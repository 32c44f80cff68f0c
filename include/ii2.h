/*
 * ii2.h — C-ABI of the B200-native hot path of lezhnev74/inverted_index_2:
 * segment compaction and multi-segment term-range reads.
 *
 * This is the header a Go maintainer would `#include` from a cgo preamble
 * (see INTEGRATION.md).  Plain pointers and sizes only.  Every entry point
 * names the reference code it replaces (paths relative to the reference repo).
 *
 * Conventions
 *   - return value: 0 (II2_OK) or a negative II2_ERR_* code; ii2_strerror()
 *     gives the text.  "No term in range" is NOT an error: the output is
 *     empty, like the vellum.ErrIteratorDone handling in shard.go:257-261.
 *   - inputs are borrowed for the duration of the call only (no Go pointer is
 *     retained across the cgo call); outputs are allocated by the library
 *     (pinned host memory) and released with the matching *_free().
 *   - re-entrant: any number of host threads may call concurrently (the
 *     reference calls this path from many goroutines: inverted_index.go:83-103,
 *     :239-285).  Each call uses its host thread's stream + scratch arena on
 *     the call's device (see ii2_init for processes that drive several GPUs).
 *     ii2_bitmask objects are NOT thread-safe, like file/bitmask.go:10.
 *   - there is no CPU fallback: without a usable CUDA device every compute
 *     entry point returns II2_ERR_NO_DEVICE.
 */
#ifndef II2_H
#define II2_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define II2_ABI_VERSION 2

/* ---- error codes -------------------------------------------------------- */
#define II2_OK 0
#define II2_ERR_INVALID (-1)     /* bad argument / malformed view              */
#define II2_ERR_NOMEM (-2)       /* host or device allocation failed           */
#define II2_ERR_CUDA (-3)        /* CUDA runtime error (see ii2_last_error)    */
#define II2_ERR_NO_DEVICE (-4)   /* no CUDA device / ii2_init not successful   */
#define II2_ERR_BITMASK_OOB (-5) /* "bitmask is out of bound" bitmask.go:41-44 */
#define II2_ERR_CORRUPT (-6)     /* undecodable _val run or roaring buffer     */
#define II2_ERR_UNSUPPORTED (-7) /* input beyond an implementation limit       */

/* ---- segment views ------------------------------------------------------ */
/* How the postings of a segment are handed over. */
#define II2_SEG_DECODED 0 /* post[] + post_off[]  (already-decoded uint32 lists)              */
#define II2_SEG_VAL 1     /* raw <key>_val bytes + the FST outputs (file/reader.go:50-52,64)  */
#define II2_SEG_DIRECT 2  /* no _val file: FST output IS the posting (file/reader.go:73-77)   */

/*
 * One immutable segment, flattened.  Terms are in ascending bytes.Compare
 * order (the order vellum iterates them, file/reader.go:147), concatenated in
 * term_bytes; term i is term_bytes[term_off[i] .. term_off[i+1]).
 * Replaces the per-term file.TermValues objects of file/types.go:9-12.
 *
 * Alignment contract: term_bytes and val_bytes may start at ANY address (a Go
 * sub-slice, an mmap offset); term_off / post / post_off / val_off must be
 * naturally aligned for their element type (4 / 4 / 8 / 8 bytes), as Go slices
 * of those types always are.  Arrays are borrowed for the call only.  Offsets
 * are validated (monotone, inside the arrays): corrupt input is II2_ERR_INVALID.
 * An empty segment (n_terms == 0) may leave every pointer NULL.
 */
typedef struct ii2_seg_view {
  uint64_t n_terms;
  const uint8_t* term_bytes;
  const uint32_t* term_off; /* n_terms + 1 */
  int32_t mode;             /* II2_SEG_*   */
  /* II2_SEG_DECODED */
  const uint32_t* post;     /* post_off[n_terms] values                    */
  const uint64_t* post_off; /* n_terms + 1, in values                      */
  /* II2_SEG_VAL: val_off[i] = FST output of term i = byte offset of its run;
   * run i ends at val_off[i+1] (file/reader.go:52) or val_size (:64).
   * II2_SEG_DIRECT: val_off[i] = FST output = the single posting, truncated
   * to uint32 exactly like file/reader.go:75. */
  const uint8_t* val_bytes;
  const uint64_t* val_off; /* n_terms */
  uint64_t val_size;
  /* II2_SEG_VAL only, optional (ABI version 2): the same FST outputs as 32-bit WORD offsets
   * (val_off[i] / 4) for `_val` files below 16 GiB; when non-NULL it is used instead of
   * val_off (which may then be NULL) and halves the offset bytes that cross the bus. */
  const uint32_t* val_woff32; /* n_terms */
} ii2_seg_view;

/* ---- lifecycle ---------------------------------------------------------- */
/* Bind the calling process to the CUDA devices devices[0 .. ndev), 1 <= ndev <= 16
 * distinct ordinals, every one an sm_100 device.  devices == NULL (or ndev == 0)
 * picks device 0.  Peer access is enabled in this process for every ordered pair of
 * the set the hardware allows.  Called from NewInvertedIndex (inverted_index.go:342).
 * Idempotent for the same set (in any order); any other set, a duplicate or an
 * out-of-range ordinal is II2_ERR_INVALID.
 *
 * Devices of a bound set
 *   - host-buffer calls (ii2_merge, ii2_read_range, ii2_ingest, ii2_prefix_search,
 *     the codecs, ii2_bitmask_new) and uploads (ii2_seg_upload, ii2_removed_upload)
 *     run on the device the calling host thread selected with ii2_set_device
 *     (devices[0] until it does);
 *   - every handle (ii2_seg, ii2_removed, ii2_result, ii2_bitmask) lives on the
 *     device that created it, and calls that take handles (the _dev calls, downloads,
 *     ii2_result_to_seg, releases, bitmask operations) run there, whatever the thread
 *     selected.  Handles of different devices in one call are II2_ERR_INVALID.
 *     Segments never move between devices;
 *   - streams, scratch memory and ii2_set_stream bindings belong to a (host thread,
 *     device) pair; pinned host outputs are process-wide and usable from every device.
 *   - a call leaves its device current on the calling thread. */
int ii2_init(const int* devices, int ndev);
int ii2_shutdown(void);
int ii2_abi_version(void);
const char* ii2_strerror(int code);
/* Thread-local detail string of the last failing call on this thread. */
const char* ii2_last_error(void);
/* Select the device of this host thread's host-buffer calls and uploads: a CUDA
 * ordinal of the bound set, else II2_ERR_INVALID.  Go moves goroutines between OS
 * threads: wrap the selection and the calls it governs in runtime.LockOSThread. */
int ii2_set_device(int device);
/* Launch on a caller-owned CUDA stream (cudaStream_t as void*) instead of a
 * pooled one, for this host thread and the device it selected (the stream must
 * belong to that device); NULL restores the pool.  Lets a host framework time the
 * kernels with its own events. */
int ii2_set_stream(void* cuda_stream);
/* Number of kernels this library launched since ii2_init (all threads). */
uint64_t ii2_kernel_launches(void);
/* Instrumentation for bench.py's roofline: while enabled, every kernel phase of the
 * pipelines is bracketed by CUDA events on the launching stream.  ii2_prof_read
 * aggregates by phase name (total ms, number of launches) since the last enable and
 * returns the number of entries written (<= cap), or a negative error. */
typedef struct ii2_prof_entry {
  const char* name;
  double ms;      /* device time between the phase's events */
  double host_ms; /* host wall time spent inside the phase (launch + allocation + waits) */
  uint64_t count;
} ii2_prof_entry;
int ii2_prof_enable(int on);
int ii2_prof_read(ii2_prof_entry* out, int cap);
/* Generic release for buffers documented as "free with ii2_free". */
void ii2_free(void* p);

/* ---- compaction: replaces the merge loop shard.go:158-212 ---------------- */
#define II2_MERGE_WANT_DECODED 1u /* also return decoded post/post_off */

typedef struct ii2_merge_out {
  /* terms appended to the new segment, i.e. non-empty after the removed
   * filter (termsCount, shard.go:211).  0 ⇒ no segment is written
   * (lazy writer, shard.go:197-205,219). */
  uint64_t terms_count;
  uint8_t* term_bytes;
  uint32_t* term_off; /* terms_count + 1 */
  /* What Writer.Append produces (file/writer.go:43-56): val_off[i] is the FST
   * output of term i (running valuesOffset), val_bytes the <key>_val file. */
  uint64_t* val_off; /* terms_count */
  uint8_t* val_bytes;
  uint64_t val_size;
  /* minTerm / maxTerm as shard.go:176-179 records them: BEFORE the removed
   * filter, so they may name dropped terms (survey quirk Q3). */
  int32_t has_minmax;
  uint8_t* min_term;
  uint32_t min_term_len;
  uint8_t* max_term;
  uint32_t max_term_len;
  /* only with II2_MERGE_WANT_DECODED */
  uint32_t* post;
  uint64_t* post_off; /* terms_count + 1 */
  /* accounting */
  uint64_t terms_merged;  /* distinct terms before the filter */
  uint64_t postings_in;   /* Σ input list lengths             */
  uint64_t postings_out;  /* Σ output list lengths            */
  void* _owner;
} ii2_merge_out;

/* k-way merge of the segments' term dictionaries (go-iterators MergingIterator
 * built at shard.go:267 with file.CompareTermValues, file/types.go:24-26),
 * per-term sorted-unique union for terms present in >= 2 segments
 * (file.MergeTermValues, file/types.go:14-22; single-source lists pass through
 * untouched, quirk Q4), removed filter by membership in removed_sorted
 * (shard.go:181-190), empty-term drop (:192-194) and intcomp encoding with
 * running offsets (file/writer.go:43-56) in one device pass.
 * removed_sorted: ascending, duplicates allowed (removed_list.go:44-54). */
int ii2_merge(const ii2_seg_view* segs, int nseg, const uint32_t* removed_sorted,
              uint64_t nrem, uint32_t flags, ii2_merge_out* out);
void ii2_merge_out_free(ii2_merge_out* out);

/* ---- ingest batching: replaces D calls of Shard.Put (shard.go:33-67) and the
 *      Shard.Merge that later folds their segments ---------------------------- */
typedef struct ii2_doc_view {
  uint64_t n_terms;
  const uint8_t* term_bytes; /* the document's terms in ANY order: Put sorts them (shard.go:34) */
  const uint32_t* term_off;  /* n_terms + 1 */
  uint32_t value;            /* every term of the document maps to [value] (shard.go:47)     */
} ii2_doc_view;

/* The segment that Put(docs[0]) .. Put(docs[n-1]) followed by one Merge of the
 * resulting direct-mode segments produces: terms sorted on the device (one
 * segmented sort over all documents), a term repeated inside a document kept
 * once, then the same pipeline as ii2_merge (union per term, removed filter,
 * intcomp `_val` stream, FST outputs).  At most 1024 documents per call. */
int ii2_ingest(const ii2_doc_view* docs, int ndocs, const uint32_t* removed_sorted,
               uint64_t nrem, uint32_t flags, ii2_merge_out* out);

/* ---- term-range read: replaces shard.go:253-278 + the iterator pulls ----- */
typedef struct ii2_read_out {
  uint64_t n_terms;
  uint8_t* term_bytes;
  uint32_t* term_off; /* n_terms + 1 */
  uint32_t* post;
  uint64_t* post_off; /* n_terms + 1 */
  void* _owner;
} ii2_read_out;

/* Union over all segments of the terms in [min,max] (both inclusive, NULL =
 * open; file/reader.go:147-155 and :54-58), ascending by term.  The reference
 * read path does not filter removed values (shard.go:72-75, quirk Q2); pass
 * removed_sorted != NULL only to reproduce the benchmark composition "read +
 * merge-style filter", which also drops emptied terms. */
int ii2_read_range(const ii2_seg_view* segs, int nseg, const uint8_t* min, size_t minlen,
                   const uint8_t* max, size_t maxlen, const uint32_t* removed_sorted,
                   uint64_t nrem, ii2_read_out* out);
void ii2_read_out_free(ii2_read_out* out);

/* ---- device-resident segments (keeps PCIe staging off the hot path) ------ */
typedef struct ii2_seg ii2_seg;         /* a segment living in HBM            */
typedef struct ii2_removed ii2_removed; /* removed list (+ bitmap) in HBM     */
typedef struct ii2_result ii2_result;   /* merge / read result in HBM         */

int ii2_seg_upload(const ii2_seg_view* view, ii2_seg** seg);
void ii2_seg_release(ii2_seg* seg);
int ii2_removed_upload(const uint32_t* removed_sorted, uint64_t nrem, ii2_removed** rem);
void ii2_removed_release(ii2_removed* rem);

/* Same work as ii2_merge / ii2_read_range on resident inputs; the result stays
 * in HBM until downloaded.  `flags` selects what a merge produces:
 * II2_RESULT_ENCODED = the intcomp `_val` stream + FST outputs (what Writer.Append
 * writes, file/writer.go:43-56), II2_RESULT_DECODED = decoded postings (needed by
 * ii2_result_to_seg / ii2_result_download_read); 0 means decoded only.
 * The result of a small read (<= 65 536 term instances in range) holds device arrays sized by
 * the range's input (it is placed before the output sizes are known: one host round trip
 * less); the counts in ii2_result_info are exact.  Release results you do not keep. */
#define II2_RESULT_ENCODED 1u
#define II2_RESULT_DECODED 2u
int ii2_merge_dev(ii2_seg* const* segs, int nseg, const ii2_removed* rem, uint32_t flags,
                  ii2_result** res);
int ii2_read_range_dev(ii2_seg* const* segs, int nseg, const uint8_t* min, size_t minlen,
                       const uint8_t* max, size_t maxlen, const ii2_removed* rem,
                       ii2_result** res);

typedef struct ii2_result_info {
  uint64_t terms_count, term_bytes, postings_out, postings_in, terms_merged, val_size;
  /* device pointers (valid until ii2_result_release) — for NCCL gathers */
  const void* d_term_bytes;
  const void* d_term_off; /* u32[terms_count+1] */
  const void* d_post;     /* u32[postings_out]  */
  const void* d_post_off; /* u64[terms_count+1] */
  const void* d_val_bytes;
  const void* d_val_off; /* u64[terms_count]   */
} ii2_result_info;
int ii2_result_info_get(const ii2_result* res, ii2_result_info* info);
int ii2_result_download_merge(const ii2_result* res, uint32_t flags, ii2_merge_out* out);
int ii2_result_download_read(const ii2_result* res, ii2_read_out* out);
/* Adopt a decoded result as a resident segment (for multi-pass compaction). */
int ii2_result_to_seg(ii2_result* res, ii2_seg** seg);
void ii2_result_release(ii2_result* res);
/* Block until everything queued by this thread's streams is done. */
int ii2_sync(void);
/* The CUDA device a result lives on (routes follow-up calls; where a gather put it). */
int ii2_result_device(const ii2_result* res, int* device);

/* ---- PrefixSearch: replaces the per-shard scan of InvertedIndex.PrefixSearch
 *      (inverted_index.go:239-292) ------------------------------------------ */
typedef struct ii2_prefix_out {
  uint64_t n_prefixes;
  /* matched[i] != 0 <=> at least one term starts with prefix i, i.e. prefix i
   * is a key of the map PrefixSearch returns (inverted_index.go:274-279; a
   * matching term with an empty list still creates the key). */
  uint8_t* matched;
  /* found[prefix i] = values[value_off[i] .. value_off[i+1]): the values of
   * every term with that prefix over all segments, sorted and compacted
   * (slices.Sort + slices.Compact, inverted_index.go:289-292). */
  uint32_t* values;
  uint64_t* value_off; /* n_prefixes + 1 */
  void* _owner;
} ii2_prefix_out;

/* Prefix i = prefix_bytes[prefix_off[i] .. prefix_off[i+1]); any order,
 * duplicates and the empty prefix allowed (the reference sorts them only to
 * bound its scan, inverted_index.go:196,266-271).  `segs` may be the segments
 * of ALL shards at once: shard selection by min/max (:211-236) only skips
 * shards that cannot match.  No removed filter (reads never filter, shard.go:72-75). */
int ii2_prefix_search_dev(ii2_seg* const* segs, int nseg, const uint8_t* prefix_bytes,
                          const uint32_t* prefix_off, uint32_t nprefix, ii2_prefix_out* out);
int ii2_prefix_search(const ii2_seg_view* segs, int nseg, const uint8_t* prefix_bytes,
                      const uint32_t* prefix_off, uint32_t nprefix, ii2_prefix_out* out);
void ii2_prefix_out_free(ii2_prefix_out* out);

/* ---- batched term lookup: InvertedIndex.Read(t, t) for many keys t in one call */
typedef struct ii2_lookup_out {
  uint64_t n_keys;
  uint8_t* found;       /* n_keys: != 0 <=> Read(key, key) yields the term          */
  uint32_t* post;       /* key i's list = post[post_off[i] .. post_off[i+1])        */
  uint64_t* post_off;   /* n_keys + 1                                               */
  uint64_t postings_in; /* Σ lengths of the source lists that were unioned          */
  void* _owner;
} ii2_lookup_out;

/* Key i = key_bytes[key_off[i] .. key_off[i+1]); any order, duplicates and the
 * empty key allowed.  For every key, found[i] and list i are exactly the term and
 * list ii2_read_range_dev(segs, nseg, key, key, rem) returns:
 *   - no segment holds the key: found = 0, empty list;
 *   - one segment holds it: that list as stored (possibly unsorted, duplicates kept);
 *   - two or more hold it: the sorted-unique union, even when some lists are empty;
 *   - without rem a key held only with empty lists is found with an empty list;
 *   - with rem the removed values are dropped after the union, and a key whose list
 *     ends empty is not found.
 * ii2_lookup_dev runs on the device of its handles (handles of two devices:
 * II2_ERR_INVALID); ii2_lookup uploads the views to the device the thread selected.
 * nkeys == 0 or nseg == 0 gives empty results.  Outputs are pinned host memory;
 * free them with ii2_lookup_out_free.  II2_ERR_INVALID: NULL out, NULL data
 * pointers, key_off not monotone.  II2_ERR_UNSUPPORTED: more than 1024 segments,
 * a key longer than 65 535 bytes, one key's union of 2^32 postings or more. */
int ii2_lookup_dev(ii2_seg* const* segs, int nseg, const uint8_t* key_bytes,
                   const uint32_t* key_off, uint32_t nkeys, const ii2_removed* rem,
                   ii2_lookup_out* out);
int ii2_lookup(const ii2_seg_view* segs, int nseg, const uint8_t* key_bytes,
               const uint32_t* key_off, uint32_t nkeys, const uint32_t* removed_sorted,
               uint64_t nrem, ii2_lookup_out* out);
void ii2_lookup_out_free(ii2_lookup_out* out);

/* ---- boolean term queries: AND / OR / NOT over exact terms and prefixes, many
 *      queries per call (an extension beyond the reference's read surface) ---- */
#define II2_ATOM_TERM 0
#define II2_ATOM_PREFIX 1
/* Q queries as three nested CSR levels: atom a = atom_bytes[atom_off[a] ..
 * atom_off[a+1]) of kind atom_kind[a]; the atoms of clause c are
 * [clause_atom_off[c], clause_atom_off[c+1]); the clauses of query q are
 * [query_clause_off[q], query_clause_off[q+1]).  Every offset array starts at 0
 * and is monotone; clause_atom_off[nclauses] == natoms and
 * query_clause_off[nqueries] == nclauses. */
typedef struct ii2_query_batch {
  const uint8_t* atom_bytes;
  const uint32_t* atom_off;         /* natoms + 1   */
  const uint8_t* atom_kind;         /* natoms: II2_ATOM_* */
  uint32_t natoms;
  const uint32_t* clause_atom_off;  /* nclauses + 1 */
  const uint8_t* clause_excluded;   /* nclauses: 0 = required, 1 = excluded */
  uint32_t nclauses;
  const uint32_t* query_clause_off; /* nqueries + 1 */
  uint32_t nqueries;
} ii2_query_batch;

typedef struct ii2_query_out {
  uint64_t n_queries;
  uint32_t* values;        /* query i = values[value_off[i] .. value_off[i+1])  */
  uint64_t* value_off;     /* n_queries + 1                                      */
  uint64_t clause_values;  /* Σ sizes of the clause unions (work accounting)     */
  void* _owner;
} ii2_query_out;

/* Semantics:
 *   - values(TERM t)   = the sorted-unique set of t's values over all segments.
 *     This is a set even when one segment holds t: unlike Read(t, t), which
 *     passes a single-source list through as stored (quirk Q4).  An absent term
 *     gives the empty set.
 *   - values(PREFIX p) = found[p] of PrefixSearch, i.e. exactly the list
 *     ii2_prefix_search_dev returns for p.  An unmatched prefix gives the empty
 *     set; the empty prefix matches every term.
 *   - values(clause)   = the union of its atoms; a clause with no atoms is the
 *     empty set.
 *   - result(query)    = the intersection of its required clauses, minus the
 *     union of its excluded clauses, minus the removed set when rem != NULL
 *     (reads never filter, quirk Q2, so rem is optional).  Ascending and unique.
 *   - a query needs at least one required clause (there is no universe):
 *     otherwise the call is II2_ERR_INVALID.  Duplicate atoms, clauses and
 *     queries are allowed.
 * ii2_query_dev runs on the device of its handles (handles of two devices:
 * II2_ERR_INVALID); ii2_query uploads the views to the device the thread
 * selected.  nqueries == 0 or nseg == 0 gives empty lists.  Outputs are pinned
 * host memory; free them with ii2_query_out_free.  On error *out is zeroed.
 * II2_ERR_INVALID (checked before any launch): NULL out or q, NULL arrays,
 * non-monotone offsets, a first offset other than 0, a last offset that
 * disagrees with the count of the next level, an unknown atom kind or clause
 * flag, a query without a required clause.  II2_ERR_UNSUPPORTED: more than 1024
 * segments, an atom longer than 65 535 bytes, a clause of more than 1024 atoms,
 * a union of 2^32 values or more, natoms x nseg >= 2^32. */
int ii2_query_dev(ii2_seg* const* segs, int nseg, const ii2_query_batch* q,
                  const ii2_removed* rem, ii2_query_out* out);
int ii2_query(const ii2_seg_view* segs, int nseg, const ii2_query_batch* q,
              const uint32_t* removed_sorted, uint64_t nrem, ii2_query_out* out);
void ii2_query_out_free(ii2_query_out* out);

/* ---- cross-shard exchange: one process per GPU, contiguous shard-key ranges per
 *      rank (shardKey, shard.go:362-378), NCCL over NVLink --------------------
 * Compaction needs no exchange (shards never interact, shard.go:19-20).  Reads
 * that span ranks do: InvertedIndex.Read concatenates the shard streams in key
 * order (inverted_index.go:330-338) and PrefixSearch unions the per-shard maps,
 * then slices.Sort + slices.Compact (inverted_index.go:274-292). */
#define II2_COMM_ID_BYTES 128
/* Rank 0 makes the id (ncclGetUniqueId) and hands it to the other processes by
 * any host channel; then every process calls ii2_comm_init on the device it
 * bound with ii2_init.  One communicator per process. */
int ii2_comm_unique_id(uint8_t* id /* II2_COMM_ID_BYTES */);
int ii2_comm_init(const uint8_t* id, int rank, int world);
int ii2_comm_info(int* rank, int* world); /* world = 0 before ii2_comm_init */
void ii2_comm_shutdown(void);
/* Collective: every rank passes its own decoded result (ii2_read_range_dev over
 * its shards).  `gathered` on rank `root` (every rank if root < 0) is the
 * rank-ordered concatenation, offsets rebased — what InvertedIndex.Read yields
 * over all shards; the other ranks get an empty result.  One size all-gather,
 * one group of sends / receives, no padding. */
int ii2_read_gather(const ii2_result* local, int root, ii2_result** gathered);
/* Collective: every rank passes its ii2_prefix_search(_dev) result for the SAME
 * prefix list.  `merged` on the root: per prefix the sorted-unique union of
 * every rank's values, matched = OR of the ranks' flags (the final sort + compact
 * runs on the root GPU).  Free with ii2_prefix_out_free. */
int ii2_prefix_gather(const ii2_prefix_out* local, int root, ii2_prefix_out* merged);
/* (ii2_comm_init is II2_ERR_INVALID in a process that bound more than one device:
 * NCCL is for one process per GPU; the calls below serve one process over many.) */

/* ---- in-process cross-device gathers: one process, several bound devices ------
 * The caller fans out (one host thread / goroutine per device, as the reference
 * fans out over shards), then gathers on a root device of the set. */
/* parts[0 .. nparts) are decoded read results (ii2_read_range_dev; an encoded-only
 * merge result is II2_ERR_INVALID) in shard-key order, on any bound devices.
 * `gathered` lives on root_device: the concatenation in part order, offsets
 * rebased — what InvertedIndex.Read's sequential concatenation yields
 * (inverted_index.go:330-338) and what ii2_read_gather gives its root.  ONE kernel
 * on the root reads every part straight from its device's HBM (peer access) and
 * writes it to its final place.  The call waits for the streams that produced the
 * parts (they must still exist) and returns when the result is complete.  Limits:
 * < 4 GiB of term bytes, < 2^32-1 terms, at most 64 parts (II2_ERR_UNSUPPORTED);
 * a part on a device the root cannot read by peer access is II2_ERR_UNSUPPORTED.
 * nparts == 0 gives an empty result on the root. */
int ii2_read_gather_devices(const ii2_result* const* parts, int nparts, int root_device,
                            ii2_result** gathered);
/* parts are ii2_prefix_search(_dev) outputs for the SAME prefix list (one per
 * device or shard group; II2_ERR_INVALID if n_prefixes differ).  `merged`: per
 * prefix the sorted-unique union of the parts' values, matched = OR of the parts'
 * flags (inverted_index.go:274-292); the union runs on root_device.  Free with
 * ii2_prefix_out_free. */
int ii2_prefix_gather_devices(const ii2_prefix_out* parts, int nparts, int root_device,
                              ii2_prefix_out* merged);

/* ---- posting codec: replaces intcomp.CompressUint32 (file/writer.go:49) and
 *      intcomp.UncompressUint32 (file/reader.go:100), batched ---------------- */
/* list i = in[off[i] .. off[i+1]); out words of list i =
 * words[word_off[i] .. word_off[i+1]).  Outputs: free with ii2_free. */
int ii2_intcomp_encode_u32(const uint32_t* in, const uint64_t* off, uint64_t nlists,
                           uint32_t** words, uint64_t** word_off);
int ii2_intcomp_decode_u32(const uint32_t* words, const uint64_t* word_off, uint64_t nlists,
                           uint32_t** out, uint64_t** out_off);

/* ---- file/bitmask.go ------------------------------------------------------ */
typedef struct ii2_bitmask ii2_bitmask;
/* NewBitmask (file/bitmask.go:20): the dictionary starts as init[0..n). */
int ii2_bitmask_new(const uint32_t* init, uint64_t n, ii2_bitmask** bm);
void ii2_bitmask_free(ii2_bitmask* bm);
/* AllValues (:24).  Free with ii2_free. */
int ii2_bitmask_all_values(const ii2_bitmask* bm, uint32_t** vals, uint64_t* n);
/* Put (:53-59): dictionary index of every value (first occurrence; appended on
 * miss in input order, :64-71), bits set in a roaring bitmap, portable
 * serialisation returned.  Free bytes with ii2_free. */
int ii2_bitmask_put(ii2_bitmask* bm, const uint32_t* vals, uint64_t n, uint8_t** bytes,
                    uint64_t* nbytes);
/* Get (:30-49): parse ONE bitmap from the front of enc (trailing bytes are
 * ignored, file/bitmask_test.go:44-46), map ascending indexes through the
 * dictionary; II2_ERR_BITMASK_OOB if an index >= len(dictionary). */
int ii2_bitmask_get(const ii2_bitmask* bm, const uint8_t* enc, uint64_t nenc, uint32_t** vals,
                    uint64_t* n);

/* ---- <key>_fst term dictionaries: blevesearch/vellum v1 FST files ----------
 * Host-side (no device work, usable without a GPU).  Replaces vellum.Open +
 * fst.Iterator(min, nil) + the manual inclusive max bound of the reader
 * (file/reader.go:139-155, :48-58) and vellum.New / Insert / Close of the writer
 * (file/writer.go:35,43,62,104-129).  Format restated from the vellum module,
 * which is not in the reference tree: bytes unverified against Go (see
 * csrc/fst_v1.cpp). */
typedef struct ii2_fst_terms {
  uint64_t n_terms;    /* keys in [min,max]                                   */
  uint8_t* term_bytes; /* ascending bytes.Compare order, 32 readable pad bytes */
  uint32_t* term_off;  /* n_terms + 1                                          */
  uint64_t* values;    /* FST outputs: `_val` byte offsets, or the posting itself
                        * in direct mode (file/writer.go:35,43)                 */
  uint64_t fst_len;    /* keys in the whole FST (its footer)                   */
  void* _owner;
} ii2_fst_terms;

/* All keys k with min <= k <= max (NULL = open), with their outputs: what the
 * reader's FST iterator yields.  The result plugs into ii2_seg_view as
 * term_bytes / term_off / val_off (modes II2_SEG_VAL and II2_SEG_DIRECT). */
int ii2_fst_read(const uint8_t* fst, uint64_t nbytes, const uint8_t* min, size_t minlen,
                 const uint8_t* max, size_t maxlen, ii2_fst_terms* out);
void ii2_fst_terms_free(ii2_fst_terms* out);
/* fst.Get: *found = 0 if the key is absent. */
int ii2_fst_get(const uint8_t* fst, uint64_t nbytes, const uint8_t* key, size_t keylen,
                uint64_t* value, int* found);
int ii2_fst_len(const uint8_t* fst, uint64_t nbytes, uint64_t* n_terms);
/* vellum.New(w, nil) + Insert(term i, values[i]) for ascending, distinct terms
 * + Close: the bytes of a `<key>_fst` file.  II2_ERR_INVALID if the terms are
 * not strictly ascending (vellum.ErrOutOfOrder).  Free with ii2_fst_free. */
int ii2_fst_build(const uint8_t* term_bytes, const uint32_t* term_off, const uint64_t* values,
                  uint64_t n_terms, uint8_t** fst, uint64_t* nbytes);
void ii2_fst_free(void* fst);

/* ---- removed.list: the gob stream of RemovedLists (removed_list.go:26-33,73-80;
 *      read/written next to the segment files, shard.go:340-358) -------------
 * Host-side.  lists[timestamps[k]] = values[off[k] .. off[k+1]).  Wire format
 * restated from the encoding/gob documentation, unverified against Go (see
 * csrc/removed_gob.cpp). */
typedef struct ii2_removed_lists {
  uint64_t n_lists;
  int64_t* timestamps; /* n_lists           */
  uint64_t* off;       /* n_lists + 1       */
  uint32_t* values;    /* off[n_lists]      */
  void* _owner;
} ii2_removed_lists;
/* RemovedLists.Serialize.  Free the bytes with ii2_fst_free. */
int ii2_removed_list_encode(const int64_t* timestamps, const uint64_t* off, const uint32_t* values,
                            uint64_t n_lists, uint8_t** bytes, uint64_t* nbytes);
/* UnserializeRemovedList. */
int ii2_removed_list_decode(const uint8_t* bytes, uint64_t nbytes, ii2_removed_lists* out);
void ii2_removed_lists_free(ii2_removed_lists* lists);

/* ---- partitioning rule: shardKey (shard.go:362-378) ---------------------- */
/* Returns the numeric shard key 0..1023 ((t[0]<<8 | t[1]) >> 6; 0 for terms
 * shorter than 2 bytes). Host-side helper, no device work. */
uint32_t ii2_shard_key(const uint8_t* term, size_t len);

#ifdef __cplusplus
}
#endif
#endif /* II2_H */
