// union.cuh — outputs of K12 (fused term merge + posting union) and inputs of the emit kernel.
#pragma once
#include "plan.cuh"

namespace ii2 {

// One record per DISTINCT term, in merged (ascending term) order inside its bucket: the
// records of bucket b start at index bk_pos[b] (an upper bound of the groups before it).
struct GroupRec {
  uint64_t dec;   // device address of the unioned + filtered postings (if kept decoded)
  uint64_t eoff;  // device address of the term's intcomp stream (if encoded)
  uint32_t inst;  // global instance id of one source (names the term bytes)
  uint32_t tlen;  // term length
  uint32_t cnt;   // values left after union + removed filter
  uint32_t enc;   // intcomp words of that list
};

// What K1b knows about a distinct term, in merged order inside its bucket (index = bucket base
// bk_pos[b] + rank, like GroupRec).
struct __align__(16) GroupIn {
  uint32_t inst;   // global instance id of one source (names the term bytes)
  uint32_t tlen;   // term length
  uint32_t src;    // first source in src_ptr / src_len (filled for heavy terms only)
  uint32_t c;      // number of sources
  uint32_t L;      // Σ source lengths if <= REG_CAP, anything larger otherwise
  uint32_t pst;    // postings of the light terms before it in the bucket: its gather slot
  uint32_t eslot;  // `_val` staging words reserved before it in the bucket
  uint32_t pad;
};


struct LargeArgs {
  const uint32_t* rec;     // record index of the term (same index in gin and recs)
  const uint32_t* bucket;
  const GroupIn* gin;
  const uint64_t* src_ptr;
  const uint32_t* src_len;
  uint64_t* len;           // Σ source lengths
  const uint64_t* off;     // offset into tmp
  const uint64_t* eoff;    // offset into enc (upper-bound slots)
  uint32_t* tmp;
  uint32_t* enc;
  GroupRec* recs;
  RemovedSet rem;
  int want_enc, keep_empty;
  int always_sort;         // sort + dedup single-source groups too (prefix search)
  const uint8_t* presorted;  // [n] groups already sorted + deduped by the bitmap path, or null
  uint64_t* bk_raw;        // per-bucket totals to add to, or null
  uint32_t nb1;
};

// ---- K12f (k12_fused.cu): a whole bucket in one kernel --------------------------------------
constexpr uint32_t F_MAXK = 256;  // segments per call on the fused path
// bk_mode[b]: how bucket b's output is laid out for the placement kernels (k6_emit.cu)
constexpr uint32_t K12F_RECORDS = 0;   // per-term GroupRec + upper-bound slots (K1b / K2b)
constexpr uint32_t K12F_DENSE = 1;     // dense, merged order, in the bucket's staging areas (K12f)
constexpr uint32_t K12F_DEFERRED = 2;  // K12f passed: the general kernels run it (-> records)

struct K12fArgs {
  const SegDesc* segs;
  int k;
  const uint32_t* part;  // boundary tables of the plan
  const uint32_t* btb;
  const uint64_t* bpo;
  const uint64_t* bk_pos;
  const uint32_t* bk_cpl;
  const uint64_t* bk_P;
  const uint64_t* bk_E;
  const uint64_t* bk_TB;
  RemovedSet rem;
  int want_enc, want_dec, keep_empty;
  uint32_t* bk_D;
  uint32_t* bk_mode;
  uint64_t* bk_raw;  // [4][nb1], zeroed
  uint32_t nb1;
  // dense staging of bucket b: term bytes at bk_TB[b], `_val` words at bk_E[b], decoded
  // postings at bk_P[b]; per surviving term (index bk_pos[b] + t) its offsets relative to the
  // bucket: first term byte, first word, first posting
  uint8_t* st_tb;
  uint32_t* st_toff;
  uint32_t* st_eoff;
  uint32_t* st_poff;
  uint32_t* st_enc;
  uint32_t* st_post;
  uint32_t* n_def;     // deferred buckets
  uint32_t* def_list;
};
bool k12f_supported(int k);
int k12f_launch(const K12fArgs& a, uint32_t n_buckets, cudaStream_t s);

int k2_large_run(LargeArgs la, uint32_t n_groups, DevBuf<uint32_t>& large_tmp,
                 DevBuf<uint32_t>& large_enc, cudaStream_t s);

struct UnionOut {
  DevBuf<GroupRec> recs;       // [N_T]
  DevBuf<uint32_t> tmp_post;   // [N_in] gather slots of the light terms, replaced by their unions
  DevBuf<uint32_t> tmp_enc;    // encoded streams, one upper-bound slot per light term
  DevBuf<uint32_t> large_enc;  // the same for heavy terms
  DevBuf<uint32_t> large_tmp;  // sort space of the multi-CTA path for heavy terms
  DevBuf<uint32_t> med_post;   // unions of the medium terms (one CTA each)
  DevBuf<uint32_t> med_enc;    // their `_val` streams
  DevBuf<uint32_t> bk_D;       // [B] distinct terms per bucket
  // fused path (K12f): dense per-bucket staging
  bool fused = false;
  DevBuf<uint8_t> st_tb;       // [Σ term bytes of all instances] merged term bytes, bucket b at bk_TB[b]
  DevBuf<uint32_t> st_off;     // [3][N_T] bucket-relative term-byte / word / posting offsets
  DevBuf<uint32_t> bk_mode;    // [B] K12F_*
  DevBuf<uint32_t> def_list;   // [B] buckets K12f left to the general kernels
  uint32_t n_def = 0;
  // [4][B+1] per bucket {surviving terms, their term bytes, postings out, encoded words}
  DevBuf<uint64_t> bk_raw;
  DevBuf<uint64_t> bk_out;     // exclusive prefixes of bk_raw
  DevBuf<uint64_t> totals;     // [4] device (+ scratch counters behind)
  uint64_t h_totals[4] = {0, 0, 0, 0};
  uint64_t terms_merged = 0;   // Σ bk_D
  bool keep_empty = false;     // reads without a filter keep terms whose list is empty
  bool want_dec = false, want_enc = false;
  // Early emit (small fused calls): the caller names the result; K12 launches the dense
  // placement into arrays sized by the input's upper bounds right behind the bucket kernel and
  // the totals, BEFORE it waits for the totals — one host round trip instead of two.  If a
  // bucket had to be deferred the placement is simply redone by k6_emit.
  struct EmitOut* early_out = nullptr;
  bool emitted_early = false;
};

// K12: per bucket, finish the k-way term merge (group equal terms, order the distinct ones) and
// union + dedup the posting lists of every term with the removed filter in the same pass
// (file.MergeTermValues file/types.go:14-22 for terms with >= 2 sources, pass-through for
// single-source terms; filter shard.go:181-190); encode (intcomp) while the list is still in
// shared memory.  Synchronises the stream once to learn the output sizes.
// keep_empty: terms left with no values are kept (plain reads) instead of dropped (merge,
// shard.go:192-194).
// n_in / tb_in: input postings / term bytes inside the windows (upper bounds size the staging).
int k12_union(const MergePlan& plan, const RemovedSet& rem, bool want_dec, bool want_enc,
              bool keep_empty, uint64_t n_in, uint64_t tb_in, UnionOut& u, cudaStream_t s);

struct EmitOut {
  DevBuf<uint8_t> term_bytes;
  DevBuf<uint32_t> term_off;  // [T+1]
  DevBuf<uint32_t> post;      // [P]    (if want_dec)
  DevBuf<uint64_t> post_off;  // [T+1]  (if want_dec)
  DevBuf<uint32_t> val_words; // [E]    (if want_enc)
  DevBuf<uint64_t> val_off;   // [T]    byte offsets (if want_enc)
};

// Emit: surviving terms (non-empty after the filter, shard.go:192-194) with compact term
// bytes/offsets, decoded postings and/or the `_val` stream with running byte offsets
// (Writer.Append, file/writer.go:43-56).  Pure gather/copy: everything was computed by K12.
int k6_emit(const MergePlan& plan, const UnionOut& u, EmitOut& out, cudaStream_t s);
// The dense placement alone, into arrays sized by upper bounds (T <= instances, term bytes <=
// tb_in, postings <= n_in); no synchronisation, reads the prefixes on the device.
int k6_emit_early(const MergePlan& plan, UnionOut& u, uint64_t n_in, uint64_t tb_in, EmitOut& out,
                  cudaStream_t s);

// Read(min == max) as one kernel (k12_union.cu, k4_point_kernel): h_segs / term live in pinned
// host memory (the kernel reads them in place), h_res = 5 pinned words {status, T, P, postings in,
// segments holding the term}; status 1 = the result is in `out` (one term or none), 2 = more than
// 4096 values: take the general path.  Decoded output only.  No synchronisation.
constexpr uint32_t kPointMaxTerm = 8192;  // term bytes the kernel stages in shared memory
int k4_point_read(const SegDesc* h_segs, int k, const uint8_t* term, uint32_t tlen,
                  const RemovedSet& rem, bool keep_empty, EmitOut& out, uint64_t* h_res,
                  cudaStream_t s);

// First and last term of the merged order (pre-filter min/max, shard.go:176-179).
// d_out: [0]=len_min [1]=len_max (u32), bytes from +8 (min then max); needs 8 + 2*65536 bytes.
int k6_minmax(const MergePlan& plan, const UnionOut& u, uint8_t* d_out, cudaStream_t s);

}  // namespace ii2
