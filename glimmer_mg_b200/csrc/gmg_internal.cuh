// glimmer_mg_b200/csrc/gmg_internal.cuh -- shared definitions of libgmgicm.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/gmg_icm.h"

#define GMG_MAX_W 32      // window bases held in one 64-bit register
#define GMG_MAX_DEPTH 12
// zero entries after the walk-ready context arrays (d_ctxf / d_ctxr): K1's software pipeline reads whole trips past the
// end of a share (k1_planes_bucketed); sized for every (contexts per thread, threads per CTA) variant it is built in
#define GMG_CTX_PAD 16384
#define GMG_PAD_WORDS 8   // 64-bit words of zero padding before/after the packed bases
#define GMG_NPROF 8
#define GMG_NSCRATCH 21
#define GMG_PROF_RING 64

void gmg_set_error(const char* fmt, ...);

#define GMG_CUDA(call)                                                                        \
  do {                                                                                        \
    cudaError_t e__ = (call);                                                                 \
    if (e__ != cudaSuccess) {                                                                 \
      gmg_set_error("CUDA error %s at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e__)); \
      return 1;                                                                               \
    }                                                                                         \
  } while (0)

#define GMG_CHECK(cond, ...)     \
  do {                           \
    if (!(cond)) {               \
      gmg_set_error(__VA_ARGS__); \
      return 1;                  \
    }                            \
  } while (0)

// device view of an ICM: only what the walks need.
//  mip   int8 [P][inner]   branch position of the nodes on levels 0..D-1 (levels that can be
//                          descended from); -1/-2 = stop here.
//  prob  float [P][N][4]   natural-log probabilities with cut nodes (mut_info_pos == -2)
//                          pre-resolved to their parent's row (icm.cc:592-597, 829-830), so a
//                          walk needs no fix-up step.
//  lut3  float [2][3][64]  only for W == 3 models (the independent model): the full-window value of
//                          every base triple, [strand][period][b(q0) | b(q0+1) << 2 | b(q0+2) << 4] where q0 is
//                          the lowest of the three sequence positions the window covers; NULL otherwise.
struct DevIcm {
  int W, D, P, N, inner;
  const int8_t* mip;
  const float* prob;
  const float* lut3;
  const float* lutp;  // W == 3 models: partial-window values [strand][lim - 1][period][raw], lim = 1, 2 unavailable positions
};

// Tables of the bucketed K1 kernel (W <= 16, D == 7, P == 3), see icm_upload:
//  mw     uint32 [P][4 + 64 + 1024]  one word per node of levels 1, 3, 5: bits 0-4 the node's shift, bits 5+5k..9+5k
//                                    the shift of child k, bit 25 / bits 26+k their stop flags.  shift = 30 - 2 *
//                                    mut_info_pos (the left shift that brings the branch base to the top two bits of
//                                    the 32-bit window register), 0 where the walk stops
//  bleaf  float [P][4][np]           log-probabilities by predicted base in the reference's dense node order (node
//                                    n's children are 4n+1 .. 4n+4) over the COMPLETED tree: descendants of a node
//                                    where walks stop carry that node's value
//  s0 / stop0                        shift / stop flag of the three roots
struct DevIcmFast {
  int valid, W, D, P, N, np;
  int s0[3], stop0[3];
  const uint32_t* mw;
  const float* bleaf;
};

struct gmg_ctx {
  int device;
  cudaStream_t stream;
  bool own_stream;
  int sm_count;
  int64_t launches;
  // scratch (grown on demand, reused across calls)
  void* scratch[GMG_NSCRATCH];
  size_t scratch_bytes[GMG_NSCRATCH];
  double* h_penalty;  // pinned staging
  int64_t* h_scalars;  // pinned: small device -> host results (totals) that must not serialise the stream
  cudaEvent_t ev_scalars;
  cudaStream_t side;   // second stream: small kernels that do not depend on the walks run beside K1 (gmg_score_orfs_g3)
  cudaEvent_t ev_fork, ev_join;
  double mg_rate[4];   // start records per base seen by the last gmg_score_orfs_mg call, by (indels, subs) mode
  int64_t train_flagged;  // nodes of the last gmg_icm_train* call that the host recomputed (gmg_ctx_train_flagged)
  int64_t indep_flagged;  // model entries of the last gmg_score_orfs_mg_gc call that the host recomputed (gmg_ctx_indep_flagged)
  struct gmg_icm* indep_tpl;  // Build_Indep_WO_Stops topology (gmg_indep_build): walk tables shared by every GC's model
  uint8_t* d_indep_src;       // [GMG_INDEP_REC] compact slot of every record entry (gmg_indep_build)
  void* h_stage;       // pinned staging for larger device -> host results (training count slabs), grown on demand
  size_t h_stage_bytes;
  // per-kernel device timing (gmg_ctx_profile): event pairs around the launches of each kernel class
  int prof_on;
  int prof_n[GMG_NPROF];
  cudaEvent_t prof_ev[GMG_NPROF][GMG_PROF_RING][2];
  double prof_ms[GMG_NPROF];
  int64_t prof_launches[GMG_NPROF];
};

// kernel classes of gmg_ctx_profile_read (values are part of the C-ABI, see gmg_icm.h)
int gmg_prof_begin(gmg_ctx* ctx, int cls);
void gmg_prof_end(gmg_ctx* ctx, int cls);

struct gmg_icm {
  gmg_ctx* ctx;
  int W, D, P, N;
  std::vector<int16_t> mip;  // [P][N]   host mirror, exactly as ICM_t::score[][].mut_info_pos
  std::vector<float> prob;   // [P][N][4] exactly as ICM_t::score[][].prob
  std::vector<float> mut_info;  // [P][N] ICM_Score_Node_t::mut_info: set by training, 0 for models read from a file
  int8_t* d_mip;
  float* d_prob;
  DevIcm dev;
  uint8_t* d_msh;
  float* d_bleaf;
  float* d_lut3;
  float* d_lutp;
  DevIcmFast fast;
  int ready;  // device views built (gmg_icm_ready)
  // value statistics of `prob` (computed with the device views, see gmg_icm_value_stats)
  int stat_valid, stat_ulp_exp;
  float stat_max_abs;
};

// smallest ulp exponent (every entry is an integer multiple of 2^ulp_exp) and largest magnitude of the model's
// log-probabilities: the inputs of the static FP64 exactness certificates (DESIGN.md)
void gmg_icm_value_stats(const gmg_icm* m, int* ulp_exp, float* max_abs);
// build the model's device views on first use (no-op afterwards); every scoring entry point calls it
int gmg_icm_ready(const gmg_icm* m);

struct gmg_seqset {
  gmg_ctx* ctx;
  int64_t n;                 // sequences
  int64_t total;             // bases
  int64_t max_len;           // longest sequence
  std::vector<int64_t> hdr_off, hdr_end;  // gmg_seqset_from_fasta: header text of record i = image[hdr_off[i], hdr_end[i])
  std::vector<int64_t> off;  // host copy, n+1
  int64_t* d_off;            // n+1
  uint64_t* d_words_base;    // allocation incl. padding
  uint64_t* d_words;         // 2-bit bases, base i at bits 2*(i%32) of word i/32
  int32_t* d_blk2seq;        // sequence holding base 32*b; bit 31 = interior block (see k_blk2seq)
  uint8_t* d_qual;           // per-base quality (input file values) or NULL
  unsigned long long* d_gc;  // {gc count, ORFs of the last g3 scoring call that took the ordered-sum fallback,
                             //  4 x bases per code (k_bucket_finish), non-acgt bytes counted by the pack}
  // every input byte that is not a / c / g / t in either case, position-sorted: (base index << 8) | tolower(byte).
  // The 2-bit pack keeps only Filter(byte); extraction needs the raw IUPAC code to complement it before Filter.
  uint64_t* d_nacgt;
  int64_t n_nacgt;
  // base buckets (k_bucket_*): the K1 planes are stored bucketed by the base at each position (see gmg_plane_index)
  uint32_t* d_bktidx;        // [nblk][4] plane index of the first base-b position at or after 32-base block blk
  // walk-ready contexts in plane-index order (model independent; K1 shifts them down by 32 - 2 W, W <= 14):
  uint32_t* d_ctxf;          // [total] forward strand: base p+j at bits 30-2j, j = 0..13; bits 0-3 min(len-1-q, 15)
  uint32_t* d_ctxr;          // [total] reverse strand: complement of base p-15+i at bits 2i, i = 2..15; bits 0-3 min(q, 15)
  int64_t n_base[4];         // positions with base a / c / g / t (host copy valid iff n_base_valid)
  int n_base_valid;
  // codon bitmaps (k_codon_bits): uint2 {start bits, stop bits} [strand][stream r][nwc]; bit i of word w <-> the
  // codon whose three bases start at global index 3 (32 w + i) + r
  uint2* d_cbits;
  int64_t nwc;
  unsigned long long cbits_key[4];  // the raw codon masks the bitmaps were built for
  // ORFs
  int64_t n_orfs;
  gmg_orf* d_orfs;
  int64_t* d_orf_off;        // n+1
  int32_t* d_orf_seq;        // sequence index of every ORF
  std::vector<int64_t> orf_off;
  // starts of the last scoring call
  int64_t n_starts;
  gmg_start* d_starts;
  int64_t* d_start_off;      // n_orfs+1
  int64_t uncertified;
  unsigned long long* uncert_pending;  // device counter still to be read into `uncertified` (fused plain path)
  int orfs_external;                   // ORF table came from gmg_set_orfs (not from the device finder)
  size_t cap_orfs, cap_starts;
  // reduced start lists of the last gmg_reduce_starts_mg call (they live in the context's SCR_RED scratch)
  int64_t n_red, n_red_fallback;
  gmg_start* d_red;
  int64_t* d_red_first;
  int32_t* d_red_cnt;
  uint8_t* d_red_status;
};

// scratch slots
enum { SCR_PLANES = 0, SCR_CUM = 1, SCR_TMP = 2, SCR_TMP2 = 3, SCR_FLAGS = 4, SCR_TMP3 = 5, SCR_QUAL = 6, SCR_TMP4 = 7,
       // flat glimmer-mg start enumeration (gmg_mg_flat.cuh): gates, root calls, per-level work arrays; reduction output
       SCR_MG_GATE = 8, SCR_MG_ROOT = 9, SCR_MG_L0 = 10, SCR_MG_CALL1 = 11, SCR_MG_L1 = 12, SCR_MG_L2 = 13, SCR_RED = 14,
       SCR_MISC = 15,
       // gmg_score_orfs_mg_gc: per-GC model records, the call's inputs (GC values, sequence -> record, ignore lengths),
       // the flagged-model list and the host's corrections
       SCR_INDEP = 16, SCR_INDEP_IN = 17, SCR_INDEP_AUX = 18, SCR_INDEP_FIX = 19,
       // plain glimmer-mg on read sets: the partial-window gene values of every sequence (k1_partial_side)
       SCR_SIDE = 20 };
int gmg_scratch(gmg_ctx* ctx, int slot, size_t bytes, void** out);
// ctx->h_stage holds at least `bytes` (grown to max(bytes, want)); its contents are not kept when it grows
int gmg_host_stage(gmg_ctx* ctx, size_t bytes, size_t want);

// ---- device helpers ---------------------------------------------------------------------

// bases [p0, p0+32) as one 64-bit value (base p0 at bits 0..1); p0 may be negative down to
// -32*GMG_PAD_WORDS and run past the end by the same amount (zero padding).
__device__ __forceinline__ uint64_t gmg_extract32(const uint64_t* __restrict__ words, int64_t p0) {
  int64_t w = p0 >> 5;  // arithmetic shift: floor
  int sh = (int)(p0 & 31) * 2;
  uint64_t lo = __ldg(words + w);
  if (sh == 0) return lo;
  uint64_t hi = __ldg(words + w + 1);
  return (lo >> sh) | (hi << (64 - sh));
}

__device__ __forceinline__ int gmg_base_at(const uint64_t* __restrict__ words, int64_t p) {
  return (int)((__ldg(words + (p >> 5)) >> ((p & 31) * 2)) & 3);
}

// One ICM walk (Full_Window_Prob icm.cc:557-610 / Partial_Window_Prob icm.cc:807-842 unified):
//  ctx   window bases: window position k at bits 2*k (k = 0 .. W-1; W-1 = predicted base)
//  lim   smallest window position whose base is available (0 = full window)
// mipf / probf already offset to the period's table.
__device__ __forceinline__ float gmg_walk(const int8_t* __restrict__ mipf, const float* __restrict__ probf,
                                          uint64_t ctx, int W, int D, int lim) {
  int node = 0;
  for (int i = 0; i < D; i++) {
    int pos = mipf[node];
    if (pos < lim) break;  // -1 leaf, -2 cut, or context base not available
    node = 4 * node + (int)((ctx >> (2 * pos)) & 3) + 1;
  }
  return __ldg(probf + 4 * (size_t)node + (int)((ctx >> (2 * (W - 1))) & 3));
}

// The six K1 planes (float [6][total]) are not stored in position order but bucketed by the base at each
// position: all 'a' positions first (ascending), then 'c', 'g', 't'.  K1's role-persistent CTAs each keep ONE
// (period, predicted base) leaf table in shared memory and stream through one bucket, reading and writing
// densely; every consumer maps a position to its plane index with one 16-byte load and a popcount:
//   index(p) = bktidx[p / 32][b] + #{ q in the same 32-base block, q < p, base(q) == b },  b = base(p).
// Consecutive positions of one base have consecutive indices, so a warp reading 32 consecutive positions touches
// four dense runs (the same number of 32-byte sectors as a position-ordered plane).
__device__ __forceinline__ uint32_t gmg_plane_index(const uint64_t* __restrict__ words,
                                                    const uint32_t* __restrict__ bktidx, int64_t p) {
  const uint64_t w = __ldg(words + (p >> 5));
  const int i = (int)(p & 31);
  const unsigned b = (unsigned)(w >> (2 * i)) & 3u;
  const uint64_t x = w ^ (0x5555555555555555ull * b);
  const uint64_t eq = ~(x | (x >> 1)) & 0x5555555555555555ull & ((1ull << (2 * i)) - 1ull);
  return __ldg(bktidx + ((p >> 5) << 2) + b) + (uint32_t)__popcll(eq);
}

// The walk-ready contexts of position p = 32 blk + i (the format of gmg_seqset::d_ctxf / d_ctxr) from the packed words of
// blocks blk - 1, blk, blk + 1 (zero padding either side of the batch); q / e = distance of p to the first / last base of
// its sequence.  k_bucket_finish stores them for K1, k1_partial_side forms them again for the partial windows of read sets.
__device__ __forceinline__ void gmg_window_ctx(uint64_t wm, uint64_t w, uint64_t wp, int i, int64_t q, int64_t e,
                                               uint32_t* cf, uint32_t* cr) {
  // forward: bases p .. p+15, order reversed (base p in the top pair)
  uint32_t f = (uint32_t)(i == 0 ? w : ((w >> (2 * i)) | (wp << (64 - 2 * i))));
  f = __brev(f);
  f = ((f >> 1) & 0x55555555u) | ((f & 0x55555555u) << 1);
  // reverse: complement of bases p-15 .. p (base p-15 in the low pair)
  const uint32_t r = ~(uint32_t)(i >= 15 ? (w >> (2 * (i - 15))) : ((wm >> (64 - 2 * (15 - i))) | (w << (2 * (15 - i)))));
  // the low four bits (the two bases farthest from p; windows of up to 14 bases never see them) hold the distance to the
  // end / start of the sequence, clipped to 15: which window positions exist
  *cf = (f & ~15u) | (uint32_t)(e < 15 ? e : 15);
  *cr = (r & ~15u) | (uint32_t)(q < 15 ? q : 15);
}

// reverse the order of the low W bases of v (base i <-> base W-1-i)
__device__ __forceinline__ uint64_t gmg_reverse_bases(uint64_t v, int W) {
  // reverse all 32 2-bit groups, then shift down
  v = ((v >> 2) & 0x3333333333333333ull) | ((v & 0x3333333333333333ull) << 2);
  v = ((v >> 4) & 0x0F0F0F0F0F0F0F0Full) | ((v & 0x0F0F0F0F0F0F0F0Full) << 4);
  v = ((v >> 8) & 0x00FF00FF00FF00FFull) | ((v & 0x00FF00FF00FF00FFull) << 8);
  v = ((v >> 16) & 0x0000FFFF0000FFFFull) | ((v & 0x0000FFFF0000FFFFull) << 16);
  v = (v >> 32) | (v << 32);
  return v >> (2 * (32 - W));
}

// ---- per-sequence independent models (gmg_score_orfs_mg_gc) ----------------------------------------------------
// Build_Indep_WO_Stops (icm.cc:65-216) on the host: mip [3][21], prob [3][21][4] of the ICM_t(3,2,3)
void gmg_indep_tables(double gc, const char* const* stops, int n_stops, int16_t* mip, float* prob);
// Subscript(Filter(ch)) (icm.cc:2008-2027)
int gmg_base_code(char ch);
// the entries of the device view's prob table ((period * N + node) * 4 + base) that the full-window table
// lut3 [384] and the partial-window table lutp [768] of a W == 3, P == 3 model take (icm_upload)
void gmg_w3_lut_index(const int16_t* mip, int N, int D, int* idx3, int* idxp);
// One record per GC value: the device view's prob [3][21][4], lut3 [384] and lutp [768] floats, in this order.  A kernel
// scores a sequence with its record by pointing a copy of the shared DevIcm (W, D, P, N, mip) at it.
#define GMG_INDEP_REC (252 + 384 + 768)
struct IndepSeqs {
  const float* rec;        // [n_models][GMG_INDEP_REC]
  const int32_t* model;    // [n_seq] record of every sequence
  const int32_t* isl;      // [n_seq] Ignore_Score_Len of every sequence
  const int32_t* orf_seq;  // [n_orfs] sequence of every ORF (for kernels that otherwise see only ORF descriptors)
};
// the n_models records for the GC values d_gc (device) / h_gc (host, the same values) with p's stop codons into the
// context's SCR_INDEP scratch; *base = the shared part of the device view
int gmg_indep_build(gmg_ctx* ctx, const double* d_gc, const double* h_gc, int64_t n_models, const gmg_params* p,
                    float** d_rec, DevIcm* base);

int gmg_seqset_ensure_buckets(gmg_ctx* ctx, gmg_seqset* s);
// kernel launchers implemented across the .cu files
int gmg_launch_pack(gmg_ctx* ctx, const uint8_t* d_ascii, int64_t total, uint64_t* d_words, unsigned long long* d_gc,
                    uint64_t* d_nacgt, int64_t cap_nacgt);
