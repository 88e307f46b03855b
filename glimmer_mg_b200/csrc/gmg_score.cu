// glimmer_mg_b200/csrc/gmg_score.cu -- the scoring kernels.
//
//   K1  k1_planes          per-position six-frame ICM tree walks            (Score_All_Frames glimmer-mg.cc:1468,
//                                                                            ICM_t::Frame_Score icm.cc:485)
//   K2  k2_prefix_lanes    per-(strand, reading-frame class) prefix sums of gene - indep log-odds, previous /
//                          next in-frame stop tables, 454 quality synthesis, FP64 exactness certificate (glimmer-mg
//                          -i / -s)                                         (Cumulative_Frame_Score glimmer-mg.cc:561,
//                                                                            Save_Prev_Stops :675, Set_Quality_454 :1865)
//       k2_g3_codon_cum    codon-boundary sums of the glimmer3 path
//   K3  k_mgf_*            per-ORF start enumeration incl. indel / substitution branches, level by level (flat form)
//       k3_mg_starts       the same with one thread per ORF         (Score_Orf_Starts :1693, Score_Indels :1513)
//       k3_mg_plain_lanes, k3_mg_plain
//                          K2 + K3 fused for plain glimmer-mg (no error branches)
//       k3_g3_count, k3_g3_heads, k3_g3_emit, k3_g3_ordered
//                          glimmer3's start enumeration                     (Score_Orfs glimmer3.cc:1275)
//   plus the device ORF finder (Find_Orfs glimmer_base.cc:638) and the scalar operator surface
//   (Score_String / Cumulative_Score / Frame_Score icm.cc:864/354/485).
//
// Data layout (all offsets are global base indices p = off[seq] + q, q = position in the sequence):
//   words   2-bit bases, 32 per 64-bit word
//   planes  float [6][total]   gene-ICM log-prob of base p under model period f (Frame_Score, icm.cc:485):
//              plane f   (forward strand): context = the W-1 bases to the RIGHT of q
//              plane 3+f (reverse strand): context = complement of the W-1 bases to the LEFT of q
//           position j of an ORF string uses period (1 + j) mod 3 (Cumulative_Score icm.cc:354); in terms of the
//           reading-frame class c of the K2 sums (forward ORFs with hi mod 3 == c, reverse ORFs with lo mod 3 == c)
//           a forward class-c sum takes period (c - q) mod 3 at position q, a reverse one (1 + q - c) mod 3.
//   cum     double [6][total]  forward planes: suffix sums  sum_{q' >= q} (gene - indep); reverse planes: prefix sums.
#include <float.h>
#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <cub/block/block_scan.cuh>
#include <cub/device/device_scan.cuh>

#include "gmg_internal.cuh"
#include "gmg_mg_flat.cuh"

// ------------------------------------------------------------------------------------------------
// small device helpers

__device__ __forceinline__ int mod3(int x) {
  int r = x % 3;
  return r < 0 ? r + 3 : r;
}

struct SeqView {
  int64_t a;  // global index of the first base
  int len;
};

__device__ __forceinline__ SeqView locate(const int64_t* __restrict__ off, const int32_t* __restrict__ blk2seq,
                                          int64_t p, int32_t* seq_out) {
  int32_t s = __ldg(blk2seq + (p >> 5)) & 0x7FFFFFFF;
  while (p >= __ldg(off + s + 1)) s++;
  SeqView v;
  v.a = __ldg(off + s);
  v.len = (int)(__ldg(off + s + 1) - v.a);
  *seq_out = s;
  return v;
}

// window register for the forward strand at global position p: window position k <-> base p + W-1-k
__device__ __forceinline__ uint64_t ctx_fwd(const uint64_t* __restrict__ words, int64_t p, int W) {
  return gmg_reverse_bases(gmg_extract32(words, p), W);
}
// reverse strand: window position k <-> complement of base p - (W-1) + k
__device__ __forceinline__ uint64_t ctx_rev(const uint64_t* __restrict__ words, int64_t p, int W) {
  return ~gmg_extract32(words, p - (W - 1));
}
// plain string order (Score_String etc.): window position k <-> base p - (W-1) + k
__device__ __forceinline__ uint64_t ctx_str(const uint64_t* __restrict__ words, int64_t p, int W) {
  return gmg_extract32(words, p - (W - 1));
}

__device__ __forceinline__ float icm_fwd(const DevIcm& m, const uint64_t* __restrict__ words, int64_t p, int q, int end,
                                         int f) {
  // `end` = exclusive end (in sequence coordinates) of the available context
  int lim = q + m.W - end;
  return gmg_walk(m.mip + (size_t)f * m.inner, m.prob + (size_t)f * m.N * 4, ctx_fwd(words, p, m.W), m.W, m.D,
                  lim > 0 ? lim : 0);
}
__device__ __forceinline__ float icm_rev(const DevIcm& m, const uint64_t* __restrict__ words, int64_t p, int q,
                                         int begin, int f) {
  int lim = m.W - 1 - (q - begin);
  return gmg_walk(m.mip + (size_t)f * m.inner, m.prob + (size_t)f * m.N * 4, ctx_rev(words, p, m.W), m.W, m.D,
                  lim > 0 ? lim : 0);
}
__device__ __forceinline__ float icm_str(const DevIcm& m, const uint64_t* __restrict__ words, int64_t p, int q, int f) {
  int lim = m.W - 1 - q;
  return gmg_walk(m.mip + (size_t)f * m.inner, m.prob + (size_t)f * m.N * 4, ctx_str(words, p, m.W), m.W, m.D,
                  lim > 0 ? lim : 0);
}

// gmg_score_orfs_mg_gc: the independent model of sequence s -- the shared view pointed at the sequence's record
__device__ __forceinline__ DevIcm indep_of(const DevIcm& base, const IndepSeqs& X, int64_t s) {
  DevIcm m = base;
  m.prob = X.rec + (size_t)__ldg(X.model + s) * GMG_INDEP_REC;
  m.lut3 = m.prob + 252;
  m.lutp = m.prob + 636;
  return m;
}

// 6-bit code (b0*16 + b1*4 + b2) of the forward-strand codon whose three bases start at global index g
__device__ __forceinline__ int codon6_at(const uint64_t* __restrict__ words, int64_t g) {
  const int raw = (int)(gmg_extract32(words, g) & 63);  // b(g) | b(g+1) << 2 | b(g+2) << 4
  return ((raw & 3) << 4) | (raw & 12) | (raw >> 4);
}
// forward codon whose 3' base is at sequence position q: S[q-2], S[q-1], S[q]
__device__ __forceinline__ int codon_fwd_ending_at(const uint64_t* __restrict__ words, int64_t a, int q) {
  return codon6_at(words, a + q - 2);
}
// reverse-strand codon occupying q, q+1, q+2 read 5'->3': c(q+2), c(q+1), c(q)
__device__ __forceinline__ int codon_rev_starting_at(const uint64_t* __restrict__ words, int64_t a, int q) {
  const int c = 63 - codon6_at(words, a + q);
  return ((c & 3) << 4) | (c & 12) | (c >> 4);
}

// Ch_Mask (Common/gene.cc:954-995): the set of bases an IUPAC letter stands for, bit b = base b (a c g t); 0 = none
static unsigned iupac_mask(char ch) {
  switch (ch | 0x20) {
    case 'a': return 0x1;
    case 'c': return 0x2;
    case 'g': return 0x4;
    case 't': return 0x8;
    case 'r': return 0x5;
    case 'y': return 0xA;
    case 's': return 0x6;
    case 'w': return 0x9;
    case 'm': return 0x3;
    case 'k': return 0xC;
    case 'b': return 0xE;
    case 'd': return 0xD;
    case 'h': return 0xB;
    case 'v': return 0x7;
    case 'n': return 0xF;
    default: return 0x0;
  }
}

// Start / stop codon PATTERNS (Codon_t masks, gene.cc:39-161: letters may be IUPAC ambiguity codes) as sets of concrete
// codons: a sequence codon (always a/c/g/t after Filter) matches pattern i iff each of its bases is in the pattern's
// letter set; `which` = the first matching start pattern (Codon_t::Can_Be's order).
static int make_codon_sets(const gmg_params* p, CodonSets* cs, DevParams* dp) {
  memset(cs, 0, sizeof *cs);
  GMG_CHECK(p->n_start >= 0 && p->n_start <= 8 && p->n_stop >= 0 && p->n_stop <= 8, "bad start/stop codon count");
  memset(cs->which, 0xFF, sizeof cs->which);
  for (int code = 0; code < 64; code++) {
    const unsigned b0 = 1u << (code >> 4), b1 = 1u << ((code >> 2) & 3), b2 = 1u << (code & 3);
    for (int i = 0; i < p->n_start; i++)
      if ((iupac_mask(p->start_codon[i][0]) & b0) && (iupac_mask(p->start_codon[i][1]) & b1) && (iupac_mask(p->start_codon[i][2]) & b2)) {
        if (!(cs->start_mask >> code & 1)) cs->which[code] = (unsigned char)i;
        cs->start_mask |= 1ull << code;
      }
    for (int i = 0; i < p->n_stop; i++)
      if ((iupac_mask(p->stop_codon[i][0]) & b0) && (iupac_mask(p->stop_codon[i][1]) & b1) && (iupac_mask(p->stop_codon[i][2]) & b2))
        cs->stop_mask |= 1ull << code;
  }
  for (int raw = 0; raw < 64; raw++) {
    const int b0 = raw & 3, b1 = (raw >> 2) & 3, b2 = raw >> 4;
    const int fc = b0 * 16 + b1 * 4 + b2, rc = (3 - b2) * 16 + (3 - b1) * 4 + (3 - b0);
    if (cs->start_mask >> fc & 1) cs->raw_mask[0] |= 1ull << raw;
    if (cs->stop_mask >> fc & 1) cs->raw_mask[1] |= 1ull << raw;
    if (cs->start_mask >> rc & 1) cs->raw_mask[2] |= 1ull << raw;
    if (cs->stop_mask >> rc & 1) cs->raw_mask[3] |= 1ull << raw;
  }
  GMG_CHECK(p->indel_max >= 0 && p->indel_max <= 2, "indel_max %d unsupported (0..2)", p->indel_max);
  // qualities live in a uint8 plane (file values clamped to 255): Clean_Quality_454's threshold + 1 must fit it, and a
  // gate test q <= threshold must not open for values the clamp brought down to 255
  GMG_CHECK(p->indel_quality_threshold <= 254, "indel_quality_threshold %d unsupported (at most 254)",
            p->indel_quality_threshold);
  dp->min_gene_len = p->min_gene_len;
  dp->allow_truncated = p->allow_truncated;
  dp->allow_indels = p->allow_indels;
  dp->allow_subs = p->allow_subs;
  dp->min_indel_orf_len = p->min_indel_orf_len;
  dp->indel_q_thresh = p->indel_quality_threshold;
  dp->indel_max = p->indel_max;
  dp->ignore_score_len = p->ignore_score_len;
  dp->have_quality_file = p->have_quality_file;
  dp->indel_suffix_thresh = p->indel_suffix_score_threshold;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// K1: per-position six-frame walks of the gene ICM.
//
// One thread per base, six independent walks per thread (ILP hides the dependent shared-memory
// lookups); the branch-position bytes of the descendable levels (P * (4^D-1)/3 bytes = 16 KB at the
// defaults) are staged in shared memory, the leaf probabilities are one 4-byte read-only gather per
// walk from the L2-resident table.  Stores are one full 128-byte line per warp and plane.

template <int NW>
__device__ __forceinline__ void walk_many(const int8_t* const* mipf, const float* const* probf, const uint64_t* ctx,
                                          const int* lim, int W, int D, float* out) {
  int node[NW];
  bool live[NW];
#pragma unroll
  for (int w = 0; w < NW; w++) {
    node[w] = 0;
    live[w] = true;
  }
  for (int i = 0; i < D; i++) {
    bool any = false;
#pragma unroll
    for (int w = 0; w < NW; w++) {
      int pos = live[w] ? (int)mipf[w][node[w]] : -1;
      live[w] = live[w] && (pos >= lim[w]);
      int b = (int)((ctx[w] >> (2 * (pos & 31))) & 3);
      node[w] = live[w] ? 4 * node[w] + b + 1 : node[w];
      any |= live[w];
    }
    if (!any) break;
  }
#pragma unroll
  for (int w = 0; w < NW; w++) out[w] = __ldg(probf[w] + 4 * (size_t)node[w] + (int)((ctx[w] >> (2 * (W - 1))) & 3));
}

__global__ void __launch_bounds__(256) k1_planes(DevIcm gene, const uint64_t* __restrict__ words,
                                                 const int64_t* __restrict__ off, const int32_t* __restrict__ blk2seq,
                                                 const uint32_t* __restrict__ bktidx, int64_t total,
                                                 float* __restrict__ planes) {
  extern __shared__ int8_t s_mip[];
  const int nmip = gene.P * gene.inner;
  for (int i = threadIdx.x; i < nmip; i += blockDim.x) s_mip[i] = gene.mip[i];
  __syncthreads();

  const int W = gene.W, D = gene.D;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += (int64_t)gridDim.x * blockDim.x) {
    int32_t s;
    SeqView sv = locate(off, blk2seq, p, &s);
    const int q = (int)(p - sv.a);
    uint64_t cf = ctx_fwd(words, p, W), cr = ctx_rev(words, p, W);
    int lf = q + W - sv.len;
    lf = lf > 0 ? lf : 0;
    int lr = W - 1 - q;
    lr = lr > 0 ? lr : 0;
    const int8_t* mipf[6];
    const float* probf[6];
    uint64_t ctx[6];
    int lim[6];
    float v[6];
#pragma unroll
    for (int f = 0; f < 3; f++) {
      mipf[f] = mipf[3 + f] = s_mip + f * gene.inner;
      probf[f] = probf[3 + f] = gene.prob + (size_t)f * gene.N * 4;
      ctx[f] = cf;
      ctx[3 + f] = cr;
      lim[f] = lf;
      lim[3 + f] = lr;
    }
    walk_many<6>(mipf, probf, ctx, lim, W, D, v);
    const size_t pi = gmg_plane_index(words, bktidx, p);
#pragma unroll
    for (int f = 0; f < 6; f++) planes[(size_t)f * total + pi] = v[f];
  }
}

// K1, bucketed form (the default for W <= 16, D <= 7): role-persistent CTAs.  The planes are stored bucketed by
// the base at each position (gmg_plane_index), so all positions whose PREDICTED base is pb -- the base itself on the
// forward strand, its complement on the reverse strand -- are one dense run of plane indices.  A CTA keeps the
// leaf probabilities of ONE (period f, predicted base pb) pair (N floats, 87 KB at depth 7) and the period's shift
// table (8 KB) in shared memory and streams through its share of that role's run: position list in (dense), window
// from the packed bases, D shared-memory byte lookups, one shared-memory float lookup, result out (dense).  No
// global gathers are left on the walk (measured, tools/gpu/ubench_leaf.cu: a warp-wide random 4-byte read costs
// 4 SM cycles from shared memory against 11 from an L1-resident and 28 from an L2-resident table).
// The 24 (f, pb, strand) segments are linearised; CTA c takes the c-th equal share of the 6 * total walks, which
// spans at most two roles unless the batch is tiny.
#define K1_PAD GMG_CTX_PAD  // entries of padding after the context arrays (gmg_internal.cuh)
struct K1Segs {
  long long lo[25];        // linearised start of segment (f * 4 + pb) * 2 + strand; lo[24] = 6 * total
  unsigned bucket_lo[4];   // plane index of the first position of each base bucket
};

// two tree levels from one merged word (DevIcmFast::mw): i = index of the node within its (odd) level on entry, of
// its grandchild on exit.  No stop test: the tables describe the completed tree.
__device__ __forceinline__ uint32_t k1_step2(uint32_t w, uint32_t c, uint32_t i) {
  const uint32_t y1 = c << (w & 31);
  const uint32_t t = w >> (5 * (y1 >> 30) + 5);
  const uint32_t y2 = c << (t & 31);
  return __funnelshift_l(y2, __funnelshift_l(y1, i, 2), 2);
}

// the same two levels for a window whose positions below `lim` are not available (lsh = 30 - 2 lim): stops at the
// first node that is a real stop or branches on an unavailable position and returns true with *res = that node's
// dense number (off = dense number of the first node of the entry level, 4 off + 1 of the next).
__device__ __forceinline__ bool k1_step2_tested(uint32_t w, uint32_t c, unsigned lsh, uint32_t off, uint32_t* i,
                                                uint32_t* res) {
  const uint32_t s1 = w & 31;
  if (((w >> 25) & 1u) || s1 > lsh) {
    *res = off + *i;
    return true;
  }
  const uint32_t y1 = c << s1, b1 = y1 >> 30;
  const uint32_t i2 = __funnelshift_l(y1, *i, 2);
  const uint32_t s2 = (w >> (5 * b1 + 5)) & 31;
  if (((w >> (26 + b1)) & 1u) || s2 > lsh) {
    *res = 4 * off + 1 + i2;
    return true;
  }
  *i = __funnelshift_l(c << s2, i2, 2);
  return false;
}

// Partial windows, separately: the W-1 first positions of a sequence have a partial reverse-strand window and the W-1
// last ones a partial forward window (icm.cc:807-842).  In bucket order nearly every warp of the bucketed kernel would
// meet one and fall to its tested path, so for read sets that kernel walks EVERY window as if it were full and one of the
// two kernels below then walks the 2 (W-1) x 3 partial entries of every sequence again.  Their walks (one per period) go
// through the same merged words as the main kernel -- read from global memory, 13 KB that stay in L1 -- and stop at the
// first node that branches on an unavailable position.
//
// The gene value of period f of the walk-ready context c (d_ctxf / d_ctxr format) whose predicted base is pb.
__device__ __forceinline__ float k1_partial_walk(const DevIcmFast& gm, uint32_t c, unsigned pb, int f) {
  constexpr int NWORDS = 4 + 64 + 1024;
  constexpr uint32_t OFF7 = (16384 - 1) / 3;
  const int W = gm.W;
  const int lim = max(W - 1 - (int)(c & 15u), 0);  // first available window position
  const unsigned lsh = 30 - 2 * lim;               // a node may be descended iff its shift <= this
  const uint32_t cw = c >> (32 - 2 * W);
  const uint32_t* __restrict__ mw = gm.mw + (size_t)f * NWORDS;
  const unsigned s0 = f == 0 ? gm.s0[0] : (f == 1 ? gm.s0[1] : gm.s0[2]);
  const bool stop0 = (f == 0 ? gm.stop0[0] : (f == 1 ? gm.stop0[1] : gm.stop0[2])) != 0;
  uint32_t res = 0;
  if (!(stop0 || s0 > lsh)) {
    uint32_t i = (cw << s0) >> 30;
    if (!k1_step2_tested(__ldg(mw + i), cw, lsh, 1, &i, &res))
      if (!k1_step2_tested(__ldg(mw + 4 + i), cw, lsh, 21, &i, &res))
        if (!k1_step2_tested(__ldg(mw + 68 + i), cw, lsh, 341, &i, &res)) res = OFF7 + i;
  }
  return __ldg(gm.bleaf + (size_t)(f * 4 + (int)pb) * gm.np + res);
}

// In place, for every consumer of complete planes: one thread per (sequence, end, offset), the entry's context read back
// from the context array, the three values stored into the planes at the position's plane index.
__global__ void __launch_bounds__(256) k1_partial_fix(DevIcmFast gm, const uint64_t* __restrict__ words,
                                                      const int64_t* __restrict__ off, int64_t n_seq,
                                                      const uint32_t* __restrict__ bktidx,
                                                      const uint32_t* __restrict__ ctxf, const uint32_t* __restrict__ ctxr,
                                                      int64_t total, float* __restrict__ planes) {
  const int W = gm.W, per = 2 * (W - 1);
  const int64_t items = n_seq * per;
  for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < items; it += (int64_t)gridDim.x * blockDim.x) {
    const int64_t sq = it / per;
    const int k = (int)(it - sq * per);
    const int64_t a = __ldg(off + sq);
    const int L = (int)(__ldg(off + sq + 1) - a);
    const bool tail = k >= W - 1;  // forward-strand partial windows at the end of the sequence
    const int q = tail ? L - 1 - (k - (W - 1)) : k;
    if (q < 0 || q >= L) continue;
    // the strand whose window is partial at this end; the other strand's entry is a full window and already right
    // (unless the sequence is so short that it is partial too: then the item of the other end rewrites it)
    const bool rev = !tail;
    const int64_t p = a + q;
    const uint32_t pi = gmg_plane_index(words, bktidx, p);
    const uint32_t c = __ldg((rev ? ctxr : ctxf) + pi);
    if ((int)(c & 15u) >= W - 1) continue;  // a full window after all
    const unsigned own = (unsigned)gmg_base_at(words, p), pb = rev ? 3u - own : own;
#pragma unroll
    for (int f = 0; f < 3; f++) planes[(size_t)(rev ? 3 + f : f) * total + pi] = k1_partial_walk(gm, c, pb, f);
  }
}

// Into a dense table, for the plain glimmer-mg pass (the only consumer on its path, see mgp_gene): side[sq][k][f] for
// k < W-1 the reverse-strand value at q = k, for k >= W-1 the forward-strand value at q = L-1-(k-(W-1)); every entry
// whose position exists is written.  One thread per (sequence, end, offset) as above, but the context is formed from the
// sequence's packed words (consecutive threads read the same few words) and the bounds it already holds, and the stores
// are dense: no bucket-index or context gather and no read-modify-write of plane sectors that have left L2.
__global__ void __launch_bounds__(256) k1_partial_side(DevIcmFast gm, const uint64_t* __restrict__ words,
                                                       const int64_t* __restrict__ off, int64_t n_seq,
                                                       float* __restrict__ side) {
  const int W = gm.W, per = 2 * (W - 1);
  const int64_t items = n_seq * per;
  for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < items; it += (int64_t)gridDim.x * blockDim.x) {
    const int64_t sq = it / per;
    const int k = (int)(it - sq * per);
    const int64_t a = __ldg(off + sq);
    const int L = (int)(__ldg(off + sq + 1) - a);
    const bool rev = k < W - 1;
    const int q = rev ? k : L - 1 - (k - (W - 1));
    if (q < 0 || q >= L) continue;
    const int64_t p = a + q, blk = p >> 5;
    const uint64_t w = __ldg(words + blk);
    uint32_t cf, cr;
    gmg_window_ctx(__ldg(words + blk - 1), w, __ldg(words + blk + 1), (int)(p & 31), q, L - 1 - q, &cf, &cr);
    const unsigned own = (unsigned)(w >> (2 * (p & 31))) & 3u, pb = rev ? 3u - own : own;
#pragma unroll
    for (int f = 0; f < 3; f++) side[it * 3 + f] = k1_partial_walk(gm, rev ? cr : cf, pb, f);
  }
}

// kAllFull: the main loop walks EVERY window as a full one (no test, no slow path); k1_partial_fix or k1_partial_side
// then walks the entries whose window is partial.  (Tried and measured slower, 0.85 against 0.62 ms per 31 Mbp of 100 bp
// reads: a second phase inside this kernel that scans a bitmap of the partial plane indices and walks them from the
// shared-memory tables -- with 24 warps per SM its dependent bitmap -> context loads are pure latency, and the extra
// registers slow the main loop.)
template <int kU, int NT = 1024, bool kAllFull = false>
__global__ void __launch_bounds__(NT, 2) k1_planes_bucketed(DevIcmFast gm, const uint32_t* __restrict__ ctxf,
                                                              const uint32_t* __restrict__ ctxr, unsigned total,
                                                              K1Segs segs, float* __restrict__ planes) {
  extern __shared__ __align__(16) uint8_t s_raw[];
  constexpr int NWORDS = 4 + 64 + 1024;      // merged words of one period (levels 1, 3, 5)
  constexpr uint32_t OFF7 = (16384 - 1) / 3;  // dense number of the first level-7 node
  uint32_t* s_mw = reinterpret_cast<uint32_t*>(s_raw);
  float* s_leaf = reinterpret_cast<float*>(s_raw + NWORDS * 4);
  const int W = gm.W, nt = NT, np = gm.np;
  const int wsh = 32 - 2 * W;
  const long long all = segs.lo[24];
  const long long w0 = all * blockIdx.x / gridDim.x, w1 = all * (blockIdx.x + 1) / gridDim.x;
  int seg = 0;
  while (segs.lo[seg + 1] <= w0 && seg < 23) seg++;
  int have_f = -1, have_role = -1;
  for (; seg < 24 && segs.lo[seg] < w1; seg++) {
    const long long a0 = max(w0, segs.lo[seg]), a1 = min(w1, segs.lo[seg + 1]);
    if (a1 <= a0) continue;
    const int role = seg >> 1, f = role >> 2, pb = role & 3, rev = seg & 1;
    if (role != have_role) {  // CTA-uniform
      __syncthreads();
      if (f != have_f) {
        const uint4* src = reinterpret_cast<const uint4*>(gm.mw + (size_t)f * NWORDS);
        uint4* dst = reinterpret_cast<uint4*>(s_mw);
        for (int i = threadIdx.x; i < NWORDS / 4; i += nt) dst[i] = __ldg(src + i);
      }
      {
        const uint4* src = reinterpret_cast<const uint4*>(gm.bleaf + (size_t)role * np);
        uint4* dst = reinterpret_cast<uint4*>(s_leaf);
        for (int i = threadIdx.x; i < (np >> 2); i += nt) dst[i] = __ldg(src + i);
      }
      __syncthreads();
      have_f = f;
      have_role = role;
    }
    const unsigned s0 = f == 0 ? gm.s0[0] : (f == 1 ? gm.s0[1] : gm.s0[2]);
    const bool stop0 = (f == 0 ? gm.stop0[0] : (f == 1 ? gm.stop0[1] : gm.stop0[2])) != 0;
    const unsigned own = rev ? 3 - pb : pb;
    // plane indices [g0, g0 + n) of this share; the strand's contexts and its period-f plane, both offset to g0
    const unsigned g0 = segs.bucket_lo[own] + (unsigned)(a0 - segs.lo[seg]);
    const unsigned n = (unsigned)(a1 - a0);
    const uint32_t* __restrict__ cx = (rev ? ctxr : ctxf) + g0;
    float* __restrict__ out = planes + (size_t)(rev ? 3 + f : f) * total + g0;
    // every thread runs the same number of trips (the body votes).  Lanes past the end of the share walk whatever
    // context lies there (the arrays are padded by K1_PAD entries) and simply do not store.
    const unsigned trips = (n + kU * NT - 1) / (kU * NT);
    unsigned i0 = threadIdx.x;
    const uint32_t* __restrict__ pc = cx + i0;
    float* __restrict__ po = out + i0;
    uint32_t nc[kU];  // software pipeline: the contexts of the next trip are in flight while this one walks
#pragma unroll
    for (int u = 0; u < kU; u++) nc[u] = __ldg(pc + NT * u);
    for (unsigned t = 0; t < trips; t++, i0 += kU * NT, po += kU * NT) {
      uint32_t c[kU];
      bool partial = false;
      pc += kU * NT;
#pragma unroll
      for (int u = 0; u < kU; u++) {
        c[u] = nc[u];
        if (!kAllFull) partial |= (int)(c[u] & 15u) < W - 1;  // some window position does not exist
        nc[u] = __ldg(pc + NT * u);
      }
      uint32_t idx[kU];
      if (!__any_sync(0xffffffffu, partial || stop0)) {
        uint32_t i[kU], w[kU];
#pragma unroll
        for (int u = 0; u < kU; u++) {
          c[u] >>= wsh;  // window position k at bits 2k
          i[u] = (c[u] << s0) >> 30;
        }
#pragma unroll
        for (int u = 0; u < kU; u++) w[u] = s_mw[i[u]];
#pragma unroll
        for (int u = 0; u < kU; u++) i[u] = k1_step2(w[u], c[u], i[u]);
#pragma unroll
        for (int u = 0; u < kU; u++) w[u] = s_mw[4 + i[u]];
#pragma unroll
        for (int u = 0; u < kU; u++) i[u] = k1_step2(w[u], c[u], i[u]);
#pragma unroll
        for (int u = 0; u < kU; u++) w[u] = s_mw[68 + i[u]];
#pragma unroll
        for (int u = 0; u < kU; u++) idx[u] = OFF7 + k1_step2(w[u], c[u], i[u]);
      } else {
#pragma unroll
        for (int u = 0; u < kU; u++) {
          const int lim = max(W - 1 - (int)(c[u] & 15u), 0);  // first available window position
          const unsigned lsh = 30 - 2 * lim;                   // a node may be descended iff its shift <= this
          const uint32_t cw = c[u] >> wsh;
          uint32_t res = 0;
          if (!(stop0 || s0 > lsh)) {
            uint32_t i = (cw << s0) >> 30;
            if (!k1_step2_tested(s_mw[i], cw, lsh, 1, &i, &res))
              if (!k1_step2_tested(s_mw[4 + i], cw, lsh, 21, &i, &res))
                if (!k1_step2_tested(s_mw[68 + i], cw, lsh, 341, &i, &res)) res = OFF7 + i;
          }
          idx[u] = res;
        }
      }
#pragma unroll
      for (int u = 0; u < kU; u++) {
        const float v = s_leaf[idx[u]];
        // predicated store (no branch): only entries of this share
        asm volatile("{ .reg .pred p; setp.lt.u32 p, %0, %1; @p st.global.f32 [%2], %3; }" ::"r"(i0 + NT * u), "r"(n),
                     "l"(po + NT * u), "f"(v)
                     : "memory");
      }
    }
  }
}

// side_out: NULL -- the planes come out complete; else the caller reads partial-window values from *side_out where it is
// not NULL (k1_partial_side's table, in the context's SCR_SIDE scratch) and the planes hold full-window walks there.
static int launch_k1(gmg_ctx* ctx, const gmg_icm* gene, gmg_seqset* s, float** planes_out, float** side_out) {
  GMG_CHECK(gene->P == 3, "six-frame scoring needs a periodicity-3 gene model (got %d)", gene->P);
  if (gmg_icm_ready(gene)) return 1;
  if (gmg_seqset_ensure_buckets(ctx, s)) return 1;
  void* planes = NULL;
  if (gmg_scratch(ctx, SCR_PLANES, (size_t)6 * (s->total + 32) * sizeof(float), &planes)) return 1;
  *planes_out = (float*)planes;
  if (side_out) *side_out = NULL;
  if (s->total == 0) return 0;
  if (gene->fast.valid && gene->W <= 14) {
    if (!s->n_base_valid) {
      unsigned long long nb[4];
      GMG_CUDA(cudaMemcpyAsync(nb, s->d_gc + 2, sizeof nb, cudaMemcpyDeviceToHost, ctx->stream));
      GMG_CUDA(cudaStreamSynchronize(ctx->stream));
      for (int b = 0; b < 4; b++) s->n_base[b] = (int64_t)nb[b];
      s->n_base_valid = 1;
    }
    K1Segs segs;
    long long acc = 0;
    for (int f = 0; f < 3; f++)
      for (int pb = 0; pb < 4; pb++)
        for (int rev = 0; rev < 2; rev++) {
          segs.lo[(f * 4 + pb) * 2 + rev] = acc;
          acc += s->n_base[rev ? 3 - pb : pb];
        }
    segs.lo[24] = acc;
    unsigned bl = 0;
    for (int b = 0; b < 4; b++) {
      segs.bucket_lo[b] = bl;
      bl += (unsigned)s->n_base[b];
    }
    const size_t smem = (size_t)(4 + 64 + 1024) * 4 + (size_t)gene->fast.np * sizeof(float);
    // Six walks in flight per thread, 384 threads per CTA: the six hide the shared-memory latency with a third of the
    // warps and pay the loop overhead once per six walks, and the 768 threads per SM leave room for the side-stream
    // kernels of gmg_score_orfs_g3 to run beside K1 (the other shapes measured took as long or longer, DESIGN.md 3.1).
    // Read sets walk every window as full (no partial-window test in the hot loop) and a second kernel walks the
    // 2 (W-1) x 3 partial entries of every sequence: into a dense table for a caller that takes one (k1_partial_side), in
    // place otherwise (k1_partial_fix).  On long sequences the test costs less than that second launch (5 Mbp contig: 71.6
    // against 78.9 us), so they keep the tested loop.  GMG_K1_FIX=0 (test hook): read sets too.
    const bool long_seqs = s->total / (s->n > 0 ? s->n : 1) >= 4096;
    const char* fix_env = getenv("GMG_K1_FIX");
    const bool fix = !long_seqs && !(fix_env && atoi(fix_env) == 0);
    long long need = (acc + 4095) / 4096;
    long long cap = (long long)ctx->sm_count * 2;
    int grid = (int)(need < cap ? need : cap);
    if (gmg_prof_begin(ctx, GMG_PROF_K1)) return 1;
    const auto k1 = fix ? k1_planes_bucketed<6, 384, true> : k1_planes_bucketed<6, 384, false>;
    GMG_CUDA(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k1<<<grid, 384, smem, ctx->stream>>>(gene->fast, s->d_ctxf, s->d_ctxr, (unsigned)s->total, segs, (float*)planes);
    if (fix) {
      const int64_t items = s->n * 2 * (gene->W - 1);
      int64_t fg = (items + 255) / 256, fcap = (int64_t)ctx->sm_count * 16;
      const unsigned fgrid = (unsigned)(fg < fcap ? fg : fcap);
      if (side_out) {
        void* side = NULL;
        if (gmg_scratch(ctx, SCR_SIDE, (size_t)items * 3 * sizeof(float), &side)) return 1;
        *side_out = (float*)side;
        k1_partial_side<<<fgrid, 256, 0, ctx->stream>>>(gene->fast, s->d_words, s->d_off, s->n, (float*)side);
      } else {
        k1_partial_fix<<<fgrid, 256, 0, ctx->stream>>>(gene->fast, s->d_words, s->d_off, s->n, s->d_bktidx, s->d_ctxf,
                                                       s->d_ctxr, s->total, (float*)planes);
      }
      ctx->launches++;
    }
    gmg_prof_end(ctx, GMG_PROF_K1);
    ctx->launches++;
    GMG_CUDA(cudaGetLastError());
    return 0;
  }
  size_t smem = (size_t)gene->dev.P * gene->dev.inner;
  GMG_CHECK(smem <= 200 * 1024, "gene model too deep for the shared-memory walk table (%zu bytes)", smem);
  if (smem > 48 * 1024)
    GMG_CUDA(cudaFuncSetAttribute(k1_planes, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int64_t need = (s->total + 255) / 256;
  int64_t cap = (int64_t)ctx->sm_count * 8;
  int grid = (int)(need < cap ? need : cap);
  if (gmg_prof_begin(ctx, GMG_PROF_K1)) return 1;
  k1_planes<<<grid, 256, smem, ctx->stream>>>(gene->dev, s->d_words, s->d_off, s->d_blk2seq, s->d_bktidx, s->total,
                                              (float*)planes);
  gmg_prof_end(ctx, GMG_PROF_K1);
  ctx->launches++;
  GMG_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int gmg_k1_score_planes(gmg_ctx* ctx, const gmg_icm* gene, gmg_seqset* s) {
  GMG_CHECK(ctx && gene && s, "gmg_k1_score_planes: NULL argument");
  float* planes;
  return launch_k1(ctx, gene, s, &planes, NULL);
}

// ------------------------------------------------------------------------------------------------
// Frame_Scores surface (Score_All_Frames): FS[f][q] = gene - indep as doubles, reference layout.

__global__ void __launch_bounds__(256) k_frame_scores(DevIcm indep, const uint64_t* __restrict__ words,
                                                      const int64_t* __restrict__ off,
                                                      const int32_t* __restrict__ blk2seq,
                                                      const uint32_t* __restrict__ bktidx, int64_t total,
                                                      const float* __restrict__ planes, double* __restrict__ fs) {
  int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= total) return;
  const size_t pi = gmg_plane_index(words, bktidx, p);
  int32_t s;
  SeqView sv = locate(off, blk2seq, p, &s);
  const int q = (int)(p - sv.a);
  double* row = fs + 6 * sv.a;
  for (int f = 0; f < 3; f++) {
    float g = planes[(size_t)f * total + pi];
    float n = icm_fwd(indep, words, p, q, sv.len, f);
    row[(size_t)f * sv.len + q] = (double)g - (double)n;
    g = planes[(size_t)(3 + f) * total + pi];
    n = icm_rev(indep, words, p, q, 0, f);
    row[(size_t)(3 + f) * sv.len + q] = (double)g - (double)n;
  }
}

extern "C" int gmg_score_all_frames(gmg_ctx* ctx, const gmg_icm* gene, const gmg_icm* indep, gmg_seqset* s,
                                    double* out, int out_on_device) {
  GMG_CHECK(ctx && gene && indep && s && out, "gmg_score_all_frames: NULL argument");
  GMG_CHECK(indep->P == 3, "independent model must have periodicity 3");
  if (gmg_icm_ready(indep)) return 1;
  float* planes;
  if (launch_k1(ctx, gene, s, &planes, NULL)) return 1;
  if (s->total == 0) return 0;
  double* d_fs = out;
  if (!out_on_device) {
    void* tmp;
    if (gmg_scratch(ctx, SCR_CUM, (size_t)6 * s->total * sizeof(double), &tmp)) return 1;
    d_fs = (double*)tmp;
  }
  if (gmg_prof_begin(ctx, GMG_PROF_FS)) return 1;
  k_frame_scores<<<(unsigned)((s->total + 255) / 256), 256, 0, ctx->stream>>>(indep->dev, s->d_words, s->d_off,
                                                                             s->d_blk2seq, s->d_bktidx, s->total, planes,
                                                                             d_fs);
  gmg_prof_end(ctx, GMG_PROF_FS);
  ctx->launches++;
  GMG_CUDA(cudaGetLastError());
  if (!out_on_device) {
    GMG_CUDA(cudaMemcpyAsync(out, d_fs, (size_t)6 * s->total * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Scalar operator surface: Score_String / Cumulative_Score / Frame_Score.
// One warp per string; lanes evaluate 32 consecutive positions, lane order is preserved when the
// FP64 sum is accumulated so the result has the reference's serial rounding (icm.cc:886-900).

// mode 0: Score_String (one double per string), 1: Cumulative_Score, 2: Frame_Score
__global__ void __launch_bounds__(128) k_string_scores(DevIcm m, const uint64_t* __restrict__ words,
                                                       const int64_t* __restrict__ off, int64_t n, int frame0,
                                                       int mode, double* __restrict__ out) {
  int64_t s = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= n) return;
  const int64_t a = off[s];
  const int len = (int)(off[s + 1] - a);
  if (m.P == 1) frame0 = 0;
  double total = 0.0;
  for (int base = 0; base < len; base += 32) {
    int q = base + lane;
    double x = 0.0;
    if (q < len) {
      int f = (mode == 2) ? frame0 : (frame0 + q) % m.P;
      x = (double)icm_str(m, words, a + q, q, f);
      if (mode == 2) out[a + q] = x;
    }
    if (mode != 2) {
      // ordered accumulation: position base+0, base+1, ... exactly like the serial loop
      double run = total;
      double mine = 0.0;
      int cnt = min(32, len - base);
      for (int l = 0; l < cnt; l++) {
        double xl = __shfl_sync(0xffffffffu, x, l);
        run += xl;
        if (l == lane) mine = run;
      }
      total = run;
      if (mode == 1 && q < len) out[a + q] = mine;
    }
  }
  if (mode == 0 && lane == 0) out[s] = total;
}

static int string_scores(gmg_ctx* ctx, const gmg_icm* m, gmg_seqset* s, int frame, int mode, double* h_out) {
  GMG_CHECK(ctx && m && s && h_out, "string score: NULL argument");
  GMG_CHECK(frame >= 0 && (frame < m->P || m->P == 1), "frame %d out of range for periodicity %d", frame, m->P);
  if (gmg_icm_ready(m)) return 1;
  if (s->n == 0) return 0;
  size_t n_out = (mode == 0) ? (size_t)s->n : (size_t)s->total;
  if (n_out == 0) return 0;
  void* d_out;
  if (gmg_scratch(ctx, SCR_CUM, n_out * sizeof(double), &d_out)) return 1;
  int64_t threads = s->n * 32;
  k_string_scores<<<(unsigned)((threads + 127) / 128), 128, 0, ctx->stream>>>(m->dev, s->d_words, s->d_off, s->n, frame,
                                                                             mode, (double*)d_out);
  ctx->launches++;
  GMG_CUDA(cudaGetLastError());
  GMG_CUDA(cudaMemcpyAsync(h_out, d_out, n_out * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Many-model read scoring (SURVEY.md section 8(f) row 4: the `simple-score` step of the Phymm / Scimm
// classification that precedes glimmer-mg, scripts/scoreReadsGlim.pl:450,482 -- Score_String of every read
// against every ICM).  gridDim.y = model: a CTA stages its model's branch-position table (int8, levels
// 0..D-1) in shared memory and gathers leaf probabilities from the L2-resident table; one warp per read, lanes
// stride the positions and sum in FP64.  Summation order is free whenever the read's certificate holds (every term an
// integer multiple of 2^g, g from the smallest float exponent the read meets, and sum|term| < 2^(g+52): no addition
// can round); the kernel flags the (model, read) pairs where it does not and k_score_many_redo repeats just those in
// the reference's serial order.
__global__ void __launch_bounds__(256) k_score_many(const DevIcm* __restrict__ models, const int* __restrict__ slot,
                                                    const uint64_t* __restrict__ words, const int64_t* __restrict__ off,
                                                    int64_t n, int frame0, double* __restrict__ out,
                                                    uint8_t* __restrict__ redo, int force_redo) {
  extern __shared__ int8_t s_mipm[];
  const DevIcm m = models[slot[blockIdx.y]];
  const int nmip = m.P * m.inner;
  for (int i = threadIdx.x; i < nmip; i += blockDim.x) s_mipm[i] = m.mip[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int fr0 = m.P == 1 ? 0 : frame0;
  double* row = out + (size_t)slot[blockIdx.y] * n;
  uint8_t* flag = redo + (size_t)slot[blockIdx.y] * n;
  for (int64_t s = (int64_t)blockIdx.x * nw + wid; s < n; s += (int64_t)gridDim.x * nw) {
    const int64_t a = off[s];
    const int len = (int)(off[s + 1] - a);
    double sum = 0.0;
    unsigned umin = 0x7fffffffu;  // certificate inputs, as in K2: smallest magnitude bits, sum of magnitudes
    double asum = 0.0;            // FP64: a float sum of len / 32 terms would eat the margin on long sequences
    for (int q = lane; q < len; q += 32) {
      const int f = m.P == 1 ? 0 : (fr0 + q) % m.P;
      const int lim = m.W - 1 - q;
      const float v = gmg_walk(s_mipm + (size_t)f * m.inner, m.prob + (size_t)f * m.N * 4, ctx_str(words, a + q, m.W), m.W,
                               m.D, lim > 0 ? lim : 0);
      sum += (double)v;
      const unsigned u = __float_as_uint(v) & 0x7fffffffu;
      umin = min(umin, u ? u : 0x7fffffffu);
      asum += (double)fabsf(v);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      sum += __shfl_xor_sync(0xffffffffu, sum, d);
      umin = min(umin, __shfl_xor_sync(0xffffffffu, umin, d));
      asum += __shfl_xor_sync(0xffffffffu, asum, d);
    }
    if (lane == 0) {
      // every term is a multiple of 2^g and every partial sum of ANY order is bounded by the sum of magnitudes:
      // below 2^(g+52) no addition can round and this sum has the bits of the reference's serial one
      const int e = (int)(umin >> 23);
      const int g = (e > 0 ? e : 1) - 150;
      const bool exact = umin == 0x7fffffffu || asum * 1.001 < ldexp(1.0, g + 52);
      row[s] = sum;
      flag[s] = (exact && !force_redo) ? 0 : 1;
    }
  }
}

// the (model, read) pairs whose certificate failed, again in the reference's serial order (icm.cc:886-900)
__global__ void __launch_bounds__(128) k_score_many_redo(const DevIcm* __restrict__ models, const int* __restrict__ slot,
                                                         int n_slots, const uint64_t* __restrict__ words,
                                                         const int64_t* __restrict__ off, int64_t n, int frame0,
                                                         double* __restrict__ out, const uint8_t* __restrict__ redo) {
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= (int64_t)n_slots * n) return;
  const int k = slot[w / n];
  const int64_t s = w % n;
  if (!redo[(size_t)k * n + s]) return;
  const DevIcm m = models[k];
  const int64_t a = off[s];
  const int len = (int)(off[s + 1] - a);
  const int fr0 = m.P == 1 ? 0 : frame0;
  double total = 0.0;
  for (int base = 0; base < len; base += 32) {
    const int q = base + lane;
    double x = 0.0;
    if (q < len) x = (double)icm_str(m, words, a + q, q, (fr0 + q) % m.P);
    const int cnt = min(32, len - base);
    for (int l = 0; l < cnt; l++) total += __shfl_sync(0xffffffffu, x, l);
  }
  if (lane == 0) out[(size_t)k * n + s] = total;
}

extern "C" int gmg_icm_score_strings_many(gmg_ctx* ctx, const gmg_icm* const* models, int n_models, gmg_seqset* s,
                                          int frame, double* h_out) {
  GMG_CHECK(ctx && models && s && h_out && n_models >= 0, "gmg_icm_score_strings_many: bad argument");
  if (n_models == 0 || s->n == 0) return 0;
  std::vector<DevIcm> dev((size_t)n_models);
  std::vector<int> fast_slots, ordered_slots;
  size_t smem = 0;
  for (int k = 0; k < n_models; k++) {
    const gmg_icm* m = models[k];
    GMG_CHECK(m != NULL, "gmg_icm_score_strings_many: model %d is NULL", k);
    if (gmg_icm_ready(m)) return 1;
    GMG_CHECK(frame >= 0 && (frame < m->P || m->P == 1), "frame %d out of range for periodicity %d (model %d)", frame, m->P, k);
    dev[(size_t)k] = m->dev;
    const size_t need = (size_t)m->dev.P * m->dev.inner;
    if (need <= 64 * 1024) {  // branch table fits in shared memory; exactness is certified per read in the kernel
      fast_slots.push_back(k);
      if (need > smem) smem = need;
    } else {
      ordered_slots.push_back(k);
    }
  }
  void *d_out, *d_models, *d_redo;
  if (gmg_scratch(ctx, SCR_CUM, (size_t)n_models * s->n * sizeof(double), &d_out)) return 1;
  if (!fast_slots.empty()) {
    const size_t mb = (size_t)n_models * sizeof(DevIcm), sb = fast_slots.size() * sizeof(int);
    if (gmg_scratch(ctx, SCR_TMP3, mb + sb + 64, &d_models)) return 1;
    if (gmg_scratch(ctx, SCR_TMP2, (size_t)n_models * s->n + 64, &d_redo)) return 1;
    int* d_slot = (int*)((char*)d_models + ((mb + 15) & ~(size_t)15));
    GMG_CUDA(cudaMemcpyAsync(d_models, dev.data(), mb, cudaMemcpyHostToDevice, ctx->stream));
    GMG_CUDA(cudaMemcpyAsync(d_slot, fast_slots.data(), sb, cudaMemcpyHostToDevice, ctx->stream));
    if (smem > 48 * 1024)
      GMG_CUDA(cudaFuncSetAttribute(k_score_many, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t need_ctas = (s->n + 7) / 8;
    int64_t gx = (int64_t)ctx->sm_count * 8 / (int64_t)fast_slots.size() + 1;
    if (gx > need_ctas) gx = need_ctas;
    if (gx < 1) gx = 1;
    dim3 grid((unsigned)gx, (unsigned)fast_slots.size());
    const char* env_redo = getenv("GMG_MANY_FORCE_REDO");  // test hook: every pair through the serial-order kernel
    const int force_redo = env_redo ? atoi(env_redo) : 0;
    if (gmg_prof_begin(ctx, GMG_PROF_FS)) return 1;
    k_score_many<<<grid, 256, smem, ctx->stream>>>((const DevIcm*)d_models, d_slot, s->d_words, s->d_off, s->n, frame,
                                                  (double*)d_out, (uint8_t*)d_redo, force_redo);
    const int64_t pairs = (int64_t)fast_slots.size() * s->n;
    k_score_many_redo<<<(unsigned)((pairs * 32 + 127) / 128), 128, 0, ctx->stream>>>(
        (const DevIcm*)d_models, d_slot, (int)fast_slots.size(), s->d_words, s->d_off, s->n, frame, (double*)d_out,
        (const uint8_t*)d_redo);
    gmg_prof_end(ctx, GMG_PROF_FS);
    ctx->launches += 2;
    GMG_CUDA(cudaGetLastError());
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));  // dev / fast_slots are host temporaries
  }
  for (int k : ordered_slots) {  // branch table too large for shared memory: the ordered kernel, model by model
    const gmg_icm* m = models[k];
    int64_t threads = s->n * 32;
    k_string_scores<<<(unsigned)((threads + 127) / 128), 128, 0, ctx->stream>>>(m->dev, s->d_words, s->d_off, s->n, frame, 0,
                                                                               (double*)d_out + (size_t)k * s->n);
    ctx->launches++;
    GMG_CUDA(cudaGetLastError());
  }
  GMG_CUDA(cudaMemcpyAsync(h_out, d_out, (size_t)n_models * s->n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int gmg_icm_score_strings(gmg_ctx* ctx, const gmg_icm* m, gmg_seqset* s, int frame, double* h_out) {
  return string_scores(ctx, m, s, frame, 0, h_out);
}
extern "C" int gmg_icm_cumulative_score(gmg_ctx* ctx, const gmg_icm* m, gmg_seqset* s, int frame, double* h_out) {
  return string_scores(ctx, m, s, frame, 1, h_out);
}
extern "C" int gmg_icm_frame_score(gmg_ctx* ctx, const gmg_icm* m, gmg_seqset* s, int frame, double* h_out) {
  return string_scores(ctx, m, s, frame, 2, h_out);
}

extern "C" int gmg_icm_full_window_prob(gmg_ctx* ctx, const gmg_icm* m, const char* w, int frame, double* out) {
  GMG_CHECK(ctx && m && w && out, "gmg_icm_full_window_prob: NULL argument");
  int64_t off[2] = {0, m->W};
  gmg_seqset* s = NULL;
  if (gmg_seqset_create(ctx, w, off, 1, NULL, &s)) return 1;
  std::vector<double> v(m->W);
  int rc = string_scores(ctx, m, s, frame, 2, v.data());
  gmg_seqset_free(s);
  if (rc == 0) *out = v[m->W - 1];
  return rc;
}

extern "C" int gmg_icm_partial_window_prob(gmg_ctx* ctx, const gmg_icm* m, int predict_pos, const char* str, int frame,
                                           double* out) {
  GMG_CHECK(ctx && m && str && out && predict_pos >= 0, "gmg_icm_partial_window_prob: bad argument");
  int64_t off[2] = {0, predict_pos + 1};
  gmg_seqset* s = NULL;
  if (gmg_seqset_create(ctx, str, off, 1, NULL, &s)) return 1;
  std::vector<double> v(predict_pos + 1);
  int rc = string_scores(ctx, m, s, frame, 2, v.data());
  gmg_seqset_free(s);
  if (rc == 0) *out = v[predict_pos];
  return rc;
}

// ------------------------------------------------------------------------------------------------
// Codon bitmaps.  For every strand and reading-frame stream r = (codon's first base) mod 3 one bit per codon
// says "start codon" and one "stop codon":  uint2 {start, stop} [strand][r][nwc],  bit i of word w <-> the codon
// at global bases 3 (32 w + i) + r .. + 2 (reverse strand: the same three bases read as their reverse
// complement).  The ORF finder and the glimmer3 start enumeration then work on 32 codons per word with
// clz / ffs / popc instead of per-codon extraction.  One thread builds the 12 words of one word index.
__global__ void __launch_bounds__(128) k_codon_bits(const uint64_t* __restrict__ words, int64_t nwc, CodonSets cs,
                                                    uint2* __restrict__ cb) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nwc) return;
  // bases 96 w .. 96 w + 127 (zero padding past the end of the batch)
  uint64_t x[4];
#pragma unroll
  for (int k = 0; k < 4; k++) x[k] = __ldg(words + 3 * w + k);
#pragma unroll
  for (int r = 0; r < 3; r++) {
    unsigned fs = 0, fp = 0, rs = 0, rp = 0;
#pragma unroll
    for (int i = 0; i < 32; i++) {
      const int o = 3 * i + r, k = o >> 5, sh = 2 * (o & 31);
      uint64_t v = x[k] >> sh;
      if (sh > 58) v |= x[k + 1] << (64 - sh);
      const int raw = (int)(v & 63);
      fs |= (unsigned)((cs.raw_mask[0] >> raw) & 1) << i;
      fp |= (unsigned)((cs.raw_mask[1] >> raw) & 1) << i;
      rs |= (unsigned)((cs.raw_mask[2] >> raw) & 1) << i;
      rp |= (unsigned)((cs.raw_mask[3] >> raw) & 1) << i;
    }
    cb[(size_t)r * nwc + w] = make_uint2(fs, fp);
    cb[(size_t)(3 + r) * nwc + w] = make_uint2(rs, rp);
  }
}

static int ensure_codon_bits(gmg_ctx* ctx, gmg_seqset* s, const CodonSets& cs) {
  if (s->d_cbits && memcmp(s->cbits_key, cs.raw_mask, sizeof s->cbits_key) == 0) return 0;
  const int64_t nwc = s->total / 96 + 2;
  if (!s->d_cbits) {
    // the last word index reads packed words up to 3 (nwc - 1) + 3 <= total / 32 + 6: inside the zero padding (8 words)
    static_assert(GMG_PAD_WORDS >= 7, "k_codon_bits reads up to seven words past the last base");
    GMG_CUDA(cudaMallocAsync(&s->d_cbits, (size_t)6 * nwc * sizeof(uint2), ctx->stream));
    s->nwc = nwc;
  }
  k_codon_bits<<<(unsigned)((nwc + 127) / 128), 128, 0, ctx->stream>>>(s->d_words, nwc, cs, s->d_cbits);
  ctx->launches++;
  GMG_CUDA(cudaGetLastError());
  memcpy(s->cbits_key, cs.raw_mask, sizeof s->cbits_key);
  return 0;
}

// One stream of the codon bitmaps as the ORF finder sees it: a CTA stages the words its tile can ask for (its own
// 12 plus ORF_HALO below them) in shared memory; anything further down comes from global memory.
#define ORF_TILE 1024      // bases per CTA, four consecutive bases per thread
#define ORF_STAGE_CAP 256  // ORF records a CTA can stage in the single-pass mode
#define ORF_HALO 2         // 2 words = 64 codons = 192 bases: every look-back of a short read stays in shared memory
#define ORF_SW (ORF_HALO + 12)
#define ORF_NB 129         // sequence bounds staged per CTA
struct CbView {
  const uint2* g;  // the six streams' words in global memory [6][nwc]
  const uint2* s;  // staged copy of words [w0, w0 + ORF_SW) of every stream [6][ORF_SW]
  int64_t nwc;
  int w0;
  __device__ __forceinline__ uint2 at(int strm, int w) const {
    const unsigned d = (unsigned)(w - w0);
    return d < (unsigned)ORF_SW ? s[strm * ORF_SW + d] : __ldg(g + (size_t)strm * nwc + w);
  }
};

// Scan one stream's codon bits downwards over the slots [s_lo, s_hi]: the highest slot with a stop bit
// (-1 = none) and, among the slots above it, the lowest (`far`) and highest (`near`) one with a start bit.
struct BackScan {
  int stop, far, near;  // slot numbers (< 2^32 / 3: batches hold fewer than 2^32 bases), -1 = none
};
__device__ __forceinline__ BackScan scan_back(const CbView& cb, int strm, int s_hi, int s_lo) {
  BackScan r;
  r.stop = r.far = r.near = -1;
  if (s_hi < s_lo) return r;
  const int w_hi = s_hi >> 5, w_lo = s_lo >> 5;
  const unsigned m_hi = (2u << (s_hi & 31)) - 1u, m_lo = ~0u << (s_lo & 31);
  for (int w = w_hi; w >= w_lo; --w) {
    const uint2 x = cb.at(strm, w);
    const unsigned m = (w == w_hi ? m_hi : ~0u) & (w == w_lo ? m_lo : ~0u);
    unsigned st = x.x & m;
    const unsigned sp = x.y & m;
    int b = -1;
    if (sp) {
      b = 31 - __clz(sp);
      st &= ~((2u << b) - 1u);  // only starts above the stop count
    }
    if (st) {
      if (r.near < 0) r.near = (w << 5) + 31 - __clz(st);
      r.far = (w << 5) + __ffs(st) - 1;
    }
    if (sp) {
      r.stop = (w << 5) + b;
      break;
    }
  }
  return r;
}

// ------------------------------------------------------------------------------------------------
// Device ORF finder (Find_Orfs, glimmer_base.cc:638-817; linear sequences, no ignore regions).
//
// Every ORF is created by the stop codon that closes it.  A base that closes an ORF (at most one forward and one
// reverse stop, plus the Finish_Orfs reverse ORFs and the three virtual forward stops at a sequence's last base)
// looks up the previous in-frame stop and the relevant start codon in the codon bitmaps (32 codons per word).
// The reference's output order -- by closing base; forward before reverse; then the end-of-sequence extras -- is
// kept by ranks: count, block scan, emit inside a CTA; a device scan of the CTA totals between CTAs.

// forward ORF closed by the (possibly virtual) stop codon whose last base is i (sequence coordinates).
__device__ bool orf_fwd_closed(const CbView& cbv, int64_t a, int L, int i, const DevParams& P, gmg_orf* o) {
  // candidate codons end at t = i-3, i-6, ... >= 2, i.e. start at i-5, i-8, ... >= 0
  // 32-bit arithmetic: global base indices are below 2^32 (build_buckets checks the batch size)
  const uint32_t a32 = (uint32_t)a;
  const int r = (int)((a32 + (uint32_t)i + 1u) % 3u);
  const int s_hi = i >= 5 ? (int)((a32 + (uint32_t)i - 5u) / 3u) : -1, s_lo = (int)((a32 - (uint32_t)r + 2u) / 3u);
  const BackScan f = scan_back(cbv, r, s_hi, s_lo);
  const int prev = f.stop >= 0 ? (int)(3u * (uint32_t)f.stop + (uint32_t)r - a32) + 1 : 0;  // 1-based first base of the previous stop
  const int first_start = f.far >= 0 ? (int)(3u * (uint32_t)f.far + (uint32_t)r - a32) + 1 : INT_MAX;
  int gene_len, orf_len;
  if (prev == 0) {
    int pos = i - 1;
    orf_len = pos - 1;
    orf_len -= orf_len % 3;
    gene_len = (first_start == INT_MAX) ? 0 : pos - first_start;
    if (P.allow_truncated && gene_len < P.min_gene_len) gene_len = orf_len;
  } else {
    gene_len = (int)((long long)i - first_start - 1);
    orf_len = i - prev - 4;
  }
  if (!(gene_len >= P.min_gene_len || ((P.allow_indels || P.allow_subs) && orf_len >= P.min_indel_orf_len)))
    return false;
  o->stop_position = i - 1;
  o->frame = 1 + (i % 3 + 1) % 3;
  o->gene_len = gene_len;
  o->orf_len = orf_len;
  return true;
}

// reverse ORF closed at i (real reverse stop whose highest base is i), or with finish = true the
// Finish_Orfs ORF of frame class fr = i % 3 where i is the last position of that class (< L).
__device__ bool orf_rev_closed(const CbView& cbv, int64_t a, int L, int i, bool finish, const DevParams& P,
                               gmg_orf* o) {
  const int t0 = finish ? i : i - 3;  // candidate codons end at t0, t0-3, ... >= 2
  const uint32_t a32 = (uint32_t)a;
  const int r = (int)((a32 + (uint32_t)(t0 + 1)) % 3u);  // t0 >= -1 in every call
  const int s_hi = t0 >= 2 ? (int)((a32 + (uint32_t)t0 - 2u) / 3u) : -1, s_lo = (int)((a32 - (uint32_t)r + 2u) / 3u);
  const BackScan f = scan_back(cbv, 3 + r, s_hi, s_lo);
  const int prev = f.stop >= 0 ? (int)(3u * (uint32_t)f.stop + (uint32_t)r - a32) + 1 : 0;
  const int last_start = f.near >= 0 ? (int)(3u * (uint32_t)f.near + (uint32_t)r - a32) + 1 : 0;  // nearest to i
  int gene_len, orf_len, orf_stop;
  if (!finish) {
    if (prev == 0) {
      if (!P.allow_truncated) {
        gene_len = 0;
        orf_stop = 0;  // glimmer_base.cc:513,999-1003: orf_stop keeps its initial value
      } else {
        orf_stop = (i - 1) % 3;
        if (orf_stop > 0) orf_stop -= 3;
        gene_len = last_start - orf_stop;
      }
    } else {
      orf_stop = prev;
      gene_len = last_start - orf_stop;
    }
    orf_len = i - orf_stop - 4;
  } else {
    const int fr = i % 3;
    orf_stop = prev ? prev : (fr == 0 ? -1 : (fr == 1 ? 0 : -2));
    orf_len = L - orf_stop - 2;
    orf_len -= orf_len % 3;
    gene_len = (last_start == 0) ? 0 : last_start - orf_stop;
    if (P.allow_truncated && gene_len < P.min_gene_len) gene_len = orf_len;
  }
  if (!(gene_len >= P.min_gene_len || ((P.allow_indels || P.allow_subs) && orf_len >= P.min_indel_orf_len)))
    return false;
  o->stop_position = orf_stop;
  o->frame = -1 - (i % 3 + 1) % 3;
  o->gene_len = gene_len;
  o->orf_len = orf_len;
  return true;
}

// One CTA per tile of ORF_TILE bases.  Staged once per CTA: the sequence bounds that fall into the tile and the codon
// bitmap words its look-backs can reach (ORF_SW per stream), so that on read sets no thread touches global memory
// between the staging and its records.
//   phase A  every thread tests the stop bits of its four bases and the "last base of a sequence" condition: a mask of
//            CANDIDATE events (base x 8 kinds: forward stop, reverse stop, the three Finish_Orfs reverse ORFs, the three
//            virtual forward stops -- the reference's order within a base); a block scan numbers them in output order
//            and they are written, as 16-bit descriptors, to a shared-memory list;
//   phase B  one thread per candidate evaluates it (orf_fwd_closed / orf_rev_closed), a block scan per 256 candidates
//            ranks the ORFs that exist, and they are written at their ranks.
// Evaluating events where they are found (one thread per base, 2-3 lanes of a warp inside the divergent look-back at any
// time) cost 25 warp instructions per BASE: 0.65-0.8 ms per 31 Mbp, all of it instruction issue; compacted, the same
// look-backs run with full warps.
// kMode 1: records at block_base[blockIdx] + rank (write pass after an overflow).  kMode 2: single pass -- per-CTA
// counts AND the records staged at slot blockIdx * ORF_STAGE_CAP + rank (a CTA with more than ORF_STAGE_CAP ORFs raises
// *overflow and the caller re-runs the batch with kMode 1); k_orfs_compact then moves the staged records to their final,
// scan-ordered places.
#define ORF_CAND_CAP 4096  // candidate descriptors per round (a tile holds at most 2 * ORF_TILE + 6 * its sequence ends)
template <int kMode>
__global__ void __launch_bounds__(256) k_orfs(const uint2* __restrict__ cb, int64_t nwc, const int64_t* __restrict__ off,
                                              const int32_t* __restrict__ blk2seq, int64_t total, DevParams P,
                                              int64_t* __restrict__ block_counts, const int64_t* __restrict__ block_base,
                                              gmg_orf* __restrict__ orfs, int32_t* __restrict__ orf_seq,
                                              int* __restrict__ overflow, int64_t n_seq) {
  typedef cub::BlockScan<int, 256> Scan;
  __shared__ typename Scan::TempStorage tmp;
  __shared__ uint2 s_cb[6][ORF_SW];
  __shared__ long long s_bound[ORF_NB];
  __shared__ int s_s0;
  __shared__ unsigned short s_cand[ORF_CAND_CAP];
  __shared__ unsigned char s_blk[ORF_TILE / 32];
  const int64_t p0 = (int64_t)blockIdx.x * ORF_TILE;
  const int w0 = (int)(((p0 >= 2 ? p0 - 2 : 0) / 3) >> 5) - ORF_HALO;
  const int t = threadIdx.x;
  if (t < 6 * ORF_SW) {
    const int strm = t / ORF_SW, k = t - strm * ORF_SW;
    const int64_t w = (int64_t)w0 + k;
    s_cb[strm][k] = (w >= 0 && w < nwc) ? __ldg(cb + (size_t)strm * nwc + w) : make_uint2(0u, 0u);
  } else if (t >= 96 && t < 96 + ORF_NB) {
    const int k = t - 96;
    const int32_t s0 = __ldg(blk2seq + (p0 >> 5)) & 0x7FFFFFFF;  // p0 is a multiple of 32: the sequence that holds it
    const int64_t idx = (int64_t)s0 + k;
    s_bound[k] = idx <= n_seq ? (long long)__ldg(off + idx) : LLONG_MAX;
    if (k == 0) s_s0 = s0;
  }
  __syncthreads();
  CbView cbv;
  cbv.g = cb;
  cbv.s = &s_cb[0][0];
  cbv.nwc = nwc;
  cbv.w0 = w0;
  const bool staged = s_bound[ORF_NB - 1] > p0 + ORF_TILE - 1;  // all of the tile's sequences are in the staged list
  // staged bound index of the sequence holding the first base of each 32-base block of the tile (one binary search per
  // block instead of one per thread and candidate)
  if (staged && t < ORF_TILE / 32) {
    const int64_t p = p0 + 32 * t;
    int lo = 0, hi = ORF_NB - 1;  // s_bound[lo] <= p < s_bound[hi]; empty sequences repeat a bound: the last one holds the base
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (s_bound[mid] <= p) lo = mid;
      else hi = mid;
    }
    s_blk[t] = (unsigned char)lo;
  }
  __syncthreads();
  // the sequence holding global base p: index, first base, length
  auto seq_of = [&](int64_t p, int32_t* sq, int64_t* a, int* L) {
    if (staged) {  // largest k with s_bound[k] <= p
      int k = s_blk[(int)(p - p0) >> 5];
      while (s_bound[k + 1] <= p) k++;
      *sq = s_s0 + k;
      *a = s_bound[k];
      *L = (int)(s_bound[k + 1] - s_bound[k]);
    } else {
      SeqView sv = locate(off, blk2seq, p, sq);
      *a = sv.a;
      *L = sv.len;
    }
  };
  // ---- phase A: candidate mask of this thread's bases pt .. pt + 3 (bit 8 m + kind)
  const int64_t pt = p0 + 4 * t;
  unsigned cm = 0;
  if (pt < total) {
    int32_t sq;
    int64_t a;
    int L;
    seq_of(pt, &sq, &a, &L);
    int64_t next = a + L;
    const uint32_t c0 = (uint32_t)(pt >= 2 ? pt - 2 : 0);
    uint32_t r = c0 % 3u, sl = c0 / 3u;
    if (pt < 2) {  // bases 0, 1 of the batch close no codon; the codon of base 2 is (r, sl) = (0, 0)
      r = (uint32_t)((pt + 1) % 3);  // so that after (2 - pt) steps r == 0
      sl = 0;
    }
#pragma unroll
    for (int m = 0; m < 4; m++) {
      const int64_t p = pt + m;
      if (p < total) {
        if (p >= next) {  // the next non-empty sequence
          seq_of(p, &sq, &a, &L);
          next = a + L;
        }
        const int q = (int)(p - a);
        if (L >= P.min_gene_len) {
          if (q >= 2) {  // the codon q-2 .. q: forward stop / reverse stop?
            const unsigned d = (unsigned)((int)(sl >> 5) - w0);  // < ORF_SW by construction of the stage
            const unsigned bit = 1u << (sl & 31u);
            if (s_cb[r][d].y & bit) cm |= 1u << (8 * m);
            if (s_cb[3 + r][d].y & bit) cm |= 2u << (8 * m);
          }
          if (q == L - 1) cm |= (P.allow_truncated ? 0xFCu : 0x1Cu) << (8 * m);
        }
      }
      if (p >= 2) {  // advance (r, sl) to the codon ending at p + 1
        if (++r == 3u) {
          r = 0;
          sl++;
        }
      } else {
        r = (r + 1u) % 3u;
      }
    }
  }
  int my_n = __popc(cm), my_off, n_cand;
  Scan(tmp).ExclusiveSum(my_n, my_off, n_cand);
  int64_t out_base = kMode == 1 ? block_base[blockIdx.x] : (int64_t)blockIdx.x * ORF_STAGE_CAP;
  int placed = 0;  // ORFs of this tile written (or counted) so far
  // ---- rounds of at most ORF_CAND_CAP candidates (one round unless the tile is full of tiny sequences)
  for (int r0 = 0; r0 < n_cand; r0 += ORF_CAND_CAP) {
    __syncthreads();  // the list (and the scan's storage) are free again
    {
      unsigned x = cm;
      int i = my_off;
      while (x) {
        const int b = __ffs(x) - 1;
        x &= x - 1u;
        if (i >= r0 && i < r0 + ORF_CAND_CAP) s_cand[i - r0] = (unsigned short)(((4 * t + (b >> 3)) << 3) | (b & 7));
        i++;
      }
    }
    __syncthreads();
    const int n_round = min(n_cand - r0, ORF_CAND_CAP);
    // ---- phase B
    for (int c0 = 0; c0 < n_round; c0 += 256) {
      const int i = c0 + t;
      gmg_orf rec;
      int32_t sq = 0;
      int ok = 0;
      if (i < n_round) {
        const unsigned dsc = s_cand[i];
        const int kind = (int)(dsc & 7u);
        const int64_t p = p0 + (int64_t)(dsc >> 3);
        int64_t a;
        int L;
        seq_of(p, &sq, &a, &L);
        const int q = (int)(p - a);
        // two code paths for the eight kinds, so a warp of mixed candidates runs each look-back at most twice
        if (kind == 0 || kind >= 5) {
          ok = orf_fwd_closed(cbv, a, L, kind == 0 ? q : L + (kind - 5), P, &rec);
        } else {
          const bool finish = kind != 1;
          const int fr = kind - 2;
          int ii = q;
          if (finish) {
            ii = L - 1 - mod3(L - 1 - fr);  // last index of class fr that is < L
            if (ii < 0) ii = fr;            // degenerate; the search range is empty
          }
          ok = orf_rev_closed(cbv, a, L, ii, finish, P, &rec);
          if (finish) rec.frame = -1 - (fr + 1) % 3;  // only depends on fr (= ii % 3 when ii >= 0)
        }
      }
      int rank, found;
      __syncthreads();
      Scan(tmp).ExclusiveSum(ok, rank, found);
      if (ok) {
        const int slot = placed + rank;
        if (kMode == 1 || slot < ORF_STAGE_CAP) {
          orfs[out_base + slot] = rec;
          orf_seq[out_base + slot] = sq;
        }
      }
      placed += found;
    }
  }
  if (kMode == 2 && t == 0) {
    block_counts[blockIdx.x] = placed;
    if (placed > ORF_STAGE_CAP) *overflow = 1;
  }
}

// staged records of CTA b -> orfs[block_base[b] ..): ORF_STAGE_CAP threads per CTA of k_orfs<2>
__global__ void __launch_bounds__(256) k_orfs_compact(const gmg_orf* __restrict__ st_orfs,
                                                      const int32_t* __restrict__ st_seq,
                                                      const int64_t* __restrict__ block_base, int64_t nblk,
                                                      gmg_orf* __restrict__ orfs, int32_t* __restrict__ orf_seq) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t b = g / ORF_STAGE_CAP;
  const int t = (int)(g % ORF_STAGE_CAP);
  if (b >= nblk) return;
  const int64_t lo = block_base[b];
  if (t >= block_base[b + 1] - lo) return;
  orfs[lo + t] = st_orfs[g];
  orf_seq[lo + t] = st_seq[g];
}

// first ORF of every sequence (orf_seq is sorted): lower bound
__global__ void k_orf_offsets(const int32_t* __restrict__ orf_seq, int64_t n_orfs, int64_t n_seq,
                              int64_t* __restrict__ orf_off) {
  int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s > n_seq) return;
  int64_t lo = 0, hi = n_orfs;  // first index with orf_seq >= s
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if (orf_seq[mid] < s) lo = mid + 1;
    else hi = mid;
  }
  orf_off[s] = lo;
}

__global__ void k_orf_seq_from_off(const int64_t* __restrict__ orf_off, int64_t n_seq, int64_t n_orfs,
                                   int32_t* __restrict__ orf_seq) {
  int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= n_orfs) return;
  int64_t lo = 0, hi = n_seq;  // largest s with orf_off[s] <= o
  while (hi - lo > 1) {
    int64_t mid = (lo + hi) >> 1;
    if (orf_off[mid] <= o) lo = mid;
    else hi = mid;
  }
  orf_seq[o] = (int32_t)lo;
}

static int exclusive_sum_i64_on(gmg_ctx* ctx, cudaStream_t stream, int64_t* d_in, int64_t* d_out, int64_t n) {
  size_t tmp_bytes = 0;
  GMG_CUDA(cub::DeviceScan::ExclusiveSum(NULL, tmp_bytes, d_in, d_out, n, stream));
  void* tmp;
  if (gmg_scratch(ctx, SCR_TMP4, tmp_bytes, &tmp)) return 1;
  GMG_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, d_in, d_out, n, stream));
  ctx->launches += 2;
  return 0;
}
static int exclusive_sum_i64(gmg_ctx* ctx, int64_t* d_in, int64_t* d_out, int64_t n) {
  return exclusive_sum_i64_on(ctx, ctx->stream, d_in, d_out, n);
}

static int ensure_orf_capacity(gmg_seqset* s, int64_t n_orfs) {
  if ((size_t)n_orfs > s->cap_orfs || !s->d_orfs) {
    if (s->d_orfs) cudaFreeAsync(s->d_orfs, s->ctx->stream);
    if (s->d_orf_seq) cudaFreeAsync(s->d_orf_seq, s->ctx->stream);
    if (s->d_start_off) cudaFreeAsync(s->d_start_off, s->ctx->stream);
    s->d_orfs = NULL; s->d_orf_seq = NULL; s->d_start_off = NULL;
    size_t cap = (size_t)n_orfs + (size_t)n_orfs / 8 + 64;
    GMG_CUDA(cudaMallocAsync(&s->d_orfs, cap * sizeof(gmg_orf), s->ctx->stream));
    GMG_CUDA(cudaMallocAsync(&s->d_orf_seq, cap * sizeof(int32_t), s->ctx->stream));
    GMG_CUDA(cudaMallocAsync(&s->d_start_off, (cap + 1) * sizeof(int64_t), s->ctx->stream));
    s->cap_orfs = cap;
  }
  if (!s->d_orf_off) GMG_CUDA(cudaMallocAsync(&s->d_orf_off, (size_t)(s->n + 2) * sizeof(int64_t), s->ctx->stream));
  return 0;
}

extern "C" int gmg_find_orfs(gmg_ctx* ctx, gmg_seqset* s, const gmg_params* p, int64_t* n_orfs) {
  GMG_CHECK(ctx && s && p, "gmg_find_orfs: NULL argument");
  CodonSets cs;
  DevParams dp;
  if (make_codon_sets(p, &cs, &dp)) return 1;
  s->n_orfs = 0;
  s->n_starts = 0;
  if (s->total == 0) {
    if (ensure_orf_capacity(s, 0)) return 1;
    GMG_CUDA(cudaMemsetAsync(s->d_orf_off, 0, (size_t)(s->n + 1) * sizeof(int64_t), ctx->stream));
    s->orf_off.assign((size_t)s->n + 1, 0);
    if (n_orfs) *n_orfs = 0;
    return 0;
  }
  if (ensure_codon_bits(ctx, s, cs)) return 1;
  int64_t nblk = (s->total + ORF_TILE - 1) / ORF_TILE;
  void* d_counts;
  if (gmg_scratch(ctx, SCR_FLAGS, (size_t)(2 * (nblk + 1)) * sizeof(int64_t), &d_counts)) return 1;
  int64_t* counts = (int64_t*)d_counts;
  int64_t* bases = counts + nblk + 1;
  GMG_CUDA(cudaMemsetAsync(counts + nblk, 0, sizeof(int64_t), ctx->stream));
  // single pass: records staged per CTA (ORF_STAGE_CAP slots each), counted, scanned, compacted
  void *d_stage;
  const size_t stage_slots = (size_t)nblk * ORF_STAGE_CAP;
  if (gmg_scratch(ctx, SCR_TMP2, stage_slots * (sizeof(gmg_orf) + sizeof(int32_t)) + 16, &d_stage)) return 1;
  gmg_orf* st_orfs = (gmg_orf*)d_stage;
  int32_t* st_seq = (int32_t*)(st_orfs + stage_slots);
  int* d_overflow = (int*)(st_seq + stage_slots);
  GMG_CUDA(cudaMemsetAsync(d_overflow, 0, sizeof(int), ctx->stream));
  if (gmg_prof_begin(ctx, GMG_PROF_ORF)) return 1;
  k_orfs<2><<<(unsigned)nblk, 256, 0, ctx->stream>>>(s->d_cbits, s->nwc, s->d_off, s->d_blk2seq, s->total, dp, counts, NULL,
                                                     st_orfs, st_seq, d_overflow, s->n);
  gmg_prof_end(ctx, GMG_PROF_ORF);
  ctx->launches++;
  GMG_CUDA(cudaGetLastError());
  if (exclusive_sum_i64(ctx, counts, bases, nblk + 1)) return 1;
  ctx->h_scalars[2] = 0;
  ctx->h_scalars[3] = 0;
  GMG_CUDA(cudaMemcpyAsync(&ctx->h_scalars[2], bases + nblk, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaMemcpyAsync(&ctx->h_scalars[3], d_overflow, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  const int64_t total_orfs = ctx->h_scalars[2];
  const char* two_pass = getenv("GMG_ORF_TWO_PASS");  // test hook: take the overflow path
  const bool overflow = (ctx->h_scalars[3] & 0xffffffff) != 0 || (two_pass && atoi(two_pass));
  if (ensure_orf_capacity(s, total_orfs)) return 1;
  if (gmg_prof_begin(ctx, GMG_PROF_ORF)) return 1;
  if (!overflow)
    k_orfs_compact<<<(unsigned)((stage_slots + 255) / 256), 256, 0, ctx->stream>>>(st_orfs, st_seq, bases, nblk, s->d_orfs,
                                                                                 s->d_orf_seq);
  else  // some CTA found more ORFs than it could stage: write pass over the whole batch
    k_orfs<1><<<(unsigned)nblk, 256, 0, ctx->stream>>>(s->d_cbits, s->nwc, s->d_off, s->d_blk2seq, s->total, dp, NULL, bases,
                                                       s->d_orfs, s->d_orf_seq, NULL, s->n);
  gmg_prof_end(ctx, GMG_PROF_ORF);
  k_orf_offsets<<<(unsigned)((s->n + 1 + 255) / 256), 256, 0, ctx->stream>>>(s->d_orf_seq, total_orfs, s->n, s->d_orf_off);
  ctx->launches += 2;
  GMG_CUDA(cudaGetLastError());
  s->n_orfs = total_orfs;
  s->orfs_external = 0;
  s->orf_off.clear();
  if (n_orfs) *n_orfs = total_orfs;
  return 0;
}

extern "C" int gmg_get_orfs(gmg_ctx* ctx, gmg_seqset* s, gmg_orf* h_orfs, int64_t* h_orf_off) {
  GMG_CHECK(ctx && s, "gmg_get_orfs: NULL argument");
  if (h_orfs && s->n_orfs)
    GMG_CUDA(cudaMemcpyAsync(h_orfs, s->d_orfs, (size_t)s->n_orfs * sizeof(gmg_orf), cudaMemcpyDeviceToHost, ctx->stream));
  if (h_orf_off && s->d_orf_off)
    GMG_CUDA(cudaMemcpyAsync(h_orf_off, s->d_orf_off, (size_t)(s->n + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost,
                             ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int gmg_set_orfs(gmg_ctx* ctx, gmg_seqset* s, const gmg_orf* h_orfs, const int64_t* h_orf_off) {
  GMG_CHECK(ctx && s && h_orf_off, "gmg_set_orfs: NULL argument");
  int64_t n_orfs = h_orf_off[s->n];
  GMG_CHECK(n_orfs >= 0 && h_orf_off[0] == 0, "gmg_set_orfs: bad offsets");
  GMG_CHECK(n_orfs == 0 || h_orfs, "gmg_set_orfs: NULL ORF table");
  // geometry: the kernels score linear sequences; a wrap-around ORF of a circular genome (Find_Orfs with
  // Genome_Is_Circular, glimmer_base.cc:760-777) would be read from the neighbouring sequence
  for (int64_t q = 0; q < s->n; q++) {
    GMG_CHECK(h_orf_off[q + 1] >= h_orf_off[q], "gmg_set_orfs: offsets not monotone at sequence %lld", (long long)q);
    const int64_t L = s->off[(size_t)q + 1] - s->off[(size_t)q];
    for (int64_t o = h_orf_off[q]; o < h_orf_off[q + 1]; o++) {
      const gmg_orf& f = h_orfs[o];
      const int af = f.frame < 0 ? -f.frame : f.frame;
      GMG_CHECK(af >= 1 && af <= 3 && f.orf_len >= 0, "gmg_set_orfs: ORF %lld has frame %d, orf_len %d", (long long)o, f.frame, f.orf_len);
      const int64_t lo = f.frame > 0 ? (int64_t)f.stop_position - 1 - f.orf_len : (int64_t)f.stop_position + 2;
      const int64_t hi = f.frame > 0 ? (int64_t)f.stop_position - 1 : (int64_t)f.stop_position + 2 + f.orf_len;
      GMG_CHECK(lo >= 0 && hi <= L, "gmg_set_orfs: ORF %lld (frame %d, stop %d, length %d) does not lie inside its %lld bp sequence: "
                "wrap-around ORFs of circular sequences are not supported", (long long)o, f.frame, f.stop_position, f.orf_len, (long long)L);
    }
  }
  if (ensure_orf_capacity(s, n_orfs)) return 1;
  if (n_orfs)
    GMG_CUDA(cudaMemcpyAsync(s->d_orfs, h_orfs, (size_t)n_orfs * sizeof(gmg_orf), cudaMemcpyHostToDevice, ctx->stream));
  GMG_CUDA(cudaMemcpyAsync(s->d_orf_off, h_orf_off, (size_t)(s->n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice,
                           ctx->stream));
  if (n_orfs) {
    k_orf_seq_from_off<<<(unsigned)((n_orfs + 255) / 256), 256, 0, ctx->stream>>>(s->d_orf_off, s->n, n_orfs, s->d_orf_seq);
    ctx->launches++;
    GMG_CUDA(cudaGetLastError());
  }
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  s->n_orfs = n_orfs;
  s->n_starts = 0;
  s->orfs_external = 1;  // caller's table: its lengths are not trusted to agree with the sequence's stop codons
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Start-list emission shared by the glimmer3 and glimmer-mg kernels.

struct Emit {
  gmg_start* out;  // NULL = counting pass
  int64_t n;
};

__device__ __forceinline__ void emit_start(Emit& e, int j, int pos, double score, int which, int truncated, int first,
                                           int n_err, const int* err_pos, const int* err_type, int ignore_len) {
  if (e.out) {
    gmg_start st;
    st.j = j;
    st.pos = pos;
    // long-ORF boost (glimmer-mg.cc:1649-1651, glimmer3.cc:1464-1466): Max(0.0, score)
    st.score = (j > ignore_len && 0.0 > score) ? 0.0 : score;
    st.which = which;
    st.truncated = truncated;
    st.first = first;
    st.n_err = n_err;
    st.err_pos[0] = n_err > 0 ? err_pos[0] : 0;
    st.err_pos[1] = n_err > 1 ? err_pos[1] : 0;
    st.err_type[0] = n_err > 0 ? err_type[0] : 0;
    st.err_type[1] = n_err > 1 ? err_type[1] : 0;
    e.out[e.n] = st;
  }
  e.n++;
}

// ------------------------------------------------------------------------------------------------
// K3 (glimmer3): Score_Orfs start enumeration on the extracted ORF string (glimmer3.cc:1275-1466).
//
// One warp per ORF.  buff[j] = S[hi-1-j] (forward) / complement S[lo+j] (reverse); the gene ICM and the
// independent model are accumulated SEPARATELY in FP64 in j order with the period cycling 1,2,0
// (Cumulative_Score icm.cc:354-405).  Positions j >= W-1 read the K1 planes; the first W-1 positions
// use partial windows that only see the ORF string (icm.cc:376-388), recomputed here.
// Lanes evaluate 32 consecutive j; the running sums are formed by an ordered in-warp accumulation, so
// every prefix has exactly the reference's serial rounding -- no reassociation.

struct G3Geom {
  int frame, lo, hi, len, k0, trunc;
};

__device__ __forceinline__ G3Geom g3_geom(const gmg_orf& o, int L, const DevParams& P) {
  G3Geom g;
  g.frame = o.frame;
  g.len = o.orf_len;
  if (o.frame > 0) {
    g.hi = o.stop_position - 1;
    if (g.hi <= 0) g.hi += L;
    g.lo = g.hi - g.len;
    g.trunc = (g.lo < 3 && P.allow_truncated);
    g.k0 = o.stop_position - g.len - 2;
  } else {
    g.lo = o.stop_position + 2;
    if (g.lo >= L) g.lo -= L;
    g.hi = g.lo + g.len;
    g.trunc = (L - g.hi < 3 && P.allow_truncated);
    g.k0 = o.stop_position + g.len + 4;
  }
  return g;
}

// is j a start position of this ORF string?  returns which (>=0), -1 = only by the truncated rule, -2 = no
__device__ __forceinline__ int g3_codon_which(const uint64_t* __restrict__ words, int64_t a, const G3Geom& g, int j,
                                              const CodonSets& cs) {
  // codon register after shifting in buff[m-1] .. buff[j]: buff[j+2], buff[j+1], buff[j]; complete iff j <= m-3
  if (j > g.len - 3) return -1;
  int c;
  if (g.frame > 0) c = codon_fwd_ending_at(words, a, g.hi - 1 - j);  // S[p-2], S[p-1], S[p], p = hi-1-j
  else c = codon_rev_starting_at(words, a, g.lo + j);                 // c(S[q+2]), c(S[q+1]), c(S[q]), q = lo+j
  return ((cs.start_mask >> c) & 1) ? (int)cs.which[c] : -1;
}

// Ordered pass (the fallback of k3_g3_emit): gene / indep running sums along j in the reference's association
// (icm.cc:390-402) and emission of the start records.  Lanes evaluate 32 consecutive j; the running sums are
// formed by a lane-ordered accumulation, so every prefix has exactly the reference's serial rounding.
__device__ void g3_accumulate_ordered(const DevIcm& gene, const DevIcm& indep, const float* __restrict__ lut,
                                      const uint64_t* __restrict__ words, int64_t a, const G3Geom& g,
                                      const float* __restrict__ plane, const uint32_t* __restrict__ bktidx,
                                      int64_t total, const CodonSets& cs, const DevParams& P, int first_j, int n_emit,
                                      gmg_start* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int W = gene.W, m = g.len;
  const int lowest_j = min(3, P.min_gene_len - 3);
  const bool use_lut = (lut != NULL);
  double run_g = 0.0, run_n = 0.0;
  int emitted_below = 0;           // records of start positions below the current chunk (ascending j)
  const int j_last = first_j - 1;  // scores are needed up to index first_j - 1
  for (int base = 0; base <= j_last; base += 32) {
    const int j = base + lane;
    float xg = 0.f, xn = 0.f;
    if (j <= j_last) {
      const int f = (1 + j) % 3;
      if (g.frame > 0) {
        const int q = g.hi - 1 - j;
        xg = (j < W - 1) ? icm_fwd(gene, words, a + q, q, g.hi, f)
                         : __ldg(plane + (size_t)f * total + gmg_plane_index(words, bktidx, a + q));
        if (use_lut && j >= 2) xn = lut[f * 64 + (int)(gmg_extract32(words, a + q) & 63)];
        else xn = icm_fwd(indep, words, a + q, q, g.hi, f);
      } else {
        const int q = g.lo + j;
        xg = (j < W - 1) ? icm_rev(gene, words, a + q, q, g.lo, f)
                         : __ldg(plane + (size_t)f * total + gmg_plane_index(words, bktidx, a + q));
        if (use_lut && j >= 2) xn = lut[(3 + f) * 64 + (int)(gmg_extract32(words, a + q - 2) & 63)];
        else xn = icm_rev(indep, words, a + q, q, g.lo, f);
      }
    }
    // position base+0, base+1, ... exactly like the serial loop
    double my_g = 0.0, my_n = 0.0;
    const int cnt = min(32, j_last + 1 - base);
    for (int l = 0; l < cnt; l++) {
      run_g += (double)__shfl_sync(0xffffffffu, xg, l);
      run_n += (double)__shfl_sync(0xffffffffu, xn, l);
      if (l == lane) {
        my_g = run_g;
        my_n = run_n;
      }
    }
    // start position js = j + 1 uses score[j]
    const int js = j + 1;
    bool cand = (j <= j_last) && (js % 3 == 0) && (js >= lowest_j) && (js <= m - 1) && (js + 3 >= P.min_gene_len);
    int w = cand ? g3_codon_which(words, a, g, js, cs) : -2;
    bool is_first = cand && (js == first_j);
    bool emits = cand && (w >= 0 || (is_first && g.trunc));
    int nrec = emits ? ((is_first && g.trunc && w >= 0) ? 2 : 1) : 0;
    // records are stored in DESCENDING j order: slot = n_emit - (records at positions <= js)
    int incl = nrec;
    for (int d = 1; d < 32; d <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    if (emits) {
      const int slot = n_emit - (emitted_below + incl);
      const double sc = my_g - my_n;
      const int kpos = (g.frame > 0) ? g.k0 + (m - 1 - js) : g.k0 - (m - 1 - js);
      Emit e;
      e.out = out;
      e.n = slot;
      if (is_first && g.trunc) {
        emit_start(e, js + 2, kpos, sc, -1, 1, 1, 0, NULL, NULL, P.ignore_score_len);
        if (w >= 0) emit_start(e, js + 2, kpos, sc, w, 0, 0, 0, NULL, NULL, P.ignore_score_len);
      } else {
        emit_start(e, js + 2, kpos, sc, w, 0, is_first ? 1 : 0, 0, NULL, NULL, P.ignore_score_len);
      }
    }
    emitted_below += __shfl_sync(0xffffffffu, incl, 31);
  }
}

// The candidate start positions of an ORF string are js = jmin, jmin+3, ..., jmax (js % 3 == 0,
// lowest_j <= js, js + 3 >= min_gene_len, codon complete: js <= m - 3); their codons are consecutive slots of ONE
// codon-bitmap stream: forward  slot(js) = s0 - js / 3,  reverse  slot(js) = s0 + js / 3.
struct G3Range {
  int jmin, jmax;  // empty iff jmax < jmin
  int r;           // stream
  int64_t s0;      // slot of js = 0
};
__device__ __forceinline__ G3Range g3_range(const G3Geom& g, int64_t a, const DevParams& P) {
  G3Range R;
  const int lowest_j = min(3, P.min_gene_len - 3);
  int jmin = max(max(lowest_j, P.min_gene_len - 3), 0);
  jmin += (3 - jmin % 3) % 3;
  int jmax = g.len - 3;
  jmax -= mod3(jmax);
  R.jmin = jmin;
  R.jmax = jmax;
  const int64_t c0 = g.frame > 0 ? a + g.hi - 3 : a + g.lo;  // first base of the codon of js = 0
  R.r = (int)(c0 % 3);
  R.s0 = c0 / 3;
  return R;
}

// Count pass, one thread per ORF: popcount of the start bits over the ORF's slot range.
// counts[oi] = records, first_js[oi] = js of the first (largest-js) one; with the truncated rule the first
// candidate position emits a (which = -1) record whatever its codon (glimmer3.cc:1423-1432).
__global__ void __launch_bounds__(128) k3_g3_count(const uint2* __restrict__ cb, int64_t nwc,
                                                   const int64_t* __restrict__ off, const gmg_orf* __restrict__ orfs,
                                                   const int32_t* __restrict__ orf_seq, int64_t n_orfs, DevParams P,
                                                   int64_t* __restrict__ counts, int32_t* __restrict__ first_js,
                                                   int* __restrict__ max_len) {
  const int64_t oi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = oi < n_orfs;
  G3Geom g;
  g.len = 0;
  int64_t a = 0;
  if (live) {
    const int32_t s = orf_seq[oi];
    a = off[s];
    g = g3_geom(orfs[oi], (int)(off[s + 1] - a), P);
  }
  {  // longest ORF string of the batch (the emit pass's exactness bound)
    const int wmax = __reduce_max_sync(0xffffffffu, g.len);
    if ((threadIdx.x & 31) == 0 && wmax > 0) atomicMax(max_len, wmax);
  }
  if (!live) return;
  const G3Range R = g3_range(g, a, P);
  int cnt = 0, first = -1;
  if (R.jmax >= R.jmin) {
    const bool fwd = g.frame > 0;
    const int64_t s_lo = fwd ? R.s0 - R.jmax / 3 : R.s0 + R.jmin / 3;
    const int64_t s_hi = fwd ? R.s0 - R.jmin / 3 : R.s0 + R.jmax / 3;
    const uint2* st = cb + (size_t)(fwd ? R.r : 3 + R.r) * nwc;
    const int64_t w_lo = s_lo >> 5, w_hi = s_hi >> 5;
    const unsigned m_lo = ~0u << (int)(s_lo & 31), m_hi = (2u << (int)(s_hi & 31)) - 1u;
    int64_t ext = -1;  // forward: lowest set slot (largest js); reverse: highest set slot
    for (int64_t w = w_lo; w <= w_hi; w++) {
      const unsigned x = __ldg(st + w).x & (w == w_lo ? m_lo : ~0u) & (w == w_hi ? m_hi : ~0u);
      if (x) {
        cnt += __popc(x);
        if (fwd) {
          if (ext < 0) ext = (w << 5) + __ffs(x) - 1;
        } else {
          ext = (w << 5) + 31 - __clz(x);
        }
      }
    }
    if (ext >= 0) first = (int)(fwd ? 3 * (R.s0 - ext) : 3 * (ext - R.s0));
  }
  if (g.trunc) {  // the largest candidate position, complete codon or not
    const int jtop = (g.len - 1) - mod3(g.len - 1);
    if (jtop >= R.jmin) {
      first = jtop;
      cnt += 1;
    }
  }
  counts[oi] = cnt;
  first_js[oi] = first;
}

// Heads, kHG lanes per ORF: positions 0 .. ja of the ORF string evaluated explicitly -- the W-1 partial windows
// only see the ORF string (icm.cc:376-388) -- and prefix-summed; heads[oi][k] = sum over j <= 3k+2 of
// (gene_j - indep_j), k < nh = (ja+1)/3, ja = first j >= W-2 with j % 3 == 2 (the anchor of k3_g3_emit).
template <int kHG>
__global__ void __launch_bounds__(128) k3_g3_heads(DevIcm gene, DevIcm indep, const uint64_t* __restrict__ words,
                                                   const int64_t* __restrict__ off, const gmg_orf* __restrict__ orfs,
                                                   const int32_t* __restrict__ orf_seq, int64_t n_orfs, DevParams P,
                                                   const int64_t* __restrict__ counts, int ja, double* __restrict__ heads) {
  constexpr unsigned FULL = 0xffffffffu;
  const int64_t oi = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / kHG;
  const int gl = threadIdx.x % kHG;
  const bool live = oi < n_orfs && counts[oi] > 0;
  double hs = 0.0;
  if (live) {
    const int32_t s = orf_seq[oi];
    const int64_t a = off[s];
    const G3Geom g = g3_geom(orfs[oi], (int)(off[s + 1] - a), P);
    if (gl <= ja && gl < g.len) {
      const bool fwd = g.frame > 0;
      const int f = (1 + gl) % 3, bound = fwd ? g.hi : g.lo;
      const int q = fwd ? g.hi - 1 - gl : g.lo + gl;
      const float xg = fwd ? icm_fwd(gene, words, a + q, q, bound, f) : icm_rev(gene, words, a + q, q, bound, f);
      float xn;
      if (gl >= 2) xn = fwd ? __ldg(indep.lut3 + f * 64 + (int)(gmg_extract32(words, a + q) & 63))
                            : __ldg(indep.lut3 + (3 + f) * 64 + (int)(gmg_extract32(words, a + q - 2) & 63));
      else xn = fwd ? icm_fwd(indep, words, a + q, q, bound, f) : icm_rev(indep, words, a + q, q, bound, f);
      hs = (double)xg - (double)xn;
    }
  }
#pragma unroll
  for (int d = 1; d < kHG; d <<= 1) {
    const double t = __shfl_up_sync(FULL, hs, d, kHG);
    if (gl >= d) hs += t;
  }
  if (live && gl <= ja && gl % 3 == 2) heads[(size_t)oi * ((ja + 1) / 3) + gl / 3] = hs;
}

// K2 (glimmer3 path): codon-boundary cumulative log-odds.
//
// Every start position js of every ORF needs score[js-1] = sum_{j < js} (gene_j - indep_j) along the ORF string
// (glimmer3.cc:1346-1371).  Past the first W-1 positions the terms are plain full-window values, i.e. K1 plane
// entries, and position p contributes to a forward ORF with the period (r - p) mod 3, r = (hi + a) mod 3 -- so
// there are only three forward and three reverse "streams" over the whole batch, and a start only ever asks
// for a stream's running sum at a position where the period is 0 (j mod 3 == 2): p mod 3 == r.  Hence every
// position is the boundary of exactly ONE forward and ONE reverse stream and 16 B/base hold all the sums:
//   CF[p] = sum of the forward stream p%3 over codon slots p, p+3, ... to the end of p's tile  (suffix sums)
//   CR[p] = sum of the reverse stream with boundary residue p%3 from the start of p's tile     (prefix sums)
// where the slot of boundary p is the three terms at p, p+1, p+2 (periods 0, 2, 1) forward and p, p-1, p-2
// (periods 0, 2, 1) reverse.  Sums restart at every tile of G3_TS codon slots, so tiles are independent CTAs;
// tileT[tile][6] keeps each stream's tile total.  An ORF's sums are differences / sums of these values; they
// carry the reference's bits because no addition can round (the static certificate of gmg_score_orfs_g3).
#define G3_TS 512  // codon slots (3 bases each) per tile = threads per CTA

__global__ void __launch_bounds__(G3_TS) k2_g3_codon_cum(const float* __restrict__ lut3,
                                                         const uint64_t* __restrict__ words, int64_t total,
                                                         const float* __restrict__ planes,
                                                         const uint32_t* __restrict__ bktidx,
                                                         double* __restrict__ cumc, int64_t tot3,
                                                         double* __restrict__ tileT) {
  constexpr int NW = G3_TS / 32;
  __shared__ float s_lut[384];
  __shared__ double s_wtot[6][NW];
  __shared__ double s_out[2][3 * G3_TS];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  for (int i = tid; i < 384; i += G3_TS) s_lut[i] = lut3[i];
  __syncthreads();
  const int64_t p0 = 3 * ((int64_t)blockIdx.x * G3_TS + tid);
  double u[3] = {0.0, 0.0, 0.0}, v[3] = {0.0, 0.0, 0.0};
  if (p0 - 2 < total) {
    const uint64_t win = gmg_extract32(words, p0 - 4);  // base b at bits 2 (b - p0 + 4)
    const size_t T = (size_t)total;
    // plane indices of the seven positions p0-2 .. p0+4 (they lie in at most two 32-base blocks)
    uint32_t pi[7];
    bool pv[7];
    {
      const int64_t nblk = (total + 31) >> 5;
      const int64_t P0 = p0 - 2;
      int64_t ba = P0 >> 5;
      ba = ba < 0 ? 0 : ba;
      int64_t bb = (P0 + 6) >> 5;
      bb = bb >= nblk ? nblk - 1 : bb;
      const uint64_t wa = __ldg(words + ba), wb = __ldg(words + bb);
      const uint4 ra = __ldg(reinterpret_cast<const uint4*>(bktidx) + ba), rb = __ldg(reinterpret_cast<const uint4*>(bktidx) + bb);
#pragma unroll
      for (int k = 0; k < 7; k++) {
        const int64_t p = P0 + k;
        pv[k] = p >= 0 && p < total;
        const bool ina = (p >> 5) <= ba;
        const uint64_t w = ina ? wa : wb;
        const uint4 r = ina ? ra : rb;
        const int i = (int)(p & 31);
        const unsigned bs = (unsigned)(w >> (2 * i)) & 3u;
        const uint64_t x = w ^ (0x5555555555555555ull * bs);
        const uint64_t eq = ~(x | (x >> 1)) & 0x5555555555555555ull & ((1ull << (2 * i)) - 1ull);
        pi[k] = (bs == 0 ? r.x : (bs == 1 ? r.y : (bs == 2 ? r.z : r.w))) + (uint32_t)__popcll(eq);
      }
    }
#pragma unroll
    for (int rho = 0; rho < 3; rho++) {
#pragma unroll
      for (int k = 0; k < 3; k++) {
        const int f = k == 0 ? 0 : (k == 1 ? 2 : 1);
        const int kf = rho + k + 2, kr = rho - k + 2;  // slots of pi[] of the forward / reverse term's position
        if (pv[kf])  // forward term at p0 + rho + k: window = bases pf, pf+1, pf+2
          u[rho] += (double)__ldg(planes + f * T + pi[kf]) - (double)s_lut[f * 64 + (int)((win >> (2 * (rho + k + 4))) & 63)];
        if (pv[kr])  // reverse term at p0 + rho - k: window = complement of bases pr-2, pr-1, pr
          v[rho] += (double)__ldg(planes + (3 + f) * T + pi[kr]) -
                    (double)s_lut[(3 + f) * 64 + (int)((win >> (2 * (rho - k + 2))) & 63)];
      }
    }
  }
  // warp level: suffix scans (forward streams), prefix scans (reverse streams)
#pragma unroll
  for (int rho = 0; rho < 3; rho++) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const double tu = __shfl_down_sync(0xffffffffu, u[rho], d), tv = __shfl_up_sync(0xffffffffu, v[rho], d);
      if (lane + d < 32) u[rho] += tu;
      if (lane >= d) v[rho] += tv;
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int rho = 0; rho < 3; rho++) s_wtot[rho][wid] = u[rho];
  }
  if (lane == 31) {
#pragma unroll
    for (int rho = 0; rho < 3; rho++) s_wtot[3 + rho][wid] = v[rho];
  }
  __syncthreads();
  // warp k < 6 turns the warp totals of stream k into exclusive offsets and writes the tile total
  if (wid < 6) {
    const bool fw = wid < 3;
    const double x = lane < NW ? s_wtot[wid][lane] : 0.0;
    double incl = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const double td = __shfl_down_sync(0xffffffffu, incl, d), tu = __shfl_up_sync(0xffffffffu, incl, d);
      if (fw && lane + d < 32) incl += td;
      if (!fw && lane >= d) incl += tu;
    }
    if (lane < NW) s_wtot[wid][lane] = incl - x;  // exclusive: warps after (forward) / before (reverse) this one
    const double tot = __shfl_sync(0xffffffffu, incl, fw ? 0 : 31);
    if (lane == 0) tileT[(size_t)blockIdx.x * 6 + wid] = tot;
  }
  __syncthreads();
#pragma unroll
  for (int rho = 0; rho < 3; rho++) {
    s_out[0][3 * tid + rho] = u[rho] + s_wtot[rho][wid];
    s_out[1][3 * tid + rho] = v[rho] + s_wtot[3 + rho][wid];
  }
  __syncthreads();
  const size_t o0 = (size_t)blockIdx.x * (3 * G3_TS);
#pragma unroll
  for (int i = 0; i < 3; i++) {
    cumc[o0 + i * G3_TS + tid] = s_out[0][i * G3_TS + tid];
    cumc[(size_t)tot3 + o0 + i * G3_TS + tid] = s_out[1][i * G3_TS + tid];
  }
}

// K3 (glimmer3) emit pass, kG lanes per ORF: every lane takes one 32-codon word of the ORF's start-bit range per
// step and writes the records of its set bits.  score[js-1] of a start is  H + (stream sum between the anchor
// position j = ja and j = js-1): H from k3_g3_heads, the stream sum read off k2_g3_codon_cum's tables -- two
// loads when both ends share a tile, plus the totals of the tiles in between otherwise.  Records are stored in
// generation order (descending js): forward ORFs walk their slots upwards, reverse ORFs downwards.
template <int kG>
__global__ void __launch_bounds__(128) k3_g3_emit(const uint64_t* __restrict__ words, const uint2* __restrict__ cb,
                                                  int64_t nwc, const int64_t* __restrict__ off,
                                                  const gmg_orf* __restrict__ orfs, const int32_t* __restrict__ orf_seq,
                                                  int64_t n_orfs, const double* __restrict__ cumc, int64_t tot3,
                                                  const double* __restrict__ tileT, const double* __restrict__ heads,
                                                  int ja, CodonSets cs, DevParams P,
                                                  const int64_t* __restrict__ start_off,
                                                  const int32_t* __restrict__ first_js, int exact_len,
                                                  gmg_start* __restrict__ starts) {
  constexpr unsigned FULL = 0xffffffffu;
  __shared__ unsigned char s_which[64];
  if (threadIdx.x < 64) s_which[threadIdx.x] = cs.which[threadIdx.x];
  __syncthreads();
  const int64_t oi = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / kG;
  const int gl = threadIdx.x % kG;
  int n_emit = 0;
  int64_t so = 0;
  if (oi < n_orfs && orfs[oi].orf_len <= exact_len) {  // longer ORFs: k3_g3_ordered
    so = start_off[oi];
    n_emit = (int)(start_off[oi + 1] - so);
  }
  const bool live = n_emit > 0;
  // per-ORF state (identical in the kG lanes of a group)
  G3Geom g;
  G3Range R;
  int64_t a = 0, s_first = 0, pa = 0, ta = 0;
  int first_j = 0, nwords = 0, strand = 0, rho = 0;
  bool fwd = true;
  double c_a = 0.0, t_a = 0.0, h_ja = 0.0;
  const double* hd = NULL;
  if (live) {
    first_j = first_js[oi];
    const int32_t s = orf_seq[oi];
    a = off[s];
    g = g3_geom(orfs[oi], (int)(off[s + 1] - a), P);
    R = g3_range(g, a, P);
    fwd = g.frame > 0;
    strand = fwd ? 0 : 1;
    // slots in generation order: from js = min(first_j, jmax) down to jmin
    const int jhi = min(first_j, R.jmax);
    s_first = fwd ? R.s0 - jhi / 3 : R.s0 + jhi / 3;
    const int64_t s_last = fwd ? R.s0 - R.jmin / 3 : R.s0 + R.jmin / 3;
    nwords = jhi >= R.jmin ? (int)(fwd ? (s_last >> 5) - (s_first >> 5) : (s_first >> 5) - (s_last >> 5)) + 1 : 0;
    hd = heads + (size_t)oi * ((ja + 1) / 3);
    if (first_j - 1 > ja) {
      pa = a + (fwd ? g.hi - 1 - ja : g.lo + ja);
      rho = (int)(pa % 3);
      ta = pa / (3 * G3_TS);
      c_a = __ldg(cumc + (size_t)strand * tot3 + pa);
      t_a = __ldg(tileT + (size_t)ta * 6 + strand * 3 + rho);
      h_ja = __ldg(hd + ja / 3);
    }
  }
  gmg_start* out = starts + so;
  int emitted = 0;
  // truncated rule: the first candidate position emits a which = -1 record whatever its codon
  const bool trunc_first = live && g.trunc;
  if (trunc_first) emitted = 1;
  const int64_t s_lo = live ? (fwd ? s_first : R.s0 + R.jmin / 3) : 0;
  const int64_t s_hi = live ? (fwd ? R.s0 - R.jmin / 3 : s_first) : 0;
  for (int wb = 0; __any_sync(FULL, wb < nwords); wb += kG) {
    const int wi = wb + gl;
    unsigned x = 0;
    int64_t w = 0;
    if (wi < nwords) {
      w = fwd ? (s_lo >> 5) + wi : (s_hi >> 5) - wi;
      x = __ldg(cb + (size_t)(fwd ? R.r : 3 + R.r) * nwc + w).x;
      if (w == (s_lo >> 5)) x &= ~0u << (int)(s_lo & 31);
      if (w == (s_hi >> 5)) x &= (2u << (int)(s_hi & 31)) - 1u;
    }
    const int cnt = __popc(x);
    int incl = cnt;
#pragma unroll
    for (int d = 1; d < kG; d <<= 1) {
      const int t = __shfl_up_sync(FULL, incl, d, kG);
      if (gl >= d) incl += t;
    }
    int slot = emitted + incl - cnt;
    while (x) {
      const int b = fwd ? __ffs(x) - 1 : 31 - __clz(x);
      x &= ~(1u << b);
      const int64_t sl = (w << 5) + b;
      const int js = (int)(fwd ? 3 * (R.s0 - sl) : 3 * (sl - R.s0));
      const int j = js - 1;
      double sc;
      if (j <= ja) {
        sc = __ldg(hd + j / 3);
      } else {
        const int64_t pj = a + (fwd ? g.hi - 1 - j : g.lo + j);
        const int64_t tj = pj / (3 * G3_TS);
        const double c_j = __ldg(cumc + (size_t)strand * tot3 + pj);
        if (tj == ta) {
          sc = h_ja + (c_j - c_a);
        } else {
          double qd = 0.0;  // totals of the tiles strictly between the anchor's and this start's
          if (fwd) for (int64_t t = ta - 1; t > tj; t--) qd += __ldg(tileT + (size_t)t * 6 + rho);
          else for (int64_t t = ta + 1; t < tj; t++) qd += __ldg(tileT + (size_t)t * 6 + 3 + rho);
          sc = h_ja + ((c_j + qd) + (t_a - c_a));
        }
      }
      // the start codon: S[c], S[c+1], S[c+2] forward / complement of S[c+2], S[c+1], S[c] reverse, c = 3 sl + r
      const int raw = (int)(gmg_extract32(words, 3 * sl + R.r) & 63);
      const int b0 = raw & 3, b1 = (raw >> 2) & 3, b2 = raw >> 4;
      const int code = fwd ? b0 * 16 + b1 * 4 + b2 : (3 - b2) * 16 + (3 - b1) * 4 + (3 - b0);
      const int which = s_which[code];
      const int m = g.len;
      const int kpos = fwd ? g.k0 + (m - 1 - js) : g.k0 - (m - 1 - js);
      Emit e;
      e.out = out;
      e.n = slot++;
      emit_start(e, js + 2, kpos, sc, which, 0, (js == first_j && !g.trunc) ? 1 : 0, 0, NULL, NULL, P.ignore_score_len);
    }
    emitted += __shfl_sync(FULL, incl, kG - 1, kG);
  }
  if (trunc_first && gl == 0) {
    const int js = first_j, j = js - 1;
    double sc;
    if (j <= ja) {
      sc = __ldg(hd + j / 3);
    } else {
      const int64_t pj = a + (fwd ? g.hi - 1 - j : g.lo + j);
      const int64_t tj = pj / (3 * G3_TS);
      const double c_j = __ldg(cumc + (size_t)strand * tot3 + pj);
      double qd = 0.0;
      if (fwd) for (int64_t t = ta - 1; t > tj; t--) qd += __ldg(tileT + (size_t)t * 6 + rho);
      else for (int64_t t = ta + 1; t < tj; t++) qd += __ldg(tileT + (size_t)t * 6 + 3 + rho);
      sc = tj == ta ? h_ja + (c_j - c_a) : h_ja + ((c_j + qd) + (t_a - c_a));
    }
    const int m = g.len;
    const int kpos = fwd ? g.k0 + (m - 1 - js) : g.k0 - (m - 1 - js);
    Emit e;
    e.out = out;
    e.n = 0;
    emit_start(e, js + 2, kpos, sc, -1, 1, 1, 0, NULL, NULL, P.ignore_score_len);
  }
}

// The reference's own association for every ORF (one warp each): used when the static exactness certificate
// of gmg_score_orfs_g3 does not hold for the model pair / sequence lengths at hand.
__global__ void __launch_bounds__(128) k3_g3_ordered(DevIcm gene, DevIcm indep, const uint64_t* __restrict__ words,
                                                     const int64_t* __restrict__ off, const gmg_orf* __restrict__ orfs,
                                                     const int32_t* __restrict__ orf_seq, int64_t n_orfs, int64_t total,
                                                     const float* __restrict__ planes,
                                                     const uint32_t* __restrict__ bktidx, CodonSets cs, DevParams P,
                                                     const int64_t* __restrict__ start_off,
                                                     const int32_t* __restrict__ first_js, int exact_len,
                                                     gmg_start* __restrict__ starts,
                                                     unsigned long long* __restrict__ n_ordered) {
  __shared__ float s_lut[384];
  if (indep.lut3)
    for (int i = threadIdx.x; i < 384; i += blockDim.x) s_lut[i] = indep.lut3[i];
  __syncthreads();
  const float* lut = indep.lut3 ? s_lut : NULL;
  const int64_t oi = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (oi >= n_orfs || orfs[oi].orf_len <= exact_len) return;
  if ((threadIdx.x & 31) == 0) atomicAdd(n_ordered, 1ull);
  const int64_t so = start_off[oi];
  const int n_emit = (int)(start_off[oi + 1] - so);
  if (n_emit == 0) return;
  const int32_t s = orf_seq[oi];
  const int64_t a = off[s];
  const G3Geom g = g3_geom(orfs[oi], (int)(off[s + 1] - a), P);
  const float* plane = planes + (size_t)(g.frame > 0 ? 0 : 3) * total;  // the strand's three period planes
  g3_accumulate_ordered(gene, indep, lut, words, a, g, plane, bktidx, total, cs, P, first_js[oi], n_emit, starts + so);
}

// ------------------------------------------------------------------------------------------------
// K2 (glimmer-mg -i / -s): per-sequence prefix sums, stop tables, quality synthesis, exactness certificate.
// One warp per sequence, every lane owns FOUR consecutive positions of a 128-position tile whose start is aligned to 4
// bases of the batch, so that a lane's four results of one array are one aligned 32-byte run (two 16-byte stores for
// doubles, one for the int32 stop tables, one 4-byte store for qualities) and its four plane indices share one block
// lookup.  Sums run serially inside the lane; one warp scan per class joins the 32 lane totals -- 6 FP64 scans per 128
// positions instead of the 24 of one position per lane -- and the independent model is the 384-entry full-window table
// (lut3) in shared memory except at the two end positions.
// Any association gives the reference's bits under the read's certificate: every term is a multiple of 2^g (g from the
// smallest float exponent among the read's terms), so while the sum of magnitudes stays below 2^(g+52) no partial sum
// can round.
#define K2_R 4
// c + i for c in 0..2, i in 0..3, reduced mod 3 without a division
__device__ __forceinline__ int k2_add3(int c, int i) {
  int t = c + i;
  t = t >= 3 ? t - 3 : t;
  return t >= 3 ? t - 3 : t;
}
// certificate inputs of one float term: smallest magnitude bits of the non-zero terms (its exponent field bounds the
// term's ulp: the value is an integer multiple of 2^(max(e,1) - 150)) and the running sum of magnitudes
__device__ __forceinline__ void k2_cert_term(float v, unsigned& umin, float& asum) {
  const unsigned u = __float_as_uint(v) & 0x7fffffffu;
  umin = min(umin, u ? u : 0x7fffffffu);
  asum += fabsf(v);
}

template <bool kPS>
__global__ void __launch_bounds__(128) k2_prefix_lanes(DevIcm indep_, IndepSeqs X, const uint64_t* __restrict__ words,
                                                       const int64_t* __restrict__ off, int64_t n_seq, int64_t total,
                                                       const float* __restrict__ planes, const uint32_t* __restrict__ bktidx,
                                                       CodonSets cs, DevParams P, const uint8_t* __restrict__ qual_in,
                                                       double* __restrict__ cum, int32_t* __restrict__ fwd_prev,
                                                       int32_t* __restrict__ rev_next, uint8_t* __restrict__ qual,
                                                       uint8_t* __restrict__ cert) {
  constexpr unsigned FULL = 0xffffffffu;
  constexpr int NONE_LO = -0x40000000, NONE_HI = 0x40000000;
  __shared__ float s_lut_sh[384];
  const bool have_lut = indep_.lut3 != NULL;
  if (!kPS && have_lut)
    for (int i = threadIdx.x; i < 384; i += blockDim.x) s_lut_sh[i] = indep_.lut3[i];
  __syncthreads();
  const int64_t s = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= n_seq) return;
  // per-sequence models (gmg_score_orfs_mg_gc): the sequence's own table, read through L1
  DevIcm own;  // kPS: the sequence's own model; the single-model form reads the kernel parameter
  if constexpr (kPS) own = indep_of(indep_, X, s);
  const DevIcm& indep = kPS ? own : indep_;
  const float* const s_lut = kPS ? indep.lut3 : s_lut_sh;
  const int64_t a = off[s];
  const int L = (int)(off[s + 1] - a);
  if (L == 0) {
    if (lane == 0) cert[s] = 1;
    return;
  }
  unsigned umin = 0x7fffffffu;
  float asum = 0.f;      // magnitudes of one tile (<= 48 terms per lane) ...
  double asum_d = 0.0;  // ... folded into FP64 tile by tile: a float sum over a long sequence would eat the margin
  const int shift = (int)(a & 3);  // tiles start at sequence position -shift: a + q0 is a multiple of 4
  const int ntile = (L + shift + 127) >> 7;
  const size_t T = (size_t)total;
  const float* const pf0 = planes;
  const float* const pf1 = planes + T;
  const float* const pf2 = planes + 2 * T;
  const float* const pr0 = planes + 3 * T;
  const float* const pr1 = planes + 4 * T;
  const float* const pr2 = planes + 5 * T;

  // ---- left to right: reverse-strand prefix sums, previous forward stops, quality ----
  {
    double carry[3] = {0.0, 0.0, 0.0};
    int last_stop[3] = {0, 1, -1};  // Save_Prev_Stops init (glimmer-mg.cc:684), by class q % 3
    for (int t = 0; t < ntile; t++) {
      const int q0 = t * 128 - shift + lane * K2_R;  // first of this lane's four positions
      double v[3][K2_R];
      int stp[K2_R];
      uint32_t qv4 = 0;
      uint64_t wblk = 0, win = 0;
      uint4 rblk = make_uint4(0, 0, 0, 0);
      const bool any_in = q0 + K2_R > 0 && q0 < L;
      if (any_in) {
        const int64_t blk = (a + q0) >> 5;
        wblk = __ldg(words + blk);
        rblk = __ldg(reinterpret_cast<const uint4*>(bktidx) + blk);
        win = gmg_extract32(words, a + q0 - 4);  // base a+q0-4+k at bits 2k
      }
      const int c0 = mod3(q0);          // class of position q0 + i is c0 + i (mod 3)
      const int rot0 = k2_add3(c0, 1);  // f of class c at q0 + i is rot0 + i - c (mod 3)
      const int bi0 = (int)((a + q0) & 31);
#pragma unroll
      for (int i = 0; i < K2_R; i++) {
        const int q = q0 + i;
        const bool in = q >= 0 && q < L;
        double d0 = 0.0, d1 = 0.0, d2 = 0.0;
        stp[i] = NONE_LO;
        if (in) {
          const int bi = bi0 + i;
          const unsigned bs = (unsigned)(wblk >> (2 * bi)) & 3u;
          const uint64_t xx = wblk ^ (0x5555555555555555ull * bs);
          const uint64_t eq = ~(xx | (xx >> 1)) & 0x5555555555555555ull & ((1ull << (2 * bi)) - 1ull);
          const uint32_t pi = (bs == 0 ? rblk.x : (bs == 1 ? rblk.y : (bs == 2 ? rblk.z : rblk.w))) + (uint32_t)__popcll(eq);
          const int raw_rev = (int)((win >> (2 * (i + 2))) & 63);  // bases q-2, q-1, q
          const float g0 = __ldg(pr0 + pi), g1 = __ldg(pr1 + pi), g2 = __ldg(pr2 + pi);
          float n0, n1, n2;
          if (have_lut && q >= 2) {
            n0 = s_lut[192 + raw_rev];
            n1 = s_lut[256 + raw_rev];
            n2 = s_lut[320 + raw_rev];
          } else if (have_lut) {  // q = 0, 1: two / one window positions missing
            const float* lp = indep.lutp + 384 + (1 - q) * 192 + raw_rev;
            n0 = __ldg(lp);
            n1 = __ldg(lp + 64);
            n2 = __ldg(lp + 128);
          } else {
            n0 = icm_rev(indep, words, a + q, q, 0, 0);
            n1 = icm_rev(indep, words, a + q, q, 0, 1);
            n2 = icm_rev(indep, words, a + q, q, 0, 2);
          }
          k2_cert_term(g0, umin, asum); k2_cert_term(g1, umin, asum); k2_cert_term(g2, umin, asum);
          k2_cert_term(n0, umin, asum); k2_cert_term(n1, umin, asum); k2_cert_term(n2, umin, asum);
          d0 = (double)g0 - (double)n0;
          d1 = (double)g1 - (double)n1;
          d2 = (double)g2 - (double)n2;
          if (q >= 2) {  // forward stop whose last base is q
            const int cd = ((raw_rev & 3) << 4) | (raw_rev & 12) | (raw_rev >> 4);
            if ((cs.stop_mask >> cd) & 1) stp[i] = q;
          }
          // Without a quality file, Set_Quality_454 (glimmer-mg.cc:1865-1906): last base of a homopolymer run of length
          // r gets 31 - 5*min(r,5), every other base 31.  With one, the file's values (already clamped to 0..255),
          // cleaned by Clean_Quality_454 (:519-546) under -i only, as main() does (:385-392): under -s alone they reach
          // Pass_Stop_Penalty as read.
          if (qual) {
            const int b = (int)bs;
            const bool last_of_run = (q == L - 1) || ((int)((win >> (2 * (i + 5))) & 3) != b);
            int qv;
            if (qual_in) {
              qv = qual_in[a + q];
              if (P.allow_indels) {
                if (qv <= 0) qv = 1;
                if (!last_of_run && qv < P.indel_q_thresh + 1) qv = P.indel_q_thresh + 1;
              }
            } else if (!last_of_run) {
              qv = 31;
            } else {
              int r = 1;
              while (r < 5 && q - r >= 0 && (int)((win >> (2 * (i + 4 - r))) & 3) == b) r++;
              qv = 31 - 5 * r;
            }
            qv4 |= (uint32_t)qv << (8 * i);
          }
        }
        // class c takes the term of period f = rot - c (mod 3), rot = rot0 + i
        const int rot = k2_add3(rot0, i);
        const double x0 = rot == 0 ? d0 : (rot == 1 ? d1 : d2);
        const double x1 = rot == 0 ? d2 : (rot == 1 ? d0 : d1);
        const double x2 = rot == 0 ? d1 : (rot == 1 ? d2 : d0);
        v[0][i] = (i ? v[0][i - 1] : 0.0) + x0;
        v[1][i] = (i ? v[1][i - 1] : 0.0) + x1;
        v[2][i] = (i ? v[2][i - 1] : 0.0) + x2;
      }
#pragma unroll
      for (int c = 0; c < 3; c++) {
        const double tot = v[c][K2_R - 1];
        double inc = tot;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const double tt = __shfl_up_sync(FULL, inc, d);
          if (lane >= d) inc += tt;
        }
        const double base = carry[c] + (inc - tot);
#pragma unroll
        for (int i = 0; i < K2_R; i++) v[c][i] += base;
        carry[c] += __shfl_sync(FULL, inc, 31);
      }
      // stop tables: running maximum per class inside the lane (classes relative to c0: position i has relative
      // class i % 3), lane summaries joined per absolute class by three int max-scans
      int rel[3] = {NONE_LO, NONE_LO, NONE_LO};
      int outp[K2_R];
#pragma unroll
      for (int i = 0; i < K2_R; i++) {
        rel[i % 3] = max(rel[i % 3], stp[i]);
        outp[i] = rel[i % 3];
      }
      // absolute class c is relative class c - c0 (mod 3)
      const int ab0 = c0 == 0 ? rel[0] : (c0 == 1 ? rel[2] : rel[1]);
      const int ab1 = c0 == 0 ? rel[1] : (c0 == 1 ? rel[0] : rel[2]);
      const int ab2 = c0 == 0 ? rel[2] : (c0 == 1 ? rel[1] : rel[0]);
      int ex[3];
      {
        int inc[3] = {ab0, ab1, ab2};
#pragma unroll
        for (int c = 0; c < 3; c++) {
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const int tt = __shfl_up_sync(FULL, inc[c], d);
            if (lane >= d) inc[c] = max(inc[c], tt);
          }
          int e = __shfl_up_sync(FULL, inc[c], 1);
          if (lane == 0) e = NONE_LO;
          ex[c] = e > NONE_LO ? e : last_stop[c];
          const int all = __shfl_sync(FULL, inc[c], 31);
          if (all > NONE_LO) last_stop[c] = all;
        }
      }
      // relative class r is absolute class c0 + r
      const int er0 = c0 == 0 ? ex[0] : (c0 == 1 ? ex[1] : ex[2]);
      const int er1 = c0 == 0 ? ex[1] : (c0 == 1 ? ex[2] : ex[0]);
      const int er2 = c0 == 0 ? ex[2] : (c0 == 1 ? ex[0] : ex[1]);
#pragma unroll
      for (int i = 0; i < K2_R; i++)
        if (outp[i] <= NONE_LO) outp[i] = (i % 3) == 0 ? er0 : ((i % 3) == 1 ? er1 : er2);
      // stores: a lane's four positions are one aligned run
      if (q0 >= 0 && q0 + K2_R <= L) {
#pragma unroll
        for (int c = 0; c < 3; c++) {
          double* d1p = cum + (size_t)(3 + c) * T + a + q0;
          if (((uintptr_t)d1p & 15) == 0) {
            reinterpret_cast<double2*>(d1p)[0] = make_double2(v[c][0], v[c][1]);
            reinterpret_cast<double2*>(d1p)[1] = make_double2(v[c][2], v[c][3]);
          } else {
            d1p[0] = v[c][0]; d1p[1] = v[c][1]; d1p[2] = v[c][2]; d1p[3] = v[c][3];
          }
        }
        int32_t* p1 = fwd_prev + a + q0;
        if (((uintptr_t)p1 & 15) == 0) *reinterpret_cast<int4*>(p1) = make_int4(outp[0], outp[1], outp[2], outp[3]);
        else { p1[0] = outp[0]; p1[1] = outp[1]; p1[2] = outp[2]; p1[3] = outp[3]; }
        if (qual) {
          uint8_t* u1 = qual + a + q0;
          if (((uintptr_t)u1 & 3) == 0) *reinterpret_cast<uint32_t*>(u1) = qv4;
          else { u1[0] = (uint8_t)qv4; u1[1] = (uint8_t)(qv4 >> 8); u1[2] = (uint8_t)(qv4 >> 16); u1[3] = (uint8_t)(qv4 >> 24); }
        }
      } else if (any_in) {
#pragma unroll
        for (int i = 0; i < K2_R; i++) {
          const int q = q0 + i;
          if (q >= 0 && q < L) {
#pragma unroll
            for (int c = 0; c < 3; c++) cum[(size_t)(3 + c) * T + a + q] = v[c][i];
            fwd_prev[a + q] = outp[i];
            if (qual) qual[a + q] = (uint8_t)(qv4 >> (8 * i));
          }
        }
      }
      asum_d += (double)asum;
      asum = 0.f;
    }
  }
  // ---- right to left: forward-strand suffix sums, next reverse stops ----
  {
    double carry[3] = {0.0, 0.0, 0.0};
    // Save_Prev_Stops reverse init (glimmer-mg.cc:706-708) by class r = (L-1-q) % 3: {L-1, L-2, L}
    int next_stop[3] = {L - 1, L - 2, L};
    for (int t = ntile - 1; t >= 0; t--) {
      const int q0 = t * 128 - shift + (31 - lane) * K2_R;  // lane 0 owns the rightmost four positions
      double v[3][K2_R];
      int stp[K2_R];
      uint64_t wblk = 0, win = 0;
      uint4 rblk = make_uint4(0, 0, 0, 0);
      const bool any_in = q0 + K2_R > 0 && q0 < L;
      if (any_in) {
        const int64_t blk = (a + q0) >> 5;
        wblk = __ldg(words + blk);
        rblk = __ldg(reinterpret_cast<const uint4*>(bktidx) + blk);
        win = gmg_extract32(words, a + q0);  // base a+q0+k at bits 2k
      }
      // f of class c at position q is c - q (mod 3); at q0 + 3 (the lane's rightmost): rotr = -(q0 + 3) = -q0 (mod 3)
      const int nq0 = mod3(-q0);
      const int bi0 = (int)((a + q0) & 31);
#pragma unroll
      for (int ii = 0; ii < K2_R; ii++) {
        const int i = K2_R - 1 - ii;  // right to left inside the lane
        const int q = q0 + i;
        const bool in = q >= 0 && q < L;
        double d0 = 0.0, d1 = 0.0, d2 = 0.0;
        stp[i] = NONE_HI;
        if (in) {
          const int bi = bi0 + i;
          const unsigned bs = (unsigned)(wblk >> (2 * bi)) & 3u;
          const uint64_t xx = wblk ^ (0x5555555555555555ull * bs);
          const uint64_t eq = ~(xx | (xx >> 1)) & 0x5555555555555555ull & ((1ull << (2 * bi)) - 1ull);
          const uint32_t pi = (bs == 0 ? rblk.x : (bs == 1 ? rblk.y : (bs == 2 ? rblk.z : rblk.w))) + (uint32_t)__popcll(eq);
          const int raw_fwd = (int)((win >> (2 * i)) & 63);  // bases q, q+1, q+2
          const float g0 = __ldg(pf0 + pi), g1 = __ldg(pf1 + pi), g2 = __ldg(pf2 + pi);
          float n0, n1, n2;
          if (have_lut && q <= L - 3) {
            n0 = s_lut[raw_fwd];
            n1 = s_lut[64 + raw_fwd];
            n2 = s_lut[128 + raw_fwd];
          } else if (have_lut) {  // q = L-2, L-1: one / two window positions missing
            const float* lp = indep.lutp + (q - (L - 2)) * 192 + raw_fwd;
            n0 = __ldg(lp);
            n1 = __ldg(lp + 64);
            n2 = __ldg(lp + 128);
          } else {
            n0 = icm_fwd(indep, words, a + q, q, L, 0);
            n1 = icm_fwd(indep, words, a + q, q, L, 1);
            n2 = icm_fwd(indep, words, a + q, q, L, 2);
          }
          k2_cert_term(g0, umin, asum); k2_cert_term(g1, umin, asum); k2_cert_term(g2, umin, asum);
          k2_cert_term(n0, umin, asum); k2_cert_term(n1, umin, asum); k2_cert_term(n2, umin, asum);
          d0 = (double)g0 - (double)n0;
          d1 = (double)g1 - (double)n1;
          d2 = (double)g2 - (double)n2;
          if (q <= L - 3) {  // reverse-strand stop occupying q, q+1, q+2
            const int cc = 63 - (((raw_fwd & 3) << 4) | (raw_fwd & 12) | (raw_fwd >> 4));
            const int cd = ((cc & 3) << 4) | (cc & 12) | (cc >> 4);
            if ((cs.stop_mask >> cd) & 1) stp[i] = q;
          }
        }
        // class c takes f = c - q = c + nq0 - i (mod 3): with m = nq0 - i (mod 3), x_c = d[(c + m) % 3]
        const int m = k2_add3(nq0, 3 - (i % 3));
        const double x0 = m == 0 ? d0 : (m == 1 ? d1 : d2);
        const double x1 = m == 0 ? d1 : (m == 1 ? d2 : d0);
        const double x2 = m == 0 ? d2 : (m == 1 ? d0 : d1);
        v[0][i] = (ii ? v[0][i + 1] : 0.0) + x0;
        v[1][i] = (ii ? v[1][i + 1] : 0.0) + x1;
        v[2][i] = (ii ? v[2][i + 1] : 0.0) + x2;
      }
#pragma unroll
      for (int c = 0; c < 3; c++) {
        const double tot = v[c][0];
        double inc = tot;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const double tt = __shfl_up_sync(FULL, inc, d);
          if (lane >= d) inc += tt;
        }
        const double base = carry[c] + (inc - tot);
#pragma unroll
        for (int i = 0; i < K2_R; i++) v[c][i] += base;
        carry[c] += __shfl_sync(FULL, inc, 31);
      }
      // next reverse stop per class r = (L-1-q) % 3: running minimum from the right.  Relative class of the
      // ii-th position from the right is ii % 3; absolute class = r3 + ii, r3 = class of the rightmost position.
      const int r3 = mod3(L - 1 - (q0 + K2_R - 1));
      int rel[3] = {NONE_HI, NONE_HI, NONE_HI};
      int outp[K2_R];
#pragma unroll
      for (int ii = 0; ii < K2_R; ii++) {
        const int i = K2_R - 1 - ii;
        rel[ii % 3] = min(rel[ii % 3], stp[i]);
        outp[i] = rel[ii % 3];
      }
      const int ab0 = r3 == 0 ? rel[0] : (r3 == 1 ? rel[2] : rel[1]);
      const int ab1 = r3 == 0 ? rel[1] : (r3 == 1 ? rel[0] : rel[2]);
      const int ab2 = r3 == 0 ? rel[2] : (r3 == 1 ? rel[1] : rel[0]);
      int ex[3];
      {
        int inc[3] = {ab0, ab1, ab2};
#pragma unroll
        for (int c = 0; c < 3; c++) {
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const int tt = __shfl_up_sync(FULL, inc[c], d);
            if (lane >= d) inc[c] = min(inc[c], tt);
          }
          int e = __shfl_up_sync(FULL, inc[c], 1);
          if (lane == 0) e = NONE_HI;
          ex[c] = e < NONE_HI ? e : next_stop[c];
          const int all = __shfl_sync(FULL, inc[c], 31);
          if (all < NONE_HI) next_stop[c] = all;
        }
      }
      const int er0 = r3 == 0 ? ex[0] : (r3 == 1 ? ex[1] : ex[2]);
      const int er1 = r3 == 0 ? ex[1] : (r3 == 1 ? ex[2] : ex[0]);
      const int er2 = r3 == 0 ? ex[2] : (r3 == 1 ? ex[0] : ex[1]);
#pragma unroll
      for (int ii = 0; ii < K2_R; ii++) {
        const int i = K2_R - 1 - ii;
        if (outp[i] >= NONE_HI) outp[i] = (ii % 3) == 0 ? er0 : ((ii % 3) == 1 ? er1 : er2);
      }
      if (q0 >= 0 && q0 + K2_R <= L) {
#pragma unroll
        for (int c = 0; c < 3; c++) {
          double* d1p = cum + (size_t)c * T + a + q0;
          if (((uintptr_t)d1p & 15) == 0) {
            reinterpret_cast<double2*>(d1p)[0] = make_double2(v[c][0], v[c][1]);
            reinterpret_cast<double2*>(d1p)[1] = make_double2(v[c][2], v[c][3]);
          } else {
            d1p[0] = v[c][0]; d1p[1] = v[c][1]; d1p[2] = v[c][2]; d1p[3] = v[c][3];
          }
        }
        int32_t* p1 = rev_next + a + q0;
        if (((uintptr_t)p1 & 15) == 0) *reinterpret_cast<int4*>(p1) = make_int4(outp[0], outp[1], outp[2], outp[3]);
        else { p1[0] = outp[0]; p1[1] = outp[1]; p1[2] = outp[2]; p1[3] = outp[3]; }
      } else if (any_in) {
#pragma unroll
        for (int i = 0; i < K2_R; i++) {
          const int q = q0 + i;
          if (q >= 0 && q < L) {
#pragma unroll
            for (int c = 0; c < 3; c++) cum[(size_t)c * T + a + q] = v[c][i];
            rev_next[a + q] = outp[i];
          }
        }
      }
      asum_d += (double)asum;
      asum = 0.f;
    }
  }
  // ---- certificate: every term is a multiple of 2^g, g from the smallest float exponent seen; every partial sum
  // of any association is bounded by the sum of magnitudes (accumulated in FP32, 0.1 % margin for its rounding) ----
  for (int d = 16; d > 0; d >>= 1) {
    umin = min(umin, __shfl_xor_sync(FULL, umin, d));
    asum_d += __shfl_xor_sync(FULL, asum_d, d);
  }
  if (lane == 0) {
    const int e = (int)(umin >> 23);
    const int g = (e > 0 ? e : 1) - 150;
    bool ok = (umin == 0x7fffffffu) || (asum_d * 1.001 < ldexp(1.0, g + 52));
    cert[s] = ok ? 1 : 0;
  }
}

// ------------------------------------------------------------------------------------------------
// K3 (glimmer-mg): Score_Orf_Starts / Score_Indels / Pass_Stop_Penalty recursion, one thread per ORF,
// explicit stack (depth <= 1 + indel_max + sub).  score[j] of any branch is a difference of two entries of
// the K2 prefix-sum planes (bit-identical to the reference's serial Cumulative_Frame_Score whenever the
// sequence's certificate holds -- see DESIGN.md).

struct MgSeq {
  const uint64_t* words;
  int64_t a;
  int L;
  int64_t total;
  const double* cum;
  const int32_t* fwd_prev;
  const int32_t* rev_next;
  const uint8_t* qual;
  const double* penalty;   // [256] log(pe/2) - log(1-pe), pe = 10^(-q/10)   (host glibc, Score_Indels :1520-1521)
  const double* stop_pen;  // [4]   Pass_Stop_Penalty without a quality file, index = 2*a1 + a2
  const double* codon_p;   // [256] 1 - 10^(-q/10)
  const double* sub_pen;   // [n_orfs] Pass_Stop_Penalty of every root call with a quality file (log taken on the host)
  // ordered mode (sequences whose exactness certificate failed): score[] of a call is re-summed in the reference's
  // own order from the six Frame_Scores rows instead of read off the prefix sums
  int ordered;
  const float* planes;
  const uint32_t* bktidx;
  DevIcm indep;
};

// Frame_Scores[plane][q] (Score_All_Frames glimmer-mg.cc:1468-1510): gene - indep in FP64
__device__ double mg_frame_score_at(const MgSeq& S, int plane, int q) {
  if (q < 0 || q >= S.L) return 0.0;
  const int64_t p = S.a + q;
  const float g = S.planes[(size_t)plane * S.total + gmg_plane_index(S.words, S.bktidx, p)];
  const float n = plane < 3 ? icm_fwd(S.indep, S.words, p, q, S.L, plane) : icm_rev(S.indep, S.words, p, q, 0, plane - 3);
  return (double)g - (double)n;
}

struct MgCall {
  int lo, hi, m;       // geometry of this call (1-based lo/hi as in the reference)
  int j;               // loop cursor
  int phase;           // 0: before deletion branch, 1: before insertion branch, 2: codon test
  int suffix_j;
  int first_pos;
  int trunc;
  int n_err;
  int err_pos[2], err_type[2];
  double suffix_score;
  double cbase;        // cumulative value subtracted to get score[] of this call
};

__device__ __forceinline__ double mg_cum_f(const MgSeq& S, int c, int q) {  // suffix sum from q (0 past the end)
  return (q >= S.L || q < 0) ? 0.0 : S.cum[(size_t)c * S.total + S.a + q];
}
__device__ __forceinline__ double mg_cum_r(const MgSeq& S, int c, int q) {  // prefix sum through q (0 before 0)
  return (q < 0 || q >= S.L) ? 0.0 : S.cum[(size_t)(3 + c) * S.total + S.a + q];
}

// score[j] of a call (Cumulative_Frame_Score glimmer-mg.cc:561-604)
__device__ __forceinline__ double mg_score(const MgSeq& S, int frame, const MgCall& c, int j) {
  if (S.ordered) {  // Cumulative_Frame_Score (glimmer-mg.cc:561-604), term by term from the call's end
    double cum_score = 0.0;
    int f = 1, si = frame > 0 ? c.hi - 1 : c.lo - 1;
    for (int i = 0; i <= j; i++) {
      cum_score = cum_score + mg_frame_score_at(S, frame > 0 ? f : 3 + f, si);
      si += frame > 0 ? -1 : 1;
      f = f == 2 ? 0 : f + 1;
    }
    return cum_score;
  }
  if (frame > 0) {
    const int cls = mod3(c.hi);
    return mg_cum_f(S, cls, c.hi - 1 - j) - c.cbase;
  } else {
    const int cls = mod3(c.lo - 1);
    return mg_cum_r(S, cls, c.lo - 1 + j) - c.cbase;
  }
}

__device__ __forceinline__ void mg_open_call(const MgSeq& S, const DevParams& P, int frame, int end_point,
                                             MgCall& c) {
  const int L = S.L;
  if (frame > 0) {
    c.hi = end_point;
    const int e = end_point - 1;
    c.lo = ((e >= 0 && e < L) ? S.fwd_prev[S.a + e] : e) + 1;
    c.m = c.hi - c.lo;
    c.trunc = (c.lo < 3 && P.allow_truncated);
    c.cbase = mg_cum_f(S, mod3(c.hi), c.hi);
  } else {
    c.lo = end_point;
    const int e = end_point - 1;
    c.hi = ((e >= 0 && e < L) ? S.rev_next[S.a + e] : e) + 1;
    c.m = c.hi - c.lo;
    c.trunc = (L - (c.hi - 1) < 3 && P.allow_truncated);
    c.cbase = mg_cum_r(S, mod3(c.lo - 1), c.lo - 2);
  }
  if (c.m < 0) c.m = 0;
  c.j = c.m - 1;
  c.phase = 0;
  c.first_pos = 0;
}

__device__ double mg_pass_stop_penalty(const MgSeq& S, const DevParams& P, int frame, int lo, int hi, int64_t oi) {
  if (S.sub_pen) return S.sub_pen[oi];  // quality file: p_stop from the device, its log-odds from the host (glibc)
  int i0, i1, i2;
  if (frame > 0) { i0 = lo - 3; i1 = lo - 2; i2 = lo - 1; }
  else { i0 = hi + 1; i1 = hi; i2 = hi - 1; }
  const int want = (frame > 0) ? 0 : 3;  // 'a' forward, 't' reverse
  const bool a1 = (i1 >= 0 && i1 < S.L) && gmg_base_at(S.words, S.a + i1) == want;
  const bool a2 = (i2 >= 0 && i2 < S.L) && gmg_base_at(S.words, S.a + i2) == want;
  if (!P.have_quality_file) return S.stop_pen[2 * (int)a1 + (int)a2];
  double cp[3];
  const int idx[3] = {i0, i1, i2};
  for (int t = 0; t < 3; t++) cp[t] = (idx[t] >= 0 && idx[t] < S.L) ? S.codon_p[S.qual[S.a + idx[t]]] : 0.999;
  double p_stop = cp[0];
  p_stop *= a1 ? (2.0 / 3.0 * cp[1] + 1.0 / 3.0) : cp[1];
  p_stop *= a2 ? (2.0 / 3.0 * cp[2] + 1.0 / 3.0) : cp[2];
  return log(1.0 - p_stop) - log(p_stop);
}

__device__ void mg_orf_starts(const MgSeq& S, const DevParams& P, const CodonSets& cs, const gmg_orf& o, int64_t oi, Emit& e) {
  const int frame = o.frame;
  const int lowest_j = min(3, P.min_gene_len - 3);
  MgCall st[5];
  int sp = 0;
  mg_open_call(S, P, frame, frame > 0 ? o.stop_position - 1 : o.stop_position + 3, st[0]);
  st[0].suffix_score = 0.0;
  st[0].suffix_j = 0;
  st[0].n_err = 0;
  bool fresh = true;  // the call on top of the stack has not run its substitution pre-step yet
  while (sp >= 0) {
    MgCall& c = st[sp];
    if (fresh) {
      fresh = false;
      // substitution through the previous stop (glimmer-mg.cc:1771-1806)
      if (P.allow_subs && c.n_err < 1) {
        int eep, epos;
        if (frame > 0) { eep = c.lo - 3; epos = c.lo - 2; }
        else { eep = c.hi + 3; epos = c.hi + 2; }
        if (eep >= 0 && eep - 2 < S.L) {
          double ess = c.suffix_score + mg_pass_stop_penalty(S, P, frame, c.lo, c.hi, oi);
          if (c.m > 0) ess += mg_score(S, frame, c, c.m - 1) - 0.0;
          MgCall& nc = st[sp + 1];
          mg_open_call(S, P, frame, eep, nc);
          nc.suffix_score = ess;
          nc.suffix_j = c.suffix_j + c.m;
          nc.n_err = c.n_err + 1;
          nc.err_pos[0] = c.err_pos[0]; nc.err_type[0] = c.err_type[0];
          nc.err_pos[c.n_err] = epos;
          nc.err_type[c.n_err] = 2;
          sp++;
          fresh = true;
          continue;
        }
      }
    }
    if (c.j < lowest_j) {
      sp--;
      continue;
    }
    const int j = c.j;
    const int k = (frame > 0) ? c.lo + c.m - 2 - j : c.lo + j + 2;
    const int bidx = (frame > 0) ? c.hi - 1 - j : c.lo - 1 + j;
    if (c.phase < 2) {
      bool branch = false;
      if (P.allow_indels && c.n_err < P.indel_max) {
        const int qv = S.qual[S.a + bidx];
        if (qv <= P.indel_q_thresh) {
          const double pen = S.penalty[qv];
          const int esj = c.suffix_j + j + 2 - (j % 3);
          while (c.phase < 2 && !branch) {
            const int ph = c.phase++;
            const double ess = c.suffix_score + mg_score(S, frame, c, ph == 0 ? j : j - 1) - 0.0 + pen;
            if (ess > P.indel_suffix_thresh) {
              int eep, epos;
              if (ph == 0) {  // deletion
                eep = (frame > 0) ? k + (j % 3) : k - (j % 3);
                epos = (frame > 0) ? k + 3 : k - 1;
              } else {        // insertion
                eep = (frame > 0) ? k - (2 - (j % 3)) : k + 2 - (j % 3);
                epos = (frame > 0) ? k + 2 : k - 2;
              }
              MgCall& nc = st[sp + 1];
              mg_open_call(S, P, frame, eep, nc);
              nc.suffix_score = ess;
              nc.suffix_j = esj;
              nc.n_err = c.n_err + 1;
              nc.err_pos[0] = c.err_pos[0]; nc.err_type[0] = c.err_type[0];
              nc.err_pos[c.n_err] = epos;
              nc.err_type[c.n_err] = (ph == 0) ? 1 : 0;
              branch = true;
            }
          }
        }
      }
      if (branch) {
        sp++;
        fresh = true;
        continue;
      }
      c.phase = 2;
    }
    // codon test at j (glimmer-mg.cc:1819-1856)
    if (j % 3 == 0) {
      int which = -1;
      if (j <= c.m - 3) {
        const int cd = (frame > 0) ? codon_fwd_ending_at(S.words, S.a, bidx) : codon_rev_starting_at(S.words, S.a, bidx);
        if ((cs.start_mask >> cd) & 1) which = cs.which[cd];
      }
      if ((which >= 0 || (c.first_pos == 0 && c.trunc)) && j + 3 + c.suffix_j >= P.min_gene_len) {
        const double sc = (mg_score(S, frame, c, j - 1) - 0.0) + c.suffix_score;
        int first = (c.first_pos == 0);
        if (which >= 0 && c.first_pos == 0 && c.trunc) {
          emit_start(e, j + 2 + c.suffix_j, k, sc, -1, 1, first, c.n_err, c.err_pos, c.err_type, P.ignore_score_len);
          first = 0;
        }
        emit_start(e, j + 2 + c.suffix_j, k, sc, which, which < 0, first, c.n_err, c.err_pos, c.err_type,
                   P.ignore_score_len);
        if (c.first_pos == 0) c.first_pos = k;
      }
    }
    c.j--;
    c.phase = 0;
  }
}

// One thread per ORF: the recursion as the reference runs it (explicit stack).  Used for read sets without error
// branches (plain glimmer-mg: one short linear walk per ORF) and, with kOnlyUncert, as the ORDERED path of the
// sequences whose FP64 exactness certificate failed in K2 (their sums are re-formed in the reference's own order).
template <bool kWrite, bool kPS>
__global__ void __launch_bounds__(128) k3_mg_starts(MgfBatch B, int64_t n_orfs, const gmg_orf* __restrict__ orfs,
                                                    const int32_t* __restrict__ orf_seq, CodonSets cs, DevParams P,
                                                    int only_uncert, const float* __restrict__ planes,
                                                    const uint32_t* __restrict__ bktidx, DevIcm indep, IndepSeqs X,
                                                    int64_t* __restrict__ counts, const int64_t* __restrict__ start_off,
                                                    gmg_start* __restrict__ starts) {
  const int64_t oi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (oi >= n_orfs) return;
  const int32_t s = orf_seq[oi];
  const bool uncert = B.cert != NULL && B.cert[s] == 0;
  if (only_uncert && !uncert) return;
  MgSeq S;
  S.words = B.words;
  S.a = B.off[s];
  S.L = (int)(B.off[s + 1] - S.a);
  S.total = B.total;
  S.cum = B.cum;
  S.fwd_prev = B.fwd_prev;
  S.rev_next = B.rev_next;
  S.qual = B.qual;
  S.penalty = B.tables;
  S.stop_pen = B.tables + 256;
  S.codon_p = B.tables + 260;
  S.sub_pen = B.sub_pen;
  S.ordered = uncert ? 1 : 0;
  S.planes = planes;
  S.bktidx = bktidx;
  S.indep = kPS ? indep_of(indep, X, s) : indep;
  Emit e;
  e.out = kWrite ? starts + start_off[oi] : NULL;
  e.n = 0;
  if constexpr (kPS) {  // the sequence's own Ignore_Score_Len
    DevParams Ps = P;
    Ps.ignore_score_len = __ldg(X.isl + s);
    mg_orf_starts(S, Ps, cs, orfs[oi], oi, e);
  } else {
    mg_orf_starts(S, P, cs, orfs[oi], oi, e);
  }
  if (!kWrite) counts[oi] = e.n;
}

// ------------------------------------------------------------------------------------------------
// K3 (glimmer-mg), flat form (the default for -i / -s): the reference's recursion enumerated level by level with
// one thread per CANDIDATE call, see gmg_mg_flat.cuh for the passes.  The kernels below only map a thread to an
// item; the bodies are the __host__ __device__ functions of that header (tests/test_mgflat_host.py runs them
// on the host against the CPU checker, the start-list parity tests run them on the device).

// gates: positions whose quality allows an indel branch (Score_Orf_Starts glimmer-mg.cc:1816)
__global__ void __launch_bounds__(256) k_gate_bits(const uint8_t* __restrict__ qual, int64_t total, int thresh, int64_t nblk,
                                                   uint32_t* __restrict__ bits, uint32_t* __restrict__ cnt) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nblk) return;
  uint32_t m = 0;
  const int64_t p0 = w << 5;
  if (p0 + 32 <= total) {
    const uint4* q4 = reinterpret_cast<const uint4*>(qual + p0);
    const uint4 x = __ldg(q4), y = __ldg(q4 + 1);
    const uint32_t v[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
#pragma unroll
    for (int k = 0; k < 8; k++)
#pragma unroll
      for (int b = 0; b < 4; b++) m |= (uint32_t)((int)((v[k] >> (8 * b)) & 255u) <= thresh) << (4 * k + b);
  } else {
    for (int i = 0; i < 32 && p0 + i < total; i++) m |= (uint32_t)((int)qual[p0 + i] <= thresh) << i;
  }
  bits[w] = m;
  cnt[w] = (uint32_t)__popc(m);
}
__global__ void __launch_bounds__(256) k_gate_pos(const uint32_t* __restrict__ bits, const uint32_t* __restrict__ rank, int64_t nblk,
                                                  uint32_t* __restrict__ pos) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nblk) return;
  uint32_t m = bits[w], r = rank[w];
  while (m) {
    const int b = __ffs(m) - 1;
    m &= m - 1;
    pos[r++] = (uint32_t)(w << 5) + (uint32_t)b;
  }
}

// Pass_Stop_Penalty with a quality file: the stop probability of every root call (the host takes the logs)
__global__ void __launch_bounds__(128) k_mg_sub_pstop(MgfBatch B, DevParams P, const gmg_orf* __restrict__ orfs,
                                                      const int32_t* __restrict__ orf_seq, uint32_t n_orfs, double* __restrict__ pstop) {
  const uint32_t o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= n_orfs) return;
  const MgfSeq S = mgf_seq_of(B, orf_seq[o]);
  const bool fwd = orfs[o].frame > 0;
  int lo, hi;
  mgf_open(B, S, fwd, fwd ? orfs[o].stop_position - 1 : orfs[o].stop_position + 3, &lo, &hi);
  pstop[o] = mgf_stop_pstop(B, S, fwd, lo, hi);
}

__global__ void __launch_bounds__(128) k_mgf_a(MgfBatch B, DevParams P, MgfWork W) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < W.n_orfs) mgf_pass_a(B, P, W, i);
}
__global__ void __launch_bounds__(256) k_mgf_fill(const uint32_t* __restrict__ off, uint32_t n, uint32_t* __restrict__ par) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < n) mgf_fill_parent(off, p, par);
}
__global__ void __launch_bounds__(128) k_mgf_b(MgfBatch B, DevParams P, MgfWork W) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < W.c1) mgf_pass_b(B, P, W, i);
}
__global__ void __launch_bounds__(128) k_mgf_c(MgfBatch B, DevParams P, MgfWork W) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < W.c2) mgf_pass_c(B, P, W, i);
}
__global__ void __launch_bounds__(256) k_mgf_d(MgfWork W) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < W.c1) mgf_pass_d(W, i);
}
__global__ void __launch_bounds__(256) k_mgf_e(MgfWork W) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < W.n_orfs) mgf_pass_e(W, i);
}
// the write passes set the records' long-ORF boost: with per-sequence ignore lengths (kPS) each thread takes its own
__device__ __forceinline__ DevParams mgf_params_of(const DevParams& P, const IndepSeqs& X, int32_t s) {
  DevParams Ps = P;
  Ps.ignore_score_len = __ldg(X.isl + s);
  return Ps;
}
template <bool kPS>
__global__ void __launch_bounds__(128) k_mgf_w0(MgfBatch B, DevParams P, CodonSets cs, MgfWork W, IndepSeqs X) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= W.n_orfs) return;
  if constexpr (kPS) mgf_write_0(B, mgf_params_of(P, X, W.orf_seq[i]), cs, W, i);
  else mgf_write_0(B, P, cs, W, i);
}
template <bool kPS>
__global__ void __launch_bounds__(128) k_mgf_w1(MgfBatch B, DevParams P, CodonSets cs, MgfWork W, IndepSeqs X) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= W.c1) return;
  if constexpr (kPS) {
    if (!W.call1[i].ok) return;  // (mgf_write_1's own test) the ORF of a call that does not exist is not set
    mgf_write_1(B, mgf_params_of(P, X, W.orf_seq[W.call1[i].orf]), cs, W, i);
  } else {
    mgf_write_1(B, P, cs, W, i);
  }
}
template <bool kPS>
__global__ void __launch_bounds__(128) k_mgf_w2(MgfBatch B, DevParams P, CodonSets cs, MgfWork W, IndepSeqs X) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= W.c2) return;
  if constexpr (kPS) mgf_write_2(B, mgf_params_of(P, X, W.orf_seq[W.call1[W.par2[i]].orf]), cs, W, i);
  else mgf_write_2(B, P, cs, W, i);
}

// test hook (GMG_MG_FORCE_UNCERT=k): withdraw the certificate of every k-th sequence so that the ordered path runs
__global__ void k_force_uncert(uint8_t* __restrict__ cert, int64_t n, int k) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && i % k == 0) cert[i] = 0;
}

static int exclusive_sum_u32(gmg_ctx* ctx, const uint32_t* d_in, uint32_t* d_out, int64_t n) {
  size_t tmp_bytes = 0;
  GMG_CUDA(cub::DeviceScan::ExclusiveSum(NULL, tmp_bytes, d_in, d_out, n, ctx->stream));
  void* tmp;
  if (gmg_scratch(ctx, SCR_TMP4, tmp_bytes, &tmp)) return 1;
  GMG_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, d_in, d_out, n, ctx->stream));
  ctx->launches += 2;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// K2 + K3 (glimmer-mg) FUSED for read sets without error branches (plain glimmer-mg, BASELINE configs[4]): the
// segmented prefix sums of Cumulative_Frame_Score (glimmer-mg.cc:561-604) are formed only over the ORFs -- one warp
// per ORF, the terms gene - indep straight from the K1 planes, codon-boundary prefixes kept in shared memory -- and
// the ORF's start records are written from them in the same kernel.  Without indel / substitution branches every
// call is a root call, so the six whole-read prefix planes (48 B/base), the stop tables and the qualities that K2
// materialises for the branching modes are never needed: 1.3 ms of K2 + K3 per 31 Mbp become one 0.1 ms-class pass.
// Exactness: the static certificate of the model pair (as in gmg_score_orfs_g3) bounds the ORF length up to which no
// FP64 addition can round; longer ORFs are accumulated by one lane in the reference's serial order.
#define MGP_SLOTS 512  // codon-boundary prefixes per warp: sequences up to 3 * (MGP_SLOTS - 1) bases

// Plain glimmer-mg on read sets: the partial-window table of k1_partial_side, [n_seq][2 (w - 1)][3], and the gene model's
// window; t == NULL when the K1 planes are complete.
struct PlainSide {
  const float* t;
  int w;
};

// The gene-model value of period f at position q of sequence S (index sq) on one strand.  With a partial-window table the
// planes hold full-window walks where the strand's window is partial -- the W-1 first positions of the reverse strand,
// the W-1 last of the forward strand -- and the value comes from the table there; from the planes everywhere else, at
// plane index pidx() (evaluated only then).  (Measured on reads100: a select of the two addresses, one load for every
// lane, makes k3_mg_plain_lanes spill and costs 0.55 ms against 0.53 for this branch.)
template <class PlaneIdx>
__device__ __forceinline__ float mgp_gene(const float* __restrict__ planes, const PlainSide& ps, const MgfBatch& B, const MgfSeq& S,
                                          int32_t sq, bool fwd, int f, int q, PlaneIdx pidx) {
  if (ps.t != NULL) {
    const int wm1 = ps.w - 1;
    const int k = fwd ? wm1 + (S.L - 1 - q) : q;  // the table's offset of (q, strand)
    if (k < (fwd ? 2 * wm1 : wm1)) return __ldg(ps.t + ((size_t)sq * (size_t)(2 * wm1) + (size_t)k) * 3 + f);
  }
  return __ldg(planes + (size_t)(fwd ? f : 3 + f) * (size_t)B.total + pidx());
}

__device__ __forceinline__ void mgp_term(const DevIcm& indep, const float* __restrict__ s_lut, const float* __restrict__ planes,
                                         const PlainSide& ps, const uint32_t* __restrict__ bktidx, const MgfBatch& B, const MgfSeq& S,
                                         int32_t sq, bool fwd, int f, int q, float* g_out, float* n_out) {
  const int64_t p = S.a + q;
  *g_out = mgp_gene(planes, ps, B, S, sq, fwd, f, q, [&]() { return gmg_plane_index(B.words, bktidx, p); });
  float n;
  if (indep.lut3 != NULL) {
    if (fwd) {
      const int raw = (int)(gmg_extract32(B.words, p) & 63);  // bases q, q+1, q+2
      n = q <= S.L - 3 ? s_lut[f * 64 + raw] : __ldg(indep.lutp + (q - (S.L - 2)) * 192 + f * 64 + raw);
    } else {
      const int raw = (int)(gmg_extract32(B.words, p - 2) & 63);  // bases q-2, q-1, q
      n = q >= 2 ? s_lut[192 + f * 64 + raw] : __ldg(indep.lutp + 384 + (1 - q) * 192 + f * 64 + raw);
    }
  } else {
    n = fwd ? icm_fwd(indep, B.words, p, q, S.L, f) : icm_rev(indep, B.words, p, q, 0, f);
  }
  *n_out = n;
}

// What the emission kernel needs of an ORF's root call, worked out once by the count kernel (one thread per ORF) instead of
// by every emission warp: sequence (first base, length), lo / hi, the eligible j range and the plan of the truncated
// records (mgf_own_open, mgf_plan).  32 bytes: two 16-byte loads, prefetched one ORF ahead.
struct PlainDesc {
  uint32_t a;    // global index of the sequence's first base (batches hold fewer than 2^32 bases)
  int32_t L;     // its length
  int32_t lo, hi;
  int32_t j_lo, j_hi, j_hs;
  uint32_t bits;  // bit 0 fwd, bit 1 trunc, bit 2 state_after, bits 4.. nT
};

__global__ void __launch_bounds__(128) k3_mg_plain_count(MgfBatch B, DevParams P, const gmg_orf* __restrict__ orfs,
                                                         const int32_t* __restrict__ orf_seq, int64_t n_orfs,
                                                         int64_t* __restrict__ counts, PlainDesc* __restrict__ desc) {
  const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= n_orfs) return;
  const MgfSeq S = mgf_seq_of(B, orf_seq[o]);
  const gmg_orf orf = orfs[o];
  const bool fwd = orf.frame > 0;
  const int hi = fwd ? orf.stop_position - 1 : orf.stop_position + 3 + orf.orf_len;
  const int lo = fwd ? hi - orf.orf_len : orf.stop_position + 3;
  MgfOwn f;
  mgf_own_open(B, S, P, fwd, lo, hi, 0, f);
  counts[o] = mgf_own_count(f, fwd, -1);
  MgfPlan pl;
  mgf_plan(f, fwd, pl);
  PlainDesc d;
  d.a = (uint32_t)S.a;
  d.L = S.L;
  d.lo = lo;
  d.hi = hi;
  d.j_lo = f.j_lo;
  d.j_hi = f.j_hi;
  d.j_hs = f.j_hs;
  d.bits = (fwd ? 1u : 0u) | (f.trunc ? 2u : 0u) | (pl.state_after ? 4u : 0u) | ((uint32_t)pl.nT << 4);
  desc[o] = d;
}

template <bool kPS>
__global__ void __launch_bounds__(128) k3_mg_plain(DevIcm indep_, IndepSeqs X, const float* __restrict__ planes, PlainSide ps,
                                                   const uint32_t* __restrict__ bktidx, MgfBatch B, DevParams P_, CodonSets cs,
                                                   const gmg_orf* __restrict__ orfs, const int32_t* __restrict__ orf_seq,
                                                   int64_t n_orfs, const int64_t* __restrict__ start_off,
                                                   gmg_start* __restrict__ starts, int exact_len,
                                                   unsigned long long* __restrict__ n_ordered, int slots, int lanes) {
  constexpr unsigned FULL = 0xffffffffu;
  extern __shared__ double s_pref_all[];  // [4 warps][slots]: sized for the batch's longest sequence (occupancy on short reads)
  __shared__ float s_lut_sh[384];
  if (!kPS && indep_.lut3 != NULL)
    for (int i = threadIdx.x; i < 384; i += blockDim.x) s_lut_sh[i] = indep_.lut3[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t o = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (o >= n_orfs) return;  // warp-uniform
  const int64_t so = start_off[o];
  if (start_off[o + 1] == so) return;
  const int32_t sq = orf_seq[o];
  const MgfSeq S = mgf_seq_of(B, sq);
  // per-sequence models (gmg_score_orfs_mg_gc): the sequence's own table (read through L1) and ignore length
  DevIcm own;  // kPS: the sequence's own model; the single-model form reads the kernel parameter
  if constexpr (kPS) own = indep_of(indep_, X, orf_seq[o]);
  const DevIcm& indep = kPS ? own : indep_;
  const float* const s_lut = kPS ? indep.lut3 : s_lut_sh;
  const DevParams P = kPS ? mgf_params_of(P_, X, orf_seq[o]) : P_;
  const gmg_orf orf = orfs[o];
  const bool fwd = orf.frame > 0;
  const int hi = fwd ? orf.stop_position - 1 : orf.stop_position + 3 + orf.orf_len;
  const int lo = fwd ? hi - orf.orf_len : orf.stop_position + 3;
  MgfOwn f;
  mgf_own_open(B, S, P, fwd, lo, hi, 0, f);
  double* pref = s_pref_all + (size_t)wid * slots;
  // score[j] for j < j_hi is all the records can ask for (score[j - 1] at their own j <= j_hi)
  const int need = f.j_hi;  // terms j = 0 .. need - 1
  if (lanes && need <= 384 && f.j_lo >= 3) return;  // an instance of k3_mg_plain_lanes has written this ORF (mgl_takes)
  if (lane == 0) pref[0] = 0.0;
  // warp-parallel scan; its sums carry the reference's bits whenever the ORF's certificate holds: every term is a
  // multiple of 2^g (g from the smallest float exponent the ORF meets) and the sum of magnitudes stays below 2^(g+52),
  // so no addition of ANY association can round (DESIGN.md section 3.2)
  unsigned umin = 0x7fffffffu;
  float asum = 0.f;
  double carry = 0.0;
  for (int base = 0; base < need; base += 32) {
    const int j = base + lane;
    double x = 0.0;
    if (j < need) {
      float g, n;
      mgp_term(indep, s_lut, planes, ps, bktidx, B, S, sq, fwd, (1 + j) % 3, fwd ? hi - 1 - j : lo - 1 + j, &g, &n);
      k2_cert_term(g, umin, asum);
      k2_cert_term(n, umin, asum);
      x = (double)g - (double)n;
    }
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const double t = __shfl_up_sync(FULL, x, d);
      if (lane >= d) x += t;
    }
    x += carry;
    if (j < need && (j + 1) % 3 == 0) pref[(j + 1) / 3] = x;
    carry = __shfl_sync(FULL, x, 31);
  }
  double asum_d = (double)asum;  // <= need / 32 + 1 float additions per lane: the 0.1 % margin covers their rounding
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    umin = min(umin, __shfl_xor_sync(FULL, umin, d));
    asum_d += __shfl_xor_sync(FULL, asum_d, d);
  }
  const int e = (int)(umin >> 23);
  const bool exact = exact_len >= 0 && (umin == 0x7fffffffu || asum_d * 1.001 < ldexp(1.0, (e > 0 ? e : 1) - 150 + 52));
  if (!exact) {  // no certificate: the reference's own order, one lane
    __syncwarp();
    if (lane == 0) {
      atomicAdd(n_ordered, 1ull);
      double run = 0.0;
      for (int j = 0; j < need; j++) {
        float g, n;
        mgp_term(indep, s_lut, planes, ps, bktidx, B, S, sq, fwd, (1 + j) % 3, fwd ? hi - 1 - j : lo - 1 + j, &g, &n);
        run = run + ((double)g - (double)n);
        if ((j + 1) % 3 == 0) pref[(j + 1) / 3] = run;
      }
    }
  }
  __syncwarp();
  if (lane == 0) {
    const int ep[2] = {0, 0}, et[2] = {0, 0};
    mgf_own_write_with(B, S, P, cs, f, fwd, 0.0, 0, 0, ep, et, starts + so, [](int) { return (int64_t)0; },
                       [&](int j) { return pref[j / 3]; });
  }
}

// The fused pass with ONE CODON PER LANE -- the default for ORFs of up to 384 scored bases (every ORF of a short-read
// set).  The warp-per-ORF kernel above spends a 5-step FP64 scan on every 32 bases and a serial record writer on lane 0:
// ~1 200 warp instructions per ORF, 0.60 ms per 31 Mbp batch.  Here a lane sums the three terms of one codon, ONE scan
// per group of lanes gives every codon-boundary prefix, and the lanes write the records of their own positions (mgf_plan /
// mgf_recs_at: the position-by-position form of the reference's start loop, held to the CPU checker on the host by
// tests/mgflat_host_check.cu).
// Exactness as above: the per-ORF certificate (smallest term exponent, sum of magnitudes); an ORF without one is summed
// by one lane in the reference's serial order into a shared-memory row and the lanes take their prefixes from there.
// ORFs with more than 384 scored bases, or with j_lo < 3, are left to k3_mg_plain (its skip test is this one).
__device__ __forceinline__ bool mgl_takes(int need, int j_lo) { return need <= 384 && j_lo >= 3; }

// CodonSets::which as four 64-bit words, one nibble per 6-bit codon (15 = not a start codon): indexing the byte array of a
// kernel parameter with a run-time subscript makes the compiler copy the whole parameter block to local memory
struct Which4 {
  unsigned long long w[4];
};
__device__ __forceinline__ int which4_of(const Which4& t, int cd) {
  const unsigned long long w = cd < 32 ? (cd < 16 ? t.w[0] : t.w[1]) : (cd < 48 ? t.w[2] : t.w[3]);
  const int v = (int)((w >> (4 * (cd & 15))) & 15ull);
  return v == 15 ? 255 : v;
}

// gene - indep of the three consecutive sequence positions q0, q0 + 1, q0 + 2 (one codon), summed in ascending order of
// q, with the certificate inputs of the six floats.  per(i) = model period of position q0 + i.  One 64-bit window of the
// packed bases serves the three independent-model codes and the three own bases; W == 3 independent models only.
__device__ __forceinline__ double mgl_codon_sum(const DevIcm& indep, const float* __restrict__ planes, const PlainSide& ps,
                                                const uint32_t* __restrict__ bktidx, const MgfBatch& B, const MgfSeq& S, int32_t sq,
                                                bool fwd, int q0, unsigned& umin, float& asum) {
  const int64_t p0 = S.a + q0;
  const uint64_t v = gmg_extract32(B.words, p0 - 2);  // base q0 - 2 + m at bits 2 m
  const uint32_t pu = (uint32_t)p0;                   // batches hold fewer than 2^32 bases
  const uint32_t blk0 = pu >> 5, blk2 = (pu + 2u) >> 5;
  const uint64_t w0 = __ldg(B.words + blk0);
  const uint64_t w2 = blk2 != blk0 ? __ldg(B.words + blk2) : w0;
  double x = 0.0;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const int q = q0 + i;
    const int f = fwd ? (3 - i) % 3 : (1 + i) % 3;
    const float g = mgp_gene(planes, ps, B, S, sq, fwd, f, q, [&]() {
      const uint32_t p = pu + (uint32_t)i, blk = p >> 5, ib = p & 31u;
      const uint64_t w = blk == blk0 ? w0 : w2;
      const unsigned b = (unsigned)(v >> (2 * (i + 2))) & 3u;
      const uint64_t y = w ^ (0x5555555555555555ull * b);
      const uint64_t eq = ~(y | (y >> 1)) & 0x5555555555555555ull & ((1ull << (2 * ib)) - 1ull);
      return __ldg(bktidx + (blk << 2) + b) + (uint32_t)__popcll(eq);
    });
    float n;
    if (fwd) {
      const int raw = (int)(v >> (2 * (i + 2))) & 63;  // bases q, q+1, q+2
      const float* tb = q <= S.L - 3 ? indep.lut3 : indep.lutp + (q - (S.L - 2)) * 192;
      n = __ldg(tb + f * 64 + raw);
    } else {
      const int raw = (int)(v >> (2 * i)) & 63;  // bases q-2, q-1, q
      const float* tb = q >= 2 ? indep.lut3 + 192 : indep.lutp + 384 + (1 - q) * 192;
      n = __ldg(tb + f * 64 + raw);
    }
    k2_cert_term(g, umin, asum);
    k2_cert_term(n, umin, asum);
    x = x + ((double)g - (double)n);
  }
  return x;
}

// G = lanes per ORF, K = chunks of G codons: an instance takes the ORFs with need_lo < need <= 3 * G * K scored bases (and
// j_lo >= 3).  Two instances: <16, 4>, TWO ORFs per warp up to 192 bases, and <32, 4>, one ORF per warp up to 384.
// The kernel is bound by the latency of a warp's dependent rounds (6 us per ORF with one ORF per warp, 40 % issue
// utilisation at 32 warps per SM): more ORFs in flight per warp at the same register count is what raises the throughput
// on short reads (0.61 -> 0.49 ms per 31 Mbp with two; four per warp gave 0.50 -- the lane's serial share grows and its
// prefix registers spill).
template <int G, int K, bool kPS>
__global__ void __launch_bounds__(128, 8) k3_mg_plain_lanes(DevIcm indep_, const float* __restrict__ planes, PlainSide ps,
                                                         const uint32_t* __restrict__ bktidx, MgfBatch B, DevParams P, Which4 which,
                                                         int64_t n_orfs, const int64_t* __restrict__ start_off,
                                                         gmg_start* __restrict__ starts, int exact_len,
                                                         unsigned long long* __restrict__ n_ordered,
                                                         const PlainDesc* __restrict__ desc, int need_lo, IndepSeqs X) {
  constexpr unsigned FULL = 0xffffffffu;
  constexpr int HPW = 32 / G;                                       // ORFs per warp
  constexpr unsigned GMASK = G == 32 ? 0xffffffffu : ((1u << (G & 31)) - 1u);
  __shared__ double s_serial[4][HPW][G * K];  // codon-boundary prefixes of an ORF summed in serial order (rare)
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int sub = lane % G, grp = lane / G, gshift = grp * G;
  // Persistent warps: a warp's life used to be five dependent load rounds (CSR -> ORF -> sequence offsets -> packed bases ->
  // bucket index -> planes) with nothing to overlap them, and ~100 instructions of call geometry that every warp derived
  // again.  The count kernel now leaves a 32-byte descriptor per ORF (sequence, lo / hi, eligible j range, plan of the
  // truncated records), fetched together with the CSR pair for the group's NEXT ORF while it works on the current one.
  const int64_t stride = (((int64_t)gridDim.x * blockDim.x) >> 5) * HPW;
  int64_t o = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * HPW + grp;
  int64_t nx_so = 0, nx_so1 = 0;
  uint4 nx_d0 = make_uint4(0u, 0u, 0u, 0u), nx_d1 = make_uint4(0u, 0u, 0u, 0u);
  int32_t nx_sq = 0;  // the ORF's sequence: its row of the partial-window table, its model (kPS)
  if (o < n_orfs) {
    nx_so = __ldg(start_off + o);
    nx_so1 = __ldg(start_off + o + 1);
    nx_d0 = __ldg(reinterpret_cast<const uint4*>(desc + o));
    nx_d1 = __ldg(reinterpret_cast<const uint4*>(desc + o) + 1);
    nx_sq = __ldg(X.orf_seq + o);
  }
  for (; o - grp < n_orfs; o += stride) {  // warp-uniform: o - grp is the warp's first ORF of this round
  const int64_t so = nx_so, so1 = nx_so1;
  const uint4 d0 = nx_d0, d1 = nx_d1;
  const int32_t xs = nx_sq;
  const bool have = o < n_orfs;
  if (o + stride < n_orfs) {
    nx_so = __ldg(start_off + o + stride);
    nx_so1 = __ldg(start_off + o + stride + 1);
    nx_d0 = __ldg(reinterpret_cast<const uint4*>(desc + o + stride));
    nx_d1 = __ldg(reinterpret_cast<const uint4*>(desc + o + stride) + 1);
    nx_sq = __ldg(X.orf_seq + o + stride);
  }
  MgfSeq S;
  S.a = (int64_t)d0.x;
  S.L = (int)d0.y;
  const int lo = (int)d0.z, hi = (int)d0.w;
  const bool fwd = (d1.w & 1u) != 0;
  MgfOwn f;  // as mgf_own_open leaves it
  f.lo = lo;
  f.hi = hi;
  f.m = hi - lo > 0 ? hi - lo : 0;
  f.trunc = (d1.w >> 1) & 1u;
  f.j_lo = (int)d1.x;
  f.j_hi = (int)d1.y;
  f.j_hs = (int)d1.z;
  f.cpos = fwd ? d0.x + (uint32_t)(hi - 3) : d0.x + (uint32_t)(lo - 1);
  f.st = B.cb + (size_t)((fwd ? 0u : 3u) + f.cpos % 3u) * (size_t)B.nwc;
  const int need = f.j_hi;  // terms j = 0 .. need - 1: score[j - 1] of the highest record position j_hi
  // this group's ORF is worked on here iff it has records and its length is this instance's
  const bool act = have && so1 != so && f.j_lo >= 3 && need > need_lo && need <= 3 * G * K;
  // per-sequence models (gmg_score_orfs_mg_gc): the ORF's own table and ignore length
  DevIcm own;  // kPS: the sequence's own model; the single-model form reads the kernel parameter
  if constexpr (kPS) own = indep_of(indep_, X, xs);
  const DevIcm& indep = kPS ? own : indep_;
  const float* s_lut = indep.lut3;  // 1.5 KB: read through L1 (staging it cost 8 % of the kernel's instructions)
  DevParams Ps;  // kPS: the records' parameters with the sequence's ignore length (the single-model form reads P)
  if constexpr (kPS) Ps = mgf_params_of(P, X, xs);
  MgfPlan pl;  // as mgf_plan leaves it
  pl.nT = (int)(d1.w >> 4);
  pl.state_after = (int)((d1.w >> 2) & 1u);
  {
    const int jt = f.j_hi - 3 * pl.nT;
    pl.jb = jt < f.j_hs ? jt : f.j_hs;
  }
  const int ncod = act ? need / 3 : 0, nch = (ncod + G - 1) / G;
  const int nch_w = G == 32 ? nch : __reduce_max_sync(FULL, nch);  // chunks the warp runs (warp-uniform)
  if (nch_w == 0) continue;
  double incl[K];
  double carry = 0.0;
  unsigned umin = 0x7fffffffu;
  float asum = 0.f;
#pragma unroll
  for (int k = 0; k < K; k++) {
    incl[k] = 0.0;
    if (k < nch_w) {  // warp-uniform
      const int c = G * k + sub;
      double x = 0.0;
      if (c < ncod) {
        if (indep.lut3 != NULL) {  // j = 3 c .. 3 c + 2: positions hi-1-3c-2 .. hi-1-3c (forward), lo-1+3c .. +2 (reverse)
          x = mgl_codon_sum(indep, planes, ps, bktidx, B, S, xs, fwd, fwd ? hi - 3 - 3 * c : lo - 1 + 3 * c, umin, asum);
        } else {
#pragma unroll
          for (int t = 0; t < 3; t++) {
            const int j = 3 * c + t;
            float g, n;
            mgp_term(indep, s_lut, planes, ps, bktidx, B, S, xs, fwd, (1 + t) % 3, fwd ? hi - 1 - j : lo - 1 + j, &g, &n);
            k2_cert_term(g, umin, asum);
            k2_cert_term(n, umin, asum);
            x = x + ((double)g - (double)n);
          }
        }
      }
#pragma unroll
      for (int d = 1; d < G; d <<= 1) {
        const double y = __shfl_up_sync(FULL, x, d, G);
        if (sub >= d) x += y;
      }
      x += carry;
      incl[k] = x;  // score[3 (c + 1) - 1]
      carry = __shfl_sync(FULL, x, G - 1, G);
    }
  }
  double asum_d = (double)asum;  // at most 6 * K float additions per lane: the 0.1 % margin covers their rounding
#pragma unroll
  for (int d = G / 2; d > 0; d >>= 1) {  // within the group (xor with d < G stays inside it)
    umin = min(umin, __shfl_xor_sync(FULL, umin, d));
    asum_d += __shfl_xor_sync(FULL, asum_d, d);
  }
  const int e = (int)(umin >> 23);
  const bool exact = exact_len >= 0 && (umin == 0x7fffffffu || asum_d * 1.001 < ldexp(1.0, (e > 0 ? e : 1) - 150 + 52));
  if (!exact && act && sub == 0) {  // no certificate: the reference's own order, one lane of the group
    atomicAdd(n_ordered, 1ull);
    double run = 0.0;
    for (int j = 0; j < need; j++) {
      float g, n;
      mgp_term(indep, s_lut, planes, ps, bktidx, B, S, xs, fwd, (1 + j) % 3, fwd ? hi - 1 - j : lo - 1 + j, &g, &n);
      run = run + ((double)g - (double)n);
      if ((j + 1) % 3 == 0) s_serial[wid][grp][j / 3] = run;
    }
  }
  __syncwarp();
  // records, from the highest position down: lane = position j = 3 (c + 1); ballots are taken by the whole warp, a group
  // reads its own G bits
  const unsigned higher = sub == G - 1 ? 0u : (~((2u << sub) - 1u)) & GMASK;
  int placed = 0;
  bool seen_nonzero = false;
  const int ep[2] = {0, 0}, et[2] = {0, 0};
  gmg_start* out = starts + so;
#pragma unroll
  for (int k = K - 1; k >= 0; k--) {
    if (k < nch_w) {  // warp-uniform
      const int c = G * k + sub, j = 3 * (c + 1);
      bool trunc_rec = false, chain = false;
      int nr = 0;
      if (c < ncod && j >= f.j_lo) nr = mgf_recs_at(f, pl, fwd, j, &trunc_rec, &chain);
      const int kp = mgf_kpos(f, fwd, j);
      const unsigned m1 = (__ballot_sync(FULL, nr >= 1) >> gshift) & GMASK, m2 = (__ballot_sync(FULL, nr == 2) >> gshift) & GMASK;
      const unsigned mnz = (__ballot_sync(FULL, chain && kp != 0) >> gshift) & GMASK;
      if (nr) {
        const int idx = placed + __popc(m1 & higher) + __popc(m2 & higher);
        const double sum = exact ? incl[k] : s_serial[wid][grp][c];
        const double sc = (sum - 0.0) + 0.0;
        if (trunc_rec) {
          mgf_put(out + idx, kPS ? Ps : P, j + 2, kp, sc, -1, 1, 1, 0, ep, et);
          if (nr == 2) mgf_put(out + idx + 1, kPS ? Ps : P, j + 2, kp, sc, which4_of(which, mgf_codon_at(B, S, f, fwd, j)), 0, 0, 0, ep, et);
        } else {
          const int first = (pl.state_after && !seen_nonzero && (mnz & higher) == 0u) ? 1 : 0;
          mgf_put(out + idx, kPS ? Ps : P, j + 2, kp, sc, which4_of(which, mgf_codon_at(B, S, f, fwd, j)), 0, first, 0, ep, et);
        }
      }
      placed += __popc(m1) + __popc(m2);
      seen_nonzero = seen_nonzero || mnz != 0u;
    }
  }
  __syncwarp();  // the serial rows are free for the warp's next ORFs
  }
}

// ------------------------------------------------------------------------------------------------
// Start-list reduction (SURVEY.md section 8 row a11b): what Score_Orfs_Errors' filter (glimmer-mg.cc:1656-1684) and
// Add_Events_Fwd / Add_Events_Rev (glimmer_base.cc:65-128, 175-235) keep of an ORF's raw start_list -- at most one
// candidate per start position -- decided on the device so that only survivors cross PCIe.
//
// One warp per ORF, two sweeps over its records and a shared-memory table indexed by start position:
//   gate 1  first_j + 1 >= Min_Gene_Len, first_j = j of the record at the lowest (forward) / highest (reverse)
//           position.  Several records can share that position with different j (std::sort is not stable): the ORF
//           is decided here only when they all agree, else it is handed back (status 2).
//   gate 2  best raw score > Start_Threshold.
//   per start position: candidates with 1 + j >= Min_Gene_Len are ranked by
//           x = ((score + prior) [+ LogOdds_Start(which)]) + LogOdds_Length(...)
//           -- the reference's event score, formed in its order, WITHOUT the RBS term: Add_PWM_Score adds the same
//           value to every candidate of a position, so it shifts all of them alike up to a rounding of the last
//           bits.  The maximum survives if x + pwm_bonus_max can exceed Event_Threshold; if a second candidate of
//           the position lies within 1e-9 of it (a tie, or close enough for the RBS term's rounding to matter) the
//           ORF is handed back as well.  The host then runs the reference's own Add_Events on the survivors (exact
//           scores, exact threshold) or, for status 2, on the raw list it fetches for that ORF.
struct DevEventModel {
  double prior, start_threshold, event_threshold, pwm_bonus_max;
  double start_lo[8];
  int n_len, n_class, min_gene_len;
  const double* len_lo;      // [n_class][2][2][n_len]
  const int32_t* seq_class;  // [n_seq] or NULL
};
struct RedSlot {
  unsigned long long best;
  unsigned int win, cnt;
};
__device__ __forceinline__ unsigned long long red_key(double x) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(x);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double red_unkey(unsigned long long k) {
  return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

__global__ void __launch_bounds__(128) k3_mg_reduce(const gmg_start* __restrict__ starts, const int64_t* __restrict__ soff,
                                                    const gmg_orf* __restrict__ orfs, const int32_t* __restrict__ orf_seq,
                                                    const int64_t* __restrict__ off, int64_t n_orfs, DevEventModel M,
                                                    int slots_per_warp, gmg_start* __restrict__ out,
                                                    unsigned long long* __restrict__ cursor, int64_t* __restrict__ red_first,
                                                    int32_t* __restrict__ red_cnt, uint8_t* __restrict__ status,
                                                    const uint32_t* __restrict__ big,
                                                    const unsigned long long* __restrict__ n_big) {
  constexpr unsigned FULL = 0xffffffffu;
  constexpr double TOL = 1e-9;
  extern __shared__ __align__(16) unsigned char s_red[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  RedSlot* tab = reinterpret_cast<RedSlot*>(s_red) + (size_t)wid * slots_per_warp;
  // the ORFs k3_mg_reduce_small left over (big != NULL: their list and its length on the device), else all of them
  const int64_t n_items = big ? (int64_t)*n_big : n_orfs;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t item = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; item < n_items; item += n_warps) {  // warp-uniform
  const int64_t o = big ? (int64_t)big[item] : item;
  const int64_t a = soff[o];
  const int n = (int)(soff[o + 1] - a);
  const gmg_start* rec = starts + a;
  int st = 0, kept = 0;
  long long first = 0;
  if (n > 0) {
    const gmg_orf orf = orfs[o];
    const bool fwd = orf.frame > 0;
    const int32_t sq = orf_seq[o];
    const int L = (int)(off[sq + 1] - off[sq]);
    // sweep 1: position range, best raw score
    int pmin = INT_MAX, pmax = INT_MIN;
    double best = -DBL_MAX;
    for (int i = lane; i < n; i += 32) {
      const int p = rec[i].pos;
      pmin = min(pmin, p);
      pmax = max(pmax, p);
      best = fmax(best, rec[i].score);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      pmin = min(pmin, __shfl_xor_sync(FULL, pmin, d));
      pmax = max(pmax, __shfl_xor_sync(FULL, pmax, d));
      best = fmax(best, __shfl_xor_sync(FULL, best, d));
    }
    const int range = pmax - pmin + 1;
    if (range > slots_per_warp) {
      st = 2;
    } else {
      for (int i = lane; i < range; i += 32) {
        tab[i].best = 0ull;
        tab[i].win = 0xffffffffu;
        tab[i].cnt = 0u;
      }
      __syncwarp();
      const int ext = fwd ? pmin : pmax;
      const int cls = M.seq_class ? M.seq_class[sq] : 0;
      const bool t3 = fwd ? orf.stop_position > L - 2 : orf.stop_position < 1;
      const double* lenrow = M.len_lo + (size_t)cls * 4 * M.n_len;
      bool pass_any = false, fail_any = false, too_long = false;
      // sweep 2: first_j gate inputs; per-position maxima of the candidates
      for (int i = lane; i < n; i += 32) {
        const gmg_start r = rec[i];
        if (r.pos == ext) {
          if (r.j + 1 >= M.min_gene_len) pass_any = true;
          else fail_any = true;
        }
        if (1 + r.j >= M.min_gene_len) {
          const int l = (1 + r.j) / 3;
          if (l >= M.n_len) {
            too_long = true;
            continue;
          }
          double x = r.score + M.prior;
          if (r.which >= 0) x += M.start_lo[r.which & 7];
          x += lenrow[(size_t)((r.truncated ? 2 : 0) + (t3 ? 1 : 0)) * M.n_len + l];
          if (x + M.pwm_bonus_max > M.event_threshold - TOL) atomicMax(&tab[r.pos - pmin].best, red_key(x));
        }
      }
      pass_any = __any_sync(FULL, pass_any);
      fail_any = __any_sync(FULL, fail_any);
      too_long = __any_sync(FULL, too_long);
      __syncwarp();
      if (too_long || (pass_any && fail_any)) {
        st = 2;
      } else if (!pass_any || !(best > M.start_threshold)) {
        st = 0;
      } else {
        // sweep 3: who is (within TOL of) the maximum of its position
        for (int i = lane; i < n; i += 32) {
          const gmg_start r = rec[i];
          if (1 + r.j >= M.min_gene_len) {
            const int l = (1 + r.j) / 3;
            double x = r.score + M.prior;
            if (r.which >= 0) x += M.start_lo[r.which & 7];
            x += lenrow[(size_t)((r.truncated ? 2 : 0) + (t3 ? 1 : 0)) * M.n_len + l];
            RedSlot* t = &tab[r.pos - pmin];
            if (t->best != 0ull && x + M.pwm_bonus_max > M.event_threshold - TOL && x >= red_unkey(t->best) - TOL) {
              atomicAdd(&t->cnt, 1u);
              atomicMin(&t->win, (unsigned)i);
            }
          }
        }
        __syncwarp();
        bool amb = false;
        int mine = 0;
        for (int i = lane; i < range; i += 32) {
          if (tab[i].cnt > 1u) amb = true;
          if (tab[i].cnt >= 1u) mine++;
        }
        amb = __any_sync(FULL, amb);
        if (amb) {
          st = 2;
        } else {
          st = 1;
          int incl = mine;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(FULL, incl, d);
            if (lane >= d) incl += t;
          }
          kept = __shfl_sync(FULL, incl, 31);
          unsigned long long base = 0;
          if (lane == 0 && kept) base = atomicAdd(cursor, (unsigned long long)kept);
          base = __shfl_sync(FULL, base, 0);
          first = (long long)base;
          // lane's slots are i = lane, lane + 32, ...: survivors go out in that (deterministic) order
          unsigned long long at = base + (unsigned long long)(incl - mine);
          for (int i = lane; i < range; i += 32)
            if (tab[i].cnt >= 1u) out[at++] = rec[tab[i].win];
        }
      }
    }
    __syncwarp();
  }
  if (lane == 0) {
    status[o] = (uint8_t)st;
    red_cnt[o] = st == 1 ? kept : 0;
    red_first[o] = first;
  }
  __syncwarp();
  }
}

// The same decisions for ORFs with at most RED_SMALL raw records, ONE THREAD per ORF, everything in registers: on plain
// read sets nearly every ORF has one to three records and a warp per ORF spent 680 instructions on each (0.38 ms per
// 31 Mbp batch, all of it instruction issue).  ORFs with more records are appended to `big` for k3_mg_reduce.
#define RED_SMALL 8
__global__ void __launch_bounds__(128) k3_mg_reduce_small(const gmg_start* __restrict__ starts, const int64_t* __restrict__ soff,
                                                          const gmg_orf* __restrict__ orfs, const int32_t* __restrict__ orf_seq,
                                                          const int64_t* __restrict__ off, int64_t n_orfs, DevEventModel M,
                                                          gmg_start* __restrict__ out, unsigned long long* __restrict__ cursor,
                                                          int64_t* __restrict__ red_first, int32_t* __restrict__ red_cnt,
                                                          uint8_t* __restrict__ status, uint32_t* __restrict__ big,
                                                          unsigned long long* __restrict__ n_big) {
  constexpr unsigned FULL = 0xffffffffu;
  constexpr double TOL = 1e-9;
  const int lane = threadIdx.x & 31;
  const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int n = 0, st = 0, kept = 0;
  int64_t a = 0;
  if (o < n_orfs) {
    a = soff[o];
    n = (int)(soff[o + 1] - a);
  }
  const bool is_big = n > RED_SMALL;
  unsigned keep_mask = 0;  // bit i: record i survives
  if (n > 0 && !is_big) {
    const gmg_start* rec = starts + a;
    const gmg_orf orf = orfs[o];
    const bool fwd = orf.frame > 0;
    const int32_t sq = orf_seq[o];
    const int L = (int)(off[sq + 1] - off[sq]);
    const int cls = M.seq_class ? M.seq_class[sq] : 0;
    const bool t3 = fwd ? orf.stop_position > L - 2 : orf.stop_position < 1;
    const double* lenrow = M.len_lo + (size_t)cls * 4 * M.n_len;
    int pos[RED_SMALL], jj[RED_SMALL];
    double x[RED_SMALL];
    bool elig[RED_SMALL];
    int pmin = INT_MAX, pmax = INT_MIN;
    double best = -DBL_MAX;
    bool too_long = false;
#pragma unroll
    for (int i = 0; i < RED_SMALL; i++) {
      pos[i] = 0;
      jj[i] = 0;
      x[i] = 0.0;
      elig[i] = false;
      if (i < n) {
        const gmg_start r = rec[i];
        pos[i] = r.pos;
        jj[i] = r.j;
        pmin = min(pmin, r.pos);
        pmax = max(pmax, r.pos);
        best = fmax(best, r.score);
        if (1 + r.j >= M.min_gene_len) {
          const int l = (1 + r.j) / 3;
          if (l >= M.n_len) {
            too_long = true;
          } else {
            double v = r.score + M.prior;
            if (r.which >= 0) v += M.start_lo[r.which & 7];
            v += lenrow[(size_t)((r.truncated ? 2 : 0) + (t3 ? 1 : 0)) * M.n_len + l];
            x[i] = v;
            elig[i] = v + M.pwm_bonus_max > M.event_threshold - TOL;
          }
        }
      }
    }
    const int ext = fwd ? pmin : pmax;
    bool pass_any = false, fail_any = false;
#pragma unroll
    for (int i = 0; i < RED_SMALL; i++)
      if (i < n && pos[i] == ext) {
        if (jj[i] + 1 >= M.min_gene_len) pass_any = true;
        else fail_any = true;
      }
    if (too_long || (pass_any && fail_any)) {
      st = 2;
    } else if (!pass_any || !(best > M.start_threshold)) {
      st = 0;
    } else {
      st = 1;
      bool amb = false;
#pragma unroll
      for (int i = 0; i < RED_SMALL; i++) {
        if (i < n && elig[i]) {
          double mx = x[i];
#pragma unroll
          for (int k = 0; k < RED_SMALL; k++)
            if (k < n && elig[k] && pos[k] == pos[i]) mx = fmax(mx, x[k]);
          if (x[i] >= mx - TOL) {  // within TOL of its position's maximum
#pragma unroll
            for (int k = 0; k < RED_SMALL; k++)
              if (k != i && k < n && elig[k] && pos[k] == pos[i] && x[k] >= mx - TOL) amb = true;
            keep_mask |= 1u << i;
          }
        }
      }
      if (amb) {
        st = 2;
        keep_mask = 0;
      }
      kept = __popc(keep_mask);
    }
  }
  // one cursor bump and one list bump per warp
  int incl = kept;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int t = __shfl_up_sync(FULL, incl, d);
    if (lane >= d) incl += t;
  }
  const int warp_kept = __shfl_sync(FULL, incl, 31);
  unsigned long long base = 0;
  if (lane == 31 && warp_kept) base = atomicAdd(cursor, (unsigned long long)warp_kept);
  base = __shfl_sync(FULL, base, 31);
  const unsigned bigs = __ballot_sync(FULL, is_big);
  unsigned long long bbase = 0;
  if (lane == 0 && bigs) bbase = atomicAdd(n_big, (unsigned long long)__popc(bigs));
  bbase = __shfl_sync(FULL, bbase, 0);
  if (o >= n_orfs) return;
  if (is_big) {
    big[bbase + (unsigned)__popc(bigs & ((1u << lane) - 1u))] = (uint32_t)o;
    return;
  }
  long long first = 0;
  if (kept) {
    first = (long long)(base + (unsigned long long)(incl - kept));
    const gmg_start* rec = starts + a;
    long long at = first;
    for (int i = 0; i < n; i++)
      if (keep_mask >> i & 1u) out[at++] = rec[i];
  }
  status[o] = (uint8_t)st;
  red_cnt[o] = st == 1 ? kept : 0;
  red_first[o] = first;
}

// ------------------------------------------------------------------------------------------------
// All_Frame_Score (glimmer3.cc:328-359), batched: for every item -- a region [lo, lo + len) of a sequence -- the six
// ICM_t::Score_String sums the reference forms for the `.detail` log: the region read downwards (context = the bases to
// its right, the orientation of a forward gene's buff) with first-base periods 0, 1, 2, and the region's complement
// read upwards (context = the complemented bases to its left) with first-base periods 0, 1, 2.  Positions past the
// first W-1 are K1 plane entries; the first W-1 of either direction see only the region itself (Partial_Window_Prob,
// icm.cc:807-842).  One warp per item; every sum is accumulated in the reference's serial order (icm.cc:886-900).
// out[item][0..2] = downward sums (period of the first base 0, 1, 2), out[item][3..5] = upward sums.
__global__ void __launch_bounds__(128) k_all_frame_scores(DevIcm gene, const uint64_t* __restrict__ words,
                                                          const int64_t* __restrict__ off, const uint32_t* __restrict__ bktidx,
                                                          int64_t total, const float* __restrict__ planes, int64_t n,
                                                          const int32_t* __restrict__ it_seq, const int32_t* __restrict__ it_lo,
                                                          const int32_t* __restrict__ it_len, double* __restrict__ out) {
  constexpr unsigned FULL = 0xffffffffu;
  const int64_t it = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (it >= n) return;
  const int64_t a = off[it_seq[it]];
  const int lo = it_lo[it], len = it_len[it], hi = lo + len;
  double tot[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  for (int base = 0; base < len; base += 32) {
    const int i = base + lane;
    float v[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (i < len) {
      const int qd = hi - 1 - i, qu = lo + i;
      const size_t pd = gmg_plane_index(words, bktidx, a + qd), pu = gmg_plane_index(words, bktidx, a + qu);
#pragma unroll
      for (int f0 = 0; f0 < 3; f0++) {
        const int f = (f0 + i) % 3;
        v[f0] = i < gene.W - 1 ? icm_fwd(gene, words, a + qd, qd, hi, f) : __ldg(planes + (size_t)f * total + pd);
        v[3 + f0] = i < gene.W - 1 ? icm_rev(gene, words, a + qu, qu, lo, f) : __ldg(planes + (size_t)(3 + f) * total + pu);
      }
    }
    const int cnt = min(32, len - base);
    for (int l = 0; l < cnt; l++)
#pragma unroll
      for (int k = 0; k < 6; k++) tot[k] += (double)__shfl_sync(FULL, v[k], l);
  }
  if (lane == 0)
#pragma unroll
    for (int k = 0; k < 6; k++) out[it * 6 + k] = tot[k];
}

extern "C" int gmg_all_frame_scores(gmg_ctx* ctx, const gmg_icm* gene, gmg_seqset* s, int64_t n, const int32_t* h_seq,
                                    const int32_t* h_lo, const int32_t* h_len, double* h_out) {
  GMG_CHECK(ctx && gene && s && (n == 0 || (h_seq && h_lo && h_len && h_out)), "gmg_all_frame_scores: NULL argument");
  if (n == 0) return 0;
  for (int64_t i = 0; i < n; i++) {
    GMG_CHECK(h_seq[i] >= 0 && h_seq[i] < s->n, "gmg_all_frame_scores: item %lld: sequence %d out of range", (long long)i, h_seq[i]);
    const int64_t L = s->off[(size_t)h_seq[i] + 1] - s->off[(size_t)h_seq[i]];
    GMG_CHECK(h_lo[i] >= 0 && h_len[i] >= 0 && (int64_t)h_lo[i] + h_len[i] <= L, "gmg_all_frame_scores: item %lld: region [%d, %d) "
              "outside its %lld bp sequence", (long long)i, h_lo[i], h_lo[i] + h_len[i], (long long)L);
  }
  float* planes;
  if (launch_k1(ctx, gene, s, &planes, NULL)) return 1;
  void* d_it;
  if (gmg_scratch(ctx, SCR_MISC, (size_t)n * (3 * sizeof(int32_t) + 6 * sizeof(double)) + 64, &d_it)) return 1;
  double* d_out = (double*)d_it;
  int32_t* d_seq = (int32_t*)(d_out + 6 * n);
  int32_t* d_lo = d_seq + n;
  int32_t* d_len = d_lo + n;
  GMG_CUDA(cudaMemcpyAsync(d_seq, h_seq, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
  GMG_CUDA(cudaMemcpyAsync(d_lo, h_lo, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
  GMG_CUDA(cudaMemcpyAsync(d_len, h_len, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
  k_all_frame_scores<<<(unsigned)((n * 32 + 127) / 128), 128, 0, ctx->stream>>>(gene->dev, s->d_words, s->d_off, s->d_bktidx, s->total,
                                                                                planes, n, d_seq, d_lo, d_len, d_out);
  ctx->launches++;
  GMG_CUDA(cudaGetLastError());
  GMG_CUDA(cudaMemcpyAsync(h_out, d_out, (size_t)n * 6 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// host drivers of the two scoring halves

static int ensure_start_capacity(gmg_seqset* s, int64_t n) {
  if ((size_t)n > s->cap_starts || !s->d_starts) {
    if (s->d_starts) cudaFreeAsync(s->d_starts, s->ctx->stream);
    s->d_starts = NULL;
    size_t cap = (size_t)n + (size_t)n / 8 + 64;
    GMG_CUDA(cudaMallocAsync(&s->d_starts, cap * sizeof(gmg_start), s->ctx->stream));
    s->cap_starts = cap;
  }
  return 0;
}

__global__ void k_count_zero_flags(const uint8_t* __restrict__ cert, int64_t n, unsigned long long* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned bad = (i < n && cert[i] == 0) ? 1u : 0u;
  bad = __popc(__ballot_sync(0xffffffffu, bad));
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(out, (unsigned long long)bad);
}

extern "C" int gmg_score_orfs_g3(gmg_ctx* ctx, const gmg_icm* gene, const gmg_icm* indep, gmg_seqset* s,
                                 const gmg_params* p, int64_t* n_starts) {
  GMG_CHECK(ctx && gene && indep && s && p, "gmg_score_orfs_g3: NULL argument");
  GMG_CHECK(gene->P == 3 && indep->P == 3, "glimmer3 scoring needs periodicity-3 models");
  if (gmg_icm_ready(gene) || gmg_icm_ready(indep)) return 1;
  if (gmg_seqset_ensure_buckets(ctx, s)) return 1;  // here, not inside K1: its scratch must not be touched once the side stream runs
  CodonSets cs;
  DevParams dp;
  if (make_codon_sets(p, &cs, &dp)) return 1;
  s->n_starts = 0;
  s->uncertified = 0;
  if (n_starts) *n_starts = 0;
  if (s->n_orfs == 0) return 0;
  if (ensure_codon_bits(ctx, s, cs)) return 1;
  // Static exactness certificate: every term is a float of the two models, i.e. an integer multiple of
  // 2^gexp (gexp = smallest ulp exponent over both tables); every sum formed for an ORF -- and every partial sum of
  // the reference's serial accumulation -- has at most orf_len + 4 tiles of terms, each bounded by max|gene| +
  // max|indep|.  While that bound stays below 2^(gexp+52) no addition can round, so any association gives the
  // reference's bits: ORFs up to exact_len bases take the scan-based path, longer ones (and every ORF when the
  // independent model is not the usual 3-base one) are accumulated in the reference's own order.
  const int ja = (gene->W - 2) + (5 - (gene->W - 2) % 3) % 3;  // first j >= W-2 with j % 3 == 2
  int exact_len = -1;
  const bool force_ordered = getenv("GMG_G3_ORDERED") && atoi(getenv("GMG_G3_ORDERED"));  // test hook
  if (indep->dev.lut3 != NULL && gene->W >= 2 && ja < 32 && !force_ordered) {
    int eg, en;
    float mg, mn;
    gmg_icm_value_stats(gene, &eg, &mg);
    gmg_icm_value_stats(indep, &en, &mn);
    const double lim = ldexp(1.0, (eg < en ? eg : en) + 52) / (((double)mg + (double)mn) * 1.01 + 1e-300) - 12.0 * G3_TS;
    exact_len = lim >= 2e9 ? INT_MAX : (lim < 0 ? -1 : (int)lim);
  }
  const bool exact = exact_len >= 0;
  GMG_CUDA(cudaMemsetAsync(s->d_gc + 1, 0, sizeof(unsigned long long), ctx->stream));
  // Start counts, their scan and the head sums only need the codon bitmaps and the packed bases: they run on the
  // context's side stream BESIDE the walks (K1) and the codon sums (K2), which fill the machine on the main stream.
  // The total travels to pinned memory behind an event, so the host sizes the output while K1 is still running; the
  // emit pass joins both streams.
  void *d_counts, *d_first;
  if (gmg_scratch(ctx, SCR_FLAGS, (size_t)(s->n_orfs + 2) * sizeof(int64_t), &d_counts)) return 1;
  if (gmg_scratch(ctx, SCR_TMP3, (size_t)s->n_orfs * sizeof(int32_t), &d_first)) return 1;
  int64_t* counts = (int64_t*)d_counts;
  int* d_maxlen = (int*)(counts + s->n_orfs + 1);
  double *cumc = NULL, *tileT = NULL, *heads = NULL;
  const int64_t ntiles = s->total / (3 * G3_TS) + 1, tot3 = ntiles * 3 * G3_TS;
  const int nh = (ja + 1) / 3;
  if (exact) {
    void *d_cum, *d_tiles, *d_heads;
    if (gmg_scratch(ctx, SCR_CUM, (size_t)2 * tot3 * sizeof(double), &d_cum)) return 1;
    if (gmg_scratch(ctx, SCR_QUAL, (size_t)ntiles * 6 * sizeof(double), &d_tiles)) return 1;
    if (gmg_scratch(ctx, SCR_TMP2, (size_t)s->n_orfs * nh * sizeof(double), &d_heads)) return 1;
    cumc = (double*)d_cum;
    tileT = (double*)d_tiles;
    heads = (double*)d_heads;
  }
  float* planes = NULL;
  void* d_planes;
  if (gmg_scratch(ctx, SCR_PLANES, (size_t)6 * (s->total + 32) * sizeof(float), &d_planes)) return 1;  // before the fork
  cudaStream_t side = ctx->side;
  GMG_CUDA(cudaEventRecord(ctx->ev_fork, ctx->stream));
  GMG_CUDA(cudaStreamWaitEvent(side, ctx->ev_fork, 0));
  GMG_CUDA(cudaMemsetAsync(counts + s->n_orfs, 0, 2 * sizeof(int64_t), side));
  k3_g3_count<<<(unsigned)((s->n_orfs + 127) / 128), 128, 0, side>>>(s->d_cbits, s->nwc, s->d_off, s->d_orfs, s->d_orf_seq,
                                                                     s->n_orfs, dp, counts, (int32_t*)d_first, d_maxlen);
  ctx->launches++;
  GMG_CUDA(cudaGetLastError());
  if (exclusive_sum_i64_on(ctx, side, counts, s->d_start_off, s->n_orfs + 1)) return 1;
  ctx->h_scalars[0] = 0;
  ctx->h_scalars[1] = 0;
  GMG_CUDA(cudaMemcpyAsync(&ctx->h_scalars[0], s->d_start_off + s->n_orfs, sizeof(int64_t), cudaMemcpyDeviceToHost, side));
  GMG_CUDA(cudaMemcpyAsync(&ctx->h_scalars[1], d_maxlen, sizeof(int), cudaMemcpyDeviceToHost, side));
  GMG_CUDA(cudaEventRecord(ctx->ev_scalars, side));
  if (exact) {
    if (ja < 16)
      k3_g3_heads<16><<<(unsigned)((s->n_orfs * 16 + 127) / 128), 128, 0, side>>>(
          gene->dev, indep->dev, s->d_words, s->d_off, s->d_orfs, s->d_orf_seq, s->n_orfs, dp, counts, ja, heads);
    else
      k3_g3_heads<32><<<(unsigned)((s->n_orfs * 32 + 127) / 128), 128, 0, side>>>(
          gene->dev, indep->dev, s->d_words, s->d_off, s->d_orfs, s->d_orf_seq, s->n_orfs, dp, counts, ja, heads);
    ctx->launches++;
    GMG_CUDA(cudaGetLastError());
  }
  GMG_CUDA(cudaEventRecord(ctx->ev_join, side));

  if (launch_k1(ctx, gene, s, &planes, NULL)) return 1;
  if (exact) {  // K2 (glimmer3 path): codon-boundary cumulative sums, tile by tile
    if (gmg_prof_begin(ctx, GMG_PROF_K2)) return 1;
    k2_g3_codon_cum<<<(unsigned)ntiles, G3_TS, 0, ctx->stream>>>(indep->dev.lut3, s->d_words, s->total, planes,
                                                                s->d_bktidx, cumc, tot3, tileT);
    gmg_prof_end(ctx, GMG_PROF_K2);
    ctx->launches++;
    GMG_CUDA(cudaGetLastError());
  }
  GMG_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
  GMG_CUDA(cudaEventSynchronize(ctx->ev_scalars));
  const int64_t total_starts = ctx->h_scalars[0];
  const int max_orf_len = (int)(ctx->h_scalars[1] & 0xffffffff);
  if (ensure_start_capacity(s, total_starts)) return 1;
  if (total_starts > 0) {
    if (gmg_prof_begin(ctx, GMG_PROF_K3)) return 1;
    if (exact) {
      k3_g3_emit<8><<<(unsigned)((s->n_orfs * 8 + 127) / 128), 128, 0, ctx->stream>>>(
          s->d_words, s->d_cbits, s->nwc, s->d_off, s->d_orfs, s->d_orf_seq, s->n_orfs, cumc, tot3, tileT, heads, ja, cs,
          dp, s->d_start_off, (const int32_t*)d_first, exact_len, s->d_starts);
      ctx->launches++;
    }
    if (max_orf_len > exact_len) {
      k3_g3_ordered<<<(unsigned)((s->n_orfs * 32 + 127) / 128), 128, 0, ctx->stream>>>(
          gene->dev, indep->dev, s->d_words, s->d_off, s->d_orfs, s->d_orf_seq, s->n_orfs, s->total, planes, s->d_bktidx,
          cs, dp, s->d_start_off, (const int32_t*)d_first, exact_len, s->d_starts, s->d_gc + 1);
      ctx->launches++;
    }
    gmg_prof_end(ctx, GMG_PROF_K3);
    GMG_CUDA(cudaGetLastError());
  }
  s->n_starts = total_starts;
  if (n_starts) *n_starts = total_starts;
  return 0;
}

// Plain glimmer-mg (no error branches): K2 and K3 fused into one pass per ORF over the K1 planes
template <bool kPS>
static int score_orfs_mg_plain(gmg_ctx* ctx, const gmg_icm* gene, const DevIcm& indep, const IndepSeqs& X, gmg_seqset* s,
                               const gmg_params* p, const CodonSets& cs, const DevParams& dp, int64_t* n_starts) {
  MgfBatch B;
  memset(&B, 0, sizeof B);
  B.words = s->d_words;
  B.off = s->d_off;
  B.total = s->total;
  B.cb = s->d_cbits;
  B.nwc = s->nwc;
  // The record counts only need the codon bitmaps: they are taken, scanned and their total sent to pinned memory BEFORE
  // the walks are launched, so the host sizes the output while K1 runs and the emission kernel follows K1 without a gap
  // (the stream used to drain between the count and the emission: a host round trip inside every step).
  if (gmg_seqset_ensure_buckets(ctx, s)) return 1;  // here, not inside K1: one host synchronisation serves both
  void* d_counts;
  if (gmg_scratch(ctx, SCR_FLAGS, (size_t)(s->n_orfs + 2) * sizeof(int64_t), &d_counts)) return 1;
  int64_t* counts = (int64_t*)d_counts;
  GMG_CUDA(cudaMemsetAsync(counts + s->n_orfs, 0, 2 * sizeof(int64_t), ctx->stream));
  if (gmg_prof_begin(ctx, GMG_PROF_K3)) return 1;
  void* d_geom;
  if (gmg_scratch(ctx, SCR_MISC, (size_t)(s->n_orfs + 1) * sizeof(PlainDesc), &d_geom)) return 1;
  PlainDesc* geom = (PlainDesc*)d_geom;
  k3_mg_plain_count<<<(unsigned)((s->n_orfs + 127) / 128), 128, 0, ctx->stream>>>(B, dp, s->d_orfs, s->d_orf_seq, s->n_orfs, counts,
                                                                                 geom);
  gmg_prof_end(ctx, GMG_PROF_K3);
  ctx->launches++;
  if (exclusive_sum_i64(ctx, counts, s->d_start_off, s->n_orfs + 1)) return 1;
  ctx->h_scalars[6] = 0;
  GMG_CUDA(cudaMemcpyAsync(&ctx->h_scalars[6], s->d_start_off + s->n_orfs, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaEventRecord(ctx->ev_scalars, ctx->stream));
  float* planes;
  float* side;
  if (launch_k1(ctx, gene, s, &planes, &side)) return 1;
  PlainSide ps;
  ps.t = side;
  ps.w = gene->W;
  IndepSeqs Xo = X;  // the emission kernels find every ORF's sequence here, with either kind of independent model
  Xo.orf_seq = s->d_orf_seq;
  // exactness is certified per ORF inside the kernel; the test hook withdraws every certificate
  const int exact_len = (getenv("GMG_MG_FORCE_UNCERT") && atoi(getenv("GMG_MG_FORCE_UNCERT")) > 0) ? -1 : INT_MAX;
  GMG_CUDA(cudaEventSynchronize(ctx->ev_scalars));
  const int64_t total_starts = ctx->h_scalars[6];
  if (ensure_start_capacity(s, total_starts)) return 1;
  if (total_starts > 0) {
    // one codon per lane for ORFs of up to 384 scored bases: two ORFs per warp up to 192 (every ORF of a 100 bp read set),
    // one beyond; the warp-per-ORF scan for whatever is left.  Test hooks: GMG_PLAIN_LANES=0 sends every ORF through the
    // latter, =1 gives one ORF per warp throughout.
    const int lanes_env = getenv("GMG_PLAIN_LANES") ? atoi(getenv("GMG_PLAIN_LANES")) : 2;
    const int plain_lanes = lanes_env == 0 || lanes_env == 1 ? lanes_env : 2;
    if (gmg_prof_begin(ctx, GMG_PROF_K3)) return 1;
    if (plain_lanes) {
      Which4 which;
      memset(&which, 0, sizeof which);
      for (int cd = 0; cd < 64; cd++)
        which.w[cd >> 4] |= (unsigned long long)(cs.which[cd] < 15 ? cs.which[cd] : 15) << (4 * (cd & 15));
      const int64_t lanes_cap = (int64_t)ctx->sm_count * 8;  // 8 CTAs per SM resident
      unsigned long long* d_nord = (unsigned long long*)(counts + s->n_orfs + 1);
      int done_to = -1;  // ORFs with need <= done_to are taken by an instance launched so far
      // one instance, G lanes per ORF: the ORFs with done_to < need <= 3 * G * 4
      auto launch_lanes = [&](auto kernel, int G) {
        const int64_t need_ctas = (s->n_orfs * G + 127) / 128;
        kernel<<<(unsigned)(need_ctas < lanes_cap ? need_ctas : lanes_cap), 128, 0, ctx->stream>>>(
            indep, planes, ps, s->d_bktidx, B, dp, which, s->n_orfs, s->d_start_off, s->d_starts, exact_len, d_nord, geom, done_to, Xo);
        ctx->launches++;
        done_to = 3 * G * 4;
      };
      if (plain_lanes == 2) launch_lanes(k3_mg_plain_lanes<16, 4, kPS>, 16);
      if (s->max_len > done_to) launch_lanes(k3_mg_plain_lanes<32, 4, kPS>, 32);
    }
    // every ORF taken above?  (need <= orf_len <= max_len; j_lo >= 3 whenever min_gene_len >= 6)
    const bool all_taken = plain_lanes && s->max_len <= 96 * 4 && p->min_gene_len >= 6;
    if (!all_taken) {
      const int slots = (int)(s->max_len / 3 + 4);
      k3_mg_plain<kPS><<<(unsigned)((s->n_orfs * 32 + 127) / 128), 128, (size_t)4 * slots * sizeof(double), ctx->stream>>>(
          indep, X, planes, ps, s->d_bktidx, B, dp, cs, s->d_orfs, s->d_orf_seq, s->n_orfs, s->d_start_off, s->d_starts, exact_len,
          (unsigned long long*)(counts + s->n_orfs + 1), slots, plain_lanes);
      ctx->launches++;
    }
    gmg_prof_end(ctx, GMG_PROF_K3);
    GMG_CUDA(cudaGetLastError());
  }
  s->n_starts = total_starts;
  s->uncert_pending = (unsigned long long*)(counts + s->n_orfs + 1);  // ORFs summed in serial order; read on demand
  if (n_starts) *n_starts = total_starts;
  return 0;
}

// K2 (prefix sums, stop tables, qualities, certificates), then K3: the flat enumeration (k3mg_mode 0) or one thread
// per ORF (1)
template <bool kPS>
static int score_orfs_mg_k2k3(gmg_ctx* ctx, const gmg_icm* gene, const DevIcm& indep, const IndepSeqs& X, gmg_seqset* s,
                              const gmg_params* p, const CodonSets& cs, const DevParams& dp, int k3mg_mode,
                              int64_t* n_starts) {
  float* planes;
  if (launch_k1(ctx, gene, s, &planes, NULL)) return 1;
  // K2
  void *d_cum, *d_tab, *d_qual, *d_cert;
  if (gmg_scratch(ctx, SCR_CUM, (size_t)6 * s->total * sizeof(double), &d_cum)) return 1;
  if (gmg_scratch(ctx, SCR_TMP, (size_t)2 * s->total * sizeof(int32_t), &d_tab)) return 1;
  if (gmg_scratch(ctx, SCR_QUAL, (size_t)s->total + 64, &d_qual)) return 1;
  if (gmg_scratch(ctx, SCR_TMP3, (size_t)s->n + 64 + 520 * sizeof(double), &d_cert)) return 1;
  int32_t* fwd_prev = (int32_t*)d_tab;
  int32_t* rev_next = fwd_prev + s->total;
  // penalty tables (host libm, FP64): indices 0..255 indel penalty, 256..259 stop penalty, 260..515 codon_p
  double* d_tables = (double*)d_cert;
  uint8_t* cert = (uint8_t*)(d_tables + 516);
  if (!ctx->h_penalty) {
    GMG_CUDA(cudaMallocHost(&ctx->h_penalty, 516 * sizeof(double)));
    for (int q = 0; q < 256; q++) {
      double pe = pow(10.0, -(double)q / 10.0);
      ctx->h_penalty[q] = log(pe / 2.0) - log(1.0 - pe);
      ctx->h_penalty[260 + q] = 1.0 - pe;
    }
    for (int t = 0; t < 4; t++) {
      const double dpv = 0.999;
      double ps = dpv;
      ps *= (t & 2) ? (2.0 / 3.0 * dpv + 1.0 / 3.0) : dpv;
      ps *= (t & 1) ? (2.0 / 3.0 * dpv + 1.0 / 3.0) : dpv;
      ctx->h_penalty[256 + t] = log(1.0 - ps) - log(ps);
    }
  }
  GMG_CUDA(cudaMemcpyAsync(d_tables, ctx->h_penalty, 516 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  const bool need_qual = p->allow_indels || p->have_quality_file;
  unsigned g2 = (unsigned)((s->n * 32 + 127) / 128);
  if (gmg_prof_begin(ctx, GMG_PROF_K2)) return 1;
  k2_prefix_lanes<kPS><<<g2, 128, 0, ctx->stream>>>(indep, X, s->d_words, s->d_off, s->n, s->total, planes, s->d_bktidx, cs,
                                                   dp, p->have_quality_file ? s->d_qual : NULL, (double*)d_cum, fwd_prev,
                                                   rev_next, need_qual ? (uint8_t*)d_qual : NULL, cert);
  gmg_prof_end(ctx, GMG_PROF_K2);
  ctx->launches++;
  GMG_CUDA(cudaGetLastError());
  {  // test hook: withdraw every k-th sequence's certificate (exercises the ordered path)
    const char* fu = getenv("GMG_MG_FORCE_UNCERT");
    const int k = fu ? atoi(fu) : 0;
    if (k > 0) {
      k_force_uncert<<<(unsigned)((s->n + 255) / 256), 256, 0, ctx->stream>>>(cert, s->n, k);
      ctx->launches++;
    }
  }

  // ---- K3 ----
  MgfBatch B;
  memset(&B, 0, sizeof B);
  B.words = s->d_words;
  B.off = s->d_off;
  B.total = s->total;
  B.cum = (const double*)d_cum;
  B.fwd_prev = fwd_prev;
  B.rev_next = rev_next;
  B.qual = need_qual ? (const uint8_t*)d_qual : NULL;
  B.cert = cert;
  B.cb = s->d_cbits;
  B.nwc = s->nwc;
  B.tables = d_tables;
  void* d_counts;
  if (gmg_scratch(ctx, SCR_FLAGS, (size_t)(s->n_orfs + 2) * sizeof(int64_t), &d_counts)) return 1;
  int64_t* counts = (int64_t*)d_counts;
  GMG_CUDA(cudaMemsetAsync(counts, 0, (size_t)(s->n_orfs + 2) * sizeof(int64_t), ctx->stream));
  const unsigned g3 = (unsigned)((s->n_orfs + 127) / 128);
  const uint32_t no = (uint32_t)s->n_orfs;
  // Pass_Stop_Penalty with a quality file needs a log per root call: p_stop from the device, glibc's log here
  if (p->allow_subs && p->have_quality_file) {
    void* d_ps;
    if (gmg_scratch(ctx, SCR_MISC, (size_t)no * sizeof(double), &d_ps)) return 1;
    k_mg_sub_pstop<<<g3, 128, 0, ctx->stream>>>(B, dp, s->d_orfs, s->d_orf_seq, no, (double*)d_ps);
    ctx->launches++;
    std::vector<double> h((size_t)no);
    GMG_CUDA(cudaMemcpyAsync(h.data(), d_ps, (size_t)no * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));
    for (uint32_t i = 0; i < no; i++) h[i] = log(1.0 - h[i]) - log(h[i]);  // glimmer-mg.cc:993
    GMG_CUDA(cudaMemcpyAsync(d_ps, h.data(), (size_t)no * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));
    B.sub_pen = (const double*)d_ps;
  }
  MgfWork W;
  memset(&W, 0, sizeof W);
  if (gmg_prof_begin(ctx, GMG_PROF_K3)) return 1;
  if (k3mg_mode == 0) {
    // gates
    const int64_t nblk = s->total / 32 + 2;
    void* d_gate;
    if (gmg_scratch(ctx, SCR_MG_GATE, (size_t)(3 * nblk + s->total + 8) * sizeof(uint32_t), &d_gate)) return 1;
    uint32_t* gate_bits = (uint32_t*)d_gate;
    uint32_t* gate_cnt = gate_bits + nblk;
    uint32_t* gate_rank = gate_cnt + nblk;
    uint32_t* gate_pos = gate_rank + nblk;
    if (p->allow_indels) {
      k_gate_bits<<<(unsigned)((nblk + 255) / 256), 256, 0, ctx->stream>>>((const uint8_t*)d_qual, s->total,
                                                                          dp.indel_q_thresh, nblk, gate_bits, gate_cnt);
      if (exclusive_sum_u32(ctx, gate_cnt, gate_rank, nblk)) return 1;
      k_gate_pos<<<(unsigned)((nblk + 255) / 256), 256, 0, ctx->stream>>>(gate_bits, gate_rank, nblk, gate_pos);
      ctx->launches += 2;
    }
    B.gate_bits = gate_bits;
    B.gate_rank = gate_rank;
    B.gate_pos = gate_pos;
    // level 0
    void *d_root, *d_l0;
    if (gmg_scratch(ctx, SCR_MG_ROOT, (size_t)no * sizeof(MgfCall), &d_root)) return 1;
    if (gmg_scratch(ctx, SCR_MG_L0, (size_t)(3 * ((size_t)no + 1)) * sizeof(uint32_t), &d_l0)) return 1;
    W.orfs = s->d_orfs;
    W.orf_seq = s->d_orf_seq;
    W.n_orfs = no;
    W.root = (MgfCall*)d_root;
    W.n1 = (uint32_t*)d_l0;
    W.off1 = W.n1 + no + 1;
    W.own0 = W.off1 + no + 1;
    W.counts = counts;
    GMG_CUDA(cudaMemsetAsync(W.n1 + no, 0, sizeof(uint32_t), ctx->stream));
    k_mgf_a<<<g3, 128, 0, ctx->stream>>>(B, dp, W);
    ctx->launches++;
    if (exclusive_sum_u32(ctx, W.n1, W.off1, (int64_t)no + 1)) return 1;
    uint32_t* hs = (uint32_t*)&ctx->h_scalars[9];
    GMG_CUDA(cudaMemcpyAsync(hs, W.off1 + no, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));
    W.c1 = hs[0];
    GMG_CHECK(W.c1 < 0x7ffffff0u, "gmg_score_orfs_mg: %u level-1 candidate calls -- split the batch", W.c1);
    // level 1
    void *d_call1, *d_l1;
    if (gmg_scratch(ctx, SCR_MG_CALL1, ((size_t)W.c1 + 1) * sizeof(MgfCall), &d_call1)) return 1;
    if (gmg_scratch(ctx, SCR_MG_L1, (size_t)(6 * ((size_t)W.c1 + 1)) * sizeof(uint32_t), &d_l1)) return 1;
    W.call1 = (MgfCall*)d_call1;
    W.n2 = (uint32_t*)d_l1;
    W.off2 = W.n2 + W.c1 + 1;
    W.own1 = W.off2 + W.c1 + 1;
    W.t1 = W.own1 + W.c1 + 1;
    W.s1 = W.t1 + W.c1 + 1;
    W.par1 = W.s1 + W.c1 + 1;
    GMG_CUDA(cudaMemsetAsync(W.n2 + W.c1, 0, sizeof(uint32_t), ctx->stream));
    GMG_CUDA(cudaMemsetAsync(W.t1 + W.c1, 0, sizeof(uint32_t), ctx->stream));
    if (W.c1) {
      k_mgf_fill<<<(no + 255) / 256, 256, 0, ctx->stream>>>(W.off1, no, W.par1);
      k_mgf_b<<<(W.c1 + 127) / 128, 128, 0, ctx->stream>>>(B, dp, W);
      ctx->launches += 2;
    }
    if (exclusive_sum_u32(ctx, W.n2, W.off2, (int64_t)W.c1 + 1)) return 1;
    GMG_CUDA(cudaMemcpyAsync(hs, W.off2 + W.c1, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));
    W.c2 = hs[0];
    GMG_CHECK(W.c2 < 0x7ffffff0u, "gmg_score_orfs_mg: %u level-2 candidate calls -- split the batch", W.c2);
    // level 2
    void* d_l2;
    if (gmg_scratch(ctx, SCR_MG_L2, (size_t)(3 * ((size_t)W.c2 + 1)) * sizeof(uint32_t), &d_l2)) return 1;
    W.cnt3 = (uint32_t*)d_l2;
    W.s3 = W.cnt3 + W.c2 + 1;
    W.par2 = W.s3 + W.c2 + 1;
    GMG_CUDA(cudaMemsetAsync(W.cnt3 + W.c2, 0, sizeof(uint32_t), ctx->stream));
    if (W.c2) {
      k_mgf_fill<<<(W.c1 + 255) / 256, 256, 0, ctx->stream>>>(W.off2, W.c1, W.par2);
      k_mgf_c<<<(W.c2 + 127) / 128, 128, 0, ctx->stream>>>(B, dp, W);
      ctx->launches += 2;
    }
    if (exclusive_sum_u32(ctx, W.cnt3, W.s3, (int64_t)W.c2 + 1)) return 1;
    if (W.c1) {
      k_mgf_d<<<(W.c1 + 255) / 256, 256, 0, ctx->stream>>>(W);
      ctx->launches++;
    }
    if (exclusive_sum_u32(ctx, W.t1, W.s1, (int64_t)W.c1 + 1)) return 1;
    k_mgf_e<<<(no + 255) / 256, 256, 0, ctx->stream>>>(W);
    ctx->launches++;
    // sequences without a certificate: counted (and later written) in the reference's serial order
    k3_mg_starts<false, kPS><<<g3, 128, 0, ctx->stream>>>(B, s->n_orfs, s->d_orfs, s->d_orf_seq, cs, dp, 1, planes, s->d_bktidx,
                                                     indep, X, counts, NULL, NULL);
    ctx->launches++;
  } else {
    k3_mg_starts<false, kPS><<<g3, 128, 0, ctx->stream>>>(B, s->n_orfs, s->d_orfs, s->d_orf_seq, cs, dp, 0, planes, s->d_bktidx,
                                                     indep, X, counts, NULL, NULL);
    ctx->launches++;
  }
  gmg_prof_end(ctx, GMG_PROF_K3);
  GMG_CUDA(cudaGetLastError());
  k_count_zero_flags<<<(unsigned)((s->n + 255) / 256), 256, 0, ctx->stream>>>(cert, s->n,
                                                                             (unsigned long long*)(counts + s->n_orfs + 1));
  ctx->launches++;
  if (exclusive_sum_i64(ctx, counts, s->d_start_off, s->n_orfs + 1)) return 1;
  ctx->h_scalars[6] = ctx->h_scalars[7] = 0;
  GMG_CUDA(cudaMemcpyAsync(&ctx->h_scalars[6], s->d_start_off + s->n_orfs, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaMemcpyAsync(&ctx->h_scalars[7], counts + s->n_orfs + 1, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  const int64_t total_starts = ctx->h_scalars[6], bad = ctx->h_scalars[7];
  s->uncertified = bad;
  GMG_CHECK(total_starts < 0xfffffff0ll || k3mg_mode != 0, "gmg_score_orfs_mg: %lld start records -- split the batch",
            (long long)total_starts);
  if (ensure_start_capacity(s, total_starts)) return 1;
  if (gmg_prof_begin(ctx, GMG_PROF_K3)) return 1;
  if (total_starts > 0) {
    if (k3mg_mode == 0) {
      W.start_off = s->d_start_off;
      W.starts = s->d_starts;
      k_mgf_w0<kPS><<<g3, 128, 0, ctx->stream>>>(B, dp, cs, W, X);
      ctx->launches++;
      if (W.c1) {
        k_mgf_w1<kPS><<<(W.c1 + 127) / 128, 128, 0, ctx->stream>>>(B, dp, cs, W, X);
        ctx->launches++;
      }
      if (W.c2) {
        k_mgf_w2<kPS><<<(W.c2 + 127) / 128, 128, 0, ctx->stream>>>(B, dp, cs, W, X);
        ctx->launches++;
      }
      if (bad > 0) {
        k3_mg_starts<true, kPS><<<g3, 128, 0, ctx->stream>>>(B, s->n_orfs, s->d_orfs, s->d_orf_seq, cs, dp, 1, planes, s->d_bktidx,
                                                        indep, X, NULL, s->d_start_off, s->d_starts);
        ctx->launches++;
      }
    } else {
      k3_mg_starts<true, kPS><<<g3, 128, 0, ctx->stream>>>(B, s->n_orfs, s->d_orfs, s->d_orf_seq, cs, dp, 0, planes, s->d_bktidx,
                                                      indep, X, NULL, s->d_start_off, s->d_starts);
      ctx->launches++;
    }
  }
  gmg_prof_end(ctx, GMG_PROF_K3);
  GMG_CUDA(cudaGetLastError());
  s->n_starts = total_starts;
  if (n_starts) *n_starts = total_starts;
  return 0;
}

// gmg_score_orfs_mg (kPS = false: one independent model) and gmg_score_orfs_mg_gc (kPS: the model and ignore length of
// every sequence from X); the kernels take the same switch, so the single-model call compiles to the work it always did
template <bool kPS>
static int score_orfs_mg(gmg_ctx* ctx, const gmg_icm* gene, const DevIcm& indep, const IndepSeqs& X, gmg_seqset* s,
                         const gmg_params* p, int64_t* n_starts) {
  CodonSets cs;
  DevParams dp;
  if (make_codon_sets(p, &cs, &dp)) return 1;
  GMG_CHECK(!(p->have_quality_file && !s->d_qual), "have_quality_file set but the seqset has no quality values");
  s->n_starts = 0;
  s->uncertified = 0;
  s->uncert_pending = NULL;
  s->n_red = s->n_red_fallback = 0;
  s->d_red = NULL;
  if (n_starts) *n_starts = 0;
  if (s->n_orfs == 0) return 0;
  GMG_CHECK(s->n_orfs < 0x7fffffffll && s->total < 0xffffffffll, "gmg_score_orfs_mg: batch too large (%lld ORFs): split it",
            (long long)s->n_orfs);
  if (ensure_codon_bits(ctx, s, cs)) return 1;  // start-codon bitmaps: the own starts of every call
  // flat form (0) when calls can branch (-i / -s); without error branches the fused per-ORF scan (2) -- or, for very
  // long sequences and caller-supplied ORF tables, K2 + one thread per ORF (1).  GMG_K3MG_MODE forces a form (tests).
  const int k3mg_env = getenv("GMG_K3MG_MODE") ? atoi(getenv("GMG_K3MG_MODE")) : -1;
  const bool branching = p->allow_indels || p->allow_subs;
  const bool fused_ok = !branching && !s->orfs_external && s->max_len <= 3 * (MGP_SLOTS - 1);
  const int k3mg_mode = k3mg_env >= 0 && !(k3mg_env == 2 && !fused_ok) ? k3mg_env : (branching ? 0 : (fused_ok ? 2 : 1));
  if (k3mg_mode == 2) return score_orfs_mg_plain<kPS>(ctx, gene, indep, X, s, p, cs, dp, n_starts);
  return score_orfs_mg_k2k3<kPS>(ctx, gene, indep, X, s, p, cs, dp, k3mg_mode, n_starts);
}

extern "C" int gmg_score_orfs_mg(gmg_ctx* ctx, const gmg_icm* gene, const gmg_icm* indep, gmg_seqset* s,
                                 const gmg_params* p, int64_t* n_starts) {
  GMG_CHECK(ctx && gene && indep && s && p, "gmg_score_orfs_mg: NULL argument");
  GMG_CHECK(gene->P == 3 && indep->P == 3, "glimmer-mg scoring needs periodicity-3 models");
  if (gmg_icm_ready(gene) || gmg_icm_ready(indep)) return 1;
  IndepSeqs none;
  memset(&none, 0, sizeof none);
  return score_orfs_mg<false>(ctx, gene, indep->dev, none, s, p, n_starts);
}

// glimmer-mg -c: every read scored with the independent model of its own GC fraction (and, optionally, its own
// Ignore_Score_Len).  The GC values are deduplicated by bit pattern in one host pass, one model record per distinct value
// is built on the device (gmg_indep_build), and the kernels of gmg_score_orfs_mg look up the record of each ORF's sequence.
extern "C" int gmg_score_orfs_mg_gc(gmg_ctx* ctx, const gmg_icm* gene, gmg_seqset* s, const double* h_gc,
                                    const int32_t* h_isl, const gmg_params* p, int64_t* n_starts) {
  GMG_CHECK(ctx && gene && s && p && (h_gc || s->n == 0), "gmg_score_orfs_mg_gc: NULL argument");
  GMG_CHECK(gene->P == 3, "glimmer-mg scoring needs periodicity-3 models");
  GMG_CHECK(p->n_stop >= 0 && p->n_stop <= 8, "gmg_score_orfs_mg_gc: %d stop codons", p->n_stop);
  const int64_t n = s->n;
  for (int64_t i = 0; i < n; i++) {
    GMG_CHECK(h_gc[i] >= 0.0 && h_gc[i] <= 1.0, "gmg_score_orfs_mg_gc: sequence %lld: GC fraction %g is not in [0, 1]",
              (long long)i, h_gc[i]);
    GMG_CHECK(!h_isl || h_isl[i] >= 0, "gmg_score_orfs_mg_gc: sequence %lld: negative ignore_score_len %d", (long long)i,
              h_isl ? h_isl[i] : 0);
  }
  if (gmg_icm_ready(gene)) return 1;
  // inputs in one page-locked block: [distinct GC values][model of every sequence][ignore length of every sequence]
  const size_t gc_bytes = (size_t)(n > 0 ? n : 1) * sizeof(double), seq_bytes = (size_t)(n > 0 ? n : 1) * sizeof(int32_t);
  if (gmg_host_stage(ctx, gc_bytes + 2 * seq_bytes, 0)) return 1;
  double* h_uniq = (double*)ctx->h_stage;
  int32_t* h_model = (int32_t*)((char*)ctx->h_stage + gc_bytes);
  int32_t* h_isl_all = h_model + (n > 0 ? n : 1);
  // dedupe by bit pattern: open addressing, table of at least 2 n slots
  int64_t n_models = 0;
  {
    int bits = 4;
    while ((int64_t(1) << bits) < 2 * n) bits++;
    const uint64_t mask = (uint64_t(1) << bits) - 1;
    std::vector<int32_t> slot((size_t)mask + 1, -1);
    for (int64_t i = 0; i < n; i++) {
      uint64_t key;
      memcpy(&key, &h_gc[i], sizeof key);
      uint64_t h = (key * 0x9E3779B97F4A7C15ull) >> (64 - bits);
      for (;; h = (h + 1) & mask) {
        const int32_t m = slot[h];
        if (m < 0) {
          slot[h] = (int32_t)n_models;
          h_uniq[n_models] = h_gc[i];
          h_model[i] = (int32_t)n_models++;
          break;
        }
        uint64_t km;
        memcpy(&km, &h_uniq[m], sizeof km);
        if (km == key) {
          h_model[i] = m;
          break;
        }
      }
      h_isl_all[i] = h_isl ? h_isl[i] : p->ignore_score_len;
    }
  }
  void* d_in;
  if (gmg_scratch(ctx, SCR_INDEP_IN, gc_bytes + 2 * seq_bytes, &d_in)) return 1;
  GMG_CUDA(cudaMemcpyAsync(d_in, ctx->h_stage, (size_t)n_models * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  GMG_CUDA(cudaMemcpyAsync((char*)d_in + gc_bytes, h_model, 2 * seq_bytes, cudaMemcpyHostToDevice, ctx->stream));
  float* d_rec;
  DevIcm base;
  if (gmg_indep_build(ctx, (const double*)d_in, h_uniq, n_models, p, &d_rec, &base)) return 1;
  IndepSeqs X;
  X.rec = d_rec;
  X.model = (const int32_t*)((char*)d_in + gc_bytes);
  X.isl = X.model + (n > 0 ? n : 1);
  X.orf_seq = s->d_orf_seq;
  return score_orfs_mg<true>(ctx, gene, base, X, s, p, n_starts);
}

extern "C" int gmg_reduce_starts_mg(gmg_ctx* ctx, gmg_seqset* s, const gmg_params* p, const gmg_event_model* em,
                                    int64_t* n_kept, int64_t* n_fallback_orfs) {
  GMG_CHECK(ctx && s && p && em, "gmg_reduce_starts_mg: NULL argument");
  GMG_CHECK(em->n_start >= 0 && em->n_start <= 8 && em->n_class >= 1 && em->n_len >= 1 && em->len_lo,
            "gmg_reduce_starts_mg: bad event model (n_start %d, n_class %d, n_len %d)", em->n_start, em->n_class, em->n_len);
  s->n_red = s->n_red_fallback = 0;
  s->d_red = NULL;
  if (n_kept) *n_kept = 0;
  if (n_fallback_orfs) *n_fallback_orfs = 0;
  if (s->n_orfs == 0) return 0;
  const size_t len_bytes = (size_t)em->n_class * 4 * em->n_len * sizeof(double);
  const size_t cls_bytes = em->seq_class ? (size_t)s->n * sizeof(int32_t) : 0;
  const size_t hdr = ((len_bytes + cls_bytes + 128 + 255) / 256) * 256;
  const size_t per_orf = sizeof(int64_t) + sizeof(int32_t) + sizeof(uint32_t) + 1;
  const size_t meta = (((size_t)s->n_orfs * per_orf + 64 + 255) / 256) * 256;
  void* d_red;
  if (gmg_scratch(ctx, SCR_RED, hdr + meta + ((size_t)s->n_starts + 1) * sizeof(gmg_start), &d_red)) return 1;
  char* base = (char*)d_red;
  double* d_len = (double*)base;
  int32_t* d_cls = em->seq_class ? (int32_t*)(base + ((len_bytes + 15) & ~(size_t)15)) : NULL;
  unsigned long long* d_cursor = (unsigned long long*)(base + hdr - 64);
  int64_t* d_first = (int64_t*)(base + hdr);
  int32_t* d_cnt = (int32_t*)(d_first + s->n_orfs);
  uint32_t* d_big = (uint32_t*)(d_cnt + s->n_orfs);
  uint8_t* d_status = (uint8_t*)(d_big + s->n_orfs);
  gmg_start* d_out = (gmg_start*)(base + hdr + meta);
  GMG_CUDA(cudaMemcpyAsync(d_len, em->len_lo, len_bytes, cudaMemcpyHostToDevice, ctx->stream));
  if (d_cls) GMG_CUDA(cudaMemcpyAsync(d_cls, em->seq_class, cls_bytes, cudaMemcpyHostToDevice, ctx->stream));
  GMG_CUDA(cudaMemsetAsync(d_cursor, 0, 64, ctx->stream));
  DevEventModel M;
  M.prior = em->prior;
  M.start_threshold = em->start_threshold;
  M.event_threshold = em->event_threshold;
  M.pwm_bonus_max = em->pwm_bonus_max;
  for (int i = 0; i < 8; i++) M.start_lo[i] = i < em->n_start ? em->start_lo[i] : 0.0;
  M.n_len = em->n_len;
  M.n_class = em->n_class;
  M.min_gene_len = p->min_gene_len;
  M.len_lo = d_len;
  M.seq_class = d_cls;
  // one table slot per start position of a sequence (start records lie inside it); capped at 2 048 per warp
  int slots = (int)(s->max_len + 8);
  if (slots > 2048) slots = 2048;
  const size_t smem = (size_t)4 * slots * sizeof(RedSlot);
  if (smem > 48 * 1024) GMG_CUDA(cudaFuncSetAttribute(k3_mg_reduce, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (gmg_prof_begin(ctx, GMG_PROF_K3)) return 1;
  // GMG_RED_SMALL=0: every ORF through the warp-per-ORF kernel (A/B and test hook)
  const int red_small = getenv("GMG_RED_SMALL") ? atoi(getenv("GMG_RED_SMALL")) : 1;
  if (red_small) {
    k3_mg_reduce_small<<<(unsigned)((s->n_orfs + 127) / 128), 128, 0, ctx->stream>>>(
        s->d_starts, s->d_start_off, s->d_orfs, s->d_orf_seq, s->d_off, s->n_orfs, M, d_out, d_cursor, d_first, d_cnt, d_status,
        d_big, d_cursor + 1);
    // the ORFs with more than RED_SMALL records: a warp each, as many warps as the machine holds
    int64_t ctas = (s->n_orfs * 32 + 127) / 128, cap = (int64_t)ctx->sm_count * 12;
    k3_mg_reduce<<<(unsigned)(ctas < cap ? ctas : cap), 128, smem, ctx->stream>>>(
        s->d_starts, s->d_start_off, s->d_orfs, s->d_orf_seq, s->d_off, s->n_orfs, M, slots, d_out, d_cursor, d_first, d_cnt,
        d_status, d_big, d_cursor + 1);
    ctx->launches++;
  } else {
    k3_mg_reduce<<<(unsigned)((s->n_orfs * 32 + 127) / 128), 128, smem, ctx->stream>>>(
        s->d_starts, s->d_start_off, s->d_orfs, s->d_orf_seq, s->d_off, s->n_orfs, M, slots, d_out, d_cursor, d_first, d_cnt,
        d_status, NULL, NULL);
  }
  gmg_prof_end(ctx, GMG_PROF_K3);
  ctx->launches++;
  GMG_CUDA(cudaGetLastError());
  ctx->h_scalars[10] = 0;
  GMG_CUDA(cudaMemcpyAsync(&ctx->h_scalars[10], d_cursor, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  s->n_red = ctx->h_scalars[10];
  s->d_red = d_out;
  s->d_red_first = d_first;
  s->d_red_cnt = d_cnt;
  s->d_red_status = d_status;
  if (n_kept) *n_kept = s->n_red;
  if (n_fallback_orfs) *n_fallback_orfs = -1;  // counted by the caller from the status bytes
  return 0;
}

extern "C" int gmg_get_reduced_starts(gmg_ctx* ctx, gmg_seqset* s, gmg_start* h_starts, int64_t* h_first, int32_t* h_count,
                                      uint8_t* h_status) {
  GMG_CHECK(ctx && s, "gmg_get_reduced_starts: NULL argument");
  GMG_CHECK(s->d_red != NULL || s->n_orfs == 0, "gmg_get_reduced_starts: no gmg_reduce_starts_mg result on this set");
  if (s->n_orfs == 0) return 0;
  if (h_starts && s->n_red)
    GMG_CUDA(cudaMemcpyAsync(h_starts, s->d_red, (size_t)s->n_red * sizeof(gmg_start), cudaMemcpyDeviceToHost, ctx->stream));
  if (h_first)
    GMG_CUDA(cudaMemcpyAsync(h_first, s->d_red_first, (size_t)s->n_orfs * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (h_count)
    GMG_CUDA(cudaMemcpyAsync(h_count, s->d_red_cnt, (size_t)s->n_orfs * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (h_status)
    GMG_CUDA(cudaMemcpyAsync(h_status, s->d_red_status, (size_t)s->n_orfs, cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int gmg_get_orf_starts(gmg_ctx* ctx, gmg_seqset* s, int64_t orf, gmg_start* h_out, int64_t cap, int64_t* n) {
  GMG_CHECK(ctx && s && n && orf >= 0 && orf < s->n_orfs, "gmg_get_orf_starts: bad argument");
  int64_t lim[2];
  GMG_CUDA(cudaMemcpyAsync(lim, s->d_start_off + orf, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  *n = lim[1] - lim[0];
  if (h_out && *n > 0) {
    GMG_CHECK(*n <= cap, "gmg_get_orf_starts: ORF %lld has %lld records, buffer holds %lld", (long long)orf, (long long)*n,
              (long long)cap);
    GMG_CUDA(cudaMemcpyAsync(h_out, s->d_starts + lim[0], (size_t)*n * sizeof(gmg_start), cudaMemcpyDeviceToHost, ctx->stream));
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  return 0;
}

extern "C" int gmg_get_starts(gmg_ctx* ctx, gmg_seqset* s, gmg_start* h_starts, int64_t* h_start_off) {
  GMG_CHECK(ctx && s, "gmg_get_starts: NULL argument");
  if (h_starts && s->n_starts)
    GMG_CUDA(cudaMemcpyAsync(h_starts, s->d_starts, (size_t)s->n_starts * sizeof(gmg_start), cudaMemcpyDeviceToHost,
                             ctx->stream));
  if (h_start_off) {
    if (s->n_orfs)
      GMG_CUDA(cudaMemcpyAsync(h_start_off, s->d_start_off, (size_t)(s->n_orfs + 1) * sizeof(int64_t),
                               cudaMemcpyDeviceToHost, ctx->stream));
    else
      h_start_off[0] = 0;
  }
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int64_t gmg_uncertified_count(const gmg_seqset* cs) {
  gmg_seqset* s = const_cast<gmg_seqset*>(cs);
  if (!s) return 0;
  if (s->uncert_pending) {  // the fused plain path leaves the counter on the device until somebody asks
    unsigned long long v = 0;
    if (cudaMemcpyAsync(&v, s->uncert_pending, sizeof v, cudaMemcpyDeviceToHost, s->ctx->stream) == cudaSuccess &&
        cudaStreamSynchronize(s->ctx->stream) == cudaSuccess)
      s->uncertified = (int64_t)v;
    s->uncert_pending = NULL;
  }
  return s->uncertified;
}

extern "C" int gmg_ordered_fallback_count(gmg_seqset* s, int64_t* out) {
  GMG_CHECK(s && out, "gmg_ordered_fallback_count: NULL argument");
  unsigned long long v = 0;
  GMG_CUDA(cudaMemcpyAsync(&v, s->d_gc + 1, sizeof v, cudaMemcpyDeviceToHost, s->ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(s->ctx->stream));
  *out = (int64_t)v;
  return 0;
}
