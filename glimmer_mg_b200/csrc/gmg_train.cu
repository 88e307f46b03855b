// glimmer_mg_b200/csrc/gmg_train.cu -- ICM_Training_t: context counting on the device (K4), the
// level-synchronous tree construction around it.
//
// Reference behaviour mirrored (paths relative to /root/reference/src/ICM/):
//   Train_Model                     icm.cc:1356-1463   root counts, root probs (float arithmetic), root MI position
//   Complete_Tree                   icm.cc:1061-1186   per level: count, MI position with the 3 % right bias, prune
//   Count_Char_Pairs                icm.cc:1841-1870   (level 0)
//   Count_Char_Pairs_Restricted     icm.cc:1190-1229   (level >= 1)
//   Get_Training_Node               icm.cc:1233-1256
//   Get_Mutual_Info                 icm.cc:1900-1954
//   Interpolate_Probs               icm.cc:1260-1330
//   Take_Logs                       icm.cc:1334-1352   (logf: float overload, see SURVEY.md section 7)
//
// K4 is the hot part (~90 % of build-icm): every window of every training string walks `level` steps
// down the tree built so far and adds 1 to W-1 pair counters of the node it lands in.  The level's
// count slab [P][4^level][W-1][16] int32 is what gets all-reduced across GPUs; mutual information,
// interpolation and logs are O(nodes) FP64/float arithmetic whose rounding decides the tree topology,
// so they run on the host with the same libm the reference uses (parallel over nodes -- every node's
// arithmetic is independent, so this is bit-identical to the serial loop).
#include <float.h>
#include <math.h>
#include <string.h>

#include <thread>

#include "gmg_internal.cuh"

// device view of one model's training strings (k4_count)
struct K4Seq {
  const uint64_t* words;
  const int64_t* off;
  const int32_t* blk2seq;
  int64_t total;
};
// windows [lo, hi) of model `model`'s strings: one unit of k4_count's work list
struct K4Chunk {
  int64_t lo, hi;
  int32_t model, pad;
};
// corrected result of a flagged node (k4_apply_flagged)
struct K4Fix {
  float prob[4];
  int32_t mip;
};

// A trainer builds M models of one shape (w, d, p, reverse) level by level; gmg_trainer_create makes M = 1 and
// gmg_icm_train_many a group.  Every per-model table is stored as M * P rows ("row" = model * P + period): the level
// finish is per node, so a batch is just more rows.
struct gmg_trainer {
  gmg_ctx* ctx;
  std::vector<gmg_seqset*> seqs;  // [M]
  int M, W, D, P, N, reverse;
  std::vector<int16_t> mip;  // [M * P][N]
  std::vector<float> prob;   // [M * P][N][4] probabilities (logs only after finish)
  std::vector<float> mut_info;  // [M * P][N] mutual information of the chosen position (icm.cc:1156, 1438)
  int8_t* d_mip;             // [M * P][N] current tree (levels not built yet are -1)
  int32_t* d_counts;         // [M][slab] of the level being counted: the trainer's own stream-ordered allocation (no
  size_t counts_cap;         // other call on the context can invalidate it between levels)
  std::vector<K4Seq> h_seqs;    // [M]
  std::vector<K4Chunk> h_chunks;  // k4_count's work list over all M models' windows
  K4Seq* d_seqs;             // device copies, uploaded by the first direct count (NULL before)
  K4Chunk* d_chunks;
  int n_chunks;
  std::vector<int32_t> h_counts;
  int next_level;
  unsigned* d_hist;          // [P][4^W] windows by (frame, content): built once, walked by every level (large sets);
  int hist_ready;            // owned by the trainer like the slab
  // device-side level finish (k4_finish_level): probabilities (not logs) and mutual information of the nodes built so
  // far, per-node results of the level being finished
  float* d_prob;             // [M * P][N][4]
  uint8_t* d_lvl;            // per node of the level: {int8 mip, uint8 flag, float mi, float prob[4]} as SoA, see finish_level
  // multi-GPU (gmg_trainer_set_shard): with the window histogram summed over all ranks, this rank walks cells
  // [cell_lo, cell_hi) of every frame's 4^W cells at every level
  int64_t n_flagged;         // nodes the host had to recompute (decision within the log error bound)
  int rank, world;
  int64_t global_bases;
  gmg_allreduce_fn ar;
  void* ar_user;
};

static inline int64_t level_nodes(int level) {
  int64_t n = 1;
  for (int i = 0; i < level; i++) n *= 4;
  return n;
}
static inline int64_t first_node_of(int level) { return (level_nodes(level) - 1) / 3; }

// add the shared-memory replicas of one model's slab into its global slab
__device__ __forceinline__ void k4_flush_smem(const int* s_cnt, int slab, int copies, int* __restrict__ dst) {
  __syncthreads();
  for (int i = threadIdx.x; i < slab; i += blockDim.x) {
    int v = 0;
    for (int c = 0; c < copies; c++) v += s_cnt[c * slab + i];
    if (v) atomicAdd(dst + i, v);
  }
}

// One thread per window.  A CTA takes chunks blockIdx.x, blockIdx.x + gridDim.x, ... of the work list; a chunk lies in
// one model's strings, and that model's tree rows (mip + model * P * N) and slab (counts + model * slab) are used.
// kSmem: the slab (times `copies` replicas to spread same-address conflicts) lives in shared memory and is flushed
// whenever the CTA moves on to another model, and at the end; otherwise global reductions.
template <bool kSmem>
__global__ void __launch_bounds__(512) k4_count(const K4Seq* __restrict__ seqs, const K4Chunk* __restrict__ chunks,
                                                int n_chunks, int W, int P, int N, int reverse, int level,
                                                int first_node, int nodes_on_level, const int8_t* __restrict__ mip,
                                                int* __restrict__ counts, int slab, int copies) {
  extern __shared__ int s_cnt[];
  int held = -1;  // model whose counts the shared slab holds (kSmem)
  const int wp = W % P;
  for (int c = blockIdx.x; c < n_chunks; c += gridDim.x) {
    const K4Chunk ch = chunks[c];
    if (kSmem && ch.model != held) {  // uniform over the CTA
      if (held >= 0) k4_flush_smem(s_cnt, slab, copies, counts + (size_t)held * slab);
      __syncthreads();
      for (int i = threadIdx.x; i < slab * copies; i += blockDim.x) s_cnt[i] = 0;
      __syncthreads();
      held = ch.model;
    }
    const K4Seq sq = seqs[ch.model];
    const uint64_t* __restrict__ words = sq.words;
    const int64_t* __restrict__ off = sq.off;
    const int32_t* __restrict__ blk2seq = sq.blk2seq;
    int* mine = kSmem ? s_cnt + ((threadIdx.x >> 5) % copies) * slab : counts + (size_t)ch.model * slab;
    const int8_t* mm = mip + (size_t)ch.model * P * N;
    for (int64_t p = ch.lo + threadIdx.x; p < ch.hi; p += blockDim.x) {
      int32_t s = __ldg(blk2seq + (p >> 5)) & 0x7FFFFFFF;
      while (p >= __ldg(off + s + 1)) s++;
      const int64_t a = __ldg(off + s);
      const int len = (int)(__ldg(off + s + 1) - a);
      const int q = (int)(p - a);
      uint64_t ctx;
      int t;  // window start in the (possibly reversed) training string
      if (!reverse) {
        if (q + W > len) continue;
        t = q;
        ctx = gmg_extract32(words, p);  // window position k <-> s[q + k]
      } else {
        if (q - (W - 1) < 0) continue;
        t = len - 1 - q;
        ctx = gmg_reverse_bases(gmg_extract32(words, p - (W - 1)), W);  // window position k <-> s[q - k]
      }
      const int f = (wp + t) % P;
      int node = 0;
      bool ok = true;
      const int8_t* mf = mm + (size_t)f * N;
      for (int i = 0; i < level; i++) {
        int j = mf[node];
        if (j < 0) {
          ok = false;
          break;
        }
        node = 4 * node + (int)((ctx >> (2 * j)) & 3) + 1;
      }
      if (!ok) continue;
      const int last = (int)((ctx >> (2 * (W - 1))) & 3);
      int* row = mine + ((size_t)f * nodes_on_level + (node - first_node)) * (W - 1) * 16 + last;
      for (int i = 0; i < W - 1; i++) {
        int b = (int)((ctx >> (2 * i)) & 3);
        atomicAdd(row + i * 16 + 4 * b, 1);
      }
    }
  }
  if (kSmem && held >= 0) k4_flush_smem(s_cnt, slab, copies, counts + (size_t)held * slab);
}

// ---- large training sets: one pass over the strings, then every level walks the DISTINCT windows -------------
// hist[f][window content] = number of training windows of frame f with that content (W <= 12: 3 * 4^12 cells =
// 201 MB).  A level pass then visits one cell per thread instead of one window per thread -- 10x fewer walks at
// 500 Mbp -- and adds the cell's multiplicity.  Counts are sums of the same +1 events, so the slab is identical.
__global__ void __launch_bounds__(512) k4_hist_build(const uint64_t* __restrict__ words, const int64_t* __restrict__ off,
                                                     const int32_t* __restrict__ blk2seq, int64_t total, int W, int P,
                                                     int reverse, unsigned* __restrict__ hist) {
  const int wp = W % P;
  const size_t cells = (size_t)1 << (2 * W);
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += (int64_t)gridDim.x * blockDim.x) {
    int32_t s = __ldg(blk2seq + (p >> 5)) & 0x7FFFFFFF;
    while (p >= __ldg(off + s + 1)) s++;
    const int64_t a = __ldg(off + s);
    const int len = (int)(__ldg(off + s + 1) - a);
    const int q = (int)(p - a);
    uint64_t ctx;
    int t;
    if (!reverse) {
      if (q + W > len) continue;
      t = q;
      ctx = gmg_extract32(words, p);
    } else {
      if (q - (W - 1) < 0) continue;
      t = len - 1 - q;
      ctx = gmg_reverse_bases(gmg_extract32(words, p - (W - 1)), W);
    }
    const int f = (wp + t) % P;
    atomicAdd(hist + (size_t)f * cells + (size_t)(ctx & (cells - 1)), 1u);
  }
}

// One thread per histogram cell.  Consecutive cells differ only in window positions 0..2 (bits 0..5), so the 32
// cells of a warp usually land in the same node and share the bases at positions >= 3 and the predicted base:
// those W-1-3 counters get ONE atomic per warp (the warp's summed multiplicity); positions 0..2 add per lane.
template <bool kSmem>
__global__ void __launch_bounds__(512) k4_hist_level(const unsigned* __restrict__ hist, int W, int P, int N, int level,
                                                     int first_node, int nodes_on_level, const int8_t* __restrict__ mip,
                                                     int* __restrict__ counts, int slab, int copies, int64_t g_lo,
                                                     int64_t g_hi) {
  extern __shared__ int s_cnt[];
  if (kSmem) {
    for (int i = threadIdx.x; i < slab * copies; i += blockDim.x) s_cnt[i] = 0;
    __syncthreads();
  }
  int* mine = kSmem ? s_cnt + ((threadIdx.x >> 5) % copies) * slab : counts;
  const int64_t cells = (int64_t)1 << (2 * W);
  const int64_t all = cells * P;
  const int lane = threadIdx.x & 31;
  // this rank's share [g_lo, g_hi) of the P * 4^W cells (multiples of 32: whole warps)
  for (int64_t g0 = g_lo + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) & ~31ll); g0 < g_hi; g0 += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = g0 + lane;  // cells is a multiple of 32 (W >= 3, checked by the caller): a warp never straddles two frames
    const unsigned cnt = g < g_hi && g < all ? __ldg(hist + g) : 0u;
    if (__ballot_sync(0xffffffffu, cnt != 0) == 0) continue;
    const int f = g < all ? (int)(g / cells) : 0;
    const uint64_t ctx = (uint64_t)(g - (int64_t)f * cells);
    int node = 0;
    bool ok = true;
    const int8_t* mf = mip + (size_t)f * N;
    for (int i = 0; i < level; i++) {
      const int j = mf[node];
      if (j < 0) {
        ok = false;
        break;
      }
      node = 4 * node + (int)((ctx >> (2 * j)) & 3) + 1;
    }
    const int last = (int)((ctx >> (2 * (W - 1))) & 3);
    const int c = ok ? (int)cnt : 0;
    int* row = mine + ((size_t)f * nodes_on_level + (ok ? node - first_node : 0)) * (W - 1) * 16 + last;
    const int node0 = __shfl_sync(0xffffffffu, ok ? node : -1, 0);
    const bool uniform = __all_sync(0xffffffffu, (ok ? node : -1) == node0);
    if (uniform) {
      if (node0 < 0) continue;
      const int sum = __reduce_add_sync(0xffffffffu, c);
      const int lo = W - 1 < 3 ? W - 1 : 3;
      if (c)
        for (int i = 0; i < lo; i++) atomicAdd(row + i * 16 + 4 * (int)((ctx >> (2 * i)) & 3), c);
      if (lane == 0 && sum)
        for (int i = 3; i < W - 1; i++) atomicAdd(row + i * 16 + 4 * (int)((ctx >> (2 * i)) & 3), sum);
    } else if (c) {
      for (int i = 0; i < W - 1; i++) atomicAdd(row + i * 16 + 4 * (int)((ctx >> (2 * i)) & 3), c);
    }
  }
  if (kSmem) {
    __syncthreads();
    for (int i = threadIdx.x; i < slab; i += blockDim.x) {
      int v = 0;
      for (int c = 0; c < copies; c++) v += s_cnt[c * slab + i];
      if (v) atomicAdd(counts + i, v);
    }
  }
}


// ---- level finish on the device ---------------------------------------------------------------------------------
// Position choice (Get_Mutual_Info, the >= / 3 % right-bias rule, pruning) and Interpolate_Probs for every node of a
// level, one thread per node, straight from the (all-reduced) count slab -- so that only 22 bytes per node instead of
// the 704-byte count table cross PCIe and the host is out of the level loop.
//
// Bit-exactness: everything but the 16 x (W-1) logarithms is IEEE +, -, *, / on the same operands in the reference's
// order (the library is built with --fmad=false), identical on host and device.  The device's log differs from
// glibc's in the last bits, so every DECISION that a mutual-information value enters carries an error bound
// (sum of |terms| x 2^-46 covers both libraries' log error and the reordered rounding): the node's result is used
// only if every comparison -- next >= best, next >= best / 1.03, best <= 1e-4, and the float rounding of the stored
// mut_info -- has a margin larger than the bounds; otherwise the node is FLAGGED and the host recomputes it from its
// counts with glibc exactly as the reference does (gmg_trainer_finish_level).  GMG_K4_MI=0 sends every node to the
// host (the round-1 path; the tests hold both to the same model bytes).
struct MiVal {
  double v, err;
};
__device__ MiVal k4_mutual_info16(const int32_t* __restrict__ ct, int sum) {
  MiVal r;
  r.v = 0.0;
  r.err = 0.0;
  if (sum == 0) return r;
  double left[4] = {0, 0, 0, 0}, right[4] = {0, 0, 0, 0};
  int c[16];
#pragma unroll
  for (int k = 0; k < 16; k++) c[k] = __ldg(ct + k);
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) {
      left[i] += c[4 * i + j];
      right[j] += c[4 * i + j];
    }
#pragma unroll
  for (int i = 0; i < 4; i++) {
    left[i] /= sum;
    right[i] /= sum;
  }
  double abs_sum = 0.0;
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const double pr = double(c[4 * i + j]) / sum;
      if (pr != 0.0 && left[i] != 0.0 && right[j] != 0.0) {
        const double t = pr * log(pr / (left[i] * right[j]));
        r.v += t;
        abs_sum += fabs(t);
      }
    }
  r.err = abs_sum * 1.5e-14;  // 2^-46: ~6x the worst case of both libraries' log error plus the reordered rounding
  return r;
}

// One thread per node of the level in every row (row = model * P + period: counts [rows][nl][W-1][16], mip [rows][N],
// prob [rows][N][4]), so one launch finishes the level of every model of a trainer.
__global__ void __launch_bounds__(128) k4_finish_level(const int32_t* __restrict__ counts, int W, int rows, int N, int level,
                                                       int first, int nl, int8_t* __restrict__ mip, float* __restrict__ prob,
                                                       int8_t* __restrict__ o_mip, uint8_t* __restrict__ o_flag,
                                                       float* __restrict__ o_mi, float* __restrict__ o_prob, int force_flag) {
  const int it = blockIdx.x * blockDim.x + threadIdx.x;
  if (it >= rows * nl) return;
  const int f = it / nl, local = it - f * nl, sub = first + local;
  const int32_t* nc = counts + (size_t)it * (W - 1) * 16;
  int8_t* mp = mip + (size_t)f * N + sub;
  float* pr = prob + ((size_t)f * N + sub) * 4;
  int out_mip = 0;
  float out_mi = 0.f, p4[4] = {0.f, 0.f, 0.f, 0.f};
  bool flag = false;
  const int par = level > 0 ? (sub - 1) / 4 : 0;
  if (level > 0 && mip[(size_t)f * N + par] < 0) {
    out_mip = -2;  // stopped at the parent (icm.cc:1104-1109)
  } else {
    int final_ct[4] = {0, 0, 0, 0}, sum = 0;
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int v = __ldg(nc + 4 * i + j);
        sum += v;
        final_ct[j] += v;
      }
    // choose_position with error bounds
    int max_pos = 0;
    MiVal best = k4_mutual_info16(nc, sum), used = best;
    for (int i = 1; i < W - 1; i++) {
      const MiVal next = k4_mutual_info16(nc + 16 * i, sum);
      const double tol = next.err + best.err;
      if (fabs(next.v - best.v) <= tol && !(next.v == best.v && tol == 0.0)) flag = true;
      if (next.v >= best.v) {
        used = best = next;
        max_pos = i;
      } else {
        const double thr = best.v / (1.0 + 0.03);
        if (fabs(next.v - thr) <= tol) flag = true;
        if (next.v >= thr) {  // MUT_INFO_BIAS: prefer positions to the right
          max_pos = i;
          used = next;
        }
      }
    }
    const MiVal kept = level == 0 ? best : used;  // root keeps the maximum (icm.cc:1438)
    out_mi = (float)kept.v;
    if ((float)(kept.v - kept.err) != out_mi || (float)(kept.v + kept.err) != out_mi) flag = true;
    if (level == 0) {
      for (int j = 0; j < 4; j++) p4[j] = ((float)final_ct[j] + float(0.001 / 4)) / float(sum + 0.001);  // icm.cc:1411-1413
    } else {
      if (sum < 400) {
        if (fabs(best.v - 1e-4) <= best.err) flag = true;
        if (best.v <= 1e-4) max_pos = -1;  // MUT_INFO_EPSILON, SAMPLE_SIZE_BOUND
      }
      // Interpolate_Probs (icm.cc:1260-1330)
      const float* pp = prob + ((size_t)f * N + par) * 4;
      const float q4[4] = {pp[0], pp[1], pp[2], pp[3]};
      double total = 0.0;
      for (int i = 0; i < 4; i++) total += final_ct[i];
      for (int i = 0; i < 4; i++) p4[i] = (float)((final_ct[i] + 0.001 * q4[i]) / (total + 0.001));
      if (total < 400) {
        const float cv[7] = {2.37f, 4.11f, 6.25f, 7.81f, 9.35f, 11.3f, 12.8f};
        const float cs[7] = {0.50f, 0.75f, 0.90f, 0.95f, 0.975f, 0.99f, 0.995f};
        double chi2 = 0.0;
        for (int i = 0; i < 4; i++) {
          const double expected = total * q4[i];
          if (expected > 0.0) {
            const double dd = final_ct[i] - expected;
            chi2 += (dd * dd) / expected;  // pow(x, 2.0) is folded to x * x by the host compiler as well
          }
        }
        int i = 0;
        while (i < 7 && cv[i] < chi2) i++;
        double lambda;
        if (i == 0) lambda = 0.0;
        else if (i == 7) lambda = 1.0;
        else lambda = cs[i - 1] + ((chi2 - cv[i - 1]) / (cv[i] - cv[i - 1])) * (cs[i] - cs[i - 1]);
        lambda *= total / 400;
        if (lambda > 1.0) lambda = 1.0;
        for (int k = 0; k < 4; k++) {
          p4[k] = (float)(p4[k] * lambda);  // two float stores, like the reference (icm.cc:1324-1326)
          p4[k] = (float)(p4[k] + (1.0 - lambda) * q4[k]);
        }
      }
    }
    out_mip = max_pos;
  }
  if (force_flag && out_mip != -2) flag = true;
  *mp = (int8_t)out_mip;
  pr[0] = p4[0]; pr[1] = p4[1]; pr[2] = p4[2]; pr[3] = p4[3];
  o_mip[it] = (int8_t)out_mip;
  o_flag[it] = flag ? 1 : 0;
  o_mi[it] = out_mi;
  o_prob[4 * (size_t)it + 0] = p4[0];
  o_prob[4 * (size_t)it + 1] = p4[1];
  o_prob[4 * (size_t)it + 2] = p4[2];
  o_prob[4 * (size_t)it + 3] = p4[3];
}

// the count tables of the flagged nodes (item = row * nl + node of the level) into one compact buffer
__global__ void __launch_bounds__(256) k4_gather_flagged(const int32_t* __restrict__ counts, const int64_t* __restrict__ items,
                                                         int64_t n, int per, int32_t* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n * per; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t k = i / per;
    out[i] = counts[items[k] * per + (i - k * per)];
  }
}

// the host's results for the flagged nodes into the device tree
__global__ void __launch_bounds__(256) k4_apply_flagged(const int64_t* __restrict__ items, const K4Fix* __restrict__ fix,
                                                        int64_t n, int nl, int first, int N, int8_t* __restrict__ mip,
                                                        float* __restrict__ prob) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    const int64_t it = items[k];
    const size_t at = (size_t)(it / nl) * N + first + (size_t)(it % nl);
    mip[at] = (int8_t)fix[k].mip;
    for (int j = 0; j < 4; j++) prob[at * 4 + j] = fix[k].prob[j];
  }
}

// the host's share of training: up to 32 threads over n independent items (nodes or models); below `serial_below`
// items, one thread
template <class F>
static void host_parallel(int64_t n, int64_t serial_below, F work) {
  unsigned hw = std::thread::hardware_concurrency();
  int nthreads = (int)(hw ? hw : 1);
  if (nthreads > 32) nthreads = 32;
  if (n < serial_below) nthreads = 1;
  else if (nthreads > n) nthreads = (int)n;
  if (nthreads <= 1) {
    if (n > 0) work((int64_t)0, n);
    return;
  }
  std::vector<std::thread> pool;
  int64_t chunk = (n + nthreads - 1) / nthreads;
  for (int i = 0; i < nthreads; i++) {
    int64_t lo = i * chunk, hi = lo + chunk < n ? lo + chunk : n;
    if (lo < hi) pool.emplace_back(work, lo, hi);
  }
  for (auto& th : pool) th.join();
}

static int check_shape(int w, int d, int p) {
  GMG_CHECK(w >= 2 && w <= GMG_MAX_W, "training: model_len %d unsupported (2..%d)", w, GMG_MAX_W);
  GMG_CHECK(d >= 1 && d <= GMG_MAX_DEPTH && d <= w - 1, "training: model_depth %d unsupported", d);
  GMG_CHECK(p >= 1 && p <= 16, "training: periodicity %d unsupported", p);
  return 0;
}

// counting route: the window histogram for large sets (W <= 12); GMG_K4_HIST=0/1 forces the direct / histogram path
// (tests).  W >= 3: 4^W cells per frame must be a multiple of the warp size, see k4_hist_level.
static bool k4_use_hist(int W, int P, int64_t bases) {
  const char* hist_env = getenv("GMG_K4_HIST");
  const int hist_mode = hist_env ? atoi(hist_env) : -1;
  return W >= 3 && W <= 12 && (hist_mode == 1 || (hist_mode < 0 && bases >= ((int64_t)P << (2 * W)) / 2));  // >= 25 M windows at 12/7/3
}

// device bytes of one model in a trainer: deepest count slab, tree, probabilities, level results
static size_t trainer_model_bytes(int w, int d, int p) {
  const size_t n = (size_t)((level_nodes(d + 1) - 1) / 3);
  return (size_t)p * level_nodes(d) * ((w - 1) * 16 * sizeof(int32_t) + 24) + (size_t)p * n * (1 + 4 * sizeof(float));
}

// a trainer of M models of one shape, one seqset each (the same seqset may appear more than once)
static int trainer_create(gmg_ctx* ctx, gmg_seqset* const* sets, int M, int w, int d, int p, int reverse, gmg_trainer** out) {
  GMG_CHECK(ctx && sets && out && M >= 1, "gmg_trainer_create: NULL argument");
  for (int k = 0; k < M; k++) GMG_CHECK(sets[k], "gmg_trainer_create: NULL argument");
  if (check_shape(w, d, p)) return 1;
  gmg_trainer* t = new gmg_trainer();
  t->ctx = ctx;
  t->seqs.assign(sets, sets + M);
  t->M = M;
  t->W = w; t->D = d; t->P = p; t->reverse = reverse;
  t->N = (int)((level_nodes(d + 1) - 1) / 3);
  const size_t rows = (size_t)M * p;
  t->mip.assign(rows * t->N, 0);
  t->prob.assign(rows * t->N * 4, 0.0f);
  t->mut_info.assign(rows * t->N, 0.0f);
  t->d_mip = NULL;
  t->d_counts = NULL;
  t->counts_cap = 0;
  t->d_seqs = NULL;
  t->d_chunks = NULL;
  t->n_chunks = 0;
  t->next_level = 0;
  t->d_hist = NULL;
  t->hist_ready = 0;
  t->d_prob = NULL;
  t->d_lvl = NULL;
  t->n_flagged = 0;
  t->rank = 0;
  t->world = 1;
  t->global_bases = -1;
  t->ar = NULL;
  t->ar_user = NULL;
  if (cudaSetDevice(ctx->device) != cudaSuccess) {
    gmg_set_error("gmg_trainer_create: cannot select device %d", ctx->device);
    delete t;
    return 1;
  }
  // k4_count's work list: each model's windows in chunks of at least 512, at most 4 per SM -- the split a model alone
  // gets, so that the CTAs in flight sweep about one model (and one model's slab in L2) at a time
  std::vector<K4Seq>& hs = t->h_seqs;
  std::vector<K4Chunk>& hc = t->h_chunks;
  hs.resize((size_t)M);
  const int64_t per_sm = (int64_t)ctx->sm_count * 4;
  for (int k = 0; k < M; k++) {
    hs[k] = {sets[k]->d_words, sets[k]->d_off, sets[k]->d_blk2seq, sets[k]->total};
    int64_t chunk = (hs[k].total + per_sm - 1) / per_sm;
    if (chunk < 512) chunk = 512;
    for (int64_t lo = 0; lo < hs[k].total; lo += chunk)
      hc.push_back({lo, lo + chunk < hs[k].total ? lo + chunk : hs[k].total, k, 0});
  }
  t->n_chunks = (int)hc.size();
  // the count slab (and the window histogram) are the trainer's own allocations from the stream-ordered pool (the
  // pool keeps freed blocks, so a model costs no cudaMalloc / cudaFree); context scratch would be invalidated by any
  // other call on the context between two levels of the step API
  const size_t cap = (size_t)p * level_nodes(d) * (w - 1) * 16;
  const size_t lvl_bytes = rows * level_nodes(d) * 24 + 256;  // deepest level: 1 + 1 + 4 + 16 bytes per node, padded
  if (cudaMallocAsync(&t->d_counts, (size_t)M * cap * sizeof(int32_t), ctx->stream) != cudaSuccess) {
    gmg_set_error("gmg_trainer_create: cannot allocate the %zu-byte count slab", (size_t)M * cap * sizeof(int32_t));
    t->d_counts = NULL;
    gmg_trainer_free(t);
    return 1;
  }
  t->counts_cap = cap;
  if (cudaMallocAsync(&t->d_mip, rows * t->N, ctx->stream) != cudaSuccess ||
      cudaMallocAsync(&t->d_prob, rows * t->N * 4 * sizeof(float), ctx->stream) != cudaSuccess ||
      cudaMallocAsync(&t->d_lvl, lvl_bytes, ctx->stream) != cudaSuccess) {
    gmg_set_error("gmg_trainer_create: cannot allocate the level buffers");
    gmg_trainer_free(t);
    return 1;
  }
  GMG_CUDA(cudaMemsetAsync(t->d_mip, 0xFF, rows * t->N, ctx->stream));
  GMG_CUDA(cudaMemsetAsync(t->d_prob, 0, rows * t->N * 4 * sizeof(float), ctx->stream));
  *out = t;
  return 0;
}

extern "C" int gmg_trainer_create(gmg_ctx* ctx, gmg_seqset* s, int w, int d, int p, int reverse, gmg_trainer** out) {
  GMG_CHECK(ctx && s && out, "gmg_trainer_create: NULL argument");
  return trainer_create(ctx, &s, 1, w, d, p, reverse, out);
}

// Multi-GPU training: this rank holds 1 / world of the training strings.  With the window histogram (large sets) the
// histogram is summed over the ranks ONCE (`ar`, an in-place int32 sum as for the level slabs) and every rank then
// walks only its 1 / world share of the histogram cells at every level, so the per-level work shrinks with the number of
// GPUs; the level slabs are summed across ranks by the caller as before (gmg_trainer_count_level's pointer) or, through
// gmg_icm_train, by the same callback.
extern "C" int gmg_trainer_set_shard(gmg_trainer* t, int rank, int world, int64_t global_bases, gmg_allreduce_fn ar,
                                     void* user) {
  GMG_CHECK(t && world >= 1 && rank >= 0 && rank < world, "gmg_trainer_set_shard: bad rank %d / world %d", rank, world);
  GMG_CHECK(world == 1 || ar != NULL, "gmg_trainer_set_shard: world %d needs an all-reduce callback", world);
  GMG_CHECK(t->next_level == 0 && !t->hist_ready, "gmg_trainer_set_shard: call before the first level is counted");
  t->rank = rank;
  t->world = world;
  t->global_bases = global_bases;  // the same number on every rank: all ranks must take the same counting path
  t->ar = ar;
  t->ar_user = user;
  return 0;
}

extern "C" void gmg_trainer_free(gmg_trainer* t) {
  if (!t) return;
  cudaSetDevice(t->ctx->device);
  if (t->d_mip) cudaFreeAsync(t->d_mip, t->ctx->stream);
  if (t->d_counts) cudaFreeAsync(t->d_counts, t->ctx->stream);
  if (t->d_hist) cudaFreeAsync(t->d_hist, t->ctx->stream);
  if (t->d_prob) cudaFreeAsync(t->d_prob, t->ctx->stream);
  if (t->d_lvl) cudaFreeAsync(t->d_lvl, t->ctx->stream);
  if (t->d_seqs) cudaFreeAsync(t->d_seqs, t->ctx->stream);
  if (t->d_chunks) cudaFreeAsync(t->d_chunks, t->ctx->stream);
  delete t;
}

extern "C" int gmg_trainer_count_level(gmg_trainer* t, int level, void** d_counts, int64_t* n_counts) {
  GMG_CHECK(t, "gmg_trainer_count_level: NULL trainer");
  GMG_CHECK(level == t->next_level && level <= t->D, "gmg_trainer_count_level: level %d out of order (next %d)", level,
            t->next_level);
  gmg_ctx* ctx = t->ctx;
  gmg_seqset* s = t->seqs[0];
  const int64_t nl = level_nodes(level);
  const int64_t slab = (int64_t)t->P * nl * (t->W - 1) * 16;  // one model's
  GMG_CUDA(cudaMemsetAsync(t->d_counts, 0, (size_t)slab * t->M * sizeof(int32_t), ctx->stream));
  // window histogram for large sets: a single model only (gmg_icm_train_many routes such models to gmg_icm_train)
  const bool use_hist = t->M == 1 && k4_use_hist(t->W, t->P, t->global_bases >= 0 ? t->global_bases : s->total);
  if (s->total > 0 && use_hist) {
    const size_t cells = (size_t)t->P << (2 * t->W);
    const int threads = 512;
    if (gmg_prof_begin(ctx, GMG_PROF_K4)) return 1;
    if (!t->hist_ready) {
      if (!t->d_hist) GMG_CUDA(cudaMallocAsync(&t->d_hist, cells * sizeof(unsigned), ctx->stream));
      GMG_CUDA(cudaMemsetAsync(t->d_hist, 0, cells * sizeof(unsigned), ctx->stream));
      int64_t need = (s->total + threads - 1) / threads;
      int64_t cap = (int64_t)ctx->sm_count * 4;
      k4_hist_build<<<(int)(need < cap ? need : cap), threads, 0, ctx->stream>>>(s->d_words, s->d_off, s->d_blk2seq, s->total,
                                                                              t->W, t->P, t->reverse, t->d_hist);
      ctx->launches++;
      t->hist_ready = 1;
      if (t->world > 1) {  // the one exchange of the histogram: afterwards every rank holds the windows of ALL strings
        GMG_CHECK(t->ar(t->ar_user, t->d_hist, (int64_t)cells, (void*)ctx->stream) == 0,
                  "gmg_trainer_count_level: all-reduce of the window histogram failed");
      }
    }
    // this rank's share of the cells (whole warps); world == 1: all of them
    const int64_t per = (((int64_t)cells + t->world - 1) / t->world + 31) & ~31ll;
    const int64_t g_lo = t->world > 1 ? per * t->rank : 0;
    int64_t g_hi = t->world > 1 ? g_lo + per : (int64_t)cells;
    if (g_hi > (int64_t)cells) g_hi = (int64_t)cells;
    const int64_t my_cells = g_hi > g_lo ? g_hi - g_lo : 0;
    const size_t smem_budget = 200 * 1024;
    const bool use_smem = (size_t)slab * sizeof(int) <= smem_budget;
    int64_t need = (my_cells + threads - 1) / threads;
    if (need < 1) need = 1;
    if (use_smem) {
      int copies = (int)(smem_budget / ((size_t)slab * sizeof(int)));
      if (copies > threads / 32) copies = threads / 32;
      if (copies < 1) copies = 1;
      size_t smem = (size_t)slab * copies * sizeof(int);
      GMG_CUDA(cudaFuncSetAttribute(k4_hist_level<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      int grid = (int)(need < ctx->sm_count ? need : ctx->sm_count);
      k4_hist_level<true><<<grid, threads, smem, ctx->stream>>>(t->d_hist, t->W, t->P, t->N, level, (int)first_node_of(level),
                                                               (int)nl, t->d_mip, t->d_counts, (int)slab, copies, g_lo, g_hi);
    } else {
      int64_t cap = (int64_t)ctx->sm_count * 4;
      k4_hist_level<false><<<(int)(need < cap ? need : cap), threads, 0, ctx->stream>>>(
          t->d_hist, t->W, t->P, t->N, level, (int)first_node_of(level), (int)nl, t->d_mip, t->d_counts, (int)slab, 1, g_lo,
          g_hi);
    }
    gmg_prof_end(ctx, GMG_PROF_K4);
    ctx->launches++;
    GMG_CUDA(cudaGetLastError());
  } else if (t->n_chunks > 0) {
    // one launch over every window of every model (the work list of trainer_create)
    if (!t->d_seqs) {  // pageable sources: the copies have read them when they return
      GMG_CUDA(cudaMallocAsync(&t->d_seqs, t->h_seqs.size() * sizeof(K4Seq), ctx->stream));
      GMG_CUDA(cudaMallocAsync(&t->d_chunks, t->h_chunks.size() * sizeof(K4Chunk), ctx->stream));
      GMG_CUDA(cudaMemcpyAsync(t->d_seqs, t->h_seqs.data(), t->h_seqs.size() * sizeof(K4Seq), cudaMemcpyHostToDevice,
                               ctx->stream));
      GMG_CUDA(cudaMemcpyAsync(t->d_chunks, t->h_chunks.data(), t->h_chunks.size() * sizeof(K4Chunk), cudaMemcpyHostToDevice,
                               ctx->stream));
    }
    const size_t smem_budget = 200 * 1024;
    const bool use_smem = (size_t)slab * sizeof(int) <= smem_budget;
    const int threads = 512;
    if (gmg_prof_begin(ctx, GMG_PROF_K4)) return 1;
    if (use_smem) {
      int copies = (int)(smem_budget / ((size_t)slab * sizeof(int)));
      if (copies > threads / 32) copies = threads / 32;
      if (copies < 1) copies = 1;
      size_t smem = (size_t)slab * copies * sizeof(int);
      GMG_CUDA(cudaFuncSetAttribute(k4_count<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      int grid = t->n_chunks < ctx->sm_count ? t->n_chunks : ctx->sm_count;
      k4_count<true><<<grid, threads, smem, ctx->stream>>>(t->d_seqs, t->d_chunks, t->n_chunks, t->W, t->P, t->N, t->reverse,
                                                          level, (int)first_node_of(level), (int)nl, t->d_mip, t->d_counts,
                                                          (int)slab, copies);
    } else {
      int64_t cap = (int64_t)ctx->sm_count * 4;
      int grid = (int)(t->n_chunks < cap ? t->n_chunks : cap);
      k4_count<false><<<grid, threads, 0, ctx->stream>>>(t->d_seqs, t->d_chunks, t->n_chunks, t->W, t->P, t->N, t->reverse,
                                                        level, (int)first_node_of(level), (int)nl, t->d_mip, t->d_counts,
                                                        (int)slab, 1);
    }
    gmg_prof_end(ctx, GMG_PROF_K4);
    ctx->launches++;
    GMG_CUDA(cudaGetLastError());
  }
  if (d_counts) *d_counts = t->d_counts;
  if (n_counts) *n_counts = slab;
  return 0;
}

// Get_Mutual_Info for a 4x4 table (icm.cc:1900-1954)
static double mutual_info16(const int32_t* ct, int sum) {
  if (sum == 0) return 0.0;
  double left[4] = {0, 0, 0, 0}, right[4] = {0, 0, 0, 0}, mi = 0.0;
  for (int i = 0, k = 0; i < 4; i++)
    for (int j = 0; j < 4; j++, k++) {
      left[i] += ct[k];
      right[j] += ct[k];
    }
  for (int i = 0; i < 4; i++) {
    left[i] /= sum;
    right[i] /= sum;
  }
  for (int i = 0, k = 0; i < 4; i++)
    for (int j = 0; j < 4; j++, k++) {
      double pr = double(ct[k]) / sum;
      if (pr != 0.0 && left[i] != 0.0 && right[j] != 0.0) mi += pr * log(pr / (left[i] * right[j]));
    }
  return mi;
}

static const float kChi2Val[7] = {2.37f, 4.11f, 6.25f, 7.81f, 9.35f, 11.3f, 12.8f};          // icm.hh:36-37
static const float kChi2Sig[7] = {0.50f, 0.75f, 0.90f, 0.95f, 0.975f, 0.99f, 0.995f};         // icm.hh:39-40

// position choice for one node; returns max_pos (no pruning applied) and best_info
static int choose_position(const int32_t* node_counts, int W, int sum, double* best_out, double* used_out) {
  int max_pos = 0;
  double best = mutual_info16(node_counts, sum), used = best;
  for (int i = 1; i < W - 1; i++) {
    double next = mutual_info16(node_counts + 16 * i, sum);
    if (next >= best) {
      used = best = next;
      max_pos = i;
    } else if (next >= best / (1.0 + 0.03)) {  // MUT_INFO_BIAS: prefer positions to the right
      max_pos = i;
      used = next;
    }
  }
  *best_out = best;
  *used_out = used;  // information of the position actually chosen (what the node stores, icm.cc:1156)
  return max_pos;
}

static void interpolate_probs(float* pr, const float* pp, const int ct[4]) {
  double total = 0.0;
  for (int i = 0; i < 4; i++) total += ct[i];
  for (int i = 0; i < 4; i++) pr[i] = (float)((ct[i] + 0.001 * pp[i]) / (total + 0.001));
  if (total >= 400) return;
  double chi2 = 0.0;
  for (int i = 0; i < 4; i++) {
    double expected = total * pp[i];
    if (expected > 0.0) chi2 += pow(ct[i] - expected, 2.0) / expected;
  }
  int i;
  for (i = 0; i < 7 && kChi2Val[i] < chi2; i++)
    ;
  double lambda;
  if (i == 0) lambda = 0.0;
  else if (i == 7) lambda = 1.0;
  else
    lambda = kChi2Sig[i - 1] +
             ((chi2 - kChi2Val[i - 1]) / (kChi2Val[i] - kChi2Val[i - 1])) * (kChi2Sig[i] - kChi2Sig[i - 1]);
  lambda *= total / 400;
  if (lambda > 1.0) lambda = 1.0;
  for (int k = 0; k < 4; k++) {
    pr[k] = (float)(pr[k] * lambda);                  // two float stores, like the reference (icm.cc:1324-1326)
    pr[k] = (float)(pr[k] + (1.0 - lambda) * pp[k]);
  }
}

// one node on the host, exactly as the reference computes it (glibc log): the fallback of k4_finish_level's flagged nodes
// and, with GMG_K4_MI=0, the path of every node
static void finish_node_host(gmg_trainer* t, int level, int f, int sub, const int32_t* nc) {
  const int W = t->W, N = t->N;
  int16_t* mp = &t->mip[(size_t)f * N + sub];
  float* pr = &t->prob[((size_t)f * N + sub) * 4];
  if (level > 0 && t->mip[(size_t)f * N + (sub - 1) / 4] < 0) {
    *mp = -2;  // stopped at the parent (icm.cc:1104-1109)
    return;
  }
  int final_ct[4] = {0, 0, 0, 0}, sum = 0;
  for (int i = 0, k = 0; i < 4; i++)
    for (int j = 0; j < 4; j++, k++) {
      sum += nc[k];
      final_ct[j] += nc[k];
    }
  double best, used;
  int max_pos = choose_position(nc, W, sum, &best, &used);
  t->mut_info[(size_t)f * N + sub] = (float)(level == 0 ? best : used);  // root keeps the maximum (icm.cc:1438)
  if (level == 0) {
    // float arithmetic (icm.cc:1411-1413)
    for (int j = 0; j < 4; j++) pr[j] = ((float)final_ct[j] + float(0.001 / 4)) / float(sum + 0.001);
    *mp = (int16_t)max_pos;
  } else {
    if (best <= 1e-4 && sum < 400) max_pos = -1;  // MUT_INFO_EPSILON, SAMPLE_SIZE_BOUND
    *mp = (int16_t)max_pos;
    interpolate_probs(pr, &t->prob[((size_t)f * N + (sub - 1) / 4) * 4], final_ct);
  }
}

int gmg_host_stage(gmg_ctx* ctx, size_t bytes, size_t want) {
  if (ctx->h_stage_bytes >= bytes) return 0;
  if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
  ctx->h_stage = NULL;
  ctx->h_stage_bytes = 0;
  const size_t cap = want > bytes ? want : bytes;
  GMG_CUDA(cudaMallocHost(&ctx->h_stage, cap));
  ctx->h_stage_bytes = cap;
  return 0;
}

extern "C" int gmg_trainer_finish_level(gmg_trainer* t, int level) {
  GMG_CHECK(t, "gmg_trainer_finish_level: NULL trainer");
  GMG_CHECK(level == t->next_level && level <= t->D, "gmg_trainer_finish_level: level %d out of order", level);
  gmg_ctx* ctx = t->ctx;
  const int W = t->W, N = t->N, rows = t->M * t->P;
  const int64_t nl = level_nodes(level), first = first_node_of(level);
  const int64_t slab = (int64_t)rows * nl * (W - 1) * 16;  // all models'
  const size_t slab_bytes = (size_t)slab * sizeof(int32_t);
  const int64_t n_items = (int64_t)rows * nl;
  const int per = (W - 1) * 16;  // counters of one node
  const char* mi_env = getenv("GMG_K4_MI");  // 0: every node on the host (round-1 path); 2: device + every node re-done on the host
  const int mi_mode = mi_env ? atoi(mi_env) : 1;
  if (mi_mode != 0) {
    // ---- device: position choice + interpolation for every node of every model; flagged nodes come back for the host ----
    int8_t* o_mip = (int8_t*)t->d_lvl;
    uint8_t* o_flag = (uint8_t*)(o_mip + n_items);
    float* o_mi = (float*)(t->d_lvl + ((2 * (size_t)n_items + 15) & ~(size_t)15));
    float* o_prob = o_mi + n_items;
    const size_t out_bytes = ((2 * (size_t)n_items + 15) & ~(size_t)15) + (size_t)n_items * 5 * sizeof(float);
    if (gmg_prof_begin(ctx, GMG_PROF_K4)) return 1;
    k4_finish_level<<<(unsigned)((n_items + 127) / 128), 128, 0, ctx->stream>>>(t->d_counts, W, rows, N, level, (int)first, (int)nl,
                                                                                t->d_mip, t->d_prob, o_mip, o_flag, o_mi, o_prob,
                                                                                mi_mode == 2 ? 1 : 0);
    gmg_prof_end(ctx, GMG_PROF_K4);
    ctx->launches++;
    GMG_CUDA(cudaGetLastError());
    if (gmg_host_stage(ctx, out_bytes, (size_t)rows * level_nodes(t->D) * 24 + 256)) return 1;
    GMG_CUDA(cudaMemcpyAsync(ctx->h_stage, t->d_lvl, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));
    const int8_t* h_mip = (const int8_t*)ctx->h_stage;
    const uint8_t* h_flag = (const uint8_t*)(h_mip + n_items);
    const float* h_mi = (const float*)((const char*)ctx->h_stage + ((2 * (size_t)n_items + 15) & ~(size_t)15));
    const float* h_prob = h_mi + n_items;
    std::vector<int64_t> flagged;
    for (int64_t it = 0; it < n_items; it++) {
      const int64_t row = it / nl;
      const size_t at = (size_t)row * N + (size_t)(first + it % nl);
      t->mip[at] = (int16_t)h_mip[it];
      t->mut_info[at] = h_mi[it];
      memcpy(&t->prob[at * 4], h_prob + 4 * it, 4 * sizeof(float));
      if (h_flag[it]) flagged.push_back(it);
    }
    const int64_t nf = (int64_t)flagged.size();
    if (nf > 0) {
      // a decision within the logarithm's error bound: these nodes again on the host with glibc, from their counts.
      // Their count tables come back gathered in one copy, their results go out in one copy.
      const size_t items_bytes = (size_t)nf * sizeof(int64_t);
      const size_t cnt_off = (items_bytes + 15) & ~(size_t)15;
      const size_t fix_off = cnt_off + (((size_t)nf * per * sizeof(int32_t) + 15) & ~(size_t)15);
      char* d_buf = NULL;
      GMG_CUDA(cudaMallocAsync((void**)&d_buf, fix_off + (size_t)nf * sizeof(K4Fix), ctx->stream));
      int64_t* d_items = (int64_t*)d_buf;
      int32_t* d_cnt = (int32_t*)(d_buf + cnt_off);
      K4Fix* d_fix = (K4Fix*)(d_buf + fix_off);
      const int64_t cells = nf * per;
      const int64_t cap = (int64_t)ctx->sm_count * 8;
      const int g_gather = (int)((cells + 255) / 256 < cap ? (cells + 255) / 256 : cap);
      const int g_apply = (int)((nf + 255) / 256 < cap ? (nf + 255) / 256 : cap);
      // the same layout in the page-locked staging buffer, whose level results have been read above; the next writer
      // of the buffer is the next level's D2H, ordered on the stream after the H2D of the fixes
      if (gmg_host_stage(ctx, fix_off + (size_t)nf * sizeof(K4Fix), 0)) {
        cudaFreeAsync(d_buf, ctx->stream);
        return 1;
      }
      memcpy(ctx->h_stage, flagged.data(), items_bytes);
      const int32_t* cnt = (const int32_t*)((const char*)ctx->h_stage + cnt_off);
      K4Fix* fix = (K4Fix*)((char*)ctx->h_stage + fix_off);
      GMG_CUDA(cudaMemcpyAsync(d_items, ctx->h_stage, items_bytes, cudaMemcpyHostToDevice, ctx->stream));
      k4_gather_flagged<<<g_gather, 256, 0, ctx->stream>>>(t->d_counts, d_items, nf, per, d_cnt);
      ctx->launches++;
      GMG_CUDA(cudaGetLastError());
      GMG_CUDA(cudaMemcpyAsync((char*)ctx->h_stage + cnt_off, d_cnt, (size_t)cells * sizeof(int32_t), cudaMemcpyDeviceToHost,
                               ctx->stream));
      GMG_CUDA(cudaStreamSynchronize(ctx->stream));
      host_parallel(nf, 256, [&](int64_t lo, int64_t hi) {
        for (int64_t k = lo; k < hi; k++) {
          const int64_t it = flagged[k];
          const int64_t row = it / nl;
          const int sub = (int)(first + it % nl);
          const size_t at = (size_t)row * N + sub;
          t->mut_info[at] = 0.0f;
          finish_node_host(t, level, (int)row, sub, &cnt[(size_t)k * per]);
          fix[k].mip = t->mip[at] < -2 ? -2 : t->mip[at];
          memcpy(fix[k].prob, &t->prob[at * 4], 4 * sizeof(float));
        }
      });
      GMG_CUDA(cudaMemcpyAsync(d_fix, fix, (size_t)nf * sizeof(K4Fix), cudaMemcpyHostToDevice, ctx->stream));
      k4_apply_flagged<<<g_apply, 256, 0, ctx->stream>>>(d_items, d_fix, nf, (int)nl, (int)first, N, t->d_mip, t->d_prob);
      ctx->launches++;
      GMG_CUDA(cudaGetLastError());
      GMG_CUDA(cudaFreeAsync(d_buf, ctx->stream));
      if (level == t->D) GMG_CUDA(cudaStreamSynchronize(ctx->stream));  // the staging buffer is free when the call returns
    }
    t->n_flagged += nf;
    t->next_level = level + 1;
    return 0;
  }
  // ---- host: the slab comes back through the context's page-locked staging buffer ----
  if (gmg_host_stage(ctx, slab_bytes, (size_t)rows * level_nodes(t->D) * per * sizeof(int32_t))) return 1;
  GMG_CUDA(cudaMemcpyAsync(ctx->h_stage, t->d_counts, slab_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  const int32_t* C = (const int32_t*)ctx->h_stage;
  host_parallel(n_items, 256, [&](int64_t lo, int64_t hi) {
    for (int64_t it = lo; it < hi; it++)
      finish_node_host(t, level, (int)(it / nl), (int)(first + it % nl), C + (size_t)it * per);
  });
  // publish this level's branch positions and probabilities to the device tree
  std::vector<int8_t> lvl((size_t)nl);
  for (int f = 0; f < rows; f++) {
    for (int64_t i = 0; i < nl; i++) {
      int v = t->mip[(size_t)f * N + first + i];
      lvl[(size_t)i] = (int8_t)(v < -2 ? -2 : v);
    }
    GMG_CUDA(cudaMemcpyAsync(t->d_mip + (size_t)f * N + first, lvl.data(), (size_t)nl, cudaMemcpyHostToDevice, ctx->stream));
    GMG_CUDA(cudaMemcpyAsync(t->d_prob + ((size_t)f * N + first) * 4, &t->prob[((size_t)f * N + first) * 4],
                             (size_t)nl * 4 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  t->next_level = level + 1;
  return 0;
}

// Take_Logs for every model of the trainer (host threads: each model's arithmetic is independent) and hand them over;
// on failure no out[k] is left allocated
static int trainer_finish_all(gmg_trainer* t, gmg_icm** out) {
  GMG_CHECK(t->next_level == t->D + 1, "gmg_trainer_finish: only %d of %d levels built", t->next_level, t->D + 1);
  const size_t per_model = (size_t)t->P * t->N;
  std::vector<float> logs(t->prob.size());
  host_parallel(t->M, 2, [&](int64_t lo, int64_t hi) {
    for (size_t i = (size_t)lo * per_model * 4; i < (size_t)hi * per_model * 4; i++)
      logs[i] = (t->prob[i] > 0.0f) ? logf(t->prob[i]) : -FLT_MAX;
  });
  for (int k = 0; k < t->M; k++) {
    out[k] = NULL;
    if (gmg_icm_from_tables(t->ctx, t->W, t->D, t->P, t->mip.data() + k * per_model, logs.data() + k * per_model * 4,
                            &out[k])) {
      for (int j = 0; j < k; j++) {
        gmg_icm_free(out[j]);
        out[j] = NULL;
      }
      return 1;
    }
    out[k]->mut_info.assign(t->mut_info.begin() + k * per_model, t->mut_info.begin() + (k + 1) * per_model);
  }
  return 0;
}

extern "C" int gmg_trainer_finish(gmg_trainer* t, gmg_icm** out) {
  GMG_CHECK(t && out, "gmg_trainer_finish: NULL argument");
  return trainer_finish_all(t, out);
}

extern "C" int gmg_icm_train_sharded(gmg_ctx* ctx, gmg_seqset* s, int w, int d, int p, int reverse, gmg_allreduce_fn ar,
                                     void* user, int rank, int world, int64_t global_bases, gmg_icm** out) {
  gmg_trainer* t = NULL;
  if (gmg_trainer_create(ctx, s, w, d, p, reverse, &t)) return 1;
  int rc = (world > 1) ? gmg_trainer_set_shard(t, rank, world, global_bases, ar, user) : 0;
  for (int level = 0; level <= d && rc == 0; level++) {
    void* dptr = NULL;
    int64_t n = 0;
    rc = gmg_trainer_count_level(t, level, &dptr, &n);
    if (rc == 0 && ar) {
      if (ar(user, dptr, n, (void*)ctx->stream)) {
        gmg_set_error("gmg_icm_train: all-reduce callback failed at level %d", level);
        rc = 1;
      }
    }
    if (rc == 0) rc = gmg_trainer_finish_level(t, level);
  }
  if (rc == 0) rc = gmg_trainer_finish(t, out);
  ctx->train_flagged = t->n_flagged;
  gmg_trainer_free(t);
  return rc;
}

// all strings of the model on every rank's callback path (each rank walks every histogram cell of its own strings)
extern "C" int gmg_icm_train(gmg_ctx* ctx, gmg_seqset* s, int w, int d, int p, int reverse, gmg_allreduce_fn ar,
                             void* user, gmg_icm** out) {
  return gmg_icm_train_sharded(ctx, s, w, d, p, reverse, ar, user, 0, 1, -1, out);
}

// Batched training: models large enough for the window histogram go through gmg_icm_train one by one (each needs its
// own 4^W-cell histogram); the others are trained in groups, every group through all levels together -- one k4_count
// and one k4_finish_level launch per level for the whole group, one level result copy, one flagged-node round trip.
// Groups are sized from the free device memory (GMG_K4_MANY_GROUP=k forces k models per group).
extern "C" int gmg_icm_train_many(gmg_ctx* ctx, gmg_seqset* const* sets, int n_models, int w, int d, int p, int reverse,
                                  gmg_icm** out) {
  GMG_CHECK(ctx && sets && out, "gmg_icm_train_many: NULL argument");
  GMG_CHECK(n_models >= 1, "gmg_icm_train_many: n_models %d < 1", n_models);
  for (int k = 0; k < n_models; k++) {
    out[k] = NULL;
    GMG_CHECK(sets[k], "gmg_icm_train_many: training set %d is NULL", k);
  }
  if (check_shape(w, d, p)) return 1;
  int64_t flagged = 0;
  int rc = 0;
  std::vector<gmg_seqset*> direct;
  std::vector<int> direct_at;
  for (int k = 0; k < n_models && rc == 0; k++) {
    if (k4_use_hist(w, p, sets[k]->total)) {
      rc = gmg_icm_train(ctx, sets[k], w, d, p, reverse, NULL, NULL, &out[k]);
      flagged += ctx->train_flagged;
    } else {
      direct.push_back(sets[k]);
      direct_at.push_back(k);
    }
  }
  int group = (int)direct.size();
  const char* g_env = getenv("GMG_K4_MANY_GROUP");
  if (g_env && atoi(g_env) >= 1) {
    if (atoi(g_env) < group) group = atoi(g_env);
  } else if (rc == 0 && group > 0) {
    size_t free_b = 0, total_b = 0;
    if (cudaSetDevice(ctx->device) != cudaSuccess || cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) {
      gmg_set_error("gmg_icm_train_many: cannot query the device memory");
      rc = 1;
    }
    // half the free memory; the count tables of flagged nodes may need up to one more slab per model
    const size_t fit = free_b / 2 / (trainer_model_bytes(w, d, p) + (size_t)p * level_nodes(d) * (w - 1) * 16 * sizeof(int32_t));
    if (fit < (size_t)group) group = fit > 1 ? (int)fit : 1;
  }
  std::vector<gmg_icm*> got;
  for (size_t g0 = 0; g0 < direct.size() && rc == 0; g0 += (size_t)group) {
    const int m = (int)(direct.size() - g0 < (size_t)group ? direct.size() - g0 : (size_t)group);
    gmg_trainer* t = NULL;
    if (trainer_create(ctx, direct.data() + g0, m, w, d, p, reverse, &t)) {
      rc = 1;
      break;
    }
    for (int level = 0; level <= d && rc == 0; level++) {
      rc = gmg_trainer_count_level(t, level, NULL, NULL);
      if (rc == 0) rc = gmg_trainer_finish_level(t, level);
    }
    got.assign((size_t)m, NULL);
    if (rc == 0) rc = trainer_finish_all(t, got.data());
    flagged += t->n_flagged;
    gmg_trainer_free(t);
    for (int k = 0; k < m && rc == 0; k++) out[direct_at[g0 + k]] = got[k];
  }
  ctx->train_flagged = flagged;
  if (rc) {
    for (int k = 0; k < n_models; k++) {
      gmg_icm_free(out[k]);
      out[k] = NULL;
    }
  }
  return rc;
}

extern "C" int64_t gmg_ctx_train_flagged(const gmg_ctx* ctx) { return ctx ? ctx->train_flagged : 0; }
