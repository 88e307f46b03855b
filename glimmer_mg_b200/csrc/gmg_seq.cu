// glimmer_mg_b200/csrc/gmg_seq.cu -- sequence batches: ASCII -> Filter -> 2-bit pack in HBM.
//
// Reference behaviour mirrored (paths relative to /root/reference/src/):
//   Filter                 Common/gene.cc:1139-1175   (every non-acgt IUPAC code -> one fixed base,
//                                                      anything else incl. 'n' -> 'c')
//   tolower(Filter(c))     Glimmer/glimmer-mg.cc:381-382, glimmer3.cc:270-271
//   Set_GC_Fraction        Glimmer/glimmer_base.cc:2564-2595
#include <limits.h>
#include <string.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <thrust/iterator/transform_iterator.h>

#include "gmg_internal.cuh"

// 2-bit code of tolower(Filter(ch)): a=0 c=1 g=2 t=3 (ALPHA_STRING "acgt", icm.hh:30)
__device__ __forceinline__ unsigned filter_code(unsigned ch) {
  switch (ch | 0x20u) {
    case 'a': return 0;
    case 'g': case 'r': case 'd': return 2;
    case 't': case 'w': case 'k': return 3;
    default: return 1;  // c, y, s, m, b, h, v and everything else
  }
}

__device__ __forceinline__ bool is_acgt(unsigned ch) {
  const unsigned c = ch | 0x20u;
  return c == 'a' || c == 'c' || c == 'g' || c == 't';
}

// g + c among the 32 bases of a packed word (codes 1 and 2: exactly one of the two bits set; zero padding is 'a')
__device__ __forceinline__ unsigned word_gc(uint64_t v) {
  return (unsigned)__popcll((v ^ (v >> 1)) & 0x5555555555555555ull);
}

// sum of every thread's count into *gc: one atomic per warp; every thread of the warp must call it
__device__ __forceinline__ void warp_add_gc(unsigned my_gc, unsigned long long* gc) {
  for (int o = 16; o > 0; o >>= 1) my_gc += __shfl_down_sync(0xffffffffu, my_gc, o);
  if ((threadIdx.x & 31) == 0 && my_gc) atomicAdd(gc, (unsigned long long)my_gc);
}

// one thread packs 32 bases (32 ASCII bytes = two 16-byte loads) into one 64-bit word and
// counts its g/c; a warp therefore reads 1 KB contiguous and writes 256 B contiguous.
// Bytes other than a / c / g / t (bit b of `odd`) go to the non-acgt list: one ballot per warp finds out whether any
// lane has one, so acgt-only input never reaches the atomic.  *n_nacgt counts every such byte, also those past `cap`
// (the caller sees the overflow and packs again with room for all of them).  The list comes out unordered.
__global__ void __launch_bounds__(256) k_pack(const uint8_t* __restrict__ ascii, int64_t total,
                                              uint64_t* __restrict__ words, unsigned long long* __restrict__ gc,
                                              uint64_t* __restrict__ nacgt, int64_t cap,
                                              unsigned long long* __restrict__ n_nacgt) {
  int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t nwords = (total + 31) >> 5;
  unsigned my_gc = 0, odd = 0;
  const int64_t base = w << 5;
  if (w < nwords) {
    uint64_t v = 0;
    if (base + 32 <= total && ((reinterpret_cast<uintptr_t>(ascii + base) & 15) == 0)) {
      const uint4* src = reinterpret_cast<const uint4*>(ascii + base);
#pragma unroll
      for (int h = 0; h < 2; h++) {
        uint4 q = __ldg(src + h);
        unsigned r[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int k = 0; k < 4; k++)
#pragma unroll
          for (int b = 0; b < 4; b++) {
            const unsigned ch = (r[k] >> (8 * b)) & 0xFF;
            v |= (uint64_t)filter_code(ch) << (2 * (h * 16 + k * 4 + b));
            odd |= (is_acgt(ch) ? 0u : 1u) << (h * 16 + k * 4 + b);
          }
      }
    } else {
      for (int b = 0; b < 32 && base + b < total; b++) {
        const unsigned ch = ascii[base + b];
        v |= (uint64_t)filter_code(ch) << (2 * b);
        odd |= (is_acgt(ch) ? 0u : 1u) << b;
      }
    }
    words[w] = v;
    my_gc = word_gc(v);
  }
  if (__ballot_sync(0xffffffffu, odd != 0)) {
    const int lane = threadIdx.x & 31;
    const unsigned cnt = (unsigned)__popc(odd);
    unsigned incl = cnt;  // inclusive warp prefix of the counts
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    unsigned long long first = 0;
    if (lane == 31) first = atomicAdd(n_nacgt, (unsigned long long)incl);
    unsigned long long e = __shfl_sync(0xffffffffu, first, 31) + (incl - cnt);
    for (; odd; odd &= odd - 1, e++) {
      const int b = __ffs(odd) - 1;
      unsigned ch = ascii[base + b];
      if (ch >= 'A' && ch <= 'Z') ch += 32;
      if (e < (unsigned long long)cap) nacgt[e] = ((uint64_t)(base + b) << 8) | ch;
    }
  }
  warp_add_gc(my_gc, gc);
}

__global__ void k_unpack(const uint64_t* __restrict__ words, int64_t total, char* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) out[i] = "acgt"[gmg_base_at(words, i)];
}

// sequence that holds base 32*b (binary search over the offsets; run once per batch), plus the interior flag
__global__ void k_blk2seq(const int64_t* __restrict__ off, int64_t n, int64_t nblk, int32_t* __restrict__ blk2seq) {
  int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nblk) return;
  int64_t p = b << 5;
  int64_t lo = 0, hi = n;  // largest s with off[s] <= p
  while (hi - lo > 1) {
    int64_t mid = (lo + hi) >> 1;
    if (off[mid] <= p) lo = mid;
    else hi = mid;
  }
  // bit 31: "interior" block -- all 32 bases lie in one sequence, at least 32 bases from either end, so no
  // window of up to GMG_MAX_W bases around them is partial (K1's fast path needs no sequence lookup at all)
  const bool interior = (p - off[lo] >= 32) && (p + 64 <= off[lo + 1]);
  blk2seq[b] = (int32_t)lo | (interior ? (int32_t)0x80000000 : 0);
}

// ---- base buckets (see gmg_plane_index) ---------------------------------------------------------------
// per 32-base block: how many a / c / g / t (positions at or past `total` are not counted)
__global__ void __launch_bounds__(256) k_bucket_count(const uint64_t* __restrict__ words, int64_t total, int64_t nblk,
                                                      uint4* __restrict__ cnt) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nblk) return;
  const uint64_t w = __ldg(words + b);
  const int n = (int)(total - (b << 5) < 32 ? total - (b << 5) : 32);
  const uint64_t valid = n >= 32 ? 0x5555555555555555ull : (0x5555555555555555ull & ((1ull << (2 * n)) - 1ull));
  const uint64_t lo = w & 0x5555555555555555ull, hi = (w >> 1) & 0x5555555555555555ull;
  uint4 c;
  c.x = (unsigned)__popcll(~lo & ~hi & valid);
  c.y = (unsigned)__popcll(lo & ~hi & valid);
  c.z = (unsigned)__popcll(~lo & hi & valid);
  c.w = (unsigned)__popcll(lo & hi & valid);
  cnt[b] = c;
}

struct Uint4Add {
  __device__ __forceinline__ uint4 operator()(const uint4& a, const uint4& b) const {
    return make_uint4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
  }
};

// exclusive per-base prefix -> absolute plane index of each block's first a / c / g / t, and the walk-ready
// contexts of every position stored at its plane index.  One CTA per tile of BKT_TILE bases (a warp takes four 32-base
// blocks); staged once per CTA: the per-base totals and the sequence bounds that fall into the tile, so that a position
// finds its distance to the ends of its sequence without dependent global loads (they were 40 % of the kernel's stalls).
#define BKT_TILE 1024
#define BKT_NB 129
__global__ void __launch_bounds__(256) k_bucket_finish(const uint64_t* __restrict__ words, int64_t total, int64_t nblk,
                                                       const int64_t* __restrict__ off, int64_t n_seq,
                                                       const int32_t* __restrict__ blk2seq,
                                                       const uint4* __restrict__ prefix, const uint4* __restrict__ cnt,
                                                       uint4* __restrict__ bktidx, uint32_t* __restrict__ ctxf,
                                                       uint32_t* __restrict__ ctxr,
                                                       unsigned long long* __restrict__ n_base) {
  __shared__ unsigned s_tot[4];
  __shared__ long long s_bound[BKT_NB];
  __shared__ unsigned char s_blk[BKT_TILE / 32];
  const int64_t p0 = (int64_t)blockIdx.x * BKT_TILE;
  const int t = threadIdx.x;
  if (t == 0) {
    const uint4 lp = prefix[nblk - 1], lc = cnt[nblk - 1];
    s_tot[0] = lp.x + lc.x;
    s_tot[1] = lp.y + lc.y;
    s_tot[2] = lp.z + lc.z;
    s_tot[3] = lp.w + lc.w;
  } else if (t >= 32 && t < 32 + BKT_NB) {
    const int k = t - 32;
    const int32_t s0 = __ldg(blk2seq + (p0 >> 5)) & 0x7FFFFFFF;  // the sequence that holds the tile's first base
    const int64_t idx = (int64_t)s0 + k;
    s_bound[k] = idx <= n_seq ? (long long)__ldg(off + idx) : LLONG_MAX;
  }
  __syncthreads();
  const bool staged = s_bound[BKT_NB - 1] > p0 + BKT_TILE - 1;  // all of the tile's sequences are in the staged list
  if (staged && t < BKT_TILE / 32) {  // staged bound index of the sequence holding the first base of each block
    const int64_t p = p0 + 32 * t;
    int lo = 0, hi = BKT_NB - 1;  // s_bound[lo] <= p < s_bound[hi]
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (s_bound[mid] <= p) lo = mid;
      else hi = mid;
    }
    s_blk[t] = (unsigned char)lo;
  }
  __syncthreads();
  const unsigned na = s_tot[0], nc = s_tot[1], ng = s_tot[2], nt = s_tot[3];
  if (blockIdx.x == 0 && t == 0) {
    n_base[0] = na; n_base[1] = nc; n_base[2] = ng; n_base[3] = nt;
  }
  const int warp = t >> 5, i = t & 31;
#pragma unroll 1
  for (int k = 0; k < BKT_TILE / 256; k++) {
    const int bt = warp + 8 * k;  // block of the tile
    const int64_t blk = (p0 >> 5) + bt, p = (blk << 5) + i;
    if (p >= total) continue;
    uint4 pre = prefix[blk];
    pre.y += na;
    pre.z += na + nc;
    pre.w += na + nc + ng;
    if (i == 0) bktidx[blk] = pre;
    // the block's word and its neighbours (warp-uniform loads; zero padding either side of the batch): every window
    // below is cut from these three
    const uint64_t wm = __ldg(words + blk - 1), w = __ldg(words + blk), wp = __ldg(words + blk + 1);
    const unsigned b = (unsigned)(w >> (2 * i)) & 3u;
    const uint64_t x = w ^ (0x5555555555555555ull * b);
    const uint64_t eq = ~(x | (x >> 1)) & 0x5555555555555555ull & ((1ull << (2 * i)) - 1ull);
    const unsigned first = b == 0 ? pre.x : (b == 1 ? pre.y : (b == 2 ? pre.z : pre.w));
    const unsigned idx = first + (unsigned)__popcll(eq);
    int64_t a, nx;
    if (staged) {
      int kb = s_blk[bt];
      while (s_bound[kb + 1] <= p) kb++;
      a = s_bound[kb];
      nx = s_bound[kb + 1];
    } else {
      int32_t sq = __ldg(blk2seq + blk) & 0x7FFFFFFF;
      nx = __ldg(off + sq + 1);
      while (p >= nx) nx = __ldg(off + (++sq) + 1);
      a = __ldg(off + sq);
    }
    uint32_t cf, cr;
    gmg_window_ctx(wm, w, wp, i, p - a, nx - 1 - p, &cf, &cr);
    ctxf[idx] = cf;
    ctxr[idx] = cr;
  }
}

// Base buckets and walk-ready contexts exist for K1 only: built on its first launch on a set (training and the
// string-scoring calls never pay for them).
int gmg_seqset_ensure_buckets(gmg_ctx* ctx, gmg_seqset* s) {
  if (s->d_bktidx || s->total == 0) return 0;
  const int64_t nblk = (s->total + 31) >> 5;
  GMG_CHECK(s->total < (1ll << 32), "batches of 2^32 bases or more are not supported (got %lld)", (long long)s->total);
  GMG_CUDA(cudaMallocAsync(&s->d_bktidx, (size_t)(nblk + 1) * sizeof(uint4), ctx->stream));
  GMG_CUDA(cudaMallocAsync(&s->d_ctxf, (size_t)(s->total + GMG_CTX_PAD) * sizeof(uint32_t), ctx->stream));
  GMG_CUDA(cudaMallocAsync(&s->d_ctxr, (size_t)(s->total + GMG_CTX_PAD) * sizeof(uint32_t), ctx->stream));
  GMG_CUDA(cudaMemsetAsync(s->d_ctxf + s->total, 0, GMG_CTX_PAD * sizeof(uint32_t), ctx->stream));
  GMG_CUDA(cudaMemsetAsync(s->d_ctxr + s->total, 0, GMG_CTX_PAD * sizeof(uint32_t), ctx->stream));
  void *d_cnt, *d_tmp;
  if (gmg_scratch(ctx, SCR_TMP3, (size_t)2 * nblk * sizeof(uint4), &d_cnt)) return 1;
  uint4* cnt = (uint4*)d_cnt;
  uint4* prefix = cnt + nblk;
  k_bucket_count<<<(unsigned)((nblk + 255) / 256), 256, 0, ctx->stream>>>(s->d_words, s->total, nblk, cnt);
  size_t tmp_bytes = 0;
  GMG_CUDA(cub::DeviceScan::ExclusiveScan(NULL, tmp_bytes, cnt, prefix, Uint4Add(), make_uint4(0, 0, 0, 0), nblk, ctx->stream));
  if (gmg_scratch(ctx, SCR_TMP4, tmp_bytes, &d_tmp)) return 1;
  GMG_CUDA(cub::DeviceScan::ExclusiveScan(d_tmp, tmp_bytes, cnt, prefix, Uint4Add(), make_uint4(0, 0, 0, 0), nblk, ctx->stream));
  k_bucket_finish<<<(unsigned)((s->total + BKT_TILE - 1) / BKT_TILE), 256, 0, ctx->stream>>>(
      s->d_words, s->total, nblk, s->d_off, s->n, s->d_blk2seq, prefix, cnt, (uint4*)s->d_bktidx, s->d_ctxf, s->d_ctxr,
      s->d_gc + 2);
  ctx->launches += 4;
  GMG_CUDA(cudaGetLastError());
  return 0;
}

// d_gc[6] counts the non-acgt bytes (d_nacgt holds the first cap_nacgt of them)
int gmg_launch_pack(gmg_ctx* ctx, const uint8_t* d_ascii, int64_t total, uint64_t* d_words, unsigned long long* d_gc,
                    uint64_t* d_nacgt, int64_t cap_nacgt) {
  int64_t nwords = (total + 31) >> 5;
  if (nwords == 0) return 0;
  if (gmg_prof_begin(ctx, GMG_PROF_PACK)) return 1;
  k_pack<<<(unsigned)((nwords + 255) / 256), 256, 0, ctx->stream>>>(d_ascii, total, d_words, d_gc, d_nacgt, cap_nacgt,
                                                                    d_gc + 6);
  gmg_prof_end(ctx, GMG_PROF_PACK);
  ctx->launches++;
  GMG_CUDA(cudaGetLastError());
  return 0;
}

// An empty set of n sequences with offsets h_off: device offsets, zeroed words and counters, blk2seq.  The creation routes
// pack bases into it, gmg_seqset_extract copies them from another set.
// copy_off_from_caller: the device copy of the offsets is made straight from h_off (gmg_seqset_create synchronises before
// it returns, so a page-locked caller buffer travels at PCIe rate and without the driver's staging copy); otherwise from
// the set's own host copy.
static int seqset_alloc(gmg_ctx* ctx, const int64_t* h_off, int64_t n, gmg_seqset** out, bool copy_off_from_caller) {
  GMG_CHECK(n >= 0 && n < (1ll << 31), "gmg_seqset_create: %lld sequences unsupported", (long long)n);
  int64_t max_len = 0;
  for (int64_t i = 0; i < n; i++) {
    GMG_CHECK(h_off[i + 1] >= h_off[i], "gmg_seqset_create: offsets not monotone at %lld", (long long)i);
    if (h_off[i + 1] - h_off[i] > max_len) max_len = h_off[i + 1] - h_off[i];
  }
  GMG_CHECK(n == 0 || h_off[0] == 0, "gmg_seqset_create: offsets must start at 0");
  gmg_seqset* s = new gmg_seqset();
  s->ctx = ctx;
  s->n = n;
  s->total = n ? h_off[n] : 0;
  s->max_len = max_len;
  s->off.assign(h_off, h_off + n + 1);
  if (n == 0) s->off.assign(1, 0);
  s->d_off = NULL; s->d_words_base = NULL; s->d_words = NULL; s->d_blk2seq = NULL; s->d_qual = NULL; s->d_gc = NULL;
  s->d_cbits = NULL; s->nwc = 0; s->d_bktidx = NULL; s->d_ctxf = NULL; s->d_ctxr = NULL; memset(s->n_base, 0, sizeof s->n_base); s->n_base_valid = 0; memset(s->cbits_key, 0, sizeof s->cbits_key);
  s->n_orfs = 0; s->d_orfs = NULL; s->d_orf_off = NULL; s->d_orf_seq = NULL;
  s->n_starts = 0; s->d_starts = NULL; s->d_start_off = NULL; s->uncertified = 0;
  s->cap_orfs = s->cap_starts = 0;
  s->d_nacgt = NULL; s->n_nacgt = 0;
  GMG_CUDA(cudaSetDevice(ctx->device));
  int64_t nwords = (s->total + 31) >> 5;
  int64_t nblk = nwords > 0 ? nwords : 1;
  size_t wbytes = (size_t)(nwords + 2 * GMG_PAD_WORDS) * sizeof(uint64_t);
  GMG_CUDA(cudaMallocAsync(&s->d_words_base, wbytes, s->ctx->stream));
  GMG_CUDA(cudaMemsetAsync(s->d_words_base, 0, wbytes, ctx->stream));
  s->d_words = s->d_words_base + GMG_PAD_WORDS;
  GMG_CUDA(cudaMallocAsync(&s->d_off, (size_t)(s->n + 1) * sizeof(int64_t), s->ctx->stream));
  GMG_CUDA(cudaMemcpyAsync(s->d_off, copy_off_from_caller && n > 0 ? h_off : s->off.data(), (size_t)(s->n + 1) * sizeof(int64_t),
                           cudaMemcpyHostToDevice, ctx->stream));
  GMG_CUDA(cudaMallocAsync(&s->d_blk2seq, (size_t)nblk * sizeof(int32_t), s->ctx->stream));
  GMG_CUDA(cudaMallocAsync(&s->d_gc, 7 * sizeof(unsigned long long), s->ctx->stream));
  GMG_CUDA(cudaMemsetAsync(s->d_gc, 0, 7 * sizeof(unsigned long long), ctx->stream));
  if (s->total > 0) {
    k_blk2seq<<<(unsigned)((nblk + 255) / 256), 256, 0, ctx->stream>>>(s->d_off, s->n, nblk, s->d_blk2seq);
    ctx->launches++;
    GMG_CUDA(cudaGetLastError());
  }
  *out = s;
  return 0;
}

// room for the pack's first pass at the non-acgt list (context scratch SCR_MISC): assembled genomes hold a few such bytes
// per Mbp; input with more packs a second time at the exact size (seqset_finish_nacgt)
static int64_t nacgt_cap(int64_t total) { return 4096 + total / 1024; }

// Pack the ASCII at d_ascii into a new set.  The count of non-acgt bytes is on its way to ctx->h_scalars[15]: synchronise
// the stream, then call seqset_finish_nacgt while d_ascii is still intact.
static int seqset_build(gmg_ctx* ctx, const void* d_ascii, const int64_t* h_off, int64_t n, const void* d_qual,
                        gmg_seqset** out, bool copy_off_from_caller = false) {
  gmg_seqset* s;
  if (seqset_alloc(ctx, h_off, n, &s, copy_off_from_caller)) return 1;
  ctx->h_scalars[15] = 0;
  if (s->total > 0) {
    void* d_list;
    if (gmg_scratch(ctx, SCR_MISC, (size_t)nacgt_cap(s->total) * sizeof(uint64_t), &d_list)) return 1;
    if (gmg_launch_pack(ctx, (const uint8_t*)d_ascii, s->total, s->d_words, s->d_gc, (uint64_t*)d_list,
                        nacgt_cap(s->total)))
      return 1;
    GMG_CUDA(cudaMemcpyAsync(ctx->h_scalars + 15, s->d_gc + 6, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (d_qual) {
      GMG_CUDA(cudaMallocAsync(&s->d_qual, (size_t)s->total, s->ctx->stream));
      GMG_CUDA(cudaMemcpyAsync(s->d_qual, d_qual, (size_t)s->total, cudaMemcpyDeviceToDevice, ctx->stream));
    }
  }
  *out = s;
  return 0;
}

// Sorts the pack's non-acgt list into the set (after the stream synchronisation that brought its count to the host).
// A list that overflowed the first pass is recorded again, at its exact size, from the same ASCII.
static int seqset_finish_nacgt(gmg_ctx* ctx, gmg_seqset* s, const void* d_ascii) {
  const int64_t cnt = ctx->h_scalars[15];
  if (cnt == 0) return 0;
  GMG_CHECK(cnt < (1ll << 31), "gmg_seqset_create: %lld bytes other than a, c, g, t -- split the batch", (long long)cnt);
  void *d_list, *d_tmp;
  if (gmg_scratch(ctx, SCR_MISC, (size_t)(cnt > nacgt_cap(s->total) ? cnt : nacgt_cap(s->total)) * sizeof(uint64_t), &d_list))
    return 1;
  if (cnt > nacgt_cap(s->total)) {
    GMG_CUDA(cudaMemsetAsync(s->d_gc, 0, 7 * sizeof(unsigned long long), ctx->stream));
    if (gmg_launch_pack(ctx, (const uint8_t*)d_ascii, s->total, s->d_words, s->d_gc, (uint64_t*)d_list, cnt)) return 1;
  }
  GMG_CUDA(cudaMallocAsync(&s->d_nacgt, (size_t)cnt * sizeof(uint64_t), ctx->stream));
  int end_bit = 8;
  while (end_bit < 64 && (s->total >> (end_bit - 8)) != 0) end_bit++;
  size_t tmp_bytes = 0;
  GMG_CUDA(cub::DeviceRadixSort::SortKeys(NULL, tmp_bytes, (const uint64_t*)d_list, s->d_nacgt, (int)cnt, 8, end_bit,
                                          ctx->stream));
  if (gmg_scratch(ctx, SCR_TMP4, tmp_bytes, &d_tmp)) return 1;
  GMG_CUDA(cub::DeviceRadixSort::SortKeys(d_tmp, tmp_bytes, (const uint64_t*)d_list, s->d_nacgt, (int)cnt, 8, end_bit,
                                          ctx->stream));
  ctx->launches++;
  s->n_nacgt = cnt;
  return 0;
}

extern "C" int gmg_seqset_create_device(gmg_ctx* ctx, const void* d_ascii, const int64_t* h_off, int64_t n,
                                        const void* d_qual, gmg_seqset** out) {
  GMG_CHECK(ctx && h_off && out, "gmg_seqset_create_device: NULL argument");
  if (seqset_build(ctx, d_ascii, h_off, n, d_qual, out)) return 1;
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  return seqset_finish_nacgt(ctx, *out, d_ascii);
}

extern "C" int gmg_seqset_create(gmg_ctx* ctx, const char* h_ascii, const int64_t* h_off, int64_t n,
                                 const uint8_t* h_qual, gmg_seqset** out) {
  GMG_CHECK(ctx && h_off && out, "gmg_seqset_create: NULL argument");
  GMG_CUDA(cudaSetDevice(ctx->device));
  int64_t total = n ? h_off[n] : 0;
  void* d_ascii = NULL;
  void* d_q = NULL;
  if (total > 0) {
    GMG_CHECK(h_ascii != NULL, "gmg_seqset_create: NULL sequence data");
    if (gmg_scratch(ctx, SCR_TMP, (size_t)total + 64, &d_ascii)) return 1;
    GMG_CUDA(cudaMemcpyAsync(d_ascii, h_ascii, (size_t)total, cudaMemcpyHostToDevice, ctx->stream));
    if (h_qual) {
      if (gmg_scratch(ctx, SCR_TMP2, (size_t)total + 64, &d_q)) return 1;
      GMG_CUDA(cudaMemcpyAsync(d_q, h_qual, (size_t)total, cudaMemcpyHostToDevice, ctx->stream));
    }
  }
  if (seqset_build(ctx, d_ascii, h_off, n, d_q, out, true)) return 1;
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));  // host buffers may be reused by the caller
  return seqset_finish_nacgt(ctx, *out, d_ascii);
}

// ------------------------------------------------------------------------------------------------
// FASTA ingest on the device (SURVEY.md section 8(f) row 1; Fasta_Read, Common/fasta.cc:236-283, and build-icm's
// Read_String, ICM/build-icm.cc:262-315): everything before the first '>' is skipped; a '>' anywhere outside a
// header line starts a record whose header runs to the end of that line; every other non-white-space byte up to
// the next '>' is a sequence character.  "Inside a header line" is a property of the LAST '>' or '\n' at or before
// a byte, i.e. an inclusive max-scan over (position, kind) keys; record numbers and compacted sequence indices are
// a second (sum) scan.  Two cub scans and two elementwise kernels replace the reference's fgetc loop.

struct FastaMaxOp {
  __device__ __forceinline__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; }
};
struct FastaSumOp {
  __device__ __forceinline__ uint2 operator()(uint2 a, uint2 b) const { return make_uint2(a.x + b.x, a.y + b.y); }
};
__device__ __forceinline__ bool fasta_is_space(unsigned ch) { return ch == ' ' || (ch >= 9 && ch <= 13); }

// key = (position + 1) * 2 + kind for '>' (kind 1) and '\n' (kind 0), 0 for every other byte
__global__ void __launch_bounds__(256) k_fasta_keys(const uint8_t* __restrict__ in, int64_t n, uint32_t* __restrict__ key) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned ch = in[i];
  key[i] = ch == '>' ? (uint32_t)((i + 1) * 2 + 1) : (ch == '\n' ? (uint32_t)((i + 1) * 2) : 0u);
}

// last[i] = inclusive max-scan of key.  flags.x = 1 for a kept sequence character, flags.y = 1 for a record start
__global__ void __launch_bounds__(256) k_fasta_flags(const uint8_t* __restrict__ in, int64_t n,
                                                     const uint32_t* __restrict__ last, uint2* __restrict__ flags) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned ch = in[i];
  const bool in_hdr = (last[i] & 1u) != 0;                 // the last '>' / '\n' at or before i is a '>'
  const bool prev_hdr = i > 0 && (last[i - 1] & 1u) != 0;  // ... before i
  const bool start = ch == '>' && !prev_hdr;
  flags[i] = make_uint2((!in_hdr && !fasta_is_space(ch)) ? 1u : 0u, start ? 1u : 0u);
}

// incl[i] = inclusive sums of flags (.x characters outside header lines, .y records started).
// Pass 1: per-record tables.  rec_chars[r] = characters counted before record r starts, hdr_off[r] = first byte of
// its header text, hdr_end[r] = the '\n' ending the header line (pre-filled with n for a header cut off by the end).
__global__ void __launch_bounds__(256) k_fasta_records(const uint8_t* __restrict__ in, int64_t n,
                                                       const uint32_t* __restrict__ last, const uint2* __restrict__ incl,
                                                       int64_t* __restrict__ rec_chars, int64_t* __restrict__ hdr_off,
                                                       int64_t* __restrict__ hdr_end) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint2 me = incl[i];
  const uint2 before = i > 0 ? incl[i - 1] : make_uint2(0u, 0u);
  if (me.y != before.y) {  // record me.y - 1 starts at this '>'
    rec_chars[me.y - 1] = before.x;
    hdr_off[me.y - 1] = i + 1;
  }
  if (in[i] == '\n' && i > 0 && (last[i - 1] & 1u) != 0 && me.y > 0) hdr_end[me.y - 1] = i;
}

// Pass 2: the sequence characters of all records, compacted (characters before the first record are dropped)
__global__ void __launch_bounds__(256) k_fasta_scatter(const uint8_t* __restrict__ in, int64_t n,
                                                       const uint2* __restrict__ incl, const int64_t* __restrict__ rec_chars,
                                                       uint8_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint2 me = incl[i];
  const uint32_t before = i > 0 ? incl[i - 1].x : 0u;
  if (me.x != before && me.y > 0) out[(int64_t)before - rec_chars[0]] = in[i];
}

__global__ void k_fill_i64(int64_t* __restrict__ p, int64_t n, int64_t v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

extern "C" int gmg_seqset_from_fasta(gmg_ctx* ctx, const char* h_bytes, int64_t n_bytes, gmg_seqset** out,
                                     int64_t* n_records) {
  GMG_CHECK(ctx && out && n_bytes >= 0 && (h_bytes || n_bytes == 0), "gmg_seqset_from_fasta: bad argument");
  GMG_CHECK(n_bytes < (1ll << 30), "gmg_seqset_from_fasta: images of 1 GiB or more must be split at record boundaries "
            "(got %lld bytes)", (long long)n_bytes);
  GMG_CUDA(cudaSetDevice(ctx->device));
  if (n_records) *n_records = 0;
  const int64_t n = n_bytes;
  int64_t n_rec = 0, n_chars = 0;
  std::vector<int64_t> h_tab;  // rec_chars | hdr_off | hdr_end
  void* d_out = NULL;
  if (n > 0) {
    void *d_in, *d_work;
    if (gmg_scratch(ctx, SCR_TMP, (size_t)n + 64, &d_in)) return 1;
    GMG_CUDA(cudaMemcpyAsync(d_in, h_bytes, (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    // keys / last (4 B per byte) and flags / sums (8 B per byte)
    if (gmg_scratch(ctx, SCR_CUM, (size_t)n * 12 + 256, &d_work)) return 1;
    uint2* d_flags = (uint2*)d_work;
    uint32_t* d_key = (uint32_t*)(d_flags + n);
    const unsigned grid = (unsigned)((n + 255) / 256);
    k_fasta_keys<<<grid, 256, 0, ctx->stream>>>((const uint8_t*)d_in, n, d_key);
    size_t tb1 = 0, tb2 = 0;
    GMG_CUDA(cub::DeviceScan::InclusiveScan(NULL, tb1, d_key, d_key, FastaMaxOp(), n, ctx->stream));
    GMG_CUDA(cub::DeviceScan::InclusiveScan(NULL, tb2, d_flags, d_flags, FastaSumOp(), n, ctx->stream));
    void* d_tmp;
    if (gmg_scratch(ctx, SCR_TMP4, tb1 > tb2 ? tb1 : tb2, &d_tmp)) return 1;
    GMG_CUDA(cub::DeviceScan::InclusiveScan(d_tmp, tb1, d_key, d_key, FastaMaxOp(), n, ctx->stream));
    k_fasta_flags<<<grid, 256, 0, ctx->stream>>>((const uint8_t*)d_in, n, d_key, d_flags);
    GMG_CUDA(cub::DeviceScan::InclusiveScan(d_tmp, tb2, d_flags, d_flags, FastaSumOp(), n, ctx->stream));
    ctx->launches += 4;
    GMG_CUDA(cudaMemcpyAsync(ctx->h_scalars + 4, d_flags + (n - 1), sizeof(uint2), cudaMemcpyDeviceToHost, ctx->stream));
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));
    uint2 tot;
    memcpy(&tot, ctx->h_scalars + 4, sizeof tot);
    n_rec = tot.y;
    if (n_rec > 0) {
      void* d_tab;
      if (gmg_scratch(ctx, SCR_TMP3, (size_t)3 * n_rec * sizeof(int64_t), &d_tab)) return 1;
      int64_t* rec_chars = (int64_t*)d_tab;
      int64_t* hdr_off = rec_chars + n_rec;
      int64_t* hdr_end = hdr_off + n_rec;
      k_fill_i64<<<(unsigned)((n_rec + 255) / 256), 256, 0, ctx->stream>>>(hdr_end, n_rec, n);
      k_fasta_records<<<grid, 256, 0, ctx->stream>>>((const uint8_t*)d_in, n, d_key, d_flags, rec_chars, hdr_off, hdr_end);
      if (gmg_scratch(ctx, SCR_TMP2, (size_t)tot.x + 64, &d_out)) return 1;
      k_fasta_scatter<<<grid, 256, 0, ctx->stream>>>((const uint8_t*)d_in, n, d_flags, rec_chars, (uint8_t*)d_out);
      ctx->launches += 3;
      GMG_CUDA(cudaGetLastError());
      h_tab.resize((size_t)3 * n_rec);
      GMG_CUDA(cudaMemcpyAsync(h_tab.data(), d_tab, h_tab.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
      GMG_CUDA(cudaStreamSynchronize(ctx->stream));
      n_chars = (int64_t)tot.x - h_tab[0];
      // Fasta_Read skips the blanks after '>' and gives up if the file ends there (Common/fasta.cc:251-255): a last
      // record whose '>' is followed by nothing but blanks does not exist; and the header text starts after the blanks
      for (int64_t r = 0; r < n_rec; r++) {
        int64_t& ho = h_tab[(size_t)(n_rec + r)];
        const int64_t he = h_tab[(size_t)(2 * n_rec + r)];
        while (ho < he && h_bytes[ho] == ' ') ho++;
      }
      {
        int64_t q = h_tab[(size_t)(2 * n_rec - 1)];  // header text of the last record
        while (q < n && h_bytes[q] == ' ') q++;
        if (q == n) {  // it has no characters either: drop it
          std::vector<int64_t> t2;
          for (int part = 0; part < 3; part++) t2.insert(t2.end(), h_tab.begin() + part * n_rec, h_tab.begin() + part * n_rec + (n_rec - 1));
          h_tab.swap(t2);
          n_rec--;
        }
      }
    }
  }
  // sequence offsets: characters counted before each record, relative to the first record
  std::vector<int64_t> off((size_t)n_rec + 1, 0);
  for (int64_t r = 0; r < n_rec; r++) off[(size_t)r] = h_tab[(size_t)r] - h_tab[0];
  off[(size_t)n_rec] = n_chars;
  gmg_seqset* s = NULL;
  if (seqset_build(ctx, d_out, off.data(), n_rec, NULL, &s)) return 1;
  s->hdr_off.assign(h_tab.begin() + (n_rec ? n_rec : 0), h_tab.begin() + (n_rec ? 2 * n_rec : 0));
  s->hdr_end.assign(h_tab.begin() + (n_rec ? 2 * n_rec : 0), h_tab.end());
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));  // d_out (scratch) has been consumed by the pack kernel
  if (seqset_finish_nacgt(ctx, s, d_out)) return 1;
  *out = s;
  if (n_records) *n_records = n_rec;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Quality-file ingest on the device (SURVEY.md section 8(f) row 1; Fasta_Qual_Vec_Read, Common/fasta.cc:115-170): records
// as in Fasta_Read -- a '>' outside a header line starts one, its header runs to the end of that line -- and in a
// record's body a value is the number formed by ALL digits since the last white-space character, taken when the next
// white-space character arrives (other characters are skipped; digits still pending at the next '>' or at the end of the
// file are dropped).  One thread per byte: a white-space byte of a body looks back to the previous white space / header
// byte for digits; the two scans of the FASTA ingest number the values and the records.
__device__ __forceinline__ bool qual_is_space(unsigned ch) { return ch == ' ' || (ch >= 9 && ch <= 13); }

// value ending at the white-space byte i (body byte): -1 if no digit since the previous reset point
__device__ __forceinline__ long long qual_value_before(const uint8_t* __restrict__ in, const uint32_t* __restrict__ last,
                                                       int64_t i, int* too_long) {
  long long val = 0, mul = 1;
  bool have = false;
  int steps = 0;
  for (int64_t j = i - 1; j >= 0; --j) {
    const unsigned ch = in[j];
    if ((last[j] & 1u) != 0 || qual_is_space(ch)) break;  // header byte (incl. the record's '>') or white space
    if (ch >= '0' && ch <= '9') {
      if (mul <= 1000000000ll) {
        val += (long long)(ch - '0') * mul;
        mul *= 10;
      } else if (ch != '0') {
        val = 0x7fffffffll;  // more than ten digits: saturate (the reference's int would overflow)
      }
      have = true;
    }
    if (++steps > 65536) {
      *too_long = 1;
      break;
    }
  }
  if (val > 0x7fffffffll) val = 0x7fffffffll;
  return have ? val : -1;
}

__global__ void __launch_bounds__(256) k_qual_flags(const uint8_t* __restrict__ in, int64_t n,
                                                    const uint32_t* __restrict__ last, uint2* __restrict__ flags,
                                                    int* __restrict__ too_long) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned ch = in[i];
  const bool in_hdr = (last[i] & 1u) != 0;
  const bool prev_hdr = i > 0 && (last[i - 1] & 1u) != 0;
  const bool start = ch == '>' && !prev_hdr;
  unsigned emit = 0;
  if (!in_hdr && qual_is_space(ch)) emit = qual_value_before(in, last, i, too_long) >= 0 ? 1u : 0u;
  flags[i] = make_uint2(emit, start ? 1u : 0u);
}

// values of all records, compacted (anything before the first record is dropped)
__global__ void __launch_bounds__(256) k_qual_scatter(const uint8_t* __restrict__ in, int64_t n,
                                                      const uint32_t* __restrict__ last, const uint2* __restrict__ incl,
                                                      const int64_t* __restrict__ rec_vals, int32_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint2 me = incl[i];
  const uint32_t before = i > 0 ? incl[i - 1].x : 0u;
  if (me.x != before && me.y > 0) {
    int dummy = 0;
    out[(int64_t)before - rec_vals[0]] = (int32_t)qual_value_before(in, last, i, &dummy);
  }
}

__global__ void __launch_bounds__(256) k_qual_clamp(const int32_t* __restrict__ v, int64_t n, uint8_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (uint8_t)(v[i] < 0 ? 0 : (v[i] > 255 ? 255 : v[i]));
}

// parse: *d_values = int32 values of all records (context scratch SCR_TMP2), off = values before each record
static int quality_parse(gmg_ctx* ctx, const char* h_bytes, int64_t n, std::vector<int64_t>* off, int32_t** d_values) {
  GMG_CHECK(n < (1ll << 30), "quality images of 1 GiB or more must be split at record boundaries (got %lld bytes)", (long long)n);
  off->assign(1, 0);
  *d_values = NULL;
  if (n == 0) return 0;
  void *d_in, *d_work;
  if (gmg_scratch(ctx, SCR_TMP, (size_t)n + 64, &d_in)) return 1;
  GMG_CUDA(cudaMemcpyAsync(d_in, h_bytes, (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  if (gmg_scratch(ctx, SCR_CUM, (size_t)n * 12 + 256, &d_work)) return 1;
  uint2* d_flags = (uint2*)d_work;
  uint32_t* d_key = (uint32_t*)(d_flags + n);
  int* d_err = (int*)(d_key + n);
  GMG_CUDA(cudaMemsetAsync(d_err, 0, sizeof(int), ctx->stream));
  const unsigned grid = (unsigned)((n + 255) / 256);
  k_fasta_keys<<<grid, 256, 0, ctx->stream>>>((const uint8_t*)d_in, n, d_key);
  size_t tb1 = 0, tb2 = 0;
  GMG_CUDA(cub::DeviceScan::InclusiveScan(NULL, tb1, d_key, d_key, FastaMaxOp(), n, ctx->stream));
  GMG_CUDA(cub::DeviceScan::InclusiveScan(NULL, tb2, d_flags, d_flags, FastaSumOp(), n, ctx->stream));
  void* d_tmp;
  if (gmg_scratch(ctx, SCR_TMP4, tb1 > tb2 ? tb1 : tb2, &d_tmp)) return 1;
  GMG_CUDA(cub::DeviceScan::InclusiveScan(d_tmp, tb1, d_key, d_key, FastaMaxOp(), n, ctx->stream));
  k_qual_flags<<<grid, 256, 0, ctx->stream>>>((const uint8_t*)d_in, n, d_key, d_flags, d_err);
  GMG_CUDA(cub::DeviceScan::InclusiveScan(d_tmp, tb2, d_flags, d_flags, FastaSumOp(), n, ctx->stream));
  ctx->launches += 4;
  GMG_CUDA(cudaMemcpyAsync(ctx->h_scalars + 4, d_flags + (n - 1), sizeof(uint2), cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaMemcpyAsync(ctx->h_scalars + 5, d_err, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  uint2 tot;
  memcpy(&tot, ctx->h_scalars + 4, sizeof tot);
  GMG_CHECK((ctx->h_scalars[5] & 0xffffffff) == 0, "quality file: more than 65536 characters without white space");
  int64_t n_rec = tot.y;
  if (n_rec == 0) return 0;
  void* d_tab;
  if (gmg_scratch(ctx, SCR_TMP3, (size_t)3 * n_rec * sizeof(int64_t), &d_tab)) return 1;
  int64_t* rec_vals = (int64_t*)d_tab;
  int64_t* hdr_off = rec_vals + n_rec;
  int64_t* hdr_end = hdr_off + n_rec;
  k_fill_i64<<<(unsigned)((n_rec + 255) / 256), 256, 0, ctx->stream>>>(hdr_end, n_rec, n);
  k_fasta_records<<<grid, 256, 0, ctx->stream>>>((const uint8_t*)d_in, n, d_key, d_flags, rec_vals, hdr_off, hdr_end);
  void* d_out;
  if (gmg_scratch(ctx, SCR_TMP2, ((size_t)tot.x + 16) * sizeof(int32_t), &d_out)) return 1;
  k_qual_scatter<<<grid, 256, 0, ctx->stream>>>((const uint8_t*)d_in, n, d_key, d_flags, rec_vals, (int32_t*)d_out);
  ctx->launches += 3;
  GMG_CUDA(cudaGetLastError());
  std::vector<int64_t> h_tab((size_t)3 * n_rec);
  GMG_CUDA(cudaMemcpyAsync(h_tab.data(), d_tab, h_tab.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  // a last record whose '>' is followed by nothing but blanks does not exist (fasta.cc:137-141)
  {
    int64_t q = h_tab[(size_t)(2 * n_rec - 1)];
    while (q < n && h_bytes[q] == ' ') q++;
    if (q == n) n_rec--;
  }
  off->assign((size_t)n_rec + 1, 0);
  for (int64_t r = 0; r < n_rec; r++) (*off)[(size_t)r] = h_tab[(size_t)r] - h_tab[0];
  (*off)[(size_t)n_rec] = (int64_t)tot.x - h_tab[0];
  *d_values = (int32_t*)d_out;
  return 0;
}

extern "C" int gmg_quality_parse_fasta(gmg_ctx* ctx, const char* h_bytes, int64_t n_bytes, int64_t* n_records,
                                       int64_t* n_values, int64_t* h_off, int32_t* h_values, int64_t cap_records,
                                       int64_t cap_values) {
  GMG_CHECK(ctx && n_bytes >= 0 && (h_bytes || n_bytes == 0), "gmg_quality_parse_fasta: bad argument");
  GMG_CUDA(cudaSetDevice(ctx->device));
  std::vector<int64_t> off;
  int32_t* d_values;
  if (quality_parse(ctx, h_bytes, n_bytes, &off, &d_values)) return 1;
  const int64_t n_rec = (int64_t)off.size() - 1, n_val = off.back();
  if (n_records) *n_records = n_rec;
  if (n_values) *n_values = n_val;
  if (h_off && cap_records >= n_rec) memcpy(h_off, off.data(), off.size() * sizeof(int64_t));
  if (h_values && cap_values >= n_val && n_val > 0) {
    GMG_CUDA(cudaMemcpyAsync(h_values, d_values, (size_t)n_val * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  return 0;
}

extern "C" int gmg_seqset_quality_from_fasta(gmg_ctx* ctx, gmg_seqset* s, const char* h_bytes, int64_t n_bytes) {
  GMG_CHECK(ctx && s && n_bytes >= 0 && (h_bytes || n_bytes == 0), "gmg_seqset_quality_from_fasta: bad argument");
  GMG_CUDA(cudaSetDevice(ctx->device));
  std::vector<int64_t> off;
  int32_t* d_values;
  if (quality_parse(ctx, h_bytes, n_bytes, &off, &d_values)) return 1;
  const int64_t n_rec = (int64_t)off.size() - 1;
  GMG_CHECK(n_rec == s->n, "quality file holds %lld records, the sequence set %lld", (long long)n_rec, (long long)s->n);
  for (int64_t r = 0; r < n_rec; r++)
    GMG_CHECK(off[(size_t)r + 1] - off[(size_t)r] == s->off[(size_t)r + 1] - s->off[(size_t)r],
              "ERROR:  record %lld sequence length does not match quality values length (%lld bases, %lld values)", (long long)r,
              (long long)(s->off[(size_t)r + 1] - s->off[(size_t)r]), (long long)(off[(size_t)r + 1] - off[(size_t)r]));
  if (s->total > 0) {
    if (!s->d_qual) GMG_CUDA(cudaMallocAsync(&s->d_qual, (size_t)s->total, ctx->stream));
    k_qual_clamp<<<(unsigned)((s->total + 255) / 256), 256, 0, ctx->stream>>>(d_values, s->total, s->d_qual);
    ctx->launches++;
    GMG_CUDA(cudaGetLastError());
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));  // the values live in context scratch
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// FASTQ ingest on the device: four-line records (header '@', sequence, '+' [header], qualities).  One scan over the
// '\n' marks gives every byte its line; record r is lines 4r .. 4r+3.  The records end at the line of the last
// non-white-space byte, so blank lines may follow the last record.  The first failure is the smallest (line, reason,
// byte) key of any check; it travels to the host with the record count in one stream synchronisation.
enum { FQ_NO_AT = 0, FQ_NO_PLUS = 1, FQ_PLUS_TEXT = 2, FQ_TRUNCATED = 3, FQ_QUAL_LEN = 4, FQ_QUAL_BYTE = 5 };

// line < 2^31, reason < 8, byte position < 2^30 (images are < 1 GiB)
__device__ __forceinline__ unsigned long long fq_key(int64_t line, unsigned reason, int64_t pos) {
  return ((unsigned long long)line << 33) | ((unsigned long long)reason << 30) | (unsigned long long)pos;
}

struct FqIsNewline {
  __host__ __device__ __forceinline__ uint32_t operator()(uint8_t c) const { return c == '\n' ? 1u : 0u; }
};

struct FqCtl {
  unsigned long long err;  // first failure (fq_key), ~0 = none
  int32_t last_nb;         // line of the last non-white-space byte, -1 = none
  uint32_t last_line;      // index of the last line (the text after a final '\n' is an empty last line)
};

// One thread per byte, line[i] = '\n' bytes before byte i.  starts[j] = first byte of line j, starts[last + 1] = n + 1,
// so line j ends (at its '\n' or at the image end) at starts[j + 1] - 1.  Also the range check of every quality byte
// (lines 4r+3 without their '\n' and one trailing '\r'): lines past the last record are blank, and a key on one of them
// sorts after every failure inside the records, so the host drops it.
__global__ void __launch_bounds__(256) k_fastq_lines(const uint8_t* __restrict__ in, int64_t n,
                                                     const uint32_t* __restrict__ line, unsigned lo,
                                                     uint32_t* __restrict__ starts, FqCtl* __restrict__ ctl) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int nb = -1;
  unsigned long long bad = ~0ull;
  if (i < n) {
    const unsigned ch = in[i];
    const uint32_t j = line[i];
    if (ch == '\n') starts[j + 1] = (uint32_t)(i + 1);
    if (i == 0) starts[0] = 0;
    if (i == n - 1) {
      const uint32_t last = j + (ch == '\n' ? 1u : 0u);
      starts[last + 1] = (uint32_t)(n + 1);
      ctl->last_line = last;
    }
    if (!fasta_is_space(ch)) nb = (int)j;
    if ((j & 3u) == 3u && ch != '\n' && !(ch == '\r' && (i + 1 == n || in[i + 1] == '\n')) && (ch < lo || ch > '~'))
      bad = fq_key(j, FQ_QUAL_BYTE, i);
  }
  nb = __reduce_max_sync(0xffffffffu, nb);
  if ((threadIdx.x & 31) == 0 && nb >= 0) atomicMax(&ctl->last_nb, nb);
  if (__any_sync(0xffffffffu, bad != ~0ull)) {
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long t = __shfl_xor_sync(0xffffffffu, bad, o);
      bad = t < bad ? t : bad;
    }
    if ((threadIdx.x & 31) == 0) atomicMin(&ctl->err, bad);
  }
}

// One warp per record (grid-stride; the record count is on the device): the '@' and '+' lines, the '+' text against the
// header, the sequence characters (non-white-space bytes of line 4r+1) and the quality line's length.  Writes the
// sequence length and the header span; seq_len[n_rec] = 0 so that an exclusive sum over n_rec + 1 entries ends in the total.
__global__ void __launch_bounds__(256) k_fastq_records(const uint8_t* __restrict__ in, const uint32_t* __restrict__ starts,
                                                       FqCtl* __restrict__ ctl, uint32_t* __restrict__ seq_len,
                                                       uint32_t* __restrict__ hdr_off, uint32_t* __restrict__ hdr_end) {
  const int lane = threadIdx.x & 31;
  const int64_t last_nb = ctl->last_nb, last_line = ctl->last_line;
  const int64_t n_rec = last_nb < 0 ? 0 : last_nb / 4 + 1;
  if (blockIdx.x == 0 && threadIdx.x == 0) seq_len[n_rec] = 0;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n_rec; r += warps) {
    const int64_t l0 = 4 * r;
    const int64_t have = last_line - l0 + 1;  // lines of the record in the image (>= 1)
    unsigned long long err = have < 4 ? fq_key(last_line + 1, FQ_TRUNCATED, 0) : ~0ull;
    // header: '@', then the text after the blanks, to the line end
    const int64_t h0 = starts[l0], h1 = (int64_t)starts[l0 + 1] - 1;
    int64_t ho = h1;
    if (h1 > h0 && in[h0] == '@') {
      ho = h0 + 1;
      while (ho < h1 && in[ho] == ' ') ho++;
    } else {
      err = min(err, fq_key(l0, FQ_NO_AT, h0));
    }
    unsigned cnt = 0;
    if (have >= 2) {
      const int64_t s0 = starts[l0 + 1], s1 = (int64_t)starts[l0 + 2] - 1;
      for (int64_t p = s0 + lane; p < s1; p += 32) cnt += fasta_is_space(in[p]) ? 0u : 1u;
      cnt = __reduce_add_sync(0xffffffffu, cnt);
    }
    if (have >= 3) {
      const int64_t p0 = starts[l0 + 2], p1 = (int64_t)starts[l0 + 3] - 1;
      if (p1 > p0 && in[p0] == '+') {
        int64_t pt = p0 + 1, pe = p1, he = h1;  // one trailing '\r' of either line does not count
        while (pt < pe && in[pt] == ' ') pt++;
        if (pe > pt && in[pe - 1] == '\r') pe--;
        if (he > ho && in[he - 1] == '\r') he--;
        if (pe > pt) {
          bool differ = pe - pt != he - ho;
          if (!differ) {
            bool d = false;
            for (int64_t k = lane; k < pe - pt; k += 32) d |= in[pt + k] != in[ho + k];
            differ = __any_sync(0xffffffffu, d);
          }
          if (differ) err = min(err, fq_key(l0 + 2, FQ_PLUS_TEXT, p0));
        }
      } else {
        err = min(err, fq_key(l0 + 2, FQ_NO_PLUS, p0));
      }
    }
    if (have >= 4) {
      const int64_t q0 = starts[l0 + 3];
      int64_t q1 = (int64_t)starts[l0 + 4] - 1;
      if (q1 > q0 && in[q1 - 1] == '\r') q1--;
      if (q1 - q0 != (int64_t)cnt) err = min(err, fq_key(l0 + 3, FQ_QUAL_LEN, q0));
    }
    if (lane == 0) {
      seq_len[r] = cnt;
      hdr_off[r] = (uint32_t)ho;
      hdr_end[r] = (uint32_t)h1;
      if (err != ~0ull) atomicMin(&ctl->err, err);
    }
  }
}

// One warp per record of a checked image: the sequence characters to seq[off[r] ..) (a ballot keeps their order past
// white space) and the quality bytes minus the Phred offset to qual[off[r] ..)
__global__ void __launch_bounds__(256) k_fastq_copy(const uint8_t* __restrict__ in, const uint32_t* __restrict__ starts,
                                                    const int64_t* __restrict__ off, int64_t n_rec, unsigned lo,
                                                    uint8_t* __restrict__ seq, uint8_t* __restrict__ qual) {
  const int lane = threadIdx.x & 31;
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n_rec) return;  // warp-uniform
  const int64_t s0 = starts[4 * r + 1], s1 = (int64_t)starts[4 * r + 2] - 1, q0 = starts[4 * r + 3];
  const int64_t o = off[r], len = off[r + 1] - o;
  int64_t k = o;
  for (int64_t p = s0; p < s1; p += 32) {
    const unsigned ch = p + lane < s1 ? in[p + lane] : ' ';
    const bool keep = !fasta_is_space(ch);
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (keep) seq[k + __popc(m & ((1u << lane) - 1u))] = (uint8_t)ch;
    k += __popc(m);
  }
  for (int64_t t = lane; t < len; t += 32) qual[o + t] = (uint8_t)(in[q0 + t] - lo);
}

// the message of the first failure (key from k_fastq_lines / k_fastq_records)
static int fastq_error(gmg_ctx* ctx, const char* h_bytes, int64_t n, int phred_offset, unsigned long long key,
                       const uint32_t* d_seq_len) {
  const int64_t line = (int64_t)(key >> 33), pos = (int64_t)(key & ((1ull << 30) - 1));
  const int reason = (int)((key >> 30) & 7);
  const long long rec = line / 4 + 1, ln = line + 1;
  switch (reason) {
    case FQ_NO_AT:
      gmg_set_error("gmg_seqset_from_fastq: record %lld (line %lld): the header line does not start with '@' "
                    "(multi-line FASTQ records are not supported)", rec, ln);
      break;
    case FQ_NO_PLUS:
      gmg_set_error("gmg_seqset_from_fastq: record %lld (line %lld): the separator line does not start with '+' "
                    "(multi-line FASTQ records are not supported)", rec, ln);
      break;
    case FQ_PLUS_TEXT:
      gmg_set_error("gmg_seqset_from_fastq: record %lld (line %lld): the text after '+' differs from the header", rec, ln);
      break;
    case FQ_TRUNCATED: {
      static const char* role[4] = {"header", "sequence", "'+'", "quality"};
      gmg_set_error("gmg_seqset_from_fastq: record %lld (line %lld): truncated last record: the image ends before its %s "
                    "line", rec, ln, role[line & 3]);
      break;
    }
    case FQ_QUAL_LEN: {
      uint32_t cnt = 0;
      GMG_CUDA(cudaMemcpyAsync(&cnt, d_seq_len + (rec - 1), sizeof cnt, cudaMemcpyDeviceToHost, ctx->stream));
      GMG_CUDA(cudaStreamSynchronize(ctx->stream));
      const char* nl = (const char*)memchr(h_bytes + pos, '\n', (size_t)(n - pos));
      int64_t q1 = nl ? nl - h_bytes : n;
      if (q1 > pos && h_bytes[q1 - 1] == '\r') q1--;
      gmg_set_error("gmg_seqset_from_fastq: record %lld (line %lld): the quality line holds %lld characters, the sequence "
                    "%lld", rec, ln, (long long)(q1 - pos), (long long)cnt);
      break;
    }
    default: {
      int64_t a = pos;
      while (a > 0 && h_bytes[a - 1] != '\n') a--;
      gmg_set_error("gmg_seqset_from_fastq: record %lld (line %lld): quality byte %d at column %lld is outside [%d, 126] "
                    "(phred offset %d)", rec, ln, (int)(uint8_t)h_bytes[pos], (long long)(pos - a + 1), phred_offset,
                    phred_offset);
      break;
    }
  }
  return 1;
}

extern "C" int gmg_seqset_from_fastq(gmg_ctx* ctx, const char* h_bytes, int64_t n_bytes, int phred_offset,
                                     gmg_seqset** out, int64_t* n_records) {
  GMG_CHECK(ctx && out && n_bytes >= 0 && (h_bytes || n_bytes == 0), "gmg_seqset_from_fastq: bad argument");
  *out = NULL;
  if (n_records) *n_records = 0;
  GMG_CHECK(phred_offset == 33 || phred_offset == 64, "gmg_seqset_from_fastq: phred_offset must be 33 or 64 (got %d)",
            phred_offset);
  GMG_CHECK(n_bytes < (1ll << 30), "gmg_seqset_from_fastq: images of 1 GiB or more must be split at record boundaries "
            "(got %lld bytes)", (long long)n_bytes);
  GMG_CUDA(cudaSetDevice(ctx->device));
  const int64_t n = n_bytes;
  const unsigned lo = (unsigned)phred_offset;
  int64_t n_rec = 0;
  std::vector<int64_t> off(1, 0), hdr_off, hdr_end;
  void *d_seq = NULL, *d_qual = NULL;
  if (n > 0) {
    void *d_in, *d_work, *d_tab, *d_tmp;
    if (gmg_scratch(ctx, SCR_TMP, (size_t)n + 64, &d_in)) return 1;
    GMG_CUDA(cudaMemcpyAsync(d_in, h_bytes, (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    // line of every byte | line starts (at most n + 1 lines, plus the end sentinel) | control block
    if (gmg_scratch(ctx, SCR_CUM, (size_t)(2 * n + 2) * sizeof(uint32_t) + 64, &d_work)) return 1;
    uint32_t* d_line = (uint32_t*)d_work;
    uint32_t* d_starts = d_line + n;
    FqCtl* d_ctl = (FqCtl*)(((uintptr_t)(d_starts + n + 2) + 15) & ~(uintptr_t)15);
    // per record (at most (n + 1) / 4 + 1 of them): offsets (int64) | sequence length | header start | header end
    const int64_t cap = n / 4 + 2;
    if (gmg_scratch(ctx, SCR_TMP3, (size_t)cap * (sizeof(int64_t) + 3 * sizeof(uint32_t)), &d_tab)) return 1;
    int64_t* d_off = (int64_t*)d_tab;
    uint32_t* d_len = (uint32_t*)(d_off + cap);
    uint32_t* d_hoff = d_len + cap;
    uint32_t* d_hend = d_hoff + cap;
    GMG_CUDA(cudaMemsetAsync(d_ctl, 0xFF, sizeof(FqCtl), ctx->stream));  // err = ~0, last_nb = -1
    const auto nl = thrust::make_transform_iterator((const uint8_t*)d_in, FqIsNewline());
    size_t tb = 0;
    GMG_CUDA(cub::DeviceScan::ExclusiveSum(NULL, tb, nl, d_line, n, ctx->stream));
    if (gmg_scratch(ctx, SCR_TMP4, tb, &d_tmp)) return 1;
    GMG_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tb, nl, d_line, n, ctx->stream));
    k_fastq_lines<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>((const uint8_t*)d_in, n, d_line, lo, d_starts,
                                                                        d_ctl);
    const int64_t rblk = (cap + 7) / 8;  // eight warps a block
    k_fastq_records<<<(unsigned)(rblk < 16 * ctx->sm_count ? rblk : 16 * ctx->sm_count), 256, 0, ctx->stream>>>(
        (const uint8_t*)d_in, d_starts, d_ctl, d_len, d_hoff, d_hend);
    ctx->launches += 3;
    GMG_CUDA(cudaGetLastError());
    GMG_CUDA(cudaMemcpyAsync(ctx->h_scalars + 4, d_ctl, sizeof(FqCtl), cudaMemcpyDeviceToHost, ctx->stream));
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));
    FqCtl c;
    memcpy(&c, ctx->h_scalars + 4, sizeof c);
    n_rec = c.last_nb < 0 ? 0 : (int64_t)c.last_nb / 4 + 1;
    if (c.err != ~0ull && (int64_t)(c.err >> 33) < 4 * n_rec) return fastq_error(ctx, h_bytes, n, phred_offset, c.err, d_len);
    if (n_rec > 0) {
      GMG_CUDA(cub::DeviceScan::ExclusiveSum(NULL, tb, d_len, d_off, n_rec + 1, ctx->stream));
      if (gmg_scratch(ctx, SCR_TMP4, tb, &d_tmp)) return 1;
      GMG_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tb, d_len, d_off, n_rec + 1, ctx->stream));
      // at most n sequence characters
      if (gmg_scratch(ctx, SCR_TMP2, (size_t)n + 64, &d_seq)) return 1;
      if (gmg_scratch(ctx, SCR_QUAL, (size_t)n + 64, &d_qual)) return 1;
      k_fastq_copy<<<(unsigned)((n_rec + 7) / 8), 256, 0, ctx->stream>>>((const uint8_t*)d_in, d_starts, d_off, n_rec, lo,
                                                                         (uint8_t*)d_seq, (uint8_t*)d_qual);
      ctx->launches += 2;
      GMG_CUDA(cudaGetLastError());
      // offsets | header starts | header ends through the context's page-locked staging
      const size_t ob = (size_t)(n_rec + 1) * sizeof(int64_t), hb = (size_t)n_rec * sizeof(uint32_t);
      if (gmg_host_stage(ctx, ob + 2 * hb, 0)) return 1;
      char* st = (char*)ctx->h_stage;
      GMG_CUDA(cudaMemcpyAsync(st, d_off, ob, cudaMemcpyDeviceToHost, ctx->stream));
      GMG_CUDA(cudaMemcpyAsync(st + ob, d_hoff, hb, cudaMemcpyDeviceToHost, ctx->stream));
      GMG_CUDA(cudaMemcpyAsync(st + ob + hb, d_hend, hb, cudaMemcpyDeviceToHost, ctx->stream));
      GMG_CUDA(cudaStreamSynchronize(ctx->stream));
      off.assign((const int64_t*)st, (const int64_t*)st + n_rec + 1);
      hdr_off.assign((const uint32_t*)(st + ob), (const uint32_t*)(st + ob) + n_rec);
      hdr_end.assign((const uint32_t*)(st + ob + hb), (const uint32_t*)(st + ob + hb) + n_rec);
    }
  }
  gmg_seqset* s = NULL;
  if (seqset_build(ctx, d_seq, off.data(), n_rec, d_qual, &s)) return 1;
  s->hdr_off.swap(hdr_off);
  s->hdr_end.swap(hdr_end);
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));  // d_seq / d_qual (scratch) have been consumed
  if (seqset_finish_nacgt(ctx, s, d_seq)) {
    gmg_seqset_free(s);
    return 1;
  }
  *out = s;
  if (n_records) *n_records = n_rec;
  return 0;
}

extern "C" int gmg_seqset_qualities(const gmg_seqset* s, uint8_t* h_out) {
  GMG_CHECK(s, "gmg_seqset_qualities: NULL set");
  GMG_CHECK(s->d_qual, "gmg_seqset_qualities: the set has no qualities");
  if (!h_out) return 0;
  GMG_CUDA(cudaSetDevice(s->ctx->device));
  GMG_CUDA(cudaMemcpyAsync(h_out, s->d_qual, (size_t)s->total, cudaMemcpyDeviceToHost, s->ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(s->ctx->stream));
  return 0;
}

extern "C" int64_t gmg_seqset_count(const gmg_seqset* s) { return s ? s->n : 0; }

extern "C" int gmg_seqset_offsets(const gmg_seqset* s, int64_t* h_off) {
  GMG_CHECK(s && h_off, "gmg_seqset_offsets: NULL argument");
  memcpy(h_off, s->off.data(), s->off.size() * sizeof(int64_t));
  return 0;
}

extern "C" int gmg_seqset_fasta_headers(const gmg_seqset* s, int64_t* h_hdr_off, int64_t* h_hdr_end) {
  GMG_CHECK(s && h_hdr_off && h_hdr_end, "gmg_seqset_fasta_headers: NULL argument");
  GMG_CHECK((int64_t)s->hdr_off.size() == s->n, "gmg_seqset_fasta_headers: the seqset was not built by gmg_seqset_from_fasta");
  memcpy(h_hdr_off, s->hdr_off.data(), s->hdr_off.size() * sizeof(int64_t));
  memcpy(h_hdr_end, s->hdr_end.data(), s->hdr_end.size() * sizeof(int64_t));
  return 0;
}

extern "C" void gmg_seqset_free(gmg_seqset* s) {
  if (!s) return;
  cudaSetDevice(s->ctx->device);
  void* ptrs[] = {s->d_off, s->d_words_base, s->d_blk2seq, s->d_qual, s->d_gc, s->d_orfs, s->d_orf_off,
                  s->d_orf_seq, s->d_starts, s->d_start_off, s->d_cbits, s->d_bktidx, s->d_ctxf, s->d_ctxr,
                  s->d_nacgt};
  for (void* p : ptrs)
    if (p) cudaFreeAsync(p, s->ctx->stream);
  delete s;
}

extern "C" int64_t gmg_seqset_total_bases(const gmg_seqset* s) { return s ? s->total : 0; }

extern "C" int gmg_seqset_gc_fraction(gmg_seqset* s, double* gc) {
  GMG_CHECK(s && gc, "gmg_seqset_gc_fraction: NULL argument");
  unsigned long long ct = 0;
  GMG_CUDA(cudaMemcpyAsync(&ct, s->d_gc, sizeof ct, cudaMemcpyDeviceToHost, s->ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(s->ctx->stream));
  // the reference counts in `unsigned int` and divides as double (glimmer_base.cc:2571-2590)
  *gc = (double)(unsigned int)ct / (double)(unsigned int)s->total;
  return 0;
}

extern "C" int gmg_seqset_unpack(gmg_seqset* s, char* h_out) {
  GMG_CHECK(s && h_out, "gmg_seqset_unpack: NULL argument");
  if (s->total == 0) return 0;
  gmg_ctx* ctx = s->ctx;
  void* d = NULL;
  if (gmg_scratch(ctx, SCR_TMP, (size_t)s->total, &d)) return 1;
  k_unpack<<<(unsigned)((s->total + 255) / 256), 256, 0, ctx->stream>>>(s->d_words, s->total, (char*)d);
  ctx->launches++;
  GMG_CUDA(cudaGetLastError());
  GMG_CUDA(cudaMemcpyAsync(h_out, d, (size_t)s->total, cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// extract (Util/extract.cc) on a resident set.  Output sequence r is region r: bases [from[r], from[r] + len_r) of the
// source (global base indices), read upwards on strand +1; on strand -1 read downwards and complemented.  The reference
// complements the raw IUPAC code (Complement, Common/delcher.cc) and build-icm applies Filter afterwards; the 2-bit
// complement 3 - code equals that for a / c / g / t only, so the positions of the source's non-acgt list that fall into
// minus regions are patched with Filter(Complement(raw)).

// Complement of a lower-case IUPAC code; every other byte becomes 'n', so the complement of a non-acgt byte is again
// non-acgt and the output list has one entry per source entry inside a region.
__device__ __forceinline__ unsigned iupac_complement(unsigned ch) {
  switch (ch) {
    case 'a': return 't';
    case 'c': return 'g';
    case 'g': return 'c';
    case 't': return 'a';
    case 'r': return 'y';
    case 'y': return 'r';
    case 'm': return 'k';
    case 'k': return 'm';
    case 'b': return 'v';
    case 'v': return 'b';
    case 'd': return 'h';
    case 'h': return 'd';
    case 's': return 's';
    case 'w': return 'w';
    default: return 'n';
  }
}

// first index of the (position-sorted) list whose position is >= p
__device__ __forceinline__ int64_t nacgt_lower_bound(const uint64_t* __restrict__ list, int64_t n, int64_t p) {
  int64_t lo = 0, hi = n;
  const uint64_t key = (uint64_t)p << 8;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (__ldg(list + mid) < key) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

// largest r < n with key[r] <= x (key ascending, key[0] <= x): the region of an output position (off) or of an output
// list entry (list_base).  Empty regions share their key with the next one, so the search lands on a non-empty one.
__device__ __forceinline__ int64_t last_at_or_below(const int64_t* __restrict__ key, int64_t n, int64_t x) {
  int64_t lo = 0, hi = n;
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (__ldg(key + mid) <= x) lo = mid;
    else hi = mid;
  }
  return lo;
}

// per region: the source list entries inside it, [first[r], first[r] + cnt[r])
__global__ void __launch_bounds__(256) k_extract_count(const uint64_t* __restrict__ list, int64_t n_list,
                                                       const int64_t* __restrict__ off, const int64_t* __restrict__ from,
                                                       int64_t n, int64_t* __restrict__ first, int64_t* __restrict__ cnt) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int64_t a = nacgt_lower_bound(list, n_list, from[r]);
  const int64_t b = nacgt_lower_bound(list, n_list, from[r] + (off[r + 1] - off[r]));
  first[r] = a;
  cnt[r] = b - a;
}

// one thread per output word: each region piece inside the word is a two-word funnel shift of the source (plus, on
// strand -1, base reversal, complement and the non-acgt patch); then the word's g + c count
__global__ void __launch_bounds__(256) k_extract_words(const uint64_t* __restrict__ src, const uint64_t* __restrict__ list,
                                                       int64_t n_list, const int64_t* __restrict__ off,
                                                       const int64_t* __restrict__ from, const int8_t* __restrict__ strand,
                                                       int64_t n, int64_t total, uint64_t* __restrict__ words,
                                                       unsigned long long* __restrict__ gc) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned my_gc = 0;
  if (w < ((total + 31) >> 5)) {
    const int64_t w0 = w << 5, end = w0 + 32 < total ? w0 + 32 : total;
    uint64_t v = 0;
    for (int64_t p = w0; p < end;) {
      const int64_t r = last_at_or_below(off, n, p);
      const int64_t a = __ldg(off + r), e = __ldg(off + r + 1);
      const int64_t q = e < end ? e : end;
      const int m = (int)(q - p);
      const int64_t k = p - a;  // offset of the piece in its region
      uint64_t x;
      if (__ldg(strand + r) > 0) {
        x = gmg_extract32(src, __ldg(from + r) + k);
      } else {
        const int64_t s0 = __ldg(from + r) + (e - a) - k - m;  // lowest source base of the piece
        x = ~gmg_reverse_bases(gmg_extract32(src, s0), m);  // 3 - code = code ^ 3
        for (int64_t i = n_list ? nacgt_lower_bound(list, n_list, s0) : 0; i < n_list; i++) {
          const uint64_t ent = __ldg(list + i);
          const int64_t ps = (int64_t)(ent >> 8);
          if (ps >= s0 + m) break;
          const int j = (int)(s0 + m - 1 - ps);  // its place in the piece
          x = (x & ~(3ull << (2 * j))) | ((uint64_t)filter_code(iupac_complement((unsigned)(ent & 0xFF))) << (2 * j));
        }
      }
      if (m < 32) x &= (1ull << (2 * m)) - 1ull;
      v |= x << (2 * (p - w0));
      p = q;
    }
    words[w] = v;
    my_gc = word_gc(v);
  }
  warp_add_gc(my_gc, gc);
}

// one thread per output list entry: its region (by the exclusive sum `base` of cnt), the source entry, the new position
// and, on strand -1, the complemented code; regions are in output order and a minus region takes its entries in reverse,
// so the output list is position-sorted
__global__ void __launch_bounds__(256) k_extract_list(const uint64_t* __restrict__ list, const int64_t* __restrict__ off,
                                                      const int64_t* __restrict__ from, const int8_t* __restrict__ strand,
                                                      int64_t n, const int64_t* __restrict__ first,
                                                      const int64_t* __restrict__ cnt, const int64_t* __restrict__ base,
                                                      int64_t n_out, uint64_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_out) return;
  const int64_t r = last_at_or_below(base, n, i);
  const int64_t k = i - base[r];
  const int64_t a = off[r], len = off[r + 1] - a;
  uint64_t ent;
  int64_t pos;
  unsigned ch;
  if (strand[r] > 0) {
    ent = list[first[r] + k];
    pos = a + ((int64_t)(ent >> 8) - from[r]);
    ch = (unsigned)(ent & 0xFF);
  } else {
    ent = list[first[r] + cnt[r] - 1 - k];
    pos = a + (from[r] + len - 1 - (int64_t)(ent >> 8));
    ch = iupac_complement((unsigned)(ent & 0xFF));
  }
  out[i] = ((uint64_t)pos << 8) | ch;
}

extern "C" int gmg_seqset_extract(gmg_ctx* ctx, gmg_seqset* src, int64_t n, const int32_t* h_seq, const int32_t* h_lo,
                                  const int32_t* h_len, const int8_t* h_strand, gmg_seqset** out) {
  GMG_CHECK(ctx && src && out && (n == 0 || (h_seq && h_lo && h_len && h_strand)), "gmg_seqset_extract: NULL argument");
  GMG_CHECK(n >= 0 && n < (1ll << 31), "gmg_seqset_extract: %lld regions unsupported", (long long)n);
  std::vector<int64_t> off((size_t)n + 1, 0), from((size_t)n);
  for (int64_t i = 0; i < n; i++) {
    GMG_CHECK(h_seq[i] >= 0 && h_seq[i] < src->n, "gmg_seqset_extract: region %lld: sequence %d out of range (the set "
              "holds %lld)", (long long)i, h_seq[i], (long long)src->n);
    const int64_t L = src->off[(size_t)h_seq[i] + 1] - src->off[(size_t)h_seq[i]];
    GMG_CHECK(h_lo[i] >= 0, "gmg_seqset_extract: region %lld: start %d is negative", (long long)i, h_lo[i]);
    GMG_CHECK(h_len[i] >= 0 && (int64_t)h_lo[i] + h_len[i] <= L, "gmg_seqset_extract: region %lld: [%d, %lld) is not "
              "inside its %lld bp sequence %d", (long long)i, h_lo[i], (long long)h_lo[i] + h_len[i], (long long)L, h_seq[i]);
    GMG_CHECK(h_strand[i] == 1 || h_strand[i] == -1, "gmg_seqset_extract: region %lld: strand %d is not +1 or -1",
              (long long)i, (int)h_strand[i]);
    off[(size_t)i + 1] = off[(size_t)i] + h_len[i];
    from[(size_t)i] = src->off[(size_t)h_seq[i]] + h_lo[i];
  }
  GMG_CUDA(cudaSetDevice(ctx->device));
  gmg_seqset* s;
  if (seqset_alloc(ctx, off.data(), n, &s, false)) return 1;
  if (s->total == 0) {
    *out = s;
    return 0;
  }
  // region table: from | first | cnt | base (int64 [n] each) | strand (int8 [n])
  void* d_tab;
  if (gmg_scratch(ctx, SCR_MISC, (size_t)n * (4 * sizeof(int64_t) + 1) + 64, &d_tab)) return 1;
  int64_t* d_from = (int64_t*)d_tab;
  int64_t* d_first = d_from + n;
  int64_t* d_cnt = d_first + n;
  int64_t* d_base = d_cnt + n;
  int8_t* d_strand = (int8_t*)(d_base + n);
  GMG_CUDA(cudaMemcpyAsync(d_from, from.data(), (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
  GMG_CUDA(cudaMemcpyAsync(d_strand, h_strand, (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  const unsigned grid_r = (unsigned)((n + 255) / 256);
  if (src->n_nacgt > 0) {
    k_extract_count<<<grid_r, 256, 0, ctx->stream>>>(src->d_nacgt, src->n_nacgt, s->d_off, d_from, n, d_first, d_cnt);
    size_t tmp_bytes = 0;
    void* d_tmp;
    GMG_CUDA(cub::DeviceScan::ExclusiveSum(NULL, tmp_bytes, d_cnt, d_base, n, ctx->stream));
    if (gmg_scratch(ctx, SCR_TMP4, tmp_bytes, &d_tmp)) return 1;
    GMG_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_cnt, d_base, n, ctx->stream));
    ctx->launches += 2;
    ctx->h_scalars[15] = ctx->h_scalars[14] = 0;
    GMG_CUDA(cudaMemcpyAsync(ctx->h_scalars + 14, d_base + n - 1, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    GMG_CUDA(cudaMemcpyAsync(ctx->h_scalars + 15, d_cnt + n - 1, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  }
  const int64_t nwords = (s->total + 31) >> 5;
  k_extract_words<<<(unsigned)((nwords + 255) / 256), 256, 0, ctx->stream>>>(src->d_words, src->d_nacgt, src->n_nacgt,
                                                                             s->d_off, d_from, d_strand, n, s->total,
                                                                             s->d_words, s->d_gc);
  ctx->launches++;
  GMG_CUDA(cudaGetLastError());
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  if (src->n_nacgt > 0) {
    const int64_t n_out = ctx->h_scalars[14] + ctx->h_scalars[15];
    if (n_out > 0) {
      GMG_CUDA(cudaMallocAsync(&s->d_nacgt, (size_t)n_out * sizeof(uint64_t), ctx->stream));
      k_extract_list<<<(unsigned)((n_out + 255) / 256), 256, 0, ctx->stream>>>(src->d_nacgt, s->d_off, d_from, d_strand, n,
                                                                               d_first, d_cnt, d_base, n_out, s->d_nacgt);
      ctx->launches++;
      GMG_CUDA(cudaGetLastError());
      s->n_nacgt = n_out;
      GMG_CUDA(cudaStreamSynchronize(ctx->stream));
    }
  }
  *out = s;
  return 0;
}
