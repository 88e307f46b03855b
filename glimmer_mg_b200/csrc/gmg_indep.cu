// glimmer_mg_b200/csrc/gmg_indep.cu -- the independent models of many GC fractions, built on the device
// (gmg_score_orfs_mg_gc: glimmer-mg -c builds Build_Indep_WO_Stops once per read, glimmer-mg.cc).
//
// Build_Indep_WO_Stops (icm.cc:65-216, gmg_indep_tables) makes an ICM_t(3,2,3) whose topology (mip) does not depend on
// the GC fraction.  Only 108 log-probabilities do: the 21 nodes of period 0, the root of period 1 and the 5 nodes of
// period 2, 4 each ("slots").  Every other node never receives a count and holds 0.  The device view (prob, lut3, lutp)
// is a GC-independent gather of those slots, so one CTA per GC value forms the 108 values and writes the model's record
// (GMG_INDEP_REC floats) through the gather table.
//
// Bit-exactness with the host build: the arithmetic is the host's, operation by operation and in its order, with
// explicit round-to-nearest FP64 intrinsics (no contraction): gc / 2.0, 0.5 - x, the codon products, the 1e-20 stop
// entries, the 64-term sum and the divisions, the float accumulators (acc += double rounds to float at every step), the
// node sums and acc / s.  The last step, (float) log(x), uses the device's log, whose error bound (1 ulp, CUDA C
// Programming Guide) differs from glibc's: an entry is CERTIFIED when every double within 4 ulps of the device's result
// rounds to the same float -- then glibc's result, also within that bound of the exact value, rounds to it as well.  The
// models with an uncertified entry are listed; one copy brings the list back, the host builds them with glibc
// (gmg_indep_tables) and one copy plus k_indep_fix write their records (the scheme of k4_gather_flagged /
// k4_apply_flagged in training).  GMG_INDEP_FORCE_HOST=1 withdraws every certificate (tests).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "gmg_internal.cuh"

#define INDEP_SLOTS 108  // GC-dependent values of a model; slot 108 (and the padding up to 112) holds 0
#define INDEP_PAD 112

// first slot of node `node` of period f, -1 for the nodes that never receive a count
__host__ __device__ __forceinline__ int indep_slot(int f, int node) {
  if (f == 0) return 4 * node;
  if (f == 1) return node == 0 ? 84 : -1;
  return node <= 4 ? 88 + 4 * node : -1;
}

struct IndepStops {
  int n;
  int j[8];  // codon index of every stop codon, reversed as Build_Indep_WO_Stops enters it
};

__global__ void __launch_bounds__(128) k_indep_build(const double* __restrict__ gc, IndepStops st,
                                                     const uint8_t* __restrict__ src, float* __restrict__ rec,
                                                     int32_t* __restrict__ flagged, unsigned long long* __restrict__ counts,
                                                     int force_host) {
  __shared__ double s_cp[64];
  __shared__ double s_sum;
  __shared__ float s_acc[INDEP_PAD];
  __shared__ float s_val[INDEP_PAD];
  __shared__ int s_nflag;
  const int64_t m = blockIdx.x;
  const int t = threadIdx.x;
  if (t == 0) s_nflag = 0;
  const double b1 = __ddiv_rn(gc[m], 2.0), b0 = __dsub_rn(0.5, b1);  // base_prob[1] = base_prob[2], [0] = [3]
  if (t < 64) {
    const int x = (t >> 4) & 3, y = (t >> 2) & 3, z = t & 3;
    const double px = (x == 1 || x == 2) ? b1 : b0, py = (y == 1 || y == 2) ? b1 : b0, pz = (z == 1 || z == 2) ? b1 : b0;
    s_cp[t] = __dmul_rn(__dmul_rn(px, py), pz);
  }
  __syncthreads();
  if (t == 0) {
    for (int i = 0; i < st.n; i++) s_cp[st.j[i]] = 1e-20;
    double sum = 0.0;
    for (int c = 0; c < 64; c++) sum = __dadd_rn(sum, s_cp[c]);
    s_sum = sum;
  }
  __syncthreads();
  if (t < 64) s_cp[t] = __ddiv_rn(s_cp[t], s_sum);
  __syncthreads();
  // accumulator of slot t: every codon whose bases select its node and predicted base, in ascending codon order
  if (t < INDEP_SLOTS) {
    const int f = t < 84 ? 0 : (t < 88 ? 1 : 2);
    const int node = f == 0 ? t >> 2 : (f == 1 ? 0 : (t - 88) >> 2), k = t & 3;
    const int sh1 = 2 * ((3 - f) % 3), sh2 = 2 * ((4 - f) % 3), sh3 = 2 * ((5 - f) % 3);  // c / pw[.] % 4 as shifts
    float a = 0.f;
    for (int c = 0; c < 64; c++) {
      bool take = ((c >> sh1) & 3) == k;
      if (node >= 1 && node <= 4) take = take && ((c >> sh2) & 3) == node - 1;
      if (node >= 5) take = take && ((c >> sh2) & 3) == (node - 5) >> 2 && ((c >> sh3) & 3) == ((node - 5) & 3);
      if (take) a = __double2float_rn(__dadd_rn((double)a, s_cp[c]));
    }
    s_acc[t] = a;
  }
  __syncthreads();
  float v = 0.f;
  if (t < INDEP_SLOTS) {
    const int b = t & ~3;
    double s = 0.0;
    for (int k = 0; k < 4; k++) s = __dadd_rn(s, (double)s_acc[b + k]);
    if (s != 0.0) {
      const double x = __ddiv_rn((double)s_acc[t], s);
      const double y = log(x);
      v = __double2float_rn(y);
      bool ok = true;
      if (x != 0.0) {  // log(0) = -inf in both libraries
        const double e = fabs(y) * 0x1p-50;  // >= 4 ulps of y
        ok = __double2float_rn(y - e) == v && __double2float_rn(y + e) == v;
      }
      if (!ok || force_host) atomicAdd(&s_nflag, 1);
    }
  }
  if (t < INDEP_PAD) s_val[t] = v;
  __syncthreads();
  if (t == 0 && s_nflag) {
    flagged[atomicAdd(counts, 1ull)] = (int32_t)m;
    atomicAdd(counts + 1, (unsigned long long)s_nflag);
  }
  float* r = rec + (size_t)m * GMG_INDEP_REC;
  for (int i = t; i < GMG_INDEP_REC; i += blockDim.x) r[i] = s_val[__ldg(src + i)];
}

// the host's values of the flagged models into their records (vals: [n][INDEP_PAD])
__global__ void __launch_bounds__(128) k_indep_fix(const int32_t* __restrict__ models, const float* __restrict__ vals,
                                                   int64_t n, const uint8_t* __restrict__ src, float* __restrict__ rec) {
  __shared__ float s_val[INDEP_PAD];
  const int64_t b = blockIdx.x;
  if (b >= n) return;  // the launch is made with at least one CTA
  if (threadIdx.x < INDEP_PAD) s_val[threadIdx.x] = vals[b * INDEP_PAD + threadIdx.x];
  __syncthreads();
  float* r = rec + (size_t)models[b] * GMG_INDEP_REC;
  for (int i = threadIdx.x; i < GMG_INDEP_REC; i += blockDim.x) r[i] = s_val[__ldg(src + i)];
}

// The shared topology (a host-built model of any GC fraction: only its walk tables are used) and the gather table
// slot <- record entry, built once per context.
static int indep_topology(gmg_ctx* ctx, const gmg_params* p) {
  if (ctx->indep_tpl) return 0;
  const char* stops[8];
  for (int i = 0; i < p->n_stop; i++) stops[i] = p->stop_codon[i];
  gmg_icm* m = NULL;
  if (gmg_icm_build_indep(ctx, 0.5, stops, p->n_stop, &m)) return 1;
  if (gmg_icm_ready(m)) {
    gmg_icm_free(m);
    return 1;
  }
  const int N = m->N;
  // slot of every entry of the device view's prob table (cut nodes take their parent's row, see icm_upload)
  auto slot_of = [&](int e) -> uint8_t {
    const int f = e / (4 * N), node = (e / 4) % N;
    const int srcn = (m->mip[(size_t)f * N + node] < -1 && node > 0) ? (node - 1) / 4 : node;
    const int sl = indep_slot(f, srcn);
    return (uint8_t)(sl < 0 ? INDEP_SLOTS : sl + (e & 3));
  };
  std::vector<int> idx3(384), idxp(768);
  gmg_w3_lut_index(m->mip.data(), N, m->D, idx3.data(), idxp.data());
  std::vector<uint8_t> tab(GMG_INDEP_REC);
  for (int e = 0; e < 252; e++) tab[e] = slot_of(e);
  for (int i = 0; i < 384; i++) tab[252 + i] = slot_of(idx3[i]);
  for (int i = 0; i < 768; i++) tab[636 + i] = slot_of(idxp[i]);
  void* d = NULL;
  cudaError_t e = cudaMalloc(&d, GMG_INDEP_REC);
  if (e == cudaSuccess) e = cudaMemcpy(d, tab.data(), GMG_INDEP_REC, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    if (d) cudaFree(d);
    gmg_icm_free(m);
    gmg_set_error("gmg_indep_build: %s", cudaGetErrorString(e));
    return 1;
  }
  ctx->indep_tpl = m;
  ctx->d_indep_src = (uint8_t*)d;
  return 0;
}

int gmg_indep_build(gmg_ctx* ctx, const double* d_gc, const double* h_gc, int64_t n_models, const gmg_params* p,
                    float** d_rec, DevIcm* base) {
  GMG_CHECK(p->n_stop >= 0 && p->n_stop <= 8, "gmg_indep_build: %d stop codons", p->n_stop);
  if (indep_topology(ctx, p)) return 1;
  IndepStops st;
  memset(&st, 0, sizeof st);
  st.n = p->n_stop;
  for (int i = 0; i < p->n_stop; i++)
    st.j[i] = gmg_base_code(p->stop_codon[i][0]) + 4 * gmg_base_code(p->stop_codon[i][1]) +
              16 * gmg_base_code(p->stop_codon[i][2]);
  void *rec, *aux;
  if (gmg_scratch(ctx, SCR_INDEP, (size_t)(n_models > 0 ? n_models : 1) * GMG_INDEP_REC * sizeof(float), &rec)) return 1;
  if (gmg_scratch(ctx, SCR_INDEP_AUX, 16 + (size_t)(n_models > 0 ? n_models : 1) * sizeof(int32_t), &aux)) return 1;
  unsigned long long* counts = (unsigned long long*)aux;  // {flagged models, flagged entries}
  int32_t* flagged = (int32_t*)(counts + 2);
  GMG_CUDA(cudaMemsetAsync(counts, 0, 16, ctx->stream));
  const int force_host = getenv("GMG_INDEP_FORCE_HOST") && atoi(getenv("GMG_INDEP_FORCE_HOST")) > 0;
  if (n_models > 0) {
    k_indep_build<<<(unsigned)n_models, 128, 0, ctx->stream>>>(d_gc, st, ctx->d_indep_src, (float*)rec, flagged, counts,
                                                               force_host);
    ctx->launches++;
    GMG_CUDA(cudaGetLastError());
  }
  GMG_CUDA(cudaMemcpyAsync(&ctx->h_scalars[12], counts, 16, cudaMemcpyDeviceToHost, ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  const int64_t nf = ctx->h_scalars[12];
  ctx->indep_flagged = ctx->h_scalars[13];
  // the flagged models again on the host with glibc: one copy of the list back, one copy of the values over, one launch
  // (made also when nothing is flagged, so that a call's launch count does not depend on its values)
  std::vector<float> vals((size_t)nf * INDEP_PAD, 0.0f);
  void* fix;
  if (gmg_scratch(ctx, SCR_INDEP_FIX, (size_t)(nf > 0 ? nf : 1) * INDEP_PAD * sizeof(float), &fix)) return 1;
  if (nf > 0) {
    std::vector<int32_t> models((size_t)nf);
    GMG_CUDA(cudaMemcpyAsync(models.data(), flagged, (size_t)nf * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));
    const char* stops[8];
    for (int i = 0; i < p->n_stop; i++) stops[i] = p->stop_codon[i];
    int16_t mip[3 * 21];
    float prob[3 * 21 * 4];
    for (int64_t k = 0; k < nf; k++) {
      gmg_indep_tables(h_gc[models[k]], stops, p->n_stop, mip, prob);
      for (int f = 0; f < 3; f++)
        for (int node = 0; node < 21; node++) {
          const int sl = indep_slot(f, node);
          if (sl >= 0)
            for (int b = 0; b < 4; b++) vals[(size_t)k * INDEP_PAD + sl + b] = prob[(f * 21 + node) * 4 + b];
        }
    }
    GMG_CUDA(cudaMemcpyAsync(fix, vals.data(), vals.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  }
  k_indep_fix<<<(unsigned)(nf > 0 ? nf : 1), 128, 0, ctx->stream>>>(flagged, (const float*)fix, nf, ctx->d_indep_src,
                                                                  (float*)rec);
  ctx->launches++;
  GMG_CUDA(cudaGetLastError());
  if (nf > 0) GMG_CUDA(cudaStreamSynchronize(ctx->stream));  // `vals` is pageable host memory going out of scope
  *d_rec = (float*)rec;
  *base = ctx->indep_tpl->dev;
  return 0;
}

extern "C" int64_t gmg_ctx_indep_flagged(const gmg_ctx* ctx) { return ctx ? ctx->indep_flagged : 0; }
