// glimmer_mg_b200/csrc/gmg_model.cu -- context, error channel and the ICM_t container:
// build-icm binary format reader/writer, Build_Indep_WO_Stops, device upload.
//
// Reference behaviour mirrored (paths relative to /root/reference/src/):
//   ICM_t::ICM_t / Input / Output / Output_Node / Write_Header   ICM/icm.cc:24-45, 614-803, 961-998
//   ICM_t::Build_Indep_WO_Stops                                   ICM/icm.cc:65-216
//   Set_Ignore_Score_Len                                          Glimmer/glimmer_base.cc:2597-2633
#include <limits.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <float.h>
#include <math.h>

#include "gmg_internal.cuh"

static thread_local char g_err[1024] = "";

void gmg_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
}

extern "C" const char* gmg_last_error(void) { return g_err; }
extern "C" int gmg_abi_version(void) { return GMG_ABI_VERSION; }

extern "C" int gmg_ctx_create(int device, void* stream, gmg_ctx** out) {
  GMG_CHECK(out != NULL, "gmg_ctx_create: out is NULL");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    gmg_set_error("gmg_ctx_create: no usable CUDA device (%s); libgmgicm has no CPU fallback",
                  e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    return 1;
  }
  GMG_CHECK(device >= 0 && device < n, "gmg_ctx_create: device %d out of range (have %d)", device, n);
  GMG_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  GMG_CUDA(cudaGetDeviceProperties(&prop, device));
  GMG_CHECK(prop.major >= 10, "gmg_ctx_create: device %d is sm_%d%d; this library is built for sm_100a only",
            device, prop.major, prop.minor);
  gmg_ctx* c = new gmg_ctx();
  memset(c, 0, sizeof *c);
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  if (stream) {
    c->stream = (cudaStream_t)stream;
    c->own_stream = false;
  } else {
    GMG_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    c->own_stream = true;
  }
  // seqset / ORF / start buffers come from the device's stream-ordered pool; keep freed blocks cached
  // so that steady-state batches allocate without touching the driver
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    unsigned long long keep = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  GMG_CUDA(cudaMallocHost(&c->h_scalars, 16 * sizeof(int64_t)));
  GMG_CUDA(cudaEventCreateWithFlags(&c->ev_scalars, cudaEventDisableTiming));
  GMG_CUDA(cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking));
  GMG_CUDA(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
  GMG_CUDA(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
  *out = c;
  return 0;
}

extern "C" int gmg_host_alloc(size_t bytes, void** out) {
  GMG_CHECK(out, "gmg_host_alloc: out is NULL");
  GMG_CUDA(cudaMallocHost(out, bytes ? bytes : 1));
  return 0;
}

extern "C" void gmg_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

extern "C" void gmg_ctx_destroy(gmg_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  gmg_icm_free(c->indep_tpl);
  if (c->d_indep_src) cudaFree(c->d_indep_src);
  for (int i = 0; i < GMG_NSCRATCH; i++)
    if (c->scratch[i]) cudaFree(c->scratch[i]);
  if (c->h_penalty) cudaFreeHost(c->h_penalty);
  if (c->h_scalars) cudaFreeHost(c->h_scalars);
  if (c->h_stage) cudaFreeHost(c->h_stage);
  if (c->ev_scalars) cudaEventDestroy(c->ev_scalars);
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev_join) cudaEventDestroy(c->ev_join);
  if (c->side) cudaStreamDestroy(c->side);
  for (int k = 0; k < GMG_NPROF; k++)
    for (int i = 0; i < GMG_PROF_RING; i++)
      for (int e = 0; e < 2; e++)
        if (c->prof_ev[k][i][e]) cudaEventDestroy(c->prof_ev[k][i][e]);
  if (c->own_stream) cudaStreamDestroy(c->stream);
  delete c;
}

// ---- per-kernel device timing ---------------------------------------------------------------
static int prof_drain(gmg_ctx* c, int cls) {
  if (c->prof_n[cls] == 0) return 0;
  GMG_CUDA(cudaStreamSynchronize(c->stream));
  for (int i = 0; i < c->prof_n[cls]; i++) {
    float ms = 0.f;
    GMG_CUDA(cudaEventElapsedTime(&ms, c->prof_ev[cls][i][0], c->prof_ev[cls][i][1]));
    c->prof_ms[cls] += ms;
  }
  c->prof_n[cls] = 0;
  return 0;
}

int gmg_prof_begin(gmg_ctx* c, int cls) {
  if (!c->prof_on) return 0;
  if (c->prof_n[cls] == GMG_PROF_RING && prof_drain(c, cls)) return 1;
  cudaEvent_t* ev = c->prof_ev[cls][c->prof_n[cls]];
  if (!ev[0]) {
    GMG_CUDA(cudaEventCreate(&ev[0]));
    GMG_CUDA(cudaEventCreate(&ev[1]));
  }
  GMG_CUDA(cudaEventRecord(ev[0], c->stream));
  return 0;
}

void gmg_prof_end(gmg_ctx* c, int cls) {
  if (!c->prof_on) return;
  cudaEventRecord(c->prof_ev[cls][c->prof_n[cls]][1], c->stream);
  c->prof_n[cls]++;
  c->prof_launches[cls]++;
}

extern "C" int gmg_ctx_profile(gmg_ctx* c, int enable) {
  GMG_CHECK(c, "gmg_ctx_profile: NULL context");
  for (int k = 0; k < GMG_NPROF; k++)
    if (prof_drain(c, k)) return 1;
  c->prof_on = enable ? 1 : 0;
  return 0;
}

extern "C" int gmg_ctx_profile_read(gmg_ctx* c, int cls, double* ms, int64_t* launches) {
  GMG_CHECK(c && cls >= 0 && cls < GMG_NPROF, "gmg_ctx_profile_read: bad argument");
  if (prof_drain(c, cls)) return 1;
  if (ms) *ms = c->prof_ms[cls];
  if (launches) *launches = c->prof_launches[cls];
  c->prof_ms[cls] = 0.0;
  c->prof_launches[cls] = 0;
  return 0;
}

extern "C" int gmg_ctx_sync(gmg_ctx* c) {
  GMG_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

extern "C" int64_t gmg_ctx_launch_count(const gmg_ctx* c) { return c->launches; }

extern "C" int gmg_ctx_memcpy_d2h(gmg_ctx* c, void* h_dst, const void* d_src, size_t bytes) {
  GMG_CUDA(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, c->stream));
  GMG_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

extern "C" int gmg_ctx_memcpy_h2d(gmg_ctx* c, void* d_dst, const void* h_src, size_t bytes) {
  GMG_CUDA(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, c->stream));
  GMG_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

int gmg_scratch(gmg_ctx* ctx, int slot, size_t bytes, void** out) {
  if (bytes == 0) bytes = 256;
  if (ctx->scratch_bytes[slot] < bytes) {
    if (ctx->scratch[slot]) {
      GMG_CUDA(cudaStreamSynchronize(ctx->stream));
      GMG_CUDA(cudaFree(ctx->scratch[slot]));
      ctx->scratch[slot] = NULL;
      ctx->scratch_bytes[slot] = 0;
    }
    size_t want = bytes + bytes / 8 + 4096;
    GMG_CUDA(cudaMalloc(&ctx->scratch[slot], want));
    ctx->scratch_bytes[slot] = want;
  }
  *out = ctx->scratch[slot];
  return 0;
}

extern "C" void gmg_params_default(gmg_params* p, int metagenomic) {
  memset(p, 0, sizeof *p);
  p->min_gene_len = 75;
  p->allow_truncated = metagenomic ? 1 : 0;
  p->min_indel_orf_len = 15;
  p->indel_quality_threshold = 18;
  p->indel_max = 2;
  p->ignore_score_len = INT_MAX;
  p->indel_suffix_score_threshold = -12.0;
  p->n_start = 3;
  strcpy(p->start_codon[0], "atg");
  strcpy(p->start_codon[1], "gtg");
  strcpy(p->start_codon[2], "ttg");
  p->n_stop = 3;
  strcpy(p->stop_codon[0], "taa");
  strcpy(p->stop_codon[1], "tag");
  strcpy(p->stop_codon[2], "tga");
}

extern "C" int gmg_ignore_score_len(double gc, const gmg_params* p) {
  double lambda = 0.0;
  for (int i = 0; i < p->n_stop; i++) {
    double x = 1.0;
    for (int j = 0; j < 3; j++) {
      char ch = p->stop_codon[i][j];
      x *= (ch == 'c' || ch == 'g') ? gc / 2.0 : (1.0 - gc) / 2.0;
    }
    lambda += x;
  }
  if (lambda == 0.0) return INT_MAX;
  return (int)(long)floor(3.0 * log(2.0 * 1000000 * lambda) / lambda);
}

// ------------------------------------------------------------------------------------------

int gmg_base_code(char ch) {
  // Subscript(Filter(ch)) (icm.cc:2008-2027, gene.cc:1139-1175)
  switch (ch | 0x20) {
    case 'a': return 0;
    case 'c': return 1;
    case 'g': return 2;
    case 't': return 3;
    case 'r': return 2;
    case 'y': return 1;
    case 's': return 1;
    case 'w': return 3;
    case 'm': return 1;
    case 'k': return 3;
    case 'b': return 1;
    case 'd': return 2;
    case 'h': return 1;
    case 'v': return 1;
    default: return 1;
  }
}

void gmg_icm_value_stats(const gmg_icm* m, int* ulp_exp, float* max_abs) {
  if (gmg_icm_ready(m)) {  // cannot upload: nothing can be certified
    *ulp_exp = -100000;
    *max_abs = 0.f;
    return;
  }
  *ulp_exp = m->stat_ulp_exp;
  *max_abs = m->stat_max_abs;
}

static int num_nodes_for(int d) {
  long n = 1, pw = 1;
  for (int i = 0; i < d; i++) {
    pw *= 4;
    n += pw;
  }
  return (int)n;
}

// Entries of the device view's prob table (cut nodes resolved to their parent's row) that the W == 3 lookup tables
// take.  lut3: full-window value of every base triple, [strand][period][raw]; lutp: the same for the partial windows at
// a sequence's ends
// (Partial_Window_Prob, icm.cc:807-842), [strand][lim - 1][period][raw] -- window positions below lim are not available,
// the walk stops at the first node that asks for one, so the entry does not depend on the raw code's bits at those
// positions and the caller may index with whatever bases lie there.
void gmg_w3_lut_index(const int16_t* mip, int N, int D, int* idx3, int* idxp) {
  for (int i = 0; i < 384 + 768; i++) {
    const bool full = i < 384;
    const int k = full ? i : i - 384;
    const int raw = k & 63, f = (k >> 6) % 3, lim = full ? 0 : 1 + (k / 192) % 2, strand = full ? k / 192 : k / 384;
    // forward strand: window position k <-> base q0 + 2 - k; reverse strand: complement of base q0 + k
    const unsigned ctx = strand == 0 ? (unsigned)(((raw >> 4) & 3) | (((raw >> 2) & 3) << 2) | ((raw & 3) << 4))
                                     : (unsigned)((~raw) & 63);
    int node = 0;
    for (int l = 0; l < D; l++) {
      const int pos = mip[(size_t)f * N + node];
      if (pos < lim) break;
      node = 4 * node + (int)((ctx >> (2 * pos)) & 3) + 1;
    }
    (full ? idx3[k] : idxp[k]) = (f * N + node) * 4 + (int)((ctx >> 4) & 3);
  }
}

static int icm_upload(gmg_icm* m) {
  gmg_ctx* ctx = m->ctx;
  GMG_CUDA(cudaSetDevice(ctx->device));
  const int P = m->P, N = m->N, D = m->D;
  const int inner = (D == 0) ? 1 : num_nodes_for(D - 1);  // nodes on levels 0..D-1
  std::vector<int8_t> mip8((size_t)P * inner);
  std::vector<float> eff((size_t)P * N * 4);
  for (int f = 0; f < P; f++) {
    for (int i = 0; i < inner; i++) {
      int v = m->mip[(size_t)f * N + i];
      mip8[(size_t)f * inner + i] = (int8_t)(v < -2 ? -2 : v);
    }
    for (int i = 0; i < N; i++) {
      // cut node -> parent's probabilities (the reference steps back one level only)
      int src = (m->mip[(size_t)f * N + i] < -1 && i > 0) ? (i - 1) / 4 : i;
      memcpy(&eff[((size_t)f * N + i) * 4], &m->prob[((size_t)f * N + src) * 4], 4 * sizeof(float));
    }
  }
  // model tables come from the device's stream-ordered pool (cached blocks: no driver call per model)
  GMG_CUDA(cudaMallocAsync(&m->d_mip, mip8.size() + 16, ctx->stream));
  GMG_CUDA(cudaMallocAsync(&m->d_prob, eff.size() * sizeof(float) + 16, ctx->stream));
  GMG_CUDA(cudaMemcpyAsync(m->d_mip, mip8.data(), mip8.size(), cudaMemcpyHostToDevice, ctx->stream));
  GMG_CUDA(cudaMemcpyAsync(m->d_prob, eff.data(), eff.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  GMG_CUDA(cudaStreamSynchronize(ctx->stream));
  // value statistics for the static exactness certificates
  {
    int ue = 1024;
    float mx = 0.f;
    for (float v : m->prob) {
      if (v == 0.f) continue;
      if (!(fabsf(v) <= FLT_MAX)) {  // inf / nan: nothing can be certified
        ue = -100000;
        continue;
      }
      int e;
      frexpf(v, &e);  // |v| in [2^(e-1), 2^e)
      e = (e - 1 < -126 ? -126 : e - 1) - 23;
      if (e < ue) ue = e;
      if (fabsf(v) > mx) mx = fabsf(v);
    }
    m->stat_valid = 1;
    m->stat_ulp_exp = ue;
    m->stat_max_abs = mx;
  }
  // tables of the bucketed K1 kernel (the build-icm defaults: window <= 16, depth 7, period 3)
  m->fast.valid = 0;
  if (m->W <= 16 && D == 7 && P == 3) {
    // Completed tree: a walk that stops at node n (leaf, cut node, or depth reached) is continued through
    // VIRTUAL descendants that all carry n's value, so the full-window fast path needs no stop test and always
    // reads a level-D entry.  stop[n] = "a real walk stops here or has stopped above".
    const size_t np = ((size_t)N + 3) & ~(size_t)3;  // row stride: 16-byte aligned rows
    const int NW = 4 + 64 + 1024;                    // merged words: nodes of levels 1, 3, 5
    std::vector<float> bleaf((size_t)P * 4 * np, 0.0f);
    std::vector<uint32_t> mw((size_t)P * NW, 0u);
    const int inner = num_nodes_for(D - 1);
    for (int f = 0; f < P; f++) {
      std::vector<int> src(N);
      std::vector<uint8_t> stop(N), sh(N, 0);
      for (int n = 0; n < N; n++) {
        const int par = n ? (n - 1) / 4 : -1;
        const bool virt = n && stop[par];
        src[n] = virt ? src[par] : n;
        const int v = n < inner ? (int)m->mip[(size_t)f * N + n] : -1;
        stop[n] = virt || v < 0;
        sh[n] = (uint8_t)(stop[n] ? 0 : 30 - 2 * v);
        for (int b = 0; b < 4; b++) bleaf[((size_t)f * 4 + b) * np + n] = eff[((size_t)f * N + src[n]) * 4 + b];
      }
      m->fast.s0[f] = sh[0];
      m->fast.stop0[f] = stop[0];
      int wbase = 0;
      for (int l = 1; l <= 5; l += 2) {
        const int first = num_nodes_for(l - 1), width = 1 << (2 * l);  // dense index of the level's first node
        for (int i = 0; i < width; i++) {
          const int n = first + i;
          uint32_t w = sh[n] | ((uint32_t)stop[n] << 25);
          for (int k = 0; k < 4; k++) {
            const int c = 4 * n + 1 + k;
            w |= (uint32_t)sh[c] << (5 + 5 * k);
            w |= (uint32_t)stop[c] << (26 + k);
          }
          mw[(size_t)f * NW + wbase + i] = w;
        }
        wbase += width;
      }
    }
    GMG_CUDA(cudaMallocAsync(&m->d_msh, mw.size() * sizeof(uint32_t) + 64, ctx->stream));
    GMG_CUDA(cudaMemcpyAsync(m->d_msh, mw.data(), mw.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    GMG_CUDA(cudaMallocAsync(&m->d_bleaf, bleaf.size() * sizeof(float) + 64, ctx->stream));
    GMG_CUDA(cudaMemcpyAsync(m->d_bleaf, bleaf.data(), bleaf.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));
    m->fast.N = N;
    m->fast.np = (int)np;
    m->fast.bleaf = m->d_bleaf;
    m->fast.mw = reinterpret_cast<const uint32_t*>(m->d_msh);
    m->fast.valid = 1;
    m->fast.W = m->W;
    m->fast.D = D;
    m->fast.P = P;
  }
  // full-window lookup table of W == 3 models (Build_Indep_WO_Stops makes an ICM_t(3,2,3))
  m->dev.lut3 = NULL;
  m->dev.lutp = NULL;
  if (m->W == 3 && P == 3) {
    std::vector<int> idx3(384), idxp(768);
    gmg_w3_lut_index(m->mip.data(), N, D, idx3.data(), idxp.data());
    std::vector<float> lut(384), lutp(768);
    for (int i = 0; i < 384; i++) lut[i] = eff[idx3[i]];
    for (int i = 0; i < 768; i++) lutp[i] = eff[idxp[i]];
    GMG_CUDA(cudaMallocAsync(&m->d_lut3, 384 * sizeof(float), ctx->stream));
    GMG_CUDA(cudaMemcpyAsync(m->d_lut3, lut.data(), 384 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    GMG_CUDA(cudaMallocAsync(&m->d_lutp, 768 * sizeof(float), ctx->stream));
    GMG_CUDA(cudaMemcpyAsync(m->d_lutp, lutp.data(), 768 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    GMG_CUDA(cudaStreamSynchronize(ctx->stream));
    m->dev.lut3 = m->d_lut3;
    m->dev.lutp = m->d_lutp;
  }
  m->dev.W = m->W;
  m->dev.D = D;
  m->dev.P = P;
  m->dev.N = N;
  m->dev.inner = inner;
  m->dev.mip = m->d_mip;
  m->dev.prob = m->d_prob;
  return 0;
}

static int icm_validate(int w, int d, int p, int n) {
  GMG_CHECK(w >= 1 && w <= GMG_MAX_W, "ICM model_len %d unsupported (1..%d)", w, GMG_MAX_W);
  GMG_CHECK(d >= 0 && d <= GMG_MAX_DEPTH && d < w + 1, "ICM model_depth %d unsupported (0..%d)", d, GMG_MAX_DEPTH);
  GMG_CHECK(p >= 1 && p <= 16, "ICM periodicity %d unsupported", p);
  GMG_CHECK(n == num_nodes_for(d), "ICM num_nodes %d does not match depth %d", n, d);
  return 0;
}

extern "C" int gmg_icm_from_tables(gmg_ctx* ctx, int w, int d, int p, const int16_t* h_mip, const float* h_prob,
                                   gmg_icm** out) {
  GMG_CHECK(ctx && out && h_mip && h_prob, "gmg_icm_from_tables: NULL argument");
  int n = num_nodes_for(d);
  if (icm_validate(w, d, p, n)) return 1;
  gmg_icm* m = new gmg_icm();
  m->ctx = ctx;
  m->W = w; m->D = d; m->P = p; m->N = n;
  m->mip.assign(h_mip, h_mip + (size_t)p * n);
  m->prob.assign(h_prob, h_prob + (size_t)p * n * 4);
  m->mut_info.assign((size_t)p * n, 0.0f);
  m->d_mip = NULL;
  m->d_prob = NULL;
  m->d_msh = NULL;
  m->d_bleaf = NULL;
  m->d_lut3 = NULL;
  m->d_lutp = NULL;
  for (size_t i = 0; i < m->mip.size(); i++)
    if (m->mip[i] >= w - 1 && w > 1) {
      gmg_set_error("ICM node %zu has mut_info_pos %d outside the context window (len %d)", i, m->mip[i], w);
      delete m;
      return 1;
    }
  // the device views (walk tables, completed tree, merged words, leaf tables by predicted base) are built when a
  // scoring call first needs them (gmg_icm_ready): a model that is only trained and written never pays for them
  m->ready = 0;
  *out = m;
  return 0;
}

int gmg_icm_ready(const gmg_icm* cm) {
  gmg_icm* m = const_cast<gmg_icm*>(cm);
  if (m->ready) return 0;
  if (icm_upload(m)) return 1;
  m->ready = 1;
  return 0;
}

// ICM_t::Input (icm.cc:614-726) over a memory image of the build-icm binary format
extern "C" int gmg_icm_load_mem(gmg_ctx* ctx, const void* image, size_t n_bytes, gmg_icm** out) {
  GMG_CHECK(ctx && out && (image || n_bytes == 0), "gmg_icm_load_mem: NULL argument");
  const unsigned char* cur = (const unsigned char*)image;
  const unsigned char* const end = cur + n_bytes;
  auto take = [&](void* dst, size_t nb) -> bool {
    if ((size_t)(end - cur) < nb) return false;
    memcpy(dst, cur, nb);
    cur += nb;
    return true;
  };
  char line[150];
  int32_t param[6];
  GMG_CHECK(take(line, 150), "ERROR reading ICM header");
  GMG_CHECK(take(param, sizeof param), "ERROR reading parameters");
  GMG_CHECK(param[0] == 200, "Bad ICM version = %d  should be %d", param[0], 200);
  GMG_CHECK(param[1] == 150, "Bad ID_STRING_LEN = %d  should be %d", param[1], 150);
  const int w = param[2], d = param[3], p = param[4], n = param[5];
  if (icm_validate(w, d, p, n)) return 1;
  std::vector<int16_t> mip((size_t)p * n, 0);
  std::vector<float> prob((size_t)p * n * 4, 0.0f);
  int period = -1, prev = 0;
  int32_t id;
  while (take(&id, sizeof id)) {
    if (id < 0) break;
    if (id == 0) period++;
    GMG_CHECK(!(period < 0 || period >= p || id >= n), "ERROR reading icm node = %d  period = %d", id, period);
    size_t at = (size_t)period * n + id;
    GMG_CHECK(take(&prob[at * 4], 4 * sizeof(float)), "ERROR reading icm node = %d  period = %d", id, period);
    GMG_CHECK(take(&mip[at], sizeof(int16_t)), "ERROR reading mut_info_pos for node = %d  period = %d", id, period);
    if (id != 0 && prev != id - 1)
      for (int i = prev + 1; i < id; i++) mip[(size_t)period * n + i] = -2;
    if (id == 0 && period > 0)
      for (int i = prev + 1; i < n; i++) mip[(size_t)(period - 1) * n + i] = -2;
    prev = id;
  }
  GMG_CHECK(period == p - 1, "ERROR:  Too few nodes for periodicity = %d", p);
  for (int i = prev + 1; i < n; i++) mip[(size_t)period * n + i] = -2;
  return gmg_icm_from_tables(ctx, w, d, p, mip.data(), prob.data(), out);
}

extern "C" int gmg_icm_load(gmg_ctx* ctx, const char* path, gmg_icm** out) {
  GMG_CHECK(ctx && path && out, "gmg_icm_load: NULL argument");
  FILE* fp = fopen(path, "rb");
  GMG_CHECK(fp != NULL, "ERROR:  Could not open file  %s", path);
  std::vector<unsigned char> image;
  unsigned char buf[1 << 16];
  size_t got;
  while ((got = fread(buf, 1, sizeof buf, fp)) > 0) image.insert(image.end(), buf, buf + got);
  fclose(fp);
  return gmg_icm_load_mem(ctx, image.data(), image.size(), out);
}

// ICM_t::Output(fp, binary = true) (icm.cc:729-803, 961-998) into memory: *n_bytes receives the image size; the image
// is copied to h_out when it fits in `cap` (call with h_out = NULL to size the buffer)
extern "C" int gmg_icm_write_mem(const gmg_icm* m, void* h_out, size_t cap, size_t* n_bytes) {
  GMG_CHECK(m && n_bytes, "gmg_icm_write_mem: NULL argument");
  std::string img;
  img.reserve(174 + (size_t)m->P * m->N * 22 + 4);
  char line[150];
  memset(line, 0, sizeof line);
  snprintf(line, sizeof line, ">ver = %.2f  len = %d  depth = %d  periodicity = %d  nodes = %d\n", 2.00, m->W, m->D,
           m->P, m->N);
  int32_t param[6] = {200, 150, m->W, m->D, m->P, m->N};
  img.append(line, 150);
  img.append((const char*)param, sizeof param);
  for (int f = 0; f < m->P; f++)
    for (int32_t i = 0; i < m->N; i++) {
      size_t at = (size_t)f * m->N + i;
      if (i != 0 && m->mip[at] < -1) continue;  // cut nodes are not stored
      img.append((const char*)&i, sizeof i);
      img.append((const char*)&m->prob[at * 4], 4 * sizeof(float));
      img.append((const char*)&m->mip[at], sizeof(int16_t));
    }
  int32_t end_marker = -1;
  img.append((const char*)&end_marker, sizeof end_marker);
  *n_bytes = img.size();
  if (h_out) {
    GMG_CHECK(cap >= img.size(), "gmg_icm_write_mem: buffer of %zu bytes, image needs %zu", cap, img.size());
    memcpy(h_out, img.data(), img.size());
  }
  return 0;
}

extern "C" int gmg_icm_write(const gmg_icm* m, const char* path) {
  GMG_CHECK(m && path, "gmg_icm_write: NULL argument");
  size_t nb = 0;
  if (gmg_icm_write_mem(m, NULL, 0, &nb)) return 1;
  std::vector<char> img(nb);
  if (gmg_icm_write_mem(m, img.data(), nb, &nb)) return 1;
  FILE* fp = fopen(path, "wb");
  GMG_CHECK(fp != NULL, "ERROR:  Could not open file  %s", path);
  bool ok = fwrite(img.data(), 1, nb, fp) == nb;
  ok = (fclose(fp) == 0) && ok;
  GMG_CHECK(ok, "ERROR writing ICM file %s", path);
  return 0;
}

extern "C" int gmg_icm_dims(const gmg_icm* m, int32_t dims[4]) {
  GMG_CHECK(m && dims, "gmg_icm_dims: NULL argument");
  dims[0] = m->W; dims[1] = m->D; dims[2] = m->P; dims[3] = m->N;
  return 0;
}

extern "C" int gmg_icm_tables(const gmg_icm* m, int16_t* h_mip, float* h_prob) {
  GMG_CHECK(m, "gmg_icm_tables: NULL model");
  if (h_mip) memcpy(h_mip, m->mip.data(), m->mip.size() * sizeof(int16_t));
  if (h_prob) memcpy(h_prob, m->prob.data(), m->prob.size() * sizeof(float));
  return 0;
}

extern "C" int gmg_icm_mut_info(const gmg_icm* m, float* h_out) {
  GMG_CHECK(m && h_out, "gmg_icm_mut_info: NULL argument");
  memcpy(h_out, m->mut_info.data(), m->mut_info.size() * sizeof(float));
  return 0;
}

extern "C" void gmg_icm_free(gmg_icm* m) {
  if (!m) return;
  cudaSetDevice(m->ctx->device);
  void* ptrs[] = {m->d_mip, m->d_prob, m->d_msh, m->d_bleaf, m->d_lut3, m->d_lutp};
  for (void* q : ptrs)
    if (q) cudaFreeAsync(q, m->ctx->stream);  // ordered after every kernel of this context that reads the tables
  delete m;
}

// Independent-nucleotide codon model without stop codons, stored as a period-3 depth-2
// ICM in the reversed orientation the gene models use (icm.cc:65-216).  The table is tiny
// (63 nodes) and is built once per run on the host in FP64 exactly like the reference
// (its float accumulators round at every += ; glibc log), then uploaded.
void gmg_indep_tables(double gc, const char* const* stops, int n_stops, int16_t* mip, float* prob) {
  double base_prob[4], codon_prob[64];
  base_prob[1] = base_prob[2] = gc / 2.0;
  base_prob[0] = base_prob[3] = 0.5 - base_prob[1];
  for (int c = 0; c < 64; c++) codon_prob[c] = base_prob[(c >> 4) & 3] * base_prob[(c >> 2) & 3] * base_prob[c & 3];
  for (int i = 0; i < n_stops; i++) {
    // the model runs 3'->5', so the stop codon enters reversed
    int j = gmg_base_code(stops[i][0]) + 4 * gmg_base_code(stops[i][1]) + 16 * gmg_base_code(stops[i][2]);
    codon_prob[j] = 1e-20;
  }
  double sum = 0.0;
  for (int c = 0; c < 64; c++) sum += codon_prob[c];
  for (int c = 0; c < 64; c++) codon_prob[c] /= sum;

  const int N = 21;
  std::vector<float> acc(3 * N * 4, 0.0f);
  static const int pw[3] = {1, 4, 16};
  for (int i = 0; i < 3 * N; i++) mip[i] = 0;
  for (int f = 0; f < 3; f++) {
    const int d1 = pw[(3 - f) % 3], d2 = pw[(4 - f) % 3], d3 = pw[(5 - f) % 3];
    mip[f * N] = (f == 1) ? -1 : 1;
    for (int c = 0; c < 64; c++) acc[(f * N) * 4 + (c / d1) % 4] += codon_prob[c];
    for (int b = 0; b < 4; b++) mip[f * N + 1 + b] = (f == 2) ? -1 : 0;
    if (f != 1)
      for (int c = 0; c < 64; c++) acc[(f * N + 1 + (c / d2) % 4) * 4 + (c / d1) % 4] += codon_prob[c];
    if (f == 0) {
      for (int b = 0; b < 16; b++) mip[f * N + 5 + b] = -1;
      for (int c = 0; c < 64; c++) acc[(f * N + 5 + 4 * ((c / d2) % 4) + (c / d3) % 4) * 4 + (c / d1) % 4] += codon_prob[c];
    }
  }
  for (int i = 0; i < 3 * N; i++) {
    double s = 0.0;
    for (int k = 0; k < 4; k++) s += acc[i * 4 + k];
    for (int k = 0; k < 4; k++) prob[i * 4 + k] = (float)(s == 0.0 ? 0.0 : log(acc[i * 4 + k] / s));
  }
}

extern "C" int gmg_icm_build_indep(gmg_ctx* ctx, double gc, const char* const* stops, int n_stops, gmg_icm** out) {
  GMG_CHECK(ctx && out, "gmg_icm_build_indep: NULL argument");
  int16_t mip[3 * 21];
  float prob[3 * 21 * 4];
  gmg_indep_tables(gc, stops, n_stops, mip, prob);
  return gmg_icm_from_tables(ctx, 3, 2, 3, mip, prob, out);
}
