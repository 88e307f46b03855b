// glimmer_mg_b200/host/icm.hh -- C++ host facade over the C-ABI (include/gmg_icm.h).
//
// Drop-in for the class interface of the reference's ICM library (/root/reference/src/ICM/icm.hh:116-213):
// the same class names (ICM_t, ICM_Training_t), method names, argument meaning and error behaviour (message on
// stderr, then exit(EXIT_FAILURE): icm.cc:635-657, 682-697, 2019-2024), so that a translation unit written against
// the reference's header compiles against this one and every model operation runs on the GPU.  Put this directory
// before the reference's src/ICM on the include path and link -lgmgicm instead of -lGLMicm (INTEGRATION.md).
//
// Nothing here computes: every method is a call into libgmgicm.so.  The scalar methods (Full_Window_Prob,
// Score_String, ...) are device round trips kept for parity and for rarely-called sites; drivers get their speed
// from the batched calls (gmg_score_orfs_g3 / gmg_score_orfs_mg), see host/g3_score_orfs_dropin.inc.
#ifndef GMG_HOST_ICM_HH
#define GMG_HOST_ICM_HH

#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include <string>
#include <vector>

#include "gmg_icm.h"

// constants callers of the reference header rely on (icm.hh:30-80)
const int DEFAULT_MODEL_LEN = 12;
const int DEFAULT_MODEL_DEPTH = 7;
const int DEFAULT_PERIODICITY = 3;
const int ICM_VERSION_ID = 200;
const int ID_STRING_LEN = 150;
const double MAX_LOG_DIFF = -46.0;  // icm.hh: used by glimmer3.cc Integerize_Scores

// One context per process: the reference's drivers are single-threaded (globals, static scratch buffers).
// GMG_DEVICE selects the GPU (default 0).  Created on first use so that file-scope ICM_t objects
// (glimmer3.cc:48,64) can be constructed before main() without touching the GPU.
inline gmg_ctx* Gmg_Context() {
  static gmg_ctx* ctx = NULL;
  if (ctx == NULL) {
    const char* dev = getenv("GMG_DEVICE");
    if (gmg_ctx_create(dev ? atoi(dev) : 0, NULL, &ctx) != 0) {
      fprintf(stderr, "ERROR:  %s\n", gmg_last_error());
      exit(EXIT_FAILURE);
    }
  }
  return ctx;
}

#define GMG_OR_DIE(call)                                  \
  do {                                                    \
    if ((call) != 0) {                                    \
      fprintf(stderr, "ERROR:  %s\n", gmg_last_error());  \
      exit(EXIT_FAILURE);                                 \
    }                                                     \
  } while (0)

class ICM_t {
 protected:
  gmg_icm* handle;  // owns host mirror + device tables (freed in the destructor, like score[] at icm.cc:48-61)
  int model_len, model_depth, periodicity;

  void Adopt(gmg_icm* h) {
    gmg_icm_free(handle);
    handle = h;
    int32_t d[4];
    GMG_OR_DIE(gmg_icm_dims(handle, d));
    model_len = d[0];
    model_depth = d[1];
    periodicity = d[2];
  }
  void Need_Model(const char* what) const {
    if (handle == NULL) {
      fprintf(stderr, "ERROR:  %s on an empty ICM\n", what);
      exit(EXIT_FAILURE);
    }
  }
  // one string as a 1-sequence batch
  gmg_seqset* One(const char* s, int64_t len) const {
    int64_t off[2] = {0, len};
    gmg_seqset* ss = NULL;
    GMG_OR_DIE(gmg_seqset_create(Gmg_Context(), s, off, 1, NULL, &ss));
    return ss;
  }

 public:
  ICM_t(int m = DEFAULT_MODEL_LEN, int d = DEFAULT_MODEL_DEPTH, int p = DEFAULT_PERIODICITY)
      : handle(NULL), model_len(m), model_depth(d), periodicity(p) {}
  ~ICM_t() { gmg_icm_free(handle); }
  ICM_t(const ICM_t&) = delete;  // the reference's Copy() is a shallow alias and unused (icm.cc:1000-1007)
  ICM_t& operator=(const ICM_t&) = delete;

  int Get_Model_Len(void) { return model_len; }
  int Get_Periodicity(void) { return periodicity; }
  gmg_icm* Handle(void) const { return handle; }  // for the batched calls

  void Read(char* path) {  // icm.cc:846-860
    gmg_icm* h = NULL;
    GMG_OR_DIE(gmg_icm_load(Gmg_Context(), path, &h));
    Adopt(h);
  }
  void Input(FILE* fp) {  // icm.cc:614-727: the model follows at the stream's current position
    // read exactly the model's bytes -- header, parameters, 22-byte node records up to the -1 terminator -- so that
    // the stream is left where the reference leaves it, and hand the image to the library
    std::vector<unsigned char> image(150 + 6 * sizeof(int32_t));
    if (fread(image.data(), 1, 150, fp) != 150) {
      fprintf(stderr, "ERROR reading ICM header\n");
      exit(EXIT_FAILURE);
    }
    if (fread(image.data() + 150, sizeof(int32_t), 6, fp) != 6) {
      fprintf(stderr, "ERROR reading parameters\n");
      exit(EXIT_FAILURE);
    }
    for (;;) {
      unsigned char rec[22];
      if (fread(rec, 1, 4, fp) != 4) break;
      image.insert(image.end(), rec, rec + 4);
      int32_t id;
      memcpy(&id, rec, 4);
      if (id < 0) break;
      const size_t got = fread(rec + 4, 1, 18, fp);
      image.insert(image.end(), rec + 4, rec + 4 + got);
      if (got != 18) break;  // the library reports the truncated node
    }
    gmg_icm* h = NULL;
    GMG_OR_DIE(gmg_icm_load_mem(Gmg_Context(), image.data(), image.size(), &h));
    Adopt(h);
  }
  void Build_Indep_WO_Stops(double gc_frac, const std::vector<const char*>& stop_codon) {  // icm.cc:65-216
    gmg_icm* h = NULL;
    GMG_OR_DIE(gmg_icm_build_indep(Gmg_Context(), gc_frac, stop_codon.data(), (int)stop_codon.size(), &h));
    Adopt(h);
  }
  void Output(FILE* fp, bool binary_form);  // icm.cc:729-803

  double Full_Window_Prob(const char* string, int frame) const {  // icm.cc:557
    Need_Model("Full_Window_Prob");
    double v;
    GMG_OR_DIE(gmg_icm_full_window_prob(Gmg_Context(), handle, string, frame, &v));
    return v;
  }
  double Partial_Window_Prob(int predict_pos, const char* string, int frame) const {  // icm.cc:807
    Need_Model("Partial_Window_Prob");
    double v;
    GMG_OR_DIE(gmg_icm_partial_window_prob(Gmg_Context(), handle, predict_pos, string, frame, &v));
    return v;
  }
  double Score_String(const char* string, int len, int frame) const {  // icm.cc:864
    Need_Model("Score_String");
    gmg_seqset* ss = One(string, len);
    double v = 0.0;
    GMG_OR_DIE(gmg_icm_score_strings(Gmg_Context(), handle, ss, frame, &v));
    gmg_seqset_free(ss);
    return v;
  }
  void Cumulative_Score(const std::string& s, std::vector<double>& score, int frame) const {  // icm.cc:354
    Need_Model("Cumulative_Score");
    score.resize(s.length());
    if (s.empty()) return;
    gmg_seqset* ss = One(s.data(), (int64_t)s.length());
    GMG_OR_DIE(gmg_icm_cumulative_score(Gmg_Context(), handle, ss, frame, score.data()));
    gmg_seqset_free(ss);
  }
  void Frame_Score(const std::string& s, std::vector<double>& score, int frame) const {  // icm.cc:485
    Need_Model("Frame_Score");
    score.resize(s.length());
    if (s.empty()) return;
    gmg_seqset* ss = One(s.data(), (int64_t)s.length());
    GMG_OR_DIE(gmg_icm_frame_score(Gmg_Context(), handle, ss, frame, score.data()));
    gmg_seqset_free(ss);
  }
};

// Output: the binary form is the build-icm model format, written by the library (byte-identical to the
// reference's, tests/test_gpu_parity.py); the text form ("for debugging only", build-icm -t) is formatted here
// from the model tables: "%6d  <context label> mut_info p(a) p(c) p(g) p(t)" for every node that is not pruned.
inline void ICM_t::Output(FILE* fp, bool binary_form) {
  Need_Model("Output");
  if (binary_form) {
    size_t nb = 0;
    GMG_OR_DIE(gmg_icm_write_mem(handle, NULL, 0, &nb));
    std::vector<char> image(nb);
    GMG_OR_DIE(gmg_icm_write_mem(handle, image.data(), nb, &nb));
    if (fwrite(image.data(), 1, nb, fp) != nb) {
      fprintf(stderr, "ERROR writing ICM\n");
      exit(EXIT_FAILURE);
    }
    return;
  }
  int32_t d[4];
  GMG_OR_DIE(gmg_icm_dims(handle, d));
  const int W = d[0], P = d[2], N = d[3];
  std::vector<int16_t> mip((size_t)P * N);
  std::vector<float> prob((size_t)P * N * 4);
  GMG_OR_DIE(gmg_icm_tables(handle, mip.data(), prob.data()));
  std::vector<float> info((size_t)P * N);
  GMG_OR_DIE(gmg_icm_mut_info(handle, info.data()));
  fprintf(fp, "ver = %.2f  len = %d  depth = %d  periodicity = %d  nodes = %d\n", ICM_VERSION_ID / 100.0, W, d[1], P, N);
  for (int f = 0; f < P; f++)
    for (int id = 0; id < N; id++) {
      const int16_t* m = &mip[(size_t)f * N];
      if (id > 0 && m[id] < -1) continue;
      // context label: '-' free position, '?' the predicted base, '*' this node's branch position, a/c/g/t the
      // bases fixed by the ancestors; '|' marks codon boundaries for periodic models (icm.cc:907-958)
      std::string label((size_t)W, '-');
      label[W - 1] = '?';
      if (m[id] >= 0) label[m[id]] = '*';
      for (int x = id; x > 0;) {
        const int parent = (x - 1) / 4;
        label[m[parent]] = "acgt"[x - 4 * parent - 1];
        x = parent;
      }
      std::string shown;
      int first_bar = (P == 1) ? -1 : (f == 0 ? W - P : W - f);
      for (int i = 0; i < W; i++) {
        if (P > 1 && i > 0 && first_bar > 0 && i <= first_bar && (first_bar - i) % P == 0) shown += '|';
        shown += label[i];
      }
      fprintf(fp, "%6d  %s", id, shown.c_str());
      fprintf(fp, " %7.4f", info[(size_t)f * N + id]);
      for (int k = 0; k < 4; k++) fprintf(fp, " %6.3f", exp((double)prob[((size_t)f * N + id) * 4 + k]));
      fputc('\n', fp);
    }
}

class ICM_Training_t : public ICM_t {
 public:
  ICM_Training_t(int m = DEFAULT_MODEL_LEN, int d = DEFAULT_MODEL_DEPTH, int p = DEFAULT_PERIODICITY) : ICM_t(m, d, p) {}

  // Train_Model (icm.cc:1356-1463): data = the training strings, already lower-cased and, for build-icm -r,
  // already reversed by the caller (build-icm.cc:111-118).
  void Train_Model(const std::vector<char*>& data) { Train_Strings(data, 0, NULL, NULL); }

  // the same with the options the device path adds: reverse on the device instead of on the host, and an
  // all-reduce callback summing each level's count slab across the GPUs of a box (include/gmg_icm.h)
  void Train_Strings(const std::vector<char*>& data, int reverse, gmg_allreduce_fn allreduce, void* user) {
    gmg_seqset* ss = Seqset_Of(data);
    gmg_icm* h = NULL;
    GMG_OR_DIE(gmg_icm_train(Gmg_Context(), ss, model_len, model_depth, periodicity, reverse, allreduce, user, &h));
    gmg_seqset_free(ss);
    Adopt(h);
  }

  // the training strings as a device seqset
  static gmg_seqset* Seqset_Of(const std::vector<char*>& data) {
    std::vector<int64_t> off(data.size() + 1, 0);
    for (size_t i = 0; i < data.size(); i++) off[i + 1] = off[i] + (int64_t)strlen(data[i]);
    char* cat = NULL;
    GMG_OR_DIE(gmg_host_alloc((size_t)off.back() + 1, (void**)&cat));  // page-locked: one H2D at PCIe rate
    for (size_t i = 0; i < data.size(); i++) memcpy(cat + off[i], data[i], (size_t)(off[i + 1] - off[i]));
    gmg_seqset* ss = NULL;
    GMG_OR_DIE(gmg_seqset_create(Gmg_Context(), cat, off.data(), (int64_t)data.size(), NULL, &ss));
    GMG_OR_DIE(gmg_ctx_sync(Gmg_Context()));  // the upload has read `cat`
    gmg_host_free(cat);
    return ss;
  }

  // Train_Model for many training sets in one device pass (gmg_icm_train_many): models[k] gets the model of sets[k];
  // every model takes this object's shape
  void Train_Many(const std::vector<gmg_seqset*>& sets, int reverse, const std::vector<ICM_Training_t*>& models) {
    std::vector<gmg_icm*> h(sets.size(), NULL);
    GMG_OR_DIE(gmg_icm_train_many(Gmg_Context(), sets.data(), (int)sets.size(), model_len, model_depth, periodicity, reverse,
                                  h.data()));
    for (size_t k = 0; k < sets.size(); k++) models[k]->Adopt(h[k]);
  }

  // Train straight from a multi-FASTA image (parsed, lower-cased and packed on the device -- no per-character
  // host loop): what build-icm does with its standard input.  Returns the number of training strings.
  int64_t Train_Fasta(const char* image, int64_t n_bytes, int reverse, gmg_allreduce_fn allreduce, void* user) {
    gmg_seqset* ss = NULL;
    int64_t n_records = 0;
    GMG_OR_DIE(gmg_seqset_from_fasta(Gmg_Context(), image, n_bytes, &ss, &n_records));
    if (n_records > 0) {
      gmg_icm* h = NULL;
      GMG_OR_DIE(gmg_icm_train(Gmg_Context(), ss, model_len, model_depth, periodicity, reverse, allreduce, user, &h));
      Adopt(h);
    }
    gmg_seqset_free(ss);
    return n_records;
  }
};

#endif  // GMG_HOST_ICM_HH
