// tests/mgflat_host_check.cu -- TEST INFRASTRUCTURE.  Runs the passes of the flat glimmer-mg start enumeration
// (glimmer_mg_b200/csrc/gmg_mg_flat.cuh, the __host__ __device__ bodies of the K3 kernels) ON THE HOST against the
// oracle port (oracle/icm_oracle.c): per read the inputs K2 would produce are rebuilt from oracle outputs
// (Frame_Scores -> prefix sums, Save_Prev_Stops, Set_Quality_454, codon bitmaps, gate lists), the passes are run as
// plain loops with std exclusive scans, and the start lists must equal orc_mg_score_orfs byte for byte.
// This is a debugging aid for kernel logic in a container without a GPU; the product never runs this way.
//
// With a quality seed the reads carry seeded Phred values as from a quality file (have_quality_file = 1): the oracle
// gets them as they are, the quality plane is built by glimmer-mg's rule (Clean_Quality_454 under -i only) and the
// Pass_Stop_Penalty of every root call is filled in as k_mg_sub_pstop + the host log fill it.
//
//   mgflat_check <model.icm> <reads.fa> <n_reads> <allow_indels> <allow_subs> <indel_max> [truncate_len [qual_seed]]
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <numeric>
#include <string>
#include <vector>

extern "C" {
#include "../oracle/icm_oracle.h"
}
#include "../glimmer_mg_b200/csrc/gmg_mg_flat.cuh"

static int code_of(char ch) {
  switch (ch | 0x20) {
    case 'a': return 0;
    case 'c': return 1;
    case 'g': return 2;
    case 't': return 3;
  }
  return 1;
}

static void make_sets(const orc_params& p, CodonSets* cs) {
  memset(cs, 0, sizeof *cs);
  memset(cs->which, 0xFF, sizeof cs->which);
  for (int i = 0; i < p.n_start; i++) {
    int code = code_of(p.start_codon[i][0]) * 16 + code_of(p.start_codon[i][1]) * 4 + code_of(p.start_codon[i][2]);
    if (!(cs->start_mask >> code & 1)) cs->which[code] = (unsigned char)i;
    cs->start_mask |= 1ull << code;
  }
  for (int i = 0; i < p.n_stop; i++)
    cs->stop_mask |= 1ull << (code_of(p.stop_codon[i][0]) * 16 + code_of(p.stop_codon[i][1]) * 4 + code_of(p.stop_codon[i][2]));
  for (int raw = 0; raw < 64; raw++) {
    const int b0 = raw & 3, b1 = (raw >> 2) & 3, b2 = raw >> 4;
    const int fc = b0 * 16 + b1 * 4 + b2, rc = (3 - b2) * 16 + (3 - b1) * 4 + (3 - b0);
    if (cs->start_mask >> fc & 1) cs->raw_mask[0] |= 1ull << raw;
    if (cs->stop_mask >> fc & 1) cs->raw_mask[1] |= 1ull << raw;
    if (cs->start_mask >> rc & 1) cs->raw_mask[2] |= 1ull << raw;
    if (cs->stop_mask >> rc & 1) cs->raw_mask[3] |= 1ull << raw;
  }
}

// seeded Phred values: half of them from the edges of the quality tables (0, the indel threshold 18 and its
// neighbours, 1 - 10^(-q/10) rounding to 1 from 163 on, 255), the rest uniform in 0..40 (splitmix64)
static std::vector<int> seeded_quality(uint64_t& st, int L) {
  static const int edge[12] = {0, 1, 2, 17, 18, 19, 20, 40, 93, 162, 163, 255};
  std::vector<int> q((size_t)L);
  for (int i = 0; i < L; i++) {
    uint64_t z = (st += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    q[i] = (z & 1) ? edge[(z >> 8) % 12] : (int)((z >> 8) % 41);
  }
  return q;
}

static std::vector<std::string> read_fasta(const char* path, int n_max) {
  std::vector<std::string> out;
  FILE* fp = fopen(path, "r");
  if (!fp) { perror(path); exit(2); }
  char line[1 << 16];
  while (fgets(line, sizeof line, fp)) {
    if (line[0] == '>') {
      if ((int)out.size() == n_max) break;
      out.push_back("");
    } else if (!out.empty()) {
      for (char* c = line; *c; c++)
        if (*c > ' ') out.back().push_back("acgt"[code_of(*c) & 3]);
    }
  }
  fclose(fp);
  return out;
}

template <class T>
static void exscan(std::vector<T>& in, std::vector<T>& out) {
  out.resize(in.size());
  T acc = 0;
  for (size_t i = 0; i < in.size(); i++) {
    out[i] = acc;
    acc += in[i];
  }
}

int main(int argc, char** argv) {
  if (argc < 7) {
    fprintf(stderr, "usage: %s model.icm reads.fa n_reads allow_indels allow_subs indel_max [truncate_len]\n", argv[0]);
    return 2;
  }
  orc_icm* gene = orc_icm_read(argv[1]);
  const int trunc_len = argc > 7 ? atoi(argv[7]) : 0;
  const bool have_qual = argc > 8;
  uint64_t qual_state = have_qual ? strtoull(argv[8], NULL, 10) : 0;
  std::vector<std::string> reads = read_fasta(argv[2], atoi(argv[3]));
  if (trunc_len > 0)
    for (auto& r : reads)
      if ((int)r.size() > trunc_len) r.resize(trunc_len);
  orc_params op;
  orc_default_params(&op, 1);
  op.allow_indels = atoi(argv[4]);
  op.allow_subs = atoi(argv[5]);
  op.indel_max = atoi(argv[6]);
  // batch layout
  const int64_t n = (int64_t)reads.size();
  std::vector<int64_t> off(n + 1, 0);
  for (int64_t i = 0; i < n; i++) off[i + 1] = off[i] + (int64_t)reads[i].size();
  const int64_t total = off[n];
  long gcn = 0;
  for (auto& r : reads)
    for (char c : r) gcn += (c == 'c' || c == 'g');
  const double gc = (double)gcn / (double)total;
  const char* stops[3] = {"taa", "tag", "tga"};
  orc_icm* indep = orc_build_indep_wo_stops(gc, stops, 3);
  op.ignore_score_len = orc_ignore_score_len(gc, &op);

  const int PADW = 8;
  std::vector<uint64_t> words_base(total / 32 + 2 + 2 * PADW, 0);
  uint64_t* words = words_base.data() + PADW;
  for (int64_t i = 0; i < n; i++)
    for (size_t q = 0; q < reads[i].size(); q++) {
      const int64_t p = off[i] + (int64_t)q;
      words[p >> 5] |= (uint64_t)code_of(reads[i][q]) << ((p & 31) * 2);
    }
  CodonSets cs;
  make_sets(op, &cs);
  DevParams P;
  P.min_gene_len = op.min_gene_len;
  P.allow_truncated = op.allow_truncated;
  P.allow_indels = op.allow_indels;
  P.allow_subs = op.allow_subs;
  P.min_indel_orf_len = op.min_indel_orf_len;
  P.indel_q_thresh = op.indel_quality_threshold;
  P.indel_max = op.indel_max;
  P.ignore_score_len = op.ignore_score_len;
  P.have_quality_file = have_qual ? 1 : 0;
  op.have_quality_file = P.have_quality_file;
  P.indel_suffix_thresh = op.indel_suffix_score_threshold;

  // codon bitmaps
  const int64_t nwc = total / 96 + 2;
  std::vector<uint2> cb((size_t)6 * nwc, uint2{0, 0});
  for (int r = 0; r < 3; r++)
    for (int64_t sl = 0; 3 * sl + r + 2 < total + 96; sl++) {
      const int64_t g = 3 * sl + r;
      if ((sl >> 5) >= nwc) break;
      int raw = 0;
      for (int t = 0; t < 3; t++) raw |= mgf_base_at(words, g + t) << (2 * t);
      uint2& f = cb[(size_t)r * nwc + (sl >> 5)];
      uint2& v = cb[(size_t)(3 + r) * nwc + (sl >> 5)];
      f.x |= (unsigned)((cs.raw_mask[0] >> raw) & 1) << (sl & 31);
      f.y |= (unsigned)((cs.raw_mask[1] >> raw) & 1) << (sl & 31);
      v.x |= (unsigned)((cs.raw_mask[2] >> raw) & 1) << (sl & 31);
      v.y |= (unsigned)((cs.raw_mask[3] >> raw) & 1) << (sl & 31);
    }
  // K2 outputs rebuilt from the oracle
  std::vector<double> cum((size_t)6 * total, 0.0);
  std::vector<int32_t> fwd_prev(total), rev_next(total);
  std::vector<uint8_t> qual(total, 31);
  std::vector<std::vector<int>> raw_qual((size_t)n);
  long n_zero = 0, n_high = 0;
  for (int64_t i = 0; i < n; i++) {
    const int L = (int)reads[i].size();
    if (L == 0) continue;
    const char* s = reads[i].c_str();
    std::vector<double> fs((size_t)6 * L);
    orc_score_all_frames(gene, indep, s, L, fs.data());
    for (int c = 0; c < 3; c++) {
      double acc = 0.0;
      for (int q = L - 1; q >= 0; q--) {  // forward class c: suffix sums of FS[(c - q) mod 3][q]
        acc += fs[(size_t)mgf_mod3(c - q) * L + q];
        cum[(size_t)c * total + off[i] + q] = acc;
      }
      acc = 0.0;
      for (int q = 0; q < L; q++) {  // reverse class c: prefix sums of FS[3 + (1 + q - c) mod 3][q]
        acc += fs[(size_t)(3 + mgf_mod3(1 + q - c)) * L + q];
        cum[(size_t)(3 + c) * total + off[i] + q] = acc;
      }
    }
    orc_save_prev_stops(s, L, &op, fwd_prev.data() + off[i], rev_next.data() + off[i]);
    std::vector<int> qv(L);
    if (have_qual) {
      raw_qual[i] = seeded_quality(qual_state, L);
      qv = raw_qual[i];
      if (op.allow_indels) orc_clean_quality_454(s, L, qv.data(), op.indel_quality_threshold);
      for (int q = 0; q < L; q++) {
        n_zero += qv[q] == 0;
        n_high += qv[q] >= 163;
      }
    } else {
      orc_set_quality_454(s, L, qv.data());
    }
    for (int q = 0; q < L; q++) qual[off[i] + q] = (uint8_t)qv[q];
  }
  const int64_t nblk = total / 32 + 2;
  std::vector<uint32_t> gate_bits(nblk, 0), gate_cnt(nblk, 0), gate_rank, gate_pos;
  for (int64_t p = 0; p < total; p++)
    if ((int)qual[p] <= P.indel_q_thresh) {
      gate_bits[p >> 5] |= 1u << (p & 31);
      gate_cnt[p >> 5]++;
      gate_pos.push_back((uint32_t)p);
    }
  exscan(gate_cnt, gate_rank);
  gate_pos.push_back(0);
  std::vector<double> tables(516);
  for (int q = 0; q < 256; q++) {
    const double pe = pow(10.0, -(double)q / 10.0);
    tables[q] = log(pe / 2.0) - log(1.0 - pe);
    tables[260 + q] = 1.0 - pe;
  }
  for (int t = 0; t < 4; t++) {
    const double dpv = 0.999;
    double ps = dpv;
    ps *= (t & 2) ? (2.0 / 3.0 * dpv + 1.0 / 3.0) : dpv;
    ps *= (t & 1) ? (2.0 / 3.0 * dpv + 1.0 / 3.0) : dpv;
    tables[256 + t] = log(1.0 - ps) - log(ps);
  }

  // ORFs + oracle start lists
  std::vector<gmg_orf> orfs;
  std::vector<int32_t> orf_seq;
  std::vector<orc_start> want;
  std::vector<int64_t> want_off(1, 0);
  for (int64_t i = 0; i < n; i++) {
    const int L = (int)reads[i].size();
    orc_orf* o = NULL;
    const int no = orc_find_orfs(reads[i].c_str(), L, &op, &o);
    std::vector<int> so(no + 1, 0);
    orc_start* st = NULL;
    const int ns = orc_mg_score_orfs(gene, indep, reads[i].c_str(), L, have_qual ? raw_qual[i].data() : NULL, &op, o, no, so.data(),
                                     &st);
    for (int k = 0; k < no; k++) {
      gmg_orf g;
      g.frame = o[k].frame;
      g.stop_position = o[k].stop_position;
      g.orf_len = o[k].orf_len;
      g.gene_len = o[k].gene_len;
      orfs.push_back(g);
      orf_seq.push_back((int32_t)i);
      want_off.push_back(want_off.back() + (so[k + 1] - so[k]));
    }
    for (int k = 0; k < ns; k++) want.push_back(st[k]);
    free(o);
    free(st);
  }
  const uint32_t n_orfs = (uint32_t)orfs.size();

  MgfBatch B;
  B.words = words;
  B.off = off.data();
  B.total = total;
  B.cum = cum.data();
  B.fwd_prev = fwd_prev.data();
  B.rev_next = rev_next.data();
  B.qual = qual.data();
  B.cert = NULL;
  B.cb = cb.data();
  B.nwc = nwc;
  B.gate_bits = gate_bits.data();
  B.gate_rank = gate_rank.data();
  B.gate_pos = gate_pos.data();
  B.tables = tables.data();
  B.sub_pen = NULL;
  // Pass_Stop_Penalty of every root call with a quality file: p_stop as k_mg_sub_pstop forms it, the log as the host takes it
  std::vector<double> sub_pen;
  if (have_qual && op.allow_subs) {
    sub_pen.resize(n_orfs);
    for (uint32_t o = 0; o < n_orfs; o++) {
      const MgfSeq S = mgf_seq_of(B, orf_seq[o]);
      const bool fwd = orfs[o].frame > 0;
      int lo, hi;
      mgf_open(B, S, fwd, fwd ? orfs[o].stop_position - 1 : orfs[o].stop_position + 3, &lo, &hi);
      const double ps = mgf_stop_pstop(B, S, fwd, lo, hi);
      sub_pen[o] = log(1.0 - ps) - log(ps);
    }
    B.sub_pen = sub_pen.data();
  }

  MgfWork W;
  memset(&W, 0, sizeof W);
  W.orfs = orfs.data();
  W.orf_seq = orf_seq.data();
  W.n_orfs = n_orfs;
  std::vector<MgfCall> root(n_orfs);
  std::vector<uint32_t> n1(n_orfs + 1, 0), off1, own0(n_orfs, 0);
  W.root = root.data();
  W.n1 = n1.data();
  W.own0 = own0.data();
  for (uint32_t o = 0; o < n_orfs; o++) mgf_pass_a(B, P, W, o);
  exscan(n1, off1);
  W.off1 = off1.data();
  W.c1 = off1[n_orfs];
  std::vector<MgfCall> call1(W.c1 + 1);
  std::vector<uint32_t> n2(W.c1 + 1, 0), off2, own1(W.c1 + 1, 0), t1(W.c1 + 1, 0), s1;
  W.call1 = call1.data();
  W.n2 = n2.data();
  W.own1 = own1.data();
  std::vector<uint32_t> par1(W.c1 + 1, 0);
  W.par1 = par1.data();
  for (uint32_t o = 0; o < n_orfs; o++) mgf_fill_parent(W.off1, o, W.par1);
  for (uint32_t i = 0; i < W.c1; i++) mgf_pass_b(B, P, W, i);
  exscan(n2, off2);
  W.off2 = off2.data();
  W.c2 = off2[W.c1];
  std::vector<uint32_t> cnt3(W.c2 + 1, 0), s3;
  W.cnt3 = cnt3.data();
  std::vector<uint32_t> par2(W.c2 + 1, 0);
  W.par2 = par2.data();
  for (uint32_t i = 0; i < W.c1; i++) mgf_fill_parent(W.off2, i, W.par2);
  for (uint32_t i = 0; i < W.c2; i++) mgf_pass_c(B, P, W, i);
  exscan(cnt3, s3);
  W.s3 = s3.data();
  W.t1 = t1.data();
  for (uint32_t i = 0; i < W.c1; i++) mgf_pass_d(W, i);
  exscan(t1, s1);
  W.s1 = s1.data();
  std::vector<int64_t> counts(n_orfs + 1, 0), start_off;
  W.counts = counts.data();
  for (uint32_t o = 0; o < n_orfs; o++) mgf_pass_e(W, o);
  exscan(counts, start_off);
  W.start_off = start_off.data();
  const int64_t n_starts = start_off[n_orfs];
  std::vector<gmg_start> starts((size_t)n_starts + 1);
  memset(starts.data(), 0xEE, starts.size() * sizeof(gmg_start));
  W.starts = starts.data();
  for (uint32_t o = 0; o < n_orfs; o++) mgf_write_0(B, P, cs, W, o);
  for (uint32_t i = 0; i < W.c1; i++) mgf_write_1(B, P, cs, W, i);
  for (uint32_t i = 0; i < W.c2; i++) mgf_write_2(B, P, cs, W, i);

  // compare
  long bad = 0;
  if (n_starts != (int64_t)want.size()) {
    printf("TOTAL starts %lld, oracle %zu\n", (long long)n_starts, want.size());
    bad++;
  }
  static_assert(sizeof(gmg_start) == sizeof(orc_start), "record layouts differ");
  for (uint32_t o = 0; o < n_orfs && bad < 10; o++) {
    const int64_t a = start_off[o], b = start_off[o + 1], wa = want_off[o], wb = want_off[o + 1];
    if (b - a != wb - wa) {
      printf("ORF %u (seq %d frame %d stop %d): %lld records, oracle %lld\n", o, orf_seq[o], orfs[o].frame, orfs[o].stop_position,
             (long long)(b - a), (long long)(wb - wa));
      bad++;
      continue;
    }
    for (int64_t k = 0; k < b - a; k++)
      if (memcmp(&starts[a + k], &want[wa + k], sizeof(gmg_start)) != 0) {
        const gmg_start& g = starts[a + k];
        const orc_start& w = want[wa + k];
        printf("ORF %u (seq %d frame %d stop %d) record %lld: got j=%d pos=%d sc=%.17g w=%d t=%d f=%d ne=%d (%d:%d %d:%d)  want j=%d pos=%d "
               "sc=%.17g w=%d t=%d f=%d ne=%d (%d:%d %d:%d)\n",
               o, orf_seq[o], orfs[o].frame, orfs[o].stop_position, (long long)k, g.j, g.pos, g.score, g.which, g.truncated, g.first,
               g.n_err, g.err_pos[0], g.err_type[0], g.err_pos[1], g.err_type[1], w.j, w.pos, w.score, w.which, w.truncated, w.first,
               w.n_err, w.err_pos[0], w.err_type[0], w.err_pos[1], w.err_type[1]);
        bad++;
        break;
      }
  }
  // plain mode: the position-by-position form of a root call's records (mgf_plan / mgf_recs_at, what the lanes of the
  // fused kernel evaluate) against the same oracle lists
  if (!op.allow_indels && !op.allow_subs) {
    for (uint32_t o = 0; o < n_orfs && bad < 10; o++) {
      const MgfSeq S = mgf_seq_of(B, orf_seq[o]);
      const gmg_orf orf = orfs[o];
      const bool fwd = orf.frame > 0;
      const int hi = fwd ? orf.stop_position - 1 : orf.stop_position + 3 + orf.orf_len;
      const int lo = fwd ? hi - orf.orf_len : orf.stop_position + 3;
      MgfOwn f;
      mgf_own_open(B, S, P, fwd, lo, hi, 0, f);
      MgfPlan pl;
      mgf_plan(f, fwd, pl);
      const double* row = mgf_row(B, S, fwd, lo, hi);
      const double cbase = mgf_cbase(B, S, fwd, lo, hi);
      std::vector<gmg_start> got;
      bool seen_nonzero = false;
      const int ep[2] = {0, 0}, et[2] = {0, 0};
      if (f.j_hi >= f.j_lo)
        for (int j = f.j_hi; j >= f.j_lo; j -= 3) {
          bool trunc_rec, chain;
          const int nr = mgf_recs_at(f, pl, fwd, j, &trunc_rec, &chain);
          if (nr == 0) continue;
          const double sc = (mgf_score(S, fwd, row, lo, hi, cbase, j - 1) - 0.0) + 0.0;
          const int k = mgf_kpos(f, fwd, j);
          gmg_start st;
          memset(&st, 0, sizeof st);
          if (trunc_rec) {
            mgf_put(&st, P, j + 2, k, sc, -1, 1, 1, 0, ep, et);
            got.push_back(st);
            if (nr == 2) {
              mgf_put(&st, P, j + 2, k, sc, mgf_which_at(B, S, cs.which, f, fwd, j), 0, 0, 0, ep, et);
              got.push_back(st);
            }
          } else {
            mgf_put(&st, P, j + 2, k, sc, mgf_which_at(B, S, cs.which, f, fwd, j), 0, (pl.state_after && !seen_nonzero) ? 1 : 0, 0, ep,
                    et);
            got.push_back(st);
            if (k != 0) seen_nonzero = true;
          }
        }
      const int64_t wa = want_off[o], wb = want_off[o + 1];
      if ((int64_t)got.size() != wb - wa) {
        printf("lane form: ORF %u: %zu records, oracle %lld\n", o, got.size(), (long long)(wb - wa));
        bad++;
        continue;
      }
      for (size_t k = 0; k < got.size(); k++) {
        gmg_start w;
        memcpy(&w, &want[wa + k], sizeof w);
        // padding bytes of the host-built record are zero as in mgf_put's full assignment: compare field by field
        const gmg_start& g = got[k];
        if (g.j != w.j || g.pos != w.pos || memcmp(&g.score, &w.score, 8) != 0 || g.which != w.which || g.truncated != w.truncated ||
            g.first != w.first || g.n_err != w.n_err) {
          printf("lane form: ORF %u record %zu: got j=%d pos=%d sc=%.17g w=%d t=%d f=%d  want j=%d pos=%d sc=%.17g w=%d t=%d f=%d\n", o, k,
                 g.j, g.pos, g.score, g.which, g.truncated, g.first, w.j, w.pos, w.score, w.which, w.truncated, w.first);
          bad++;
          break;
        }
      }
    }
  }
  long n_inf = 0, n_ninf = 0;
  for (const orc_start& w : want) {
    n_inf += isinf(w.score) && w.score > 0;
    n_ninf += isinf(w.score) && w.score < 0;
  }
  printf("%s: %lld reads, %u ORFs, %u level-1 candidates, %u level-2 candidates, %lld starts (oracle %zu); qualities 0: %ld, "
         ">= 163: %ld; scores +inf: %ld, -inf: %ld\n",
         bad ? "MISMATCH" : "OK", (long long)n, n_orfs, W.c1, W.c2, (long long)n_starts, want.size(), n_zero, n_high, n_inf, n_ninf);
  return bad ? 1 : 0;
}
