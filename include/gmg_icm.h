/* include/gmg_icm.h -- C-ABI of libgmgicm.so, the B200 (sm_100a) implementation of
 * Glimmer-MG's ICM scoring and training hot path.
 *
 * This is the drop-in boundary.  The reference has no FFI; its seam is the C++ class
 * interface of libGLMicm.a (src/ICM/icm.hh:116-213) plus the file-static scoring
 * functions of the two drivers (src/Glimmer/glimmer-mg.cc, glimmer3.cc).  Every entry
 * point below names the reference interface it replaces (paths relative to
 * /root/reference/src/).  Plain pointers and sizes only; no C++ / torch types.
 *
 * Conventions
 *  - every function returns 0 on success, non-zero on error; gmg_last_error() returns
 *    the message (the C++ facade turns it into the reference's "message on stderr +
 *    exit(EXIT_FAILURE)" behaviour, icm.cc:635-657).
 *  - there is NO CPU fallback: gmg_ctx_create fails if no CUDA device is usable.
 *  - "h_" pointers are host memory, "d_" pointers are device memory of the context's
 *    device.  All work is enqueued on the context's stream; functions that return
 *    host data synchronise that stream before returning, functions documented
 *    "async" do not.
 *  - sequences are ASCII; every character goes through tolower(Filter(c))
 *    (Common/gene.cc:1139-1175) on the device, exactly like the drivers do
 *    (glimmer-mg.cc:381-382, glimmer3.cc:270-271), and is then held 2 bits/base.
 */
#ifndef GMG_ICM_H
#define GMG_ICM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GMG_ABI_VERSION 1

typedef struct gmg_ctx gmg_ctx;       /* one per GPU / host thread: device, stream, scratch */
typedef struct gmg_icm gmg_icm;       /* ICM_t: host mirror + device tables */
typedef struct gmg_seqset gmg_seqset; /* a batch of sequences packed 2-bit in HBM */
typedef struct gmg_trainer gmg_trainer; /* ICM_Training_t */

/* Orf_t (Common/gene.hh:101-136) */
typedef struct {
  int32_t frame;         /* +-(1..3) */
  int32_t stop_position; /* 1-based lowest coordinate of the stop codon (may be <1 or >len-2) */
  int32_t orf_len, gene_len;
} gmg_orf;

/* Start_t (Glimmer/glimmer_base.hh:80-88), error vector flattened (<= 2 entries) */
typedef struct {
  int32_t j, pos;
  double score;
  int32_t which;      /* index into the start-codon list, -1 = truncated */
  int32_t truncated, first;
  int32_t n_err;
  int32_t err_pos[2];
  int32_t err_type[2]; /* 0 insertion, 1 deletion, 2 substitution (gene.hh:138-146) */
} gmg_start;

/* Options of the scoring half.  gmg_params_default fills the reference's defaults
 * (glimmer_base.hh:24-34, glimmer-mg.cc:12,107-138, glimmer3.cc:23). */
typedef struct {
  int32_t min_gene_len;            /* Min_Gene_Len, 75 */
  int32_t allow_truncated;         /* Allow_Truncated_Orfs: glimmer-mg 1, glimmer3 0 (-X) */
  int32_t allow_indels;            /* glimmer-mg -i */
  int32_t allow_subs;              /* glimmer-mg -s */
  int32_t min_indel_orf_len;       /* Min_Indel_ORF_Len, 15 */
  int32_t indel_quality_threshold; /* 18 (<= 254 supported: threshold + 1 must fit the uint8 quality plane) */
  int32_t indel_max;               /* 2 (<= 2 supported) */
  int32_t ignore_score_len;        /* Ignore_Score_Len; INT32_MAX = off */
  double indel_suffix_score_threshold; /* -12 */
  int32_t have_quality_file;       /* Quality_File_Name != NULL (changes Pass_Stop_Penalty); the set's qualities are
                                      cleaned (Clean_Quality_454) under allow_indels only, as glimmer-mg does */
  int32_t n_start, n_stop;
  char start_codon[8][4];          /* lower-case, e.g. "atg" */
  char stop_codon[8][4];
} gmg_params;

/* ---- context -------------------------------------------------------------------- */
int gmg_abi_version(void);
const char* gmg_last_error(void);
/* stream: a cudaStream_t (e.g. torch's current stream) or NULL for a private stream */
int gmg_ctx_create(int device, void* stream, gmg_ctx** out);
void gmg_ctx_destroy(gmg_ctx* ctx);
int gmg_ctx_sync(gmg_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
int64_t gmg_ctx_launch_count(const gmg_ctx* ctx);
/* Per-kernel device timing for bench.py's roofline: while enabled, CUDA events on the context's
 * stream bracket every launch of the hot kernels.  gmg_ctx_profile_read synchronises the stream and
 * returns (and resets) the summed duration and launch count of one kernel class. */
#define GMG_PROF_K1 0   /* k1_planes: six-frame tree walks */
#define GMG_PROF_K2 1   /* k2_prefix: prefix sums / stop tables / quality */
#define GMG_PROF_K3 2   /* k3_*_starts: start enumeration (count + write passes) */
#define GMG_PROF_K4 3   /* k4_count: training context counts */
#define GMG_PROF_ORF 4  /* ORF finder */
#define GMG_PROF_PACK 5 /* Filter + 2-bit pack */
#define GMG_PROF_FS 6   /* Frame_Scores surface (gene - indep as FP64) */
int gmg_ctx_profile(gmg_ctx* ctx, int enable);
int gmg_ctx_profile_read(gmg_ctx* ctx, int kernel_class, double* ms, int64_t* launches);
/* page-locked host memory (cudaMallocHost) for callers without a CUDA runtime of their own: input
 * and output buffers allocated here make the H2D / D2H copies of the calls below run at PCIe rate */
int gmg_host_alloc(size_t bytes, void** out);
void gmg_host_free(void* p);
/* plain copies on the context's stream (for callers without a CUDA runtime of their own); both sync */
int gmg_ctx_memcpy_d2h(gmg_ctx* ctx, void* h_dst, const void* d_src, size_t bytes);
int gmg_ctx_memcpy_h2d(gmg_ctx* ctx, void* d_dst, const void* h_src, size_t bytes);
void gmg_params_default(gmg_params* p, int metagenomic);
/* Set_Ignore_Score_Len (glimmer_base.cc:2597-2633) */
int gmg_ignore_score_len(double gc, const gmg_params* p);

/* ---- models: ICM_t ---------------------------------------------------------------- */
/* ICM_t::Read / Input (icm.cc:846, 614-726): build-icm binary format */
int gmg_icm_load(gmg_ctx* ctx, const char* path, gmg_icm** out);
/* ICM_t::Input(FILE*) (icm.cc:614-726) for callers that hold the model file's bytes (an open FILE* read to memory, an
 * mmap, a network buffer): the same format from a memory image */
int gmg_icm_load_mem(gmg_ctx* ctx, const void* image, size_t n_bytes, gmg_icm** out);
/* ICM_t(w,d,p) filled from caller tables: mip int16 [p][nodes], prob float [p][nodes][4] */
int gmg_icm_from_tables(gmg_ctx* ctx, int w, int d, int p, const int16_t* h_mip, const float* h_prob,
                        gmg_icm** out);
/* ICM_t::Build_Indep_WO_Stops (icm.cc:65-216) on an ICM_t(3,2,3) */
int gmg_icm_build_indep(gmg_ctx* ctx, double gc, const char* const* stops, int n_stops, gmg_icm** out);
/* ICM_t::Output(fp, binary=true) (icm.cc:729-803, 961-998) */
int gmg_icm_write(const gmg_icm* m, const char* path);
/* the same image into caller memory (ICM_t::Output(FILE*, true) without a file): *n_bytes = image size; copied to
 * h_out when cap >= *n_bytes (h_out = NULL sizes the buffer) */
int gmg_icm_write_mem(const gmg_icm* m, void* h_out, size_t cap, size_t* n_bytes);
/* {model_len, model_depth, periodicity, num_nodes}  (Get_Model_Len / Get_Periodicity) */
int gmg_icm_dims(const gmg_icm* m, int32_t dims[4]);
int gmg_icm_tables(const gmg_icm* m, int16_t* h_mip, float* h_prob);
/* ICM_Score_Node_t::mut_info (icm.hh:106-113, STORE_MUT_INFO): [P][N] floats, the mutual information of each
 * node's branch position as stored by Train_Model (icm.cc:1156,1438); 0 for models read from a file (the
 * binary format does not carry it, icm.cc:614-727).  Only the text form of ICM_t::Output prints it. */
int gmg_icm_mut_info(const gmg_icm* m, float* h_out);
void gmg_icm_free(gmg_icm* m);

/* ---- sequence batches -------------------------------------------------------------- */
/* n sequences, concatenated ASCII in h_ascii, sequence i = [h_off[i], h_off[i+1]).
 * H2D copy + device Filter/2-bit pack (+ GC count).  h_qual (optional, may be NULL):
 * one Phred value per base (Fasta_Qual_Vec_Read, fasta.cc:115). */
int gmg_seqset_create(gmg_ctx* ctx, const char* h_ascii, const int64_t* h_off, int64_t n,
                      const uint8_t* h_qual, gmg_seqset** out);
/* same, ASCII already resident in HBM (d_ascii); offsets still from the host.  Returns once d_ascii has been read. */
int gmg_seqset_create_device(gmg_ctx* ctx, const void* d_ascii, const int64_t* h_off, int64_t n,
                             const void* d_qual, gmg_seqset** out);
void gmg_seqset_free(gmg_seqset* s);
/* FASTA ingest on the device (Fasta_Read, Common/fasta.cc:236-283; build-icm's Read_String, ICM/build-icm.cc:262-315):
 * `h_bytes` is a multi-FASTA image in host memory (page-locked memory from gmg_host_alloc makes the copy run at
 * PCIe rate).  Bytes before the first '>' are skipped; a '>' outside a header line starts a record whose header
 * runs to the end of the line; every other non-white-space byte up to the next '>' is a sequence character
 * (Filter + lower-case applied as in gmg_seqset_create).  Images must be < 1 GiB (split larger files at record
 * boundaries).  gmg_seqset_offsets returns the n+1 sequence offsets of any seqset; gmg_seqset_fasta_headers the
 * header text of record i as image[hdr_off[i], hdr_end[i]) (after the '>', up to the line end). */
int gmg_seqset_from_fasta(gmg_ctx* ctx, const char* h_bytes, int64_t n_bytes, gmg_seqset** out, int64_t* n_records);
int64_t gmg_seqset_count(const gmg_seqset* s);
int gmg_seqset_offsets(const gmg_seqset* s, int64_t* h_off);
int gmg_seqset_fasta_headers(const gmg_seqset* s, int64_t* h_hdr_off, int64_t* h_hdr_end);
/* Quality values from the image of a quality file (Fasta_Qual_Vec_Read, Common/fasta.cc:115-170: a '>' header line per
 * record, then integers separated by white space; a value is taken when white space follows it, characters that are
 * neither digits nor white space are skipped, digits still pending at the next '>' or at the end of the file are
 * dropped), parsed on the device.
 * gmg_quality_parse_fasta: *n_records / *n_values always; h_off (n_records + 1 entries: values before each record) and
 *   h_values are filled when their capacities suffice (call once with NULL / 0 to size them).
 * gmg_seqset_quality_from_fasta: attaches the values (clamped to 0..255, as the bindings pass them) to a set as its
 *   per-base qualities -- what gmg_seqset_create's h_qual does; the records must match the set's sequences in number and
 *   length (glimmer-mg.cc:534-537: "sequence length does not match quality values length"). */
int gmg_quality_parse_fasta(gmg_ctx* ctx, const char* h_bytes, int64_t n_bytes, int64_t* n_records, int64_t* n_values,
                            int64_t* h_off, int32_t* h_values, int64_t cap_records, int64_t cap_values);
int gmg_seqset_quality_from_fasta(gmg_ctx* ctx, gmg_seqset* s, const char* h_bytes, int64_t n_bytes);
/* FASTQ ingest on the device: the sequences and Phred qualities of a FASTQ image in host memory (page-locked memory from
 * gmg_host_alloc makes the copy run at PCIe rate).  Four-line records, LF or CRLF line ends:
 *   line 1  '@' and the header.  Its text is what gmg_seqset_fasta_headers reports for the same line with '>' in place of
 *           '@' (blanks after the marker skipped, the text runs to the line end), so FASTQ converted to FASTA keeps its
 *           headers.  gmg_seqset_fasta_headers returns it as offsets into the FASTQ image.
 *   line 2  the sequence: every non-white-space byte is a sequence character (Filter + lower-case + 2-bit pack as in
 *           gmg_seqset_create, and the set keeps its non-acgt list, so gmg_seqset_extract works on it).
 *   line 3  '+', optionally followed by the header text again (blanks after the '+' skipped; one trailing '\r' of either
 *           line does not count).  Any other text is an error.
 *   line 4  the qualities: as many bytes as line 2 has sequence characters (one trailing '\r' does not count), each in
 *           [phred_offset, '~']; the value is byte - phred_offset.  phred_offset is 33 or 64.
 * An empty sequence with an empty quality line is a record of length 0.  The last line may lack its '\n' (the text after
 * a final '\n' is an empty last line).  Blank lines may follow the last record, nowhere else: the records end at the line
 * of the last non-white-space byte.  Multi-line records are not supported (they fail the '@' / '+' checks).  Images must
 * be < 1 GiB (split larger files at record boundaries).
 * Every violation fails the call, with a message (gmg_last_error) naming the first bad record and its line (1-based) and
 * the reason: no '@' / '+', '+' text other than the header, quality length other than the sequence length, a quality
 * byte out of range, or a truncated last record.  Nothing is allocated for a rejected image (*out = NULL) and the
 * context stays usable.
 * The set carries its qualities exactly as gmg_seqset_quality_from_fasta attaches them, so gmg_score_orfs_mg with
 * have_quality_file = 1 runs on it directly. */
int gmg_seqset_from_fastq(gmg_ctx* ctx, const char* h_bytes, int64_t n_bytes, int phred_offset, gmg_seqset** out,
                          int64_t* n_records);
/* per-base qualities of any set (0..255, as attached: total_bases bytes to h_out); returns non-zero if the set has none
 * (a set without bases has none).  h_out = NULL only asks whether it has them. */
int gmg_seqset_qualities(const gmg_seqset* s, uint8_t* h_out);
int64_t gmg_seqset_total_bases(const gmg_seqset* s);
/* Set_GC_Fraction (glimmer_base.cc:2564-2595): (#c + #g after Filter) / total */
int gmg_seqset_gc_fraction(gmg_seqset* s, double* gc);
/* unpack to lower-case acgt (what the drivers hold in `Sequence`) */
int gmg_seqset_unpack(gmg_seqset* s, char* h_out);
/* extract (Util/extract.cc) on a resident set: n regions [lo[i], lo[i] + len[i]) of sequence seq[i] (0-based) become the
 * n sequences of a new set; strand[i] = -1 takes the reverse complement of the region, complementing raw IUPAC codes before
 * Filter as extract + build-icm do.  Regions must lie inside their sequence (no wrap-around).  The new set is an ordinary
 * set (score, find ORFs, train, unpack, extract again); it carries no qualities and no headers.  Every set keeps the
 * position and raw code of each input byte other than a / c / g / t for this; a minus region's output holds the
 * complemented code, so extracting from an extracted set equals extracting from the source directly. */
int gmg_seqset_extract(gmg_ctx* ctx, gmg_seqset* src, int64_t n, const int32_t* h_seq, const int32_t* h_lo,
                       const int32_t* h_len, const int8_t* h_strand, gmg_seqset** out);

/* ---- scalar operator surface (each call = device work over one string) -------------- */
/* ICM_t::Score_String (icm.cc:864-903) for n strings of a seqset; frame = first base's period */
int gmg_icm_score_strings(gmg_ctx* ctx, const gmg_icm* m, gmg_seqset* s, int frame, double* h_out);
/* ICM_t::Cumulative_Score (icm.cc:354-405): out[off[i]+t] for every string */
/* Score_String of every sequence against every model in one launch (the many-model read scoring that precedes
 * glimmer-mg: Phymm / Scimm `simple-score`, scripts/scoreReadsGlim.pl:450,482).  h_out[k * n_seqs + i] = score of
 * sequence i under models[k]; models may differ in window, depth and periodicity.  Bit-identical to
 * gmg_icm_score_strings model by model. */
int gmg_icm_score_strings_many(gmg_ctx* ctx, const gmg_icm* const* models, int n_models, gmg_seqset* s, int frame,
                               double* h_out);
int gmg_icm_cumulative_score(gmg_ctx* ctx, const gmg_icm* m, gmg_seqset* s, int frame, double* h_out);
/* ICM_t::Frame_Score (icm.cc:485-509): per-position log-prob, fixed period */
int gmg_icm_frame_score(gmg_ctx* ctx, const gmg_icm* m, gmg_seqset* s, int frame, double* h_out);
/* ICM_t::Full_Window_Prob / Partial_Window_Prob (icm.cc:557-610, 807-842) for one window
 * (convenience wrappers over the kernels above) */
int gmg_icm_full_window_prob(gmg_ctx* ctx, const gmg_icm* m, const char* w, int frame, double* out);
int gmg_icm_partial_window_prob(gmg_ctx* ctx, const gmg_icm* m, int predict_pos, const char* s, int frame,
                                double* out);

/* ---- batched scoring half ------------------------------------------------------------ */
/* Score_All_Frames (glimmer-mg.cc:1468-1510): Frame_Scores[f][i] = gene - indep for the 6
 * frames of every sequence.  out layout: for sequence i, six rows of len_i doubles starting
 * at 6*off[i].  out may be a host pointer (copied back, sync) or, with out_on_device != 0, a
 * device pointer (async). */
int gmg_score_all_frames(gmg_ctx* ctx, const gmg_icm* gene, const gmg_icm* indep, gmg_seqset* s,
                         double* out, int out_on_device);
/* K1 alone (the dominant kernel): gene log-probs of all six (strand, reading-frame class)
 * planes into the context's scratch; nothing copied out.  async.  For benchmarking/profiling. */
int gmg_k1_score_planes(gmg_ctx* ctx, const gmg_icm* gene, gmg_seqset* s);

/* Find_Orfs (glimmer_base.cc:638-817) on the device, linear sequences, no ignore regions.
 * Results stay on the device inside the seqset; *n_orfs receives the total. orfs of sequence i
 * are [orf_off[i], orf_off[i+1]) in reference order. */
int gmg_find_orfs(gmg_ctx* ctx, gmg_seqset* s, const gmg_params* p, int64_t* n_orfs);
int gmg_get_orfs(gmg_ctx* ctx, gmg_seqset* s, gmg_orf* h_orfs, int64_t* h_orf_off /* n+1, may be NULL */);
/* caller-supplied ORF table instead (the reference boundary: host Find_Orfs -> orf_list) */
int gmg_set_orfs(gmg_ctx* ctx, gmg_seqset* s, const gmg_orf* h_orfs, const int64_t* h_orf_off);

/* glimmer3 Score_Orfs start enumeration (glimmer3.cc:1275-1466): per ORF, Cumulative_Score
 * of the gene ICM and the independent model over the ORF string and the start_list
 * (j, pos, score, which, truncated, first) in generation order, long-ORF boost applied.
 * Needs ORFs (gmg_find_orfs / gmg_set_orfs).  *n_starts = total. async until gmg_get_starts. */
int gmg_score_orfs_g3(gmg_ctx* ctx, const gmg_icm* gene, const gmg_icm* indep, gmg_seqset* s,
                      const gmg_params* p, int64_t* n_starts);
/* All_Frame_Score (glimmer3.cc:328-359), batched, for the `.detail` log: for each of n regions [lo, lo + len) (0-based)
 * of sequence h_seq[i] the six Score_String sums of the gene ICM the reference forms -- h_out[6 i + k], k = 0..2: the
 * region read downwards (a forward gene's buff) with the first base in period k; k = 3..5: the region's complement
 * read upwards (a reverse gene's buff) with the first base in period k - 3.  Sums in the reference's serial order. */
int gmg_all_frame_scores(gmg_ctx* ctx, const gmg_icm* gene, gmg_seqset* s, int64_t n, const int32_t* h_seq,
                         const int32_t* h_lo, const int32_t* h_len, double* h_out);
/* glimmer-mg Score_Orfs_Errors up to the boost (glimmer-mg.cc:1605-1651): Score_All_Frames,
 * Save_Prev_Stops, Set_Quality_454 / Clean_Quality_454, Cumulative_Frame_Score and the
 * Score_Orf_Starts / Score_Indels / Pass_Stop_Penalty recursion for every ORF. */
int gmg_score_orfs_mg(gmg_ctx* ctx, const gmg_icm* gene, const gmg_icm* indep, gmg_seqset* s,
                      const gmg_params* p, int64_t* n_starts);
/* gmg_score_orfs_mg with a per-sequence independent model (glimmer-mg -c, which builds the model from each read's GC
 * fraction): sequence i is scored as gmg_score_orfs_mg scores it in a set of its own with
 * indep = Build_Indep_WO_Stops(h_gc[i], p's stop codons) and p->ignore_score_len replaced by h_isl[i] (h_isl = NULL:
 * p->ignore_score_len for all).  Results (raw start lists, gmg_get_starts / gmg_get_orf_starts / gmg_reduce_starts_mg
 * afterwards) are bit-identical to that.  Needs ORFs (gmg_find_orfs / gmg_set_orfs); every mode of gmg_score_orfs_mg.
 * The models are built on the device, one per distinct GC value (exact bit pattern); the launch count does not depend
 * on the number of sequences or of distinct values.  Rejected before any device work, with a message naming the first
 * bad sequence: a GC value that is NaN or outside [0, 1], a negative ignore length; the context stays usable. */
int gmg_score_orfs_mg_gc(gmg_ctx* ctx, const gmg_icm* gene, gmg_seqset* s, const double* h_gc, const int32_t* h_isl,
                         const gmg_params* p, int64_t* n_starts);
/* The models of gmg_score_orfs_mg_gc take their logarithms on the device where the result provably rounds to the float
 * that glibc's log gives; the other entries are recomputed on the host.  This returns how many entries the last
 * gmg_score_orfs_mg_gc call on the context recomputed (diagnostic; results are exact either way). */
int64_t gmg_ctx_indep_flagged(const gmg_ctx* ctx);
/* ---- start-list reduction (the consumer side of Score_Orfs_Errors, glimmer-mg.cc:1656-1684, and the per-position
 * arg-max of Add_Events_Fwd / Add_Events_Rev, glimmer_base.cc:65-128, 175-235) ------------------------------------
 * With -i nearly every raw start record is dominated by another candidate at the same start position; the
 * reduction keeps, per ORF that passes the reference's two gates (first_j + 1 >= Min_Gene_Len, best score >
 * Start_Threshold), the one record per start position that can win Add_Events' `ne->score > best->score` test, so
 * that only survivors cross PCIe.  Candidates are ranked by the reference's event score without the RBS term
 * (score + prior [+ LogOdds_Start(which)] + LogOdds_Length(...), added in the reference's order); the RBS term is the
 * same for all candidates of a position.  The host then runs the reference's own Add_Events on the survivors.
 * Whenever the decision could depend on the last bits (two candidates of a position within 1e-9, records sharing the
 * extreme position with different j around Min_Gene_Len, a length beyond the table) the ORF gets status 2 and the host
 * fetches its raw list (gmg_get_orf_starts) and proceeds exactly as the reference does. */
typedef struct {
  double prior;            /* LogOdds_Prior (a float in the reference, glimmer-mg.cc:119), widened */
  double start_threshold;  /* Start_Threshold, -6 (glimmer-mg.cc:123) */
  double event_threshold;  /* Event_Threshold, -3 (glimmer-mg.cc:107) */
  double pwm_bonus_max;    /* upper bound of what Add_PWM_Score can add (glimmer_base.cc:267-295); 0 without an RBS
                              model, INFINITY if unknown (then no candidate is dropped by the threshold) */
  int32_t n_start;
  double start_lo[8];      /* LogOdds_Start.Score(which) */
  int32_t n_class;         /* fragment-length classes of LogOdds_Length (Length_Dist_t::Choose_Frag_Dist) */
  int32_t n_len;           /* table length: gene lengths (1 + j) / 3 below n_len */
  const double* len_lo;    /* host, [n_class][2 truncated_5p][2 truncated_3p][n_len]: LogOdds_Length.Score(l, t5, t3, frag) */
  const int32_t* seq_class; /* host, class of every sequence (from Sequence_Len / 3), or NULL: all class 0 */
} gmg_event_model;
/* Reduce the raw start lists of the last gmg_score_orfs_mg call on the device.  *n_kept = surviving records. */
int gmg_reduce_starts_mg(gmg_ctx* ctx, gmg_seqset* s, const gmg_params* p, const gmg_event_model* em, int64_t* n_kept,
                         int64_t* n_fallback_orfs /* unused, set to -1 */);
/* survivors: ORF i owns h_starts[h_first[i] .. h_first[i] + h_count[i]); h_status[i]: 0 = the ORF fails a gate or
 * has no surviving candidate, 1 = reduced list, 2 = undecided (take the raw list).  Any output may be NULL. */
int gmg_get_reduced_starts(gmg_ctx* ctx, gmg_seqset* s, gmg_start* h_starts, int64_t* h_first, int32_t* h_count,
                           uint8_t* h_status);
/* the raw start_list of one ORF of the last gmg_score_orfs_* call (*n = its length; h_out may be NULL to query) */
int gmg_get_orf_starts(gmg_ctx* ctx, gmg_seqset* s, int64_t orf, gmg_start* h_out, int64_t cap, int64_t* n);
/* start lists of the last gmg_score_orfs_* call: h_start_off has n_orfs+1 entries */
int gmg_get_starts(gmg_ctx* ctx, gmg_seqset* s, gmg_start* h_starts, int64_t* h_start_off);
/* FP64 sums are formed by parallel scans where an exactness certificate proves them bit-identical to the reference's
 * serial sums (DESIGN.md section 3.2); sequences (glimmer-mg with -i / -s) or ORFs (plain glimmer-mg) without one are
 * summed again in the reference's own serial order.  This returns how many took that route in the last call; results
 * are exact either way. */
int64_t gmg_uncertified_count(const gmg_seqset* s);
/* gmg_score_orfs_g3 forms its FP64 sums with warp-parallel scans where an exactness certificate proves
 * them bit-identical to the reference's serial sums, and re-does every other ORF in the reference's
 * order; this returns how many ORFs of the last call took that ordered path (results are exact either way). */
int gmg_ordered_fallback_count(gmg_seqset* s, int64_t* out);

/* ---- training: ICM_Training_t ---------------------------------------------------------- */
/* strings as given to Train_Model (icm.cc:1356): the seqset holds the training strings in
 * the orientation to be modelled (build-icm -r reverses on the host or with reverse != 0). */
int gmg_trainer_create(gmg_ctx* ctx, gmg_seqset* s, int w, int d, int p, int reverse, gmg_trainer** out);
void gmg_trainer_free(gmg_trainer* t);
/* K4: Count_Char_Pairs (level 0, icm.cc:1841-1870) / Count_Char_Pairs_Restricted +
 * Get_Training_Node (level >= 1, icm.cc:1190-1256) over this rank's strings.  Returns the device
 * pointer and element count of the level's int32 count slab [period][nodes_on_level][w-1][16]
 * so the caller can all-reduce it in place (NCCL sum) before gmg_trainer_finish_level. async. */
int gmg_trainer_count_level(gmg_trainer* t, int level, void** d_counts, int64_t* n_counts);
/* mutual-information position choice + Interpolate_Probs for the level (icm.cc:1097-1176,
 * 1401-1439, 1260-1330) from the (all-reduced) counts. */
int gmg_trainer_finish_level(gmg_trainer* t, int level);
/* Multi-GPU: this rank's seqset holds 1 / world of the training strings.  For large sets (window histogram) the
 * histogram is summed over the ranks once through `ar` and each rank then walks 1 / world of its cells per level, so
 * the level passes shrink with the number of GPUs.  Call before the first gmg_trainer_count_level. */
typedef int (*gmg_allreduce_fn)(void* user, void* d_buf, int64_t count, void* stream);
int gmg_trainer_set_shard(gmg_trainer* t, int rank, int world, int64_t global_bases /* training bases of ALL ranks: every
                          rank must choose the same counting path */, gmg_allreduce_fn ar, void* user);
/* Take_Logs (icm.cc:1334-1352) and hand the trained model over as a gmg_icm */
int gmg_trainer_finish(gmg_trainer* t, gmg_icm** out);
/* convenience: all levels, optional all-reduce callback (NULL = single GPU).  The callback
 * must sum `count` int32 at d_buf across ranks, ordered on `stream`. */
int gmg_icm_train(gmg_ctx* ctx, gmg_seqset* s, int w, int d, int p, int reverse, gmg_allreduce_fn ar,
                  void* user, gmg_icm** out);
/* the same with the strings dealt to `world` ranks (gmg_trainer_set_shard): `ar` sums the window histogram once and
 * every level's count slab across the ranks; every rank returns the identical model */
int gmg_icm_train_sharded(gmg_ctx* ctx, gmg_seqset* s, int w, int d, int p, int reverse, gmg_allreduce_fn ar, void* user,
                          int rank, int world, int64_t global_bases, gmg_icm** out);
/* Train_Model (icm.cc:1356) for n_models independent training sets in one call: out[k] is the model of sets[k], byte-identical
 * (gmg_icm_write) to gmg_icm_train(ctx, sets[k], w, d, p, reverse, NULL, NULL, &m).  All models share (w, d, p, reverse).
 * gmg_ctx_train_flagged afterwards returns the number of flagged nodes summed over the batch.  A set may appear more than
 * once.  On failure no out[k] is left allocated (all are NULL). */
int gmg_icm_train_many(gmg_ctx* ctx, gmg_seqset* const* sets, int n_models, int w, int d, int p, int reverse, gmg_icm** out);
/* Position choice and interpolation of a level run on the device; nodes whose choice lies within the error bound of the
 * device's logarithm are recomputed on the host with the reference's own libm.  This returns how many nodes of the
 * last gmg_icm_train* call on the context took that path (diagnostic). */
int64_t gmg_ctx_train_flagged(const gmg_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* GMG_ICM_H */
