// glimmer_mg_b200/host/build-icm.cc -- build-icm on the B200 training path.
//
// Same command line, input format and output file as the reference's build-icm
// (/root/reference/src/ICM/build-icm.cc:49-127, options :130-260, usage :366-403):
//
//     build-icm [options] output_file < input-file
//     build-icm [options] -B list          (each non-blank line of list: input_fasta output_file)
//       -d <num>  depth          -F  skip strings with in-frame stops     -h  help
//       -p <num>  period         -r  train on the reversed strings        -t  text output
//       -v <num>  verbosity      -w <num>  window length
//       -z <n>    stop codons of Genbank translation table n              -Z  comma-separated stop codons
//       -B <list> train one model per line of <list> in one device pass (not in the reference)
//
// The host side only parses FASTA and options; counting runs on the device (K4) through the ICM_Training_t
// facade (host/icm.hh -> gmg_icm_train, gmg_icm_train_many for -B).  Additional environment: GMG_DEVICE = GPU index.
#include <ctype.h>
#include <getopt.h>

#include <memory>
#include <string>
#include <vector>

#include "icm.hh"

static int Model_Len = DEFAULT_MODEL_LEN, Model_Depth = DEFAULT_MODEL_DEPTH, Model_Periodicity = DEFAULT_PERIODICITY;
static bool Print_Binary = true, Reverse_Strings = false, Skip_In_Frame_Stop_Strings = false;
static int Verbose = 0;
static std::vector<std::string> Stop_Codon;
static const char* Batch_List = NULL;

static void Usage() {
  fprintf(stderr,
          "USAGE:  build-icm [options] output_file < input-file\n"
          "        build-icm [options] -B <list>\n\n"
          "Read sequences from standard input and output to  output-file\n"
          "the interpolated context model built from them (counted on the GPU).\n"
          "If <output-file> is \"-\", then output goes to standard output\n"
          "With -B, every non-blank line of <list> is  input_fasta output_file :\n"
          "all inputs are read and checked, then one model per line is trained in\n"
          "one pass on the GPU and written to its output file; standard input is\n"
          "not read.  The other options apply to every model.\n\n"
          "Options:\n"
          " -B <list>  Build one model per line of <list> (see above)\n"
          " -d <num>   Set depth of model to <num>\n"
          " -F         Ignore input strings with in-frame stop codons\n"
          " -h         Print this message\n"
          " -p <num>   Set period of model to <num>\n"
          " -r         Use the reverse of input strings to build the model\n"
          " -t         Output model as text (for debugging only)\n"
          " -v <num>   Set verbose level\n"
          " -w <num>   Set length of model window to <num>\n"
          " -z <n>     Use Genbank translation table number <n> for stop codons\n"
          " -Z <list>  Comma-separated list of stop codons\n\n");
}

// stop codons of a Genbank translation table (the table the reference keeps in Common/gene.cc:1560-1640)
static bool Stops_By_Code(int code, std::vector<std::string>& out) {
  struct Row { int code; const char* stops; };
  static const Row rows[] = {{1, "taa,tag,tga"}, {11, "taa,tag,tga"}, {12, "taa,tag,tga"}, {2, "taa,tag,aga,agg"},
                             {3, "taa,tag"},     {4, "taa,tag"},      {5, "taa,tag"},      {9, "taa,tag"},
                             {10, "taa,tag"},    {13, "taa,tag"},     {21, "taa,tag"},     {6, "tga"},
                             {14, "tag"},        {15, "taa,tga"},     {16, "taa,tga"},     {22, "taa,tga,tca"},
                             {23, "taa,tag,tga,tta"}};
  out.clear();
  for (const Row& r : rows)
    if (r.code == code) {
      std::string s(r.stops);
      for (size_t a = 0; a < s.size(); a += 4) out.push_back(s.substr(a, 3));
      return true;
    }
  return false;
}

static bool Number(const char* arg, int* out, bool positive) {
  char* end;
  long v = strtol(arg, &end, 10);
  if (end == arg || (positive && v <= 0)) return false;
  *out = (int)v;
  return true;
}

// multi-FASTA image in memory -> training strings (host parser, used for -F and for images of 1 GiB or more):
// header lines start with '>', sequence characters are concatenated with white space removed and letters
// lower-cased (build-icm.cc:262-343)
static void Read_Training_Data(const char* image, size_t n, std::vector<char*>& data) {
  size_t i = 0;
  while (i < n && image[i] != '>') i++;
  while (i < n) {
    while (i < n && image[i] != '\n') i++;  // header line
    std::string cur;
    while (i < n && image[i] != '>') {
      const unsigned char ch = (unsigned char)image[i++];
      if (!isspace(ch)) cur.push_back((char)tolower(ch));
    }
    data.push_back(strdup(cur.c_str()));
  }
}

// -F (build-icm.cc:77-108): drop strings with an in-frame stop codon
static void Skip_In_Frame_Stops(std::vector<char*>& training) {
  if (Stop_Codon.empty()) Stops_By_Code(1, Stop_Codon);
  size_t kept = 0, total = training.size();
  for (size_t i = 0; i < total; i++) {
    const char* s = training[i];
    const long len = (long)strlen(s);
    bool skip = false;
    for (long j = 0; j < len - 2 && !skip; j += 3)
      for (const std::string& stop : Stop_Codon)
        if (strncmp(s + j, stop.c_str(), 3) == 0) { skip = true; break; }
    if (!skip) training[kept++] = training[i];
  }
  fprintf(stderr, "Skipped %d strings with in-frame stops of %d total strings\n", (int)(total - kept), (int)total);
  training.resize(kept);
}

// the whole stream into page-locked memory (free with gmg_host_free)
static char* Read_Image(FILE* fp, size_t* n) {
  size_t cap = (size_t)64 << 20, used = 0;
  char* image = NULL;
  GMG_OR_DIE(gmg_host_alloc(cap, (void**)&image));
  for (;;) {
    if (used == cap) {
      char* bigger = NULL;
      GMG_OR_DIE(gmg_host_alloc(cap * 2, (void**)&bigger));
      memcpy(bigger, image, used);
      gmg_host_free(image);
      image = bigger;
      cap *= 2;
    }
    const size_t got = fread(image + used, 1, cap - used, fp);
    if (got == 0) break;
    used += got;
  }
  *n = used;
  return image;
}

// -B: read and check every input (the single-model ingest per file), then train all models with one
// gmg_icm_train_many call and write each output.  An input without data stops the run before anything is written.
static int Build_Batch(const char* list_path) {
  FILE* lf = fopen(list_path, "r");
  if (lf == NULL) {
    fprintf(stderr, "ERROR:  Could not open file  %s \n", list_path);
    return EXIT_FAILURE;
  }
  std::vector<std::string> in_names, out_names;
  char line[8192];
  for (int line_no = 1; fgets(line, sizeof line, lf) != NULL; line_no++) {
    char a[4096], b[4096], extra[2];
    const int got = sscanf(line, "%4095s %4095s %1s", a, b, extra);
    if (got <= 0) continue;  // blank line
    if (got != 2) {
      fprintf(stderr, "ERROR:  %s line %d: expected  input_fasta output_file\n", list_path, line_no);
      fclose(lf);
      return EXIT_FAILURE;
    }
    in_names.push_back(a);
    out_names.push_back(b);
  }
  fclose(lf);
  if (in_names.empty()) {
    fprintf(stderr, "ERROR:  Cannot create model--no input data\n  (%s lists no input files)\n", list_path);
    return EXIT_FAILURE;
  }
  std::vector<gmg_seqset*> sets;
  std::vector<int64_t> n_strings;
  for (size_t k = 0; k < in_names.size(); k++) {
    FILE* fp = fopen(in_names[k].c_str(), "rb");
    if (fp == NULL) {
      fprintf(stderr, "ERROR:  Could not open file  %s \n", in_names[k].c_str());
      return EXIT_FAILURE;
    }
    size_t used = 0;
    char* image = Read_Image(fp, &used);
    fclose(fp);
    gmg_seqset* ss = NULL;
    int64_t n = 0;
    if (!Skip_In_Frame_Stop_Strings && used < ((size_t)1 << 30)) {
      GMG_OR_DIE(gmg_seqset_from_fasta(Gmg_Context(), image, (int64_t)used, &ss, &n));
      GMG_OR_DIE(gmg_ctx_sync(Gmg_Context()));  // the parse has read `image`
    } else {
      std::vector<char*> training;
      Read_Training_Data(image, used, training);
      const std::vector<char*> all = training;
      n = (int64_t)training.size();  // checked before -F, as for a single model
      if (n > 0) {
        if (Skip_In_Frame_Stop_Strings) Skip_In_Frame_Stops(training);
        ss = ICM_Training_t::Seqset_Of(training);
      }
      for (char* s : all) free(s);
    }
    gmg_host_free(image);
    if (n == 0) {
      fprintf(stderr, "ERROR:  Cannot create model--no input data\n  (%s)\n", in_names[k].c_str());
      return EXIT_FAILURE;
    }
    sets.push_back(ss);
    n_strings.push_back(n);
  }
  std::vector<std::unique_ptr<ICM_Training_t>> models;
  std::vector<ICM_Training_t*> ptrs;
  for (size_t k = 0; k < sets.size(); k++) {
    models.emplace_back(new ICM_Training_t(Model_Len, Model_Depth, Model_Periodicity));
    ptrs.push_back(models.back().get());
  }
  models[0]->Train_Many(sets, Reverse_Strings ? 1 : 0, ptrs);
  for (gmg_seqset* ss : sets) gmg_seqset_free(ss);
  for (size_t k = 0; k < models.size(); k++) {
    FILE* out = fopen(out_names[k].c_str(), Print_Binary ? "wb" : "w");
    if (out == NULL) {
      fprintf(stderr, "ERROR:  Could not open file  %s \n", out_names[k].c_str());
      return EXIT_FAILURE;
    }
    if (Verbose > 0) fprintf(stderr, "%s: trained on %lld strings\n", in_names[k].c_str(), (long long)n_strings[k]);
    models[k]->Output(out, Print_Binary);
    fclose(out);
  }
  return 0;
}

int main(int argc, char** argv) {
  bool err = false;
  int ch;
  static struct option long_options[] = {{"depth", 1, 0, 'd'},  {"no_stops", 0, 0, 'F'}, {"help", 0, 0, 'h'},
                                         {"period", 1, 0, 'p'}, {"reverse", 0, 0, 'r'},  {"text", 0, 0, 't'},
                                         {"verbose", 1, 0, 'v'}, {"width", 1, 0, 'w'},   {"trans_table", 1, 0, 'z'},
                                         {"stop_codons", 1, 0, 'Z'}, {"batch", 1, 0, 'B'}, {0, 0, 0, 0}};
  while (!err && (ch = getopt_long(argc, argv, "B:d:Fhp:rtv:w:z:Z:", long_options, NULL)) != EOF) switch (ch) {
      case 'B': Batch_List = optarg; break;
      case 'd':
        if (!Number(optarg, &Model_Depth, true)) { fprintf(stderr, "Bad model depth value \"%s\"\n", optarg); err = true; }
        break;
      case 'F': Skip_In_Frame_Stop_Strings = true; break;
      case 'h': err = true; break;
      case 'p':
        if (!Number(optarg, &Model_Periodicity, true)) { fprintf(stderr, "Bad model period value \"%s\"\n", optarg); err = true; }
        break;
      case 'r': Reverse_Strings = true; break;
      case 't': Print_Binary = false; break;
      case 'v':
        if (!Number(optarg, &Verbose, false)) { fprintf(stderr, "Bad verbose value \"%s\"\n", optarg); err = true; }
        break;
      case 'w':
        if (!Number(optarg, &Model_Len, true)) { fprintf(stderr, "Bad model length value \"%s\"\n", optarg); err = true; }
        break;
      case 'z': {
        int code = 0;
        if (!Number(optarg, &code, false) || !Stops_By_Code(code, Stop_Codon)) {
          fprintf(stderr, "Bad translation table code \"%s\"\n", optarg);
          err = true;
        }
        break;
      }
      case 'Z': {
        Stop_Codon.clear();
        for (char* p = strtok(optarg, ","); p != NULL; p = strtok(NULL, ",")) {
          std::string s(p);
          for (char& c : s) c = (char)tolower(c);
          Stop_Codon.push_back(s);
        }
        break;
      }
      case '?': fprintf(stderr, "Unrecognized option -%c\n", optopt);  // fall through
      default: err = true;
    }
  if (err || optind != argc - (Batch_List ? 0 : 1)) {
    Usage();
    exit(EXIT_FAILURE);
  }
  if (Batch_List) return Build_Batch(Batch_List);
  const char* out_name = argv[optind];
  FILE* out = strcmp(out_name, "-") == 0 ? stdout : fopen(out_name, Print_Binary ? "wb" : "w");
  if (out == NULL) {
    fprintf(stderr, "ERROR:  Could not open file  %s \n", out_name);
    exit(EXIT_FAILURE);
  }

  ICM_Training_t model(Model_Len, Model_Depth, Model_Periodicity);
  int64_t n_strings = 0;
  size_t used = 0;
  char* image = Read_Image(stdin, &used);
  if (!Skip_In_Frame_Stop_Strings && used < ((size_t)1 << 30)) {
    // parsed, lower-cased and packed on the device (gmg_seqset_from_fasta)
    n_strings = model.Train_Fasta(image, (int64_t)used, Reverse_Strings ? 1 : 0, NULL, NULL);
    gmg_host_free(image);
    if (n_strings == 0) {
      fprintf(stderr, "ERROR:  Cannot create model--no input data\n");
      fclose(out);
      exit(EXIT_FAILURE);
    }
  } else {
  std::vector<char*> training;
  Read_Training_Data(image, used, training);
  gmg_host_free(image);
  if (training.empty()) {
    fprintf(stderr, "ERROR:  Cannot create model--no input data\n");
    fclose(out);
    exit(EXIT_FAILURE);
  }
  if (Skip_In_Frame_Stop_Strings) Skip_In_Frame_Stops(training);
  // -r: the device reads the packed strings back to front instead of reversing them on the host
  model.Train_Strings(training, Reverse_Strings ? 1 : 0, NULL, NULL);
  n_strings = (int64_t)training.size();
  }
  if (Verbose > 0) fprintf(stderr, "trained on %lld strings\n", (long long)n_strings);
  model.Output(out, Print_Binary);
  if (out != stdout) fclose(out);
  return 0;
}
