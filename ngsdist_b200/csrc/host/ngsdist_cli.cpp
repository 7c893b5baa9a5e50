// ngsDist drop-in command line on top of libngsdist_b200.so.
//
// Same flags, input formats and `.dist` layout as the reference's main() (ngsDist.cpp:29-320, parse_args.cpp:52-221):
// this file is the host side that stays C++ -- option parsing, the readers' tokenising rules, labels, the host RNG
// stream and the writer -- and it hands RAW values to the CUDA hot path through the C ABI (include/ngsdist_b200.h).
// The readers, labels, RNG stream and writer are written from the behaviour documented in SURVEY.md §3/App. E.  ONE
// block restates the reference on purpose: parse_args() below reproduces the option table, the getopt string, the banner
// format and the nine validation messages of /root/reference/parse_args.cpp:54-83,167-220 -- they are the flag schema
// and the user-visible strings a drop-in must keep.  The reference is GPL-3 (its LICENSE); see LICENSE-NOTE.md.
//
// Differences on purpose (documented in DESIGN.md): text lines may be longer than the reference's 500 000-character
// buffer; input is streamed in chunks (the whole data set is never held on the host); --verbose >= 5 per-site dumps are
// not produced; additive flags: --device N (first GPU), --tree FILE (a neighbour-joining tree per matrix, and FILE.support with bootstrap support values),
// --nni_bme (with --tree: balanced minimum-evolution trees refined from the neighbour-joining ones), --n_gpus N and
// --shard auto|replicated|sites (multi-GPU inside
// the library, SURVEY §8e).  The tail of gen_dist (ngsDist.cpp:372-386: division, -log(1-d), JC69) runs HERE with the
// host's libm on the raw distance the device returns, so that the written values are the reference's to the last digit.
#include <fcntl.h>
#include <getopt.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>
#include <zlib.h>

#include <condition_variable>
#include <mutex>
#include <algorithm>
#include <functional>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/ngsdist_b200.h"
#include "fast_io.h"

static const char *kVersion = "1.0.10-b200";

struct Pars {
  const char *in_geno = nullptr;
  bool in_bin = false, in_probs = false, in_logscale = false;
  uint64_t n_ind = 0, n_sites = 0, tot_sites = 0;
  const char *in_labels = nullptr; bool in_labels_header = false;
  const char *in_pos = nullptr; bool in_pos_header = false;
  bool call_geno = false; double N_thresh = 0, call_thresh = 0;
  bool pairwise_del = false;
  double score[9] = {0, 0.5, 1, 0.5, 0, 0.5, 1, 0.5, 0};
  uint64_t evol_model = 1;
  bool indep_geno = false;
  uint64_t n_boot_rep = 0, boot_block_size = 1;
  const char *out = nullptr;
  unsigned n_threads = 1, verbose = 1, seed = 0;
  int device = 0, n_gpus = 1, shard = 0;
  const char *tree = nullptr;   // --tree FILE: one neighbour-joining tree (Newick) per matrix
  bool nni_bme = false;         // --nni_bme: with --tree, refine each tree by balanced minimum-evolution NNIs (ngsd_bme_tree)
};

// error(): same shape as the reference's (shared/gen_func.cpp:12-18): banner on stderr, perror, exit(-1)
[[noreturn]] static void die(const char *func, const char *msg) {
  fflush(stdout);
  fprintf(stderr, "\n=====\nERROR: [%s] %s\n=====\n\n", func, msg);
  perror("\t");
  fflush(stderr);
  exit(-1);
}

static const char *kModels[] = {"Raw p-distance", "Log transf. p-distance", "JC69", "K80", "F81", "HKY85/F84", "TN93"};

static bool is_vcf_name(const char *name) {
  const size_t len = name ? strlen(name) : 0;
  return (len > 7 && strcmp(name + len - 7, ".vcf.gz") == 0) || (len > 4 && strcmp(name + len - 4, ".vcf") == 0);
}

static void parse_args(Pars *p, int argc, char **argv) {
  static struct option lopts[] = {
      {"geno", required_argument, nullptr, 'g'},       {"probs", no_argument, nullptr, 'p'},
      {"log_scale", no_argument, nullptr, 'l'},        {"n_ind", required_argument, nullptr, 'n'},
      {"n_sites", required_argument, nullptr, 's'},    {"tot_sites", required_argument, nullptr, 'S'},
      {"labels", required_argument, nullptr, 'L'},     {"labelsH", required_argument, nullptr, 'H'},
      {"pos", required_argument, nullptr, 'a'},        {"posH", required_argument, nullptr, 'A'},
      {"call_geno", no_argument, nullptr, 'c'},        {"N_thresh", required_argument, nullptr, 'N'},
      {"call_thresh", required_argument, nullptr, 'C'}, {"pairwise_del", no_argument, nullptr, 'D'},
      {"avg_nuc_dist", no_argument, nullptr, 'd'},     {"evol_model", required_argument, nullptr, 'm'},
      {"indep_geno", no_argument, nullptr, 'I'},       {"n_boot_rep", required_argument, nullptr, 'b'},
      {"boot_block_size", required_argument, nullptr, 'B'}, {"out", required_argument, nullptr, 'o'},
      {"n_threads", required_argument, nullptr, 'x'},  {"verbose", required_argument, nullptr, 'V'},
      {"seed", required_argument, nullptr, 'r'},       {"device", required_argument, nullptr, 1000},
      {"n_gpus", required_argument, nullptr, 1001},    {"shard", required_argument, nullptr, 1002},
      {"tree", required_argument, nullptr, 1003},      {"nni_bme", no_argument, nullptr, 1004},
      {nullptr, 0, nullptr, 0}};
  p->seed = (unsigned) time(nullptr);
  int c;
  while ((c = getopt_long_only(argc, argv, "g:pln:s:S:a:A:L:H:cN:C:Ddm:Ib:B:o:x:V:r:", lopts, nullptr)) != -1) {
    switch (c) {
      case 'g': p->in_geno = optarg; break;
      case 'p': p->in_probs = true; break;
      case 'l': p->in_logscale = true; p->in_probs = true; break;
      case 'n': p->n_ind = (uint64_t) atol(optarg); break;
      case 's': p->n_sites = (uint64_t) atol(optarg); break;
      case 'S': p->tot_sites = (uint64_t) atol(optarg); break;
      case 'L': p->in_labels = optarg; p->in_labels_header = false; break;
      case 'H': p->in_labels = optarg; p->in_labels_header = true; break;
      case 'a': p->in_pos = optarg; p->in_pos_header = false; break;
      case 'A': p->in_pos = optarg; p->in_pos_header = true; break;
      case 'c': p->call_geno = true; break;
      case 'N': p->N_thresh = atof(optarg); p->call_geno = true; break;
      case 'C': p->call_thresh = atof(optarg); p->call_geno = true; break;
      case 'D': p->pairwise_del = true; break;
      case 'd': p->score[4] = 0.5; break;
      case 'm': p->evol_model = (uint64_t) atol(optarg); break;
      case 'I': p->indep_geno = true; break;
      case 'b': p->n_boot_rep = (uint64_t) atol(optarg); break;
      case 'B': p->boot_block_size = (uint64_t) atol(optarg); break;
      case 'o': p->out = optarg; break;
      case 'x': p->n_threads = (unsigned) atoi(optarg); break;
      case 'V': p->verbose = (unsigned) atoi(optarg); break;
      case 'r': p->seed = (unsigned) atoi(optarg); break;
      case 1000: p->device = atoi(optarg); break;
      case 1001: p->n_gpus = atoi(optarg); break;
      case 1003: p->tree = optarg; break;
      case 1004: p->nni_bme = true; break;
      case 1002:
        if (strcmp(optarg, "auto") == 0) p->shard = NGSD_SHARD_AUTO;
        else if (strcmp(optarg, "replicated") == 0) p->shard = NGSD_SHARD_REPLICATED;
        else if (strcmp(optarg, "sites") == 0) p->shard = NGSD_SHARD_SITES;
        else die("parse_cmd_args", "--shard takes auto, replicated or sites!");
        break;
      default: exit(-1);
    }
  }
  if (is_vcf_name(p->in_geno)) p->in_probs = p->in_logscale = true;   // a VCF holds log-scale likelihoods whatever the flags say
  if (p->verbose >= 1) {
    fprintf(stderr, "==> Input Arguments:\n");
    fprintf(stderr,
            "\tgeno: %s\n\tprobs: %s\n\tlog_scale: %s\n\tn_ind: %lu\n\tn_sites: %lu\n\ttot_sites: %lu\n\tlabels: %s (%s header)\n"
            "\tpositions: %s (%s header)\n\tcall_geno: %s\n\tN_thresh: %f\n\tcall_thresh: %f\n\tpairwise_del: %s\n\tavg_nuc_dist: %s\n"
            "\tevol_model: %s\n\tgeno_indep: %s\n\tn_boot_rep: %lu\n\tboot_block_size: %lu\n\tout: %s\n\tn_threads: %d\n\tverbose: %d\n"
            "\tseed: %d\n\tversion: %s (CUDA sm_100a, device %d)\n\n",
            p->in_geno, p->in_probs ? "true" : "false", p->in_logscale ? "true" : "false", p->n_ind, p->n_sites, p->tot_sites,
            p->in_labels, p->in_labels_header ? "WITH" : "WITHOUT", p->in_pos, p->in_pos_header ? "WITH" : "WITHOUT",
            p->call_geno ? "true" : "false", p->N_thresh, p->call_thresh, p->pairwise_del ? "true" : "false",
            p->score[4] == 0.5 ? "true" : "false", p->evol_model <= 6 ? kModels[p->evol_model] : "?", p->indep_geno ? "true" : "false",
            p->n_boot_rep, p->boot_block_size, p->out, p->n_threads, p->verbose, p->seed, kVersion, p->device);
  }
  if (p->verbose > 4)
    fprintf(stderr, "==> Verbose values greater than 4 for debugging purpose only. Expect large amounts of info on screen\n");
  // the checks of parse_args.cpp:203-220, same order and messages
  if (p->in_geno == nullptr) die("parse_cmd_args", "genotype input file (--geno) missing!");
  if (p->n_ind == 0) die("parse_cmd_args", "number of individuals (--n_ind) missing!");
  if (p->n_sites == 0) die("parse_cmd_args", "number of sites (--n_sites) missing!");
  if (p->tot_sites > 0 && p->pairwise_del)
    die("parse_cmd_args", "cannot specify total number of sites (--tot_sites) with pairwise deletion (--pairwise_del)!");
  if (p->call_geno && !p->in_probs) die("parse_cmd_args", "can only call genotypes from likelihoods/probabilities!");
  if (p->evol_model > 6) die("parse_cmd_args", "invalid correction method specified!");
  if (p->evol_model > 2 && p->in_pos == nullptr)
    die("parse_cmd_args", "use of more complex evolutionary models requires position information!");
  if (p->out == nullptr) die("parse_cmd_args", "output prefix (--out) missing!");
  if (p->n_threads < 1) die("parse_cmd_args", "number of threads cannot be less than 1!");
  if (p->n_gpus < 1) die("parse_cmd_args", "number of GPUs (--n_gpus) cannot be less than 1!");
  if (p->nni_bme && p->tree == nullptr) die("parse_cmd_args", "balanced NNI refinement (--nni_bme) needs a tree output file (--tree)!");
}

// ---- line-oriented gz reading (labels, positions, text genotypes) --------------------------------------------

static gzFile open_gz(const char *name, const char *mode) {
  gzFile fh = strcmp(name, "-") == 0 ? gzdopen(fileno(stdin), mode) : gzopen(name, mode);
  if (fh) gzbuffer(fh, 1 << 20);
  return fh;
}

// one line of any length, trailing "\n" / "\r\n" removed; false at end of file
static bool read_line(gzFile fh, std::string &line) {
  line.clear();
  char buf[65536];
  bool got = false;
  while (gzgets(fh, buf, sizeof(buf)) != nullptr) {
    got = true;
    line += buf;
    if (!line.empty() && line.back() == '\n') break;
  }
  if (!got) return false;
  while (!line.empty() && (line.back() == '\n' || line.back() == '\r')) line.pop_back();
  return true;
}

// numeric tokens of a line: separators are blanks and tabs, a token counts only if it parses completely as a double
// (shared/gen_func.cpp:390-417)
static void numeric_fields(const std::string &line, std::vector<double> &out) {
  out.clear();
  const char *s = line.c_str();
  while (*s) {
    while (*s == ' ' || *s == '\t') s++;
    if (!*s) break;
    const char *e = s;
    while (*e && *e != ' ' && *e != '\t') e++;
    double v;
    if (fastio::parse_number(s, e, &v)) out.push_back(v);
    s = e;
  }
}

static std::vector<std::string> read_labels(const Pars &p) {
  std::vector<std::string> lab;
  if (!p.in_labels) {
    for (uint64_t i = 0; i < p.n_ind; i++) lab.push_back("Ind_" + std::to_string(i));   // ngsDist.cpp:118-124
    return lab;
  }
  if (p.verbose >= 1) fprintf(stderr, "==> Reading labels\n");
  gzFile fh = open_gz(p.in_labels, "r");
  if (!fh) die("read_file", "cannot open file!");
  std::string line;
  uint64_t skip = p.in_labels_header ? 1 : 0;
  while (read_line(fh, line)) {
    if (line.empty() || line[0] == '#') continue;          // shared/gen_func.cpp:258-261
    if (skip) { skip--; continue; }
    size_t tab = line.find('\t');                            // cut at the first tab (ngsDist.cpp:111-116)
    lab.push_back(tab == std::string::npos ? line : line.substr(0, tab));
  }
  gzclose(fh);
  if (lab.size() != p.n_ind) die("main", "invalid LABELS file!");
  return lab;
}

static void check_positions(const Pars &p) {   // only validated, never used (models 3-6 are rejected), ngsDist.cpp:133-149
  if (!p.in_pos) return;
  if (p.verbose >= 1) fprintf(stderr, "==> Reading positions file\n");
  gzFile fh = open_gz(p.in_pos, "r");
  if (!fh) die("read_file", "cannot open file!");
  std::string line;
  uint64_t skip = p.in_pos_header ? 1 : 0, rows = 0, cols = 0;
  while (read_line(fh, line)) {
    if (line.empty() || line[0] == '#') continue;
    if (skip) { skip--; continue; }
    uint64_t n = 1;
    for (char ch : line) n += (ch == '\t');
    if (cols == 0) cols = n;
    if (cols != n) die("read_split", "invalid number of fields in file!");
    rows++;
  }
  gzclose(fh);
  if (rows != p.n_sites || cols < 2) die("main", "invalid POS file!");
}

// ---- writer (ngsDist.cpp:282-287; "%.10f" as gen_func.cpp:479-496) ------------------------------------------------

static void format_rows(const std::vector<std::string> &lab, const double *d, uint64_t n, uint64_t r0, uint64_t r1, std::string *out) {
  out->clear();
  char num[512];
  for (uint64_t i = r0; i < r1; i++) {
    out->append(lab[i]);
    for (uint64_t j = 0; j < n; j++) {
      const double v = d[i * n + j];
      num[0] = '\t';
      int len;
      if (fabs(v) < 4503599627370496.0 || !(v == v) || isinf(v)) len = 1 + fastio::fmt_fixed10(num + 1, v);
      else len = snprintf(num, sizeof(num), "\t%.10f", v);
      out->append(num, len);
    }
    out->push_back('\n');
  }
}

// One matrix in the reference's layout: "\n<n>\n" then label<TAB>v0<TAB>...<TAB>v{n-1} per row, "%.10f" values.
// Rows are formatted by n_threads threads in bands (bounded memory) and written in order.
static void write_matrix(FILE *fh, const std::vector<std::string> &lab, const double *d, uint64_t n, unsigned n_threads) {
  fprintf(fh, "\n%lu\n", n);
  const unsigned T = (unsigned) std::max<uint64_t>(1, std::min<uint64_t>(n_threads, n / 64 + 1));
  const uint64_t band = std::max<uint64_t>(1, std::min<uint64_t>(n, ((uint64_t) 64 << 20) / (n * 14 + 64) + 1));   // ~64 MB of text per round
  std::vector<std::string> parts(T);
  for (uint64_t b0 = 0; b0 < n; b0 += band) {
    const uint64_t b1 = std::min(n, b0 + band), rows = b1 - b0;
    if (T == 1) {
      format_rows(lab, d, n, b0, b1, &parts[0]);
    } else {
      std::vector<std::thread> th;
      for (unsigned t = 0; t < T; t++)
        th.emplace_back(format_rows, std::cref(lab), d, n, b0 + rows * t / T, b0 + rows * (t + 1) / T, &parts[t]);
      for (auto &x : th) x.join();
    }
    for (unsigned t = 0; t < T; t++) fwrite(parts[t].data(), 1, parts[t].size(), fh);
  }
}

// The evolutionary correction of gen_dist (ngsDist.cpp:378-386) on the raw distances d = dist / cnt the device returned,
// with the host's libm -- the same log() the reference calls -- on n_threads threads.  NaN spelling as the reference's
// x86 arithmetic gives it: 0/0 is the negative default NaN ("-nan", model 0), which -log(1 - d) turns positive ("nan").
static void apply_model(double *d, uint64_t n, uint64_t model, unsigned n_threads) {
  auto rows = [&](uint64_t r0, uint64_t r1) {
    for (uint64_t i = r0; i < r1; i++)
      for (uint64_t j = 0; j < n; j++) {
        if (i == j) continue;
        double v = d[i * n + j];
        if (v != v) v = -fabs(v);                       // whatever the device's NaN looks like: the sign x86 gives 0/0
        if (model == 1) v = -log(1 - v);
        else if (model == 2) v = -log(1 - (v * 4 / 3)) * 3 / 4;
        d[i * n + j] = v;
      }
  };
  const unsigned T = (unsigned) std::max<uint64_t>(1, std::min<uint64_t>(n_threads, n / 64 + 1));
  if (T == 1) { rows(0, n); return; }
  std::vector<std::thread> th;
  for (unsigned t = 0; t < T; t++) th.emplace_back(rows, n * t / T, n * (t + 1) / T);
  for (auto &x : th) x.join();
}

// --selftest_io N: the exact fast "%.10f" and the fast number parser against libc on N random values (no GPU needed)
static int selftest_io(uint64_t n) {
  uint64_t x = 0x9E3779B97F4A7C15ull, bad = 0;
  auto next = [&]() { x ^= x << 13; x ^= x >> 7; x ^= x << 17; return x; };
  char a[512], b[512];
  auto check = [&](double v) {
    const int la = fastio::fmt_fixed10(a, v);
    a[la] = 0;
    snprintf(b, sizeof(b), "%.10f", v);
    if (strcmp(a, b) != 0) { if (bad < 10) fprintf(stderr, "fmt mismatch: %s vs %s (%a)\n", a, b, v); bad++; }
    if (v == v) {                                   // parse back what libc prints with 17 / 10 / 6 digits
      for (const char *f : {"%.17g", "%.10f", "%.6f", "%g"}) {
        snprintf(b, sizeof(b), f, v);
        double w1 = 0, w2 = strtod(b, nullptr);
        const bool ok = fastio::parse_number(b, b + strlen(b), &w1);
        if (!ok || memcmp(&w1, &w2, 8) != 0) { if (bad < 10) fprintf(stderr, "parse mismatch on '%s'\n", b); bad++; }
      }
    }
  };
  const double specials[] = {0.0, -0.0, 1.0, 0.5, 0.25, 0.125, 1e-10, 5e-11, 0.00000000005, 1.00000000005, 2.5e-10, 0.99999999995,
                             123456.00000000005, INFINITY, -INFINITY, NAN, -NAN, 4503599627370495.5, 1e300, 1e-300, 4.9e-324, 0.1, 0.3, 2.0 / 3};
  for (double v : specials) { check(v); check(-v); }
  for (uint64_t k = 0; k < n; k++) {
    const uint64_t r = next();
    double v;
    switch (k % 6) {
      case 0: v = (double) (r >> 11) * 0x1p-53; break;                                // [0,1)
      case 1: v = (double) (r >> 11) * 0x1p-53 * 10.0; break;                         // typical distances
      case 2: v = (double) (r % 20000000001ull) * 5e-11; break;                        // near decimal half-way points
      case 3: v = ldexp((double) (r >> 11) * 0x1p-53, (int) (next() % 80) - 60); break;
      case 4: memcpy(&v, &r, 8); if (!(fabs(v) < 1e15)) v = 0.75; break;               // random bit patterns
      default: v = (double) ((int64_t) (r % 2000001) - 1000000) / 1e6; break;         // short decimals
    }
    check(v);
  }
  double w;
  const char *not_numbers[] = {"", "-", "+", ".", "abc", "1.2.3", "1e", "0x", "--1", "1-", "marker"};
  for (const char *t : not_numbers)
    if (fastio::parse_number(t, t + strlen(t), &w)) { fprintf(stderr, "parsed a non-number: '%s'\n", t); bad++; }
  fprintf(stderr, "selftest_io: %lu values, %lu mismatches\n", n, bad);
  return bad ? 1 : 0;
}

// --tree: the step the reference's workflow (README.md:83-98) runs FastME for -- one neighbour-joining tree per matrix
// (with --nni_bme: refined by balanced minimum-evolution NNIs, FastME's criterion), computed on the device from the
// matrices as written (after the host's -log / JC69 tail).  The matrices are kept until `cap` of them are held (a fixed
// host budget, at least one per GPU) and their trees are then built by one ngsd_trees_batch call, written in order.
struct TreeBatch {
  FILE *fh = nullptr;
  ngsd_ctx *ctx = nullptr;
  int32_t method = NGSD_TREE_NJ;
  uint64_t n2 = 0, cap = 1, held = 0;
  std::vector<const char *> names;
  std::vector<double> mats;
  std::vector<std::string> *keep = nullptr;

  void add(const double *d) {
    memcpy(mats.data() + held * n2, d, n2 * sizeof(double));
    if (++held == cap) flush();
  }
  void flush() {
    if (!held) return;
    std::vector<uint64_t> offsets(held + 1);
    std::vector<int32_t> status(held);
    std::vector<char> buf(held * (64 * names.size() + 1024));
    int rc = ngsd_trees_batch(ctx, mats.data(), held, method, names.data(), buf.data(), buf.size(), offsets.data(), nullptr, status.data());
    if (rc && offsets[held] > buf.size()) {
      buf.resize(offsets[held]);
      rc = ngsd_trees_batch(ctx, mats.data(), held, method, names.data(), buf.data(), buf.size(), offsets.data(), nullptr, status.data());
    }
    if (rc) die("main", ngsd_last_error(ctx));
    for (uint64_t k = 0; k < held; k++) {
      if (status[k]) {
        fprintf(stderr, "> no tree for this matrix: it holds non-finite values (pairs without shared sites?)\n");
        fprintf(fh, "NA\n");
        keep->push_back("NA");
        continue;
      }
      const uint64_t len = offsets[k + 1] - offsets[k] - 1;
      fwrite(buf.data() + offsets[k], 1, len, fh);
      fputc('\n', fh);
      keep->emplace_back(buf.data() + offsets[k], len);
    }
    held = 0;
  }
};

// FILE.support: the main tree with, on every internal edge, the percentage of bootstrap trees that hold it -- what the
// reference's workflow gets from `raxmlHPC -f b -t main -z boots` (README.md:83-98)
static void write_support(const char *tree_path, const std::vector<std::string> &trees) {
  if (trees.size() < 2 || trees[0] == "NA") return;
  std::vector<const char *> reps;
  for (size_t k = 1; k < trees.size(); k++) reps.push_back(trees[k].c_str());
  uint64_t need = 0;
  std::vector<char> buf(2 * trees[0].size() + 64);
  int rc = ngsd_tree_support(trees[0].c_str(), reps.data(), reps.size(), 1, buf.data(), buf.size(), &need);
  if (rc && need + 1 > buf.size()) {
    buf.resize(need + 1);
    rc = ngsd_tree_support(trees[0].c_str(), reps.data(), reps.size(), 1, buf.data(), buf.size(), &need);
  }
  if (rc) {
    fprintf(stderr, "> no support values: the trees do not share one set of labels\n");
    return;
  }
  const std::string path = std::string(tree_path) + ".support";
  FILE *fh = fopen(path.c_str(), "w");
  if (!fh) die("main", "cannot open tree support output file!");
  fwrite(buf.data(), 1, need, fh);
  fputc('\n', fh);
  fclose(fh);
}

// NGSD_CLI_TIMING=1: wall-clock stamps of the phases on stderr (development aid)
static void stamp(const char *what) {
  static const bool on = getenv("NGSD_CLI_TIMING") != nullptr;
  static struct timespec t0 = {0, 0};
  if (!on) return;
  struct timespec t;
  clock_gettime(CLOCK_MONOTONIC, &t);
  if (t0.tv_sec == 0 && t0.tv_nsec == 0) t0 = t;
  fprintf(stderr, "[timing] %-28s %8.3f s\n", what, (double) (t.tv_sec - t0.tv_sec) + 1e-9 * (double) (t.tv_nsec - t0.tv_nsec));
}

int main(int argc, char **argv) {
  stamp("start");
  if (argc >= 2 && strcmp(argv[1], "--selftest_io") == 0) return selftest_io(argc >= 3 ? (uint64_t) atol(argv[2]) : 1000000);
  Pars p;
  parse_args(&p, argc, argv);
  const bool in_vcf = is_vcf_name(p.in_geno);
  const uint64_t n_comb = (uint64_t) ((pow((double) p.n_ind, 2) - p.n_ind) / 2);
  if (p.verbose >= 1) fprintf(stderr, "==> Analysis will be run in %lu combinations\n", n_comb);
  // forcing rules of ngsDist.cpp:55-65
  if (!p.in_probs && !p.indep_geno) {
    fprintf(stderr, "==> Using faster algorithm (assuming independence of genotypes) since input are genotypes!\n");
    p.indep_geno = true;
  } else if (p.call_geno && !p.indep_geno) {
    fprintf(stderr, "==> Using faster algorithm (assuming independence of genotypes) since calling genotypes!\n");
    p.indep_geno = true;
  } else if (p.indep_geno && p.verbose >= 1) {
    fprintf(stderr, "==> Using faster algorithm (assuming independence of genotypes)!\n");
  }
  // input kind (ngsDist.cpp:73-95)
  bool in_bed = false;
  if (in_vcf) {
    // Extension (SURVEY §8f N3): genotype likelihoods straight from a VCF -- FORMAT/GL (log10) or FORMAT/PL (phred) of
    // biallelic records, one site per record, samples in column order.  They enter the front end as natural-log
    // likelihoods through the text reader's --log_scale path (read_data.cpp:83-87,98), i.e. exactly as if the same
    // numbers had been written to a .gz text file and read with --probs --log_scale.
    if (p.verbose >= 1) fprintf(stderr, "==> VCF input file (FORMAT/GL or FORMAT/PL genotype likelihoods)\n");
    p.in_bin = false;
  } else if (strcmp(p.in_geno, "-") == 0) {
    if (p.verbose >= 1) fprintf(stderr, "==> Reading from STDIN (BINARY)\n");
    p.in_bin = true;
  } else {
    struct stat st;
    if (stat(p.in_geno, &st) != 0) die("main", "cannot check GENO file size!");
    const char *dot = strrchr(p.in_geno, '.');
    if (dot && strcmp(dot, ".bed") == 0) {
      // Extension (SURVEY §8f N3): a variant-major PLINK .bed holds the called genotypes at 2 bits per individual-site
      // and goes to the device as it is (ngsd_push_packed_genotypes); the reference would take it for a binary
      // likelihood file and stop at the size check below.
      if (p.verbose >= 1) fprintf(stderr, "==> PLINK .bed input file (2-bit genotypes)\n");
      if (p.in_probs) die("main", "a .bed file holds genotypes, not probabilities (--probs)!");
      in_bed = true;
      if ((uint64_t) st.st_size != 3 + p.n_sites * ((p.n_ind + 3) / 4)) die("main", "invalid/corrupt genotype input file!");
    } else if (dot && strcmp(dot, ".gz") == 0) {
      if (p.verbose >= 1) fprintf(stderr, "==> GZIP input file (never BINARY)\n");
      p.in_bin = false;
    } else {
      if (p.verbose >= 1) fprintf(stderr, "==> BINARY input file\n");
      p.in_bin = true;
      p.in_probs = true;
      if (p.n_sites != (uint64_t) st.st_size / sizeof(double) / p.n_ind / 3) die("main", "invalid/corrupt genotype input file!");
    }
  }
  std::vector<std::string> labels = read_labels(p);
  if (p.verbose >= 4)
    for (auto &l : labels) fprintf(stderr, "%s\n", l.c_str());
  check_positions(p);

  // ---- context ----
  ngsd_cfg cfg;
  ngsd_default_cfg(&cfg);
  cfg.n_ind = p.n_ind; cfg.n_sites = p.n_sites; cfg.tot_sites = p.tot_sites;
  memcpy(cfg.score, p.score, sizeof(cfg.score));
  // models 0..2: the device returns the raw distance dist / cnt (evol_model 0) and apply_model() below does
  // ngsDist.cpp:378-386 with the host's libm; models 3..6 are passed on so that ngsd_create reports them like gen_dist
  const bool host_model = p.evol_model <= 2 && !getenv("NGSD_CLI_DEVICE_MODEL");
  cfg.evol_model = host_model ? 0 : (int32_t) p.evol_model;
  cfg.n_gpus = p.n_gpus > 1 ? p.n_gpus : 0;
  cfg.shard = p.shard;
  cfg.boot_block_size = p.n_boot_rep > 0 ? p.boot_block_size : 0;
  cfg.pairwise_del = p.pairwise_del; cfg.indep_geno = p.indep_geno; cfg.call_geno = p.call_geno;
  cfg.N_thresh = p.N_thresh; cfg.call_thresh = p.call_thresh; cfg.input_is_log = p.in_logscale;
  const bool codes_input = !p.in_probs && !p.in_bin;
  cfg.input_kind = codes_input ? NGSD_INPUT_GENOTYPES : (p.in_bin ? NGSD_INPUT_BINARY_GL : NGSD_INPUT_TEXT_GL);
  cfg.device = p.device;
  ngsd_ctx *ctx = nullptr;
  if (ngsd_create(&cfg, &ctx)) die(p.evol_model > 2 ? "gen_dist" : "main", ngsd_last_error(nullptr));
  stamp("context created");

  // ---- read + front end, chunk by chunk (replaces read_geno + ngsDist.cpp:161-174) ----
  // A reader thread fills one of two pinned chunk buffers (file read / inflate, text parsing on --n_threads threads)
  // while the main thread pushes the other one through the front end: disk, parser, PCIe and GPU overlap.
  if (p.verbose >= 1) fprintf(stderr, "==> Reading genotype data\n");
  if (in_bed) {
    const int fd = open(p.in_geno, O_RDONLY);
    unsigned char magic[3] = {0, 0, 0};
    if (fd < 0 || read(fd, magic, 3) != 3) die("read_geno", "cannot open GENO file!");
    if (magic[0] != 0x6c || magic[1] != 0x1b) die("read_geno", "wrong GENO file format. Not a PLINK .bed file!");
    if (magic[2] != 0x01) die("read_geno", "wrong GENO file format. Only variant-major .bed files are supported!");
    const uint64_t stride = (p.n_ind + 3) / 4;
    uint64_t bchunk = std::max<uint64_t>(64, ((uint64_t) 64 << 20) / stride / 64 * 64);
    if (const char *e = getenv("NGSD_CLI_CHUNK")) bchunk = std::max<uint64_t>(64, (uint64_t) atol(e) / 64 * 64);
    unsigned char *buf = (unsigned char *) ngsd_host_alloc(std::min(bchunk, (p.n_sites + 63) / 64 * 64) * stride);
    if (!buf) die("main", "cannot allocate pinned host buffer");
    static const int8_t bed_codes[4] = {0, -1, 1, 2};   // fields: 00 homozygous A1, 01 missing, 10 heterozygous, 11 homozygous A2
    for (uint64_t s0 = 0; s0 < p.n_sites; s0 += bchunk) {
      const uint64_t n = std::min(bchunk, p.n_sites - s0);
      for (uint64_t got = 0; got < n * stride;) {
        const ssize_t r = read(fd, buf + got, n * stride - got);
        if (r <= 0) die("read_geno", "GENO file at premature EOF. Check GENO file and number of sites!");
        got += (uint64_t) r;
      }
      if (ngsd_push_packed_genotypes(ctx, buf, stride, bed_codes, s0, n)) die("read_geno", ngsd_last_error(ctx));
    }
    close(fd);
    ngsd_host_free(buf);
  }
  if (!in_bed) {
  gzFile fh = open_gz(p.in_geno, p.in_bin ? "rb" : "r");
  if (!fh) die("read_geno", "cannot open GENO file!");
  const uint64_t per_site = p.n_ind * 3;
  uint64_t chunk = ((uint64_t) 32 << 20) / (per_site * sizeof(double)) / 64 * 64;
  if (chunk < 64) chunk = 64;
  if (const char *e = getenv("NGSD_CLI_CHUNK")) chunk = std::max<uint64_t>(64, (uint64_t) atol(e) / 64 * 64);   // tests: force many chunks
  const uint64_t n_geno = p.in_probs ? 3 : 1;
  struct Slot {
    double *raw = nullptr;
    uint64_t *packed = nullptr;   // text posteriors that are k / 10^6 with k < 2^20 travel as 3 x 20 bits (NGSD_XFER_U20X3)
    bool packable = false;
    std::vector<int8_t> codes;
    uint64_t s0 = 0, n = 0;
    bool full = false;
  } slots[2];
  // 6-decimal text posteriors (what ANGSD -doGeno 8 writes and the reference's test inputs hold) are exactly k / 10^6:
  // 8 bytes per individual-site over PCIe instead of 24, and the device's (double) k / 1e6 is the very double strtod gave
  const bool try_pack = !p.in_bin && p.in_probs && !p.in_logscale && !getenv("NGSD_CLI_NO_PACK");
  for (auto &sl : slots) {
    if (codes_input) sl.codes.resize(chunk * p.n_ind);
    else if (!(sl.raw = (double *) ngsd_host_alloc(chunk * per_site * sizeof(double)))) die("main", "cannot allocate pinned host buffer");
    if (try_pack && !(sl.packed = (uint64_t *) ngsd_host_alloc(chunk * p.n_ind * sizeof(uint64_t)))) die("main", "cannot allocate pinned host buffer");
  }
  std::mutex mu;
  std::condition_variable cv;

  // A plain (not gzip-compressed) binary file is read with read(2) straight into the pinned buffer; zlib's transparent
  // mode (what gzopen gives the reference, read_data.cpp:24-31) is kept for stdin and for compressed binaries.
  int raw_fd = -1;
  if (p.in_bin && strcmp(p.in_geno, "-") != 0) {
    FILE *probe = fopen(p.in_geno, "rb");
    unsigned char magic[2] = {0, 0};
    const bool is_gz = probe && fread(magic, 1, 2, probe) == 2 && magic[0] == 0x1f && magic[1] == 0x8b;
    if (probe) fclose(probe);
    if (!is_gz) raw_fd = open(p.in_geno, O_RDONLY);
  }
  auto fill_binary = [&](Slot &sl) {
    const uint64_t bytes = sl.n * per_site * sizeof(double);
    uint64_t got = 0;
    while (raw_fd >= 0 && got < bytes) {
      const ssize_t r = read(raw_fd, (char *) sl.raw + got, bytes - got);
      if (r == 0) die("read_geno", "GENO file at premature EOF. Check GENO file and number of sites!");
      if (r < 0) die("read_geno", "cannot read binary GENO file. Check GENO file and number of sites!");
      got += (uint64_t) r;
    }
    while (got < bytes) {
      const unsigned want = (unsigned) ((bytes - got > (1u << 30)) ? (1u << 30) : bytes - got);
      int r = gzread(fh, (char *) sl.raw + got, want);
      if (r <= 0) {
        if (gzeof(fh)) die("read_geno", "GENO file at premature EOF. Check GENO file and number of sites!");
        die("read_geno", "cannot read binary GENO file. Check GENO file and number of sites!");
      }
      got += (uint64_t) r;
    }
  };
  bool first_data_seen = false;   // the header rule only applies before the first data line
  std::vector<std::string> lines;
  std::vector<std::vector<double>> fields;
  auto fill_text = [&](Slot &sl) {
    uint64_t s = 0;
    sl.packable = try_pack;
    while (s < sl.n) {
      // (1) sequential: the next batch of lines, at most one per site still missing
      const uint64_t want = sl.n - s;
      if (lines.size() < want) { lines.resize(want); fields.resize(want); }
      for (uint64_t k = 0; k < want; k++)
        if (!read_line(fh, lines[k])) {
          if (gzeof(fh)) die("read_geno", "GENO file at premature EOF. Check GENO file and number of sites!");
          die("read_geno", "cannot read GZip GENO file. Check GENO file and number of sites!");
        }
      // (2) parallel: tokenise + convert (the expensive part of a text input)
      const unsigned T = (unsigned) std::max<uint64_t>(1, std::min<uint64_t>(p.n_threads, want / 8 + 1));
      auto parse_range = [&](uint64_t k0, uint64_t k1) { for (uint64_t k = k0; k < k1; k++) numeric_fields(lines[k], fields[k]); };
      if (T == 1) {
        parse_range(0, want);
      } else {
        std::vector<std::thread> th;
        for (unsigned t = 0; t < T; t++) th.emplace_back(parse_range, want * t / T, want * (t + 1) / T);
        for (auto &x : th) x.join();
      }
      // (3) sequential: the reference's per-line rules, in file order
      for (uint64_t k = 0; k < want; k++) {
        const std::string &line = lines[k];
        const std::vector<double> &f = fields[k];
        if (line.empty()) {
          // consumes a site and leaves the reference's values at their -1e15 fill (read_data.cpp:58-59): (0,0,0) after
          // exp, plain missing data under --call_geno -- the front end reproduces both from this marker
          sl.packable = false;                                  // the marker is a NaN: this chunk travels as doubles
          double blank;
          const uint64_t bits = NGSD_BLANK_SITE_BITS;
          memcpy(&blank, &bits, sizeof(blank));
          for (uint64_t i = 0; i < p.n_ind; i++) {
            if (codes_input) sl.codes[s * p.n_ind + i] = (int8_t) NGSD_BLANK_SITE_CODE;
            else sl.raw[(s * p.n_ind + i) * 3 + 0] = sl.raw[(s * p.n_ind + i) * 3 + 1] = sl.raw[(s * p.n_ind + i) * 3 + 2] = blank;
          }
          s++;
          continue;
        }
        if (f.empty() || (!first_data_seen && sl.s0 + s == 0 && f.size() < p.n_ind * n_geno)) {
          fprintf(stderr, "> Header found! Skipping line...\n");
          continue;                                             // header: does not consume a site
        }
        first_data_seen = true;
        if (f.size() < p.n_ind * n_geno) die("read_geno", "wrong GENO file format. Less fields than expected!");
        const double *ptr = f.data() + (f.size() - p.n_ind * n_geno);   // last n_ind*n_geno numeric columns
        if (codes_input) {
          for (uint64_t i = 0; i < p.n_ind; i++) {
            int g = (int) ptr[i];
            if (g > 2) die("read_geno", "wrong GENO file format. Genotypes must be coded as {-1,0,1,2} !");
            sl.codes[s * p.n_ind + i] = (int8_t) (g < 0 ? -1 : g);
          }
        } else {
          memcpy(sl.raw + s * per_site, ptr, per_site * sizeof(double));
          for (uint64_t i = 0; i < p.n_ind && sl.packable; i++) {
            uint64_t w = 0;
            for (int g = 0; g < 3; g++) {
              const double v = ptr[i * 3 + g];
              const double qd = nearbyint(v * 1e6);
              if (!(v >= 0) || signbit(v) || !(qd < 1048576.0) || qd / 1e6 != v) { sl.packable = false; break; }
              w |= (uint64_t) qd << (20 * g);
            }
            sl.packed[s * p.n_ind + i] = w;
          }
        }
        s++;
      }
    }
  };
  // VCF records -> natural-log likelihood triples (see in_vcf above)
  auto parse_vcf_record = [&](const std::string &line, double *dst) {
    std::vector<const char *> col;
    col.reserve(p.n_ind + 9);
    const char *b = line.c_str();
    col.push_back(b);
    for (const char *c = b; *c; c++)
      if (*c == '\t') col.push_back(c + 1);
    if (col.size() != p.n_ind + 9) die("read_geno", "wrong VCF file format. Number of sample columns differs from --n_ind!");
    auto field_end = [](const char *c) { while (*c && *c != '\t') c++; return c; };
    for (const char *c = col[4]; c < field_end(col[4]); c++)
      if (*c == ',') die("read_geno", "wrong VCF file format. Only biallelic records are supported!");
    // position of GL / PL inside FORMAT
    int idx = -1, k = 0;
    bool phred = false;
    for (const char *c = col[8], *e = field_end(col[8]); c < e; k++) {
      const char *q = c;
      while (q < e && *q != ':') q++;
      if (q - c == 2 && c[0] == 'G' && c[1] == 'L') { idx = k; phred = false; break; }
      if (q - c == 2 && c[0] == 'P' && c[1] == 'L' && idx < 0) { idx = k; phred = true; }
      c = q + 1;
    }
    if (idx < 0) die("read_geno", "wrong VCF file format. FORMAT holds neither GL nor PL!");
    const double ln10 = 2.302585092994046;
    for (uint64_t i = 0; i < p.n_ind; i++) {
      const char *c = col[9 + i], *e = field_end(c);
      for (int f = 0; f < idx && c < e; f++) { while (c < e && *c != ':') c++; if (c < e) c++; }
      const char *fe = c;
      while (fe < e && *fe != ':') fe++;
      double v[3];
      int got = 0;
      while (c < fe && got < 3) {
        const char *q = c;
        while (q < fe && *q != ',') q++;
        if (!fastio::parse_number(c, q, &v[got])) break;
        got++;
        c = q + 1;
      }
      for (int g = 0; g < 3; g++) {
        if (got < 3) dst[i * 3 + g] = log(1.0 / 3);                      // "." = no data: equal likelihoods -> missing
        else dst[i * 3 + g] = phred ? -v[g] / 10 * ln10 : v[g] * ln10;
      }
    }
  };
  auto fill_vcf = [&](Slot &sl) {
    uint64_t s = 0;
    sl.packable = false;
    while (s < sl.n) {
      const uint64_t want = sl.n - s;
      if (lines.size() < want) lines.resize(want);
      uint64_t have = 0;
      while (have < want) {
        if (!read_line(fh, lines[have])) {
          if (gzeof(fh)) die("read_geno", "GENO file at premature EOF. Check GENO file and number of sites!");
          die("read_geno", "cannot read GZip GENO file. Check GENO file and number of sites!");
        }
        if (lines[have].empty() || lines[have][0] == '#') continue;       // meta lines and the #CHROM header
        have++;
      }
      const unsigned T = (unsigned) std::max<uint64_t>(1, std::min<uint64_t>(p.n_threads, want / 8 + 1));
      auto range = [&](uint64_t k0, uint64_t k1) { for (uint64_t k = k0; k < k1; k++) parse_vcf_record(lines[k], sl.raw + (s + k) * per_site); };
      if (T == 1) {
        range(0, want);
      } else {
        std::vector<std::thread> th;
        for (unsigned t = 0; t < T; t++) th.emplace_back(range, want * t / T, want * (t + 1) / T);
        for (auto &x : th) x.join();
      }
      s += want;
    }
  };
  std::thread reader([&]() {
    int w = 0;
    for (uint64_t s0 = 0; s0 < p.n_sites; s0 += chunk, w ^= 1) {
      Slot &sl = slots[w];
      {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return !sl.full; });
      }
      sl.s0 = s0;
      sl.n = (p.n_sites - s0 < chunk) ? p.n_sites - s0 : chunk;
      if (p.in_bin) fill_binary(sl); else if (in_vcf) fill_vcf(sl); else fill_text(sl);
      {
        std::lock_guard<std::mutex> lk(mu);
        sl.full = true;
      }
      cv.notify_all();
    }
  });
  {
    int r = 0;
    for (uint64_t s0 = 0; s0 < p.n_sites; s0 += chunk, r ^= 1) {
      Slot &sl = slots[r];
      {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return sl.full; });
      }
      int rc = codes_input    ? ngsd_push_genotypes(ctx, sl.codes.data(), sl.s0, sl.n)
               : sl.packable ? ngsd_push_sites_packed(ctx, sl.packed, NGSD_XFER_U20X3, 1e6, sl.s0, sl.n)
                             : ngsd_push_sites(ctx, sl.raw, sl.s0, sl.n);
      if (rc) die("read_geno", ngsd_last_error(ctx));
      {
        std::lock_guard<std::mutex> lk(mu);
        sl.full = false;
      }
      cv.notify_all();
    }
  }
  reader.join();
  {  // the file must be at EOF (read_data.cpp:106-109)
    char extra;
    if (raw_fd >= 0) {
      if (read(raw_fd, &extra, 1) != 0) die("read_geno", "GENO file not at EOF. Check GENO file and number of sites!");
      close(raw_fd);
    } else {
      int r = gzread(fh, &extra, 1);
      if (!(r <= 0 && gzeof(fh))) die("read_geno", "GENO file not at EOF. Check GENO file and number of sites!");
    }
  }
  gzclose(fh);
  for (auto &sl : slots) {
    if (sl.raw) ngsd_host_free(sl.raw);
    if (sl.packed) ngsd_host_free(sl.packed);
  }
  }   // !in_bed
  if (ngsd_frontend(ctx)) die("read_geno", ngsd_last_error(ctx));
  stamp("input read + front end");

  if (p.verbose >= 2) fprintf(stderr, "==> Setting seed for random number generator\n");
  uint32_t rng[3];
  ngsd_taus_seed(rng, p.seed);                                        // gsl_rng_taus + gsl_rng_set (ngsDist.cpp:179-180)

  FILE *out_fh = fopen(p.out, "w");
  if (!out_fh) die("main", "cannot open output file!");
  std::vector<std::string> trees;                                      // --tree: the Newick strings, for FILE.support
  FILE *tree_fh = p.tree ? fopen(p.tree, "w") : nullptr;
  if (p.tree && !tree_fh) die("main", "cannot open tree output file!");
  TreeBatch tb;
  if (tree_fh) {
    const uint64_t budget = 2ull << 30, per = p.n_ind * p.n_ind * sizeof(double);   // host bytes of the held matrices
    tb.fh = tree_fh;
    tb.ctx = ctx;
    tb.method = p.nni_bme ? NGSD_TREE_BME : NGSD_TREE_NJ;
    tb.n2 = p.n_ind * p.n_ind;
    tb.cap = std::min<uint64_t>(p.n_boot_rep + 1, std::max<uint64_t>({1, (uint64_t) p.n_gpus, budget / per}));
    for (auto &l : labels) tb.names.push_back(l.c_str());
    tb.mats.resize(tb.cap * tb.n2);
    tb.keep = &trees;
  }
  static char obuf[1 << 22];
  setvbuf(out_fh, obuf, _IOFBF, sizeof(obuf));

  const uint64_t n2 = p.n_ind * p.n_ind;
  // several GPUs: the bootstrap replicates go to the library n_gpus at a time (ngsd_distances_batch deals them out and
  // every GPU returns its matrix over its own PCIe link); they are written in replicate order as the reference does
  const uint64_t round = (p.n_gpus > 1 && p.verbose < 3) ? (uint64_t) p.n_gpus : 1;
  std::vector<double> dist(n2 * round), num;
  std::vector<uint64_t> cnt;
  if (p.verbose >= 3) { num.resize(n2); cnt.resize(n2); }
  std::vector<uint32_t> counts;
  uint64_t n_sites = p.n_sites;
  for (uint64_t rep = 0; rep <= p.n_boot_rep; rep++) {
    if (rep > 0 && round > 1) {
      n_sites -= n_sites % p.boot_block_size;                         // persistent truncation (ngsDist.cpp:236)
      const uint64_t n_blocks = n_sites / p.boot_block_size, k = std::min<uint64_t>(round, p.n_boot_rep - rep + 1);
      counts.resize(std::max<uint64_t>(1, n_blocks * k));             // (n_blocks == 0: --boot_block_size > n_sites, still a non-NULL pointer)
      for (uint64_t q = 0; q < k; q++) ngsd_boot_block_counts(rng, n_blocks, counts.data() + q * n_blocks);
      if (p.verbose >= 1)
        for (uint64_t q = 0; q < k; q++) fprintf(stderr, "==> Bootstrap replicate # %lu ...\n", rep + q);
      if (ngsd_distances_batch(ctx, counts.data(), k, n_blocks, p.boot_block_size, dist.data())) die("gen_dist", ngsd_last_error(ctx));
      for (uint64_t q = 0; q < k; q++) {
        if (host_model) apply_model(dist.data() + q * n2, p.n_ind, p.evol_model, p.n_threads);
        if (p.verbose >= 2) fprintf(stderr, "> Printing distance matrix\n");
        write_matrix(out_fh, labels, dist.data() + q * n2, p.n_ind, p.n_threads);
        if (tree_fh) tb.add(dist.data() + q * n2);
      }
      rep += k - 1;
      continue;
    }
    if (p.verbose >= 1) {
      if (rep == 0) fprintf(stderr, "==> Analyzing full dataset...\n");
      else fprintf(stderr, "==> Bootstrap replicate # %lu ...\n", rep);
    }
    int rc;
    if (rep == 0) {
      rc = ngsd_distances(ctx, nullptr, 0, 1, dist.data(), num.empty() ? nullptr : num.data(), cnt.empty() ? nullptr : cnt.data());
    } else {
      n_sites -= n_sites % p.boot_block_size;                         // persistent truncation (ngsDist.cpp:236)
      const uint64_t n_blocks = n_sites / p.boot_block_size;
      counts.resize(std::max<uint64_t>(1, n_blocks));                 // non-NULL even for zero blocks: NULL means replicate 0
      ngsd_boot_block_counts(rng, n_blocks, counts.data());           // the draws of rnd_map_data (ngsDist.cpp:421-423)
      rc = ngsd_distances(ctx, counts.data(), n_blocks, p.boot_block_size, dist.data(), num.empty() ? nullptr : num.data(),
                          cnt.empty() ? nullptr : cnt.data());
    }
    if (rc) die("gen_dist", ngsd_last_error(ctx));
    if (p.verbose >= 3)
      for (uint64_t i1 = 0; i1 < p.n_ind; i1++)
        for (uint64_t i2 = i1 + 1; i2 < p.n_ind; i2++)
          fprintf(stderr, "\tDistance of %f from %lu valid sites (%f) between %s (ind %lu) and %s (ind %lu)!\n", num[i1 * p.n_ind + i2],
                  cnt[i1 * p.n_ind + i2], num[i1 * p.n_ind + i2] / (double) cnt[i1 * p.n_ind + i2], labels[i1].c_str(), i1,
                  labels[i2].c_str(), i2);
    if (rep == 0) stamp("first matrix computed");
    if (host_model) apply_model(dist.data(), p.n_ind, p.evol_model, p.n_threads);
    if (p.verbose >= 2) fprintf(stderr, "> Printing distance matrix\n");
    write_matrix(out_fh, labels, dist.data(), p.n_ind, p.n_threads);
    if (tree_fh) tb.add(dist.data());
  }
  fclose(out_fh);
  if (tree_fh) {
    tb.flush();
    fclose(tree_fh);
  }
  if (tree_fh && p.n_boot_rep > 0) write_support(p.tree, trees);
  stamp("all matrices written");
  if (p.verbose >= 1) fprintf(stderr, "==> Freeing memory...\n");
  ngsd_destroy(ctx);
  stamp("context destroyed");
  if (p.verbose >= 1) fprintf(stderr, "Done!\n");
  return 0;
}
