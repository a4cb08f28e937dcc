// kmerust-b200 -- command line front end with the reference's flag semantics (src/cli.rs:36-70,
// src/main.rs:34-281) on top of the GPU engine:
//   kmerust-b200 <k> [path|-] [-f fasta|tsv|json|histogram] [-m N] [-q] [-i auto|fasta|fastq] [--save X.kmix] [-Q q]
//   kmerust-b200 query <index> <kmer>
// Differences from the reference: output records come out key-sorted (the reference prints in HashMap
// order, i.e. nondeterministically), and the index is written straight from the device table.
#include <cstdlib>
#include <sys/stat.h>

#include "kmerust.hpp"

using namespace kmerust;

static void die(const std::string &head, const std::string &msg) {
  fprintf(stderr, "%s\n %s\n", head.c_str(), msg.c_str());
  exit(1);
}

static int run_query(int argc, char **argv) {
  if (argc != 4) { fprintf(stderr, "usage: %s query <index> <kmer>\n", argv[0]); return 2; }
  try {
    std::string kmer = argv[3];
    const std::string ipath = argv[2];
    if (ipath.size() >= 3 && ipath.compare(ipath.size() - 3, 3, ".gz") == 0) {  // gzip-wrapped index: host reader
      KmerIndex idx = load_index(ipath);
      for (auto &c : kmer) c = (char)toupper((unsigned char)c);
      if (kmer.size() != idx.k().get())
        die("Query error:", "k-mer length mismatch: query has " + std::to_string(kmer.size()) + " bases, index has k=" + std::to_string(idx.k().get()));
      uint64_t packed;
      try { packed = canonical_packed(kmer); } catch (const InvalidBaseError &e) { die("Invalid k-mer:", e.what()); return 1; }
      printf("%llu\n", (unsigned long long)idx.get(packed).value_or(0));
      return 0;
    }
    auto idx = open_index_on_device(ipath);  // records go to HBM, the look-up (canonicalisation included) runs there
    if (kmer.size() != idx->k().get())
      die("Query error:", "k-mer length mismatch: query has " + std::to_string(kmer.size()) + " bases, index has k=" + std::to_string(idx->k().get()));
    uint64_t bad = 0;
    const std::vector<uint64_t> got = idx->query({kmer}, &bad);
    if (bad) { try { canonical_packed(kmer); } catch (const InvalidBaseError &e) { die("Invalid k-mer:", e.what()); } return 1; }
    printf("%llu\n", (unsigned long long)got[0]);
  } catch (const KmeRustError &e) {
    die("Failed to load index:", e.what());
  }
  return 0;
}

int main(int argc, char **argv) {
  if (argc > 1 && std::string(argv[1]) == "query") return run_query(argc, argv);
  size_t k = 0;
  bool have_k = false, quiet = false;
  std::string path = "-", save;
  OutputFormat format = OutputFormat::Fasta;
  SequenceFormat input_format = SequenceFormat::Auto;
  uint64_t min_count = 1;
  std::optional<uint8_t> min_quality;
  int positional = 0;
  auto need = [&](int &i) -> std::string { if (i + 1 >= argc) { fprintf(stderr, "error: %s needs a value\n", argv[i]); exit(2); } return argv[++i]; };
  for (int i = 1; i < argc; ++i) {
    std::string a = argv[i];
    if (a == "-f" || a == "--format") {
      std::string v = need(i);
      if (v == "fasta") format = OutputFormat::Fasta; else if (v == "tsv") format = OutputFormat::Tsv;
      else if (v == "json") format = OutputFormat::Json; else if (v == "histogram") format = OutputFormat::Histogram;
      else { fprintf(stderr, "error: invalid value '%s' for '--format'\n", v.c_str()); return 2; }
    } else if (a == "-m" || a == "--min-count") min_count = strtoull(need(i).c_str(), nullptr, 10);
    else if (a == "-q" || a == "--quiet") quiet = true;
    else if (a == "-i" || a == "--input-format") {
      std::string v = need(i);
      if (v == "auto") input_format = SequenceFormat::Auto; else if (v == "fasta") input_format = SequenceFormat::Fasta;
      else if (v == "fastq") input_format = SequenceFormat::Fastq;
      else { fprintf(stderr, "error: invalid value '%s' for '--input-format'\n", v.c_str()); return 2; }
    } else if (a == "--save") save = need(i);
    else if (a == "-Q" || a == "--min-quality") {
      long q = strtol(need(i).c_str(), nullptr, 10);
      if (q < 0 || q > 255) { fprintf(stderr, "error: invalid value for '--min-quality'\n"); return 2; }
      min_quality = (uint8_t)q;
    } else if (a == "-h" || a == "--help") {
      printf("usage: %s <k> [path|-] [-f fasta|tsv|json|histogram] [-m N] [-q] [-i auto|fasta|fastq] [--save PATH] [-Q q]\n       %s query <index> <kmer>\n", argv[0], argv[0]);
      return 0;
    } else if (a.size() > 1 && a[0] == '-' && a != "-") { fprintf(stderr, "error: unexpected argument '%s'\n", a.c_str()); return 2; }
    else if (positional == 0) {
      char *end = nullptr;
      unsigned long long v = strtoull(a.c_str(), &end, 10);
      if (!end || *end || a.empty()) { fprintf(stderr, "error: invalid value '%s' for '<K>': '%s' is not a valid number\n", a.c_str(), a.c_str()); return 2; }
      if (v == 0) { fprintf(stderr, "error: invalid value '%s' for '<K>': k-mer length must be at least 1\n", a.c_str()); return 2; }   // src/cli.rs:103-114
      if (v > 32) { fprintf(stderr, "error: invalid value '%s' for '<K>': k-mer length must be at most 32\n", a.c_str()); return 2; }
      k = (size_t)v; have_k = true; ++positional;
    } else if (positional == 1) { path = a; ++positional; }
    else { fprintf(stderr, "error: unexpected argument '%s'\n", a.c_str()); return 2; }
  }
  if (!have_k) { fprintf(stderr, "error: the following required arguments were not provided:\n  <K>\n"); return 2; }
  if (path != "-") {
    struct stat sb;
    if (stat(path.c_str(), &sb) != 0) die("Problem with arguments:", "File not found: " + path);  // src/main.rs:58-67
  }
  const SequenceFormat resolved = resolve_format(input_format, path == "-" ? nullptr : &path);
  if (!quiet) {
    fprintf(stderr, "k-length: %zu\ndata: %s\ninput-format: %s%s\nreader: kmerust-b200 host\noutput-format: %s\n", k,
            path == "-" ? "stdin" : path.c_str(), resolved == SequenceFormat::Fastq ? "fastq" : "fasta",
            input_format == SequenceFormat::Auto ? " (auto-detected)" : "",
            format == OutputFormat::Fasta ? "fasta" : format == OutputFormat::Tsv ? "tsv" : format == OutputFormat::Json ? "json" : "histogram");
    if (min_count > 1) fprintf(stderr, "min-count: %llu\n", (unsigned long long)min_count);
    if (min_quality) fprintf(stderr, "min-quality: %u\n", (unsigned)*min_quality);
    if (!save.empty()) fprintf(stderr, "save-index: %s\n", save.c_str());
    fprintf(stderr, "\n");
  }
  if (min_quality && resolved == SequenceFormat::Fasta) fprintf(stderr, "warning: --min-quality is ignored for FASTA input\n");
  try {
    const KmerLength kl = KmerLength::create(k);
    GpuKmerCounter counter(kl, min_quality);
    const bool is_fastq = resolved == SequenceFormat::Fastq;
    if (path == "-") {  // stdin and .gz files stream through the device parser, in host memory bounded by its staging ring
      struct stat sb;
      const uint64_t hint = fstat(fileno(stdin), &sb) == 0 && S_ISREG(sb.st_mode) ? (uint64_t)sb.st_size : 0;
      counter.count_stream(stdin, is_fastq, hint);
    } else if (ends_with(lower(path), ".gz")) {
      gzFile g = gzopen(path.c_str(), "rb");
      if (!g) throw SequenceReadError("failed to read sequences from '" + path + "'");
      gzbuffer(g, 1u << 20);
      try { counter.count_stream(g, is_fastq); } catch (...) { gzclose(g); throw; }
      gzclose(g);
    } else {  // file image -> device parser; refused inputs (multi-line FASTQ ...) take the host splitter
      const std::vector<uint8_t> image = slurp(path);
      if (!counter.count_file_image(image.data(), image.size(), is_fastq)) counter.count(read_with_quality(path, resolved));
    }
    kmg_summary s = counter.finalize();
    if (!save.empty()) {  // the index holds ALL k-mers; --min-count only filters stdout (src/main.rs:155-212)
      try { counter.save_kmix(save); } catch (const KmeRustError &e) { die("Failed to save index:", e.what()); }
      if (!quiet) fprintf(stderr, "saved: %s (%llu k-mers)\n", save.c_str(), (unsigned long long)s.n_distinct);
    }
    std::ios::sync_with_stdio(false);
    if (format == OutputFormat::Histogram) {
      for (auto &kv : counter.histogram(min_count)) std::cout << kv.first << '\t' << kv.second << '\n';
    } else {
      std::cout.flush();
      counter.write_text("-", format, min_count);  // fasta / tsv / json records are formatted on the device
    }
    std::cout.flush();
  } catch (const KmeRustError &e) {
    die("Application error:", e.what());
  }
  return 0;
}
