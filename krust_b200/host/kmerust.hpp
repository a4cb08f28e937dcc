// kmerust.hpp -- C++ host side above the C ABI (include/kmerust_gpu.h), mirroring the reference's
// library interface for the counting path: same names, argument meaning and error behaviour
// (the reference is compiled Rust; no Rust toolchain exists in this image, so the host that a
// Rust `kmerust-gpu` wrapper crate would be is written in C++ -- INTEGRATION.md shows the Rust
// binding).  Citations are into the kmerust repository.  Header-only; link with -lkmerust_gpu.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iostream>
#include <map>
#include <memory>
#include <optional>
#include <sstream>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include <zlib.h>

#include "../../include/kmerust_gpu.h"

namespace kmerust {

// ---- errors (src/error.rs) ---------------------------------------------------------------------
struct KmeRustError : std::runtime_error { using std::runtime_error::runtime_error; };
struct KmerLengthError : KmeRustError {  // src/error.rs:88-97
  size_t k; uint8_t min, max;
  KmerLengthError(size_t k_, uint8_t mn, uint8_t mx)
      : KmeRustError("k-mer length " + std::to_string(k_) + " is out of range (must be " + std::to_string(mn) + "-" + std::to_string(mx) + ")"),
        k(k_), min(mn), max(mx) {}
};
struct InvalidBaseError : KmeRustError {  // src/error.rs:99-110
  uint8_t base; size_t position;
  InvalidBaseError(uint8_t b, size_t p) : KmeRustError("invalid base '" + std::string(1, (char)b) + "' at position " + std::to_string(p)), base(b), position(p) {}
};
struct SequenceParseError : KmeRustError { using KmeRustError::KmeRustError; };   // src/error.rs:27-30
struct SequenceReadError : KmeRustError { using KmeRustError::KmeRustError; };    // src/error.rs:20-26
struct InvalidIndexError : KmeRustError { using KmeRustError::KmeRustError; };    // src/error.rs:62-70
struct IndexIoError : KmeRustError { using KmeRustError::KmeRustError; };
struct BuilderError : KmeRustError { using KmeRustError::KmeRustError; };         // src/error.rs:159
struct GpuError : KmeRustError {
  kmg_status status;
  GpuError(kmg_status s, const std::string &m) : KmeRustError(m), status(s) {}
};

// ---- KmerLength (src/kmer.rs:74-145) -------------------------------------------------------------
class KmerLength {
  uint8_t k_;
  explicit KmerLength(uint8_t k) : k_(k) {}
 public:
  static constexpr uint8_t MIN = 1, MAX = 32;
  static KmerLength create(size_t k) {
    if (k < MIN || k > MAX) throw KmerLengthError(k, MIN, MAX);
    return KmerLength((uint8_t)k);
  }
  size_t get() const { return k_; }
  uint8_t as_u8() const { return k_; }
  bool operator==(const KmerLength &o) const { return k_ == o.k_; }
};

// src/kmer.rs:431-456
inline std::string unpack_to_string(uint64_t bits, KmerLength k) {
  std::string s(k.get(), 'A');
  for (size_t i = 0; i < k.get(); ++i) s[i] = "ACGT"[(bits >> (2 * (k.get() - 1 - i))) & 3];
  return s;
}

// from_sub + pack + canonical for ONE query k-mer (src/kmer.rs:266-390); used by `query` only -- the
// counting path does this on the GPU.
inline uint64_t canonical_packed(const std::string &kmer) {
  uint64_t fwd = 0, rc = 0;
  const size_t k = kmer.size();
  for (size_t i = 0; i < k; ++i) {
    int c;
    switch (kmer[i]) {
      case 'A': case 'a': c = 0; break;
      case 'C': case 'c': c = 1; break;
      case 'G': case 'g': c = 2; break;
      case 'T': case 't': c = 3; break;
      default: throw InvalidBaseError((uint8_t)kmer[i], i);
    }
    fwd = (fwd << 2) | (uint64_t)c;
    rc |= (uint64_t)(3 - c) << (2 * i);
  }
  return fwd < rc ? fwd : rc;
}

// ---- formats (src/format.rs, src/cli.rs) ------------------------------------------------------------
enum class SequenceFormat { Auto, Fasta, Fastq };
enum class OutputFormat { Fasta, Tsv, Json, Histogram };

inline std::string lower(std::string s) { for (auto &c : s) c = (char)tolower((unsigned char)c); return s; }
inline bool ends_with(const std::string &s, const std::string &suf) { return s.size() >= suf.size() && s.compare(s.size() - suf.size(), suf.size(), suf) == 0; }

inline SequenceFormat format_from_extension(const std::string &path) {  // src/format.rs:47-70
  std::string name = lower(path.substr(path.find_last_of('/') == std::string::npos ? 0 : path.find_last_of('/') + 1));
  if (ends_with(name, ".gz")) name.resize(name.size() - 3);
  const size_t dot = name.find_last_of('.');
  const std::string ext = dot == std::string::npos ? "" : name.substr(dot + 1);
  return (ext == "fq" || ext == "fastq") ? SequenceFormat::Fastq : SequenceFormat::Fasta;
}
inline SequenceFormat resolve_format(SequenceFormat f, const std::string *path) {  // src/format.rs:97-102
  if (f != SequenceFormat::Auto) return f;
  return path ? format_from_extension(*path) : SequenceFormat::Fasta;
}

// ---- reader stand-in (src/reader.rs:167-247): whole input -> records laid back to back ----------------
struct Records {
  std::vector<uint8_t> seq, qual;
  std::vector<uint64_t> offsets{0};
  bool has_qual = false;
  uint64_t n_records() const { return offsets.size() - 1; }
};

inline std::vector<uint8_t> slurp(const std::string &path) {
  std::vector<uint8_t> data;
  if (path == "-") {
    uint8_t buf[1 << 16];
    size_t n;
    while ((n = fread(buf, 1, sizeof buf, stdin)) > 0) data.insert(data.end(), buf, buf + n);
    return data;
  }
  if (ends_with(lower(path), ".gz")) {  // flate2::GzDecoder stand-in (src/reader.rs:102-144)
    gzFile g = gzopen(path.c_str(), "rb");
    if (!g) throw SequenceReadError("failed to read sequences from '" + path + "'");
    uint8_t buf[1 << 16];
    int n;
    while ((n = gzread(g, buf, sizeof buf)) > 0) data.insert(data.end(), buf, buf + n);
    const bool bad = n < 0;
    gzclose(g);
    if (bad) throw SequenceReadError("failed to decompress '" + path + "'");
    return data;
  }
  std::ifstream f(path, std::ios::binary | std::ios::ate);
  if (!f) throw SequenceReadError("failed to read sequences from '" + path + "'");
  const std::streamsize n = f.tellg();
  data.resize((size_t)n);
  f.seekg(0);
  if (n && !f.read(reinterpret_cast<char *>(data.data()), n)) throw SequenceReadError("failed to read sequences from '" + path + "'");
  return data;
}

inline Records parse_records(const std::vector<uint8_t> &data, bool is_fastq) {
  Records r;
  r.has_qual = is_fastq;
  r.seq.resize(data.size() + 1);
  if (is_fastq) r.qual.resize(data.size() + 1);
  uint64_t max_rec = 1;
  for (uint8_t b : data) max_rec += (b == (is_fastq ? '@' : '>'));
  r.offsets.assign(max_rec + 1, 0);
  uint64_t n = 0;
  char err[256] = {0};
  kmg_status st = kmg_parse_fastx(data.data(), data.size(), is_fastq, r.seq.data(), is_fastq ? r.qual.data() : nullptr,
                                  r.offsets.data(), max_rec, &n, err, sizeof err);
  if (st != KMG_OK) throw SequenceParseError(std::string("failed to parse sequence: ") + err);
  r.offsets.resize(n + 1);
  r.seq.resize(r.offsets.back());
  if (is_fastq) r.qual.resize(r.offsets.back());
  return r;
}

inline Records read_with_quality(const std::string &path, SequenceFormat fmt) {
  const SequenceFormat f = resolve_format(fmt, path == "-" ? nullptr : &path);
  return parse_records(slurp(path), f == SequenceFormat::Fastq);
}

// ---- the engine handle: replaces KmerMap / StreamingKmerCounter (src/run.rs:491-583) -----------------
using PackedCounts = std::unordered_map<uint64_t, uint64_t>;
using KmerHistogram = std::map<uint64_t, uint64_t>;  // src/histogram.rs:33
struct Progress { uint64_t sequences_processed, bases_processed; };  // src/progress.rs:26-31

class GpuKmerCounter {
  kmg_ctx *ctx_ = nullptr;
  KmerLength k_;
  void check(kmg_status s) const {
    if (s == KMG_OK) return;
    const char *m = kmg_last_error(ctx_);
    std::string msg = (m && *m) ? m : kmg_status_string(s);
    if (s == KMG_ERR_PARSE) throw SequenceParseError(msg);
    if (s == KMG_ERR_IO) throw IndexIoError(msg);
    throw GpuError(s, msg);
  }
 public:
  GpuKmerCounter(KmerLength k, std::optional<uint8_t> min_quality = std::nullopt, uint64_t expected_distinct = 0, uint32_t flags = 0)
      : k_(k) {
    kmg_config cfg{};
    cfg.abi_version = KMG_ABI_VERSION;
    cfg.k = (uint32_t)k.get();
    cfg.device = -1;
    cfg.flags = flags;
    cfg.has_min_quality = min_quality.has_value();
    cfg.min_quality = min_quality.value_or(0);
    cfg.expected_distinct = expected_distinct;
    kmg_status s = kmg_create(&cfg, &ctx_);
    if (s != KMG_OK) throw GpuError(s, kmg_last_error(nullptr));
  }
  ~GpuKmerCounter() { kmg_destroy(ctx_); }
  GpuKmerCounter(const GpuKmerCounter &) = delete;
  GpuKmerCounter &operator=(const GpuKmerCounter &) = delete;
  KmerLength k() const { return k_; }

  void count(const Records &r) {
    if (r.n_records() == 0) return;
    check(kmg_count_ascii(ctx_, r.seq.data(), r.has_qual ? r.qual.data() : nullptr, r.offsets.data(), r.n_records()));
  }
  void count_sequences(const std::vector<std::string> &seqs) {
    Records r;
    for (auto &s : seqs) { r.seq.insert(r.seq.end(), s.begin(), s.end()); r.offsets.push_back(r.seq.size()); }
    count(r);
  }
  kmg_summary finalize() { kmg_summary s{}; check(kmg_finalize(ctx_, &s)); return s; }
  void export_counts(uint64_t min_count, bool sorted, std::vector<uint64_t> &keys, std::vector<uint64_t> &counts) {
    uint64_t n = 0;
    check(kmg_export_counts(ctx_, min_count, sorted, nullptr, nullptr, 0, &n));
    keys.resize(n); counts.resize(n);
    if (n) check(kmg_export_counts(ctx_, min_count, sorted, keys.data(), counts.data(), n, &n));
  }
  KmerHistogram histogram(uint64_t min_count) {
    uint64_t n = 0;
    check(kmg_histogram(ctx_, min_count, nullptr, nullptr, 0, &n));
    std::vector<uint64_t> v(n), f(n);
    if (n) check(kmg_histogram(ctx_, min_count, v.data(), f.data(), n, &n));
    KmerHistogram h;
    for (uint64_t i = 0; i < n; ++i) h[v[i]] = f[i];
    return h;
  }
  // A whole FASTA / FASTQ file image: records are found on the device (kmg_count_fastx).  false: the device parser refused the
  // input (multi-line FASTQ ...) and the counter was reset -- feed it through read_with_quality() + count() instead.
  bool count_file_image(const uint8_t *bytes, uint64_t len, bool is_fastq) {
    uint64_t n = 0;
    const kmg_status s = kmg_count_fastx(ctx_, bytes, len, is_fastq, &n);
    if (s == KMG_ERR_PARSE) { check(kmg_reset(ctx_)); return false; }
    check(s);
    return true;
  }
  // A FASTA / FASTQ byte stream (stdin through fread, a .gz file through gzread) parsed on the device in blocks of 64 MiB; host
  // memory stays bounded by the block and the staging ring (kmg_fastx_stream_*).  A stream the device parser refuses (multi-line
  // FASTQ ...) goes on through the host splitter: the bytes it did not count plus the rest of the input are split with
  // kmg_parse_fastx and counted with count().  Returns the records of the whole stream.
  uint64_t count_stream(FILE *f, bool is_fastq, uint64_t size_hint = 0) {
    return count_stream_from([f](uint8_t *b, size_t cap) -> long { const size_t n = fread(b, 1, cap, f); return ferror(f) ? -1 : (long)n; },
                             is_fastq, size_hint);
  }
  uint64_t count_stream(gzFile g, bool is_fastq, uint64_t size_hint = 0) {
    return count_stream_from([g](uint8_t *b, size_t cap) -> long { return (long)gzread(g, b, (unsigned)cap); }, is_fastq, size_hint);
  }
  // read(buf, cap): bytes read, 0 at the end, < 0 on a read error
  template <class Read>
  uint64_t count_stream_from(Read &&read, bool is_fastq, uint64_t size_hint) {
    constexpr size_t BLOCK = 64u << 20;
    const uint64_t r0 = progress().sequences_processed;
    check(kmg_fastx_stream_begin(ctx_, is_fastq, size_hint));
    std::vector<uint8_t> block(BLOCK);
    kmg_status s = KMG_OK;
    long n = 0;
    while (s == KMG_OK && (n = read(block.data(), BLOCK)) > 0) s = kmg_fastx_stream_push(ctx_, block.data(), (uint64_t)n);
    if (n < 0) { kmg_reset(ctx_); throw SequenceReadError("failed to read sequences from the input stream"); }
    if (s == KMG_OK) { uint64_t recs = 0; s = kmg_fastx_stream_end(ctx_, &recs); }
    if (s != KMG_OK) {
      const std::string msg = kmg_last_error(ctx_);
      uint64_t n_rest = 0;
      if (s != KMG_ERR_PARSE || kmg_fastx_stream_rest(ctx_, nullptr, 0, &n_rest) != KMG_OK) {
        if (s == KMG_ERR_PARSE) throw SequenceParseError(msg);
        throw GpuError(s, msg);
      }
      std::vector<uint8_t> data(n_rest);
      check(kmg_fastx_stream_rest(ctx_, data.data(), n_rest, &n_rest));
      while ((n = read(block.data(), BLOCK)) > 0) data.insert(data.end(), block.data(), block.data() + n);
      if (n < 0) throw SequenceReadError("failed to read sequences from the input stream");
      count(parse_records(data, is_fastq));
    }
    return progress().sequences_processed - r0;
  }
  // fasta / tsv / json records formatted on the device, sorted by k-mer (kmg_write_text; "-" = stdout)
  uint64_t write_text(const std::string &path, OutputFormat fmt, uint64_t min_count) {
    if (fmt == OutputFormat::Histogram) throw KmeRustError("write_text formats fasta, tsv or json; the histogram comes from histogram()");
    const int code = fmt == OutputFormat::Tsv ? KMG_TEXT_TSV : fmt == OutputFormat::Json ? KMG_TEXT_JSON : KMG_TEXT_FASTA;
    uint64_t recs = 0, bytes = 0;
    check(kmg_write_text(ctx_, min_count, code, path.c_str(), &recs, &bytes));
    return recs;
  }
  std::vector<uint64_t> query(const std::vector<std::string> &kmers, uint64_t *n_invalid = nullptr) {
    std::string blob;
    for (auto &q : kmers) blob += q;
    std::vector<uint64_t> out(kmers.size());
    uint64_t bad = 0;
    if (!kmers.empty()) check(kmg_query_ascii(ctx_, reinterpret_cast<const uint8_t *>(blob.data()), kmers.size(), out.data(), &bad));
    if (n_invalid) *n_invalid = bad;
    return out;
  }
  // adopt a context opened by kmg_index_open
  GpuKmerCounter(kmg_ctx *ctx, KmerLength k) : ctx_(ctx), k_(k) {}
  void save_kmix(const std::string &path);  // defined after save_index (a .gz path goes through the host writer)
  Progress progress() const { Progress p{}; kmg_progress(ctx_, &p.sequences_processed, &p.bases_processed); return p; }
};

// ---- reference-named entry points --------------------------------------------------------------------
inline PackedCounts to_map(const std::vector<uint64_t> &k, const std::vector<uint64_t> &c) {
  PackedCounts m; m.reserve(k.size());
  for (size_t i = 0; i < k.size(); ++i) m.emplace(k[i], c[i]);
  return m;
}
// src/streaming.rs:198-204
inline PackedCounts count_kmers_from_sequences(const std::vector<std::string> &sequences, KmerLength k) {
  GpuKmerCounter c(k);
  c.count_sequences(sequences);
  c.finalize();
  std::vector<uint64_t> keys, counts;
  c.export_counts(1, false, keys, counts);
  return to_map(keys, counts);
}
// src/streaming.rs:158-167
inline PackedCounts count_kmers_streaming_packed(const std::string &path, KmerLength k) {
  GpuKmerCounter c(k);
  c.count(read_with_quality(path, SequenceFormat::Auto));
  c.finalize();
  std::vector<uint64_t> keys, counts;
  c.export_counts(1, false, keys, counts);
  return to_map(keys, counts);
}
// src/run.rs:304-344 (and :221, :245 through the defaults)
inline std::unordered_map<std::string, uint64_t> count_kmers_with_quality(const std::string &path, size_t k,
                                                                          SequenceFormat fmt = SequenceFormat::Auto,
                                                                          std::optional<uint8_t> min_quality = std::nullopt) {
  const KmerLength kl = KmerLength::create(k);
  GpuKmerCounter c(kl, min_quality);
  c.count(read_with_quality(path, fmt));
  c.finalize();
  std::vector<uint64_t> keys, counts;
  c.export_counts(1, false, keys, counts);
  std::unordered_map<std::string, uint64_t> m; m.reserve(keys.size());
  for (size_t i = 0; i < keys.size(); ++i) m.emplace(unpack_to_string(keys[i], kl), counts[i]);  // into_hashmap, src/run.rs:573-582
  return m;
}
inline std::unordered_map<std::string, uint64_t> count_kmers(const std::string &path, size_t k) { return count_kmers_with_quality(path, k); }

// src/histogram.rs:110-116 on an exported map (host glue; the GPU version is GpuKmerCounter::histogram)
inline KmerHistogram compute_histogram_packed(const PackedCounts &counts) {
  KmerHistogram h;
  for (auto &kv : counts) h[kv.second] += 1;
  return h;
}

// text emitters (src/run.rs:452-481); keys arrive sorted -> deterministic output order
inline void output_counts(std::ostream &out, const std::vector<uint64_t> &keys, const std::vector<uint64_t> &counts, KmerLength k,
                          OutputFormat fmt) {
  switch (fmt) {
    case OutputFormat::Fasta:
      for (size_t i = 0; i < keys.size(); ++i) out << '>' << counts[i] << '\n' << unpack_to_string(keys[i], k) << '\n';
      break;
    case OutputFormat::Tsv:
      for (size_t i = 0; i < keys.size(); ++i) out << unpack_to_string(keys[i], k) << '\t' << counts[i] << '\n';
      break;
    case OutputFormat::Json:
      out << "[";
      for (size_t i = 0; i < keys.size(); ++i)
        out << (i ? ",\n" : "\n") << "  {\n    \"kmer\": \"" << unpack_to_string(keys[i], k) << "\",\n    \"count\": " << counts[i] << "\n  }";
      out << (keys.empty() ? "]" : "\n]") << '\n';
      break;
    case OutputFormat::Histogram: {
      KmerHistogram h;
      for (uint64_t c : counts) h[c] += 1;
      for (auto &kv : h) out << kv.first << '\t' << kv.second << '\n';
      break;
    }
  }
}

// ---- builder (src/builder.rs:62-526) ----------------------------------------------------------------------
class KmerCounter {
  std::optional<KmerLength> k_;
  uint64_t min_count_ = 1;
  OutputFormat format_ = OutputFormat::Fasta;
  SequenceFormat input_format_ = SequenceFormat::Auto;
  KmerLength need_k() const { if (!k_) throw BuilderError("k-mer length must be set before counting"); return *k_; }
 public:
  KmerCounter &k(size_t k) { k_ = KmerLength::create(k); return *this; }
  KmerCounter &min_count(uint64_t m) { min_count_ = m; return *this; }
  KmerCounter &format(OutputFormat f) { format_ = f; return *this; }
  KmerCounter &input_format(SequenceFormat f) { input_format_ = f; return *this; }
  std::unordered_map<std::string, uint64_t> count(const std::string &path) const {  // src/builder.rs:242-260
    auto m = count_kmers_with_quality(path, need_k().get(), input_format_);
    if (min_count_ > 1)
      for (auto it = m.begin(); it != m.end();) it = it->second >= min_count_ ? std::next(it) : m.erase(it);
    return m;
  }
  KmerHistogram histogram(const std::string &path) const {  // src/builder.rs:286-294, on the GPU
    GpuKmerCounter c(need_k());
    c.count(read_with_quality(path, input_format_));
    c.finalize();
    return c.histogram(min_count_);
  }
  void count_to_writer(const std::string &path, std::ostream &out) const {  // src/builder.rs:399-442
    GpuKmerCounter c(need_k());
    c.count(read_with_quality(path, input_format_));
    c.finalize();
    std::vector<uint64_t> keys, counts;
    c.export_counts(min_count_, true, keys, counts);
    output_counts(out, keys, counts, need_k(), format_);
  }
};

// ---- .kmix index (src/index.rs) -----------------------------------------------------------------------------
class KmerIndex {
  KmerLength k_;
  PackedCounts counts_;
 public:
  KmerIndex(KmerLength k, PackedCounts c) : k_(k), counts_(std::move(c)) {}
  KmerLength k() const { return k_; }
  size_t len() const { return counts_.size(); }
  bool is_empty() const { return counts_.empty(); }
  const PackedCounts &counts() const { return counts_; }
  std::optional<uint64_t> get(uint64_t packed) const { auto it = counts_.find(packed); return it == counts_.end() ? std::nullopt : std::optional<uint64_t>(it->second); }
};

inline void put_le(std::string &s, uint64_t v, int n) { for (int i = 0; i < n; ++i) s.push_back((char)(v >> (8 * i))); }
inline uint64_t get_le(const uint8_t *p, int n) { uint64_t v = 0; for (int i = 0; i < n; ++i) v |= (uint64_t)p[i] << (8 * i); return v; }

// src/index.rs:156-196, :222-279 (host writer for an exported map; GpuKmerCounter::save_kmix streams from the device table)
inline void save_index(const KmerIndex &idx, const std::string &path) {
  std::string body = "KMIX";
  body.push_back(1); body.push_back((char)idx.k().as_u8());
  put_le(body, idx.len(), 8);
  std::vector<std::pair<uint64_t, uint64_t>> items(idx.counts().begin(), idx.counts().end());
  std::sort(items.begin(), items.end());
  for (auto &kv : items) { put_le(body, kv.first, 8); put_le(body, kv.second, 8); }
  put_le(body, crc32_z(0L, reinterpret_cast<const Bytef *>(body.data()), body.size()), 4);  // crc32_z: size_t length (indexes pass 4 GiB)
  if (ends_with(path, ".gz")) {
    gzFile g = gzopen(path.c_str(), "wb");
    if (!g || gzwrite(g, body.data(), (unsigned)body.size()) != (int)body.size()) { if (g) gzclose(g); throw IndexIoError("failed to write index to '" + path + "'"); }
    gzclose(g);
    return;
  }
  std::ofstream f(path, std::ios::binary);
  if (!f || !f.write(body.data(), (std::streamsize)body.size())) throw IndexIoError("failed to write index to '" + path + "'");
}

// src/index.rs:199-216, :282-401: same checks, same order
inline KmerIndex load_index(const std::string &path) {
  std::vector<uint8_t> d;
  try { d = slurp(path); } catch (const KmeRustError &) { throw IndexIoError("failed to read index from '" + path + "'"); }
  if (d.size() < 18) throw InvalidIndexError("invalid index file '" + path + "': file too small");
  if (memcmp(d.data(), "KMIX", 4) != 0) throw InvalidIndexError("invalid index file '" + path + "': invalid magic bytes (not a kmerust index file)");
  const uint32_t stored = (uint32_t)get_le(d.data() + d.size() - 4, 4);
  const uint32_t computed = (uint32_t)crc32_z(0L, d.data(), d.size() - 4);
  if (stored != computed) {
    char buf[128];
    snprintf(buf, sizeof buf, "checksum mismatch (expected %#x, got %#x)", stored, computed);
    throw InvalidIndexError("invalid index file '" + path + "': " + buf);
  }
  if (d[4] != 1) throw InvalidIndexError("invalid index file '" + path + "': unsupported version " + std::to_string(d[4]));
  if (d[5] < 1 || d[5] > 32) throw InvalidIndexError("invalid index file '" + path + "': invalid k-mer length: " + std::to_string(d[5]));
  const uint64_t n = get_le(d.data() + 6, 8);
  if (d.size() - 18 != n * 16) throw InvalidIndexError("invalid index file '" + path + "': data size mismatch");
  PackedCounts m; m.reserve(n);
  for (uint64_t i = 0; i < n; ++i) m[get_le(d.data() + 14 + 16 * i, 8)] = get_le(d.data() + 22 + 16 * i, 8);
  return KmerIndex(KmerLength::create(d[5]), std::move(m));
}

// src/index.rs:156-196: the index straight from the device table; a path ending in .gz is gzip-wrapped like the reference does
// (kmg_save_kmix itself refuses .gz names rather than writing raw bytes under them)
inline void GpuKmerCounter::save_kmix(const std::string &path) {
  if (!ends_with(path, ".gz")) { check(kmg_save_kmix(ctx_, path.c_str())); return; }
  std::vector<uint64_t> keys, counts;
  export_counts(0, false, keys, counts);
  save_index(KmerIndex(k_, to_map(keys, counts)), path);
}

// src/index.rs:199-216 into device memory: a ready-to-query counter (kmg_index_open; .gz indexes go through load_index)
inline std::unique_ptr<GpuKmerCounter> open_index_on_device(const std::string &path) {
  kmg_ctx *ctx = nullptr;
  const kmg_status s = kmg_index_open(path.c_str(), -1, &ctx);
  if (s == KMG_ERR_PARSE) throw InvalidIndexError("invalid index file '" + path + "': " + kmg_last_error(nullptr));
  if (s == KMG_ERR_IO) throw IndexIoError(kmg_last_error(nullptr));
  if (s != KMG_OK) throw GpuError(s, kmg_last_error(nullptr));
  return std::unique_ptr<GpuKmerCounter>(new GpuKmerCounter(ctx, KmerLength::create(kmg_ctx_k(ctx))));
}

}  // namespace kmerust
