/*
 * kmerust_gpu.h -- C ABI (v1) of the B200-native canonical k-mer counting engine.
 *
 * This is the drop-in boundary for kmerust's counting path (SURVEY.md section 8b).  The reference
 * (crate kmerust v0.3.1, paths below relative to its repository root) has no FFI of its own; its
 * de-facto operator interface is Rust-internal:
 *     in : Iterator<Item = Bytes> / IntoIter<SequenceWithQuality> + KmerLength + Option<u8> min_quality
 *     out: HashMap<u64, u64>  (packed canonical k-mer -> count)
 * (src/streaming.rs:198-204 count_kmers_from_sequences, :158-167 count_kmers_streaming_packed,
 *  src/run.rs:491-583 KmerMap, src/reader.rs:13-16 SequenceWithQuality).
 * Each entry point below names the reference item it replaces.  INTEGRATION.md shows the Rust
 * `-sys` binding a maintainer would add.
 *
 * Conventions
 *  - plain C, no exceptions cross the boundary; every call returns a kmg_status;
 *    kmg_last_error() returns a UTF-8 message for the last failing call on that context.
 *  - keys and counts are u64 little-endian, exactly the (packed_bits, count) pairs of
 *    HashMap<u64,u64> and of the .kmix DATA section (src/index.rs:7-23).
 *  - a context is driven by ONE feeder thread at a time (Rust wrapper: Send + !Sync).
 *  - ownership: the context, its pinned staging buffers and all device memory belong to the
 *    library; every result array belongs to the caller.
 *  - there is NO CPU fallback: without a CUDA device kmg_create() fails with KMG_ERR_CUDA.
 */
#ifndef KMERUST_GPU_H
#define KMERUST_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KMG_ABI_VERSION 1u

typedef enum kmg_status {
  KMG_OK = 0,
  KMG_ERR_INVALID_K = 1,   /* maps to KmerLengthError{k,min:1,max:32}  (src/kmer.rs:100-111, src/error.rs:88) */
  KMG_ERR_INVALID_ARG = 2,
  KMG_ERR_CUDA = 3,        /* no device / driver error; message carries cudaGetErrorString */
  KMG_ERR_OOM = 4,         /* device or pinned allocation failed */
  KMG_ERR_TABLE_FULL = 5,  /* table cannot grow any further; nothing is ever silently dropped */
  KMG_ERR_STATE = 6,       /* call not valid in the context's current state */
  KMG_ERR_IO = 7,          /* maps to KmeRustError::IndexWrite / SequenceRead (src/error.rs:20-60) */
  KMG_ERR_ABI = 8,         /* abi_version mismatch */
  KMG_ERR_CAPACITY = 9,    /* caller's output arrays are too small; *n_out holds the needed size */
  KMG_ERR_PARSE = 10       /* maps to KmeRustError::SequenceParse{details} (src/error.rs:27-30) */
} kmg_status;

enum {
  KMG_FLAG_FORCE_HASH = 1u,         /* use the single open-addressing HBM table (never the 4^k array / partitions) */
  KMG_FLAG_FORCE_DIRECT = 2u,       /* use the direct-indexed 4^k array (k <= 14 only) */
  KMG_FLAG_NO_PREAGG = 4u,          /* disable duplicate pre-aggregation (for A/B measurements) */
  KMG_FLAG_FORCE_PARTITIONED = 8u   /* use the partitioned pipeline (hash partitions counted in shared-memory tables) */
};

/* Replaces: KmerLength::new (src/kmer.rs:100) + the Option<u8> min_quality argument of
 * KmerMap::build_with_quality (src/run.rs:505-520) + capacity planning DashMap does implicitly. */
typedef struct kmg_config {
  uint32_t abi_version;       /* KMG_ABI_VERSION */
  uint32_t k;                 /* 1..=32 */
  int32_t device;             /* CUDA device ordinal; -1 = current device */
  uint32_t flags;             /* KMG_FLAG_* */
  uint8_t has_min_quality;    /* 0 = None */
  uint8_t min_quality;        /* Phred; a base passes iff qual_byte >= saturating_add(min_quality, 33) (src/run.rs:538) */
  uint8_t parts_log2;         /* partitioned pipeline: log2(#partitions), 0 = choose from the input size (max 20) */
  uint8_t reserved[5];
  uint64_t expected_distinct; /* capacity hint (distinct canonical k-mers, or simply the number of bases to come); 0 = plan from
                                 the first call and adapt: the hash table migrates to the partitioned pipeline past 2^26 keys,
                                 an outgrown partition plan is re-split.  A good hint avoids that extra work. */
  uint64_t batch_bases;       /* bases per staging chunk of kmg_count_ascii (4 chunks in flight) and capacity of a pre-packed
                                 batch; 0 = default (2^28) */
  void *stream;               /* cudaStream_t to run on; NULL = library-owned stream (pass cudaStreamLegacy, 0x1, to
                                 share the legacy default stream with e.g. a torch process) */
} kmg_config;

typedef struct kmg_ctx kmg_ctx;

/* What the reference reports through Progress{sequences_processed, bases_processed}
 * (src/progress.rs:26-31) plus what HashMap::len() / values().sum() would give. */
typedef struct kmg_summary {
  uint64_t n_records;
  uint64_t n_bases;
  uint64_t n_windows;       /* counted windows == sum of all counts */
  uint64_t n_distinct;      /* distinct canonical k-mers in the table */
  uint64_t max_count;
  uint64_t table_capacity;  /* slots (hash path) or 4^k (direct path) */
  uint32_t path;            /* 0 = hash table, 1 = direct-indexed array, 2 = partitioned pipeline */
  uint32_t n_grows;         /* number of rehash/grow events (path 0; + 1 for a migration to path 2) or consolidation passes (path 2) */
  uint64_t kernel_ns;       /* device time spent in the counting kernels (CUDA events on the launching stream) */
  uint64_t h2d_bytes;
  uint64_t scan_ns;         /* of kernel_ns: tile scan (+ upsert on paths 0/1, + partition scatter on path 2) */
  uint64_t consolidate_ns;  /* of kernel_ns: path 2 phase B (one CTA per hash partition, table in shared memory) */
} kmg_summary;

/* One pinned, library-owned staging buffer for the pre-packed feed (the Rust reader packs
 * straight into it).  Layout: base j of the batch lives in bases2bit[j/32] at bit shift
 * 62 - 2*(j%32) (MSB first, i.e. a full word read as an integer is the reference's packed
 * 32-mer, src/kmer.rs:467-471); valid_bits[j/32] bit 31-(j%32) is 1 iff base j may be part of
 * a counted window (ACGTacgt and quality >= threshold).  Record boundaries are expressed by
 * start_bits (same bit layout; 1 on the first base of every record) so that windows never
 * span records (src/run.rs:500-503 processes each record separately). */
typedef struct kmg_batch {
  uint64_t *bases2bit;
  uint32_t *valid_bits;
  uint32_t *start_bits;
  uint64_t capacity_bases;
  uint64_t n_bases;    /* filled by the producer */
  uint64_t n_records;  /* filled by the producer (progress accounting only) */
  uint32_t slot;       /* which slot of the ring this is (library-private) */
} kmg_batch;

uint32_t kmg_abi_version(void);
const char *kmg_status_string(kmg_status s);
/* Message of the last failure on `ctx` (or of the last failing kmg_create when ctx == NULL). */
const char *kmg_last_error(const kmg_ctx *ctx);

/* Replaces KmerMap::new / StreamingKmerCounter::new (src/run.rs:494-498, src/streaming.rs:838-843). */
kmg_status kmg_create(const kmg_config *cfg, kmg_ctx **out);
void kmg_destroy(kmg_ctx *ctx);
/* The context's k (KmerIndex::k, src/index.rs:95; what kmg_index_open read from the file header). */
uint32_t kmg_ctx_k(const kmg_ctx *ctx);
/* Forget all counts but keep the allocations (benchmark steps, repeated use). */
kmg_status kmg_reset(kmg_ctx *ctx);

/* Replaces KmerMap::build_with_quality / StreamingKmerCounter::count_sequences over a batch of
 * records (src/run.rs:505-520, src/streaming.rs:1058-1066): `seq` holds n_records ASCII records
 * back to back, record r = seq[offsets[r] .. offsets[r+1]); `qual` (same layout, Phred+33) may be
 * NULL (FASTA: the quality filter is then ignored, tests/quality_tests.rs:88-114).  HOST pointers;
 * the call stages through pinned double buffers, overlapping H2D copies with the kernels, and
 * returns when everything is queued (results are complete after kmg_finalize). */
kmg_status kmg_count_ascii(kmg_ctx *ctx, const uint8_t *seq, const uint8_t *qual,
                           const uint64_t *offsets, uint64_t n_records);

/* Replaces reader::read / read_with_quality + the counting call for a whole FASTA / FASTQ FILE IMAGE in host memory (an mmap of
 * the file, src/mmap.rs:33-71; src/reader.rs:82-247 materialises every record on the host first): the raw bytes are copied to
 * the device in chunks cut at line / record boundaries and parsed THERE (line classification, trim_end of every sequence and
 * quality line, record starts), then ingested and scanned as usual.  Well-formed single- or multi-line FASTA and 4-line FASTQ
 * (\n or \r\n); multi-line FASTQ or a line longer than batch_bases gives KMG_ERR_PARSE -- fall back to kmg_parse_fastx +
 * kmg_count_ascii after kmg_reset.  *n_records_out: records (header lines) seen. */
kmg_status kmg_count_fastx(kmg_ctx *ctx, const uint8_t *buf, uint64_t len, int is_fastq, uint64_t *n_records_out);

/* Replaces count_kmers_from_reader_packed (src/streaming.rs:295-509) and the stdin / gzip readers (src/reader.rs:102-144): a
 * FASTA / FASTQ byte STREAM parsed on the device like kmg_count_fastx, in host memory bounded by the context's four pinned
 * staging slots whatever the stream's length.  For any split of a byte string into pushes the result (table, histogram, text,
 * .kmix, and the summary's records / bases / windows) equals kmg_count_fastx on the whole string wherever that call accepts it.
 *   begin: size_hint = bytes expected (0 = unknown: the table is planned from the first chunk and adapts).  Refused with
 *     KMG_ERR_STATE on a context of a shard group or with a stream already open.
 *   push: any number of bytes, cut anywhere; they are copied, so the buffer can be reused on return.  A slot that holds
 *     min(batch_bases, 2^30) bytes is cut at its last line start (FASTA) / record start (FASTQ), its copy to the device is queued
 *     and the chunk before it is parsed and counted; the bytes after the cut go to the front of the next slot.  A FASTA slot
 *     without a newline is cut inside its sequence line (between two non-blank bytes, not before a '>'), so unwrapped lines of
 *     any length are counted.
 *   end: parses and counts what is left (a last line without '\n' is fine) and closes the stream; *n_records_out: records of
 *     the whole stream.
 *   rest: after a KMG_ERR_PARSE that leaves the context usable, the bytes that were not counted (two-call protocol: bytes ==
 *     NULL gives the size in *n_out; KMG_ERR_CAPACITY when cap is too small).  That is every byte when byte 0 is no header
 *     ('>' / '@'), else the bytes from the first byte of the refused chunk on -- a FASTQ chunk refused before it was counted
 *     (multi-line FASTQ, no '+' line where one is expected, no record start near a slot end) or a FASTA slot without a
 *     possible cut.  The table then holds exactly the records of the earlier chunks, which all end at record starts: split the
 *     rest plus the remainder of the input with kmg_parse_fastx and feed it to kmg_count_ascii on the same context.
 * Every other failure (a quality line whose length differs from its sequence, CUDA errors, a full table) is final, as for
 * kmg_count_fastx: the stream is closed, rest gives KMG_ERR_STATE and the context needs kmg_reset.  While a stream is open
 * every other feed, kmg_finalize, export, histogram, text, index and query call returns KMG_ERR_STATE; kmg_progress advances
 * per counted chunk; kmg_reset and kmg_destroy abandon the stream. */
kmg_status kmg_fastx_stream_begin(kmg_ctx *ctx, int is_fastq, uint64_t size_hint);
kmg_status kmg_fastx_stream_push(kmg_ctx *ctx, const uint8_t *bytes, uint64_t n);
kmg_status kmg_fastx_stream_end(kmg_ctx *ctx, uint64_t *n_records_out);
kmg_status kmg_fastx_stream_rest(kmg_ctx *ctx, uint8_t *bytes, uint64_t cap, uint64_t *n_out);

/* Pre-packed, zero-copy feed for the Rust reader layer (src/reader.rs, src/streaming.rs, src/mmap.rs): a ring of four pinned
 * batches (zeroed when handed out), each with its own device buffers.  kmg_submit_batch queues the batch's H2D copy on the copy
 * stream at once and scans the batch submitted before it, so copies overlap the kernels while the producer fills the next
 * batch; the last batch is scanned by kmg_finalize (or whichever call reads the table next). */
kmg_status kmg_acquire_batch(kmg_ctx *ctx, kmg_batch *batch);
kmg_status kmg_submit_batch(kmg_ctx *ctx, const kmg_batch *batch);

/* Same work with inputs already resident in HBM (device pointers).  d_offsets may be NULL when
 * the buffer is one record.  d_seq must be 16-byte aligned. */
kmg_status kmg_count_ascii_device(kmg_ctx *ctx, const uint8_t *d_seq, const uint8_t *d_qual,
                                  const uint64_t *d_offsets, uint64_t n_records, uint64_t n_bytes);
/* Weighted upsert of already-canonical keys (device pointers; d_counts NULL = 1 each): the
 * receive side of the multi-GPU exchange.  Replaces process_valid_kmer (src/run.rs:565-571). */
kmg_status kmg_insert_keys_device(kmg_ctx *ctx, const uint64_t *d_keys, const uint64_t *d_counts, uint64_t n);
/* Scan only: emit the canonical key of every counted window, bucketed by owner shard
 * (owner = kmg_owner_of(key, n_shards)); d_keys_out has room for cap keys in total and is laid
 * out shard-major; shard_counts_out[n_shards] (HOST) receives the bucket sizes. */
kmg_status kmg_extract_keys_device(kmg_ctx *ctx, const uint8_t *d_seq, const uint8_t *d_qual,
                                   const uint64_t *d_offsets, uint64_t n_records, uint64_t n_bytes,
                                   uint32_t n_shards, uint64_t *d_keys_out, uint64_t cap,
                                   uint64_t *shard_counts_out);
uint32_t kmg_owner_of(uint64_t canonical_key, uint32_t n_shards);
/* Multi-GPU fast path.  kmg_partition_plan puts the context on the partitioned pipeline (sized for
 * expected_keys) and reports its partition plan: n_coarse coarse hash bins, each split into n_sub sub-bins.
 * A sender buckets its keys with kmg_extract_keys_device(n_shards = world * n_coarse): bins
 * [r*n_coarse, (r+1)*n_coarse) belong to rank r, so one all-to-all moves contiguous ranges.  The owner
 * then hands each received block to kmg_adopt_coarse_device (keys already grouped by ITS n_coarse bins,
 * bin_counts on the HOST), which only has to refine and count them -- no re-partitioning. */
kmg_status kmg_partition_plan(kmg_ctx *ctx, uint64_t expected_keys, uint32_t *n_coarse, uint32_t *n_sub);
kmg_status kmg_adopt_coarse_device(kmg_ctx *ctx, const uint64_t *d_keys, const uint64_t *bin_counts, uint32_t n_bins, uint64_t n);

/* ---- hash-sharded counting across the GPUs of one box (SURVEY.md 8e) ------------------------------------------------------
 * One context per GPU -- one process per device (torchrun, a Rust host that forks per GPU) or one thread per device -- joined
 * into a group.  The table shards by k-mer hash; every rank scatters its keys by (owner, hash bin) into its own send buffer,
 * and the exchange is fused into the owner's refine kernel, whose tile loads read the owner's bins straight out of all ranks'
 * send buffers through P2P-mapped memory (NVLink loads): no key is copied, it crosses NVLink on its way into the kernel that
 * partitions it further.  Only sizes, flags and results cross on the host, through a POSIX shared-memory segment named after
 * `group` (created by rank 0, unlinked once everybody is attached) -- no NCCL inside the library.  All kmg_shard_* calls are
 * COLLECTIVE: every rank makes the same sequence of them (a rank without input passes n_bytes / n_records = 0); a rank that
 * fails marks the group aborted, so its peers return KMG_ERR_STATE instead of waiting.  Results of the whole group: summary,
 * histogram, one .kmix and one sorted text file (kmg_shard_write_text: the key space cut into pieces, each merged by one owner
 * straight out of its peers' staging buffers).  world == 1 degenerates to the plain
 * single-GPU calls.  Local feeds (kmg_count_ascii, kmg_insert_keys_device ...) are refused on a grouped context.
 *   kmg_shard_join: before the first feed; identical k / batch_bases / expected_keys_total (keys of the WHOLE job; 0 = the
 *   config's expected_distinct) on every rank.  One round moves at most batch_bases bases per rank.
 * Replaces the single shared DashMap of src/run.rs:489-583 by `world` disjoint tables. */
kmg_status kmg_shard_join(kmg_ctx *ctx, uint32_t world, uint32_t rank, const char *group, uint64_t expected_keys_total);
kmg_status kmg_shard_leave(kmg_ctx *ctx);
/* THIS rank's slice of the records; layouts as kmg_count_ascii_device / kmg_count_ascii. */
kmg_status kmg_shard_count_ascii_device(kmg_ctx *ctx, const uint8_t *d_seq, const uint8_t *d_qual, const uint64_t *d_offsets,
                                        uint64_t n_records, uint64_t n_bytes);
kmg_status kmg_shard_count_ascii(kmg_ctx *ctx, const uint8_t *seq, const uint8_t *qual, const uint64_t *offsets, uint64_t n_records);
/* kmg_count_fastx for the whole group: every rank passes the SAME whole file image (each process may mmap the file, thread ranks
 * may share one buffer) and parses only its own slice of it on the device.  With t = len * r / world, rank r's slice begins at
 * the first line start (FASTA) / record start (FASTQ: a '@' line whose line after next begins with '+') at or after t; every rank
 * computes all cuts from the same bytes.  A FASTA slice that begins inside a record is preceded by the record's last k-1 bases,
 * so every window is counted once, by the rank that holds its last base; the union of the shards equals what kmg_count_fastx
 * gives on one context, whatever the world size.  Each parsed chunk (at most batch_bases - (k-1) raw bytes) is one fused round.
 * *n_records_out: records of the whole image, on every rank.  Join with expected_keys_total = len (FASTA) or len / 2 (FASTQ).
 * Every rank returns an error when byte 0 is no header, a line is longer than a chunk, the FASTQ is multi-line or has a quality
 * of a different length than its sequence (KMG_ERR_PARSE; peers of a rank that fails mid-stream return KMG_ERR_STATE), or the
 * ranks passed images of different lengths / cuts (KMG_ERR_INVALID_ARG).  The group is then aborted: leave it, destroy the
 * contexts, and count the input with a new group through kmg_parse_fastx + kmg_shard_count_ascii.  Outside a group it is
 * kmg_count_fastx. */
kmg_status kmg_shard_count_fastx(kmg_ctx *ctx, const uint8_t *buf, uint64_t len, int is_fastq, uint64_t *n_records_out);
/* kmg_finalize + the summary of the WHOLE table (sums over the shards; kernel timings stay this rank's). */
kmg_status kmg_shard_finalize(kmg_ctx *ctx, kmg_summary *summary);
/* kmg_histogram merged over the shards (element-wise sum); the size query does the merge, the second call copies it out. */
kmg_status kmg_shard_histogram(kmg_ctx *ctx, uint64_t min_count, uint64_t *count_vals, uint64_t *freqs, uint64_t cap, uint64_t *n_out);
/* ONE .kmix from all shards: rank 0 writes header and combined CRC, every rank its own records (src/index.rs:222-279). */
kmg_status kmg_shard_save_kmix(kmg_ctx *ctx, const char *path, uint64_t *n_records_out);
/* ONE file holding the records of ALL shards with count >= min_count (0 behaves as 1) in ascending k-mer order, formatted as
 * KMG_TEXT_FASTA / KMG_TEXT_TSV / KMG_TEXT_JSON: byte-identical to what kmg_write_text writes for a single context that counted
 * the same input.
 * COLLECTIVE, same arguments on every rank; every rank writes its own byte ranges of the file.  *n_records_out / *n_bytes_out:
 * totals of the whole file, on every rank.  On a context outside a group it is kmg_write_text.  Inside a group "-" (stdout) is
 * refused with KMG_ERR_INVALID_ARG on every rank; ranks that disagree on min_count / format abort the group. */
kmg_status kmg_shard_write_text(kmg_ctx *ctx, uint64_t min_count, int format, const char *path,
                                uint64_t *n_records_out, uint64_t *n_bytes_out);
/* Diagnostics: keys written to other ranks, keys received, rounds, rounds that took the exact (count + prefix) route. */
kmg_status kmg_shard_stats(const kmg_ctx *ctx, uint64_t *sent_keys, uint64_t *recv_keys, uint64_t *rounds, uint64_t *exact_rounds);

/* Waits for all queued work; replaces into_hashmap()'s barrier role (src/run.rs:573-582). */
kmg_status kmg_finalize(kmg_ctx *ctx, kmg_summary *summary);

/* Replaces the HashMap<u64,u64> result + the min-count retain (src/run.rs:447-450,
 * src/builder.rs:251-258).  Two-call protocol: with keys == NULL only *n_out is written.
 * sorted != 0 gives ascending key order (== lexicographic order of the k-mer strings). */
kmg_status kmg_export_counts(kmg_ctx *ctx, uint64_t min_count, int sorted, uint64_t *keys,
                             uint64_t *counts, uint64_t cap, uint64_t *n_out);
kmg_status kmg_export_counts_device(kmg_ctx *ctx, uint64_t min_count, int sorted, uint64_t *d_keys,
                                    uint64_t *d_counts, uint64_t cap, uint64_t *n_out);

/* The same result in pieces: shard s of n_shards holds the entries with key % n_shards == s (n_shards <= 1: everything).  For
 * tables larger than the caller's memory -- the 3.1 Gbp configuration's HashMap<u64,u64> is 50 GB -- and for sampled checks. */
kmg_status kmg_export_shard(kmg_ctx *ctx, uint64_t min_count, int sorted, uint64_t n_shards, uint64_t shard, uint64_t *keys,
                            uint64_t *counts, uint64_t cap, uint64_t *n_out);
kmg_status kmg_export_shard_device(kmg_ctx *ctx, uint64_t min_count, int sorted, uint64_t n_shards, uint64_t shard,
                                   uint64_t *d_keys, uint64_t *d_counts, uint64_t cap, uint64_t *n_out);

/* Replaces compute_histogram_packed after the min-count filter (src/histogram.rs:110-116,
 * src/run.rs:471-481): ascending (count, number of distinct k-mers with that count). */
kmg_status kmg_histogram(kmg_ctx *ctx, uint64_t min_count, uint64_t *count_vals, uint64_t *freqs,
                         uint64_t cap, uint64_t *n_out);

/* Replaces the fasta / tsv / json text emitters of output_counts and count_to_writer (src/run.rs:452-481, src/builder.rs:399-442)
 * and unpack_to_string (src/kmer.rs:431-456): entries with count >= min_count (0 behaves as 1) in ascending k-mer order -- the
 * reference prints HashMap iteration order, parity is defined on the sorted text -- formatted on the device
 * (tsv "{kmer}\t{count}\n", fasta ">{count}\n{kmer}\n", json the serde_json::to_string_pretty array of {"kmer", "count"}
 * objects plus "\n", "[]\n" when no entry passes) and delivered to `sink` in chunks of at most 64 MiB; a non-zero return from
 * the sink aborts with KMG_ERR_IO.  *n_bytes_out counts every byte delivered, json's "[" and closing "]\n" included.
 * kmg_write_text writes the same bytes to a file ("-" = stdout). */
enum { KMG_TEXT_FASTA = 0, KMG_TEXT_TSV = 1, KMG_TEXT_JSON = 2 };
typedef int (*kmg_text_sink)(void *user, const uint8_t *bytes, size_t n);
kmg_status kmg_emit_text(kmg_ctx *ctx, uint64_t min_count, int format, kmg_text_sink sink, void *user, uint64_t *n_records_out,
                         uint64_t *n_bytes_out);
kmg_status kmg_write_text(kmg_ctx *ctx, uint64_t min_count, int format, const char *path, uint64_t *n_records_out, uint64_t *n_bytes_out);

/* Replaces counts_to_packed + KmerIndex::new + save_index (src/main.rs:155-202, :284-299,
 * src/index.rs:156-196, :222-279).  Writes ALL k-mers (the index is never min-count filtered). */
kmg_status kmg_save_kmix(kmg_ctx *ctx, const char *path);
/* The same index written from several shards (one context per GPU, hash-sharded table): kmg_kmix_begin creates the file; every
 * shard writes its records at record_offset (= records of the shards before it; sizes from kmg_finalize) and reports their
 * number and CRC-32; kmg_kmix_finish writes the header (n = sum over shards) and the CRC of the whole file combined from the
 * shard CRCs (the format allows any record order, src/index.rs:7-23).  Paths ending in .gz are refused (no compression here). */
kmg_status kmg_kmix_begin(const char *path);
kmg_status kmg_save_kmix_shard(kmg_ctx *ctx, const char *path, uint64_t record_offset, uint64_t *n_records_out, uint32_t *crc_out);
kmg_status kmg_kmix_finish(const char *path, uint32_t k, const uint64_t *shard_records, const uint32_t *shard_crcs, uint32_t n_shards);

/* Batched look-ups (replaces KmerIndex::get, src/index.rs:127-131, and the canonicalisation the `query` subcommand does first,
 * src/main.rs:254-266).  HOST arrays.  kmg_query_keys: canonical packed keys -> counts (0 = absent).  kmg_query_ascii: n k-mers
 * of k ASCII bytes each, any case, canonicalised on the device; a k-mer with a byte outside ACGTacgt counts 0 and is reported in
 * *n_invalid_out.  A context of a shard group answers for the keys it owns (0 for the others: sum the ranks' answers). */
kmg_status kmg_query_keys(kmg_ctx *ctx, const uint64_t *keys, uint64_t n, uint64_t *counts_out);
kmg_status kmg_query_ascii(kmg_ctx *ctx, const uint8_t *kmers, uint64_t n, uint64_t *counts_out, uint64_t *n_invalid_out);
/* Replaces load_index / read_index (src/index.rs:199-216, :282-401): opens an uncompressed .kmix file as a ready-to-query
 * context on `device` (-1 = current).  Same checks in the same order: size >= 18, magic, CRC-32, version, k, data size == n * 16.
 * KMG_ERR_IO = cannot read, KMG_ERR_PARSE = invalid index (message: kmg_last_error(NULL)). */
kmg_status kmg_index_open(const char *path, int32_t device, kmg_ctx **out);

/* Replaces ProgressTracker::snapshot (src/progress.rs). */
kmg_status kmg_progress(const kmg_ctx *ctx, uint64_t *records, uint64_t *bases);

/* Diagnostics: number of this library's own CUDA kernels launched so far in this process. */
uint64_t kmg_kernel_launches(void);

/* Diagnostics (no reference counterpart): device time of the partitioned pipeline's stages since the last kmg_reset, CUDA events on
 * the launching stream.  out_ns4[0] = ingest + A1 (tile scan + coarse scatter), [1] = A2 (refine to fine partitions, on N GPUs the
 * pull over NVLink), [2] = phase B (count the partitions), [3] = everything else timed (paths 0 / 1: the scan-and-count kernel). */
kmg_status kmg_phase_times(kmg_ctx *ctx, uint64_t *out_ns4);

/* Test/bench helper: fill d_out[n] with the deterministic synthetic base stream
 * (same generator as oracle/kmer_oracle.c orc_synth_uniform). */
kmg_status kmg_synth_uniform_device(kmg_ctx *ctx, uint64_t seed, uint64_t first_base, uint64_t n, uint8_t *d_out);

/* Test/bench helper: n_reads synthetic 150 bp reads laid back to back (d_seq, and d_qual unless NULL: n_reads * 150 bytes
 * each); profile 3 = the R20M shape of config C3 (N bases, Phred qualities), 5 = the R200M shape of config C5 (10 % satellite
 * reads).  Same generator as oracle/kmer_oracle.c orc_synth_reads. */
kmg_status kmg_synth_reads_device(kmg_ctx *ctx, uint64_t seed, uint32_t profile, uint64_t first_read, uint64_t n_reads,
                                  uint8_t *d_seq, uint8_t *d_qual);

/* Host utility (no CUDA): FASTA/FASTQ record splitter for hosts without the Rust reader layer; stands
 * in for bio::io::{fasta,fastq}::Reader as used by src/reader.rs:91,96,176,181.  seq_out (and
 * qual_out for FASTQ, may be NULL) need room for `len` bytes, offsets_out for max_records+1
 * entries.  Errors map to KmeRustError::SequenceParse{details} with the message in errbuf. */
kmg_status kmg_parse_fastx(const uint8_t *buf, uint64_t len, int is_fastq, uint8_t *seq_out, uint8_t *qual_out,
                           uint64_t *offsets_out, uint64_t max_records, uint64_t *n_records_out, char *errbuf,
                           size_t errbuf_len);

#ifdef __cplusplus
}
#endif
#endif /* KMERUST_GPU_H */
