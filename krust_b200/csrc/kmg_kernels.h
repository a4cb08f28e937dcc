// Internal C++ interface between the C-ABI layer (kmg_api.cu) and the kernels (kmg_kernels.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace kmg {

// packed-stream view handed to the scan kernels; pointers include the zero lead-in words.
struct ScanInput {
  const uint64_t *bases;
  const uint32_t *valid;
  const uint32_t *start;  // nullptr: single record / no boundaries inside the stream
  uint64_t n_tiles;
  int k;
  // speculative scatter (no count pass): partition p owns out[p * part_cap, (p + 1) * part_cap); a reservation that does not
  // fit raises *overflow_flag and writes nothing.  part_cap == 0: exact layout from the counted prefix.
  uint64_t part_cap = 0;
  uint32_t *overflow_flag = nullptr;
};

struct HashTable {
  uint64_t *slots;  // cap x {key, count}
  uint64_t cap;
};

// read-side view over either table kind
struct TableView {
  const uint64_t *slots;             // v1 hash table (key, occurrences-1) slots
  const unsigned long long *dense;   // direct path: 4^k counters
  const uint64_t *pair_keys;         // partitioned path: consolidated run, SoA
  const uint64_t *pair_counts;
  uint64_t n;                        // slots, 4^k or number of pairs
  uint64_t shard_mod = 0, shard_rem = 0;  // stats (entry count) / compaction only: keep keys with key % shard_mod == shard_rem (<= 1: all)
  uint64_t range_lo = 0, range_hi = ~0ull;  // ... and range_lo <= key <= range_hi
  __host__ __device__ bool keeps(uint64_t key) const {
    return (shard_mod <= 1 || key % shard_mod == shard_rem) && key >= range_lo && key <= range_hi;
  }
};
constexpr int KEY_BUCKETS = 4096;  // kmg_save_kmix sizes its sorted pieces from a histogram over the top 12 bits of the 2k-bit keys

// ---- partitioned pipeline (kmg_partition.cu) ----------------------------------------------------------
constexpr int CONS_MAX_RUNS = 32;  // one warp scans the segment table of a partition
constexpr int MAX_PARTS = 8192;        // bins of ONE scatter level (shared-memory histogram)
constexpr int REFINE_THREADS = 512;
constexpr int REFINE_TILE = 8192;      // keys per level-2 tile (staged in shared memory: 64 KiB, 128 KiB with counts)
constexpr int REFINE_ROWS_THREADS = 1024;   // single-pass level-2 scatter: one CTA per SM
constexpr int REFINE_ROWS_SLOTS = 16384;    // n_sub rows of 2^cap_log2 keys (128 KiB)
constexpr int REFINE_ROWS_OVERFLOW = 4096;  // keys whose row was full (a coarse bin holding a hot key puts hundreds per tile there)
constexpr int COUNT_THREADS = 512;
constexpr int COUNT_CTAS_PER_SM = 2;
constexpr int SMEM_COUNT_THREADS = 512;    // phase B primary variant: table in shared memory, 2 CTAs/SM
constexpr int SMEM_TABLE_SLOTS = 8192;      // 64 KiB of u64 keys + 32 KiB of u32 (count-1)

// A run: partition-indexed keys (every key counts 1) or (key, count) pairs.  Partition p of the run is
// entries [seg_start[p], seg_start[p] + seg_len[p]).
struct ConsRun {
  const uint64_t *keys;
  const uint64_t *counts;     // nullptr: every key counts 1
  const uint64_t *seg_start;  // device, n_parts entries
  const uint64_t *seg_len;    // device, n_parts entries
};
struct RefineParams {
  const uint64_t *keys, *counts;          // coarse-partitioned input (counts may be nullptr)
  const uint64_t *coarse_start;           // n_coarse + 1
  const uint64_t *coarse_len;             // nullptr: partition c ends where c + 1 starts (exact layout)
  const uint32_t *tile_prefix;            // n_coarse + 1: first global tile number of each coarse partition
  uint32_t n_coarse, n_sub, n_tiles, row_cap;   // row_cap / row_magic: row size of the single-pass scatter (set by launch_refine)
  uint32_t row_magic, pad;
  // bin of a key inside input partition c: sub_of_mix(mix, sub_total) - (c % sub_old) * n_sub.  Plain refinement of coarse bins:
  // sub_total = n_sub, sub_old = 1.  Re-splitting a fine-partitioned run m ways (the sub-bin function nests: floor(x * P2 * m) / m ==
  // floor(x * P2)): n_sub = m, sub_old = old sub-bins per coarse bin, sub_total = sub_old * m.
  uint32_t sub_total, sub_old;
  // sharded pull: input partition c is read from src[c % in_group] (the send buffer of source rank c % in_group, P2P-mapped:
  // the tile loads below are the NVLink transfer); n_src == 0: everything comes from `keys`
  const uint64_t *src[8];
  uint32_t n_src, pad2;
  uint32_t in_keys, in_group;             // in_keys 1: the input holds plain keys (adopted from another rank) -- mix on load; the output is always mixed
                                          // in_group g > 1: input partitions c*g .. c*g+g-1 are g pieces of coarse bin c (one per source rank of the sharded scatter)
  unsigned long long *fine_counts;        // count pass
  const unsigned long long *fine_start;   // scatter pass: exclusive prefix of fine_counts
  unsigned long long *fine_cursor;        // scatter pass: zeroed
  uint64_t *out_keys, *out_counts;
  // speculative layout (no count pass): fine partition f owns out[f * fine_cap, (f + 1) * fine_cap); fine_cursor[] then ends
  // up as the partition sizes.  A reservation that does not fit raises *overflow_flag and writes nothing (the host redoes
  // the chunk with exact counts).  fine_cap == 0: exact layout, fine_start[] is the prefix of the counted sizes.
  uint64_t fine_cap;
  uint32_t *overflow_flag;
};
struct CountParams {
  uint32_t n_parts, R, scratch_log2, preagg;
  uint32_t split_log2;               // shared-memory kernel: partitions larger than a table are counted in up to 2^split_log2 passes
  // sieve in place (one raw run in a strided layout: partition p owns entries [p * part_cap, (p + 1) * part_cap)): the
  // output run IS the input run.  Its keys are never written -- a repeated key's further entries keep their key and get count 0 --
  // and the counts cover every partition's whole capacity (0 behind the segment).  0: the keys are copied to out_keys.
  uint32_t part_cap;
  ConsRun runs[CONS_MAX_RUNS];
  const uint32_t *order;             // partitions in processing order (largest first); nullptr = 0, 1, 2, ...
  uint64_t *scratch;                 // gridDim.x private tables of 2^scratch_log2 (key, count-1) slots, clean
  uint64_t *out_keys, *out_counts;
  unsigned long long *out_cursor;    // zeroed; ends up = entries of the output run (distinct keys + skipped filler entries)
  unsigned long long *out_distinct;  // zeroed; ends up = number of distinct keys
  uint64_t *out_seg_start, *out_seg_len;  // n_parts each: where partition p landed in the output
  uint32_t *next, *error_flag;       // zeroed
  // the output run holds out_cap entries (the host sizes it from the expected number of DISTINCT keys, not from the input
  // entries: read sets repeat every k-mer many times); a partition whose reservation does not fit writes nothing and raises
  // *nospace_flag -- the host then retries with a larger run
  unsigned long long out_cap;
  uint32_t *nospace_flag;            // zeroed
  // count-of-counts of the OUTPUT, built while compacting (zeroed by the host; nullptr = skip):
  // hist[c] for 2 <= c < HIST_DENSE_BINS, hist[HIST_DENSE_BINS] = number of overflow entries;
  // counts >= HIST_DENSE_BINS are appended to hist_overflow.  hist[1] is implied (distinct - the rest).
  unsigned long long *hist;
  uint64_t *hist_overflow;
  uint64_t hist_overflow_cap;
  // sieve variant only: partitions it hands to the compacting variant (more repeated keys than its side table holds, or more
  // entries than one batch), appended as partition numbers
  uint32_t *redo_list, *redo_count;  // redo_count zeroed
  // ... together with the output range a partition had already reserved (redo_base[i] = ~0: none).  The launch that takes the list
  // over passes them back as pre_base / pre_len (indexed like `order`): such a partition is written into its range, the unused
  // tail filled with skipped entries.
  unsigned long long *redo_base;
  uint32_t *redo_len;
  const unsigned long long *pre_base;
  const uint32_t *pre_len;
};

enum { CTR_WINDOWS = 0, CTR_DISTINCT = 1, CTR_FULL = 2, CTR_SCRATCH = 3, CTR_N = 8 };

constexpr int SCAN_CTAS_PER_SM = 4;
constexpr int DENSE_SMEM_MAX_K = 6;      // 4^6 u32 = 16 KiB privatised per CTA
constexpr int DENSE_MAX_K = 14;          // 4^14 u64 = 2 GiB
constexpr int DENSE_DEFAULT_MAX_K = 13;  // automatic choice of the direct path
constexpr int HIST_SMEM_BINS = 2048;
constexpr int HIST_DENSE_BINS = 65536;
constexpr int HIST_CTA_BINS = 32;        // phase B keeps the lowest bins per CTA in shared memory
constexpr uint64_t HIST_OVERFLOW_CAP = 1 << 16;

cudaError_t launch_ingest(const uint8_t *d_seq, const uint8_t *d_qual, uint64_t n_bytes, uint32_t thr, uint64_t n_words_total,
                          uint64_t *d_bases, uint32_t *d_valid, cudaStream_t s);
cudaError_t launch_start_bits(const uint64_t *d_offsets, uint64_t n_records, uint64_t base_offset, uint64_t n_bytes,
                              uint64_t n_words_total, uint32_t *d_start, cudaStream_t s);
cudaError_t launch_synth_uniform(uint64_t seed, uint64_t first_base, uint64_t n, uint8_t *d_out, cudaStream_t s);
cudaError_t launch_synth_reads(uint64_t seed, uint32_t profile, uint64_t first_read, uint64_t n_reads, uint8_t *d_seq, uint8_t *d_qual,
                               cudaStream_t s);
cudaError_t launch_count_windows(const uint32_t *d_valid, const uint32_t *d_start, uint64_t n_words, int k, unsigned long long *d_out,
                                 cudaStream_t s);
cudaError_t launch_scan_emit_keys(const ScanInput &in, uint64_t *d_out, unsigned long long *d_cursor, cudaStream_t s);
cudaError_t launch_scan_hash(const ScanInput &in, HashTable t, unsigned long long *counters, uint32_t flags, cudaStream_t s);
cudaError_t launch_scan_dense(const ScanInput &in, unsigned long long *dense, unsigned long long *counters, uint32_t flags,
                              cudaStream_t s);
// scatter == false: part_counts[p] += keys of partition p.  scatter == true: keys are written to
// out[part_start[p] + ...]; part_cursor[] (zeroed) hands out ranges inside each partition.
cudaError_t launch_scan_partition(const ScanInput &in, uint32_t n_parts, bool scatter, unsigned long long *part_counts,
                                  const unsigned long long *part_start, unsigned long long *part_cursor, uint64_t *out,
                                  unsigned long long *counters, cudaStream_t s, bool mixed = false);  // mixed: write mix64(key)
bool scan_scatter_supports_cap(uint32_t n_parts);
cudaError_t launch_keys_coarse(const uint64_t *d_keys, const uint64_t *d_counts, uint64_t n, uint32_t n_coarse, bool scatter,
                               unsigned long long *coarse_counts, const unsigned long long *coarse_start,
                               unsigned long long *coarse_cursor, uint64_t *out_keys, uint64_t *out_counts, cudaStream_t s);
cudaError_t launch_refine(const RefineParams &P, bool scatter, cudaStream_t s);
bool refine_single_pass_available(uint32_t n_sub, bool weighted);  // the rows kernel applies (it can run without a count pass)
cudaError_t launch_fill_strided(uint64_t *d, uint64_t n, uint64_t stride, cudaStream_t s);  // d[i] = i * stride
cudaError_t launch_sum_lens(const CountParams &P, unsigned long long *d_totals, unsigned long long *d_max, cudaStream_t s);
cudaError_t launch_count_partitions(const CountParams &P, unsigned grid, cudaStream_t s);
// weighted: some input run carries counts, or a partition is large enough to want run-length pre-aggregation
// direct: unweighted, mostly distinct keys -- new keys go straight to the output, no compaction pass (the output then holds one
// entry per INPUT entry, the duplicates' as skipped fillers)
cudaError_t launch_count_partitions_smem(const CountParams &P, bool weighted, bool direct, cudaStream_t s);
// sieve: unweighted, mostly distinct keys -- a bitmap finds the few keys that MAY repeat, only those enter a (small) table; every
// other key is copied to the output in place.  Partitions it cannot take are listed in P.redo_list for the variants above.
// The input runs are raw runs, whose segments are 16-byte aligned and padded to an even length (launch_pad_segments): the copies go
// through the TMA unit and the output segments are the padded inputs.  With P.part_cap set the sieve runs in place.
constexpr uint32_t SIEVE_MAX_ENTRIES = 4096;  // entries of one partition the sieve variant takes (one batch)
cudaError_t launch_count_partitions_sieve(const CountParams &P, cudaStream_t s);
uint32_t sieve_redo_limit_host(uint32_t n_parts);  // more partitions handed back than this: the sieve stopped early, repeat the launch without it
// keys[seg_start[p] + seg_len[p]] = EMPTY_MIX for every segment of odd length (the layout must leave room for it)
cudaError_t launch_pad_segments(uint64_t *keys, const uint64_t *seg_start, const uint64_t *seg_len, uint32_t n_parts, cudaStream_t s);
cudaError_t launch_even_lengths(const uint64_t *seg_len, uint64_t *even_len, uint32_t n_parts, cudaStream_t s);  // even_len[p] = seg_len[p] rounded up to even
// tmp == nullptr: returns the scratch size needed for n items in *tmp_bytes.  Asynchronous on s.
cudaError_t exclusive_sum_u64(const uint64_t *d_in, uint64_t *d_out, uint64_t n, void *tmp, size_t *tmp_bytes, cudaStream_t s);
int num_sms();
cudaError_t launch_table_init(HashTable t, cudaStream_t s, uint64_t empty = ~0ull);  // empty: EMPTY_KEY, or EMPTY_MIX for phase B scratch
cudaError_t launch_insert_keys(HashTable t, const uint64_t *d_keys, const uint64_t *d_counts, uint64_t n,
                               unsigned long long *counters, cudaStream_t s);
cudaError_t launch_insert_keys_dense(unsigned long long *dense, const uint64_t *d_keys, const uint64_t *d_counts, uint64_t n,
                                     unsigned long long *counters, cudaStream_t s);
cudaError_t launch_rehash(HashTable from, HashTable to, unsigned long long *counters, cudaStream_t s);
cudaError_t launch_table_stats(const TableView &v, uint64_t min_count, unsigned long long *d_stats3, cudaStream_t s);
cudaError_t launch_compact(const TableView &v, uint64_t min_count, uint64_t *d_keys, uint64_t *d_counts, uint64_t cap_out,
                           unsigned long long *d_cursor, cudaStream_t s);
cudaError_t launch_histogram(const TableView &v, uint64_t min_count, unsigned long long *d_bins, uint64_t *d_overflow,
                             uint64_t overflow_cap, unsigned long long *d_overflow_n, cudaStream_t s);
// bucket_counts[key >> shift] += 1 for every entry (KEY_BUCKETS bins, zeroed by this call)
cudaError_t launch_key_buckets(const TableView &v, int shift, unsigned long long *d_bucket_counts, cudaStream_t s);
// FASTA / FASTQ parsing on the device (kmg_count_fastx): see kmg_kernels.cu
cudaError_t launch_fastx_parse(const uint8_t *d_buf, uint64_t n, int is_fastq, uint8_t *d_kind, uint8_t *d_keep, uint32_t *d_lineno, uint32_t *d_pos_s,
                               uint32_t *d_pos_q, void *d_scan_tmp, size_t scan_tmp_bytes, uint64_t carry, uint8_t *d_out_seq, uint8_t *d_out_qual,
                               uint8_t *d_out_mark, unsigned long long *d_n_records, uint32_t *d_err, uint32_t *h_totals_pinned, cudaStream_t s);
size_t fastx_scan_tmp_bytes(uint64_t n);
cudaError_t launch_fastx_scatter(const uint8_t *d_buf, uint64_t n, int is_fastq, const uint8_t *d_kind, const uint32_t *d_lineno, const uint8_t *d_keep,
                                 const uint32_t *d_pos_s, const uint32_t *d_pos_q, uint64_t carry, uint64_t total_s, uint8_t *d_out_seq, uint8_t *d_out_qual,
                                 uint8_t *d_out_mark, unsigned long long *d_n_records, uint32_t *d_err, cudaStream_t s);
cudaError_t launch_fastx_apply_pending(uint32_t *d_pending, uint8_t *d_mark_first_new, cudaStream_t s);
cudaError_t launch_marks_to_bits(const uint8_t *d_mark, uint64_t n_bases, uint64_t n_words_total, uint32_t *d_start, cudaStream_t s);
// index queries / loading
cudaError_t launch_query_pack(const uint8_t *d_kmers, uint64_t n, int k, uint64_t *d_keys, cudaStream_t s);
cudaError_t launch_query(const TableView &v, HashTable t, const uint64_t *d_seg_start, const uint64_t *d_seg_len, uint32_t n_coarse, uint32_t n_sub,
                         uint32_t shard_world, uint32_t shard_rank, const uint64_t *d_keys, uint64_t n, uint64_t *d_counts, cudaStream_t s);
cudaError_t launch_deinterleave_pairs(const void *d_in, uint64_t n, uint64_t *d_keys, uint64_t *d_counts, cudaStream_t s);
// text emitters / index records of a sorted piece (formatting happens on the device).  format is a KMG_TEXT_* code; first != 0:
// record 0 of the piece is the first record of the whole output (json puts no "," in front of it)
cudaError_t launch_text_len(const uint64_t *d_counts, uint64_t n, int k, int format, int first, uint64_t *d_lens, cudaStream_t s);
cudaError_t launch_text_write(const uint64_t *d_keys, const uint64_t *d_counts, const uint64_t *d_offs, uint64_t n, int k, int format, int first,
                              uint8_t *d_out, cudaStream_t s);
cudaError_t launch_interleave_pairs(const uint64_t *d_keys, const uint64_t *d_counts, uint64_t n, void *d_out, cudaStream_t s);
// text file of a shard group: up to MERGE_MAX_RUNS sorted (key, count) runs, possibly in other GPUs' memory (P2P / IPC mapped),
// merged into one sorted local run.  The runs' keys must be pairwise distinct (a key lives on one shard only).
constexpr int MERGE_MAX_RUNS = 8;
struct MergeRuns {
  const uint64_t *keys[MERGE_MAX_RUNS];
  const uint64_t *counts[MERGE_MAX_RUNS];
  uint64_t len[MERGE_MAX_RUNS];
  uint32_t n_runs;
};
// d_out[i] = lower_bound(d_keys[0, n), cut_keys[i]) for i < n_cuts (<= MERGE_MAX_RUNS + 1): where each piece of a step starts
cudaError_t launch_piece_bounds(const uint64_t *d_keys, uint64_t n, const uint64_t *cut_keys, uint32_t n_cuts, uint64_t *d_out, cudaStream_t s);
// out[0, sum of len) = the merged runs; *d_placed (zeroed here) += records written in ascending order (== the total unless two
// runs shared a key)
cudaError_t launch_merge_shard_pieces(const MergeRuns &R, uint64_t *d_keys_out, uint64_t *d_counts_out, unsigned long long *d_placed,
                                      cudaStream_t s);
uint64_t kernel_launches();  // number of kernels of this library launched so far (process-wide)
cudaError_t sort_pairs(uint64_t *d_keys, uint64_t *d_counts, uint64_t n, int key_bits, cudaStream_t s);

}  // namespace kmg
