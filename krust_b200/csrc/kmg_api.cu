// C-ABI layer of libkmerust_gpu (include/kmerust_gpu.h): context, device memory pool, the staging ring of the
// host feed, the choice between the three counting paths (direct 4^k array, one HBM table, partitioned pipeline) and
// its adaptation to a growing input (table growth, migration to the partitioned path, speculative layouts with
// exact fallback, re-split / multi-pass when the partition plan is outgrown), consolidation of the runs, result export.
// The counting itself happens in the sm_100a kernels of kmg_kernels.cu / kmg_partition.cu.  There is no CPU
// fallback: every entry point needs a CUDA device.
#include <fcntl.h>
#include <sched.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/kmerust_gpu.h"
#include "kmg_device.cuh"
#include "kmg_kernels.h"

using namespace kmg;

#define KMG_EXPORT extern "C" __attribute__((visibility("default")))

namespace {

thread_local std::string g_create_error;

constexpr double LOAD_TARGET = 0.60;  // sizing goal when memory allows
constexpr double LOAD_SOFT = 0.70;    // grow after a batch if exceeded and memory allows
constexpr double LOAD_HARD = 0.90;    // never start a batch that could exceed this
constexpr uint64_t DEFAULT_BATCH_BASES = 1ull << 28;  // per staging slot; every batch becomes one run of the partitioned pipeline
constexpr int N_STAGE = 4;                             // ASCII staging ring: copies run up to 3 chunks ahead of the kernels
constexpr uint64_t MIN_TABLE_SLOTS = 1ull << 16;

struct Staging {
  uint8_t *h_seq = nullptr, *h_qual = nullptr;  // pinned (lazily allocated; skipped for pinned callers)
  uint64_t *h_off = nullptr;
  uint8_t *d_seq = nullptr, *d_qual = nullptr;
  uint64_t *d_off = nullptr;
  uint64_t off_cap = 0;
  cudaEvent_t h2d_done = nullptr, compute_done = nullptr;
  bool h2d_pending = false, compute_pending = false;
  // pre-packed feed (kmg_acquire_batch)
  uint64_t *hp_bases = nullptr;
  uint32_t *hp_valid = nullptr, *hp_start = nullptr;
  uint64_t *dp_bases = nullptr;                      // the slot's packed stream on the device (with the zero lead-in words)
  uint32_t *dp_valid = nullptr, *dp_start = nullptr;
  uint64_t hp_used_words = 0;                        // words the last producer may have written
};

}  // namespace

// A run is a partition-indexed list of keys (phase A output, every key counts 1) or of (key, count)
// pairs (phase B output / weighted inserts).  All runs of a context share the same partition count;
// partition p of a run is entries [seg_start[p], seg_start[p] + seg_len[p]).  A run built by refine_to_run (a raw run, or weighted
// keys) is padded: its segments start on 16-byte boundaries and an EMPTY_MIX key follows every segment of odd length.
struct Run {
  uint64_t *d_keys = nullptr, *d_counts = nullptr, *d_seg_start = nullptr, *d_seg_len = nullptr;
  uint64_t n = 0;        // entries (a consolidated run may hold skipped filler entries, see count_partitions_smem_kernel)
  uint64_t n_valid = 0;  // consolidated runs: distinct keys
  uint64_t part_cap = 0;  // raw run in the speculative layout: partition p owns entries [p * part_cap, (p + 1) * part_cap); 0: exact layout
};

struct kmg_ctx {
  kmg_config cfg{};
  int device = 0;
  int k = 0;
  bool use_dense = false;
  cudaStream_t stream = nullptr, copy_stream = nullptr;
  bool own_stream = false;
  std::string err;

  // table
  HashTable table{nullptr, 0};
  unsigned long long *dense = nullptr;
  uint64_t dense_n = 0;
  uint64_t distinct_ub = 0;  // upper bound of distinct keys currently in the table
  uint32_t n_grows = 0;

  unsigned long long *d_counters = nullptr;  // CTR_N
  unsigned long long *h_counters = nullptr;  // pinned mirror
  unsigned long long *d_stats = nullptr;     // 3 + cursor + overflow_n

  // packed stream buffers (grown on demand)
  uint64_t *d_bases = nullptr;
  uint32_t *d_valid = nullptr, *d_start = nullptr;
  uint64_t packed_words = 0;  // capacity in words (excluding lead-in)

  uint64_t batch_bases = DEFAULT_BATCH_BASES;
  Staging st[N_STAGE];
  bool staging_ready = false, packed_feed_ready = false;
  uint64_t staging_cap = 0;
  uint32_t next_slot = 0;    // pre-packed feed: next ring slot to hand out
  int pending_slot = -1;     // pre-packed feed: batch whose copy is queued but which has not been scanned yet
  uint64_t pending_words = 0, dp_words = 0;
  uint32_t next_ascii = 0;   // ASCII staging ring

  // partitioned pipeline (v2)
  enum Mode { MODE_UNDECIDED, MODE_DENSE, MODE_TABLE, MODE_PARTITIONED } mode = MODE_UNDECIDED;
  uint32_t n_parts = 0, n_coarse = 0, n_sub = 0, scratch_log2 = 13;
  std::vector<Run> runs;      // pending, not yet consolidated
  Run result;                 // consolidated (key, count) run
  bool has_result = false;
  bool spec_coarse_ok = true;  // same for the level-1 scatter
  bool spec_fine_ok = true;  // level-2 scatter without a count pass until a partition overflows its share
  size_t total_mem = 0;                      // device memory size (cudaMemGetInfo is slow; asked once)
  void *d_scan_tmp = nullptr;                // CUB scan scratch for scan_tmp_items items
  size_t scan_tmp_bytes = 0;
  uint64_t scan_tmp_items = 0, fine_cursor_items = 0;
  bool in_resplit = false;
  struct FxStream *fxs = nullptr;    // an open FASTA / FASTQ stream (kmg_fastx_stream_begin .. _end)
  std::vector<uint8_t> fx_rest;      // the bytes a refused stream did not count (kmg_fastx_stream_rest)
  bool fx_rest_ok = false;
  struct ShardShm *shm = nullptr;     // sharded mode (kmg_shard_join): the group's shared segment
  uint32_t sh_world = 1, sh_rank = 0;
  uint64_t *sh_recv = nullptr;        // this rank's SEND buffer: two halves of sh_recv_entries keys (owners pull their regions over NVLink)
  uint64_t sh_recv_entries = 0;
  uint64_t *sh_peer[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // every rank's send buffer as seen from here
  bool sh_peer_ipc[8] = {false, false, false, false, false, false, false, false};
  int sh_pid[8] = {}, sh_device[8] = {};  // every rank's process and device (kmg_shard_join)
  uint64_t sh_gathers = 0;                // shard_allgather calls since kmg_shard_join: the parity picks the post area's half
  uint64_t sh_sent = 0, sh_recv_keys = 0, sh_rounds = 0, sh_exact_rounds = 0;
  std::vector<uint64_t> sh_hist_vals, sh_hist_freqs;  // merged histogram of the last kmg_shard_histogram
  int feed_kind = 0;        // partitioned path: 1 = runs binned by this context's own coarse function, 2 = blocks adopted from a sender
                            // that binned by (owner, bin) -- the two bin functions differ, so one context takes only one kind
  bool poisoned = false;    // a re-split failed half way: runs with different partitionings coexist; only kmg_reset / kmg_destroy are safe
  double dedup_ratio = 1.0;  // distinct keys per raw entry seen by the last consolidation (sizes the next consolidated run)
  double plan_scale = 1.0;  // kmg_count_ascii with a quality filter: (bases of the whole call) / (bases of its first chunk)
  int building_run = 0;  // > 0 while refine_to_run derives a run from the current plan: a nested consolidate must not re-split
  // count-of-counts of `result`, produced by phase B itself (consolidate)
  unsigned long long *d_hist = nullptr;      // HIST_DENSE_BINS bins + overflow counter
  uint64_t *d_hist_ov = nullptr;             // HIST_OVERFLOW_CAP counts >= HIST_DENSE_BINS
  bool fused_valid = false, fused_cached = false;
  std::vector<unsigned long long> h_bins;    // host copy, bins[1] filled in
  std::vector<uint64_t> h_ov;                // ascending
  uint64_t fused_sum = 0, fused_max = 0;
  uint64_t pending_bytes = 0;
  unsigned long long *d_part = nullptr;  // 3 * MAX_PARTS scratch: coarse counts, starts, cursors
  unsigned long long *d_fine_cursor = nullptr;  // n_parts
  uint32_t n_consolidations = 0;
  uint64_t sieve_redo = 0;  // partitions the sieve variant of phase B handed to the compacting variant (diagnostic)

  // device-memory pool for the partitioned pipeline's large, short-lived buffers: cudaMalloc/cudaFree of tens
  // of GB cost ~10 ms each and a counting job needs a dozen of them, so freed blocks are kept for reuse
  std::vector<std::pair<void *, size_t>> pool_idle;
  std::unordered_map<void *, size_t> pool_live;

  uint64_t n_records = 0, n_bases = 0, h2d_bytes = 0;
  cudaEvent_t ev_a = nullptr, ev_b = nullptr;
  double kernel_ms = 0.0;
  double cat_ms[3] = {0.0, 0.0, 0.0};  // 0: scan / partition kernels (includes 2), 1: consolidation kernel, 2: refine (A2) launches, nested inside 0
  struct Timer { cudaEvent_t a, b; int cat; };
  std::vector<Timer> pending_timers;
};

namespace {

void shard_release(kmg_ctx *c);  // defined with the shard group code below
void fx_stream_close(kmg_ctx *c, bool failed);  // abandons an open FASTA / FASTQ stream (defined with kmg_fastx_stream_begin)
kmg_status scan_pending_batch(kmg_ctx *c);  // pre-packed feed: scan the batch whose copy is in flight (defined with kmg_submit_batch)

kmg_status fail(kmg_ctx *ctx, kmg_status s, const std::string &msg) {
  if (ctx) ctx->err = msg; else g_create_error = msg;
  return s;
}
kmg_status cuda_fail(kmg_ctx *ctx, cudaError_t e, const char *what) {
  kmg_status s = (e == cudaErrorMemoryAllocation) ? KMG_ERR_OOM : KMG_ERR_CUDA;
  return fail(ctx, s, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU(ctx, call)                                            \
  do {                                                           \
    cudaError_t _e = (call);                                     \
    if (_e != cudaSuccess) return cuda_fail(ctx, _e, #call);     \
  } while (0)

// every feed and every call that reads the table waits for an open FASTA / FASTQ stream to end
#define NO_OPEN_STREAM(ctx)                                                                                                        \
  do {                                                                                                                             \
    if ((ctx)->fxs) return fail(ctx, KMG_ERR_STATE, "a FASTA / FASTQ stream is open on this context: end it with kmg_fastx_stream_end (or kmg_reset)"); \
  } while (0)

inline uint64_t round_up(uint64_t x, uint64_t m) { return (x + m - 1) / m * m; }

void pool_release_idle(kmg_ctx *c) {
  for (auto &b : c->pool_idle) cudaFree(b.first);
  c->pool_idle.clear();
}
cudaError_t pool_alloc(kmg_ctx *c, void **p, size_t bytes) {
  bytes = std::max<size_t>(bytes, 256);
  size_t best = SIZE_MAX, best_i = 0;
  for (size_t i = 0; i < c->pool_idle.size(); ++i) {
    const size_t sz = c->pool_idle[i].second;
    if (sz >= bytes && sz <= bytes + bytes / 8 + (1u << 20) && sz < best) { best = sz; best_i = i; }
  }
  if (best != SIZE_MAX) {
    *p = c->pool_idle[best_i].first;
    c->pool_live[*p] = best;
    c->pool_idle.erase(c->pool_idle.begin() + best_i);
    return cudaSuccess;
  }
  cudaError_t e = cudaMalloc(p, bytes);
  if (e != cudaSuccess) {  // give idle blocks back to the driver and retry once
    cudaGetLastError();
    pool_release_idle(c);
    e = cudaMalloc(p, bytes);
  }
  if (e == cudaSuccess) c->pool_live[*p] = bytes;
  return e;
}
template <class T>
cudaError_t pool_alloc(kmg_ctx *c, T **p, size_t bytes) { return pool_alloc(c, reinterpret_cast<void **>(p), bytes); }
void pool_free(kmg_ctx *c, void *p) {
  if (!p) return;
  auto it = c->pool_live.find(p);
  if (it == c->pool_live.end()) { cudaFree(p); return; }
  c->pool_idle.emplace_back(p, it->second);
  c->pool_live.erase(it);
}

TableView view_of(const kmg_ctx *c) {
  TableView v{nullptr, nullptr, nullptr, nullptr, 0};
  if (c->mode == kmg_ctx::MODE_PARTITIONED) { v.pair_keys = c->result.d_keys; v.pair_counts = c->result.d_counts; v.n = c->has_result ? c->result.n : 0; }
  else if (c->use_dense) { v.dense = c->dense; v.n = c->dense_n; }
  else { v.slots = c->table.slots; v.n = c->table.slots ? c->table.cap : 0; }
  return v;
}

void free_run(kmg_ctx *c, Run &r) {
  pool_free(c, r.d_keys); pool_free(c, r.d_counts); pool_free(c, r.d_seg_start); pool_free(c, r.d_seg_len);
  r = Run();
}

kmg_status alloc_table(kmg_ctx *c, uint64_t cap, HashTable *out) {
  cap = std::max<uint64_t>(cap, MIN_TABLE_SLOTS);
  cap = round_up(cap, 2);
  uint64_t *p = nullptr;
  cudaError_t e = cudaMalloc(&p, cap * 16);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(c, KMG_ERR_OOM, "cudaMalloc(table) failed: " + std::string(cudaGetErrorString(e))); }
  out->slots = p; out->cap = cap;
  CU(c, launch_table_init(*out, c->stream));
  return KMG_OK;
}

// Try target loads from generous to tight until an allocation succeeds.
kmg_status alloc_table_for(kmg_ctx *c, uint64_t need_keys, HashTable *out) {
  const double loads[3] = {LOAD_TARGET, 0.75, LOAD_HARD};
  kmg_status s = KMG_ERR_OOM;
  for (double l : loads) {
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    uint64_t cap = (uint64_t)((double)need_keys / l) + 2;
    if (cap * 16 > (uint64_t)free_b) continue;
    s = alloc_table(c, cap, out);
    if (s == KMG_OK) return s;
  }
  return fail(c, KMG_ERR_TABLE_FULL, "cannot allocate a table for " + std::to_string(need_keys) + " keys");
}

kmg_status read_counters(kmg_ctx *c) {
  CU(c, cudaMemcpyAsync(c->h_counters, c->d_counters, CTR_N * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  if (c->h_counters[CTR_FULL]) return fail(c, KMG_ERR_TABLE_FULL, "hash table filled up during a batch (capacity planning bug)");
  return KMG_OK;
}

kmg_status grow_table(kmg_ctx *c, uint64_t need_keys) {
  HashTable nt{nullptr, 0};
  kmg_status s = alloc_table_for(c, need_keys, &nt);
  if (s != KMG_OK) return s;
  if (nt.cap <= c->table.cap) { cudaFree(nt.slots); return fail(c, KMG_ERR_TABLE_FULL, "table cannot grow any further"); }
  CU(c, launch_rehash(c->table, nt, c->d_counters, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  cudaFree(c->table.slots);
  c->table = nt;
  c->n_grows++;
  return KMG_OK;
}

// Make sure `incoming` more upserts cannot push the load above LOAD_HARD.  Returns how many of them
// may be issued now (>= 1 tile's worth or an error).
kmg_status reserve_capacity(kmg_ctx *c, uint64_t incoming, uint64_t *granted) {
  *granted = incoming;
  if (c->use_dense) return KMG_OK;
  auto room = [&]() -> uint64_t {
    uint64_t lim = (uint64_t)(LOAD_HARD * (double)c->table.cap);
    return lim > c->distinct_ub ? lim - c->distinct_ub : 0;
  };
  if (incoming <= room()) { c->distinct_ub += incoming; return KMG_OK; }
  kmg_status s = read_counters(c);  // exact distinct count
  if (s != KMG_OK) return s;
  c->distinct_ub = c->h_counters[CTR_DISTINCT];
  if (incoming <= room() && (double)c->distinct_ub <= LOAD_SOFT * (double)c->table.cap) { c->distinct_ub += incoming; return KMG_OK; }
  // grow: enough for what is there plus the incoming batch
  s = grow_table(c, c->distinct_ub + incoming);
  if (s != KMG_OK) {
    // could not grow: hand out whatever room is left (caller splits the batch)
    uint64_t r = room();
    if (r < (uint64_t)TILE_WORDS * 32) return s;
    c->err.clear();
    *granted = std::min(incoming, r);
  }
  c->distinct_ub += *granted;
  return KMG_OK;
}

kmg_status ensure_packed(kmg_ctx *c, uint64_t n_words_total) {
  if (n_words_total <= c->packed_words) return KMG_OK;
  CU(c, cudaStreamSynchronize(c->stream));
  cudaFree(c->d_bases); cudaFree(c->d_valid); cudaFree(c->d_start);
  c->d_bases = nullptr; c->d_valid = c->d_start = nullptr; c->packed_words = 0;
  CU(c, cudaMalloc(&c->d_bases, (LEAD_BASE_WORDS + n_words_total) * 8));
  CU(c, cudaMalloc(&c->d_valid, (LEAD_MASK_WORDS + n_words_total) * 4));
  CU(c, cudaMalloc(&c->d_start, (LEAD_MASK_WORDS + n_words_total) * 4));
  CU(c, cudaMemsetAsync(c->d_bases, 0, LEAD_BASE_WORDS * 8, c->stream));
  CU(c, cudaMemsetAsync(c->d_valid, 0, LEAD_MASK_WORDS * 4, c->stream));
  CU(c, cudaMemsetAsync(c->d_start, 0, LEAD_MASK_WORDS * 4, c->stream));
  c->packed_words = n_words_total;
  return KMG_OK;
}

size_t timer_begin(kmg_ctx *c, int cat = 0) {
  cudaEvent_t a, b;
  cudaEventCreate(&a); cudaEventCreate(&b);
  cudaEventRecord(a, c->stream);
  c->pending_timers.push_back(kmg_ctx::Timer{a, b, cat});
  return c->pending_timers.size() - 1;
}
void timer_end(kmg_ctx *c, size_t idx) { cudaEventRecord(c->pending_timers[idx].b, c->stream); }
void timers_collect(kmg_ctx *c) {
  for (auto &p : c->pending_timers) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) { if (p.cat != 2) c->kernel_ms += ms; c->cat_ms[p.cat] += ms; }
    cudaEventDestroy(p.a); cudaEventDestroy(p.b);
  }
  c->pending_timers.clear();
}


// =================================================================================================
// Partitioned pipeline: A1 coarse scatter, A2 refine to fine partitions, B per-CTA counting
// (kernels and rationale: kmg_partition.cu).
// =================================================================================================
constexpr uint64_t TARGET_KEYS_PER_PART = 3600;  // <= 4096 with 8 sigma to spare: one upsert round per partition; load ~0.44
// entries one refine_to_run call takes: the exact layout places them at 32-bit positions, with room for one pad entry per
// partition (at most 2048 x 2048)
constexpr uint64_t REFINE_MAX_ENTRIES = (1ull << 32) - 2048ull * 2048;

// n_coarse / n_sub are set: allocate the partitioned pipeline's bookkeeping
kmg_status init_partitioned(kmg_ctx *c) {
  c->n_parts = c->n_coarse * c->n_sub;
  CU(c, cudaMalloc(&c->d_part, 3 * (size_t)MAX_PARTS * sizeof(unsigned long long)));
  CU(c, cudaMalloc(&c->d_fine_cursor, (size_t)c->n_parts * sizeof(unsigned long long)));
  c->fine_cursor_items = c->n_parts;
  return KMG_OK;
}

// Decide how this context counts.  Called at the first feeding call, when the input size is known.
kmg_status decide_mode(kmg_ctx *c, uint64_t first_call_windows) {
  if (c->mode != kmg_ctx::MODE_UNDECIDED) return KMG_OK;
  if (c->use_dense) { c->mode = kmg_ctx::MODE_DENSE; return KMG_OK; }
  const uint32_t f = c->cfg.flags;
  const uint64_t hint = c->cfg.expected_distinct ? c->cfg.expected_distinct : first_call_windows;  // an explicit hint is taken at its word
  const bool part = (f & KMG_FLAG_FORCE_PARTITIONED) || (!(f & KMG_FLAG_FORCE_HASH) && hint >= (1ull << 25));
  if (!part) {
    c->mode = kmg_ctx::MODE_TABLE;
    if (!c->table.slots) {
      kmg_status s = c->cfg.expected_distinct ? alloc_table_for(c, c->cfg.expected_distinct, &c->table) : alloc_table(c, 1ull << 22, &c->table);
      if (s != KMG_OK) return s;
    }
    return KMG_OK;
  }
  c->mode = kmg_ctx::MODE_PARTITIONED;
  if (c->cfg.parts_log2) {
    const uint32_t lg = std::min<uint32_t>(c->cfg.parts_log2, 20);
    c->n_coarse = 1u << (lg / 2);
    c->n_sub = 1u << (lg - lg / 2);
  } else {
    const uint64_t want = std::max<uint64_t>(4, (hint + TARGET_KEYS_PER_PART - 1) / TARGET_KEYS_PER_PART);
    uint64_t p1 = 1;
    while (p1 * p1 < want) ++p1;
    p1 = std::min<uint64_t>(p1, 2048);
    c->n_coarse = (uint32_t)p1;
    c->n_sub = (uint32_t)std::min<uint64_t>((want + p1 - 1) / p1, 2048);
  }
  return init_partitioned(c);
}

kmg_status consolidate(kmg_ctx *c, bool recompact = false);

kmg_status add_run(kmg_ctx *c, Run &&r) {
  if (r.n == 0) { free_run(c, r); return KMG_OK; }
  c->pending_bytes += r.n * (r.d_counts ? 16 : 8);
  c->runs.push_back(std::move(r));
  if (!c->total_mem) { size_t free_b = 0; cudaMemGetInfo(&free_b, &c->total_mem); }
  const size_t total_b = c->total_mem;
  // consolidate early when the pending runs get numerous or large (keeps streaming inputs bounded in memory)
  if (c->runs.size() + (c->has_result ? 1 : 0) >= (size_t)CONS_MAX_RUNS - 1 || c->pending_bytes > (uint64_t)total_b * 20 / 100)
    return consolidate(c);
  return KMG_OK;
}

// allocate with one retry after consolidating what is pending (frees the pending runs' buffers)
kmg_status alloc_or_consolidate(kmg_ctx *c, void **p, size_t bytes, const char *what) {
  cudaError_t e = pool_alloc(c, p, bytes ? bytes : 1);
  if (e == cudaSuccess) return KMG_OK;
  cudaGetLastError();
  if (c->in_resplit) return fail(c, KMG_ERR_OOM, std::string("cudaMalloc(") + what + ") failed while re-splitting the runs");
  kmg_status s = consolidate(c);
  if (s != KMG_OK) return s;
  e = pool_alloc(c, p, bytes ? bytes : 1);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(c, KMG_ERR_OOM, std::string("cudaMalloc(") + what + ") failed"); }
  return KMG_OK;
}

// A2: coarse-partitioned keys (+counts) -> fine-partitioned run.  Takes ownership of the coarse buffers when `owns`.
// `sync`: wait for the scatter before returning (needed when the input belongs to the caller).  Without it the coarse
// buffers go back to the pool while the kernels are still queued, which is safe because every pool block is only ever
// touched by work on c->stream (stream-ordered reuse).
// coarse_len == nullptr: coarse partition p is [coarse_off[p], coarse_off[p + 1]); otherwise [coarse_off[p], coarse_off[p] + len[p]).
// `split` != nullptr: the input is a fine-partitioned run (split->n_in partitions) that is re-split split->m ways; the new run is
// returned in *split->out instead of being added to the pending runs.
struct SplitPlan { uint32_t n_in, m, sub_old; Run *out; };
kmg_status refine_to_run(kmg_ctx *c, uint64_t *d_ckeys, uint64_t *d_ccounts, const std::vector<uint64_t> &coarse_off, bool owns = true,
                         bool sync = true, const std::vector<uint64_t> *coarse_len = nullptr, const SplitPlan *split = nullptr,
                         bool in_keys = false,    // in_keys: the input holds plain keys, not mixes (blocks adopted from another rank)
                         uint32_t in_group = 1,   // in_group g: coarse bin b arrives as the g input partitions b*g .. b*g+g-1 (sharded: one per source rank)
                         const uint64_t *const *src = nullptr) {  // src[s]: input partition p is read from src[p % in_group] (other ranks' send buffers)
  struct BuildGuard {
    kmg_ctx *c;
    explicit BuildGuard(kmg_ctx *c_) : c(c_) { ++c->building_run; }
    void release() { if (c) { --c->building_run; c = nullptr; } }
    ~BuildGuard() { release(); }
  } guard(c);
  const uint32_t P1 = split ? split->n_in : c->n_coarse * in_group;  // input partitions
  const uint32_t n_sub = split ? split->m : c->n_sub;
  const uint32_t P = split ? split->n_in * split->m : c->n_parts;
  auto len_of = [&](uint32_t p) { return coarse_len ? (*coarse_len)[p] : coarse_off[p + 1] - coarse_off[p]; };
  uint64_t n = 0;
  for (uint32_t p = 0; p < P1; ++p) n += len_of(p);
  Run r;
  uint64_t *d_cstart = nullptr, *d_clen = nullptr;
  uint32_t *d_tprefix = nullptr;
  auto cleanup = [&]() { if (owns) { pool_free(c, d_ckeys); pool_free(c, d_ccounts); } pool_free(c, d_cstart); pool_free(c, d_clen); pool_free(c, d_tprefix); };
  if (n + P > (1ull << 32)) { cleanup(); return fail(c, KMG_ERR_STATE, "refine: more entries than 32-bit positions hold with a pad entry per partition"); }
  // both layouts end here: the pad entries behind odd segments, then the run is handed over
  auto finish = [&]() -> kmg_status {
    const cudaError_t pe = launch_pad_segments(r.d_keys, r.d_seg_start, r.d_seg_len, P, c->stream);
    if (pe != cudaSuccess) { free_run(c, r); return cuda_fail(c, pe, "pad segments"); }
    r.n = n;
    if (split) { *split->out = std::move(r); return KMG_OK; }
    guard.release();  // the run is complete: a consolidation triggered by add_run may re-split it with the others
    return add_run(c, std::move(r));
  };
  std::vector<uint32_t> tprefix(P1 + 1, 0);
  uint64_t tiles = 0;
  for (uint32_t p = 0; p < P1; ++p) { tprefix[p] = (uint32_t)tiles; tiles += (len_of(p) + REFINE_TILE - 1) / REFINE_TILE; }
  tprefix[P1] = (uint32_t)tiles;
  cudaError_t e = cudaSuccess;
  if (c->fine_cursor_items < P) {  // the partition count grew (re-split)
    CU(c, cudaStreamSynchronize(c->stream));
    cudaFree(c->d_fine_cursor); c->d_fine_cursor = nullptr; c->fine_cursor_items = 0;
    CU(c, cudaMalloc(&c->d_fine_cursor, (size_t)P * sizeof(unsigned long long)));
    c->fine_cursor_items = P;
  }
  e = pool_alloc(c, &d_cstart, (P1 + 1) * 8);
  if (e == cudaSuccess && coarse_len) {
    e = pool_alloc(c, &d_clen, (size_t)P1 * 8);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_clen, coarse_len->data(), (size_t)P1 * 8, cudaMemcpyHostToDevice, c->stream);
  }
  if (e == cudaSuccess) e = pool_alloc(c, &d_tprefix, (P1 + 1) * 4);
  if (e == cudaSuccess) e = pool_alloc(c, &r.d_seg_start, (size_t)P * 8);
  if (e == cudaSuccess) e = pool_alloc(c, &r.d_seg_len, (size_t)P * 8);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_cstart, coarse_off.data(), (P1 + 1) * 8, cudaMemcpyHostToDevice, c->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_tprefix, tprefix.data(), (P1 + 1) * 4, cudaMemcpyHostToDevice, c->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(r.d_seg_len, 0, (size_t)P * 8, c->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(c->d_fine_cursor, 0, (size_t)P * 8, c->stream);
  if (e != cudaSuccess) { cleanup(); free_run(c, r); return cuda_fail(c, e, "refine setup"); }
  RefineParams rp{};
  rp.keys = d_ckeys; rp.counts = d_ccounts; rp.coarse_start = d_cstart; rp.coarse_len = d_clen; rp.tile_prefix = d_tprefix;
  rp.n_coarse = P1; rp.n_sub = n_sub; rp.n_tiles = (uint32_t)tiles;
  if (split) { rp.sub_total = split->sub_old * split->m; rp.sub_old = split->sub_old; }
  rp.in_keys = in_keys ? 1u : 0u;
  rp.in_group = in_group;
  if (src) { rp.n_src = in_group; for (uint32_t i = 0; i < in_group && i < 8; ++i) rp.src[i] = src[i]; }
  // Speculative layout first: hash partitions are Poisson-sized, so every fine partition gets mean + 7 sigma + 16 slots
  // and the count pass (a full read of the keys) is skipped.  Skewed input overflows a share: the kernel then raises a
  // flag, and this chunk -- and, sticky, the rest of the job -- takes the exact count + prefix + scatter route below.
  const double mu = (double)n / P;
  const uint64_t cap_f = ((uint64_t)(mu + 7.0 * std::sqrt(mu) + 16.0) + 7) & ~7ull;
  if (c->spec_fine_ok && mu >= 64.0 && cap_f * P < (1ull << 32) && refine_single_pass_available(n_sub, d_ccounts != nullptr)) {
    kmg_status s = alloc_or_consolidate(c, reinterpret_cast<void **>(&r.d_keys), cap_f * P * 8, "fine keys");
    if (s != KMG_OK) { cleanup(); free_run(c, r); return s; }
    rp.fine_cap = cap_f;
    rp.fine_cursor = reinterpret_cast<unsigned long long *>(r.d_seg_len);  // zeroed above; ends up as the partition sizes
    rp.overflow_flag = reinterpret_cast<uint32_t *>(c->d_stats + 5);
    rp.out_keys = r.d_keys;
    uint32_t h_flag = 0;
    e = cudaMemsetAsync(rp.overflow_flag, 0, 4, c->stream);
    if (e == cudaSuccess) e = launch_fill_strided(r.d_seg_start, P, cap_f, c->stream);
    const size_t tmr2 = timer_begin(c, 2);
    if (e == cudaSuccess) e = launch_refine(rp, true, c->stream);
    timer_end(c, tmr2);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h_flag, rp.overflow_flag, 4, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) { cleanup(); free_run(c, r); return cuda_fail(c, e, "refine scatter (speculative layout)"); }
    if (!h_flag) {
      cleanup();
      r.part_cap = cap_f;
      return finish();
    }
    c->spec_fine_ok = false;
    pool_free(c, r.d_keys); r.d_keys = nullptr;
    rp.fine_cap = 0; rp.overflow_flag = nullptr; rp.out_keys = nullptr;
    e = cudaMemsetAsync(r.d_seg_len, 0, (size_t)P * 8, c->stream);
    if (e != cudaSuccess) { cleanup(); free_run(c, r); return cuda_fail(c, e, "refine setup"); }
  }
  rp.fine_counts = reinterpret_cast<unsigned long long *>(r.d_seg_len);
  rp.fine_start = reinterpret_cast<const unsigned long long *>(r.d_seg_start);
  rp.fine_cursor = c->d_fine_cursor;
  const size_t tmr3 = timer_begin(c, 2);
  e = launch_refine(rp, false, c->stream);
  timer_end(c, tmr3);
  if (e == cudaSuccess && (!c->d_scan_tmp || c->scan_tmp_items < P)) {
    cudaFree(c->d_scan_tmp); c->d_scan_tmp = nullptr;
    e = exclusive_sum_u64(nullptr, nullptr, P, nullptr, &c->scan_tmp_bytes, c->stream);
    if (e == cudaSuccess) e = cudaMalloc(&c->d_scan_tmp, c->scan_tmp_bytes ? c->scan_tmp_bytes : 16);
    c->scan_tmp_items = P;
  }

  // segment p starts at the prefix of the lengths rounded up to even: room for its pad entry, and a 16-byte aligned start
  if (e == cudaSuccess) e = launch_even_lengths(r.d_seg_len, r.d_seg_start, P, c->stream);
  if (e == cudaSuccess) e = exclusive_sum_u64(r.d_seg_start, r.d_seg_start, P, c->d_scan_tmp, &c->scan_tmp_bytes, c->stream);
  if (e != cudaSuccess) { cleanup(); free_run(c, r); return cuda_fail(c, e, "refine count"); }
  kmg_status s = alloc_or_consolidate(c, reinterpret_cast<void **>(&r.d_keys), (n + P) * 8, "fine keys");
  if (s == KMG_OK && d_ccounts) s = alloc_or_consolidate(c, reinterpret_cast<void **>(&r.d_counts), (n + P) * 8, "fine counts");
  if (s != KMG_OK) { cleanup(); free_run(c, r); return s; }
  rp.out_keys = r.d_keys; rp.out_counts = r.d_counts;
  const size_t tmr4 = timer_begin(c, 2);
  e = launch_refine(rp, true, c->stream);
  timer_end(c, tmr4);
  if (e == cudaSuccess && sync) e = cudaStreamSynchronize(c->stream);
  cleanup();
  if (e != cudaSuccess) { free_run(c, r); return cuda_fail(c, e, "refine scatter"); }
  return finish();
}

// A1 over the packed stream: coarse count pass, exact offsets, coarse scatter; then A2.
kmg_status scan_to_run(kmg_ctx *c, uint64_t n_words_total, bool has_start) {
  if (c->poisoned) return fail(c, KMG_ERR_STATE, "context is inconsistent after a failed re-split: kmg_reset it");
  if (c->feed_kind == 2) return fail(c, KMG_ERR_STATE, "context holds blocks adopted from a sender (kmg_adopt_coarse_device): it cannot also scan input itself");
  c->feed_kind = 1;
  const uint64_t n_tiles = n_words_total / TILE_WORDS;
  const uint64_t max_tiles = REFINE_MAX_ENTRIES / ((uint64_t)TILE_WORDS * 32);  // < 2^32 windows per launch, one refine_to_run each
  const uint32_t P1 = c->n_coarse;
  unsigned long long *d_cnt = c->d_part, *d_start = c->d_part + MAX_PARTS, *d_cur = c->d_part + 2 * MAX_PARTS;
  for (uint64_t tile0 = 0; tile0 < n_tiles; tile0 += max_tiles) {
    ScanInput in;
    in.bases = c->d_bases + tile0 * TILE_WORDS;
    in.valid = c->d_valid + tile0 * TILE_WORDS;
    in.start = has_start ? c->d_start + tile0 * TILE_WORDS : nullptr;
    in.n_tiles = std::min(max_tiles, n_tiles - tile0);
    in.k = c->k;
    const size_t tmr = timer_begin(c, 0);
    CU(c, cudaMemsetAsync(c->d_part, 0, 3 * (size_t)MAX_PARTS * sizeof(unsigned long long), c->stream));
    // Speculative layout first (no count pass): hash bins are Poisson-sized, so every coarse bin gets an equal share of
    // (windows of this launch) / P1 + 7 sigma + 1024 slots.  A bin that outgrows its share (heavily repeated k-mers) raises
    // a flag; this launch -- and, sticky, the rest of the job -- then takes the exact count + prefix + scatter route.
    {
      const uint64_t n_ub = in.n_tiles * (uint64_t)TILE_WORDS * 32;
      const double mu = (double)n_ub / P1;
      const uint64_t cap_c = ((uint64_t)(mu + 7.0 * std::sqrt(mu) + 1024.0) + 15) & ~15ull;
      if (c->spec_coarse_ok && cap_c * P1 < (1ull << 32) && scan_scatter_supports_cap(P1)) {
        uint64_t *d_ckeys = nullptr;
        kmg_status s = alloc_or_consolidate(c, reinterpret_cast<void **>(&d_ckeys), cap_c * P1 * 8, "coarse keys");
        if (s != KMG_OK) return s;
        std::vector<uint64_t> off(P1 + 1, 0), lens(P1, 0);
        for (uint32_t p = 0; p <= P1; ++p) off[p] = (uint64_t)p * cap_c;
        ScanInput sin = in;
        sin.part_cap = cap_c;
        sin.overflow_flag = reinterpret_cast<uint32_t *>(c->d_stats + 5);
        uint32_t h_flag = 0;
        cudaError_t e = cudaMemsetAsync(sin.overflow_flag, 0, 4, c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_start, off.data(), P1 * 8, cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess) e = launch_scan_partition(sin, P1, true, d_cnt, d_start, d_cur, d_ckeys, c->d_counters, c->stream, /*mixed=*/true);
        if (e == cudaSuccess) e = cudaMemcpyAsync(lens.data(), d_cur, P1 * 8, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(&h_flag, sin.overflow_flag, 4, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) { pool_free(c, d_ckeys); return cuda_fail(c, e, "coarse scatter (speculative layout)"); }
        if (!h_flag) {
          uint64_t n = 0;
          for (uint32_t p = 0; p < P1; ++p) n += lens[p];
          if (n == 0) { pool_free(c, d_ckeys); timer_end(c, tmr); continue; }
          s = refine_to_run(c, d_ckeys, nullptr, off, /*owns=*/true, /*sync=*/false, &lens);
          timer_end(c, tmr);
          if (s != KMG_OK) return s;
          continue;
        }
        c->spec_coarse_ok = false;
        pool_free(c, d_ckeys);
        CU(c, cudaMemsetAsync(c->d_part, 0, 3 * (size_t)MAX_PARTS * sizeof(unsigned long long), c->stream));
      }
    }
    CU(c, launch_scan_partition(in, P1, false, d_cnt, d_start, d_cur, nullptr, c->d_counters, c->stream));
    std::vector<unsigned long long> counts(P1);
    CU(c, cudaMemcpyAsync(counts.data(), d_cnt, P1 * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    std::vector<uint64_t> off(P1 + 1, 0);
    for (uint32_t p = 0; p < P1; ++p) off[p + 1] = off[p] + counts[p];
    const uint64_t n = off[P1];
    if (n == 0) { timer_end(c, tmr); continue; }
    uint64_t *d_ckeys = nullptr;
    kmg_status s = alloc_or_consolidate(c, reinterpret_cast<void **>(&d_ckeys), n * 8, "coarse keys");
    if (s != KMG_OK) return s;
    CU(c, cudaMemcpyAsync(d_start, off.data(), P1 * 8, cudaMemcpyHostToDevice, c->stream));
    CU(c, launch_scan_partition(in, P1, true, d_cnt, d_start, d_cur, d_ckeys, c->d_counters, c->stream, /*mixed=*/true));
    s = refine_to_run(c, d_ckeys, nullptr, off, /*owns=*/true, /*sync=*/false);  // input is the context's own packed stream
    timer_end(c, tmr);
    if (s != KMG_OK) return s;
  }
  return KMG_OK;
}

// weighted keys (device) -> one run (the receive side of the multi-GPU exchange)
kmg_status keys_to_run(kmg_ctx *c, const uint64_t *d_keys, const uint64_t *d_counts, uint64_t n) {
  if (c->poisoned) return fail(c, KMG_ERR_STATE, "context is inconsistent after a failed re-split: kmg_reset it");
  if (c->feed_kind == 2) return fail(c, KMG_ERR_STATE, "context holds blocks adopted from a sender (kmg_adopt_coarse_device): it cannot also take plain keys");
  c->feed_kind = 1;
  const uint32_t P1 = c->n_coarse;
  unsigned long long *d_cnt = c->d_part, *d_start = c->d_part + MAX_PARTS, *d_cur = c->d_part + 2 * MAX_PARTS;
  const uint64_t max_n = REFINE_MAX_ENTRIES;
  for (uint64_t i0 = 0; i0 < n; i0 += max_n) {
    const uint64_t m = std::min(max_n, n - i0);
    const size_t tmr = timer_begin(c, 0);
    CU(c, cudaMemsetAsync(c->d_part, 0, 3 * (size_t)MAX_PARTS * sizeof(unsigned long long), c->stream));
    CU(c, launch_keys_coarse(d_keys + i0, d_counts ? d_counts + i0 : nullptr, m, P1, false, d_cnt, d_start, d_cur, nullptr, nullptr, c->stream));
    std::vector<unsigned long long> counts(P1);
    CU(c, cudaMemcpyAsync(counts.data(), d_cnt, P1 * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    std::vector<uint64_t> off(P1 + 1, 0);
    for (uint32_t p = 0; p < P1; ++p) off[p + 1] = off[p] + counts[p];
    uint64_t *d_ckeys = nullptr, *d_ccounts = nullptr;
    kmg_status s = alloc_or_consolidate(c, reinterpret_cast<void **>(&d_ckeys), m * 8, "coarse keys");
    if (s == KMG_OK && d_counts) s = alloc_or_consolidate(c, reinterpret_cast<void **>(&d_ccounts), m * 8, "coarse counts");
    if (s != KMG_OK) { pool_free(c, d_ckeys); return s; }
    CU(c, cudaMemcpyAsync(d_start, off.data(), P1 * 8, cudaMemcpyHostToDevice, c->stream));
    CU(c, launch_keys_coarse(d_keys + i0, d_counts ? d_counts + i0 : nullptr, m, P1, true, d_cnt, d_start, d_cur, d_ckeys, d_ccounts, c->stream));
    s = refine_to_run(c, d_ckeys, d_ccounts, off);  // synchronises: the caller may reuse d_keys when we return
    timer_end(c, tmr);
    if (s != KMG_OK) return s;
  }
  return KMG_OK;
}

// The input outgrew the partition plan: split every fine partition of every run m ways (one streaming pass per run; the
// sub-bin function nests, so partition p becomes partitions p*m .. p*m + m-1).  Afterwards n_sub and n_parts are m times larger.
kmg_status resplit_runs(kmg_ctx *c, uint32_t m) {
  const uint32_t P_old = c->n_parts;
  std::vector<Run *> all;
  if (c->has_result && c->result.n) all.push_back(&c->result);
  for (auto &r : c->runs) all.push_back(&r);
  for (auto *r : all) if (r->n > REFINE_MAX_ENTRIES) return KMG_OK;  // refine launches index with 32 bits: leave it to the multi-pass kernel
  c->in_resplit = true;
  kmg_status st = KMG_OK;
  std::vector<uint64_t> off(P_old + 1), lens(P_old);
  for (auto *r : all) {
    cudaError_t e = cudaMemcpyAsync(off.data(), r->d_seg_start, (size_t)P_old * 8, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(lens.data(), r->d_seg_len, (size_t)P_old * 8, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) { st = cuda_fail(c, e, "re-split (segment table)"); break; }
    off[P_old] = P_old ? off[P_old - 1] + lens[P_old - 1] : 0;
    Run nr;
    SplitPlan sp{P_old, m, c->n_sub, &nr};
    st = refine_to_run(c, r->d_keys, r->d_counts, off, /*owns=*/false, /*sync=*/true, &lens, &sp);
    if (st != KMG_OK) break;
    nr.n_valid = r->n_valid;
    free_run(c, *r);
    *r = std::move(nr);
  }
  c->in_resplit = false;
  if (st != KMG_OK) {  // runs already re-split and runs not yet re-split coexist now: refuse everything but a reset
    c->poisoned = true;
    return fail(c, st, c->err + " (while re-splitting the runs: the context must be reset)");
  }
  c->n_sub *= m;
  c->n_parts = P_old * m;
  return KMG_OK;
}

// phase B: merge the consolidated result (if any) and all pending runs into a new consolidated run
// recompact: rewrite the consolidated result alone (its entries are mostly skipped fillers after a direct-emit launch on
// duplicate-rich input) with the compacting kernel
kmg_status consolidate(kmg_ctx *c, bool recompact) {
  if (c->runs.empty() && !(recompact && c->has_result && c->result.n)) return KMG_OK;
  {  // partitions several times larger than planned: refine the plan before counting
    uint64_t entries = c->has_result ? c->result.n_valid : 0;
    for (auto &r : c->runs) entries += r.n;
    const uint64_t avg = entries / std::max<uint32_t>(c->n_parts, 1);
    // (not while refine_to_run is building a run from the current plan -- its allocations may land here -- : the run would be
    // finished with the old partition count and sub-bin function; partitions are counted in passes instead)
    if (avg > 2 * TARGET_KEYS_PER_PART && c->n_sub * 2 <= 2048 && !c->cfg.parts_log2 && !c->building_run) {  // an explicit partition count is respected
      const uint32_t m = (uint32_t)std::min<uint64_t>((avg + TARGET_KEYS_PER_PART - 1) / TARGET_KEYS_PER_PART, 2048 / c->n_sub);
      // Re-splitting costs one tile (~3.5 us of one SM) per input partition or per 8192 entries of every run plus a streaming
      // pass; counting in m passes instead costs ~7 ps per entry and extra pass, again at every later consolidation.  Many small
      // runs over a slightly outgrown plan are cheaper in passes, one big run over a badly outgrown plan is cheaper re-split.
      double resplit_ns = (double)entries * 0.006, passes_ns = (double)entries * (m - 1) * 0.007 * 2.0;
      auto tiles_of = [&](const Run &r) { return (double)std::max<uint64_t>(c->n_parts, r.n / REFINE_TILE); };
      if (c->has_result && c->result.n) resplit_ns += tiles_of(c->result) * 3500.0 / num_sms();
      for (auto &r : c->runs) resplit_ns += tiles_of(r) * 3500.0 / num_sms();
      if (m >= 2 && resplit_ns < passes_ns) { kmg_status rs = resplit_runs(c, m); if (rs != KMG_OK) return rs; }
    }
  }
  std::vector<Run *> in;
  if (c->has_result && c->result.n) in.push_back(&c->result);
  for (auto &r : c->runs) in.push_back(&r);
  const uint32_t P = c->n_parts, R = (uint32_t)in.size();
  if (R > (uint32_t)CONS_MAX_RUNS) return fail(c, KMG_ERR_STATE, "too many pending runs");
  uint64_t total = 0;
  for (auto *r : in) total += r->n;

  CountParams prm{};
  prm.n_parts = P; prm.R = R; prm.preagg = !(c->cfg.flags & KMG_FLAG_NO_PREAGG);
  for (uint32_t r = 0; r < R; ++r) prm.runs[r] = ConsRun{in[r]->d_keys, in[r]->d_counts, in[r]->d_seg_start, in[r]->d_seg_len};

  // processing order: partitions with many entries first (a partition is counted by ONE CTA).  Only when some partition is
  // heavy (> 8x the average) is the per-partition table fetched and sorted; otherwise partitions are taken as they come.
  unsigned long long *d_totals = nullptr;
  uint32_t *d_order = nullptr;
  unsigned long long h_max = 0;
  cudaError_t e = pool_alloc(c, &d_totals, (size_t)P * 8);
  if (e == cudaSuccess) e = launch_sum_lens(prm, d_totals, c->d_stats + 6, c->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(&h_max, c->d_stats + 6, 8, cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  if (e != cudaSuccess) { pool_free(c, d_totals); return cuda_fail(c, e, "consolidate setup"); }
  const uint64_t max_total = h_max;
  const uint64_t heavy = 8 * std::max<uint64_t>(total / P, 1024);
  if (max_total > heavy) {
    std::vector<unsigned long long> totals(P);
    e = pool_alloc(c, &d_order, (size_t)P * 4);
    if (e == cudaSuccess) e = cudaMemcpyAsync(totals.data(), d_totals, (size_t)P * 8, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) { pool_free(c, d_totals); pool_free(c, d_order); return cuda_fail(c, e, "consolidate setup"); }
    std::vector<uint32_t> order, big;
    order.reserve(P);
    for (uint32_t p = 0; p < P; ++p) if (totals[p] > heavy) big.push_back(p);
    std::sort(big.begin(), big.end(), [&](uint32_t a, uint32_t b) { return totals[a] > totals[b]; });
    order = big;
    for (uint32_t p = 0; p < P; ++p) if (totals[p] <= heavy) order.push_back(p);
    e = cudaMemcpy(d_order, order.data(), (size_t)P * 4, cudaMemcpyHostToDevice);  // synchronous: `order` dies with this scope
  }
  pool_free(c, d_totals);
  prm.order = d_order;

  // The output run holds one entry per DISTINCT key.  `total` (one per input entry) is always enough, but read sets repeat every
  // k-mer many times (C5: 26 G windows, 2.4 G distinct) and a run sized for the input would not fit next to the inputs.  So the
  // run is sized from the dedup ratio the previous consolidation observed (1.0 at first), and a launch that runs out of space
  // (nospace flag, nothing written past the capacity) is repeated with whatever memory allows.
  Run out;
  uint64_t raw_entries = 0;
  for (auto *r : in) if (!r->d_counts) raw_entries += r->n;
  // Direct emit (count_partitions_smem_kernel<false, true>): only unweighted runs of keys that are mostly distinct (a genome, not a
  // deep read set), partitions within the plan.  Its output holds one entry per input entry.
  bool direct = !recompact && raw_entries == total && c->dedup_ratio >= 0.5 && max_total <= 0xffffu &&
                total / std::max<uint32_t>(P, 1) <= SMEM_TABLE_SLOTS / 2 && !(c->cfg.flags & KMG_FLAG_NO_PREAGG);
  // Sieve variant (count_partitions_sieve_tma_kernel): same precondition; it leaves the partitions it cannot take (too many repeated keys,
  // more than one batch of entries) to the compacting variant, so no bound on the largest partition is needed.
  bool sieve = !recompact && raw_entries == total && c->dedup_ratio >= 0.5 &&
               total / std::max<uint32_t>(P, 1) <= SIEVE_MAX_ENTRIES * 15 / 16 && !(c->cfg.flags & KMG_FLAG_NO_PREAGG);
  uint32_t *d_redo = nullptr;
  unsigned long long *d_redo_base = nullptr;
  if (sieve && (pool_alloc(c, &d_redo, (size_t)P * 8) != cudaSuccess || pool_alloc(c, &d_redo_base, (size_t)P * 8) != cudaSuccess)) {  // d_redo: partition numbers, then range lengths
    cudaGetLastError(); pool_free(c, d_redo); pool_free(c, d_redo_base); d_redo = nullptr; d_redo_base = nullptr; sieve = false;
  }
  // In place (count_partitions_sieve_in_place_kernel): one raw run in the speculative layout is counted where it lies.  The
  // result takes over its keys and segment starts and gets a count for every slot of the layout (0: repeat, pad entry or slack), so
  // phase B writes 8 bytes per slot instead of 16 per entry and no second key array is held.  Each fallback below leaves the route
  // for the copying one: the kernel never writes the keys, so the input is intact until the compacting variant has run.  The
  // partitions it hands over are compacted into their own capacity, which is only safe while that variant cannot overflow: a
  // capacity of at most two batches (2 x 4096 entries) fits its 8192-slot table and, at 256 claims per warp and batch, its warp lists.
  bool in_place = sieve && R == 1 && in[0]->part_cap != 0 && in[0]->part_cap <= 2ull * SMEM_COUNT_THREADS * 8;
  const uint64_t in_place_n = in_place ? (uint64_t)P * in[0]->part_cap : 0;
  uint64_t out_cap = std::max<uint64_t>(total, 1) + (sieve ? (uint64_t)P * R : 0);  // padded segments: up to one filler entry per partition and run
  if (recompact) out_cap = std::min<uint64_t>(out_cap, c->result.n_valid + (1ull << 20));
  else if (total > (1ull << 28) && !direct && !sieve) {
    const uint64_t est = (total - raw_entries) + (uint64_t)((double)raw_entries * std::min(1.0, c->dedup_ratio * 1.25 + 0.02)) + (1ull << 24);
    out_cap = std::min(out_cap, est);
  }
  auto alloc_out = [&](uint64_t cap) -> cudaError_t {
    cudaError_t ae = pool_alloc(c, &out.d_keys, cap * 8);
    if (ae == cudaSuccess) ae = pool_alloc(c, &out.d_counts, cap * 8);
    if (ae != cudaSuccess) { pool_free(c, out.d_keys); pool_free(c, out.d_counts); out.d_keys = out.d_counts = nullptr; cudaGetLastError(); }
    return ae;
  };
  auto alloc_copy_out = [&]() -> cudaError_t {
    cudaError_t ae = alloc_out(out_cap);
    if (ae != cudaSuccess && out_cap > (1ull << 26)) {  // not even the estimate fits: take what is there
      size_t free_b = 0, total_b = 0;
      pool_release_idle(c);
      cudaMemGetInfo(&free_b, &total_b);
      const uint64_t room = free_b > (3ull << 30) ? (free_b - (2ull << 30)) / 16 : 0;
      if (room >= (1ull << 26)) { out_cap = std::min(out_cap, room); ae = alloc_out(out_cap); }
    }
    prm.out_keys = out.d_keys; prm.out_counts = out.d_counts; prm.out_cap = out_cap; prm.part_cap = 0;
    return ae;
  };
  if (e == cudaSuccess && in_place) {
    if (pool_alloc(c, &out.d_counts, in_place_n * 8) == cudaSuccess) {
      prm.out_keys = in[0]->d_keys; prm.out_counts = out.d_counts; prm.out_cap = in_place_n; prm.part_cap = (uint32_t)in[0]->part_cap;
    } else { cudaGetLastError(); in_place = false; }
  }
  if (e == cudaSuccess && !in_place) e = alloc_copy_out();
  if (e == cudaSuccess) e = pool_alloc(c, &out.d_seg_start, (size_t)P * 8);
  if (e == cudaSuccess) e = pool_alloc(c, &out.d_seg_len, (size_t)P * 8);
  if (e != cudaSuccess) { pool_free(c, d_order); pool_free(c, d_redo); pool_free(c, d_redo_base); free_run(c, out); return cuda_fail(c, e, "cudaMalloc(consolidated run)"); }
  prm.out_seg_start = out.d_seg_start; prm.out_seg_len = out.d_seg_len;

  if (!c->d_hist) {
    e = cudaMalloc(&c->d_hist, (HIST_DENSE_BINS + 1) * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMalloc(&c->d_hist_ov, HIST_OVERFLOW_CAP * 8);
    if (e != cudaSuccess) { pool_free(c, d_order); pool_free(c, d_redo); pool_free(c, d_redo_base); free_run(c, out); return cuda_fail(c, e, "cudaMalloc(histogram)"); }
  }
  prm.hist = c->d_hist; prm.hist_overflow = c->d_hist_ov; prm.hist_overflow_cap = HIST_OVERFLOW_CAP;
  c->fused_valid = c->fused_cached = false;

  const unsigned grid = (unsigned)std::min<uint64_t>(P, (uint64_t)num_sms() * COUNT_CTAS_PER_SM);
  kmg_status st = KMG_OK;
  unsigned long long n_out = 0;
  // attempt 0: shared-memory tables (primary).  If a partition holds more distinct keys than such a table
  // (inputs much larger than the partition plan), fall back to L2-resident scratch tables of growing size.
  // The shared-memory kernel counts partitions that outgrew the plan in several passes (split_log2, from the average
  // partition size); if a partition still overflows its table the split is refined twice before the L2-scratch variant
  // takes over.
  uint32_t split_log2 = 0;
  while (split_log2 < 8 && (3600ull << split_log2) * 5 / 4 < total / std::max<uint32_t>(P, 1)) ++split_log2;
  unsigned long long n_valid = 0;
  int smem_attempts = 0;
  for (int attempt = 0;; ++attempt) {
    const bool use_smem = smem_attempts < 3 && split_log2 <= 8;
    uint64_t *d_scratch = nullptr;
    unsigned long long *d_sync = nullptr;  // [0] out_cursor, [1] next (u32) | error (u32), [2] distinct keys, [3] no-space flag (u32)
    const uint64_t slots = use_smem ? 0 : (uint64_t)grid << c->scratch_log2;
    prm.split_log2 = split_log2;
    e = pool_alloc(c, &d_sync, 32);
    if (e == cudaSuccess && slots) e = pool_alloc(c, &d_scratch, slots * 16);
    if (e != cudaSuccess) { pool_free(c, d_scratch); pool_free(c, d_sync); st = cuda_fail(c, e, "cudaMalloc(count scratch)"); break; }
    prm.scratch = d_scratch; prm.scratch_log2 = c->scratch_log2;
    prm.out_cursor = d_sync;
    prm.out_distinct = d_sync + 2;
    prm.next = reinterpret_cast<uint32_t *>(d_sync + 1);
    prm.error_flag = reinterpret_cast<uint32_t *>(d_sync + 1) + 1;
    prm.nospace_flag = reinterpret_cast<uint32_t *>(d_sync + 3);
    e = cudaMemsetAsync(d_sync, 0, 32, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->d_hist, 0, (HIST_DENSE_BINS + 1) * sizeof(unsigned long long), c->stream);
    if (e == cudaSuccess && slots) e = launch_table_init(HashTable{d_scratch, slots}, c->stream, EMPTY_MIX);
    const size_t tmr = timer_begin(c, 1);
    bool weighted = max_total > ((2ull * SMEM_COUNT_THREADS * 8) << split_log2);  // partitions oversized beyond the split want the pre-aggregating variant
    for (uint32_t r = 0; r < R; ++r) weighted |= in[r]->d_counts != nullptr;
    if (weighted || split_log2 || !use_smem) direct = sieve = false;
    if (in_place && !sieve) {  // the copying route takes over
      pool_free(c, out.d_counts); out.d_counts = nullptr;
      in_place = false;
      if (e == cudaSuccess) e = alloc_copy_out();
    }
    static const bool dbg_sieve = getenv("KMG_DEBUG_SIEVE") != nullptr;
    unsigned long long h_sync[4] = {0, 0, 0, 0};
    if (sieve) {
      prm.redo_list = d_redo; prm.redo_count = reinterpret_cast<uint32_t *>(d_sync + 3) + 1;
      prm.redo_len = d_redo + P; prm.redo_base = d_redo_base;
      if (e == cudaSuccess) e = launch_count_partitions_sieve(prm, c->stream);
      timer_end(c, tmr);
      if (e == cudaSuccess) e = cudaMemcpyAsync(h_sync, d_sync, 32, cudaMemcpyDeviceToHost, c->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
      const uint32_t n_redo = (uint32_t)(h_sync[3] >> 32);
      if (e == cudaSuccess && (n_redo > sieve_redo_limit_host(P) || (uint32_t)h_sync[3])) {
        // duplicate-rich input (the reserved ranges of the partitions handed back are lost as fillers, the sieve stops early):
        // the launch is repeated without the sieve
        if (dbg_sieve) fprintf(stderr, "[kmg] sieve: %u partitions, %u handed back, repeated without the sieve, %s\n", P, n_redo, in_place ? "leaves the in-place route" : "copied");
        pool_free(c, d_scratch); pool_free(c, d_sync);
        sieve = direct = false;
        c->dedup_ratio = std::min(c->dedup_ratio, 0.49);
        continue;
      }
      if (e == cudaSuccess && n_redo) {
        // the partitions the sieve left alone: compacting variant, continuing the same output cursor, distinct count and histogram
        CountParams redo = prm;
        redo.order = d_redo; redo.n_parts = n_redo; redo.redo_list = nullptr; redo.redo_count = nullptr;
        redo.pre_base = d_redo_base; redo.pre_len = d_redo + P; redo.redo_base = nullptr; redo.redo_len = nullptr;
        e = cudaMemsetAsync(prm.next, 0, 4, c->stream);
        const size_t tmr2 = timer_begin(c, 1);
        if (e == cudaSuccess) e = launch_count_partitions_smem(redo, false, false, c->stream);
        timer_end(c, tmr2);
        if (e == cudaSuccess) e = cudaMemcpyAsync(h_sync, d_sync, 32, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        c->sieve_redo += n_redo;
      }
      if (dbg_sieve)
        fprintf(stderr, "[kmg] sieve: %u partitions, %u left to the compacting variant, %llu entries, %llu distinct, %s\n", P, n_redo,
                in_place ? (unsigned long long)in_place_n : (unsigned long long)h_sync[0], (unsigned long long)h_sync[2], in_place ? "in place" : "copied");
    } else {
      if (e == cudaSuccess) e = use_smem ? launch_count_partitions_smem(prm, weighted, direct, c->stream) : launch_count_partitions(prm, grid, c->stream);
      timer_end(c, tmr);
      if (e == cudaSuccess) e = cudaMemcpyAsync(h_sync, d_sync, 32, cudaMemcpyDeviceToHost, c->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    }
    pool_free(c, d_scratch); pool_free(c, d_sync);
    if (e != cudaSuccess) { st = cuda_fail(c, e, "count_partitions"); break; }
    if ((uint32_t)h_sync[3] && !(h_sync[1] >> 32)) {  // the run was too small for the distinct keys: enlarge it and repeat
      const uint64_t need = std::min<uint64_t>(total, h_sync[0] + (1ull << 20));  // out_cursor kept counting: the exact demand (plus filler entries)
      if (out_cap >= total || attempt >= 16) { st = fail(c, KMG_ERR_OOM, "the consolidated run does not fit in device memory"); break; }
      pool_free(c, out.d_keys); pool_free(c, out.d_counts); out.d_keys = out.d_counts = nullptr;
      out_cap = need;
      if (alloc_out(out_cap) != cudaSuccess) {
        pool_release_idle(c);
        if (alloc_out(out_cap) != cudaSuccess) { st = fail(c, KMG_ERR_OOM, "the consolidated run (" + std::to_string(need) + " entries) does not fit in device memory"); break; }
      }
      prm.out_keys = out.d_keys; prm.out_counts = out.d_counts; prm.out_cap = out_cap;
      c->dedup_ratio = 1.0;
      continue;
    }
    n_out = h_sync[0]; n_valid = h_sync[2];
    if (!(h_sync[1] >> 32)) break;  // no overflow
    if (sieve && in_place) {
      // Not reached: the route is only taken for capacities the compacting variant always holds (see above).  Its other
      // partitions were compacted into the input, so the launch cannot be repeated from it.
      c->poisoned = true;
      st = fail(c, KMG_ERR_STATE, "phase B in place: the compacting variant overflowed on a partition of the speculative layout (the context must be reset)");
      break;
    }
    if (sieve) { sieve = false; continue; }    // a left-over partition was beyond the compacting variant too: the whole launch is repeated without the sieve
    if (direct) { direct = false; continue; }  // a partition beyond the direct variant's limits: the compacting variant takes the launch
    if (attempt >= 16 || c->scratch_log2 >= 30) { st = fail(c, KMG_ERR_TABLE_FULL, "partition table overflow could not be resolved"); break; }
    if (use_smem) {  // finer split first (weights beyond 32 bits are not cured by it: the L2 variant follows after three tries)
      ++smem_attempts;
      split_log2 += 2;
      c->scratch_log2 = std::max<uint32_t>(c->scratch_log2, 14);
    } else ++c->scratch_log2;  // retry with larger tables
  }
  pool_free(c, d_order); pool_free(c, d_redo); pool_free(c, d_redo_base);
  if (st != KMG_OK) { free_run(c, out); return st; }
  out.n = n_out; out.n_valid = n_valid;
  if (in_place) {  // the result takes over the input run's keys and layout (free_run below leaves them alone)
    out.n = in_place_n;
    out.d_keys = in[0]->d_keys; in[0]->d_keys = nullptr;
    pool_free(c, out.d_seg_start); out.d_seg_start = in[0]->d_seg_start; in[0]->d_seg_start = nullptr;
  }
  if (raw_entries > (1ull << 24)) {  // distinct keys the raw runs added per raw entry (an upper estimate: keys already in the result count as new)
    const uint64_t before = total - raw_entries;
    c->dedup_ratio = std::min(1.0, (double)(n_valid > before / 2 ? n_valid - before / 2 : 0) / (double)raw_entries);
  }
  if (c->has_result) free_run(c, c->result);
  for (auto &r : c->runs) free_run(c, r);
  c->runs.clear();
  c->pending_bytes = 0;
  // give back the slack (upper bound was one slot per input entry) when it is worth a copy (an in-place result has no spare
  // allocation: its slack is the layout's)
  if (!in_place && out.n && out.n < total / 2) {
    uint64_t *k2 = nullptr, *c2 = nullptr;
    if (pool_alloc(c, &k2, out.n * 8) == cudaSuccess && pool_alloc(c, &c2, out.n * 8) == cudaSuccess) {
      cudaMemcpyAsync(k2, out.d_keys, out.n * 8, cudaMemcpyDeviceToDevice, c->stream);
      cudaMemcpyAsync(c2, out.d_counts, out.n * 8, cudaMemcpyDeviceToDevice, c->stream);
      cudaStreamSynchronize(c->stream);
      pool_free(c, out.d_keys); pool_free(c, out.d_counts);
      out.d_keys = k2; out.d_counts = c2;
    } else { cudaGetLastError(); pool_free(c, k2); pool_free(c, c2); }
  }
  c->result = std::move(out);
  c->has_result = true;
  c->fused_valid = true;
  c->n_consolidations++;
  if ((direct || sieve) && c->result.n > (1ull << 20) && c->result.n_valid < c->result.n / 2) {
    // duplicate-rich input went through the direct variant (nothing was known about it yet): most entries are fillers.
    // Rewrite the run compactly once; dedup_ratio now steers later consolidations to the compacting variant.
    kmg_status rs = consolidate(c, /*recompact=*/true);
    if (rs != KMG_OK) return rs;
    c->n_consolidations--;
  }
  return KMG_OK;
}

// Host copy of the count-of-counts phase B left behind for `result`.  false: not available (no consolidated
// result, or more than HIST_OVERFLOW_CAP counts >= HIST_DENSE_BINS) -- the caller then runs the table kernels.
bool fetch_fused_hist(kmg_ctx *c) {
  if (c->mode != kmg_ctx::MODE_PARTITIONED || !c->has_result || !c->runs.empty() || !c->fused_valid) return false;
  if (c->fused_cached) return true;
  c->h_bins.assign(HIST_DENSE_BINS + 1, 0);
  if (cudaMemcpyAsync(c->h_bins.data(), c->d_hist, (HIST_DENSE_BINS + 1) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
      cudaStreamSynchronize(c->stream) != cudaSuccess) { cudaGetLastError(); c->fused_valid = false; return false; }
  const uint64_t ov_n = c->h_bins[HIST_DENSE_BINS];
  if (ov_n > HIST_OVERFLOW_CAP) { c->fused_valid = false; return false; }
  c->h_ov.resize(ov_n);
  if (ov_n && cudaMemcpy(c->h_ov.data(), c->d_hist_ov, ov_n * 8, cudaMemcpyDeviceToHost) != cudaSuccess) { cudaGetLastError(); c->fused_valid = false; return false; }
  std::sort(c->h_ov.begin(), c->h_ov.end());
  c->h_bins.resize(HIST_DENSE_BINS);
  uint64_t others = ov_n, sum = 0, mx = 0;
  for (uint64_t b = 2; b < (uint64_t)HIST_DENSE_BINS; ++b) if (c->h_bins[b]) { others += c->h_bins[b]; sum += b * c->h_bins[b]; mx = b; }
  c->h_bins[0] = 0;
  c->h_bins[1] = c->result.n_valid - others;  // counts of 1 are not recorded by the kernel
  sum += c->h_bins[1];
  if (c->h_bins[1] && mx < 1) mx = 1;
  for (uint64_t v : c->h_ov) sum += v;
  if (ov_n) mx = c->h_ov.back();
  c->fused_sum = sum; c->fused_max = mx;
  c->fused_cached = true;
  return true;
}

// Run the counting scan over a packed stream of n_words_total words (already in d_bases/d_valid/d_start).
// A context that started small sits on the single HBM table (random atomics: fine while it fits L2, ~6x slower than the
// partitioned pipeline beyond).  Once the table plus the incoming batch pass MIGRATE_KEYS it is emptied into a weighted run
// and the context continues on the partitioned path, planned for 16x what it has seen (over-partitioning is cheap at this size;
// re-splitting / multi-pass counting covers streams that grow further).
constexpr uint64_t MIGRATE_KEYS = 1ull << 26;
kmg_status migrate_to_partitioned(kmg_ctx *c, uint64_t incoming) {
  kmg_status s = read_counters(c);
  if (s != KMG_OK) return s;
  const uint64_t n = c->h_counters[CTR_DISTINCT];
  uint64_t *dk = nullptr, *dc = nullptr;
  if (n) {
    cudaError_t e = pool_alloc(c, &dk, n * 8);
    if (e == cudaSuccess) e = pool_alloc(c, &dc, n * 8);
    if (e == cudaSuccess) e = launch_compact(view_of(c), 1, dk, dc, n, c->d_stats + 3, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) { pool_free(c, dk); pool_free(c, dc); return cuda_fail(c, e, "migrate to the partitioned path"); }
  }
  cudaFree(c->table.slots);
  c->table = HashTable{nullptr, 0};
  c->mode = kmg_ctx::MODE_UNDECIDED;
  c->cfg.flags |= KMG_FLAG_FORCE_PARTITIONED;
  c->cfg.expected_distinct = std::max<uint64_t>(c->cfg.expected_distinct, 16 * (n + incoming));  // the hint was too small (or absent)
  s = decide_mode(c, c->cfg.expected_distinct);
  if (s == KMG_OK && n) s = keys_to_run(c, dk, dc, n);
  pool_free(c, dk); pool_free(c, dc);
  c->n_grows++;
  return s;
}

kmg_status scan_packed(kmg_ctx *c, uint64_t n_words_total, bool has_start) {
  const uint64_t n_tiles = n_words_total / TILE_WORDS;
  uint64_t incoming = n_words_total * 32;  // upper bound of the keys this stream adds
  bool incoming_exact = false;
  if (!c->use_dense && c->cfg.has_min_quality) {
    // a quality filter can remove almost every window (config C3 keeps ~3 %): plan the table / the partitions from the
    // countable windows (masks only, 0.25 B/base), not from the bases
    unsigned long long h_ok = 0;
    CU(c, launch_count_windows(c->d_valid, has_start ? c->d_start : nullptr, n_words_total, c->k, c->d_stats + 7, c->stream));
    CU(c, cudaMemcpyAsync(&h_ok, c->d_stats + 7, 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    incoming = h_ok; incoming_exact = true;
  }
  uint64_t plan_windows = incoming;
  if (incoming_exact && c->plan_scale > 1.0) plan_windows = (uint64_t)((double)incoming * c->plan_scale * 1.25) + 1024;  // first chunk of a longer call
  c->plan_scale = 1.0;
  kmg_status ms = decide_mode(c, plan_windows);
  if (ms != KMG_OK) return ms;
  if (c->mode == kmg_ctx::MODE_TABLE && !(c->cfg.flags & KMG_FLAG_FORCE_HASH) && c->distinct_ub + incoming > MIGRATE_KEYS) {
    ms = migrate_to_partitioned(c, incoming);
    if (ms != KMG_OK) return ms;
  }
  if (c->mode == kmg_ctx::MODE_PARTITIONED) {
    if (incoming_exact && !c->shm && incoming * 8 < n_words_total * 32 && incoming < (1ull << 32) - 1) {
      // sparse route: fewer than one window in eight survives the quality filter -- scan + compact the surviving keys, then partition
      // those (the scatter kernels would pay their per-sub-tile work for every tile of the input)
      if (incoming == 0) return KMG_OK;
      uint64_t *d_keys = nullptr;
      kmg_status st = alloc_or_consolidate(c, reinterpret_cast<void **>(&d_keys), incoming * 8, "sparse keys");
      if (st != KMG_OK) return st;
      const size_t tmr = timer_begin(c, 0);
      unsigned long long h_n = 0;
      cudaError_t e = cudaMemsetAsync(c->d_stats + 7, 0, 8, c->stream);
      for (uint64_t tile0 = 0; e == cudaSuccess && tile0 < n_tiles;) {
        const uint64_t tiles = std::min<uint64_t>(n_tiles - tile0, ((1ull << 32) - 1) / ((uint64_t)TILE_WORDS * 32));
        ScanInput in;
        in.bases = c->d_bases + tile0 * TILE_WORDS; in.valid = c->d_valid + tile0 * TILE_WORDS;
        in.start = has_start ? c->d_start + tile0 * TILE_WORDS : nullptr;
        in.n_tiles = tiles; in.k = c->k;
        e = launch_scan_emit_keys(in, d_keys, c->d_stats + 7, c->stream);
        tile0 += tiles;
      }
      if (e == cudaSuccess) e = cudaMemcpyAsync(&h_n, c->d_stats + 7, 8, cudaMemcpyDeviceToHost, c->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
      timer_end(c, tmr);
      if (e != cudaSuccess) { pool_free(c, d_keys); return cuda_fail(c, e, "sparse scan"); }
      if (h_n != incoming) { pool_free(c, d_keys); return fail(c, KMG_ERR_STATE, "sparse scan: emitted keys differ from the counted windows"); }
      st = keys_to_run(c, d_keys, nullptr, incoming);
      pool_free(c, d_keys);
      return st;
    }
    return scan_to_run(c, n_words_total, has_start);
  }
  uint64_t tile0 = 0;
  const size_t tmr = timer_begin(c);
  while (tile0 < n_tiles) {
    uint64_t want = (n_tiles - tile0) * TILE_WORDS * 32, granted = 0;
    if (incoming_exact && tile0 == 0) want = std::max<uint64_t>(incoming, 1);  // the whole stream adds exactly this many keys
    kmg_status s = reserve_capacity(c, want, &granted);
    if (s != KMG_OK) return s;
    uint64_t tiles = granted >= want ? n_tiles - tile0 : granted / ((uint64_t)TILE_WORDS * 32);
    if (tiles == 0) return fail(c, KMG_ERR_TABLE_FULL, "no table capacity left for even one tile");
    ScanInput in;
    in.bases = c->d_bases + tile0 * TILE_WORDS;
    in.valid = c->d_valid + tile0 * TILE_WORDS;
    in.start = has_start ? c->d_start + tile0 * TILE_WORDS : nullptr;
    in.n_tiles = tiles;
    in.k = c->k;
    if (c->use_dense) CU(c, launch_scan_dense(in, c->dense, c->d_counters, c->cfg.flags, c->stream));
    else CU(c, launch_scan_hash(in, c->table, c->d_counters, c->cfg.flags, c->stream));
    tile0 += tiles;
  }
  timer_end(c, tmr);
  return KMG_OK;
}

// The lowest quality byte a base needs to count under the context's filter: min_quality + 33, saturating (src/run.rs:538).
uint32_t quality_threshold(const kmg_ctx *c) { return std::min<uint32_t>(255u, (uint32_t)c->cfg.min_quality + 33u); }

// Ingest n_bytes > 0 of raw ASCII already on the device into the context's packed buffers, with the start bits of d_starts[n_starts]
// (byte offsets, minus base_offset, of record starts inside these bytes).  The scan over them is the caller's.
kmg_status pack_device_ascii(kmg_ctx *c, const uint8_t *d_seq, const uint8_t *d_qual, const uint64_t *d_starts, uint64_t n_starts,
                             uint64_t base_offset, uint64_t n_bytes, uint64_t *n_words_total, bool *has_start) {
  const uint64_t words = round_up((n_bytes + 31) / 32, TILE_WORDS);
  kmg_status s = ensure_packed(c, words);
  if (s != KMG_OK) return s;
  const bool use_q = c->cfg.has_min_quality && d_qual != nullptr;
  CU(c, launch_ingest(d_seq, use_q ? d_qual : nullptr, n_bytes, quality_threshold(c), words, c->d_bases, c->d_valid, c->stream));
  *has_start = d_starts != nullptr && n_starts > 0;
  if (*has_start) CU(c, launch_start_bits(d_starts, n_starts, base_offset, n_bytes, words, c->d_start, c->stream));
  *n_words_total = words;
  return KMG_OK;
}

kmg_status ensure_staging(kmg_ctx *c, bool need_pinned, bool need_qual, uint64_t need_bytes) {
  // staging slots are sized for the largest chunk seen so far (at most batch_bases), not for batch_bases up front
  const uint64_t want = std::min<uint64_t>(c->batch_bases, std::max<uint64_t>(need_bytes, 1u << 20)) + 64;
  if (want > c->staging_cap) {
    CU(c, cudaStreamSynchronize(c->stream));
    CU(c, cudaStreamSynchronize(c->copy_stream));
    for (auto &s : c->st) {
      cudaFree(s.d_seq); cudaFree(s.d_qual); s.d_seq = s.d_qual = nullptr;
      if (s.h_seq) cudaFreeHost(s.h_seq);
      if (s.h_qual) cudaFreeHost(s.h_qual);
      s.h_seq = s.h_qual = nullptr;
      s.h2d_pending = s.compute_pending = false;
    }
    c->staging_cap = want;
  }
  for (auto &s : c->st) {
    if (!s.d_seq) CU(c, cudaMalloc(&s.d_seq, c->staging_cap));
    if (need_qual && !s.d_qual) CU(c, cudaMalloc(&s.d_qual, c->staging_cap));
    if (!s.h2d_done) {
      CU(c, cudaEventCreateWithFlags(&s.h2d_done, cudaEventDisableTiming));
      CU(c, cudaEventCreateWithFlags(&s.compute_done, cudaEventDisableTiming));
    }
    if (need_pinned && !s.h_seq) CU(c, cudaHostAlloc(&s.h_seq, c->staging_cap, cudaHostAllocDefault));
    if (need_pinned && need_qual && !s.h_qual) CU(c, cudaHostAlloc(&s.h_qual, c->staging_cap, cudaHostAllocDefault));
  }
  c->staging_ready = true;
  return KMG_OK;
}

kmg_status ensure_offsets(kmg_ctx *c, Staging &s, uint64_t n) {
  if (n <= s.off_cap) return KMG_OK;
  CU(c, cudaStreamSynchronize(c->stream));
  CU(c, cudaStreamSynchronize(c->copy_stream));
  if (s.h_off) cudaFreeHost(s.h_off);
  if (s.d_off) cudaFree(s.d_off);
  s.h_off = nullptr; s.d_off = nullptr; s.off_cap = 0;
  uint64_t cap = std::max<uint64_t>(n, 1024) * 2;
  CU(c, cudaHostAlloc(&s.h_off, cap * 8, cudaHostAllocDefault));
  CU(c, cudaMalloc(&s.d_off, cap * 8));
  s.off_cap = cap;
  return KMG_OK;
}

bool is_pinned_host(const void *p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

// ---- CRC32 (IEEE, reflected 0xEDB88320; src/index.rs:404-431), slicing-by-8 ----------------------------
struct Crc32 {
  uint32_t t[8][256];
  Crc32() {
    for (uint32_t i = 0; i < 256; i++) {
      uint32_t c = i;
      for (int j = 0; j < 8; j++) c = (c & 1) ? (c >> 1) ^ 0xEDB88320u : c >> 1;
      t[0][i] = c;
    }
    for (uint32_t i = 0; i < 256; i++)
      for (int s = 1; s < 8; s++) t[s][i] = (t[s - 1][i] >> 8) ^ t[0][t[s - 1][i] & 0xFF];
  }
  uint32_t update(uint32_t crc, const uint8_t *p, size_t n) const {
    while (n >= 8) {
      uint32_t a, b;
      memcpy(&a, p, 4); memcpy(&b, p + 4, 4);
      a ^= crc;
      crc = t[7][a & 0xFF] ^ t[6][(a >> 8) & 0xFF] ^ t[5][(a >> 16) & 0xFF] ^ t[4][a >> 24] ^
            t[3][b & 0xFF] ^ t[2][(b >> 8) & 0xFF] ^ t[1][(b >> 16) & 0xFF] ^ t[0][b >> 24];
      p += 8; n -= 8;
    }
    while (n--) crc = t[0][(crc ^ *p++) & 0xFF] ^ (crc >> 8);
    return crc;
  }
};
const Crc32 &crc_tables() { static Crc32 c; return c; }

}  // namespace

// =================================================================================================
KMG_EXPORT uint32_t kmg_abi_version(void) { return KMG_ABI_VERSION; }
KMG_EXPORT uint32_t kmg_ctx_k(const kmg_ctx *c) { return c ? (uint32_t)c->k : 0u; }

KMG_EXPORT const char *kmg_status_string(kmg_status s) {
  switch (s) {
    case KMG_OK: return "ok";
    case KMG_ERR_INVALID_K: return "invalid k-mer length (must be 1..=32)";
    case KMG_ERR_INVALID_ARG: return "invalid argument";
    case KMG_ERR_CUDA: return "CUDA error";
    case KMG_ERR_OOM: return "out of memory";
    case KMG_ERR_TABLE_FULL: return "k-mer table full";
    case KMG_ERR_STATE: return "invalid state";
    case KMG_ERR_IO: return "I/O error";
    case KMG_ERR_ABI: return "ABI version mismatch";
    case KMG_ERR_CAPACITY: return "output capacity too small";
    case KMG_ERR_PARSE: return "sequence parse error";
  }
  return "unknown";
}

KMG_EXPORT const char *kmg_last_error(const kmg_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

KMG_EXPORT uint32_t kmg_owner_of(uint64_t canonical_key, uint32_t n_shards) { return n_shards <= 1 ? 0 : part_of(canonical_key, n_shards); }

KMG_EXPORT void kmg_destroy(kmg_ctx *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
  timers_collect(c);
  if (c->fxs) fx_stream_close(c, true);
  if (c->shm || c->sh_recv) shard_release(c);
  for (auto &r : c->runs) free_run(c, r);
  if (c->has_result) free_run(c, c->result);
  pool_release_idle(c);
  for (auto &kv : c->pool_live) cudaFree(kv.first);
  cudaFree(c->d_part); cudaFree(c->d_fine_cursor);
  cudaFree(c->table.slots); cudaFree(c->dense); cudaFree(c->d_counters); cudaFree(c->d_stats); cudaFree(c->d_hist); cudaFree(c->d_hist_ov); cudaFree(c->d_scan_tmp);
  cudaFree(c->d_bases); cudaFree(c->d_valid); cudaFree(c->d_start);
  if (c->h_counters) cudaFreeHost(c->h_counters);
  for (auto &s : c->st) {
    if (s.h_seq) cudaFreeHost(s.h_seq);
    if (s.h_qual) cudaFreeHost(s.h_qual);
    if (s.h_off) cudaFreeHost(s.h_off);
    if (s.hp_bases) cudaFreeHost(s.hp_bases);
    if (s.hp_valid) cudaFreeHost(s.hp_valid);
    if (s.hp_start) cudaFreeHost(s.hp_start);
    cudaFree(s.d_seq); cudaFree(s.d_qual); cudaFree(s.d_off);
    cudaFree(s.dp_bases); cudaFree(s.dp_valid); cudaFree(s.dp_start);
    if (s.h2d_done) cudaEventDestroy(s.h2d_done);
    if (s.compute_done) cudaEventDestroy(s.compute_done);
  }
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

KMG_EXPORT kmg_status kmg_create(const kmg_config *cfg, kmg_ctx **out) {
  if (!cfg || !out) return fail(nullptr, KMG_ERR_INVALID_ARG, "cfg and out must not be NULL");
  *out = nullptr;
  if (cfg->abi_version != KMG_ABI_VERSION)
    return fail(nullptr, KMG_ERR_ABI, "abi_version " + std::to_string(cfg->abi_version) + " != " + std::to_string(KMG_ABI_VERSION));
  if (cfg->k < 1 || cfg->k > 32)  // KmerLengthError (src/kmer.rs:100-111)
    return fail(nullptr, KMG_ERR_INVALID_K, "k-mer length " + std::to_string(cfg->k) + " is out of range (must be 1-32)");
  if ((cfg->flags & KMG_FLAG_FORCE_DIRECT) && (cfg->flags & KMG_FLAG_FORCE_HASH))
    return fail(nullptr, KMG_ERR_INVALID_ARG, "FORCE_DIRECT and FORCE_HASH are mutually exclusive");
  if ((cfg->flags & KMG_FLAG_FORCE_DIRECT) && cfg->k > (uint32_t)DENSE_MAX_K)
    return fail(nullptr, KMG_ERR_INVALID_ARG, "direct-indexed path supports k <= 14");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(nullptr, KMG_ERR_CUDA, std::string("no CUDA device available (this library has no CPU fallback): ") +
                                           (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
  }
  kmg_ctx *c = new kmg_ctx();
  c->cfg = *cfg;
  c->k = (int)cfg->k;
  if (cfg->device >= 0) c->device = cfg->device; else cudaGetDevice(&c->device);
  auto bail = [&](kmg_status s) { g_create_error = c->err; kmg_destroy(c); return s; };
#define CUC(call)                                                                  \
  do {                                                                             \
    cudaError_t _e = (call);                                                       \
    if (_e != cudaSuccess) { cuda_fail(c, _e, #call); return bail(_e == cudaErrorMemoryAllocation ? KMG_ERR_OOM : KMG_ERR_CUDA); } \
  } while (0)
  CUC(cudaSetDevice(c->device));
  if (cfg->stream) c->stream = (cudaStream_t)cfg->stream;
  else { CUC(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)); c->own_stream = true; }
  CUC(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  CUC(cudaMalloc(&c->d_counters, CTR_N * sizeof(unsigned long long)));
  CUC(cudaMemsetAsync(c->d_counters, 0, CTR_N * sizeof(unsigned long long), c->stream));
  CUC(cudaMalloc(&c->d_stats, 8 * sizeof(unsigned long long)));
  CUC(cudaHostAlloc(&c->h_counters, 16 * sizeof(unsigned long long), cudaHostAllocDefault));
  if (cfg->batch_bases) c->batch_bases = std::max<uint64_t>(round_up(cfg->batch_bases, 32), 4096);
  c->use_dense = (cfg->flags & KMG_FLAG_FORCE_DIRECT) ||
                 (!(cfg->flags & (KMG_FLAG_FORCE_HASH | KMG_FLAG_FORCE_PARTITIONED)) && cfg->k <= (uint32_t)DENSE_DEFAULT_MAX_K);
  if (c->use_dense) {
    c->dense_n = 1ull << (2 * c->k);
    CUC(cudaMalloc(&c->dense, c->dense_n * 8));
    CUC(cudaMemsetAsync(c->dense, 0, c->dense_n * 8, c->stream));
  }
  // hash table / partition buffers are allocated by decide_mode() at the first feeding call, when the
  // input size is known (small inputs: one HBM table; large inputs: the partitioned pipeline)
  if ((cfg->flags & KMG_FLAG_FORCE_PARTITIONED) && (cfg->flags & (KMG_FLAG_FORCE_HASH | KMG_FLAG_FORCE_DIRECT))) {
    c->err = "FORCE_PARTITIONED excludes FORCE_HASH / FORCE_DIRECT";
    return bail(KMG_ERR_INVALID_ARG);
  }
  if (cfg->parts_log2 > 20) { c->err = "parts_log2 must be <= 20"; return bail(KMG_ERR_INVALID_ARG); }
  if (cfg->flags & KMG_FLAG_FORCE_PARTITIONED) c->use_dense = false;
  CUC(cudaStreamSynchronize(c->stream));
#undef CUC
  *out = c;
  return KMG_OK;
}

KMG_EXPORT kmg_status kmg_reset(kmg_ctx *c) {
  if (!c) return KMG_ERR_INVALID_ARG;
  CU(c, cudaSetDevice(c->device));
  if (c->fxs) fx_stream_close(c, true);  // an open stream is abandoned with everything else
  std::vector<uint8_t>().swap(c->fx_rest);
  c->fx_rest_ok = false;
  CU(c, cudaStreamSynchronize(c->copy_stream));
  c->pending_slot = -1;  // a submitted but unscanned pre-packed batch is forgotten with everything else
  if (c->use_dense) CU(c, cudaMemsetAsync(c->dense, 0, c->dense_n * 8, c->stream));
  else if (c->mode == kmg_ctx::MODE_TABLE) CU(c, launch_table_init(c->table, c->stream));
  else if (c->mode == kmg_ctx::MODE_PARTITIONED) {
    CU(c, cudaStreamSynchronize(c->stream));
    for (auto &r : c->runs) free_run(c, r);
    c->runs.clear();
    if (c->has_result) free_run(c, c->result);
    c->has_result = false; c->pending_bytes = 0; c->n_consolidations = 0; c->dedup_ratio = 1.0;
    c->feed_kind = 0; c->poisoned = false;
    c->fused_valid = c->fused_cached = false;
  }
  CU(c, cudaMemsetAsync(c->d_counters, 0, CTR_N * sizeof(unsigned long long), c->stream));
  c->distinct_ub = 0; c->n_records = c->n_bases = c->h2d_bytes = 0;
  CU(c, cudaStreamSynchronize(c->stream));
  timers_collect(c);
  c->kernel_ms = c->cat_ms[0] = c->cat_ms[1] = c->cat_ms[2] = 0.0;
  return KMG_OK;
}

KMG_EXPORT kmg_status kmg_count_ascii_device(kmg_ctx *c, const uint8_t *d_seq, const uint8_t *d_qual, const uint64_t *d_offsets,
                                             uint64_t n_records, uint64_t n_bytes) {
  if (!c) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  if (c->shm) return fail(c, KMG_ERR_STATE, "context belongs to a shard group: feed it with kmg_shard_count_ascii(_device)");
  if (n_bytes && !d_seq) return fail(c, KMG_ERR_INVALID_ARG, "d_seq is NULL");
  if (((uintptr_t)d_seq & 15) || ((uintptr_t)d_qual & 15)) return fail(c, KMG_ERR_INVALID_ARG, "d_seq / d_qual must be 16-byte aligned");
  CU(c, cudaSetDevice(c->device));
  if (n_bytes) {
    uint64_t n_words_total = 0;
    bool has_start = false;
    // offsets[0] (== 0) needs no start bit; a single record needs none at all
    kmg_status s = pack_device_ascii(c, d_seq, d_qual, n_records > 1 ? d_offsets : nullptr, n_records, 0, n_bytes, &n_words_total, &has_start);
    if (s == KMG_OK) s = scan_packed(c, n_words_total, has_start);
    if (s != KMG_OK) return s;
  }
  c->n_records += n_records; c->n_bases += n_bytes;
  return KMG_OK;
}


namespace {

// The layout checks of kmg_count_ascii and kmg_shard_count_ascii.  A call without records, or with only empty records and no seq,
// passes with nothing to stage.
kmg_status check_ascii_layout(kmg_ctx *c, const uint8_t *seq, const uint64_t *offsets, uint64_t n_records) {
  if (n_records == 0 || (!seq && offsets && offsets[n_records] == offsets[0])) return KMG_OK;
  if (!offsets || !seq) return fail(c, KMG_ERR_INVALID_ARG, "seq / offsets must not be NULL");
  for (uint64_t r = 0; r < n_records; ++r)
    if (offsets[r + 1] < offsets[r]) return fail(c, KMG_ERR_INVALID_ARG, "offsets must be non-decreasing");
  return KMG_OK;
}

// The host ASCII feed of one checked call over the context's staging ring: seq[offsets[0], offsets[n_records]) in chunks of at most
// batch_bases bytes that overlap by k-1, each with the starts of the records that begin strictly inside it.  The H2D copies run up
// to N_STAGE - 1 chunks ahead of the kernels (processing contains host syncs).  step() packs a chunk and hands it to the caller's
// scan (scan_packed on one context, shard_scan_round in a group).
struct AsciiFeed {
  struct Chunk { uint64_t pos, len, r_lo, nrec; };
  kmg_ctx *c;
  const uint8_t *seq, *qual;
  const uint64_t *offsets;
  uint64_t begin, end;
  bool use_q, src_pinned = false;
  std::vector<Chunk> chunks;
  uint32_t slot0 = 0;
  size_t staged = 0;

  AsciiFeed(kmg_ctx *ctx, const uint8_t *s, const uint8_t *q, const uint64_t *off, uint64_t n_records)
      : c(ctx), seq(s), qual(q), offsets(off), begin(n_records ? off[0] : 0), end(n_records ? off[n_records] : 0),
        use_q(ctx->cfg.has_min_quality && q != nullptr) {
    const uint64_t K1 = (uint64_t)c->k - 1, B = c->batch_bases, step = B - K1;  // B: bytes per chunk including the k-1 overlap
    uint64_t r_lo = 0;
    for (uint64_t pos = begin; pos < end; pos += step) {
      const uint64_t len = std::min<uint64_t>(B, end - pos);
      if (pos != begin && len <= K1) break;  // only the overlap is left: no new windows
      while (r_lo < n_records && offsets[r_lo] <= pos) ++r_lo;  // records with a start strictly inside (pos, pos+len)
      uint64_t r_hi = r_lo;
      while (r_hi < n_records && offsets[r_hi] < pos + len) ++r_hi;
      chunks.push_back(Chunk{pos, len, r_lo, r_hi - r_lo});
    }
  }

  kmg_status open() {
    slot0 = c->next_ascii;
    src_pinned = end > begin && is_pinned_host(seq + begin) && (!use_q || is_pinned_host(qual + begin));
    return ensure_staging(c, !src_pinned, use_q, end - begin);
  }

  // chunk i lives in ring slot (slot0 + i) % N_STAGE; reusing a slot waits for its previous chunk's compute_done
  kmg_status stage(const Chunk &ch, Staging &st) {
    if (st.h2d_pending) { CU(c, cudaEventSynchronize(st.h2d_done)); st.h2d_pending = false; }
    if (st.compute_pending) { CU(c, cudaStreamWaitEvent(c->copy_stream, st.compute_done, 0)); }
    kmg_status es = ensure_offsets(c, st, ch.nrec);
    if (es != KMG_OK) return es;
    const uint8_t *src_seq = seq + ch.pos, *src_qual = use_q ? qual + ch.pos : nullptr;
    if (!src_pinned) {
      memcpy(st.h_seq, src_seq, ch.len); src_seq = st.h_seq;
      if (use_q) { memcpy(st.h_qual, src_qual, ch.len); src_qual = st.h_qual; }
    }
    CU(c, cudaMemcpyAsync(st.d_seq, src_seq, ch.len, cudaMemcpyHostToDevice, c->copy_stream));
    if (use_q) CU(c, cudaMemcpyAsync(st.d_qual, src_qual, ch.len, cudaMemcpyHostToDevice, c->copy_stream));
    if (ch.nrec) {
      memcpy(st.h_off, offsets + ch.r_lo, ch.nrec * 8);
      CU(c, cudaMemcpyAsync(st.d_off, st.h_off, ch.nrec * 8, cudaMemcpyHostToDevice, c->copy_stream));
    }
    c->h2d_bytes += ch.len * (use_q ? 2 : 1) + ch.nrec * 8;
    CU(c, cudaEventRecord(st.h2d_done, c->copy_stream));
    st.h2d_pending = true;
    return KMG_OK;
  }

  template <class Scan>
  kmg_status step(size_t i, Scan &&scan) {
    for (; staged < chunks.size() && staged < i + N_STAGE; ++staged) {
      kmg_status ss = stage(chunks[staged], c->st[(slot0 + staged) % N_STAGE]);
      if (ss != KMG_OK) return ss;
    }
    Staging &st = c->st[(slot0 + i) % N_STAGE];
    const Chunk &ch = chunks[i];
    CU(c, cudaStreamWaitEvent(c->stream, st.h2d_done, 0));
    uint64_t n_words_total = 0;
    bool has_start = false;
    kmg_status s = pack_device_ascii(c, st.d_seq, use_q ? st.d_qual : nullptr, ch.nrec ? st.d_off : nullptr, ch.nrec, ch.pos, ch.len,
                                     &n_words_total, &has_start);
    if (s != KMG_OK) return s;
    CU(c, cudaEventRecord(st.compute_done, c->stream));  // the staging slot is free once the chunk is packed
    st.compute_pending = true;
    return scan(n_words_total, has_start);
  }

  // After the last step: the copies read the CALLER's buffer when it is pinned, and it must be reusable when the call returns.
  kmg_status close() {
    c->next_ascii = (slot0 + (uint32_t)chunks.size()) % N_STAGE;
    if (src_pinned)
      for (auto &st : c->st)
        if (st.h2d_pending) { CU(c, cudaEventSynchronize(st.h2d_done)); st.h2d_pending = false; }
    return KMG_OK;
  }
};

constexpr int FASTQ_SYNC_LINES = 64;  // lines searched for a FASTQ record start at a chunk end (backward) or a rank cut (forward)

// Does the line at p open a FASTQ record?  '@' first, and the line after next begins with '+' (a quality line may begin with '@',
// but the line after next of a quality line is a sequence line).
bool fastq_record_start(const uint8_t *buf, uint64_t len, uint64_t p) {
  if (p >= len || buf[p] != '@') return false;
  const void *l1 = memchr(buf + p, '\n', (size_t)(len - p));
  const void *l2 = l1 ? memchr((const uint8_t *)l1 + 1, '\n', (size_t)(buf + len - ((const uint8_t *)l1 + 1))) : nullptr;
  return l2 && (const uint8_t *)l2 + 1 < buf + len && ((const uint8_t *)l2)[1] == '+';
}

struct FxChunk { uint64_t pos, len; };

const char *const FX_NO_NEWLINE = "a line is longer than a staging chunk (raise batch_bases or use the host splitter)";
const char *const FX_NO_RECORD = "no FASTQ record boundary found near a chunk end (multi-line FASTQ? use the host splitter)";

// The last chunk boundary in buf[pos, stop) above pos (the lines after it are read up to len): the start of the last line
// (FASTA), or the last line start within FASTQ_SYNC_LINES lines that opens a record (FASTQ).  nullptr, or why there is none.
const char *last_fastx_cut(const uint8_t *buf, uint64_t len, uint64_t pos, uint64_t stop, bool is_fastq, uint64_t *cut) {
  const void *nl = memrchr(buf + pos, '\n', (size_t)(stop - pos));
  if (!nl) return FX_NO_NEWLINE;
  uint64_t p = (uint64_t)((const uint8_t *)nl - buf) + 1;
  if (is_fastq) {  // step back line by line to a line that opens a record
    bool found = false;
    for (int tries = 0; tries < FASTQ_SYNC_LINES && p > pos; ++tries) {
      if (fastq_record_start(buf, len, p)) { found = true; break; }
      const void *prev = p >= 2 ? memrchr(buf + pos, '\n', (size_t)(p - 1 - pos)) : nullptr;  // start of the previous line
      if (!prev) break;
      p = (uint64_t)((const uint8_t *)prev - buf) + 1;
    }
    if (!found || p <= pos) return FX_NO_RECORD;
  }
  *cut = p;
  return nullptr;
}

// Staging chunks of buf[begin, end) (begin and end at line starts (FASTA) / record starts (FASTQ), or end == len): each holds at
// most cb bytes and ends at a line start (FASTA) or a record start (FASTQ).
kmg_status plan_fastx_chunks(kmg_ctx *c, const uint8_t *buf, uint64_t len, uint64_t begin, uint64_t end, bool is_fastq, uint64_t cb,
                             std::vector<FxChunk> &chunks) {
  for (uint64_t pos = begin; pos < end;) {
    uint64_t stop = std::min(end, pos + cb);
    if (stop < end) {
      const char *why = last_fastx_cut(buf, len, pos, stop, is_fastq, &stop);
      if (why) return fail(c, KMG_ERR_PARSE, why);
    }
    chunks.push_back(FxChunk{pos, stop - pos});
    pos = stop;
  }
  return KMG_OK;
}

// The device parser's driver over chunks that are cut at line (FASTA) / record (FASTQ) starts -- or, in a stream, inside a FASTA
// sequence line between two non-blank bytes: pooled parse buffers, per chunk the parse kernels, the scatter of sequence
// (+ quality) bytes and record marks, the carry of a FASTA record's last k-1 bases into the next chunk, and the error words.
// parse() takes a chunk whose bytes are in (or on their way to) a staging slot and leaves it packed in the context's stream for the
// caller's scan (scan_packed on one context, shard_scan_round in a group).  Over the planned chunks of one file image, step()
// stages the raw chunks through the context's ring itself, up to N_STAGE - 1 chunks ahead; a stream fills the slots (FxStream).
struct FastxFeed {
  kmg_ctx *c;
  const uint8_t *buf;                  // the file image, or nullptr for a stream
  const std::vector<FxChunk> *chunks;  // the image's planned chunks
  bool is_fastq, use_q, src_pinned = false;
  bool refused = false;  // the last parse() refused its chunk's layout before anything of the chunk was counted
  uint64_t K1 = 0, max_len = 0, prev_n = 0, bases = 0;  // prev_n: sequence bases the last chunk left (their tail is the next carry)
  uint8_t *d_kind = nullptr, *d_keep = nullptr, *d_seq = nullptr, *d_qual = nullptr, *d_mark = nullptr, *d_carry = nullptr;
  uint32_t *d_lineno = nullptr, *d_pos_s = nullptr, *d_pos_q = nullptr, *d_misc = nullptr, *h_tot = nullptr;
  void *d_tmp = nullptr;
  size_t tmp_bytes = 0, staged = 0;
  uint32_t slot0 = 0, thr = 0;

  FastxFeed(kmg_ctx *ctx, bool fq, const uint8_t *b = nullptr, const std::vector<FxChunk> *ch = nullptr)
      : c(ctx), buf(b), chunks(ch), is_fastq(fq), use_q(fq && ctx->cfg.has_min_quality) {}
  unsigned long long *d_nrec() const { return reinterpret_cast<unsigned long long *>(d_misc); }  // [0..1] n_records (u64)
  uint32_t *d_err() const { return d_misc + 4; }  // [2..3] totals, [4] error word, [5] pending record start

  // stream_len: the largest chunk of a stream (the slots are filled by the caller, from pinned memory)
  kmg_status open(uint64_t stream_len = 0) {
    K1 = (uint64_t)c->k - 1;
    slot0 = c->next_ascii;
    max_len = stream_len;
    if (chunks) for (auto &ch : *chunks) max_len = std::max(max_len, ch.len);
    src_pinned = buf && is_pinned_host(buf);
    kmg_status s = ensure_staging(c, buf && !src_pinned, false, max_len);  // a stream pins the slots it uses itself
    if (s != KMG_OK) return s;
    tmp_bytes = fastx_scan_tmp_bytes(max_len);
    cudaError_t e = pool_alloc(c, &d_kind, max_len);
    if (e == cudaSuccess) e = pool_alloc(c, &d_keep, max_len);
    if (e == cudaSuccess) e = pool_alloc(c, &d_pos_s, max_len * 4);
    if (e == cudaSuccess && is_fastq) e = pool_alloc(c, &d_lineno, max_len * 4);
    if (e == cudaSuccess && is_fastq) e = pool_alloc(c, &d_pos_q, max_len * 4);
    if (e == cudaSuccess) e = pool_alloc(c, &d_seq, max_len + K1 + 64);
    if (e == cudaSuccess && use_q) e = pool_alloc(c, &d_qual, max_len + K1 + 64);
    if (e == cudaSuccess) e = pool_alloc(c, &d_mark, max_len + K1 + 64);
    if (e == cudaSuccess) e = pool_alloc(c, &d_carry, 2 * 64);
    if (e == cudaSuccess) e = pool_alloc(c, &d_misc, 64);
    if (e == cudaSuccess) e = pool_alloc(c, &d_tmp, tmp_bytes);
    if (e == cudaSuccess) e = cudaHostAlloc(&h_tot, 16, cudaHostAllocDefault);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_misc, 0, 64, c->stream);
    if (e != cudaSuccess) return cuda_fail(c, e, "cudaMalloc(fastx parse buffers)");
    thr = quality_threshold(c);
    return KMG_OK;
  }

  // The first chunk continues a FASTA record that began before it (a rank's slice in a group): its last n <= k-1 bases and their
  // record marks, and whether a header line ends right before the chunk (its record then starts with the chunk's first base).
  kmg_status seed_carry(const uint8_t *seq, const uint8_t *mark, uint64_t n, bool pending) {
    if (n) {
      CU(c, cudaMemcpyAsync(d_carry + (K1 - n), seq, n, cudaMemcpyHostToDevice, c->stream));
      CU(c, cudaMemcpyAsync(d_carry + 64 + (K1 - n), mark, n, cudaMemcpyHostToDevice, c->stream));
    }
    if (pending) CU(c, cudaMemsetAsync(d_err() + 1, 1, 1, c->stream));
    prev_n = n;
    return KMG_OK;
  }

  // Queue the copy of len bytes at src (pinned) into the slot's device buffer once the slot's previous chunk has been consumed.
  kmg_status copy_to_slot(Staging &st, const uint8_t *src, uint64_t len) {
    if (st.compute_pending) { CU(c, cudaStreamWaitEvent(c->copy_stream, st.compute_done, 0)); }
    CU(c, cudaMemcpyAsync(st.d_seq, src, len, cudaMemcpyHostToDevice, c->copy_stream));
    c->h2d_bytes += len;
    CU(c, cudaEventRecord(st.h2d_done, c->copy_stream));
    st.h2d_pending = true;
    return KMG_OK;
  }

  kmg_status stage(const FxChunk &ch, Staging &st) {
    if (st.h2d_pending) { CU(c, cudaEventSynchronize(st.h2d_done)); st.h2d_pending = false; }
    const uint8_t *src = buf + ch.pos;
    if (!src_pinned) { memcpy(st.h_seq, src, ch.len); src = st.h_seq; }
    return copy_to_slot(st, src, ch.len);
  }

  // Chunk i of the image: staged ahead, then parsed.
  template <class Scan>
  kmg_status step(size_t i, Scan &&scan, bool *scanned) {
    *scanned = false;
    for (; staged < chunks->size() && staged < i + N_STAGE; ++staged) {
      kmg_status ss = stage((*chunks)[staged], c->st[(slot0 + staged) % N_STAGE]);
      if (ss != KMG_OK) return ss;
    }
    const FxChunk &ch = (*chunks)[i];
    return parse(c->st[(slot0 + i) % N_STAGE], ch.len, buf[ch.pos] == '>', scan, scanned);
  }

  // The chunk of len bytes whose copy into st was queued last (opens_header: its first byte is '>'): parse, pack, and -- when it
  // holds sequence bases (with the carry) -- scan(n_words_total).  *scanned tells whether it did.
  template <class Scan>
  kmg_status parse(Staging &st, uint64_t len, bool opens_header, Scan &&scan, bool *scanned) {
    *scanned = false;
    refused = false;
    uint32_t *err = d_err();
    CU(c, cudaStreamWaitEvent(c->stream, st.h2d_done, 0));
    // a FASTA chunk that does not open with a header continues the previous chunk's last record: its last k-1 bases (and their
    // record marks) are put in front, so that the windows spanning the cut are counted -- and none twice (k-1 bases hold no window)
    const uint64_t carry = (!is_fastq && !opens_header) ? std::min<uint64_t>(K1, prev_n) : 0;
    CU(c, cudaMemsetAsync(d_mark, 0, len + K1 + 64, c->stream));
    CU(c, cudaMemsetAsync(err, 0, 4, c->stream));
    if (carry) {
      CU(c, cudaMemcpyAsync(d_seq, d_carry + (K1 - carry), carry, cudaMemcpyDeviceToDevice, c->stream));
      CU(c, cudaMemcpyAsync(d_mark, d_carry + 64 + (K1 - carry), carry, cudaMemcpyDeviceToDevice, c->stream));
    }
    CU(c, launch_fastx_parse(st.d_seq, len, is_fastq, d_kind, d_keep, d_lineno, d_pos_s, d_pos_q, d_tmp, tmp_bytes, carry, d_seq, d_qual, d_mark,
                             d_nrec(), err, h_tot, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    const uint32_t total_s = h_tot[0], total_q = h_tot[1], perr = h_tot[2];
    refused = (perr & 3u) != 0;
    if (perr & 1u) return fail(c, KMG_ERR_PARSE, "FASTQ record does not start with '@' (multi-line FASTQ is not handled by the device parser)");
    if (perr & 2u) return fail(c, KMG_ERR_PARSE, "FASTQ record without a '+' separator line where one is expected");
    if (is_fastq && total_s != total_q) return fail(c, KMG_ERR_PARSE, "sequence and quality lengths differ");
    // a record whose header closed the previous chunk starts with this chunk's first base (the scatter below may raise the flag anew)
    if (!is_fastq && total_s) CU(c, launch_fastx_apply_pending(err + 1, d_mark + carry, c->stream));
    CU(c, launch_fastx_scatter(st.d_seq, len, is_fastq, d_kind, d_lineno, d_keep, d_pos_s, d_pos_q, carry, total_s, d_seq, use_q ? d_qual : nullptr,
                               d_mark, d_nrec(), err, c->stream));
    CU(c, cudaEventRecord(st.compute_done, c->stream));  // the raw chunk has been consumed
    st.compute_pending = true;
    const uint64_t n = carry + total_s;
    bases += total_s;
    prev_n = n;
    if (!n) return KMG_OK;
    const uint64_t n_words_total = round_up((n + 31) / 32, TILE_WORDS);
    kmg_status ps = ensure_packed(c, n_words_total);
    if (ps != KMG_OK) return ps;
    CU(c, launch_ingest(d_seq, use_q ? d_qual : nullptr, n, thr, n_words_total, c->d_bases, c->d_valid, c->stream));
    CU(c, launch_marks_to_bits(d_mark, n, n_words_total, c->d_start, c->stream));
    if (!is_fastq) {  // keep the tail for the next chunk
      const uint64_t t = std::min<uint64_t>(K1, n);
      if (t) {
        CU(c, cudaMemcpyAsync(d_carry + (K1 - t), d_seq + (n - t), t, cudaMemcpyDeviceToDevice, c->stream));
        CU(c, cudaMemcpyAsync(d_carry + 64 + (K1 - t), d_mark + (n - t), t, cudaMemcpyDeviceToDevice, c->stream));
      }
    }
    *scanned = true;
    ps = scan(n_words_total);
    if (ps != KMG_OK) return ps;
    if (is_fastq && use_q) {  // a quality mismatch inside a record shows up at the next record start (checked in the scatter)
      uint32_t e2 = 0;
      CU(c, cudaMemcpyAsync(&e2, err, 4, cudaMemcpyDeviceToHost, c->stream));
      CU(c, cudaStreamSynchronize(c->stream));
      if (e2 & 8u) return fail(c, KMG_ERR_PARSE, "sequence and quality lengths differ");
    }
    return KMG_OK;
  }

  // Records (header lines) the parsed chunks held.
  kmg_status records(uint64_t *n) {
    unsigned long long h = 0;
    CU(c, cudaMemcpyAsync(&h, d_nrec(), 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    *n = h;
    return KMG_OK;
  }

  // After the last step (or a failed one): the caller's buffer must be reusable when the call returns.
  void close(bool failed) {
    if (failed) { cudaStreamSynchronize(c->stream); cudaStreamSynchronize(c->copy_stream); }
    if (chunks) c->next_ascii = (slot0 + (uint32_t)chunks->size()) % N_STAGE;
    for (auto &st : c->st) if (st.h2d_pending && src_pinned) { cudaEventSynchronize(st.h2d_done); st.h2d_pending = false; }
    pool_free(c, d_kind); pool_free(c, d_keep); pool_free(c, d_seq); pool_free(c, d_qual); pool_free(c, d_mark); pool_free(c, d_carry);
    pool_free(c, d_lineno); pool_free(c, d_pos_s); pool_free(c, d_pos_q); pool_free(c, d_misc); pool_free(c, d_tmp);
    if (h_tot) cudaFreeHost(h_tot);
    h_tot = nullptr;
  }
};

}  // namespace

KMG_EXPORT kmg_status kmg_count_ascii(kmg_ctx *c, const uint8_t *seq, const uint8_t *qual, const uint64_t *offsets, uint64_t n_records) {
  if (!c) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  if (c->shm) return fail(c, KMG_ERR_STATE, "context belongs to a shard group: feed it with kmg_shard_count_ascii(_device)");
  kmg_status s = check_ascii_layout(c, seq, offsets, n_records);
  if (s != KMG_OK) return s;
  if (n_records == 0 || !seq) { c->n_records += n_records; return KMG_OK; }
  CU(c, cudaSetDevice(c->device));
  AsciiFeed feed(c, seq, qual, offsets, n_records);
  const uint64_t bases = feed.end - feed.begin;
  if (feed.use_q && !c->cfg.expected_distinct && c->mode == kmg_ctx::MODE_UNDECIDED && !c->use_dense)
    c->plan_scale = (double)bases / (double)std::min<uint64_t>(bases, c->batch_bases);  // decided after the first chunk's ingest (scan_packed)
  else s = decide_mode(c, bases);  // plan for the whole call, not for its first staging chunk
  if (s == KMG_OK) s = feed.open();
  for (size_t i = 0; s == KMG_OK && i < feed.chunks.size(); ++i)
    s = feed.step(i, [&](uint64_t n_words_total, bool has_start) { return scan_packed(c, n_words_total, has_start); });
  if (s != KMG_OK) return s;
  c->n_records += n_records; c->n_bases += bases;
  return feed.close();
}

// FASTA / FASTQ file image (HOST bytes, e.g. an mmap'ed file: src/mmap.rs:33-71) -> counts, with the records found ON THE DEVICE:
// the raw bytes go over PCIe in chunks cut at line (FASTA) / record (FASTQ) boundaries, a few small kernels classify the lines,
// compact sequence (+ quality) bytes, mark the record starts, and the usual ingest + scan follow.  Replaces reader::read /
// read_with_quality (src/reader.rs:82-247: whole file -> Vec<Record> -> Vec<SequenceWithQuality>, two host copies) for
// well-formed input; multi-line FASTQ, or a line longer than a chunk, is refused with KMG_ERR_PARSE -- nothing has been
// counted then only if it happens in the first chunk, so callers fall back to kmg_parse_fastx + kmg_count_ascii after kmg_reset.
KMG_EXPORT kmg_status kmg_count_fastx(kmg_ctx *c, const uint8_t *buf, uint64_t len, int is_fastq, uint64_t *n_records_out) {
  if (!c || (len && !buf)) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  if (c->shm) return fail(c, KMG_ERR_STATE, "context belongs to a shard group: feed it with kmg_shard_count_fastx / kmg_shard_count_ascii(_device)");
  if (n_records_out) *n_records_out = 0;
  if (len == 0) return KMG_OK;
  const uint8_t marker = is_fastq ? '@' : '>';
  if (buf[0] != marker) return fail(c, KMG_ERR_PARSE, is_fastq ? "FASTQ record does not start with '@' (record 0)" : "FASTA record does not start with '>' (record 0)");
  CU(c, cudaSetDevice(c->device));
  const bool use_q = is_fastq && c->cfg.has_min_quality;
  std::vector<FxChunk> chunks;
  kmg_status s = plan_fastx_chunks(c, buf, len, 0, len, is_fastq, std::min<uint64_t>(c->batch_bases, 1ull << 30), chunks);
  if (s != KMG_OK) return s;
  uint64_t max_len = 0;
  for (auto &ch : chunks) max_len = std::max(max_len, ch.len);
  if (max_len >= (1ull << 32)) return fail(c, KMG_ERR_INVALID_ARG, "staging chunks must stay below 4 GiB");
  // ---- plan the table / partitions for the whole file
  if (use_q && !c->cfg.expected_distinct && c->mode == kmg_ctx::MODE_UNDECIDED && !c->use_dense) c->plan_scale = (double)len / (double)chunks[0].len;
  else s = decide_mode(c, is_fastq ? len / 2 : len);
  if (s != KMG_OK) return s;
  FastxFeed feed(c, is_fastq, buf, &chunks);
  s = feed.open();
  uint64_t n_rec = 0;
  for (size_t i = 0; s == KMG_OK && i < chunks.size(); ++i) {
    bool scanned = false;
    s = feed.step(i, [&](uint64_t n_words_total) { return scan_packed(c, n_words_total, true); }, &scanned);
  }
  if (s == KMG_OK) s = feed.records(&n_rec);
  feed.close(s != KMG_OK);
  if (s != KMG_OK) return s;
  c->n_records += n_rec; c->n_bases += feed.bases;
  if (n_records_out) *n_records_out = n_rec;
  return KMG_OK;
}

// ---- FASTA / FASTQ byte streams (kmg_fastx_stream_*): the file-image parser over input that arrives in pieces ----------------
// Pushed bytes fill the ring slot `cur` in place.  A full slot is cut at its last line / record start (plan_fastx_chunks' rules;
// a FASTA slot without a newline inside its sequence line), the copy of the chunk in front of the cut is queued at once, and then
// the chunk before it (`pend`) is parsed and scanned, so the copy of chunk i overlaps the kernels of chunk i-1; the bytes after
// the cut open the other slot.  The stream alternates between two slots of the ring (pinned on first use): host memory is those
// two slots whatever the stream's length.
struct FxStream {
  FastxFeed feed;
  uint64_t cb = 0;         // bytes a slot holds when it is cut
  uint32_t slot[2] = {0, 1};  // the ring slots the stream alternates between
  uint32_t cur = 0;        // the slot being filled
  uint64_t fill = 0;
  int pend = -1;           // the slot whose chunk has been queued for the device but not parsed
  uint64_t pend_len = 0;
  bool started = false;    // byte 0 has been checked
  bool mid_line = false;   // the slot being filled continues a FASTA sequence line that the last cut split
  uint64_t plan_len = 0;   // size hint that scales the quality-filtered plan of the first chunk (as kmg_count_fastx does)
  uint64_t rec0 = 0, bases0 = 0;           // the context's records / bases before the stream
  unsigned long long *h_nrec = nullptr;    // pinned: records of the chunks parsed so far, read back without a synchronisation
  FxStream(kmg_ctx *c, bool fq) : feed(c, fq) {}
};

namespace {

void fx_stream_close(kmg_ctx *c, bool failed) {
  FxStream *x = c->fxs;
  x->feed.close(failed);
  c->next_ascii = (x->cur + 1) % N_STAGE;
  if (x->h_nrec) cudaFreeHost(x->h_nrec);
  delete x;
  c->fxs = nullptr;
}

// A refusal that leaves the context usable: the bytes from the refused chunk on -- the pending chunk if it is the refused one,
// the slot being filled, the caller's bytes this push has not consumed -- become the stream's rest, and the stream closes.
kmg_status fx_stream_refuse(kmg_ctx *c, const uint8_t *more, uint64_t n_more) {
  FxStream *x = c->fxs;
  std::vector<uint8_t>().swap(c->fx_rest);
  if (x->pend >= 0) c->fx_rest.insert(c->fx_rest.end(), c->st[x->pend].h_seq, c->st[x->pend].h_seq + x->pend_len);
  c->fx_rest.insert(c->fx_rest.end(), c->st[x->cur].h_seq, c->st[x->cur].h_seq + x->fill);
  if (n_more) c->fx_rest.insert(c->fx_rest.end(), more, more + n_more);
  // the records and bases of exactly the chunks counted before the refused one (the refused chunk reached no scatter)
  const std::string why = c->err;
  uint64_t n_rec = 0;
  if (x->feed.records(&n_rec) != KMG_OK) { fx_stream_close(c, true); return KMG_ERR_CUDA; }
  c->n_records = x->rec0 + n_rec; c->n_bases = x->bases0 + x->feed.bases;
  c->err = why;
  c->fx_rest_ok = true;
  fx_stream_close(c, true);
  return KMG_ERR_PARSE;
}

// A failed step: a layout refusal before anything of the chunk was counted keeps the context usable, everything else is final.
kmg_status fx_stream_fail(kmg_ctx *c, kmg_status s, const uint8_t *more, uint64_t n_more) {
  if (s == KMG_ERR_PARSE && c->fxs->feed.refused) return fx_stream_refuse(c, more, n_more);
  fx_stream_close(c, true);
  return s;
}

// Parse and scan the pending chunk; the context's progress then counts the bases of every parsed chunk and the records of all
// chunks before it.
kmg_status fx_stream_parse_pending(kmg_ctx *c) {
  FxStream *x = c->fxs;
  if (x->pend < 0) return KMG_OK;
  Staging &st = c->st[x->pend];
  if (x->plan_len) { c->plan_scale = (double)x->plan_len / (double)x->pend_len; x->plan_len = 0; }
  bool scanned = false;
  kmg_status s = x->feed.parse(st, x->pend_len, st.h_seq[0] == '>', [&](uint64_t n_words_total) { return scan_packed(c, n_words_total, true); },
                               &scanned);
  if (s != KMG_OK) return s;
  x->pend = -1;
  c->n_records = x->rec0 + *x->h_nrec;  // copied behind the previous chunk, complete since the parse synchronised
  CU(c, cudaMemcpyAsync(x->h_nrec, x->feed.d_nrec(), 8, cudaMemcpyDeviceToHost, c->stream));
  c->n_bases = x->bases0 + x->feed.bases;
  return KMG_OK;
}

// The slot being filled holds cb bytes: cut it, queue the chunk's copy, count the pending chunk, move the rest to the next slot.
// more / n_more: the bytes of the current push not consumed yet (part of the rest if the stream is refused).
kmg_status fx_stream_flush(kmg_ctx *c, const uint8_t *more, uint64_t n_more) {
  FxStream *x = c->fxs;
  Staging &st = c->st[x->cur];
  const uint8_t *b = st.h_seq;
  uint64_t cut = 0;
  const char *why = last_fastx_cut(b, x->fill, 0, x->fill, x->feed.is_fastq, &cut);
  bool mid = false;
  if (why == FX_NO_NEWLINE && !x->feed.is_fastq) {
    // a sequence line longer than a slot is cut between two non-blank bytes, not before a '>' (the next chunk must not open a
    // header); a slot that opens a header line holds no such position
    why = "a FASTA header line is longer than a staging chunk, or a sequence line holds no cut between two non-blank bytes";
    if (x->mid_line || b[0] != '>') {
      auto blank = [](uint8_t v) { return v == ' ' || (v >= 9 && v <= 13); };
      for (uint64_t p = x->fill - 1; p > 0; --p)
        if (!blank(b[p - 1]) && !blank(b[p]) && b[p] != '>') { cut = p; why = nullptr; mid = true; break; }
    }
  }
  kmg_status s = KMG_OK;
  if (why) {
    if ((s = fx_stream_parse_pending(c)) != KMG_OK) return fx_stream_fail(c, s, more, n_more);
    fail(c, KMG_ERR_PARSE, why);
    return fx_stream_refuse(c, more, n_more);
  }
  if ((s = x->feed.copy_to_slot(st, b, cut)) != KMG_OK) return fx_stream_fail(c, s, more, n_more);
  if ((s = fx_stream_parse_pending(c)) != KMG_OK) return fx_stream_fail(c, s, more, n_more);
  const uint32_t nxt = x->cur == x->slot[0] ? x->slot[1] : x->slot[0];
  Staging &ns = c->st[nxt];
  if (ns.h2d_pending) {
    const cudaError_t e = cudaEventSynchronize(ns.h2d_done);  // the slot's last chunk has left the host
    if (e != cudaSuccess) { cuda_fail(c, e, "cudaEventSynchronize(h2d_done)"); return fx_stream_fail(c, KMG_ERR_CUDA, more, n_more); }
    ns.h2d_pending = false;
  }
  memcpy(ns.h_seq, b + cut, x->fill - cut);
  x->pend = (int)x->cur; x->pend_len = cut;
  x->cur = nxt; x->fill -= cut; x->mid_line = mid;
  return KMG_OK;
}

}  // namespace

KMG_EXPORT kmg_status kmg_fastx_stream_begin(kmg_ctx *c, int is_fastq, uint64_t size_hint) {
  if (!c) return KMG_ERR_INVALID_ARG;
  if (c->shm) return fail(c, KMG_ERR_STATE, "context belongs to a shard group: a stream is counted on a context of its own");
  if (c->fxs) return fail(c, KMG_ERR_STATE, "a FASTA / FASTQ stream is already open on this context");
  CU(c, cudaSetDevice(c->device));
  std::vector<uint8_t>().swap(c->fx_rest);
  c->fx_rest_ok = false;
  kmg_status s = scan_pending_batch(c);  // the pre-packed feed's last batch uses the ring's events
  if (s != KMG_OK) return s;
  // a slot holds a chunk of min(batch_bases, 2^30) bytes; a known small stream gets smaller slots (1 MiB at least)
  uint64_t cb = std::min<uint64_t>(c->batch_bases, 1ull << 30);
  if (size_hint) cb = std::min<uint64_t>(cb, std::max<uint64_t>(round_up(size_hint, 64), 1ull << 20));
  const bool use_q = is_fastq && c->cfg.has_min_quality;
  FxStream *x = new FxStream(c, is_fastq != 0);
  x->cb = cb;
  if (size_hint) {  // plan the table / partitions for the whole stream, as kmg_count_fastx does for a file
    if (use_q && !c->cfg.expected_distinct && c->mode == kmg_ctx::MODE_UNDECIDED && !c->use_dense) x->plan_len = size_hint;
    else s = decide_mode(c, is_fastq ? size_hint / 2 : size_hint);
  }
  if (s == KMG_OK) s = x->feed.open(cb);
  cudaError_t e = cudaSuccess;
  if (s == KMG_OK) {
    x->slot[0] = x->cur = c->next_ascii;
    x->slot[1] = (c->next_ascii + 1) % N_STAGE;
    e = cudaHostAlloc(&x->h_nrec, 8, cudaHostAllocDefault);
    for (uint32_t i : x->slot) {
      Staging &st = c->st[i];
      if (e == cudaSuccess && !st.h_seq) e = cudaHostAlloc(&st.h_seq, c->staging_cap, cudaHostAllocDefault);
    }
    Staging &st = c->st[x->cur];
    if (e == cudaSuccess && st.h2d_pending) e = cudaEventSynchronize(st.h2d_done);
    if (e == cudaSuccess) { *x->h_nrec = 0; st.h2d_pending = false; }
    else s = cuda_fail(c, e, "stream ring");
  }
  x->rec0 = c->n_records; x->bases0 = c->n_bases;
  c->fxs = x;
  if (s != KMG_OK) fx_stream_close(c, true);
  return s;
}

KMG_EXPORT kmg_status kmg_fastx_stream_push(kmg_ctx *c, const uint8_t *bytes, uint64_t n) {
  if (!c) return KMG_ERR_INVALID_ARG;
  if (!c->fxs) return fail(c, KMG_ERR_STATE, "no FASTA / FASTQ stream is open on this context (kmg_fastx_stream_begin)");
  if (n && !bytes) return fail(c, KMG_ERR_INVALID_ARG, "bytes is NULL");
  CU(c, cudaSetDevice(c->device));
  FxStream *x = c->fxs;
  if (n && !x->started) {
    x->started = true;
    if (bytes[0] != (x->feed.is_fastq ? '@' : '>')) {
      fail(c, KMG_ERR_PARSE, x->feed.is_fastq ? "FASTQ record does not start with '@' (record 0)" : "FASTA record does not start with '>' (record 0)");
      return fx_stream_refuse(c, bytes, n);
    }
  }
  while (n) {
    const uint64_t take = std::min<uint64_t>(n, x->cb - x->fill);
    memcpy(c->st[x->cur].h_seq + x->fill, bytes, take);
    x->fill += take; bytes += take; n -= take;
    if (x->fill == x->cb) {
      const kmg_status s = fx_stream_flush(c, bytes, n);
      if (s != KMG_OK) return s;
    }
  }
  return KMG_OK;
}

KMG_EXPORT kmg_status kmg_fastx_stream_end(kmg_ctx *c, uint64_t *n_records_out) {
  if (!c) return KMG_ERR_INVALID_ARG;
  if (n_records_out) *n_records_out = 0;
  if (!c->fxs) return fail(c, KMG_ERR_STATE, "no FASTA / FASTQ stream is open on this context (kmg_fastx_stream_begin)");
  CU(c, cudaSetDevice(c->device));
  FxStream *x = c->fxs;
  Staging &st = c->st[x->cur];
  kmg_status s = x->fill ? x->feed.copy_to_slot(st, st.h_seq, x->fill) : KMG_OK;
  if (s == KMG_OK) s = fx_stream_parse_pending(c);
  if (s == KMG_OK && x->fill) {  // the last chunk: whatever is left, a last line without '\n' included
    x->pend = (int)x->cur; x->pend_len = x->fill; x->fill = 0;
    s = fx_stream_parse_pending(c);
  }
  uint64_t n_rec = 0;
  if (s == KMG_OK) s = x->feed.records(&n_rec);
  if (s != KMG_OK) return fx_stream_fail(c, s, nullptr, 0);
  c->n_records = x->rec0 + n_rec; c->n_bases = x->bases0 + x->feed.bases;
  fx_stream_close(c, false);
  if (n_records_out) *n_records_out = n_rec;
  return KMG_OK;
}

KMG_EXPORT kmg_status kmg_fastx_stream_rest(kmg_ctx *c, uint8_t *bytes, uint64_t cap, uint64_t *n_out) {
  if (!c || !n_out) return KMG_ERR_INVALID_ARG;
  if (!c->fx_rest_ok) return fail(c, KMG_ERR_STATE, "no refused stream: the rest exists after a KMG_ERR_PARSE that left the context usable");
  *n_out = c->fx_rest.size();
  if (!bytes) return KMG_OK;
  if (cap < c->fx_rest.size()) return fail(c, KMG_ERR_CAPACITY, "rest needs " + std::to_string(c->fx_rest.size()) + " bytes");
  if (!c->fx_rest.empty()) memcpy(bytes, c->fx_rest.data(), c->fx_rest.size());
  return KMG_OK;
}

// ---- pre-packed, zero-copy feed (the Rust reader layer packs 2-bit words + masks straight into pinned memory) ------------------
// N_STAGE pinned slots, each with its own packed device buffers.  kmg_submit_batch queues the slot's H2D copy on the copy stream
// at once and then scans the batch submitted BEFORE it, so the copy of batch i overlaps the kernels of batch i-1 while the
// producer fills batch i+1; the last batch is scanned by whichever call needs the table next (finalize, export, ...).
namespace {
kmg_status scan_pending_batch(kmg_ctx *c) {
  if (c->pending_slot < 0) return KMG_OK;
  Staging &s = c->st[c->pending_slot];
  const uint64_t n_words_total = c->pending_words;
  c->pending_slot = -1;
  CU(c, cudaStreamWaitEvent(c->stream, s.h2d_done, 0));
  // the scan reads the context's packed stream: point it at this slot's buffers for the duration of the call
  uint64_t *sb = c->d_bases; uint32_t *sv = c->d_valid, *ss = c->d_start; const uint64_t sw = c->packed_words;
  c->d_bases = s.dp_bases; c->d_valid = s.dp_valid; c->d_start = s.dp_start; c->packed_words = c->dp_words;
  const kmg_status st = scan_packed(c, n_words_total, true);
  c->d_bases = sb; c->d_valid = sv; c->d_start = ss; c->packed_words = sw;
  if (st != KMG_OK) return st;
  CU(c, cudaEventRecord(s.compute_done, c->stream));
  s.compute_pending = true;
  return KMG_OK;
}
}  // namespace

KMG_EXPORT kmg_status kmg_acquire_batch(kmg_ctx *c, kmg_batch *b) {
  if (!c || !b) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  CU(c, cudaSetDevice(c->device));
  const uint64_t words = round_up((c->batch_bases + 31) / 32, TILE_WORDS);
  if (!c->packed_feed_ready) {
    for (int i = 0; i < N_STAGE; ++i) {
      Staging &s = c->st[i];
      CU(c, cudaHostAlloc(&s.hp_bases, words * 8, cudaHostAllocDefault));
      CU(c, cudaHostAlloc(&s.hp_valid, words * 4, cudaHostAllocDefault));
      CU(c, cudaHostAlloc(&s.hp_start, words * 4, cudaHostAllocDefault));
      memset(s.hp_bases, 0, words * 8); memset(s.hp_valid, 0, words * 4); memset(s.hp_start, 0, words * 4);
      CU(c, cudaMalloc(&s.dp_bases, (LEAD_BASE_WORDS + words) * 8));
      CU(c, cudaMalloc(&s.dp_valid, (LEAD_MASK_WORDS + words) * 4));
      CU(c, cudaMalloc(&s.dp_start, (LEAD_MASK_WORDS + words) * 4));
      CU(c, cudaMemsetAsync(s.dp_bases, 0, LEAD_BASE_WORDS * 8, c->stream));
      CU(c, cudaMemsetAsync(s.dp_valid, 0, LEAD_MASK_WORDS * 4, c->stream));
      CU(c, cudaMemsetAsync(s.dp_start, 0, LEAD_MASK_WORDS * 4, c->stream));
      if (!s.h2d_done) {
        CU(c, cudaEventCreateWithFlags(&s.h2d_done, cudaEventDisableTiming));
        CU(c, cudaEventCreateWithFlags(&s.compute_done, cudaEventDisableTiming));
      }
    }
    CU(c, cudaStreamSynchronize(c->stream));
    c->dp_words = words;
    c->packed_feed_ready = true;
  }
  if ((int)c->next_slot == c->pending_slot) {  // the ring is full: the oldest submitted batch must be scanned before its slot is handed out again
    kmg_status st = scan_pending_batch(c);
    if (st != KMG_OK) return st;
  }
  Staging &s = c->st[c->next_slot];
  if (s.h2d_pending) { CU(c, cudaEventSynchronize(s.h2d_done)); s.h2d_pending = false; }  // the pinned words have left the host
  if (s.hp_used_words) {  // hand out zeroed words (producers OR their bits in): only what the previous user touched
    memset(s.hp_bases, 0, s.hp_used_words * 8); memset(s.hp_valid, 0, s.hp_used_words * 4); memset(s.hp_start, 0, s.hp_used_words * 4);
    s.hp_used_words = 0;
  }
  b->bases2bit = s.hp_bases; b->valid_bits = s.hp_valid; b->start_bits = s.hp_start;
  b->capacity_bases = c->batch_bases; b->n_bases = 0; b->n_records = 0; b->slot = c->next_slot;
  c->next_slot = (c->next_slot + 1) % N_STAGE;
  return KMG_OK;
}

KMG_EXPORT kmg_status kmg_submit_batch(kmg_ctx *c, const kmg_batch *b) {
  if (!c || !b) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  if (c->shm) return fail(c, KMG_ERR_STATE, "context belongs to a shard group: feed it with kmg_shard_count_ascii(_device)");
  if (b->slot >= (uint32_t)N_STAGE || !c->packed_feed_ready || b->bases2bit != c->st[b->slot].hp_bases)
    return fail(c, KMG_ERR_STATE, "batch was not obtained from kmg_acquire_batch");
  if (b->n_bases > b->capacity_bases) return fail(c, KMG_ERR_INVALID_ARG, "n_bases exceeds the batch capacity");
  if (b->n_bases == 0) return KMG_OK;
  CU(c, cudaSetDevice(c->device));
  Staging &s = c->st[b->slot];
  const uint64_t n_words = (b->n_bases + 31) / 32, n_words_total = round_up(n_words, TILE_WORDS);
  s.hp_used_words = n_words_total;
  // the copy goes out now, on the copy stream, as soon as the slot's device buffers are free (its previous scan has finished)
  if (s.compute_pending) { CU(c, cudaStreamWaitEvent(c->copy_stream, s.compute_done, 0)); s.compute_pending = false; }
  CU(c, cudaMemcpyAsync(s.dp_bases + LEAD_BASE_WORDS, s.hp_bases, n_words_total * 8, cudaMemcpyHostToDevice, c->copy_stream));
  CU(c, cudaMemcpyAsync(s.dp_valid + LEAD_MASK_WORDS, s.hp_valid, n_words_total * 4, cudaMemcpyHostToDevice, c->copy_stream));
  CU(c, cudaMemcpyAsync(s.dp_start + LEAD_MASK_WORDS, s.hp_start, n_words_total * 4, cudaMemcpyHostToDevice, c->copy_stream));
  CU(c, cudaEventRecord(s.h2d_done, c->copy_stream));
  s.h2d_pending = true;
  c->h2d_bytes += n_words_total * 16;
  c->n_records += b->n_records; c->n_bases += b->n_bases;
  // ... and while it travels, the batch submitted before this one is scanned
  kmg_status st = scan_pending_batch(c);
  c->pending_slot = (int)b->slot; c->pending_words = n_words_total;
  return st;
}

KMG_EXPORT kmg_status kmg_insert_keys_device(kmg_ctx *c, const uint64_t *d_keys, const uint64_t *d_counts, uint64_t n) {
  if (!c) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  if (c->shm) return fail(c, KMG_ERR_STATE, "context belongs to a shard group: feed it with kmg_shard_count_ascii(_device)");
  if (n == 0) return KMG_OK;
  if (!d_keys) return fail(c, KMG_ERR_INVALID_ARG, "d_keys is NULL");
  CU(c, cudaSetDevice(c->device));
  kmg_status ms = decide_mode(c, n);
  if (ms != KMG_OK) return ms;
  if (c->use_dense) { CU(c, launch_insert_keys_dense(c->dense, d_keys, d_counts, n, c->d_counters, c->stream)); return KMG_OK; }
  if (c->mode == kmg_ctx::MODE_PARTITIONED) return keys_to_run(c, d_keys, d_counts, n);
  uint64_t done = 0;
  while (done < n) {
    uint64_t granted = 0;
    kmg_status s = reserve_capacity(c, n - done, &granted);
    if (s != KMG_OK) return s;
    CU(c, launch_insert_keys(c->table, d_keys + done, d_counts ? d_counts + done : nullptr, granted, c->d_counters, c->stream));
    done += granted;
  }
  return KMG_OK;
}

KMG_EXPORT kmg_status kmg_partition_plan(kmg_ctx *c, uint64_t expected_keys, uint32_t *n_coarse, uint32_t *n_sub) {
  if (!c) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  CU(c, cudaSetDevice(c->device));
  if (c->mode == kmg_ctx::MODE_UNDECIDED) {
    if (c->use_dense) return fail(c, KMG_ERR_STATE, "context uses the direct-indexed path; create it with KMG_FLAG_FORCE_PARTITIONED");
    c->cfg.flags |= KMG_FLAG_FORCE_PARTITIONED;
    c->cfg.flags &= ~(uint32_t)KMG_FLAG_FORCE_HASH;
    kmg_status s = decide_mode(c, expected_keys);
    if (s != KMG_OK) return s;
  }
  if (c->mode != kmg_ctx::MODE_PARTITIONED) return fail(c, KMG_ERR_STATE, "context is not on the partitioned path");
  if (n_coarse) *n_coarse = c->n_coarse;
  if (n_sub) *n_sub = c->n_sub;
  return KMG_OK;
}

KMG_EXPORT kmg_status kmg_adopt_coarse_device(kmg_ctx *c, const uint64_t *d_keys, const uint64_t *bin_counts, uint32_t n_bins, uint64_t n) {
  if (!c || !bin_counts) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  if (c->shm) return fail(c, KMG_ERR_STATE, "context belongs to a shard group: feed it with kmg_shard_count_ascii(_device)");
  if (c->mode != kmg_ctx::MODE_PARTITIONED) return fail(c, KMG_ERR_STATE, "call kmg_partition_plan first");
  if (n_bins != c->n_coarse) return fail(c, KMG_ERR_INVALID_ARG, "n_bins must equal the context's coarse partition count");
  if (n > REFINE_MAX_ENTRIES) return fail(c, KMG_ERR_INVALID_ARG, "at most 2^32 - 2^22 keys per call");
  std::vector<uint64_t> off(n_bins + 1, 0);
  for (uint32_t b = 0; b < n_bins; ++b) off[b + 1] = off[b] + bin_counts[b];
  if (off[n_bins] != n) return fail(c, KMG_ERR_INVALID_ARG, "bin_counts do not add up to n");
  if (n == 0) return KMG_OK;
  if (!d_keys) return fail(c, KMG_ERR_INVALID_ARG, "d_keys is NULL");
  if (c->poisoned) return fail(c, KMG_ERR_STATE, "context is inconsistent after a failed re-split: kmg_reset it");
  if (c->feed_kind == 1) return fail(c, KMG_ERR_STATE, "context already holds runs binned by its own coarse function: adopted blocks (binned by owner and bin) cannot be mixed in");
  c->feed_kind = 2;
  CU(c, cudaSetDevice(c->device));
  const size_t tmr = timer_begin(c, 0);
  kmg_status s = refine_to_run(c, const_cast<uint64_t *>(d_keys), nullptr, off, /*owns=*/false, /*sync=*/true, nullptr, nullptr, /*in_keys=*/true);
  timer_end(c, tmr);
  return s;
}

KMG_EXPORT kmg_status kmg_extract_keys_device(kmg_ctx *c, const uint8_t *d_seq, const uint8_t *d_qual, const uint64_t *d_offsets,
                                              uint64_t n_records, uint64_t n_bytes, uint32_t n_shards, uint64_t *d_keys_out,
                                              uint64_t cap, uint64_t *shard_counts_out) {
  if (!c || !shard_counts_out) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  if (n_shards < 1 || n_shards > (uint32_t)MAX_PARTS) return fail(c, KMG_ERR_INVALID_ARG, "n_shards must be in 1..=8192");
  if (((uintptr_t)d_seq & 15) || ((uintptr_t)d_qual & 15)) return fail(c, KMG_ERR_INVALID_ARG, "d_seq / d_qual must be 16-byte aligned");
  CU(c, cudaSetDevice(c->device));
  for (uint32_t i = 0; i < n_shards; ++i) shard_counts_out[i] = 0;
  if (n_bytes == 0) return KMG_OK;
  uint64_t n_words_total = 0;
  bool has_start = false;
  kmg_status s = pack_device_ascii(c, d_seq, d_qual, n_records > 1 ? d_offsets : nullptr, n_records, 0, n_bytes, &n_words_total, &has_start);
  if (s != KMG_OK) return s;
  if (n_bytes >= (1ull << 32)) return fail(c, KMG_ERR_INVALID_ARG, "kmg_extract_keys_device handles < 2^32 bytes per call");
  unsigned long long *d_pc = nullptr;
  CU(c, pool_alloc(c, &d_pc, 3 * (size_t)n_shards * 8 + 64));  // pooled: a cudaMalloc / cudaFree pair per call synchronises the device
  unsigned long long *d_cur = d_pc + n_shards;
  unsigned long long *d_ps = d_cur + n_shards;
  unsigned long long *d_ctr = d_ps + n_shards;  // scratch counters (windows of this call only)
  CU(c, cudaMemsetAsync(d_pc, 0, 3 * (size_t)n_shards * 8 + 64, c->stream));
  ScanInput in{c->d_bases, c->d_valid, has_start ? c->d_start : nullptr, n_words_total / TILE_WORDS, c->k};
  cudaError_t e = launch_scan_partition(in, n_shards, false, d_pc, d_ps, d_cur, nullptr, d_ctr, c->stream);
  std::vector<unsigned long long> h(n_shards);
  if (e == cudaSuccess) e = cudaMemcpyAsync(h.data(), d_pc, n_shards * 8, cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  if (e != cudaSuccess) { pool_free(c, d_pc); return cuda_fail(c, e, "partition count pass"); }
  uint64_t total = 0;
  std::vector<unsigned long long> prefix(n_shards);
  for (uint32_t i = 0; i < n_shards; ++i) { prefix[i] = total; total += h[i]; shard_counts_out[i] = h[i]; }
  if (total > cap || (total && !d_keys_out)) { pool_free(c, d_pc); return fail(c, KMG_ERR_CAPACITY, "d_keys_out too small: need " + std::to_string(total)); }
  e = cudaMemcpyAsync(d_ps, prefix.data(), n_shards * 8, cudaMemcpyHostToDevice, c->stream);
  if (e == cudaSuccess) e = launch_scan_partition(in, n_shards, true, d_pc, d_ps, d_cur, d_keys_out, d_ctr, c->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  pool_free(c, d_pc);
  if (e != cudaSuccess) return cuda_fail(c, e, "partition scatter pass");
  c->n_records += n_records; c->n_bases += n_bytes;
  return KMG_OK;
}


// =================================================================================================
// Sharded (multi-GPU) counting: one context per GPU -- processes (torchrun, a Rust host with one process per device) or
// threads of one process -- joined into a group on ONE box.  The count table shards by hash: global coarse bin
// g = coarse_of_mix(mix, world * P1) belongs to rank g / P1.  Every rank scatters its keys into its own send buffer, one
// region per global bin; the exchange is FUSED into the owner's refine kernel (A2), whose tile loads read the owner's regions
// straight out of all ranks' send buffers through P2P-mapped pointers (NVLink loads, prefetched a tile ahead), so no key is
// ever copied: it crosses NVLink once, on its way into the kernel that partitions it further.  Only metadata crosses between
// the ranks on the host: a POSIX shared-memory segment carries a sense-reversing barrier and one double-buffered post area,
// through which every collective exchanges its messages (region sizes, flags, summaries, histograms) with one all-gather
// (shard_allgather).  The host ASCII feed and the file-image feed are the ones a single context uses (AsciiFeed, FastxFeed);
// only the scan of a chunk differs.  No NCCL, no staging copies, no count pass on the fast path.
// (Measured alternative, round 2: the scatter kernel writing into the owners' buffers with P2P STORES.  A sub-tile yields only
// ~8 keys per bin, and 64-byte NVLink writes cost more than they move: 4.45 ms per 310 M-base round against 2.05 ms for the
// local scatter; fewer bins made the stores longer but the owner's refine slower -- profiles/r2_summary.md.)
// =================================================================================================
constexpr uint32_t SHARD_MAX_WORLD = 8;
constexpr uint32_t SHARD_MAX_BINS = 2048;        // world * P1 (the single-scan rows kernel's limit)
constexpr uint32_t SHARD_HIST_MAX = 2 * 65536;   // (value, frequency) pairs a rank can post
constexpr uint32_t SHARD_MAGIC = 0x4b4d4753u;
constexpr double SHARD_TIMEOUT_S = 120.0;

constexpr uint32_t SHARD_POST_WORDS = 1 + 2 * SHARD_HIST_MAX;  // the largest message: a histogram's pair count and its pairs

struct PeerBuf {  // a rank's device buffer as its peers open it: raw pointer (threads of one process) or CUDA IPC handle
  cudaIpcMemHandle_t handle;
  uint64_t raw_ptr;
};
constexpr size_t PEER_BUF_WORDS = sizeof(PeerBuf) / 8;
static_assert(sizeof(PeerBuf) % 8 == 0, "a PeerBuf is posted as whole words");

struct ShardShm {
  uint32_t ready, world;
  uint32_t bar_count, bar_gen, abort, spec_disabled;
  uint64_t post[2][SHARD_MAX_WORLD][SHARD_POST_WORDS];  // [gather parity][rank]: the rank's message of a shard_allgather
};

namespace {

double now_s() { timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec; }

kmg_status shard_fail(kmg_ctx *c, kmg_status st, const std::string &msg) {
  if (c->shm) __atomic_store_n(&c->shm->abort, 1u, __ATOMIC_RELEASE);  // peers waiting in a barrier give up instead of hanging
  return fail(c, st, msg);
}

// sense-reversing barrier over the group's shared segment (processes or threads)
kmg_status shard_barrier(kmg_ctx *c) {
  ShardShm *S = c->shm;
  const uint32_t gen = __atomic_load_n(&S->bar_gen, __ATOMIC_ACQUIRE);
  if (__atomic_add_fetch(&S->bar_count, 1u, __ATOMIC_ACQ_REL) == S->world) {
    __atomic_store_n(&S->bar_count, 0u, __ATOMIC_RELAXED);
    __atomic_add_fetch(&S->bar_gen, 1u, __ATOMIC_RELEASE);
    return KMG_OK;
  }
  const double t0 = now_s();
  for (uint32_t spins = 0;; ++spins) {
    if (__atomic_load_n(&S->bar_gen, __ATOMIC_ACQUIRE) != gen) return KMG_OK;
    if (__atomic_load_n(&S->abort, __ATOMIC_ACQUIRE)) return fail(c, KMG_ERR_STATE, "a peer rank of the shard group failed");
    if (spins > 2000) {
      sched_yield();
      if ((spins & 1023) == 0 && now_s() - t0 > SHARD_TIMEOUT_S) return shard_fail(c, KMG_ERR_STATE, "shard group barrier timed out (a peer did not make the matching call)");
    }
  }
}
#define SB(c) do { kmg_status _s = shard_barrier(c); if (_s != KMG_OK) return _s; } while (0)
#define SCU(c, call) do { cudaError_t _e = (call); if (_e != cudaSuccess) { cuda_fail(c, _e, #call); return shard_fail(c, _e == cudaErrorMemoryAllocation ? KMG_ERR_OOM : KMG_ERR_CUDA, c->err); } } while (0)

// The one exchange of host metadata between the ranks: every rank posts n_words words, and all[r * n_words, (r + 1) * n_words) is
// rank r's message afterwards, on every rank.  counted_pairs: a variable-length message, word 0 the number m of pairs that follow as
// 2m words (n_words = 1 + 2m); every rank's row is copied with its own length, back to back.  Every rank makes the same sequence
// of calls.
// One barrier suffices because gathers alternate between the two halves of the post area: a rank writes the half of gather i
// again only in gather i+2, after it has passed the barrier of gather i+1, and no rank reaches that barrier before it has
// finished reading gather i.
kmg_status shard_allgather(kmg_ctx *c, const void *mine, size_t n_words, std::vector<uint64_t> &all, bool counted_pairs = false) {
  if (n_words > SHARD_POST_WORDS) return shard_fail(c, KMG_ERR_STATE, "shard group message larger than the post area");
  uint64_t (*post)[SHARD_POST_WORDS] = c->shm->post[c->sh_gathers & 1];
  memcpy(post[c->sh_rank], mine, n_words * 8);
  kmg_status st = shard_barrier(c);
  if (st != KMG_OK) return st;
  all.clear();
  for (uint32_t r = 0; r < c->sh_world; ++r) all.insert(all.end(), post[r], post[r] + (counted_pairs ? 1 + 2 * post[r][0] : n_words));
  c->sh_gathers++;
  return KMG_OK;
}

// A device buffer every rank can read: each rank posts its own, and after the gather opens all of them.
void publish_peer_buffer(PeerBuf &slot, void *mine) {
  slot.raw_ptr = (uint64_t)(uintptr_t)mine;
  cudaError_t e = cudaIpcGetMemHandle(&slot.handle, mine);
  if (e != cudaSuccess) { cudaGetLastError(); memset(&slot.handle, 0, sizeof slot.handle); }  // same-process groups do not need it
}
// peers[r] = rank r's buffer as seen from here, from the PeerBuf at the start of rank r's row of a gather: threads of one process use
// plain pointers (+ peer access between different devices), other processes a CUDA IPC mapping (ipc[r]).  Returns why a buffer
// could not be opened, or "".
std::string open_peer_buffers(kmg_ctx *c, const std::vector<uint64_t> &all, size_t row_words, uint64_t **peers, bool *ipc) {
  for (uint32_t r = 0; r < c->sh_world; ++r) {
    PeerBuf b;
    memcpy(&b, all.data() + r * row_words, sizeof b);
    const int dev = c->sh_device[r];
    if (r == c->sh_rank) {
      peers[r] = reinterpret_cast<uint64_t *>((uintptr_t)b.raw_ptr);
    } else if (c->sh_pid[r] == c->sh_pid[c->sh_rank]) {
      if (dev != c->device) {
        int can = 0;
        cudaDeviceCanAccessPeer(&can, c->device, dev);
        if (!can) return "no peer access between devices " + std::to_string(c->device) + " and " + std::to_string(dev);
        cudaError_t pe = cudaDeviceEnablePeerAccess(dev, 0);
        cudaGetLastError();
        if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) return std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(pe);
      }
      peers[r] = reinterpret_cast<uint64_t *>((uintptr_t)b.raw_ptr);
    } else {
      void *pp = nullptr;
      cudaError_t pe = cudaIpcOpenMemHandle(&pp, b.handle, cudaIpcMemLazyEnablePeerAccess);
      if (pe != cudaSuccess) { cudaGetLastError(); return std::string("cudaIpcOpenMemHandle(rank ") + std::to_string(r) + "): " + cudaGetErrorString(pe); }
      peers[r] = static_cast<uint64_t *>(pp); ipc[r] = true;
    }
  }
  return "";
}
void close_peer_buffers(uint64_t **peers, bool *ipc) {
  for (uint32_t r = 0; r < SHARD_MAX_WORLD; ++r) {
    if (peers[r] && ipc[r]) cudaIpcCloseMemHandle(peers[r]);
    peers[r] = nullptr; ipc[r] = false;
  }
}

void shard_release(kmg_ctx *c) {
  close_peer_buffers(c->sh_peer, c->sh_peer_ipc);
  if (c->sh_recv) { cudaFree(c->sh_recv); c->sh_recv = nullptr; }
  if (c->shm) { munmap(c->shm, sizeof(ShardShm)); c->shm = nullptr; }
  c->sh_world = 1; c->sh_rank = 0;
}

// One round of the sharded pipeline over the context's packed stream (n_words_total may be 0: a rank that has run out of
// input still takes part).  A1 scatters this rank's keys into ITS OWN send buffer, one region per global bin (owner-major);
// after the barrier every owner runs A2 straight over the regions that belong to it in ALL ranks' send buffers -- the tile
// loads of the refine kernel are P2P loads, i.e. the NVLink transfer happens inside A2, tile by tile, prefetched one tile ahead.
// Send buffers are double buffered: round i+1 scatters into the other half while slower owners may still be pulling round i.
kmg_status shard_scan_round(kmg_ctx *c, uint64_t n_words_total, bool has_start) {
  ShardShm *S = c->shm;
  const uint32_t W = c->sh_world, me = c->sh_rank, P1 = c->n_coarse, G = W * P1;
  unsigned long long *d_cnt = c->d_part, *d_start = c->d_part + MAX_PARTS, *d_cur = c->d_part + 2 * MAX_PARTS;
  static const bool trace = getenv("KMG_SHARD_TIMING") != nullptr;  // per-round wall times (every phase ends in a sync anyway)
  const double tr0 = now_s();
  // 1. the round's size is known to all (and everybody has finished the round before the previous one: see the buffers' reuse)
  std::vector<uint64_t> all;
  const uint64_t my_bytes = n_words_total * 32;
  kmg_status gs = shard_allgather(c, &my_bytes, 1, all);
  if (gs != KMG_OK) return gs;
  const uint64_t max_w = *std::max_element(all.begin(), all.end());
  if (max_w == 0) return KMG_OK;
  if (max_w >= (1ull << 32) || max_w > c->sh_recv_entries) return shard_fail(c, KMG_ERR_INVALID_ARG, "a sharded round handles at most batch_bases (< 2^32) bases per rank");
  const uint64_t parity = c->sh_rounds & 1;
  c->sh_rounds++;
  uint64_t *send = c->sh_recv + parity * c->sh_recv_entries;
  const uint64_t *src[SHARD_MAX_WORLD];
  for (uint32_t r = 0; r < W; ++r) src[r] = c->sh_peer[r] + parity * c->sh_recv_entries;
  ScanInput in;
  in.bases = c->d_bases; in.valid = c->d_valid; in.start = has_start ? c->d_start : nullptr;
  in.n_tiles = n_words_total / TILE_WORDS; in.k = c->k;
  // what this rank posts after its scatter: the overflow flag, then its G region lengths
  std::vector<uint64_t> h_start(G), post(1 + G);
  uint64_t *h_len = post.data() + 1;
  auto len_of = [&](uint32_t s, uint32_t g) { return all[(size_t)s * (G + 1) + 1 + g]; };  // source s's region of global bin g
  const size_t tmr = timer_begin(c, 0);
  bool done = false;
  double tr1 = tr0, tr2 = tr0;
  // 2. speculative layout: every global bin owns cap slots of the send buffer (cap from the largest rank's round, so that owners
  //    know where to read without being told); no count pass
  const double mu = (double)max_w / G;
  const uint64_t cap = ((uint64_t)(mu + 7.0 * std::sqrt(mu) + 64.0) + 15) & ~15ull;
  if (!__atomic_load_n(&S->spec_disabled, __ATOMIC_ACQUIRE) && cap * G <= c->sh_recv_entries && scan_scatter_supports_cap(G)) {
    for (uint32_t g = 0; g < G; ++g) h_start[g] = (uint64_t)g * cap;
    ScanInput sin = in;
    sin.part_cap = cap;
    sin.overflow_flag = reinterpret_cast<uint32_t *>(c->d_stats + 5);
    uint32_t h_flag = 0;
    SCU(c, cudaMemsetAsync(c->d_part, 0, 3 * (size_t)MAX_PARTS * sizeof(unsigned long long), c->stream));
    SCU(c, cudaMemsetAsync(sin.overflow_flag, 0, 4, c->stream));
    SCU(c, cudaMemcpyAsync(d_start, h_start.data(), G * 8, cudaMemcpyHostToDevice, c->stream));
    if (in.n_tiles) SCU(c, launch_scan_partition(sin, G, true, d_cnt, d_start, d_cur, send, c->d_counters, c->stream, /*mixed=*/true));
    SCU(c, cudaMemcpyAsync(h_len, d_cur, G * 8, cudaMemcpyDeviceToHost, c->stream));
    SCU(c, cudaMemcpyAsync(&h_flag, sin.overflow_flag, 4, cudaMemcpyDeviceToHost, c->stream));
    SCU(c, cudaStreamSynchronize(c->stream));
    tr1 = now_s();
    post[0] = h_flag;
    if ((gs = shard_allgather(c, post.data(), 1 + G, all)) != KMG_OK) return gs;  // every rank's regions are complete in its send buffer
    tr2 = now_s();
    bool any = false;
    for (uint32_t r = 0; r < W; ++r) any |= all[(size_t)r * (G + 1)] != 0;
    if (!any) {
      std::vector<uint64_t> off((size_t)P1 * W + 1), lens((size_t)P1 * W);
      uint64_t n_in = 0;
      for (uint32_t cl = 0; cl < P1; ++cl)
        for (uint32_t s2 = 0; s2 < W; ++s2) {
          const size_t j = (size_t)cl * W + s2;
          off[j] = (uint64_t)(me * P1 + cl) * cap; lens[j] = len_of(s2, me * P1 + cl); n_in += lens[j];
        }
      off[(size_t)P1 * W] = 0;  // unused: lengths are explicit
      for (uint32_t g = 0; g < G; ++g) if (g / P1 != me) c->sh_sent += h_len[g];
      c->sh_recv_keys += n_in;
      if (n_in) {
        kmg_status st = refine_to_run(c, nullptr, nullptr, off, /*owns=*/false, /*sync=*/true, &lens, nullptr, false, W, src);
        if (st != KMG_OK) return shard_fail(c, st, c->err);
      }
      done = true;
    } else {
      __atomic_store_n(&S->spec_disabled, 1u, __ATOMIC_RELEASE);  // sticky for the whole group: skewed input
    }
  }
  // 3. exact route (skewed input): count pass, exact prefix inside the own send buffer, scatter; owners derive every source's
  //    region offsets from the size matrix in the shared segment
  if (!done) {
    c->sh_exact_rounds++;
    SCU(c, cudaMemsetAsync(c->d_part, 0, 3 * (size_t)MAX_PARTS * sizeof(unsigned long long), c->stream));
    if (in.n_tiles) SCU(c, launch_scan_partition(in, G, false, d_cnt, d_start, d_cur, nullptr, c->d_counters, c->stream));
    SCU(c, cudaMemcpyAsync(h_len, d_cnt, G * 8, cudaMemcpyDeviceToHost, c->stream));
    SCU(c, cudaStreamSynchronize(c->stream));
    uint64_t run = 0;
    for (uint32_t g = 0; g < G; ++g) { h_start[g] = run; run += h_len[g]; }
    if (run > c->sh_recv_entries) return shard_fail(c, KMG_ERR_STATE, "send buffer smaller than a round (internal sizing error)");
    SCU(c, cudaMemcpyAsync(d_start, h_start.data(), G * 8, cudaMemcpyHostToDevice, c->stream));
    if (in.n_tiles) SCU(c, launch_scan_partition(in, G, true, d_cnt, d_start, d_cur, send, c->d_counters, c->stream, /*mixed=*/true));
    SCU(c, cudaStreamSynchronize(c->stream));
    tr1 = now_s();
    post[0] = 0;
    if ((gs = shard_allgather(c, post.data(), 1 + G, all)) != KMG_OK) return gs;
    tr2 = now_s();
    std::vector<uint64_t> off((size_t)P1 * W + 1), lens((size_t)P1 * W);
    uint64_t n_in = 0;
    for (uint32_t s2 = 0; s2 < W; ++s2) {
      uint64_t pre = 0;
      for (uint32_t g = 0; g < G; ++g) {
        if (g / P1 == me) { const size_t j = (size_t)(g - me * P1) * W + s2; off[j] = pre; lens[j] = len_of(s2, g); n_in += lens[j]; }
        pre += len_of(s2, g);
      }
    }
    off[(size_t)P1 * W] = 0;
    for (uint32_t g = 0; g < G; ++g) if (g / P1 != me) c->sh_sent += h_len[g];
    c->sh_recv_keys += n_in;
    if (n_in) {
      kmg_status st = refine_to_run(c, nullptr, nullptr, off, /*owns=*/false, /*sync=*/true, &lens, nullptr, false, W, src);
      if (st != KMG_OK) return shard_fail(c, st, c->err);
    }
  }
  timer_end(c, tmr);
  if (trace && me == 0)
    fprintf(stderr, "[shard round %llu] bases %llu  scatter %.2f ms  wait-for-peers %.2f ms  pull+refine %.2f ms  (G=%u, %s)\n",
            (unsigned long long)c->sh_rounds, (unsigned long long)(n_words_total * 32), (tr1 - tr0) * 1e3, (tr2 - tr1) * 1e3, (now_s() - tr2) * 1e3,
            G, done ? "speculative" : "exact");
  return KMG_OK;
}

}  // namespace

KMG_EXPORT kmg_status kmg_shard_join(kmg_ctx *c, uint32_t world, uint32_t rank, const char *group, uint64_t expected_keys_total) {
  if (!c || !group || !*group) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  if (world < 1 || world > SHARD_MAX_WORLD || rank >= world) return fail(c, KMG_ERR_INVALID_ARG, "world must be 1..=8 and rank < world");
  if (c->shm || c->sh_world > 1) return fail(c, KMG_ERR_STATE, "context already belongs to a shard group");
  if (c->mode != kmg_ctx::MODE_UNDECIDED) return fail(c, KMG_ERR_STATE, "kmg_shard_join must come before the first feeding call");
  if (world == 1) return KMG_OK;  // a group of one is the plain single-GPU path
  if (c->cfg.flags & (KMG_FLAG_FORCE_HASH | KMG_FLAG_FORCE_DIRECT)) return fail(c, KMG_ERR_INVALID_ARG, "the sharded path is the partitioned pipeline: FORCE_HASH / FORCE_DIRECT do not apply");
  CU(c, cudaSetDevice(c->device));
  // ---- partition plan: every rank derives the same one from the same arguments
  if (c->use_dense) { cudaFree(c->dense); c->dense = nullptr; c->dense_n = 0; c->use_dense = false; }
  c->cfg.flags |= KMG_FLAG_FORCE_PARTITIONED;
  c->mode = kmg_ctx::MODE_PARTITIONED;
  {
    const uint64_t per_rank = std::max<uint64_t>(expected_keys_total ? expected_keys_total : c->cfg.expected_distinct, 1) / world + 1;
    const uint64_t want = std::max<uint64_t>(4, (per_rank + TARGET_KEYS_PER_PART - 1) / TARGET_KEYS_PER_PART);
    uint64_t p1 = 1;
    while (p1 * p1 < want) ++p1;
    p1 = std::min<uint64_t>(p1, SHARD_MAX_BINS / world);  // world * P1 global bins in one scatter (the single-scan rows kernel's limit)
    c->n_coarse = (uint32_t)std::max<uint64_t>(p1, 1);
    c->n_sub = (uint32_t)std::min<uint64_t>((want + c->n_coarse - 1) / c->n_coarse, 2048);
    kmg_status st = init_partitioned(c);
    if (st != KMG_OK) return st;
  }
  // ---- send buffer (double buffered, one allocation so that one IPC handle covers both halves): a round scatters at most
  // batch_bases keys into it; the speculative layout needs mean + 7 sigma + 64 slots per global bin
  const uint64_t G = (uint64_t)world * c->n_coarse;
  const uint64_t round_max = round_up(c->batch_bases, (uint64_t)TILE_WORDS * 32);  // rounds are padded to whole tiles
  const double mu = (double)round_max / (double)G;
  c->sh_recv_entries = std::min<uint64_t>(round_max + G * (uint64_t)(7.0 * std::sqrt(mu) + 96.0), REFINE_MAX_ENTRIES);
  CU(c, cudaMalloc(&c->sh_recv, 2 * c->sh_recv_entries * 8));
  // ---- shared segment: rank 0 creates, the others attach
  const std::string name = std::string("/kmg-") + group;
  int fd = -1;
  const double t0 = now_s();
  if (rank == 0) {
    shm_unlink(name.c_str());
    fd = shm_open(name.c_str(), O_CREAT | O_EXCL | O_RDWR, 0600);
    if (fd < 0 || ftruncate(fd, (off_t)sizeof(ShardShm)) != 0) { if (fd >= 0) close(fd); shard_release(c); return fail(c, KMG_ERR_IO, "cannot create the shard group's shared segment " + name); }
  } else {
    while ((fd = shm_open(name.c_str(), O_RDWR, 0600)) < 0) {
      if (now_s() - t0 > SHARD_TIMEOUT_S) { shard_release(c); return fail(c, KMG_ERR_STATE, "shard group " + name + " did not appear (rank 0 missing?)"); }
      usleep(1000);
    }
    struct stat sb;
    while (fstat(fd, &sb) == 0 && (size_t)sb.st_size < sizeof(ShardShm)) {
      if (now_s() - t0 > SHARD_TIMEOUT_S) { close(fd); shard_release(c); return fail(c, KMG_ERR_STATE, "shard group segment was never sized"); }
      usleep(1000);
    }
  }
  void *mem = mmap(nullptr, sizeof(ShardShm), PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
  close(fd);
  if (mem == MAP_FAILED) { shard_release(c); return fail(c, KMG_ERR_IO, "cannot map the shard group's shared segment"); }
  c->shm = static_cast<ShardShm *>(mem);
  c->sh_world = world; c->sh_rank = rank;
  ShardShm *S = c->shm;
  if (rank == 0) {  // ftruncate zero-filled the segment
    S->world = world;
    __atomic_store_n(&S->ready, SHARD_MAGIC, __ATOMIC_RELEASE);
  } else {
    while (__atomic_load_n(&S->ready, __ATOMIC_ACQUIRE) != SHARD_MAGIC) {
      if (now_s() - t0 > SHARD_TIMEOUT_S) { shard_release(c); return fail(c, KMG_ERR_STATE, "shard group segment was never initialised"); }
      usleep(200);
    }
    if (S->world != world) { shard_release(c); return fail(c, KMG_ERR_INVALID_ARG, "ranks disagree on the world size"); }
  }
  // every rank's send buffer, process, device and plan
  constexpr size_t JW = PEER_BUF_WORDS + 6;
  uint64_t mine[JW];
  PeerBuf send;
  publish_peer_buffer(send, c->sh_recv);
  memcpy(mine, &send, sizeof send);
  uint64_t *m = mine + PEER_BUF_WORDS;
  m[0] = (uint64_t)getpid(); m[1] = (uint64_t)c->device; m[2] = c->n_coarse; m[3] = c->n_sub; m[4] = (uint64_t)c->k; m[5] = c->sh_recv_entries;
  c->sh_gathers = 0;
  std::vector<uint64_t> all;
  kmg_status st = shard_allgather(c, mine, JW, all);
  if (st != KMG_OK) { shard_release(c); return st; }
  std::string why;
  for (uint32_t r = 0; r < world; ++r) {
    const uint64_t *o = all.data() + r * JW + PEER_BUF_WORDS;
    c->sh_pid[r] = (int)o[0]; c->sh_device[r] = (int)o[1];
    if (o[2] != c->n_coarse || o[3] != c->n_sub || o[4] != (uint64_t)c->k || o[5] != c->sh_recv_entries)
      why = "ranks disagree on k / the partition plan / batch_bases (pass identical arguments on every rank)";
  }
  if (why.empty()) why = open_peer_buffers(c, all, JW, c->sh_peer, c->sh_peer_ipc);
  if (!why.empty()) __atomic_store_n(&S->abort, 1u, __ATOMIC_RELEASE);
  st = shard_barrier(c);  // every rank has opened its peers (or the group is aborted)
  if (rank == 0) shm_unlink(name.c_str());  // the mapping lives on; no name is left behind
  if (!why.empty() || st != KMG_OK) { shard_release(c); c->mode = kmg_ctx::MODE_PARTITIONED; return why.empty() ? st : fail(c, KMG_ERR_CUDA, why); }
  return KMG_OK;
}

KMG_EXPORT kmg_status kmg_shard_leave(kmg_ctx *c) {
  if (!c) return KMG_ERR_INVALID_ARG;
  if (!c->shm) return KMG_OK;
  CU(c, cudaSetDevice(c->device));
  cudaStreamSynchronize(c->stream);
  shard_barrier(c);  // nobody may still be writing into a buffer that is about to be unmapped / freed
  shard_release(c);
  return KMG_OK;
}

// Collective: every rank of the group calls it the same number of times (a rank without input passes n_bytes = 0).
// Input: THIS rank's slice of the records (device pointers), layout as kmg_count_ascii_device.
KMG_EXPORT kmg_status kmg_shard_count_ascii_device(kmg_ctx *c, const uint8_t *d_seq, const uint8_t *d_qual, const uint64_t *d_offsets,
                                                   uint64_t n_records, uint64_t n_bytes) {
  if (!c) return KMG_ERR_INVALID_ARG;
  if (!c->shm) return kmg_count_ascii_device(c, d_seq, d_qual, d_offsets, n_records, n_bytes);
  if (n_bytes && !d_seq) return shard_fail(c, KMG_ERR_INVALID_ARG, "d_seq is NULL");
  if (((uintptr_t)d_seq & 15) || ((uintptr_t)d_qual & 15)) return shard_fail(c, KMG_ERR_INVALID_ARG, "d_seq / d_qual must be 16-byte aligned");
  CU(c, cudaSetDevice(c->device));
  // rounds of at most batch_bases bases (k-1 overlap, records may span rounds); the ranks agree on the number of rounds
  // (round starts stay 16-byte aligned for the ingest kernel's vector loads: step is rounded down, a round covers step + k-1 bases)
  const uint64_t K1 = (uint64_t)c->k - 1, B = c->batch_bases, step = (B - K1) & ~15ull;
  if (step == 0) return shard_fail(c, KMG_ERR_INVALID_ARG, "batch_bases is too small for sharded rounds");
  uint64_t my_rounds = 0;
  for (uint64_t pos = 0; pos < n_bytes; pos += step) { if (pos && n_bytes - pos <= K1) break; ++my_rounds; }
  std::vector<uint64_t> all;
  kmg_status st = shard_allgather(c, &my_rounds, 1, all);
  if (st != KMG_OK) return st;
  const uint64_t rounds = *std::max_element(all.begin(), all.end());
  for (uint64_t i = 0; i < rounds; ++i) {
    const uint64_t pos = i * step;
    const uint64_t len = i < my_rounds ? std::min<uint64_t>(step + K1, n_bytes - pos) : 0;
    uint64_t n_words_total = 0;
    bool has_start = false;
    if (len) {
      st = pack_device_ascii(c, d_seq + pos, d_qual ? d_qual + pos : nullptr, n_records > 1 ? d_offsets : nullptr, n_records, pos, len,
                             &n_words_total, &has_start);
      if (st != KMG_OK) return shard_fail(c, st, c->err);
    }
    st = shard_scan_round(c, n_words_total, has_start);
    if (st != KMG_OK) return st;
  }
  c->n_records += n_records; c->n_bases += n_bytes;
  return KMG_OK;
}

// The same with HOST pointers (this rank's slice): staged through the context's pinned ring like kmg_count_ascii.
KMG_EXPORT kmg_status kmg_shard_count_ascii(kmg_ctx *c, const uint8_t *seq, const uint8_t *qual, const uint64_t *offsets, uint64_t n_records) {
  if (!c) return KMG_ERR_INVALID_ARG;
  if (!c->shm) return kmg_count_ascii(c, seq, qual, offsets, n_records);
  kmg_status s = check_ascii_layout(c, seq, offsets, n_records);
  if (s != KMG_OK) return shard_fail(c, s, c->err);
  CU(c, cudaSetDevice(c->device));
  // the ranks agree on the number of rounds; a rank without chunks left takes part with empty rounds
  AsciiFeed feed(c, seq, qual, offsets, n_records);
  if ((s = feed.open()) != KMG_OK) return shard_fail(c, s, c->err);
  const uint64_t my_rounds = feed.chunks.size();
  std::vector<uint64_t> all;
  if ((s = shard_allgather(c, &my_rounds, 1, all)) != KMG_OK) return s;
  const uint64_t rounds = *std::max_element(all.begin(), all.end());
  auto scan = [&](uint64_t n_words_total, bool has_start) { return shard_scan_round(c, n_words_total, has_start); };
  for (uint64_t i = 0; s == KMG_OK && i < rounds; ++i) s = i < my_rounds ? feed.step(i, scan) : scan(0, false);
  if (s != KMG_OK) return shard_fail(c, s, c->err);
  c->n_records += n_records; c->n_bases += feed.end - feed.begin;
  return feed.close();
}

namespace {

// Where a rank's slice of a file image begins, given t = len * r / W: the first line start at or after t (FASTA), or the first
// record start at or after t within FASTQ_SYNC_LINES lines (FASTQ).  len when the image ends first; false: no record start found.
bool fastx_rank_cut(const uint8_t *buf, uint64_t len, uint64_t t, bool is_fastq, uint64_t *cut) {
  auto next_line = [&](uint64_t p) -> uint64_t {
    const void *nl = memchr(buf + p, '\n', (size_t)(len - p));
    return nl ? (uint64_t)((const uint8_t *)nl - buf) + 1 : len;
  };
  uint64_t p = (t == 0 || t >= len || buf[t - 1] == '\n') ? std::min(t, len) : next_line(t);
  for (int tries = 0; tries < FASTQ_SYNC_LINES; ++tries) {
    if (!is_fastq || p >= len || fastq_record_start(buf, len, p)) { *cut = p; return true; }
    p = next_line(p);
  }
  return false;
}

// The carry of a FASTA slice that begins at the line start p inside a record: the last bases (at most k-1) of that record before
// p, collected backward line by line with the parser's trim_end (' ' and \t..\r), stopping at the record's header.  A carry that
// starts at the record's first base carries its record mark; *pending: the record's header is the last line before p that is not
// blank, so the record starts with the first base of the slice.
void fasta_carry_at(const uint8_t *buf, uint64_t p, uint64_t K1, std::vector<uint8_t> &seq, std::vector<uint8_t> &mark, bool *pending) {
  seq.clear();
  bool at_header = false;
  for (uint64_t le = p; le > 0 && seq.size() < K1;) {  // the line [ls, le), its '\n' at le - 1
    const void *nl = le >= 2 ? memrchr(buf, '\n', (size_t)(le - 1)) : nullptr;
    const uint64_t ls = nl ? (uint64_t)((const uint8_t *)nl - buf) + 1 : 0;
    if (buf[ls] == '>') { at_header = true; break; }
    uint64_t t = le;
    while (t > ls && (buf[t - 1] == ' ' || (buf[t - 1] >= 9 && buf[t - 1] <= 13))) --t;
    const uint64_t take = std::min<uint64_t>(t - ls, K1 - seq.size());
    seq.insert(seq.begin(), buf + t - take, buf + t);
    le = ls;
  }
  mark.assign(seq.size(), 0);
  if (at_header && !seq.empty()) mark[0] = 1;
  *pending = at_header && seq.empty();
}

}  // namespace

// One file image counted by the whole group: every rank passes the SAME image and parses only its own slice of it on the device,
// every parsed chunk is one fused scatter + exchange round.  Slices are cut at line (FASTA) / record (FASTQ) starts that every rank
// computes from the same bytes; a FASTA slice that begins inside a record gets that record's last k-1 bases in front of its first
// chunk (collected on the host), so every window is counted by exactly one rank: the one that holds its last base.
KMG_EXPORT kmg_status kmg_shard_count_fastx(kmg_ctx *c, const uint8_t *buf, uint64_t len, int is_fastq, uint64_t *n_records_out) {
  if (!c) return KMG_ERR_INVALID_ARG;
  if (!c->shm) return kmg_count_fastx(c, buf, len, is_fastq, n_records_out);
  if (n_records_out) *n_records_out = 0;
  if (len && !buf) return shard_fail(c, KMG_ERR_INVALID_ARG, "buf is NULL");
  if (len && buf[0] != (is_fastq ? '@' : '>'))
    return shard_fail(c, KMG_ERR_PARSE, is_fastq ? "FASTQ record does not start with '@' (record 0)" : "FASTA record does not start with '>' (record 0)");
  SCU(c, cudaSetDevice(c->device));
  const uint32_t W = c->sh_world, me = c->sh_rank;
  const uint64_t K1 = (uint64_t)c->k - 1;
  // ---- rank cuts (every rank computes all of them) and this rank's chunks: raw chunk + carry <= batch_bases bases, one round each
  uint64_t cuts[SHARD_MAX_WORLD + 1];
  cuts[0] = 0; cuts[W] = len;
  for (uint32_t r = 1; r < W; ++r)
    if (!fastx_rank_cut(buf, len, len / W * r + len % W * r / W, is_fastq, &cuts[r]))
      return shard_fail(c, KMG_ERR_PARSE, "no FASTQ record start found near a rank cut (multi-line FASTQ? use the host splitter)");
  const uint64_t begin = cuts[me], end = cuts[me + 1];
  std::vector<FxChunk> chunks;
  const kmg_status plan = plan_fastx_chunks(c, buf, len, begin, end, is_fastq, std::min<uint64_t>(c->batch_bases - K1, 1ull << 30), chunks);
  // ---- the ranks compare their images (length and cuts) and plans, and agree on the number of rounds
  const size_t FW = W + 4;  // image length, plan status, rounds, cuts
  uint64_t mine[SHARD_MAX_WORLD + 4] = {len, (uint64_t)plan, plan == KMG_OK ? chunks.size() : 0};
  memcpy(mine + 3, cuts, (W + 1) * 8);
  std::vector<uint64_t> all;
  kmg_status s = shard_allgather(c, mine, FW, all);
  if (s != KMG_OK) return s;
  bool same = true, planned = true;
  uint64_t rounds = 0;
  for (uint32_t r = 0; r < W; ++r) {
    const uint64_t *o = all.data() + r * FW;
    same = same && o[0] == len && memcmp(o + 3, cuts, (W + 1) * 8) == 0;
    planned = planned && o[1] == (uint64_t)KMG_OK;
    rounds = std::max<uint64_t>(rounds, o[2]);
  }
  if (!same) return shard_fail(c, KMG_ERR_INVALID_ARG, "ranks passed different file images (pass the same whole image on every rank)");
  if (!planned)
    return shard_fail(c, KMG_ERR_PARSE, plan != KMG_OK ? c->err : "another rank's slice cannot be cut into staging chunks (a line longer than a chunk, or multi-line FASTQ)");
  // ---- rounds: parse -> pack -> fused scatter + exchange; a rank without chunks left takes part with empty rounds
  FastxFeed feed(c, is_fastq, buf, &chunks);
  if (!chunks.empty()) {
    s = feed.open();
    if (s == KMG_OK && !is_fastq && buf[begin] != '>') {
      std::vector<uint8_t> cseq, cmark;
      bool pending = false;
      fasta_carry_at(buf, begin, K1, cseq, cmark, &pending);
      s = feed.seed_carry(cseq.data(), cmark.data(), cseq.size(), pending);
    }
  }
  for (uint64_t i = 0; s == KMG_OK && i < rounds; ++i) {
    bool scanned = false;
    if (i < chunks.size()) s = feed.step(i, [&](uint64_t n_words_total) { return shard_scan_round(c, n_words_total, true); }, &scanned);
    if (s == KMG_OK && !scanned) s = shard_scan_round(c, 0, false);
  }
  uint64_t n_rec = 0;
  if (s == KMG_OK && !chunks.empty()) s = feed.records(&n_rec);
  if (!chunks.empty()) feed.close(s != KMG_OK);
  if (s != KMG_OK) return shard_fail(c, s, c->err);
  // ---- records of the whole image, on every rank
  if ((s = shard_allgather(c, &n_rec, 1, all)) != KMG_OK) return s;
  uint64_t total = 0;
  for (uint64_t n : all) total += n;
  c->n_records += n_rec; c->n_bases += feed.bases;
  if (n_records_out) *n_records_out = total;
  return KMG_OK;
}

KMG_EXPORT kmg_status kmg_finalize(kmg_ctx *c, kmg_summary *out) {
  if (!c) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  CU(c, cudaSetDevice(c->device));
  { kmg_status _fs = scan_pending_batch(c); if (_fs != KMG_OK) return _fs; }
  CU(c, cudaStreamSynchronize(c->copy_stream));
  kmg_status s = read_counters(c);
  if (s != KMG_OK) return s;
  for (auto &st : c->st) { st.h2d_pending = false; st.compute_pending = false; }
  if (c->mode == kmg_ctx::MODE_PARTITIONED && (s = consolidate(c)) != KMG_OK) return s;
  timers_collect(c);
  if (c->mode == kmg_ctx::MODE_TABLE) c->distinct_ub = c->h_counters[CTR_DISTINCT];
  if (!out) return KMG_OK;
  memset(out, 0, sizeof *out);
  unsigned long long h[3];
  if (fetch_fused_hist(c)) { h[0] = c->result.n_valid; h[1] = c->fused_max; h[2] = c->fused_sum; }
  else {
    CU(c, launch_table_stats(view_of(c), 1, c->d_stats, c->stream));
    CU(c, cudaMemcpyAsync(h, c->d_stats, sizeof h, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
  }
  out->n_records = c->n_records; out->n_bases = c->n_bases;
  out->n_windows = h[2];
  out->n_distinct = h[0]; out->max_count = h[1];
  out->table_capacity = c->use_dense ? c->dense_n : c->mode == kmg_ctx::MODE_PARTITIONED ? c->n_parts : c->table.cap;
  out->path = c->use_dense ? 1 : c->mode == kmg_ctx::MODE_PARTITIONED ? 2 : 0;
  out->n_grows = c->mode == kmg_ctx::MODE_PARTITIONED ? c->n_consolidations : c->n_grows;
  out->kernel_ns = (uint64_t)(c->kernel_ms * 1e6);
  out->scan_ns = (uint64_t)(c->cat_ms[0] * 1e6);
  out->consolidate_ns = (uint64_t)(c->cat_ms[1] * 1e6);
  out->h2d_bytes = c->h2d_bytes;
  return KMG_OK;
}

namespace {
kmg_status count_filtered(kmg_ctx *c, uint64_t min_count, uint64_t *n, uint64_t shard_mod = 0, uint64_t shard_rem = 0) {
  { kmg_status _fs = scan_pending_batch(c); if (_fs != KMG_OK) return _fs; }
  CU(c, cudaStreamSynchronize(c->copy_stream));
  if (c->mode == kmg_ctx::MODE_PARTITIONED) { kmg_status s = consolidate(c); if (s != KMG_OK) return s; }
  if (shard_mod <= 1 && fetch_fused_hist(c)) {
    uint64_t m = 0;
    for (uint64_t b = std::max<uint64_t>(min_count, 1); b < (uint64_t)HIST_DENSE_BINS; ++b) m += c->h_bins[b];
    m += c->h_ov.end() - std::lower_bound(c->h_ov.begin(), c->h_ov.end(), min_count);
    *n = m;
    return KMG_OK;
  }
  TableView v = view_of(c);
  v.shard_mod = shard_mod; v.shard_rem = shard_rem;
  CU(c, launch_table_stats(v, min_count, c->d_stats, c->stream));
  unsigned long long h[3];
  CU(c, cudaMemcpyAsync(h, c->d_stats, sizeof h, cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  *n = h[0];
  return KMG_OK;
}

kmg_status export_device(kmg_ctx *c, uint64_t min_count, int sorted, uint64_t shard_mod, uint64_t shard_rem, uint64_t *d_keys,
                         uint64_t *d_counts, uint64_t cap, uint64_t *n_out) {
  if (!c || !n_out) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  if (shard_mod > 1 && shard_rem >= shard_mod) return fail(c, KMG_ERR_INVALID_ARG, "shard must be < n_shards");
  CU(c, cudaSetDevice(c->device));
  uint64_t n = 0;
  kmg_status s = count_filtered(c, min_count, &n, shard_mod, shard_rem);
  if (s != KMG_OK) return s;
  *n_out = n;
  if (!d_keys || !d_counts) return KMG_OK;
  if (cap < n) return fail(c, KMG_ERR_CAPACITY, "output arrays hold " + std::to_string(cap) + " entries, need " + std::to_string(n));
  TableView v = view_of(c);
  v.shard_mod = shard_mod; v.shard_rem = shard_rem;
  CU(c, launch_compact(v, min_count, d_keys, d_counts, cap, c->d_stats + 3, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  if (sorted) CU(c, sort_pairs(d_keys, d_counts, n, 2 * c->k, c->stream));
  return KMG_OK;
}

kmg_status export_host(kmg_ctx *c, uint64_t min_count, int sorted, uint64_t shard_mod, uint64_t shard_rem, uint64_t *keys,
                       uint64_t *counts, uint64_t cap, uint64_t *n_out) {
  if (!c || !n_out) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  if (shard_mod > 1 && shard_rem >= shard_mod) return fail(c, KMG_ERR_INVALID_ARG, "shard must be < n_shards");
  CU(c, cudaSetDevice(c->device));
  uint64_t n = 0;
  kmg_status s = count_filtered(c, min_count, &n, shard_mod, shard_rem);
  if (s != KMG_OK) return s;
  *n_out = n;
  if (!keys || !counts) return KMG_OK;
  if (cap < n) return fail(c, KMG_ERR_CAPACITY, "output arrays hold " + std::to_string(cap) + " entries, need " + std::to_string(n));
  if (n == 0) return KMG_OK;
  uint64_t *dk = nullptr, *dc = nullptr;
  CU(c, pool_alloc(c, &dk, n * 8));
  cudaError_t e = pool_alloc(c, &dc, n * 8);
  if (e != cudaSuccess) { pool_free(c, dk); return cuda_fail(c, e, "cudaMalloc(export)"); }
  uint64_t n2 = 0;
  s = export_device(c, min_count, sorted, shard_mod, shard_rem, dk, dc, n, &n2);
  if (s == KMG_OK) {
    e = cudaMemcpyAsync(keys, dk, n * 8, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(counts, dc, n * 8, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) s = cuda_fail(c, e, "D2H export");
  }
  pool_free(c, dk); pool_free(c, dc);
  return s;
}
}  // namespace

KMG_EXPORT kmg_status kmg_export_counts_device(kmg_ctx *c, uint64_t min_count, int sorted, uint64_t *d_keys, uint64_t *d_counts,
                                               uint64_t cap, uint64_t *n_out) {
  return export_device(c, min_count, sorted, 0, 0, d_keys, d_counts, cap, n_out);
}

KMG_EXPORT kmg_status kmg_export_counts(kmg_ctx *c, uint64_t min_count, int sorted, uint64_t *keys, uint64_t *counts, uint64_t cap,
                                        uint64_t *n_out) {
  return export_host(c, min_count, sorted, 0, 0, keys, counts, cap, n_out);
}

KMG_EXPORT kmg_status kmg_export_shard(kmg_ctx *c, uint64_t min_count, int sorted, uint64_t n_shards, uint64_t shard, uint64_t *keys,
                                       uint64_t *counts, uint64_t cap, uint64_t *n_out) {
  return export_host(c, min_count, sorted, n_shards, shard, keys, counts, cap, n_out);
}

KMG_EXPORT kmg_status kmg_export_shard_device(kmg_ctx *c, uint64_t min_count, int sorted, uint64_t n_shards, uint64_t shard,
                                              uint64_t *d_keys, uint64_t *d_counts, uint64_t cap, uint64_t *n_out) {
  return export_device(c, min_count, sorted, n_shards, shard, d_keys, d_counts, cap, n_out);
}

KMG_EXPORT kmg_status kmg_histogram(kmg_ctx *c, uint64_t min_count, uint64_t *count_vals, uint64_t *freqs, uint64_t cap, uint64_t *n_out) {
  if (!c || !n_out) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  CU(c, cudaSetDevice(c->device));
  { kmg_status _fs = scan_pending_batch(c); if (_fs != KMG_OK) return _fs; }
  CU(c, cudaStreamSynchronize(c->copy_stream));
  kmg_status s = read_counters(c);
  if (s != KMG_OK) return s;
  if (c->mode == kmg_ctx::MODE_PARTITIONED && (s = consolidate(c)) != KMG_OK) return s;
  if (fetch_fused_hist(c)) {  // phase B already built it
    const uint64_t lo = std::max<uint64_t>(min_count, 1);
    const auto ov0 = std::lower_bound(c->h_ov.begin(), c->h_ov.end(), min_count);
    uint64_t n = 0;
    for (uint64_t b = lo; b < (uint64_t)HIST_DENSE_BINS; ++b) if (c->h_bins[b]) ++n;
    for (auto it = ov0; it != c->h_ov.end(); ++it) if (it == ov0 || *it != *(it - 1)) ++n;
    *n_out = n;
    if (!count_vals || !freqs) return KMG_OK;
    if (cap < n) return fail(c, KMG_ERR_CAPACITY, "histogram arrays hold " + std::to_string(cap) + " bins, need " + std::to_string(n));
    uint64_t o = 0;
    for (uint64_t b = lo; b < (uint64_t)HIST_DENSE_BINS; ++b) if (c->h_bins[b]) { count_vals[o] = b; freqs[o] = c->h_bins[b]; ++o; }
    for (auto it = ov0; it != c->h_ov.end();) {
      auto j = it;
      while (j != c->h_ov.end() && *j == *it) ++j;
      count_vals[o] = *it; freqs[o] = (uint64_t)(j - it); ++o;
      it = j;
    }
    return KMG_OK;
  }
  // counts >= HIST_DENSE_BINS: at most (sum of counts) / HIST_DENSE_BINS distinct keys can reach that
  CU(c, launch_table_stats(view_of(c), 1, c->d_stats, c->stream));
  unsigned long long hs[3];
  CU(c, cudaMemcpyAsync(hs, c->d_stats, sizeof hs, cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  const uint64_t ov_cap = hs[2] / HIST_DENSE_BINS + 16;
  unsigned long long *d_bins = nullptr;
  uint64_t *d_ov = nullptr;
  CU(c, pool_alloc(c, &d_bins, HIST_DENSE_BINS * 8));
  cudaError_t e = pool_alloc(c, &d_ov, ov_cap * 8);
  if (e != cudaSuccess) { pool_free(c, d_bins); return cuda_fail(c, e, "cudaMalloc(histogram overflow)"); }
  std::vector<unsigned long long> bins(HIST_DENSE_BINS);
  std::vector<uint64_t> ov;
  unsigned long long ov_n = 0;
  e = launch_histogram(view_of(c), min_count, d_bins, d_ov, ov_cap, c->d_stats + 4, c->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(bins.data(), d_bins, HIST_DENSE_BINS * 8, cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(&ov_n, c->d_stats + 4, 8, cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  if (e == cudaSuccess && ov_n > ov_cap) { pool_free(c, d_bins); pool_free(c, d_ov); return fail(c, KMG_ERR_STATE, "histogram overflow list exceeded its bound"); }
  if (e == cudaSuccess && ov_n) { ov.resize(ov_n); e = cudaMemcpy(ov.data(), d_ov, ov_n * 8, cudaMemcpyDeviceToHost); }
  pool_free(c, d_bins); pool_free(c, d_ov);
  if (e != cudaSuccess) return cuda_fail(c, e, "histogram");
  // assemble ascending (count, frequency) pairs: dense bins first, then the (tiny) overflow tail
  std::sort(ov.begin(), ov.end());
  uint64_t n = 0;
  for (uint64_t b = 0; b < HIST_DENSE_BINS; ++b) if (bins[b]) ++n;
  for (size_t i = 0; i < ov.size(); ++i) if (i == 0 || ov[i] != ov[i - 1]) ++n;
  *n_out = n;
  if (!count_vals || !freqs) return KMG_OK;
  if (cap < n) return fail(c, KMG_ERR_CAPACITY, "histogram arrays hold " + std::to_string(cap) + " bins, need " + std::to_string(n));
  uint64_t o = 0;
  for (uint64_t b = 0; b < HIST_DENSE_BINS; ++b) if (bins[b]) { count_vals[o] = b; freqs[o] = bins[b]; ++o; }
  for (size_t i = 0; i < ov.size();) {
    size_t j = i;
    while (j < ov.size() && ov[j] == ov[i]) ++j;
    count_vals[o] = ov[i]; freqs[o] = j - i; ++o;
    i = j;
  }
  return KMG_OK;
}

namespace {
// CRC-32 of a concatenation from the parts' CRCs (zlib's crc32_combine idea: advance crc1 over len2 zero bytes with
// GF(2) matrix squaring, then xor crc2) -- lets every GPU shard checksum its own records (src/index.rs:434-456 streams one CRC).
uint32_t gf2_times(const uint32_t *mat, uint32_t vec) {
  uint32_t sum = 0;
  for (; vec; vec >>= 1, ++mat) if (vec & 1) sum ^= *mat;
  return sum;
}
void gf2_square(uint32_t *sq, const uint32_t *mat) { for (int n = 0; n < 32; ++n) sq[n] = gf2_times(mat, mat[n]); }
uint32_t crc32_combine(uint32_t crc1, uint32_t crc2, uint64_t len2) {
  if (len2 == 0) return crc1;
  uint32_t even[32], odd[32];
  odd[0] = 0xEDB88320u;  // operator for one zero bit
  for (uint32_t n = 1, row = 1; n < 32; ++n, row <<= 1) odd[n] = row;
  gf2_square(even, odd);  // two zero bits
  gf2_square(odd, even);  // four zero bits
  do {
    gf2_square(even, odd);
    if (len2 & 1) crc1 = gf2_times(even, crc1);
    len2 >>= 1;
    if (!len2) break;
    gf2_square(odd, even);
    if (len2 & 1) crc1 = gf2_times(odd, crc1);
    len2 >>= 1;
  } while (len2);
  return crc1 ^ crc2;
}

// CRC-32 of a large buffer on all host cores: the parts' CRCs are combined (a single core manages ~2 GB/s, an index is tens of GB)
uint32_t crc32_parallel(const uint8_t *p, size_t n) {
  const Crc32 &T = crc_tables();
  unsigned nt = std::min<unsigned>(std::max(1u, std::thread::hardware_concurrency()), 16u);
  if (n < (8u << 20) || nt == 1) return ~T.update(~0u, p, n);
  const size_t per = (n + nt - 1) / nt;
  std::vector<uint32_t> part(nt, 0);
  std::vector<size_t> len(nt, 0);
  std::vector<std::thread> th;
  for (unsigned t = 0; t < nt; ++t) {
    const size_t lo = std::min(n, t * per), hi = std::min(n, lo + per);
    len[t] = hi - lo;
    th.emplace_back([&, t, lo, hi] { part[t] = ~T.update(~0u, p + lo, hi - lo); });
  }
  for (auto &x : th) x.join();
  uint32_t crc = part[0];
  for (unsigned t = 1; t < nt; ++t) crc = crc32_combine(crc, part[t], len[t]);
  return crc;
}

// The sorted walkers below cut the key space on the boundaries of KEY_BUCKETS buckets over the top bits of the 2k-bit keys.
int key_bucket_shift(const kmg_ctx *c) { return 2 * c->k > 12 ? 2 * c->k - 12 : 0; }

// hb[b] = entries of the table (any count) in key bucket b
kmg_status key_histogram(kmg_ctx *c, uint64_t *hb) {
  unsigned long long *d_b = nullptr;
  CU(c, pool_alloc(c, &d_b, KEY_BUCKETS * 8));
  cudaError_t e = launch_key_buckets(view_of(c), key_bucket_shift(c), d_b, c->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(hb, d_b, KEY_BUCKETS * 8, cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  pool_free(c, d_b);
  if (e != cudaSuccess) return cuda_fail(c, e, "key histogram");
  return KMG_OK;
}

// Cuts of the bucket range into pieces of at most max(~piece_target, largest bucket) entries: piece i is buckets [cuts[i], cuts[i+1]).
// Empty buckets at the end belong to no piece; an empty histogram gives no piece.
std::vector<int> piece_cuts(const uint64_t *hb, uint64_t piece_target) {
  uint64_t n_all = 0, piece_cap = 0;
  for (int b = 0; b < KEY_BUCKETS; ++b) { n_all += hb[b]; piece_cap = std::max<uint64_t>(piece_cap, hb[b]); }
  piece_cap = std::max<uint64_t>(piece_cap, std::min<uint64_t>(n_all, piece_target));
  std::vector<int> cuts{0};
  for (int b0 = 0; b0 < KEY_BUCKETS;) {
    uint64_t ub = hb[b0];
    int b1 = b0 + 1;
    while (b1 < KEY_BUCKETS && ub + hb[b1] <= piece_cap) ub += hb[b1++];
    if (ub) cuts.push_back(b1);
    b0 = b1;
  }
  return cuts;
}

// Entries of the largest piece of `cuts` (its sorted part fits a buffer of that size)
uint64_t largest_piece(const uint64_t *hb, const std::vector<int> &cuts) {
  uint64_t m = 0;
  for (size_t i = 0; i + 1 < cuts.size(); ++i) {
    uint64_t n = 0;
    for (int b = cuts[i]; b < cuts[i + 1]; ++b) n += hb[b];
    m = std::max(m, n);
  }
  return m;
}

// Walk the table in ascending key order WITHOUT a second copy of it: each piece of `cuts` is compacted (count >= min_count) into
// dk / dc (room for cap entries), sorted, and handed to fn(dk, dc, m), empty pieces too.  The pieces concatenate to the sorted result.
template <class F>
kmg_status for_each_sorted_piece(kmg_ctx *c, uint64_t min_count, const std::vector<int> &cuts, uint64_t *dk, uint64_t *dc, uint64_t cap,
                                 F &&fn) {
  const int shift = key_bucket_shift(c);
  kmg_status s = KMG_OK;
  for (size_t i = 0; s == KMG_OK && i + 1 < cuts.size(); ++i) {
    TableView v = view_of(c);
    v.range_lo = (uint64_t)cuts[i] << shift;
    v.range_hi = cuts[i + 1] == KEY_BUCKETS ? ~0ull : ((uint64_t)cuts[i + 1] << shift) - 1;
    unsigned long long m = 0;
    cudaError_t e = launch_compact(v, min_count, dk, dc, cap, c->d_stats + 3, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&m, c->d_stats + 3, 8, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e == cudaSuccess && m > cap) return fail(c, KMG_ERR_STATE, "sorted piece larger than its key histogram");
    if (e == cudaSuccess && m) e = sort_pairs(dk, dc, m, 2 * c->k, c->stream);
    if (e != cudaSuccess) return cuda_fail(c, e, "sorted piece");
    s = fn(dk, dc, (uint64_t)m);
  }
  return s;
}

// The whole table of one context, in pieces of about piece_target entries.
template <class F>
kmg_status for_each_sorted_piece(kmg_ctx *c, uint64_t min_count, uint64_t piece_target, F &&fn) {
  uint64_t n_all = 0;
  kmg_status s = count_filtered(c, 0, &n_all);
  if (s != KMG_OK || n_all == 0) return s;
  std::vector<uint64_t> hb(KEY_BUCKETS);
  if ((s = key_histogram(c, hb.data())) != KMG_OK) return s;
  const std::vector<int> cuts = piece_cuts(hb.data(), piece_target);
  const uint64_t cap = largest_piece(hb.data(), cuts);
  uint64_t *dk = nullptr, *dc = nullptr;
  CU(c, pool_alloc(c, &dk, cap * 8));
  cudaError_t e = pool_alloc(c, &dc, cap * 8);
  if (e != cudaSuccess) { pool_free(c, dk); return cuda_fail(c, e, "cudaMalloc(sorted piece)"); }
  s = for_each_sorted_piece(c, min_count, cuts, dk, dc, cap, [&](const uint64_t *k, const uint64_t *n, uint64_t m) -> kmg_status {
    return m ? fn(k, n, m) : KMG_OK;
  });
  pool_free(c, dk); pool_free(c, dc);
  return s;
}

// Device bytes -> sink through two pinned staging buffers (the copy of chunk i+1 overlaps the sink of chunk i).
struct HostStager {
  kmg_ctx *c;
  uint8_t *h[2] = {nullptr, nullptr};
  size_t cap = 0;
  explicit HostStager(kmg_ctx *c_, size_t cap_) : c(c_), cap(cap_) {}
  ~HostStager() { for (auto *p : h) if (p) cudaFreeHost(p); }
  template <class Sink>
  kmg_status drain(const uint8_t *d_src, size_t n, Sink &&sink) {
    for (int i = 0; i < 2; ++i)
      if (!h[i] && cudaHostAlloc(&h[i], cap, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return fail(c, KMG_ERR_OOM, "pinned staging buffer"); }
    size_t issued = 0;
    int slot = 0;
    size_t len_prev = 0;
    if (n) { len_prev = std::min(cap, n); CU(c, cudaMemcpyAsync(h[0], d_src, len_prev, cudaMemcpyDeviceToHost, c->stream)); issued = len_prev; }
    while (len_prev) {
      CU(c, cudaStreamSynchronize(c->stream));
      const size_t len_next = std::min(cap, n - issued);
      if (len_next) { CU(c, cudaMemcpyAsync(h[slot ^ 1], d_src + issued, len_next, cudaMemcpyDeviceToHost, c->stream)); issued += len_next; }
      kmg_status s = sink(h[slot], len_prev);
      if (s != KMG_OK) { cudaStreamSynchronize(c->stream); return s; }
      slot ^= 1; len_prev = len_next;
    }
    return KMG_OK;
  }
};

// A sorted (key, count) piece -> its fasta / tsv / json text in d_text, formatted on the device (record lengths, their exclusive
// sum = record offsets, then every record written at its offset).  The buffers grow as pieces need and are reused across pieces.
// first: record 0 of the piece is the first record of the whole output.
struct TextFormatter {
  kmg_ctx *c;
  int text_format;
  uint64_t *d_off = nullptr;
  uint8_t *d_text = nullptr;
  uint64_t off_cap = 0, text_cap = 0;
  TextFormatter(kmg_ctx *c_, int text_format_) : c(c_), text_format(text_format_) {}
  ~TextFormatter() { pool_free(c, d_off); pool_free(c, d_text); }
  kmg_status format(const uint64_t *dk, const uint64_t *dc, uint64_t m, bool first, uint64_t *bytes_out) {
    if (m + 1 > off_cap) { pool_free(c, d_off); d_off = nullptr; off_cap = std::max<uint64_t>(m + 1, 1ull << 20); CU(c, pool_alloc(c, &d_off, off_cap * 8)); }
    CU(c, launch_text_len(dc, m, c->k, text_format, first, d_off, c->stream));
    CU(c, cudaMemsetAsync(d_off + m, 0, 8, c->stream));
    if (!c->d_scan_tmp || c->scan_tmp_items < m + 1) {
      CU(c, cudaStreamSynchronize(c->stream));
      cudaFree(c->d_scan_tmp); c->d_scan_tmp = nullptr;
      CU(c, exclusive_sum_u64(nullptr, nullptr, m + 1, nullptr, &c->scan_tmp_bytes, c->stream));
      CU(c, cudaMalloc(&c->d_scan_tmp, c->scan_tmp_bytes ? c->scan_tmp_bytes : 16));
      c->scan_tmp_items = m + 1;
    }
    CU(c, exclusive_sum_u64(d_off, d_off, m + 1, c->d_scan_tmp, &c->scan_tmp_bytes, c->stream));  // entry m = bytes of the piece
    uint64_t total = 0;
    CU(c, cudaMemcpyAsync(&total, d_off + m, 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (total > text_cap) { pool_free(c, d_text); d_text = nullptr; text_cap = total + total / 8; CU(c, pool_alloc(c, &d_text, text_cap)); }
    CU(c, launch_text_write(dk, dc, d_off, m, c->k, text_format, first, d_text, c->stream));
    *bytes_out = total;
    return KMG_OK;
  }
};
// json framing around the records: "[" in front of them, then "\n]\n" after them, or "]\n" when there is none ("[]\n")
constexpr char JSON_OPEN[] = "[";
const char *json_close(uint64_t records) { return records ? "\n]\n" : "]\n"; }

// Stream all (key, count) records of the context to `f` in ascending key order (16-byte records interleaved on the device).
// *crc_out is the finished CRC-32 of the bytes written here (standard init / xor-out).
kmg_status write_kmix_records(kmg_ctx *c, FILE *f, uint32_t *crc_out, uint64_t *n_out) {
  uint64_t n = 0;
  kmg_status s = count_filtered(c, 0, &n);
  if (s != KMG_OK) return s;
  *n_out = n;
  uint32_t crc = 0;  // CRC of the empty string
  uint64_t written = 0;
  bool first = true;
  HostStager stage(c, 64u << 20);
  void *d_pairs = nullptr;
  uint64_t pairs_cap = 0;
  s = for_each_sorted_piece(c, 0, 1ull << 25, [&](const uint64_t *dk, const uint64_t *dc, uint64_t m) -> kmg_status {
    if (m > pairs_cap) {
      pool_free(c, d_pairs); d_pairs = nullptr;
      pairs_cap = std::max<uint64_t>(m, std::min<uint64_t>(n, 1ull << 25));
      CU(c, pool_alloc(c, &d_pairs, pairs_cap * 16));
    }
    CU(c, launch_interleave_pairs(dk, dc, m, d_pairs, c->stream));
    written += m;
    return stage.drain(static_cast<const uint8_t *>(d_pairs), m * 16, [&](const uint8_t *p, size_t len) -> kmg_status {
      if (fwrite(p, 1, len, f) != len) return fail(c, KMG_ERR_IO, "short write to the index file");
      const uint32_t part = crc32_parallel(p, len);
      crc = first ? part : crc32_combine(crc, part, len);
      first = false;
      return KMG_OK;
    });
  });
  pool_free(c, d_pairs);
  if (s != KMG_OK) return s;
  if (written != n) return fail(c, KMG_ERR_STATE, "kmix writer: pieces do not add up to the table");
  *crc_out = crc;
  return KMG_OK;
}

bool has_gz_suffix(const char *path) { const size_t l = strlen(path); return l >= 3 && strcmp(path + l - 3, ".gz") == 0; }
}  // namespace

KMG_EXPORT kmg_status kmg_save_kmix(kmg_ctx *c, const char *path) {
  if (!c || !path) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  // src/index.rs:159-168 gzips when the path ends in .gz; this writer does not compress -- refuse rather than write raw bytes
  // under a .gz name (the reference's load_index would reject that file)
  if (has_gz_suffix(path)) return fail(c, KMG_ERR_INVALID_ARG, "kmg_save_kmix writes uncompressed .kmix files; gzip on the host side for a .gz path");
  CU(c, cudaSetDevice(c->device));
  uint64_t n = 0;
  kmg_status s = count_filtered(c, 0, &n);
  if (s != KMG_OK) return s;
  FILE *f = fopen(path, "wb");
  if (!f) return fail(c, KMG_ERR_IO, std::string("cannot open ") + path + " for writing");
  const Crc32 &T = crc_tables();
  uint8_t hdr[14] = {'K', 'M', 'I', 'X', 1, (uint8_t)c->k};
  for (int b = 0; b < 8; ++b) hdr[6 + b] = (uint8_t)(n >> (8 * b));
  bool ok = fwrite(hdr, 1, 14, f) == 14;
  uint32_t crc = ~T.update(~0u, hdr, 14), body_crc = 0;
  uint64_t n2 = 0;
  s = write_kmix_records(c, f, &body_crc, &n2);
  if (s != KMG_OK) { fclose(f); return s; }
  crc = crc32_combine(crc, body_crc, n2 * 16);
  uint8_t tail[4] = {(uint8_t)crc, (uint8_t)(crc >> 8), (uint8_t)(crc >> 16), (uint8_t)(crc >> 24)};
  ok = ok && n2 == n && fwrite(tail, 1, 4, f) == 4;
  ok = (fclose(f) == 0) && ok;
  if (!ok) return fail(c, KMG_ERR_IO, std::string("short write to ") + path);
  return KMG_OK;
}

// .kmix from several shards (one context per GPU / process; src/index.rs:222-279 writes header, n records in arbitrary order,
// CRC).  Every shard writes its records into ITS byte range of the same file -- record_offset = number of records of the shards
// before it -- and reports their count and CRC; kmg_kmix_finish then writes the header (n = sum) and the trailing CRC combined
// from the shards' CRCs.  The file must exist (kmg_kmix_begin creates / truncates it).
KMG_EXPORT kmg_status kmg_kmix_begin(const char *path) {
  if (!path || has_gz_suffix(path)) return KMG_ERR_INVALID_ARG;
  FILE *f = fopen(path, "wb");
  if (!f) return KMG_ERR_IO;
  return fclose(f) == 0 ? KMG_OK : KMG_ERR_IO;
}
KMG_EXPORT kmg_status kmg_save_kmix_shard(kmg_ctx *c, const char *path, uint64_t record_offset, uint64_t *n_records_out, uint32_t *crc_out) {
  if (!c || !path || !n_records_out || !crc_out) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  CU(c, cudaSetDevice(c->device));
  FILE *f = fopen(path, "r+b");
  if (!f) return fail(c, KMG_ERR_IO, std::string("cannot open ") + path + " (call kmg_kmix_begin first)");
  if (fseeko(f, (off_t)(14 + 16 * record_offset), SEEK_SET) != 0) { fclose(f); return fail(c, KMG_ERR_IO, "seek failed"); }
  kmg_status s = write_kmix_records(c, f, crc_out, n_records_out);
  const bool ok = fclose(f) == 0;
  if (s != KMG_OK) return s;
  return ok ? KMG_OK : fail(c, KMG_ERR_IO, std::string("short write to ") + path);
}
KMG_EXPORT kmg_status kmg_kmix_finish(const char *path, uint32_t k, const uint64_t *shard_records, const uint32_t *shard_crcs, uint32_t n_shards) {
  if (!path || k < 1 || k > 32 || (n_shards && (!shard_records || !shard_crcs))) return KMG_ERR_INVALID_ARG;
  uint64_t n = 0;
  for (uint32_t i = 0; i < n_shards; ++i) n += shard_records[i];
  FILE *f = fopen(path, "r+b");
  if (!f) return KMG_ERR_IO;
  const Crc32 &T = crc_tables();
  uint8_t hdr[14] = {'K', 'M', 'I', 'X', 1, (uint8_t)k};
  for (int b = 0; b < 8; ++b) hdr[6 + b] = (uint8_t)(n >> (8 * b));
  uint32_t crc = ~T.update(~0u, hdr, 14);
  for (uint32_t i = 0; i < n_shards; ++i) crc = crc32_combine(crc, shard_crcs[i], shard_records[i] * 16);
  uint8_t tail[4] = {(uint8_t)crc, (uint8_t)(crc >> 8), (uint8_t)(crc >> 16), (uint8_t)(crc >> 24)};
  bool ok = fseeko(f, 0, SEEK_SET) == 0 && fwrite(hdr, 1, 14, f) == 14;
  ok = ok && fseeko(f, (off_t)(14 + 16 * n), SEEK_SET) == 0 && fwrite(tail, 1, 4, f) == 4;
  ok = (fclose(f) == 0) && ok;
  return ok ? KMG_OK : KMG_ERR_IO;
}


// ---- results of a shard group (collective calls: every rank makes the same sequence of them) ---------------------------
// Global summary: sums over the (disjoint) shards, maximum of max_count; the timing fields stay this rank's own.
KMG_EXPORT kmg_status kmg_shard_finalize(kmg_ctx *c, kmg_summary *out) {
  if (!c) return KMG_ERR_INVALID_ARG;
  kmg_summary loc;
  kmg_status s = kmg_finalize(c, &loc);
  if (!c->shm) { if (out) *out = loc; return s; }
  if (s != KMG_OK) return shard_fail(c, s, c->err);
  const uint64_t m[5] = {loc.n_windows, loc.n_distinct, loc.n_records, loc.n_bases, loc.max_count};
  std::vector<uint64_t> all;
  if ((s = shard_allgather(c, m, 5, all)) != KMG_OK) return s;
  if (out) {
    *out = loc;
    out->n_windows = out->n_distinct = out->n_records = out->n_bases = out->max_count = 0;
    for (uint32_t r = 0; r < c->sh_world; ++r) {
      const uint64_t *o = all.data() + 5 * r;
      out->n_windows += o[0]; out->n_distinct += o[1]; out->n_records += o[2]; out->n_bases += o[3];
      out->max_count = std::max<uint64_t>(out->max_count, o[4]);
    }
  }
  return KMG_OK;
}

// Count-of-counts over all shards: the element-wise sum of the shard histograms (a k-mer lives in exactly one shard).
// Replaces compute_histogram_packed (src/histogram.rs:110-116) for the sharded table.  Two-call protocol like kmg_histogram;
// the size query does the merge (collective), the call with arrays returns that merged result.
KMG_EXPORT kmg_status kmg_shard_histogram(kmg_ctx *c, uint64_t min_count, uint64_t *count_vals, uint64_t *freqs, uint64_t cap, uint64_t *n_out) {
  if (!c || !n_out) return KMG_ERR_INVALID_ARG;
  if (!c->shm) return kmg_histogram(c, min_count, count_vals, freqs, cap, n_out);
  if (!count_vals || !freqs) {
    uint64_t n = 0;
    kmg_status s = kmg_histogram(c, min_count, nullptr, nullptr, 0, &n);
    if (s != KMG_OK) return shard_fail(c, s, c->err);
    if (n > SHARD_HIST_MAX) return shard_fail(c, KMG_ERR_CAPACITY, "shard histogram has too many distinct count values");
    std::vector<uint64_t> mine(1 + 2 * n), posted;  // n, the n values, their n frequencies
    mine[0] = n;
    if (n && (s = kmg_histogram(c, min_count, &mine[1], &mine[1 + n], n, &n)) != KMG_OK) return shard_fail(c, s, c->err);
    if ((s = shard_allgather(c, mine.data(), mine.size(), posted, /*counted_pairs=*/true)) != KMG_OK) return s;
    std::vector<std::pair<uint64_t, uint64_t>> all;
    for (size_t o = 0; o < posted.size(); o += 1 + 2 * posted[o])
      for (uint64_t i = 0; i < posted[o]; ++i) all.emplace_back(posted[o + 1 + i], posted[o + 1 + posted[o] + i]);
    std::sort(all.begin(), all.end());
    c->sh_hist_vals.clear(); c->sh_hist_freqs.clear();
    for (size_t i = 0; i < all.size();) {
      uint64_t f = 0;
      size_t j = i;
      for (; j < all.size() && all[j].first == all[i].first; ++j) f += all[j].second;
      c->sh_hist_vals.push_back(all[i].first); c->sh_hist_freqs.push_back(f);
      i = j;
    }
    *n_out = c->sh_hist_vals.size();
    return KMG_OK;
  }
  const uint64_t n = c->sh_hist_vals.size();
  *n_out = n;
  if (cap < n) return fail(c, KMG_ERR_CAPACITY, "histogram arrays hold " + std::to_string(cap) + " bins, need " + std::to_string(n));
  if (n) { memcpy(count_vals, c->sh_hist_vals.data(), n * 8); memcpy(freqs, c->sh_hist_freqs.data(), n * 8); }
  return KMG_OK;
}

// ONE .kmix index from all shards of the group (src/index.rs:222-279; records in shard order, each shard ascending): rank 0
// creates the file, every rank writes its records into its own byte range, rank 0 writes the header (n = sum) and the CRC of
// the whole file combined from the shards' CRCs.  *n_records_out: records of the whole index.
KMG_EXPORT kmg_status kmg_shard_save_kmix(kmg_ctx *c, const char *path, uint64_t *n_records_out) {
  if (!c || !path) return KMG_ERR_INVALID_ARG;
  if (!c->shm) {
    kmg_status s = kmg_save_kmix(c, path);
    if (s == KMG_OK && n_records_out) { uint64_t n = 0; s = count_filtered(c, 0, &n); *n_records_out = n; }
    return s;
  }
  if (has_gz_suffix(path)) return shard_fail(c, KMG_ERR_INVALID_ARG, "kmg_shard_save_kmix writes uncompressed .kmix files");
  CU(c, cudaSetDevice(c->device));
  uint64_t n = 0;
  kmg_status s = count_filtered(c, 0, &n);
  if (s != KMG_OK) return shard_fail(c, s, c->err);
  if (c->sh_rank == 0 && kmg_kmix_begin(path) != KMG_OK) return shard_fail(c, KMG_ERR_IO, std::string("cannot create ") + path);
  std::vector<uint64_t> recs, crcs;  // every shard's records, then the CRCs of their bytes
  if ((s = shard_allgather(c, &n, 1, recs)) != KMG_OK) return s;
  uint64_t before = 0, total = 0;
  for (uint32_t r = 0; r < c->sh_world; ++r) { if (r < c->sh_rank) before += recs[r]; total += recs[r]; }
  uint64_t n2 = 0;
  uint32_t crc = 0;
  s = kmg_save_kmix_shard(c, path, before, &n2, &crc);
  if (s != KMG_OK) return shard_fail(c, s, c->err);
  if (n2 != n) return shard_fail(c, KMG_ERR_STATE, "shard index writer wrote an unexpected number of records");
  const uint64_t my_crc = crc;
  if ((s = shard_allgather(c, &my_crc, 1, crcs)) != KMG_OK) return s;
  if (c->sh_rank == 0) {
    uint32_t crc32s[SHARD_MAX_WORLD];
    for (uint32_t r = 0; r < c->sh_world; ++r) crc32s[r] = (uint32_t)crcs[r];
    const kmg_status fs = kmg_kmix_finish(path, (uint32_t)c->k, recs.data(), crc32s, c->sh_world);
    if (fs != KMG_OK) return shard_fail(c, fs, std::string("cannot finish ") + path);
  }
  SB(c);  // no rank returns before rank 0 has finished the file
  if (n_records_out) *n_records_out = total;
  return KMG_OK;
}

// Diagnostics of the exchange: keys this rank wrote into other ranks' buffers, keys it received, rounds, exact-route rounds.
KMG_EXPORT kmg_status kmg_shard_stats(const kmg_ctx *c, uint64_t *sent_keys, uint64_t *recv_keys, uint64_t *rounds, uint64_t *exact_rounds) {
  if (!c) return KMG_ERR_INVALID_ARG;
  if (sent_keys) *sent_keys = c->sh_sent;
  if (recv_keys) *recv_keys = c->sh_recv_keys;
  if (rounds) *rounds = c->sh_rounds;
  if (exact_rounds) *exact_rounds = c->sh_exact_rounds;
  return KMG_OK;
}


// Text emitters of output_counts / count_to_writer (src/run.rs:452-481, src/builder.rs:399-442) for --format tsv, fasta and json:
// records with count >= min_count in ascending k-mer order (the reference prints HashMap order; parity is on the sorted text),
// formatted ON THE DEVICE (2-bit unpack + decimal count), delivered to `sink` in chunks of at most 64 MiB.  json's framing goes
// to the sink before the first piece and after the last one.
KMG_EXPORT kmg_status kmg_emit_text(kmg_ctx *c, uint64_t min_count, int format, kmg_text_sink sink, void *user, uint64_t *n_records_out,
                                    uint64_t *n_bytes_out) {
  if (!c || !sink) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  if (format != KMG_TEXT_FASTA && format != KMG_TEXT_TSV && format != KMG_TEXT_JSON)
    return fail(c, KMG_ERR_INVALID_ARG, "format must be KMG_TEXT_FASTA, KMG_TEXT_TSV or KMG_TEXT_JSON");
  CU(c, cudaSetDevice(c->device));
  if (min_count == 0) min_count = 1;
  uint64_t records = 0, bytes = 0;
  auto to_sink = [&](const uint8_t *p, size_t len) -> kmg_status {
    return sink(user, p, len) == 0 ? KMG_OK : fail(c, KMG_ERR_IO, "the text sink reported an error");
  };
  auto frame = [&](const char *t) -> kmg_status {
    bytes += strlen(t);
    return to_sink(reinterpret_cast<const uint8_t *>(t), strlen(t));
  };
  kmg_status s = format == KMG_TEXT_JSON ? frame(JSON_OPEN) : KMG_OK;
  HostStager stage(c, 64u << 20);
  TextFormatter fmt(c, format);
  if (s == KMG_OK)
    s = for_each_sorted_piece(c, min_count, 1ull << 24, [&](const uint64_t *dk, const uint64_t *dc, uint64_t m) -> kmg_status {
      uint64_t total = 0;
      kmg_status fs = fmt.format(dk, dc, m, records == 0, &total);
      if (fs != KMG_OK) return fs;
      records += m; bytes += total;
      return stage.drain(fmt.d_text, total, to_sink);
    });
  if (s == KMG_OK && format == KMG_TEXT_JSON) s = frame(json_close(records));
  if (n_records_out) *n_records_out = records;
  if (n_bytes_out) *n_bytes_out = bytes;
  return s;
}

namespace {
int file_sink(void *user, const uint8_t *p, size_t n) { return fwrite(p, 1, n, static_cast<FILE *>(user)) == n ? 0 : 1; }
}  // namespace

// The same into a file ("-" = stdout): what `kmerust <k> <path> --format tsv|fasta|json --min-count m > file` produces, sorted.
KMG_EXPORT kmg_status kmg_write_text(kmg_ctx *c, uint64_t min_count, int format, const char *path, uint64_t *n_records_out, uint64_t *n_bytes_out) {
  if (!c || !path) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  const bool to_stdout = strcmp(path, "-") == 0;
  FILE *f = to_stdout ? stdout : fopen(path, "wb");
  if (!f) return fail(c, KMG_ERR_IO, std::string("cannot open ") + path + " for writing");
  kmg_status s = kmg_emit_text(c, min_count, format, file_sink, f, n_records_out, n_bytes_out);
  const bool ok = to_stdout ? fflush(f) == 0 : fclose(f) == 0;
  if (s == KMG_OK && !ok) return fail(c, KMG_ERR_IO, std::string("short write to ") + path);
  return s;
}

// The same file from all shards of a group, byte for byte.  The shards split the keys by hash, so every key range is spread over
// all ranks.  The key space is cut into pieces of ~2^24 records from the ranks' summed key histograms; W consecutive pieces make a
// step.  In each step every rank compacts and sorts its part of the step's key range into a staging buffer its peers can read;
// rank j then owns piece j of the step: it merges the piece's W sorted parts straight out of the peers' memory
// (merge_shard_pieces_kernel), formats it on the device and writes it at its offset in the file (the bytes of all earlier pieces).
// json: every piece lands after the "[" that rank 0 writes at offset 0; the owner of the first non-empty piece of the file formats
// its first record without the "," separator; rank 0 writes the closing bracket after the last step.
KMG_EXPORT kmg_status kmg_shard_write_text(kmg_ctx *c, uint64_t min_count, int format, const char *path, uint64_t *n_records_out,
                                           uint64_t *n_bytes_out) {
  if (!c || !path) return KMG_ERR_INVALID_ARG;
  if (!c->shm) return kmg_write_text(c, min_count, format, path, n_records_out, n_bytes_out);
  // every rank sees the same path: all of them refuse here, before any barrier
  if (strcmp(path, "-") == 0) return fail(c, KMG_ERR_INVALID_ARG, "a shard group writes its text to a file: ranks cannot write one stream at given offsets");
  if (format != KMG_TEXT_FASTA && format != KMG_TEXT_TSV && format != KMG_TEXT_JSON)
    return shard_fail(c, KMG_ERR_INVALID_ARG, "format must be KMG_TEXT_FASTA, KMG_TEXT_TSV or KMG_TEXT_JSON");
  const bool json = format == KMG_TEXT_JSON;
  const uint64_t head = json ? strlen(JSON_OPEN) : 0;  // bytes in front of the first piece
  if (min_count == 0) min_count = 1;
  SCU(c, cudaSetDevice(c->device));
  const uint32_t W = c->sh_world, me = c->sh_rank;
  // 1. arguments, records that pass min_count and key histogram of every shard; rank 0 creates / truncates the file
  constexpr size_t AW = 3 + KEY_BUCKETS;  // min_count, format, records, key histogram
  std::vector<uint64_t> mine(AW), args;
  mine[0] = min_count; mine[1] = (uint64_t)format;
  kmg_status s = count_filtered(c, min_count, &mine[2]);
  if (s == KMG_OK) s = key_histogram(c, &mine[3]);
  if (s != KMG_OK) return shard_fail(c, s, c->err);
  if (me == 0) {
    FILE *f = fopen(path, "wb");
    if (!f || fclose(f) != 0) return shard_fail(c, KMG_ERR_IO, std::string("cannot create ") + path);
  }
  if ((s = shard_allgather(c, mine.data(), AW, args)) != KMG_OK) return s;
  auto hist_of = [&](uint32_t r) { return args.data() + r * AW + 3; };
  for (uint32_t r = 0; r < W; ++r)
    if (args[r * AW] != min_count || args[r * AW + 1] != (uint64_t)format)
      return shard_fail(c, KMG_ERR_INVALID_ARG, "ranks disagree on min_count / format (pass identical arguments on every rank)");
  // 2. the same pieces on every rank; staging buffers sized for the largest part of a step any rank holds, merge buffers for the
  //    largest piece this rank owns
  std::vector<uint64_t> sum(KEY_BUCKETS, 0);
  for (uint32_t r = 0; r < W; ++r)
    for (int b = 0; b < KEY_BUCKETS; ++b) sum[b] += hist_of(r)[b];
  const std::vector<int> cuts = piece_cuts(sum.data(), 1ull << 24);
  const size_t n_pieces = cuts.size() - 1;
  std::vector<int> step_cuts;
  for (size_t p = 0; p < n_pieces; p += W) step_cuts.push_back(cuts[p]);
  if (n_pieces) step_cuts.push_back(cuts[n_pieces]);
  uint64_t stage_cap = 1, own_cap = 1;
  for (uint32_t r = 0; r < W; ++r) stage_cap = std::max(stage_cap, largest_piece(hist_of(r), step_cuts));
  for (size_t p = me; p < n_pieces; p += W) own_cap = std::max(own_cap, largest_piece(sum.data(), {cuts[p], cuts[p + 1]}));
  const int shift = key_bucket_shift(c);
  uint64_t *stage = nullptr, *dk = nullptr, *dc = nullptr, *d_aux = nullptr;
  uint64_t *peer[SHARD_MAX_WORLD] = {};
  bool peer_ipc[SHARD_MAX_WORLD] = {};
  int fd = -1;
  uint64_t records = 0, file_bytes = 0;
  std::vector<uint64_t> all;
  auto run = [&]() -> kmg_status {
    SCU(c, cudaMalloc(&stage, 2 * stage_cap * 8));  // (key, count) SoA: keys [0, stage_cap), counts [stage_cap, 2 * stage_cap)
    SCU(c, pool_alloc(c, &dk, own_cap * 8));
    SCU(c, pool_alloc(c, &dc, own_cap * 8));
    SCU(c, pool_alloc(c, &d_aux, (SHARD_MAX_WORLD + 2) * 8));  // piece bounds + the merge's placed-record counter
    PeerBuf mine_stage;
    publish_peer_buffer(mine_stage, stage);
    kmg_status gs = shard_allgather(c, &mine_stage, PEER_BUF_WORDS, all);
    if (gs != KMG_OK) return gs;
    const std::string why = open_peer_buffers(c, all, PEER_BUF_WORDS, peer, peer_ipc);
    if (!why.empty()) return shard_fail(c, KMG_ERR_CUDA, why);
    if ((fd = open(path, O_WRONLY)) < 0) return shard_fail(c, KMG_ERR_IO, std::string("cannot open ") + path + " for writing");
    HostStager staged(c, 64u << 20);
    TextFormatter fmt(c, format);
    uint64_t written = 0;
    auto put = [&](const uint8_t *p, size_t len, uint64_t off) -> kmg_status {
      for (size_t done = 0; done < len;) {
        const ssize_t w = pwrite(fd, p + done, len - done, (off_t)(off + done));
        if (w <= 0) return shard_fail(c, KMG_ERR_IO, std::string("short write to ") + path);
        done += (size_t)w; written += (uint64_t)w;
      }
      return KMG_OK;
    };
    size_t step = 0;
    kmg_status st = for_each_sorted_piece(c, min_count, step_cuts, stage, stage + stage_cap, stage_cap,
                                          [&](const uint64_t *sk, const uint64_t *, uint64_t m) -> kmg_status {
      // 3. this rank's part of the step is sorted in its staging buffer: where does each piece start in it
      const size_t p0 = step++ * W;
      const uint32_t n_own = (uint32_t)std::min<size_t>(W, n_pieces - p0);
      uint64_t cut_keys[SHARD_MAX_WORLD + 1], bounds[SHARD_MAX_WORLD + 1];
      for (uint32_t j = 0; j < n_own; ++j) cut_keys[j] = (uint64_t)cuts[p0 + j] << shift;
      SCU(c, launch_piece_bounds(sk, m, cut_keys, n_own, d_aux, c->stream));
      SCU(c, cudaMemcpyAsync(bounds, d_aux, n_own * 8, cudaMemcpyDeviceToHost, c->stream));
      SCU(c, cudaStreamSynchronize(c->stream));
      bounds[n_own] = m;
      kmg_status gst = shard_allgather(c, bounds, n_own + 1, all);  // every rank's part of the step is in its staging buffer
      if (gst != KMG_OK) return gst;
      // 4. the owner merges its piece out of all staging buffers and formats it
      uint64_t expect = 0, bytes = 0;
      unsigned long long placed = 0;
      if (me < n_own) {
        MergeRuns R{};
        R.n_runs = W;
        uint64_t before = records;  // records of the file in front of this piece: earlier steps + earlier pieces of this step
        for (uint32_t q = 0; q < W; ++q) {
          const uint64_t lo = all[q * (n_own + 1) + me], hi = all[q * (n_own + 1) + me + 1];
          R.keys[q] = peer[q] + lo; R.counts[q] = peer[q] + stage_cap + lo; R.len[q] = hi - lo;
          expect += hi - lo; before += lo;
        }
        if (expect > own_cap) return shard_fail(c, KMG_ERR_STATE, "merged piece larger than its key histogram");
        unsigned long long *d_placed = reinterpret_cast<unsigned long long *>(d_aux + SHARD_MAX_WORLD + 1);
        SCU(c, launch_merge_shard_pieces(R, dk, dc, d_placed, c->stream));
        SCU(c, cudaMemcpyAsync(&placed, d_placed, 8, cudaMemcpyDeviceToHost, c->stream));
        kmg_status fs = fmt.format(dk, dc, expect, before == 0 && expect > 0, &bytes);  // ends in a stream synchronize
        if (fs != KMG_OK) return shard_fail(c, fs, c->err);
      }
      const uint64_t piece[3] = {expect, placed, bytes};  // records expected, records the merge placed in order, bytes
      // nobody reads a staging buffer of this step any more after this gather: the next step may overwrite them
      if ((gst = shard_allgather(c, piece, 3, all)) != KMG_OK) return gst;
      // 5. file offset = json's "[" + bytes of all earlier pieces; every merged piece holds as many ordered records as its parts
      uint64_t off = head + file_bytes;
      for (uint32_t j = 0; j < n_own; ++j) {
        const uint64_t *tp = all.data() + 3 * j;
        if (tp[0] != tp[1]) return shard_fail(c, KMG_ERR_STATE, "piece " + std::to_string(p0 + j) + ": the merge placed " + std::to_string(tp[1]) + " records in order, its parts hold " + std::to_string(tp[0]));
        if (j < me) off += tp[2];
        file_bytes += tp[2]; records += tp[0];
      }
      return staged.drain(fmt.d_text, bytes, [&](const uint8_t *p, size_t len) -> kmg_status {
        kmg_status ps = put(p, len, off);
        off += len;
        return ps;
      });
    });
    if (st != KMG_OK) return shard_fail(c, st, c->err);
    if (json) {  // every rank knows the group's records now; rank 0 writes the framing around the pieces
      const char *tail = json_close(records);
      if (me == 0) {
        if ((st = put(reinterpret_cast<const uint8_t *>(JSON_OPEN), head, 0)) != KMG_OK) return st;
        if ((st = put(reinterpret_cast<const uint8_t *>(tail), strlen(tail), head + file_bytes)) != KMG_OK) return st;
      }
      file_bytes += head + strlen(tail);
    }
    const int closed = close(fd);
    fd = -1;
    if (closed != 0) return shard_fail(c, KMG_ERR_IO, std::string("short write to ") + path);
    if ((gs = shard_allgather(c, &written, 1, all)) != KMG_OK) return gs;
    // 6. the file holds every record of every shard that passes min_count, and every byte the owners formatted
    uint64_t want_records = 0, total_written = 0;
    for (uint32_t r = 0; r < W; ++r) { want_records += args[r * AW + 2]; total_written += all[r]; }
    if (records != want_records) return shard_fail(c, KMG_ERR_STATE, "text file holds " + std::to_string(records) + " records, the shards " + std::to_string(want_records));
    if (total_written != file_bytes) return shard_fail(c, KMG_ERR_STATE, "bytes written differ from the bytes of the formatted pieces");
    close_peer_buffers(peer, peer_ipc);
    SB(c);  // every peer has closed its mapping of this rank's staging buffer
    return KMG_OK;
  };
  s = run();
  close_peer_buffers(peer, peer_ipc);
  if (fd >= 0) close(fd);
  cudaStreamSynchronize(c->stream);
  cudaFree(stage);
  pool_free(c, dk); pool_free(c, dc); pool_free(c, d_aux);
  if (s != KMG_OK) return s;
  if (n_records_out) *n_records_out = records;
  if (n_bytes_out) *n_bytes_out = file_bytes;
  return KMG_OK;
}


// ---- index queries and loading (src/index.rs:127-131 KmerIndex::get, :199-216 load_index, :282-401 read_index; the consumer is
// the `query` subcommand, src/main.rs:233-281) --------------------------------------------------------------------------------
namespace {
kmg_status query_device_keys(kmg_ctx *c, const uint64_t *d_keys, uint64_t n, uint64_t *counts_out) {
  { kmg_status _fs = scan_pending_batch(c); if (_fs != KMG_OK) return _fs; }
  CU(c, cudaStreamSynchronize(c->copy_stream));
  if (c->mode == kmg_ctx::MODE_PARTITIONED) { kmg_status s = consolidate(c); if (s != KMG_OK) return s; }
  uint64_t *d_counts = nullptr;
  CU(c, pool_alloc(c, &d_counts, std::max<uint64_t>(n, 1) * 8));
  const bool part = c->mode == kmg_ctx::MODE_PARTITIONED;
  TableView v = view_of(c);
  cudaError_t e = cudaSuccess;
  if (part && !c->has_result) e = cudaMemsetAsync(d_counts, 0, n * 8, c->stream);  // nothing counted yet
  else e = launch_query(v, c->table, part ? c->result.d_seg_start : nullptr, part ? c->result.d_seg_len : nullptr, std::max<uint32_t>(c->n_coarse, 1),
                        std::max<uint32_t>(c->n_sub, 1), c->shm ? c->sh_world : 1, c->shm ? c->sh_rank : 0, d_keys, n, d_counts, c->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(counts_out, d_counts, n * 8, cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  pool_free(c, d_counts);
  if (e != cudaSuccess) return cuda_fail(c, e, "query");
  return KMG_OK;
}
}  // namespace

// counts_out[i] = count of the canonical packed key keys[i] (0 when absent).  HOST arrays.
KMG_EXPORT kmg_status kmg_query_keys(kmg_ctx *c, const uint64_t *keys, uint64_t n, uint64_t *counts_out) {
  if (!c || (n && (!keys || !counts_out))) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  if (n == 0) return KMG_OK;
  CU(c, cudaSetDevice(c->device));
  uint64_t *d_keys = nullptr;
  CU(c, pool_alloc(c, &d_keys, n * 8));
  cudaError_t e = cudaMemcpyAsync(d_keys, keys, n * 8, cudaMemcpyHostToDevice, c->stream);
  kmg_status s = e == cudaSuccess ? query_device_keys(c, d_keys, n, counts_out) : cuda_fail(c, e, "H2D query keys");
  pool_free(c, d_keys);
  return s;
}

// n k-mers as ASCII, k bytes each, back to back, any case: canonicalised on the device (upper-case, pack, min(fwd, rc) -- what the
// query subcommand does on the host) and looked up.  A k-mer with a byte outside ACGTacgt counts 0 and sets *n_invalid_out.
KMG_EXPORT kmg_status kmg_query_ascii(kmg_ctx *c, const uint8_t *kmers, uint64_t n, uint64_t *counts_out, uint64_t *n_invalid_out) {
  if (!c || (n && (!kmers || !counts_out))) return KMG_ERR_INVALID_ARG;
  NO_OPEN_STREAM(c);
  if (n_invalid_out) *n_invalid_out = 0;
  if (n == 0) return KMG_OK;
  CU(c, cudaSetDevice(c->device));
  uint8_t *d_kmers = nullptr;
  uint64_t *d_keys = nullptr;
  CU(c, pool_alloc(c, &d_kmers, n * (uint64_t)c->k));
  cudaError_t e = pool_alloc(c, &d_keys, n * 8);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_kmers, kmers, n * (uint64_t)c->k, cudaMemcpyHostToDevice, c->stream);
  if (e == cudaSuccess) e = launch_query_pack(d_kmers, n, c->k, d_keys, c->stream);
  kmg_status s = e == cudaSuccess ? query_device_keys(c, d_keys, n, counts_out) : cuda_fail(c, e, "query (pack)");
  if (s == KMG_OK && n_invalid_out) {
    std::vector<uint64_t> hk(n);
    e = cudaMemcpy(hk.data(), d_keys, n * 8, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) s = cuda_fail(c, e, "query (invalid k-mers)");
    else for (uint64_t x : hk) *n_invalid_out += x == EMPTY_KEY;
  }
  pool_free(c, d_kmers); pool_free(c, d_keys);
  return s;
}

// Open a .kmix index as a ready-to-query context on `device`: the checks of read_index in the reference's order (size >= 18,
// magic, CRC, version, k, n * 16 == data size; src/index.rs:282-401), then the records are streamed to the device and
// upserted.  Errors: KMG_ERR_IO (cannot read) / KMG_ERR_PARSE (invalid index; message via kmg_last_error(NULL)).
KMG_EXPORT kmg_status kmg_index_open(const char *path, int32_t device, kmg_ctx **out) {
  if (!path || !out) return KMG_ERR_INVALID_ARG;
  *out = nullptr;
  if (has_gz_suffix(path)) return fail(nullptr, KMG_ERR_INVALID_ARG, "kmg_index_open reads uncompressed .kmix files; gunzip on the host side");
  FILE *f = fopen(path, "rb");
  if (!f) return fail(nullptr, KMG_ERR_IO, std::string("failed to read index from '") + path + "'");
  struct Closer { FILE *f; ~Closer() { if (f) fclose(f); } } closer{f};
  if (fseeko(f, 0, SEEK_END) != 0) return fail(nullptr, KMG_ERR_IO, "seek failed");
  const uint64_t size = (uint64_t)ftello(f);
  rewind(f);
  if (size < 18) return fail(nullptr, KMG_ERR_PARSE, "file too small");
  uint8_t hdr[14];
  if (fread(hdr, 1, 14, f) != 14) return fail(nullptr, KMG_ERR_IO, "short read");
  if (memcmp(hdr, "KMIX", 4) != 0) return fail(nullptr, KMG_ERR_PARSE, "invalid magic bytes (not a kmerust index file)");
  // CRC over everything before the last four bytes, streamed (the reference buffers the whole file)
  const Crc32 &T = crc_tables();
  uint32_t crc = ~T.update(~0u, hdr, 14);
  const uint64_t body = size - 18;
  std::vector<uint8_t> buf((size_t)std::min<uint64_t>(std::max<uint64_t>(body, 16), 256ull << 20));
  for (uint64_t done = 0; done < body;) {
    const size_t m = (size_t)std::min<uint64_t>(buf.size(), body - done);
    if (fread(buf.data(), 1, m, f) != m) return fail(nullptr, KMG_ERR_IO, "short read");
    crc = crc32_combine(crc, crc32_parallel(buf.data(), m), m);
    done += m;
  }
  uint8_t tail[4];
  if (fread(tail, 1, 4, f) != 4) return fail(nullptr, KMG_ERR_IO, "short read");
  const uint32_t stored = (uint32_t)tail[0] | (uint32_t)tail[1] << 8 | (uint32_t)tail[2] << 16 | (uint32_t)tail[3] << 24;
  if (stored != crc) { char m[96]; snprintf(m, sizeof m, "checksum mismatch (expected %#x, got %#x)", stored, crc); return fail(nullptr, KMG_ERR_PARSE, m); }
  if (hdr[4] != 1) return fail(nullptr, KMG_ERR_PARSE, "unsupported version " + std::to_string(hdr[4]));
  const uint32_t k = hdr[5];
  if (k < 1 || k > 32) return fail(nullptr, KMG_ERR_PARSE, "invalid k-mer length: k-mer length " + std::to_string(k) + " is out of range (must be 1-32)");
  uint64_t n = 0;
  for (int b = 0; b < 8; ++b) n |= (uint64_t)hdr[6 + b] << (8 * b);
  if (body != n * 16) return fail(nullptr, KMG_ERR_PARSE, "data size mismatch (expected " + std::to_string(n * 16) + " bytes, got " + std::to_string(body) + " bytes)");
  kmg_config cfg{};
  cfg.abi_version = KMG_ABI_VERSION; cfg.k = k; cfg.device = device; cfg.expected_distinct = std::max<uint64_t>(n, 1);
  kmg_ctx *c = nullptr;
  kmg_status s = kmg_create(&cfg, &c);
  if (s != KMG_OK) return s;
  auto bail = [&](kmg_status st) { g_create_error = c->err; kmg_destroy(c); return st; };
  if (n) {
    if (fseeko(f, 14, SEEK_SET) != 0) return bail(fail(c, KMG_ERR_IO, "seek failed"));
    const uint64_t CH = std::min<uint64_t>(n, 1ull << 24);  // records per piece (256 MiB)
    void *d_pairs = nullptr;
    uint64_t *dk = nullptr, *dc = nullptr;
    cudaError_t e = pool_alloc(c, &d_pairs, CH * 16);
    if (e == cudaSuccess) e = pool_alloc(c, &dk, CH * 8);
    if (e == cudaSuccess) e = pool_alloc(c, &dc, CH * 8);
    if (e != cudaSuccess) return bail(cuda_fail(c, e, "cudaMalloc(index load)"));
    buf.resize((size_t)(CH * 16));
    for (uint64_t done = 0; done < n && s == KMG_OK;) {
      const uint64_t m = std::min<uint64_t>(CH, n - done);
      if (fread(buf.data(), 16, m, f) != m) { s = fail(c, KMG_ERR_IO, "short read"); break; }
      e = cudaMemcpyAsync(d_pairs, buf.data(), m * 16, cudaMemcpyHostToDevice, c->stream);
      if (e == cudaSuccess) e = launch_deinterleave_pairs(d_pairs, m, dk, dc, c->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
      if (e != cudaSuccess) { s = cuda_fail(c, e, "index load"); break; }
      s = kmg_insert_keys_device(c, dk, dc, m);
      done += m;
    }
    pool_free(c, d_pairs); pool_free(c, dk); pool_free(c, dc);
    if (s == KMG_OK) s = kmg_finalize(c, nullptr);
    if (s != KMG_OK) return bail(s);
  }
  *out = c;
  return KMG_OK;
}

KMG_EXPORT kmg_status kmg_progress(const kmg_ctx *c, uint64_t *records, uint64_t *bases) {
  if (!c) return KMG_ERR_INVALID_ARG;
  if (records) *records = c->n_records;
  if (bases) *bases = c->n_bases;
  return KMG_OK;
}

KMG_EXPORT uint64_t kmg_kernel_launches(void) { return kernel_launches(); }

KMG_EXPORT kmg_status kmg_phase_times(kmg_ctx *c, uint64_t *out_ns) {
  if (!c || !out_ns) return KMG_ERR_INVALID_ARG;
  CU(c, cudaSetDevice(c->device));
  CU(c, cudaStreamSynchronize(c->stream));
  timers_collect(c);
  const double a2 = c->cat_ms[2], a1 = std::max(0.0, c->cat_ms[0] - a2), b = c->cat_ms[1];
  out_ns[0] = (uint64_t)(a1 * 1e6); out_ns[1] = (uint64_t)(a2 * 1e6); out_ns[2] = (uint64_t)(b * 1e6);
  out_ns[3] = (uint64_t)(std::max(0.0, c->kernel_ms - c->cat_ms[0] - b) * 1e6);
  return KMG_OK;
}

KMG_EXPORT kmg_status kmg_synth_uniform_device(kmg_ctx *c, uint64_t seed, uint64_t first_base, uint64_t n, uint8_t *d_out) {
  if (!c) return KMG_ERR_INVALID_ARG;
  CU(c, cudaSetDevice(c->device));
  if (n) CU(c, launch_synth_uniform(seed, first_base, n, d_out, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  return KMG_OK;
}

KMG_EXPORT kmg_status kmg_synth_reads_device(kmg_ctx *c, uint64_t seed, uint32_t profile, uint64_t first_read, uint64_t n_reads,
                                             uint8_t *d_seq, uint8_t *d_qual) {
  if (!c) return KMG_ERR_INVALID_ARG;
  if (profile != 3 && profile != 5) return fail(c, KMG_ERR_INVALID_ARG, "profile must be 3 (R20M shape) or 5 (R200M shape)");
  if (n_reads && !d_seq) return fail(c, KMG_ERR_INVALID_ARG, "d_seq is NULL");
  CU(c, cudaSetDevice(c->device));
  CU(c, launch_synth_reads(seed, profile, first_read, n_reads, d_seq, d_qual, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  return KMG_OK;
}
