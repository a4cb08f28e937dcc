// Partitioned pipeline, phases A2 and B (phase A1, the scan-side coarse scatter, lives in kmg_kernels.cu).
//
// Why partition at all: an upsert into one big HBM-resident table is bounded by ~20 G random atomics/s
// on a B200 and moves 144 B of DRAM traffic per k-mer (profiles/r1_summary.md), while HBM streams at
// 6.5 TB/s.  So the keys are radix-partitioned by hash with streaming writes until a partition is so
// small (~3.5 K keys) that ONE CTA can count it in a SHARED-MEMORY table, compact it into the output and
// move on -- no cross-CTA dependencies, no grid barriers, HBM sees only streams.
//
//   A1  scan -> mixed canonical keys -> P1 coarse bins            (partition_scatter_rows2_kernel, kmg_kernels.cu)
//   A2  coarse bin -> P2 sub-bins each (P = P1*P2 fine)           (refine_rows4_kernel: big rows, tiles interleaved over the grid;
//                                                                  refine_rows_kernel: few sub-bins, and keys pulled from other GPUs;
//                                                                  refine_kernel<> = exact route)
//   B   one CTA per fine partition: count, emit, histogram        (count_partitions_sieve_tma_kernel, and _in_place_kernel for one
//                                                                  raw run in the speculative layout: bit-map sieve for raw runs of
//                                                                  mostly distinct keys; count_partitions_smem_kernel: table variant
//                                                                  for weighted / repeat-rich runs; count_partitions_kernel = L2-scratch
//                                                                  fallback)
//
// The streams between the stages hold MIXED keys v = mix64(key) (kmg_device.cuh): coarse bin = top bits of v's high
// half, sub-bin = top bits of its low half, table slot = its lowest bits.  Both scatter levels write into speculative
// fixed shares per bin (mean + 7 sigma), so neither needs a count pass; overflow -> exact route (kmg_api.cu).
// Two levels because a scatter needs runs per (tile, bin) long enough to write whole sectors: with ~900 bins per
// level an 8 K-key tile yields ~9-key runs, while a single level with 860 K bins would not.
//
// Replaces the DashMap upsert + iteration of src/run.rs:565-582 for large inputs; results are the same
// multiset of (canonical key, count) pairs.
#include <algorithm>
#include <atomic>

#include "kmg_device.cuh"
#include "kmg_kernels.h"

namespace kmg {

extern std::atomic<uint64_t> g_launches;

// ---------------------------------------------------------------------------------------------------
// level 1 for keys that are already extracted (receive side of the multi-GPU exchange, weighted inserts)
// ---------------------------------------------------------------------------------------------------
template <bool SCATTER>
__global__ void __launch_bounds__(256) keys_coarse_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ counts,
                                                          uint64_t n, uint32_t n_coarse, unsigned long long *coarse_counts,
                                                          const unsigned long long *coarse_start, unsigned long long *coarse_cursor,
                                                          uint64_t *out_keys, uint64_t *out_counts) {
  extern __shared__ uint32_t sm[];
  uint32_t *hist = sm;  // histogram, then ABSOLUTE output cursors (the atomic's return value is the destination)
  constexpr uint32_t TILE = 16384;
  for (uint32_t p = threadIdx.x; p < n_coarse; p += blockDim.x) hist[p] = 0;
  __syncthreads();
  constexpr int U = 8;  // keys in flight per thread: the loops are otherwise serialised on one global load each
  for (uint64_t t0 = (uint64_t)blockIdx.x * TILE; t0 < n; t0 += (uint64_t)gridDim.x * TILE) {
    const uint32_t m = (uint32_t)(n - t0 < TILE ? n - t0 : TILE);
    for (uint32_t i0 = 0; i0 < m; i0 += U * 256) {
      uint64_t key[U];
#pragma unroll
      for (int j = 0; j < U; ++j) { const uint32_t i = i0 + j * 256 + threadIdx.x; key[j] = i < m ? keys[t0 + i] : EMPTY_KEY; }
#pragma unroll
      for (int j = 0; j < U; ++j) if (i0 + j * 256 + threadIdx.x < m) atomicAdd(hist + coarse_of_mix(mix64(key[j]), n_coarse), 1u);
    }
    if (SCATTER) {
      __syncthreads();
      for (uint32_t p = threadIdx.x; p < n_coarse; p += blockDim.x) {
        const uint32_t c = hist[p];
        hist[p] = c ? (uint32_t)(coarse_start[p] + atomicAdd(coarse_cursor + p, (unsigned long long)c)) : 0u;
      }
      __syncthreads();
      for (uint32_t i0 = 0; i0 < m; i0 += U * 256) {
        uint64_t key[U], cnt[U];
        uint32_t p[U], o[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
          const uint32_t i = i0 + j * 256 + threadIdx.x;
          key[j] = i < m ? keys[t0 + i] : EMPTY_KEY;
          cnt[j] = (i < m && counts) ? counts[t0 + i] : 1ull;
        }
#pragma unroll
        for (int j = 0; j < U; ++j) { key[j] = mix64(key[j]); p[j] = coarse_of_mix(key[j], n_coarse); o[j] = 0; if (i0 + j * 256 + threadIdx.x < m) o[j] = atomicAdd(hist + p[j], 1u); }
#pragma unroll
        for (int j = 0; j < U; ++j)
          if (i0 + j * 256 + threadIdx.x < m) {
            out_keys[o[j]] = key[j];  // the runs carry MIXED keys (kmg_device.cuh)
            if (out_counts) out_counts[o[j]] = cnt[j];
          }
      }
      __syncthreads();
      for (uint32_t p = threadIdx.x; p < n_coarse; p += blockDim.x) hist[p] = 0;
      __syncthreads();
    }
  }
  if (!SCATTER) {
    __syncthreads();
    for (uint32_t p = threadIdx.x; p < n_coarse; p += blockDim.x)
      if (hist[p]) atomicAdd(coarse_counts + p, (unsigned long long)hist[p]);
  }
}

cudaError_t launch_keys_coarse(const uint64_t *d_keys, const uint64_t *d_counts, uint64_t n, uint32_t n_coarse, bool scatter,
                               unsigned long long *coarse_counts, const unsigned long long *coarse_start,
                               unsigned long long *coarse_cursor, uint64_t *out_keys, uint64_t *out_counts, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  const size_t smem = (size_t)n_coarse * sizeof(uint32_t);
  const uint64_t want = (n + 16383) / 16384, cap = (uint64_t)num_sms() * 2;
  const unsigned grid = (unsigned)std::min(want, cap);
  cudaError_t e;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  if (scatter) {
    if ((e = cudaFuncSetAttribute(keys_coarse_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    keys_coarse_kernel<true><<<grid, 256, smem, s>>>(d_keys, d_counts, n, n_coarse, coarse_counts, coarse_start, coarse_cursor, out_keys, out_counts);
  } else {
    if ((e = cudaFuncSetAttribute(keys_coarse_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    keys_coarse_kernel<false><<<grid, 256, smem, s>>>(d_keys, d_counts, n, n_coarse, coarse_counts, coarse_start, coarse_cursor, out_keys, out_counts);
  }
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// level 2: split every coarse partition into n_sub sub-bins.  Work unit = a tile of REFINE_TILE keys that
// lies inside ONE coarse partition (tile_prefix[] maps a global tile number to its partition).
// SCATTER == false: fine_counts[c*n_sub + s] += ...      SCATTER == true: fine_start[] is the exclusive
// prefix of those counts and fine_cursor[] starts at zero.
// ---------------------------------------------------------------------------------------------------
// where sub-bin f of this tile lands in the output: exact layout = counted prefix + running cursor; speculative layout =
// f * fine_cap + running cursor, refused (marker, nothing is written) when the partition's share is exhausted
constexpr uint32_t NO_BASE = 0xffffffffu;
constexpr unsigned long long NO_SPACE = ~0ull;  // phase B: the partition's output reservation did not fit the run (CountParams::out_cap)
__device__ __forceinline__ uint32_t refine_reserve(const RefineParams &P, uint64_t f, uint32_t h) {
  if (!h) return 0u;
  const unsigned long long off = atomicAdd(P.fine_cursor + f, (unsigned long long)h);
  if (P.fine_cap) {
    if (off + h > P.fine_cap) { atomicExch(P.overflow_flag, 1u); return NO_BASE; }
    return (uint32_t)(f * P.fine_cap + off);
  }
  return (uint32_t)(P.fine_start[f] + off);
}

// where input partition c's keys live (RefineParams::src)
__device__ __forceinline__ const uint64_t *refine_keys_of(const RefineParams &P, uint32_t c) {
  return P.n_src ? P.src[c % P.in_group] : P.keys;  // once per tile, never per key
}

// One tile, exact two-pass procedure: histogram -> (count: add to fine_counts | scatter: prefix, one global reservation
// per sub-bin, rank the keys into `staging` in sub-bin order, coalesced copy-out).  hist[] is zero on entry and on exit.
// FILLERS: the input may be a consolidated run (refine_kernel; the rows kernels only see raw runs, which hold no fillers).
template <int THREADS, bool SCATTER, bool FILLERS = false>
__device__ __forceinline__ void refine_tile_two_pass(const RefineParams &P, const uint64_t *__restrict__ kbase, const uint64_t begin, const uint32_t m, const uint64_t f0, const uint32_t sub_base,
                                                     uint64_t *staging, uint64_t *staging_c, uint32_t *hist, uint32_t *s_off,
                                                     uint32_t *g_base, uint32_t *s_scan) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int U = 8;  // keys in flight per thread
  // sub-bin of a mixed key of the tile.  A consolidated run being re-split holds filler entries inside its segments (EMPTY_MIX
  // with count 0: the pad entry of an odd segment, a repeat of the copying sieve); their mix lies in no particular partition, so
  // they stay fillers in the last sub-bin of their own partition instead of indexing past hist[].
  auto bin_of = [&](uint64_t mixed) {
    const uint32_t b = sub_of_mix(mixed, P.sub_total) - sub_base;
    return FILLERS ? min(b, P.n_sub - 1u) : b;
  };
  for (uint32_t i0 = 0; i0 < m; i0 += U * THREADS) {
    uint64_t key[U];
#pragma unroll
    for (int j = 0; j < U; ++j) {
      const uint32_t i = i0 + j * THREADS + tid;
      key[j] = i < m ? (SCATTER ? kbase[begin + i] : __ldcs(kbase + begin + i)) : EMPTY_KEY;
    }
#pragma unroll
    for (int j = 0; j < U; ++j) if (i0 + j * THREADS + tid < m) atomicAdd(hist + bin_of(P.in_keys ? mix64(key[j]) : key[j]), 1u);
  }
  __syncthreads();
  if (!SCATTER) {
    for (uint32_t s = tid; s < P.n_sub; s += THREADS) {
      const uint32_t h = hist[s];
      if (h) { atomicAdd(P.fine_counts + f0 + s, (unsigned long long)h); hist[s] = 0; }
    }
    return;
  }
  // exclusive prefix over the sub-bins (staging offsets) + one global reservation per sub-bin
  const uint32_t per = (P.n_sub + THREADS - 1) / THREADS;
  const uint32_t b0 = min((uint32_t)tid * per, P.n_sub), b1 = min(b0 + per, P.n_sub);
  uint32_t mine = 0;
  for (uint32_t s = b0; s < b1; ++s) mine += hist[s];
  uint32_t incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { uint32_t v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
  if (lane == 31) s_scan[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    uint32_t v = lane < THREADS / 32 ? s_scan[lane] : 0, inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { uint32_t u = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += u; }
    if (lane < THREADS / 32) s_scan[lane] = inc - v;
  }
  __syncthreads();
  uint32_t run = s_scan[warp] + (incl - mine);
  for (uint32_t s = b0; s < b1; ++s) {
    const uint32_t h = hist[s];
    s_off[s] = run;
    g_base[s] = refine_reserve(P, f0 + s, h);
    hist[s] = run;  // becomes the staging cursor
    run += h;
  }
  __syncthreads();
  for (uint32_t i0 = 0; i0 < m; i0 += U * THREADS) {  // second read of the tile comes from L2
    uint64_t key[U], cnt[U];
    uint32_t sb[U], o[U];
#pragma unroll
    for (int j = 0; j < U; ++j) {
      const uint32_t i = i0 + j * THREADS + tid;
      key[j] = i < m ? __ldcs(kbase + begin + i) : EMPTY_KEY;  // last use of this tile
      cnt[j] = (i < m && P.counts) ? __ldcs(P.counts + begin + i) : 1ull;
    }
#pragma unroll
    for (int j = 0; j < U; ++j) { if (P.in_keys) key[j] = mix64(key[j]); sb[j] = bin_of(key[j]); o[j] = 0; if (i0 + j * THREADS + tid < m) o[j] = atomicAdd(hist + sb[j], 1u); }
#pragma unroll
    for (int j = 0; j < U; ++j)
      if (i0 + j * THREADS + tid < m) { staging[o[j]] = key[j]; if (P.counts) staging_c[o[j]] = cnt[j]; }
  }
  __syncthreads();
  for (uint32_t i = tid; i < m; i += THREADS) {  // coalesced copy-out; destination recomputed from the key
    const uint64_t key = staging[i];
    const uint32_t sbin = bin_of(key);  // staged values are mixed keys
    if (g_base[sbin] == NO_BASE) continue;
    const uint64_t dst = (uint64_t)g_base[sbin] + (i - s_off[sbin]);
    P.out_keys[dst] = key;
    if (P.out_counts) P.out_counts[dst] = P.counts ? staging_c[i] : 1ull;
  }
  __syncthreads();
  for (uint32_t s = tid; s < P.n_sub; s += THREADS) hist[s] = 0;
}

// the key range [begin, begin + m) of tile g, which lies in coarse partition c
__device__ __forceinline__ void refine_tile_range(const RefineParams &P, uint32_t g, uint32_t c, uint64_t &begin, uint32_t &m) {
  begin = P.coarse_start[c] + (uint64_t)(g - P.tile_prefix[c]) * REFINE_TILE;
  const uint64_t end_c = P.coarse_len ? P.coarse_start[c] + P.coarse_len[c] : P.coarse_start[c + 1];
  m = (uint32_t)(end_c - begin < (uint64_t)REFINE_TILE ? end_c - begin : (uint64_t)REFINE_TILE);
}

// which coarse partition owns tile g (largest c with tile_prefix[c] <= g), and the tile's key range
__device__ __forceinline__ void refine_locate_tile(const RefineParams &P, uint32_t g, uint32_t *s_c, uint32_t &c, uint64_t &begin, uint32_t &m) {
  if (threadIdx.x == 0) {
    uint32_t lo = 0, hi = P.n_coarse;
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (P.tile_prefix[mid] <= g) lo = mid; else hi = mid; }
    *s_c = lo;
  }
  __syncthreads();
  c = *s_c;
  refine_tile_range(P, g, c, begin, m);
}

// the coarse partition of tile g, searched from `hint` (the partition of the tile located before it): consecutive tiles of a
// CTA mostly share their partition or lie in the next non-empty one
__device__ __forceinline__ uint32_t refine_partition_from(const RefineParams &P, uint32_t g, uint32_t hint) {
  if (P.tile_prefix[hint] > g || hint >= P.n_coarse) hint = 0;
  if (P.tile_prefix[hint + 1] <= g) {  // not in the same or the next non-empty partition: binary search
    uint32_t lo = hint, hi = P.n_coarse;
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (P.tile_prefix[mid] <= g) lo = mid; else hi = mid; }
    hint = lo;
  }
  return hint;
}

template <bool SCATTER>
__global__ void __launch_bounds__(REFINE_THREADS) refine_kernel(RefineParams P) {
  extern __shared__ __align__(16) uint8_t rsm[];
  // count pass: one histogram.  scatter pass (weighted keys): the tile's keys are ranked into a
  // shared-memory staging buffer in sub-bin order and copied out by consecutive lanes (scattered 8-byte stores, one L2
  // transaction each, were 60 % of the unstaged kernels).
  uint64_t *staging = reinterpret_cast<uint64_t *>(rsm);                                // SCATTER only: REFINE_TILE keys
  uint64_t *staging_c = staging + REFINE_TILE;                                          // SCATTER with counts only
  uint32_t *hist = reinterpret_cast<uint32_t *>(rsm + (SCATTER ? (size_t)REFINE_TILE * 8 * (P.counts ? 2 : 1) : 0));
  uint32_t *s_off = hist + P.n_sub, *g_base = s_off + P.n_sub;
  const int tid = threadIdx.x;
  __shared__ uint32_t s_c, s_scan[REFINE_THREADS / 32 + 1];
  for (uint32_t s = tid; s < P.n_sub; s += REFINE_THREADS) hist[s] = 0;
  __syncthreads();
  for (uint32_t g = blockIdx.x; g < P.n_tiles; g += gridDim.x) {
    uint32_t c, m;
    uint64_t begin;
    refine_locate_tile(P, g, &s_c, c, begin, m);
    const uint32_t cb = c / P.in_group;  // coarse bin of input partition c
    refine_tile_two_pass<REFINE_THREADS, SCATTER, true>(P, refine_keys_of(P, c), begin, m, (uint64_t)cb * P.n_sub, (cb % P.sub_old) * P.n_sub, staging, staging_c, hist, s_off, g_base, s_scan);
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------
// level 2 scatter, single pass (unweighted keys -- the scan path): every sub-bin owns a ROW of 2^cap_log2 key slots in
// shared memory.  A key is read once, hashed once, ranked inside its sub-bin by one shared atomic (with return) and
// dropped into its row; the few keys whose row is full (sub-bin sizes are Poisson around 9/16 of the row) go to a
// small overflow list together with their rank.  Then one global reservation per sub-bin and a copy-out in which
// consecutive lanes write consecutive keys of a row.  Compared with histogram + prefix + re-read + re-hash this is
// ~1/3 of the instructions per key (the two-pass kernel was issue bound, profiles/r1_v4_phaseA_lines.txt).
// A tile whose overflow list does not suffice (heavily repeated keys) is redone with the exact two-pass procedure.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(REFINE_ROWS_THREADS, 1) refine_rows_kernel(RefineParams P) {
  extern __shared__ __align__(16) uint8_t rsm[];
  const uint32_t cap = P.row_cap, n_slots = P.n_sub * cap, magic = P.row_magic;  // x / cap == __umulhi(x, magic) for x < 2^16
  uint64_t *rows = reinterpret_cast<uint64_t *>(rsm);  // REFINE_ROWS_SLOTS
  uint64_t *ov_key = rows + REFINE_ROWS_SLOTS;         // REFINE_ROWS_OVERFLOW
  uint32_t *ov_meta = reinterpret_cast<uint32_t *>(ov_key + REFINE_ROWS_OVERFLOW);
  uint32_t *cnt = ov_meta + REFINE_ROWS_OVERFLOW, *s_off = cnt + P.n_sub, *g_base = s_off + P.n_sub;
  __shared__ uint32_t s_c[2], s_ovn, s_scan[REFINE_ROWS_THREADS / 32 + 1];
  const int tid = threadIdx.x;
  constexpr int U = REFINE_TILE / REFINE_ROWS_THREADS;  // the whole tile is in registers: one exposed load latency per tile
  static_assert(U * REFINE_ROWS_THREADS == REFINE_TILE, "tile must be a multiple of the CTA size");
  // a CTA owns a CONTIGUOUS range of tiles, so consecutive tiles mostly share their coarse partition
  const uint32_t per_cta = (P.n_tiles + gridDim.x - 1) / gridDim.x;
  const uint32_t g_begin = blockIdx.x * per_cta, g_end = min(g_begin + per_cta, P.n_tiles);
  if (g_begin >= g_end) return;
  uint32_t c_hint = 0;  // thread 0: coarse partition of the tile located last
  for (uint32_t s = tid; s < P.n_sub; s += REFINE_ROWS_THREADS) cnt[s] = 0;
  if (tid == 0) s_ovn = 0;
  if (tid == 0) s_c[0] = c_hint = refine_partition_from(P, g_begin, c_hint);
  __syncthreads();
  uint32_t c = s_c[0], m;
  uint64_t begin;
  refine_tile_range(P, g_begin, c, begin, m);
  uint64_t key[U];
  {
    const uint64_t *kb = refine_keys_of(P, c) + begin;
#pragma unroll
    for (int j = 0; j < U; ++j) { const uint32_t i = j * REFINE_ROWS_THREADS + tid; key[j] = i < m ? __ldcs(kb + i) : EMPTY_KEY; }
  }

  for (uint32_t g = g_begin; g < g_end; ++g) {
    const uint32_t cb = P.in_group > 1 ? c / P.in_group : c;  // coarse bin of input partition c
    const uint64_t f0 = (uint64_t)cb * P.n_sub;
    const uint32_t sub_base = (cb % P.sub_old) * P.n_sub;
    {  // ---- rank the tile's keys into the rows
      uint32_t sb[U], r[U];
#pragma unroll
      for (int j = 0; j < U; ++j) {
        if (P.in_keys) key[j] = mix64(key[j]);
        sb[j] = sub_of_mix(key[j], P.sub_total) - sub_base;
        r[j] = 0;
        if (j * REFINE_ROWS_THREADS + tid < m) r[j] = atomicAdd(cnt + sb[j], 1u);
      }
#pragma unroll
      for (int j = 0; j < U; ++j) {
        if (j * REFINE_ROWS_THREADS + tid >= m) continue;
        if (r[j] < cap) rows[sb[j] * cap + r[j]] = key[j];
        else {
          const uint32_t o = atomicAdd(&s_ovn, 1u);
          if (o < REFINE_ROWS_OVERFLOW) { ov_key[o] = key[j]; ov_meta[o] = (sb[j] << 16) | r[j]; }  // r < REFINE_TILE <= 65536
        }
      }
    }
    const int nslot = (g - g_begin + 1) & 1;
    if (g + 1 < g_end && tid == 0) s_c[nslot] = c_hint = refine_partition_from(P, g + 1, c_hint);
    __syncthreads();
    const uint32_t n_ov = s_ovn;
    const bool exact = n_ov > REFINE_ROWS_OVERFLOW;  // block-uniform: skewed tile, take the exact route
    if (exact) {
      for (uint32_t s = tid; s < P.n_sub; s += REFINE_ROWS_THREADS) cnt[s] = 0;
      __syncthreads();
      refine_tile_two_pass<REFINE_ROWS_THREADS, true>(P, refine_keys_of(P, c), begin, m, f0, sub_base, rows, nullptr, cnt, s_off, g_base, s_scan);
    } else {
      for (uint32_t s = tid; s < P.n_sub; s += REFINE_ROWS_THREADS) {
        const uint32_t h = cnt[s];
        g_base[s] = refine_reserve(P, f0 + s, h);
        if (g_base[s] == NO_BASE) cnt[s] = 0;  // refused: nothing of this sub-bin is written
      }
    }
    // ---- the next tile's keys are requested now, so their latency hides behind this tile's copy-out
    uint32_t c_next = c, m_next = 0;
    uint64_t begin_next = 0;
    if (g + 1 < g_end) {
      c_next = s_c[nslot];
      refine_tile_range(P, g + 1, c_next, begin_next, m_next);
      const uint64_t *kb = refine_keys_of(P, c_next) + begin_next + tid;
      uint32_t mn = m_next;
      asm volatile("" : "+l"(kb), "+r"(mn));  // pinned in registers: the compiler otherwise re-derives the tile's base (segment tables, source select) for every load
#pragma unroll
      for (int j = 0; j < U; ++j) key[j] = (uint32_t)(j * REFINE_ROWS_THREADS + tid) < mn ? __ldcs(kb + j * REFINE_ROWS_THREADS) : EMPTY_KEY;
    }
    __syncthreads();
    if (!exact) {
      if (cap <= 24u) {  // eight lanes per row, lanes along the row: contiguous destinations, row size / base fetched once per row (see partition_scatter_rows_kernel)
        const uint32_t l = tid & 7u;
#pragma unroll 2
        for (uint32_t s2 = tid >> 3; s2 < P.n_sub; s2 += REFINE_ROWS_THREADS / 8) {
          const uint32_t h = min(cnt[s2], cap);
          uint64_t *dst = P.out_keys + (uint64_t)g_base[s2] + l;
          const uint64_t *row = rows + s2 * cap + l;
          if (l == 0u) cnt[s2] = 0;  // read by all eight lanes in the same instruction: no separate clearing pass + barrier
          if (l < h) dst[0] = row[0];
          if (l + 8u < h) dst[8] = row[8];
          if (h > 16u && l + 16u < h) dst[16] = row[16];
        }
      } else {
#pragma unroll 4
        for (uint32_t x = tid; x < n_slots; x += REFINE_ROWS_THREADS) {  // lanes walk along the rows: contiguous destinations
          const uint32_t s2 = __umulhi(x, magic), e = x - s2 * cap;
          if (e < cnt[s2]) P.out_keys[(uint64_t)g_base[s2] + e] = rows[x];
        }
      }
      for (uint32_t o = tid; o < n_ov; o += REFINE_ROWS_THREADS) {
        const uint32_t meta = ov_meta[o];
        if (g_base[meta >> 16] != NO_BASE) P.out_keys[(uint64_t)g_base[meta >> 16] + (meta & 0xffffu)] = ov_key[o];
      }
      if (cap > 24u) {
        __syncthreads();
        for (uint32_t s = tid; s < P.n_sub; s += REFINE_ROWS_THREADS) cnt[s] = 0;
      }
    }
    if (tid == 0) s_ovn = 0;
    __syncthreads();
    c = c_next; m = m_next; begin = begin_next;
  }
}

// The rows scheme for 128 sub-bins and more when the keys are local (refine_rows_kernel above takes fewer sub-bins and keys pulled
// from other GPUs).  What the measurements on C4 said (profiles/r4_summary.md), in the order they were made:
//   * cutting the instructions per key by a third (32-bit shared-space addresses, predicated stores and copies instead of
//     BSSY / BRA / BSYNC regions that re-derive the shared window per key) changed nothing: 20.0 -> 19.9 ms.  Not issue bound.
//   * TILE ORDER is what mattered: with a contiguous tile range per CTA the grid appends to 148 x 928 output regions at once and
//     DRAM sees line-sized writes all over 4 GB; with the tiles INTERLEAVED over the grid (in chunks of C tile pairs) it works in
//     a handful of coarse bins at a time: 19.9 -> 16.0 ms at C = 1, 14.6 ms at C = 16 (C = 1 makes all CTAs reserve in the same
//     sub-bins at the same instant, C = 64 spreads the writes too far again: 15.7 ms).
//   * the cost per (row, drain) -- one global reservation, a row header, two half-filled sectors at the ends of every run -- is
//     real: two 512-thread CTAs on half tiles (runs of 4.4 keys) 19.8 ms, one CTA draining once per tile (8.8) 16.7 ms, once per
//     TWO tiles (17.7) 16.2 ms (all interleaved, C = 1).  So the rows take all the shared memory there is (28 slots for 928
//     sub-bins, mean fill 0.63, ~0.1 % of the keys overflow to the list) and are drained once per two tiles.
//   * the next group's two tiles are prefetched into L2 a group ahead (one line per thread): the register batches (four keys per
//     thread; the first tile of a group requested before the previous group's copy-out, the second one batch ahead) then wait
//     for L2 instead of DRAM: 16.2 -> 16.0 ms.
constexpr int R4_OVERFLOW = 1024, R4_BATCH = 4096;
constexpr size_t R4_SMEM = 226 * 1024;  // rows + overflow list + three arrays of n_sub words
// the exact route of a skewed tile, out of line: it is rare, and inlined it costs the hot loop its registers
__device__ __noinline__ void refine_tile_exact_1024(const RefineParams P, const uint64_t *kbase, uint64_t begin, uint32_t m, uint64_t f0, uint32_t sub_base,
                                                    uint64_t *staging, uint32_t *hist, uint32_t *s_off, uint32_t *g_base, uint32_t *s_scan) {
  refine_tile_two_pass<REFINE_ROWS_THREADS, true>(P, kbase, begin, m, f0, sub_base, staging, nullptr, hist, s_off, g_base, s_scan);
}
__host__ __device__ inline double rows_overflow_fraction(double mean, uint32_t cap) {  // E[(X - cap)+] / mean, X ~ Poisson(mean)
  double p = exp(-mean), s = 0.0;
  for (uint32_t k = 0; k <= cap; ++k) { s += (double)(cap - k) * p; p *= mean / (double)(k + 1); }
  return (mean - (double)cap + s) / mean;
}
template <bool IN_KEYS>
__global__ void __launch_bounds__(REFINE_ROWS_THREADS, 1) refine_rows4_kernel(RefineParams P, uint32_t tiles_per_group, uint32_t n_slots) {
  extern __shared__ __align__(16) uint8_t rsm[];
  const uint32_t cap = P.row_cap;
  uint64_t *rows = reinterpret_cast<uint64_t *>(rsm);  // n_slots >= n_sub * cap
  uint64_t *ov_key = rows + n_slots;                    // R4_OVERFLOW
  uint32_t *ov_meta = reinterpret_cast<uint32_t *>(ov_key + R4_OVERFLOW);
  uint32_t *cnt = ov_meta + R4_OVERFLOW, *s_off = cnt + P.n_sub, *g_base = s_off + P.n_sub;
  const uint32_t rows_s = smem_u32(rows), cnt_s = smem_u32(cnt), gb_s = smem_u32(g_base);
  __shared__ uint32_t s_c[2], s_ovn, s_scan[REFINE_ROWS_THREADS / 32 + 1];
  const int tid = threadIdx.x;
  constexpr int T = REFINE_ROWS_THREADS, U = R4_BATCH / T;  // 4 keys per thread and batch
  static_assert(2 * R4_BATCH == REFINE_TILE, "a host-side tile is two batches");
  // tile order: P.pad = C > 0 -> INTERLEAVED in chunks of C tile pairs (pair q holds tiles 2q, 2q + 1; CTA b takes pairs
  // [b*C, b*C + C) of every block of gridDim * C pairs): the whole grid works in a handful of coarse bins and appends to the same
  // few thousand output regions at a time, which is what DRAM wants (C4, A2: 20.0 ms with contiguous ranges, 16.7 ms interleaved);
  // C > 1 keeps the CTAs from reserving in the same sub-bins at the same instant.  P.pad = 0 (a contiguous range of tiles per CTA)
  // is never launched: launch_refine sets C >= 1.  The branches for it stay because the kernel compiled without them measured
  // slower on a B200 (A2 +0.6 % on C4, +2 % on C1: the register allocation of the whole loop changes).
  const uint32_t C = P.pad;
  const bool il = C != 0;
  uint32_t pi = 0;  // interleaved: this CTA's pair counter
  auto pair_of = [&](uint32_t i) { return (i / C) * (gridDim.x * C) + blockIdx.x * C + (i % C); };
  const uint32_t per_cta = (P.n_tiles + gridDim.x - 1) / gridDim.x;
  const uint32_t g_begin = il ? 2u * pair_of(0) : blockIdx.x * per_cta, g_end = il ? P.n_tiles : min(g_begin + per_cta, P.n_tiles);
  if (g_begin >= g_end) return;
  uint32_t c_hint = 0;  // thread 0: coarse partition of the tile located last
  // batch `half` (0 / 1) of the tile whose keys start at kb and which holds m keys
  auto load_batch = [&](uint64_t (&k)[U], const uint64_t *kb, uint32_t m, uint32_t half) {
    const uint64_t *p = kb + half * R4_BATCH + tid;
    uint32_t left = m > half * R4_BATCH ? m - half * R4_BATCH : 0u;
    asm volatile("" : "+l"(p), "+r"(left));  // pinned in registers: the compiler otherwise re-derives the tile's base for every load
#pragma unroll
    for (int j = 0; j < U; ++j) k[j] = (uint32_t)(j * T + tid) < left ? __ldcs(p + j * T) : EMPTY_KEY;
  };
  uint32_t sub_base = 0;
  auto rank_batch = [&](uint64_t (&k)[U], uint32_t m, uint32_t half) {
    const uint32_t left = m > half * R4_BATCH ? m - half * R4_BATCH : 0u;  // block-uniform
    uint32_t sb[U], r[U], over = 0;
    if (left >= (uint32_t)R4_BATCH) {  // a full batch needs no bounds tests
#pragma unroll
      for (int j = 0; j < U; ++j) {
        if (IN_KEYS) k[j] = mix64(k[j]);
        sb[j] = sub_of_mix(k[j], P.sub_total) - sub_base;
        r[j] = atoms_add(cnt_s + 4u * sb[j], 1u);
      }
#pragma unroll
      for (int j = 0; j < U; ++j) {
        const bool fit = r[j] < cap;
        sts64_if(fit, rows_s + 8u * (sb[j] * cap + r[j]), k[j]);
        over |= (fit ? 0u : 1u) << j;
      }
    } else if (left) {
#pragma unroll
      for (int j = 0; j < U; ++j) {
        const bool live = (uint32_t)(j * T + tid) < left;
        if (IN_KEYS) k[j] = mix64(k[j]);
        sb[j] = live ? sub_of_mix(k[j], P.sub_total) - sub_base : 0u;
        r[j] = live ? atoms_add(cnt_s + 4u * sb[j], 1u) : 0u;
      }
#pragma unroll
      for (int j = 0; j < U; ++j) {
        const bool live = (uint32_t)(j * T + tid) < left, fit = r[j] < cap;
        sts64_if(live && fit, rows_s + 8u * (sb[j] * cap + r[j]), k[j]);
        over |= ((live && !fit) ? 1u : 0u) << j;
      }
    }
    if (over) {  // this thread holds keys whose row was full
#pragma unroll
      for (int j = 0; j < U; ++j) {
        if (!((over >> j) & 1u)) continue;
        const uint32_t o = atomicAdd(&s_ovn, 1u);
        if (o < (uint32_t)R4_OVERFLOW) { ov_key[o] = k[j]; ov_meta[o] = (sb[j] << 16) | r[j]; }  // r < 2 * REFINE_TILE <= 65536
      }
    }
  };
  for (uint32_t s = tid; s < P.n_sub; s += T) cnt[s] = 0;
  if (tid == 0) s_ovn = 0;
  if (tid == 0) s_c[0] = c_hint = refine_partition_from(P, g_begin, c_hint);
  __syncthreads();
  uint32_t c = s_c[0], m;
  uint64_t begin;
  refine_tile_range(P, g_begin, c, begin, m);
  uint64_t kA[U], kB[U];
  load_batch(kA, refine_keys_of(P, c) + begin, m, 0);
  load_batch(kB, refine_keys_of(P, c) + begin, m, 1);
  int slot = 0;
  for (uint32_t g = g_begin; g < g_end;) {
    const uint32_t cb = P.in_group > 1 ? c / P.in_group : c;  // coarse bin of input partition c
    const uint64_t f0 = (uint64_t)cb * P.n_sub;
    sub_base = (cb % P.sub_old) * P.n_sub;
    // the group: this tile and, when it lies in the same partition (and in this CTA's range), the next one
    const bool two = tiles_per_group > 1u && g + 1 < g_end && P.tile_prefix[c + 1] > g + 1 && !(il && (g & 1u));
    uint64_t begin2 = 0;
    uint32_t m2 = 0;
    const uint64_t *kbase = refine_keys_of(P, c);
    if (two) refine_tile_range(P, g + 1, c, begin2, m2);
    if (!P.n_src) {  // L2 prefetch of this CTA's NEXT group (one 128-byte line per thread = two tiles), assuming it lies in the same
                     // partition (it does for all but one group in ~200): its loads then wait for L2, not for DRAM
      const uint64_t end_c = P.coarse_len ? P.coarse_start[c] + P.coarse_len[c] : P.coarse_start[c + 1];
      const uint64_t pf = begin + (uint64_t)(il ? 2u * pair_of(pi + 1) - g : 2u) * REFINE_TILE + (uint64_t)tid * 16u;
      if (pf < end_c) asm volatile("prefetch.global.L2 [%0];" ::"l"(kbase + pf));
    }
    {  // one code instance per register batch (merged call sites would force the batches into local memory)
      uint32_t mt = m;
      for (uint32_t t = 0, nt = two ? 2u : 1u; t < nt; ++t) {
        rank_batch(kA, mt, 0);
        if (t + 1 < nt) load_batch(kA, kbase + begin2, m2, 0);
        rank_batch(kB, mt, 1);
        if (t + 1 < nt) load_batch(kB, kbase + begin2, m2, 1);
        mt = m2;
      }
    }
    // interleaved: a pair that straddles two partitions is two groups of one tile; then on to this CTA's next pair
    uint32_t g_next = g + (two ? 2u : 1u);
    if (il && ((g & 1u) || two || g + 1 >= g_end)) g_next = 2u * pair_of(++pi);
    slot ^= 1;
    if (g_next < g_end && tid == 0) s_c[slot] = c_hint = refine_partition_from(P, g_next, c_hint);
    __syncthreads();
    const uint32_t n_ov = s_ovn;
    const bool exact = n_ov > (uint32_t)R4_OVERFLOW;  // block-uniform: skewed group, take the exact route tile by tile
    if (exact) {
      for (uint32_t s = tid; s < P.n_sub; s += T) cnt[s] = 0;
      __syncthreads();
      refine_tile_exact_1024(P, kbase, begin, m, f0, sub_base, rows, cnt, s_off, g_base, s_scan);
      if (two) {
        __syncthreads();
        refine_tile_exact_1024(P, kbase, begin2, m2, f0, sub_base, rows, cnt, s_off, g_base, s_scan);
      }
    } else {
      for (uint32_t s = tid; s < P.n_sub; s += T) {
        const uint32_t h = cnt[s];
        g_base[s] = refine_reserve(P, f0 + s, h);
        if (g_base[s] == NO_BASE) cnt[s] = 0;  // refused: nothing of this sub-bin is written
      }
    }
    // ---- the next group's first tile is requested now, so its latency hides behind this group's copy-out
    uint32_t c_next = c, m_next = 0;
    uint64_t begin_next = 0;
    if (g_next < g_end) {
      c_next = s_c[slot];
      refine_tile_range(P, g_next, c_next, begin_next, m_next);
      const uint64_t *kb = refine_keys_of(P, c_next) + begin_next;
      load_batch(kA, kb, m_next, 0);
      load_batch(kB, kb, m_next, 1);
    }
    __syncthreads();
    if (!exact) {
      const uint32_t l = tid & 7u;  // eight lanes per row, lanes along the row
#pragma unroll 1
      for (uint32_t s2 = tid >> 3; s2 < P.n_sub; s2 += T / 8) {
        const uint32_t h = min(lds32(cnt_s + 4u * s2), cap);
        uint64_t *dst = P.out_keys + (uint64_t)lds32(gb_s + 4u * s2) + l;
        const uint32_t row = rows_s + 8u * (s2 * cap + l);
        sts32_if(l == 0u, cnt_s + 4u * s2, 0u);  // read by all eight lanes in the same instruction: the row is handed back clean
        copy64_if_lt<false>(l, h, dst, row);
        copy64_if_lt<false>(l + 8u, h, dst + 8, row + 64u);
        copy64_if_lt<false>(l + 16u, h, dst + 16, row + 128u);
        for (uint32_t e = 24u; e < h; e += 8u) copy64_if_lt<false>(l + e, h, dst + e, row + 8u * e);  // rows of more than 24 slots
      }
      for (uint32_t o = tid; o < n_ov; o += T) {
        const uint32_t meta = ov_meta[o];
        if (g_base[meta >> 16] != NO_BASE) P.out_keys[(uint64_t)g_base[meta >> 16] + (meta & 0xffffu)] = ov_key[o];
      }
    }
    if (tid == 0) s_ovn = 0;
    __syncthreads();
    g = g_next; c = c_next; m = m_next; begin = begin_next;
  }
}

bool refine_single_pass_available(uint32_t n_sub, bool weighted) { return !weighted && n_sub <= REFINE_ROWS_SLOTS / 8; }

__global__ void fill_strided_kernel(uint64_t *d, uint64_t n, uint64_t stride) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) d[i] = i * stride;
}
cudaError_t launch_fill_strided(uint64_t *d, uint64_t n, uint64_t stride, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  fill_strided_kernel<<<(unsigned)std::min<uint64_t>((n + 255) / 256, (uint64_t)num_sms() * 8), 256, 0, s>>>(d, n, stride);
  return cudaGetLastError();
}

cudaError_t launch_refine(const RefineParams &P_in, bool scatter, cudaStream_t s) {
  if (P_in.n_tiles == 0) return cudaSuccess;
  RefineParams P = P_in;
  if (!P.sub_total) { P.sub_total = P.n_sub; P.sub_old = 1; }  // plain refinement of coarse bins
  if (!P.in_group) P.in_group = 1;
  cudaError_t e;
  if (scatter && refine_single_pass_available(P.n_sub, P.counts || P.out_counts)) {
    P.row_cap = std::min<uint32_t>((uint32_t)REFINE_ROWS_SLOTS / P.n_sub, REFINE_TILE);  // mean fill 8192 / (n_sub * cap) ~ 0.5
    P.row_magic = (uint32_t)(((1ull << 32) + P.row_cap - 1) / P.row_cap);
    const size_t smem = (size_t)REFINE_ROWS_SLOTS * 8 + (size_t)REFINE_ROWS_OVERFLOW * 12 + 3 * (size_t)P.n_sub * sizeof(uint32_t);
    // big rows, drained once per two tiles, tiles interleaved over the grid -- for LOCAL keys.  When the keys are pulled from other
    // GPUs (n_src) the round-3 kernel stays: measured on two GPUs (profiles/r4_summary.md) it pulls and refines a step's keys in
    // 10.4 ms against 12.4 ms (13.7 ms with one tile per drain): NVLink, not the drain pattern, sets its pace.
    if (P.n_sub >= 128u && P.n_src == 0) {
      const uint32_t n_slots = (uint32_t)((R4_SMEM - (size_t)R4_OVERFLOW * 12 - 3 * (size_t)P.n_sub * sizeof(uint32_t)) / 8) & ~1u;
      P.row_cap = n_slots / P.n_sub;
      const uint32_t tg = rows_overflow_fraction(2.0 * REFINE_TILE / P.n_sub, P.row_cap) <= 0.035 ? 2u : 1u;  // two tiles per drain unless the rows would overflow too often
      const size_t smem4 = (size_t)n_slots * 8 + (size_t)R4_OVERFLOW * 12 + 3 * (size_t)P.n_sub * sizeof(uint32_t);
      const unsigned grid = (unsigned)std::min<uint64_t>(P.n_tiles, (uint64_t)num_sms());
      // chunk of the interleaved tile order: 16 pairs, less when the input is so small that some CTAs would get nothing
      P.pad = 16;
      while (P.pad > 1 && (uint64_t)grid * P.pad * 8 > P.n_tiles) P.pad >>= 1;
      auto kern = P.in_keys ? refine_rows4_kernel<true> : refine_rows4_kernel<false>;
      if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4)) != cudaSuccess) return e;
      g_launches.fetch_add(1, std::memory_order_relaxed);
      kern<<<grid, REFINE_ROWS_THREADS, smem4, s>>>(P, tg, n_slots);
      return cudaGetLastError();
    }
    if ((e = cudaFuncSetAttribute(refine_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    refine_rows_kernel<<<(unsigned)std::min<uint64_t>(P.n_tiles, (uint64_t)num_sms()), REFINE_ROWS_THREADS, smem, s>>>(P);
    return cudaGetLastError();
  }
  const size_t smem = scatter ? (size_t)REFINE_TILE * 8 * (P.counts ? 2 : 1) + 3 * (size_t)P.n_sub * sizeof(uint32_t) : (size_t)P.n_sub * sizeof(uint32_t);
  const unsigned grid = (unsigned)std::min<uint64_t>(P.n_tiles, (uint64_t)num_sms() * ((scatter && smem > 110 * 1024) ? 1 : 2));
  g_launches.fetch_add(1, std::memory_order_relaxed);
  if (scatter) {
    if ((e = cudaFuncSetAttribute(refine_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    refine_kernel<true><<<grid, REFINE_THREADS, smem, s>>>(P);
  } else {
    if ((e = cudaFuncSetAttribute(refine_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    refine_kernel<false><<<grid, REFINE_THREADS, smem, s>>>(P);
  }
  return cudaGetLastError();
}

// per-partition totals over all input runs (for load-balanced ordering on the host)
__global__ void sum_lens_kernel(CountParams P, unsigned long long *totals, unsigned long long *max_total) {
  unsigned long long mx = 0;
  for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < P.n_parts; p += gridDim.x * blockDim.x) {
    unsigned long long t = 0;
    for (uint32_t r = 0; r < P.R; ++r) t += P.runs[r].seg_len[p];
    totals[p] = t;
    mx = t > mx ? t : mx;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { const unsigned long long v = __shfl_xor_sync(0xffffffffu, mx, o); mx = v > mx ? v : mx; }
  if ((threadIdx.x & 31) == 0 && mx) atomicMax(max_total, mx);
}
// d_max (zeroed by this call) receives the largest per-partition total: the host only fetches the whole table when some
// partition is heavy enough to need the largest-first processing order
cudaError_t launch_sum_lens(const CountParams &P, unsigned long long *d_totals, unsigned long long *d_max, cudaStream_t s) {
  cudaError_t e = cudaMemsetAsync(d_max, 0, sizeof(unsigned long long), s);
  if (e != cudaSuccess) return e;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  sum_lens_kernel<<<(unsigned)std::min<uint64_t>((P.n_parts + 255) / 256, (uint64_t)num_sms() * 8), 256, 0, s>>>(P, d_totals, d_max);
  return cudaGetLastError();
}

// Count-of-counts while compacting (src/histogram.rs:88-116 computes it from the finished map; here it falls out
// of phase B for free).  Must be called by all 32 lanes together.  Counts of 1 -- the bulk on most inputs -- are
// not recorded at all: hist[1] = distinct - everything else.  Equal counts within the warp are merged first, so
// a popular count value costs one atomic per warp; the lowest bins live in shared memory until the CTA retires.
__device__ __forceinline__ void hist_note(bool ok, unsigned long long cnt, uint32_t *s_hist, const CountParams &P, int lane) {
  const bool agg = ok && cnt > 1 && cnt < (unsigned long long)HIST_DENSE_BINS;
  uint32_t pending = __ballot_sync(0xffffffffu, agg);
  while (pending) {
    const int leader = __ffs(pending) - 1;
    const uint32_t v = __shfl_sync(0xffffffffu, (uint32_t)cnt, leader);
    const uint32_t same = __ballot_sync(0xffffffffu, agg && (uint32_t)cnt == v);
    if (lane == leader) {
      if (v < (uint32_t)HIST_CTA_BINS) atomicAdd(&s_hist[v], (uint32_t)__popc(same));
      else atomicAdd(P.hist + v, (unsigned long long)__popc(same));
    }
    pending &= ~same;
  }
  if (ok && cnt >= (unsigned long long)HIST_DENSE_BINS) {
    const unsigned long long o = atomicAdd(P.hist + HIST_DENSE_BINS, 1ull);
    if (o < P.hist_overflow_cap) P.hist_overflow[o] = cnt;
  }
}
__device__ __forceinline__ void hist_flush(const uint32_t *s_hist, const CountParams &P, int tid) {
  if (tid < HIST_CTA_BINS && s_hist[tid]) atomicAdd(P.hist + tid, (unsigned long long)s_hist[tid]);
}

// ---------------------------------------------------------------------------------------------------
// phase B: one CTA counts one fine partition at a time in its private scratch table (L2-resident: the whole
// grid's scratch is ~39 MB), then compacts it into the output run and hands the slots back clean.
// Slots are (key, occurrences-1): a new key costs one CAS, duplicates one more RED.
// The table cannot overflow by construction (capacity >= 1.6 x the partition's ENTRIES when small, and for
// oversized -- i.e. high-multiplicity -- partitions the number of DISTINCT keys is bounded by the hash-uniform
// share of a partition); should that bound ever be violated the kernel raises error_flag and the host retries
// with larger scratch tables.  Nothing is dropped silently.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(COUNT_THREADS, COUNT_CTAS_PER_SM) count_partitions_kernel(CountParams P) {
  __shared__ uint64_t seg_begin[CONS_MAX_RUNS];
  __shared__ uint64_t seg_prefix[CONS_MAX_RUNS + 1];
  __shared__ uint32_t s_work, s_warp[COUNT_THREADS / 32 + 1], s_hist[HIST_CTA_BINS];
  __shared__ unsigned long long s_base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < HIST_CTA_BINS) s_hist[tid] = 0;
  unsigned long long *table = reinterpret_cast<unsigned long long *>(P.scratch) + (uint64_t)blockIdx.x * (2ull << P.scratch_log2);
  uint32_t next_work = 0;
  if (tid == 0) next_work = atomicAdd(P.next, 1u);

  for (;;) {
    // ---- fetch a partition (the next one is drawn early so the atomic's latency hides behind this one's work)
    if (warp == 0) {
      uint32_t w = 0;
      if (lane == 0) { w = next_work; if (w < P.n_parts) next_work = atomicAdd(P.next, 1u); }
      w = __shfl_sync(0xffffffffu, w, 0);
      if (w < P.n_parts) {
        const uint32_t p = P.order ? P.order[w] : w;
        uint64_t b = 0, len = 0;
        if (lane < (int)P.R) { b = P.runs[lane].seg_start[p]; len = P.runs[lane].seg_len[p]; }
        uint64_t incl = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { uint64_t v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
        if (lane < (int)P.R) { seg_begin[lane] = b; seg_prefix[lane] = incl - len; }
        if (lane == (int)P.R - 1) seg_prefix[P.R] = incl;
      }
      if (lane == 0) s_work = w;
    }
    __syncthreads();
    const uint32_t work = s_work;
    if (work >= P.n_parts) break;
    const uint32_t p = P.order ? P.order[work] : work;
    const uint64_t n_p = seg_prefix[P.R];
    if (n_p == 0) {  // block-uniform
      if (tid == 0) { P.out_seg_start[p] = 0; P.out_seg_len[p] = 0; }
      __syncthreads();
      continue;
    }
    // capacity: 1.6x the entries, at least 256 slots, at most the scratch table
    uint32_t cap_log2 = 8;
    while (cap_log2 < P.scratch_log2 && (1ull << cap_log2) * 5 < n_p * 8) ++cap_log2;
    const uint64_t mask = (1ull << cap_log2) - 1;

    // ---- upsert all entries of partition p
    constexpr int G = 4;
    uint32_t new_keys = 0;
    uint32_t r = 0;  // run holding the thread's current entry: entries are visited in ascending order
#pragma unroll 1
    for (uint64_t base = 0; base < n_p; base += (uint64_t)COUNT_THREADS * G) {
      uint64_t key[G], w[G], slot[G], cur[G];
#pragma unroll
      for (int j = 0; j < G; ++j) {
        const uint64_t idx = base + (uint64_t)j * COUNT_THREADS + tid;
        w[j] = 0; key[j] = EMPTY_MIX;
        if (idx < n_p) {
          while (r + 1 < P.R && idx >= seg_prefix[r + 1]) ++r;
          const uint64_t src = seg_begin[r] + (idx - seg_prefix[r]);
          key[j] = __ldcs(P.runs[r].keys + src);
          w[j] = P.runs[r].counts ? __ldcs(P.runs[r].counts + src) : 1ull;
        }
      }
      if (P.preagg) {
        // Warp run-length pre-aggregation: the scatter passes keep the keys of consecutive windows close together,
        // so homopolymer / tandem-repeat runs tend to arrive as runs of equal keys in adjacent lanes.  The head lane
        // of each run upserts once with the run length; this bounds same-address atomic bursts on skewed inputs.
#pragma unroll
        for (int j = 0; j < G; ++j) {
          const uint64_t kk = w[j] ? key[j] : EMPTY_MIX;
          const uint64_t kp = __shfl_up_sync(0xffffffffu, kk, 1);
          const bool head = lane == 0 || kp != kk;
          const uint32_t heads = __ballot_sync(0xffffffffu, head);
          if (__all_sync(0xffffffffu, w[j] <= 1ull)) {  // unit weights only (keys-runs); pair-runs are distinct per run
            const uint32_t above = lane == 31 ? 0u : heads & ~((2u << lane) - 1u);
            const uint32_t end = above ? (uint32_t)__ffs(above) - 1u : 32u;
            if (w[j]) w[j] = head ? (uint64_t)(end - lane) : 0ull;
          }
        }
      }
      uint32_t pend = 0;
#pragma unroll
      for (int j = 0; j < G; ++j) {  // first probes of all G keys in flight together
        slot[j] = key[j] & mask;  // the stored values ARE the mixes: lowest bits here, coarse / sub-bin used the top bits of each half
        cur[j] = 0;
        if (w[j]) cur[j] = atomicCAS(table + 2 * slot[j], EMPTY_MIX, key[j]);
      }
#pragma unroll
      for (int j = 0; j < G; ++j) {
        if (!w[j]) continue;
        if (cur[j] == EMPTY_MIX) { ++new_keys; if (w[j] > 1) atomicAdd(table + 2 * slot[j] + 1, (unsigned long long)(w[j] - 1)); }
        else if (cur[j] == key[j]) atomicAdd(table + 2 * slot[j] + 1, (unsigned long long)w[j]);
        else pend |= 1u << j;
      }
      uint64_t tries = 0;
      while (pend) {  // linear probing; all still-pending keys of the thread advance together (keeps MLP)
        if (++tries > mask) { atomicExch(P.error_flag, 1u); break; }
#pragma unroll
        for (int j = 0; j < G; ++j)
          if (pend >> j & 1u) { slot[j] = (slot[j] + 1) & mask; cur[j] = *reinterpret_cast<volatile unsigned long long *>(table + 2 * slot[j]); }
#pragma unroll
        for (int j = 0; j < G; ++j)
          if ((pend >> j & 1u) && cur[j] == EMPTY_MIX) cur[j] = atomicCAS(table + 2 * slot[j], EMPTY_MIX, key[j]);
#pragma unroll
        for (int j = 0; j < G; ++j) {
          if (!(pend >> j & 1u)) continue;
          if (cur[j] == EMPTY_MIX) { ++new_keys; if (w[j] > 1) atomicAdd(table + 2 * slot[j] + 1, (unsigned long long)(w[j] - 1)); pend &= ~(1u << j); }
          else if (cur[j] == key[j]) { atomicAdd(table + 2 * slot[j] + 1, (unsigned long long)w[j]); pend &= ~(1u << j); }
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) new_keys += __shfl_xor_sync(0xffffffffu, new_keys, o);
    if (lane == 0) s_warp[warp] = new_keys;
    __threadfence_block();
    __syncthreads();  // all upserts of this CTA are done (they are L2 atomics issued by this CTA only)
    if (tid == 0) {
      uint32_t d = 0;
      for (int w2 = 0; w2 < COUNT_THREADS / 32; ++w2) d += s_warp[w2];
      unsigned long long b = atomicAdd(P.out_cursor, (unsigned long long)d);  // the partition's contiguous output range
      if (b + d > P.out_cap) { atomicExch(P.nospace_flag, 1u); b = NO_SPACE; }
      P.out_seg_start[p] = b; P.out_seg_len[p] = d;
      if (d) atomicAdd(P.out_distinct, (unsigned long long)d);
      s_base = b;
    }
    __syncthreads();

    // ---- compact the table into the output run and clean it
    const unsigned long long out0 = s_base;
    const bool fits = out0 != NO_SPACE;
    uint32_t mine = 0;
    for (uint64_t i = tid; i <= mask; i += COUNT_THREADS) mine += __ldcg(table + 2 * i) != EMPTY_MIX;
    uint32_t incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { uint32_t v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      uint32_t v = lane < COUNT_THREADS / 32 ? s_warp[lane] : 0, inc = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { uint32_t u = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += u; }
      if (lane < COUNT_THREADS / 32) s_warp[lane] = inc - v;
    }
    __syncthreads();
    uint64_t o = out0 + s_warp[warp] + (incl - mine);
    const ulonglong2 *tab2 = reinterpret_cast<const ulonglong2 *>(table);
    for (uint64_t i = tid; i <= mask; i += COUNT_THREADS) {  // trip count is warp-uniform (mask + 1 is a multiple of 256)
      const ulonglong2 sl = __ldcg(tab2 + i);
      const bool used = sl.x != EMPTY_MIX;
      if (used) {
        if (fits) {
          __stcs(P.out_keys + o, sl.x);
          __stcs(P.out_counts + o, sl.y + 1);  // slots store occurrences - 1
        }
        ++o;
        reinterpret_cast<ulonglong2 *>(table)[i] = make_ulonglong2(EMPTY_MIX, 0ull);
      }
      if (P.hist) hist_note(used, sl.y + 1, s_hist, P, lane);
    }
    __syncthreads();  // table clean (same-CTA visibility) before the next partition's upserts
  }
  if (P.hist) hist_flush(s_hist, P, tid);
}


// ---------------------------------------------------------------------------------------------------
// phase B, primary variant: the partition's table lives in SHARED memory.  The kernel is instruction-issue
// bound (profiles/), so everything here is about warp-instructions per key:
//  * layout: SoA, 8192 x u64 keys + 8192 x u32 (occurrences - 1) + 8192 x u16 claimed-slot lists = 112 KiB, so
//    TWO 512-thread CTAs fit per SM and one CTA's bubbles (metadata, key loads, output reservation) overlap
//    with the other's work;
//  * a key's home is a BUCKET of two adjacent slots read with one 16-byte load; all first probes of a batch
//    of 8 keys per thread are issued together (4 at a time in flight);
//  * the few keys whose bucket is taken are then finished lane by lane (no warp-wide rendezvous per key), walking
//    further buckets with an odd stride taken from the high mix bits (double hashing: short chains);
//  * every warp lists the slots IT claimed (ballot + popc, no atomics); compaction walks those lists, so it
//    touches only occupied slots, writes coalesced output and leaves the table clean;
//  * WEIGHTED = false (no input run carries counts, no oversized partition): no per-key weights in registers.
// If a partition holds more distinct keys than the table, a warp claims more than its list holds, or a count does
// not fit 32 bits, error_flag is raised and the host re-runs phase B with the L2-scratch variant.
// ---------------------------------------------------------------------------------------------------
//  * DIRECT (unweighted runs of mostly distinct keys, e.g. a genome: no oversized partitions): no compaction pass at all.  The
//    partition's output range is reserved for all its entries when its segment table is fetched; a key that claims a fresh slot
//    is written to the output right away with count 1 -- positions from ballots taken in the converged code after the two probe
//    rounds, so consecutive lanes write consecutive entries -- and remembers its output index in the slot (u16, where the other
//    variant keeps its slot lists).  Duplicates only bump the slot's counter; after the partition a sweep over the table patches
//    the few entries whose counter is non-zero, feeds the count-of-counts, and cleans the slots.  The unused tail of the
//    reservation (one entry per duplicate) is filled with (EMPTY, 0) entries that every reader skips.
template <bool WEIGHTED, bool DIRECT = false>
__global__ void __launch_bounds__(SMEM_COUNT_THREADS, 2) count_partitions_smem_kernel(CountParams P) {
  static_assert(!(WEIGHTED && DIRECT), "the direct variant counts unweighted keys");
  extern __shared__ __align__(16) unsigned long long skeys[];
  constexpr uint32_t SLOTS = SMEM_TABLE_SLOTS;
  constexpr int NW = SMEM_COUNT_THREADS / 32;
  constexpr uint32_t WLIST = SLOTS / NW;  // claimed-slot list entries per warp
  uint32_t *scnt = reinterpret_cast<uint32_t *>(skeys + SLOTS);
  uint16_t *slist = reinterpret_cast<uint16_t *>(scnt + SLOTS);  // DIRECT: sidx[slot] = output index of the slot's key
  __shared__ uint64_t seg_begin[CONS_MAX_RUNS];
  __shared__ uint64_t seg_prefix[CONS_MAX_RUNS + 1];
  __shared__ uint32_t s_work, s_hist[HIST_CTA_BINS], s_wn[NW];
  __shared__ unsigned long long s_base;
  __shared__ uint32_t s_run;  // entries of the current partition already written (multi-pass partitions)
  __shared__ uint32_t s_emit; // DIRECT: entries of the current partition written so far
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint16_t *wlist = slist + warp * WLIST;
  if (tid < HIST_CTA_BINS) s_hist[tid] = 0;
  for (uint32_t i = tid; i < SLOTS; i += SMEM_COUNT_THREADS) { skeys[i] = EMPTY_MIX; scnt[i] = 0; }
  uint32_t next_work = 0;
  if (tid == 0) next_work = atomicAdd(P.next, 1u);
  if (tid < NW) s_wn[tid] = 0;
  __syncthreads();

  for (;;) {
    if (warp == 0) {
      uint32_t w = 0;
      if (lane == 0) { w = next_work; if (w < P.n_parts) next_work = atomicAdd(P.next, 1u); }
      w = __shfl_sync(0xffffffffu, w, 0);
      if (w < P.n_parts) {
        const uint32_t p = P.order ? P.order[w] : w;
        uint64_t b = 0, len = 0;
        if (lane < (int)P.R) { b = P.runs[lane].seg_start[p]; len = P.runs[lane].seg_len[p]; }
        uint64_t incl = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { uint64_t v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
        if (lane < (int)P.R) { seg_begin[lane] = b; seg_prefix[lane] = incl - len; }
        if (lane == (int)P.R - 1) {
          seg_prefix[P.R] = incl;
          if (DIRECT) {  // the output range for ALL entries of the partition, reserved while the others still wait at the barrier
            unsigned long long ob = 0;
            if (incl) { ob = atomicAdd(P.out_cursor, (unsigned long long)incl); if (ob + incl > P.out_cap) { atomicExch(P.nospace_flag, 1u); ob = NO_SPACE; } }
            s_base = ob; s_emit = 0;
          }
        }
      }
      if (lane == 0) s_work = w;
    }
    __syncthreads();
    const uint32_t work = s_work;
    if (work >= P.n_parts) break;
    const uint32_t p = P.order ? P.order[work] : work;
    const uint64_t n_p = seg_prefix[P.R];
    if (n_p == 0) {
      if (tid == 0) { P.out_seg_start[p] = 0; P.out_seg_len[p] = 0; }
      __syncthreads();
      continue;
    }
    uint32_t cap_log2 = 8;  // small partitions use a prefix of the table
    while ((1u << cap_log2) < SLOTS && (1ull << cap_log2) * 5 < n_p * 8) ++cap_log2;
    const uint32_t mask = (1u << cap_log2) - 1, bmask = mask & ~1u;
    if (DIRECT && n_p > 0xffffu) {  // block-uniform: output indices are 16 bits; such a partition needs the multi-pass variant
      if (tid == 0) { atomicExch(P.error_flag, 1u); P.out_seg_start[p] = 0; P.out_seg_len[p] = 0; }
      __syncthreads();
      continue;
    }
    // A partition with more entries than one table comfortably holds (the input outgrew the partition plan) is counted in
    // m passes: pass q takes the keys whose spare mix bits equal q, so every pass sees ~1/m of the distinct keys.  Its
    // output range is then reserved up front for all n_p entries; what stays unused is filled with (EMPTY, 0) entries
    // that every reader skips.  m is capped by the launch-wide P.split_log2 (set from the AVERAGE partition size): a
    // partition that is large only because a few keys are hot does not need more passes than its neighbours.
    uint32_t m_log2 = 0;
    while (!DIRECT && m_log2 < P.split_log2 && ((uint64_t)(SLOTS / 2) << m_log2) < n_p) ++m_log2;
    const uint32_t n_pass = 1u << m_log2;
    if (n_pass > 1 && tid == 0) {
      unsigned long long b = atomicAdd(P.out_cursor, (unsigned long long)n_p);
      if (b + n_p > P.out_cap) { atomicExch(P.nospace_flag, 1u); b = NO_SPACE; }
      s_base = b; s_run = 0;
    }

    constexpr int G = 8, H = 4;
    static_assert(G == 8, "slot bookkeeping below packs 8 x 16 bits");
#pragma unroll 1
    for (uint32_t pass = 0; pass < n_pass; ++pass) {
    if (pass) __syncthreads();  // the previous pass's list counters are reset
    // entry idx of the partition is kq[idx] while idx < hi (the pointers are biased by the run's first index)
    uint32_t r = 0;
    uint64_t hi = seg_prefix[1];
    const uint64_t *kq = P.runs[0].keys + seg_begin[0];
    const uint64_t *cq = (WEIGHTED && P.runs[0].counts) ? P.runs[0].counts + seg_begin[0] : nullptr;
#pragma unroll 1
    for (uint64_t base = 0; base < n_p; base += (uint64_t)SMEM_COUNT_THREADS * G) {
      uint64_t key[G];
      uint32_t w[WEIGHTED ? G : 1];
      uint32_t live = 0;  // bit j: key j is a real entry with a non-zero weight
#pragma unroll
      for (int j = 0; j < G; ++j) {
        const uint64_t idx = base + (uint64_t)j * SMEM_COUNT_THREADS + tid;
        key[j] = EMPTY_MIX;
        if (WEIGHTED) w[j] = 0;
        if (idx < n_p) {
          while (idx >= hi) {  // entries are visited in ascending order: runs only ever advance
            ++r;
            hi = seg_prefix[r + 1];
            kq = P.runs[r].keys + seg_begin[r] - seg_prefix[r];
            if (WEIGHTED) cq = P.runs[r].counts ? P.runs[r].counts + seg_begin[r] - seg_prefix[r] : nullptr;
          }
          key[j] = n_pass > 1 ? __ldg(kq + idx) : __ldcs(kq + idx);  // multi-pass: the entries are read again, keep them in L2
          if (n_pass == 1 || (((uint32_t)key[j] >> 13) & (n_pass - 1)) == pass) live |= 1u << j;
          if (WEIGHTED) {
            uint64_t w64 = 1;
            if (cq) w64 = __ldcs(cq + idx);
            if (w64 > 0xffffffffull) { atomicExch(P.error_flag, 1u); w64 = 0; }  // needs the u64 (L2-scratch) variant
            w[j] = (uint32_t)w64;
            if (!w64) live &= ~(1u << j);
          }
        }
      }
      if (WEIGHTED && (P.preagg & 1u) && n_p > 2 * SMEM_COUNT_THREADS * G) {
        // Warp run-length pre-aggregation, only for oversized (= skewed) partitions: the scatter passes keep the keys of
        // consecutive windows close together, so homopolymer / tandem-repeat runs arrive as runs of equal keys in
        // adjacent lanes.  The head lane of each run upserts once with the run length.
#pragma unroll
        for (int j = 0; j < G; ++j) {
          const uint64_t kk = (live >> j & 1u) ? key[j] : EMPTY_MIX;
          const uint64_t kp = __shfl_up_sync(0xffffffffu, kk, 1);
          const bool head = lane == 0 || kp != kk;
          const uint32_t heads = __ballot_sync(0xffffffffu, head);
          if (__all_sync(0xffffffffu, w[j] <= 1u)) {
            const uint32_t above = lane == 31 ? 0u : heads & ~((2u << lane) - 1u);
            const uint32_t end = above ? (uint32_t)__ffs(above) - 1u : 32u;
            if (live >> j & 1u) { w[j] = head ? end - lane : 0u; if (!head) live &= ~(1u << j); }
          }
        }
      }
      // ---- two straight-line probe rounds, H keys in flight each: the home bucket (one 16-byte load), then -- for the
      // keys that lost -- the next position of their sequence.  Both rounds run converged; only the ~2 % of keys that are
      // still homeless afterwards enter the divergent loop below.
      // Probe sequence of a (mixed) key: bucket t = b0 + t * step2 (b0 = its lowest bits, the odd stride from bits 40+), slots (t,0), (t,1).
      uint32_t pend = 0, newm = 0;    // bit j: key j still to place / key j claimed a fresh slot
      uint32_t odd = 0, adv = 0;      // pending key j lost slot (adv, odd) last: it continues at u = 2 * adv + odd + 1
      uint64_t fs_lo = 0, fs_hi = 0;  // slot of key j, 16 bits each (keys 0-3 / 4-7), meaningful for the keys in newm
#pragma unroll
      for (int h0 = 0; h0 < G; h0 += H) {
        uint32_t sl[H];
#pragma unroll
        for (int j = 0; j < H; ++j) sl[j] = (uint32_t)key[h0 + j] & bmask;
#pragma unroll
        for (int round = 0; round < 2; ++round) {
          const uint32_t act = round ? pend : live;
          ulonglong2 cur[H];
          unsigned long long got[H];
#pragma unroll
          for (int j = 0; j < H; ++j) {
            const int q = h0 + j;
            if (round && (odd >> q & 1u)) sl[j] = ((sl[j] & ~1u) + ((((uint32_t)(key[q] >> 40)) | 1u) << 1)) & mask;  // both home slots lost: next bucket
            else sl[j] &= ~1u;
            cur[j] = make_ulonglong2(0ull, 0ull);
            if (act >> q & 1u) cur[j] = *reinterpret_cast<const ulonglong2 *>(&skeys[sl[j]]);
          }
          const uint32_t was_odd = odd;
#pragma unroll
          for (int j = 0; j < H; ++j) {
            const int q = h0 + j;
            const unsigned long long k = key[q];
            got[j] = 0ull;
            if (!(act >> q & 1u)) continue;
            const bool x_known_taken = round && !(was_odd >> q & 1u);  // lost the race for the first home slot in round 0
            if (x_known_taken || (cur[j].x != k && cur[j].x != EMPTY_MIX)) { sl[j] |= 1u; cur[j].x = cur[j].y; }
            got[j] = cur[j].x;
            if (cur[j].x == EMPTY_MIX) got[j] = atomicCAS(&skeys[sl[j]], EMPTY_MIX, k);
          }
          if (round == 0) {
            // second chance inside the home bucket: the whole partition is inserted concurrently, so most conflicts are lost RACES for
            // the first slot -- the loser takes the second slot right away instead of waiting for round 1, which then already looks
            // at the next bucket; only keys that lose three slots reach the divergent loop below
#pragma unroll
            for (int j = 0; j < H; ++j) {
              const int q = h0 + j;
              const unsigned long long k = key[q];
              if ((act >> q & 1u) && !(sl[j] & 1u) && got[j] != EMPTY_MIX && got[j] != k) {
                sl[j] |= 1u;
                got[j] = cur[j].y;  // as loaded with the bucket; re-checked by the CAS when it looked empty
                if (cur[j].y == EMPTY_MIX) got[j] = atomicCAS(&skeys[sl[j]], EMPTY_MIX, k);
              }
            }
          }
#pragma unroll
          for (int j = 0; j < H; ++j) {
            const int q = h0 + j;
            if (!(act >> q & 1u)) continue;
            const bool is_new = got[j] == EMPTY_MIX;
            if (is_new || got[j] == key[q]) {
              const uint32_t wj = WEIGHTED ? w[q] : 1u;
              const uint32_t add = wj - (is_new ? 1u : 0u);  // slots store occurrences - 1
              if (add) { const uint32_t old = atomicAdd(&scnt[sl[j]], add); if (old > 0xffffffffu - add) atomicExch(P.error_flag, 1u); }
              if (is_new) { newm |= 1u << q; (q < 4 ? fs_lo : fs_hi) |= (uint64_t)sl[j] << (16 * (q & 3)); }
              pend &= ~(1u << q);
            } else {
              pend |= 1u << q;
              if (round) adv |= (was_odd >> q & 1u) << q;  // this round looked at the next bucket iff both home slots were lost before
              odd = (odd & ~(1u << q)) | ((sl[j] & 1u) << q);
            }
          }
        }
      }
      if (DIRECT) {
        // ---- the keys that claimed a slot in the two rounds go to the output now: key q of all lanes forms one run, lanes in
        // order, so a warp store covers consecutive entries.  Still converged code: the ballots are plain votes.
        uint32_t bal[G], tot = 0;
#pragma unroll
        for (int q = 0; q < G; ++q) { bal[q] = __ballot_sync(0xffffffffu, newm >> q & 1u); tot += __popc(bal[q]); }
        uint32_t wb = 0;
        if (lane == 0 && tot) wb = atomicAdd(&s_emit, tot);
        wb = __shfl_sync(0xffffffffu, wb, 0);
        const uint32_t lt = (1u << lane) - 1u;
        const bool fits = s_base != NO_SPACE;
#pragma unroll
        for (int q = 0; q < G; ++q) {
          if (newm >> q & 1u) {
            const uint32_t oi = wb + __popc(bal[q] & lt);
            slist[(uint32_t)((q < 4 ? fs_lo : fs_hi) >> (16 * (q & 3))) & 0xffffu] = (uint16_t)oi;
            if (fits) { __stcs(P.out_keys + s_base + oi, (uint64_t)key[q]); __stcs(P.out_counts + s_base + oi, (uint64_t)1); }
          }
          wb += __popc(bal[q]);
        }
      }
      // ---- what is left: every lane works through ITS pending keys on its own, continuing behind the slot it lost
      while (pend) {
        const int j = __ffs(pend) - 1;
        uint64_t kj = key[0];
        uint32_t wj = WEIGHTED ? w[0] : 1u;
#pragma unroll
        for (int q = 1; q < G; ++q) if (j == q) { kj = key[q]; if (WEIGHTED) wj = w[q]; }
        const uint32_t b0 = (uint32_t)kj & bmask, step2 = (((uint32_t)(kj >> 40)) | 1u) << 1;
        uint32_t s2 = 0;
        unsigned long long c2 = 0;
        for (uint32_t u = 2u * (adv >> j & 1u) + (odd >> j & 1u) + 1u;; ++u) {
          s2 = ((b0 + (u >> 1) * step2) & mask) | (u & 1u);
          c2 = skeys[s2];
          if (c2 == EMPTY_MIX) c2 = atomicCAS(&skeys[s2], EMPTY_MIX, kj);
          if (c2 == EMPTY_MIX || c2 == kj) break;
          if (u > mask + 4) { atomicExch(P.error_flag, 1u); break; }  // every slot visited: the host re-runs with the L2 variant
        }
        const bool is_new = c2 == EMPTY_MIX;
        if (is_new || c2 == kj) {
          const uint32_t add = wj - (is_new ? 1u : 0u);
          if (add) { const uint32_t old = atomicAdd(&scnt[s2], add); if (old > 0xffffffffu - add) atomicExch(P.error_flag, 1u); }
          if (is_new) {
            if (DIRECT) {  // rare (~2 % of the keys): one shared atomic hands out the output index
              const uint32_t oi = atomicAdd(&s_emit, 1u);
              slist[s2] = (uint16_t)oi;
              if (s_base != NO_SPACE) { __stcs(P.out_keys + s_base + oi, (uint64_t)kj); __stcs(P.out_counts + s_base + oi, (uint64_t)1); }
            } else {
              newm |= 1u << j;
              const uint64_t f = (uint64_t)s2 << (16 * (j & 3));
              if (j < 4) fs_lo |= f; else fs_hi |= f;
            }
          }
        }
        pend &= pend - 1;
      }
      __syncwarp();  // reconverge here: otherwise the rest of the batch runs once per fragment of the warp
      if (DIRECT) continue;  // everything of this batch has been written
      // ---- every lane appends the slots it claimed to its warp's list.  One same-address shared atomic per lane
      // and batch hands out the positions; deliberately no warp collective here: this point follows divergent
      // code, where a *_sync intrinsic costs a software convergence routine per call.
      if (newm) {
        uint32_t pos = atomicAdd(&s_wn[warp], (uint32_t)__popc(newm));
#pragma unroll
        for (int q = 0; q < G; ++q)
          if (newm >> q & 1u) { if (pos < WLIST) wlist[pos] = (uint16_t)((q < 4 ? fs_lo : fs_hi) >> (16 * (q & 3))); ++pos; }
      }
    }
    __syncthreads();  // all upserts done
    if (DIRECT) {
      const uint32_t d = s_emit;  // distinct keys of the partition, all of them already in the output with count 1
      const bool fits = s_base != NO_SPACE;
      // sweep the table: patch the entries of the keys that were seen again, note their counts, clean the slots
      for (uint32_t i = 2 * tid; i <= mask; i += 2 * SMEM_COUNT_THREADS) {
        const uint2 c2 = *reinterpret_cast<const uint2 *>(&scnt[i]);
        if (c2.x | c2.y) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const uint32_t cc = h ? c2.y : c2.x;
            if (!cc) continue;
            const unsigned long long cnt = (unsigned long long)cc + 1;  // slots store occurrences - 1
            if (fits) __stcs(P.out_counts + s_base + slist[i + h], (uint64_t)cnt);
            if (P.hist) {
              if (cnt < (unsigned long long)HIST_CTA_BINS) atomicAdd(&s_hist[cnt], 1u);
              else if (cnt < (unsigned long long)HIST_DENSE_BINS) atomicAdd(P.hist + cnt, 1ull);
              else { const unsigned long long o = atomicAdd(P.hist + HIST_DENSE_BINS, 1ull); if (o < P.hist_overflow_cap) P.hist_overflow[o] = cnt; }
            }
          }
          *reinterpret_cast<uint2 *>(&scnt[i]) = make_uint2(0u, 0u);
        }
        *reinterpret_cast<ulonglong2 *>(&skeys[i]) = make_ulonglong2(EMPTY_MIX, EMPTY_MIX);
      }
      for (uint64_t i = d + tid; i < n_p && fits; i += SMEM_COUNT_THREADS) {  // one unused entry per duplicate: readers skip them
        __stcs(P.out_keys + s_base + i, (uint64_t)EMPTY_MIX);
        __stcs(P.out_counts + s_base + i, (uint64_t)0);
      }
      if (tid == 0) {
        P.out_seg_start[p] = fits ? s_base : 0; P.out_seg_len[p] = d;
        if (d) atomicAdd(P.out_distinct, (unsigned long long)d);
      }
      __syncthreads();  // table clean, s_base / s_emit free for the next partition
      continue;
    }
    uint32_t wn = s_wn[warp];  // slots this warp claimed for the partition
    if (wn > WLIST) { if (lane == 0) atomicExch(P.error_flag, 1u); wn = WLIST; }  // list full: results are discarded, stay in bounds
    // ---- compact: the partition gets one contiguous output range (one global atomic), each warp a sub-range of it
    uint32_t pre, pass_d;
    {
      const uint32_t raw = lane < NW ? s_wn[lane] : 0u, v = min(raw, WLIST);
      const bool lost = __any_sync(0xffffffffu, raw > WLIST);  // some warp's list overflowed: the partition's results are void
      uint32_t incl = v;
#pragma unroll
      for (int o = 1; o < NW; o <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += u; }
      const uint32_t d = __shfl_sync(0xffffffffu, incl, NW - 1);
      pre = __shfl_sync(0xffffffffu, incl - v, warp);
      if (n_pass == 1 && tid == 0) {
        unsigned long long b = P.pre_base ? P.pre_base[work] : NO_SPACE;  // a range the sieve variant had reserved (it holds >= n_p >= d entries)
        if (b == NO_SPACE) {
          b = atomicAdd(P.out_cursor, (unsigned long long)d);
          if (b + d > P.out_cap) { atomicExch(P.nospace_flag, 1u); b = NO_SPACE; }
        } else if (lost || *reinterpret_cast<volatile uint32_t *>(P.error_flag)) {
          // void results stay out of a pre-reserved range: on the in-place route it is the partition's input, which the host's
          // fallback reads again (this CTA's table overflow was flagged before the barrier above)
          b = NO_SPACE;
        }
        P.out_seg_start[p] = b; P.out_seg_len[p] = d;
        s_base = b; s_run = 0;
        if (d) atomicAdd(P.out_distinct, (unsigned long long)d);
      }
      pass_d = d;
    }
    __syncthreads();
    {
      const bool fits = s_base != NO_SPACE;  // otherwise the table is only cleaned (the host retries with a larger run)
      const unsigned long long out0 = s_base + s_run + pre;
      for (uint32_t i0 = 0; i0 < wn; i0 += 32) {  // warp-uniform trip count
        const uint32_t i = i0 + lane;
        const bool ok = i < wn;
        unsigned long long cnt = 0;
        if (ok) {
          const uint32_t slot = wlist[i];
          cnt = (unsigned long long)scnt[slot] + 1;  // slots store occurrences - 1
          if (fits) {
            __stcs(P.out_keys + out0 + i, (uint64_t)skeys[slot]);
            __stcs(P.out_counts + out0 + i, (uint64_t)cnt);
          }
          skeys[slot] = EMPTY_MIX; scnt[slot] = 0;
        }
        if (P.hist) hist_note(ok, cnt, s_hist, P, lane);
      }
    }
    if (n_pass == 1 && P.pre_base && P.pre_base[work] != NO_SPACE && s_base != NO_SPACE) {  // the rest of the pre-reserved range: entries every reader skips
      const unsigned long long b = s_base;
      for (uint32_t i = pass_d + tid; i < P.pre_len[work]; i += SMEM_COUNT_THREADS) { __stcs(P.out_keys + b + i, (uint64_t)EMPTY_MIX); __stcs(P.out_counts + b + i, (uint64_t)0); }
    }
    __syncthreads();  // table clean before the next pass / partition (and every warp has read the list counters)
    if (tid < NW) s_wn[tid] = 0;  // ordered before the next appends by the barrier that opens the next pass / follows the metadata fetch
    if (tid == 0) s_run += pass_d;
    }  // pass
    if (n_pass > 1) {
      __syncthreads();
      const uint32_t done = s_run;  // <= n_p: every entry contributes at most one distinct key
      for (uint64_t i = done + tid; i < n_p && s_base != NO_SPACE; i += SMEM_COUNT_THREADS) {  // unused tail of the reservation: entries every reader skips
        __stcs(P.out_keys + s_base + i, (uint64_t)EMPTY_MIX);
        __stcs(P.out_counts + s_base + i, (uint64_t)0);
      }
      if (tid == 0) {
        P.out_seg_start[p] = s_base; P.out_seg_len[p] = done;
        if (done) atomicAdd(P.out_distinct, (unsigned long long)done);
      }
      __syncthreads();  // s_base / s_run are rewritten by the next partition
    }
  }
  if (P.hist) hist_flush(s_hist, P, tid);
}

// ---------------------------------------------------------------------------------------------------
// phase B, sieve (unweighted runs of mostly distinct keys: a genome).  The table variants above pay a compare-and-swap protocol for
// EVERY key although almost every key of such a partition occurs once.  Here a key first sets its bit in a 2^18-bit map (one shared
// atomic OR, no retry): with ~3600 keys per partition only ~0.7 % of them find the bit already set.  Only those SUSPECTS and the keys
// they met are resolved in a small table; every other key occurs once and stays at its input position with count 1.  The input runs
// are raw runs, whose segments start on 16-byte boundaries and are padded to an even number of entries with EMPTY_MIX (refine_to_run,
// launch_pad_segments), so the key copies are handed to the TMA unit.  A sieve that copied the keys with plain loads and stores and
// resolved each suspect on the spot spent 3.9 warp-instr per key (ncu), a third of them in the one-lane-active detours of the
// suspects, and half of all warp time at block barriers.  So here
//   * the partition's keys arrive by 1-D bulk loads (one per input run) in one of two key stages, requested half a partition ahead,
//     and leave by ONE bulk store of the stage (fillers and repeats are patched in the stage); counts go out as plain coalesced
//     8-byte stores of 1 / 0 while the keys are read, and are patched afterwards where a key repeats;
//   * nothing divergent happens in the two passes over the keys: pass 1 is the bit-map test-and-set (a suspect only sets a bit in a
//     4096-bit filter indexed like the map), pass 2 tests that filter and queues the indices of the keys it flags -- the suspects,
//     the earlier keys they met in the bit map, a few chance hits;
//   * the queue (~100 of ~3600 entries) is then resolved by as many threads in parallel in a small table of stage indices
//     (32-bit CAS; the key of a slot is read from the stage): first claimant = the entry that stays, the others become fillers;
//   * two 512-thread CTAs per SM, so one CTA's barriers overlap the other's work; output ranges are reserved when the segment
//     table is fetched (two partitions ahead), so no global atomic sits on the critical path.
// The output segment is the padded input: entries (EMPTY, 0) are fillers every reader skips.  A partition with more suspects than
// the table holds, or more entries than one stage, is appended to P.redo_list and left to the compacting variant.  The in-place
// variant of this scheme (count_partitions_sieve_in_place_kernel) follows it.
// ---------------------------------------------------------------------------------------------------
constexpr uint32_t SV_BM_LOG2 = 18;
constexpr uint32_t SV_BM_WORDS = 1u << (SV_BM_LOG2 - 5);  // 32 KiB
constexpr int SVT_THREADS = 512, SVT_G = 8, SVT_NS = 2, SVT_META = 3;
__host__ __device__ __forceinline__ uint32_t sieve_redo_limit_impl(uint32_t n_parts) { return n_parts / 8 + 64; }
__device__ __forceinline__ uint32_t sieve_redo_limit(uint32_t n_parts) { return sieve_redo_limit_impl(n_parts); }
constexpr uint32_t SVT_CAP = SIEVE_MAX_ENTRIES;  // entries per key stage
constexpr uint32_t SVT_L_SLOTS = 1024, SVT_L_MAX = 704, SVT_Q = 2048, SVT_BLOOM_WORDS = 128;
static_assert(SVT_THREADS * SVT_G == (int)SVT_CAP, "one batch per partition");
constexpr size_t SVT_SMEM = (size_t)SVT_CAP * 8 * SVT_NS + (size_t)SV_BM_WORDS * 4 + (size_t)SVT_L_SLOTS * 8 + (size_t)SVT_Q * 2;

__device__ __forceinline__ void tma_store_1d(void *gmem_dst, const void *smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_wait_group_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void hist_add(uint32_t *s_hist, const CountParams &P, unsigned long long cnt) {
  if (cnt < (unsigned long long)HIST_CTA_BINS) atomicAdd(&s_hist[cnt], 1u);
  else if (cnt < (unsigned long long)HIST_DENSE_BINS) atomicAdd(P.hist + cnt, 1ull);
  else { const unsigned long long o = atomicAdd(P.hist + HIST_DENSE_BINS, 1ull); if (o < P.hist_overflow_cap) P.hist_overflow[o] = cnt; }
}
template <bool ONE_RUN>
__global__ void __launch_bounds__(SVT_THREADS, 2) count_partitions_sieve_tma_kernel(CountParams P) {
  extern __shared__ __align__(128) unsigned char svt_raw[];
  constexpr int G = SVT_G, T = SVT_THREADS, NS = SVT_NS, NM = SVT_META;
  unsigned long long *stage = reinterpret_cast<unsigned long long *>(svt_raw);  // [NS][SVT_CAP] keys
  uint32_t *bm = reinterpret_cast<uint32_t *>(stage + (size_t)NS * SVT_CAP);    // bit map
  uint32_t *Lslot = bm + SV_BM_WORDS;                                           // stage index + 1 of the entry that owns the slot, 0 = free
  uint32_t *Lcnt = Lslot + SVT_L_SLOTS;                                         // further occurrences of that entry's key
  uint16_t *Q = reinterpret_cast<uint16_t *>(Lcnt + SVT_L_SLOTS);               // stage indices of the flagged entries
  __shared__ __align__(8) uint64_t bar[NS];
  __shared__ uint64_t m_src[NM][CONS_MAX_RUNS];  // run r's segment of the partition (global address)
  __shared__ uint32_t m_len[NM][CONS_MAX_RUNS];  // its padded length in entries
  __shared__ uint32_t m_npad[NM], m_np[NM], m_work[NM], m_state[NM];  // state: 0 empty, 1 staged, 2 left to the compacting variant
  __shared__ unsigned long long m_base[NM];
  __shared__ uint32_t s_hist[HIST_CTA_BINS], s_bloom[SVT_BLOOM_WORDS];
  __shared__ uint32_t s_nq, s_nL, s_fail, s_holes;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t R = P.R;

  auto fetch = [&](uint32_t w, uint64_t &b, uint64_t &len) {
    b = 0; len = 0;
    if (w < P.n_parts && lane < (int)R) {
      const uint32_t p = P.order ? P.order[w] : w;
      b = P.runs[lane].seg_start[p]; len = P.runs[lane].seg_len[p];
    }
  };
  // warp 0: work item w (lane r holds run r's segment) -> metadata slot sl.  The output range is reserved here, but the atomic's
  // result is only looked at one iteration later (settle): its latency must not sit in this single-warp section.
  unsigned long long pend_ob = 0;  // lane 0
  uint32_t pend_npad = 0;
  int pend_slot = -1;
  auto settle = [&]() {  // lane 0
    if (pend_slot < 0) return;
    unsigned long long ob = pend_ob;
    if (ob + pend_npad > P.out_cap) { atomicExch(P.nospace_flag, 1u); ob = NO_SPACE; }
    m_base[pend_slot] = ob;
    pend_slot = -1;
  };
  auto publish = [&](int sl, uint32_t w, uint64_t b, uint64_t len) {
    const bool big = __any_sync(0xffffffffu, len > (uint64_t)SVT_CAP);
    const uint32_t l32 = big ? 0u : (uint32_t)len, pl = (l32 + 1u) & ~1u;
    uint32_t incl = pl, np = l32;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) np += __shfl_xor_sync(0xffffffffu, np, o);
    const uint32_t npad = __shfl_sync(0xffffffffu, incl, 31);
    const uint32_t state = w >= P.n_parts ? 0u : (big || npad > SVT_CAP) ? 2u : npad ? 1u : 0u;
    if (lane < (int)R) { m_src[sl][lane] = reinterpret_cast<uint64_t>(P.runs[lane].keys + b); m_len[sl][lane] = pl; }
    if (lane == 0) {
      if (state == 1u) { pend_ob = atomicAdd(P.out_cursor, (unsigned long long)npad); pend_npad = npad; pend_slot = sl; }
      m_npad[sl] = npad; m_np[sl] = np; m_work[sl] = w; m_state[sl] = state;
    }
    __syncwarp();
  };
  // thread 0: bulk loads of the partition in metadata slot sl into key stage ks
  auto issue = [&](int sl, int ks) {
    if (m_state[sl] != 1u) return;
    mbar_expect_tx(&bar[ks], m_npad[sl] * 8u);
    uint32_t off = 0;
    for (uint32_t r = 0; r < R; ++r) {
      const uint32_t pl = m_len[sl][r];
      if (pl) tma_load_1d(stage + (size_t)ks * SVT_CAP + off, reinterpret_cast<const void *>(m_src[sl][r]), pl * 8u, &bar[ks]);
      off += pl;
    }
  };

  if (tid < HIST_CTA_BINS) s_hist[tid] = 0;
  if (tid < (int)SVT_BLOOM_WORDS) s_bloom[tid] = 0;
  for (uint32_t i = tid; i < SVT_L_SLOTS; i += T) { Lslot[i] = 0; Lcnt[i] = 0; }
  for (uint32_t i = tid; i < SV_BM_WORDS; i += T) bm[i] = 0;
  if (tid == 0) {
    s_nq = 0; s_nL = 0; s_fail = 0; s_holes = 0;
    for (int i = 0; i < NS; ++i) mbar_init(&bar[i], 1);
    mbar_fence_init();
  }
  uint32_t w_ahead = 0;  // lane 0 of warp 0: the work item two after the current one
  __syncthreads();
  if (warp == 0) {
    uint32_t w0 = 0, w1 = 0;
    if (lane == 0) { w0 = atomicAdd(P.next, 1u); w1 = atomicAdd(P.next, 1u); w_ahead = atomicAdd(P.next, 1u); }
    w0 = __shfl_sync(0xffffffffu, w0, 0); w1 = __shfl_sync(0xffffffffu, w1, 0);
    uint64_t b, len;
    fetch(w0, b, len); publish(0, w0, b, len);
    if (lane == 0) settle();
    fetch(w1, b, len); publish(1, w1, b, len);
    if (lane == 0) { issue(0, 0); settle(); }
  }
  __syncthreads();

  unsigned long long my_entries = 0;  // tid 0: distinct keys of the partitions this CTA counted
  uint32_t ph = 0;                    // bit s: parity of key stage s's next completion
  for (uint32_t it = 0;; ++it) {
    const int sl = (int)(it % NM), ks = (int)(it & 1u);
    const uint32_t work = m_work[sl];
    if (work >= P.n_parts) break;
    const uint32_t state = m_state[sl], npad = m_npad[sl], np = m_np[sl];
    const unsigned long long base = m_base[sl];
    const bool fits = base != NO_SPACE;
    const uint32_t p = P.order ? P.order[work] : work;
    // segment table of the partition two ahead: loads issued now, published at the end of this iteration
    uint32_t wn = 0, handed_back = 0;
    uint64_t nb = 0, nlen = 0;
    if (warp == 0) {
      wn = __shfl_sync(0xffffffffu, w_ahead, 0);
      fetch(wn, nb, nlen);
      if (lane == 0 && wn < P.n_parts) w_ahead = atomicAdd(P.next, 1u);
      if (lane == 0) handed_back = *reinterpret_cast<volatile uint32_t *>(P.redo_count);  // looked at when this iteration ends
    }
    if (state != 1u) {
      if (tid == 0) {
        if (state == 0u) { P.out_seg_start[p] = 0; P.out_seg_len[p] = 0; }
        else {
          const uint32_t ri = atomicAdd(P.redo_count, 1u);
          P.redo_list[ri] = p; P.redo_base[ri] = NO_SPACE; P.redo_len[ri] = 0u;
        }
        tma_wait_group_read<0>();
        issue((int)((it + 1) % NM), ks ^ 1);  // the next partition's keys
      }
    } else {
      unsigned long long *st = stage + (size_t)ks * SVT_CAP;
      // the previous partition's queue / table counters: everybody read them before barrier A, nobody touches them before barrier B
      if (tid == 0) { s_nq = 0; s_nL = 0; s_fail = 0; s_holes = 0; }
      mbar_wait(&bar[ks], (ph >> ks) & 1u);
      ph ^= 1u << ks;
      // ---- pass 1: read the staged keys, write the counts (1 per live entry), test-and-set in the bit map
      unsigned long long key[G];
      uint32_t live = 0;
      {
        uint32_t old[G];
        const uint32_t last = npad - 1u;
#pragma unroll
        for (int j = 0; j < G; ++j) {
          const uint32_t idx = (uint32_t)j * T + tid;
          key[j] = st[min(idx, last)];  // rows past the end re-read the last entry and stay dead
          const bool lv = ONE_RUN ? idx < np : (idx < npad && key[j] != EMPTY_MIX);  // not the pad entry behind a segment of odd length
          live |= (lv ? 1u : 0u) << j;
          if (fits && idx < npad) __stcs(P.out_counts + base + idx, lv ? 1ull : 0ull);
          const uint32_t lo = (uint32_t)key[j];
          old[j] = lv ? atomicOr(&bm[(lo >> 5) & (SV_BM_WORDS - 1)], __funnelshift_l(0u, 1u, lo)) : 0u;
        }
#pragma unroll
        for (int j = 0; j < G; ++j) {  // a suspect (its bit was already set) marks the filter; no detour, a predicated shared atomic
          const uint32_t lo = (uint32_t)key[j];
          if (__funnelshift_r(old[j], 0u, lo) & 1u) atomicOr(&s_bloom[(lo >> 5) & (SVT_BLOOM_WORDS - 1)], __funnelshift_l(0u, 1u, lo));
        }
      }
      if (tid == 0) {  // the other key stage: its last store has had this pass to leave shared memory
        tma_wait_group_read<0>();
        issue((int)((it + 1) % NM), ks ^ 1);
      }
      __syncthreads();  // B: bit map and filter complete
      {
        uint4 *bm4 = reinterpret_cast<uint4 *>(bm);
#pragma unroll
        for (uint32_t i = 0; i < SV_BM_WORDS / 4 / T; ++i) bm4[i * T + tid] = make_uint4(0u, 0u, 0u, 0u);
      }
      // ---- pass 2: the entries the filter flags are queued
      {
        uint32_t hit = 0;
#pragma unroll
        for (int j = 0; j < G; ++j) {
          const uint32_t lo = (uint32_t)key[j];
          hit |= ((s_bloom[(lo >> 5) & (SVT_BLOOM_WORDS - 1)] & __funnelshift_l(0u, 1u, lo)) ? 1u : 0u) << j;
        }
        hit &= live;
        if (hit) {
          uint32_t q = atomicAdd(&s_nq, (uint32_t)__popc(hit));
          while (hit) {
            const uint32_t j = (uint32_t)__ffs((int)hit) - 1u;
            if (q < SVT_Q) Q[q] = (uint16_t)(j * T + tid);
            ++q;
            hit &= hit - 1u;
          }
        }
      }
      __syncthreads();  // C: the queue is complete
      const uint32_t nq = s_nq;
      // ---- resolve the queue: entry e claims a slot of L for its key or meets the entry that did
      constexpr int E = SVT_Q / T;
      uint32_t my_slot[E], my_idx[E], reps = 0;
      if (nq <= SVT_Q && (uint32_t)tid < nq) {
#pragma unroll
        for (int u = 0; u < E; ++u) {
          const uint32_t e = (uint32_t)u * T + tid;
          my_slot[u] = 0; my_idx[u] = 0;
          if (e >= nq) continue;
          const uint32_t idx = Q[e];
          const unsigned long long k = st[idx];
          uint32_t s = (uint32_t)(k >> 32) & (SVT_L_SLOTS - 1);
          for (uint32_t t = 0;; ++t) {
            if (t > SVT_L_SLOTS) { atomicExch(&s_fail, 1u); break; }
            uint32_t cur = *reinterpret_cast<volatile uint32_t *>(&Lslot[s]);
            if (cur == 0u) {
              if (*reinterpret_cast<volatile uint32_t *>(&s_fail)) break;  // bounds the entries: every thread has at most one claim past this test
              cur = atomicCAS(&Lslot[s], 0u, idx + 1u);
              if (cur == 0u) {
                if (atomicAdd(&s_nL, 1u) >= SVT_L_MAX) atomicExch(&s_fail, 1u);
                reps |= 1u << u; my_slot[u] = s; my_idx[u] = idx;
                break;
              }
            }
            if (st[cur - 1u] == k) {  // the owner of a slot is never patched: its key stays readable
              atomicAdd(&Lcnt[s], 1u);
              st[idx] = EMPTY_MIX;
              if (fits) P.out_counts[base + idx] = 0ull;  // after this entry's own 1 (two barriers ago)
              atomicAdd(&s_holes, 1u);  // of this partition
              break;
            }
            s = (s + 1u) & (SVT_L_SLOTS - 1);
          }
        }
      }
      fence_proxy_async_smem();  // this thread's patches of the stage, ahead of the bulk store
      __syncthreads();           // D: L's counters are final
      const bool fail = nq > SVT_Q || s_fail != 0;
      if (!fail) {
        if (reps)
#pragma unroll
        for (int u = 0; u < E; ++u) {
          if (!(reps >> u & 1u)) continue;
          const unsigned long long cnt = 1ull + Lcnt[my_slot[u]];
          if (cnt > 1) {
            if (fits) P.out_counts[base + my_idx[u]] = cnt;
            if (P.hist) hist_add(s_hist, P, cnt);
          }
          Lslot[my_slot[u]] = 0; Lcnt[my_slot[u]] = 0;
        }
        if (tid == 0) {
          if (fits) tma_store_1d(P.out_keys + base, st, npad * 8u);
          P.out_seg_start[p] = fits ? base : 0;
          P.out_seg_len[p] = npad;
          my_entries += np - s_holes;
        }
      } else {  // too many repeated keys: the partition goes to the compacting variant, which writes into the range reserved here
        for (uint32_t i = tid; i < SVT_L_SLOTS; i += T) { Lslot[i] = 0; Lcnt[i] = 0; }
        if (tid == 0) {
          const uint32_t ri = atomicAdd(P.redo_count, 1u);
          P.redo_list[ri] = p; P.redo_base[ri] = base; P.redo_len[ri] = npad;
        }
      }
      if (tid < (int)SVT_BLOOM_WORDS) s_bloom[tid] = 0;
    }
    if (warp == 0) {
      if (lane == 0) { tma_commit_group(); settle(); }  // settle: the partition published one iteration ago (it is processed next)
      // a duplicate-rich input (most partitions handed back) is not this variant's business: stop early, the host repeats the launch without it
      if (__shfl_sync(0xffffffffu, handed_back, 0) > sieve_redo_limit(P.n_parts)) { wn = 0xffffffffu; nb = 0; nlen = 0; }
      publish((int)((it + 2) % NM), wn, nb, nlen);
    }
    __syncthreads();  // A
  }
  if (tid == 0) {
    tma_wait_group_read<0>();
    if (my_entries) atomicAdd(P.out_distinct, my_entries);
  }
  if (P.hist) hist_flush(s_hist, P, tid);
}

// ---------------------------------------------------------------------------------------------------
// The sieve in place (one raw run in a strided layout, P.part_cap): the stored keys would be byte-identical to the loaded ones
// except for the rare repeats, so the output run keeps the input's key array and layout and only counts are written -- 8 B in and
// 8 B per slot of capacity out per key instead of 8 in and 16 out.  A repeat keeps its key and gets count 0; the pad entry and the
// slack behind the segment get count 0 too, so whole-array readers skip them whatever keys sit there.  The keys are never written,
// so every fallback of the host (early stop, the launch without the sieve) rereads an intact input.
// The passes are those of the TMA sieve above.  Without a bulk store the stage only has to live until the queue is resolved, so a
// CTA has one key stage and keeps no keys in registers across its barriers (pass 2 and the queue re-read the stage); the next
// partition's bulk load is issued right after barrier D.  The shared memory a second stage would take holds more partitions in
// flight instead: four 256-thread CTAs per SM, whose chains of a bulk load and four block barriers per partition overlap.
// The map is 2^16 bits (2048 words), and a key sets TWO bits of one word with one atomic OR: word (lo >> 5) & 2047, bits lo & 31
// and (lo >> 16) & 31 of the key's low half lo.  A key is a suspect iff both were already set.  Of two equal keys, the one whose OR
// comes second sees both bits of the other, so every repeat makes a suspect; a distinct key is a (false) suspect only when both
// its bits were set by other keys of its word.  Bits 0-20 of lo vary freely inside a partition (sub_of_mix takes at most 11 top
// bits of lo, the coarse bin comes from the high half).  A partition of ~3500 keys has ~22 suspects and a queue of ~50 entries
// (one bit per key: ~90 and ~250), well inside SVT_Q and SVT_L_MAX.  The queue is dealt out across the warps (entry e to lane
// e / 8 of warp e % 8), so that no warp carries a chain of probes that the others wait for at barrier D, and the entry that claims
// a slot of L notes the slot in its queue entry: after barrier D only the claimed slots are read and cleaned.
// ---------------------------------------------------------------------------------------------------
constexpr int SVI_THREADS = 256, SVI_G = 16, SVI_BATCH = 8, SVI_CTAS_PER_SM = 4;
constexpr uint32_t SVI_BM_WORDS = 1u << (16 - 5);  // 8 KiB
static_assert(SVI_THREADS * SVI_G == (int)SVT_CAP, "one stage per partition");
static_assert(SVT_CAP <= 0x8000u && SVT_L_SLOTS <= 0x8000u, "a queue entry holds a stage index or a flagged slot of L");
constexpr size_t SVI_SMEM = (size_t)SVT_CAP * 8 + (size_t)SVI_BM_WORDS * 4 + (size_t)SVT_L_SLOTS * 8 + (size_t)SVT_Q * 2;
__device__ __forceinline__ uint32_t svi_map_bits(uint32_t lo) { return __funnelshift_l(0u, 1u, lo) | __funnelshift_l(0u, 1u, lo >> 16); }

__global__ void __launch_bounds__(SVI_THREADS, SVI_CTAS_PER_SM) count_partitions_sieve_in_place_kernel(CountParams P) {
  extern __shared__ __align__(128) unsigned char svi_raw[];
  constexpr int G = SVI_G, T = SVI_THREADS, NM = SVT_META;
  unsigned long long *st = reinterpret_cast<unsigned long long *>(svi_raw);  // [SVT_CAP] keys
  const uint32_t *st32 = reinterpret_cast<const uint32_t *>(st);             // st32[2 * i]: low half of key i
  uint32_t *bm = reinterpret_cast<uint32_t *>(st + SVT_CAP);                 // bit map
  uint32_t *Lslot = bm + SVI_BM_WORDS;
  uint32_t *Lcnt = Lslot + SVT_L_SLOTS;
  uint16_t *Q = reinterpret_cast<uint16_t *>(Lcnt + SVT_L_SLOTS);
  __shared__ __align__(8) uint64_t bar;
  __shared__ unsigned long long m_base[NM];  // the partition's segment: its first slot in the input (and output) run
  __shared__ uint32_t m_npad[NM], m_np[NM], m_work[NM], m_state[NM];  // state: 0 empty, 1 staged, 2 left to the compacting variant
  __shared__ uint32_t s_hist[HIST_CTA_BINS], s_bloom[SVT_BLOOM_WORDS];
  __shared__ uint32_t s_nq, s_nL, s_fail, s_holes;
  const int tid = threadIdx.x;

  // thread 0 only: the segment table of work item w is loaded when an iteration starts and published when it ends
  auto fetch = [&](uint32_t w, uint64_t &b, uint64_t &len) {
    b = 0; len = 0;
    if (w < P.n_parts) {
      const uint32_t p = P.order ? P.order[w] : w;
      b = P.runs[0].seg_start[p]; len = P.runs[0].seg_len[p];
    }
  };
  auto publish = [&](int sl, uint32_t w, uint64_t b, uint64_t len) {
    const uint32_t np = len > (uint64_t)SVT_CAP ? 0u : (uint32_t)len;
    m_base[sl] = b; m_npad[sl] = (np + 1u) & ~1u; m_np[sl] = np; m_work[sl] = w;
    m_state[sl] = w >= P.n_parts ? 0u : len > (uint64_t)SVT_CAP ? 2u : np ? 1u : 0u;
  };
  auto issue = [&](int sl) {  // the bulk load of the partition in metadata slot sl into the key stage
    if (m_state[sl] != 1u) return;
    mbar_expect_tx(&bar, m_npad[sl] * 8u);
    tma_load_1d(st, P.runs[0].keys + m_base[sl], m_npad[sl] * 8u, &bar);
  };

  if (tid < HIST_CTA_BINS) s_hist[tid] = 0;
  if (tid < (int)SVT_BLOOM_WORDS) s_bloom[tid] = 0;
  for (uint32_t i = tid; i < SVT_L_SLOTS; i += T) { Lslot[i] = 0; Lcnt[i] = 0; }
  for (uint32_t i = tid; i < SVI_BM_WORDS; i += T) bm[i] = 0;
  uint32_t w_ahead = 0;  // thread 0: the work item two after the current one
  if (tid == 0) {
    s_nq = 0; s_nL = 0; s_fail = 0; s_holes = 0;
    mbar_init(&bar, 1);
    mbar_fence_init();
    const uint32_t w0 = atomicAdd(P.next, 1u), w1 = atomicAdd(P.next, 1u);
    w_ahead = atomicAdd(P.next, 1u);
    uint64_t b, len;
    fetch(w0, b, len); publish(0, w0, b, len);
    fetch(w1, b, len); publish(1, w1, b, len);
    issue(0);
  }
  __syncthreads();

  unsigned long long my_entries = 0;  // tid 0: distinct keys of the partitions this CTA counted
  uint32_t ph = 0;                    // parity of the key stage's next completion
  for (uint32_t it = 0;; ++it) {
    const int sl = (int)(it % NM), sl_next = (int)((it + 1) % NM);
    const uint32_t work = m_work[sl];
    if (work >= P.n_parts) break;
    const uint32_t state = m_state[sl], npad = m_npad[sl], np = m_np[sl];
    const unsigned long long base = m_base[sl];
    const uint32_t p = P.order ? P.order[work] : work;
    uint32_t wn = 0, handed_back = 0;
    uint64_t nb = 0, nlen = 0;
    if (tid == 0) {
      wn = w_ahead;
      fetch(wn, nb, nlen);
      if (wn < P.n_parts) w_ahead = atomicAdd(P.next, 1u);
      handed_back = *reinterpret_cast<volatile uint32_t *>(P.redo_count);  // looked at when this iteration ends
    }
    if (state != 1u) {
      if (state == 0u)  // an empty partition: its whole capacity is slack
        for (uint32_t i = tid; i < P.part_cap; i += T) __stcs(P.out_counts + base + i, 0ull);
      if (tid == 0) {
        if (state == 0u) P.out_seg_len[p] = 0;
        else {  // the compacting variant writes the partition into its own capacity
          const uint32_t ri = atomicAdd(P.redo_count, 1u);
          P.redo_list[ri] = p; P.redo_base[ri] = base; P.redo_len[ri] = P.part_cap;
        }
        issue(sl_next);
      }
    } else {
      // the previous partition's queue / table counters: everybody read them before barrier A, nobody touches them before barrier B
      if (tid == 0) { s_nq = 0; s_nL = 0; s_fail = 0; s_holes = 0; }
      mbar_wait(&bar, ph);
      ph ^= 1u;
      // ---- pass 1: read the staged keys' low halves, write the counts (1 per live entry), test-and-set in the bit map
      const uint32_t last = npad - 1u;
      uint32_t live = 0;
#pragma unroll
      for (int h = 0; h < G; h += SVI_BATCH) {
        uint32_t lo[SVI_BATCH], old[SVI_BATCH];
#pragma unroll
        for (int j = 0; j < SVI_BATCH; ++j) {
          const uint32_t idx = (uint32_t)(h + j) * T + tid;
          lo[j] = st32[2u * min(idx, last)];  // rows past the end re-read the last entry and stay dead
          const bool lv = idx < np;           // not the pad entry behind a segment of odd length
          live |= (lv ? 1u : 0u) << (h + j);
          if (idx < P.part_cap) __stcs(P.out_counts + base + idx, lv ? 1ull : 0ull);
          old[j] = lv ? atomicOr(&bm[(lo[j] >> 5) & (SVI_BM_WORDS - 1)], svi_map_bits(lo[j])) : 0u;
        }
#pragma unroll
        for (int j = 0; j < SVI_BATCH; ++j) {  // a suspect (both its bits were already set) marks the filter
          const uint32_t m = svi_map_bits(lo[j]);
          if ((old[j] & m) == m) atomicOr(&s_bloom[(lo[j] >> 5) & (SVT_BLOOM_WORDS - 1)], __funnelshift_l(0u, 1u, lo[j]));
        }
      }
      for (uint32_t i = (uint32_t)G * T + tid; i < P.part_cap; i += T) __stcs(P.out_counts + base + i, 0ull);  // the capacity may exceed one stage
      __syncthreads();  // B: bit map and filter complete
      {
        uint4 *bm4 = reinterpret_cast<uint4 *>(bm);
#pragma unroll
        for (uint32_t i = 0; i < SVI_BM_WORDS / 4 / T; ++i) bm4[i * T + tid] = make_uint4(0u, 0u, 0u, 0u);
      }
      // ---- pass 2: the entries the filter flags are queued
      {
        uint32_t hit = 0;
#pragma unroll
        for (int j = 0; j < G; ++j) {
          const uint32_t lo = st32[2u * min((uint32_t)j * T + tid, last)];
          hit |= ((s_bloom[(lo >> 5) & (SVT_BLOOM_WORDS - 1)] & __funnelshift_l(0u, 1u, lo)) ? 1u : 0u) << j;
        }
        hit &= live;
        if (hit) {
          uint32_t q = atomicAdd(&s_nq, (uint32_t)__popc(hit));
          while (hit) {
            const uint32_t j = (uint32_t)__ffs((int)hit) - 1u;
            if (q < SVT_Q) Q[q] = (uint16_t)(j * T + tid);
            ++q;
            hit &= hit - 1u;
          }
        }
      }
      __syncthreads();  // C: the queue is complete
      const uint32_t nq = s_nq;
      // ---- resolve the queue: entry e claims a slot of L for its key or meets the entry that did
      const uint32_t e0 = (uint32_t)(tid & 31) * (T / 32) + (uint32_t)(tid >> 5);  // this thread's first entry
      if (nq <= SVT_Q)
        for (uint32_t e = e0; e < nq; e += T) {
          const uint32_t idx = Q[e];
          const unsigned long long k = st[idx];
          uint32_t s = (uint32_t)(k >> 32) & (SVT_L_SLOTS - 1);
          for (uint32_t t = 0;; ++t) {
            if (t > SVT_L_SLOTS) { atomicExch(&s_fail, 1u); break; }
            uint32_t cur = *reinterpret_cast<volatile uint32_t *>(&Lslot[s]);
            if (cur == 0u) {
              if (*reinterpret_cast<volatile uint32_t *>(&s_fail)) break;  // bounds the entries: every thread has at most one claim past this test
              cur = atomicCAS(&Lslot[s], 0u, idx + 1u);
              if (cur == 0u) {
                if (atomicAdd(&s_nL, 1u) >= SVT_L_MAX) atomicExch(&s_fail, 1u);
                Q[e] = (uint16_t)(0x8000u | s);  // read back after barrier D
                break;
              }
            }
            if (st[cur - 1u] == k) {
              atomicAdd(&Lcnt[s], 1u);
              P.out_counts[base + idx] = 0ull;  // after this entry's own 1 (two barriers ago)
              atomicAdd(&s_holes, 1u);          // of this partition
              break;
            }
            s = (s + 1u) & (SVT_L_SLOTS - 1);
          }
        }
      __syncthreads();  // D: L's counters are final; nobody reads the stage any more
      if (tid == 0) issue(sl_next);
      const bool fail = nq > SVT_Q || s_fail != 0;
      // the entries that own a slot of L carry their key's count, and their threads clean the slot
      if (nq <= SVT_Q)
        for (uint32_t e = e0; e < nq; e += T) {
          const uint32_t q = Q[e];
          if (!(q & 0x8000u)) continue;
          const uint32_t s = q & (SVT_L_SLOTS - 1), more = Lcnt[s];
          if (!fail && more) {
            const unsigned long long cnt = 1ull + more;
            P.out_counts[base + Lslot[s] - 1u] = cnt;
            if (P.hist) hist_add(s_hist, P, cnt);
          }
          Lslot[s] = 0; Lcnt[s] = 0;
        }
      if (tid == 0) {
        if (!fail) {
          P.out_seg_len[p] = npad;
          my_entries += np - s_holes;
        } else {  // too many repeated keys: the compacting variant writes the partition into its own capacity
          const uint32_t ri = atomicAdd(P.redo_count, 1u);
          P.redo_list[ri] = p; P.redo_base[ri] = base; P.redo_len[ri] = P.part_cap;
        }
      }
      s_bloom[tid % SVT_BLOOM_WORDS] = 0;  // by every thread: a predicate kept across the loop would cost a register
    }
    if (tid == 0) {
      // a duplicate-rich input (most partitions handed back) is not this variant's business: stop early, the host repeats the launch without it
      if (handed_back > sieve_redo_limit(P.n_parts)) { wn = 0xffffffffu; nb = 0; nlen = 0; }
      publish((int)((it + 2) % NM), wn, nb, nlen);
    }
    __syncthreads();  // A
  }
  if (tid == 0 && my_entries) atomicAdd(P.out_distinct, my_entries);
  if (P.hist) hist_flush(s_hist, P, tid);
}

// Every raw run (refine_to_run) has its segments start on 16-byte boundaries and an EMPTY_MIX entry behind every segment of odd
// length, so that phase B may copy whole 16-byte units.  The speculative layout has room for that entry because it gives every
// partition an even capacity; the exact layout because its segment starts are the prefix of the lengths rounded up to even
// (even_lengths_kernel).
__global__ void pad_segments_kernel(uint64_t *keys, const uint64_t *__restrict__ seg_start, const uint64_t *__restrict__ seg_len, uint32_t n_parts) {
  for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n_parts; p += gridDim.x * blockDim.x) {
    const uint64_t len = seg_len[p];
    if (len & 1ull) keys[seg_start[p] + len] = EMPTY_MIX;
  }
}
cudaError_t launch_pad_segments(uint64_t *keys, const uint64_t *seg_start, const uint64_t *seg_len, uint32_t n_parts, cudaStream_t s) {
  if (!n_parts) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  pad_segments_kernel<<<(unsigned)std::min<uint64_t>((n_parts + 255) / 256, (uint64_t)num_sms() * 8), 256, 0, s>>>(keys, seg_start, seg_len, n_parts);
  return cudaGetLastError();
}
__global__ void even_lengths_kernel(const uint64_t *__restrict__ seg_len, uint64_t *even_len, uint32_t n_parts) {
  for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n_parts; p += gridDim.x * blockDim.x) even_len[p] = (seg_len[p] + 1) & ~1ull;
}
cudaError_t launch_even_lengths(const uint64_t *seg_len, uint64_t *even_len, uint32_t n_parts, cudaStream_t s) {
  if (!n_parts) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  even_lengths_kernel<<<(unsigned)std::min<uint64_t>((n_parts + 255) / 256, (uint64_t)num_sms() * 8), 256, 0, s>>>(seg_len, even_len, n_parts);
  return cudaGetLastError();
}

uint32_t sieve_redo_limit_host(uint32_t n_parts) { return sieve_redo_limit_impl(n_parts); }
cudaError_t launch_count_partitions_sieve(const CountParams &P, cudaStream_t s) {
  if (P.n_parts == 0) return cudaSuccess;
  if (!P.redo_list || !P.redo_count || !P.redo_base || !P.redo_len) return cudaErrorInvalidValue;
  if (P.part_cap) {
    if (P.R != 1) return cudaErrorInvalidValue;
    cudaError_t e = cudaFuncSetAttribute(count_partitions_sieve_in_place_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SVI_SMEM);
    if (e != cudaSuccess) return e;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    count_partitions_sieve_in_place_kernel<<<(unsigned)std::min<uint64_t>(P.n_parts, (uint64_t)num_sms() * SVI_CTAS_PER_SM), SVI_THREADS,
                                             SVI_SMEM, s>>>(P);
    return cudaGetLastError();
  }
  auto kern = P.R == 1 ? count_partitions_sieve_tma_kernel<true> : count_partitions_sieve_tma_kernel<false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SVT_SMEM);
  if (e != cudaSuccess) return e;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  kern<<<(unsigned)std::min<uint64_t>(P.n_parts, (uint64_t)num_sms() * 2), SVT_THREADS, SVT_SMEM, s>>>(P);
  return cudaGetLastError();
}

cudaError_t launch_count_partitions_smem(const CountParams &P, bool weighted, bool direct, cudaStream_t s) {
  if (P.n_parts == 0) return cudaSuccess;
  const size_t smem = (size_t)SMEM_TABLE_SLOTS * 14;  // u64 keys + u32 counts + u16 slot lists / output indices
  const unsigned grid = (unsigned)std::min<uint64_t>(P.n_parts, (uint64_t)num_sms() * 2);
  if (weighted && direct) return cudaErrorInvalidValue;
  auto kern = weighted ? count_partitions_smem_kernel<true, false> : direct ? count_partitions_smem_kernel<false, true> : count_partitions_smem_kernel<false, false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  kern<<<grid, SMEM_COUNT_THREADS, smem, s>>>(P);
  return cudaGetLastError();
}

cudaError_t launch_count_partitions(const CountParams &P, unsigned grid, cudaStream_t s) {
  if (P.n_parts == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  count_partitions_kernel<<<grid, COUNT_THREADS, 0, s>>>(P);
  return cudaGetLastError();
}

}  // namespace kmg
