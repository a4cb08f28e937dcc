// sm_100a kernels of libkmerust_gpu: ingest (ASCII -> 2-bit + masks), tile scan with rolling
// forward / reverse-complement words, open-addressing HBM table upsert, direct-indexed 4^k
// counters, owner bucketing, compaction, count-of-counts histogram.
//
// Reference behaviour reproduced (paths relative to the kmerust repository):
//   src/kmer.rs:21-47, :266-286, :304-312, :348-390   validate / pack / canonical
//   src/run.rs:526-571                                  window predicate + upsert
//   src/run.rs:447-450, src/histogram.rs:88-116         min-count filter, histogram
// All arithmetic is integer; results are bit-exact by construction (tests/ prove it against oracle/).
#include "kmg_kernels.h"

#include <algorithm>
#include <atomic>
#include <cstdlib>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <thrust/iterator/transform_iterator.h>

#include "../../include/kmerust_gpu.h"
#include "kmg_device.cuh"

namespace kmg {

// =================================================================================================
// K8 ingest: ASCII (+ Phred+33 quality) -> packed bases + valid mask.  One thread per 32-base word.
// =================================================================================================
__device__ __forceinline__ void ingest4(uint32_t x, uint32_t q, bool use_q, uint32_t thr4, uint64_t &bases, uint32_t &valid) {
  // x: 4 ASCII bytes, byte 0 = earliest base.  code = ((b>>1)^(b>>2))&3 maps A/a,C/c,G/g,T/t -> 0,1,2,3
  // (src/kmer.rs:21-32); validity = upper-cased byte is one of A C G T (src/kmer.rs:270-277).
  uint32_t c = ((x >> 1) ^ (x >> 2)) & 0x03030303u;
  uint32_t u = x & 0xDFDFDFDFu;
  uint32_t ok = __vcmpeq4(u, 0x41414141u) | __vcmpeq4(u, 0x43434343u) | __vcmpeq4(u, 0x47474747u) | __vcmpeq4(u, 0x54545454u);
  if (use_q) ok &= __vcmpgeu4(q, thr4);  // q >= saturating_add(min_quality, 33)  (src/run.rs:538, :544)
  uint32_t packed8 = (c * 0x40100401u) >> 24;                    // c0<<6 | c1<<4 | c2<<2 | c3
  uint32_t nib = ((ok & 0x01010101u) * 0x80402010u) >> 28;        // v0<<3 | v1<<2 | v2<<1 | v3
  bases = (bases << 8) | packed8;
  valid = (valid << 4) | nib;
}

__global__ void __launch_bounds__(256) ingest_kernel(const uint8_t *__restrict__ seq, const uint8_t *__restrict__ qual,
                                                     uint64_t n_bytes, uint32_t thr, uint64_t n_words_total,
                                                     uint64_t *__restrict__ bases_out, uint32_t *__restrict__ valid_out) {
  const bool use_q = qual != nullptr;
  const uint32_t thr4 = thr * 0x01010101u;
  for (uint64_t w = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; w < n_words_total;
       w += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t b0 = w * 32;
    uint64_t bases = 0;
    uint32_t valid = 0;
    if (b0 + 32 <= n_bytes) {
      const uint4 *p = reinterpret_cast<const uint4 *>(seq + b0);
      uint4 s0 = __ldg(p), s1 = __ldg(p + 1);
      uint4 q0 = make_uint4(0, 0, 0, 0), q1 = q0;
      if (use_q) {
        const uint4 *qp = reinterpret_cast<const uint4 *>(qual + b0);
        q0 = __ldg(qp); q1 = __ldg(qp + 1);
      }
      ingest4(s0.x, q0.x, use_q, thr4, bases, valid); ingest4(s0.y, q0.y, use_q, thr4, bases, valid);
      ingest4(s0.z, q0.z, use_q, thr4, bases, valid); ingest4(s0.w, q0.w, use_q, thr4, bases, valid);
      ingest4(s1.x, q1.x, use_q, thr4, bases, valid); ingest4(s1.y, q1.y, use_q, thr4, bases, valid);
      ingest4(s1.z, q1.z, use_q, thr4, bases, valid); ingest4(s1.w, q1.w, use_q, thr4, bases, valid);
    } else if (b0 < n_bytes) {
      for (int g = 0; g < 8; ++g) {
        uint32_t x = 0, q = 0;
        for (int j = 0; j < 4; ++j) {
          uint64_t i = b0 + g * 4 + j;
          if (i < n_bytes) {
            x |= (uint32_t)seq[i] << (8 * j);
            if (use_q) q |= (uint32_t)qual[i] << (8 * j);
          }
        }
        ingest4(x, q, use_q, thr4, bases, valid);  // bytes past the end are 0 -> invalid
      }
    }
    bases_out[LEAD_BASE_WORDS + w] = bases;
    valid_out[LEAD_MASK_WORDS + w] = valid;
  }
}

__global__ void start_bits_kernel(const uint64_t *__restrict__ offsets, uint64_t n_records, uint64_t base_offset,
                                  uint64_t n_bytes, uint32_t *__restrict__ start_out) {
  for (uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; r < n_records;
       r += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t o = offsets[r];
    if (o < base_offset) continue;
    o -= base_offset;
    if (o == 0 || o >= n_bytes) continue;  // position 0 has no predecessor; trailing empty records
    atomicOr(&start_out[LEAD_MASK_WORDS + (o >> 5)], 1u << (31 - (uint32_t)(o & 31)));
  }
}

__global__ void synth_uniform_kernel(uint64_t seed, uint64_t first_base, uint64_t n, uint8_t *__restrict__ out) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t g = first_base + i;
    uint64_t x = seed * 0x9E3779B97F4A7C15ull + (g >> 5);
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    x ^= x >> 31;
    out[i] = "ACGT"[(x >> (62 - 2 * (g & 31))) & 3];
  }
}

// Synthetic READS (test / bench helper, SURVEY.md 8d: R20M for C3, R200M for C5).  Same counter-based specification as
// oracle/kmer_oracle.c orc_synth_reads (written from the spec in that file's comment, not shared code): one thread per base.
__device__ __forceinline__ uint64_t splitmix64_dev(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
__device__ __forceinline__ uint32_t synth_genome_code(uint64_t g) {
  return (uint32_t)(splitmix64_dev(42ull * 0x9E3779B97F4A7C15ull + (g >> 5)) >> (62 - 2 * (g & 31))) & 3u;
}
__global__ void synth_reads_kernel(uint64_t seed, uint32_t profile, uint64_t first_read, uint64_t n_reads, uint8_t *__restrict__ seq,
                                   uint8_t *__restrict__ qual) {
  constexpr uint32_t L = 150;
  constexpr uint64_t GOLD = 0x9E3779B97F4A7C15ull, GENOME = 100000000ull;
  const uint64_t n = n_reads * L;
  for (uint64_t x = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; x < n; x += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t rr = x / L, r = first_read + rr;
    const uint32_t i = (uint32_t)(x - rr * L);
    const uint64_t a = splitmix64_dev(seed * GOLD + 2 * r), b = splitmix64_dev(seed * GOLD + 2 * r + 1);
    const uint64_t h = splitmix64_dev((seed ^ 0xABCDEFull) * GOLD + 256 * r + i);
    uint32_t code;
    if (profile == 5 && ((b >> 1) % 10) == 0) {  // satellite read
      const uint32_t u = (uint32_t)((b >> 8) % 64), ulen = u == 0 ? 1u : u == 1 ? 2u : 3u + u % 29u;
      const uint32_t j = ((uint32_t)((b >> 16) % ulen) + i) % ulen;
      code = u == 0 ? 0u : u == 1 ? (j & 1u) : (uint32_t)(splitmix64_dev(0x5A7E111Eull + u) >> (62 - 2 * j)) & 3u;
    } else {
      const uint64_t start = ((a >> 32) * (GENOME - L + 1)) >> 32;
      code = (b & 1) ? 3u - synth_genome_code(start + (L - 1 - i)) : synth_genome_code(start + i);
    }
    if ((h & 0xFFFF) < (profile == 3 ? 655u : 328u)) code = (code + 1u + (uint32_t)((h >> 16) & 0xFF) % 3u) & 3u;
    uint8_t base = "ACGT"[code], q = 'I';
    if (profile == 3) {
      const uint32_t npos = (uint32_t)((b >> 16) % (L - 9));
      if (((h >> 24) & 0xFFFF) < 328u || (((b >> 1) % 100) == 0 && i >= npos && i < npos + 10)) base = 'N';
      const uint32_t uq = (uint32_t)((h >> 40) & 0xFFFF);
      const bool late = i >= L - 30;
      const uint32_t t0 = late ? 3932u : 1311u, t1 = late ? 19661u : 6554u, t2 = late ? 32768u : 19661u;
      q = (uint8_t)(33 + (uq < t0 ? 2 : uq < t1 ? 11 : uq < t2 ? 25 : 37));
    }
    seq[x] = base;
    if (qual) qual[x] = q;
  }
}

// =================================================================================================
// Tile pipeline: double-buffered TMA bulk copies of the packed stream into shared memory.
// =================================================================================================
struct TileSmem {
  uint64_t bases[TILE_WORDS + LEAD_BASE_WORDS];
  uint32_t valid[TILE_WORDS + LEAD_MASK_WORDS];
  uint32_t start[TILE_WORDS + LEAD_MASK_WORDS];
};
constexpr uint32_t TILE_BASE_BYTES = (TILE_WORDS + LEAD_BASE_WORDS) * 8;
constexpr uint32_t TILE_MASK_BYTES = (TILE_WORDS + LEAD_MASK_WORDS) * 4;

__device__ __forceinline__ void issue_tile(const ScanInput &in, TileSmem *dst, uint64_t *bar, uint64_t tile) {
  // arrays carry LEAD_* zero words, so word index (tile*TILE_WORDS - lead) is array index tile*TILE_WORDS
  const uint64_t w0 = tile * TILE_WORDS;
  uint32_t bytes = TILE_BASE_BYTES + TILE_MASK_BYTES + (in.start ? TILE_MASK_BYTES : 0);
  mbar_expect_tx(bar, bytes);
  tma_load_1d(dst->bases, in.bases + w0, TILE_BASE_BYTES, bar);
  tma_load_1d(dst->valid, in.valid + w0, TILE_MASK_BYTES, bar);
  if (in.start) tma_load_1d(dst->start, in.start + w0, TILE_MASK_BYTES, bar);
}

// Walk the 32 windows ending in word `i` of the staged tile, handing groups of G canonical keys to
// the emitter.  fwd/rc are rolled one base at a time; canonical = min(fwd, rc) which equals the
// reference's bytewise lexicographic choice (src/kmer.rs:348-365) because A<C<G<T in both orders.
template <int G, class Emit>
__device__ __forceinline__ uint32_t scan_word(const TileSmem *ts, int i, int k, bool has_start, Emit &emit) {
  const uint64_t prev = ts->bases[LEAD_BASE_WORDS + i - 1];
  const uint64_t cur = ts->bases[LEAD_BASE_WORDS + i];
  const uint32_t vprev = ts->valid[LEAD_MASK_WORDS + i - 1], vcur = ts->valid[LEAD_MASK_WORDS + i];
  uint32_t sprev = 0, scur = 0;
  if (has_start) { sprev = ts->start[LEAD_MASK_WORDS + i - 1]; scur = ts->start[LEAD_MASK_WORDS + i]; }
  const uint32_t ok = window_ok_mask(vprev, vcur, sprev, scur, k, has_start);
  if (ok == 0) return 0;
  const uint64_t mask = kmer_mask(k);
  const int rc_shift = 2 * (k - 1);
  uint64_t fwd = prev & mask;
  uint64_t rc = revcomp(fwd, k);
#pragma unroll
  for (int g = 0; g < 32 / G; ++g) {
    uint64_t key[G];
    uint32_t okg = 0;
#pragma unroll
    for (int j = 0; j < G; ++j) {
      const int e = g * G + j;
      const uint64_t c = (cur >> (62 - 2 * e)) & 3ull;
      fwd = ((fwd << 2) | c) & mask;
      rc = (rc >> 2) | ((3ull - c) << rc_shift);
      key[j] = fwd < rc ? fwd : rc;
      okg |= ((ok >> (31 - e)) & 1u) << j;
    }
    if (okg) emit.template group<G>(key, okg);
  }
  return __popc(ok);
}

// In-thread pre-aggregation: adjacent (distance 1 and 2) equal keys inside a group are merged, which
// collapses homopolymer and dinucleotide-repeat runs before they reach the atomics.
template <int G>
__device__ __forceinline__ void preaggregate(const uint64_t (&key)[G], uint32_t okg, uint32_t (&cnt)[G], bool enable) {
#pragma unroll
  for (int j = 0; j < G; ++j) cnt[j] = (okg >> j) & 1u;
  if (!enable) return;
#pragma unroll
  for (int j = 1; j < G; ++j)
    if (cnt[j] && cnt[j - 1] && key[j] == key[j - 1]) { cnt[j] += cnt[j - 1]; cnt[j - 1] = 0; }
#pragma unroll
  for (int j = 2; j < G; ++j)
    if (cnt[j] && cnt[j - 2] && key[j] == key[j - 2]) { cnt[j] += cnt[j - 2]; cnt[j - 2] = 0; }
}

// ---- K2: open-addressing table upsert (AoS 16-byte slots: key, count-1) -------------------------------
// A slot stores (key, occurrences - 1): the CAS that claims an empty slot IS the first count, so a new
// key costs one atomic instead of two (the measured HBM-resident ceiling is ~20 G single atomics/s but
// only ~10.5 G CAS+RED pairs/s, profiles/microbench_r1.jsonl).  Duplicates add with one more RED.
__device__ __forceinline__ void table_add_slow(HashTable t, uint64_t key, uint64_t add, uint64_t slot, uint32_t &new_keys,
                                               unsigned long long *full_flag) {
  for (uint64_t probe = 1; probe < t.cap; ++probe) {
    slot = slot + 1 == t.cap ? 0 : slot + 1;
    unsigned long long *kp = reinterpret_cast<unsigned long long *>(t.slots + 2 * slot);
    uint64_t cur = *reinterpret_cast<volatile unsigned long long *>(kp);
    if (cur == EMPTY_KEY) cur = atomicCAS(kp, EMPTY_KEY, key);
    if (cur == EMPTY_KEY) { ++new_keys; if (add > 1) atomicAdd(kp + 1, add - 1); return; }
    if (cur == key) { atomicAdd(kp + 1, add); return; }
  }
  atomicExch(full_flag, 1ull);
}

__device__ __forceinline__ void table_add(HashTable t, uint64_t key, uint64_t add, uint32_t &new_keys,
                                          unsigned long long *full_flag) {
  uint64_t slot = slot_of(key, t.cap);
  unsigned long long *kp = reinterpret_cast<unsigned long long *>(t.slots + 2 * slot);
  uint64_t old = atomicCAS(kp, EMPTY_KEY, key);
  if (old == EMPTY_KEY) { ++new_keys; if (add > 1) atomicAdd(kp + 1, add - 1); }
  else if (old == key) atomicAdd(kp + 1, add);
  else table_add_slow(t, key, add, slot, new_keys, full_flag);
}

struct HashEmit {
  HashTable t;
  unsigned long long *full_flag;
  uint32_t new_keys;
  bool preagg;
  template <int G>
  __device__ __forceinline__ void group(const uint64_t (&key)[G], uint32_t okg) {
    uint32_t cnt[G];
    preaggregate<G>(key, okg, cnt, preagg);
    uint64_t slot[G], old[G];
    // phase 1: all first probes in flight together (memory-level parallelism G per thread)
#pragma unroll
    for (int j = 0; j < G; ++j) {
      old[j] = 0;
      slot[j] = slot_of(key[j], t.cap);
      if (cnt[j]) old[j] = atomicCAS(reinterpret_cast<unsigned long long *>(t.slots + 2 * slot[j]), EMPTY_KEY, key[j]);
    }
    // phase 2: resolve
#pragma unroll
    for (int j = 0; j < G; ++j) {
      if (!cnt[j]) continue;
      unsigned long long *cp = reinterpret_cast<unsigned long long *>(t.slots + 2 * slot[j] + 1);
      if (old[j] == EMPTY_KEY) { ++new_keys; if (cnt[j] > 1) atomicAdd(cp, (unsigned long long)(cnt[j] - 1)); }
      else if (old[j] == key[j]) atomicAdd(cp, (unsigned long long)cnt[j]);
      else table_add_slow(t, key[j], cnt[j], slot[j], new_keys, full_flag);
    }
  }
};

// ---- K3: direct-indexed counters ----------------------------------------------------------------------
struct DenseGlobalEmit {
  unsigned long long *dense;
  bool preagg;
  template <int G>
  __device__ __forceinline__ void group(const uint64_t (&key)[G], uint32_t okg) {
    uint32_t cnt[G];
    preaggregate<G>(key, okg, cnt, preagg);
#pragma unroll
    for (int j = 0; j < G; ++j)
      if (cnt[j]) atomicAdd(dense + key[j], (unsigned long long)cnt[j]);
  }
};
struct DenseSmemEmit {
  uint32_t *hist;  // 4^k u32 counters in shared memory
  template <int G>
  __device__ __forceinline__ void group(const uint64_t (&key)[G], uint32_t okg) {
#pragma unroll
    for (int j = 0; j < G; ++j)
      if ((okg >> j) & 1u) atomicAdd(hist + (uint32_t)key[j], 1u);
  }
};

__device__ __forceinline__ uint64_t warp_sum(uint64_t v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

enum ScanMode { MODE_HASH = 0, MODE_DENSE_GLOBAL = 1, MODE_DENSE_SMEM = 2 };

template <int MODE, int G>
__global__ void __launch_bounds__(SCAN_THREADS) scan_count_kernel(ScanInput in, HashTable table, unsigned long long *dense,
                                                                  unsigned long long *counters, uint32_t flags) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  TileSmem *stages = reinterpret_cast<TileSmem *>(smem_raw);
  __shared__ __align__(8) uint64_t bars[2];
  uint32_t *hist = reinterpret_cast<uint32_t *>(smem_raw + 2 * sizeof(TileSmem));
  const int tid = threadIdx.x;
  const bool has_start = in.start != nullptr;
  const bool preagg = !(flags & 4u);

  if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_fence_init(); }
  if (MODE == MODE_DENSE_SMEM) {
    const uint32_t nbins = 1u << (2 * in.k);
    for (uint32_t b = tid; b < nbins; b += SCAN_THREADS) hist[b] = 0;
  }
  __syncthreads();

  uint64_t windows = 0;
  uint32_t new_keys = 0;
  uint64_t tile = blockIdx.x;
  int stage = 0;
  uint32_t phase0 = 0, phase1 = 0;
  if (tile < in.n_tiles && tid == 0) issue_tile(in, &stages[0], &bars[0], tile);
  for (; tile < in.n_tiles; tile += gridDim.x) {
    const uint64_t next = tile + gridDim.x;
    if (next < in.n_tiles && tid == 0) issue_tile(in, &stages[stage ^ 1], &bars[stage ^ 1], next);
    if (stage == 0) { mbar_wait(&bars[0], phase0); phase0 ^= 1; } else { mbar_wait(&bars[1], phase1); phase1 ^= 1; }
    const TileSmem *ts = &stages[stage];
#pragma unroll 1
    for (int r = 0; r < WORDS_PER_THREAD; ++r) {
      const int i = r * SCAN_THREADS + tid;
      if (MODE == MODE_HASH) {
        HashEmit e{table, counters + CTR_FULL, 0, preagg};
        windows += scan_word<G>(ts, i, in.k, has_start, e);
        new_keys += e.new_keys;
      } else if (MODE == MODE_DENSE_GLOBAL) {
        DenseGlobalEmit e{dense, preagg};
        windows += scan_word<G>(ts, i, in.k, has_start, e);
      } else {
        DenseSmemEmit e{hist};
        windows += scan_word<G>(ts, i, in.k, has_start, e);
      }
    }
    __syncthreads();  // everyone is done with this stage before it is refilled
    stage ^= 1;
  }

  if (MODE == MODE_DENSE_SMEM) {
    const uint32_t nbins = 1u << (2 * in.k);
    for (uint32_t b = tid; b < nbins; b += SCAN_THREADS) {
      uint32_t c = hist[b];
      if (c) atomicAdd(dense + b, (unsigned long long)c);
    }
  }
  windows = warp_sum(windows);
  uint64_t nk = warp_sum(new_keys);
  if ((tid & 31) == 0) {
    if (windows) atomicAdd(counters + CTR_WINDOWS, (unsigned long long)windows);
    if (nk) atomicAdd(counters + CTR_DISTINCT, (unsigned long long)nk);
  }
}

// number of countable windows of a packed stream (masks only): lets the host plan the table / partition count for inputs
// whose quality filter removes most windows (config C3 keeps ~3 % of them) before any key is produced
__global__ void __launch_bounds__(256) count_windows_kernel(const uint32_t *__restrict__ valid, const uint32_t *__restrict__ start,
                                                            uint64_t n_words, int k, unsigned long long *out) {
  uint64_t n = 0;
  for (uint64_t w = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; w < n_words; w += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t vprev = valid[LEAD_MASK_WORDS + w - 1], vcur = valid[LEAD_MASK_WORDS + w];
    uint32_t sprev = 0, scur = 0;
    if (start) { sprev = start[LEAD_MASK_WORDS + w - 1]; scur = start[LEAD_MASK_WORDS + w]; }
    n += __popc(window_ok_mask(vprev, vcur, sprev, scur, k, start != nullptr));
  }
  n = warp_sum(n);
  if ((threadIdx.x & 31) == 0 && n) atomicAdd(out, (unsigned long long)n);
}

// ---- K4: owner / partition bucketing ------------------------------------------------------------------
struct PartCountEmit {
  uint32_t *hist;
  uint32_t n_parts;
  template <int G>
  __device__ __forceinline__ void group(const uint64_t (&key)[G], uint32_t okg) {
#pragma unroll
    for (int j = 0; j < G; ++j)
      if ((okg >> j) & 1u) atomicAdd(hist + part_of(key[j], n_parts), 1u);
  }
};
// Scatter emitter.  The G shared-memory atomics of a group are issued back to back, then the G base loads,
// then the G stores: consuming each atomic's return immediately serialises a thread's 32 atomics on their
// latency (45 % of the stall samples sat right behind the ATOMS in profiles/r1_summary.md).  The cursors hold
// absolute output indices, so the atomic's return value IS the destination: no second shared-memory lookup
// (the scatter kernels are bound by the shared-memory pipe: every access costs ~2.5 wavefronts of bank conflicts).
struct PartScatterEmit {
  uint32_t *cursor;  // smem: ABSOLUTE next index in `out` for each partition (seeded with the tile's reservation)
  uint64_t *out;
  uint32_t n_parts;
  template <int G>
  __device__ __forceinline__ void group(const uint64_t (&key)[G], uint32_t okg) {
    uint32_t p[G], o[G];
#pragma unroll
    for (int j = 0; j < G; ++j) p[j] = part_of(key[j], n_parts);
#pragma unroll
    for (int j = 0; j < G; ++j) { o[j] = 0; if ((okg >> j) & 1u) o[j] = atomicAdd(cursor + p[j], 1u); }
#pragma unroll
    for (int j = 0; j < G; ++j)
      if ((okg >> j) & 1u) __stcs(out + o[j], key[j]);
  }
};

// Synchronously stage one tile (used at pass boundaries where there is nothing to overlap with).
__device__ __forceinline__ void wait_stage(uint64_t *bars, int stage, uint32_t &phase0, uint32_t &phase1) {
  if (stage == 0) { mbar_wait(&bars[0], phase0); phase0 ^= 1; } else { mbar_wait(&bars[1], phase1); phase1 ^= 1; }
}

// ---- sparse inputs: scan + compact.  When a quality filter leaves only a few per cent of the windows (config C3: 2.5 %), the
// partition scatter would still pay its per-sub-tile machinery for every tile.  This kernel only scans -- a word without a
// countable window costs a mask test -- and appends the canonical keys of the survivors to a dense array: staged per sub-tile of
// 8192 windows in shared memory (so the buffer can never overflow), one global reservation and a coalesced copy per sub-tile
// that has keys at all.  The keys then take the ordinary keys -> run path (kmg_api.cu keys_to_run).
constexpr int EMITK_SUB_WORDS = SCAN_THREADS;        // one word per thread and sub-tile
constexpr int EMITK_CAP = EMITK_SUB_WORDS * 32;      // 8192 staged keys (64 KiB)
struct KeyAppendEmit {
  uint64_t *kbuf;  // smem staging
  uint32_t *s_n;   // smem: keys staged so far in this sub-tile
  template <int G>
  __device__ __forceinline__ void group(const uint64_t (&key)[G], uint32_t okg) {
    uint32_t pos = atomicAdd(s_n, (uint32_t)__popc(okg));
#pragma unroll
    for (int j = 0; j < G; ++j) if ((okg >> j) & 1u) kbuf[pos++] = key[j];
  }
};
__global__ void __launch_bounds__(SCAN_THREADS, 2) scan_emit_keys_kernel(ScanInput in, uint64_t *__restrict__ out, unsigned long long *cursor) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  TileSmem *stages = reinterpret_cast<TileSmem *>(smem_raw);
  uint64_t *kbuf = reinterpret_cast<uint64_t *>(smem_raw + 2 * sizeof(TileSmem));
  __shared__ __align__(8) uint64_t bars[2];
  __shared__ uint32_t s_n;
  __shared__ unsigned long long s_gbase;
  const int tid = threadIdx.x;
  const bool has_start = in.start != nullptr;
  if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_fence_init(); s_n = 0; }
  __syncthreads();
  uint64_t tile = blockIdx.x;
  int stage = 0;
  uint32_t phase0 = 0, phase1 = 0;
  if (tile < in.n_tiles && tid == 0) issue_tile(in, &stages[0], &bars[0], tile);
  for (; tile < in.n_tiles; tile += gridDim.x) {
    const uint64_t next = tile + gridDim.x;
    if (next < in.n_tiles && tid == 0) issue_tile(in, &stages[stage ^ 1], &bars[stage ^ 1], next);
    wait_stage(bars, stage, phase0, phase1);
    for (int sub = 0; sub < TILE_WORDS / EMITK_SUB_WORDS; ++sub) {
      KeyAppendEmit e{kbuf, &s_n};
      scan_word<8>(&stages[stage], sub * EMITK_SUB_WORDS + tid, in.k, has_start, e);
      __syncthreads();
      const uint32_t n = s_n;  // block-uniform
      if (n) {
        if (tid == 0) s_gbase = atomicAdd(cursor, (unsigned long long)n);
        __syncthreads();
        const unsigned long long g = s_gbase;
        for (uint32_t i = tid; i < n; i += SCAN_THREADS) out[g + i] = kbuf[i];
        __syncthreads();
        if (tid == 0) s_n = 0;
        __syncthreads();
      }
    }
    __syncthreads();  // everyone is done with this stage before it is refilled
    stage ^= 1;
  }
}

// pass 1 (count_pass_kernel): per-partition totals of the whole launch into part_counts[].
__global__ void __launch_bounds__(SCAN_THREADS) partition_count_kernel(ScanInput in, uint32_t n_parts,
                                                                       unsigned long long *part_counts,
                                                                       unsigned long long *counters) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  TileSmem *stages = reinterpret_cast<TileSmem *>(smem_raw);
  __shared__ __align__(8) uint64_t bars[2];
  uint32_t *hist = reinterpret_cast<uint32_t *>(smem_raw + 2 * sizeof(TileSmem));
  const int tid = threadIdx.x;
  const bool has_start = in.start != nullptr;
  if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_fence_init(); }
  for (uint32_t p = tid; p < n_parts; p += SCAN_THREADS) hist[p] = 0;
  __syncthreads();
  uint64_t windows = 0;
  uint64_t tile = blockIdx.x;
  int stage = 0;
  uint32_t phase0 = 0, phase1 = 0;
  if (tile < in.n_tiles && tid == 0) issue_tile(in, &stages[0], &bars[0], tile);
  for (; tile < in.n_tiles; tile += gridDim.x) {
    const uint64_t next = tile + gridDim.x;
    if (next < in.n_tiles && tid == 0) issue_tile(in, &stages[stage ^ 1], &bars[stage ^ 1], next);
    wait_stage(bars, stage, phase0, phase1);
    PartCountEmit e{hist, n_parts};
#pragma unroll 1
    for (int r = 0; r < WORDS_PER_THREAD; ++r) windows += scan_word<8>(&stages[stage], r * SCAN_THREADS + tid, in.k, has_start, e);
    __syncthreads();
    stage ^= 1;
  }
  for (uint32_t p = tid; p < n_parts; p += SCAN_THREADS) {
    const uint32_t c = hist[p];
    if (c) atomicAdd(part_counts + p, (unsigned long long)c);
  }
  windows = warp_sum(windows);
  if ((tid & 31) == 0 && windows && counters) atomicAdd(counters + CTR_WINDOWS, (unsigned long long)windows);
}

// pass 2: scatter.  part_start[] holds the exclusive prefix of the totals, part_cursor[] starts at zero.
// A CTA works on SUPER consecutive tiles at a time: it histograms them in shared memory, reserves ONE
// contiguous range per partition for the whole super-tile (a single global atomic), then re-scans the
// same tiles (they come from L2 now) and writes the keys into those ranges.  Long per-partition runs
// keep the 8-byte stores mergeable into full sectors in L2; keys are re-derived rather than staged.
// A launch never carries more than 2^32-1 windows, so indices into `out` fit 32 bits.
// pass 2: scatter.  part_start[] holds the exclusive prefix of the totals, part_cursor[] starts at zero.
// Per tile: histogram in shared memory, ONE contiguous reservation per partition (a single global atomic),
// then the tile is re-scanned (it is still in shared memory) and the keys are written into those ranges;
// keys are re-derived rather than staged.  At most 2 CTAs/SM so that the tiles' open output (256 KiB each)
// stays mergeable in L2.  A launch never carries more than 2^32-1 windows, so indices into `out` fit 32 bits.
// (A single-pass variant drawing one L2 atomic per key from per-partition cursors was measured at 162 ms
// against 88 ms for this scheme on C4: a few hundred hot addresses serialise in L2.)
constexpr int SCATTER_THREADS = 512;
__global__ void __launch_bounds__(SCATTER_THREADS, 2) partition_scatter_kernel(ScanInput in, uint32_t n_parts,
                                                                            const unsigned long long *part_start,
                                                                            unsigned long long *part_cursor, uint64_t *out) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  TileSmem *stages = reinterpret_cast<TileSmem *>(smem_raw);
  __shared__ __align__(8) uint64_t bars[2];
  uint32_t *hist = reinterpret_cast<uint32_t *>(smem_raw + 2 * sizeof(TileSmem));
  const int tid = threadIdx.x;
  const bool has_start = in.start != nullptr;
  if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_fence_init(); }
  for (uint32_t p = tid; p < n_parts; p += SCATTER_THREADS) hist[p] = 0;
  __syncthreads();
  uint64_t tile = blockIdx.x;
  int stage = 0;
  uint32_t phase0 = 0, phase1 = 0;
  if (tile < in.n_tiles && tid == 0) issue_tile(in, &stages[0], &bars[0], tile);
  for (; tile < in.n_tiles; tile += gridDim.x) {
    const uint64_t next = tile + gridDim.x;
    if (next < in.n_tiles && tid == 0) issue_tile(in, &stages[stage ^ 1], &bars[stage ^ 1], next);
    wait_stage(bars, stage, phase0, phase1);
    const TileSmem *ts = &stages[stage];
    {
      PartCountEmit e{hist, n_parts};
#pragma unroll 1
      for (int r = 0; r < TILE_WORDS / SCATTER_THREADS; ++r) scan_word<8>(ts, r * SCATTER_THREADS + tid, in.k, has_start, e);
    }
    __syncthreads();
    for (uint32_t p = tid; p < n_parts; p += SCATTER_THREADS) {  // histogram -> absolute cursors
      const uint32_t c = hist[p];
      hist[p] = c ? (uint32_t)(part_start[p] + atomicAdd(part_cursor + p, (unsigned long long)c)) : 0u;
    }
    __syncthreads();
    {
      PartScatterEmit e{hist, out, n_parts};
#pragma unroll 1
      for (int r = 0; r < TILE_WORDS / SCATTER_THREADS; ++r) scan_word<8>(ts, r * SCATTER_THREADS + tid, in.k, has_start, e);
    }
    __syncthreads();
    for (uint32_t p = tid; p < n_parts; p += SCATTER_THREADS) hist[p] = 0;
    __syncthreads();
    stage ^= 1;
  }
}

// pass 2, STAGED variant: measured with ablation switches on an earlier unstaged scatter, 60 % of the scatter pass
// was the stores themselves -- a warp store of 32 keys to 32 different partitions is 32 separate L2 transactions.
// Here each sub-tile's keys are first ranked into a shared-memory staging buffer in partition order, then copied
// out by consecutive lanes: a warp instruction now covers a few contiguous runs (one sector per ~4 keys).
//   per sub-tile: histogram (POPC.INC) -> exclusive prefix over the partitions (staging offsets) + ONE global
//   reservation per partition -> rank pass (shared atomic returns the staging slot) -> coalesced copy-out, the
//   destination recomputed from the staged key itself.
constexpr int STAGE_THREADS = 512;
constexpr int STAGE_SUB_WORDS = 512;                 // 16384 windows per sub-tile
constexpr int STAGE_KEYS = STAGE_SUB_WORDS * 32;     // staging capacity (128 KiB)
// MIXED: what is staged / written is mix64(key) (the partitioned pipeline's internal streams, kmg_device.cuh); otherwise the key
// itself (kmg_extract_keys_device hands keys to the caller).
template <bool MIXED>
struct StageEmit {
  uint32_t *cursor;   // smem: next staging slot of each partition
  uint64_t *staging;  // smem
  uint32_t n_parts;
  template <int G>
  __device__ __forceinline__ void group(const uint64_t (&key)[G], uint32_t okg) {
    uint32_t p[G], o[G];
    uint64_t v[G];
#pragma unroll
    for (int j = 0; j < G; ++j) { const uint64_t m = mix64(key[j]); p[j] = coarse_of_mix(m, n_parts); v[j] = MIXED ? m : key[j]; }
#pragma unroll
    for (int j = 0; j < G; ++j) { o[j] = 0; if ((okg >> j) & 1u) o[j] = atomicAdd(cursor + p[j], 1u); }
#pragma unroll
    for (int j = 0; j < G; ++j)
      if ((okg >> j) & 1u) staging[o[j]] = v[j];
  }
};
// where partition p's share of this sub-tile lands in `out` (see ScanInput::part_cap)
constexpr uint32_t NO_BASE = 0xffffffffu;
__device__ __forceinline__ uint32_t part_reserve(const ScanInput &in, const unsigned long long *part_start, unsigned long long *part_cursor,
                                                 uint32_t p, uint32_t h) {
  if (!h) return 0u;
  const unsigned long long off = atomicAdd(part_cursor + p, (unsigned long long)h);
  if (in.part_cap && off + h > in.part_cap) { atomicExch(in.overflow_flag, 1u); return NO_BASE; }
  return (uint32_t)(part_start[p] + off);
}

// One sub-tile (n_words words starting at w0), exact: histogram -> prefix + one global reservation per partition ->
// rank pass into `staging` -> coalesced copy-out.  hist[] is zero on entry and on exit; ends with a barrier.
template <int THREADS, bool MIXED>
__device__ __forceinline__ void stage_subtile_exact(const TileSmem *ts, int w0, int n_words, const ScanInput &in, bool has_start,
                                                    uint32_t n_parts, const unsigned long long *part_start, unsigned long long *part_cursor,
                                                    uint64_t *out, uint64_t *staging, uint32_t *hist, uint32_t *s_off, uint32_t *g_base,
                                                    uint32_t *s_scan) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  {
    PartCountEmit e{hist, n_parts};
#pragma unroll 1
    for (int w = tid; w < n_words; w += THREADS) scan_word<8>(ts, w0 + w, in.k, has_start, e);
  }
  __syncthreads();
  // exclusive prefix over the partitions: thread t owns the contiguous chunk [t*per, (t+1)*per)
  const uint32_t per = (n_parts + THREADS - 1) / THREADS;
  const uint32_t b0 = min((uint32_t)tid * per, n_parts), b1 = min(b0 + per, n_parts);
  uint32_t mine = 0;
  for (uint32_t p = b0; p < b1; ++p) mine += hist[p];
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
    if (lane == 31) s_scan[THREADS / 32] = inc;  // keys in this sub-tile
  }
  __syncthreads();
  uint32_t run = s_scan[warp] + (incl - mine);
  for (uint32_t p = b0; p < b1; ++p) {
    const uint32_t c = hist[p];
    s_off[p] = run;
    g_base[p] = part_reserve(in, part_start, part_cursor, p, c);
    hist[p] = run;  // becomes the staging cursor
    run += c;
  }
  const uint32_t n_sub = s_scan[THREADS / 32];
  __syncthreads();
  {
    StageEmit<MIXED> e{hist, staging, n_parts};
#pragma unroll 1
    for (int w = tid; w < n_words; w += THREADS) scan_word<8>(ts, w0 + w, in.k, has_start, e);
  }
  __syncthreads();
  for (uint32_t i = tid; i < n_sub; i += THREADS) {  // coalesced copy-out
    const uint64_t key = staging[i];
    const uint32_t p = MIXED ? coarse_of_mix(key, n_parts) : part_of(key, n_parts);
    if (g_base[p] != NO_BASE) __stcs(out + ((uint64_t)g_base[p] + (i - s_off[p])), key);
  }
  __syncthreads();
  for (uint32_t p = tid; p < n_parts; p += THREADS) hist[p] = 0;
  __syncthreads();
}

template <bool MIXED>
__global__ void __launch_bounds__(STAGE_THREADS, 1) partition_scatter_staged_kernel(ScanInput in, uint32_t n_parts,
                                                                                     const unsigned long long *part_start,
                                                                                     unsigned long long *part_cursor, uint64_t *out) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  TileSmem *stages = reinterpret_cast<TileSmem *>(smem_raw);
  __shared__ __align__(8) uint64_t bars[2];
  __shared__ uint32_t s_scan[STAGE_THREADS / 32 + 1];
  uint64_t *staging = reinterpret_cast<uint64_t *>(smem_raw + 2 * sizeof(TileSmem));
  uint32_t *hist = reinterpret_cast<uint32_t *>(staging + STAGE_KEYS);  // histogram, then staging cursors
  uint32_t *s_off = hist + n_parts;                                     // staging offset of each partition
  uint32_t *g_base = s_off + n_parts;                                   // index in `out` of the partition's reservation
  const int tid = threadIdx.x;
  const bool has_start = in.start != nullptr;
  if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_fence_init(); }
  for (uint32_t p = tid; p < n_parts; p += STAGE_THREADS) hist[p] = 0;
  __syncthreads();
  uint64_t tile = blockIdx.x;
  int stage = 0;
  uint32_t phase0 = 0, phase1 = 0;
  if (tile < in.n_tiles && tid == 0) issue_tile(in, &stages[0], &bars[0], tile);
  for (; tile < in.n_tiles; tile += gridDim.x) {
    const uint64_t next = tile + gridDim.x;
    if (next < in.n_tiles && tid == 0) issue_tile(in, &stages[stage ^ 1], &bars[stage ^ 1], next);
    wait_stage(bars, stage, phase0, phase1);
    for (int sub = 0; sub < TILE_WORDS / STAGE_SUB_WORDS; ++sub)
      stage_subtile_exact<STAGE_THREADS, MIXED>(&stages[stage], sub * STAGE_SUB_WORDS, STAGE_SUB_WORDS, in, has_start, n_parts, part_start,
                                         part_cursor, out, staging, hist, s_off, g_base, s_scan);
    stage ^= 1;
  }
}

// pass 2, ROWS variant (up to 2048 partitions): ONE scan of the input.  Every partition owns a row of
// 2^cl key slots in shared memory; a window's key is ranked inside its partition by one shared atomic (with return)
// and dropped into the row, the few keys whose row is full (partition sizes per sub-tile are Poisson around 9/16 of
// a row) go to a small overflow list with their rank.  Then one global reservation per partition and a copy-out
// in which consecutive lanes write consecutive keys of a row.  The staged variant above scans and hashes every window
// twice and was issue bound (4.4 warp-instructions per window, profiles/r1_v4_phaseA_lines.txt).
// 1024 threads, one CTA per SM, sub-tiles of 256 words: a thread owns 8 consecutive windows of one word.
// A sub-tile whose overflow list does not suffice (heavily repeated keys) is redone with the exact staged procedure.
constexpr int ROWS_THREADS = 1024;
constexpr int ROWS_SUB_WORDS = ROWS_THREADS / 4;   // 8192 windows per sub-tile
constexpr int ROWS_SLOTS = 16384;                  // n_parts rows of 2^cl keys (128 KiB; also the staging buffer of the exact route)
constexpr int ROWS_OVERFLOW = 1536;   // keys whose row was full (repeat-rich reads put ~200 per sub-tile there; beyond it the sub-tile takes the exact route)
// the 8 windows ending at bases 8g .. 8g+7 of word i
template <class Emit>
__device__ __forceinline__ void scan_octet(const TileSmem *ts, int i, int g, int k, bool has_start, Emit &emit) {
  const uint64_t prev = ts->bases[LEAD_BASE_WORDS + i - 1];
  const uint64_t cur = ts->bases[LEAD_BASE_WORDS + i];
  const uint32_t vprev = ts->valid[LEAD_MASK_WORDS + i - 1], vcur = ts->valid[LEAD_MASK_WORDS + i];
  uint32_t sprev = 0, scur = 0;
  if (has_start) { sprev = ts->start[LEAD_MASK_WORDS + i - 1]; scur = ts->start[LEAD_MASK_WORDS + i]; }
  // 64 valid bases and no record start among them (the normal case inside a genome): every window ending in this word counts
  const uint32_t okw = ((vprev & vcur) == 0xffffffffu && !(sprev | scur)) ? 0xffffffffu : window_ok_mask(vprev, vcur, sprev, scur, k, has_start);
  const uint32_t ok8 = (okw >> (24 - 8 * g)) & 0xffu;  // window 8g+j at bit 7-j
  if (ok8 == 0) return;
  const uint64_t mask = kmer_mask(k);
  const int rc_shift = 2 * (k - 1), e0 = 8 * g;
  uint64_t fwd = (e0 ? ((prev << (2 * e0)) | (cur >> (64 - 2 * e0))) : prev) & mask;  // the k-mer ending just before base e0
  uint64_t rc = revcomp(fwd, k);
  uint64_t key[8];
  uint32_t okg = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const uint64_t c = (cur >> (62 - 2 * (e0 + j))) & 3ull;
    fwd = ((fwd << 2) | c) & mask;
    rc = (rc >> 2) | ((3ull - c) << rc_shift);
    key[j] = fwd < rc ? fwd : rc;
    okg |= ((ok8 >> (7 - j)) & 1u) << j;
  }
  emit.template group<8>(key, okg);
}

// The inner loops are written against 32-bit shared-space addresses (kmg_device.cuh: atoms_add / sts64_if / copy64_if_lt).  An
// octet whose eight windows all count (the normal case inside a record) is ranked without per-window tests, a row store is one
// predicated STS, overflow keys are handled after the eight stores from a bit mask, the copy-out is three predicated load + store pairs per row.
template <bool MIXED>
struct RowsEmit2 {
  uint32_t cnt_s, rows_s;  // shared-space addresses
  uint64_t *ov_key;
  uint32_t *ov_meta, *ov_n;
  uint32_t n_parts, cap;
  template <int G>
  __device__ __forceinline__ void group(const uint64_t (&key)[G], uint32_t okg) {
    uint32_t p[G], r[G], over = 0;
    uint64_t v[G];
#pragma unroll
    for (int j = 0; j < G; ++j) { const uint64_t m = mix64(key[j]); p[j] = coarse_of_mix(m, n_parts); v[j] = MIXED ? m : key[j]; }
    if (okg == (1u << G) - 1u) {
#pragma unroll
      for (int j = 0; j < G; ++j) r[j] = atoms_add(cnt_s + 4u * p[j], 1u);
#pragma unroll
      for (int j = 0; j < G; ++j) {
        const bool fit = r[j] < cap;
        sts64_if(fit, rows_s + 8u * (p[j] * cap + r[j]), v[j]);
        over |= (fit ? 0u : 1u) << j;
      }
    } else {
#pragma unroll
      for (int j = 0; j < G; ++j) { r[j] = 0; if ((okg >> j) & 1u) r[j] = atoms_add(cnt_s + 4u * p[j], 1u); }
#pragma unroll
      for (int j = 0; j < G; ++j) {
        const bool live = (okg >> j) & 1u, fit = r[j] < cap;
        sts64_if(live && fit, rows_s + 8u * (p[j] * cap + r[j]), v[j]);
        over |= ((live && !fit) ? 1u : 0u) << j;
      }
    }
    if (over) {  // rare: keys whose row was full
#pragma unroll
      for (int j = 0; j < G; ++j) {
        if (!((over >> j) & 1u)) continue;
        const uint32_t o = atomicAdd(ov_n, 1u);
        if (o < (uint32_t)ROWS_OVERFLOW) { ov_key[o] = v[j]; ov_meta[o] = (p[j] << 16) | r[j]; }  // r < 8192, p < 2048
      }
    }
  }
};
template <bool MIXED>
__global__ void __launch_bounds__(ROWS_THREADS, 1) partition_scatter_rows2_kernel(ScanInput in, uint32_t n_parts, uint32_t cap, uint32_t magic,
                                                                                   const unsigned long long *part_start,
                                                                                   unsigned long long *part_cursor, uint64_t *out) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  TileSmem *stages = reinterpret_cast<TileSmem *>(smem_raw);
  __shared__ __align__(8) uint64_t bars[2];
  __shared__ uint32_t s_scan[ROWS_THREADS / 32 + 1], s_ovn;
  uint64_t *rows = reinterpret_cast<uint64_t *>(smem_raw + 2 * sizeof(TileSmem));
  uint64_t *ov_key = rows + ROWS_SLOTS;
  uint32_t *ov_meta = reinterpret_cast<uint32_t *>(ov_key + ROWS_OVERFLOW);
  uint32_t *cnt = ov_meta + ROWS_OVERFLOW, *s_off = cnt + n_parts, *g_base = s_off + n_parts;
  const uint32_t rows_s = smem_u32(rows), cnt_s = smem_u32(cnt), gb_s = smem_u32(g_base);
  const uint32_t n_slots = n_parts * cap;  // x / cap == __umulhi(x, magic) for x < 2^16
  const int tid = threadIdx.x;
  const bool has_start = in.start != nullptr;
  if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_fence_init(); s_ovn = 0; }
  for (uint32_t p = tid; p < n_parts; p += ROWS_THREADS) cnt[p] = 0;
  __syncthreads();
  uint64_t tile = blockIdx.x;
  int stage = 0;
  uint32_t phase0 = 0, phase1 = 0;
  if (tile < in.n_tiles && tid == 0) issue_tile(in, &stages[0], &bars[0], tile);
  for (; tile < in.n_tiles; tile += gridDim.x) {
    const uint64_t next = tile + gridDim.x;
    if (next < in.n_tiles && tid == 0) issue_tile(in, &stages[stage ^ 1], &bars[stage ^ 1], next);
    wait_stage(bars, stage, phase0, phase1);
    const TileSmem *ts = &stages[stage];
    for (int sub = 0; sub < TILE_WORDS / ROWS_SUB_WORDS; ++sub) {
      const int w0 = sub * ROWS_SUB_WORDS;
      {
        RowsEmit2<MIXED> e{cnt_s, rows_s, ov_key, ov_meta, &s_ovn, n_parts, cap};
        scan_octet(ts, w0 + (tid >> 2), tid & 3, in.k, has_start, e);
      }
      __syncthreads();
      const uint32_t n_ov = s_ovn;
      if (n_ov > (uint32_t)ROWS_OVERFLOW) {  // block-uniform: skewed sub-tile, take the exact route
        for (uint32_t p = tid; p < n_parts; p += ROWS_THREADS) cnt[p] = 0;
        __syncthreads();
        stage_subtile_exact<ROWS_THREADS, MIXED>(ts, w0, ROWS_SUB_WORDS, in, has_start, n_parts, part_start, part_cursor, out, rows, cnt, s_off,
                                          g_base, s_scan);
      } else {
        for (uint32_t p = tid; p < n_parts; p += ROWS_THREADS) {
          const uint32_t h = cnt[p];
          g_base[p] = part_reserve(in, part_start, part_cursor, p, h);
          if (g_base[p] == NO_BASE) cnt[p] = 0;  // refused: nothing of this partition is written
        }
        __syncthreads();
        // copy-out, lanes along the rows (contiguous destinations).  Rows of up to 24 slots (more than ~680 partitions): EIGHT LANES PER
        // ROW, the row's size and base fetched once per lane and row, up to three predicated slot copies, no slot -> row division and no
        // loop (the flat walk over all slots cost ~20 instructions per slot visit and 1.4 of 4.4 warp-instr per window,
        // profiles/r2_v1_lines.txt; a half-warp per row with a strided loop was worse still: 2.2).
        // (two slots per lane through one 16-byte row load was measured SLOWER, 44.8 vs 40.9 ms of phase A on C4: the stores of a warp
        //  then stride by 16 bytes and touch twice the sectors)
        if (cap <= 24u) {
          const uint32_t l = tid & 7u;
#pragma unroll 2
          for (uint32_t p = tid >> 3; p < n_parts; p += ROWS_THREADS / 8) {
            const uint32_t c = min(lds32(cnt_s + 4u * p), cap);
            uint64_t *dst = out + (uint64_t)lds32(gb_s + 4u * p) + l;
            const uint32_t row = rows_s + 8u * (p * cap + l);
            sts32_if(l == 0u, cnt_s + 4u * p, 0u);  // all eight lanes have read it (same instruction): the row is handed back clean
            // default cache policy: measured 0.3 ms faster on C4 than streaming (.cs) stores -- the lines are completed by later
            // sub-tiles; and the third pair only when the row needs it: a predicated-off load / store pair still costs its MIO slots (0.5 ms)
            copy64_if_lt<false>(l, c, dst, row);
            copy64_if_lt<false>(l + 8u, c, dst + 8, row + 64u);
            if (c > 16u) copy64_if_lt<false>(l + 16u, c, dst + 16, row + 128u);
          }
        } else {
#pragma unroll 4
          for (uint32_t x = tid; x < n_slots; x += ROWS_THREADS) {
            const uint32_t p = __umulhi(x, magic), e = x - p * cap;
            if (e < cnt[p]) __stcs(out + (uint64_t)g_base[p] + e, rows[x]);
          }
        }
        for (uint32_t o = tid; o < n_ov; o += ROWS_THREADS) {
          const uint32_t meta = ov_meta[o];
          if (g_base[meta >> 16] != NO_BASE) __stcs(out + (uint64_t)g_base[meta >> 16] + (meta & 0xffffu), ov_key[o]);
        }
        if (cap > 24u) {
          __syncthreads();
          for (uint32_t p = tid; p < n_parts; p += ROWS_THREADS) cnt[p] = 0;
        }
      }
      if (tid == 0) s_ovn = 0;
      __syncthreads();
    }
    stage ^= 1;
  }
}

// =================================================================================================
// Table maintenance, weighted inserts, compaction (K5), histogram (K6)
// =================================================================================================
__global__ void table_init_kernel(uint64_t *slots, uint64_t cap, uint64_t empty) {
  ulonglong2 *p = reinterpret_cast<ulonglong2 *>(slots);
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < cap; i += (uint64_t)gridDim.x * blockDim.x)
    p[i] = make_ulonglong2(empty, 0ull);
}

__global__ void insert_keys_kernel(HashTable t, const uint64_t *__restrict__ keys, const uint64_t *__restrict__ counts,
                                   uint64_t n, unsigned long long *counters) {
  uint32_t new_keys = 0;
  uint64_t windows = 0;
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t c = counts ? counts[i] : 1ull;
    if (c == 0) continue;
    table_add(t, keys[i], c, new_keys, counters + CTR_FULL);
    windows += c;
  }
  windows = warp_sum(windows);
  uint64_t nk = warp_sum(new_keys);
  if ((threadIdx.x & 31) == 0) {
    if (windows) atomicAdd(counters + CTR_WINDOWS, (unsigned long long)windows);
    if (nk) atomicAdd(counters + CTR_DISTINCT, (unsigned long long)nk);
  }
}

__global__ void insert_keys_dense_kernel(unsigned long long *dense, const uint64_t *__restrict__ keys,
                                         const uint64_t *__restrict__ counts, uint64_t n, unsigned long long *counters) {
  uint64_t windows = 0;
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t c = counts ? counts[i] : 1ull;
    if (c == 0) continue;
    atomicAdd(dense + keys[i], (unsigned long long)c);
    windows += c;
  }
  windows = warp_sum(windows);
  if ((threadIdx.x & 31) == 0 && windows) atomicAdd(counters + CTR_WINDOWS, (unsigned long long)windows);
}

// re-insert every occupied slot of `from` into `to` (grow / rehash)
__global__ void rehash_kernel(HashTable from, HashTable to, unsigned long long *counters) {
  uint32_t new_keys = 0;
  const ulonglong2 *p = reinterpret_cast<const ulonglong2 *>(from.slots);
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < from.cap; i += (uint64_t)gridDim.x * blockDim.x) {
    ulonglong2 s = p[i];
    if (s.x != EMPTY_KEY) table_add(to, s.x, s.y + 1, new_keys, counters + CTR_FULL);
  }
}

// A "view" unifies both table kinds for the read-side kernels: entry i is (key, count); empty if count == 0.
__device__ __forceinline__ bool view_get(const TableView &v, uint64_t i, uint64_t &key, uint64_t &count) {
  if (v.pair_keys) { key = unmix64(v.pair_keys[i]); count = v.pair_counts[i]; return count != 0; }  // runs hold mixed keys; count 0: filler entry, repeat left in place or slack of a strided layout (any key)
  if (v.dense) { key = i; count = v.dense[i]; return count != 0; }
  ulonglong2 s = reinterpret_cast<const ulonglong2 *>(v.slots)[i];
  key = s.x; count = s.y + 1;  // slots store occurrences - 1
  return s.x != EMPTY_KEY;
}

// stats[0] += #entries with count >= min_count ; stats[1] = max count ; stats[2] += sum of counts (all entries)
__global__ void table_stats_kernel(TableView v, uint64_t min_count, unsigned long long *stats) {
  uint64_t n = 0, mx = 0, sum = 0;
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < v.n; i += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t key, c;
    if (view_get(v, i, key, c)) {
      sum += c;
      if (c >= min_count && v.keeps(key)) ++n;
      mx = c > mx ? c : mx;
    }
  }
  n = warp_sum(n); sum = warp_sum(sum);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { uint64_t other = __shfl_xor_sync(0xffffffffu, mx, o); mx = other > mx ? other : mx; }
  if ((threadIdx.x & 31) == 0) {
    if (n) atomicAdd(stats + 0, (unsigned long long)n);
    if (mx) atomicMax(stats + 1, (unsigned long long)mx);
    if (sum) atomicAdd(stats + 2, (unsigned long long)sum);
  }
}

// K5: stream-compact entries with count >= min_count into (keys_out, counts_out).  Warp-aggregated
// reservation: one atomic per warp per 32 entries.
__global__ void compact_kernel(TableView v, uint64_t min_count, uint64_t *__restrict__ keys_out,
                               uint64_t *__restrict__ counts_out, uint64_t cap_out, unsigned long long *cursor) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  const uint64_t n_round = (v.n + 31) & ~31ull;
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_round; i += stride) {
    uint64_t key = 0, c = 0;
    bool take = i < v.n && view_get(v, i, key, c) && c >= min_count && v.keeps(key);
    const uint32_t ballot = __ballot_sync(0xffffffffu, take);
    if (ballot == 0) continue;
    const int lane = threadIdx.x & 31;
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(cursor, (unsigned long long)__popc(ballot));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (take) {
      const uint64_t o = base + __popc(ballot & ((1u << lane) - 1u));
      if (o < cap_out) { keys_out[o] = key; counts_out[o] = c; }
    }
  }
}

// entries per key bucket (top bits of the 2k-bit key): lets the .kmix writer cut the key space into pieces of bounded size
__global__ void __launch_bounds__(256) key_buckets_kernel(TableView v, int shift, unsigned long long *buckets) {
  __shared__ uint32_t sh[KEY_BUCKETS];
  for (int b = threadIdx.x; b < KEY_BUCKETS; b += blockDim.x) sh[b] = 0;
  __syncthreads();
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < v.n; i += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t key, c;
    if (view_get(v, i, key, c)) atomicAdd(&sh[(uint32_t)(key >> shift) & (KEY_BUCKETS - 1)], 1u);
  }
  __syncthreads();
  for (int b = threadIdx.x; b < KEY_BUCKETS; b += blockDim.x)
    if (sh[b]) atomicAdd(buckets + b, (unsigned long long)sh[b]);
}

// =================================================================================================
// FASTA / FASTQ parsing on the device (replaces the record iteration of bio::io::{fasta,fastq}::Reader as used by
// src/reader.rs:82-247 for well-formed files): raw file bytes -> compacted sequence (+ quality) bytes + record-start marks.
// A chunk always starts at a line start (FASTQ: at a record).  Line kinds: FASTA 0 = sequence, 1 = header ('>' first);
// FASTQ = line number mod 4 (0 header '@', 1 sequence, 2 '+', 3 quality; multi-line FASTQ is left to the host splitter).
// Every sequence / quality line is trim_end()-ed like the reference's parser does (trailing blanks, \r, \n).
// =================================================================================================
__device__ __forceinline__ bool fx_is_ws(uint8_t b) { return b == ' ' || (b >= 9 && b <= 13); }
// seed of the line-kind scan: the kind at a line start, "inherit" (0xff) elsewhere; FASTQ: newline flags for the line counter
__global__ void fx_seed_kernel(const uint8_t *__restrict__ buf, uint64_t n, int is_fastq, uint8_t *__restrict__ seed) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    if (is_fastq) seed[i] = buf[i] == '\n';
    else seed[i] = (i == 0 || buf[i - 1] == '\n') ? (buf[i] == '>' ? 1 : 0) : 0xff;
  }
}
struct FxBit0 { __host__ __device__ __forceinline__ uint32_t operator()(uint8_t k) const { return k == 1; } };
struct FxBit1 { __host__ __device__ __forceinline__ uint32_t operator()(uint8_t k) const { return k == 2; } };
struct FxInherit {  // scan operator: the kind of the most recent line start
  __host__ __device__ __forceinline__ uint8_t operator()(uint8_t a, uint8_t b) const { return b == 0xff ? a : b; }
};
// keep flags: byte i belongs to the compacted sequence (bit 0) / quality (bit 1) stream.
// err bits: 1 header line without its marker, 2 '+' line missing, 4 first line of a FASTA chunk that opens the file is no header
__global__ void fx_keep_kernel(const uint8_t *__restrict__ buf, uint64_t n, int is_fastq, const uint8_t *__restrict__ kind8,
                               const uint32_t *__restrict__ lineno, uint8_t *__restrict__ keep, uint32_t *err) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint8_t b = buf[i];
    const uint32_t kind = is_fastq ? (lineno[i] & 3u) : kind8[i];
    const bool line_start = i == 0 || buf[i - 1] == '\n';
    if (line_start) {
      if (is_fastq && kind == 0 && b != '@') atomicOr(err, 1u);
      if (is_fastq && kind == 2 && b != '+') atomicOr(err, 2u);
    }
    uint8_t k = 0;
    const bool payload = is_fastq ? (kind == 1 || kind == 3) : kind == 0;
    if (payload && b != '\n') {
      bool trailing = false;
      if (fx_is_ws(b)) {  // trim_end: blanks that run up to the end of the line are dropped, interior ones stay (and count as invalid bases)
        uint64_t j = i + 1;
        while (j < n && buf[j] != '\n' && fx_is_ws(buf[j])) ++j;
        trailing = j == n || buf[j] == '\n';
      }
      if (!trailing) k = (is_fastq && kind == 3) ? 2 : 1;
    }
    keep[i] = k;
  }
}
// positions: pos_s[i] / pos_q[i] = kept sequence / quality bytes before i (exclusive prefix sums of the keep bits, by CUB)
__global__ void fx_scatter_kernel(const uint8_t *__restrict__ buf, uint64_t n, int is_fastq, const uint8_t *__restrict__ kind8,
                                  const uint32_t *__restrict__ lineno, const uint8_t *__restrict__ keep, const uint32_t *__restrict__ pos_s,
                                  const uint32_t *__restrict__ pos_q, uint64_t carry, uint64_t total_s, uint8_t *__restrict__ out_seq,
                                  uint8_t *__restrict__ out_qual, uint8_t *__restrict__ out_mark, unsigned long long *n_records, uint32_t *err) {
  unsigned long long recs = 0;
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint8_t k = keep[i];
    if (k == 1) out_seq[carry + pos_s[i]] = buf[i];
    else if (k == 2 && out_qual) out_qual[carry + pos_q[i]] = buf[i];
    if (i == 0 || buf[i - 1] == '\n') {  // a header line opens a record: its first base is the next kept sequence byte
      const uint32_t kind = is_fastq ? (lineno[i] & 3u) : kind8[i];
      if (kind == (is_fastq ? 0u : 1u)) {
        ++recs;
        if (pos_s[i] < total_s) out_mark[carry + pos_s[i]] = 1;
        else atomicOr(err + 1, 1u);  // the record's first base lies in the NEXT chunk: remembered in the word behind the error word
        if (is_fastq && pos_s[i] != pos_q[i]) atomicOr(err, 8u);  // an earlier record's quality length differs from its sequence length
      }
    }
  }
  recs = warp_sum(recs);
  if ((threadIdx.x & 31) == 0 && recs) atomicAdd(n_records, recs);
}
// a record that opened at the very end of the previous chunk starts with this chunk's first new base
__global__ void fx_apply_pending_kernel(uint32_t *pending, uint8_t *mark_at_first_new_base) {
  if (*pending) { *mark_at_first_new_base = 1; *pending = 0; }
}
__global__ void fx_totals_kernel(const uint8_t *keep, const uint32_t *pos_s, const uint32_t *pos_q, uint64_t n, int is_fastq, uint32_t *totals) {
  totals[0] = pos_s[n - 1] + (keep[n - 1] == 1);
  totals[1] = is_fastq ? pos_q[n - 1] + (keep[n - 1] == 2) : 0u;
}
// record-start marks (one byte per base) -> the start bit stream of the packed layout (bit 31 - j%32 of word j/32)
__global__ void fx_marks_to_bits_kernel(const uint8_t *__restrict__ mark, uint64_t n_bases, uint64_t n_words_total, uint32_t *__restrict__ start_out) {
  for (uint64_t w = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; w < n_words_total; w += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t bits = 0;
    const uint64_t b0 = w * 32;
    if (b0 < n_bases) {
      const uint64_t m = n_bases - b0 < 32 ? n_bases - b0 : 32;
      for (uint64_t j = 0; j < m; ++j) bits |= (uint32_t)(mark[b0 + j] != 0) << (31 - j);
      if (w == 0) bits &= 0x7fffffffu;  // position 0 has no predecessor
    }
    start_out[LEAD_MASK_WORDS + w] = bits;
  }
}

// =================================================================================================
// Index queries (replaces KmerIndex::get, src/index.rs:127-131, and the canonicalisation the `query` subcommand does first,
// src/main.rs:254-266): batched look-ups against whichever table the context holds.
// =================================================================================================
// ASCII k-mers (n x k bytes, any case) -> canonical packed keys; ~0 for a k-mer with a non-ACGT byte (never a canonical key)
__global__ void query_pack_kernel(const uint8_t *__restrict__ kmers, uint64_t n, int k, uint64_t *__restrict__ keys) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint8_t *p = kmers + i * (uint64_t)k;
    uint64_t fwd = 0;
    bool ok = true;
    for (int j = 0; j < k; ++j) {
      const uint8_t b = p[j] & 0xDF;
      ok &= b == 'A' || b == 'C' || b == 'G' || b == 'T';
      fwd = (fwd << 2) | (uint64_t)(((p[j] >> 1) ^ (p[j] >> 2)) & 3u);
    }
    const uint64_t rc = revcomp(fwd & kmer_mask(k), k);
    fwd &= kmer_mask(k);
    keys[i] = ok ? (fwd < rc ? fwd : rc) : EMPTY_KEY;
  }
}
// one warp per query: hash table -> probe sequence; dense array -> direct; partitioned run -> the lanes sweep the key's partition
__global__ void __launch_bounds__(256) query_kernel(TableView v, HashTable t, const uint64_t *__restrict__ seg_start, const uint64_t *__restrict__ seg_len,
                                                    uint32_t n_coarse, uint32_t n_sub, uint32_t shard_world, uint32_t shard_rank,
                                                    const uint64_t *__restrict__ keys, uint64_t n, uint64_t *__restrict__ counts) {
  const int lane = threadIdx.x & 31;
  const uint64_t warp0 = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5, n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  for (uint64_t i = warp0; i < n; i += n_warps) {
    const uint64_t key = keys[i];
    uint64_t found = 0;
    if (key == EMPTY_KEY) { if (lane == 0) counts[i] = 0; continue; }
    if (v.dense) {
      if (lane == 0) found = key < v.n ? v.dense[key] : 0;
    } else if (v.pair_keys) {
      const uint64_t m = mix64(key);
      uint32_t g = coarse_of_mix(m, n_coarse * shard_world);
      if (g / n_coarse == shard_rank) {  // a sharded table answers for its own keys only
        const uint64_t p = (uint64_t)(g - shard_rank * n_coarse) * n_sub + sub_of_mix(m, n_sub);
        const uint64_t b = seg_start[p], e = b + seg_len[p];
        for (uint64_t j = b + lane; j < e; j += 32)  // a repeat that phase B left in place holds the key once more, with count 0
          if (v.pair_keys[j] == m) found |= v.pair_counts[j];
      }
    } else if (t.slots && lane == 0) {
      uint64_t slot = slot_of(key, t.cap);
      for (uint64_t probe = 0; probe < t.cap; ++probe) {
        const ulonglong2 sl = reinterpret_cast<const ulonglong2 *>(t.slots)[slot];
        if (sl.x == key) { found = sl.y + 1; break; }
        if (sl.x == EMPTY_KEY) break;
        slot = slot + 1 == t.cap ? 0 : slot + 1;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) found |= __shfl_xor_sync(0xffffffffu, found, o);  // at most one lane holds a non-zero count
    if (lane == 0) counts[i] = found;
  }
}
__global__ void deinterleave_pairs_kernel(const ulonglong2 *__restrict__ in, uint64_t n, uint64_t *__restrict__ keys, uint64_t *__restrict__ counts) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const ulonglong2 r = in[i];
    keys[i] = r.x; counts[i] = r.y;
  }
}

// ---- output formatting on the device (replaces the per-k-mer writeln! of src/run.rs:452-470 / src/builder.rs:406-429 and
// unpack_to_string, src/kmer.rs:431-456): record i of a sorted piece becomes "{kmer}\t{count}\n" (tsv), ">{count}\n{kmer}\n" (fasta)
// or, for json (serde_json::to_string_pretty of the {kmer, count} vector), ",\n" + body with body = "  {\n    \"kmer\": \"{kmer}\",\n
// \"count\": {count}\n  }".  The separator goes in front of a record, so only the first record of the whole output differs (its
// prefix is "\n"): `first` says that record 0 of this piece is that one.  The "[" and the trailer are framing the caller writes.
__device__ __forceinline__ uint32_t dec_digits(uint64_t v) {
  uint32_t d = 1;
  while (v >= 10) { v /= 10; ++d; }
  return d;
}
constexpr uint32_t JSON_HEAD = 17;  // `  {\n    "kmer": "`
constexpr uint32_t JSON_MID = 16;   // `",\n    "count": `
__global__ void text_len_kernel(const uint64_t *__restrict__ counts, uint64_t n, int k, int format, int first, uint64_t *__restrict__ lens) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t fixed = format == KMG_TEXT_FASTA ? 3u : format == KMG_TEXT_TSV ? 2u : (i == 0 && first ? 1u : 2u) + JSON_HEAD + JSON_MID + 4u;
    lens[i] = (uint64_t)k + dec_digits(counts[i]) + fixed;
  }
}
__global__ void text_write_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ counts, const uint64_t *__restrict__ offs,
                                  uint64_t n, int k, int format, int first, uint8_t *__restrict__ out) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t key = keys[i];
    uint64_t cnt = counts[i];
    uint8_t *p = out + offs[i];
    const uint32_t nd = dec_digits(cnt);
    uint8_t *num, *mer;  // where the decimal count and the k-mer go
    if (format == KMG_TEXT_FASTA) {
      num = p + 1; mer = p + 1 + nd + 1;
      p[0] = '>'; p[1 + nd] = '\n'; p[1 + nd + 1 + k] = '\n';
    } else if (format == KMG_TEXT_TSV) {
      num = p + k + 1; mer = p;
      p[k] = '\t'; p[k + 1 + nd] = '\n';
    } else {
      if (!(i == 0 && first)) *p++ = ',';
      const char head[] = "\n  {\n    \"kmer\": \"", mid[] = "\",\n    \"count\": ", tail[] = "\n  }";
      for (uint32_t j = 0; j < JSON_HEAD + 1; ++j) p[j] = (uint8_t)head[j];
      mer = p + JSON_HEAD + 1;
      for (uint32_t j = 0; j < JSON_MID; ++j) mer[k + j] = (uint8_t)mid[j];
      num = mer + k + JSON_MID;
      for (uint32_t j = 0; j < 4; ++j) num[nd + j] = (uint8_t)tail[j];
    }
    for (int d = (int)nd - 1; d >= 0; --d) { num[d] = (uint8_t)('0' + cnt % 10); cnt /= 10; }
    for (int j = 0; j < k; ++j) mer[j] = "ACGT"[(key >> (2 * (k - 1 - j))) & 3];  // base j = (bits >> 2(k-1-j)) & 3 (src/kmer.rs:431-440)
  }
}
// (key, count) SoA -> the 16-byte little-endian records of the .kmix DATA section (src/index.rs:7-23)
__global__ void interleave_pairs_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ counts, uint64_t n, ulonglong2 *__restrict__ out) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
    out[i] = make_ulonglong2(keys[i], counts[i]);
}

// ---- ONE sorted text file from a shard group (kmg_shard_write_text): every rank holds a sorted step of the key space in a staging
// buffer its peers can read; the owner of a piece merges the piece's parts straight out of the peers' memory.
__device__ __forceinline__ uint64_t lower_bound_u64(const uint64_t *a, uint64_t n, uint64_t key) {
  uint64_t lo = 0, hi = n;
  while (lo < hi) {
    const uint64_t mid = (lo + hi) >> 1;
    if (a[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}
struct PieceCuts { uint64_t key[MERGE_MAX_RUNS + 1]; };
__global__ void piece_bounds_kernel(const uint64_t *__restrict__ keys, uint64_t n, PieceCuts cuts, uint32_t n_cuts, uint64_t *__restrict__ out) {
  const uint32_t i = threadIdx.x;
  if (i < n_cuts) out[i] = lower_bound_u64(keys, n, cuts.key[i]);
}

constexpr int MERGE_THREADS = 256;
constexpr int MERGE_TILE = 2048;  // output records per CTA: keys and counts staged in 32 KiB of shared memory
constexpr int MERGE_PER_THREAD = MERGE_TILE / MERGE_THREADS;
// The runs come from different shards, and a key lives on exactly one shard: no key appears in two runs.  So the record at index i
// of run r has the global rank i + sum over q != r of lower_bound_q(key), every output position has exactly one split across the
// runs, and no ties need breaking.  Each CTA writes the fixed output range [d0, d1): it finds where that range starts and ends in
// every run (binary search over i of the rank above, one warp per (boundary, run), lane q searching run q), loads the sub-ranges
// with coalesced (peer) loads into shared memory, and puts every record at its rank inside the tile.
__global__ void __launch_bounds__(MERGE_THREADS) merge_shard_pieces_kernel(MergeRuns R, uint64_t total, uint64_t *__restrict__ keys_out,
                                                                          uint64_t *__restrict__ counts_out, unsigned long long *placed) {
  __shared__ uint64_t s_key[MERGE_TILE], s_cnt[MERGE_TILE];
  __shared__ const uint64_t *s_rk[MERGE_MAX_RUNS], *s_rc[MERGE_MAX_RUNS];
  __shared__ uint64_t s_len[MERGE_MAX_RUNS], s_lo[MERGE_MAX_RUNS], s_hi[MERGE_MAX_RUNS];
  __shared__ uint32_t s_off[MERGE_MAX_RUNS + 1];
  const uint32_t W = R.n_runs;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x < W) { s_rk[threadIdx.x] = R.keys[threadIdx.x]; s_rc[threadIdx.x] = R.counts[threadIdx.x]; s_len[threadIdx.x] = R.len[threadIdx.x]; }
  __syncthreads();
  const uint64_t d0 = blockIdx.x * (uint64_t)MERGE_TILE, d1 = d0 + MERGE_TILE < total ? d0 + MERGE_TILE : total;
  for (uint32_t job = warp; job < 2 * W; job += MERGE_THREADS / 32) {
    const uint32_t r = job % W;
    const uint64_t d = job < W ? d0 : d1;
    uint64_t lo = 0, hi = s_len[r];
    while (lo < hi) {  // warp-uniform: every lane sees the same mid and the same sum
      const uint64_t mid = (lo + hi) >> 1;
      const uint64_t key = s_rk[r][mid];
      const uint64_t below = warp_sum(lane < (int)W && lane != (int)r ? lower_bound_u64(s_rk[lane], s_len[lane], key) : 0);
      if (mid + below < d) lo = mid + 1; else hi = mid;
    }
    if (lane == 0) (job < W ? s_lo : s_hi)[r] = lo;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t o = 0;
    for (uint32_t r = 0; r < W; ++r) { s_off[r] = o; o += (uint32_t)(s_hi[r] - s_lo[r]); }
    s_off[W] = o;  // == d1 - d0
  }
  __syncthreads();
  const uint32_t n = s_off[W];
  for (uint32_t t = threadIdx.x; t < n; t += MERGE_THREADS) {
    uint32_t r = 0;
    while (r + 1 < W && t >= s_off[r + 1]) ++r;
    const uint64_t i = s_lo[r] + (t - s_off[r]);
    s_key[t] = s_rk[r][i];
    s_cnt[t] = s_rc[r][i];
  }
  __syncthreads();
  uint64_t k_[MERGE_PER_THREAD], c_[MERGE_PER_THREAD];
  uint32_t pos[MERGE_PER_THREAD];
#pragma unroll
  for (int j = 0; j < MERGE_PER_THREAD; ++j) {
    const uint32_t t = threadIdx.x + j * MERGE_THREADS;
    pos[j] = ~0u;
    if (t < n) {
      uint32_t r = 0;
      while (r + 1 < W && t >= s_off[r + 1]) ++r;
      const uint64_t key = s_key[t];
      uint32_t p = t - s_off[r];
      for (uint32_t q = 0; q < W; ++q)
        if (q != r) p += (uint32_t)lower_bound_u64(s_key + s_off[q], s_off[q + 1] - s_off[q], key);
      k_[j] = key; c_[j] = s_cnt[t]; pos[j] = p;
    }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < MERGE_PER_THREAD; ++j)
    if (pos[j] < n) { s_key[pos[j]] = k_[j]; s_cnt[pos[j]] = c_[j]; }
  __syncthreads();
  uint64_t asc = 0;
  for (uint32_t t = threadIdx.x; t < n; t += MERGE_THREADS) {
    const uint64_t key = s_key[t];
    keys_out[d0 + t] = key;
    counts_out[d0 + t] = s_cnt[t];
    asc += t == 0 || s_key[t - 1] < key;
  }
  asc = warp_sum(asc);
  if (lane == 0 && asc) atomicAdd(placed, (unsigned long long)asc);
}

// K6: count-of-counts.  Counts below HIST_DENSE_BINS go to dense bins (the first HIST_SMEM_BINS of them
// privatised in shared memory); larger counts are appended to an overflow list (at most
// total_windows / HIST_DENSE_BINS entries can ever land there).
__global__ void __launch_bounds__(256) histogram_kernel(TableView v, uint64_t min_count, unsigned long long *bins,
                                                        uint64_t *overflow, uint64_t overflow_cap,
                                                        unsigned long long *overflow_n) {
  __shared__ uint32_t sh[HIST_SMEM_BINS];
  for (int b = threadIdx.x; b < HIST_SMEM_BINS; b += blockDim.x) sh[b] = 0;
  __syncthreads();
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < v.n; i += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t key, c;
    if (!view_get(v, i, key, c) || c < min_count) continue;
    if (c < HIST_SMEM_BINS) atomicAdd(&sh[c], 1u);
    else if (c < HIST_DENSE_BINS) atomicAdd(bins + c, 1ull);
    else {
      unsigned long long o = atomicAdd(overflow_n, 1ull);
      if (o < overflow_cap) overflow[o] = c;
    }
  }
  __syncthreads();
  for (int b = threadIdx.x; b < HIST_SMEM_BINS; b += blockDim.x)
    if (sh[b]) atomicAdd(bins + b, (unsigned long long)sh[b]);
}

// =================================================================================================
// Host-side launch wrappers
// =================================================================================================
std::atomic<uint64_t> g_launches{0};
uint64_t kernel_launches() { return g_launches.load(std::memory_order_relaxed); }
static int g_num_sms = 0;
int num_sms() {
  if (!g_num_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) g_num_sms = 148;
  }
  return g_num_sms;
}
static inline unsigned grid_for(uint64_t n_items, int threads, int ctas_per_sm) {
  uint64_t want = (n_items + threads - 1) / threads;
  uint64_t cap = (uint64_t)num_sms() * ctas_per_sm;
  if (want < 1) want = 1;
  return (unsigned)(want < cap ? want : cap);
}

cudaError_t launch_ingest(const uint8_t *d_seq, const uint8_t *d_qual, uint64_t n_bytes, uint32_t thr, uint64_t n_words_total,
                          uint64_t *d_bases, uint32_t *d_valid, cudaStream_t s) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  ingest_kernel<<<grid_for(n_words_total, 256, 8), 256, 0, s>>>(d_seq, d_qual, n_bytes, thr, n_words_total, d_bases, d_valid);
  return cudaGetLastError();
}

cudaError_t launch_start_bits(const uint64_t *d_offsets, uint64_t n_records, uint64_t base_offset, uint64_t n_bytes,
                              uint64_t n_words_total, uint32_t *d_start, cudaStream_t s) {
  cudaError_t e = cudaMemsetAsync(d_start, 0, (LEAD_MASK_WORDS + n_words_total) * sizeof(uint32_t), s);
  if (e != cudaSuccess) return e;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  start_bits_kernel<<<grid_for(n_records, 256, 8), 256, 0, s>>>(d_offsets, n_records, base_offset, n_bytes, d_start);
  return cudaGetLastError();
}

cudaError_t launch_synth_uniform(uint64_t seed, uint64_t first_base, uint64_t n, uint8_t *d_out, cudaStream_t s) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  synth_uniform_kernel<<<grid_for(n, 256, 8), 256, 0, s>>>(seed, first_base, n, d_out);
  return cudaGetLastError();
}

cudaError_t launch_count_windows(const uint32_t *d_valid, const uint32_t *d_start, uint64_t n_words, int k, unsigned long long *d_out,
                                 cudaStream_t s) {
  cudaError_t e = cudaMemsetAsync(d_out, 0, sizeof(unsigned long long), s);
  if (e != cudaSuccess || n_words == 0) return e;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  count_windows_kernel<<<grid_for(n_words, 256, 8), 256, 0, s>>>(d_valid, d_start, n_words, k, d_out);
  return cudaGetLastError();
}

cudaError_t launch_synth_reads(uint64_t seed, uint32_t profile, uint64_t first_read, uint64_t n_reads, uint8_t *d_seq, uint8_t *d_qual,
                               cudaStream_t s) {
  if (n_reads == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  synth_reads_kernel<<<grid_for(n_reads * 150, 256, 8), 256, 0, s>>>(seed, profile, first_read, n_reads, d_seq, d_qual);
  return cudaGetLastError();
}

template <class K>
static cudaError_t set_smem(K kernel, size_t bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// canonical keys of all countable windows, appended to d_out from *d_cursor on (d_cursor is NOT reset here)
cudaError_t launch_scan_emit_keys(const ScanInput &in, uint64_t *d_out, unsigned long long *d_cursor, cudaStream_t s) {
  if (in.n_tiles == 0) return cudaSuccess;
  const size_t smem = 2 * sizeof(TileSmem) + (size_t)EMITK_CAP * 8;
  cudaError_t e = set_smem(scan_emit_keys_kernel, smem);
  if (e != cudaSuccess) return e;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  const unsigned grid = (unsigned)std::min<uint64_t>(in.n_tiles, (uint64_t)num_sms() * 2);
  scan_emit_keys_kernel<<<grid, SCAN_THREADS, smem, s>>>(in, d_out, d_cursor);
  return cudaGetLastError();
}

cudaError_t launch_scan_hash(const ScanInput &in, HashTable t, unsigned long long *counters, uint32_t flags, cudaStream_t s) {
  const size_t smem = 2 * sizeof(TileSmem);
  auto kern = scan_count_kernel<MODE_HASH, 8>;
  cudaError_t e = set_smem(kern, smem);
  if (e != cudaSuccess) return e;
  unsigned grid = (unsigned)(in.n_tiles < (uint64_t)num_sms() * SCAN_CTAS_PER_SM ? in.n_tiles : (uint64_t)num_sms() * SCAN_CTAS_PER_SM);
  if (grid == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  kern<<<grid, SCAN_THREADS, smem, s>>>(in, t, nullptr, counters, flags);
  return cudaGetLastError();
}

cudaError_t launch_scan_dense(const ScanInput &in, unsigned long long *dense, unsigned long long *counters, uint32_t flags,
                              cudaStream_t s) {
  unsigned grid = (unsigned)(in.n_tiles < (uint64_t)num_sms() * SCAN_CTAS_PER_SM ? in.n_tiles : (uint64_t)num_sms() * SCAN_CTAS_PER_SM);
  if (grid == 0) return cudaSuccess;
  HashTable none{nullptr, 0};
  if (in.k <= DENSE_SMEM_MAX_K) {
    const size_t smem = 2 * sizeof(TileSmem) + (sizeof(uint32_t) << (2 * in.k));
    auto kern = scan_count_kernel<MODE_DENSE_SMEM, 8>;
    cudaError_t e = set_smem(kern, smem);
    if (e != cudaSuccess) return e;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    kern<<<grid, SCAN_THREADS, smem, s>>>(in, none, dense, counters, flags);
  } else {
    const size_t smem = 2 * sizeof(TileSmem);
    auto kern = scan_count_kernel<MODE_DENSE_GLOBAL, 8>;
    cudaError_t e = set_smem(kern, smem);
    if (e != cudaSuccess) return e;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    kern<<<grid, SCAN_THREADS, smem, s>>>(in, none, dense, counters, flags);
  }
  return cudaGetLastError();
}

bool scan_scatter_supports_cap(uint32_t n_parts) {  // the rows / staged kernels honour ScanInput::part_cap
  const size_t stsmem = 2 * sizeof(TileSmem) + (size_t)STAGE_KEYS * 8 + 3 * (size_t)n_parts * sizeof(uint32_t);
  return n_parts <= (uint32_t)ROWS_SLOTS / 8 || stsmem <= 220 * 1024;
}

cudaError_t launch_scan_partition(const ScanInput &in, uint32_t n_parts, bool scatter, unsigned long long *part_counts,
                                  const unsigned long long *part_start, unsigned long long *part_cursor, uint64_t *out,
                                  unsigned long long *counters, cudaStream_t s, bool mixed) {
  if (in.n_tiles == 0) return cudaSuccess;
  const size_t smem = 2 * sizeof(TileSmem) + (size_t)n_parts * sizeof(uint32_t);
  const uint64_t max_ctas = (uint64_t)num_sms() * (smem > 100 * 1024 ? 1 : smem > 72 * 1024 ? 2 : SCAN_CTAS_PER_SM);
  cudaError_t e;
  const size_t stsmem = 2 * sizeof(TileSmem) + (size_t)STAGE_KEYS * 8 + 3 * (size_t)n_parts * sizeof(uint32_t);
  const size_t rwsmem = 2 * sizeof(TileSmem) + (size_t)ROWS_SLOTS * 8 + (size_t)ROWS_OVERFLOW * 12 + 3 * (size_t)n_parts * sizeof(uint32_t);
  if (scatter && n_parts <= (uint32_t)ROWS_SLOTS / 8) {  // single-scan rows variant
    const uint32_t cap = std::min<uint32_t>((uint32_t)ROWS_SLOTS / n_parts, ROWS_SUB_WORDS * 32);  // mean fill 8192 / (n_parts * cap) ~ 0.5
    const uint32_t magic = (uint32_t)(((1ull << 32) + cap - 1) / cap);
    const unsigned grid = (unsigned)std::min<uint64_t>(in.n_tiles, (uint64_t)num_sms());
    if ((e = mixed ? set_smem(partition_scatter_rows2_kernel<true>, rwsmem) : set_smem(partition_scatter_rows2_kernel<false>, rwsmem)) != cudaSuccess) return e;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (mixed) partition_scatter_rows2_kernel<true><<<grid, ROWS_THREADS, rwsmem, s>>>(in, n_parts, cap, magic, part_start, part_cursor, out);
    else partition_scatter_rows2_kernel<false><<<grid, ROWS_THREADS, rwsmem, s>>>(in, n_parts, cap, magic, part_start, part_cursor, out);
  } else if (scatter && stsmem <= 220 * 1024) {  // staged variant (> 2048 partitions)
    const unsigned grid = (unsigned)std::min<uint64_t>(in.n_tiles, (uint64_t)num_sms());
    if ((e = mixed ? set_smem(partition_scatter_staged_kernel<true>, stsmem) : set_smem(partition_scatter_staged_kernel<false>, stsmem)) != cudaSuccess) return e;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (mixed) partition_scatter_staged_kernel<true><<<grid, STAGE_THREADS, stsmem, s>>>(in, n_parts, part_start, part_cursor, out);
    else partition_scatter_staged_kernel<false><<<grid, STAGE_THREADS, stsmem, s>>>(in, n_parts, part_start, part_cursor, out);
  } else if (scatter && mixed) {
    return cudaErrorInvalidValue;  // > 5100-ish partitions with mixed output: no kernel variant (the plan never asks for it)
  } else if (scatter) {
    if ((e = set_smem(partition_scatter_kernel, smem)) != cudaSuccess) return e;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    const uint64_t ctas = (uint64_t)num_sms() * 2;
    partition_scatter_kernel<<<(unsigned)std::min(in.n_tiles, ctas), SCATTER_THREADS, smem, s>>>(in, n_parts, part_start, part_cursor, out);
  } else {
    if ((e = set_smem(partition_count_kernel, smem)) != cudaSuccess) return e;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    partition_count_kernel<<<(unsigned)std::min(in.n_tiles, max_ctas), SCAN_THREADS, smem, s>>>(in, n_parts, part_counts, counters);
  }
  return cudaGetLastError();
}

cudaError_t launch_table_init(HashTable t, cudaStream_t s, uint64_t empty) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  table_init_kernel<<<grid_for(t.cap, 256, 8), 256, 0, s>>>(t.slots, t.cap, empty);
  return cudaGetLastError();
}
cudaError_t launch_insert_keys(HashTable t, const uint64_t *d_keys, const uint64_t *d_counts, uint64_t n,
                               unsigned long long *counters, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  insert_keys_kernel<<<grid_for(n, 256, 8), 256, 0, s>>>(t, d_keys, d_counts, n, counters);
  return cudaGetLastError();
}
cudaError_t launch_insert_keys_dense(unsigned long long *dense, const uint64_t *d_keys, const uint64_t *d_counts, uint64_t n,
                                     unsigned long long *counters, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  insert_keys_dense_kernel<<<grid_for(n, 256, 8), 256, 0, s>>>(dense, d_keys, d_counts, n, counters);
  return cudaGetLastError();
}
cudaError_t launch_rehash(HashTable from, HashTable to, unsigned long long *counters, cudaStream_t s) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  rehash_kernel<<<grid_for(from.cap, 256, 8), 256, 0, s>>>(from, to, counters);
  return cudaGetLastError();
}
cudaError_t launch_table_stats(const TableView &v, uint64_t min_count, unsigned long long *d_stats3, cudaStream_t s) {
  cudaError_t e = cudaMemsetAsync(d_stats3, 0, 3 * sizeof(unsigned long long), s);
  if (e != cudaSuccess) return e;
  if (v.n == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  table_stats_kernel<<<grid_for(v.n, 256, 8), 256, 0, s>>>(v, min_count, d_stats3);
  return cudaGetLastError();
}
cudaError_t launch_compact(const TableView &v, uint64_t min_count, uint64_t *d_keys, uint64_t *d_counts, uint64_t cap_out,
                           unsigned long long *d_cursor, cudaStream_t s) {
  cudaError_t e = cudaMemsetAsync(d_cursor, 0, sizeof(unsigned long long), s);
  if (e != cudaSuccess) return e;
  if (v.n == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  compact_kernel<<<grid_for(v.n, 256, 8), 256, 0, s>>>(v, min_count, d_keys, d_counts, cap_out, d_cursor);
  return cudaGetLastError();
}
cudaError_t launch_key_buckets(const TableView &v, int shift, unsigned long long *d_bucket_counts, cudaStream_t s) {
  cudaError_t e = cudaMemsetAsync(d_bucket_counts, 0, KEY_BUCKETS * sizeof(unsigned long long), s);
  if (e != cudaSuccess || v.n == 0) return e;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  key_buckets_kernel<<<grid_for(v.n, 256, 4), 256, 0, s>>>(v, shift, d_bucket_counts);
  return cudaGetLastError();
}
// One parse pass over n raw bytes (device).  tmp layout is managed by the caller: seed/kind (n bytes), keep (n bytes), lineno / pos_s / pos_q
// (n u32 each), scan scratch.  Totals (kept sequence / quality bytes) come back through d_totals[2] (u32), records are ADDED to *d_n_records.
cudaError_t launch_fastx_parse(const uint8_t *d_buf, uint64_t n, int is_fastq, uint8_t *d_kind, uint8_t *d_keep, uint32_t *d_lineno, uint32_t *d_pos_s,
                               uint32_t *d_pos_q, void *d_scan_tmp, size_t scan_tmp_bytes, uint64_t carry, uint8_t *d_out_seq, uint8_t *d_out_qual,
                               uint8_t *d_out_mark, unsigned long long *d_n_records, uint32_t *d_err, uint32_t *h_totals_pinned, cudaStream_t s) {
  if (n == 0) { h_totals_pinned[0] = h_totals_pinned[1] = 0; return cudaSuccess; }
  const unsigned grid = grid_for(n, 256, 8);
  cudaError_t e;
  g_launches.fetch_add(4, std::memory_order_relaxed);
  fx_seed_kernel<<<grid, 256, 0, s>>>(d_buf, n, is_fastq, d_kind);
  size_t tb = scan_tmp_bytes;
  if (is_fastq) e = cub::DeviceScan::ExclusiveSum(d_scan_tmp, tb, d_kind, d_lineno, (int64_t)n, s);           // newlines before i = line number
  else e = cub::DeviceScan::InclusiveScan(d_scan_tmp, tb, d_kind, d_kind, FxInherit(), (int64_t)n, s);         // kind of the current line
  if (e != cudaSuccess) return e;
  fx_keep_kernel<<<grid, 256, 0, s>>>(d_buf, n, is_fastq, d_kind, d_lineno, d_keep, d_err);
  // exclusive prefix sums of the two keep bits (transform iterators would save a pass; these streams are tiny next to the PCIe copy)
  tb = scan_tmp_bytes;
  e = cub::DeviceScan::ExclusiveSum(d_scan_tmp, tb, thrust::make_transform_iterator(d_keep, FxBit0()), d_pos_s, (int64_t)n, s);
  if (e != cudaSuccess) return e;
  if (is_fastq) {
    tb = scan_tmp_bytes;
    e = cub::DeviceScan::ExclusiveSum(d_scan_tmp, tb, thrust::make_transform_iterator(d_keep, FxBit1()), d_pos_q, (int64_t)n, s);
    if (e != cudaSuccess) return e;
  }
  // totals[0..1] = kept sequence / quality bytes (last prefix + last flag); totals[2] is the error word: one 16-byte D2H for the caller
  g_launches.fetch_add(1, std::memory_order_relaxed);
  fx_totals_kernel<<<1, 1, 0, s>>>(d_keep, d_pos_s, d_pos_q, n, is_fastq, d_err - 2);
  e = cudaMemcpyAsync(h_totals_pinned, d_err - 2, 16, cudaMemcpyDeviceToHost, s);
  return e;
}
size_t fastx_scan_tmp_bytes(uint64_t n) {
  size_t a = 0, b = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, a, (const uint8_t *)nullptr, (uint32_t *)nullptr, (int64_t)n);
  cub::DeviceScan::InclusiveScan(nullptr, b, (uint8_t *)nullptr, (uint8_t *)nullptr, FxInherit(), (int64_t)n);
  return std::max(a, b) + 256;
}
cudaError_t launch_fastx_scatter(const uint8_t *d_buf, uint64_t n, int is_fastq, const uint8_t *d_kind, const uint32_t *d_lineno, const uint8_t *d_keep,
                                 const uint32_t *d_pos_s, const uint32_t *d_pos_q, uint64_t carry, uint64_t total_s, uint8_t *d_out_seq, uint8_t *d_out_qual,
                                 uint8_t *d_out_mark, unsigned long long *d_n_records, uint32_t *d_err, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  fx_scatter_kernel<<<grid_for(n, 256, 8), 256, 0, s>>>(d_buf, n, is_fastq, d_kind, d_lineno, d_keep, d_pos_s, d_pos_q, carry, total_s, d_out_seq, d_out_qual,
                                                        d_out_mark, d_n_records, d_err);
  return cudaGetLastError();
}
cudaError_t launch_fastx_apply_pending(uint32_t *d_pending, uint8_t *d_mark_first_new, cudaStream_t s) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  fx_apply_pending_kernel<<<1, 1, 0, s>>>(d_pending, d_mark_first_new);
  return cudaGetLastError();
}
cudaError_t launch_marks_to_bits(const uint8_t *d_mark, uint64_t n_bases, uint64_t n_words_total, uint32_t *d_start, cudaStream_t s) {
  if (n_words_total == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  fx_marks_to_bits_kernel<<<grid_for(n_words_total, 256, 8), 256, 0, s>>>(d_mark, n_bases, n_words_total, d_start);
  return cudaGetLastError();
}

cudaError_t launch_query_pack(const uint8_t *d_kmers, uint64_t n, int k, uint64_t *d_keys, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  query_pack_kernel<<<grid_for(n, 256, 8), 256, 0, s>>>(d_kmers, n, k, d_keys);
  return cudaGetLastError();
}
cudaError_t launch_query(const TableView &v, HashTable t, const uint64_t *d_seg_start, const uint64_t *d_seg_len, uint32_t n_coarse, uint32_t n_sub,
                         uint32_t shard_world, uint32_t shard_rank, const uint64_t *d_keys, uint64_t n, uint64_t *d_counts, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  query_kernel<<<grid_for(n * 32, 256, 8), 256, 0, s>>>(v, t, d_seg_start, d_seg_len, n_coarse, n_sub, shard_world, shard_rank, d_keys, n, d_counts);
  return cudaGetLastError();
}
cudaError_t launch_deinterleave_pairs(const void *d_in, uint64_t n, uint64_t *d_keys, uint64_t *d_counts, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  deinterleave_pairs_kernel<<<grid_for(n, 256, 8), 256, 0, s>>>(static_cast<const ulonglong2 *>(d_in), n, d_keys, d_counts);
  return cudaGetLastError();
}
cudaError_t launch_text_len(const uint64_t *d_counts, uint64_t n, int k, int format, int first, uint64_t *d_lens, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  text_len_kernel<<<grid_for(n, 256, 8), 256, 0, s>>>(d_counts, n, k, format, first, d_lens);
  return cudaGetLastError();
}
cudaError_t launch_text_write(const uint64_t *d_keys, const uint64_t *d_counts, const uint64_t *d_offs, uint64_t n, int k, int format, int first,
                              uint8_t *d_out, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  text_write_kernel<<<grid_for(n, 256, 8), 256, 0, s>>>(d_keys, d_counts, d_offs, n, k, format, first, d_out);
  return cudaGetLastError();
}
cudaError_t launch_interleave_pairs(const uint64_t *d_keys, const uint64_t *d_counts, uint64_t n, void *d_out, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  interleave_pairs_kernel<<<grid_for(n, 256, 8), 256, 0, s>>>(d_keys, d_counts, n, static_cast<ulonglong2 *>(d_out));
  return cudaGetLastError();
}
cudaError_t launch_piece_bounds(const uint64_t *d_keys, uint64_t n, const uint64_t *cut_keys, uint32_t n_cuts, uint64_t *d_out, cudaStream_t s) {
  if (n_cuts == 0 || n_cuts > MERGE_MAX_RUNS + 1) return n_cuts ? cudaErrorInvalidValue : cudaSuccess;
  PieceCuts cuts{};
  for (uint32_t i = 0; i < n_cuts; ++i) cuts.key[i] = cut_keys[i];
  g_launches.fetch_add(1, std::memory_order_relaxed);
  piece_bounds_kernel<<<1, 32, 0, s>>>(d_keys, n, cuts, n_cuts, d_out);
  return cudaGetLastError();
}
cudaError_t launch_merge_shard_pieces(const MergeRuns &R, uint64_t *d_keys_out, uint64_t *d_counts_out, unsigned long long *d_placed,
                                      cudaStream_t s) {
  if (R.n_runs == 0 || R.n_runs > MERGE_MAX_RUNS) return cudaErrorInvalidValue;
  cudaError_t e = cudaMemsetAsync(d_placed, 0, sizeof(unsigned long long), s);
  uint64_t total = 0;
  for (uint32_t r = 0; r < R.n_runs; ++r) total += R.len[r];
  if (e != cudaSuccess || total == 0) return e;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  merge_shard_pieces_kernel<<<(unsigned)((total + MERGE_TILE - 1) / MERGE_TILE), MERGE_THREADS, 0, s>>>(R, total, d_keys_out, d_counts_out, d_placed);
  return cudaGetLastError();
}
cudaError_t launch_histogram(const TableView &v, uint64_t min_count, unsigned long long *d_bins, uint64_t *d_overflow,
                             uint64_t overflow_cap, unsigned long long *d_overflow_n, cudaStream_t s) {
  cudaError_t e = cudaMemsetAsync(d_bins, 0, HIST_DENSE_BINS * sizeof(unsigned long long), s);
  if (e != cudaSuccess) return e;
  if ((e = cudaMemsetAsync(d_overflow_n, 0, sizeof(unsigned long long), s)) != cudaSuccess) return e;
  if (v.n == 0) return cudaSuccess;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  histogram_kernel<<<grid_for(v.n, 256, 4), 256, 0, s>>>(v, min_count, d_bins, d_overflow, overflow_cap, d_overflow_n);
  return cudaGetLastError();
}

// K7: ascending key order == lexicographic order of the unpacked strings (A<C<G<T <-> 0<1<2<3).
// Library radix sort (CUB, ships with the CUDA toolkit) on the already-compacted pairs; not on the
// counting hot path.
cudaError_t sort_pairs(uint64_t *d_keys, uint64_t *d_counts, uint64_t n, int key_bits, cudaStream_t s) {
  if (n < 2) return cudaSuccess;
  uint64_t *alt_k = nullptr, *alt_c = nullptr;
  void *tmp = nullptr;
  size_t tmp_bytes = 0;
  cudaError_t e;
  if ((e = cudaMalloc(&alt_k, n * 8)) != cudaSuccess) return e;
  if ((e = cudaMalloc(&alt_c, n * 8)) != cudaSuccess) { cudaFree(alt_k); return e; }
  cub::DoubleBuffer<uint64_t> kb(d_keys, alt_k), cb(d_counts, alt_c);
  e = cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, kb, cb, n, 0, key_bits, s);
  if (e == cudaSuccess) e = cudaMalloc(&tmp, tmp_bytes ? tmp_bytes : 1);
  if (e == cudaSuccess) e = cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, kb, cb, n, 0, key_bits, s);
  if (e == cudaSuccess && kb.Current() != d_keys) {
    e = cudaMemcpyAsync(d_keys, kb.Current(), n * 8, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_counts, cb.Current(), n * 8, cudaMemcpyDeviceToDevice, s);
  }
  cudaError_t e2 = cudaStreamSynchronize(s);
  cudaFree(tmp); cudaFree(alt_k); cudaFree(alt_c);
  return e != cudaSuccess ? e : e2;
}


// exclusive prefix sum of per-partition sizes (library scan, bookkeeping only); scratch comes from the caller
cudaError_t exclusive_sum_u64(const uint64_t *d_in, uint64_t *d_out, uint64_t n, void *tmp, size_t *tmp_bytes, cudaStream_t s) {
  if (!tmp) { *tmp_bytes = 0; return cub::DeviceScan::ExclusiveSum(nullptr, *tmp_bytes, d_in, d_out, n ? n : 1, s); }
  if (n == 0) return cudaSuccess;
  return cub::DeviceScan::ExclusiveSum(tmp, *tmp_bytes, d_in, d_out, n, s);
}

}  // namespace kmg
