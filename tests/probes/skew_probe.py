"""Throughput and parity on a repeat-rich synthetic genome (satellite arrays, homopolymer runs, a segmental duplication):
the speculative layouts overflow here, so this exercises the sticky exact route, the rows kernels' per-tile fallback and
phase B's weighted / oversized-partition handling at scale.  Run under gpurun; prints one line per case."""
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")  # run from the repository root: python tests/probes/skew_probe.py 1e9 --no-oracle
import krust_b200 as kb  # noqa: E402
from oracle import oracle as orc  # noqa: E402  (checker only)

n = int(float(sys.argv[1])) if len(sys.argv) > 1 else 100_000_000
k = 21
rng = np.random.default_rng(7)
t0 = time.perf_counter()
seq = rng.integers(0, 4, size=n, dtype=np.uint8)
seq = np.frombuffer(b"ACGT", dtype=np.uint8)[seq]
motif = seq[1000:1171].copy()
for pos in rng.integers(0, n - 200_000, size=max(1, n // 2_500_000)):      # satellite arrays: 171-mer x 1000
    seq[pos:pos + 171_000] = np.tile(motif, 1000)
for pos in rng.integers(0, n - 20_000, size=max(1, n // 1_000_000)):       # homopolymer / dinucleotide runs
    seq[pos:pos + 10_000] = ord("A")
    seq[pos + 10_000:pos + 20_000] = np.frombuffer(b"AC" * 5000, dtype=np.uint8)
seg = n // 8
seq[5 * seg:6 * seg] = seq[seg:2 * seg]                                      # segmental duplication (12.5 % of the genome)
seq[rng.integers(0, n, size=n // 100_000)] = ord("N")
offsets = np.linspace(0, n, 33).astype(np.uint64)   # 32 records
print(f"generated {n} bases in {time.perf_counter() - t0:.1f} s", flush=True)

h = torch.from_numpy(seq).pin_memory()
h_np = h.numpy()
with kb.GpuKmerCounter(k) as c:
    best = 1e9
    for it in range(3):
        c.reset()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        c.count_batch(h_np, None, offsets)
        s = c.finalize(True)
        vals, freqs = c.histogram(1)
        best = min(best, time.perf_counter() - t0)
    print(f"{'auto':15s}: {best * 1e3:8.1f} ms  {s['n_windows'] / best / 1e9:6.2f} G k-mers/s  windows {s['n_windows']} distinct {s['n_distinct']} "
          f"max {s['max_count']} consolidations {s['n_grows']} | phase A {s['scan_ns'] / 1e6:.1f} ms, phase B {s['consolidate_ns'] / 1e6:.1f} ms", flush=True)
    gpu_hist = (vals.copy(), freqs.copy())
if "--stream" in sys.argv:
    # the same genome fed record by record with no size hint: the plan is made from the first call alone
    rec = [(int(offsets[i]), int(offsets[i + 1])) for i in range(len(offsets) - 1)]
    with kb.GpuKmerCounter(k) as c:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        per_call = []
        for a, b in rec:
            t1 = time.perf_counter()
            c.count_batch(h_np[a:b], None, np.array([0, b - a], dtype=np.uint64))
            per_call.append((time.perf_counter() - t1) * 1e3)
        print("per-call ms:", " ".join(f"{x:.1f}" for x in per_call), flush=True)
        s2 = c.finalize(True)
        dt = time.perf_counter() - t0
        print(f"streamed in {len(rec)} calls, no hint: {dt * 1e3:8.1f} ms  {s2['n_windows'] / dt / 1e9:6.2f} G k-mers/s  distinct {s2['n_distinct']} "
              f"consolidations {s2['n_grows']} | phase A {s2['scan_ns'] / 1e6:.1f} ms, phase B {s2['consolidate_ns'] / 1e6:.1f} ms", flush=True)
        assert s2["n_distinct"] == s["n_distinct"] and s2["n_windows"] == s["n_windows"]
if "--stream-part" in sys.argv:
    # 128 calls on the partitioned path: with and without a size hint (31 runs pending -> LSM-style consolidation)
    from krust_b200 import _lib
    cuts = np.linspace(0, n, 129).astype(np.int64)
    for hint in (n, 0):
        with kb.GpuKmerCounter(k, flags=_lib.KMG_FLAG_FORCE_PARTITIONED, expected_distinct=hint) as c:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for a, b in zip(cuts[:-1], cuts[1:]):
                a2 = max(0, a - (k - 1)) if a else 0   # callers of a chunked feed overlap by k-1 themselves; here: separate records
                c.count_batch(h_np[a:b], None, np.array([0, b - a], dtype=np.uint64))
            s3 = c.finalize(True)
            dt = time.perf_counter() - t0
            print(f"128 calls, partitioned, hint {hint:>10}: {dt * 1e3:8.1f} ms  {s3['n_windows'] / dt / 1e9:6.2f} G k-mers/s  distinct {s3['n_distinct']} "
                  f"consolidations {s3['n_grows']} | phase A {s3['scan_ns'] / 1e6:.1f} ms, phase B {s3['consolidate_ns'] / 1e6:.1f} ms", flush=True)
if "--no-oracle" in sys.argv:
    sys.exit(0)
t0 = time.perf_counter()
ow, od, ok, oc = orc.reference_path_count(k, seq, None, offsets, None, export=True)   # all host cores
ov, of = orc.histogram(oc, 1)
print(f"oracle: {time.perf_counter() - t0:.1f} s, windows {ow} distinct {len(ok)}", flush=True)
assert ow == s["n_windows"] and len(ok) == s["n_distinct"], "PARITY FAILURE (summary)"
assert (ov == gpu_hist[0]).all() and (of == gpu_hist[1]).all(), "PARITY FAILURE (histogram)"
print("parity OK (windows, distinct, count-of-counts)")
