#!/usr/bin/env python
"""Benchmark of the canonical k-mer counting path on the five BASELINE.json configurations.

    python bench.py --gpus N --steps K --warmup W            # our CUDA path, headline config C4 (k=21, 3.1 Gbp)
    python bench.py --config C1|C2|C3|C4|C5 ...              # the other configurations (single GPU unless stated)
    python bench.py --impl reference --gpus N ...            # the reference's CPU algorithm (oracle port), same config

A "step" is one complete counting job: clear the table, ingest + scan the synthetic input (ASCII already in HBM for
`value`; pinned HOST memory for `e2e`), exchange for N>1, table final, the configuration's device-side result.
Prints ONE JSON line on rank 0.  DESIGN.md section "Measurement" explains every field.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "canonical k-mers counted/sec"
UNIT = "kmers/s"
READ_LEN = 150
ATOMIC_CEILING = 20.4e9   # measured random u64 atomics/s on an HBM-resident table (profiles/microbench_r1.jsonl, 8-64 GB tables)

# name -> workload (SURVEY.md 8d: generators, seeds, algorithmic bytes per counted k-mer)
CONFIGS = {
    "C1": dict(k=21, gen="uniform", seed=42, bases=100_000_000, records=100, alg=32.375, result="export",
               what="k=21 canonical k-mer counting, 100 Mbp uniform-random FASTA (G100: 100 records x 1 Mbp), --format tsv"),
    "C2": dict(k=12, gen="uniform", seed=42, bases=100_000_000, records=100, alg=16.375, result="histogram", also_k=5, also_alg=0.375,
               what="k=12 (and k=5) direct-indexed 4^k array on the same 100 Mbp FASTA, --format histogram"),
    "C3": dict(k=31, gen="reads", profile=3, seed=43, reads=20_000_000, min_quality=20, min_count=2, alg=24.5, result="export",
               what="k=31, 20 M x 150 bp FASTQ-shaped reads with N bases, -Q 20, --min-count 2"),
    "C4": dict(k=21, gen="uniform", seed=44, bases=3_100_000_000, records=31, alg=32.375, result="histogram",
               what="k=21 canonical k-mer counting, 3.1 Gbp uniform-random FASTA (31 records x 100 Mbp), hash-sharded across N GPUs"),
    "C5": dict(k=21, gen="reads", profile=5, seed=45, reads=200_000_000, alg=24.4, result="histogram+kmix",
               what="k=21, 200 M x 150 bp skewed reads (~30 Gbp, 10 % satellite / poly-A), --format histogram + .kmix from GPU shards"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C4", choices=sorted(CONFIGS))
    ap.add_argument("--k", type=int, default=0, help="override the configuration's k")
    ap.add_argument("--bases", type=float, default=0, help="override the genome size (uniform generators)")
    ap.add_argument("--reads", type=float, default=0, help="override the number of reads (read generators)")
    ap.add_argument("--records", type=int, default=0)
    ap.add_argument("--cpu-sample-bases", type=float, default=0, help="bases of the CPU sample (0 = largest that fits the time budget, <= 310 Mbp)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--kmix", default="", help="C5: also time kmg_save_kmix(_shard) into this path (needs ~16 B x distinct of disk)")
    ap.add_argument("--flags", type=int, default=0)
    ap.add_argument("--plan-bases", type=float, default=0, help="profiling aid: plan the partitions for this many bases (a slice of C4 then runs "
                    "phase A with the full job's bin counts; phase B sees proportionally smaller partitions)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float64): the summary, the histogram of the "
                         "histogram configurations, and for the export configurations the (filtered, key-sorted) table entries whose "
                         "key %% ceil(bases / 1e6) == 0, keys split into 32-bit halves")
    return ap.parse_args()


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(names, r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        # "under load" = the upper half of the samples (idle samples before/after the region drag the median down)
        load = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def resolve(args) -> dict:
    cfg = dict(CONFIGS[args.config])
    cfg["name"] = args.config
    if args.k:
        cfg["k"] = args.k
    if args.bases and cfg["gen"] == "uniform":
        cfg["bases"] = int(args.bases)
    if args.reads and cfg["gen"] == "reads":
        cfg["reads"] = int(args.reads)
    if args.records and cfg["gen"] == "uniform":
        cfg["records"] = args.records
    if cfg["gen"] == "reads":
        cfg["bases"] = cfg["reads"] * READ_LEN
        cfg["records"] = cfg["reads"]
    return cfg


def expected_windows_uniform(total: int, records: int, k: int) -> int:
    rec_len = total // records
    last = total - rec_len * (records - 1)
    return (records - 1) * max(0, rec_len - k + 1) + max(0, last - k + 1)


# --------------------------------------------------------------------------------------------- --dump-outputs
DUMP_LIMIT_BYTES = 64 << 20
TABLE_SAMPLE_BASES = 1_000_000   # the dumped table sample keeps about one entry per this many input bases


def table_sample(counter, cfg, min_count: int, world: int):
    """The key-space sample key % ceil(bases / 1e6) == 0 of the (key, count) table a caller would export, key-sorted over all
    ranks.  The modulus depends on the arguments only, so two builds sample the same keys."""
    import numpy as np
    m = max(1, -(-cfg["bases"] // TABLE_SAMPLE_BASES))
    keys, counts = counter.export_shard(m, 0, min_count, True)
    if world > 1:
        import torch.distributed as dist
        parts = [None] * world
        dist.all_gather_object(parts, (keys, counts))
        keys = np.concatenate([p[0] for p in parts]); counts = np.concatenate([p[1] for p in parts])
        order = np.argsort(keys, kind="stable")
        keys, counts = keys[order], counts[order]
    return {"table_keys_hi": keys >> np.uint64(32), "table_keys_lo": keys & np.uint64(0xFFFFFFFF), "table_counts": counts}


def write_outputs(out_dir: str, arrays: dict):
    """Each array as out_dir/<name>.npy in float64 (exact: every value is an integer below 2^53)."""
    import numpy as np
    total = sum(8 * np.asarray(a).size for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES} byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a).astype(np.float64))


# --------------------------------------------------------------------------------------------- reference arm
def cpu_sample(cfg, sample_bases: int):
    """A bounded sample of the configuration's own generator for the CPU arm: (seq, qual, offsets, description)."""
    import numpy as np
    from oracle import oracle as orc
    if cfg["gen"] == "uniform":
        rec = max(1, cfg["records"])
        rec_len = max(cfg["k"], sample_bases // rec)
        n = rec_len * rec
        seq = orc.synth_uniform(cfg["seed"], 0, n)
        return seq, None, np.arange(0, n + 1, rec_len, dtype=np.uint64), f"{rec} records x {rec_len} bp uniform ACGT (seed {cfg['seed']})"
    n_reads = max(1, sample_bases // READ_LEN)
    seq, qual, off = orc.synth_reads(cfg["seed"], cfg["profile"], 0, n_reads, want_qual=cfg.get("min_quality") is not None)
    return seq, qual, off, f"{n_reads} reads x {READ_LEN} bp of the profile-{cfg['profile']} read generator (seed {cfg['seed']})"


def run_reference(args, rank: int):
    """The reference's own CPU algorithm (oracle port: the Rust crate cannot be built here) on a bounded sample of the same
    workload, all host threads.  Sample per step: the largest prefix (<= 310 Mbp, what the packed map of a 62 GB host holds)
    such that W/8 + K steps stay within ~3 minutes at the rate measured during warm-up."""
    if rank != 0:
        return
    from oracle import oracle as orc
    cfg = resolve(args)
    cores = os.cpu_count() or 1
    k, q = cfg["k"], cfg.get("min_quality")
    probe = cpu_sample(cfg, 16_000_000)
    t0 = time.perf_counter()
    orc.reference_path_count(k, probe[0], probe[1], probe[2], min_quality=q, threads=cores)
    rate = float(probe[2][-1]) / max(time.perf_counter() - t0, 1e-3)   # bases/s, small-map regime (optimistic)
    if args.cpu_sample_bases:
        n = int(args.cpu_sample_bases)
    else:
        n = int(min(310e6, max(32e6, 0.6 * 180.0 * rate / max(1, args.steps))))
    n = min(n, cfg["bases"])
    seq, qual, offsets, what = cpu_sample(cfg, n)
    for _ in range(max(0, args.warmup - 1)):
        m = max(1, (len(offsets) - 1) // 8)
        orc.reference_path_count(k, seq[: int(offsets[m])], None if qual is None else qual[: int(offsets[m])], offsets[: m + 1], min_quality=q, threads=cores)
    t0 = time.perf_counter()
    windows = 0
    for _ in range(args.steps):
        w, d = orc.reference_path_count(k, seq, qual, offsets, min_quality=q, threads=cores)
        windows += w
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"summary": [w, d]})   # n_windows, n_distinct of the last step
    value = windows / dt
    sample = f"{what}, k={k}, per step; restated reference CPU path (oracle/kmer_oracle.c orc_reference_path_count)"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": f"{cfg['name']}: {cfg['what']}; bounded CPU sample", "k": k, "sample_bases": int(offsets[-1]),
                       "full_bases": cfg["bases"]},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


_REAL_STDOUT = None


def claim_stdout():
    """The driver parses stdout as ONE JSON line: route everything libraries print there (e.g. NCCL's version banner)
    to stderr and keep the real stdout for emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


# --------------------------------------------------------------------------------------------- our arm
def main():
    args = parse_args()
    claim_stdout()
    if os.environ.get("KMG_BENCH_DEBUG"):
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["KMG_BENCH_DEBUG"]), repeat=True, file=sys.stderr)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import krust_b200 as kb  # noqa: F401
    from krust_b200 import _lib
    from krust_b200.dist import GpuShardEngine, ShardedKmerCounter, slice_for_rank

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: krust_b200 has no CPU fallback")
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.load()
    cfg = resolve(args)
    k = cfg["k"]
    reads = cfg["gen"] == "reads"
    min_q = cfg.get("min_quality")
    min_count = cfg.get("min_count", 1)

    # ---- this rank's slice of the synthetic input, generated on the device (same counter-based generators as the oracle)
    if reads:
        r0, r1 = cfg["reads"] * rank // world, cfg["reads"] * (rank + 1) // world
        n_local = (r1 - r0) * READ_LEN
        n_rec_local = r1 - r0
    else:
        a, b = slice_for_rank(cfg["bases"], world, rank, k)
        n_local = b - a
        rec_len = cfg["bases"] // cfg["records"]
        inside = [s - a for s in (r * rec_len for r in range(cfg["records"])) if a < s < b]
        offsets_np = np.array([0] + inside + [n_local], dtype=np.uint64)
        n_rec_local = len(offsets_np) - 1
        exp_windows = expected_windows_uniform(cfg["bases"], cfg["records"], k)
    d_seq = torch.empty(n_local + 64, dtype=torch.uint8, device=dev)[:n_local]
    d_qual = torch.empty(n_local + 64, dtype=torch.uint8, device=dev)[:n_local] if (reads and min_q is not None) else None
    hint = int(cfg["bases"] / world * 1.03) + 1024 if (not reads or min_q is None) else 0   # quality-filtered: planned from the data
    if args.plan_bases:
        hint = int(args.plan_bases / world * 1.03) + 1024
    CH_READS = 1 << 24   # reads per device call (2.5 GB of ASCII): every call leaves a run; large jobs consolidate while streaming
    bb = 0
    if world > 1:   # sharded: one fused scatter + exchange round moves <= batch_bases bases per rank (identical on every rank)
        per_rank = (cfg["bases"] + world - 1) // world + k
        rounds = max(1, round(per_rank / 3.0e8)) if not reads else max(1, -(-per_rank // (CH_READS * READ_LEN)))
        bb = ((per_rank + rounds - 1) // rounds + k + 31) // 32 * 32
    engine = GpuShardEngine(k, dev, min_quality=min_q, expected_distinct=hint, flags=args.flags, batch_bases=bb)
    if reads:
        engine.counter.synth_reads_device(cfg["seed"], cfg["profile"], r0, n_rec_local, d_seq.data_ptr(), d_qual.data_ptr() if d_qual is not None else 0)
        d_off = torch.arange(0, (min(CH_READS, n_rec_local) + 1) * READ_LEN, READ_LEN, dtype=torch.int64, device=dev)
    else:
        engine.counter.synth_uniform_device(cfg["seed"], a, n_local, d_seq.data_ptr())
        d_off = torch.from_numpy(offsets_np.astype(np.int64)).to(dev)
    sharded = ShardedKmerCounter(engine)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def feed_device():
        if not reads:
            sharded.count(d_seq, d_off if n_rec_local > 1 else None,
                          expected_keys_per_rank=int(args.plan_bases) // world if args.plan_bases else exp_windows // world + 1024)
            return
        for c0 in range(0, n_rec_local, CH_READS):
            c1 = min(n_rec_local, c0 + CH_READS)
            sl = slice(c0 * READ_LEN, c1 * READ_LEN)
            sharded.count(d_seq[sl], d_off[: c1 - c0 + 1], None if d_qual is None else d_qual[sl],
                          expected_keys_per_rank=cfg["bases"] // world)

    def device_result():
        """the configuration's result, device side: table final (+ the count-of-counts for the histogram outputs)"""
        engine.finalize(False)
        if "histogram" in cfg["result"]:
            return sharded.histogram(min_count)
        return None

    def step_device():
        engine.reset()
        feed_device()
        return device_result()

    # ---- device-resident timing: W warm-up, then exactly K steps between barriers, CUDA events, max over ranks
    for _ in range(args.warmup):
        step_device()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = L.kmg_kernel_launches()
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        res = step_device()
    ev1.record()
    barrier()
    launches = L.kmg_kernel_launches() - launches0
    clocks = sampler.stop() if rank == 0 else None
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    ms_per_step = ms_total / args.steps
    summary = sharded.finalize()   # global sums over shards
    if reads:
        exp_windows = summary["n_windows"]        # reads: no closed form (N bases, quality filter); parity is checked in tests/
        if min_q is None and exp_windows != cfg["reads"] * (READ_LEN - k + 1):
            raise SystemExit(f"PARITY FAILURE: counted {exp_windows} windows, expected {cfg['reads'] * (READ_LEN - k + 1)}")
    elif summary["n_windows"] != exp_windows:
        raise SystemExit(f"PARITY FAILURE: counted {summary['n_windows']} windows, expected {exp_windows}")
    if args.dump_outputs:   # before the legs below reset the table
        out = {"summary": [summary["n_windows"], summary["n_distinct"], summary["max_count"]]}
        if res is not None:
            out["histogram_values"], out["histogram_frequencies"] = res
        else:
            out.update(table_sample(engine.counter, cfg, min_count, world))
        if rank == 0:
            write_outputs(args.dump_outputs, out)
    local = summary.get("local", summary)
    value = exp_windows / (ms_per_step * 1e-3)

    # ---- roofline.  frac_job: the design-independent algorithmic bytes of SURVEY.md 8(d) over the whole step;
    # frac / achieved: the dominant kernel alone with ITS algorithmic bytes, timed live with CUDA events on its stream
    peak, peak_src = peaks()
    gpu_windows = exp_windows / world   # per-GPU share (strong scaling)
    input_bytes = 0.375 * cfg["bases"] / world
    new_frac = summary["n_distinct"] / max(1, exp_windows)
    if local["path"] == 1:
        alg_job = gpu_windows * (16.0 if k > 6 else 0.0) + input_bytes
    else:
        alg_job = gpu_windows * 24.0 + 8.0 * summary["n_distinct"] / world + input_bytes
    pipeline = None
    if local["path"] == 2:
        # partitioned pipeline: phase A (ingest, A1 partition_scatter_rows2, A2 refine_rows4) and phase B (count_partitions_sieve_tma); reset()
        # clears the timers, so these are the last step's kernels on this rank.  Per k-mer: A1 = 0.375 in + 8 out, A2 = 8 in + 8 out,
        # B = 8 in + 16 out per DISTINCT key.
        a_ms, b_ms = local["scan_ns"] / 1e6, local["consolidate_ns"] / 1e6
        pt = engine.counter.phase_times()
        a1_ms, a2_ms = pt["a1_ns"] / 1e6, pt["a2_ns"] / 1e6
        b_bytes = gpu_windows * 8.0 + 16.0 * summary["n_distinct"] / world
        a1_bytes, a2_bytes = gpu_windows * 8.0 + input_bytes, gpu_windows * 16.0
        gbs = lambda by, ms: by / (ms * 1e-3) / 1e9 if ms else 0.0
        pipeline = {"phase_a_ms": a_ms, "phase_b_ms": b_ms,
                    "phase_a_gbs": gbs(gpu_windows * 24.0 + input_bytes, a_ms), "phase_b_gbs": gbs(b_bytes, b_ms),
                    "a1_ms": a1_ms, "a2_ms": a2_ms,
                    "a1_frac": gbs(a1_bytes, a1_ms) / peak, "a2_frac": gbs(a2_bytes, a2_ms) / peak, "b_frac": gbs(b_bytes, b_ms) / peak,
                    "consolidations": local["n_grows"]}
        # the dominant kernel = the stage with the most device time (its own algorithmic bytes; all three fractions are in `pipeline`)
        stages = [(a1_ms, a1_bytes, "partition_scatter_rows2_kernel (A1: tile scan, canonical k-mers, mix, coarse scatter through shared-memory rows; instruction / "
                                    "shared-memory-pipe bound, not HBM bound; "
                                    "0.375 B in + 8 B out per k-mer)"),
                  (a2_ms, a2_bytes, "refine_rows4_kernel (A2: coarse bins -> fine partitions through shared-memory rows, tiles interleaved over the grid; on N GPUs "
                                    "refine_rows_kernel pulling over NVLink; "
                                    "8 B in + 8 B out per k-mer)"),
                  (b_ms, b_bytes, "count_partitions_sieve_tma_kernel (phase B: one CTA per hash partition, bit-map sieve + bulk copies; compacting "
                                  "count_partitions_smem_kernel for repeat-rich input; 8 B in + 16 B out per k-mer)")]
        kern_ms, alg_bytes, kern_name = max(stages, key=lambda t: t[0])
    else:
        kern_ms = local["kernel_ns"] / 1e6          # scan_count_kernel of the last step (reset() clears the timer)
        alg_bytes = alg_job
        kern_name = ("scan_count_kernel<DENSE> (tile scan + direct-indexed 4^k array: shared-memory privatised for k <= 6, L2 atomics above)"
                     if local["path"] == 1 else "scan_count_kernel<HASH> (tile scan + upsert into one HBM-resident table)")
    # DRAM traffic of the dominant kernel: bytes per k-mer from the committed `ncu --set full` capture (taken on a 5e8-base
    # slice of C4: the full job would make ncu save/restore ~100 GB per pass), scaled to this launch -- not measured in this run
    traffic = None
    try:
        tpk = json.load(open(os.path.join(ROOT, "profiles", "traffic_per_kmer.json")))
        for name, v in tpk.items():
            if name in kern_name:
                traffic = v * gpu_windows
    except Exception:
        traffic = None
    achieved = alg_bytes / (kern_ms * 1e-3) / 1e9 if kern_ms > 0 else 0.0
    job_gbs = alg_job / (ms_per_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": "scaled from the committed ncu --set full capture of a 5e8-base C4 slice (profiles/traffic_per_kmer.json)" if traffic else None,
                "kernel": kern_name, "kernel_ms": kern_ms, "alg_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                "frac_job": job_gbs / peak, "job_gbs": job_gbs, "alg_bytes_per_kmer_job": alg_job / max(1.0, gpu_windows),
                "survey_alg_bytes_per_kmer": cfg["alg"], "new_key_fraction": new_frac,
                "atomic_ceiling_frac": value / world / ATOMIC_CEILING,
                "atomic_ceiling": "20.4 G random u64 atomics/s on an HBM-resident table (profiles/microbench_r1.jsonl): what ONE open-addressing "
                                  "HBM table could reach at best; > 1 means the partitioned design beats that ceiling",
                "pipeline": pipeline}

    # ---- C2 also names k=5: one more device-resident measurement on the same input (shared-memory privatised counters)
    also = None
    if cfg.get("also_k") and world == 1:
        k2 = cfg["also_k"]
        with kb.GpuKmerCounter(k2, device=dev.index) as c2:
            def step2():
                c2.reset()
                c2.count_device(d_seq.data_ptr(), n_local, d_offsets=d_off.data_ptr(), n_records=n_rec_local)
                c2.finalize(False)
                return c2.histogram(1)
            for _ in range(args.warmup):
                step2()
            torch.cuda.synchronize(dev)
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(torch.cuda.current_stream(dev))
            t0 = time.perf_counter()
            for _ in range(args.steps):
                hv2, hf2 = step2()
            torch.cuda.synchronize(dev)
            ms2 = (time.perf_counter() - t0) * 1e3 / args.steps
            s2 = c2.finalize()
            w2 = expected_windows_uniform(cfg["bases"], cfg["records"], k2)
            if s2["n_windows"] != w2 or int((hv2 * hf2).sum()) != w2:
                raise SystemExit("PARITY FAILURE in the k=5 leg")
            km = s2["kernel_ns"] / 1e6
            also = {"k": k2, "value": w2 / (ms2 * 1e-3), "unit": UNIT, "ms_per_step": ms2, "kernel_ms": km, "path": s2["path"],
                    "input_gbs": 0.375 * cfg["bases"] / (km * 1e-3) / 1e9 if km else None,
                    "frac": 0.375 * cfg["bases"] / (km * 1e-3) / 1e9 / peak if km else None,
                    "note": "k=5: 512 canonical keys, counters privatised per CTA in shared memory; bound by shared-memory atomic issue, "
                            "algorithmic bytes = packed input only (0.375 B/k-mer)"}

    # ---- end to end: HOST (pinned) ASCII in, the configuration's result on the HOST, through the public C-ABI calls
    e2e = None
    if not args.no_e2e:
        import psutil
        need = n_local * (2 if d_qual is not None else 1)
        avail = psutil.virtual_memory().available
        frac_e2e = 1.0
        n_e2e_rec, n_e2e = n_rec_local, n_local
        if need > 0.6 * avail:   # C5 at full size wants 30 GB of pinned memory: take the largest prefix the host can pin
            frac_e2e = 0.6 * avail / need
            n_e2e_rec = max(1, int(n_rec_local * frac_e2e))
            n_e2e = n_e2e_rec * READ_LEN if reads else int(n_local * frac_e2e)
        h_seq = torch.empty(n_e2e, dtype=torch.uint8, pin_memory=True)
        h_seq.copy_(d_seq[:n_e2e])
        h_qual = None
        if d_qual is not None:
            h_qual = torch.empty(n_e2e, dtype=torch.uint8, pin_memory=True)
            h_qual.copy_(d_qual[:n_e2e])
        torch.cuda.synchronize(dev)
        h_np = h_seq.numpy()
        hq_np = h_qual.numpy() if h_qual is not None else None
        if reads:
            off_e2e = np.arange(0, (n_e2e_rec + 1) * READ_LEN, READ_LEN, dtype=np.uint64)
        elif frac_e2e < 1.0:
            off_e2e = np.append(offsets_np[offsets_np < n_e2e], np.uint64(n_e2e)).astype(np.uint64)
        else:
            off_e2e = offsets_np
        d2h_bytes = 0
        e2e_windows = 0
        pin_k = pin_c = None
        if cfg["result"] == "export":   # the (filtered) map lands in pinned host arrays: what the FFI wrapper would hand to HashMap::from_iter
            cap_out = int(summary["n_distinct"] * (frac_e2e if frac_e2e < 1.0 else 1.0)) + 1024
            pin_k = torch.empty(cap_out, dtype=torch.int64, pin_memory=True)
            pin_c = torch.empty(cap_out, dtype=torch.int64, pin_memory=True)

        def step_e2e():
            nonlocal d2h_bytes, e2e_windows
            engine.reset()
            if world == 1:
                engine.counter.count_batch(h_np, hq_np, off_e2e)     # kmg_count_ascii: chunked H2D overlapped with the kernels
            else:
                sharded.count_host(h_np, off_e2e, hq_np, expected_keys_per_rank=cfg["bases"] // world + 1024)
            engine.finalize(False)
            if cfg["result"] == "export":                            # what count_kmers_streaming_packed returns: the (filtered) map
                n_out = engine.counter.export_into(pin_k.numpy().view(np.uint64), pin_c.numpy().view(np.uint64), min_count, sorted=False)
                d2h_bytes = 16 * n_out
                e2e_windows = -1
                return pin_k.numpy()[:n_out], pin_c.numpy()[:n_out]
            vals, freqs = sharded.histogram(min_count)               # D2H of the count-of-counts
            d2h_bytes = (vals.nbytes + freqs.nbytes) + 65536 * 8
            e2e_windows = int((vals * freqs).sum())
            return vals, freqs

        for _ in range(max(2, args.warmup // 2)):   # the first host-fed step sizes the staging ring and the pool
            step_e2e()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            res = step_e2e()
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        s_e2e = sharded.finalize()
        if frac_e2e == 1.0 and s_e2e["n_windows"] != exp_windows:
            raise SystemExit("PARITY FAILURE in the end-to-end path")
        e2e = {"value": s_e2e["n_windows"] / (dt / args.steps), "unit": UNIT,
               "h2d_bytes_per_step": int(n_e2e * (2 if hq_np is not None else 1) + off_e2e.nbytes),
               "d2h_bytes_per_step": int(d2h_bytes), "ms_per_step": dt / args.steps * 1e3,
               "result": ("filtered (key, count) arrays on the host (min_count %d): %d entries" % (min_count, len(res[0]))) if cfg["result"] == "export"
                         else "count-of-counts histogram + summary to host; table stays in HBM",
               "input_fraction": frac_e2e}
        del h_seq, h_qual
    else:
        pin_k = pin_c = None

    # ---- from FILE BYTES: an in-RAM FASTA / FASTQ image of the workload (80-column FASTA lines; 4-line FASTQ), records found
    # on the device by kmg_count_fastx (SURVEY.md 8f-1).  Timed like e2e: raw bytes in pinned host memory -> result on the host.
    e2e_file = None
    if not args.no_e2e and world == 1 and cfg["bases"] <= 4_000_000_000:
        host_seq = d_seq.cpu().numpy()
        if reads:
            n_r = n_rec_local
            img_t = torch.empty(n_r * 316, dtype=torch.uint8, pin_memory=True)
            img = img_t.numpy().reshape(n_r, 316)
            idx = np.arange(n_r, dtype=np.int64)
            img[:, 0] = ord("@"); img[:, 1] = ord("r")
            for j in range(9):
                img[:, 2 + j] = ((idx // 10 ** (8 - j)) % 10 + 48).astype(np.uint8)
            img[:, 11] = 10
            img[:, 12:162] = host_seq.reshape(n_r, READ_LEN)
            img[:, 162] = 10; img[:, 163] = ord("+"); img[:, 164] = 10
            img[:, 165:315] = d_qual.cpu().numpy().reshape(n_r, READ_LEN) if d_qual is not None else ord("I")
            img[:, 315] = 10
            image = img_t.numpy()
        else:
            rec_len = cfg["bases"] // cfg["records"]
            assert rec_len % 80 == 0 and rec_len * cfg["records"] == cfg["bases"]
            hdrs = [b">chr%d\n" % r for r in range(cfg["records"])]
            per = rec_len + rec_len // 80
            img_t = torch.empty(sum(len(h) for h in hdrs) + per * cfg["records"], dtype=torch.uint8, pin_memory=True)
            image = img_t.numpy()
            o = 0
            for r, h in enumerate(hdrs):
                image[o:o + len(h)] = np.frombuffer(h, dtype=np.uint8); o += len(h)
                body = image[o:o + per].reshape(-1, 81)
                body[:, :80] = host_seq[r * rec_len:(r + 1) * rec_len].reshape(-1, 80)
                body[:, 80] = 10
                o += per
        del host_seq

        def step_file():
            engine.reset()
            engine.counter.count_fastx(image, reads)
            engine.finalize(False)
            if cfg["result"] == "export" and pin_k is not None:
                return engine.counter.export_into(pin_k.numpy().view(np.uint64), pin_c.numpy().view(np.uint64), min_count, sorted=False)
            return sharded.histogram(min_count)

        for _ in range(2):
            step_file()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_file()
        dt = (time.perf_counter() - t0) / args.steps
        s_f = sharded.finalize()
        if s_f["n_windows"] != exp_windows or s_f["n_records"] != cfg["records"]:
            raise SystemExit("PARITY FAILURE in the file-image path")
        e2e_file = {"value": exp_windows / dt, "unit": UNIT, "ms_per_step": dt * 1e3, "file_bytes": int(image.nbytes),
                    "file_gbs": image.nbytes / dt / 1e9,
                    "format": "4-line FASTQ image, 316 B per read" if reads else "FASTA image, 80-column lines",
                    "parser": "kmg_count_fastx: raw bytes over PCIe, records found on the device"}
        del image, img_t

    # ---- C5: the .kmix index written from the GPU shard(s) (timed once, outside the steps: it is disk-bound)
    kmix = None
    if args.kmix and "kmix" in cfg["result"]:
        engine.reset(); feed_device(); engine.finalize(False)
        t0 = time.perf_counter()
        info = sharded.save_kmix(args.kmix)
        barrier()
        kmix = {"seconds": max_over_ranks(time.perf_counter() - t0), "records": info["records"], "bytes": 18 + 16 * info["records"], "path": args.kmix}

    # ---- CPU baseline on the box's host cores (rank 0, N=1 only; bounded sample of the same generator)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as orc
        cores = os.cpu_count() or 1
        n = int(args.cpu_sample_bases) if args.cpu_sample_bases else int(min(310e6, cfg["bases"]))
        seq, qual, offs, what = cpu_sample(cfg, n)
        t0 = time.perf_counter()
        w, _d = orc.reference_path_count(k, seq, qual, offs, min_quality=min_q, threads=cores)
        dt = time.perf_counter() - t0
        cpu = {"value": w / dt, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{what}, k={k}: the largest prefix whose packed map fits a 62 GB host (<= 310 Mbp); restated reference CPU path, {dt:.1f} s"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64",
                "data": "synthetic",
                "config": {"workload": f"{cfg['name']}: {cfg['what']}",
                           "k": k, "bases": cfg["bases"], "records": cfg["records"], "windows": exp_windows,
                           "distinct": summary["n_distinct"], "max_count": summary["max_count"],
                           "min_quality": min_q, "min_count": min_count,
                           "path": {0: "hbm-table", 1: "direct-4^k", 2: "partitioned"}[local["path"]],
                           "table_slots_or_partitions_per_gpu": local["table_capacity"],
                           "l2_policy": "inputs and tables are far larger than L2 (no flush needed)" if cfg["bases"] > 5e8 else
                                        "input (>= 100 MB ASCII + packed streams) exceeds the 126 MB L2 between steps; the k=12 counter array (134 MB) does too",
                           "step": "table clear + ingest + scan/upsert (+ fused bucket/exchange over NVLink for N>1) + finalize + device-side result",
                           "parallelism": f"hash-shard x{world}" if world > 1 else "single GPU"},
                "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches)}
        if e2e_file:
            line["e2e_file"] = e2e_file
        if also:
            line["also"] = also
        if kmix:
            line["kmix"] = kmix
        if world > 1:
            line["exchange"] = sharded.stats()
        emit(line)
    engine.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
