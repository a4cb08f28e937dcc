"""Where does the time of ONE sorted text file from a shard group go?  Writes C1's tsv (k = 21, the 100 Mbp genome of seed 42 in
100 records: 2.4 GB) under OUT_DIR with a single context, with groups of 2 and 4 thread ranks on one GPU, and with 2 / 4 / 8 process
ranks (one per GPU) where that many GPUs exist.  For each run: wall time of the write call, records, GB/s of text, and the device
time of merge_shard_pieces_kernel (summed over the ranks, from a second, profiled call).  Every file must be byte-identical to the
single-context file; all files are deleted afterwards.  Prints one JSON line per run, the GPU's name and power limit first.

    python tools/shard_text_probe.py [OUT_DIR]
"""
import json
import os
import socket
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import krust_b200 as kb  # noqa: E402
from krust_b200.dist import slice_for_rank  # noqa: E402

K, N, N_REC, SEED = 21, 100_000_000, 100, 42
OFFSETS = np.arange(0, N + 1, N // N_REC, dtype=np.int64)
MERGE_KERNEL = "merge_shard_pieces_kernel"


def gpu_line() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return {"gpus": torch.cuda.device_count(), "nvidia_smi": [x.strip() for x in q.strip().splitlines()], "torch_name": torch.cuda.get_device_name(0)}


def genome_slice(c: "kb.GpuKmerCounter", world: int, rank: int, dev):
    """This rank's slice of the genome, synthesised on the device, and its record offsets."""
    a, b = slice_for_rank(N, world, rank, K)
    d = torch.empty(b - a, dtype=torch.uint8, device=dev)
    c.synth_uniform_device(SEED, a, b - a, d.data_ptr())
    inside = OFFSETS[(OFFSETS > a) & (OFFSETS < b)] - a
    off = torch.from_numpy(np.concatenate([[0], inside, [b - a]]).astype(np.int64)).to(dev)
    return d, off


def merge_ms(prof) -> float:
    return sum(e.device_time_total for e in prof.key_averages() if MERGE_KERNEL in e.key) / 1e3


def profiled(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return merge_ms(prof)


def same_file(a, b) -> bool:
    x, y = np.memmap(a, dtype=np.uint8, mode="r"), np.memmap(b, dtype=np.uint8, mode="r")
    if len(x) != len(y):
        return False
    return all((x[i:i + (1 << 28)] == y[i:i + (1 << 28)]).all() for i in range(0, len(x), 1 << 28))


def report(kind, world, wall, rec, nbytes, merge, path, ref):
    ok = ref is None or same_file(path, ref)
    print(json.dumps({"run": kind, "world": world, "wall_s": round(wall, 3), "records": rec, "bytes": nbytes,
                      "GB_per_s": round(nbytes / wall / 1e9, 3), "merge_kernel_ms": round(merge, 3), "identical_to_single": ok}), flush=True)
    if not ok:
        raise SystemExit(f"{path} differs from the single-context file")


def single(out_dir) -> str:
    dev = torch.device("cuda:0")
    p = os.path.join(out_dir, "single.tsv")
    with kb.GpuKmerCounter(K, expected_distinct=N) as c:
        d, off = genome_slice(c, 1, 0, dev)
        c.count_device(d.data_ptr(), d.numel(), 0, off.data_ptr(), off.numel() - 1)
        c.finalize(False)
        t0 = time.perf_counter()
        rec, nbytes = c.write_text(p, "tsv", 1)
        wall = time.perf_counter() - t0
    report("single", 1, wall, rec, nbytes, 0.0, p, None)
    return p


def thread_group(world, out_dir, ref):
    dev = torch.device("cuda:0")
    group = f"probe{os.getpid()}-{world}"
    p = os.path.join(out_dir, f"threads{world}.tsv")
    ctxs = [kb.GpuKmerCounter(K) for _ in range(world)]
    errors, res = [], [None] * world

    def each(fn):
        def run(r):
            try:
                res[r] = fn(ctxs[r], r)
            except Exception as e:  # noqa: BLE001
                errors.append(repr(e))
        ts = [threading.Thread(target=run, args=(r,)) for r in range(world)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        if errors:
            raise SystemExit(errors)

    try:
        each(lambda c, r: c.shard_join(world, r, group, N))
        def feed(c, r):
            d, off = genome_slice(c, world, r, dev)
            c.shard_count_device(d.data_ptr(), d.numel(), 0, off.data_ptr(), off.numel() - 1)
            torch.cuda.synchronize(dev)
        each(feed)
        each(lambda c, r: c.shard_finalize())
        t0 = time.perf_counter()
        each(lambda c, r: c.shard_write_text(p, "tsv", 1))
        wall = time.perf_counter() - t0
        rec, nbytes = res[0]
        merge = profiled(lambda: each(lambda c, r: c.shard_write_text(p, "tsv", 1)))
        report("threads", world, wall, rec, nbytes, merge, p, ref)
        each(lambda c, r: c.shard_leave())
    finally:
        for c in ctxs:
            c.close()
        if os.path.exists(p):
            os.remove(p)


def _proc(rank, world, port, out_dir, ref):
    import torch.distributed as dist
    from krust_b200.dist import GpuShardEngine, ShardedKmerCounter
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dev = torch.device(f"cuda:{rank}")
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        eng = GpuShardEngine(K, dev)
        sc = ShardedKmerCounter(eng)
        d, off = genome_slice(eng.counter, world, rank, dev)
        sc.count(d, off)
        sc.finalize()
        p = os.path.join(out_dir, f"procs{world}.tsv")
        dist.barrier()
        t0 = time.perf_counter()
        rec, nbytes = sc.write_text(p, "tsv", 1)
        dist.barrier()
        wall = time.perf_counter() - t0
        merge = torch.tensor([profiled(lambda: sc.write_text(p, "tsv", 1))], device=dev)
        dist.all_reduce(merge)
        if rank == 0:
            report("processes", world, wall, rec, nbytes, float(merge.item()), p, ref)
            os.remove(p)
        dist.barrier()
        eng.close()
    finally:
        dist.destroy_process_group()


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else tempfile.mkdtemp(prefix="shard_text_")
    os.makedirs(out_dir, exist_ok=True)
    print(json.dumps(gpu_line()), flush=True)
    ref = single(out_dir)
    try:
        for w in (2, 4):
            thread_group(w, out_dir, ref)
        import torch.multiprocessing as mp
        for w in (2, 4, 8):
            if torch.cuda.device_count() >= w:
                s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
                mp.spawn(_proc, args=(w, port, out_dir, ref), nprocs=w, join=True)
    finally:
        os.remove(ref)


if __name__ == "__main__":
    main()
