"""What does parsing a genome file on the device buy a multi-GPU shard group?  Builds the C4-shaped FASTA image of bench.py (31 x 100
Mbp of the synthetic genome of seed 44, 80-column lines: 3.14 GB) in a file under /dev/shm (or the temp directory), then times, with
2 warm-ups and STEPS timed calls, one call = count + shard_finalize + shard_histogram:
  world 1        one context, kmg_count_fastx;
  world 2/4/8    one process per GPU (as far as the box has GPUs), (a) kmg_shard_count_fastx of the whole image on every rank,
                 (b) the path without it: kmg_parse_fastx of the image on the host, then kmg_shard_count_ascii of the rank's share
                 of the records.
Each with the image in pinned host memory (what bench.py's e2e_file uses) and in pageable memory (an mmap of the file).  Every call
is checked against the one-context n_windows / n_records.  Writes one JSON line per case to OUT (default
profiles/r8_shard_fastx_probe.jsonl), the GPU's name and power limit (nvidia-smi, read-only) first; the image file is deleted at the end.

    python tools/shard_fastx_probe.py [OUT] [STEPS]
"""
import json
import mmap
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import krust_b200 as kb  # noqa: E402
from krust_b200.api import parse_fastx  # noqa: E402

K, SEED, N_REC, REC_LEN = 21, 44, 31, 100_000_000
WARMUP = 2


def gpu_line() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return {"gpus": torch.cuda.device_count(), "nvidia_smi": [x.strip() for x in q.strip().splitlines()], "torch_name": torch.cuda.get_device_name(0)}


def write_image(path):
    """bench.py's C4 FASTA image: '>chrR' headers, 80-column lines of the device-synthesised genome."""
    dev = torch.device("cuda:0")
    with kb.GpuKmerCounter(K) as c, open(path, "wb") as f:
        d = torch.empty(REC_LEN, dtype=torch.uint8, device=dev)
        body = np.empty((REC_LEN // 80, 81), dtype=np.uint8)
        body[:, 80] = 10
        for r in range(N_REC):
            c.synth_uniform_device(SEED, r * REC_LEN, REC_LEN, d.data_ptr())
            body[:, :80] = d.cpu().numpy().reshape(-1, 80)
            f.write(b">chr%d\n" % r)
            f.write(body.tobytes())


def load(path, pinned):
    """The image in pinned memory (a copy) or pageable (the mmap itself).  Returns (array, keep-alive objects)."""
    f = open(path, "rb")
    m = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ)
    if not pinned:
        return np.frombuffer(m, dtype=np.uint8), (f, m)
    t = torch.empty(len(m), dtype=torch.uint8, pin_memory=True)
    a = t.numpy()
    a[:] = np.frombuffer(m, dtype=np.uint8)
    return a, (t,)


def timed(call, steps):
    for _ in range(WARMUP):
        call()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        out = call()
        ts.append(time.perf_counter() - t0)
    return ts, out


def single(path, steps):
    torch.cuda.set_device(0)
    rows = []
    for pinned in (True, False):
        image, keep = load(path, pinned)
        with kb.GpuKmerCounter(K, expected_distinct=len(image)) as c:
            def call():
                c.reset()
                n = c.count_fastx(image, False)
                s = c.finalize()
                c.histogram(1)
                return n, s
            ts, (n, s) = timed(call, steps)
        rows.append(dict(world=1, path="kmg_count_fastx", memory="pinned" if pinned else "pageable", ts=ts, n_windows=int(s["n_windows"]),
                         n_records=int(n), file_bytes=len(image)))
        del image, keep
    return rows


def _rank(rank, world, group, path, pinned, which, steps, q):
    dev = torch.device(f"cuda:{rank}")
    torch.cuda.set_device(dev)
    image, keep = load(path, pinned)
    c = kb.GpuKmerCounter(K, device=rank)
    try:
        c.shard_join(world, rank, group, len(image))
        if which == "shard_count_fastx":
            def feed():
                return c.shard_count_fastx(image, False)
        else:
            def feed():
                seq, _, offsets = parse_fastx(image, False)
                n = len(offsets) - 1
                lo, hi = n * rank // world, n * (rank + 1) // world
                a, b = int(offsets[lo]), int(offsets[hi])
                c.shard_count_batch(seq[a:b], None, (offsets[lo:hi + 1] - a).astype(np.uint64))
                return n

        def call():
            c.reset()
            n = feed()
            s = c.shard_finalize()
            c.shard_histogram(1)
            return n, s
        ts, (n, s) = timed(call, steps)
        q.put(dict(rank=rank, ts=ts, n_windows=int(s["n_windows"]), n_records=int(s["n_records"]), n_out=int(n)))
        c.shard_leave()
    except Exception as e:  # noqa: BLE001
        q.put(dict(rank=rank, error=repr(e)))
    finally:
        c.close()


def group(path, world, pinned, which, steps):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    name = f"fxprobe{os.getpid()}-{world}-{time.time_ns() & 0xffffff:x}"
    ps = [ctx.Process(target=_rank, args=(r, world, name, path, pinned, which, steps, q)) for r in range(world)]
    for p in ps:
        p.start()
    got = [q.get(timeout=1800) for _ in range(world)]
    for p in ps:
        p.join()
    errs = [g["error"] for g in got if "error" in g]
    if errs:
        raise SystemExit(f"world {world} {which}: {errs}")
    ts = np.max(np.array([g["ts"] for g in got]), axis=0).tolist()   # a call ends when its slowest rank returns
    g0 = got[0]
    return dict(world=world, path="kmg_shard_count_fastx" if which == "shard_count_fastx" else "kmg_parse_fastx + kmg_shard_count_ascii",
                memory="pinned" if pinned else "pageable", ts=ts, n_windows=g0["n_windows"], n_records=g0["n_records"],
                file_bytes=os.path.getsize(path))


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r8_shard_fastx_probe.jsonl")
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    tmp = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    path = os.path.join(tmp, f"shard_fastx_probe_{os.getpid()}.fa")
    lines = [gpu_line()]
    try:
        write_image(path)
        rows = single(path, steps)
        ref = rows[0]
        n_gpus = torch.cuda.device_count()
        for w in (2, 4, 8):
            if n_gpus < w:
                lines.append({"world": w, "measured": False, "why": f"{n_gpus} GPU(s) on this box"})
                continue
            for which in ("shard_count_fastx", "parse_then_shard_count_ascii"):
                for pinned in (True, False):
                    rows.append(group(path, w, pinned, which, steps))
        for r in rows:
            ms = float(np.median(r["ts"])) * 1e3
            parity = r["n_windows"] == ref["n_windows"] and r["n_records"] == ref["n_records"] == N_REC
            lines.append({"world": r["world"], "path": r["path"], "memory": r["memory"], "calls": len(r["ts"]),
                          "ms_per_call": round(ms, 2), "ms_min": round(min(r["ts"]) * 1e3, 2), "ms_max": round(max(r["ts"]) * 1e3, 2),
                          "G_kmers_per_s": round(r["n_windows"] / ms / 1e6, 2), "file_GB_per_s": round(r["file_bytes"] / ms / 1e6, 2),
                          "n_windows": r["n_windows"], "n_records": r["n_records"], "parity": parity})
    finally:
        if os.path.exists(path):
            os.remove(path)
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")
            print(json.dumps(ln), flush=True)
    if not all(ln.get("parity", True) for ln in lines):
        raise SystemExit("PARITY FAILURE")


if __name__ == "__main__":
    main()
