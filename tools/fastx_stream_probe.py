"""What does counting a FASTA byte stream cost next to counting the same file as one image?  Builds bench.py's C4-shaped FASTA
image (31 x 100 Mbp of the synthetic genome of seed 44, 80-column lines: 3.14 GB; tools/shard_fastx_probe.py's write_image) in a
file under /dev/shm (or the temp directory), then times, with 1 warm-up and STEPS timed calls, one call = count + finalize +
histogram on one context:
  stream 4 MiB / 64 MiB   kmg_fastx_stream_begin / push / end, the pushes read from the mmap of the file (pageable memory);
  image pageable / pinned kmg_count_fastx of the mmap / of a pinned copy;
  cli stdin               kmerust-b200 21 - -f histogram, the image piped into its stdin by a `cat` child process (wall time of
                          the whole process, CUDA start-up included), with the CLI's peak RSS (getrusage of the children).
Every call is checked against the first one's n_windows / n_records.  Writes one JSON line per case to OUT (default
profiles/r9_fastx_stream_probe.jsonl), the GPU's name and power limit (nvidia-smi, read-only) first; the image file is deleted at
the end.

    python tools/fastx_stream_probe.py [OUT] [STEPS]
"""
import ctypes as C
import json
import mmap
import os
import resource
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import krust_b200 as kb  # noqa: E402
from krust_b200 import _lib  # noqa: E402
from shard_fastx_probe import K, gpu_line, load, write_image  # noqa: E402

BIN = os.path.join(ROOT, "krust_b200", "host", "kmerust-b200")


def stream(c, image, block):
    L, ctx = c._L, c._ctx
    assert L.kmg_fastx_stream_begin(ctx, 0, 0) == _lib.KMG_OK
    base = image.ctypes.data
    for pos in range(0, len(image), block):
        assert L.kmg_fastx_stream_push(ctx, base + pos, min(block, len(image) - pos)) == _lib.KMG_OK, L.kmg_last_error(ctx)
    n = C.c_uint64(0)
    assert L.kmg_fastx_stream_end(ctx, C.byref(n)) == _lib.KMG_OK, L.kmg_last_error(ctx)
    return n.value


def timed_calls(c, feed, steps):
    ts, out = [], None
    for i in range(1 + steps):
        c.reset()
        t0 = time.perf_counter()
        n = feed()
        s = c.finalize()
        c.histogram(1)
        dt = time.perf_counter() - t0
        if i:
            ts.append(dt)
        got = (n, s["n_records"], s["n_windows"])
        assert out is None or got == out, (got, out)
        out = got
    return ts, out


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r9_fastx_stream_probe.jsonl")
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    torch.cuda.set_device(0)
    tmpdir = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    path = os.path.join(tmpdir, f"c4_stream_probe_{os.getpid()}.fa")
    rows = [dict(case="gpu", **gpu_line())]
    try:
        write_image(path)
        size = os.path.getsize(path)
        # the CLI first: RUSAGE_CHILDREN keeps the largest child seen so far, and `cat` / nvidia-smi stay small
        cli_ts = []
        for i in range(1 + steps):
            with open(path, "rb") as f:
                cat = subprocess.Popen(["cat"], stdin=f, stdout=subprocess.PIPE)
                t0 = time.perf_counter()
                r = subprocess.run([BIN, str(K), "-", "-f", "histogram", "-q"], stdin=cat.stdout, capture_output=True)
                dt = time.perf_counter() - t0
                cat.stdout.close()
                cat.wait()
            assert r.returncode == 0, r.stderr
            if i:
                cli_ts.append(dt)
            windows = sum(int(a) * int(b) for a, b in (ln.split(b"\t") for ln in r.stdout.splitlines()))
        peak = resource.getrusage(resource.RUSAGE_CHILDREN).ru_maxrss * 1024
        rows.append(dict(case="cli stdin", image_bytes=size, seconds=cli_ts, median_ms=1e3 * float(np.median(cli_ts)), peak_rss_bytes=peak,
                         n_windows=windows))
        with kb.GpuKmerCounter(K) as c:
            for label, pinned in (("image pageable", False), ("image pinned", True)):
                image, keep = load(path, pinned)
                ts, (n, recs, win) = timed_calls(c, lambda: c.count_fastx(image, False), steps)
                rows.append(dict(case=label, image_bytes=size, seconds=ts, median_ms=1e3 * float(np.median(ts)), n_records=recs, n_windows=win))
                del image, keep
            image, keep = load(path, False)
            for block in (4 << 20, 64 << 20):
                ts, (n, recs, win) = timed_calls(c, lambda: stream(c, image, block), steps)
                rows.append(dict(case=f"stream {block >> 20} MiB pushes (pageable)", image_bytes=size, seconds=ts,
                                 median_ms=1e3 * float(np.median(ts)), n_records=recs, n_windows=win))
            del image, keep
        assert len({r["n_windows"] for r in rows[1:]}) == 1, "the cases disagree"
    finally:
        if os.path.exists(path):
            os.remove(path)
    os.makedirs(os.path.dirname(out_path), exist_ok=True)
    with open(out_path, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")
            print(json.dumps(r))


if __name__ == "__main__":
    main()
