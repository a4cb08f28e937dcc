"""How long does --format json take on C1 (k = 21, the 100 Mbp genome of seed 42 in 100 records: ~10^8 records, ~6 GB of json)?

Runs, each printed as one JSON line (the GPU's name and power limit first):
  - device: kmg_write_text json of one context, into a file under OUT_DIR and into /dev/null (wall time of the call), and the device
    time of text_len_kernel + text_write_kernel from a second, profiled call into /dev/null;
  - host route as the CLI took it before json was formatted on the device: kmg_export_counts of the sorted table, then kmerust.hpp's
    output_counts through std::ostream (a small C++ program built into a temporary directory), into a file and into /dev/null;
  - write_counts (Python json.dumps of one dict per record) on a stated prefix of the sorted table, into /dev/null: it holds the
    whole document in memory, which for all 10^8 records does not fit a host comfortably;
  - kmg_shard_write_text json with groups of 2 and 4 thread ranks on one GPU.
Every file must be byte-identical to the device file of one context; all files are deleted afterwards.

    python tools/json_text_probe.py [OUT_DIR]
"""
import io
import json
import os
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
TEXT_KERNELS = ("text_len_kernel", "text_write_kernel")
WRITE_COUNTS_PREFIX = 10_000_000

OUTPUT_COUNTS_MAIN = r"""
#include <chrono>
#include <cstdio>
#include <fstream>
#include <iostream>
#include "kmerust.hpp"
// argv: k  keys.u64  counts.u64  out  -> prints the seconds output_counts took
int main(int argc, char **argv) {
  if (argc != 5) return 2;
  const size_t k = std::stoul(argv[1]);
  auto load = [](const char *p) {
    std::ifstream f(p, std::ios::binary | std::ios::ate);
    std::vector<uint64_t> v((size_t)f.tellg() / 8);
    f.seekg(0);
    f.read(reinterpret_cast<char *>(v.data()), (std::streamsize)(v.size() * 8));
    return v;
  };
  const std::vector<uint64_t> keys = load(argv[2]), counts = load(argv[3]);
  std::ofstream out(argv[4], std::ios::binary);
  const auto t0 = std::chrono::steady_clock::now();
  kmerust::output_counts(out, keys, counts, kmerust::KmerLength::create(k), kmerust::OutputFormat::Json);
  out.flush();
  const double s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  if (!out) return 1;
  printf("%.6f\n", s);
  return 0;
}
"""


def gpu_line() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return {"gpus": torch.cuda.device_count(), "nvidia_smi": [x.strip() for x in q.strip().splitlines()], "torch_name": torch.cuda.get_device_name(0)}


def emit(**kw):
    print(json.dumps(kw), flush=True)


def genome_slice(c, world: int, rank: int, dev):
    a, b = slice_for_rank(N, world, rank, K)
    d = torch.empty(b - a, dtype=torch.uint8, device=dev)
    c.synth_uniform_device(SEED, a, b - a, d.data_ptr())
    inside = OFFSETS[(OFFSETS > a) & (OFFSETS < b)] - a
    off = torch.from_numpy(np.concatenate([[0], inside, [b - a]]).astype(np.int64)).to(dev)
    return d, off


def kernel_ms(fn) -> float:
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(e.device_time_total for e in prof.key_averages() if any(n in e.key for n in TEXT_KERNELS)) / 1e3


def same_file(a, b) -> bool:
    x, y = np.memmap(a, dtype=np.uint8, mode="r"), np.memmap(b, dtype=np.uint8, mode="r")
    if len(x) != len(y):
        return False
    return all((x[i:i + (1 << 28)] == y[i:i + (1 << 28)]).all() for i in range(0, len(x), 1 << 28))


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return r, time.perf_counter() - t0


def device_and_host_routes(out_dir, build_dir) -> str:
    dev = torch.device("cuda:0")
    ref = os.path.join(out_dir, "single.json")
    with kb.GpuKmerCounter(K, expected_distinct=N) as c:
        d, off = genome_slice(c, 1, 0, dev)
        c.count_device(d.data_ptr(), d.numel(), 0, off.data_ptr(), off.numel() - 1)
        c.finalize(False)
        del d
        (rec, nbytes), wall = timed(lambda: c.write_text(ref, "json", 1))
        emit(run="device kmg_write_text", sink="file", wall_s=round(wall, 3), records=rec, bytes=nbytes, GB_per_s=round(nbytes / wall / 1e9, 3))
        (rec, nbytes), wall = timed(lambda: c.write_text(os.devnull, "json", 1))
        emit(run="device kmg_write_text", sink="/dev/null", wall_s=round(wall, 3), records=rec, bytes=nbytes, GB_per_s=round(nbytes / wall / 1e9, 3))
        ms = kernel_ms(lambda: c.write_text(os.devnull, "json", 1))
        emit(run="device formatting kernels", kernels=list(TEXT_KERNELS), device_ms=round(ms, 3), bytes=nbytes,
             GB_per_s_of_kernel_time=round(nbytes / (ms / 1e3) / 1e9, 1))
        (keys, counts), export_s = timed(lambda: c.export(1, True))
    emit(run="host export (kmg_export_counts, sorted)", wall_s=round(export_s, 3), records=len(keys))

    # export + output_counts, as the CLI did it: a C++ program over the exported arrays
    exe = os.path.join(build_dir, "output_counts_json")
    src = exe + ".cpp"
    with open(src, "w") as f:
        f.write(OUTPUT_COUNTS_MAIN)
    host = os.path.join(ROOT, "krust_b200", "host")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I", host, src, "-o", exe, "-L", os.path.join(ROOT, "krust_b200"), "-lkmerust_gpu", "-lz",
                           "-Wl,-rpath," + os.path.join(ROOT, "krust_b200")])
    kp, cp = os.path.join(out_dir, "keys.u64"), os.path.join(out_dir, "counts.u64")
    keys.tofile(kp); counts.tofile(cp)
    host_file = os.path.join(out_dir, "host.json")
    try:
        for sink, path in (("file", host_file), ("/dev/null", os.devnull)):
            s = float(subprocess.run([exe, str(K), kp, cp, path], capture_output=True, text=True, check=True).stdout)
            emit(run="host output_counts (std::ostream)", sink=sink, output_counts_s=round(s, 3), export_plus_output_counts_s=round(s + export_s, 3),
                 bytes=nbytes)
        ok = same_file(host_file, ref)
        emit(run="host output_counts file identical to the device file", identical=ok)
        if not ok:
            raise SystemExit("output_counts json differs from the device json")
    finally:
        for p in (kp, cp, host_file):
            if os.path.exists(p):
                os.remove(p)

    # write_counts on a prefix: one dict per record and one string of the document
    n = min(WRITE_COUNTS_PREFIX, len(keys))
    with open(os.devnull, "wb") as f:
        _, s = timed(lambda: kb.write_counts(f, keys[:n], counts[:n], K, "json"))
    buf = io.BytesIO()
    kb.write_counts(buf, keys[:1000], counts[:1000], K, "json")
    with open(ref, "rb") as f:
        head = f.read(len(buf.getvalue()) - 3)
    emit(run="host write_counts (Python json.dumps)", sink="/dev/null", prefix_records=n, wall_s=round(s, 3),
         records_per_s=round(n / s), prefix_matches_device_file=buf.getvalue()[:-3] == head)
    return ref


def thread_group(world, out_dir, ref):
    dev = torch.device("cuda:0")
    group = f"jprobe{os.getpid()}-{world}"
    p = os.path.join(out_dir, f"threads{world}.json")
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
        _, wall = timed(lambda: each(lambda c, r: c.shard_write_text(p, "json", 1)))
        rec, nbytes = res[0]
        ms = kernel_ms(lambda: each(lambda c, r: c.shard_write_text(p, "json", 1)))
        ok = same_file(p, ref)
        emit(run="threads kmg_shard_write_text", world=world, wall_s=round(wall, 3), records=rec, bytes=nbytes,
             GB_per_s=round(nbytes / wall / 1e9, 3), formatting_kernels_ms_all_ranks=round(ms, 3), identical_to_single=ok)
        if not ok:
            raise SystemExit(f"{p} differs from the single-context file")
        each(lambda c, r: c.shard_leave())
    finally:
        for c in ctxs:
            c.close()
        if os.path.exists(p):
            os.remove(p)


def run(out_dir):
    emit(**gpu_line())
    with tempfile.TemporaryDirectory(prefix="json_probe_build_") as build_dir:
        ref = device_and_host_routes(out_dir, build_dir)
    try:
        for w in (2, 4):
            thread_group(w, out_dir, ref)
    finally:
        os.remove(ref)


def main():
    if len(sys.argv) > 1:
        os.makedirs(sys.argv[1], exist_ok=True)
        run(sys.argv[1])
    else:
        with tempfile.TemporaryDirectory(prefix="json_text_") as out_dir:
            run(out_dir)


if __name__ == "__main__":
    main()
