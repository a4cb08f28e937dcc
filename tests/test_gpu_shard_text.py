"""kmg_shard_write_text: ONE sorted fasta / tsv file from all shards of a group, byte-identical to what kmg_write_text writes for a
single context that counted the same input, and to the sorted oracle table formatted line by line.  Ranks are threads with their own
contexts on one device (as in test_gpu_shard_group.py); the last test runs one process per GPU where a box has several."""
import os
import pickle
import socket
import threading
import time

import numpy as np
import pytest

import krust_b200 as kb
from krust_b200.dist import slice_for_rank
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


def run_group(world, k, seq, offsets, action, batch_bases=0):
    """Every rank counts its slice_for_rank(...) of the stream in a fresh group, then returns action(counter, rank).
    Returns (per-rank results, errors)."""
    import torch
    dev = torch.device("cuda:0")
    total = len(seq)
    group = f"txt{os.getpid()}-{time.time_ns() & 0xffffff:x}"
    results, errors = [None] * world, []

    def worker(r):
        c = None
        try:
            a, b = slice_for_rank(total, world, r, k)
            inside = [int(o) - a for o in offsets[1:-1] if a < int(o) < b]
            off = np.array([0] + inside + [b - a], dtype=np.int64)
            c = kb.GpuKmerCounter(k, batch_bases=batch_bases)
            c.shard_join(world, r, group, total)
            d_seq = torch.from_numpy(np.array(seq[a:b])).to(dev)
            d_off = torch.from_numpy(off).to(dev)
            c.shard_count_device(d_seq.data_ptr() if b > a else 0, b - a, 0, d_off.data_ptr(), len(off) - 1)
            del d_seq
            results[r] = action(c, r)
            c.shard_leave()
        except Exception as e:  # noqa: BLE001
            errors.append((r, repr(e)))
        finally:
            if c is not None:
                c.close()

    threads = [threading.Thread(target=worker, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout=600)
    assert not any(t.is_alive() for t in threads), "a rank hung"
    return results, errors


def single_context_file(k, seq, offsets, path, fmt, min_count):
    with kb.GpuKmerCounter(k) as c:
        c.count_batch(seq, None, offsets)
        return c.write_text(path, fmt, min_count)


def _oracle_text(keys, counts, k, fmt) -> bytes:
    names = kb.unpack_many(keys, k).tolist()
    if fmt == "tsv":
        return b"".join(b"%s\t%d\n" % (s, int(c)) for s, c in zip(names, counts.tolist()))
    return b"".join(b">%d\n%s\n" % (int(c), s) for s, c in zip(names, counts.tolist()))


def _genome(rng, n, p_n=0.01):
    return rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8), p=[(1 - p_n) / 4] * 4 + [p_n], size=n).astype(np.uint8)


CASES = [(fmt, m) for fmt in ("tsv", "fasta") for m in (0, 1, 2, 50)]


def check_files(tmp_path, k, seq, offsets, results, errors, oracle):
    """Every (format, min_count) file of the group equals the single-context file and the oracle text; totals on every rank."""
    assert not errors, errors
    okeys, ocounts, _ = oracle
    for fmt, m in CASES:
        fk, fc = orc.filter_min_count(okeys, ocounts, max(m, 1))
        want = _oracle_text(fk, fc, k, fmt)
        one = tmp_path / f"one-{fmt}-{m}"
        assert single_context_file(k, seq, offsets, one, fmt, m) == (len(fk), len(want))
        got = (tmp_path / f"group-{fmt}-{m}").read_bytes()
        assert got == one.read_bytes() == want, (fmt, m)
        for res in results:
            assert res[(fmt, m)] == (len(fk), len(want))


def write_all(tmp_path):
    def action(c, r):
        return {(fmt, m): c.shard_write_text(tmp_path / f"group-{fmt}-{m}", fmt, m) for fmt, m in CASES}
    return action


@pytest.mark.parametrize("world,k", [(2, 21), (3, 32), (4, 31), (8, 15)])
def test_group_text_equals_single_context_and_oracle(world, k, tmp_path):
    rng = np.random.default_rng(world * 100 + k)
    seq = _genome(rng, 1_500_000)
    offsets = np.array([0, 1, 400_000, 400_000, 1_100_000, 1_100_777, len(seq)], dtype=np.uint64)   # records of mixed length
    oracle = orc.count_batch_mt(k, seq, None, offsets)
    results, errors = run_group(world, k, seq, offsets, write_all(tmp_path))
    check_files(tmp_path, k, seq, offsets, results, errors, oracle)


def test_group_text_skewed_input_and_empty_outputs(tmp_path):
    """poly-A / satellite input (multi-digit counts, very uneven pieces); then poly-A alone, where all ranks but one own nothing;
    and a min_count above the largest count, which gives an empty file."""
    world, k = 4, 21
    rng = np.random.default_rng(5)
    seq = np.concatenate([_genome(rng, 600_000, 0.0), np.frombuffer(b"A" * 900_000, dtype=np.uint8), np.frombuffer(b"ACGTTGCA" * 60_000, dtype=np.uint8),
                          _genome(rng, 500_000, 0.0)])
    offsets = np.array([0, 600_000, 1_500_000, len(seq)], dtype=np.uint64)
    oracle = orc.count_batch_mt(k, seq, None, offsets)
    above = int(oracle[1].max()) + 1

    def action(c, r):
        out = write_all(tmp_path)(c, r)
        out["above"] = c.shard_write_text(tmp_path / "above", "tsv", above)
        out["stats"] = c.shard_stats()
        return out

    results, errors = run_group(world, k, seq, offsets, action, batch_bases=1 << 20)
    check_files(tmp_path, k, seq, offsets, results, errors, oracle)
    assert all(r["stats"]["exact_rounds"] >= 1 for r in results)
    assert all(r["above"] == (0, 0) for r in results) and os.path.getsize(tmp_path / "above") == 0

    polya = np.frombuffer(b"A" * 300_000, dtype=np.uint8)
    off1 = np.array([0, len(polya)], dtype=np.uint64)
    p = tmp_path / "polya.fa"
    results, errors = run_group(3, k, polya, off1, lambda c, r: (c.shard_write_text(p, "fasta", 1), c.export(1, True)[0].size))
    assert not errors, errors
    assert sorted(r[1] for r in results) == [0, 0, 1]
    want = b">%d\n%s\n" % (len(polya) - k + 1, b"A" * k)
    assert p.read_bytes() == want and all(r[0] == (1, len(want)) for r in results)


def test_group_text_c1_100mbp_many_steps(tmp_path):
    """C1's 100 Mbp genome (~10^8 keys, ~6 pieces of 2^24) at world 4: one full step and one in which two ranks own no piece.
    Equal to the single-context file (compared in blocks) and to the oracle (one-digit counts: the text as a matrix)."""
    world, n, n_rec, k = 4, 100_000_000, 100, 21
    host = orc.synth_uniform(42, 0, n)
    offs = np.arange(0, n + 1, n // n_rec, dtype=np.uint64)
    okeys, ocounts, _ = orc.count_batch_mt(k, host, None, offs)
    assert int(ocounts.max()) < 10 and 5 * (1 << 24) < len(okeys) <= 6 * (1 << 24)
    pg, p1 = tmp_path / "group.tsv", tmp_path / "one.tsv"
    results, errors = run_group(world, k, host, offs, lambda c, r: c.shard_write_text(pg, "tsv", 1))
    assert not errors, errors
    assert all(r == (len(okeys), len(okeys) * (k + 3)) for r in results)
    assert single_context_file(k, host, offs, p1, "tsv", 1) == results[0]
    got = np.memmap(pg, dtype=np.uint8, mode="r")
    one = np.memmap(p1, dtype=np.uint8, mode="r")
    assert len(got) == len(one) == len(okeys) * (k + 3)
    block = 1 << 28
    for i in range(0, len(got), block):
        assert (got[i:i + block] == one[i:i + block]).all()
    del one
    os.remove(p1)
    got = got.reshape(-1, k + 3)
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    shifts = (np.arange(k - 1, -1, -1, dtype=np.uint64) * np.uint64(2))
    step = 4_000_000
    for i in range(0, len(okeys), step):
        kk = okeys[i:i + step]
        want = np.empty((len(kk), k + 3), dtype=np.uint8)
        want[:, :k] = lut[((kk[:, None] >> shifts[None, :]) & np.uint64(3)).astype(np.uint8)]
        want[:, k] = ord("\t"); want[:, k + 1] = ocounts[i:i + step].astype(np.uint8) + ord("0"); want[:, k + 2] = ord("\n")
        assert (got[i:i + step] == want).all()


def test_group_text_with_small_batches(tmp_path):
    """batch_bases = 200 000: many counting rounds and small send buffers; the text staging buffers do not depend on them."""
    world, k = 3, 25
    seq, _, offsets = orc.synth_reads(43, 3, 0, 12_000)
    oracle = orc.count_batch_mt(k, seq, None, offsets)

    def action(c, r):
        return dict(write_all(tmp_path)(c, r), stats=c.shard_stats())

    results, errors = run_group(world, k, seq, offsets, action, batch_bases=200_000)
    assert not errors, errors
    assert all(r["stats"]["rounds"] >= 3 for r in results)   # 600 kbp per rank
    for r in results:
        del r["stats"]
    check_files(tmp_path, k, seq, offsets, results, errors, oracle)


def _errors_group(action, world=3, k=21):
    rng = np.random.default_rng(1)
    seq = _genome(rng, 200_000)
    t0 = time.time()
    results, errors = run_group(world, k, seq, np.array([0, len(seq)], dtype=np.uint64), action)
    return results, errors, time.time() - t0


def test_group_text_errors_do_not_hang(tmp_path):
    # "-" is refused on every rank before any barrier; the group stays usable
    p = tmp_path / "after.tsv"

    def stdout_then_file(c, r):
        with pytest.raises(kb.GpuError):
            c.shard_write_text("-", "tsv", 1)
        return c.shard_write_text(p, "tsv", 1)

    results, errors, _ = _errors_group(stdout_then_file)
    assert not errors, errors
    assert len({r for r in results}) == 1 and results[0][1] == os.path.getsize(p) > 0

    # a path in a missing directory fails on every rank, long before the barrier timeout
    def missing_dir(c, r):
        try:
            c.shard_write_text(tmp_path / "no" / "such" / "dir.tsv", "tsv", 1)
            return "no error"
        except kb.GpuError as e:
            return str(e)

    results, errors, dt = _errors_group(missing_dir)
    assert not errors and all(r != "no error" for r in results) and dt < 100, (results, errors, dt)

    # ranks passing different min_count values all fail
    def mismatch(c, r):
        try:
            c.shard_write_text(tmp_path / "mismatch.tsv", "tsv", 1 + (r == 1))
            return "no error"
        except kb.GpuError as e:
            return str(e)

    results, errors, dt = _errors_group(mismatch)
    assert not errors and all(r != "no error" for r in results) and dt < 100, (results, errors, dt)


def test_ungrouped_context_shard_write_text_is_write_text(tmp_path):
    rng = np.random.default_rng(7)
    seq = _genome(rng, 300_000)
    offsets = np.array([0, 100_000, len(seq)], dtype=np.uint64)
    with kb.GpuKmerCounter(21) as c:
        c.count_batch(seq, None, offsets)
        for fmt in ("tsv", "fasta"):
            a = c.shard_write_text(tmp_path / f"a.{fmt}", fmt, 1)
            b = c.write_text(tmp_path / f"b.{fmt}", fmt, 1)
            assert a == b and (tmp_path / f"a.{fmt}").read_bytes() == (tmp_path / f"b.{fmt}").read_bytes()


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _worker(rank, world, port, k, data_path, out_dir):
    import torch
    import torch.distributed as dist
    from krust_b200.dist import GpuShardEngine, ShardedKmerCounter
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    os.environ["KMG_DIST_FUSED"] = "1"
    dev = torch.device(f"cuda:{rank}")
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        with open(data_path, "rb") as f:
            seq_np, offsets_np = pickle.load(f)
        a, b = slice_for_rank(len(seq_np), world, rank, k)
        inside = [int(o) - a for o in offsets_np[1:-1] if a < int(o) < b]
        off = torch.tensor([0] + inside + [b - a], dtype=torch.int64, device=dev)
        eng = GpuShardEngine(k, dev, batch_bases=400_000)
        sc = ShardedKmerCounter(eng)
        sc.count(torch.from_numpy(seq_np[a:b].copy()).to(dev), off)
        out = {fmt: sc.write_text(os.path.join(out_dir, f"multi.{fmt}"), fmt, 2 if fmt == "fasta" else 1) for fmt in ("tsv", "fasta")}
        with open(os.path.join(out_dir, f"r{rank}.pkl"), "wb") as f:
            pickle.dump(out, f)
        eng.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(_n_gpus() < 2, reason="needs >= 2 GPUs")
def test_multi_gpu_processes_write_one_text_file(tmp_path):
    """One process per GPU: the staging buffers are mapped through CUDA IPC and the merge kernel's loads cross NVLink."""
    import torch.multiprocessing as mp
    world, k = min(_n_gpus(), 4), 21
    rng = np.random.default_rng(11)
    seq = _genome(rng, 2_000_000)
    offsets = np.array([0, 300_000, 300_000, 1_200_000, len(seq)], dtype=np.uint64)
    data = tmp_path / "d.pkl"
    with open(data, "wb") as f:
        pickle.dump((seq, offsets), f)
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_worker, args=(world, port, k, str(data), str(tmp_path)), nprocs=world, join=True)
    okeys, ocounts, _ = orc.count_batch_mt(k, seq, None, offsets)
    for fmt, m in (("tsv", 1), ("fasta", 2)):
        fk, fc = orc.filter_min_count(okeys, ocounts, m)
        want = _oracle_text(fk, fc, k, fmt)
        assert (tmp_path / f"multi.{fmt}").read_bytes() == want
        one = tmp_path / f"one.{fmt}"
        assert single_context_file(k, seq, offsets, one, fmt, m) == (len(fk), len(want)) and one.read_bytes() == want
        for r in range(world):
            with open(tmp_path / f"r{r}.pkl", "rb") as f:
                assert pickle.load(f)[fmt] == (len(fk), len(want))
