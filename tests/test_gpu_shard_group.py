"""The fused scatter + exchange path (kmg_shard_* calls) with several ranks on ONE device: every rank is a thread with its
own context; the peers' receive buffers are then plain same-device pointers, everything else -- the shared-memory group, the
barrier, the speculative / exact region layouts, owner-side refine + count, merged summary / histogram, the index written
from shards -- is exactly what runs across GPUs (tests/test_gpu_multi.py, which needs >= 2 devices).  Against the oracle."""
import os
import threading
import time

import numpy as np
import pytest

import krust_b200 as kb
from krust_b200 import _lib
from krust_b200.dist import slice_for_rank
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


def run_group(world, k, seq, offsets, qual=None, min_quality=None, batch_bases=0, host_feed=False, kmix_path=None, uneven=False, cuts=None):
    """Returns (per-rank results, errors).  Rank r scans slice_for_rank(...) of the stream (or, with `uneven`, rank 0 gets 70 %; with
    `cuts`, the byte range cuts[r])."""
    import torch
    dev = torch.device("cuda:0")
    total = len(seq)
    group = f"t{os.getpid()}-{time.time_ns() & 0xffffff:x}"
    results, errors = [None] * world, []

    def cut(r):
        if cuts is not None:
            return cuts[r]
        if not uneven:
            return slice_for_rank(total, world, r, k)
        edges = [0] + [int(total * (0.7 + 0.3 * i / (world - 1))) for i in range(world - 1)] + [total]
        a, b = edges[r], edges[r + 1]
        return a, (min(total, b + k - 1) if r + 1 < world else b)

    def worker(r):
        c = None
        try:
            a, b = cut(r)
            inside = [int(o) - a for o in offsets[1:-1] if a < int(o) < b]
            off = np.array([0] + inside + [b - a], dtype=np.uint64)
            c = kb.GpuKmerCounter(k, min_quality=min_quality, batch_bases=batch_bases)
            c.shard_join(world, r, group, total)
            if host_feed:
                c.shard_count_batch(np.ascontiguousarray(seq[a:b]), None if qual is None else np.ascontiguousarray(qual[a:b]), off)
            else:
                d_seq = torch.from_numpy(np.ascontiguousarray(seq[a:b])).to(dev)
                d_qual = None if qual is None else torch.from_numpy(np.ascontiguousarray(qual[a:b])).to(dev)
                d_off = torch.from_numpy(off.astype(np.int64)).to(dev)
                c.shard_count_device(d_seq.data_ptr() if b > a else 0, b - a, d_qual.data_ptr() if d_qual is not None and b > a else 0,
                                     d_off.data_ptr(), len(off) - 1)
            summary = c.shard_finalize()
            hist = c.shard_histogram(1)
            hist2 = c.shard_histogram(2)
            n_kmix = c.shard_save_kmix(kmix_path) if kmix_path else None
            keys, counts = c.export(1, True)
            results[r] = dict(summary=summary, hist=hist, hist2=hist2, keys=keys, counts=counts, stats=c.shard_stats(), n_kmix=n_kmix,
                              local=c.finalize())
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
        t.join(timeout=300)
    assert not any(t.is_alive() for t in threads), "a rank hung"
    return results, errors


def check(results, errors, world, oracle, kmix_path=None, k=None):
    assert not errors, errors
    okeys, ocounts, owin = oracle
    allk = np.concatenate([r["keys"] for r in results]); allc = np.concatenate([r["counts"] for r in results])
    assert len(allk) == len(okeys)                      # shards are disjoint: no key twice
    order = np.argsort(allk, kind="stable")
    assert (allk[order] == okeys).all() and (allc[order] == ocounts).all()
    ov, of = orc.histogram(ocounts, 1)
    ov2, of2 = orc.histogram(ocounts, 2)
    for r, res in enumerate(results):
        s = res["summary"]
        assert s["n_windows"] == owin and s["n_distinct"] == len(okeys) and s["max_count"] == (int(ocounts.max()) if len(ocounts) else 0)
        assert (res["hist"][0] == ov).all() and (res["hist"][1] == of).all()
        assert (res["hist2"][0] == ov2).all() and (res["hist2"][1] == of2).all()
        assert all(kb.owner_of(int(x), world) == r for x in res["keys"][:300])   # every key lives on its owner
        assert res["local"]["n_distinct"] == len(res["keys"])
    assert sum(r["stats"]["recv_keys"] for r in results) == owin   # every counted window arrived at exactly one owner
    if kmix_path:
        kk, ikeys, icounts = orc.kmix_decode(open(kmix_path, "rb").read())
        assert kk == k and results[0]["n_kmix"] == len(okeys) == len(ikeys)
        o2 = np.argsort(ikeys, kind="stable")
        assert (ikeys[o2] == okeys).all() and (icounts[o2] == ocounts).all()


def _genome(rng, n, p_n=0.01):
    return rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8), p=[(1 - p_n) / 4] * 4 + [p_n], size=n).astype(np.uint8)


@pytest.mark.parametrize("world,k", [(2, 21), (4, 31), (8, 15), (3, 32)])
def test_fused_exchange_equals_oracle(world, k, tmp_path):
    rng = np.random.default_rng(world * 10 + k)
    seq = _genome(rng, 3_000_000)
    offsets = np.array([0, 700_000, 700_000, 1_900_000, len(seq)], dtype=np.uint64)
    oracle = orc.count_batch_mt(k, seq, None, offsets)
    p = str(tmp_path / "g.kmix")
    results, errors = run_group(world, k, seq, offsets, kmix_path=p)
    check(results, errors, world, oracle, p, k)
    assert all(r["stats"]["rounds"] == 1 and r["stats"]["exact_rounds"] == 0 for r in results)


def test_fused_exchange_many_rounds_uneven_ranks_and_quality():
    """Small batch_bases: many rounds with k-1 overlaps and records spanning rounds; rank 0 holds 70 % of the input, so the other
    ranks take part in rounds without input; FASTQ-style qualities with -Q 20."""
    world, k = 3, 25
    seq, qual, offsets = orc.synth_reads(43, 3, 0, 12_000)
    oracle = orc.count_batch_mt(k, seq, qual, offsets, 20)
    for host_feed in (False, True):
        results, errors = run_group(world, k, seq, offsets, qual=qual, min_quality=20, batch_bases=200_000, host_feed=host_feed, uneven=True)
        check(results, errors, world, oracle)
        assert results[0]["stats"]["rounds"] >= 6 and len({r["stats"]["rounds"] for r in results}) == 1


def test_fused_exchange_skew_takes_the_exact_route():
    """poly-A / satellite input overflows the speculative per-region shares: the whole group must switch to the exact
    (count + sizes through the shared segment + exact offsets) route and stay exact."""
    world, k = 4, 21
    rng = np.random.default_rng(5)
    seq = np.concatenate([_genome(rng, 600_000, 0.0), np.frombuffer(b"A" * 900_000, dtype=np.uint8), np.frombuffer(b"ACGTTGCA" * 60_000, dtype=np.uint8),
                          _genome(rng, 500_000, 0.0)])
    offsets = np.array([0, 600_000, 1_500_000, len(seq)], dtype=np.uint64)
    oracle = orc.count_batch_mt(k, seq, None, offsets)
    results, errors = run_group(world, k, seq, offsets, batch_bases=1 << 20)
    check(results, errors, world, oracle)
    assert all(r["stats"]["exact_rounds"] >= 1 for r in results)


def test_host_feed_rank_with_an_empty_slice():
    """A rank whose slice holds one empty record and no bytes (seq NULL, offsets [0, 0]) takes part in every round of the host feed."""
    world, k = 3, 21
    seq = _genome(np.random.default_rng(9), 1_500_000)
    offsets = np.array([0, 400_000, len(seq)], dtype=np.uint64)
    oracle = orc.count_batch_mt(k, seq, None, offsets)
    mid = 800_000
    results, errors = run_group(world, k, seq, offsets, batch_bases=200_000, host_feed=True, cuts=[(0, mid + k - 1), (mid, mid), (mid, len(seq))])
    check(results, errors, world, oracle)
    assert results[0]["stats"]["rounds"] >= 4 and len({r["stats"]["rounds"] for r in results}) == 1


def test_host_feed_refuses_decreasing_offsets_and_peers_do_not_hang():
    """Decreasing offsets fail the rank that passes them, as kmg_count_ascii does, and its peer returns instead of waiting."""
    world, k = 2, 21
    group = f"d{os.getpid()}-{time.time_ns() & 0xffffff:x}"
    seq = np.frombuffer(b"ACGT" * 50, dtype=np.uint8)
    out = [None, None]

    def worker(r):
        c = kb.GpuKmerCounter(k)
        try:
            c.shard_join(world, r, group, 1_000_000)
            try:
                c.shard_count_batch(seq, None, np.array([0, 120, 60, 200] if r == 0 else [0, 200], dtype=np.uint64))
                c.shard_finalize()
                out[r] = "no error"
            except kb.GpuError as e:
                out[r] = e
        finally:
            c.close()

    ts = [threading.Thread(target=worker, args=(r,)) for r in range(world)]
    t0 = time.time()
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=200)
    assert not any(t.is_alive() for t in ts) and time.time() - t0 < 100
    assert isinstance(out[0], kb.GpuError) and out[0].status == _lib.KMG_ERR_INVALID_ARG and "offsets must be non-decreasing" in str(out[0])
    assert isinstance(out[1], kb.GpuError) and "peer rank" in str(out[1])


def test_grouped_context_refuses_local_feeds_and_peers_do_not_hang():
    """A rank that fails marks the group aborted: its peers return an error instead of waiting for it."""
    world, k = 2, 21
    group = f"x{os.getpid()}-{time.time_ns() & 0xffffff:x}"
    out = [None, None]

    def worker(r):
        c = kb.GpuKmerCounter(k)
        try:
            c.shard_join(world, r, group, 1_000_000)
            if r == 0:
                with pytest.raises(kb.GpuError):
                    c.count_records([b"ACGT" * 20])           # local feed on a grouped context
                with pytest.raises(kb.GpuError):
                    c.shard_count_device(1, 100)               # misaligned pointer: this rank fails and aborts the group
                out[r] = "failed as expected"
            else:
                try:
                    c.shard_count_device(0, 0)
                    c.shard_finalize()
                    out[r] = "no error"
                except kb.GpuError as e:
                    out[r] = str(e)
        finally:
            c.close()

    ts = [threading.Thread(target=worker, args=(r,)) for r in range(world)]
    t0 = time.time()
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=200)
    assert not any(t.is_alive() for t in ts) and time.time() - t0 < 100
    assert out[0] == "failed as expected" and "peer rank" in out[1]
