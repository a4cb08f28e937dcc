"""Phase B in place: one raw run in the speculative layout is counted where it lies (count_partitions_sieve_in_place_kernel).
The result keeps the run's key array; a repeated key's further entries keep their key with count 0, the slack behind every
segment gets count 0.  Every case is compared against the oracle, and each runs in a subprocess with KMG_DEBUG_SIEVE set so
that the route phase B took (in place, or left for the copying route) can be read from its stderr line."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DONE = re.compile(r"\[kmg\] sieve: (\d+) partitions, (\d+) left to the compacting variant, (\d+) entries, (\d+) distinct, (in place|copied)$")
STOPPED = re.compile(r"\[kmg\] sieve: (\d+) partitions, (\d+) handed back, repeated without the sieve, (leaves the in-place route|copied)$")


def _run(case, *args):
    """Runs _case_<case>(*args) in a fresh process; returns its phase B debug lines."""
    env = dict(os.environ, KMG_DEBUG_SIEVE="1")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), case] + [str(a) for a in args]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, f"case {case} failed:\n{r.stdout[-4000:]}\n{r.stderr[-4000:]}"
    return [ln for ln in r.stderr.splitlines() if ln.startswith("[kmg] sieve:")]


def _assert_same(got, want):
    assert len(got[0]) == len(want[0]), (len(got[0]), len(want[0]))
    assert (got[0] == want[0]).all() and (got[1] == want[1]).all()


def _check_queries(c, okeys, ocounts, rng, k):
    """Device queries: keys seen 2-4 times (in place, each shares its segment with a count-0 twin), keys seen once, absent keys."""
    rep = okeys[(ocounts >= 2) & (ocounts <= 4)]
    assert len(rep) > 0
    once = okeys[ocounts == 1][:20_000]
    absent = rng.integers(0, 1 << (2 * k), size=20_000, dtype=np.uint64)
    absent = np.minimum(absent, _revcomp(absent, k))
    absent = absent[~np.isin(absent, okeys)]
    q = np.concatenate([rep, once, absent])
    want = np.concatenate([ocounts[(ocounts >= 2) & (ocounts <= 4)], np.ones(len(once), np.uint64), np.zeros(len(absent), np.uint64)])
    assert (c.query_keys(q) == want).all()


def _revcomp(x, k):
    x = np.asarray(x, dtype=np.uint64)
    rc = np.zeros_like(x)
    for j in range(k):
        rc = (rc << np.uint64(2)) | (np.uint64(3) - ((x >> np.uint64(2 * j)) & np.uint64(3)))
    return rc


def _partition_of(keys, parts_log2):
    """The fine partition of canonical keys (mix64, coarse bin from the high half, sub-bin from the low half; kmg_device.cuh)."""
    m = np.asarray(keys, dtype=np.uint64).copy()
    with np.errstate(over="ignore"):
        m ^= m >> np.uint64(33); m *= np.uint64(0xff51afd7ed558ccd)
        m ^= m >> np.uint64(33); m *= np.uint64(0xc4ceb9fe1a85ec53)
        m ^= m >> np.uint64(33)
    nc, ns = 1 << (parts_log2 // 2), 1 << (parts_log2 - parts_log2 // 2)
    coarse = ((m >> np.uint64(32)) * np.uint64(nc)) >> np.uint64(32)
    sub = ((m & np.uint64(0xffffffff)) * np.uint64(ns)) >> np.uint64(32)
    return (coarse * np.uint64(ns) + sub).astype(np.int64)


def _one_window_input(seed, k, parts_log2, per_part, hot_every):
    """Records of exactly k bases (one window each), so every partition's content is chosen: in every hot_every-th partition
    per_part / 2 keys occur twice each (more repeated keys than the sieve's side table holds: the partition goes to the
    compacting variant), in the others per_part keys of which 2 % occur 2-4 times (repeats the sieve leaves in place)."""
    rng = np.random.default_rng(seed)
    P = 1 << parts_log2
    x = rng.integers(0, 1 << (2 * k), size=int(P * per_part * 1.3), dtype=np.uint64)
    x = np.unique(np.minimum(x, _revcomp(x, k)))
    part = _partition_of(x, parts_log2)
    order = np.argsort(part, kind="stable")
    x, part = x[order], part[order]
    rank = np.arange(len(x)) - np.searchsorted(part, part)
    hot = part % hot_every == 0
    take = rank < np.where(hot, per_part // 2, per_part)
    assert (np.bincount(part[take], minlength=P) == np.where(np.arange(P) % hot_every == 0, per_part // 2, per_part)).all()
    x, hot = x[take], hot[take]
    mult = np.where(hot, 2, 1).astype(np.int64)
    cold = np.flatnonzero(~hot)
    rep = cold[rng.random(len(cold)) < 0.02]
    mult[rep] = rng.integers(2, 5, size=len(rep))
    keys = rng.permutation(np.repeat(x, mult))
    seq = np.empty((len(keys), k), dtype=np.uint8)
    for j in range(k):
        seq[:, j] = np.frombuffer(b"ACGT", dtype=np.uint8)[((keys >> np.uint64(2 * (k - 1 - j))) & np.uint64(3)).astype(np.intp)]
    seq = seq.reshape(-1)
    offsets = np.arange(0, len(seq) + 1, k, dtype=np.uint64)
    return seq, offsets


# ----------------------------------------------------------------------------------------------- cases (run in the subprocess)
def _case_c4_geometry():
    """C4's bin geometry (2^20 partitions) on 100 Mbp in one call, then a second, overlapping call."""
    import krust_b200 as kb
    from krust_b200 import _lib
    from oracle import oracle as orc
    k, n, n_rec = 21, 100_000_000, 10
    host = orc.synth_uniform(4242, 0, n)
    off = np.arange(0, n + 1, n // n_rec, dtype=np.uint64)
    okeys, ocounts, owin = orc.count_batch_mt(k, host, None, off)
    rng = np.random.default_rng(5)
    with kb.GpuKmerCounter(k, flags=_lib.KMG_FLAG_FORCE_PARTITIONED, parts_log2=20) as c:
        c.count_batch(host, None, off)
        s = c.finalize()
        assert s["path"] == 2 and s["n_windows"] == owin and s["n_distinct"] == len(okeys)
        for m in (1, 2):
            _assert_same(c.export(m, True), orc.filter_min_count(okeys, ocounts, m))
        hv, hf = c.histogram(1)
        ov, of = orc.histogram(ocounts, 1)
        assert (hv == ov).all() and (hf == of).all()
        _check_queries(c, okeys, ocounts, rng, k)
        # the first 30 Mbp (3 records) once more: the in-place result re-enters phase B as a weighted run
        m = 3 * (n // n_rec)
        c.count_batch(host[:m], None, off[:4])
        c.finalize()
        k2, c2, _ = orc.count_batch_mt(k, host[:m], None, off[:4])
        want = ocounts.copy()
        want[np.searchsorted(okeys, k2)] += c2
        _assert_same(c.export(1, True), (okeys, want))
        _check_queries(c, okeys, want, rng, k)


def _case_compacting(kmix_path):
    """Partitions the sieve hands to the compacting variant are compacted into their own capacity; a .kmix of the in-place
    result; then a second, overlapping call."""
    import krust_b200 as kb
    from krust_b200 import _lib
    from oracle import oracle as orc
    k, parts_log2 = 21, 10
    seq, off = _one_window_input(11, k, parts_log2, 2000, hot_every=64)
    okeys, ocounts, owin = orc.count_batch(k, seq, None, off)
    rng = np.random.default_rng(6)
    with kb.GpuKmerCounter(k, flags=_lib.KMG_FLAG_FORCE_PARTITIONED, parts_log2=parts_log2) as c:
        c.count_batch(seq, None, off)
        s = c.finalize()
        assert s["n_windows"] == owin and s["n_distinct"] == len(okeys)
        for m in (1, 2):
            _assert_same(c.export(m, True), orc.filter_min_count(okeys, ocounts, m))
        hv, hf = c.histogram(1)
        ov, of = orc.histogram(ocounts, 1)
        assert (hv == ov).all() and (hf == of).all()
        _check_queries(c, okeys, ocounts, rng, k)
        c.save_kmix(kmix_path)
        with open(kmix_path, "rb") as f:
            blob = f.read()
        assert blob == orc.kmix_encode(k, okeys, ocounts)
        half = (len(off) - 1) // 2
        c.count_batch(seq[:int(off[half])], None, off[:half + 1])
        c.finalize()
        k2, c2, _ = orc.count_batch(k, seq[:int(off[half])], None, off[:half + 1])
        want = ocounts.copy()
        want[np.searchsorted(okeys, k2)] += c2
        _assert_same(c.export(1, True), (okeys, want))
        _check_queries(c, okeys, want, rng, k)


def _case_every_key_repeats():
    """Every partition holds more repeated keys than the sieve takes: it stops early and the launch is repeated on the copying
    route, which reads the input the in-place attempt left intact."""
    import krust_b200 as kb
    from krust_b200 import _lib
    from oracle import oracle as orc
    k, parts_log2 = 21, 10
    seq, off = _one_window_input(12, k, parts_log2, 2000, hot_every=1)
    okeys, ocounts, owin = orc.count_batch(k, seq, None, off)
    with kb.GpuKmerCounter(k, flags=_lib.KMG_FLAG_FORCE_PARTITIONED, parts_log2=parts_log2) as c:
        c.count_batch(seq, None, off)
        s = c.finalize()
        assert s["n_windows"] == owin and s["n_distinct"] == len(okeys)
        _assert_same(c.export(1, True), (okeys, ocounts))
        hv, hf = c.histogram(1)
        ov, of = orc.histogram(ocounts, 1)
        assert (hv == ov).all() and (hf == of).all()


def _case_resplit():
    """An in-place result (with repeats left in place as count-0 twins) is re-split when a much larger second call outgrows the
    automatic partition plan: the twins are scattered with their keys and must stay invisible to the weighted count."""
    import krust_b200 as kb
    from krust_b200 import _lib
    from oracle import oracle as orc
    rng = np.random.default_rng(21)
    k, n1, n2 = 21, 2_000_000, 20_000_000
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    g1 = acgt[rng.integers(0, 4, size=n1, dtype=np.uint8)].copy()
    for _ in range(20):   # second copies of 5 kbp blocks: repeats the sieve leaves in place
        a, b = (int(x) for x in rng.integers(0, n1 - 5000, size=2))
        g1[b:b + 5000] = g1[a:a + 5000]
    g2 = np.concatenate([g1, acgt[rng.integers(0, 4, size=n2 - n1, dtype=np.uint8)]])
    okeys, ocounts, owin = orc.count_batch(k, np.concatenate([g1, g2]), None, np.array([0, n1, n1 + n2], dtype=np.uint64))
    with kb.GpuKmerCounter(k, flags=_lib.KMG_FLAG_FORCE_PARTITIONED) as c:
        c.count_batch(g1, None, np.array([0, n1], dtype=np.uint64))
        p1 = c.finalize()["table_capacity"]
        c.count_batch(g2, None, np.array([0, n2], dtype=np.uint64))
        s = c.finalize()
        assert s["table_capacity"] > p1, (p1, s["table_capacity"])   # the plan was refined: the runs were re-split
        assert s["n_windows"] == owin and s["n_distinct"] == len(okeys)
        _assert_same(c.export(1, True), (okeys, ocounts))
        hv, hf = c.histogram(1)
        ov, of = orc.histogram(ocounts, 1)
        assert (hv == ov).all() and (hf == of).all()
        _check_queries(c, okeys, ocounts, rng, k)


# ----------------------------------------------------------------------------------------------- tests
@pytest.mark.gpu
def test_one_call_at_c4_bin_geometry_in_place():
    lines = _run("c4_geometry")
    assert len(lines) == 1, lines  # the second call's consolidation merges two runs: no sieve
    m = DONE.match(lines[0])
    assert m and m.group(1) == str(1 << 20) and m.group(5) == "in place", lines


@pytest.mark.gpu
def test_compacting_variant_writes_into_the_input_in_place(tmp_path):
    lines = _run("compacting", tmp_path / "in_place.kmix")
    assert len(lines) == 1, lines
    m = DONE.match(lines[0])
    assert m and m.group(5) == "in place", lines
    assert int(m.group(2)) >= 1024 // 64, lines  # every hot partition went to the compacting variant


@pytest.mark.gpu
def test_every_key_repeated_leaves_the_in_place_route():
    lines = _run("every_key_repeats")
    assert len(lines) == 1, lines  # the repeated launch runs without the sieve
    m = STOPPED.match(lines[0])
    assert m and m.group(3) == "leaves the in-place route", lines


@pytest.mark.gpu
def test_in_place_result_is_re_split_when_the_plan_is_outgrown():
    lines = _run("resplit")
    m = DONE.match(lines[0]) if lines else None
    assert m and m.group(5) == "in place", lines  # the first call's consolidation; the merge after the re-split has two runs


if __name__ == "__main__":
    globals()["_case_" + sys.argv[1]](*sys.argv[2:])
