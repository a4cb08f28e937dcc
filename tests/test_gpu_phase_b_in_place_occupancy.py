"""Phase B in place (count_partitions_sieve_in_place_kernel): one key stage per CTA, a 2^16-bit map, four CTAs per SM.  The
cases aim at what the smaller map and the single stage exercise: partitions whose keys all collide in the bit map, partitions
that fill the stage exactly (4096 entries), one short of it and empty ones, and the plans of C1 and of a C4 slice.  Each case
runs in a subprocess with KMG_DEBUG_SIEVE set, so the route phase B took can be read from its stderr line, and is compared
against the oracle (keys, counts, count-of-counts)."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests.test_gpu_phase_b_in_place import DONE, _assert_same, _check_queries, _partition_of, _revcomp  # noqa: E402

_M1, _M2 = np.uint64(0xff51afd7ed558ccd), np.uint64(0xc4ceb9fe1a85ec53)
_U1, _U2 = np.uint64(0x4f74430c22a54005), np.uint64(0x9cb4b2f8129337db)   # their inverses mod 2^64


def _mix64(x):
    x = np.asarray(x, dtype=np.uint64).copy()
    with np.errstate(over="ignore"):
        x ^= x >> np.uint64(33); x *= _M1
        x ^= x >> np.uint64(33); x *= _M2
        x ^= x >> np.uint64(33)
    return x


def _unmix64(x):
    x = np.asarray(x, dtype=np.uint64).copy()
    with np.errstate(over="ignore"):
        x ^= x >> np.uint64(33); x *= _U2
        x ^= x >> np.uint64(33); x *= _U1
        x ^= x >> np.uint64(33)
    return x


def _run(case, *args):
    """Runs _case_<case>(*args) in a fresh process; returns its phase B debug lines."""
    env = dict(os.environ, KMG_DEBUG_SIEVE="1")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), case] + [str(a) for a in args]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, f"case {case} failed:\n{r.stdout[-4000:]}\n{r.stderr[-4000:]}"
    return [ln for ln in r.stderr.splitlines() if ln.startswith("[kmg] sieve:")]


def _records(keys, k):
    """One record of exactly k bases per key, so every key lands in the partition it was chosen for."""
    seq = np.empty((len(keys), k), dtype=np.uint8)
    for j in range(k):
        seq[:, j] = np.frombuffer(b"ACGT", dtype=np.uint8)[((keys >> np.uint64(2 * (k - 1 - j))) & np.uint64(3)).astype(np.intp)]
    return seq.reshape(-1), np.arange(0, len(keys) * k + 1, k, dtype=np.uint64)


def _random_partitions(rng, k, parts_log2, per_part, skip):
    """per_part distinct canonical keys in every partition not in `skip`, 2 % of them occurring 2-4 times."""
    P = 1 << parts_log2
    x = rng.integers(0, 1 << (2 * k), size=int(P * per_part * 1.3), dtype=np.uint64)
    x = np.unique(np.minimum(x, _revcomp(x, k)))
    part = _partition_of(x, parts_log2)
    order = np.argsort(part, kind="stable")
    x, part = x[order], part[order]
    rank = np.arange(len(x)) - np.searchsorted(part, part)
    x = x[(rank < per_part) & ~np.isin(part, list(skip))]
    mult = np.ones(len(x), dtype=np.int64)
    rep = rng.random(len(x)) < 0.02
    mult[rep] = rng.integers(2, 5, size=int(rep.sum()))
    return np.repeat(x, mult)


def _count_and_check(k, parts_log2, keys, rng, **kw):
    """Counts the keys (shuffled, one record each) in one call and compares export, histogram and device queries with the oracle."""
    import krust_b200 as kb
    from krust_b200 import _lib
    from oracle import oracle as orc
    seq, off = _records(rng.permutation(keys), k)
    okeys, ocounts, owin = orc.count_batch(k, seq, None, off)
    with kb.GpuKmerCounter(k, flags=_lib.KMG_FLAG_FORCE_PARTITIONED, parts_log2=parts_log2, **kw) as c:
        c.count_batch(seq, None, off)
        s = c.finalize()
        assert s["path"] == 2 and s["n_windows"] == owin and s["n_distinct"] == len(okeys)
        for m in (1, 2):
            _assert_same(c.export(m, True), orc.filter_min_count(okeys, ocounts, m))
        hv, hf = c.histogram(1)
        ov, of = orc.histogram(ocounts, 1)
        assert (hv == ov).all() and (hf == of).all()
        _check_queries(c, okeys, ocounts, rng, k)


# ----------------------------------------------------------------------------------------------- cases (run in the subprocess)
def _colliding_keys(rng, k, parts_log2, part, low16, n):
    """n distinct canonical k-mers of fine partition `part` whose mixed values all end in the 16 bits low16: chosen mixed values
    (coarse bin from the high half, sub-bin from the top bits of the low half) mapped back through unmix64."""
    lc, ls = parts_log2 // 2, parts_log2 - parts_log2 // 2
    coarse, sub = part >> ls, part & ((1 << ls) - 1)
    got = np.empty(0, dtype=np.uint64)
    while len(got) < n:
        hi = (np.uint64(coarse) << np.uint64(32 - lc)) | rng.integers(0, 1 << (32 - lc), size=8 * n, dtype=np.uint64)
        mid = rng.integers(0, 1 << (16 - ls), size=8 * n, dtype=np.uint64)
        lo = (np.uint64(sub) << np.uint64(32 - ls)) | (mid << np.uint64(16)) | np.uint64(low16)
        key = _unmix64((hi << np.uint64(32)) | lo)
        key = key[key < np.uint64(1 << (2 * k))]
        key = key[key <= _revcomp(key, k)]
        got = np.unique(np.concatenate([got, key]))
    got = rng.permutation(got)[:n]
    assert (_partition_of(got, parts_log2) == part).all() and ((_mix64(got) & np.uint64(0xffff)) == np.uint64(low16)).all()
    return got


def _case_bit_map_collisions():
    """Partition 100: 1500 keys that all share one bit of the map (every one a suspect: more than the table takes, the partition
    goes to the compacting variant).  Partition 101: 600 such keys, 100 of them twice (a long queue the table still holds: it
    stays in place).  Every other partition holds ~2000 ordinary keys."""
    rng = np.random.default_rng(31)
    k, parts_log2 = 31, 10
    full = _colliding_keys(rng, k, parts_log2, 100, 0x5a5a, 1500)
    held = _colliding_keys(rng, k, parts_log2, 101, 0x0123, 600)
    keys = np.concatenate([_random_partitions(rng, k, parts_log2, 2000, {100, 101}), full, held, held[:100]])
    _count_and_check(k, parts_log2, keys, rng)


def _case_partition_sizes():
    """Partitions of exactly 4096 entries (a full key stage), 4095 (odd: the pad entry shares the stage) and 0, with 50 repeated
    keys each in the first two; the others hold ~3750 entries, so the speculative capacity exceeds 4096."""
    rng = np.random.default_rng(32)
    k, parts_log2 = 21, 10
    P = 1 << parts_log2
    special = {7: 4096, 300: 4095, 301: 0, 302: 0, 900: 4096}
    keys = [_random_partitions(rng, k, parts_log2, 3600, set(special))]
    x = rng.integers(0, 1 << (2 * k), size=P * 6000, dtype=np.uint64)
    x = np.unique(np.minimum(x, _revcomp(x, k)))
    part = _partition_of(x, parts_log2)
    for p, n in special.items():
        if n:
            mine = rng.permutation(x[part == p])[:n - 50]
            assert len(mine) == n - 50
            keys.append(np.concatenate([mine, mine[:50]]))
    keys = np.concatenate(keys)
    sizes = np.bincount(_partition_of(keys, parts_log2), minlength=P)
    assert all(sizes[p] == n for p, n in special.items())
    _count_and_check(k, parts_log2, keys, rng)


def _case_plan(plan_bases):
    """100 Mbp (C1's generator and records) counted in one call with the partition plan for plan_bases bases, as bench.py plans C1
    (plan_bases = 1e8) and a slice of C4 (--plan-bases 3.1e9)."""
    import krust_b200 as kb
    from oracle import oracle as orc
    k, n, n_rec = 21, 100_000_000, 100
    host = orc.synth_uniform(42, 0, n)
    off = np.arange(0, n + 1, n // n_rec, dtype=np.uint64)
    okeys, ocounts, owin = orc.count_batch_mt(k, host, None, off)
    rng = np.random.default_rng(7)
    with kb.GpuKmerCounter(k, expected_distinct=int(float(plan_bases) * 1.03) + 1024) as c:
        c.count_batch(host, None, off)
        s = c.finalize()
        assert s["path"] == 2 and s["n_windows"] == owin and s["n_distinct"] == len(okeys)
        _assert_same(c.export(1, True), (okeys, ocounts))
        hv, hf = c.histogram(1)
        ov, of = orc.histogram(ocounts, 1)
        assert (hv == ov).all() and (hf == of).all()
        _check_queries(c, okeys, ocounts, rng, k)


# ----------------------------------------------------------------------------------------------- tests
@pytest.mark.gpu
def test_bit_map_collisions_go_to_the_compacting_variant():
    lines = _run("bit_map_collisions")
    assert len(lines) == 1, lines
    m = DONE.match(lines[0])
    assert m and m.group(5) == "in place", lines
    assert int(m.group(2)) == 1, lines  # only the partition of 1500 colliding keys


@pytest.mark.gpu
def test_full_odd_and_empty_partitions_in_place():
    lines = _run("partition_sizes")
    assert len(lines) == 1, lines
    m = DONE.match(lines[0])
    assert m and m.group(1) == "1024" and m.group(2) == "0" and m.group(5) == "in place", lines


@pytest.mark.gpu
@pytest.mark.parametrize("plan_bases", ["1e8", "3.1e9"])
def test_plan_geometry_in_place(plan_bases):
    lines = _run("plan", plan_bases)
    assert lines, lines
    m = DONE.match(lines[0])
    assert m and m.group(5) == "in place", lines


if __name__ == "__main__":
    globals()["_case_" + sys.argv[1]](*sys.argv[2:])
