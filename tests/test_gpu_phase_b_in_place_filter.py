"""Phase B in place (count_partitions_sieve_in_place_kernel) sets two bits of one map word per key: word (lo >> 5) & 2047, bits
lo & 31 and (lo >> 16) & 31 of the mixed key's low half lo; a key is a suspect iff both were already set.  The cases aim at that
test: a partition whose keys all share the word and both bits (every key after the first a false suspect), repeated keys alone in
their word (each first occurrence sets its bits before any other key, so only the later occurrences are suspects and the first
one is found through the filter), and partitions whose queue holds exactly SVT_L_MAX distinct keys (in place) or one more (handed
to the compacting variant).  Each case runs in a subprocess with KMG_DEBUG_SIEVE set, so the route phase B took can be read from
its stderr line, and is compared against the oracle (keys, counts, count-of-counts, device queries)."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests.test_gpu_phase_b_in_place import DONE, _partition_of, _revcomp  # noqa: E402
from tests.test_gpu_phase_b_in_place_occupancy import _count_and_check, _mix64, _random_partitions, _unmix64  # noqa: E402

SVT_L_MAX = 704  # distinct keys the side table of one partition takes (kmg_partition.cu)


def _run(case, *args):
    """Runs _case_<case>(*args) in a fresh process; returns its phase B debug lines."""
    env = dict(os.environ, KMG_DEBUG_SIEVE="1")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), case] + [str(a) for a in args]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, f"case {case} failed:\n{r.stdout[-4000:]}\n{r.stderr[-4000:]}"
    return [ln for ln in r.stderr.splitlines() if ln.startswith("[kmg] sieve:")]


def _keys_with_low_bits(rng, k, parts_log2, part, low, nbits, n):
    """n distinct canonical k-mers of fine partition `part` whose mixed values all end in the nbits bits `low`: chosen mixed values
    (coarse bin from the high half, sub-bin from the top bits of the low half) mapped back through unmix64."""
    lc, ls = parts_log2 // 2, parts_log2 - parts_log2 // 2
    coarse, sub = part >> ls, part & ((1 << ls) - 1)
    got = np.empty(0, dtype=np.uint64)
    while len(got) < n:
        hi = (np.uint64(coarse) << np.uint64(32 - lc)) | rng.integers(0, 1 << (32 - lc), size=8 * n, dtype=np.uint64)
        mid = rng.integers(0, 1 << (32 - ls - nbits), size=8 * n, dtype=np.uint64)
        lo = (np.uint64(sub) << np.uint64(32 - ls)) | (mid << np.uint64(nbits)) | np.uint64(low)
        key = _unmix64((hi << np.uint64(32)) | lo)
        key = key[key < np.uint64(1 << (2 * k))]
        key = key[key <= _revcomp(key, k)]
        got = np.unique(np.concatenate([got, key]))
    got = rng.permutation(got)[:n]
    assert (_partition_of(got, parts_log2) == part).all()
    assert ((_mix64(got) & np.uint64((1 << nbits) - 1)) == np.uint64(low)).all()
    return got


def _map_word(keys):
    return ((_mix64(keys) >> np.uint64(5)) & np.uint64(2047)).astype(np.int64)


# ----------------------------------------------------------------------------------------------- cases (run in the subprocess)
def _case_false_suspects():
    """Partition 100: 700 distinct keys that share the low 21 bits of their mixed value, hence the map word and both bits (every
    key after the first a false suspect; they all share one filter bit, so all are queued, and the table still takes them).
    Partition 101: 600 keys that share the word and the first bit, but spread their second bit over all 32 values, 100 of them
    twice.  Every other partition holds ~2000 ordinary keys."""
    rng = np.random.default_rng(41)
    k, parts_log2 = 31, 10
    same = _keys_with_low_bits(rng, k, parts_log2, 100, 0x0f0f0f, 21, 700)
    half = _keys_with_low_bits(rng, k, parts_log2, 101, 0x4321, 16, 600)
    assert len(np.unique((_mix64(half) >> np.uint64(16)) & np.uint64(31))) == 32
    keys = np.concatenate([_random_partitions(rng, k, parts_log2, 2000, {100, 101}), same, half, half[:100]])
    _count_and_check(k, parts_log2, keys, rng)


def _case_lone_repeats():
    """Partitions 200-215: 1200 keys each, every one alone in its map word, 300 of them occurring 2-4 times.  Whichever
    occurrence of a repeated key comes first sets both bits of a word no other key touches; only its later occurrences are
    suspects, and the first one is queued through the filter alone."""
    rng = np.random.default_rng(42)
    k, parts_log2 = 31, 10
    lone = set(range(200, 216))
    pool = np.unique(_random_partitions(rng, k, parts_log2, 3000, set()))
    part, word = _partition_of(pool, parts_log2), _map_word(pool)
    keys = [_random_partitions(rng, k, parts_log2, 2000, lone)]
    for p in sorted(lone):
        mine = pool[part == p]
        _, first = np.unique(word[part == p], return_index=True)
        mine = rng.permutation(mine[first])[:1200]
        assert len(mine) == 1200 and len(np.unique(_map_word(mine))) == 1200
        keys += [mine, np.repeat(mine[:300], rng.integers(1, 4, size=300))]
    _count_and_check(k, parts_log2, np.concatenate(keys), rng)


def _case_table_limit(n_distinct):
    """Partition 100: n_distinct keys that share the low 16 bits of their mixed value (all queued: each claims a slot of the side
    table), 100 of them twice.  Every other partition holds ~2000 ordinary keys."""
    rng = np.random.default_rng(43)
    k, parts_log2 = 31, 10
    full = _keys_with_low_bits(rng, k, parts_log2, 100, 0xa5a5, 16, int(n_distinct))
    keys = np.concatenate([_random_partitions(rng, k, parts_log2, 2000, {100}), full, full[:100]])
    _count_and_check(k, parts_log2, keys, rng)


# ----------------------------------------------------------------------------------------------- tests
@pytest.mark.gpu
def test_false_suspects_sharing_word_and_both_bits_stay_in_place():
    lines = _run("false_suspects")
    assert len(lines) == 1, lines
    m = DONE.match(lines[0])
    assert m and m.group(2) == "0" and m.group(5) == "in place", lines


@pytest.mark.gpu
def test_repeats_alone_in_their_map_word_are_found():
    lines = _run("lone_repeats")
    assert len(lines) == 1, lines
    m = DONE.match(lines[0])
    assert m and m.group(2) == "0" and m.group(5) == "in place", lines


@pytest.mark.gpu
@pytest.mark.parametrize("n_distinct, handed_back", [(SVT_L_MAX, 0), (SVT_L_MAX + 1, 1)])
def test_side_table_limit(n_distinct, handed_back):
    lines = _run("table_limit", n_distinct)
    assert len(lines) == 1, lines
    m = DONE.match(lines[0])
    assert m and m.group(5) == "in place" and int(m.group(2)) == handed_back, lines


if __name__ == "__main__":
    globals()["_case_" + sys.argv[1]](*sys.argv[2:])
