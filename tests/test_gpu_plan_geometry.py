"""The partitioned pipeline across its partition-plan range, against the oracle.

decide_mode (kmg_api.cu) plans P1 coarse bins x P2 sub-bins from the size hint: want = ceil(hint / 3600), P1 = ceil(sqrt(want))
and P2 = ceil(want / P1), both capped at 2048.  The plan picks the row size of the coarse scatter (partition_scatter_rows2:
16384 / P1 slots), the level-2 kernel (refine_rows below 128 sub-bins, refine_rows4 from 128 on, its rows carved from what
226 KiB leave after 3 * P2 counter words) and the level-2 layout (speculative from 64 keys per partition, exact below).  Each
geometry below names the corner of that space it reaches; each is counted whole by the oracle, then a prefix of the input is
counted once more (the first result re-enters phase B as a weighted run).  The CPU test at the end checks the reciprocal the
scatter kernels use to map a row slot to its row, for every row size a plan can produce."""
import functools
import os
import re
from typing import NamedTuple, Tuple

import numpy as np
import pytest

import krust_b200 as kb
from krust_b200 import _lib
from oracle import oracle as orc

PART = _lib.KMG_FLAG_FORCE_PARTITIONED
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "krust_b200", "csrc")


class Geometry(NamedTuple):
    hint: int                 # expected_distinct
    plan: Tuple[int, int]     # (P1, P2) the hint must plan
    n: int                    # bases
    n_rec: int                # equal records (the features below may add boundaries)
    k: int
    shape: str                # "uniform", "n_runs", "poly_a", "skewed"
    seed: int
    prefix_rec: int           # records counted again by the second call


GEOMETRIES = {
    # rows of 8 slots in A1, refine_rows4 at 2048 sub-bins (rows of 11), speculative level-2 layout (~71 keys per partition);
    # the second call (~21 keys per partition) takes the exact layout
    "G1_2048x2048": Geometry(17_000_000_000, (2048, 2048), 300_000_000, 30, 21, "uniform", 71, 9),
    # the same rows on the exact level-2 layout from the first call (~9.5 keys per partition), k=31, N runs
    "G2_2048x2048_exact": Geometry(17_000_000_000, (2048, 2048), 40_000_000, 8, 31, "n_runs", 72, 3),
    # refine_rows one sub-bin below the switch (rows of 129), and refine_rows4 at it (rows of 212); A1 rows of 128 in both
    "G3_128x127": Geometry(58_068_000, (128, 127), 60_000_000, 6, 25, "uniform", 73, 2),
    "G4_128x128": Geometry(58_982_400, (128, 128), 60_000_000, 6, 25, "uniform", 73, 2),
    # the C4 plan (A1 rows of 17, A2 rows of 28) at a size the oracle counts whole; k=32 with a poly-A record: key 0, whose mix
    # is 0, with ~10^5 windows (its bins outgrow their speculative shares: the exact routes of both levels)
    "G5_928x928_k17": Geometry(3_100_000_000, (928, 928), 100_000_000, 10, 17, "uniform", 74, 3),
    "G5_928x928_k32": Geometry(3_100_000_000, (928, 928), 100_000_000, 10, 32, "poly_a", 74, 3),
    # non-power-of-two rows (A1 11, A2 17) on the skewed input of test_c4_bin_geometry_on_skewed_input: overflow lists, the
    # per-tile exact route, and the exact layouts once the poly-A bin outgrows its share (~69 keys per partition: the
    # speculative layouts are tried first)
    "G6_1444x1443": Geometry(7_500_000_000, (1444, 1443), 144_000_000, 3, 21, "skewed", 76, 2),
}


def _offsets(n: int, n_rec: int, shape: str) -> np.ndarray:
    off = np.arange(0, n + 1, n // n_rec, dtype=np.uint64)
    if shape == "poly_a":   # a 100 kbp record of A's after the first record
        off = np.insert(off, 2, off[1] + 100_000)
    return off


def _apply_features(host: np.ndarray, off: np.ndarray, shape: str, seed: int):
    """Edits the uniform genome in place into the geometry's input."""
    n = len(host)
    rng = np.random.default_rng(seed)
    if shape == "n_runs":
        for pos, ln in zip(rng.integers(0, n - 400, size=4000), rng.integers(1, 400, size=4000)):
            host[pos:pos + ln] = ord("N")
    elif shape == "poly_a":
        host[int(off[1]):int(off[2])] = ord("A")
    elif shape == "skewed":
        u = n // 24
        block = host[1000:1600].copy()
        for pos in range(2 * u, 8 * u, 9_000):                # 600-base block every 9 kbp
            host[pos:pos + 600] = block
        sat = host[5000:5040].copy()
        host[9 * u:10 * u] = np.tile(sat, u // 40 + 1)[:u]   # satellite
        host[12 * u:13 * u + u // 2] = ord("A")               # poly-A
        host[15 * u:15 * u + (2 * u) // 5] = ord("T")         # its reverse complement: the same canonical key
        for pos in rng.integers(0, n - 10, size=300):
            host[pos:pos + 10] = ord("N")


@functools.lru_cache(maxsize=1)   # G3 and G4 count the same input
def _input_and_oracle(n: int, n_rec: int, seed: int, shape: str, k: int):
    host = orc.synth_uniform(seed, 0, n)
    off = _offsets(n, n_rec, shape)
    _apply_features(host, off, shape, seed)
    okeys, ocounts, owin = orc.count_batch_mt(k, host, None, off)
    return host, off, okeys, ocounts, owin


def _canonical(x: np.ndarray, k: int) -> np.ndarray:
    """min(x, reverse complement of x) of packed k-mers (2 bits per base, first base highest)."""
    y = ~x
    for shift, mask in ((2, 0x3333333333333333), (4, 0x0F0F0F0F0F0F0F0F), (8, 0x00FF00FF00FF00FF),
                        (16, 0x0000FFFF0000FFFF), (32, 0x00000000FFFFFFFF)):
        m = np.uint64(mask)
        y = ((y >> np.uint64(shift)) & m) | ((y & m) << np.uint64(shift))
    return np.minimum(x, y >> np.uint64(64 - 2 * k))


def _query_set(okeys, k, seed, n_present=100_000, n_absent=100_000):
    """Queries: ~n_present keys of the table spread over the key space (their indices in it), then n_absent canonical keys
    that are not in it."""
    idx = np.arange(0, len(okeys), max(1, len(okeys) // n_present))
    rng = np.random.default_rng(seed)
    cand = np.unique(_canonical(rng.integers(0, 1 << (2 * k), size=2 * n_absent, dtype=np.uint64), k))
    pos = np.minimum(np.searchsorted(okeys, cand), len(okeys) - 1)
    absent = cand[okeys[pos] != cand][:n_absent]
    assert len(absent) == n_absent
    return np.concatenate([okeys[idx], absent]), idx


def _assert_table(c, okeys, ocounts, min_counts=(1,)):
    for m in min_counts:
        gk, gc = c.export(m, True)
        fk, fc = (okeys, ocounts) if m == 1 else orc.filter_min_count(okeys, ocounts, m)
        assert len(gk) == len(fk), (m, len(gk), len(fk))
        assert (gk == fk).all() and (gc == fc).all(), m
    hv, hf = c.histogram(1)
    ov, of = orc.histogram(ocounts, 1)
    assert len(hv) == len(ov) and (hv == ov).all() and (hf == of).all()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GEOMETRIES))
def test_plan_geometry_against_oracle(name):
    import torch
    g = GEOMETRIES[name]
    if g.n >= 200_000_000:
        if torch.cuda.get_device_properties(0).total_memory < 40e9:
            pytest.skip("needs a device with 40 GB for the 300 Mbp job at 4 M partitions")
        import psutil
        if psutil.virtual_memory().available < 32e9:
            pytest.skip("the oracle and the compared tables need ~25 GB of host memory at 300 Mbp")
    dev = torch.device("cuda:0")
    host, off_np, okeys, ocounts, owin = _input_and_oracle(g.n, g.n_rec, g.seed, g.shape, g.k)
    n_rec = len(off_np) - 1
    buf = torch.empty(g.n + 64, dtype=torch.uint8, device=dev)
    offsets = torch.from_numpy(off_np.astype(np.int64)).to(dev)
    with kb.GpuKmerCounter(g.k, flags=PART, expected_distinct=g.hint) as c:
        c.synth_uniform_device(g.seed, 0, g.n, buf.data_ptr())
        if g.shape == "uniform":
            assert torch.equal(buf[:g.n].cpu(), torch.from_numpy(host))   # the device generator made the oracle's input
        else:
            buf[:g.n].copy_(torch.from_numpy(host))
        c.count_device(buf.data_ptr(), g.n, d_offsets=offsets.data_ptr(), n_records=n_rec)
        assert c.partition_plan(g.hint) == g.plan   # a changed plan formula must not go on to test another geometry
        s = c.finalize()
        assert s["path"] == 2
        assert s["n_windows"] == owin and s["n_distinct"] == len(okeys) and s["max_count"] == int(ocounts.max())
        _assert_table(c, okeys, ocounts, (1, 2))
        qk, qidx = _query_set(okeys, g.k, g.seed)
        got = c.query_keys(qk)
        assert (got[:len(qidx)] == ocounts[qidx]).all() and not got[len(qidx):].any()
        if name.startswith("G1"):
            for rem in (0, 517):   # key-space samples of the table, against the oracle counting only those keys
                gk, gc = c.export_shard(1009, rem, 1, True)
                sk, sc, _ = orc.count_batch_mt(g.k, host, None, off_np, filter_mod=1009, filter_rem=rem)
                assert len(gk) == len(sk) and (gk == sk).all() and (gc == sc).all()
        # the first records once more: the table re-enters phase B as a weighted run next to the new keys
        m = int(off_np[g.prefix_rec])
        c.count_device(buf.data_ptr(), m, d_offsets=offsets.data_ptr(), n_records=g.prefix_rec)
        s2 = c.finalize()
        assert c.partition_plan(g.hint) == g.plan
        pk, pc, pwin = orc.count_batch_mt(g.k, host[:m], None, off_np[:g.prefix_rec + 1])
        want = ocounts.copy()
        want[np.searchsorted(okeys, pk)] += pc
        assert s2["n_windows"] == owin + pwin and s2["n_distinct"] == len(okeys) and s2["max_count"] == int(want.max())
        _assert_table(c, okeys, want)
        got = c.query_keys(qk)
        assert (got[:len(qidx)] == want[qidx]).all() and not got[len(qidx):].any()


def _source_constant(path: str, name: str) -> int:
    with open(os.path.join(CSRC, path)) as f:
        m = re.search(r"constexpr\s+\w+\s+%s\s*=\s*(\d+)\s*;" % name, f.read())
    assert m, f"{name} not found in {path}"
    return int(m.group(1))


def test_row_reciprocal_is_exact_for_every_planned_row_size():
    """The scatter kernels map a row slot x to its row as __umulhi(x, magic) with magic = ceil(2^32 / cap) (the flat copy-outs
    of partition_scatter_rows(2)_kernel and refine_rows_kernel): that equals x / cap for every slot of every row size a plan can
    produce -- A1 rows of min(16384 / P1, 8192) slots for P1 in 1..2048, refine_rows rows of min(16384 / P2, 8192) slots for every
    P2 it may run with (1..127 from a plan, up to 2048 for keys pulled from other GPUs)."""
    rows_slots = _source_constant("kmg_kernels.cu", "ROWS_SLOTS")
    rows_sub_windows = _source_constant("kmg_kernels.cu", "ROWS_THREADS") // 4 * 32   # ROWS_SUB_WORDS * 32
    refine_slots = _source_constant("kmg_kernels.h", "REFINE_ROWS_SLOTS")
    refine_tile = _source_constant("kmg_kernels.h", "REFINE_TILE")
    assert (rows_slots, rows_sub_windows, refine_slots, refine_tile) == (16384, 8192, 16384, 8192)
    slots_of_cap = {}   # row size -> most slots a plan walks with it
    for slots, cap_max, n_rows_max in ((rows_slots, rows_sub_windows, rows_slots // 8), (refine_slots, refine_tile, refine_slots // 8)):
        for n_rows in range(1, n_rows_max + 1):
            cap = min(slots // n_rows, cap_max)
            assert cap >= 8 and n_rows * cap <= slots
            slots_of_cap[cap] = max(slots_of_cap.get(cap, 0), n_rows * cap)
    assert max(slots_of_cap.values()) <= 1 << 16   # the bound the kernels' comments state
    assert {8, 11, 17, 128, 129, 8192} <= set(slots_of_cap)
    for cap, n_slots in slots_of_cap.items():
        magic = ((1 << 32) + cap - 1) // cap
        assert magic < 1 << 32   # fits the kernels' uint32_t
        x = np.arange(n_slots, dtype=np.uint64)
        row = (x * np.uint64(magic)) >> np.uint64(32)
        assert (row == x // np.uint64(cap)).all(), cap
