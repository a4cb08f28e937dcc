"""Parity tests proper: the CUDA path, called through the C ABI, against the CPU oracle on the same
inputs (bit-exact: integer work).  All of these need a GPU (`-m gpu`)."""
import os

import numpy as np
import pytest

import krust_b200 as kb
from krust_b200 import _lib
from oracle import oracle as orc
from tests import kats

pytestmark = pytest.mark.gpu

PART = _lib.KMG_FLAG_FORCE_PARTITIONED
FLAG_SETS = {"auto": 0, "hash": _lib.KMG_FLAG_FORCE_HASH, "hash_nopreagg": _lib.KMG_FLAG_FORCE_HASH | _lib.KMG_FLAG_NO_PREAGG,
             "part": PART, "part_nopreagg": PART | _lib.KMG_FLAG_NO_PREAGG}


def gpu_count(k, records, quals=None, min_quality=None, flags=0, batch_bases=0, min_count=1, expected_distinct=0, parts_log2=0):
    if (flags & PART) and parts_log2 == 0:
        parts_log2 = 1 + (k % 7)  # exercise many different partition counts (2..128) on small inputs
    with kb.GpuKmerCounter(k, min_quality=min_quality, flags=flags, batch_bases=batch_bases,
                           expected_distinct=expected_distinct, parts_log2=parts_log2) as c:
        c.count_records(records, quals)
        s = c.finalize()
        keys, counts = c.export(min_count, sorted=True)
        return keys, counts, s


def assert_same(gpu, oracle):
    gk, gc = gpu[0], gpu[1]
    ok, oc = oracle[0], oracle[1]
    assert len(gk) == len(ok), (len(gk), len(ok))
    assert (gk == ok).all() and (gc == oc).all()


@pytest.mark.parametrize("flags", list(FLAG_SETS), ids=list(FLAG_SETS))
@pytest.mark.parametrize("kat", kats.COUNT_KATS, ids=[k[0] for k in kats.COUNT_KATS])
def test_reference_kats_through_c_abi(kat, flags):
    _, _, k, records, quals, q, expected = kat
    keys, counts, s = gpu_count(k, records, quals, q, FLAG_SETS[flags])
    got = {kb.unpack_to_string(a, k): int(b) for a, b in zip(keys.tolist(), counts.tolist())}
    assert got == expected
    assert s["n_windows"] == sum(expected.values()) and s["n_distinct"] == len(expected)
    assert s["n_records"] == len(records)


def _random_records(rng, n_rec, max_len, alphabet, min_len=0):
    recs, quals = [], []
    for _ in range(n_rec):
        n = int(rng.integers(min_len, max_len))
        recs.append(bytes(rng.choice(alphabet, size=n).tolist()))
        quals.append(bytes((rng.integers(0, 42, size=n) + 33).astype(np.uint8).tolist()))
    return recs, quals


@pytest.mark.parametrize("flags", ["auto", "hash", "part"])
def test_randomised_differential_all_k(flags):
    """Random records with N / IUPAC / blanks / lower case, quality thresholds, every k in 1..32."""
    rng = np.random.default_rng(77)
    alphabet = list(b"ACGT" * 12 + b"acgtNnRY -")
    for k in range(1, 33):
        recs, quals = _random_records(rng, int(rng.integers(1, 40)), 400, alphabet)
        q = [None, 0, 19, 20, 30, 93, 250][k % 7]
        use_qual = k % 3 != 0
        oracle = orc.count_records(k, recs, quals if use_qual else None, q, mode="literal")
        gpu = gpu_count(k, recs, quals if use_qual else None, q, FLAG_SETS[flags])
        assert_same(gpu, oracle)
        assert gpu[2]["n_windows"] == oracle[2]


@pytest.mark.parametrize("k", [1, 2, 13, 21, 31, 32])
def test_chunked_feed_equals_single_shot(k):
    """Tiny staging buffers force many chunks (record-spanning, k-1 overlap) -- results must not change."""
    rng = np.random.default_rng(k)
    recs, quals = _random_records(rng, 60, 3000, list(b"ACGT" * 30 + b"N"), min_len=0)
    recs.append(bytes(rng.choice(list(b"ACGT"), size=50_000).tolist()))  # one record much longer than a chunk
    quals.append(b"I" * 50_000)
    oracle = orc.count_records(k, recs, quals, 20, mode="rolling")
    for bb in (4096, 10_000):
        gpu = gpu_count(k, recs, quals, 20, _lib.KMG_FLAG_FORCE_HASH, batch_bases=bb)
        assert_same(gpu, oracle)
        # partitioned pipeline: every chunk becomes a run; > 31 runs force intermediate consolidations (result + runs merge)
        gpu = gpu_count(k, recs, quals, 20, PART, batch_bases=bb, parts_log2=5)
        assert_same(gpu, oracle)
        assert gpu[2]["path"] == 2 and gpu[2]["n_grows"] >= 1 and gpu[2]["n_windows"] == oracle[2]


def test_many_short_reads_record_boundaries():
    """150 bp reads back to back: windows must never span records (src/run.rs:500-503)."""
    rng = np.random.default_rng(150)
    genome = rng.choice(list(b"ACGT"), size=20_000).astype(np.uint8)
    recs = []
    for _ in range(3000):
        s = int(rng.integers(0, len(genome) - 150))
        r = genome[s:s + 150].copy()
        if rng.random() < 0.2:
            r[int(rng.integers(0, 150))] = ord("N")
        recs.append(r.tobytes())
    for k in (21, 31):
        oracle = orc.count_records(k, recs, mode="rolling")
        assert_same(gpu_count(k, recs, flags=_lib.KMG_FLAG_FORCE_HASH), oracle)
        assert_same(gpu_count(k, recs, flags=_lib.KMG_FLAG_FORCE_HASH, batch_bases=8192), oracle)
        assert_same(gpu_count(k, recs, flags=PART, parts_log2=6), oracle)
        assert_same(gpu_count(k, recs, flags=PART, batch_bases=8192, parts_log2=13), oracle)


def test_k32_poly_t_and_empty_sentinel():
    """EMPTY = ~0 is TTT..T for k=32, which is never canonical; key 0 (AAA..A) is a real key."""
    recs = [b"T" * 40, b"A" * 35, b"ACGT" * 20]
    oracle = orc.count_records(32, recs, mode="literal")
    gpu = gpu_count(32, recs)
    assert_same(gpu, oracle)
    assert gpu[0][0] == 0 and gpu[1][0] == 9 + 4


def test_skewed_high_multiplicity():
    """poly-A / dinucleotide / satellite repeats exercise the in-thread pre-aggregation and contended atomics."""
    recs = [b"A" * 100_000, b"AC" * 50_000, b"ACGTTGCA" * 20_000, b"GATTACA" * 10_000]
    for k in (5, 21, 32):
        oracle = orc.count_records(k, recs, mode="rolling")
        for f in ("auto", "hash", "hash_nopreagg", "part", "part_nopreagg"):
            assert_same(gpu_count(k, recs, flags=FLAG_SETS[f]), oracle)


def test_table_growth_never_drops_keys():
    rng = np.random.default_rng(5)
    recs = [bytes(rng.choice(list(b"ACGT"), size=300_000).tolist()) for _ in range(8)]
    oracle = orc.count_records(25, recs, mode="rolling")
    with kb.GpuKmerCounter(25, batch_bases=200_000) as c:  # starts at 4 Mi slots... force growth with a tiny hint
        pass
    with kb.GpuKmerCounter(25, batch_bases=100_000, expected_distinct=1000) as c:
        for r in recs:
            c.count_records([r])
        s = c.finalize()
        keys, counts = c.export(1, True)
    assert s["n_grows"] >= 1
    assert_same((keys, counts), oracle)
    assert s["n_distinct"] == len(oracle[0]) and s["n_windows"] == oracle[2]


def test_min_count_histogram_and_kmix(tmp_path):
    rng = np.random.default_rng(8)
    genome = bytes(rng.choice(list(b"ACGT"), size=5000).tolist())
    recs = [genome[i:i + 200] for i in rng.integers(0, 4800, size=2000)]
    for k, flags in ((12, 0), (21, _lib.KMG_FLAG_FORCE_HASH), (21, PART), (12, PART)):
        okeys, ocounts, _ = orc.count_records(k, recs, mode="rolling")
        with kb.GpuKmerCounter(k, flags=flags, parts_log2=4 if flags & PART else 0) as c:
            c.count_records(recs)
            s = c.finalize()
            assert s["max_count"] == int(ocounts.max())
            for m in (0, 1, 2, 5, 10**9):
                fk, fc = orc.filter_min_count(okeys, ocounts, m)
                assert_same(c.export(m, True), (fk, fc))
                hv, hf = c.histogram(m)
                ov, of = orc.histogram(ocounts, m)
                assert (hv == ov).all() and (hf == of).all()
                text = b"".join(b"%d\t%d\n" % (int(a), int(b)) for a, b in zip(hv, hf))
                assert text == b"".join(b"%d\t%d\n" % (int(a), int(b)) for a, b in zip(ov, of))
            # unsorted export is the same multiset
            uk, uc = c.export(1, False)
            order = np.argsort(uk)
            assert_same((uk[order], uc[order]), (okeys, ocounts))
            p = tmp_path / f"k{k}.kmix"
            c.save_kmix(p)
        blob = p.read_bytes()
        kk, ikeys, icounts = orc.kmix_decode(blob)  # header + CRC valid, record set equal (parity definition v)
        order = np.argsort(ikeys)
        assert kk == k and len(blob) == 18 + 16 * len(okeys)
        assert_same((ikeys[order], icounts[order]), (okeys, ocounts))
        assert kb.load_index(p).counts() == dict(zip(okeys.tolist(), ocounts.tolist()))
        assert blob == orc.kmix_encode(k, okeys, ocounts)  # sorted writer => byte-identical to a sorted reference-format file


def test_histogram_overflow_tail():
    """counts >= 65536 leave the dense bins and go through the overflow list."""
    recs = [b"A" * 70_000, b"C" * 200_000, b"ACGT" * 10]
    okeys, ocounts, _ = orc.count_records(4, recs, mode="rolling")
    for flags in (0, _lib.KMG_FLAG_FORCE_HASH, PART):
        with kb.GpuKmerCounter(4, flags=flags) as c:
            c.count_records(recs)
            c.finalize()
            hv, hf = c.histogram(1)
        ov, of = orc.histogram(ocounts, 1)
        assert (hv == ov).all() and (hf == of).all() and hv.max() >= 65536


def test_reference_named_entry_points(golden_dir, tmp_path):
    fx = os.path.join(golden_dir, "fixtures")
    # tests/library_tests.rs:36-52, :262-270 and the derived fixture answers (SURVEY 8c)
    assert kb.count_kmers(os.path.join(fx, "simple.fa"), 3) == {"AAT": 1, "ACA": 1, "ACG": 4, "ATC": 1, "GTA": 3, "TAA": 1}
    assert kb.count_kmers(os.path.join(fx, "soft_masked.fa"), 3) == {"AAA": 2}
    assert kb.count_kmers(os.path.join(fx, "with_n.fa"), 4) == {"AATC": 1, "ACGT": 2, "ATTA": 1, "GTAA": 1, "TACA": 1}
    # FASTA == FASTQ (tests/integration_tests.rs:486-523)
    assert kb.count_kmers(os.path.join(fx, "simple.fa"), 3) == kb.count_kmers(os.path.join(fx, "simple.fq"), 3)
    assert kb.count_kmers_streaming(os.path.join(fx, "with_n.fq"), 3) == kb.count_kmers(os.path.join(fx, "with_n.fa"), 3)
    # quality (tests/quality_tests.rs; src/streaming.rs:1165-1189)
    lq = os.path.join(fx, "low_quality.fq")
    assert kb.count_kmers_with_quality(lq, 4, "auto", 20) == {"AATC": 1, "ACGT": 1, "ATTA": 1, "GTAA": 1, "TACA": 1}
    assert kb.count_kmers_with_quality(lq, 4, "auto", None) == kb.count_kmers(os.path.join(fx, "simple.fa"), 4)
    assert kb.count_kmers_with_quality(os.path.join(fx, "simple.fa"), 4, "auto", 40) == kb.count_kmers(os.path.join(fx, "simple.fa"), 4)
    # packed seams
    packed = kb.count_kmers_from_sequences(iter([b"ACGTACGT", b"TGCATGCA"]), kb.KmerLength(4))
    okeys, ocounts, _ = orc.count_records(4, [b"ACGTACGT", b"TGCATGCA"])
    assert packed == dict(zip(okeys.tolist(), ocounts.tolist()))
    assert kb.count_kmers_streaming_packed(os.path.join(fx, "simple.fa"), kb.KmerLength(3)) == kb.count_kmers_sequential(os.path.join(fx, "simple.fa"), 3)
    with pytest.raises(kb.KmerLengthError):
        kb.count_kmers(os.path.join(fx, "simple.fa"), 0)
    with pytest.raises(kb.KmerLengthError):
        kb.count_kmers(os.path.join(fx, "simple.fa"), 33)
    # builder (src/builder.rs): min_count, histogram, writer
    b = kb.KmerCounter.new().k(3).min_count(2)
    assert b.count(os.path.join(fx, "simple.fa")) == {"ACG": 4, "GTA": 3}
    assert b.histogram(os.path.join(fx, "simple.fa")) == {3: 1, 4: 1}
    a8 = tmp_path / "a8.fa"; a8.write_bytes(b">s\nAAAAAAAA\n")
    assert kb.KmerCounter.new().k(3).histogram(a8) == {6: 1}  # tests/integration_tests.rs:767-799
    import io
    out = io.BytesIO()
    kb.KmerCounter.new().k(3).format("tsv").count_to_writer(os.path.join(fx, "soft_masked.fa"), out)
    assert out.getvalue() == b"AAA\t2\n"  # tests/integration_tests.rs:263-281
    out = io.BytesIO()
    kb.KmerCounter.new().k(3).format("histogram").count_to_writer(a8, out)
    assert out.getvalue() == b"6\t1\n"
    empty = tmp_path / "empty.fa"; empty.write_bytes(b"")
    assert kb.count_kmers(empty, 3) == {}
    seen = []
    kb.KmerCounter.new().k(3).count_with_progress(os.path.join(fx, "simple.fa"), seen.append)
    assert seen and seen[-1] == {"sequences_processed": 2, "bases_processed": 15}


def test_prepacked_batch_feed():
    """kmg_acquire_batch / kmg_submit_batch: the Rust reader's zero-copy path (2-bit words + valid/start bits), a ring of four
    pinned batches whose copies overlap the previous batch's scan.  Ten batches (the ring wraps twice), every engine path."""
    rng = np.random.default_rng(31)
    recs = [bytes(rng.choice(list(b"ACGTN"), p=[.24, .24, .24, .24, .04], size=int(rng.integers(1, 900))).tolist()) for _ in range(500)]
    code = np.full(256, 255, dtype=np.uint8)
    for ch, v in zip(b"ACGTacgt", [0, 1, 2, 3, 0, 1, 2, 3]):
        code[ch] = v
    for k, flags, pl in ((17, _lib.KMG_FLAG_FORCE_HASH, 0), (21, PART, 5), (12, 0, 0), (31, 0, 0)):
        oracle = orc.count_records(k, recs, mode="rolling")
        with kb.GpuKmerCounter(k, batch_bases=32768, flags=flags, parts_log2=pl) as c:
            per = len(recs) // 10
            for bi in range(10):
                b = c.acquire_batch()
                words = (b.capacity_bases + 31) // 32
                bases = np.ctypeslib.as_array(b.bases2bit, shape=(words,))
                valid = np.ctypeslib.as_array(b.valid_bits, shape=(words,))
                start = np.ctypeslib.as_array(b.start_bits, shape=(words,))
                assert not bases.any() and not valid.any() and not start.any()     # handed out zeroed
                pos = 0
                chunk = recs[bi * per:(bi + 1) * per] if bi < 9 else recs[9 * per:]
                for r in chunk:
                    start[pos // 32] |= np.uint32(1 << (31 - pos % 32))
                    for ch in r:
                        cd = code[ch]
                        if cd != 255:
                            bases[pos // 32] |= np.uint64(int(cd) << (62 - 2 * (pos % 32)))
                            valid[pos // 32] |= np.uint32(1 << (31 - pos % 32))
                        pos += 1
                assert pos <= b.capacity_bases
                b.n_bases = pos
                b.n_records = len(chunk)
                c.submit_batch(b)
            s = c.finalize()
            assert_same(c.export(1, True), oracle)
            assert s["n_windows"] == oracle[2] and s["n_records"] == len(recs)


def test_device_resident_path_and_synthetic_generator():
    """kmg_count_ascii_device on a synthetic genome generated on the device; the generator must agree with
    the oracle's host generator, and the counts with the oracle's."""
    import torch
    n = 3_000_000
    dev = torch.device("cuda:0")
    buf = torch.empty(n, dtype=torch.uint8, device=dev)
    for k, flags in ((21, 0), (12, 0), (5, 0), (31, 0), (9, _lib.KMG_FLAG_FORCE_HASH), (21, PART), (32, PART), (7, PART)):
        with kb.GpuKmerCounter(k, flags=flags) as c:
            c.synth_uniform_device(42, 0, n, buf.data_ptr())
            host = buf.cpu().numpy()
            assert (host == orc.synth_uniform(42, 0, n)).all()
            offsets = torch.tensor([0, 1_000_000, 1_000_000, 2_500_000, n], dtype=torch.int64, device=dev)  # incl. an empty record
            c.count_device(buf.data_ptr(), n, d_offsets=offsets.data_ptr(), n_records=4)
            s = c.finalize()
            gpu = c.export(1, True)
        oracle = orc.count_batch(k, host, None, offsets.cpu().numpy().astype(np.uint64), mode="rolling")
        assert_same(gpu, oracle)
        assert s["n_windows"] == oracle[2] and s["n_windows"] == n - 3 * (k - 1)


def test_extract_and_insert_equal_direct_count():
    """Owner bucketing (K4) + weighted upsert: the multi-GPU data path on one device."""
    import torch
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(12)
    host = rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8), p=[.245, .245, .245, .245, .02], size=1_500_000).astype(np.uint8)
    seq = torch.from_numpy(host).to(dev)
    offsets_np = np.array([0, 400_000, 900_000, len(host)], dtype=np.uint64)
    offsets = torch.from_numpy(offsets_np.astype(np.int64)).to(dev)
    for k in (11, 21, 32):
        oracle = orc.count_batch(k, host, None, offsets_np, mode="rolling")
        for n_shards in (1, 2, 8, 64, 4096, 8192):  # 4096: the staged scatter kernel, 8192: partition_scatter_kernel
            out = torch.empty(len(host), dtype=torch.int64, device=dev)
            with kb.GpuKmerCounter(k) as c:
                counts = c.extract_keys_device(seq.data_ptr(), len(host), n_shards, out.data_ptr(), len(host),
                                               d_offsets=offsets.data_ptr(), n_records=3)
            assert int(counts.sum()) == oracle[2]
            keys = out[: int(counts.sum())].cpu().numpy().view(np.uint64)
            # every key sits in its owner's bucket
            bounds = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
            for p in range(n_shards):
                sample = keys[bounds[p]:bounds[p + 1]][:50]
                assert all(kb.owner_of(int(x), n_shards) == p for x in sample)
            uk, uc = np.unique(keys, return_counts=True)
            assert_same((uk, uc.astype(np.uint64)), oracle)
            # upsert the buckets into a fresh table, half of them as (key, count) pairs
            for flags2 in (_lib.KMG_FLAG_FORCE_HASH, PART):
              with kb.GpuKmerCounter(k, flags=flags2, parts_log2=5 if flags2 == PART else 0) as c2:
                half = len(keys) // 2
                c2.insert_keys_device(out.data_ptr(), half)
                rest_k, rest_c = np.unique(keys[half:], return_counts=True)
                rk = torch.from_numpy(rest_k.view(np.int64)).to(dev); rc = torch.from_numpy(rest_c.astype(np.int64)).to(dev)
                c2.insert_keys_device(rk.data_ptr(), len(rest_k), rc.data_ptr())
                c2.finalize()
                assert_same(c2.export(1, True), oracle)


@pytest.mark.parametrize("k,flags", [(21, 0), (21, _lib.KMG_FLAG_FORCE_HASH), (12, 0), (5, 0)])
def test_full_size_100mbp_oracle_and_properties(k, flags):
    """BASELINE configs C1 (k=21) and C2 (k=12, k=5) at full size (G100: 100 Mbp, 100 records, seed 42): the sorted
    (key, count) list and the histogram text against the multi-threaded rolling oracle, plus size-independent properties --
    sum of counts == windows, reverse-complement invariance of the whole table, linearity (counting the genome twice
    doubles every count), histogram consistency."""
    import torch
    dev = torch.device("cuda:0")
    n, n_rec = 100_000_000, 100
    buf = torch.empty(n, dtype=torch.uint8, device=dev)
    offsets = torch.arange(0, n + 1, n // n_rec, dtype=torch.int64, device=dev)
    with kb.GpuKmerCounter(k, flags=flags, expected_distinct=n if k > 13 else 0) as c:
        c.synth_uniform_device(42, 0, n, buf.data_ptr())
        c.count_device(buf.data_ptr(), n, d_offsets=offsets.data_ptr(), n_records=n_rec)
        s = c.finalize()
        assert s["n_windows"] == n - n_rec * (k - 1)
        keys, counts = c.export(1, True)
        assert int(counts.sum()) == s["n_windows"] and len(keys) == s["n_distinct"]
        assert (np.diff(keys.astype(np.int64)) > 0).all()  # sorted, no duplicates
        hv, hf = c.histogram(1)
        assert int(hf.sum()) == s["n_distinct"] and int((hv * hf).sum()) == s["n_windows"]
        assert (np.diff(hv.astype(np.int64)) > 0).all()
        # the oracle on the same bytes (generated on the host by the oracle's own generator)
        host = orc.synth_uniform(42, 0, n)
        okeys, ocounts, owin = orc.count_batch_mt(k, host, None, np.arange(0, n + 1, n // n_rec, dtype=np.uint64))
        del host
        assert owin == s["n_windows"] and s["n_distinct"] == len(okeys)
        assert_same((keys, counts), (okeys, ocounts))
        ov, of = orc.histogram(ocounts, 1)
        assert b"".join(b"%d\t%d\n" % (int(a), int(b)) for a, b in zip(hv, hf)) == b"".join(b"%d\t%d\n" % (int(a), int(b)) for a, b in zip(ov, of))
        del okeys, ocounts
        # linearity
        c.count_device(buf.data_ptr(), n, d_offsets=offsets.data_ptr(), n_records=n_rec)
        c.finalize()
        keys2, counts2 = c.export(1, True)
        assert (keys2 == keys).all() and (counts2 == 2 * counts).all()
    # reverse complement of every record gives the identical table
    lut = torch.zeros(256, dtype=torch.uint8, device=dev)
    for a, b in zip(b"ACGT", b"TGCA"):
        lut[a] = b
    rc = lut[buf.view(n_rec, n // n_rec).flip(1).long()].contiguous().view(-1)
    with kb.GpuKmerCounter(k, flags=flags, expected_distinct=n if k > 13 else 0) as c:
        c.count_device(rc.data_ptr(), n, d_offsets=offsets.data_ptr(), n_records=n_rec)
        c.finalize()
        keys3, counts3 = c.export(1, True)
    assert (keys3 == keys).all() and (counts3 == counts).all()


def test_partitioned_fallbacks_large_weights_and_overfull_partitions():
    """Phase B's shared-memory tables hold 8192 distinct keys and 32-bit counts; anything beyond must take the
    L2-scratch fallback (u64 counts, growing tables) and still be exact."""
    import torch
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(99)
    k = 21
    keys = rng.integers(0, 4**k, size=200_000, dtype=np.uint64)
    keys[:1000] = keys[0]  # one hot key
    weights = rng.integers(1, 5, size=len(keys), dtype=np.uint64)
    weights[:10] = np.uint64(2**33 + 7)  # does not fit 32 bits
    uk, inv = np.unique(keys, return_inverse=True)
    uc = np.zeros(len(uk), dtype=np.uint64)
    np.add.at(uc, inv, weights)
    tk = torch.from_numpy(keys.view(np.int64)).to(dev)
    tw = torch.from_numpy(weights.view(np.int64)).to(dev)
    torch.cuda.synchronize()
    for pl in (2, 6, 12):  # 4 partitions of 50 K keys overflow a shared-memory table; 4096 partitions do not
        with kb.GpuKmerCounter(k, flags=PART, parts_log2=pl) as c:
            c.insert_keys_device(tk.data_ptr(), len(keys), tw.data_ptr())
            s = c.finalize()
            assert_same(c.export(1, True), (uk, uc))
            assert s["n_windows"] == int(uc.sum()) and s["max_count"] == int(uc.max())


def test_input_outgrows_the_partition_plan():
    """The plan is made from the first call; when far more data follows, partitions hold many times what one shared-memory
    table takes.  Phase B must then count them in several passes (and still be exact), not fall off a cliff."""
    rng = np.random.default_rng(2024)
    k = 23
    small = [bytes(rng.choice(list(b"ACGT"), size=30_000).tolist())]
    big = [bytes(rng.choice(list(b"ACGT"), size=600_000).tolist()) for _ in range(4)]
    big.append(b"ACGTTGCAAT" * 40_000)  # plus a block of hot keys
    oracle = orc.count_records(k, small + big, mode="rolling")
    with kb.GpuKmerCounter(k, flags=PART) as c:   # ~9 partitions planned for 30 K windows, 2.8 M windows arrive
        for recs in (small, big):
            c.count_records(recs)
        s = c.finalize()
        keys, counts = c.export(1, True)
        assert s["path"] == 2
        assert_same((keys, counts, s), oracle)
        hv, hf = c.histogram(2)
        ov, of = orc.histogram(oracle[1], 2)
        assert (hv == ov).all() and (hf == of).all()


def test_small_start_migrates_from_the_table_to_the_partitioned_path():
    """A context whose first call is small starts on the single hash table; when the stream keeps growing it must move
    its contents to the partitioned pipeline (weighted run) without losing or double counting anything."""
    rng = np.random.default_rng(77)
    k = 25
    parts = [np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=30_000_000, dtype=np.uint8)] for _ in range(3)]
    parts[2][:5_000_000] = parts[0][:5_000_000]  # shared sequence: counts of 2 across the migration boundary
    with kb.GpuKmerCounter(k) as c:
        for p in parts:
            c.count_batch(p, None, np.array([0, len(p)], dtype=np.uint64))
        s = c.finalize()
        got = c.export(1, True)
        hist = c.histogram(1)
    assert s["path"] == 2 and s["n_windows"] == 3 * (30_000_000 - k + 1)
    seq = np.concatenate(parts)
    off = np.array([0, 30_000_000, 60_000_000, 90_000_000], dtype=np.uint64)
    with kb.GpuKmerCounter(k, flags=PART) as c:
        c.count_batch(seq, None, off)
        s2 = c.finalize()
        want = c.export(1, True)
        hist2 = c.histogram(1)
    assert s2["n_distinct"] == s["n_distinct"] and s2["max_count"] == s["max_count"]
    assert (got[0] == want[0]).all() and (got[1] == want[1]).all()
    assert (hist[0] == hist2[0]).all() and (hist[1] == hist2[1]).all()
    # and an oracle check on a slice of the key space: the 5 Mbp shared block alone
    ok, oc, _ = orc.count_batch(k, parts[0][:200_000], None, np.array([0, 200_000], dtype=np.uint64))
    idx = np.searchsorted(got[0], ok)
    assert (got[0][idx] == ok).all() and (got[1][idx] >= 2 * oc).all()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_exchange_shapes_on_one_device(world):
    """The bucket counts of the N-GPU exchange (world x P1 global coarse bins: ~1300, ~1850 and > 2048, which takes the
    staged scatter kernel instead of the rows kernel) exercised on ONE device: extract into world x P1 bins, then every
    'rank' adopts its P1 bins from every source and the union of the shard tables must equal the oracle count."""
    import torch
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(40 + world)
    k = 21
    host = rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8), p=[.248, .248, .248, .248, .008], size=3_000_000).astype(np.uint8)
    offsets_np = np.array([0, 1_200_000, len(host)], dtype=np.uint64)
    oracle = orc.count_batch(k, host, None, offsets_np, mode="rolling")
    seq = torch.from_numpy(host).to(dev)
    offsets = torch.from_numpy(offsets_np.astype(np.int64)).to(dev)
    p1 = {2: 657, 4: 464, 8: 328}[world]   # what the plan gives for C4 split over `world` ranks
    shards = []
    for r in range(world):
        c = kb.GpuKmerCounter(k, flags=PART, expected_distinct=p1 * p1 * 3600)
        assert c.partition_plan(p1 * p1 * 3600)[0] == p1
        shards.append(c)
    try:
        out = torch.empty(len(host), dtype=torch.int64, device=dev)
        counts = shards[0].extract_keys_device(seq.data_ptr(), len(host), world * p1, out.data_ptr(), len(host),
                                               d_offsets=offsets.data_ptr(), n_records=2)
        assert int(counts.sum()) == oracle[2]
        bounds = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        got_k, got_c = [], []
        for r in range(world):
            lo, hi = bounds[r * p1], bounds[(r + 1) * p1]
            block = out[lo:hi]
            if hi > lo:
                shards[r].adopt_coarse_device(block.data_ptr(), counts[r * p1:(r + 1) * p1].astype(np.uint64), int(hi - lo))
            shards[r].finalize()
            kk, cc = shards[r].export(1, True)
            assert all(kb.owner_of(int(x), world) == r for x in kk[:200])
            got_k.append(kk); got_c.append(cc)
        allk = np.concatenate(got_k); allc = np.concatenate(got_c)
        order = np.argsort(allk, kind="stable")
        assert_same((allk[order], allc[order]), oracle)
    finally:
        for c in shards:
            c.close()


@pytest.mark.parametrize("shape", ["distinct", "repeats", "triple", "few_partitions", "small", "exact_layout", "exact_layout_one_run"])
def test_phase_b_sieve_variants(shape):
    """Phase B's sieve (bit map + small side table, TMA-staged keys copied in place) on inputs it takes whole, inputs with a
    repeat fraction its side table still holds, and inputs it must hand to the compacting variant (every key repeated; partitions
    larger than a batch) -- several runs per partition (three calls).  "exact_layout": ~30 keys per partition and run, too few
    for the speculative level-2 layout, so the sieve reads raw runs in the exact layout (three runs; "exact_layout_one_run": the
    first call alone, one run, which is copied rather than counted in place)."""
    rng = np.random.default_rng(4242)
    k = 21
    n = 100_000 if shape == "small" else 2_000_000   # "small": the same kernels at a size compute-sanitizer's racecheck finishes (tools/sanitize.sh)
    g = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=3 * n, dtype=np.uint8)].copy()
    if shape == "small":
        g[250_000:255_000] = g[10_000:15_000]
    if shape == "repeats":  # ~30 % of the sequence are second copies of earlier 5 kbp blocks
        for _ in range(180):
            a, b = (int(x) for x in rng.integers(0, 3 * n - 5000, size=2))
            g[b:b + 5000] = g[a:a + 5000]
    if shape == "triple":
        g[n:2 * n] = g[:n]
        g[2 * n:] = g[:n]
    n_calls = 1 if shape == "exact_layout_one_run" else 3
    g = g[:n_calls * n]
    chunks = [g[i * n:(i + 1) * n] for i in range(n_calls)]
    kw = dict(flags=PART, expected_distinct=3 * n)
    if shape == "few_partitions":
        kw = dict(flags=PART, parts_log2=6)   # 64 partitions of ~94 K entries: beyond a batch, beyond one table
    if shape.startswith("exact_layout"):
        kw = dict(flags=PART, parts_log2=16)
    with kb.GpuKmerCounter(k, **kw) as c:
        for ch in chunks:
            c.count_batch(ch, None, np.array([0, len(ch)], dtype=np.uint64))
        s = c.finalize()
        got = c.export(1, True)
        hv, hf = c.histogram(1)
    ok, oc, _ = orc.count_batch(k, g, None, np.arange(n_calls + 1, dtype=np.uint64) * n)   # the calls are records
    assert s["path"] == 2 and s["n_windows"] == n_calls * (n - k + 1) and s["n_distinct"] == len(ok)
    assert_same(got, (ok, oc))
    ov, of = orc.histogram(oc, 1)
    assert (hv == ov).all() and (hf == of).all()


def test_c4_bin_geometry_on_100mbp():
    """The bin counts of the full C4 job (~1000 x 1000: rows of 16 slots, eight lanes per row in the copy-out of both scatter
    levels, speculative layouts, sieve in place) on an input the oracle counts in seconds: 100 Mbp with
    2^20 partitions, the whole table and the histogram against the oracle; then a second, overlapping call (the first result
    re-enters phase B as a weighted run)."""
    import torch
    dev = torch.device("cuda:0")
    k, n, n_rec = 21, 100_000_000, 10
    buf = torch.empty(n, dtype=torch.uint8, device=dev)
    offsets = torch.arange(0, n + 1, n // n_rec, dtype=torch.int64, device=dev)
    host = orc.synth_uniform(4242, 0, n)
    off_np = np.arange(0, n + 1, n // n_rec, dtype=np.uint64)
    with kb.GpuKmerCounter(k, flags=PART, parts_log2=20) as c:
        c.synth_uniform_device(4242, 0, n, buf.data_ptr())
        c.count_device(buf.data_ptr(), n, d_offsets=offsets.data_ptr(), n_records=n_rec)
        s = c.finalize()
        got = c.export(1, True)
        okeys, ocounts, owin = orc.count_batch_mt(k, host, None, off_np)
        assert s["path"] == 2 and owin == s["n_windows"] and s["n_distinct"] == len(okeys)
        assert_same(got, (okeys, ocounts))
        hv, hf = c.histogram(1)
        ov, of = orc.histogram(ocounts, 1)
        assert (hv == ov).all() and (hf == of).all()
        # the first 30 Mbp (3 records) once more
        m = 3 * (n // n_rec)
        c.count_device(buf.data_ptr(), m, d_offsets=offsets.data_ptr(), n_records=3)
        c.finalize()
        got2 = c.export(1, True)
        k2, c2, _ = orc.count_batch_mt(k, host[:m], None, off_np[:4])
        idx = np.searchsorted(okeys, k2)
        want = ocounts.copy()
        want[idx] += c2
        assert_same(got2, (okeys, want))


@pytest.mark.parametrize("size", ["full", "small"])
def test_c4_bin_geometry_on_skewed_input(size):
    """The C4 bin counts (2^10 x 2^10: rows of 16 / 27 slots, the scatter kernels partition_scatter_rows2 / refine_rows4) on an input
    whose sub-tiles overflow their rows in every way: blocks copied many times (a few overflow keys per sub-tile: the overflow
    lists), a 40-base satellite and poly-A stretches (thousands of equal keys per sub-tile: the per-sub-tile exact route, then the
    job-wide exact layout once a partition outgrows its speculative share), N runs.  "small": the same at a size compute-sanitizer
    finishes (tools/sanitize.sh)."""
    rng = np.random.default_rng(777)
    k = 21
    n = 24_000_000 if size == "full" else 800_000
    u = n // 24   # unit: the features below are placed in 24ths of the input
    g = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=n, dtype=np.uint8)].copy()
    block = g[1000:1600].copy()
    for pos in range(2 * u, 8 * u, 9_000):            # 600-base block every 9 kbp
        g[pos:pos + 600] = block
    sat = g[5000:5040].copy()
    g[9 * u:10 * u] = np.tile(sat, u // 40 + 1)[:u]   # satellite
    g[12 * u:13 * u + u // 2] = ord("A")              # poly-A
    g[15 * u:15 * u + (2 * u) // 5] = ord("T")        # its reverse complement: the same canonical key
    for pos in rng.integers(0, n - 10, size=300 if size == "full" else 30):
        g[pos:pos + 10] = ord("N")
    cut = 12 * u + (7 * u) // 10
    off_np = np.array([0, 5 * u, cut, n], dtype=np.uint64)
    okeys, ocounts, owin = orc.count_batch_mt(k, g, None, off_np)
    ov, of = orc.histogram(ocounts, 1)
    for parts_log2 in (20, 19):   # 1024 x 1024 and 512 x 1024 bins
        with kb.GpuKmerCounter(k, flags=PART, parts_log2=parts_log2) as c:
            c.count_batch(g[:cut], None, off_np[:3])
            c.count_batch(g[cut:], None, np.array([0, n - cut], dtype=np.uint64))
            s = c.finalize()
            got = c.export(1, True)
            hv, hf = c.histogram(1)
        assert s["path"] == 2 and s["n_windows"] == owin and s["n_distinct"] == len(okeys)
        assert_same(got, (okeys, ocounts))
        assert (hv == ov).all() and (hf == of).all()
