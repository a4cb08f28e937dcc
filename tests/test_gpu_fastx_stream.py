"""kmg_fastx_stream_*: FASTA / FASTQ byte streams parsed on the device, pushed in pieces of any size, against the oracle's
bio-compatible record parser + counter and against kmg_count_fastx on the whole image.  Small staging chunks (batch_bases 4096)
make slot cuts and tail moves happen every few pushes; unwrapped FASTA lines are cut inside the line; refused FASTQ falls back to
the host splitter through kmg_fastx_stream_rest; the CLI and the Python front ends stream stdin and .gz files."""
import ctypes as C
import gzip
import os
import subprocess
import threading
import time

import numpy as np
import pytest

import krust_b200 as kb
from krust_b200 import _lib
from oracle import oracle as orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FX = os.path.join(ROOT, "tests", "golden", "fixtures")
BIN = os.path.join(ROOT, "krust_b200", "host", "kmerust-b200")
OK, PARSE, STATE = _lib.KMG_OK, _lib.KMG_ERR_PARSE, _lib.KMG_ERR_STATE


# ----------------------------------------------------------------------------- fixtures and helpers
def fasta_image(rng, n_rec, width, eol=b"\n", trailing_blank=False, final_newline=True, blank_lines=False, max_len=3000):
    out = []
    for r in range(n_rec):
        n = int(rng.integers(0, max_len))
        seq = bytes(rng.choice(list(b"ACGTacgtNn"), p=[.2, .2, .2, .2, .04, .04, .04, .04, .02, .02], size=n).tolist())
        out.append(b">rec%d some description" % r + eol)
        for i in range(0, n, width):
            out.append(seq[i:i + width] + (b"  \t" if trailing_blank and i % (3 * width) == 0 else b"") + eol)
            if blank_lines and i % (7 * width) == 0:
                out.append(eol)
    data = b"".join(out)
    return data if final_newline else data.rstrip(b"\r\n")


def fastq_image(n_reads, seed=43, at_quals=True, eol=b"\n"):
    seq, qual, off = orc.synth_reads(seed, 3, 0, n_reads)
    s2, q2 = seq.reshape(n_reads, 150), qual.reshape(n_reads, 150).copy()
    if at_quals:
        q2[::5, 0] = ord("@")  # quality lines that look like headers
    return b"".join(b"@read%d/1" % i + eol + s2[i].tobytes() + eol + b"+" + eol + q2[i].tobytes() + eol for i in range(n_reads))


def oracle_counts(data, is_fastq, k, q=None):
    seq, qual, offsets = orc.parse_fastx(data, is_fastq)
    keys, counts, windows = orc.count_batch(k, seq, qual, offsets, q, mode="rolling")
    return dict(keys=keys, counts=counts, windows=windows, records=len(offsets) - 1, bases=int(offsets[-1]))


def pieces(data, how, rng=None):
    if how == "whole":
        return [data]
    if how == "random":
        cuts = np.sort(rng.integers(0, len(data) + 1, size=max(1, len(data) // 1500)))
        return [data[a:b] for a, b in zip([0, *cuts.tolist()], [*cuts.tolist(), len(data)])]
    return [data[i:i + how] for i in range(0, len(data), how)]


def results(c):
    s = c.finalize()
    keys, counts = c.export(1, True)
    hv, hf = c.histogram(1)
    return dict(summary=s, keys=keys, counts=counts, hv=hv, hf=hf)


def push_all(c, chunks, is_fastq, hint=0):
    L, ctx = c._L, c._ctx
    assert L.kmg_fastx_stream_begin(ctx, int(is_fastq), hint) == OK
    for p in chunks:
        buf = np.frombuffer(p, dtype=np.uint8) if p else np.zeros(1, dtype=np.uint8)
        st = L.kmg_fastx_stream_push(ctx, buf.ctypes.data, len(p))
        assert st == OK, L.kmg_last_error(ctx)
    n = C.c_uint64(0)
    st = L.kmg_fastx_stream_end(ctx, C.byref(n))
    assert st == OK, L.kmg_last_error(ctx)
    return n.value


def stream_counts(data, is_fastq, k, q=None, how="whole", batch_bases=4096, rng=None, hint=0):
    with kb.GpuKmerCounter(k, min_quality=q, batch_bases=batch_bases) as c:
        n = push_all(c, pieces(data, how, rng), is_fastq, hint)
        r = results(c)
    r["n"] = n
    return r


def image_counts(data, is_fastq, k, q=None, batch_bases=0):
    with kb.GpuKmerCounter(k, min_quality=q, batch_bases=batch_bases) as c:
        n = c.count_fastx(data, is_fastq)
        r = results(c)
    r["n"] = n
    return r


def same_as_oracle(r, o):
    assert len(r["keys"]) == len(o["keys"]) and (r["keys"] == o["keys"]).all() and (r["counts"] == o["counts"]).all()
    s = r["summary"]
    assert s["n_windows"] == o["windows"] and s["n_records"] == o["records"] and s["n_bases"] == o["bases"]
    if "n" in r:
        assert r["n"] == o["records"]
    hv, hf = orc.histogram(o["counts"], 1) if len(o["counts"]) else (np.zeros(0), np.zeros(0))
    assert (r["hv"] == hv).all() and (r["hf"] == hf).all()


def same_as_image(r, i):
    assert (r["keys"] == i["keys"]).all() and (r["counts"] == i["counts"]).all() and (r["hv"] == i["hv"]).all() and (r["hf"] == i["hf"]).all()
    for f in ("n_records", "n_bases", "n_windows", "n_distinct"):
        assert r["summary"][f] == i["summary"][f]
    assert r["n"] == i["n"]


# ----------------------------------------------------------------------------- 1. splits
def test_fixture_images_in_every_split():
    rng = np.random.default_rng(1)
    for name, is_fastq in (("simple.fa", False), ("simple.fq", True), ("with_n.fa", False), ("with_n.fq", True), ("soft_masked.fa", False),
                           ("low_quality.fq", True)):
        data = open(os.path.join(FX, name), "rb").read()
        for k in (1, 3, 21):
            for q in ((None, 20) if is_fastq else (None,)):
                o = oracle_counts(data, is_fastq, k, q)
                for how in ("whole", 1, 7, 4096, "random"):
                    same_as_oracle(stream_counts(data, is_fastq, k, q, how, rng=rng), o)


@pytest.mark.parametrize("k", [1, 3, 21, 31, 32])
def test_generated_fasta_variants_in_pieces(k):
    rng = np.random.default_rng(k)
    for width, eol, tb, fn, bl in ((80, b"\n", False, True, False), (60, b"\r\n", True, True, True), (100, b"\n", True, False, False),
                                   (7, b"\n", False, True, True)):
        data = fasta_image(rng, 25, width, eol, tb, fn, bl)
        o = oracle_counts(data, False, k)
        img = image_counts(data, False, k, batch_bases=4096)
        for how in ("whole", 7, 4096, "random"):
            r = stream_counts(data, False, k, how=how, rng=rng)
            same_as_oracle(r, o)
            same_as_image(r, img)
    small = fasta_image(rng, 6, 13, b"\r\n", True, False, True, max_len=60)
    same_as_oracle(stream_counts(small, False, k, how=1), oracle_counts(small, False, k))


@pytest.mark.parametrize("k,q", [(1, None), (3, 20), (21, None), (31, 20), (32, 20)])
def test_fastq_with_at_leading_quality_lines_in_pieces(k, q):
    rng = np.random.default_rng(k)
    data = fastq_image(300)
    assert b"\n@" in data.replace(b"\n@read", b"")
    o = oracle_counts(data, True, k, q)
    img = image_counts(data, True, k, q, batch_bases=4096)
    for how in ("whole", 7, 4096, "random"):
        r = stream_counts(data, True, k, q, how=how, rng=rng)
        same_as_oracle(r, o)
        same_as_image(r, img)
    crlf = fastq_image(40, seed=7, eol=b"\r\n")
    same_as_oracle(stream_counts(crlf, True, k, q, how=1), oracle_counts(crlf, True, k, q))


def test_two_pushes_split_at_every_offset():
    rng = np.random.default_rng(5)
    fa = fasta_image(rng, 4, 11, b"\r\n", True, False, True, max_len=60)
    fq = fastq_image(2, seed=3)[:-1]  # no final newline
    for data, is_fastq, k in ((fa, False, 5), (fq, True, 7)):
        o = oracle_counts(data, is_fastq, k)
        with kb.GpuKmerCounter(k) as c:
            for cut in range(len(data) + 1):
                c.reset()
                n = push_all(c, [data[:cut], data[cut:]], is_fastq)
                same_as_oracle(dict(results(c), n=n), o)


def test_small_staging_slots_with_size_hint_and_partitioned_path():
    rng = np.random.default_rng(9)
    data = fasta_image(rng, 200, 70, max_len=20_000)
    o = oracle_counts(data, False, 21)
    same_as_oracle(stream_counts(data, False, 21, how=65536, batch_bases=0, hint=len(data)), o)
    with kb.GpuKmerCounter(21, batch_bases=1 << 16, flags=_lib.KMG_FLAG_FORCE_PARTITIONED, parts_log2=4) as c:
        n = push_all(c, pieces(data, 10_000), False)
        same_as_oracle(dict(results(c), n=n), o)


# ----------------------------------------------------------------------------- 2. FASTA lines longer than a chunk
def test_unwrapped_fasta_lines_longer_than_a_chunk():
    rng = np.random.default_rng(11)
    line = bytearray(rng.choice(list(b"ACGTN"), p=[.24, .24, .24, .24, .04], size=40_000).tolist())
    for pos, junk in ((3000, b" "), (5000, b"\t\t"), (7000, b"\r"), (9000, b">"), (12000, b"> >"), (15000, b"NNNN")):
        line[pos:pos + len(junk)] = junk
    line[20_000:23_000] = b"A " * 1500          # no valid cut for 3000 bytes
    line[30_000:31_000] = b">A" * 500           # cuts only after a '>'
    recs = [b">one\n" + bytes(line) + b"\n", b">two\n" + bytes(line[::-1]) + b"\n", b">three\n" + bytes(line[:9000]),
            b">four\n" + bytes(line[1000:5000]) + b"\nACGT\n"]
    data = b"".join(recs)
    for k in (1, 3, 21, 32):
        o = oracle_counts(data, False, k)
        for how in ("whole", 1000, "random"):
            same_as_oracle(stream_counts(data, False, k, how=how, rng=rng), o)
    with pytest.raises(kb.SequenceParseError):
        image_counts(data, False, 21, batch_bases=4096)   # the file-image call keeps refusing them


def test_header_longer_than_a_chunk_is_refused_and_falls_back():
    data = b">" + b"h" * 10_000 + b"\nACGTACGTTT\n>b\nGGGACC\n"
    o = oracle_counts(data, False, 3)
    got = fallback_count(data, False, 3, 1000)
    same_as_oracle(got, o)
    assert got["refused_at"] == 0


# ----------------------------------------------------------------------------- 3. fallback through rest
def fallback_count(data, is_fastq, k, piece, q=None, batch_bases=4096):
    """Push in pieces; on KMG_ERR_PARSE take the rest + the pieces not pushed through the host splitter into kmg_count_ascii."""
    with kb.GpuKmerCounter(k, min_quality=q, batch_bases=batch_bases) as c:
        L, ctx = c._L, c._ctx
        assert L.kmg_fastx_stream_begin(ctx, int(is_fastq), 0) == OK
        parts = pieces(data, piece)
        st, i, refused_at = OK, 0, None
        for i, p in enumerate(parts):
            buf = np.frombuffer(p, dtype=np.uint8)
            st = L.kmg_fastx_stream_push(ctx, buf.ctypes.data, len(p))
            if st != OK:
                break
        if st == OK:
            st = L.kmg_fastx_stream_end(ctx, C.byref(C.c_uint64(0)))
            i = len(parts)
        if st != OK:
            assert st == PARSE, L.kmg_last_error(ctx)
            n = C.c_uint64(0)
            assert L.kmg_fastx_stream_rest(ctx, None, 0, C.byref(n)) == OK
            rest = np.zeros(max(n.value, 1), dtype=np.uint8)
            assert L.kmg_fastx_stream_rest(ctx, rest.ctypes.data, n.value, C.byref(n)) == OK
            tail = rest[:n.value].tobytes() + b"".join(parts[i + 1:])
            refused_at = len(data) - len(tail)
            assert data.endswith(tail)
            seq, qual, offsets = kb.parse_fastx(tail, is_fastq)
            c.count_batch(seq, qual, offsets)
        r = results(c)
    r["refused_at"] = refused_at
    return r


def test_multiline_fastq_falls_back_in_the_first_and_in_a_later_chunk():
    good = fastq_image(120, seed=17)
    ml = b"@ml1\nACGTAC\nGTACGT\n+\nIIIIII\nIIII!!\n@ml2\nGATTACA\n+\nIIIIIII\n"
    for data in (ml + good, good + ml + good):
        for q in (None, 20):
            o = oracle_counts(data, True, 4, q)
            for piece in (1000, 4096, 100_000):
                got = fallback_count(data, True, 4, piece, q)
                same_as_oracle(got, o)
                assert got["refused_at"] is not None
                if data.startswith(ml):
                    assert got["refused_at"] == 0
                else:
                    assert 0 < got["refused_at"] <= len(good)   # the earlier chunks were counted on the device


def test_missing_header_at_byte_zero():
    with kb.GpuKmerCounter(3) as c:
        L, ctx = c._L, c._ctx
        for is_fastq, data in ((False, b"ACGT\n>x\nAC\n"), (True, b"ACGT\n+\nIIII\n")):
            assert L.kmg_fastx_stream_begin(ctx, int(is_fastq), 0) == OK
            buf = np.frombuffer(data, dtype=np.uint8)
            assert L.kmg_fastx_stream_push(ctx, buf.ctypes.data, len(data)) == PARSE
            n = C.c_uint64(0)
            assert L.kmg_fastx_stream_rest(ctx, None, 0, C.byref(n)) == OK and n.value == len(data)
            rest = np.zeros(len(data), dtype=np.uint8)
            assert L.kmg_fastx_stream_rest(ctx, rest.ctypes.data, 2, C.byref(n)) == _lib.KMG_ERR_CAPACITY
            assert L.kmg_fastx_stream_rest(ctx, rest.ctypes.data, len(data), C.byref(n)) == OK and rest.tobytes() == data
            with pytest.raises(kb.SequenceParseError):
                kb.parse_fastx(data, is_fastq)   # the host splitter refuses it too
        assert c.finalize()["n_windows"] == 0


# ----------------------------------------------------------------------------- 4. final errors and states
def test_quality_length_mismatch_is_final():
    data = fastq_image(50) + b"@bad\nACGTACGT\n+\nIII\n" + fastq_image(50, seed=2)
    with kb.GpuKmerCounter(21, batch_bases=4096) as c:
        L, ctx = c._L, c._ctx
        assert L.kmg_fastx_stream_begin(ctx, 1, 0) == OK
        buf = np.frombuffer(data, dtype=np.uint8)
        st = L.kmg_fastx_stream_push(ctx, buf.ctypes.data, len(data))
        if st == OK:
            st = L.kmg_fastx_stream_end(ctx, C.byref(C.c_uint64(0)))
        assert st == PARSE and b"quality" in L.kmg_last_error(ctx)
        assert L.kmg_fastx_stream_rest(ctx, None, 0, C.byref(C.c_uint64(0))) == STATE
        with pytest.raises(kb.SequenceParseError):
            kb.parse_fastx(data, True)
        c.reset()
        good = fastq_image(30)
        n = push_all(c, pieces(good, 999), True)
        same_as_oracle(dict(results(c), n=n), oracle_counts(good, True, 21))


def test_every_other_call_waits_for_an_open_stream():
    data = fastq_image(200)
    o = oracle_counts(data, True, 5)
    with kb.GpuKmerCounter(5, batch_bases=4096) as c:
        L, ctx = c._L, c._ctx
        assert L.kmg_fastx_stream_begin(ctx, 1, 0) == OK
        assert L.kmg_fastx_stream_begin(ctx, 1, 0) == STATE
        buf = np.frombuffer(data, dtype=np.uint8)
        assert L.kmg_fastx_stream_push(ctx, buf.ctypes.data, 5000) == OK
        r0, _ = c.progress()
        assert L.kmg_fastx_stream_push(ctx, buf[5000:].ctypes.data, len(data) - 5000) == OK
        r1, b1 = c.progress()
        assert r0 <= r1 and 0 < r1 < 200 and b1 > 0                   # progress advances per counted chunk
        seq = np.frombuffer(b"ACGTACGT", dtype=np.uint8)
        off = np.array([0, 8], dtype=np.uint64)
        u64 = C.c_uint64(0)
        keys = np.zeros(4, dtype=np.uint64)
        summ = _lib.KmgSummary()
        b = _lib.KmgBatch()
        for st in (L.kmg_count_ascii(ctx, seq.ctypes.data, None, off.ctypes.data, 1),
                   L.kmg_count_fastx(ctx, buf.ctypes.data, len(data), 1, C.byref(u64)),
                   L.kmg_acquire_batch(ctx, C.byref(b)),
                   L.kmg_finalize(ctx, C.byref(summ)),
                   L.kmg_export_counts(ctx, 1, 1, None, None, 0, C.byref(u64)),
                   L.kmg_export_shard(ctx, 1, 1, 2, 0, None, None, 0, C.byref(u64)),
                   L.kmg_histogram(ctx, 1, None, None, 0, C.byref(u64)),
                   L.kmg_write_text(ctx, 1, _lib.KMG_TEXT_TSV, b"/dev/null", C.byref(u64), C.byref(u64)),
                   L.kmg_save_kmix(ctx, b"/dev/null"),
                   L.kmg_query_keys(ctx, keys.ctypes.data, 4, keys.ctypes.data)):
            assert st == STATE
        n = C.c_uint64(0)
        assert L.kmg_fastx_stream_end(ctx, C.byref(n)) == OK and n.value == 200
        assert L.kmg_fastx_stream_end(ctx, None) == STATE
        same_as_oracle(dict(results(c), n=n.value), o)
        assert c.progress() == (200, o["bases"])


def test_reset_and_destroy_mid_stream_empty_stream_and_grouped_context():
    data = fasta_image(np.random.default_rng(2), 30, 60)
    o = oracle_counts(data, False, 21)
    with kb.GpuKmerCounter(21, batch_bases=4096) as c:
        L, ctx = c._L, c._ctx
        assert L.kmg_fastx_stream_begin(ctx, 0, 0) == OK
        buf = np.frombuffer(data, dtype=np.uint8)
        assert L.kmg_fastx_stream_push(ctx, buf.ctypes.data, len(data) // 2) == OK
        c.reset()                                                         # abandons the stream
        assert L.kmg_fastx_stream_push(ctx, buf.ctypes.data, 10) == STATE
        n = push_all(c, pieces(data, 3333), False)
        same_as_oracle(dict(results(c), n=n), o)
        c.reset()
        assert push_all(c, [], False) == 0 and c.finalize()["n_windows"] == 0   # an empty stream
    c = kb.GpuKmerCounter(21, batch_bases=4096)
    assert c._L.kmg_fastx_stream_begin(c._ctx, 0, 0) == OK
    assert c._L.kmg_fastx_stream_push(c._ctx, buf.ctypes.data, len(data) - 100) == OK
    t0 = time.time()
    c.close()                                                             # destroy with a stream open
    assert time.time() - t0 < 30
    group = f"st{os.getpid()}-{time.time_ns() & 0xffffff:x}"
    got = [None, None]

    def rank(r):
        g = kb.GpuKmerCounter(21)
        try:
            g.shard_join(2, r, group, 1 << 20)
            got[r] = g._L.kmg_fastx_stream_begin(g._ctx, 0, 0)
        finally:
            g.shard_leave()
            g.close()
    ts = [threading.Thread(target=rank, args=(r,)) for r in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert got == [STATE, STATE]


# ----------------------------------------------------------------------------- 5. scale and memory
def test_c1_streamed_in_64_mib_pushes():
    n, n_rec, k = 100_000_000, 100, 21
    host = orc.synth_uniform(42, 0, n)
    rec = n // n_rec
    body = host.reshape(n_rec, rec // 80, 80)
    lines = np.concatenate([body, np.full((n_rec, rec // 80, 1), 10, dtype=np.uint8)], axis=2).reshape(n_rec, -1)
    data = b"".join(b">c1_%d\n" % r + lines[r].tobytes() for r in range(n_rec))
    okeys, ocounts, owin = orc.count_batch_mt(k, host, None, np.arange(0, n + 1, rec, dtype=np.uint64))
    with kb.GpuKmerCounter(k) as c:
        got = push_all(c, pieces(data, 64 << 20), False)
        r = results(c)
    assert got == n_rec and r["summary"]["n_windows"] == owin and r["summary"]["n_bases"] == n
    assert len(r["keys"]) == len(okeys) and (r["keys"] == okeys).all() and (r["counts"] == ocounts).all()
    hv, hf = orc.histogram(ocounts, 1)
    assert (r["hv"] == hv).all() and (r["hf"] == hf).all()


def test_cli_stdin_of_a_4_gib_fasta_in_bounded_memory(tmp_path):
    """A 4.3 GB FASTA generated by a child process and piped into the CLI's stdin: the CLI's peak RSS (getrusage of a wrapper's
    children) stays far below the input; the windows total (-f histogram) and a sample of the key space (the k-mers of a -m 2 tsv
    run with key % 1009 == 3) equal the oracle's."""
    import psutil
    if psutil.virtual_memory().available < 24e9:
        pytest.skip("the oracle needs ~10 GB of host memory for the 4.3 Gbp stream")
    n_rec, rec, k = 43, 100_000_000, 21
    gen = (
        "import sys, numpy as np\n"
        f"sys.path.insert(0, {ROOT!r})\n"
        "from oracle import oracle as orc\n"
        "out = sys.stdout.buffer\n"
        f"for r in range({n_rec}):\n"
        f"    b = orc.synth_uniform(45, r * {rec}, {rec}).reshape(-1, 80)\n"
        "    out.write(b'>s%d\\n' % r)\n"
        "    out.write(np.concatenate([b, np.full((len(b), 1), 10, dtype=np.uint8)], axis=1).tobytes())\n")
    wrap = ("import resource, subprocess, sys\n"
            "r = subprocess.run(sys.argv[1:])\n"
            "sys.stderr.write('RSS %d\\n' % resource.getrusage(resource.RUSAGE_CHILDREN).ru_maxrss)\n"
            "sys.exit(r.returncode)\n")

    def cli(args, out_path):
        g = subprocess.Popen(["python", "-c", gen], stdout=subprocess.PIPE)
        with open(out_path, "wb") as out:
            r = subprocess.run(["python", "-c", wrap, BIN, str(k), "-", "-q", *args], stdin=g.stdout, stdout=out, stderr=subprocess.PIPE,
                               timeout=1800)
        g.stdout.close()
        assert g.wait() == 0 and r.returncode == 0, r.stderr
        peak = int(r.stderr.splitlines()[-1].split()[1]) * 1024
        assert peak < 2 << 30, f"peak RSS {peak / 2**30:.2f} GiB for a {n_rec * rec / 2**30:.1f} GiB input"
        return open(out_path, "rb").read()

    n = n_rec * rec
    hist = np.array([[int(x) for x in ln.split(b"\t")] for ln in cli(["-f", "histogram"], tmp_path / "h.txt").splitlines()], dtype=np.uint64)
    assert int((hist[:, 0] * hist[:, 1]).sum()) == n - n_rec * (k - 1)
    tsv = cli(["-f", "tsv", "-m", "2"], tmp_path / "m2.tsv").splitlines()
    kmers = np.frombuffer(b"".join(ln[:k] for ln in tsv), dtype=np.uint8).reshape(-1, k)
    codes = ((kmers >> 1) ^ (kmers >> 2)) & 3      # A C G T -> 0 1 2 3
    keys = np.zeros(len(kmers), dtype=np.uint64)
    for j in range(k):
        keys = (keys << np.uint64(2)) | codes[:, j].astype(np.uint64)
    counts = np.array([int(ln[k + 1:]) for ln in tsv], dtype=np.uint64)
    assert int(counts.sum()) == int((hist[:, 0] * hist[:, 1])[hist[:, 0] >= 2].sum())
    sel = keys % np.uint64(1009) == np.uint64(3)
    host = orc.synth_uniform(45, 0, n)
    okeys, ocounts, owin = orc.count_batch_mt(k, host, None, np.arange(0, n + 1, rec, dtype=np.uint64), filter_mod=1009, filter_rem=3)
    del host
    assert owin == n - n_rec * (k - 1)
    keep = ocounts >= 2
    assert (keys[sel] == okeys[keep]).all() and (counts[sel] == ocounts[keep]).all() and sel.sum() == keep.sum() > 0
    hv, hf = np.unique(ocounts, return_counts=True)
    for v, f in zip(hv.tolist(), hf.tolist()):   # the sample's share of the count-of-counts is consistent with the whole
        exp = float(hist[hist[:, 0] == v, 1].sum()) / 1009
        assert abs(f - exp) < 6 * exp ** 0.5 + 10


# ----------------------------------------------------------------------------- 6. front ends
def test_cli_and_kmer_counter_on_stdin_and_gz_equal_the_file_path(tmp_path):
    rng = np.random.default_rng(21)
    cases = [("g.fa", fasta_image(rng, 60, 70, max_len=20_000)), ("r.fq", fastq_image(500)),
             ("ml.fq", fastq_image(200) + b"@ml\nACGTAC\nGTACGT\n+\nIIIIII\nIIII!!\n" + fastq_image(10, seed=5))]
    for name, data in cases:
        p = tmp_path / name
        p.write_bytes(data)
        gz = tmp_path / (name + ".gz")
        gz.write_bytes(gzip.compress(data))
        fmt = "fastq" if name.endswith(".fq") else "fasta"
        for args in (["-f", "tsv"], ["-f", "histogram"], ["-f", "tsv", "-Q", "20"]):
            want = subprocess.run([BIN, "21", str(p), "-q", *args], capture_output=True, timeout=300)
            assert want.returncode == 0 and want.stdout
            got_gz = subprocess.run([BIN, "21", str(gz), "-q", *args], capture_output=True, timeout=300)
            got_in = subprocess.run([BIN, "21", "-", "-q", "-i", fmt, *args], input=data, capture_output=True, timeout=300)
            with open(p, "rb") as f:   # stdin that is a regular file: its size is the hint
                got_file = subprocess.run([BIN, "21", "-", "-q", "-i", fmt, *args], stdin=f, capture_output=True, timeout=300)
            assert got_gz.stdout == want.stdout and got_in.stdout == want.stdout and got_file.stdout == want.stdout
        q = 20 if fmt == "fastq" else None
        want = kb.KmerCounter.new().k(21).min_quality(q).count_packed(p)
        got = kb.KmerCounter.new().k(21).min_quality(q).count_packed(gz)
        assert (got[0] == want[0]).all() and (got[1] == want[1]).all()
        code = ("import sys, numpy as np; sys.path.insert(0, %r); import krust_b200 as kb; "
                "k, c = kb.KmerCounter.new().k(21).input_format(%r).count_packed('-'); sys.stdout.buffer.write(k.tobytes() + c.tobytes())" % (ROOT, fmt))
        out = subprocess.run(["python", "-c", code], input=data, capture_output=True, timeout=300)
        assert out.returncode == 0, out.stderr
        want = kb.KmerCounter.new().k(21).count_packed(p)
        assert out.stdout == want[0].tobytes() + want[1].tobytes()
    bad = tmp_path / "bad.fq.gz"
    bad.write_bytes(gzip.compress(b"@r1\nACGT\n+\nIII\n"))
    r = subprocess.run([BIN, "3", str(bad), "-q"], capture_output=True, timeout=120)
    assert r.returncode == 1 and r.stderr.startswith(b"Application error:")
    with pytest.raises(kb.KmeRustError):
        kb.count_kmers(bad, 3)
