"""kmg_shard_count_fastx: one FASTA / FASTQ file image counted by a shard group, every rank parsing its own slice on the device.
Thread ranks on ONE device (as tests/test_gpu_shard_group.py), each case against the oracle (orc.parse_fastx + count_batch) AND
against one context's kmg_count_fastx: the union of the shards, disjoint shards, every window counted once at the rank cuts,
records / bases / histogram, the records of the whole image on every rank.  The cut-sweep test puts rank cuts on every kind of
line the carry rule has to handle; the error tests feed malformed input and check that no rank waits for the barrier timeout."""
import mmap
import os
import socket
import threading
import time

import numpy as np
import pytest

import krust_b200 as kb
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


def hint(data, is_fastq):
    return max(len(data) // 2 if is_fastq else len(data), 1)


def oracle_of(data: bytes, is_fastq: bool, k: int, q=None):
    seq, qual, offsets = orc.parse_fastx(data, is_fastq)
    keys, counts, windows = orc.count_batch_mt(k, seq, qual, offsets, q)
    return dict(keys=keys, counts=counts, windows=windows, records=len(offsets) - 1, bases=int(offsets[-1]))


def one_context(data: bytes, is_fastq: bool, k: int, q=None, batch_bases=0, text_path=None):
    with kb.GpuKmerCounter(k, min_quality=q, batch_bases=batch_bases) as c:
        n = c.count_fastx(data, is_fastq)
        s = c.finalize()
        keys, counts = c.export(1, True)
        hist = c.histogram(1)
        if text_path:
            c.write_text(text_path, "tsv", 1)
    return dict(n=n, summary=s, keys=keys, counts=counts, hist=hist)


def run_group(world, k, data, is_fastq, q=None, batch_bases=1 << 20, images=None, text_path=None, kmix_path=None):
    """Every rank joins, calls shard_count_fastx on the image (or on images[r]) and reads the group's results.
    Returns (per-rank results, per-rank exceptions, seconds)."""
    group = f"fx{os.getpid()}-{time.time_ns() & 0xffffff:x}"
    results, errors = [None] * world, [None] * world

    def worker(r):
        c = None
        try:
            c = kb.GpuKmerCounter(k, min_quality=q, batch_bases=batch_bases)
            c.shard_join(world, r, group, hint(data, is_fastq))
            n = c.shard_count_fastx(data if images is None else images[r], is_fastq)
            summary = c.shard_finalize()
            hist = c.shard_histogram(1)
            text = c.shard_write_text(text_path, "tsv", 1) if text_path else None
            n_kmix = c.shard_save_kmix(kmix_path) if kmix_path else None
            keys, counts = c.export(1, True)
            results[r] = dict(n=n, summary=summary, hist=hist, keys=keys, counts=counts, stats=c.shard_stats(), text=text, n_kmix=n_kmix)
        except Exception as e:  # noqa: BLE001
            errors[r] = e
        finally:
            if c is not None:
                try:
                    c.shard_leave()
                finally:
                    c.close()

    t0 = time.time()
    threads = [threading.Thread(target=worker, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout=300)
    assert not any(t.is_alive() for t in threads), "a rank hung"
    return results, errors, time.time() - t0


def check(results, errors, world, ora, single):
    assert not any(errors), errors
    allk = np.concatenate([r["keys"] for r in results]); allc = np.concatenate([r["counts"] for r in results])
    assert len(allk) == len(ora["keys"])                     # shards are disjoint: no key twice
    order = np.argsort(allk, kind="stable")
    assert (allk[order] == ora["keys"]).all() and (allc[order] == ora["counts"]).all()
    assert (single["keys"] == ora["keys"]).all() and (single["counts"] == ora["counts"]).all()
    ov, of = orc.histogram(ora["counts"], 1)
    for r, res in enumerate(results):
        s = res["summary"]
        assert s["n_windows"] == ora["windows"] == single["summary"]["n_windows"]
        assert s["n_distinct"] == len(ora["keys"]) and s["max_count"] == single["summary"]["max_count"]
        assert s["n_records"] == ora["records"] == single["summary"]["n_records"] and res["n"] == single["n"] == ora["records"]
        assert s["n_bases"] == ora["bases"] == single["summary"]["n_bases"]
        assert (res["hist"][0] == ov).all() and (res["hist"][1] == of).all()
        assert (single["hist"][0] == ov).all() and (single["hist"][1] == of).all()
        assert all(kb.owner_of(int(x), world) == r for x in res["keys"][:300])
    assert sum(r["stats"]["recv_keys"] for r in results) == ora["windows"]   # no window counted twice at a cut


def same_as_one_context(world, k, data, is_fastq, q=None, batch_bases=1 << 20):
    ora = oracle_of(data, is_fastq, k, q)
    single = one_context(data, is_fastq, k, q)
    results, errors, _ = run_group(world, k, data, is_fastq, q, batch_bases)
    check(results, errors, world, ora, single)
    return results


def _fasta_image(rng, n_rec, width, eol, trailing_blank=False, final_newline=True, blank_lines=False, max_len=5000):
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


VARIANTS = ((80, b"\n", False, True, False), (60, b"\r\n", True, True, True), (100, b"\n", True, False, False), (7, b"\n", False, True, True))


@pytest.mark.parametrize("world,k", [(2, 21), (3, 32), (4, 31), (8, 15)])
def test_multiline_fasta_variants(world, k):
    rng = np.random.default_rng(world * 100 + k)
    for width, eol, tb, fn, bl in VARIANTS:
        data = _fasta_image(rng, 40, width, eol, tb, fn, bl)
        same_as_one_context(world, k, data, False)
        # small chunks: several rounds per rank, records spanning chunks and slices
        same_as_one_context(world, k, data, False, batch_bases=10_000)


# ---- every kind of rank cut ----------------------------------------------------------------------------------------------
def _short_records_image(rng, pad):
    """Many records of 0-40 bases (often 1, 2, 8 or 15) on 7-base lines, some \\r\\n lines, blank lines and trailing blanks; the
    first header is padded by `pad` bytes so that the rank cuts move across the line structure."""
    out = [b">r0" + b"x" * pad + b"\n"]
    for r in range(200):
        if r:
            out.append(b">r%d\n" % r)
        n = int(rng.choice([1, 2, 8, 15])) if rng.random() < 0.4 else int(rng.integers(0, 41))
        seq = bytes(rng.choice(list(b"ACGTacgN"), size=n).tolist())
        for i in range(0, n, 7):
            eol = b"\r\n" if rng.random() < 0.3 else b"\n"
            out.append(seq[i:i + 7] + (b" \t" if rng.random() < 0.1 else b"") + eol)
            if rng.random() < 0.25:
                out.append(b"\r\n" if rng.random() < 0.5 else b"\n")
    return b"".join(out)


def _trimmed(line: bytes) -> bytes:
    return line.rstrip(b" \t\n\v\f\r")


def cut_kinds(data: bytes, world: int, k: int):
    """The rule of kmg_shard_count_fastx, in Python: where each rank cut falls and what kind of line structure it meets."""
    kinds = set()
    for r in range(1, world):
        t = len(data) * r // world
        p = t if t == 0 or t >= len(data) or data[t - 1] == 10 else data.find(b"\n", t) + 1 or len(data)
        if p >= len(data) or data[p] == ord(">"):
            continue
        ls_next = data.find(b"\n", p)
        line = data[p:(ls_next + 1 if ls_next >= 0 else len(data))]
        if _trimmed(line) == b"":
            kinds.add("blank line")
        if line.endswith(b"\r\n"):
            kinds.add("crlf line")
        # walk back to the record's header: bases since the header, lines the carry spans
        lines, le = [], p
        while le > 0:
            ls = data.rfind(b"\n", 0, le - 1) + 1
            if data[ls] == ord(">"):
                break
            lines.insert(0, _trimmed(data[ls:le]))
            le = ls
        before = b"".join(lines)
        if not lines:
            kinds.add("right after a header")
        elif len(before) < k - 1:
            kinds.add("fewer than k-1 bases since the header")
        carried, spanned = 0, 0
        for piece in reversed(lines):
            if carried >= k - 1:
                break
            if piece:
                spanned += 1
            carried += len(piece)
        if spanned >= 2:
            kinds.add("carry spans several lines")
        nxt = data.find(b"\n>", p)
        after = b"".join(_trimmed(x) for x in data[p:(nxt + 1 if nxt >= 0 else len(data))].split(b"\n"))
        if len(before) + len(after) < k:
            kinds.add("record shorter than k")
    return kinds


ALL_KINDS = {"right after a header", "fewer than k-1 bases since the header", "blank line", "crlf line", "record shorter than k",
             "carry spans several lines"}


@pytest.mark.parametrize("k", [21, 32, 3])
def test_every_kind_of_cut(k):
    seen = set()
    for pad in range(64):
        data = _short_records_image(np.random.default_rng(2), pad)
        ora = oracle_of(data, False, k)
        single = one_context(data, False, k)
        for world in (3, 8):
            seen |= cut_kinds(data, world, k)
            results, errors, _ = run_group(world, k, data, False, batch_bases=4096)
            check(results, errors, world, ora, single)
    assert seen == ALL_KINDS, ALL_KINDS - seen


def test_one_long_record_spans_all_ranks():
    rng = np.random.default_rng(3)
    seq = bytes(rng.choice(list(b"ACGTN"), p=[.24, .24, .24, .24, .04], size=1_500_000).tolist())
    data = b">chr1 long\n" + b"\n".join(seq[i:i + 80] for i in range(0, len(seq), 80)) + b"\n"
    for world, k in ((3, 31), (4, 21)):
        # unequal slices of whole lines: ranks make many rounds, not all the same number
        results = same_as_one_context(world, k, data, False, batch_bases=40_000)
        assert min(r["stats"]["rounds"] for r in results) >= 8


# ---- FASTQ -----------------------------------------------------------------------------------------------------------------
def _fastq_image(n_reads):
    seq, qual, off = orc.synth_reads(43, 3, 0, n_reads)
    n = len(off) - 1
    s2, q2 = seq.reshape(n, 150), qual.reshape(n, 150).copy()
    q2[::7, 0] = ord("@")      # every 7th quality line begins with '@': it looks like a header
    return b"".join(b"@read%d/1\n" % i + s2[i].tobytes() + b"\n+\n" + q2[i].tobytes() + b"\n" for i in range(n))


@pytest.mark.parametrize("world", [2, 4, 8])
def test_fastq_reads_with_qualities(world):
    data = _fastq_image(12_000)
    for q in (None, 2, 20):
        same_as_one_context(world, 31, data, True, q)
    same_as_one_context(world, 21, data, True, 20, batch_bases=100_000)   # many rounds per rank
    crlf = _fastq_image(4000).replace(b"\n", b"\r\n")
    same_as_one_context(world, 25, crlf, True, 20, batch_bases=70_001)


# ---- edge sizes, ungrouped context -----------------------------------------------------------------------------------------
def test_empty_image_fixtures_at_world_8_and_ungrouped(golden_dir):
    results, errors, _ = run_group(8, 21, b"", False)
    assert not any(errors), errors
    assert all(r["n"] == 0 and r["summary"]["n_windows"] == 0 and r["summary"]["n_records"] == 0 for r in results)
    fx = os.path.join(golden_dir, "fixtures")
    for name, is_fastq in (("simple.fa", False), ("simple.fq", True), ("with_n.fa", False), ("with_n.fq", True), ("soft_masked.fa", False),
                           ("low_quality.fq", True)):
        data = open(os.path.join(fx, name), "rb").read()
        for k in (3, 7):
            for q in ((None, 20) if is_fastq else (None,)):
                same_as_one_context(8, k, data, is_fastq, q)
    data = _fasta_image(np.random.default_rng(1), 30, 60, b"\n")
    single = one_context(data, False, 21)
    with kb.GpuKmerCounter(21) as c:      # outside a group the call is kmg_count_fastx
        assert c.shard_count_fastx(data, False) == single["n"]
        s = c.finalize()
        keys, counts = c.export(1, True)
    assert s["n_windows"] == single["summary"]["n_windows"] and (keys == single["keys"]).all() and (counts == single["counts"]).all()


# ---- results of the group --------------------------------------------------------------------------------------------------
def same_file(a, b) -> bool:
    x, y = np.memmap(a, dtype=np.uint8, mode="r"), np.memmap(b, dtype=np.uint8, mode="r")
    return len(x) == len(y) and all((x[i:i + (1 << 28)] == y[i:i + (1 << 28)]).all() for i in range(0, len(x), 1 << 28))


def _check_files(data, is_fastq, k, tmp_path, batch_bases, kmix=True):
    ref = str(tmp_path / "one.tsv")
    single = one_context(data, is_fastq, k, text_path=ref)
    ora = oracle_of(data, is_fastq, k)
    tsv, kmix_path = str(tmp_path / "group.tsv"), (str(tmp_path / "group.kmix") if kmix else None)
    results, errors, _ = run_group(4, k, data, is_fastq, batch_bases=batch_bases, text_path=tsv, kmix_path=kmix_path)
    check(results, errors, 4, ora, single)
    assert same_file(tsv, ref)
    os.remove(tsv); os.remove(ref)
    if kmix:
        kk, ikeys, icounts = orc.kmix_decode(open(kmix_path, "rb").read())
        o2 = np.argsort(ikeys, kind="stable")
        assert kk == k and results[0]["n_kmix"] == len(ora["keys"]) and (ikeys[o2] == ora["keys"]).all() and (icounts[o2] == ora["counts"]).all()
    return results


def test_group_text_and_index_equal_one_context(tmp_path):
    _check_files(_fasta_image(np.random.default_rng(11), 60, 70, b"\r\n", True, True, True), False, 21, tmp_path, 1 << 20)
    _check_files(_fastq_image(4000), True, 31, tmp_path, 1 << 20)


def test_c1_sized_image(tmp_path):
    """100 records x 1 Mbp on 80-column lines (101 MB): several rounds per rank."""
    g = orc.synth_uniform(42, 0, 100_000_000).tobytes()
    parts = []
    for r in range(100):
        s = g[r * 1_000_000:(r + 1) * 1_000_000]
        parts.append(b">chr%d\n" % r + b"\n".join(s[i:i + 80] for i in range(0, len(s), 80)) + b"\n")
    results = _check_files(b"".join(parts), False, 21, tmp_path, 1 << 23, kmix=False)
    assert all(r["stats"]["rounds"] >= 3 for r in results)


# ---- errors: every rank returns well before the barrier timeout, and the documented fallback gives the oracle --------------
def fallback(world, k, data, is_fastq, q=None):
    """A fresh group on fresh contexts: kmg_parse_fastx on the host, each rank its share of the records."""
    from krust_b200.api import parse_fastx
    seq, qual, offsets = parse_fastx(data, is_fastq)
    n = len(offsets) - 1
    group = f"fb{os.getpid()}-{time.time_ns() & 0xffffff:x}"
    results, errors = [None] * world, []

    def worker(r):
        c = kb.GpuKmerCounter(k, min_quality=q)
        try:
            c.shard_join(world, r, group, max(len(seq), 1))
            lo, hi = n * r // world, n * (r + 1) // world
            a, b = int(offsets[lo]), int(offsets[hi])
            c.shard_count_batch(np.ascontiguousarray(seq[a:b]), None if qual is None else np.ascontiguousarray(qual[a:b]),
                                (offsets[lo:hi + 1] - a).astype(np.uint64))
            s = c.shard_finalize()
            results[r] = (s, *c.export(1, True))
            c.shard_leave()
        except Exception as e:  # noqa: BLE001
            errors.append(repr(e))
        finally:
            c.close()

    ts = [threading.Thread(target=worker, args=(r,)) for r in range(world)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=300)
    assert not any(t.is_alive() for t in ts) and not errors, errors
    keys, counts, windows = orc.count_batch(k, seq, qual, offsets, q)
    allk = np.concatenate([r[1] for r in results]); allc = np.concatenate([r[2] for r in results])
    o = np.argsort(allk, kind="stable")
    assert (allk[o] == keys).all() and (allc[o] == counts).all() and results[0][0]["n_windows"] == windows


def _fails_everywhere(world, k, data, is_fastq, images=None, batch_bases=1 << 20):
    results, errors, secs = run_group(world, k, data, is_fastq, batch_bases=batch_bases, images=images)
    assert all(e is not None for e in errors), errors
    assert secs < 60, f"ranks took {secs:.0f} s to give up"
    return errors


def test_errors_return_on_every_rank_and_the_fallback_counts():
    k = 21
    ml = b"".join(b"@r%d\nACGTACGTAC\nGTACGTACGT\n+\nIIIIIIIIII\nIIIIIIIIII\n" % i for i in range(400))   # multi-line FASTQ
    errs = _fails_everywhere(3, k, ml, True)
    assert all(isinstance(e, kb.SequenceParseError) for e in errs), errs
    fallback(3, k, ml, True, 20)
    rng = np.random.default_rng(5)
    long_line = b">a\n" + bytes(rng.choice(list(b"ACGT"), size=300_000).tolist()) + b"\n>b\nACGTACGTACGTACGTACGTACGTA\n"
    errs = _fails_everywhere(4, k, long_line, False, batch_bases=8192)     # a line longer than a chunk
    assert all(isinstance(e, kb.SequenceParseError) for e in errs), errs
    fallback(4, k, long_line, False)
    errs = _fails_everywhere(2, k, b"ACGT\n>r\nACGTACGT\n", False)           # no header at byte 0
    assert all(isinstance(e, kb.SequenceParseError) for e in errs), errs
    data = _fasta_image(rng, 20, 60, b"\n")
    errs = _fails_everywhere(3, k, data, False, images=[data, data, data[: len(data) - 1000]])   # one rank passes a shorter image
    assert all(isinstance(e, kb.GpuError) and e.status == kb._lib.KMG_ERR_INVALID_ARG for e in errs), errs
    fallback(3, k, data, False)


# ---- process ranks: one process per GPU, each maps the same file -------------------------------------------------------------
def _proc(rank, world, port, path, out_dir):
    import torch
    import torch.distributed as dist
    from krust_b200.dist import GpuShardEngine, ShardedKmerCounter
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dev = torch.device(f"cuda:{rank}")
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        eng = GpuShardEngine(21, dev)
        sc = ShardedKmerCounter(eng)
        with open(path, "rb") as f, mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ) as m:
            image = np.frombuffer(m, dtype=np.uint8)
            n = sc.count_file_image(image, False)
            del image
        s = sc.finalize()
        keys, counts = sc.export_gathered(1)
        if rank == 0:
            np.savez(os.path.join(out_dir, "procs.npz"), keys=keys, counts=counts, n=n, windows=s["n_windows"], records=s["n_records"])
        dist.barrier()
        eng.close()
    finally:
        dist.destroy_process_group()


def test_process_ranks_map_the_same_file(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    world = min(torch.cuda.device_count(), 4)
    data = _fasta_image(np.random.default_rng(9), 200, 80, b"\n", max_len=40_000)
    p = tmp_path / "g.fa"
    p.write_bytes(data)
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_proc, args=(world, port, str(p), str(tmp_path)), nprocs=world, join=True)
    got = np.load(tmp_path / "procs.npz")
    ora = oracle_of(data, False, 21)
    assert int(got["n"]) == int(got["records"]) == ora["records"] and int(got["windows"]) == ora["windows"]
    assert (got["keys"] == ora["keys"]).all() and (got["counts"] == ora["counts"]).all()
