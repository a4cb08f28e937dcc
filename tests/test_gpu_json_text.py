"""--format json formatted on the device: kmg_emit_text / kmg_write_text of one context and kmg_shard_write_text of a group write
the bytes of output_counts / write_counts (serde_json::to_string_pretty of the sorted {kmer, count} vector plus a newline, which
is also json.dumps(..., indent=2) + "\\n").  Ranks of a group are threads with their own contexts on one device (as in
test_gpu_shard_text.py); the last test runs one process per GPU where a box has several."""
import hashlib
import io
import json
import os
import pickle
import socket
import subprocess
import threading
import time

import numpy as np
import pytest

import krust_b200 as kb
from krust_b200 import _lib
from krust_b200.dist import slice_for_rank
from oracle import oracle as orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FX = os.path.join(ROOT, "tests", "golden", "fixtures")
BIN = os.path.join(ROOT, "krust_b200", "host", "kmerust-b200")
PART, HASH, DIRECT = _lib.KMG_FLAG_FORCE_PARTITIONED, _lib.KMG_FLAG_FORCE_HASH, _lib.KMG_FLAG_FORCE_DIRECT

SIMPLE_K3 = (b'[\n'
             b'  {\n    "kmer": "AAT",\n    "count": 1\n  },\n'
             b'  {\n    "kmer": "ACA",\n    "count": 1\n  },\n'
             b'  {\n    "kmer": "ACG",\n    "count": 4\n  },\n'
             b'  {\n    "kmer": "ATC",\n    "count": 1\n  },\n'
             b'  {\n    "kmer": "GTA",\n    "count": 3\n  },\n'
             b'  {\n    "kmer": "TAA",\n    "count": 1\n  }\n'
             b']\n')


def ref_json(keys, counts, k) -> bytes:
    out = io.BytesIO()
    kb.write_counts(out, keys, counts, k, "json")
    return out.getvalue()


def emit(c, m):
    out = io.BytesIO()
    n_rec, n_bytes = c.emit_text(out, "json", m)
    return out.getvalue(), n_rec, n_bytes


def np_json_records(keys, counts, k, first) -> bytes:
    """Vectorised json records (no framing): every record is ",\\n" + body, the first of the output "\\n" + body."""
    n = len(keys)
    if n == 0:
        return b""
    counts = np.ascontiguousarray(counts, dtype=np.uint64)
    nd = np.ones(n, dtype=np.int64)
    v = counts.copy()
    for _ in range(19):
        v //= np.uint64(10)
        nd += v > 0
    head, mid, tail = b',\n  {\n    "kmer": "', b'",\n    "count": ', b"\n  }"
    w = len(head) + k + len(mid) + 20 + len(tail)
    mat = np.zeros((n, w), dtype=np.uint8)
    mat[:, :len(head)] = np.frombuffer(head, dtype=np.uint8)
    o = len(head)
    mat[:, o:o + k] = kb.unpack_many(keys, k).view(np.uint8).reshape(n, k)
    o += k
    mat[:, o:o + len(mid)] = np.frombuffer(mid, dtype=np.uint8)
    o += len(mid)
    cols = np.arange(20)
    digits = np.zeros((n, 20), dtype=np.uint8)   # the count's digits, most significant in column 0
    v = counts.copy()
    for i in range(20):                          # i-th digit from the right goes to column nd - 1 - i
        col = nd - 1 - i
        rows = np.nonzero(col >= 0)[0]
        digits[rows, col[rows]] = (v[rows] % np.uint64(10)).astype(np.uint8) + ord("0")
        v //= np.uint64(10)
    mat[:, o:o + 20] = digits
    t = np.frombuffer(tail, dtype=np.uint8)
    mat[np.arange(n)[:, None], o + nd[:, None] + np.arange(len(tail))[None, :]] = t
    mask = np.ones((n, w), dtype=bool)
    mask[:, o:o + 20] = cols[None, :] < nd[:, None]
    mask[:, o + 20:] = False
    mask[np.arange(n)[:, None], o + nd[:, None] + np.arange(len(tail))[None, :]] = True
    if first:
        mask[0, 0] = False
    return mat[mask].tobytes()


def np_json(keys, counts, k) -> bytes:
    return b"[" + np_json_records(keys, counts, k, True) + (b"\n]\n" if len(keys) else b"]\n")


# ------------------------------------------------------------------------------------------------------------------ one context
def test_known_answer_simple_fa_k3_from_count_batch_and_count_fastx():
    path = os.path.join(FX, "simple.fa")
    seq, qual, offsets = kb.read_records(path)
    docs = []
    with kb.GpuKmerCounter(3) as c:
        c.count_batch(seq, qual, offsets)
        c.finalize(False)
        keys, counts = c.export(1, True)
        docs.append(emit(c, 1))
    with kb.GpuKmerCounter(3) as c:
        with open(path, "rb") as f:
            c.count_fastx(f.read(), False)
        c.finalize(False)
        docs.append(emit(c, 0))
    for got, n_rec, n_bytes in docs:
        assert got == SIMPLE_K3 and n_rec == 6 and n_bytes == len(SIMPLE_K3)
    assert ref_json(keys, counts, 3) == SIMPLE_K3
    names = kb.unpack_many(keys, 3).tolist()
    assert json.dumps([{"kmer": s.decode(), "count": int(n)} for s, n in zip(names, counts.tolist())], indent=2).encode() + b"\n" == SIMPLE_K3
    assert np_json(keys, counts, 3) == SIMPLE_K3


@pytest.mark.parametrize("k,flags", [(1, 0), (2, 0), (13, DIRECT), (13, PART), (21, 0), (21, PART), (31, PART), (32, HASH), (32, PART)])
def test_every_engine_path_and_k_equals_write_counts_of_the_oracle(k, flags, tmp_path):
    rng = np.random.default_rng(k * 16 + flags)
    recs = [b"A" * 3000, b"ACGTTGCA" * 150] + [bytes(rng.choice(list(b"ACGTN"), p=[.24, .24, .24, .24, .04], size=int(rng.integers(0, 2000))).tolist())
                                              for _ in range(300)]
    okeys, ocounts, _ = orc.count_records(k, recs, mode="rolling")
    above = int(ocounts.max()) + 1
    with kb.GpuKmerCounter(k, flags=flags, parts_log2=3 if flags == PART else 0) as c:
        c.count_records(recs)
        c.finalize(False)
        for m in (0, 1, 2, 50, above):
            fk, fc = orc.filter_min_count(okeys, ocounts, max(m, 1))
            want = ref_json(fk, fc, k)
            got, n_rec, n_bytes = emit(c, m)
            assert got == want and n_rec == len(fk) and n_bytes == len(want), (k, flags, m)
            assert json.loads(got) == [{"kmer": s.decode(), "count": int(n)} for s, n in zip(kb.unpack_many(fk, k).tolist(), fc.tolist())]
        assert emit(c, above)[0] == b"[]\n"
        p = tmp_path / "o.json"
        assert c.write_text(p, "json", 2) == (len(orc.filter_min_count(okeys, ocounts, 2)[0]), os.path.getsize(p))
        assert p.read_bytes() == ref_json(*orc.filter_min_count(okeys, ocounts, 2), k)


def test_every_count_width_from_1_to_20_digits():
    """Weighted keys: counts 1, 9, 10, 99, 100, ..., 10^19 and 2^64 - 1 (every decimal width), in random key order."""
    import torch
    k = 21
    widths = [1] + [x for e in range(1, 20) for x in (10 ** e - 1, 10 ** e)] + [2 ** 64 - 1]
    rng = np.random.default_rng(3)
    keys = np.unique(rng.integers(0, 4 ** k, size=4 * len(widths), dtype=np.uint64))[:len(widths)]
    counts = np.array(widths, dtype=np.uint64)
    rng.shuffle(counts)
    with kb.GpuKmerCounter(k, flags=HASH) as c:
        d_k = torch.from_numpy(keys.view(np.int64)).cuda()
        d_c = torch.from_numpy(counts.view(np.int64)).cuda()
        c.insert_keys_device(d_k.data_ptr(), len(keys), d_c.data_ptr())
        torch.cuda.synchronize()
        c.finalize(False)
        gk, gc = c.export(1, True)
        assert (gk == keys).all() and sorted(gc.tolist()) == sorted(widths)
        for m in (1, 10 ** 10, 2 ** 64 - 1):
            fk, fc = orc.filter_min_count(gk, gc, m)
            got, n_rec, n_bytes = emit(c, m)
            want = ref_json(fk, fc, k)
            assert got == want == np_json(fk, fc, k) and n_rec == len(fk) and n_bytes == len(got), m
    assert {len(str(w)) for w in widths} == set(range(1, 21))


def _piece_cuts(keys, k, target=1 << 24):
    """The cuts of kmg's sorted-piece walker (piece_cuts in kmg_api.cu) over the key histogram of the top 12 key bits."""
    shift = 2 * k - 12 if 2 * k > 12 else 0
    hb = np.bincount((keys >> np.uint64(shift)).astype(np.int64), minlength=4096)
    cap = max(int(hb.max()), min(int(hb.sum()), target))
    cuts, b0 = [0], 0
    while b0 < 4096:
        ub, b1 = int(hb[b0]), b0 + 1
        while b1 < 4096 and ub + int(hb[b1]) <= cap:
            ub += int(hb[b1]); b1 += 1
        if ub:
            cuts.append(b1)
        b0 = b1
    return cuts, shift


def test_several_pieces_and_sink_chunks_first_piece_filtered_out():
    """40 M weighted keys: ~3 sorted pieces of 2^24 records and ~40 chunks of 64 MiB.  Every key of the first piece has count 1,
    so with min_count 2 the first record of the output opens the second piece.  Compared as a streamed hash against the
    vectorised formatter."""
    import torch
    k, n = 21, 40_000_000
    rng = np.random.default_rng(12)
    keys = np.unique(rng.integers(0, 4 ** k, size=n + n // 100, dtype=np.uint64))[:n]
    keys = keys[rng.permutation(len(keys))]
    cuts, shift = _piece_cuts(keys, k)
    assert len(cuts) >= 4
    counts = rng.integers(2, 100, size=len(keys), dtype=np.uint64)
    counts[(keys >> np.uint64(shift)) < np.uint64(cuts[1])] = 1
    order = np.argsort(keys)
    skeys, scounts = keys[order], counts[order]
    with kb.GpuKmerCounter(k, flags=HASH, expected_distinct=len(keys)) as c:
        d_k = torch.from_numpy(keys.view(np.int64)).cuda()
        d_c = torch.from_numpy(counts.view(np.int64)).cuda()
        c.insert_keys_device(d_k.data_ptr(), len(keys), d_c.data_ptr())
        torch.cuda.synchronize()
        del d_k, d_c
        c.finalize(False)
        for m in (1, 2):
            keep = scounts >= m
            fk, fc = skeys[keep], scounts[keep]
            assert len(fk) > 1 << 24
            if m == 2:
                assert (fk[0] >> np.uint64(shift)) == cuts[1]   # the first passing record is the first key of piece 2
            h, size = hashlib.sha256(), [0]

            class Hasher:
                def write(self, b):
                    h.update(b); size[0] += len(b)

            n_rec, n_bytes = c.emit_text(Hasher(), "json", m)
            want, want_size = hashlib.sha256(b"["), 1
            step = 4_000_000
            for i in range(0, len(fk), step):
                part = np_json_records(fk[i:i + step], fc[i:i + step], k, i == 0)
                want.update(part); want_size += len(part)
            want.update(b"\n]\n"); want_size += 3
            assert n_rec == len(fk) and n_bytes == size[0] == want_size and h.hexdigest() == want.hexdigest(), m


# ------------------------------------------------------------------------------------------------------------------ shard groups
def run_group(world, k, seq, offsets, action, expected_keys=0):
    """Every rank counts its slice_for_rank(...) of the stream in a fresh group, then returns action(counter, rank)."""
    import torch
    dev = torch.device("cuda:0")
    total = len(seq)
    group = f"json{os.getpid()}-{time.time_ns() & 0xffffff:x}"
    results, errors = [None] * world, []

    def worker(r):
        c = None
        try:
            a, b = slice_for_rank(total, world, r, k)
            mid = np.asarray(offsets[1:-1], dtype=np.int64)
            inside = mid[(mid > a) & (mid < b)] - a
            off = np.concatenate([[0], inside, [b - a]]).astype(np.int64)
            c = kb.GpuKmerCounter(k)
            c.shard_join(world, r, group, expected_keys or total)
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


def _genome(rng, n, p_n=0.01):
    return rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8), p=[(1 - p_n) / 4] * 4 + [p_n], size=n).astype(np.uint8)


@pytest.mark.parametrize("world,k", [(2, 21), (3, 32), (4, 31), (8, 15)])
def test_group_json_equals_single_context_and_oracle(world, k, tmp_path):
    rng = np.random.default_rng(world * 100 + k + 1)
    seq = _genome(rng, 1_500_000)
    offsets = np.array([0, 1, 400_000, 400_000, 1_100_000, 1_100_777, len(seq)], dtype=np.uint64)
    okeys, ocounts, _ = orc.count_batch_mt(k, seq, None, offsets)
    mins = (0, 1, 2, 50)
    results, errors = run_group(world, k, seq, offsets, lambda c, r: {m: c.shard_write_text(tmp_path / f"group-{m}.json", "json", m) for m in mins})
    assert not errors, errors
    for m in mins:
        fk, fc = orc.filter_min_count(okeys, ocounts, max(m, 1))
        want = ref_json(fk, fc, k)
        one = tmp_path / f"one-{m}.json"
        with kb.GpuKmerCounter(k) as c:
            c.count_batch(seq, None, offsets)
            assert c.write_text(one, "json", m) == (len(fk), len(want))
        assert (tmp_path / f"group-{m}.json").read_bytes() == one.read_bytes() == want, m
        assert all(res[m] == (len(fk), len(want)) for res in results)


def test_group_json_poly_a_alone_and_empty_output(tmp_path):
    """poly-A: one rank holds the only record, and rank 0, which owns the file's only piece, merges it out of that rank's staging
    buffer as the file's first record; a min_count above every count: "[]\\n".  A first record formatted by a rank other than 0
    is tested by test_group_json_many_pieces_and_steps."""
    k = 21
    polya = np.frombuffer(b"A" * 300_000, dtype=np.uint8)
    off1 = np.array([0, len(polya)], dtype=np.uint64)
    p, e = tmp_path / "polya.json", tmp_path / "empty.json"
    n = len(polya) - k + 1

    def action(c, r):
        return c.shard_write_text(p, "json", 1), c.export(1, True)[0].size, c.shard_write_text(e, "json", n + 1)

    results, errors = run_group(3, k, polya, off1, action)
    assert not errors, errors
    assert sorted(r[1] for r in results) == [0, 0, 1]
    want = b'[\n  {\n    "kmer": "%s",\n    "count": %d\n  }\n]\n' % (b"A" * k, n)
    assert p.read_bytes() == want and all(r[0] == (1, len(want)) for r in results)
    assert e.read_bytes() == b"[]\n" and all(r[2] == (0, 3) for r in results)


def _revcomp(x, k):
    c = x ^ np.uint64(4 ** k - 1)
    r = np.zeros_like(c)
    for i in range(k):
        r = (r << np.uint64(2)) | ((c >> np.uint64(2 * i)) & np.uint64(3))
    return r


def _sha_of_file(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for block in iter(lambda: f.read(1 << 26), b""):
            h.update(block)
    return h.hexdigest()


def _sha_of_emit(c, m):
    h, size = hashlib.sha256(), [0]

    class Hasher:
        def write(self, b):
            h.update(b); size[0] += len(b)

    n_rec, n_bytes = c.emit_text(Hasher(), "json", m)
    assert n_bytes == size[0]
    return n_rec, n_bytes, h.hexdigest()


def _sha_of_np_json(keys, counts, k):
    h, size = hashlib.sha256(b"["), 1
    for i in range(0, len(keys), 4_000_000):
        part = np_json_records(keys[i:i + 4_000_000], counts[i:i + 4_000_000], k, i == 0)
        h.update(part); size += len(part)
    tail = b"\n]\n" if len(keys) else b"]\n"
    h.update(tail)
    return size + len(tail), h.hexdigest()


def test_group_json_many_pieces_and_steps(tmp_path):
    """~40 M distinct 21-mers, each fed as records of exactly k bases, so that every key's count is chosen: three sorted pieces of
    ~2^24 records.  Every key of the first piece occurs once, every other key twice.  At world 2 the pieces make two steps (rank 0
    owns pieces 0 and 2, rank 1 piece 1); at world 4 they make one step in which rank 3 owns no piece.  min_count 1: rank 0 formats
    the file's first record, and the pieces of later ranks and of the later step land at their offsets with "," in front of their
    first record; min_count 2: the first piece is empty, so rank 1 formats the file's first record.  The group's file equals the
    json of one context and the vectorised formatter (compared as streamed hashes); totals on every rank."""
    k, n = 21, 40_000_000
    rng = np.random.default_rng(31)
    x = rng.integers(0, 4 ** k, size=n, dtype=np.uint64)
    keys, first = np.unique(np.minimum(x, _revcomp(x, k)), return_index=True)   # canonical keys, sorted; k odd: no palindromes
    x = x[first]
    cuts, shift = _piece_cuts(keys, k)
    assert len(cuts) - 1 == 3
    counts = np.where((keys >> np.uint64(shift)) < np.uint64(cuts[1]), 1, 2).astype(np.uint64)
    recs = np.repeat(x, counts.astype(np.int64))
    recs = recs[rng.permutation(len(recs))]
    del x
    seq = np.empty(len(recs) * k, dtype=np.uint8)
    for i in range(0, len(recs), 4_000_000):
        part = recs[i:i + 4_000_000]
        seq[i * k:(i + len(part)) * k] = kb.unpack_many(part, k).view(np.uint8)
    offsets = np.arange(0, (len(recs) + 1) * k, k, dtype=np.uint64)
    want = {}
    for m in (1, 2):
        keep = counts >= m
        fk, fc = keys[keep], counts[keep]
        assert len(fk) > 1 << 24
        if m == 2:
            assert int(fk[0] >> np.uint64(shift)) == cuts[1]   # the output opens with the first key of piece 1
        want[m] = (len(fk),) + _sha_of_np_json(fk, fc, k)
    with kb.GpuKmerCounter(k, expected_distinct=len(keys)) as c:
        c.count_batch(seq, None, offsets)
        assert c.finalize()["n_distinct"] == len(keys)
        for m in (1, 2):
            assert _sha_of_emit(c, m) == want[m], m
    for world in (2, 4):
        def action(c, r):
            out = {}
            for m in (1, 2):
                out[m] = c.shard_write_text(tmp_path / f"group{world}-{m}.json", "json", m)
            return out

        results, errors = run_group(world, k, seq, offsets, action, expected_keys=len(recs))
        assert not errors, errors
        for m in (1, 2):
            p = tmp_path / f"group{world}-{m}.json"
            n_rec, size, sha = want[m]
            assert all(res[m] == (n_rec, size) for res in results), (world, m)
            assert os.path.getsize(p) == size and _sha_of_file(p) == sha, (world, m)
            os.remove(p)


def test_group_ranks_disagreeing_on_json_and_tsv_all_fail(tmp_path):
    rng = np.random.default_rng(1)
    seq = _genome(rng, 200_000)

    def mismatch(c, r):
        try:
            c.shard_write_text(tmp_path / "mismatch", "json" if r != 1 else "tsv", 1)
            return "no error"
        except kb.GpuError as e:
            return str(e)

    t0 = time.time()
    results, errors = run_group(3, 21, seq, np.array([0, len(seq)], dtype=np.uint64), mismatch)
    assert not errors and all(r != "no error" for r in results) and time.time() - t0 < 100, results


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
        out = sc.write_text(os.path.join(out_dir, "multi.json"), "json", 2)
        with open(os.path.join(out_dir, f"r{rank}.pkl"), "wb") as f:
            pickle.dump(out, f)
        eng.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(_n_gpus() < 2, reason="needs >= 2 GPUs")
def test_multi_gpu_processes_sharded_counter_writes_json(tmp_path):
    """One process per GPU through ShardedKmerCounter.write_text(path, "json") on the fused group."""
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
    fk, fc = orc.filter_min_count(*orc.count_batch_mt(k, seq, None, offsets)[:2], 2)
    want = ref_json(fk, fc, k)
    assert (tmp_path / "multi.json").read_bytes() == want
    for r in range(world):
        with open(tmp_path / f"r{r}.pkl", "rb") as f:
            assert pickle.load(f) == (len(fk), len(want))


# ------------------------------------------------------------------------------------------------------------------ public layers
def _cli(*args):
    if not os.path.exists(BIN):
        subprocess.check_call(["make", "-C", os.path.dirname(BIN), "-s"])
    return subprocess.run([BIN, *args], capture_output=True, timeout=300)


def test_cli_json_equals_output_counts_of_the_sorted_export(tmp_path):
    """kmerust-b200 -f json (device formatting) against write_counts over the sorted export, the bytes of output_counts."""
    rng = np.random.default_rng(21)
    recs = [bytes(rng.choice(list(b"ACGTN"), p=[.24, .24, .24, .24, .04], size=int(rng.integers(1, 400))).tolist()) for _ in range(500)]
    quals = [bytes((rng.choice([2, 11, 25, 37], p=[.1, .1, .2, .6], size=len(s)) + 33).astype(np.uint8).tolist()) for s in recs]
    fa, fq = tmp_path / "multi.fa", tmp_path / "multi.fq"
    fa.write_bytes(b"".join(b">r%d\n%s\n" % (i, s) for i, s in enumerate(recs)))
    fq.write_bytes(b"".join(b"@r%d\n%s\n+\n%s\n" % (i, s, q) for i, (s, q) in enumerate(zip(recs, quals))))
    cases = [(3, os.path.join(FX, name), []) for name in ("simple.fa", "simple.fq", "with_n.fa", "with_n.fq", "soft_masked.fa", "low_quality.fq")]
    cases += [(4, os.path.join(FX, "low_quality.fq"), ["-Q", "20"]), (11, str(fa), []), (11, str(fa), ["-m", "2"]),
              (15, str(fq), ["-Q", "20"]), (7, str(fq), ["-Q", "20", "-m", "3"]), (21, str(fa), ["-m", "1000000"])]
    for k, path, extra in cases:
        r = _cli(str(k), path, "-f", "json", "-q", *extra)
        assert r.returncode == 0, r.stderr
        m = int(extra[extra.index("-m") + 1]) if "-m" in extra else 1
        q = int(extra[extra.index("-Q") + 1]) if "-Q" in extra else None
        seq, qual, offsets = kb.read_records(path)
        with kb.GpuKmerCounter(k, min_quality=q) as c:
            c.count_batch(seq, qual, offsets)
            c.finalize(False)
            keys, counts = c.export(m, True)
        assert r.stdout == ref_json(keys, counts, k), (k, path, extra)
    assert _cli("3", os.path.join(FX, "simple.fa"), "-f", "json", "-q").stdout == SIMPLE_K3


def test_builder_count_to_writer_json_equals_write_counts():
    for k, name, m in ((3, "simple.fa", 1), (3, "simple.fq", 2), (3, "soft_masked.fa", 1), (4, "with_n.fq", 1), (3, "simple.fa", 99)):
        path = os.path.join(FX, name)
        out = io.BytesIO()
        kb.KmerCounter.new().k(k).min_count(m).format("json").count_to_writer(path, out)
        keys, counts = kb.KmerCounter.new().k(k).min_count(m).count_packed(path)
        order = np.argsort(keys)
        assert out.getvalue() == ref_json(keys[order], counts[order], k), (k, name, m)
    out = io.BytesIO()
    kb.KmerCounter.new().k(3).format("json").count_to_writer(os.path.join(FX, "simple.fa"), out)
    assert out.getvalue() == SIMPLE_K3
