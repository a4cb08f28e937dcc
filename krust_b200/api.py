"""Host-side mirror of kmerust's counting API on top of the C ABI (include/kmerust_gpu.h).

Same names, argument meaning and error behaviour as the reference so that the parity tests read like
the reference's own tests.  Citations are into the kmerust repository.  All counting happens on the
GPU through libkmerust_gpu.so; there is no CPU fallback (importing works without a GPU, creating a
counter does not).
"""
from __future__ import annotations

import ctypes as C
import gzip
import os
import stat
import sys
import zlib
from typing import Dict, IO, Iterable, Iterator, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import KmgBatch, KmgConfig, KmgSummary


# ----------------------------------------------------------------------------- errors (src/error.rs)
class KmeRustError(Exception):
    """Base error (src/error.rs:11-83)."""


class KmerLengthError(KmeRustError, ValueError):
    """src/error.rs:88-97 -- k outside 1..=32."""

    def __init__(self, k: int, min: int = 1, max: int = 32):
        super().__init__(f"k-mer length {k} is out of range (must be {min}-{max})")
        self.k, self.min, self.max = k, min, max


class SequenceParseError(KmeRustError):
    """KmeRustError::SequenceParse{details} (src/error.rs:27-30)."""


class InvalidIndexError(KmeRustError):
    """KmeRustError::InvalidIndex{details, path} (src/index.rs:296-340)."""


class BuilderError(KmeRustError):
    """src/error.rs:159 -- e.g. KmerLengthNotSet."""


class GpuError(KmeRustError):
    """Any failing C-ABI status that has no reference equivalent (CUDA, OOM, table full)."""

    def __init__(self, status: int, message: str):
        super().__init__(f"[kmg status {status}] {message}")
        self.status = status


def _check(status: int, ctx=None):
    if status == _lib.KMG_OK:
        return
    L = _lib.load()
    msg = (L.kmg_last_error(ctx) or b"").decode() or L.kmg_status_string(status).decode()
    if status == _lib.KMG_ERR_INVALID_K:
        raise KmeRustError(msg)
    if status == _lib.KMG_ERR_PARSE:
        raise SequenceParseError(msg)
    raise GpuError(status, msg)


# output formats the device text emitters write (kmg_emit_text / kmg_write_text / kmg_shard_write_text)
_TEXT_FORMATS = {"fasta": _lib.KMG_TEXT_FASTA, "tsv": _lib.KMG_TEXT_TSV, "json": _lib.KMG_TEXT_JSON}


# ----------------------------------------------------------------------------- k-mer primitives (src/kmer.rs)
class KmerLength:
    """Validated k in 1..=32 (src/kmer.rs:74-145)."""
    MIN, MAX = 1, 32

    def __init__(self, k: int):
        if not (self.MIN <= int(k) <= self.MAX):
            raise KmerLengthError(int(k), self.MIN, self.MAX)
        self._k = int(k)

    new = classmethod(lambda cls, k: cls(k))

    def get(self) -> int:
        return self._k

    def as_u8(self) -> int:
        return self._k

    def __int__(self):
        return self._k

    def __eq__(self, other):
        return int(other) == self._k

    def __hash__(self):
        return hash(self._k)

    def __repr__(self):
        return f"KmerLength({self._k})"


def _k(k) -> int:
    return k.get() if isinstance(k, KmerLength) else KmerLength(k).get()


def unpack_to_string(packed_bits: int, k) -> str:
    """src/kmer.rs:431-456: base i = (bits >> 2(k-1-i)) & 3 -> ACGT."""
    k = _k(k)
    return "".join("ACGT"[(int(packed_bits) >> (2 * (k - 1 - i))) & 3] for i in range(k))


def unpack_many(keys: np.ndarray, k) -> np.ndarray:
    """Vectorised unpack_to_string: (n,) u64 -> (n,) |S{k} byte strings."""
    k = _k(k)
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    shifts = (np.arange(k - 1, -1, -1, dtype=np.uint64) * np.uint64(2))
    codes = ((keys[:, None] >> shifts[None, :]) & np.uint64(3)).astype(np.uint8)
    return np.frombuffer(b"ACGT", dtype=np.uint8)[codes].view(f"S{k}").ravel()


# ----------------------------------------------------------------------------- formats (src/format.rs)
class SequenceFormat:
    AUTO, FASTA, FASTQ = "auto", "fasta", "fastq"

    @staticmethod
    def from_extension(path) -> str:
        """src/format.rs:47-70: .fq/.fastq (optionally .gz) -> FASTQ, everything else FASTA."""
        name = os.path.basename(os.fspath(path)).lower()
        if name.endswith(".gz"):
            name = name[:-3]
        ext = name.rsplit(".", 1)[-1] if "." in name else ""
        return SequenceFormat.FASTQ if ext in ("fq", "fastq") else SequenceFormat.FASTA

    @staticmethod
    def resolve(fmt: str, path=None) -> str:
        """src/format.rs:97-102."""
        if fmt == SequenceFormat.AUTO:
            return SequenceFormat.FASTA if path is None else SequenceFormat.from_extension(path)
        return fmt


def read_records(path, fmt: str = SequenceFormat.AUTO):
    """Stand-in for reader::read_with_quality (src/reader.rs:167-247): whole file -> records laid back
    to back.  Returns (seq u8[], qual u8[]|None, offsets u64[n+1])."""
    p = os.fspath(path)
    if p == "-":
        data = sys.stdin.buffer.read()
        resolved = SequenceFormat.resolve(fmt, None)
    else:
        try:
            with open(p, "rb") as f:
                data = f.read()
        except OSError as e:
            raise KmeRustError(f"failed to read sequences from '{p}': {e}") from e
        if p.lower().endswith(".gz"):
            try:
                data = gzip.decompress(data)
            except (OSError, EOFError, zlib.error) as e:
                raise KmeRustError(f"failed to read sequences from '{p}': {e}") from e
        resolved = SequenceFormat.resolve(fmt, p)
    return parse_fastx(data, resolved == SequenceFormat.FASTQ)


def parse_fastx(data: bytes, is_fastq: bool):
    L = _lib.load()
    n = len(data)
    src = np.frombuffer(data, dtype=np.uint8) if n else np.zeros(1, dtype=np.uint8)
    seq = np.empty(max(n, 1), dtype=np.uint8)
    qual = np.empty(max(n, 1), dtype=np.uint8) if is_fastq else None
    max_records = data.count(b">" if not is_fastq else b"@") + 1
    offsets = np.zeros(max_records + 1, dtype=np.uint64)
    n_rec = C.c_uint64(0)
    err = C.create_string_buffer(256)
    st = L.kmg_parse_fastx(src.ctypes.data, n, int(is_fastq), seq.ctypes.data, qual.ctypes.data if is_fastq else None,
                           offsets.ctypes.data, max_records, C.byref(n_rec), err, 256)
    if st != _lib.KMG_OK:
        raise SequenceParseError(err.value.decode() or "sequence parse error")
    offsets = offsets[: n_rec.value + 1].copy()
    total = int(offsets[-1])
    return seq[:total], (qual[:total] if is_fastq else None), offsets


# ----------------------------------------------------------------------------- the engine handle
class GpuKmerCounter:
    """Owns one kmg_ctx.  Replaces KmerMap / StreamingKmerCounter (src/run.rs:491-583,
    src/streaming.rs:833-1114) behind the same feed -> finalize -> results life cycle."""

    def __init__(self, k, min_quality: Optional[int] = None, expected_distinct: int = 0, batch_bases: int = 0,
                 flags: int = 0, device: int = -1, stream: Optional[int] = None, parts_log2: int = 0):
        self.k = _k(k)
        self._L = _lib.load()
        cfg = KmgConfig()
        cfg.abi_version = _lib.KMG_ABI_VERSION
        cfg.k = self.k
        cfg.device = device
        cfg.flags = flags
        cfg.has_min_quality = int(min_quality is not None)
        cfg.min_quality = int(min_quality or 0)
        cfg.expected_distinct = int(expected_distinct)
        cfg.batch_bases = int(batch_bases)
        cfg.parts_log2 = int(parts_log2)
        cfg.stream = stream
        self._ctx = C.c_void_p()
        _check(self._L.kmg_create(C.byref(cfg), C.byref(self._ctx)), None)

    # -- life cycle
    def close(self):
        if getattr(self, "_ctx", None):
            self._L.kmg_destroy(self._ctx)
            self._ctx = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def reset(self):
        _check(self._L.kmg_reset(self._ctx), self._ctx)

    # -- feeding (host buffers)
    def count_batch(self, seq: np.ndarray, qual: Optional[np.ndarray], offsets: np.ndarray):
        """kmg_count_ascii over records laid back to back (host arrays; pinned torch tensors' numpy views
        are DMA'd directly)."""
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n_rec = len(offsets) - 1
        if n_rec <= 0:
            return
        assert seq.dtype == np.uint8 and seq.flags.c_contiguous
        if qual is not None:
            assert qual.dtype == np.uint8 and qual.flags.c_contiguous and len(qual) >= int(offsets[-1])
        assert len(seq) >= int(offsets[-1])
        _check(self._L.kmg_count_ascii(self._ctx, seq.ctypes.data if len(seq) else None,
                                       qual.ctypes.data if qual is not None and len(qual) else None,
                                       offsets.ctypes.data, n_rec), self._ctx)

    def count_fastx(self, data, is_fastq: bool) -> int:
        """kmg_count_fastx: a whole FASTA / FASTQ file image (bytes, bytearray, numpy u8 or mmap) parsed on the device.
        Returns the number of records."""
        arr = data if isinstance(data, np.ndarray) else np.frombuffer(data, dtype=np.uint8)
        assert arr.dtype == np.uint8 and arr.flags.c_contiguous
        n = C.c_uint64(0)
        _check(self._L.kmg_count_fastx(self._ctx, arr.ctypes.data if len(arr) else None, len(arr), int(is_fastq), C.byref(n)), self._ctx)
        return n.value

    def count_stream(self, readable, is_fastq: bool, size_hint: int = 0, block: int = 64 << 20) -> int:
        """kmg_fastx_stream_*: a FASTA / FASTQ byte stream (sys.stdin.buffer, gzip.open(...), any object with readinto or read)
        parsed on the device, pushed in blocks of `block` bytes; host memory stays bounded by the block and the staging ring.
        size_hint: bytes expected (0 = unknown).  A stream the device parser refuses (multi-line FASTQ ...) goes on through the
        host splitter: the bytes it did not count plus the rest of the stream are split with parse_fastx and fed to count_batch.
        Returns the records of the whole stream.  An exception from the reader abandons the stream with kmg_reset."""
        L, ctx = self._L, self._ctx
        r0 = self.progress()[0]
        _check(L.kmg_fastx_stream_begin(ctx, int(is_fastq), int(size_hint)), ctx)
        buf = bytearray(block)
        addr = C.addressof((C.c_char * block).from_buffer(buf))
        view = memoryview(buf)
        st = _lib.KMG_OK
        try:
            while st == _lib.KMG_OK:
                if hasattr(readable, "readinto"):
                    n = readable.readinto(view) or 0
                else:
                    data = readable.read(block)
                    n = len(data)
                    view[:n] = data
                if n == 0:
                    break
                st = L.kmg_fastx_stream_push(ctx, addr, n)
        except BaseException:
            L.kmg_reset(ctx)
            raise
        if st == _lib.KMG_OK:
            st = L.kmg_fastx_stream_end(ctx, C.byref(C.c_uint64(0)))
        if st != _lib.KMG_OK:
            msg = (L.kmg_last_error(ctx) or b"").decode() or L.kmg_status_string(st).decode()
            n_rest = C.c_uint64(0)
            if st != _lib.KMG_ERR_PARSE or L.kmg_fastx_stream_rest(ctx, None, 0, C.byref(n_rest)) != _lib.KMG_OK:
                raise SequenceParseError(msg) if st == _lib.KMG_ERR_PARSE else GpuError(st, msg)
            rest = np.empty(n_rest.value, dtype=np.uint8)
            _check(L.kmg_fastx_stream_rest(ctx, rest.ctypes.data, n_rest.value, C.byref(n_rest)), ctx)
            tail = readable.read()
            seq, qual, offsets = parse_fastx(rest.tobytes() + (tail or b""), is_fastq)
            self.count_batch(seq, qual, offsets)
        return self.progress()[0] - r0

    def count_records(self, records: Iterable[bytes], quals: Optional[Iterable[bytes]] = None):
        records = [bytes(r) for r in records]
        offsets = np.zeros(len(records) + 1, dtype=np.uint64)
        if records:
            offsets[1:] = np.cumsum([len(r) for r in records], dtype=np.uint64)
        seq = np.frombuffer(b"".join(records), dtype=np.uint8)
        qual = None
        if quals is not None:
            quals = [bytes(q) for q in quals]
            if any(len(q) != len(r) for q, r in zip(quals, records)):
                raise SequenceParseError("sequence and quality lengths differ")
            qual = np.frombuffer(b"".join(quals), dtype=np.uint8)
        self.count_batch(seq, qual, offsets)

    # -- feeding (pre-packed pinned batches: the Rust reader's path)
    def acquire_batch(self) -> KmgBatch:
        b = KmgBatch()
        _check(self._L.kmg_acquire_batch(self._ctx, C.byref(b)), self._ctx)
        return b

    def submit_batch(self, b: KmgBatch):
        _check(self._L.kmg_submit_batch(self._ctx, C.byref(b)), self._ctx)

    # -- feeding (device-resident; raw pointers so torch stays plumbing)
    def count_device(self, d_seq: int, n_bytes: int, d_qual: int = 0, d_offsets: int = 0, n_records: int = 1):
        _check(self._L.kmg_count_ascii_device(self._ctx, d_seq, d_qual or None, d_offsets or None, n_records, n_bytes),
               self._ctx)

    def insert_keys_device(self, d_keys: int, n: int, d_counts: int = 0):
        _check(self._L.kmg_insert_keys_device(self._ctx, d_keys, d_counts or None, n), self._ctx)

    def extract_keys_device(self, d_seq: int, n_bytes: int, n_shards: int, d_keys_out: int, cap: int, d_qual: int = 0,
                            d_offsets: int = 0, n_records: int = 1) -> np.ndarray:
        counts = np.zeros(n_shards, dtype=np.uint64)
        _check(self._L.kmg_extract_keys_device(self._ctx, d_seq, d_qual or None, d_offsets or None, n_records, n_bytes,
                                               n_shards, d_keys_out or None, cap, counts.ctypes.data), self._ctx)
        return counts

    def partition_plan(self, expected_keys: int) -> Tuple[int, int]:
        a, b = C.c_uint32(0), C.c_uint32(0)
        _check(self._L.kmg_partition_plan(self._ctx, int(expected_keys), C.byref(a), C.byref(b)), self._ctx)
        return a.value, b.value

    def adopt_coarse_device(self, d_keys: int, bin_counts: np.ndarray, n: int):
        bin_counts = np.ascontiguousarray(bin_counts, dtype=np.uint64)
        _check(self._L.kmg_adopt_coarse_device(self._ctx, d_keys or None, bin_counts.ctypes.data, len(bin_counts), int(n)), self._ctx)

    def synth_uniform_device(self, seed: int, first_base: int, n: int, d_out: int):
        _check(self._L.kmg_synth_uniform_device(self._ctx, seed, first_base, n, d_out), self._ctx)

    # -- hash-sharded group of contexts, one per GPU (collective calls; see include/kmerust_gpu.h)
    def shard_join(self, world: int, rank: int, group: str, expected_keys_total: int = 0):
        _check(self._L.kmg_shard_join(self._ctx, world, rank, group.encode(), int(expected_keys_total)), self._ctx)

    def shard_leave(self):
        _check(self._L.kmg_shard_leave(self._ctx), self._ctx)

    def shard_count_device(self, d_seq: int, n_bytes: int, d_qual: int = 0, d_offsets: int = 0, n_records: int = 1):
        _check(self._L.kmg_shard_count_ascii_device(self._ctx, d_seq or None, d_qual or None, d_offsets or None, n_records, n_bytes), self._ctx)

    def shard_count_batch(self, seq: np.ndarray, qual: Optional[np.ndarray], offsets: np.ndarray):
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n_rec = max(0, len(offsets) - 1)
        assert seq.dtype == np.uint8 and seq.flags.c_contiguous
        _check(self._L.kmg_shard_count_ascii(self._ctx, seq.ctypes.data if len(seq) else None,
                                             qual.ctypes.data if qual is not None and len(qual) else None,
                                             offsets.ctypes.data if n_rec else None, n_rec), self._ctx)

    def shard_count_fastx(self, data, is_fastq: bool) -> int:
        """kmg_shard_count_fastx (collective): every rank passes the SAME whole FASTA / FASTQ file image (same input types as
        count_fastx) and parses its own slice of it on the device.  Returns the records of the whole image."""
        arr = data if isinstance(data, np.ndarray) else np.frombuffer(data, dtype=np.uint8)
        assert arr.dtype == np.uint8 and arr.flags.c_contiguous
        n = C.c_uint64(0)
        _check(self._L.kmg_shard_count_fastx(self._ctx, arr.ctypes.data if len(arr) else None, len(arr), int(is_fastq), C.byref(n)), self._ctx)
        return n.value

    def shard_finalize(self) -> dict:
        s = KmgSummary()
        _check(self._L.kmg_shard_finalize(self._ctx, C.byref(s)), self._ctx)
        return {f: getattr(s, f) for f, _ in KmgSummary._fields_}

    def shard_histogram(self, min_count: int = 1) -> Tuple[np.ndarray, np.ndarray]:
        n = C.c_uint64(0)
        _check(self._L.kmg_shard_histogram(self._ctx, min_count, None, None, 0, C.byref(n)), self._ctx)
        vals = np.empty(n.value, dtype=np.uint64)
        freqs = np.empty(n.value, dtype=np.uint64)
        if n.value:
            _check(self._L.kmg_shard_histogram(self._ctx, min_count, vals.ctypes.data, freqs.ctypes.data, n.value, C.byref(n)), self._ctx)
        return vals, freqs

    def shard_save_kmix(self, path) -> int:
        n = C.c_uint64(0)
        _check(self._L.kmg_shard_save_kmix(self._ctx, os.fspath(path).encode(), C.byref(n)), self._ctx)
        return n.value

    def shard_write_text(self, path, fmt: str = "tsv", min_count: int = 1) -> Tuple[int, int]:
        """kmg_shard_write_text (collective): ONE sorted fasta / tsv / json file from all shards of the group, the same bytes as write_text
        on a single context.  Returns (records, bytes) of the whole file."""
        code = _TEXT_FORMATS[fmt]
        n_rec, n_bytes = C.c_uint64(0), C.c_uint64(0)
        _check(self._L.kmg_shard_write_text(self._ctx, min_count, code, os.fspath(path).encode(), C.byref(n_rec), C.byref(n_bytes)), self._ctx)
        return n_rec.value, n_bytes.value

    def shard_stats(self) -> dict:
        a, b, r, x = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        _check(self._L.kmg_shard_stats(self._ctx, C.byref(a), C.byref(b), C.byref(r), C.byref(x)), self._ctx)
        return {"sent_keys": a.value, "recv_keys": b.value, "rounds": r.value, "exact_rounds": x.value}

    def synth_reads_device(self, seed: int, profile: int, first_read: int, n_reads: int, d_seq: int, d_qual: int = 0):
        _check(self._L.kmg_synth_reads_device(self._ctx, seed, profile, first_read, n_reads, d_seq, d_qual or None), self._ctx)

    # -- results
    def finalize(self, want_summary: bool = True) -> Optional[dict]:
        if not want_summary:
            _check(self._L.kmg_finalize(self._ctx, None), self._ctx)
            return None
        s = KmgSummary()
        _check(self._L.kmg_finalize(self._ctx, C.byref(s)), self._ctx)
        return {f: getattr(s, f) for f, _ in KmgSummary._fields_}

    def phase_times(self) -> dict:
        """Device time (ns) of the partitioned pipeline's stages since the last reset: kmg_phase_times."""
        out = (C.c_uint64 * 4)()
        _check(self._L.kmg_phase_times(self._ctx, out), self._ctx)
        return {"a1_ns": int(out[0]), "a2_ns": int(out[1]), "b_ns": int(out[2]), "other_ns": int(out[3])}

    def export(self, min_count: int = 1, sorted: bool = True) -> Tuple[np.ndarray, np.ndarray]:
        n = C.c_uint64(0)
        _check(self._L.kmg_export_counts(self._ctx, min_count, int(sorted), None, None, 0, C.byref(n)), self._ctx)
        keys = np.empty(n.value, dtype=np.uint64)
        counts = np.empty(n.value, dtype=np.uint64)
        if n.value:
            _check(self._L.kmg_export_counts(self._ctx, min_count, int(sorted), keys.ctypes.data, counts.ctypes.data,
                                             n.value, C.byref(n)), self._ctx)
        return keys, counts

    def export_into(self, keys: np.ndarray, counts: np.ndarray, min_count: int = 1, sorted: bool = False) -> int:
        """kmg_export_counts into caller-owned arrays (e.g. numpy views of pinned memory: the D2H copy then runs at PCIe speed).
        Returns the number of entries written; raises when the arrays are too small."""
        assert keys.dtype == np.uint64 and counts.dtype == np.uint64 and keys.flags.c_contiguous and counts.flags.c_contiguous
        n = C.c_uint64(0)
        _check(self._L.kmg_export_counts(self._ctx, min_count, int(sorted), keys.ctypes.data, counts.ctypes.data,
                                         min(len(keys), len(counts)), C.byref(n)), self._ctx)
        return n.value

    def export_shard(self, n_shards: int, shard: int, min_count: int = 1, sorted: bool = True) -> Tuple[np.ndarray, np.ndarray]:
        """The entries with key % n_shards == shard (kmg_export_shard): the result in pieces that fit the host."""
        n = C.c_uint64(0)
        _check(self._L.kmg_export_shard(self._ctx, min_count, int(sorted), n_shards, shard, None, None, 0, C.byref(n)), self._ctx)
        keys = np.empty(n.value, dtype=np.uint64)
        counts = np.empty(n.value, dtype=np.uint64)
        if n.value:
            _check(self._L.kmg_export_shard(self._ctx, min_count, int(sorted), n_shards, shard, keys.ctypes.data,
                                            counts.ctypes.data, n.value, C.byref(n)), self._ctx)
        return keys, counts

    def export_device(self, d_keys: int, d_counts: int, cap: int, min_count: int = 1, sorted: bool = False) -> int:
        n = C.c_uint64(0)
        _check(self._L.kmg_export_counts_device(self._ctx, min_count, int(sorted), d_keys or None, d_counts or None, cap,
                                                C.byref(n)), self._ctx)
        return n.value

    def histogram(self, min_count: int = 1) -> Tuple[np.ndarray, np.ndarray]:
        n = C.c_uint64(0)
        _check(self._L.kmg_histogram(self._ctx, min_count, None, None, 0, C.byref(n)), self._ctx)
        vals = np.empty(n.value, dtype=np.uint64)
        freqs = np.empty(n.value, dtype=np.uint64)
        if n.value:
            _check(self._L.kmg_histogram(self._ctx, min_count, vals.ctypes.data, freqs.ctypes.data, n.value, C.byref(n)),
                   self._ctx)
        return vals, freqs

    def emit_text(self, writer: IO[bytes], fmt: str = "tsv", min_count: int = 1) -> Tuple[int, int]:
        """kmg_emit_text: sorted fasta / tsv lines or the json document formatted on the device, written to `writer` chunk by
        chunk.  Returns (records, bytes); json's bytes include its "[" and closing bracket."""
        code = _TEXT_FORMATS[fmt]

        def sink(_user, ptr, n):
            try:
                writer.write(C.string_at(ptr, n))
                return 0
            except Exception:  # noqa: BLE001 -- reported through the status code
                return 1

        cb = _lib.TEXT_SINK(sink)
        n_rec, n_bytes = C.c_uint64(0), C.c_uint64(0)
        _check(self._L.kmg_emit_text(self._ctx, min_count, code, cb, None, C.byref(n_rec), C.byref(n_bytes)), self._ctx)
        return n_rec.value, n_bytes.value

    def write_text(self, path, fmt: str = "tsv", min_count: int = 1) -> Tuple[int, int]:
        code = _TEXT_FORMATS[fmt]
        n_rec, n_bytes = C.c_uint64(0), C.c_uint64(0)
        _check(self._L.kmg_write_text(self._ctx, min_count, code, os.fspath(path).encode(), C.byref(n_rec), C.byref(n_bytes)), self._ctx)
        return n_rec.value, n_bytes.value

    def query_keys(self, keys: np.ndarray) -> np.ndarray:
        """Counts of canonical packed keys (0 = absent), looked up on the device (kmg_query_keys)."""
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        out = np.zeros(len(keys), dtype=np.uint64)
        if len(keys):
            _check(self._L.kmg_query_keys(self._ctx, keys.ctypes.data, len(keys), out.ctypes.data), self._ctx)
        return out

    def query_kmers(self, kmers: Sequence[bytes]) -> Tuple[np.ndarray, int]:
        """Counts of k-mer strings (any case; canonicalised on the device like the `query` subcommand does on the host).
        Returns (counts, number of invalid k-mers)."""
        blob = b"".join(bytes(x) for x in kmers)
        if len(blob) != len(kmers) * self.k:
            raise KmeRustError(f"every query k-mer must have length {self.k}")
        arr = np.frombuffer(blob, dtype=np.uint8)
        out = np.zeros(len(kmers), dtype=np.uint64)
        bad = C.c_uint64(0)
        if len(kmers):
            _check(self._L.kmg_query_ascii(self._ctx, arr.ctypes.data, len(kmers), out.ctypes.data, C.byref(bad)), self._ctx)
        return out, bad.value

    @classmethod
    def open_index(cls, path, device: int = -1) -> "GpuKmerCounter":
        """kmg_index_open: a .kmix file as a ready-to-query counter on the device (src/index.rs:199-216, :282-401)."""
        L = _lib.load()
        ctx = C.c_void_p()
        st = L.kmg_index_open(os.fspath(path).encode(), device, C.byref(ctx))
        if st != _lib.KMG_OK:
            msg = (L.kmg_last_error(None) or b"").decode() or L.kmg_status_string(st).decode()
            if st == _lib.KMG_ERR_PARSE:
                raise InvalidIndexError(msg)
            if st == _lib.KMG_ERR_IO:
                raise KmeRustError(msg)
            raise GpuError(st, msg)
        self = cls.__new__(cls)
        self._L, self._ctx = L, ctx
        self.k = 0
        s = self.finalize()
        self.k = int(L.kmg_ctx_k(ctx))
        return self

    def save_kmix(self, path):
        _check(self._L.kmg_save_kmix(self._ctx, os.fspath(path).encode()), self._ctx)

    def save_kmix_shard(self, path, record_offset: int) -> Tuple[int, int]:
        """Write this shard's records into its byte range of `path`; returns (records, crc32 of those bytes)."""
        n, crc = C.c_uint64(0), C.c_uint32(0)
        _check(self._L.kmg_save_kmix_shard(self._ctx, os.fspath(path).encode(), int(record_offset), C.byref(n), C.byref(crc)), self._ctx)
        return n.value, crc.value

    def progress(self) -> Tuple[int, int]:
        r, b = C.c_uint64(0), C.c_uint64(0)
        _check(self._L.kmg_progress(self._ctx, C.byref(r), C.byref(b)), self._ctx)
        return r.value, b.value


def kmix_begin(path):
    st = _lib.load().kmg_kmix_begin(os.fspath(path).encode())
    if st != _lib.KMG_OK:
        raise KmeRustError(f"failed to write index to '{os.fspath(path)}'")


def kmix_finish(path, k: int, shard_records: Sequence[int], shard_crcs: Sequence[int]):
    rec = np.asarray(list(shard_records), dtype=np.uint64)
    crc = np.asarray(list(shard_crcs), dtype=np.uint32)
    st = _lib.load().kmg_kmix_finish(os.fspath(path).encode(), int(k), rec.ctypes.data, crc.ctypes.data, len(rec))
    if st != _lib.KMG_OK:
        raise KmeRustError(f"failed to write index to '{os.fspath(path)}'")


def owner_of(key: int, n_shards: int) -> int:
    return int(_lib.load().kmg_owner_of(int(key), n_shards))


# ----------------------------------------------------------------------------- reference-named entry points
def count_kmers_from_sequences(sequences: Iterable[bytes], k: KmerLength) -> Dict[int, int]:
    """src/streaming.rs:198-204 -- Iterator<Bytes> -> HashMap<u64,u64>."""
    with GpuKmerCounter(k) as c:
        c.count_records(sequences)
        c.finalize(False)
        keys, counts = c.export(1, sorted=True)
    return dict(zip(keys.tolist(), counts.tolist()))


def _read_file_image(path, fmt: str):
    """(bytes of an uncompressed file, is_fastq)."""
    p = os.fspath(path)
    try:
        with open(p, "rb") as f:
            data = f.read()
    except OSError as e:
        raise KmeRustError(f"failed to read sequences from '{p}': {e}") from e
    return data, SequenceFormat.resolve(fmt, p) == SequenceFormat.FASTQ


def _feed_file(c: "GpuKmerCounter", path, fmt: str):
    """File -> counter: records are found on the device -- stdin ("-") and .gz files as a stream (count_stream), other files as
    one image (kmg_count_fastx); inputs the device parser refuses (multi-line FASTQ, broken records) go through the host splitter,
    which reports the reference's parse errors."""
    p = os.fspath(path)
    if p == "-":
        try:
            st = os.fstat(sys.stdin.buffer.fileno())
            hint = st.st_size if stat.S_ISREG(st.st_mode) else 0
        except (OSError, ValueError, AttributeError):
            hint = 0
        c.count_stream(sys.stdin.buffer, SequenceFormat.resolve(fmt, None) == SequenceFormat.FASTQ, hint)
        return
    if p.lower().endswith(".gz"):
        try:
            with gzip.open(p, "rb") as g:
                c.count_stream(g, SequenceFormat.resolve(fmt, p) == SequenceFormat.FASTQ)
        except (OSError, EOFError, zlib.error) as e:
            raise KmeRustError(f"failed to read sequences from '{p}': {e}") from e
        return
    data, is_fastq = _read_file_image(path, fmt)
    try:
        c.count_fastx(data, is_fastq)
    except SequenceParseError:
        c.reset()
        seq, qual, offsets = parse_fastx(data, is_fastq)
        c.count_batch(seq, qual, offsets)


def _count_path_packed(path, k, fmt=SequenceFormat.AUTO, min_quality: Optional[int] = None, min_count: int = 1):
    with GpuKmerCounter(k, min_quality=min_quality) as c:
        _feed_file(c, path, fmt)
        c.finalize(False)
        return c.export(min_count, sorted=True)


def count_kmers_streaming_packed(path, k: KmerLength) -> Dict[int, int]:
    """src/streaming.rs:158-167."""
    keys, counts = _count_path_packed(path, k)
    return dict(zip(keys.tolist(), counts.tolist()))


def count_kmers_sequential(path, k: int) -> Dict[int, int]:
    """src/streaming.rs:252-260 (same result as the parallel packed path)."""
    return count_kmers_streaming_packed(path, KmerLength(k))


def _stringify(keys: np.ndarray, counts: np.ndarray, k: int) -> Dict[str, int]:
    names = unpack_many(keys, k)
    return {a.decode(): int(b) for a, b in zip(names.tolist(), counts.tolist())}


def count_kmers_streaming(path, k: int) -> Dict[str, int]:
    """src/streaming.rs:95-119."""
    kl = KmerLength(k)
    keys, counts = _count_path_packed(path, kl)
    return _stringify(keys, counts, kl.get())


def count_kmers(path, k: int) -> Dict[str, int]:
    """src/run.rs:221-226."""
    return count_kmers_with_quality(path, k, SequenceFormat.AUTO, None)


def count_kmers_with_format(path, k: int, fmt: str) -> Dict[str, int]:
    """src/run.rs:245-281."""
    return count_kmers_with_quality(path, k, fmt, None)


def count_kmers_with_quality(path, k: int, fmt: str = SequenceFormat.AUTO, min_quality: Optional[int] = None) -> Dict[str, int]:
    """src/run.rs:304-344."""
    kl = KmerLength(k)
    keys, counts = _count_path_packed(path, kl, fmt, min_quality)
    return _stringify(keys, counts, kl.get())


def compute_histogram_packed(counts: Dict[int, int]) -> Dict[int, int]:
    """src/histogram.rs:110-116 on an already exported map (host glue; the GPU histogram is
    GpuKmerCounter.histogram / KmerCounter.histogram)."""
    vals, freqs = np.unique(np.fromiter(counts.values(), dtype=np.uint64, count=len(counts)), return_counts=True)
    return dict(zip(vals.tolist(), freqs.tolist()))


compute_histogram = compute_histogram_packed  # src/histogram.rs:88-94 (same arithmetic, String keys)


def histogram_stats(histogram: Dict[int, int]) -> dict:
    """src/histogram.rs:148-169."""
    distinct = sum(histogram.values())
    total = sum(c * f for c, f in histogram.items())
    mode_count, mode_frequency = 0, 0
    for c in sorted(histogram):  # max_by_key keeps the last maximum
        if histogram[c] >= mode_frequency:
            mode_count, mode_frequency = c, histogram[c]
    return dict(total_kmers=total, distinct_kmers=distinct, mode_count=mode_count, mode_frequency=mode_frequency,
                mean_count=(total / distinct) if distinct else 0.0)


# ----------------------------------------------------------------------------- output (src/run.rs:441-486)
class OutputFormat:
    FASTA, TSV, JSON, HISTOGRAM = "fasta", "tsv", "json", "histogram"


def write_counts(writer: IO[bytes], keys: np.ndarray, counts: np.ndarray, k: int, fmt: str):
    """Text emitters of output_counts / count_to_writer (src/run.rs:452-481, src/builder.rs:399-442).
    Keys arrive sorted, so unlike the reference the output order is deterministic."""
    if fmt == OutputFormat.HISTOGRAM:
        vals, freqs = np.unique(counts, return_counts=True)
        writer.write(b"".join(b"%d\t%d\n" % (int(v), int(f)) for v, f in zip(vals, freqs)))
        return
    names = unpack_many(keys, k).tolist()
    if fmt == OutputFormat.FASTA:
        writer.write(b"".join(b">%d\n%s\n" % (int(c), s) for s, c in zip(names, counts.tolist())))
    elif fmt == OutputFormat.TSV:
        writer.write(b"".join(b"%s\t%d\n" % (s, int(c)) for s, c in zip(names, counts.tolist())))
    elif fmt == OutputFormat.JSON:
        import json
        data = [{"kmer": s.decode(), "count": int(c)} for s, c in zip(names, counts.tolist())]
        writer.write(json.dumps(data, indent=2).encode() + b"\n")
    else:
        raise ValueError(f"unknown output format {fmt}")


# ----------------------------------------------------------------------------- builder (src/builder.rs)
class KmerCounter:
    """Fluent builder with the reference's methods (src/builder.rs:62-526)."""

    def __init__(self):
        self._k: Optional[KmerLength] = None
        self._min_count = 1
        self._format = OutputFormat.FASTA
        self._input_format = SequenceFormat.AUTO
        self._min_quality: Optional[int] = None  # extension: the reference builder has no setter (CLI -Q only)

    @staticmethod
    def new() -> "KmerCounter":
        return KmerCounter()

    def k(self, k: int) -> "KmerCounter":
        self._k = KmerLength(k)  # raises KmerLengthError
        return self

    def min_count(self, m: int) -> "KmerCounter":
        self._min_count = int(m)
        return self

    def format(self, fmt: str) -> "KmerCounter":
        self._format = fmt
        return self

    def input_format(self, fmt: str) -> "KmerCounter":
        self._input_format = fmt
        return self

    def min_quality(self, q: Optional[int]) -> "KmerCounter":
        self._min_quality = q
        return self

    def _need_k(self) -> KmerLength:
        if self._k is None:
            raise BuilderError("k-mer length must be set before counting")  # BuilderError::KmerLengthNotSet
        return self._k

    def count_packed(self, path) -> Tuple[np.ndarray, np.ndarray]:
        return _count_path_packed(path, self._need_k(), self._input_format, self._min_quality, self._min_count)

    def count(self, path) -> Dict[str, int]:
        """src/builder.rs:242-260."""
        keys, counts = self.count_packed(path)
        return _stringify(keys, counts, self._need_k().get())

    count_streaming = count   # src/builder.rs:508-526
    count_mmap = count        # src/builder.rs:468-486

    def histogram(self, path) -> Dict[int, int]:
        """src/builder.rs:286-294 -- computed on the GPU (kmg_histogram)."""
        seq, qual, offsets = read_records(path, self._input_format)
        with GpuKmerCounter(self._need_k(), min_quality=self._min_quality) as c:
            c.count_batch(seq, qual, offsets)
            c.finalize(False)
            vals, freqs = c.histogram(self._min_count)
        return dict(zip(vals.tolist(), freqs.tolist()))

    def count_with_progress(self, path, callback) -> Dict[str, int]:
        """src/builder.rs:322-344: callback(Progress) -- invoked per submitted batch here."""
        seq, qual, offsets = read_records(path, self._input_format)
        with GpuKmerCounter(self._need_k(), min_quality=self._min_quality) as c:
            c.count_batch(seq, qual, offsets)
            r, b = c.progress()
            callback({"sequences_processed": r, "bases_processed": b})
            c.finalize(False)
            keys, counts = c.export(self._min_count, sorted=True)
        return _stringify(keys, counts, self._need_k().get())

    def count_to_writer(self, path, writer: IO[bytes]):
        """src/builder.rs:399-442.  fasta / tsv / json are formatted on the GPU (kmg_emit_text), sorted by k-mer; histogram
        comes from kmg_histogram."""
        k = self._need_k()
        if self._format not in _TEXT_FORMATS and self._format != OutputFormat.HISTOGRAM:
            raise ValueError(f"unknown output format {self._format}")
        seq, qual, offsets = read_records(path, self._input_format)
        with GpuKmerCounter(k, min_quality=self._min_quality) as c:
            c.count_batch(seq, qual, offsets)
            c.finalize(False)
            if self._format == OutputFormat.HISTOGRAM:
                vals, freqs = c.histogram(self._min_count)
                writer.write(b"".join(b"%d\t%d\n" % (int(v), int(f)) for v, f in zip(vals, freqs)))
            else:
                c.emit_text(writer, self._format, self._min_count)

    def run(self, path):
        """src/builder.rs:366-375 -- to stdout."""
        self.count_to_writer(path, sys.stdout.buffer)


# ----------------------------------------------------------------------------- .kmix index (src/index.rs)
class KmerIndex:
    """src/index.rs:69-153."""

    def __init__(self, k: KmerLength, counts: Dict[int, int]):
        self._k = k if isinstance(k, KmerLength) else KmerLength(k)
        self._counts = counts

    def k(self) -> KmerLength:
        return self._k

    def __len__(self):
        return len(self._counts)

    def is_empty(self) -> bool:
        return not self._counts

    def counts(self) -> Dict[int, int]:
        return self._counts

    def get(self, packed_bits: int) -> Optional[int]:
        return self._counts.get(packed_bits)


def save_index(index: KmerIndex, path):
    """src/index.rs:156-196, :222-279 -- host-side writer for an already exported map (the GPU-side
    writer that streams straight from the device table is GpuKmerCounter.save_kmix)."""
    items = sorted(index.counts().items())
    body = bytearray(b"KMIX" + bytes([1, index.k().get()]) + len(items).to_bytes(8, "little"))
    arr = np.array(items, dtype="<u8").reshape(-1, 2)
    body += arr.tobytes()
    body += (zlib.crc32(bytes(body)) & 0xFFFFFFFF).to_bytes(4, "little")
    p = os.fspath(path)
    opener = gzip.open if p.endswith(".gz") else open
    with opener(p, "wb") as f:
        f.write(bytes(body))


def load_index(path) -> KmerIndex:
    """src/index.rs:199-216, :282-401 -- same checks in the same order."""
    p = os.fspath(path)
    opener = gzip.open if p.endswith(".gz") else open
    try:
        with opener(p, "rb") as f:
            data = f.read()
    except OSError as e:
        raise KmeRustError(f"failed to read index from '{p}': {e}") from e
    if len(data) < 18:
        raise InvalidIndexError("file too small")
    if data[:4] != b"KMIX":
        raise InvalidIndexError("invalid magic bytes (not a kmerust index file)")
    content, stored = data[:-4], int.from_bytes(data[-4:], "little")
    computed = zlib.crc32(content) & 0xFFFFFFFF
    if computed != stored:
        raise InvalidIndexError(f"checksum mismatch (expected {stored:#x}, got {computed:#x})")
    if content[4] != 1:
        raise InvalidIndexError(f"unsupported version {content[4]}")
    try:
        k = KmerLength(content[5])
    except KmerLengthError as e:
        raise InvalidIndexError(f"invalid k-mer length: {e}") from e
    n = int.from_bytes(content[6:14], "little")
    if len(content) - 14 != n * 16:
        raise InvalidIndexError(f"data size mismatch (expected {n * 16} bytes, got {len(content) - 14} bytes)")
    arr = np.frombuffer(content, dtype="<u8", offset=14).reshape(-1, 2)
    return KmerIndex(k, dict(zip(arr[:, 0].tolist(), arr[:, 1].tolist())))
