"""Hash-sharded multi-GPU counting: one process per GPU, torch.distributed for launch / rendezvous.

The count table shards by k-mer hash (SURVEY.md 8e).  With the CUDA engine the exchange is FUSED into the pipeline
(`kmg_shard_*` in include/kmerust_gpu.h): every rank scatters its keys by (owner, hash bin) into its own send buffer and the
owner's refine kernel pulls its bins out of all ranks' buffers over NVLink (P2P-mapped memory) while it partitions them
further; sizes, flags, summaries and histograms cross through a shared-memory segment inside the library.
torch.distributed only names the group and times the run.

A generic path (bucket -> all_to_all_single -> adopt) remains for engines without the fused calls: it is what the CPU tests
drive with the gloo backend and a stand-in engine (tests/test_dist_gloo.py), and it can be forced on GPUs with
KMG_DIST_FUSED=0 for A/B measurements (NCCL all-to-all of raw keys: the round-1 design).

The reference has no distributed mode; this replaces the single shared DashMap of src/run.rs:489-583 by `world`
disjoint tables.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import os
import time

import numpy as np
import torch
import torch.distributed as dist

_TIMING = bool(os.environ.get("KMG_DIST_TIMING"))


def slice_for_rank(total: int, world: int, rank: int, k: int) -> Tuple[int, int]:
    """Byte range [a, b) of a `total`-byte stream that `rank` scans: equal cuts, each extended by the
    k-1 halo so that every window is seen by exactly one rank (windows are assigned to the rank
    that owns their first base)."""
    a = total * rank // world
    b = total * (rank + 1) // world
    if rank + 1 < world:
        b = min(total, b + k - 1)
    return a, b


def merge_histograms(parts: List[Tuple[np.ndarray, np.ndarray]]) -> Tuple[np.ndarray, np.ndarray]:
    """Element-wise sum of (count value -> frequency) maps; ascending by count value."""
    acc: Dict[int, int] = {}
    for vals, freqs in parts:
        for v, f in zip(vals.tolist(), freqs.tolist()):
            acc[v] = acc.get(v, 0) + f
    keys = sorted(acc)
    return np.array(keys, dtype=np.uint64), np.array([acc[x] for x in keys], dtype=np.uint64)


class GpuShardEngine:
    """One rank's CUDA engine: thin adapter from torch tensors to the raw-pointer C ABI."""

    fused = True   # offers the kmg_shard_* calls (the owners' refine kernels pull their bins over NVLink)

    def __init__(self, k: int, device: torch.device, min_quality: Optional[int] = None, expected_distinct: int = 0,
                 flags: int = 0, batch_bases: int = 0):
        from .api import GpuKmerCounter
        self.device = device
        torch.cuda.set_device(device)
        self.stream = torch.cuda.current_stream(device)
        # The engine must run on the SAME stream torch orders its NCCL work against.  torch's default "current
        # stream" is the legacy default stream, whose handle is 0 -- which the C ABI reads as "use a private
        # stream" -- so it is passed as cudaStreamLegacy (0x1) instead.
        handle = self.stream.cuda_stream or 1
        if dist.is_initialized() and dist.get_world_size() > 1:
            from ._lib import KMG_FLAG_FORCE_PARTITIONED
            flags |= KMG_FLAG_FORCE_PARTITIONED  # the exchange moves hash-partitioned keys, whatever k is
        self.counter = GpuKmerCounter(k, min_quality=min_quality, expected_distinct=expected_distinct, flags=flags,
                                      device=device.index, stream=handle, batch_bases=batch_bases)
        self.k = k
        self.batch_bases = batch_bases
        self.joined = False

    def join(self, world: int, rank: int, group: str, expected_keys_total: int):
        self.counter.shard_join(world, rank, group, expected_keys_total)
        self.joined = True

    def count_fused(self, seq: torch.Tensor, offsets: Optional[torch.Tensor] = None, qual: Optional[torch.Tensor] = None):
        n_rec = 1 if offsets is None else offsets.numel() - 1
        self.counter.shard_count_device(seq.data_ptr() if seq.numel() else 0, seq.numel(), qual.data_ptr() if qual is not None and qual.numel() else 0,
                                        offsets.data_ptr() if offsets is not None else 0, n_rec)

    def count_local(self, seq: torch.Tensor, offsets: Optional[torch.Tensor] = None, qual: Optional[torch.Tensor] = None):
        n_rec = 1 if offsets is None else offsets.numel() - 1
        self.counter.count_device(seq.data_ptr(), seq.numel(), qual.data_ptr() if qual is not None else 0,
                                  offsets.data_ptr() if offsets is not None else 0, n_rec)

    def extract(self, seq: torch.Tensor, n_shards: int, offsets: Optional[torch.Tensor] = None,
                qual: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, np.ndarray]:
        """Canonical keys of every counted window, bucketed shard-major.  Returns (keys int64[n], counts[n_shards])."""
        n_rec = 1 if offsets is None else offsets.numel() - 1
        cap = max(int(seq.numel()), 1)
        out = torch.empty(cap, dtype=torch.int64, device=self.device)
        counts = self.counter.extract_keys_device(seq.data_ptr(), seq.numel(), n_shards, out.data_ptr(), cap,
                                                  qual.data_ptr() if qual is not None else 0,
                                                  offsets.data_ptr() if offsets is not None else 0, n_rec)
        return out[: int(counts.sum())], counts

    def insert(self, keys: torch.Tensor, counts: Optional[torch.Tensor] = None):
        if keys.numel():
            self.counter.insert_keys_device(keys.data_ptr(), keys.numel(), counts.data_ptr() if counts is not None else 0)

    def plan(self, expected_keys: int) -> int:
        """Put the engine on the partitioned pipeline; returns its number of coarse hash bins."""
        return self.counter.partition_plan(expected_keys)[0]

    def adopt(self, keys: torch.Tensor, bin_counts: np.ndarray):
        """Take a block of keys that is already grouped by this engine's coarse bins (counts on the host)."""
        if keys.numel():
            self.counter.adopt_coarse_device(keys.data_ptr(), bin_counts, keys.numel())

    def finalize(self, want_summary: bool = True):
        return self.counter.finalize(want_summary)

    def export(self, min_count: int = 1):
        return self.counter.export(min_count, sorted=True)

    def histogram(self, min_count: int = 1):
        return self.counter.histogram(min_count)

    def reset(self):
        self.counter.reset()

    def close(self):
        if self.joined:
            try:
                self.counter.shard_leave()
            except Exception:
                pass
            self.joined = False
        self.counter.close()


class ShardedKmerCounter:
    """Drives one engine per rank through scan -> bucket -> all-to-all -> local upsert."""

    def __init__(self, engine, group=None, n_chunks: int = 0):
        self.engine = engine
        self.group = group
        self.n_chunks = n_chunks   # 0 = automatic: two pieces for slices of >= 2^30 bases, else one.  Measured on 2 x B200 (C4,
                                   # 1.55 G bases per rank): 1 piece 63.3 ms/step, 2 pieces 59.8, 3 pieces 68.5, 5 pieces 71 -- every
                                   # piece costs a few host round trips, which soon outweigh the overlap
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.sent_keys = 0
        self.recv_keys = 0
        self._p1 = None
        self.fused = bool(getattr(engine, "fused", False)) and os.environ.get("KMG_DIST_FUSED", "1") != "0" and self.world > 1

    def _join(self, expected_keys_total: int):
        """All ranks join ONE shard group with identical arguments (name from rank 0, size hint = the largest proposal)."""
        dev0 = getattr(self.engine, "device", torch.device("cpu"))
        t = torch.tensor([int(expected_keys_total)], dtype=torch.int64, device=dev0)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        name = [f"{os.getpid()}-{time.time_ns() & 0xffffffffff:x}" if self.rank == 0 else None]
        dist.broadcast_object_list(name, src=dist.get_global_rank(self.group, 0) if self.group is not None else 0, group=self.group)
        self.engine.join(self.world, self.rank, name[0], int(t.item()))

    def count(self, seq, offsets=None, qual=None, expected_keys_per_rank: int = 0, n_chunks: Optional[int] = None):
        """`seq` is THIS rank's slice (see slice_for_rank); offsets/qual are relative to it.

        Every rank buckets its keys straight into world x P1 global coarse hash bins (P1 = the engines' common
        coarse-partition count); bins [r*P1, (r+1)*P1) belong to rank r, so ONE all-to-all moves contiguous
        ranges and the owner adopts each received block as already coarse-partitioned input.

        With `n_chunks` > 1 the slice is processed in pieces (k-1 bases of overlap, every window counted by exactly
        one piece) so that the key exchange of piece j runs on NCCL's stream while the engine refines piece j-1 and
        scans piece j+1 (see __init__ for the default)."""
        if self.world == 1:
            self.engine.count_local(seq, offsets, qual)
            return
        if self.fused:
            if not self.engine.joined:
                self._join(max(int(expected_keys_per_rank), int(seq.numel()), 1) * self.world)
            self.engine.count_fused(seq, offsets, qual)   # rounds of batch_bases; the ranks agree on their number inside
            return
        if self._p1 is None:
            # all ranks must agree on P1: take the plan of the rank expecting the most keys
            mine = self.engine.plan(max(int(expected_keys_per_rank), int(seq.numel()), 1))
            dev0 = getattr(self.engine, "device", torch.device("cpu"))
            t = torch.tensor([mine, -mine], dtype=torch.int64, device=dev0)
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
            self._p1 = int(t[0].item())
            if self._p1 != -int(t[1].item()):   # EVERY rank sees the disagreement and raises: nobody is left waiting in a collective
                raise RuntimeError(f"ranks disagree on the partition plan ({-int(t[1].item())}..{self._p1} coarse bins); pass the same expected_keys_per_rank")
        p1, world, k = self._p1, self.world, int(self.engine.k)
        n = int(seq.numel())
        # every rank must run the same number of exchanges: agree on the largest slice's choice
        if n_chunks is None:
            n_chunks = self.n_chunks if self.n_chunks else int(os.environ.get("KMG_DIST_CHUNKS", "2" if n >= (1 << 30) else "1"))
        dev0 = getattr(self.engine, "device", torch.device("cpu"))
        t = torch.tensor([int(n_chunks)], dtype=torch.int64, device=dev0)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        n_chunks = int(t.item())
        cuts = [((n * j) // n_chunks) & ~15 for j in range(n_chunks)] + [n]   # 16-byte aligned piece starts
        off_host = None if offsets is None else offsets.detach().cpu().numpy().astype(np.int64)

        def finish(p):
            work, recv, recv_split, recv_m, _keep = p
            if work is not None:
                work.wait()
            o = 0
            for src in range(world):
                self.engine.adopt(recv[o:o + recv_split[src]], recv_m[src].astype(np.uint64))
                o += recv_split[src]

        def lap(tag, t0):
            if _TIMING and self.rank == 0:
                if seq.is_cuda:
                    torch.cuda.synchronize(seq.device)
                print(f"[dist timing] {tag}: {(time.perf_counter() - t0) * 1e3:.2f} ms", flush=True)
            return time.perf_counter()

        pending = None
        t0 = time.perf_counter()
        for j in range(n_chunks):
            a = cuts[j]
            b = n if j + 1 == n_chunks else min(n, cuts[j + 1] + k - 1)
            if b <= a:
                sub_seq, sub_qual, sub_off = seq[:0], (None if qual is None else qual[:0]), None
            else:
                sub_seq = seq[a:b]
                sub_qual = None if qual is None else qual[a:b]
                sub_off = None
                if off_host is not None:
                    inside = off_host[(off_host > a) & (off_host < b)] - a
                    sub_off = torch.from_numpy(np.concatenate([[0], inside, [b - a]]).astype(np.int64)).to(seq.device)
            keys, bin_counts = self.engine.extract(sub_seq, world * p1, sub_off, sub_qual)
            t0 = lap("extract", t0)
            dev = keys.device
            send_m = torch.as_tensor(bin_counts.astype(np.int64), device=dev)       # [world * p1], owner-major
            recv_m = torch.empty_like(send_m)
            dist.all_to_all_single(recv_m, send_m, group=self.group)                # row s = what source s holds for my bins
            recv_m = recv_m.cpu().numpy().reshape(world, p1)
            send_split = bin_counts.reshape(world, p1).sum(axis=1).astype(np.int64).tolist()
            recv_split = recv_m.sum(axis=1).astype(np.int64).tolist()
            recv = torch.empty(int(sum(recv_split)), dtype=torch.int64, device=dev)
            t0 = lap("count exchange", t0)
            work = dist.all_to_all_single(recv, keys, output_split_sizes=recv_split, input_split_sizes=send_split, group=self.group,
                                          async_op=True)
            self.sent_keys += int(sum(send_split)) - send_split[self.rank]
            self.recv_keys += int(sum(recv_split)) - recv_split[self.rank]
            if _TIMING:
                work.wait()
                t0 = lap("key exchange", t0)
            if pending is not None:
                finish(pending)          # refine piece j-1 while piece j is on the wire
            pending = (work, recv, recv_split, recv_m, keys)
        if pending is not None:
            finish(pending)
            t0 = lap("adopt", t0)

    def count_host(self, seq: np.ndarray, offsets: np.ndarray, qual: Optional[np.ndarray] = None, expected_keys_per_rank: int = 0):
        """THIS rank's slice in HOST memory (pinned arrays are DMA'd directly): kmg_shard_count_ascii stages it through the
        context's pinned ring, chunk by chunk, every chunk one fused scatter + exchange round."""
        if self.world == 1:
            self.engine.counter.count_batch(seq, qual, offsets)
        elif self.fused:
            if not self.engine.joined:
                self._join(max(int(expected_keys_per_rank), len(seq), 1) * self.world)
            self.engine.counter.shard_count_batch(seq, qual, offsets)
        else:
            dev = self.engine.device
            self.count(torch.from_numpy(seq).to(dev, non_blocking=True), torch.from_numpy(np.asarray(offsets).astype(np.int64)).to(dev),
                       None if qual is None else torch.from_numpy(qual).to(dev, non_blocking=True), expected_keys_per_rank=expected_keys_per_rank)

    def count_file_image(self, image, is_fastq: bool) -> int:
        """The WHOLE FASTA / FASTQ file image, the same on every rank (e.g. each rank's mmap of the file): kmg_shard_count_fastx
        parses only this rank's slice of it on the device.  Returns the records of the whole image.  At world 1 it is count_fastx."""
        if self.world == 1:
            return self.engine.counter.count_fastx(image, is_fastq)
        if not self.fused:
            raise RuntimeError("count_file_image needs the fused shard group (kmg_shard_*)")
        if not self.engine.joined:
            self._join(max(len(image) // 2 if is_fastq else len(image), 1))   # the size hint kmg_count_fastx plans with
        return self.engine.counter.shard_count_fastx(image, is_fastq)

    def finalize(self) -> dict:
        """Global summary: sums over shards (shards are disjoint), max of max_count."""
        if self.fused and self.engine.joined:
            out = self.engine.counter.shard_finalize()      # kmg_shard_finalize: merged inside the library
            out["local"] = self.engine.finalize(True)
            st = self.engine.counter.shard_stats()
            self.sent_keys, self.recv_keys = st["sent_keys"], st["recv_keys"]
            return out
        s = self.engine.finalize(True)
        if self.world == 1:
            return s
        dev = getattr(self.engine, "device", torch.device("cpu"))
        sums = torch.tensor([s["n_windows"], s["n_distinct"], s["n_records"], s["n_bases"]], dtype=torch.int64, device=dev)
        mx = torch.tensor([s["max_count"]], dtype=torch.int64, device=dev)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=self.group)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX, group=self.group)
        out = dict(s)
        out["n_windows"], out["n_distinct"], out["n_records"], out["n_bases"] = [int(x) for x in sums.cpu().tolist()]
        out["max_count"] = int(mx.item())
        out["local"] = s
        return out

    def histogram(self, min_count: int = 1):
        """Count-of-counts over all shards (every rank gets the merged result)."""
        if self.fused and self.engine.joined:
            return self.engine.counter.shard_histogram(min_count)
        vals, freqs = self.engine.histogram(min_count)
        if self.world == 1:
            return vals, freqs
        parts: List = [None] * self.world
        dist.all_gather_object(parts, (vals, freqs), group=self.group)
        return merge_histograms(parts)

    def export_gathered(self, min_count: int = 1):
        """All shards' (key, count) lists concatenated and key-sorted on every rank (tests / small outputs)."""
        keys, counts = self.engine.export(min_count)
        if self.world == 1:
            return keys, counts
        parts: List = [None] * self.world
        dist.all_gather_object(parts, (keys, counts), group=self.group)
        k = np.concatenate([p[0] for p in parts]); c = np.concatenate([p[1] for p in parts])
        order = np.argsort(k, kind="stable")
        return k[order], c[order]

    def save_kmix(self, path) -> dict:
        """ONE .kmix index from all shards (rank 0 writes header + combined CRC, every rank its own records)."""
        if self.world == 1 or (self.fused and self.engine.joined):
            n = self.engine.counter.shard_save_kmix(path)
            return {"records": int(n)}
        # generic path: the same protocol driven from here (kmg_kmix_begin / kmg_save_kmix_shard / kmg_kmix_finish)
        from .api import kmix_begin, kmix_finish
        s = self.engine.finalize(True)
        sizes: List = [None] * self.world
        dist.all_gather_object(sizes, int(s["n_distinct"]), group=self.group)
        if self.rank == 0:
            kmix_begin(path)
        dist.barrier(group=self.group)
        n, crc = self.engine.counter.save_kmix_shard(path, sum(sizes[: self.rank]))
        parts: List = [None] * self.world
        dist.all_gather_object(parts, (int(n), int(crc)), group=self.group)
        if self.rank == 0:
            kmix_finish(path, int(self.engine.k), [p[0] for p in parts], [p[1] for p in parts])
        dist.barrier(group=self.group)
        return {"records": int(sum(p[0] for p in parts))}

    def write_text(self, path, fmt: str = "tsv", min_count: int = 1) -> Tuple[int, int]:
        """ONE sorted fasta / tsv / json file from all shards, byte-identical to what one GPU writes for the same input
        (collective).  Returns (records, bytes) of the whole file on every rank."""
        if self.world == 1:
            return self.engine.counter.write_text(path, fmt, min_count)
        if self.fused and self.engine.joined:
            return self.engine.counter.shard_write_text(path, fmt, min_count)
        raise RuntimeError("write_text needs the fused shard group (kmg_shard_*): the generic bucket + all-to-all path has no "
                           "cross-shard text writer")

    def stats(self) -> dict:
        out = {"path": "fused exchange (owners' refine kernels pull their bins from all ranks' send buffers over NVLink)" if self.fused else "bucket + NCCL all_to_all_single + adopt",
               "sent_keys": int(self.sent_keys), "recv_keys": int(self.recv_keys)}
        if self.fused and getattr(self.engine, "joined", False):
            out.update(self.engine.counter.shard_stats())
        return out
