"""Multi-GPU sharding of the per-line transform (SURVEY.md 8e) -- the reference's producer + worker pool
(main.go:345-396) with GPUs as the workers.

Lines are independent, so the data region of a VCF is cut into newline-aligned byte ranges; every GPU runs the
same kernel pipeline on its ranges with its own host thread, context and streams, and the host writes the
outputs back in input order.  There is no cross-shard reduction, hence no collective (no NCCL): the only thing
every GPU needs is the small constant context (config + header).

Two partitions are provided:
  * `partition`      N contiguous shards of ~equal size (one per GPU / rank): what `bench.py`'s strong-scaling arm
                     and the world_size-2 gloo test use;
  * `read_vcf_multi` the product path: the data region is cut into chunks (config.chunkBytes), chunk k goes to GPU
                     k mod N, results are written in chunk order.  Output streams while the GPUs work and host
                     memory stays bounded (a few chunks per GPU), which N contiguous shards cannot offer: shard 1's
                     whole output would have to wait for shard 0's.  A bgzf (.vcf.gz) input is cut into groups of
                     whole blocks (bgzf.plan_groups, libbvcf's bvcf_bgzf_plan): the compressed bytes go to the GPUs, which inflate them.
Both are pure host logic around bvcf_submit / bvcf_collect.
"""
from __future__ import annotations

import ctypes as C
import mmap
import os
import queue
import stat
import threading
from typing import BinaryIO, List, Optional, Sequence, Tuple

from . import bgzf
from ._lib import BvcfError
from .host import Config, PinnedRing, Sink, Transformer, locus_at, read_preamble


def partition(data, begin: int, end: int, n: int) -> List[Tuple[int, int]]:
    """Split data[begin:end] into n byte ranges of ~equal size whose boundaries follow a newline.

    `data` only needs find(b"\\n", lo, hi) (bytes, bytearray, mmap).  Ranges are contiguous, cover [begin, end)
    exactly, and every range except possibly the last ends just after a b"\\n" (so does the last one when the
    input is newline-terminated).  Empty ranges are possible when there are fewer lines than shards."""
    cuts = [begin]
    for k in range(1, n):
        target = begin + (end - begin) * k // n
        target = max(target, cuts[-1])
        if target >= end:
            cuts.append(end)
            continue
        if target == begin or data[target - 1:target] == b"\n":
            cuts.append(target)
            continue
        nl = data.find(b"\n", target, end)
        cuts.append(end if nl < 0 else nl + 1)
    cuts.append(end)
    return [(cuts[i], cuts[i + 1]) for i in range(n)]


def chunk_ranges(data, lo: int, hi: int, chunk_bytes: int) -> List[Tuple[int, int]]:
    """Newline-aligned sub-chunks of one shard (what bvcf_submit is fed)."""
    out = []
    p = lo
    while p < hi:
        q = min(p + chunk_bytes, hi)
        if q < hi:
            nl = data.rfind(b"\n", p, q)
            if nl < 0:  # a single line longer than the chunk: extend to its end
                nl = data.find(b"\n", q, hi)
                q = hi if nl < 0 else nl + 1
            else:
                q = nl + 1
        out.append((p, q))
        p = q
    return out


def _stage(dst: int, data, lo: int, hi: int) -> None:
    """data[lo:hi] -> pinned memory at address dst (one memmove; ctypes drops the GIL for it)."""
    n = hi - lo
    if n == 0:
        return
    if isinstance(data, bytes):
        src = C.cast(C.c_char_p(data), C.c_void_p).value + lo
        C.memmove(dst, src, n)
    else:
        try:  # writable buffers (bytearray, pinned numpy views ...)
            src = C.addressof((C.c_char * len(data)).from_buffer(data)) + lo
            C.memmove(dst, src, n)
        except (TypeError, BufferError):  # read-only mmap and friends
            C.memmove(dst, bytes(data[lo:hi]), n)


def _gpu_worker(cfg: Config, device: int, eol_width: int, chrom_line: bytes, data, chunks, my_ids, results, errors,
                n_slots: int):
    """One GPU: its chunks in order, n_slots in flight; results (chunk id, ChunkResult) into `results`.  A chunk is a
    (lo, hi) byte range of plain text or a bgzf.Group."""
    ring = None
    try:
        c = Config(**{**cfg.__dict__, "device": device})
        gz = bool(chunks) and isinstance(chunks[0], bgzf.Group)
        cap = max((chunks[i][1] - chunks[i][0] for i in my_ids), default=0) + 1
        text_cap = max((chunks[i].text + len(chunks[i].tail) for i in my_ids), default=0) + 1 if gz else cap
        ring = PinnedRing(n_slots + 1, cap)
        with Transformer(c, eol_width=eol_width, n_slots=n_slots, max_chunk_bytes=text_cap) as tr:
            tr.set_header(chrom_line)
            if cfg.regions is not None:
                tr.set_regions(cfg.regions)
            sub = col = 0
            while col < len(my_ids):
                while sub < len(my_ids) and sub - col < n_slots:
                    ch = chunks[my_ids[sub]]
                    buf = ring.ptrs[sub % (n_slots + 1)]
                    _stage(buf, data, ch[0], ch[1])
                    if gz:
                        tr.submit_bgzf(sub, (buf, ch.hi - ch.lo), ch.skip, ch.tail)
                    else:
                        tr.submit(sub, (buf, ch[1] - ch[0]))
                    sub += 1
                res = tr.collect(col, diag_fields=gz)
                results.put((my_ids[col], res))  # blocks when the writer is behind: bounded host memory
                col += 1
    except BaseException as e:  # surfaced by the caller
        errors.append(e)
        results.put((None, None))
    finally:
        if ring is not None:
            ring.close()


def whole_input(reader: BinaryIO, head: bytes = b""):
    """The whole input of `reader`, of which `head` has been read already: the file mapped read-only when the reader is
    a regular file read from its start, otherwise head + the rest read."""
    try:
        st = os.fstat(reader.fileno())
        if stat.S_ISREG(st.st_mode) and st.st_size > 0 and reader.tell() == len(head):
            return mmap.mmap(reader.fileno(), 0, access=mmap.ACCESS_READ)
    except (AttributeError, OSError, ValueError):  # io.BytesIO and other readers without a file behind them
        pass
    return bytes(head) + reader.read()


def read_vcf_multi(config: Config, data, writer: Optional[BinaryIO], devices: Sequence[int], diag_sink=None,
                   n_slots: int = 3) -> dict:
    """readVcf (main.go:241-396) over several GPUs of one box.  `data` is the whole uncompressed VCF as a bytes-like
    object or mmap, or a whole bgzf (.vcf.gz) file.  Chunk k of the data region goes to devices[k mod N] (a device may
    be listed more than once); rows, dosage batches and diagnostics leave in input order while the GPUs are still
    working."""
    chunk_bytes = max(int(config.chunkBytes), 1 << 16)
    gz = bgzf.is_bgzf(data)
    width, chrom_line, off = read_preamble(data, gz)
    if gz:
        try:
            # with regions and an index beside the file, only the blocks of the index's spans are read
            views = bgzf.index_views(data, config.inPath, config.regions) if config.regions and config.inPath else None
            cap = 2 * chunk_bytes + (64 << 20)
            chunks = bgzf.plan_groups(data, off, chunk_bytes, cap) if views is None else bgzf.plan_views(data, views, chunk_bytes, cap)
        except ValueError as e:
            raise BvcfError(str(e)) from None
        end = off + sum(g.text - g.skip + len(g.tail) for g in chunks)
    else:
        last_nl = data.rfind(b"\n", off, len(data))
        end = off if last_nl < 0 else last_nl + 1  # an unterminated last line is dropped (main.go:354-357)
        chunks = chunk_ranges(data, off, end, chunk_bytes)
    n_dev = len(devices)
    sink = Sink(config, chrom_line, writer, diag_sink)
    errors: list = []
    queues = [queue.Queue(maxsize=n_slots + 1) for _ in range(n_dev)]
    threads = []
    for g, dev in enumerate(devices):
        ids = list(range(g, len(chunks), n_dev))
        t = threading.Thread(target=_gpu_worker, args=(config, dev, width, chrom_line, data, chunks, ids, queues[g], errors,
                                                       n_slots), daemon=True)
        t.start()
        threads.append(t)
    try:
        for k in range(len(chunks)):  # chunk order == input order
            cid, res = queues[k % n_dev].get()
            if cid is None:
                raise errors[0]
            assert cid == k
            sink.put(res, res.diag_fields if gz else (locus_at(data, chunks[k][0] + st) for st in res.diag_starts))
    finally:
        sink.close()
        for q in queues:  # unblock workers if we are bailing out
            while True:
                try:
                    q.get_nowait()
                except queue.Empty:
                    break
        for t in threads:
            t.join(timeout=60)
    if errors:
        raise errors[0]
    return {**sink.totals, "in_bytes": end - off, "n_chunks": len(chunks), "devices": list(devices)}
