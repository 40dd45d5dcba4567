"""bgzf (block gzip, SAM spec 4.1: what bgzip / htslib write and what .vcf.gz files are) on the host side: thin wrappers
of libbvcf's bgzf module (csrc/bvcf_bgzf.cpp, which the C++ host calls too) for the block header rule, the host inflate
and the plan that cuts a file into groups of whole blocks for the streaming path (plan_groups); the views an index gives
a run with regions; and a writer used by the tests and the bench to make compressed workloads.  The DEFLATE payloads
themselves are inflated on the GPU (csrc/bvcf_inflate.cuh: bvcf_submit_bgzf, bvcf_resident_inflate_bgzf)."""
from __future__ import annotations

import ctypes as C
import struct
import zlib
from concurrent.futures import ThreadPoolExecutor
from typing import List, NamedTuple

import numpy as np

from . import _lib

MAGIC = b"\x1f\x8b\x08\x04"
EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
MAX_TEXT = 65280  # text bytes per block (bgzip's choice: the compressed block always fits 64 KiB)
LINE_TOO_LONG = "a single line exceeds the chunk capacity; raise --chunkBytes"


def _addr(buf) -> int:
    """the address of a bytes-like object or mmap (read-only ones too)"""
    return np.frombuffer(buf, dtype=np.uint8).ctypes.data


def _reason(rc: int, why) -> str:
    return why.value.decode() if why.value else _lib.lib().bvcf_strerror(rc).decode()


def _block(buf, p: int, check: bool = True):
    """(BSIZE, ISIZE) of the bgzf block at buf[p] (bvcf_bgzf_block): BSIZE 0 while its header is not complete, ISIZE 0
    unless the whole block is there.  ValueError (with check) when it is not a bgzf block or claims ISIZE 0 but holds
    text."""
    size, isize, why = C.c_size_t(), C.c_uint32(), C.c_char_p()
    rc = _lib.lib().bvcf_bgzf_block(_addr(buf) + p, len(buf) - p, C.byref(size), C.byref(isize), C.byref(why))
    if rc and check:
        raise ValueError("%s at byte %d" % (_reason(rc, why), p))
    return size.value, isize.value


def is_bgzf(head) -> bool:
    """the first bytes of an input start with a whole bgzf header (a first block that is then refused as corrupt still
    counts: reading it reports that)"""
    return _block(head, 0, check=False)[0] > 0


def block_size(buf, p: int) -> int:
    """total size of the bgzf block that starts at buf[p] (0 when its header is not complete yet)"""
    return _block(buf, p)[0]


def _walk(buf):
    """offset, size and ISIZE (numpy arrays) of every block of a whole bgzf buffer, walked by bvcf_bgzf_blocks"""
    base, n, p, parts = _addr(buf), len(buf), 0, []
    got, why = C.c_size_t(), C.c_char_p()
    while p < n:
        cap = min((n - p) // 26 + 1, 1 << 20)  # a bgzf block has at least 26 bytes
        size, isize = np.empty(cap, np.uint32), np.empty(cap, np.uint32)
        rc = _lib.lib().bvcf_bgzf_blocks(base + p, n - p, size.ctypes.data, isize.ctypes.data, cap, C.byref(got), C.byref(why))
        if rc:
            raise ValueError("%s at byte %d" % (_reason(rc, why), p + int(size[:got.value].sum())))
        if got.value == 0:
            raise ValueError("truncated bgzf block at byte %d" % p)
        parts.append((size[:got.value], isize[:got.value]))
        p += int(parts[-1][0].sum())
    size = np.concatenate([s for s, _ in parts] or [np.zeros(0, np.uint32)]).astype(np.uint64)
    isize = np.concatenate([i for _, i in parts] or [np.zeros(0, np.uint32)]).astype(np.uint64)
    return np.cumsum(size) - size, size, isize


def blocks(buf) -> List[tuple]:
    """(offset, size, ISIZE) of every block of a whole bgzf file.  A truncated last block or bytes that are not a bgzf
    block raise ValueError, and so does a block that claims ISIZE 0 (normally only the EOF block) unless it holds no
    text: its text would otherwise be dropped without a word."""
    return list(zip(*(a.tolist() for a in _walk(buf))))


class Group(NamedTuple):
    """A chunk of the streaming path: its text is inflate(buf[lo:hi])[skip:] + tail (bvcf_submit_bgzf)."""
    lo: int
    hi: int
    skip: int
    tail: bytes
    text: int  # bytes of inflate(buf[lo:hi])


# bvcf_bgzf_blk
BLK = np.dtype([("bytes", np.uint64), ("size", np.uint64), ("start", np.uint64), ("isize", np.uint32)], align=True)


def plan_blocks(block, data_off: int, chunk_bytes: int, cap: int) -> List[tuple]:
    """bvcf_bgzf_plan over block(i) -> the address of block i's bvcf_bgzf_blk (BLK), or None past the last: the groups as
    (lo_block, hi_block, skip, tail).  An exception raised by block() ends the plan and is raised here (ctypes would
    swallow it); a refusal raises ValueError with the library's reason."""
    out, err = [], []

    def block_fn(_, i, b):
        try:
            a = block(i)
        except BaseException as e:
            err.append(e)
            return -1
        if a is None:
            return 0
        C.memmove(b, a, BLK.itemsize)
        return 1

    def emit_fn(_, lo, hi, skip, tail, n):
        out.append((lo, hi, skip, C.string_at(tail, n) if n else b""))
        return 0

    why = C.c_char_p()
    rc = _lib.lib().bvcf_bgzf_plan(_lib.BGZF_BLOCK_FN(block_fn), _lib.BGZF_EMIT_FN(emit_fn), None, data_off, chunk_bytes,
                                   cap, C.byref(why))
    if err:
        raise err[0]
    if rc:
        raise ValueError(_reason(rc, why))
    return out


def block_table(buf):
    """the blocks with text of a whole bgzf buffer as bvcf_bgzf_blk (BLK) records, and their offsets with len(buf) after
    the last"""
    off, size, isize = _walk(buf)
    keep = isize > 0
    table = np.zeros(int(keep.sum()), BLK)
    table["bytes"], table["size"], table["isize"] = off[keep] + _addr(buf), size[keep], isize[keep]
    table["start"] = np.cumsum(table["isize"]) - table["isize"]
    return table, np.append(off[keep], np.uint64(len(buf)))


def plan_groups(buf, data_off: int, chunk_bytes: int, cap: int) -> List[Group]:
    """Cut a whole bgzf file into groups of whole blocks of about chunk_bytes of text, data lines from text offset
    data_off (the end of the #CHROM line) on, by bvcf_bgzf_plan (include/bvcf.h states the rule).  A group whose text
    plus tail exceeds cap raises ValueError(LINE_TOO_LONG)."""
    table, lo_of = block_table(buf)
    a0, n = table.ctypes.data, len(table)
    starts = np.append(table["start"], table["start"][-1] + table["isize"][-1] if n else np.uint64(0)).tolist()
    lo_of = lo_of.tolist()
    return [Group(lo_of[lo], lo_of[hi], skip, tail, starts[hi] - starts[lo]) for lo, hi, skip, tail in
            plan_blocks(lambda i: a0 + i * BLK.itemsize if i < n else None, data_off, chunk_bytes, cap)]


def index_views(buf, in_path: str, regions):
    """What a run with regions reads of the whole bgzf file buf (read from in_path) when a tabix or CSI index lies beside
    it (in_path + ".tbi", else + ".csi"): (lo, hi, skip) per span the index gives (bvcf_index_spans) -- buf[lo:hi] holds
    the blocks from the span's first to its last, its data lines start at text offset skip.  The C++ host's reader
    (csrc/bvcf_host.cpp index_pieces) follows the same rule.  None when there is no index; ValueError when the index is
    malformed or points at bytes that are not a bgzf block of buf."""
    import gzip
    import os

    path = next((in_path + e for e in (".tbi", ".csi") if os.path.exists(in_path + e)), None)
    if path is None:
        return None
    with gzip.open(path, "rb") as f:
        idx = f.read()
    L, n = _lib.lib(), len(regions)
    names = (C.c_char_p * max(n, 1))(*[c for c, _, _ in regions])
    beg = (C.c_int64 * max(n, 1))(*[b for _, b, _ in regions])
    end = (C.c_int64 * max(n, 1))(*[e for _, _, e in regions])
    cap, got = 1024, C.c_size_t()
    while True:
        sp = (C.c_uint64 * (2 * cap))()
        rc = L.bvcf_index_spans(idx, len(idx), names, beg, end, n, sp, cap, C.byref(got))
        if rc != -5:  # BVCF_E_TOO_LARGE: got says how many
            break
        cap = got.value
    if rc:
        raise ValueError("%s: not a tabix or CSI index (%d)" % (path, rc))

    def block_at(off: int) -> int:
        try:
            bs = block_size(buf, off) if off < len(buf) else 0
        except ValueError:
            bs = 0
        if bs == 0 or off + bs > len(buf):
            raise ValueError("%s: virtual offset %d << 16 is not a bgzf block of %s" % (path, off, in_path))
        return bs

    views = []
    for k in range(got.value):
        cb, ce, ue = sp[2 * k] >> 16, sp[2 * k + 1] >> 16, sp[2 * k + 1] & 0xFFFF
        block_at(cb)
        hi = ce + block_at(ce) if ue else ce
        if hi > len(buf):
            raise ValueError("%s: virtual offset %d << 16 is past the end of %s" % (path, ce, in_path))
        if hi > cb:
            views.append((cb, hi, sp[2 * k] & 0xFFFF))
    return views


def plan_views(buf, views, chunk_bytes: int, cap: int) -> List[Group]:
    """plan_groups over each (lo, hi, skip) of index_views, the groups' offsets into buf"""
    mv = memoryview(buf)
    return [g._replace(lo=g.lo + lo, hi=g.hi + lo) for lo, hi, skip in views
            for g in plan_groups(mv[lo:hi], skip, chunk_bytes, cap)]


def _one_block(args) -> bytes:
    chunk, level, strategy = args
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    payload = c.compress(chunk) + c.flush()
    bsize = len(payload) + 26
    assert bsize <= 65536
    return (MAGIC + b"\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", bsize - 1) + payload +
            struct.pack("<II", zlib.crc32(chunk), len(chunk)))


def compress(data, level: int = 6, block_text: int = MAX_TEXT, threads: int = 0, strategy: int = zlib.Z_DEFAULT_STRATEGY,
             eof: bool = True) -> bytes:
    """data -> bgzf bytes (independent 64 KiB blocks; zlib drops the GIL, so blocks are compressed in parallel)"""
    import os

    mv = memoryview(data)
    jobs = [(mv[i:i + block_text], level, strategy) for i in range(0, len(mv), block_text)]
    if len(jobs) < 4:
        parts = [_one_block(j) for j in jobs]
    else:
        with ThreadPoolExecutor(threads or (os.cpu_count() or 1)) as ex:
            parts = list(ex.map(_one_block, jobs, chunksize=16))
    return b"".join(parts) + (EOF_BLOCK if eof else b"")


def inflate_host(buf, max_text: int) -> bytes:
    """the text of the whole blocks at the start of a bgzf buffer, until there are at least max_text bytes of it, inflated
    on the host and checked against each block's CRC-32 and ISIZE: only used to read the VCF preamble"""
    out, n, p = [], 0, 0
    while p < len(buf) and n < max_text:
        bs, isize = _block(buf, p)
        if bs == 0 or p + bs > len(buf):
            break
        text, why = C.create_string_buffer(isize), C.c_char_p()
        rc = _lib.lib().bvcf_bgzf_inflate(_addr(buf) + p, bs, text, isize, C.byref(why))
        if rc:
            raise ValueError("%s at byte %d" % (_reason(rc, why), p))
        out.append(text.raw)
        n += isize
        p += bs
    return b"".join(out)
