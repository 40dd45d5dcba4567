"""bgzf (block gzip, SAM spec 4.1: what bgzip / htslib write and what .vcf.gz files are) on the host side:
walking block headers, cutting a file into groups of whole blocks for the streaming path (plan_groups), and a writer
used by the tests and the bench to make compressed workloads.  The DEFLATE payloads themselves are inflated on the
GPU (csrc/bvcf_inflate.cuh: bvcf_submit_bgzf, bvcf_resident_inflate_bgzf)."""
from __future__ import annotations

import bisect
import struct
import zlib
from concurrent.futures import ThreadPoolExecutor
from typing import List, NamedTuple

MAGIC = b"\x1f\x8b\x08\x04"
EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
MAX_TEXT = 65280  # text bytes per block (bgzip's choice: the compressed block always fits 64 KiB)


def _header(buf, p: int) -> int:
    """The header of the bgzf block at buf[p]: a gzip member with FLG.FEXTRA whose extra field holds a BC subfield with
    SLEN 2 -- anywhere in the field (SAM spec 4.1).  The subfields are walked in order, one that runs past the end of the
    field ends the walk, and the first BC subfield gives BSIZE - 1.  The C++ host (bgzf_header) and the library
    (bgzf_walk) follow the same rule.  Returns the block size, or 0 when the header is not complete yet; raises
    ValueError when it is not a bgzf header."""
    if len(buf) - p < 18:
        return 0
    if buf[p] != 0x1F or buf[p + 1] != 0x8B or buf[p + 2] != 8 or not buf[p + 3] & 4:
        raise ValueError("not a bgzf block")
    xlen = buf[p + 10] | (buf[p + 11] << 8)
    if len(buf) - p < 12 + xlen:
        return 0
    q, end = p + 12, p + 12 + xlen
    while q + 4 <= end:
        slen = buf[q + 2] | (buf[q + 3] << 8)
        if q + 4 + slen > end:
            break
        if buf[q] == 66 and buf[q + 1] == 67 and slen == 2:
            bsize = (buf[q + 4] | (buf[q + 5] << 8)) + 1
            if bsize < 12 + xlen + 8:
                raise ValueError("bgzf block size %d is smaller than its header and trailer" % bsize)
            return bsize
        q += 4 + slen
    raise ValueError("gzip member without the bgzf BC subfield")


def is_bgzf(head) -> bool:
    """the first bytes of an input start with a whole bgzf header"""
    try:
        return _header(head, 0) > 0
    except ValueError:
        return False


def block_size(buf, p: int) -> int:
    """total size of the bgzf block that starts at buf[p] (0 when its header is not complete yet)"""
    return _header(buf, p)


def _payload_text(buf, p: int, bs: int) -> bytes:
    """the text of the bgzf block at buf[p:p + bs], inflated with zlib and checked against its CRC-32 and ISIZE"""
    xlen = buf[p + 10] | (buf[p + 11] << 8)
    try:
        text = zlib.decompress(bytes(buf[p + 12 + xlen:p + bs - 8]), -15)
    except zlib.error as e:
        raise ValueError("corrupt bgzf block at byte %d: %s" % (p, e)) from None
    crc, isize = struct.unpack("<II", bytes(buf[p + bs - 8:p + bs]))
    if len(text) != isize or zlib.crc32(text) != crc:
        raise ValueError("bgzf block at byte %d fails its CRC-32 / ISIZE check" % p)
    return text


def blocks(buf) -> List[tuple]:
    """(offset, size, ISIZE) of every block of a whole bgzf file.  A truncated last block or bytes that are not a bgzf
    block raise ValueError.  A block that claims ISIZE 0 (normally only the EOF block) is inflated here, and raises
    ValueError unless it holds no text and CRC-32 0: its text would otherwise be dropped without a word."""
    out = []
    p, n = 0, len(buf)
    while p < n:
        bs = block_size(buf, p)
        if bs == 0 or p + bs > n:
            raise ValueError("truncated bgzf block at byte %d" % p)
        isize = int.from_bytes(buf[p + bs - 4:p + bs], "little")
        if isize == 0:
            _payload_text(buf, p, bs)
        out.append((p, bs, isize))
        p += bs
    return out


class Group(NamedTuple):
    """A chunk of the streaming path: its text is inflate(buf[lo:hi])[skip:] + tail (bvcf_submit_bgzf)."""
    lo: int
    hi: int
    skip: int
    tail: bytes
    text: int  # bytes of inflate(buf[lo:hi])


LINE_TOO_LONG = "a single line exceeds the chunk capacity; raise --chunkBytes"


def plan_groups(buf, data_off: int, chunk_bytes: int, cap: int) -> List[Group]:
    """Cut a whole bgzf file into groups of whole blocks of about chunk_bytes of text, data lines from text offset
    data_off (the end of the #CHROM line) on.  The same rule as the C++ host's reader (csrc/bvcf_host.cpp):

    * a group's blocks are taken while its text is below chunk_bytes (empty blocks, the EOF block among them, add none);
      the first group starts at the block that holds text byte data_off, its skip is where data_off falls in it;
    * the line that crosses into the next group belongs to this one: its continuation -- the next group's text up to and
      including its first newline, inflated here -- is this group's tail, and the next group's skip jumps past it.  A next
      group with no newline at all is merged into this one;
    * the last group ends at the file's last newline (an unterminated last line is dropped, main.go:354-357): the blocks
      from the one holding that newline on are inflated here and left out, their text up to the newline is the tail;
    * a group whose text plus tail exceeds cap raises ValueError(LINE_TOO_LONG)."""
    bl = [b for b in blocks(buf) if b[2]]
    n = len(bl)
    starts = [0] * (n + 1)
    for i, b in enumerate(bl):
        starts[i + 1] = starts[i] + b[2]
    if data_off >= starts[n]:
        return []
    text_of = lambda i: _payload_text(buf, bl[i][0], bl[i][1])  # noqa: E731
    lo_of = lambda i: bl[i][0] if i < n else len(buf)  # noqa: E731
    b = bisect.bisect_right(starts, data_off) - 1
    skip = data_off - starts[b]
    out: List[Group] = []

    def take(i: int) -> int:  # end block of the group candidate that starts at block i
        e = i
        while e < n and starts[e] - starts[i] < chunk_bytes:
            e += 1
        return e

    def emit(lo_b: int, hi_b: int, skip_: int, tail: bytes) -> None:
        text = starts[hi_b] - starts[lo_b]
        if text + len(tail) > cap:
            raise ValueError(LINE_TOO_LONG)
        if text - skip_ + len(tail) > 0:
            out.append(Group(lo_of(lo_b), lo_of(hi_b), skip_, tail, text))

    while True:
        e = take(b)
        tail = None
        while e < n and tail is None:
            e2 = take(e)
            parts = []
            for j in range(e, e2):  # the continuation: inflated until its newline
                t = text_of(j)
                k = t.find(b"\n")
                if k >= 0:
                    parts.append(t[:k + 1])
                    tail = b"".join(parts)
                    break
                parts.append(t)
            if tail is None:
                e = e2  # no newline in the next group: it joins this one
        if tail is not None:
            emit(b, e, skip, tail)
            b, skip = e, len(tail)
            continue
        # the last group [b, n): it ends at the file's last newline
        f, tail = n, None
        while f > b and tail is None:
            f -= 1
            t = text_of(f)
            k = t.rfind(b"\n")
            if k >= 0:
                tail = t[:k + 1]
        if tail is None:
            return out  # nothing but an unterminated last line
        data_start = starts[b] + skip
        if data_start < starts[f]:
            emit(b, f, skip, tail)
        elif data_start - starts[f] < len(tail):  # the rest is inside the block of the last newline
            rest = tail[data_start - starts[f]:]
            if out:  # the previous group's tail takes it
                g = out.pop()
                lo_b = bisect.bisect_left(starts, starts[b] - g.text)
                emit(lo_b, b, g.skip, g.tail + rest)
            else:
                emit(f, f, 0, rest)
        return out


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
    out = []
    n = 0
    p = 0
    while p < len(buf) and n < max_text:
        bs = block_size(buf, p)
        if bs == 0 or p + bs > len(buf):
            break
        out.append(_payload_text(buf, p, bs))
        n += len(out[-1])
        p += bs
    return b"".join(out)
