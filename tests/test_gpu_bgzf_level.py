"""bgzf output at levels 2..9 (bvcf_deflate_dyn_kernel: a bounded multi-candidate search, lazy matching from level 4,
dynamic Huffman codes built on the device): zlib and the GPU inflate read it back, the block type is the cheapest of
stored / fixed / dynamic, overlong codes are limited to 15 bits, degenerate alphabets stay valid, the output is
deterministic and within 10 % of zlib -6, level 1 is bvcf_resident_download_bgzf byte for byte, and both CLIs take
--bgzfLevel end to end."""
import ctypes as C
import gzip
import heapq
import itertools
import os
import random
import zlib

import pytest

from test_gpu_parity import _cfg
from test_host_drivers import BIN, PY, _cli, _vcf

pytestmark = pytest.mark.gpu

SLICE = 49152
ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]


def _members(comp):
    from bystro_vcf_b200 import bgzf

    out, p = [], 0
    while p < len(comp):
        bs = bgzf.block_size(comp, p)
        assert bs > 0 and p + bs <= len(comp)
        out.append(comp[p:p + bs])
        p += bs
    return out


def _check_members(comp, text_len):
    ms = _members(comp)
    assert len(ms) == -(-text_len // SLICE)
    for m in ms:
        assert int.from_bytes(m[-4:], "little") <= SLICE
    return ms


class _Bits:
    def __init__(self, b):
        self.b, self.p = b, 0

    def get(self, n):
        v = 0
        for i in range(n):
            v |= ((self.b[self.p >> 3] >> (self.p & 7)) & 1) << i
            self.p += 1
        return v


def _first_block(member):
    """BTYPE of the member's first block and, for a dynamic one, its literal/length code lengths (RFC 1951 3.2.7)"""
    r = _Bits(member[18:])
    r.get(1)
    bt = r.get(2)
    if bt != 2:
        return bt, None
    hlit, hdist, hclen = r.get(5) + 257, r.get(5) + 1, r.get(4) + 4
    pl = [0] * 19
    for i in range(hclen):
        pl[ORDER[i]] = r.get(3)
    codes, code = {}, 0
    for ln in range(1, 8):
        for s in range(19):
            if pl[s] == ln:
                codes[(ln, code)] = s
                code += 1
        code <<= 1
    out = []
    while len(out) < hlit + hdist:
        c = ln = 0
        while (ln, c) not in codes:
            c, ln = (c << 1) | r.get(1), ln + 1
            assert ln <= 7
        s = codes[(ln, c)]
        if s < 16:
            out.append(s)
        elif s == 16:
            out += [out[-1]] * (3 + r.get(2))
        elif s == 17:
            out += [0] * (3 + r.get(3))
        else:
            out += [0] * (11 + r.get(7))
    return bt, out[:hlit]


def _huffman_depth(freqs):
    """the longest code of an unlimited Huffman code for these frequencies"""
    h = [(f, i) for i, f in enumerate(freqs) if f]
    heapq.heapify(h)
    par, ids = {}, itertools.count(len(freqs))
    while len(h) > 1:
        (f1, a), (f2, b) = heapq.heappop(h), heapq.heappop(h)
        k = next(ids)
        par[a] = par[b] = k
        heapq.heappush(h, (f1 + f2, k))

    def depth(x):
        n = 0
        while x in par:
            x, n = par[x], n + 1
        return n

    return max(depth(i) for i, f in enumerate(freqs) if f)


def _fibonacci_slice(n=SLICE, seed=0):
    """n bytes in which no 4-byte string repeats (so every byte is a literal), drawn with Fibonacci weights for 14 bytes
    and flat ones for 64 more: the literal histogram's unlimited Huffman code is deeper than 15 bits"""
    fib = [1, 1]
    while len(fib) < 14:
        fib.append(fib[-1] + fib[-2])
    weights = fib + [fib[-1]] * 64
    syms = list(range(len(weights)))
    rng, seen, out = random.Random(seed), set(), bytearray()
    while len(out) < n:
        for s in rng.choices(syms, weights=weights, k=16):
            g = bytes(out[-3:]) + bytes([s])
            if len(out) < 3 or g not in seen:
                break
        else:
            continue
        if len(out) >= 3:
            seen.add(g)
        out.append(s)
    return bytes(out)


def _de_bruijn(k, n):
    """B(k, n) over bytes 'a'.. (every n-byte string over k letters exactly once, cyclically)"""
    a, seq = [0] * k * n, []

    def db(t, p):
        if t > n:
            if n % p == 0:
                seq.extend(a[1:p + 1])
        else:
            a[t] = a[t - p]
            db(t + 1, p)
            for j in range(a[t - p] + 1, k):
                a[t] = j
                db(t + 1, t)

    db(1, 1)
    return bytes(97 + x for x in seq)


@pytest.fixture(scope="module")
def rows_tr(chr1_fixture):
    """the chr1 fixture's rows (--keepId --keepInfo) resident in a Transformer's output region"""
    from bystro_vcf_b200 import Config, Transformer, parse_preamble

    vcf = chr1_fixture[:40 << 20].rsplit(b"\n", 1)[0] + b"\n"
    w, chrom, off = parse_preamble(vcf)
    body = vcf[off:]
    c = Config()
    c.allowedFilters = {"PASS": True, ".": True}
    c.keepID = c.keepInfo = True
    with Transformer(c, eol_width=w) as tr:
        tr.set_header(chrom)
        tr.resident_alloc(len(body), len(body) // 4 + (1 << 20))
        tr.resident_upload(0, body)
        stats, _ = tr.resident_run(len(body))
        n = stats["out_bytes"]
        yield tr, tr.resident_download(0, n)


@pytest.fixture(scope="module")
def raw_tr():
    """a Transformer whose output region takes arbitrary bytes"""
    from bystro_vcf_b200 import Transformer

    with Transformer(_cfg()) as tr:
        tr.set_header(b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO")
        tr.resident_alloc(1 << 20, 1 << 20)
        yield tr


def _deflate(tr, data, level):
    from bystro_vcf_b200 import bgzf

    tr.resident_write_output(0, data)
    comp = tr.resident_download_bgzf(0, len(data), level)
    assert gzip.decompress(comp + bgzf.EOF_BLOCK) == data
    _check_members(comp, len(data))
    return comp


@pytest.mark.parametrize("level", [2, 6, 9])
def test_round_trip_through_zlib(rows_tr, level):
    """zlib checks every CRC-32 and ISIZE and refuses over-subscribed or otherwise invalid codes"""
    from bystro_vcf_b200 import bgzf

    tr, rows = rows_tr
    n = len(rows)
    comp = tr.resident_download_bgzf(0, n, level)
    assert gzip.decompress(comp + bgzf.EOF_BLOCK) == rows
    _check_members(comp, n)
    for o, ln in ((0, 1), (3, SLICE - 1), (5, SLICE), (7, SLICE + 1), (12345, 200001)):
        part = tr.resident_download_bgzf(o, ln, level)
        assert gzip.decompress(part + bgzf.EOF_BLOCK) == rows[o:o + ln]
        _check_members(part, ln)


def test_gpu_inflate_reads_level_6(rows_tr):
    """both directions on the device: the level-6 members inflated by bvcf_resident_inflate_bgzf give the rows back"""
    from bystro_vcf_b200 import Transformer

    tr, rows = rows_tr
    comp = tr.resident_download_bgzf(0, len(rows), 6)
    with Transformer(_cfg()) as t2:
        t2.set_header(b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO")
        t2.resident_alloc(len(rows) + (1 << 20), 1 << 20)
        assert t2.resident_inflate_bgzf(comp, 0) == len(rows)
        assert t2.resident_peek(0, len(rows)) == rows


def test_block_types(rows_tr, raw_tr):
    """row text gets dynamic codes (BTYPE 10); random bytes get stored blocks (BTYPE 00), never bigger than
    header + 5 + text + trailer"""
    tr, rows = rows_tr
    comp = tr.resident_download_bgzf(0, len(rows), 6)
    assert all(_first_block(m)[0] == 2 for m in _members(comp))
    rng = random.Random(41)
    data = bytes(rng.randrange(256) for _ in range(120000))
    for m in _members(_deflate(raw_tr, data, 6)):
        assert _first_block(m)[0] == 0 and len(m) <= SLICE + 5 + 26


@pytest.mark.parametrize("level", [2, 6])
def test_length_limited_codes(raw_tr, level):
    """a slice whose literal histogram wants codes deeper than 15 bits: the emitted code has 15-bit lengths, no more"""
    data = _fibonacci_slice()
    assert len({data[i:i + 4] for i in range(len(data) - 3)}) == len(data) - 3  # no match possible: all literals
    freqs = [data.count(bytes([b])) for b in range(256)] + [1]  # + end of block
    assert _huffman_depth(freqs) > 15
    (m,) = _members(_deflate(raw_tr, data, level))
    bt, lens = _first_block(m)
    assert bt == 2 and max(lens) == 15


@pytest.mark.parametrize("data", [
    b"A" * 150000,                       # one literal, one distance code
    _de_bruijn(16, 4)[:SLICE],           # no match at all: zero distance codes, 16 literals
    b"0|0\t1|1\t" * 20000,
    b"x",
    b"ab" * 3,
], ids=["one-byte", "de-bruijn", "genotypes", "single", "short"])
@pytest.mark.parametrize("level", [2, 4, 9])
def test_degenerate_alphabets(raw_tr, data, level):
    _deflate(raw_tr, data, level)


def test_ratio_against_zlib_and_level_1(rows_tr):
    """level 6 within 10 % of zlib -6 on the same 48 KiB slices, and at most 3/4 of level 1"""
    tr, rows = rows_tr
    n = len(rows)
    l6 = len(tr.resident_download_bgzf(0, n, 6))
    l1 = len(tr.resident_download_bgzf(0, n, 1))
    z6 = 0
    for o in range(0, n, SLICE):
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        z6 += len(c.compress(rows[o:o + SLICE]) + c.flush()) + 26  # + the bgzf header and trailer
    print("rows %d B: level 6 %d B (%.3f of zlib -6's %d B), level 1 %d B (level 6 = %.3f of it)"
          % (n, l6, l6 / z6, z6, l1, l6 / l1))
    assert l6 <= 1.10 * z6, (l6, z6)
    assert l6 <= 0.75 * l1, (l6, l1)


def test_deterministic(rows_tr):
    tr, rows = rows_tr
    assert tr.resident_download_bgzf(0, len(rows), 6) == tr.resident_download_bgzf(0, len(rows), 6)


def test_level_1_is_the_level_1_entry_point(rows_tr):
    """bvcf_resident_download_bgzf_level(..., 1, ...) == bvcf_resident_download_bgzf; levels 0 and 10 are refused"""
    tr, rows = rows_tr
    n = len(rows)
    cap = n + n // 4 + (1 << 16)
    a, b = C.create_string_buffer(cap), C.create_string_buffer(cap)
    na, nb = C.c_size_t(), C.c_size_t()
    assert tr._L.bvcf_resident_download_bgzf(tr._ctx, 0, n, a, cap, C.byref(na)) == 0
    assert tr._L.bvcf_resident_download_bgzf_level(tr._ctx, 0, n, 1, b, cap, C.byref(nb)) == 0
    assert na.value == nb.value and a.raw[:na.value] == b.raw[:nb.value]
    for bad in (0, 10, -1):
        assert tr._L.bvcf_resident_download_bgzf_level(tr._ctx, 0, n, bad, b, cap, C.byref(nb)) == -1  # BVCF_E_ARG


def _hosts():
    return [("python", PY)] + ([("cpp", [BIN])] if os.path.exists(BIN) else [])


@pytest.mark.parametrize("host", ["cpp", "python"])
def test_cli_level_1_flag_changes_no_byte(tmp_path, host):
    cmds = dict(_hosts())
    if host not in cmds:
        pytest.skip("the C++ host is not built")
    vcf = _vcf(20, 3000)
    outs = []
    for extra in ([], ["--bgzfLevel", "1"]):
        r = _cli(cmds[host] + ["--keepId", "--bgzfOut"] + extra, vcf)
        assert r.returncode == 0, r.stderr.decode()[-2000:]
        outs.append(r.stdout)
    assert outs[0] == outs[1]


@pytest.mark.parametrize("route", ["pipe", "file"])
@pytest.mark.parametrize("host", ["cpp", "python"])
def test_cli_level_6_end_to_end(tmp_path, host, route):
    """--in x.vcf.gz --bgzfOut --bgzfLevel 6 with --dosageOutput and --sample: the rows, the Arrow file, the sample list
    and the log lines of the plain run"""
    import pyarrow as pa

    from bystro_vcf_b200 import bgzf

    cmds = dict(_hosts())
    if host not in cmds:
        pytest.skip("the C++ host is not built")
    vcf = _vcf(40, 6000)
    data = bgzf.compress(vcf, block_text=9000)
    inp = tmp_path / "in.vcf.gz"
    inp.write_bytes(data)
    got = {}
    for mode, extra in (("plain", []), ("level6", ["--bgzfOut", "--bgzfLevel", "6"])):
        d, s = tmp_path / ("d_%s.feather" % mode), tmp_path / ("s_%s.txt" % mode)
        cmd = cmds[host] + ["--keepId", "--keepInfo", "--dosageOutput", str(d), "--sample", str(s)] + extra
        r = _cli(cmd + (["--in", str(inp)] if route == "file" else []), b"" if route == "file" else data)
        assert r.returncode == 0, r.stderr.decode()[-2000:]
        rows = r.stdout if mode == "plain" else gzip.decompress(r.stdout)
        got[mode] = (rows, d.read_bytes(), s.read_bytes(), r.stderr.decode().split("\n"))
    rows, dos, samples, log = got["plain"]
    assert rows.count(b"\n") > 1000 and len([x for x in log if x]) > 500
    assert got["level6"][0] == rows
    assert got["level6"][2:] == got["plain"][2:]
    read = lambda b: pa.ipc.open_file(pa.py_buffer(b)).read_all()  # noqa: E731
    assert read(got["level6"][1]).equals(read(dos))
