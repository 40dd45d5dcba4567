"""--regions / --regionsFile without a GPU: the flag grammar and every refusal in both CLIs, before any device work; and
bvcf_index_spans (host only) on tabix and CSI indexes written here by a small writer that follows the SAM spec (5.1-5.2)
and CSIv1, as htslib fills them: the spans are sorted, disjoint, and cover every record whose POS is in a region."""
import ctypes as C
import os
import random
import struct
import subprocess
import sys

import pytest

from bystro_vcf_b200 import bgzf, host

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAX = (1 << 63) - 1
VCF_HEAD = b"##fileformat=VCFv4.1\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n"


def _clis():
    cmds = [[sys.executable, "-m", "bystro_vcf_b200"]]
    binary = os.path.join(ROOT, "bystro_vcf_b200", "bin", "bystro-vcf-b200")
    if os.path.exists(binary):
        cmds.append([binary])
    return cmds


# ---- flags ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("arg,exp", [
    ("chr1", [(b"chr1", 1, MAX)]),
    ("chr1:5", [(b"chr1", 5, 5)]),
    ("chr1:5-9", [(b"chr1", 5, 9)]),
    ("chr1:5-", [(b"chr1", 5, MAX)]),
    ("1:007-8,2,HLA-A*01:01:3-4", [(b"1", 7, 8), (b"2", 1, MAX), (b"HLA-A*01:01", 3, 4)]),
])
def test_regions_grammar(arg, exp):
    assert host.setup(["--regions", arg]).regions == exp
    assert host.setup(["-regions=" + arg, "--keepId"]).regions == exp
    for cmd in _clis():  # gets past the flags to the input (not a VCF here)
        r = subprocess.run(cmd + ["--regions", arg], input=b"hello\n", capture_output=True, cwd=ROOT)
        assert r.returncode == 1 and b"Not a VCF file" in r.stderr, (cmd, r.stderr)


def test_no_flag_no_regions():
    assert host.setup([]).regions is None


def test_regions_file_and_union(tmp_path):
    bed = tmp_path / "r.bed"
    bed.write_bytes(b"track name=t\nbrowser position chr1\n# comment\n\nchr1\t0\t10\tname\t0\t+\n"
                    b"chr2 99 100\nchr3\t5\t5\n2\t1\t2\r\n")
    c = host.setup(["--regions", "chrX:3", "--regionsFile", str(bed)])
    assert c.regions == [(b"chrX", 3, 3), (b"chr1", 1, 10), (b"chr2", 100, 100), (b"2", 2, 2)]


@pytest.mark.parametrize("flags,msg", [
    (["--regions", ""], b'--regions: malformed region ""'),
    (["--regions", "chr1,"], b'--regions: malformed region ""'),
    (["--regions", ":5"], b'--regions: malformed region ":5"'),
    (["--regions", "chr1:x"], b'--regions: malformed region "chr1:x"'),
    (["--regions", "chr1:0"], b'--regions: malformed region "chr1:0"'),
    (["--regions", "chr1:0-5"], b'--regions: malformed region "chr1:0-5"'),
    (["--regions", "chr1:9-5"], b'--regions: malformed region "chr1:9-5"'),
    (["--regions", "chr1:-5"], b'--regions: malformed region "chr1:-5"'),
    (["--regions", "chr1:5-x"], b'--regions: malformed region "chr1:5-x"'),
    (["--regions", "chr1:99999999999999999999"], b"--regions: malformed region"),
    (["--regionsFile", "/nonexistent/r.bed"], b"--regionsFile: /nonexistent/r.bed: "),
    (["--regionsFile", "@2col"], b"line 2: fewer than three columns"),
    (["--regionsFile", "@backwards"], b"line 1: start > end"),
    (["--regionsFile", "@text"], b"line 1: start and end must be non-negative integers"),
    (["--regionsFile", "@empty"], b"--regionsFile: no intervals"),
])
def test_refusals_before_any_device_work(flags, msg, tmp_path):
    beds = {"@2col": b"chr1\t1\t2\nchr1\t5\n", "@backwards": b"chr1\t9\t5\n", "@text": b"chr1\tx\t5\n",
            "@empty": b"# nothing\n"}
    flags = list(flags)
    if flags[-1] in beds:
        p = tmp_path / "r.bed"
        p.write_bytes(beds[flags[-1]])
        flags[-1] = str(p)
    with pytest.raises(ValueError, match=msg.decode().replace("*", r"\*")):
        host.setup(flags)
    for cmd in _clis():
        # a valid VCF on stdin: only the flag check can stop the run before the device is needed
        r = subprocess.run(cmd + flags, input=VCF_HEAD, capture_output=True, cwd=ROOT)
        assert r.returncode == 1, (cmd, r.stderr)
        assert r.stderr.strip().count(b"\n") == 0 and msg in r.stderr, (cmd, r.stderr)
        assert r.stdout == b""


# ---- a tabix / CSI writer ---------------------------------------------------------------------------------------------

def reg2bin(beg, end, min_shift, depth):
    """SAM spec 5.3 (0-based, half-open), generalised to CSI's min_shift and depth"""
    end -= 1
    s, t = min_shift, ((1 << depth * 3) - 1) // 7
    for l in range(depth, 0, -1):
        if beg >> s == end >> s:
            return t + (beg >> s)
        s += 3
        t -= 1 << ((l - 1) * 3)
    return 0


def records(seed, contigs, n, max_pos, block_text):
    """a sorted VCF with long deletions among its records, its bgzf bytes, and each record's (contig, POS, REF length,
    virtual offsets [start, end))"""
    rng = random.Random(seed)
    lines, meta = [], []
    for c in contigs:
        for p in sorted(rng.sample(range(1, max_pos), n)):
            rlen = rng.choice([1, 1, 1, 2, 40, 20000])
            lines.append(b"%s\t%d\t.\t%s\tA\t.\tPASS\t.\n" % (c, p, b"A" * rlen))
            meta.append((c, p, rlen))
    text = VCF_HEAD + b"".join(lines)
    comp = bgzf.compress(text, block_text=block_text)
    coff = [b[0] for b in bgzf.blocks(comp)]

    def voff(t):  # text offset -> virtual offset; a record ends one past its last byte, in the block of that byte
        return coff[t // block_text] << 16 | (t % block_text)

    out, t = [], len(VCF_HEAD)
    for line, m in zip(lines, meta):
        out.append(m + (voff(t), voff(t + len(line) - 1) + 1))
        t += len(line)
    return comp, out


def write_index(recs, contigs, csi=False, min_shift=14, depth=5):
    """the index htslib would write: chunks per bin (consecutive records merged), the linear index of the first record
    overlapping each window with empty windows filled from the left, and (CSI) a bin's loffset from the linear index
    at its first window"""
    names = b"".join(c + b"\0" for c in contigs)
    conf = struct.pack("<6i", 2, 1, 2, 0, ord("#"), 0) + struct.pack("<i", len(names)) + names
    body = b""
    for c in contigs:
        bins, lin = {}, {}
        for (rc, p, rlen, vb, ve) in (r for r in recs if r[0] == c):
            beg, end = p - 1, p - 1 + rlen
            ch = bins.setdefault(reg2bin(beg, end, min_shift, depth), [])
            if ch and ch[-1][1] == vb:
                ch[-1][1] = ve
            else:
                ch.append([vb, ve])
            for w in range(beg >> min_shift, ((end - 1) >> min_shift) + 1):
                lin.setdefault(w, vb)
        n_lin = max(lin) + 1
        li = [0] * n_lin
        prev = min(lin.values())
        for w in range(n_lin):
            prev = li[w] = lin.get(w, prev)
        body += struct.pack("<i", len(bins))
        for b, ch in sorted(bins.items()):
            body += struct.pack("<I", b)
            if csi:
                l = next(l for l in range(depth, -1, -1) if b >= ((1 << 3 * l) - 1) // 7)
                bot = (b - ((1 << 3 * l) - 1) // 7) << 3 * (depth - l)
                body += struct.pack("<Q", li[bot] if bot < n_lin else 0)
            body += struct.pack("<i", len(ch)) + b"".join(struct.pack("<QQ", *x) for x in ch)
        if not csi:
            body += struct.pack("<i", n_lin) + b"".join(struct.pack("<Q", x) for x in li)
    if csi:
        return b"CSI\1" + struct.pack("<3i", min_shift, depth, len(conf)) + conf + struct.pack("<i", len(contigs)) + body
    return b"TBI\1" + struct.pack("<i", len(contigs)) + conf + body


def spans(index, regions, cap=1 << 16):
    from bystro_vcf_b200 import _lib

    L = _lib.lib()
    n = len(regions)
    names = (C.c_char_p * max(n, 1))(*[r[0] for r in regions])
    beg = (C.c_int64 * max(n, 1))(*[r[1] for r in regions])
    end = (C.c_int64 * max(n, 1))(*[r[2] for r in regions])
    out = (C.c_uint64 * (2 * max(cap, 1)))()
    got = C.c_size_t()
    rc = L.bvcf_index_spans(index, len(index), names, beg, end, n, out, cap, C.byref(got))
    return rc, [(out[2 * k], out[2 * k + 1]) for k in range(min(got.value, cap))], got.value


def check_cover(recs, regions, sp):
    for a, b in zip(sp, sp[1:]):
        assert a[0] < a[1] <= b[0], "spans sorted and disjoint"
    for (c, p, rlen, vb, ve) in recs:
        if any(c == rc and rb <= p <= re for rc, rb, re in regions):
            assert any(s <= vb and ve <= e for s, e in sp), (c, p)


CONTIGS = [b"1", b"10", b"chr1"]
INDEXES = {"tbi": dict(), "csi": dict(csi=True), "csi-10-7": dict(csi=True, min_shift=10, depth=7),
           "csi-16-4": dict(csi=True, min_shift=16, depth=4)}


@pytest.mark.parametrize("kind", list(INDEXES))
def test_index_spans_cover_every_record_in_the_regions(kind):
    comp, recs = records(1, CONTIGS, 1500, 3_000_000, 3000)
    idx = write_index(recs, CONTIGS, **INDEXES[kind])
    rng = random.Random(2)
    edges = [16384 * k for k in (1, 2, 7, 8, 64)] + [1 << 17, 1 << 20, 1 << 23]
    sets = [[(rng.choice(CONTIGS), b, b + rng.randint(0, 50000)) for b in rng.sample(range(1, 3_000_000), 20)],
            [(c, e + d, e + d) for c in CONTIGS for e in edges for d in (-1, 0, 1)],
            [(c, e - 5, e + 5) for c in CONTIGS for e in edges],
            [(r[0], r[1], r[1]) for r in rng.sample(recs, 200)],
            [(b"10", 1, MAX)], [(b"1", 2_999_000, MAX), (b"chr1", 1, 3)]]
    whole = len(comp) << 16
    for regions in sets:
        rc, sp, n = spans(idx, regions)
        assert rc == 0 and n == len(sp)
        check_cover(recs, regions, sp)
        if len(regions) < 40 and regions[0][2] != MAX:
            assert sum((e >> 16) - (s >> 16) for s, e in sp) < whole // 4, "small regions read a small part"


def test_index_spans_absent_contig_cap_and_malformed():
    comp, recs = records(3, CONTIGS, 300, 3_000_000, 2000)
    for kind in ("tbi", "csi"):
        idx = write_index(recs, CONTIGS, **INDEXES[kind])
        assert spans(idx, [(b"chr10", 1, MAX), (b"2", 1, 5)]) == (0, [], 0)
        assert spans(idx, []) == (0, [], 0)
        regions = [(r[0], r[1], r[1]) for r in recs[::25]]
        rc, sp, n = spans(idx, regions)
        assert rc == 0 and n > 2
        rc, _, need = spans(idx, regions, cap=n - 1)
        assert rc == -5 and need == n  # BVCF_E_TOO_LARGE, and the count it takes
        assert spans(idx, regions, cap=n)[1] == sp
        for bad in (idx[:3], idx[:len(idx) // 2], idx[:40], b"TBJ\1" + idx[4:], bytes(64),
                    idx[:4] + struct.pack("<i", -1) + idx[8:]):
            assert spans(bad, regions)[0] == -1  # BVCF_E_ARG
        for bad_region in ([(b"1", 0, 5)], [(b"1", 6, 5)], [(b"", 1, 5)]):
            assert spans(idx, bad_region)[0] == -1


def index_of(text: bytes, block_text: int, level: int = 6, **kw) -> bytes:
    """the index of bgzf.compress(text, level, block_text): every data line whose POS is a number is placed"""
    comp = bgzf.compress(text, level=level, block_text=block_text)
    coff = [b[0] for b in bgzf.blocks(comp)]

    def voff(t):
        return coff[t // block_text] << 16 | (t % block_text)

    t = text.index(b"\n", text.index(b"\n#CHROM") + 1) + 1
    recs, contigs = [], []
    for line in text[t:].splitlines(keepends=True):
        f = line.split(b"\t", 4)
        if len(f) > 3 and f[1].isdigit() and 0 < int(f[1]) < 1 << 29:
            if f[0] not in contigs:
                contigs.append(f[0])
            recs.append((f[0], int(f[1]), len(f[3]), voff(t), voff(t + len(line) - 1) + 1))
        t += len(line)
    return write_index(recs, contigs, **kw)
