"""bgzf input on the host, without a GPU: the DEFLATE corpus of deflate_writer.py checked against zlib (before any GPU
decodes it), the one bgzf header rule (libbvcf's bvcf_bgzf.cpp) as both CLIs apply it, and members that claim ISIZE 0 checked instead of
skipped."""
import ctypes
import os
import random
import subprocess
import sys
import zlib

import pytest

import deflate_writer as D

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "bystro_vcf_b200", "bin", "bystro-vcf-b200")
PY = [sys.executable, "-m", "bystro_vcf_b200"]
VCF = (b"##fileformat=VCFv4.1\n##source=conformance\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n" +
       b"".join(b"1\t%d\t.\tA\tG\t.\tPASS\t.\n" % (100 + i) for i in range(50)))
# what the CLIs print when they refuse a bgzf input (before any device work)
REFUSALS = (b"bgzf", b"BC subfield", b"Not a VCF file")


def _cli(cmd, data):
    return subprocess.run(cmd, input=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE, cwd=ROOT, timeout=600)


# ---- the writer's streams against zlib ----

def test_writer_valid_streams_match_zlib():
    for name, payload, text in D.valid_cases():
        assert D.inflate(payload) == text, name
        assert len(text) <= D.MAX_TEXT and len(D.member(payload, text)) <= 65536, name  # a bgzf member's limits
    for n in D.TEXT_LENGTHS:
        payload, text = D.text_of_length(n)
        assert len(text) == n and D.inflate(payload) == text, n
    for seed in range(200):
        payload, text = D.random_member_payload(random.Random(seed))
        assert len(text) <= D.MAX_TEXT and D.inflate(payload) == text, seed


def test_writer_invalid_streams_are_refused_by_zlib():
    cases = D.invalid_cases()
    assert D.SINGLE_CODE_CASES <= {name for name, _, _ in cases}
    for name, payload, _ in cases:
        with pytest.raises(zlib.error):
            D.inflate(payload)
        with pytest.raises(zlib.error):
            zlib.decompress(payload, -15)


def test_writer_codes_reach_every_length():
    """the hand-made corpus really holds literal/length and distance codes of every length 1..15"""
    chain = D.random_lengths(random.Random(0), 16, deep=True)
    assert sorted(set(chain)) == list(range(1, 16))
    for _ in range(50):
        lens = D.random_lengths(random.Random(_), random.Random(_).randrange(2, 287))
        assert sum(1 << (15 - L) for L in lens) == 1 << 15 and max(lens) <= 15


# ---- one header rule ----

def _with_extra(extra_of, payload, text, flg=4):
    """a gzip member whose extra field is extra_of(BSIZE - 1) (its length must not depend on the value)"""
    import struct

    xlen = len(extra_of(0))
    total = 12 + xlen + len(payload) + 8
    return (b"\x1f\x8b\x08" + bytes([flg]) + b"\x00\x00\x00\x00\x00\xff" + struct.pack("<H", xlen) + extra_of(total - 1) +
            payload + struct.pack("<II", zlib.crc32(text), len(text)))


def _bc(v, slen=2):
    return b"BC" + bytes([slen, 0]) + (v & 0xFFFF).to_bytes(2, "little") + b"\x00" * (slen - 2)


def _header_table():
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    p = c.compress(VCF) + c.flush()
    sub = D.subfield
    return [
        ("bc-first", _with_extra(lambda v: _bc(v), p, VCF), True),
        ("bc-after-another-subfield", _with_extra(lambda v: sub(b"XY", b"abcd") + _bc(v), p, VCF), True),
        ("bc-after-an-empty-subfield", _with_extra(lambda v: sub(b"AB", b"") + _bc(v), p, VCF), True),
        ("xlen-more-than-6", _with_extra(lambda v: _bc(v) + sub(b"ZZ", b"0123456789"), p, VCF), True),
        ("two-bc-the-first-right", _with_extra(lambda v: _bc(v) + _bc(17), p, VCF), True),
        ("two-bc-the-first-too-small", _with_extra(lambda v: _bc(17) + _bc(v), p, VCF), False),
        ("bc-with-slen-4", _with_extra(lambda v: _bc(v, 4), p, VCF), False),
        ("bc-with-slen-4-then-bc", _with_extra(lambda v: _bc(v, 4) + _bc(v), p, VCF), True),
        ("stray-bytes-after-bc", _with_extra(lambda v: _bc(v) + b"\x00\x00", p, VCF), True),
        ("field-ends-inside-a-later-subfield", _with_extra(lambda v: _bc(v) + b"XY\x08\x00ab", p, VCF), True),
        ("field-ends-inside-bc", _with_extra(lambda v: _bc(v)[:5], p, VCF), False),
        ("field-ends-inside-a-subfield-around-bc", _with_extra(lambda v: b"XY\x0a\x00" + _bc(v), p, VCF), False),
        ("no-fextra", _with_extra(lambda v: _bc(v), p, VCF, flg=0), False),
    ]


@pytest.mark.parametrize("case", [c[0] for c in _header_table()])
def test_bgzf_header_parsers_agree(case, tmp_path):
    """the one header rule -- BC anywhere in the extra field, the first BC subfield with SLEN 2 inside the field -- as
    bgzf.is_bgzf / block_size / blocks, bvcf_bgzf_text_bytes (the library's walk) and the C++ CLI's refusals see it:
    they accept the same headers and agree on the block size"""
    from bystro_vcf_b200 import _lib, bgzf

    name, first, ok = next(c for c in _header_table() if c[0] == case)
    data = first + D.EOF_BLOCK
    assert bgzf.is_bgzf(data) is ok
    if ok:
        assert bgzf.block_size(data, 0) == len(first)
        assert [b[:2] for b in bgzf.blocks(data)] == [(0, len(first)), (len(first), len(D.EOF_BLOCK))]
    else:
        with pytest.raises(ValueError):
            bgzf.blocks(data)
    L = _lib.lib()
    text, n = ctypes.c_uint64(), ctypes.c_uint64()
    rc = L.bvcf_bgzf_text_bytes(data, len(data), ctypes.byref(text), ctypes.byref(n))
    assert (rc == 0) is ok, rc
    if ok:
        assert (text.value, n.value) == (len(VCF), 2)
    if os.path.exists(BIN):
        inp = tmp_path / "in.vcf.gz"
        inp.write_bytes(data)
        for r in (_cli([BIN, "--in", str(inp)], b""), _cli([BIN], data)):
            refused = r.returncode == 1 and any(m in r.stderr for m in REFUSALS)
            assert refused is not ok, (case, r.returncode, r.stderr[-400:])


# ---- members that claim ISIZE 0 ----

def _hidden(text=b"1\t7\t.\tC\tT\t.\tPASS\t.\n", crc=None):
    """a member whose text is `text` but whose trailer claims ISIZE 0"""
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    return D.member(c.compress(text) + c.flush(), text, crc=crc, isize=0)


def _empty_members():
    out = [D.EOF_BLOCK]
    for kind in ("stored", "fixed", "dynamic"):
        w = D.BitWriter()
        if kind == "stored":
            D.stored(w, b"", True)
        elif kind == "fixed":
            D.fixed(w, [], True)
        else:
            ll = [0] * 257
            ll[256] = 1
            D.dynamic(w, [], True, ll, [0])
        out.append(D.member(w.getvalue(), b""))
    return out


def test_blocks_check_members_that_claim_no_text():
    from bystro_vcf_b200 import bgzf

    good = bgzf.compress(VCF, block_text=300, eof=False)
    for e in _empty_members():  # empty members of every block type are fine
        assert len(bgzf.blocks(good + e + good + D.EOF_BLOCK)) == 2 * len(bgzf.blocks(good)) + 2
    for bad in (_hidden(), _hidden(crc=0), D.member(b"\x03\x00", b"", crc=1)):
        with pytest.raises(ValueError):
            bgzf.blocks(good + bad + D.EOF_BLOCK)


@pytest.mark.parametrize("where", ["preamble", "middle", "after-the-last-newline"])
def test_plan_groups_refuses_hidden_text(where):
    from bystro_vcf_b200 import bgzf

    parts = [bgzf.compress(VCF[i:i + 300], eof=False) for i in range(0, len(VCF), 300)]
    k = {"preamble": 0, "middle": len(parts) // 2, "after-the-last-newline": len(parts)}[where]
    data = b"".join(parts[:k]) + _hidden() + b"".join(parts[k:]) + D.EOF_BLOCK
    data_off = VCF.index(b"\n", VCF.index(b"#CHROM")) + 1
    plain = b"".join(parts) + D.EOF_BLOCK
    assert bgzf.plan_groups(plain, data_off, 1 << 16, 1 << 20)
    with pytest.raises(ValueError):
        bgzf.plan_groups(data, data_off, 1 << 16, 1 << 20)


def test_hidden_text_in_the_preamble_is_refused_by_both_clis(tmp_path):
    """a member inside the ## lines -- or the first member -- whose trailer claims ISIZE 0 but which inflates to text, or
    an empty first member with a wrong CRC-32: exit 1 before any device work, piped or from --in, with the bgzf refusal
    (the input is still told to be bgzf by its header, not taken for plain text)"""
    from bystro_vcf_b200 import bgzf

    head = VCF[:VCF.index(b"#CHROM")]
    for data in (bgzf.compress(head[:20], eof=False) + _hidden() + bgzf.compress(VCF[20:]),
                 _hidden() + bgzf.compress(VCF), D.member(b"\x03\x00", b"", crc=1) + bgzf.compress(VCF)):
        assert bgzf.is_bgzf(data)
        inp = tmp_path / "in.vcf.gz"
        inp.write_bytes(data)
        for cmd in [PY] + ([[BIN]] if os.path.exists(BIN) else []):
            for r in (_cli(cmd + ["--in", str(inp)], b""), _cli(cmd, data)):
                assert r.returncode == 1, (cmd, r.stderr[-400:])
                assert b"bgzf" in r.stderr and b"CRC-32" in r.stderr, (cmd, r.stderr[-400:])
                assert b"Not a VCF file" not in r.stderr and b"Traceback" not in r.stderr, (cmd, r.stderr[-400:])
