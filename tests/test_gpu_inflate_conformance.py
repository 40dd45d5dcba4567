"""The GPU inflate kernel (csrc/bvcf_inflate.cuh) on DEFLATE streams zlib never writes: codes of every length 1..15,
hand-made precodes and code-length runs, degenerate codes, every length and distance symbol, many blocks per member,
text sizes around the kernel's CRC runs and flush pieces -- byte-identical to zlib; and every stream zlib refuses,
refused, with a trailer that would otherwise match.  The streams come from deflate_writer.py, whose valid and invalid
cases test_bgzf_conformance.py checks against zlib on the host."""
import gzip
import io
import os
import random
import subprocess
import sys
import zlib

import pytest

import deflate_writer as D

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "bystro_vcf_b200", "bin", "bystro-vcf-b200")
PY = [sys.executable, "-m", "bystro_vcf_b200"]
HDR = b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO"


@pytest.fixture(scope="module")
def tr():
    from bystro_vcf_b200 import Config, Transformer

    with Transformer(Config()) as t:
        t.set_header(HDR)
        t.resident_alloc(64 << 20, 1 << 20)
        yield t


def _inflate_many(tr, members):
    """[(member, text)] in one call per 32 MiB of text: the texts, back to back, exactly"""
    k = 0
    while k < len(members):
        batch, n = [], 0
        while k < len(members) and n + len(members[k][1]) <= 32 << 20:
            batch.append(members[k])
            n += len(members[k][1])
            k += 1
        comp = b"".join(m for m, _ in batch)
        want = b"".join(t for _, t in batch)
        assert tr.resident_inflate_bgzf(comp) == len(want)
        got = tr.resident_peek(0, len(want)) if want else b""
        if got != want:  # name the first member that differs
            off = 0
            for m, t in batch:
                assert got[off:off + len(t)] == t, "member of %d text bytes at text offset %d" % (len(t), off)
                off += len(t)
        assert got == want


def _refused(tr, member):
    from bystro_vcf_b200 import BvcfError

    with pytest.raises(BvcfError):
        tr.resident_inflate_bgzf(member)


def test_valid_corpus_matches_zlib(tr):
    """codes of every length (10 and 11 bits for literal/length, 9 and 10 for distance: the lookup tables' widths and
    one past them), 15-bit codes on the most frequent symbols, HCLEN 5 and 19, precode lengths up to 7, HLIT 257 / 286,
    HDIST 1 / 30, runs of 16 / 17 / 18 across the literal/length-distance boundary and 16 as the first distance entry,
    a single 1-bit distance code, no distance code, end-of-block-only blocks, every length and distance symbol with its
    extra bits, 258 both ways, 32,768, overlapping matches at distances 1..40, length-3 matches from beyond the 16 KiB
    ring, stored / fixed / dynamic / empty blocks in one member"""
    cases = D.valid_cases()
    _inflate_many(tr, [(D.member(p, t), t) for _, p, t in cases])
    for name, p, t in cases:  # one at a time as well: a member alone in its launch
        _inflate_many(tr, [(D.member(p, t), t)])


def test_text_sizes_and_crc(tr):
    """0..130 bytes (where the warp CRC's run length changes), the 4 KiB flush pieces and the 64 KiB maximum; one bit of
    the CRC-32 flipped is refused at each size, and 65,537 bytes are refused"""
    members = []
    for n in D.TEXT_LENGTHS:
        p, t = D.text_of_length(n)
        members.append((D.member(p, t), t))
    _inflate_many(tr, members)
    for n in D.TEXT_LENGTHS:
        p, t = D.text_of_length(n)
        _refused(tr, D.member(p, t, crc=zlib.crc32(t) ^ (1 << (n % 32))))
    p, t = D.text_of_length(65537)
    assert D.inflate(p) == t
    _refused(tr, D.member(p, t))


@pytest.mark.parametrize("case", [c[0] for c in D.invalid_cases()])
def test_invalid_stream_is_refused(tr, case):
    """each stream zlib refuses, alone in its call, with the CRC-32 and ISIZE of the text a decoder that missed the error
    would make"""
    name, p, t = next(c for c in D.invalid_cases() if c[0] == case)
    _refused(tr, D.member(p, t))


def test_trailer_only_refusals(tr):
    """a valid stream whose text is one byte longer or shorter than its ISIZE"""
    for n in (1, 100, 4096, 65535):
        p, t = D.text_of_length(n, seed=3)
        _refused(tr, D.member(p, t, isize=n + 1))
        _refused(tr, D.member(p, t, isize=n - 1))
        _refused(tr, D.member(p, t, isize=0))


_FUZZ_OFF = int(os.environ.get("BVCF_FUZZ_OFFSET", "0"))


@pytest.mark.parametrize("seed", range(_FUZZ_OFF, _FUZZ_OFF + int(os.environ.get("BVCF_FUZZ5_N", "3"))))
def test_random_members(tr, seed):
    """random stored / fixed / dynamic / empty block sequences with random complete codes of up to 15 bits: identical
    to zlib in one batch; a copy of each with one bit flipped is refused, or gives exactly what zlib gives"""
    rng = random.Random(seed * 7919 + 5)
    cases = [D.random_member_payload(rng) for _ in range(250)]
    _inflate_many(tr, [(D.member(p, t), t) for p, t in cases])
    for p, t in cases:
        if not p:
            continue
        bad = bytearray(p)
        bit = rng.randrange(8 * len(bad))
        bad[bit >> 3] ^= 1 << (bit & 7)
        d = zlib.decompressobj(-15)
        try:
            got = d.decompress(bytes(bad)) + d.flush()
            same = d.eof and got == t
        except zlib.error:
            same = False
        m = D.member(bytes(bad), t)
        if same:
            _inflate_many(tr, [(m, t)])
        else:
            _refused(tr, m)


def test_deflate_worst_case_literals(tr):
    """the GPU deflate at its largest output: bytes of 0x90 and more (9-bit literals) with almost no 4-byte repeats"""
    from bystro_vcf_b200 import bgzf

    rng = random.Random(77)
    data = bytes(rng.randrange(0x90, 0x100) for _ in range(300000))
    tr.resident_write_output(0, data)
    comp = tr.resident_download_bgzf(0, len(data))
    assert gzip.decompress(comp + bgzf.EOF_BLOCK) == data


def _cli(cmd, data):
    return subprocess.run(cmd, input=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE, cwd=ROOT, timeout=600)


def test_end_to_end_with_long_codes(chr1_sample, tmp_path):
    """chr1 lines re-encoded as bgzf with random codes of up to 15 bits: read_vcf (auto-detected, small chunks: groups
    and host-inflated tails), the C++ CLI from --in and from a pipe, and --bgzfOut in both CLIs give the plain run's
    rows; with one middle member's ISIZE set to 0 both CLIs exit 1"""
    from bystro_vcf_b200 import Config, bgzf, read_vcf

    vcf = chr1_sample
    comp = D.bgzf_file(vcf, random.Random(11))
    assert gzip.decompress(comp) == vcf
    c = Config()
    plain = io.BytesIO()
    read_vcf(c, io.BytesIO(vcf), plain)
    assert plain.getvalue().count(b"\n") > 300
    c.chunkBytes = 1 << 16
    out = io.BytesIO()
    read_vcf(c, io.BytesIO(comp), out)
    assert out.getvalue() == plain.getvalue()
    inp = tmp_path / "in.vcf.gz"
    inp.write_bytes(comp)
    hosts = [PY] + ([[BIN, "--chunkBytes", str(1 << 16)]] if os.path.exists(BIN) else [])
    for cmd in hosts:
        ref = _cli(cmd, vcf)  # the plain-text run: the TSV header line, then the rows
        assert ref.returncode == 0 and ref.stdout.endswith(plain.getvalue()), ref.stderr.decode()[-2000:]
        for flags in ([], ["--bgzfOut"]):
            for r in (_cli(cmd + flags + ["--in", str(inp)], b""), _cli(cmd + flags, comp)):
                assert r.returncode == 0, (cmd, flags, r.stderr.decode()[-2000:])
                assert (gzip.decompress(r.stdout) if flags else r.stdout) == ref.stdout, (cmd, flags)
    # a middle member whose ISIZE claims no text
    blocks = bgzf.blocks(comp)
    off, bs, _ = blocks[len(blocks) // 2]
    bad = bytearray(comp)
    bad[off + bs - 4:off + bs] = b"\x00\x00\x00\x00"
    inp.write_bytes(bytes(bad))
    for cmd in hosts:
        for flags in ([], ["--bgzfOut"]):
            for r in (_cli(cmd + flags + ["--in", str(inp)], b""), _cli(cmd + flags, bytes(bad))):
                assert r.returncode == 1, (cmd, flags, r.stderr.decode()[-2000:])
