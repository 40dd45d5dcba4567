"""bgzf.plan_groups, the host rule that cuts a .vcf.gz into groups of whole blocks for bvcf_submit_bgzf: every group's
text is inflate(comp)[skip:] + tail, ends with a newline, and the groups give back the data region exactly."""
import random
import zlib

import pytest

from bystro_vcf_b200 import bgzf

PRE = b"##fileformat=VCFv4.1\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n"
_ALPHA = bytes(b"ACGT\t0|1."[i % 9] for i in range(256))


def _inflate(buf) -> bytes:
    out, p = [], 0
    while p < len(buf):
        bs = bgzf.block_size(buf, p)
        xlen = buf[p + 10] | (buf[p + 11] << 8)
        out.append(zlib.decompress(bytes(buf[p + 12 + xlen:p + bs - 8]), -15))
        p += bs
    return b"".join(out)


def _random_text(rng, max_line):
    lines = []
    for _ in range(rng.randrange(0, 40)):
        n = rng.choice([1, 2, 9, 80, 1000, 30000, max_line])
        eol = b"\r\n" if rng.random() < 0.3 else b"\n"
        lines.append(rng.randbytes(max(0, n - len(eol))).translate(_ALPHA) + eol)
    data = PRE + b"".join(lines)
    if rng.random() < 0.5:
        data += b"1\t5\tunterminated" * rng.randrange(1, 3000)
    return data


def _check(comp, data, groups):
    end = max(data.rfind(b"\n") + 1, len(PRE))
    got, prev = [], None
    for g in groups:
        t = _inflate(comp[g.lo:g.hi])
        assert len(t) == g.text and g.skip <= g.text
        text = t[g.skip:] + g.tail
        assert text.endswith(b"\n")
        if prev is not None:
            assert g.skip == len(prev.tail)
        got.append(text)
        prev = g
    assert b"".join(got) == data[len(PRE):end]


@pytest.mark.parametrize("seed", range(12))
def test_groups_rebuild_the_data_region(seed):
    rng = random.Random(seed)
    for _ in range(6):
        data = _random_text(rng, 200000)
        block_text = rng.choice([1, 17, 777, 4096, 20000, 65280]) if len(data) < 150000 else rng.choice([777, 20000, 65280])
        comp = bgzf.compress(data, level=rng.choice([0, 1, 6]), block_text=block_text)
        chunk = rng.choice([1 << 16, 100000, 1 << 18, 1 << 20])
        groups = bgzf.plan_groups(comp, len(PRE), chunk, 1 << 30)
        _check(comp, data, groups)


def test_line_longer_than_a_group_is_merged_or_refused():
    rng = random.Random(7)
    long_line = rng.randbytes(300000).translate(_ALPHA) + b"\n"
    data = PRE + b"1\t1\tx\n" * 5000 + long_line + b"1\t2\ty\n" * 5000
    comp = bgzf.compress(data, block_text=5000)
    groups = bgzf.plan_groups(comp, len(PRE), 1 << 16, 1 << 30)
    _check(comp, data, groups)
    assert len(groups) > 2 and any(g.text + len(g.tail) > len(long_line) for g in groups)  # merged, whole in one group
    with pytest.raises(ValueError, match="a single line exceeds the chunk capacity"):
        bgzf.plan_groups(comp, len(PRE), 1 << 16, 200000)


def test_preamble_in_later_blocks_and_empty_data():
    data = PRE + b"1\t1\tx\n" * 100
    comp = bgzf.compress(data, block_text=7)  # the #CHROM line ends several blocks in
    _check(comp, data, bgzf.plan_groups(comp, len(PRE), 1 << 16, 1 << 30))
    assert bgzf.plan_groups(bgzf.compress(PRE), len(PRE), 1 << 16, 1 << 30) == []
    assert bgzf.plan_groups(bgzf.compress(PRE + b"1\t1\tno newline"), len(PRE), 1 << 16, 1 << 30) == []


def test_truncated_or_garbage_input_is_an_error():
    data = PRE + b"1\t1\tx\n" * 20000
    comp = bgzf.compress(data, block_text=4000)
    for bad in (comp[:-5], comp[:len(comp) - 28 - 100], comp + b"trailing garbage", comp + b"\x1f\x8b\x08\x04\x00"):
        with pytest.raises(ValueError):
            bgzf.plan_groups(bad, len(PRE), 1 << 16, 1 << 30)
    # a block whose BSIZE is smaller than its own header and trailer
    small = bytearray(bgzf.EOF_BLOCK)
    small[16], small[17] = 10, 0
    with pytest.raises(ValueError, match="smaller than its header"):
        bgzf.block_size(bytes(small), 0)
    # a corrupt block inflated on the host (a tail block) fails its CRC-32
    flipped = bytearray(comp)
    flipped[len(comp) - 28 - 8] ^= 1
    with pytest.raises(ValueError, match="CRC-32"):
        bgzf.plan_groups(bytes(flipped), len(PRE), 1 << 16, 1 << 30)
