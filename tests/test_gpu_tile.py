"""bvcf_tile_kernel's corners vs the CPU oracle, through the C ABI: variable-size locus strings, the slow path
(records that do not fit the shared-memory arena), capacity retries of the diagnostics buffer and the line
slots, INFO spans appended at copy-out, many tiles (decoupled look-back)."""
import io
import random

import pytest

import ref_vectors as V
from test_gpu_parity import _cfg, gpu_rows, oracle_rows

pytestmark = pytest.mark.gpu


def _process(vcf, cfg, **tr_kw):
    from bystro_vcf_b200 import Transformer, parse_preamble

    w, chrom, off = parse_preamble(vcf)
    with Transformer(cfg, eol_width=w, **tr_kw) as tr:
        tr.set_header(chrom)
        return tr.process(vcf[off:])


def _hdr(n):
    return V.HDR8 + ["FORMAT"] + ["S%04d_ab" % i for i in range(n)]


def test_dosage_locus_longer_than_63_bytes():
    """ADVICE r1: "chrom:pos:ref:+INS" keys used to live in 64-byte slots.  A 200-bp insertion, a 300-bp padded
    insertion, a long contig name and a 150-bp deletion: loci, dosages and rows all match (main.go:577)."""
    import numpy as np

    from oracle import oracle as O

    rng = random.Random(5)
    ins200 = "A" + "".join(rng.choice("ACGT") for _ in range(200))
    pad = "".join(rng.choice("ACGT") for _ in range(40))
    ins300 = pad + "".join(rng.choice("ACGT") for _ in range(300))
    contig = "GL000207.1_some_very_long_unplaced_scaffold_name_that_goes_on_and_on_0123456789"
    n = 12
    gts = ["0|1", "1|1", "0|0", ".|.", "1|0", "0|0", "0|0", "1", "0|0", "0/1", "0|0", "1|1"]
    recs = [["1", "1000", "rs1", "A", ins200, ".", "PASS", "DP=1", "GT"] + gts,
            [contig, "123456789", "rs2", pad, ins300, ".", "PASS", "DP=2", "GT"] + gts,
            ["chr7", "55", "rs3", "G" + "T" * 150, "G", ".", "PASS", "DP=3", "GT"] + gts,
            [contig, "77", "rs4", "A", "C," + ins200 + ",G", ".", "PASS", "DP=4", "GT"] + ["1|2", "2|3", "0|3"] + gts[3:]]
    vcf = V._vcf(_hdr(n), recs)
    ref = O.read_vcf(O.OracleConfig(want_dosage=True, keep_id=True, keep_info=True), vcf)
    assert max(len(x) for x in ref.loci) > 300
    c = _cfg(keep_id=True, keep_info=True)
    c.dosageMatrixOutPath = "unused.feather"
    res = _process(vcf, c)
    assert res.tsv == ref.tsv
    assert res.loci == ref.loci
    assert np.array_equal(res.dosage, ref.dosage)


@pytest.mark.parametrize("with_samples", [False, True])
def test_slow_path_records(with_samples):
    """Records whose rows do not fit the tile's arena -- a 3,000-base insertion, a 70-base MNP (70 rows), a 40-ALT
    site, a 5,000-character ID -- next to ordinary ones, with and without samples, keepId/keepInfo/keepPos on."""
    rng = random.Random(11)
    seq = lambda k: "".join(rng.choice("ACGT") for _ in range(k))
    n = 9 if with_samples else 0
    hdr = _hdr(n) if with_samples else V.HDR8
    tail = lambda: (["GT"] + [rng.choice(["0|0", "0|1", "1|1", "1|0", ".|.", "2|1", "0|2"]) for _ in range(n)]) if with_samples else []
    recs = []
    for i in range(400):
        k = i % 8
        pos = str(1000 + 7 * i)
        if k == 0:
            recs.append(["1", pos, "rs%d" % i, "A", "A" + seq(3000), ".", "PASS", "X=%d" % i] + tail())
        elif k == 1:
            r = seq(70)
            a = "".join({"A": "C", "C": "G", "G": "T", "T": "A"}[ch] for ch in r)
            recs.append(["2", pos, ".", r, a, ".", "PASS", "MNP"] + tail())
        elif k == 2:
            recs.append(["3", pos, ".", "A", ",".join(rng.choice(["C", "G", "T", "AT", "ACC"]) for _ in range(40)), ".", "PASS",
                         "M"] + tail())
        elif k == 3:
            recs.append(["4", pos, "r" * 5000, "G", "T", ".", "PASS", "ID"] + tail())
        else:
            recs.append(["5", pos, "rs%d" % i, "C", "T", ".", "PASS", "DP=%d" % i] + tail())
    vcf = V._vcf(hdr, recs)
    for kw in (dict(), dict(keep_id=True, keep_info=True, keep_pos=True)):
        assert gpu_rows(vcf, **kw) == oracle_rows(vcf, **kw)


def _sites_recs(rng, n, heavy=0.3):
    """sites-only records at BASELINE's mix: SNPs, multi-allelic sites, MNPs, padded indels, rejected alleles"""
    seq = lambda k: "".join(rng.choice("ACGT") for _ in range(k))
    recs = []
    for i in range(n):
        pos = str(10_000 + 13 * i)
        u = rng.random()
        if u > heavy:
            recs.append([rng.choice(["1", "chr2", "X", "chrM"]), pos, "rs%d" % i, rng.choice("ACGT"), rng.choice("ACGT"), ".", "PASS", "AC=%d" % i])
            continue
        k = rng.randrange(7)
        if k == 0:    # multi-allelic, 2..8 ALTs of mixed shapes
            ref = seq(rng.choice([1, 1, 2, 4]))
            alts = [rng.choice([seq(1), seq(2), ref[0] + seq(3), ref[:1], "<DEL>", "*", ref + seq(2)]) for _ in range(rng.randrange(2, 9))]
            recs.append(["3", pos, ".", ref, ",".join(alts), ".", "PASS", "M=%d" % i])
        elif k == 1:  # MNP
            r = seq(rng.randrange(2, 9))
            recs.append(["4", pos, ".", r, "".join(rng.choice("ACGT") for _ in r), ".", "PASS", "."])
        elif k == 2:  # deletion, padded
            r = seq(rng.randrange(2, 30))
            recs.append(["5", pos, "", r, r[:rng.randrange(1, len(r))], ".", "PASS", ""])
        elif k == 3:  # insertion, padded on both sides
            r = seq(rng.randrange(1, 6))
            recs.append(["chr6", pos, ".", r, r[:1] + seq(rng.randrange(1, 40)) + r[1:], ".", "PASS", "I"])
        elif k == 4:  # POS that is not a number / negative / huge, REF longer than one base
            recs.append(["7", rng.choice(["abc", "-5", "99999999999", "1e3", "007"]), ".", "AC", rng.choice(["A", "ACG", "GT", "A,ACT"]), ".", "PASS", "P"])
        elif k == 5:  # FILTER variety
            recs.append(["8", pos, ".", "A", "G", ".", rng.choice(["q10", ".", "PASS", "LowQual"]), "F"])
        else:         # REF == ALT, empty fields
            recs.append(["9", pos, ".", rng.choice(["A", ""]), rng.choice(["A", "", "."]), ".", "PASS", "E"])
    return recs


@pytest.mark.parametrize("kw", [dict(), dict(keep_info=True), dict(keep_id=True, keep_pos=True), dict(keep_id=True, keep_info=True, keep_pos=True)])
def test_sites_only_rows_spread_over_lanes(kw):
    """bvcf_compose_sites_kernel: rows planned per record and composed a row per lane, dense blocks copied out whole;
    --keepInfo takes the row-table path.  20,000 records, 30 % with two to eight candidate rows (main.go:723-1038)."""
    rng = random.Random(2024)
    vcf = V._vcf(V.HDR8, _sites_recs(rng, 20_000))
    assert gpu_rows(vcf, **kw) == oracle_rows(vcf, **kw)


def test_sites_only_overfull_tiles():
    """tiles whose rows exceed the row table (96) or the arena (3.5 KiB): the tail records take the slow path, the
    others stay staged; tiles where every record fails; a 70-row MNP next to SNPs"""
    rng = random.Random(77)
    seq = lambda k: "".join(rng.choice("ACGT") for _ in range(k))
    recs = []
    for i in range(3000):
        pos = str(500 + 3 * i)
        blk = (i // 32) % 6
        if blk == 0:    # 32 records x 8 rows = 256 rows in one tile
            recs.append(["1", pos, ".", "A", ",".join(rng.choice("CGT") for _ in range(8)), ".", "PASS", "."])
        elif blk == 1:  # 32 records x ~400 text bytes
            recs.append(["2", pos, ".", "A", "A" + seq(350), ".", "PASS", "."])
        elif blk == 2:  # a record on its own too large for the arena, SNPs around it
            recs.append(["3", pos, ".", "A", "A" + seq(7000), ".", "PASS", "."] if i % 32 == 7 else ["3", pos, ".", "C", "T", ".", "PASS", "."])
        elif blk == 3:  # 70-row MNP
            r = seq(70)
            a = "".join({"A": "C", "C": "G", "G": "T", "T": "A"}[ch] for ch in r)
            recs.append(["4", pos, ".", r, a, ".", "PASS", "."] if i % 32 in (0, 31) else ["4", pos, ".", "G", "A", ".", "PASS", "."])
        elif blk == 4:  # nothing comes out of the whole tile
            recs.append(["5", pos, ".", "A", "A", ".", "PASS", "."])
        else:
            recs.append(["6", pos, "rs%d" % i, "T", "C", ".", "PASS", "DP=%d" % i])
    vcf = V._vcf(V.HDR8, recs)
    for kw in (dict(), dict(keep_info=True, keep_id=True)):
        assert gpu_rows(vcf, **kw) == oracle_rows(vcf, **kw)


def test_sites_only_matches_thread_per_record_composer(monkeypatch):
    """the two sites-only composers (BVCF_SITES_OLD selects round 2's first one) give the same bytes and diagnostics"""
    from oracle import oracle as O

    rng = random.Random(4)
    vcf = V._vcf(V.HDR8, _sites_recs(rng, 6000, heavy=0.6))
    ref = O.read_vcf(O.OracleConfig(keep_info=True), vcf)
    a = _process(vcf, _cfg(keep_info=True))
    monkeypatch.setenv("BVCF_SITES_OLD", "1")
    b = _process(vcf, _cfg(keep_info=True))
    assert a.tsv == b.tsv == ref.tsv
    assert sorted(a.diags) == sorted(b.diags) == sorted(ref.diags)


def test_long_info_spans_appended_at_copy_out():
    """--keepInfo with INFO fields from 0 to 9,000 bytes: the span is copied from the input line after the staged row"""
    rng = random.Random(3)
    n = 5
    recs = []
    for i in range(700):
        ln = rng.choice([0, 1, 7, 8, 9, 15, 16, 17, 100, 1000, 9000])
        info = "".join(rng.choice("ABCdef=;0123") for _ in range(ln)) if ln else ""
        gts = [rng.choice(["0|0", "0|1", "1|1"]) for _ in range(n)]
        recs.append(["1", str(100 + i), "rs%d" % i, "A", "G", ".", "PASS", info, "GT"] + gts)
    vcf = V._vcf(_hdr(n), recs)
    assert gpu_rows(vcf, keep_info=True) == oracle_rows(vcf, keep_info=True)
    assert gpu_rows(vcf, keep_info=True, keep_id=True) == oracle_rows(vcf, keep_info=True, keep_id=True)


def test_diagnostics_beyond_first_capacity(monkeypatch):
    """ADVICE r1: diagnostics past the buffer's capacity used to be dropped; now the buffer grows and the chunk runs again"""
    from oracle import oracle as O

    monkeypatch.setenv("BVCF_DIAG_CAP", "16")
    recs = [["1", str(5 + i), ".", "A", "<DEL>" if i % 2 else "A", ".", "PASS", "."] for i in range(500)]
    vcf = V._vcf(V.HDR8, recs)
    ref = O.read_vcf(O.OracleConfig(), vcf)
    res = _process(vcf, _cfg())
    assert res.retries > 0
    assert sorted(res.diags) == sorted(ref.diags) and len(ref.diags) == 500
    assert res.tsv == ref.tsv


def test_short_lines_grow_the_line_slots():
    """ADVICE r1: with 8 <= H < 16 and lines shorter than 16 bytes the per-range line slots ran out and the chunk failed"""
    recs = [["1", str(i % 10), "", "A", "C", "", ".", ""] for i in range(40000)]  # 12-byte lines
    vcf = V._vcf(V.HDR8, recs)
    exp = oracle_rows(vcf)
    res = _process(vcf, _cfg())
    assert res.retries > 0
    assert res.tsv == exp and res.n_rows == 40000


def test_many_tiles_look_back(chr1_fixture):
    """1,000+ tiles of 128 records with very different sizes: every tile's offset comes from the look-back chain"""
    from oracle import oracle as O

    rng = random.Random(17)
    n = 40
    recs = []
    for i in range(150000):
        dense = i % 97 == 0
        gts = [rng.choice(["0|1", "1|1", "1|0"]) if dense or rng.random() < 0.02 else "0|0" for _ in range(n)]
        recs.append(["1", str(10 + i), ".", "A", "G", ".", "PASS", ".", "GT"] + gts)
    vcf = V._vcf(_hdr(n), recs)
    assert gpu_rows(vcf) == oracle_rows(vcf)


# ---- bgzf input: DEFLATE inflated on the GPU (SURVEY 8f-3) -------------------------------------------------
def _inflate_on_gpu(comp: bytes, n_text: int) -> bytes:
    from bystro_vcf_b200 import Transformer

    with Transformer(_cfg()) as tr:
        tr.set_header(b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO")
        tr.resident_alloc(max(n_text, 1), 4096)
        got = tr.resident_inflate_bgzf(comp)
        assert got == n_text
        return tr.resident_peek(0, n_text) if n_text else b""


@pytest.mark.parametrize("kind", ["dynamic", "fixed", "stored", "mixed-levels"])
def test_gpu_inflate_block_types(kind):
    """stored, fixed-Huffman and dynamic-Huffman DEFLATE blocks, matches at every distance / length class, literals of
    all 256 byte values, blocks from 1 byte to the 65,280-byte bgzf maximum: byte-identical to zlib on the host"""
    import zlib

    from bystro_vcf_b200 import bgzf

    rng = random.Random(29)
    parts = [bytes(rng.randrange(256) for _ in range(70000)),                      # literals, all byte values
             b"0|0\t" * 50000,                                                     # distance-4 matches of length 258
             b"".join(b"chr%d\t%d\trs%d\tA\tG\t100\tPASS\tAC=%d;AF=0.%d\tGT\t" % (i % 22, 1000 + 7 * i, i, i % 9, i) +
                      b"\t".join(rng.choice([b"0|0", b"0|0", b"0|0", b"0|1", b"1|1", b".|."]) for _ in range(300)) + b"\n"
                      for i in range(400)),
             bytes(rng.choice(b"ACGT") for _ in range(100000)),                    # four symbols: short codes
             b"x", b""]
    data = b"".join(parts)
    if kind == "dynamic":
        comp = bgzf.compress(data, level=6)
    elif kind == "fixed":
        comp = bgzf.compress(data, level=6, strategy=zlib.Z_FIXED)
    elif kind == "stored":
        comp = bgzf.compress(data, level=0)
    else:
        comp = b"".join(bgzf.compress(data[i:i + 100001], level=lv, block_text=bt, eof=False)
                        for i, (lv, bt) in zip(range(0, len(data), 100001), [(1, 1), (9, 65280), (4, 777), (6, 65280), (2, 31000)] * 10)) + bgzf.EOF_BLOCK
    import gzip

    assert gzip.decompress(comp) == data
    assert _inflate_on_gpu(comp, len(data)) == data


@pytest.mark.parametrize("gap", [15000, 16126, 16127, 16384, 20000, 32000, 32768])
def test_gpu_inflate_far_matches(gap):
    """matches whose source has left the 16 KiB shared-memory ring (distance up to DEFLATE's 32 KiB) are read back from
    the flushed text in global memory; sources that straddle the ring's edge; a stored block as the far source"""
    import gzip
    import zlib

    from bystro_vcf_b200 import bgzf

    rng = random.Random(gap)
    motif = bytes(rng.randrange(256) for _ in range(600))          # incompressible, so it can only come back as a match
    filler = bytes(rng.randrange(256) for _ in range(gap - 600))
    tail = b"".join(motif[j:j + 37] + bytes([j & 255]) for j in range(0, 560, 7))
    block = motif + filler + motif + filler[:500] + motif[100:400] + tail   # second motif: distance == gap
    data = block * 3
    for level, strategy in ((9, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_FIXED)):
        comp = bgzf.compress(data, level=level, block_text=65280, strategy=strategy)
        assert gzip.decompress(comp) == data
        assert _inflate_on_gpu(comp, len(data)) == data
    # one member = stored block(s) holding the first motif and the filler, then compressed blocks whose matches reach
    # back into the stored text (the compressor gets that text as its preset dictionary)
    import struct

    text = block[:gap + 600]
    c2 = zlib.compressobj(9, zlib.DEFLATED, -15, 9, zlib.Z_DEFAULT_STRATEGY, text[-32768:])
    rest = block[gap + 600:]
    stored = b"".join(struct.pack("<BHH", 0, len(text[i:i + 65535]), len(text[i:i + 65535]) ^ 0xFFFF) + text[i:i + 65535]
                      for i in range(0, len(text), 65535))
    member_payload = stored + c2.compress(rest) + c2.flush()
    whole = text + rest
    assert zlib.decompress(member_payload, -15) == whole
    if len(whole) <= 65280 and len(member_payload) + 26 <= 65536:
        member = (bgzf.MAGIC + b"\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(member_payload) + 25) +
                  member_payload + struct.pack("<II", zlib.crc32(whole), len(whole)))
        assert _inflate_on_gpu(member + bgzf.EOF_BLOCK, len(whole)) == whole


def test_gpu_inflate_rejects_corrupt_blocks():
    from bystro_vcf_b200 import BvcfError, Transformer, bgzf

    comp = bytearray(bgzf.compress(b"0|0\t1|1\t" * 30000, eof=False))
    comp[40] ^= 0x55  # inside the first block's DEFLATE payload
    with Transformer(_cfg()) as tr:
        tr.set_header(b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO")
        tr.resident_alloc(1 << 20, 4096)
        with pytest.raises(BvcfError):
            tr.resident_inflate_bgzf(bytes(comp))
        with pytest.raises(BvcfError):
            tr.resident_inflate_bgzf(b"not bgzf at all, just text\n")


def test_bgzf_vcf_resident_and_streaming_match_plain(chr1_fixture):
    """a .vcf.gz (bgzf) through the resident (bgzfOut) driver: compressed bytes to the device, inflated there, rows
    identical to the plain path; groups smaller than the file, so partial lines are carried from group to group.  Then
    through read_vcf, which runs it on the streaming path."""
    import dataclasses
    import gzip
    import io

    from bystro_vcf_b200 import Config, bgzf, host, read_vcf

    vcf = chr1_fixture[:60 << 20].rsplit(b"\n", 1)[0] + b"\nunterminated last line"
    comp = bgzf.compress(vcf)
    assert len(comp) < len(vcf) // 10
    c = Config()
    c.allowedFilters = {"PASS": True, ".": True}
    c.keepID = c.keepInfo = True
    plain = io.BytesIO()
    st0 = read_vcf(c, io.BytesIO(vcf), plain)
    for batch in (512 << 20, 7 << 20):
        out = io.BytesIO()
        st = host._read_vcf_resident(dataclasses.replace(c, bgzfOut=True), comp[:1 << 20], io.BytesIO(comp[1 << 20:]), out,
                                     batch_text=batch)
        assert gzip.decompress(out.getvalue()) == plain.getvalue()
        assert st["n_rows"] == st0["n_rows"] and st["compressed_bytes"] <= len(comp)
    out = io.BytesIO()
    read_vcf(c, io.BytesIO(comp), out)  # auto-detected
    assert out.getvalue() == plain.getvalue()


# ---- bgzf output: rows deflated on the GPU (SURVEY 8f-4) ------------------------------------------------------
def test_gpu_deflate_output_is_valid_bgzf(chr1_fixture):
    """The rows of a resident run leave as bgzf blocks made on the GPU (LZ77 + fixed Huffman + CRC-32): gzip on the host
    -- which verifies every member's CRC-32 and ISIZE -- gives the uncompressed rows back, block headers are bgzf's."""
    import gzip

    from bystro_vcf_b200 import Config, Transformer, bgzf, parse_preamble

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
        rows = tr.resident_download(0, n)
        comp = tr.resident_download_bgzf(0, n)
        assert gzip.decompress(comp + bgzf.EOF_BLOCK) == rows
        assert len(comp) < n * 0.6  # sample-name lists and repeated columns do compress
        p = k = 0
        while p < len(comp):  # whole bgzf blocks of at most 48 KiB of text
            bs = bgzf.block_size(comp, p)
            assert bs > 0 and int.from_bytes(comp[p + bs - 4:p + bs], "little") <= 49152
            p += bs
            k += 1
        assert p == len(comp) and k == -(-n // 49152)
        # odd sizes and offsets: one byte, a slice boundary +- 1, an unaligned start
        for o, ln in ((0, 1), (3, 49151), (5, 49152), (7, 49153), (12345, 200001)):
            assert gzip.decompress(tr.resident_download_bgzf(o, ln) + bgzf.EOF_BLOCK) == rows[o:o + ln]


def test_gpu_deflate_incompressible_and_repetitive():
    """random bytes (every literal, 9-bit codes: the block grows) and one byte repeated (distance-1 matches of 258)"""
    import gzip

    from bystro_vcf_b200 import Transformer, bgzf

    rng = random.Random(41)
    for data in (bytes(rng.randrange(256) for _ in range(120000)), b"A" * 150000, b"0|0\t1|1\t" * 20000 + b"\n"):
        with Transformer(_cfg()) as tr:
            tr.set_header(b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO")
            tr.resident_alloc(1 << 20, len(data) + 4096)
            tr.resident_write_output(0, data)
            assert gzip.decompress(tr.resident_download_bgzf(0, len(data)) + bgzf.EOF_BLOCK) == data
