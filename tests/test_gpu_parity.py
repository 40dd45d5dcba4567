"""CUDA path vs CPU oracle / reference vectors.  Every call goes through the C ABI (libbvcf.so)."""
import hashlib
import io

import pytest

import ref_vectors as V

pytestmark = pytest.mark.gpu


def _cfg(**kw):
    from bystro_vcf_b200 import Config

    c = Config()
    m = {"keep_id": "keepID", "keep_info": "keepInfo", "keep_pos": "keepPos"}
    for k, v in kw.items():
        if k == "allow":
            c.allowedFilters = None if v is None else {x: True for x in v}
        elif k == "exclude":
            c.excludedFilters = None if v is None else {x: True for x in v}
        else:
            setattr(c, m[k], v)
    if "allow" not in kw:
        c.allowedFilters = {"PASS": True, ".": True}
    return c


def gpu_rows(vcf: bytes, **kw) -> bytes:
    from bystro_vcf_b200 import read_vcf

    out = io.BytesIO()
    read_vcf(_cfg(**kw), io.BytesIO(vcf), out)
    return out.getvalue()


def oracle_rows(vcf: bytes, **kw) -> bytes:
    from oracle import oracle as O

    return O.read_vcf(O.OracleConfig(**kw), vcf).tsv


def rows_of(tsv: bytes):
    return [r.split("\t") for r in tsv.decode().split("\n")[:-1]] if tsv else []


@pytest.mark.parametrize("name,cfg,vcf,exp", V.STREAM_CASES, ids=[c[0] for c in V.STREAM_CASES])
def test_reference_stream_vectors(name, cfg, vcf, exp):
    got = gpu_rows(vcf, **cfg)
    assert rows_of(got) == exp
    assert got == oracle_rows(vcf, **cfg)


@pytest.mark.parametrize("fields,a,nhom,nhet,nmiss,ac,an", V.GT_VECTORS)
def test_genotype_vectors(fields, a, nhom, nhet, nmiss, ac, an):
    """makeHetHomozygotes vectors (main_test.go:652-951) through a synthetic one-line VCF whose ALT list
    makes `a` an output allele."""
    n_alt = int(a)
    alts = ",".join(["C", "G", "T"][:max(n_alt, 1)])
    hdr = V.HDR8 + ["FORMAT"] + ["S%d" % i for i in range(len(fields))]
    vcf = V._vcf(hdr, [["1", "100", ".", "A", alts, ".", "PASS", ".", "GT"] + fields])
    got = rows_of(gpu_rows(vcf))
    exp = rows_of(oracle_rows(vcf))
    assert got == exp
    row = [r for r in got if r[4] == ["C", "G", "T"][n_alt - 1]]
    if ac == 0:
        assert row == []
    else:
        r = row[0]
        assert (r[12], r[13]) == (str(ac), str(an))
        assert (0 if r[6] == "!" else len(r[6].split(";"))) == nhet
        assert (0 if r[8] == "!" else len(r[8].split(";"))) == nhom
        assert (0 if r[10] == "!" else len(r[10].split(";"))) == nmiss


@pytest.mark.parametrize("inp,exp", V.ALLELE_VECTORS)
def test_allele_vectors(inp, exp):
    pos, ref, alt = inp
    vcf = V._vcf(V.HDR8, [["chr1", pos, ".", ref, alt, ".", "PASS", "."]])
    got = rows_of(gpu_rows(vcf))
    typ, poss, refs, alts, _ = exp
    assert [(r[0], r[1], r[2], r[3], r[4]) for r in got] == [("chr1", p, typ, r_, a_) for p, r_, a_ in zip(poss, refs, alts)]


def test_golden_chr1(chr1_fixture):
    got = gpu_rows(chr1_fixture)
    assert len(got) == 32496849
    assert hashlib.md5(got).hexdigest() == V.GOLDEN_MD5_INPUT_ORDER


def test_golden_chr1_keepid_keepinfo_small_chunks(chr1_fixture):
    from bystro_vcf_b200 import read_vcf

    cfg = _cfg(keep_id=True, keep_info=True)
    cfg.chunkBytes = 7 << 20  # many chunks, lines straddle every read boundary
    out = io.BytesIO()
    st = read_vcf(cfg, io.BytesIO(chr1_fixture), out)
    assert st["n_lines"] == 19600 and st["n_rows"] == 20090
    assert hashlib.md5(out.getvalue()).hexdigest() == V.GOLDEN_MD5_KEEPID_KEEPINFO


def test_query_fixture_matches_oracle(query_fixture):
    for kw in ({}, {"allow": None, "keep_pos": True, "keep_id": True, "keep_info": True}):
        got = gpu_rows(query_fixture, **kw)
        exp = oracle_rows(query_fixture, **kw)
        assert got == exp


def test_dosage_matrix_vector():
    """main_test.go:2911-2977 TestGenotypeMatrix through the C ABI (dosage batch of bvcf_collect)."""
    from bystro_vcf_b200 import Config, Transformer, parse_preamble

    vcf, loci, dos = V.DOSAGE_CASE
    c = _cfg()
    c.dosageMatrixOutPath = "unused.feather"
    w, chrom, off = parse_preamble(vcf)
    with Transformer(c, eol_width=w) as tr:
        tr.set_header(chrom)
        res = tr.process(vcf[off:])
    assert res.loci == loci
    assert res.dosage.tolist() == dos


def test_dosage_matrix_chr1_vs_oracle(chr1_fixture):
    import numpy as np

    from bystro_vcf_b200 import Config, Transformer, parse_preamble
    from oracle import oracle as O

    n = chr1_fixture.index(b"\n", 30 << 20) + 1  # ~30 MB: header + ~2,900 records
    data = chr1_fixture[:n]
    ref = O.read_vcf(O.OracleConfig(want_dosage=True), data)
    c = _cfg()
    c.dosageMatrixOutPath = "unused.feather"
    w, chrom, off = parse_preamble(data)
    with Transformer(c, eol_width=w) as tr:
        tr.set_header(chrom)
        res = tr.process(data[off:])
    assert res.tsv == ref.tsv
    assert res.loci == ref.loci
    assert np.array_equal(res.dosage, ref.dosage)


def test_diagnostics_match_oracle():
    """the reference's log.Printf sites (main.go:730-986) as (line, alt, code) triples"""
    from bystro_vcf_b200 import Transformer, parse_preamble
    from oracle import oracle as O

    recs = [["1", "5", ".", "A", "A", ".", "PASS", "."], ["1", "6", ".", "A", "<DEL>", ".", "PASS", "."],
            ["1", "7", ".", "AT", "G", ".", "PASS", "."], ["1", "x", ".", "AT", "A", ".", "PASS", "."],
            ["1", "9", ".", "A", "GT,C,N", ".", "PASS", "."], ["1", "10", ".", "TAGCTT", "TAC,T", ".", "PASS", "."],
            ["1", "y", ".", "AT", "A,ATT", ".", "PASS", "."], ["1", "12", ".", "AT", "C,ATT", ".", "PASS", "."]]
    vcf = V._vcf(V.HDR8, recs)
    ref = O.read_vcf(O.OracleConfig(), vcf)
    w, chrom, off = parse_preamble(vcf)
    with Transformer(_cfg(), eol_width=w) as tr:
        tr.set_header(chrom)
        res = tr.process(vcf[off:])
    assert res.tsv == ref.tsv
    assert sorted(res.diags) == sorted(ref.diags)
    assert len(ref.diags) >= 8


def test_long_fields_beyond_64k():
    """tab offsets past 64 KiB (huge INFO / ALT): the rows kernel rescans the line itself"""
    info = "X=" + "A" * 70000
    ins = "A" + "ACGT" * 20000
    hdr = V.HDR8 + ["FORMAT", "S1", "S2", "S3"]
    recs = [["1", "100", "rs1", "A", "C", ".", "PASS", info, "GT", "0|1", "1|1", "0|0"],
            ["1", "200", "rs2", "A", ins, ".", "PASS", "Y=1", "GT", "0|1", "0|0", ".|."],
            ["1", "300", "rs3", "A", "G", ".", "PASS", "Z", "GT:PL", "0/1:" + "9," * 40000 + "9", "1/1:0", "0/0:1"]]
    vcf = V._vcf(hdr, recs)
    for kw in ({}, {"keep_info": True, "keep_id": True, "keep_pos": True}):
        assert gpu_rows(vcf, **kw) == oracle_rows(vcf, **kw)


def test_slash_separated_and_mixed_width_fields():
    """'/'-separated 1000G-style block (T1/T2 tiers follow the separator) with odd-width fields mixed in"""
    import random

    rnd = random.Random(7)
    ns = 700
    hdr = V.HDR8 + ["FORMAT"] + ["N%04d" % i for i in range(ns)]
    recs = []
    for i in range(300):
        sep = "/" if i % 3 else "|"
        gts = []
        for s in range(ns):
            r = rnd.random()
            if r < 0.9: g = "0" + sep + "0"
            elif r < 0.95: g = "0" + sep + "1"
            elif r < 0.97: g = "1" + sep + "1"
            elif r < 0.98: g = "." + sep + "."
            elif r < 0.985: g = "1"
            elif r < 0.99: g = "10" + sep + "0"
            elif r < 0.995: g = "0" + sep + "1" + sep + "1"
            else: g = "0" + ("|" if sep == "/" else "/") + "1"
            gts.append(g)
        recs.append(["2", str(1000 + i), ".", "A", "C,G", ".", "PASS", ".", "GT"] + gts)
    vcf = V._vcf(hdr, recs)
    assert gpu_rows(vcf) == oracle_rows(vcf)


def test_dense_genotype_block_grows_event_scratch():
    """every sample non-reference and haploid: 4 event bytes per 2 input bytes overflows the default event
    slice; the library must notice, grow the scratch and re-run the chunk (retries > 0), byte-identically"""
    from bystro_vcf_b200 import Transformer, parse_preamble
    from oracle import oracle as O

    ns = 6000
    hdr = V.HDR8 + ["FORMAT"] + ["H%05d" % i for i in range(ns)]
    recs = [["3", str(100 + i), ".", "A", "C", ".", "PASS", ".", "GT"] + ["1"] * ns for i in range(200)]
    vcf = V._vcf(hdr, recs)
    ref = O.read_vcf(O.OracleConfig(), vcf)
    w, chrom, off = parse_preamble(vcf)
    with Transformer(_cfg(), eol_width=w) as tr:
        tr.set_header(chrom)
        res = tr.process(vcf[off:])
    assert res.retries > 0
    assert res.tsv == ref.tsv


def test_dosage_arrow_file_like_reference(tmp_path):
    """main_test.go:2911-2977 TestGenotypeMatrix end to end: --dosageOutput writes an Arrow IPC file (zstd) with
    schema locus: utf8 + one non-nullable int8 column per sample; read it back like the reference test does."""
    import pyarrow as pa

    from bystro_vcf_b200 import read_vcf

    vcf, loci, dos = V.DOSAGE_CASE
    path = tmp_path / "dosage.feather"
    c = _cfg()
    c.dosageMatrixOutPath = str(path)
    out = io.BytesIO()
    read_vcf(c, io.BytesIO(vcf), out)
    with pa.OSFile(str(path), "rb") as f:
        t = pa.ipc.open_file(f).read_all()
    assert t.schema.names == ["locus", "S1", "S2", "S3"]
    assert t.schema.field("locus").type == pa.string() and not t.schema.field("locus").nullable
    assert all(t.schema.field(n).type == pa.int8() and not t.schema.field(n).nullable for n in ("S1", "S2", "S3"))
    got = {l: [t.column(n)[i].as_py() for n in ("S1", "S2", "S3")] for i, l in enumerate(t.column("locus").to_pylist())}
    assert got == {l.decode(): d for l, d in zip(loci, dos)}
    # TestNoOut (main_test.go:2980-3029): --noOut still writes the matrix and no TSV
    c.noOut = True
    out2 = io.BytesIO()
    read_vcf(c, io.BytesIO(vcf), out2)
    assert out2.getvalue() == b""
    with pa.OSFile(str(path), "rb") as f:
        assert pa.ipc.open_file(f).read_all().num_rows == 3


def test_odd_bytes_in_regular_genotype_zones():
    """Bytes that are neither a digit nor '.' where an allele belongs, inside otherwise regular `x|y` zones (the
    vector tiers of the scan kernel must hand such windows to the field-by-field path): high-bit bytes whose low
    nibble looks like a digit, '/', ':' and letters, next to missing and multi-allelic samples."""
    import random

    rng = random.Random(7)
    n = 700  # several 512-byte windows per line
    hdr = V.HDR8 + ["FORMAT"] + ["ZZ%05d" % i for i in range(n)]  # 7-character names: the vector names path
    odd = [b"\xba", b"\xbf", b"\x8a", b"/", b"?", b"N", b"\x1e", b"\x3a", b"\xb1", b"\xfe"]
    recs = []
    for r in range(40):
        fields = []
        for i in range(n):
            u = rng.random()
            if u < 0.90:
                f = b"0|0"
            elif u < 0.93:
                f = b"0|1" if rng.random() < 0.5 else b"1|1"
            elif u < 0.95:
                f = b".|." if rng.random() < 0.5 else b"0|."
            elif u < 0.97:
                f = b"2|1"
            else:
                a = odd[rng.randrange(len(odd))]
                f = (a + b"|1") if rng.random() < 0.5 else (b"1|" + a)
            fields.append(f)
        fixed = [b"1", str(1000 + r).encode(), b".", b"A", b"C,G", b".", b"PASS", b".", b"GT"]
        recs.append(b"\t".join(fixed + fields))
    vcf = (V.VERSION + "\n" + "\t".join(hdr) + "\n").encode() + b"\n".join(recs) + b"\n"
    got = gpu_rows(vcf)
    exp = oracle_rows(vcf)
    assert got == exp
    assert len(got) > 1000


def _fuzz_vcf(rng, n_samples, n_lines, name_w):
    """A random VCF whose lines differ in every dimension the scan kernel's tiers care about: prefix length (the
    field phase modulo 4 and where the 512-byte windows cut), GT shapes, FORMAT suffixes, field counts."""
    names = [("%0*d" % (name_w, i))[-name_w:] if name_w else "s%d" % (i * 37 % 1000) for i in range(n_samples)]
    hdr = V.HDR8 + (["FORMAT"] + names if n_samples else [])
    gts_common = ["0|0"] * 30 + ["0|1", "1|0", "1|1", ".|.", "0|.", "2|1", "0|2", "3|3"]
    gts_odd = ["0/0", "0/1", "1", "0", ".", "", "10|1", "1|10", "0|1|1", "1/1/1", "0|1:35", "1|1:0,3:99", "./.", "0/1|1",
               "A|1", "1|?", "01|1", "1|", "|1", "1||1"]
    alts = ["C", "G", "T", "C,G", "G,T,C", "AC", "ACG,AT", "<DEL>", "*", "N", "a", "C,<CN0>,G", "AT,ATT"]
    refs = ["A", "A", "A", "AT", "ATG", "ACGT"]
    filts = ["PASS", "PASS", "PASS", ".", "q10", "PASS;q10"]
    recs = []
    for i in range(n_lines):
        info = "AC=%d;AN=%d;X=%s" % (rng.randrange(100), rng.randrange(5000), "k" * rng.randrange(0, 90))
        if rng.random() < 0.05:
            info += ";LONG=" + "z" * rng.randrange(400, 3000)  # the fixed fields span several 512-byte windows
        ident = rng.choice([".", "rs%d" % rng.randrange(10 ** rng.randrange(1, 9))])
        chrom = rng.choice(["1", "22", "X", "chr7", "GL000207.1"])
        fixed = [chrom, str(rng.randrange(1, 10 ** rng.randrange(1, 9))), ident, rng.choice(refs), rng.choice(alts), "100",
                 rng.choice(filts), info]
        if not n_samples:
            recs.append(fixed)
            continue
        mode = rng.random()
        p_odd = 0.0 if mode < 0.5 else (0.002 if mode < 0.8 else 0.05)
        p_alt = rng.choice([0.0, 0.001, 0.02, 0.5])
        fmt = "GT" if rng.random() < 0.9 else "GT:DP"
        fields = []
        for s in range(n_samples):
            u = rng.random()
            if u < p_odd:
                g = rng.choice(gts_odd)
            elif u < p_odd + p_alt:
                g = rng.choice(gts_common[30:])
            else:
                g = "0|0"
            if fmt != "GT" and rng.random() < 0.5:
                g += ":%d" % rng.randrange(100)
            fields.append(g)
        n_keep = n_samples if rng.random() < 0.97 else rng.randrange(0, n_samples + 3)  # wrong field counts vanish
        fields = (fields + ["0|0"] * 3)[:n_keep]
        recs.append(fixed + [fmt] + fields)
        if rng.random() < 0.03:
            recs.append(rng.choice([[], [""], ["1"], ["1", "5"], fixed[:5]]))  # blank and truncated lines vanish
    return V._vcf(hdr, recs)


import os as _os


_FUZZ_OFF = int(_os.environ.get("BVCF_FUZZ_OFFSET", "0"))


@pytest.mark.parametrize("seed", range(_FUZZ_OFF, _FUZZ_OFF + int(_os.environ.get("BVCF_FUZZ_N", "24"))))
def test_fuzz_line_shapes_vs_oracle(seed):
    import random

    rng = random.Random(1000 + seed)
    n_samples = rng.choice([0, 1, 3, 31, 127, 128, 129, 300, 700, 1500])
    name_w = rng.choice([7, 7, 0, 4])  # 7-character names take the 8-byte-item kernels, the others the general ones
    vcf = _fuzz_vcf(rng, n_samples, rng.randrange(20, 120), name_w)
    kw = rng.choice([{}, {"keep_info": True, "keep_id": True}, {"keep_pos": True}, {"allow": None}, {"exclude": ["q10"]}])
    assert gpu_rows(vcf, **kw) == oracle_rows(vcf, **kw)


def test_empty_last_sample_field():
    """A line whose last sample field is empty (a tab right before the newline) inside an otherwise regular `x|y`
    zone: the empty token still counts one allele towards `an` (main.go:1143,1166)."""
    ns = 300
    hdr = V.HDR8 + ["FORMAT"] + ["Q%06d" % i for i in range(ns)]
    recs = []
    for i in range(8):
        gts = ["0|0"] * ns
        gts[5 + i] = "0|1"
        gts[-1] = ""  # the empty last field
        recs.append(["1", str(100 + 13 * i), ".", "A" * (1 + i % 4), "C", ".", "PASS", "X" * i, "GT"] + gts)
    vcf = V._vcf(hdr, recs)
    got = gpu_rows(vcf)
    assert got == oracle_rows(vcf)
    assert all(r[13] == str(2 * (ns - 1) + 1) for r in rows_of(got))


@pytest.mark.parametrize("seed", range(_FUZZ_OFF, _FUZZ_OFF + int(_os.environ.get("BVCF_FUZZ2_N", "16"))))
def test_fuzz_options_dosage_chunks_vs_oracle(seed):
    """The same random line shapes under the other axes: CRLF line ends, 64 KiB chunks through submit/collect,
    multi-character emptyField / fieldDelimiter, the dosage matrix, diagnostics."""
    import random

    import numpy as np

    from bystro_vcf_b200 import Transformer, parse_preamble, read_vcf
    from oracle import oracle as O

    rng = random.Random(5000 + seed)
    n_samples = rng.choice([1, 5, 128, 257, 700, 1500, 3500])
    name_w = rng.choice([7, 7, 3])
    vcf = _fuzz_vcf(rng, n_samples, rng.randrange(30, 160), name_w)
    if rng.random() < 0.3:
        vcf = vcf.replace(b"\n", b"\r\n")
    empty, delim = rng.choice([("!", ";"), ("NA", "|"), ("", ";;"), ("!", ",")])
    okw = {"empty_field": empty, "field_delim": delim, "keep_id": rng.random() < 0.5, "keep_info": rng.random() < 0.3}
    want_dosage = rng.random() < 0.5
    ref = O.read_vcf(O.OracleConfig(want_dosage=want_dosage, **okw), vcf)
    c = _cfg(keep_id=okw["keep_id"], keep_info=okw["keep_info"])
    c.emptyField, c.fieldDelimiter = empty, delim
    if want_dosage:
        c.dosageMatrixOutPath = "unused.feather"
    w, chrom, off = parse_preamble(vcf)
    with Transformer(c, eol_width=w) as tr:
        tr.set_header(chrom)
        res = tr.process(vcf[off:])
    assert res.tsv == ref.tsv
    assert sorted(res.diags) == sorted(ref.diags)
    if want_dosage:
        assert res.loci == ref.loci
        assert np.array_equal(res.dosage, ref.dosage)
    # and the streaming driver with the smallest chunks
    c2 = _cfg(keep_id=okw["keep_id"], keep_info=okw["keep_info"])
    c2.emptyField, c2.fieldDelimiter = empty, delim
    c2.chunkBytes = 1 << 16
    out = io.BytesIO()
    read_vcf(c2, io.BytesIO(vcf), out)
    assert out.getvalue() == ref.tsv


@pytest.mark.parametrize("n_samples,dens,name_fmt", [(3000, 0.9, "W%06d"), (9000, 0.5, "W%06d"), (20000, 0.6, "W%06d"),
                                                     (20000, 0.15, "W%06d"), (70000, 0.3, "W%06d"), (3000, 0.8, "ID%08d"),
                                                     (20000, 0.5, "s%04d"[:6] + "x"), (9000, 0.6, "LONGNAME%07d")])
def test_wide_dense_rows_name_kernels(n_samples, dens, name_fmt):
    """Rows whose name lists outgrow the per-warp index buffer (chunked sweep) and whose event lists exceed 4,096 quads
    (CTA-per-row kernel), with 16-bit (<= 65,000 samples) and 32-bit sample indices; multi-allelic and missing
    samples mixed in; with and without the dosage matrix."""
    import random

    import numpy as np

    from bystro_vcf_b200 import Transformer, parse_preamble
    from oracle import oracle as O

    rng = random.Random(n_samples + int(dens * 100))
    # 7-character names: 8-byte items; 10 and 15 characters: 16-byte padded items; "s%04dx" grows from 6 to 7 characters
    # (variable width: the general kernels)
    hdr = V.HDR8 + ["FORMAT"] + [name_fmt % i for i in range(n_samples)]
    pool = ["0|1", "1|0", "1|1", "1|1", ".|.", "2|1", "0|2", "1", "1|1|0"]
    recs = []
    for i in range(6):
        d = dens if i % 2 == 0 else dens / 8
        gts = [rng.choice(pool) if rng.random() < d else "0|0" for _ in range(n_samples)]
        recs.append(["7", str(500 + i), ".", "A", "C,G" if i % 3 == 0 else "C", ".", "PASS", ".", "GT"] + gts)
    vcf = V._vcf(hdr, recs)
    for want_dosage in (False, True):
        ref = O.read_vcf(O.OracleConfig(want_dosage=want_dosage), vcf)
        c = _cfg()
        if want_dosage:
            c.dosageMatrixOutPath = "unused.feather"
        w, chrom, off = parse_preamble(vcf)
        with Transformer(c, eol_width=w) as tr:
            tr.set_header(chrom)
            res = tr.process(vcf[off:])
        assert res.tsv == ref.tsv
        if want_dosage:
            assert res.loci == ref.loci
            assert np.array_equal(res.dosage, ref.dosage)


@pytest.mark.parametrize("seed", range(_FUZZ_OFF, _FUZZ_OFF + int(_os.environ.get("BVCF_FUZZ3_N", "12"))))
def test_fuzz_resident_tiny_subchunks_vs_oracle(seed):
    """The device-resident entry points (bvcf_resident_*) on random line shapes, cut into 64 KiB sub-chunks so that
    lines straddle sub-chunk and range boundaries everywhere."""
    import random

    from bystro_vcf_b200 import Transformer, parse_preamble
    from oracle import oracle as O

    rng = random.Random(9000 + seed)
    n_samples = rng.choice([0, 2, 128, 700, 1500, 4000])
    vcf = _fuzz_vcf(rng, n_samples, rng.randrange(40, 200), 7)
    ref = O.read_vcf(O.OracleConfig(), vcf)
    w, chrom, off = parse_preamble(vcf)
    body = vcf[off:]
    with Transformer(_cfg(), eol_width=w, resident_subchunk_bytes=1 << 16) as tr:
        tr.set_header(chrom)
        tr.resident_alloc(len(body), max(len(body), 1 << 20))
        tr.resident_upload(0, body)
        stats, _ = tr.resident_run(len(body))
        out = tr.resident_download(0, stats["out_bytes"]) if stats["out_bytes"] else b""
    assert out == ref.tsv
    assert stats["n_rows"] == ref.n_rows


def test_output_and_row_capacity_retries():
    """Outputs larger than the library's first guess: the kernels flag the overflow, the host grows the buffer and
    re-runs the chunk (output several times the input: every ALT of a sites-only line is a row; eight rows per
    record with samples: an 8-base MNP), through submit/collect and through the resident entry points."""
    from bystro_vcf_b200 import Transformer, parse_preamble
    from oracle import oracle as O

    # sites-only, three rows per 30-byte line
    recs = [["1", str(10 + i), ".", "A", "C,G,T", ".", "PASS", "."] for i in range(60000)]
    vcf = V._vcf(V.HDR8, recs)
    ref = O.read_vcf(O.OracleConfig(), vcf)
    assert len(ref.tsv) > 3 * len(vcf)
    w, chrom, off = parse_preamble(vcf)
    body = vcf[off:]
    with Transformer(_cfg(), eol_width=w) as tr:
        tr.set_header(chrom)
        res = tr.process(body)
        assert res.retries > 0 and res.tsv == ref.tsv
        tr.resident_alloc(len(body), 4096)  # absurdly small output region
        tr.resident_upload(0, body)
        stats, _ = tr.resident_run(len(body))
        assert stats["retries"] > 0
        assert tr.resident_download(0, stats["out_bytes"]) == ref.tsv
    # samples + MNPs: more rows than row descriptors
    hdr = V.HDR8 + ["FORMAT", "S1", "S2", "S3"]
    recs = [["2", str(100 + 10 * i), ".", "ACGTACGT", "TGCATGCA", ".", "PASS", ".", "GT", "0|1", "1|1", "0|0"] for i in range(40000)]
    vcf = V._vcf(hdr, recs)
    ref = O.read_vcf(O.OracleConfig(), vcf)
    assert ref.n_rows == 8 * 40000
    w, chrom, off = parse_preamble(vcf)
    with Transformer(_cfg(), eol_width=w) as tr:
        tr.set_header(chrom)
        res = tr.process(vcf[off:])
    assert res.tsv == ref.tsv
    assert res.retries > 0


def _fuzz_alleles_vcf(rng, n_lines, with_samples):
    """Random REF/ALT pairs around getAlleles' decision tree (main.go:723-1038): SNPs, MNPs, insertions and deletions
    with shared prefixes/suffixes, mixed and malformed alleles, odd POS, multi-allelic lists."""
    B = "ACGT"

    def bases(n):
        return "".join(rng.choice(B) for _ in range(n))

    def alt_of(ref):
        u = rng.random()
        if u < 0.25:  # SNP / MNP
            a = list(ref)
            for _ in range(rng.randrange(1, len(a) + 1)):
                i = rng.randrange(len(a)); a[i] = rng.choice(B)
            return "".join(a)
        if u < 0.45:  # insertion after a shared prefix, maybe a shared suffix
            k = rng.randrange(0, len(ref) + 1)
            return ref[:k] + bases(rng.randrange(1, 6)) + ref[k:]
        if u < 0.65 and len(ref) > 1:  # deletion
            k = rng.randrange(1, len(ref)); m = rng.randrange(k, len(ref) + 1)
            return ref[:k] + ref[m:] if ref[:k] + ref[m:] else ref[0]
        if u < 0.72:
            return bases(rng.randrange(1, 9))  # unrelated
        if u < 0.80:
            return rng.choice(["<DEL>", "*", ".", "N", "acgt", "A[chr1:5[", "", ref])
        return rng.choice(B)

    hdr = V.HDR8 + (["FORMAT", "S1", "S2", "S3"] if with_samples else [])
    recs = []
    for i in range(n_lines):
        ref = bases(rng.choice([1, 1, 1, 2, 3, 4, 8, 9, 13]))  # 9, 13: beyond the eight REF bases the generator keeps in registers
        alts = ",".join(alt_of(ref) for _ in range(rng.choice([1, 1, 1, 2, 3, 5])))
        odd_pos = [str(rng.randrange(1, 10 ** rng.randrange(1, 10))), "x", "+5", "-3", "007", "9223372036854775807"]
        pos = rng.choice(odd_pos) if rng.random() < 0.1 else str(rng.randrange(1, 250000000))
        rec = [rng.choice(["1", "chr1", "MT", "GL000207.1", "c"]), pos, rng.choice([".", "rs1;rs2"]), ref, alts, ".",
               rng.choice(["PASS", "PASS", ".", "q10"]), "AC=1"]
        if with_samples:
            n_alt = alts.count(",") + 1
            gts = ["%s|%s" % (rng.randrange(0, n_alt + 1), rng.randrange(0, n_alt + 1)) for _ in range(3)]
            rec += ["GT"] + gts
        recs.append(rec)
    return V._vcf(hdr, recs)


@pytest.mark.parametrize("seed", range(_FUZZ_OFF, _FUZZ_OFF + int(_os.environ.get("BVCF_FUZZ4_N", "12"))))
def test_fuzz_alleles_vs_oracle(seed):
    import random

    from bystro_vcf_b200 import Transformer, parse_preamble
    from oracle import oracle as O

    rng = random.Random(77000 + seed)
    vcf = _fuzz_alleles_vcf(rng, rng.randrange(50, 400), rng.random() < 0.5)
    okw = {"keep_id": rng.random() < 0.5, "keep_info": rng.random() < 0.5, "keep_pos": rng.random() < 0.5}
    ref = O.read_vcf(O.OracleConfig(**okw), vcf)
    w, chrom, off = parse_preamble(vcf)
    with Transformer(_cfg(**okw), eol_width=w) as tr:
        tr.set_header(chrom)
        res = tr.process(vcf[off:])
    assert res.tsv == ref.tsv
    assert sorted(res.diags) == sorted(ref.diags)
