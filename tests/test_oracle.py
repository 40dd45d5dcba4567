"""Pins the CPU oracle (oracle/) against the reference's own vectors and golden output.  CPU only."""
import gzip
import hashlib
import os
import subprocess

import pytest

import ref_vectors as V
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rows_of(tsv: bytes):
    return [r.split("\t") for r in tsv.decode().split("\n")[:-1]] if tsv else []


@pytest.mark.parametrize("inp,exp", V.ALLELE_VECTORS)
def test_get_alleles(inp, exp):
    assert O.get_alleles("chr1", *inp) == exp


@pytest.mark.parametrize("alt,exp", V.ALT_VALID_VECTORS)
def test_alt_is_valid(alt, exp):
    assert O.alt_is_valid(alt) is exp


@pytest.mark.parametrize("fields,a,nhom,nhet,nmiss,ac,an", V.GT_VECTORS)
def test_het_hom(fields, a, nhom, nhet, nmiss, ac, an):
    names = ["S%d" % i for i in range(len(fields))]
    homs, hets, miss, dos, rac, ran = O.het_hom(fields, a, names)
    assert (len(homs), len(hets), len(miss), rac, ran) == (nhom, nhet, nmiss, ac, an)


@pytest.mark.parametrize("k,n,exp", V.FLOAT_VECTORS)
def test_float_text(k, n, exp):
    assert O.format_float(k / n) == exp


def test_header():
    assert O.header(O.OracleConfig()).split("\t") == V.BASE_HEADER
    assert O.header(O.OracleConfig(keep_pos=True, keep_id=True, keep_info=True)).split("\t") == \
        V.BASE_HEADER + ["vcfPos", "id", "alleleIdx", "info"]
    assert O.header(O.OracleConfig(keep_info=True)).split("\t") == V.BASE_HEADER + ["alleleIdx", "info"]


@pytest.mark.parametrize("name,cfg,vcf,exp", V.STREAM_CASES, ids=[c[0] for c in V.STREAM_CASES])
def test_stream_cases(name, cfg, vcf, exp):
    r = O.read_vcf(O.OracleConfig(**cfg), vcf)
    assert r.error == 0
    assert rows_of(r.tsv) == exp


def test_dosage_matrix():
    vcf, loci, dos = V.DOSAGE_CASE
    r = O.read_vcf(O.OracleConfig(want_dosage=True), vcf)
    assert r.loci == loci
    assert r.dosage.tolist() == dos


def test_not_a_vcf_and_no_header():
    assert O.read_vcf(O.OracleConfig(), b"hello\n#CHROM\tPOS\n").error == 1
    assert O.read_vcf(O.OracleConfig(), b"##fileformat=VCFv4.2\n##x\n1\t2\n").error == 2


def test_unterminated_last_line_dropped():
    vcf = V._vcf(V.HDR8, [["1", "5", ".", "A", "C", ".", "PASS", "X"], ["1", "6", ".", "A", "G", ".", "PASS", "X"]])
    r = O.read_vcf(O.OracleConfig(), vcf[:-1])  # main.go:354-357
    assert [x[1] for x in rows_of(r.tsv)] == ["5"]


def test_golden_chr1(chr1_sample, chr1_fixture, tmp_path):
    """previous_out_check/README.md:3-10 on the sampled lines: sort both, compare.  Plus the input-order md5 of the
    sample repeated (chr1_fixture), which is the sample's rows as often."""
    r = O.read_vcf(O.OracleConfig(), chr1_sample)
    assert r.n_lines == V.GOLDEN_SAMPLE_LINES and r.n_rows == V.GOLDEN_SAMPLE_ROWS
    big = O.read_vcf(O.OracleConfig(), chr1_fixture)
    assert big.tsv == r.tsv * V.CHR1_REPEATS
    assert hashlib.md5(big.tsv).hexdigest() == V.GOLDEN_MD5_INPUT_ORDER
    with gzip.open(os.path.join(ROOT, "tests", "golden", "chr1_400lines.golden_out_10_3_18.tsv.gz")) as f:
        gold = f.read()
    head, _, body = gold.partition(b"\n")
    assert head.decode() == O.header(O.OracleConfig())
    a, b = tmp_path / "ours.tsv", tmp_path / "gold.tsv"
    a.write_bytes(r.tsv)
    b.write_bytes(body)
    env = dict(os.environ, LC_ALL="C")
    sa = subprocess.check_output(["sort", "-k1,1", "-k2,2n", "-k5,5", str(a)], env=env)
    sb = subprocess.check_output(["sort", "-k1,1", "-k2,2n", "-k5,5", str(b)], env=env)
    assert sa == sb
    assert hashlib.md5(sa).hexdigest() == V.GOLDEN_MD5_SORTED
    # threads: same bytes in the same order
    assert O.read_vcf(O.OracleConfig(), chr1_fixture, threads=4).tsv == big.tsv


def test_query_fixture_counts(query_fixture):
    """examples/test.query.vcf has no golden; SURVEY 8c probe: 879 rows, 757 SNP / 70 DEL / 52 INS."""
    r = O.read_vcf(O.OracleConfig(), query_fixture)
    rows = rows_of(r.tsv)
    assert len(rows) == 879
    types = [x[2] for x in rows]
    assert (types.count("SNP"), types.count("DEL"), types.count("INS")) == (757, 70, 52)
    assert sum(1 for x in rows if x[10] != "!") == 490
