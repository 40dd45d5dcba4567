"""--regions / --regionsFile on a real GPU: the records outside the regions are dropped by the region filter stage, and the
output equals the unchanged program's on the input with those data lines deleted -- rows, dosage rows, diagnostics and
log lines -- on the streaming slots, the resident path and both CLIs."""
import bisect
import gzip
import os
import random
import subprocess
import sys

import pytest

import ref_vectors as V

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "bystro_vcf_b200", "bin", "bystro-vcf-b200")
MAX = (1 << 63) - 1
CHROMS = ["1", "10", "chr1", "chr10", "1_random"]  # names that are prefixes of each other
LONG = "L" * 70000                                 # a CHROM that ends past the scan kernel's 64 KiB tab window


def _cfg(**kw):
    from bystro_vcf_b200 import Config

    c = Config(allowedFilters={"PASS": True, ".": True})
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def synth(seed, n, n_samples=4, crlf=False, long_chrom=False, sort=False):
    """a VCF with leading-zero, non-digit and 19-digit POS, wrong-width lines and alleles that log diagnostics"""
    rng = random.Random(seed)
    hdr = V.HDR8 + (["FORMAT"] + ["S%d.x" % i for i in range(n_samples)] if n_samples else [])
    pos = {c: 0 for c in CHROMS + [LONG]}
    recs = []
    for i in range(n):
        c = LONG if long_chrom and i % 50 == 7 else rng.choice(CHROMS)
        pos[c] += rng.randint(1, 40)
        p, r = str(pos[c]), rng.random()
        if r < 0.03:
            p = "0" * rng.randint(1, 3) + p
        elif r < 0.05:
            p = p + "a"
        elif r < 0.06:
            p = "1" * 19
        alt = rng.choice(["G", "T", "G,T", "<DEL>", "A", "AT", "C"])
        rec = [c, p, "rs%d" % i, "A", alt, ".", rng.choice(["PASS", ".", "q10"]), "DP=%d" % i]
        if n_samples:
            rec += ["GT"] + [rng.choice(["0|0", "0|1", "1|1", ".|.", "1|2", "0/1"]) for _ in range(n_samples)]
        if rng.random() < 0.02:
            rec = rec[:-1]  # wrong width: not a record
        recs.append(rec)
    if sort:
        recs.sort(key=lambda r: (CHROMS.index(r[0]) if r[0] in CHROMS else 99, int(r[1]) if r[1].isdigit() else 0))
    eol = "\r\n" if crlf else "\n"
    return ("%s%s%s%s" % (V.VERSION, eol, "\t".join(hdr), eol) + "".join("\t".join(r) + eol for r in recs)).encode()


def merged(regions):
    m = {}
    for c, b, e in sorted((c if isinstance(c, bytes) else c.encode(), b, e) for c, b, e in regions):
        iv = m.setdefault(c, [])
        if iv and b <= iv[-1][1] + 1:
            iv[-1][1] = max(iv[-1][1], e)
        else:
            iv.append([b, e])
    return {c: ([x[0] for x in v], [x[1] for x in v]) for c, v in m.items()}


def in_regions(line: bytes, m) -> bool:
    f = line.split(b"\t", 2)
    if len(f) < 3 or not (1 <= len(f[1]) <= 18 and f[1].isdigit()) or f[0] not in m:
        return False
    v, (begs, ends) = int(f[1]), m[f[0]]
    k = bisect.bisect_right(begs, v) - 1
    return k >= 0 and v <= ends[k]


def split(vcf: bytes):
    """(meta lines + #CHROM line, data lines)"""
    end = vcf.index(b"\n", vcf.index(b"\n#CHROM") + 1) + 1
    return vcf[:end], vcf[end:].splitlines(keepends=True)


def prefiltered(vcf: bytes, regions) -> bytes:
    head, lines = split(vcf)
    m = merged(regions)
    return head + b"".join(l for l in lines if in_regions(l, m))


def random_regions(seed, n, span=400, max_pos=6000):
    rng = random.Random(seed)
    out = []
    for _ in range(n):
        b = rng.randint(1, max_pos)
        out.append((rng.choice(CHROMS).encode(), b, b + rng.randint(0, span)))
    return out


FLAGSETS = {
    "default": {},
    "keep": dict(keepID=True, keepInfo=True, keepPos=True),
    "filters": dict(allowedFilters={"PASS": True, "q10": True}, excludedFilters={"q10": True}),
    "dosage": dict(dosageMatrixOutPath="x.arrow"),
}
ORACLE = {
    "default": {},
    "keep": dict(keep_id=True, keep_info=True, keep_pos=True),
    "filters": dict(allow=["PASS", "q10"], exclude=["q10"]),
    "dosage": dict(want_dosage=True),
}


def diag_texts(lines, diags):
    """(line text, ALT number, code) of each diagnostic: line numbers are chunk-relative, the lines themselves are not"""
    return sorted((lines[ln], alt, code) for ln, alt, code in diags)


def check_chunk(vcf, regions, flags, **tr_kw):
    """one streaming-slot chunk through the C ABI against the CPU oracle on the pre-filtered input"""
    from bystro_vcf_b200 import Transformer, parse_preamble
    from oracle import oracle as O

    w, chrom, off = parse_preamble(vcf)
    cfg = _cfg(**FLAGSETS[flags])
    ref_in = prefiltered(vcf, regions)
    ref = O.read_vcf(O.OracleConfig(**ORACLE[flags]), ref_in)
    with Transformer(cfg, eol_width=w, **tr_kw) as tr:
        tr.set_header(chrom)
        tr.set_regions(regions)
        res = tr.process(vcf[off:])
    assert res.tsv == ref.tsv
    assert res.n_rows == ref.n_rows
    if flags == "dosage" and ref.n_rows:
        assert res.loci == ref.loci
        assert (res.dosage == ref.dosage).all()
    got = sorted((vcf[off + s:vcf.index(b"\n", off + s) + 1], a, c) for s, (_, a, c) in zip(res.diag_starts, res.diags))
    assert got == diag_texts(split(ref_in)[1], ref.diags)
    return res, ref


@pytest.mark.parametrize("flags", list(FLAGSETS))
@pytest.mark.parametrize("seed", [1, 2])
def test_slot_parity_random_regions(flags, seed):
    vcf = synth(seed, 3000, crlf=seed == 2, long_chrom=True)
    regions = random_regions(seed, 12) + [(LONG, 1, 3000)]
    res, ref = check_chunk(vcf, regions, flags)
    assert 0 < ref.n_rows < res.n_records


def test_slot_parity_edges_of_intervals():
    """records at exactly beg / end and one off, overlapping and adjacent intervals, a 0-based-looking beg"""
    vcf = synth(3, 2000, n_samples=0)
    _, lines = split(vcf)
    regions = []
    for l in lines[::97]:
        f = l.split(b"\t")
        if f[1].isdigit() and 1 < int(f[1]) < 10 ** 17:
            p = int(f[1])
            regions += [(f[0], p, p + 5), (f[0], p + 6, p + 9), (f[0], p - 1, p - 1), (f[0], p + 3, p + 4)]
    check_chunk(vcf, regions, "keep")
    check_chunk(vcf, [(c, b + 1, e - 1) for c, b, e in regions if e - 1 >= b + 1], "default")


def test_slot_keeps_nothing_and_everything():
    vcf = synth(4, 1500)
    res, ref = check_chunk(vcf, [(b"chr1", 10 ** 17, MAX), (b"absent", 1, MAX)], "dosage")
    assert res.tsv == b"" and ref.n_rows == 0 and res.n_records > 0
    res, ref = check_chunk(vcf, [(c.encode(), 1, MAX) for c in CHROMS], "default")
    assert ref.n_rows > 500


def test_slot_100k_intervals():
    vcf = synth(5, 4000, n_samples=2)
    rng = random.Random(5)
    regions = [(rng.choice(CHROMS), b, b + rng.randint(0, 3)) for b in (rng.randint(1, 40000) for _ in range(100000))]
    res, ref = check_chunk(vcf, regions, "keep")
    assert ref.n_rows > 0


def test_resident_small_subchunks_with_an_empty_one():
    """the resident path cut into 64 KiB sub-chunks, the later ones keeping nothing"""
    from bystro_vcf_b200 import Transformer, parse_preamble
    from oracle import oracle as O

    vcf = synth(6, 6000, sort=True)
    regions = [(b"1", 1, 3000), (b"10", 500, 900)]
    w, chrom, off = parse_preamble(vcf)
    ref = O.read_vcf(O.OracleConfig(keep_id=True), prefiltered(vcf, regions))
    with Transformer(_cfg(keepID=True), eol_width=w, resident_subchunk_bytes=64 << 10) as tr:
        tr.set_header(chrom)
        tr.set_regions(regions)
        tr.resident_alloc(len(vcf), len(vcf) * 4)
        tr.resident_upload(0, vcf)
        stats, times = tr.resident_run(len(vcf), begin=off)
        assert tr.resident_download(0, stats["out_bytes"]) == ref.tsv
        _, _, diags = tr.resident_results()
        assert len(diags) == len(ref.diags)
        assert stats["n_rows"] == ref.n_rows


def test_streaming_64k_chunks_rows_and_log_lines():
    """read_vcf in 64 KiB chunks (some keep nothing) against the unchanged program on the pre-filtered input"""
    import io

    from bystro_vcf_b200 import read_vcf

    vcf = synth(7, 8000, sort=True, long_chrom=True)
    regions = [(b"chr1", 1, 2000), (b"1_random", 100, 99999), (LONG, 1, MAX)]
    got, exp = [], []
    out1, out2 = io.BytesIO(), io.BytesIO()
    read_vcf(_cfg(chunkBytes=1 << 16, regions=regions), io.BytesIO(vcf), out1, diag_sink=lambda t, *a: got.append(t))
    read_vcf(_cfg(chunkBytes=1 << 16), io.BytesIO(prefiltered(vcf, regions)), out2, diag_sink=lambda t, *a: exp.append(t))
    assert out1.getvalue() == out2.getvalue() and out1.getvalue()
    assert got == exp and got


def test_no_regions_means_no_extra_launch():
    from bystro_vcf_b200 import Transformer, parse_preamble

    vcf = synth(8, 2000)
    w, chrom, off = parse_preamble(vcf)
    counts = []
    for regions in (None, [], [(b"1", 1, MAX)]):
        with Transformer(_cfg(), eol_width=w) as tr:
            tr.set_header(chrom)
            if regions is not None:
                tr.set_regions([(b"chr1", 1, 5)])
                tr.set_regions(regions)  # [] clears
            tr.process(vcf[off:])
            counts.append(tr.launches)
    assert counts[0] == counts[1]
    assert counts[2] == counts[0] + 2


def test_set_regions_refusals():
    from bystro_vcf_b200 import Transformer
    from bystro_vcf_b200._lib import BvcfError

    with Transformer(_cfg()) as tr:
        for bad in ([(b"1", 0, 5)], [(b"1", 6, 5)], [(b"", 1, 5)]):
            with pytest.raises(BvcfError, match=r"\(-1\)"):
                tr.set_regions(bad)
        tr.set_header(b"\t".join(x.encode() for x in V.HDR8))
        tr.submit(0, b"1\t5\t.\tA\tG\t.\tPASS\t.\n")
        with pytest.raises(BvcfError, match=r"\(-3\)"):
            tr.set_regions([(b"1", 1, 5)])
        tr.collect(0)


# ---- both CLIs --------------------------------------------------------------------------------------------------------

def _run(cmd, stdin=b""):
    p = subprocess.run(cmd, input=stdin, capture_output=True, cwd=ROOT, timeout=600)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    return p.stdout, p.stderr


def _clis():
    """the two CLIs; the C++ one cut into 64 KiB chunks"""
    return {"cpp": [BIN, "--chunkBytes", str(1 << 16)], "python": [sys.executable, "-m", "bystro_vcf_b200"]}


@pytest.mark.parametrize("host", ["cpp", "python"])
def test_cli_inputs_agree(host, tmp_path):
    """plain --in, a pipe, bgzf --in; several workers; --bgzfOut at levels 1 and 6: all equal the plain run on the
    pre-filtered input (rows, sample list, log lines)"""
    from bystro_vcf_b200 import bgzf

    vcf = synth(9, 20000, sort=True)
    regions = "chr1:1-3000,10:2000-,1_random"
    parsed = [(b"chr1", 1, 3000), (b"10", 2000, MAX), (b"1_random", 1, MAX)]
    bed = tmp_path / "r.bed"
    bed.write_bytes(b"track name=x\n# c\nchr1\t0\t3000\textra\n10\t1999\t%d\n1_random\t0\t%d\n" % (MAX, MAX))
    plain, gz, ref = tmp_path / "in.vcf", tmp_path / "in.vcf.gz", tmp_path / "ref.vcf"
    plain.write_bytes(vcf)
    gz.write_bytes(bgzf.compress(vcf, block_text=4000))
    ref.write_bytes(prefiltered(vcf, parsed))
    cmd = _clis()[host]
    common = ["--keepId", "--sample"]
    exp_out, exp_err = _run(cmd + common + [str(tmp_path / "s0.txt"), "--in", str(ref)])
    assert exp_out.count(b"\n") > 100
    runs = [["--in", str(plain), "--regions", regions], ["--in", str(gz), "--regionsFile", str(bed)],
            ["--regions", regions]]
    if host == "cpp":
        runs.append(["--in", str(gz), "--regions", regions, "--devices", "0,0"])
    runs.append(["--regions", regions])  # bgzf through a pipe
    for i, extra in enumerate(runs):
        s = tmp_path / ("s%d.txt" % (i + 1))
        stdin = b"" if "--in" in extra else (gz.read_bytes() if i == len(runs) - 1 else vcf)
        out, err = _run(cmd + common + [str(s)] + extra, stdin=stdin)
        assert out == exp_out, extra
        assert sorted(err.splitlines()) == sorted(exp_err.splitlines()), extra
        assert s.read_bytes() == (tmp_path / "s0.txt").read_bytes()
    for level in ([], ["--bgzfLevel", "6"]):
        for src in (plain, gz):
            out, err = _run(cmd + ["--keepId", "--bgzfOut", "--in", str(src), "--regions", regions] + level)
            assert gzip.decompress(out) == exp_out
            assert sorted(err.splitlines()) == sorted(exp_err.splitlines())


@pytest.mark.parametrize("flags", list(FLAGSETS))
def test_slot_parity_chr1(chr1_sample, flags):
    _, lines = split(chr1_sample)
    rng = random.Random(11)
    pos = sorted(int(l.split(b"\t")[1]) for l in lines)
    regions = [(b"1", p, p + rng.randint(0, 20000)) for p in rng.sample(pos, 15)] + [(b"chr1", 1, MAX)]
    res, ref = check_chunk(chr1_sample, regions, flags)
    assert 0 < ref.n_rows


@pytest.mark.parametrize("host", ["cpp", "python"])
def test_cli_index_prunes(host, tmp_path):
    """with a .tbi or .csi beside the file only the blocks of its spans are read: the payloads of every other block (past
    the first megabyte, which the preamble reader inflates) are corrupted, and the run still equals the plain run on the
    pre-filtered input -- without the index the same file fails on a corrupt block"""
    from bystro_vcf_b200 import bgzf
    from test_regions_cpu import index_of

    vcf = synth(12, 60000, n_samples=2, sort=True)
    regions = "chr10:2000-5000,1_random:30000-60000,1_random:90000-90000"
    parsed = [(b"chr10", 2000, 5000), (b"1_random", 30000, 60000), (b"1_random", 90000, 90000)]
    cmd = _clis()[host] + ["--keepId", "--keepInfo"]
    ref = tmp_path / "ref.vcf"
    ref.write_bytes(prefiltered(vcf, parsed))
    exp_out, exp_err = _run(cmd + ["--in", str(ref)])
    assert exp_out.count(b"\n") > 50
    comp = bytearray(bgzf.compress(vcf, block_text=4000))
    gz = tmp_path / "in.vcf.gz"
    for kind, ext in (("tbi", ".tbi"), ("csi", ".csi")):
        gz.write_bytes(bytes(comp))
        idx = tmp_path / ("in.vcf.gz" + ext)
        idx.write_bytes(bgzf.compress(index_of(vcf, 4000, **({"csi": True} if kind == "csi" else {}))))
        views = bgzf.index_views(bytes(comp), str(gz), parsed)
        assert views and sum(hi - lo for lo, hi, _ in views) < len(comp) // 4
        for extra in ([], ["--bgzfOut"]):
            out, err = _run(cmd + ["--in", str(gz), "--regions", regions] + extra)
            assert (gzip.decompress(out) if extra else out) == exp_out
            assert sorted(err.splitlines()) == sorted(exp_err.splitlines())
        bad = bytearray(comp)
        used = [False] * len(bad)
        for lo, hi, _ in views:
            used[lo:hi] = [True] * (hi - lo)
        n_bad = 0
        for off, size, isize in bgzf.blocks(bytes(comp)):
            if off > (1 << 20) // 2 and not used[off] and isize:
                bad[off + 18:off + size - 8] = bytes(size - 26)
                n_bad += 1
        assert n_bad > 100
        gz.write_bytes(bytes(bad))
        for extra in ([], ["--bgzfOut"]):
            out, err = _run(cmd + ["--in", str(gz), "--regions", regions] + extra)
            assert (gzip.decompress(out) if extra else out) == exp_out
        os.remove(idx)
        p = subprocess.run(cmd + ["--in", str(gz), "--regions", regions], capture_output=True, cwd=ROOT, timeout=600)
        assert p.returncode == 1 and (b"corrupt" in p.stderr or b"failed to inflate" in p.stderr), p.stderr[-500:]
