"""CPU-only: host logic that mirrors the reference interface, the C ABI surface, the workload generator."""
import ctypes as C
import io
import os
import re

import pytest

import ref_vectors as V
import bystro_vcf_b200 as B
from bystro_vcf_b200 import _lib, host, shard, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_setup_flags_like_reference():
    """main_test.go:19-57 TestKeepFlagsTrue"""
    c = B.setup(["--keepInfo", "--keepId", "--keepPos", "--in", "/path/to/file", "--err", "/path/to/err",
                 "--cpuProfile", "/path/to/profile", "--emptyField", ".", "--out", "/path/to/out",
                 "--fieldDelimiter", "&", "--allowFilter", "PASS,., somethingElse ",
                 "--excludeFilter", "unwanted_one, unwanted_two "])
    assert c.keepInfo and c.keepID and c.keepPos
    assert (c.inPath, c.errPath, c.cpuProfile, c.outPath) == ("/path/to/file", "/path/to/err", "/path/to/profile", "/path/to/out")
    assert (c.emptyField, c.fieldDelimiter) == (".", "&")
    assert c.allowedFilters == {"PASS": True, ".": True, "somethingElse": True}
    assert c.excludedFilters == {"unwanted_one": True, "unwanted_two": True}


def test_setup_defaults_and_go_flag_syntax():
    c = B.setup([])
    assert c.allowedFilters == {"PASS": True, ".": True} and c.excludedFilters is None  # main.go:98-99
    assert (c.emptyField, c.fieldDelimiter) == ("!", ";")
    assert B.setup(["--allowFilter", "*"]).allowedFilters is None  # main.go:108
    assert B.setup(["-allowFilter="]).allowedFilters is None
    c = B.setup(["-keepId=false", "--keepInfo=true", "-out=x", "positional", "--keepPos"])
    assert (c.keepID, c.keepInfo, c.outPath, c.keepPos) == (False, True, "x", False)  # parsing stops at the first non-flag
    with pytest.raises(ValueError):
        B.setup(["--nope"])
    with pytest.raises(ValueError):
        B.setup(["--keepId=maybe"])


def test_header_like_reference():
    """main_test.go:74-169 TestHeader"""
    assert B.header(B.Config()) == V.BASE_HEADER
    assert B.header(B.Config(keepPos=True)) == V.BASE_HEADER + ["vcfPos"]
    assert B.header(B.Config(keepID=True)) == V.BASE_HEADER + ["id"]
    assert B.header(B.Config(keepInfo=True)) == V.BASE_HEADER + ["alleleIdx", "info"]
    assert B.header(B.Config(keepPos=True, keepID=True, keepInfo=True)) == V.BASE_HEADER + ["vcfPos", "id", "alleleIdx", "info"]
    assert B.string_header(B.Config()) == "\t".join(V.BASE_HEADER)


def test_c_abi_loads_and_exports_every_declared_symbol():
    L = _lib.lib()
    hdr = open(os.path.join(ROOT, "include", "bvcf.h")).read()
    declared = set(re.findall(r"\b(bvcf_[a-z_0-9]+)\s*\(", hdr))
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for s in declared:
        assert hasattr(L, s), s
    assert L.bvcf_abi_version() == 2
    assert L.bvcf_strerror(0) == b"ok" and b"newline" in L.bvcf_strerror(-4)


def test_c_abi_header_line_matches_reference():
    L = _lib.lib()
    for kw in ({}, {"keep_pos": 1}, {"keep_id": 1, "keep_info": 1}, {"keep_pos": 1, "keep_id": 1, "keep_info": 1}):
        c = _lib.CConfig()
        for k, v in kw.items():
            setattr(c, k, v)
        buf = C.create_string_buffer(512)
        n = L.bvcf_header_line(C.byref(c), buf, 512)
        cfg = B.Config(keepPos=bool(kw.get("keep_pos")), keepID=bool(kw.get("keep_id")), keepInfo=bool(kw.get("keep_info")))
        assert buf.value.decode() == B.string_header(cfg) and n == len(buf.value)


def test_no_cpu_fallback_without_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(B.BvcfError):
        B.Transformer(B.Config())


def test_parse_preamble():
    vcf = b"##fileformat=VCFv4.2\n##x=1\n#CHROM\tPOS\tID\n1\t2\t3\n"
    w, chrom, off = B.parse_preamble(vcf)
    assert (w, chrom, vcf[off:]) == (1, b"#CHROM\tPOS\tID", b"1\t2\t3\n")
    w, chrom, off = B.parse_preamble(vcf.replace(b"\n", b"\r\n"))
    assert (w, chrom) == (2, b"#CHROM\tPOS\tID")
    with pytest.raises(B.NotAVcfError, match="Not a VCF file"):
        B.parse_preamble(b"hello\n#CHROM\tPOS\n")
    with pytest.raises(B.NotAVcfError, match="No header found"):
        B.parse_preamble(b"##fileformat=VCFv4.2\n1\t2\n")


def test_sink_writes_sample_list_like_reference(tmp_path):
    """main_test.go:171-293"""
    p = tmp_path / "s.list"
    host.Sink(B.Config(sampleListPath=str(p)), "\t".join(V.HDR_S4).encode())
    assert p.read_text().split() == ["Sample1", "Sample2", "Sample3", "Sample4"]
    p2 = tmp_path / "none.list"
    host.Sink(B.Config(sampleListPath=str(p2)), "\t".join(V.HDR8).encode())
    assert p2.read_text() == ""


def test_partition_is_newline_aligned_and_exact():
    import random

    rnd = random.Random(3)
    lines = [b"x" * rnd.randint(0, 200) + b"\n" for _ in range(500)]
    data = b"HEAD\n" + b"".join(lines)
    for n in (1, 2, 3, 4, 8, 64, 1000):
        parts = shard.partition(data, 5, len(data), n)
        assert parts[0][0] == 5 and parts[-1][1] == len(data)
        assert all(a[1] == b[0] for a, b in zip(parts, parts[1:]))
        for lo, hi in parts:
            assert lo == hi or data[hi - 1:hi] == b"\n"
        assert b"".join(data[lo:hi] for lo, hi in parts) == data[5:]
    for lo, hi in shard.chunk_ranges(data, 5, len(data), 300):
        assert data[hi - 1:hi] == b"\n"
    assert b"".join(data[lo:hi] for lo, hi in shard.chunk_ranges(data, 5, len(data), 300)) == data[5:]


def test_synth_is_a_pure_function_of_seed_and_line():
    a = synth.host_lines(20130502, 2504, "chr1", 0, 64, 4)
    assert synth.host_lines(20130502, 2504, "chr1", 0, 64, 1) == a
    assert synth.host_lines(20130502, 2504, "chr1", 17, 5, 2) in a
    assert synth.host_lines(20130503, 2504, "chr1", 0, 64, 4) != a
    ls = a.split(b"\n")[:-1]
    assert len(ls) == 64 and all(len(l.split(b"\t")) == 9 + 2504 for l in ls)
    h = synth.header(20130502, 2504)
    assert h.startswith(b"##fileformat=VCFv4") and len(synth.chrom_line(20130502, 2504).rstrip().split(b"\t")) == 9 + 2504
    assert b"." not in b"".join(synth.chrom_line(20130502, 2504).split(b"\t")[9:])  # NormalizeHeader stays unexercised


def test_synth_shapes_through_the_oracle():
    from oracle import oracle as O

    for shape, ns, n, kw in (("chr1", 2504, 400, {}), ("sites", 0, 20000, {}), ("biobank", 3000, 40, {}),
                             ("chr1_filters", 2504, 400, {"allow": None, "exclude": ["LowQual"]})):
        body = synth.host_lines(7, ns, shape, 0, n)
        r = O.read_vcf(O.OracleConfig(**kw), synth.header(7, ns) + body, threads=4)
        assert r.n_lines == n and r.n_rows > n * 0.8


def test_bgzf_helpers_round_trip():
    """bystro_vcf_b200.bgzf (host side of the GPU inflate path): blocks gzip can read, header walking, preamble inflate"""
    import gzip

    from bystro_vcf_b200 import bgzf

    data = b"##fileformat=VCFv4.1\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n" + b"1\t5\t.\tA\tG\t.\tPASS\t.\n" * 20000
    comp = bgzf.compress(data, level=6, block_text=5000)
    assert gzip.decompress(comp) == data
    assert bgzf.is_bgzf(comp) and not bgzf.is_bgzf(data)
    p = n = 0
    while p < len(comp):
        bs = bgzf.block_size(comp, p)
        assert bs > 0
        p += bs
        n += 1
    assert p == len(comp) and n == -(-len(data) // 5000) + 1  # + the EOF block
    assert bgzf.block_size(comp[:10], 0) == 0  # header not complete yet
    assert bgzf.inflate_host(comp, 12000) == data[:15000]  # whole blocks until at least 12,000 bytes


def test_read_vcf_multi_is_chunk_round_robin():
    """shard.chunk_ranges cuts on newlines and covers the region; chunk k goes to device k mod N (pure host logic)"""
    from bystro_vcf_b200.shard import chunk_ranges

    data = b"".join(b"line%d\tx\n" % i for i in range(5000))
    ch = chunk_ranges(data, 0, len(data), 700)
    assert ch[0][0] == 0 and ch[-1][1] == len(data)
    assert all(a[1] == b[0] for a, b in zip(ch, ch[1:]))
    assert all(data[hi - 1:hi] == b"\n" and hi - lo <= 700 for lo, hi in ch)
    one_long = b"x" * 5000 + b"\n" + b"y\n"
    assert chunk_ranges(one_long, 0, len(one_long), 100)[0] == (0, 5001)  # a line longer than a chunk stays whole


def test_bgzf_out_flag_and_its_refusals():
    """--bgzfOut (extension): parsed like a Go bool flag by both hosts; several GPUs are refused before any device
    work, after the (compressed) header line has gone out (main.go:199 writes it before reading input)"""
    import gzip
    import subprocess
    import sys

    from bystro_vcf_b200 import host

    assert host.setup(["--bgzfOut"]).bgzfOut is True
    assert host.setup(["--bgzfOut=false", "--keepId"]).bgzfOut is False
    assert host.setup([]).bgzfOut is False
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmds = [[sys.executable, "-m", "bystro_vcf_b200"]]
    binary = os.path.join(root, "bystro_vcf_b200", "bin", "bystro-vcf-b200")
    if os.path.exists(binary):
        cmds.append([binary])
    for cmd in cmds:
        r = subprocess.run(cmd + ["--bgzfOut", "--gpus", "2"], input=b"##fileformat=VCFv4.1\n", capture_output=True, cwd=root)
        assert r.returncode == 1 and b"--bgzfOut runs on one GPU" in r.stderr
        assert gzip.decompress(r.stdout).decode().split("\t")[:3] == ["chrom", "pos", "type"]


@pytest.mark.parametrize("data,msg", [(b"hello\nworld\n", b"Not a VCF file"), (b"##fileformat=VCFv4.2\n##x\n", b"No header found")])
def test_cli_fatal_paths_like_reference(data, msg):
    """log.Fatal of readVcf (main.go:263,293) in both hosts: the TSV header line is out already (main.go:199), the
    message goes to stderr, exit status 1 -- before any device is touched"""
    import subprocess
    import sys

    cmds = [[sys.executable, "-m", "bystro_vcf_b200"]]
    binary = os.path.join(ROOT, "bystro_vcf_b200", "bin", "bystro-vcf-b200")
    if os.path.exists(binary):
        cmds.append([binary])
    for cmd in cmds:
        r = subprocess.run(cmd, input=data, capture_output=True, cwd=ROOT)
        assert r.returncode == 1
        assert msg in r.stderr
        assert r.stdout.decode().rstrip("\n").split("\t") == V.BASE_HEADER


def test_cli_flag_errors_like_reference():
    """main.go:160,164: --noOut with --out, --noOut without --dosageOutput"""
    import subprocess
    import sys

    cmds = [[sys.executable, "-m", "bystro_vcf_b200"]]
    binary = os.path.join(ROOT, "bystro_vcf_b200", "bin", "bystro-vcf-b200")
    if os.path.exists(binary):
        cmds.append([binary])
    for cmd in cmds:
        r = subprocess.run(cmd + ["--noOut", "--out", "x.tsv"], input=b"", capture_output=True, cwd=ROOT)
        assert r.returncode == 1 and b"Cannot specify --noOut and --out" in r.stderr
        r = subprocess.run(cmd + ["--noOut"], input=b"", capture_output=True, cwd=ROOT)
        assert r.returncode == 1 and b"When specifying --noOut, must specify --dosageOutput" in r.stderr
