"""The two readVcf drivers of each CLI (the streaming one, and the resident one that --bgzfOut runs) share the preamble,
the sample list, the dosage file and the log lines: --bgzfOut gives what the streaming run gives, with every output on,
from plain and .vcf.gz input, piped and from --in; a corrupt block inside the preamble is refused by both."""
import gzip
import os
import subprocess
import sys

import pytest

import ref_vectors as V

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "bystro_vcf_b200", "bin", "bystro-vcf-b200")
PY = [sys.executable, "-m", "bystro_vcf_b200"]


def _cli(cmd, data):
    return subprocess.run(cmd, input=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE, cwd=ROOT, timeout=600)


def _hosts():
    return [PY] + ([[BIN]] if os.path.exists(BIN) else [])


def _vcf(n_samples, n_rec, meta_lines=0):
    """lines that raise every kind of diagnostic, genotypes with dotted sample names, `meta_lines` long ## lines"""
    hdr = V.HDR8 + (["FORMAT"] + ["S.%03d" % i for i in range(n_samples)] if n_samples else [])
    alts = ["G", "A", "<DEL>", "G,T", "C,ATT", "TAC,T", "GT,C,N"]
    recs = []
    for i in range(n_rec):
        ref = "TAGCTT" if i % 7 == 5 else ("AT" if i % 7 in (4, 6) else "A")
        pos = "x" if i % 101 == 7 else str(100 + i)
        r = ["chr%d" % (1 + i % 3), pos, "rs%d" % i, ref, alts[i % 7], ".", "PASS", "DP=%d" % i]
        if n_samples:
            r += ["GT"] + [("0|0", "0|1", "1|1", ".|.", "1|0")[(i * 7 + j) % 5] for j in range(n_samples)]
        recs.append(r)
    vcf = V._vcf(hdr, recs)
    meta = b"".join(b"##contig=<ID=c%d,length=%s>\n" % (k, b"9" * 400) for k in range(meta_lines))
    first, _, rest = vcf.partition(b"\n")
    return first + b"\n" + meta + rest


@pytest.mark.gpu
@pytest.mark.parametrize("n_samples", [40, 0])
@pytest.mark.parametrize("route", ["pipe", "file"])
@pytest.mark.parametrize("compressed_in", [False, True])
@pytest.mark.parametrize("host", ["cpp", "python"])
def test_bgzf_out_equals_streaming_with_every_output(tmp_path, host, compressed_in, route, n_samples):
    """--bgzfOut with --dosageOutput, --sample and diagnosed lines: the decompressed rows, the Arrow file, the sample list
    and the log lines equal the streaming run's"""
    import pyarrow as pa

    from bystro_vcf_b200 import bgzf

    if host == "cpp" and not os.path.exists(BIN):
        pytest.skip("the C++ host is not built")
    vcf = _vcf(n_samples, 6000) + b"1\t5\tunterminated"
    data = bgzf.compress(vcf, block_text=9000) if compressed_in else vcf
    inp = tmp_path / ("in.vcf.gz" if compressed_in else "in.vcf")
    inp.write_bytes(data)
    base = ([BIN, "--chunkBytes", str(1 << 16)] if host == "cpp" else list(PY)) + ["--keepId", "--keepInfo"]
    got = {}
    for mode in ("stream", "bgzfOut"):
        d, s = tmp_path / ("d_%s.feather" % mode), tmp_path / ("s_%s.txt" % mode)
        cmd = base + ["--dosageOutput", str(d), "--sample", str(s)] + (["--bgzfOut"] if mode == "bgzfOut" else [])
        r = _cli(cmd + (["--in", str(inp)] if route == "file" else []), b"" if route == "file" else data)
        assert r.returncode == 0, r.stderr.decode()[-2000:]
        rows = gzip.decompress(r.stdout) if mode == "bgzfOut" else r.stdout
        got[mode] = (rows, d.read_bytes(), s.read_bytes(), r.stderr.decode().split("\n"))
    rows, dos, samples, log = got["stream"]
    assert rows.count(b"\n") > 1000 and len([x for x in log if x]) > 500
    if n_samples:
        assert samples == b"".join(b"S_%03d\n" % i for i in range(n_samples))
        assert pa.ipc.open_file(pa.py_buffer(dos)).read_all().num_rows > 1000
    else:
        assert samples == b"" and dos == b""
        assert ("No samples found in VCF file; writing empty dosage matrix file" in log) == (host == "cpp")
    assert got["bgzfOut"][0] == rows
    assert got["bgzfOut"][2:] == got["stream"][2:]
    if n_samples:
        other = got["bgzfOut"][1]
        assert pa.ipc.open_file(pa.py_buffer(other)).read_all().equals(pa.ipc.open_file(pa.py_buffer(dos)).read_all())
    else:
        assert got["bgzfOut"][1] == b""


@pytest.mark.gpu
def test_bgzf_out_mapped_bgzf_file_over_several_groups(chr1_fixture, tmp_path):
    """--bgzfOut --in x.vcf.gz: the mapped file cut into groups of whole blocks, an empty block inside the stream, text
    carried from group to group; gzip reads the rows back to what the streaming run writes"""
    from bystro_vcf_b200 import bgzf

    vcf = chr1_fixture[:140 << 20]
    cut = len(vcf) // 3 + 12345
    comp = bgzf.compress(vcf[:cut], eof=False) + bgzf.EOF_BLOCK + bgzf.compress(vcf[cut:])
    inp = tmp_path / "in.vcf.gz"
    inp.write_bytes(comp)
    plain = _cli([BIN, "--keepId"], vcf)
    assert plain.returncode == 0, plain.stderr.decode()[-2000:]
    for cmd in ([BIN, "--chunkBytes", str(1 << 16)], PY):  # C++: groups of 64 MiB of text
        r = _cli(cmd + ["--keepId", "--bgzfOut", "--in", str(inp)], b"")
        assert r.returncode == 0, r.stderr.decode()[-2000:]
        assert gzip.decompress(r.stdout) == plain.stdout


@pytest.mark.parametrize("bgzf_out", [False, True])
def test_corrupt_block_in_the_preamble_is_refused(tmp_path, bgzf_out):
    """a preamble block whose CRC-32 does not match its text: exit status 1 and the reason on stderr, piped or from --in,
    before any device work"""
    from bystro_vcf_b200 import bgzf

    vcf = _vcf(4, 50, meta_lines=60)
    comp = bytearray(bgzf.compress(vcf, block_text=5000))
    assert vcf.index(b"#CHROM") > 3 * 5000
    p = 0
    for _ in range(2):  # the third block: inside the ## lines
        p += bgzf.block_size(comp, p)
    comp[p + bgzf.block_size(comp, p) - 8] ^= 0x01  # its CRC-32
    inp = tmp_path / "in.vcf.gz"
    inp.write_bytes(bytes(comp))
    flags = ["--bgzfOut"] if bgzf_out else []
    for cmd in _hosts():
        for route in ("pipe", "file"):
            r = _cli(cmd + flags + (["--in", str(inp)] if route == "file" else []), b"" if route == "file" else bytes(comp))
            assert r.returncode == 1, (cmd, route, r.stderr[-500:])
            assert b"CRC-32" in r.stderr, (cmd, route, r.stderr[-500:])
