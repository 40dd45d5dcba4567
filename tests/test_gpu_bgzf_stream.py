"""bgzf (.vcf.gz) input on the streaming path: groups of whole blocks through bvcf_submit_bgzf, inflated on the GPU with
every member's CRC-32 checked there, several chunks in flight; the CLIs on several workers; corrupt members rejected."""
import os
import random
import struct
import subprocess
import sys
import zlib

import pytest

import ref_vectors as V
from test_gpu_parity import _cfg

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "bystro_vcf_b200", "bin", "bystro-vcf-b200")


def _vcf_with_diags(n_samples, n_rec, seed=5):
    rng = random.Random(seed)
    hdr = V.HDR8 + (["FORMAT"] + ["SM%05d" % i for i in range(n_samples)] if n_samples else [])
    recs = []
    for i in range(n_rec):
        alt = "<DEL>" if i % 37 == 3 else ("G,T" if i % 7 == 0 else ("A" if i % 53 == 1 else "G"))
        r = ["chr%d" % (1 + i % 3), str(100 + i), "rs%d" % i, "A", alt, ".", "PASS", "DP=%d" % i]
        if n_samples:
            r += ["GT"] + [rng.choice(["0|0", "0|0", "0|1", "1|1", ".|."]) for _ in range(n_samples)]
        recs.append(r)
    return V._vcf(hdr, recs)


def _stream(vcf, cfg, chunk_bytes, block_text, level=6, **tr_kw):
    """vcf -> bgzf -> plan_groups -> submit_bgzf with three chunks in flight; results in group order"""
    from bystro_vcf_b200 import Transformer, bgzf, parse_preamble

    w, chrom, off = parse_preamble(vcf)
    comp = bgzf.compress(vcf, level=level, block_text=block_text)
    groups = bgzf.plan_groups(comp, off, chunk_bytes, 1 << 30)
    res = []
    with Transformer(cfg, eol_width=w, n_slots=3, **tr_kw) as tr:
        tr.set_header(chrom)
        sub = 0
        for col in range(len(groups)):
            while sub < len(groups) and sub - col < 3:
                g = groups[sub]
                tr.submit_bgzf(sub, comp[g.lo:g.hi], g.skip, g.tail)
                sub += 1
            res.append(tr.collect(col, diag_fields=True))
    return groups, res


@pytest.mark.parametrize("n_samples,n_rec,chunk,block", [(0, 20000, 1 << 16, 777), (40, 6000, 1 << 16, 20000),
                                                         (30000, 12, 1 << 16, 65280), (3, 3000, 1 << 17, 1)])
def test_submit_bgzf_matches_process(n_samples, n_rec, chunk, block):
    """rows, dosage matrix, diagnostics and their CHROM / POS fields: byte for byte what process() gives on the plain
    text; the 30,000-sample lines are longer than a group"""
    import numpy as np

    from bystro_vcf_b200 import Transformer, parse_preamble
    from bystro_vcf_b200.host import locus_at

    vcf = _vcf_with_diags(n_samples, n_rec)
    cfg = _cfg()
    cfg.dosageMatrixOutPath = "unused" if n_samples else ""
    w, chrom, off = parse_preamble(vcf)
    with Transformer(cfg, eol_width=w, max_chunk_bytes=len(vcf) + 1) as tr:
        tr.set_header(chrom)
        ref = tr.process(vcf[off:])
    groups, res = _stream(vcf, cfg, chunk, block, max_chunk_bytes=1 << 30)
    assert len(groups) > 1
    assert b"".join(r.tsv for r in res) == ref.tsv
    assert sum(r.n_lines for r in res) == ref.n_lines
    diags, fields, base = [], [], 0
    for r in res:
        diags += [(ln + base, a, c) for ln, a, c in r.diags]
        fields += r.diag_fields
        base += r.n_lines
    assert diags == ref.diags and len(diags) > 0
    assert fields == [locus_at(vcf, off + st) for st in ref.diag_starts]
    if n_samples:
        assert sum((r.loci for r in res), []) == ref.loci
        assert np.array_equal(np.concatenate([r.dosage for r in res if r.dosage is not None]), ref.dosage)


def test_diagnostics_across_slots(monkeypatch):
    """a diagnostics buffer of 16 entries, many groups with hundreds of diagnostics each, three in flight: every slot
    grows to what it needs and every diagnostic arrives"""
    from oracle import oracle as O

    monkeypatch.setenv("BVCF_DIAG_CAP", "16")
    recs = [["1", str(5 + i), ".", "A", "<DEL>" if i % 2 else "A", ".", "PASS", "."] for i in range(30000)]
    vcf = V._vcf(V.HDR8, recs)
    ref = O.read_vcf(O.OracleConfig(), vcf)
    groups, res = _stream(vcf, _cfg(), 1 << 16, 4000)
    assert len(groups) >= 8
    got, base = [], 0
    for r in res:
        got += [(ln + base, a, c) for ln, a, c in r.diags]
        base += r.n_lines
    assert got == ref.diags and len(got) == 30000
    assert b"".join(r.tsv for r in res) == ref.tsv


# ---- corrupt members -----------------------------------------------------------------------------------------------
def _member(payload, text, crc=None):
    from bystro_vcf_b200 import bgzf

    return (bgzf.MAGIC + b"\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(payload) + 25) + payload +
            struct.pack("<II", zlib.crc32(text) if crc is None else crc, len(text)))


def _corrupt_cases(text):
    """(name, bgzf bytes) of three corrupt single-member files whose ISIZE matches the text"""
    from bystro_vcf_b200 import bgzf

    good = bgzf.compress(text, eof=False)
    crc_flipped = bytearray(good)
    crc_flipped[-8] ^= 0x01
    stored = bytearray(bgzf.compress(text, level=0, eof=False))
    stored[18 + 5 + len(text) // 2] ^= 0x20  # a literal of the stored block: same length, other text
    # empty fixed-Huffman blocks, none of them final: 10 bits each (BFINAL 0, BTYPE 01, end-of-block code 0000000)
    bits = "0" + "10" + "0000000"
    chain = (bits * 400)[:8 * 500]
    payload = bytes(int(chain[i:i + 8][::-1], 2) for i in range(0, len(chain), 8))
    return [("crc", bytes(crc_flipped)), ("stored-literal", bytes(stored)), ("empty-chain", _member(payload, text))]


def _text_vcf():
    return _vcf_with_diags(4, 300)


def test_corrupt_members_rejected_by_both_entry_points():
    from bystro_vcf_b200 import BvcfError, Transformer, parse_preamble

    vcf = _text_vcf()
    w, chrom, off = parse_preamble(vcf)
    body = vcf[off:]
    for name, comp in _corrupt_cases(body):
        with Transformer(_cfg(), eol_width=w) as tr:
            tr.set_header(chrom)
            tr.submit_bgzf(0, comp, 0, b"")
            with pytest.raises(BvcfError) as e:
                tr.collect(0)
            assert "(-1)" in str(e.value), name
            if name != "empty-chain":
                assert "CRC-32" in str(e.value), name
            tr.resident_alloc(len(body) + 1024, 4096)
            with pytest.raises(BvcfError):
                tr.resident_inflate_bgzf(comp + b"")
        # the same member intact goes through
    from bystro_vcf_b200 import bgzf

    with Transformer(_cfg(), eol_width=w) as tr:
        tr.set_header(chrom)
        tr.submit_bgzf(0, bgzf.compress(body, eof=False), 0, b"")
        assert tr.collect(0).n_lines == 300


def _cli(cmd, data, **kw):
    return subprocess.run(cmd, input=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE, cwd=ROOT, timeout=600, **kw)


def _devices():
    """two workers: two GPUs when the box has them, the same GPU twice otherwise"""
    import torch

    return "0,1" if torch.cuda.device_count() >= 2 else "0,0"


def _python_two_workers():
    """the Python CLI on two workers: --gpus 2, or on a one-GPU box the same host code on device 0 twice"""
    if _devices() == "0,1":
        return [sys.executable, "-m", "bystro_vcf_b200", "--gpus", "2"]
    code = ("import sys; from bystro_vcf_b200 import host, shard; from bystro_vcf_b200.__main__ import main; "
            "f = shard.read_vcf_multi; shard.read_vcf_multi = lambda c, d, w, devs, **k: f(c, d, w, [0, 0], **k); "
            "sys.exit(main(['--gpus', '2'] + sys.argv[1:]))")
    return [sys.executable, "-c", code]


def test_corrupt_members_rejected_by_both_clis(tmp_path):
    from bystro_vcf_b200 import bgzf, parse_preamble

    vcf = _text_vcf()
    _, _, off = parse_preamble(vcf)
    for name, comp in _corrupt_cases(vcf[off:]):
        data = bgzf.compress(vcf[:off], eof=False) + comp + bgzf.EOF_BLOCK
        p = tmp_path / "in.vcf.gz"
        p.write_bytes(data)
        for cmd in ([BIN, "--devices", _devices()], [BIN, "--in", str(p)], _python_two_workers(), [sys.executable, "-m", "bystro_vcf_b200"]):
            r = _cli(cmd, data if "--in" not in cmd else b"")
            assert r.returncode == 1, (name, cmd, r.stderr[-500:])
            assert r.stderr.strip(), (name, cmd)


@pytest.mark.parametrize("host", ["cpp-file", "cpp-pipe", "python"])
def test_cli_bgzf_several_workers_match_plain(chr1_fixture, tmp_path, host):
    """two workers (two GPUs, or one GPU twice) and one: exactly the bytes of the plain single-GPU run, small groups and
    777-byte blocks, an unterminated last line"""
    from bystro_vcf_b200 import bgzf

    vcf = chr1_fixture[:12 << 20].rsplit(b"\n", 1)[0] + b"\n" + b"1\t5\tunterminated"
    flags = ["--keepId", "--keepInfo"]
    plain = _cli([BIN] + flags, vcf).stdout
    comp = bgzf.compress(vcf, block_text=777)
    p = tmp_path / "in.vcf.gz"
    p.write_bytes(comp)
    for workers in (["--devices", _devices()], ["--gpus", "1"]):
        if host == "python":
            cmd = _python_two_workers() if workers[0] == "--devices" else [sys.executable, "-m", "bystro_vcf_b200", "--gpus", "1"]
        else:
            cmd = [BIN, "--chunkBytes", str(1 << 20)] + workers
        if host == "cpp-file":
            r = _cli(cmd + ["--in", str(p)] + flags, b"")
        else:
            r = _cli(cmd + flags, comp)
        assert r.returncode == 0, r.stderr.decode()[-2000:]
        assert r.stdout == plain


@pytest.mark.parametrize("host", ["cpp", "python"])
def test_cli_bgzf_two_workers_dosage_and_log_lines(tmp_path, host):
    """the Arrow dosage file and the log lines from a .vcf.gz on two workers equal the oracle's"""
    import numpy as np
    import pyarrow as pa

    from bystro_vcf_b200 import bgzf
    from oracle import oracle as O

    n = 40
    vcf = _vcf_with_diags(n, 8000)
    ref = O.read_vcf(O.OracleConfig(want_dosage=True), vcf)
    comp = bgzf.compress(vcf, block_text=5000)
    path = tmp_path / "d.feather"
    if host == "cpp":
        cmd = [BIN, "--devices", _devices(), "--chunkBytes", str(1 << 16)]
    else:
        cmd = _python_two_workers()
    r = _cli(cmd + ["--dosageOutput", str(path)], comp)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    assert r.stdout.partition(b"\n")[2] == ref.tsv
    tab = pa.ipc.open_file(str(path)).read_all()
    assert [x.encode() for x in tab.column(0).to_pylist()] == ref.loci
    assert np.array_equal(np.stack([tab.column(j + 1).to_numpy() for j in range(n)], axis=1), ref.dosage)
    from bystro_vcf_b200 import parse_preamble
    from bystro_vcf_b200.host import format_diag

    _, _, off = parse_preamble(vcf)
    lines = vcf[off:].split(b"\n")
    exp = [format_diag(*(lines[ln].split(b"\t")[0].decode(), lines[ln].split(b"\t")[1].decode()), a, c) for ln, a, c in ref.diags]
    assert sorted(r.stderr.decode().strip().split("\n")) == sorted(exp) and len(exp) > 100
