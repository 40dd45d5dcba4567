"""--bgzfLevel (extension): parsed like a Go int flag by both CLIs, and refused before any device work when it is not an
integer, outside 1..9, or given without --bgzfOut."""
import os
import subprocess
import sys

import pytest

from bystro_vcf_b200 import host

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _clis():
    cmds = [[sys.executable, "-m", "bystro_vcf_b200"]]
    binary = os.path.join(ROOT, "bystro_vcf_b200", "bin", "bystro-vcf-b200")
    if os.path.exists(binary):
        cmds.append([binary])
    return cmds


def test_default_level_is_one():
    assert host.setup([]).bgzfLevel == 1
    assert host.setup(["--bgzfOut"]).bgzfLevel == 1


@pytest.mark.parametrize("flags", [["--bgzfLevel=6"], ["--bgzfLevel", "6"], ["-bgzfLevel", "6"], ["-bgzfLevel=6"]])
def test_level_syntax(flags):
    assert host.setup(["--bgzfOut"] + flags).bgzfLevel == 6
    assert host.setup(flags + ["--bgzfOut", "--keepId"]).bgzfLevel == 6
    # the C++ CLI takes the same flags: it gets as far as the input (not a VCF here), past the flag check
    for cmd in _clis():
        r = subprocess.run(cmd + ["--bgzfOut"] + flags, input=b"hello\n", capture_output=True, cwd=ROOT)
        assert r.returncode == 1 and b"Not a VCF file" in r.stderr


@pytest.mark.parametrize("flags,msg", [
    (["--bgzfOut", "--bgzfLevel", "0"], b"--bgzfLevel must be 1..9"),
    (["--bgzfOut", "--bgzfLevel", "10"], b"--bgzfLevel must be 1..9"),
    (["--bgzfOut", "--bgzfLevel", "x"], b'invalid value "x" for flag -bgzfLevel'),
    (["--bgzfOut", "--bgzfLevel=6.5"], b'invalid value "6.5" for flag -bgzfLevel'),
    (["--bgzfLevel", "6"], b"--bgzfLevel needs --bgzfOut"),
])
def test_refusals_before_any_device_work(flags, msg):
    with pytest.raises(ValueError, match=msg.decode().replace(".", r"\.")):
        host.setup(flags)
    for cmd in _clis():
        # a valid VCF on stdin: only the flag check can stop the run before the device is needed
        r = subprocess.run(cmd + flags, input=b"##fileformat=VCFv4.1\n#CHROM\tPOS\n", capture_output=True, cwd=ROOT)
        assert r.returncode == 1, (cmd, r.stderr)
        assert r.stderr.strip().count(b"\n") == 0 and msg in r.stderr, (cmd, r.stderr)
        assert r.stdout == b""
