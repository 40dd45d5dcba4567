import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def chr1_sample():
    """400 of the 19,747 data lines of the reference's 20k-line 1000G chr1 slice (previous_out_check/) under its header,
    in input order, decompressed: 300 drawn at random among the lines with one-base REF and ALT and FILTER PASS or '.',
    100 among the others (indels, MNPs, multi-allelic sites, other filters).  tests/golden/ holds the reference's rows
    for exactly these lines."""
    import gzip

    with gzip.open(os.path.join(ROOT, "tests", "golden", "chr1_400lines.vcf.gz")) as f:
        return f.read()


@pytest.fixture(scope="session")
def chr1_fixture(chr1_sample):
    """chr1_sample's data lines CHR1_REPEATS times over under its header: about the 200 MB of the slice they come from,
    so that tests cutting tens of megabytes or many chunks out of it still see real chr1 lines at that size."""
    import ref_vectors as V

    end = chr1_sample.index(b"\n", chr1_sample.index(b"\n#CHROM") + 1) + 1
    return chr1_sample[:end] + chr1_sample[end:] * V.CHR1_REPEATS


@pytest.fixture(scope="session")
def query_fixture():
    """The reference's examples/test.query.vcf (60 samples, GT:AD:DP:GQ:PL, '/' separated)."""
    import gzip

    with gzip.open(os.path.join(ROOT, "tests", "golden", "test.query.vcf.gz")) as f:
        return f.read()
