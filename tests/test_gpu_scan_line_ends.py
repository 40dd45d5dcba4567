"""Line ends at every byte position of the scan kernel's 1 KiB window pairs, against the CPU oracle.

The scan reads its input as pairs of 512-byte windows and routes a pair that holds a newline window by window:
the window before the newline through the vector tiers, the one holding it through the general path, the one after
it through the vector tiers again when the next line's sample zone has begun.  Every line here is 1 (mod 1024) bytes
long, so over 1,024 lines the newline visits every offset of a pair, in window A and in window B, at every phase of
the sample zone mod 4, and on a window's last byte.  The fixed fields span one, two or three windows; the field
before the newline is a regular genotype, a '.' genotype, a multi-digit allele or empty; the lines end in LF or
CRLF.  Rows and diagnostics must equal the oracle's byte for byte."""
import random

import pytest

import ref_vectors as V

pytestmark = pytest.mark.gpu

N_SAMPLES = 200
LAST = {
    "regular": ["0|0", "0|1", "1|1", "1|0"],
    "dot": [".|.", "./.", ".", "0|.", ".|1"],
    "multi": ["10|1", "1|12", "0|10", "2|10"],
    "empty": [""],
}


def _line_end_vcf(rng, last, eol):
    hdr = V.HDR8 + ["FORMAT"] + ["S%06d" % i for i in range(N_SAMPLES)]
    lines = []
    for i in range(1024):
        sep = "/" if i % 5 == 4 else "|"
        gts = []
        for _ in range(N_SAMPLES - 1):
            u = rng.random()
            g = "0|0" if u < 0.85 else "0|1" if u < 0.93 else "1|1" if u < 0.96 else ".|." if u < 0.98 else "1|2"
            gts.append(g.replace("|", sep))
        gts.append(rng.choice(LAST[last]))
        ref, alt = ("A", "A") if i % 37 == 5 else ("A", "C,G") if i % 3 else ("AT", "A")  # REF == ALT: a diagnostic
        fixed = ["chr1", str(10000 + 7 * i), "rs%d" % i, ref, alt, "50", "PASS", "", "GT"]
        bare = len("\t".join(fixed + gts) + eol)
        # INFO pads the line to 1 (mod 1024) bytes; two lines in three have fixed fields one or two windows longer
        n_info = (1 - bare) % 1024
        n_info += (1024 if n_info < 3 else 0) + 1024 * (i % 3)
        fixed[7] = "X=" + "".join(rng.choice("ACGT") for _ in range(n_info - 2))
        line = "\t".join(fixed + gts) + eol
        assert len(line.encode()) % 1024 == 1
        lines.append(line)
    head = "".join(x + eol for x in [V.VERSION, "\t".join(hdr)])
    return (head + "".join(lines)).encode()


@pytest.mark.parametrize("eol", ["\n", "\r\n"], ids=["lf", "crlf"])
@pytest.mark.parametrize("last", sorted(LAST))
def test_line_end_positions_vs_oracle(last, eol):
    from bystro_vcf_b200 import Config, Transformer, parse_preamble
    from oracle import oracle as O

    vcf = _line_end_vcf(random.Random("%s-%d" % (last, len(eol))), last, eol)
    ref = O.read_vcf(O.OracleConfig(), vcf)
    w, chrom, off = parse_preamble(vcf)
    assert w == len(eol)
    c = Config()
    c.allowedFilters = {"PASS": True, ".": True}
    with Transformer(c, eol_width=w) as tr:
        tr.set_header(chrom)
        res = tr.process(vcf[off:])
    assert res.tsv == ref.tsv
    assert sorted(res.diags) == sorted(ref.diags)
    assert ref.n_rows > 900 and len(ref.diags) > 0
