"""Known-answer vectors transcribed from the reference's own tests (/root/reference/main_test.go).

Each block cites the main_test.go lines it was transcribed from.  Full expected rows were written
out by hand from the reference semantics and agree with every column the Go test asserts.
These vectors are shared by the oracle tests (CPU) and the CUDA parity tests (GPU).
"""

VERSION = "##fileformat=VCFv4.x"
HDR8 = ["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO"]
HDR_S4 = HDR8 + ["FORMAT", "Sample1", "Sample2", "Sample3", "Sample4"]

# ---- getAlleles: main_test.go:295-522 (TestUpdateFieldsWithAlt) ----
# (pos, ref, alt) -> (type, positions, refs, alts, altIndices)
ALLELE_VECTORS = [
    (("100", "T", "C"), ("SNP", ["100"], ["T"], ["C"], [0])),  # :296-308
    (("100", "TCCT", "TCCA"), ("SNP", ["103"], ["T"], ["A"], [0])),  # :310-318
    (("100", "TGCT", "TGAT"), ("SNP", ["102"], ["C"], ["A"], [0])),  # :320-328
    (("100", "TGCT", "AGCT"), ("SNP", ["100"], ["T"], ["A"], [0])),  # :330-338
    (("100", "TCGT", "GTAA"), ("MNP", ["100", "101", "102", "103"], list("TCGT"), list("GTAA"), [0, 0, 0, 0])),  # :340-371
    (("100", "TCGT", "TAGC"), ("MNP", ["101", "103"], ["C", "T"], ["A", "C"], [0, 0])),  # :373-404
    (("100", "TCGT", "TCGC"), ("SNP", ["103"], ["T"], ["C"], [0])),  # :406-436
    (("100", "TC", "T"), ("DEL", ["101"], ["C"], ["-1"], [0])),  # :438-447
    (("100", "TAGCGT", "T"), ("DEL", ["101"], ["A"], ["-5"], [0])),  # :449-457
    (("100", "TAGCTT", "TA"), ("DEL", ["102"], ["G"], ["-4"], [0])),  # :459-468
    (("100", "TAGCTT", "TAC"), ("", [], [], [], [])),  # :470-479 malformed
    (("100", "TAGCTT", "TAT"), ("DEL", ["102"], ["G"], ["-3"], [0])),  # :481-497
    (("100", "T", "TAGCTT"), ("INS", ["100"], ["T"], ["+AGCTT"], [0])),  # :499-509
    (("100", "TT", "TAGCTT"), ("INS", ["100"], ["T"], ["+AGCT"], [0])),  # :511-521
]

# ---- altIsValid: main_test.go:571-650 ----
ALT_VALID_VECTORS = [
    ("ACTG", True), (".", False), ("]13 : 123456]T", False), ("C[2 : 321682[", False),
    (".A", False), ("G.", False), ("<DUP>", False), ("A,C", False),
]

# ---- linePasses: main_test.go:524-569 (FILTER value, allow, exclude) -> passes ----
FILTER_VECTORS = [
    ("PASS", ["PASS", "."], None, True),
    (".", ["PASS", "."], None, True),
    ("blah", None, None, True),
    ("blah", None, ["blah"], False),
]

# ---- makeHetHomozygotes: main_test.go:652-951 ----
# (sample fields, alleleNum, n_hom, n_het, n_missing, ac, an)
GT_VECTORS = [
    (["0|0", "0|0", "0|0", "0|0"], "1", 0, 0, 0, 0, 8),  # :660-677
    (["0|1", "0|1", "0|1", "0|1"], "1", 0, 4, 0, 4, 8),  # :679-697
    ([".|.", ".|.", ".|1", "1|."], "1", 0, 0, 4, 0, 0),  # :699-717
    ([".|1", "0|1", "0|1", "0|1"], "1", 0, 3, 1, 3, 6),  # :719-739
    (["1|.", "0|1", "0|1", "0|1"], "1", 0, 3, 1, 3, 6),  # :741-759
    (["1|1", "1|1", "0|1", "0|1"], "1", 2, 2, 0, 6, 8),  # :761-779
    (["1|2", "1|1", "0|1", "0|1"], "1", 1, 3, 0, 5, 8),  # :781-802
    (["1|2", "1|1", "0|1", "0|1"], "2", 0, 1, 0, 1, 8),  # :804-822
    (["1|2:-0.03,-1.12,-5.00", "1|1:-0.03,-1.12,-5.00", "0|1:-0.03,-1.12,-5.00", "0|1:-0.03,-1.12,-5.00"], "2", 0, 1, 0, 1, 8),  # :824-842
    (["1|2|1:-0.03,-1.12,-5.00", "1|1:-0.03,-1.12,-5.00", "0|1:-0.03,-1.12,-5.00", "0|1:-0.03,-1.12,-5.00"], "2", 0, 1, 0, 1, 9),  # :844-862
    (["1|2|1", "1|1", "0|1", "0|1"], "2", 0, 1, 0, 1, 9),  # :864-882
    (["2|2|2:-0.03,-1.12,-5.00", "1|1:-0.03,-1.12,-5.00", "0|1:-0.03,-1.12,-5.00", "0|1:-0.03,-1.12,-5.00"], "2", 1, 0, 0, 3, 9),  # :884-894
    (["2|2|2", "1|1", "0|1", "0|1"], "2", 1, 0, 0, 3, 9),  # :896-905
    (["0", ".", "1", "0"], "1", 1, 0, 1, 1, 3),  # :908-930 haploid
    (["0:1", ".:1", "1:1", "0:1"], "1", 1, 0, 1, 1, 3),  # :932-950 haploid + FORMAT
]

# ---- float text: main_test.go:1399-1436,2026-2070 + golden pins (SURVEY Appendix B) ----
FLOAT_VECTORS = [
    (1, 3, "0.333"), (1, 4, "0.25"), (2, 5, "0.4"), (1, 6, "0.167"), (3, 10, "0.3"), (3, 6, "0.5"),
    (1, 5008, "0.0002"), (2, 5008, "0.000399"), (939, 5008, "0.188"), (1565, 5008, "0.312"),
    (4695, 5008, "0.938"), (1, 2504, "0.000399"), (1, 1, "1"), (5008, 5008, "1"), (5007, 5008, "1"),
    # E-notation regime: unpinned by the reference (Go's documented 'G' rules == C "%.3G")
    (1, 400000, "2.5E-06"), (1, 10016, "9.98E-05"), (1, 500000, "2E-06"), (1, 10000, "0.0001"),
]


def _vcf(header, records):
    return ("\n".join([VERSION, "\t".join(header)] + ["\t".join(r) for r in records]) + "\n").encode()


E3 = ["!", "0", "!", "0", "!", "0", "0", "0", "0"]  # columns 7-15 with no samples (main_test.go:2553-2572)

# name, config kwargs, vcf bytes, expected rows (list of column lists)
STREAM_CASES = [
    # main_test.go:959-1001 TestHandlesAllMissing
    ("all_missing", {}, _vcf(HDR_S4, [
        ["10", "1000", "rs123", "A", "T", "100", "PASS", "AC=1", "GT", "./.", "./1", "1/.", "./0"],
        ["10", "1000", "rs124", "A", "C", "100", "PASS", "AC=1", "GT", ".|.", "1|.", "1|.", ".|0"]]), []),
    # main_test.go:1003-1105 TestOutputsInfo
    ("info_snp", {"keep_info": True}, _vcf(HDR8, [["10", "1000", "rs#", "C", "T", "100", "PASS", "AC=1"]]),
     [["chr10", "1000", "SNP", "C", "T", "1"] + E3 + ["0", "AC=1"]]),
    ("info_multi", {"keep_info": True}, _vcf(HDR8, [["10", "1000", "rs#", "C", "T,G", "100", "PASS", "AC=1"]]),
     [["chr10", "1000", "MULTIALLELIC", "C", "T", "0"] + E3 + ["0", "AC=1"],
      ["chr10", "1000", "MULTIALLELIC", "C", "G", "0"] + E3 + ["1", "AC=1"]]),
    # main_test.go:1107-1197 TestOutputsId
    ("id_snp", {"keep_id": True}, _vcf(HDR8, [["10", "1000", "rs123", "C", "T", "100", "PASS", "AC=1"]]),
     [["chr10", "1000", "SNP", "C", "T", "1"] + E3 + ["rs123"]]),
    ("id_multi", {"keep_id": True}, _vcf(HDR8, [["10", "1000", "rs456", "C", "T,G", "100", "PASS", "AC=1"]]),
     [["chr10", "1000", "MULTIALLELIC", "C", "T", "0"] + E3 + ["rs456"],
      ["chr10", "1000", "MULTIALLELIC", "C", "G", "0"] + E3 + ["rs456"]]),
    # main_test.go:1199-1274 TestOutputsVcfPos (deletion shifts pos; vcfPos keeps the input)
    ("vcfpos_del", {"keep_pos": True}, _vcf(HDR8, [["10", "1000", "rs#", "CTT", "CT", "100", "PASS", "AC=1"]]),
     [["chr10", "1001", "DEL", "T", "-1", "0"] + E3 + ["1000"]]),
    ("vcfpos_multi", {"keep_pos": True}, _vcf(HDR8, [["10", "1003", "rs#", "C", "T,G", "100", "PASS", "AC=1"]]),
     [["chr10", "1003", "MULTIALLELIC", "C", "T", "0"] + E3 + ["1003"],
      ["chr10", "1003", "MULTIALLELIC", "C", "G", "0"] + E3 + ["1003"]]),
    # main_test.go:1276-1331 TestOutputsVcfPosIdAndInfo
    ("vcfpos_id_info", {"keep_pos": True, "keep_id": True, "keep_info": True},
     _vcf(HDR8, [["10", "1000", "rs123", "C", "T", "100", "PASS", "AC=1"]]),
     [["chr10", "1000", "SNP", "C", "T", "1"] + E3 + ["1000", "rs123", "0", "AC=1"]]),
    # main_test.go:1333-1460 TestOutputsSamplesVcfPosIdAndInfo ('/' separated)
    ("samples_slash", {"keep_pos": True, "keep_id": True, "keep_info": True}, _vcf(HDR_S4, [
        ["10", "1000", "rs123", "A", "T", "100", "PASS", "AC=1", "GT", "0/0", "0/1", "1/1", "./."]]),
     [["chr10", "1000", "SNP", "A", "T", "2", "Sample2", "0.333", "Sample3", "0.333", "Sample4", "0.25",
       "3", "6", "0.5", "1000", "rs123", "0", "AC=1"]]),
    # same family, '|' separated and GT:GQ suffix (main_test.go:1462-2340 sub-cases)
    ("samples_pipe_fmt", {"keep_pos": True, "keep_id": True, "keep_info": True}, _vcf(HDR_S4, [
        ["10", "1000", "rs123", "A", "T", "100", "PASS", "AC=1", "GT:GQ", "0|0:1", "0|1:1", "1|1:1", ".|.:1"]]),
     [["chr10", "1000", "SNP", "A", "T", "2", "Sample2", "0.333", "Sample3", "0.333", "Sample4", "0.25",
       "3", "6", "0.5", "1000", "rs123", "0", "AC=1"]]),
    # main_test.go:2342-2518 TestOutputMultiallelic
    ("multiallelic", {}, _vcf(HDR8 + ["Format", "Sample1", "Sample2", "Sample3", "Sample4"], [
        ["20", "4", ".", "GCACG", "G,GTCACACG", ".", "PASS", "DP=100", "GT", "0|0", "0|1", "2|2", ".|."]]),
     [["chr20", "5", "MULTIALLELIC", "C", "-4", "0", "Sample2", "0.333", "!", "0", "Sample4", "0.25", "1", "6", "0.167"],
      ["chr20", "4", "MULTIALLELIC", "G", "+TCA", "0", "!", "0", "Sample3", "0.333", "Sample4", "0.25", "2", "6", "0.333"]]),
    # main_test.go:2520-2596 TestOutputComplexMultiDel
    ("complex_multi_del", {}, _vcf(HDR8, [
        ["16", "84034434", "rs141446650", "GAGGGAGACAGAGGGAAGT", "G,GGGGAGACAGAGGGAAGT", ".", "PASS", "DP=100"]]),
     [["chr16", "84034435", "MULTIALLELIC", "A", "-18", "0"] + E3,
      ["chr16", "84034435", "MULTIALLELIC", "A", "-1", "0"] + E3]),
    # main_test.go:2598-2671 TestOutputComplexDel
    ("complex_del", {}, _vcf(HDR8, [
        ["1", "874816", "rs200996316", "CCCCCTCATCACCTCCCCAGCCACGGTGAGGACCCACCCTGGCATGATCT",
         "CCCCCTCATCACCTCCCCAGCCACGGTGAGGACCCACCCTGGCATGATCTCCCCTCATCACCTCCCCAGCCACGGTGAGGACCCACCCTGGCATGATCT,"
         "GCCCCTCATCACCTCCCCAGCCACGGTGAGGACCCACCCTGGCATGATCT,C,"
         "CTCCCCTCATCACCTCCCCAGCCACGGTGAGGACCCACCCTGGCATGATCT", ".", "PASS", "DP=100"]]),
     [["chr1", "874816", "MULTIALLELIC", "C", "+CCCCTCATCACCTCCCCAGCCACGGTGAGGACCCACCCTGGCATGATCT", "0"] + E3,
      ["chr1", "874816", "MULTIALLELIC", "C", "G", "0"] + E3,
      ["chr1", "874817", "MULTIALLELIC", "C", "-49", "0"] + E3,
      ["chr1", "874816", "MULTIALLELIC", "C", "+T", "0"] + E3]),
    # main_test.go:2673-2729 TestOutputMultiallelicSnp
    ("multiallelic_snp", {}, _vcf(HDR8, [
        ["1", "1265061", "rs138351882;rs563042459", "CGT", "TGT,C", ".", "PASS", "DP=100"]]),
     [["chr1", "1265061", "MULTIALLELIC", "C", "T", "0"] + E3,
      ["chr1", "1265062", "MULTIALLELIC", "G", "-2", "0"] + E3]),
    # main_test.go:2731-2778 TestComplexSnp
    ("complex_snp", {}, _vcf(HDR8, [
        ["1", "1265062", "rs138351882;rs563042459", "CGT", "CGA", ".", "PASS", "DP=100"]]),
     [["chr1", "1265064", "SNP", "T", "A", "2"] + E3]),
    # main_test.go:2780-2852 TestMNP  (trTv per base is [inferred]: parity unpinned by the reference)
    ("mnp", {}, _vcf(HDR8, [["1", "1000", "rs138351882;rs563042459", "ACGT", "GATC", ".", "PASS", "DP=100"]]),
     [["chr1", "1000", "MNP", "A", "G", "1"] + E3, ["chr1", "1001", "MNP", "C", "A", "2"] + E3,
      ["chr1", "1002", "MNP", "G", "T", "2"] + E3, ["chr1", "1003", "MNP", "T", "C", "1"] + E3]),
    # main_test.go:2854-2909 TestManyAlleles (allele numbers >= 10, haploid sample)
    ("many_alleles", {}, _vcf(
        HDR8 + ["FORMAT", "S1", "S1_2", "S2", "S3", "S4", "S5", "S6", "S7", "S8", "S9", "S10", "S11", "S11_HAPLOID"],
        [["1", "1000", "rs1", "A", "AA,AC,AG,AT,C,G,T,ATA,ATC,ATG,ATT", ".", "PASS", "DP=100", "GT",
          "1|1", "1|1", "2|2", "3|3", "4|4", "5|5", "6|6", "7|7", "8|8", "9|9", "10|10", "11|11", "11"]]),
     [["chr1", "1000", "MULTIALLELIC", "A", alt, "0", "!", "0", homs, hz, "!", "0", ac, "25", maf]
      for alt, homs, hz, ac, maf in [
          ("+A", "S1;S1_2", "0.154", "4", "0.16"), ("+C", "S2", "0.0769", "2", "0.08"),
          ("+G", "S3", "0.0769", "2", "0.08"), ("+T", "S4", "0.0769", "2", "0.08"),
          ("C", "S5", "0.0769", "2", "0.08"), ("G", "S6", "0.0769", "2", "0.08"),
          ("T", "S7", "0.0769", "2", "0.08"), ("+TA", "S8", "0.0769", "2", "0.08"),
          ("+TC", "S9", "0.0769", "2", "0.08"), ("+TG", "S10", "0.0769", "2", "0.08"),
          ("+TT", "S11;S11_HAPLOID", "0.154", "3", "0.12")]]),
    # FILTER handling through the stream (main_test.go:524-569 semantics end to end)
    ("filter_default_drops", {}, _vcf(HDR8, [["1", "5", ".", "A", "C", ".", "q10", "X"]]), []),
    ("filter_allow_all", {"allow": None}, _vcf(HDR8, [["1", "5", ".", "A", "C", ".", "q10", "X"]]),
     [["chr1", "5", "SNP", "A", "C", "2"] + E3]),
    ("filter_exclude", {"allow": None, "exclude": ["q10"]}, _vcf(HDR8, [
        ["1", "5", ".", "A", "C", ".", "q10", "X"], ["chr1", "6", ".", "G", "A", ".", "PASS;q10", "X"]]),
     [["chr1", "6", "SNP", "G", "A", "1"] + E3]),
]

# ---- dosage matrix: main_test.go:2911-2977 TestGenotypeMatrix ----
DOSAGE_CASE = (
    _vcf(HDR8 + ["FORMAT", "S1", "S2", "S3"], [
        ["1", "1000", "rs1", "A", "T", ".", "PASS", "DP=100", "GT", "1|1", "0|1", "0|0"],
        ["2", "200", "rs2", "C", "G", ".", "PASS", "DP=100", "GT", "0|1", "0|0", "1|1"],
        ["22", "300", "rs2", "G", "T", ".", "PASS", "DP=100", "GT", "0|.", "0|.", "1|1"]]),
    [b"chr1:1000:A:T", b"chr2:200:C:G", b"chr22:300:G:T"],
    [[2, 1, 0], [1, 0, 2], [-1, -1, 2]],
)

# ---- header: main_test.go:74-169 TestHeader ----
BASE_HEADER = ["chrom", "pos", "type", "ref", "alt", "trTv", "heterozygotes", "heterozygosity", "homozygotes",
               "homozygosity", "missingGenos", "missingness", "ac", "an", "sampleMaf"]

# chr1 goldens (tests/conftest.py): the 400-line sample and the sample CHR1_REPEATS times over (chr1_fixture)
CHR1_REPEATS = 49
GOLDEN_SAMPLE_LINES, GOLDEN_SAMPLE_ROWS = 400, 410
GOLDEN_MD5_SORTED = "9d2c0824f4f6d584d711e65519b8acae"  # sample, LC_ALL=C sort -k1,1 -k2,2n -k5,5 (reference procedure)
GOLDEN_MD5_INPUT_ORDER = "548d4a7464de83108ca88130c7a5e065"  # chr1_fixture, default flags, body only, 32,496,849 B
GOLDEN_MD5_KEEPID_KEEPINFO = "39f2056b35704d34a6aad24630eb2b2a"  # chr1_fixture, oracle-derived (no reference golden exists)
