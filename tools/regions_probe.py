#!/usr/bin/env python
"""--regions on one B200: what the region filter stage costs, and what an index saves.

a) bench.py's c2 workload, device-resident: one step (Transformer.resident_run) without regions and with region sets that
   keep all, about half and none of the records, the arms alternated, `--rounds` rounds of `--steps` steps each.  The
   filter runs inside the compact_ms window of bvcf_kernel_times, so compact_ms minus the no-region arm's is the filter's
   device time.  Rows are checked against the unchanged pipeline on the pre-filtered input: the whole input (all), the
   records up to the half region's end (the input is sorted by POS: a prefix of it), nothing (none).
b) the C++ binary file to /dev/null on a generated c2-shape .vcf.gz of `--gb` GB of text, with a .tbi written here:
   --regions spanning about 1 %, 10 % and 100 % of the records, with and without the index beside the file.

Prints the card and power limit.  python tools/regions_probe.py [--steps 5] [--rounds 3] [--gb 3] [--skip-b]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
BIN = os.path.join(ROOT, "bystro_vcf_b200", "bin", "bystro-vcf-b200")
MAX = (1 << 63) - 1


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    rows = [x.strip() for x in r.stdout.strip().split("\n") if x.strip()]
    return rows[0] if rows else "unknown"


def line_at(tr, off, need):
    """(start, CHROM, POS) of the first line that starts at or after byte off"""
    if off:
        b = tr.resident_peek(off - 1, min(1 << 16, need - off + 1))
        off += b.index(b"\n")
    f = tr.resident_peek(off, min(4096, need - off)).split(b"\t", 2)
    return off, f[0], int(f[1])


def probe_a(a):
    import bench
    from bystro_vcf_b200 import Transformer, synth

    spec = bench.CONFIGS["c2"]
    seed, ns, shape, n = spec["seed"], spec["n_samples"], spec["shape"], spec["lines"]
    tr = Transformer(bench.make_config(spec, 0), eol_width=1)
    tr.set_header(synth.chrom_line(seed, ns))
    _, need = synth.device_lines(seed, ns, shape, 0, n, 0, 0, 0)
    d_in, _ = tr.resident_alloc(need, int(need * 0.12) + (64 << 20))
    assert synth.device_lines(seed, ns, shape, 0, n, d_in, need, 0)[0] == need
    _, chrom, first = line_at(tr, 0, need)
    _, _, last = line_at(tr, need - 20000, need)
    mid = (first + last) // 2
    lo, hi = 0, need  # the first line whose POS is past mid: the half arm's input is the lines before it
    while hi - lo > 1 << 16:
        m = (lo + hi) // 2
        if line_at(tr, m, need)[2] <= mid:
            lo = m
        else:
            hi = m
    cut = lo
    while cut < need and line_at(tr, cut, need)[2] <= mid:
        cut = line_at(tr, cut + 1, need)[0]
    arms = {"off": None, "all": [(chrom, 1, MAX)], "half": [(chrom, 1, mid)], "none": [(chrom, last + 1, MAX)]}

    def run(regions, length):
        tr.set_regions(regions)
        stats, times = tr.resident_run(length)
        return stats, times

    md5 = {}
    for name, length in (("off", need), ("half-ref", cut)):
        stats, _ = run(None, length)
        md5[name] = (hashlib.md5(tr.resident_download(0, stats["out_bytes"])).hexdigest(), stats["n_rows"])
    res = {k: [] for k in arms}
    for rnd in range(a.rounds):
        for name, regions in arms.items():
            for _ in range(a.warmup):
                run(regions, need)
            c = t = 0.0
            for _ in range(a.steps):
                stats, times = run(regions, need)
                c += times["compact_ms"]
                t += times["total_ms"]
            got = (hashlib.md5(tr.resident_download(0, stats["out_bytes"])).hexdigest(), stats["n_rows"])
            exp = {"off": md5["off"], "all": md5["off"], "half": md5["half-ref"], "none": (hashlib.md5(b"").hexdigest(), 0)}[name]
            assert got == exp, (name, got, exp)
            res[name].append({"compact_ms": c / a.steps, "total_ms": t / a.steps, "n_rows": stats["n_rows"]})
            print(json.dumps({"probe": "a", "arm": name, "round": rnd, **res[name][-1]}), flush=True)
    tr.close()
    base = sum(r["compact_ms"] for r in res["off"]) / a.rounds
    for name, rs in res.items():
        c = [r["compact_ms"] - base for r in rs]
        t = [r["total_ms"] for r in rs]
        print("# a) c2 step, %s: filter %.3f ms (%.3f..%.3f) over the no-region compaction, step %.2f ms (%.2f..%.2f), "
              "%d rows; rows equal the pre-filtered run" % (name, sum(c) / len(c), min(c), max(c), sum(t) / len(t),
                                                           min(t), max(t), rs[-1]["n_rows"]), flush=True)


def probe_b(a):
    from bystro_vcf_b200 import bgzf, synth
    from test_regions_cpu import index_of

    seed, ns = 20130502, 2504
    per = len(synth.host_lines(seed, ns, "chr1", 0, 1000)) / 1000
    n = int(a.gb * 1e9 / per)
    d = tempfile.mkdtemp(dir=a.tmp)
    text = synth.header(seed, ns) + synth.host_lines(seed, ns, "chr1", 0, n)
    gz = os.path.join(d, "c2.vcf.gz")
    with open(gz, "wb") as f:
        f.write(bgzf.compress(text, level=1, block_text=bgzf.MAX_TEXT))
    tbi = bgzf.compress(index_of(text, bgzf.MAX_TEXT, level=1))
    t0 = text.index(b"\n", text.index(b"\n#CHROM") + 1) + 1
    chrom, first = text[t0:t0 + 100].split(b"\t")[:2]
    last = int(text[text.rindex(b"\n", 0, len(text) - 1) + 1:].split(b"\t")[1])
    first = int(first)
    del text
    print("# b) %s: %.2f GB of text, %d records, %.2f GB compressed" % (gz, n * per / 1e9, n, os.path.getsize(gz) / 1e9))
    rows = []
    for frac in (0.01, 0.10, 1.0):
        reg = "%s:%d-%d" % (chrom.decode(), first, first + int((last - first) * frac))
        for indexed in (True, False):
            if indexed:
                open(gz + ".tbi", "wb").write(tbi)
            elif os.path.exists(gz + ".tbi"):
                os.remove(gz + ".tbi")
            t = time.perf_counter()
            r = subprocess.run([BIN, "--in", gz, "--out", "/dev/null", "--regions", reg], capture_output=True)
            dt = time.perf_counter() - t
            assert r.returncode == 0, r.stderr[-2000:]
            rows.append({"probe": "b", "region_frac": frac, "index": indexed, "wall_s": round(dt, 3)})
            print(json.dumps(rows[-1]), flush=True)
    t = time.perf_counter()
    subprocess.run([BIN, "--in", gz, "--out", "/dev/null"], check=True, capture_output=True)
    print("# b) no --regions: %.3f s" % (time.perf_counter() - t), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--gb", type=float, default=3.0)
    ap.add_argument("--tmp", default=None)
    ap.add_argument("--skip-a", action="store_true")
    ap.add_argument("--skip-b", action="store_true")
    a = ap.parse_args()
    print("# card, power limit: %s" % card(), flush=True)
    if not a.skip_a:
        probe_a(a)
    if not a.skip_b:
        probe_b(a)


if __name__ == "__main__":
    main()
