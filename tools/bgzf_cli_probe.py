#!/usr/bin/env python
"""File-to-file rate of the C++ host on .vcf.gz input against plain .vcf input, on 1, 2, 4 and 8 GPUs.

A C2-shape VCF (synthetic 1000G chr1 shape, 2,504 samples) is generated on the GPU, copied to the host, written to
/dev/shm as .vcf and as .vcf.gz (bgzf, zlib level 6), and `bystro-vcf-b200 --in X --out /dev/null --gpus N` is timed
around the whole process (context creation included).  With --old BIN (a build of another commit) old and new runs
alternate in the same call.  Prints one JSON line per run and a summary; --out writes them to a file.

    python tools/bgzf_cli_probe.py --gb 2 --gpus 1,2,4,8 [--old /path/to/old/bystro-vcf-b200] [--out profiles/x.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
BIN = os.path.join(ROOT, "bystro_vcf_b200", "bin", "bystro-vcf-b200")


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    rows = [x.strip() for x in r.stdout.strip().split("\n") if x.strip()]
    return rows[0] if rows else "unknown", len(rows)


def make_inputs(gb, d):
    from bystro_vcf_b200 import Config, Transformer, bgzf, synth

    seed, ns = 20130502, 2504
    n = max(1000, int(gb * 1e9 / 10200))
    c = Config()
    with Transformer(c) as tr:
        tr.set_header(synth.chrom_line(seed, ns))
        _, need = synth.device_lines(seed, ns, "chr1", 0, n, 0, 0, 0)
        d_in, _ = tr.resident_alloc(need, 1 << 20)
        synth.device_lines(seed, ns, "chr1", 0, n, d_in, need, 0)
        body = tr.resident_peek(0, need)
    text = synth.header(seed, ns) + body
    plain, gz = os.path.join(d, "bvcf_probe.vcf"), os.path.join(d, "bvcf_probe.vcf.gz")
    with open(plain, "wb") as f:
        f.write(text)
    t0 = time.perf_counter()
    comp = bgzf.compress(text, level=6, threads=os.cpu_count() or 1)
    with open(gz, "wb") as f:
        f.write(comp)
    print("# %d variants, %.2f GB of text, %.3f GB bgzf (%.1fx, compressed in %.1f s)"
          % (n, len(text) / 1e9, len(comp) / 1e9, len(text) / len(comp), time.perf_counter() - t0), flush=True)
    return plain, gz, n, len(text)


def run(binary, path, gpus):
    t0 = time.perf_counter()
    r = subprocess.run([binary, "--in", path, "--out", "/dev/null", "--gpus", str(gpus)], stdout=subprocess.DEVNULL,
                       stderr=subprocess.PIPE, timeout=1800)
    dt = time.perf_counter() - t0
    if r.returncode != 0:
        raise RuntimeError("%s %s --gpus %d: exit %d: %s" % (binary, path, gpus, r.returncode, r.stderr.decode()[-1000:]))
    return dt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=2.0, help="GB of VCF text")
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--old", default="", help="a second binary (another commit's build), alternated with this one")
    ap.add_argument("--dir", default="/dev/shm" if os.access("/dev/shm", os.W_OK) else "/tmp")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    name, n_dev = card()
    print("# card: %s, %d visible" % (name, n_dev), flush=True)
    plain = gz = None
    rows = []
    try:
        plain, gz, n_var, n_text = make_inputs(a.gb, a.dir)
        bins = [("new", BIN)] + ([("old", a.old)] if a.old else [])
        for g in [int(x) for x in a.gpus.split(",") if x]:
            if g > n_dev:
                continue
            for rep in range(a.reps):
                for tag, b in bins:
                    for kind, path in (("vcf.gz", gz), ("vcf", plain)):
                        dt = run(b, path, g)
                        row = {"binary": tag, "input": kind, "gpus": g, "rep": rep, "seconds": round(dt, 3),
                               "variants_per_s": round(n_var / dt), "text_GB_per_s": round(n_text / 1e9 / dt, 3),
                               "card": name}
                        rows.append(row)
                        print(json.dumps(row), flush=True)
    finally:
        for p in (plain, gz):
            if p and os.path.exists(p):
                os.remove(p)
    summary = {}
    for r in rows:
        k = "%s %s %d GPU" % (r["binary"], r["input"], r["gpus"])
        summary[k] = max(summary.get(k, 0), r["variants_per_s"])
    print("# best of %d, M variants/s (context creation included):" % a.reps)
    for k, v in summary.items():
        print("#   %-24s %7.2f" % (k, v / 1e6))
    if a.out:
        with open(a.out, "w") as f:
            json.dump({"card": name, "gb_text": a.gb, "runs": rows, "best_variants_per_s": summary}, f, indent=1)


if __name__ == "__main__":
    main()
