#!/usr/bin/env python
"""Device-resident step time of the genotype scan and of the whole pipeline on bench.py's c2 (full size), c4 (biobank
width, T2-bound) and c3 (sites-only, HAS_SAMPLES=false) workloads.

Every measurement runs in a child process that generates the workload on the device, warms up, times `--steps`
`Transformer.resident_run` passes with CUDA events and prints one JSON line: mean scan_ms and total_ms per step, plus
an md5 of the rows.  With --old LIB (libbvcf.so of another commit) old and new children alternate, `--rounds` rounds
each, in the same call; the rows of both arms must be identical.  Prints the card name and power limit.

    python tools/scan_probe.py [--old /path/to/old/libbvcf.so] [--configs c2,c4,c3] [--out profiles/x.json]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    rows = [x.strip() for x in r.stdout.strip().split("\n") if x.strip()]
    return rows[0] if rows else "unknown"


def child(lib, config, steps, warmup):
    from bystro_vcf_b200 import _lib
    if lib:
        _lib.LIB_PATH = os.path.abspath(lib)
    import bench
    from bystro_vcf_b200 import Transformer, synth

    spec = bench.CONFIGS[config]
    seed, ns, shape, n = spec["seed"], spec["n_samples"], spec["shape"], spec["lines"]
    tr = Transformer(bench.make_config(spec, 0), eol_width=1)
    tr.set_header(synth.chrom_line(seed, ns))
    _, need = synth.device_lines(seed, ns, shape, 0, n, 0, 0, 0)
    d_in, _ = tr.resident_alloc(need, int(need * (0.55 if ns == 0 else 0.12)) + (64 << 20))
    got, _ = synth.device_lines(seed, ns, shape, 0, n, d_in, need, 0)
    assert got == need, "device generator failed"
    for _ in range(warmup):
        stats, _ = tr.resident_run(need)
    assert stats["n_lines"] == n, stats
    scan = total = 0.0
    for _ in range(steps):
        stats, times = tr.resident_run(need)
        scan += times["scan_ms"]
        total += times["total_ms"]
    md5 = hashlib.md5(tr.resident_download(0, stats["out_bytes"])).hexdigest()
    tr.close()
    print(json.dumps({"scan_ms": scan / steps, "total_ms": total / steps, "n_rows": stats["n_rows"],
                      "out_bytes": stats["out_bytes"], "md5": md5}), flush=True)


def run_child(lib, config, steps, warmup):
    cmd = [sys.executable, os.path.abspath(__file__), "--child", config, "--lib", lib, "--steps", str(steps),
           "--warmup", str(warmup)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1800, cwd=ROOT)
    if r.returncode != 0:
        raise RuntimeError("%s: exit %d\n%s" % (" ".join(cmd), r.returncode, r.stderr[-3000:]))
    return json.loads(r.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="c2,c4,c3")
    ap.add_argument("--old", default="", help="libbvcf.so of another commit, alternated with this tree's build")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="")
    ap.add_argument("--child", default="", help=argparse.SUPPRESS)
    ap.add_argument("--lib", default="", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        child(a.lib, a.child, a.steps, a.warmup)
        return
    name = card()
    print("# card, power limit: %s" % name, flush=True)
    arms = [("new", "")] + ([("old", a.old)] if a.old else [])
    rows, fail = [], False
    for config in [c for c in a.configs.split(",") if c]:
        for rnd in range(a.rounds):
            for tag, lib in arms:
                t0 = time.perf_counter()
                r = run_child(lib, config, a.steps, a.warmup)
                r.update({"config": config, "arm": tag, "round": rnd, "card": name,
                          "child_s": round(time.perf_counter() - t0, 1)})
                rows.append(r)
                print(json.dumps(r), flush=True)
    print("# mean over rounds, ms per step (min..max); %d timed steps per run" % a.steps)
    for config in dict.fromkeys(r["config"] for r in rows):
        line = []
        for tag, _ in arms:
            rs = [r for r in rows if r["config"] == config and r["arm"] == tag]
            for k in ("scan_ms", "total_ms"):
                v = [r[k] for r in rs]
                line.append("%s %s %.3f (%.3f..%.3f)" % (tag, k, sum(v) / len(v), min(v), max(v)))
        if a.old:
            same = len({(r["md5"], r["n_rows"], r["out_bytes"]) for r in rows if r["config"] == config}) == 1
            fail |= not same
            line.append("rows identical: %s" % same)
        print("#   %s: %s" % (config, "; ".join(line)), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump({"card": name, "runs": rows}, f, indent=1)
    sys.exit(1 if fail else 0)


if __name__ == "__main__":
    main()
