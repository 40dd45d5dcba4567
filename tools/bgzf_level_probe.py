#!/usr/bin/env python
"""--bgzfOut at level 1 against level 6 (or any --levels) on one GPU, and against zlib -6 on the same machine's cores.

1. C2 rows (BASELINE configs[1] shape, 2,504 samples) are made on the device: the lines are generated into the resident
   input region and transformed; the rows stay in the resident output region.
2. bvcf_resident_download_bgzf_level is timed on those rows at each level, the levels alternating over --rounds rounds
   (host clock around the call, which ends in a stream synchronise: deflate, pack and the D2H copy of the compressed
   bytes into a pinned buffer allocated once).  Reported: GB/s of rows in, the ratio, and the spread over the rounds.
3. zlib -6 on a sample of the same 48 KiB slices: its ratio, and its rate on all host cores (one process per core, each
   compressing whole slices, wall clock around the lot).
4. The C++ CLI file to file: `--in x.vcf.gz --bgzfOut [--bgzfLevel N] --out /dev/null` on a generated C2-shape .vcf.gz,
   the levels alternating.

    python tools/bgzf_level_probe.py [--variants 600000] [--levels 1,6] [--rounds 3] [--cli-gb 1] [--out x.json]
"""
import argparse
import ctypes as C
import json
import multiprocessing as mp
import os
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bgzf_cli_probe import BIN, make_inputs  # noqa: E402

SLICE = 49152
_SAMPLE = b""


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    rows = [x.strip() for x in r.stdout.strip().split("\n") if x.strip()]
    return rows[0] if rows else "unknown"


def _zlib6(span):
    lo, hi = span
    n = 0
    for o in range(lo, hi, SLICE):
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        n += len(c.compress(_SAMPLE[o:min(o + SLICE, hi)]) + c.flush()) + 26  # + bgzf header and trailer
    return n


def zlib_all_cores(sample):
    """(compressed bytes, seconds) of zlib -6 over the sample's slices on every core"""
    global _SAMPLE
    _SAMPLE = sample
    cores = os.cpu_count() or 1
    per = -(-len(sample) // SLICE // cores) * SLICE
    spans = [(lo, min(lo + per, len(sample))) for lo in range(0, len(sample), per)]
    with mp.get_context("fork").Pool(cores) as pool:
        pool.map(_zlib6, [(0, SLICE)] * cores)  # the workers are up
        t0 = time.perf_counter()
        n = sum(pool.map(_zlib6, spans))
        return n, time.perf_counter() - t0, cores


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--variants", type=int, default=600000)
    ap.add_argument("--levels", default="1,6")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--zlib-mb", type=int, default=256, help="MB of rows (whole slices, spread over the rows) for zlib")
    ap.add_argument("--cli-gb", type=float, default=1.0, help="GB of VCF text for the CLI runs (0: skip them)")
    ap.add_argument("--dir", default="/dev/shm" if os.access("/dev/shm", os.W_OK) else "/tmp")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    from bystro_vcf_b200 import Config, Transformer, _lib, synth

    levels = [int(x) for x in a.levels.split(",") if x]
    res = {"card": card(), "levels": {}, "cli": []}
    print("# card (name, power limit): %s" % res["card"], flush=True)
    seed, ns = 20130502, 2504
    with Transformer(Config()) as tr:
        tr.set_header(synth.chrom_line(seed, ns))
        _, need = synth.device_lines(seed, ns, "chr1", 0, a.variants, 0, 0, 0)
        d_in, _ = tr.resident_alloc(need, need // 6 + (64 << 20))
        synth.device_lines(seed, ns, "chr1", 0, a.variants, d_in, need, 0)
        stats, _ = tr.resident_run(need, want_times=False)
        n = stats["out_bytes"]
        print("# %d variants, %.3f GB of rows" % (a.variants, n / 1e9), flush=True)
        cap, host, zn = n + n // 4 + (1 << 20), C.c_void_p(), C.c_size_t()
        _lib.check(tr._L.bvcf_host_alloc(C.byref(host), cap), None, "bvcf_host_alloc")

        def deflate(lv):
            _lib.check(tr._L.bvcf_resident_download_bgzf_level(tr._ctx, 0, n, lv, host, cap, C.byref(zn)), tr._ctx,
                       "bvcf_resident_download_bgzf_level")
            return zn.value

        for lv in levels:  # warm-up: modules, device buffers
            deflate(lv)
        times = {lv: [] for lv in levels}
        sizes = {}
        for _ in range(a.rounds):
            for lv in levels:
                t0 = time.perf_counter()
                sizes[lv] = deflate(lv)
                times[lv].append(time.perf_counter() - t0)
        tr._L.bvcf_host_free(host)
        # zlib -6 on whole slices spread over the rows
        step = max(1, n // SLICE // max(1, (a.zlib_mb << 20) // SLICE)) * SLICE
        sample = b"".join(tr.resident_download(o, min(SLICE, n - o)) for o in range(0, n, step))
    for lv in levels:
        ts = times[lv]
        gbs = [n / 1e9 / t for t in ts]
        row = {"level": lv, "rows_GB": round(n / 1e9, 3), "ratio": round(n / sizes[lv], 3),
               "GB_per_s_best": round(max(gbs), 2), "GB_per_s_worst": round(min(gbs), 2),
               "spread_pct": round(100 * (max(ts) - min(ts)) / min(ts), 1), "seconds": [round(t, 4) for t in ts]}
        res["levels"][lv] = row
        print(json.dumps(row), flush=True)
    zn, zt, cores = zlib_all_cores(sample)
    res["zlib6"] = {"sample_MB": round(len(sample) / 1e6, 1), "ratio": round(len(sample) / zn, 3), "cores": cores,
                    "all_core_GB_per_s": round(len(sample) / 1e9 / zt, 3)}
    print(json.dumps({"zlib6": res["zlib6"]}), flush=True)
    for lv in levels:
        x = res["levels"][lv]
        print("# level %d: %.2fx, %.2f GB/s = %.1fx all-core zlib -6 (%.2fx, %.3f GB/s on %d cores)"
              % (lv, x["ratio"], x["GB_per_s_best"], x["GB_per_s_best"] / res["zlib6"]["all_core_GB_per_s"],
                 res["zlib6"]["ratio"], res["zlib6"]["all_core_GB_per_s"], cores), flush=True)
    if a.cli_gb > 0:
        plain = gz = None
        try:
            plain, gz, n_var, n_text = make_inputs(a.cli_gb, a.dir)
            for rnd in range(2):
                for lv in levels:
                    cmd = [BIN, "--in", gz, "--bgzfOut", "--out", "/dev/null"] + (["--bgzfLevel", str(lv)] if lv != 1 else [])
                    t0 = time.perf_counter()
                    r = subprocess.run(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, timeout=1800)
                    dt = time.perf_counter() - t0
                    if r.returncode:
                        raise RuntimeError("%s: exit %d: %s" % (cmd, r.returncode, r.stderr.decode()[-1000:]))
                    row = {"cli_level": lv, "round": rnd, "seconds": round(dt, 3), "variants_per_s": round(n_var / dt),
                           "text_GB_per_s": round(n_text / 1e9 / dt, 3)}
                    res["cli"].append(row)
                    print(json.dumps(row), flush=True)
        finally:
            for p in (plain, gz):
                if p and os.path.exists(p):
                    os.remove(p)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
