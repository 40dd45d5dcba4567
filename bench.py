#!/usr/bin/env python
"""bench.py -- the per-line VCF transform on the BASELINE.json workload (configs[1]: synthetic 1000G Phase 3
chr1-shape VCF, 6.2M variants x 2,504 phased diploid samples).

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA, libbvcf)
  python bench.py --impl reference --gpus N ...            the reference's CPU implementation of the path
                                                           (oracle port: Go cannot be built in this image)

A step = one pass of the whole pipeline over one rank's shard, input resident in HBM (`value`), and the
same metric through the C ABI with host buffers, H2D + D2H inside the timed region (`e2e`).
Multi-GPU: one process per GPU (torchrun), shards are independent line ranges, no data-path collective.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "variants/s"

# BASELINE.json configs (SURVEY.md 8d).  `lines` = variants per GPU at the default size; c2 is the headline
# (configs[1]), the others are the driver-visible lines VERDICT r1 asked for (`--config c3|c4|c5`).
CONFIGS = {
    "c2": dict(name="configs[1]: synthetic 1000G Phase 3 chr1-shape VCF", shape="chr1", n_samples=2504, seed=20130502,
               lines=6_200_000, flags="default PASS/. filter", cfg={}),
    "c3": dict(name="configs[2]: sites-only synthetic VCF (0 samples), 30% multiallelic/MNP + padded indels", shape="sites",
               n_samples=0, seed=50, lines=50_000_000, flags="default PASS/. filter", cfg={}),
    "c4": dict(name="configs[3]: biobank-width synthetic VCF, 200,000 samples with 2% missing GT (a slice of the 1M-variant "
                    "file per GPU: the whole file is 800 GB)", shape="biobank", n_samples=200_000, seed=200000, lines=32_000,
               flags="default PASS/. filter", cfg={}),
    "c5": dict(name="configs[4]: chr1-shape VCF with --keepInfo, --allowFilter '*' --excludeFilter LowQual and the dosage "
                    "matrix (arrow/ schema)", shape="chr1_filters", n_samples=2504, seed=20130502, lines=6_200_000,
               flags="--keepInfo --allowFilter * --excludeFilter LowQual --dosageOutput", cfg=dict(keepInfo=True, allow=None,
                                                                                                  exclude=["LowQual"], dosage=True)),
}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe):
    one long-running `nvidia-smi -lms 100` started before the region and stopped after it."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self._p = None

    def __enter__(self):
        try:
            self._p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                        "--format=csv,noheader,nounits", "-lms", "100"],
                                       stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.25)  # let the first sample land before the timed region starts
        except Exception:
            self._p = None
        return self

    def __exit__(self, *a):
        if self._p is None:
            return
        time.sleep(0.12)
        self._p.terminate()
        try:
            out, _ = self._p.communicate(timeout=5)
        except Exception:
            self._p.kill()
            out = ""
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 6:
                self.rows.append(f)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i].lower() == "active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def scan_traffic_ratio():
    """DRAM bytes (read+write) per algorithmic byte of the scan kernel, from the committed ncu --set full
    capture (profiles/r02_scan_traffic.json); None when no capture is committed."""
    p = os.path.join(ROOT, "profiles", "r02_scan_traffic.json")
    try:
        with open(p) as f:
            d = json.load(f)
        return (d["dram_bytes_read"] + d["dram_bytes_write"]) / d["algorithmic_bytes"], d.get("source", p)
    except Exception:
        return None, None


def newline_cuts(view, total: int, chunk: int):
    """Newline-aligned chunk boundaries of a host buffer (numpy uint8 view)."""
    import numpy as np

    cuts = [0]
    while cuts[-1] < total:
        end = min(cuts[-1] + chunk, total)
        if end < total:
            lo = max(cuts[-1], end - (4 << 20))
            nl = np.flatnonzero(view[lo:end] == 10)
            end = lo + int(nl[-1]) + 1
        cuts.append(end)
    return cuts


def make_config(spec, dev):
    from bystro_vcf_b200 import Config

    cfg = Config()
    cfg.allowedFilters = {"PASS": True, ".": True}
    c = spec["cfg"]
    if "allow" in c:
        cfg.allowedFilters = None if c["allow"] is None else {x: True for x in c["allow"]}
    if c.get("exclude"):
        cfg.excludedFilters = {x: True for x in c["exclude"]}
    cfg.keepInfo = bool(c.get("keepInfo"))
    if c.get("dosage"):
        cfg.dosageMatrixOutPath = "resident"  # any non-empty path: the library produces the dosage rows + loci
    cfg.device = dev
    return cfg


def oracle_config(spec):
    from oracle import oracle as O

    c = spec["cfg"]
    return O.OracleConfig(keep_info=bool(c.get("keepInfo")), allow=c["allow"] if "allow" in c else ("PASS", "."),
                          exclude=c.get("exclude"), want_dosage=bool(c.get("dosage")))


DUMP_SEED = 20130502
DUMP_ROW_WINDOWS, DUMP_WINDOW_BYTES = 128, 64 << 10  # 8 MiB of row text -> 32 MiB as float32
DUMP_DOSAGE_BYTES = 20 << 20  # whole dosage rows as float32 (2,093 rows of 2,504 samples)
DUMP_DIAGS = 1 << 16  # x 4 float64


def dump_outputs(tr, stats, out_dir):
    """What the last timed resident run returned to its caller, as .npy files in out_dir (under 60 MB in all): the
    run's counts, the TSV rows, the dosage matrix and loci of dosage configs, the diagnostics.  Outputs larger than
    that are sampled at positions drawn from DUMP_SEED, the same for every run of the same arguments."""
    import random

    import numpy as np

    from bystro_vcf_b200 import _lib

    os.makedirs(out_dir, exist_ok=True)
    rng = random.Random(DUMP_SEED)

    def save(name, a, dtype):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=dtype))

    keys = ("n_lines", "n_records", "n_rows", "in_bytes", "out_bytes")
    save("stats", [stats[k] for k in keys], np.float64)
    n = stats["out_bytes"]
    if n <= DUMP_ROW_WINDOWS * DUMP_WINDOW_BYTES:
        offsets, width = [0], n
    else:  # one window in each of DUMP_ROW_WINDOWS equal strata of the output
        stratum = n // DUMP_ROW_WINDOWS
        offsets = [i * stratum + rng.randrange(stratum - DUMP_WINDOW_BYTES + 1) for i in range(DUMP_ROW_WINDOWS)]
        width = DUMP_WINDOW_BYTES
    rows = [np.frombuffer(tr.resident_download(o, width), dtype=np.uint8) for o in offsets]
    save("rows", np.stack(rows), np.float32)  # [windows, bytes]: byte values of the row text
    save("rows_offsets", offsets, np.float64)

    dos = _lib.CDosageBatch()
    dg = C.POINTER(_lib.CDiag)()
    nd = C.c_size_t()
    _lib.check(_lib.lib().bvcf_resident_results(tr._ctx, C.byref(dos), C.byref(dg), C.byref(nd)), tr._ctx,
               "bvcf_resident_results")
    if dos.n_rows:
        nr, ns = dos.n_rows, dos.n_samples
        pick = sorted(rng.sample(range(nr), min(nr, max(1, DUMP_DOSAGE_BYTES // (4 * ns)))))
        mat = np.ctypeslib.as_array(dos.dosage, shape=(nr, ns))
        save("dosage", mat[pick], np.float32)  # [sampled rows, samples]
        save("dosage_rows", pick, np.float64)
        offs = np.ctypeslib.as_array(dos.loci_off, shape=(nr + 1,))
        base = C.cast(dos.loci, C.c_void_p).value
        loci = b"\n".join(C.string_at(base + int(offs[i]), int(offs[i + 1] - offs[i])) for i in pick) + b"\n"
        save("loci", np.frombuffer(loci, dtype=np.uint8), np.float32)  # the sampled rows' loci, newline-separated
    picked = sorted(rng.sample(range(nd.value), min(nd.value, DUMP_DIAGS)))
    diags = [(dg[i].line_no, dg[i].alt_no, dg[i].code, dg[i].line_start) for i in picked]
    save("diagnostics", np.asarray(diags, dtype=np.float64).reshape(-1, 4), np.float64)  # line, alt, code, line start


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from bystro_vcf_b200 import Transformer, synth
    from bystro_vcf_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = local
    spec = CONFIGS[args.config]
    n_lines = args.lines or spec["lines"]
    n_samples, seed, shape = spec["n_samples"], spec["seed"], spec["shape"]
    first_line = rank * n_lines  # rank r owns lines [r*n, (r+1)*n): newline-aligned shards of one N*n-line file

    cfg = make_config(spec, dev)
    dosage = bool(spec["cfg"].get("dosage"))
    tr = Transformer(cfg, eol_width=1, n_slots=3, max_chunk_bytes=(args.chunk_mb << 20) + (64 << 20))
    chrom = synth.chrom_line(seed, n_samples)
    tr.set_header(chrom)
    L = _lib.lib()

    # ---- workload: generated on the device, straight into the resident input region ----
    _, need = synth.device_lines(seed, n_samples, shape, first_line, n_lines, 0, 0, dev)
    out_cap = int(need * (0.55 if n_samples == 0 else 0.12)) + (64 << 20)
    d_in, d_out = tr.resident_alloc(need, out_cap)
    got, _ = synth.device_lines(seed, n_samples, shape, first_line, n_lines, d_in, need, dev)
    assert got == need, "device generator failed"

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    stage_keys = ("scan_ms", "compact_ms", "stats_ms", "rows_ms", "names_ms", "total_ms", "compose_ms", "copyout_ms")

    def resident_steps(length, expect_lines):
        """warm-up, then `steps` timed passes of the whole pipeline over the resident input"""
        for _ in range(args.warmup):
            stats, times = tr.resident_run(length)
        assert stats["n_lines"] == expect_lines, stats
        launches0 = tr.launches
        acc = {k: 0.0 for k in stage_keys}
        barrier()
        with ClockSampler(dev) as clk:
            t0 = time.perf_counter()
            for _ in range(args.steps):
                stats, times = tr.resident_run(length)
                for k in acc:
                    acc[k] += times[k]
            barrier()
            wall_ms = (time.perf_counter() - t0) * 1e3
        return stats, acc, wall_ms, tr.launches - launches0, clk

    # ---- device-resident steps (weak: every GPU its own n_lines) ----
    stats, acc, wall_ms, gpu_launches, clk = resident_steps(need, n_lines)
    dev_ms = acc["total_ms"]  # CUDA events on the launching stream, first to last launch of every step
    out_bytes, n_rows = stats["out_bytes"], stats["n_rows"]
    if args.dump_outputs and rank == 0:  # before anything else runs on the resident regions
        dump_outputs(tr, stats, args.dump_outputs)

    # ---- parity of what was just timed: the rows of the first lines against the CPU oracle (outside the timed region) ----
    parity = None
    if rank == 0:
        import hashlib

        from oracle import oracle as O

        bpl = need / n_lines
        probe = int(min(need, 64 << 20, max(args.parity_lines * bpl, 4 * bpl + 4096, 1 << 20)))
        head = tr.resident_peek(0, probe)
        head = head[:head.rfind(b"\n") + 1]
        ref = O.process_block(oracle_config(spec), chrom, head, threads=os.cpu_count() or 1)
        got_rows = tr.resident_download(0, len(ref.tsv)) if ref.tsv else b""
        ok = got_rows == ref.tsv and len(ref.tsv) <= out_bytes
        parity = {"checked": bool(ok), "lines": ref.n_lines, "rows": ref.n_rows, "bytes": len(ref.tsv),
                  "md5": hashlib.md5(got_rows).hexdigest(),
                  "how": "rows of the first %d lines of the timed device-resident output == oracle rows for the same lines"
                         % ref.n_lines}
        assert ok, "device-resident rows differ from the oracle"

    # ---- end to end through the C ABI: pinned host buffers, H2D + kernels + D2H per chunk ----
    def host_slice(n_want):
        """the first n_want lines of the resident input, copied once to pinned host memory; newline-aligned cuts"""
        bpl = need / n_lines
        probe = int(min(tr_len, n_want * bpl * 1.02 + (1 << 20)))
        hp = C.c_void_p()
        _lib.check(L.bvcf_host_alloc(C.byref(hp), probe), None, "bvcf_host_alloc")
        tr.resident_peek(0, probe, hp.value)
        hv = np.ctypeslib.as_array(C.cast(hp, C.POINTER(C.c_uint8)), shape=(probe,))
        nl = np.flatnonzero(hv[max(0, probe - (8 << 20)):probe] == 10)
        nbytes = max(0, probe - (8 << 20)) + int(nl[-1]) + 1
        return hp, hv, nbytes, newline_cuts(hv, nbytes, args.chunk_mb << 20)

    def e2e_steps(hp, cuts):
        dos = _lib.CDosageBatch()
        tsv, n = C.c_void_p(), C.c_size_t()
        st = _lib.CChunkStats()
        nl_tot = out_tot = dos_tot = 0
        first = None
        for it in range(args.warmup + args.steps):
            if it == args.warmup:
                barrier()
                t0 = time.perf_counter()
                nl_tot = out_tot = dos_tot = 0
            nchunks = len(cuts) - 1
            sub = col = 0
            while col < nchunks:
                while sub < nchunks and sub - col < tr.n_slots:
                    _lib.check(L.bvcf_submit(tr._ctx, sub, hp.value + cuts[sub], cuts[sub + 1] - cuts[sub]), tr._ctx, "submit")
                    sub += 1
                _lib.check(L.bvcf_collect(tr._ctx, col, C.byref(tsv), C.byref(n), C.byref(dos) if dosage else None, None, None,
                                          C.byref(st)), tr._ctx, "collect")
                if first is None:  # the rows of the first chunk, for the parity check below
                    first = C.string_at(tsv, min(n.value, 4 << 20))
                nl_tot += st.n_lines
                out_tot += n.value
                if dosage:
                    dos_tot += dos.n_rows * dos.n_samples + (dos.loci_off[dos.n_rows] if dos.n_rows else 0) + 8 * dos.n_rows
                _lib.check(L.bvcf_release(tr._ctx, col), tr._ctx, "release")
                col += 1
        barrier()
        ms = (time.perf_counter() - t0) * 1e3
        return ms, nl_tot // args.steps, out_tot // args.steps, dos_tot // args.steps, first

    tr_len = need
    e2e_lines = max(1, min(n_lines, int(args.e2e_lines * 10400 / (need / n_lines))))  # a byte budget: --e2e-lines chr1-shape lines
    host_ptr, hview, e2e_bytes, cuts = host_slice(e2e_lines)
    # PCIe H2D bound, measured in the same run: pinned -> device copies of the slice
    tr.resident_upload(0, (host_ptr.value, min(e2e_bytes, 1 << 30)))  # warm
    tp0 = time.perf_counter()
    n_up = 3
    for _ in range(n_up):
        tr.resident_upload(0, (host_ptr.value, e2e_bytes))
    pcie_gbs = n_up * e2e_bytes / (time.perf_counter() - tp0) / 1e9
    # the same with every rank copying at once: what the host side (DRAM, root complexes) can feed N GPUs together
    barrier()
    tp0 = time.perf_counter()
    for _ in range(n_up):
        tr.resident_upload(0, (host_ptr.value, e2e_bytes))
    barrier()
    h2d_concurrent_gbs = n_up * e2e_bytes / (time.perf_counter() - tp0) / 1e9  # this rank's share; summed below
    e2e_ms, e2e_lines_per_step, e2e_out_per_step, e2e_dos_per_step, e2e_first = e2e_steps(host_ptr, cuts)
    if rank == 0 and parity is not None:  # the e2e path returns the same rows
        k = min(len(e2e_first), parity["bytes"])
        parity["e2e_checked"] = bool(k == 0 or e2e_first[:k] == got_rows[:k])
        assert parity["e2e_checked"], "end-to-end rows differ from the device-resident rows"

    # ---- the same end-to-end step with bgzf-COMPRESSED host buffers (SURVEY 8f-3): only the compressed bytes cross
    # PCIe, the GPU inflates them into the resident region, runs the transform there, rows come back.  Beside `e2e`,
    # not instead of it: the north star's e2e is uncompressed input. ----
    e2e_bgzf = None
    if not args.no_bgzf and n_samples > 0:
        from bystro_vcf_b200 import bgzf

        bz_bytes = int(min(e2e_bytes, args.bgzf_mb << 20))
        nlb = np.flatnonzero(hview[max(0, bz_bytes - (8 << 20)):bz_bytes] == 10)
        bz_bytes = max(0, bz_bytes - (8 << 20)) + int(nlb[-1]) + 1
        text = hview[:bz_bytes].tobytes()
        t0 = time.perf_counter()
        comp = bgzf.compress(text, level=6, threads=max(1, (os.cpu_count() or 1) // world))
        t_comp = time.perf_counter() - t0
        cp = C.c_void_p()
        _lib.check(L.bvcf_host_alloc(C.byref(cp), len(comp)), None, "bvcf_host_alloc")
        C.memmove(cp.value, comp, len(comp))
        out_host = C.c_void_p()
        _lib.check(L.bvcf_host_alloc(C.byref(out_host), int(bz_bytes * 0.2) + (16 << 20)), None, "bvcf_host_alloc")
        inf_ms = 0.0
        for it in range(args.warmup + args.steps):
            if it == args.warmup:
                barrier()
                tb0 = time.perf_counter()
            t0 = time.perf_counter()
            got_n = tr.resident_inflate_bgzf((cp.value, len(comp)))
            t1 = time.perf_counter()
            st_b, _ = tr.resident_run(got_n, want_times=False)
            _lib.check(L.bvcf_resident_download(tr._ctx, 0, out_host, st_b["out_bytes"]), tr._ctx, "download")
            if it >= args.warmup:
                inf_ms += (t1 - t0) * 1e3
        barrier()
        bz_ms = (time.perf_counter() - tb0) * 1e3
        assert got_n == bz_bytes
        rows_b = C.string_at(out_host, min(st_b["out_bytes"], parity["bytes"])) if parity else b""
        ok_b = (not parity) or rows_b == got_rows[:len(rows_b)]
        bz_lines_all = st_b["n_lines"]
        if world > 1:
            tt = torch.tensor([bz_ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            bz_ms = float(tt.item())
            tv = torch.tensor([float(st_b["n_lines"])], dtype=torch.float64, device="cuda")
            dist.all_reduce(tv, op=dist.ReduceOp.SUM)
            bz_lines_all = float(tv.item())
        # ... and with the rows deflated on the GPU as well (SURVEY 8f-4): compressed in, compressed out
        out_cap_b = int(bz_bytes * 0.2) + (16 << 20)
        zn = C.c_size_t()
        def_ms = 0.0
        for it in range(args.warmup + args.steps):
            if it == args.warmup:
                barrier()
                tz0 = time.perf_counter()
            got_n = tr.resident_inflate_bgzf((cp.value, len(comp)))
            st_z, _ = tr.resident_run(got_n, want_times=False)
            t0 = time.perf_counter()
            _lib.check(L.bvcf_resident_download_bgzf(tr._ctx, 0, st_z["out_bytes"], out_host, out_cap_b, C.byref(zn)), tr._ctx, "download_bgzf")
            if it >= args.warmup:
                def_ms += (time.perf_counter() - t0) * 1e3
        barrier()
        zz_ms = (time.perf_counter() - tz0) * 1e3
        if world > 1:
            tt = torch.tensor([zz_ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            zz_ms = float(tt.item())
        import gzip as _gz
        ok_z = (not parity) or _gz.decompress(C.string_at(out_host, zn.value) + bgzf.EOF_BLOCK)[:len(rows_b)] == rows_b
        assert ok_z, "rows deflated on the GPU do not inflate back to the rows"
        e2e_bgzf = {"value": bz_lines_all * args.steps / (bz_ms / 1e3), "unit": "variants/s", "n_gpus": world,
                    "compressed_rows_too": {"value": bz_lines_all * args.steps / (zz_ms / 1e3), "unit": "variants/s",
                                            "d2h_bytes_per_step": zn.value, "rows_bytes_per_step": st_z["out_bytes"],
                                            "rows_compression_ratio": st_z["out_bytes"] / max(zn.value, 1),
                                            "deflate_gb_per_s": st_z["out_bytes"] * args.steps / (def_ms / 1e3) / 1e9,
                                            "parity_checked": bool(ok_z),
                                            "what": "rows deflated on the GPU (bgzf blocks) before the D2H copy; the rate includes that copy"},
                    "h2d_bytes_per_step": len(comp), "d2h_bytes_per_step": st_b["out_bytes"], "text_bytes_per_step": bz_bytes,
                    "variants_per_step": st_b["n_lines"], "compression_ratio": bz_bytes / len(comp),
                    "inflate_gb_per_s": bz_bytes * args.steps / (inf_ms / 1e3) / 1e9,
                    "text_gb_per_s": world * bz_bytes * args.steps / (bz_ms / 1e3) / 1e9, "parity_checked": bool(ok_b),
                    "sample": "first %d variants of each rank's shard, bgzf level 6 (%d blocks), pinned host memory; H2D of the compressed bytes + "
                              "GPU inflate + transform + D2H of the rows, one group, no overlap between the stages"
                              % (st_b["n_lines"], -(-bz_bytes // bgzf.MAX_TEXT)),
                    "host_compress_s": t_comp}
        assert ok_b, "rows from bgzf input differ"
        L.bvcf_host_free(cp)
        L.bvcf_host_free(out_host)
        # the resident region was overwritten: put the workload back for the strong-scaling arm / later use
        synth.device_lines(seed, n_samples, shape, first_line, n_lines, d_in, need, dev)

    # ---- CPU baseline sample (N=1 only), taken while the weak slice is still in host memory ----
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as O

        bpl = need / n_lines
        cb_lines = max(1, min(e2e_lines_per_step, int(args.cpu_lines * 10400 / bpl)))
        idx = np.flatnonzero(hview[:min(e2e_bytes, int(cb_lines * bpl * 1.02) + 4096)] == 10)
        cb_lines = min(cb_lines, len(idx))
        cb_bytes = int(idx[cb_lines - 1]) + 1
        threads = os.cpu_count() or 1
        t0 = time.perf_counter()
        r = O.process_block(oracle_config(spec), chrom, host_ptr.value, cb_bytes, 1, threads)
        dt = time.perf_counter() - t0
        cpu_baseline = {"value": r.n_lines / dt, "unit": "variants/s", "cores": threads, "kind": "port",
                        "sample": "first %d variants of the workload, in RAM, output to memory; %.2f s" % (r.n_lines, dt),
                        "note": "C restatement of main.go (oracle/), not the Go binary: no Go toolchain in this image"}
    L.bvcf_host_free(host_ptr)

    # ---- strong scaling: ONE n_lines-variant file partitioned over the N GPUs by newline-aligned line ranges ----
    strong = None
    if world > 1:
        s_lines = n_lines // world
        s_first = rank * s_lines
        got, s_need = synth.device_lines(seed, n_samples, shape, s_first, s_lines, d_in, need, dev)
        assert got == s_need <= need
        s_stats, s_acc, _, _, _ = resident_steps(s_need, s_lines)
        tr_len = s_need
        s_hp, s_hv, s_bytes, s_cuts = host_slice(max(1, e2e_lines // world))
        s_e2e_ms, s_e2e_lines, s_e2e_out, _, _ = e2e_steps(s_hp, s_cuts)
        L.bvcf_host_free(s_hp)
        t = torch.tensor([s_acc["total_ms"], s_e2e_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        v = torch.tensor([float(s_e2e_lines), float(s_bytes), float(s_stats["out_bytes"])], dtype=torch.float64, device="cuda")
        dist.all_reduce(v, op=dist.ReduceOp.SUM)
        s_dev_ms, s_e2e_ms = (float(x) for x in t.tolist())
        tot_e2e_lines, tot_e2e_bytes, tot_out = (float(x) for x in v.tolist())
        strong = {"scaling": "strong", "total_variants": s_lines * world, "variants_per_gpu": s_lines,
                  "value": s_lines * world * args.steps / (s_dev_ms / 1e3), "unit": "variants/s",
                  "ms_per_step": s_dev_ms / args.steps,
                  "e2e": {"value": tot_e2e_lines * args.steps / (s_e2e_ms / 1e3), "unit": "variants/s",
                          "total_variants_per_step": int(tot_e2e_lines), "h2d_bytes_per_step": int(tot_e2e_bytes),
                          "input_gb_per_s": tot_e2e_bytes * args.steps / (s_e2e_ms / 1e3) / 1e9,
                          "sample": "one %d-variant slice of the file, 1/%d per GPU (newline-aligned), pinned host memory"
                                    % (int(tot_e2e_lines), world)},
                  "note": "the same total work as the 1-GPU run split over %d GPUs; no collective (shards never interact)" % world}

    # ---- max over ranks ----
    h2d_all = h2d_concurrent_gbs
    if world > 1:
        t = torch.tensor([dev_ms, wall_ms, e2e_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, wall_ms, e2e_ms = (float(x) for x in t.tolist())
        t = torch.tensor([h2d_concurrent_gbs], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        h2d_all = float(t.item())

    result = None
    if rank == 0:
        peak, peak_src = measured_peaks()
        value = world * n_lines * args.steps / (dev_ms / 1e3)
        in_gbs = world * need * args.steps / (dev_ms / 1e3) / 1e9
        scan_ms = acc["scan_ms"] / args.steps
        dos_bytes = (n_rows * (n_samples + 4)) if dosage else 0  # + locus strings (a few bytes per row more)
        alg_bytes = need + out_bytes + dos_bytes
        # dominant kernel = the fused index+genotype scan: it must read every input byte once
        roof = {"bound": "hbm", "kernel": "bvcf_scan_genotype_kernel", "achieved": need / (scan_ms / 1e3) / 1e9,
                "peak": peak, "peak_source": peak_src, "unit": "GB/s", "traffic": None,
                "algorithmic_bytes_per_step": need, "avg_ms_per_step": scan_ms}
        roof["frac"] = roof["achieved"] / peak
        # the kernel is launched once per 16 GiB sub-chunk of the resident input: per-launch figures beside the per-step ones
        n_launch = max(1, -(-need // (16 << 30)))
        roof["launches_per_step"] = n_launch
        roof["algorithmic_bytes_per_launch"] = need / n_launch
        roof["avg_ms_per_launch"] = scan_ms / n_launch
        ratio, src = scan_traffic_ratio()
        if ratio is not None and args.config == "c2":  # DRAM read+write bytes per launch, scaled from the committed ncu --set full capture
            roof["traffic"] = ratio * need / n_launch
            roof["traffic_per_step"] = ratio * need
            roof["traffic_source"] = src
        pipe = {"achieved": alg_bytes / (dev_ms / args.steps / 1e3) / 1e9, "unit": "GB/s",
                "algorithmic_bytes_per_step": alg_bytes, "bytes_per_variant": alg_bytes / n_lines}
        pipe["frac"] = pipe["achieved"] / peak
        e2e_val = world * e2e_lines_per_step * args.steps / (e2e_ms / 1e3)
        result = {
            "metric": METRIC, "value": value, "unit": "variants/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "%s, %d variants x %d samples per GPU (seed %d), %s"
                                   % (spec["name"], n_lines, n_samples, seed, spec["flags"]),
                       "variants_per_gpu": n_lines, "samples": n_samples, "input_bytes_per_gpu": need,
                       "output_bytes_per_gpu": out_bytes, "rows_per_gpu": n_rows,
                       "l2": "input (%.1f GB) >> 126 MB L2, no flush needed" % (need / 1e9),
                       "parallelism": "%d independent newline-aligned shards, no collective" % world},
            "input_gb_per_s": in_gbs,
            "wall_ms_per_step": wall_ms / args.steps,
            "kernel_ms_per_step": {k: v / args.steps for k, v in acc.items()},
            "roofline": roof, "roofline_pipeline": pipe,
            "e2e": {"value": e2e_val, "unit": "variants/s", "h2d_bytes_per_step": e2e_bytes,
                    "d2h_bytes_per_step": e2e_out_per_step + e2e_dos_per_step, "variants_per_step": e2e_lines_per_step,
                    "input_gb_per_s": world * e2e_bytes * args.steps / (e2e_ms / 1e3) / 1e9,
                    "pcie_h2d_gbs_measured": pcie_gbs,
                    "h2d_gbs_all_ranks_at_once": h2d_all,
                    "frac_of_concurrent_h2d_bound": (world * e2e_bytes * args.steps / (e2e_ms / 1e3) / 1e9) / h2d_all,
                    "host": {"cpus": len(os.sched_getaffinity(0)), "numa_nodes": len([d for d in os.listdir("/sys/devices/system/node")
                                                                                       if d.startswith("node")])
                             if os.path.isdir("/sys/devices/system/node") else None},
                    "frac_of_pcie_h2d_bound": (e2e_bytes * args.steps / (e2e_ms / 1e3) / 1e9) / pcie_gbs,
                    "sample": "first %d variants of each rank's shard, pinned host memory, %d MiB chunks, 3 slots"
                              % (e2e_lines_per_step, args.chunk_mb)},
            "gpu_launches": int(gpu_launches),
            "parity_checked": bool(parity and parity["checked"] and parity.get("e2e_checked", True)), "parity": parity,
            "clocks": clk.summary(),
        }
        if e2e_bgzf is not None:
            result["e2e_bgzf"] = e2e_bgzf
        if strong is not None:
            result["strong"] = strong
        if cpu_baseline is not None:
            result["cpu_baseline"] = cpu_baseline
    tr.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(result))


def run_reference(args):
    """The reference's CPU implementation of the path on the host cores: the oracle port (cpu_baseline.kind
    "port"), all host threads, a bounded sample of the same workload per step."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from bystro_vcf_b200 import synth
    from oracle import oracle as O

    spec = CONFIGS[args.config]
    n_samples, seed, shape = spec["n_samples"], spec["seed"], spec["shape"]
    lines = args.lines or spec["lines"]
    threads = os.cpu_count() or 1
    bpl = {"chr1": 10200, "chr1_filters": 10200, "sites": 175, "biobank": 800_100}[shape]
    n = max(16, min(lines, int(args.ref_lines * 10400 / bpl)))  # a byte budget: --ref-lines chr1-shape lines
    body = synth.host_lines(seed, n_samples, shape, 0, n, threads)
    chrom = synth.chrom_line(seed, n_samples)
    cfg = oracle_config(spec)
    for _ in range(args.warmup):
        O.process_block(cfg, chrom, body, threads=threads)
    t0 = time.perf_counter()
    rows = 0
    for _ in range(args.steps):
        r = O.process_block(cfg, chrom, body, threads=threads)
        rows = r.n_rows
    dt = time.perf_counter() - t0
    value = n * args.steps / dt
    sample = ("first %d variants of the workload per step (%.1f MB), in RAM, rows to memory; a per-variant rate: the "
              "whole workload is %d variants per GPU" % (n, len(body) / 1e6, lines))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "variants/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "%s, %d variants x %d samples per GPU (seed %d), %s"
                               % (spec["name"], lines, n_samples, seed, spec["flags"]),
                   "variants_per_gpu": lines, "samples": n_samples, "sample_variants_per_step": n},
        "cpu_baseline": {"value": value, "unit": "variants/s", "cores": threads, "kind": "port", "sample": sample,
                         "rows_per_step": rows,
                         "note": "oracle/ C restatement of main.go; the Go reference cannot be built here (no Go toolchain)"},
        "e2e": {"value": value, "unit": "variants/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="BASELINE.json workload (default c2 = configs[1], the headline)")
    ap.add_argument("--lines", type=int, default=int(os.environ.get("BVCF_BENCH_LINES", "0")),
                    help="variants per GPU (default: the config's full size)")
    ap.add_argument("--e2e-lines", type=int, default=400000, help="variants in the host-resident e2e slice (chr1-shape lines)")
    ap.add_argument("--cpu-lines", type=int, default=200000, help="variants in the CPU-baseline sample")
    ap.add_argument("--ref-lines", type=int, default=100000, help="variants per step of the reference arm")
    ap.add_argument("--parity-lines", type=int, default=2000, help="lines of the timed output checked against the oracle")
    ap.add_argument("--chunk-mb", type=int, default=128)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-bgzf", action="store_true", help="skip the bgzf-compressed end-to-end line")
    ap.add_argument("--bgzf-mb", type=int, default=1024, help="text bytes of the bgzf end-to-end sample")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rows, counts, dosage) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the timed CUDA path (--impl ours)")
    if args.warmup < 3:
        args.warmup = 3 if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
