"""`python -m bystro_vcf_b200 [flags]` -- main() of the reference (main.go:134-217) on the GPU path.

Same flags, same stdin/stdout behaviour: header line first (main.go:199), then rows in input order; the
reference's log.Printf lines ("chrom:pos ALT #k message", main.go:730-986) on stderr, or appended to --err.
`--gpus N` (extension) shards the input -- plain or bgzf (.vcf.gz) -- over N GPUs of the box (shard.read_vcf_multi, which
also runs a .vcf.gz on one GPU); `--bgzfOut` (extension) writes the rows as bgzf blocks deflated on the GPU -- with a
.vcf.gz input the command stands for the whole `pigz -d -c in.vcf.gz | bystro-vcf ... | pigz -c > out.gz` of README.md:10."""
from __future__ import annotations

import os
import sys

from ._lib import BvcfError
from .host import NotAVcfError, read_vcf, setup, string_header


def main(argv=None) -> int:
    a = list(sys.argv[1:] if argv is None else argv)
    gpus = 1
    for i, s in enumerate(list(a)):  # extension flag, not in the reference: taken out before setup() sees the rest
        if s in ("--gpus", "-gpus") and i + 1 < len(a):
            gpus = max(1, int(a[i + 1]))
            del a[i:i + 2]
            break
        if s.startswith("--gpus=") or s.startswith("-gpus="):
            gpus = max(1, int(s.split("=", 1)[1]))
            del a[i]
            break
    try:
        cfg = setup(a)
    except ValueError as e:  # a flag error: one line, before anything is read or written
        print(str(e), file=sys.stderr)
        return 1
    err = sys.stderr
    if cfg.errPath:
        # main.go:150-156 opens the file read-only and re-points os.Stderr, which Go's `log` package never
        # looks at again; what the flag evidently means is honoured here: diagnostics are appended to the file.
        try:
            err = open(cfg.errPath, "a")
        except OSError as e:
            print(str(e), file=sys.stderr)
            return 1
    if cfg.noOut and cfg.outPath:
        print("Cannot specify --noOut and --out", file=err)  # main.go:160
        return 1
    if cfg.noOut and not cfg.dosageMatrixOutPath:
        print("When specifying --noOut, must specify --dosageOutput", file=err)  # main.go:164
        return 1
    inp = open(cfg.inPath, "rb") if cfg.inPath else sys.stdin.buffer
    out = None
    if not cfg.noOut:
        if cfg.outPath:
            # os.OpenFile(path, O_WRONLY|O_CREATE, 0644) main.go:172: an existing file is overwritten from offset
            # 0 and NOT truncated, like the reference
            out = os.fdopen(os.open(cfg.outPath, os.O_WRONLY | os.O_CREAT, 0o644), "wb")
        else:
            out = sys.stdout.buffer
        hdr = string_header(cfg).encode() + b"\n"  # main.go:199
        if cfg.bgzfOut:
            from . import bgzf

            hdr = bgzf.compress(hdr, eof=False)
        out.write(hdr)

    def log(text, line_no, alt_no, code):  # the reference's log.Printf sites (main.go:730-986)
        print(text, file=err)

    try:
        if gpus > 1 and cfg.bgzfOut:
            print("--bgzfOut runs on one GPU", file=err)
            return 1
        if gpus > 1:
            from . import shard

            shard.read_vcf_multi(cfg, shard.whole_input(inp), out, list(range(gpus)), diag_sink=log)
        else:
            read_vcf(cfg, inp, out, diag_sink=log)
        if out is not None and cfg.bgzfOut:
            from . import bgzf

            out.write(bgzf.EOF_BLOCK)
    except NotAVcfError as e:
        print(str(e), file=err)  # log.Fatal main.go:263,293
        return 1
    except BvcfError as e:  # a corrupt .vcf.gz member, a line longer than a chunk ...
        print(str(e), file=sys.stderr)
        return 1
    finally:
        if out is not None:
            out.flush()
        if err is not sys.stderr:
            err.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
