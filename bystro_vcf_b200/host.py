"""Host side of the B200 transform, mirroring the reference's own interface for this path.

Reference (Go, /root/reference/main.go)      ->  here
  type Config            main.go:63-80       ->  Config
  setup(args)            main.go:82-126      ->  setup(args)
  header / stringHeader  main.go:219-239     ->  header(config) / string_header(config)
  readVcf(cfg, r, w)     main.go:241-396     ->  read_vcf(config, reader, writer)
  processLines(...)      main.go:476-721     ->  Transformer (libbvcf: CUDA kernels behind the C ABI)

The per-line work never runs on the CPU: Transformer raises if libbvcf.so or a CUDA device is missing.
"""
from __future__ import annotations

import ctypes as C
import re
from dataclasses import dataclass, field
from typing import BinaryIO, Dict, List, Optional, Sequence, Tuple

from . import _lib
from ._lib import BvcfError, CChunkStats, CConfig, CDiag, CDosageBatch, CKernelTimes, check

# message table main.go:41-51, indexed by BVCF_DIAG_* code
DIAG_TEXT = {
    1: "REF == ALT",
    2: "ALT not ACTG",
    3: "1st base REF != ALT",
    4: "Invalid POS",
    5: "1st base ALT != REF",
    6: "Mixed indel/snp sites not supported",
    7: "1st base REF != ALT",   # inside the ALT list: logged as "ALT#%d" (main.go:835)
    8: "Invalid POS",           # inside the ALT list: logged without an ALT number (main.go:827)
}


def format_diag(chrom: str, pos: str, alt_no: int, code: int) -> str:
    """The reference's log.Printf line for one diagnostic (formats differ per call site, main.go:730-986)."""
    msg = DIAG_TEXT.get(code, "?")
    if code == 1:
        return "%s:%s : %s" % (chrom, pos, msg)
    if code in (6, 7):
        return "%s:%s ALT#%d %s" % (chrom, pos, alt_no, msg)
    if code == 8:
        return "%s:%s %s" % (chrom, pos, msg)
    return "%s:%s ALT #%d %s" % (chrom, pos, alt_no, msg)

# parse.Header of github.com/bystrogenomics/bystro-utils (pinned by main_test.go:79-80)
PARSE_HEADER = ["chrom", "pos", "type", "ref", "alt", "trTv", "heterozygotes", "heterozygosity", "homozygotes",
                "homozygosity", "missingGenos", "missingness", "ac", "an", "sampleMaf"]


class NotAVcfError(ValueError):
    """log.Fatal("Not a VCF file") main.go:263 / log.Fatal("No header found") main.go:293"""


@dataclass
class Config:
    """main.go:63-80.  Field names follow the reference's flags."""

    inPath: str = ""
    outPath: str = ""
    noOut: bool = False
    dosageMatrixOutPath: str = ""
    sampleListPath: str = ""
    famPath: str = ""
    errPath: str = ""
    emptyField: str = "!"
    fieldDelimiter: str = ";"
    keepID: bool = False
    keepInfo: bool = False
    keepQual: bool = False
    keepPos: bool = False
    cpuProfile: str = ""
    allowedFilters: Optional[Dict[str, bool]] = None   # None == nil map: every FILTER allowed
    excludedFilters: Optional[Dict[str, bool]] = None  # None == nil map: nothing excluded
    # not in the reference: which GPU, chunking
    device: int = 0
    chunkBytes: int = 64 << 20
    normalizeHeader: bool = True
    # not in the reference: the rows leave as bgzf blocks deflated on the GPU (stands in for the `| pigz -c` behind the
    # reference, README.md:10,71); --bgzfOut
    bgzfOut: bool = False
    # --bgzfLevel N: how hard the GPU deflates those rows, 1..9 as `bgzip -l` / `pigz -N` take it; 1 is the fast
    # single-candidate kernel with fixed codes, 2..9 search more and write dynamic Huffman codes
    bgzfLevel: int = 1
    # --regions / --regionsFile: only the records inside these (contig, 1-based inclusive beg, end) are transformed; None:
    # every record (bvcf_set_regions)
    regions: Optional[List[Tuple[bytes, int, int]]] = None


_STRING_FLAGS = {"in": "inPath", "fam": "famPath", "err": "errPath", "out": "outPath", "dosageOutput": "dosageMatrixOutPath",
                 "sample": "sampleListPath", "emptyField": "emptyField", "fieldDelimiter": "fieldDelimiter",
                 "cpuProfile": "cpuProfile", "allowFilter": None, "excludeFilter": None, "regions": None,
                 "regionsFile": None}
_BOOL_FLAGS = {"noOut": "noOut", "keepId": "keepID", "keepQual": "keepQual", "keepPos": "keepPos", "keepInfo": "keepInfo",
               "bgzfOut": "bgzfOut"}
_INT_FLAGS = {"bgzfLevel": "bgzfLevel"}
REGION_MAX = (1 << 63) - 1  # the end of an open region ("chr", "chr:beg-")


def _pos_int(s: str) -> Optional[int]:
    """a decimal number of 0..2^63-1 without a sign, or None"""
    return int(s) if s and len(s) <= 19 and s.isascii() and s.isdigit() and int(s) <= REGION_MAX else None


def parse_regions(arg: str) -> List[Tuple[bytes, int, int]]:
    """--regions chr|chr:pos|chr:beg-end|chr:beg-[,...] (bcftools -r): 1-based inclusive (contig, beg, end); the position
    part follows the last ':'.  ValueError on a malformed item."""
    out = []
    for item in arg.split(","):
        chrom, beg, end = item, 1, REGION_MAX
        if ":" in item:
            chrom, r = item.rsplit(":", 1)
            b, dash, e = r.partition("-")
            beg = _pos_int(b)
            end = beg if not dash else (REGION_MAX if e == "" else _pos_int(e))
            if beg is None or end is None or beg < 1 or beg > end:
                chrom = ""
        if not chrom:
            raise ValueError(f'--regions: malformed region "{item}"')
        out.append((chrom.encode(), beg, end))
    return out


def read_regions_file(path: str) -> List[Tuple[bytes, int, int]]:
    """--regionsFile: BED (0-based, half-open) -> 1-based inclusive (contig, beg, end).  "#", "track" and "browser" lines
    and blank lines are skipped, columns past the third are ignored; an empty interval holds no position.  ValueError on
    an unreadable file, a line with fewer than three columns or start > end."""
    try:
        with open(path, "rb") as f:
            data = f.read()
    except OSError as e:
        raise ValueError(f"--regionsFile: {path}: {e.strerror}") from None
    out = []
    for no, line in enumerate(data.split(b"\n"), 1):
        col = line.rstrip(b"\r").replace(b"\t", b" ").split()
        if not col or col[0].startswith(b"#") or col[0] in (b"track", b"browser"):
            continue
        where = f"--regionsFile: {path} line {no}: "
        if len(col) < 3:
            raise ValueError(where + "fewer than three columns")
        b, e = _pos_int(col[1].decode("latin-1")), _pos_int(col[2].decode("latin-1"))
        if b is None or e is None:
            raise ValueError(where + "start and end must be non-negative integers")
        if b > e:
            raise ValueError(where + "start > end")
        if b < e:
            out.append((col[0], b + 1, e))
    return out


def _go_int(val: str) -> Optional[int]:
    """strconv.ParseInt(val, 0, 64), what Go's `flag` package reads an int flag with (0x.., 0o.., 0b.., 0.. octal,
    underscores between digits); None when val is not such an integer"""
    digits = val.lstrip("+-")
    if val != val.strip() or len(val) - len(digits) > 1:
        return None
    try:
        v = int(val, 8) if len(digits) > 1 and digits[0] == "0" and digits[1] in "01234567_" else int(val, 0)
    except ValueError:
        return None
    return v if -(1 << 63) <= v < (1 << 63) else None


def setup(args: Optional[Sequence[str]] = None) -> Config:
    """main.go:82-126 with Go `flag` syntax: -x/--x, --x=v / --x v, bool flags --x / --x=true|false,
    parsing stops at the first non-flag argument or after "--"."""
    import sys

    a = list(sys.argv[1:] if args is None else args)
    cfg = Config()
    allow, exclude = "PASS,.", ""
    level_given = False
    regions = None
    i = 0
    while i < len(a):
        s = a[i]
        if len(s) < 2 or s[0] != "-":
            break
        if s == "--":
            break
        name = s[2:] if s.startswith("--") else s[1:]
        if not name or name[0] in "-=":
            raise ValueError(f"bad flag syntax: {s}")
        val = None
        if "=" in name:
            name, val = name.split("=", 1)
        if name in _BOOL_FLAGS:
            if val is None:
                b = True
            else:
                lv = val
                if lv in ("1", "t", "T", "true", "TRUE", "True"):
                    b = True
                elif lv in ("0", "f", "F", "false", "FALSE", "False"):
                    b = False
                else:
                    raise ValueError(f"invalid boolean value {val!r} for -{name}")
            setattr(cfg, _BOOL_FLAGS[name], b)
        elif name in _INT_FLAGS:
            if val is None:
                i += 1
                if i >= len(a):
                    raise ValueError(f"flag needs an argument: -{name}")
                val = a[i]
            v = _go_int(val)
            if v is None:
                raise ValueError(f'invalid value "{val}" for flag -{name}: parse error')
            setattr(cfg, _INT_FLAGS[name], v)
            level_given = True
        elif name in _STRING_FLAGS:
            if val is None:
                i += 1
                if i >= len(a):
                    raise ValueError(f"flag needs an argument: -{name}")
                val = a[i]
            if name in ("regions", "regionsFile"):
                regions = (regions or []) + (read_regions_file(val) if name == "regionsFile" else parse_regions(val))
            elif name == "allowFilter":
                allow = val
            elif name == "excludeFilter":
                exclude = val
            else:
                setattr(cfg, _STRING_FLAGS[name], val)
        else:
            raise ValueError(f"flag provided but not defined: -{name}")
        i += 1
    if allow != "" and allow != "*":  # main.go:108-114
        cfg.allowedFilters = {v.strip(): True for v in allow.split(",")}
    if exclude != "":  # main.go:117-123
        cfg.excludedFilters = {v.strip(): True for v in exclude.split(",")}
    if not 1 <= cfg.bgzfLevel <= 9:
        raise ValueError(f"--bgzfLevel must be 1..9, not {cfg.bgzfLevel}")
    if level_given and not cfg.bgzfOut:
        raise ValueError("--bgzfLevel needs --bgzfOut")
    if regions is not None and not regions:
        raise ValueError("--regionsFile: no intervals")
    cfg.regions = regions
    return cfg


def header(config: Config) -> List[str]:
    """main.go:223-239"""
    h = list(PARSE_HEADER)
    if config.keepPos:
        h.append("vcfPos")
    if config.keepID:
        h.append("id")
    if config.keepInfo:
        h += ["alleleIdx", "info"]
    return h


def string_header(config: Config) -> str:
    """main.go:219-221"""
    return "\t".join(header(config))


@dataclass
class ChunkResult:
    tsv: bytes
    n_lines: int
    n_records: int
    n_rows: int
    diags: List[tuple] = field(default_factory=list)          # (line_no, alt_no, code)
    diag_starts: List[int] = field(default_factory=list)      # byte offset of each diagnostic's line in the chunk
    loci: List[bytes] = field(default_factory=list)
    dosage: Optional[object] = None  # numpy int8 [rows, samples]
    retries: int = 0
    diag_fields: List[tuple] = field(default_factory=list)    # (CHROM, POS) of each diagnostic's line, when asked for


def _unpack_dosage(dos):
    """bvcf_dosage_batch -> (list of locus strings, numpy int8 [rows, samples]) copies"""
    import numpy as np

    if not dos.n_rows:
        return [], None
    nr, ns = dos.n_rows, dos.n_samples
    dosage = np.frombuffer(C.string_at(dos.dosage, nr * ns), dtype=np.int8).reshape(nr, ns).copy()
    offs = np.ctypeslib.as_array(dos.loci_off, shape=(nr + 1,)).tolist()
    blob = C.string_at(dos.loci, offs[-1])
    return [blob[offs[i]:offs[i + 1]] for i in range(nr)], dosage


def locus_at(block, start: int):
    """CHROM and POS text of the line that starts at block[start]: what the reference's log lines start with
    (main.go:730-986 "%s:%s ...")."""
    f = bytes(block[start:start + 4096]).split(b"\t", 2)
    if len(f) < 3:
        return "?", "?"
    return f[0].decode("latin-1"), f[1].decode("latin-1")


class Transformer:
    """One GPU's processLines: owns a bvcf_ctx.  Not thread-safe (one host thread per GPU)."""

    def __init__(self, config: Config, eol_width: int = 1, n_slots: int = 3, max_chunk_bytes: int = 0,
                 resident_subchunk_bytes: int = 0):
        L = _lib.lib()
        self._L = L
        self._keep = []
        c = CConfig()
        c.empty_field = config.emptyField.encode()
        c.field_delim = config.fieldDelimiter.encode()
        c.keep_id, c.keep_info, c.keep_pos = int(config.keepID), int(config.keepInfo), int(config.keepPos)
        c.want_tsv = int(not config.noOut)
        c.want_dosage = int(config.dosageMatrixOutPath != "")
        if config.allowedFilters is None:
            c.n_allow, c.allow = -1, None
        else:
            vals = [k.encode() for k, v in config.allowedFilters.items() if v]
            arr = (C.c_char_p * max(1, len(vals)))(*vals)
            self._keep.append(arr)
            c.allow, c.n_allow = arr, len(vals)
        if not config.excludedFilters:
            c.n_exclude, c.exclude = 0, None
        else:
            vals = [k.encode() for k, v in config.excludedFilters.items() if v]
            arr = (C.c_char_p * max(1, len(vals)))(*vals)
            self._keep.append(arr)
            c.exclude, c.n_exclude = arr, len(vals)
        c.eol_width = eol_width
        c.normalize_dots = int(config.normalizeHeader)
        c.n_slots = n_slots
        c.max_chunk_bytes = max_chunk_bytes
        c.resident_subchunk_bytes = resident_subchunk_bytes
        self._cconfig = c
        self.config = config
        self.n_slots = n_slots
        ctx = C.c_void_p()
        rc = L.bvcf_create(C.byref(ctx), config.device, C.byref(c))
        if rc != 0:
            raise BvcfError(f"bvcf_create failed ({rc}): {L.bvcf_strerror(rc).decode()} -- a CUDA device is required, "
                            "there is no CPU fallback")
        self._ctx = ctx
        self.n_samples = 0

    def close(self):
        if getattr(self, "_ctx", None):
            self._L.bvcf_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- header ---------------------------------------------------------------------------------
    def set_header(self, chrom_line: bytes) -> None:
        check(self._L.bvcf_set_header(self._ctx, chrom_line, len(chrom_line)), self._ctx, "bvcf_set_header")
        n = len(chrom_line.rstrip(b"\r\n").split(b"\t"))
        self.n_samples = max(n - 9, 0)

    def set_regions(self, regions: Optional[Sequence[Tuple[bytes, int, int]]]) -> None:
        """Only the records inside these (contig, 1-based inclusive beg, end) are transformed, on both paths
        (bvcf_set_regions); None or an empty list: every record."""
        regions = list(regions or [])
        n = len(regions)
        names = (C.c_char_p * max(n, 1))(*[c.encode() if isinstance(c, str) else bytes(c) for c, _, _ in regions])
        beg = (C.c_int64 * max(n, 1))(*[b for _, b, _ in regions])
        end = (C.c_int64 * max(n, 1))(*[e for _, _, e in regions])
        check(self._L.bvcf_set_regions(self._ctx, names, beg, end, n), self._ctx, "bvcf_set_regions")

    # -- streaming path ---------------------------------------------------------------------------
    def submit(self, seq: int, chunk) -> None:
        """chunk: bytes-like or (address, length).  It must stay alive until collect(seq)."""
        if isinstance(chunk, tuple):
            addr, n = chunk
        else:
            n = len(chunk)
            if isinstance(chunk, bytes):
                addr = C.cast(C.c_char_p(chunk), C.c_void_p).value
            else:
                addr = C.addressof((C.c_char * n).from_buffer(chunk)) if n else 0
            self._keep_chunk = getattr(self, "_keep_chunk", {})
            self._keep_chunk[seq] = chunk
        check(self._L.bvcf_submit(self._ctx, seq, addr, n), self._ctx, "bvcf_submit")

    def submit_bgzf(self, seq: int, comp, skip: int = 0, tail: bytes = b"") -> None:
        """A chunk given as whole bgzf blocks: its text is inflate(comp)[skip:] + tail and must end with a newline.
        comp: bytes-like or (address, length).  The blocks are inflated on the GPU and every member's CRC-32 and ISIZE
        checked there: collect(seq) raises BvcfError for a corrupt member."""
        if isinstance(comp, tuple):
            addr, n = comp
        else:
            comp = bytes(comp) if not isinstance(comp, bytes) else comp
            n = len(comp)
            addr = C.cast(C.c_char_p(comp), C.c_void_p).value
        tail = bytes(tail)
        self._keep_chunk = getattr(self, "_keep_chunk", {})
        self._keep_chunk[seq] = (comp, tail)
        check(self._L.bvcf_submit_bgzf(self._ctx, seq, addr, n, skip, C.cast(C.c_char_p(tail), C.c_void_p).value, len(tail)),
              self._ctx, "bvcf_submit_bgzf")

    def _diag_fields(self, seq: int, n: int) -> List[tuple]:
        """(CHROM, POS) of each diagnostic of collected chunk seq, gathered on the device (bvcf_diag_fields)"""
        text, off = C.c_void_p(), C.POINTER(C.c_uint64)()
        check(self._L.bvcf_diag_fields(self._ctx, seq, C.byref(text), C.byref(off)), self._ctx, "bvcf_diag_fields")
        if n == 0:
            return []
        blob = C.string_at(text, off[n]) if off[n] else b""
        out = []
        for i in range(n):
            f = blob[off[i]:off[i + 1]].split(b"\t", 1)
            out.append((f[0].decode("latin-1"), f[1].decode("latin-1")) if len(f) == 2 else ("?", "?"))
        return out

    def collect(self, seq: int, copy: bool = True, diag_fields: bool = False) -> ChunkResult:
        """Rows, dosage batch and diagnostics of chunk seq, in input order.  diag_fields: also the CHROM and POS of each
        diagnostic's line (out.diag_fields), read on the device -- what a bgzf chunk's log lines need."""
        import numpy as np

        tsv = C.c_void_p()
        n = C.c_size_t()
        dos = CDosageBatch()
        dg = C.POINTER(CDiag)()
        nd = C.c_size_t()
        st = CChunkStats()
        check(self._L.bvcf_collect(self._ctx, seq, C.byref(tsv), C.byref(n), C.byref(dos), C.byref(dg), C.byref(nd),
                                   C.byref(st)), self._ctx, "bvcf_collect")
        out = ChunkResult(tsv=C.string_at(tsv, n.value) if n.value else b"", n_lines=st.n_lines,
                          n_records=st.n_records, n_rows=st.n_rows, retries=st.retries)
        out.diags = [(dg[i].line_no, dg[i].alt_no, dg[i].code) for i in range(nd.value)]
        out.diag_starts = [dg[i].line_start for i in range(nd.value)]
        out.loci, out.dosage = _unpack_dosage(dos)
        if diag_fields:
            out.diag_fields = self._diag_fields(seq, nd.value)
        check(self._L.bvcf_release(self._ctx, seq), self._ctx, "bvcf_release")
        if hasattr(self, "_keep_chunk"):
            self._keep_chunk.pop(seq, None)
        return out

    def process(self, block: bytes) -> ChunkResult:
        """One newline-aligned block of data lines in, rows out (blocking convenience)."""
        self.submit(0, block)
        return self.collect(0)

    # -- device-resident path -----------------------------------------------------------------------
    def resident_alloc(self, in_bytes: int, out_capacity: int):
        d_in, d_out = C.c_void_p(), C.c_void_p()
        check(self._L.bvcf_resident_alloc(self._ctx, in_bytes, out_capacity, C.byref(d_in), C.byref(d_out)), self._ctx,
              "bvcf_resident_alloc")
        return d_in.value, d_out.value

    def resident_upload(self, offset: int, data) -> None:
        if isinstance(data, tuple):
            addr, n = data
        else:
            n = len(data)
            addr = C.cast(C.c_char_p(bytes(data)), C.c_void_p).value if not isinstance(data, bytes) else \
                C.cast(C.c_char_p(data), C.c_void_p).value
        check(self._L.bvcf_resident_upload(self._ctx, offset, addr, n), self._ctx, "bvcf_resident_upload")

    def resident_inflate_bgzf(self, comp, dst_offset: int = 0) -> int:
        """bgzf blocks (bytes-like or (address, length), pinned for full PCIe speed) -> text in the resident input
        region at dst_offset, inflated on the GPU.  Returns the number of text bytes."""
        if isinstance(comp, tuple):
            addr, n = comp
        else:
            n = len(comp)
            comp = bytes(comp) if not isinstance(comp, bytes) else comp
            self._keep_comp = comp
            addr = C.cast(C.c_char_p(comp), C.c_void_p).value
        out = C.c_size_t()
        check(self._L.bvcf_resident_inflate_bgzf(self._ctx, addr, n, dst_offset, C.byref(out)), self._ctx,
              "bvcf_resident_inflate_bgzf")
        return out.value

    def resident_run(self, length: int, want_times: bool = True, begin: int = 0):
        st, kt = CChunkStats(), CKernelTimes()
        check(self._L.bvcf_resident_run_at(self._ctx, begin, length, C.byref(st), C.byref(kt) if want_times else None), self._ctx,
              "bvcf_resident_run")
        stats = {k: getattr(st, k) for k, _ in CChunkStats._fields_}
        times = {k: getattr(kt, k) for k, _ in CKernelTimes._fields_}
        return stats, times

    def resident_results(self):
        """(loci, dosage, [(line_no, alt_no, code, line_start)]) of the last resident run"""
        dos = CDosageBatch()
        dg = C.POINTER(CDiag)()
        nd = C.c_size_t()
        check(self._L.bvcf_resident_results(self._ctx, C.byref(dos), C.byref(dg), C.byref(nd)), self._ctx, "bvcf_resident_results")
        loci, dosage = _unpack_dosage(dos)
        return loci, dosage, [(dg[i].line_no, dg[i].alt_no, dg[i].code, dg[i].line_start) for i in range(nd.value)]

    def resident_write_output(self, offset: int, data: bytes) -> None:
        check(self._L.bvcf_resident_write_output(self._ctx, offset, data, len(data)), self._ctx, "bvcf_resident_write_output")

    def resident_download_bgzf(self, offset: int, length: int, level: int = 1) -> bytes:
        """rows [offset, offset + length) of the resident output, deflated on the GPU at `level` (1..9, see
        bvcf_resident_download_bgzf_level): whole bgzf blocks (append bgzf.EOF_BLOCK at the end of a file)"""
        cap = length + length // 4 + (1 << 16)
        buf = C.create_string_buffer(cap)
        n = C.c_size_t()
        check(self._L.bvcf_resident_download_bgzf_level(self._ctx, offset, length, level, buf, cap, C.byref(n)), self._ctx,
              "bvcf_resident_download_bgzf_level")
        return buf.raw[:n.value]

    def resident_download(self, offset: int, length: int) -> bytes:
        buf = C.create_string_buffer(max(length, 1))
        check(self._L.bvcf_resident_download(self._ctx, offset, buf, length), self._ctx, "bvcf_resident_download")
        return buf.raw[:length]

    def resident_peek(self, offset: int, length: int, addr: int = 0) -> bytes:
        """bytes of the resident INPUT region (device-generated workloads); into `addr` when given."""
        if addr:
            check(self._L.bvcf_resident_peek(self._ctx, offset, addr, length), self._ctx, "bvcf_resident_peek")
            return b""
        buf = C.create_string_buffer(max(length, 1))
        check(self._L.bvcf_resident_peek(self._ctx, offset, buf, length), self._ctx, "bvcf_resident_peek")
        return buf.raw[:length]

    def resident_line_index(self, cap: int):
        import numpy as np

        starts = np.zeros(cap, dtype=np.uint64)
        lens = np.zeros(cap, dtype=np.uint32)
        an = np.zeros(cap, dtype=np.uint32)
        n = C.c_size_t()
        check(self._L.bvcf_resident_line_index(
            self._ctx, starts.ctypes.data_as(C.POINTER(C.c_uint64)), lens.ctypes.data_as(C.POINTER(C.c_uint32)),
            an.ctypes.data_as(C.POINTER(C.c_uint32)), cap, C.byref(n)), self._ctx, "bvcf_resident_line_index")
        k = min(cap, n.value)
        return starts[:k], lens[:k], an[:k], n.value

    @property
    def launches(self) -> int:
        return self._L.bvcf_launch_count(self._ctx)


# ---- stream driver ------------------------------------------------------------------------------------

def find_end_of_line(first: bytes):
    """parse.FindEndOfLine (main.go:250): (eol byte, numChars, first line without EOL, bytes consumed)."""
    m = re.search(rb"[\r\n]", first)
    if not m:
        return None
    i = m.start()
    if first[i:i + 1] == b"\r":
        if first[i + 1:i + 2] == b"\n":
            return b"\n", 2, first[:i], i + 2
        return b"\r", 1, first[:i], i + 1
    return b"\n", 1, first[:i], i + 1


def parse_preamble(data: bytes):
    """main.go:250-294: version-line check, locate the #CHROM line.
    Returns (eol_width, chrom_line_without_eol, offset_of_first_data_line) or raises NotAVcfError.
    `data` only has to hold the meta lines + header."""
    r = find_end_of_line(data)
    if r is None:
        raise NotAVcfError("Not a VCF file")
    eol, width, version, p = r
    if b"##fileformat=VCFv4" not in version:  # regexp.MatchString main.go:256
        raise NotAVcfError("Not a VCF file")
    if eol != b"\n":
        raise NotAVcfError("bare-CR line endings are not supported by the GPU path")
    while True:
        e = data.find(eol, p)
        if e < 0:
            raise NotAVcfError("No header found")
        row = data[p:e + 1]
        content = row[:len(row) - width] if len(row) >= width else b""
        if content.split(b"\t")[0] == b"#CHROM":
            return width, content, e + 1
        p = e + 1


class PinnedRing:
    """n pinned host buffers (bvcf_host_alloc) with writable views: chunks are read or copied into them so that
    bvcf_submit's H2D copy is a true asynchronous DMA."""

    def __init__(self, n: int, cap: int):
        self.cap = cap
        self.ptrs = []
        self.views = []
        L = _lib.lib()
        for _ in range(n):
            p = C.c_void_p()
            check(L.bvcf_host_alloc(C.byref(p), cap), None, "bvcf_host_alloc")
            self.ptrs.append(p.value)
            self.views.append(memoryview((C.c_char * cap).from_address(p.value)).cast("B"))
        libc = C.CDLL(None)
        libc.memrchr.restype = C.c_void_p
        libc.memrchr.argtypes = [C.c_void_p, C.c_int, C.c_size_t]
        self._memrchr = libc.memrchr

    def last_newline(self, i: int, n: int) -> int:
        """length of the longest newline-terminated prefix of buffer i's first n bytes, or -1"""
        if n <= 0:
            return -1
        r = self._memrchr(self.ptrs[i], 10, n)
        return -1 if not r else r - self.ptrs[i] + 1

    def close(self):
        L = _lib.lib()
        self.views = []
        for p in self.ptrs:
            L.bvcf_host_free(p)
        self.ptrs = []


def read_preamble(buf, gz: bool, reader: Optional[BinaryIO] = None):
    """parse_preamble on the first bytes of an input: (eol_width, chrom_line, data_off), data_off counted in text bytes.
    buf holds the input read so far -- a bytearray that grows from `reader` until the #CHROM line is in sight, or the
    whole input (bytes, mmap) when there is no reader.  A bgzf input's first blocks are inflated on the host, each one
    checked against its CRC-32 (BvcfError when one fails)."""
    from . import bgzf

    want = 1 << 20
    while True:
        while reader is not None and len(buf) < want:
            more = reader.read(want - len(buf))
            if not more:
                reader = None
            buf += more
        try:
            text = bgzf.inflate_host(buf, want) if gz else bytes(buf[:want])
        except ValueError as e:
            raise BvcfError(str(e)) from None
        try:
            return parse_preamble(text)
        except NotAVcfError as e:
            if (str(e) == "Not a VCF file" and re.search(rb"[\r\n]", text)) or (reader is None and len(text) < want):
                raise
            want *= 4


class Sink:
    """Where the results of a run go (main.go:296-343, 398-445): rows to the writer, dosage batches to the Arrow file, the
    reference's log lines to diag_sink(text, line_no, alt_no, code), and the totals.  Built once from the #CHROM line:
    it writes the sample list and opens the dosage file -- or, when the VCF has no samples, writes an empty one."""

    def __init__(self, config: Config, chrom_line: bytes, writer: Optional[BinaryIO] = None, diag_sink=None):
        self.config, self.writer, self.diag_sink = config, writer, diag_sink
        names = [s.replace(b".", b"_") if config.normalizeHeader else s for s in chrom_line.split(b"\t")[9:]]
        if config.sampleListPath and not config.noOut:  # writeSampleListIfWanted / makeSampleList main.go:398-445
            with open(config.sampleListPath, "wb") as fh:
                fh.write(b"".join(s + b"\n" for s in names))
        self.arrow = None
        if config.dosageMatrixOutPath and not names:
            open(config.dosageMatrixOutPath, "wb").close()  # main.go:308-318: no samples, an empty dosage file
        elif config.dosageMatrixOutPath:
            from .dosage import DosageWriter  # Arrow IPC framing (SURVEY 8f-2)

            self.arrow = DosageWriter(config.dosageMatrixOutPath, names)
        self.totals = {"n_lines": 0, "n_records": 0, "n_rows": 0, "out_bytes": 0}

    def put(self, res: ChunkResult, loci) -> None:
        """one chunk's results, in input order.  res.tsv is written as it is (bgzf blocks with bgzfOut); loci yields the
        (CHROM, POS) of each diagnostic's line -- read from the chunk's text with locus_at, or res.diag_fields."""
        if self.writer is not None and not self.config.noOut:
            self.writer.write(res.tsv)
        if self.arrow is not None and res.dosage is not None:
            self.arrow.write(res.loci, res.dosage)
        if self.diag_sink is not None and res.diags:
            for (ln, alt_no, code), (chrom, pos) in zip(res.diags, loci):
                self.diag_sink(format_diag(chrom, pos, alt_no, code), self.totals["n_lines"] + ln, alt_no, code)
        self.totals["n_lines"] += res.n_lines
        self.totals["n_records"] += res.n_records
        self.totals["n_rows"] += res.n_rows
        self.totals["out_bytes"] += len(res.tsv)

    def close(self) -> None:
        if self.arrow is not None:
            self.arrow.close()
            self.arrow = None


def _read_vcf_resident(config: Config, head: bytes, reader: BinaryIO, writer: Optional[BinaryIO], batch_text: int = 512 << 20,
                       diag_sink=None) -> dict:
    """readVcf (main.go:241-396) for bgzfOut: the rows are deflated where they are made (replaces the `| pigz -c` behind
    the reference, README.md:10), so the input goes through one GPU's resident regions a group at a time -- plain text
    uploaded, or whole bgzf blocks inflated on the GPU.  The partial line at a group's end is carried into the next."""
    from . import bgzf

    buf = bytearray(head)
    gz = bgzf.is_bgzf(buf)
    width, chrom_line, data_off = read_preamble(buf, gz, reader)
    eof = False

    def fill(n: int):
        nonlocal eof
        while not eof and len(buf) < n:
            more = reader.read(max(n - len(buf), 8 << 20))
            if not more:
                eof = True
            else:
                buf.extend(more)

    compressed_bytes = in_bytes = 0
    max_line = 8 << 20  # room for the carried partial line
    # what is read: the input from its data lines on, or -- with regions and an index beside a bgzf file -- the index's
    # spans (bgzf.index_views), each from its first block to its last; a partial line at a span's end is dropped
    sources = [(buf, data_off)]
    if gz and config.regions and config.inPath:
        import mmap

        with open(config.inPath, "rb") as f:
            whole = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ)
        try:
            views = bgzf.index_views(whole, config.inPath, config.regions)
        except ValueError as e:
            raise BvcfError(str(e)) from None
        if views is not None:
            sources = [(bytearray(whole[lo:hi]), skip) for lo, hi, skip in views]
            eof = True
    sink = Sink(config, chrom_line, writer, diag_sink)
    try:
        with Transformer(config, eol_width=width) as tr:
            tr.set_header(chrom_line)
            if config.regions is not None:
                tr.set_regions(config.regions)
            tr.resident_alloc(batch_text + max_line + (1 << 20), batch_text // 4 + (64 << 20))
            for buf, begin in sources:  # a source's first group holds what comes before its data lines: skipped on the device
                carry = b""
                while True:
                    # ---- a group: whole blocks worth about batch_text bytes of text, or batch_text bytes of plain text ----
                    p = text = 0
                    if not gz:
                        fill(batch_text)
                        p = min(len(buf), batch_text)
                    while gz and text < batch_text:
                        fill(p + (1 << 16) + 18)
                        try:
                            bs = bgzf.block_size(buf, p)
                        except ValueError as e:  # not bgzf, or a block that claims ISIZE 0 but holds text
                            raise BvcfError("bgzf input: %s" % e) from None
                        if bs == 0 or p + bs > len(buf):
                            if not eof:
                                fill(p + max(bs, 1 << 16) + 18)
                                continue
                            if p < len(buf):
                                raise BvcfError("bgzf input: truncated block at the end")
                            break
                        text += int.from_bytes(buf[p + bs - 4:p + bs], "little")
                        p += bs
                    if p == 0:
                        break
                    group = bytes(buf[:p])
                    del buf[:p]
                    if carry:
                        tr.resident_upload(0, carry)
                    if gz:
                        n_text = tr.resident_inflate_bgzf(group, len(carry))
                    else:
                        tr.resident_upload(len(carry), group)
                        n_text = len(group)
                    total = len(carry) + n_text
                    compressed_bytes += len(group)
                    # ---- the longest newline-terminated prefix; what follows it is carried into the next group ----
                    tail_n = min(total - begin, max_line)
                    tail = tr.resident_peek(total - tail_n, tail_n) if tail_n > 0 else b""
                    k = tail.rfind(b"\n")
                    if k < 0:
                        if tail_n == total - begin:  # no complete line in this group at all
                            carry = carry + tr.resident_peek(len(carry), n_text) if begin == 0 else tr.resident_peek(begin, total - begin)
                            begin = 0
                            continue
                        raise BvcfError("a single line exceeds %d bytes" % max_line)
                    end = total - tail_n + k + 1
                    stats, _ = tr.resident_run(end, want_times=False, begin=begin)
                    rows = b""
                    if writer is not None and not config.noOut and stats["out_bytes"]:
                        rows = tr.resident_download_bgzf(0, stats["out_bytes"], config.bgzfLevel)
                    loci, dosage, diags = tr.resident_results()
                    res = ChunkResult(tsv=rows, n_lines=stats["n_lines"], n_records=stats["n_records"], n_rows=stats["n_rows"],
                                      diags=[d[:3] for d in diags], diag_starts=[d[3] for d in diags], loci=loci, dosage=dosage)
                    sink.put(res, (locus_at(tr.resident_peek(st, min(4096, end - st)), 0) for st in res.diag_starts))
                    in_bytes += end - begin
                    carry = tail[k + 1:]
                    begin = 0
            # an unterminated last line (carry) is dropped (main.go:354-357)
    finally:
        sink.close()
    return {**sink.totals, "in_bytes": in_bytes, "compressed_bytes": compressed_bytes}


def read_vcf(config: Config, reader: BinaryIO, writer: Optional[BinaryIO], diag_sink=None) -> dict:
    """readVcf (main.go:241-396) on the GPU: header discovery on the host, every data line on the device.

    reader/writer are binary file objects (the reference's *bufio.Reader / *bufio.Writer).  Rows are
    written in input order.  The TSV header line is NOT written here (main() does that, main.go:199).
    diag_sink(text, line_no, alt_no, code) receives the reference's log.Printf line for every skipped allele.
    A .vcf.gz (bgzf) input runs on the streaming path of shard.read_vcf_multi with config.device as its one GPU."""
    from . import bgzf, shard

    chunk_bytes = max(int(config.chunkBytes), 1 << 16)
    head = bytearray(reader.read(1 << 20))
    if config.bgzfOut:  # the rows are deflated where they are: on the device
        return _read_vcf_resident(config, head, reader, writer, diag_sink=diag_sink)
    if bgzf.is_bgzf(head):  # .vcf.gz: the compressed bytes go to the GPU, which inflates them (SURVEY 8f-3)
        return shard.read_vcf_multi(config, shard.whole_input(reader, head), writer, [config.device], diag_sink=diag_sink)
    width, chrom_line, off = read_preamble(head, False, reader)
    # chunks are staged in pinned host buffers (bvcf_host_alloc) and read into them directly: a pageable source
    # would make the driver bounce every H2D copy through its own staging buffer
    cap = 2 * chunk_bytes + (64 << 20)
    in_bytes = 0
    sink = Sink(config, chrom_line, writer, diag_sink)
    try:
        with Transformer(config, eol_width=width, max_chunk_bytes=cap) as tr:
            tr.set_header(chrom_line)
            if config.regions is not None:
                tr.set_regions(config.regions)
            ring = PinnedRing(tr.n_slots + 1, cap)
            seq_in = seq_out = 0
            pending = {}  # seq -> the chunk's text (a view of its ring buffer) while it is in flight

            def drain(upto: int):
                nonlocal seq_out
                while seq_out < upto:
                    res = tr.collect(seq_out)
                    text = pending.pop(seq_out)
                    sink.put(res, (locus_at(text, st) for st in res.diag_starts))
                    seq_out += 1

            try:
                slot = 0
                fill = len(head) - off  # bytes waiting in the current buffer
                if fill > cap:
                    raise BvcfError("the VCF preamble does not fit a chunk buffer; raise chunkBytes")
                C.memmove(ring.ptrs[0], bytes(head[off:]), fill)
                eof = False
                while not eof or fill:
                    view = ring.views[slot]
                    while not eof and fill < chunk_bytes:
                        n = reader.readinto(view[fill:min(cap, chunk_bytes)])
                        if not n:
                            eof = True
                            break
                        fill += n
                    cut = ring.last_newline(slot, fill)
                    if cut < 0:
                        if eof:
                            break  # an unterminated last line is dropped (main.go:354-357)
                        if fill >= cap:
                            raise BvcfError("a single line exceeds the chunk capacity; raise chunkBytes")
                        n = reader.readinto(view[fill:cap])
                        if not n:
                            eof = True
                        fill += n or 0
                        continue
                    nxt = (slot + 1) % len(ring.ptrs)
                    if seq_in - seq_out >= tr.n_slots:
                        drain(seq_out + 1)  # frees the next ring buffer too (n_slots + 1 buffers, n_slots in flight)
                    C.memmove(ring.ptrs[nxt], ring.ptrs[slot] + cut, fill - cut)  # carry the partial line
                    pending[seq_in] = view[:cut]
                    tr.submit(seq_in, (ring.ptrs[slot], cut))
                    in_bytes += cut
                    seq_in += 1
                    fill -= cut
                    slot = nxt
                drain(seq_in)
            finally:
                pending.clear()
                ring.close()
    finally:
        sink.close()
    return {**sink.totals, "in_bytes": in_bytes}
