"""A raw DEFLATE (RFC 1951) writer for the tests: streams built from explicit choices that zlib's encoder never makes --
codes of any length up to 15 bits, hand-made precodes and code-length runs, single-code and empty distance codes, length
258 written both ways, many blocks per member -- and bgzf members (SAM spec 4.1) around them.  Imported like
ref_vectors.py.  Every stream it builds is checked against zlib.decompress(wbits=-15) by test_bgzf_conformance.py."""
from __future__ import annotations

import random
import struct
import zlib
from typing import List, Optional, Sequence, Tuple, Union

LBASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEXT = [0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0]
DBASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
         6145, 8193, 12289, 16385, 24577]
DEXT = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
FIXED_L = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_D = [5] * 30
MAX_TEXT = 65536  # text bytes a bgzf member may hold

# A token is a literal byte (an int) or a match (length symbol 257..285, its extra bits, distance symbol 0..29, its
# extra bits).  An int 256 is the end-of-block code where a caller wants to place it by hand.
Token = Union[int, Tuple[int, int, int, int]]


class BitWriter:
    """DEFLATE's bit order: values least significant bit first, Huffman codes most significant bit first"""

    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    def bits(self, v: int, n: int) -> None:
        assert 0 <= v < (1 << n) or n == 0 and v == 0
        self.acc |= v << self.n
        self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 0xFF)
            self.acc >>= 8
            self.n -= 8

    def code(self, code: int, length: int) -> None:
        # (the low bits: an over-subscribed code, written for a decoder to refuse, runs past `length` bits)
        self.bits(int(format(code & ((1 << length) - 1), "0%db" % length)[::-1], 2), length)

    def align(self) -> None:
        if self.n:
            self.bits(0, 8 - self.n)

    def raw(self, data: bytes) -> None:
        assert self.n == 0
        self.out += data

    def getvalue(self) -> bytes:
        return bytes(self.out) + (bytes([self.acc]) if self.n else b"")


def canonical(lengths: Sequence[int]) -> List[Optional[int]]:
    """the canonical Huffman codes of a list of code lengths (RFC 1951 3.2.2); None for length 0"""
    bl_count = [0] * 16
    for L in lengths:
        bl_count[L] += 1
    bl_count[0] = 0
    nxt, code = [0] * 16, 0
    for b in range(1, 16):
        code = (code + bl_count[b - 1]) << 1
        nxt[b] = code
    out: List[Optional[int]] = []
    for L in lengths:
        if L:
            out.append(nxt[L])
            nxt[L] += 1
        else:
            out.append(None)
    return out


def limited_lengths(freqs: Sequence[int], maxbits: int) -> List[int]:
    """complete code lengths of at most maxbits bits for the symbols with freqs > 0 (at least two of them get a code: a
    second symbol is added when only one is used)"""
    import heapq

    syms = [s for s, f in enumerate(freqs) if f > 0]
    if len(syms) < 2:
        syms = (syms + [s for s in range(len(freqs)) if s not in syms])[:2]
    lens = [0] * len(freqs)
    heap = [(max(freqs[s], 1), i, [s]) for i, s in enumerate(syms)]
    heapq.heapify(heap)
    k = len(heap)
    while len(heap) > 1:
        fa, _, a = heapq.heappop(heap)
        fb, _, b = heapq.heappop(heap)
        for s in a + b:
            lens[s] += 1
        heapq.heappush(heap, (fa + fb, k, a + b))
        k += 1
    unit = lambda L: 1 << (maxbits - L)  # noqa: E731
    lens = [min(L, maxbits) for L in lens]
    total = sum(unit(L) for L in lens if L)
    full = 1 << maxbits
    by_len = sorted((s for s in syms), key=lambda s: -lens[s])
    while total > full:  # over-subscribed: lengthen the longest code that can still grow
        s = next(s for s in by_len if lens[s] < maxbits)
        total -= unit(lens[s]) - unit(lens[s] + 1)
        lens[s] += 1
        by_len.sort(key=lambda s: -lens[s])
    while total < full:  # incomplete: shorten the longest code that still fits
        s = next(s for s in by_len if total + unit(lens[s]) <= full)
        total += unit(lens[s])
        lens[s] -= 1
        by_len.sort(key=lambda s: -lens[s])
    return lens


def random_lengths(rng: random.Random, n_codes: int, maxbits: int = 15, deep: bool = False) -> List[int]:
    """a multiset of code lengths of a complete code with n_codes >= 2 codes, made by splitting random leaves (deep:
    always the deepest splittable one, so the lengths run 1, 2, 3, ... down to maxbits)"""
    leaves = [1, 1]
    while len(leaves) < n_codes:
        cand = [i for i, L in enumerate(leaves) if L < maxbits]
        i = max(cand, key=lambda i: leaves[i]) if deep else rng.choice(cand)
        L = leaves.pop(i)
        leaves += [L + 1, L + 1]
    return sorted(leaves)


def rle(lengths: Sequence[int]) -> List[Tuple[int, int]]:
    """code-length symbols (sym, extra) for a list of lengths, with runs of 16, 17 and 18 where they fit (over the whole
    list: runs cross from the literal/length lengths into the distance lengths)"""
    out: List[Tuple[int, int]] = []
    i, n = 0, len(lengths)
    while i < n:
        L = lengths[i]
        j = i
        while j < n and lengths[j] == L:
            j += 1
        run = j - i
        if L == 0:
            while run >= 11:
                r = min(run, 138)
                out.append((18, r - 11))
                run -= r
            if run >= 3:
                out.append((17, run - 3))
                run = 0
            out += [(0, 0)] * run
        else:
            out.append((L, 0))
            run -= 1
            while run >= 3:
                r = min(run, 6)
                out.append((16, r - 3))
                run -= r
            out += [(L, 0)] * run
        i = j
    return out


def run_lengths(runs: Sequence[Tuple[int, int]]) -> List[int]:
    """the lengths a list of code-length symbols spells out"""
    out: List[int] = []
    for sym, extra in runs:
        if sym < 16:
            out.append(sym)
        elif sym == 16:
            out += [out[-1]] * (3 + extra)
        elif sym == 17:
            out += [0] * (3 + extra)
        else:
            out += [0] * (11 + extra)
    return out


def match(length: int, dist: int) -> Tuple[int, int, int, int]:
    """the match token of (length, distance); 258 as symbol 285"""
    lc = 28 if length == 258 else max(i for i in range(28) if LBASE[i] <= length)
    dc = max(i for i in range(30) if DBASE[i] <= dist)
    return (257 + lc, length - LBASE[lc], dc, dist - DBASE[dc])


def token_length(t) -> Tuple[int, int]:
    lsym, lx, dsym, dx = t
    return LBASE[lsym - 257] + lx, DBASE[dsym] + dx


def apply(tokens: Sequence[Token], text: bytearray) -> None:
    """append the text of `tokens` to `text` (which holds what the member produced before them)"""
    for t in tokens:
        if isinstance(t, int):
            if t < 256:
                text.append(t)
            continue
        length, dist = token_length(t)
        assert 1 <= dist <= len(text), (dist, len(text))
        src = text[len(text) - dist:len(text) - dist + length]
        text += (src * (length // dist + 1))[:length]  # an overlapping match repeats its last `dist` bytes


def write_tokens(w: BitWriter, tokens: Sequence[Token], llens: Sequence[int], dlens: Sequence[int], eob: bool = True) -> None:
    lc, dc = canonical(llens), canonical(dlens)
    for t in list(tokens) + ([256] if eob else []):
        if isinstance(t, int):
            w.code(lc[t], llens[t])
            continue
        lsym, lx, dsym, dx = t
        w.code(lc[lsym], llens[lsym])
        if lsym <= 284:
            w.bits(lx, LEXT[lsym - 257])
        else:
            assert lx == 0
        w.code(dc[dsym], dlens[dsym])
        w.bits(dx, DEXT[dsym] if dsym < 30 else 0)  # (distance symbols 30 and 31 are invalid: no extra bits)


def stored(w: BitWriter, data: bytes, final: bool, nlen: Optional[int] = None) -> None:
    w.bits(int(final), 1)
    w.bits(0, 2)
    w.align()
    w.raw(struct.pack("<HH", len(data), (len(data) ^ 0xFFFF) if nlen is None else nlen) + data)


def fixed(w: BitWriter, tokens: Sequence[Token], final: bool, eob: bool = True) -> None:
    w.bits(int(final), 1)
    w.bits(1, 2)
    write_tokens(w, tokens, FIXED_L, FIXED_D, eob)


def dynamic(w: BitWriter, tokens: Sequence[Token], final: bool, llens: Sequence[int], dlens: Sequence[int],
            runs: Optional[Sequence[Tuple[int, int]]] = None, precode: Optional[Sequence[int]] = None,
            hclen: Optional[int] = None, hlit: Optional[int] = None, hdist: Optional[int] = None, eob: bool = True) -> None:
    """a dynamic block.  llens / dlens are the code lengths the tokens are written with; runs (default rle(llens + dlens))
    the code-length symbols sent for them, precode (default: limited to 7 bits from the runs) the code-length code,
    hclen / hlit / hdist the header counts (default: what the lengths need)."""
    if runs is None:
        runs = rle(list(llens) + list(dlens))
    if precode is None:
        freq = [0] * 19
        for sym, _ in runs:
            freq[sym] += 1
        precode = limited_lengths(freq, 7)
    if hclen is None:
        hclen = max([4] + [i + 1 for i in range(19) if precode[ORDER[i]]])
    hlit = len(llens) if hlit is None else hlit
    hdist = len(dlens) if hdist is None else hdist
    w.bits(int(final), 1)
    w.bits(2, 2)
    w.bits(hlit - 257, 5)
    w.bits(hdist - 1, 5)
    w.bits(hclen - 4, 4)
    for i in range(hclen):
        w.bits(precode[ORDER[i]], 3)
    pc = canonical(precode)
    for sym, extra in runs:
        w.code(pc[sym], precode[sym])
        if sym >= 16:
            w.bits(extra, (2, 3, 7)[sym - 16])
    write_tokens(w, tokens, llens, dlens, eob)


def subfield(si: bytes, data: bytes) -> bytes:
    return si + struct.pack("<H", len(data)) + data


def member(payload: bytes, text: bytes, crc: Optional[int] = None, isize: Optional[int] = None, before: bytes = b"",
           after: bytes = b"", bsize: Optional[int] = None) -> bytes:
    """a bgzf member around a raw DEFLATE payload: the extra field is `before`, the BC subfield, `after`; the trailer
    is the CRC-32 and size of `text` unless crc / isize override it (bsize overrides the BC value + 1)"""
    xlen = len(before) + 6 + len(after)
    total = 12 + xlen + len(payload) + 8
    bs = total if bsize is None else bsize
    head = b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff" + struct.pack("<H", xlen)
    return (head + before + b"BC\x02\x00" + struct.pack("<H", bs - 1) + after + payload +
            struct.pack("<II", zlib.crc32(text) if crc is None else crc, len(text) if isize is None else isize))


EOF_BLOCK = member(b"\x03\x00", b"")


def inflate(payload: bytes) -> bytes:
    """zlib's raw inflate, which must consume the whole payload"""
    d = zlib.decompressobj(-15)
    out = d.decompress(payload) + d.flush()
    if not d.eof:
        raise zlib.error("incomplete stream")
    return out


# ---- random valid streams ----

def random_code(rng: random.Random, alphabet: Sequence[int], n_codes: int, must: Sequence[int] = (), maxbits: int = 15,
                deep: bool = False, n_total: int = 0) -> List[int]:
    """lengths of n_total symbols: a random complete code over n_codes of `alphabet` (the `must` symbols among them)"""
    lens = [0] * n_total
    chosen = list(must) + rng.sample([s for s in alphabet if s not in must], n_codes - len(must))
    rng.shuffle(chosen)
    if n_codes == 1:
        lens[chosen[0]] = 1
        return lens
    for s, L in zip(chosen, random_lengths(rng, n_codes, maxbits, deep)):
        lens[s] = L
    return lens


def random_tokens(rng: random.Random, text: bytearray, budget: int, llens: Sequence[int], dlens: Sequence[int],
                  n_max: int) -> List[Token]:
    """up to n_max random tokens the codes can write, with at most `budget` bytes of text; appended to text"""
    lits = [s for s in range(256) if llens[s]]
    lsyms = [s for s in range(257, 286) if s < len(llens) and llens[s]]
    dsyms = [s for s in range(30) if s < len(dlens) and dlens[s]]
    out: List[Token] = []
    for _ in range(n_max):
        if budget <= 0:
            break
        produced = len(text)
        ok_d = [d for d in dsyms if DBASE[d] <= min(produced, 32768)]
        ok_l = [s for s in lsyms if LBASE[s - 257] <= budget]
        if ok_d and ok_l and (not lits or rng.random() < 0.5):
            lsym = rng.choice(ok_l)
            lx = 0 if lsym == 285 else rng.randrange(min(1 << LEXT[lsym - 257], budget - LBASE[lsym - 257] + 1))
            d = rng.choice(ok_d)
            dx = rng.randrange(min(1 << DEXT[d], min(produced, 32768) - DBASE[d] + 1))
            t = (lsym, lx, d, dx)
        elif lits:
            t = rng.choice(lits)
        else:
            break
        before = len(text)
        apply([t], text)
        budget -= len(text) - before
        out.append(t)
    return out


def random_member_payload(rng: random.Random, max_text: int = MAX_TEXT) -> Tuple[bytes, bytes]:
    """(payload, text): a random sequence of stored, fixed, dynamic and empty blocks with at most max_text of text"""
    w = BitWriter()
    text = bytearray()
    n_blocks = rng.choice([1, 1, 2, 3, 5, 8])
    target = rng.choice([rng.randrange(0, 200), rng.randrange(0, 5000), rng.randrange(0, max_text + 1)])
    for k in range(n_blocks):
        final = k == n_blocks - 1
        budget = min(max_text - len(text), max(0, (target - len(text)) // max(1, n_blocks - k - 1) if not final
                                                 else target - len(text)))
        kind = rng.choice(["stored", "fixed", "dynamic", "dynamic", "empty"])
        if kind == "empty":
            kind2 = rng.choice(["stored", "fixed", "dynamic"])
            if kind2 == "stored":
                stored(w, b"", final)
            elif kind2 == "fixed":
                fixed(w, [], final)
            else:
                llens = random_code(rng, range(257), rng.choice([1, 2, 3]), must=[256], n_total=257)
                dlens = [0] if rng.random() < 0.5 else [1]
                dynamic(w, [], final, llens, dlens)
        elif kind == "stored":
            n = min(budget, 65535, rng.choice([0, rng.randrange(0, 300), rng.randrange(0, 65536)]))
            data = bytes(rng.getrandbits(8) for _ in range(min(n, 64))) * (n // 64 + 1)
            data = data[:n]
            stored(w, data, final)
            text += data
        elif kind == "fixed":
            toks = random_tokens(rng, text, budget, FIXED_L[:286], FIXED_D, rng.randrange(0, 3000))
            fixed(w, toks, final)
        else:
            hlit = rng.choice([257, 286, rng.randrange(257, 287)])
            hdist = rng.choice([1, 30, rng.randrange(1, 31)])
            n_l = rng.randrange(2, hlit + 1) if rng.random() < 0.9 else 1
            llens = random_code(rng, range(hlit), n_l, must=[256] + ([rng.randrange(256)] if n_l > 1 else []),
                                deep=rng.random() < 0.3, n_total=hlit)
            n_d = rng.choice([0, 1, rng.randrange(1, hdist + 1)]) if hdist > 1 else rng.choice([0, 1])
            dlens = random_code(rng, range(hdist), n_d, deep=rng.random() < 0.3, n_total=hdist) if n_d else [0] * hdist
            toks = random_tokens(rng, text, budget, llens, dlens, rng.randrange(0, 4000))
            dynamic(w, toks, final, llens, dlens)
    return w.getvalue(), bytes(text)


# ---- the conformance corpus: named streams, each (name, payload, text) ----

def _lits(rng: random.Random, n: int, alphabet: Sequence[int]) -> List[int]:
    return [rng.choice(alphabet) for _ in range(n)]


def _code_length_cases() -> list:
    """codes of every length 1..15: a 16-code chain (lengths 1, 2, ..., 15, 15) rotated over 16 literal/length symbols
    and 16 distance symbols, so that each symbol is sent at each length -- the lookup-table widths and one past them
    among them; then blocks whose most frequent symbols carry the 15-bit codes (the canonical walk decodes them)"""
    out = []
    chain = random_lengths(random.Random(0), 16, deep=True)
    assert chain == list(range(1, 16)) + [15]
    for r in range(16):
        rng = random.Random(100 + r)
        syms = [ord(c) for c in "ACGT|0\t\n"] + [256, 257, 258, 265, 270, 277, 284, 285]
        llens = [0] * 286
        for k, s in enumerate(syms):
            llens[s] = chain[(k + r) % 16]
        dlens = [0] * 30
        for d in range(16):
            dlens[d] = chain[(d + 3 * r) % 16]
        text = bytearray()
        toks: List[Token] = []
        lit = [s for s in syms if s < 256]
        for _ in range(3):  # every symbol, whatever its length, several times
            t = _lits(rng, 300, lit)
            apply(t, text)
            toks += t
            for ls in syms[9:]:
                for d in range(16):
                    lx = rng.randrange(1 << LEXT[ls - 257]) if ls < 285 else 0
                    m = (ls, lx, d, rng.randrange(1 << DEXT[d]))
                    apply([m], text)
                    toks.append(m)
        w = BitWriter()
        dynamic(w, toks, True, llens, dlens)
        out.append(("code-lengths-rot%d" % r, w.getvalue(), bytes(text)))
    # the most frequent symbols carry the longest codes
    rng = random.Random(7)
    llens = [0] * 286
    chain = list(range(1, 15)) + [15] * 2
    syms = [256, 257, 258, 259, 260, 261, 262, 263, 264, 265, 266, 267, 268, 269, 0x41, 0x42]
    for s, L in zip(syms, chain):
        llens[s] = L
    dlens = [0] * 30
    for d, L in zip(range(16), chain):
        dlens[d] = L
    dlens[15], dlens[0] = dlens[0], dlens[15]  # distance 1: a 15-bit code
    text = bytearray()
    toks = _lits(rng, 20000, [0x41, 0x42])
    apply(toks, text)
    w = BitWriter()
    dynamic(w, toks, True, llens, dlens)
    out.append(("code-lengths-15-bit-literals", w.getvalue(), bytes(text)))
    toks2 = _lits(rng, 40, [0x41, 0x42]) + [(259, 0, 0, 0)] * 3000  # every match: 15-bit length and distance codes
    text = bytearray()
    apply(toks2, text)
    w = BitWriter()
    llens[259], llens[0x41] = llens[0x41], llens[259]
    dynamic(w, toks2, True, llens, dlens)
    out.append(("code-lengths-15-bit-matches", w.getvalue(), bytes(text)))
    return out


def _precode_cases() -> list:
    out = []
    rng = random.Random(11)
    for hlit in (257, 286):
        for hdist in (1, 30):
            for pc_kind in ("hclen19-deep", "hclen5"):
                text = bytearray()
                if pc_kind == "hclen5":  # code-length symbols 16, 17, 18, 0, 8 only: 256 codes of 8 bits
                    llens = [0] * hlit
                    for s in range(255):
                        llens[s] = 8
                    llens[256] = 8
                    dlens = [0] * hdist
                    lit = list(range(255))
                    toks = _lits(rng, 3000, lit)
                    precode = [0] * 19
                    precode[16], precode[17], precode[18], precode[0], precode[8] = 2, 3, 3, 2, 2
                    runs = rle(list(llens) + list(dlens))
                    w = BitWriter()
                    apply(toks, text)
                    dynamic(w, toks, True, llens, dlens, runs=runs, precode=precode, hclen=5)
                else:  # all 19 precode lengths sent, up to 7 bits
                    llens = random_code(rng, range(hlit), min(hlit, 60), must=[256, 65], n_total=hlit)
                    dlens = random_code(rng, range(hdist), hdist, n_total=hdist) if hdist > 1 else [1]
                    precode = [0] * 19
                    for s, L in zip(rng.sample(range(19), 19), random_lengths(rng, 19, 7)):
                        precode[s] = L
                    assert max(precode) == 7
                    toks = random_tokens(rng, text, 20000, llens, dlens, 4000)
                    w = BitWriter()
                    dynamic(w, toks, True, llens, dlens, precode=precode, hclen=19)
                out.append(("precode-%s-hlit%d-hdist%d" % (pc_kind, hlit, hdist), w.getvalue(), bytes(text)))
    # runs that cross from the literal/length lengths into the distance lengths
    letters = list(range(97, 123))
    for kind in ("zeros-18", "zeros-17", "repeat-16", "16-first-distance"):
        rngk = random.Random(len(kind))
        if kind == "zeros-18":  # 10 unused length symbols + 5 unused distance symbols: one run of 18
            llens = random_code(rngk, letters + list(range(256, 276)), 40, must=[256, 97], n_total=286)
            dlens = [0] * 5 + random_code(rngk, range(25), 20, n_total=25)
        elif kind == "zeros-17":  # 2 + 2 unused: one run of 17
            llens = random_code(rngk, letters + list(range(256, 284)), 40, must=[256, 97, 283], n_total=286)
            dlens = [0, 0] + random_code(rngk, range(28), 20, must=[0], n_total=28)
        else:  # 32 codes of 5 bits; the distance code starts with the same length: 16 repeats it across
            llens = [0] * 286
            for s in letters + [256] + list(range(281, 286)):
                llens[s] = 5
            dlens = [5] * 28 + [4, 4]
        runs = rle(llens + dlens) if kind != "16-first-distance" else rle(llens) + [(16, 0)] + rle(dlens[3:])
        assert run_lengths(runs) == llens + dlens
        text = bytearray()
        toks = random_tokens(rngk, text, 30000, llens, dlens, 5000)
        w = BitWriter()
        dynamic(w, toks, True, llens, dlens, runs=runs)
        out.append(("runs-across-boundary-%s" % kind, w.getvalue(), bytes(text)))
    return out


def _one_block(tokens: Sequence[Token], llens: Sequence[int], dlens: Sequence[int], prefix: bytes = b"") -> Tuple[bytes, bytes]:
    """(payload, text): `prefix` as a stored block (the history later matches reach into), then one dynamic block"""
    w = BitWriter()
    text = bytearray(prefix)
    if prefix:
        for i in range(0, len(prefix), 65535):
            stored(w, prefix[i:i + 65535], False)
    apply(tokens, text)
    dynamic(w, tokens, True, llens, dlens)
    return w.getvalue(), bytes(text)


def _degenerate_cases() -> list:
    out = []
    rng = random.Random(5)
    lit = list(range(97, 105))
    llens = [0] * 286
    for s in lit + [256, 257, 258, 259, 260, 261, 262, 263]:
        llens[s] = 4
    for d in (0, 3, 29):  # a single distance code of one bit, as symbol 0, 3 or 29 (HDIST 1, 4 or 30)
        dlens = [0] * (d + 1)
        dlens[d] = 1
        toks = _lits(rng, 40000 if d == 29 else 50, lit)
        for k in range(200):
            toks.append((257 + rng.randrange(7), 0, d, rng.randrange(1 << DEXT[d])))
        out.append(("single-distance-code-%d" % d,) + _one_block(toks, llens, dlens))
    lonly = [8] * 257  # 255 codes of 8 bits, 2 of 9: complete
    lonly[0], lonly[1] = 9, 9
    for hdist in (1, 30):  # a literal-only block without any distance code
        toks = _lits(rng, 5000, list(range(256)))
        out.append(("no-distance-codes-hdist%d" % hdist,) + _one_block(toks, lonly, [0] * hdist))
    eob = [0] * 257
    eob[256] = 1
    for hdist, dl in ((1, [0]), (1, [1]), (30, [0] * 30)):  # an end-of-block-only block with a 1-bit code
        w = BitWriter()
        dynamic(w, [], False, eob, dl)
        fixed(w, [97, 98, 99], True)
        out.append(("end-of-block-only-1-bit-hdist%d-%s" % (hdist, dl[0]), w.getvalue(), b"abc"))
    return out


def _length_distance_cases() -> list:
    out = []
    rng = random.Random(9)
    # every length symbol with every extra-bits value, 258 written both ways (285, and 284 with extra bits 31)
    toks: List[Token] = [97, 98, 99, 100]
    for ls in range(257, 286):
        for lx in range(1 << LEXT[ls - 257]) if ls < 285 else [0]:
            toks.append((ls, lx, rng.randrange(4), 0))
            toks.append(rng.randrange(256))
    toks += [(284, 31, 0, 0), (285, 0, 1, 0), (284, 31, 2, 0)]
    w, text = BitWriter(), bytearray()
    apply(toks, text)
    fixed(w, toks, True)
    out.append(("every-length-fixed", w.getvalue(), bytes(text)))
    llens = [0] * 286
    for s, L in zip(list(range(256)) + list(range(256, 286)), [8] * 226 + [9] * 60):
        llens[s] = L
    assert sum(1 << (15 - x) for x in llens if x) == 1 << 15
    out.append(("every-length-dynamic",) + _one_block(toks, llens, [2, 2, 2, 2]))
    # every distance symbol, with its smallest, largest and a random extra-bits value; 32,768 among them
    hist = bytes(rng.randrange(256) for _ in range(32768))
    toks = []
    for d in range(30):
        for dx in sorted({0, (1 << DEXT[d]) - 1, rng.randrange(1 << DEXT[d])}):
            toks.append((257 + rng.randrange(28), 0, d, dx))
    toks.append((285, 0, 29, 8191))  # 32,768
    out.append(("every-distance-fixed-history",) + _fixed_after(hist, toks))
    dl = [4, 4] + [5] * 28
    assert sum(1 << (15 - x) for x in dl) == 1 << 15
    out.append(("every-distance-dynamic",) + _one_block(toks, llens, dl, prefix=hist))
    # overlapping matches at every distance 1..40, at lengths around the warp's 32-byte steps
    toks = [rng.randrange(256) for _ in range(40)]
    for dist in range(1, 41):
        for length in (3, 31, 32, 33, 63, 64, 65, 95, 97, 129, 200, 257, 258):
            if length > dist:
                toks.append(match(length, dist))
                toks.append(rng.randrange(256))
    w, text = BitWriter(), bytearray()
    apply(toks, text)
    fixed(w, toks, True)
    out.append(("overlapping-matches", w.getvalue(), bytes(text)))
    # length-3 matches from beyond the 16 KiB ring (and from just inside it)
    hist = bytes(rng.randrange(256) for _ in range(34000))
    toks = []
    for k in range(600):
        dist = rng.choice([16383, 16384, 16385, 16126, 16127, 20000, rng.randrange(16000, 32769), 32768])
        toks.append(match(rng.choice([3, 3, 4, 5]), dist))
    out.append(("far-length-3-matches",) + _fixed_after(hist, toks))
    return out


def _fixed_after(hist: bytes, toks: Sequence[Token]) -> Tuple[bytes, bytes]:
    """stored blocks holding `hist`, then one fixed block of `toks`"""
    w = BitWriter()
    for i in range(0, len(hist), 65535):
        stored(w, hist[i:i + 65535], False)
    text = bytearray(hist)
    apply(toks, text)
    fixed(w, toks, True)
    return w.getvalue(), bytes(text)


def _multi_block_cases() -> list:
    out = []
    for seed in range(6):
        rng = random.Random(300 + seed)
        w, text = BitWriter(), bytearray()
        kinds = ["stored", "fixed", "dynamic", "empty-stored", "empty-fixed", "empty-dynamic", "dynamic", "stored"] * 2
        rng.shuffle(kinds)
        kinds = ["dynamic", "stored"] + kinds  # a stored block right after a dynamic block that ended mid-byte
        for k, kind in enumerate(kinds):
            final = k == len(kinds) - 1
            budget = min(3000, MAX_TEXT - len(text))
            if kind == "stored":
                data = bytes(rng.choice(b"ACGT\t\n") for _ in range(rng.randrange(1, 1500)))[:budget]
                stored(w, data, final)
                text += data
            elif kind == "fixed":
                fixed(w, random_tokens(rng, text, budget, FIXED_L[:286], FIXED_D, 800), final)
            elif kind == "dynamic":
                hlit, hdist = rng.randrange(257, 287), rng.randrange(1, 31)
                llens = random_code(rng, range(hlit), rng.randrange(3, hlit), must=sorted({256, 65, hlit - 1}), n_total=hlit)
                dlens = random_code(rng, range(hdist), rng.randrange(1, hdist + 1), n_total=hdist)
                dynamic(w, random_tokens(rng, text, budget, llens, dlens, 800), final, llens, dlens)
            elif kind == "empty-stored":
                stored(w, b"", final)
            elif kind == "empty-fixed":
                fixed(w, [], final)
            else:
                llens = random_code(rng, range(257), 3, must=[256], n_total=257)
                dynamic(w, [], final, llens, [0])
        out.append(("multi-block-%d" % seed, w.getvalue(), bytes(text)))
    return out


def text_of_length(n: int, seed: int = 0) -> Tuple[bytes, bytes]:
    """(payload, text) of exactly n text bytes: VCF-like text in a random dynamic code, matches of every kind"""
    rng = random.Random(seed * 100003 + n)
    llens = random_code(rng, range(286), 120, must=[256] + list(b"0|1\t\n.") + [257, 285], n_total=286)
    dlens = random_code(rng, range(30), 30, n_total=30)
    text = bytearray()
    toks = random_tokens(rng, text, n, llens, dlens, 1 << 30)
    lits = [s for s in range(256) if llens[s]]
    while len(text) < n:  # (the budget can end on a length no match fits)
        t = rng.choice(lits)
        toks.append(t)
        text.append(t)
    w = BitWriter()
    dynamic(w, toks, True, llens, dlens)
    return w.getvalue(), bytes(text)


TEXT_LENGTHS = (list(range(0, 131)) + [255, 256, 257, 1023, 1024, 1025, 4095, 4096, 4097, 8191, 8192, 8193, 8192 + 258,
                                       12288, 16384, 32768, 65535, 65536])


def valid_cases() -> list:
    """(name, payload, text) of every hand-made valid stream"""
    return (_code_length_cases() + _precode_cases() + _degenerate_cases() + _length_distance_cases() +
            _multi_block_cases())


def invalid_cases() -> list:
    """(name, payload, text) of streams zlib refuses; text is what a decoder that missed the error would produce (the
    trailer is made from it, so that only the stream itself can fail)"""
    out = []
    abc = [97, 98, 99, 100]

    def blk(fn, text=b"abcd"):
        w = BitWriter()
        fn(w)
        out.append((fn.__name__, w.getvalue(), text))

    def btype_3(w):
        w.bits(1, 1)
        w.bits(3, 2)
        w.bits(0, 16)

    def stored_nlen_mismatch(w):
        stored(w, b"abcd", True, nlen=(4 ^ 0xFFFF) ^ 0x100)

    l5 = [0] * 286
    for s in list(range(97, 123)) + [256] + list(range(281, 286)):
        l5[s] = 5
    d5 = [5] * 28 + [4, 4]

    def hlit_287(w):
        dynamic(w, abc, True, l5 + [0], d5)

    def hlit_288(w):
        dynamic(w, abc, True, l5 + [0, 0], d5)

    def hdist_31(w):
        dynamic(w, abc, True, l5, d5 + [0])

    def hdist_32(w):
        dynamic(w, abc, True, l5, d5 + [0, 0])

    def precode_oversubscribed(w):
        pre = [0] * 19
        pre[5], pre[16], pre[0], pre[17], pre[18], pre[4] = 1, 1, 1, 2, 3, 3
        dynamic(w, abc, True, l5, d5, precode=pre, runs=rle(l5 + d5))

    def precode_incomplete(w):
        pre = [0] * 19
        pre[5], pre[16], pre[0], pre[17], pre[18], pre[4] = 2, 2, 3, 3, 3, 4
        dynamic(w, abc, True, l5, d5, precode=pre, runs=rle(l5 + d5))

    def symbol_16_first(w):
        dynamic(w, abc, True, l5, d5, runs=[(16, 0)] + rle(l5 + d5)[:-1])

    def repeat_past_the_end(w):
        runs = rle(l5 + d5)
        dynamic(w, abc, True, l5, d5, runs=runs[:-1] + [(16, 0)])

    def no_end_of_block_length(w):
        ll = list(l5)
        ll[256], ll[255] = 0, 5
        dynamic(w, abc, True, ll, d5, eob=False)
        w.bits(0, 20)

    def literal_code_oversubscribed(w):
        ll = list(l5)
        ll[98] = 4
        dynamic(w, abc, True, ll, d5)

    def literal_code_incomplete(w):
        ll = list(l5)
        ll[122] = 0
        dynamic(w, abc, True, ll, d5)

    def single_literal_code_of_2_bits(w):  # end-of-block only, as a 2-bit code
        ll = [0] * 257
        ll[256] = 2
        dynamic(w, [], False, ll, [0])
        fixed(w, abc, True)

    def single_literal_code_of_3_bits(w):
        ll = [0] * 257
        ll[256] = 3
        dynamic(w, [], False, ll, [1])
        fixed(w, abc, True)

    def single_distance_code_of_2_bits(w):
        dynamic(w, abc + [(281, 0, 0, 0)], True, l5, [2])

    def single_distance_code_of_5_bits(w):
        dl = [0] * 30
        dl[2] = 5
        dynamic(w, abc + [(281, 0, 2, 0)], True, l5, dl)

    def fixed_literal_286(w):
        fixed(w, abc + [286], True)

    def fixed_literal_287(w):
        fixed(w, abc + [287], True)

    def fixed_distance_30(w):
        w.bits(1, 1)
        w.bits(1, 2)
        write_tokens(w, abc + [(258, 0, 30, 0)], FIXED_L, FIXED_D + [5, 5])

    def fixed_distance_31(w):
        w.bits(1, 1)
        w.bits(1, 2)
        write_tokens(w, abc + [(258, 0, 31, 0)], FIXED_L, FIXED_D + [5, 5])

    def distance_before_the_start(w):
        fixed(w, abc + [(257, 0, 4, 0)], True)  # distance 5 after 4 bytes

    def missing_end_of_block(w):
        fixed(w, abc, True, eob=False)

    def bfinal_never_set(w):
        fixed(w, abc[:2], False)
        stored(w, b"cd", False)

    for fn in (btype_3, stored_nlen_mismatch, hlit_287, hlit_288, hdist_31, hdist_32, precode_oversubscribed,
               precode_incomplete, symbol_16_first, repeat_past_the_end, no_end_of_block_length,
               literal_code_oversubscribed, literal_code_incomplete, single_literal_code_of_2_bits,
               single_literal_code_of_3_bits, single_distance_code_of_2_bits, single_distance_code_of_5_bits,
               fixed_literal_286, fixed_literal_287, fixed_distance_30, fixed_distance_31, distance_before_the_start,
               missing_end_of_block, bfinal_never_set):
        text = bytearray(b"abcd")
        if fn is single_distance_code_of_2_bits:
            apply([(281, 0, 0, 0)], text)
        elif fn is single_distance_code_of_5_bits:
            apply([(281, 0, 2, 0)], text)
        blk(fn, bytes(text))
    return out


SINGLE_CODE_CASES = {"single_literal_code_of_2_bits", "single_literal_code_of_3_bits", "single_distance_code_of_2_bits",
                     "single_distance_code_of_5_bits"}


def deflate_text(text: bytes, rng: random.Random) -> bytes:
    """text (at most MAX_TEXT bytes) as one dynamic block: greedy matches of 4 bytes and more, then random complete
    codes of up to 15 bits over the symbols used -- often the 15-bit ones on frequent symbols"""
    toks: List[Token] = []
    last = {}
    i, n = 0, len(text)
    while i < n:
        key = text[i:i + 4]
        j = last.get(key, -1)
        last[key] = i
        if j >= 0 and i - j <= 32768 and len(key) == 4:
            L = 4
            while L < 258 and i + L < n and text[j + L] == text[i + L]:
                L += 1
            toks.append(match(L, i - j))
            for k in range(i + 1, min(i + L, n - 3), 3):
                last[text[k:k + 4]] = k
            i += L
        else:
            toks.append(text[i])
            i += 1
    lsyms = sorted({t if isinstance(t, int) else t[0] for t in toks} | {256})
    dsyms = sorted({t[2] for t in toks if not isinstance(t, int)})
    if len(lsyms) < 2:
        lsyms.append(0 if lsyms[0] != 0 else 1)
    llens, dlens = [0] * 286, [0] * 30
    for s, L in zip(rng.sample(lsyms, len(lsyms)), random_lengths(rng, len(lsyms), deep=rng.random() < 0.3)):
        llens[s] = L
    if len(dsyms) == 1:
        dlens[dsyms[0]] = 1
    elif dsyms:
        for s, L in zip(rng.sample(dsyms, len(dsyms)), random_lengths(rng, len(dsyms), deep=rng.random() < 0.3)):
            dlens[s] = L
    w = BitWriter()
    dynamic(w, toks, True, llens, dlens)
    return w.getvalue()


def bgzf_file(text: bytes, rng: random.Random, block_text: int = 60000) -> bytes:
    """text as bgzf members made by deflate_text (drawn again while a member would exceed 64 KiB), then the EOF block"""
    out = []
    for i in range(0, len(text), block_text):
        piece = text[i:i + block_text]
        payload = deflate_text(piece, rng)
        while len(payload) + 26 > 65536:
            payload = deflate_text(piece, rng)
        out.append(member(payload, piece))
    return b"".join(out) + EOF_BLOCK
