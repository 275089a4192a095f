"""Deflate stream forge: writes raw Deflate (RFC 1951) streams block by block, including streams zlib never writes and streams
that are malformed on purpose.  Bit order is BitByteData's LsbBitWriter (helpers.LsbBitWriter).

A stream is a list of blocks (`Stored`, `Fixed`, `Dynamic`); Huffman blocks carry a list of symbols:

    int 0..255              literal
    ("m", length, dist)     match, written with the RFC 1951 length / distance codes
    ("L", sym, extra, n)    raw lit/len symbol `sym` followed by `n` extra bits of value `extra` (286/287, 284 + 31, ...)
    ("D", sym, extra, n)    raw distance symbol (30/31, ...), same form
    ("bits", value, n)      `n` raw bits (a code that has no length assigned, junk)

`forge(blocks)` returns (stream, expected) where `expected` is what a decoder that follows RFC 1951 produces, computed while
the stream is written, or None when the blocks contain something the writer cannot decode by construction (raw bits, raw
symbols outside the alphabets, a code shadowed by a shorter one, a distance past the output).  `corpus()` builds the families the
tests run: each unit declares the status the reference returns for it (read off Sources/Deflate/Deflate.swift), "error"
for inputs cut short at a byte boundary, or None where only the oracle can say (cuts at a bit boundary, whose zero-filled
last byte may still decode)."""
import random
from fractions import Fraction

from helpers import LsbBitWriter

LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
             6145, 8193, 12289, 16385, 24577]
DIST_EXTRA = [0] * 4 + [k for k in range(1, 14) for _ in range(2)]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_DIST = [5] * 32

# include/swc_status.h
OK, TRAP, WRONG_LENGTHS, WRONG_BLOCK_TYPE, WRONG_SYMBOL, SYMBOL_NOT_FOUND = 0, 2, 101, 102, 103, 104


def len_code(length):
    for s in range(28, -1, -1):
        if length >= LEN_BASE[s]:
            return 257 + s, length - LEN_BASE[s], LEN_EXTRA[s]
    raise ValueError(length)


def dist_code(dist):
    for s in range(29, -1, -1):
        if dist >= DIST_BASE[s]:
            return s, dist - DIST_BASE[s], DIST_EXTRA[s]
    raise ValueError(dist)


def kraft(lengths):
    return sum((Fraction(1, 1 << l) for l in lengths if l), Fraction(0))


def canonical(lengths):
    """Canonical code of a length vector, assigned like Code.huffmanCodes (sorted by (length, symbol), a counter shifted left
    at every new length; bits above the length are dropped, so an over-subscribed set reuses codes).
    -> ({symbol: (code, length)} with the code MSB first, Kraft sum)"""
    codes, counter, loop_bits = {}, -1, -1
    for length, sym in sorted((l, s) for s, l in enumerate(lengths) if l):
        counter += 1
        if length != loop_bits:
            counter <<= length - loop_bits
            loop_bits = length
        codes[sym] = (counter & ((1 << length) - 1), length)
    return codes, kraft(lengths)


def decodes_as(lengths):
    """What the reference's decoding tree (DecodingTree.swift:15-50) returns for each symbol's code.  Codes go into the tree
    in canonical order, a later code that lands on the same slot replaces the earlier one, and decoding stops at the first
    leaf on the path.  -> {symbol: the symbol read back from its code with the same number of bits (itself unless the set
    is over-subscribed), or None when a shorter code is a prefix of it}"""
    codes, _ = canonical(lengths)
    slot = {}
    for sym, (code, length) in sorted(codes.items(), key=lambda kv: (kv[1][1], kv[0])):
        slot[(length, code)] = sym
    out = {}
    for sym, (code, length) in codes.items():
        for k in range(1, length + 1):
            owner = slot.get((k, code >> (length - k)))
            if owner is not None:
                out[sym] = owner if k == length else None
                break
    return out


def rev(code, n):
    return int(format(code, f"0{n}b")[::-1], 2) if n else 0


class Stored:
    def __init__(self, data, final=False, nlen=None, pad=0):
        self.data, self.final, self.nlen, self.pad = bytes(data), final, nlen, pad


class Fixed:
    def __init__(self, symbols, final=False, eob=True):
        self.symbols, self.final, self.eob = symbols, final, eob


class Dynamic:
    """lit_lengths / dist_lengths: the code-length vectors (their sizes give HLIT / HDIST unless `hlit` / `hdist` set the
    5-bit fields directly).  cl_lengths: the 19 code-length-code lengths by symbol (default: a complete code over the symbols
    the run-length pass uses).  cl_ops: explicit [(symbol, extra)] run-length program replacing the default one, which codes
    the concatenated vector with 16/17/18 (a 16 may cross from the lit/len into the distance lengths).  hclen: the 4-bit field."""

    def __init__(self, symbols, lit_lengths, dist_lengths, final=False, eob=True, hlit=None, hdist=None, hclen=None,
                 cl_lengths=None, cl_ops=None, rle=True):
        self.symbols, self.final, self.eob = symbols, final, eob
        self.lit, self.dist = list(lit_lengths), list(dist_lengths)
        self.hlit, self.hdist, self.hclen, self.cl_lengths, self.cl_ops, self.rle = hlit, hdist, hclen, cl_lengths, cl_ops, rle


def rle_ops(lengths, use_repeats=True):
    ops, i, n = [], 0, len(lengths)
    while i < n:
        v, j = lengths[i], i
        while j < n and lengths[j] == v:
            j += 1
        run = j - i
        if not use_repeats:
            ops += [(v, 0)] * run
        elif v == 0:
            while run >= 11:
                k = min(run, 138); ops.append((18, k - 11)); run -= k
            if run >= 3:
                ops.append((17, run - 3)); run = 0
            ops += [(0, 0)] * run
        else:
            ops.append((v, 0)); run -= 1
            while run >= 3:
                k = min(run, 6); ops.append((16, k - 3)); run -= k
            ops += [(v, 0)] * run
        i = j
    return ops


def complete_lengths(used, nsyms, maxlen=15):
    """a complete code (Kraft sum 1) over the symbols in `used` (at least two: a lone symbol gets a partner)"""
    used = sorted(set(used))
    if len(used) == 1:
        used.append(next(s for s in range(nsyms) if s not in used))
    k = len(used)
    n = (k - 1).bit_length()
    short = (1 << n) - k                       # symbols one bit shorter
    assert n <= maxlen
    lengths = [0] * nsyms
    for i, s in enumerate(used):
        lengths[s] = n - 1 if i < short else n
    return lengths


_EXTRA_OF_CL = {16: 2, 17: 3, 18: 7}


class _Out:
    """expected output, tracked while the stream is written; `ok` drops to False on anything not decodable by construction.
    `ended`: the final block's end-of-block symbol has been read (what follows is trailing input).  `max_run`: the longest
    run of literal bytes (Huffman literals and stored bytes) that ends in a match."""

    def __init__(self):
        self.buf, self.ok, self.ended = bytearray(), True, False
        self.run = self.max_run = 0

    def literals(self, data):
        if not self.ended:
            self.buf += data
            self.run += len(data)

    def match(self, length, dist):
        if self.ended:
            return
        if not (3 <= length <= 258) or not (1 <= dist <= len(self.buf)):
            self.ok = False
            return
        s = len(self.buf) - dist
        for i in range(length):
            self.buf.append(self.buf[s + i])
        self.max_run = max(self.max_run, self.run)
        self.run = 0


_FIXED = None


def _fixed_tables():
    global _FIXED
    if _FIXED is None:
        _FIXED = (canonical(FIXED_LIT)[0], canonical(FIXED_DIST)[0], decodes_as(FIXED_LIT), decodes_as(FIXED_DIST))
    return _FIXED


def _write_symbols(w, out, symbols, lit_codes, dist_codes, lit_map, dist_map, eob, final):
    """writes each symbol with its own code; the expected output follows what the decoder reads back (`lit_map`, `dist_map`:
    decodes_as of the two sets), so a code another symbol took over in an over-subscribed set is decoded as that symbol"""
    def put(codes, sym):
        c = codes.get(sym)
        if c is None:
            raise ValueError(f"symbol {sym} has no code")
        w.write_number(rev(*c), c[1])

    pending_len = None

    def litlen(sym, extra, n, closing=False):
        nonlocal pending_len
        put(lit_codes, sym); w.write_number(extra, n)
        if out.ended:
            return
        d = lit_map.get(sym)
        if d is None or pending_len is not None or (d != sym and n):
            out.ok = False
        elif d < 256:
            out.literals(bytes([d]))
        elif d == 256:
            if final:
                out.ended = True
            elif not closing:
                out.ok = False                 # a block that ends early: the rest of it would be read as the next block
        elif d <= 285 and n == LEN_EXTRA[d - 257] and extra < (1 << n):
            pending_len = LEN_BASE[d - 257] + extra
        else:
            out.ok = False

    def distance(sym, extra, n):
        nonlocal pending_len
        put(dist_codes, sym); w.write_number(extra, n)
        if out.ended:
            return
        d = dist_map.get(sym)
        if pending_len is not None and d is not None and d <= 29 and n == DIST_EXTRA[d] and extra < (1 << n):
            out.match(pending_len, DIST_BASE[d] + extra)
        else:
            out.ok = False
        pending_len = None

    for s in symbols:
        if isinstance(s, int):
            litlen(s, 0, 0)
        elif s[0] == "m":
            _, length, dist = s
            litlen(*len_code(length))
            distance(*dist_code(dist))
        elif s[0] == "L":
            litlen(*s[1:])
        elif s[0] == "D":
            distance(*s[1:])
        elif s[0] == "bits":
            w.write_number(s[1], s[2])
            if not out.ended:
                out.ok = False
        else:
            raise ValueError(s)
    if eob:
        litlen(256, 0, 0, closing=True)
    if pending_len is not None:
        out.ok = False


def _write_dynamic(w, b, out):
    """-> the largest Kraft sum of the block's three code sets"""
    lit_codes, kl = canonical(b.lit)
    dist_codes, kd = canonical(b.dist)
    ops = b.cl_ops if b.cl_ops is not None else rle_ops(b.lit + b.dist, b.rle)
    cl = list(b.cl_lengths) if b.cl_lengths is not None else complete_lengths([s for s, _ in ops], 19, 7)
    cl_codes, kc = canonical(cl)
    cl_map = decodes_as(cl)
    if any(cl_map.get(sym) != sym for sym, _ in ops):
        out.ok = False                         # a code-length code another one took over: the header reads differently
    hclen = b.hclen
    if hclen is None:
        hclen = max([4] + [i + 1 for i, s in enumerate(CL_ORDER) if cl[s]]) - 4
    w.write_number(len(b.lit) - 257 if b.hlit is None else b.hlit, 5)
    w.write_number(len(b.dist) - 1 if b.hdist is None else b.hdist, 5)
    w.write_number(hclen, 4)
    for i in range(hclen + 4):
        w.write_number(cl[CL_ORDER[i]], 3)
    for sym, extra in ops:
        c = cl_codes[sym]
        w.write_number(rev(*c), c[1])
        if sym in _EXTRA_OF_CL:
            w.write_number(extra, _EXTRA_OF_CL[sym])
    _write_symbols(w, out, b.symbols, lit_codes, dist_codes, decodes_as(b.lit), decodes_as(b.dist), b.eob, b.final)
    return max(kl, kd, kc)


def forge(blocks, writer=None, stats=None):
    """-> (stream bytes, expected output bytes or None).  `stats` (a dict) receives "kraft", the largest Kraft sum of any
    dynamic block's code sets (0 without one), and "max_run", the longest literal run that ends in a match."""
    w = writer or LsbBitWriter()
    out = _Out()
    k = Fraction(0)
    for b in blocks:
        w.write_number(1 if b.final else 0, 1)
        if isinstance(b, Stored):
            w.write_number(0, 2)
            w.align(fill=b.pad)
            n = len(b.data)
            w.write_number(n, 16)
            nlen = (~n & 0xFFFF) if b.nlen is None else b.nlen
            w.write_number(nlen, 16)
            if n & nlen:
                out.ok = False
            w.write_bytes(b.data)
            out.literals(b.data)
            out.ended = out.ended or b.final
        elif isinstance(b, Fixed):
            w.write_number(1, 2)
            _write_symbols(w, out, b.symbols, *_fixed_tables(), b.eob, b.final)
        else:
            w.write_number(2, 2)
            k = max(k, _write_dynamic(w, b, out))
    if stats is not None:
        stats.update(kraft=k, max_run=out.max_run)
    return w.data, (bytes(out.buf) if out.ok else None)


# ------------------------------------------------------------------------------------------------ symbol streams
def random_symbols(rng, lit_lengths, dist_lengths, n, out_len=0, match_p=0.3):
    """`n` random symbols that only use coded symbols: literals, and matches whose distance fits the output so far
    (`out_len` bytes precede the block)."""
    lits = [s for s in range(256) if lit_lengths[s]]
    lens = [s for s in range(257, min(len(lit_lengths), 286)) if lit_lengths[s]]
    dists = [s for s in range(min(len(dist_lengths), 30)) if dist_lengths[s]]
    syms, pos = [], out_len
    for _ in range(n):
        ok_d = [d for d in dists if DIST_BASE[d] <= pos]
        if lens and ok_d and rng.random() < match_p:
            ls, d = rng.choice(lens), rng.choice(ok_d)
            le = rng.randrange(1 << LEN_EXTRA[ls - 257])
            de = rng.randrange(min(1 << DIST_EXTRA[d], pos - DIST_BASE[d] + 1))
            syms += [("L", ls, le, LEN_EXTRA[ls - 257]), ("D", d, de, DIST_EXTRA[d])]
            pos += LEN_BASE[ls - 257] + le
        elif lits:
            syms.append(rng.choice(lits))
            pos += 1
    return syms


def lengths_by_count(counts, symbols, nsyms):
    """code lengths giving counts[L] symbols length L (counts indexed 1..15), taken in order from `symbols`"""
    out, it = [0] * nsyms, iter(symbols)
    for L in range(1, len(counts)):
        for _ in range(counts[L]):
            out[next(it)] = L
    return out


class Unit:
    """`stats`: forge()'s stats of the stream, where a test needs them; `lengths`: (lit/len, distance) code lengths of a
    single-dynamic-block stream"""

    def __init__(self, family, name, data, expect, status, zlib_ok=None, stats=None, lengths=None):
        self.family, self.name, self.data, self.expect, self.status = family, name, data, expect, status
        self.zlib_ok, self.stats, self.lengths = zlib_ok, stats, lengths

    @property
    def oversub(self):
        """a code set of the stream has a Kraft sum > 1, so the batch decoders hand it to inflate_slow_kernel"""
        return self.stats is not None and self.stats["kraft"] > 1

    def __repr__(self):
        return f"<{self.family}/{self.name} {len(self.data)} B>"


# every lit/len length 1..15 in use, complete: lengths 1..14 once and 15 twice (1/2 + ... + 1/2^14 + 2/2^15 = 1)
LONG_LIT_COUNTS = [0] + [1] * 14 + [2]
# every distance length 1..15 in use, complete
LONG_DIST_COUNTS = [0] + [1] * 14 + [2]


def _long_codes(units, rng):
    # 15-bit EOB and length symbols; every other length carries a mix of literals and length symbols
    for k in range(12):
        lit_syms = rng.sample(range(256), 12)
        len_syms = rng.sample(range(257, 286), 3)
        tail = [256, 284 if k % 2 else len_syms[0]]                 # the two 15-bit codes
        order = lit_syms + [s for s in len_syms if s not in tail] + [rng.randrange(256)]
        order = [s for s in dict.fromkeys(order) if s not in tail][:14] + tail
        lit = lengths_by_count(LONG_LIT_COUNTS, order, 286)
        if k % 4 == 3:                                                # a literal on a 15-bit code instead of the length symbol
            lit[tail[1]] = 0
            spare = next(s for s in range(256) if lit[s] == 0)
            lit[spare] = 15
        dsyms = rng.sample(range(30), 16)
        if k % 2:
            dsyms.remove(29) if 29 in dsyms else dsyms.pop()
            dsyms.append(29)                                          # distance 29 on a 15-bit code
        dist = lengths_by_count(LONG_DIST_COUNTS, dsyms, 30)
        head = random_symbols(rng, lit, [0] * 30, 40000 if k < 4 else 3000, 0, 0)
        body = random_symbols(rng, lit, dist, 3000, len(head), 0.4)
        data, exp = forge([Dynamic(head + body, lit, dist, final=True)])
        units.append(Unit("long_codes", f"k{k}", data, exp, OK, zlib_ok=True, lengths=(lit, dist)))


def _sym48(units, rng):
    # back-to-back matches of 15-bit 284 + 5 extra bits and 15-bit distance 29 + 13 extra bits: 48 bits per match
    for k in range(4):
        lit_syms = rng.sample(range(256), 13) + [257 + k]
        lit = lengths_by_count(LONG_LIT_COUNTS, lit_syms + [284, 256], 286)
        dist = lengths_by_count(LONG_DIST_COUNTS, rng.sample(range(29), 15) + [29], 30)
        head = random_symbols(rng, lit, [0] * 30, 33000, 0, 0)
        body = []
        for i in range(200 + 50 * k):
            body += [("L", 284, rng.randrange(32), 5), ("D", 29, rng.randrange(8192), 13)]
            if i % 37 == 36:
                body.append(lit_syms[i % 13])
        data, exp = forge([Dynamic(head + body, lit, dist, final=True)])
        units.append(Unit("sym48", f"k{k}", data, exp, OK, zlib_ok=True, lengths=(lit, dist)))


def _uniform(units, rng):
    # 254 literals on 8-bit codes: every bit offset decodes as some literal, so a lane started at a wrong offset never
    # resynchronises by luck
    for k in range(4):
        nine = rng.sample(range(256), 2)
        lit = [8] * 256 + [9] + [9] + [0] * 28
        for s in nine:
            lit[s] = 9
        syms = [rng.choice([s for s in range(256) if s not in nine]) for _ in range(6000 + 3000 * k)]
        data, exp = forge([Dynamic(syms, lit, [1], final=True)])
        units.append(Unit("uniform", f"k{k}", data, exp, OK, zlib_ok=True))


def _incomplete(units, rng):
    base = complete_lengths(range(258), 286)
    for k in range(4):
        # one distance code of length 1 (symbol k); matches use it
        dist = [0] * 30
        dist[k] = 1
        syms = random_symbols(rng, base, dist, 2000, 0, 0.3)
        data, exp = forge([Dynamic(syms, base, dist, final=True)])
        units.append(Unit("incomplete", f"one_dist_{k}", data, exp, OK, zlib_ok=True))
    # no distance codes at all, literal-only block (HDIST 1, its length 0)
    for k in range(2):
        syms = [rng.randrange(256) for _ in range(500 * (k + 1))]
        data, exp = forge([Dynamic(syms, base, [0] * (k + 1), final=True)])
        units.append(Unit("incomplete", f"no_dist_{k}", data, exp, OK, zlib_ok=True))
    # incomplete lit/len set (Kraft 1/2 + ...); the stream reaches a code no symbol owns
    lit = [0] * 286
    for s in range(64):
        lit[s] = 8                                        # Kraft 1/4
    lit[256] = 8
    codes, _ = canonical(lit)
    top = max(c for c, l in codes.values())               # every 8-bit code above `top` is unassigned
    for k in range(4):
        syms = [rng.randrange(64) for _ in range(100 + 200 * k)] + [("bits", rev(top + 1 + k, 8), 8)]
        data, _ = forge([Dynamic(syms, lit, [1], final=True)])
        units.append(Unit("incomplete", f"unassigned_{k}", data, None, SYMBOL_NOT_FOUND))
    # an unassigned distance code: one distance code of length 2, the stream sends another 2-bit pattern
    dist = [0] * 30
    dist[3] = 2
    syms = [rng.randrange(200) for _ in range(50)] + [("L", 257, 0, 0), ("bits", 0b11, 2)]
    data, _ = forge([Dynamic(syms, base, dist, final=True)])
    units.append(Unit("incomplete", "unassigned_dist", data, None, SYMBOL_NOT_FOUND))


def _oversub(units, rng):
    """Over-subscribed sets (Kraft sum > 1), which the reference accepts: later codes overwrite heap slots and shorter codes
    shadow longer ones.  The streams use the codes that survive; in the 'collide' units two codes another symbol took over
    are used as well (a literal read back as length symbol 257, and one read back as end of block), so every unit decodes
    to bytes the forge knows."""
    for k in range(24):
        kind = ("lit", "dist", "cl", "collide")[k % 4]
        lit = [0] * 286
        for s in range(256, 266):                               # end of block and nine length symbols on 7-bit codes
            lit[s] = 7
        order = rng.sample(range(256), 256)
        for s in order[:236]:                                   # 236 literals on 8-bit codes: complete
            lit[s] = 8
        dist = complete_lengths(range(30), 30)
        cl = None
        if kind == "lit":
            for s in order[236:237 + k % 20]:                   # more 8-bit literals: their codes wrap onto the 7-bit ones
                lit[s] = 8
        elif kind == "dist":
            for s in rng.sample(range(30), 1 + k % 5):
                dist[s] = 3
        elif kind == "cl":
            cl = complete_lengths(sorted({s for s, _ in rle_ops(lit + dist)}), 19, 7)
            for s in [s for s in range(19) if not cl[s]][:1 + k % 3]:
                cl[s] = 7
        else:
            lit = [8] * 258 + [0] * 28                          # 256 -> literal 0's slot, 257 -> literal 1's slot
        lmap, dmap = decodes_as(lit), decodes_as(dist)
        assert lmap[256] == 256
        usable_lit = [l if lmap.get(s) == s else 0 for s, l in enumerate(lit)]
        usable_dist = [l if dmap.get(s) == s else 0 for s, l in enumerate(dist)]
        syms = random_symbols(rng, usable_lit, usable_dist, 1500 + 100 * k, 0, 0.3)
        if kind == "collide":
            syms += [1, ("D", 0, 0, 0)] + syms[:40] + [0] + syms[40:80]      # 1 reads as length 3, 0 ends the block
        st = {}
        data, exp = forge([Dynamic(syms, lit, dist, final=True, cl_lengths=cl)], stats=st)
        assert exp is not None and st["kraft"] > 1
        units.append(Unit("oversub", f"{kind}_{k}", data, exp, OK, stats=st))


def _header_edges(units, rng):
    def simple(nlit, ndist):
        lit = complete_lengths(range(nlit), nlit)
        dist = [0] * ndist
        dist[0], dist[ndist - 1] = 1, 1
        return lit, dist

    for nlit in (257, 286):                                   # HLIT 257 and 286
        lit, dist = simple(nlit, 30)
        syms = random_symbols(rng, lit, dist, 800, 0, 0.3)
        data, exp = forge([Dynamic(syms, lit, dist, final=True)])
        units.append(Unit("header", f"hlit_{nlit}", data, exp, OK, zlib_ok=True))
    # a small dynamic block: the truncation family cuts it at every bit length
    lit = complete_lengths([97, 98, 99, 256, 257], 286)
    data, exp = forge([Dynamic([97, 98, 99, 97, ("m", 3, 1), 98, 99], lit, [1], final=True)])
    units.append(Unit("header", "small_dynamic", data, exp, OK, zlib_ok=True))
    for field in (30, 31):                                    # HLIT field 30/31 = 287/288 symbols
        lit, dist = simple(286, 30)
        data, _ = forge([Dynamic([65], lit, dist, final=True, hlit=field)])
        units.append(Unit("header", f"hlit_field_{field}", data, None, WRONG_SYMBOL))
    # HDIST 32: distance symbols 30/31 assigned, unused (valid for the reference) and used (wrongSymbol)
    lit, _ = simple(286, 30)
    dist = [5] * 32
    syms = random_symbols(rng, lit, dist[:30], 900, 0, 0.3)
    data, exp = forge([Dynamic(syms, lit, dist, final=True)])
    units.append(Unit("header", "hdist_32_unused", data, exp, OK, zlib_ok=False))
    for ds in (30, 31):
        data, _ = forge([Dynamic([1, 2, 3, ("L", 285, 0, 0), ("D", ds, 0, 0)], lit, dist, final=True)])
        units.append(Unit("header", f"hdist_32_uses_{ds}", data, None, WRONG_SYMBOL))
    # HCLEN 4: only code-length symbols 16, 17, 18, 0 can have codes -> every length is 0 -> no lit/len code at all
    ops = [(18, 127), (18, 127), (17, 1)]                    # 138 + 138 + 4 = 280 ... + 6 zeros below
    ops += [(0, 0)] * 6 + [(0, 0)]                           # 286 lit/len + 1 distance
    cl = [0] * 19
    cl[16], cl[17], cl[18], cl[0] = 2, 2, 2, 2
    data, _ = forge([Dynamic([], [0] * 286, [0], final=True, cl_ops=ops, cl_lengths=cl, hclen=0, eob=False)])
    units.append(Unit("header", "hclen_4", data + b"\x00", None, SYMBOL_NOT_FOUND))
    # HCLEN 19: all 19 code-length-code lengths written
    lit, dist = simple(286, 30)
    syms = random_symbols(rng, lit, dist, 600, 0, 0.3)
    used = {s for s, _ in rle_ops(lit + dist)}
    cl = complete_lengths(sorted(used | {15}), 19, 7)
    data, exp = forge([Dynamic(syms, lit, dist, final=True, cl_lengths=cl, hclen=15)])
    units.append(Unit("header", "hclen_19", data, exp, OK, zlib_ok=True))
    # 16 as the first code-length code
    ops = [(16, 0)] + rle_ops(lit + dist)
    cl = complete_lengths(sorted({s for s, _ in ops}), 19, 7)
    data, _ = forge([Dynamic([65], lit, dist, final=True, cl_ops=ops, cl_lengths=cl)])
    units.append(Unit("header", "first_16", data, None, WRONG_SYMBOL))
    # 138-long 18 runs: 256 literals unused except a few, so the lengths vector has long zero runs
    lit = [0] * 286
    for s in (1, 2, 200, 250, 256, 257):
        lit[s] = 3
    lit[285] = 2
    dist = [0] * 30
    dist[0] = 1; dist[29] = 1
    syms = random_symbols(rng, lit, dist, 2000, 0, 0.4)
    ops = rle_ops(lit + dist)
    assert (18, 127) in ops
    data, exp = forge([Dynamic(syms, lit, dist, final=True)])
    units.append(Unit("header", "runs_138", data, exp, OK, zlib_ok=True))
    # a 16 that crosses from the lit/len lengths into the distance lengths (RFC 1951 allows it)
    lit = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 6        # 286 = fixed lengths
    dist = [8] * 2 + [5] * 28
    lit[284], lit[285] = 8, 8
    # lit/len 285 = 8, then a 16 repeating it 3 times: distance lengths 0..2
    ops = rle_ops(lit[:285]) + [(8, 0), (16, 0)] + rle_ops(dist[3:])
    dist2 = [8, 8, 8] + dist[3:]
    syms = random_symbols(rng, lit, dist2, 1200, 0, 0.3)
    data, exp = forge([Dynamic(syms, lit, dist2, final=True, cl_ops=ops)])
    units.append(Unit("header", "repeat_16_crosses", data, exp, OK, zlib_ok=False))      # incomplete sets: zlib refuses
    # overshooting repeats: 16 past the count (wrongSymbol at once), 17 / 18 past the count (n != count, wrongSymbol)
    lit, dist = simple(286, 30)
    base_ops = rle_ops(lit + dist)
    tail = rle_ops(dist)
    head_ops = base_ops[:len(base_ops) - len(tail)]
    for name, extra_ops in (("over_16", [(5, 0)] * 27 + [(16, 3)]), ("over_17", [(5, 0)] * 25 + [(17, 7)]),
                            ("over_18", [(18, 20)])):
        ops = head_ops + extra_ops
        cl = complete_lengths(sorted({s for s, _ in ops}), 19, 7)
        data, _ = forge([Dynamic([], lit, dist, final=True, cl_ops=ops, cl_lengths=cl, eob=False)])
        units.append(Unit("header", name, data + b"\xff\xff", None, WRONG_SYMBOL))
    # HCLEN / HLIT present but the input ends inside the code-length-code lengths
    data, _ = forge([Dynamic([65], *simple(286, 30), final=True, hclen=15)])
    units.append(Unit("header", "cut_in_cl_lengths", data[:4], None, SYMBOL_NOT_FOUND))


def _static_edges(units, rng):
    pre = [rng.randrange(256) for _ in range(40)]
    for sym in (286, 287):
        data, _ = forge([Fixed(pre + [("L", sym, 0, 0)], final=True)])
        units.append(Unit("static", f"lit_{sym}", data + b"\0\0", None, WRONG_SYMBOL))
    for ds in (30, 31):
        data, _ = forge([Fixed(pre + [("L", 260, 0, 0), ("D", ds, 0, 0)], final=True)])
        units.append(Unit("static", f"dist_{ds}", data + b"\0\0", None, WRONG_SYMBOL))
    # length 258 as code 285 and as code 284 + extra 31 (RFC 1951 3.2.5 leaves the second form out; the reference decodes it)
    for form, sym in (("285", ("L", 285, 0, 0)), ("284_31", ("L", 284, 31, 5))):
        syms = pre + [sym, ("D", 0, 0, 0)] + pre
        data, exp = forge([Fixed(syms, final=True)])
        if form == "284_31":
            exp = bytes(pre) + bytes([pre[-1]]) * 258 + bytes(pre)
        units.append(Unit("static", f"len258_{form}", data, exp, OK, zlib_ok=True))


def _matches(units, rng):
    # distance == output so far (valid), output + 1 (trap)
    for n in (1, 2, 3, 100, 1000, 32768):
        lits = [rng.randrange(256) for _ in range(n)]
        data, exp = forge([Fixed(lits + [("m", 10, n)], final=True)])
        units.append(Unit("matches", f"dist_eq_out_{n}", data, exp, OK, zlib_ok=True))
        if n < 32768:
            data, _ = forge([Fixed(lits + [("m", 10, n + 1)], final=True)])
            units.append(Unit("matches", f"dist_out_plus_1_{n}", data, None, TRAP))
    # a match with nothing before it
    data, _ = forge([Fixed([("m", 3, 1)], final=True)])
    units.append(Unit("matches", "dist_at_start", data, None, TRAP))
    # distance 32768, a chain of them
    lits = [rng.randrange(256) for _ in range(40000)]
    data, exp = forge([Fixed(lits + [("m", 258, 32768)] * 20 + [("m", 3, 32768)], final=True)])
    units.append(Unit("matches", "dist_32768", data, exp, OK, zlib_ok=True))
    # distances 1..40 x lengths 3..258: period < length, every phase of src[i % d]
    for d0 in range(1, 41, 4):
        syms = [rng.randrange(256) for _ in range(41)]
        for d in range(d0, d0 + 4):
            for length in range(3, 259, 1 if d < 9 else 5):
                syms.append(("m", length, d))
                syms.append(rng.randrange(256))
        data, exp = forge([Fixed(syms, final=True)])
        units.append(Unit("matches", f"periodic_{d0}", data, exp, OK, zlib_ok=True))
    # sources in an earlier stored block and in an earlier Huffman block
    for k in range(4):
        raw = bytes(rng.randrange(256) for _ in range(3000 + 700 * k))
        syms = [("m", rng.randrange(3, 259), rng.randrange(1, len(raw) + 1)) for _ in range(60)]
        data, exp = forge([Stored(raw), Fixed([7, 8, 9]), Fixed(syms, final=True)])
        units.append(Unit("matches", f"src_in_stored_{k}", data, exp, OK, zlib_ok=True))
        h = [rng.randrange(256) for _ in range(2000)]
        lit = complete_lengths(range(286), 286)
        dist = complete_lengths(range(30), 30)
        syms2 = random_symbols(rng, lit, dist, 1000, 2000 + 3, 0.5)
        data, exp = forge([Fixed(h), Stored(b"abc"), Dynamic(syms2, lit, dist, final=True)])
        units.append(Unit("matches", f"src_in_huffman_{k}", data, exp, OK, zlib_ok=True))


RUNS = (255, 256, 257, 511, 512, 32767, 32768, 32769, 65535, 65536, 100003)


def _literal_runs(units, rng):
    for n in RUNS:
        lits = [rng.randrange(256) for _ in range(n)]
        raw = bytes(lits)
        tail = [("m", 17, 5), 1, 2, ("m", 3, 1)]
        forms = {
            "huffman": [Fixed(lits + tail, final=True)],
            "stored": [Stored(raw[i:i + 65535]) for i in range(0, n, 65535)] + [Fixed(tail, final=True)],
            # the run continues across block boundaries: Huffman literals, a stored block, Huffman literals, the match
            "mixed": [Fixed(lits[:n // 2]), Stored(raw[n // 2:n // 2 + 60000]), Fixed(lits[n // 2 + 60000:] + tail, final=True)],
        }
        for form, blocks in forms.items():
            st = {}
            data, exp = forge(blocks, stats=st)
            units.append(Unit("literal_runs", f"{form}_{n}", data, exp, OK, zlib_ok=True, stats=st))


def _block_structure(units, rng):
    for size in (0, 65535):
        raw = bytes(rng.randrange(256) for _ in range(size))
        for m in range(8):                                   # fixed block of m 9-bit literals: the stored header starts at bit 2 + m
            lead = [144 + rng.randrange(112) for _ in range(m)]
            for pad in (0, 1):
                data, exp = forge([Fixed(lead), Stored(raw, pad=pad), Fixed([1, 2, 3], final=True)])
                units.append(Unit("blocks", f"stored_{size}_off{(2 + m) % 8}_pad{pad}", data, exp, OK, zlib_ok=True))
    # bogus NLEN: the reference only checks LEN & NLEN == 0
    for nlen in (0, 0x00F0):
        data, exp = forge([Stored(b"abcde", nlen=nlen, final=True)])
        units.append(Unit("blocks", f"nlen_{nlen}", data, b"abcde", OK, zlib_ok=False))
    data, _ = forge([Stored(b"abcde", nlen=0xFFFF, final=True)])
    units.append(Unit("blocks", "nlen_overlaps", data, None, WRONG_LENGTHS))
    data, _ = forge([Stored(b"abcde" * 20, final=True)])
    units.append(Unit("blocks", "stored_cut", data[:50], None, WRONG_LENGTHS))
    # 300 one-symbol blocks, fixed and stored mixed
    for k in range(2):
        blocks = [Fixed([rng.randrange(256)]) if (i + k) % 3 else Stored(bytes([i & 255])) for i in range(300)]
        blocks[-1].final = True
        data, exp = forge(blocks)
        units.append(Unit("blocks", f"blocks_300_{k}", data, exp, OK, zlib_ok=True))
    # trailing bytes after the final block (consumed bits stop at the end of the final block)
    for k in range(4):
        data, exp = forge([Fixed([rng.randrange(256) for _ in range(10 + k)], final=True)])
        units.append(Unit("blocks", f"trailing_{k}", data + bytes(rng.randrange(256) for _ in range(1 + 7 * k)), exp, OK,
                          zlib_ok=True))
    # no final block: the reader runs out of bits at the next header
    for k in range(6):
        data, _ = forge([Fixed([rng.randrange(144) for _ in range(3 + k)])])
        w_bits = 3 + 8 * (3 + k) + 7                       # header + 8-bit literals (0..143 only) + EOB
        pad = (8 - w_bits % 8) % 8
        # < 3 padding bits: the BFINAL/BTYPE read traps; >= 3 zero bits: a stored header, then < 4 bytes for LEN/NLEN
        units.append(Unit("blocks", f"no_final_{k}", data, None, TRAP if pad < 3 else WRONG_LENGTHS))
    # block type 3
    units.append(Unit("blocks", "btype_3", bytes([0b111]) + b"\0\0", None, WRONG_BLOCK_TYPE))
    units.append(Unit("blocks", "too_short", b"\x03", None, WRONG_BLOCK_TYPE))


def _truncations(units, rng, sources):
    for src in sources:
        for cut in range(1, len(src.data)):
            units.append(Unit("truncation", f"{src.family}/{src.name}@{cut}B", src.data[:cut], None, "error"))
    small = [s for s in sources if len(s.data) <= 48]
    for src in small:
        for bits in range(1, len(src.data) * 8):
            b = bytearray(src.data[:(bits + 7) // 8])
            if bits % 8:
                b[-1] &= (1 << (bits % 8)) - 1
            units.append(Unit("truncation", f"{src.family}/{src.name}@{bits}b", bytes(b), None, None))


def corpus(seed=20261017):
    """the forged units, a few hundred distinct ones"""
    rng = random.Random(seed)
    units = []
    _long_codes(units, rng)
    _sym48(units, rng)
    _uniform(units, rng)
    _incomplete(units, rng)
    _oversub(units, rng)
    _header_edges(units, rng)
    _static_edges(units, rng)
    _matches(units, rng)
    _literal_runs(units, rng)
    _block_structure(units, rng)
    srcs = [u for u in units if u.status == OK and len(u.data) < 400][:8]
    srcs += [u for u in units if u.family == "header" and u.name in ("hclen_19", "small_dynamic")]
    _truncations(units, rng, srcs)
    seen, distinct = set(), []
    for u in units:                       # a bit cut that ends on a byte boundary repeats a byte cut
        if u.data not in seen:
            seen.add(u.data)
            distinct.append(u)
    return distinct
