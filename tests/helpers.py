"""Shared test helpers: golden fixtures, synthetic corpora, a Python LsbBitWriter (BitByteData semantics)."""
import ctypes as C
import json
import os
import random
import struct
import zlib

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

with open(os.path.join(GOLDEN, "manifest.json")) as _f:
    MANIFEST = json.load(_f)


def answer(name):
    a = MANIFEST["answers"][name]
    if "literal" in a:
        return a["literal"].encode().decode("unicode_escape").encode("latin1")
    return bytes(a["zeros"])


def fixture(rel):
    with open(os.path.join(GOLDEN, rel), "rb") as f:
        return f.read()


def fixtures(prefix):
    return [(rel, meta["answer"]) for rel, meta in sorted(MANIFEST["fixtures"].items()) if rel.startswith(prefix)]


class LsbBitWriter:
    """BitByteData.LsbBitWriter: bits fill each byte from bit 0 upward; numbers are written LSB first."""

    # Whole bytes go to `out`; the < 8 pending bits sit in the integer `acc` (bit k of acc = stream bit nbits_done + k).
    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.nacc = 0

    def __len__(self):
        """number of bits written so far"""
        return len(self.out) * 8 + self.nacc

    def write_bits(self, bits):
        for b in bits:
            self.write_number(b & 1, 1)

    def write_number(self, value, count):
        self.acc |= (value & ((1 << count) - 1)) << self.nacc
        self.nacc += count
        if self.nacc >= 8:
            k = self.nacc >> 3
            self.out += (self.acc & ((1 << (8 * k)) - 1)).to_bytes(k, "little")
            self.acc >>= 8 * k
            self.nacc &= 7

    def write_bytes(self, data):
        """bytes at the current bit position (a byte-aligned writer appends them as they are)"""
        if self.nacc == 0:
            self.out += data
        else:
            for byte in data:
                self.write_number(byte, 8)

    def align(self, fill=0):
        """pad to a byte boundary with `fill` bits (0 or 1)"""
        if self.nacc:
            pad = 8 - self.nacc
            self.write_number((1 << pad) - 1 if fill else 0, pad)

    @property
    def data(self):
        self.align()
        return bytes(self.out)


# literal round-trip vectors of the reference's compression tests (DeflateCompressionTests.swift:7-83,
# BZip2CompressionTests.swift:11-95, LZ4CompressionTests.swift:11-171)
ROUNDTRIP_STRINGS = [
    b"ban", b"banana", b"abaaba", b"abracadabra", b"cabbage", b"baabaabac", b"AAAAAAABBBBCCCD", b"AAAAAAA",
    b"abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789", bytes(range(256)), b"", b"a",
    b"Hello, World!\n", b"the quick brown fox jumps over the lazy dog " * 40,
]


def textlike(n, seed):
    """SURVEY.md §8(d) corpus: order-1 Markov over a 64-symbol Zipf(1.2) alphabet + ~30 % back-references."""
    rng = np.random.Generator(np.random.PCG64(seed))
    ranks = np.arange(1, 65, dtype=np.float64)
    p = ranks ** -1.2
    p /= p.sum()
    alphabet = np.frombuffer(b"etaoinshrdlucmfwypvbgkjqxz ETAOINSHRDLUCMFWYPVBGKJQXZ.,;:!?-'\"()\n", dtype=np.uint8)[:64]
    # order-1 flavour: each previous symbol rotates the Zipf ranking
    base = rng.choice(64, size=n, p=p)
    prev = np.concatenate([[0], base[:-1]])
    sym = (base + (prev * 7)) % 64
    out = alphabet[sym].copy()
    # back-references
    i = 64
    while i < n - 70:
        if rng.random() < 0.12:
            ln = int(rng.integers(3, 65))
            dist = int(rng.integers(1, min(i, 32768) + 1))
            for k in range(ln):
                out[i + k] = out[i + k - dist]
            i += ln
        else:
            i += int(rng.integers(1, 12))
    return out.tobytes()


def raw_deflate(data, level=6, mem_level=9):
    c = zlib.compressobj(level, zlib.DEFLATED, -15, mem_level)
    return c.compress(data) + c.flush()


_lz4 = None


def liblz4():
    global _lz4
    if _lz4 is None:
        _lz4 = C.CDLL("liblz4.so.1")
        _lz4.LZ4_compressBound.restype = C.c_int
        _lz4.LZ4_compress_default.restype = C.c_int
        _lz4.LZ4_compress_default.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_int]
    return _lz4


def lz4_block_compress(data):
    L = liblz4()
    cap = L.LZ4_compressBound(len(data))
    dst = C.create_string_buffer(max(cap, 16))
    n = L.LZ4_compress_default(data, dst, len(data), cap)
    assert n > 0 or len(data) == 0
    return dst.raw[:n]


def lz4_frame_independent(blocks_raw, bd=0x40, content_checksum=False, block_checksum=False):
    """B4 independent-block frame built by hand (FLG version 01, B.Indep=1)."""
    import oracle_xxh
    flg = 0x60 | (0x10 if block_checksum else 0) | (0x04 if content_checksum else 0)
    desc = bytes([flg, bd])
    out = bytearray(struct.pack("<I", 0x184D2204) + desc + bytes([(oracle_xxh.xxh32(desc) >> 8) & 0xFF]))
    for raw in blocks_raw:
        comp = lz4_block_compress(raw)
        if len(comp) >= len(raw):
            out += struct.pack("<I", len(raw) | 0x80000000) + raw
            blk = raw
        else:
            out += struct.pack("<I", len(comp)) + comp
            blk = comp
        if block_checksum:
            out += struct.pack("<I", oracle_xxh.xxh32(blk))
    out += struct.pack("<I", 0)
    if content_checksum:
        out += struct.pack("<I", oracle_xxh.xxh32(b"".join(blocks_raw)))
    return bytes(out)
