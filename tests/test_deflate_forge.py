"""Pins the Deflate stream forge (tests/deflate_forge.py) on the CPU: every unit meant to be valid decodes to the bytes the
forge wrote under the oracle and, where zlib accepts the stream, under zlib; every malformed family gets the status it
declares (read off Sources/Deflate/Deflate.swift) from the oracle.  The GPU tests rely on both."""
import collections
import zlib

import pytest

import deflate_forge as F
import helpers as H


@pytest.fixture(scope="module")
def units():
    return F.corpus()


def zlib_verdict(data):
    try:
        d = zlib.decompressobj(-15)
        return d.decompress(data) + d.flush()
    except zlib.error:
        return None


def test_bit_writer_layout():
    w = H.LsbBitWriter()
    w.write_number(0b101, 3)
    w.write_number(0x1FF, 9)
    w.write_bytes(b"\x80")
    assert len(w) == 20
    assert w.data == bytes([0b1111_1101, 0b0000_1111, 0b0000_1000])
    w = H.LsbBitWriter()
    w.write_bits([1, 0, 1, 1])
    w.align(fill=1)
    assert w.data == b"\xfd"


def test_canonical_codes_and_kraft():
    codes, k = F.canonical([2, 1, 3, 3])                     # RFC 1951 3.2.2 example
    assert codes == {1: (0b0, 1), 0: (0b10, 2), 2: (0b110, 3), 3: (0b111, 3)} and k == 1
    assert F.canonical([2, 2, 2])[1] < 1
    codes, k = F.canonical([1, 1, 1])                        # over-subscribed: the third code wraps onto the first
    assert k > 1 and codes[2] == codes[0]


def test_corpus_families(units):
    fams = collections.Counter(u.family for u in units)
    assert set(fams) == {"long_codes", "sym48", "uniform", "incomplete", "oversub", "header", "static", "matches",
                         "literal_runs", "blocks", "truncation"}
    assert len({u.data for u in units}) == len(units), "distinct units"


def test_long_codes_use_every_length(units):
    long = [u for u in units if u.family == "long_codes"]
    assert len(long) >= 12
    for u in long:
        lit, dist = u.lengths
        assert {l for l in lit if l} == set(range(1, 16)), u        # every lit/len code length 1..15 in use
        assert {l for l in dist if l} >= set(range(6, 16)), u       # distance codes of 6..15 bits
        assert F.kraft(lit) == 1 and F.kraft(dist) == 1, u
    assert any(u.lengths[0][256] == 15 for u in long), "end of block on a 15-bit code"
    assert any(any(l == 15 for l in u.lengths[0][257:]) and u.lengths[0][256] == 15 for u in long), "length symbol on a 15-bit code"
    assert any(any(l == 15 for l in u.lengths[0][:256]) for u in long), "literal on a 15-bit code"
    assert any(u.lengths[1][29] == 15 for u in long), "distance 29 on a 15-bit code"
    for u in (u for u in units if u.family == "sym48"):
        lit, dist = u.lengths
        assert lit[284] == 15 and dist[29] == 15, u                 # 15 + 5 + 15 + 13 = 48 bits per match


def test_oversubscribed_family(units):
    """every unit of the family really has a set with Kraft sum > 1, of each kind, and decodes to bytes the forge knows"""
    over = [u for u in units if u.family == "oversub"]
    assert all(u.oversub for u in over)
    assert not any(u.oversub for u in units if u.family != "oversub")
    kinds = {u.name.split("_")[0] for u in over}
    assert kinds == {"lit", "dist", "cl", "collide"}
    assert all(u.status == F.OK and u.expect is not None for u in over)


def test_decodes_as_follows_reference_tree():
    # complete set: every code reads back as its own symbol
    assert all(k == v for k, v in F.decodes_as(F.complete_lengths(range(286), 286)).items())
    # 258 codes of 8 bits: 256 and 257 wrap onto the slots of literals 0 and 1 and replace them
    m = F.decodes_as([8] * 258)
    assert m[0] == 256 and m[1] == 257 and m[256] == 256 and m[257] == 257 and m[2] == 2
    # [1, 1, 1, 2]: symbol 2 wraps onto symbol 0's slot; symbol 3 (code 11 0 -> wraps to 00) lies under that leaf
    m = F.decodes_as([1, 1, 1, 2])
    assert m[0] == 2 and m[1] == 1 and m[2] == 2 and m[3] is None


def test_oracle_agrees_with_forge_and_declared_status(oracle, units):
    seen = collections.Counter()
    for u in units:
        st, out, used = oracle.deflate_decompress(u.data)
        seen[(u.family, st)] += 1
        if u.status == "error":
            assert st != F.OK, u
        elif u.status is not None:
            assert st == u.status, (u, st)
        if u.expect is not None:
            assert st == F.OK and out == u.expect, u
        if st == F.OK:
            assert 0 < used <= 8 * len(u.data), u
    print("\noracle status per family:", dict(sorted(seen.items())))


def test_zlib_agrees_where_rfc_allows(units):
    verdicts = collections.Counter()
    for u in units:
        if u.zlib_ok is None:
            continue
        z = zlib_verdict(u.data)
        verdicts[(u.family, u.name.split("_")[0], z is not None)] += 1
        assert (z is not None) == u.zlib_ok, u
        if z is not None:
            assert z == u.expect, u
    print("\nzlib verdicts:", dict(sorted(verdicts.items())))


def test_consumed_bits_end_at_final_block(oracle, units):
    for u in units:
        if u.family == "blocks" and u.name.startswith("trailing"):
            st, out, used = oracle.deflate_decompress(u.data)
            d = zlib.decompressobj(-15)
            d.decompress(u.data)
            assert st == 0 and (used + 7) // 8 == len(u.data) - len(d.unused_data), u


def test_literal_runs_end_in_a_match(units):
    # a literal run of >= 32 768 bytes ending in a match is what sets the high half of an escape record
    runs = [u for u in units if u.family == "literal_runs"]
    assert len(runs) == 3 * len(F.RUNS)
    for u in runs:
        assert u.stats["max_run"] == int(u.name.split("_")[1]), u
    assert sum(u.stats["max_run"] >= 32768 for u in runs) == 3 * sum(n >= 32768 for n in F.RUNS)


def test_truncations_cut_a_dynamic_header_at_every_bit(units):
    src = next(u for u in units if u.name == "small_dynamic")
    have = {u.data for u in units}                 # a cut that changes no byte is the stream itself
    for bits in range(1, 8 * len(src.data)):
        cut = bytearray(src.data[:(bits + 7) // 8])
        if bits % 8:
            cut[-1] &= (1 << (bits % 8)) - 1
        assert bytes(cut) in have, bits


def test_header_offsets_of_stored_blocks(units):
    names = {u.name for u in units if u.family == "blocks"}
    for size in (0, 65535):
        assert {f"stored_{size}_off{k}_pad0" for k in range(8)} <= names
