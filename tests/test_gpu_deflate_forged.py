"""Forged Deflate streams (tests/deflate_forge.py) through every Huffman stage of the batched call, compared unit by unit with the
oracle (status; out_len, consumed bits and bytes when the oracle decodes) and with the bytes the forge wrote:

  a. small batch  -> inflate_warp_kernel (K1w) + lz_resolve_kernel (K2) + inflate_slow_kernel
  b. >= 20 000 units, every in_off % 16 -> inflate_lut_kernel (K1L) + K2 + inflate_slow_kernel
  c. start_bits (k junk bits before each stream) at both batch sizes
  d. output fences: capacities around the decoded size, every byte outside the units' capacities keeps its canary
  e. the same fences for LZ4 blocks (lz4_parse_kernel + lz4_exec_kernel)
  f. the thread-per-unit K1 (SWC_DEFLATE_K1=thread) on the small corpus, in a subprocess
  g. a 2^28-byte unit inside a K1L batch: SWC_ERR_UNSUPPORTED (DESIGN §6), its neighbours decode"""
import ctypes as C
import os
import random
import subprocess
import sys
import time

import numpy as np
import pytest

import deflate_forge as F
import helpers as H

pytestmark = pytest.mark.gpu

LARGE = 20480               # batches of >= 20 000 units take K1L
CANARY = 0xA5
S_OVERFLOW, S_UNSUPPORTED = 1, 6
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module", autouse=True)
def timer():
    t0 = time.time()
    yield
    print(f"\n{__name__}: {time.time() - t0:.1f} s")


@pytest.fixture(scope="module")
def corpus(oracle):
    units = F.corpus()
    ref = [oracle.deflate_decompress(u.data) for u in units]
    return units, ref


def _align(v, a=16):
    return (v + a - 1) // a * a


def pack(datas, shifts=None):
    """input buffer with unit i at a 16-byte boundary + shifts[i] bytes"""
    n = len(datas)
    shifts = np.zeros(n, dtype=np.int64) if shifts is None else np.asarray(shifts)
    offs = np.zeros(n, dtype=np.uint64)
    cur = 0
    for i, d in enumerate(datas):
        offs[i] = _align(cur) + int(shifts[i])
        cur = int(offs[i]) + len(d)
    buf = np.zeros(_align(cur) + 64, dtype=np.uint8)
    for d, o in zip(datas, offs):
        buf[int(o):int(o) + len(d)] = np.frombuffer(d, dtype=np.uint8)
    return buf, offs, np.array([len(d) for d in datas], dtype=np.uint64)


def out_layout(caps, gap=16):
    """16-byte aligned output regions with `gap` bytes between them (fence bytes no unit may touch)"""
    caps = np.asarray(caps, dtype=np.uint64)
    ends = np.cumsum(((caps + np.uint64(15)) // np.uint64(16) * np.uint64(16)) + np.uint64(gap))
    offs = np.concatenate([[0], ends[:-1]]).astype(np.uint64)
    return offs, int(ends[-1]) if len(caps) else 0


class Run:
    """one batched call through the C ABI with hand-built offsets; d_out starts as CANARY"""

    def __init__(self, codec, buf, in_off, in_len, caps, start_bits=None):
        import torch
        from swcompression_b200 import _lib
        L = _lib.lib()
        self.n = n = len(in_off)
        self.caps = np.asarray(caps, dtype=np.uint64)
        self.out_off, self.out_total = out_layout(self.caps)
        dev = torch.device("cuda:0")
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        d_in, d_ioff, d_ilen = t(buf), t(in_off.view(np.int64)), t(in_len.view(np.int64))
        d_ooff, d_ocap = t(self.out_off.view(np.int64)), t(self.caps.view(np.int64))
        self.d_out = torch.full((self.out_total + 64,), CANARY, dtype=torch.uint8, device=dev)
        d_len = torch.zeros(n, dtype=torch.int64, device=dev)
        d_used = torch.zeros(n, dtype=torch.int64, device=dev)
        d_st = torch.full((n,), -1, dtype=torch.int32, device=dev)
        d_sb = None if start_bits is None else t(np.asarray(start_bits, dtype=np.uint8))
        p = lambda x: C.c_void_p(x.data_ptr()) if x is not None else None
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        if codec == "deflate":
            scratch = torch.empty(L.swc_deflate_batch_scratch_bytes(n, self.out_total), dtype=torch.uint8, device=dev)
            rc = L.swc_deflate_decompress_batch(p(d_in), p(d_ioff), p(d_ilen), p(d_sb), p(self.d_out), p(d_ooff), p(d_ocap),
                                                self.out_total, p(d_len), p(d_used), p(d_st), n, p(scratch), scratch.numel(),
                                                stream)
        else:
            rc = L.swc_lz4_block_decompress_batch(p(d_in), p(d_ioff), p(d_ilen), None, 0, p(self.d_out), p(d_ooff), p(d_ocap),
                                                  p(d_len), p(d_st), n, stream)
        assert rc == 0, _lib.status_name(rc)
        torch.cuda.synchronize(dev)
        self.st, self.ln, self.used = d_st.cpu().numpy(), d_len.cpu().numpy(), d_used.cpu().numpy()
        self.keep = (d_in, d_ioff, d_ilen, d_ooff, d_ocap, d_sb)

    def host_out(self):
        return self.d_out.cpu().numpy()

    def output(self, host, i):
        o = int(self.out_off[i])
        return bytes(host[o:o + int(self.ln[i])])

    def fence_intact(self, host=None):
        """every byte outside [out_off[i], out_off[i] + cap[i]) still holds the canary (64-byte tail included)"""
        host = self.host_out() if host is None else host
        inside = np.zeros(len(host), dtype=bool)
        for o, c in zip(self.out_off, self.caps):
            inside[int(o):int(o) + int(c)] = True
        bad = np.flatnonzero(~inside & (host != CANARY))
        if len(bad):
            unit = int(np.searchsorted(self.out_off, bad[0], side="right")) - 1
            return f"{len(bad)} fence bytes overwritten, first at {int(bad[0])} (after unit {unit}, cap {int(self.caps[unit])})"
        return None


def check(run, ref, names, host=None, expect=None):
    """status / out_len / consumed / bytes of every unit against the oracle results `ref` (and the forge's bytes)"""
    host = run.host_out() if host is None else host
    for i in range(run.n):
        ost, oout, oused = ref[i]
        tag = (i, names[i], int(run.st[i]), ost)
        if ost == 0 and len(oout) > int(run.caps[i]):
            assert run.st[i] == S_OVERFLOW and run.ln[i] == len(oout), tag + (int(run.ln[i]), len(oout))
        elif ost == 0:
            assert run.st[i] == 0 and run.ln[i] == len(oout) and run.used[i] == oused, tag + (int(run.ln[i]), len(oout), int(run.used[i]), oused)
            got = run.output(host, i)
            assert got == oout, tag + (next(k for k in range(len(got)) if got[k] != oout[k]),)
            if expect is not None and expect[i] is not None:
                assert got == expect[i], tag
        else:
            assert run.st[i] == ost, tag


def _caps_for(ref, slack=4096):
    return [len(o) if st == 0 else slack for st, o, _ in ref]


# ---------------------------------------------------------------------------------------------------------------- a
def test_a_small_batch(corpus):
    units, ref = corpus
    assert len(units) < 20000
    buf, off, ln = pack([u.data for u in units])
    run = Run("deflate", buf, off, ln, _caps_for(ref))
    check(run, ref, units, expect=[u.expect for u in units])
    assert run.fence_intact() is None


# ---------------------------------------------------------------------------------------------------------------- b
def test_b_large_batch_lut_kernel(corpus):
    import torch
    units, ref = corpus
    n0 = len(units)
    tiles = max(16, -(-LARGE // n0))
    rng = np.random.default_rng(7)
    order = rng.permutation(n0 * tiles)
    uid, tile = order % n0, order // n0
    datas = [units[k].data for k in uid]
    buf, off, ln = pack(datas, shifts=tile % 16)
    assert len(datas) >= 20000 and len(set((off % np.uint64(16)).tolist())) == 16
    oversub = sum(units[k].oversub for k in uid)
    assert oversub >= 300, "the batch must send a few hundred units to inflate_slow_kernel"
    caps = np.array(_caps_for(ref), dtype=np.uint64)[uid]
    run = Run("deflate", buf, off, ln, caps)
    ost = np.array([r[0] for r in ref])[uid]
    olen = np.array([len(r[1]) for r in ref])[uid]
    oused = np.array([r[2] for r in ref])[uid]
    okm = ost == 0
    bad = np.flatnonzero(run.st != ost)
    assert len(bad) == 0, [(int(j), units[uid[j]], int(run.st[j]), int(ost[j])) for j in bad[:10]]
    assert (run.ln[okm] == olen[okm]).all() and (run.used[okm] == oused[okm]).all()
    # every unit's bytes against one expected buffer, compared on the device: the decoded bytes of every unit, and the canary
    # everywhere outside the capacities (inside a capacity but past the decoded length, bytes may change)
    exp = np.full(run.out_total + 64, CANARY, dtype=np.uint8)
    checked = np.ones(run.out_total + 64, dtype=bool)
    for j in range(run.n):
        o = int(run.out_off[j])
        checked[o:o + int(run.caps[j])] = False
        if okm[j]:
            exp[o:o + olen[j]] = np.frombuffer(ref[uid[j]][1], dtype=np.uint8)
            checked[o:o + olen[j]] = True
    wrong = (run.d_out != torch.from_numpy(exp).cuda()) & torch.from_numpy(checked).cuda()
    if bool(wrong.any()):
        first = int(torch.nonzero(wrong)[0])
        j = int(np.searchsorted(run.out_off, first, side="right")) - 1
        pytest.fail(f"byte {first} wrong: unit {j} = {units[uid[j]]}, offset {first - int(run.out_off[j])}, cap {int(run.caps[j])}")


# ---------------------------------------------------------------------------------------------------------------- c
def _with_junk(data, k, rng):
    w = H.LsbBitWriter()
    w.write_number(rng.getrandbits(8), k)
    w.write_bytes(data)
    return w.data


@pytest.mark.parametrize("large", [False, True], ids=["small", "large"])
def test_c_start_bits(corpus, oracle, large):
    units, _ = corpus
    rng = random.Random(3)
    base = [u for u in units if u.family != "truncation"] + [u for u in units if u.family == "truncation"][::4]
    tiles = -(-LARGE // len(base)) if large else 1
    datas, ks, names, ref = [], [], [], []
    cache = {}
    for t in range(tiles):
        for i, u in enumerate(base):
            k = (i + t) % 8
            key = (i, k)
            if key not in cache:
                d = _with_junk(u.data, k, rng)
                cache[key] = (d, oracle.deflate_decompress(d, k))
            d, r = cache[key]
            datas.append(d); ks.append(k); names.append(u); ref.append(r)
    shifts = np.arange(len(datas)) % 16 if large else None
    buf, off, ln = pack(datas, shifts)
    run = Run("deflate", buf, off, ln, _caps_for(ref), start_bits=ks)
    assert (run.n >= 20000) == large
    check(run, ref, names)
    assert run.fence_intact() is None


# ---------------------------------------------------------------------------------------------------------------- d
def _fence_set(units, ref, max_need):
    datas, caps, refs, names = [], [], [], []
    for u, r in zip(units, ref):
        if r[0] != 0 or len(r[1]) > max_need:
            continue
        need = len(r[1])
        cs = sorted({c for c in range(need - 17, need + 18) if c >= 0} | {need & ~7, 0})
        for c in cs:
            datas.append(u.data); caps.append(c); refs.append(r); names.append(u)
    return datas, caps, refs, names


@pytest.mark.parametrize("large", [False, True], ids=["small", "large"])
def test_d_output_fences(corpus, large):
    units, ref = corpus
    datas, caps, refs, names = _fence_set(units, ref, 70000 if not large else 20000)
    if large:
        tiles = -(-LARGE // len(datas))
        datas, caps, refs, names = datas * tiles, caps * tiles, refs * tiles, names * tiles
    else:
        assert len(datas) < 20000
    buf, off, ln = pack(datas, np.arange(len(datas)) % 16)
    run = Run("deflate", buf, off, ln, caps)
    assert (run.n >= 20000) == large
    host = run.host_out()
    check(run, refs, names, host=host)
    msg = run.fence_intact(host)
    assert msg is None, msg


# ---------------------------------------------------------------------------------------------------------------- e
def _lz4_raws(rng):
    raws = []
    for p in range(2, 16):
        pat = bytes(rng.getrandbits(8) for _ in range(p))
        for n in (64, 65, 100, 257, 1000, 4099):
            pre = bytes(rng.getrandbits(8) for _ in range(rng.randrange(0, 20)))
            raws.append(pre + (pat * (n // p + 2))[:n] + b"tail" + pre)
    raws += [H.textlike(n, 900 + n) for n in (70, 300, 5000, 30000)]
    raws += [bytes(n) for n in (13, 64, 100, 1000, 20000)]
    return raws


@pytest.mark.parametrize("large", [False, True], ids=["small", "large"])
def test_e_lz4_block_fences(oracle, large):
    rng = random.Random(21)
    raws = _lz4_raws(rng)
    datas, caps, raw_of = [], [], []
    for r in raws:
        comp = H.lz4_block_compress(r)
        st, out, _ = oracle.lz4_block(comp)
        assert st == 0 and out == r
        need = len(r)
        for c in sorted({c for c in range(need - 17, need + 18, 3) if c >= 0} | {need, need & ~7, 0}):
            datas.append(comp); caps.append(c); raw_of.append(r)
    if large:
        tiles = -(-LARGE // len(datas))
        datas, caps, raw_of = datas * tiles, caps * tiles, raw_of * tiles
    buf, off, ln = pack(datas, np.arange(len(datas)) % 16)
    run = Run("lz4_block", buf, off, ln, caps)
    assert (run.n >= 20000) == large
    host = run.host_out()
    for i, r in enumerate(raw_of):
        if len(r) > caps[i]:
            assert run.st[i] == S_OVERFLOW and run.ln[i] == len(r), (i, len(r), caps[i], int(run.st[i]), int(run.ln[i]))
        else:
            assert run.st[i] == 0 and run.output(host, i) == r, (i, len(r), caps[i], int(run.st[i]))
    msg = run.fence_intact(host)
    assert msg is None, msg


# ---------------------------------------------------------------------------------------------------------------- f
_CHILD = r"""
import sys, numpy as np
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests", sys.argv[1] + "/oracle"]
import test_gpu_deflate_forged as T
z = np.load(sys.argv[2])
run = T.Run("deflate", z["buf"], z["off"], z["ln"], z["caps"])
np.savez(sys.argv[3], st=run.st, ln=run.ln, used=run.used, out=run.host_out())
"""


def test_f_round1_thread_kernel(corpus, tmp_path):
    units, ref = corpus
    buf, off, ln = pack([u.data for u in units])
    caps = np.array(_caps_for(ref), dtype=np.uint64)
    np.savez(tmp_path / "in.npz", buf=buf, off=off, ln=ln, caps=caps)
    env = dict(os.environ, SWC_DEFLATE_K1="thread")
    subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(tmp_path / "in.npz"), str(tmp_path / "res.npz")], env=env,
                   check=True, timeout=600)
    thr = np.load(tmp_path / "res.npz")
    run = Run("deflate", buf, off, ln, caps)                  # K1w, as run a
    assert (thr["st"] == run.st).all(), [(i, units[i], int(thr["st"][i]), int(run.st[i])) for i in np.flatnonzero(thr["st"] != run.st)[:10]]
    ok = run.st == 0
    assert (thr["ln"][ok] == run.ln[ok]).all() and (thr["used"][ok] == run.used[ok]).all()
    host = run.host_out()
    for i in np.flatnonzero(ok):
        o, n = int(run.out_off[i]), int(run.ln[i])
        assert bytes(thr["out"][o:o + n]) == bytes(host[o:o + n]), (i, units[i])


# ---------------------------------------------------------------------------------------------------------------- g
def test_g_unit_past_32bit_positions(corpus):
    units, ref = corpus
    good = [(u, r) for u, r in zip(units, ref) if r[0] == 0 and len(u.data) < 4096 and len(r[1]) < 4096]
    n = 20000
    big_at = 10007
    datas, refs = [], []
    for i in range(n):
        u, r = good[i % len(good)]
        datas.append(u.data); refs.append(r)
    buf, off, ln = pack(datas)
    big = 1 << 28
    # the big unit sits after the others; its contents do not matter, the length alone decides
    off[big_at] = np.uint64(len(buf))
    ln[big_at] = np.uint64(big)
    buf = np.concatenate([buf, np.zeros(big + 64, dtype=np.uint8)])
    caps = [len(r[1]) for r in refs]
    caps[big_at] = 4096
    run = Run("deflate", buf, off, ln, caps)
    assert run.st[big_at] == S_UNSUPPORTED
    host = run.host_out()
    for i in range(n):
        if i == big_at:
            continue
        assert run.st[i] == 0 and run.output(host, i) == refs[i][1] and run.used[i] == refs[i][2], i
