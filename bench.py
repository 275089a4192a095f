#!/usr/bin/env python3
"""bench.py — headline benchmark of the hot path (BASELINE.json config 2): batched Deflate decode of independent
64 KiB dynamic-Huffman blocks on B200, measured as decompressed GB/s (10^9 B/s).

    python bench.py --gpus N --steps K --warmup W            # product arm (CUDA, through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...   # reference arm: the reference's algorithm on host cores

One "step" = one batched call of the hot path over the whole workload (262 144 units x 65 536 B = 16 GiB decoded per
GPU; 4096 distinct synthetic units tiled x64 on the device to bound host prep time).  `value` is measured with the
compressed batch resident in HBM; `e2e` goes through swc_deflate_decompress_batch_host with pinned HOST buffers, i.e.
host->device and device->host copies inside the timed region (the same 262 144 units).
`--dump-outputs DIR` writes what the last timed step returned (result tables, a seeded sample of decoded units) as
DIR/*.npy; the corpus is seeded, so the same flags give the same inputs and two builds can be compared output for output.
Multi-GPU: units are independent, every rank decodes its own shard with no data-path collective (weak scaling);
rank 0 owns the unit list and scatters byte-balanced shards over NCCL; `multi_gpu.legs` adds the gather / all-gather variants.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time
import zlib
from multiprocessing import Pool

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

UNIT = 65536
N_UNITS = 262144          # BASELINE.json configs[1]
DISTINCT = 4096
METRIC = "decompressed_GB_per_s"


def _make_unit(seed):
    import helpers as H
    raw = H.textlike(UNIT, seed)
    comp = H.raw_deflate(raw)           # zlib level 6, raw deflate, memLevel 9 -> one final dynamic block
    assert comp[0] & 7 == 0b101
    return comp, zlib.crc32(raw)


def make_corpus(distinct, seed0=2, world=1):
    """-> (compressed units, crc32 of every unit's raw bytes)"""
    procs = max(1, min((os.cpu_count() or 1) // max(world, 1), 32))
    with Pool(procs) as pool:
        res = pool.map(_make_unit, range(seed0, seed0 + distinct), chunksize=16)
    return [r[0] for r in res], [r[1] for r in res]


def workload_config(n_units, distinct, world):
    """The config both arms print (identical by construction): the workload, not how it was sampled or timed."""
    tile = n_units // distinct
    return {"workload": f"batched Deflate: {n_units} independent 64 KiB single-block dynamic-Huffman units per GPU "
                        f"(BASELINE configs[1]); {distinct} distinct units tiled x{tile}",
            "units_per_gpu": n_units, "unit_bytes": UNIT, "decompressed_bytes_per_gpu": n_units * UNIT,
            "parallelism": f"independent units sharded over {world} GPU(s), no data-path collective",
            "l2": "inputs+outputs (>20 GB) exceed the 126 MB L2; no flush needed",
            "corpus": "order-1 Markov/Zipf text + back-references (tests/helpers.textlike), zlib level 6 raw deflate memLevel 9"}


def host_memory_budget():
    """Bytes of host memory this job may use: MemAvailable, clipped by the cgroup limit when there is one."""
    avail = 1 << 62
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                avail = int(line.split()[1]) * 1024
    except OSError:
        pass
    for path in ("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory/memory.limit_in_bytes"):
        try:
            v = open(path).read().strip()
            if v != "max":
                lim = int(v)
                try:
                    used = int(open(path.replace("memory.max", "memory.current").replace("limit_in_bytes", "usage_in_bytes")).read())
                except (OSError, ValueError):
                    used = 0
                avail = min(avail, max(lim - used, 0))
        except (OSError, ValueError):
            pass
    return avail


DUMP_TABLE_UNITS = 1 << 18     # result-table rows dumped: 4 float64 columns = 8 MiB
DUMP_OUTPUT_UNITS = 192        # decoded units dumped as float32 rows: 48 MiB (56 MiB in all with the tables, under 64 MB)


def dump_outputs(b, out_dir, seed=0):
    """Writes what the last b.run() returned to its caller as .npy files: status, decoded length and consumed bits of every
    unit (of a seeded sample of 2^18 units in larger batches; `units.npy` holds their indices), and the decoded bytes of a
    seeded sample of 192 units (`output.npy`, one row of UNIT values per unit in `output_units.npy`, zero past the decoded
    length).  The same seed and batch give the same sample, so two builds can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    st, ln, used = b.results()
    rng = np.random.default_rng(seed)
    n = b.n
    rows = np.arange(n) if n <= DUMP_TABLE_UNITS else np.sort(rng.choice(n, DUMP_TABLE_UNITS, replace=False))
    picks = np.sort(rng.choice(n, min(n, DUMP_OUTPUT_UNITS), replace=False))
    out = np.zeros((len(picks), UNIT), dtype=np.float32)
    for r, i in enumerate(picks):
        o, m = int(b.h_out_off[i]), min(int(ln[i]), UNIT)
        out[r, :m] = b.d_out[o:o + m].cpu().numpy()
    arrays = {"units": rows, "status": st[rows], "out_len": ln[rows], "consumed_bits": used[rows], "output_units": picks}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float64))
    np.save(os.path.join(out_dir, "output.npy"), out)


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------- CPU legs (oracle)
def cpu_decode_throughput(units, seconds_budget, threads):
    """Times the CPU restatement of the reference (oracle/) on `threads` host threads over a bounded sample.  The threads are
    pthreads inside oracle/batch_mt.c pulling units from an atomic counter — no interpreter in the timed loop."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import swco
    swco.lib()
    sec, nbytes, fails = swco.batch_mt("deflate", units, max(2 * threads, 16), threads)      # calibration (also warms the pages)
    assert fails == 0
    per_unit = sec / max(2 * threads, 16)
    total = max(int(seconds_budget / per_unit), threads)
    sec, nbytes, fails = swco.batch_mt("deflate", units, total, threads)
    assert fails == 0 and nbytes == total * UNIT
    return nbytes / sec / 1e9, total, sec


def cgroup_cpu_limit():
    """CPUs the container may actually use (cgroup v2 cpu.max / v1 cfs quota), or None when unlimited / unknown."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        return None if q == "max" else float(q) / float(per)
    except Exception:
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else q / per
    except Exception:
        return None


def best_thread_count(units):
    """The box shows 128 logical CPUs but may schedule far fewer for this container (measured: linear to 16 threads, flat at
    32, slower at 128).  "All the host threads it can use" = the count with the highest measured throughput."""
    ncpu = os.cpu_count() or 1
    cands = sorted({max(1, ncpu >> k) for k in range(0, 5)} | {min(ncpu, 16), min(ncpu, 24), min(ncpu, 48)})
    sweep = {}
    for th in cands:
        v, _, _ = cpu_decode_throughput(units, 1.5, th)
        sweep[th] = v
    best = max(sweep, key=sweep.get)
    return best, {str(k): round(v, 4) for k, v in sweep.items()}


def physical_cores():
    try:
        pairs = set()
        phys = core = None
        for line in open("/proc/cpuinfo"):
            if line.startswith("physical id"):
                phys = line.split(":")[1].strip()
            elif line.startswith("core id"):
                core = line.split(":")[1].strip()
            elif not line.strip():
                if phys is not None and core is not None:
                    pairs.add((phys, core))
                phys = core = None
        return len(pairs) or None
    except Exception:
        return None


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    n_units = (args.units // min(args.distinct, args.units)) * min(args.distinct, args.units)
    units, _ = make_corpus(256)
    threads, sweep = best_thread_count(units)
    per_step = 6.0
    vals, n_total = [], 0
    for _ in range(args.steps):
        v, n, dt = cpu_decode_throughput(units, per_step, threads)
        vals.append(v); n_total += n
    value = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": workload_config(n_units, min(args.distinct, n_units), args.gpus),
        "cpu_baseline": {"value": value, "unit": "GB/s", "cores": threads, "logical_cpus": os.cpu_count(), "physical_cores": physical_cores(),
                         "cgroup_cpu_limit": cgroup_cpu_limit(), "thread_sweep_GBps": sweep, "kind": "port",
                         "sample": f"{n_total} units of 64 KiB (256 distinct, same generator/compressor as the GPU workload) in "
                                   f"{args.steps} steps of ~{per_step:.0f} s on {threads} pthreads (oracle/batch_mt.c)",
                         "note": "the Swift reference cannot be built here (no Swift toolchain); this arm times the C restatement of "
                                 "its algorithm (oracle/, bit-by-bit tree walk like DecodingTree.findNextSymbol) on all host threads"},
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_line(line)
    return 0


# --------------------------------------------------------------------------------------------- product arm
def run_product(args):
    import torch
    import torch.distributed as dist
    from swcompression_b200 import _lib
    from swcompression_b200.batch import Batch, pack_units

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    from swcompression_b200 import shard
    n_units = args.units
    distinct = min(args.distinct, n_units)
    tile = n_units // distinct
    n_units = tile * distinct
    nominal_units = n_units
    # Rank 0 owns the unit list (SURVEY §8e): it builds the corpus, the other ranks receive their shard over NCCL.
    units, crcs = make_corpus(distinct, seed0=2) if rank == 0 else (None, None)      # fork the generator pool BEFORE CUDA is initialised
    assert torch.cuda.is_available(), "bench.py product arm needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/nccl_%h_%p.log")     # NCCL's version / debug lines go to a file: stdout = the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()
    L.swc_timing_collect.argtypes = [C.c_void_p, C.c_int32]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    scatter_ms = 0.0
    if rank == 0:
        buf, offs, lens = pack_units(units)                   # 16-byte aligned unit starts: stride[i] = padded length
        strides = np.diff(np.concatenate([offs, [len(buf) - 64]])).astype(np.int64)
        d_one = torch.from_numpy(buf[:len(buf) - 64]).to(dev)
    if world == 1:
        d_in = torch.cat([d_one.repeat(tile), torch.zeros(64, dtype=torch.uint8, device=dev)])
        l_stride, l_len, begin = np.tile(strides, tile), np.tile(lens.astype(np.int64), tile), 0
        crc_t = torch.tensor(crcs, dtype=torch.int64, device=dev)
    else:
        # the whole job = world x n_units units, tiled from the distinct corpus on rank 0's GPU; byte-balanced contiguous
        # shards go out with one table broadcast + one NCCL send per rank (timed: scatter_ms)
        crc_t = torch.zeros(distinct, dtype=torch.int64, device=dev)
        g_buf = g_stride = g_len = None
        if rank == 0:
            crc_t = torch.tensor(crcs, dtype=torch.int64, device=dev)
            g_buf = d_one.repeat(tile * world)
            g_stride, g_len = np.tile(strides, tile * world), np.tile(lens.astype(np.int64), tile * world)
        dist.broadcast(crc_t, src=0)
        barrier()
        t0 = time.perf_counter()
        d_loc, l_stride, l_cap, (begin, end), l_len = shard.scatter_units(g_buf, g_stride, None if g_stride is None else np.full(len(g_stride), UNIT), dev, extra=g_len)
        barrier()
        scatter_ms = (time.perf_counter() - t0) * 1e3
        del g_buf
        d_in = torch.cat([d_loc, torch.zeros(64, dtype=torch.uint8, device=dev)])
        n_units = end - begin
    all_off = np.concatenate([[0], np.cumsum(l_stride)[:-1]]).astype(np.uint64)
    all_len = l_len.astype(np.uint64)
    b = Batch.__new__(Batch)
    Batch.__init__(b, "deflate", np.zeros(1, dtype=np.uint8), all_off, all_len, UNIT, device=str(dev))
    b.d_in = d_in
    total_in = int(all_len.sum())
    total_out = n_units * UNIT
    torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        b.run()
    barrier()
    # parity check of the workload itself (outside the timed region): the CRC-32 of EVERY decoded unit (device-side, batched
    # swc_crc32_batch) against the CRC-32 of the raw bytes it was compressed from; a sample against the oracle byte by byte
    st, ln, used = b.results()
    assert (st == 0).all() and (ln == UNIT).all(), "decode failed"
    d_crc = torch.zeros(n_units, dtype=torch.int32, device=dev)
    pp = lambda t: C.c_void_p(t.data_ptr())
    assert L.swc_crc32_batch(pp(b.d_out), pp(b.d_out_off), pp(b.d_out_len), pp(b.d_status), pp(d_crc), n_units,
                             C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)) == 0
    want = crc_t[(torch.arange(n_units, device=dev) + begin) % distinct]
    assert torch.equal(d_crc.to(torch.int64) & 0xFFFFFFFF, want), "a decoded unit has the wrong CRC-32"
    if rank == 0:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import swco
        host_out = b.d_out[: distinct * UNIT].cpu().numpy()
        for i in range(0, distinct, max(distinct // 16, 1)):
            ost, oout, oused = swco.deflate_decompress(units[i])
            assert ost == 0 and host_out[i * UNIT:(i + 1) * UNIT].tobytes() == oout and used[i] == oused, "parity vs oracle failed"

    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = L.swc_kernel_launches()
    L.swc_timing_enable(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        b.run()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    tbuf = (C.c_float * (args.steps * 5 + 8))()
    nint = L.swc_timing_collect(tbuf, len(tbuf))
    L.swc_timing_enable(0)
    launches = L.swc_kernel_launches() - launches0
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    ms_per_step = ms_max / args.steps
    job = torch.tensor([total_out, total_in], dtype=torch.float64, device=dev)     # whole job = the units ALL ranks decoded
    if world > 1:
        dist.all_reduce(job, op=dist.ReduceOp.SUM)
    value = float(job[0].item()) / (ms_per_step * 1e-3) / 1e9
    if args.dump_outputs and rank == 0:
        dump_outputs(b, args.dump_outputs)

    # ---- SURVEY §8e legs: decode-only / + gather to rank 0 / + all-gather, on a sub-batch whose gathered size fits every GPU ----
    legs = None
    if world > 1 and not args.no_legs:
        n_leg = min(n_units, args.leg_units)
        lb = Batch.__new__(Batch)
        Batch.__init__(lb, "deflate", np.zeros(1, dtype=np.uint8), all_off[:n_leg], all_len[:n_leg], UNIT, device=str(dev))
        lb.d_in = d_in
        leg_bytes = torch.tensor([n_leg * UNIT], dtype=torch.float64, device=dev)
        dist.all_reduce(leg_bytes, op=dist.ReduceOp.SUM)

        def timed(fn, reps=3):
            fn(); barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            barrier()
            tt = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(leg_bytes.item()) / (float(tt.item()) * 1e-3) / 1e9, float(tt.item())

        out_view = lambda: lb.d_out[: n_leg * UNIT]
        g0, t_0 = timed(lambda: lb.run())
        g1, t_1 = timed(lambda: (lb.run(), shard.gather_to_root(out_view())))
        g2, t_2 = timed(lambda: (lb.run(), shard.allgather(out_view())))
        legs = {"units_per_gpu": int(n_leg), "decode_only_GBps": g0, "decode_gather_to_root_GBps": g1, "decode_allgather_GBps": g2,
                "ms": {"decode_only": t_0, "decode_gather_to_root": t_1, "decode_allgather": t_2},
                "note": "whole-job decompressed GB/s over all ranks; gathers move decoded bytes over NCCL/NVLink (gather: grouped "
                        "send/recv to rank 0, all-gather: ncclAllGather); sub-batch sized so that world x shard fits one GPU"}
        del lb


    # per-kernel durations: 4 marks per step -> intervals [K1L table-lookup decode, slow path (no-op here), K2 record replay, gap]
    iv = np.array(list(tbuf)[:nint], dtype=np.float64)
    k1 = float(iv[0::4].mean()) if nint >= 3 else None
    ks = float(iv[1::4].mean()) if nint >= 3 else None
    k2 = float(iv[2::4].mean()) if nint >= 3 else None
    peak, peak_src = read_peaks()
    alg_bytes = total_in + total_out
    roof = None
    if k1:
        dom, dom_ms = ("inflate_lut_kernel", k1) if k1 >= k2 else ("lz_resolve_kernel", k2)
        achieved = alg_bytes / (dom_ms * 1e-3) / 1e9
        path = alg_bytes / ((k1 + ks + k2) * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                per_unit = json.load(open(tp)).get("bytes_per_unit", {}).get(dom)
                traffic = per_unit * n_units if per_unit else None
            except Exception:
                traffic = None
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "kernel": dom, "kernel_ms": dom_ms, "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                "kernels_ms": {"inflate_lut_kernel": k1, "inflate_slow_kernel(no-op)": ks, "lz_resolve_kernel": k2},
                "path_achieved": path, "path_frac": path / peak,
                "read_only_frac": total_in / ((k1 + ks + k2) * 1e-3) / 1e9 / peak,
                "write_only_frac": total_out / ((k1 + ks + k2) * 1e-3) / 1e9 / peak}

    # ---- end to end through the host-buffer C-ABI call (pinned host memory, H2D + D2H inside the timed region) ----
    e2e = None
    if not args.no_e2e:
        n_e = min(args.e2e_units, n_units)
        # every rank pins its own buffers: keep the job's pinned total under half of what the host (or its cgroup) can give
        n_e = max(2048, min(n_e, int(host_memory_budget() * 0.5 / world / (UNIT * 1.4))))
        if world > 1:                                                  # one figure for the whole job
            tn = torch.tensor([n_e], dtype=torch.int64, device=dev)
            dist.all_reduce(tn, op=dist.ReduceOp.MIN)
            n_e = int(tn.item())
        in_total = int(all_off[n_e - 1] + l_stride[n_e - 1]) + 64
        out_total = n_e * UNIT
        p_in = L.swc_alloc_pinned(in_total)
        p_out = L.swc_alloc_pinned(out_total)
        assert p_in and p_out, "pinned allocation failed"
        h_in = torch.from_numpy(np.ctypeslib.as_array(C.cast(p_in, C.POINTER(C.c_uint8)), shape=(in_total,)))
        h_in[: in_total - 64].copy_(d_in[: in_total - 64])            # the same compressed bytes, now in pinned HOST memory
        torch.cuda.synchronize(dev)
        e_off = np.ascontiguousarray(all_off[:n_e]); e_len = np.ascontiguousarray(all_len[:n_e])
        o_off = (np.arange(n_e, dtype=np.uint64) * np.uint64(UNIT)); o_cap = np.full(n_e, UNIT, dtype=np.uint64)
        r_len = np.zeros(n_e, dtype=np.uint64); r_used = np.zeros(n_e, dtype=np.uint64); r_st = np.zeros(n_e, dtype=np.int32)
        vp = lambda a: a.ctypes.data_as(C.c_void_p)

        def call():
            rc = L.swc_deflate_decompress_batch_host(C.c_void_p(p_in), vp(e_off), vp(e_len), in_total, C.c_void_p(p_out), vp(o_off), vp(o_cap),
                                                     out_total, vp(r_len), vp(r_used), vp(r_st), n_e)
            assert rc == 0, _lib.status_name(rc)

        call()
        assert (r_st == 0).all() and (r_len == UNIT).all()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            call()
        torch.cuda.synchronize(dev)
        dt = (time.perf_counter() - t0) / args.e2e_steps
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": out_total * world / float(tt.item()) / 1e9, "unit": "GB/s",
               "h2d_bytes_per_step": int(in_total + n_e * 8 * 4), "d2h_bytes_per_step": int(out_total + n_e * 20),
               "units_per_step": int(n_e), "ms_per_step": float(tt.item()) * 1e3,
               "api": "swc_deflate_decompress_batch_host (pinned host buffers; per call: H2D + K1/K2 + D2H, up to 32 slices of >= 2048 units pipelined over 3 streams)"}
        L.swc_free_pinned(C.c_void_p(p_in)); L.swc_free_pinned(C.c_void_p(p_out))

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cores, sweep = best_thread_count(units[:256])
        v1, n1, dt1 = cpu_decode_throughput(units[:256], 4.0, 1)
        vN, nN, dtN = cpu_decode_throughput(units[:256], 10.0, cores)
        cpu = {"value": vN, "unit": "GB/s", "cores": cores, "logical_cpus": os.cpu_count(), "physical_cores": physical_cores(),
               "cgroup_cpu_limit": cgroup_cpu_limit(), "thread_sweep_GBps": sweep, "kind": "port",
               "sample": f"{nN} units of 64 KiB (same generator/compressor as the GPU workload) in {dtN:.1f} s on {cores} pthreads "
                         f"(oracle/batch_mt.c, no interpreter in the loop)",
               "single_thread_value": v1, "thread_scaling": vN / v1 if v1 else None,
               "note": "C restatement of the Swift reference's algorithm (oracle/); the Swift reference itself cannot be built here"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": workload_config(nominal_units, distinct, world),
            "compressed_bytes_per_gpu": total_in, "units_this_rank": int(n_units),
            "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "multi_gpu": None if world == 1 else {"unit_list_owner": "rank 0", "scatter_ms": scatter_ms,
                                                  "partition": "contiguous ranges balanced by compressed+decompressed bytes (shard.partition)",
                                                  "legs": legs},
        }
        emit_line(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


_REAL_STDOUT = None


def guard_stdout():
    """stdout carries exactly ONE JSON line: everything else that libraries write to fd 1 (NCCL prints its version line there
    when NCCL_DEBUG is set in the environment, whatever NCCL_DEBUG_FILE says) is sent to stderr."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit_line(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    guard_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="product", choices=["product", "reference"])
    ap.add_argument("--units", type=int, default=N_UNITS)
    ap.add_argument("--distinct", type=int, default=DISTINCT)
    ap.add_argument("--e2e-units", type=int, default=N_UNITS)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-legs", action="store_true")
    ap.add_argument("--leg-units", type=int, default=32768)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned as DIR/*.npy "
                                                          "(product arm, rank 0's units; see dump_outputs)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_product(args)


if __name__ == "__main__":
    sys.exit(main())
