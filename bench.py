#!/usr/bin/env python
"""Benchmark of the .spz per-gaussian codec hot path (BASELINE.json: encode/decode Mgaussians/s and
HBM GB/s vs roofline at 1/2/4/8 B200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--points P] [--sh-degree D] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference's own CPU pack/unpack on the host cores

Workload (config 5 of BASELINE.json; it fits one GPU, so it is also the N=1 workload): ONE synthetic
100M-gaussian SH-degree-3 cloud (counter-seeded: every float is a function of the seed and its global
index), v3 stream, sharded by contiguous point range over the N ranks -- rank r generates and owns
gaussians [a_r, b_r) of that cloud (strong scaling; no collective on the data path).  One "step" =
encode the rank's shard (float planes -> byte planes), then decode the result back (byte planes ->
float planes, with a coordinate flip folded in).

  value     gaussians through that encode+decode round trip per second, whole job, inputs resident in
            HBM, timed with CUDA events on the launching stream, max over ranks.
  parity    outside the timed region: sampled 64k-point blocks of every rank's encode and decode output
            against the CPU checker (oracle/), and order-sensitive hashes of ALL output planes that add up
            over the shards -- the same two numbers must come out for every N.
  e2e       the same step through the host-pointer C-ABI (spzb200_encode_host / spzb200_decode_host:
            pinned host planes in and out, H2D and D2H inside the timed region), issued full duplex --
            step i's encode and the decode of step i-1's stream run concurrently from two host threads
            so both directions of the PCIe link are busy; the one-thread figure is e2e.sequential.
            e2e.link_ceiling_gbs is the bare link measured in the same run by the same processes (plain
            pinned cudaMemcpyAsync, all ranks at once); e2e.frac_of_link = achieved / that ceiling.
  e2e_multi (N > 1) rank 0 alone drives all N GPUs through spzb200_encode_host_multi /
            spzb200_decode_host_multi on the whole cloud in pinned host memory -- the library's own
            multi-GPU entry point; its planes must hash to the parity hashes.

The working set (30.1 GB per step at N=1) is far larger than the 126 MB L2, so no explicit flush is
needed between iterations.

The oracle / reference build under oracle/ is used here ONLY as the checker of `parity` and as the
timed CPU baseline (`cpu_baseline`, `--impl reference`), never on the measured GPU path.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "encode+decode Mgaussians/s (v3, SH3)"
UNIT = "Mgaussians/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--points", type=int, default=100_000_000, help="gaussians in the whole cloud")
    ap.add_argument("--sh-degree", type=int, default=3)
    ap.add_argument("--from-coord", type=int, default=6, help="PackOptions.from (6 = RDF)")
    ap.add_argument("--to-coord", type=int, default=6, help="UnpackOptions.to (6 = RDF)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-chunk-sweep", default="", help="comma-separated pipeline range sizes (points) to re-time the duplex e2e step with")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ply", action="store_true", help="skip the fused PLY-rows kernel timings (N=1 only)")
    ap.add_argument("--cpu-sample-points", type=int, default=0, help="0 = auto")
    ap.add_argument("--traffic-bytes", type=float, default=None,
                    help="dram bytes per launch of the dominant kernel from an ncu --set full capture")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of the last step's encoded and decoded planes to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the B200 arm computed; the reference arm has no outputs to dump")
    return args


def workload_name(n, deg):
    return f"synthetic {n / 1e6:g}M gaussians SH degree {deg} v3 encode+decode, sharded by point range"


# -------------------------------------------------------------------------------------------------
# clocks: NVML sampled from a thread during the timed region
# -------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.005)

    def start(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join()
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# -------------------------------------------------------------------------------------------------
# the reference's CPU implementation, timed (cpu_baseline and --impl reference)
# -------------------------------------------------------------------------------------------------
def cpu_reference_run(points_total, deg, frm, to, steps, warmup, threads, sample_points, best=False):
    """Times encode+decode of a bounded sample of the workload with the reference's own code
    (oracle/_ref/libspz_ref.so = the unmodified C++ compiled in place) or, if that build is not
    present, the C restatement (oracle/_build/libspz_oracle.so).  `threads` independent point
    ranges run concurrently (the reference itself is single-threaded; points are independent)."""
    from concurrent.futures import ThreadPoolExecutor

    import numpy as np

    import oracle as O
    from spz_b200.synth import numpy_cloud

    kind = "reference"
    try:
        impl_factory = O.Ref
        impl_factory()
    except Exception:  # noqa: BLE001
        kind = "port"
        impl_factory = O.Oracle
    per_thread = max(1, sample_points // threads)
    clouds = []
    for t in range(threads):
        c = numpy_cloud(per_thread, deg, seed=1000 + t)
        clouds.append(O.Cloud(per_thread, deg, *c.planes()))
    impls = [impl_factory() for _ in range(threads)]

    def one(i):
        p = impls[i].pack(clouds[i], frm)
        t_pack = impls[i].last_seconds
        g = impls[i].unpack(p, to)
        t_unpack = impls[i].last_seconds
        return t_pack, t_unpack, int(g.n)

    times, inner = [], []
    with ThreadPoolExecutor(threads) as ex:
        for s in range(warmup + steps):
            t0 = time.perf_counter()
            res = list(ex.map(one, range(threads)))
            dt = time.perf_counter() - t0
            if s >= warmup:
                times.append(dt)
                inner.append(res)
    n_step = per_thread * threads
    if best:  # best of `steps` (BASELINE.md section 4), judged on the time inside the two functions
        k = min(range(len(times)), key=lambda i: sum(max(r[j] for r in inner[i]) for j in (0, 1)) if inner[i][0][0] is not None else times[i])
        times, inner = [times[k]], [inner[k]]
    mean = sum(times) / len(times)
    out = {"value": n_step / mean / 1e6, "unit": UNIT, "cores": threads, "kind": kind,
           "sample": f"{n_step} gaussians per step ({threads} x {per_thread}-point ranges of the synthetic SH{deg} "
                     f"workload), {'best of ' if best else ''}{steps} steps; wall time of pack+unpack calls incl. marshalling copies",
           "ms_per_step": mean * 1e3}
    if kind == "reference" and inner and inner[0][0][0] is not None:
        # time inside packGaussians / unpackGaussians alone (marshalling excluded), slowest thread
        pk = statistics.mean(max(r[0] for r in step) for step in inner)
        up = statistics.mean(max(r[1] for r in step) for step in inner)
        out["pack_mgs"] = n_step / pk / 1e6
        out["unpack_mgs"] = n_step / up / 1e6
        out["value"] = n_step / (pk + up) / 1e6
        out["ms_per_step"] = (pk + up) * 1e3
        out["sample"] += "; value = time inside packGaussians+unpackGaussians only"
    return out


def traffic_for(kernel, gaussians, override):
    """(DRAM bytes per launch of `kernel`, how that figure was obtained).  Not a measurement of this run: the
    ncu --set full capture recorded in profiles/traffic.json was taken at another launch size and is scaled
    per gaussian to this launch; --traffic-bytes passes a capture of this very configuration instead."""
    if override is not None:
        return override, "ncu_capture_passed_on_the_command_line"
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[kernel]
        return t["dram_bytes"] / t["gaussians"] * gaussians, f"scaled_from_ncu_{t['gaussians'] // 1000000}M"
    except Exception:  # noqa: BLE001
        return None, None


def ply_rows_kernels(ctx, codec, dev, deg, n=40_000_000, steps=8):
    """SURVEY.md 8f-3: the fused kernels on the other side of the codec, .ply vertex records <-> packed
    planes (canonical property order), device-resident, CUDA events, median of `steps`."""
    import torch
    names = codec.ply_property_names(deg)
    w = len(names)
    rows = torch.empty(n * w, dtype=torch.float32, device=dev).uniform_(-1, 1)
    out = codec.alloc_packed(n, deg, 3, device=dev)
    back = torch.empty_like(rows)
    per = 4 * w + codec.packed_bytes_per_gaussian(deg)
    res = {"points": n, "sh_degree": deg, "bytes_per_gaussian": per,
           "note": "packGaussians(loadSplatFromPly(...)) / saveSplatToPly(unpackGaussians(...)) row layout in one kernel each; "
                   "not part of `value`"}
    for key, fn in (("rows_to_packed", lambda: ctx.encode_ply_device(rows, n, names, deg, 6, out=out)),
                    ("packed_to_rows", lambda: ctx.decode_ply_device(out, names, 6, out=back))):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(steps):
            e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            e[0].record()
            fn()
            e[1].record()
            torch.cuda.synchronize()
            ts.append(e[0].elapsed_time(e[1]))
        ms = statistics.median(ts)
        res[key] = {"ms": ms, "hbm_gbs": per * n / ms / 1e6, "mgaussians_s": n / ms / 1e3}
    return res


def small_cloud_latency(ctx, codec, torch_cloud, dev, n, deg, args):
    import torch
    c = torch_cloud(n, deg, dev, seed=60)
    p = codec.alloc_packed(n, deg, 3, device=dev)
    g = codec.alloc_cloud(n, deg, device=dev)
    dev_us, host_us = [], []
    for i in range(60):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        e[0].record()
        ctx.encode_device(c, args.from_coord, out=p)
        ctx.decode_device(p, args.to_coord, out=g)
        e[1].record()
        torch.cuda.synchronize()
        if i >= 10:
            dev_us.append(e[0].elapsed_time(e[1]) * 1e3)
    # the same pair captured once in a CUDA graph and replayed: what a consumer that decodes every frame would do, and
    # the kernels' own latency without the Python -> ctypes launch path (~10-20 us per call)
    graph_us = None
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            ctx.encode_device(c, args.from_coord, out=p)
            ctx.decode_device(p, args.to_coord, out=g)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            ctx.encode_device(c, args.from_coord, out=p)
            ctx.decode_device(p, args.to_coord, out=g)
        ts = []
        for i in range(60):
            e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            e[0].record()
            graph.replay()
            e[1].record()
            torch.cuda.synchronize()
            if i >= 10:
                ts.append(e[0].elapsed_time(e[1]) * 1e3)
        graph_us = statistics.median(ts)
        del graph
    except Exception as ex:  # noqa: BLE001 -- an optional extra; the bench line does not depend on it
        graph_us = f"unavailable: {ex!r}"[:200]
    hc = codec.alloc_cloud(n, deg, pinned=True, numpy_arrays=True)
    hp = codec.alloc_packed(n, deg, 3, pinned=True, numpy_arrays=True)
    hb = codec.alloc_cloud(n, deg, pinned=True, numpy_arrays=True)
    for src, dst in zip(c.planes(), hc.planes()):
        if dst.size:
            torch.from_numpy(dst).copy_(src)
    torch.cuda.synchronize()
    for i in range(60):
        t0 = time.perf_counter()
        ctx.encode_host(hc, args.from_coord, out=hp)
        ctx.decode_host(hp, args.to_coord, out=hb)
        if i >= 10:
            host_us.append((time.perf_counter() - t0) * 1e6)
    return {"points": n, "sh_degree": deg, "device_encode_plus_decode_us": statistics.median(dev_us),
            "device_encode_plus_decode_cuda_graph_us": graph_us,
            "host_api_encode_plus_decode_us": statistics.median(host_us),
            "note": "median of 50; device = two launches (encode, decode; the sub-tile remainder rides in each) on resident planes, issued from Python through ctypes, so it is launch-bound, not bandwidth-bound (the data moves in ~6 us); cuda_graph = the same two launches captured once and replayed (no host launch path); host = spzb200_encode_host + spzb200_decode_host with pinned planes, i.e. 18 MB over PCIe each way"}


def time_host_zlib(packed, deg, sample_points):
    """gzip stays on the host (north star) and is reported apart from the codec: deflate / inflate of
    the container bytes of the first `sample_points` encoded gaussians with the reference's zlib
    parameters (default level, gzip wrapper, memLevel 9; load-spz.cc:186-214), one thread."""
    import struct
    import zlib

    from spz_b200 import codec
    widths = codec.byte_plane_widths(deg, 3)
    planes = [p[:w * sample_points].cpu().numpy().tobytes() for p, w in zip(packed.planes(), widths)]
    order = [planes[0], planes[3], planes[4], planes[1], planes[2], planes[5]]  # stream order
    stream = struct.pack("<IIIBBBB", 0x5053474e, 3, sample_points, deg, 12, 0, 0) + b"".join(order)
    threads = host_threads()
    t0 = time.perf_counter()
    gz = codec.gzip_bytes(stream, 1)          # the reference's single-thread zlib stream, byte for byte
    t1 = time.perf_counter()
    back = codec.gunzip_bytes(gz, 1)
    t2 = time.perf_counter()
    gzp = codec.gzip_bytes(stream, threads)   # block-parallel zlib, one standard gzip member
    t3 = time.perf_counter()
    backp = codec.gunzip_bytes(gzp, threads)
    t4 = time.perf_counter()
    assert back == stream and backp == stream and zlib.decompress(gzp, 16 + zlib.MAX_WBITS) == stream
    mg = lambda dt: sample_points / dt / 1e6  # noqa: E731
    return {"sample": f"container of the first {sample_points} encoded gaussians ({len(stream)} bytes), zlib {zlib.ZLIB_RUNTIME_VERSION}",
            "reference_1_thread": {"deflate_mb_s": len(stream) / (t1 - t0) / 1e6, "inflate_mb_s": len(stream) / (t2 - t1) / 1e6,
                                   "deflate_mgaussians_s": mg(t1 - t0), "inflate_mgaussians_s": mg(t2 - t1), "ratio": len(gz) / len(stream)},
            "block_parallel": {"threads": threads, "deflate_mb_s": len(stream) / (t3 - t2) / 1e6, "inflate_mb_s": len(stream) / (t4 - t3) / 1e6,
                               "deflate_mgaussians_s": mg(t3 - t2), "inflate_mgaussians_s": mg(t4 - t3), "ratio": len(gzp) / len(stream)}}


def host_memory_available():
    """min(MemAvailable, cgroup limit - usage) in bytes, or None."""
    vals = []
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable:"):
                vals.append(int(ln.split()[1]) * 1024)
    except OSError:
        pass
    try:
        mx = open("/sys/fs/cgroup/memory.max").read().strip()
        if mx != "max":
            vals.append(int(mx) - int(open("/sys/fs/cgroup/memory.current").read()))
    except (OSError, ValueError):
        pass
    return min(vals) if vals else None


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        return os.cpu_count() or 1


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = max(1, min(host_threads(), 32))
    sample = args.cpu_sample_points or threads * 250_000
    r = cpu_reference_run(args.points, args.sh_degree, args.from_coord, args.to_coord, args.steps, args.warmup, threads, sample)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32->u8", "data": "synthetic",
            "config": bench_config(args, max(1, args.gpus)),
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    for k in ("pack_mgs", "unpack_mgs"):
        if k in r:
            line[k] = r[k]
    print(json.dumps(line), flush=True)
    return 0


# -------------------------------------------------------------------------------------------------
# multi-rank plumbing (no data-path collective: only the barrier and these scalar reductions)
# -------------------------------------------------------------------------------------------------
def reduce_scalar(dist, x, op, device):
    """max / sum of a python scalar over all ranks; identity when not distributed."""
    if dist is None:
        return x
    import torch
    t = torch.tensor([float(x)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
    return t.item()


def allsum_u64(dist, x, device):
    """sum mod 2^64 of one unsigned 64-bit value per rank (the shard hashes); identity when not distributed."""
    if dist is None:
        return x
    import torch
    t = torch.tensor([x - (1 << 64) if x >= (1 << 63) else x], dtype=torch.int64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return int(t.item()) & 0xFFFFFFFFFFFFFFFF


def rank_shard(points_total, sh_degree, world, rank):
    """[a, b) of this rank: contiguous point range with tile-aligned boundaries (spzb200_shard_range)."""
    from spz_b200 import codec
    return codec.shard_range(points_total, sh_degree, world, rank)


# -------------------------------------------------------------------------------------------------
# parity inside the bench (outside every timed region): sampled blocks against the oracle, and
# order-sensitive 64-bit hashes of whole planes that add up across shards
# -------------------------------------------------------------------------------------------------
_HASH_C1 = -7046029254386353131   # 0x9E3779B97F4A7C15 as int64
_HASH_C2 = -4658895280553007687   # 0xBF58476D1CE4E5B9 as int64


def plane_hash(t, global_byte_offset, salt, dev):
    """sum over 8-byte words w_i (global word index i) of mix(w_i, i) mod 2^64.  Additive over contiguous
    shards (every shard boundary is a multiple of 8 bytes in every plane), sensitive to any changed or
    moved word.  `t`: device tensor or host numpy array; hashed on `dev` in bounded slices."""
    import numpy as np
    import torch
    assert global_byte_offset % 8 == 0
    flat = t.view(np.uint8).reshape(-1) if isinstance(t, np.ndarray) else t.view(torch.uint8).reshape(-1)
    n = flat.shape[0]
    total = 0
    step = 1 << 29  # bytes per slice
    for s in range(0, n, step):
        e = min(n, s + step)
        chunk = flat[s:e]
        if isinstance(chunk, np.ndarray):
            chunk = torch.from_numpy(chunk).to(dev, non_blocking=False)
        if (e - s) % 8:
            chunk = torch.cat([chunk, torch.zeros(8 - (e - s) % 8, dtype=torch.uint8, device=dev)])
        w = chunk.view(torch.int64)
        i = torch.arange(w.numel(), dtype=torch.int64, device=dev) + ((global_byte_offset + s) // 8 + salt * 0x100000001B3)
        x = (w ^ (i * _HASH_C1)) * _HASH_C2
        x = x ^ (x >> 29)
        total = (total + int(x.sum().item())) & 0xFFFFFFFFFFFFFFFF
        del w, i, x, chunk
    return total


def planes_hash(planes, widths_bytes, a, dev):
    """hash of a set of planes holding gaussians [a, a + n) of the whole cloud"""
    h = 0
    for k, (t, wb) in enumerate(zip(planes, widths_bytes)):
        size = t.size if hasattr(t, "size") and not callable(t.size) else t.numel()
        if size:
            h = (h + plane_hash(t, a * wb, k + 1, dev)) & 0xFFFFFFFFFFFFFFFF
    return h


def oracle_block_parity(cloud, packed, decoded, n, deg, frm, to, rank, blocks=6, block_points=65536):
    """Sampled blocks of this rank's shard: the device-resident encoder / decoder outputs against the CPU
    checker (the unmodified reference compiled in place where its build is present, else the C restatement),
    byte for byte and float bit for float bit.  Returns (blocks checked, blocks equal, checker kind)."""
    import numpy as np

    import oracle as O
    from spz_b200 import codec
    try:
        checker, kind = O.Ref(), "reference"
    except Exception:  # noqa: BLE001
        checker, kind = O.Oracle(), "port"
    tg = codec.tile_gaussians(deg)
    bp = min(block_points, n)
    rng = np.random.default_rng(1234 + rank)
    starts = {0, max(0, n - bp)}  # the first block and the last one (which holds the sub-tile remainder)
    while len(starts) < min(blocks, max(1, n // max(bp, 1))):
        starts.add(int(rng.integers(0, max(1, (n - bp) // tg + 1))) * tg)
    fw, bw = codec.float_plane_widths(deg), codec.byte_plane_widths(deg, 3)
    ok = 0
    for s0 in sorted(starts):
        src = [t[s0 * w:(s0 + bp) * w].cpu().numpy() for t, w in zip(cloud.planes(), fw)]
        want = checker.pack(O.Cloud(bp, deg, *src), frm)
        same = all(np.array_equal(t[s0 * w:(s0 + bp) * w].cpu().numpy(), e) for t, w, e in zip(packed.planes(), bw, want.planes()))
        back = checker.unpack(want, to)
        same = same and all(np.array_equal(O.bits(t[s0 * w:(s0 + bp) * w].cpu().numpy()), O.bits(e))
                            for t, w, e in zip(decoded.planes(), fw, back.planes()))
        ok += int(same)
    return len(starts), ok, kind


DUMP_POINTS = 65536  # 32.5 MB of .npy files at SH degree 3


def dump_outputs(out_dir, packed, decoded, n_total, deg, a, b, rank, world):
    """What encode_device and decode_device returned in the last timed step, for gaussians drawn from the whole
    cloud with a fixed seed (so every build and every N dumps the same ones): `encoded_<plane>.npy` holds the byte
    planes and `decoded_<plane>.npy` the float planes, both float32 with one row per gaussian, and `indices.npy`
    (float64) the global index of each row.  With N > 1 ranks each writes the rows of its shard, as
    `<name>.rank<r>.npy`."""
    import numpy as np
    import torch

    from spz_b200 import codec
    idx = np.sort(np.random.default_rng(0).choice(n_total, size=min(n_total, DUMP_POINTS), replace=False))
    idx = idx[(idx >= a) & (idx < b)]
    rows = torch.from_numpy(idx - a).to(packed.positions.device)
    arrays = {"indices": idx.astype(np.float64)}
    for kind, planes, widths in (("encoded", packed.planes(), codec.byte_plane_widths(deg, 3)),
                                 ("decoded", decoded.planes(), codec.float_plane_widths(deg))):
        for name, t, w in zip(codec.PLANES, planes, widths):
            arrays[f"{kind}_{name}"] = (t.view(-1, w)[rows].to(torch.float32).cpu().numpy() if w
                                        else np.zeros((idx.size, 0), np.float32))
    os.makedirs(out_dir, exist_ok=True)
    suffix = "" if world == 1 else f".rank{rank}"
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), arr)


def link_ceiling(dev, barrier, seconds=1.0, mb=1024):
    """Bare host<->device link of this rank while every other rank does the same: plain pinned
    cudaMemcpyAsync (torch copy_ on pinned tensors), nothing of the codec.  H2D alone, D2H alone, both at
    once; GB/s of this rank per phase and direction (scripts/link_probe.py is the standalone form).  Each
    phase is run in two shapes -- one stream per direction with 256 MiB pieces, and three streams per
    direction with 64 MiB pieces (the shape of the codec's own pipeline) -- and the better one counts: on
    some boxes the single-stream shape leaves 10 % of a contended link unused, and a ceiling must not
    be something the measured path can beat."""
    import torch
    nbytes = mb << 20
    host_in = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    host_out = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    host_in.fill_(1)
    d_in = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    d_out = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
    streams = [[torch.cuda.Stream(dev) for _ in range(3)] for _ in range(2)]

    def loop(secs, h2d, d2h, nstreams, chunk):
        torch.cuda.synchronize(dev)
        moved = 0
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < secs:
            for k, a in enumerate(range(0, nbytes, chunk)):
                if h2d:
                    with torch.cuda.stream(streams[0][k % nstreams]):
                        d_in[a:a + chunk].copy_(host_in[a:a + chunk], non_blocking=True)
                if d2h:
                    with torch.cuda.stream(streams[1][k % nstreams]):
                        host_out[a:a + chunk].copy_(d_out[a:a + chunk], non_blocking=True)
            for group in streams:
                for st in group:
                    st.synchronize()
            moved += nbytes
        return moved / (time.perf_counter() - t0) / 1e9

    loop(0.2, True, True, 1, 256 << 20)
    out = {}
    for name, h2d, d2h in (("h2d_alone", True, False), ("d2h_alone", False, True), ("duplex", True, True)):
        best = 0.0
        for nstreams, chunk in ((1, 256 << 20), (3, 64 << 20)):
            barrier()
            best = max(best, loop(seconds * 0.6, h2d, d2h, nstreams, chunk))  # each direction moves `moved` bytes: GB/s per direction
        out[name] = best
    barrier()
    del host_in, host_out, d_in, d_out
    return out


def shard_range_py(n, sh_degree, num_shards, index):
    """spzb200_shard_range restated in Python (whole tiles dealt out evenly, the remainder on the last shard), so the
    reference arm can describe the workload without loading this repo's library; tests/test_multirank_host_logic.py
    checks it against the C-ABI."""
    g = 6400 if sh_degree == 1 else 1280
    tiles = n // g
    a = tiles * index // num_shards * g
    b = n if index == num_shards - 1 else tiles * (index + 1) // num_shards * g
    return a, b


def bench_config(args, world):
    """The `config` object of the JSON line; identical for the B200 arm and the reference arm."""
    n_total, deg = args.points, args.sh_degree
    a0, b0 = shard_range_py(n_total, deg, world, 0)
    return {"workload": workload_name(n_total, deg), "points_total": n_total, "points_per_gpu": b0 - a0,
            "sh_degree": deg, "stream_version": 3, "from": args.from_coord, "to": args.to_coord,
            "l2": "working set per step >> 126 MB L2, no flush needed", "sharding": f"point-range x{world}, no collective",
            "data": "one counter-seeded cloud (seed 1); rank r holds slice [a_r, b_r) of it"}


# -------------------------------------------------------------------------------------------------
# the B200 arm
# -------------------------------------------------------------------------------------------------
def run_b200_arm(args):
    import numpy as np
    import torch

    from spz_b200 import codec
    from spz_b200.synth import counter_cloud_torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the codec has no CPU path (use --impl reference for the CPU arm)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py: --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import datetime

        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(minutes=20))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    deg, n_total = args.sh_degree, args.points
    a, b = rank_shard(n_total, deg, world, rank)
    n = b - a
    ctx = codec.Context(local)
    dev = torch.device("cuda", local)
    # ONE cloud for every N: rank r generates gaussians [a_r, b_r) of it (counter-based, SURVEY.md 8d)
    cloud = counter_cloud_torch(n_total, deg, dev, a, b, seed=1)
    packed = codec.alloc_packed(n, deg, 3, device=dev)
    decoded = codec.alloc_cloud(n, deg, device=dev)
    alg_bytes = codec.algorithmic_bytes_per_gaussian(deg, 3)
    fwb = [4 * w for w in codec.float_plane_widths(deg)]
    bwb = list(codec.byte_plane_widths(deg, 3))

    def step(evs=None):
        if evs:
            evs[0].record()
        ctx.encode_device(cloud, args.from_coord, out=packed)
        if evs:
            evs[1].record()
        ctx.decode_device(packed, args.to_coord, out=decoded)
        if evs:
            evs[2].record()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    launches0 = ctx.info()["kernel_launches"]
    sampler = ClockSampler(local)
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    barrier()
    e0.record()
    for s in range(args.steps):
        step(evs[s])
    e1.record()
    barrier()
    clocks = sampler.stop()
    total_ms = e0.elapsed_time(e1)
    launches = ctx.info()["kernel_launches"] - launches0
    enc_ms = statistics.mean(ev[0].elapsed_time(ev[1]) for ev in evs)
    dec_ms = statistics.mean(ev[1].elapsed_time(ev[2]) for ev in evs)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, packed, decoded, n_total, deg, a, b, rank, world)

    # ---- parity of what was just timed (outside the timed region) ---------------------------------
    # (1) sampled 64k-point blocks of this rank's shard against the CPU checker; (2) order-sensitive
    # hashes of every output plane, which add up over the shards: the all-reduced value is a function
    # of the cloud alone, so the lines of N = 1, 2, 4, 8 must print the same two numbers.
    par_blocks, par_ok, par_kind = oracle_block_parity(cloud, packed, decoded, n, deg, args.from_coord, args.to_coord, rank)
    enc_hash_local = planes_hash(packed.planes(), bwb, a, dev)
    dec_hash_local = planes_hash(decoded.planes(), fwb, a, dev)

    enc_hash, dec_hash = allsum_u64(dist, enc_hash_local, dev), allsum_u64(dist, dec_hash_local, dev)

    # ---- the bare link, every rank at once: the ceiling e2e is measured against ---------------------
    link = None
    if not args.no_e2e:
        link = link_ceiling(dev, barrier)

    # ---- e2e: the same step through the host-pointer C-ABI with pinned host planes ---------------
    e2e = None
    need = 2 * codec.float_bytes_per_gaussian(deg) * n + 2 * codec.packed_bytes_per_gaussian(deg) * n
    avail = host_memory_available()
    if not args.no_e2e and avail is not None and need * world > 0.6 * avail:
        raise SystemExit(f"bench.py: e2e needs {need * world / 1e9:.1f} GB of pinned host memory, only {avail / 1e9:.1f} GB "
                         "available; rerun with --no-e2e or fewer --points")
    if not args.no_e2e:
        del decoded
        torch.cuda.empty_cache()
        h_cloud = codec.alloc_cloud(n, deg, pinned=True, numpy_arrays=True)
        h_packed = codec.alloc_packed(n, deg, 3, pinned=True, numpy_arrays=True)
        h_back = codec.alloc_cloud(n, deg, pinned=True, numpy_arrays=True)
        for src, dst in zip(cloud.planes(), h_cloud.planes()):
            if dst.size:
                torch.from_numpy(dst).copy_(src)
        torch.cuda.synchronize()
        phases = []

        def e2e_step():
            _, t_enc = ctx.encode_host(h_cloud, args.from_coord, out=h_packed)
            _, t_dec = ctx.decode_host(h_packed, args.to_coord, out=h_back)
            return t_enc, t_dec

        e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            phases.append(e2e_step())
        barrier()
        e2e_s = (time.perf_counter() - t0) / args.e2e_steps
        h2d = phases[-1][0]["h2d_bytes"] + phases[-1][1]["h2d_bytes"]
        d2h = phases[-1][0]["d2h_bytes"] + phases[-1][1]["d2h_bytes"]
        e2e = {"s": e2e_s, "h2d": h2d, "d2h": d2h,
               "enc": {k: statistics.mean(p[0][k] for p in phases) for k in ("h2d_ms", "kernel_ms", "d2h_ms", "wall_ms")},
               "dec": {k: statistics.mean(p[1][k] for p in phases) for k in ("h2d_ms", "kernel_ms", "d2h_ms", "wall_ms")}}

        # Full-duplex form of the same step: a second host thread (own context) decodes the stream
        # the previous step produced while this step's cloud is being encoded, so both directions of
        # the PCIe link carry a step's worth of planes at once.  Same calls, same bytes per step.
        from concurrent.futures import ThreadPoolExecutor
        ctx2 = codec.Context(local)
        h_packed2 = codec.alloc_packed(n, deg, 3, pinned=True, numpy_arrays=True)
        streams = [h_packed, h_packed2]
        ctx.encode_host(h_cloud, args.from_coord, out=streams[1])  # step 0 decodes this one
        pool = ThreadPoolExecutor(2)

        def duplex_step(i):
            fa = pool.submit(ctx.encode_host, h_cloud, args.from_coord, streams[i % 2])
            fb = pool.submit(ctx2.decode_host, streams[(i + 1) % 2], args.to_coord, h_back)
            return fa.result()[1], fb.result()[1]

        def measure_duplex(steps):
            duplex_step(0)
            barrier()
            t0 = time.perf_counter()
            ph = [duplex_step(1 + i) for i in range(steps)]
            barrier()
            return (time.perf_counter() - t0) / steps, ph

        e2e["duplex_s"], dphases = measure_duplex(args.e2e_steps)
        e2e["duplex_enc_wall_ms"] = statistics.mean(p[0]["wall_ms"] for p in dphases)
        e2e["duplex_dec_wall_ms"] = statistics.mean(p[1]["wall_ms"] for p in dphases)
        e2e["chunk_sweep"] = None
        if args.e2e_chunk_sweep:  # development: the same duplex step with other pipeline range sizes (all ranks together)
            e2e["chunk_sweep"] = []
            for pts in [int(x) for x in args.e2e_chunk_sweep.split(",")]:
                ctx.set_chunk_points(pts)
                ctx2.set_chunk_points(pts)
                s_step, _ = measure_duplex(2)
                e2e["chunk_sweep"].append({"chunk_points": pts, "s": s_step})
            ctx.set_chunk_points(0)
            ctx2.set_chunk_points(0)
            measure_duplex(1)  # the planes hashed below come from the default configuration again
        pool.shutdown()
        ctx2.close()
        # what the e2e path produced, whole planes, against what the device-resident path produced
        e2e["hash_ok"] = (planes_hash(h_packed.planes(), bwb, a, dev) == enc_hash_local and
                          planes_hash(h_packed2.planes(), bwb, a, dev) == enc_hash_local and
                          planes_hash(h_back.planes(), fwb, a, dev) == dec_hash_local)
        if not e2e["hash_ok"]:
            raise SystemExit("bench.py: the host-pointer (e2e) path produced different planes than the device-resident path")
        del h_cloud, h_packed, h_packed2, h_back, streams

    # ---- e2e_multi: the library's own multi-GPU entry point, one process driving all N GPUs -------
    # rank 0 holds the WHOLE cloud in pinned host memory and calls spzb200_encode_host_multi /
    # spzb200_decode_host_multi over devices 0..N-1 (what spz::packGaussians does under
    # SPZ_B200_DEVICES); the other ranks idle at the barrier.  Its planes must hash to the same values.
    e2e_multi = None
    if not args.no_e2e and world > 1:
        barrier()
        if rank == 0:
            need_multi = 2 * (codec.float_bytes_per_gaussian(deg) + codec.packed_bytes_per_gaussian(deg)) * n_total
            avail = host_memory_available()
            if avail is not None and need_multi > 0.7 * avail:
                e2e_multi = {"skipped": f"needs {need_multi / 1e9:.1f} GB of pinned host memory for the whole cloud, {avail / 1e9:.1f} GB available"}
            else:
                e2e_multi = run_e2e_multi(args, codec, dev, world, n_total, deg, fwb, bwb, enc_hash, dec_hash)
        barrier()

    # ---- reduce over ranks (max time; sums of bytes and launches) -----------------------------------
    def allmax(x):
        return reduce_scalar(dist, x, "max", dev)

    def allsum(x):
        return reduce_scalar(dist, x, "sum", dev)

    total_ms = allmax(total_ms)
    enc_ms_max, dec_ms_max = allmax(enc_ms), allmax(dec_ms)
    launches = int(allsum(launches))
    par_blocks, par_ok = int(allsum(par_blocks)), int(allsum(par_ok))
    if e2e:
        e2e["s"] = allmax(e2e["s"])
        e2e["duplex_s"] = allmax(e2e["duplex_s"])
        for row in e2e["chunk_sweep"] or []:
            row["s"] = allmax(row["s"])
        e2e["h2d"] = int(allsum(e2e["h2d"]))
        e2e["d2h"] = int(allsum(e2e["d2h"]))
    if link:
        link = {k: {"sum": allsum(v), "min_rank": -allmax(-v)} for k, v in link.items()}

    # ---- config 1 of BASELINE.json is a 60k-gaussian file: far too small to be bandwidth-bound, so
    # what matters there is latency.  Device-resident launch pair and the host-pointer call, median of 50.
    latency = None
    if rank == 0:
        from spz_b200.synth import torch_cloud
        latency = small_cloud_latency(ctx, codec, torch_cloud, dev, 60_000, deg, args)

    ply_rows = None
    if rank == 0 and world == 1 and not args.no_ply:
        ply_rows = ply_rows_kernels(ctx, codec, dev, deg, n=min(n, 40_000_000))

    host_zlib = None
    if rank == 0 and not args.no_cpu_baseline:
        host_zlib = time_host_zlib(packed, deg, min(n, 400_000))

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # BASELINE.md section 4 / SURVEY.md 8d: the reference's pack + unpack, ONE thread, best of 3 on 10M points
        sample = args.cpu_sample_points or min(n_total, 10_000_000)
        cpu = cpu_reference_run(n_total, deg, args.from_coord, args.to_coord, steps=3, warmup=0, threads=1, sample_points=sample, best=True)
        cpu = {k: cpu[k] for k in cpu if k != "ms_per_step"}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:  # noqa: BLE001
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        ms_per_step = total_ms / args.steps
        value = n_total / (ms_per_step * 1e-3) / 1e6
        # per-kernel roofline on this rank's shard (rank 0's durations; all shards are equal-sized)
        enc_gbs = alg_bytes * n / (enc_ms * 1e-3) / 1e9
        dec_gbs = alg_bytes * n / (dec_ms * 1e-3) / 1e9
        dec_env = os.environ.get("SPZB200_DECODE")
        dec_kernel = ("decodeTilesKernel" if deg == 0 or dec_env == "direct" else
                      "decodeTilesBulkKernel" if dec_env == "bulk" else "decodePerGaussianKernel")
        enc_env = os.environ.get("SPZB200_ENCODE")
        enc_kernel = ("encodePerGaussianKernel" if enc_env == "bulk" or (enc_env != "tiles" and ((deg == 3 and n <= 24_000_000) or (deg == 1 and n <= 6_000_000)))
                      else "encodeTilesKernel")
        dom = (enc_kernel, enc_gbs, enc_ms) if enc_ms >= dec_ms else (dec_kernel, dec_gbs, dec_ms)
        traffic, traffic_kind = traffic_for(dom[0], n, args.traffic_bytes)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32->u8", "data": "synthetic",
            "config": bench_config(args, world),
            "encode_mgs": n_total / (enc_ms_max * 1e-3) / 1e6, "decode_mgs": n_total / (dec_ms_max * 1e-3) / 1e6,
            "encode_ms": enc_ms_max, "decode_ms": dec_ms_max,
            "hbm_gbs_per_gpu": {"encode": enc_gbs, "decode": dec_gbs},
            "roofline": {"bound": "hbm", "kernel": dom[0], "achieved": dom[1], "peak": peak, "unit": "GB/s",
                         "frac": dom[1] / peak, "frac_of_nominal_8TBs": dom[1] / 8000.0, "peak_source": peak_src,
                         "algorithmic_bytes_per_gaussian": alg_bytes, "gaussians_per_launch": n,
                         "avg_launch_ms": dom[2], "traffic": traffic, "traffic_kind": traffic_kind,
                         "encode": {"achieved": enc_gbs, "frac": enc_gbs / peak, "avg_launch_ms": enc_ms},
                         "decode": {"achieved": dec_gbs, "frac": dec_gbs / peak, "avg_launch_ms": dec_ms}},
            "gpu_launches": launches, "clocks": clocks,
            "parity": {"ok": par_ok == par_blocks, "blocks": par_blocks, "blocks_equal": par_ok, "block_points": min(65536, n),
                       "checker": par_kind, "what": "sampled blocks of every rank's device-resident encode and decode output vs the CPU checker, "
                                                   "bytes and float bits; outside the timed region",
                       "encode_hash": f"{enc_hash:016x}", "decode_hash": f"{dec_hash:016x}",
                       "hash": "order-sensitive 64-bit sum over all output planes of all ranks; a function of the cloud alone, so equal for every N"},
        }
        if e2e:
            step_s = e2e["duplex_s"]
            line["e2e"] = {"value": n_total / step_s / 1e6, "unit": UNIT, "h2d_bytes_per_step": e2e["h2d"],
                           "d2h_bytes_per_step": e2e["d2h"], "ms_per_step": step_s * 1e3, "steps": args.e2e_steps,
                           "api": "spzb200_encode_host + spzb200_decode_host (pinned host planes)",
                           "mode": "full duplex: step i's encode_host and the decode_host of step i-1's stream are issued concurrently "
                                   "from two host threads (one context each), so H2D and D2H of a step's planes overlap on the PCIe link",
                           "encode_call_ms": e2e["duplex_enc_wall_ms"], "decode_call_ms": e2e["duplex_dec_wall_ms"],
                           "planes_equal_device_path": True,
                           "sequential": {"value": n_total / e2e["s"] / 1e6, "ms_per_step": e2e["s"] * 1e3,
                                          "mode": "one host thread: encode_host, then decode_host of its result",
                                          "phases_note": "h2d/kernel/d2h_ms are sums over point ranges of per-range stream time; ranges run on 3 streams and overlap, wall_ms is the call",
                                          "encode_phases_ms": e2e["enc"], "decode_phases_ms": e2e["dec"]}}
            if e2e["chunk_sweep"]:
                line["e2e"]["chunk_sweep"] = [{"chunk_points": r["chunk_points"], "value": n_total / r["s"] / 1e6} for r in e2e["chunk_sweep"]]
            if link:
                ach_h2d, ach_d2h = e2e["h2d"] / step_s / 1e9, e2e["d2h"] / step_s / 1e9
                line["e2e"]["link_ceiling_gbs"] = {
                    "how": "bare pinned cudaMemcpyAsync (torch copy_), 1 GiB per direction per rank, all ranks at once, each phase in two shapes (1 stream x 256 MiB pieces, "
                           "3 streams x 64 MiB pieces; the better counts), 0.6 s each; GB/s per direction, summed over ranks (and the slowest rank)",
                    "h2d_alone": link["h2d_alone"], "d2h_alone": link["d2h_alone"], "duplex_each_direction": link["duplex"]}
                line["e2e"]["achieved_gbs"] = {"h2d": ach_h2d, "d2h": ach_d2h}
                line["e2e"]["frac_of_link"] = min(ach_h2d, ach_d2h) / link["duplex"]["sum"]
        if e2e_multi:
            line["e2e_multi"] = e2e_multi
        if cpu:
            line["cpu_baseline"] = cpu
        if host_zlib:
            line["host_zlib"] = host_zlib
        if latency:
            line["latency_60k"] = latency
        if ply_rows:
            line["ply_rows"] = ply_rows
        print(json.dumps(line), flush=True)
    ctx.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_e2e_multi(args, codec, dev, world, n_total, deg, fwb, bwb, enc_hash, dec_hash):
    """spzb200_encode_host_multi + spzb200_decode_host_multi over all `world` GPUs from this one process, on the
    whole cloud in pinned host memory."""
    import torch

    from spz_b200.synth import counter_cloud_torch
    devices = list(range(world))
    h_cloud = codec.alloc_cloud(n_total, deg, pinned=True, numpy_arrays=True)
    h_packed = codec.alloc_packed(n_total, deg, 3, pinned=True, numpy_arrays=True)
    h_back = codec.alloc_cloud(n_total, deg, pinned=True, numpy_arrays=True)
    fw = codec.float_plane_widths(deg)
    piece = 5_000_000 // 1280 * 1280
    for a in range(0, n_total, piece):  # the same counter-seeded cloud, generated piecewise on this GPU
        b = min(n_total, a + piece)
        part = counter_cloud_torch(n_total, deg, dev, a, b, seed=1)
        for src, dst, w in zip(part.planes(), h_cloud.planes(), fw):
            if w:
                torch.from_numpy(dst[a * w:b * w]).copy_(src)
        del part
    torch.cuda.synchronize()

    def one():
        _, te = codec.encode_host_multi(devices, h_cloud, args.from_coord, out=h_packed)
        _, td = codec.decode_host_multi(devices, h_packed, args.to_coord, out=h_back)
        return te, td

    one()  # warm: creates the pooled contexts of every device
    t0 = time.perf_counter()
    tms = [one() for _ in range(args.e2e_steps)]
    step_s = (time.perf_counter() - t0) / args.e2e_steps
    ok = planes_hash(h_packed.planes(), bwb, 0, dev) == enc_hash and planes_hash(h_back.planes(), fwb, 0, dev) == dec_hash
    # full duplex, as for the per-rank e2e: step i's encode and the decode of step i-1's stream run concurrently (two
    # pooled contexts per device), so every link carries planes in both directions at once
    from concurrent.futures import ThreadPoolExecutor
    h_packed2 = codec.alloc_packed(n_total, deg, 3, pinned=True, numpy_arrays=True)
    streams = [h_packed, h_packed2]
    codec.encode_host_multi(devices, h_cloud, args.from_coord, out=streams[1])
    pool = ThreadPoolExecutor(2)

    def duplex(i):
        fa = pool.submit(codec.encode_host_multi, devices, h_cloud, args.from_coord, streams[i % 2])
        fb = pool.submit(codec.decode_host_multi, devices, streams[(i + 1) % 2], args.to_coord, h_back)
        return fa.result()[1], fb.result()[1]

    duplex(0)
    t0 = time.perf_counter()
    for i in range(args.e2e_steps):
        duplex(1 + i)
    duplex_s = (time.perf_counter() - t0) / args.e2e_steps
    pool.shutdown()
    ok = ok and planes_hash(h_packed2.planes(), bwb, 0, dev) == enc_hash and planes_hash(h_back.planes(), fwb, 0, dev) == dec_hash
    if not ok:
        raise SystemExit("bench.py: spzb200_*_host_multi produced different planes than the per-rank device-resident path")
    best_s = min(duplex_s, step_s)
    return {"value": n_total / best_s / 1e6, "unit": UNIT, "ms_per_step": best_s * 1e3, "steps": args.e2e_steps, "devices": devices,
            "api": "spzb200_encode_host_multi + spzb200_decode_host_multi: ONE process, the whole cloud in pinned host memory, "
                   "sharded by point range over the devices (what spz::packGaussians / unpackGaussians do under SPZ_B200_DEVICES)",
            "mode": "the better of the two forms below (which one wins depends on how the box shares its links)",
            "full_duplex": {"value": n_total / duplex_s / 1e6, "ms_per_step": duplex_s * 1e3,
                            "mode": "step i's encode and the decode of step i-1's stream issued concurrently from two host threads"},
            "sequential": {"value": n_total / step_s / 1e6, "ms_per_step": step_s * 1e3,
                           "encode_call_ms": statistics.mean(t[0]["wall_ms"] for t in tms),
                           "decode_call_ms": statistics.mean(t[1]["wall_ms"] for t in tms)},
            "h2d_bytes_per_step": tms[-1][0]["h2d_bytes"] + tms[-1][1]["h2d_bytes"],
            "d2h_bytes_per_step": tms[-1][0]["d2h_bytes"] + tms[-1][1]["d2h_bytes"],
            "planes_hash_equals_parity_hash": True}


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_b200_arm(args)


if __name__ == "__main__":
    sys.exit(main())
