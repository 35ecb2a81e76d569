"""Batches of .spz files of device clouds against loops of single calls, one JSON line per measurement
(B200 only).

    python scripts/device_batch_timing.py > profiles/r7_device_batch_timing.jsonl

Batches: K = 1, 8, 64, 256 synthetic 60K-point SH3 scenes, K = 1, 8 of 1M SH3 and K = 64 of 60K SH0
(synth.torch_cloud, seeded).  For each batch, in one run with the profiler off:
  * save_spz_device_batch against a loop of save_spz_device, and load_spz_device_batch against a loop of
    load_spz_device, alternating, wall time (host clock ending in a synchronise), median of five;
  * for loading, also the host route per file composed from public pieces: gunzip_bytes(threads=16), a
    pageable H2D of the container and decode_device of its planes;
  * the outputs of the batch and of the loop compared (file bytes, cloud bits).
Then, in a run of its own, the deflate, inflate and plane-move kernels' device time (torch.profiler, CUDA
activities) of one batch call and of one loop.  Last, gunzip_device of one 10M SH3 file: inflate kernel
time and wall time.  The first line names the card and its power limit."""
from __future__ import annotations

import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from spz_b200.codec import PackedPlanes, Context, byte_plane_widths, gunzip_bytes  # noqa: E402
from spz_b200.synth import torch_cloud  # noqa: E402

REPS = 5
BATCHES = ((60_000, 3, 1), (60_000, 3, 8), (60_000, 3, 64), (60_000, 3, 256), (1_000_000, 3, 1), (1_000_000, 3, 8), (60_000, 0, 64))
DEFLATE = ("deflateSegmentsKernel", "segmentOffsetsKernel", "packSlotsKernel")


def emit(**kw):
    print(json.dumps(kw), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3, r


def alternate(a, b):
    """Medians of REPS timings of a and b taken in turns, after one warm-up call of each; their last results."""
    ra, rb = a(), b()
    ta, tb = [], []
    for _ in range(REPS):
        t, ra = timed(a)
        ta.append(t)
        t, rb = timed(b)
        tb.append(t)
    return float(np.median(ta)), float(np.median(tb)), ra, rb


def kernel_ms(fn):
    """Device time of fn's deflate, inflate and move kernels (torch.profiler), one call after a warm-up."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {"deflate": 0.0, "inflate": 0.0, "move": 0.0, "deflate_launches": 0, "inflate_launches": 0, "move_launches": 0}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        key = "deflate" if any(k in e.name for k in DEFLATE) else "inflate" if "inflateBlocksKernel" in e.name else \
            "move" if "moveSpansKernel" in e.name else None
        if key:
            out[key] += e.device_time / 1e3
            out[key + "_launches"] += 1
    return {k: round(v, 4) if isinstance(v, float) else v for k, v in out.items()}


def same_clouds(xs, ys):
    return all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for x, y in zip(xs, ys) for a, b in zip(x.planes(), y.planes()))


def host_route(ctx, blob, n, deg):
    """gunzip_bytes(threads=16) + pageable H2D of the container + decode_device of its aligned planes."""
    container = gunzip_bytes(blob, threads=16)
    dev = torch.from_numpy(np.frombuffer(bytearray(container), np.uint8)).to("cuda")
    w = byte_plane_widths(deg)
    planes, off = [None] * 6, 16
    for s in (0, 3, 4, 1, 2, 5):  # stream order -> struct index
        planes[s] = dev[off:off + w[s] * n].clone()
        off += w[s] * n
    return ctx.decode_device(PackedPlanes(n, deg, *planes, fractional_bits=int(container[13]), version=3))


def measure(ctx, n, deg, k):
    clouds = [torch_cloud(n, deg, "cuda", seed=1000 * deg + i) for i in range(k)]
    label = dict(n=n, sh_degree=deg, files=k)
    save_batch, save_loop, files, loop_files = alternate(lambda: ctx.save_spz_device_batch(clouds),
                                                         lambda: [ctx.save_spz_device(c) for c in clouds])
    emit(kind="save", **label, file_bytes=sum(map(len, files)), batch_ms=round(save_batch, 2), loop_ms=round(save_loop, 2),
         speedup=round(save_loop / save_batch, 2), outputs_equal=files == loop_files)
    load_batch, load_loop, got, loop_got = alternate(lambda: [c for c, _ in ctx.load_spz_device_batch(files)],
                                                     lambda: [ctx.load_spz_device(f)[0] for f in files])
    host_ms, host_got = timed(lambda: [host_route(ctx, f, n, deg) for f in files])
    emit(kind="load", **label, batch_ms=round(load_batch, 2), loop_ms=round(load_loop, 2), speedup=round(load_loop / load_batch, 2),
         host_route_loop_ms=round(host_ms, 2), outputs_equal=same_clouds(got, loop_got) and same_clouds(got, host_got))
    del got, loop_got, host_got
    emit(kind="kernels", **label, save_batch=kernel_ms(lambda: ctx.save_spz_device_batch(clouds)),
         save_loop=kernel_ms(lambda: [ctx.save_spz_device(c) for c in clouds]),
         load_batch=kernel_ms(lambda: ctx.load_spz_device_batch(files)), load_loop=kernel_ms(lambda: [ctx.load_spz_device(f) for f in files]))
    del clouds, files, loop_files
    torch.cuda.empty_cache()


def single_10m(ctx):
    blob = ctx.save_spz_device(torch_cloud(10_000_000, 3, "cuda", seed=1))
    torch.cuda.empty_cache()
    out = torch.empty(len(gunzip_bytes(blob, threads=16)), dtype=torch.uint8, device="cuda")
    walls = [timed(lambda: ctx.gunzip_device(blob, out=out))[0] for _ in range(REPS + 1)][1:]
    emit(kind="single_10m_sh3", file_bytes=len(blob), gunzip_device_ms=round(float(np.median(walls)), 2),
         kernels=kernel_ms(lambda: ctx.gunzip_device(blob, out=out)))


def main():
    emit(kind="card", **card())
    ctx = Context(0)
    for n, deg, k in BATCHES:
        measure(ctx, n, deg, k)
    single_10m(ctx)
    ctx.close()


if __name__ == "__main__":
    main()
