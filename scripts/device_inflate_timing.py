"""The inflate stage on the device against the host route, one JSON line per measurement (B200 only).

    python scripts/device_inflate_timing.py > profiles/r4_device_inflate_timing.jsonl

Files: 1M and 10M SH3 and 10M SH0 device clouds (synth.torch_cloud) saved by save_spz_device (64 KiB
segments in table blocks of 64 KiB), and the 10M SH3 cloud saved by the host saveSpz (zlib blocks of
1 MiB).  For each: the inflate kernel's time (torch.profiler, CUDA activities, over repeated
gunzip_device calls) and GB/s of inflated output; gunzip_device and load_spz_device wall time (host
clock, ending in a synchronise).  In the same run the host route composed from public pieces, step by
step: gunzip_bytes(threads=16), a pageable H2D of the container, decode_device of its planes.  The
first line names the card and its power limit.

    --compare-lib PATH   also time spzb200_load_spz_device of another build of the library (e.g. the parent
                         commit's, which inflates on the host) on the same files, alternating with this one."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from spz_b200 import _native as N  # noqa: E402
from spz_b200 import build as B  # noqa: E402
from spz_b200.codec import (PLANES, Context, PackedPlanes, _cloud_struct, alloc_cloud, byte_plane_widths,  # noqa: E402
                            gunzip_bytes, gzip_table_info)
from spz_b200.synth import torch_cloud  # noqa: E402

REPS = 5


def emit(**kw):
    print(json.dumps(kw), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def wall_ms(fn, reps=REPS):
    r = fn()
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t) * 1e3)
    return float(np.median(out)), r


def inflate_kernel_ms(ctx, blob, out, reps=REPS):
    from torch.profiler import ProfilerActivity, profile
    ctx.gunzip_device(blob, out=out)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.gunzip_device(blob, out=out)
    return sum(e.device_time for e in prof.events() if e.device_type.name == "CUDA" and "inflateBlocksKernel" in e.name) / 1e3 / reps


def packed_from_container(dev, n, deg):
    """Aligned device planes of a version-3 container already on the device (struct order)."""
    w = byte_plane_widths(deg)  # positions, scales, rotations, alphas, colors, sh
    order = [0, 3, 4, 1, 2, 5]  # stream order -> struct index
    planes, off = [None] * 6, 16
    for s in order:
        planes[s] = dev[off:off + w[s] * n].clone()
        off += w[s] * n
    frac = int(dev[13].item())
    return PackedPlanes(n, deg, *planes, fractional_bits=frac, version=3)


class OtherBuild:
    """spzb200_load_spz_device of another build of the library, through a context of its own."""

    def __init__(self, path):
        self.lib = C.CDLL(path)
        self.lib.spzb200_create.argtypes = [C.c_int32, C.POINTER(C.c_void_p)]
        self.lib.spzb200_load_spz_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int32, C.POINTER(N.Cloud),
                                                     C.POINTER(C.c_int32), C.c_void_p]
        self.h = C.c_void_p(None)
        assert self.lib.spzb200_create(0, C.byref(self.h)) == 0

    def load(self, blob, out):
        buf = np.frombuffer(blob, np.uint8)
        cs, aa = _cloud_struct(out, True), C.c_int32(0)
        rc = self.lib.spzb200_load_spz_device(self.h, C.c_void_p(buf.ctypes.data), buf.size, 0, C.byref(cs), C.byref(aa),
                                              C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0


def compare_load(ctx, other, label, blob, n, deg):
    """load_spz_device of this build and of the other one, alternating, into the same planes; the planes must agree."""
    mine, theirs = alloc_cloud(n, deg, device="cuda"), alloc_cloud(n, deg, device="cuda")
    a, b = [], []
    for _ in range(REPS):
        a.append(wall_ms(lambda: ctx.load_spz_device(blob, out=mine), reps=1)[0])
        b.append(wall_ms(lambda: other.load(blob, theirs), reps=1)[0])
    same = all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in zip(mine.planes(), theirs.planes()))
    emit(kind="load_ab", file=label, n=n, sh_degree=deg, load_spz_device_ms=round(float(np.median(a)), 2),
         other_build_load_spz_device_ms=round(float(np.median(b)), 2), speedup=round(float(np.median(b) / np.median(a)), 2),
         planes_equal=same)
    del mine, theirs


def measure(ctx, label, blob, n, deg, other=None):
    size, blocks = gzip_table_info(blob)
    out = torch.empty(size, dtype=torch.uint8, device="cuda")
    kern = inflate_kernel_ms(ctx, blob, out)
    gun_ms, (_, on_device) = wall_ms(lambda: ctx.gunzip_device(blob, out=out))
    load_ms, _ = wall_ms(lambda: ctx.load_spz_device(blob))
    emit(kind="device_route", file=label, n=n, sh_degree=deg, file_bytes=len(blob), container_bytes=size, table_blocks=blocks,
         block_bytes=int.from_bytes(blob[16:20], "little"), on_device=on_device, inflate_kernel_ms=round(kern, 3),
         inflate_output_GBps=round(size / kern / 1e6, 1) if kern else None, gunzip_device_ms=round(gun_ms, 2),
         load_spz_device_ms=round(load_ms, 2))
    # the host route from public pieces
    host_inflate_ms, container = wall_ms(lambda: gunzip_bytes(blob, threads=16))
    pageable = np.frombuffer(bytearray(container), np.uint8)
    h2d_ms, dev = wall_ms(lambda: torch.from_numpy(pageable).to("cuda"))
    packed = packed_from_container(dev, n, deg)
    decode_ms, _ = wall_ms(lambda: ctx.decode_device(packed))
    emit(kind="host_route", file=label, n=n, sh_degree=deg, gunzip_bytes_16_threads_ms=round(host_inflate_ms, 2),
         h2d_pageable_container_ms=round(h2d_ms, 2), decode_device_ms=round(decode_ms, 3),
         sum_ms=round(host_inflate_ms + h2d_ms + decode_ms, 2))
    del out, dev, packed
    torch.cuda.empty_cache()
    if other is not None:
        compare_load(ctx, other, label, blob, n, deg)
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--compare-lib", default=None)
    args = ap.parse_args()
    B.build_python_module()
    from spz_b200.pyspz import spz
    emit(kind="card", **card())
    ctx = Context(0)
    other = OtherBuild(args.compare_lib) if args.compare_lib else None
    for n, deg in ((1_000_000, 3), (10_000_000, 3), (10_000_000, 0)):
        c = torch_cloud(n, deg, "cuda", seed=1)
        blob = ctx.save_spz_device(c)
        measure(ctx, "save_spz_device", blob, n, deg, other)
        if n == 10_000_000 and deg == 3:
            g = spz.GaussianCloud()
            g.sh_degree = deg
            for name, p in zip(PLANES, c.planes()):
                setattr(g, name, p.cpu().numpy())
            with tempfile.TemporaryDirectory() as tmp:
                path = os.path.join(tmp, "x.spz")
                assert spz.save_spz(g, spz.PackOptions(), path)
                with open(path, "rb") as f:
                    host_blob = f.read()
            del g
            measure(ctx, "host saveSpz", host_blob, n, deg, other)
        del c
        torch.cuda.empty_cache()
    ctx.close()


if __name__ == "__main__":
    main()
