"""Device-resident .spz files against the host route, one JSON line per measurement (B200 only).

    python scripts/device_file_timing.py > profiles/r3_device_file_timing.jsonl
    bash scripts/gpu.sh sweep r3_device_file_timing.jsonl device_file_timing.py   (the same, through the runner)

For 1M and 10M SH3 and 10M SH0 device clouds (synth.torch_cloud): the device deflater's kernel time
(torch.profiler, CUDA activities, over repeated gzip_device calls on the container) and its input GB/s;
encode time (CUDA events); D2H of the compressed bytes (events, pageable destination, as the library
copies); save_spz_device and load_spz_device wall time (host clock, ending in a synchronise); the file
size.  In the same run the existing route: D2H of the cloud into numpy planes, then spz.save_spz and
spz.load_spz (the C++ saveSpz / loadSpz) through a temporary file.  The first line names the card and
its power limit."""
from __future__ import annotations

import gzip
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from spz_b200 import build as B  # noqa: E402
from spz_b200.codec import Context, PLANES  # noqa: E402
from spz_b200.synth import torch_cloud  # noqa: E402

REPS = 3


def emit(**kw):
    print(json.dumps(kw), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def events_ms(fn, reps=REPS):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def wall_ms(fn, reps=REPS):
    fn()
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t) * 1e3)
    return float(np.median(out)), r


def deflate_kernel_ms(ctx, data, reps=REPS):
    from torch.profiler import ProfilerActivity, profile
    ctx.gzip_device(data)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.gzip_device(data)
    per = {}
    for e in prof.events():
        if e.device_type.name == "CUDA":
            for k in ("deflateSegmentsKernel", "segmentOffsetsKernel", "packSlotsKernel"):
                if k in e.name:
                    per[k] = per.get(k, 0.0) + e.device_time / 1e3 / reps
    return per


def main():
    B.build_python_module()
    from spz_b200.pyspz import spz
    emit(kind="card", **card())
    ctx = Context(0)
    for n, deg in ((1_000_000, 3), (10_000_000, 3), (10_000_000, 0)):
        c = torch_cloud(n, deg, "cuda", seed=1)
        torch.cuda.synchronize()
        enc_ms = events_ms(lambda: ctx.encode_device(c))
        save_ms, blob = wall_ms(lambda: ctx.save_spz_device(c))
        load_ms, _ = wall_ms(lambda: ctx.load_spz_device(blob))
        container = gzip.decompress(blob)
        dev_container = torch.frombuffer(bytearray(container), dtype=torch.uint8).cuda()
        kern = deflate_kernel_ms(ctx, dev_container)
        comp = torch.empty(len(blob), dtype=torch.uint8, device="cuda")
        d2h_ms, _ = wall_ms(lambda: comp.cpu())
        deflate_ms = sum(kern.values())
        emit(kind="device_route", n=n, sh_degree=deg, container_bytes=len(container), file_bytes=len(blob),
             ratio=round(len(blob) / len(container), 4), encode_ms=round(enc_ms, 3),
             deflate_kernels_ms={k: round(v, 3) for k, v in kern.items()},
             deflate_input_GBps=round(len(container) / deflate_ms / 1e6, 1) if deflate_ms else None,
             d2h_compressed_ms=round(d2h_ms, 2), save_spz_device_ms=round(save_ms, 2), load_spz_device_ms=round(load_ms, 2))
        # the existing route: cloud to host vectors, then saveSpz / loadSpz
        d2h_cloud_ms, host = wall_ms(lambda: [p.cpu().numpy() for p in c.planes()], reps=1)
        g = spz.GaussianCloud()
        g.sh_degree = deg
        for name, a in zip(PLANES, host):
            setattr(g, name, a)
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "x.spz")
            t = time.perf_counter()
            assert spz.save_spz(g, spz.PackOptions(), path)
            host_save_ms = (time.perf_counter() - t) * 1e3
            t = time.perf_counter()
            back = spz.load_spz(path)
            host_load_ms = (time.perf_counter() - t) * 1e3
            assert back.num_points == n
            size = os.path.getsize(path)
        emit(kind="host_route", n=n, sh_degree=deg, file_bytes=size, d2h_cloud_ms=round(d2h_cloud_ms, 1),
             save_spz_ms=round(host_save_ms, 1), load_spz_ms=round(host_load_ms, 1),
             save_speedup_device_vs_host=round((d2h_cloud_ms + host_save_ms) / save_ms, 1))
        del c, dev_container, comp
        torch.cuda.empty_cache()
    ctx.close()


if __name__ == "__main__":
    main()
