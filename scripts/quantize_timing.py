"""quantize_device against encode_device + decode_device, one JSON line per measurement (B200 only).

    python scripts/quantize_timing.py > profiles/r5_quantize_timing.jsonl

Clouds (synth.torch_cloud, seed 1): 1M and 10M SH3, 10M SH0 and, where it fits, 100M SH3.  Every input is
larger than the 126 MB L2 (1M SH3 is 236 MB of floats).  Times are kernel times from CUDA events recorded
right before and after each launch, median over REPS launches after WARMUP, so the host's pace does not
enter them; the two-kernel route is timed per kernel, back to back as a caller runs it (the decoder may
find part of the encoder's packed planes still in L2).  Bytes are algorithmic: 2 x the float bytes per
gaussian for quantize_device (read and write each float once), and 2 x (float + packed) bytes for the two
kernels.  The share of HBM is against the 7.7 TB/s data-sheet figure.  Each line says whether the outputs of
both routes are bit-identical.  The first line names the card and its power limit."""
from __future__ import annotations

import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from spz_b200.codec import (Context, alloc_cloud, alloc_packed, float_bytes_per_gaussian,  # noqa: E402
                            packed_bytes_per_gaussian)
from spz_b200.synth import torch_cloud  # noqa: E402

WARMUP, REPS = 5, 50
HBM_BYTES_PER_S = 7.7e12


def emit(**kw):
    print(json.dumps(kw), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def alternating_ms(fns):
    """Median GPU time of each function's work -- an event pair around every call -- with the functions
    taken in turns (REPS rounds) so that drift hits all alike."""
    for fn in fns:
        for _ in range(WARMUP):
            fn()
    pairs = [[] for _ in fns]
    for _ in range(REPS):
        for k, fn in enumerate(fns):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            pairs[k].append((a, b))
    torch.cuda.synchronize()
    return [float(np.median([a.elapsed_time(b) for a, b in p])) for p in pairs]


def measure(ctx, n, deg):
    c = torch_cloud(n, deg, "cuda", seed=1)
    out = alloc_cloud(n, deg, device="cuda")
    packed = alloc_packed(n, deg, 3, device="cuda")
    dec = alloc_cloud(n, deg, device="cuda")
    q_ms, enc_ms, dec_ms = alternating_ms([lambda: ctx.quantize_device(c, 6, out=out),
                                           lambda: ctx.encode_device(c, 6, out=packed),
                                           lambda: ctx.decode_device(packed, 6, out=dec)])
    torch.cuda.synchronize()
    same = all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in zip(out.planes(), dec.planes()))
    fb, pb = float_bytes_per_gaussian(deg), packed_bytes_per_gaussian(deg)
    q_bytes, route_bytes = 2 * fb * n, 2 * (fb + pb) * n
    emit(kind="quantize", n=n, sh_degree=deg, version=3, frm=6, to=6, launches_per_call=1,
         quantize_kernel_ms=round(q_ms, 4), quantize_bytes=q_bytes, quantize_GBps=round(q_bytes / q_ms / 1e6, 1),
         quantize_share_of_hbm=round(q_bytes / (q_ms * 1e-3) / HBM_BYTES_PER_S, 3),
         encode_kernel_ms=round(enc_ms, 4), decode_kernel_ms=round(dec_ms, 4), encode_plus_decode_ms=round(enc_ms + dec_ms, 4),
         route_bytes=route_bytes, route_GBps=round(route_bytes / (enc_ms + dec_ms) / 1e6, 1),
         speedup=round((enc_ms + dec_ms) / q_ms, 3), outputs_bit_identical=same)
    del c, out, packed, dec
    torch.cuda.empty_cache()


def main():
    emit(kind="card", **card())
    ctx = Context(0)
    for n, deg in ((1_000_000, 3), (10_000_000, 3), (10_000_000, 0), (100_000_000, 3)):
        need = n * (3 * float_bytes_per_gaussian(deg) + packed_bytes_per_gaussian(deg))
        free, _ = torch.cuda.mem_get_info()
        if need > 0.8 * free:
            emit(kind="skipped", n=n, sh_degree=deg, bytes_needed=need, bytes_free=free)
            continue
        measure(ctx, n, deg)
    ctx.close()


if __name__ == "__main__":
    main()
