"""-m gpu: .spz files from and to device-resident clouds (Context.gzip_device / save_spz_device /
load_spz_device), against the host deflater model (tests/host_emul/deflate_host.cc), Python's gzip,
the host saveSpz / loadSpz of the `spz` module and, where built, the reference."""
from __future__ import annotations

import gzip
import os
import struct

import numpy as np
import pytest

from test_device_deflate_host import RUN_MIN, SEG, build_deflate_host, host_gzip

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.fixture(scope="module")
def dfl():
    return build_deflate_host()


@pytest.fixture(scope="module")
def spz():
    from spz_b200 import build as B
    B.build_python_module()
    from spz_b200.pyspz import spz as module
    return module


def dev_bytes(torch, data: bytes):
    return torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda() if data else torch.empty(0, dtype=torch.uint8, device="cuda")


def gzip_cases():
    rng = np.random.default_rng(11)
    for size in (0, 1, 65535, 65536, 65537, 3 * 65536 + 7, 20_000_000):
        yield f"zeros {size}", bytes(size)
        yield f"0x80 {size}", b"\x80" * size
        yield f"random {size}", rng.integers(0, 256, size, dtype=np.uint8).tobytes()
        fib = np.array([1, 1, 2, 3, 5, 8, 13, 21, 34, 55, 89, 144, 233, 377, 610], np.float64)
        yield f"fibonacci {size}", rng.choice(len(fib), size, p=fib / fib.sum()).astype(np.uint8).tobytes()
    base = bytearray(rng.integers(0, 4, 4 * SEG, dtype=np.uint8).tobytes())
    for run in (RUN_MIN - 1, RUN_MIN, RUN_MIN + 1, 258, 259, 516):
        b = bytearray(base)
        for edge in (SEG, 2 * SEG, 3 * SEG):  # across, ending at and starting at segment edges
            b[edge - run // 2:edge - run // 2 + run] = b"\x09" * run
        b[SEG - run:SEG] = b"\x0a" * run
        b[2 * SEG:2 * SEG + run] = b"\x0b" * run
        yield f"runs {run}", bytes(b)
    # runs that span thread slices (128 bytes) of one segment
    yield "slice-spanning runs", b"".join(bytes([i % 7]) * (i * 37 % 700 + 1) for i in range(2000))[:5 * SEG]


def test_gzip_device_round_trip(torch, gpu_ctx, dfl):
    from spz_b200.codec import gunzip_bytes
    for name, data in gzip_cases():
        member = gpu_ctx.gzip_device(dev_bytes(torch, data))
        assert member == host_gzip(dfl, data), name  # the kernels compute exactly the format's model
        assert gzip.decompress(member) == data, name  # CRC and ISIZE checked
        assert gunzip_bytes(member, threads=8) == data, name
        if name.startswith("random"):
            assert len(member) <= len(data) * 1.001 + 64, name


def test_gzip_device_encoded_containers(torch, gpu_ctx, dfl):
    from spz_b200.codec import CloudPlanes
    from spz_b200.synth import numpy_cloud
    for deg in range(4):
        c = numpy_cloud(70_000, deg, seed=deg)
        blob = gpu_ctx.save_spz_device(CloudPlanes(c.n, deg, *[torch.from_numpy(p).cuda() for p in c.planes()]))
        container = gzip.decompress(blob)
        member = gpu_ctx.gzip_device(dev_bytes(torch, container))
        assert member == host_gzip(dfl, container) and gzip.decompress(member) == container


def test_gzip_device_deterministic(torch, gpu_ctx):
    from spz_b200.codec import Context
    data = dev_bytes(torch, np.random.default_rng(3).geometric(0.05, 3_000_000).astype(np.uint8).tobytes())
    first = gpu_ctx.gzip_device(data)
    assert gpu_ctx.gzip_device(data) == first
    s = torch.cuda.Stream()
    with Context(0) as other:
        assert other.gzip_device(data, stream=s) == first
    if torch.cuda.device_count() > 1:
        with Context(1) as second:
            assert second.gzip_device(data.to("cuda:1"), stream=torch.cuda.current_stream(1)) == first


def host_save(spz, tmp_path, c, frm, antialiased):
    g = spz.GaussianCloud()
    g.sh_degree = c.sh_degree
    g.antialiased = antialiased
    for name in ("positions", "scales", "rotations", "alphas", "colors", "sh"):
        setattr(g, name, np.asarray(getattr(c, name)))
    o = spz.PackOptions()
    o.from_coord = spz.CoordinateSystem(frm)
    path = str(tmp_path / "host.spz")
    assert spz.save_spz(g, o, path)
    with open(path, "rb") as f:
        return f.read()


def to_device(torch, c):
    from spz_b200.codec import CloudPlanes
    return CloudPlanes(c.n, c.sh_degree, *[torch.from_numpy(np.asarray(p)).cuda() for p in c.planes()])


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_save_spz_device_inflates_to_host_container(torch, gpu_ctx, spz, tmp_path, deg):
    from oracle import Ref
    from spz_b200.synth import numpy_cloud
    c = numpy_cloud(50_000 + 17 * deg, deg, seed=20 + deg)
    dc = to_device(torch, c)
    for frm in (0, 2, 6):
        for aa in (False, True):
            blob = gpu_ctx.save_spz_device(dc, frm, antialiased=aa)
            host = host_save(spz, tmp_path, c, frm, aa)
            assert gzip.decompress(blob) == gzip.decompress(host), (frm, aa)
    if Ref.available():
        back = Ref().load_spz(gpu_ctx.save_spz_device(dc, 0))
        want = Ref().load_spz(host_save(spz, tmp_path, c, 0, False))
        from util import assert_cloud_bits_equal
        assert_cloud_bits_equal(back, want, "reference loadSpz")


def host_load(spz, tmp_path, blob, to):
    path = str(tmp_path / "in.spz")
    with open(path, "wb") as f:
        f.write(blob)
    o = spz.UnpackOptions()
    o.to_coord = spz.CoordinateSystem(to)
    return spz.load_spz(path, o)


def assert_same_cloud(dev, host, what):
    from util import PLANES
    from oracle import bits
    assert dev.n == host.num_points and dev.sh_degree == host.sh_degree, what
    for name in PLANES:
        got = getattr(dev, name).cpu().numpy() if dev.n else np.zeros(0, np.float32)
        assert np.array_equal(bits(got), bits(np.asarray(getattr(host, name), np.float32))), f"{what}: {name}"


def version_container(rng, n, deg, ver):
    from util import random_stream
    p = random_stream(rng, n, deg, ver)
    head = struct.pack("<IIIBBBB", 0x5053474E, ver, n, deg, 12, 1, 0)
    return head + b"".join(np.asarray(x).tobytes() for x in (p.positions, p.alphas, p.colors, p.scales, p.rotations, p.sh))


def test_load_spz_device_matches_host_load(torch, gpu_ctx, spz, tmp_path, monkeypatch):
    from oracle import Ref
    from spz_b200.synth import numpy_cloud
    rng = np.random.default_rng(4)
    c = numpy_cloud(40_000, 3, seed=8)
    files = {"save_spz_device": gpu_ctx.save_spz_device(to_device(torch, c), 1, antialiased=True),
             "version 1": gzip.compress(version_container(rng, 3000, 2, 1)),
             "version 2": gzip.compress(version_container(rng, 3000, 3, 2))}
    monkeypatch.setenv("SPZ_B200_GZIP_THREADS", "4")  # the block-parallel host writer, at any size
    files["block-parallel saveSpz"] = host_save(spz, tmp_path, c, 0, False)
    monkeypatch.delenv("SPZ_B200_GZIP_THREADS")
    if Ref.available():
        from oracle import Cloud
        files["reference"] = Ref().save_spz(Cloud(c.n, 3, *c.planes()), 0)
    for name, blob in files.items():
        for to in (range(9) if name == "save_spz_device" else (0, 6)):
            got, aa = gpu_ctx.load_spz_device(blob, to=to)
            want = host_load(spz, tmp_path, blob, to)
            assert_same_cloud(got, want, f"{name} to={to}")
            assert aa == want.antialiased


def test_load_spz_device_rejects_bad_files(torch, gpu_ctx):
    from spz_b200 import _native as N
    from spz_b200.codec import alloc_cloud
    from spz_b200.synth import numpy_cloud
    c = numpy_cloud(5000, 1, seed=2)
    good = gpu_ctx.save_spz_device(to_device(torch, c))
    container = bytearray(gzip.decompress(good))
    bad_magic = bytearray(container)
    bad_magic[0] ^= 0xFF
    oversized = bytearray(container)
    struct.pack_into("<I", oversized, 8, 5001)  # the header claims more points than the planes hold
    out = alloc_cloud(5000, 1, device="cuda")
    for p in out.planes():
        p.fill_(7.0)
    for blob in (good[:len(good) // 2], good[:30], gzip.compress(bytes(bad_magic)), gzip.compress(bytes(oversized))):
        with pytest.raises(N.CodecError) as e:
            gpu_ctx.load_spz_device(blob, out=out)
        assert e.value.code == N.ERR_INVALID
        torch.cuda.synchronize()
        assert all(bool((p == 7.0).all()) for p in out.planes())


def peaked(c, rng):
    c.sh[:] = rng.normal(0, 0.05, c.sh.size).astype(np.float32)
    c.scales[:] = rng.normal(-4.5, 1, c.scales.size).astype(np.float32)
    c.alphas[:] = rng.normal(2, 1, c.alphas.size).astype(np.float32)
    c.colors[:] = rng.normal(0, 0.3, c.colors.size).astype(np.float32)
    return c


def test_compression_ratio(torch, gpu_ctx, spz, tmp_path):
    from spz_b200.synth import numpy_cloud
    rng = np.random.default_rng(6)
    n = 1_000_000
    for c in (numpy_cloud(n, 3, seed=1), peaked(numpy_cloud(n, 3, seed=2), rng)):
        dev = len(gpu_ctx.save_spz_device(to_device(torch, c)))
        host = len(host_save(spz, tmp_path, c, 0, False))
        assert dev <= host, (dev, host)
    c = numpy_cloud(n, 3, seed=3)
    c.sh[:] = 0
    with_sh = len(gpu_ctx.save_spz_device(to_device(torch, c)))
    from spz_b200.codec import CloudPlanes
    c0 = CloudPlanes(n, 0, c.positions, c.scales, c.rotations, c.alphas, c.colors, np.zeros(0, np.float32))
    without = len(gpu_ctx.save_spz_device(to_device(torch, c0)))
    assert with_sh - without < 0.01 * 45 * n


def test_large_cloud_both_routes(torch, gpu_ctx):
    from spz_b200.synth import torch_cloud
    n = 20_000_000
    c = torch_cloud(n, 3, "cuda", seed=5)
    blob = gpu_ctx.save_spz_device(c, 0)
    block_size, blocks = struct.unpack_from("<II", blob, 16)
    container = 16 + 65 * n
    assert -(-container // SEG) > 16000 and block_size > SEG and blocks <= 16000
    back, _ = gpu_ctx.load_spz_device(blob)
    want = gpu_ctx.decode_device(gpu_ctx.encode_device(c))
    for x, y in zip(back.planes(), want.planes()):
        assert torch.equal(x.view(torch.int32), y.view(torch.int32))


def test_save_on_a_stream_right_after_the_fill(torch, gpu_ctx):
    from spz_b200.synth import torch_cloud
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        c = torch_cloud(3_000_000, 3, "cuda", seed=9)  # queued on s
        blob = gpu_ctx.save_spz_device(c, 0, stream=s)
    s.synchronize()
    assert blob == gpu_ctx.save_spz_device(c, 0)
