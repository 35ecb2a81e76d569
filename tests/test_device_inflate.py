"""-m gpu: the inflate stage on the device (Context.gunzip_device, and load_spz_device's route for
block-table members) against Python's gzip, spzb200_gunzip and the host loadSpz of the `spz` module.
The damaged members are ones the host build of the decoder (test_device_inflate_host.py) handles
safely."""
from __future__ import annotations

import gzip
import struct

import numpy as np
import pytest

from test_device_deflate_host import SEG
from test_device_file import assert_same_cloud, dev_bytes, gzip_cases, host_load, host_save, to_device, version_container
from test_device_inflate_host import damaged_copies, damaged_source, mixed

pytestmark = pytest.mark.gpu

GUARD = 4096


@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.fixture(scope="module")
def spz():
    from spz_b200 import build as B
    B.build_python_module()
    from spz_b200.pyspz import spz as module
    return module


def gunzip_guarded(torch, ctx, blob, size):
    """gunzip_device into the middle of a tensor with guard bands; checks the bands after the call."""
    buf = torch.full((size + 2 * GUARD,), 0xA5, dtype=torch.uint8, device="cuda")
    try:
        got, on_device = ctx.gunzip_device(blob, out=buf[GUARD:GUARD + size])
        result = (got.cpu().numpy().tobytes(), on_device)
    finally:
        torch.cuda.synchronize()
        assert bool((buf[:GUARD] == 0xA5).all()) and bool((buf[GUARD + size:] == 0xA5).all()), "guard band overwritten"
    return result


def test_gunzip_device_device_deflater_members(torch, gpu_ctx):
    from spz_b200.codec import gzip_table_info
    for name, data in gzip_cases():
        member = gpu_ctx.gzip_device(dev_bytes(torch, data))
        if not data:
            continue  # an empty member has no table: covered below
        size, blocks = gzip_table_info(member)
        assert size == len(data), name
        got, on_device = gunzip_guarded(torch, gpu_ctx, member, size)
        assert got == gzip.decompress(member) == data, name
        assert on_device, name


@pytest.mark.parametrize("level", [1, 6])
def test_gunzip_device_host_parallel_members(torch, gpu_ctx, monkeypatch, level):
    from spz_b200.codec import gzip_bytes
    monkeypatch.setenv("SPZ_B200_GZIP_LEVEL", str(level))
    data = mixed(np.random.default_rng(level), (9 << 20) + 77)
    member = gzip_bytes(data, threads=4)
    got, on_device = gunzip_guarded(torch, gpu_ctx, member, len(data))
    assert got == data and on_device
    t, on = gpu_ctx.gunzip_device(member)  # allocated from the table's size
    assert t.numel() == len(data) and on and t.cpu().numpy().tobytes() == data


def test_gunzip_device_without_table_fails(torch, gpu_ctx):
    from spz_b200 import _native as N
    from spz_b200.codec import gzip_table_info
    for blob in (gzip.compress(b"x" * 100000), gpu_ctx.gzip_device(dev_bytes(torch, b""))):
        with pytest.raises(N.CodecError) as e:
            gzip_table_info(blob)
        assert e.value.code == N.ERR_INVALID
        out = torch.zeros(200000, dtype=torch.uint8, device="cuda")
        with pytest.raises(N.CodecError) as e:
            gpu_ctx.gunzip_device(blob, out=out)
        assert e.value.code == N.ERR_INVALID


def test_gunzip_device_damaged_members(torch, gpu_ctx):
    from spz_b200 import _native as N
    from spz_b200.codec import gunzip_bytes, gzip_table_info
    member = gpu_ctx.gzip_device(dev_bytes(torch, damaged_source()))
    for name, blob in damaged_copies(member):
        try:
            want = gunzip_bytes(blob, threads=8)
        except N.CodecError:
            want = None
        size, _ = gzip_table_info(blob)
        try:
            got, _ = gunzip_guarded(torch, gpu_ctx, blob, size)
        except N.CodecError as e:
            assert e.code == N.ERR_INVALID, name
            got = None
        assert got == want, name


def test_load_spz_device_block_table_members_match_host_load(torch, gpu_ctx, spz, tmp_path, monkeypatch):
    """64 KiB table blocks (save_spz_device, and version-1/2 containers framed by the device deflater's
    host model) take the device route; 1 MiB zlib blocks (saveSpz, gzip_bytes) the host route.  Both give
    host loadSpz's planes, and the device inflater vouches for every one of these members."""
    from spz_b200.codec import gzip_bytes
    from spz_b200.synth import numpy_cloud
    from test_device_deflate_host import build_deflate_host, host_gzip
    dfl = build_deflate_host()
    rng = np.random.default_rng(31)
    files = {}
    for deg in range(4):
        c = numpy_cloud(60_000 + deg, deg, seed=40 + deg)
        files[f"save_spz_device SH{deg}"] = gpu_ctx.save_spz_device(to_device(torch, c), 1, antialiased=deg == 2)
    monkeypatch.setenv("SPZ_B200_GZIP_THREADS", "4")  # the block-parallel host writer, at any size
    c = numpy_cloud(150_000, 3, seed=9)
    files["block-parallel saveSpz"] = host_save(spz, tmp_path, c, 0, False)
    monkeypatch.delenv("SPZ_B200_GZIP_THREADS")
    files["version 1 by gzip_bytes"] = gzip_bytes(version_container(rng, 60_000, 2, 1), threads=4)
    files["version 2 by gzip_bytes"] = gzip_bytes(version_container(rng, 60_000, 3, 2), threads=4)
    files["version 1, 64 KiB blocks"] = host_gzip(dfl, version_container(rng, 40_000, 1, 1))
    files["version 2, 64 KiB blocks"] = host_gzip(dfl, version_container(rng, 40_000, 3, 2))
    for name, blob in files.items():
        _, on_device = gpu_ctx.gunzip_device(blob)
        assert on_device, name
        for to in (0, 6):
            got, aa = gpu_ctx.load_spz_device(blob, to=to)
            want = host_load(spz, tmp_path, blob, to)
            assert_same_cloud(got, want, f"{name} to={to}")
            assert aa == want.antialiased, name


def test_load_spz_device_damaged_member_keeps_host_verdict(torch, gpu_ctx, spz, tmp_path):
    from spz_b200 import _native as N
    from spz_b200.codec import alloc_cloud
    from spz_b200.synth import numpy_cloud
    c = numpy_cloud(30_000, 1, seed=3)
    good = bytearray(gpu_ctx.save_spz_device(to_device(torch, c)))
    good[-8] ^= 1  # trailer CRC: the device cannot vouch, and the host route rejects the member
    out = alloc_cloud(30_000, 1, device="cuda")
    for p in out.planes():
        p.fill_(7.0)
    with pytest.raises(N.CodecError) as e:
        gpu_ctx.load_spz_device(bytes(good), out=out)
    assert e.value.code == N.ERR_INVALID
    torch.cuda.synchronize()
    assert all(bool((p == 7.0).all()) for p in out.planes())


def test_load_spz_device_20m_sh3(torch, gpu_ctx):
    from spz_b200.codec import gzip_table_info
    from spz_b200.synth import torch_cloud
    n = 20_000_000
    c = torch_cloud(n, 3, "cuda", seed=5)
    blob = gpu_ctx.save_spz_device(c, 0)
    block_size, _ = struct.unpack_from("<II", blob, 16)
    assert block_size == 2 * SEG  # 128 KiB table blocks
    size, _ = gzip_table_info(blob)
    t, on_device = gpu_ctx.gunzip_device(blob)
    assert on_device and t.numel() == size
    del t
    back, _ = gpu_ctx.load_spz_device(blob)
    want = gpu_ctx.decode_device(gpu_ctx.encode_device(c))
    for x, y in zip(back.planes(), want.planes()):
        assert torch.equal(x.view(torch.int32), y.view(torch.int32))
