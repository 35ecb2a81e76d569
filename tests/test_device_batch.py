"""Batches of .spz files of device clouds (DESIGN.md section 10c): Context.gzip_device_batch,
save_spz_device_batch, gunzip_device_batch and load_spz_device_batch.

Entry i of every batch must be exactly what the single-file call gives for input i alone -- the same
bytes, the same cloud bits, the same verdict and `on_device` -- whatever its neighbours are and in any
order, and the batch must really share its launches: one inflate and one plane-move launch for a load
batch, three deflate launches and one plane-move launch for a save batch.

The descriptor tables (batch_plan.hpp) need no GPU: they are checked against a Python restatement
through tests/host_emul/batch_host.cc.  Every other test is -m gpu."""
from __future__ import annotations

import ctypes as C
import gzip
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from test_device_deflate_host import RUN_MIN, SEG, build_deflate_host, host_gzip
from test_device_inflate_host import build_inflate_host, crafted_streams, hostile_corpus, mixed, zlib_verdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu

GUARD = 4096
FILL = 0xA5
MAX_TABLE_BLOCKS = 16000  # deflate_format.cuh: kMaxTableBlocks


# ---- descriptor tables, no GPU ------------------------------------------------------------------------


class DeflateSegment(C.Structure):
    _fields_ = [("src", C.c_uint64), ("len", C.c_uint32), ("last", C.c_uint32)]


class InflateBlock(C.Structure):
    _fields_ = [("inp", C.c_uint64), ("out", C.c_uint64), ("in_bytes", C.c_uint32), ("out_bytes", C.c_uint32)]


@pytest.fixture(scope="module")
def plan():
    """tests/host_emul/_build/libbatch_host.so: batch_plan.hpp compiled for the host."""
    here = os.path.join(ROOT, "tests", "host_emul")
    out_dir = os.path.join(here, "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libbatch_host.so")
    deps = [os.path.join(here, "batch_host.cc")] + [os.path.join(ROOT, "spz_b200", "csrc", h) for h in ("batch_plan.hpp", "deflate_format.cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", deps[0], "-o", so], check=True)
    lib = C.CDLL(so)
    u64p, u32p = C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)
    lib.bp_plan_deflate.restype = C.c_longlong
    lib.bp_plan_deflate.argtypes = [u64p, u64p, C.c_int, u64p, C.POINTER(DeflateSegment), C.c_longlong]
    lib.bp_member_bodies.restype = C.c_longlong
    lib.bp_member_bodies.argtypes = [u32p, u64p, C.c_int, u64p, u32p, u64p, C.c_longlong]
    lib.bp_plan_inflate.argtypes = [C.c_int, u64p, u64p, u64p, u32p, u64p, C.POINTER(InflateBlock), u64p, u64p]
    lib.bp_plan_aligned.argtypes = [u64p, C.c_int, u64p]
    lib.bp_sizes.argtypes = [C.POINTER(C.c_int)] * 3
    return lib


def _arr(ctype, values):
    values = list(values)
    return (ctype * max(len(values), 1))(*values)


# restatement: segments of one input, the table blocks of one member
def py_segments(size):
    n = max(1, -(-size // SEG))
    return [(s * SEG, min(SEG, size - s * SEG), int(s + 1 == n)) for s in range(n)]


def py_blocks(seg_bytes):
    per = -(-len(seg_bytes) // MAX_TABLE_BLOCKS)
    return [sum(seg_bytes[k:k + per]) for k in range(0, len(seg_bytes), per)]


PLAN_SIZES = [0, 1, SEG - 1, SEG, SEG + 1, 1024 * SEG + 1, 16000 * SEG + 1]


def test_descriptor_layouts(plan):
    seg, block, span = C.c_int(), C.c_int(), C.c_int()
    assert plan.bp_sizes(C.byref(seg), C.byref(block), C.byref(span)) == SEG
    assert (seg.value, block.value, span.value) == (16, 24, 24) == (C.sizeof(DeflateSegment), C.sizeof(InflateBlock), 24)


@pytest.mark.parametrize("order", ["ascending", "mixed"])
def test_deflate_plan_matches_restatement(plan, order):
    sizes = PLAN_SIZES if order == "ascending" else [16000 * SEG + 1, 0, SEG + 1, 1, 1024 * SEG + 1, SEG, SEG - 1, 0]
    base = [(1 << 40) * (i + 1) + i for i in range(len(sizes))]  # distinct addresses, some unaligned
    total = sum(len(py_segments(s)) for s in sizes)
    first = (C.c_uint64 * (len(sizes) + 1))()
    segs = (DeflateSegment * total)()
    got = plan.bp_plan_deflate(_arr(C.c_uint64, base), _arr(C.c_uint64, sizes), len(sizes), first, segs, total)
    assert got == total
    at = 0
    for i, size in enumerate(sizes):
        assert first[i] == at
        for off, length, last in py_segments(size):
            d = segs[at]
            assert (d.src, d.len, d.last) == (base[i] + off, length, last), (size, off)
            at += 1
    assert first[len(sizes)] == total
    # body ranges and table blocks from synthetic segment sizes
    rng = np.random.default_rng(1)
    seg_bytes = rng.integers(0, SEG + 64, total).astype(np.uint32)
    body = (C.c_uint64 * (len(sizes) + 1))()
    nblocks = (C.c_uint64 * len(sizes))()
    want_blocks, want_start, acc = [], [0], 0
    for i in range(len(sizes)):
        mine = seg_bytes[first[i]:first[i + 1]].astype(np.int64).tolist()
        want_blocks.append(py_blocks(mine))
        acc += sum(mine)
        want_start.append(acc)
    cap = sum(len(b) for b in want_blocks)
    flat = (C.c_uint32 * cap)()
    assert plan.bp_member_bodies(seg_bytes.ctypes.data_as(C.POINTER(C.c_uint32)), first, len(sizes), body, flat, nblocks, cap) == cap
    assert list(body) == want_start
    at = 0
    for i, b in enumerate(want_blocks):
        assert nblocks[i] == len(b) and list(flat[at:at + len(b)]) == b, sizes[i]
        at += len(b)
    if order == "ascending":  # the two table-size regimes: one segment per block, and two past 16000 segments
        assert [len(b) for b in want_blocks] == [1, 1, 1, 1, 2, 1025, 8001]


def test_inflate_plan_matches_restatement(plan):
    rng = np.random.default_rng(2)
    members = [(65536, 1), (65536, 65536), (65536, 3 * 65536 + 7), (1 << 20, 5 * (1 << 20) + 1), (4097, 20 * 4097 + 3), (1, 17),
               (262144, 262144 * 3)]
    block_size = [b for b, _ in members]
    total = [t for _, t in members]
    nblocks = [max(1, -(-t // b)) for b, t in members]
    compressed = rng.integers(1, 70000, sum(nblocks)).tolist()
    out = [(1 << 36) * (i + 1) + 3 * i for i in range(len(members))]
    blocks = (InflateBlock * sum(nblocks))()
    first = (C.c_uint64 * (len(members) + 1))()
    body = (C.c_uint64 * (len(members) + 1))()
    plan.bp_plan_inflate(len(members), _arr(C.c_uint64, block_size), _arr(C.c_uint64, total), _arr(C.c_uint64, nblocks),
                         _arr(C.c_uint32, compressed), _arr(C.c_uint64, out), blocks, first, body)
    at, inp = 0, 0
    for i, (b, t) in enumerate(members):
        assert first[i] == at and body[i] == inp
        for k in range(nblocks[i]):
            d = blocks[at]
            want_out = t - k * b if k + 1 == nblocks[i] else b
            assert (d.inp, d.out, d.in_bytes, d.out_bytes) == (inp, out[i] + k * b, compressed[at], want_out), (i, k)
            inp += compressed[at]
            at += 1
        assert sum(blocks[j].out_bytes for j in range(first[i], at)) == t  # the blocks tile the member's output
    assert first[len(members)] == at and body[len(members)] == inp


def test_aligned_places(plan):
    sizes = [0, 1, 15, 16, 17, 16000 * SEG + 1, 3]
    at = (C.c_uint64 * (len(sizes) + 1))()
    plan.bp_plan_aligned(_arr(C.c_uint64, sizes), len(sizes), at)
    want = np.concatenate([[0], np.cumsum([-(-s // 16) * 16 for s in sizes])]).tolist()
    assert list(at) == want


# ---- inputs ---------------------------------------------------------------------------------------------


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
def ifl():
    return build_inflate_host()


@pytest.fixture(scope="module")
def spz():
    from spz_b200 import build as B
    B.build_python_module()
    from spz_b200.pyspz import spz as module
    return module


def fibonacci(count, first=(1, 2)):
    f = list(first)
    while len(f) < count:
        f.append(f[-1] + f[-2])
    return f[:count]


def _longest_run(a):
    starts = np.concatenate([[0], np.flatnonzero(a[1:] != a[:-1]) + 1])
    return int(np.diff(np.append(starts, a.size)).max())


def deep_literal_segment(pad_to=None):
    """21 literal values with Fibonacci counts (a Huffman tree 21 levels deep): the 15-bit limit has to
    rearrange the code.  No run reaches RUN_MIN."""
    counts = fibonacci(21)
    if pad_to:
        counts.append(pad_to - sum(counts))
    base = np.repeat(np.arange(len(counts), dtype=np.uint8) * 7 + 3, counts)
    for seed in range(100):
        a = np.random.default_rng(seed).permutation(base)
        if _longest_run(a) < RUN_MIN:
            return a.tobytes()
    raise AssertionError("no seed keeps every run below RUN_MIN")


def deep_length_segment():
    """A Fibonacci histogram whose twelve rarest symbols are length codes: runs of 0xaa of 259, 228, ..., 44
    bytes with multiplicities 1, 2, 3, ..., 233 between literals of seven other values.  63902 bytes."""
    runs = [259, 228, 196, 164, 132, 116, 100, 84, 68, 60, 52, 44]
    fib = fibonacci(20)
    run_counts, lit_counts = fib[:12], fib[12:13] + fib[14:]
    for seed in range(100):
        rng = np.random.default_rng(seed)
        pool = rng.permutation(np.repeat(np.array([0x11, 0x22, 0x33, 0x44, 0x55, 0x66, 0x77], np.uint8), lit_counts))
        if _longest_run(pool) >= RUN_MIN:
            continue
        order = rng.permutation(np.repeat(np.arange(12), run_counts))
        cuts = np.sort(rng.choice(np.arange(1, pool.size), order.size, replace=False))
        parts, at = [b"\xaa"], 0
        for cut, r in zip(cuts.tolist(), order.tolist()):
            parts += [pool[at:cut].tobytes(), b"\xaa" * runs[r]]
            at = cut
        parts += [pool[at:].tobytes(), b"\xaa"]
        data = b"".join(parts)
        assert len(data) == 63902
        return data
    raise AssertionError("no seed keeps every literal run below RUN_MIN")


def tie_heavy_segment():
    """Four heavy byte values and 220 light ones of equal counts, shuffled: code lengths decided among ties."""
    light = [v for v in range(256) if v % 16][:220]
    base = np.concatenate([np.repeat(np.array([0x10, 0x20, 0x30, 0x40], np.uint8), 9000), np.repeat(np.array(light, np.uint8), 120)])
    return np.random.default_rng(4).permutation(base).tobytes()


def device_at(torch, data: bytes, offset=0):
    """data as a CUDA tensor starting `offset` bytes into a 16-byte-aligned allocation."""
    buf = torch.zeros(len(data) + offset + 16, dtype=torch.uint8, device="cuda")
    if data:
        buf[offset:offset + len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    return buf[offset:offset + len(data)]


def guarded(torch, size, offset=0):
    """(buffer, slice of `size` bytes at GUARD + offset) of a FILL-ed buffer with guard bands."""
    buf = torch.full((size + 2 * GUARD + 16,), FILL, dtype=torch.uint8, device="cuda")
    return buf, buf[GUARD + offset:GUARD + offset + size]


def bands_intact(buf, size, offset=0):
    return bool((buf[:GUARD + offset] == FILL).all()) and bool((buf[GUARD + offset + size:] == FILL).all())


def launches(ctx):
    return ctx.info()["kernel_launches"]


def to_device(torch, c):
    from spz_b200.codec import CloudPlanes
    return CloudPlanes(c.n, c.sh_degree, *[torch.from_numpy(np.asarray(p)).cuda() for p in c.planes()])


def cloud_bits(torch, c):
    return [p.view(torch.int32).cpu().numpy() for p in c.planes()]


def same_cloud(torch, a, b):
    return a.n == b.n and a.sh_degree == b.sh_degree and all(np.array_equal(x, y) for x, y in zip(cloud_bits(torch, a), cloud_bits(torch, b)))


# ---- gzip_device_batch ------------------------------------------------------------------------------------


def gzip_batch_inputs(torch):
    rng = np.random.default_rng(70)
    items = [("empty", b"", 0), ("one byte", b"\x07", 0)]
    for size in (65535, 65536, 65537):
        items.append((f"mixed {size}", mixed(rng, size), 0))
    for offset in range(1, 16):
        items.append((f"source at offset {offset}", mixed(rng, 3 * SEG + 97 * offset), offset))
    items += [("Fibonacci literals", deep_literal_segment(), 0), ("Fibonacci literals, whole segment", deep_literal_segment(SEG), 3),
              ("Fibonacci length codes", deep_length_segment(), 0), ("tie-heavy", tie_heavy_segment(), 5),
              ("deep and tied between ordinary segments",
               mixed(rng, SEG) + deep_literal_segment(SEG) + mixed(rng, SEG) + deep_length_segment() + tie_heavy_segment(), 0)]
    return [(name, data, device_at(torch, data, off)) for name, data, off in items]


@gpu
def test_gzip_device_batch_equals_single(torch, gpu_ctx, dfl):
    from spz_b200.codec import gunzip_bytes
    items = gzip_batch_inputs(torch)
    members = gpu_ctx.gzip_device_batch([t for _, _, t in items])
    assert len(members) == len(items)
    for (name, data, t), member in zip(items, members):
        assert member == gpu_ctx.gzip_device(t), name
        assert member == host_gzip(dfl, data), name
        assert gunzip_bytes(member, threads=8) == data, name
        if not data:
            continue  # an empty member's table is not one the parallel inflaters take
        got, on_device = gpu_ctx.gunzip_device(member)
        assert on_device and got.cpu().numpy().tobytes() == data, name
    assert gpu_ctx.gzip_device_batch([]) == []


@gpu
def test_gzip_device_batch_past_16000_segments(torch, gpu_ctx):
    """A member of 16000 * SEG + 1 bytes (two segments per table block) beside small ones."""
    from spz_b200.codec import gunzip_bytes, gzip_table_info
    big = (torch.arange(16000 * SEG + 1, device="cuda", dtype=torch.int64) * 2654435761 >> 13).remainder(7).to(torch.uint8)
    small = [device_at(torch, b"abc" * 1000), device_at(torch, b"", 0), device_at(torch, mixed(np.random.default_rng(71), SEG + 1), 9)]
    batch = gpu_ctx.gzip_device_batch([small[0], big, small[1], small[2]])
    assert batch[1] == gpu_ctx.gzip_device(big)
    for t, member in zip(small, [batch[0], batch[2], batch[3]]):
        assert member == gpu_ctx.gzip_device(t)
    assert gzip_table_info(batch[1]) == (16000 * SEG + 1, 8001)
    host = big.cpu().numpy().tobytes()
    assert gunzip_bytes(batch[1], threads=16) == host
    got, on_device = gpu_ctx.gunzip_device(batch[1])
    assert on_device and torch.equal(got, big)


# ---- save_spz_device_batch ----------------------------------------------------------------------------------


@gpu
def test_save_spz_device_batch_equals_single(torch, gpu_ctx):
    from spz_b200.synth import torch_cloud
    clouds, flags = [], []
    for deg in range(4):
        for n in (0, 1, 15, 16, 17, 60_000):
            clouds.append(torch_cloud(n, deg, "cuda", seed=100 * deg + n % 97))
            flags.append(bool((deg + n) % 2))
    clouds.append(torch_cloud(1_000_007, 3, "cuda", seed=5))
    flags.append(True)
    for frm in (0, 6):
        files = gpu_ctx.save_spz_device_batch(clouds, frm, antialiased=flags)
        for c, aa, blob in zip(clouds, flags, files):
            assert blob == gpu_ctx.save_spz_device(c, frm, antialiased=aa), (c.n, c.sh_degree, frm, aa)
    same_flag = gpu_ctx.save_spz_device_batch(clouds[:3], 2, antialiased=True)
    assert same_flag == [gpu_ctx.save_spz_device(c, 2, antialiased=True) for c in clouds[:3]]
    assert gpu_ctx.save_spz_device_batch([]) == []


# ---- gunzip_device_batch -------------------------------------------------------------------------------------


def zlib_member(data: bytes, block_size: int):
    """data in table blocks of block_size bytes, each a raw zlib stream of its own, framed with the "SZ" table."""
    n = max(1, -(-len(data) // block_size))
    blocks = []
    for i in range(n):
        z = zlib.compressobj(6, zlib.DEFLATED, -15)
        blocks.append(z.compress(data[i * block_size:(i + 1) * block_size]) + z.flush(zlib.Z_FINISH if i + 1 == n else zlib.Z_SYNC_FLUSH))
    return frame_member(blocks, block_size, data)


def frame_member(blocks_raw, block_size, data):
    sub = struct.pack("<IIII", block_size, len(blocks_raw), len(data) & 0xFFFFFFFF, len(data) >> 32)
    sub += b"".join(struct.pack("<I", len(b)) for b in blocks_raw)
    extra = b"SZ" + struct.pack("<H", len(sub)) + sub
    head = b"\x1f\x8b\x08\x04" + bytes(4) + b"\x00\x03" + struct.pack("<H", len(extra)) + extra
    return head + b"".join(blocks_raw) + struct.pack("<II", zlib.crc32(data), len(data) & 0xFFFFFFFF)


def single_gunzip(torch, ctx, blob, size):
    """(status, bytes, on_device) of gunzip_device alone into a buffer of `size` bytes."""
    from spz_b200 import _native as N
    out = torch.empty(max(size, 0), dtype=torch.uint8, device="cuda")
    try:
        got, on_device = ctx.gunzip_device(blob, out=out)
        return N.OK, got.cpu().numpy().tobytes(), on_device
    except N.CodecError as e:
        return e.code, None, False


def gunzip_batch_and_compare(torch, ctx, blobs, sizes, offsets=None):
    """gunzip_device_batch into guard-banded outs; every member's (status, bytes, on_device) must be what
    gunzip_device gives alone.  Returns the batch's (status, on_device) per member."""
    from spz_b200 import _native as N
    offsets = offsets or [0] * len(blobs)
    bufs = [guarded(torch, s, o) for s, o in zip(sizes, offsets)]
    failed = []
    try:
        results = ctx.gunzip_device_batch(blobs, outs=[o for _, o in bufs])
    except N.CodecError as e:
        assert e.code == N.ERR_INVALID
        failed, results = e.failed, None
    torch.cuda.synchronize()
    seen = []
    for i, (blob, size, off) in enumerate(zip(blobs, sizes, offsets)):
        buf, out = bufs[i]
        assert bands_intact(buf, size, off), f"member {i}: guard band overwritten"
        want = single_gunzip(torch, ctx, blob, size)
        if i in failed:
            assert want[0] == N.ERR_INVALID, f"member {i} failed in the batch, alone it gives {want[0]}"
            seen.append((N.ERR_INVALID, False))
            continue
        assert want[0] == N.OK, f"member {i} passed in the batch, alone it fails"
        if results is not None:
            got, on_device = results[i]
            assert got.cpu().numpy().tobytes() == want[1] and on_device == want[2], f"member {i}"
            seen.append((N.OK, on_device))
        else:  # outs of members that passed are complete; their size is the table's
            assert out[:len(want[1])].cpu().numpy().tobytes() == want[1], f"member {i}"
            seen.append((N.OK, want[2]))
    return seen


@gpu
def test_gunzip_device_batch_mixed_members(torch, gpu_ctx, dfl, monkeypatch):
    from spz_b200.codec import gzip_bytes
    monkeypatch.setenv("SPZ_B200_GZIP_THREADS", "8")
    rng = np.random.default_rng(72)
    datas = [mixed(rng, n) for n in (1, 65536, 3 * SEG + 11, 9 << 20)]
    blobs, sizes, kinds = [], [], []
    for d in datas:
        blobs.append(gpu_ctx.gzip_device(device_at(torch, d)))
        kinds.append("device deflater")
    big = mixed(rng, (9 << 20) + 5)
    blobs.append(gzip_bytes(big, threads=8))  # zlib-parallel, 1 MiB blocks
    kinds.append("zlib-parallel")
    datas.append(big)
    blobs.append(gzip.compress(datas[2]))  # no table: fails as it does alone
    kinds.append("no table")
    datas.append(datas[2])
    flipped = bytearray(blobs[2])
    flipped[-8] ^= 0x01  # CRC-32 of the trailer: the device cannot vouch, the host gives the verdict
    blobs.append(bytes(flipped))
    kinds.append("flipped CRC")
    datas.append(datas[2])
    sizes = [len(d) for d in datas]
    offsets = [i % 16 for i in range(len(blobs))]
    seen = gunzip_batch_and_compare(torch, gpu_ctx, blobs, sizes, offsets)
    for kind, (st, on_device) in zip(kinds, seen):
        if kind == "device deflater":
            assert st == 0 and on_device, kind
        if kind in ("no table", "flipped CRC"):
            assert st != 0, kind


@gpu
def test_gunzip_device_batch_hostile_members_between_valid_ones(torch, gpu_ctx, ifl, dfl, monkeypatch):
    monkeypatch.setenv("SPZ_B200_GZIP_THREADS", "8")
    rng = np.random.default_rng(73)
    blobs, sizes, valid = [], [], []
    streams = list(crafted_streams()) + list(hostile_corpus(dfl, count=600))
    for k, (name, raw, n) in enumerate(streams):
        if k % 8 == 0:
            d = mixed(rng, int(rng.integers(1, 3 * SEG)))
            blobs.append(zlib_member(d, 65536))
            sizes.append(len(d))
            valid.append(len(blobs) - 1)
        _, want = zlib_verdict(ifl, raw, n)
        blobs.append(frame_member([raw], n, want))
        sizes.append(n)
    seen = gunzip_batch_and_compare(torch, gpu_ctx, blobs, sizes)
    for i in valid:
        assert seen[i] == (0, True), f"valid member {i} did not come back on_device"


# ---- load_spz_device_batch ----------------------------------------------------------------------------------


def host_save(spz, tmp_path, c, frm=0, antialiased=False):
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


def version_container(rng, n, deg, ver):
    from util import random_stream
    p = random_stream(rng, n, deg, ver)
    head = struct.pack("<IIIBBBB", 0x5053474E, ver, n, deg, 12, 1, 0)
    return head + b"".join(np.asarray(x).tobytes() for x in (p.positions, p.alphas, p.colors, p.scales, p.rotations, p.sh))


def load_inputs(torch, ctx, spz, tmp_path, monkeypatch):
    """(name, blob, should_fail) of every kind of file the load routes see."""
    from spz_b200.synth import numpy_cloud, torch_cloud
    rng = np.random.default_rng(74)
    files = []
    for deg in range(4):
        files.append((f"save_spz_device SH{deg}", ctx.save_spz_device(torch_cloud(20_000 + 7 * deg, deg, "cuda", seed=deg), 1,
                                                                       antialiased=bool(deg % 2)), False))
    files.append(("save_spz_device 60K SH3", ctx.save_spz_device(torch_cloud(60_000, 3, "cuda", seed=9)), False))
    files.append(("0 points", ctx.save_spz_device(torch_cloud(0, 2, "cuda", seed=1)), False))
    c = numpy_cloud(30_000, 3, seed=8)
    files.append(("host saveSpz, no table", host_save(spz, tmp_path, c, 0, True), False))
    monkeypatch.setenv("SPZ_B200_GZIP_THREADS", "4")
    files.append(("host saveSpz, table", host_save(spz, tmp_path, c, 0, False), False))
    monkeypatch.delenv("SPZ_B200_GZIP_THREADS")
    for ver in (1, 2, 3):
        container = version_container(rng, 3000 + ver, ver, ver)
        files.append((f"version {ver}, no table", gzip.compress(container), False))
        files.append((f"version {ver}, 64 KiB table", zlib_member(container, 65536), False))
    good = files[1][1]
    damaged = bytearray(good)
    damaged[len(damaged) // 2] ^= 0x5A
    files.append(("damaged", bytes(damaged), True))
    files.append(("truncated", good[:len(good) // 2], True))
    return files


def guarded_cloud(torch, n, deg, fill=7.0):
    """A CloudPlanes whose planes are slices of FILL-ed buffers with guard bands: (cloud, [buffers])."""
    from spz_b200.codec import CloudPlanes, float_plane_widths
    bufs, planes = [], []
    for w in float_plane_widths(deg):
        b = torch.full((n * w + 2 * GUARD,), fill, dtype=torch.float32, device="cuda")
        bufs.append((b, n * w))
        planes.append(b[GUARD:GUARD + n * w])
    return CloudPlanes(n, deg, *planes), bufs


def guards_ok(torch, bufs, fill=7.0):
    return all(bool((b[:GUARD] == fill).all()) and bool((b[GUARD + k:] == fill).all()) for b, k in bufs)


def run_load_batch(torch, ctx, files, to):
    """load_spz_device_batch into guard-banded clouds sized from each good file: (clouds, guard buffers, failed)."""
    from spz_b200 import _native as N
    from spz_b200.codec import spz_info
    outs, guards = [], []
    for name, blob, bad in files:
        n, deg = spz_info(files[1][1] if name == "truncated" else blob)  # a damaged file's header is still readable
        cloud, bufs = guarded_cloud(torch, n, deg)
        outs.append(cloud)
        guards.append(bufs)
    failed = []
    try:
        ctx.load_spz_device_batch([b for _, b, _ in files], to=to, outs=outs)
    except N.CodecError as e:
        assert e.code == N.ERR_INVALID
        failed = e.failed
    torch.cuda.synchronize()
    return outs, guards, failed


@gpu
def test_load_spz_device_batch_equals_single(torch, gpu_ctx, spz, tmp_path, monkeypatch):
    from spz_b200 import _native as N
    files = load_inputs(torch, gpu_ctx, spz, tmp_path, monkeypatch)
    for to in (0, 6):
        outs, guards, failed = run_load_batch(torch, gpu_ctx, files, to)
        assert failed == [i for i, f in enumerate(files) if f[2]], failed
        for i, ((name, blob, bad), out, bufs) in enumerate(zip(files, outs, guards)):
            assert guards_ok(torch, bufs), f"{name}: guard band overwritten"
            if bad:
                with pytest.raises(N.CodecError) as e:
                    gpu_ctx.load_spz_device(blob, to=to)
                assert e.value.code == N.ERR_INVALID, name
                assert all(bool((p == 7.0).all()) for p in out.planes()), f"{name}: out touched"
                continue
            want, aa = gpu_ctx.load_spz_device(blob, to=to)
            assert same_cloud(torch, out, want), f"{name} to={to}"
            assert out.antialiased == aa, name
    # without outs: the clouds are allocated from the headers
    good = [(n, b) for n, b, bad in files if not bad]
    got = gpu_ctx.load_spz_device_batch([b for _, b in good], to=3)
    for (name, blob), (cloud, aa) in zip(good, got):
        want, want_aa = gpu_ctx.load_spz_device(blob, to=3)
        assert same_cloud(torch, cloud, want) and aa == want_aa, name
    assert gpu_ctx.load_spz_device_batch([]) == []


# ---- order, launches, errors ----------------------------------------------------------------------------


@gpu
def test_batches_are_order_independent(torch, gpu_ctx, spz, tmp_path, monkeypatch):
    from spz_b200.synth import torch_cloud
    rng = np.random.default_rng(75)
    clouds = [torch_cloud(int(n), d, "cuda", seed=s) for s, (n, d) in enumerate([(5000, 0), (17, 3), (0, 1), (40_000, 2), (70_001, 3), (1, 1)])]
    flags = [bool(i % 2) for i in range(len(clouds))]
    perm = rng.permutation(len(clouds)).tolist()
    files = gpu_ctx.save_spz_device_batch(clouds, 0, flags)
    permuted = gpu_ctx.save_spz_device_batch([clouds[p] for p in perm], 0, [flags[p] for p in perm])
    assert permuted == [files[p] for p in perm]
    tensors = [device_at(torch, mixed(rng, int(k)), int(o)) for k, o in zip(rng.integers(0, 5 * SEG, 9), rng.integers(0, 16, 9))]
    members = gpu_ctx.gzip_device_batch(tensors)
    perm9 = rng.permutation(9).tolist()
    assert gpu_ctx.gzip_device_batch([tensors[p] for p in perm9]) == [members[p] for p in perm9]
    inputs = load_inputs(torch, gpu_ctx, spz, tmp_path, monkeypatch)
    good = [b for _, b, bad in inputs if not bad]
    loaded = gpu_ctx.load_spz_device_batch(good)
    permn = rng.permutation(len(good)).tolist()
    again = gpu_ctx.load_spz_device_batch([good[p] for p in permn])
    for k, p in enumerate(permn):
        assert same_cloud(torch, again[k][0], loaded[p][0]) and again[k][1] == loaded[p][1]
    blobs = [m for m in members]
    unz = gpu_ctx.gunzip_device_batch(blobs)
    unz_p = gpu_ctx.gunzip_device_batch([blobs[p] for p in perm9])
    for k, p in enumerate(perm9):
        assert torch.equal(unz_p[k][0], unz[p][0]) and unz_p[k][1] == unz[p][1]


@gpu
def test_batches_share_their_launches(torch, gpu_ctx):
    """64 files: a load batch costs one inflate and one plane-move launch plus each cloud's decode launches; a save
    batch three deflate launches and one plane-move launch (which also writes the headers) plus each cloud's
    encode launches.  Loops of single calls pay the shared launches once per file."""
    from spz_b200.synth import torch_cloud
    clouds = [torch_cloud(2000 + 37 * i, i % 4, "cuda", seed=i) for i in range(64)]
    before = launches(gpu_ctx)
    singles = []
    for c in clouds:
        b = launches(gpu_ctx)
        gpu_ctx.save_spz_device(c)
        singles.append(launches(gpu_ctx) - b)
    single_total = launches(gpu_ctx) - before
    assert all(s >= 5 for s in singles)  # encode + move + 3 deflate, per file
    b = launches(gpu_ctx)
    files = gpu_ctx.save_spz_device_batch(clouds)
    assert launches(gpu_ctx) - b == single_total - 4 * (len(clouds) - 1)
    b = launches(gpu_ctx)
    for f in files:
        gpu_ctx.load_spz_device(f)
    load_single = launches(gpu_ctx) - b
    b = launches(gpu_ctx)
    gpu_ctx.load_spz_device_batch(files)
    assert launches(gpu_ctx) - b == load_single - 2 * (len(files) - 1)
    # the deflater alone: three launches for the batch, three per input in a loop
    tensors = [device_at(torch, bytes([i]) * (1000 * i)) for i in range(64)]
    b = launches(gpu_ctx)
    gpu_ctx.gzip_device_batch(tensors)
    assert launches(gpu_ctx) - b == 3
    b = launches(gpu_ctx)
    for t in tensors:
        gpu_ctx.gzip_device(t)
    assert launches(gpu_ctx) - b == 3 * len(tensors)
    b = launches(gpu_ctx)
    gpu_ctx.gunzip_device_batch(files)
    assert launches(gpu_ctx) - b == 1


@gpu
def test_batch_argument_errors_queue_nothing(torch, gpu_ctx):
    from spz_b200 import _native as N
    from spz_b200.codec import CloudPlanes, _cloud_struct, alloc_cloud
    from spz_b200.synth import torch_cloud
    L, h, stream = N.lib(), gpu_ctx._h, C.c_void_p(torch.cuda.current_stream().cuda_stream)
    sentinel = C.c_void_p(12345)
    outs, sizes = (C.c_void_p * 2)(sentinel, sentinel), (C.c_size_t * 2)(7, 7)
    b = launches(gpu_ctx)
    # null arrays
    assert L.spzb200_gzip_device_batch(h, None, None, 2, outs, sizes, stream) == N.ERR_INVALID
    assert list(outs) == [None, None] and list(sizes) == [0, 0]
    assert L.spzb200_gzip_device_batch(h, None, None, 1, None, None, stream) == N.ERR_INVALID
    assert L.spzb200_save_spz_device_batch(h, None, 2, 0, None, outs, sizes, stream) == N.ERR_INVALID
    assert L.spzb200_gunzip_device_batch(h, None, None, 2, None, None, None, None, None, stream) == N.ERR_INVALID
    assert L.spzb200_load_spz_device_batch(h, None, None, 2, 0, None, None, None, stream) == N.ERR_INVALID
    assert L.spzb200_gzip_device_batch(None, None, None, 0, None, None, stream) == N.ERR_INVALID
    assert L.spzb200_gzip_device_batch(h, None, None, -1, None, None, stream) == N.ERR_INVALID
    assert L.spzb200_gzip_device_batch(h, None, None, 0, None, None, stream) == N.OK  # count 0
    # a cloud checkSizes rejects (a null plane), beside good ones; a bad coordinate system
    good = torch_cloud(100, 1, "cuda", seed=1)
    bad = CloudPlanes(100, 1, good.positions, good.scales, good.rotations, good.alphas, good.colors, good.sh)
    structs = (N.Cloud * 3)(_cloud_struct(good, True), _cloud_struct(bad, True), _cloud_struct(good, True))
    structs[1].sh = None
    outs3, sizes3 = (C.c_void_p * 3)(sentinel, sentinel, sentinel), (C.c_size_t * 3)(1, 1, 1)
    assert L.spzb200_save_spz_device_batch(h, structs, 3, 0, None, outs3, sizes3, stream) == N.ERR_INVALID
    assert list(outs3) == [None] * 3 and list(sizes3) == [0] * 3
    structs[1].sh = structs[0].sh
    structs[1].num_points = -1
    assert L.spzb200_save_spz_device_batch(h, structs, 3, 0, None, outs3, sizes3, stream) == N.ERR_INVALID
    structs[1].num_points = 100
    assert L.spzb200_save_spz_device_batch(h, structs, 3, 9, None, outs3, sizes3, stream) == N.ERR_INVALID
    assert list(outs3) == [None] * 3
    with pytest.raises(N.CodecError):
        gpu_ctx.save_spz_device_batch([good, good], -1)
    assert launches(gpu_ctx) == b, "an argument error queued work"
    blob = gpu_ctx.save_spz_device(good)
    b = launches(gpu_ctx)
    out, bufs = guarded_cloud(torch, 100, 1)
    with pytest.raises(N.CodecError) as e:
        gpu_ctx.load_spz_device_batch([blob, blob], to=9, outs=[out, alloc_cloud(100, 1, device="cuda")])
    assert e.value.code == N.ERR_INVALID
    torch.cuda.synchronize()
    assert guards_ok(torch, bufs) and all(bool((p == 7.0).all()) for p in out.planes())
    assert launches(gpu_ctx) == b, "an argument error queued work"
