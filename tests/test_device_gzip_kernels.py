"""The device deflate and inflate kernels held to their host builds (test_device_deflate_host.py,
test_device_inflate_host.py) on every input those builds are vetted on, at the geometries only the GPU
runs: the inflater's lane-parallel table fill, copies and CRC tree, both of its warp geometries and
under-aligned outputs; the deflater's per-slice tokens, package-merge at the 15-bit limit, tie order,
stored/dynamic choice, unaligned staging and segment-count boundaries.

Every input first passes the host build in the same test.  Then the GPU must agree exactly: the same
bytes, the same verdict, and -- since a member whose kernel output fails its CRC quietly takes the host
route and still returns the right bytes -- `on_device` wherever the host build vouches for the member.

The block-table framer, the deep-code and tie-heavy segments and their checks against zlib need no GPU;
every other test is -m gpu."""
from __future__ import annotations

import bisect
import gzip
import hashlib
import struct
import zlib

import numpy as np
import pytest

from test_device_deflate_host import RUN_MIN, SEG, build_deflate_host, encode_segment, host_gzip, huffman_depth
from test_device_inflate_host import (assert_member_on_device_route, build_inflate_host, crafted_streams, hostile_corpus,
                                      inflate_guarded, member_on_device_route, mixed, skewed, zlib_verdict)

gpu = pytest.mark.gpu

GUARD = 4096
FILL = 0xA5


@pytest.fixture(scope="module")
def ifl():
    return build_inflate_host()


@pytest.fixture(scope="module")
def dfl():
    return build_deflate_host()


@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


# ---- members framed block by block -----------------------------------------------------------------------


def frame_member(blocks_raw, block_size, data):
    """A gzip member with the "SZ" block table laid out as frameBlockMember writes it (block size, count, total
    as lo / hi, one compressed size per block), the blocks' raw deflate bytes, then CRC-32 and ISIZE of data."""
    sub = struct.pack("<IIII", block_size, len(blocks_raw), len(data) & 0xFFFFFFFF, len(data) >> 32)
    sub += b"".join(struct.pack("<I", len(b)) for b in blocks_raw)
    extra = b"SZ" + struct.pack("<H", len(sub)) + sub
    head = b"\x1f\x8b\x08\x04" + bytes(4) + b"\x00\x03" + struct.pack("<H", len(extra)) + extra
    return head + b"".join(blocks_raw) + struct.pack("<II", zlib.crc32(data), len(data) & 0xFFFFFFFF)


# (level, strategy, sync flush every n bytes inside the block): every block type and match shape zlib writes
STYLES = {
    "level 0": (0, zlib.Z_DEFAULT_STRATEGY, 0),
    "level 1": (1, zlib.Z_DEFAULT_STRATEGY, 0),
    "level 6": (6, zlib.Z_DEFAULT_STRATEGY, 0),
    "level 9": (9, zlib.Z_DEFAULT_STRATEGY, 0),
    "Z_FIXED": (6, zlib.Z_FIXED, 0),
    "Z_RLE": (6, zlib.Z_RLE, 0),
    "Z_HUFFMAN_ONLY": (6, zlib.Z_HUFFMAN_ONLY, 0),
    "sync-flushed": (6, zlib.Z_DEFAULT_STRATEGY, 50_000),
}


def deflate_block(chunk: bytes, last: bool, style="level 6"):
    """One table block: a fresh raw stream, so it decodes on its own; ended by Z_SYNC_FLUSH, or Z_FINISH when last."""
    level, strategy, flush_every = STYLES[style]
    z = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    out = b""
    step = flush_every or max(len(chunk), 1)
    for i in range(0, len(chunk), step):
        out += z.compress(chunk[i:i + step])
        if flush_every:
            out += z.flush(zlib.Z_SYNC_FLUSH)
    return out + z.flush(zlib.Z_FINISH if last else zlib.Z_SYNC_FLUSH)


def zlib_member(data: bytes, block_size: int, styles=("level 6",)):
    """data in table blocks of block_size bytes, block i deflated in styles[i % len(styles)]."""
    n = max(1, -(-len(data) // block_size))
    blocks = [deflate_block(data[i * block_size:(i + 1) * block_size], i + 1 == n, styles[i % len(styles)]) for i in range(n)]
    return frame_member(blocks, block_size, data)


def test_framer_members_read_everywhere(ifl):
    """No GPU: framed members are gzip members, carry a table the library trusts, and pass the host build of
    the device route -- so a GPU test that fails on them fails because of the kernel."""
    from spz_b200.codec import gunzip_bytes, gzip_table_info
    rng = np.random.default_rng(60)
    data = mixed(rng, 300_001)
    for block_size, styles in ((65536, tuple(STYLES)), (4097, ("level 0", "Z_FIXED", "level 9")), (300_001, ("level 1",)),
                               (17, ("level 6",))):
        what = f"block size {block_size}"
        part = data if block_size > 17 else data[:5000]
        member = zlib_member(part, block_size, styles)
        assert member[12:14] == b"SZ"
        assert gzip_table_info(member) == (len(part), -(-len(part) // block_size)), what
        assert gzip.decompress(member) == part, what
        assert gunzip_bytes(member, threads=8) == part, what
        assert member_on_device_route(ifl, member) == (1, part), what
    one = frame_member([deflate_block(b"x", True)], 1, b"x")
    assert gzip.decompress(one) == b"x" and gzip_table_info(one) == (1, 1)


# ---- segments the deflater's code has to cope with ----------------------------------------------------


_LENGTH_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]


def segment_histogram(data: bytes):
    """The literal/length symbol counts of one segment as the format tokenizes it (maximal runs, runTokens),
    end-of-block included: a restatement in Python, so tests can state what a segment's code must cope with."""
    freq = np.zeros(286, np.int64)
    a = np.frombuffer(data, np.uint8)
    if a.size:
        starts = np.concatenate([[0], np.flatnonzero(a[1:] != a[:-1]) + 1])
        for s, n in zip(starts.tolist(), np.diff(np.append(starts, a.size)).tolist()):
            if n < RUN_MIN:
                freq[a[s]] += n
                continue
            freq[a[s]] += 1
            m = n - 1
            while m >= 3:
                take = min(m, 258)
                if 0 < m - take < 3:
                    take = m - 3
                freq[256 + bisect.bisect_right(_LENGTH_BASE, take)] += 1
                m -= take
            freq[a[s]] += m
    freq[256] = 1
    return freq


def fibonacci(count, first=(1, 2)):
    f = list(first)
    while len(f) < count:
        f.append(f[-1] + f[-2])
    return f[:count]


def _longest_run(a):
    starts = np.concatenate([[0], np.flatnonzero(a[1:] != a[:-1]) + 1])
    return int(np.diff(np.append(starts, a.size)).max())


def deep_literal_segment(pad_to=None):
    """21 literal values with Fibonacci counts 1, 2, 3, ..., 17711 (46366 bytes): with the end-of-block code's
    count of 1 the histogram is the Fibonacci sequence itself, whose Huffman tree is 21 levels deep, so the
    15-bit limit has to rearrange the code.  Shuffled with the first seed that leaves no run of RUN_MIN."""
    counts = fibonacci(21)
    if pad_to:
        counts.append(pad_to - sum(counts))
    base = np.repeat(np.arange(len(counts), dtype=np.uint8) * 7 + 3, counts)
    for seed in range(100):
        a = np.random.default_rng(seed).permutation(base)
        if _longest_run(a) < RUN_MIN:
            return a.tobytes()
    raise AssertionError("no seed keeps every run below RUN_MIN")


def deep_length_segment(pad_to=None):
    """A Fibonacci histogram (with end-of-block) whose twelve rarest symbols are length codes: runs of one byte
    value A of 259, 228, 196, ..., 44 bytes (length symbols 285 down to 274, one run length each) with
    multiplicities 1, 2, 3, ..., 233, each run between literals of seven other values counted 377, 987, ...,
    10946; A's literal count (one per run, plus an A at either end) is 610.  63902 bytes."""
    runs = [259, 228, 196, 164, 132, 116, 100, 84, 68, 60, 52, 44]
    fib = fibonacci(20)  # 1, 2, 3, ..., 10946
    run_counts, a_count, lit_counts = fib[:12], fib[13], fib[12:13] + fib[14:]
    assert a_count == sum(run_counts) + 2
    if pad_to:
        lit_counts.append(pad_to - 63902)
    for seed in range(100):
        rng = np.random.default_rng(seed)
        pool = rng.permutation(np.repeat(np.array([0x11, 0x22, 0x33, 0x44, 0x55, 0x66, 0x77, 0x88][:len(lit_counts)], np.uint8), lit_counts))
        if _longest_run(pool) >= RUN_MIN:
            continue
        order = rng.permutation(np.repeat(np.arange(12), run_counts))
        cuts = np.sort(rng.choice(np.arange(1, pool.size), order.size, replace=False))  # distinct: a literal between runs
        parts, at = [b"\xaa"], 0
        for cut, r in zip(cuts.tolist(), order.tolist()):
            parts += [pool[at:cut].tobytes(), b"\xaa" * runs[r]]
            at = cut
        parts += [pool[at:].tobytes(), b"\xaa"]
        data = b"".join(parts)
        assert len(data) == (pad_to or 63902)
        return data
    raise AssertionError("no seed keeps every literal run below RUN_MIN")


def tie_heavy_segment():
    """Four heavy byte values of 9000 each and 220 light ones of 120 each, shuffled: compressible, with the
    code's lengths decided among hundreds of equal frequencies (the (frequency, symbol) rank order)."""
    light = [v for v in range(256) if v % 16][:220]
    base = np.concatenate([np.repeat(np.array([0x10, 0x20, 0x30, 0x40], np.uint8), 9000),
                           np.repeat(np.array(light, np.uint8), 120)])
    return np.random.default_rng(4).permutation(base).tobytes()


def test_deep_and_tied_segments_are_what_they_claim(dfl):
    """No GPU: the segments' histograms are what their names say, and the host model codes them dynamic."""
    lit = segment_histogram(deep_literal_segment())
    assert sorted(lit[lit > 0].tolist()) == [1] + fibonacci(21)
    ln = segment_histogram(deep_length_segment())
    assert sorted(ln[ln > 0].tolist()) == [1] + fibonacci(20)
    assert set((np.flatnonzero(ln[257:]) + 257).tolist()) == set(range(274, 286))  # the rarest twelve after end-of-block
    assert sorted(ln[274:286].tolist()) == fibonacci(12)
    for make in (deep_literal_segment, deep_length_segment):
        for pad in (None, SEG):
            data = make(pad)
            assert huffman_depth(segment_histogram(data)) > 15, make.__name__
            assert encode_segment(dfl, data, False)[1], make.__name__
    tie = segment_histogram(tie_heavy_segment())
    assert np.count_nonzero(tie == 120) >= 200
    assert encode_segment(dfl, tie_heavy_segment(), False)[1]


def deep_and_tied_segments():
    """(name, segment): codes the 15-bit limit has to rearrange, and a code built among hundreds of tied frequencies."""
    yield "Fibonacci literals", deep_literal_segment()
    yield "Fibonacci literals, whole segment", deep_literal_segment(SEG)
    yield "Fibonacci length codes", deep_length_segment()
    yield "Fibonacci length codes, whole segment", deep_length_segment(SEG)
    yield "tie-heavy", tie_heavy_segment()


def _inflate_raw(data: bytes) -> bytes:
    z = zlib.decompressobj(-15)
    return z.decompress(data) + z.flush()


@pytest.mark.parametrize("last", [True, False])
def test_deep_and_tied_segments_inflate_with_zlib(dfl, last):
    """No GPU: the host model against zlib on these segments as whole segments, not only as histograms."""
    for name, data in deep_and_tied_segments():
        coded, dynamic = encode_segment(dfl, data, last)
        assert dynamic, name
        assert _inflate_raw(coded) == data, name
        assert len(coded) < len(data), name
        if not last:  # ends byte-aligned with a sync marker: segments concatenate
            assert zlib.decompressobj(-15).decompress(coded + coded) == data + data, name


# ---- the inflater on the GPU ------------------------------------------------------------------------------


def gunzip_at(torch, ctx, blob, size, offset=0):
    """gunzip_device into out = a slice at byte `offset` of a guard-banded buffer; (bytes, on_device).  The
    bands are checked after the call, whether it returned or raised."""
    buf = torch.full((size + 2 * GUARD,), FILL, dtype=torch.uint8, device="cuda")
    try:
        got, on_device = ctx.gunzip_device(blob, out=buf[GUARD + offset:GUARD + offset + size])
        result = (got.cpu().numpy().tobytes(), on_device)
    finally:
        torch.cuda.synchronize()
        assert bool((buf[:GUARD + offset] == FILL).all()), "guard band before out overwritten"
        assert bool((buf[GUARD + offset + size:] == FILL).all()), "guard band after out overwritten"
    return result


def assert_inflates_on_device(torch, ctx, ifl, member, data, what, offset=0):
    assert_member_on_device_route(ifl, member, data, what)  # the host build vouches for it first
    got, on_device = gunzip_at(torch, ctx, member, len(data), offset)
    assert on_device, f"{what}: the kernel did not vouch for a member its host build inflates"
    assert got == data, what


@gpu
@pytest.mark.parametrize("style", list(STYLES))
def test_zlib_styles(torch, gpu_ctx, ifl, style):
    data = mixed(np.random.default_rng(61), (3 << 20) + 4321)
    assert_inflates_on_device(torch, gpu_ctx, ifl, zlib_member(data, 262144, (style,)), data, style)


def long_match_cases():
    rng = np.random.default_rng(62)
    window = rng.integers(0, 256, 32768, dtype=np.uint8).tobytes()
    yield "distance 32768", window + window[:258] + window
    for length in (255, 256, 257, 258):  # one match of each length, near and at the window's far end
        phrase = rng.integers(0, 256, length, dtype=np.uint8).tobytes()
        filler = rng.integers(0, 256, 500, dtype=np.uint8).tobytes()
        yield f"length {length}", phrase + filler + phrase + window[:32768 - length] + phrase
    for d in range(1, 41):  # overlapping copies below, at and above the 32 lanes
        yield f"overlapping distance {d}", bytes([(7 * i + d) & 0xFF for i in range(d)]) * (6000 // d + 1) + b"\x00" * (d % 5)


@gpu
def test_long_and_overlapping_matches(torch, gpu_ctx, ifl):
    for name, data in long_match_cases():
        for level in (1, 9):
            for block_size in (len(data), 4099):
                what = f"{name}, level {level}, blocks of {block_size}"
                assert_inflates_on_device(torch, gpu_ctx, ifl, zlib_member(data, block_size, (f"level {level}",)), data, what)


@gpu
@pytest.mark.parametrize("block_size", [1, 15, 16, 17, 31, 32, 33, 4095, 4097, 65536, 65537])
def test_block_sizes(torch, gpu_ctx, ifl, block_size):
    """Slices that start unaligned, lanes whose CRC chunk is empty, slices shorter than one lane's chunk; the last
    block of one byte and of a whole block."""
    blocks = 40 if block_size < 64 else 5
    rng = np.random.default_rng(63 + block_size)
    styles = ("level 0", "Z_FIXED", "level 6", "Z_RLE", "level 9")
    for total in (block_size * (blocks - 1) + 1, block_size * blocks):
        data = mixed(rng, total) if block_size > 64 else skewed(rng, total, 0.3)
        assert_inflates_on_device(torch, gpu_ctx, ifl, zlib_member(data, block_size, styles), data, f"{block_size} x {blocks}, {total} bytes")


@gpu
def test_warp_geometry_boundary(torch, gpu_ctx, ifl):
    """8 * SMs blocks is the first count that runs 8 warps per CTA (one below runs 1); one above leaves 7 idle
    warps in the last CTA.  4 KiB blocks with stored, fixed and dynamic blocks side by side."""
    sm = gpu_ctx.info()["sm_count"]
    assert sm > 0
    data = mixed(np.random.default_rng(64), (8 * sm + 1) * 4096)
    styles = ("level 0", "Z_FIXED", "level 6", "Z_HUFFMAN_ONLY", "level 1", "Z_RLE", "level 9")
    for blocks in (8 * sm - 1, 8 * sm, 8 * sm + 1):
        part = data[:blocks * 4096 - 1000]
        assert_inflates_on_device(torch, gpu_ctx, ifl, zlib_member(part, 4096, styles), part, f"{blocks} blocks")


@gpu
def test_under_aligned_out(torch, gpu_ctx, ifl):
    data = mixed(np.random.default_rng(65), 20 * 4097 + 3)
    member = zlib_member(data, 4097, ("level 6", "level 0", "Z_FIXED"))
    for offset in range(1, 16):
        assert_inflates_on_device(torch, gpu_ctx, ifl, member, data, f"out at byte offset {offset}", offset)


@gpu
def test_crafted_and_hostile_streams_get_the_host_builds_verdict(torch, gpu_ctx, ifl, dfl, monkeypatch):
    """Every stream of the hostile corpus as a one-block member: the kernel vouches exactly when the host build
    accepts, and gunzip_device returns what gunzip_bytes returns (bytes or the error)."""
    from spz_b200 import _native as N
    from spz_b200.codec import gunzip_bytes, gzip_table_info
    monkeypatch.setenv("SPZ_B200_GZIP_THREADS", "8")  # gunzip_device's host route as gunzip_bytes(threads=8)
    streams = list(crafted_streams()) + list(hostile_corpus(dfl))
    ran = 0
    for name, raw, n in streams:
        st, _ = inflate_guarded(ifl, raw, n)
        assert st >= 0, f"{name}: the host build touched memory outside the block ({st})"
        ok, want = zlib_verdict(ifl, raw, n)
        member = frame_member([raw], n, want)  # the trailer CRC is zlib's bytes' when zlib accepts
        try:
            gzip_table_info(member)
        except N.CodecError:
            continue  # a table the parser refuses (beyond 1032:1): no route reaches the kernel
        try:
            expected = gunzip_bytes(member, threads=8)
        except N.CodecError as e:
            expected = e.code
        try:
            got, on_device = gunzip_at(torch, gpu_ctx, member, n)
        except N.CodecError as e:
            got, on_device = e.code, False
        assert on_device == (st == 0), f"{name}: host build status {st}, kernel vouched {on_device}"
        assert got == expected, name
        ran += 1
    assert ran >= 0.9 * len(streams), (ran, len(streams))


# ---- the deflater on the GPU ------------------------------------------------------------------------------


def device_buffer(torch, data: bytes, offset=0):
    """data as a CUDA tensor starting `offset` bytes into its allocation, which is at least 16-byte aligned."""
    buf = torch.zeros(len(data) + offset + 16, dtype=torch.uint8, device="cuda")
    if data:
        buf[offset:offset + len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    return buf[offset:offset + len(data)]


def assert_deflates_like_host(torch, ctx, dfl, data: bytes, what, offset=0):
    want = host_gzip(dfl, data)
    assert gzip.decompress(want) == data, what  # the host build first
    src = device_buffer(torch, data, offset)
    assert src.data_ptr() % 16 == offset % 16
    member = ctx.gzip_device(src)
    assert member == want, f"{what}: the kernels' member differs from the host build's"
    assert gzip.decompress(member) == data, what
    got, on_device = gunzip_at(torch, ctx, member, len(data))
    assert on_device and got == data, what


def ordinary(seed, size=SEG):
    return mixed(np.random.default_rng(seed), size)


@gpu
def test_deep_codes(torch, gpu_ctx, dfl):
    """Segments whose Huffman code is deeper than 15 bits: package-merge's length limit on the device."""
    for make in (deep_literal_segment, deep_length_segment):
        for pad in (None, SEG):
            seg = make(pad)
            assert huffman_depth(segment_histogram(seg)) > 15, make.__name__
            assert encode_segment(dfl, seg, True)[1] and encode_segment(dfl, seg, False)[1], make.__name__
            assert_deflates_like_host(torch, gpu_ctx, dfl, seg, f"{make.__name__}({pad}) alone")
            if pad:
                data = ordinary(70) + seg + ordinary(71) + seg + ordinary(72, 999)
                assert_deflates_like_host(torch, gpu_ctx, dfl, data, f"{make.__name__} between ordinary segments")


@gpu
def test_tie_heavy_segments(torch, gpu_ctx, dfl):
    seg = tie_heavy_segment()
    assert np.count_nonzero(segment_histogram(seg) == 120) >= 200
    assert encode_segment(dfl, seg, False)[1]
    assert_deflates_like_host(torch, gpu_ctx, dfl, seg, "tie-heavy alone")
    padded = seg + skewed(np.random.default_rng(73), SEG - len(seg), 0.02)
    assert encode_segment(dfl, padded, False)[1]
    assert_deflates_like_host(torch, gpu_ctx, dfl, ordinary(74) + padded + padded + seg, "tie-heavy between segments")


def boundary_pair(dfl, size, last):
    """Two segments of `size` bytes one byte apart on the way from skewed to random bytes, the first coded
    dynamic and the second stored: bisected with the host model."""
    rng = np.random.default_rng(75 + size)
    rnd, sk = rng.integers(0, 256, size, dtype=np.uint8).tobytes(), skewed(rng, size, 0.02)
    seg = lambda k: rnd[:k] + sk[k:]  # noqa: E731
    lo, hi = 0, size
    assert encode_segment(dfl, seg(lo), last)[1] and not encode_segment(dfl, seg(hi), last)[1]
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if encode_segment(dfl, seg(mid), last)[1]:
            lo = mid
        else:
            hi = mid
    return seg(lo), seg(hi)


@gpu
def test_dynamic_stored_boundary(torch, gpu_ctx, dfl):
    dyn, stored = boundary_pair(dfl, SEG, False)
    for tail_size in (SEG - 1, 4097):
        tail_dyn, tail_stored = boundary_pair(dfl, tail_size, True)
        for tail in (tail_dyn, tail_stored):
            data = dyn + stored + stored + dyn + dyn + stored + tail
            assert_deflates_like_host(torch, gpu_ctx, dfl, data, f"alternating, last segment of {tail_size} bytes")


@gpu
def test_under_aligned_sources(torch, gpu_ctx, dfl):
    """Sources at src & 15 != 0 are staged without the bulk copy; aligned sizes just past a segment take its tail."""
    rng = np.random.default_rng(76)
    base = bytearray(skewed(rng, 3 * SEG + 64, 0.2))
    base[SEG - 20:SEG + 20] = b"\xee" * 40  # a run across a segment edge
    for size in (1, 15, 16, 17, SEG - 1, SEG, SEG + 1, 3 * SEG + 5):
        for offset in range(1, 16):
            assert_deflates_like_host(torch, gpu_ctx, dfl, bytes(base[:size]), f"{size} bytes at offset {offset}", offset)
    for size in (SEG + 15, SEG + 16, SEG + 17):
        assert_deflates_like_host(torch, gpu_ctx, dfl, bytes(base[:size]), f"{size} bytes aligned")


def slice_edge_segment(rng):
    """Runs of a byte the background never holds, placed against the kernel's 128-byte slices."""
    seg = bytearray(rng.integers(0, 4, SEG, dtype=np.uint8).tobytes())
    S = 128
    runs = [(5 * S, 40),                  # starts at a slice boundary
            (9 * S - 40, 40),             # ends at one
            (12 * S - 1, RUN_MIN),        # RUN_MIN, one byte before the boundary
            (15 * S - RUN_MIN + 1, RUN_MIN),  # RUN_MIN, one byte past it
            (18 * S - RUN_MIN, RUN_MIN),  # RUN_MIN ending at it
            (21 * S, RUN_MIN - 1),        # one short of a match, from a boundary
            (24 * S, S),                  # exactly one slice
            (27 * S, 2 * S),              # exactly two slices
            (31 * S - 5, 3 * S + 10),     # through two whole slices
            (40 * S - 1, 259 + 1)]        # a 258-match crossing
    for at, n in runs:
        seg[at:at + n] = b"\xee" * n
    return bytes(seg)


@gpu
def test_slice_edges(torch, gpu_ctx, dfl):
    rng = np.random.default_rng(77)
    edge = slice_edge_segment(rng)
    assert_deflates_like_host(torch, gpu_ctx, dfl, edge, "runs at slice edges")
    all_but_last = b"\x5c" * (SEG - 1) + b"\x5d"
    all_but_first = b"\x5d" + b"\x5c" * (SEG - 1)
    data = ordinary(78) + all_but_last + edge + all_but_first + all_but_last + ordinary(79, 3 * 128 + 7)
    assert_deflates_like_host(torch, gpu_ctx, dfl, data, "whole-segment runs between segments")


def tiled(seed, size):
    """size bytes of a mixed pattern whose period is not a multiple of the segment, so segments differ."""
    return np.resize(np.frombuffer(ordinary(seed, 3 * SEG + 12345), np.uint8), size).tobytes()


@gpu
def test_segment_offsets_scan_past_1024_segments(torch, gpu_ctx, dfl):
    """Above 1024 segments a thread of the offset scan sums several."""
    for size in (1024 * SEG, 1024 * SEG + 1):
        assert_deflates_like_host(torch, gpu_ctx, dfl, tiled(80, size), f"{size} bytes")


@gpu
def test_two_segments_per_table_block_past_16000_segments(torch, gpu_ctx, dfl):
    """Above 16000 segments each table block holds two.  About 1 GiB each: compared by SHA-256."""
    data = tiled(81, 16000 * SEG + 1)
    for size in (16000 * SEG, 16000 * SEG + 1):
        view = memoryview(data)[:size]
        want = host_gzip(dfl, view)
        digest = hashlib.sha256(view).digest()
        assert hashlib.sha256(gzip.decompress(want)).digest() == digest, size
        _, blocks = struct.unpack_from("<II", want, 16)
        assert blocks == (16000 if size == 16000 * SEG else 8001), size
        member = gpu_ctx.gzip_device(device_buffer(torch, bytes(view)))
        assert hashlib.sha256(member).digest() == hashlib.sha256(want).digest(), size  # so it inflates as want did
        del want
        out, on_device = gpu_ctx.gunzip_device(member)
        assert on_device and hashlib.sha256(out.cpu().numpy()).digest() == digest, size
        del out, member
        torch.cuda.empty_cache()
