"""The device deflater's format (spz_b200/csrc/deflate_format.cuh) compiled for the HOST
(tests/host_emul/deflate_host.cc) and checked without a GPU: length-limited code lengths against
Huffman and package-merge optima computed here, single segments against Python's zlib inflater, and
whole members -- framed by the library's own block-table writer -- against gzip and spzb200_gunzip.
The -m gpu tests (test_device_file.py) compare the kernels' output with this host build byte for byte."""
from __future__ import annotations

import ctypes as C
import gzip
import heapq
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEG = 65536
RUN_MIN = 12  # deflate_format.cuh: kRunMin
SLOT = SEG + 64


def build_deflate_host():
    """tests/host_emul/_build/libdeflate_host.so, linked against the in-tree library (its gzip framing)."""
    from spz_b200 import _native
    from spz_b200 import build as B
    _native.lib()
    here = os.path.join(ROOT, "tests", "host_emul")
    out_dir = os.path.join(here, "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libdeflate_host.so")
    deps = [os.path.join(here, "deflate_host.cc"), B.LIB] + [os.path.join(ROOT, "spz_b200", "csrc", h)
                                                            for h in ("deflate_format.cuh", "spz_internal.hpp")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", deps[0], "-o", so, "-L", B.OUT_DIR, "-lspz_b200",
                        "-Wl,-rpath," + B.OUT_DIR], check=True)
    lib = C.CDLL(so)
    lib.dfl_build_lengths.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.dfl_encode_segment.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
    lib.dfl_gzip.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
    lib.dfl_free.argtypes = [C.c_void_p]
    return lib


@pytest.fixture(scope="module")
def dfl():
    return build_deflate_host()


def lengths(dfl, freq, max_bits):
    f = np.ascontiguousarray(freq, np.uint32)
    out = np.zeros(f.size, np.uint8)
    assert dfl.dfl_build_lengths(f.ctypes.data, f.size, max_bits, out.ctypes.data) == 0
    return out.astype(np.int64)


def encode_segment(dfl, data: bytes, last: bool):
    a = np.frombuffer(data, np.uint8)
    out = np.zeros(SLOT, np.uint8)
    dyn = C.c_int(0)
    n = dfl.dfl_encode_segment(a.ctypes.data if a.size else None, a.size, int(last), out.ctypes.data, C.byref(dyn))
    return out[:n].tobytes(), bool(dyn.value)


def host_gzip(dfl, data: bytes) -> bytes:
    a = np.frombuffer(data, np.uint8)
    p, n = C.c_void_p(None), C.c_size_t(0)
    assert dfl.dfl_gzip(a.ctypes.data if a.size else None, a.size, C.byref(p), C.byref(n)) == 0
    try:
        return C.string_at(p.value, n.value)
    finally:
        dfl.dfl_free(p)


def huffman_cost(freq):
    f = [int(x) for x in freq if x]
    if len(f) < 2:
        return sum(f)
    h = list(f)
    heapq.heapify(h)
    cost = 0
    while len(h) > 1:
        a, b = heapq.heappop(h), heapq.heappop(h)
        cost += a + b
        heapq.heappush(h, a + b)
    return cost


def huffman_depth(freq):
    f = [int(x) for x in freq if x]
    h = [(x, 0, i) for i, x in enumerate(f)]
    heapq.heapify(h)
    k = len(f)
    while len(h) > 1:
        a, b = heapq.heappop(h), heapq.heappop(h)
        heapq.heappush(h, (a[0] + b[0], max(a[1], b[1]) + 1, k))
        k += 1
    return h[0][1]


def package_merge_cost(freq, max_bits):
    """Optimal length-limited cost: coin collector over symbol-count vectors."""
    w = np.array([int(x) for x in freq if x], np.int64)
    n = w.size
    leaves = [(int(w[i]), np.eye(n, dtype=np.int64)[i]) for i in np.argsort(w, kind="stable")]
    cur = list(leaves)
    for _ in range(max_bits - 1):
        pk = [(cur[2 * i][0] + cur[2 * i + 1][0], cur[2 * i][1] + cur[2 * i + 1][1]) for i in range(len(cur) // 2)]
        cur = sorted(leaves + pk, key=lambda t: t[0])
    lens = sum(v for _, v in cur[:2 * n - 2])
    return int((lens * w).sum())


def check_prefix_code(lens, max_bits):
    used = lens[lens > 0]
    assert used.size >= 2 and used.max() <= max_bits
    assert sum(2.0 ** -int(x) for x in used) == 1.0  # complete: Kraft sum exactly one


@pytest.mark.parametrize("max_bits,nsym", [(15, 286), (15, 40), (7, 19)])
def test_code_lengths_random_histograms(dfl, max_bits, nsym):
    rng = np.random.default_rng(max_bits * 1000 + nsym)
    for trial in range(40):
        freq = rng.integers(0, [2, 20, 1000, 65536][trial % 4], nsym).astype(np.uint32)
        freq[rng.random(nsym) < 0.3] = 0
        if np.count_nonzero(freq) < 2:
            freq[:2] = 1
        lens = lengths(dfl, freq, max_bits)
        check_prefix_code(lens, max_bits)
        assert np.all((lens > 0) == (freq > 0))
        cost = int((lens * freq.astype(np.int64)).sum())
        if huffman_depth(freq) <= max_bits:
            assert cost == huffman_cost(freq)
        else:
            assert cost <= package_merge_cost(freq, max_bits) * 1.005


@pytest.mark.parametrize("max_bits,nsym", [(15, 286), (7, 19)])
def test_code_lengths_one_and_two_symbols(dfl, max_bits, nsym):
    for used in ([5], [0], [nsym - 1], [3, 9], [0, 1]):
        freq = np.zeros(nsym, np.uint32)
        freq[used] = [7] * len(used)
        lens = lengths(dfl, freq, max_bits)
        check_prefix_code(lens, max_bits)  # a lone symbol gets a partner: two codes of one bit
        assert all(lens[u] == 1 for u in used) and np.count_nonzero(lens) == 2


@pytest.mark.parametrize("max_bits,nsym,count", [(15, 286, 18), (15, 286, 24), (15, 40, 40), (7, 19, 9), (7, 19, 19)])
def test_code_lengths_fibonacci_deeper_than_limit(dfl, max_bits, nsym, count):
    fib = [1, 1]
    while len(fib) < count:
        fib.append(fib[-1] + fib[-2])
    freq = np.zeros(nsym, np.uint32)
    freq[:count] = [min(f, 4096) for f in fib]  # a segment's symbol counts sum to at most 65536 + 1
    assert huffman_depth(freq) > max_bits
    lens = lengths(dfl, freq, max_bits)
    check_prefix_code(lens, max_bits)
    cost = int((lens * freq.astype(np.int64)).sum())
    assert cost <= package_merge_cost(freq, max_bits) * 1.005


def _inflate_raw(data: bytes) -> bytes:
    z = zlib.decompressobj(-15)
    return z.decompress(data) + z.flush()


def segment_cases():
    rng = np.random.default_rng(5)
    skew = np.minimum(rng.geometric(0.25, SEG), 255).astype(np.uint8).tobytes()
    yield "empty", b"", False
    yield "one byte", b"\x07", False
    yield "zeros", bytes(SEG), True
    yield "constant 0x80", b"\x80" * SEG, True
    yield "uniform random", rng.integers(0, 256, SEG, dtype=np.uint8).tobytes(), False
    yield "skewed", skew, True
    yield "short skewed", skew[:1000], True
    for run in (RUN_MIN - 1, RUN_MIN, RUN_MIN + 1, 258, 259, 260, 261, 516, 40000):
        body = bytearray(skew[:5000])
        body[100:100 + run] = b"\x33" * run
        yield f"run {run}", bytes(body), True
    yield "runs everywhere", b"".join(bytes([i % 251]) * (i % 40 + 1) for i in range(3000))[:SEG], True


@pytest.mark.parametrize("last", [True, False])
def test_single_segments_inflate_with_zlib(dfl, last):
    for name, data, want_dynamic in segment_cases():
        coded, dynamic = encode_segment(dfl, data, last)
        assert dynamic == want_dynamic, name
        assert _inflate_raw(coded) == data, name
        assert len(coded) <= len(data) + 10, name
        if not last:  # ends byte-aligned with a sync marker or a stored block: segments concatenate
            z = zlib.decompressobj(-15)
            assert z.decompress(coded + coded) == data + data, name


def test_run_segment_is_small(dfl):
    coded, _ = encode_segment(dfl, bytes(SEG), False)
    assert len(coded) < SEG // 500


def test_member_with_64k_blocks_reads_with_gzip_and_gunzip(dfl):
    from spz_b200.codec import gunzip_bytes
    rng = np.random.default_rng(9)
    for size in (0, 1, SEG - 1, SEG, SEG + 1, 3 * SEG + 7, 20 * SEG + 123):
        data = np.minimum(rng.geometric(0.1, size), 255).astype(np.uint8).tobytes()
        if size > 2 * SEG:
            data = data[:SEG] + rng.integers(0, 256, SEG, dtype=np.uint8).tobytes() + bytes(SEG) + data[3 * SEG:]
        member = host_gzip(dfl, data)
        assert gzip.decompress(member) == data
        assert gunzip_bytes(member, threads=8) == data
        xlen, = struct.unpack_from("<H", member, 10)
        assert member[12:14] == b"SZ"
        block_size, blocks = struct.unpack_from("<II", member, 16)
        assert block_size == SEG and blocks == max(1, -(-size // SEG))


def test_damaged_member_is_rejected(dfl):
    from spz_b200 import _native as N
    from spz_b200.codec import gunzip_bytes
    data = np.minimum(np.random.default_rng(2).geometric(0.1, 5 * SEG), 255).astype(np.uint8).tobytes()
    member = bytearray(host_gzip(dfl, data))
    member[-8] ^= 1  # CRC
    with pytest.raises(N.CodecError):
        gunzip_bytes(bytes(member), threads=8)
