"""The device inflater's decoder (spz_b200/csrc/inflate_format.cuh) compiled for the HOST
(tests/host_emul/inflate_host.cc) and checked without a GPU: valid members and raw streams against
zlib, a seeded corpus of hostile streams against zlib's verdict with the input and the output slice
placed against inaccessible pages, and the shared block-table parser against forged tables.  The -m gpu
tests (test_device_inflate.py) run the kernels on members and damaged members this file vouches for."""
from __future__ import annotations

import ctypes as C
import gzip
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from test_device_deflate_host import build_deflate_host, host_gzip

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build_inflate_host():
    """tests/host_emul/_build/libinflate_host.so, linked against the in-tree library (its table parser)."""
    from spz_b200 import _native
    from spz_b200 import build as B
    _native.lib()
    here = os.path.join(ROOT, "tests", "host_emul")
    out_dir = os.path.join(here, "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libinflate_host.so")
    deps = [os.path.join(here, "inflate_host.cc"), B.LIB] + [os.path.join(ROOT, "spz_b200", "csrc", h)
                                                            for h in ("inflate_format.cuh", "deflate_format.cuh", "spz_internal.hpp")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", deps[0], "-o", so, "-L", B.OUT_DIR, "-lspz_b200", "-lz",
                        "-Wl,-rpath," + B.OUT_DIR], check=True)
    lib = C.CDLL(so)
    for name in ("ifl_inflate", "ifl_inflate_guarded", "ifl_zlib"):
        getattr(lib, name).argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint32]
    lib.ifl_member.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
    lib.ifl_table.argtypes = [C.c_void_p, C.c_size_t] + [C.POINTER(C.c_uint64)] * 3 + [C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
    return lib


@pytest.fixture(scope="module")
def ifl():
    return build_inflate_host()


@pytest.fixture(scope="module")
def dfl():
    return build_deflate_host()


def _buf(data: bytes):
    a = np.frombuffer(data, np.uint8) if data else np.zeros(1, np.uint8)
    return a, a.ctypes.data


def inflate_guarded(ifl, raw: bytes, out_len: int):
    """(status, slice) of the decoder with guard pages; status -100 means a canary changed."""
    a, p = _buf(raw)
    out = np.zeros(max(out_len, 1), np.uint8)
    st = ifl.ifl_inflate_guarded(p, len(raw), out.ctypes.data, out_len)
    return st, out[:out_len].tobytes()


def zlib_verdict(ifl, raw: bytes, out_len: int):
    """(filled, slice) of one zlib inflate() into out_len bytes, as the block-parallel host inflater calls it."""
    a, p = _buf(raw)
    out = np.zeros(max(out_len, 1), np.uint8)
    ok = ifl.ifl_zlib(p, len(raw), out.ctypes.data, out_len)
    return ok == 1, out[:out_len].tobytes()


def member_on_device_route(ifl, member: bytes):
    """The device route for a whole member, on the host: (1 vouched / 0 host fallback / -1 no table, bytes)."""
    size, _ = table_of(ifl, member) or (0, None)
    out = np.zeros(max(size, 1), np.uint8)
    a, p = _buf(member)
    got = C.c_size_t(0)
    rc = ifl.ifl_member(p, len(member), out.ctypes.data, out.size, C.byref(got))
    return rc, out[:got.value].tobytes()


def table_of(ifl, member: bytes):
    a, p = _buf(member)
    bs, total, body, n = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0), C.c_size_t(0)
    comp = np.zeros(20000, np.uint32)
    if ifl.ifl_table(p, len(member), C.byref(bs), C.byref(total), C.byref(body), comp.ctypes.data, comp.size, C.byref(n)) != 0:
        return None
    return total.value, (bs.value, body.value, comp[:n.value].tolist())


def table_blocks(ifl, member: bytes):
    """[(raw deflate bytes, inflated length)] of every table block."""
    total, (bs, off, comp) = table_of(ifl, member)
    out = []
    for i, c in enumerate(comp):
        out.append((member[off:off + c], bs if i + 1 < len(comp) else total - bs * (len(comp) - 1)))
        off += c
    return out


def raw_deflate(data: bytes, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, flush_every=0, wbits=-15):
    z = zlib.compressobj(level, zlib.DEFLATED, wbits, 9, strategy)
    if not flush_every:
        return z.compress(data) + z.flush()
    out = b""
    for i in range(0, len(data), flush_every):
        out += z.compress(data[i:i + flush_every]) + z.flush(zlib.Z_SYNC_FLUSH)
    return out + z.flush()


def skewed(rng, n, p=0.1):
    return np.minimum(rng.geometric(p, n), 255).astype(np.uint8).tobytes()


def mixed(rng, n):
    """Random bytes, runs, repeated phrases and skewed bytes: every block type and match shape."""
    parts, size = [], 0
    while size < n:
        k = int(rng.integers(0, 5))
        m = int(rng.integers(1, 40000))
        if k == 0:
            part = rng.integers(0, 256, m, dtype=np.uint8).tobytes()
        elif k == 1:
            part = bytes([int(rng.integers(0, 256))]) * m
        elif k == 2:
            phrase = rng.integers(0, 256, int(rng.integers(1, 300)), dtype=np.uint8).tobytes()
            part = (phrase * (m // len(phrase) + 1))[:m]
        else:
            part = skewed(rng, m, 0.05 * k)
        parts.append(part)
        size += len(part)
    return b"".join(parts)[:n]


# ---- valid streams ------------------------------------------------------------------------------------


def assert_inflates_like_zlib(ifl, raw: bytes, data: bytes, what: str):
    st, got = inflate_guarded(ifl, raw, len(data))
    assert st == 0, f"{what}: status {st}"
    assert got == data, what


def assert_member_on_device_route(ifl, member: bytes, data: bytes, what: str):
    assert gzip.decompress(member) == data, what
    rc, got = member_on_device_route(ifl, member)
    if not data:  # a table cannot describe an empty member: the host inflater takes it
        assert rc == -1, what
        return
    assert rc == 1, f"{what}: rc {rc}"
    assert got == data, what
    for raw, n in table_blocks(ifl, member):
        ok, want = zlib_verdict(ifl, raw, n)
        assert ok, what
        assert_inflates_like_zlib(ifl, raw, want, what)


def test_device_deflater_members(ifl, dfl):
    from test_device_file import gzip_cases
    for name, data in gzip_cases():
        if len(data) > 4_000_000:
            data = data[:4_000_000]
        assert_member_on_device_route(ifl, host_gzip(dfl, data), data, name)


@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_host_parallel_members(ifl, monkeypatch, level):
    from spz_b200.codec import gzip_bytes
    monkeypatch.setenv("SPZ_B200_GZIP_LEVEL", str(level))
    rng = np.random.default_rng(100 + level)
    data = mixed(rng, (5 << 20) + 12345)
    member = gzip_bytes(data, threads=4)
    assert member[12:14] == b"SZ"
    assert_member_on_device_route(ifl, member, data, f"level {level}")


@pytest.mark.parametrize("strategy", ["fixed", "rle", "huffman_only", "default_flushed"])
def test_zlib_strategies(ifl, strategy):
    rng = np.random.default_rng(7)
    data = mixed(rng, 700_000)
    if strategy == "default_flushed":
        raw = raw_deflate(data, 6, flush_every=50_000)
    else:
        raw = raw_deflate(data, 6, {"fixed": zlib.Z_FIXED, "rle": zlib.Z_RLE, "huffman_only": zlib.Z_HUFFMAN_ONLY}[strategy])
    assert_inflates_like_zlib(ifl, raw, data, strategy)


def test_long_matches_and_overlapping_copies(ifl):
    rng = np.random.default_rng(8)
    window = rng.integers(0, 256, 32768, dtype=np.uint8).tobytes()
    cases = {
        "258 at distance 32768": window + window[:258] * 1 + window,  # matches reaching back the whole window
        "overlapping distance 1": b"x" + b"y" * 100_000,
        "overlapping distance 3": b"abc" * 40_000,
        "overlapping distance 31": (bytes(range(31)) * 5000),
        "overlapping distance 33": (bytes(range(33)) * 5000),
    }
    for name, data in cases.items():
        for level in (1, 9):
            assert_inflates_like_zlib(ifl, raw_deflate(data, level), data, f"{name} level {level}")
    # the stop rule: a slice shorter than the stream ends inside a literal run, a match or a stored block
    for name, data in cases.items():
        raw = raw_deflate(data, 9)
        for cut in (1, 259, len(data) // 2 + 1, len(data) - 1):
            ok, want = zlib_verdict(ifl, raw, cut)
            st, got = inflate_guarded(ifl, raw, cut)
            assert ok and st == 0 and got == want == data[:cut], (name, cut)
        st, _ = inflate_guarded(ifl, raw, len(data) + 1)  # the final block ends first
        assert st != 0 and not zlib_verdict(ifl, raw, len(data) + 1)[0], name
    stored = raw_deflate(rng.integers(0, 256, 200_000, dtype=np.uint8).tobytes(), 0)
    assert_inflates_like_zlib(ifl, stored, zlib.decompress(stored, -15), "stored")


def test_encoded_containers(ifl, dfl):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_device_file import version_container
    rng = np.random.default_rng(12)
    for deg in range(4):
        container = version_container(rng, 60_000, deg, 3)
        assert_member_on_device_route(ifl, host_gzip(dfl, container), container, f"device deflater SH{deg}")
        from spz_b200.codec import gzip_bytes
        big = version_container(rng, 200_000, deg, 3)
        assert_member_on_device_route(ifl, gzip_bytes(big, threads=4), big, f"zlib blocks SH{deg}")


# ---- hostile streams ----------------------------------------------------------------------------------


class Bits:
    def __init__(self):
        self.v, self.n = 0, 0

    def put(self, value, n):
        self.v |= (value & ((1 << n) - 1)) << self.n
        self.n += n
        return self

    def code(self, code, n):  # Huffman codes go MSB first
        return self.put(int(format(code, f"0{n}b")[::-1], 2), n)

    def align(self):
        self.n = (self.n + 7) // 8 * 8
        return self

    def bytes(self):
        return self.v.to_bytes((self.n + 7) // 8, "little")


def fixed_lit(b: Bits, sym: int):
    if sym < 144:
        return b.code(0x30 + sym, 8)
    if sym < 256:
        return b.code(0x190 + sym - 144, 9)
    if sym < 280:
        return b.code(sym - 256, 7)
    return b.code(0xC0 + sym - 280, 8)


def dynamic_header(b: Bits, final, hlit, hdist, cl_lens):
    b.put(final, 1).put(2, 2).put(hlit - 257, 5).put(hdist - 1, 5).put(len(cl_lens) - 4, 4)
    for x in cl_lens:
        b.put(x, 3)
    return b


def crafted_streams():
    """(name, raw, slice length) of streams zlib rejects or that stress a rule of the decoder."""
    b = fixed_lit(Bits().put(1, 1).put(1, 2), ord("a"))
    yield "lit/len symbol 286", fixed_lit(Bits().put(1, 1).put(1, 2), 286).put(0, 8).bytes(), 4
    yield "lit/len symbol 287 after a literal", fixed_lit(fixed_lit(Bits().put(1, 1).put(1, 2), 65), 287).put(0, 8).bytes(), 4
    yield "distance symbol 30", fixed_lit(b, 257).code(30, 5).put(0, 16).bytes(), 4
    yield "distance symbol 31", fixed_lit(fixed_lit(Bits().put(1, 1).put(1, 2), 65), 257).code(31, 5).put(0, 16).bytes(), 4
    yield "distance too far", fixed_lit(fixed_lit(Bits().put(1, 1).put(1, 2), 65), 257).code(1, 5).put(0, 16).bytes(), 4
    yield "distance too far after full", fixed_lit(fixed_lit(Bits().put(1, 1).put(1, 2), 65), 257).code(9, 5).put(0, 16).bytes(), 1
    yield "symbol 286 after full", fixed_lit(fixed_lit(Bits().put(1, 1).put(1, 2), 65), 286).put(0, 8).bytes(), 1
    yield "block type 3", Bits().put(0, 1).put(3, 2).put(0, 13).bytes(), 1
    yield "block type 3 after full", fixed_lit(fixed_lit(Bits().put(0, 1).put(1, 2), 65), 256).put(0, 1).put(3, 2).put(0, 8).bytes(), 1
    stored = Bits().put(1, 1).put(0, 2).align().put(5, 16).put(0xFFFF ^ 5 ^ 1, 16)
    yield "stored LEN != ~NLEN", stored.bytes() + b"hello", 5
    yield "stored truncated", Bits().put(1, 1).put(0, 2).align().put(5, 16).put(0xFFFF ^ 5, 16).bytes() + b"hel", 5
    yield "HLIT 287", dynamic_header(Bits(), 1, 287, 1, [0] * 4).put(0, 32).bytes(), 4
    yield "HLIT 288", dynamic_header(Bits(), 1, 288, 1, [0] * 4).put(0, 32).bytes(), 4
    yield "HDIST 31", dynamic_header(Bits(), 1, 257, 31, [0] * 4).put(0, 32).bytes(), 4
    yield "HDIST 32", dynamic_header(Bits(), 1, 257, 32, [0] * 4).put(0, 32).bytes(), 4
    yield "code-length code over-subscribed", dynamic_header(Bits(), 1, 257, 1, [1] * 19).put(0, 32).bytes(), 4
    yield "code-length code incomplete", dynamic_header(Bits(), 1, 257, 1, [1] + [0] * 18).put(0, 32).bytes(), 4
    yield "code-length code empty", dynamic_header(Bits(), 1, 257, 1, [0] * 19).put(0, 64).bytes(), 4
    # code-length code: symbols 16, 17, 18 and 0 (the first four of the header's order) with 2 bits each,
    # so canonical codes 0 -> 0, 16 -> 1, 17 -> 2, 18 -> 3
    cl = [2, 2, 2, 2]
    yield "repeat with no previous length", dynamic_header(Bits(), 1, 257, 1, cl).code(1, 2).put(0, 2).put(0, 32).bytes(), 4
    b = dynamic_header(Bits(), 1, 257, 1, cl)
    for _ in range(2):  # 18: 138 zeros, twice -> past HLIT + HDIST
        b.code(3, 2).put(127, 7)
    yield "repeat past the lengths", b.put(0, 32).bytes(), 4
    b = dynamic_header(Bits(), 1, 257, 1, cl)  # 258 zero lengths: no end-of-block code
    b.code(3, 2).put(127, 7).code(3, 2).put(109, 7)
    yield "no end-of-block code", b.put(0, 32).bytes(), 4


def damaged(rng, raw: bytes):
    """Seeded damage: bit flips, truncations, a byte overwritten, a range zeroed."""
    k = int(rng.integers(0, 4))
    r = bytearray(raw)
    if k == 0:
        for _ in range(int(rng.integers(1, 4))):
            i = int(rng.integers(0, len(r) * 8))
            r[i // 8] ^= 1 << (i % 8)
    elif k == 1:
        r = r[:int(rng.integers(0, len(r)))]
    elif k == 2:
        r[int(rng.integers(0, len(r)))] = int(rng.integers(0, 256))
    else:
        i, m = int(rng.integers(0, len(r))), int(rng.integers(1, 16))
        r[i:i + m] = bytes(len(r[i:i + m]))
    return bytes(r)


def hostile_corpus(dfl, seed=1, count=1500):
    rng = np.random.default_rng(seed)
    bases = []
    data = mixed(rng, 60_000)
    bases.append((raw_deflate(data, 6), len(data)))
    bases.append((raw_deflate(data, 1, zlib.Z_FIXED), len(data)))
    bases.append((raw_deflate(data[:3000], 0), 3000))
    bases.append((raw_deflate(data, 9, flush_every=7000), len(data)))
    small = skewed(rng, 5000)
    bases.append((raw_deflate(small, 6), len(small)))
    member = host_gzip(dfl, small + bytes(70_000))
    xlen, = struct.unpack_from("<H", member, 10)
    body = member[12 + xlen:-8]
    bases.append((body, len(small) + 70_000))  # one device-deflater table block (two segments)
    for name, raw, n in crafted_streams():
        yield name, raw, n
    for i in range(count):
        raw, n = bases[i % len(bases)]
        cut = n if i % 5 else int(rng.integers(1, n + 2))
        yield f"damaged {i}", damaged(rng, raw), cut


def test_hostile_streams_never_pass_what_zlib_rejects(ifl, dfl):
    agree = disagree = 0
    for name, raw, n in hostile_corpus(dfl):
        st, got = inflate_guarded(ifl, raw, n)
        assert st >= 0, f"{name}: memory outside the block's range was touched ({st})"
        ok, want = zlib_verdict(ifl, raw, n)
        if st == 0:
            assert ok, f"{name}: accepted a stream zlib rejects"
            assert got == want, f"{name}: accepted with bytes other than zlib's"
        if (st == 0) == ok:
            agree += 1
        else:
            disagree += 1  # stricter than zlib: allowed, costs a host fallback
    assert disagree <= 0.02 * (agree + disagree), (agree, disagree)


def damaged_copies(member: bytes):
    """A short fixed list of damaged copies of a block-table member: (name, bytes).  The -m gpu tests run
    the kernels on these copies of a gzip_device member; test_damaged_copies_are_safe checks them here first."""
    xlen, = struct.unpack_from("<H", member, 10)
    body = 12 + xlen
    out = []
    for i in (body + 3, body + 700, body + 40000, len(member) - 20):
        for bit in (0, 5):
            m = bytearray(member)
            m[i] ^= 1 << bit
            out.append((f"bit {bit} of byte {i}", bytes(m)))
    crc = bytearray(member)
    crc[-8] ^= 1
    out.append(("trailer CRC", bytes(crc)))
    zeroed = bytearray(member)
    zeroed[body + 100:body + 140] = bytes(40)
    out.append(("zeroed run", bytes(zeroed)))
    return out


def damaged_source():
    return mixed(np.random.default_rng(21), 6 * 65536 + 999)


def test_damaged_copies_are_safe(ifl, dfl):
    """host_gzip is byte for byte what gzip_device writes (test_device_file.py), so these are the GPU test's members."""
    from spz_b200 import _native as N
    from spz_b200.codec import gunzip_bytes
    for name, blob in damaged_copies(host_gzip(dfl, damaged_source())):
        for raw, n in table_blocks(ifl, blob):
            st, got = inflate_guarded(ifl, raw, n)
            assert st >= 0, name
            ok, want = zlib_verdict(ifl, raw, n)
            assert st != 0 or (ok and got == want), name
        rc, got = member_on_device_route(ifl, blob)
        try:
            want = gunzip_bytes(blob, threads=8)
        except N.CodecError:
            want = None
        assert rc == 0 or (rc == 1 and got == want), name


def test_crafted_streams_get_zlibs_verdict(ifl):
    accepted = {"distance too far after full"}  # zlib stops before checking the distance of a match it has no room for
    for name, raw, n in crafted_streams():
        st, got = inflate_guarded(ifl, raw, n)
        ok, want = zlib_verdict(ifl, raw, n)
        assert ok == (name in accepted), (name, ok)
        assert (st == 0) == ok, (name, st)
        if ok:
            assert got == want, name


# ---- the table parser --------------------------------------------------------------------------------


def test_table_info_rejects_forged_tables(ifl):
    from spz_b200 import _native as N
    from spz_b200.codec import gzip_bytes, gzip_table_info
    data = bytes(3 << 20)
    z = bytearray(gzip_bytes(data, 4))
    assert gzip_table_info(bytes(z)) == (len(data), 3)

    def forged(block_size, total):
        f = bytearray(z)
        struct.pack_into("<IIII", f, 16, block_size, 3, total & 0xffffffff, total >> 32)
        struct.pack_into("<I", f, len(f) - 4, total & 0xffffffff)  # ISIZE agrees with the table
        return bytes(f)

    # beyond deflate's 1032:1 expansion or 2 GiB blocks: refused before anything is sized from them
    for block_size, total in ((1 << 30, (2 << 30) + 5), (0xffff0000, 2 * 0xffff0000 + 1), (1 << 31, (2 << 31) + 1)):
        with pytest.raises(N.CodecError) as e:
            gzip_table_info(forged(block_size, total))
        assert e.value.code == N.ERR_INVALID
        assert member_on_device_route(ifl, forged(block_size, total))[0] == -1
    # a plausible lie passes the parser, but no block fills its slice: the host inflater gives the verdict
    lie = forged((1 << 20) + 4096, 2 * ((1 << 20) + 4096) + 1)
    assert gzip_table_info(lie) == (2 * ((1 << 20) + 4096) + 1, 3)
    assert member_on_device_route(ifl, lie)[0] == 0
    bad_isize = bytearray(z)
    bad_isize[-4] ^= 1
    truncated = bytes(z[:-9])
    no_table = gzip.compress(data)
    for blob in (bytes(bad_isize), truncated, no_table, b"", b"\x1f\x8b"):
        with pytest.raises(N.CodecError) as e:
            gzip_table_info(blob)
        assert e.value.code == N.ERR_INVALID


def test_damaged_member_falls_back(ifl, dfl):
    data = skewed(np.random.default_rng(3), 5 * 65536)
    member = bytearray(host_gzip(dfl, data))
    member[-8] ^= 1  # CRC
    assert member_on_device_route(ifl, bytes(member))[0] == 0
