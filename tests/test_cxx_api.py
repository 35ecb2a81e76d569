"""The drop-in C++ API (include/spz_b200/spz.hpp, spz_b200/csrc/spz_api.cc) against the reference's
own C++ through one consumer source compiled against both (tests/cxx/api_shim.cc).

not-gpu tests: everything that is host glue in both implementations -- container writer/reader and
plane order, gzip bytes, loadSpzPacked of v1/v2/v3 files, PackedGaussians::at, coordinateConverter,
convertCoordinates, medianVolume, data(), half conversions, small math, error behaviour, and that
the codec entry points fail loudly without a device.
gpu tests: packGaussians / unpackGaussians / saveSpz / loadSpz / unpack(i) vs the reference, bit for bit."""
from __future__ import annotations

import ctypes as C
import gzip
import os
import struct
import subprocess
import sys
import zlib

import time

import numpy as np
import pytest

from oracle import SH_DIM, Cloud, Packed, bits
from util import PLANES, assert_cloud_bits_equal, assert_packed_equal, random_cloud, random_stream

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CXX = os.path.join(ROOT, "tests", "cxx")

_f32p, _u8p = C.POINTER(C.c_float), C.POINTER(C.c_uint8)


class Shim:
    """ctypes front end of one build of tests/cxx/api_shim.cc."""

    def __init__(self, prefix: str):
        self.prefix = prefix
        so = os.path.join(CXX, "_build", f"libshim_{prefix}.so")
        target = {"b200": "all", "ref": "ref", "xlink": "xlink"}[prefix]
        can_build = prefix == "b200" or os.path.isdir("/root/reference/src/cc")
        if can_build:
            from spz_b200 import _native
            _native.lib()  # make sure libspz_b200.so exists before linking against it
            subprocess.run(["make", "-s", "-C", CXX, target], check=True)
        if not os.path.exists(so):
            pytest.skip(f"{so} not built and cannot be built here")
        self.lib = C.CDLL(so)
        for name, res in (("save_spz", C.c_void_p), ("load_spz", C.c_void_p), ("load_spz_file", C.c_void_p), ("load_ply", C.c_void_p),
                          ("load_packed", C.c_void_p), ("serialize", C.c_void_p), ("gzip", C.c_void_p),
                          ("cloud_ops", C.c_float)):
            self.fn(name).restype = res

    def fn(self, name):
        return getattr(self.lib, f"{self.prefix}_{name}")

    @staticmethod
    def _fplanes(arrs):
        arrs = [np.ascontiguousarray(a, np.float32).reshape(-1) for a in arrs]
        return arrs, (_f32p * 6)(*[a.ctypes.data_as(_f32p) for a in arrs])

    @staticmethod
    def _bplanes(arrs):
        arrs = [np.ascontiguousarray(a, np.uint8).reshape(-1) for a in arrs]
        return arrs, (_u8p * 6)(*[a.ctypes.data_as(_u8p) for a in arrs])

    def _take(self, ptr, size):
        try:
            return C.string_at(ptr, size.value)
        finally:
            self.fn("free")(C.c_void_p(ptr))

    # ---- codec ------------------------------------------------------------------------------
    def pack(self, c: Cloud, frm=0):
        d = SH_DIM.get(c.sh_degree, 0) * 3
        out = [np.zeros(c.n * w, np.uint8) for w in (9, 3, 4, 1, 3, d)]
        _, ip = self._fplanes(c.planes())
        _, op = self._bplanes(out)
        meta = (C.c_int32 * 5)()
        rc = self.fn("pack")(C.c_int32(c.n), C.c_int32(c.sh_degree), C.c_int32(frm), ip, op, meta)
        return rc, Packed(c.n, c.sh_degree, meta[2], 3, *out), list(meta)

    def unpack(self, p: Packed, to=0):
        d = SH_DIM.get(p.sh_degree, 0) * 3
        out = [np.zeros(p.n * w, np.float32) for w in (3, 3, 4, 1, 3, d)]
        _, ip = self._bplanes(p.planes())
        _, op = self._fplanes(out)
        # _fplanes copies; rebuild pointer table over the real outputs
        op = (_f32p * 6)(*[a.ctypes.data_as(_f32p) for a in out])
        meta = (C.c_int32 * 3)()
        rc = self.fn("unpack")(C.c_int32(p.n), C.c_int32(p.sh_degree), C.c_int32(p.fractional_bits), C.c_int32(p.version),
                               C.c_int32(to), ip, op, meta)
        return rc, Cloud(p.n, p.sh_degree, *out), list(meta)

    def save_spz(self, c: Cloud, frm=0):
        _, ip = self._fplanes(c.planes())
        size = C.c_uint64(0)
        ptr = self.fn("save_spz")(C.c_int32(c.n), C.c_int32(c.sh_degree), C.c_int32(int(c.antialiased)), C.c_int32(frm), ip, C.byref(size))
        return None if not ptr else self._take(ptr, size)

    def save_spz_v2(self, c: Cloud, frm=0):
        _, ip = self._fplanes(c.planes())
        size = C.c_uint64(0)
        f = self.fn("save_spz_v2")
        f.restype = C.c_void_p
        ptr = f(C.c_int32(c.n), C.c_int32(c.sh_degree), C.c_int32(int(c.antialiased)), C.c_int32(frm), ip, C.byref(size))
        return None if not ptr else self._take(ptr, size)

    def save_spz_file(self, c: Cloud, path: str, frm=0) -> bool:
        _, ip = self._fplanes(c.planes())
        return bool(self.fn("save_spz_file")(C.c_int32(c.n), C.c_int32(c.sh_degree), C.c_int32(int(c.antialiased)), C.c_int32(frm), ip, path.encode()))

    def _cloud_from_handle(self, h):
        try:
            m = (C.c_int64 * 9)()
            self.fn("cloud_info")(C.c_void_p(h), m)
            out = [np.zeros(m[3 + k], np.float32) for k in range(6)]
            op = (_f32p * 6)(*[a.ctypes.data_as(_f32p) for a in out])
            self.fn("cloud_copy")(C.c_void_p(h), op)
            return Cloud(int(m[0]), int(m[1]), *out, antialiased=bool(m[2]))
        finally:
            self.fn("cloud_free")(C.c_void_p(h))

    def load_spz(self, blob: bytes, to=0, via_vector=False) -> Cloud:
        buf = np.frombuffer(blob, np.uint8)
        h = self.fn("load_spz")(buf.ctypes.data_as(_u8p), C.c_int32(buf.size), C.c_int32(to), C.c_int32(int(via_vector)))
        return self._cloud_from_handle(h)

    def load_spz_file(self, path: str, to=0) -> Cloud:
        return self._cloud_from_handle(self.fn("load_spz_file")(path.encode(), C.c_int32(to)))

    def save_ply(self, c: Cloud, path: str, frm=0) -> bool:
        _, ip = self._fplanes(c.planes())
        return bool(self.fn("save_ply")(C.c_int32(c.n), C.c_int32(c.sh_degree), C.c_int32(frm), ip, path.encode()))

    def load_ply(self, path: str, to=0) -> Cloud:
        return self._cloud_from_handle(self.fn("load_ply")(path.encode(), C.c_int32(to)))

    # ---- host glue --------------------------------------------------------------------------
    def load_packed(self, blob: bytes, which=0):
        buf = np.frombuffer(blob, np.uint8) if blob else np.zeros(0, np.uint8)
        h = self.fn("load_packed")(buf.ctypes.data_as(_u8p), C.c_int32(buf.size), C.c_int32(which))
        try:
            m = (C.c_int64 * 12)()
            self.fn("packed_info")(C.c_void_p(h), m)
            out = [np.zeros(m[6 + k], np.uint8) for k in range(6)]
            op = (_u8p * 6)(*[a.ctypes.data_as(_u8p) for a in out])
            self.fn("packed_copy")(C.c_void_p(h), op)
            return dict(n=int(m[0]), deg=int(m[1]), fb=int(m[2]), aa=bool(m[3]), s3=bool(m[4]), half=bool(m[5])), out
        finally:
            self.fn("packed_free")(C.c_void_p(h))

    def serialize(self, p: Packed) -> bytes:
        _, ip = self._bplanes(p.planes())
        size = C.c_uint64(0)
        ptr = self.fn("serialize")(C.c_int32(p.n), C.c_int32(p.sh_degree), C.c_int32(p.fractional_bits), C.c_int32(p.version),
                                   C.c_int32(int(p.antialiased)), ip, C.byref(size))
        return self._take(ptr, size)

    def gzip(self, data: bytes):
        buf = np.frombuffer(data, np.uint8) if data else np.zeros(0, np.uint8)
        size = C.c_uint64(0)
        ptr = self.fn("gzip")(buf.ctypes.data_as(_u8p), C.c_uint64(buf.size), C.byref(size))
        return None if not ptr else self._take(ptr, size)

    def ply_to_spz(self, path: str, frm: int):
        self.fn("ply_to_spz").restype = C.c_void_p
        size = C.c_uint64(0)
        ptr = self.fn("ply_to_spz")(path.encode(), C.c_int32(frm), C.byref(size))
        return None if not ptr else self._take(ptr, size)

    def spz_to_ply(self, blob: bytes, to: int, path: str) -> bool:
        buf = np.frombuffer(blob, np.uint8)
        return bool(self.fn("spz_to_ply")(buf.ctypes.data_as(_u8p), C.c_uint64(buf.size), C.c_int32(to), path.encode()))

    def gzip_parallel(self, data: bytes, threads: int):
        self.fn("gzip_parallel").restype = C.c_void_p
        buf = np.frombuffer(data, np.uint8) if data else np.zeros(0, np.uint8)
        size = C.c_uint64(0)
        ptr = self.fn("gzip_parallel")(buf.ctypes.data_as(_u8p), C.c_uint64(buf.size), C.c_int32(threads), C.byref(size))
        return None if not ptr else self._take(ptr, size)

    def gunzip(self, data: bytes, threads: int):
        self.fn("gunzip").restype = C.c_void_p
        buf = np.frombuffer(data, np.uint8) if data else np.zeros(0, np.uint8)
        size = C.c_uint64(0)
        ptr = self.fn("gunzip")(buf.ctypes.data_as(_u8p), C.c_uint64(buf.size), C.c_int32(threads), C.byref(size))
        return None if not ptr else self._take(ptr, size)

    def at(self, p: Packed, i: int) -> np.ndarray:
        _, ip = self._bplanes(p.planes())
        out = np.zeros(65, np.uint8)
        self.fn("packed_at")(C.c_int32(p.n), C.c_int32(p.sh_degree), C.c_int32(p.fractional_bits), C.c_int32(p.version), ip, C.c_int32(i), out.ctypes.data_as(_u8p))
        return out

    def unpack_one(self, p: Packed, i: int, frm: int, to: int) -> np.ndarray:
        _, ip = self._bplanes(p.planes())
        out = np.zeros(59, np.float32)
        self.fn("packed_unpack_one")(C.c_int32(p.n), C.c_int32(p.sh_degree), C.c_int32(p.fractional_bits), C.c_int32(p.version), ip,
                                     C.c_int32(i), C.c_int32(frm), C.c_int32(to), out.ctypes.data_as(_f32p))
        return out

    def unpack_many(self, p: Packed, idx, conv21, batch: bool) -> np.ndarray:
        _, ip = self._bplanes(p.planes())
        idx = np.ascontiguousarray(idx, np.int32)
        conv = np.ascontiguousarray(conv21, np.float32)
        out = np.zeros((idx.size, 59), np.float32)
        got = self.fn("packed_unpack_many")(C.c_int32(p.n), C.c_int32(p.sh_degree), C.c_int32(p.fractional_bits), C.c_int32(p.version), ip,
                                            idx.ctypes.data_as(C.POINTER(C.c_int32)), C.c_int32(idx.size), conv.ctypes.data_as(_f32p),
                                            C.c_int32(int(batch)), out.ctypes.data_as(_f32p))
        return out[:got]

    def unpack_walk(self, p: Packed, idx, conv21, every: int) -> np.ndarray:
        _, ip = self._bplanes(p.planes())
        idx = np.ascontiguousarray(idx, np.int32)
        conv = np.ascontiguousarray(conv21, np.float32)
        out = np.zeros((idx.size, 59), np.float32)
        self.fn("packed_unpack_walk")(C.c_int32(p.n), C.c_int32(p.sh_degree), C.c_int32(p.fractional_bits), C.c_int32(p.version), ip,
                                      idx.ctypes.data_as(C.POINTER(C.c_int32)), C.c_int32(idx.size), conv.ctypes.data_as(_f32p),
                                      C.c_int32(every), out.ctypes.data_as(_f32p))
        return out

    def short_lived_threads(self, c: Cloud, frm: int, threads: int, concurrently) -> float:
        _, ip = self._fplanes(c.planes())
        f = self.fn("short_lived_threads")
        f.restype = C.c_double
        return f(C.c_int32(c.n), C.c_int32(c.sh_degree), C.c_int32(frm), ip, C.c_int32(threads), C.c_int32(int(concurrently)))

    def converter(self, frm, to) -> np.ndarray:
        out = np.zeros(21, np.float32)
        self.fn("converter")(C.c_int32(frm), C.c_int32(to), out.ctypes.data_as(_f32p))
        return out

    def cloud_ops(self, c: Cloud, frm, to):
        arrs = [np.ascontiguousarray(a, np.float32).copy() for a in c.planes()]
        ip = (_f32p * 6)(*[a.ctypes.data_as(_f32p) for a in arrs])
        vol = self.fn("cloud_ops")(C.c_int32(c.n), C.c_int32(c.sh_degree), C.c_int32(frm), C.c_int32(to), ip)
        return Cloud(c.n, c.sh_degree, *arrs), float(vol)

    def half_tables(self, samples: np.ndarray):
        to_float = np.zeros(65536, np.float32)
        samples = np.ascontiguousarray(samples, np.float32)
        to_half = np.zeros(samples.size, np.uint16)
        self.fn("half_tables")(to_float.ctypes.data_as(_f32p), samples.ctypes.data_as(_f32p), C.c_int32(samples.size),
                               to_half.ctypes.data_as(C.POINTER(C.c_uint16)))
        return to_float, to_half

    def math(self, axis, qa, qb, v) -> np.ndarray:
        a = [np.ascontiguousarray(x, np.float32) for x in (axis, qa, qb, v)]
        out = np.zeros(16, np.float32)
        self.fn("math")(*[x.ctypes.data_as(_f32p) for x in a], out.ctypes.data_as(_f32p))
        return out


@pytest.fixture(scope="module")
def mine():
    return Shim("b200")


@pytest.fixture(scope="module")
def theirs():
    return Shim("ref")


class OracleCodec:
    """The codec calls of Shim (pack, unpack, unpack_one) answered by the C restatement, oracle/spz_oracle.c, which
    tests/test_oracle.py pins bit for bit to vectors the unmodified reference made.  The meta fields are what the shim
    reports for the structs it builds: antialiased is always set (makeCloud / makePacked in api_shim.cc)."""

    prefix = "oracle"

    def __init__(self, oracle):
        self.oracle = oracle

    def pack(self, c: Cloud, frm=0):
        p = self.oracle.pack(c, frm)
        return 0, p, [p.n, p.sh_degree, p.fractional_bits, 1, int(p.version >= 3)]

    def unpack(self, p: Packed, to=0):
        g = self.oracle.unpack(p, to)
        return 0, g, [g.n, g.sh_degree, 1]

    def unpack_one(self, p: Packed, i: int, frm: int, to: int) -> np.ndarray:
        return self.oracle.unpack_at(p, [i], self.oracle.converter(frm, to))[0]


@pytest.fixture(scope="module")
def theirs_codec(oracle):
    """The reference's packGaussians / unpackGaussians / PackedGaussians::unpack(i, c) where its build is present or can
    be made, otherwise the C restatement of the same functions."""
    try:
        return Shim("ref")
    except pytest.skip.Exception:
        return OracleCodec(oracle)


@pytest.fixture(scope="module")
def relinked():
    """The consumer compiled against the REFERENCE's headers but linked against libspz_b200.so: what
    an existing application gets when only the library is swapped (layout-identical structs, same
    mangled symbols)."""
    return Shim("xlink")


def container(p: Packed, version=None, n_override=None, magic=0x5053474e) -> bytes:
    """Header + planes in stream order, written by hand (load-spz.cc:131-139, 533-546)."""
    ver = p.version if version is None else version
    hdr = struct.pack("<IIIBBBB", magic, ver, p.n if n_override is None else n_override, p.sh_degree, p.fractional_bits & 255,
                      1 if p.antialiased else 0, 0)
    return hdr + b"".join(np.ascontiguousarray(a).tobytes() for a in (p.positions, p.alphas, p.colors, p.scales, p.rotations, p.sh))


# =================================================================================================
# host glue (no GPU)
# =================================================================================================

@pytest.mark.parametrize("ver", [1, 2, 3])
def test_serialize_and_gzip_bytes_match_reference(mine, theirs, ver):
    rng = np.random.default_rng(ver)
    p = random_stream(rng, 1000, 2, ver, 12)
    p.antialiased = bool(ver % 2)
    a, b = mine.serialize(p), theirs.serialize(p)
    assert a == b
    assert a[:4] == b"NGSP" and a[4] == 3  # the writer always stamps version 3 (load-spz.cc:133)
    assert a[16:] == container(p)[16:]
    for data in (a, b"", b"x" * 100000, rng.integers(0, 256, 300000).astype(np.uint8).tobytes()):
        za, zb = mine.gzip(data), theirs.gzip(data)
        assert za == zb
        assert gzip.decompress(za) == data


@pytest.mark.parametrize("ver", [1, 2, 3])
@pytest.mark.parametrize("which", [0, 1])
def test_load_packed_all_versions(mine, theirs, ver, which):
    rng = np.random.default_rng(10 + ver)
    for deg in range(4):
        p = random_stream(rng, 333, deg, ver, 11)
        p.antialiased = True
        blob = gzip.compress(container(p), 6)
        ma, pa = mine.load_packed(blob, which)
        mb, pb = theirs.load_packed(blob, which)
        assert ma == mb == dict(n=333, deg=deg, fb=11, aa=True, s3=ver >= 3, half=ver == 1)
        for x, y, z in zip(pa, pb, p.planes()):
            assert np.array_equal(x, y) and np.array_equal(x, z)


def test_load_packed_rejects_what_the_reference_rejects(mine, theirs, tmp_path):
    rng = np.random.default_rng(20)
    p = random_stream(rng, 50, 1, 3)
    good = container(p)
    empty = dict(n=0, deg=0, fb=0, aa=False, s3=True, half=True)  # a default PackedGaussians
    cases = {
        "not gzip": good,
        "empty input": b"",
        "truncated gzip": gzip.compress(good)[:40],
        "bad magic": gzip.compress(container(p, magic=0x12345678)),
        "version 0": gzip.compress(container(p, version=0)),
        "version 4": gzip.compress(container(p, version=4)),
        "sh degree 4": gzip.compress(good[:12] + bytes([4]) + good[13:]),
        "short planes": gzip.compress(good[:-7]),
        "short header": gzip.compress(good[:9]),
        "count larger than data": gzip.compress(container(p, n_override=51)),
    }
    for name, blob in cases.items():
        ma, _ = mine.load_packed(blob)
        mb, _ = theirs.load_packed(blob)
        assert ma == mb == empty, name
    # trailing bytes after the planes are ignored by both
    ma, pa = mine.load_packed(gzip.compress(good + b"tail"))
    mb, pb = theirs.load_packed(gzip.compress(good + b"tail"))
    assert ma == mb and ma["n"] == 50 and all(np.array_equal(x, y) for x, y in zip(pa, pb))
    # file variant: missing file -> empty; real file -> same as bytes
    path = str(tmp_path / "a.spz")
    assert mine.load_packed(path.encode(), 2)[0] == empty
    open(path, "wb").write(gzip.compress(good))
    assert mine.load_packed(path.encode(), 2)[0] == theirs.load_packed(path.encode(), 2)[0] == ma


def test_load_packed_fuzz_against_the_reference(mine, theirs):
    """Seeded corruption fuzz of the container reader (load-spz.cc:548-596): header bytes overwritten, the stream
    truncated or extended at random, gzip payloads cut short.  Whatever the reference makes of a blob -- the
    empty struct or some set of planes -- the drop-in reader makes the same of it.  Point counts stay far
    below the reference's 10M cap, the one documented divergence of this reader."""
    rng = np.random.default_rng(21)
    agree_empty = agree_data = 0
    spent = [0.0, 0.0]
    for trial in range(400):
        ver = int(rng.integers(1, 4))
        deg = int(rng.integers(0, 4))
        n = int(rng.integers(1, 40))
        p = random_stream(rng, n, deg, ver, int(rng.integers(0, 25)))
        raw = bytearray(container(p))
        kind = trial % 5
        if kind == 0:    # one to three header bytes replaced
            for _ in range(int(rng.integers(1, 4))):  # (not the count's high bytes: the reference would zero-fill up to 650 MB per trial)
                raw[int(rng.choice([0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 12, 13, 14, 15]))] = int(rng.integers(0, 256))
        elif kind == 1:  # point count nudged (kept small: the cap is a documented divergence)
            raw[8:12] = int(rng.integers(0, 80)).to_bytes(4, "little")
        elif kind == 2:  # truncated or padded
            cut = int(rng.integers(0, len(raw) + 20))
            raw = raw[:cut] if cut <= len(raw) else raw + bytes(rng.integers(0, 256, cut - len(raw), dtype=np.uint8))
        elif kind == 3:  # sh degree / version / flags fields swept
            raw[4:8] = int(rng.integers(0, 6)).to_bytes(4, "little")
            raw[12] = int(rng.integers(0, 6))
            raw[14] = int(rng.integers(0, 256))
        blob = gzip.compress(bytes(raw), 1)
        if kind == 4:    # the gzip stream itself damaged
            blob = blob[:int(rng.integers(0, len(blob)))] if trial % 2 else blob[:10] + bytes(rng.integers(0, 256, 8, dtype=np.uint8)) + blob[18:]
        t0 = time.perf_counter()
        ma, pa = mine.load_packed(blob, trial % 2)
        t1 = time.perf_counter()
        mb, pb = theirs.load_packed(blob, trial % 2)
        spent[0] += t1 - t0
        spent[1] += time.perf_counter() - t1
        assert ma == mb, (trial, kind, ma, mb)
        for x, y in zip(pa, pb):
            assert np.array_equal(x, y), (trial, kind)
        if ma["n"] == 0:
            agree_empty += 1
        else:
            agree_data += 1
    assert agree_empty > 30 and agree_data > 30, (agree_empty, agree_data)  # the fuzz reaches both outcomes
    # a damaged blob must not cost more than a sound one (a truncated member's last four bytes once sized a 4 GiB buffer)
    assert spent[0] < 10 * spent[1] + 1.0, spent


def test_zero_fill_free_vectors_and_their_fallback(tmp_path):
    """spz_internal.hpp: resizeUninitialized (reserve + end pointer, no value-initialisation) and its
    SPZ_B200_ZEROFILL=1 fallback to resize() read the same file to the same planes (file API -> readFile,
    gunzip buffer, deserialize), each in a fresh process because the switch is read once."""
    import sys
    rng = np.random.default_rng(23)
    p = random_stream(rng, 5000, 3, 3, 12)
    path = str(tmp_path / "z.spz")
    open(path, "wb").write(gzip.compress(container(p), 1))
    code = ("import sys, hashlib; sys.path[:0] = [%r, %r]; import test_cxx_api as T; m, planes = T.Shim('b200').load_packed(%r.encode(), 2); "
            "print(m['n'], hashlib.sha256(b''.join(a.tobytes() for a in planes)).hexdigest())") % (os.path.dirname(__file__), ROOT, path)
    outs = []
    for env in ({}, {"SPZ_B200_ZEROFILL": "1"}):
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=dict(os.environ, **env), timeout=300)
        assert r.returncode == 0, r.stderr[-800:]
        outs.append(r.stdout.strip().splitlines()[-1])
    import hashlib
    want = "5000 " + hashlib.sha256(b"".join(a.tobytes() for a in p.planes())).hexdigest()
    assert outs[0] == outs[1] == want, outs


def test_point_cap_is_lifted_and_restorable(mine, theirs):
    """Documented divergence: the reference refuses > 10,000,000 points (load-spz.cc:549)."""
    n = 10_000_001
    z = lambda k: np.zeros(k, np.uint8)  # noqa: E731
    p = Packed(n, 0, 12, 3, z(9 * n), z(3 * n), z(4 * n), z(n), z(3 * n), z(0))
    blob = gzip.compress(container(p), 1)
    assert theirs.load_packed(blob)[0]["n"] == 0
    assert mine.load_packed(blob)[0]["n"] == n
    os.environ["SPZ_B200_MAX_POINTS"] = "10000000"
    try:
        assert mine.load_packed(blob)[0]["n"] == 0
    finally:
        del os.environ["SPZ_B200_MAX_POINTS"]


def test_at_gathers_the_same_65_bytes(mine, theirs):
    rng = np.random.default_rng(30)
    for ver in (1, 2, 3):
        for deg in range(4):
            p = random_stream(rng, 17, deg, ver)
            for i in (0, 5, 16):
                a, b = mine.at(p, i), theirs.at(p, i)
                if ver == 1:  # only 6 of the 9 position bytes are defined for float16 positions
                    a[6:9] = b[6:9] = 0
                if ver < 3:   # and 3 of the 4 rotation bytes
                    a[12] = b[12] = 0
                assert np.array_equal(a, b), (ver, deg, i)


def test_converter_cloud_ops_and_math(mine, theirs):
    for frm in range(9):
        for to in range(9):
            assert np.array_equal(bits(mine.converter(frm, to)), bits(theirs.converter(frm, to)))
    rng = np.random.default_rng(40)
    for deg in range(4):
        c = random_cloud(rng, 501, deg, True)
        for frm, to in ((4, 6), (6, 7), (0, 8), (1, 8), (5, 5)):
            (ca, va), (cb, vb) = mine.cloud_ops(c, frm, to), theirs.cloud_ops(c, frm, to)
            assert_cloud_bits_equal(ca, cb, f"convertCoordinates deg{deg} {frm}->{to}")
            assert va == vb or (np.isnan(va) and np.isnan(vb))
    empty = Cloud(0, 0, *[np.zeros(0, np.float32)] * 6)
    assert mine.cloud_ops(empty, 4, 6)[1] == theirs.cloud_ops(empty, 4, 6)[1] == np.float32(0.01)
    samples = np.concatenate([rng.normal(size=5000).astype(np.float32) * np.float32(10.0) ** rng.integers(-12, 8, 5000).astype(np.float32),
                              np.array([0, -0.0, np.inf, -np.inf, np.nan, 65504, 65520, 1e-8, 6e-8, 6.1e-5, -6.1e-5, 1e-45], np.float32)])
    (fa, ha), (fb, hb) = mine.half_tables(samples), theirs.half_tables(samples)
    assert np.array_equal(bits(fa), bits(fb)) and np.array_equal(ha, hb)
    for _ in range(20):
        axis, qa, qb, v = (rng.normal(size=k).astype(np.float32) for k in (3, 4, 4, 3))
        assert np.array_equal(bits(mine.math(axis, qa, qb, v)), bits(theirs.math(axis, qa, qb, v)))
    z3 = np.zeros(3, np.float32)
    assert np.array_equal(bits(mine.math(z3, qa, qb, v)), bits(theirs.math(z3, qa, qb, v)))


def test_ply_io_matches_reference(mine, theirs, tmp_path):
    rng = np.random.default_rng(70)
    for deg in range(4):
        c = random_cloud(rng, 257, deg, False)
        for frm in (0, 4, 6):
            pa, pb = str(tmp_path / f"a{deg}{frm}.ply"), str(tmp_path / f"b{deg}{frm}.ply")
            assert mine.save_ply(c, pa, frm) and theirs.save_ply(c, pb, frm)
            assert open(pa, "rb").read() == open(pb, "rb").read()
            for to in (0, 4, 8):
                ga, gb = mine.load_ply(pb, to), theirs.load_ply(pb, to)
                assert ga.n == gb.n == 257 and ga.sh_degree == gb.sh_degree == deg
                assert_cloud_bits_equal(ga, gb, f"ply deg{deg} from{frm} to{to}")
    assert not mine.save_ply(c, "/nonexistent_dir/x.ply", 0)
    # a cloud large enough for the multi-threaded shuffles (>= 64K points; 300K points = two write batches)
    for n_big, deg_big in ((70_001, 1), (300_000, 0)):
        big = random_cloud(rng, n_big, deg_big, False)
        pa, pb2 = str(tmp_path / "big_a.ply"), str(tmp_path / "big_b.ply")
        assert mine.save_ply(big, pa, 8) and theirs.save_ply(big, pb2, 8)
        assert open(pa, "rb").read() == open(pb2, "rb").read()
        assert_cloud_bits_equal(mine.load_ply(pb2, 7), theirs.load_ply(pb2, 7), f"large ply {n_big}")
    # malformed files: both hand back an empty cloud
    good = open(pb, "rb").read()
    body = good.index(b"end_header\n") + len(b"end_header\n")
    variants = {
        "missing": None,
        "not ply": b"plx\n" + good[4:],
        "ascii": good.replace(b"binary_little_endian", b"ascii"),
        "double property": good.replace(b"property float opacity", b"property double opacity"),
        "missing field": good.replace(b"property float rot_3\n", b""),
        "truncated body": good[:body + 100],
        "zero vertices": good.replace(b"element vertex 257", b"element vertex 0"),
        "comment and blank lines ok": good.replace(b"format binary", b"comment hello\n\n  format binary", 1),
    }
    for name, data in variants.items():
        path = str(tmp_path / "v.ply")
        if data is None:
            path = str(tmp_path / "nope.ply")
        else:
            open(path, "wb").write(data)
        ga, gb = mine.load_ply(path, 0), theirs.load_ply(path, 0)
        assert ga.n == gb.n, name
        if gb.n:
            assert_cloud_bits_equal(ga, gb, name)
    # A header that names a property twice: the reference sizes a vertex record by its name -> column map and then
    # indexes it with the (larger) line numbers, i.e. past the end of its buffer (load-spz.cc:740,801), so there is
    # nothing to compare with.  Here a record is as wide as the header has property lines and the later line wins.
    last = good[body:]
    rows = np.frombuffer(last, np.float32).reshape(257, -1)
    wide = np.concatenate([rows, rows[:, :1] + 100.0], axis=1)  # one more column at the end: the second "x"
    dup = good[:body].replace(b"end_header\n", b"property float x\nend_header\n") + wide.astype(np.float32).tobytes()
    open(str(tmp_path / "dup.ply"), "wb").write(dup)
    gd = mine.load_ply(str(tmp_path / "dup.ply"), 0)
    ref_last = theirs.load_ply(pb, 0)
    assert gd.n == 257
    assert np.array_equal(gd.positions[0::3], ref_last.positions[0::3] + np.float32(100.0))
    assert np.array_equal(bits(gd.positions[1::3]), bits(ref_last.positions[1::3])) and np.array_equal(bits(gd.sh), bits(ref_last.sh))


def test_parallel_gzip_is_a_standard_member_with_identical_content(mine, theirs):
    """Block-parallel zlib (spz_gzip.cc): every inflater recovers the exact input -- Python's gzip,
    the reference's loadSpzPacked, this repo's serial and parallel inflaters -- and the parallel
    inflater also reads members it did not write."""
    rng = np.random.default_rng(80)
    # a real container so the reference's loader can be the judge: 120k SH3 points = 7.8 MB, 8 blocks
    p = random_stream(rng, 120_000, 3, 3)
    # compressible planes (real splats are): quantise the noise
    p.sh = (p.sh & 0xF0).astype(np.uint8)
    p.scales = (p.scales & 0xFC).astype(np.uint8)
    stream = container(p)
    for threads in (2, 5, 16):
        z = mine.gzip_parallel(stream, threads)
        assert z[:4] == b"\x1f\x8b\x08\x04"            # one member, FEXTRA set
        assert gzip.decompress(z) == stream
        assert zlib.decompress(z, 16 + zlib.MAX_WBITS) == stream
        assert mine.gunzip(z, 0) == stream                 # serial inflater
        assert mine.gunzip(z, threads) == stream           # block-parallel inflater
        meta, planes = theirs.load_packed(z)               # the unmodified reference reads it
        assert meta["n"] == 120_000 and all(np.array_equal(a, b) for a, b in zip(planes, p.planes()))
        serial = mine.gzip(stream)
        assert len(z) < len(serial) * 1.02                 # independent 1 MiB blocks cost < 2 % in ratio
    # a faster zlib level for the parallel path only; content unchanged
    os.environ["SPZ_B200_GZIP_LEVEL"] = "1"
    try:
        fast = mine.gzip_parallel(stream, 4)
        assert gzip.decompress(fast) == stream and mine.gunzip(fast, 4) == stream and fast != z
        assert mine.gzip(stream) == theirs.gzip(stream)    # the serial stream ignores the knob
    finally:
        del os.environ["SPZ_B200_GZIP_LEVEL"]
    # one thread, or an input below two blocks: the reference's byte-identical serial stream
    assert mine.gzip_parallel(stream, 1) == theirs.gzip(stream)
    small = stream[:1_500_000]
    assert mine.gzip_parallel(small, 8) == theirs.gzip(small)
    # sizes around the block boundaries
    for size in (2 << 20, (2 << 20) + 1, (3 << 20) - 1, 5 * (1 << 20)):
        data = rng.integers(0, 64, size).astype(np.uint8).tobytes()
        z = mine.gzip_parallel(data, 4)
        assert gzip.decompress(z) == data and mine.gunzip(z, 4) == data
    # members written by others (no block table) go down the serial path
    assert mine.gunzip(theirs.gzip(stream), 8) == stream
    assert mine.gunzip(gzip.compress(stream, 1), 8) == stream
    # damage: flipped payload byte, truncated tail, lying table -> the same refusal as a serial inflater
    z = bytearray(mine.gzip_parallel(stream, 4))
    bad = bytes(z[:len(z) // 2]) + bytes([z[len(z) // 2] ^ 0x55]) + bytes(z[len(z) // 2 + 1:])
    assert mine.gunzip(bad, 4) is None and mine.gunzip(bad, 0) is None
    assert mine.gunzip(bytes(z[:-9]), 4) is None
    lying = bytearray(z)
    lying[20] ^= 0x10  # block size field
    assert mine.gunzip(bytes(lying), 4) in (None, stream)  # falls back to the serial inflater, which ignores FEXTRA
    assert mine.gunzip(b"", 4) is None and mine.gunzip(b"\x1f\x8b", 4) is None


def test_parallel_gunzip_rejects_a_hostile_block_table(mine):
    """ADVICE r1: the 'SZ' FEXTRA table is untrusted and used to size the output before a byte is inflated.  A
    table that claims terabytes (or just more than deflate's 1032:1 ceiling for a block's compressed length) must
    neither allocate that nor throw across the API: the serial inflater -- whose buffer grows only with what zlib
    really produces -- gives the verdict, through the C++ API, the loader and the extern "C" entry point."""
    import resource
    from spz_b200 import codec
    data = bytes(3 << 20)  # zeros: three 1 MiB blocks of ~1 KB each
    z = bytearray(mine.gzip_parallel(data, 4))
    assert z[3] == 4 and z[12:14] == b"SZ"
    blocks = struct.unpack_from("<I", z, 20)[0]
    assert blocks == 3 and struct.unpack_from("<I", z, 16)[0] == 1 << 20

    def forged(block_size, total):
        f = bytearray(z)
        struct.pack_into("<IIII", f, 16, block_size, blocks, total & 0xffffffff, total >> 32)
        struct.pack_into("<I", f, len(f) - 4, total & 0xffffffff)  # ISIZE agrees with the table
        return bytes(f)

    before = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss
    for block_size, total in ((1 << 30, (2 << 30) + 5), (0xffff0000, 2 * 0xffff0000 + 1), (1 << 31, (2 << 31) + 1),
                              ((1 << 20) + 4096, 2 * ((1 << 20) + 4096) + 1)):
        blob = forged(block_size, total)
        for call in (lambda b: mine.gunzip(b, 4), lambda b: codec.gunzip_bytes(b, 4)):
            try:
                got = call(blob)
            except Exception as e:  # noqa: BLE001 -- a clean refusal (CodecError) is fine too
                assert "zlib" in str(e) or "memory" in str(e)
                got = None
            assert got is None  # the serial inflater sees ISIZE disagree with what the stream really holds
        meta, _ = mine.load_packed(blob)
        assert meta["n"] == 0
    after = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss
    assert after - before < 512 * 1024  # KiB: nothing near the forged gigabytes was ever touched
    assert mine.gunzip(bytes(z), 4) == data


def test_parallel_gunzip_fuzz(mine):
    """Seeded damage to block-parallel gzip members (the block table in FEXTRA, block bodies, the trailer,
    truncation): the inflater never crashes, and gives Python's gzip module's verdict -- the same bytes
    when that accepts the member, failure when it rejects it."""
    rng = np.random.default_rng(22)
    accepted = rejected = 0
    for trial in range(120):
        n = int(rng.integers(1, 6)) << 20
        data = (rng.integers(0, 40, n, dtype=np.uint8) * 3).tobytes() if trial % 3 else rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        blob = bytearray(mine.gzip_parallel(data, 4))
        kind = trial % 4
        if kind == 0:    # a byte of the header / block table
            blob[int(rng.integers(0, 64))] ^= 1 << int(rng.integers(0, 8))
        elif kind == 1:  # a byte somewhere in the bodies
            blob[int(rng.integers(64, len(blob) - 8))] ^= 1 << int(rng.integers(0, 8))
        elif kind == 2:  # the CRC / ISIZE trailer
            blob[len(blob) - 1 - int(rng.integers(0, 8))] ^= 1 << int(rng.integers(0, 8))
        else:            # truncated (or, one time in four, left intact)
            blob = blob if trial % 16 == 3 else blob[:int(rng.integers(1, len(blob)))]
        try:
            want = gzip.decompress(bytes(blob))
        except Exception:  # noqa: BLE001  (BadGzipFile, EOFError, zlib.error)
            want = None
        for threads in (1, 4):
            got = mine.gunzip(bytes(blob), threads)
            assert got == want, (trial, kind, threads, None if got is None else len(got), None if want is None else len(want))
        accepted += want is not None
        rejected += want is None
    assert accepted >= 5 and rejected >= 60, (accepted, rejected)


def test_save_load_use_parallel_gzip_when_asked(mine, theirs, tmp_path):
    """SPZ_B200_GZIP_THREADS switches loadSpzPacked to the parallel inflater (the save side needs the
    GPU for its planes and is covered by the gpu test below)."""
    rng = np.random.default_rng(81)
    p = random_stream(rng, 100_000, 3, 3)
    z = mine.gzip_parallel(container(p), 4)
    os.environ["SPZ_B200_GZIP_THREADS"] = "4"
    try:
        meta, planes = mine.load_packed(z)
    finally:
        del os.environ["SPZ_B200_GZIP_THREADS"]
    assert meta["n"] == 100_000 and all(np.array_equal(a, b) for a, b in zip(planes, p.planes()))
    # the default policy (variable unset): a member that carries the block table is inflated block-parallel, one the
    # reference wrote serially; SPZ_B200_GZIP_THREADS=1 pins the serial inflater for both.  Same container every way.
    for blob in (z, theirs.gzip(container(p))):
        for env in (None, "1"):
            if env:
                os.environ["SPZ_B200_GZIP_THREADS"] = env
            try:
                meta, planes = mine.load_packed(blob)
            finally:
                os.environ.pop("SPZ_B200_GZIP_THREADS", None)
            assert meta["n"] == 100_000 and all(np.array_equal(a, b) for a, b in zip(planes, p.planes()))


def test_relinked_consumer_host_glue(relinked, theirs, tmp_path):
    rng = np.random.default_rng(90)
    p = random_stream(rng, 777, 3, 3)
    p.antialiased = True
    assert relinked.serialize(p) == theirs.serialize(p)
    assert relinked.gzip(container(p)) == theirs.gzip(container(p))
    for ver in (1, 2, 3):
        q = random_stream(rng, 99, 2, ver, 9)
        blob = gzip.compress(container(q))
        (ma, pa), (mb, pb) = relinked.load_packed(blob), theirs.load_packed(blob)
        assert ma == mb and all(np.array_equal(x, y) for x, y in zip(pa, pb))
        assert np.array_equal(relinked.at(q, 7)[13:], theirs.at(q, 7)[13:])
    c = random_cloud(rng, 300, 3, False)
    (ca, va), (cb, vb) = relinked.cloud_ops(c, 6, 7), theirs.cloud_ops(c, 6, 7)
    assert_cloud_bits_equal(ca, cb, "convertCoordinates")
    assert va == vb
    pa, pb = str(tmp_path / "a.ply"), str(tmp_path / "b.ply")
    assert relinked.save_ply(c, pa, 4) and theirs.save_ply(c, pb, 4)
    assert open(pa, "rb").read() == open(pb, "rb").read()
    assert_cloud_bits_equal(relinked.load_ply(pb, 8), theirs.load_ply(pb, 8), "ply")
    empty = Cloud(0, 0, *[np.zeros(0, np.float32)] * 6, antialiased=True)
    assert relinked.save_spz(empty, 6) == theirs.save_spz(empty, 6)


def test_size_checks_and_empty_cloud_need_no_device(mine, theirs):
    """Rejections happen before any device work, so they behave the same with and without a GPU."""
    rng = np.random.default_rng(50)
    c = random_cloud(rng, 10, 1, False)
    bad = Cloud(10, 1, c.positions, c.scales, c.rotations, c.alphas, c.colors, c.sh[:-3])
    # the shim's makeCloud assigns by the declared sizes, so build the mismatch through sh_degree
    wrong_degree = Cloud(10, 4, *c.planes())
    for cloud in (wrong_degree,):
        ra, _, ma = mine.pack(cloud, 0)
        rb, _, mb = theirs.pack(cloud, 0)
        assert ra == rb == 1 and ma == mb
    del bad
    # empty cloud: packs to an empty v3 struct and saves to the reference's bytes, no GPU touched
    empty = Cloud(0, 0, *[np.zeros(0, np.float32)] * 6, antialiased=True)
    ra, pa, ma = mine.pack(empty, 6)
    rb, pb, mb = theirs.pack(empty, 6)
    assert ra == rb == 0 and ma == mb == [0, 0, 12, 1, 1]
    assert mine.save_spz(empty, 6) == theirs.save_spz(empty, 6)
    g = mine.load_spz(theirs.save_spz(empty, 6), 8)
    assert g.n == 0 and g.antialiased
    # garbage in -> empty cloud out, no exception (load_spz_test.py:842-863)
    assert mine.load_spz(b"garbage", 0).n == 0
    assert mine.load_spz_file("/nonexistent/file.spz", 0).n == 0


def test_codec_fails_loudly_without_a_device(mine):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    rng = np.random.default_rng(60)
    c = random_cloud(rng, 10, 1, False)
    rc, _, meta = mine.pack(c, 0)
    assert rc == 1 and meta[0] == 0          # empty struct, like any rejected call
    assert mine.save_spz(c, 0) is None       # and saveSpz returns false rather than writing an empty file
    p = random_stream(rng, 10, 1, 3)
    rc, _, meta = mine.unpack(p, 0)
    assert rc == 1 and meta[0] == 0


# =================================================================================================
# the codec through the C++ API (GPU)
# =================================================================================================

@pytest.mark.gpu
@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_pack_unpack_match_reference(mine, theirs_codec, deg):
    theirs = theirs_codec
    rng = np.random.default_rng(100 + deg)
    for special in (False, True):
        c = random_cloud(rng, 20011, deg, special)
        for frm in (0, 4, 6, 7, 8):
            (ra, pa, ma), (rb, pb, mb) = mine.pack(c, frm), theirs.pack(c, frm)
            assert ra == rb == 0 and ma == mb
            assert_packed_equal(pa, pb, f"deg{deg} from{frm}")
        for to in (0, 4, 6, 7, 8):
            (ra, ga, ma), (rb, gb, mb) = mine.unpack(pb, to), theirs.unpack(pb, to)
            assert ra == rb == 0 and ma == mb
            assert_cloud_bits_equal(ga, gb, f"deg{deg} to{to}")


@pytest.mark.gpu
@pytest.mark.parametrize("ver", [1, 2, 3, 4])
def test_unpack_legacy_flavours(mine, theirs_codec, ver):
    theirs = theirs_codec
    rng = np.random.default_rng(200 + ver)
    for fb in (12, 7):
        s = random_stream(rng, 7001, 2, ver, fb)
        for to in (0, 7):
            (ra, ga, _), (rb, gb, _) = mine.unpack(s, to), theirs.unpack(s, to)
            assert ra == rb == 0
            assert_cloud_bits_equal(ga, gb, f"v{ver} fb{fb} to{to}")


@pytest.mark.gpu
def test_save_load_spz_bytes_and_files(mine, theirs, tmp_path):
    rng = np.random.default_rng(300)
    for deg in (0, 3):
        c = random_cloud(rng, 5003, deg, False)
        c.antialiased = True
        blob_a, blob_b = mine.save_spz(c, 6), theirs.save_spz(c, 6)
        assert blob_a == blob_b  # same planes, same container, same zlib parameters
        for via_vector in (False, True):
            ga, gb = mine.load_spz(blob_b, 8, via_vector), theirs.load_spz(blob_b, 8, via_vector)
            assert ga.n == gb.n == 5003 and ga.antialiased and ga.sh_degree == deg
            assert_cloud_bits_equal(ga, gb, "loadSpz")
        pa, pb = str(tmp_path / "a.spz"), str(tmp_path / "b.spz")
        assert mine.save_spz_file(c, pa, 6) and theirs.save_spz_file(c, pb, 6)
        assert open(pa, "rb").read() == open(pb, "rb").read()
        assert_cloud_bits_equal(mine.load_spz_file(pb, 7), theirs.load_spz_file(pb, 7), "loadSpz(file)")
        assert not mine.save_spz_file(c, "/nonexistent_dir/x.spz", 0)


@pytest.mark.gpu
def test_save_spz_with_parallel_gzip_is_readable_by_the_reference(mine, theirs):
    rng = np.random.default_rng(310)
    c = random_cloud(rng, 150_000, 3, False)
    os.environ["SPZ_B200_GZIP_THREADS"] = "1"
    try:
        serial = mine.save_spz(c, 6)
        os.environ["SPZ_B200_GZIP_THREADS"] = "8"
        par = mine.save_spz(c, 6)
        back = mine.load_spz(par, 8)
    finally:
        del os.environ["SPZ_B200_GZIP_THREADS"]
    assert serial == theirs.save_spz(c, 6), "SPZ_B200_GZIP_THREADS=1 pins the reference's file bytes"
    assert par != serial and gzip.decompress(par) == gzip.decompress(serial)
    assert_cloud_bits_equal(theirs.load_spz(par, 8), theirs.load_spz(serial, 8), "reference reads the parallel member")
    assert_cloud_bits_equal(back, theirs.load_spz(serial, 8), "parallel inflate + decode")


@pytest.mark.gpu
def test_save_spz_default_gzip_policy(mine, theirs):
    """With SPZ_B200_GZIP_THREADS unset, a container below 8 MiB is deflated as the reference does it (same file bytes);
    from 8 MiB up saveSpz takes the block-parallel framing on its own -- a different, standard gzip member holding the
    identical container, which the unmodified reference loads to the same cloud.  SPZ_B200_GZIP_THREADS=1 pins the
    reference's bytes at every size."""
    rng = np.random.default_rng(311)
    small = random_cloud(rng, 20_000, 3, False)
    assert mine.save_spz(small, 6) == theirs.save_spz(small, 6)
    c = random_cloud(rng, 400_000, 3, False)  # 16 + 65 * 400K = 26 MB of container
    auto = mine.save_spz(c, 6)
    assert auto[3] & 4, "FEXTRA block table expected above the threshold"
    stream = gzip.decompress(auto)
    assert len(stream) == 16 + 65 * c.n
    r, p, m = theirs.pack(c, 6)
    assert stream == container(p)
    assert_cloud_bits_equal(mine.load_spz(auto, 8), theirs.unpack(p, 8)[1], "default policy: parallel member, parallel inflate")
    assert theirs.load_spz(auto, 8).n == c.n


@pytest.mark.gpu
@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_fused_ply_to_spz_matches_load_then_save(mine, theirs, tmp_path, deg):
    """plyToSpz (records -> GPU -> packed planes, ply_kernels.cu) against the reference's two-step
    loadSplatFromPly + saveSpz: identical container bytes for every frame choice."""
    rng = np.random.default_rng(340 + deg)
    n = 3 * 512 + 57  # full tiles on the staged kernel (128..512 gaussians by degree) + a scalar remainder
    c = random_cloud(rng, n, deg, deg == 3)
    path = str(tmp_path / "in.ply")
    assert theirs.save_ply(c, path, 0)
    for to in (4, 7, 8):  # records are RDF; the loader converts to X, the encoder from X back to RUB
        want = theirs.save_spz(theirs.load_ply(path, to), to)
        got = mine.ply_to_spz(path, 6)
        assert gzip.decompress(got) == gzip.decompress(want), (deg, to)
    assert gzip.decompress(mine.ply_to_spz(path, 0)) == gzip.decompress(theirs.save_spz(theirs.load_ply(path, 0), 0))
    assert mine.ply_to_spz(str(tmp_path / "missing.ply"), 0) is None


@pytest.mark.gpu
@pytest.mark.parametrize("ver", [2, 3])
def test_fused_spz_to_ply_matches_load_then_save(mine, theirs, tmp_path, ver):
    """spzToPly (packed planes -> GPU -> finished vertex records) against the reference's two-step
    loadSpz + saveSplatToPly: the same .ply file byte for byte, for v3 and legacy v2 streams."""
    rng = np.random.default_rng(350 + ver)
    for deg in range(4):
        n = 2 * 512 + 131
        s = random_stream(rng, n, deg, ver, 12)
        if ver == 3:
            # magnitudes <= 255 of 511: three squares sum below 1, so sqrt(1 - sum) is a number and the
            # files can be compared raw (an invalid payload yields NaN, whose bits differ x86 vs sm_100a)
            s.rotations.view("<u4")[:] &= np.uint32(0xEFFBFEFF)
        blob = gzip.compress(container(s), 1)
        for x in (4, 7):
            want_path, got_path = str(tmp_path / "want.ply"), str(tmp_path / "got.ply")
            assert theirs.save_ply(theirs.load_spz(blob, x), want_path, x)
            assert mine.spz_to_ply(blob, 6, got_path)
            assert open(got_path, "rb").read() == open(want_path, "rb").read(), (ver, deg, x)
        assert theirs.save_ply(theirs.load_spz(blob, 0), want_path, 0) and mine.spz_to_ply(blob, 0, got_path)
        assert open(got_path, "rb").read() == open(want_path, "rb").read(), (ver, deg, "unspecified")
    assert not mine.spz_to_ply(blob, 0, "/nonexistent_dir/x.ply")


@pytest.mark.gpu
def test_relinked_consumer_codec(relinked, theirs, tmp_path):
    rng = np.random.default_rng(330)
    for deg in (0, 3):
        c = random_cloud(rng, 30_011, deg, True)
        c.antialiased = True
        (ra, pa, ma), (rb, pb, mb) = relinked.pack(c, 6), theirs.pack(c, 6)
        assert ra == rb == 0 and ma == mb
        assert_packed_equal(pa, pb, f"relinked pack deg{deg}")
        (ra, ga, ma), (rb, gb, mb) = relinked.unpack(pb, 8), theirs.unpack(pb, 8)
        assert ra == rb == 0 and ma == mb
        assert_cloud_bits_equal(ga, gb, f"relinked unpack deg{deg}")
        assert relinked.save_spz(c, 6) == theirs.save_spz(c, 6)
        assert_cloud_bits_equal(relinked.load_spz(theirs.save_spz(c, 6), 7), theirs.load_spz(theirs.save_spz(c, 6), 7), "relinked loadSpz")
    s = random_stream(rng, 5, 3, 3)
    s.rotations.view("<u4")[:] &= np.uint32(0xEFFBFEFF)
    assert np.array_equal(bits(relinked.unpack_one(s, 3, 4, 6)), bits(theirs.unpack_one(s, 3, 4, 6)))


@pytest.mark.gpu
def test_concurrent_callers_each_get_their_own_context(mine, theirs):
    rng = np.random.default_rng(320)
    c = random_cloud(rng, 40_000, 3, False)
    _, ip = mine._fplanes(c.planes())
    for shim in (mine, theirs):
        diff = shim.fn("concurrent_roundtrip")(C.c_int32(c.n), C.c_int32(3), C.c_int32(6), C.c_int32(8), ip, C.c_int32(4))
        assert diff == 0, shim.prefix


@pytest.mark.gpu
def test_unpack_one_matches_reference(mine, theirs_codec):
    theirs = theirs_codec
    rng = np.random.default_rng(400)
    for ver in (1, 2, 3):
        for deg in (0, 2, 3):
            s = random_stream(rng, 9, deg, ver, 12)
            if ver == 3:
                # keep smallest-three payloads valid so sqrt(1 - sum) is a number in both
                comp = s.rotations.view("<u4")
                comp &= np.uint32(0xEFFBFEFF)  # magnitudes <= 255: a valid unit quaternion
            for i in (0, 8):
                for frm, to in ((0, 0), (4, 6), (4, 7)):
                    a, b = mine.unpack_one(s, i, frm, to), theirs.unpack_one(s, i, frm, to)
                    assert np.array_equal(bits(a), bits(b)), (ver, deg, i, frm, to)


@pytest.mark.gpu
def test_unpack_many_matches_a_loop_over_the_reference(mine, theirs, relinked):
    """SURVEY.md 8f-4: batched at()/unpack(i) -- one launch for a list of indices -- against the reference's
    PackedGaussians::unpack (load-spz.cc:383-463) called in a loop, every stream flavour and SH degree, the
    nine coordinate converters and a hand-built converter with arbitrary factors (applied by multiplication,
    in the reference's order)."""
    rng = np.random.default_rng(410)
    odd = (rng.normal(size=21) * 3).astype(np.float32)
    odd[[2, 9]] = [0.0, -0.0]
    convs = [mine.converter(frm, to) for frm, to in ((0, 0), (4, 6), (4, 7), (1, 8), (6, 3))] + [odd]
    for ver in (1, 2, 3, 4):
        for deg in range(4):
            n = 700
            s = random_stream(rng, n, deg, ver, int(rng.choice([0, 5, 12, 20])))
            if ver >= 3:
                s.rotations.view("<u4")[::2] &= np.uint32(0xEFFBFEFF)  # half of them valid unit quaternions, half NaN roots
            idx = np.concatenate([[0, n - 1, n - 1, 3], rng.integers(0, n, 300)]).astype(np.int32)
            for conv in convs:
                want = theirs.unpack_many(s, idx, conv, False)
                got = mine.unpack_many(s, idx, conv, True)
                assert got.shape == want.shape
                assert np.array_equal(bits(got), bits(want)), (ver, deg, conv[:3])
            # the one-at-a-time accessor, through this library and through a consumer built against the reference's headers
            few = idx[:6]
            want = theirs.unpack_many(s, few, odd, False)
            assert np.array_equal(bits(mine.unpack_many(s, few, odd, False)), bits(want))
            assert np.array_equal(bits(relinked.unpack_many(s, few, odd, False)), bits(want))
    # an index outside the cloud is refused (empty result), not read out of bounds
    assert mine.unpack_many(s, np.array([0, n], np.int32), convs[0], True).shape[0] == 0
    # a list longer than one staged chunk (65536 records) exercises the double-buffered path
    big = random_stream(rng, 5000, 3, 3)
    big.rotations.view("<u4")[:] &= np.uint32(0xEFFBFEFF)
    idx = rng.integers(0, 5000, 150_000).astype(np.int32)
    got = mine.unpack_many(big, idx, convs[1], True)
    uniq = theirs.unpack_many(big, np.arange(5000, dtype=np.int32), convs[1], False)
    assert np.array_equal(bits(got), bits(uniq[idx]))


@pytest.mark.gpu
def test_unpack_walk_reads_ahead_without_going_stale(mine, theirs, relinked):
    """A loop over packed.unpack(i, c) (load-spz.cc:461-463) is served from a read-ahead window after the first two
    consecutive indices.  The window is a memo keyed on the record's own bytes, the stream flavour, fractionalBits and
    the converter, so a caller that edits the planes, the header fields or the converter in the middle of the walk --
    here: three gaussians AHEAD of the cursor every 5th step, fractionalBits and flipP.x at the half-way point -- gets
    exactly what the reference returns.  Walks: in order over the whole cloud (windows of 16, 64, ... 4096 and a ragged
    last one), in order with jumps back and forth, and a shuffled one (no read-ahead at all)."""
    rng = np.random.default_rng(430)
    odd = (rng.normal(size=21) * 2).astype(np.float32)
    for ver, deg, n in ((3, 3, 6000), (2, 1, 300), (1, 0, 77), (4, 2, 1500)):
        s = random_stream(rng, n, deg, ver, 12)
        if ver >= 3:
            s.rotations.view("<u4")[:] &= np.uint32(0xEFFBFEFF)
        walks = [np.arange(n), np.concatenate([np.arange(40), np.arange(10, 200 if n > 200 else n), np.arange(n - 50, n), np.arange(0, n, 1)]),
                 rng.permutation(n)[:200]]
        for w, walk in enumerate(walks):
            for every in (0, 5):
                want = theirs.unpack_walk(s, walk, odd, every)
                assert np.array_equal(bits(mine.unpack_walk(s, walk, odd, every)), bits(want)), (ver, deg, w, every)
        assert np.array_equal(bits(relinked.unpack_walk(s, walks[0], odd, 5)), bits(theirs.unpack_walk(s, walks[0], odd, 5)))


@pytest.mark.gpu
def test_version2_files_are_read_by_the_reference(mine, theirs):
    """saveSpzV2 (extension, parity unpinned: the reference has no version-2 encoder): the container says version 2,
    the UNMODIFIED reference loads it down its first-three path, and this library's loader decodes the same bytes to
    the same floats; the quaternions come back within the 8-bit step of the normalised, w >= 0 input."""
    rng = np.random.default_rng(430)
    for deg in (0, 3):
        c = random_cloud(rng, 5000, deg, False)
        blob = mine.save_spz_v2(c, 6)
        raw = gzip.decompress(blob)
        assert struct.unpack_from("<III", raw, 0) == (0x5053474e, 2, 5000) and len(raw) == 16 + 5000 * (19 + 3 * SH_DIM[deg])
        a, b = mine.load_spz(blob, 8), theirs.load_spz(blob, 8)
        assert_cloud_bits_equal(a, b, f"v2 file deg{deg}")
        v3 = theirs.load_spz(theirs.save_spz(c, 6), 8)
        for name in ("positions", "scales", "alphas", "colors", "sh"):
            assert np.array_equal(bits(getattr(a, name)), bits(getattr(v3, name))), name
        q = c.rotations.reshape(-1, 4).astype(np.float64)
        q /= np.linalg.norm(q, axis=1, keepdims=True)
        q *= np.where(q[:, 3:4] < 0, -1.0, 1.0)
        want = q * np.concatenate([theirs.converter(6, 8)[3:6], [1.0]])
        assert np.abs(a.rotations.reshape(-1, 4)[:, :3] - want[:, :3]).max() <= 0.5 / 127.5 + 1e-6


@pytest.mark.gpu
def test_short_lived_threads_share_pooled_contexts(mine):
    """VERDICT r1 item 5: a server that packs from threads that come and go must not rebuild the GPU context
    (streams, tables, device staging, and above all the pinned bounce buffers: 0.1 - 0.4 s per context on these
    VMs) per thread.  400k SH3 points = 120 MB per call, so the bounce path is in play.  64 threads that each pack
    once and exit -- one after the other, and all at once -- take less than twice as long as 64 packs from one
    thread -- asserted with a generous 3x bound, since per-thread contexts cost 64 x the pinned allocation, an order of
    magnitude more; results identical."""
    rng = np.random.default_rng(420)
    c = random_cloud(rng, 400_000, 3, False)
    for _ in range(2):
        assert mine.short_lived_threads(c, 6, 8, True) >= 0      # warm: the pool's contexts and their buffers exist
    steady_ms = min(mine.short_lived_threads(c, 6, 64, 2) for _ in range(2))
    serial_ms = mine.short_lived_threads(c, 6, 64, False)
    burst_ms = min(mine.short_lived_threads(c, 6, 64, True) for _ in range(2))
    assert serial_ms >= 0 and burst_ms >= 0, "results differ between threads"
    print(f"64 packs of 400k SH3: one thread {steady_ms:.1f} ms, 64 one-shot threads in turn {serial_ms:.1f} ms, at once {burst_ms:.1f} ms")
    # measured: 464 / 455 / 183 ms (profiles/r2_pool_sweep.jsonl); per-thread contexts would add ~64 x 0.1-0.4 s of pinned allocation
    assert serial_ms < 3 * steady_ms + 50
    assert burst_ms < 3 * steady_ms + 50


@pytest.mark.gpu
@pytest.mark.parametrize("max_contexts", ["1", "3"])
def test_pool_limit_makes_callers_wait_not_fail(max_contexts):
    """SPZ_B200_MAX_CONTEXTS bounds the contexts per device; callers beyond it block until a lease comes back.  With
    a pool of ONE context, eight concurrent threads packing and unpacking still all finish with identical results
    (no deadlock, no failure); the variable is read when the pool is first used, hence the fresh process."""
    worker = (
        "import os, sys\n"
        "sys.path.insert(0, os.environ['REPO']); sys.path.insert(0, os.path.join(os.environ['REPO'], 'tests'))\n"
        "import ctypes as C, numpy as np\n"
        "from test_cxx_api import Shim\n"
        "from util import random_cloud\n"
        "mine = Shim('b200')\n"
        "c = random_cloud(np.random.default_rng(5), 300_000, 3, False)\n"
        "_, ip = mine._fplanes(c.planes())\n"
        "diff = mine.fn('concurrent_roundtrip')(C.c_int32(c.n), C.c_int32(3), C.c_int32(6), C.c_int32(8), ip, C.c_int32(8))\n"
        "print('diff', diff)\n")
    r = subprocess.run([sys.executable, "-c", worker], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, REPO=ROOT, SPZ_B200_MAX_CONTEXTS=max_contexts, SPZB200_NO_REBUILD="1"))
    assert r.returncode == 0 and "diff 0" in r.stdout, (r.stdout[-500:], r.stderr[-1500:])


@pytest.mark.gpu
def test_reference_suite_fixture_roundtrip(mine, theirs):
    """The reference test-suite's canonical 2-gaussian fixture (load_spz_test.py:72-147) through
    saveSpz -> loadSpz, with its tolerances, and bit-equality with the reference itself."""
    c = Cloud(2, 3, np.array([0, .1, -.2, .3, .4, .5], np.float32), np.array([-3, -2, -1.5, -1, 0, .1], np.float32),
              np.array([-.5, .2, 1, -.2, .1, -.4, -.3, .5], np.float32), np.array([-1, 1], np.float32),
              np.array([-1, 0, 1, -.5, .5, .1], np.float32), (np.arange(90, dtype=np.float32) / 45.0 - 1.0).astype(np.float32), True)
    blob = mine.save_spz(c, 0)
    assert len(blob) == 126 and blob == theirs.save_spz(c, 0)
    g = mine.load_spz(blob, 0)
    assert g.n == 2 and g.sh_degree == 3 and g.antialiased
    assert np.allclose(g.positions, c.positions, atol=1 / 2048)
    assert np.allclose(g.scales, c.scales, atol=1 / 32)
    assert np.allclose(g.alphas, c.alphas, atol=0.01 * 8)
    assert np.allclose(g.sh, np.clip(c.sh, -1, 0.9922), atol=2 / 32 + 0.5 / 255)
    assert_cloud_bits_equal(g, theirs.load_spz(blob, 0), "fixture")


# =================================================================================================
# the reference's command-line tools, relinked
# =================================================================================================

def _cli(tool: str, flavour: str) -> str:
    """tests/cxx/_build/<tool>_<flavour>: cli_tools/src/<tool>.cpp of the reference, compiled unchanged against the
    reference's headers and linked to libspz_b200.so (`b200`) or to the reference's own sources (`ref`)."""
    exe = os.path.join(CXX, "_build", f"{tool}_{flavour}")
    if os.path.isdir("/root/reference/cli_tools/src"):
        from spz_b200 import _native
        _native.lib()
        subprocess.run(["make", "-s", "-C", CXX, "cli"], check=True)
    if not os.path.exists(exe):
        pytest.skip(f"{exe} not built and cannot be built here")
    return exe


def _run(exe: str, *args: str):
    r = subprocess.run([exe, *args], capture_output=True, text=True, timeout=300)
    return r.returncode, r.stdout, r.stderr


def test_reference_cli_tools_link_against_this_library(tmp_path):
    """SURVEY.md 8b 'callers of the hot path: CLIs via the file API': the three tools build from the reference's
    unchanged sources against libspz_b200.so with no undefined symbol, and behave like the reference's where no device is
    needed (usage text; an unreadable or empty input)."""
    for tool in ("ply_to_spz", "spz_to_ply", "spz_info"):
        a, b = _cli(tool, "b200"), _cli(tool, "ref")
        assert _run(a) == _run(b)  # usage
    junk = tmp_path / "junk.spz"
    junk.write_bytes(b"not a gzip member")
    mine_out, ref_out = _run(_cli("spz_info", "b200"), str(junk)), _run(_cli("spz_info", "ref"), str(junk))
    assert mine_out[0] == ref_out[0] == 0 and mine_out[1].splitlines()[-1] == ref_out[1].splitlines()[-1] == "Number of points: 0"
    empty = tmp_path / "empty.spz"
    empty.write_bytes(Shim("ref").save_spz(Cloud(0, 0, *[np.zeros(0, np.float32)] * 6), 0))
    assert _run(_cli("spz_info", "b200"), str(empty)) == _run(_cli("spz_info", "ref"), str(empty))


@pytest.mark.gpu
@pytest.mark.parametrize("deg", [0, 3])
def test_reference_cli_tools_relinked_produce_the_same_files(theirs, tmp_path, deg):
    """ply_to_spz, spz_to_ply and spz_info of the reference, relinked to this library, against the same tools built with
    the reference's sources: identical .spz bytes, identical .ply bytes, identical report."""
    rng = np.random.default_rng(700 + deg)
    c = random_cloud(rng, 12_345, deg, False)
    ply = str(tmp_path / "in.ply")
    assert theirs.save_ply(c, ply, 0)
    out = {}
    for flavour in ("b200", "ref"):
        spz_file, back = str(tmp_path / f"{flavour}.spz"), str(tmp_path / f"{flavour}.ply")
        assert _run(_cli("ply_to_spz", flavour), ply, spz_file)[0] == 0
        assert _run(_cli("spz_to_ply", flavour), spz_file, back)[0] == 0
        info = _run(_cli("spz_info", flavour), spz_file)
        assert info[0] == 0
        out[flavour] = (open(spz_file, "rb").read(), open(back, "rb").read(), info[1])
    assert out["b200"][0] == out["ref"][0], "ply_to_spz: .spz bytes"
    assert out["b200"][1] == out["ref"][1], "spz_to_ply: .ply bytes"
    assert out["b200"][2] == out["ref"][2] and f"Number of points: {c.n}" in out["ref"][2], "spz_info report"
    # and crosswise: each side's tool reads the other side's file
    assert _run(_cli("spz_info", "b200"), str(tmp_path / "ref.spz"))[1] == out["ref"][2]
    assert _run(_cli("spz_info", "ref"), str(tmp_path / "b200.spz"))[1] == out["ref"][2]
