"""Parity tests proper: the sm_100a kernels, called through the C-ABI, against the CPU oracle
(oracle/spz_oracle.c, itself pinned to the unmodified reference by tests/test_oracle.py) and the
reference-made golden fixtures.  Bit-exact: encoded planes byte-equal, decoded floats bit-equal
(NaNs compared as a class -- x86 and sm_100a mint different NaN payloads, see oracle.bits)."""
from __future__ import annotations

import numpy as np
import pytest

from oracle import SH_DIM, Cloud, Packed, bits
from util import (PLANES, assert_cloud_bits_equal, assert_packed_equal, golden_cloud, golden_packed,
                  random_cloud, random_stream)

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    return torch


def to_dev_cloud(c: Cloud):
    from spz_b200.codec import CloudPlanes
    t = _torch()
    return CloudPlanes(c.n, c.sh_degree, *[t.from_numpy(np.ascontiguousarray(p, np.float32).copy()).cuda() for p in c.planes()])


def to_dev_packed(p: Packed):
    from spz_b200.codec import PackedPlanes
    t = _torch()
    return PackedPlanes(p.n, p.sh_degree, *[t.from_numpy(np.ascontiguousarray(a, np.uint8).copy()).cuda() for a in p.planes()],
                        fractional_bits=p.fractional_bits, version=p.version)


def host_packed(pp) -> Packed:
    _torch().cuda.synchronize()
    return Packed(pp.n, pp.sh_degree, pp.fractional_bits, pp.version, *[a.cpu().numpy() if hasattr(a, "cpu") else a for a in pp.planes()])


def host_cloud(cp) -> Cloud:
    _torch().cuda.synchronize()
    return Cloud(cp.n, cp.sh_degree, *[a.cpu().numpy() if hasattr(a, "cpu") else a for a in cp.planes()])


def gpu_pack(ctx, c: Cloud, frm=0) -> Packed:
    return host_packed(ctx.encode_device(to_dev_cloud(c), frm))


def gpu_unpack(ctx, p: Packed, to=0) -> Cloud:
    return host_cloud(ctx.decode_device(to_dev_packed(p), to))


# ---- golden fixtures (made by the unmodified reference) ---------------------------------------

def test_context_is_a_b200_and_loaded_native_code(gpu_ctx):
    info = gpu_ctx.info()
    assert info["sm_count"] >= 100
    thr, lut = gpu_ctx.tables()
    assert np.isposinf(thr[255]) and np.isneginf(lut[0]) and np.isposinf(lut[255])


def test_golden_kat(gpu_ctx, golden):
    c = golden_cloud(golden, "kat_in", 2, 3)
    for frm in (0, 6):
        assert_packed_equal(gpu_pack(gpu_ctx, c, frm), golden_packed(golden, f"kat_pack_from{frm}", 2, 3), f"kat from{frm}")
    p0 = golden_packed(golden, "kat_pack_from0", 2, 3)
    for to in (0, 8):
        g = gpu_unpack(gpu_ctx, p0, to)
        for name, plane in zip(PLANES, g.planes()):
            assert np.array_equal(bits(plane), golden[f"kat_unpack_to{to}_{name}"]), (to, name)


def test_golden_sh_known_answer(gpu_ctx, golden):
    edge = golden["shedge_in"]
    c = Cloud(1, 1, np.zeros(3, np.float32), np.zeros(3, np.float32), np.array([0, 0, 0, 1], np.float32),
              np.zeros(1, np.float32), np.zeros(3, np.float32), edge)
    p = gpu_pack(gpu_ctx, c, 0)
    assert np.array_equal(p.sh, golden["shedge_bytes"])
    assert np.array_equal(bits(gpu_unpack(gpu_ctx, p, 0).sh), golden["shedge_decoded"])


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
@pytest.mark.parametrize("tag", ["tame", "wild"])
def test_golden_clouds(gpu_ctx, golden, deg, tag):
    key = f"c{deg}_{tag}"
    c = golden_cloud(golden, key + "_in", 257, deg)
    for frm in (0, 6, 7):
        assert_packed_equal(gpu_pack(gpu_ctx, c, frm), golden_packed(golden, f"{key}_pack_from{frm}", 257, deg), f"{key} from{frm}")
    p0 = golden_packed(golden, f"{key}_pack_from0", 257, deg)
    for to in (0, 6, 8):
        g = gpu_unpack(gpu_ctx, p0, to)
        for name, plane in zip(PLANES, g.planes()):
            assert np.array_equal(bits(plane), golden[f"{key}_unpack_to{to}_{name}"]), (key, to, name)


@pytest.mark.parametrize("ver", [1, 2, 3])
@pytest.mark.parametrize("fb", [12, 0, 5, 31, 35])
def test_golden_streams(gpu_ctx, golden, ver, fb):
    deg = 3 if ver == 3 else 2
    key = f"s{ver}_fb{fb}"
    pk = golden_packed(golden, key + "_in", 131, deg, fb, ver)
    for to in (0, 7, 8):
        g = gpu_unpack(gpu_ctx, pk, to)
        for name, plane in zip(PLANES, g.planes()):
            assert np.array_equal(bits(plane), golden[f"{key}_unpack_to{to}_{name}"]), (key, to, name)


# ---- seeded random clouds against the oracle: vector path + remainder path ---------------------

@pytest.mark.parametrize("deg", [0, 1, 2, 3])
@pytest.mark.parametrize("special", [False, True])
def test_encode_all_coordinate_systems(gpu_ctx, oracle, deg, special):
    from spz_b200.codec import tile_gaussians
    rng = np.random.default_rng(1000 + deg * 2 + special)
    n = 3 * tile_gaussians(deg) + 77  # three full tiles on the vector kernel + a scalar remainder
    c = random_cloud(rng, n, deg, special)
    dc = to_dev_cloud(c)
    for frm in range(9):
        got = host_packed(gpu_ctx.encode_device(dc, frm))
        assert_packed_equal(got, oracle.pack(c, frm), f"deg{deg} from{frm}")


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
@pytest.mark.parametrize("ver", [1, 2, 3])
def test_decode_all_coordinate_systems(gpu_ctx, oracle, deg, ver):
    from spz_b200.codec import tile_gaussians
    rng = np.random.default_rng(2000 + deg * 3 + ver)
    n = 2 * tile_gaussians(deg) + 131
    for fb in (12, 9):
        s = random_stream(rng, n, deg, ver, fb)
        ds = to_dev_packed(s)
        for to in range(9):
            got = host_cloud(gpu_ctx.decode_device(ds, to))
            assert_cloud_bits_equal(got, oracle.unpack(s, to), f"deg{deg} v{ver} fb{fb} to{to}")


@pytest.mark.parametrize("deg", [0, 3])
def test_scalar_kernels_agree_with_vector_kernels(gpu_ctx, oracle, deg):
    from spz_b200.codec import tile_gaussians
    rng = np.random.default_rng(3000 + deg)
    n = 2 * tile_gaussians(deg) + 5
    c = random_cloud(rng, n, deg, True)
    want = oracle.pack(c, 6)
    try:
        gpu_ctx.set_force_generic(True)
        assert_packed_equal(gpu_pack(gpu_ctx, c, 6), want, "generic encode")
        assert_cloud_bits_equal(gpu_unpack(gpu_ctx, want, 7), oracle.unpack(want, 7), "generic decode")
    finally:
        gpu_ctx.set_force_generic(False)
    assert_packed_equal(gpu_pack(gpu_ctx, c, 6), want, "vector encode")
    assert_cloud_bits_equal(gpu_unpack(gpu_ctx, want, 7), oracle.unpack(want, 7), "vector decode")


def test_both_byte_packers(gpu_ctx, oracle):
    from spz_b200.codec import tile_gaussians
    rng = np.random.default_rng(3100)
    c = random_cloud(rng, 2 * tile_gaussians(3), 3, True)
    want = oracle.pack(c, 0)
    before = gpu_ctx.info()["pack_mode"]
    try:
        for cvt in (False, True):
            gpu_ctx.set_pack_mode(cvt)
            assert_packed_equal(gpu_pack(gpu_ctx, c, 0), want, f"cvt={cvt}")
    finally:
        gpu_ctx.set_pack_mode(before == "cvt.pack")


def test_under_aligned_pointers_take_the_scalar_path(gpu_ctx, oracle):
    """Slices that start at an odd gaussian are not 16-byte aligned: still exact."""
    from spz_b200.codec import CloudPlanes, tile_gaussians
    t = _torch()
    rng = np.random.default_rng(3200)
    deg = 3
    n = tile_gaussians(deg) + 9
    c = random_cloud(rng, n + 1, deg, False)
    full = to_dev_cloud(c)
    ws = (3, 3, 4, 1, 3, 45)
    sl = CloudPlanes(n, deg, *[p[w:] for p, w in zip(full.planes(), ws)])
    got = host_packed(gpu_ctx.encode_device(sl, 6))
    assert_packed_equal(got, oracle.pack(c.slice(1, n + 1), 6), "unaligned encode")
    del t


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_kernels_write_only_their_planes(gpu_ctx, oracle, deg):
    """Guard bands (compute-sanitizer is closed on this GPU pool): every output plane sits inside a
    larger 0xA5-filled buffer; after encode and decode of assorted sizes -- tile multiples, one off
    either side, sub-tile, odd counts that end in the scalar kernel -- the bands are untouched."""
    from spz_b200.codec import CloudPlanes, PackedPlanes, byte_plane_widths, float_plane_widths, tile_gaussians
    t = _torch()
    tg = tile_gaussians(deg)
    rng = np.random.default_rng(3300 + deg)
    pad = 4096
    for n in (1, 3, 31, tg - 1, tg, tg + 1, 2 * tg + 7, 3 * tg):
        c = random_cloud(rng, n, deg, False)
        want = oracle.pack(c, 6)
        bufs = [t.full((n * w + 2 * pad,), 0xA5, dtype=t.uint8, device="cuda") for w in byte_plane_widths(deg, 3)]
        out = PackedPlanes(n, deg, *[b[pad:pad + n * w] for b, w in zip(bufs, byte_plane_widths(deg, 3))])
        gpu_ctx.encode_device(to_dev_cloud(c), 6, out=out)
        t.cuda.synchronize()
        for name, b, w, exp in zip(PLANES, bufs, byte_plane_widths(deg, 3), want.planes()):
            assert bool((b[:pad] == 0xA5).all()) and bool((b[pad + n * w:] == 0xA5).all()), (n, name, "encode wrote outside its plane")
            assert np.array_equal(b[pad:pad + n * w].cpu().numpy(), exp), (n, name)
        fb = [t.full((n * w + 2 * pad,), float("nan"), dtype=t.float32, device="cuda") for w in float_plane_widths(deg)]
        fout = CloudPlanes(n, deg, *[b[pad:pad + n * w] for b, w in zip(fb, float_plane_widths(deg))])
        gpu_ctx.decode_device(to_dev_packed(want), 8, out=fout)
        t.cuda.synchronize()
        back = oracle.unpack(want, 8)
        for name, b, w, exp in zip(PLANES, fb, float_plane_widths(deg), back.planes()):
            assert bool(t.isnan(b[:pad]).all()) and bool(t.isnan(b[pad + n * w:]).all()), (n, name, "decode wrote outside its plane")
            assert np.array_equal(bits(b[pad:pad + n * w].cpu().numpy()), bits(exp)), (n, name)


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
@pytest.mark.parametrize("extra", [False, True])
def test_ply_kernels_write_only_their_planes(gpu_ctx, oracle, deg, extra):
    """Guard bands around every output of the fused PLY-rows kernels -- the bulk-copy kernels of the canonical
    property order (extra=False) and the column-map kernels (an extra column makes the layout non-canonical) --
    for sizes on both sides of every tile size in use (64 .. 512 gaussians) and odd remainders."""
    from spz_b200.codec import PackedPlanes, byte_plane_widths, ply_property_names
    from util import cloud_to_ply_rows
    t = _torch()
    rng = np.random.default_rng(3600 + 2 * deg + extra)
    names = ply_property_names(deg) + (["extra"] if extra else [])
    w, pad = len(names), 4096
    for n in (1, 63, 64, 65, 127, 128, 129, 255, 256, 257, 511, 512, 513, 3 * 512 + 77):
        c = random_cloud(rng, n, deg, False)
        rows = cloud_to_ply_rows(c, names).reshape(-1)
        want = oracle.pack(c, 6)
        bufs = [t.full((n * bw + 2 * pad,), 0xA5, dtype=t.uint8, device="cuda") for bw in byte_plane_widths(deg, 3)]
        out = PackedPlanes(n, deg, *[b[pad:pad + n * bw] for b, bw in zip(bufs, byte_plane_widths(deg, 3))])
        gpu_ctx.encode_ply_device(t.from_numpy(rows).cuda(), n, names, deg, 6, out=out)
        t.cuda.synchronize()
        for name, b, bw, exp in zip(PLANES, bufs, byte_plane_widths(deg, 3), want.planes()):
            assert bool((b[:pad] == 0xA5).all()) and bool((b[pad + n * bw:] == 0xA5).all()), (n, name, "PLY encode wrote outside its plane")
            assert np.array_equal(b[pad:pad + n * bw].cpu().numpy(), exp), (n, name)
        fb = t.full((n * w + 2 * pad,), float("nan"), dtype=t.float32, device="cuda")
        gpu_ctx.decode_ply_device(to_dev_packed(want), names, 8, out=fb[pad:pad + n * w])
        t.cuda.synchronize()
        assert bool(t.isnan(fb[:pad]).all()) and bool(t.isnan(fb[pad + n * w:]).all()), (n, "PLY decode wrote outside its records")
        exp = cloud_to_ply_rows(oracle.unpack(want, 8), names).reshape(-1)
        assert np.array_equal(bits(fb[pad:pad + n * w].cpu().numpy()), bits(exp)), n


@pytest.mark.parametrize("env", [{"SPZB200_GRID": "persistent"}, {"SPZB200_GRID": "persistent", "SPZB200_CTAS_PER_SM": "1"},
                                 {"SPZB200_DECODE": "direct"}, {"SPZB200_DECODE": "bulk"}, {"SPZB200_DECODE": "bulk", "SPZB200_GRID": "persistent"},
                                 {"SPZB200_DECODE": "pergaussian"}, {"SPZB200_DECODE": "pergaussian", "SPZB200_GRID": "persistent"},
                                 {"SPZB200_ENCODE": "bulk"}, {"SPZB200_ENCODE": "bulk", "SPZB200_GRID": "persistent"}, {"SPZB200_ENCODE": "tiles"},
                                 {"SPZB200_ENCODE": "tiles", "SPZB200_GRID": "persistent"},
                                 {"SPZB200_PACK": "alu"}, {"SPZB200_PLY": "mapped"},
                                 {"SPZB200_TILE": "128"}, {"SPZB200_TILE": "320"}, {"SPZB200_TILE": "128", "SPZB200_REST": "separate"},
                                 {"SPZB200_REST": "separate"}, {"SPZB200_PDL": "0"}, {"SPZB200_PDL": "0", "SPZB200_REST": "separate"}])
def test_alternate_launch_shapes(env):
    """The development knobs select other code paths of the same kernels (persistent multi-tile CTAs,
    which exercise the bulk decoder's mbarrier phase flip and buffer hand-over between tiles; the
    register-path decoder; the ALU byte packer).  scripts/sanitize_case.py runs every kernel variant
    against the oracle under each."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "scripts", "sanitize_case.py")], capture_output=True, text=True,
                       env=dict(os.environ, SPZB200_NO_REBUILD="1", **env), timeout=600)
    assert r.returncode == 0 and "sanitize_case ok" in r.stdout, (env, r.stdout[-1500:], r.stderr[-1500:])


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_fused_ply_rows_encoder(gpu_ctx, oracle, deg):
    """spzb200_encode_ply_device / _host: row-major .ply records -> packed planes, against the oracle's
    pack of the same cloud; shuffled column order, extra columns, tile multiples and remainders,
    an unaligned base pointer (scalar kernel) and the chunked host pipeline."""
    from spz_b200.codec import SH_DIM as DIM, ply_property_names
    t = _torch()
    rng = np.random.default_rng(3400 + deg)
    names = ply_property_names(deg)
    d = DIM[deg]
    for n, shuffle in ((512 * 3, False), (512 * 2 + 128 * 3 + 77, True), (90, False)):
        c = random_cloud(rng, n, deg, True)
        cols = {"x": c.positions[0::3], "y": c.positions[1::3], "z": c.positions[2::3],
                "nx": np.zeros(n, np.float32), "ny": np.zeros(n, np.float32), "nz": np.zeros(n, np.float32),
                "f_dc_0": c.colors[0::3], "f_dc_1": c.colors[1::3], "f_dc_2": c.colors[2::3], "opacity": c.alphas,
                "scale_0": c.scales[0::3], "scale_1": c.scales[1::3], "scale_2": c.scales[2::3],
                "rot_0": c.rotations[3::4], "rot_1": c.rotations[0::4], "rot_2": c.rotations[1::4], "rot_3": c.rotations[2::4]}
        sh = c.sh.reshape(n, d, 3) if d else np.zeros((n, 0, 3), np.float32)
        for ch in range(3):
            for s in range(d):
                cols[f"f_rest_{ch * d + s}"] = sh[:, s, ch]
        order = list(names)
        if shuffle:
            order = list(rng.permutation(order)) + ["extra_a", "extra_b"]
            cols["extra_a"] = rng.normal(size=n).astype(np.float32)
            cols["extra_b"] = rng.normal(size=n).astype(np.float32)
        rows = np.ascontiguousarray(np.stack([cols[k] for k in order], axis=1), np.float32).reshape(-1)
        for frm in (0, 6, 7):
            want = oracle.pack(c, frm)
            got = host_packed(gpu_ctx.encode_ply_device(t.from_numpy(rows).cuda(), n, order, deg, frm))
            assert_packed_equal(got, want, f"ply device deg{deg} n{n} from{frm}")
        # base pointer off by one float: not 16-byte aligned -> scalar kernel
        padded = t.from_numpy(np.concatenate([np.zeros(1, np.float32), rows])).cuda()
        got = host_packed(gpu_ctx.encode_ply_device(padded[1:], n, order, deg, 6))
        assert_packed_equal(got, oracle.pack(c, 6), "ply device unaligned")
        try:
            gpu_ctx.set_chunk_points(512)
            got, tm = gpu_ctx.encode_ply_host(rows, n, order, deg, 6)
            assert tm["chunks"] == (n + 511) // 512
            assert_packed_equal(Packed(n, deg, 12, 3, *got.planes()), oracle.pack(c, 6), "ply host")
        finally:
            gpu_ctx.set_chunk_points(0)


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
@pytest.mark.parametrize("ver", [1, 2, 3, 4])
def test_fused_ply_rows_decoder(gpu_ctx, oracle, deg, ver):
    """spzb200_decode_ply_device / _host: packed planes -> row-major records, against the oracle's
    unpack scattered into the same column layout."""
    from spz_b200.codec import SH_DIM as DIM, ply_property_names
    rng = np.random.default_rng(3500 + 4 * deg + ver)
    _fused_ply_rows_decoder_case(gpu_ctx, oracle, deg, ver, rng, ply_property_names(deg) + ["extra"])  # column-map kernels
    _fused_ply_rows_decoder_case(gpu_ctx, oracle, deg, ver, rng, ply_property_names(deg))  # canonical-layout kernel


def _fused_ply_rows_decoder_case(gpu_ctx, oracle, deg, ver, rng, names):
    from spz_b200.codec import SH_DIM as DIM
    d, w = DIM[deg], len(names)
    col = {k: i for i, k in enumerate(names)}
    for n in (512 * 2 + 300, 77):
        s = random_stream(rng, n, deg, ver, 11)
        for to in (0, 6):
            g = oracle.unpack(s, to)
            want = np.zeros((n, w), np.float32)
            for ax, k in enumerate("xyz"):
                want[:, col[k]] = g.positions[ax::3]
                want[:, col[f"scale_{ax}"]] = g.scales[ax::3]
                want[:, col[f"f_dc_{ax}"]] = g.colors[ax::3]
            want[:, col["opacity"]] = g.alphas
            for i, k in enumerate(("rot_1", "rot_2", "rot_3", "rot_0")):
                want[:, col[k]] = g.rotations[i::4]
            sh = g.sh.reshape(n, d, 3) if d else None
            for ch in range(3):
                for c in range(d):
                    want[:, col[f"f_rest_{ch * d + c}"]] = sh[:, c, ch]
            got = gpu_ctx.decode_ply_device(to_dev_packed(s), names, to)
            _torch().cuda.synchronize()
            assert np.array_equal(bits(got.cpu().numpy()), bits(want.reshape(-1))), (deg, ver, n, to)
        try:
            gpu_ctx.set_chunk_points(512)
            from spz_b200.codec import PackedPlanes
            got, tm = gpu_ctx.decode_ply_host(PackedPlanes(n, deg, *s.planes(), fractional_bits=11, version=ver), names, 6)
            assert tm["chunks"] == (n + 511) // 512
            assert np.array_equal(bits(got), bits(want.reshape(-1)))
        finally:
            gpu_ctx.set_chunk_points(0)


def test_empty_cloud(gpu_ctx):
    from spz_b200.codec import alloc_cloud, alloc_packed
    for deg in range(4):
        c = alloc_cloud(0, deg, device="cuda")
        p = gpu_ctx.encode_device(c, 6)
        assert p.n == 0 and p.version == 3 and p.fractional_bits == 12
        g = gpu_ctx.decode_device(alloc_packed(0, deg, 3, device="cuda"), 8)
        assert g.n == 0


def test_roundtrip_tolerances_of_the_reference_suite(gpu_ctx):
    """The per-attribute tolerances the reference's own tests assert (load_spz_test.py:113-178)."""
    rng = np.random.default_rng(1)
    n = 50_000
    c = Cloud(n, 3, rng.uniform(-10, 10, 3 * n).astype(np.float32), rng.uniform(-5, 2, 3 * n).astype(np.float32),
              rng.normal(size=4 * n).astype(np.float32), rng.uniform(-3, 3, n).astype(np.float32),
              rng.uniform(-1, 1, 3 * n).astype(np.float32), rng.uniform(-1, 1, 45 * n).astype(np.float32))
    g = gpu_unpack(gpu_ctx, gpu_pack(gpu_ctx, c, 0), 0)
    assert np.allclose(g.positions, c.positions, atol=1 / 2048)
    assert np.allclose(g.scales, c.scales, atol=1 / 16)
    sig = lambda x: 1 / (1 + np.exp(-x))  # noqa: E731
    assert np.allclose(sig(g.alphas), sig(c.alphas), atol=0.01)
    assert np.allclose(g.sh, c.sh, atol=2 / 32 + 1 / 255)
    q = g.rotations.reshape(-1, 4)
    assert np.allclose(np.linalg.norm(q, axis=1), 1, atol=1e-6 * 4)
    r = c.rotations.reshape(-1, 4)
    r = r / np.linalg.norm(r, axis=1, keepdims=True)
    assert np.all(np.abs(np.sum(q * r, axis=1)) > 1 - 1e-3)


# ---- exhaustive per-value sweeps on the real kernels ---------------------------------------------

def _sweep_cloud(vals_u32: np.ndarray, plane: str):
    """A degree-1 cloud whose `plane` carries the given float bit patterns."""
    f = vals_u32.view(np.float32)
    per = {"positions": 3, "scales": 3, "alphas": 1, "colors": 3, "sh": 9}[plane]
    n = f.size // per
    z3 = np.zeros(3 * n, np.float32)
    planes = dict(positions=z3, scales=z3, rotations=np.tile(np.array([0, 0, 0, 1], np.float32), n),
                  alphas=np.zeros(n, np.float32), colors=z3, sh=np.zeros(9 * n, np.float32))
    planes[plane] = f[:per * n]
    return Cloud(n, 1, *[planes[k] for k in PLANES])


@pytest.mark.parametrize("plane,which", [("alphas", 0), ("scales", 1), ("colors", 2)])
def test_quantizer_sweeps_all_float_classes(gpu_ctx, oracle, plane, which):
    """Strided over all 2^32 bit patterns (stride coprime to 2^32: NaNs, Infs, denormals, both
    signs) plus dense windows; the byte must equal the oracle's for every one."""
    stride = 2053
    count = ((1 << 32) // stride) // 36 * 36
    u = (np.arange(count, dtype=np.uint64) * stride + 17).astype(np.uint32)
    c = _sweep_cloud(u, plane)
    got = getattr(gpu_pack(gpu_ctx, c, 0), plane)
    want = oracle.sweep_u8(which, 17, stride, got.size)
    assert np.array_equal(got, want)


def test_alpha_every_float_near_every_threshold(gpu_ctx, oracle):
    thr, _ = gpu_ctx.tables()
    tb = thr[:255].view(np.uint32).astype(np.int64)
    win = np.arange(-64, 64, dtype=np.int64)
    u = (tb[:, None] + win[None, :]).reshape(-1).astype(np.uint32)
    u = np.resize(u, (u.size + 35) // 36 * 36)
    c = _sweep_cloud(u, "alphas")
    got = gpu_pack(gpu_ctx, c, 0).alphas
    want = np.array([oracle.lib.oracle_quant_alpha(float(x)) for x in u.view(np.float32)[:got.size]], np.uint8)
    assert np.array_equal(got, want)


def test_sh_sweep_both_buckets_and_flips(gpu_ctx, oracle):
    """SH values as float bit patterns strided over the full range, at degree 3 so both the 5-bit
    (first 9 values) and 4-bit buckets and every flipSh phase are exercised, from=LDF flips."""
    stride = 4099
    n = ((1 << 32) // stride) // 45
    u = (np.arange(45 * n, dtype=np.uint64) * stride + 5).astype(np.uint32)
    z3 = np.zeros(3 * n, np.float32)
    c = Cloud(n, 3, z3, z3, np.tile(np.array([0, 0, 0, 1], np.float32), n), np.zeros(n, np.float32), z3, u.view(np.float32))
    for frm in (0, 5, 6):
        assert np.array_equal(gpu_pack(gpu_ctx, c, frm).sh, oracle.pack(c, frm).sh), frm


def test_decode_every_byte_value_and_every_24bit_position(gpu_ctx, oracle):
    n = (1 << 24) // 3 + 1
    codes = np.resize(np.arange(1 << 24, dtype=np.uint32), 3 * n)
    pb = np.stack([codes & 255, (codes >> 8) & 255, codes >> 16], axis=1).astype(np.uint8).reshape(-1)
    rng = np.random.default_rng(5)
    ramp = np.resize(np.arange(256, dtype=np.uint8), 45 * n)
    s = Packed(n, 3, 12, 3, pb, ramp[:3 * n].copy(), rng.integers(0, 256, 4 * n).astype(np.uint8),
               ramp[:n].copy(), ramp[:3 * n].copy(), ramp.copy())
    for to in (0, 5):
        assert_cloud_bits_equal(gpu_unpack(gpu_ctx, s, to), oracle.unpack(s, to), f"to{to}")


def test_rotation_decode_first_three_exhaustive(gpu_ctx, oracle):
    n = 1 << 24
    b = np.arange(n, dtype=np.uint32)
    rb = np.stack([b & 255, (b >> 8) & 255, b >> 16], axis=1).astype(np.uint8).reshape(-1)
    z = np.zeros(9 * n, np.uint8)
    s = Packed(n, 0, 12, 2, z, z[:3 * n], rb, z[:n], z[:3 * n], np.zeros(0, np.uint8))
    got = gpu_unpack(gpu_ctx, s, 7)
    want = oracle.unpack(s, 7)
    assert np.array_equal(bits(got.rotations), bits(want.rotations))


def test_division_identities_on_the_device(gpu_ctx):
    """The quotients the smallest-three packer computes without a division (codec_math.cuh: one shared
    reciprocal + FMA residual corrections) equal the device's IEEE division bit for bit: exhaustively for
    the constant divisor sqrt1_2, and on 4e10 pseudo-random operand pairs of the guarded domain."""
    wrong, checked = gpu_ctx.selfcheck_division(0)
    assert wrong == 0 and checked == 0x3f8147ae - 0x17000000 + 2, (wrong, checked)  # 6.8e8 floats
    for seed in (1, 2):
        wrong, checked = gpu_ctx.selfcheck_division(1, 1 << 16, seed)
        assert wrong == 0 and checked >= 148 * 2048 * (1 << 16), (wrong, checked)


def test_rotation_encode_guard_boundaries(gpu_ctx, oracle):
    """As tests/test_device_math_host.py::test_rotations_encode_guard_boundaries, on the device: the
    Markstein-quotient fast path of the smallest-three packer and the general form behind its guard."""
    from util import rotation_guard_stress
    rng = np.random.default_rng(78)
    n = 2_000_000
    rot = rotation_guard_stress(rng, n)
    z3, z1 = np.zeros(3 * n, np.float32), np.zeros(n, np.float32)
    c = Cloud(n, 0, z3, z3, rot, z1, z3, np.zeros(0, np.float32))
    for frm in (0, 5, 8):
        got = gpu_pack(gpu_ctx, c, frm)
        want = oracle.pack(c, frm)
        bad = np.flatnonzero(got.rotations.view("<u4") != want.rotations.view("<u4"))
        assert bad.size == 0, (frm, bad[:5], rot.reshape(-1, 4)[bad[:5]])


def test_rotation_encode_decode_large_random(gpu_ctx, oracle):
    rng = np.random.default_rng(77)
    n = 4_000_000 // 1260 * 1260
    rot = rng.uniform(-1, 1, 4 * n).astype(np.float32)
    rot.reshape(-1, 4)[rng.integers(0, n, 5000), rng.integers(0, 4, 5000)] = 0.0
    rot[:8] = [0.5, 0.5, 0.5, 0.5, -0.5, 0.5, -0.5, 0.5]
    z3 = np.zeros(3 * n, np.float32)
    c = Cloud(n, 0, z3, z3, rot, np.zeros(n, np.float32), z3, np.zeros(0, np.float32))
    for frm in (0, 7):
        got = gpu_pack(gpu_ctx, c, frm)
        want = oracle.pack(c, frm)
        assert np.array_equal(got.rotations, want.rotations)
    # decode: all 2^22 combinations of two fields x index, third field random
    m = 1 << 22
    comp = rng.integers(0, 1 << 32, m, dtype=np.uint64).astype(np.uint32)
    comp = (comp & np.uint32(0x000003FF)) | (np.arange(m, dtype=np.uint32) << 10)
    z = np.zeros(9 * m, np.uint8)
    s = Packed(m, 0, 12, 3, z, z[:3 * m], comp.view(np.uint8).copy(), z[:m], z[:3 * m], np.zeros(0, np.uint8))
    for to in (0, 6):
        assert np.array_equal(bits(gpu_unpack(gpu_ctx, s, to).rotations), bits(oracle.unpack(s, to).rotations))


@pytest.mark.parametrize("deg,n", [(2, 1_200_037), (1, 1_100_011), (3, 1_000_003), (2, 999_000)])
def test_default_encoder_dispatch_by_size(gpu_ctx, oracle, deg, n):
    """The default encoder depends on the launch size: one thread per gaussian with bulk copies for SH degree 3 up to
    24M gaussians, degree 2 from 1M to 24M (128-bit shared-memory reads of the 24-word SH records), degree 1 up to 6M;
    register-path tiles elsewhere (pergaussian_kernels.cu: launchEncodePerGaussianPlanar).  Sizes on both sides of the
    degree-2 switch, with a ragged remainder, against the oracle -- NaN / Inf / huge inputs included."""
    rng = np.random.default_rng(5200 + deg)
    c = random_cloud(rng, n, deg, True)
    assert_packed_equal(gpu_pack(gpu_ctx, c, 7), oracle.pack(c, 7), f"deg{deg} n{n}")


# ---- the host-pointer pipeline (what the C++/Python drop-in API calls) -----------------------------

@pytest.mark.parametrize("deg", [0, 3])
def test_host_pipeline_chunked(gpu_ctx, oracle, deg):
    from spz_b200.codec import CloudPlanes, PackedPlanes, tile_gaussians
    rng = np.random.default_rng(4000 + deg)
    tg = tile_gaussians(deg)
    n = 7 * tg + 333
    c = random_cloud(rng, n, deg, True)
    want = oracle.pack(c, 6)
    try:
        gpu_ctx.set_chunk_points(2 * tg)  # 4 chunks: both stages, the drain, a ragged tail
        got, tm = gpu_ctx.encode_host(CloudPlanes(n, deg, *c.planes()), 6)
        assert tm["chunks"] == 4 and tm["kernel_launches"] >= 4
        assert tm["h2d_bytes"] == sum(p.nbytes for p in c.planes())
        assert tm["d2h_bytes"] == sum(p.nbytes for p in want.planes())
        assert_packed_equal(Packed(n, deg, 12, 3, *got.planes()), want, "encode_host")
        back, tm2 = gpu_ctx.decode_host(PackedPlanes(n, deg, *want.planes()), 7)
        assert tm2["chunks"] == 4
        assert_cloud_bits_equal(Cloud(n, deg, *back.planes()), oracle.unpack(want, 7), "decode_host")
    finally:
        gpu_ctx.set_chunk_points(0)


def test_host_pipeline_pageable_pinned_and_unstaged_agree(gpu_ctx, oracle):
    """Pageable planes are bounced through pinned buffers by host threads, pinned planes are copied
    directly, and the bounce can be switched off: three routes, one result."""
    from spz_b200.codec import CloudPlanes, PackedPlanes, alloc_cloud, alloc_packed, tile_gaussians
    rng = np.random.default_rng(4200)
    deg = 2
    n = 11 * tile_gaussians(deg) + 17
    c = random_cloud(rng, n, deg, False)
    want = oracle.pack(c, 7)
    want_back = oracle.unpack(want, 5)
    try:
        gpu_ctx.set_chunk_points(3 * tile_gaussians(deg))  # 4 ranges over 3 stages
        for label, pinned, bounce, staged in (("pageable", False, 2, 3), ("pinned", True, 2, 0), ("unstaged", False, 0, 0), ("auto-small", False, 1, 3)):
            gpu_ctx.set_host_staging(bounce, 3)
            src = alloc_cloud(n, deg, numpy_arrays=True, pinned=pinned)
            for a, b in zip(src.planes(), c.planes()):
                a[...] = b
            out = alloc_packed(n, deg, 3, numpy_arrays=True, pinned=pinned)
            got, tm = gpu_ctx.encode_host(src, 7, out=out)
            assert tm["staged"] == staged and tm["chunks"] == 4, (label, tm)
            assert_packed_equal(Packed(n, deg, 12, 3, *got.planes()), want, label)
            back = alloc_cloud(n, deg, numpy_arrays=True, pinned=pinned)
            got_back, tm = gpu_ctx.decode_host(out, 5, out=back)
            assert tm["staged"] == staged
            assert_cloud_bits_equal(Cloud(n, deg, *got_back.planes()), want_back, label)
    finally:
        gpu_ctx.set_chunk_points(0)
        gpu_ctx.set_host_staging(1, 0)


@pytest.mark.parametrize("deg,n,threads", [(3, 700_001, 0), (3, 300_000, 1), (0, 2_200_123, 3), (1, 1_000_000, 2)])
def test_host_pipeline_bounced_pieces(gpu_ctx, oracle, deg, n, threads):
    """The bounced pipeline at the sizes where it is more than one piece per plane and more ranges than stages: planes of
    tens of MB cut into 2 MiB pieces copied by the pool while earlier pieces are on the link, down pieces copied out
    behind their events, stages reused (9 ranges at SH degree 0).  Pageable on both sides, on the input side only and on
    the output side only; one copy thread (the calling thread does everything), a few, and the default."""
    from spz_b200.codec import alloc_cloud, alloc_packed
    rng = np.random.default_rng(4300 + deg)
    c = random_cloud(rng, n, deg, False)
    want = oracle.pack(c, 7)
    want_back = oracle.unpack(want, 5)
    try:
        gpu_ctx.set_host_staging(2, threads)
        for pin_in, pin_out in ((False, False), (False, True), (True, False)):
            src = alloc_cloud(n, deg, numpy_arrays=True, pinned=pin_in)
            for a, b in zip(src.planes(), c.planes()):
                a[...] = b
            out = alloc_packed(n, deg, 3, numpy_arrays=True, pinned=pin_out)
            got, tm = gpu_ctx.encode_host(src, 7, out=out)
            assert tm["staged"] == (0 if pin_in else 1) | (0 if pin_out else 2), tm
            assert tm["chunks"] == -(-n // (1 << 18)), tm  # 256K-point ranges
            assert_packed_equal(Packed(n, deg, 12, 3, *got.planes()), want, f"encode pinned={pin_in},{pin_out}")
            # decode: the packed planes take the role of the input
            pk = alloc_packed(n, deg, 3, numpy_arrays=True, pinned=pin_in)
            for a, b in zip(pk.planes(), want.planes()):
                a[...] = b
            back = alloc_cloud(n, deg, numpy_arrays=True, pinned=pin_out)
            got_back, tm = gpu_ctx.decode_host(pk, 5, out=back)
            assert tm["staged"] == (0 if pin_in else 1) | (0 if pin_out else 2), tm
            assert_cloud_bits_equal(Cloud(n, deg, *got_back.planes()), want_back, f"decode pinned={pin_in},{pin_out}")
    finally:
        gpu_ctx.set_host_staging(1, 0)


def test_host_multi_entry_point_single_device(oracle):
    """spzb200_*_host_multi with the devices present (1 here; more on a multi-GPU box): shards
    land at their precomputed offsets and the result is byte-identical to the unsharded one."""
    from spz_b200.codec import CloudPlanes, PackedPlanes, decode_host_multi, encode_host_multi, tile_gaussians
    t = _torch()
    devs = list(range(t.cuda.device_count()))
    rng = np.random.default_rng(4100)
    n = 9 * tile_gaussians(3) + 41
    c = random_cloud(rng, n, 3, False)
    want = oracle.pack(c, 0)
    for dl in (devs, devs + devs[:1]):  # the second form shards 2-ways even on one GPU
        got, tm = encode_host_multi(dl, CloudPlanes(n, 3, *c.planes()), 0)
        assert_packed_equal(Packed(n, 3, 12, 3, *got.planes()), want, f"multi encode {dl}")
        back, _ = decode_host_multi(dl, PackedPlanes(n, 3, *want.planes()), 8)
        assert_cloud_bits_equal(Cloud(n, 3, *back.planes()), oracle.unpack(want, 8), f"multi decode {dl}")


# ---- full-size, size-independent properties (BASELINE.json config 3: 10M SH3) ------------------

def test_full_size_10m_sh3_properties(gpu_ctx, oracle):
    """10M SH-degree-3 gaussians on the device.  The oracle checks sampled 64k-point blocks bit for
    bit; the whole cloud is checked through properties that need no CPU pass: decode(encode(x))
    re-encodes to the same bytes (idempotence of the quantizer on its own output), the flip of a
    flip is the identity, and shard-wise encoding equals whole-cloud encoding (checksum of planes)."""
    from spz_b200.codec import CloudPlanes, shard_range
    from spz_b200.synth import torch_cloud
    t = _torch()
    n, deg = 10_000_000, 3
    c = torch_cloud(n, deg, "cuda", seed=1)
    p = gpu_ctx.encode_device(c, 0)
    t.cuda.synchronize()
    # (1) sampled blocks against the oracle
    ws_f = (3, 3, 4, 1, 3, 45)
    for start in (0, 4_999_937, n - 65_536):
        blk = Cloud(65_536, deg, *[pl[w * start:w * (start + 65_536)].cpu().numpy() for pl, w in zip(c.planes(), ws_f)])
        want = oracle.pack(blk, 0)
        ws_b = (9, 3, 4, 1, 3, 45)
        for name, pl, w, wnt in zip(PLANES, p.planes(), ws_b, want.planes()):
            assert np.array_equal(pl[w * start:w * (start + 65_536)].cpu().numpy(), wnt), (start, name)
        dec = gpu_ctx.decode_device(to_dev_packed(want), 6)
        assert_cloud_bits_equal(host_cloud(dec), oracle.unpack(want, 6), f"decode block {start}")
    # (2) idempotence: encode(decode(p)) == p on every plane, all 10M points
    d = gpu_ctx.decode_device(p, 0)
    p2 = gpu_ctx.encode_device(d, 0)
    t.cuda.synchronize()
    for name, a, b in zip(PLANES, p.planes(), p2.planes()):
        if name == "rotations":
            continue  # smallest-three re-quantisation may move a component by one step (not idempotent in the reference either)
        assert t.equal(a, b), name
    # (3) a flip folded into the encoder equals the same flip folded into the decoder
    p_rdf = gpu_ctx.encode_device(c, 6)          # RDF -> RUB on the way in
    d_a = gpu_ctx.decode_device(p_rdf, 6)        # RUB -> RDF on the way out: flips cancel
    d_b = gpu_ctx.decode_device(p, 0)
    t.cuda.synchronize()
    for name, a, b in zip(PLANES, d_a.planes(), d_b.planes()):
        if name in ("sh", "rotations"):
            continue  # the SH bucket rounding ((q + b/2) / b * b) is not an odd function: ties move
        same = (a.view(t.int32) == b.view(t.int32)) | ((a == 0) & (b == 0))
        assert bool(same.all()), name  # round-half-away is odd, so flipped positions match exactly
    # (4) sharded encoding writes the same bytes as whole-cloud encoding
    from spz_b200.codec import alloc_packed, PackedPlanes
    out = alloc_packed(n, deg, 3, device="cuda")
    ws_b = (9, 3, 4, 1, 3, 45)
    for i in range(8):
        a, b = shard_range(n, deg, 8, i)
        ci = CloudPlanes(b - a, deg, *[pl[w * a:w * b] for pl, w in zip(c.planes(), ws_f)])
        oi = PackedPlanes(b - a, deg, *[pl[w * a:w * b] for pl, w in zip(out.planes(), ws_b)])
        gpu_ctx.encode_device(ci, 0, out=oi)
    t.cuda.synchronize()
    for name, a, b in zip(PLANES, p.planes(), out.planes()):
        assert t.equal(a, b), name


# ---- batched per-gaussian access (SURVEY.md 8f-4; load-spz.cc:383-463) ---------------------------

def test_unpack_gather_golden(gpu_ctx):
    """spzb200_unpack_gather_host / _device / _records_host against vectors made by the reference's own
    PackedGaussians::unpack(i, c): every stream flavour x SH degree x {identity, RUB->RDF, arbitrary factors}."""
    import os
    from spz_b200 import codec
    t = _torch()
    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_unpack_at.npz"))
    convs = G["converters"]
    for ver in (1, 2, 3, 4):
        for deg in range(4):
            key = f"v{ver}d{deg}"
            s = Packed(64, deg, int(G[f"{key}_fb"]), ver, *[G[f"{key}_{p}"] for p in PLANES])
            hp = codec.PackedPlanes(64, deg, *[np.ascontiguousarray(a) for a in s.planes()], fractional_bits=s.fractional_bits, version=ver)
            dp = to_dev_packed(s)
            idx = G[f"{key}_idx"]
            for k, conv in enumerate(convs):
                want = G[f"{key}_out{k}"]
                assert np.array_equal(bits(gpu_ctx.unpack_gather_host(hp, idx, conv)), want), (key, k, "host")
                got = gpu_ctx.unpack_gather_device(dp, t.from_numpy(idx).cuda(), conv)
                t.cuda.synchronize()
                assert np.array_equal(bits(got.cpu().numpy()), want), (key, k, "device")
                rec = codec.gather_records(hp, idx)
                assert np.array_equal(bits(gpu_ctx.unpack_records_host(rec, ver, s.fractional_bits, conv)), want), (key, k, "records")


def test_unpack_gather_against_the_oracle(gpu_ctx, oracle):
    """Larger random streams: all three entry points against oracle_unpack_at; a list longer than one staged chunk;
    indices == None; the small zero-copy path (n <= 2048) and the staged path give the same floats; and with a
    +-1 converter the gather equals the bulk decoder on the same gaussians."""
    from spz_b200 import codec
    from spz_b200._native import CodecError
    t = _torch()
    rng = np.random.default_rng(811)
    for ver, deg, n in ((3, 3, 70_001), (2, 1, 5_000), (1, 2, 3_001), (4, 0, 777), (3, 0, 129)):
        s = random_stream(rng, n, deg, ver, int(rng.choice([0, 7, 12, 31, 35])))
        if ver >= 3:
            s.rotations.view("<u4")[::3] &= np.uint32(0xEFFBFEFF)
        hp = codec.PackedPlanes(n, deg, *[np.ascontiguousarray(a) for a in s.planes()], fractional_bits=s.fractional_bits, version=ver)
        dp = to_dev_packed(s)
        conv = (rng.normal(size=21) * 2).astype(np.float32)
        for count in (1, 5, 2048, 2049, min(n, 40_000), 140_000):
            idx = rng.integers(0, n, count).astype(np.int64)
            want = bits(oracle.unpack_at(s, idx, conv))
            assert np.array_equal(bits(gpu_ctx.unpack_gather_host(hp, idx, conv)), want), (ver, deg, count, "host")
            got = gpu_ctx.unpack_gather_device(dp, t.from_numpy(idx).cuda(), conv)
            t.cuda.synchronize()
            assert np.array_equal(bits(got.cpu().numpy()), want), (ver, deg, count, "device")
        # no index list: gaussians 0..n-1 in order, no converter: identity
        want = bits(oracle.unpack_at(s, np.arange(n), oracle.converter(0, 0)))
        assert np.array_equal(bits(gpu_ctx.unpack_gather_host(hp)), want)
        got = gpu_ctx.unpack_gather_device(dp)
        t.cuda.synchronize()
        assert np.array_equal(bits(got.cpu().numpy()), want)
        # the bulk decoder with the same flips
        full = gpu_unpack(gpu_ctx, s, 6)
        rows = gpu_ctx.unpack_gather_host(hp, None, oracle.converter(4, 6))
        assert np.array_equal(bits(rows[:, 0:3].reshape(-1)), bits(full.positions))
        assert np.array_equal(bits(rows[:, 3:7].reshape(-1)), bits(full.rotations))
        assert np.array_equal(bits(rows[:, 7:10].reshape(-1)), bits(full.scales))
        assert np.array_equal(bits(rows[:, 13]), bits(full.alphas))
        with pytest.raises(CodecError):
            gpu_ctx.unpack_gather_host(hp, [0, n])
        with pytest.raises(CodecError):
            gpu_ctx.unpack_gather_host(hp, [-1])
    assert gpu_ctx.unpack_gather_host(hp, np.zeros(0, np.int64)).shape == (0, 59)


# ---- version-2 encoder (SURVEY.md 8f-4): PARITY UNPINNED, the reference has only the decoder -----------

@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_v2_encoder_against_its_restatement_and_the_reference_decoder(gpu_ctx, oracle, deg):
    """spzb200_encode_device_as / _host_as with stream version 2.  What CAN be pinned is pinned: (1) every plane but
    the rotations is byte-identical to the version-3 encoder's (which is pinned to the reference); (2) the rotation
    bytes equal oracle_pack_v2, the restatement of upstream's pre-smallest-three encoder; (3) the REFERENCE's own
    decoder (unpackQuaternionFirstThree, load-spz.cc:333-345; its C restatement where no build of the reference is
    present) turns them back into the normalised input quaternion
    (sign-fixed to w >= 0) within the 8-bit step; (4) tile kernel, scalar remainder, scalar-only path and host
    pipeline agree."""
    from oracle import Ref
    from spz_b200 import codec
    ref = Ref() if Ref.available() else oracle
    rng = np.random.default_rng(5200 + deg)
    n = 3 * codec.tile_gaussians(deg) + 333
    c = random_cloud(rng, n, deg, False)
    for frm in (0, 6, 7):
        v3 = gpu_pack(gpu_ctx, c, frm)
        got = host_packed(gpu_ctx.encode_device(to_dev_cloud(c), frm, version=2))
        assert got.version == 2 and got.rotations.size == 3 * n
        want = oracle.pack_v2(c, frm)
        for name in ("positions", "scales", "alphas", "colors", "sh"):
            assert np.array_equal(getattr(got, name), getattr(v3, name)), (frm, name)
        assert np.array_equal(got.rotations, want.rotations), frm
        # through the reference's decoder: q / |q|, flipped, sign chosen so that w >= 0
        back = ref.unpack(Packed(n, deg, 12, 2, *got.planes()), 0)
        q = c.rotations.reshape(n, 4).astype(np.float64)
        q /= np.linalg.norm(q, axis=1, keepdims=True)
        fq = np.concatenate([oracle.flips(frm, 4)[1], [1.0]])
        q = q * fq * np.where(q[:, 3:4] < 0, -1.0, 1.0)
        r = back.rotations.reshape(n, 4)
        assert np.abs(r[:, :3] - q[:, :3]).max() <= 0.5 / 127.5 + 1e-6
        ok = np.abs(q[:, 3]) > 0.2  # w = sqrt(1 - |xyz|^2) amplifies the byte error by (|x| + |y| + |z|) / w <= sqrt(3) / 0.2
        assert np.abs(r[ok, 3] - q[ok, 3]).max() < 0.04
    gpu_ctx.set_force_generic(True)
    try:
        assert np.array_equal(host_packed(gpu_ctx.encode_device(to_dev_cloud(c), 6, version=2)).rotations, oracle.pack_v2(c, 6).rotations)
    finally:
        gpu_ctx.set_force_generic(False)
    hp, _ = gpu_ctx.encode_host(codec.CloudPlanes(n, deg, *c.planes()), 6, version=2)
    assert np.array_equal(hp.rotations, oracle.pack_v2(c, 6).rotations) and np.array_equal(hp.sh, oracle.pack(c, 6).sh)
    # specials (NaN / Inf / zero quaternions): the restatement's x86 answers, byte for byte
    s = random_cloud(rng, 2 * codec.tile_gaussians(deg) + 5, deg, True)
    s.rotations[:8] = 0
    assert np.array_equal(host_packed(gpu_ctx.encode_device(to_dev_cloud(s), 1, version=2)).rotations, oracle.pack_v2(s, 1).rotations)
    with pytest.raises(Exception):
        gpu_ctx.encode_device(to_dev_cloud(c), 0, version=1)


def test_counter_seeded_cloud_is_the_same_on_host_and_device(gpu_ctx):
    """bench.py's workload (SURVEY.md 8d: counter-based, so shards generate identical data): the torch generator on the
    GPU gives, bit for bit, the numpy generator's slice of the same cloud -- whatever the slice and the scratch size."""
    from spz_b200.synth import counter_cloud_numpy, counter_cloud_torch
    t = _torch()
    n_total = 3_000_000
    for deg, a, b in ((3, 1280 * 700, 1280 * 700 + 40_001), (0, 0, 70_000), (1, n_total - 50_000, n_total)):
        host = counter_cloud_numpy(n_total, deg, a, b, seed=1)
        dev = counter_cloud_torch(n_total, deg, t.device("cuda", 0), a, b, seed=1, slice_elems=1 << 16)
        for name, x, y in zip(PLANES, host.planes(), dev.planes()):
            assert np.array_equal(x.view(np.uint32), y.cpu().numpy().view(np.uint32)), (deg, name)
    # and it is a sensible cloud: the encoder's output of a slice equals the oracle's
    c = counter_cloud_numpy(n_total, 3, 5 * 1280, 5 * 1280 + 3000, seed=1)
    from oracle import Oracle
    assert_packed_equal(gpu_pack(gpu_ctx, Cloud(3000, 3, *c.planes()), 6), Oracle().pack(Cloud(3000, 3, *c.planes()), 6), "counter cloud")


@pytest.mark.parametrize("deg", [0, 3])
def test_bench_dump_outputs_are_the_timed_step_results(oracle, tmp_path, deg):
    """bench.py --dump-outputs: the sampled rows of the last timed step's encoded and decoded planes equal the oracle's
    on the same counter-seeded cloud, every file is float32 or float64, and together they stay under 64 MB."""
    import json
    import os
    import subprocess
    import sys

    from spz_b200.codec import byte_plane_widths, float_plane_widths
    from spz_b200.synth import counter_cloud_numpy
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    n, out = 300_007, tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--points", str(n), "--sh-degree", str(deg),
                        "--steps", "2", "--warmup", "1", "--no-e2e", "--no-cpu-baseline", "--no-ply", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600, env=dict(os.environ, SPZB200_NO_REBUILD="1"))
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    assert sum(f.stat().st_size for f in out.iterdir()) <= 64 << 20
    idx = np.load(out / "indices.npy")
    assert idx.dtype == np.float64 and idx.size == 65536 and np.all(np.diff(idx) > 0) and idx[-1] < n
    rows = idx.astype(np.int64)
    want = oracle.pack(Cloud(n, deg, *counter_cloud_numpy(n, deg, seed=1).planes()), 6)
    back = oracle.unpack(want, 6)
    for name, wb, wf, pb, pf in zip(PLANES, byte_plane_widths(deg, 3), float_plane_widths(deg), want.planes(), back.planes()):
        enc, dec = np.load(out / f"encoded_{name}.npy"), np.load(out / f"decoded_{name}.npy")
        assert enc.dtype == dec.dtype == np.float32 and enc.shape == (rows.size, wb) and dec.shape == (rows.size, wf), name
        assert np.array_equal(enc, pb.reshape(n, wb)[rows].astype(np.float32)), name
        assert np.array_equal(bits(dec), bits(pf.reshape(n, wf)[rows])), name
