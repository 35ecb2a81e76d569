"""Context.quantize_device / spzb200_quantize_device and codec.quantize_straight_through: the codec's round
trip on float planes in one kernel.  The exact oracle is the device encoder followed by the device decoder:
every output float must equal theirs bit for bit (compared as uint32, NaN payloads included, since both run
the same device arithmetic).  The CPU oracle and the reference-made golden fixtures pin it from outside."""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from oracle import Cloud, bits
from util import PLANES, SPECIALS, golden_cloud, random_cloud, rotation_guard_stress

pytestmark = pytest.mark.gpu

SENTINEL = 0x7FA5A5A5  # a NaN payload the kernels never produce


def _torch():
    import torch
    return torch


def to_dev_cloud(c: Cloud):
    from spz_b200.codec import CloudPlanes
    t = _torch()
    return CloudPlanes(c.n, c.sh_degree, *[t.from_numpy(np.ascontiguousarray(p, np.float32).copy()).cuda() for p in c.planes()])


def dev_random_cloud(n, deg, seed, special=True):
    """random_cloud's value ranges and special-value salting, generated on the device."""
    from spz_b200.codec import CloudPlanes, float_plane_widths
    t = _torch()
    g = t.Generator(device="cuda").manual_seed(seed)
    specials = t.from_numpy(SPECIALS).cuda()
    ranges = [(-10, 10), (-12, 8), (-1, 1), (-8, 8), (-4, 4), (-1.2, 1.2)]

    def f(k, lo, hi):
        a = t.rand(k, generator=g, device="cuda") * (hi - lo) + lo
        if special and k:
            m = max(1, k // 12)
            a[t.randint(0, k, (m,), generator=g, device="cuda")] = specials[t.randint(0, specials.numel(), (m,), generator=g, device="cuda")]
        return a

    return CloudPlanes(n, deg, *[f(n * w, lo, hi) for w, (lo, hi) in zip(float_plane_widths(deg), ranges)])


def encode_decode(ctx, cloud, frm, to, version):
    return ctx.decode_device(ctx.encode_device(cloud, frm, version=version), to)


def assert_same_bits(got, want, what=""):
    t = _torch()
    for name, x, y in zip(PLANES, got.planes(), want.planes()):
        assert x.shape == y.shape, (what, name, x.shape, y.shape)
        neq = x.view(t.int32) != y.view(t.int32)
        if bool(neq.any()):
            i = neq.nonzero().flatten()[:5]
            raise AssertionError(f"{what} {name}: {int(neq.sum())} mismatches, first at {i.tolist()}: "
                                 f"{[hex(v & 0xffffffff) for v in x.view(t.int32)[i].tolist()]} vs "
                                 f"{[hex(v & 0xffffffff) for v in y.view(t.int32)[i].tolist()]}")


def sentinel_cloud(n, deg):
    from spz_b200.codec import CloudPlanes, float_plane_widths
    t = _torch()
    return CloudPlanes(n, deg, *[t.full((n * w,), SENTINEL, dtype=t.int32, device="cuda").view(t.float32) for w in float_plane_widths(deg)])


def all_sentinel(c):
    t = _torch()
    t.cuda.synchronize()
    return all(bool((p.view(t.int32) == SENTINEL).all()) for p in c.planes())


# ---- bit equality with encode_device + decode_device ----------------------------------------------

@pytest.mark.parametrize("version", [2, 3])
@pytest.mark.parametrize("deg", [0, 1, 2, 3])
@pytest.mark.parametrize("size", ["0", "1", "tile-1", "tile", "tile+1", "1M+7"])
def test_matches_encode_then_decode(gpu_ctx, deg, version, size):
    from spz_b200.codec import tile_gaussians
    tg = tile_gaussians(deg)
    n = {"0": 0, "1": 1, "tile-1": tg - 1, "tile": tg, "tile+1": tg + 1, "1M+7": 1_000_007}[size]
    c = dev_random_cloud(n, deg, 100 + 10 * deg + version)
    c.antialiased = True
    launches = gpu_ctx.info()["kernel_launches"]
    got = gpu_ctx.quantize_device(c, 6, version=version)
    assert gpu_ctx.info()["kernel_launches"] - launches == (1 if n else 0)
    assert got.n == n and got.sh_degree == deg and got.antialiased
    assert_same_bits(got, encode_decode(gpu_ctx, c, 6, 6, version), f"n={n}")


@pytest.mark.parametrize("version", [2, 3])
@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_every_coordinate_system_and_cross_pairs(gpu_ctx, deg, version):
    from spz_b200.codec import tile_gaussians
    c = dev_random_cloud(2 * tile_gaussians(deg) + 77, deg, 200 + 10 * deg + version)
    pairs = [(s, s) for s in range(9)] + [(0, 8), (8, 0), (4, 6), (6, 1), (1, 4), (2, 7), (7, 3), (5, 2)]
    for frm, to in pairs:
        assert_same_bits(gpu_ctx.quantize_device(c, frm, to, version), encode_decode(gpu_ctx, c, frm, to, version), f"{frm}->{to}")


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
@pytest.mark.parametrize("tag", ["tame", "wild"])
def test_golden_clouds(gpu_ctx, golden, deg, tag):
    """The reference-made golden clouds: equal to the device route, and to the reference's own
    unpackGaussians(packGaussians(c, from = 0), to) (NaNs as a class)."""
    key = f"c{deg}_{tag}"
    c = to_dev_cloud(golden_cloud(golden, key + "_in", 257, deg))
    for version in (2, 3):
        for frm, to in ((0, 0), (6, 6), (7, 8), (0, 6)):
            assert_same_bits(gpu_ctx.quantize_device(c, frm, to, version), encode_decode(gpu_ctx, c, frm, to, version), (key, frm, to))
    for to in (0, 6, 8):
        got = gpu_ctx.quantize_device(c, 0, to)
        for name, plane in zip(PLANES, got.planes()):
            assert np.array_equal(bits(plane.cpu().numpy()), golden[f"{key}_unpack_to{to}_{name}"]), (key, to, name)


def test_known_answer_cloud(gpu_ctx, golden):
    c = to_dev_cloud(golden_cloud(golden, "kat_in", 2, 3))
    for to in (0, 8):
        got = gpu_ctx.quantize_device(c, 0, to)
        for name, plane in zip(PLANES, got.planes()):
            assert np.array_equal(bits(plane.cpu().numpy()), golden[f"kat_unpack_to{to}_{name}"]), (to, name)


def test_float_sweeps_in_every_plane(gpu_ctx):
    """Every plane carries float bit patterns strided over all 2^32 (NaNs, Infs, denormals, both signs, the
    rounding ties of the quantizer sweeps), at SH degree 3 so both SH buckets and every flip phase occur."""
    from spz_b200.codec import CloudPlanes, float_plane_widths
    t = _torch()
    stride = 4099
    n = ((1 << 32) // stride) // 45
    planes = []
    for k, w in enumerate(float_plane_widths(3)):
        u = (t.arange(w * n, dtype=t.int64, device="cuda") * stride + 5 + k) & 0xffffffff
        planes.append(((u ^ (1 << 31)) - (1 << 31)).to(t.int32).view(t.float32))  # the low 32 bits as int32
    c = CloudPlanes(n, 3, *planes)
    for version in (2, 3):
        for frm, to in ((0, 0), (5, 5), (6, 8)):
            assert_same_bits(gpu_ctx.quantize_device(c, frm, to, version), encode_decode(gpu_ctx, c, frm, to, version), (version, frm, to))


def test_alpha_every_float_near_every_threshold(gpu_ctx):
    from spz_b200.codec import CloudPlanes
    t = _torch()
    thr, _ = gpu_ctx.tables()
    tb = thr[:255].view(np.uint32).astype(np.int64)
    u = (tb[:, None] + np.arange(-64, 64, dtype=np.int64)[None, :]).reshape(-1).astype(np.uint32)
    n = u.size
    z = lambda k: t.zeros(k, device="cuda")  # noqa: E731
    c = CloudPlanes(n, 0, z(3 * n), z(3 * n), z(4 * n), t.from_numpy(u.view(np.float32).copy()).cuda(), z(3 * n), z(0))
    assert_same_bits(gpu_ctx.quantize_device(c), encode_decode(gpu_ctx, c, 0, 0, 3))


def test_rotation_guard_boundaries(gpu_ctx):
    from spz_b200.codec import CloudPlanes
    t = _torch()
    rng = np.random.default_rng(78)
    n = 2_000_000
    rot = t.from_numpy(rotation_guard_stress(rng, n)).cuda()
    z = lambda k: t.zeros(k, device="cuda")  # noqa: E731
    c = CloudPlanes(n, 0, z(3 * n), z(3 * n), rot, z(n), z(3 * n), z(0))
    for version in (2, 3):
        for frm, to in ((0, 0), (5, 5), (8, 3)):
            assert_same_bits(gpu_ctx.quantize_device(c, frm, to, version), encode_decode(gpu_ctx, c, frm, to, version), (version, frm, to))


def test_10m_sh3(gpu_ctx):
    n = 10_000_000
    c = dev_random_cloud(n, 3, 7)
    for version in (3, 2):
        assert_same_bits(gpu_ctx.quantize_device(c, 6, version=version), encode_decode(gpu_ctx, c, 6, 6, version), f"v{version}")


# ---- the CPU oracle --------------------------------------------------------------------------------

@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_against_the_cpu_oracle(gpu_ctx, oracle, deg):
    """oracle unpack(pack(c, from), to) on a sample of the gaussians of a salted cloud, version 3."""
    rng = np.random.default_rng(400 + deg)
    n = 300_001
    c = random_cloud(rng, n, deg, special=True)
    dc = to_dev_cloud(c)
    idx = np.sort(rng.choice(n, 20_000, replace=False))
    d = c.sh.size // n if n else 0
    widths = (3, 3, 4, 1, 3, d)
    sub = Cloud(idx.size, deg, *[p.reshape(n, w)[idx].reshape(-1) if w else p for p, w in zip(c.planes(), widths)])
    for frm, to in ((0, 0), (6, 6), (3, 8)):
        got = gpu_ctx.quantize_device(dc, frm, to)
        want = oracle.unpack(oracle.pack(sub, frm), to)
        for name, g, wnt, w in zip(PLANES, got.planes(), want.planes(), widths):
            if not w:
                continue
            gs = g.cpu().numpy().reshape(n, w)[idx].reshape(-1)
            assert np.array_equal(bits(gs), bits(wnt)), (deg, frm, to, name)


# ---- in place, under-aligned planes, guard bands ---------------------------------------------------

@pytest.mark.parametrize("deg", [0, 3])
def test_in_place_equals_out_of_place(gpu_ctx, deg):
    from spz_b200.codec import CloudPlanes, tile_gaussians
    c = dev_random_cloud(3 * tile_gaussians(deg) + 5, deg, 500 + deg)
    for version in (2, 3):
        want = gpu_ctx.quantize_device(c, 7, 7, version)
        work = CloudPlanes(c.n, deg, *[p.clone() for p in c.planes()], antialiased=True)
        got = gpu_ctx.quantize_device(work, 7, 7, version, out=work)
        assert got is work and work.antialiased
        assert_same_bits(work, want, f"in place v{version}")


@pytest.mark.parametrize("deg", [0, 1, 3])
def test_under_aligned_planes(gpu_ctx, deg):
    """Planes that start one float into their buffer (4 bytes past 16-byte alignment), as input, as output
    and both, give the aligned result."""
    from spz_b200.codec import CloudPlanes, tile_gaussians
    t = _torch()
    n = 2 * tile_gaussians(deg) + 9
    c = dev_random_cloud(n, deg, 600 + deg)
    want = gpu_ctx.quantize_device(c, 5, 2)

    def shifted(src):
        return CloudPlanes(n, deg, *[t.cat([t.zeros(1, device="cuda"), p])[1:] for p in src.planes()])

    sin = shifted(c)
    assert all(p.data_ptr() % 16 == 4 for p in sin.planes() if p.numel())
    for src, dst in ((sin, None), (c, shifted(sentinel_cloud(n, deg))), (sin, shifted(sentinel_cloud(n, deg)))):
        got = gpu_ctx.quantize_device(src, 5, 2, out=dst)
        assert_same_bits(got, want, "under-aligned")
    got = gpu_ctx.quantize_device(sin, 5, 2, out=sin)  # in place, under-aligned
    assert_same_bits(got, want, "under-aligned in place")


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_writes_only_its_planes(gpu_ctx, deg):
    """Guard bands: every output plane sits inside a larger sentinel-filled buffer; after assorted sizes --
    one off either side of the encoder's tile and of this kernel's slices, odd counts whose planes end inside
    a float4 -- the bands are untouched.  Also in place inside such buffers."""
    from spz_b200.codec import CloudPlanes, float_plane_widths, tile_gaussians
    t = _torch()
    tg = tile_gaussians(deg)
    pad = 4096
    ws = float_plane_widths(deg)
    for n in (1, 3, 31, 87, 89, 167, 169, 451, 453, 1363, 1365, tg - 1, tg, tg + 1, 2 * tg + 7):
        c = dev_random_cloud(n, deg, 700 + n)
        want = encode_decode(gpu_ctx, c, 6, 6, 3)
        for in_place in (False, True):
            bufs = [t.full((n * w + 2 * pad,), SENTINEL, dtype=t.int32, device="cuda").view(t.float32) for w in ws]
            out = CloudPlanes(n, deg, *[b[pad:pad + n * w] for b, w in zip(bufs, ws)])
            if in_place:
                for o, p in zip(out.planes(), c.planes()):
                    o.copy_(p)
            gpu_ctx.quantize_device(out if in_place else c, 6, out=out)
            t.cuda.synchronize()
            for name, b, w in zip(PLANES, bufs, ws):
                bi = b.view(t.int32)
                assert bool((bi[:pad] == SENTINEL).all()) and bool((bi[pad + n * w:] == SENTINEL).all()), (n, name, in_place)
            assert_same_bits(out, want, f"n={n} in_place={in_place}")


# ---- the straight-through estimator ---------------------------------------------------------------

@pytest.mark.parametrize("deg", [0, 3])
def test_straight_through_forward_and_gradient(gpu_ctx, deg):
    from spz_b200.codec import CloudPlanes, quantize_straight_through
    t = _torch()
    n = 10_007
    base = dev_random_cloud(n, deg, 800 + deg, special=False)
    leaves = [p.clone().requires_grad_(True) for p in base.planes()]
    c = CloudPlanes(n, deg, *leaves, antialiased=True)
    for version in (2, 3):
        out = quantize_straight_through(gpu_ctx, c, 6, version)
        assert out.antialiased and out.n == n and out.sh_degree == deg
        assert_same_bits(CloudPlanes(n, deg, *[p.detach() for p in out.planes()]), gpu_ctx.quantize_device(base, 6, 6, version))
        assert all(p.requires_grad for p in out.planes() if p.numel())
        g = t.Generator(device="cuda").manual_seed(version)
        ups = [t.randn(p.shape, generator=g, device="cuda") for p in out.planes()]
        used = [i for i, p in enumerate(out.planes()) if p.numel()]
        grads = t.autograd.grad([out.planes()[i] for i in used], [leaves[i] for i in used], [ups[i] for i in used])
        for i, gr in zip(used, grads):
            assert t.equal(gr, ups[i]), (version, PLANES[i])
    # a scalar loss through it: d(sum(w * q(x)))/dx = w
    w = [t.rand(p.shape, device="cuda") for p in leaves]
    loss = sum((wi * q).sum() for wi, q in zip(w, quantize_straight_through(gpu_ctx, c, 6).planes()))
    loss.backward()
    for leaf, wi in zip(leaves, w):
        assert t.equal(leaf.grad, wi)
    # the input is not modified and nothing requires grad that should not
    assert_same_bits(CloudPlanes(n, deg, *[p.detach() for p in leaves]), base)
    with t.no_grad():
        assert not any(p.requires_grad for p in quantize_straight_through(gpu_ctx, c, 6).planes())
    plain = quantize_straight_through(gpu_ctx, base, 6)
    assert not any(p.requires_grad for p in plain.planes()) and not any(p.requires_grad for p in base.planes())


def test_straight_through_some_planes_without_grad(gpu_ctx):
    from spz_b200.codec import CloudPlanes, quantize_straight_through
    t = _torch()
    base = dev_random_cloud(1000, 1, 900, special=False)
    pos = base.positions.clone().requires_grad_(True)
    c = CloudPlanes(1000, 1, pos, *base.planes()[1:])
    out = quantize_straight_through(gpu_ctx, c, 0)
    assert out.positions.requires_grad and not out.colors.requires_grad
    (out.positions * 3).sum().backward()
    assert t.equal(pos.grad, t.full_like(pos, 3))


# ---- argument errors ------------------------------------------------------------------------------

def test_argument_errors_raise_and_leave_out_untouched(gpu_ctx):
    from spz_b200._native import ERR_INVALID, CodecError
    from spz_b200.codec import CloudPlanes
    t = _torch()
    n, deg = 1000, 2
    c = dev_random_cloud(n, deg, 1000)

    def expect_invalid(call, out):
        with pytest.raises(CodecError) as e:
            call()
        assert e.value.code == ERR_INVALID, e.value
        assert all_sentinel(out)

    out = sentinel_cloud(n, deg)
    # a wrong plane size, in the input and in the output
    short = CloudPlanes(n, deg, c.positions[:-1], *c.planes()[1:])
    expect_invalid(lambda: gpu_ctx.quantize_device(short, out=out), out)
    bad_out = CloudPlanes(n, deg, *out.planes()[:5], t.full((n * 24 + 1,), SENTINEL, dtype=t.int32, device="cuda").view(t.float32))
    expect_invalid(lambda: gpu_ctx.quantize_device(c, out=bad_out), bad_out)
    # out for another point count or SH degree
    other = sentinel_cloud(n + 1, deg)
    expect_invalid(lambda: gpu_ctx.quantize_device(c, out=other), other)
    # SH degree above 3
    expect_invalid(lambda: gpu_ctx.quantize_device(CloudPlanes(n, 4, *c.planes()), out=out), out)
    # versions other than 2 and 3, coordinate systems out of range
    for version in (0, 1, 4, 5):
        expect_invalid(lambda: gpu_ctx.quantize_device(c, version=version, out=out), out)
    for frm, to in ((9, 0), (0, 9), (-1, 0)):
        expect_invalid(lambda: gpu_ctx.quantize_device(c, frm, to, out=out), out)
    # partial overlaps: an output plane shifted against its input, an output plane on another input plane,
    # two output planes on one buffer
    big = t.full((3 * n + 3,), SENTINEL, dtype=t.int32, device="cuda").view(t.float32)
    cin = CloudPlanes(n, deg, big[:3 * n], *c.planes()[1:])
    o1 = CloudPlanes(n, deg, big[3:], *out.planes()[1:])
    expect_invalid(lambda: gpu_ctx.quantize_device(cin, out=o1), o1)
    o2 = CloudPlanes(n, deg, out.positions, c.positions, *out.planes()[2:])  # scales written over the positions read
    expect_invalid(lambda: gpu_ctx.quantize_device(c, out=o2), out)
    o3 = CloudPlanes(n, deg, out.positions, out.colors, *out.planes()[2:])  # scales and colours on one buffer
    expect_invalid(lambda: gpu_ctx.quantize_device(c, out=o3), o3)


def test_c_abi_rejects_bad_degree_and_null_planes(gpu_ctx):
    """The checks behind the Python ones, called through the C-ABI directly."""
    from spz_b200 import _native as N
    t = _torch()
    n = 64
    planes = [t.zeros(n * 45, device="cuda") for _ in range(6)]

    def cloud(deg, drop=None):
        s = N.Cloud()
        s.num_points, s.sh_degree = n, deg
        for i, (name, p) in enumerate(zip(PLANES, planes)):
            setattr(s, name, None if i == drop else p.data_ptr())
        return s

    stream = C.c_void_p(t.cuda.current_stream().cuda_stream)
    for cin, cout, version in ((cloud(4), cloud(4), 3), (cloud(3), cloud(3, drop=5), 3), (cloud(3, drop=0), cloud(3), 3),
                               (cloud(-1), cloud(-1), 3), (cloud(3), cloud(2), 3), (cloud(3), cloud(3), 1)):
        assert N.lib().spzb200_quantize_device(gpu_ctx._h, C.byref(cin), 0, 0, version, C.byref(cout), stream) == N.ERR_INVALID
    assert N.lib().spzb200_quantize_device(gpu_ctx._h, None, 0, 0, 3, C.byref(cloud(3)), stream) == N.ERR_INVALID
    assert N.lib().spzb200_quantize_device(None, C.byref(cloud(3)), 0, 0, 3, C.byref(cloud(3)), stream) == N.ERR_INVALID
