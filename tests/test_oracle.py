"""Pins oracle/spz_oracle.c (the CPU restatement) bit-for-bit against
  (a) the known answers SURVEY.md section 8c extracted from the reference,
  (b) tests/golden/golden.npz, produced by the UNMODIFIED reference (tests/golden/make_golden.py),
  (c) the live reference build oracle/_ref/libspz_ref.so wherever it is present.
No GPU, no product code."""
from __future__ import annotations

import numpy as np
import pytest

from oracle import SH_DIM, Cloud, Packed, bits
from util import (PLANES, assert_cloud_bits_equal, assert_packed_equal, golden_cloud, golden_packed,
                  random_cloud, random_stream)


def hexbytes(s: str) -> np.ndarray:
    return np.frombuffer(bytes.fromhex(s.replace("|", " ").replace(" ", "")), np.uint8)


def kat_cloud() -> Cloud:
    """The reference test-suite's canonical 2-gaussian fixture (tests/python/load_spz_test.py:72-100)."""
    return Cloud(2, 3,
                 np.array([0, .1, -.2, .3, .4, .5], np.float32),
                 np.array([-3, -2, -1.5, -1, 0, .1], np.float32),
                 np.array([-.5, .2, 1, -.2, .1, -.4, -.3, .5], np.float32),
                 np.array([-1, 1], np.float32),
                 np.array([-1, 0, 1, -.5, .5, .1], np.float32),
                 (np.arange(90, dtype=np.float32) / 45.0 - 1.0).astype(np.float32), True)


# ---- (a) SURVEY.md 8c known answers (typed in from the survey's probe of the reference) ---------

def test_kat_pack_unspecified(oracle):
    p = oracle.pack(kat_cloud(), 0)
    assert np.array_equal(p.positions, hexbytes("00 00 00 9a 01 00 cd fc ff | cd 04 00 66 06 00 00 08 00"))
    assert np.array_equal(p.alphas, hexbytes("45 ba"))
    assert np.array_equal(p.colors, hexbytes("59 80 a6 6c 93 83"))
    assert np.array_equal(p.scales, hexbytes("70 80 88 90 a0 a2"))
    assert np.array_equal(p.rotations, hexbytes("7d f6 91 b3 | 30 57 5e c6"))
    assert np.array_equal(p.sh[:18], hexbytes("00 00 08 08 08 10 10 18 18 20 20 20 20 20 30 30 30 30"))
    assert np.array_equal(p.sh[88:90], hexbytes("ff ff"))


def test_kat_pack_rdf(oracle):
    p = oracle.pack(kat_cloud(), 6)
    assert np.array_equal(p.positions, hexbytes("00 00 00 66 fe ff 33 03 00 | cd 04 00 9a f9 ff 00 f8 ff"))
    assert np.array_equal(p.rotations, hexbytes("7d f4 91 93 | 30 55 56 c6"))
    assert np.array_equal(p.sh[:6], hexbytes("ff ff f8 f8 f8 f0"))


def test_kat_unpack(oracle):
    p = oracle.pack(kat_cloud(), 0)
    g = oracle.unpack(p, 0)
    u = lambda s: np.array([int(x, 16) for x in s.replace("|", " ").split()], np.uint32)  # noqa: E731
    assert np.array_equal(bits(g.positions), u("00000000 3dcd0000 be4cc000 3e99a000 3eccc000 3f000000"))
    assert np.array_equal(bits(g.rotations), u("beddc1ee 3e311f65 3f5e14f3 be311f65 | 3e0f1d77 bf0f7826 bed76192 3f33186e"))
    assert np.array_equal(bits(g.alphas), u("bf7ddc20 3f7ddc23"))
    assert np.array_equal(bits(g.colors), u("bf80d62b 3c562c55 3f80d62c bf028282 3f028285 3dbb662a"))
    g8 = oracle.unpack(p, 8)
    assert bits(g8.positions)[2] == 0x3e4cc000 and bits(g8.positions)[5] == 0xbf000000
    assert np.array_equal(bits(g8.rotations), u("3eddc1ee be311f65 3f5e14f3 be311f65 | be0f1d77 3f0f7826 bed76192 3f33186e"))


def test_kat_v2_and_table_ends(oracle):
    n = 1
    pk = Packed(n, 0, 12, 2, np.zeros(9, np.uint8), np.zeros(3, np.uint8), np.array([0x00, 0x7f, 0xff], np.uint8),
                np.zeros(1, np.uint8), np.array([0x00, 0x80, 0xff], np.uint8), np.zeros(0, np.uint8))
    g = oracle.unpack(pk, 7)  # LUF
    assert [hex(v) for v in bits(g.rotations)] == ["0x3f800000", "0xbb808000", "0xbf800000", "0x0"]
    assert bits(g.alphas)[0] == 0xff800000
    assert [hex(v) for v in bits(g.colors)] == ["0xc0555555", "0x3c562c55", "0x40555555"]
    assert bits(g.positions)[0] == 0x80000000  # zero position under a -1 flip is -0.0
    pk.alphas[:] = 0xff
    assert bits(oracle.unpack(pk, 0).alphas)[0] == 0x7f800000


def test_sh_known_answer_of_reference_suite(oracle, golden):
    """test_sh_encoding_for_zeros_and_edges (load_spz_test.py:180-207): the reference's only KAT."""
    edge = np.array([-.01, 0, .01, -1, -.99, -.95, .95, .99, 1], np.float32)
    c = Cloud(1, 1, np.zeros(3, np.float32), np.zeros(3, np.float32), np.array([0, 0, 0, 1], np.float32),
              np.zeros(1, np.float32), np.zeros(3, np.float32), edge)
    p = oracle.pack(c, 0)
    assert np.array_equal(p.sh, golden["shedge_bytes"])
    dec = oracle.unpack(p, 0).sh
    assert np.array_equal(bits(dec), golden["shedge_decoded"])
    expected = np.array([0, 0, 0, -1, -1, -.9375, .9375, .9922, .9922], np.float32)
    assert np.allclose(dec, expected, atol=2e-5)  # the tolerance the reference test states


# ---- (b) golden fixtures made by the unmodified reference -------------------------------------

def test_golden_kat(oracle, golden):
    c = golden_cloud(golden, "kat_in", 2, 3)
    for frm in (0, 6):
        assert_packed_equal(oracle.pack(c, frm), golden_packed(golden, f"kat_pack_from{frm}", 2, 3), f"kat from{frm}")
    p0 = oracle.pack(c, 0)
    for to in (0, 8):
        g = oracle.unpack(p0, to)
        for name, plane in zip(PLANES, g.planes()):
            assert np.array_equal(bits(plane), golden[f"kat_unpack_to{to}_{name}"]), (to, name)


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
@pytest.mark.parametrize("tag", ["tame", "wild"])
def test_golden_clouds(oracle, golden, deg, tag):
    key = f"c{deg}_{tag}"
    c = golden_cloud(golden, key + "_in", 257, deg)
    for frm in (0, 6, 7):
        assert_packed_equal(oracle.pack(c, frm), golden_packed(golden, f"{key}_pack_from{frm}", 257, deg), f"{key} from{frm}")
    p0 = oracle.pack(c, 0)
    for to in (0, 6, 8):
        g = oracle.unpack(p0, to)
        for name, plane in zip(PLANES, g.planes()):
            assert np.array_equal(bits(plane), golden[f"{key}_unpack_to{to}_{name}"]), (key, to, name)


@pytest.mark.parametrize("ver", [1, 2, 3])
@pytest.mark.parametrize("fb", [12, 0, 5, 31, 35])
def test_golden_streams(oracle, golden, ver, fb):
    deg = 3 if ver == 3 else 2
    key = f"s{ver}_fb{fb}"
    pk = golden_packed(golden, key + "_in", 131, deg, fb, ver)
    for to in (0, 7, 8):
        g = oracle.unpack(pk, to)
        for name, plane in zip(PLANES, g.planes()):
            assert np.array_equal(bits(plane), golden[f"{key}_unpack_to{to}_{name}"]), (key, to, name)


def test_golden_alpha_steps_and_tables(oracle, golden):
    thr = golden["alpha_thresholds"].view(np.float32)
    assert thr.size == 255 and np.all(np.diff(thr) > 0)
    at = np.array([oracle.lib.oracle_quant_alpha(float(t)) for t in thr], np.uint8)
    assert np.array_equal(at, golden["alpha_at_threshold"])
    assert np.array_equal(at, np.arange(1, 256, dtype=np.uint8))
    below = np.nextafter(thr, np.float32(-np.inf))
    bl = np.array([oracle.lib.oracle_quant_alpha(float(t)) for t in below], np.uint8)
    assert np.array_equal(bl, golden["alpha_below_threshold"])
    assert np.array_equal(bits(oracle.dequant_table("alpha")), golden["table_alpha"])
    assert np.array_equal(bits(oracle.dequant_table("scale")), golden["table_scale"])
    assert np.array_equal(bits(oracle.dequant_table("color")), golden["table_color"])


# ---- (c) the live reference ------------------------------------------------------------------

@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_live_reference_pack_unpack(oracle, ref, deg):
    rng = np.random.default_rng(100 + deg)
    for special in (False, True):
        c = random_cloud(rng, 1531, deg, special)
        for frm in range(9):
            assert_packed_equal(oracle.pack(c, frm), ref.pack(c, frm), f"deg{deg} from{frm}")
        p = ref.pack(c, 4)
        for to in range(9):
            assert_cloud_bits_equal(oracle.unpack(p, to), ref.unpack(p, to), f"deg{deg} to{to}")


@pytest.mark.parametrize("ver", [1, 2, 3])
def test_live_reference_random_streams(oracle, ref, ver):
    rng = np.random.default_rng(200 + ver)
    for fb in (12, 8, 23):
        s = random_stream(rng, 777, 3, ver, fb)
        for to in (0, 1, 4, 6, 7, 8):
            assert_cloud_bits_equal(oracle.unpack(s, to), ref.unpack(s, to), f"v{ver} fb{fb} to{to}")


def test_live_reference_container_matches_golden(ref, golden):
    c = golden_cloud(golden, "kat_in", 2, 3)
    c.antialiased = True
    assert np.array_equal(np.frombuffer(ref.serialize(c, 0), np.uint8), golden["kat_container"])
    blob = ref.save_spz(c, 0)
    assert len(blob) == 126 and blob[:10] == bytes.fromhex("1f8b0800000000000003")  # SURVEY 8c
    back = ref.load_spz(blob, 0)
    assert back.n == 2 and back.sh_degree == 3 and back.antialiased


def test_empty_and_bad_degree(oracle):
    for deg in range(4):
        e = Cloud(0, deg, *[np.zeros(0, np.float32)] * 6)
        p = oracle.pack(e, 6)
        assert all(a.size == 0 for a in p.planes())
        g = oracle.unpack(p, 8)
        assert all(a.size == 0 for a in g.planes())
    bad = Cloud(1, 4, *[np.zeros(64, np.float32)] * 6)
    with pytest.raises((ValueError, KeyError)):
        oracle.pack(bad, 0)


def test_alpha_quantizer_is_a_monotone_step_function(oracle):
    """The property the device alpha quantizer rests on (SURVEY.md section 7): over ALL floats in
    ascending order the reference's alpha byte never decreases.  Exhaustive over the interval that
    contains every threshold, [-8, 8]; sampled outside (the function is constant there)."""
    from concurrent.futures import ThreadPoolExecutor

    def run(first_bits, count, descending):
        out = oracle.sweep_u8(0, first_bits, 1, count)
        d = np.diff(out.astype(np.int16))
        return (d.max(initial=0) <= 0) if descending else (d.min(initial=0) >= 0), out[0], out[-1]

    # positive floats 0 .. 8.0 ascend with their bit patterns; negative -0 .. -8.0 descend
    hi = int(np.array([8.0], np.float32).view(np.uint32)[0])
    jobs = []
    step = 1 << 26
    for a in range(0, hi + 1, step):
        jobs.append((a, min(step, hi + 1 - a), False))
        jobs.append((0x80000000 + a, min(step, hi + 1 - a), True))
    with ThreadPoolExecutor(8) as ex:
        res = list(ex.map(lambda j: run(*j), jobs))
    assert all(r[0] for r in res)
    # chunk boundaries chain monotonically too
    pos = [r for j, r in zip(jobs, res) if not j[2]]
    assert all(pos[i][2] <= pos[i + 1][1] for i in range(len(pos) - 1))
    neg = [r for j, r in zip(jobs, res) if j[2]]
    assert all(neg[i][2] >= neg[i + 1][1] for i in range(len(neg) - 1))
    assert oracle.lib.oracle_quant_alpha(8.0) == 255 and oracle.lib.oracle_quant_alpha(-8.0) == 0
    assert oracle.lib.oracle_quant_alpha(float("inf")) == 255 and oracle.lib.oracle_quant_alpha(float("-inf")) == 0
    assert oracle.lib.oracle_quant_alpha(3e38) == 255 and oracle.lib.oracle_quant_alpha(-3e38) == 0


def test_unpack_at_restatement_matches_golden(oracle):
    """oracle_unpack_at (PackedGaussians::at + unpack, load-spz.cc:383-463) against vectors the reference made
    (tests/golden/make_golden_unpack_at.py), and against the bulk decoder on the same gaussians."""
    import os
    from util import PLANES, random_stream
    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_unpack_at.npz"))
    convs = G["converters"]
    assert np.array_equal(convs[1], oracle.converter(4, 6))
    for ver in (1, 2, 3, 4):
        for deg in range(4):
            key = f"v{ver}d{deg}"
            s = Packed(64, deg, int(G[f"{key}_fb"]), ver, *[G[f"{key}_{p}"] for p in PLANES])
            for k, conv in enumerate(convs):
                assert np.array_equal(bits(oracle.unpack_at(s, G[f"{key}_idx"], conv)), G[f"{key}_out{k}"]), (key, k)
    rng = np.random.default_rng(77)
    # with +-1 converters the gather equals the bulk decoder (unpackGaussians) on the same gaussians
    s = random_stream(rng, 100, 2, 3)
    s.rotations.view("<u4")[:] &= np.uint32(0xEFFBFEFF)
    full = oracle.unpack(s, 6)  # RUB -> RDF
    rows = oracle.unpack_at(s, np.arange(100), oracle.converter(4, 6))
    assert np.array_equal(bits(rows[:, 0:3].reshape(-1)), bits(full.positions))
    assert np.array_equal(bits(rows[:, 3:7].reshape(-1)), bits(full.rotations))
    assert np.array_equal(bits(rows[:, 14:22]), bits(full.sh.reshape(100, 8, 3)[:, :, 0]))
    assert np.all(rows[:, 22:29] == 0)  # coefficients the stream does not carry decode from the pad byte 128
    with pytest.raises(ValueError):
        oracle.unpack_at(s, [100], convs[0])


def test_unpack_at_restatement_matches_golden_and_live_reference(oracle, ref):
    """oracle_unpack_at against the reference library itself on fresh streams (the stored vectors are checked by
    test_unpack_at_restatement_matches_golden)."""
    from util import random_stream
    rng = np.random.default_rng(77)
    for ver in (1, 2, 3, 4):
        for deg in (0, 1, 3):
            s = random_stream(rng, 300, deg, ver, int(rng.integers(0, 40)))
            idx = rng.integers(0, 300, 500)
            conv = (rng.normal(size=21) * 2).astype(np.float32)
            assert np.array_equal(bits(oracle.unpack_at(s, idx, conv)), bits(ref.unpack_at(s, idx, conv))), (ver, deg)
