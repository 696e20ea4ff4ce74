"""CPU tier: the rd_update stages the shipped configuration leaves off — bufscale (render.c:1765-1790),
transform_smooth (render.c:694-718), keyframe interpolation (render.c:1792-1809, 2347-2353) — in the oracle,
pinned against the reference's compiled code where the reference has code to compile (transform_smooth)."""
import os

import numpy as np
import pytest

import glava_b200 as g
from oracle.oracle import OracleStream, ext_from, params_from
from tests.conftest import GOLDEN
from tests.reference_record import same


def test_transform_smooth_golden(orc):
    z = np.load(os.path.join(GOLDEN, "smooth.npz"))
    for n in (1024, 4096):
        for name, (d, ratio) in (("default", (0.01, 4.0)), ("wide", (0.2, 2.0))):
            got = orc.transform_smooth(z[f"in_{n}"], d, ratio)
            assert np.array_equal(got, z[f"out_{n}_{name}"], equal_nan=True), (n, name)
            assert np.isnan(got[0]) and not np.isnan(got[1:]).any()        # log(0): empty window, 0/0


@pytest.mark.parametrize("n", [256, 2048, 16384])
def test_transform_smooth_live_reference_bit_exact(orc, ref, n):
    rng = np.random.default_rng(n)
    for d, ratio in ((0.01, 4.0), (0.05, 3.0), (0.3, 1.0)):
        x = (rng.random(n) ** 2).astype(np.float32); x[rng.random(n) < 0.3] = 0
        assert same(orc.transform_smooth(x, d, ratio), ref.smooth(x, d, ratio), equal_nan=True)
    silent = np.zeros(n, np.float32)                                         # every window empty: NaN over the head
    a, b = orc.transform_smooth(silent), ref.smooth(silent)
    assert same(a, b, equal_nan=True) and np.isnan(a[: n // 4]).all() and not np.isnan(a[n // 4:]).any()


def test_bufscale_is_a_sequential_float_mean(orc):
    rng = np.random.default_rng(3)
    x = ((rng.random(4096) - 0.5) * 0.9).astype(np.float32)
    for k in (2, 4, 8):
        want = np.zeros(4096 // k, np.float32)
        for a in range(k):
            want = (want + x[a::k]).astype(np.float32)
        want = (want / np.float32(k)).astype(np.float32)
        assert np.array_equal(orc.bufscale(x, k), want)


def test_interp_formula(orc):
    rng = np.random.default_rng(4)
    s = rng.random(512).astype(np.float32); e = rng.random(512).astype(np.float32)
    ur, fr = np.float32(86.1328125), np.float32(240.0)
    for k in (0, 1, 2, 3, 7):
        mod = min(np.float32(ur / fr) * np.float32(k), np.float32(1.0))
        want = (s + ((e - s) * mod).astype(np.float32)).astype(np.float32)
        assert np.array_equal(orc.interp(s, e, ur, fr, k), want)
    assert np.array_equal(orc.interp(s, e, ur, fr, 0), s) and np.allclose(orc.interp(s, e, ur, fr, 3), e, atol=1e-6)   # s + (e - s) rounds


def _pcm(n, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(n, dtype=np.float32)
    return (0.05 * np.sin(t * 0.07 * (seed + 1)) + 0.01 * rng.standard_normal(n)).astype(np.float32)


def test_stream_interpolation_shows_an_update_one_update_late(orc):
    """pipeline A, fr = 4 ur: every frame shows the lerp of the two keyframes pushed by PREVIOUS modified updates
    (render.c:1792-1809, 2347-2353): the output runs one update late (rc.glsl:129-130)."""
    p = orc.default_params("bars", n=1024, accel_fft=0, smooth_pass=0)
    x = ext_from(interpolate=1, fr=p.ur * 4)
    st = OracleStream(orc, p, x)
    plain = OracleStream(orc, p, ext_from())
    specs, texs = [], []
    for u in range(4):
        lb, rb = _pcm(1024, u), _pcm(1024, 10 + u)
        specs.append(plain.update(lb, rb, True)[0])
        frames = [st.update(lb, rb, True)[2]] + [st.update(lb, rb, False)[2] for _ in range(3)]
        texs.append(frames)
    q = lambda v: np.where(v > 0, np.where(v < 1, np.rint((v * np.float32(65535.0)).astype(np.float32)).astype(np.int64), 65535), 0).astype(np.uint16)
    # kcounter is reset AFTER a modified frame (render.c:2380-2383), so with 3 sub-frames per update the modifier runs
    # 0, 1/4, 2/4 on the sub-frames and 3/4 on the next modified frame, whose lerp still uses the old keyframes
    zero = np.zeros(1024, np.float32)
    key = lambda u: specs[u] if u >= 0 else zero
    fr = p.ur * 4
    for u in range(4):
        if u >= 1:
            assert np.array_equal(texs[u][0], q(orc.interp(key(u - 2), key(u - 1), p.ur, fr, 3))), u
        for j in (1, 2, 3):
            assert np.array_equal(texs[u][j], q(orc.interp(key(u - 1), key(u), p.ur, fr, j - 1))), (u, j)
    assert np.array_equal(texs[2][1], q(specs[1]))          # modifier 0: exactly the previous update's spectrum


def test_stream_interpolation_is_forced_off(orc):
    lb, rb = _pcm(1024, 1), _pcm(1024, 2)
    # update rate close to the frame rate (render.c:1761-1763)
    p = orc.default_params("bars", n=1024, accel_fft=0)
    a, b = OracleStream(orc, p, ext_from(interpolate=1, fr=p.ur)), OracleStream(orc, p, ext_from())
    for _ in range(3):
        assert np.array_equal(a.update(lb, rb, True)[2], b.update(lb, rb, True)[2])
    # fft chain pushed to the GL passes (render.c:2161-2168)
    p = orc.default_params("bars", n=1024, accel_fft=1)
    a, b = OracleStream(orc, p, ext_from(interpolate=1, fr=p.ur * 4)), OracleStream(orc, p, ext_from())
    for _ in range(3):
        assert np.array_equal(a.update(lb, rb, True)[2], b.update(lb, rb, True)[2])
    # ... but `wave` has no fft transform: interpolation stays on even under setaccelfft
    p = orc.default_params("wave", n=1024, accel_fft=1)
    a, b = OracleStream(orc, p, ext_from(interpolate=1, fr=p.ur * 4)), OracleStream(orc, p, ext_from())
    a.update(lb, rb, True); b.update(lb, rb, True)
    assert not np.array_equal(a.update(lb, rb, True)[2], b.update(lb, rb, True)[2])


def test_stream_transform_smooth_forces_the_cpu_chain(orc):
    """a transform after "fft" under setaccelfft: the bind runs fft + gravity + average on the CPU (render.c:2143-2154)"""
    lb, rb = _pcm(1024, 5), _pcm(1024, 6)
    pa = orc.default_params("bars", n=1024, accel_fft=0)
    pb = orc.default_params("bars", n=1024, accel_fft=1)
    x = ext_from(transform_smooth=1)
    a, b, plain = OracleStream(orc, pa, x), OracleStream(orc, pb, x), OracleStream(orc, pa, ext_from())
    for _ in range(3):
        ra, rb_, rp = a.update(lb, rb, True), b.update(lb, rb, True), plain.update(lb, rb, True)
    assert np.array_equal(ra[0], rb_[0], equal_nan=True) and np.array_equal(ra[2], rb_[2])
    assert np.array_equal(ra[0], orc.transform_smooth(rp[0]), equal_nan=True)
    assert ra[0].shape == (1024,) and np.isnan(ra[0][0])


def test_stream_bufscale_shrinks_the_textures(orc):
    p = orc.default_params("bars", n=2048)
    st = OracleStream(orc, p, ext_from(bufscale=2))
    p2 = orc.default_params("bars", n=1024)
    half = OracleStream(orc, p2, ext_from())
    lb, rb = _pcm(2048, 7), _pcm(2048, 8)
    got = st.update(lb, rb, True)
    want = half.update(orc.bufscale(lb, 2), orc.bufscale(rb, 2), True)
    assert st.n == 1024 and all(np.array_equal(x, y) for x, y in zip(got, want))


# ---- config surface ------------------------------------------------------------------------------------
def test_requests_reach_the_parameters(built):
    p = g.load_config(requests=["setbufscale 2", "setinterpolate true", "setsmooth 0.05", "setsmoothratio 3",
                                "setframerate 240", 'transform audio_l "smooth"', 'transform audio_l "fft"'])
    assert (p.bufscale, p.interpolate, p.transform_smooth) == (2, 1, 1)
    assert abs(p.smooth_distance - 0.05) < 1e-7 and p.smooth_ratio == 3.0 and p.fr == 240.0
    d = g.load_config()
    assert (d.bufscale, d.interpolate, d.transform_smooth, d.fr) == (1, 0, 0, 0.0)          # rc.glsl:131,236
    assert abs(d.smooth_distance - 0.01) < 1e-9 and d.smooth_ratio == 4.0                     # render.c:917-918
    x = ext_from(p)
    assert (x.bufscale, x.interpolate, x.transform_smooth, x.fr) == (2, 1, 1, 240.0)
    assert params_from(p).n == p.n


def test_unknown_transform_is_an_error(built):
    with pytest.raises(g.GlavaError, match="transform function does not exist"):
        g.load_config(requests=['transform audio_l "bogus"'])


def test_bad_bufscale_is_rejected_without_a_gpu(built):
    import ctypes as C
    L = g.api.lib()
    p = g.default_params("bars", n=1024, bufscale=8)            # 1024 / 8 = 128 < 256
    assert not L.glava_b200_new(C.byref(p), 1, 0)
    assert b"setbufscale" in L.glava_b200_last_error()
