"""-m gpu: the fused spectrum kernel through the C ABI against the oracle / reference golden vectors."""
import os

import numpy as np
import pytest

import glava_b200 as g
from glava_b200.synth import fifo_to_float
from oracle.oracle import OracleChannel, params_from
from tests.conftest import GOLDEN

pytestmark = pytest.mark.gpu
HOP = 256


def _peak_err(got, want):
    want = np.asarray(want, dtype=np.float64)
    return np.abs(np.asarray(got, dtype=np.float64) - want).max() / max(np.abs(want).max(), 1e-30)


@pytest.mark.parametrize("n", [512, 1024, 4096])
def test_config1_pipeline_a_vs_reference_golden(n, built):
    """BASELINE configs[0]: single stream, Hann(sic)+FFT+|X|+gravity(+avg) via render.c's CPU transform.
    Golden = the reference's own compiled render.c (tests/golden/make_golden.py).  Tolerance: 1e-5 of peak."""
    gold = np.load(os.path.join(GOLDEN, f"spectrum_a_n{n}.npz"))
    p = g.default_params("bars", n=n, w=64, h=16, accel_fft=0, smooth_pass=0)
    ring = np.zeros((1, n), np.float32)
    with g.Renderer(p, batch=1) as r:
        for u, c in enumerate(gold["chunks"], start=1):
            l, _ = fifo_to_float(c)
            ring[0] = np.concatenate([ring[0, HOP:], l])
            r.update(ring, ring, True)
            if u in (1, 6, 12):
                sl, sr = r.spectrum()
                assert _peak_err(sl[0], gold[f"out_{u}"]) <= 1e-5, (n, u)
                assert np.array_equal(sl, sr)


@pytest.mark.parametrize("n", [256, 512, 1024, 2048, 4096, 8192, 16384])
@pytest.mark.parametrize("accel", [0, 1])
def test_all_sizes_both_pipelines(orc_pm, n, accel, built):
    batch = 3
    p = g.default_params("bars", n=n, w=64, h=16, accel_fft=accel); op = params_from(p)
    rings = g.StreamRings(batch, n)
    chans = [[OracleChannel(orc_pm, op), OracleChannel(orc_pm, op)] for _ in range(batch)]
    with g.Renderer(p, batch=batch) as r:
        for _ in range(9):
            rings.advance()
            r.update(rings.lb, rings.rb, True)
            want = [[chans[s][0].update(rings.lb[s]), chans[s][1].update(rings.rb[s])] for s in range(batch)]
        sl, sr = r.spectrum(); tl, tr = r.textures()
    tol = 1e-5 if n <= 4096 else 2.5e-5           # reference's own float recurrence error above 4096 (SURVEY §7)
    for s in range(batch):
        for got, gtex, (spec, tex) in ((sl[s], tl[s], want[s][0]), (sr[s], tr[s], want[s][1])):
            assert _peak_err(got, spec) <= tol, (n, accel, s)
            assert np.abs(gtex.astype(int) - tex.astype(int)).max() <= 2, (n, accel, s)     # R16 texels, 2 LSB16 = 3e-5
    if accel:   # accel returns the raw transform_fft output: also compare with exact (float64) arithmetic
        d = orc_pm.fft_f64(op, rings.lb[0])
        assert _peak_err(sl[0], d) <= 2e-6


def test_avg_frame_variants(orc_pm, built):
    for F, win in ((1, 1), (2, 1), (3, 1), (6, 0), (16, 1)):
        for accel in (0, 1):
            n = 1024
            p = g.default_params("bars", n=n, w=64, h=16, accel_fft=accel, avg_frames=F, avg_window=win); op = params_from(p)
            rings = g.StreamRings(1, n, first_stream=5)
            oc = OracleChannel(orc_pm, op)
            with g.Renderer(p, batch=1) as r:
                for _ in range(F + 3):
                    rings.advance(); r.update(rings.lb, rings.rb, True); spec, tex = oc.update(rings.lb[0])
                sl, _ = r.spectrum(); tl, _ = r.textures()
            assert _peak_err(sl[0], spec) <= 1e-5, (F, win, accel)
            assert np.abs(tl[0].astype(int) - tex.astype(int)).max() <= 2, (F, win, accel)


@pytest.mark.parametrize("mode,formula", [(0, 0), (1, 0), (2, 0), (0, 1), (0, 2)])
def test_smooth_pass_kernel_bit_exact(orc_pm, mode, formula, built):
    n = 4096
    p = g.default_params("bars", n=n, w=64, h=16, sample_mode=mode, round_formula=formula); op = params_from(p)
    rng = np.random.default_rng(7)
    tex = (rng.random((6, n)) ** 2 * 65535).astype(np.uint16)
    tex[4] = 0; tex[5] = 65535
    with g.Renderer(p, batch=1) as r:
        got = r.smooth_pass(tex)
    for i in range(tex.shape[0]):
        assert np.array_equal(got[i], orc_pm.smooth_pass(op, tex[i])), i


def test_wave_chain_bit_exact(orc_pm, built):
    n, batch = 2048, 2
    p = g.default_params("wave", n=n, w=64, h=16); op = params_from(p)
    rings = g.StreamRings(batch, n)
    with g.Renderer(p, batch=batch) as r:
        for _ in range(9):
            rings.advance()
        r.update(rings.lb, None, True)
        sl, _ = r.spectrum(); tl, _ = r.textures()
    for s in range(batch):
        spec, tex = OracleChannel(orc_pm, op).update(rings.lb[s], is_fft=False)
        assert np.array_equal(sl[s], spec) and np.array_equal(tl[s], tex)


def test_streams_are_independent_and_deterministic(built):
    """size-independent property at the headline size: stream s of a big batch == the same stream alone"""
    n, batch = 4096, 64
    p = g.default_params("bars", n=n, w=64, h=16)
    rings = g.StreamRings(batch, n)
    hist = []
    with g.Renderer(p, batch=batch) as r:
        for _ in range(7):
            rings.advance(); hist.append((rings.lb.copy(), rings.rb.copy()))
            r.update(rings.lb, rings.rb, True)
        sl, sr = r.spectrum(); tl, tr = r.textures()
    for s in (0, 17, 63):
        with g.Renderer(p, batch=1) as r1:
            for lb, rb in hist:
                r1.update(lb[s:s + 1], rb[s:s + 1], True)
            a, b = r1.spectrum(); c, d = r1.textures()
        assert np.array_equal(a[0], sl[s]) and np.array_equal(b[0], sr[s])
        assert np.array_equal(c[0], tl[s]) and np.array_equal(d[0], tr[s])


def test_silence_and_gravity_decay(built):
    n = 1024
    p = g.default_params("bars", n=n, w=64, h=16, accel_fft=0, avg_frames=1, avg_window=0, smooth_pass=0)
    loud = (np.sin(np.arange(n) * 0.3) * 0.4).astype(np.float32)[None, :]
    zero = np.zeros((1, n), np.float32)
    gstep = np.float32(p.gravity_step) * (np.float32(1.0) / np.float32(p.ur))
    with g.Renderer(p, batch=1) as r:
        r.update(loud, loud, True); prev, _ = r.spectrum()
        for _ in range(4):
            r.update(zero, zero, True); cur, _ = r.spectrum()
            falling = prev[0] > 2 * gstep
            assert np.allclose((prev[0] - cur[0])[falling], gstep, atol=1e-6)
            prev = cur


def test_fifo_ingest_matches_fifo_c(orc_pm, built):
    n, batch, hop = 1024, 3, 256
    for channels in (2, 1):
        p = g.default_params("bars", n=n, w=64, h=16, channels=channels)
        rl = np.zeros((batch, n), np.float32); rr = np.zeros((batch, n), np.float32)
        rng = np.random.default_rng(3)
        with g.Renderer(p, batch=batch) as r, g.Renderer(p, batch=batch) as r2:
            for _ in range(6):
                chunks = rng.integers(-32768, 32767, size=(batch, hop * 2), dtype=np.int16)
                for s in range(batch):
                    orc_pm.fifo_ingest(rl[s], rr[s], chunks[s], channels)
                r.ingest_fifo(chunks)
            r.update_rings(True)
            r2.update(rl, rr, True)
            a = r.spectrum(); b = r2.spectrum()
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_bad_arguments_fail_loudly(built):
    p = g.default_params("bars", n=1024, w=64, h=16)
    with g.Renderer(p, batch=2) as r:
        with pytest.raises(AssertionError):
            r.update(np.zeros((2, 512), np.float32), None, True)
        rc = r._L.glava_b200_update(r._h, np.zeros((2, 512), np.float32).ctypes.data, None, 512, 1)
        assert rc != 0 and b"bsz" in r._L.glava_b200_last_error()
    with pytest.raises(g.GlavaError):
        g.Renderer(g.default_params("bars", n=1000), batch=1)


@pytest.mark.parametrize("n,w", [(1024, 320), (4096, 1920), (8192, 1920), (16384, 1920)])
def test_kernel_variants_give_identical_textures_and_frames(built, monkeypatch, n, w):
    """the spectrum path exists in several launch structures (tuning knobs, DESIGN 6.2): plane-per-CTA kernel with in-kernel
    epilogue and K5; K5 as its own kernel over (texel, stream) pairs (through L2, or out of shared-memory tiles); the R16 state
    update as an elementwise kernel; FFT passes in place / out of place, 128 / 256 threads.  All of them are the same arithmetic: textures and frames must be identical."""
    batch = 70                                                    # not a multiple of 32: partial stream groups in k5_need_kernel
    p = g.default_params("bars", n=n, w=w, h=32, lazy_smooth=1)
    rng = np.random.default_rng(n)
    seq = [((rng.random((batch, n), np.float32) - 0.5) * 0.4, (rng.random((batch, n), np.float32) - 0.5) * 0.4) for _ in range(7)]
    masks = [None, None, rng.random(batch) < 0.5, None, rng.random(batch) < 0.5, None, None]

    def run(env):
        for k in ("GLAVA_B200_K5_SPLIT", "GLAVA_B200_SPLIT_EPI", "GLAVA_B200_SPEC_OOP", "GLAVA_B200_SPEC_T", "GLAVA_B200_K5N_SMEM",
                  "GLAVA_B200_K5N_ROWS", "GLAVA_B200_K5N_TPB", "GLAVA_B200_K5N_WARPS", "GLAVA_B200_K5N_S", "GLAVA_B200_SPEC_CTAS_PER_SM"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        with g.Renderer(p, batch=batch) as r:
            for (lb, rb), m in zip(seq, masks):
                if m is None:
                    r.update(lb, rb, True)
                else:
                    r.update_masked(lb, rb, m)
            tl, tr = r.textures()
            need = tl.any(axis=0) | tr.any(axis=0)                 # lazy: only the sampled texels are defined
            return tl[:, need], tr[:, need], [r.readback(s) for s in (0, 33, batch - 1)], r.spectrum()

    base = run({"GLAVA_B200_K5_SPLIT": "0", "GLAVA_B200_SPEC_OOP": "0", "GLAVA_B200_SPEC_T": "0"})
    assert base[0].any()
    for env in ({"GLAVA_B200_K5_SPLIT": "1", "GLAVA_B200_SPLIT_EPI": "0"}, {"GLAVA_B200_K5_SPLIT": "1", "GLAVA_B200_SPLIT_EPI": "1"},
                {"GLAVA_B200_K5_SPLIT": "1", "GLAVA_B200_SPLIT_EPI": "1", "GLAVA_B200_SPEC_OOP": "1", "GLAVA_B200_SPEC_T": "256"},
                {"GLAVA_B200_K5_SPLIT": "0", "GLAVA_B200_SPEC_OOP": "1", "GLAVA_B200_SPEC_T": "128"},
                # K5 over (texel, stream) pairs: through L2 from a transposed copy / out of shared-memory tiles over blocks of texels
                {"GLAVA_B200_K5_SPLIT": "1", "GLAVA_B200_K5N_SMEM": "0"},
                {"GLAVA_B200_K5_SPLIT": "1", "GLAVA_B200_K5N_SMEM": "0", "GLAVA_B200_K5N_S": "4"},     # (4 streams per lane: only through the knob)
                {"GLAVA_B200_K5_SPLIT": "1", "GLAVA_B200_K5N_SMEM": "1"},
                {"GLAVA_B200_K5_SPLIT": "1", "GLAVA_B200_K5N_SMEM": "1", "GLAVA_B200_K5N_ROWS": "64", "GLAVA_B200_K5N_TPB": "3", "GLAVA_B200_K5N_WARPS": "2"},
                {}):                                                                                             # {} = this size's defaults
        got = run(env)
        assert np.array_equal(got[0], base[0]) and np.array_equal(got[1], base[1]), env
        for a, b in zip(got[2], base[2]):
            assert np.array_equal(a, b), env
        if env.get("GLAVA_B200_SPLIT_EPI") == "0":                 # (the three-kernel form writes only the bins that matter into `spec`)
            bad = np.argwhere(got[3][0] != base[3][0])
            assert len(bad) == 0, (env, len(bad), bad[:5].tolist(), got[3][0][tuple(bad[0])], base[3][0][tuple(bad[0])])
