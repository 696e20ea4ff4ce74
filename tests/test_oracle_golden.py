"""The oracle is pinned here: against golden vectors generated from the reference's own compiled
render.c (tests/golden/make_golden.py) and against it on fresh input: live where oracle/_ref is built, its recorded
results elsewhere (tests/reference_record.py)."""
import os

import numpy as np
import pytest

from tests.conftest import GOLDEN
from tests.reference_record import same
from glava_b200.synth import fifo_to_float

HOP = 256


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _replay(n, chunks):
    ring = np.zeros(n, np.float32)
    for c in chunks:
        l, _ = fifo_to_float(c)
        ring = np.concatenate([ring[HOP:], l])
        yield ring


@pytest.mark.parametrize("n", [512, 1024, 4096])
def test_pipeline_a_matches_reference_golden(orc, n):
    from oracle.oracle import OracleChannel
    gold = np.load(os.path.join(GOLDEN, f"spectrum_a_n{n}.npz"))
    p = orc.default_params("bars", n=n, accel_fft=0, smooth_pass=0, ur=float(gold["ur"]))
    ch = OracleChannel(orc, p)
    for u, ring in enumerate(_replay(n, gold["chunks"]), start=1):
        spec, tex = ch.update(ring)
        if u in (1, 6, 12):
            assert np.array_equal(_bits(spec), _bits(gold[f"out_{u}"])), f"update {u}"
        if u == 12:
            assert np.array_equal(_bits(orc.fft_f32(p, ring)), _bits(gold["raw_fft_12"]))
            # texture = GL_R16 upload of the float result (render.c:521-524)
            want = np.rint((np.clip(spec, 0, 1).astype(np.float32) * np.float32(65535)).astype(np.float32))
            assert np.array_equal(tex, want.astype(np.uint16))


def test_fft_known_answers(orc):
    gold = np.load(os.path.join(GOLDEN, "fft_kat.npz"))
    p = orc.default_params("bars", n=1024)
    for k in ("sine", "impulse"):
        assert np.array_equal(_bits(orc.fft_f32(p, gold[k])), _bits(gold[k + "_out"]))
    # SURVEY fact 3: N real samples = N/2 interleaved complex; a 64-cycle sine peaks at complex
    # bins 64 and 448 -> float indices 128/129 and 896/897
    out = gold["sine_out"]
    assert int(out.argmax()) in (896, 897)                 # the index ramp favours the upper image
    assert int(out[:512].argmax()) in (128, 129)


def test_window_is_phase_shifted_hamming(orc):
    # SURVEY fact 4: window(i, sz - 1) expands to cos(TWOPI*i/sz - 1)
    n = 1024
    w = orc.window(n)
    i = np.arange(n)
    assert np.allclose(w, 0.53836 - 0.46164 * np.cos(6.28318530718 * i / n - 1), atol=1e-15)
    intended = 0.53836 - 0.46164 * np.cos(6.28318530718 * i / (n - 1))
    assert np.abs(w - intended).max() > 0.3


def test_f64_restatement_tracks_reference(orc):
    # the float64 "truth" companion: reference's own float32 recurrence is ~7e-6 of peak away at N=4096
    gold = np.load(os.path.join(GOLDEN, "spectrum_a_n4096.npz"))
    p = orc.default_params("bars", n=4096)
    ring = list(_replay(4096, gold["chunks"]))[-1]
    d = orc.fft_f64(p, ring)
    ref = gold["raw_fft_12"].astype(np.float64)
    assert np.abs(d - ref).max() / ref.max() < 2e-5


def test_wrange_golden(orc):
    from oracle.oracle import OracleChannel
    gold = np.load(os.path.join(GOLDEN, "wrange.npz"))
    p = orc.default_params("wave", n=1024, smooth_pass=0)
    spec, tex = OracleChannel(orc, p).update(gold["ramp"], is_fft=False)
    assert np.array_equal(_bits(spec), _bits(gold["out"]))


def test_live_reference_bit_exact(orc, ref):
    """restatement vs the reference's compiled transforms on fresh random input, several sizes"""
    from oracle.oracle import OracleChannel
    rng = np.random.default_rng(123)
    for n in (256, 512, 2048, 8192, 16384):
        for avg_window in (1, 0):
            p = orc.default_params("bars", n=n, accel_fft=0, smooth_pass=0, avg_window=avg_window, avg_frames=4)
            rc = ref.chan(p)
            oc = OracleChannel(orc, p)
            for _ in range(6):
                x = (rng.standard_normal(n) * 0.15).astype(np.float32)
                spec, _ = oc.update(x)
                assert same(spec, ref.update_a(rc, x)), (n, avg_window)


def test_gravity_decays_monotonically(orc):
    from oracle.oracle import OracleChannel
    n = 512
    p = orc.default_params("bars", n=n, accel_fft=0, smooth_pass=0, avg_frames=1, avg_window=0)
    ch = OracleChannel(orc, p)
    loud = (np.sin(np.arange(n) * 0.3) * 0.4).astype(np.float32)
    first, _ = ch.update(loud)
    prev = first
    g = np.float32(p.gravity_step) * (np.float32(1.0) / np.float32(p.ur))
    for _ in range(5):
        cur, _ = ch.update(np.zeros(n, np.float32))     # silence: fft output 0 -> pure decay
        assert np.all(cur <= prev + 1e-7)
        falling = prev > 2 * g                            # below that the max() with the input (0) takes over
        assert np.allclose((prev - cur)[falling], g, atol=1e-6)
        assert np.all(cur[~falling] >= -g - 1e-7)
        prev = cur


def test_live_reference_bit_exact_random_parameters(orc, ref):
    """the same, over random setfftscale / setfftcutoff / setgravitystep / ur / setavgframes / setavgwindow and input
    regimes (silence, clipping-level, tiny, a DC offset, an impulse): 40 parameter sets x 7 updates, bit for bit"""
    from oracle.oracle import OracleChannel
    rng = np.random.default_rng(2026)
    for trial in range(40):
        n = int(rng.choice([256, 512, 1024, 4096]))
        p = orc.default_params("bars", n=n, accel_fft=0, smooth_pass=0, avg_window=int(rng.integers(0, 2)),
                               avg_frames=int(rng.integers(1, 9)), fft_scale=float(rng.uniform(0.5, 20)),
                               fft_cutoff=float(rng.uniform(0.0, 1.2)), gravity_step=float(rng.uniform(0.0, 12)),
                               ur=float(rng.uniform(20, 250)))
        rc = ref.chan(p)
        oc = OracleChannel(orc, p)
        for k in range(7):
            regime = int(rng.integers(0, 6))
            x = (rng.standard_normal(n) * [0.15, 0.5, 1e-6, 0.0, 0.05, 0.0][regime]).astype(np.float32)
            if regime == 4:
                x += np.float32(0.3)
            if regime == 5:
                x[int(rng.integers(0, n))] = np.float32(0.5)
            spec, _ = oc.update(x)
            assert same(spec, ref.update_a(rc, x)), (trial, n, k, regime)
