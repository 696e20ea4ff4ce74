"""CPU tier: the product's kernel maths (glava_b200/csrc/*_core.h, compiled for the host by
tests/emul) against the oracle.  Same checks the -m gpu tests make through the C ABI, so that
arithmetic bugs are caught before GPU time is spent."""
import numpy as np
import pytest

import glava_b200 as g
from oracle.oracle import OracleChannel, params_from
from tests.reference_record import same
from tests import emul


def _tex(n, seed):
    return (np.random.default_rng(seed).random(n) ** 2 * 65535).astype(np.uint16)


@pytest.mark.parametrize("n", [256, 512, 1024, 2048, 4096, 8192, 16384])
def test_stockham_fft_vs_reference_restatement(orc_pm, n, built):
    p = g.default_params("bars", n=n); op = params_from(p)
    x = (np.random.default_rng(n).standard_normal(n) * 0.2).astype(np.float32)
    got = emul.fft(x)
    f32 = orc_pm.fft_f32(op, x); f64 = orc_pm.fft_f64(op, x)
    # north_star tolerance: 1e-5 of peak against render.c's transform.  The reference's own float
    # twiddle recurrence is 1.2e-5 / 1.6e-5 away from exact arithmetic at N = 8192 / 16384 (SURVEY §7),
    # so above 4096 the bar is 1e-5 against the float64 evaluation and 2.5e-5 against the float32 one.
    assert np.abs(got - f64).max() / f64.max() <= 2e-6
    assert np.abs(got - f32).max() / f32.max() <= (1e-5 if n <= 4096 else 2.5e-5)


@pytest.mark.parametrize("accel", [0, 1])
@pytest.mark.parametrize("n", [1024, 4096])
def test_update_chain(orc_pm, accel, n, built):
    p = g.default_params("bars", n=n, accel_fft=accel); op = params_from(p)
    rings = g.StreamRings(1, n)
    oc = OracleChannel(orc_pm, op); ec = emul.Channel(p)
    for _ in range(n // 256 + 7):
        rings.advance()
        s0, t0 = oc.update(rings.lb[0]); s1, t1 = ec.update(rings.lb[0])
    assert np.abs(s0 - s1).max() / np.abs(s0).max() <= 1e-5
    assert np.abs(t0.astype(int) - t1.astype(int)).max() <= 2          # R16 texels: <= 2 LSB16 (3e-5)


@pytest.mark.parametrize("mode,formula", [(0, 0), (1, 0), (2, 0), (0, 1), (0, 2)])
def test_smooth_pass_bit_exact(orc_pm, mode, formula, built):
    n = 2048
    p = g.default_params("bars", n=n, sample_mode=mode, round_formula=formula); op = params_from(p)
    tex = _tex(n, 5)
    assert np.array_equal(orc_pm.smooth_pass(op, tex), emul.smooth(p, tex))


def test_wave_chain_bit_exact(orc_pm, built):
    n = 2048
    p = g.default_params("wave", n=n); op = params_from(p)
    x = (np.random.default_rng(1).standard_normal(n) * 0.2).astype(np.float32)
    s0, t0 = OracleChannel(orc_pm, op).update(x, is_fft=False)
    s1, t1 = emul.Channel(p).update(x, is_fft=False)
    assert np.array_equal(s0, s1) and np.array_equal(t0, t1)


@pytest.mark.parametrize("module", g.MODULES)
@pytest.mark.parametrize("w,h", [(640, 360), (333, 97)])
def test_raster_bit_exact(orc_pm, module, w, h, built):
    n = 2048
    p = g.default_params(module, n=n, w=w, h=h); op = params_from(p)
    tl = orc_pm.smooth_pass(op, _tex(n, 1)); tr = orc_pm.smooth_pass(op, _tex(n, 2))
    want = orc_pm.raster(op, tl, tr)
    assert np.array_equal(want, emul.raster(p, tl, tr))
    if module in ("bars", "graph", "wave", "circle"):
        assert np.array_equal(want, emul.raster(p, tl, tr, fast=True))      # hoisted evaluation of the kernels


@pytest.mark.parametrize("over", [dict(bars_direction=1), dict(bars_invert=1), dict(bars_flip=1), dict(bars_mirror_yx=1),
                                  dict(channels=1), dict(channels=1, bars_invert=1), dict(bars_outline_width=0.0),
                                  dict(bars_outline_mode=1), dict(bars_width=3.0, bars_gap=2.0), dict(smooth_pass=0)])
def test_bars_options(orc_pm, over, built):
    n = 1024
    p = g.default_params("bars", n=n, w=320, h=200, **over)
    if over.get("bars_outline_mode") == 1:
        p.bars_outline[0], p.bars_outline[1], p.bars_outline[2], p.bars_outline[3] = 0.9, 0.1, 0.2, 1.0
    op = params_from(p)
    tl, tr = _tex(n, 3), _tex(n, 4)
    want = orc_pm.raster(op, tl, tr)
    assert np.array_equal(want, emul.raster(p, tl, tr))
    if not over.get("bars_mirror_yx"):
        assert np.array_equal(want, emul.raster(p, tl, tr, fast=True))


@pytest.mark.parametrize("module,over", [("radial", dict(radial_invert=1)), ("radial", dict(premultiply_alpha=0)),
                                         ("circle", dict(circle_fill=1)), ("circle", dict(circle_smooth=0)),
                                         ("circle", dict(circle_invert=1)), ("graph", dict(graph_direction=-1)),
                                         ("graph", dict(graph_invert=1)), ("graph", dict(graph_draw_outline=1)),
                                         ("graph", dict(graph_draw_highlight=0))])
def test_module_options(orc_pm, module, over, built):
    n = 1024
    p = g.default_params(module, n=n, w=400, h=300, **over); op = params_from(p)
    tl, tr = _tex(n, 6), _tex(n, 7)
    assert np.array_equal(orc_pm.raster(op, tl, tr), emul.raster(p, tl, tr))


def test_unorm_fetch_is_exact_division(built):
    """from8 / from16 use reciprocal + fma correction instead of a divide: must equal u / MAX for every u"""
    assert emul.lib().emul_unorm_fetch_mismatches() == 0


# ---- optional rd_update stages: the product's chain_core.h arithmetic on the host against the oracle -------------
def test_chain_core_bufscale_and_transform_smooth_bit_exact(orc, built):
    from tests import emul
    rng = np.random.default_rng(11)
    for n in (256, 4096, 16384):
        x = ((rng.random(n) - 0.5) * 0.9).astype(np.float32)
        for k in (2, 4, 8):
            assert np.array_equal(emul.bufscale(x, k), orc.bufscale(x, k))
        y = (rng.random(n) ** 3).astype(np.float32); y[rng.random(n) < 0.25] = 0
        for d, ratio in ((0.01, 4.0), (0.2, 2.0), (0.3, 1.0)):
            assert np.array_equal(emul.transform_smooth(y, d, ratio), orc.transform_smooth(y, d, ratio), equal_nan=True)
        z = np.zeros(n, np.float32)
        assert np.array_equal(emul.transform_smooth(z), orc.transform_smooth(z), equal_nan=True)


def test_chain_core_transform_smooth_vs_compiled_reference(ref, built):
    from tests import emul
    rng = np.random.default_rng(12)
    y = (rng.random(2048) ** 2).astype(np.float32); y[rng.random(2048) < 0.3] = 0
    assert same(emul.transform_smooth(y, 0.05, 3.0), ref.smooth(y, 0.05, 3.0), equal_nan=True)


def test_chain_core_keyframe_upload_bit_exact(orc, built):
    from tests import emul
    rng = np.random.default_rng(13)
    s = (rng.random(1024) * 1.2 - 0.1).astype(np.float32); e = (rng.random(1024) * 1.2 - 0.1).astype(np.float32)
    s[5] = np.nan
    q = lambda v: np.where(v > 0, np.where(v < 1, np.rint((v * np.float32(65535.0)).astype(np.float32)).astype(np.int64), 65535), 0).astype(np.uint16)
    ur, fr = np.float32(86.1328125), np.float32(240.0)
    for k in (0, 1, 2, 5):
        with np.errstate(invalid="ignore"):
            assert np.array_equal(emul.upload(s, e, ur, fr, k), q(orc.interp(s, e, ur, fr, k)))
    with np.errstate(invalid="ignore"):
        assert np.array_equal(emul.upload(s, None, ur, fr, 0), q(s)) and emul.upload(s, None, ur, fr, 0)[5] == 0   # NaN -> 0


# ---- K5 from the precomputed tables (glava_b200/csrc/tables.h), walked as the kernels walk them ---------------------
@pytest.mark.parametrize("mode,formula", [(0, 0), (1, 0), (2, 0), (0, 1), (0, 2), (2, 2)])
@pytest.mark.parametrize("n", [256, 1024, 4096])
def test_full_plane_k5_table_bit_exact(orc_pm, n, mode, formula, built):
    p = g.default_params("bars", n=n, sample_mode=mode, round_formula=formula)
    op = params_from(p)
    for seed in (1, 2):
        tex = _tex(n, seed)
        assert np.array_equal(emul.k5_table(p, tex), orc_pm.smooth_pass(op, tex)), (n, mode, formula, seed)
    for const in (0, 65535):
        tex = np.full(n, const, np.uint16)
        assert np.array_equal(emul.k5_table(p, tex), orc_pm.smooth_pass(op, tex))


def test_full_plane_k5_table_wide_window(orc_pm, built):
    """a smoothing factor large enough that taps run past the texture (texelFetch reads 0 there)"""
    p = g.default_params("bars", n=512, smooth_factor=0.3, sample_range=0.999, sample_scale=2.0)
    op = params_from(p)
    tex = _tex(512, 5)
    assert np.array_equal(emul.k5_table(p, tex), orc_pm.smooth_pass(op, tex))


@pytest.mark.parametrize("module,n,w,h", [("bars", 4096, 1920, 1080), ("bars", 1024, 333, 200), ("radial", 2048, 800, 600),
                                          ("graph", 2048, 1280, 720), ("wave", 2048, 1280, 720)])
def test_lazy_k5_tables_give_the_oracle_texels(orc_pm, module, n, w, h, built):
    """need-list + tap table: every texel the module samples equals the oracle's smooth pass there, through both table
    layouts and through the blocks-of-texels tiling (every counting tap inside its block's tile, every texel in exactly one
    block), and the pruning bound epi_n covers every input a tap reads"""
    p = g.default_params(module, n=n, w=w, h=h, lazy_smooth=1)
    op = params_from(p)
    epi = emul.lazy_epi_n(p)
    assert 0 < epi <= n
    for chan in (0, 1):
        tex = _tex(n, 7 + chan)
        want = orc_pm.smooth_pass(op, tex)
        got = {}
        for path in (0, 1, 2, 40):             # 2, 40: blocks of texels out of a tile (k5_need_smem_kernel), default / small blocks
            idx, val = emul.lazy_k5(p, chan, path, tex)
            if module == "wave" and chan == 1:
                assert idx is not None and len(idx) == 0               # audio_r is never sampled (wave/1.frag:7)
                continue
            assert len(idx) > 0 and np.array_equal(val, want[idx]), (module, chan, path)
            got[path] = (idx, val)
        if got:
            assert np.array_equal(got[0][0], got[1][0])
            for path in (2, 40):               # the same texels, widest windows first inside each block
                assert np.array_equal(np.sort(got[path][0]), got[0][0]), (module, chan, path)
            # inputs at or beyond epi_n cannot influence a sampled texel
            tex2 = tex.copy(); tex2[epi:] = 0
            assert np.array_equal(emul.lazy_k5(p, chan, 1, tex2)[1], got[1][1])


@pytest.mark.parametrize("module,n,w,h", [("bars", 8192, 1920, 1080), ("bars", 16384, 1920, 1080), ("radial", 8192, 3840, 2160),
                                          ("graph", 4096, 1920, 1080), ("bars", 512, 1280, 720), ("bars", 256, 64, 16)])
def test_need_list_blocks_at_the_sweep_sizes(orc_pm, module, n, w, h, built):
    """the blocks-of-texels tiling (k5_need_smem_kernel) at the sizes of BASELINE configs[2] and [4]: default tile height, a
    height below every window (one texel per block, tiles as tall as the window) and a tall one"""
    p = g.default_params(module, n=n, w=w, h=h, lazy_smooth=1)
    op = params_from(p)
    for chan in (0, 1):
        tex = _tex(n, 11 + chan)
        want = orc_pm.smooth_pass(op, tex)
        base = emul.lazy_k5(p, chan, 1, tex)
        for path in (2, 4, 4000):
            idx, val = emul.lazy_k5(p, chan, path, tex)
            assert np.array_equal(np.sort(idx), base[0]) and np.array_equal(val, want[idx]), (module, n, chan, path)


def test_circle_has_no_need_list(built):
    p = g.default_params("circle", n=1024, w=320, h=240, lazy_smooth=1)
    assert emul.lazy_k5(p, 0, 0, _tex(1024, 1))[0] is None


def test_need_list_covers_the_join_channels_middle_taps(built):
    """JOIN_CHANNELS samples audio_l around coordinate 1 and audio_r around 0 for `middle` (graph/1.frag:126)"""
    n, w = 1024, 320
    av = np.arange(n, dtype=np.uint16)
    plain = g.default_params("graph", n=n, w=w, h=200, lazy_smooth=1)
    join = g.default_params("graph", n=n, w=w, h=200, lazy_smooth=1, graph_join_channels=1)
    for chan, texel in ((0, int(np.rint((1 - 1 / w) * n))), (1, 0), (1, int(np.rint(1 / w * n)))):
        idx, _ = emul.lazy_k5(join, chan, 0, av)
        assert texel in idx.tolist(), (chan, texel)
    ia, _ = emul.lazy_k5(plain, 0, 0, av); ib, _ = emul.lazy_k5(join, 0, 0, av)
    assert set(ia.tolist()) <= set(ib.tolist())


def test_update_chain_random_parameters(orc_pm, built):
    """product spectrum arithmetic vs the (reference-pinned) oracle over random parameters, both pipelines"""
    rng = np.random.default_rng(77)
    for trial in range(24):
        n = int(rng.choice([256, 1024, 2048]))
        p = g.default_params("bars", n=n, accel_fft=int(trial % 2), avg_window=int(rng.integers(0, 2)),
                             avg_frames=int(rng.integers(1, 9)), fft_scale=float(rng.uniform(0.5, 20)),
                             fft_cutoff=float(rng.uniform(0.0, 1.2)), gravity_step=float(rng.uniform(0.0, 12)),
                             ur=float(rng.uniform(20, 250)), smooth_factor=float(rng.uniform(0.005, 0.06)),
                             sample_mode=int(rng.integers(0, 3)), round_formula=int(rng.integers(0, 3)))
        op = params_from(p)
        oc = OracleChannel(orc_pm, op); ec = emul.Channel(p)
        amp = float(rng.choice([0.004, 0.05, 0.3]))
        for _ in range(n // 256 + 9):
            x = (rng.standard_normal(n) * amp).astype(np.float32)
            s0, t0 = oc.update(x); s1, t1 = ec.update(x)
        peak = max(np.abs(s0).max(), 1e-30)
        assert np.abs(s0 - s1).max() / peak <= 1e-5, (trial, n)
        assert np.abs(t0.astype(int) - t1.astype(int)).max() <= 2, (trial, n)


# ---- the need-list is complete: a lazy frame reads no texel outside it -----------------------------------------------
_RASTER_OPTIONS = ([("bars", o) for o in (dict(bars_direction=1), dict(bars_invert=1), dict(bars_flip=1), dict(bars_mirror_yx=1),
                                          dict(channels=1), dict(channels=1, bars_invert=1), dict(bars_outline_width=0.0),
                                          dict(bars_width=3.0, bars_gap=2.0), dict(smooth_pass=0), dict(bars_width=1.0, bars_gap=0.0))]
                   + [("radial", o) for o in (dict(radial_invert=1), dict(radial_off_x=40.0, radial_off_y=-25.0), dict(radial_nbars=37),
                                              dict(radial_nbars=181), dict(radial_rotate=0.7), dict(radial_amplify=-120.0))]
                   + [("graph", o) for o in (dict(graph_direction=-1), dict(graph_invert=1), dict(graph_draw_outline=1),
                                             dict(graph_draw_highlight=0), dict(graph_join_channels=1))]
                   + [(m, {}) for m in ("bars", "radial", "graph", "wave")])


@pytest.mark.parametrize("w,h", [(320, 200), (333, 97), (802, 601)])
@pytest.mark.parametrize("module,over", _RASTER_OPTIONS, ids=[f"{m}-{'-'.join(f'{k}={v}' for k, v in o.items()) or 'default'}" for m, o in _RASTER_OPTIONS])
def test_lazy_frame_reads_only_need_list_texels(orc_pm, module, over, w, h, built):
    """lazy_smooth = 1 smooths only the texels of emul.lazy_k5's list (tables.h build_need_list): every other texel of the
    texture is stale on the device, so randomising all of them must leave the oracle's frame unchanged"""
    n = 1024
    p = g.default_params(module, n=n, w=w, h=h, lazy_smooth=1, **over)
    op = params_from(p)
    tl, tr = orc_pm.smooth_pass(op, _tex(n, 21)), orc_pm.smooth_pass(op, _tex(n, 22))
    if module == "wave":
        tl = (tl.astype(int) // 4 + 24576).astype(np.uint16)             # PCM-like values around 0.5
    want = orc_pm.raster(op, tl, tr)
    assert want.any()
    rng = np.random.default_rng(w * h)
    stale = []
    for chan, t in ((0, tl), (1, tr)):
        idx, _ = emul.lazy_k5(p, chan, 1, t)
        keep = np.zeros(n, bool); keep[idx] = True
        s = t.copy(); s[~keep] = rng.integers(0, 65536, int((~keep).sum()), dtype=np.uint16)
        stale.append(s)
    assert np.array_equal(orc_pm.raster(op, stale[0], stale[1]), want), (module, over, w, h)


# ---- parameter sets that select a K5 fallback stay on their side of capi.cu's size thresholds -------------------------
# capi.cu build_tables: lazy tap table <= 64 MB (:351), one channel's blob + the FFT buffers <= 112 KB for the one-kernel form
# (:363), tallest need-block tile * 33 floats <= 200 KB for the shared-memory K5 tiles, else the L2 form (:382);
# build_k5_table: full-plane table <= 256 MB and 2 spans <= 200 KB, else k5_planes_kernel evaluates the taps itself (:308).
# tests/test_z_gpu_launch_structures.py runs these parameter sets on the device and counts their launches.
MB = 1 << 20


def _sizes(n, w=1920, **over):
    return emul.table_sizes(g.default_params("bars", n=n, w=w, h=48, lazy_smooth=1, **over))


@pytest.mark.parametrize("over", [dict(), dict(sample_mode=1)])
def test_l2_fallback_parameters_exceed_the_tile_limit(over, built):
    s = _sizes(16384, smooth_factor=0.1, **over)
    assert s["lazy_tab_bytes"] <= 64 * MB and s["lazy_blob_bytes"] > 112 * 1024
    assert s["need_tile_rows"] * 33 * 4 > 200 * 1024, s


def test_full_plane_parameters_exceed_the_table_limit(built):
    s = _sizes(16384, smooth_factor=0.3)
    assert s["full_bytes"] > 256 * MB, s
    assert s["need_tile_rows"] * 33 * 4 > 200 * 1024                   # (its lazy form: the L2 fallback)


def test_split_below_4096_parameters_do_not_fit_next_to_the_fft(built):
    s = _sizes(2048, w=7680)
    assert s["lazy_blob_bytes"] > 112 * 1024 and s["need_tile_rows"] * 33 * 4 <= 200 * 1024, s


@pytest.mark.parametrize("n", [512, 1024, 2048, 4096, 8192, 16384])
def test_sweep_points_use_shared_memory_k5_tiles(n, built):
    """every benchmarked shape at default parameters keeps its K5 out of the L2 fallback and its full-plane table uploaded"""
    for w in (1280, 1920, 3840, 7680):
        s = _sizes(n, w=w)
        assert s["lazy_tab_bytes"] <= 64 * MB and s["need_tile_rows"] * 33 * 4 <= 200 * 1024, (n, w, s)
        assert s["full_bytes"] <= 256 * MB and 2 * s["full_span"] * 4 <= 200 * 1024, (n, w, s)
