"""Frames computed from the REFERENCE'S OWN SHADER TEXT (tests/golden/glsl_golden.npz, made by
tests/golden/make_glsl_golden.py with oracle/glsl_interp.py) against the C restatement (oracle), the product arithmetic
compiled for the host (tests/emul) and — -m gpu — the kernels.  Round 1's pin of the raster half and the GL passes
K2 / K4 / K5: the interpreter takes macro precedence, int / float typing, operand order, stage chaining and quantisation
from the .frag / .glsl files themselves.  Since round 2 the pin is the reference itself on Mesa llvmpipe
(tests/test_llvmpipe_golden.py); these frames stay as EXACT (same-libm) single-stage checks on chosen textures."""
import ctypes as C
import json
import os
import zlib

import numpy as np
import pytest

import glava_b200 as g
from oracle.oracle import params_from
from tests.conftest import GOLDEN
from tests.reference_record import same

W, H, N = 96, 54, 512
REF_SHADERS = "/root/reference/shaders/glava"
OWN_CONFIG = os.path.join(os.path.dirname(g.__file__), "config")      # the reader's fallback on our side


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(GOLDEN, "glsl_golden.npz"))


def _cases():
    z = np.load(os.path.join(GOLDEN, "glsl_golden.npz"))
    return [str(c) for c in z["case_names"]]


def _params(gold, case):
    module = str(gold[f"{case}_module"])
    over = json.loads(str(gold[f"{case}_params"]))
    w, h = (int(v) for v in gold[f"{case}_size"])
    return module, g.default_params(module, n=N, w=w, h=h, **over)


def _lsb(a, b):
    return int(np.abs(a.astype(int) - b.astype(int)).max())


@pytest.mark.parametrize("case", _cases())
def test_oracle_equals_the_reference_shader_frames(orc, orc_pm, gold, case, built):
    module, p = _params(gold, case)
    op = params_from(p)
    tl, tr, want = gold[f"{case}_tl"], gold[f"{case}_tr"], gold[f"{case}_frame"]
    assert want.any()
    got = orc.raster(op, tl, tr)
    assert np.array_equal(got, want), (case, int((got != want).any(axis=2).sum()))      # same libm as the interpreter: exact
    assert _lsb(orc_pm.raster(op, tl, tr), want) <= 1                                      # product-maths build


@pytest.mark.parametrize("case", _cases())
def test_product_arithmetic_equals_the_reference_shader_frames(orc_pm, gold, case, built):
    from tests import emul
    module, p = _params(gold, case)
    tl, tr, want = gold[f"{case}_tl"], gold[f"{case}_tr"], gold[f"{case}_frame"]
    got = emul.raster(p, tl, tr)
    assert _lsb(got, want) <= 1 and (got != want).any(axis=2).sum() <= 0.002 * want.shape[0] * want.shape[1], case
    if module in ("bars", "graph", "wave", "circle") and not p.bars_mirror_yx and p.premultiply_alpha and not p.graph_join_channels and not p.graph_anti_alias:
        assert np.array_equal(emul.raster(p, tl, tr, fast=True), got)                      # the kernels' hoisted evaluation (native
                                                                                           # opacity only: launch_raster's rule)


def _native_cases():
    """non-native opacity (GL blending over the clear colour) runs in tests/test_zz_gpu_blend.py"""
    return [c for c in _cases() if not (c.endswith("_blend") or c.endswith("_blend_opaque") or c.endswith("_nopremult")
                                        or c in ("radial_outline", "graph_join", "graph_aa", "graph_aa_invert"))]   # (per-pixel kernels: same file)


@pytest.mark.gpu
@pytest.mark.parametrize("case", _native_cases())
def test_kernels_equal_the_reference_shader_frames(orc_pm, gold, case, built):
    module, p = _params(gold, case)
    tl, tr, want = gold[f"{case}_tl"], gold[f"{case}_tr"], gold[f"{case}_frame"]
    with g.Renderer(p, batch=2) as r:
        r.raster_textures(np.stack([tl, tl]), np.stack([tr, tr]))
        got = r.readback(1)
    assert _lsb(got, want) <= 1 and (got != want).any(axis=2).sum() <= 0.002 * want.shape[0] * want.shape[1], case


# ---- the GL passes on 1-D R16 textures --------------------------------------------------------------------------------------
MODES = {"average": 0, "maximum": 1, "hybrid": 2}
FORMULAS = {"sinusoidal": 0, "linear": 1, "circular": 2}


@pytest.mark.parametrize("mode,formula", [("average", "sinusoidal"), ("average", "linear"), ("average", "circular"),
                                          ("maximum", "sinusoidal"), ("hybrid", "sinusoidal")])
def test_k5_smooth_pass_equals_smooth_pass_frag(orc, orc_pm, gold, mode, formula, built):
    from tests import emul
    tex, want = gold["k5_in"], gold[f"k5_{mode}_{formula}"]
    p = g.default_params("bars", n=len(tex), sample_mode=MODES[mode], round_formula=FORMULAS[formula])
    op = params_from(p)
    assert _lsb(orc.smooth_pass(op, tex), want) <= 1                       # same libm as the interpreter
    # product maths (gl_math.h log / sin polynomials, <= 1 ulp from libm): 1 LSB16, except `circular`, whose
    # sqrt(1 - (x - 1)^2) has an infinite slope at the window edge and turns an ulp of the log into tens of LSB16 of one
    # edge tap's weight (still < 0.2 LSB of an 8-bit pixel)
    tol = 64 if formula == "circular" else 1
    assert _lsb(orc_pm.smooth_pass(op, tex), want) <= tol
    assert _lsb(emul.smooth(p, tex), want) <= tol and _lsb(emul.k5_table(p, tex), want) <= tol


def _from16(u):
    return (u.astype(np.float32) / np.float32(65535.0)).astype(np.float32)


def _unorm16(v):
    v = np.asarray(v, np.float32)
    q = np.rint((v * np.float32(65535.0)).astype(np.float32))       # GL's float -> R16: one rounding, ties to even (Mesa; llvmpipe goldens)
    return np.where(v > 0, np.where(v < 1, q.astype(np.int64), 65535), 0).astype(np.uint16)


def test_gravity_and_pass_frag(gold):
    """K2 = texel - diff, K1 / K3 = copy (the restatement in oracle/glava_oracle.c orc_chan_update and the kernel's
    gravity_b use exactly this arithmetic)"""
    tex = gold["k5_in"]
    assert np.array_equal(gold["pass_out"], tex)
    assert np.array_equal(gold["gravity_out"], _unorm16(_from16(tex) - np.float32(gold["gravity_diff"])))


@pytest.mark.parametrize("F,win", [(5, 1), (3, 1), (2, 1), (5, 0)])
def test_average_pass_frag(gold, F, win):
    """K4: r += window(I, _AVG_FRAMES - 1) * t_I with the macro expanding to cos(TWOPI * I / F - 1), newest frame first;
    no window for two frames (average_pass.frag:27-29); r / F without normalising the window"""
    frames = gold["avg_frames_in"][:F]
    r = np.zeros(frames.shape[1], np.float32)
    windowed = win and F != 2
    for i in range(F):
        tx = _from16(frames[i])
        if windowed:
            w = np.float32(0.53836) - np.float32(0.46164) * np.cos(np.float32(np.float32(6.28318530718) * np.float32(i) / np.float32(F)) - np.float32(1.0), dtype=np.float32)
            r = (r + (np.float32(w) * tx).astype(np.float32)).astype(np.float32)
        else:
            r = (r + tx).astype(np.float32)
    want = gold[f"avg_F{F}_w{win}"]
    assert _lsb(_unorm16(r / np.float32(F)), want) <= 1


# ---- the interpreter against the oracle on a fresh configuration (recorded where the reference tree is absent) ----------------
def _interpret(module, w, h, tl, tr, **kw):
    """one frame of the module's shaders from the reference tree, run by the interpreter"""
    from oracle import glsl_interp as gi
    prog = gi.ModuleProgram(REF_SHADERS, module, w, h, tl, tr, **kw)
    got = np.zeros((h, w, 4), np.uint8)
    for y in range(h):
        for x in range(w):
            got[y, x] = prog.pixel(x, y)
    return got


@pytest.mark.parametrize("module,gl_over,p_over", [
    ("bars", {"AMPLIFY": "30", "BAR_WIDTH": "3", "BAR_GAP": "1"}, dict(bars_amplify=30.0, bars_width=3.0, bars_gap=1.0)),
    ("radial", {"C_RADIUS": "9", "AMPLIFY": "20", "NBARS": "32"}, dict(radial_radius=9.0, radial_amplify=20.0, radial_nbars=32)),
    ("circle", {"C_RADIUS": "15", "AMPLIFY": "25"}, dict(circle_radius=15.0, circle_amplify=25.0)),
    ("graph", {"VSCALE": "30"}, dict(graph_vscale=30.0)),
    ("wave", {"AMPLIFY": "30"}, dict(wave_amplify=30.0)),
])
def test_interpreter_live_against_the_oracle(orc, ref_record, module, gl_over, p_over, built):
    w, h, n = 64, 40, 256
    p = orc.default_params(module, n=n, w=w, h=h, **p_over)
    rng = np.random.default_rng(zlib.crc32(module.encode()) % 1000)
    tl = orc.smooth_pass(p, (rng.random(n) ** 2 * 65535).astype(np.uint16))
    tr = orc.smooth_pass(p, (rng.random(n) ** 3 * 65535).astype(np.uint16))
    if module == "wave":
        tl = np.clip(tl.astype(int) // 4 + 24576, 0, 65535).astype(np.uint16)
    want = orc.raster(p, tl, tr)
    got = ref_record.call("interpret", lambda a, b: _interpret(module, w, h, a, b, overrides=gl_over), (tl, tr))
    assert same(want, got), module


@pytest.mark.skipif(not os.path.isdir(REF_SHADERS), reason="reference tree not present")
def test_interpreter_reproduces_the_reference_known_answer(built):
    from oracle import glsl_interp as gi
    z = np.zeros(256, np.uint16)
    prog = gi.ModuleProgram(REF_SHADERS, "test", 8, 4, z, z)
    assert len(prog.stages) == 3 and prog.pixel(3, 2) == (0x55, 0, 0, 0x55)              # test_rc.glsl:27


# ---- the config reader (glava_b200/csrc/config.cpp) against the shader semantics of the same config text (recorded where the
# reference tree is absent) ------------------------------------------------------------------------------------------------------
USER_CONFIGS = {
    "bars": """
#define BAR_WIDTH 3
#define BAR_GAP 2
#define BAR_OUTLINE_WIDTH 1
#define AMPLIFY (20 + 15)
#define GRADIENT 30
#define COLOR mix(#ff8000, #2040ff, clamp(d / GRADIENT, 0, 1))
#define BAR_OUTLINE #20c040
#define DIRECTION 1
""",
    "radial": """
#define C_RADIUS 11
#define C_LINE 3
#define OUTLINE #808020
#define NBARS 36
#define BAR_WIDTH 2.5
#define AMPLIFY 25
#define GRADIENT 12
#define COLOR mix(#10e0e0, #e010e0, clamp(d / GRADIENT, 0, 1))
#define ROTATE (PI / 4)
#define INVERT 1
""",
    "bars:conditionals": """
#define FANCY 2
#ifdef FANCY
#define BAR_WIDTH 3
#else
#define BAR_WIDTH 7
#endif
#if FANCY > 1 && !defined(NOPE)
#define BAR_GAP 2
#elif FANCY == 1
#define BAR_GAP 5
#else
#define BAR_GAP 0
#endif
#ifndef AMPLIFY_OVERRIDE
#undef AMPLIFY
#define AMPLIFY (FANCY * 15)
#endif
#if 0
#define COLOR #ff0000
#define BAR_WIDTH 1
#endif
#if (FANCY - 2) || defined FANCY
#define BAR_OUTLINE_WIDTH 0
#endif
""",
    "radial:outline": """
#define C_RADIUS 10
#define NBARS 20
#define BAR_WIDTH 5
#define AMPLIFY 25
#define BAR_OUTLINE_WIDTH 2
#define OUTLINE #4080c0
""",
    "circle": """
#define C_RADIUS 14
#define C_LINE 2
#define OUTLINE vec4(0.9, 0.5, 0.1, 1)
#define AMPLIFY 22
#define ROTATE (TWOPI / 3)
""",
    "graph": """
#define VSCALE 35
#define GRADIENT 20
#define COLOR mix(#a0ff20, #2020c0, clamp(pos / GRADIENT, 0, 1))
#define DRAW_OUTLINE 1
#define OUTLINE #ff00ff
#define DIRECTION -1
""",
    "wave": """
#define MIN_THICKNESS 2
#define MAX_THICKNESS 5
#define BASE_COLOR vec4(0.2, 0.6, 0.3, 1)
#define AMPLIFY 35
#define OUTLINE #101010
""",
}


@pytest.mark.parametrize("module", sorted(USER_CONFIGS))
def test_config_reader_agrees_with_the_shaders_on_a_user_config(orc, ref_record, tmp_path, module, built):
    key, module = module, module.split(":")[0]
    """a user's <module>.glsl goes (a) through glava_b200_load_config -> parameters -> oracle raster and (b) as text through
    the reference's shaders in the interpreter: same pixels.  Covers colour literals / mix() gradients / constant
    vec4 colours / integer vs float macro values / parenthesised arithmetic in #defines."""
    w, h, n = 72, 44, 256
    user = tmp_path / "user"
    user.mkdir()
    (user / "rc.glsl").write_text("#request mod %s\n#request setbufsize %d\n#request setgeometry 0 0 %d %d\n" % (module, n, w, h))
    (user / (module + ".glsl")).write_text(USER_CONFIGS[key])
    p = g.load_config([str(user), OWN_CONFIG])
    assert p.module_name == module and (p.w, p.h, p.n) == (w, h, n)
    op = params_from(p)
    rng = np.random.default_rng(len(module))
    tl = orc.smooth_pass(op, (rng.random(n) ** 2 * 65535).astype(np.uint16))
    tr = orc.smooth_pass(op, (rng.random(n) ** 3 * 65535).astype(np.uint16))
    if module == "wave":
        tl = np.clip(tl.astype(int) // 4 + 24576, 0, 65535).astype(np.uint16)
    want = orc.raster(op, tl, tr)
    got = ref_record.call("interpret", lambda d, a, b: _interpret(module, w, h, a, b, config_dir=d), (str(user), tl, tr))
    assert want.any() and same(want, got), module


def _pass_shader_chain(n, F, win, diff, bs):
    """K1..K5 over the updates `bs`, every pass executed from the reference's util/*.frag by the interpreter; -> the K5
    texture after every update"""
    from oracle import glsl_interp as gi
    util = os.path.join(REF_SHADERS, "util")
    hdr = dict(avg_frames=F, avg_window=win)
    grav = gi.load_stage(os.path.join(util, "gravity_pass.frag"), REF_SHADERS, None, **hdr)
    copy = gi.load_stage(os.path.join(util, "pass.frag"), REF_SHADERS, None, **hdr)
    avg = gi.load_stage(os.path.join(util, "average_pass.frag"), REF_SHADERS, None, **hdr) if F > 1 else None
    k5 = gi.load_stage(os.path.join(util, "smooth_pass.frag"), REF_SHADERS, None, **hdr)

    def run(sh, uniforms):
        out = np.zeros(n, np.uint16)
        for x in range(n):
            out[x] = gi.unorm16(sh.run(dict(uniforms), x, 0)["fragment"].v[0])
        return out

    gr_store = np.zeros(n, np.uint16)
    ring = [np.zeros(n, np.uint16) for _ in range(F)]
    out_idx = 0
    outs = []
    for b in bs:
        upload = _unorm16(b)                                                          # glTexImage1D GL_R16, render.c:521-524
        gr_store = np.maximum(gr_store, run(copy, {"tex": gi.Sampler1D(upload)}))     # K1: pass.frag blended with GL_MAX
        gr_store = run(grav, {"tex": gi.Sampler1D(gr_store), "diff": diff})           # K2 in place
        tex = gr_store
        if F > 1:
            ring[out_idx] = run(copy, {"tex": gi.Sampler1D(gr_store)})                # K3
            uni = {f"t{t}": gi.Sampler1D(ring[(out_idx - t) % F]) for t in range(F)}  # t0 = most recent (render.c:2250-2255)
            tex = run(avg, uni)                                                       # K4
            out_idx = (out_idx + 1) % F
        outs.append(run(k5, {"tex": gi.Sampler1D(tex), "sz": n, "w": n}))             # K5
    return np.stack(outs)


@pytest.mark.parametrize("F,win", [(5, 1), (3, 1), (2, 1), (1, 1), (4, 0)])
def test_pipeline_b_chain_through_the_reference_pass_shaders(orc, ref_record, F, win, built):
    """the accelerated chain of one channel over several updates — R16 upload, K1 GL_MAX into gr_store, K2
    gravity_pass.frag in place, K3 pass.frag into the ring slot, K4 average_pass.frag over the ring newest-first,
    K5 smooth_pass.frag (render.c:2188-2303) — with every shader pass EXECUTED from the reference's source by the
    interpreter, against orc_chan_update's restatement of the same chain: identical textures after every update."""
    from oracle.oracle import OracleChannel
    n = 128
    p = orc.default_params("bars", n=n, accel_fft=1, avg_frames=F, avg_window=win)
    ch = OracleChannel(orc, p)
    rng = np.random.default_rng(F * 10 + win)
    bs = np.stack([(rng.random(n) ** 2 * (1.3 if u % 3 else 0.2)).astype(np.float32)  # "transform_fft output", some > 1
                   for u in range(2 * F + 3)])
    diff = np.float32(p.gravity_step) * (np.float32(1.0) / np.float32(p.ur))          # render.c:2224
    gots = ref_record.call("pass_shader_chain", lambda d, b: _pass_shader_chain(n, F, win, d, b), (diff, bs), whole=True)
    assert gots.shape == (2 * F + 3, n)
    for u, (b, got) in enumerate(zip(bs, gots)):
        spec = np.empty(n, np.float32); tex_o = np.empty(n, np.uint16)
        orc.L.orc_chan_update(ch.h, C.byref(p), b.ctypes.data, 2, spec.ctypes.data, tex_o.ctypes.data)   # 2: `b` is transform_fft's output
        assert np.abs(got.astype(int) - tex_o.astype(int)).max() <= 1, (F, win, u)
        assert (got != tex_o).mean() < 0.02


def _smooth_pass_frag(d, sf, tex):
    """util/smooth_pass.frag of the reference tree with user config dir d, run by the interpreter"""
    from oracle import glsl_interp as gi
    n = tex.shape[0]
    sh = gi.load_stage(os.path.join(REF_SHADERS, "util", "smooth_pass.frag"), REF_SHADERS, None, config_dir=d, smooth_factor=sf)
    return np.array([gi.unorm16(sh.run({"tex": gi.Sampler1D(tex), "sz": n, "w": n}, x, 0)["fragment"].v[0]) for x in range(n)], np.uint16)


def test_k5_random_smooth_parameters_through_smooth_pass_frag(orc, orc_pm, ref_record, tmp_path, built):
    """smooth_pass.frag (K5) run from the reference's text with a random user smooth_parameters.glsl and setsmoothfactor,
    against the oracle and the product arithmetic (direct evaluation and the precomputed tap table): R16 texels within
    2 / 3 LSB16 (3e-5 / 5e-5 of full scale; the serial tap sums round differently by an ulp here and there)"""
    from tests import emul
    rng = np.random.default_rng(31)
    n = 256
    for trial in range(10):
        mode = str(rng.choice(["average", "maximum", "hybrid"])); formula = str(rng.choice(["sinusoidal", "linear"]))
        scale, rng_, hyb = float(np.float32(rng.uniform(4, 10))), float(np.float32(rng.uniform(0.5, 0.95))), float(np.float32(rng.uniform(0.3, 0.9)))
        # (a window narrower than one texel gives weight 0 and the shader returns 0 / 0: which texels hit that knife edge
        # depends on the last ulp of log() — any two GL implementations disagree there; the draw stays clear of it)
        sf = float(np.float32(rng.uniform(0.025, 0.06)))
        user = tmp_path / f"u{trial}"
        user.mkdir()
        (user / "rc.glsl").write_text("#request setbufsize 256\n")
        (user / "smooth_parameters.glsl").write_text(      # (a setsmoothfactor in rc.glsl would lose to smooth_parameters.glsl:72)
            f"#request setsmoothfactor {sf!r}\n#define SAMPLE_MODE {mode}\n#define ROUND_FORMULA {formula}\n#define SAMPLE_SCALE {scale!r}\n"
            f"#define SAMPLE_RANGE {rng_!r}\n#define SAMPLE_HYBRID_WEIGHT {hyb!r}\n")
        p = g.load_config([str(user), OWN_CONFIG])
        p.n = n
        assert (p.sample_mode, p.round_formula) == (MODES[mode], FORMULAS[formula]) and p.smooth_factor == np.float32("%.6f" % sf)      # `#define _SMOOTH_FACTOR %.6f`
        tex = (rng.random(n) ** 2 * 65535).astype(np.uint16)
        want = ref_record.call("smooth_pass_frag", _smooth_pass_frag, (str(user), sf, tex), whole=True)
        assert want.any()
        assert _lsb(orc.smooth_pass(params_from(p), tex), want) <= 2, (trial, mode, formula)
        assert _lsb(emul.smooth(p, tex), want) <= 3 and _lsb(emul.k5_table(p, tex), want) <= 3, (trial, mode, formula)
