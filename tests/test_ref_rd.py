"""The reference's OWN rd_new / rd_update (glava/render.c compiled where it lies) on a null OpenGL driver and a null
window backend (oracle/ref_shim.c, oracle/_ref/libglava_ref_rd.so):

* what rd_new's request handlers make of a configuration — rc.glsl, smooth_parameters.glsl, CLI requests — against the
  product's config reader, field by field;
* what rd_update uploads as the audio textures over a sequence of frames — transform chain, `modified` handling, buffer
  scaling, keyframe interpolation as the reference orchestrates them — against the oracle's restatement (orc_stream_*),
  which is what the kernels are tested against.

rd_new / rd_update need the reference tree (the shipped shaders are what rd_new loads) and an executable stack; where
either is missing their recorded results stand in (tests/reference_record.py: the configuration rd_new read, and every
upload as digests of its floats and of its R16 texture — the comparisons here are bit for bit).  Our side reads the
test's own files and the package's config directory, never the reference tree.  Tests that hand the reference's own
shader text to either side still need the tree."""
import os

import numpy as np
import pytest

import glava_b200 as g
from oracle.oracle import OracleStream, OrcExt, ReferenceRenderer, params_from
from tests.reference_record import Recorded, Session, same

REF_SHADERS = "/root/reference/shaders/glava"
OWN_CONFIG = os.path.join(os.path.dirname(g.__file__), "config")
pytestmark = pytest.mark.timeout(300)
needs_tree = pytest.mark.skipif(not os.path.isdir(REF_SHADERS), reason="reference tree not present")


def _live():
    return os.path.isdir(REF_SHADERS) and ReferenceRenderer.lib() is not None


class _Renderer:
    """ReferenceRenderer through a Session: .cfg as rd_new read it, frame() -> {texture: Recorded upload}"""

    def __init__(self, s, paths, requests):
        self.s = s
        self.r = ReferenceRenderer(paths, requests=requests) if s.live else None
        key = ["<reference tree>" if p == REF_SHADERS else p for p in paths]
        self.cfg = s.call("rd_new", lambda *a: self.r.cfg, (key, list(requests)))
        self.lb = np.zeros(self.cfg["bufsize"], np.float32)
        self.rb = np.zeros(self.cfg["bufsize"], np.float32)

    def set_rates(self, ur, fr):
        self.s.call("set_rates", lambda *a: self.r.set_rates(ur, fr), (float(ur), float(fr)))

    def frame(self, pcm_l=None, pcm_r=None):
        if pcm_l is not None:
            self.lb[:] = pcm_l; self.rb[:] = pcm_r

        def live(*a):
            with np.errstate(over="ignore", invalid="ignore"):         # (uploads of never-initialised keyframe buffers)
                return {str(k): {"raw": Recorded.digest(v), "nan": Recorded.digest(v, True), "tex": Recorded.digest(_unorm16(v)),
                                 "len": int(v.shape[0])} for k, v in self.r.frame(pcm_l, pcm_r).items()}
        # (until two keyframes are pushed, interpolation uploads buffers the reference never initialised: check_live=False)
        return {int(k): Recorded(d) for k, d in self.s.call("frame", live, (pcm_l, pcm_r), check_live=False).items()}

    def close(self):
        if self.r is not None:
            self.r.close()


@pytest.fixture
def rd(built, request):
    s = Session(request, _live())
    return lambda paths, requests=(): _Renderer(s, paths, requests)


@pytest.fixture(scope="module")
def rd_live(built):
    if not os.path.isdir(REF_SHADERS):
        pytest.skip("reference tree not present")
    if ReferenceRenderer.lib() is None:
        pytest.skip("oracle/_ref/libglava_ref_rd.so not built or not loadable (needs an executable stack)")
    return ReferenceRenderer


def _tex(up):
    """the R16 texture of a recorded upload (GL's float -> R16 conversion of its floats)"""
    return Recorded({"raw": up.d["tex"], "nan": up.d["tex"]})


def _user_dir(path, files):
    """a user configuration directory the way `glava --copy-config` lays it out: the user's own files, symlinks to the
    installed shaders / modules for everything else (render.c:1318-1320; only where the reference tree is present — only
    the reference reads them)"""
    path.mkdir()
    for name, text in files.items():
        (path / name).write_text(text)
    if os.path.isdir(REF_SHADERS):
        for entry in os.listdir(REF_SHADERS):
            if entry not in files:
                os.symlink(os.path.join(REF_SHADERS, entry), path / entry)
    return str(path)


def _own(path, files):
    """the same user files for our config reader, which falls back to the package's config directory"""
    path.mkdir()
    for name, text in files.items():
        (path / name).write_text(text)
    return [str(path), OWN_CONFIG]


def _unorm16(v):
    v = np.asarray(v, np.float32)
    q = np.rint((v * np.float32(65535.0)).astype(np.float32))       # GL's float -> R16: one rounding, ties to even (Mesa; llvmpipe goldens)
    with np.errstate(invalid="ignore"):
        return np.where(v > 0, np.where(v < 1, q.astype(np.int64), 65535), 0).astype(np.uint16)


CONFIGS = [
    ("shipped", "", "", []),
    ("user rc", '#request mod radial\n#request setbufsize 2048\n#request setgeometry 5 6 640 360\n#request setopacity "none"\n'
     "#request setbg 10203040\n#request setmirror true\n#request setsamplerate 44100\n#request setsamplesize 512\n"
     "#request setaccelfft false\n#request setinterpolate true\n#request setbufscale 2\n#request setframerate 120\n", "", []),
    ("user smooth parameters", "#request mod graph\n",
     "#request setfftscale 7.5\n#request setfftcutoff 0.45\n#request setavgframes 3\n#request setavgwindow false\n"
     "#request setgravitystep 2.25\n#request setsmoothfactor 0.0438713878\n#request setsmoothpass false\n", []),
    # one CLI request per run: rd_new reuses one `struct glsl_ext` for all of them and ext_free() leaves its destructor list
    # dangling, so a second `--request` corrupts the reference's heap (render.c:1415-1435, glsl_ext.c:124-136)
    ("cli request wins", "#request mod wave\n#request setbufsize 1024\n", "", ["setbufsize 8192"]),
    ("cli setbgf", "#request mod wave\n", "", ["setbgf 0.25 0.5 0.75 1.0"]),
    ("cli xroot", "#request mod circle\n#request setsmooth 0.02\n#request setsmoothratio 3.5\n", "", ['setopacity "xroot"']),
    ("rc leaves everything to rd_new's initialisers", "#request mod bars\n", "", []),
]


@pytest.mark.parametrize("name,rc,sp,requests", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_config_reader_reads_what_rd_new_reads(rd, tmp_path, name, rc, sp, requests):
    paths, ours = [REF_SHADERS], [OWN_CONFIG]
    if rc or sp:
        files = {"rc.glsl": rc or "#request mod bars\n"}
        if sp:
            files["smooth_parameters.glsl"] = sp
        paths = [_user_dir(tmp_path / "user", files), REF_SHADERS]
        ours = _own(tmp_path / "own", files)
    r = rd(paths, requests=requests)
    try:
        c = r.cfg
        p = g.load_config(ours, requests=requests)
        assert (p.n, p.rate_request, p.samplesize_request) == (c["bufsize"], c["rate"], c["samplesize"])
        assert p.channels == (1 if c["mirror_input"] else 2)
        assert (p.avg_frames, p.avg_window, p.smooth_pass, p.accel_fft) == (c["avg_frames"], c["avg_window"], c["smooth_pass"], c["accel_fft"])
        assert (p.interpolate, p.bufscale, p.premultiply_alpha) == (c["interpolate"], c["bufscale"], c["premultiply_alpha"])
        assert (p.w, p.h) == (c["w"], c["h"])
        for ours, theirs in (("fft_scale", "fft_scale"), ("fft_cutoff", "fft_cutoff"), ("gravity_step", "gravity_step"),
                             ("smooth_distance", "smooth_distance"), ("smooth_ratio", "smooth_ratio")):
            assert getattr(p, ours) == np.float32(c[theirs]), ours
        assert p.smooth_factor == np.float32("%.6f" % c["smooth_factor"])     # the shaders get the "%.6f" literal (render.c:315-324)
        assert list(p.clear_color) == [np.float32(c[k]) for k in ("clear_r", "clear_g", "clear_b", "clear_a")]
        if c["framerate"] > 0:
            assert p.fr == c["framerate"]
    finally:
        r.close()


def _chain_case(rd, tmp_path, extra_rc, ur, fr, pattern, seed):
    """pipeline A with the R16 texture taken straight from the upload (setsmoothpass false): reference uploads vs oracle"""
    files = {"rc.glsl": "#request mod bars\n#request setbufsize 1024\n#request setaccelfft false\n" + extra_rc,
             "smooth_parameters.glsl": "#request setsmoothpass false\n"}
    paths = [_user_dir(tmp_path / "u", files), REF_SHADERS]
    r = rd(paths)
    try:
        p = g.load_config(_own(tmp_path / "own", files))
        assert p.smooth_pass == 0 and p.accel_fft == 0
        p.ur = ur
        ext = OrcExt(bufscale=p.bufscale, interpolate=p.interpolate, fr=fr, transform_smooth=0, smooth_distance=0.01, smooth_ratio=4.0)
        from oracle.oracle import Oracle
        orc = Oracle("libm")
        st = OracleStream(orc, params_from(p), ext)
        r.set_rates(ur, fr)
        rng = np.random.default_rng(seed)
        n = p.n
        checked = 0
        pushed = 0                                        # keyframes pushed so far (render.c:2347-2353)
        for k, modified in enumerate(pattern):
            if modified:
                amp = [0.15, 0.02, 0.4][k % 3]
                pl = (rng.standard_normal(n) * amp).astype(np.float32); pr = (rng.standard_normal(n) * amp).astype(np.float32)
                up = r.frame(pl, pr)
                sl, sr, tl, tr = st.update(pl, pr, True)
            else:
                up = r.frame()
                sl, sr, tl, tr = st.update(np.zeros(n, np.float32), np.zeros(n, np.float32), False)
            assert set(up) >= {0, 1}, (k, up.keys())
            assert up[0].d["len"] == st.n
            interp_active = bool(p.interpolate) and ur / fr <= 0.9
            settled = pushed >= 2
            pushed += 1 if modified else 0
            if interp_active and not settled:
                continue      # the reference lerps between malloc'd, never initialised keyframe buffers until two have been pushed
            if p.bufscale > 1 and not modified and not (p.interpolate and ur / fr <= 0.9):
                # Known deviation, deliberately not reproduced: with setbufscale > 1 the reference's transforms run on a
                # stack copy (nlb / nrb, render.c:1765-1790) that is gone by the next frame, so a frame without new audio
                # uploads the RAW box-averaged PCM — one untransformed frame flashes.  Oracle and product re-show the last
                # spectrum, as the reference itself does when bufscale is 1 (lb / rb keep the transformed data).
                assert same(orc.bufscale(r.lb, p.bufscale), up[0]) and not same(tl, _tex(up[0]))
                checked += 1
                continue
            assert same(tl, _tex(up[0])) and same(tr, _tex(up[1])), (k, modified)
            if modified and not (p.interpolate and ur / fr <= 0.9):
                assert same(sl, up[0]) and same(sr, up[1]), k                        # the float chain result itself, bit for bit
            checked += 1
        return checked
    finally:
        r.close()


def test_transform_chain_and_modified_handling(rd, tmp_path):
    assert _chain_case(rd, tmp_path, "", 86.1328125, 86.1328125, [1, 1, 0, 1, 0, 0, 1, 1, 1, 0, 1], 1) == 11


def test_buffer_scaling(rd, tmp_path):
    assert _chain_case(rd, tmp_path, "#request setbufscale 2\n", 86.1328125, 86.1328125, [1, 1, 1, 0, 1, 1], 2) == 6
    (tmp_path / "b").mkdir()
    assert _chain_case(rd, tmp_path / "b", "#request setbufscale 4\n", 50.0, 50.0, [1, 0, 1, 1], 3) == 4


def test_keyframe_interpolation(rd, tmp_path):
    # ur / fr = 0.25: three interpolated frames between updates; output runs one update late (rc.glsl:129-130)
    assert _chain_case(rd, tmp_path, "#request setinterpolate true\n", 30.0, 120.0, [1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0, 0, 0, 1, 0], 4) == 11   # 5 unsettled frames skipped
    (tmp_path / "b").mkdir()
    # ur / fr > 0.9: the reference switches interpolation off for the frame (render.c:1761-1763)
    assert _chain_case(rd, tmp_path / "b", "#request setinterpolate true\n", 100.0, 105.0, [1, 0, 1, 1, 0, 1], 5) == 6
    (tmp_path / "c").mkdir()
    assert _chain_case(rd, tmp_path / "c", "#request setinterpolate true\n#request setbufscale 2\n", 40.0, 100.0, [1, 0, 1, 0, 0, 1, 0, 1], 6) == 5


def test_pipeline_b_uploads_transform_fft_only(rd, tmp_path):
    """setaccelfft true (shipped): on a modified frame rd_update uploads transform_fft's output and leaves gravity / average
    to the GL passes (render.c:2131-2180) — the oracle's `spec` in pipeline B is that buffer, bit for bit; interpolation is
    forced off for such a bind (render.c:2161-2168) even though rd_new's initialiser has it on"""
    from oracle.oracle import Oracle
    files = {"rc.glsl": "#request mod bars\n#request setbufsize 2048\n"}
    paths = [_user_dir(tmp_path / "u", files), REF_SHADERS]
    r = rd(paths)
    try:
        p = g.load_config(_own(tmp_path / "own", files))
        assert p.accel_fft == 1 and p.interpolate == 1 and r.cfg["interpolate"] == 1
        p.ur = 30.0
        st = OracleStream(Oracle("libm"), params_from(p), OrcExt(bufscale=1, interpolate=1, fr=120.0, transform_smooth=0, smooth_distance=0.01, smooth_ratio=4.0))
        r.set_rates(30.0, 120.0)
        rng = np.random.default_rng(9)
        for k in range(5):
            pl = (rng.standard_normal(p.n) * 0.2).astype(np.float32); pr = (rng.standard_normal(p.n) * 0.2).astype(np.float32)
            up = r.frame(pl, pr)
            sl, sr, _, _ = st.update(pl, pr, True)
            assert same(sl, up[0]) and same(sr, up[1]), k
    finally:
        r.close()


def test_wave_chain_window_wrange(rd, tmp_path):
    """wave/1.frag:7-10 binds audio_l only, with the transforms "window" (a no-op) and "wrange": the uploaded buffer is
    (pcm + 1) / 2 (render.c:773-781); keyframe interpolation stays available to it (no fft transform on the bind)"""
    from oracle.oracle import Oracle
    for extra, ur, fr, pattern in (("#request setinterpolate false\n", 86.0, 86.0, [1, 1, 0, 1]),
                                   ("", 30.0, 120.0, [1, 0, 1, 0, 0, 1, 0, 0, 0, 1, 0])):       # rd_new's initialiser: interpolation on
        d = tmp_path / ("w%d" % len(pattern))
        files = {"rc.glsl": "#request mod wave\n#request setbufsize 1024\n" + extra}
        paths = [_user_dir(d, files), REF_SHADERS]
        cli = ["setsmoothpass false"]             # (smooth_parameters.glsl cannot switch it off for wave; one CLI request can)
        r = rd(paths, requests=cli)
        try:
            p = g.load_config(_own(tmp_path / ("own%d" % len(pattern)), files), requests=cli)
            assert p.smooth_pass == 0 and r.cfg["smooth_pass"] == 0
            p.ur = ur
            st = OracleStream(Oracle("libm"), params_from(p), OrcExt(bufscale=1, interpolate=p.interpolate, fr=fr, transform_smooth=0,
                                                                     smooth_distance=0.01, smooth_ratio=4.0))
            r.set_rates(ur, fr)
            rng = np.random.default_rng(13)
            pushed = 0
            for k, modified in enumerate(pattern):
                if modified:
                    pl = (rng.standard_normal(p.n) * 0.2).astype(np.float32)
                    up = r.frame(pl, pl)
                    sl, _, tl, _ = st.update(pl, pl, True)
                else:
                    up = r.frame()
                    sl, _, tl, _ = st.update(np.zeros(p.n, np.float32), np.zeros(p.n, np.float32), False)
                assert 0 in up and 1 not in up                               # audio_r is not bound by this module
                active = bool(p.interpolate) and ur / fr <= 0.9
                settled = pushed >= 2
                pushed += 1 if modified else 0
                if active and not settled:
                    continue
                assert same(tl, _tex(up[0])), (extra, k, modified)                   # lerped or not: what the texture holds
                if modified and not active:
                    assert same(sl, up[0]), (extra, k)
                    assert same((pl + np.float32(1.0)) / np.float32(2.0), up[0])
        finally:
            r.close()


def test_random_configs_against_rd_new(rd, tmp_path):
    """random rc.glsl / smooth_parameters.glsl request sets (each request present or left to rd_new's initialiser, in random
    order, some repeated): the product's reader and the real rd_new agree on every field"""
    rng = np.random.default_rng(55)

    def pick(name, maker, prob=0.6):
        return [f"#request {name} {maker()}"] if rng.random() < prob else []

    for trial in range(24):
        module = str(rng.choice(["bars", "radial", "circle", "graph", "wave"]))
        b = lambda: str(rng.choice(["true", "false", "t", "f", "1", "0"]))                  # noqa: E731
        rc = [f"#request mod {module}"]
        rc += pick("setbufsize", lambda: str(rng.choice([512, 1024, "0x800", 4096, 8192])))
        rc += pick("setgeometry", lambda: "%d %d %d %d" % tuple(rng.integers(100, 2000, 4)))
        rc += pick("setopacity", lambda: '"%s"' % rng.choice(["native", "none", "xroot"]))
        rc += pick("setmirror", b) + pick("setaccelfft", b) + pick("setinterpolate", b)
        rc += pick("setsamplerate", lambda: str(rng.choice([22050, 44100, 48000]))) + pick("setsamplesize", lambda: str(rng.choice([256, 512, 1024])))
        rc += pick("setbufscale", lambda: str(rng.choice([1, 2])), 0.3) + pick("setframerate", lambda: str(rng.choice([0, 60, 144])))
        rc += pick("setbg", lambda: "%08x" % int(rng.integers(0, 1 << 32)), 0.4) + pick("setbgf", lambda: "%.3f %.3f %.3f %.3f" % tuple(rng.random(4)), 0.3)
        rc += pick("setsmooth", lambda: "%.4f" % rng.uniform(0.005, 0.05), 0.3) + pick("setsmoothratio", lambda: "%.2f" % rng.uniform(1, 6), 0.3)
        rc += pick("setbufsize", lambda: str(rng.choice([1024, 2048])), 0.2)                # a later request overrides
        tail = rc[1:]; rng.shuffle(tail); rc = rc[:1] + tail
        sp = pick("setfftscale", lambda: "%.3f" % rng.uniform(1, 20)) + pick("setfftcutoff", lambda: "%.3f" % rng.uniform(0, 1))
        sp += pick("setavgframes", lambda: str(int(rng.integers(1, 9)))) + pick("setavgwindow", b) + pick("setgravitystep", lambda: "%.3f" % rng.uniform(0, 10))
        sp += pick("setsmoothfactor", lambda: "%.7f" % rng.uniform(0.005, 0.08)) + pick("setsmoothpass", b)
        files = {"rc.glsl": "\n".join(rc) + "\n"}
        if sp and rng.random() < 0.8:
            files["smooth_parameters.glsl"] = "\n".join(sp) + "\n"
        paths = [_user_dir(tmp_path / f"t{trial}", files), REF_SHADERS]
        r = rd(paths)
        try:
            c = r.cfg
            p = g.load_config(_own(tmp_path / f"own{trial}", files))
            got = dict(bufsize=p.n, rate=p.rate_request, samplesize=p.samplesize_request, mirror_input=2 - p.channels,
                       avg_frames=p.avg_frames, avg_window=p.avg_window, smooth_pass=p.smooth_pass, accel_fft=p.accel_fft,
                       interpolate=p.interpolate, bufscale=p.bufscale, premultiply_alpha=p.premultiply_alpha, w=p.w, h=p.h)
            assert got == {k: c[k] for k in got}, (trial, files)
            for ours, theirs in (("fft_scale", "fft_scale"), ("fft_cutoff", "fft_cutoff"), ("gravity_step", "gravity_step"),
                                 ("smooth_distance", "smooth_distance"), ("smooth_ratio", "smooth_ratio")):
                assert getattr(p, ours) == np.float32(c[theirs]), (trial, ours, files)
            assert p.smooth_factor == np.float32("%.6f" % c["smooth_factor"]), (trial, files)
            assert list(p.clear_color) == [np.float32(c[k]) for k in ("clear_r", "clear_g", "clear_b", "clear_a")], (trial, files)
            assert (p.fr if c["framerate"] > 0 else 0) == max(c["framerate"], 0) or c["framerate"] <= 0
        finally:
            r.close()


def test_smooth_transform_after_fft_forces_the_cpu_order_chain(rd_live, tmp_path):
    """a module whose bind lists "smooth" after "fft" (render.c:1218-1286): under setaccelfft the reference can no longer
    leave gravity / average to the GL passes and runs fft -> gravity -> average -> smooth on the CPU (render.c:2143-2154);
    the uploaded buffer is the oracle's transform_smooth chain, NaN head included"""
    from oracle.oracle import Oracle
    src = open(os.path.join(REF_SHADERS, "bars", "1.frag")).read()
    for ch in ("audio_l", "audio_r"):
        anchor = f'#request transform {ch} "avg"\n'
        assert anchor in src
        src = src.replace(anchor, anchor + f'#request transform {ch} "smooth"\n')
    d = tmp_path / "u"
    paths = [_user_dir(d, {"rc.glsl": "#request mod bars\n#request setbufsize 1024\n#request setinterpolate false\n"
                                     "#request setsmooth 0.02\n#request setsmoothratio 3.0\n"}), REF_SHADERS]
    os.unlink(d / "bars"); (d / "bars").mkdir()                           # a private copy of the module with the extra transform
    for f in os.listdir(os.path.join(REF_SHADERS, "bars")):
        (d / "bars" / f).write_text(src if f == "1.frag" else open(os.path.join(REF_SHADERS, "bars", f)).read())
    r = rd_live(paths)
    try:
        p = g.load_config(paths)
        assert p.accel_fft == 1 and p.smooth_distance == np.float32(0.02) and p.smooth_ratio == np.float32(3.0)
        p.ur = 86.1328125
        st = OracleStream(Oracle("libm"), params_from(p), OrcExt(bufscale=1, interpolate=0, fr=0.0, transform_smooth=1,
                                                                 smooth_distance=p.smooth_distance, smooth_ratio=p.smooth_ratio))
        r.set_rates(86.1328125, 86.1328125)
        rng = np.random.default_rng(17)
        for k in range(7):
            pl = (rng.standard_normal(p.n) * 0.2).astype(np.float32); pr = (rng.standard_normal(p.n) * 0.2).astype(np.float32)
            up = r.frame(pl, pr)
            sl, sr, _, _ = st.update(pl, pr, True)
            assert np.array_equal(up[0], sl, equal_nan=True) and np.array_equal(up[1], sr, equal_nan=True), k
            assert np.isnan(up[0][0])                                      # transform_smooth's b[0] = 0 / 0 (render.c:694-718)
    finally:
        r.close()


@pytest.mark.parametrize("accel", ["true", "false"])
def test_smooth_transform_before_fft_runs_on_the_pcm(rd_live, tmp_path, accel):
    """a module whose bind lists "smooth" BEFORE "window" / "fft": handle_audio applies it on the CPU to the PCM ring, then
    meets "fft" and carries on as usual — GL passes under setaccelfft (the upload is transform_fft of the smoothed ring),
    the whole CPU chain otherwise (render.c:2131-2156).  transform_smooth = 2 in the oracle / product."""
    from oracle.oracle import Oracle
    src = open(os.path.join(REF_SHADERS, "bars", "1.frag")).read()
    for ch in ("audio_l", "audio_r"):
        anchor = f'#request transform {ch} "window"\n'
        assert anchor in src
        src = src.replace(anchor, f'#request transform {ch} "smooth"\n' + anchor)
    d = tmp_path / "u"
    paths = [_user_dir(d, {"rc.glsl": "#request mod bars\n#request setbufsize 1024\n#request setinterpolate false\n"
                                     f"#request setaccelfft {accel}\n#request setsmooth 0.02\n#request setsmoothratio 3.0\n"}), REF_SHADERS]
    os.unlink(d / "bars"); (d / "bars").mkdir()
    for f in os.listdir(os.path.join(REF_SHADERS, "bars")):
        (d / "bars" / f).write_text(src if f == "1.frag" else open(os.path.join(REF_SHADERS, "bars", f)).read())
    r = rd_live(paths)
    try:
        p = g.load_config(paths)
        assert p.accel_fft == (1 if accel == "true" else 0)
        p.ur = 86.1328125
        st = OracleStream(Oracle("libm"), params_from(p), OrcExt(bufscale=1, interpolate=0, fr=0.0, transform_smooth=2,
                                                                 smooth_distance=p.smooth_distance, smooth_ratio=p.smooth_ratio))
        r.set_rates(86.1328125, 86.1328125)
        rng = np.random.default_rng(23)
        from oracle.oracle import Reference
        ref = Reference()
        for k in range(6):
            pl = (rng.standard_normal(p.n) * 0.2).astype(np.float32); pr = (rng.standard_normal(p.n) * 0.2).astype(np.float32)
            up = r.frame(pl, pr)
            sl, sr, _, _ = st.update(pl, pr, True)
            if accel == "false" or k == 0:
                assert np.array_equal(up[0], sl, equal_nan=True) and np.array_equal(up[1], sr, equal_nan=True), k
            elif k >= 2:
                # REFERENCE DEFECT, not reproduced: frame 0 set optimize_fft and truncated the bind's list to [smooth, window]
                # (render.c:2170-2172); frame 1 then takes "smooth" for a transform AFTER an optimised fft, runs the CPU chain
                # once and clears optimize_fft (:2143-2154) — and from frame 2 on nothing transforms the ring but "smooth":
                # GLava uploads the smoothed raw PCM as if it were a spectrum, forever.  The oracle / product keep doing what
                # frame 0 did: transform_fft of the smoothed ring, then the GL passes.
                assert np.array_equal(up[0], ref.smooth(pl, 0.02, 3.0), equal_nan=True), k
    finally:
        r.close()


@pytest.mark.parametrize("rc_extra,sp,state", [
    ("", "", (1, 0)),                                                                       # shipped: consistent
    ("#request setsmoothpass false\n", "#request setsmoothpass false\n", (0, 0)),           # off everywhere: shader smooths
    ("", "#request setsmoothpass false\n", (0, 1)),                                         # off where the shipped config sets it
    ("#request setsmoothpass false\n", "", (1, 2)),                                         # off in rc.glsl only: smoothed twice
])
def test_stage1_header_is_built_before_its_includes_run_their_requests(rd_live, tmp_path, rc_extra, sp, state):
    """shaderload forms `#define _PRE_SMOOTHED_AUDIO ...` (EBIND list, render.c:284-293) before ext_process runs the shader's
    own includes (:312): the module's FIRST shader believes smooth_pass as of the end of rc.glsl, the K5 pass follows the final
    value.  (params.smooth_pass, params.shader_pre_smoothed) must say exactly that."""
    import re
    files = {"rc.glsl": "#request mod bars\n" + rc_extra}
    if sp:
        files["smooth_parameters.glsl"] = open(os.path.join(REF_SHADERS, "smooth_parameters.glsl")).read() + sp
    paths = [_user_dir(tmp_path / "u", files), REF_SHADERS]
    r = rd_live(paths)
    try:
        p = g.load_config(paths)
        assert (p.smooth_pass, p.shader_pre_smoothed) == state
        assert r.cfg["smooth_pass"] == p.smooth_pass                                        # whether K5 runs
        stage1 = next(s for s in r.sources if "BAR_WIDTH" in s)                              # bars/1.frag, the first shader loaded
        believed = int(re.search(r"#define _PRE_SMOOTHED_AUDIO (\d)", stage1).group(1))
        assert believed == ((p.shader_pre_smoothed == 1) if p.shader_pre_smoothed else p.smooth_pass)
        k5 = next(s for s in r.sources if "smooth_audio(tex, sz" in s)                       # util/smooth_pass.frag is loaded later
        assert "#define _PRE_SMOOTHED_AUDIO %d" % p.smooth_pass in k5
    finally:
        r.close()


@pytest.mark.parametrize("module", ["bars", "radial", "circle", "graph", "wave", "test"])
def test_interpreter_consumes_what_rd_new_hands_to_the_glsl_compiler(rd_live, module):
    """every fragment shader text the real rd_new passes to glShaderSource — injected header (render.c:315-327) + glsl_ext
    output — preprocesses to the same token stream as the interpreter's own pipeline (header_macros + ext_process) for the
    same file: module stages in order, then util/smooth_pass, gravity_pass, average_pass, pass.  Stages that `#error
    __disablestage` do so on both sides."""
    from oracle import glsl_interp as gi
    r = rd_live([REF_SHADERS], requests=[f"mod {module}"])
    try:
        frags = r.sources[0::2]                                            # a raw vertex shader follows every fragment shader
        avg = r.cfg["avg_frames"]                                          # 5 from smooth_parameters.glsl; wave never reads it: 6
        assert avg == (6 if module == "wave" else 5)
        files = []
        k = 1
        while os.path.exists(os.path.join(REF_SHADERS, module, f"{k}.frag")):
            files.append(os.path.join(REF_SHADERS, module, f"{k}.frag")); k += 1
        files += [os.path.join(REF_SHADERS, "util", f) for f in ("smooth_pass.frag", "gravity_pass.frag", "average_pass.frag", "pass.frag")]
        assert len(frags) == len(files), (len(frags), files)
        for path, real in zip(files, frags):
            def tokens(lines, predefine):
                pp = gi.Preprocessor()
                if predefine:
                    gi.header_macros(pp, avg_frames=avg)
                try:
                    return [t for t in pp.run(lines) if t[1] not in ("#",)]
                except gi.DisabledStage:
                    return "disabled"
            cd = os.path.dirname(path)
            mine = tokens(gi.ext_process(path, gi.ExtCtx(cd, REF_SHADERS, REF_SHADERS, {"_AVG_FRAMES": avg}, fallback=REF_SHADERS)), True)
            theirs = tokens(gi._strip_comments(real).split("\n"), False)
            if mine == "disabled" or theirs == "disabled":
                assert mine == theirs, path
                continue
            # the real header declares `uniform <type> STDIN;` inside `#if USE_STDIN == 1` (inactive) and nothing else beyond macros
            assert mine == theirs, (path, next((i, a, b) for i, (a, b) in enumerate(zip(mine, theirs)) if a != b))
    finally:
        r.close()


def test_pipe_line_parser_against_the_one_inside_rd_update(request, built):
    """the `--pipe` stdin parser is part of rd_update (render.c:1846-2005): the real one gets a pipe as stdin and one line per
    frame (oracle/ref_pipe_driver.py, a subprocess); the uniform writes it makes are what glava_b200_pipe_feed must store"""
    import json
    import subprocess
    import sys
    binds = [["fg", "vec4"], ["bg", "vec4"], ["amp", "float"], ["on", "bool"], ["k", "int"], ["p2", "vec2"], ["p3", "vec3"]]
    lines = ["fg = #ff8000", "  bg=#10203040   ", "fg = 0.5, 0.25,1,0.75", "#0xabcdef", "a = 3.5", "= #000000ff", "on = true", "on = 0",
             "on = TRUE", "on = False", "on = maybe", "k = 42abc", "k = -7", "p2 = 1.5,2.5", "p2 = 9", "p3 = 1,2,3", "p3 = 4", "nope = 1",
             "fg =   ", "bg = #12x456", "amp = 1e3", "amp=-0.125", "f = 1,2", "b = #80", "bg = #123", "0.1,0.2,0.3,0.4", "amp = abc",
             "p = 7,8", "fg=#FFFFFFFF", "k=0x10", "on=1"]
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def driver(binds, lines):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_pipe_driver.py"),
                              json.dumps({"shaders": REF_SHADERS, "binds": binds, "lines": lines})], capture_output=True, text=True, timeout=120)
        assert out.returncode == 0, out.stderr[-2000:]
        return json.loads(next(ln for ln in out.stdout.splitlines() if ln.startswith("RESULT "))[7:])
    ref = Session(request, _live()).call("pipe_driver", driver, (binds, lines))
    assert len(ref) == len(lines)
    with g.Pipe([f"{n}:{t}" for n, t in binds]) as pipe:
        width = {"vec4": 4, "vec3": 3, "vec2": 2, "float": 1}
        for line, writes in zip(lines, ref):
            before = pipe.binds()
            changed = pipe.feed(line + "\n")
            after = pipe.binds()
            assert changed == (1 if writes else 0), (line, writes)
            for name, (typ, val) in after.items():
                hit = [w for w in writes if w[0] == name]
                if not hit:
                    assert val == before[name][1], (line, name)          # untouched by this line
                    continue
                _, count, vals = hit[0]
                if typ in ("bool", "int"):
                    assert count == -1 and val[0] == vals[0], (line, name, val, vals)
                else:
                    assert count == width[typ] and list(val[:count]) == [np.float32(v) for v in vals[:count]], (line, name, val, vals)


@pytest.mark.parametrize("args,ours", [
    (["--pipe=1abc"], lambda: g.Pipe(["1abc"])), (["--pipe=a-b"], lambda: g.Pipe(["a-b"])), (["--pipe=:vec4"], lambda: g.Pipe([":vec4"])),
    (["--pipe=x:mat4"], lambda: g.Pipe(["x:mat4"])), (["--pipe=fg", "--pipe=fg:float"], lambda: g.Pipe(["fg", "fg:float"])),
    (["--audio=nope"], lambda: __import__("glava_b200").audio.find_backend("nope")),
])
def test_argument_errors_word_for_word(request, built, args, ours):
    """what the reference's glava_entry prints when it rejects `--pipe NAME[:TYPE]` / `--audio NAME` is what the library
    reports for the same argument"""
    import subprocess
    import sys
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def driver(args):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_entry_driver.py")] + args, capture_output=True, text=True, timeout=60)
        return [out.stderr.strip(), out.returncode]
    theirs, rc = Session(request, _live()).call("entry_driver", driver, (args,))
    assert theirs and rc != 0
    with pytest.raises(g.GlavaError) as e:
        ours()
    assert str(e.value).strip() == theirs


@pytest.mark.parametrize("mirror", [False, True])
def test_whole_program_fifo_to_uploads(rd_live, orc, tmp_path, mirror):
    """The whole reference program — glava_entry's argument parsing, rd_new, fifo.c's audio thread on a real named pipe, the
    frame loop's locked ring copy (glava.c:523-552), rd_update with the shipped setaccelfft — on the null driver for half a
    second (oracle/ref_program_driver.py).  Every frame that saw new audio uploads transform_fft of the rings as they stood;
    the oracle's FIFO ingest + transform_fft over the same bytes must reproduce those uploads bit for bit, in order, for both
    channels.  (Frames without new audio re-transform their buffer in place — the reference's own artefact — and are ignored.)"""
    import json
    import subprocess
    import sys
    n, samplesz, nchunks = 4096, 1024, 12                                # 16 hops per ring: the chunks stay visible for 16 slides
    hop = samplesz // 4
    cfg = tmp_path / "cfg" / "glava"
    cfg.parent.mkdir()
    fifo = str(tmp_path / "audio.fifo")
    os.mkfifo(fifo)
    _user_dir(cfg, {"rc.glsl": f'#request mod bars\n#request setbufsize {n}\n#request setsamplesize {samplesz}\n#request setsource "{fifo}"\n'
                               "#request setprintframes false\n#request setframerate 0\n" + ("#request setmirror true\n" if mirror else "")})
    rng = np.random.default_rng(3)
    chunks = rng.integers(-20000, 20000, size=(nchunks, hop * 2), dtype=np.int16)
    np.save(tmp_path / "chunks.npy", chunks)
    log = str(tmp_path / "uploads.bin")
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = dict(config_home=str(tmp_path / "cfg"), fifo=fifo, chunks_file=str(tmp_path / "chunks.npy"), run_ms=500, log=log, hold=0.4)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_program_driver.py"), json.dumps(spec)],
                         capture_output=True, text=True, timeout=120)
    assert "DONE 0" in out.stdout, out.stderr[-2000:]
    raw = open(log, "rb").read()
    recs, off = [], 0
    while off < len(raw):
        tex, w = np.frombuffer(raw, np.int32, 2, off); off += 8
        recs.append((int(tex), raw[off:off + 4 * int(w)])); off += 4 * int(w)
        assert w == n
    # ring states the audio thread goes through: the chunks, then zero slides once the FIFO runs dry (fifo.c:67-79)
    p = orc.default_params("bars", n=n)
    rl = np.zeros(n, np.float32); rr = np.zeros(n, np.float32)
    want = {}
    for k in range(nchunks + 3 * (n // hop)):
        orc.fifo_ingest(rl, rr, chunks[k] if k < nchunks else np.zeros(hop * 2, np.int16), 1 if mirror else 2)   # glava.c:504
        want.setdefault(orc.fft_f32(p, rl).tobytes(), ("l", k)); want.setdefault(orc.fft_f32(p, rr).tobytes(), ("r", k))
    seen = {"l": [], "r": []}
    tex_of = {}
    by_tex = {}
    for tex, data in recs:
        hit = want.get(data) if any(data) else None                        # (the silent ring's spectrum is the same for both channels)
        if hit:
            seen[hit[0]].append(hit[1]); tex_of.setdefault(hit[0], set()).add(tex)
            by_tex.setdefault(tex, []).append(hit[1])
    if mirror:
        # setmirror: fifo.c writes the integer mean of L and R into BOTH rings (fifo.c:98-102): the two audio textures get
        # the same uploads, each equal to the oracle's mono ingest
        assert np.array_equal(rl, rr) and len(by_tex) == 2
        a, b = by_tex.values()
        assert a == b and len(set(a)) >= 3 and a == sorted(a) and max(a) >= nchunks - 1
        return
    for ch in "lr":
        ks = [k for i, k in enumerate(seen[ch]) if i == 0 or k != seen[ch][i - 1]]   # (the all-zero ring recurs)
        assert len(ks) >= 3 and ks == sorted(set(ks)), (ch, ks)           # several audio frames, strictly in the audio thread's order
        assert len(tex_of[ch]) == 1                                        # always the same texture object
    assert seen["l"] == seen["r"] and tex_of["l"] != tex_of["r"]           # both channels of every frame, from the same ring state
    assert max(seen["l"]) >= nchunks - 1                                   # the last chunk made it to the screen


def test_whole_program_cpu_chain_state_by_state(rd_live, orc, tmp_path):
    """the whole program with setaccelfft false: the writer paces its chunks, so the (much faster) frame loop sees EVERY ring
    state; each distinct upload must then be the oracle's fft -> gravity -> average chain advanced by exactly one ring update —
    the next chunk, or a zero slide where fifo.c's poll timed out in between (the log tells which).  `ur` stays at rd_new's
    initialiser 1.0 on the null window's clock, so gravity falls by setgravitystep per update."""
    import json
    import subprocess
    import sys
    from oracle.oracle import OracleChannel
    n, samplesz, nchunks = 2048, 1024, 24
    hop = samplesz // 4
    cfg = tmp_path / "cfg" / "glava"
    cfg.parent.mkdir()
    fifo = str(tmp_path / "audio.fifo")
    os.mkfifo(fifo)
    _user_dir(cfg, {"rc.glsl": f'#request mod bars\n#request setbufsize {n}\n#request setsamplesize {samplesz}\n#request setsource "{fifo}"\n'
                               "#request setprintframes false\n#request setframerate 0\n#request setaccelfft false\n#request setinterpolate false\n"})
    rng = np.random.default_rng(21)
    chunks = rng.integers(-20000, 20000, size=(nchunks, hop * 2), dtype=np.int16)
    np.save(tmp_path / "chunks.npy", chunks)
    log = str(tmp_path / "uploads.bin")
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = dict(config_home=str(tmp_path / "cfg"), fifo=fifo, chunks_file=str(tmp_path / "chunks.npy"), run_ms=600, log=log, hold=1.5, pace_ms=8)
    # (hold > run: once the writer exits, fifo.c spins on POLLHUP re-sliding its stale read buffer — not part of this check)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_program_driver.py"), json.dumps(spec)],
                         capture_output=True, text=True, timeout=120)
    assert "DONE 0" in out.stdout, out.stderr[-2000:]
    raw = open(log, "rb").read()
    per_tex, off = {}, 0
    while off < len(raw):
        tex, w = np.frombuffer(raw, np.int32, 2, off); off += 8
        per_tex.setdefault(int(tex), []).append(np.frombuffer(raw, np.float32, int(w), off).copy()); off += 4 * int(w)
    assert len(per_tex) == 2
    p = orc.default_params("bars", n=n, accel_fft=0, smooth_pass=0, avg_frames=5, ur=1.0)
    zero = np.zeros(hop * 2, np.int16)
    matched_channels = 0
    for uploads in per_tex.values():
        for side in (0, 1):                                                # which ring this texture shows
            ring = [np.zeros(n, np.float32), np.zeros(n, np.float32)]
            ch = OracleChannel(orc, p)
            nxt, steps, ok = 0, 0, True
            # leading records: the never-initialised lb of glava.c:487-490 until the first ring update arrives
            start = next((i for i, u in enumerate(uploads) if _step_matches(orc, p, ring, chunks[0], side, u)), None)
            if start is None:
                continue
            for u in uploads[start:]:
                # one ring update per logged upload as a rule; two when the frame loop was held up for a moment (it then
                # transforms only the later state — the earlier one never reaches gravity / average, here neither)
                singles = ([("c", 1)] if nxt < nchunks else []) + [("z", 0)]
                doubles = [a + b for a in ("c", "z") for b in ("c", "z")]
                hit = None
                for seq in [t[0] for t in singles] + doubles:
                    r2 = [ring[0].copy(), ring[1].copy()]
                    k = nxt
                    if seq.count("c") > nchunks - nxt:
                        continue
                    for step in seq:
                        orc.fifo_ingest(r2[0], r2[1], chunks[k] if step == "c" else zero, 2)
                        k += step == "c"
                    if np.array_equal(_replay(orc, p, getattr(ch, "_log", []), r2[side]), u):
                        hit = (seq, r2, k)
                        break
                if hit is None:
                    ok = False
                    break
                ring, nxt = hit[1], hit[2]
                ch._log = getattr(ch, "_log", []) + [ring[side].copy()]
                steps += len(hit[0])
            if ok and steps >= nchunks and nxt == nchunks:
                matched_channels += 1
    assert matched_channels == 2                                           # one texture follows the left ring, the other the right


def _replay(orc, p, log, ring_now):
    """the chain's result after the logged ring states followed by `ring_now` (OracleChannel has no copy: replay)"""
    from oracle.oracle import OracleChannel
    ch = OracleChannel(orc, p)
    out = None
    for state in list(log) + [ring_now]:
        out, _ = ch.update(state)
    return out


def _step_matches(orc, p, ring, chunk, side, upload):
    r2 = [ring[0].copy(), ring[1].copy()]
    orc.fifo_ingest(r2[0], r2[1], chunk, 2)
    return np.array_equal(_replay(orc, p, [], r2[side]), upload)
