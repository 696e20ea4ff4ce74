"""The reference's OWN source extension (glava/glsl_ext.c, compiled where it lies into oracle/_ref/libglava_ref.so) run on
real text, against (a) the interpreter's restatement of it — the front end of every shader-derived golden frame — and
(b) the product's config reader: `#request` tokenising and typed argument conversion, `#include` with the ':' / '@'
directory rules, `#rrggbb[aa]` literals, `@name:default` binds, and what counts as a parse error."""
import os
import re

import numpy as np
import pytest

import glava_b200 as g

REF_SHADERS = "/root/reference/shaders/glava"


def _auto_undef_removed(text):
    """glsl_ext.c:143-159 puts `#ifdef X / #undef X / #endif` + a #line in front of every #define; the interpreter's
    preprocessor lets a later #define override instead.  Hand-written #undef blocks of the shaders stay."""
    text = re.sub(r"#ifdef (\w+)\n#undef \1\n#endif\n\n#line \d+ \d+\n(?=#define \1\b)", "", text)
    return "\n".join(ln for ln in text.split("\n") if not ln.startswith("#line"))


@pytest.mark.skipif(not os.path.isdir(REF_SHADERS), reason="reference tree not present")
def test_interpreter_front_end_is_token_identical_to_glsl_ext_c(ref_live, built):
    ref = ref_live
    import glob
    from oracle import glsl_interp as gi
    files = sorted(glob.glob(REF_SHADERS + "/*/*.frag"))
    assert len(files) >= 20
    for f in files:
        cd = os.path.dirname(f)
        real, _ = ref.ext_process(f, cd, REF_SHADERS, REF_SHADERS)
        mine = "\n".join(gi.ext_process(f, gi.ExtCtx(cd, REF_SHADERS, REF_SHADERS, {"_AVG_FRAMES": 5}, fallback=REF_SHADERS)))
        a = gi.tokenize(gi._strip_comments(_auto_undef_removed(real))); b = gi.tokenize(mine)
        assert a == b, (f, next(i for i, (x, y) in enumerate(zip(a, b)) if x != y))


@pytest.mark.skipif(not os.path.isdir(REF_SHADERS), reason="reference tree not present")
def test_shipped_rc_requests_as_the_reference_parses_them(ref_live, built):
    ref = ref_live
    _, reqs = ref.ext_process(REF_SHADERS + "/rc.glsl", REF_SHADERS, None, REF_SHADERS)
    got = {r[0]: r[1:] for r in reqs}
    p = g.load_config([REF_SHADERS])
    assert got["mod"] == [p.module_name] and got["setbufsize"] == [str(p.n)] and got["setgeometry"][2:] == [str(p.w), str(p.h)]
    assert got["setopacity"] == ["native"] and p.premultiply_alpha == 1 and got["setmirror"] == [str(2 - p.channels)]
    assert got["setsamplerate"] == [str(p.rate_request)] and got["setsamplesize"] == [str(p.samplesize_request)]
    assert got["setaccelfft"] == [str(p.accel_fft)] and got["setinterpolate"] == [str(p.interpolate)] and got["setbufscale"] == [str(p.bufscale)]
    # smooth_parameters.glsl is read through the module shader's `#include "@..."` / `":..."` pair
    _, reqs = ref.ext_process(REF_SHADERS + "/bars/1.frag", REF_SHADERS + "/bars", REF_SHADERS, REF_SHADERS)
    got = {r[0]: r[1:] for r in reqs if r[0].startswith("set")}
    assert np.float32(got["setfftscale"][0]) == p.fft_scale and np.float32(got["setfftcutoff"][0]) == p.fft_cutoff
    assert np.float32(got["setgravitystep"][0]) == p.gravity_step and np.float32(got["setsmoothfactor"][0]) == p.smooth_factor
    assert got["setavgframes"] == [str(p.avg_frames)] and got["setavgwindow"] == [str(p.avg_window)] and got["setsmoothpass"] == [str(p.smooth_pass)]


RC = """
#request mod radial
#request setbufsize 0x800
#request setgeometry 10 20 640 360
#request setopacity "none"
#request setbg 10203040
#request setmirror t
#request setsamplerate 44100
#request setsamplesize 0400
#request setaccelfft 0
#request setinterpolate f
#include "extra.glsl"
#request setbgf 0.25 .5 75e-2 1
"""
EXTRA = """
/* a comment with #request setbufsize 512 inside */
#request setfftscale 1.25e1
#request setfftcutoff  0.5    // trailing comment
#request setavgframes 0x7
#request setavgwindow false
#request setgravitystep 3
#request setsmoothfactor .0625
#request setsmoothpass 1
#request settitle "a title with spaces"
"""


def test_request_tokenising_and_typed_arguments(ref, tmp_path, built):
    (tmp_path / "rc.glsl").write_text(RC); (tmp_path / "extra.glsl").write_text(EXTRA)
    _, reqs = ref.ext_process(str(tmp_path / "rc.glsl"), str(tmp_path), None, str(tmp_path))
    got = {}
    for r in reqs:
        got[r[0]] = r[1:]                                                 # a later request overrides
    p = g.load_config([str(tmp_path)])
    assert got["mod"] == ["radial"] == [p.module_name]
    assert int(got["setbufsize"][0]) == p.n == 2048                       # strtol(.., 0): hex, and 0400 is octal 256
    assert [int(v) for v in got["setgeometry"][2:]] == [p.w, p.h] == [640, 360]
    assert got["setopacity"] == ["none"] and p.premultiply_alpha == 0
    assert int(got["setmirror"][0]) == 1 and p.channels == 1
    assert int(got["setsamplerate"][0]) == p.rate_request and int(got["setsamplesize"][0]) == p.samplesize_request == 256
    assert int(got["setaccelfft"][0]) == p.accel_fft == 0 and int(got["setinterpolate"][0]) == p.interpolate == 0
    for name, field in (("setfftscale", "fft_scale"), ("setfftcutoff", "fft_cutoff"), ("setgravitystep", "gravity_step"),
                        ("setsmoothfactor", "smooth_factor")):
        assert np.float32(got[name][0]) == getattr(p, field), name
    assert int(got["setavgframes"][0]) == p.avg_frames == 7 and int(got["setavgwindow"][0]) == p.avg_window == 0
    assert got["settitle"] == ["a title with spaces"]
    assert [np.float32(v) for v in got["setbgf"]] == list(p.clear_color)  # setbgf after setbg wins
    assert "512" not in [a for r in reqs for a in r]                      # the commented-out request is not one


@pytest.mark.parametrize("line", ["#request setavgwindow maybe", "#request frobnicate 1", "#request setgeometry 1 2 3",
                                  '#include "missing.glsl"'])
def test_what_the_reference_rejects_the_reader_rejects(ref, tmp_path, line, built):
    (tmp_path / "rc.glsl").write_text("#request mod bars\n" + line + "\n")
    with pytest.raises(ValueError):
        ref.ext_process(str(tmp_path / "rc.glsl"), str(tmp_path), None, str(tmp_path))
    with pytest.raises(g.GlavaError):
        g.load_config([str(tmp_path)])


MODULE = """
#define GRADIENT (20 + 20)
#define COLOR @fg:mix(#3366b2, #A0a0B2ff, clamp(d / GRADIENT, 0, 1))
/* (a bound `@name:f(...)` swallows its line's newline in glsl_ext.c, so — as in the shipped configs — a comment line follows) */
#define BAR_OUTLINE @bg:#20c04080
#define AMPLIFY 123
"""


def test_colour_literals_and_binds_as_the_reference_rewrites_them(ref, tmp_path, built):
    (tmp_path / "rc.glsl").write_text("#request mod bars\n"); (tmp_path / "bars.glsl").write_text(MODULE)
    text, _ = ref.ext_process(str(tmp_path / "bars.glsl"), str(tmp_path), None, str(tmp_path))
    colour = re.search(r"#define COLOR (.*)", text).group(1)
    lits = [[float(v) for v in m] for m in re.findall(r"vec4\(([\d.]+), ([\d.]+), ([\d.]+), ([\d.]+)\)", colour)]
    assert "@" not in colour and len(lits) == 2                            # unbound: the default, literals as "%.6f" decimals
    p = g.load_config([str(tmp_path)])
    assert p.bars_color.mode == 0 and p.bars_color.gradient == 40
    assert [np.float32(v) for v in lits[0]] == list(p.bars_color.lo) and [np.float32(v) for v in lits[1]] == list(p.bars_color.hi)
    outl = [np.float32(v) for v in re.search(r"#define BAR_OUTLINE\s+vec4\(([^)]*)\)", text).group(1).split(",")]
    assert p.bars_outline_mode == 1 and outl == list(p.bars_outline)
    # bound: the macro becomes the uniform `_IN_name` (glsl_ext.c:571-576); the reader substitutes the bind's value
    text, _ = ref.ext_process(str(tmp_path / "bars.glsl"), str(tmp_path), None, str(tmp_path), binds=["fg"])
    assert re.search(r"#define COLOR\s+_IN_fg\b", text) and "_IN_bg" not in text and "mix" not in text
    q = g.load_config([str(tmp_path)], binds={"fg": "vec4(0.5, 0.25, 0.125, 1)"})
    assert q.bars_color.mode == 1 and list(q.bars_color.lo) == [0.5, 0.25, 0.125, 1.0] and list(q.bars_outline) == outl


def test_include_directory_rules(ref, tmp_path, built):
    """':' switches to the config dir, '@' to the defaults dir, and the switch sticks for the rest of the file"""
    user, sysd = tmp_path / "user", tmp_path / "sys"
    user.mkdir(); sysd.mkdir()
    (user / "rc.glsl").write_text('#request mod bars\n#include "@part.glsl"\n#include "next.glsl"\n#include ":part.glsl"\n')
    (sysd / "part.glsl").write_text("#request setbufsize 1024\n"); (sysd / "next.glsl").write_text("#request setavgframes 3\n")
    (user / "part.glsl").write_text("#request setbufsize 2048\n"); (user / "next.glsl").write_text("#request setavgframes 9\n")
    _, reqs = ref.ext_process(str(user / "rc.glsl"), str(user), str(user), str(sysd))
    assert [r for r in reqs if r[0] != "mod"] == [["setbufsize", "1024"], ["setavgframes", "3"], ["setbufsize", "2048"]]
    # rc.glsl itself is read without a config / defaults dir (render.c:1356-1361): '@' is an error there, ':' is inert
    with pytest.raises(ValueError):
        ref.ext_process(str(user / "rc.glsl"), str(user), None, None or str(user) + "/nonexistent")


def test_requests_inside_a_dead_conditional_still_run(ref, tmp_path, built):
    """glsl_ext.c does not evaluate #if / #ifdef: a `#request` acts wherever it stands; only the #defines are the GLSL
    compiler's to select — the config reader follows both halves"""
    (tmp_path / "rc.glsl").write_text("#request mod graph\n")
    (tmp_path / "graph.glsl").write_text("#ifdef NOPE\n#request setavgframes 9\n#define VSCALE 77\n#endif\n#if 0\n#request setgravitystep 2.5\n#endif\n")
    text, reqs = ref.ext_process(str(tmp_path / "graph.glsl"), str(tmp_path), None, str(tmp_path))
    assert ["setavgframes", "9"] in reqs and ["setgravitystep", "2.5"] in reqs and "#ifdef NOPE" in text
    p = g.load_config([str(tmp_path)])
    assert p.avg_frames == 9 and p.gravity_step == 2.5 and p.graph_vscale == 300
