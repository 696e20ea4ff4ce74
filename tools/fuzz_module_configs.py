"""Randomised differential over the module option space (test infrastructure; needs the reference tree).

For every seed: a random user <module>.glsl (integer AND float spellings of the numeric macros, #rrggbb / #rrggbbaa / vec4
colours, every option flag), sometimes `setopacity "none"` with a random `setbgf`, sometimes `setmirror`.  The SAME text goes
  (a) through the reference's own module shaders in oracle/glsl_interp.py (what GLava would render),
  (b) through the product's config reader -> parameters -> the C oracle, and
  (c) through the config reader -> the host build of the product's raster arithmetic (tests/emul).
(a) == (b) must hold exactly; (c) within 1 LSB on a handful of pixels (the product's own sin / atan / log polynomials).

    python tools/fuzz_module_configs.py 0 200        # seeds [0, 200)

Found with it: circle/2.frag is a pass-through, not a disabled stage, when C_SMOOTH is 0 (one more blend in non-native
opacity), and setsmoothfactor reaches the shaders as the "%.6f" literal of the injected header.
tests/test_module_config_fuzz.py runs a fixed slice of seeds in the CPU tier."""
import os
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import glava_b200 as g
from oracle import glsl_interp as gi
from oracle.oracle import Oracle, params_from
from tests import emul
REF="/root/reference/shaders/glava"
orc=Oracle("libm")

def num(rng, lo, hi, int_ok=True):
    if int_ok and rng.random()<0.5: return str(int(rng.integers(int(np.ceil(lo)), int(hi)+1)))
    return "%.2f" % rng.uniform(lo,hi)
def col(rng):
    k=rng.integers(0,3)
    if k==0: return "#%06x" % int(rng.integers(0,1<<24))
    if k==1: return "#%08x" % int(rng.integers(0,1<<32))
    return "vec4(%.2f, %.2f, %.2f, %.2f)" % tuple(rng.uniform(0,1,4))
def gen(rng, module):
    L=[]
    D=lambda k,v: L.append(f"#define {k} {v}")
    if module=="bars":
        # BAR_OUTLINE_WIDTH is tested in `#if BAR_OUTLINE_WIDTH > 0` (bars/1.frag:116): integers only compile; the same draw
        # as before is consumed (so the other macros of a seed stay what they were) and its integer part is kept
        D("BAR_WIDTH", num(rng,1,6)); D("BAR_GAP", num(rng,0,3)); D("BAR_OUTLINE_WIDTH", str(int(float(num(rng,0,2))))); D("AMPLIFY", num(rng,10,40))
        D("GRADIENT", num(rng,5,40)); D("COLOR", f"mix({col(rng)}, {col(rng)}, clamp(d / GRADIENT, 0, 1))")
        if rng.random()<0.5: D("BAR_OUTLINE", col(rng))
        for k in ("DIRECTION","INVERT","FLIP","MIRROR_YX"): D(k, int(rng.integers(0,2)))
    if module=="radial":
        D("C_RADIUS", num(rng,4,10)); D("C_LINE", num(rng,1,4)); D("OUTLINE", col(rng)); D("NBARS", int(rng.integers(4,30))*2)
        D("BAR_WIDTH", num(rng,1,5)); D("AMPLIFY", num(rng,8,25)); D("GRADIENT", num(rng,4,20))
        D("COLOR", f"mix({col(rng)}, {col(rng)}, clamp(d / GRADIENT, 0, 1))"); D("ROTATE", rng.choice(["(PI / 2)","0","1.3","(TWOPI / 5)"]))
        D("INVERT", int(rng.integers(0,2))); D("BAR_ALIAS_FACTOR", num(rng,0.5,2,False)); D("C_ALIAS_FACTOR", num(rng,0.5,2.5,False))
        D("CENTER_OFFSET_X", num(rng,-4,4)); D("CENTER_OFFSET_Y", num(rng,-3,3)); D("BAR_OUTLINE_WIDTH", (lambda c: {"0.5": "1"}.get(c, c))(str(rng.choice(["0","0","1","0.5"]))))   # (`#if BAR_OUTLINE_WIDTH > 0`, radial/1.frag:87: integers only)
    if module=="circle":
        D("C_RADIUS", num(rng,4,10)); D("C_LINE", num(rng,1,3)); D("OUTLINE", col(rng)); D("AMPLIFY", num(rng,5,20))
        D("ROTATE", rng.choice(["(PI / 2)","0","2.1"])); D("INVERT", int(rng.integers(0,2))); D("C_FILL", int(rng.integers(0,2))); D("C_SMOOTH", int(rng.integers(0,2)))
    if module=="graph":
        D("VSCALE", num(rng,10,40)); D("DIRECTION", rng.choice(["1","-1"])); D("GRADIENT", num(rng,5,30))
        D("COLOR", f"mix({col(rng)}, {col(rng)}, clamp(pos / GRADIENT, 0, 1))")
        for k in ("DRAW_OUTLINE","DRAW_HIGHLIGHT","ANTI_ALIAS","INVERT"): D(k, int(rng.integers(0,2)))
        D("JOIN_CHANNELS", int(rng.random()<0.25)); D("OUTLINE", col(rng))
    if module=="wave":
        D("MIN_THICKNESS", num(rng,1,2)); D("MAX_THICKNESS", num(rng,2,6)); D("BASE_COLOR", col(rng)); D("AMPLIFY", num(rng,10,60)); D("OUTLINE", col(rng))
    return "\n".join(L)+"\n"

def shader_frame(d, module, w, h, tl, tr, clear, hdr):
    """the frame the reference's module shaders draw with user config dir d, run by the interpreter"""
    prog=gi.ModuleProgram(REF, module, w, h, tl, tr, config_dir=d, clear_color=clear, **hdr)
    return np.array([[prog.pixel(x,y) for x in range(w)] for y in range(h)],np.uint8)

def run(seed, module, w, h, n=128, native=True, smooth_in_shader=False, config_tail=REF, frame=shader_frame):
    """config_tail: the directory the reader falls back to after the user's; frame: shader_frame or a stand-in with its
    arguments and result"""
    rng=np.random.default_rng(seed)
    text=gen(rng, module)
    d=tempfile.mkdtemp()
    rc=f"#request mod {module}\n#request setbufsize 256\n#request setgeometry 0 0 {w} {h}\n"
    clear=(0,0,0,0)
    if not native:
        clear=tuple(float(np.float32(v)) for v in rng.uniform(0,1,4))
        rc+='#request setopacity "none"\n#request setbgf %r %r %r %r\n' % clear
    if rng.random()<0.3: rc+="#request setmirror true\n"
    hdr_extra = {}
    want_state = None
    if smooth_in_shader:
        # setsmoothpass and the module's belief about its textures.  The stage-1 header (`_PRE_SMOOTHED_AUDIO`) is built from
        # smooth_pass as of the end of rc.glsl, BEFORE the shader's own includes run smooth_parameters.glsl's requests
        # (render.c:284-293 vs :312), while the K5 pass follows the final value:
        #   variant 0  false in rc.glsl and in smooth_parameters.glsl -> shader smooths the raw texture itself   (0, 0)
        #   variant 1  false only in smooth_parameters.glsl           -> shader believes "smoothed", K5 is off   (0, 1)
        #   variant 2  false only in rc.glsl                          -> K5 runs AND the shader smooths again    (1, 2)
        variant = int(smooth_in_shader) - 1 if smooth_in_shader is not True else 0
        sf = float(np.float32(rng.uniform(0.01, 0.05)))
        final = "true" if variant == 2 else "false"
        sp = "#request setsmoothpass %s\n#request setsmoothfactor %r\n" % (final, sf)
        sp += "#define SAMPLE_MODE %s\n#define ROUND_FORMULA %s\n" % (rng.choice(["average", "maximum", "hybrid"]), rng.choice(["sinusoidal", "linear", "circular"]))
        sp += "#define SAMPLE_SCALE %s\n#define SAMPLE_RANGE %s\n#define SAMPLE_HYBRID_WEIGHT %s\n" % (num(rng, 4, 10), num(rng, 0.5, 0.95, False), num(rng, 0.3, 0.9, False))
        open(d+"/smooth_parameters.glsl","w").write(sp)
        if variant != 1: rc += "#request setsmoothpass false\n"
        hdr_extra = dict(pre_smoothed=1 if variant == 1 else 0, smooth_factor=sf)
        want_state = [(0, 0), (0, 1), (1, 2)][variant]
    open(d+"/rc.glsl","w").write(rc); open(f"{d}/{module}.glsl","w").write(text)
    p=g.load_config([d, config_tail])
    n=p.n
    op=params_from(p)
    if smooth_in_shader and want_state != (1, 2):
        tl=(rng.random(n)**2*65535).astype(np.uint16); tr=(rng.random(n)**3*65535).astype(np.uint16)
    else:
        tl=orc.smooth_pass(op,(rng.random(n)**2*65535).astype(np.uint16)); tr=orc.smooth_pass(op,(rng.random(n)**3*65535).astype(np.uint16))
    if module=="wave": tl=np.clip(tl.astype(int)//4+24576,0,65535).astype(np.uint16)
    hdr=dict(premultiply_alpha=p.premultiply_alpha, channels=p.channels, **hdr_extra)
    assert (p.smooth_pass, p.shader_pre_smoothed) == (want_state or (1, 0)), (p.smooth_pass, p.shader_pre_smoothed, want_state)
    want=frame(d, module, w, h, tl, tr, clear, hdr)
    o=orc.raster(op,tl,tr); e=emul.raster(p,tl,tr)
    return text, want, o, e

if __name__=="__main__":
    bad=0; t0=time.time()
    for seed in range(int(sys.argv[1]), int(sys.argv[2])):
        module=["bars","radial","circle","graph","wave"][seed%5]
        w,h=[(40,28),(41,27),(38,30)][seed%3]
        try:
            text,want,o,e=run(seed,module,w,h,native=(seed%4!=3),smooth_in_shader=((1 + seed // 7 % 3) if (seed%7==5 and module in ('bars','radial','circle','graph')) else False))
        except Exception as ex:
            print(seed,module,"EXC",repr(ex)[:300]); bad+=1; continue
        do=(o!=want).any(axis=2).sum(); de=(e!=want).any(axis=2).sum(); lsb=int(np.abs(e.astype(int)-want.astype(int)).max())
        flag = "" if do==0 and lsb<=1 and de<=0.005*w*h else "  <<<<<<"
        if flag: bad+=1
        print(seed,module,(w,h),"oracle!=shader:",do,"product!=shader:",de,"lsb",lsb,flag, flush=True)
        if flag: print(text)
    print("bad",bad,"time",time.time()-t0)
