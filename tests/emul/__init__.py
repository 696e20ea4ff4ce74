"""TEST INFRASTRUCTURE — host emulation of the CUDA kernels' arithmetic (see emul.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def lib():
    global _lib
    if _lib is None:
        so = os.path.join(HERE, "libglava_emul.so")
        src = os.path.join(HERE, "emul.cpp")
        csrc = os.path.join(HERE, "..", "..", "glava_b200", "csrc")
        newest = max(os.path.getmtime(os.path.join(csrc, f)) for f in os.listdir(csrc) if f.endswith(".h"))
        if not os.path.exists(so) or os.path.getmtime(so) < max(newest, os.path.getmtime(src)):
            subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas",
                            "-o", so, src], check=True)
        L = C.CDLL(so)
        vp, i32 = C.c_void_p, C.c_int
        L.emul_fft.argtypes = [i32, vp, vp, C.c_float, C.c_float]
        L.emul_chan_new.restype = vp
        L.emul_chan_new.argtypes = [vp]
        L.emul_chan_free.argtypes = [vp]
        L.emul_chan_update.argtypes = [vp, vp, vp, i32, vp, vp]
        L.emul_smooth.argtypes = [vp, vp, vp]
        L.emul_raster.argtypes = [vp, vp, vp, vp, i32, i32]
        L.emul_raster_fast.argtypes = [vp, vp, vp, vp]
        L.emul_eval_color.argtypes = [vp, C.c_float, vp]
        L.emul_lazy_k5.argtypes = [vp, i32, i32, vp, vp, vp]
        L.emul_lazy_epi_n.argtypes = [vp]
        L.emul_k5_table.argtypes = [vp, vp, vp]
        L.emul_table_sizes.argtypes = [vp, i32, i32, vp]
        L.emul_bufscale.argtypes = [vp, i32, i32, vp]
        L.emul_transform_smooth.argtypes = [vp, i32, C.c_float, C.c_float]
        L.emul_upload.argtypes = [vp, vp, i32, C.c_float, C.c_float, i32, vp]
        _lib = L
    return _lib


def fft(pcm, fft_scale=10.2, fft_cutoff=0.3):
    x = np.ascontiguousarray(pcm, dtype=np.float32)
    out = np.empty_like(x)
    assert lib().emul_fft(x.shape[0], x.ctypes.data, out.ctypes.data, fft_scale, fft_cutoff) == 0
    return out


class Channel:
    def __init__(self, params):
        self.p = params
        self.h = lib().emul_chan_new(C.addressof(params))

    def update(self, pcm, is_fft=True):
        x = np.ascontiguousarray(pcm, dtype=np.float32)
        spec = np.empty(self.p.n, np.float32); tex = np.empty(self.p.n, np.uint16)
        assert lib().emul_chan_update(self.h, C.addressof(self.p), x.ctypes.data, 1 if is_fft else 0,
                                      spec.ctypes.data, tex.ctypes.data) == 0
        return spec, tex

    def __del__(self):
        try: lib().emul_chan_free(self.h)
        except Exception: pass


def smooth(params, tex):
    t = np.ascontiguousarray(tex, dtype=np.uint16)
    out = np.empty_like(t)
    lib().emul_smooth(C.addressof(params), t.ctypes.data, out.ctypes.data)
    return out


def raster(params, tex_l, tex_r, fast=False):
    tl = np.ascontiguousarray(tex_l, dtype=np.uint16)
    tr = np.ascontiguousarray(tex_r if tex_r is not None else tex_l, dtype=np.uint16)
    out = np.zeros((params.h, params.w, 4), dtype=np.uint8)
    if fast:
        assert lib().emul_raster_fast(C.addressof(params), tl.ctypes.data, tr.ctypes.data, out.ctypes.data) == 0
    else:
        lib().emul_raster(C.addressof(params), tl.ctypes.data, tr.ctypes.data, out.ctypes.data, 0, params.h)
    return out


def bufscale(pcm, k):
    x = np.ascontiguousarray(pcm, dtype=np.float32)
    out = np.empty(x.shape[0] // k, np.float32)
    lib().emul_bufscale(x.ctypes.data, x.shape[0], k, out.ctypes.data)
    return out


def transform_smooth(buf, smooth_distance=0.01, smooth_ratio=4.0):
    b = np.array(buf, dtype=np.float32, copy=True)
    lib().emul_transform_smooth(b.ctypes.data, b.shape[0], smooth_distance, smooth_ratio)
    return b


def upload(start, end, ur, fr, kcounter):
    s = np.ascontiguousarray(start, dtype=np.float32)
    e = None if end is None else np.ascontiguousarray(end, dtype=np.float32)
    out = np.empty(s.shape[0], np.uint16)
    lib().emul_upload(s.ctypes.data, None if e is None else e.ctypes.data, s.shape[0], ur, fr, kcounter, out.ctypes.data)
    return out


def lazy_k5(p, chan, path, av):
    """(texel indices, values) of the need-list texels of channel `chan`, through the tap-major table (path 0) or the
    texel-major blob (path 1)"""
    av = np.ascontiguousarray(av, dtype=np.uint16)
    out = np.zeros(p.n, np.uint16); need = np.zeros(p.n, np.int32)
    cnt = lib().emul_lazy_k5(C.byref(p), chan, path, av.ctypes.data, out.ctypes.data, need.ctypes.data)
    if cnt < -1:
        raise AssertionError(f"blocks-of-texels walk: error {cnt} (emul.cpp emul_lazy_k5)")
    if cnt < 0:
        return None, None
    idx = need[:cnt].copy()
    return idx, out[idx]


def lazy_epi_n(p):
    return lib().emul_lazy_epi_n(C.byref(p))


def table_sizes(p, target_rows=-105, texels_per_block=16):
    """host table sizes the K5 launch structure is chosen from (capi.cu build_tables; the block shape defaults to its
    own): dict(lazy_tab_bytes, lazy_blob_bytes, need_tile_rows, full_span, full_bytes); the lazy_* / need_* entries are
    None for a module without a need-list"""
    out = np.zeros(5, np.int64)
    rc = lib().emul_table_sizes(C.byref(p), target_rows, texels_per_block, out.ctypes.data)
    lazy = [int(v) for v in out[:3]] if rc == 0 else [None] * 3
    return dict(lazy_tab_bytes=lazy[0], lazy_blob_bytes=lazy[1], need_tile_rows=lazy[2], full_span=int(out[3]), full_bytes=int(out[4]))


def k5_table(p, tex):
    tex = np.ascontiguousarray(tex, dtype=np.uint16)
    out = np.empty_like(tex)
    lib().emul_k5_table(C.byref(p), tex.ctypes.data, out.ctypes.data)
    return out


def eval_color(prog, x):
    """a compiled colour expression (glava_b200.api.ColorProg) at X -> float32[4]"""
    out = np.zeros(4, np.float32)
    lib().emul_eval_color(C.byref(prog), float(x), out.ctypes.data)
    return out
