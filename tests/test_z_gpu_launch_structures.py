"""-m gpu: every launch structure of the lazy pipeline-B update (capi.cu build_tables / run_update, DESIGN 4.1a) at the batch
sizes and shapes that bench.py and tools/sweep_configs.py time, against the oracle chain.

  * persistent spectrum grid: with the K5 taps in shared memory spectrum_kernel runs 2 x SM-count CTAs, and above that many
    work units a CTA walks u, u + gridDim.x, ... with the next unit's PCM prefetched by the TMA engine (A);
  * every benchmarked shape (bench.workload() names and the sweep grid) at a batch of 2 x SM count + 37 streams (B);
  * K5 structures that a parameter set selects without any tuning knob: the L2 form of the need-list K5 (transposed copy +
    k5_need_kernel, S = 1 and S = 2), the in-kernel full-plane k5_planes_kernel, the three-kernel split below setbufsize
    4096, and SAMPLE_MODE / ROUND_FORMULA on the lazy path (C).

Which structure ran is asserted through the spectrum-side launches of one update; that the parameter sets sit on the
intended side of capi.cu's size thresholds is asserted on the host by tests/test_emul_parity.py.

Tolerances (the same as the rest of the suite): spectrum <= 1e-5 of the plane's peak up to setbufsize 4096 and 2.5e-5 above
against the oracle chain, 1e-5 against the float64 transform, over the leading epi_n bins (the three-kernel form writes only those); R16 texels at the need-list <= 2 LSB16; frames bit-exact
against the oracle's raster of the GPU's own textures and within 1 LSB of the oracle chain's frames except at most
2e-4 * w * h pixels; lazy and full K5 frames bit-identical."""
import numpy as np
import pytest

import bench
import glava_b200 as g
from oracle.oracle import OracleChannel, params_from
from tests import emul

pytestmark = pytest.mark.gpu

# spectrum-side launches of one modified update (capi.cu run_update): one kernel (taps in shared memory, or lazy_smooth = 0
# + a full-plane K5 kernel: 2), three kernels with K5 out of shared-memory tiles, four with the L2 form (transpose + K5)
ONE, FULL, TILES, L2 = 1, 2, 3, 4


def _sm():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _peak_err(got, want, peak):
    """max |got - want| over the compared bins, relative to the peak of the whole reference plane"""
    return np.abs(np.asarray(got, dtype=np.float64) - np.asarray(want, dtype=np.float64)).max() / max(float(np.abs(peak).max()), 1e-30)


_CHUNKS = {}


def _chunks(batch, steps):
    """the synthetic FIFO chunks of streams 0..batch-1 for `steps` hops (g.StreamRings.chunks), generated once per batch"""
    have = _CHUNKS.setdefault(batch, [])
    if len(have) < steps:
        rings = g.StreamRings(batch, 256)
        rings.t = 256 * len(have)
        while len(have) < steps:
            have.append(rings.chunks()); rings.t += 256
    return have[:steps]


class Run:
    """`steps` updates of one renderer through update_device / update_device_masked (the entry points bench.py times), fed
    from g.StreamRings.  Per probe stream: the oracle chain and / or a batch-1 renderer driven with that stream's own flag."""

    def __init__(self, p, batch, steps, masks=None, probes=(), orc=None, singles=False):
        import torch
        self.p, self.batch, self.fft = p, batch, p.module_name != "wave"
        op = params_from(p)
        rings = g.StreamRings(batch, p.n)
        chans = {s: [OracleChannel(orc, op), OracleChannel(orc, op)] for s in probes} if orc is not None else {}
        one = {s: g.Renderer(p, batch=1) for s in probes} if singles else {}
        self.want, self.single = {}, {}
        dl = torch.zeros((batch, p.n), device="cuda"); dr = torch.zeros_like(dl)
        self.r = g.Renderer(p, batch=batch)
        try:
            mod_launches = None
            for t, c in enumerate(_chunks(batch, steps)):
                rings.push(c)
                m = None if masks is None else masks[t]
                self.r.sync()                                    # the previous update has read dl / dr
                dl.copy_(torch.from_numpy(rings.lb)); dr.copy_(torch.from_numpy(rings.rb)); torch.cuda.synchronize()
                before = self.r.launch_count
                if m is None:
                    self.r.update_device(dl.data_ptr(), dr.data_ptr(), True)
                    mod_launches = self.r.launch_count - before
                else:
                    self.r.update_device_masked(dl.data_ptr(), dr.data_ptr(), m)
                for s in probes:
                    on = m is None or bool(m[s])
                    if s in chans and on:
                        self.want[s] = (chans[s][0].update(rings.lb[s], self.fft), chans[s][1].update(rings.rb[s], self.fft))
                    if s in one:
                        one[s].update(rings.lb[s:s + 1], rings.rb[s:s + 1], on)
            self.last_l, self.last_r = rings.lb.copy(), rings.rb.copy()
            before = self.r.launch_count
            self.r.update_device(dl.data_ptr(), dr.data_ptr(), False)     # raster only: the same frames again
            self.spec_launches = mod_launches - (self.r.launch_count - before)
            for s, q in one.items():
                self.single[s] = (q.spectrum(), q.textures(), q.readback(0))
        finally:
            for q in one.values():
                q.close()
        self.spec = self.r.spectrum(); self.tex = self.r.textures()

    def close(self):
        self.r.close()

    def holds_frame(self, s):
        slots = self.p.fb_slots if 0 < self.p.fb_slots < self.batch else self.batch
        return s >= self.batch - slots


def _need(p):
    """need-list texels of each channel (all texels where the module has no need-list)"""
    out = []
    for c in (0, 1):
        idx, _ = emul.lazy_k5(p, c, 1, np.zeros(p.n, np.uint16))
        out.append(np.arange(p.n) if idx is None else idx)
    return out


def _bands(p):
    if p.w * p.h <= 1920 * 1080:
        return [(0, p.h)]
    h = p.h
    return [(0, 6), (96, 104), (188, 200), (h // 2 - 3, h // 2 + 3), (h // 2 + 120, h // 2 + 134), (h - 5, h)]


def _check_oracle(run, orc, probes, frames=()):
    """probe streams against the oracle chain: spectrum over [:epi_n], textures at the need-list, frames (row bands at 4K / 8K)"""
    p = run.p; op = params_from(p)
    epi = emul.lazy_epi_n(p) if p.lazy_smooth else p.n
    epi = p.n if epi <= 0 else epi
    tol = 1e-5 if p.n <= 4096 else 2.5e-5
    need = _need(p)
    for s in probes:
        for c in ((0, 1) if run.fft else (0,)):
            spec_w, tex_w = run.want[s][c]
            assert _peak_err(run.spec[c][s][:epi], spec_w[:epi], spec_w) <= tol, (s, c)
            idx = need[c] if p.lazy_smooth else np.arange(p.n)
            assert np.abs(run.tex[c][s][idx].astype(int) - tex_w[idx].astype(int)).max() <= 2, (s, c)
    for s in frames:
        assert run.holds_frame(s)
        got = run.r.readback(s)
        gl, gr = run.tex[0][s], (run.tex[1][s] if run.fft else run.tex[0][s])
        wl, wr = run.want[s][0][1], (run.want[s][1][1] if run.fft else run.want[s][0][1])
        bad = 0
        for y0, y1 in _bands(p):
            own = orc.raster(op, gl, gr, rows=(y0, y1))
            assert np.array_equal(got[y0:y1], own[y0:y1]), (s, y0, y1)
            chain = orc.raster(op, wl, wr, rows=(y0, y1)).astype(int)
            bad += int((np.abs(got[y0:y1].astype(int) - chain[y0:y1]).max(axis=2) > 1).sum())
        assert bad <= 2e-4 * p.w * p.h, (s, bad)


# ---- A. the persistent spectrum grid: CTAs that walk several units ---------------------------------------------------
def _walk_masks(batch, sm, steps, seed):
    """None = plain update; random masks, one all-off step, and one that switches off every stream of CTA 2's whole walk
    (grid = 2 x SM count CTAs, unit u = 2 * stream + channel: CTA c walks streams c // 2 + k * SM)"""
    rng = np.random.default_rng(seed)
    masks = [None] * steps
    for t in (2, 7):
        masks[t] = rng.random(batch) < 0.6
    masks[4] = np.zeros(batch, bool)
    walk = rng.random(batch) < 0.7
    walk[[s for s in range(1, batch, sm)]] = False
    masks[5] = walk
    return masks


A_SHAPES = [("bars", n, w, 64) for n in (256, 512, 1024, 2048) for w in (1920, 3840)] + [("radial", 2048, 800, 600), ("graph", 1024, 320, 64)]


@pytest.mark.parametrize("module,n,w,h", A_SHAPES)
def test_persistent_walk_against_one_cta_per_unit_single_streams_and_oracle(orc_pm, monkeypatch, module, n, w, h, built):
    sm = _sm()
    batch = 2 * sm + 37                                  # each of the 2 x SM CTAs walks 2 or 3 units; ragged tail, partial 32-stream group
    p = g.default_params(module, n=n, w=w, h=h, lazy_smooth=1)
    probes = (0, 1, sm - 1, sm, 2 * sm - 1, batch - 1)
    masks = _walk_masks(batch, sm, 10, n + w)
    sample = sorted(set(probes) | {2, sm + 1, 2 * sm + 1, batch // 2})
    monkeypatch.delenv("GLAVA_B200_SPEC_CTAS_PER_SM", raising=False)
    walk = Run(p, batch, 10, masks, probes, orc_pm, singles=True)
    try:
        assert walk.spec_launches == ONE, walk.spec_launches
        frames = {s: walk.r.readback(s) for s in sample}
        for s in probes:
            (sl, sr), (tl, tr), fr = walk.single[s]
            assert np.array_equal(walk.spec[0][s], sl[0]) and np.array_equal(walk.spec[1][s], sr[0]), s
            assert np.array_equal(walk.tex[0][s], tl[0]) and np.array_equal(walk.tex[1][s], tr[0]), s
            assert np.array_equal(frames[s], fr), s
        _check_oracle(walk, orc_pm, probes, frames=(0, sm, batch - 1))
    finally:
        walk.close()
    monkeypatch.setenv("GLAVA_B200_SPEC_CTAS_PER_SM", "0")                  # one CTA per unit: nothing walks
    flat = Run(p, batch, 10, masks)
    try:
        assert flat.spec_launches == ONE
        for c in (0, 1):
            assert np.array_equal(walk.spec[c], flat.spec[c]), c
            assert np.array_equal(walk.tex[c], flat.tex[c]), (c, np.argwhere(walk.tex[c] != flat.tex[c])[:5].tolist())
        for s in sample:
            assert np.array_equal(frames[s], flat.r.readback(s)), s
    finally:
        flat.close()


# ---- B. every benchmarked shape against the oracle -------------------------------------------------------------------
def _sweep_names():
    """bench.workload() names and tools/sweep_configs.py's grid (main()), one entry per distinct shape"""
    names = ["headline", "radial4k", "graph720", "wave720", "circle1080", "radial1080", "graph1080", "wave1080"]
    names += [f"sweep:{n}:{w}x{h}" for n in (512, 1024, 2048, 4096, 8192, 16384)
              for w, h in ((1280, 720), (1920, 1080), (3840, 2160), (7680, 4320))]
    out, seen = [], set()
    for nm in names:
        wl = bench.workload(nm)
        key = (wl["module"], wl["n"], wl["w"], wl["h"])
        if key not in seen:
            seen.add(key); out.append(nm)
    return out


def _bench_params(wl):
    p = g.default_params(wl["module"], n=wl["n"], w=wl["w"], h=wl["h"])   # as bench.py builds them
    p.lazy_smooth = 1
    if wl["w"] * wl["h"] > 1920 * 1080:
        p.fb_slots = 16                                                    # frame ring: bounds the framebuffer memory
    return p


def _bench_shape(orc, wl, batch, probes):
    p = _bench_params(wl)
    steps = p.n // 256 + p.avg_frames + 2
    run = Run(p, batch, steps, None, probes, orc)
    try:
        tiles = TILES if run.fft else TILES - 1                                 # (wave has no separate state-update kernel)
        if p.module_name == "circle":
            assert run.spec_launches == FULL                                     # no need-list: full-plane K5 kernel
        elif p.n >= 4096:
            assert run.spec_launches == tiles, run.spec_launches                 # need-list K5 as its own kernel from 4096 up
        else:
            assert run.spec_launches in (ONE, tiles), run.spec_launches          # one kernel where the taps fit shared memory
        # every stream: pipeline B's spectrum is transform_fft of this update's ring (wave: wrange of it), against the exact
        # (float64) transform — the reference's float one is itself 1.2e-5 off it on some of these streams (SURVEY 7)
        epi = emul.lazy_epi_n(p); epi = p.n if epi <= 0 else epi
        op = params_from(p)
        for s in range(batch):
            for c, ring in ((0, run.last_l), (1, run.last_r)):
                if run.fft:
                    want = orc.fft_f64(op, ring[s])
                    assert _peak_err(run.spec[c][s][:epi], want[:epi], want) <= 1e-5, (s, c)
                elif c == 0:
                    assert np.array_equal(run.spec[0][s][:epi], ((ring[s] + np.float32(1)) / np.float32(2))[:epi]), s
        _check_oracle(run, orc, probes, [s for s in probes if run.holds_frame(s)])
    finally:
        run.close()


@pytest.mark.parametrize("name", _sweep_names())
def test_benchmarked_shape_against_oracle(orc_pm, name, built):
    sm = _sm()
    batch = 2 * sm + 37
    _bench_shape(orc_pm, bench.workload(name), batch, probes=(0, sm, batch - 1))


@pytest.mark.parametrize("name", ["radial4k", "sweep:16384:1920x1080"])
def test_benchmarked_shape_at_the_bench_batch(orc_pm, name, built):
    wl = bench.workload(name)
    batch = wl["batch"]
    _bench_shape(orc_pm, wl, batch, probes=(0, batch // 2 + 1, batch - 1))


# ---- C. K5 structures a parameter set selects on its own -------------------------------------------------------------
C_CASES = [
    ("L2 fallback, S = 1", dict(n=16384, smooth_factor=0.1), None, L2),
    ("L2 fallback, S = 2", dict(n=16384, smooth_factor=0.1), 1024, L2),
    ("split below 4096", dict(n=2048, w=7680), None, TILES),
    ("L2 fallback, sample_mode 1", dict(n=16384, smooth_factor=0.1, sample_mode=1), None, L2),
] + [(f"{k} {v} at {n}", {"n": n, k: v}, None, ONE if n < 4096 else TILES)
     for n in (1024, 4096, 16384) for k in ("sample_mode", "round_formula") for v in (1, 2)]


@pytest.mark.parametrize("what,over,batch,launches", C_CASES, ids=[c[0] for c in C_CASES])
def test_parameter_selected_k5_structures(orc_pm, monkeypatch, what, over, batch, launches, built):
    for k in ("GLAVA_B200_K5_SPLIT", "GLAVA_B200_K5N_SMEM", "GLAVA_B200_K5N_S", "GLAVA_B200_SPEC_CTAS_PER_SM", "GLAVA_B200_NO_SMEM_TAPS"):
        monkeypatch.delenv(k, raising=False)
    batch = batch or 2 * _sm() + 37
    over = dict(over)
    p = g.default_params("bars", n=over.pop("n"), w=over.pop("w", 1920), h=48, lazy_smooth=1, **over)
    probes = (0, batch - 1)
    lazy = Run(p, batch, 12, None, probes, orc_pm)
    try:
        assert lazy.spec_launches == launches, (what, lazy.spec_launches)
        _check_oracle(lazy, orc_pm, probes, frames=probes)
        frames = {s: lazy.r.readback(s) for s in probes}
    finally:
        lazy.close()
    p.lazy_smooth = 0
    full = Run(p, batch, 12)
    try:
        assert full.spec_launches == FULL
        for s in probes:
            assert np.array_equal(frames[s], full.r.readback(s)), (what, s)
    finally:
        full.close()


def test_in_kernel_full_plane_k5(orc_pm, built):
    """bars at setbufsize 16384 with smooth_factor 0.3: the full-plane tap table is over its size limit, so lazy_smooth = 0
    evaluates the taps inside k5_planes_kernel; the lazy path at the same parameters takes the L2 form"""
    batch = 40
    p = g.default_params("bars", n=16384, w=1920, h=48, smooth_factor=0.3, lazy_smooth=0)
    probes = (0, batch - 1)
    full = Run(p, batch, 8, None, probes, orc_pm)
    try:
        assert full.spec_launches == FULL
        _check_oracle(full, orc_pm, probes, frames=probes)
        frames = {s: full.r.readback(s) for s in probes}
    finally:
        full.close()
    p.lazy_smooth = 1
    lazy = Run(p, batch, 8)
    try:
        assert lazy.spec_launches == L2
        for s in probes:
            assert np.array_equal(frames[s], lazy.r.readback(s)), s
    finally:
        lazy.close()
