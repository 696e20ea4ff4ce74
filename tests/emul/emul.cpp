// TEST INFRASTRUCTURE — host emulation of the CUDA kernels' arithmetic.
//
// Compiles the product's *_core.h headers for the host (g++ -ffp-contract=off) and drives them
// with the same thread/phase structure the kernels use (threads emulated sequentially, one
// loop per __syncthreads phase).  Lets the CPU-only test tier check the kernels' maths against
// the oracle before any GPU time is spent.  NOT part of libglava_b200.so and never loaded by it.
#include "../../glava_b200/csrc/raster_core.h"
#include "../../glava_b200/csrc/chain_core.h"
#include "../../glava_b200/csrc/tables.h"

#include <cmath>
#include <cstring>
#include <vector>

using namespace glb;

namespace {

template <int M, int T, int NS>
void emul_passes(std::vector<cpx>& buf, const std::vector<cpx>& raw, const double* window, const cpx* tw) {
    constexpr int REM = M / NS;
    if constexpr (REM > 1) {
        constexpr int R = (REM >= 8) ? 8 : REM;
        using Pass = StockhamPass<M, T, R, NS>;
        std::vector<cpx> regs((size_t) T * Pass::PER * R);
        for (int tid = 0; tid < T; ++tid) {                       // read phase
            cpx (&reg)[Pass::PER][R] = *reinterpret_cast<cpx (*)[Pass::PER][R]>(&regs[(size_t) tid * Pass::PER * R]);
            if constexpr (NS == 1) {
                Pass::load([&](int i) {
                    cpx v = raw[i];
                    cpx r = { (float) ((double) v.x * window[2 * i]), (float) ((double) v.y * window[2 * i + 1]) };
                    return r; }, tw, tid, reg);
            } else Pass::load([&](int i) { return buf[fft_pad(i)]; }, tw, tid, reg);
        }
        for (int tid = 0; tid < T; ++tid) {                       // write phase
            cpx (&reg)[Pass::PER][R] = *reinterpret_cast<cpx (*)[Pass::PER][R]>(&regs[(size_t) tid * Pass::PER * R]);
            Pass::store(buf.data(), tid, reg);
        }
        emul_passes<M, T, NS * R>(buf, raw, window, tw);
    }
}

template <int LOG2N>
void emul_fft_t(const float* pcm, float* out, float fft_scale, float fft_cutoff) {
    constexpr int N = 1 << LOG2N, M = N / 2;
    constexpr int T = (M / 8 < 128) ? 128 : ((M / 8 > 512) ? 512 : M / 8);
    std::vector<double> w(N);
    for (int i = 0; i < N; ++i) w[i] = 0.53836 - (0.46164 * cos(6.28318530718 * (double) i / (double) N - 1));
    std::vector<cpx> tw(M);
    for (int k = 0; k < M; ++k) { double a = -2.0 * M_PI * (double) k / (double) M; tw[k] = { (float) cos(a), (float) sin(a) }; }
    std::vector<cpx> raw(M), buf(fft_padded_size(M));
    memcpy(raw.data(), pcm, sizeof(float) * N);
    emul_passes<M, T, 1>(buf, raw, w.data(), tw.data());
    for (int n = 0; n < N; ++n) {
        cpx z = buf[fft_pad(n >> 1)];
        out[n] = fft_post((n & 1) ? z.y : z.x, n, N, fft_scale, fft_cutoff);
    }
}

}  // namespace

extern "C" {

int emul_fft(int n, const float* pcm, float* out, float fft_scale, float fft_cutoff) {
    switch (n) {
        case 256: emul_fft_t<8>(pcm, out, fft_scale, fft_cutoff); break;
        case 512: emul_fft_t<9>(pcm, out, fft_scale, fft_cutoff); break;
        case 1024: emul_fft_t<10>(pcm, out, fft_scale, fft_cutoff); break;
        case 2048: emul_fft_t<11>(pcm, out, fft_scale, fft_cutoff); break;
        case 4096: emul_fft_t<12>(pcm, out, fft_scale, fft_cutoff); break;
        case 8192: emul_fft_t<13>(pcm, out, fft_scale, fft_cutoff); break;
        case 16384: emul_fft_t<14>(pcm, out, fft_scale, fft_cutoff); break;
        default: return -1;
    }
    return 0;
}

// persistent state of one (stream, channel) plane, laid out like the kernel's HBM arrays
struct emul_chan {
    int n, F;
    std::vector<float> applied, ring_f;
    std::vector<uint16_t> gr_store, ring_u;
    unsigned long long update;
};
emul_chan* emul_chan_new(const glava_b200_params* p) {
    emul_chan* c = new emul_chan();
    c->n = p->n; c->F = p->avg_frames; c->update = 0;
    c->applied.assign(p->n, 0.0f); c->ring_f.assign((size_t) p->n * p->avg_frames, 0.0f);
    c->gr_store.assign(p->n, 0); c->ring_u.assign((size_t) p->n * p->avg_frames, 0);
    return c;
}
void emul_chan_free(emul_chan* c) { delete c; }

// mirrors spectrum_kernel's epilogue + K5 (spectrum_kernels.cu) for one plane
int emul_chan_update(emul_chan* c, const glava_b200_params* pp, const float* pcm, int is_fft, float* spec, uint16_t* tex) {
    const glava_b200_params& p = *pp;
    const int N = p.n, F = p.avg_frames;
    std::vector<float> v(N);
    std::vector<uint16_t> av(N);
    if (is_fft) {
        if (emul_fft(N, pcm, v.data(), p.fft_scale, p.fft_cutoff)) return -1;
        if (!p.accel_fft) {
            const float g = p.gravity_step * (1.0f / p.ur);
            const int newest = (int) (c->update % (unsigned long long) F);
            for (int n = 0; n < N; ++n) {
                float x = gravity_a(v[n], &c->applied[n], g);
                c->ring_f[(size_t) newest * N + n] = x;
                float acc = 0.0f;
                for (int f = 0; f < F; ++f) {
                    int slot = newest + 1 + f; if (slot >= F) slot -= F;
                    float b = (f == F - 1) ? x : c->ring_f[(size_t) slot * N + n];
                    double w = 0.6 - (0.4 * cos(6.28318530718 * (double) f / (double) F - 1));
                    if (p.avg_window) acc = (float) ((double) acc + w * (double) b); else acc += b;
                }
                float out = acc / (float) F;
                spec[n] = out; av[n] = (uint16_t) unorm16(out);
            }
        } else {
            const float diff = p.gravity_step * (1.0f / p.ur);
            const int out_idx = (int) (c->update % (unsigned long long) F);
            const int windowed = (p.avg_window && F != 2) ? 1 : 0;
            for (int n = 0; n < N; ++n) {
                spec[n] = v[n];
                uint32_t gq = gravity_b(unorm16(v[n]), c->gr_store[n], diff);
                c->gr_store[n] = (uint16_t) gq;
                uint32_t texel = gq;
                if (F > 1) {
                    c->ring_u[(size_t) out_idx * N + n] = (uint16_t) gq;
                    float r = 0.0f;
                    for (int i = 0; i < F; ++i) {
                        int fr = out_idx - i; if (fr < 0) fr += F;
                        float tx = from16(i == 0 ? gq : (uint32_t) c->ring_u[(size_t) fr * N + n]);
                        float w = 0.53836f - (0.46164f * cosf(6.28318530718f * (float) i / (float) F - 1.0f));
                        if (windowed) r += w * tx; else r += tx;
                    }
                    texel = unorm16(r / (float) F);
                }
                av[n] = (uint16_t) texel;
            }
        }
        ++c->update;
    } else {
        for (int n = 0; n < N; ++n) { float b = pcm[n]; b += 1.0f; b /= 2.0f; spec[n] = b; av[n] = (uint16_t) unorm16(b); }
    }
    if (p.smooth_pass) {
        SmoothParams sp = smooth_params(p);
        for (int x = 0; x < N; ++x) tex[x] = (uint16_t) smooth_pass_texel(sp, av.data(), N, x);
    } else memcpy(tex, av.data(), sizeof(uint16_t) * N);
    return 0;
}

// exhaustive check helper: returns the number of u for which from8/from16 differ from true division
int emul_unorm_fetch_mismatches(void) {
    int bad = 0;
    for (uint32_t u = 0; u < 256; ++u) { volatile float d = (float) u / 255.0f; if (from8(u) != d) ++bad; }
    for (uint32_t u = 0; u < 65536; ++u) { volatile float d = (float) u / 65535.0f; if (from16(u) != d) ++bad; }
    return bad;
}

void emul_smooth(const glava_b200_params* p, const uint16_t* in, uint16_t* out) {
    SmoothParams sp = smooth_params(*p);
    for (int x = 0; x < p->n; ++x) out[x] = (uint16_t) smooth_pass_texel(sp, in, p->n, x);
}

// one compiled colour expression at X (the interpreter the kernels run: raster_core.h eval_color_prog)
void emul_eval_color(const glava_b200_color_prog* prog, float x, float out[4]) {
    const f4 r = eval_color_prog(*prog, x);
    out[0] = r.r; out[1] = r.g; out[2] = r.b; out[3] = r.a;
}

// per-pixel reference semantics (raster_generic_kernel)
void emul_raster(const glava_b200_params* pp, const uint16_t* tl, const uint16_t* tr, uint8_t* out, int y0, int y1) {
    const glava_b200_params& p = *pp;
    AudioTex t; t.l = tl; t.r = tr; t.n = p.n; t.pre_smoothed = p.shader_pre_smoothed ? (p.shader_pre_smoothed == 1) : p.smooth_pass;   /* capi.cu run_update: the raster launch's view */ t.sp = smooth_params(p);
    uint32_t* dst = reinterpret_cast<uint32_t*>(out);
    for (int y = y0; y < y1; ++y) for (int x = 0; x < p.w; ++x) dst[(size_t) y * p.w + x] = module_px(p, t, x, y);
}

// hoisted evaluation exactly as raster_bars_kernel / raster_graph_kernel / raster_wave_kernel do it
int emul_raster_fast(const glava_b200_params* pp, const uint16_t* tl, const uint16_t* tr, uint8_t* out) {
    const glava_b200_params& p = *pp;
    AudioTex t; t.l = tl; t.r = tr; t.n = p.n; t.pre_smoothed = p.shader_pre_smoothed ? (p.shader_pre_smoothed == 1) : p.smooth_pass;   /* capi.cu run_update: the raster launch's view */ t.sp = smooth_params(p);
    uint32_t* dst = reinterpret_cast<uint32_t*>(out);
    if (p.module == GLAVA_B200_MOD_BARS && !p.bars_mirror_yx) {
        std::vector<BarsCol> col(p.w);
        for (int x = 0; x < p.w; ++x) col[x] = bars_column(p, t, (float) x + 0.5f, p.w);
        const bool has_outline = p.bars_outline_width > 0.0f;
        for (int y = 0; y < p.h; ++y) {
            float fy = (float) y + 0.5f, d = p.bars_flip ? (float) p.h - fy : fy;
            BarsRow rc = bars_row(p, d);
            for (int x = 0; x < p.w; ++x) {
                uint32_t below = (col[x].cls == 1) ? rc.fill : rc.outl;
                uint32_t v = (d < col[x].vm) ? below : ((has_outline && d <= col[x].v) ? rc.outl : 0u);
                dst[(size_t) y * p.w + x] = col[x].cls ? v : 0u;
            }
        }
        return 0;
    }
    if (p.module == GLAVA_B200_MOD_GRAPH) {
        std::vector<float> s(p.w + 2, 0.0f);
        for (int x = 0; x < p.w; ++x) s[x + 1] = graph_height(p, t, x);
        for (int y = 0; y < p.h; ++y) {
            uint32_t row3[3] = { y > 0 ? graph_row(p, y - 1) : 0u, graph_row(p, y), y + 1 < p.h ? graph_row(p, y + 1) : 0u };
            for (int x = 0; x < p.w; ++x) {
                const float s3[3] = { s[x], s[x + 1], s[x + 2] };
                dst[(size_t) y * p.w + x] = graph_px_cols(p, s3, row3, x, y);
            }
        }
        return 0;
    }
    if (p.module == GLAVA_B200_MOD_CIRCLE && p.smooth_pass) {
        // raster_circle_kernel: stage 1 from the cached geometry (texel references), stages 2-3 from the tile
        std::vector<uint32_t> s1((size_t) (p.w + 2) * (p.h + 2), 0u);
        auto at = [&](int x, int y) -> uint32_t& { return s1[(size_t) (y + 1) * (p.w + 2) + (x + 1)]; };
        for (int y = 0; y < p.h; ++y) for (int x = 0; x < p.w; ++x) at(x, y) = circle_stage1_geo(p, t, circle_geometry(p, x, y));
        for (int y = 0; y < p.h; ++y) for (int x = 0; x < p.w; ++x) {
            const int xm = x > 0 ? x - 1 : x, ym = y > 0 ? y - 1 : y;       // the kernel's lxm / lym: int(-0.5) = 0 at the border
            const uint32_t nb[6] = { at(x + 1, y), at(x + 1, y + 1), at(x, y + 1), at(xm, y), at(xm, ym), at(x, ym) };
            dst[(size_t) y * p.w + x] = circle_finish(p, at(x, y), nb);
        }
        return 0;
    }
    if (p.module == GLAVA_B200_MOD_WAVE) {
        std::vector<WaveCol> c(p.w + 2);
        for (int x = -1; x <= p.w; ++x) { int xc = x < 0 ? 0 : (x >= p.w ? p.w - 1 : x); c[x + 1] = wave_column(p, t, xc); }
        for (int y = 0; y < p.h; ++y) for (int x = 0; x < p.w; ++x) {
            const WaveCol c3[3] = { c[x], c[x + 1], c[x + 2] };
            dst[(size_t) y * p.w + x] = wave_px_cols(p, c3, x, y);
        }
        return 0;
    }
    return -1;
}

// ---- optional rd_update stages (chain_core.h): the kernels' per-element functions driven the way the kernels do ----
void emul_bufscale(const float* in, int n_in, int k, float* out) {
    for (int i = 0; i < n_in / k; ++i) out[i] = bufscale_mean(in + (size_t) i * k, k);       // bufscale_kernel: thread i
}
void emul_transform_smooth(float* b, int sz, float smooth_distance, float smooth_ratio) {
    std::vector<SmoothWin> tab; int lim = 0;
    const int asz = transform_smooth_windows(sz, smooth_distance, smooth_ratio, &tab, &lim);   // capi.cu build_tables
    std::vector<float> sm(b, b + lim);                                                         // kernel: head staged in smem
    transform_smooth_serial(sm.data(), tab.data(), asz);
    for (int i = 0; i < asz; ++i) b[i] = sm[i];
}
void emul_upload(const float* s, const float* e, int n, float ur, float fr, int kcounter, uint16_t* out) {
    const float mod = keyframe_mod(ur, fr, kcounter);
    for (int i = 0; i < n; ++i) out[i] = (uint16_t) upload_texel(e ? keyframe_lerp(s[i], e[i], mod) : s[i]);
}

// ---- K5 from the precomputed tables (tables.h), walked the way the kernels walk them ------------------------------------
// lazy K5 of one channel: out[x] for the need-list texels only (others left untouched); path 0 = tap-major table (the
// spectrum kernel's L2 path), 1 = texel-major blob (its shared-memory path).  Returns the number of texels written.
int emul_lazy_k5(const glava_b200_params* pp, int chan, int path, const uint16_t* av, uint16_t* out, int* need_out) {
    const glava_b200_params& p = *pp;
    std::vector<int> lists[2];
    if (!build_need_list(p, lists)) return -1;
    LazyTables t;
    build_lazy_tables(p, lists, &t);
    const SmoothParams sp = smooth_params(p);
    const int N = p.n;
    int written = 0;
    if (path >= 2) {
        // k5_need_smem_kernel: blocks of sampled texels (path = 2: default block shape; otherwise target rows = path, 3 texels
        // per block), a tile of from16() values per block, tap rows clamped into the tile
        NeedBlocks nb;
        if (path == 2) build_need_blocks(t, N, 384, 16, &nb); else build_need_blocks(t, N, path, 3, &nb);
        const unsigned char* blob = t.csr.data() + (size_t) chan * t.blob;
        const float* tw = reinterpret_cast<const float*>(blob);
        const uint16_t* ti = reinterpret_cast<const uint16_t*>(blob + t.idx_off);
        const int* to = reinterpret_cast<const int*>(blob + t.off_off);
        std::vector<char> seen(t.cnt, 0);
        for (int b = 0; b < nb.nblk; ++b) {
            const int* bk = nb.blk.data() + ((size_t) chan * nb.nblk + b) * 4;
            const int k0 = bk[0], k1 = bk[1], lo = bk[2], rows = bk[3];
            if (k1 <= k0) continue;
            if ((lo & 1) || (rows & 1) || lo < 0 || lo + rows > N || rows > nb.max_rows) return -2;
            std::vector<float> tile(rows);
            for (int i = 0; i < rows; ++i) tile[i] = from16(av[lo + i]);
            for (int k = k1 - 1; k >= k0; --k) {
                const int x = t.need[chan * t.cnt + k];
                if (x < 0 || x >= N) continue;
                if (seen[k]) return -3;
                seen[k] = 1;
                SmoothAcc acc; acc.init();
                for (int o = to[k]; o < to[k + 1]; ++o) {
                    int r = (int) ti[o] - lo;
                    if ((r < 0 || r >= rows) && !(ti[o] == 0 && tw[o] == 0.0f)) return -4;      // a counting tap outside its block's tile
                    r = r < 0 ? 0 : (r >= rows ? rows - 1 : r);
                    acc.add_noweight(tile[r], tw[o]);
                }
                acc.weight = t.wsum[chan * t.cnt + k];
                out[x] = (uint16_t) unorm16(acc.result(sp));
                if (need_out) need_out[written] = x;
                ++written;
            }
        }
        for (size_t k = 0; k < t.cnt; ++k) { const int x = t.need[chan * t.cnt + k]; if (x >= 0 && x < N && !seen[k]) return -5; }
        return written;
    }
    for (size_t k = 0; k < t.cnt; ++k) {                                   // kernel: thread k (+ T, ...)
        const int x = t.need[chan * t.cnt + k];
        if (x < 0 || x >= N) continue;
        SmoothAcc acc; acc.init();
        if (path == 0) {
            const TapEntry* col = t.tab.data() + (size_t) chan * t.tap_max * t.cnt + k;
            const int cnt = t.tcnt[chan * t.cnt + k];
            for (int j = 0; j < cnt; ++j) { const TapEntry e = col[(size_t) j * t.cnt]; acc.add_noweight(from16(av[e.idx]), e.w); }
        } else {
            const unsigned char* blob = t.csr.data() + (size_t) chan * t.blob;
            const float* tw = reinterpret_cast<const float*>(blob);
            const uint16_t* ti = reinterpret_cast<const uint16_t*>(blob + t.idx_off);
            const int* to = reinterpret_cast<const int*>(blob + t.off_off);
            for (int o = to[k]; o < to[k + 1]; ++o) acc.add_noweight(from16(av[ti[o]]), tw[o]);
        }
        acc.weight = t.wsum[chan * t.cnt + k];
        out[x] = (uint16_t) unorm16(acc.result(sp));
        if (need_out) need_out[written] = x;
        ++written;
    }
    return written;
}
int emul_lazy_epi_n(const glava_b200_params* pp) {
    std::vector<int> lists[2];
    if (!build_need_list(*pp, lists)) return -1;
    LazyTables t;
    build_lazy_tables(*pp, lists, &t);
    return t.epi_n;
}
// The host table sizes capi.cu's build_tables chooses a K5 launch structure from: out = {lazy tap-major table bytes, lazy
// texel-major blob bytes of one channel, tallest need-block tile in rows (build_need_blocks with target_rows / tpb), full-
// plane table's widest input span, full-plane table entry bytes}.  Returns -1 where the module has no need-list (the lazy
// entries are then 0).
int emul_table_sizes(const glava_b200_params* pp, int target_rows, int tpb, long long out[5]) {
    const glava_b200_params& p = *pp;
    for (int i = 0; i < 5; ++i) out[i] = 0;
    K5TableHost k;
    build_k5_table_host(p, &k);
    out[3] = k.max_span; out[4] = (long long) (k.ent.size() * sizeof(K5Ent));
    std::vector<int> lists[2];
    if (!build_need_list(p, lists)) return -1;
    LazyTables t;
    build_lazy_tables(p, lists, &t);
    NeedBlocks nb;
    build_need_blocks(t, p.n, target_rows, tpb, &nb);
    out[0] = (long long) (t.tab.size() * sizeof(TapEntry)); out[1] = (long long) t.blob; out[2] = nb.max_rows;
    return 0;
}

// full-plane K5 of one plane through the per-block table, as k5_table_kernel does it (float staging, padded uniform loop)
void emul_k5_table(const glava_b200_params* pp, const uint16_t* in, uint16_t* out) {
    const glava_b200_params& p = *pp;
    K5TableHost t;
    build_k5_table_host(p, &t);
    const SmoothParams sp = smooth_params(p);
    const bool avg_only = sp.sample_mode == 0;
    std::vector<float> seg;
    for (size_t b = 0; b < t.blk.size(); ++b) {
        const K5Blk d = t.blk[b];
        seg.resize((size_t) d.span);
        for (int k = 0; k < d.span; ++k) seg[k] = from16(in[d.lo + k]);
        for (int tid = 0; tid < K5_BLOCK; ++tid) {
            const int x = (int) b * K5_BLOCK + tid;
            if (x >= p.n) continue;
            SmoothAcc acc; acc.init();
            for (int j = 0; j < d.taps; ++j) {
                const K5Ent e = t.ent[(size_t) d.base + (size_t) j * K5_BLOCK + tid];
                float w; memcpy(&w, &e.wbits, 4);
                const float v = seg[e.idx] * w;
                acc.avg += v;
                if (!avg_only) { if (acc.vmax < v) acc.vmax = v; }
            }
            acc.weight = t.wsum[x];
            out[x] = (uint16_t) unorm16(acc.result(sp));
        }
    }
}

}  // extern "C"
