// f2_fused.cu -- fused gammatone filterbank + Hilbert envelope + low-pass + decimation.
//
// Replaces, for every (utterance, channel) pair, the reference's
//   erb_filterbank            gammatone/filters.py:228-237   (4x lfilter + /gain)
//   paddedHilbert + abs       scripts/processing/EnvelopeExtraction.py:20-36,58
//   lowPassFilter             scripts/processing/EnvelopeExtraction.py:39-48
//   the 160-sample grid read by InputGenerator.py:73-80
// in ONE pass over the samples, so the full-rate (C,n) matrices only reach HBM when the
// caller asks for .GFB / .ENV1 output.
//
// Mapping: one CTA = one warp = one work item = (utterance, group of 32 adjacent channels,
// output samples [t0,t1)); one thread = one channel, so every sample is a shared-memory
// broadcast and every store is a coalesced 128-byte line.  Tiles of 256 samples of the
// utterance's ring buffers (x, Im hilbert(x)) and of the edge-injection kernel G are streamed
// into shared memory by 1-D TMA bulk copies through a 4-deep mbarrier pipeline; 16 CTAs are
// resident per SM.
//
// Arithmetic: FP32, no tensor cores (there is no contraction on this path).  The real and
// the imaginary (Hilbert) cascades share coefficients, so they run as the two halves of
// packed FFMA2/FADD2 instructions.  The sections (f2_sections.cuh) take one form per group of
// 32 channels (the form is uniform in a CTA):
//   direct form  (FORM 1)                                    3 packed + 1 scalar instruction
//   delta form   (FORM 0)                                    4 packed + 1 scalar instruction
// The delta form keeps float32 round-off and coefficient quantisation harmless for poles
// 0.039 rad from z=1 (SURVEY.md H2); the direct form is used where 1+B1+B2 = |1-pole|^2 is
// large enough for it to be as accurate (FusedParams::direct_min_cy, DESIGN.md section 3).
// FORM 2 (float64 direct form, exact coefficients) runs the groups a plan created with
// F2_PLAN_FLOAT64_SECTIONS found float32 unable to hold to the tolerance, in the float64
// instantiations fused_kernel<true, ...> (DESIGN.md 2 (iii)).
// Every stage is computed WITHOUT its common numerator gain a0 = A0/gain^(1/4): stage k holds
// y_k / a0^k, and the single factor a0^4 = A0^4/gain is applied where a value leaves the
// kernel (folded into the low-pass b0 when the low-pass is on).  In delta form that is 40
// FMA-pipe lane-cycles per channel-sample for filterbank + envelope + low-pass, exactly the
// algorithmic count of SURVEY.md section 8d; 32 in direct form.
// The imaginary half solves the N2-periodic ring equation that the reference's
// zero-padded FFT Hilbert transform implies (SURVEY.md H1): e_k are the residuals of the
// zero-padded real cascade at ring positions n and n+1, G[t] is the circular Hilbert
// kernel (2/N2)cot(pi*l/N2) at the odd one of (t-n), (t-n-1).
//
// Time chunking: all sections are strictly stable, so a chunk that starts at t0>0 is
// warm-started from zero state w_casc (+ w_lpf) samples earlier; the truncated history is
// below float32 resolution (pole radius^W).  The same truncation gives the edge residuals
// (real cascade over the last w_edge samples) and the periodic steady state of the
// imaginary path (w_imag samples before t=0 on the ring).  The plan's lengths are those of the
// bank's slowest channel; every group of 32 channels scales them to its own slowest pole
// (group_warmup, f2_common.cuh): 256 / 512 / 1024 / 1536 samples for the four groups of the
// 128-channel bank instead of 1536 for all.
#include "f2_fused.cuh"
#include "f2_sections.cuh"

#include <stdlib.h>

namespace f2 {

// ENV: 0 = cascade only, 1 = magnitude, 2 = magnitude + low-pass.
// OUT: 0 = nothing leaves the kernel (warm-up), 1 = decimated frames only, 2 = full-rate
//      stores: (C, n) when CN, time-major envelope when asked (and decimated frames when
//      asked), 3 = every decimated frame goes straight into the (up to win_dots) window rows
//      that contain it.
struct OutCtx {
    float* env;     // time-major envelope: points at sample t of this thread's channel (or null)
    float* dec;     // OUT 1/2: the next decimated frame of this channel (or null).  OUT 3: slot 0 of the
                    // window that STARTS at the next decimated frame
    int next_dec;   // time index of the next decimated frame
    int step;
    size_t C;
    float env_scale;  // g4 (no low-pass) or g4*b0 (low-pass): applied when a value is stored
    int wk;         // OUT 3: index (within the utterance) of the next decimated frame
    int nwin;       // OUT 3: windows of this utterance
    // CN: (C, n) outputs in the reference's layout.  Each lane stages its channel's samples in a 32 x (kCnW+1)
    // shared-memory tile; every kCnW samples the warp writes the tile out row by row -- 32 consecutive samples
    // of one channel per store instruction (128 / 256 contiguous bytes), kCnW per row.
    float* tr_g;    // shared-memory tiles (or null)
    float* tr_e;
    char* cn_g;     // element (first channel of this CTA, sample 0) of the utterance's (C, n) block (or null)
    char* cn_e;
    int cn_n;       // samples per row
    int cn_rows;    // channels of this CTA that exist (<= 32)
};

// (C, n) staging tile: 32 channels x kCnW samples (+1 column of padding).  Longer runs per channel row make
// the stores friendlier to DRAM pages (every row of a tile lands in a different page of the (C, n) matrix).
constexpr int kCnW = 128;
constexpr int kCnP = kCnW + 1;

// rows of the staged tile -> global: samples [tb, tb + cnt) of every channel of this CTA, as float64 or float32
__device__ __forceinline__ void flush_cn(const float* tr, char* base, int f64, const OutCtx& o, int tb, int cnt) {
    __syncwarp();
    const int lane = threadIdx.x;
    if (f64) {
        double* row = reinterpret_cast<double*>(base) + tb + lane;
        for (int r = 0; r < o.cn_rows; ++r, row += o.cn_n)
#pragma unroll
            for (int h = 0; h < kCnW; h += 32)
                if (lane + h < cnt) __stcs(row + h, (double)tr[r * kCnP + lane + h]);
    } else {
        float* row = reinterpret_cast<float*>(base) + tb + lane;
        for (int r = 0; r < o.cn_rows; ++r, row += o.cn_n)
#pragma unroll
            for (int h = 0; h < kCnW; h += 32)
                if (lane + h < cnt) __stcs(row + h, tr[r * kCnP + lane + h]);
    }
    __syncwarp();
}

// OUT 3: decimated frame j = o.wk with value v goes to slot s of window j-s, s < dots, where that
// window exists: ((row0 + j - s)*dots + s)*C = (row0 + j)*dots*C - s*(dots-1)*C.  dots and C are
// read from the kernel parameters so that the per-slot offsets stay on the uniform datapath.
__device__ __forceinline__ void store_window_entries(const FusedParams& p, OutCtx& o, float v, bool active) {
    const int dots = p.win_dots;
    const long long back = (long long)(dots - 1) * (long long)p.C;
    float* wp = o.dec;
    if (o.wk >= dots - 1 && o.wk < o.nwin) {  // interior frame: all `dots` windows exist
        if (active)
            for (int s = 0; s < dots; ++s) __stcs(wp - (long long)s * back, v);
    } else {
        for (int s = 0; s < dots; ++s) {
            const int k = o.wk - s;
            if (k >= 0 && k < o.nwin && active) __stcs(wp - (long long)s * back, v);
        }
    }
    o.dec += (size_t)dots * (size_t)p.C;
    o.wk += 1;
}

// Unscaled envelope sample.  ENV 1: |y|.  ENV 2: the one-pole state w[t] = k*w[t-1] + |y[t]|; the
// butter(1) low-pass output is b0*(w[t] + w[t-1]) (same transfer function (1+z^-1)/(1-k*z^-1) as
// the reference's lfilter, EnvelopeExtraction.py:47-48), and that sum is only formed for the
// samples that are stored -- one FMA per sample instead of an add and an FMA.
template <int ENV, class S>
__device__ __forceinline__ float envelope(const FusedParams& p, S& s, float2 y) {
    float e = fast_sqrt(fmaf(y.x, y.x, y.y * y.y));
    if (ENV == 2) {
        e = fmaf(p.lp_k, s.l, e);
        s.l = e;
    }
    return e;
}

template <int FORM, int ENV, int OUT, bool ZEROX, int U, bool CN = false, class K, class S, class E>
__device__ __forceinline__ void run_tile(const FusedParams& p, const K& k, S& s, const E (&ee)[4],
                                         const E (&eo)[4], const float2* __restrict__ sxz,
                                         const float* __restrict__ sg, int t, int cnt, bool active, OutCtx& o) {
    int i = 0;
    for (; i + U <= cnt; i += U) {
        float xv[2 * U];
        float gv[U];
#pragma unroll
        for (int j = 0; j < U / 2; ++j) {
            const float4 v = *reinterpret_cast<const float4*>(sxz + i + 2 * j);
            xv[4 * j + 0] = v.x;
            xv[4 * j + 1] = v.y;
            xv[4 * j + 2] = v.z;
            xv[4 * j + 3] = v.w;
        }
#pragma unroll
        for (int j = 0; j < U / 4; ++j) {
            const float4 v = *reinterpret_cast<const float4*>(sg + i + 4 * j);
            gv[4 * j + 0] = v.x;
            gv[4 * j + 1] = v.y;
            gv[4 * j + 2] = v.z;
            gv[4 * j + 3] = v.w;
        }
        float ev[U];
        const float wprev = s.wprev;  // ENV 2: w of the sample before this block
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const float2 u = make_float2(ZEROX ? 0.f : xv[2 * j], xv[2 * j + 1]);
            const float2 y = (j & 1) ? cascade<FORM>(k, s, u, gv[j], eo) : cascade<FORM>(k, s, u, gv[j], ee);
            if (ENV > 0) ev[j] = envelope<ENV>(p, s, y);
            if (OUT == 2 && ENV > 0 && o.env && active) {
                const float v = ENV == 2 ? ev[j] + (j > 0 ? ev[j > 0 ? j - 1 : 0] : wprev) : ev[j];
                __stcs(o.env + (size_t)j * o.C, o.env_scale * v);
            }
            if (OUT == 2 && CN) {
                const int col = (t + i + j) & (kCnW - 1);
                if (o.cn_g) o.tr_g[threadIdx.x * kCnP + col] = k.g4 * y.x;
                if (ENV > 0 && o.cn_e) {
                    const float v = ENV == 2 ? ev[j] + (j > 0 ? ev[j > 0 ? j - 1 : 0] : wprev) : ev[j];
                    o.tr_e[threadIdx.x * kCnP + col] = o.env_scale * v;
                }
            }
        }
        if (ENV == 2) s.wprev = ev[U - 1];
        if (OUT == 2 && o.env) o.env += U * o.C;
        if (OUT == 2 && CN && ((t + i + U) & (kCnW - 1)) == 0) {
            if (o.cn_g) flush_cn(o.tr_g, o.cn_g, p.gfb_cn_f64, o, t + i + U - kCnW, kCnW);
            if (ENV > 0 && o.cn_e) flush_cn(o.tr_e, o.cn_e, p.env_cn_f64, o, t + i + U - kCnW, kCnW);
        }
        if (OUT > 0 && ENV > 0 && o.dec) {
            while (o.next_dec < t + i + U) {
                const int r = o.next_dec - (t + i);
                float v = ev[0];
                float vp = wprev;
#pragma unroll
                for (int j = 1; j < U; ++j) {
                    v = (r == j) ? ev[j] : v;
                    if (ENV == 2) vp = (r == j) ? ev[j - 1] : vp;
                }
                if (ENV == 2) v += vp;
                if (OUT == 3) {
                    store_window_entries(p, o, o.env_scale * v, active);
                } else {
                    if (active) __stcs(o.dec, o.env_scale * v);
                    o.dec += o.C;
                }
                o.next_dec += o.step;
            }
        }
    }
    for (; i < cnt; ++i) {
        const float2 xz = sxz[i];
        const float2 u = make_float2(ZEROX ? 0.f : xz.x, xz.y);
        const float2 y = (i & 1) ? cascade<FORM>(k, s, u, sg[i], eo) : cascade<FORM>(k, s, u, sg[i], ee);
        float e = 0.f;
        if (ENV > 0) e = envelope<ENV>(p, s, y);
        const float out = ENV == 2 ? e + s.wprev : e;
        if (ENV == 2) s.wprev = e;
        if (OUT == 2 && ENV > 0 && o.env) {
            if (active) __stcs(o.env, o.env_scale * out);
            o.env += o.C;
        }
        if (OUT == 2 && CN) {
            const int col = (t + i) & (kCnW - 1);
            if (o.cn_g) o.tr_g[threadIdx.x * kCnP + col] = k.g4 * y.x;
            if (ENV > 0 && o.cn_e) o.tr_e[threadIdx.x * kCnP + col] = o.env_scale * out;
            if (col == kCnW - 1) {
                if (o.cn_g) flush_cn(o.tr_g, o.cn_g, p.gfb_cn_f64, o, t + i - (kCnW - 1), kCnW);
                if (ENV > 0 && o.cn_e) flush_cn(o.tr_e, o.cn_e, p.env_cn_f64, o, t + i - (kCnW - 1), kCnW);
            }
        }
        if (OUT > 0 && ENV > 0 && o.dec && o.next_dec == t + i) {
            if (OUT == 3) {
                store_window_entries(p, o, o.env_scale * out, active);
            } else {
                if (active) __stcs(o.dec, o.env_scale * out);
                o.dec += o.C;
            }
            o.next_dec += o.step;
        }
    }
    if (OUT == 2 && CN && ((t + cnt) & (kCnW - 1)) != 0) {   // the utterance ends inside a block of kCnW
        const int rest = (t + cnt) & (kCnW - 1);
        if (o.cn_g) flush_cn(o.tr_g, o.cn_g, p.gfb_cn_f64, o, t + cnt - rest, rest);
        if (ENV > 0 && o.cn_e) flush_cn(o.tr_e, o.cn_e, p.env_cn_f64, o, t + cnt - rest, rest);
    }
}

// ---- cutoff sweep: one cascade, up to kMaxCutoffs envelope settings -------------------------------------
// Every low-pass setting keeps its own one-pole state w (the operations of envelope<2>); |y| is formed once.
// A plane's value is captured at the stored sample itself, from w[t] and w[t-1] = the state before this
// sample's update, so no block of U envelope values per setting is held.  The stored values are the same
// operations in the same order as run_tile's OUT 1 path: (w[t] + w[t-1]) * (g4 * b0), or g4 * |y|.
template <int NL>
__device__ __forceinline__ void store_planes(const FusedParams& p, float g4, OutCtx& o, float mag, const float (&w)[NL],
                                             const float (&wp)[NL], bool active) {
    if (active) {
        float* d = o.dec;
#pragma unroll
        for (int j = 0; j < kMaxCutoffs; ++j) {
            if (j < p.sw_planes) {
                const int q = p.sw_state[j];
                float v = mag, scale = g4;
#pragma unroll
                for (int r = 0; r < NL; ++r) {
                    if (q == r) {
                        v = w[r] + wp[r];
                        scale = g4 * p.sw_b0[r];
                    }
                }
                __stcs(d, scale * v);
                d += p.plane_stride;
            }
        }
    }
    o.dec += o.C;
    o.next_dec += o.step;
}

// One sample of the sweep.  CHECK: a decimated frame may fall on it.
template <int FORM, int NL, bool CHECK, class K, class S, class E>
__device__ __forceinline__ void sweep_sample(const FusedParams& p, const K& k, S& s, float (&w)[NL], float2 u, float g,
                                             const E (&e)[4], int t, bool active, OutCtx& o) {
    const float2 y = cascade<FORM>(k, s, u, g, e);
    const float mag = fast_sqrt(fmaf(y.x, y.x, y.y * y.y));
    float wp[NL];
#pragma unroll
    for (int r = 0; r < NL; ++r) {
        wp[r] = w[r];
        w[r] = fmaf(p.sw_k[r], w[r], mag);
    }
    if (CHECK && o.next_dec == t) store_planes<NL>(p, k.g4, o, mag, w, wp, active);
}

// STORE = false: the low-pass warm-up of a time chunk (run_tile<FORM, 2, 0> for every setting).
template <int FORM, int NL, bool STORE, int U, class K, class S, class E>
__device__ __forceinline__ void run_tile_sweep(const FusedParams& p, const K& k, S& s, float (&w)[NL], const E (&ee)[4],
                                               const E (&eo)[4], const float2* __restrict__ sxz,
                                               const float* __restrict__ sg, int t, int cnt, bool active, OutCtx& o) {
    int i = 0;
    for (; i + U <= cnt; i += U) {
        float xv[2 * U];
        float gv[U];
#pragma unroll
        for (int j = 0; j < U / 2; ++j) {
            const float4 v = *reinterpret_cast<const float4*>(sxz + i + 2 * j);
            xv[4 * j + 0] = v.x;
            xv[4 * j + 1] = v.y;
            xv[4 * j + 2] = v.z;
            xv[4 * j + 3] = v.w;
        }
#pragma unroll
        for (int j = 0; j < U / 4; ++j) {
            const float4 v = *reinterpret_cast<const float4*>(sg + i + 4 * j);
            gv[4 * j + 0] = v.x;
            gv[4 * j + 1] = v.y;
            gv[4 * j + 2] = v.z;
            gv[4 * j + 3] = v.w;
        }
        // the frame test is uniform in the warp: trips without a frame (most of them at step 160) run
        // without the per-sample compare
        if (STORE && o.next_dec < t + i + U) {
#pragma unroll
            for (int j = 0; j < U; ++j) {
                const float2 u = make_float2(xv[2 * j], xv[2 * j + 1]);
                if (j & 1) sweep_sample<FORM, NL, true>(p, k, s, w, u, gv[j], eo, t + i + j, active, o);
                else sweep_sample<FORM, NL, true>(p, k, s, w, u, gv[j], ee, t + i + j, active, o);
            }
        } else {
#pragma unroll
            for (int j = 0; j < U; ++j) {
                const float2 u = make_float2(xv[2 * j], xv[2 * j + 1]);
                if (j & 1) sweep_sample<FORM, NL, false>(p, k, s, w, u, gv[j], eo, t + i + j, active, o);
                else sweep_sample<FORM, NL, false>(p, k, s, w, u, gv[j], ee, t + i + j, active, o);
            }
        }
    }
    for (; i < cnt; ++i) {
        const float2 xz = sxz[i];
        if (i & 1) sweep_sample<FORM, NL, STORE>(p, k, s, w, xz, sg[i], eo, t + i, active, o);
        else sweep_sample<FORM, NL, STORE>(p, k, s, w, xz, sg[i], ee, t + i, active, o);
    }
}

struct Smem {
    float2 (*xz)[kTile];
    float (*g)[kTile];
    uint64_t* full;
    float* tr;   // CN: two 32 x (kCnW + 1) transposition tiles
};

// The whole CTA (= one warp = 32 adjacent channels) for one section form.
// EDGE: the edge residuals come from the per-utterance table (time-chunked batches) instead of
// the in-kernel pass.  SW > 0: the cutoff sweep (p.sw_planes planes of decimated frames) with SW one-pole
// states.
template <int FORM, int U, bool EDGE, bool WIN, bool CN, int SW = 0>
__device__ __forceinline__ void fused_body(const FusedParams& p, const Item& item, const Smem& sm, const int c) {
    const UttDesc ut = p.utts[item.utt];
    const int tid = threadIdx.x;
    const bool active = c < p.C;
    const int n = ut.n;
    const int N2 = ut.N2;
    const int mask = N2 - 1;
    const bool big = N2 >= kTile;  // TMA path: tiles never straddle the ring wrap

    using E = typename SectionTypes<FORM>::E;
    typename SectionTypes<FORM>::K k;
    load_coef<FORM>(p.chan, p.chan64, p.c_pad, c, active, k);

    // ---- tile schedule: E stream [tE0, n) (edge residuals), then M stream [ts, t1) ----
    // truncated-history lengths of THIS channel group (uniform in the CTA): the plan's lengths belong to
    // the bank's slowest channel
    const float wscale = p.chan[P_WSCALE * p.c_pad + item.cblock * kChanPerBlock];
    const int w_edge_g = group_warmup(p.w_edge, wscale);
    const int w_casc_g = group_warmup(p.w_casc, wscale);
    const int w_imag_g = group_warmup(p.w_imag, wscale);
    const int t0 = item.t0, t1 = item.t1;
    int tE0 = n - w_edge_g;
    tE0 = tE0 > 0 ? (tE0 / kTile) * kTile : 0;
    const bool need_env = WIN || p.env_t != nullptr || p.dec != nullptr || (CN && p.env_cn != nullptr);
    const bool need_imag = need_env && N2 > 2;  // N2 <= 2: the analytic signal is real
    // WIN: the window-store instantiation (f2_run_args.windows; no full-rate outputs by contract)
    const bool full_out = !WIN && (CN || p.env_t != nullptr);
    const int nE = (need_imag && !EDGE) ? (n - tE0 + kTile - 1) / kTile : 0;
    const int w_lpf = (p.lpf && need_env) ? p.w_lpf : 0;
    int ts, tenv;
    if (t0 - w_lpf - w_casc_g <= 0) {
        ts = need_imag ? -w_imag_g : 0;
        tenv = w_lpf > 0 ? 0 : t0;
    } else {
        ts = t0 - w_lpf - w_casc_g;
        tenv = t0 - w_lpf;
    }
    const int nM = (t1 - ts + kTile - 1) / kTile;
    const int total = nE + nM;

    const float2* xz_ring = p.xz + ut.ring_off;
    const float* g_ring = ut.g_tab ? ut.g_tab : p.G + ut.ring_off;
    const int g_shift = ut.g_tab ? ut.g_shift : 0;

    auto tile_time = [&](int kk) { return kk < nE ? tE0 + kk * kTile : ts + (kk - nE) * kTile; };
    auto issue = [&](int kk) {
        const int b = kk % kStages;
        const int tau = tile_time(kk) & mask;
        mbar_expect_tx(&sm.full[b], kTile * 12);
        tma_load_1d(&sm.xz[b][0], xz_ring + tau, kTile * 8, &sm.full[b]);
        tma_load_1d(&sm.g[b][0], g_ring + ((tau + g_shift) & mask), kTile * 4, &sm.full[b]);
    };

    if (big && tid == 0) {
        const int pre = total < kStages ? total : kStages;
        for (int kk = 0; kk < pre; ++kk) issue(kk);
    }

    typename SectionTypes<FORM>::S s;
    reset(s);
    float wsw[SW > 0 ? SW : 1];   // SW: the sweep's one-pole states
#pragma unroll
    for (int r = 0; r < (SW > 0 ? SW : 1); ++r) wsw[r] = 0.f;
    E ee[4] = {0, 0, 0, 0}, eo[4] = {0, 0, 0, 0};
    if (EDGE && need_imag && active) {
        if constexpr (FORM == 2) load_edge_entry(p.edge64, item.utt, p.C, c, ee, eo);
        else load_edge_entry(p.edge, item.utt, p.C, c, ee, eo);
    }
    OutCtx o;
    o.C = (size_t)p.C;
    o.step = p.step;
    o.env_scale = p.lpf ? k.g4 * p.lp_b0 : k.g4;
    o.env = p.env_t ? p.env_t + (size_t)(ut.full_off + t0) * o.C + (active ? c : 0) : nullptr;
    o.tr_g = o.tr_e = nullptr;
    o.cn_g = o.cn_e = nullptr;
    o.cn_n = n;
    o.cn_rows = 0;
    if (CN) {
        const int c0 = item.cblock * kChanPerBlock;
        o.cn_rows = min(kChanPerBlock, p.C - c0);
        const size_t elems = (size_t)ut.full_off * o.C + (size_t)c0 * (size_t)n;   // (C, n_u) blocks back to back
        o.tr_g = sm.tr;
        o.tr_e = p.gfb_cn ? sm.tr + 32 * kCnP : sm.tr;   // envelope alone: the only tile
        o.cn_g = p.gfb_cn ? reinterpret_cast<char*>(p.gfb_cn) + elems * (p.gfb_cn_f64 ? 8 : 4) : nullptr;
        o.cn_e = p.env_cn ? reinterpret_cast<char*>(p.env_cn) + elems * (p.env_cn_f64 ? 8 : 4) : nullptr;
    }
    {
        // first decimated frame at or after t0: t = phase + j*step
        int j0 = 0;
        if (t0 > p.phase) j0 = (t0 - p.phase + p.step - 1) / p.step;
        o.next_dec = p.phase + j0 * p.step;
        o.dec = p.dec ? p.dec + (size_t)(ut.dec_off + j0) * o.C + (active ? c : 0) : nullptr;
        o.wk = j0;
        o.nwin = 0;
        if (WIN) {  // window mode: o.dec walks the slot-0 entries instead
            const long long row0 = p.win_off[item.utt];
            o.nwin = (int)(p.win_off[item.utt + 1] - row0);
            o.dec = p.win + (size_t)(row0 + j0) * (size_t)p.win_dots * o.C + (active ? c : 0);
        }
    }

    for (int kk = 0; kk < total; ++kk) {
        const int b = kk % kStages;
        const int t = tile_time(kk);
        if (big) {
            mbar_wait(&sm.full[b], (uint32_t)((kk / kStages) & 1));
        } else {
            for (int i = tid; i < kTile; i += kChanPerBlock) {
                const int tau = (t + i) & mask;
                sm.xz[b][i] = xz_ring[tau];
                sm.g[b][i] = g_ring[(tau + g_shift) & mask];
            }
            __syncwarp();
        }
        const float2* sxz = &sm.xz[b][0];
        const float* sg = &sm.g[b][0];

        if (kk < nE) {
            // real cascade only, zero state at tE0 (exact when tE0 == 0)
            const int cnt = min(kTile, n - t);
            for (int i = 0; i < cnt; ++i) cascade_real<FORM>(k, s, sxz[i].x);
            if (kk == nE - 1) {
                E e0[4], e1[4];
                edge_residuals<FORM>(k, s, e0, e1);
                edge_parity(n, e0, e1, ee, eo);
                reset(s);
            }
        } else {
            const int cnt = min(kTile, t1 - t);
            if (t < 0) {
                // periodic warm-up of the imaginary path (t is a multiple of kTile: parity of t+i = parity of i)
#pragma unroll 2
                for (int i = 0; i < cnt; i += 2) {
                    const float4 xz2 = *reinterpret_cast<const float4*>(sxz + i);
                    const float2 g2 = *reinterpret_cast<const float2*>(sg + i);
                    cascade_imag<FORM>(k, s, xz2.y, g2.x, ee);
                    cascade_imag<FORM>(k, s, xz2.w, g2.y, eo);
                }
            } else if (t < tenv) {
                run_tile<FORM, 0, 0, false, U>(p, k, s, ee, eo, sxz, sg, t, cnt, active, o);
            } else if (t < t0) {
                if constexpr (SW > 0) run_tile_sweep<FORM, SW, false, U>(p, k, s, wsw, ee, eo, sxz, sg, t, cnt, active, o);
                else run_tile<FORM, 2, 0, false, U>(p, k, s, ee, eo, sxz, sg, t, cnt, active, o);
            } else if constexpr (SW > 0) {
                run_tile_sweep<FORM, SW, true, U>(p, k, s, wsw, ee, eo, sxz, sg, t, cnt, active, o);
            } else if (full_out) {
                // full-rate stores: the 8-sample unroll is the faster one (3.9 vs 4.9 ms on 256 utterances)
                constexpr int UF = U < 8 ? U : 8;
                if (p.lpf && need_env) run_tile<FORM, 2, 2, false, UF, CN>(p, k, s, ee, eo, sxz, sg, t, cnt, active, o);
                else if (need_env) run_tile<FORM, 1, 2, false, UF, CN>(p, k, s, ee, eo, sxz, sg, t, cnt, active, o);
                else run_tile<FORM, 0, 2, false, UF, CN>(p, k, s, ee, eo, sxz, sg, t, cnt, active, o);
            } else if (WIN) {
                if (p.lpf) run_tile<FORM, 2, 3, false, U>(p, k, s, ee, eo, sxz, sg, t, cnt, active, o);
                else run_tile<FORM, 1, 3, false, U>(p, k, s, ee, eo, sxz, sg, t, cnt, active, o);
            } else {
                if (p.lpf) run_tile<FORM, 2, 1, false, U>(p, k, s, ee, eo, sxz, sg, t, cnt, active, o);
                else run_tile<FORM, 1, 1, false, U>(p, k, s, ee, eo, sxz, sg, t, cnt, active, o);
            }
        }
        __syncwarp();  // every lane is done with buffer b
        if (big && tid == 0 && kk + kStages < total) issue(kk + kStages);
    }
}

// One CTA = one warp: the sections' form is uniform in the CTA, so the two float32 forms are two
// separate straight-line programs behind one branch, and a warp that finishes early (direct
// form: 3 FMAs per section instead of 4) frees its slot for the next work item instead of
// waiting at a CTA barrier for slower warps (measured: DESIGN.md section 6).
// F64: the work items of FORM 2 groups (float64 sections), in instantiations of their own: a third
// branch in the float32 instantiations would raise their register count for every bank.
template <bool F64, int MINB, int U, bool EDGE, bool WIN, bool CN>
__global__ void __launch_bounds__(kChanPerBlock, MINB) fused_kernel(const FusedParams p) {
    static_assert(kChanPerBlock == 32, "one warp per CTA: __syncwarp is the only barrier used");
    __shared__ __align__(128) float2 s_xz[kStages][kTile];
    __shared__ __align__(128) float s_g[kStages][kTile];
    __shared__ __align__(8) uint64_t s_full[kStages];
    extern __shared__ float s_tr[];   // CN: one 32 x (kCnW + 1) staging tile per (C, n) output (dynamic: 0, 1 or 2 tiles)
    if (threadIdx.x == 0) {
        for (int b = 0; b < kStages; ++b) mbar_init(&s_full[b], 1);
        mbar_fence_init();
    }
    __syncwarp();
    const Item item = p.items[blockIdx.x];
    const int c = item.cblock * kChanPerBlock + threadIdx.x;
    const Smem sm{s_xz, s_g, s_full, s_tr};
    if constexpr (F64) {
        fused_body<2, U, EDGE, WIN, CN>(p, item, sm, c);
    } else {
        // per group of 32 channels (c_pad = C rounded up to 32): min over the group of 1 + B1 + B2
        const float group_cy = p.chan[P_FORM * p.c_pad + c];
        if (group_cy >= p.direct_min_cy) fused_body<1, U, EDGE, WIN, CN>(p, item, sm, c);
        else fused_body<0, U, EDGE, WIN, CN>(p, item, sm, c);
    }
}

// The cutoff sweep (FusedParams::sw_planes > 0): decimated frames only, NL one-pole states.
template <bool F64, int MINB, int U, bool EDGE, int NL>
__global__ void __launch_bounds__(kChanPerBlock, MINB) fused_sweep_kernel(const FusedParams p) {
    __shared__ __align__(128) float2 s_xz[kStages][kTile];
    __shared__ __align__(128) float s_g[kStages][kTile];
    __shared__ __align__(8) uint64_t s_full[kStages];
    if (threadIdx.x == 0) {
        for (int b = 0; b < kStages; ++b) mbar_init(&s_full[b], 1);
        mbar_fence_init();
    }
    __syncwarp();
    const Item item = p.items[blockIdx.x];
    const int c = item.cblock * kChanPerBlock + threadIdx.x;
    const Smem sm{s_xz, s_g, s_full, nullptr};
    if constexpr (F64) {
        fused_body<2, U, EDGE, false, false, NL>(p, item, sm, c);
    } else {
        const float group_cy = p.chan[P_FORM * p.c_pad + c];
        if (group_cy >= p.direct_min_cy) fused_body<1, U, EDGE, false, false, NL>(p, item, sm, c);
        else fused_body<0, U, EDGE, false, false, NL>(p, item, sm, c);
    }
}

template <bool F64, int MINB, int U, int NL>
static void launch_sweep_nl(const FusedParams& p, int n_items, cudaStream_t stream) {
    if (F64 ? p.edge64 != nullptr : p.edge != nullptr)
        fused_sweep_kernel<F64, MINB, U, true, NL><<<n_items, kChanPerBlock, 0, stream>>>(p);
    else
        fused_sweep_kernel<F64, MINB, U, false, NL><<<n_items, kChanPerBlock, 0, stream>>>(p);
}

template <bool F64, int MINB, int U>
static void launch_variant(const FusedParams& p, int n_items, cudaStream_t stream) {
    const bool edge = F64 ? p.edge64 != nullptr : p.edge != nullptr;
    if (p.win) {
        if (edge) fused_kernel<F64, MINB, U, true, true, false><<<n_items, kChanPerBlock, 0, stream>>>(p);
        else fused_kernel<F64, MINB, U, false, true, false><<<n_items, kChanPerBlock, 0, stream>>>(p);
    } else if (p.gfb_cn || p.env_cn) {
        // (C, n) outputs written by the kernel itself (own instantiation: two transposition tiles per CTA)
        const size_t tiles = ((p.gfb_cn ? 1 : 0) + (p.env_cn ? 1 : 0)) * (size_t)(32 * kCnP) * sizeof(float);
        if (edge) fused_kernel<F64, MINB, U, true, false, true><<<n_items, kChanPerBlock, tiles, stream>>>(p);
        else fused_kernel<F64, MINB, U, false, false, true><<<n_items, kChanPerBlock, tiles, stream>>>(p);
    } else {
        if (edge) fused_kernel<F64, MINB, U, true, false, false><<<n_items, kChanPerBlock, 0, stream>>>(p);
        else fused_kernel<F64, MINB, U, false, false, false><<<n_items, kChanPerBlock, 0, stream>>>(p);
    }
}

cudaError_t launch_fused(const FusedParams& p, int n_items, bool float64, cudaStream_t stream) {
    if (n_items <= 0) return cudaSuccess;
    if (p.sw_planes > 0) {
        // float32: one instantiation per number of one-pole states, so that a setting without low-pass
        // costs no FMA per sample.  Four states do not fit 128 registers (16 CTAs per SM) with 16 samples per
        // loop trip without spilling: that instantiation loads 8 per trip.  FORM 2 (float64 sections dominate
        // its time): four states always.
        if (float64) launch_sweep_nl<true, 12, 8, 4>(p, n_items, stream);
        else if (p.sw_lp <= 1) launch_sweep_nl<false, 16, 16, 1>(p, n_items, stream);
        else if (p.sw_lp == 2) launch_sweep_nl<false, 16, 16, 2>(p, n_items, stream);
        else if (p.sw_lp == 3) launch_sweep_nl<false, 16, 16, 3>(p, n_items, stream);
        else launch_sweep_nl<false, 16, 8, 4>(p, n_items, stream);
        return cudaGetLastError();
    }
    // float32: 16 one-warp CTAs per SM, 16 samples per loop trip (profiles/r01j_tune_*.log, r01m); the
    // window-store mode is its own instantiation so that the other modes keep their code.  FORM 2: 12 and 8.
    if (float64) launch_variant<true, 12, 8>(p, n_items, stream);
    else launch_variant<false, 16, 16>(p, n_items, stream);
    return cudaGetLastError();
}

}  // namespace f2
