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
// packed FFMA2/FADD2 instructions.  Input of a section (z_k = A1k/A0):
//     in = u[t] + z_k*u[t-1]     (+ e_k*G[t] on the imaginary half)
// Section, per group of 32 channels (the form is uniform in a CTA):
//   direct form  y = (in - B2*y[t-2]) - B1*y[t-1]           3 packed + 1 scalar instruction
//   delta form   q = cq*q + in - cy*y ;  y = y + q           4 packed + 1 scalar instruction
//                (state y[t-1] and q = y[t-1]-y[t-2]; cq = B2, cy = 1+B1+B2)
// The delta form keeps float32 round-off and coefficient quantisation harmless for poles
// 0.039 rad from z=1 (SURVEY.md H2); the direct form is used where 1+B1+B2 = |1-pole|^2 is
// large enough for it to be as accurate (FusedParams::direct_min_cy, DESIGN.md section 3).
// FORM 2 (float64 direct form, exact coefficients) runs the groups a plan created with
// F2_PLAN_FLOAT64_SECTIONS found float32 unable to hold to the tolerance, in fused_kernel64 (DESIGN.md 2 (iii)).
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

#include <stdlib.h>

namespace f2 {

// FORM 0 (delta form): cq = B2, ncy = -(1+B1+B2); state q = y[t-1]-y[t-2].
// FORM 1 (direct form): cq holds -B2, ncy holds -B1;   state q = y[t-2].
struct Coef {
    float2 z[4];    // A1k/A0 (the stage's zero), broadcast to both halves
    float2 cq[4];
    float2 ncy[4];
    float2 zn[3];   // direct form only: z[i+1] - B1 of section i (next section's input from this one's state)
    float g4;       // A0^4/gain: the cascade's output scale
};

struct State {
    float2 y[4];
    float2 q[4];
    float2 up;    // previous stage-1 input (x[t-1], xi[t-1])
    float l;      // one-pole low-pass state w[t] = k*w[t-1] + |y[t]|
    float wprev;  // w[t-1] (the low-pass output is b0*(w[t] + w[t-1]))
};

__device__ __forceinline__ void reset(State& s) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        s.y[i] = make_float2(0.f, 0.f);
        s.q[i] = make_float2(0.f, 0.f);
    }
    s.up = make_float2(0.f, 0.f);
    s.l = 0.f;
    s.wprev = 0.f;
}

// One sample through the packed (real, imag) 4-stage cascade.  e[] = injection
// coefficients for this sample's parity, g = G[t].
template <int FORM>
__device__ __forceinline__ float2 cascade(const Coef& k, State& s, float2 u, float g, const float (&e)[4]) {
    float2 up = s.up;
    s.up = u;
    if (FORM == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float2 in = __ffma2_rn(k.z[i], up, u);
            in.y = fmaf(e[i], g, in.y);
            const float2 yo = s.y[i];
            float2 qn = __ffma2_rn(k.cq[i], s.q[i], in);
            qn = __ffma2_rn(k.ncy[i], yo, qn);
            const float2 yn = __fadd2_rn(yo, qn);
            s.q[i] = qn;
            s.y[i] = yn;
            up = yo;
            u = yn;
        }
        return u;
    }
    // Direct form.  With acc = in - B2*y[t-2], the section output is y = acc - B1*y[t-1] and the
    // NEXT section's input is z'*y[t-1] + y = acc + (z' - B1)*y[t-1]: both read (y[t-1], acc), so
    // the second issues right behind the first without waiting for y (k.zn = z' - B1).
    float2 in = __ffma2_rn(k.z[0], up, u);
    in.y = fmaf(e[0], g, in.y);
    float2 yn;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 yo = s.y[i];
        const float2 acc = __ffma2_rn(k.cq[i], s.q[i], in);
        yn = __ffma2_rn(k.ncy[i], yo, acc);
        if (i < 3) {
            in = __ffma2_rn(k.zn[i], yo, acc);
            in.y = fmaf(e[i + 1], g, in.y);
        }
        s.q[i] = yo;
        s.y[i] = yn;
    }
    return yn;
}

template <int FORM>
__device__ __forceinline__ void cascade_real(const Coef& k, State& s, float u) {
    float up = s.up.x;
    s.up.x = u;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float in = fmaf(k.z[i].x, up, u);
        const float yo = s.y[i].x;
        float yn;
        if (FORM == 0) {
            float qn = fmaf(k.cq[i].x, s.q[i].x, in);
            qn = fmaf(k.ncy[i].x, yo, qn);
            yn = yo + qn;
            s.q[i].x = qn;
        } else {
            yn = fmaf(k.ncy[i].x, yo, fmaf(k.cq[i].x, s.q[i].x, in));
            s.q[i].x = yo;
        }
        s.y[i].x = yn;
        up = yo;
        u = yn;
    }
}

// Imaginary half only (scalar): the periodic warm-up before t = 0, where the real half is
// identically zero -- 16 scalar FMAs per sample instead of 12-16 packed instructions.
template <int FORM>
__device__ __forceinline__ void cascade_imag(const Coef& k, State& s, float u, float g, const float (&e)[4]) {
    float up = s.up.y;
    s.up.y = u;
    if (FORM == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float in = fmaf(e[i], g, fmaf(k.z[i].x, up, u));
            const float yo = s.y[i].y;
            float qn = fmaf(k.cq[i].x, s.q[i].y, in);
            qn = fmaf(k.ncy[i].x, yo, qn);
            const float yn = yo + qn;
            s.q[i].y = qn;
            s.y[i].y = yn;
            up = yo;
            u = yn;
        }
    } else {
        float in = fmaf(e[0], g, fmaf(k.z[0].x, up, u));
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float yo = s.y[i].y;
            const float acc = fmaf(k.cq[i].x, s.q[i].y, in);
            const float yn = fmaf(k.ncy[i].x, yo, acc);
            if (i < 3) in = fmaf(e[i + 1], g, fmaf(k.zn[i].x, yo, acc));
            s.q[i].y = yo;
            s.y[i].y = yn;
        }
    }
}

// Residuals of the zero-padded ring equation at ring positions n and n+1, from the stage states
// after sample n-1 (y = y[n-1]; u = the stage's input at n-1), in the scaled stage variables:
//   e0 = b1*y[n-1] + b2*y[n-2] - z_k*u[n-1]      e1 = b2*y[n-1]
// FORM 0: b1*y[n-1] + b2*y[n-2] = (cy-1)*y - cq*q with q = y[n-1]-y[n-2];  FORM 1: directly.
template <int FORM>
__device__ __forceinline__ void edge_residuals(const Coef& k, const State& s, float (&e0)[4], float (&e1)[4]) {
    float uprev = s.up.x;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (FORM == 0) {
            const float cy = -k.ncy[i].x;
            e0[i] = fmaf(cy - 1.0f, s.y[i].x, -k.cq[i].x * s.q[i].x) - k.z[i].x * uprev;
            e1[i] = k.cq[i].x * s.y[i].x;
        } else {
            e0[i] = -fmaf(k.ncy[i].x, s.y[i].x, k.cq[i].x * s.q[i].x) - k.z[i].x * uprev;
            e1[i] = -k.cq[i].x * s.y[i].x;
        }
        uprev = s.y[i].x;
    }
}

// ---- FORM 2: float64 direct-form sections (groups float32 cannot hold to the tolerance) ----------------
// Exact design coefficients (no dither), y = in - b1*y[t-1] - b2*y[t-2] with the same zn = z' - b1 trick as
// FORM 1.  Ring samples and G stay float and are widened when read; the injection e*G is formed in double;
// g4 is applied in double, so the value that leaves the cascade is the float of the scaled output and the
// float code after it (magnitude, low-pass, stores) runs with a unit scale.
struct Coef64 {
    double z[4];
    double nb1, nb2;  // -b1, -b2
    double zn[3];     // z[i+1] - b1
    double gd;        // A0^4/gain
    float g4;         // 1: the float-side output scale of run_tile
};

struct State64 {
    double yr[4], yi[4];    // y[t-1]
    double qr[4], qi[4];    // y[t-2]
    double upr, upi;        // previous stage-1 input
    float l;
    float wprev;
};

__device__ __forceinline__ void reset(State64& s) {
#pragma unroll
    for (int i = 0; i < 4; ++i) s.yr[i] = s.yi[i] = s.qr[i] = s.qi[i] = 0.0;
    s.upr = s.upi = 0.0;
    s.l = 0.f;
    s.wprev = 0.f;
}

template <int FORM>
__device__ __forceinline__ float2 cascade(const Coef64& k, State64& s, float2 u, float g, const double (&e)[4]) {
    const double ur = u.x, ui = u.y, gd = g;
    double inr = fma(k.z[0], s.upr, ur);
    double ini = fma(e[0], gd, fma(k.z[0], s.upi, ui));
    s.upr = ur;
    s.upi = ui;
    double yr = 0.0, yi = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const double ar = fma(k.nb2, s.qr[i], inr), ai = fma(k.nb2, s.qi[i], ini);
        const double yor = s.yr[i], yoi = s.yi[i];
        yr = fma(k.nb1, yor, ar);
        yi = fma(k.nb1, yoi, ai);
        if (i < 3) {
            inr = fma(k.zn[i], yor, ar);
            ini = fma(e[i + 1], gd, fma(k.zn[i], yoi, ai));
        }
        s.qr[i] = yor;
        s.qi[i] = yoi;
        s.yr[i] = yr;
        s.yi[i] = yi;
    }
    return make_float2((float)(k.gd * yr), (float)(k.gd * yi));
}

template <int FORM>
__device__ __forceinline__ void cascade_real(const Coef64& k, State64& s, float u) {
    const double ur = u;
    double in = fma(k.z[0], s.upr, ur);
    s.upr = ur;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const double a = fma(k.nb2, s.qr[i], in);
        const double yo = s.yr[i];
        if (i < 3) in = fma(k.zn[i], yo, a);
        s.qr[i] = yo;
        s.yr[i] = fma(k.nb1, yo, a);
    }
}

template <int FORM>
__device__ __forceinline__ void cascade_imag(const Coef64& k, State64& s, float u, float g, const double (&e)[4]) {
    const double ui = u, gd = g;
    double in = fma(e[0], gd, fma(k.z[0], s.upi, ui));
    s.upi = ui;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const double a = fma(k.nb2, s.qi[i], in);
        const double yo = s.yi[i];
        if (i < 3) in = fma(e[i + 1], gd, fma(k.zn[i], yo, a));
        s.qi[i] = yo;
        s.yi[i] = fma(k.nb1, yo, a);
    }
}

// e0 = b1*y[n-1] + b2*y[n-2] - z_k*u[n-1],  e1 = b2*y[n-1]  (as FORM 1, in double)
template <int FORM>
__device__ __forceinline__ void edge_residuals(const Coef64& k, const State64& s, double (&e0)[4], double (&e1)[4]) {
    double uprev = s.upr;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        e0[i] = -fma(k.nb1, s.yr[i], k.nb2 * s.qr[i]) - k.z[i] * uprev;
        e1[i] = -k.nb2 * s.yr[i];
        uprev = s.yr[i];
    }
}

// Coefficients of this thread's channel (inactive lanes: zeros, as the float forms do)
template <int FORM>
__device__ __forceinline__ void load_coef(const FusedParams& p, int c, bool active, Coef& k) {
    const float* cp = p.chan + (active ? c : 0);
    const float on = active ? 1.f : 0.f;
    k.g4 = on * cp[P_G4 * p.c_pad];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float z = on * cp[(P_Z + i) * p.c_pad];
        const float cq = on * (FORM == 1 ? -cp[(P_CQ + i) * p.c_pad] : cp[(P_CQ + i) * p.c_pad]);
        const float ncy = on * cp[((FORM == 1 ? P_NB1 : P_NCY) + i) * p.c_pad];
        k.z[i] = make_float2(z, z);
        k.cq[i] = make_float2(cq, cq);
        k.ncy[i] = make_float2(ncy, ncy);
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const float zn = FORM == 1 ? k.z[i + 1].x + k.ncy[i].x : 0.f;
        k.zn[i] = make_float2(zn, zn);
    }
}

template <int FORM>
__device__ __forceinline__ void load_coef(const FusedParams& p, int c, bool active, Coef64& k) {
    const double* cp = p.chan64 + (active ? c : 0);
    const double on = active ? 1.0 : 0.0;
    k.gd = on * cp[P64_G4 * p.c_pad];
    k.g4 = 1.f;
    k.nb1 = -on * cp[P64_B1 * p.c_pad];
    k.nb2 = -on * cp[P64_B2 * p.c_pad];
#pragma unroll
    for (int i = 0; i < 4; ++i) k.z[i] = on * cp[(P64_Z + i) * p.c_pad];
#pragma unroll
    for (int i = 0; i < 3; ++i) k.zn[i] = k.z[i + 1] + k.nb1;
}

// Time-chunked batches: this channel's edge residuals from the per-utterance table
__device__ __forceinline__ void load_edge(const FusedParams& p, int utt, int c, float (&ee)[4], float (&eo)[4]) {
    const float4* e = reinterpret_cast<const float4*>(p.edge + ((size_t)utt * p.C + c) * 8);
    const float4 v0 = __ldg(e), v1 = __ldg(e + 1);
    ee[0] = v0.x; ee[1] = v0.y; ee[2] = v0.z; ee[3] = v0.w;
    eo[0] = v1.x; eo[1] = v1.y; eo[2] = v1.z; eo[3] = v1.w;
}

__device__ __forceinline__ void load_edge(const FusedParams& p, int utt, int c, double (&ee)[4], double (&eo)[4]) {
    const double* e = p.edge64 + ((size_t)utt * p.C + c) * 8;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        ee[i] = __ldg(e + i);
        eo[i] = __ldg(e + 4 + i);
    }
}

template <int FORM> struct SectionTypes { using K = Coef; using S = State; using E = float; };
template <> struct SectionTypes<2> { using K = Coef64; using S = State64; using E = double; };

// ENV: 0 = cascade only, 1 = magnitude, 2 = magnitude + low-pass.
// OUT: 0 = nothing leaves the kernel (warm-up), 1 = decimated frames only, 2 = full-rate
//      time-major stores (and decimated frames when asked), 3 = every decimated frame goes
//      straight into the (up to win_dots) window rows that contain it.
struct OutCtx {
    float* gfb;     // points at sample t of this thread's channel (or null)
    float* env;
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
    // of one channel per store instruction (128 / 256 contiguous bytes), kCnW per row instead of a time-major scratch
    // matrix and a transposing second kernel.
    float* tr_g;    // shared-memory tiles (or null)
    float* tr_e;
    char* cn_g;     // element (first channel of this CTA, sample 0) of the utterance's (C, n) block (or null)
    char* cn_e;
    int cn_n;       // samples per row
    int cn_rows;    // channels of this CTA that exist (<= 32)
    int cn_f64;
};

// (C, n) staging tile: 32 channels x kCnW samples (+1 column of padding).  Longer runs per channel row make
// the stores friendlier to DRAM pages (every row of a tile lands in a different page of the (C, n) matrix).
#ifndef F2_CN_W
#define F2_CN_W 128
#endif
constexpr int kCnW = F2_CN_W;
constexpr int kCnP = kCnW + 1;

// rows of the staged tile -> global: samples [tb, tb + cnt) of every channel of this CTA
__device__ __forceinline__ void flush_cn(const float* tr, char* base, const OutCtx& o, int tb, int cnt) {
    __syncwarp();
    const int lane = threadIdx.x;
    if (o.cn_f64) {
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
            if (OUT == 2 && !CN) {
                if (o.gfb && active) __stcs(o.gfb + (size_t)j * o.C, k.g4 * y.x);
                if (ENV > 0 && o.env && active) {
                    const float v = ENV == 2 ? ev[j] + (j > 0 ? ev[j > 0 ? j - 1 : 0] : wprev) : ev[j];
                    __stcs(o.env + (size_t)j * o.C, o.env_scale * v);
                }
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
        if (OUT == 2 && !CN) {
            if (o.gfb) o.gfb += U * o.C;
            if (o.env) o.env += U * o.C;
        }
        if (OUT == 2 && CN && ((t + i + U) & (kCnW - 1)) == 0) {
            if (o.cn_g) flush_cn(o.tr_g, o.cn_g, o, t + i + U - kCnW, kCnW);
            if (ENV > 0 && o.cn_e) flush_cn(o.tr_e, o.cn_e, o, t + i + U - kCnW, kCnW);
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
        if (OUT == 2 && !CN) {
            if (o.gfb) {
                if (active) __stcs(o.gfb, k.g4 * y.x);
                o.gfb += o.C;
            }
            if (ENV > 0 && o.env) {
                if (active) __stcs(o.env, o.env_scale * out);
                o.env += o.C;
            }
        }
        if (OUT == 2 && CN) {
            const int col = (t + i) & (kCnW - 1);
            if (o.cn_g) o.tr_g[threadIdx.x * kCnP + col] = k.g4 * y.x;
            if (ENV > 0 && o.cn_e) o.tr_e[threadIdx.x * kCnP + col] = o.env_scale * out;
            if (col == kCnW - 1) {
                if (o.cn_g) flush_cn(o.tr_g, o.cn_g, o, t + i - (kCnW - 1), kCnW);
                if (ENV > 0 && o.cn_e) flush_cn(o.tr_e, o.cn_e, o, t + i - (kCnW - 1), kCnW);
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
        if (o.cn_g) flush_cn(o.tr_g, o.cn_g, o, t + cnt - rest, rest);
        if (ENV > 0 && o.cn_e) flush_cn(o.tr_e, o.cn_e, o, t + cnt - rest, rest);
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
// the in-kernel pass.
template <int FORM, int U, bool EDGE, bool WIN, bool CN>
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
    load_coef<FORM>(p, c, active, k);

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
    const bool full_out = !WIN && (CN || p.gfb_t != nullptr || p.env_t != nullptr);
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
    E ee[4] = {0, 0, 0, 0}, eo[4] = {0, 0, 0, 0};
    if (EDGE && need_imag && active) load_edge(p, item.utt, c, ee, eo);
    OutCtx o;
    o.C = (size_t)p.C;
    o.step = p.step;
    o.env_scale = p.lpf ? k.g4 * p.lp_b0 : k.g4;
    o.gfb = p.gfb_t ? p.gfb_t + (size_t)(ut.full_off + t0) * o.C + (active ? c : 0) : nullptr;
    o.env = p.env_t ? p.env_t + (size_t)(ut.full_off + t0) * o.C + (active ? c : 0) : nullptr;
    o.tr_g = o.tr_e = nullptr;
    o.cn_g = o.cn_e = nullptr;
    o.cn_n = n;
    o.cn_f64 = p.cn_f64;
    o.cn_rows = 0;
    if (CN) {
        const int c0 = item.cblock * kChanPerBlock;
        o.cn_rows = min(kChanPerBlock, p.C - c0);
        const size_t esize = p.cn_f64 ? 8 : 4;
        const size_t block = ((size_t)ut.full_off * o.C + (size_t)c0 * (size_t)n) * esize;   // (C, n_u) blocks back to back
        o.tr_g = sm.tr;
        o.tr_e = p.gfb_cn ? sm.tr + 32 * kCnP : sm.tr;   // envelope alone: the only tile
        o.cn_g = p.gfb_cn ? reinterpret_cast<char*>(p.gfb_cn) + block : nullptr;
        o.cn_e = p.env_cn ? reinterpret_cast<char*>(p.env_cn) + block : nullptr;
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
                // (t - n) odd -> e0 multiplies G[t]; even -> e1
                const bool n_odd = (n & 1) != 0;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    ee[i] = n_odd ? e0[i] : e1[i];
                    eo[i] = n_odd ? e1[i] : e0[i];
                }
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
                run_tile<FORM, 2, 0, false, U>(p, k, s, ee, eo, sxz, sg, t, cnt, active, o);
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

// One CTA = one warp: the sections' form is uniform in the CTA, so the two forms are two
// separate straight-line programs behind one branch, and a warp that finishes early (direct
// form: 3 FMAs per section instead of 4) frees its slot for the next work item instead of
// waiting at a CTA barrier for slower warps (measured: DESIGN.md section 6).
template <int MINB, int U, bool EDGE, bool WIN, bool CN>
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
    // per group of 32 channels (c_pad = C rounded up to 32): min over the group of 1 + B1 + B2
    const float group_cy = p.chan[P_FORM * p.c_pad + c];
#ifdef F2_SINGLE_FORM
    (void)group_cy;
    fused_body<F2_SINGLE_FORM, U, EDGE, WIN, CN>(p, item, sm, c);
#else
    if (group_cy >= p.direct_min_cy) fused_body<1, U, EDGE, WIN, CN>(p, item, sm, c);
    else fused_body<0, U, EDGE, WIN, CN>(p, item, sm, c);
#endif
}

template <int MINB, int U>
static void launch_variant(const FusedParams& p, int n_items, cudaStream_t stream) {
    if (p.win) {
        if (p.edge) fused_kernel<MINB, U, true, true, false><<<n_items, kChanPerBlock, 0, stream>>>(p);
        else fused_kernel<MINB, U, false, true, false><<<n_items, kChanPerBlock, 0, stream>>>(p);
    } else if (p.gfb_cn || p.env_cn) {
        // (C, n) outputs written by the kernel itself (own instantiation: two transposition tiles per CTA)
        const size_t tiles = ((p.gfb_cn ? 1 : 0) + (p.env_cn ? 1 : 0)) * (size_t)(32 * kCnP) * sizeof(float);
        if (p.edge) fused_kernel<MINB, U, true, false, true><<<n_items, kChanPerBlock, tiles, stream>>>(p);
        else fused_kernel<MINB, U, false, false, true><<<n_items, kChanPerBlock, tiles, stream>>>(p);
    } else {
        if (p.edge) fused_kernel<MINB, U, true, false, false><<<n_items, kChanPerBlock, 0, stream>>>(p);
        else fused_kernel<MINB, U, false, false, false><<<n_items, kChanPerBlock, 0, stream>>>(p);
    }
}

// FORM 2 (float64 sections) in its own kernel: a third branch in fused_kernel would raise the register
// count of the float32 forms for every bank.
template <int MINB, int U, bool EDGE, bool WIN, bool CN>
__global__ void __launch_bounds__(kChanPerBlock, MINB) fused_kernel64(const FusedParams p) {
    __shared__ __align__(128) float2 s_xz[kStages][kTile];
    __shared__ __align__(128) float s_g[kStages][kTile];
    __shared__ __align__(8) uint64_t s_full[kStages];
    extern __shared__ float s_tr[];
    if (threadIdx.x == 0) {
        for (int b = 0; b < kStages; ++b) mbar_init(&s_full[b], 1);
        mbar_fence_init();
    }
    __syncwarp();
    const Item item = p.items[blockIdx.x];
    const int c = item.cblock * kChanPerBlock + threadIdx.x;
    const Smem sm{s_xz, s_g, s_full, s_tr};
    fused_body<2, U, EDGE, WIN, CN>(p, item, sm, c);
}

cudaError_t launch_fused64(const FusedParams& p, int n_items, cudaStream_t stream) {
    if (n_items <= 0) return cudaSuccess;
    constexpr int MINB = 12, U = 8;
    const bool edge = p.edge64 != nullptr;
    if (p.win) {
        if (edge) fused_kernel64<MINB, U, true, true, false><<<n_items, kChanPerBlock, 0, stream>>>(p);
        else fused_kernel64<MINB, U, false, true, false><<<n_items, kChanPerBlock, 0, stream>>>(p);
    } else if (p.gfb_cn || p.env_cn) {
        const size_t tiles = ((p.gfb_cn ? 1 : 0) + (p.env_cn ? 1 : 0)) * (size_t)(32 * kCnP) * sizeof(float);
        if (edge) fused_kernel64<MINB, U, true, false, true><<<n_items, kChanPerBlock, tiles, stream>>>(p);
        else fused_kernel64<MINB, U, false, false, true><<<n_items, kChanPerBlock, tiles, stream>>>(p);
    } else {
        if (edge) fused_kernel64<MINB, U, true, false, false><<<n_items, kChanPerBlock, 0, stream>>>(p);
        else fused_kernel64<MINB, U, false, false, false><<<n_items, kChanPerBlock, 0, stream>>>(p);
    }
    return cudaGetLastError();
}

cudaError_t launch_fused(const FusedParams& p, int n_items, cudaStream_t stream) {
    if (n_items <= 0) return cudaSuccess;
#ifdef F2_FUSED_TUNING
    // development build (make EXTRA=-DF2_FUSED_TUNING): F2_FUSED_VARIANT = "<min CTAs per SM><unroll>"
    static int variant = -1;
    if (variant < 0) {
        const char* v = getenv("F2_FUSED_VARIANT");
        variant = v ? atoi(v) : 0;
    }
    if (variant == 168) {
        launch_variant<16, 8>(p, n_items, stream);
        return cudaGetLastError();
    }
    if (variant == 208) {
        launch_variant<20, 8>(p, n_items, stream);
        return cudaGetLastError();
    }
#endif
    // 16 one-warp CTAs per SM, 16 samples per loop trip (profiles/r01j_tune_*.log, r01m); the
    // window-store mode is its own instantiation so that the other modes keep their code
    launch_variant<16, 16>(p, n_items, stream);
    return cudaGetLastError();
}

}  // namespace f2
