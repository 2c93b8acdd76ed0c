// f2_sections.cuh -- the four-section gammatone cascade, defined once for every kernel that runs it
// (f2_fused.cu, f2_edge.cu) and for the host probe that predicts its float32 error (f2_capi.cu).
//
// Input of a section (z_k = A1k/A0):
//     in = u[t] + z_k*u[t-1]     (+ e_k*G[t] on the imaginary half)
// Section forms:
//   FORM 0  delta form   q = cq*q + in - cy*y ;  y = y + q      (state y[t-1], q = y[t-1]-y[t-2]; cq = B2, cy = 1+B1+B2)
//   FORM 1  direct form  y = (in - B2*y[t-2]) - B1*y[t-1]
//   FORM 2  float64 direct form with the exact design coefficients
// Every stage is computed without its common numerator gain a0 (stage k holds y_k / a0^k); g4 = a0^4 is
// applied where a value leaves the cascade.
#pragma once
#include "f2_common.cuh"

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

__host__ __device__ __forceinline__ void reset(State& s) {
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

// Real half only (scalar): the edge-residual passes, and on the host the float32 half of the bank probe.
template <int FORM>
__host__ __device__ __forceinline__ void cascade_real(const Coef& k, State& s, float u) {
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

template <int FORM> struct SectionTypes { using K = Coef; using S = State; using E = float; };
template <> struct SectionTypes<2> { using K = Coef64; using S = State64; using E = double; };

// Coefficients of channel c from the parameter block chan[i * c_pad + c] (FORM 0/1) or the float64 block
// chan64 (FORM 2); the other block is not read.  Inactive lanes get zeros.
template <int FORM>
__host__ __device__ __forceinline__ void load_coef(const float* chan, const double* chan64, int c_pad, int c,
                                                   bool active, Coef& k) {
    const float* cp = chan + (active ? c : 0);
    const float on = active ? 1.f : 0.f;
    k.g4 = on * cp[P_G4 * c_pad];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float z = on * cp[(P_Z + i) * c_pad];
        const float cq = on * (FORM == 1 ? -cp[(P_CQ + i) * c_pad] : cp[(P_CQ + i) * c_pad]);
        const float ncy = on * cp[((FORM == 1 ? P_NB1 : P_NCY) + i) * c_pad];
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
__device__ __forceinline__ void load_coef(const float* chan, const double* chan64, int c_pad, int c, bool active,
                                          Coef64& k) {
    const double* cp = chan64 + (active ? c : 0);
    const double on = active ? 1.0 : 0.0;
    k.gd = on * cp[P64_G4 * c_pad];
    k.g4 = 1.f;
    k.nb1 = -on * cp[P64_B1 * c_pad];
    k.nb2 = -on * cp[P64_B2 * c_pad];
#pragma unroll
    for (int i = 0; i < 4; ++i) k.z[i] = on * cp[(P64_Z + i) * c_pad];
#pragma unroll
    for (int i = 0; i < 3; ++i) k.zn[i] = k.z[i + 1] + k.nb1;
}

// ---- edge table: per (utterance, channel) the residuals in the order the cascade reads them ------------
// Entry [utt][C][8]: ee (0..3) multiplies G[t] at even t, eo (4..7) at odd t.  (t - n) odd -> e0 multiplies
// G[t]; even -> e1.
template <class E>
__device__ __forceinline__ void edge_parity(int n, const E (&e0)[4], const E (&e1)[4], E (&ee)[4], E (&eo)[4]) {
    const bool n_odd = (n & 1) != 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        ee[i] = n_odd ? e0[i] : e1[i];
        eo[i] = n_odd ? e1[i] : e0[i];
    }
}

__device__ __forceinline__ void store_edge_entry(float* table, size_t utt, int C, int c, const float (&ee)[4],
                                                 const float (&eo)[4]) {
    float4* o = reinterpret_cast<float4*>(table + (utt * C + c) * 8);
    o[0] = make_float4(ee[0], ee[1], ee[2], ee[3]);
    o[1] = make_float4(eo[0], eo[1], eo[2], eo[3]);
}

__device__ __forceinline__ void store_edge_entry(double* table, size_t utt, int C, int c, const double (&ee)[4],
                                                 const double (&eo)[4]) {
    double* o = table + (utt * C + c) * 8;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        o[i] = ee[i];
        o[4 + i] = eo[i];
    }
}

__device__ __forceinline__ void load_edge_entry(const float* table, size_t utt, int C, int c, float (&ee)[4],
                                                float (&eo)[4]) {
    const float4* e = reinterpret_cast<const float4*>(table + (utt * C + c) * 8);
    const float4 v0 = __ldg(e), v1 = __ldg(e + 1);
    ee[0] = v0.x; ee[1] = v0.y; ee[2] = v0.z; ee[3] = v0.w;
    eo[0] = v1.x; eo[1] = v1.y; eo[2] = v1.z; eo[3] = v1.w;
}

__device__ __forceinline__ void load_edge_entry(const double* table, size_t utt, int C, int c, double (&ee)[4],
                                                double (&eo)[4]) {
    const double* e = table + (utt * C + c) * 8;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        ee[i] = __ldg(e + i);
        eo[i] = __ldg(e + 4 + i);
    }
}

}  // namespace f2
