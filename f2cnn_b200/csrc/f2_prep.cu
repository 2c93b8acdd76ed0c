// f2_prep.cu -- per-utterance pre-pass: zero-padded ring, its circular Hilbert transform
// and the edge-injection kernel.
//
// The reference takes one FFT pair per CHANNEL of the filtered signal
// (scripts/processing/EnvelopeExtraction.py:20-36 paddedHilbert -> scipy.signal.hilbert).
// The ring formulation used by the fused kernel needs only ONE Hilbert transform per
// utterance, of the zero-padded INPUT: xi = Im(hilbert(pad(x, N2))), N2 = 2^ceil(log2 n).
// It is computed here with a hand-written FP32 FFT (no cuFFT):
//   real N2-point FFT as a packed complex M = N2/2 point FFT; M <= 4096 in one pass, larger
//   M as a four-step (columns, twiddle, rows) FFT with <= 4096-point shared-memory legs
//   (radix-4 steps); untangle, multiply by -i*sgn(k), tangle; inverse FFT.
// Launch sequence (A, B = N2 floats per utterance, XZ = N2 float2):
//   fft_cols<fwd>  wave -> A      (int16/f32/f64 -> packed complex fused into the load)
//   fft_rows<fwd>  A    -> B      (single-pass sizes: wave -> B)
//   hilbert_mask   B in place; also tabulates the injection kernel G into A
//   fft_cols<inv>  B in place
//   fft_rows<inv>  B    -> XZ     ((x, xi) interleaved ring, x re-read from the wave)
// The same kernels serve the stand-alone envelope path (rows of an arbitrary matrix).
#include "f2_prep.cuh"

#include <cooperative_groups.h>
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <mutex>

namespace f2 {

constexpr int kFftThreads = 256;
constexpr int kFftSmemPts = 4096;  // complex points per CTA (33 KB + swizzle padding: 6 CTAs per SM)
constexpr int kTwLog = 12;         // twiddle table covers legs up to 4096 points

__device__ float2 g_twiddle[1 << (kTwLog - 1)];  // exp(-2*pi*i*j/4096), j < 2048

__global__ void init_twiddle_kernel() {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < (1 << (kTwLog - 1))) {
        double s, c;
        sincospi(-2.0 * (double)j / (double)(1 << kTwLog), &s, &c);
        g_twiddle[j] = make_float2((float)c, (float)s);
    }
}

// four-step twiddles of the cluster kernel's two sizes: g_step14[k1*128 + n2] = exp(-2*pi*i*n2*k1/2^14),
// g_step15[k1*256 + n2] = exp(-2*pi*i*n2*k1/2^15), k1 < 128 (384 KB, L2-resident; the inverse conjugates)
__device__ float2 g_step14[1 << 14];
__device__ float2 g_step15[1 << 15];
__device__ float2 g_step16[1 << 16];   // [k1*256 + n2] = exp(-2*pi*i*n2*k1/2^16), k1 < 256

__global__ void init_step_twiddle_kernel() {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double s, c;
    if (i < (1 << 14)) {
        sincospi(-2.0 * (double)((i & 127) * (i >> 7)) / (double)(1 << 14), &s, &c);
        g_step14[i] = make_float2((float)c, (float)s);
    }
    if (i < (1 << 15)) {
        sincospi(-2.0 * (double)((i & 255) * (i >> 8)) / (double)(1 << 15), &s, &c);
        g_step15[i] = make_float2((float)c, (float)s);
    }
    if (i < (1 << 16)) {
        sincospi(-2.0 * (double)((i & 255) * (i >> 8)) / (double)(1 << 16), &s, &c);
        g_step16[i] = make_float2((float)c, (float)s);
    }
}

cudaError_t init_twiddles(cudaStream_t stream) {
    init_twiddle_kernel<<<(1 << (kTwLog - 1)) / 256, 256, 0, stream>>>();
    init_step_twiddle_kernel<<<(1 << 16) / 256, 256, 0, stream>>>();
    return cudaGetLastError();
}

// Shared-memory index swizzle: one float2 of padding per 16 keeps the strided accesses of the
// first radix-4 steps (stride 4 and 16 elements) off the same banks.
__host__ __device__ __forceinline__ int sw(int i) { return i + (i >> 4); }

__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
    return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 cconj(float2 a) { return make_float2(a.x, -a.y); }

// packed sample pair (x[2m], x[2m+1]) of an utterance, zero beyond n
__device__ __forceinline__ float2 load_pair(const void* base, int dtype, long long off, int m, int n) {
    const int t = 2 * m;
    float a = 0.f, b = 0.f;
    if (t < n) {
        const bool two = t + 1 < n;
        switch (dtype) {
            case F2_DT_I16: {
                const short* p = reinterpret_cast<const short*>(base) + off + t;
                if (two && (reinterpret_cast<size_t>(p) & 3) == 0) {  // aligned pair: one 32-bit load
                    const int v = __ldg(reinterpret_cast<const int*>(p));
                    a = (float)(short)(v & 0xffff);
                    b = (float)(short)(v >> 16);
                } else {
                    a = (float)p[0];
                    if (two) b = (float)p[1];
                }
                break;
            }
            case F2_DT_F32: {
                const float* p = reinterpret_cast<const float*>(base) + off + t;
                a = p[0];
                if (two) b = p[1];
                break;
            }
            default: {
                const double* p = reinterpret_cast<const double*>(base) + off + t;
                a = (float)p[0];
                if (two) b = (float)p[1];
            }
        }
    }
    return make_float2(a, b);
}

// ---- in-shared-memory DIT FFT on `batch` arrays of length 2^logL (data stored bit-reversed).
// Two radix-2 stages are fused into one radix-4 step (half the passes and barriers); an odd
// logL ends with one radix-2 stage.  INV conjugates the twiddles (unnormalised inverse).
template <bool INV>
__device__ __forceinline__ void smem_fft(float2* s, int pitch, int logL, int batch) {
    int st = 0;
    for (; st + 2 <= logL; st += 2) {
        const int h = 1 << st;
        const int per = 1 << (logL - 2);  // radix-4 butterflies per array
        const int total = batch << (logL - 2);
        for (int bf = threadIdx.x; bf < total; bf += blockDim.x) {
            const int arr = bf >> (logL - 2);
            const int j = bf & (per - 1);
            const int pos = j & (h - 1);
            const int i0 = ((j >> st) << (st + 2)) + pos;
            float2* a = s + arr * pitch;
            const int j0 = sw(i0), j1 = sw(i0 + h), j2 = sw(i0 + 2 * h), j3 = sw(i0 + 3 * h);
            float2 w1 = g_twiddle[pos << (kTwLog - 1 - st)];  // w_{2h}^pos
            float2 w2 = g_twiddle[pos << (kTwLog - 2 - st)];  // w_{4h}^pos
            if (INV) {
                w1.y = -w1.y;
                w2.y = -w2.y;
            }
            const float2 x0 = a[j0], x1 = cmul(a[j1], w1), x2 = a[j2], x3 = cmul(a[j3], w1);
            const float2 p0 = cadd(x0, x1), p1 = csub(x0, x1);  // stage st: (0,1)
            const float2 q0 = cadd(x2, x3), q1 = csub(x2, x3);  //           (2,3)
            // stage st+1: (p0,q0) with w2; (p1,q1) with w2 * w_{4h}^h = w2 * (-i) fwd / (+i) inv
            const float2 t0 = cmul(q0, w2);
            const float2 t1r = cmul(q1, w2);
            const float2 t1 = INV ? make_float2(-t1r.y, t1r.x) : make_float2(t1r.y, -t1r.x);
            a[j0] = cadd(p0, t0);
            a[j2] = csub(p0, t0);
            a[j1] = cadd(p1, t1);
            a[j3] = csub(p1, t1);
        }
        __syncthreads();
    }
    if (st < logL) {
        const int half = 1 << st;
        const int halfL = 1 << (logL - 1);
        const int total = batch << (logL - 1);
        for (int bf = threadIdx.x; bf < total; bf += blockDim.x) {
            const int arr = bf >> (logL - 1);
            const int j = bf & (halfL - 1);
            const int pos = j & (half - 1);
            const int i0 = ((j >> st) << (st + 1)) + pos;
            float2* a = s + arr * pitch;
            float2 w = g_twiddle[pos << (kTwLog - 1 - st)];
            if (INV) w.y = -w.y;
            const int j0 = sw(i0), j1 = sw(i0 + half);
            const float2 u = a[j0];
            const float2 v = cmul(a[j1], w);
            a[j0] = cadd(u, v);
            a[j1] = csub(u, v);
        }
        __syncthreads();
    }
}

// N2 = 32768 / 65536 / 131072 are transformed by one cluster kernel (ring_cluster_kernel, ring_cluster8_kernel below)
__host__ __device__ inline bool ring_cluster_size(int log2N2) { return log2N2 >= 15 && log2N2 <= 17; }

__device__ __forceinline__ int bitrev(int v, int bits) { return bits ? (int)(__brev((unsigned)v) >> (32 - bits)) : 0; }

__host__ __device__ inline void fft_split(int log2M, int& l1, int& l2) {
    if (log2M <= kTwLog) {
        l1 = 0;
        l2 = log2M;
    } else {
        l1 = log2M / 2;
        l2 = log2M - l1;
    }
}

// ---- pass A (columns): M1-point FFTs down the columns of the M1 x M2 matrix, then the
// four-step twiddle w_M^(n2*k1).  SRC_WAVE: read the packed input straight from the wave
// and write to `buf`; otherwise in place on `buf`. ----------------------------------------
template <bool INV, bool SRC_WAVE>
__global__ void __launch_bounds__(kFftThreads) fft_cols_kernel(PrepParams p, float* buf) {
    extern __shared__ float2 s_fft[];
    const UttDesc ut = p.utts[blockIdx.x];
    const int log2M = ut.log2N2 - 1;
    if (log2M <= kTwLog) return;  // single-pass sizes skip the column pass
    int l1, l2;
    fft_split(log2M, l1, l2);
    if (p.cluster && ring_cluster_size(ut.log2N2)) return;  // taken by ring_cluster_kernel
    const int M1 = 1 << l1, M2 = 1 << l2;
    int B = kFftSmemPts >> l1;
    if (B > M2) B = M2;
    const int c0 = blockIdx.y * B;
    if (c0 >= M2) return;
    float2* z = reinterpret_cast<float2*>(buf + ut.ring_off);
    const int pitch = sw(M1) + 1;
    const int logB = 31 - __clz(B);
#pragma unroll 4
    for (int idx = threadIdx.x; idx < (B << l1); idx += blockDim.x) {
        const int n1 = idx >> logB, b = idx & (B - 1);
        const int e = n1 * M2 + c0 + b;
        s_fft[b * pitch + sw(bitrev(n1, l1))] = SRC_WAVE ? load_pair(p.wave, p.wave_dtype, ut.wave_off, e, ut.n) : z[e];
    }
    __syncthreads();
    smem_fft<INV>(s_fft, pitch, l1, B);
    const float sgn = INV ? 2.0f : -2.0f;
    const float invM = 1.0f / (float)(1 << log2M);
    for (int idx = threadIdx.x; idx < (B << l1); idx += blockDim.x) {
        const int k1 = idx >> logB, b = idx & (B - 1);
        const int n2 = c0 + b;
        float sn, cs;
        sincospif(sgn * (float)(n2 * k1) * invM, &sn, &cs);  // n2*k1 < M <= 2^24: exact in float
        z[(size_t)k1 * M2 + n2] = cmul(s_fft[b * pitch + sw(k1)], make_float2(cs, sn));
    }
}

// ---- pass B (rows): M2-point FFTs along the rows, output index k1 + M1*k2.
// SRC_WAVE: single-pass forward transform reading the wave.  DST_RING: last pass of the
// inverse: output m holds (xi[2m], xi[2m+1]); write the interleaved (x, xi) ring directly. ----
template <bool INV, bool SRC_WAVE, bool DST_RING>
__global__ void __launch_bounds__(kFftThreads) fft_rows_kernel(PrepParams p, const float* in_buf, float* out_buf) {
    extern __shared__ float2 s_fft[];
    const UttDesc ut = p.utts[blockIdx.x];
    const int log2M = ut.log2N2 - 1;
    if (log2M < 1) return;
    int l1, l2;
    fft_split(log2M, l1, l2);
    if (SRC_WAVE && l1 != 0) return;   // two-pass sizes were packed by the column pass
    if (!SRC_WAVE && !INV && l1 == 0) return;  // forward single-pass sizes take the SRC_WAVE launch
    if (p.cluster && ring_cluster_size(ut.log2N2)) return;  // taken by ring_cluster_kernel
    const int M1 = 1 << l1, M2 = 1 << l2;
    int B = kFftSmemPts >> l2;
    if (B > M1) B = M1;
    const int r0 = blockIdx.y * B;
    if (r0 >= M1) return;
    const float2* zin = reinterpret_cast<const float2*>(in_buf + ut.ring_off);
    const int pitch = sw(M2) + 1;
#pragma unroll 4
    for (int idx = threadIdx.x; idx < (B << l2); idx += blockDim.x) {
        const int b = idx >> l2, n2 = idx & (M2 - 1);
        const int e = (r0 + b) * M2 + n2;
        s_fft[b * pitch + sw(bitrev(n2, l2))] = SRC_WAVE ? load_pair(p.wave, p.wave_dtype, ut.wave_off, e, ut.n) : zin[e];
    }
    __syncthreads();
    smem_fft<INV>(s_fft, pitch, l2, B);
    const int logB = 31 - __clz(B);
    if (DST_RING) {
        float4* ring = reinterpret_cast<float4*>(p.xz + ut.ring_off);
        for (int idx = threadIdx.x; idx < (B << l2); idx += blockDim.x) {
            const int k2 = idx >> logB, b = idx & (B - 1);
            const int m = k2 * M1 + r0 + b;
            const float2 w = s_fft[b * pitch + sw(k2)];
            const float2 x = load_pair(p.wave, p.wave_dtype, ut.wave_off, m, ut.n);
            ring[m] = make_float4(x.x, w.x, x.y, w.y);
        }
    } else {
        float2* zout = reinterpret_cast<float2*>(out_buf + ut.ring_off);
        for (int idx = threadIdx.x; idx < (B << l2); idx += blockDim.x) {
            const int k2 = idx >> logB, b = idx & (B - 1);
            zout[(size_t)k2 * M1 + r0 + b] = s_fft[b * pitch + sw(k2)];
        }
    }
}

// =============================================================================================
// Register transforms for the legs of the cluster kernel below (128 and 256 points: N2 = 32768 ... 131072).
// Each leg is two register passes -- L = R1 x R2 with R1 = 16, R2 = L/16 -- around ONE
// shared-memory exchange, instead of log4(L) shared-memory passes:
//   pass 1: thread (fft b, n2) loads x[n1*R2 + n2], n1 < 16, runs a 16-point FFT in registers,
//           multiplies by w_L^(n2*k1) and writes A[b][k1][n2];
//   pass 2: thread (fft b, k1) reads A[b][k1][n2], n2 < R2, runs an R2-point FFT in registers:
//           X[k1 + 16*k2].
// =============================================================================================
// complex add / subtract as ONE packed instruction (FADD2; FFMA2 with -1): same IEEE results as the scalar pairs
__device__ __forceinline__ float2 padd(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 psub(float2 a, float2 b) { return __ffma2_rn(b, make_float2(-1.f, -1.f), a); }

template <bool INV>
__device__ __forceinline__ void fft4(float2& a0, float2& a1, float2& a2, float2& a3) {
    const float2 s02 = padd(a0, a2), d02 = psub(a0, a2), s13 = padd(a1, a3), d13 = psub(a1, a3);
    a0 = padd(s02, s13);
    a2 = psub(s02, s13);
    if (INV) {   // a1 = d02 + i*d13, a3 = d02 - i*d13
        a1 = make_float2(d02.x - d13.y, d02.y + d13.x);
        a3 = make_float2(d02.x + d13.y, d02.y - d13.x);
    } else {
        a1 = make_float2(d02.x + d13.y, d02.y - d13.x);
        a3 = make_float2(d02.x - d13.y, d02.y + d13.x);
    }
}

template <bool INV>
__device__ __forceinline__ float2 cmul_w16(float2 v, int m) {  // v * w_16^m, m = 0..9 (compile-time after unrolling)
    constexpr float C1 = 0.92387953251128674f, S1 = 0.38268343236508977f, R2 = 0.70710678118654752f;
    float c, s;  // w_16^m = cos(2 pi m/16) - i sin(2 pi m/16)
    switch (m) {
        case 0: return v;
        case 1: c = C1; s = S1; break;
        case 2: c = R2; s = R2; break;
        case 3: c = S1; s = C1; break;
        case 4: c = 0.f; s = 1.f; break;
        case 6: c = -R2; s = R2; break;
        default: c = -C1; s = -S1; break;  // m = 9
    }
    const float2 w = make_float2(c, INV ? s : -s);
    return cmul(v, w);
}

// 16-point FFT in registers; result for frequency k = (r >> 2) + 4 * (r & 3) is left in v[r].
template <bool INV>
__device__ __forceinline__ void fft16(float2 (&v)[16]) {
#pragma unroll
    for (int n2 = 0; n2 < 4; ++n2) fft4<INV>(v[n2], v[4 + n2], v[8 + n2], v[12 + n2]);
#pragma unroll
    for (int k1 = 1; k1 < 4; ++k1)
#pragma unroll
        for (int n2 = 1; n2 < 4; ++n2) v[4 * k1 + n2] = cmul_w16<INV>(v[4 * k1 + n2], n2 * k1);
#pragma unroll
    for (int k1 = 0; k1 < 4; ++k1) fft4<INV>(v[4 * k1], v[4 * k1 + 1], v[4 * k1 + 2], v[4 * k1 + 3]);
}
__device__ __forceinline__ constexpr int out16(int r) { return (r >> 2) + 4 * (r & 3); }

// 8-point FFT in registers; result for frequency k = (r >> 1) + 4 * (r & 1) is left in v[r].
template <bool INV>
__device__ __forceinline__ void fft8(float2 (&v)[8]) {
    fft4<INV>(v[0], v[2], v[4], v[6]);
    fft4<INV>(v[1], v[3], v[5], v[7]);
    v[3] = cmul_w16<INV>(v[3], 2);  // w_8^1
    v[5] = cmul_w16<INV>(v[5], 4);  // w_8^2
    v[7] = cmul_w16<INV>(v[7], 6);  // w_8^3
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float2 a = v[2 * j], b = v[2 * j + 1];
        v[2 * j] = cadd(a, b);
        v[2 * j + 1] = csub(a, b);
    }
}
__device__ __forceinline__ constexpr int out8(int r) { return (r >> 1) + 4 * (r & 1); }
// 8- or 16-point register transform chosen by the array length
template <bool INV> __device__ __forceinline__ void fft_rc(float2 (&v)[8]) { fft8<INV>(v); }
template <bool INV> __device__ __forceinline__ void fft_rc(float2 (&v)[16]) { fft16<INV>(v); }
template <int R> __device__ __forceinline__ constexpr int out_rc(int r) { return R == 16 ? out16(r) : out8(r); }

template <bool INV>
__device__ __forceinline__ float2 leg_twiddle(int m, int logL) {  // w_L^m for 0 <= m < L
    int idx = m << (kTwLog - logL);
    float2 w;
    if (idx >= (1 << (kTwLog - 1))) {
        w = g_twiddle[idx - (1 << (kTwLog - 1))];
        w = make_float2(-w.x, -w.y);
    } else {
        w = g_twiddle[idx];
    }
    if (INV) w.y = -w.y;
    return w;
}

// One pair (Z[k], Z[M-k]) of the packed spectrum -> the pair (W[k], W[M-k]) the inverse packed transform
// needs (see the derivation above hilbert_mask_kernel); valid for any 0 < k < M, k = M/2 included (a == b).
__device__ __forceinline__ void hilbert_pair(float2 a, float2 b, int k, float invN, float2& Wk, float2& Wm) {
    float sn, cs;
    sincospif(-2.0f * (float)k * invN, &sn, &cs);  // e = exp(-2 pi i k / N)
    const float2 e = make_float2(cs, sn);
    // X[k]
    const float2 sp = make_float2(a.x + b.x, a.y - b.y);  // a + conj(b)
    const float2 dm = make_float2(a.x - b.x, a.y + b.y);  // a - conj(b)
    const float2 ed = cmul(e, dm);
    const float2 Xk = make_float2(0.5f * (sp.x + ed.y), 0.5f * (sp.y - ed.x));  // sp/2 - (i/2) ed
    // X[M-k] = conj(sp)/2 - (i/2) e2 * (-conj(dm)),  e2 = exp(-2 pi i (M-k)/N) = -conj(e)
    // => X[M-k] = conj(sp)/2 - (i/2) conj(ed)
    const float2 Xm = make_float2(0.5f * (sp.x - ed.y), 0.5f * (-sp.y - ed.x));
    // Y = -i X
    const float2 Yk = make_float2(Xk.y, -Xk.x);
    const float2 Ym = make_float2(Xm.y, -Xm.x);
    // W[k] = (Yk + conj(Ym)) + i conj(e) (Yk - conj(Ym))
    const float2 s2 = make_float2(Yk.x + Ym.x, Yk.y - Ym.y);
    const float2 d2 = make_float2(Yk.x - Ym.x, Yk.y + Ym.y);
    const float2 ce = make_float2(e.x, -e.y);
    const float2 t2 = cmul(ce, d2);
    Wk = make_float2((s2.x - t2.y) * invN, (s2.y + t2.x) * invN);
    // W[M-k] = conj(s2) + i conj(t2)
    Wm = make_float2((s2.x + t2.y) * invN, (-s2.y + t2.x) * invN);
}

// H[m], m = (t - n) mod N2: the circular Hilbert kernel h[l] = (2/N2) cot(pi l / N2) at the odd one of m, m-1.
__device__ __forceinline__ float injection_tap(int m, int N2, float invN) {
    int l = m;
    if (!(l & 1)) l = (l - 1) & (N2 - 1);
    if (l > N2 / 2) l -= N2;  // cot is odd and pi-periodic: keep |l| <= N2/2 for accuracy
    float sn, cs;
    sincospif((float)l * invN, &sn, &cs);
    return 2.0f * invN * cs / sn;
}

// four shifted copies of H for one ring size: tab[s*(N2+256) + m] = H[(m + s) mod N2]
__global__ void injection_table_kernel(float* tab, int N2) {
    const float invN = 1.0f / (float)N2;
    const int len = N2 + 256;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 4 * len; i += gridDim.x * blockDim.x) {
        const int s = i / len, m = i - s * len;
        tab[i] = injection_tap((m + s) & (N2 - 1), N2, invN);
    }
}

// ---- untangle the packed real FFT, apply the Hilbert multiplier, tangle for the inverse ----
// Z = FFT_M(z).  X[k] = (Z[k]+conj(Z[M-k]))/2 - (i/2) e^{-2 pi i k/N} (Z[k]-conj(Z[M-k])).
// scipy.signal.hilbert keeps h[0]=h[N/2]=1, doubles 0<k<N/2, zeroes the rest: the imaginary
// part of its output has spectrum Y[k] = -i X[k] (0<k<N/2), Y[0]=Y[N/2]=0.  Packed inverse:
// W[k] = (Y[k]+conj(Y[M-k])) + i e^{+2 pi i k/N} (Y[k]-conj(Y[M-k])), scaled by 1/N.
//
// The same launch tabulates the injection kernel into `gtab` (when non-null):
// G[tau] = h[l], l = the odd one of (tau-n) mod N2, (tau-n-1) mod N2,
// h[l] = (2/N2) cot(pi l / N2): the circular Hilbert kernel for even N2 that matches scipy's
// one-sided mask.
__global__ void hilbert_mask_kernel(const UttDesc* utts, float* buf, float* gtab, int cluster) {
    const UttDesc ut = utts[blockIdx.x];
    const int N2 = ut.N2;
    const int M = N2 >> 1;
    const float invN = 1.0f / (float)N2;
    if (gtab && !ut.g_tab) {
        float* G = gtab + ut.ring_off;
        for (int tau = blockIdx.y * blockDim.x + threadIdx.x; tau < N2; tau += gridDim.y * blockDim.x) {
            G[tau] = N2 > 2 ? injection_tap((tau - ut.n) & (N2 - 1), N2, invN) : 0.f;
        }
    }
    if (!buf || M < 1) return;
    if (cluster && ring_cluster_size(ut.log2N2)) return;  // done in shared memory by ring_cluster_kernel
    float2* Z = reinterpret_cast<float2*>(buf + ut.ring_off);
    for (int k = blockIdx.y * blockDim.x + threadIdx.x; k <= M / 2; k += gridDim.y * blockDim.x) {
        if (k == 0) {
            Z[0] = make_float2(0.f, 0.f);
            continue;
        }
        const float2 a = Z[k], b = Z[M - k];
        float2 Wk, Wm;
        hilbert_pair(a, b, k, invN, Wk, Wm);
        Z[k] = Wk;
        if (k != M - k) Z[M - k] = Wm;
    }
}

// ---- rings without a Hilbert transform: filterbank-only runs (xi = 0) and utterances with
// N2 <= 2, whose analytic signal is real. -------------------------------------------------
__global__ void plain_ring_kernel(PrepParams p, int only_tiny) {
    const UttDesc ut = p.utts[blockIdx.x];
    const int N2 = ut.N2;
    if (only_tiny && N2 > 2) return;
    float4* ring = reinterpret_cast<float4*>(p.xz + ut.ring_off);
    const int M = N2 > 1 ? N2 >> 1 : 1;  // N2 == 1: one float4 inside the 256-sample allocation
    for (int m = blockIdx.y * blockDim.x + threadIdx.x; m < M; m += gridDim.y * blockDim.x) {
        const float2 x = load_pair(p.wave, p.wave_dtype, ut.wave_off, m, ut.n);
        ring[m] = make_float4(x.x, 0.f, x.y, 0.f);
    }
}


// =============================================================================================
// The whole ring transform of an utterance in ONE kernel (N2 = 32768, 65536 and 131072: utterances of
// 1 ... 8.2 s): a thread-block cluster keeps the packed spectrum in its distributed shared
// memory, so HBM sees the wave once (plus one L2-resident re-read) and the (x, xi) ring once --
// 0.6 MB per utterance where the five-kernel sequence above moves 3 MB through two scratch rings.
//
//   M = N2/2 = M1 x M2 packed complex points z[n1*M2 + n2] (M1 = 128; 256 for N2 = 131072, in a cluster of 8).  CTA `rank` of the CL in the cluster owns
//   columns [rank*M2/CL, +M2/CL) in the column phases and a mirror-closed set of 128/CL rows in the row
//   phase (row k1 and row 128-k1 sit in adjacent slots, because the Hilbert step pairs Z[k] with Z[M-k]).
//   1  columns forward: 128-point FFTs (16 x 8 in registers around one shared exchange), read straight
//      from the wave; four-step twiddle; every thread then holds 32 values in registers across a
//      cluster barrier and stores them into the row owners' shared memory (DSMEM): the transposition
//      never leaves the chip and needs no second buffer.
//   2  rows: forward M2-point FFT in place (results stay in digit-swapped order), Hilbert pair step,
//      inverse M2-point FFT in place (the same two register passes, mirrored), inverse twiddle, and
//      the transposition back through registers + DSMEM.
//   3  columns inverse: 128-point FFTs, output m = m1*M2 + n2 holds (xi[2m], xi[2m+1]): written with
//      (x[2m], x[2m+1]) as one float4 of the interleaved ring, 512 contiguous bytes per warp.
// =============================================================================================

template <int L1, int L2, int CL, int T>
struct RingCl {
    static constexpr int M1 = 1 << L1, M2 = 1 << L2, M = M1 * M2;
    static constexpr int RC = M1 / 16;   // second radix of the column transform: 8 (128 points) or 16 (256)
    static constexpr int NC = M2 / CL;   // columns per CTA
    static constexpr int NR = M1 / CL;   // rows per CTA
    static constexpr int PC = M1 + 1;    // column pitch (float2): odd, so that column-major tasks spread over the banks
    static constexpr int PSH = L2 - 4;   // one float2 of padding per 16 (M2 = 256) / 8 (M2 = 128) row elements
    static constexpr int PR = M2 + (M2 >> PSH) + (L2 == 7 ? 8 : 0);   // row pitch
    static constexpr int PB3 = NC + 1;   // phase 3 keeps its columns as [k1][b]: the transposing stores of a warp are contiguous
    static constexpr int kE1 = (NC * PC > NR * PR) ? NC * PC : NR * PR;
    static constexpr int kElems = kE1 > M1 * PB3 ? kE1 : M1 * PB3;
    __device__ static __forceinline__ int pad(int q) { return q + (q >> PSH); }
    // row k1 -> (owner CTA, slot).  f = min(k1, M1-k1); rows f and M1-f go to CTA f % CL, slots 2*(f/CL)
    // and 2*(f/CL)+1; the two self-mirrored rows 0 and M1/2 share pair 0 of CTA 0.
    __device__ static __forceinline__ void owner(int k1, int& cta, int& slot) {
        const int f = k1 <= M1 / 2 ? k1 : M1 - k1;
        cta = f % CL;
        slot = k1 == M1 / 2 ? 1 : 2 * (f / CL) + (k1 > M1 / 2 ? 1 : 0);
    }
    __device__ static __forceinline__ int row_of(int cta, int slot) {
        const int f = (slot >> 1) * CL + cta;
        if (f == 0) return (slot & 1) ? M1 / 2 : 0;
        return (slot & 1) ? M1 - f : f;
    }
    // position of row frequency k2 after the forward row transform (its second pass leaves k2 = k1' + 16*k2'
    // at k1'*R2 + k2', R2 = M2/16)
    __device__ static __forceinline__ int pos(int k2) { return pad((k2 & 15) * (M2 / 16) + (k2 >> 4)); }
};

template <int L1, int L2, int CL, int T>
__device__ __forceinline__ void ring_cluster_body(const PrepParams& p, const UttDesc& ut, float2* sm) {
    using S = RingCl<L1, L2, CL, T>;
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int tid = threadIdx.x;
    constexpr int M2 = S::M2, NC = S::NC, NR = S::NR, PC = S::PC, PR = S::PR;
    constexpr int R2 = M2 / 16;           // second radix of the row transform (16 or 8)
    constexpr int RC = S::RC;             // ... of the column transform
    const float invN = 0.5f / (float)S::M;
    // leg twiddles in shared memory behind the data, the index that varies across the threads of a warp
    // innermost: tw_a[k*8 + n] = w_128^(k*n) (k < 16, n < 8), tw_b[k*16 + n] = w_128^(k*n) (k < 8, n < 16),
    // tw_r[k*16 + n] = w_256^(k*n) (forward values; the inverse conjugates)
    float2* tw_a = sm + S::kElems;
    float2* tw_b = tw_a + 128;
    float2* tw_r = tw_b + 128;
    for (int i = tid; i < 128; i += T) {
        tw_a[i] = leg_twiddle<false>((i >> 3) * (i & 7), 7);
        tw_b[i] = leg_twiddle<false>((i >> 4) * (i & 15), 7);
    }
    if (L2 == 8 || L1 == 8)
        for (int i = tid; i < 256; i += T) tw_r[i] = leg_twiddle<false>((i >> 4) * (i & 15), 8);
    const float2* __restrict__ step = L1 + L2 == 14 ? g_step14 : (L1 + L2 == 15 ? g_step15 : g_step16);   // [k1*M2 + n2]
    const float2* tw_c = L1 == 8 ? tw_r : tw_a;   // column legs: [k*RC + n] = w_M1^(k*n)
    __syncthreads();

    // ---- 1: columns forward ----
    for (int task = tid; task < NC * RC; task += T) {
        const int b = task % NC, n2p = task / NC;
        float2 v[16];
#pragma unroll
        for (int n1p = 0; n1p < 16; ++n1p)
            v[n1p] = load_pair(p.wave, p.wave_dtype, ut.wave_off, (n1p * RC + n2p) * M2 + rank * NC + b, ut.n);
        fft16<false>(v);
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            const int k1p = out16(r);
            sm[b * PC + k1p * RC + n2p] = cmul(v[r], tw_c[k1p * RC + n2p]);
        }
    }
    __syncthreads();
    {
        constexpr int NT = NC * 16 / T;
        static_assert(NT * T == NC * 16, "column pass 2 tasks must divide evenly");
        float2 h[NT][RC];
#pragma unroll
        for (int i = 0; i < NT; ++i) {
            const int task = tid + i * T;
            const int b = task % NC, k1p = task / NC;
#pragma unroll
            for (int n2p = 0; n2p < RC; ++n2p) h[i][n2p] = sm[b * PC + k1p * RC + n2p];
            fft_rc<false>(h[i]);
            const int n2 = rank * NC + b;
#pragma unroll
            for (int r = 0; r < RC; ++r) {
                const int k1 = k1p + 16 * out_rc<RC>(r);
                h[i][r] = cmul(h[i][r], __ldg(step + k1 * M2 + n2));
            }
        }
        cluster.sync();   // every CTA has its column data in registers: the buffers may be overwritten
#pragma unroll
        for (int i = 0; i < NT; ++i) {
            const int task = tid + i * T;
            const int b = task % NC, k1p = task / NC;
            const int n2 = rank * NC + b;
#pragma unroll
            for (int r = 0; r < RC; ++r) {
                int cta, slot;
                S::owner(k1p + 16 * out_rc<RC>(r), cta, slot);
                float2* dst = cluster.map_shared_rank(sm, cta);
                dst[slot * PR + S::pad(n2)] = h[i][r];
            }
        }
        cluster.sync();
    }

    // ---- 2a: rows forward, in place ----
    for (int task = tid; task < NR * R2; task += T) {
        const int n2p = task % R2, slot = task / R2;
        float2* row = sm + slot * PR;
        float2 v[16];
#pragma unroll
        for (int n1p = 0; n1p < 16; ++n1p) v[n1p] = row[S::pad(n1p * R2 + n2p)];
        fft16<false>(v);
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            const int k1p = out16(r);
            row[S::pad(k1p * R2 + n2p)] = cmul(v[r], L2 == 8 ? tw_r[k1p * 16 + n2p] : tw_a[k1p * 8 + n2p]);
        }
    }
    __syncthreads();
    for (int task = tid; task < NR * 16; task += T) {
        const int k1p = task % 16, slot = task / 16;
        float2* row = sm + slot * PR;
        if (R2 == 16) {
            float2 v[16];
#pragma unroll
            for (int n2p = 0; n2p < 16; ++n2p) v[n2p] = row[S::pad(k1p * 16 + n2p)];
            fft16<false>(v);
#pragma unroll
            for (int r = 0; r < 16; ++r) row[S::pad(k1p * 16 + out16(r))] = v[r];   // k2 = k1p + 16*out16(r)
        } else {
            float2 v[8];
#pragma unroll
            for (int n2p = 0; n2p < 8; ++n2p) v[n2p] = row[S::pad(k1p * 8 + n2p)];
            fft8<false>(v);
#pragma unroll
            for (int r = 0; r < 8; ++r) row[S::pad(k1p * 8 + out8(r))] = v[r];
        }
    }
    __syncthreads();

    // ---- 2b: Hilbert multiplier on the pairs (k, M-k), k = k1 + 128*k2 ----
    for (int task = tid; task < (NR / 2) * M2; task += T) {
        const int k2 = task % M2, j = task / M2;
        if (rank == 0 && j == 0) continue;   // rows 0 and 64: below
        const int k1 = S::row_of(rank, 2 * j);
        float2* pa = sm + (2 * j) * PR + S::pos(k2);
        float2* pb = sm + (2 * j + 1) * PR + S::pos(M2 - 1 - k2);
        float2 Wk, Wm;
        hilbert_pair(*pa, *pb, k1 + S::M1 * k2, invN, Wk, Wm);
        *pa = Wk;
        *pb = Wm;
    }
    if (rank == 0) {
        for (int task = tid; task < M2 + 1; task += T) {
            if (task <= M2 / 2) {   // row 0: k = 128*k2 pairs with 128*(M2-k2)
                float2* pa = sm + S::pos(task);
                if (task == 0) {
                    *pa = make_float2(0.f, 0.f);
                } else {
                    float2* pb = sm + S::pos(M2 - task);
                    float2 Wk, Wm;
                    hilbert_pair(*pa, *pb, S::M1 * task, invN, Wk, Wm);
                    *pa = Wk;
                    if (task != M2 / 2) *pb = Wm;
                }
            } else {                // row 64: k = 64 + 128*k2 pairs with 64 + 128*(M2-1-k2)
                const int k2 = task - (M2 / 2 + 1);
                float2* pa = sm + PR + S::pos(k2);
                float2* pb = sm + PR + S::pos(M2 - 1 - k2);
                float2 Wk, Wm;
                hilbert_pair(*pa, *pb, S::M1 / 2 + S::M1 * k2, invN, Wk, Wm);
                *pa = Wk;
                *pb = Wm;
            }
        }
    }
    __syncthreads();

    // ---- 2c: rows inverse, in place; natural index i sits at pos(i) ----
    if (R2 == 16) {
        for (int task = tid; task < NR * 16; task += T) {
            const int n2p = task % 16, slot = task / 16;
            float2* row = sm + slot * PR;
            float2 v[16];
#pragma unroll
            for (int n1p = 0; n1p < 16; ++n1p) v[n1p] = row[S::pad(n2p * 16 + n1p)];   // i = n1p*16 + n2p
            fft16<true>(v);
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                const int k1p = out16(r);
                row[S::pad(n2p * 16 + k1p)] = cmul(v[r], cconj(tw_r[k1p * 16 + n2p]));
            }
        }
    } else {
        // 128 = 8 x 16: 8-point transforms over n1 (i = n1*16 + n2 at pos = n2*8 + n1), then 16-point over n2
        for (int task = tid; task < NR * 16; task += T) {
            const int n2p = task % 16, slot = task / 16;
            float2* row = sm + slot * PR;
            float2 v[8];
#pragma unroll
            for (int n1p = 0; n1p < 8; ++n1p) v[n1p] = row[S::pad(n2p * 8 + n1p)];
            fft8<true>(v);
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const int k1p = out8(r);
                row[S::pad(n2p * 8 + k1p)] = cmul(v[r], cconj(tw_b[k1p * 16 + n2p]));
            }
        }
    }
    __syncthreads();
    {
        constexpr int R1 = M2 / 16;   // first radix of the inverse row transform: 16 (M2 = 256) or 8
        constexpr int NT = NR * R1 / T > 0 ? NR * R1 / T : 1;
        static_assert(NR * R1 % T == 0 || NR * R1 < T, "row pass 2 tasks");
        float2 g[NT][16];
        bool live[NT];
#pragma unroll
        for (int i = 0; i < NT; ++i) {
            const int task = tid + i * T;
            live[i] = task < NR * R1;
            const int k1p = task % R1, slot = live[i] ? task / R1 : 0;
            const float2* row = sm + slot * PR;
#pragma unroll
            for (int n2p = 0; n2p < 16; ++n2p) g[i][n2p] = row[S::pad(n2p * R1 + k1p)];
            fft16<true>(g[i]);
            const int k1 = S::row_of(rank, slot);
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                const int m2 = k1p + R1 * out16(r);
                g[i][r] = cmul(g[i][r], cconj(__ldg(step + k1 * M2 + m2)));
            }
        }
        cluster.sync();
#pragma unroll
        for (int i = 0; i < NT; ++i) {
            const int task = tid + i * T;
            const int k1p = task % R1, slot = live[i] ? task / R1 : 0;
            const int k1 = S::row_of(rank, slot);
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                const int m2 = k1p + R1 * out16(r);
                float2* dst = cluster.map_shared_rank(sm, m2 / NC);
                if (live[i]) dst[k1 * S::PB3 + (m2 % NC)] = g[i][r];
            }
        }
        cluster.sync();
    }

    // ---- 3: columns inverse (data as [k1][b]), ring store ----
    for (int task = tid; task < NC * RC; task += T) {
        const int b = task % NC, n2p = task / NC;
        float2* col = sm + b;
        float2 v[16];
#pragma unroll
        for (int n1p = 0; n1p < 16; ++n1p) v[n1p] = col[(n1p * RC + n2p) * S::PB3];
        fft16<true>(v);
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            const int k1p = out16(r);
            col[(k1p * RC + n2p) * S::PB3] = cmul(v[r], cconj(tw_c[k1p * RC + n2p]));
        }
    }
    __syncthreads();
    float4* ring = reinterpret_cast<float4*>(p.xz + ut.ring_off);
    for (int task = tid; task < NC * 16; task += T) {
        const int b = task % NC, k1p = task / NC;
        const float2* col = sm + b;
        float2 v[RC], x[8];
        if (RC == 8) {
#pragma unroll
            for (int r = 0; r < 8; ++r)   // the wave again (L2): issued before the transform that hides their latency
                x[r] = load_pair(p.wave, p.wave_dtype, ut.wave_off, (k1p + 16 * out8(r)) * M2 + rank * NC + b, ut.n);
        }
#pragma unroll
        for (int n2p = 0; n2p < RC; ++n2p) v[n2p] = col[(k1p * RC + n2p) * S::PB3];
        fft_rc<true>(v);
#pragma unroll
        for (int r = 0; r < RC; ++r) {
            const int m = (k1p + 16 * out_rc<RC>(r)) * M2 + rank * NC + b;
            // 16 results per thread: no registers left to hold the wave pairs across the transform
            const float2 xv = RC == 8 ? x[r & 7] : load_pair(p.wave, p.wave_dtype, ut.wave_off, m, ut.n);
            ring[m] = make_float4(xv.x, v[r].x, xv.y, v[r].y);
        }
    }
}

constexpr int kRingCl = 4;            // CTAs per cluster
constexpr int kRingCtas = 2;          // CTAs per SM
constexpr int kRingClThreads = 512;
constexpr int kRingAhead = 148 * kRingCtas / kRingCl;   // clusters resident at a time
constexpr int kRingCl8 = 8;           // CTAs per cluster for rings of 131072 samples (M = 256 x 256)
constexpr int kRingAhead8 = 148 * kRingCtas / kRingCl8;
constexpr int kRingClElems = RingCl<7, 8, kRingCl, kRingClThreads>::kElems > RingCl<7, 7, kRingCl, kRingClThreads>::kElems
                                 ? RingCl<7, 8, kRingCl, kRingClThreads>::kElems
                                 : RingCl<7, 7, kRingCl, kRingClThreads>::kElems;
constexpr int kRingClSmem = (kRingClElems + 512) * (int)sizeof(float2);
constexpr int kRingCl8Smem = (RingCl<8, 8, kRingCl8, kRingClThreads>::kElems + 512) * (int)sizeof(float2);

// The first thing a cluster does is wait for its wave from HBM with nothing to overlap it with: pull the wave of
// the cluster that will run here one generation later into L2 now (one 128-byte line per thread).
template <int CL>
__device__ __forceinline__ void prefetch_next_wave(const PrepParams& p, int u, int n_utts, int ahead_by) {
    const int ahead = u + ahead_by;
    if (ahead >= n_utts) return;
    const UttDesc nx = p.utts[ahead];
    const int esz = p.wave_dtype == F2_DT_I16 ? 2 : (p.wave_dtype == F2_DT_F32 ? 4 : 8);
    const char* base = reinterpret_cast<const char*>(p.wave) + nx.wave_off * esz;
    const long long bytes = (long long)nx.n * esz;
    for (long long o = ((long long)(blockIdx.x % CL) * kRingClThreads + threadIdx.x) * 128; o < bytes;
         o += (long long)CL * kRingClThreads * 128)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(base + o));
}

__global__ void __cluster_dims__(kRingCl, 1, 1) __launch_bounds__(kRingClThreads, kRingCtas) ring_cluster_kernel(PrepParams p) {
    extern __shared__ float2 s_fft[];
    const int u = blockIdx.x / kRingCl, n_utts = gridDim.x / kRingCl;
    const UttDesc ut = p.utts[u];
    prefetch_next_wave<kRingCl>(p, u, n_utts, kRingAhead);
    if (ut.log2N2 == 16) ring_cluster_body<7, 8, kRingCl, kRingClThreads>(p, ut, s_fft);
    else if (ut.log2N2 == 15) ring_cluster_body<7, 7, kRingCl, kRingClThreads>(p, ut, s_fft);
}

// rings of 131072 samples (utterances of 4.1 ... 8.2 s): M = 256 x 256 packed points, a cluster of 8 CTAs
__global__ void __cluster_dims__(kRingCl8, 1, 1) __launch_bounds__(kRingClThreads, kRingCtas) ring_cluster8_kernel(PrepParams p) {
    extern __shared__ float2 s_fft[];
    const int u = blockIdx.x / kRingCl8, n_utts = gridDim.x / kRingCl8;
    const UttDesc ut = p.utts[u];
    if (ut.log2N2 != 17) return;
    prefetch_next_wave<kRingCl8>(p, u, n_utts, kRingAhead8);
    ring_cluster_body<8, 8, kRingCl8, kRingClThreads>(p, ut, s_fft);
}

// One injection table per (device, ring size), built on first use and kept for the life of the process
// (16 bytes per ring sample: 1 MB for N2 = 65536); immutable afterwards, so every stream may read it.
const float* injection_table(int log2N2, int* stride) {
    if (log2N2 < kGTabMinLog || log2N2 > kGTabMaxLog) return nullptr;
    static std::mutex mu;
    static float* cache[64][kGTabMaxLog + 1] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev >= 64) return nullptr;
    const int N2 = 1 << log2N2;
    if (stride) *stride = N2 + 256;
    std::lock_guard<std::mutex> lock(mu);
    if (!cache[dev][log2N2]) {
        float* t = nullptr;
        if (cudaMalloc(&t, sizeof(float) * 4 * (size_t)(N2 + 256)) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;   // the caller falls back to per-utterance tables
        }
        injection_table_kernel<<<std::min(1024, (4 * (N2 + 256) + 255) / 256), 256>>>(t, N2);
        if (cudaDeviceSynchronize() != cudaSuccess) {
            cudaGetLastError();
            cudaFree(t);
            return nullptr;
        }
        cache[dev][log2N2] = t;
    }
    return cache[dev][log2N2];
}

static int max_blocks(const HostPrepInfo& h, bool cols) {
    int best = 1;
    for (int lg = h.min_log2N2; lg <= h.max_log2N2; ++lg) {
        const int log2M = lg - 1;
        if (log2M < 1) continue;
        int l1, l2;
        fft_split(log2M, l1, l2);
        int blocks;
        if (cols) {
            if (l1 == 0) continue;
            int B = kFftSmemPts >> l1;
            if (B > (1 << l2)) B = 1 << l2;
            blocks = (1 << l2) / B;
        } else {
            int B = kFftSmemPts >> l2;
            if (B > (1 << l1)) B = 1 << l1;
            blocks = (1 << l1) / B;
        }
        if (blocks > best) best = blocks;
    }
    return best;
}

// development knob: F2CNN_B200_RING_CLUSTER=0 sends every size through the multi-pass kernels
bool ring_cluster_enabled() {
    static const bool on = [] { const char* v = getenv("F2CNN_B200_RING_CLUSTER"); return !(v && v[0] == '0'); }();
    return on;
}

cudaError_t launch_prep(const PrepParams& p_in, const HostPrepInfo& h, cudaStream_t stream) {
    if (h.n_utts <= 0) return cudaSuccess;
    PrepParams p = p_in;
    p.cluster = ring_cluster_enabled() && p.hilbert && h.min_log2N2 <= 17 && h.max_log2N2 >= 15;
    if (h.max_log2N2 - 1 > 2 * kTwLog) return cudaErrorInvalidValue;
    // per device: the attribute belongs to the current device's copy of the function
    static bool attr_done[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    const int smem = (kFftSmemPts + kFftSmemPts / 16 + 512) * (int)sizeof(float2);
    if (dev >= 64 || !attr_done[dev]) {
        cudaFuncSetAttribute(fft_cols_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        cudaFuncSetAttribute(fft_cols_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        cudaFuncSetAttribute(fft_rows_kernel<false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        cudaFuncSetAttribute(fft_rows_kernel<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        cudaFuncSetAttribute(fft_rows_kernel<true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        cudaFuncSetAttribute(ring_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kRingClSmem);
        cudaFuncSetAttribute(ring_cluster8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kRingCl8Smem);
        if (dev < 64) attr_done[dev] = true;
    }
    const int maxN2 = 1 << h.max_log2N2;
    int ew_blocks = (maxN2 / 2 + 1023) / 1024;
    ew_blocks = ew_blocks < 1 ? 1 : (ew_blocks > 2048 ? 2048 : ew_blocks);
    const dim3 g_ew(h.n_utts, ew_blocks);
    if (!p.hilbert || h.max_log2N2 < 2) {
        plain_ring_kernel<<<g_ew, 256, 0, stream>>>(p, 0);
        if (p.G) hilbert_mask_kernel<<<g_ew, 256, 0, stream>>>(p.utts, nullptr, p.G, 0);  // N2 <= 2: G = 0
        return cudaGetLastError();
    }
    const bool one = h.min_log2N2 - 1 <= kTwLog;  // some utterances take the single-pass path
    bool two = false;                              // some take the two-pass path: not a cluster kernel's size
    for (int lg = h.min_log2N2; lg <= h.max_log2N2; ++lg)
        if (lg - 1 > kTwLog && !(p.cluster && ring_cluster_size(lg))) two = true;
    const dim3 g_cols(h.n_utts, max_blocks(h, true));
    const dim3 g_rows(h.n_utts, max_blocks(h, false));
    float* A = p.bufA;
    float* B = p.bufB;
    // whole transform in one cluster kernel for the corpus sizes (its utterances are skipped by everything below
    // except the G table)
    if (p.cluster && h.min_log2N2 <= 16) ring_cluster_kernel<<<kRingCl * h.n_utts, kRingClThreads, kRingClSmem, stream>>>(p);
    if (p.cluster && h.max_log2N2 >= 17) ring_cluster8_kernel<<<kRingCl8 * h.n_utts, kRingClThreads, kRingCl8Smem, stream>>>(p);
    // forward
    if (two) fft_cols_kernel<false, true><<<g_cols, kFftThreads, smem, stream>>>(p, A);
    if (two) fft_rows_kernel<false, false, false><<<g_rows, kFftThreads, smem, stream>>>(p, A, B);
    if (one) fft_rows_kernel<false, true, false><<<g_rows, kFftThreads, smem, stream>>>(p, nullptr, B);
    // Hilbert multiplier in place on B; the injection kernel goes to A (free from here on)
    const bool all_cluster = p.cluster && h.min_log2N2 >= 15 && h.max_log2N2 <= 17;
    if (!all_cluster || (p.G && h.private_g > 0)) hilbert_mask_kernel<<<g_ew, 256, 0, stream>>>(p.utts, B, p.G, p.cluster);
    // inverse, last pass writes the (x, xi) ring
    if (two) fft_cols_kernel<true, false><<<g_cols, kFftThreads, smem, stream>>>(p, B);
    if (one || two) fft_rows_kernel<true, false, true><<<g_rows, kFftThreads, smem, stream>>>(p, B, nullptr);
    if (h.min_log2N2 < 2) plain_ring_kernel<<<g_ew, 256, 0, stream>>>(p, 1);
    return cudaGetLastError();
}

}  // namespace f2
