// f2_post.cu -- layout / windowing kernels either side of the fused kernel (all HBM-bound).
//
//   gather_rows         window gather of InputGenerator.py:73-80 from decimated frames
//   dense_frames        dense stride-1 framing of Evaluating.py:70-78 (+ normalizeInput,
//                       scripts/CNN/Training.py:13-28)
//   rows_envelope       abs(analytic) + lowPassFilter for the stand-alone
//                       ExtractEnvelopeFromMatrix path; the 1st-order low-pass is a chunked
//                       linear-recurrence scan with warp-shuffle carry propagation.
#include "f2_post.cuh"

namespace f2 {

// ------------------------------------------------------------------------------------------
// out[(row*dots + j)*C + c] = src[(base[row] + j*stride)*C + c]
__global__ void gather_rows_kernel(const float* __restrict__ src, const long long* __restrict__ base, int dots,
                                   long long stride, int C, float* __restrict__ out) {
    const long long row = blockIdx.x;
    const long long b = base[row];
    const int total = dots * C;
    float* o = out + (size_t)row * total;
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
        const int j = i / C, c = i - j * C;
        o[i] = src[(size_t)(b + (long long)j * stride) * C + c];
    }
}

// 16-byte version (C % 4 == 0, 16-byte aligned buffers): one warp per window row group, each
// thread moves float4s; stride-1 windows are `dots` consecutive source rows = one contiguous run.
__global__ void gather_rows_vec_kernel(const float4* __restrict__ src, const long long* __restrict__ base,
                                       long long n_rows, int dots, long long stride, int C4,
                                       float4* __restrict__ out) {
    const int total = dots * C4;
    for (long long row = blockIdx.x; row < n_rows; row += gridDim.x) {
        const long long b = base[row];
        float4* o = out + (size_t)row * total;
        if (stride == 1) {
            const float4* s = src + (size_t)b * C4;
            for (int i = threadIdx.x; i < total; i += blockDim.x) __stcs(o + i, __ldg(s + i));
        } else {
            for (int i = threadIdx.x; i < total; i += blockDim.x) {
                const int j = i / C4, c = i - j * C4;
                __stcs(o + i, __ldg(src + (size_t)(b + (long long)j * stride) * C4 + c));
            }
        }
    }
}

cudaError_t launch_gather_rows(const float* src, const long long* base, long long n_rows, int dots,
                               long long stride, int C, float* out, cudaStream_t stream) {
    if (n_rows <= 0) return cudaSuccess;
    if (C % 4 == 0 && ((size_t)src % 16 == 0) && ((size_t)out % 16 == 0)) {
        const long long blocks = n_rows < 148 * 32 ? n_rows : 148 * 32;
        gather_rows_vec_kernel<<<(unsigned)blocks, 128, 0, stream>>>((const float4*)src, base, n_rows, dots, stride,
                                                                     C / 4, (float4*)out);
    } else {
        gather_rows_kernel<<<(unsigned)n_rows, 256, 0, stream>>>(src, base, dots, stride, C, out);
    }
    return cudaGetLastError();
}

// out[(i*dots + j)*C + c] = src[idx[i*dots + j]*C + c]   (arbitrary, e.g. off-grid timepoints)
__global__ void gather_index_kernel(const float* __restrict__ src, const long long* __restrict__ idx, int C,
                                    float* __restrict__ out) {
    const long long r = blockIdx.x;
    const long long b = idx[r];
    for (int c = threadIdx.x; c < C; c += blockDim.x) out[(size_t)r * C + c] = src[(size_t)b * C + c];
}

cudaError_t launch_gather_index(const float* src, const long long* idx, long long n_idx, int C, float* out,
                                cudaStream_t stream) {
    if (n_idx <= 0) return cudaSuccess;
    gather_index_kernel<<<(unsigned)n_idx, 128, 0, stream>>>(src, idx, C, out);
    return cudaGetLastError();
}

// out[(w*dots + j)*C + c] = (float) env[c*n + idx[w*dots + j]]: the gather of
// InputGenerator.py:73-80 from a (C,n) matrix in the reference's own layout (loaded .ENV1.npy);
// the float64 -> float32 conversion rounds to nearest even like numpy.astype (:83).
template <typename T>
__global__ void gather_cn_kernel(const T* __restrict__ env, int C, long long n, const long long* __restrict__ idx,
                                 float* __restrict__ out) {
    const long long r = blockIdx.x;
    const long long t = idx[r];
    for (int c = threadIdx.x; c < C; c += blockDim.x) out[(size_t)r * C + c] = (float)env[(size_t)c * n + t];
}

cudaError_t launch_gather_cn(const void* env, int dtype, int C, long long n, const long long* idx, long long n_idx,
                             float* out, cudaStream_t stream) {
    if (n_idx <= 0) return cudaSuccess;
    if (dtype == F2_DT_F64)
        gather_cn_kernel<double><<<(unsigned)n_idx, 128, 0, stream>>>((const double*)env, C, n, idx, out);
    else if (dtype == F2_DT_F32)
        gather_cn_kernel<float><<<(unsigned)n_idx, 128, 0, stream>>>((const float*)env, C, n, idx, out);
    else
        return cudaErrorInvalidValue;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// Dense framing: frame i (i0 <= i < i1) = rows env_t[i + k*step], k < dots.  With
// `normalize`, Training.normalizeInput per frame: (log v - log min)/(log max - log min),
// all-equal frame -> zeros, min <= 0 -> flag set (the reference raises ValueError).
template <typename T>
__global__ void dense_frames_kernel(const float* __restrict__ env_t, int C, int dots, int step, long long i0,
                                    int normalize, T* __restrict__ out, int* __restrict__ bad_flag) {
    __shared__ float s_min[32], s_max[32];
    const long long i = i0 + blockIdx.x;
    const int total = dots * C;
    const float* src = env_t + (size_t)i * C;
    T* o = out + (size_t)blockIdx.x * total;
    float mn = INFINITY, mx = -INFINITY;
    if (normalize) {
        for (int e = threadIdx.x; e < total; e += blockDim.x) {
            const int k = e / C, c = e - k * C;
            const float v = src[(size_t)k * step * C + c];
            mn = fminf(mn, v);
            mx = fmaxf(mx, v);
        }
        for (int off = 16; off; off >>= 1) {
            mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, off));
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
        }
        if ((threadIdx.x & 31) == 0) {
            s_min[threadIdx.x >> 5] = mn;
            s_max[threadIdx.x >> 5] = mx;
        }
        __syncthreads();
        const int nw = blockDim.x >> 5;
        mn = s_min[0];
        mx = s_max[0];
        for (int w = 1; w < nw; ++w) {
            mn = fminf(mn, s_min[w]);
            mx = fmaxf(mx, s_max[w]);
        }
        if (threadIdx.x == 0 && !(mn > 0.f)) atomicOr(bad_flag, 1);
    }
    // In double: in float32, log(max) - log(min) of a frame whose span is a few ulps cancels to 0 (then
    // NaN) or to one ulp of log(min), several times the true span.
    const bool flat = normalize && (mn == mx);
    const double lmn = normalize ? log((double)mn) : 0.0;
    const double inv = normalize ? 1.0 / (log((double)mx) - lmn) : 1.0;
    for (int e = threadIdx.x; e < total; e += blockDim.x) {
        const int k = e / C, c = e - k * C;
        const float v = src[(size_t)k * step * C + c];
        if (normalize)
            o[e] = (T)(flat ? 0.0 : (log((double)v) - lmn) * inv);
        else
            o[e] = (T)v;
    }
}

cudaError_t launch_dense_frames(const float* env_t, int C, int dots, int step, long long i0, long long i1,
                                int normalize, void* out, int out_dtype, int* bad_flag, cudaStream_t stream) {
    if (i1 <= i0) return cudaSuccess;
    const unsigned nb = (unsigned)(i1 - i0);
    if (out_dtype == F2_DT_F64)
        dense_frames_kernel<double><<<nb, 256, 0, stream>>>(env_t, C, dots, step, i0, normalize, (double*)out,
                                                            bad_flag);
    else if (out_dtype == F2_DT_F32)
        dense_frames_kernel<float><<<nb, 256, 0, stream>>>(env_t, C, dots, step, i0, normalize, (float*)out,
                                                           bad_flag);
    else
        return cudaErrorInvalidValue;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// Stand-alone envelope of matrix rows: e[t] = |x[t] + i xi[t]| from the (x, xi) ring, then
// (optionally) y[t] = b0 (e[t] + e[t-1]) + k y[t-1]  (butter(1), zero initial state).
// One warp per row.  Per iteration the warp covers 32 lanes x 8 samples; every lane runs
// its 8 samples from zero state, the (k^8, local end state) pairs are composed across the
// lanes with a Kogge-Stone scan over warp shuffles, the carry of the previous iteration is
// folded in, and each lane then corrects its 8 outputs with k^(j+1) * (state at chunk start).
constexpr int kScanPerLane = 8;

// op: 0 = envelope |x + i xi|, 1 = xi alone (imaginary part of paddedHilbert), 2 = x alone
// (lowPassFilter of the raw rows).
template <typename T>
__global__ void rows_envelope_kernel(const UttDesc* rows, const float2* __restrict__ xz, int op, int lpf, float lp_k,
                                     float lp_b0, T* __restrict__ out) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const UttDesc ut = rows[warp];
    const int n = ut.n;
    const float2* src = xz + ut.ring_off;
    T* dst = out + ut.wave_off;  // same element offset as the input row
    float kp[kScanPerLane + 1];  // k^j
    kp[0] = 1.f;
#pragma unroll
    for (int j = 1; j <= kScanPerLane; ++j) kp[j] = kp[j - 1] * lp_k;
    float carry_l = 0.f;  // low-pass state (scaled by 1/b0) at the end of the previous iteration
    float carry_e = 0.f;  // last envelope sample of the previous iteration
    for (int base = 0; base < n; base += 32 * kScanPerLane) {
        const int t0 = base + lane * kScanPerLane;
        float e[kScanPerLane];
#pragma unroll
        for (int j = 0; j < kScanPerLane; ++j) {
            const int t = t0 + j;
            float2 v = make_float2(0.f, 0.f);
            if (t < n) v = src[t];
            e[j] = op == 0 ? sqrtf(fmaf(v.x, v.x, v.y * v.y)) : (op == 1 ? v.y : v.x);
        }
        if (!lpf) {
#pragma unroll
            for (int j = 0; j < kScanPerLane; ++j)
                if (t0 + j < n) dst[t0 + j] = (T)e[j];
            continue;
        }
        // previous envelope sample for this lane's first step
        float eprev = __shfl_up_sync(0xffffffffu, e[kScanPerLane - 1], 1);
        if (lane == 0) eprev = carry_e;
        // local pass from zero state
        float loc[kScanPerLane];
        float l = 0.f, ep = eprev;
#pragma unroll
        for (int j = 0; j < kScanPerLane; ++j) {
            l = fmaf(lp_k, l, e[j] + ep);
            ep = e[j];
            loc[j] = l;
        }
        // inclusive scan of (a, b): state_out = a*state_in + b
        float a = kp[kScanPerLane], b = l;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const float a1 = __shfl_up_sync(0xffffffffu, a, off);
            const float b1 = __shfl_up_sync(0xffffffffu, b, off);
            if (lane >= off) {
                b = fmaf(a, b1, b);
                a = a * a1;
            }
        }
        const float end_state = fmaf(a, carry_l, b);  // state after this lane's chunk
        float init = __shfl_up_sync(0xffffffffu, end_state, 1);
        if (lane == 0) init = carry_l;
#pragma unroll
        for (int j = 0; j < kScanPerLane; ++j)
            if (t0 + j < n) dst[t0 + j] = (T)(lp_b0 * fmaf(kp[j + 1], init, loc[j]));
        carry_l = __shfl_sync(0xffffffffu, end_state, 31);
        carry_e = __shfl_sync(0xffffffffu, e[kScanPerLane - 1], 31);
    }
}

cudaError_t launch_rows_envelope(const UttDesc* rows, int n_rows, const float2* xz, int op, int lpf, float lp_k,
                                 float lp_b0, void* out, int out_dtype, cudaStream_t stream) {
    if (n_rows <= 0) return cudaSuccess;
    // one warp per row, 4 warps per CTA; n_rows is padded by the caller to a multiple of 4
    const int blocks = (n_rows + 3) / 4;
    if (out_dtype == F2_DT_F64)
        rows_envelope_kernel<double><<<blocks, 128, 0, stream>>>(rows, xz, op, lpf, lp_k, lp_b0, (double*)out);
    else if (out_dtype == F2_DT_F32)
        rows_envelope_kernel<float><<<blocks, 128, 0, stream>>>(rows, xz, op, lpf, lp_k, lp_b0, (float*)out);
    else
        return cudaErrorInvalidValue;
    return cudaGetLastError();
}

}  // namespace f2
