// f2_edge.cu -- edge residuals e_k of the zero-padded ring equation (DESIGN.md section 3, H1).
//
// For every (utterance, channel) the real cascade's state after the last sample n-1 gives
//   e0_k = b1*y_k[n-1] + b2*y_k[n-2] - z_k*u_k[n-1] = (cy-1)*y - cq*q - z_k*u,   e1_k = cq*y
// (a0-free stage variables).  All sections are strictly stable, so the state depends on the
// last w_edge samples only (to float32 resolution).
//
// Two kernels produce the same [utt][C][8] table (entries 0..3 multiply G at even t, 4..7 at
// odd t):
//  * edge_kernel      -- one thread per channel, sequential over the window.  Used when there
//                        are enough (utterance, channel) pairs to fill the GPU.
//  * edge_scan_kernel -- chunked parallel linear-recurrence scan for small batches (a single
//                        utterance would otherwise wait for 2048 sequential steps): one warp
//                        per (utterance, channel); every lane runs one block of 64 samples
//                        from zero state; the 8-element cascade states are then composed
//                        across the 32 lanes, S_j <- S_j + M^(2^d) S_(j-2^d), d = 0..4, with
//                        __shfl_up_sync.  M = A^64 is the block transition of the four coupled
//                        biquads (lower block-triangular, one 2x2 block per section on the
//                        diagonal), its powers are precomputed per channel in float64.
#include "f2_edge.cuh"

#include <math.h>

namespace f2 {

__device__ __forceinline__ void real_step(const float (&z)[4], const float (&cq)[4], const float (&ncy)[4],
                                          float (&y)[4], float (&q)[4], float u, float up) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float in = fmaf(z[i], up, u);
        const float yo = y[i];
        float qn = fmaf(cq[i], q[i], in);
        qn = fmaf(ncy[i], yo, qn);
        const float yn = yo + qn;
        q[i] = qn;
        y[i] = yn;
        up = yo;
        u = yn;
    }
}

__device__ __forceinline__ void store_edge(const float (&z)[4], const float (&cq)[4], const float (&ncy)[4],
                                           const float (&y)[4], const float (&q)[4], float x_last, int n, bool real_only,
                                           float* __restrict__ dst) {
    float e0[4], e1[4];
    float uprev = x_last;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float cy = -ncy[i];
        e0[i] = real_only ? 0.f : fmaf(cy - 1.0f, y[i], -cq[i] * q[i]) - z[i] * uprev;
        e1[i] = real_only ? 0.f : cq[i] * y[i];
        uprev = y[i];
    }
    const bool n_odd = (n & 1) != 0;  // (t - n) odd -> e0 multiplies G[t]
    float4* o = reinterpret_cast<float4*>(dst);
    o[0] = n_odd ? make_float4(e0[0], e0[1], e0[2], e0[3]) : make_float4(e1[0], e1[1], e1[2], e1[3]);
    o[1] = n_odd ? make_float4(e1[0], e1[1], e1[2], e1[3]) : make_float4(e0[0], e0[1], e0[2], e0[3]);
}

__global__ void __launch_bounds__(kEdgeChanPerBlock) edge_kernel(const UttDesc* utts, const float* __restrict__ chan,
                                                             int C, int c_pad, const float2* __restrict__ xz,
                                                             int w_edge, float* __restrict__ edge) {
    const UttDesc ut = utts[blockIdx.x];
    const int c = blockIdx.y * kEdgeChanPerBlock + threadIdx.x;
    if (c >= C || ut.n <= 0) return;
    float z[4], cq[4], ncy[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        z[i] = chan[(P_Z + i) * c_pad + c];
        cq[i] = chan[(P_CQ + i) * c_pad + c];
        ncy[i] = chan[(P_NCY + i) * c_pad + c];
    }
    float y[4] = {0.f, 0.f, 0.f, 0.f}, q[4] = {0.f, 0.f, 0.f, 0.f};
    float up = 0.f;
    const int n = ut.n;
    const int t0 = n - w_edge > 0 ? n - w_edge : 0;
    const float2* src = xz + ut.ring_off;
    if (ut.N2 > 2) {
#pragma unroll 4
        for (int t = t0; t < n; ++t) {
            const float u = __ldg(&src[t].x);
            real_step(z, cq, ncy, y, q, u, up);
            up = u;
        }
    }
    store_edge(z, cq, ncy, y, q, up, n, ut.N2 <= 2, edge + ((size_t)blockIdx.x * C + c) * 8);
}

cudaError_t launch_edge(const UttDesc* utts, int n_utts, const float* chan, int C, int c_pad, const float2* xz,
                        int w_edge, float* edge, cudaStream_t stream) {
    if (n_utts <= 0) return cudaSuccess;
    dim3 grid(n_utts, (C + kEdgeChanPerBlock - 1) / kEdgeChanPerBlock);
    edge_kernel<<<grid, kEdgeChanPerBlock, 0, stream>>>(utts, chan, C, c_pad, xz, w_edge, edge);
    return cudaGetLastError();
}

// ---- FORM 2 groups: float64 direct-form residuals ---------------------------------------------
// One CTA per (utterance, group of 32 channels); groups that are not FORM 2 leave at once.  The same
// recurrence as cascade_real / edge_residuals of the fused kernel's FORM 2, from zero state w_edge
// samples before the end.
__global__ void __launch_bounds__(32) edge_kernel64(const UttDesc* utts, const float* __restrict__ chan,
                                                    const double* __restrict__ chan64, int C, int c_pad,
                                                    const float2* __restrict__ xz, int w_edge,
                                                    double* __restrict__ edge) {
    const UttDesc ut = utts[blockIdx.x];
    const int c = blockIdx.y * 32 + threadIdx.x;
    if (chan[P_FORM * c_pad + blockIdx.y * 32] != kForm2Marker || c >= C || ut.n <= 0) return;
    double z[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) z[i] = chan64[(P64_Z + i) * c_pad + c];
    const double b1 = chan64[P64_B1 * c_pad + c], b2 = chan64[P64_B2 * c_pad + c];
    double y[4] = {0.0, 0.0, 0.0, 0.0}, y2[4] = {0.0, 0.0, 0.0, 0.0};
    double up = 0.0;
    const int n = ut.n;
    const int t0 = n - w_edge > 0 ? n - w_edge : 0;
    const float2* src = xz + ut.ring_off;
    if (ut.N2 > 2) {
#pragma unroll 4
        for (int t = t0; t < n; ++t) {
            double u = __ldg(&src[t].x), upi = up;
            up = u;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const double yn = fma(-b1, y[i], fma(-b2, y2[i], fma(z[i], upi, u)));
                upi = y[i];
                y2[i] = y[i];
                y[i] = yn;
                u = yn;
            }
        }
    }
    double e0[4], e1[4];
    double uprev = up;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const bool real_only = ut.N2 <= 2;
        e0[i] = real_only ? 0.0 : fma(b1, y[i], b2 * y2[i]) - z[i] * uprev;
        e1[i] = real_only ? 0.0 : b2 * y[i];
        uprev = y[i];
    }
    const bool n_odd = (n & 1) != 0;  // (t - n) odd -> e0 multiplies G[t]
    double* o = edge + ((size_t)blockIdx.x * C + c) * 8;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        o[i] = n_odd ? e0[i] : e1[i];
        o[4 + i] = n_odd ? e1[i] : e0[i];
    }
}

cudaError_t launch_edge64(const UttDesc* utts, int n_utts, const float* chan, const double* chan64, int C, int c_pad,
                          const float2* xz, int w_edge, double* edge, cudaStream_t stream) {
    if (n_utts <= 0) return cudaSuccess;
    dim3 grid(n_utts, (C + 31) / 32);
    edge_kernel64<<<grid, 32, 0, stream>>>(utts, chan, chan64, C, c_pad, xz, w_edge, edge);
    return cudaGetLastError();
}

// ---- scan version ----------------------------------------------------------------------------
constexpr int kScanWarps = 4;                  // channels per CTA (they share the staged window)
constexpr int kScanPitch = kScanBlock + 1;     // floats per lane block in shared memory (bank spread)

__global__ void __launch_bounds__(kScanWarps * 32) edge_scan_kernel(const UttDesc* utts,
                                                                     const float* __restrict__ chan,
                                                                     const float* __restrict__ mats, int C, int c_pad,
                                                                     const float2* __restrict__ xz,
                                                                     float* __restrict__ edge) {
    __shared__ float s_x[32 * kScanPitch + 1];  // s_x[0] = x[t0-1], block b at 1 + b*pitch
    const UttDesc ut = utts[blockIdx.x];
    const int n = ut.n;
    if (n <= 0) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int t0 = n - kScanWindow;  // may be negative: zeros before the first sample
    const float2* src = xz + ut.ring_off;
    for (int i = threadIdx.x; i < kScanWindow + 1; i += blockDim.x) {
        const int t = t0 - 1 + i;
        const float v = t >= 0 ? __ldg(&src[t].x) : 0.f;
        if (i == 0) s_x[0] = v;
        else s_x[1 + ((i - 1) / kScanBlock) * kScanPitch + ((i - 1) % kScanBlock)] = v;
    }
    __syncthreads();
    const int c = blockIdx.y * kScanWarps + warp;
    if (c >= C) return;
    float z[4], cq[4], ncy[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        z[i] = chan[(P_Z + i) * c_pad + c];
        cq[i] = chan[(P_CQ + i) * c_pad + c];
        ncy[i] = chan[(P_NCY + i) * c_pad + c];
    }
    // 1. every lane: its block of 64 samples from zero state (the true previous input sample
    //    is part of the block's input response, not of the carried state)
    float y[4] = {0.f, 0.f, 0.f, 0.f}, q[4] = {0.f, 0.f, 0.f, 0.f};
    const float* xb = s_x + 1 + lane * kScanPitch;
    float up = lane == 0 ? s_x[0] : s_x[1 + (lane - 1) * kScanPitch + kScanBlock - 1];
#pragma unroll 4
    for (int i = 0; i < kScanBlock; ++i) {
        const float u = xb[i];
        real_step(z, cq, ncy, y, q, u, up);
        up = u;
    }
    const float x_last = __shfl_sync(0xffffffffu, up, 31);
    // 2. Kogge-Stone composition of the carries: S_j += M^(2^d) * S_(j - 2^d)
    float S[8] = {y[0], q[0], y[1], q[1], y[2], q[2], y[3], q[3]};
    const float* M = mats + (size_t)c * kScanLevels * 64;
#pragma unroll
    for (int d = 0; d < kScanLevels; ++d) {
        float P[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) P[k] = __shfl_up_sync(0xffffffffu, S[k], 1 << d);
        if (lane >= (1 << d)) {
            const float* Md = M + d * 64;
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                float acc = S[r];
#pragma unroll
                for (int k = 0; k < 8; ++k) acc = fmaf(__ldg(Md + r * 8 + k), P[k], acc);
                S[r] = acc;
            }
        }
    }
    // 3. lane 31 holds the state after sample n-1
    if (lane == 31) {
        const float yy[4] = {S[0], S[2], S[4], S[6]}, qq[4] = {S[1], S[3], S[5], S[7]};
        store_edge(z, cq, ncy, yy, qq, x_last, n, ut.N2 <= 2, edge + ((size_t)blockIdx.x * C + c) * 8);
    }
}

cudaError_t launch_edge_scan(const UttDesc* utts, int n_utts, const float* chan, const float* scan_mats, int C,
                             int c_pad, const float2* xz, float* edge, cudaStream_t stream) {
    if (n_utts <= 0) return cudaSuccess;
    dim3 grid(n_utts, (C + kScanWarps - 1) / kScanWarps);
    edge_scan_kernel<<<grid, kScanWarps * 32, 0, stream>>>(utts, chan, scan_mats, C, c_pad, xz, edge);
    return cudaGetLastError();
}

// ---- host: block transition powers ----------------------------------------------------------
void build_scan_matrices(const float* par, int c_pad, int c, float* out) {
    double z[4], cq[4], ncy[4];
    for (int i = 0; i < 4; ++i) {
        z[i] = par[(size_t)(P_Z + i) * c_pad + c];
        cq[i] = par[(size_t)(P_CQ + i) * c_pad + c];
        ncy[i] = par[(size_t)(P_NCY + i) * c_pad + c];
    }
    // one homogeneous step (input 0, previous input 0) applied to the unit vectors
    double A[8][8];
    for (int col = 0; col < 8; ++col) {
        double y[4] = {0, 0, 0, 0}, q[4] = {0, 0, 0, 0};
        (col & 1 ? q : y)[col >> 1] = 1.0;
        double u = 0.0, up = 0.0;
        for (int i = 0; i < 4; ++i) {
            const double in = z[i] * up + u;
            const double yo = y[i];
            const double qn = cq[i] * q[i] + in + ncy[i] * yo;
            const double yn = yo + qn;
            q[i] = qn;
            y[i] = yn;
            up = yo;
            u = yn;
        }
        for (int i = 0; i < 4; ++i) {
            A[2 * i][col] = y[i];
            A[2 * i + 1][col] = q[i];
        }
    }
    auto mul = [](const double (&X)[8][8], const double (&Y)[8][8], double (&Z)[8][8]) {
        double T[8][8];
        for (int i = 0; i < 8; ++i)
            for (int j = 0; j < 8; ++j) {
                double s = 0.0;
                for (int k = 0; k < 8; ++k) s += X[i][k] * Y[k][j];
                T[i][j] = s;
            }
        for (int i = 0; i < 8; ++i)
            for (int j = 0; j < 8; ++j) Z[i][j] = T[i][j];
    };
    double Mp[8][8];
    for (int i = 0; i < 8; ++i)
        for (int j = 0; j < 8; ++j) Mp[i][j] = A[i][j];
    for (int s = 1; s < kScanBlock; s <<= 1) mul(Mp, Mp, Mp);  // A^64 by repeated squaring (64 = 2^6)
    for (int d = 0; d < kScanLevels; ++d) {
        for (int i = 0; i < 8; ++i)
            for (int j = 0; j < 8; ++j) out[d * 64 + i * 8 + j] = (float)Mp[i][j];
        mul(Mp, Mp, Mp);
    }
}

}  // namespace f2
