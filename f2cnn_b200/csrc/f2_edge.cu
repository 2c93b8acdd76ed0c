// f2_edge.cu -- edge residuals e_k of the zero-padded ring equation (DESIGN.md section 3, H1).
//
// For every (utterance, channel) the real cascade's state after the last sample n-1 gives the
// residuals e0_k, e1_k (edge_residuals, f2_sections.cuh).  All sections are strictly stable, so
// the state depends on the last w_edge samples only (to float32 resolution).
//
// Two kernels produce the same float [utt][C][8] table (f2_sections.cuh: store_edge_entry):
//  * edge_kernel<0>   -- one thread per channel, sequential over the window.  Used when there
//                        are enough (utterance, channel) pairs to fill the GPU.
//  * edge_scan_kernel -- chunked parallel linear-recurrence scan for small batches (a single
//                        utterance would otherwise wait for 2048 sequential steps): one warp
//                        per (utterance, channel); every lane runs one block of 64 samples
//                        from zero state; the 8-element cascade states are then composed
//                        across the 32 lanes, S_j <- S_j + M^(2^d) S_(j-2^d), d = 0..4, with
//                        __shfl_up_sync.  M = A^64 is the block transition of the four coupled
//                        biquads (lower block-triangular, one 2x2 block per section on the
//                        diagonal), its powers are precomputed per channel in float64.
// edge_kernel<2> fills the float64 table of the FORM 2 groups with the fused kernel's FORM 2 sections.
#include "f2_edge.cuh"

#include <math.h>

namespace f2 {

// Residuals of channel c from the real cascade's state after sample n-1, into the table entry of utterance utt.
// real_only (N2 <= 2): the analytic signal is real, nothing is injected.
template <int FORM, class K, class S, class E>
__device__ __forceinline__ void write_edge(const K& k, const S& s, int n, bool real_only, E* edge, size_t utt, int C,
                                           int c) {
    E e0[4], e1[4], ee[4], eo[4];
    edge_residuals<FORM>(k, s, e0, e1);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        e0[i] = real_only ? E(0) : e0[i];
        e1[i] = real_only ? E(0) : e1[i];
    }
    edge_parity(n, e0, e1, ee, eo);
    store_edge_entry(edge, utt, C, c, ee, eo);
}

// Sequential pass, one thread per channel, from zero state w_edge samples before the end.  The float32 pass
// runs the delta form (FORM 0) for every group, the form build_scan_matrices describes, so that it and the
// scan give the same table.  FORM 2: one warp per group of 32 channels; groups that are not FORM 2 leave at
// once, and their entries of the float64 table are not written.
template <int FORM>
__global__ void __launch_bounds__(FORM == 2 ? kChanPerBlock : kEdgeChanPerBlock)
    edge_kernel(const UttDesc* utts, const float* __restrict__ chan, int C, int c_pad, const float2* __restrict__ xz,
                int w_edge, typename SectionTypes<FORM>::E* __restrict__ edge, const double* __restrict__ chan64) {
    constexpr int W = FORM == 2 ? kChanPerBlock : kEdgeChanPerBlock;
    const UttDesc ut = utts[blockIdx.x];
    const int c = blockIdx.y * W + threadIdx.x;
    if (FORM == 2 && chan[P_FORM * c_pad + blockIdx.y * W] != kForm2Marker) return;
    if (c >= C || ut.n <= 0) return;
    typename SectionTypes<FORM>::K k;
    load_coef<FORM>(chan, chan64, c_pad, c, true, k);
    typename SectionTypes<FORM>::S s;
    reset(s);
    const int n = ut.n;
    const int t0 = n - w_edge > 0 ? n - w_edge : 0;
    const float2* src = xz + ut.ring_off;
    if (ut.N2 > 2) {
#pragma unroll 4
        for (int t = t0; t < n; ++t) cascade_real<FORM>(k, s, __ldg(&src[t].x));
    }
    write_edge<FORM>(k, s, n, ut.N2 <= 2, edge, blockIdx.x, C, c);
}

template <int FORM>
cudaError_t launch_edge(const UttDesc* utts, int n_utts, const float* chan, const double* chan64, int C, int c_pad,
                        const float2* xz, int w_edge, typename SectionTypes<FORM>::E* edge, cudaStream_t stream) {
    if (n_utts <= 0) return cudaSuccess;
    constexpr int W = FORM == 2 ? kChanPerBlock : kEdgeChanPerBlock;
    dim3 grid(n_utts, (C + W - 1) / W);
    edge_kernel<FORM><<<grid, W, 0, stream>>>(utts, chan, C, c_pad, xz, w_edge, edge, chan64);
    return cudaGetLastError();
}
template cudaError_t launch_edge<0>(const UttDesc*, int, const float*, const double*, int, int, const float2*, int,
                                    float*, cudaStream_t);
template cudaError_t launch_edge<2>(const UttDesc*, int, const float*, const double*, int, int, const float2*, int,
                                    double*, cudaStream_t);

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
    Coef k;
    load_coef<0>(chan, nullptr, c_pad, c, true, k);
    // 1. every lane: its block of 64 samples from zero state (the true previous input sample
    //    is part of the block's input response, not of the carried state)
    State s;
    reset(s);
    const float* xb = s_x + 1 + lane * kScanPitch;
    s.up.x = lane == 0 ? s_x[0] : s_x[1 + (lane - 1) * kScanPitch + kScanBlock - 1];
#pragma unroll 4
    for (int i = 0; i < kScanBlock; ++i) cascade_real<0>(k, s, xb[i]);
    const float x_last = __shfl_sync(0xffffffffu, s.up.x, 31);
    // 2. Kogge-Stone composition of the carries: S_j += M^(2^d) * S_(j - 2^d)
    float S[8] = {s.y[0].x, s.q[0].x, s.y[1].x, s.q[1].x, s.y[2].x, s.q[2].x, s.y[3].x, s.q[3].x};
    const float* M = mats + (size_t)c * kScanLevels * 64;
#pragma unroll
    for (int d = 0; d < kScanLevels; ++d) {
        float P[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) P[j] = __shfl_up_sync(0xffffffffu, S[j], 1 << d);
        if (lane >= (1 << d)) {
            const float* Md = M + d * 64;
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                float acc = S[r];
#pragma unroll
                for (int j = 0; j < 8; ++j) acc = fmaf(__ldg(Md + r * 8 + j), P[j], acc);
                S[r] = acc;
            }
        }
    }
    // 3. lane 31 holds the state after sample n-1
    if (lane == 31) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            s.y[i].x = S[2 * i];
            s.q[i].x = S[2 * i + 1];
        }
        s.up.x = x_last;
        write_edge<0>(k, s, n, ut.N2 <= 2, edge, blockIdx.x, C, c);
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
