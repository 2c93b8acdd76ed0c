// f2_common.cuh -- shared device-side definitions for the F2CNN feature-extraction kernels.
//
// Hot path (reference file:line, relative to tictacmenthe/F2CNN):
//   gammatone/filters.py:195-239      erb_filterbank  (4 cascaded biquads per channel)
//   scripts/processing/EnvelopeExtraction.py:20-67  paddedHilbert / lowPassFilter /
//                                     ExtractEnvelopeFromMatrix
//   scripts/processing/InputGenerator.py:73-80, scripts/CNN/Evaluating.py:70-81  windowing
//
// Everything here is sm_100a-only device code; there is no host/CPU implementation of
// the path in this package.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace f2 {

constexpr int kTile = 256;        // samples per shared-memory tile (divides every ring >= 256)
constexpr int kStages = 4;        // TMA pipeline depth
constexpr int kChanPerBlock = 32;  // channels (threads) per CTA of the fused kernel: one warp
constexpr int kEdgeChanPerBlock = 128;           // channels (threads) per CTA of the sequential edge kernel
constexpr int kRingAlign = 256;   // ring allocations are multiples of this many samples
constexpr int kNumChanPar = 19;   // floats per channel in the parameter block

// Per-channel parameter block, parameter-major: par[i * c_pad + c].
//   0      g4      = A0^4 / gain: output scale of the cascade (filters.py:148,174-182,237)
//   1..4   z[k]    = A1k / A0: the stage's zero           (filters.py:167-170)
//   5..8   cq[k]   = B2 rounded per stage (dithered)      (filters.py:152)
//   9..12  ncy[k]  = -(1 + B1 + B2) rounded per stage     (filters.py:151-152)
//   13..16 nb1[k]  = -B1 rounded per stage: direct-form feedback (with -cq[k]) for the
//                    channel groups whose poles are far enough from z = 1
//   17     group_cy = min over the channel's group of 32 of 1 + B1 + B2 (the fused kernel picks
//                    the section form per group from it)
//   18     group_wscale = (smallest -ln|pole| of the bank) / (smallest -ln|pole| of the channel's group of
//                    32), in (0, 1]: the group's truncated-history lengths are the plan's times this --
//                    a group of wide high-frequency channels forgets its past ten times sooner than
//                    the 100 Hz channels the plan's lengths are derived from
enum ChanPar { P_G4 = 0, P_Z = 1, P_CQ = 5, P_NCY = 9, P_NB1 = 13, P_FORM = 17, P_WSCALE = 18 };

// Groups whose float32 error is predicted above the tolerance (f2_plan_create_ex with
// F2_PLAN_FLOAT64_SECTIONS) run their cascade in float64 (FORM 2): their group_cy entry holds this
// marker, and their exact design coefficients live in a second block of doubles, par64[i * c_pad + c]:
//   0 g4 = A0^4/gain   1..4 z[k] = A1k/A0   5 b1 = B1/B0   6 b2 = B2/B0
constexpr float kForm2Marker = -1.0f;
constexpr int kNumChanPar64 = 7;
enum ChanPar64 { P64_G4 = 0, P64_Z = 1, P64_B1 = 5, P64_B2 = 6 };

// A plan-wide truncated-history length scaled to one channel group, in whole tiles (never longer than
// the plan's, never shorter than one tile).  Host and device use the same expression.
__host__ __device__ __forceinline__ int group_warmup(int w_plan, float wscale) {
    const int v = (int)ceilf((float)w_plan * wscale);
    const int tiles = (v + kTile - 1) / kTile;
    const int w = (tiles < 1 ? 1 : tiles) * kTile;
    return w < w_plan ? w : w_plan;
}

// One utterance (or one matrix row for the stand-alone envelope path).
struct UttDesc {
    long long wave_off;  // first sample in the flat input buffer
    long long ring_off;  // first sample of this utterance's ring in xz / G / Z buffers
    long long full_off;  // first sample (time index) in full-rate time-major outputs
    long long dec_off;   // first frame in the decimated output
    int n;               // samples
    int N2;              // ring length = 2^ceil(log2 n)   (EnvelopeExtraction.py:29)
    int n_dec;           // decimated frames: t = phase + j*step < n
    int log2N2;
    // Injection kernel G[t] = H[(t - n) mod N2]: H depends on the ring size only.  g_tab != null: one of four
    // copies of H (shifted by 0..3 samples, so that every tile start is 16-byte aligned for the bulk copies;
    // each N2 + 256 long, so that a tile never wraps), shared by all utterances of this ring size and
    // L2-resident; tile of ring position tau starts at g_tab[(tau + g_shift) & (N2 - 1)].  null: a private
    // table in the workspace (FusedParams::G + ring_off), filled by the pre-pass.
    const float* g_tab;
    int g_shift;
    int pad_;
};

// One CTA (= one warp) of work: channels [cblock*32, +32) of utterance `utt`, output samples [t0, t1).
struct Item {
    int utt;
    int cblock;
    int t0;
    int t1;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}

// TMA 1-D bulk copy global -> shared, completion signalled on an mbarrier (UBLKCP in SASS).
// dst/src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ float fast_sqrt(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

}  // namespace f2
