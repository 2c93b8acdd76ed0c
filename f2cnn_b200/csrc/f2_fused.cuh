// f2_fused.cuh -- launch interface of the fused filterbank+envelope kernel (f2_fused.cu).
#pragma once
#include "f2_common.cuh"

namespace f2 {

struct FusedParams {
    const UttDesc* utts;
    const Item* items;
    const float* chan;   // [kNumChanPar][c_pad] per-channel parameter block
    const float2* xz;    // rings: (x[t], Im hilbert(x_padded)[t])
    const float* G;      // rings: circular Hilbert kernel aligned to each utterance's edge
    float* gfb_t;        // full-rate filterbank output, time-major [t][C]   (nullable)
    float* env_t;        // full-rate envelope, time-major [t][C]            (nullable)
    void* gfb_cn;        // full-rate filterbank output in the REFERENCE layout: (C, n_u) blocks back to back,
    void* env_cn;        //   float64 or float32 -- stored by the kernel through a shared-memory transpose (nullable)
    int cn_f64;          // element type of gfb_cn / env_cn: 1 = float64, 0 = float32
    float* dec;          // decimated envelope frames [frame][C]             (nullable)
    float* win;          // windows of win_dots consecutive frames [row][win_dots][C]   (nullable)
    const long long* win_off;  // [n_utts+1] first window row of each utterance
    int win_dots;
    const float* edge;   // precomputed edge residuals [utt][C][8] (f2_edge.cu); null: compute in-kernel
    int C;
    int c_pad;
    int step;            // decimation step: int(fs * SAMPLING_PERIOD / 1e6)   (InputGenerator.py:65)
    int phase;           // first decimated sample
    int lpf;             // apply the butter(1) low-pass                      (EnvelopeExtraction.py:61-64)
    float lp_k;          // -a1 of butter(1, cutoff/8000)
    float lp_b0;         // b0 of the same
    int w_imag;          // warm-up lengths, multiples of kTile
    int w_edge;
    int w_casc;
    int w_lpf;
    float direct_min_cy; // groups of 32 channels with min(1+B1+B2) >= this run the direct-form sections
    const double* chan64;  // [kNumChanPar64][c_pad] float64 block of the FORM 2 groups (launch_fused64 only)
    const double* edge64;  // float64 edge residuals [utt][C][8] of the FORM 2 groups (f2_edge.cu; null: in-kernel)
};

cudaError_t launch_fused(const FusedParams& p, int n_items, cudaStream_t stream);
// The work items of FORM 2 groups (float64 sections): its own instantiation of the fused kernel.
cudaError_t launch_fused64(const FusedParams& p, int n_items, cudaStream_t stream);

}  // namespace f2
