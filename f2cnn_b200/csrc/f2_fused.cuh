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
    float* env_t;        // full-rate envelope, time-major [t][C]            (nullable)
    void* gfb_cn;        // full-rate filterbank output in the REFERENCE layout: (C, n_u) blocks back to back,
    void* env_cn;        //   float64 or float32 (gfb_cn_f64, env_cn_f64) -- stored by the kernel through a
                         //   shared-memory transpose (nullable)
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
    const double* chan64;  // [kNumChanPar64][c_pad] float64 block of the FORM 2 groups (FORM 2 launch only)
    const double* edge64;  // float64 edge residuals [utt][C][8] of the FORM 2 groups (f2_edge.cu; null: in-kernel)
    int gfb_cn_f64;      // element type of gfb_cn: 1 = float64, 0 = float32
    int env_cn_f64;      // element type of env_cn: 1 = float64, 0 = float32
    // Cutoff sweep (f2_batch_run_cutoffs; 0 = off): plane j of the decimated frames is stored at
    // dec + j * plane_stride.  Plane j reads one-pole state sw_state[j] (-1: no low-pass); states
    // 0 .. sw_lp-1 have their own lp_k and b0.  lpf and w_lpf then describe the slowest of them.
    int sw_planes;
    int sw_lp;
    int sw_state[4];
    float sw_k[4];
    float sw_b0[4];
    long long plane_stride;
};

constexpr int kMaxCutoffs = 4;

// float64: p.items are work items of FORM 2 groups (float64 sections), run by their own instantiations.
cudaError_t launch_fused(const FusedParams& p, int n_items, bool float64, cudaStream_t stream);

}  // namespace f2
