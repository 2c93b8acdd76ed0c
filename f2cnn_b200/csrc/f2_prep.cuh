// f2_prep.cuh -- launch interface of the ring / Hilbert pre-pass (f2_prep.cu).
#pragma once
#include "f2_common.cuh"

// sample dtypes accepted at the C-ABI (mirrors include/f2cnn_b200.h)
#define F2_DT_I16 0
#define F2_DT_F32 1
#define F2_DT_F64 2

namespace f2 {

struct PrepParams {
    const UttDesc* utts;
    const void* wave;  // flat samples, dtype wave_dtype
    int wave_dtype;
    float* bufA;       // FFT scratch, ring_len floats per utterance
    float* bufB;       // FFT scratch, ring_len floats per utterance
    float2* xz;        // out: (x, xi) rings
    float* G;          // out: injection kernel rings; must alias bufA (free once the forward
                       // transform is done) or be null (plain Hilbert, no table)
    int hilbert;       // 0: filterbank-only run, skip the FFTs and leave xi = 0
    int cluster;       // set by launch_prep: N2 = 32768 ... 131072 go through the cluster kernels
};

struct HostPrepInfo {
    int n_utts;
    int min_log2N2;
    int max_log2N2;
    int private_g;   // utterances whose injection table lives in the workspace (UttDesc::g_tab == null)
};

constexpr int kGTabMinLog = 8, kGTabMaxLog = 20;   // ring sizes that share one injection table per device
// device pointer to the four shifted copies (stride floats apart) of the table for N2 = 2^log2N2 on the
// current device, or null (size out of range / out of memory: use per-utterance tables)
const float* injection_table(int log2N2, int* stride);
bool ring_cluster_enabled();   // false only under F2CNN_B200_RING_CLUSTER=0
cudaError_t init_twiddles(cudaStream_t stream);
cudaError_t launch_prep(const PrepParams& p, const HostPrepInfo& h, cudaStream_t stream);

}  // namespace f2
