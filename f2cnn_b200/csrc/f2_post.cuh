// f2_post.cuh -- launch interfaces of the layout / windowing kernels (f2_post.cu).
#pragma once
#include "f2_common.cuh"
#include "f2_prep.cuh"

namespace f2 {

cudaError_t launch_gather_rows(const float* src, const long long* base, long long n_rows, int dots,
                               long long stride, int C, float* out, cudaStream_t stream);
cudaError_t launch_gather_index(const float* src, const long long* idx, long long n_idx, int C, float* out,
                                cudaStream_t stream);
cudaError_t launch_dense_frames(const float* env_t, int C, int dots, int step, long long i0, long long i1,
                                int normalize, void* out, int out_dtype, int* bad_flag, cudaStream_t stream);
cudaError_t launch_gather_cn(const void* env, int dtype, int C, long long n, const long long* idx, long long n_idx,
                             float* out, cudaStream_t stream);
cudaError_t launch_rows_envelope(const UttDesc* rows, int n_rows, const float2* xz, int op, int lpf, float lp_k,
                                 float lp_b0, void* out, int out_dtype, cudaStream_t stream);

}  // namespace f2
