// f2_cnn.cuh -- launch interface of the tcgen05 CNN forward kernels (f2_cnn.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace f2 {

// Device pointers to the network's parameters, packed on the host (f2_capi.cu: f2_cnn_create) into the
// K-major plane layout the kernels copy straight into shared memory; biases and the last layer in float32.
struct CnnWeights {
    const uint8_t* w1;  // conv1 [2 planes][32 out][8]: taps 0..7 | tap 8 + zeros           (bf16)
    const uint8_t* w2;  // conv2 [9 taps][4 planes][32 out][8 in]
    const uint8_t* w3;  // conv3 [9 taps][4 planes][64 out][8 in]
    const uint8_t* w4;  // conv4 [9 taps][8 planes][64 out][8 in]
    const uint8_t* w5;  // dense1 [3 passes][30 K chunks][8 planes][176 out][8 in], out padded 516 -> 528
    const float* b1;
    const float* b2;
    const float* b3;
    const float* b4;
    const float* b5;    // [516]
    const float* w6;    // dense2 [516][2]
    const float* b6;    // [2]
};

// Frames of one chunk that come from one segment, back to back: chunk frames first .. (the next run's first) - 1
// belong to segment `seg` and read env_t from row `row` on.  cnn_front_kernel looks a frame's run up
// in the chunk's table, ordered by `first`.
struct alignas(16) CnnRun {
    int first;
    int seg;
    long long row;
};
// The run table of one chunk as a kernel parameter: up to kInline runs travel with the launch, so that no copy
// precedes the kernel in the stream (a chunk of utterances of 0.7 s or more has at most four runs; the parameter
// is kept small because every launch uploads it); a longer table is uploaded to the workspace and `table` points
// to it.
struct CnnRuns {
    static constexpr int kInline = 4;
    CnnRun inline_runs[kInline];
    const CnnRun* table;
    int n;
};

// Pooled conv2 output, features and the run table of one chunk of chunk_frames frames.
size_t cnn_workspace_bytes(long long chunk_frames);
// Raises the dynamic shared-memory limit of the three CNN kernels on the CURRENT device.  A function
// attribute belongs to one device's copy of the kernel, so every device that runs the network needs this
// once (f2_cnn_create calls it under its device guard).
cudaError_t configure_cnn_kernels();
// Segment s = seg_frames[s] frames of the time-major envelope env_t ([rows][128] float32) starting at row
// seg_rows[s]: frame i of it = rows seg_rows[s] + i + k*step, k < 11 (Evaluating.py:70-78).  The segments' frames
// lie back to back in scores ([sum seg_frames][2] float32 softmax) and are run in chunks of chunk_frames, a chunk
// crossing segment boundaries.  flags[s] != 0 when a frame of segment s held a value <= 0, flags[n_segs] != 0
// when the tensor-core pipeline did not complete.  seg_rows / seg_frames are host arrays.
cudaError_t launch_cnn_forward(const CnnWeights& w, const float* env_t, int step, const long long* seg_rows,
                               const long long* seg_frames, int n_segs, long long chunk_frames, float* scores, int* flags,
                               void* workspace, int sm_count, cudaStream_t stream);

cudaError_t launch_umma_selftest(const void* A, int a_rows, const void* B, int N, int K, int shift, int variant, float* D,
                                 int* status, cudaStream_t stream);

}  // namespace f2
