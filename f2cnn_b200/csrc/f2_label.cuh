// f2_label.cuh -- launch interface of the slope-label and label-accuracy kernels (f2_label.cu).
#pragma once
#include <cuda_runtime.h>

namespace f2 {

// out[i] = (slope, intercept, r, p) of item i; see f2_label.cu.
cudaError_t launch_label_fit(const double* formant, const long long* first, const int* center, long long n_items,
                             int dots, int step, double* out, cudaStream_t stream);

// hits[u], counted[u] (zeroed here) = the label accuracy counts of utterance u's frames; see f2_label.cu.
cudaError_t launch_label_accuracy(const float* scores, const long long* score_offsets, const long long* times,
                                  const int* classes, const long long* label_offsets, int n_utts, int step,
                                  long long* hits, long long* counted, cudaStream_t stream);

}  // namespace f2
