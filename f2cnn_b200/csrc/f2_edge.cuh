// f2_edge.cuh -- edge residuals of the zero-padded ring equation, one pass per utterance
// (f2_edge.cu): sequential kernel for full GPUs, chunked scan kernel for small batches.
#pragma once
#include "f2_sections.cuh"

namespace f2 {

constexpr int kScanBlock = 64;    // samples per lane block of the edge scan
constexpr int kScanLevels = 5;    // Kogge-Stone offsets 1, 2, 4, 8, 16 blocks
constexpr int kScanWindow = 32 * kScanBlock;  // 2048 samples: the last w_edge samples

// seq: one thread per channel runs the real cascade over the last w_edge samples.  FORM 0: the float32
// delta-form pass of every group into the float table.  FORM 2: the groups with P_FORM == kForm2Marker in
// float64 into a float64 table of the same layout; the entries of other groups are not written.
template <int FORM>
cudaError_t launch_edge(const UttDesc* utts, int n_utts, const float* chan, const double* chan64, int C, int c_pad,
                        const float2* xz, int w_edge, typename SectionTypes<FORM>::E* edge, cudaStream_t stream);
// scan: one warp per (utterance, channel); lane = block of 64 samples run from zero state;
// the 8-state cascade carries are composed across lanes with precomputed block transition
// powers M^(2^d) (lower block-triangular, 2x2 blocks per biquad) and warp shuffles.
// scan_mats: [C][kScanLevels][8][8] float32.
cudaError_t launch_edge_scan(const UttDesc* utts, int n_utts, const float* chan, const float* scan_mats, int C,
                             int c_pad, const float2* xz, float* edge, cudaStream_t stream);

// Host: one-step homogeneous transition of the a0-free delta-form cascade (state order
// y1,q1,...,y4,q4) for a channel's float32 parameters, raised to kScanBlock * 2^d.
void build_scan_matrices(const float* par, int c_pad, int c, float* out /* [kScanLevels][8][8] */);

}  // namespace f2
