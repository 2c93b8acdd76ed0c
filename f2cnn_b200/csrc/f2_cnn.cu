// f2_cnn.cu -- tcgen05 (5th-generation tensor core) forward pass of the reference's F2-direction CNN
// for `cnn eval*` (scripts/CNN/Training.py:93-114, scripts/CNN/Evaluating.py:70-87): the one dense
// contraction next to the feature-extraction hot path (SURVEY.md section 8f rank 1).
//
// See f2_umma.cuh for the operand layout all kernels here share.
#include "f2_cnn.cuh"

#include <cuda_bf16.h>

#include <algorithm>
#include <vector>

#include "f2_umma.cuh"

namespace f2 {

// =====================================================================================================
// Geometry of the reference network for the configured front end (RADIUS = 5 -> 11 dots, 128 channels):
//   input 11 x 128 x 1 -> conv1 3x3 same, 32 -> conv2 3x3 valid, 32 (9 x 126) -> maxpool 2 (4 x 63)
//   -> conv3 3x3 same, 64 -> conv4 3x3 valid, 64 (2 x 61) -> maxpool 2 (1 x 30) -> flatten 1920
//   -> dense 516 relu -> dense 2 softmax                      (Training.py:93-114; dropout is inactive)
// Every convolution is an implicit GEMM with M = 128 output pixels per tensor-core instruction: the
// activations sit in shared memory as [channel / 8][pixel][8 channels] planes (f2_umma.cuh), and filter
// tap (dy, dx) reads the SAME planes through a descriptor advanced by dy * W + dx pixels -- no im2col
// is ever materialised (except the 9-tap patch matrix of the single-channel first layer).  Output
// pixels whose window would wrap around a row end are computed and thrown away (2 of 128..130 columns).
// Three kernels, chained through L2-sized global buffers:
//   cnn_front_kernel   normalizeInput + conv1 + conv2 + pool   (frames straight from the envelope)
//   cnn_mid_kernel     conv3 + conv4 + pool -> 1920 features per frame
//   cnn_dense_kernel   dense 516 + relu + dense 2 + softmax
// A launch scores a list of segments (frame ranges of one envelope, e.g. the utterances of a batch) whose scores
// lie back to back; frames run in chunks that cross segment boundaries.  Only cnn_front_kernel knows where a frame
// comes from (a per-chunk run table, CnnRuns); mid and dense index chunk-local frames.
// =====================================================================================================
namespace cnn {

constexpr int kDots = 11, kChan = 128;
constexpr int kW0 = 130;                     // padded input grid 13 x 130 (zero halo of the `same` conv1)
constexpr int kG0 = 1800;                    // bf16 entries of the padded grid incl. slack for the last tile's taps
constexpr int kTiles1 = 12;                  // conv1: rows q = y*130 + x, q < 1430 -> 12 tiles of 128
constexpr int kRows1 = kTiles1 * 128;        // 1536 rows of the patch matrix
constexpr int kRowsC1 = 1416;                // conv1 output rows p = y*128 + x (1408) + slack for conv2's taps
constexpr int kTiles2 = 9;                   // conv2: one tile per output row y
constexpr int kPool2 = 4 * 63;               // pooled pixels per frame after conv2
constexpr int kW3 = 65;                      // padded conv3 input grid 6 x 65
constexpr int kRowsIn3 = 520;                // 390 + slack for the taps of the third tile
constexpr int kTiles3 = 3;                   // conv3: rows q = y*65 + x, q < 260 -> 3 tiles
constexpr int kRowsC3 = 256;                 // conv3 output rows p = y*63 + x (252) + slack for conv4's taps
constexpr int kFeat = 1920;
constexpr int kHidden = 516, kHiddenPad = 528, kNChunk = 176, kPasses = 3;
constexpr int kKChunk = 64;                  // K per pipeline stage of the dense kernel

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}

__device__ __forceinline__ void copy_to_smem(void* dst, const void* src, int bytes, int tid, int nthreads) {
    const uint4* s = reinterpret_cast<const uint4*>(src);
    uint4* d = reinterpret_cast<uint4*>(dst);
    for (int i = tid; i < bytes / 16; i += nthreads) d[i] = __ldg(s + i);
}

// ---- front: normalizeInput + conv1 + relu + conv2 + relu + maxpool -----------------------------------------
struct FrontSmem {
    static constexpr int w1 = 0;                                   // [2 planes][32][8] bf16
    static constexpr int w2 = w1 + 2 * 32 * 16;                    // [9 taps][4 planes][32][8]
    static constexpr int g0 = w2 + 9 * 4 * 32 * 16;                // padded input grid, bf16
    static constexpr int a1 = (g0 + kG0 * 2 + 127) / 128 * 128;    // patch matrix [2 planes][1536][8]
    static constexpr int c1 = a1 + 2 * kRows1 * 16;                // conv1 output [4 planes][1416][8]
    static constexpr int total = c1 + 4 * kRowsC1 * 16;
};

// Warp roles (front and mid kernels): 16 WORKER warps stage operands and drain accumulators -- warp w reads
// TMEM lanes 32*(w % 4) .., the four warps of a lane quarter share the tiles / columns -- and one ISSUER warp
// does nothing but feed the tensor core (tcgen05.mma from its elected lane).  The two sides meet only on
// mbarriers, never on a CTA-wide barrier, so the issuer can run ahead of the epilogues.
constexpr int kWorkers = 512;
constexpr int kThreads = kWorkers + 32;

__device__ __forceinline__ void worker_sync() { asm volatile("bar.sync 1, 512;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__global__ void __launch_bounds__(kThreads, 1)
cnn_front_kernel(const float* __restrict__ env_t, int step, const CnnRuns runs, int n_frames,
                 const uint8_t* __restrict__ w1p, const uint8_t* __restrict__ w2p, const float* __restrict__ b1,
                 const float* __restrict__ b2, uint8_t* __restrict__ pooled2, int* __restrict__ bad_flags,
                 int* __restrict__ status) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ __align__(8) uint64_t bar[2];   // issuer -> workers: conv1 / conv2 of the current frame have completed
    __shared__ __align__(8) uint64_t rdy[2];   // workers -> issuer: patch matrix staged + TMEM drained / conv1 output written
    __shared__ uint32_t tmem_slot;
    __shared__ float red[32];
    __shared__ float s_b1[32], s_b2[32];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int quarter = warp & 3, group = warp >> 2;
    copy_to_smem(smem + FrontSmem::w1, w1p, 2 * 32 * 16, tid, kThreads);
    copy_to_smem(smem + FrontSmem::w2, w2p, 9 * 4 * 32 * 16, tid, kThreads);
    for (int i = tid; i < (FrontSmem::total - FrontSmem::g0) / 16; i += kThreads)
        reinterpret_cast<uint4*>(smem + FrontSmem::g0)[i] = make_uint4(0, 0, 0, 0);   // halo, slack rows
    if (tid < 32) {
        s_b1[tid] = b1[tid];
        s_b2[tid] = b2[tid];
    }
    if (warp == 0) umma::tmem_alloc(&tmem_slot, 512);
    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        mbar_init(&rdy[0], kWorkers);
        mbar_init(&rdy[1], kWorkers);
        mbar_fence_init();
    }
    umma::fence_smem_to_async();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = tmem_slot;
    const uint32_t s_base = smem_u32(smem);
    constexpr uint32_t kPlaneA1 = kRows1 * 16, kPlaneC1 = kRowsC1 * 16;
    const uint32_t idesc32 = umma::instr_desc_bf16(128, 32);
    uint32_t phase = 0;
    bool alive = true;

    if (warp == kWorkers / 32) {
        // ================================ issuer warp ================================
        const uint64_t da1 = umma::smem_desc(s_base + FrontSmem::a1, kPlaneA1, 128);
        const uint64_t db1 = umma::smem_desc(s_base + FrontSmem::w1, 32 * 16, 128);
        const uint64_t dc1 = umma::smem_desc(s_base + FrontSmem::c1, kPlaneC1, 128);
        const uint64_t db2 = umma::smem_desc(s_base + FrontSmem::w2, 512, 128);
        for (int f = blockIdx.x; f < n_frames && alive; f += gridDim.x) {
            // ---- conv1: 12 tiles x (M128, N32, K16) ----
            alive = umma::mbar_wait_bounded(&rdy[0], phase);
            umma::fence_after_sync();
            if (!alive) break;
            if (umma::elect_one()) {
#pragma unroll
                for (int t = 0; t < kTiles1; ++t) umma::mma_bf16(tmem + (uint32_t)t * 32u, da1 + (uint64_t)(t * 128), db1, idesc32, false);
                umma::mma_commit(&bar[0]);
            }
            __syncwarp();
            // ---- conv2: 9 tiles x 9 taps x 2 x (M128, N32, K16), taps are descriptor shifts ----
            alive = umma::mbar_wait_bounded(&rdy[1], phase);
            umma::fence_after_sync();
            if (!alive) break;
            if (umma::elect_one()) {
#pragma unroll 1
                for (int y = 0; y < kTiles2; ++y) {
#pragma unroll
                    for (int tap = 0; tap < 9; ++tap) {
                        const uint32_t shift = (uint32_t)(y * kChan + (tap / 3) * kChan + (tap % 3));
#pragma unroll
                        for (int kk = 0; kk < 2; ++kk)
                            umma::mma_bf16(tmem + (uint32_t)y * 32u, dc1 + (uint64_t)(shift + (uint32_t)(2 * kk) * (kPlaneC1 / 16)),
                                           db2 + (uint64_t)((tap * 2048 + 2 * kk * 512) / 16), idesc32, tap > 0 || kk > 0);
                    }
                }
                umma::mma_commit(&bar[1]);
            }
            __syncwarp();
            phase ^= 1;
        }
        if (!alive && lane == 0) atomicExch(status, 1);
    } else {
        // ================================ worker warps ================================
        __nv_bfloat16* g0 = reinterpret_cast<__nv_bfloat16*>(smem + FrontSmem::g0);
        const unsigned short* g0u = reinterpret_cast<const unsigned short*>(smem + FrontSmem::g0);
        const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
        // The envelope samples of a frame are fetched one whole iteration before they are needed (global
        // latency is far longer than anything four warps per scheduler can hide): this thread holds channel
        // c, dots k0, k0 + 4, k0 + 8 of the NEXT frame to be staged, and v_seg the segment that frame belongs to.
        const int c = tid & 127, k0 = tid >> 7;
        float v[3] = {1.f, 1.f, 1.f};
        int v_seg = 0;
        auto fetch_input = [&](int f) {
            // the last run that starts at or before chunk frame f (every thread looks at the same entries): a
            // short table is read from the launch parameters at fixed indices (constant bank, no dependent
            // global load ahead of the envelope reads), a long one is binary-searched in the workspace
            CnnRun r = runs.inline_runs[0];
            if (runs.n <= CnnRuns::kInline) {
#pragma unroll
                for (int i = 1; i < CnnRuns::kInline; ++i)
                    if (i < runs.n && runs.inline_runs[i].first <= f) r = runs.inline_runs[i];
            } else {
                int a = 0, b = runs.n - 1;
                while (a < b) {
                    const int m = (a + b + 1) >> 1;
                    if (__ldg(&runs.table[m].first) <= f) a = m;
                    else b = m - 1;
                }
                r = runs.table[a];
            }
            v_seg = r.seg;
            const float* src = env_t + (size_t)(r.row + (f - r.first)) * kChan + c;
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const int k = k0 + 4 * j;
                if (k < kDots) v[j] = __ldg(src + (size_t)k * (size_t)step * kChan);
            }
        };
        // normalizeInput (Training.py:13-28) of the fetched frame into the padded grid, then the 9-tap patch matrix
        auto stage_input = [&]() {
            float lo = INFINITY, hi = -INFINITY;
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                if (k0 + 4 * j < kDots) {
                    lo = fminf(lo, v[j]);
                    hi = fmaxf(hi, v[j]);
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
                hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
            }
            worker_sync();   // `red` of the previous frame has been read by everybody
            if (lane == 0) {
                red[warp] = lo;
                red[16 + warp] = hi;
            }
            worker_sync();
            lo = red[lane & 15];
            hi = red[16 + (lane & 15)];
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) {
                lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
                hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
            }
            if (!(lo > 0.f) && tid == 0) atomicOr(bad_flags + v_seg, 1);   // the reference raises ValueError
            // Within a factor 2 of lo, v - lo and hi - lo are exact and log1pf keeps the digits that
            // logf(v) - logf(lo) would cancel (a frame spanning a few ulps gave NaN or several times its span);
            // beyond it (hi - lo) / lo may overflow and the log difference has no cancellation to speak of.
            const bool close = hi <= 2.f * lo;
            const float llo = logf(lo);
            const float inv = hi > lo ? 1.0f / (close ? log1pf((hi - lo) / lo) : logf(hi) - llo) : 0.f;
            if (close) {   // the same lo and hi in every worker thread: a uniform branch
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const int k = k0 + 4 * j;
                    if (k < kDots) g0[(k + 1) * kW0 + c + 1] = __float2bfloat16(log1pf((v[j] - lo) / lo) * inv);
                }
            } else {
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const int k = k0 + 4 * j;
                    if (k < kDots) g0[(k + 1) * kW0 + c + 1] = __float2bfloat16((logf(v[j]) - llo) * inv);
                }
            }
            worker_sync();
            for (int q = tid; q < kRows1; q += kWorkers) {
                unsigned short t[9];
#pragma unroll
                for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                    for (int dx = 0; dx < 3; ++dx) t[dy * 3 + dx] = g0u[q + dy * kW0 + dx];
                uint4 p0, p1;
                p0.x = (uint32_t)t[0] | ((uint32_t)t[1] << 16);
                p0.y = (uint32_t)t[2] | ((uint32_t)t[3] << 16);
                p0.z = (uint32_t)t[4] | ((uint32_t)t[5] << 16);
                p0.w = (uint32_t)t[6] | ((uint32_t)t[7] << 16);
                p1 = make_uint4((uint32_t)t[8], 0, 0, 0);
                *reinterpret_cast<uint4*>(smem + FrontSmem::a1 + (size_t)q * 16) = p0;
                *reinterpret_cast<uint4*>(smem + FrontSmem::a1 + kPlaneA1 + (size_t)q * 16) = p1;
            }
            umma::fence_smem_to_async();
        };

        int f = blockIdx.x;
        if (f < n_frames) {
            fetch_input(f);
            stage_input();
            if (f + (int)gridDim.x < n_frames) fetch_input(f + gridDim.x);
            umma::fence_before_sync();
            mbar_arrive(&rdy[0]);
        }
        for (; f < n_frames && alive; f += gridDim.x) {
            alive = umma::mbar_wait_bounded(&bar[0], phase);
            umma::fence_after_sync();
            if (!alive) break;
            // ---- epilogue 1: bias + relu -> bf16 planes, rows re-strided from 130 to 128 ----
#pragma unroll 1
            for (int t = group; t < kTiles1; t += 4) {
                float a[32];
                umma::tmem_ld32(tmem + lane_addr + (uint32_t)t * 32u, a);
                const int q = t * 128 + quarter * 32 + lane;
                const int y = q / kW0, x = q - y * kW0;
                if (y < kDots && x < kChan) {
                    uint8_t* dst = smem + FrontSmem::c1 + (size_t)(y * kChan + x) * 16;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        uint4 o;
                        o.x = pack_bf16(fmaxf(a[8 * j + 0] + s_b1[8 * j + 0], 0.f), fmaxf(a[8 * j + 1] + s_b1[8 * j + 1], 0.f));
                        o.y = pack_bf16(fmaxf(a[8 * j + 2] + s_b1[8 * j + 2], 0.f), fmaxf(a[8 * j + 3] + s_b1[8 * j + 3], 0.f));
                        o.z = pack_bf16(fmaxf(a[8 * j + 4] + s_b1[8 * j + 4], 0.f), fmaxf(a[8 * j + 5] + s_b1[8 * j + 5], 0.f));
                        o.w = pack_bf16(fmaxf(a[8 * j + 6] + s_b1[8 * j + 6], 0.f), fmaxf(a[8 * j + 7] + s_b1[8 * j + 7], 0.f));
                        *reinterpret_cast<uint4*>(dst + (size_t)j * kPlaneC1) = o;
                    }
                }
            }
            umma::fence_smem_to_async();
            umma::fence_before_sync();
            mbar_arrive(&rdy[1]);
            // the input grid and the patch matrix are free since conv1 completed: stage the next frame
            // while the tensor core works through conv2
            const bool more = f + (int)gridDim.x < n_frames;
            if (more) {
                stage_input();
                if (f + 2 * (int)gridDim.x < n_frames) fetch_input(f + 2 * gridDim.x);
            }
            alive = umma::mbar_wait_bounded(&bar[1], phase);
            umma::fence_after_sync();
            if (!alive) break;
            // ---- epilogue 2: 2x2 max pool (rows: two tiles, columns: lane pairs) + bias + relu -> global ----
            {
                uint8_t* out = pooled2 + (size_t)f * (4 * kPool2 * 16);
                const int x = quarter * 32 + lane, py = group;
                float a[32], b[32];
                umma::tmem_ld32(tmem + lane_addr + (uint32_t)(2 * py) * 32u, a);
                umma::tmem_ld32(tmem + lane_addr + (uint32_t)(2 * py + 1) * 32u, b);
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    float m = fmaxf(a[j], b[j]);
                    m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));
                    a[j] = fmaxf(m + s_b2[j], 0.f);
                }
                if ((x & 1) == 0 && x < 126) {
                    uint8_t* dst = out + (size_t)(py * 63 + (x >> 1)) * 16;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        uint4 o;
                        o.x = pack_bf16(a[8 * j + 0], a[8 * j + 1]);
                        o.y = pack_bf16(a[8 * j + 2], a[8 * j + 3]);
                        o.z = pack_bf16(a[8 * j + 4], a[8 * j + 5]);
                        o.w = pack_bf16(a[8 * j + 6], a[8 * j + 7]);
                        *reinterpret_cast<uint4*>(dst + (size_t)j * (kPool2 * 16)) = o;
                    }
                }
            }
            if (more) {   // next frame: patch matrix staged, accumulators drained
                umma::fence_before_sync();
                mbar_arrive(&rdy[0]);
            }
            phase ^= 1;
        }
        if (!alive && tid == 0) atomicExch(status, 1);
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem, 512);
}

// ---- mid: conv3 + relu + conv4 + relu + maxpool -> features ------------------------------------------------------
struct MidSmem {
    static constexpr int w3 = 0;                                   // [9][4 planes][64][8]
    static constexpr int w4 = w3 + 9 * 4 * 64 * 16;                // [9][8 planes][64][8]
    static constexpr int in3 = w4 + 9 * 8 * 64 * 16;               // 2 x [4 planes][520][8]
    static constexpr int in3_bytes = 4 * kRowsIn3 * 16;
    static constexpr int c3 = in3 + 2 * in3_bytes;                 // [8 planes][256][8]
    static constexpr int total = c3 + 8 * kRowsC3 * 16;
};

__global__ void __launch_bounds__(kThreads, 1)
cnn_mid_kernel(const uint8_t* __restrict__ pooled2, int n_frames, const uint8_t* __restrict__ w3p, const uint8_t* __restrict__ w4p,
               const float* __restrict__ b3, const float* __restrict__ b4, __nv_bfloat16* __restrict__ feat,
               int* __restrict__ status) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ __align__(8) uint64_t bar[2];    // issuer -> workers: conv3 / conv4 of the current frame have completed
    __shared__ __align__(8) uint64_t rdy_c3;    // workers -> issuer: conv3 output written (and every older accumulator drained)
    __shared__ __align__(8) uint64_t full[2];   // bulk copies of a frame's input have landed
    __shared__ uint32_t tmem_slot;
    __shared__ float s_b3[64], s_b4[64];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int quarter = warp & 3, group = warp >> 2;   // group g handles output channels 16g .. 16g+15
    copy_to_smem(smem + MidSmem::w3, w3p, 9 * 4 * 64 * 16, tid, kThreads);
    copy_to_smem(smem + MidSmem::w4, w4p, 9 * 8 * 64 * 16, tid, kThreads);
    for (int i = tid; i < (MidSmem::total - MidSmem::in3) / 16; i += kThreads)
        reinterpret_cast<uint4*>(smem + MidSmem::in3)[i] = make_uint4(0, 0, 0, 0);   // halo of the `same` conv3, slack rows
    if (tid < 64) {
        s_b3[tid] = b3[tid];
        s_b4[tid] = b4[tid];
    }
    if (warp == 0) umma::tmem_alloc(&tmem_slot, 256);
    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        mbar_init(&rdy_c3, kWorkers);
        mbar_init(&full[0], 1);
        mbar_init(&full[1], 1);
        mbar_fence_init();
    }
    umma::fence_smem_to_async();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = tmem_slot;
    const uint32_t s_base = smem_u32(smem);
    constexpr uint32_t kPlaneIn3 = kRowsIn3 * 16, kPlaneC3 = kRowsC3 * 16;
    const uint32_t idesc64 = umma::instr_desc_bf16(128, 64);
    bool alive = true;

    // interior rows of one frame's pooled conv2 output -> padded grid in buffer b (16 bulk copies of 63 pixels)
    auto fetch = [&](int f, int b) {
        const uint8_t* src = pooled2 + (size_t)f * (4 * kPool2 * 16);
        uint8_t* dst = smem + MidSmem::in3 + (size_t)b * MidSmem::in3_bytes;
        mbar_expect_tx(&full[b], 4 * kPool2 * 16);
        for (int pl = 0; pl < 4; ++pl)
            for (int y = 0; y < 4; ++y)
                tma_load_1d(dst + (size_t)pl * kPlaneIn3 + (size_t)((y + 1) * kW3 + 1) * 16,
                            src + (size_t)pl * (kPool2 * 16) + (size_t)y * 63 * 16, 63 * 16, &full[b]);
    };

    if (warp == kWorkers / 32) {
        // ================================ issuer warp ================================
        // Program order on the tensor pipe makes most hazards vanish: conv3 of frame f+1 is issued behind conv4
        // of frame f, whose issue waited for the epilogue that drained conv3(f)'s columns; conv4(f+1) waits for
        // rdy_c3(f+1), which the workers signal after they are done with everything of frame f.
        const uint64_t dw3 = umma::smem_desc(s_base + MidSmem::w3, 1024, 128);
        const uint64_t dw4 = umma::smem_desc(s_base + MidSmem::w4, 1024, 128);
        const uint64_t dc3 = umma::smem_desc(s_base + MidSmem::c3, kPlaneC3, 128);
        uint32_t phase = 0, full_phase0 = 0, full_phase1 = 0;
        int it = 0;
        for (int f = blockIdx.x; f < n_frames && alive; f += gridDim.x, ++it) {
            const int b = it & 1;
            alive = umma::mbar_wait_bounded(&full[b], b ? full_phase1 : full_phase0);
            if (b) full_phase1 ^= 1; else full_phase0 ^= 1;
            umma::fence_after_sync();
            if (!alive) break;
            if (umma::elect_one()) {
                const uint64_t din = umma::smem_desc(s_base + MidSmem::in3 + (uint32_t)b * MidSmem::in3_bytes, kPlaneIn3, 128);
#pragma unroll 1
                for (int t = 0; t < kTiles3; ++t) {
#pragma unroll
                    for (int tap = 0; tap < 9; ++tap) {
                        const uint32_t shift = (uint32_t)(t * 128 + (tap / 3) * kW3 + (tap % 3));
#pragma unroll
                        for (int kk = 0; kk < 2; ++kk)
                            umma::mma_bf16(tmem + (uint32_t)t * 64u, din + (uint64_t)(shift + (uint32_t)(2 * kk) * (kPlaneIn3 / 16)),
                                           dw3 + (uint64_t)((tap * 4096 + 2 * kk * 1024) / 16), idesc64, tap > 0 || kk > 0);
                    }
                }
                umma::mma_commit(&bar[0]);
            }
            __syncwarp();
            alive = umma::mbar_wait_bounded(&rdy_c3, phase);
            umma::fence_after_sync();
            if (!alive) break;
            if (umma::elect_one()) {
#pragma unroll
                for (int tap = 0; tap < 9; ++tap) {
                    const uint32_t shift = (uint32_t)((tap / 3) * 63 + (tap % 3));
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        umma::mma_bf16(tmem + 192u, dc3 + (uint64_t)(shift + (uint32_t)(2 * kk) * (kPlaneC3 / 16)),
                                       dw4 + (uint64_t)((tap * 8192 + 2 * kk * 1024) / 16), idesc64, tap > 0 || kk > 0);
                }
                umma::mma_commit(&bar[1]);
            }
            __syncwarp();
            phase ^= 1;
        }
        if (!alive && lane == 0) atomicExch(status, 2);
    } else {
        // ================================ worker warps ================================
        const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
        uint32_t phase = 0;
        int it = 0;
        if (tid == 0) {
            if ((int)blockIdx.x < n_frames) fetch(blockIdx.x, 0);
            if ((int)(blockIdx.x + gridDim.x) < n_frames) fetch(blockIdx.x + gridDim.x, 1);
        }
        for (int f = blockIdx.x; f < n_frames && alive; f += gridDim.x, ++it) {
            const int b = it & 1;
            alive = umma::mbar_wait_bounded(&bar[0], phase);
            umma::fence_after_sync();
            if (!alive) break;
            // ---- epilogue 3: bias + relu -> bf16 planes, rows re-strided from 65 to 63; group g: channels 16g.. ----
#pragma unroll
            for (int t = 0; t < kTiles3; ++t) {
                const int q = t * 128 + quarter * 32 + lane;
                const int y = q / kW3, x = q - y * kW3;
                float v[16];
                umma::tmem_ld16(tmem + lane_addr + (uint32_t)t * 64u + (uint32_t)group * 16u, v);
                if (y < 4 && x < 63) {
                    uint8_t* dst = smem + MidSmem::c3 + (size_t)(y * 63 + x) * 16 + (size_t)(2 * group) * kPlaneC3;
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const int c = group * 16 + 8 * j;
                        uint4 o;
                        o.x = pack_bf16(fmaxf(v[8 * j + 0] + s_b3[c + 0], 0.f), fmaxf(v[8 * j + 1] + s_b3[c + 1], 0.f));
                        o.y = pack_bf16(fmaxf(v[8 * j + 2] + s_b3[c + 2], 0.f), fmaxf(v[8 * j + 3] + s_b3[c + 3], 0.f));
                        o.z = pack_bf16(fmaxf(v[8 * j + 4] + s_b3[c + 4], 0.f), fmaxf(v[8 * j + 5] + s_b3[c + 5], 0.f));
                        o.w = pack_bf16(fmaxf(v[8 * j + 6] + s_b3[c + 6], 0.f), fmaxf(v[8 * j + 7] + s_b3[c + 7], 0.f));
                        *reinterpret_cast<uint4*>(dst + (size_t)j * kPlaneC3) = o;
                    }
                }
            }
            umma::fence_smem_to_async();
            umma::fence_before_sync();
            mbar_arrive(&rdy_c3);
            alive = umma::mbar_wait_bounded(&bar[1], phase);
            umma::fence_after_sync();
            if (!alive) break;
            // ---- epilogue 4: bias + relu -> staging [p][64] bf16 (over this frame's input buffer, now dead) ----
            uint8_t* stage = smem + MidSmem::in3 + (size_t)b * MidSmem::in3_bytes;   // 128 rows x 128 bytes
            {
                const int p = quarter * 32 + lane;
                float v[16];
                umma::tmem_ld16(tmem + lane_addr + 192u + (uint32_t)group * 16u, v);
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int c = group * 16 + 8 * j;
                    uint4 o;
                    o.x = pack_bf16(fmaxf(v[8 * j + 0] + s_b4[c + 0], 0.f), fmaxf(v[8 * j + 1] + s_b4[c + 1], 0.f));
                    o.y = pack_bf16(fmaxf(v[8 * j + 2] + s_b4[c + 2], 0.f), fmaxf(v[8 * j + 3] + s_b4[c + 3], 0.f));
                    o.z = pack_bf16(fmaxf(v[8 * j + 4] + s_b4[c + 4], 0.f), fmaxf(v[8 * j + 5] + s_b4[c + 5], 0.f));
                    o.w = pack_bf16(fmaxf(v[8 * j + 6] + s_b4[c + 6], 0.f), fmaxf(v[8 * j + 7] + s_b4[c + 7], 0.f));
                    // 16-byte chunks of a row are rotated by the row index: conflict-free column reads below
                    *reinterpret_cast<uint4*>(stage + (size_t)p * 128 + (size_t)(((2 * group + j) + p) & 7) * 16) = o;
                }
            }
            worker_sync();
            // ---- 2x2 max pool over (y, x) in {0,1} x {2px, 2px+1} -> 30 x 64 features (Keras flatten order x*64 + c) ----
            if (tid < 30 * 8) {
                const int px = tid >> 3, g = tid & 7;
                __nv_bfloat162 m[4];
                bool first = true;
#pragma unroll
                for (int yy = 0; yy < 2; ++yy)
#pragma unroll
                    for (int xx = 0; xx < 2; ++xx) {
                        const int p = yy * 63 + 2 * px + xx;
                        const uint4 r = *reinterpret_cast<const uint4*>(stage + (size_t)p * 128 + (size_t)((g + p) & 7) * 16);
                        const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
                        for (int k = 0; k < 4; ++k) m[k] = first ? h2[k] : __hmax2(m[k], h2[k]);
                        first = false;
                    }
                *reinterpret_cast<uint4*>(feat + (size_t)f * kFeat + (size_t)px * 64 + (size_t)g * 8) = *reinterpret_cast<uint4*>(m);
            }
            worker_sync();
            // restore the zero halo the staging rows overwrote and hand the buffer back to the bulk-copy engine
            for (int i = tid; i < 128 * 8; i += kWorkers) reinterpret_cast<uint4*>(stage)[i] = make_uint4(0, 0, 0, 0);
            umma::fence_smem_to_async();
            worker_sync();
            if (tid == 0 && f + 2 * (int)gridDim.x < n_frames) fetch(f + 2 * gridDim.x, b);
            phase ^= 1;
        }
        if (!alive && tid == 0) atomicExch(status, 2);
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem, 256);
}

// ---- dense: 1920 -> 516 relu -> 2 softmax ----------------------------------------------------------------------------
struct DenseSmem {
    static constexpr int a_bytes = 8 * 128 * 16;        // one K chunk of 128 frames
    static constexpr int b_bytes = 8 * kNChunk * 16;    // one K chunk of 176 hidden units
    static constexpr int stage_bytes = a_bytes + b_bytes;
    static constexpr int stages = 3;
    static constexpr int total = stages * stage_bytes;
};

__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}

__global__ void __launch_bounds__(128, 1)
cnn_dense_kernel(const __nv_bfloat16* __restrict__ feat, int n_frames, const uint8_t* __restrict__ w5p, const float* __restrict__ b5,
                 const float* __restrict__ w6, const float* __restrict__ b6, float* __restrict__ scores, int* __restrict__ status) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ __align__(8) uint64_t bar_stage[DenseSmem::stages];
    __shared__ __align__(8) uint64_t bar_acc;
    __shared__ uint32_t tmem_slot;
    __shared__ float s_b5[kHiddenPad], s_w6[kHiddenPad * 2];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (int i = tid; i < kHiddenPad; i += 128) {
        s_b5[i] = i < kHidden ? b5[i] : 0.f;
        s_w6[2 * i] = i < kHidden ? w6[2 * i] : 0.f;
        s_w6[2 * i + 1] = i < kHidden ? w6[2 * i + 1] : 0.f;
    }
    if (warp == 0) umma::tmem_alloc(&tmem_slot, 256);
    if (tid == 0) {
        for (int s = 0; s < DenseSmem::stages; ++s) mbar_init(&bar_stage[s], 1);
        mbar_init(&bar_acc, 1);
        mbar_fence_init();
    }
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = tmem_slot;
    const uint32_t s_base = smem_u32(smem);
    const int row0 = blockIdx.x * 128;
    constexpr int kChunks = kFeat / kKChunk;            // 30
    constexpr int kIters = kPasses * kChunks;           // 90
    const uint32_t idesc = umma::instr_desc_bf16(128, kNChunk);

    auto load = [&](int it) {
        const int pass = it / kChunks, kc = it % kChunks, s = it % DenseSmem::stages;
        uint8_t* sa = smem + (size_t)s * DenseSmem::stage_bytes;
        uint8_t* sb = sa + DenseSmem::a_bytes;
        for (int i = tid; i < 128 * 8; i += 128) {
            const int r = i >> 3, p8 = i & 7;
            const int row = min(row0 + r, n_frames - 1);
            cp_async16(sa + (size_t)p8 * 2048 + (size_t)r * 16, feat + (size_t)row * kFeat + (size_t)kc * kKChunk + (size_t)p8 * 8);
        }
        const uint8_t* wsrc = w5p + ((size_t)pass * kChunks + (size_t)kc) * DenseSmem::b_bytes;
        for (int i = tid; i < DenseSmem::b_bytes / 16; i += 128) cp_async16(sb + (size_t)i * 16, wsrc + (size_t)i * 16);
    };

    uint32_t stage_phase[DenseSmem::stages] = {0, 0, 0};
    uint32_t acc_phase = 0;
    bool alive = true;
    float l0 = 0.f, l1 = 0.f;
    load(0);
    asm volatile("cp.async.commit_group;" ::: "memory");
    load(1);
    asm volatile("cp.async.commit_group;" ::: "memory");
    for (int it = 0; it < kIters && alive; ++it) {
        const int s = it % DenseSmem::stages, kc = it % kChunks;
        if (it + 2 < kIters) {
            const int s2 = (it + 2) % DenseSmem::stages;
            if (it >= 1) {   // stage s2 was read by the MMAs of iteration it - 1
                alive = umma::mbar_wait_bounded(&bar_stage[s2], stage_phase[s2]);
                stage_phase[s2] ^= 1;
                if (!alive) break;
            }
            load(it + 2);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 2;" ::: "memory");
        umma::fence_smem_to_async();
        umma::fence_before_sync();
        __syncthreads();
        if (tid == 0) {
            umma::fence_after_sync();
            const uint32_t sa = s_base + (uint32_t)s * DenseSmem::stage_bytes, sb = sa + DenseSmem::a_bytes;
            for (int kk = 0; kk < kKChunk / 16; ++kk) {
                const uint64_t da = umma::smem_desc(sa + (uint32_t)(2 * kk) * 2048u, 2048, 128);
                const uint64_t db = umma::smem_desc(sb + (uint32_t)(2 * kk) * (kNChunk * 16u), kNChunk * 16, 128);
                umma::mma_bf16(tmem, da, db, idesc, kc > 0 || kk > 0);
            }
            umma::mma_commit(&bar_stage[s]);
            if (kc == kChunks - 1) umma::mma_commit(&bar_acc);
        }
        if (kc == kChunks - 1) {
            // ---- epilogue of one pass: 176 hidden units of this thread's frame -> two logits ----
            alive = umma::mbar_wait_bounded(&bar_acc, acc_phase);
            acc_phase ^= 1;
            umma::fence_after_sync();
            if (!alive) break;
            const int n0 = (it / kChunks) * kNChunk;
            for (int c0 = 0; c0 < kNChunk; c0 += 16) {
                float v[16];
                umma::tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int n = n0 + c0 + j;
                    const float h = fmaxf(v[j] + s_b5[n], 0.f);
                    l0 = fmaf(h, s_w6[2 * n], l0);
                    l1 = fmaf(h, s_w6[2 * n + 1], l1);
                }
            }
            umma::fence_before_sync();
            __syncthreads();   // every warp has read the accumulator before the next pass overwrites it
        }
    }
    if (alive) {
        const int row = row0 + warp * 32 + lane;
        if (row < n_frames) {
            l0 += b6[0];
            l1 += b6[1];
            const float m = fmaxf(l0, l1);
            const float e0 = __expf(l0 - m), e1 = __expf(l1 - m);
            const float inv = 1.0f / (e0 + e1);
            scores[(size_t)row * 2] = e0 * inv;
            scores[(size_t)row * 2 + 1] = e1 * inv;
        }
    } else if (tid == 0) {
        atomicExch(status, 3);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem, 256);
}

}  // namespace cnn

size_t cnn_workspace_bytes(long long chunk_frames) {
    const size_t pooled = (size_t)chunk_frames * 4 * cnn::kPool2 * 16;
    const size_t feat = (size_t)chunk_frames * cnn::kFeat * 2;
    const size_t runs = (size_t)chunk_frames * sizeof(CnnRun);   // a chunk holds at most one run per frame
    return ((pooled + 255) / 256 + (feat + 255) / 256 + (runs + 255) / 256) * 256 + 256;
}

cudaError_t configure_cnn_kernels() {
    using namespace cnn;
    cudaError_t e = cudaFuncSetAttribute(cnn_front_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FrontSmem::total);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(cnn_mid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MidSmem::total);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(cnn_dense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DenseSmem::total);
    return e;
}

cudaError_t launch_cnn_forward(const CnnWeights& w, const float* env_t, int step, const long long* seg_rows,
                               const long long* seg_frames, int n_segs, long long chunk_frames, float* scores, int* flags,
                               void* workspace, int sm_count, cudaStream_t stream) {
    using namespace cnn;
    uint8_t* pooled2 = (uint8_t*)(((size_t)workspace + 255) / 256 * 256);
    const size_t pooled_bytes = ((size_t)chunk_frames * 4 * kPool2 * 16 + 255) / 256 * 256;
    __nv_bfloat16* feat = (__nv_bfloat16*)(pooled2 + pooled_bytes);
    const size_t feat_bytes = ((size_t)chunk_frames * kFeat * 2 + 255) / 256 * 256;
    CnnRun* runs_dev = (CnnRun*)((uint8_t*)feat + feat_bytes);
    long long total = 0;
    for (int s = 0; s < n_segs; ++s) total += seg_frames[s];
    std::vector<CnnRun> runs;
    CnnRuns param{};
    param.table = runs_dev;
    int s0 = 0;            // first segment that still has frames at or after f0
    long long g0 = 0;      // its first frame in the scores
    for (long long f0 = 0; f0 < total; f0 += chunk_frames) {
        const int nf = (int)std::min<long long>(chunk_frames, total - f0);
        while (s0 < n_segs && g0 + seg_frames[s0] <= f0) g0 += seg_frames[s0++];
        runs.clear();
        for (long long s = s0, g = g0; s < n_segs && g < f0 + nf; g += seg_frames[s++]) {
            if (seg_frames[s] == 0) continue;
            const long long skip = std::max<long long>(f0 - g, 0);   // frames of the segment in earlier chunks
            runs.push_back(CnnRun{(int)(g + skip - f0), (int)s, seg_rows[s] + skip});
        }
        param.n = (int)runs.size();
        if (param.n <= CnnRuns::kInline) {
            std::copy(runs.begin(), runs.end(), param.inline_runs);
        } else {
            // pageable source: the copy is staged before the call returns, so `runs` may be refilled right away;
            // stream order keeps the table of the previous chunk until its front kernel has read it
            cudaError_t e = cudaMemcpyAsync(runs_dev, runs.data(), runs.size() * sizeof(CnnRun), cudaMemcpyHostToDevice, stream);
            if (e != cudaSuccess) return e;
        }
        const int grid = std::min(nf, sm_count);
        cnn_front_kernel<<<grid, kThreads, FrontSmem::total, stream>>>(env_t, step, param, nf, w.w1, w.w2, w.b1, w.b2, pooled2,
                                                                  flags, flags + n_segs);
        cnn_mid_kernel<<<grid, kThreads, MidSmem::total, stream>>>(pooled2, nf, w.w3, w.w4, w.b3, w.b4, feat, flags + n_segs);
        cnn_dense_kernel<<<(nf + 127) / 128, 128, DenseSmem::total, stream>>>(feat, nf, w.w5, w.b5, w.w6, w.b6, scores + (size_t)f0 * 2,
                                                                              flags + n_segs);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// ---- self-test: one 128 x N x K product through the exact descriptor conventions of the CNN kernels ---
// D[r][n] = sum_k A[shift + r][k] * B[n][k], r < 128.  A: [a_rows][K], B: [N][K] row-major bf16 in global
// memory; both are re-laid into K-major planes in shared memory, A's descriptor is advanced by `shift`
// rows (the convolution-tap trick).  variant 1 swaps the leading / stride byte offsets (must be WRONG:
// kept so that the test proves the convention rather than assuming it).
__global__ void __launch_bounds__(128, 1)
umma_selftest_kernel(const __nv_bfloat16* __restrict__ A, int a_rows, const __nv_bfloat16* __restrict__ B, int N, int K,
                     int shift, int variant, float* __restrict__ D, int* __restrict__ status) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int planes = K / 8;
    const uint32_t plane_a = (uint32_t)a_rows * 16u, plane_b = (uint32_t)N * 16u;
    uint8_t* sa = smem;
    uint8_t* sb = smem + (size_t)planes * plane_a;
    for (int i = tid; i < a_rows * planes; i += blockDim.x) {
        const int r = i / planes, p = i % planes;
        *reinterpret_cast<uint4*>(sa + (size_t)p * plane_a + (size_t)r * 16) =
            *reinterpret_cast<const uint4*>(A + (size_t)r * K + (size_t)p * 8);
    }
    for (int i = tid; i < N * planes; i += blockDim.x) {
        const int r = i / planes, p = i % planes;
        *reinterpret_cast<uint4*>(sb + (size_t)p * plane_b + (size_t)r * 16) =
            *reinterpret_cast<const uint4*>(B + (size_t)r * K + (size_t)p * 8);
    }
    uint32_t cols = 32;
    while ((int)cols < N) cols <<= 1;
    if (warp == 0) umma::tmem_alloc(&tmem_slot, cols);
    if (tid == 0) {
        mbar_init(&bar, 1);
        mbar_fence_init();
    }
    umma::fence_smem_to_async();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = tmem_slot;
    if (tid == 0) {
        const uint32_t idesc = umma::instr_desc_bf16(128, N);
        for (int kk = 0; kk < K / 16; ++kk) {
            const uint32_t a_addr = smem_u32(sa) + (uint32_t)(2 * kk) * plane_a + (uint32_t)shift * 16u;
            const uint32_t b_addr = smem_u32(sb) + (uint32_t)(2 * kk) * plane_b;
            const uint64_t da = variant == 1 ? umma::smem_desc(a_addr, 128, plane_a) : umma::smem_desc(a_addr, plane_a, 128);
            const uint64_t db = variant == 1 ? umma::smem_desc(b_addr, 128, plane_b) : umma::smem_desc(b_addr, plane_b, 128);
            umma::mma_bf16(tmem, da, db, idesc, kk > 0);
        }
        umma::mma_commit(&bar);
    }
    const bool ok = umma::mbar_wait_bounded(&bar, 0);
    umma::fence_after_sync();
    if (!ok) {
        if (tid == 0) *status = 1;  // the MMAs never completed
    } else {
        for (int c0 = 0; c0 < N; c0 += 16) {
            float v[16];
            umma::tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
#pragma unroll
            for (int j = 0; j < 16; ++j) D[(size_t)(warp * 32 + lane) * N + c0 + j] = v[j];
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem, cols);
}

cudaError_t launch_umma_selftest(const void* A, int a_rows, const void* B, int N, int K, int shift, int variant, float* D,
                                 int* status, cudaStream_t stream) {
    const size_t smem = (size_t)(K / 8) * ((size_t)a_rows + (size_t)N) * 16;
    cudaError_t e = cudaFuncSetAttribute(umma_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    umma_selftest_kernel<<<1, 128, smem, stream>>>((const __nv_bfloat16*)A, a_rows, (const __nv_bfloat16*)B, N, K, shift,
                                                    variant, D, status);
    return cudaGetLastError();
}


}  // namespace f2
