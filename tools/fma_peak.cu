// fma_peak.cu -- register-resident FP32 FMA microbenchmark (SURVEY.md section 8d asks for the
// sustained FMA peak next to the nominal 148*128*2*f).  Measures scalar FFMA, packed FFMA2 and
// float64 DFMA issue rates with 8 independent chains per thread, all SMs busy, for ~2 s each so
// that the power-capped clock is the one observed.  The DFMA rate is what the float64 sections
// (FORM 2) of the fused kernel run at.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

// MODE 0: scalar FFMA, register operands (what the fused kernel's per-channel coefficients
// are); 1: packed FFMA2, register operands; 2: scalar FFMA with constant-bank operands;
// 3: float64 DFMA, register operands (the same 128 FMAs per iteration).
template <int MODE>
__global__ void __launch_bounds__(256) fma_kernel(float* out, int iters, float a_in, float b_in) {
    constexpr int PACKED = (MODE == 1);
    const float a = MODE == 2 ? a_in : a_in + threadIdx.x * 1e-9f;
    const float b = MODE == 2 ? b_in : b_in + threadIdx.x * 1e-9f;
    float2 x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = make_float2(threadIdx.x * 1e-3f + i, blockIdx.x * 1e-4f - i);
    const float2 a2 = make_float2(a, a), b2 = make_float2(b, b);
    if (MODE == 3) {
        double2 d[8];
        const double ad = a, bd = b;
#pragma unroll
        for (int i = 0; i < 8; ++i) d[i] = make_double2(x[i].x, x[i].y);
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int r = 0; r < 8; ++r) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    d[i].x = fma(d[i].x, ad, bd);
                    d[i].y = fma(d[i].y, ad, bd);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = make_float2((float)d[i].x, (float)d[i].y);
    } else
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                if (PACKED) x[i] = __ffma2_rn(x[i], a2, b2);
                else { x[i].x = fmaf(x[i].x, a, b); x[i].y = fmaf(x[i].y, a, b); }
            }
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += x[i].x + x[i].y;
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

static void launch(int mode, int blocks, int threads, float* out, int iters) {
    if (mode == 1) fma_kernel<1><<<blocks, threads>>>(out, iters, 0.999f, 1e-3f);
    else if (mode == 2) fma_kernel<2><<<blocks, threads>>>(out, iters, 0.999f, 1e-3f);
    else if (mode == 3) fma_kernel<3><<<blocks, threads>>>(out, iters, 0.999f, 1e-3f);
    else fma_kernel<0><<<blocks, threads>>>(out, iters, 0.999f, 1e-3f);
}

int main(int argc, char** argv) {
    double secs = argc > 1 ? atof(argv[1]) : 2.0;
    cudaDeviceProp p;
    cudaGetDeviceProperties(&p, 0);
    const int blocks = p.multiProcessorCount * 8, threads = 256;
    float* out;
    cudaMalloc(&out, sizeof(float) * blocks * threads);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    for (int packed = 0; packed < 4; ++packed) {
        int iters = 2000;
        float ms = 0.f;
        double total_ms = 0.0, best = 0.0, flops_sum = 0.0;
        int reps = 0;
        // warm-up, then repeat launches for `secs` seconds
        for (int w = 0; w < 3; ++w) {
            launch(packed, blocks, threads, out, iters);
        }
        cudaDeviceSynchronize();
        while (total_ms < secs * 1e3) {
            cudaEventRecord(e0);
            launch(packed, blocks, threads, out, iters);
            cudaEventRecord(e1);
            cudaEventSynchronize(e1);
            cudaEventElapsedTime(&ms, e0, e1);
            const double flops = 2.0 * 2.0 * 64.0 * (double)iters * blocks * threads;  // 64 float2 FMAs/iter
            const double tf = flops / (ms * 1e-3) / 1e12;
            if (tf > best) best = tf;
            flops_sum += flops;
            total_ms += ms;
            ++reps;
        }
        static const char* kinds[] = {"ffma_reg", "ffma2_reg", "ffma_const", "dfma_reg"};
        printf("{\"kind\": \"%s\", \"device\": \"%s\", \"sms\": %d, \"burst_tflops\": %.2f, \"sustained_tflops\": %.2f, "
               "\"reps\": %d}\n", kinds[packed], p.name, p.multiProcessorCount, best, flops_sum / (total_ms * 1e-3) / 1e12, reps);
    }
    return 0;
}
