// f2_capi.cu -- the C ABI declared in include/f2cnn_b200.h: plans, batches, launch sequences.
// Host-side only; every FLOP of the hot path runs in the kernels of f2_prep.cu, f2_fused.cu
// and f2_post.cu.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <vector>

#include "../../include/f2cnn_b200.h"
#include "f2_cnn.cuh"
#include "f2_edge.cuh"
#include "f2_fused.cuh"
#include "f2_label.cuh"
#include "f2_post.cuh"
#include "f2_prep.cuh"
#include "f2_sections.cuh"

static_assert(F2_I16 == F2_DT_I16 && F2_F32 == F2_DT_F32 && F2_F64 == F2_DT_F64, "dtype codes");

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define F2_CUDA(expr)                                                                        \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) return fail(F2_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() {
        int cur = -1;
        if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
    }
};

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
int round_up_tile(double v) { return (int)(ceil(v / f2::kTile) * f2::kTile); }
constexpr float kDirectMinCyGfb = 0.25f;
constexpr float kDirectMinCyEnv = 0.035f;
constexpr double kDirectCost = 0.85;  // time per sample of a direct-form group / delta-form group (measured)
// the same for a FORM 2 (float64) group: 20.3 ms for the float64 group of a 16 kHz / 128 ch / LOW_FREQ 20 bank over
// the bench corpus against ~11.7 ms for the same group in float32 delta form (B200 at 1000 W,
// tools/float64_sections_bench.py, profiles/r03b_float64_sections.log)
constexpr double kForm2Cost = 1.75;

// Per-stage float32 rounding whose SUM over the four stages is as close to 4*c as the
// float32 lattice allows.  The four sections share their poles, so the first-order error of
// the cascade response depends only on the sum of the per-stage denominator errors: choosing
// m of 4 stages one ulp up cuts the effective coefficient error from ulp/2 to ulp/8.
void dither4(double c, float out[4]) {
    float r = (float)c;
    float lo = ((double)r <= c) ? r : nextafterf(r, -INFINITY);
    float hi = nextafterf(lo, INFINITY);
    double frac = (c - (double)lo) / ((double)hi - (double)lo);
    int m = (int)floor(4.0 * frac + 0.5);
    for (int k = 0; k < 4; ++k) out[k] = (k < m) ? hi : lo;
}

void butter1(double cutoff_hz, double* b0, double* a1) {
    // scipy.signal.butter(1, Wn, 'low'), Wn = cutoff/8000 (EnvelopeExtraction.py:47):
    // pre-warp with fs=2, bilinear transform of 1/(s+1).
    const double Wn = cutoff_hz / 8000.0;
    const double w = 4.0 * tan(M_PI * Wn / 2.0);
    *b0 = w / (4.0 + w);
    *a1 = -(4.0 - w) / (4.0 + w);
}

// ---- section coefficients of a make_erb_filters row k = [A0, A11, A12, A13, A14, A2, B0, B1, B2, gain] -----
// 1 + B1 + B2 = |1 - pole|^2: how close the channel's poles come to z = 1
double chan_cy(const double* k) { return 1.0 + (k[7] + k[8]) / k[6]; }

// min of 1 + B1 + B2 over group g of 32 channels (one warp of the fused kernel, whose section form the
// group takes from it)
double group_min_cy(const double* coefs, int C, int g) {
    double cy = 1e300;
    for (int c = g * 32; c < std::min(C, g * 32 + 32); ++c) cy = std::min(cy, chan_cy(coefs + (size_t)c * 10));
    return cy;
}

// The exact values of one channel's sections (FORM 2 runs them; the probe's float64 reference too)
struct Sections {
    double g4;     // A0^4/gain (A0 = A0/B0)
    double z[4];   // A1k/A0
    double b1, b2; // B1/B0, B2/B0
    double nlr;    // -ln |pole|
};

// The channel's float32 entries of the parameter block (g4, z, dithered cq / ncy / nb1) written to
// col[i * stride], and its exact values.
Sections chan_sections(const double* k, float* col, size_t stride) {
    Sections d;
    const double a0n = k[0] / k[6];
    d.g4 = a0n * a0n * a0n * a0n / k[9];
    d.b1 = k[7] / k[6];
    d.b2 = k[8] / k[6];
    d.nlr = -0.5 * log(d.b2);
    float cq[4], ncy[4], nb1[4];
    dither4(d.b2, cq);
    dither4(-(1.0 + d.b1 + d.b2), ncy);
    dither4(-d.b1, nb1);
    col[(size_t)f2::P_G4 * stride] = (float)d.g4;
    for (int s = 0; s < 4; ++s) {
        d.z[s] = k[1 + s] / k[0];
        col[(size_t)(f2::P_Z + s) * stride] = (float)d.z[s];
        col[(size_t)(f2::P_CQ + s) * stride] = cq[s];
        col[(size_t)(f2::P_NCY + s) * stride] = ncy[s];
        col[(size_t)(f2::P_NB1 + s) * stride] = nb1[s];
    }
    return d;
}

// ---- float32 tolerance guard -------------------------------------------------------------------
// The kernels compute in float32 and are held to 1e-4 x channel RMS against the reference's float64
// (north star).  How close a bank's poles may come to z = 1 before float32 round-off breaks that
// depends on more than 1 + B1 + B2 (LOW_FREQ = 20 Hz passes at width 1 and 0.5 and fails at width 2
// under a loud tone in the stop band, profiles/r01o_fuzz.log), so instead of a formula the plan is
// TRIED: the real cascade of the channels nearest to z = 1 is run here on the host, once in float32
// through the kernels' own cascade_real (f2_sections.cuh: same fmaf calls in the same order, on the
// parameter-block column the plan uploads, in the section form of the channel's group) and once in
// float64, on probe signals that cover the observed worst cases -- loud tones far above the channel and
// white noise.  The error is measured the way the parity tests measure it: max |y32 - y64| over
// max(channel RMS, 1 % of the loudest channel's).
template <int FORM>
double probe_channel(const float* col, const Sections& d, const float* x, int n, double loudest_rms) {
    f2::Coef k;
    f2::load_coef<FORM>(col, nullptr, 1, 0, true, k);
    f2::State s;
    f2::reset(s);
    double Y[4] = {0, 0, 0, 0}, Y2[4] = {0, 0, 0, 0}, UP0 = 0.0;
    double err = 0.0, power = 0.0;
    for (int t = 0; t < n; ++t) {
        f2::cascade_real<FORM>(k, s, x[t]);
        // float64, exact coefficients: y[t] = in - b1 y[t-1] - b2 y[t-2]
        double U = x[t], UP = UP0;
        UP0 = U;
        for (int i = 0; i < 4; ++i) {
            const double in = U + d.z[i] * UP;
            const double yo = Y[i];
            const double yn = in - d.b1 * yo - d.b2 * Y2[i];
            Y2[i] = yo;
            Y[i] = yn;
            UP = yo;
            U = yn;
        }
        const double ref = Y[3] * d.g4;
        err = std::max(err, fabs((double)(k.g4 * s.y[3].x) - ref));
        power += ref * ref;
    }
    const double scale = std::max(sqrt(power / n), 0.01 * loudest_rms);
    return scale > 0.0 ? err / scale : 0.0;
}

constexpr int kProbeChannels = 6;

// the (up to kProbeChannels) channels of [c0, c1) nearest to z = 1
std::vector<int> nearest_to_one(const double* coefs, int c0, int c1) {
    std::vector<int> order;
    for (int c = c0; c < c1; ++c) order.push_back(c);
    std::sort(order.begin(), order.end(),
              [&](int a, int b) { return chan_cy(coefs + (size_t)a * 10) < chan_cy(coefs + (size_t)b * 10); });
    order.resize((size_t)std::min(c1 - c0, kProbeChannels));
    return order;
}

// worst predicted error of the channels `order`, in units of the 1e-4 tolerance
double probe_float32_error(const double* coefs, int C, const std::vector<int>& order, int* worst_channel) {
    constexpr int kProbeLen = 8192;
    constexpr double kAmp = 8000.0;
    std::vector<float> x((size_t)kProbeLen);
    double worst = 0.0;
    if (worst_channel) *worst_channel = order.empty() ? 0 : order[0];
    const double tones[] = {M_PI / 2.0, M_PI / 8.0, 0.1727875959474386 /* 440 Hz at 16 kHz */, 0.0 /* white noise */};
    for (double w : tones) {
        double loudest;
        if (w > 0.0) {
            for (int t = 0; t < kProbeLen; ++t) x[(size_t)t] = (float)rint(kAmp * sin(w * t));
            loudest = kAmp / M_SQRT2;  // the channel centred on the tone passes it with unit gain
        } else {
            uint64_t st = 0x9E3779B97F4A7C15ull;
            for (int t = 0; t < kProbeLen; ++t) {  // sum of 4 uniforms: near-Gaussian, sigma ~ 3000 like the bench input
                double acc = 0.0;
                for (int k = 0; k < 4; ++k) {
                    st = st * 6364136223846793005ull + 1442695040888963407ull;
                    acc += (double)(st >> 40) / (double)(1 << 24) - 0.5;
                }
                x[(size_t)t] = (float)rint(acc * 3000.0 * sqrt(3.0));
            }
            loudest = 0.0;  // broadband: every channel is held to its own RMS
        }
        for (int c : order) {
            float col[f2::kNumChanPar] = {};
            const Sections d = chan_sections(coefs + (size_t)c * 10, col, 1);
            const bool direct = group_min_cy(coefs, C, c / 32) >= kDirectMinCyGfb;
            const double e = (direct ? probe_channel<1>(col, d, x.data(), kProbeLen, loudest)
                                     : probe_channel<0>(col, d, x.data(), kProbeLen, loudest)) / 1e-4;
            if (e > worst) {
                worst = e;
                if (worst_channel) *worst_channel = c;
            }
        }
    }
    return worst;
}

// worst predicted error of the bank: its channels nearest to z = 1
double bank_float32_error(const double* coefs, int C, int* worst_channel) {
    return probe_float32_error(coefs, C, nearest_to_one(coefs, 0, C), worst_channel);
}

// the same per group of 32 channels (one warp of the fused kernel): the group's channels nearest to z = 1
void group_float32_errors(const double* coefs, int C, double* per_group) {
    for (int g = 0; g * 32 < C; ++g)
        per_group[g] = probe_float32_error(coefs, C, nearest_to_one(coefs, g * 32, std::min(C, g * 32 + 32)), nullptr);
}

int check_coefs(const double* coefs, int n_channels) {
    for (int c = 0; c < n_channels; ++c) {
        const double* k = coefs + (size_t)c * 10;
        if (!(k[6] != 0.0) || !(k[0] != 0.0) || !(k[9] > 0.0) || !isfinite(k[9]))
            return fail(F2_ERR_INVALID, "channel %d: A0 == 0, B0 == 0 or gain <= 0", c);
    }
    return F2_OK;
}

}  // namespace

// error channel of the other translation units of the library (f2_host.cpp); not exported
extern "C" int f2_set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

struct f2_plan {
    int device = 0;
    int C = 0;
    int c_pad = 0;
    float* d_chan = nullptr;
    float* d_scan_mats = nullptr;  // [C][kScanLevels][8][8] block transition powers for the edge scan
    std::vector<float> h_chan;  // host copy of the parameter block (for the __constant__ upload)
    long long id = 0;
    int w_imag = 0, w_edge = 0, w_casc = 0;
    double min_neg_log_r = 0.0;
    double* d_chan64 = nullptr;  // [kNumChanPar64][c_pad] float64 block of the FORM 2 groups (null: none)
    std::vector<unsigned char> f64_group;  // per group of 32 channels: runs FORM 2
    int n_f64 = 0;
};

namespace {
// time per sample of a channel group relative to a delta-form group: direct form kDirectCost, FORM 2 kForm2Cost
double group_cost(const f2_plan* plan, int cb) {
    const float cy = plan->h_chan[(size_t)f2::P_FORM * plan->c_pad + (size_t)cb * 32];
    if (cy == f2::kForm2Marker) return kForm2Cost;
    return cy >= kDirectMinCyEnv ? kDirectCost : 1.0;
}
}  // namespace

struct f2_batch {
    f2_plan* plan = nullptr;
    int n_utts = 0;
    int step = 1, phase = 0;
    std::vector<f2::UttDesc> utts;
    std::vector<long long> frame_off;
    long long n_items = 0;
    long long n_whole = 0;  // items if no utterance were split in time
    f2::UttDesc* d_utts = nullptr;
    f2::Item* d_items = nullptr;
    // equal-LENGTH chunks for the runs that store the full-rate filterbank output (store-bound: every
    // channel group costs the same per sample); null when the two decompositions coincide
    f2::Item* d_items_uniform = nullptr;
    long long n_items_uniform = 0;
    // the last n_items_f64 (n_items_uniform_f64) of each list belong to FORM 2 groups
    long long n_items_f64 = 0, n_items_uniform_f64 = 0;
    long long total_samples = 0, total_frames = 0, total_ring = 0;
    int min_log2 = 0, max_log2 = 0;
    int private_g = 0;  // utterances without a shared injection table
};

extern "C" {

const char* f2_last_error(void) { return g_err; }
int f2_abi_version(void) { return 6; }

int f2_lowpass_coefficients(double cutoff_hz, double* b0, double* a1) {
    if (!b0 || !a1 || !(cutoff_hz > 0.0) || !(cutoff_hz < 8000.0))
        return fail(F2_ERR_INVALID, "cutoff must be in (0, 8000) Hz, got %g", cutoff_hz);
    butter1(cutoff_hz, b0, a1);
    return F2_OK;
}

int f2_bank_check(const double* coefs, int n_channels, double* predicted, int* worst_channel) {
    if (!coefs || n_channels <= 0 || !predicted) return fail(F2_ERR_INVALID, "f2_bank_check: bad arguments");
    if (const int rc = check_coefs(coefs, n_channels)) return rc;
    *predicted = bank_float32_error(coefs, n_channels, worst_channel);
    return F2_OK;
}

int f2_bank_check_groups(const double* coefs, int n_channels, double* per_group) {
    if (!coefs || n_channels <= 0 || !per_group) return fail(F2_ERR_INVALID, "f2_bank_check_groups: bad arguments");
    if (const int rc = check_coefs(coefs, n_channels)) return rc;
    group_float32_errors(coefs, n_channels, per_group);
    return F2_OK;
}

int f2_plan_create(const double* coefs, int n_channels, int device, f2_plan** out) {
    return f2_plan_create_ex(coefs, n_channels, device, 0u, out);
}

int f2_plan_create_ex(const double* coefs, int n_channels, int device, unsigned flags, f2_plan** out) {
    if (!coefs || !out || n_channels <= 0) return fail(F2_ERR_INVALID, "f2_plan_create: bad arguments");
    if (flags & ~(unsigned)F2_PLAN_FLOAT64_SECTIONS) return fail(F2_ERR_INVALID, "f2_plan_create_ex: unknown flags 0x%x", flags);
    int ndev = 0;
    F2_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(F2_ERR_INVALID, "device %d out of range (%d visible)", device, ndev);
    DeviceGuard guard(device);
    if (!guard.ok) return fail(F2_ERR_CUDA, "cannot select device %d", device);
    cudaDeviceProp prop;
    F2_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(F2_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                    prop.major, prop.minor);

    const int C = n_channels;
    const int c_pad = (int)align_up((size_t)C, 32);
    std::vector<float> par((size_t)f2::kNumChanPar * c_pad, 0.f);
    std::vector<Sections> sec((size_t)C);
    double min_nlr = 1e300;
    for (int c = 0; c < C; ++c) {
        const double* k = coefs + (size_t)c * 10;
        const double A0 = k[0], A2 = k[5], B0 = k[6], B1 = k[7], B2 = k[8], gain = k[9];
        if (A2 != 0.0) return fail(F2_ERR_UNSUPPORTED, "channel %d: A2 != 0 is not a make_erb_filters bank", c);
        if (!(B0 != 0.0) || !(gain > 0.0) || !isfinite(gain))
            return fail(F2_ERR_INVALID, "channel %d: B0 == 0 or gain <= 0", c);
        const double b1 = B1 / B0, b2 = B2 / B0;
        if (!(b2 > 0.0 && b2 < 1.0) || !(fabs(b1) < 1.0 + b2))
            return fail(F2_ERR_UNSUPPORTED, "channel %d: poles are not a stable complex pair", c);
        if (!(A0 != 0.0)) return fail(F2_ERR_INVALID, "channel %d: A0 == 0", c);
        sec[(size_t)c] = chan_sections(k, par.data() + c, (size_t)c_pad);
        min_nlr = std::min(min_nlr, sec[(size_t)c].nlr);
    }
    for (int g0 = 0; g0 < c_pad; g0 += 32) {
        // Per group of 32 channels (one warp of the fused kernel): min of 1 + B1 + B2.  The fused kernel
        // runs the direct form (3 FMAs per section) where this is large enough for its float32 round-off
        // to match the delta form's, and the delta form nearer to z = 1.
        const float cy = (float)group_min_cy(coefs, C, g0 / 32);
        // How much sooner than the bank's slowest channel the group's slowest channel forgets
        // (ratio of -ln|pole|, rounded up a little so that float32 never shortens a length).
        double nlr = 1e300;
        for (int c = g0; c < std::min(C, g0 + 32); ++c) nlr = std::min(nlr, sec[(size_t)c].nlr);
        const float scale = (float)std::min(1.0, min_nlr / nlr * (1.0 + 1e-6));
        for (int c = g0; c < g0 + 32; ++c) {
            par[(size_t)f2::P_FORM * c_pad + c] = cy;
            par[(size_t)f2::P_WSCALE * c_pad + c] = scale;
        }
    }
    // F2_PLAN_FLOAT64_SECTIONS: in a bank f2_bank_check refuses, the groups predicted to leave the tolerance in
    // float32 run FORM 2.  A bank it accepts keeps float32 everywhere, so that the flag never changes its
    // outputs.  A refused bank always flags a group: its worst channel is among the probed channels of its
    // own group, so that group's prediction is at least the bank's.
    const int n_groups = c_pad / 32;
    std::vector<unsigned char> f64_group((size_t)n_groups, 0);
    std::vector<double> par64;
    if ((flags & F2_PLAN_FLOAT64_SECTIONS) && bank_float32_error(coefs, C, nullptr) > 1.0) {
        std::vector<double> per_group((size_t)n_groups);
        group_float32_errors(coefs, C, per_group.data());
        for (int g = 0; g < n_groups; ++g) f64_group[(size_t)g] = per_group[(size_t)g] > 1.0;
        par64.assign((size_t)f2::kNumChanPar64 * c_pad, 0.0);
        for (int c = 0; c < C; ++c) {
            if (!f64_group[(size_t)(c / 32)]) continue;
            const Sections& d = sec[(size_t)c];
            par64[(size_t)f2::P64_G4 * c_pad + c] = d.g4;
            for (int s = 0; s < 4; ++s) par64[(size_t)(f2::P64_Z + s) * c_pad + c] = d.z[s];
            par64[(size_t)f2::P64_B1 * c_pad + c] = d.b1;
            par64[(size_t)f2::P64_B2 * c_pad + c] = d.b2;
        }
        for (int c = 0; c < c_pad; ++c)
            if (f64_group[(size_t)(c / 32)]) par[(size_t)f2::P_FORM * c_pad + c] = f2::kForm2Marker;
    }
    const int n_f64 = (int)std::count(f64_group.begin(), f64_group.end(), (unsigned char)1);
    if (!(flags & F2_PLAN_FLOAT64_SECTIONS)) {
        // a bank whose float32 result would leave the stated tolerance is refused, not answered quietly
        int bad = 0;
        const double predicted = bank_float32_error(coefs, C, &bad);
        if (predicted > 1.0 && !getenv("F2CNN_B200_ALLOW_IMPRECISE"))
            return fail(F2_ERR_UNSUPPORTED,
                        "filterbank too close to z = 1 for float32: channel %d (1+B1+B2 = %.3g) is predicted to miss "
                        "the 1e-4 x RMS tolerance by %.1fx (f2_bank_check); widen LOW_FREQ / lower `width`, or set "
                        "F2CNN_B200_ALLOW_IMPRECISE=1 to run anyway", bad, chan_cy(coefs + (size_t)bad * 10), predicted);
    }
    f2_plan* p = new (std::nothrow) f2_plan();
    if (!p) return fail(F2_ERR_INVALID, "out of host memory");
    static long long next_id = 1;
    p->id = next_id++;
    p->h_chan = par;
    p->device = device;
    p->C = C;
    p->c_pad = c_pad;
    p->min_neg_log_r = min_nlr;
    p->f64_group = f64_group;
    p->n_f64 = n_f64;
    // truncated-history lengths.  The cascade's impulse response decays like t^3 r^t, so for an
    // input that adds up coherently (a tone on the slowest channel's centre) the part of the steady
    // state older than W samples is Gamma(4, -W ln r)/6 of the whole: 7e-7 at 21.5/-ln r (w_imag),
    // 2e-9 at 29/-ln r (w_edge, w_casc) -- below float32 resolution.  On broadband input the error is
    // flat down to 18/-ln r (tools/warmup_sweep.py), but that would leave 1.5e-5 in the coherent
    // case (and 4e-3 on a 3-sample input, whose 4-sample ring is nothing but coherent) for a 1 % gain.
    p->w_imag = round_up_tile(21.5 / min_nlr);
    p->w_edge = round_up_tile(29.0 / min_nlr);
    p->w_casc = p->w_edge;
    std::vector<float> mats((size_t)C * f2::kScanLevels * 64);
    for (int c = 0; c < C; ++c) f2::build_scan_matrices(par.data(), c_pad, c, mats.data() + (size_t)c * f2::kScanLevels * 64);
    cudaError_t e = cudaMalloc(&p->d_chan, par.size() * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(p->d_chan, par.data(), par.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_scan_mats, mats.size() * sizeof(float));
    if (e == cudaSuccess)
        e = cudaMemcpy(p->d_scan_mats, mats.data(), mats.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess && n_f64 > 0) {
        e = cudaMalloc(&p->d_chan64, par64.size() * sizeof(double));
        if (e == cudaSuccess)
            e = cudaMemcpy(p->d_chan64, par64.data(), par64.size() * sizeof(double), cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess) e = f2::init_twiddles(0);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        if (p->d_chan) cudaFree(p->d_chan);
        if (p->d_chan64) cudaFree(p->d_chan64);
        if (p->d_scan_mats) cudaFree(p->d_scan_mats);
        delete p;
        return fail(F2_ERR_CUDA, "plan upload: %s", cudaGetErrorString(e));
    }
    *out = p;
    return F2_OK;
}

int f2_plan_destroy(f2_plan* plan) {
    if (!plan) return F2_OK;
    DeviceGuard guard(plan->device);
    if (plan->d_chan) cudaFree(plan->d_chan);
    if (plan->d_chan64) cudaFree(plan->d_chan64);
    if (plan->d_scan_mats) cudaFree(plan->d_scan_mats);
    delete plan;
    return F2_OK;
}

int f2_plan_channels(const f2_plan* plan) { return plan ? plan->C : 0; }

int f2_plan_float64_groups(const f2_plan* plan, unsigned char* mask, int n_groups) {
    if (!plan || n_groups < 0 || (n_groups > 0 && !mask)) {
        fail(F2_ERR_INVALID, "f2_plan_float64_groups: bad arguments");
        return -1;
    }
    for (int g = 0; g < n_groups; ++g) mask[g] = g < (int)plan->f64_group.size() ? plan->f64_group[(size_t)g] : 0;
    return plan->n_f64;
}

int f2_plan_set_warmup(f2_plan* plan, int w_imag, int w_edge, int w_casc) {
    if (!plan) return fail(F2_ERR_INVALID, "null plan");
    if (w_imag > 0) plan->w_imag = round_up_tile(w_imag);
    if (w_edge > 0) plan->w_edge = round_up_tile(w_edge);
    if (w_casc > 0) plan->w_casc = round_up_tile(w_casc);
    return F2_OK;
}

int f2_plan_get_warmup(const f2_plan* plan, int* w_imag, int* w_edge, int* w_casc) {
    if (!plan) return fail(F2_ERR_INVALID, "null plan");
    if (w_imag) *w_imag = plan->w_imag;
    if (w_edge) *w_edge = plan->w_edge;
    if (w_casc) *w_casc = plan->w_casc;
    return F2_OK;
}

int f2_batch_create(f2_plan* plan, const int64_t* lengths, int n_utts, int step, int phase, int64_t target_items,
                    f2_batch** out) {
    if (!plan || !out || n_utts < 0 || (n_utts > 0 && !lengths) || step <= 0 || phase < 0)
        return fail(F2_ERR_INVALID, "f2_batch_create: bad arguments");
    f2_batch* b = new (std::nothrow) f2_batch();
    if (!b) return fail(F2_ERR_INVALID, "out of host memory");
    b->plan = plan;
    b->n_utts = n_utts;
    b->step = step;
    b->phase = phase;
    b->utts.resize((size_t)n_utts);
    b->frame_off.assign((size_t)n_utts + 1, 0);
    b->min_log2 = 64;
    b->max_log2 = 0;
    long long wave = 0, ring = 0, frames = 0;
    for (int u = 0; u < n_utts; ++u) {
        const int64_t n = lengths[u];
        if (n < 0 || n > ((int64_t)1 << 25)) {
            delete b;
            return fail(F2_ERR_UNSUPPORTED, "utterance %d: %lld samples (supported: 0 .. 2^25)", u, (long long)n);
        }
        int lg = 0;
        while (((int64_t)1 << lg) < n) ++lg;  // N2 = 2^ceil(log2 n)   (EnvelopeExtraction.py:29)
        f2::UttDesc& d = b->utts[(size_t)u];
        d.wave_off = wave;
        d.ring_off = ring;
        d.full_off = wave;
        d.dec_off = frames;
        d.n = (int)n;
        d.N2 = 1 << lg;
        d.log2N2 = lg;
        d.n_dec = n > phase ? (int)((n - phase + step - 1) / step) : 0;
        d.g_tab = nullptr;   // filled below, on the plan's device
        d.g_shift = 0;
        d.pad_ = 0;
        b->frame_off[(size_t)u] = frames;
        wave += n;
        ring += (long long)align_up((size_t)d.N2, f2::kRingAlign);
        frames += d.n_dec;
        if (n > 0) {
            b->min_log2 = std::min(b->min_log2, lg);
            b->max_log2 = std::max(b->max_log2, lg);
        }
    }
    if (b->min_log2 > b->max_log2) b->min_log2 = b->max_log2 = 0;
    b->frame_off[(size_t)n_utts] = frames;
    b->total_samples = wave;
    b->total_frames = frames;
    b->total_ring = ring;

    int sm_count = 148;
    cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, plan->device);
    // ---- work items: (utterance, channel block, time chunk) -------------------------------
    const int cblocks = (plan->C + f2::kChanPerBlock - 1) / f2::kChanPerBlock;
    // Time chunking policy, counted in units of 128 channels (512 such units are resident on the
    // 148 SMs at a time, whatever the CTA width).  Whole utterances when they already give ~1 wave;
    // otherwise chunks, preferably >= 16384 samples (each chunk pays w_casc (+ w_lpf) samples of
    // warm-up) and a whole number of waves, never below 2048.
    const int units = (plan->C + 127) / 128;
    const long long wave_ctas = 148 * 4;
    long long whole = 0;
    for (int u = 0; u < n_utts; ++u) whole += lengths[u] > 0 ? units : 0;
    long long seg = (long long)1 << 40;  // no splitting
    if (target_items > 0) {
        if (whole < target_items && wave > 0)
            seg = (long long)align_up((size_t)std::max<long long>(wave * units / target_items, 2048), f2::kTile);
    } else if (whole < wave_ctas && wave > 0) {
        long long best = std::max<long long>(wave * units / wave_ctas, 2048);
        for (int waves = 4; waves >= 2; --waves) {
            const long long cand = wave * units / (waves * wave_ctas);
            if (cand >= 16384) { best = cand; break; }
        }
        seg = (long long)align_up((size_t)best, f2::kTile);
    }
    // Chunks of equal COST, not equal length (automatic policy only): a direct-form group runs a
    // sample in kDirectCost of a delta-form group's time and every group pays its own warm-up W_g per
    // chunk (group_warmup), so  (seg_g + W_g) * cost_g = T  for all groups, with T such that the total
    // number of chunks stays what equal chunks of `seg` samples would give.  With about one wave of
    // CTAs (a single long stream) all CTAs then finish together instead of the slow groups finishing last.
    std::vector<long long> seg_of((size_t)cblocks, seg);
    if (target_items <= 0 && seg < ((long long)1 << 40) && cblocks > 1) {
        std::vector<double> cost((size_t)cblocks), W((size_t)cblocks);
        for (int cb = 0; cb < cblocks; ++cb) {
            const size_t c0 = (size_t)cb * 32;
            cost[(size_t)cb] = group_cost(plan, cb);
            W[(size_t)cb] = (double)f2::group_warmup(plan->w_casc, plan->h_chan[(size_t)f2::P_WSCALE * plan->c_pad + c0]) + 2048.0;
        }
        auto seg_at = [&](double T, int cb) { return std::max(2048.0, T / cost[(size_t)cb] - W[(size_t)cb]); };
        double lo = 0.0, hi = 4.0 * ((double)seg + (double)plan->w_casc + 2048.0);
        for (int it = 0; it < 80; ++it) {
            const double T = 0.5 * (lo + hi);
            double chunks = 0.0;  // chunks per sample, summed over the groups
            for (int cb = 0; cb < cblocks; ++cb) chunks += 1.0 / seg_at(T, cb);
            if (chunks > (double)cblocks / (double)seg) lo = T; else hi = T;
        }
        for (int cb = 0; cb < cblocks; ++cb)
            seg_of[(size_t)cb] = (long long)align_up((size_t)seg_at(0.5 * (lo + hi), cb), f2::kTile);
    }
    auto build_items = [&](const std::vector<long long>& segs, bool same_for_all) {
        std::vector<f2::Item> out;
        auto push = [&](int u, int cb, long long t0, long long len, int n) {
            f2::Item it;
            it.utt = u;
            it.cblock = cb;
            it.t0 = (int)t0;
            it.t1 = (int)std::min<long long>(n, t0 + len);
            out.push_back(it);
        };
        for (int u = 0; u < n_utts; ++u) {
            const int n = b->utts[(size_t)u].n;
            if (n <= 0) continue;
            auto chunk_len = [&](long long sg) {
                const long long nseg = std::max<long long>(1, (n + sg - 1) / sg);
                return (long long)align_up((size_t)((n + nseg - 1) / nseg), f2::kTile);
            };
            if (same_for_all) {
                // the channel groups of one time chunk next to each other: they share ring tiles and, in
                // the full-rate modes, write the same time-major rows
                const long long len = chunk_len(segs[0]);
                for (long long t0 = 0; t0 < n; t0 += len)
                    for (int cb = 0; cb < cblocks; ++cb) push(u, cb, t0, len, n);
            } else {
                for (int cb = 0; cb < cblocks; ++cb) {
                    const long long len = chunk_len(segs[(size_t)cb]);
                    for (long long t0 = 0; t0 < n; t0 += len) push(u, cb, t0, len, n);
                }
            }
        }
        // Longest first -- the hardware dispatches CTAs in index order, and the channel groups of an utterance stay
        // neighbours, so they share its ring tiles in L2 -- except for the last two waves of the launch, which go
        // most expensive first: cost = (samples + the group's warm-up, which runs as scalar code at ~0.6 of a
        // sample's price) x the group's section form (a direct-form group runs a sample in kDirectCost of a
        // delta-form group's time), so that the launch does not end on slow delta-form items.  On the corpus:
        // 38.85 ms by length alone, 38.43 ms with the two-wave tail (4.3 GB read), 38.34 ms with the whole list by
        // cost (5.6 GB read: the delta-form group of an utterance then runs far ahead of its siblings).
        std::vector<double> gcost((size_t)cblocks), gwarm((size_t)cblocks);
        for (int cb = 0; cb < cblocks; ++cb) {
            const size_t c0 = (size_t)cb * 32;
            const float wscale = plan->h_chan[(size_t)f2::P_WSCALE * plan->c_pad + c0];
            gcost[(size_t)cb] = group_cost(plan, cb);
            gwarm[(size_t)cb] = 0.6 * (f2::group_warmup(plan->w_imag, wscale) + f2::group_warmup(plan->w_edge, wscale));
        }
        const bool whole_utterances = seg >= ((long long)1 << 40);
        auto by_length = [](const f2::Item& a, const f2::Item& c) { return (a.t1 - a.t0) > (c.t1 - c.t0); };
        auto by_cost = [&](const f2::Item& a, const f2::Item& c) {
            return ((a.t1 - a.t0) + gwarm[(size_t)a.cblock]) * gcost[(size_t)a.cblock] >
                   ((c.t1 - c.t0) + gwarm[(size_t)c.cblock]) * gcost[(size_t)c.cblock];
        };
        std::stable_sort(out.begin(), out.end(), by_length);
        if (whole_utterances) {   // time chunks are cut to equal cost already
            const size_t tail = std::min(out.size(), (size_t)sm_count * 16 * 2);
            std::stable_sort(out.end() - (long)tail, out.end(), by_cost);
        }
        // One wave or less (a shard of the corpus on one of eight GPUs): the CTAs are handed to the SMs round
        // after round, so with items in descending order the first SMs collect the most expensive item of every
        // round.  Every other round reversed ("snake"), all SMs get about the same sum: 5.92 -> 5.82 ms on a
        // 1/8 shard (rounds of two CTAs per SM measured best; tools/shard_sweep.py).
        if (whole_utterances && out.size() <= (size_t)sm_count * 16) {
            const size_t round = (size_t)sm_count * 2;
            for (size_t r0 = round; r0 < out.size(); r0 += 2 * round)
                std::reverse(out.begin() + (long)r0, out.begin() + (long)std::min(out.size(), r0 + round));
        }
        return out;
    };
    const std::vector<long long> seg_same((size_t)cblocks, seg);
    const bool equal_cost = seg_of != seg_same;
    std::vector<f2::Item> items = build_items(seg_of, !equal_cost);
    std::vector<f2::Item> items_uniform;
    if (equal_cost) items_uniform = build_items(seg_same, true);
    // the items of FORM 2 groups go last: the second launch (launch_fused with float64) runs them
    auto split_form2 = [&](std::vector<f2::Item>& v) {
        if (plan->n_f64 == 0) return 0LL;
        auto mid = std::stable_partition(v.begin(), v.end(),
                                         [&](const f2::Item& it) { return !plan->f64_group[(size_t)it.cblock]; });
        return (long long)(v.end() - mid);
    };
    b->n_items_f64 = split_form2(items);
    b->n_items_uniform_f64 = split_form2(items_uniform);
    b->n_items = (long long)items.size();
    b->n_items_uniform = (long long)items_uniform.size();
    b->n_whole = whole / units * cblocks;  // same utterance count, in CTAs

    DeviceGuard guard(plan->device);
    // injection tables shared per ring size (f2_prep.cu): utterance u reads copy s = (-n) mod 4 from (t - n - s) mod N2
    for (int u = 0; u < n_utts; ++u) {
        f2::UttDesc& d = b->utts[(size_t)u];
        int stride = 0;
        const float* tab = d.n > 0 ? f2::injection_table(d.log2N2, &stride) : nullptr;
        if (!tab) {
            if (d.n > 0) b->private_g += 1;
            continue;
        }
        const int s = (int)((4 - (d.n & 3)) & 3);
        d.g_tab = tab + (size_t)s * (size_t)stride;
        d.g_shift = (int)(((long long)d.N2 * 2 - d.n - s) & (d.N2 - 1));
    }
    cudaError_t e = cudaSuccess;
    if (n_utts > 0) {
        e = cudaMalloc(&b->d_utts, sizeof(f2::UttDesc) * (size_t)n_utts);
        if (e == cudaSuccess)
            e = cudaMemcpy(b->d_utts, b->utts.data(), sizeof(f2::UttDesc) * (size_t)n_utts, cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess && !items.empty()) {
        e = cudaMalloc(&b->d_items, sizeof(f2::Item) * items.size());
        if (e == cudaSuccess)
            e = cudaMemcpy(b->d_items, items.data(), sizeof(f2::Item) * items.size(), cudaMemcpyHostToDevice);
        if (e == cudaSuccess && !items_uniform.empty()) {
            e = cudaMalloc(&b->d_items_uniform, sizeof(f2::Item) * items_uniform.size());
            if (e == cudaSuccess)
                e = cudaMemcpy(b->d_items_uniform, items_uniform.data(), sizeof(f2::Item) * items_uniform.size(),
                               cudaMemcpyHostToDevice);
        }
    }
    if (e != cudaSuccess) {
        if (b->d_utts) cudaFree(b->d_utts);
        if (b->d_items) cudaFree(b->d_items);
        if (b->d_items_uniform) cudaFree(b->d_items_uniform);
        delete b;
        return fail(F2_ERR_CUDA, "batch upload: %s", cudaGetErrorString(e));
    }
    *out = b;
    return F2_OK;
}

int f2_batch_destroy(f2_batch* batch) {
    if (!batch) return F2_OK;
    DeviceGuard guard(batch->plan->device);
    if (batch->d_utts) cudaFree(batch->d_utts);
    if (batch->d_items) cudaFree(batch->d_items);
    if (batch->d_items_uniform) cudaFree(batch->d_items_uniform);
    delete batch;
    return F2_OK;
}

int64_t f2_batch_total_samples(const f2_batch* b) { return b ? b->total_samples : 0; }
int64_t f2_batch_total_frames(const f2_batch* b) { return b ? b->total_frames : 0; }
int64_t f2_batch_num_items(const f2_batch* b) { return b ? b->n_items : 0; }

int f2_batch_frame_offsets(const f2_batch* b, int64_t* frame_offsets) {
    if (!b || !frame_offsets) return fail(F2_ERR_INVALID, "f2_batch_frame_offsets: bad arguments");
    for (size_t i = 0; i < b->frame_off.size(); ++i) frame_offsets[i] = b->frame_off[i];
    return F2_OK;
}

// workspace: [Z floats][xz float2][G floats][edge][edge64], each section 256-byte aligned
static size_t ws_ring_bytes(long long total_ring) { return align_up((size_t)total_ring * 4, 256); }

static size_t ws_edge_bytes(const f2_batch* b) {
    return align_up((size_t)b->n_utts * (size_t)b->plan->C * 8 * sizeof(float), 256);
}

// float64 edge residuals of the FORM 2 groups (none without such groups)
static size_t ws_edge64_bytes(const f2_batch* b) {
    return b->plan->n_f64 ? align_up((size_t)b->n_utts * (size_t)b->plan->C * 8 * sizeof(double), 256) : 0;
}

// Ring sections of the workspace: xz (two floats per ring sample) always; the two FFT scratch rings (the
// second doubles as the per-utterance injection table) only when some utterance needs them -- a batch whose
// rings are all transformed by the cluster kernel and read shared injection tables (every corpus batch)
// holds (x, xi) alone: 8 bytes per ring sample instead of 16.
static int ws_ring_units(const f2_batch* b) {
    const bool compact = f2::ring_cluster_enabled() && b->private_g == 0 && b->min_log2 >= 15 && b->max_log2 <= 17;
    return compact ? 2 : 4;
}

size_t f2_batch_workspace_bytes(const f2_batch* b, int, int) {
    if (!b) return 0;
    return (size_t)ws_ring_units(b) * ws_ring_bytes(b->total_ring) + ws_edge_bytes(b) + ws_edge64_bytes(b) + 256;
}

}  // extern "C"

namespace {
// The launch sequence f2_batch_run and f2_batch_run_cutoffs share: the Hilbert pre-pass, the edge residuals of a
// time-chunked batch and the fused kernel (float32 groups, then FORM 2 groups).  The caller has checked its
// arguments and the workspace, and filled fp's outputs and envelope settings; the rest of fp is filled here.
int run_sequence(f2_batch* b, const void* wave, int wave_dtype, bool need_env, bool gfb, f2::FusedParams fp,
                 void* workspace, void* ev_start, void* ev_stop, void* stream_) {
    f2_plan* plan = b->plan;
    DeviceGuard guard(plan->device);
    if (!guard.ok) return fail(F2_ERR_CUDA, "cannot select device %d", plan->device);
    cudaStream_t stream = (cudaStream_t)stream_;

    char* ws = (char*)align_up((size_t)workspace, 256);
    const size_t rb = ws_ring_bytes(b->total_ring);
    const int units = ws_ring_units(b);   // 2: no FFT scratch, no private injection tables (see ws_ring_units)
    float* Z = units == 4 ? (float*)ws : nullptr;
    float2* xz = (float2*)(units == 4 ? ws + rb : ws);
    float* G = units == 4 ? (float*)(ws + 3 * rb) : nullptr;
    float* edge = (float*)(ws + (size_t)units * rb);
    double* edge64 = (double*)(ws + (size_t)units * rb + ws_edge_bytes(b));

    f2::PrepParams pp;
    pp.utts = b->d_utts;
    pp.wave = wave;
    pp.wave_dtype = wave_dtype;
    pp.bufA = G;   // the table ends up where the forward transform's first scratch was
    pp.bufB = Z;
    pp.xz = xz;
    pp.G = G;
    pp.hilbert = need_env ? 1 : 0;
    f2::HostPrepInfo hp;
    hp.n_utts = b->n_utts;
    hp.min_log2N2 = b->min_log2;
    hp.max_log2N2 = b->max_log2;
    hp.private_g = b->private_g;
    F2_CUDA(f2::launch_prep(pp, hp, stream));

    fp.utts = b->d_utts;
    // the filterbank output is store-bound and uses the direct form for fewer groups: equal-length chunks
    const bool uniform_chunks = gfb && b->d_items_uniform != nullptr;
    fp.items = uniform_chunks ? b->d_items_uniform : b->d_items;
    fp.chan = plan->d_chan;
    fp.xz = xz;
    fp.G = G;
    fp.edge = nullptr;
    fp.chan64 = plan->d_chan64;
    fp.edge64 = nullptr;
    if (need_env && b->n_items > b->n_whole) {
        // time-chunked batch: the edge residuals are per utterance, compute them once instead of
        // in every chunk.  Few (utterance, channel) pairs -> chunked scan (low latency), many ->
        // one sequential thread per channel.
        const long long scan_ctas = (long long)b->n_utts * ((plan->C + 3) / 4);
        if (plan->w_edge <= f2::kScanWindow && scan_ctas <= 148 * 16)
            F2_CUDA(f2::launch_edge_scan(b->d_utts, b->n_utts, plan->d_chan, plan->d_scan_mats, plan->C, plan->c_pad, xz,
                                         edge, stream));
        else
            F2_CUDA(f2::launch_edge<0>(b->d_utts, b->n_utts, plan->d_chan, nullptr, plan->C, plan->c_pad, xz,
                                       plan->w_edge, edge, stream));
        fp.edge = edge;
        if (plan->n_f64)
            F2_CUDA(f2::launch_edge<2>(b->d_utts, b->n_utts, plan->d_chan, plan->d_chan64, plan->C, plan->c_pad, xz,
                                       plan->w_edge, edge64, stream));
    }
    fp.C = plan->C;
    fp.c_pad = plan->c_pad;
    // Direct-form threshold (measured against the float64 oracle, DESIGN.md section 3): round-off of
    // the direct form grows like 1/(1+B1+B2).  The envelope stays at the delta form's error level
    // (<= 1e-5 of the channel RMS) down to 0.035; the filterbank output itself only down to 0.25.
    fp.direct_min_cy = gfb ? kDirectMinCyGfb : kDirectMinCyEnv;
    fp.step = b->step;
    fp.phase = b->phase;
    fp.w_imag = plan->w_imag;
    fp.w_edge = plan->w_edge;
    fp.w_casc = plan->w_casc;
    if (ev_start) F2_CUDA(cudaEventRecord((cudaEvent_t)ev_start, stream));
    const long long n_items = uniform_chunks ? b->n_items_uniform : b->n_items;
    const long long n_f64 = uniform_chunks ? b->n_items_uniform_f64 : b->n_items_f64;
    F2_CUDA(f2::launch_fused(fp, (int)(n_items - n_f64), false, stream));
    if (n_f64 > 0) {
        f2::FusedParams fp64 = fp;
        fp64.items = fp.items + (n_items - n_f64);
        fp64.edge64 = fp.edge ? edge64 : nullptr;
        F2_CUDA(f2::launch_fused(fp64, (int)n_f64, true, stream));
    }
    if (ev_stop) F2_CUDA(cudaEventRecord((cudaEvent_t)ev_stop, stream));
    return F2_OK;
}

// Low-pass warm-up of a mid-signal chunk: |a1|^W < 1e-7, for either sign of the pole (a1 > 0 above 4 kHz).
// At least one tile: the output at t0 reads the one-pole state at t0 - 1 even when a1 = 0.  At most
// kMaxLowpassWarmup, past the longest utterance (2^25 samples): a warm-up that reaches t = 0 starts there, and
// t0 - w_lpf - w_casc in the fused kernel cannot overflow (cutoffs near 0 or 8000 Hz put |a1| within 1e-9 of 1).
constexpr int kMaxLowpassWarmup = 1 << 26;
int lowpass_warmup(double a1) {
    const double k = fabs(a1);
    if (!(k < 1.0)) return kMaxLowpassWarmup;
    const double w = k > 0.0 ? log(1e-7) / log(k) : 0.0;
    return w < kMaxLowpassWarmup ? std::max(round_up_tile(w), f2::kTile) : kMaxLowpassWarmup;
}
}  // namespace

extern "C" {

int f2_batch_run(f2_batch* b, const f2_run_args* a, void* workspace, size_t workspace_bytes, void* stream_) {
    if (!b || !a) return fail(F2_ERR_INVALID, "f2_batch_run: null batch/args");
    if (a->struct_size < sizeof(f2_run_args))
        return fail(F2_ERR_INVALID, "f2_batch_run: f2_run_args.struct_size is %u, this library (ABI %d) needs %zu -- "
                    "the caller was built against an older include/f2cnn_b200.h", a->struct_size, f2_abi_version(),
                    sizeof(f2_run_args));
    if (b->total_samples == 0) return F2_OK;
    if (!a->wave || a->wave_dtype < F2_I16 || a->wave_dtype > F2_F64)
        return fail(F2_ERR_INVALID, "f2_batch_run: wave pointer/dtype");
    if ((a->gfb && a->gfb_dtype != F2_F32 && a->gfb_dtype != F2_F64) ||
        (a->env && a->env_dtype != F2_F32 && a->env_dtype != F2_F64))
        return fail(F2_ERR_INVALID, "f2_batch_run: output dtype must be F2_F32 or F2_F64");
    if (a->windows) {
        if (a->gfb || a->env || a->env_t || a->dec)
            return fail(F2_ERR_INVALID, "f2_batch_run: `windows` is a stand-alone output mode (no gfb/env/env_t/dec)");
        if (!a->win_offsets || a->win_dots < 1)
            return fail(F2_ERR_INVALID, "f2_batch_run: `windows` needs win_offsets and win_dots >= 1");
    }
    const size_t need = f2_batch_workspace_bytes(b, 0, 0);
    if (!workspace || workspace_bytes < need)
        return fail(F2_ERR_WORKSPACE, "workspace %zu bytes, need %zu", workspace_bytes, need);
    double b0 = 0.0, a1 = 0.0;
    if (a->lpf) {
        if (!(a->cutoff_hz > 0.0) || !(a->cutoff_hz < 8000.0))
            return fail(F2_ERR_INVALID, "cutoff must be in (0, 8000) Hz, got %g", a->cutoff_hz);
        butter1(a->cutoff_hz, &b0, &a1);
    }
    const bool need_env = a->env_t != nullptr || a->dec != nullptr || a->windows != nullptr || a->env != nullptr;

    f2::FusedParams fp{};
    fp.env_t = a->env_t;
    // (C, n) outputs: written by the fused kernel itself through a shared-memory transpose, each in its own dtype
    fp.gfb_cn = a->gfb;
    fp.env_cn = a->env;
    fp.gfb_cn_f64 = a->gfb && a->gfb_dtype == F2_F64 ? 1 : 0;
    fp.env_cn_f64 = a->env && a->env_dtype == F2_F64 ? 1 : 0;
    fp.dec = a->dec;
    fp.win = a->windows;
    fp.win_off = reinterpret_cast<const long long*>(a->win_offsets);
    fp.win_dots = a->win_dots;
    fp.lpf = a->lpf ? 1 : 0;
    fp.lp_k = (float)(-a1);
    fp.lp_b0 = (float)b0;
    fp.w_lpf = a->lpf ? lowpass_warmup(a1) : 0;
    return run_sequence(b, a->wave, a->wave_dtype, need_env, a->gfb != nullptr, fp, workspace, a->ev_fused_start,
                        a->ev_fused_stop, stream_);
}

int f2_batch_run_cutoffs(f2_batch* b, const void* wave, int wave_dtype, const double* cutoffs_hz, int n_settings,
                         float* dec, int64_t plane_stride, void* workspace, size_t workspace_bytes, void* stream) {
    if (!b) return fail(F2_ERR_INVALID, "f2_batch_run_cutoffs: null batch");
    if (n_settings < 1 || n_settings > f2::kMaxCutoffs)
        return fail(F2_ERR_INVALID, "f2_batch_run_cutoffs: %d settings (1 .. %d)", n_settings, f2::kMaxCutoffs);
    if (!cutoffs_hz) return fail(F2_ERR_INVALID, "f2_batch_run_cutoffs: null cutoffs");
    f2::FusedParams fp{};
    fp.sw_planes = n_settings;
    double slowest = 0.0;   // a1 of the largest |a1| (the lowest cutoff or the highest): the longest warm-up
    for (int j = 0; j < n_settings; ++j) {
        const double f = cutoffs_hz[j];
        fp.sw_state[j] = -1;
        if (f == 0.0) continue;   // no low-pass
        if (!(f > 0.0) || !(f < 8000.0))
            return fail(F2_ERR_INVALID, "f2_batch_run_cutoffs: setting %d: cutoff must be 0 (no low-pass) or in (0, 8000) Hz, "
                        "got %g", j, f);
        double b0, a1;
        butter1(f, &b0, &a1);
        const int q = fp.sw_lp++;
        fp.sw_state[j] = q;
        fp.sw_k[q] = (float)(-a1);
        fp.sw_b0[q] = (float)b0;
        if (fp.sw_lp == 1 || fabs(a1) > fabs(slowest)) slowest = a1;
    }
    if (!dec) return fail(F2_ERR_INVALID, "f2_batch_run_cutoffs: null dec");
    const int64_t plane = b->total_frames * (int64_t)b->plan->C;
    if (plane_stride < plane)
        return fail(F2_ERR_INVALID, "f2_batch_run_cutoffs: plane_stride %lld < total_frames x C = %lld",
                    (long long)plane_stride, (long long)plane);
    if (b->total_samples == 0) return F2_OK;
    if (!wave || wave_dtype < F2_I16 || wave_dtype > F2_F64)
        return fail(F2_ERR_INVALID, "f2_batch_run_cutoffs: wave pointer/dtype");
    const size_t need = f2_batch_workspace_bytes(b, 0, 0);
    if (!workspace || workspace_bytes < need)
        return fail(F2_ERR_WORKSPACE, "workspace %zu bytes, need %zu", workspace_bytes, need);
    fp.dec = dec;
    fp.plane_stride = plane_stride;
    // the chunk warm-up of the slowest setting serves every setting
    fp.lpf = fp.sw_lp > 0 ? 1 : 0;
    fp.w_lpf = fp.sw_lp > 0 ? lowpass_warmup(slowest) : 0;
    return run_sequence(b, wave, wave_dtype, true, false, fp, workspace, nullptr, nullptr, stream);
}

// ---- stand-alone envelope rows ------------------------------------------------------------
namespace {
struct RowLayout {
    int lg;
    long long ring_len;
    long long rows_pad;
};
RowLayout row_layout(int64_t rows, int64_t n) {
    RowLayout r;
    r.lg = 0;
    while (((int64_t)1 << r.lg) < n) ++r.lg;
    r.ring_len = (long long)align_up((size_t)1 << r.lg, f2::kRingAlign);
    r.rows_pad = (long long)align_up((size_t)rows, 4);
    return r;
}
__global__ void rows_desc_kernel(f2::UttDesc* d, long long rows, long long rows_pad, int n, int lg,
                                 long long ring_len) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows_pad) return;
    f2::UttDesc u;
    u.wave_off = r * n;
    u.ring_off = (r < rows ? r : 0) * ring_len;
    u.full_off = r * n;
    u.dec_off = 0;
    u.n = r < rows ? n : 0;
    u.N2 = 1 << lg;
    u.n_dec = 0;
    u.log2N2 = lg;
    u.g_tab = nullptr;
    u.g_shift = 0;
    u.pad_ = 0;
    d[r] = u;
}
}  // namespace

size_t f2_envelope_rows_workspace_bytes(int64_t rows, int64_t n) {
    if (rows <= 0 || n <= 0) return 256;
    const RowLayout r = row_layout(rows, n);
    return align_up((size_t)r.rows_pad * sizeof(f2::UttDesc), 256) + 4 * ws_ring_bytes(r.ring_len * rows) + 256;
}

int f2_envelope_rows(f2_plan* plan, const void* matrix, int dtype, int64_t rows, int64_t n, int lpf,
                     double cutoff_hz, void* out, int out_dtype, void* workspace, size_t workspace_bytes,
                     void* stream_) {
    return f2_rows_op(plan, matrix, dtype, rows, n, F2_ROWS_ENVELOPE, lpf, cutoff_hz, out, out_dtype, workspace,
                      workspace_bytes, stream_);
}

int f2_rows_op(f2_plan* plan, const void* matrix, int dtype, int64_t rows, int64_t n, int op, int lpf,
               double cutoff_hz, void* out, int out_dtype, void* workspace, size_t workspace_bytes, void* stream_) {
    if (!plan || rows < 0 || n < 0 || op < F2_ROWS_ENVELOPE || op > F2_ROWS_LOWPASS || (op == F2_ROWS_LOWPASS && !lpf))
        return fail(F2_ERR_INVALID, "f2_rows_op: bad arguments (F2_ROWS_LOWPASS needs lpf = 1)");
    if (rows == 0 || n == 0) return F2_OK;
    if (!matrix || !out || dtype < F2_I16 || dtype > F2_F64 || (out_dtype != F2_F32 && out_dtype != F2_F64))
        return fail(F2_ERR_INVALID, "f2_envelope_rows: pointer/dtype");
    if (n > ((int64_t)1 << 25)) return fail(F2_ERR_UNSUPPORTED, "row length %lld > 2^25", (long long)n);
    if (rows > (1 << 24)) return fail(F2_ERR_UNSUPPORTED, "too many rows");
    const size_t need = f2_envelope_rows_workspace_bytes(rows, n);
    if (!workspace || workspace_bytes < need)
        return fail(F2_ERR_WORKSPACE, "workspace %zu bytes, need %zu", workspace_bytes, need);
    double b0 = 0.0, a1 = 0.0;
    if (lpf) {
        if (!(cutoff_hz > 0.0) || !(cutoff_hz < 8000.0))
            return fail(F2_ERR_INVALID, "cutoff must be in (0, 8000) Hz, got %g", cutoff_hz);
        butter1(cutoff_hz, &b0, &a1);
    }
    DeviceGuard guard(plan->device);
    if (!guard.ok) return fail(F2_ERR_CUDA, "cannot select device %d", plan->device);
    cudaStream_t stream = (cudaStream_t)stream_;
    const RowLayout r = row_layout(rows, n);
    char* ws = (char*)align_up((size_t)workspace, 256);
    f2::UttDesc* d_rows = (f2::UttDesc*)ws;
    ws += align_up((size_t)r.rows_pad * sizeof(f2::UttDesc), 256);
    const size_t rb = ws_ring_bytes(r.ring_len * rows);
    float* Z = (float*)ws;
    float2* xz = (float2*)(ws + rb);
    float* Z2 = (float*)(ws + 3 * rb);
    rows_desc_kernel<<<(unsigned)((r.rows_pad + 127) / 128), 128, 0, stream>>>(d_rows, rows, r.rows_pad, (int)n, r.lg,
                                                                              r.ring_len);
    F2_CUDA(cudaGetLastError());
    f2::PrepParams pp;
    pp.utts = d_rows;
    pp.wave = matrix;
    pp.wave_dtype = dtype;
    pp.bufA = Z;
    pp.bufB = Z2;
    pp.xz = xz;
    pp.G = nullptr;
    pp.hilbert = op == F2_ROWS_LOWPASS ? 0 : 1;
    f2::HostPrepInfo hp;
    hp.n_utts = (int)rows;
    hp.min_log2N2 = hp.max_log2N2 = r.lg;
    hp.private_g = 0;
    F2_CUDA(f2::launch_prep(pp, hp, stream));
    F2_CUDA(f2::launch_rows_envelope(d_rows, (int)r.rows_pad, xz, op, lpf ? 1 : 0, (float)(-a1), (float)b0, out,
                                     out_dtype, stream));
    return F2_OK;
}

// ---- CNN forward ----------------------------------------------------------------------------------
struct f2_cnn {
    int device = 0;
    int sm_count = 148;
    void* blob = nullptr;  // one allocation holding every packed parameter
    f2::CnnWeights w{};
};

namespace {
constexpr long long kCnnChunkFrames = 32768;

uint16_t bf16_rne(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);  // NaN stays NaN
    u += 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}

// Keras conv kernel HWIO [3][3][cin][cout] -> [tap][cin / 8][cout][8] bf16
void pack_conv(const float* k, int cin, int cout, uint16_t* out) {
    for (int tap = 0; tap < 9; ++tap)
        for (int p = 0; p < cin / 8; ++p)
            for (int n = 0; n < cout; ++n)
                for (int j = 0; j < 8; ++j)
                    out[(((size_t)tap * (cin / 8) + p) * cout + n) * 8 + j] = bf16_rne(k[((size_t)tap * cin + 8 * p + j) * cout + n]);
}
}  // namespace

int f2_cnn_create(int device, const float* const* arrays, int dots, int channels, f2_cnn** out) {
    if (!arrays || !out) return fail(F2_ERR_INVALID, "f2_cnn_create: null arguments");
    for (int i = 0; i < 12; ++i)
        if (!arrays[i]) return fail(F2_ERR_INVALID, "f2_cnn_create: parameter array %d is null", i);
    if (dots != 11 || channels != 128)
        return fail(F2_ERR_UNSUPPORTED, "f2_cnn_create: the tensor-core kernels are built for the configured front end "
                    "(RADIUS = 5 -> 11 dots, 128 channels), got %d x %d", dots, channels);
    int ndev = 0;
    F2_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(F2_ERR_INVALID, "device %d out of range (%d visible)", device, ndev);
    DeviceGuard guard(device);
    if (!guard.ok) return fail(F2_ERR_CUDA, "cannot select device %d", device);
    cudaDeviceProp prop;
    F2_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(F2_ERR_UNSUPPORTED, "device %d is sm_%d%d; tcgen05 needs sm_100a", device, prop.major, prop.minor);
    // the kernels' shared-memory limit is a per-device attribute: set it for the device this network lives on
    F2_CUDA(f2::configure_cnn_kernels());
    // Keras order: conv kernels HWIO + biases (Training.py:95-108), dense kernels (in, out) + biases (:111-114)
    const float *k1 = arrays[0], *b1 = arrays[1], *k2 = arrays[2], *b2 = arrays[3], *k3 = arrays[4], *b3 = arrays[5],
                *k4 = arrays[6], *b4 = arrays[7], *W5 = arrays[8], *b5 = arrays[9], *W6 = arrays[10], *b6 = arrays[11];
    const size_t n_w1 = 2 * 32 * 8, n_w2 = 9 * 4 * 32 * 8, n_w3 = 9 * 4 * 64 * 8, n_w4 = 9 * 8 * 64 * 8;
    const size_t n_w5 = (size_t)3 * 30 * 8 * 176 * 8;
    const size_t bf_total = n_w1 + n_w2 + n_w3 + n_w4 + n_w5;
    const size_t f_total = 32 + 32 + 64 + 64 + 516 + 516 * 2 + 2;
    std::vector<uint16_t> hb(bf_total, 0);
    std::vector<float> hf(f_total);
    uint16_t* w1 = hb.data();
    uint16_t* w2 = w1 + n_w1;
    uint16_t* w3 = w2 + n_w2;
    uint16_t* w4 = w3 + n_w3;
    uint16_t* w5 = w4 + n_w4;
    for (int n = 0; n < 32; ++n) {
        for (int j = 0; j < 8; ++j) w1[(size_t)n * 8 + j] = bf16_rne(k1[(size_t)j * 32 + n]);      // taps 0..7 (cin = 1)
        w1[(size_t)(32 + n) * 8] = bf16_rne(k1[(size_t)8 * 32 + n]);                                 // tap 8, then zeros
    }
    pack_conv(k2, 32, 32, w2);
    pack_conv(k3, 32, 64, w3);
    pack_conv(k4, 64, 64, w4);
    for (int pass = 0; pass < 3; ++pass)
        for (int kc = 0; kc < 30; ++kc)
            for (int p = 0; p < 8; ++p)
                for (int nn = 0; nn < 176; ++nn) {
                    const int n = pass * 176 + nn;
                    if (n >= 516) continue;
                    for (int j = 0; j < 8; ++j)
                        w5[((((size_t)pass * 30 + kc) * 8 + p) * 176 + nn) * 8 + j] = bf16_rne(W5[(size_t)(kc * 64 + 8 * p + j) * 516 + n]);
                }
    float* f = hf.data();
    memcpy(f, b1, 32 * 4);
    memcpy(f + 32, b2, 32 * 4);
    memcpy(f + 64, b3, 64 * 4);
    memcpy(f + 128, b4, 64 * 4);
    memcpy(f + 192, b5, 516 * 4);
    memcpy(f + 708, W6, 516 * 2 * 4);
    memcpy(f + 1740, b6, 2 * 4);
    f2_cnn* c = new (std::nothrow) f2_cnn();
    if (!c) return fail(F2_ERR_INVALID, "out of host memory");
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    const size_t bf_bytes = align_up(bf_total * 2, 256);
    cudaError_t e = cudaMalloc(&c->blob, bf_bytes + f_total * 4);
    if (e == cudaSuccess) e = cudaMemcpy(c->blob, hb.data(), bf_total * 2, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy((char*)c->blob + bf_bytes, hf.data(), f_total * 4, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        if (c->blob) cudaFree(c->blob);
        delete c;
        return fail(F2_ERR_CUDA, "cnn parameter upload: %s", cudaGetErrorString(e));
    }
    const uint8_t* b = (const uint8_t*)c->blob;
    c->w.w1 = b;
    c->w.w2 = c->w.w1 + n_w1 * 2;
    c->w.w3 = c->w.w2 + n_w2 * 2;
    c->w.w4 = c->w.w3 + n_w3 * 2;
    c->w.w5 = c->w.w4 + n_w4 * 2;
    const float* df = (const float*)(b + bf_bytes);
    c->w.b1 = df;
    c->w.b2 = df + 32;
    c->w.b3 = df + 64;
    c->w.b4 = df + 128;
    c->w.b5 = df + 192;
    c->w.w6 = df + 708;
    c->w.b6 = df + 1740;
    *out = c;
    return F2_OK;
}

int f2_cnn_destroy(f2_cnn* c) {
    if (!c) return F2_OK;
    DeviceGuard guard(c->device);
    if (c->blob) cudaFree(c->blob);
    delete c;
    return F2_OK;
}

size_t f2_cnn_workspace_bytes(const f2_cnn* c, int64_t n_frames) {
    if (!c || n_frames <= 0) return 256;
    return f2::cnn_workspace_bytes(std::min<long long>(n_frames, kCnnChunkFrames));
}

int f2_cnn_workspace_layout(int64_t n_frames, int64_t* chunk_frames, size_t* features_offset) {
    const long long chunk = std::max<long long>(1, std::min<long long>(n_frames, kCnnChunkFrames));
    if (chunk_frames) *chunk_frames = chunk;
    if (features_offset) *features_offset = align_up((size_t)chunk * 4 * 252 * 16, 256);
    return F2_OK;
}

namespace {
int cnn_launch(f2_cnn* c, const float* env_t, int step, const int64_t* seg_rows, const int64_t* seg_frames, int n_segs,
               int64_t total, float* scores, int* flags, void* workspace, size_t workspace_bytes, void* stream) {
    const size_t need = f2_cnn_workspace_bytes(c, total);
    if (!workspace || workspace_bytes < need) return fail(F2_ERR_WORKSPACE, "workspace %zu bytes, need %zu", workspace_bytes, need);
    DeviceGuard guard(c->device);
    if (!guard.ok) return fail(F2_ERR_CUDA, "cannot select device %d", c->device);
    static_assert(sizeof(long long) == sizeof(int64_t), "int64_t layout");
    F2_CUDA(f2::launch_cnn_forward(c->w, env_t, step, reinterpret_cast<const long long*>(seg_rows),
                                   reinterpret_cast<const long long*>(seg_frames), n_segs,
                                   std::min<long long>(total, kCnnChunkFrames), scores, flags, workspace, c->sm_count,
                                   (cudaStream_t)stream));
    return F2_OK;
}
}  // namespace

int f2_cnn_forward(f2_cnn* c, const float* env_t, int64_t n_rows, int step, int64_t i0, int64_t i1, float* scores,
                   int* flags, void* workspace, size_t workspace_bytes, void* stream) {
    if (!c) return fail(F2_ERR_INVALID, "f2_cnn_forward: null network");
    if (i1 <= i0) return F2_OK;
    // i1 + 10*step > n_rows, written so that no caller value can overflow it
    if (!env_t || !scores || !flags || step <= 0 || i0 < 0 || n_rows < 0 || i1 > n_rows - (int64_t)10 * step)
        return fail(F2_ERR_INVALID, "f2_cnn_forward: frames [%lld, %lld) x 11 dots of step %d leave the %lld envelope rows",
                    (long long)i0, (long long)i1, step, (long long)n_rows);
    const int64_t frames = i1 - i0;
    return cnn_launch(c, env_t, step, &i0, &frames, 1, frames, scores, flags, workspace, workspace_bytes, stream);
}

int f2_cnn_forward_segments(f2_cnn* c, const float* env_t, int64_t n_rows, int step, const int64_t* seg_rows,
                            const int64_t* seg_frames, int n_segs, float* scores, int* flags, void* workspace,
                            size_t workspace_bytes, void* stream) {
    if (!c) return fail(F2_ERR_INVALID, "f2_cnn_forward_segments: null network");
    if (n_segs < 0 || (n_segs > 0 && (!seg_rows || !seg_frames)))
        return fail(F2_ERR_INVALID, "f2_cnn_forward_segments: %d segments, null segment arrays", n_segs);
    int64_t total = 0;
    for (int s = 0; s < n_segs; ++s) {
        if (seg_rows[s] < 0 || seg_frames[s] < 0 || seg_frames[s] > INT64_MAX - total)
            return fail(F2_ERR_INVALID, "f2_cnn_forward_segments: segment %d has row %lld, %lld frames", s,
                        (long long)seg_rows[s], (long long)seg_frames[s]);
        total += seg_frames[s];
    }
    if (total == 0) return F2_OK;
    if (!env_t || !scores || !flags || step <= 0 || n_rows < 0)
        return fail(F2_ERR_INVALID, "f2_cnn_forward_segments: null pointer, step %d or %lld envelope rows", step,
                    (long long)n_rows);
    // frame f of segment s reads rows up to seg_rows[s] + f + 10*step: seg_rows + seg_frames + 10*step <= n_rows,
    // compared without a sum that caller values could overflow
    const int64_t last_row = n_rows - (int64_t)10 * step;   // rows a frame may start before
    for (int s = 0; s < n_segs; ++s)
        if (seg_frames[s] > 0 && (seg_frames[s] > last_row || seg_rows[s] > last_row - seg_frames[s]))
            return fail(F2_ERR_INVALID, "f2_cnn_forward_segments: segment %d, %lld frames from row %lld x 11 dots of step %d "
                        "leave the %lld envelope rows", s, (long long)seg_frames[s], (long long)seg_rows[s], step,
                        (long long)n_rows);
    return cnn_launch(c, env_t, step, seg_rows, seg_frames, n_segs, total, scores, flags, workspace, workspace_bytes, stream);
}

int f2_umma_selftest(const void* a, int a_rows, const void* b, int n, int k, int shift, int variant, float* d, int* status,
                     void* stream) {
    if (!a || !b || !d || !status || n < 16 || n > 256 || (n & 15) || k < 16 || (k & 15) || shift < 0 ||
        a_rows < shift + 128 || (a_rows & 7))
        return fail(F2_ERR_INVALID, "f2_umma_selftest: N a multiple of 16 in [16, 256], K a multiple of 16, "
                    "a_rows a multiple of 8 and >= shift + 128");
    if ((size_t)(k / 8) * ((size_t)a_rows + (size_t)n) * 16 > 200 * 1024)
        return fail(F2_ERR_UNSUPPORTED, "f2_umma_selftest: operands exceed 200 KiB of shared memory");
    F2_CUDA(f2::launch_umma_selftest(a, a_rows, b, n, k, shift, variant, d, status, (cudaStream_t)stream));
    return F2_OK;
}

int f2_upload_spans(void* dst_device, const void* src_host, const int64_t* src_off, const int64_t* dst_off,
                    const int64_t* nbytes, int64_t n_spans, void* stream) {
    if (n_spans == 0) return F2_OK;
    if (!dst_device || !src_host || !src_off || !dst_off || !nbytes || n_spans < 0)
        return fail(F2_ERR_INVALID, "f2_upload_spans: bad arguments");
    for (int64_t i = 0; i < n_spans; ++i) {
        if (nbytes[i] < 0 || src_off[i] < 0 || dst_off[i] < 0) return fail(F2_ERR_INVALID, "f2_upload_spans: span %lld is negative", (long long)i);
        if (nbytes[i] == 0) continue;
        F2_CUDA(cudaMemcpyAsync((char*)dst_device + dst_off[i], (const char*)src_host + src_off[i], (size_t)nbytes[i],
                                cudaMemcpyHostToDevice, (cudaStream_t)stream));
    }
    return F2_OK;
}

// ---- events -------------------------------------------------------------------------------
int f2_event_create(void** event) {
    if (!event) return fail(F2_ERR_INVALID, "null event pointer");
    cudaEvent_t e;
    F2_CUDA(cudaEventCreate(&e));
    *event = (void*)e;
    return F2_OK;
}
int f2_event_destroy(void* event) {
    if (event) F2_CUDA(cudaEventDestroy((cudaEvent_t)event));
    return F2_OK;
}
int f2_event_record(void* event, void* stream) {
    F2_CUDA(cudaEventRecord((cudaEvent_t)event, (cudaStream_t)stream));
    return F2_OK;
}
int f2_event_synchronize(void* event) {
    F2_CUDA(cudaEventSynchronize((cudaEvent_t)event));
    return F2_OK;
}
int f2_event_elapsed_ms(void* start, void* stop, float* ms) {
    if (!ms) return fail(F2_ERR_INVALID, "null ms pointer");
    F2_CUDA(cudaEventElapsedTime(ms, (cudaEvent_t)start, (cudaEvent_t)stop));
    return F2_OK;
}

// ---- windowing ----------------------------------------------------------------------------
int f2_gather_windows(const float* frames, int n_channels, const int64_t* base_rows, int64_t n_windows, int dots,
                      int64_t stride_rows, float* out, void* stream) {
    if (n_windows == 0) return F2_OK;
    if (!frames || !base_rows || !out || n_channels <= 0 || dots <= 0 || n_windows < 0)
        return fail(F2_ERR_INVALID, "f2_gather_windows: bad arguments");
    static_assert(sizeof(long long) == sizeof(int64_t), "int64");
    F2_CUDA(f2::launch_gather_rows(frames, (const long long*)base_rows, n_windows, dots, stride_rows, n_channels, out,
                                   (cudaStream_t)stream));
    return F2_OK;
}

int f2_gather_index(const float* src, int n_channels, const int64_t* idx, int64_t n_idx, float* out, void* stream) {
    if (n_idx == 0) return F2_OK;
    if (!src || !idx || !out || n_channels <= 0 || n_idx < 0) return fail(F2_ERR_INVALID, "f2_gather_index: bad arguments");
    F2_CUDA(f2::launch_gather_index(src, (const long long*)idx, n_idx, n_channels, out, (cudaStream_t)stream));
    return F2_OK;
}

int f2_gather_windows_cn(const void* env, int dtype, int n_channels, int64_t n, const int64_t* idx, int64_t n_idx,
                         float* out, void* stream) {
    if (n_idx == 0) return F2_OK;
    if (!env || !idx || !out || n_channels <= 0 || n <= 0 || n_idx < 0 || (dtype != F2_F32 && dtype != F2_F64))
        return fail(F2_ERR_INVALID, "f2_gather_windows_cn: bad arguments");
    F2_CUDA(f2::launch_gather_cn(env, dtype, n_channels, n, (const long long*)idx, n_idx, out, (cudaStream_t)stream));
    return F2_OK;
}

int f2_dense_frames(const float* env_t, int64_t n_rows, int n_channels, int dots, int step, int64_t i0, int64_t i1,
                    int normalize, void* out, int out_dtype, int* bad_flag, void* stream) {
    if (i1 <= i0) return F2_OK;
    if (!env_t || !out || n_channels <= 0 || dots <= 0 || step <= 0 || i0 < 0 || (normalize && !bad_flag))
        return fail(F2_ERR_INVALID, "f2_dense_frames: bad arguments");
    if (i1 + (int64_t)(dots - 1) * step > n_rows)
        return fail(F2_ERR_INVALID, "f2_dense_frames: frames up to %lld x %d dots of step %d leave the %lld rows of env_t",
                    (long long)i1, dots, step, (long long)n_rows);
    F2_CUDA(f2::launch_dense_frames(env_t, n_channels, dots, step, i0, i1, normalize, out, out_dtype, bad_flag,
                                    (cudaStream_t)stream));
    return F2_OK;
}

int f2_label_fit(const double* formant, const int64_t* first, const int32_t* center, int64_t n_items, int dots,
                 int step, double* out, void* stream) {
    if (n_items <= 0) return F2_OK;
    if (!formant || !first || !center || !out || dots < 2 || (dots & 1) == 0 || step <= 0)
        return fail(F2_ERR_INVALID, "f2_label_fit: bad arguments (dots must be odd and >= 3, step > 0)");
    static_assert(sizeof(long long) == sizeof(int64_t), "int64_t layout");
    F2_CUDA(f2::launch_label_fit(formant, reinterpret_cast<const long long*>(first), center, (long long)n_items, dots,
                                 step, out, (cudaStream_t)stream));
    return F2_OK;
}

int f2_label_accuracy(const float* scores, const int64_t* score_offsets, const int64_t* label_times,
                      const int32_t* label_classes, const int64_t* label_offsets, int n_utts, int step, int64_t* hits,
                      int64_t* counted, void* stream) {
    if (n_utts == 0) return F2_OK;
    if (n_utts < 0 || step <= 0 || !scores || !score_offsets || !label_times || !label_classes || !label_offsets ||
        !hits || !counted || ((uintptr_t)scores & 7) != 0)
        return fail(F2_ERR_INVALID, "f2_label_accuracy: bad arguments (%d utterances, step %d; every pointer non-null, "
                    "scores 8-byte aligned)", n_utts, step);
    static_assert(sizeof(long long) == sizeof(int64_t), "int64_t layout");
    F2_CUDA(f2::launch_label_accuracy(scores, reinterpret_cast<const long long*>(score_offsets),
                                      reinterpret_cast<const long long*>(label_times), label_classes,
                                      reinterpret_cast<const long long*>(label_offsets), n_utts, step,
                                      reinterpret_cast<long long*>(hits), reinterpret_cast<long long*>(counted),
                                      (cudaStream_t)stream));
    return F2_OK;
}

}  // extern "C"
