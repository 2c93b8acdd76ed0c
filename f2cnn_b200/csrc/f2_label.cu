// f2_label.cu -- the numeric core of label generation (SURVEY.md section 8f, rank 2).
//
// Replaces, for every kept timepoint of every utterance, the body of the reference's step loop
//   scripts/processing/LabelDataGenerator.py:60-68
//     x = [step + (k - RADIUS)*STEP for k in range(DOTSPERINPUT)]
//     [a, b] = numpy.linalg.lstsq([x, 1], FormantValues)            (least-squares line)
//     r, p   = scipy.stats.pearsonr(FormantValues, a*x + b)         (p-value of the slope)
// where FormantValues are the 2*RADIUS+1 formant frames around the timepoint
// (FBFileReader.py:66-89).  The reference spends its time here (one SVD and one scipy call per
// timepoint, 1.3 M timepoints for the TIMIT-TRAIN-sized corpus); the arithmetic is 11-point sums
// and one incomplete beta function, so the whole corpus is ONE launch with one thread per
// timepoint, in float64 (the CSV keeps 5 decimals of slope and p).
//
// Closed forms used (equal to the library calls up to float64 round-off):
//   a = Sxv/Sxx, b = mean(v) - a*mean(x)             with centred sums Sxx, Sxv, Svv
//   r = corr(v, a*x+b) = |Sxv| / sqrt(Sxx*Svv)        (the fitted line has the sign of a)
//   p = 2*sf(|r|) of the beta(n/2-1, n/2-1) distribution on (-1,1)
//     = 2 * I_{(1-|r|)/2}(n/2-1, n/2-1)              (scipy/stats/_stats_py.py pearsonr)
// Constant FormantValues (Svv == 0): r = p = NaN like scipy's ConstantInputWarning path; the
// caller then drops the row because `p < RISK` is false (LabelDataGenerator.py:74).
#include "f2_label.cuh"

#include <math.h>

namespace f2 {

// Regularised incomplete beta I_x(a, b) for 0 <= x <= (a+1)/(a+b+2), by the continued fraction
// of the incomplete beta function evaluated with the modified Lentz recurrence.
__device__ double inc_beta(double a, double b, double x) {
    if (!(x > 0.0)) return 0.0;
    const double tiny = 1e-300, eps = 1e-16;
    const double qab = a + b, qap = a + 1.0, qam = a - 1.0;
    double c = 1.0;
    double d = 1.0 - qab * x / qap;
    if (fabs(d) < tiny) d = tiny;
    d = 1.0 / d;
    double h = d;
    for (int m = 1; m <= 300; ++m) {
        const double m2 = 2.0 * m;
        double aa = m * (b - m) * x / ((qam + m2) * (a + m2));
        d = 1.0 + aa * d;
        if (fabs(d) < tiny) d = tiny;
        c = 1.0 + aa / c;
        if (fabs(c) < tiny) c = tiny;
        d = 1.0 / d;
        h *= d * c;
        aa = -(a + m) * (qab + m) * x / ((a + m2) * (qap + m2));
        d = 1.0 + aa * d;
        if (fabs(d) < tiny) d = tiny;
        c = 1.0 + aa / c;
        if (fabs(c) < tiny) c = tiny;
        d = 1.0 / d;
        const double del = d * c;
        h *= del;
        if (fabs(del - 1.0) < eps) break;
    }
    const double front = exp(lgamma(qab) - lgamma(a) - lgamma(b) + a * log(x) + b * log1p(-x));
    return front * h / a;
}

__global__ void __launch_bounds__(128) label_fit_kernel(const double* __restrict__ formant,
                                                        const long long* __restrict__ first,
                                                        const int* __restrict__ center, long long n_items, int dots,
                                                        int step, double* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_items) return;
    const double* v = formant + first[i];
    const int radius = (dots - 1) / 2;
    const double x0 = (double)center[i] - (double)radius * step;
    double sv = 0.0;
    for (int k = 0; k < dots; ++k) sv += v[k];
    const double mv = sv / dots;
    const double mx = x0 + 0.5 * (dots - 1) * step;  // x is an arithmetic progression
    double sxx = 0.0, svv = 0.0, sdv = 0.0;
    bool constant = true;
    for (int k = 0; k < dots; ++k) {
        const double dx = (x0 + (double)k * step) - mx;
        const double dv = v[k] - mv;
        sxx += dx * dx;
        svv += dv * dv;
        sdv += dv;
        constant = constant && (v[k] == v[0]);
    }
    // mv is the mean rounded to float64: on a track whose spread is a few ulps of its level (one value 1 ulp
    // off a constant) the deviations from it are off by as much as they are wide.  The corrected two-pass sum
    // removes that from svv.  sxv pairs the abscissae +-j*step around the centre, so it takes no mean at all and
    // is exactly 0 on a track symmetric about its centre (slope 0: r = p = NaN, as lstsq + pearsonr give).
    svv -= sdv * sdv / dots;
    double sxv = 0.0;
    for (int j = 1; j <= radius; ++j) sxv += (double)j * step * (v[radius + j] - v[radius - j]);
    const double a = sxv / sxx;
    const double b = mv - a * mx;
    double r, p;
    if (constant || !(svv > 0.0)) {
        r = p = nan("");
    } else {
        r = fabs(sxv) / sqrt(sxx * svv);
        if (r > 1.0) r = 1.0;
        if (a == 0.0) {
            r = p = nan("");  // the fitted line is constant: correlation undefined
        } else if (dots == 2) {
            r = 1.0;
            p = 1.0;
        } else {
            const double ab = 0.5 * dots - 1.0;
            p = 2.0 * inc_beta(ab, ab, 0.5 * (1.0 - r));
            if (p > 1.0) p = 1.0;
        }
    }
    double4 o;
    o.x = a;
    o.y = b;
    o.z = r;
    o.w = p;
    reinterpret_cast<double4*>(out)[i] = o;
}

cudaError_t launch_label_fit(const double* formant, const long long* first, const int* center, long long n_items,
                             int dots, int step, double* out, cudaStream_t stream) {
    if (n_items <= 0) return cudaSuccess;
    const long long blocks = (n_items + 127) / 128;
    label_fit_kernel<<<(unsigned)blocks, 128, 0, stream>>>(formant, first, center, n_items, dots, step, out);
    return cudaGetLastError();
}

// Label accuracy of `cnn eval*` (scripts/CNN/Evaluating.py:87-110, Evaluating._label_accuracy) for every frame of
// many utterances.  Frame i of utterance u (utterance-local, compared with the label times in samples as the
// reference does) decides 1 when s[1] > s[0] (equal scores and NaN decide 0).  The reference scores it against the
// label pair t_j < i < t_{j+1} whose nearer end is closer than `step`, ties going to the earlier label.  With times
// non-decreasing the open intervals are disjoint, so the one pair the reference's loop can find is j = (number of
// times < i) - 1, found by binary search; duplicate times give an empty interval there as well.
//
// The frame count lives on the device (score_offsets[n_utts]), so the grid strides over it.  A warp's lanes hold
// consecutive frames: lanes of one utterance (__match_any_sync) add their ballots with one 64-bit atomic each, and
// integer sums in any order are exact.
__global__ void __launch_bounds__(256) label_accuracy_kernel(const float2* __restrict__ scores,
                                                             const long long* __restrict__ score_offsets,
                                                             const long long* __restrict__ times,
                                                             const int* __restrict__ classes,
                                                             const long long* __restrict__ label_offsets, int n_utts,
                                                             int step, unsigned long long* __restrict__ hits,
                                                             unsigned long long* __restrict__ counted) {
    const int lane = threadIdx.x & 31;
    const long long first = score_offsets[0], end = score_offsets[n_utts];
    const long long stride = (long long)gridDim.x * blockDim.x;
    // the loop test is on the warp's first frame, so whole warps run every iteration (the shuffles need all lanes)
    for (long long f = first + (long long)blockIdx.x * blockDim.x + threadIdx.x; f - lane < end; f += stride) {
        int u = -1;
        bool count = false, hit = false;
        if (f < end) {
            // utterance: the last u < n_utts with score_offsets[u] <= f (zero-frame utterances are passed over)
            int lo = 0, hi = n_utts - 1;
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (score_offsets[mid] <= f) lo = mid; else hi = mid - 1;
            }
            u = lo;
            const long long i = f - score_offsets[u];
            const long long l0 = label_offsets[u], l1 = label_offsets[u + 1];
            // first label at or after i: [l0, a) holds the times < i
            long long a = l0, b = l1;
            while (a < b) {
                const long long mid = a + ((b - a) >> 1);
                if (times[mid] < i) a = mid + 1; else b = mid;
            }
            if (a > l0 && a < l1 && times[a] > i) {
                // the distances are positive and below 2^64 for any int64 times: exact in unsigned arithmetic
                const unsigned long long d_lo = (unsigned long long)i - (unsigned long long)times[a - 1];
                const unsigned long long d_hi = (unsigned long long)times[a] - (unsigned long long)i;
                if (d_lo < (unsigned long long)step || d_hi < (unsigned long long)step) {
                    const int target = d_lo <= d_hi ? classes[a - 1] : classes[a];
                    const float2 s = scores[f];
                    count = true;
                    hit = (s.y > s.x ? 1 : 0) == target;
                }
            }
        }
        const unsigned same = __match_any_sync(0xffffffffu, u);
        const unsigned n_count = __popc(__ballot_sync(0xffffffffu, count) & same);
        const unsigned n_hit = __popc(__ballot_sync(0xffffffffu, hit) & same);
        if (u >= 0 && n_count != 0 && lane == __ffs(same) - 1) {
            atomicAdd(counted + u, (unsigned long long)n_count);
            if (n_hit != 0) atomicAdd(hits + u, (unsigned long long)n_hit);
        }
    }
}

cudaError_t launch_label_accuracy(const float* scores, const long long* score_offsets, const long long* times,
                                  const int* classes, const long long* label_offsets, int n_utts, int step,
                                  long long* hits, long long* counted, cudaStream_t stream) {
    if (n_utts <= 0) return cudaSuccess;
    cudaError_t e = cudaMemsetAsync(hits, 0, sizeof(long long) * (size_t)n_utts, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(counted, 0, sizeof(long long) * (size_t)n_utts, stream);
    if (e != cudaSuccess) return e;
    int device = 0, sms = 0;
    if ((e = cudaGetDevice(&device)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device)) != cudaSuccess) return e;
    // eight 256-thread CTAs fill an SM; the grid strides over frame counts it does not know on the host
    label_accuracy_kernel<<<(unsigned)sms * 8, 256, 0, stream>>>(
        reinterpret_cast<const float2*>(scores), score_offsets, times, classes, label_offsets, n_utts, step,
        reinterpret_cast<unsigned long long*>(hits), reinterpret_cast<unsigned long long*>(counted));
    return cudaGetLastError();
}

}  // namespace f2
