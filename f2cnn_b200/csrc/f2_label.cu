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

}  // namespace f2
