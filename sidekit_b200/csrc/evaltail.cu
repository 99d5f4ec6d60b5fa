// Evaluation tail of the verification pipeline (SURVEY.md 8f rank 2): PAV / ROC convex hull / EER on the host and the
// z-/t-norm statistics on the device.
//
// The reference does all of this in Python + numpy: `pavx` is a Python loop over every trial, `rocch` re-sums the
// whole label vector once per hull vertex (sidekit/bosaris/detplot.py:289-347, :391-441) and `eer` is a hand-rolled
// search (sidekit/nnet/xvector.py:101-209).  Here the sequential parts are native C++ with the SAME floating-point
// operations in the same order (the pooled means decide which bins merge, so the arithmetic must match bit for bit;
// this file is compiled without FMA contraction on the host), and the per-row / per-column statistics of
// znorm / tnorm (sidekit/score_normalization.py:44-95) are CUDA kernels over the device-resident score matrix.
#include "sidekit_b200.h"
#include "common.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <numeric>
#include <vector>

namespace skb {

// ----------------------------------------------------------------------------- PAV
// detplot.py:289-347.  Returns the number of bins.  `ghat` reproduces the reference's output INCLUDING its quirk: the
// final fill loop starts at index 0 for the first bin and, through Python's negative indexing, overwrites the LAST
// element with the first bin's height.
static int64_t pav(const double* y, int64_t n, double* ghat, int64_t* width, double* height) {
    std::vector<int64_t> index(n), length(n);
    int64_t ci = 0;
    index[0] = 0;
    length[0] = 1;
    ghat[0] = y[0];
    for (int64_t j = 1; j < n; ++j) {
        ++ci;
        index[ci] = j + 1;
        length[ci] = 1;
        ghat[ci] = y[j];
        while (ci >= 1 && ghat[ci - 1] >= ghat[ci]) {
            const int64_t nw = length[ci - 1] + length[ci];
            const double frac = (double)length[ci] / (double)nw;
            const double diff = ghat[ci] - ghat[ci - 1];
            const double prod = frac * diff;                 // kept as separate statements: no fused multiply-add
            ghat[ci - 1] = ghat[ci - 1] + prod;
            length[ci - 1] = nw;
            --ci;
        }
    }
    const int64_t n_bins = ci + 1;
    for (int64_t i = 0; i < n_bins; ++i) { height[i] = ghat[i]; width[i] = length[i]; }
    int64_t m = n;
    while (m >= 0 && ci >= 0) {
        const double v = ghat[ci];
        for (int64_t j = index[ci]; j <= m; ++j) ghat[j == 0 ? n - 1 : j - 1] = v;   // j == 0: ghat[-1] in the reference
        m = index[ci] - 1;
        --ci;
    }
    return n_bins;
}

// ----------------------------------------------------------------------------- z-/t-norm statistics on the device
// axis 1: one warp per row (mean(1), std(1) of numpy: population std); axis 0: one thread per column.
// sym (znorm(sym=True), score_normalization.py:63-66): the diagonal is excluded, the divisor is N-1 and the second
// statistic is the VARIANCE, not its square root (as in the reference).
template <typename T>
__global__ void stats_rows_kernel(const T* __restrict__ S, int M, int N, long long ld, int sym, double* __restrict__ mean,
                                  double* __restrict__ sd) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= M) return;
    const T* r = S + (size_t)row * ld;
    double s = 0.0;
    for (int j = lane; j < N; j += 32) s += (double)r[j];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const double diag = (sym && row < N) ? (double)r[row] : 0.0;
    const double mu = sym ? (s - diag) / (double)(N - 1) : s / (double)N;
    double v = 0.0;
    for (int j = lane; j < N; j += 32) {
        const double d = (double)r[j] - mu;
        v += d * d;
    }
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) {
        mean[row] = mu;
        if (!sym) sd[row] = sqrt(v / (double)N);          // sym: second pass below (it needs every row's mean)
    }
}

// znorm(sym=True), score_normalization.py:64-66: `numpy.square(scoremat - mean_per_model)` broadcasts the per-model
// means against the LAST axis, so element (i, j) is centred with the mean of model j; the row sums of that, minus the
// diagonal term, divided by N - 1, are what the reference then divides by (a variance, not a standard deviation).
template <typename T>
__global__ void sym_var_kernel(const T* __restrict__ S, int M, int N, long long ld, const double* __restrict__ mean, double* __restrict__ sd) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= M) return;
    const T* r = S + (size_t)row * ld;
    double v = 0.0;
    for (int j = lane; j < N; j += 32) {
        const double d = (double)r[j] - mean[j];
        v += d * d;
    }
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) {
        const double dd = (double)r[row] - mean[row];
        sd[row] = (v - dd * dd) / (double)(N - 1);
    }
}

template <typename T>
__global__ void stats_cols_kernel(const T* __restrict__ S, int M, int N, long long ld, double* __restrict__ mean, double* __restrict__ sd) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= N) return;
    double s = 0.0;
    for (int i = 0; i < M; ++i) s += (double)S[(size_t)i * ld + col];
    const double mu = s / (double)M;
    double v = 0.0;
    for (int i = 0; i < M; ++i) {
        const double d = (double)S[(size_t)i * ld + col] - mu;
        v += d * d;
    }
    mean[col] = mu;
    sd[col] = sqrt(v / (double)M);
}

// out[i][j] = (S[i][j] - sub[j]) / div[j]: numpy broadcasting of an (N,) vector against the LAST axis -- which is what
// both `scoremat - mean_per_segment` (tnorm) and `scoremat - mean_per_model` (znorm: needs a square matrix) do.
template <typename T>
__global__ void normalise_kernel(const T* __restrict__ S, int M, int N, long long ld, const double* __restrict__ sub,
                                 const double* __restrict__ div, T* __restrict__ out, long long ld_out) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)M * N) return;
    const int i = (int)(idx / N), j = (int)(idx - (long long)i * N);
    out[(size_t)i * ld_out + j] = (T)(((double)S[(size_t)i * ld + j] - sub[j]) / div[j]);
}

}  // namespace skb

using namespace skb;

extern "C" {

int skb_pavx(const double* y, int64_t n, double* ghat, int64_t* width, double* height, int64_t* n_bins) {
    if (!y || !ghat || !width || !height || !n_bins || n <= 0) {
        set_last_error(__FILE__, __LINE__, "pavx: input array is empty or a pointer is NULL");
        return SKB_ERR_ARG;
    }
    *n_bins = pav(y, n, ghat, width, height);
    return SKB_OK;
}

int skb_rocch(const double* tar, int64_t n_tar, const double* non, int64_t n_non, double* pmiss, double* pfa, int64_t* n_points) {
    if (!tar || !non || !pmiss || !pfa || !n_points || n_tar <= 0 || n_non <= 0) {
        set_last_error(__FILE__, __LINE__, "rocch: need at least one target and one non-target score");
        return SKB_ERR_ARG;
    }
    const int64_t N = n_tar + n_non;
    // stable ascending order of the concatenated scores (targets first): equal scores are NOT swapped (detplot.py:412-415)
    std::vector<int64_t> order(N);
    std::iota(order.begin(), order.end(), (int64_t)0);
    auto score = [&](int64_t i) { return i < n_tar ? tar[i] : non[i - n_tar]; };
    std::stable_sort(order.begin(), order.end(), [&](int64_t a, int64_t b) { return score(a) < score(b); });
    std::vector<double> ideal(N), ghat(N), height(N);
    std::vector<int64_t> width(N);
    for (int64_t i = 0; i < N; ++i) ideal[i] = order[i] < n_tar ? 1.0 : 0.0;
    const int64_t nbins = pav(ideal.data(), N, ghat.data(), width.data(), height.data());
    // running counts instead of the reference's per-vertex re-summation: the counts are integers, so the quotients are
    // the same doubles
    std::vector<int64_t> tar_prefix(N + 1, 0);
    for (int64_t i = 0; i < N; ++i) tar_prefix[i + 1] = tar_prefix[i] + (order[i] < n_tar ? 1 : 0);
    int64_t left = 0, fa = n_non, miss = 0;
    for (int64_t i = 0; i < nbins; ++i) {
        pmiss[i] = (double)miss / (double)n_tar;
        pfa[i] = (double)fa / (double)n_non;
        left += width[i];
        miss = tar_prefix[left];
        fa = N - left - (tar_prefix[N] - tar_prefix[left]);
    }
    pmiss[nbins] = (double)miss / (double)n_tar;
    pfa[nbins] = (double)fa / (double)n_non;
    *n_points = nbins + 1;
    return SKB_OK;
}

// sidekit/nnet/xvector.py:101-209.  Indices that the reference would read out of range (an IndexError there) are
// reported as SKB_ERR_ARG; negative indices wrap like Python's.
int skb_eer(const double* negatives, int64_t n_neg, const double* positives, int64_t n_pos, double* eer_out) {
    if (!negatives || !positives || !eer_out || n_neg <= 0 || n_pos <= 0) {
        set_last_error(__FILE__, __LINE__, "eer: empty score arrays");
        return SKB_ERR_ARG;
    }
    std::vector<double> pos(positives, positives + n_pos), neg(negatives, negatives + n_neg);
    std::sort(pos.begin(), pos.end());
    std::sort(neg.begin(), neg.end(), [](double a, double b) { return a > b; });
    bool oob = false;
    auto P = [&](int64_t i) { if (i < 0) i += n_pos; if (i < 0 || i >= n_pos) { oob = true; return 0.0; } return pos[i]; };
    auto Q = [&](int64_t i) { if (i < 0) i += n_neg; if (i < 0 || i >= n_neg) { oob = true; return 0.0; } return neg[i]; };
#define SKB_EER_OOB()                                                                                  \
    if (oob) { set_last_error(__FILE__, __LINE__, "eer: index out of range (the reference raises IndexError here)"); return SKB_ERR_ARG; }
    double p_score = pos[0], n_score = neg[0];
    int64_t pi = 0, ni = 0, pjump = n_pos / 2, njump = n_neg / 2;
    // bisection on both sorted lists at once
    for (;;) {
        if (pi < 0 || ni < 0) { *eer_out = 0.0; return SKB_OK; }
        if (pi > n_pos || ni > n_neg) { *eer_out = 100.0; return SKB_OK; }
        if (p_score < n_score) {
            pi += pjump; ni += njump;
            if (pjump == 0 && njump == 0) break;
        } else if (p_score >= n_score) {
            pi -= pjump; ni -= njump;
            if (pjump == 0 && njump == 0) break;
        }
        p_score = P(pi); n_score = Q(ni);
        SKB_EER_OOB();
        pjump /= 2; njump /= 2;
    }
    double best_gap = 100.0, eer = 0.0;
    double tfr = (double)(pi < 0 ? -pi : pi) / (double)n_pos;
    double tfa = (double)(1 + (ni < 0 ? -ni : ni)) / (double)n_neg;
    if (p_score == n_score && tfr == tfa) { *eer_out = tfr; return SKB_OK; }
    // walk to the crossing point
    while (P(pi) < Q(ni)) {
        SKB_EER_OOB();
        if (pi < n_pos - 1) ++pi;
        else if (ni < n_neg - 1) ++ni;
        else break;
    }
    SKB_EER_OOB();
    while (P(pi) > Q(ni) && ni >= 1) --ni;
    SKB_EER_OOB();
    tfr = (double)(1 + pi) / (double)n_pos;
    tfa = (double)(1 + ni) / (double)n_neg;
    while (tfa > tfr) {
        ++pi;
        while (P(pi) > Q(ni) && ni >= 1) --ni;
        SKB_EER_OOB();
        tfr = (double)(1 + pi) / (double)n_pos;
        tfa = (double)(1 + ni) / (double)n_neg;
    }
    // refine: keep the candidate with the smallest |FR - FA|
    if (std::fabs(tfr - tfa) <= best_gap) { best_gap = std::fabs(tfr - tfa); eer = (tfr + tfa) / 2; }
    else { *eer_out = best_gap; return SKB_OK; }
    tfr = (double)pi / (double)n_pos;
    tfa = (double)(1 + ni) / (double)n_neg;
    if (std::fabs(tfr - tfa) <= best_gap) { best_gap = std::fabs(tfr - tfa); eer = (tfr + tfa) / 2; }
    else { *eer_out = eer; return SKB_OK; }
    for (;;) {
        while (Q(ni + 1) <= P(pi - 1)) {
            SKB_EER_OOB();
            --pi;
            tfr = (double)pi / (double)n_pos;
            tfa = (double)(1 + ni) / (double)n_neg;
            if (std::fabs(tfr - tfa) <= best_gap) { best_gap = std::fabs(tfr - tfa); eer = (tfr + tfa) / 2; }
            else { *eer_out = eer; return SKB_OK; }
        }
        SKB_EER_OOB();
        while (Q(ni + 1) > P(pi - 1)) {
            SKB_EER_OOB();
            ++ni;
            tfr = (double)pi / (double)n_pos;
            tfa = (double)(1 + ni) / (double)n_neg;
            if (std::fabs(tfr - tfa) <= best_gap) { best_gap = std::fabs(tfr - tfa); eer = (tfr + tfa) / 2; }
            else { *eer_out = eer; return SKB_OK; }
        }
        SKB_EER_OOB();
    }
#undef SKB_EER_OOB
}

int skb_scoremat_stats(const void* S_dev, int M, int N, int64_t ld, int is_f64, int axis, int sym, double* mean_dev, double* std_dev,
                       void* stream) {
    if (!S_dev || !mean_dev || !std_dev || M <= 0 || N <= 0 || ld < N || (axis != 0 && axis != 1) || (sym && (axis != 1 || N < 2 || M != N))) {
        set_last_error(__FILE__, __LINE__, "scoremat_stats: bad arguments");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const double* S64 = (const double*)S_dev;
    const float* S32 = (const float*)S_dev;
    if (axis == 1) {
        if (is_f64) SKB_CUDA_CHECK(launch_kernel(false, stats_rows_kernel<double>, (M + 7) / 8, 256, 0, st, S64, M, N, ld, sym, mean_dev, std_dev));
        else SKB_CUDA_CHECK(launch_kernel(false, stats_rows_kernel<float>, (M + 7) / 8, 256, 0, st, S32, M, N, ld, sym, mean_dev, std_dev));
        if (sym) {
            if (is_f64) SKB_CUDA_CHECK(launch_kernel(false, sym_var_kernel<double>, (M + 7) / 8, 256, 0, st, S64, M, N, ld, mean_dev, std_dev));
            else SKB_CUDA_CHECK(launch_kernel(false, sym_var_kernel<float>, (M + 7) / 8, 256, 0, st, S32, M, N, ld, mean_dev, std_dev));
        }
    } else {
        if (is_f64) SKB_CUDA_CHECK(launch_kernel(false, stats_cols_kernel<double>, (N + 127) / 128, 128, 0, st, S64, M, N, ld, mean_dev, std_dev));
        else SKB_CUDA_CHECK(launch_kernel(false, stats_cols_kernel<float>, (N + 127) / 128, 128, 0, st, S32, M, N, ld, mean_dev, std_dev));
    }
    return SKB_OK;
}

int skb_scoremat_normalise(const void* S_dev, int M, int N, int64_t ld, int is_f64, const double* sub_dev, const double* div_dev,
                           void* out_dev, int64_t ld_out, void* stream) {
    if (!S_dev || !sub_dev || !div_dev || !out_dev || M <= 0 || N <= 0 || ld < N || ld_out < N) {
        set_last_error(__FILE__, __LINE__, "scoremat_normalise: bad arguments");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const long long total = (long long)M * N;
    const unsigned blocks = (unsigned)((total + 255) / 256);
    if (is_f64)
        SKB_CUDA_CHECK(launch_kernel(false, normalise_kernel<double>, blocks, 256, 0, st, (const double*)S_dev, M, N, ld, sub_dev, div_dev,
                                     (double*)out_dev, ld_out));
    else
        SKB_CUDA_CHECK(launch_kernel(false, normalise_kernel<float>, blocks, 256, 0, st, (const float*)S_dev, M, N, ld, sub_dev, div_dev,
                                     (float*)out_dev, ld_out));
    return SKB_OK;
}

}  // extern "C"
