// PLDA training on the device (SURVEY.md 8f rank 3): the EM loop of FactorAnalyser.plda
// (sidekit/factor_analyser.py:830-932, per-class E-step of fa_model_loop :166-205) as a handful of float64 kernels per
// iteration with NO host round trip inside the loop.
//
// The reference whitens the class statistics and the eigenvoice matrix with sqrt(Sigma)^-1 (an eigendecomposition per
// iteration, statserver.py:852-884), loops over the classes in Python and un-whitens again.  Every quantity of the E-
// and M-step only depends on the whitening W through W W' = Sigma^-1:
//     F_w' F_w = F' Sigma^-1 F,   aux_i = (s_i - n_i mu)' Sigma^-1 F,   C = E[h]' (S - n mu')        (W cancels)
// so the loop below never whitens: one Cholesky factorisation of Sigma (D x D) and of (n A0 + I) per distinct session
// count n (R x R, batched over the counts -- the reference inverts one matrix per CLASS), GEMMs over all classes at once,
// and Cholesky solves for the M-step.  Agreement with the reference's (mean, F, Sigma): 1e-9 after 5 iterations
// (tests/test_plda_training.py against tests/golden/plda_training.npz).
// All matrices are row-major float64; sizes are a few hundred, so the kernels are simple and latency-oriented.
#include "sidekit_b200.h"
#include "common.cuh"
#include "class_sum.cuh"

#include <vector>

namespace skb {

// C[M][N] = alpha * op(A) op(B) + beta * C, op = identity or transpose; 16 x 16 tiles through shared memory
__global__ void __launch_bounds__(256) dgemm_kernel(int ta, int tb, int M, int N, int K, double alpha, const double* __restrict__ A, int lda,
                                                    const double* __restrict__ B, int ldb, double beta, double* __restrict__ C, int ldc) {
    __shared__ double As[16][17], Bs[16][17];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int m = blockIdx.y * 16 + ty, n = blockIdx.x * 16 + tx;
    double acc = 0.0;
    for (int k0 = 0; k0 < K; k0 += 16) {
        const int ka = k0 + tx, am = blockIdx.y * 16 + ty;
        As[ty][tx] = (am < M && ka < K) ? (ta ? A[(size_t)ka * lda + am] : A[(size_t)am * lda + ka]) : 0.0;
        const int kb = k0 + ty, bn = blockIdx.x * 16 + tx;
        Bs[ty][tx] = (kb < K && bn < N) ? (tb ? B[(size_t)bn * ldb + kb] : B[(size_t)kb * ldb + bn]) : 0.0;
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 16; ++k) acc = fma(As[ty][k], Bs[k][tx], acc);
        __syncthreads();
    }
    if (m < M && n < N) C[(size_t)m * ldc + n] = alpha * acc + (beta != 0.0 ? beta * C[(size_t)m * ldc + n] : 0.0);
}

static int dgemm(int ta, int tb, int M, int N, int K, double alpha, const double* A, int lda, const double* B, int ldb, double beta,
                 double* C, int ldc, cudaStream_t st) {
    SKB_CUDA_CHECK(launch_kernel(false, dgemm_kernel, dim3((N + 15) / 16, (M + 15) / 16), 256, 0, st, ta, tb, M, N, K, alpha, A, lda, B, ldb,
                                 beta, C, ldc));
    return SKB_OK;
}

// In-place lower Cholesky factor of `batch` SPD matrices (n x n, row-major, leading dimension n): one CTA each, right-looking.
// The strictly upper triangle is left untouched.  A non-positive pivot sets *flag.
__global__ void __launch_bounds__(1024) dpotrf_kernel(double* __restrict__ A, int n, int* __restrict__ flag) {
    double* a = A + (size_t)blockIdx.x * n * n;
    __shared__ double piv;
    for (int j = 0; j < n; ++j) {
        if (threadIdx.x == 0) {
            const double d = a[(size_t)j * n + j];
            if (!(d > 0.0)) *flag = 1;
            piv = sqrt(d);
            a[(size_t)j * n + j] = piv;
        }
        __syncthreads();
        const double inv = 1.0 / piv;
        for (int i = j + 1 + threadIdx.x; i < n; i += blockDim.x) a[(size_t)i * n + j] *= inv;
        __syncthreads();
        // trailing update of the lower triangle: a[i][k] -= a[i][j] * a[k][j], j < k <= i
        const int rem = n - j - 1;
        for (int idx = threadIdx.x; idx < rem * rem; idx += blockDim.x) {
            const int i = j + 1 + idx / rem, k = j + 1 + idx % rem;
            if (k <= i) a[(size_t)i * n + k] -= a[(size_t)i * n + j] * a[(size_t)k * n + j];
        }
        __syncthreads();
    }
}

// Solve L L' X = B in place for `batch` systems: L (n x n lower, row-major), B (n x nrhs, row-major).  One thread per
// right-hand-side column (the columns are independent; a row of B is contiguous, so the warp's accesses coalesce and the
// L element is a broadcast).
__global__ void dpotrs_kernel(const double* __restrict__ L, int n, double* __restrict__ B, int nrhs, long long strideL, long long strideB) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nrhs) return;
    const double* l = L + (size_t)blockIdx.y * strideL;
    double* b = B + (size_t)blockIdx.y * strideB;
    for (int i = 0; i < n; ++i) {                       // forward: L y = b
        double s = b[(size_t)i * nrhs + c];
        for (int k = 0; k < i; ++k) s -= l[(size_t)i * n + k] * b[(size_t)k * nrhs + c];
        b[(size_t)i * nrhs + c] = s / l[(size_t)i * n + i];
    }
    for (int i = n - 1; i >= 0; --i) {                  // backward: L' x = y
        double s = b[(size_t)i * nrhs + c];
        for (int k = i + 1; k < n; ++k) s -= l[(size_t)k * n + i] * b[(size_t)k * nrhs + c];
        b[(size_t)i * nrhs + c] = s / l[(size_t)i * n + i];
    }
}

__global__ void colmean_kernel(const double* __restrict__ X, int N, int D, double* __restrict__ mean) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= D) return;
    double s = 0.0;
    for (int i = 0; i < N; ++i) s += X[(size_t)i * D + d];
    mean[d] = s / N;
}

// out[i][d] = X[i][d] - w[i] * mu[d]   (w == nullptr: weight 1)
__global__ void center_rows_kernel(const double* __restrict__ X, const double* __restrict__ w, const double* __restrict__ mu, long long n, int D,
                                   double* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = X[i] - (w ? w[i / D] : 1.0) * mu[i % D];
}

// M[u] = n_u * A0 + I  (R x R each)
__global__ void lambda_kernel(const double* __restrict__ A0, const double* __restrict__ uniq_n, int R, int U, double* __restrict__ M) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)U * R * R) return;
    const int u = (int)(i / ((long long)R * R)), rc = (int)(i % ((long long)R * R));
    M[i] = uniq_n[u] * A0[rc] + ((rc / R) == (rc % R) ? 1.0 : 0.0);
}

__global__ void identity_kernel(double* __restrict__ M, int R, int U) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)U * R * R) return;
    const int rc = (int)(i % ((long long)R * R));
    M[i] = (rc / R) == (rc % R) ? 1.0 : 0.0;
}

// e_h[i] = aux[i] . Linv[u_i]   (Linv symmetric);  e_hn[i] = n_i * e_h[i].  One CTA per class.
__global__ void __launch_bounds__(128) posterior_mean_kernel(const double* __restrict__ aux, const double* __restrict__ Linv,
                                                             const int* __restrict__ cls_u, const double* __restrict__ cls_n, int R,
                                                             double* __restrict__ e_h, double* __restrict__ e_hn) {
    extern __shared__ double a[];
    const int i = blockIdx.x;
    for (int k = threadIdx.x; k < R; k += blockDim.x) a[k] = aux[(size_t)i * R + k];
    __syncthreads();
    const double* L = Linv + (size_t)cls_u[i] * R * R;
    for (int r = threadIdx.x; r < R; r += blockDim.x) {
        double s = 0.0;
        for (int k = 0; k < R; ++k) s = fma(a[k], L[(size_t)k * R + r], s);
        e_h[(size_t)i * R + r] = s;
        e_hn[(size_t)i * R + r] = s * cls_n[i];
    }
}

// Rm = (sum_u cnt_u Linv_u + EhEh) / C ;  Am = sum_u cnt_u n_u Linv_u + EhnEh
__global__ void accumulators_kernel(const double* __restrict__ Linv, const double* __restrict__ cnt, const double* __restrict__ uniq_n, int U, int R,
                                    double inv_classes, double* __restrict__ Rm /* in: Eh'Eh */, double* __restrict__ Am /* in: Eh'diag(n)Eh */) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R * R) return;
    double sl = 0.0, snl = 0.0;
    for (int u = 0; u < U; ++u) {
        const double l = Linv[(size_t)u * R * R + i];
        sl += cnt[u] * l;
        snl += cnt[u] * uniq_n[u] * l;
    }
    Rm[i] = (sl + Rm[i]) * inv_classes;
    Am[i] = snl + Am[i];
}

__global__ void transpose_kernel(const double* __restrict__ in, int rows, int cols, double* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)rows * cols) return;
    const int r = (int)(i / cols), c = (int)(i % cols);
    out[(size_t)c * rows + r] = in[i];
}

// zero the strictly upper triangle (the Cholesky kernel leaves it as it was)
__global__ void tril_kernel(double* __restrict__ M, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n * n && (i % n) > (i / n)) M[i] = 0.0;
}

struct DBuf {
    double* p = nullptr;
    int alloc(size_t n) { return cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(double)) == cudaSuccess ? SKB_OK : SKB_ERR_CUDA; }
    ~DBuf() { cudaFree(p); }
};

}  // namespace skb

using namespace skb;

extern "C" {

// First half: the statistics the initialisation needs on the host (mean, total covariance, per-class sums).
int skb_plda_stats(const double* X_dev, int n_sess, int D, const int* cls_ptr_dev, const int* cls_rows_dev, int n_cls, double scaling,
                   double* mean_dev, double* sigma_obs_dev, double* S1_dev, void* stream) {
    if (!X_dev || !cls_ptr_dev || !cls_rows_dev || !mean_dev || !sigma_obs_dev || !S1_dev || n_sess <= 0 || D <= 0 || n_cls <= 0) {
        set_last_error(__FILE__, __LINE__, "plda_stats: bad arguments");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    DBuf xc;
    if (xc.alloc((size_t)n_sess * D)) { set_last_error(__FILE__, __LINE__, "plda_stats: out of memory"); return SKB_ERR_CUDA; }
    SKB_CUDA_CHECK(launch_kernel(false, colmean_kernel, (D + 127) / 128, 128, 0, st, X_dev, n_sess, D, mean_dev));
    const long long n = (long long)n_sess * D;
    SKB_CUDA_CHECK(launch_kernel(false, center_rows_kernel, (unsigned)((n + 255) / 256), 256, 0, st, X_dev, nullptr, mean_dev, n, D, xc.p));
    int rc = dgemm(1, 0, D, D, n_sess, 1.0 / n_sess, xc.p, D, xc.p, D, 0.0, sigma_obs_dev, D, st);     // statserver.py:920-928
    if (rc) return rc;
    SKB_CUDA_CHECK(launch_kernel(false, class_sum_kernel<double>, dim3((D + 127) / 128, n_cls), 128, 0, st, X_dev, D, (long long)D, cls_ptr_dev,
                                 cls_rows_dev, n_cls, scaling, S1_dev));
    SKB_CUDA_CHECK(cudaStreamSynchronize(st));
    return SKB_OK;
}

// Second half: nb_iter EM iterations.  S1 (n_cls, D) scaled class sums, cls_n (n_cls) scaled session counts, cls_u (n_cls)
// index of each class's count in uniq_n (U), cnt_u (U) number of classes per count; F_dev (D, R) in: the eigenvoice
// initialisation, out: the trained matrix; Sigma_dev (D, D) in: sigma_obs, out: the residual covariance.
int skb_plda_em(const double* S1_dev, const double* cls_n_dev, const int* cls_u_dev, int n_cls, const double* uniq_n_dev,
                const double* cnt_u_dev, int U, const double* mean_dev, const double* sigma_obs_dev, int D, int R, int nb_iter,
                double sum_n, double* F_dev, double* Sigma_dev, void* stream) {
    if (!S1_dev || !cls_n_dev || !cls_u_dev || !uniq_n_dev || !cnt_u_dev || !mean_dev || !sigma_obs_dev || !F_dev || !Sigma_dev ||
        n_cls <= 0 || U <= 0 || D <= 0 || R <= 0 || R > D || nb_iter < 0) {
        set_last_error(__FILE__, __LINE__, "plda_em: bad arguments");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    DBuf Ls, P, A0, Lam, Linv, Xc, aux, eh, ehn, Rm, Am, Cm, Xs, Ft;
    int* flag = nullptr;
    if (Ls.alloc((size_t)D * D) || P.alloc((size_t)D * R) || A0.alloc((size_t)R * R) || Lam.alloc((size_t)U * R * R) ||
        Linv.alloc((size_t)U * R * R) || Xc.alloc((size_t)n_cls * D) || aux.alloc((size_t)n_cls * R) || eh.alloc((size_t)n_cls * R) ||
        ehn.alloc((size_t)n_cls * R) || Rm.alloc((size_t)R * R) || Am.alloc((size_t)R * R) || Cm.alloc((size_t)R * D) ||
        Xs.alloc((size_t)R * D) || Ft.alloc((size_t)D * R) || cudaMalloc(&flag, sizeof(int)) != cudaSuccess) {
        cudaFree(flag);
        set_last_error(__FILE__, __LINE__, "plda_em: out of memory");
        return SKB_ERR_CUDA;
    }
    cudaMemsetAsync(flag, 0, sizeof(int), st);
    const long long nx = (long long)n_cls * D;
    const long long nl = (long long)U * R * R;
    // a failed launch leaves the EM loop with its error code, for the clean-up below
    int rc = [&]() -> int {
        // the centred class statistics S - n mu' never change (the mean is not re-estimated, factor_analyser.py:857)
        SKB_CUDA_CHECK(launch_kernel(false, center_rows_kernel, (unsigned)((nx + 255) / 256), 256, 0, st, S1_dev, cls_n_dev, mean_dev, nx, D,
                                     Xc.p));
        for (int it = 0; it < nb_iter; ++it) {
            // P = Sigma^-1 F  (Cholesky of Sigma; the strictly upper triangle of the copy is never read)
            cudaMemcpyAsync(Ls.p, Sigma_dev, (size_t)D * D * sizeof(double), cudaMemcpyDeviceToDevice, st);
            cudaMemcpyAsync(P.p, F_dev, (size_t)D * R * sizeof(double), cudaMemcpyDeviceToDevice, st);
            SKB_CUDA_CHECK(launch_kernel(false, dpotrf_kernel, 1, 1024, 0, st, Ls.p, D, flag));
            SKB_CUDA_CHECK(launch_kernel(false, dpotrs_kernel, dim3((R + 63) / 64, 1), 64, 0, st, Ls.p, D, P.p, R, 0, 0));
            // A0 = F' Sigma^-1 F ;  Linv_u = (n_u A0 + I)^-1 for every distinct session count (fa_model_loop :183-186)
            if (int e = dgemm(1, 0, R, R, D, 1.0, F_dev, R, P.p, R, 0.0, A0.p, R, st)) return e;
            SKB_CUDA_CHECK(launch_kernel(false, lambda_kernel, (unsigned)((nl + 255) / 256), 256, 0, st, A0.p, uniq_n_dev, R, U, Lam.p));
            SKB_CUDA_CHECK(launch_kernel(false, identity_kernel, (unsigned)((nl + 255) / 256), 256, 0, st, Linv.p, R, U));
            SKB_CUDA_CHECK(launch_kernel(false, dpotrf_kernel, U, 1024, 0, st, Lam.p, R, flag));
            SKB_CUDA_CHECK(launch_kernel(false, dpotrs_kernel, dim3((R + 63) / 64, U), 64, 0, st, Lam.p, R, Linv.p, R, (long long)R * R,
                                         (long long)R * R));
            // aux = (S - n mu') Sigma^-1 F ;  E[h_i] = aux_i Linv_{n_i}  (:188-190)
            if (int e = dgemm(0, 0, n_cls, R, D, 1.0, Xc.p, D, P.p, R, 0.0, aux.p, R, st)) return e;
            SKB_CUDA_CHECK(launch_kernel(false, posterior_mean_kernel, n_cls, 128, (size_t)R * sizeof(double), st, aux.p, Linv.p, cls_u_dev,
                                         cls_n_dev, R, eh.p, ehn.p));
            // accumulators (:907-912): R = sum E[hh'] / C,  A = sum n_i E[hh'],  C = E[h]' (S - n mu')
            if (int e = dgemm(1, 0, R, R, n_cls, 1.0, eh.p, R, eh.p, R, 0.0, Rm.p, R, st)) return e;
            if (int e = dgemm(1, 0, R, R, n_cls, 1.0, ehn.p, R, eh.p, R, 0.0, Am.p, R, st)) return e;
            SKB_CUDA_CHECK(launch_kernel(false, accumulators_kernel, (R * R + 255) / 256, 256, 0, st, Linv.p, cnt_u_dev, uniq_n_dev, U, R,
                                         1.0 / n_cls, Rm.p, Am.p));
            if (int e = dgemm(1, 0, R, D, n_cls, 1.0, eh.p, R, Xc.p, D, 0.0, Cm.p, D, st)) return e;
            // M-step (:915): F = solve(A, C)'  -- A is symmetric positive definite
            cudaMemcpyAsync(Xs.p, Cm.p, (size_t)R * D * sizeof(double), cudaMemcpyDeviceToDevice, st);
            SKB_CUDA_CHECK(launch_kernel(false, dpotrf_kernel, 1, 1024, 0, st, Am.p, R, flag));
            SKB_CUDA_CHECK(launch_kernel(false, dpotrs_kernel, dim3((D + 63) / 64, 1), 64, 0, st, Am.p, R, Xs.p, D, 0, 0));
            const long long nf = (long long)R * D;
            SKB_CUDA_CHECK(launch_kernel(false, transpose_kernel, (unsigned)((nf + 255) / 256), 256, 0, st, Xs.p, R, D, Ft.p));   // F_new (D, R)
            // residual covariance (:918): Sigma = sigma_obs - F_new C / sum n
            cudaMemcpyAsync(Sigma_dev, sigma_obs_dev, (size_t)D * D * sizeof(double), cudaMemcpyDeviceToDevice, st);
            if (int e = dgemm(0, 0, D, D, R, -1.0 / sum_n, Ft.p, R, Cm.p, D, 1.0, Sigma_dev, D, st)) return e;
            // minimum divergence (:921): F = F_new chol(R), scipy's upper factor U = L'
            SKB_CUDA_CHECK(launch_kernel(false, dpotrf_kernel, 1, 1024, 0, st, Rm.p, R, flag));
            SKB_CUDA_CHECK(launch_kernel(false, tril_kernel, (R * R + 255) / 256, 256, 0, st, Rm.p, R));
            if (int e = dgemm(0, 1, D, R, R, 1.0, Ft.p, R, Rm.p, R, 0.0, F_dev, R, st)) return e;
        }
        return SKB_OK;
    }();
    int bad = 0;
    if (!rc) {
        // cudaGetLastError: the unchecked device-to-device copies of the loop
        if (cudaGetLastError() != cudaSuccess || cudaMemcpyAsync(&bad, flag, sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess) {
            set_last_error(__FILE__, __LINE__, cudaGetErrorString(cudaGetLastError()));
            rc = SKB_ERR_CUDA;
        } else if (bad) {
            set_last_error(__FILE__, __LINE__, "plda_em: a covariance matrix is not positive definite");
            rc = SKB_ERR_ARG;
        }
    } else {
        cudaStreamSynchronize(st);
    }
    cudaFree(flag);
    return rc;
}

}  // extern "C"
