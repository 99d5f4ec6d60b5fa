// Embedding conditioning on the device (statserver.py:789-1054, :1279-1333): the float64 scatter matrices behind the
// covariances, LDA, WCCN and spectral normalisation, and the row transforms that apply them.
//
// Everything is float64 arithmetic.  tcgen05 has no f64 kind, so the matrix products run on mma.sync m8n8k4 .f64 (SASS
// DMMA.8x8x4).  Inputs are float32 or float64 row-major matrices with a row stride; float32 is widened exactly on load.
//
// skb_gram_f64     G = scale * sum_i w_i (x_i - s_k(i)) (x_i - s_k(i))'.  The shift is subtracted while the operand is
//                  loaded (never the raw-moment shortcut, never a centred copy of X).  Only the lower triangle of 64 x 64
//                  tiles is computed; every row chunk writes its partial tiles to a workspace and one kernel sums the
//                  partials in chunk order and mirrors the triangle, so G is symmetric bit for bit.  The chunking is a
//                  function of (N, D) alone: results are bitwise reproducible from call to call and from card to card.
// skb_class_stats  column mean (row-chunk partials, summed in chunk order), per-class sums (class_sum_kernel over CSR
//                  lists, rows in input order) and per-class counts.
// skb_affine_rows  y_i = ((x_i - mu) .* d) W, optionally scaled to unit norm (floored at 1e-8) in the same pass when
//                  D_out <= 256.
#include "sidekit_b200.h"
#include "common.cuh"
#include "class_sum.cuh"

#include <algorithm>

namespace skb {

namespace {

constexpr int kMaxDim = 1024;

__device__ __forceinline__ double load_x(const float* p) { return (double)__ldg(p); }
__device__ __forceinline__ double load_x(const double* p) { return __ldg(p); }

// D (8x8) += A (8x4, row) B (4x8, col).  Lane (g = lane / 4, t = lane % 4) holds A[g][t], B[t][g] and D[g][2t], D[g][2t+1].
__device__ __forceinline__ void dmma884(double (&d)[2], double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d[0]), "+d"(d[1])
                 : "d"(a), "d"(b));
}

// ------------------------------------------------------------------------------------------------------------ Gram
// CTA = 4 warps (2 x 2), output tile 64 x 64 of the lower triangle, K (= rows of X) in steps of 16.  A warp owns 32 x 32
// of the tile: 4 x 4 DMMA tiles.  The operand tiles are stored k-major (Xs[k][column]); a row stride of 72 doubles puts
// the four k of one fragment load on disjoint bank halves, so every 32-lane LDS.64 takes the minimum two wavefronts.
constexpr int kGT = 64, kGK = 16, kGS = kGT + 8, kGThreads = 128;
constexpr int kGramTargetCtas = 2048;     // row chunks x triangle tiles aimed at; a constant, so the split depends on the shape only

struct GramPlan {
    int tiles_side, tiles;
    long long chunk_rows, chunks;
};
inline GramPlan gram_plan(long long N, int D) {
    GramPlan p;
    p.tiles_side = (D + kGT - 1) / kGT;
    p.tiles = p.tiles_side * (p.tiles_side + 1) / 2;
    long long want = std::max(1, (kGramTargetCtas + p.tiles - 1) / p.tiles);
    want = std::min(want, std::max(1LL, (N + 255) / 256));          // at least 256 rows a chunk
    p.chunk_rows = ((N + want - 1) / want + kGK - 1) / kGK * kGK;
    p.chunks = (N + p.chunk_rows - 1) / p.chunk_rows;
    return p;
}

template <typename T>
__global__ void __launch_bounds__(kGThreads) gram_f64_kernel(const T* __restrict__ X, long long N, int D, long long ld,
                                                             const double* __restrict__ shift, const int* __restrict__ shift_idx,
                                                             const double* __restrict__ w, long long chunk_rows,
                                                             double* __restrict__ partial) {
    __shared__ __align__(16) double As[kGK][kGS];
    __shared__ __align__(16) double Bs[kGK][kGS];
    // lower-triangle tile p -> (ti >= tj)
    const int p = blockIdx.x;
    int ti = 0;
    while ((ti + 1) * (ti + 2) / 2 <= p) ++ti;
    const int tj = p - ti * (ti + 1) / 2;
    const bool diag = ti == tj;
    const int ca0 = ti * kGT, cb0 = tj * kGT;
    const long long r0 = (long long)blockIdx.y * chunk_rows, r1 = min(N, r0 + chunk_rows);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int wm = (warp >> 1) * 32, wn = (warp & 1) * 32;
    // loader: column lc of both strips, rows lr + 2 j (j < 8) of the K step
    const int lc = tid & 63, lr = tid >> 6;
    const int ca = ca0 + lc, cb = cb0 + lc;

    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    double va[8], vb[8];
    auto fetch = [&](long long k0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const long long r = k0 + lr + 2 * j;
            double a = 0.0, b = 0.0;
            if (r < r1) {
                const T* row = X + r * ld;
                const double* s = shift ? shift + (size_t)(shift_idx ? shift_idx[r] : 0) * D : nullptr;
                if (ca < D) a = load_x(row + ca) - (s ? s[ca] : 0.0);
                if (diag) b = a;
                else if (cb < D) b = load_x(row + cb) - (s ? s[cb] : 0.0);
                if (w) a *= w[r];
            }
            va[j] = a;
            vb[j] = b;
        }
    };
    fetch(r0);
    for (long long k0 = r0; k0 < r1; k0 += kGK) {
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            As[lr + 2 * j][lc] = va[j];
            Bs[lr + 2 * j][lc] = vb[j];
        }
        __syncthreads();
        if (k0 + kGK < r1) fetch(k0 + kGK);
#pragma unroll
        for (int kk = 0; kk < kGK; kk += 4) {
            double fa[4], fb[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) fa[i] = As[kk + t][wm + 8 * i + g];
#pragma unroll
            for (int j = 0; j < 4; ++j) fb[j] = Bs[kk + t][wn + 8 * j + g];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) dmma884(acc[i][j], fa[i], fb[j]);
        }
    }
    double* out = partial + ((size_t)blockIdx.y * gridDim.x + p) * (kGT * kGT);
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = wm + 8 * i + g, c = wn + 8 * j + 2 * t;
            *reinterpret_cast<double2*>(out + r * kGT + c) = make_double2(acc[i][j][0], acc[i][j][1]);
        }
}

// G[a][b] = G[b][a] = scale * sum over chunks (in chunk order) of the partial tile element (a, b), a >= b
__global__ void gram_reduce_kernel(const double* __restrict__ partial, long long chunks, int tiles, int D, double scale,
                                   double* __restrict__ G) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)D * D) return;
    const int a = (int)(e / D), b = (int)(e % D);
    if (b > a) return;
    const int ti = a / kGT, tj = b / kGT;
    const size_t off = (size_t)(ti * (ti + 1) / 2 + tj) * (kGT * kGT) + (a % kGT) * kGT + (b % kGT);
    double s = 0.0;
    for (long long c = 0; c < chunks; ++c) s += partial[(size_t)c * tiles * (kGT * kGT) + off];
    s *= scale;
    G[(size_t)a * D + b] = s;
    G[(size_t)b * D + a] = s;
}

// ------------------------------------------------------------------------------------------------------------ mean
constexpr int kMeanRows = 2048;           // rows per partial: a function of N only

template <typename T>
__global__ void colsum_partial_kernel(const T* __restrict__ X, long long N, int D, long long ld, double* __restrict__ partial) {
    const int d = blockIdx.y * blockDim.x + threadIdx.x;
    if (d >= D) return;
    const long long r0 = (long long)blockIdx.x * kMeanRows, r1 = min(N, r0 + kMeanRows);
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    long long r = r0;
    for (; r + 4 <= r1; r += 4) {
        s0 += load_x(X + r * ld + d);
        s1 += load_x(X + (r + 1) * ld + d);
        s2 += load_x(X + (r + 2) * ld + d);
        s3 += load_x(X + (r + 3) * ld + d);
    }
    for (; r < r1; ++r) s0 += load_x(X + r * ld + d);
    partial[(size_t)blockIdx.x * D + d] = (s0 + s1) + (s2 + s3);
}

__global__ void colsum_final_kernel(const double* __restrict__ partial, long long chunks, int D, double inv_n, double* __restrict__ mean) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= D) return;
    double s = 0.0;
    for (long long c = 0; c < chunks; ++c) s += partial[(size_t)c * D + d];
    mean[d] = s * inv_n;
}

__global__ void class_count_kernel(const int* __restrict__ cls_ptr, int n_cls, double* __restrict__ counts) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < n_cls) counts[c] = (double)(cls_ptr[c + 1] - cls_ptr[c]);
}

// ------------------------------------------------------------------------------------------------------------ affine
// CTA = 8 warps, 32 rows x 256 output columns; warp w owns columns 32 w .. 32 w + 31 (4 x 4 DMMA tiles).  K = input
// dimension in steps of 16.  A = ((x - mu) .* d) is built by the loader (two elements a thread); the W tile is copied
// with cp.async into a double buffer.  Strides: 20 (A, k-contiguous) and 264 (B, n-contiguous) doubles give the
// minimum two wavefronts per fragment load.
constexpr int kAM = 32, kAN = 256, kAK = 16, kAThreads = 256, kASa = kAK + 4, kASb = kAN + 8;
constexpr size_t kAffineSmem = (size_t)(2 * kAM * kASa + 2 * kAK * kASb) * sizeof(double);

__device__ __forceinline__ void cp_async8(double* dst, const double* src, bool valid) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(valid ? 8 : 0) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

template <typename T> __device__ __forceinline__ void store_y(T* p, double v);
template <> __device__ __forceinline__ void store_y<float>(float* p, double v) { *p = (float)v; }
template <> __device__ __forceinline__ void store_y<double>(double* p, double v) { *p = v; }

template <typename T, typename U>
__global__ void __launch_bounds__(kAThreads) affine_dmma_kernel(const T* __restrict__ X, long long N, int D, long long ld,
                                                                const double* __restrict__ mu, const double* __restrict__ dsc,
                                                                const double* __restrict__ W, int D_out, int unit_norm,
                                                                U* __restrict__ Y, long long ld_out) {
    extern __shared__ __align__(16) double sm[];
    double* As = sm;                                   // [2][kAM][kASa]
    double* Bs = sm + 2 * kAM * kASa;                  // [2][kAK][kASb]
    __shared__ double red[8][kAM];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const long long row0 = (long long)blockIdx.x * kAM;
    const int col0 = blockIdx.y * kAN;
    // A loader: row ar, k = ak, ak + 1
    const int ar = tid >> 3, ak = (tid & 7) * 2;
    const long long arow = row0 + ar;
    const int bc = col0 + tid;                         // B loader: column bc, k rows 0..15

    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    double va[2];
    auto fetch_a = [&](int k0) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int k = k0 + ak + q;
            double v = 0.0;
            if (arow < N && k < D) {
                v = load_x(X + arow * ld + k);
                if (mu) v -= mu[k];
                if (dsc) v *= dsc[k];
            }
            va[q] = v;
        }
    };
    auto fetch_b = [&](int k0, int buf) {
        double* b = Bs + buf * kAK * kASb;
#pragma unroll
        for (int k = 0; k < kAK; ++k) {
            const bool ok = (k0 + k) < D && bc < D_out;
            cp_async8(b + k * kASb + tid, ok ? W + (size_t)(k0 + k) * D_out + bc : W, ok);
        }
        cp_async_commit();
    };
    const int nk = (D + kAK - 1) / kAK;
    fetch_a(0);
    fetch_b(0, 0);
    for (int kt = 0; kt < nk; ++kt) {
        const int buf = kt & 1;
        double* a = As + buf * kAM * kASa;
        a[ar * kASa + ak] = va[0];
        a[ar * kASa + ak + 1] = va[1];
        cp_async_wait_all();
        __syncthreads();                               // tile kt visible; everyone is done with tile kt - 1
        if (kt + 1 < nk) {
            fetch_a((kt + 1) * kAK);
            fetch_b((kt + 1) * kAK, buf ^ 1);
        }
        const double* b = Bs + buf * kAK * kASb;
#pragma unroll
        for (int kk = 0; kk < kAK; kk += 4) {
            double fa[4], fb[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) fa[i] = a[(8 * i + g) * kASa + kk + t];
#pragma unroll
            for (int j = 0; j < 4; ++j) fb[j] = b[(kk + t) * kASb + warp * 32 + 8 * j + g];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) dmma884(acc[i][j], fa[i], fb[j]);
        }
    }
    // fused length normalisation: this CTA holds whole rows (D_out <= 256); sums in a fixed order
    double nrm[4] = {1.0, 1.0, 1.0, 1.0};
    if (unit_norm) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            double s = 0.0;
#pragma unroll
            for (int j = 0; j < 4; ++j) s += acc[i][j][0] * acc[i][j][0] + acc[i][j][1] * acc[i][j][1];
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            if (t == 0) red[warp][8 * i + g] = s;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            double s = 0.0;
#pragma unroll
            for (int v = 0; v < 8; ++v) s += red[v][8 * i + g];
            nrm[i] = fmax(sqrt(s), 1e-8);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const long long r = row0 + 8 * i + g;
        if (r >= N) continue;
        U* y = Y + r * ld_out;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = col0 + warp * 32 + 8 * j + 2 * t;
            if (c < D_out) store_y(y + c, acc[i][j][0] / nrm[i]);
            if (c + 1 < D_out) store_y(y + c + 1, acc[i][j][1] / nrm[i]);
        }
    }
}

// Row pass, one warp per row: y = (x - mu) .* d (W absent), optionally scaled to unit norm (floored at 1e-8, norm_stat1).
template <typename T, typename U>
__global__ void affine_diag_rows_kernel(const T* __restrict__ X, long long N, int D, long long ld, const double* __restrict__ mu,
                                        const double* __restrict__ dsc, int unit_norm, U* __restrict__ Y, long long ld_out) {
    const long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= N) return;
    const T* x = X + r * ld;
    double nrm = 1.0;
    if (unit_norm) {
        double s = 0.0;
        for (int k = lane; k < D; k += 32) {
            double v = load_x(x + k);
            if (mu) v -= mu[k];
            if (dsc) v *= dsc[k];
            s += v * v;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        nrm = fmax(sqrt(s), 1e-8);
    }
    U* y = Y + r * ld_out;
    for (int k = lane; k < D; k += 32) {
        double v = load_x(x + k);
        if (mu) v -= mu[k];
        if (dsc) v *= dsc[k];
        store_y(y + k, v / nrm);
    }
}

// Second pass of an affine transform with D_out > 256: rows of Y scaled to unit norm in place.
template <typename U>
__global__ void unit_norm_rows_kernel(U* Y, long long N, int D, long long ld) {
    const long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= N) return;
    U* y = Y + r * ld;
    double s = 0.0;
    for (int k = lane; k < D; k += 32) s += (double)y[k] * (double)y[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const double nrm = fmax(sqrt(s), 1e-8);
    for (int k = lane; k < D; k += 32) store_y(y + k, (double)y[k] / nrm);
}

struct Workspace {
    double* p = nullptr;
    cudaStream_t st;
    explicit Workspace(cudaStream_t s) : st(s) {}
    cudaError_t alloc(size_t n) { return cudaMallocAsync((void**)&p, std::max<size_t>(n, 1) * sizeof(double), st); }
    ~Workspace() {
        if (p) cudaFreeAsync(p, st);
    }
};

bool bad_matrix(const void* X, long long N, int D, long long ld) { return !X || N <= 0 || D <= 0 || D > kMaxDim || ld < D; }

template <typename T>
int gram_launch(const T* X, long long N, int D, long long ld, const double* shift, const int* shift_idx, const double* w,
                double scale, double* G, cudaStream_t st) {
    const GramPlan p = gram_plan(N, D);
    Workspace ws(st);
    SKB_CUDA_CHECK(ws.alloc((size_t)p.chunks * p.tiles * kGT * kGT));
    SKB_CUDA_CHECK(launch_kernel(false, gram_f64_kernel<T>, dim3(p.tiles, (unsigned)p.chunks), kGThreads, 0, st, X, N, D, ld, shift, shift_idx, w,
                                 p.chunk_rows, ws.p));
    const long long n = (long long)D * D;
    SKB_CUDA_CHECK(launch_kernel(false, gram_reduce_kernel, (unsigned)((n + 255) / 256), 256, 0, st, ws.p, p.chunks, p.tiles, D, scale, G));
    return SKB_OK;
}

template <typename T>
int class_stats_launch(const T* X, long long N, int D, long long ld, const int* cls_ptr, const int* cls_rows, int n_cls,
                       double* mean, double* sums, double* counts, cudaStream_t st) {
    if (mean) {
        const long long chunks = (N + kMeanRows - 1) / kMeanRows;
        Workspace ws(st);
        SKB_CUDA_CHECK(ws.alloc((size_t)chunks * D));
        SKB_CUDA_CHECK(launch_kernel(false, colsum_partial_kernel<T>, dim3((unsigned)chunks, (D + 127) / 128), 128, 0, st, X, N, D, ld, ws.p));
        SKB_CUDA_CHECK(launch_kernel(false, colsum_final_kernel, (D + 127) / 128, 128, 0, st, ws.p, chunks, D, 1.0 / (double)N, mean));
    }
    if (sums)
        SKB_CUDA_CHECK(launch_kernel(false, class_sum_kernel<T>, dim3((D + 127) / 128, n_cls), 128, 0, st, X, D, ld, cls_ptr, cls_rows, n_cls, 1.0,
                                     sums));
    if (counts) SKB_CUDA_CHECK(launch_kernel(false, class_count_kernel, (n_cls + 255) / 256, 256, 0, st, cls_ptr, n_cls, counts));
    return SKB_OK;
}

template <typename T, typename U>
int affine_launch(const T* X, long long N, int D, long long ld, const double* mu, const double* dsc, const double* W, int D_out,
                  int unit_norm, U* Y, long long ld_out, cudaStream_t st) {
    if (!W) {
        const long long threads = N * 32;
        SKB_CUDA_CHECK(launch_kernel(false, affine_diag_rows_kernel<T, U>, (unsigned)((threads + 255) / 256), 256, 0, st, X, N, D, ld, mu, dsc,
                                     unit_norm, Y, ld_out));
        return SKB_OK;
    }
    static PerDeviceOnce once;
    if (once.first())
        SKB_CUDA_CHECK(cudaFuncSetAttribute(affine_dmma_kernel<T, U>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kAffineSmem));
    const bool fused = D_out <= kAN;
    dim3 grid((unsigned)((N + kAM - 1) / kAM), (D_out + kAN - 1) / kAN);
    SKB_CUDA_CHECK(launch_kernel(false, affine_dmma_kernel<T, U>, grid, kAThreads, kAffineSmem, st, X, N, D, ld, mu, dsc, W, D_out,
                                 unit_norm && fused, Y, ld_out));
    if (unit_norm && !fused) {
        const long long threads = N * 32;
        SKB_CUDA_CHECK(launch_kernel(false, unit_norm_rows_kernel<U>, (unsigned)((threads + 255) / 256), 256, 0, st, Y, N, D_out, ld_out));
    }
    return SKB_OK;
}

}  // namespace
}  // namespace skb

using namespace skb;

extern "C" {

int skb_gram_f64(const void* X_dev, int x_is_f64, int64_t N, int D, int64_t ld, const double* shift_dev, const int* shift_idx_dev,
                 const double* w_dev, double scale, double* G_dev, void* stream) {
    if (bad_matrix(X_dev, N, D, ld) || !G_dev || (shift_idx_dev && !shift_dev)) {
        set_last_error(__FILE__, __LINE__, "gram_f64: bad arguments");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    return x_is_f64 ? gram_launch((const double*)X_dev, N, D, ld, shift_dev, shift_idx_dev, w_dev, scale, G_dev, st)
                    : gram_launch((const float*)X_dev, N, D, ld, shift_dev, shift_idx_dev, w_dev, scale, G_dev, st);
}

int skb_class_stats(const void* X_dev, int x_is_f64, int64_t N, int D, int64_t ld, const int* cls_ptr_dev, const int* cls_rows_dev,
                    int n_cls, double* mean_dev, double* sums_dev, double* counts_dev, void* stream) {
    const bool classes = sums_dev || counts_dev;
    if (bad_matrix(X_dev, N, D, ld) || (!mean_dev && !classes) || (classes && (!cls_ptr_dev || n_cls <= 0)) ||
        (sums_dev && !cls_rows_dev)) {
        set_last_error(__FILE__, __LINE__, "class_stats: bad arguments");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    return x_is_f64 ? class_stats_launch((const double*)X_dev, N, D, ld, cls_ptr_dev, cls_rows_dev, n_cls, mean_dev, sums_dev, counts_dev, st)
                    : class_stats_launch((const float*)X_dev, N, D, ld, cls_ptr_dev, cls_rows_dev, n_cls, mean_dev, sums_dev, counts_dev, st);
}

int skb_affine_rows(const void* X_dev, int x_is_f64, int64_t N, int D, int64_t ld, const double* mu_dev, const double* d_dev,
                    const double* W_dev, int D_out, int unit_norm, void* Y_dev, int y_is_f64, int64_t ld_out, void* stream) {
    if (bad_matrix(X_dev, N, D, ld) || !Y_dev || D_out <= 0 || (!W_dev && D_out != D) || ld_out < D_out) {
        set_last_error(__FILE__, __LINE__, "affine_rows: bad arguments");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (x_is_f64)
        return y_is_f64 ? affine_launch((const double*)X_dev, N, D, ld, mu_dev, d_dev, W_dev, D_out, unit_norm, (double*)Y_dev, ld_out, st)
                        : affine_launch((const double*)X_dev, N, D, ld, mu_dev, d_dev, W_dev, D_out, unit_norm, (float*)Y_dev, ld_out, st);
    return y_is_f64 ? affine_launch((const float*)X_dev, N, D, ld, mu_dev, d_dev, W_dev, D_out, unit_norm, (double*)Y_dev, ld_out, st)
                    : affine_launch((const float*)X_dev, N, D, ld, mu_dev, d_dev, W_dev, D_out, unit_norm, (float*)Y_dev, ld_out, st);
}

}  // extern "C"
