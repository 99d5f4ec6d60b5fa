// Per-class sums shared by PLDA training (plda_train.cu) and embedding conditioning (conditioning.cu).
#pragma once
#include <cuda_runtime.h>

namespace skb {

// per-class sums: S1[c] = sum of the rows of X whose class is c (fixed order: rows are visited in input order by one
// thread per (class, column) through the CSR lists) ; statserver.py:1335-1355.  X (rows, D) with row stride ld; float32
// rows are widened exactly.
template <typename T>
__global__ void class_sum_kernel(const T* __restrict__ X, int D, long long ld, const int* __restrict__ cls_ptr,
                                 const int* __restrict__ cls_rows, int n_cls, double scale, double* __restrict__ S1) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x, c = blockIdx.y;
    if (d >= D || c >= n_cls) return;
    double s = 0.0;
    for (int k = cls_ptr[c]; k < cls_ptr[c + 1]; ++k) s += (double)X[(size_t)cls_rows[k] * ld + d];
    S1[(size_t)c * D + d] = s * scale;
}

}  // namespace skb
