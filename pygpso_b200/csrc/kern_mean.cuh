// Linear mean function m(x) = x . A + b (gpflow.mean_functions.Linear).  The constant b travels as c0 through the residual and
// cross-covariance kernels, exactly like the constant of gpflow.mean_functions.Constant; these kernels add the x . A part.
//   linear_offset_kernel  out[i] += sgn * (x_i . A): candidate means (sgn = +1) and the training residual (sgn = -1)
//   linear_grad_kernel    out[k] = sum_j X[j][k] alpha[j]: d LML / d A
#pragma once

#include "common.cuh"

namespace gpso {

// x . A in a fixed order, s = fma(x[k], A[k], s) for k = 0..d-1: the value depends on the row alone, so duplicated candidates,
// shards and window positions get bit-identical offsets.  With A = 0 it is +0, and y - b - 0 = y - b exactly.
__global__ void __launch_bounds__(256) linear_offset_kernel(const double* __restrict__ X, long long rows, int d,
                                                            const double* __restrict__ A, double sgn, double* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows) return;
    const double* x = X + i * d;
    double s = 0.0;
    for (int k = 0; k < d; k++) s = fma(x[k], A[k], s);
    out[i] += sgn * s;  // sgn = +-1: the product is exact
}

// one block per input dimension k; fixed per-thread order and a fixed reduction tree (deterministic)
__global__ void __launch_bounds__(256) linear_grad_kernel(const double* __restrict__ X, const double* __restrict__ alpha, int N, int d,
                                                          double* __restrict__ out) {
    __shared__ double sRed[8];
    const int k = blockIdx.x;
    double s = 0.0;
    for (int j = threadIdx.x; j < N; j += 256) s = fma(X[(size_t)j * d + k], alpha[j], s);
    const double v = block_sum<256>(s, sRed);
    if (threadIdx.x == 0) out[k] = v;
}

}  // namespace gpso
