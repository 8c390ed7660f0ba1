// Device helpers of the Kzz whitening shared by the in-shared-memory kernels (whiten.cu, M <= GPODE_MAX_M) and the
// blocked float64 kernels (whiten_blocked.cu, GPODE_MAX_M < M <= GPODE_MAX_M_BLOCKED).
#pragma once
#include "common.cuh"
#include <math.h>

namespace {

// K_k(Z_m, Z_n) in double from the float32 parameters (direct squared-distance form)
__device__ __forceinline__ double rbf_entry(const float* __restrict__ Z, const double* __restrict__ inv_l, double vark,
                                            int D, int m, int n) {
    double e = 0.0;
    for (int j = 0; j < D; ++j) {
        const double d = ((double)Z[m * D + j] - (double)Z[n * D + j]) * inv_l[j];
        e += d * d;
    }
    return vark * exp(-0.5 * e);
}

// p_m = sum_s a_sk cos(theta_msk) for one inducing point m, by the calling warp: lanes over features, float32 angle
// like the reference (dsvgp.py:131-136) but double accumulation. Every lane returns the sum. ak = sqrt(var_k / S).
__device__ __forceinline__ double rff_at_point(const gpode_cache_t& c, int k, int m, float ak) {
    const int lane = threadIdx.x & 31, D = c.D, S = c.S;
    double acc = 0.0;
    for (int s = lane; s < S; s += 32) {
        float th = c.phase[s * D + k];
        for (int j = 0; j < D; ++j) th = fmaf(c.Z[m * D + j], c.omega[((size_t)j * S + s) * D + k], th);
        acc += (double)(c.w[s * D + k] * ak) * (double)gpode_cos_cw(th);   // 9e-8 at any angle, no libm slow path
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    return acc;
}

// This lane's share of G_j = d(pbm p_m)/dZ_mj of the above (the RFF VJP at x = Z_m, output dim k): the caller adds
// the lanes of the warp.
__device__ __forceinline__ void rff_vjp_at_point(const gpode_cache_t& c, int k, int m, double pbm, float ak,
                                                 double* G) {
    const int lane = threadIdx.x & 31, D = c.D, S = c.S;
    for (int j = 0; j < D; ++j) G[j] = 0.0;
    for (int s = lane; s < S; s += 32) {
        float th = c.phase[s * D + k];
        for (int j = 0; j < D; ++j) th = fmaf(c.Z[m * D + j], c.omega[((size_t)j * S + s) * D + k], th);
        const double g = -pbm * (double)(c.w[s * D + k] * ak) * (double)gpode_sin_cw(th);
        for (int j = 0; j < D; ++j) G[j] += g * (double)c.omega[((size_t)j * S + s) * D + k];
    }
}

// In-place right-looking Cholesky of the leading M x M block of A (row-major, leading dim ld); `rows` >= M extra
// rows below the block are carried along, so row r >= M ends up holding (L^-1 a_r)^T.
// dinv[c] receives 1 / L_cc: the triangular solves multiply by it instead of dividing (a float64 division is a ~40
// instruction dependent chain, and the column loop is the critical path of the whole kernel).
template <typename Real>
__device__ void chol_inplace(Real* A, int M, int rows, int ld, Real* dinv) {
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5, ny = blockDim.x >> 5;
    for (int c = 0; c < M; ++c) {
        __syncthreads();
        const Real acc_ = A[c * ld + c];
        const Real inv = rsqrt(acc_);        // one reciprocal square root instead of sqrt + division
        const Real dcc = acc_ * inv;
        if (threadIdx.x == 0) dinv[c] = inv;
        for (int i = c + 1 + ty; i < rows; i += ny) {
            const Real lic = A[i * ld + c] * inv;
            const int jmax = i < M ? i : M - 1;
            for (int j = c + 1 + tx; j <= jmax; j += 32) A[i * ld + j] -= lic * (A[j * ld + c] * inv);
        }
        __syncthreads();
        for (int i = c + 1 + threadIdx.x; i < rows; i += blockDim.x) A[i * ld + c] *= inv;
        if (threadIdx.x == 0) A[c * ld + c] = dcc;
    }
    __syncthreads();
}

}  // namespace
