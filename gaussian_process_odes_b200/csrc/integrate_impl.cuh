// Vector-field evaluation, fixed-grid RK4 (3/8 rule) forward and its discrete adjoint.
//
// Replaces (reference paths): DSVGP_Layer.forward src/core/dsvgp.py:172-197; torchdiffeq 0.2.0
// odeint(method='rk4') as called from Flow.forward src/core/flow.py:84-90 (step function rk4_alt_step_func, restated
// in oracle/torchdiffeq_shim); autograd through the unrolled solver (use_adjoint=False, train_vdp_gpode.py:52).
//
// Mapping: one thread owns R trajectories; their state, stage derivatives and adjoints live in registers for the
// whole time grid; the sampled function (RFF weights, Z, nu, lengthscales) lives in shared memory, staged once per
// CTA with a bulk async copy. Global traffic is only x0 in, xs (and stage checkpoints) out, all coalesced in the
// [time][row][dim] layout torchdiffeq itself returns.
#pragma once
#include <stdlib.h>
#include "vjp_mma.cuh"
#include "shoot.cuh"

namespace {

constexpr int kThreads = 128;

// rows (trajectories) per thread: as many as the register file allows without spills (ptxas -v, see DESIGN.md)
template <int D>
struct RowsFwd {
    static constexpr int value = D <= 2 ? 4 : (D <= 5 ? 2 : 1);
};
template <int D>
struct RowsBwd {
    static constexpr int value = D <= 2 ? 4 : (D <= 5 ? 2 : 1);
};

template <int D, int R>
__device__ __forceinline__ void load_rows(float (&v)[R][D], const float* __restrict__ base, const int64_t row0,
                                          const int64_t B, const int stride) {
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int64_t row = row0 + (int64_t)r * stride;
#pragma unroll
        for (int j = 0; j < D; ++j) v[r][j] = row < B ? __ldg(base + row * D + j) : 0.f;
    }
}

template <int D, int R>
__device__ __forceinline__ void store_rows(const float (&v)[R][D], float* __restrict__ base, const int64_t row0,
                                           const int64_t B, const int stride) {
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int64_t row = row0 + (int64_t)r * stride;
        if (row < B) {
#pragma unroll
            for (int j = 0; j < D; ++j) base[row * D + j] = v[r][j];
        }
    }
}

// Adjoint side of the fused shooting epilogue (shoot.cuh): the adjoint starts from lambda_T = g_ll seed_ll + g_cons seed_c
// and the gradient w.r.t. the sampled states also receives the constraint's pull on the NEXT state of the sequence,
// d cons / d ss[row + 1] = -seed_c[row].
struct ShootBwd {
    const float* seeds;   // [2, B, D]: d loglik / d pred | d constraint / d pred
    const float* g_ll;    // upstream gradient of the log-likelihood SUM (device scalar)
    const float* g_cons;  // upstream gradient of the constraint SUM (device scalar)
    float* grad_ss;       // [n_total, D] gradient w.r.t. all sampled states (rows outside this launch pre-zeroed)
    int64_t row_lo, n_total;
};

template <int D, int R>
__device__ __forceinline__ void shoot_lambda(float (&lam)[R][D], const ShootBwd& sb, const int64_t row0, const int64_t B,
                                             const int stride) {
    const float a = __ldg(sb.g_ll), b = __ldg(sb.g_cons);
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int64_t row = row0 + (int64_t)r * stride;
#pragma unroll
        for (int j = 0; j < D; ++j)
            lam[r][j] = row < B ? a * __ldg(sb.seeds + row * D + j) + b * __ldg(sb.seeds + (B + row) * D + j) : 0.f;
    }
}

template <int D, int R>
__device__ __forceinline__ void shoot_store_grad(const float (&lam)[R][D], const ShootBwd& sb, const int64_t row0,
                                                 const int64_t B, const int stride) {
    const float b = __ldg(sb.g_cons);
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int64_t row = row0 + (int64_t)r * stride;
        if (row < B) {
#pragma unroll
            for (int j = 0; j < D; ++j) {
                // the previous row's constraint pulls on this row's state (its seed is zero at a sequence end)
                const float pull = row >= 1 ? -b * __ldg(sb.seeds + (B + row - 1) * D + j) : 0.f;
                sb.grad_ss[(sb.row_lo + row) * D + j] = lam[r][j] + pull;
            }
            if (row == B - 1 && sb.row_lo + B < sb.n_total) {  // sharded launch: the state just past our last row
#pragma unroll
                for (int j = 0; j < D; ++j)
                    sb.grad_ss[(sb.row_lo + B) * D + j] = -b * __ldg(sb.seeds + (B + row) * D + j);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// f = vf(x)
// ------------------------------------------------------------------------------------------------------------------
template <int D, int R>
__global__ void __launch_bounds__(kThreads)
vf_fwd_kernel(const float* __restrict__ packed, const int M, const int S, const int total,
              const float* __restrict__ x, float* __restrict__ f, const int64_t B) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const float* sp = stage_params(smem_raw, packed, total);
    const int64_t tile_rows = (int64_t)blockDim.x * R;
    const int64_t ntiles = (B + tile_rows - 1) / tile_rows;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t row0 = tile * tile_rows + threadIdx.x;
        float xr[R][D], fr[R][D];
        load_rows<D, R>(xr, x, row0, B, blockDim.x);
        vf_eval<D, R>(sp, M, S, xr, fr);
        store_rows<D, R>(fr, f, row0, B, blockDim.x);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// RK4 3/8 rule, operation order of torchdiffeq 0.2.0 rk4_alt_step_func (no FMA contraction in the stage algebra so
// that, given identical stage derivatives, the step is bit-identical to the float32 torch ops):
//   k2 = f(y + dt*k1*(1/3)); k3 = f(y + dt*(k2 - k1*(1/3))); k4 = f(y + dt*(k1 - k2 + k3));
//   y1 = y + (k1 + 3*(k2 + k3) + k4) * dt * 0.125
// ------------------------------------------------------------------------------------------------------------------
#define GPODE_THIRD 0.3333333432674407958984375f  // float32(1/3), what torch multiplies by

template <int D, int R>
__device__ __forceinline__ void stage2(float (&o)[R][D], const float (&y)[R][D], const float (&k1)[R][D], float dt) {
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < D; ++j)
            o[r][j] = __fadd_rn(y[r][j], __fmul_rn(__fmul_rn(dt, k1[r][j]), GPODE_THIRD));
}
template <int D, int R>
__device__ __forceinline__ void stage3(float (&o)[R][D], const float (&y)[R][D], const float (&k1)[R][D],
                                       const float (&k2)[R][D], float dt) {
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < D; ++j)
            o[r][j] = __fadd_rn(y[r][j], __fmul_rn(dt, __fsub_rn(k2[r][j], __fmul_rn(k1[r][j], GPODE_THIRD))));
}
template <int D, int R>
__device__ __forceinline__ void stage4(float (&o)[R][D], const float (&y)[R][D], const float (&k1)[R][D],
                                       const float (&k2)[R][D], const float (&k3)[R][D], float dt) {
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < D; ++j)
            o[r][j] = __fadd_rn(y[r][j], __fmul_rn(dt, __fadd_rn(__fsub_rn(k1[r][j], k2[r][j]), k3[r][j])));
}

template <int D, int R, bool kShoot = false>
__global__ void __launch_bounds__(kThreads)
rk4_fwd_kernel(const float* __restrict__ packed, const int M, const int S, const int total,
               const float* __restrict__ x0, const float* __restrict__ ts, const int Tg, const int64_t B,
               float* __restrict__ xs, float* __restrict__ kst, const ShootArgs sh) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const float* sp = stage_params(smem_raw, packed, total);
    ShootSmem<D> ssm;
    double sh_ll = 0.0, sh_cs = 0.0;
    if constexpr (kShoot) ssm.init(smem_raw + 16 + (size_t)total * 4, sh);
    const int64_t tile_rows = (int64_t)blockDim.x * R;
    const int64_t ntiles = (B + tile_rows - 1) / tile_rows;
    const int64_t plane = B * D;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t row0 = tile * tile_rows + threadIdx.x;
        float y[R][D];
        load_rows<D, R>(y, x0, row0, B, blockDim.x);
        if constexpr (!kShoot) store_rows<D, R>(y, xs, row0, B, blockDim.x);
        for (int i = 0; i + 1 < Tg; ++i) {
            const float dt = __fsub_rn(__ldg(ts + i + 1), __ldg(ts + i));
            float k1[R][D], k2[R][D], k3[R][D], k4[R][D], ys[R][D];
            vf_eval<D, R>(sp, M, S, y, k1);
            stage2<D, R>(ys, y, k1, dt);
            vf_eval<D, R>(sp, M, S, ys, k2);
            stage3<D, R>(ys, y, k1, k2, dt);
            vf_eval<D, R>(sp, M, S, ys, k3);
            stage4<D, R>(ys, y, k1, k2, k3, dt);
            vf_eval<D, R>(sp, M, S, ys, k4);
            if (kst != nullptr) {
                float* kb = kst + (int64_t)i * 4 * plane;
                store_rows<D, R>(k1, kb, row0, B, blockDim.x);
                store_rows<D, R>(k2, kb + plane, row0, B, blockDim.x);
                store_rows<D, R>(k3, kb + 2 * plane, row0, B, blockDim.x);
                store_rows<D, R>(k4, kb + 3 * plane, row0, B, blockDim.x);
            }
#pragma unroll
            for (int r = 0; r < R; ++r)
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    const float sum = __fadd_rn(
                        __fadd_rn(k1[r][j], __fmul_rn(3.0f, __fadd_rn(k2[r][j], k3[r][j]))), k4[r][j]);
                    y[r][j] = __fadd_rn(y[r][j], __fmul_rn(__fmul_rn(sum, dt), 0.125f));
                }
            if constexpr (!kShoot) store_rows<D, R>(y, xs + (int64_t)(i + 1) * plane, row0, B, blockDim.x);
        }
        if constexpr (kShoot) {  // ELBO terms on the end point while it is in registers (shoot.cuh)
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int64_t row = row0 + (int64_t)r * blockDim.x;
                shoot_epilogue<D, true>(sh, ssm, row < B, row, B, y[r], sh_ll, sh_cs);
            }
        }
    }
    if constexpr (kShoot) shoot_finish<D>(sh, ssm, sh_ll, sh_cs);
}

// ------------------------------------------------------------------------------------------------------------------
// Discrete adjoint of the kernel above (SURVEY.md section 8a row A7). For every step, walking backwards:
//   kb4 = h/8 lam;                          yb4 = J(y4)^T kb4
//   kb3 = 3h/8 lam + h yb4;                 yb3 = J(y3)^T kb3
//   kb2 = 3h/8 lam + h yb3 - h yb4;         yb2 = J(y2)^T kb2
//   kb1 = h/8 lam + (h/3)(yb2 - yb3) + h yb4; yb1 = J(y1)^T kb1
//   lam <- grad_xs[i] + lam + yb1 + yb2 + yb3 + yb4
// Stage inputs are rebuilt bit-exactly from the checkpointed stage derivatives; (stage input, cotangent) pairs are
// written out as "virtual rows" for the per-inducing-point gradient kernel (param_grad.cu).
// ------------------------------------------------------------------------------------------------------------------
template <int D, int R, bool kShoot = false>
__global__ void __launch_bounds__(kThreads)
rk4_bwd_kernel(const float* __restrict__ packed, const int M, const int S, const int total,
               const float* __restrict__ ts, const int Tg, const int64_t B, const float* __restrict__ xs,
               const float* __restrict__ kst, const float* __restrict__ gxs, float* __restrict__ gx0,
               float* __restrict__ vy, float* __restrict__ vk, float* __restrict__ acc, const ShootBwd sb) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const float* sp = stage_params(smem_raw, packed, total);
    float* red = reinterpret_cast<float*>(smem_raw + 16) + total;

    float A[D][D], V[D];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        V[k] = 0.f;
#pragma unroll
        for (int j = 0; j < D; ++j) A[k][j] = 0.f;
    }

    const int64_t tile_rows = (int64_t)blockDim.x * R;
    const int64_t ntiles = (B + tile_rows - 1) / tile_rows;
    const int64_t plane = B * D;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t row0 = tile * tile_rows + threadIdx.x;
        float lam[R][D];
        if constexpr (kShoot) shoot_lambda<D, R>(lam, sb, row0, B, blockDim.x);
        else load_rows<D, R>(lam, gxs + (int64_t)(Tg - 1) * plane, row0, B, blockDim.x);
        for (int i = Tg - 2; i >= 0; --i) {
            const float h = __fsub_rn(__ldg(ts + i + 1), __ldg(ts + i));
            const float* kb = kst + (int64_t)i * 4 * plane;
            float* vyi = vy + (int64_t)i * 4 * plane;
            float* vki = vk + (int64_t)i * 4 * plane;
            float y[R][D], k1[R][D], k2[R][D], ks[R][D], ys[R][D], kbar[R][D], yb[R][D];
            float sumyb[R][D], yb4[R][D], yb23[R][D];
            load_rows<D, R>(y, xs + (int64_t)i * plane, row0, B, blockDim.x);
            load_rows<D, R>(k1, kb, row0, B, blockDim.x);
            load_rows<D, R>(k2, kb + plane, row0, B, blockDim.x);

            // ---- stage 4 ----
            load_rows<D, R>(ks, kb + 2 * plane, row0, B, blockDim.x);  // k3
            stage4<D, R>(ys, y, k1, k2, ks, h);
            load_rows<D, R>(ks, kb + 3 * plane, row0, B, blockDim.x);  // k4 = f(y4)
#pragma unroll
            for (int r = 0; r < R; ++r)
#pragma unroll
                for (int j = 0; j < D; ++j) kbar[r][j] = 0.125f * h * lam[r][j];
            store_rows<D, R>(ys, vyi + 3 * plane, row0, B, blockDim.x);
            store_rows<D, R>(kbar, vki + 3 * plane, row0, B, blockDim.x);
            vf_vjp<D, R>(sp, M, S, ys, kbar, ks, yb4, A, V);

            // ---- stage 3 ----
            stage3<D, R>(ys, y, k1, k2, h);
            load_rows<D, R>(ks, kb + 2 * plane, row0, B, blockDim.x);  // k3 = f(y3)
#pragma unroll
            for (int r = 0; r < R; ++r)
#pragma unroll
                for (int j = 0; j < D; ++j) kbar[r][j] = fmaf(0.375f * h, lam[r][j], h * yb4[r][j]);
            store_rows<D, R>(ys, vyi + 2 * plane, row0, B, blockDim.x);
            store_rows<D, R>(kbar, vki + 2 * plane, row0, B, blockDim.x);
            vf_vjp<D, R>(sp, M, S, ys, kbar, ks, yb, A, V);
#pragma unroll
            for (int r = 0; r < R; ++r)
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    sumyb[r][j] = yb4[r][j] + yb[r][j];
                    kbar[r][j] = fmaf(0.375f * h, lam[r][j], h * (yb[r][j] - yb4[r][j]));  // kb2
                    yb23[r][j] = -yb[r][j];
                }

            // ---- stage 2 ----
            stage2<D, R>(ys, y, k1, h);
            store_rows<D, R>(ys, vyi + plane, row0, B, blockDim.x);
            store_rows<D, R>(kbar, vki + plane, row0, B, blockDim.x);
            vf_vjp<D, R>(sp, M, S, ys, kbar, k2, yb, A, V);
#pragma unroll
            for (int r = 0; r < R; ++r)
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    sumyb[r][j] += yb[r][j];
                    yb23[r][j] += yb[r][j];  // yb2 - yb3
                    kbar[r][j] = fmaf(0.125f * h, lam[r][j], fmaf(h * GPODE_THIRD, yb23[r][j], h * yb4[r][j]));
                }

            // ---- stage 1 ----
            store_rows<D, R>(y, vyi, row0, B, blockDim.x);
            store_rows<D, R>(kbar, vki, row0, B, blockDim.x);
            vf_vjp<D, R>(sp, M, S, y, kbar, k1, yb, A, V);

            float gi[R][D];
            if constexpr (kShoot) {
#pragma unroll
                for (int r = 0; r < R; ++r)
#pragma unroll
                    for (int j = 0; j < D; ++j) gi[r][j] = 0.f;   // the segment start is not an output of the fused op
            } else {
                load_rows<D, R>(gi, gxs + (int64_t)i * plane, row0, B, blockDim.x);
            }
#pragma unroll
            for (int r = 0; r < R; ++r)
#pragma unroll
                for (int j = 0; j < D; ++j) lam[r][j] = gi[r][j] + lam[r][j] + (sumyb[r][j] + yb[r][j]);
        }
        if constexpr (kShoot) shoot_store_grad<D, R>(lam, sb, row0, B, blockDim.x);
        else store_rows<D, R>(lam, gx0, row0, B, blockDim.x);
    }
    __syncthreads();
    reduce_AV<D>(A, V, acc, red);
}

// VJP of a single vector-field evaluation (autograd through DSVGP_Layer.forward)
template <int D, int R>
__global__ void __launch_bounds__(kThreads)
vf_bwd_kernel(const float* __restrict__ packed, const int M, const int S, const int total,
              const float* __restrict__ x, const float* __restrict__ f, const float* __restrict__ gf,
              float* __restrict__ gx, const int64_t B, float* __restrict__ acc) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const float* sp = stage_params(smem_raw, packed, total);
    float* red = reinterpret_cast<float*>(smem_raw + 16) + total;
    float A[D][D], V[D];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        V[k] = 0.f;
#pragma unroll
        for (int j = 0; j < D; ++j) A[k][j] = 0.f;
    }
    const int64_t tile_rows = (int64_t)blockDim.x * R;
    const int64_t ntiles = (B + tile_rows - 1) / tile_rows;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t row0 = tile * tile_rows + threadIdx.x;
        float xr[R][D], fr[R][D], kb[R][D], xb[R][D];
        load_rows<D, R>(xr, x, row0, B, blockDim.x);
        load_rows<D, R>(fr, f, row0, B, blockDim.x);
        load_rows<D, R>(kb, gf, row0, B, blockDim.x);
        vf_vjp<D, R>(sp, M, S, xr, kb, fr, xb, A, V);
        store_rows<D, R>(xb, gx, row0, B, blockDim.x);
    }
    __syncthreads();
    reduce_AV<D>(A, V, acc, red);
}

// ------------------------------------------------------------------------------------------------------------------
// Warp-per-row variants for small batches (the reference's own training shapes: N = 1 / 6 trajectories over 75-100
// sequential steps, or a few thousand shooting segments). One warp owns one trajectory: its 32 lanes split the S
// Fourier features and the M inducing points of every evaluation and combine the partial sums with an xor-shuffle
// all-reduce, so the state stays replicated in registers and one evaluation costs ~(S+M)/32 feature visits instead
// of S+M. Same arithmetic per term; only the summation order differs from the row-per-thread kernels.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kWarpsPerCta = 4;

template <int D>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
vf_fwd_warp_kernel(const float* __restrict__ packed, const int M, const int S, const int total,
                   const float* __restrict__ x, float* __restrict__ f, const int64_t B) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const float* sp = stage_params(smem_raw, packed, total);
    const int lane = threadIdx.x & 31;
    for (int64_t row = (int64_t)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5); row < B;
         row += (int64_t)gridDim.x * kWarpsPerCta) {
        float xr[1][D], fr[1][D];
        load_rows<D, 1>(xr, x, row, B, 0);
        vf_eval_warp<D>(sp, M, S, xr, fr, lane);
        if (lane == 0) store_rows<D, 1>(fr, f, row, B, 0);
    }
}

// one trajectory, one warp: the whole fixed grid
template <int D>
__device__ __forceinline__ void rk4_row_warp(const float* sp, const int M, const int S, const float* __restrict__ x0,
                                             const float* __restrict__ ts, const int Tg, const int64_t row,
                                             const int64_t B, float* __restrict__ xs, float* __restrict__ kst,
                                             const int lane, float (&y)[1][D]) {
    const int64_t plane = B * D;
    load_rows<D, 1>(y, x0, row, B, 0);
    if (lane == 0 && xs != nullptr) store_rows<D, 1>(y, xs, row, B, 0);
    for (int i = 0; i + 1 < Tg; ++i) {
        const float dt = __fsub_rn(__ldg(ts + i + 1), __ldg(ts + i));
        float k1[1][D], k2[1][D], k3[1][D], k4[1][D], ys[1][D];
        vf_eval_warp<D>(sp, M, S, y, k1, lane);
        stage2<D, 1>(ys, y, k1, dt);
        vf_eval_warp<D>(sp, M, S, ys, k2, lane);
        stage3<D, 1>(ys, y, k1, k2, dt);
        vf_eval_warp<D>(sp, M, S, ys, k3, lane);
        stage4<D, 1>(ys, y, k1, k2, k3, dt);
        vf_eval_warp<D>(sp, M, S, ys, k4, lane);
        if (kst != nullptr && lane == 0) {
            float* kb = kst + (int64_t)i * 4 * plane;
            store_rows<D, 1>(k1, kb, row, B, 0);
            store_rows<D, 1>(k2, kb + plane, row, B, 0);
            store_rows<D, 1>(k3, kb + 2 * plane, row, B, 0);
            store_rows<D, 1>(k4, kb + 3 * plane, row, B, 0);
        }
#pragma unroll
        for (int j = 0; j < D; ++j) {
            const float sum = __fadd_rn(__fadd_rn(k1[0][j], __fmul_rn(3.0f, __fadd_rn(k2[0][j], k3[0][j]))),
                                        k4[0][j]);
            y[0][j] = __fadd_rn(y[0][j], __fmul_rn(__fmul_rn(sum, dt), 0.125f));
        }
        if (lane == 0 && xs != nullptr) store_rows<D, 1>(y, xs + (int64_t)(i + 1) * plane, row, B, 0);
    }
}

template <int D, bool kShoot = false>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
rk4_fwd_warp_kernel(const float* __restrict__ packed, const int M, const int S, const int total,
                    const float* __restrict__ x0, const float* __restrict__ ts, const int Tg, const int64_t B,
                    float* __restrict__ xs, float* __restrict__ kst, const ShootArgs sh) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const float* sp = stage_params(smem_raw, packed, total);
    ShootSmem<D> ssm;
    double sh_ll = 0.0, sh_cs = 0.0;
    if constexpr (kShoot) ssm.init(smem_raw + 16 + (size_t)total * 4, sh);
    const int lane = threadIdx.x & 31;
    for (int64_t row = (int64_t)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5); row < B;
         row += (int64_t)gridDim.x * kWarpsPerCta) {
        float y[1][D];
        rk4_row_warp<D>(sp, M, S, x0, ts, Tg, row, B, kShoot ? nullptr : xs, kst, lane, y);
        if constexpr (kShoot) {  // every lane holds the same end point: lane 0 evaluates the ELBO terms of the row
            if (lane == 0) shoot_epilogue<D, false>(sh, ssm, true, row, B, y[0], sh_ll, sh_cs);
        }
    }
    if constexpr (kShoot) shoot_finish<D>(sh, ssm, sh_ll, sh_cs);
}

// ---- batched Monte-Carlo prediction: blockIdx.y = parameter set; set q owns rows [q set_rows, (q+1) set_rows) and the
// packed block at packed + q set_stride (SURVEY.md 8b item 1 "n_sets", 8f item 3) ------------------------------------
template <int D>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
vf_fwd_sets_kernel(const float* __restrict__ packed, const int M, const int S, const int total,
                   const int64_t set_stride, const int64_t set_rows, const float* __restrict__ x,
                   float* __restrict__ f) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const float* sp = stage_params(smem_raw, packed + blockIdx.y * set_stride, total);
    const int lane = threadIdx.x & 31;
    const int64_t B = set_rows * gridDim.y;
    for (int64_t r = (int64_t)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5); r < set_rows;
         r += (int64_t)gridDim.x * kWarpsPerCta) {
        const int64_t row = blockIdx.y * set_rows + r;
        float xr[1][D], fr[1][D];
        load_rows<D, 1>(xr, x, row, B, 0);
        vf_eval_warp<D>(sp, M, S, xr, fr, lane);
        if (lane == 0) store_rows<D, 1>(fr, f, row, B, 0);
    }
}

template <int D>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
rk4_fwd_sets_kernel(const float* __restrict__ packed, const int M, const int S, const int total,
                    const int64_t set_stride, const int64_t set_rows, const float* __restrict__ x0,
                    const float* __restrict__ ts, const int Tg, float* __restrict__ xs) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const float* sp = stage_params(smem_raw, packed + blockIdx.y * set_stride, total);
    const int lane = threadIdx.x & 31;
    const int64_t B = set_rows * gridDim.y;
    for (int64_t r = (int64_t)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5); r < set_rows;
         r += (int64_t)gridDim.x * kWarpsPerCta)
    {
        float yend[1][D];
        rk4_row_warp<D>(sp, M, S, x0, ts, Tg, blockIdx.y * set_rows + r, B, xs, nullptr, lane, yend);
    }
}

template <int D, bool kShoot = false>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
rk4_bwd_warp_kernel(const float* __restrict__ packed, const int M, const int S, const int total,
                    const float* __restrict__ ts, const int Tg, const int64_t B, const float* __restrict__ xs,
                    const float* __restrict__ kst, const float* __restrict__ gxs, float* __restrict__ gx0,
                    float* __restrict__ vy, float* __restrict__ vk, float* __restrict__ acc, const ShootBwd sb) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const float* sp = stage_params(smem_raw, packed, total);
    double* slabs = reinterpret_cast<double*>(reinterpret_cast<float*>(smem_raw + 16) + total);
    WarpAcc64<D> wa;
    wa.init(slabs);
    const int lane = threadIdx.x & 31;
    const int64_t plane = B * D;
    for (int64_t row = (int64_t)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5); row < B;
         row += (int64_t)gridDim.x * kWarpsPerCta) {
        float lam[1][D];
        if constexpr (kShoot) shoot_lambda<D, 1>(lam, sb, row, B, 0);
        else load_rows<D, 1>(lam, gxs + (int64_t)(Tg - 1) * plane, row, B, 0);
        for (int i = Tg - 2; i >= 0; --i) {
            const float h = __fsub_rn(__ldg(ts + i + 1), __ldg(ts + i));
            const float* kb = kst + (int64_t)i * 4 * plane;
            float* vyi = vy + (int64_t)i * 4 * plane;
            float* vki = vk + (int64_t)i * 4 * plane;
            float y[1][D], k1[1][D], k2[1][D], k3[1][D], k4[1][D], ys[1][D], kbar[1][D], yb[1][D];
            float sumyb[1][D], yb4[1][D], yb23[1][D];
            load_rows<D, 1>(y, xs + (int64_t)i * plane, row, B, 0);
            load_rows<D, 1>(k1, kb, row, B, 0);
            load_rows<D, 1>(k2, kb + plane, row, B, 0);
            load_rows<D, 1>(k3, kb + 2 * plane, row, B, 0);
            load_rows<D, 1>(k4, kb + 3 * plane, row, B, 0);
            // stage 4
            stage4<D, 1>(ys, y, k1, k2, k3, h);
#pragma unroll
            for (int j = 0; j < D; ++j) kbar[0][j] = 0.125f * h * lam[0][j];
            if (lane == 0) {
                store_rows<D, 1>(ys, vyi + 3 * plane, row, B, 0);
                store_rows<D, 1>(kbar, vki + 3 * plane, row, B, 0);
            }
            vf_vjp_warp<D>(sp, M, S, ys, kbar, k4, yb4, wa, lane);
            // stage 3
            stage3<D, 1>(ys, y, k1, k2, h);
#pragma unroll
            for (int j = 0; j < D; ++j) kbar[0][j] = fmaf(0.375f * h, lam[0][j], h * yb4[0][j]);
            if (lane == 0) {
                store_rows<D, 1>(ys, vyi + 2 * plane, row, B, 0);
                store_rows<D, 1>(kbar, vki + 2 * plane, row, B, 0);
            }
            vf_vjp_warp<D>(sp, M, S, ys, kbar, k3, yb, wa, lane);
#pragma unroll
            for (int j = 0; j < D; ++j) {
                sumyb[0][j] = yb4[0][j] + yb[0][j];
                kbar[0][j] = fmaf(0.375f * h, lam[0][j], h * (yb[0][j] - yb4[0][j]));
                yb23[0][j] = -yb[0][j];
            }
            // stage 2
            stage2<D, 1>(ys, y, k1, h);
            if (lane == 0) {
                store_rows<D, 1>(ys, vyi + plane, row, B, 0);
                store_rows<D, 1>(kbar, vki + plane, row, B, 0);
            }
            vf_vjp_warp<D>(sp, M, S, ys, kbar, k2, yb, wa, lane);
#pragma unroll
            for (int j = 0; j < D; ++j) {
                sumyb[0][j] += yb[0][j];
                yb23[0][j] += yb[0][j];
                kbar[0][j] = fmaf(0.125f * h, lam[0][j], fmaf(h * GPODE_THIRD, yb23[0][j], h * yb4[0][j]));
            }
            // stage 1
            if (lane == 0) {
                store_rows<D, 1>(y, vyi, row, B, 0);
                store_rows<D, 1>(kbar, vki, row, B, 0);
            }
            vf_vjp_warp<D>(sp, M, S, y, kbar, k1, yb, wa, lane);
            float gi[1][D];
            if constexpr (kShoot) {
#pragma unroll
                for (int j = 0; j < D; ++j) gi[0][j] = 0.f;
            } else {
                load_rows<D, 1>(gi, gxs + (int64_t)i * plane, row, B, 0);
            }
#pragma unroll
            for (int j = 0; j < D; ++j) lam[0][j] = gi[0][j] + lam[0][j] + (sumyb[0][j] + yb[0][j]);
        }
        if (lane == 0) {
            if constexpr (kShoot) shoot_store_grad<D, 1>(lam, sb, row, B, 0);
            else store_rows<D, 1>(lam, gx0, row, B, 0);
        }
    }
    __syncthreads();
    reduce_AV64<D>(wa, acc, slabs + kWarpsPerCta * WarpAcc64<D>::kSlabDoubles);
}

template <int D>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
vf_bwd_warp_kernel(const float* __restrict__ packed, const int M, const int S, const int total,
                   const float* __restrict__ x, const float* __restrict__ f, const float* __restrict__ gf,
                   float* __restrict__ gx, const int64_t B, float* __restrict__ acc) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const float* sp = stage_params(smem_raw, packed, total);
    double* slabs = reinterpret_cast<double*>(reinterpret_cast<float*>(smem_raw + 16) + total);
    WarpAcc64<D> wa;
    wa.init(slabs);
    const int lane = threadIdx.x & 31;
    for (int64_t row = (int64_t)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5); row < B;
         row += (int64_t)gridDim.x * kWarpsPerCta) {
        float xr[1][D], fr[1][D], kb[1][D], xb[1][D];
        load_rows<D, 1>(xr, x, row, B, 0);
        load_rows<D, 1>(fr, f, row, B, 0);
        load_rows<D, 1>(kb, gf, row, B, 0);
        vf_vjp_warp<D>(sp, M, S, xr, kb, fr, xb, wa, lane);
        if (lane == 0) store_rows<D, 1>(xb, gx, row, B, 0);
    }
    __syncthreads();
    reduce_AV64<D>(wa, acc, slabs + kWarpsPerCta * WarpAcc64<D>::kSlabDoubles);
}

// ---- tensor-core adjoint kernels (vjp_mma.cuh) -------------------------------------------------------------------
// One CTA of kHWarps warps per SM (the f16 operand records take ~92 KB at D = 5, S = 256, so they are staged once per
// SM); a warp owns 32 rows, lane = row.
// dynamic shared memory: [0,16) mbarrier | [kern | il] | mmah records | (D*D + D) block-reduction floats | per-warp stage;
// the RK4 adjoint drops the block-reduction floats (its reduction reuses the per-warp row state, dead by then) and
// appends the per-warp row state and, when it sums the inducing-point gradients itself, the per-warp row sums
#ifndef GPODE_HWARPS
#define GPODE_HWARPS 12
#endif
constexpr int kHWarps = GPODE_HWARPS;
constexpr int kHThreads = kHWarps * 32;

struct HParams {
    int M, S8P, off_kern, n_small, off_mmah, n_mmah;
};

constexpr int kHRowFields = 7;  // rk4_bwd_mma_kernel: adjoint state per row kept in shared memory (D floats each)
template <int D>
struct HSmem {
    const float* small;
    const uint32_t* mmah;
    float* red;
    float* stage;
    float* rows;  // rk4 adjoint: kHWarps x kHRowFields x D x 32 floats of row state, then kHWarps x M x 2D row sums
    __device__ __forceinline__ HSmem(unsigned char* smem_raw, const HParams& p, const bool rk4 = false) {
        float* sp = reinterpret_cast<float*>(smem_raw + 16);
        small = sp;
        mmah = reinterpret_cast<const uint32_t*>(sp + p.n_small);
        float* q = sp + p.n_small + p.n_mmah;
        red = q;
        if (!rk4) q += kRedFloats<D>;
        stage = q + (threadIdx.x >> 5) * HShape<D>::kStageFloats;
        rows = q + kHWarps * HShape<D>::kStageFloats;
        if (rk4) red = rows;  // kHWarps * kHRowFields * D * 32 >= kRedFloats<D>
    }
};

template <int D>
__device__ __forceinline__ void hacc_reduce(const HAcc<D>& qa, const float* __restrict__ small, const int M,
                                            float* __restrict__ acc, float* red) {
    float A[D][D], V[D];
    qa.expand(small + M * VfShape<D>::KS, threadIdx.x & 3, A, V);
    __syncthreads();
    reduce_AV<D>(A, V, acc, red);
}

template <int D>
__global__ void __launch_bounds__(kHThreads, 1)
vf_bwd_mma_kernel(const float* __restrict__ packed, const HParams p, const float* __restrict__ x,
                  const float* __restrict__ f, const float* __restrict__ gf, float* __restrict__ gx, const int64_t B,
                  float* __restrict__ acc) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    stage_params_h(smem_raw, packed, p.off_kern, p.n_small, p.off_mmah, p.n_mmah);
    const HSmem<D> sm(smem_raw, p);
    HAcc<D> qa;
    qa.clear();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t nblocks = (B + 31) / 32;
    for (int64_t blk = (int64_t)blockIdx.x * kHWarps + warp; blk < nblocks; blk += (int64_t)gridDim.x * kHWarps) {
        const int64_t row = blk * 32 + lane;
        float xr[1][D], fr[1][D], kb[1][D], xb[1][D];
        load_rows<D, 1>(xr, x, row, B, 0);
        load_rows<D, 1>(fr, f, row, B, 0);
        load_rows<D, 1>(kb, gf, row, B, 0);
        vf_vjp_h<D>(sm.small, sm.mmah, sm.stage, p.M, p.S8P, xr, kb, fr, xb, qa, lane);
        store_rows<D, 1>(xb, gx, row, B, 0);
    }
    hacc_reduce<D>(qa, sm.small, p.M, acc, sm.red);
}

// ---- tensor-core forward kernels (vf_eval_h): staging and CTA shape as the adjoint ----
constexpr int kHFWarps = 12;  // measured: rk4 step 2.03 ms at 12 warps, 2.07 at 16 (single evaluation: 0.553 vs 0.530)
constexpr int kHFThreads = kHFWarps * 32;
template <int D>
__global__ void __launch_bounds__(kHFThreads, 1)
vf_fwd_h_kernel(const float* __restrict__ packed, const HParams p, const float* __restrict__ x, float* __restrict__ f,
                const int64_t B) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    stage_params_h(smem_raw, packed, p.off_kern, p.n_small, p.off_mmah, p.n_mmah);
    const HSmem<D> sm(smem_raw, p);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t nblocks = (B + 31) / 32;
    for (int64_t blk = (int64_t)blockIdx.x * kHFWarps + warp; blk < nblocks; blk += (int64_t)gridDim.x * kHFWarps) {
        const int64_t row = blk * 32 + lane;
        float xr[1][D], fr[1][D];
        load_rows<D, 1>(xr, x, row, B, 0);
        vf_eval_h<D>(sm.small, sm.mmah, sm.stage, p.M, p.S8P, xr, fr, lane);
        store_rows<D, 1>(fr, f, row, B, 0);
    }
}

// rk4_fwd_kernel<D, 1> with the evaluations on the tensor cores; the four stages loop around ONE inlined evaluation
template <int D, bool kShoot = false>
__global__ void __launch_bounds__(kHFThreads, 1)
rk4_fwd_h_kernel(const float* __restrict__ packed, const HParams p, const float* __restrict__ x0,
                 const float* __restrict__ ts, const int Tg, const int64_t B, float* __restrict__ xs,
                 float* __restrict__ kst, const ShootArgs sh, const int shoot_off) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    stage_params_h(smem_raw, packed, p.off_kern, p.n_small, p.off_mmah, p.n_mmah);
    const HSmem<D> sm(smem_raw, p);
    ShootSmem<D> ssm;
    double sh_ll = 0.0, sh_cs = 0.0;
    if constexpr (kShoot) ssm.init(smem_raw + shoot_off, sh);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int R = 1;
    const int64_t nblocks = (B + 31) / 32;
    const int64_t plane = B * D;
    for (int64_t blk = (int64_t)blockIdx.x * kHFWarps + warp; blk < nblocks; blk += (int64_t)gridDim.x * kHFWarps) {
        const int64_t row0 = blk * 32 + lane;
        float y[R][D];
        load_rows<D, R>(y, x0, row0, B, 0);
        if constexpr (!kShoot) store_rows<D, R>(y, xs, row0, B, 0);
        for (int i = 0; i + 1 < Tg; ++i) {
            const float dt = __fsub_rn(__ldg(ts + i + 1), __ldg(ts + i));
            float k1[R][D], k2[R][D], k3[R][D], k4[R][D], ys[R][D], kk[R][D];
#pragma unroll
            for (int j = 0; j < D; ++j) {
                ys[0][j] = y[0][j];
                k1[0][j] = k2[0][j] = k3[0][j] = k4[0][j] = 0.f;
            }
#pragma unroll 1
            for (int st = 1; st <= 4; ++st) {
                vf_eval_h<D>(sm.small, sm.mmah, sm.stage, p.M, p.S8P, ys, kk, lane);
                if (kst != nullptr) store_rows<D, R>(kk, kst + ((int64_t)i * 4 + (st - 1)) * plane, row0, B, 0);
                if (st == 1) {
#pragma unroll
                    for (int j = 0; j < D; ++j) k1[0][j] = kk[0][j];
                    stage2<D, R>(ys, y, k1, dt);
                } else if (st == 2) {
#pragma unroll
                    for (int j = 0; j < D; ++j) k2[0][j] = kk[0][j];
                    stage3<D, R>(ys, y, k1, k2, dt);
                } else if (st == 3) {
#pragma unroll
                    for (int j = 0; j < D; ++j) k3[0][j] = kk[0][j];
                    stage4<D, R>(ys, y, k1, k2, k3, dt);
                } else {
#pragma unroll
                    for (int j = 0; j < D; ++j) k4[0][j] = kk[0][j];
                }
            }
#pragma unroll
            for (int j = 0; j < D; ++j) {
                const float sum = __fadd_rn(__fadd_rn(k1[0][j], __fmul_rn(3.0f, __fadd_rn(k2[0][j], k3[0][j]))), k4[0][j]);
                y[0][j] = __fadd_rn(y[0][j], __fmul_rn(__fmul_rn(sum, dt), 0.125f));
            }
            if constexpr (!kShoot) store_rows<D, R>(y, xs + (int64_t)(i + 1) * plane, row0, B, 0);
        }
        if constexpr (kShoot) shoot_epilogue<D, true>(sh, ssm, row0 < B, row0, B, y[0], sh_ll, sh_cs);
    }
    if constexpr (kShoot) shoot_finish<D>(sh, ssm, sh_ll, sh_cs);
}

// Discrete adjoint of the 3/8-rule RK4 grid: the recursion, checkpoint reads and virtual-row outputs of
// rk4_bwd_kernel<D, 1>, with the four VJPs of a step on the tensor cores. The adjoint state that merely waits while a
// VJP runs (lambda, y, k1, k2 and the three running cotangent sums: 7 D floats per row) rests in shared memory
// ([field][component][lane], conflict-free), so the VJP has the 168 registers of a 12-warp CTA to itself -- with that
// state in registers ptxas spilled inside the VJP loops (3.82 ms; 8 warps at 239 registers: 3.69 ms).
// kRowSums: no virtual rows; the VJPs sum the inducing-point gradients over the warp's rows (vf_vjp_h) into a per-warp
// shared-memory accumulator, and the CTA adds its warps in warp order, in float64, into its row-sum row of `acc`.
template <int D, bool kShoot = false, bool kRowSums = false>
__global__ void __launch_bounds__(kHThreads, 1)
rk4_bwd_mma_kernel(const float* __restrict__ packed, const HParams p, const float* __restrict__ ts, const int Tg,
                   const int64_t B, const float* __restrict__ xs, const float* __restrict__ kst,
                   const float* __restrict__ gxs, float* __restrict__ gx0, float* __restrict__ vy,
                   float* __restrict__ vk, float* __restrict__ acc, const ShootBwd sb) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    stage_params_h(smem_raw, packed, p.off_kern, p.n_small, p.off_mmah, p.n_mmah);
    const HSmem<D> sm(smem_raw, p, true);
    HAcc<D> qa;
    qa.clear();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int R = 1;
    enum { F_LAM = 0, F_Y = 1, F_K1 = 2, F_K2 = 3, F_SUM = 4, F_YB4 = 5, F_Y23 = 6 };
    float* __restrict__ rs = sm.rows + warp * (kHRowFields * D * 32) + lane;
    constexpr int NV = 2 * D;
    float* __restrict__ rsum_all = sm.rows + kHWarps * kHRowFields * D * 32;
    float* __restrict__ rsum = rsum_all + warp * p.M * NV;
    if constexpr (kRowSums) {
        for (int i = lane; i < p.M * NV; i += 32) rsum[i] = 0.f;
        __syncwarp();
    }
    auto put = [&](const int f, const float (&v)[R][D]) {
#pragma unroll
        for (int j = 0; j < D; ++j) rs[(f * D + j) * 32] = v[0][j];
    };
    auto get = [&](const int f, float (&v)[R][D]) {
#pragma unroll
        for (int j = 0; j < D; ++j) v[0][j] = rs[(f * D + j) * 32];
    };

    const int64_t nblocks = (B + 31) / 32;
    const int64_t plane = B * D;
    for (int64_t blk = (int64_t)blockIdx.x * kHWarps + warp; blk < nblocks; blk += (int64_t)gridDim.x * kHWarps) {
        const int64_t row0 = blk * 32 + lane;
        {
            float lam[R][D];
            if constexpr (kShoot) shoot_lambda<D, R>(lam, sb, row0, B, 0);
            else load_rows<D, R>(lam, gxs + (int64_t)(Tg - 1) * plane, row0, B, 0);
            put(F_LAM, lam);
        }
        for (int i = Tg - 2; i >= 0; --i) {
            const float h = __fsub_rn(__ldg(ts + i + 1), __ldg(ts + i));
            const float* kb = kst + (int64_t)i * 4 * plane;
            float ks[R][D], ys[R][D], kbar[R][D], yb[R][D];
            {
                float t[R][D];
                load_rows<D, R>(t, xs + (int64_t)i * plane, row0, B, 0);
                put(F_Y, t);
                load_rows<D, R>(t, kb, row0, B, 0);
                put(F_K1, t);
                load_rows<D, R>(t, kb + plane, row0, B, 0);
                put(F_K2, t);
                get(F_LAM, t);
#pragma unroll
                for (int j = 0; j < D; ++j) kbar[0][j] = 0.125f * h * t[0][j];
            }
            // the four stages share ONE inlined VJP (code size): stage input, forward value and the cotangent
            // bookkeeping are selected by uniform branches around it
#pragma unroll 1
            for (int st = 4; st >= 1; --st) {
                {
                    float y[R][D], k1[R][D], k2[R][D];
                    get(F_Y, y);
                    get(F_K1, k1);
                    get(F_K2, k2);
                    if (st == 4) {
                        load_rows<D, R>(ks, kb + 2 * plane, row0, B, 0);  // k3
                        stage4<D, R>(ys, y, k1, k2, ks, h);
                        load_rows<D, R>(ks, kb + 3 * plane, row0, B, 0);  // k4 = f(y4)
                    } else if (st == 3) {
                        stage3<D, R>(ys, y, k1, k2, h);
                        load_rows<D, R>(ks, kb + 2 * plane, row0, B, 0);  // k3 = f(y3)
                    } else if (st == 2) {
                        stage2<D, R>(ys, y, k1, h);
#pragma unroll
                        for (int j = 0; j < D; ++j) ks[0][j] = k2[0][j];
                    } else {
#pragma unroll
                        for (int j = 0; j < D; ++j) {
                            ys[0][j] = y[0][j];
                            ks[0][j] = k1[0][j];
                        }
                    }
                }
                if constexpr (!kRowSums) {
                    store_rows<D, R>(ys, vy + ((int64_t)i * 4 + st - 1) * plane, row0, B, 0);
                    store_rows<D, R>(kbar, vk + ((int64_t)i * 4 + st - 1) * plane, row0, B, 0);
                }
                vf_vjp_h<D, kRowSums>(sm.small, sm.mmah, sm.stage, p.M, p.S8P, ys, kbar, ks, yb, qa, lane, rsum);
                float lam[R][D];
                get(F_LAM, lam);
                if (st == 4) {
                    put(F_YB4, yb);
#pragma unroll
                    for (int j = 0; j < D; ++j) kbar[0][j] = fmaf(0.375f * h, lam[0][j], h * yb[0][j]);
                } else if (st == 3) {
                    float yb4[R][D], sum[R][D], y23[R][D];
                    get(F_YB4, yb4);
#pragma unroll
                    for (int j = 0; j < D; ++j) {
                        sum[0][j] = yb4[0][j] + yb[0][j];
                        kbar[0][j] = fmaf(0.375f * h, lam[0][j], h * (yb[0][j] - yb4[0][j]));  // kb2
                        y23[0][j] = -yb[0][j];
                    }
                    put(F_SUM, sum);
                    put(F_Y23, y23);
                } else if (st == 2) {
                    float yb4[R][D], sum[R][D], y23[R][D];
                    get(F_YB4, yb4);
                    get(F_SUM, sum);
                    get(F_Y23, y23);
#pragma unroll
                    for (int j = 0; j < D; ++j) {
                        sum[0][j] += yb[0][j];
                        y23[0][j] += yb[0][j];  // yb2 - yb3
                        kbar[0][j] = fmaf(0.125f * h, lam[0][j], fmaf(h * GPODE_THIRD, y23[0][j], h * yb4[0][j]));
                    }
                    put(F_SUM, sum);
                } else {
                    float sum[R][D], gi[R][D];
                    get(F_SUM, sum);
                    if constexpr (kShoot) {
#pragma unroll
                        for (int j = 0; j < D; ++j) gi[0][j] = 0.f;
                    } else {
                        load_rows<D, R>(gi, gxs + (int64_t)i * plane, row0, B, 0);
                    }
#pragma unroll
                    for (int j = 0; j < D; ++j) lam[0][j] = gi[0][j] + lam[0][j] + (sum[0][j] + yb[0][j]);
                    put(F_LAM, lam);
                }
            }
        }
        float lam[R][D];
        get(F_LAM, lam);
        if constexpr (kShoot) shoot_store_grad<D, R>(lam, sb, row0, B, 0);
        else store_rows<D, R>(lam, gx0, row0, B, 0);
    }
    hacc_reduce<D>(qa, sm.small, p.M, acc, sm.red);   // its barrier also orders every warp's row sums before the reads
    if constexpr (kRowSums) {
        const GpodeAcc a = gpode_acc_layout(D, p.M);
        double* __restrict__ row = reinterpret_cast<double*>(acc + a.off_rs) + (size_t)blockIdx.x * p.M * NV;
        for (int i = threadIdx.x; i < p.M * NV; i += blockDim.x) {
            double s = 0.0;
            for (int w = 0; w < kHWarps; ++w) s += (double)rsum_all[w * p.M * NV + i];
            row[i] = s;
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) reinterpret_cast<int*>(acc)[2] = (int)gridDim.x;
    }
}

// ------------------------------------------------------------------------------------------------------------------
// host-side launch helpers
// ------------------------------------------------------------------------------------------------------------------
struct LaunchShape {
    int threads, grid;
    size_t smem;
};

inline int num_sms() {
    static int g_num_sms = 0;
    if (g_num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
        if (g_num_sms <= 0) g_num_sms = 148;
    }
    return g_num_sms;
}

template <typename K>
inline int shape_for(K kernel, int R, int64_t B, size_t smem, LaunchShape* out) {
    // small batches: narrow CTAs so the rows spread over more SMs; large: 128 threads, grid = SMs x resident CTAs
    int threads = (B <= (int64_t)num_sms() * 32 * R) ? 32 : kThreads;
    if (int rc = check_smem_fits(smem)) return rc;
    GPODE_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    GPODE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, smem));
    if (occ < 1) {
        gpode_set_error("kernel does not fit on an SM (smem %zu bytes)", smem);
        return -2;
    }
    const int64_t tile_rows = (int64_t)threads * R;
    const int64_t ntiles = (B + tile_rows - 1) / tile_rows;
    int64_t cap = (int64_t)num_sms() * occ;
    if (cap > GPODE_ACC_CAP_AV) cap = GPODE_ACC_CAP_AV;  // one accumulator row per CTA (common.cuh, GpodeAcc)
    out->threads = threads;
    out->grid = (int)(ntiles < cap ? ntiles : cap);
    out->smem = smem;
    return 0;
}

}  // namespace

// ------------------------------------------------------------------------------------------------------------------
// per-D launchers: wide tiles (R rows per thread) when the batch fills the machine twice over, else one row per thread
// ------------------------------------------------------------------------------------------------------------------
// batches up to this many rows go to the warp-per-row kernels (above it, row-per-thread fills the machine)
constexpr int64_t kWarpPathMaxRows = 16384;

template <typename K>
inline int warp_shape_for(K kernel, int64_t B, size_t smem, LaunchShape* out) {
    if (int rc = check_smem_fits(smem)) return rc;
    GPODE_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    GPODE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, kWarpsPerCta * 32, smem));
    if (occ < 1) {
        gpode_set_error("kernel does not fit on an SM (smem %zu bytes)", smem);
        return -2;
    }
    const int64_t want = (B + kWarpsPerCta - 1) / kWarpsPerCta;
    int64_t cap = (int64_t)num_sms() * occ;
    if (cap > GPODE_ACC_CAP_AV) cap = GPODE_ACC_CAP_AV;  // one accumulator row per CTA (common.cuh, GpodeAcc)
    out->threads = kWarpsPerCta * 32;
    out->grid = (int)(want < cap ? want : cap);
    out->smem = smem;
    return 0;
}

template <int D, int R>
inline bool use_wide(int64_t B) {
    return R > 1 && B >= (int64_t)num_sms() * 2 * kThreads * R;
}


// Tensor-core adjoint (vjp_mma.cuh): state dimensions whose three split parts fit one k = 16 contraction, batches that
// fill the machine. GPODE_BWD_MMA=0 keeps the FFMA2 adjoint.
template <int D>
constexpr bool kMmaBwd = (D >= 4 && D <= GPODE_MMAH_MAX_D);  // D = 3: measured slower than FFMA2 (1.77 vs 1.56 ms)
inline bool use_mma_bwd(int64_t B) {
    if (gpode_option(GPODE_OPT_BWD_MMA) == 0) return false;  // the parity tests run both adjoints in one process
    return B >= (int64_t)num_sms() * kHThreads;
}
inline bool use_mma_fwd(int64_t B) {
    if (gpode_option(GPODE_OPT_FWD_MMA) == 0) return false;  // 0 keeps the FFMA2 forward kernels
    return B >= (int64_t)num_sms() * kHFThreads;
}
template <int D>
inline HParams h_params(const GpodeLayout& L) {
    HParams p;
    p.M = L.M; p.S8P = L.S8P;
    p.off_kern = L.off_kern; p.n_small = L.total - L.off_kern;
    p.off_mmah = L.off_mmah; p.n_mmah = D * L.S8P * GPODE_MMAH_REC;
    return p;
}
template <int D>
inline size_t h_smem(const HParams& p, bool rk4 = true, int warps = kHWarps, bool row_sums = false) {
    return 16 + ((size_t)p.n_small + p.n_mmah + (rk4 ? 0 : kRedFloats<D>) + (size_t)warps * HShape<D>::kStageFloats +
                 (rk4 ? (size_t)warps * kHRowFields * D * 32 : 0) + (row_sums ? (size_t)warps * p.M * 2 * D : 0)) * 4;
}
// The shooting adjoint sums the inducing-point gradients inside the tensor-core kernel (no virtual rows, no
// gpode_param_grad) when that kernel is selected and its per-warp row sums fit in shared memory next to the operand
// records: at S = 256, D = 5 up to M = 101 inducing points, D = 4 up to M = 201.
template <int D>
inline bool use_mma_row_sums(int M, int S, int64_t B) {
    if constexpr (kMmaBwd<D>) {
        return use_mma_bwd(B) && h_smem<D>(h_params<D>(gpode_layout(D, M, S)), true, kHWarps, true) <= 227 * 1024;
    } else {
        return false;
    }
}
template <typename K>
inline int h_grid(K kernel, int64_t B, size_t smem, int* grid, int threads = kHThreads) {
    if (smem > 227 * 1024) {
        gpode_set_error("tensor-core adjoint needs %zu bytes of shared memory", smem);
        return -2;
    }
    GPODE_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t want = (B + threads - 1) / threads, cap = num_sms();
    *grid = (int)(want < cap ? want : cap);
    return 0;
}

template <int D>
int launch_vf_fwd(const float* packed, int M, int S, const float* x, float* f, int64_t B, cudaStream_t st) {
    const GpodeLayout L = gpode_layout(D, M, S);
    const size_t smem = 16 + (size_t)L.total * 4;
    LaunchShape ls;
    constexpr int RW = RowsFwd<D>::value;
    if constexpr (kMmaBwd<D>) {
        const HParams hp = h_params<D>(L);
        const size_t hs = h_smem<D>(hp, false, kHFWarps);
        if (use_mma_fwd(B) && hs <= 227 * 1024) {
            int grid = 0;
            if (int rc = h_grid(vf_fwd_h_kernel<D>, B, hs, &grid, kHFThreads)) return rc;
            vf_fwd_h_kernel<D><<<grid, kHFThreads, hs, st>>>(packed, hp, x, f, B);
            GPODE_LAUNCH_CHECK();
            return 0;
        }
    }
    if (B <= kWarpPathMaxRows) {
        if (int rc = warp_shape_for(vf_fwd_warp_kernel<D>, B, smem, &ls)) return rc;
        vf_fwd_warp_kernel<D><<<ls.grid, ls.threads, ls.smem, st>>>(packed, M, S, L.total, x, f, B);
    } else if (use_wide<D, RW>(B)) {
        if (int rc = shape_for(vf_fwd_kernel<D, RW>, RW, B, smem, &ls)) return rc;
        vf_fwd_kernel<D, RW><<<ls.grid, ls.threads, ls.smem, st>>>(packed, M, S, L.total, x, f, B);
    } else {
        if (int rc = shape_for(vf_fwd_kernel<D, 1>, 1, B, smem, &ls)) return rc;
        vf_fwd_kernel<D, 1><<<ls.grid, ls.threads, ls.smem, st>>>(packed, M, S, L.total, x, f, B);
    }
    GPODE_LAUNCH_CHECK();
    return 0;
}

template <int D, bool kShoot = false>
int launch_rk4_fwd(const float* packed, int M, int S, const float* x0, const float* t, int Tg, int64_t B, float* xs,
                   float* kst, cudaStream_t st, const ShootArgs sh = ShootArgs{}, int* grid_out = nullptr) {
    const GpodeLayout L = gpode_layout(D, M, S);
    auto shoot_bytes = [&](int nwarps) { return kShoot ? shoot_smem_bytes(D, sh.Dobs, nwarps) : (size_t)0; };
    const size_t smem = 16 + (size_t)L.total * 4 + shoot_bytes(kThreads / 32);
    LaunchShape ls;
    constexpr int RW = RowsFwd<D>::value;
    if constexpr (kMmaBwd<D>) {
        const HParams hp = h_params<D>(L);
        const size_t hs0 = (h_smem<D>(hp, false, kHFWarps) + 15) & ~(size_t)15;
        const size_t hs = hs0 + shoot_bytes(kHFWarps);
        if (use_mma_fwd(B) && hs <= 227 * 1024) {
            int grid = 0;
            if (int rc = h_grid(rk4_fwd_h_kernel<D, kShoot>, B, hs, &grid, kHFThreads)) return rc;
            rk4_fwd_h_kernel<D, kShoot><<<grid, kHFThreads, hs, st>>>(packed, hp, x0, t, Tg, B, xs, kst, sh, (int)hs0);
            GPODE_LAUNCH_CHECK();
            if (grid_out) *grid_out = grid;
            return 0;
        }
    }
    if (B <= kWarpPathMaxRows) {
        const size_t smem_w = 16 + (size_t)L.total * 4 + shoot_bytes(kWarpsPerCta);
        if (int rc = warp_shape_for(rk4_fwd_warp_kernel<D, kShoot>, B, smem_w, &ls)) return rc;
        rk4_fwd_warp_kernel<D, kShoot><<<ls.grid, ls.threads, ls.smem, st>>>(packed, M, S, L.total, x0, t, Tg, B, xs,
                                                                             kst, sh);
    } else if (use_wide<D, RW>(B)) {
        if (int rc = shape_for(rk4_fwd_kernel<D, RW, kShoot>, RW, B, smem, &ls)) return rc;
        rk4_fwd_kernel<D, RW, kShoot><<<ls.grid, ls.threads, ls.smem, st>>>(packed, M, S, L.total, x0, t, Tg, B, xs,
                                                                            kst, sh);
    } else {
        if (int rc = shape_for(rk4_fwd_kernel<D, 1, kShoot>, 1, B, smem, &ls)) return rc;
        rk4_fwd_kernel<D, 1, kShoot><<<ls.grid, ls.threads, ls.smem, st>>>(packed, M, S, L.total, x0, t, Tg, B, xs, kst,
                                                                           sh);
    }
    GPODE_LAUNCH_CHECK();
    if (grid_out) *grid_out = ls.grid;
    return 0;
}

// sets: grid = (CTAs per set, n_sets); a CTA never mixes rows of two sets
template <int D>
int launch_fwd_sets(const float* packed, int M, int S, int n_sets, int64_t set_rows, const float* x0, const float* t,
                    int Tg, float* out, cudaStream_t st) {
    const GpodeLayout L = gpode_layout(D, M, S);
    const size_t smem = 16 + (size_t)L.total * 4;
    const int threads = kWarpsPerCta * 32;
    const int64_t per_set = (set_rows + kWarpsPerCta - 1) / kWarpsPerCta;
    // enough CTAs per set to spread over the machine, never more than its rows need
    int64_t want = ((int64_t)num_sms() * 4 + n_sets - 1) / n_sets;
    if (want > per_set) want = per_set;
    if (want < 1) want = 1;
    const dim3 grid((unsigned)want, (unsigned)n_sets);
    if (int rc = check_smem_fits(smem)) return rc;
    if (t == nullptr) {
        GPODE_CUDA(cudaFuncSetAttribute(vf_fwd_sets_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        vf_fwd_sets_kernel<D><<<grid, threads, smem, st>>>(packed, M, S, L.total, L.n_packed, set_rows, x0, out);
    } else {
        GPODE_CUDA(cudaFuncSetAttribute(rk4_fwd_sets_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        rk4_fwd_sets_kernel<D><<<grid, threads, smem, st>>>(packed, M, S, L.total, L.n_packed, set_rows, x0, t, Tg,
                                                            out);
    }
    GPODE_LAUNCH_CHECK();
    return 0;
}

template <int D, bool kShoot = false>
int launch_rk4_bwd(const float* packed, int M, int S, const float* t, int Tg, int64_t B, const float* xs,
                   const float* kst, const float* gxs, float* gx0, float* vy, float* vk, float* acc,
                   cudaStream_t st, const ShootBwd sb = ShootBwd{}) {
    const GpodeLayout L = gpode_layout(D, M, S);
    const size_t smem = 16 + (size_t)(L.total + kRedFloats<D>) * 4;
    LaunchShape ls;
    constexpr int RW = RowsBwd<D>::value;
    if constexpr (kMmaBwd<D>) {
        const HParams hp = h_params<D>(L);
        if (kShoot && vy == nullptr) {   // no virtual rows: the caller checked use_mma_row_sums (gpode_shoot_bwd)
            const size_t hs = h_smem<D>(hp, true, kHWarps, true);
            int grid = 0;
            if (int rc = h_grid(rk4_bwd_mma_kernel<D, true, true>, B, hs, &grid)) return rc;
            rk4_bwd_mma_kernel<D, true, true><<<grid, kHThreads, hs, st>>>(packed, hp, t, Tg, B, xs, kst, gxs, gx0,
                                                                          nullptr, nullptr, acc, sb);
            GPODE_LAUNCH_CHECK();
            return 0;
        }
        if (use_mma_bwd(B) && h_smem<D>(hp) <= 227 * 1024) {
            int grid = 0;
            if (int rc = h_grid(rk4_bwd_mma_kernel<D, kShoot>, B, h_smem<D>(hp), &grid)) return rc;
            rk4_bwd_mma_kernel<D, kShoot><<<grid, kHThreads, h_smem<D>(hp), st>>>(packed, hp, t, Tg, B, xs, kst, gxs,
                                                                                  gx0, vy, vk, acc, sb);
            GPODE_LAUNCH_CHECK();
            return 0;
        }
    }
    if (B <= kWarpPathMaxRows) {
        const size_t smem_w = 16 + (size_t)L.total * 4 + (size_t)kWarpAccDoubles<D>(kWarpsPerCta) * 8;
        if (int rc = warp_shape_for(rk4_bwd_warp_kernel<D, kShoot>, B, smem_w, &ls)) return rc;
        rk4_bwd_warp_kernel<D, kShoot><<<ls.grid, ls.threads, ls.smem, st>>>(packed, M, S, L.total, t, Tg, B, xs, kst,
                                                                             gxs, gx0, vy, vk, acc, sb);
    } else if (use_wide<D, RW>(B)) {
        if (int rc = shape_for(rk4_bwd_kernel<D, RW, kShoot>, RW, B, smem, &ls)) return rc;
        rk4_bwd_kernel<D, RW, kShoot><<<ls.grid, ls.threads, ls.smem, st>>>(packed, M, S, L.total, t, Tg, B, xs, kst,
                                                                            gxs, gx0, vy, vk, acc, sb);
    } else {
        if (int rc = shape_for(rk4_bwd_kernel<D, 1, kShoot>, 1, B, smem, &ls)) return rc;
        rk4_bwd_kernel<D, 1, kShoot><<<ls.grid, ls.threads, ls.smem, st>>>(packed, M, S, L.total, t, Tg, B, xs, kst,
                                                                           gxs, gx0, vy, vk, acc, sb);
    }
    GPODE_LAUNCH_CHECK();
    return 0;
}

template <int D>
int launch_vf_bwd(const float* packed, int M, int S, const float* x, const float* f, const float* gf, float* gx,
                  int64_t B, float* acc, cudaStream_t st) {
    const GpodeLayout L = gpode_layout(D, M, S);
    const size_t smem = 16 + (size_t)(L.total + kRedFloats<D>) * 4;
    LaunchShape ls;
    constexpr int RW = RowsBwd<D>::value;
    if constexpr (kMmaBwd<D>) {
        const HParams hp = h_params<D>(L);
        if (use_mma_bwd(B) && h_smem<D>(hp) <= 227 * 1024) {
            int grid = 0;
            if (int rc = h_grid(vf_bwd_mma_kernel<D>, B, h_smem<D>(hp, false), &grid)) return rc;
            vf_bwd_mma_kernel<D><<<grid, kHThreads, h_smem<D>(hp, false), st>>>(packed, hp, x, f, gf, gx, B, acc);
            GPODE_LAUNCH_CHECK();
            return 0;
        }
    }
    if (B <= kWarpPathMaxRows) {
        const size_t smem_w = 16 + (size_t)L.total * 4 + (size_t)kWarpAccDoubles<D>(kWarpsPerCta) * 8;
        if (int rc = warp_shape_for(vf_bwd_warp_kernel<D>, B, smem_w, &ls)) return rc;
        vf_bwd_warp_kernel<D><<<ls.grid, ls.threads, ls.smem, st>>>(packed, M, S, L.total, x, f, gf, gx, B, acc);
    } else if (use_wide<D, RW>(B)) {
        if (int rc = shape_for(vf_bwd_kernel<D, RW>, RW, B, smem, &ls)) return rc;
        vf_bwd_kernel<D, RW><<<ls.grid, ls.threads, ls.smem, st>>>(packed, M, S, L.total, x, f, gf, gx, B, acc);
    } else {
        if (int rc = shape_for(vf_bwd_kernel<D, 1>, 1, B, smem, &ls)) return rc;
        vf_bwd_kernel<D, 1><<<ls.grid, ls.threads, ls.smem, st>>>(packed, M, S, L.total, x, f, gf, gx, B, acc);
    }
    GPODE_LAUNCH_CHECK();
    return 0;
}
