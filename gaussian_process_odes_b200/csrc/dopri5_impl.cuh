// Adaptive Dormand-Prince 5(4) with torchdiffeq 0.2.0's controller, as ONE cooperative persistent kernel.
//
// Replaces odeint(func, y0, t, rtol, atol, method='dopri5') (the reference's default solver, src/core/flow.py:41,84-90;
// algorithm restated in oracle/torchdiffeq_shim from torchdiffeq 0.2.0: rk_common._runge_kutta_step / _adaptive_step,
// misc._select_initial_step / _optimal_step_size / _compute_error_ratio, interp._interp_fit / _interp_evaluate).
//
// The reference decides accept/reject on the HOST after every attempt (one device->host sync per attempt, ~40 tiny
// kernels in between). Here every thread owns rows of the batch, keeps the controller state (t, dt in float64,
// pending output index) replicated in registers, and the only cross-thread quantity -- the whole-batch RMS error
// norm -- is reduced through a float64 atomic accumulator and ONE grid-wide barrier per attempt.
#pragma once
#include <cooperative_groups.h>
#include "vf.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int kDpThreads = 128;
constexpr int kDpMaxGrid = 2048;  // cooperative grid cap: 3 rotating error sums x one float64 slot per CTA
constexpr int kDpSetThreads = 256;  // sets mode: one CTA per parameter set, up to 8 warps = 8 rows in flight

// Dormand-Prince / Shampine tableau (float32 copies, like torchdiffeq's tableau cast to the state dtype)
__device__ __constant__ float kBeta[6][6] = {
    {1.f / 5, 0, 0, 0, 0, 0},
    {3.f / 40, 9.f / 40, 0, 0, 0, 0},
    {44.f / 45, -56.f / 15, 32.f / 9, 0, 0, 0},
    {(float)(19372.0 / 6561), (float)(-25360.0 / 2187), (float)(64448.0 / 6561), (float)(-212.0 / 729), 0, 0},
    {(float)(9017.0 / 3168), (float)(-355.0 / 33), (float)(46732.0 / 5247), (float)(49.0 / 176),
     (float)(-5103.0 / 18656), 0},
    {(float)(35.0 / 384), 0.f, (float)(500.0 / 1113), (float)(125.0 / 192), (float)(-2187.0 / 6784),
     (float)(11.0 / 84)}};
__device__ __constant__ float kCErr[7] = {
    (float)(35.0 / 384 - 1951.0 / 21600), 0.f, (float)(500.0 / 1113 - 22642.0 / 50085),
    (float)(125.0 / 192 - 451.0 / 720), (float)(-2187.0 / 6784 + 12231.0 / 42400), (float)(11.0 / 84 - 649.0 / 6300),
    (float)(-1.0 / 60)};
__device__ __constant__ float kCMid[7] = {
    (float)(6025192743.0 / 30085553152.0 / 2), 0.f, (float)(51252292925.0 / 65400821598.0 / 2),
    (float)(-2691868925.0 / 45128329728.0 / 2), (float)(187940372067.0 / 1594534317056.0 / 2),
    (float)(-1776094331.0 / 19743644256.0 / 2), (float)(11237099.0 / 235043384.0 / 2)};

struct Dopri5Args {
    const float* packed;
    int M, S, total;
    const float* x0;
    const double* t;  // [Tg] device, float64 ("all time-like objects use float64")
    int Tg;
    int64_t B;
    double rtol, atol;
    float* xs;        // [Tg,B,D]
    float* work;      // y | f | y1 | f1 | ymid  (5 x [B,D])
    double* red;      // [3][kDpMaxGrid] per-CTA partial sums of the three rotating error norms
    int32_t* stats;   // nfe, accepted, rejected, status  (sets mode: 4 per set)
    // sets mode (batched Monte-Carlo prediction): CTA q integrates rows [q set_rows, (q+1) set_rows) with the packed
    // block at packed + q set_stride and ITS OWN controller (error norm over the set's rows, as if called per set)
    int64_t set_rows, set_stride;
    int max_attempts;
    // optional checkpoints of the ACCEPTED steps for the discrete adjoint (all NULL when not training)
    float* ck_y;      // [cap][B][D]    state at the start of accepted step n
    float* ck_k;      // [cap][7][B][D] the seven stage derivatives of accepted step n (as integrated: sign included)
    float* ck_dt;     // [cap]          float32 step size used by the stage algebra
    int32_t* out_step;  // [Tg] accepted-step index that produced output j (-1 for j = 0)
    float* out_x;     // [Tg] interpolation abscissa of output j inside its step
    int cap;
};

__device__ __forceinline__ double block_sum_to(double v, double* smem_red) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) smem_red[w] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += smem_red[i];
    return t;  // valid on thread 0
}

template <int D>
__device__ __forceinline__ void ldrow(float (&v)[1][D], const float* p, int64_t row) {
#pragma unroll
    for (int j = 0; j < D; ++j) v[0][j] = p[row * D + j];
}
template <int D>
__device__ __forceinline__ void strow(const float (&v)[1][D], float* p, int64_t row) {
#pragma unroll
    for (int j = 0; j < D; ++j) p[row * D + j] = v[0][j];
}

// kWarp: one WARP per row (lanes split the features / inducing points, xor-shuffle all-reduce) for small batches;
// otherwise one thread per row.
template <int D, bool kWarp>
__device__ __forceinline__ void vf_signed(const float* sp, int M, int S, float sgn, const float (&x)[1][D],
                                          float (&f)[1][D]) {
    if constexpr (kWarp) {
        vf_eval<D, 1, true>(sp, M, S, x, f, threadIdx.x & 31, 32);
#pragma unroll
        for (int j = 0; j < D; ++j) f[0][j] = (float)gpode_warp_sum_f64((double)f[0][j]) * sgn;
    } else {
        vf_eval<D, 1>(sp, M, S, x, f);
#pragma unroll
        for (int j = 0; j < D; ++j) f[0][j] *= sgn;
    }
}

template <int D, bool kWarp, bool kSets = false>
__global__ void __launch_bounds__(kSets ? kDpSetThreads : kDpThreads) dopri5_kernel(const Dopri5Args a) {
    static_assert(!kSets || kWarp, "sets mode is warp-per-row");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ double sred[kDpSetThreads / 32];
    __shared__ double sset[4];
    cg::grid_group grid = cg::this_grid();
    const float* sp = stage_params(smem_raw, a.packed + (kSets ? blockIdx.x * a.set_stride : 0), a.total);
    const int M = a.M, S = a.S;
    const int64_t B = a.B, plane = B * D;
    // gtid / gstride index ROWS: threads in the row-per-thread mode, warps in the warp-per-row mode (where every lane
    // of a warp carries the same row and only lane 0 stores and contributes to the error norm)
    const int64_t gtid = kSets ? (threadIdx.x >> 5)
                               : ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / (kWarp ? 32 : 1);
    const int64_t gstride = kSets ? (blockDim.x >> 5) : ((int64_t)gridDim.x * blockDim.x) / (kWarp ? 32 : 1);
    const int64_t row_begin = kSets ? blockIdx.x * a.set_rows : 0;
    const int64_t row_end = kSets ? row_begin + a.set_rows : B;
    int32_t* const stats = a.stats + (kSets ? 4 * blockIdx.x : 0);
    const bool writer = !kWarp || (threadIdx.x & 31) == 0;
    // the only cross-thread quantities: three sums of squares. Grid mode: every CTA writes its float64 partial sum to a
    // slot of its own and, after the grid barrier, warp 0 of every CTA adds the slots in a FIXED order (no atomics: the
    // norm, hence every accept / reject decision and step size, is bitwise reproducible); sets mode: the CTA is the
    // whole "batch", so shared memory + __syncthreads.
    auto publish = [&](double v, int slot) {
        const double b = block_sum_to(v, sred);
        if (threadIdx.x == 0) {
            if constexpr (kSets) sset[slot] = b;
            else a.red[(size_t)slot * kDpMaxGrid + blockIdx.x] = b;
        }
    };
    auto barrier = [&]() {
        if constexpr (kSets) __syncthreads();
        else grid.sync();
    };
    auto total_of = [&](int slot) -> double {
        if constexpr (kSets) {
            return sset[slot];
        } else {
            __syncthreads();   // sset[3] may still be read from the previous call
            if (threadIdx.x < 32) {
                const double* __restrict__ p = a.red + (size_t)slot * kDpMaxGrid;
                double v = 0.0;
                for (int i = threadIdx.x; i < (int)gridDim.x; i += 32) v += __ldcg(p + i);
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                if (threadIdx.x == 0) sset[3] = v;
            }
            __syncthreads();
            return sset[3];
        }
    };
    float* Y = a.work;
    float* F = a.work + plane;
    float* Y1 = a.work + 2 * plane;
    float* F1 = a.work + 3 * plane;
    float* YM = a.work + 4 * plane;
    const float rtol = (float)a.rtol, atol = (float)a.atol;
    const double n_elem = (double)(row_end - row_begin) * (double)D;
    // a decreasing grid is integrated as -f over -t, exactly what torchdiffeq's odeint does
    const double dir = (a.Tg > 1 && a.t[a.Tg - 1] < a.t[0]) ? -1.0 : 1.0;
    const float fsign = (float)dir;

    // ---- y = x0, f0 = f(t0, y0); d0, d1 of _select_initial_step ----
    double s0 = 0.0, s1 = 0.0;
    for (int64_t row = row_begin + gtid; row < row_end; row += gstride) {
        float y[1][D], f[1][D];
        ldrow<D>(y, a.x0, row);
        vf_signed<D, kWarp>(sp, M, S, fsign, y, f);
        if (writer) {
            strow<D>(y, Y, row);
            strow<D>(f, F, row);
            strow<D>(y, a.xs, row);
        }
#pragma unroll
        for (int j = 0; j < D; ++j) {
            const float sc = atol + fabsf(y[0][j]) * rtol;
            const float q0 = y[0][j] / sc, q1 = f[0][j] / sc;
            s0 += (double)(q0 * q0);
            s1 += (double)(q1 * q1);
        }
    }
    if (!writer) s0 = s1 = 0.0;  // warp-per-row mode: a row counts once
    publish(s0, 0);
    publish(s1, 1);
    barrier();
    const float d0 = (float)sqrt(total_of(0) / n_elem), d1 = (float)sqrt(total_of(1) / n_elem);
    float h0 = (d0 < 1e-5f || d1 < 1e-5f) ? 1e-6f : 0.01f * d0 / d1;
    double s2 = 0.0;
    for (int64_t row = row_begin + gtid; row < row_end; row += gstride) {
        float y[1][D], f[1][D], y1[1][D], f1[1][D];
        ldrow<D>(y, Y, row);
        ldrow<D>(f, F, row);
#pragma unroll
        for (int j = 0; j < D; ++j) y1[0][j] = y[0][j] + h0 * f[0][j];
        vf_signed<D, kWarp>(sp, M, S, fsign, y1, f1);
#pragma unroll
        for (int j = 0; j < D; ++j) {
            const float sc = atol + fabsf(y[0][j]) * rtol;
            const float q = (f1[0][j] - f[0][j]) / sc;
            s2 += (double)(q * q);
        }
    }
    if (!writer) s2 = 0.0;
    publish(s2, 2);
    barrier();
    double dt;
    {
        const float d2 = (float)sqrt(total_of(2) / n_elem) / h0;
        float h1;
        if (d1 <= 1e-15f && d2 <= 1e-15f) h1 = fmaxf(1e-6f, h0 * 1e-3f);
        else h1 = powf(0.01f / fmaxf(d1, d2), 1.0f / 5.0f);
        dt = (double)fminf(100.f * h0, h1);
    }
    barrier();  // everyone has read the three sums before their slots are recycled as the rotating error sums

    // ---- main loop: controller state replicated in every thread ----
    double t0 = dir * a.t[0], t1 = dir * a.t[0];
    int jout = 1, nfe = 2, n_acc = 0, n_rej = 0, status = 0;
    int attempt = 0;
    while (jout < a.Tg) {
        if (!(dir * a.t[jout] > t1)) {  // output time already covered by the last accepted step (handled at accept time)
            ++jout;
            continue;
        }
        if (attempt >= a.max_attempts || !(t1 + dt > t1)) {
            status = attempt >= a.max_attempts ? 1 : 2;  // too many attempts / step-size underflow
            break;
        }
        if (a.ck_k != nullptr && n_acc >= a.cap) {
            status = 3;  // checkpoint capacity exhausted: the caller retries with a larger one
            break;
        }
        const float dts = (float)dt;
        double se = 0.0;
        for (int64_t row = row_begin + gtid; row < row_end; row += gstride) {
            float y[1][D], k[7][1][D], yi[1][D];
            ldrow<D>(y, Y, row);
            ldrow<D>(k[0], F, row);
#pragma unroll
            for (int i = 0; i < 6; ++i) {
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    float s = 0.f;
#pragma unroll
                    for (int l = 0; l <= i; ++l) s = fmaf(k[l][0][j], __fmul_rn(kBeta[i][l], dts), s);
                    yi[0][j] = y[0][j] + s;
                }
                vf_signed<D, kWarp>(sp, M, S, fsign, yi, k[i + 1]);
            }
            float ym[1][D];
#pragma unroll
            for (int j = 0; j < D; ++j) {
                float e = 0.f, m = 0.f;
#pragma unroll
                for (int l = 0; l < 7; ++l) {
                    e = fmaf(k[l][0][j], __fmul_rn(dts, kCErr[l]), e);
                    m = fmaf(k[l][0][j], __fmul_rn(dts, kCMid[l]), m);
                }
                ym[0][j] = y[0][j] + m;
                const float tol = atol + rtol * fmaxf(fabsf(y[0][j]), fabsf(yi[0][j]));
                const float q = e / tol;
                se += (double)(q * q);
            }
            if (writer) {
                strow<D>(yi, Y1, row);
                strow<D>(k[6], F1, row);
                strow<D>(ym, YM, row);
            }
            if (writer && a.ck_k != nullptr && n_acc < a.cap) {  // slot n_acc is simply overwritten if this attempt is rejected
                strow<D>(y, a.ck_y + (int64_t)n_acc * plane, row);
#pragma unroll
                for (int l = 0; l < 7; ++l) strow<D>(k[l], a.ck_k + ((int64_t)n_acc * 7 + l) * plane, row);
            }
        }
        if (!writer) se = 0.0;
        publish(se, attempt % 3);
        barrier();
        const float ratio = (float)sqrt(total_of(attempt % 3) / n_elem);
        const bool accept = ratio <= 1.0f;
        nfe += 6;
        if (accept) {
            const double t1n = t1 + dt;
            // outputs that fall inside (t1, t1n]
            int jend = jout;
            while (jend < a.Tg && !(dir * a.t[jend] > t1n)) ++jend;
            for (int64_t row = row_begin + gtid; row < row_end; row += gstride) {
                float y[1][D], f[1][D], y1[1][D], f1[1][D], ym[1][D];
                ldrow<D>(y1, Y1, row);
                ldrow<D>(f1, F1, row);
                if (jend > jout) {
                    ldrow<D>(y, Y, row);
                    ldrow<D>(f, F, row);
                    ldrow<D>(ym, YM, row);
#pragma unroll
                    for (int j = 0; j < D; ++j) {
                        const float y0 = y[0][j], yn = y1[0][j], f0 = f[0][j], fn = f1[0][j], ymj = ym[0][j];
                        const float ca = 2 * dts * (fn - f0) - 8 * (yn + y0) + 16 * ymj;
                        const float cb = dts * (5 * f0 - 3 * fn) + 18 * y0 + 14 * yn - 32 * ymj;
                        const float cc = dts * (fn - 4 * f0) - 11 * y0 - 5 * yn + 16 * ymj;
                        const float cd = dts * f0;
                        for (int jo = jout; jo < jend; ++jo) {
                            const float x = (float)((dir * a.t[jo] - t1) / (t1n - t1));
                            if (a.out_x != nullptr && gtid == 0 && j == 0) {
                                a.out_step[jo] = n_acc;
                                a.out_x[jo] = x;
                            }
                            float total = y0 + x * cd;
                            float xp = x * x;
                            total = total + xp * cc;
                            xp = xp * x;
                            total = total + xp * cb;
                            xp = xp * x;
                            total = total + xp * ca;
                            if (writer) a.xs[(int64_t)jo * plane + row * D + j] = total;
                        }
                    }
                }
                // warp-per-row mode: every lane has read the old state before lane 0 overwrites it, and the next
                // attempt's loads see the new one (lanes of a warp are not guaranteed to run in lockstep)
                if constexpr (kWarp) __syncwarp();
                if (writer) {
                    strow<D>(y1, Y, row);
                    strow<D>(f1, F, row);
                }
                if constexpr (kWarp) __syncwarp();
            }
            if (a.ck_dt != nullptr && gtid == 0) a.ck_dt[n_acc] = dts;
            jout = jend;
            t0 = t1;
            t1 = t1n;
            ++n_acc;
        } else {
            ++n_rej;
        }
        // _optimal_step_size (safety 0.9, ifactor 10, dfactor 0.2, order 5)
        if (ratio == 0.f) {
            dt = dt * 10.0;
        } else {
            const double dfac = ratio < 1.f ? 1.0 : 0.2;
            const double fac = fmin(10.0, fmax(0.9 / pow((double)ratio, 0.2), dfac));
            dt = dt * fac;
        }
        ++attempt;
    }
    (void)t0;
    if (gtid == 0) {
        if (a.out_step != nullptr) a.out_step[0] = -1;
        stats[0] = nfe;
        stats[1] = n_acc;
        stats[2] = n_rej;
        stats[3] = status;
    }
}

}  // namespace

// checkpoint block layout documented at gpode_dopri5_ckpt_floats
inline void dopri5_set_ckpt(Dopri5Args& a, float* ckpt, int cap, int64_t plane, int Tg) {
    a.ck_y = a.ck_k = a.ck_dt = a.out_x = nullptr;
    a.out_step = nullptr;
    a.cap = 0;
    if (ckpt != nullptr && cap > 0) {
        a.cap = cap;
        a.ck_y = ckpt;
        a.ck_k = a.ck_y + (int64_t)cap * plane;
        a.ck_dt = a.ck_k + (int64_t)cap * 7 * plane;
        a.out_x = a.ck_dt + cap;
        a.out_step = reinterpret_cast<int32_t*>(a.out_x + Tg);
    }
}

template <int D>
int launch_dopri5_sets(const float* packed, int M, int S, int n_sets, int64_t set_rows, const float* x0,
                       const double* t, int Tg, double rtol, double atol, float* xs, float* work, int32_t* stats,
                       cudaStream_t st, float* ckpt = nullptr, int cap = 0);

// a batch this small is one "set": a single CTA (one warp per row, __syncthreads instead of the grid barrier) runs the
// whole solve -- the reference's own plain-GPODE shapes (N = 1 / 6 trajectories)
constexpr int64_t kDpOneCtaRows = 16;
// dopri5_kernel's own __shared__ arrays (sred, sset): they count against the 227 KB next to the packed block
constexpr size_t kDpStaticSmem = sizeof(double) * (kDpSetThreads / 32 + 4);

template <int D>
int launch_dopri5(const float* packed, int M, int S, const float* x0, const double* t, int Tg, int64_t B, double rtol,
                  double atol, float* xs, float* work, int32_t* stats, float* ckpt, int cap, cudaStream_t st) {
    if (B <= kDpOneCtaRows)
        return launch_dopri5_sets<D>(packed, M, S, 1, B, x0, t, Tg, rtol, atol, xs, work, stats, st, ckpt, cap);
    const GpodeLayout L = gpode_layout(D, M, S);
    const size_t smem = 16 + (size_t)L.total * 4;
    // small batches: one warp per row (the reference's N = 1 / 6 trajectories, a few thousand shooting segments)
    const bool warp_mode = B <= 1024;
    const void* kern = warp_mode ? (const void*)dopri5_kernel<D, true> : (const void*)dopri5_kernel<D, false>;
    if (int rc = check_smem_fits(smem, kDpStaticSmem)) return rc;
    GPODE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0, sms = 148, dev = 0;
    GPODE_CUDA(cudaGetDevice(&dev));
    GPODE_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    if (warp_mode) {
        GPODE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, dopri5_kernel<D, true>, kDpThreads, smem));
    } else {
        GPODE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, dopri5_kernel<D, false>, kDpThreads, smem));
    }
    if (occ < 1) {
        gpode_set_error("dopri5 kernel does not fit on an SM (smem %zu bytes)", smem);
        return -2;
    }
    const int64_t rows_per_cta = warp_mode ? kDpThreads / 32 : kDpThreads;
    const int64_t want = (B + rows_per_cta - 1) / rows_per_cta;
    const int64_t grid_cap = (int64_t)sms * occ;
    int grid = (int)(want < grid_cap ? want : grid_cap);
    if (grid > kDpMaxGrid) grid = kDpMaxGrid;   // one float64 slot per CTA and rotating sum
    Dopri5Args a;
    a.packed = packed; a.M = M; a.S = S; a.total = L.total; a.x0 = x0; a.t = t; a.Tg = Tg; a.B = B;
    a.rtol = rtol; a.atol = atol; a.xs = xs;
    const int64_t plane = B * D;
    a.work = work;
    a.red = reinterpret_cast<double*>(work + 5 * plane + ((5 * plane) & 1));
    a.stats = stats;
    a.set_rows = 0;
    a.set_stride = 0;
    a.max_attempts = 1 << 20;
    dopri5_set_ckpt(a, ckpt, cap, plane, Tg);
    void* params[] = {(void*)&a};
    GPODE_CUDA(cudaLaunchCooperativeKernel(kern, dim3(grid), dim3(kDpThreads), params, smem, st));
    return 0;
}

// Batched Monte-Carlo prediction (no checkpoints): one CTA per parameter set, plain launch (no grid barrier needed).
template <int D>
int launch_dopri5_sets(const float* packed, int M, int S, int n_sets, int64_t set_rows, const float* x0,
                       const double* t, int Tg, double rtol, double atol, float* xs, float* work, int32_t* stats,
                       cudaStream_t st, float* ckpt, int cap) {
    const GpodeLayout L = gpode_layout(D, M, S);
    const size_t smem = 16 + (size_t)L.total * 4;
    int warps = (int)(set_rows < kDpSetThreads / 32 ? set_rows : kDpSetThreads / 32);
    if (warps < 1) warps = 1;
    if (int rc = check_smem_fits(smem, kDpStaticSmem)) return rc;
    GPODE_CUDA(cudaFuncSetAttribute(dopri5_kernel<D, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    GPODE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, dopri5_kernel<D, true, true>, warps * 32, smem));
    if (occ < 1) {
        gpode_set_error("dopri5 kernel does not fit on an SM (smem %zu bytes)", smem);
        return -2;
    }
    Dopri5Args a;
    a.packed = packed; a.M = M; a.S = S; a.total = L.total; a.x0 = x0; a.t = t; a.Tg = Tg;
    a.B = set_rows * n_sets;
    a.rtol = rtol; a.atol = atol; a.xs = xs;
    a.work = work;
    a.red = nullptr;
    a.stats = stats;
    a.set_rows = set_rows;
    a.set_stride = L.n_packed;
    a.max_attempts = 1 << 20;
    dopri5_set_ckpt(a, n_sets == 1 ? ckpt : nullptr, cap, a.B * D, Tg);  // checkpoints: single-set (training) use only
    dopri5_kernel<D, true, true><<<n_sets, warps * 32, smem, st>>>(a);
    GPODE_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------------------------------------
// Discrete adjoint of the accepted steps (step sizes are constants, exactly as torchdiffeq computes them under
// no_grad): walking the accepted steps backwards, each is an explicit 7-stage RK step
//     Y_i = y0 + dt sum_{l<i} beta_il k_l,  k_i = f(Y_i),  y1 = Y_7,  y_mid = y0 + dt sum c_mid_l k_l,  f1 = k_7 (FSAL)
// and every requested output inside it is the quartic through (y0, y_mid, y1, f0, f1). Warp-per-row mapping (lanes
// split features / inducing points), so it serves the small training batches dopri5 is used with.
// ------------------------------------------------------------------------------------------------------------------
struct Dopri5BwdArgs {
    const float* packed;
    int M, S, total;
    const double* t;
    int Tg;
    int64_t B;
    const float* gxs;     // [Tg,B,D]
    const float* ckpt;    // forward checkpoints
    int cap, n_acc;
    const int32_t* stats_dev;  // optional: the forward's stats block; n_acc is then read on the device (stats[1]) so
                               // that no host round trip sits between forward and backward (CUDA-graph capture)
    float* gx0;           // [B,D]
    float* vy;            // virtual rows: stage inputs  [(6 n_acc + 1)][B][D]
    float* vk;            //               cotangents
    float* acc;
};

template <int D>
__global__ void __launch_bounds__(kDpThreads) dopri5_bwd_kernel(const Dopri5BwdArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const float* sp = stage_params(smem_raw, a.packed, a.total);
    double* slabs = reinterpret_cast<double*>(reinterpret_cast<float*>(smem_raw + 16) + a.total);
    WarpAcc64<D> wa;
    wa.init(slabs);
    const int M = a.M, S = a.S, Tg = a.Tg, cap = a.cap;
    const int n_acc = a.stats_dev != nullptr ? min(a.stats_dev[1], cap) : a.n_acc;
    const int64_t B = a.B, plane = B * D;
    const float* ck_y = a.ckpt;
    const float* ck_k = ck_y + (int64_t)cap * plane;
    const float* ck_dt = ck_k + (int64_t)cap * 7 * plane;
    const float* out_x = ck_dt + cap;
    const int32_t* out_step = reinterpret_cast<const int32_t*>(out_x + Tg);
    const float fsign = (Tg > 1 && a.t[Tg - 1] < a.t[0]) ? -1.f : 1.f;
    const int lane = threadIdx.x & 31, wpc = blockDim.x >> 5;

    for (int64_t row = (int64_t)blockIdx.x * wpc + (threadIdx.x >> 5); row < B; row += (int64_t)gridDim.x * wpc) {
        float lam[D], kap[D];  // adjoints of y (end of the current step) and of f1 = k7
#pragma unroll
        for (int j = 0; j < D; ++j) lam[j] = kap[j] = 0.f;
        int jo = Tg - 1;
        for (int n = n_acc - 1; n >= 0; --n) {
            const float dt = ck_dt[n];
            float y0[1][D], k[7][1][D];
            ldrow<D>(y0, ck_y + (int64_t)n * plane, row);
#pragma unroll
            for (int l = 0; l < 7; ++l) ldrow<D>(k[l], ck_k + ((int64_t)n * 7 + l) * plane, row);
            // cotangents of the outputs interpolated inside this step
            float yb0[D], yb1[D], ybm[D], fb0[D], fb1[D];
#pragma unroll
            for (int j = 0; j < D; ++j) {
                yb0[j] = 0.f; yb1[j] = lam[j]; ybm[j] = 0.f; fb0[j] = 0.f; fb1[j] = kap[j];
            }
            while (jo >= 1 && out_step[jo] == n) {
                const float x = out_x[jo], x2 = x * x, x3 = x2 * x, x4 = x2 * x2;
                const float p0 = 1.f - 11.f * x2 + 18.f * x3 - 8.f * x4;
                const float p1 = -5.f * x2 + 14.f * x3 - 8.f * x4;
                const float pm = 16.f * x2 - 32.f * x3 + 16.f * x4;
                const float q0 = dt * (x - 4.f * x2 + 5.f * x3 - 2.f * x4);
                const float q1 = dt * (x2 - 3.f * x3 + 2.f * x4);
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    const float g = __ldg(a.gxs + (int64_t)jo * plane + row * D + j);
                    yb0[j] = fmaf(g, p0, yb0[j]);
                    yb1[j] = fmaf(g, p1, yb1[j]);
                    ybm[j] = fmaf(g, pm, ybm[j]);
                    fb0[j] = fmaf(g, q0, fb0[j]);
                    fb1[j] = fmaf(g, q1, fb1[j]);
                }
                --jo;
            }
            float kb[7][D];
#pragma unroll
            for (int l = 0; l < 7; ++l)
#pragma unroll
                for (int j = 0; j < D; ++j)
                    kb[l][j] = (l < 6 ? __fmul_rn(kBeta[5][l], dt) * yb1[j] : 0.f) + __fmul_rn(dt, kCMid[l]) * ybm[j];
#pragma unroll
            for (int j = 0; j < D; ++j) {
                kb[6][j] += fb1[j];
                kb[0][j] += fb0[j];
                yb0[j] += yb1[j] + ybm[j];
            }
            // stages 7 .. 2
#pragma unroll
            for (int i = 6; i >= 1; --i) {
                float Yi[1][D], kbi[1][D], fst[1][D], Yb[1][D];
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    float s = 0.f;
#pragma unroll
                    for (int l = 0; l < i; ++l) s = fmaf(k[l][0][j], __fmul_rn(kBeta[i - 1][l], dt), s);
                    Yi[0][j] = y0[0][j] + s;
                    kbi[0][j] = fsign * kb[i][j];   // cotangent of f(Y_i); the integrated k is fsign * f
                    fst[0][j] = fsign * k[i][0][j];
                }
                const int64_t slot = (int64_t)n * 6 + (i - 1);
                if (lane == 0) {
                    strow<D>(Yi, a.vy + slot * plane, row);
                    strow<D>(kbi, a.vk + slot * plane, row);
                }
                vf_vjp_warp<D>(sp, M, S, Yi, kbi, fst, Yb, wa, lane);
#pragma unroll
                for (int j = 0; j < D; ++j) yb0[j] += Yb[0][j];
#pragma unroll
                for (int l = 0; l < i; ++l)
#pragma unroll
                    for (int j = 0; j < D; ++j) kb[l][j] = fmaf(__fmul_rn(kBeta[i - 1][l], dt), Yb[0][j], kb[l][j]);
            }
            if (n > 0) {
#pragma unroll
                for (int j = 0; j < D; ++j) kap[j] = kb[0][j];  // k1 of this step is k7 of the previous one (FSAL)
            } else {
                float kbi[1][D], fst[1][D], Yb[1][D];
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    kbi[0][j] = fsign * kb[0][j];
                    fst[0][j] = fsign * k[0][0][j];
                }
                const int64_t slot = (int64_t)n_acc * 6;
                if (lane == 0) {
                    strow<D>(y0, a.vy + slot * plane, row);
                    strow<D>(kbi, a.vk + slot * plane, row);
                }
                vf_vjp_warp<D>(sp, M, S, y0, kbi, fst, Yb, wa, lane);
#pragma unroll
                for (int j = 0; j < D; ++j) yb0[j] += Yb[0][j];
            }
#pragma unroll
            for (int j = 0; j < D; ++j) lam[j] = yb0[j];
        }
        if (lane == 0) {
#pragma unroll
            for (int j = 0; j < D; ++j) {
                float g = lam[j] + __ldg(a.gxs + row * D + j);  // output 0 is y0 itself
                // outputs that were never reached by a step (status != 0) cannot occur for a successful forward
                a.gx0[row * D + j] = g;
            }
        }
    }
    __syncthreads();
    reduce_AV64<D>(wa, a.acc, slabs + (kDpThreads / 32) * WarpAcc64<D>::kSlabDoubles);
}

template <int D>
int launch_dopri5_bwd(const float* packed, int M, int S, const double* t, int Tg, int64_t B, const float* gxs,
                      const float* ckpt, int cap, int n_acc, const int32_t* stats_dev, float* gx0, float* vrows,
                      float* acc, cudaStream_t st) {
    const GpodeLayout L = gpode_layout(D, M, S);
    const size_t smem = 16 + (size_t)L.total * 4 + (size_t)kWarpAccDoubles<D>(kDpThreads / 32) * 8;
    if (int rc = check_smem_fits(smem)) return rc;
    GPODE_CUDA(cudaFuncSetAttribute(dopri5_bwd_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0, sms = 148, dev = 0;
    GPODE_CUDA(cudaGetDevice(&dev));
    GPODE_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    GPODE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, dopri5_bwd_kernel<D>, kDpThreads, smem));
    if (occ < 1) {
        gpode_set_error("dopri5 backward kernel does not fit on an SM (smem %zu bytes)", smem);
        return -2;
    }
    const int wpc = kDpThreads / 32;
    const int64_t want = (B + wpc - 1) / wpc;
    int64_t cap_grid = (int64_t)sms * occ;
    if (cap_grid > GPODE_ACC_CAP_AV) cap_grid = GPODE_ACC_CAP_AV;  // one accumulator row per CTA
    Dopri5BwdArgs a;
    a.packed = packed; a.M = M; a.S = S; a.total = L.total; a.t = t; a.Tg = Tg; a.B = B; a.gxs = gxs; a.ckpt = ckpt;
    a.cap = cap; a.n_acc = n_acc; a.stats_dev = stats_dev; a.gx0 = gx0;
    // cotangent rows start after the stage-input rows: exact count, or the capacity when the count lives on the device
    const int64_t VR = ((int64_t)6 * (stats_dev != nullptr ? cap : n_acc) + 1) * B;
    a.vy = vrows;
    a.vk = vrows + VR * D;
    a.acc = acc;
    dopri5_bwd_kernel<D><<<(unsigned)(want < cap_grid ? want : cap_grid), kDpThreads, smem, st>>>(a);
    GPODE_LAUNCH_CHECK();
    return 0;
}
