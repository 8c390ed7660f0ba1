// Adaptive dopri5 for 8 < D <= 64 with the controller ON THE DEVICE, and its discrete adjoint.
//
// torchdiffeq 0.2.0's dopri5 as called by Flow.forward (reference src/core/flow.py:84-90; restated in
// oracle/torchdiffeq_shim): Dormand-Prince 5(4), FSAL, whole-batch RMS error norm, float64 time, Hairer initial step,
// quartic dense output. The reference synchronises the host once per attempt (accept / reject is a Python `if`); round 1
// of this library did the same at these state dimensions (an eager host loop around the tiled vector-field kernel).
// Here one attempt is a short chain of launches -- six stage evaluations on the tcgen05 vector-field kernels
// (large_umma.cu), element-wise stage / error kernels, a one-CTA controller kernel that decides accept / reject, updates
// (t, dt) in float64 and names the outputs to interpolate, and an element-wise accept kernel -- and the chain is the body
// of a CUDA-graph WHILE node whose condition the controller kernel sets with cudaGraphSetConditional: the loop runs on
// the device until the last output time is covered, the host enqueues one graph launch and never reads a value.
// Arithmetic (operation order, float32 state, float64 time) follows dopri5_impl.cuh, which serves D <= 8.
//
// Training: the accept kernel can also record every accepted step (state at its start, the seven raw stage values, the
// float32 step size, and which step / abscissa produced each output) in the checkpoint block of
// gpode_dopri5_ckpt_floats. gpode_dopri5_bwd_large walks those steps backwards -- the algorithm of
// dopri5_impl.cuh::dopri5_bwd_kernel as a stream-ordered chain of launches around the large-D VJP (large_bwd.cu), the
// way gpode_rk4_bwd_large restates rk4_bwd_kernel. Step sizes are constants there, as in torchdiffeq, whose controller
// runs on a detached error ratio, so the two initial-step evaluations get no cotangent.
#include "common.cuh"
#include "../../include/gpode_b200.h"
#include <cstddef>
#include <deque>
#include <mutex>

int gpode_vf_large_eval(const float* packed_large, const gpode_cache_t* c, const float* x, float* tmp, float* f,
                        const GpodeDraws& dr, cudaStream_t st);  // large_umma.cu

namespace {

__device__ __constant__ float ldBeta[6][6] = {
    {1.f / 5, 0, 0, 0, 0, 0},
    {3.f / 40, 9.f / 40, 0, 0, 0, 0},
    {44.f / 45, -56.f / 15, 32.f / 9, 0, 0, 0},
    {(float)(19372.0 / 6561), (float)(-25360.0 / 2187), (float)(64448.0 / 6561), (float)(-212.0 / 729), 0, 0},
    {(float)(9017.0 / 3168), (float)(-355.0 / 33), (float)(46732.0 / 5247), (float)(49.0 / 176),
     (float)(-5103.0 / 18656), 0},
    {(float)(35.0 / 384), 0.f, (float)(500.0 / 1113), (float)(125.0 / 192), (float)(-2187.0 / 6784),
     (float)(11.0 / 84)}};
__device__ __constant__ float ldCErr[7] = {
    (float)(35.0 / 384 - 1951.0 / 21600), 0.f, (float)(500.0 / 1113 - 22642.0 / 50085),
    (float)(125.0 / 192 - 451.0 / 720), (float)(-2187.0 / 6784 + 12231.0 / 42400), (float)(11.0 / 84 - 649.0 / 6300),
    (float)(-1.0 / 60)};
__device__ __constant__ float ldCMid[7] = {
    (float)(6025192743.0 / 30085553152.0 / 2), 0.f, (float)(51252292925.0 / 65400821598.0 / 2),
    (float)(-2691868925.0 / 45128329728.0 / 2), (float)(187940372067.0 / 1594534317056.0 / 2),
    (float)(-1776094331.0 / 19743644256.0 / 2), (float)(11237099.0 / 235043384.0 / 2)};

struct LdCtrl {
    double t1, dt, dir;        // current time (already multiplied by dir), step size, +1 / -1
    double t1_used, t1n_used;  // the interval of the attempt just decided (for the accept kernel)
    float dts_used, h0, d1;
    int jout, jlo, jhi, accept, done;
    int nfe, n_acc, n_rej, status, attempt, max_attempts;
    int cap;                   // checkpoint capacity in accepted steps; 0: no checkpoints
};

// checkpoint block (layout of gpode_dopri5_ckpt_floats): y [cap][B][D] | k [cap][7][B][D] | dt [cap] | out_x [Tg] |
// out_step [Tg]. k holds the RAW vector-field values (the direction sign is applied where they are used).
struct LdCkpt {
    float* y;
    float* k;
    float* dt;
    float* out_x;
    int32_t* out_step;
};

LdCkpt ld_ckpt(float* ckpt, int cap, int64_t n, int Tg) {
    LdCkpt k;
    k.y = ckpt;
    k.k = ckpt ? ckpt + (int64_t)cap * n : nullptr;
    k.dt = ckpt ? k.k + (int64_t)cap * 7 * n : nullptr;
    k.out_x = ckpt ? k.dt + cap : nullptr;
    k.out_step = ckpt ? reinterpret_cast<int32_t*>(k.out_x + Tg) : nullptr;
    return k;
}

constexpr int kLdThreads = 256;
constexpr int kLdMaxBlocks = 2368;

inline unsigned ld_grid(int64_t n) {
    const int64_t g = (n + kLdThreads - 1) / kLdThreads;
    return (unsigned)(g < kLdMaxBlocks ? (g < 1 ? 1 : g) : kLdMaxBlocks);
}

// block sum of up to two float64 values -> partial[blockIdx.x (+ gridDim.x)]
__device__ __forceinline__ void ld_block_sums(double a, double b, double* __restrict__ partial, const bool two) {
    __shared__ double sa[kLdThreads / 32], sb[kLdThreads / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if ((threadIdx.x & 31) == 0) {
        sa[threadIdx.x >> 5] = a;
        sb[threadIdx.x >> 5] = b;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ta = 0.0, tb = 0.0;
        for (int i = 0; i < kLdThreads / 32; ++i) {
            ta += sa[i];
            tb += sb[i];
        }
        partial[blockIdx.x] = ta;
        if (two) partial[gridDim.x + blockIdx.x] = tb;
    }
}

// fixed-order sum of n partials by one CTA (thread-strided, then warps and lanes in index order)
__device__ double ld_total(const double* __restrict__ partial, const int n) {
    __shared__ double s[kLdThreads];
    double a = 0.0;
    for (int i = threadIdx.x; i < n; i += kLdThreads) a += partial[i];
    s[threadIdx.x] = a;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int i = 0; i < kLdThreads; ++i) t += s[i];
    __syncthreads();
    if (threadIdx.x == 0) s[0] = t;
    __syncthreads();
    t = s[0];
    __syncthreads();
    return t;
}

// +1 / -1: a decreasing grid is integrated as -f over -t
__device__ __forceinline__ double ld_dir(const double* __restrict__ t, const int Tg) {
    return (Tg > 1 && t[Tg - 1] < t[0]) ? -1.0 : 1.0;
}

// Batched prediction (n_sets draws, gpode_dopri5_fwd_large_sets): one LdCtrl per draw. The kernels with one CTA per
// draw index it by blockIdx.x; the element-wise kernels run on a (blocks, draws) grid, see the offsets of draw
// blockIdx.y into every [n_sets][n] buffer, and sum into their draw's slice of 2 gridDim.x partials.
__global__ void ld_start_kernel(LdCtrl* c, const double* __restrict__ t, const int Tg, const int max_attempts,
                                const int cap, int32_t* __restrict__ out_step) {
    c += blockIdx.x;
    const double dir = ld_dir(t, Tg);
    c->dir = dir;
    c->t1 = dir * t[0];
    c->dt = 0.0;
    c->jout = 1; c->jlo = c->jhi = 0; c->accept = 0; c->done = Tg <= 1;
    c->nfe = 2; c->n_acc = 0; c->n_rej = 0; c->status = 0; c->attempt = 0; c->max_attempts = max_attempts;
    c->cap = cap;
    if (out_step != nullptr)   // outputs no accepted step produces (output 0, or a failed solve) stay -1
        for (int j = 0; j < Tg; ++j) out_step[j] = -1;
}

// s0 = sum (y / sc)^2, s1 = sum (f / sc)^2, sc = atol + |y| rtol
__global__ void __launch_bounds__(kLdThreads)
ld_norm01_kernel(const float* __restrict__ y, const float* __restrict__ f, const float rtol, const float atol,
                 const int64_t n, double* __restrict__ partial) {
    y += blockIdx.y * n;
    f += blockIdx.y * n;
    double s0 = 0.0, s1 = 0.0;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const float sc = atol + fabsf(y[e]) * rtol;
        const float q0 = y[e] / sc, q1 = f[e] / sc;
        s0 += (double)(q0 * q0);
        s1 += (double)(q1 * q1);
    }
    ld_block_sums(s0, s1, partial + (size_t)blockIdx.y * 2 * gridDim.x, true);
}

__global__ void __launch_bounds__(kLdThreads)
ld_init1_kernel(LdCtrl* c, const double* __restrict__ partial, const int nb, const double n_elem) {
    c += blockIdx.x;
    partial += (size_t)blockIdx.x * 2 * nb;
    const double t0 = ld_total(partial, nb), t1 = ld_total(partial + nb, nb);
    if (threadIdx.x == 0) {
        const float d0 = (float)sqrt(t0 / n_elem), d1 = (float)sqrt(t1 / n_elem);
        c->h0 = (d0 < 1e-5f || d1 < 1e-5f) ? 1e-6f : 0.01f * d0 / d1;
        c->d1 = d1;
    }
}

// out = y + h0 * fsign * f
__global__ void ld_euler_kernel(const LdCtrl* __restrict__ c, const float* __restrict__ y, const float* __restrict__ f,
                                float* __restrict__ out, const int64_t n) {
    c += blockIdx.y;
    y += blockIdx.y * n;
    f += blockIdx.y * n;
    out += blockIdx.y * n;
    const float h0 = c->h0, fs = (float)c->dir;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x)
        out[e] = y[e] + h0 * (fs * f[e]);
}

__global__ void __launch_bounds__(kLdThreads)
ld_norm2_kernel(const float* __restrict__ y, const float* __restrict__ f0, const float* __restrict__ f1, const float rtol,
                const float atol, const int64_t n, double* __restrict__ partial) {
    y += blockIdx.y * n;
    f0 += blockIdx.y * n;
    f1 += blockIdx.y * n;
    partial += (size_t)blockIdx.y * 2 * gridDim.x;
    double s2 = 0.0;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const float sc = atol + fabsf(y[e]) * rtol;
        const float q = (f1[e] - f0[e]) / sc;   // the direction sign cancels in the square
        s2 += (double)(q * q);
    }
    ld_block_sums(s2, 0.0, partial, false);
}

// the part of the controller that decides whether another attempt is needed (top of torchdiffeq's while loop)
__device__ void ld_loop_head(LdCtrl* c, const double* __restrict__ t, const int Tg) {
    while (c->jout < Tg && !(c->dir * t[c->jout] > c->t1)) ++c->jout;
    if (c->jout >= Tg) {
        c->done = 1;
    } else if (c->attempt >= c->max_attempts || !(c->t1 + c->dt > c->t1)) {
        c->status = c->attempt >= c->max_attempts ? 1 : 2;   // attempt limit / step-size underflow
        c->done = 1;
    } else if (c->cap > 0 && c->n_acc >= c->cap) {
        c->status = 3;   // checkpoint capacity exhausted: the caller retries with a larger one
        c->done = 1;
    }
}

__global__ void __launch_bounds__(kLdThreads)
ld_init2_kernel(LdCtrl* c, const double* __restrict__ partial, const int nb, const double n_elem,
                const double* __restrict__ t, const int Tg) {
    c += blockIdx.x;
    partial += (size_t)blockIdx.x * 2 * nb;
    const double t2 = ld_total(partial, nb);
    if (threadIdx.x == 0) {
        const float h0 = c->h0, d1 = c->d1;
        const float d2 = (float)sqrt(t2 / n_elem) / h0;
        float h1;
        if (d1 <= 1e-15f && d2 <= 1e-15f) h1 = fmaxf(1e-6f, h0 * 1e-3f);
        else h1 = powf(0.01f / fmaxf(d1, d2), 1.0f / 5.0f);
        c->dt = (double)fminf(100.f * h0, h1);
        if (!c->done) ld_loop_head(c, t, Tg);
    }
}

struct LdBufs {
    float* Y;      // current state
    float* K[7];   // raw vector-field values of the attempt's stages; K[0] = f(Y) (FSAL)
    float* Ys;     // stage input
    float* Y1;     // 7th stage input = the proposed state
    float* YM;     // dense-output midpoint
    float* tmp;    // scratch of the vector-field evaluation
};

// stage input i (1..6) at element e: Y_i = Y + sum_{l < i} (fsign K_l) (beta_{i-1,l} dt), bd[l] = beta_{i-1,l} dt.
// The forward and the backward both evaluate it here, so the adjoint linearises at bit-identical stage inputs.
__device__ __forceinline__ void ld_stage_coefs(const int i, const float dts, float (&bd)[6]) {
#pragma unroll
    for (int l = 0; l < 6; ++l) bd[l] = __fmul_rn(ldBeta[i - 1][l], dts);
}
__device__ __forceinline__ float ld_stage_input(const LdBufs& b, const int i, const float (&bd)[6], const float fs,
                                                const int64_t e) {
    float s = 0.f;
#pragma unroll
    for (int l = 0; l < 6; ++l)
        if (l < i) s = fmaf(fs * b.K[l][e], bd[l], s);
    return b.Y[e] + s;
}

// the buffers of draw q: every [n_sets][n] buffer advanced by q n
__device__ __forceinline__ LdBufs ld_bufs_at(LdBufs b, const int64_t o) {
    b.Y += o;
#pragma unroll
    for (int l = 0; l < 7; ++l) b.K[l] += o;
    b.Ys += o;
    b.Y1 += o;
    b.YM += o;
    b.tmp += o;
    return b;
}

__global__ void ld_stage_kernel(const LdCtrl* __restrict__ c, const int i, LdBufs b, float* __restrict__ out,
                                const int64_t n) {
    c += blockIdx.y;
    if (c->done) return;
    b = ld_bufs_at(b, blockIdx.y * n);
    out += blockIdx.y * n;
    const float fs = (float)c->dir;
    float bd[6];
    ld_stage_coefs(i, (float)c->dt, bd);
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x)
        out[e] = ld_stage_input(b, i, bd, fs, e);
}

__global__ void __launch_bounds__(kLdThreads)
ld_err_kernel(const LdCtrl* __restrict__ c, LdBufs b, const float rtol, const float atol, const int64_t n,
              double* __restrict__ partial) {
    c += blockIdx.y;
    if (c->done) return;   // the controller does not read the partial sums of a finished draw
    b = ld_bufs_at(b, blockIdx.y * n);
    partial += (size_t)blockIdx.y * 2 * gridDim.x;
    double se = 0.0;
    const float dts = (float)c->dt, fs = (float)c->dir;
    float ce[7], cm[7];
#pragma unroll
    for (int l = 0; l < 7; ++l) {
        ce[l] = __fmul_rn(dts, ldCErr[l]);
        cm[l] = __fmul_rn(dts, ldCMid[l]);
    }
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        float er = 0.f, m = 0.f;
#pragma unroll
        for (int l = 0; l < 7; ++l) {
            const float k = fs * b.K[l][e];
            er = fmaf(k, ce[l], er);
            m = fmaf(k, cm[l], m);
        }
        const float y = b.Y[e];
        b.YM[e] = y + m;
        const float tol = atol + rtol * fmaxf(fabsf(y), fabsf(b.Y1[e]));
        const float q = er / tol;
        se += (double)(q * q);
    }
    ld_block_sums(se, 0.0, partial, false);
}

// accept / reject, step-size update (_optimal_step_size: safety 0.9, ifactor 10, dfactor 0.2, order 5), loop condition
__global__ void __launch_bounds__(kLdThreads)
ld_ctrl_kernel(LdCtrl* c, const double* __restrict__ partial, const int nb, const double n_elem,
               const double* __restrict__ t, const int Tg, const cudaGraphConditionalHandle handle, const int set_cond) {
    c += blockIdx.x;
    partial += (size_t)blockIdx.x * 2 * nb;
    const double tot = ld_total(partial, nb);
    if (threadIdx.x != 0) return;
    if (!c->done) {
        const float ratio = (float)sqrt(tot / n_elem);
        const bool accept = ratio <= 1.0f;
        c->nfe += 6;
        c->accept = accept ? 1 : 0;
        c->dts_used = (float)c->dt;
        if (accept) {
            const double t1n = c->t1 + c->dt;
            int jend = c->jout;
            while (jend < Tg && !(c->dir * t[jend] > t1n)) ++jend;
            c->jlo = c->jout;
            c->jhi = jend;
            c->t1_used = c->t1;
            c->t1n_used = t1n;
            c->jout = jend;
            c->t1 = t1n;
            ++c->n_acc;
        } else {
            ++c->n_rej;
        }
        if (ratio == 0.f) {
            c->dt = c->dt * 10.0;
        } else {
            const double dfac = ratio < 1.f ? 1.0 : 0.2;
            c->dt = c->dt * fmin(10.0, fmax(0.9 / pow((double)ratio, 0.2), dfac));
        }
        ++c->attempt;
        ld_loop_head(c, t, Tg);
    } else {
        c->accept = 0;
    }
    if (set_cond) cudaGraphSetConditional(handle, c->done ? 0u : 1u);
}

// several draws: the loop goes on while any draw is not done
__global__ void __launch_bounds__(kLdThreads)
ld_any_kernel(const LdCtrl* __restrict__ c, const int n_sets, const cudaGraphConditionalHandle handle) {
    __shared__ int any;
    if (threadIdx.x == 0) any = 0;
    __syncthreads();
    for (int q = threadIdx.x; q < n_sets; q += kLdThreads)
        if (!c[q].done) any = 1;
    __syncthreads();
    if (threadIdx.x == 0) cudaGraphSetConditional(handle, any ? 1u : 0u);
}

// accepted step: dense output at the requested times inside it, then Y <- Y1, K0 <- K6 (FSAL). With checkpoints
// (ck.y != NULL) the step's start state, its seven stage values, dt and its outputs' step / abscissa go to slot n_acc-1.
__global__ void ld_accept_kernel(const LdCtrl* __restrict__ c, LdBufs b, const double* __restrict__ t,
                                 float* __restrict__ xs, const int64_t n, const LdCkpt ck) {
    c += blockIdx.y;
    if (!c->accept) return;
    b = ld_bufs_at(b, blockIdx.y * n);
    xs += blockIdx.y * n;
    const int64_t xs_stride = n * gridDim.y;   // xs [Tg][n_sets][n]
    const float dts = c->dts_used, fs = (float)c->dir;
    const int jlo = c->jlo, jhi = c->jhi;
    const double t1 = c->t1_used, t1n = c->t1n_used, dir = c->dir;
    const int64_t slot = (int64_t)c->n_acc - 1;
    if (ck.y != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {
        ck.dt[slot] = dts;
        for (int jo = jlo; jo < jhi; ++jo) {
            ck.out_step[jo] = (int32_t)slot;
            ck.out_x[jo] = (float)((dir * t[jo] - t1) / (t1n - t1));
        }
    }
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        if (ck.y != nullptr) {
            ck.y[slot * n + e] = b.Y[e];
#pragma unroll
            for (int l = 0; l < 7; ++l) ck.k[(slot * 7 + l) * n + e] = b.K[l][e];
        }
        const float yn = b.Y1[e], kn = b.K[6][e];
        if (jhi > jlo) {
            const float y0 = b.Y[e], f0 = fs * b.K[0][e], fn = fs * kn, ymj = b.YM[e];
            const float ca = 2 * dts * (fn - f0) - 8 * (yn + y0) + 16 * ymj;
            const float cb = dts * (5 * f0 - 3 * fn) + 18 * y0 + 14 * yn - 32 * ymj;
            const float cc = dts * (fn - 4 * f0) - 11 * y0 - 5 * yn + 16 * ymj;
            const float cd = dts * f0;
            for (int jo = jlo; jo < jhi; ++jo) {
                const float x = (float)((dir * t[jo] - t1) / (t1n - t1));
                float total = y0 + x * cd;
                float xp = x * x;
                total = total + xp * cc;
                xp = xp * x;
                total = total + xp * cb;
                xp = xp * x;
                total = total + xp * ca;
                xs[(int64_t)jo * xs_stride + e] = total;
            }
        }
        b.Y[e] = yn;
        b.K[0][e] = kn;
    }
}

__global__ void ld_stats_kernel(const LdCtrl* __restrict__ c, int32_t* __restrict__ stats) {
    c += blockIdx.x;
    stats += 4 * blockIdx.x;
    stats[0] = c->nfe;
    stats[1] = c->n_acc;
    stats[2] = c->n_rej;
    stats[3] = c->status;
}

// executable graphs of earlier calls: destroyed once the event recorded behind their launch has completed
struct LdPending {
    cudaGraphExec_t exec;
    cudaGraph_t graph;
    cudaEvent_t ev;
};
std::mutex g_ld_mutex;
std::deque<LdPending> g_ld_pending;
cudaStream_t g_ld_capture_stream = nullptr;

void ld_reap(bool all) {
    while (!g_ld_pending.empty()) {
        LdPending& p = g_ld_pending.front();
        if (!all && cudaEventQuery(p.ev) != cudaSuccess) {
            (void)cudaGetLastError();
            break;
        }
        if (all) cudaEventSynchronize(p.ev);
        cudaGraphExecDestroy(p.exec);
        cudaGraphDestroy(p.graph);
        cudaEventDestroy(p.ev);
        g_ld_pending.pop_front();
    }
}

// ---- discrete adjoint (restates dopri5_impl.cuh::dopri5_bwd_kernel; kb are cotangents of the INTEGRATED stage values
// fsign K, so the VJP of the raw field at stage i takes the cotangent fsign kb_i) ---------------------------------------
struct LdAdj {
    float* kb[7];  // cotangents of the seven stage values of the current step; kb[0] is kappa (FSAL) for the step before
    float* yb0;    // cotangent of the step's start state; lambda for the step before
    float* Yi;     // stage input of the next VJP
    float* cot;    // fsign kb_i: cotangent of the raw field value at that stage
    float* Yb;     // result of the VJP
};

// accepted step n as the forward saw it: Y = its start state, K = its seven raw stage values
LdBufs ld_step_view(const LdCkpt& ck, const int64_t slot, const int64_t n) {
    LdBufs b = {};
    b.Y = ck.y + slot * n;
    for (int l = 0; l < 7; ++l) b.K[l] = ck.k + (slot * 7 + l) * n;
    return b;
}

// Step `step` begins: lambda / kappa (yb0 / kb[0] of the step after it, zero for the last one) and the cotangents of the
// outputs interpolated inside it seed kb[0..6] and yb0 through the dense-output quartic; then stage 7's input / cotangent.
__global__ void ld_adj_seed_kernel(const LdCkpt ck, const LdBufs sv, const int step, const int first,
                                   const double* __restrict__ t, const int Tg, const float* __restrict__ gxs,
                                   const LdAdj a, const int64_t n) {
    const float dt = ck.dt[step], fs = (float)ld_dir(t, Tg);
    int jlo = Tg, jhi = 0;   // outputs of this step: a contiguous run of the (monotone) output table
    for (int j = 1; j < Tg; ++j)
        if (ck.out_step[j] == step) {
            jlo = min(jlo, j);
            jhi = j + 1;
        }
    float bd[6], cm[7];   // bd: row 6 of beta times dt -- stage 7's input, which is also the step's end state y1
    ld_stage_coefs(6, dt, bd);
#pragma unroll
    for (int l = 0; l < 7; ++l) cm[l] = __fmul_rn(dt, ldCMid[l]);
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        float yb0 = 0.f, yb1 = first ? 0.f : a.yb0[e], ybm = 0.f, fb0 = 0.f, fb1 = first ? 0.f : a.kb[0][e];
        for (int jo = jhi - 1; jo >= jlo; --jo) {
            if (ck.out_step[jo] != step) continue;
            const float x = ck.out_x[jo], x2 = x * x, x3 = x2 * x, x4 = x2 * x2;
            const float g = gxs[(int64_t)jo * n + e];
            yb0 = fmaf(g, 1.f - 11.f * x2 + 18.f * x3 - 8.f * x4, yb0);
            yb1 = fmaf(g, -5.f * x2 + 14.f * x3 - 8.f * x4, yb1);
            ybm = fmaf(g, 16.f * x2 - 32.f * x3 + 16.f * x4, ybm);
            fb0 = fmaf(g, dt * (x - 4.f * x2 + 5.f * x3 - 2.f * x4), fb0);
            fb1 = fmaf(g, dt * (x2 - 3.f * x3 + 2.f * x4), fb1);
        }
        float kb6 = 0.f;
#pragma unroll
        for (int l = 0; l < 7; ++l) {
            float v = (l < 6 ? bd[l] * yb1 : 0.f) + cm[l] * ybm;
            if (l == 0) v += fb0;
            if (l == 6) v += fb1;
            a.kb[l][e] = v;
            if (l == 6) kb6 = v;
        }
        a.yb0[e] = yb0 + (yb1 + ybm);
        a.Yi[e] = ld_stage_input(sv, 6, bd, fs, e);
        a.cot[e] = fs * kb6;
    }
}

// After the VJP of stage i (1..6): yb0 += Yb, kb_l += beta_{i-1,l} dt Yb (l < i); then the input / cotangent of stage
// i-1, or for i == 1 of the first step the cotangent of f(y0) (the VJP at y0 itself).
__global__ void ld_adj_stage_kernel(const LdCkpt ck, const LdBufs sv, const int step, const int i,
                                    const double* __restrict__ t, const int Tg, const LdAdj a, const int64_t n) {
    const float dt = ck.dt[step], fs = (float)ld_dir(t, Tg);
    float bd[6], bn[6];
    ld_stage_coefs(i, dt, bd);
    if (i > 1) ld_stage_coefs(i - 1, dt, bn);
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const float yb = a.Yb[e];
        a.yb0[e] += yb;
        float kbn = 0.f;
#pragma unroll
        for (int l = 0; l < 6; ++l)
            if (l < i) {
                const float v = fmaf(bd[l], yb, a.kb[l][e]);
                a.kb[l][e] = v;
                if (l == i - 1) kbn = v;
            }
        if (i > 1) {
            a.Yi[e] = ld_stage_input(sv, i - 1, bn, fs, e);
            a.cot[e] = fs * kbn;
        } else if (step == 0) {
            a.cot[e] = fs * kbn;
        }
    }
}

// grad_x0 = lambda + grad_xs[0] (output 0 is x0 itself), lambda = yb0 + the VJP at y0
__global__ void ld_adj_x0_kernel(const LdAdj a, const float* __restrict__ gxs, float* __restrict__ gx0, const int64_t n) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x)
        gx0[e] = (a.yb0[e] + a.Yb[e]) + gxs[e];
}

}  // namespace

// work layout (floats): Y | K0..K6 | Ys | Y1 | YM | tmp  (12 n_sets B D; draw q at q B D inside each), then 8-byte
// aligned: partial sums (2 * kLdMaxBlocks float64 per draw) and the controller blocks (one per draw)
static int64_t ld_work_floats(int D, int n_sets, int64_t B) {
    return 12 * n_sets * B * (int64_t)D + 2 + n_sets * (2 * (2 * (int64_t)kLdMaxBlocks) + (int64_t)(sizeof(LdCtrl) + 3) / 4) +
           2;
}

extern "C" int64_t gpode_dopri5_large_work_floats(int D, int64_t B) { return ld_work_floats(D, 1, B); }

extern "C" int64_t gpode_dopri5_large_sets_work_floats(int D, int n_sets, int64_t set_rows) {
    return ld_work_floats(D, n_sets, set_rows);
}

namespace {

// n_sets draws of B rows each (draw q: rows [q B, (q + 1) B) of x0 / xs, packed block q), one controller per draw
int ld_fwd(const float* packed_large, const gpode_cache_t* c, const float* x0, const double* t, int Tg, int n_sets,
           int64_t B, double rtol, double atol, float* xs, float* work, int32_t* stats_out, int max_attempts, float* ckpt,
           int cap, cudaStream_t st) {
    GPODE_CHECK_ARG(c != nullptr && c->D > GPODE_MAX_D && c->D <= GPODE_MAX_D_LARGE, "large-D path needs %d < D <= %d",
                    GPODE_MAX_D, GPODE_MAX_D_LARGE);
    GPODE_CHECK_ARG(Tg >= 1 && B >= 0 && max_attempts >= 1, "bad sizes Tg=%d B=%lld", Tg, (long long)B);
    GPODE_CHECK_ARG(packed_large && x0 && t && xs && work && stats_out, "NULL argument");
    cudaStreamCaptureStatus capturing = cudaStreamCaptureStatusNone;
    GPODE_CUDA(cudaStreamIsCapturing(st, &capturing));
    GPODE_CHECK_ARG(capturing == cudaStreamCaptureStatusNone,
                    "gpode_dopri5_fwd_large builds its own CUDA graph (device-side while loop) and cannot run inside a "
                    "stream capture");
    const int D = c->D;
    const int64_t n = B * D;          // elements of one draw
    const int64_t na = n * n_sets;    // ... of all draws
    if (B == 0) {
        GPODE_CUDA(cudaMemsetAsync(stats_out, 0, 4 * sizeof(int32_t) * n_sets, st));
        return 0;
    }
    LdBufs b;
    b.Y = work;
    for (int l = 0; l < 7; ++l) b.K[l] = work + (1 + l) * na;
    b.Ys = work + 8 * na;
    b.Y1 = work + 9 * na;
    b.YM = work + 10 * na;
    b.tmp = work + 11 * na;
    uintptr_t p = reinterpret_cast<uintptr_t>(work + 12 * na);
    p = (p + 7) & ~(uintptr_t)7;
    double* partial = reinterpret_cast<double*>(p);
    LdCtrl* ctrl = reinterpret_cast<LdCtrl*>(partial + 2 * kLdMaxBlocks * n_sets);
    const unsigned g = ld_grid(n);
    const dim3 grid(g, (unsigned)n_sets);
    const double n_elem = (double)n;
    const float rt = (float)rtol, at = (float)atol;
    const LdCkpt ck = ld_ckpt(ckpt, cap, n, Tg);
    const int64_t stride = gpode_packed_large_floats(D, c->M, c->S);
    // the start evaluates every draw; inside the loop the tiles of the draws that are done are skipped
    const GpodeDraws all{n_sets, B, stride, nullptr, 0};
    const GpodeDraws live{n_sets, B, stride,
                          n_sets > 1 ? reinterpret_cast<const int*>(reinterpret_cast<const char*>(ctrl) +
                                                                    offsetof(LdCtrl, done))
                                     : nullptr,
                          (int)(sizeof(LdCtrl) / sizeof(int))};

    // ---- start: y = x0, f0, initial step (two evaluations) ----
    GPODE_CUDA(cudaMemcpyAsync(b.Y, x0, sizeof(float) * na, cudaMemcpyDeviceToDevice, st));
    GPODE_CUDA(cudaMemcpyAsync(xs, x0, sizeof(float) * na, cudaMemcpyDeviceToDevice, st));
    ld_start_kernel<<<n_sets, 1, 0, st>>>(ctrl, t, Tg, max_attempts, ckpt ? cap : 0, ck.out_step);
    if (int rc = gpode_vf_large_eval(packed_large, c, b.Y, b.tmp, b.K[0], all, st)) return rc;
    ld_norm01_kernel<<<grid, kLdThreads, 0, st>>>(b.Y, b.K[0], rt, at, n, partial);
    ld_init1_kernel<<<n_sets, kLdThreads, 0, st>>>(ctrl, partial, (int)g, n_elem);
    ld_euler_kernel<<<grid, kLdThreads, 0, st>>>(ctrl, b.Y, b.K[0], b.Ys, n);
    if (int rc = gpode_vf_large_eval(packed_large, c, b.Ys, b.tmp, b.K[1], all, st)) return rc;
    ld_norm2_kernel<<<grid, kLdThreads, 0, st>>>(b.Y, b.K[0], b.K[1], rt, at, n, partial);
    ld_init2_kernel<<<n_sets, kLdThreads, 0, st>>>(ctrl, partial, (int)g, n_elem, t, Tg);
    GPODE_LAUNCH_CHECK();

    // ---- the attempt loop as a WHILE node (condition: "not done", set by the controller kernel; with several draws
    // "any draw not done", set by ld_any_kernel) ----
    std::lock_guard<std::mutex> lock(g_ld_mutex);
    ld_reap(false);
    if (g_ld_capture_stream == nullptr) GPODE_CUDA(cudaStreamCreateWithFlags(&g_ld_capture_stream, cudaStreamNonBlocking));
    cudaGraph_t graph;
    GPODE_CUDA(cudaGraphCreate(&graph, 0));
    cudaGraphConditionalHandle handle;
    // default value 1: the body's first kernels return at once when the start kernels already set `done`
    GPODE_CUDA(cudaGraphConditionalHandleCreate(&handle, graph, 1, cudaGraphCondAssignDefault));
    cudaGraphNodeParams np = {};
    np.type = cudaGraphNodeTypeConditional;
    np.conditional.handle = handle;
    np.conditional.type = cudaGraphCondTypeWhile;
    np.conditional.size = 1;
    cudaGraphNode_t node;
    GPODE_CUDA(cudaGraphAddNode(&node, graph, nullptr, 0, &np));
    cudaGraph_t body = np.conditional.phGraph_out[0];
    cudaStream_t cs = g_ld_capture_stream;
    GPODE_CUDA(cudaStreamBeginCaptureToGraph(cs, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
    int rc = 0;
    for (int i = 1; i <= 6 && rc == 0; ++i) {
        float* out = i == 6 ? b.Y1 : b.Ys;
        ld_stage_kernel<<<grid, kLdThreads, 0, cs>>>(ctrl, i, b, out, n);
        rc = gpode_vf_large_eval(packed_large, c, out, b.tmp, b.K[i], live, cs);
    }
    if (rc == 0) {
        ld_err_kernel<<<grid, kLdThreads, 0, cs>>>(ctrl, b, rt, at, n, partial);
        ld_ctrl_kernel<<<n_sets, kLdThreads, 0, cs>>>(ctrl, partial, (int)g, n_elem, t, Tg, handle, n_sets == 1);
        if (n_sets > 1) ld_any_kernel<<<1, kLdThreads, 0, cs>>>(ctrl, n_sets, handle);
        ld_accept_kernel<<<grid, kLdThreads, 0, cs>>>(ctrl, b, t, xs, n, ck);
    }
    cudaGraph_t captured = nullptr;
    cudaError_t ce = cudaStreamEndCapture(cs, &captured);
    if (rc != 0 || ce != cudaSuccess) {
        cudaGraphDestroy(graph);
        if (rc == 0) {
            gpode_set_error("capturing the dopri5 attempt failed: %s", cudaGetErrorString(ce));
            rc = (int)ce;
        }
        return rc;
    }
    cudaGraphExec_t exec;
    ce = cudaGraphInstantiate(&exec, graph, 0);
    if (ce != cudaSuccess) {
        cudaGraphDestroy(graph);
        gpode_set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(ce));
        return (int)ce;
    }
    GPODE_CUDA(cudaGraphLaunch(exec, st));
    ld_stats_kernel<<<n_sets, 1, 0, st>>>(ctrl, stats_out);
    LdPending pend;
    pend.exec = exec;
    pend.graph = graph;
    GPODE_CUDA(cudaEventCreateWithFlags(&pend.ev, cudaEventDisableTiming));
    GPODE_CUDA(cudaEventRecord(pend.ev, st));
    g_ld_pending.push_back(pend);
    GPODE_LAUNCH_CHECK();
    return 0;
}

}  // namespace

extern "C" int gpode_dopri5_fwd_large(const float* packed_large, const gpode_cache_t* c, const float* x0, const double* t,
                                      int Tg, int64_t B, double rtol, double atol, float* xs, float* work,
                                      int32_t* stats_out, int max_attempts, void* stream) {
    return ld_fwd(packed_large, c, x0, t, Tg, 1, B, rtol, atol, xs, work, stats_out, max_attempts, nullptr, 0,
                  (cudaStream_t)stream);
}

extern "C" int gpode_dopri5_fwd_large_ckpt(const float* packed_large, const gpode_cache_t* c, const float* x0,
                                           const double* t, int Tg, int64_t B, double rtol, double atol, float* xs,
                                           float* work, int32_t* stats_out, int max_attempts, float* ckpt, int cap,
                                           void* stream) {
    GPODE_CHECK_ARG(ckpt != nullptr && cap > 0, "checkpointing needs a block and cap > 0 (cap=%d)", cap);
    return ld_fwd(packed_large, c, x0, t, Tg, 1, B, rtol, atol, xs, work, stats_out, max_attempts, ckpt, cap,
                  (cudaStream_t)stream);
}

// n_sets draws of the "sets" cache (packed by gpode_pack_cache_large_sets), one controller each: draw q's rows of xs and
// its stats are those of gpode_dopri5_fwd_large called on draw q alone
extern "C" int gpode_dopri5_fwd_large_sets(const float* packed_large, const gpode_cache_t* c, int n_sets,
                                           int64_t set_rows, const float* x0, const double* t, int Tg, double rtol,
                                           double atol, float* xs, float* work, int32_t* stats_out, int max_attempts,
                                           void* stream) {
    GPODE_CHECK_ARG(n_sets >= 1 && n_sets <= 65535 && set_rows >= 0, "n_sets=%d outside 1..65535 or set_rows < 0",
                    n_sets);
    if (set_rows == 0) {
        GPODE_CHECK_ARG(stats_out != nullptr, "stats_out is NULL");
        GPODE_CUDA(cudaMemsetAsync(stats_out, 0, 4 * sizeof(int32_t) * n_sets, (cudaStream_t)stream));
        return 0;
    }
    return ld_fwd(packed_large, c, x0, t, Tg, n_sets, set_rows, rtol, atol, xs, work, stats_out, max_attempts, nullptr,
                  0, (cudaStream_t)stream);
}

// work: 11 B D floats (kb[0..6], yb0, stage input, cotangent, VJP result)
extern "C" int gpode_dopri5_bwd_large(const float* packed_bwd, const gpode_cache_t* c, const double* t, int Tg, int64_t B,
                                      const float* grad_xs, const float* ckpt, int cap, int n_accepted, float* grad_x0,
                                      float* acc_large, float* work, void* stream) {
    GPODE_CHECK_ARG(c != nullptr && c->D > GPODE_MAX_D && c->D <= GPODE_MAX_D_LARGE, "large-D path needs %d < D <= %d",
                    GPODE_MAX_D, GPODE_MAX_D_LARGE);
    GPODE_CHECK_ARG(Tg >= 1 && B >= 0, "bad sizes Tg=%d B=%lld", Tg, (long long)B);
    GPODE_CHECK_ARG(cap > 0 && n_accepted >= 0 && n_accepted <= cap, "n_accepted=%d outside 0..cap=%d", n_accepted, cap);
    if (B == 0) return 0;
    GPODE_CHECK_ARG(packed_bwd && t && grad_xs && ckpt && grad_x0 && acc_large && work, "NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int D = c->D, M = c->M, S = c->S;
    const int64_t n = B * D;
    if (Tg == 1 || n_accepted == 0) {   // no step: x0 reaches the loss only as output 0
        GPODE_CUDA(cudaMemcpyAsync(grad_x0, grad_xs, sizeof(float) * n, cudaMemcpyDeviceToDevice, st));
        return 0;
    }
    const LdCkpt ck = ld_ckpt(const_cast<float*>(ckpt), cap, n, Tg);
    LdAdj a;
    for (int l = 0; l < 7; ++l) a.kb[l] = work + l * n;
    a.yb0 = work + 7 * n;
    a.Yi = work + 8 * n;
    a.cot = work + 9 * n;
    a.Yb = work + 10 * n;
    const unsigned g = ld_grid(n);
    for (int step = n_accepted - 1; step >= 0; --step) {
        const LdBufs sv = ld_step_view(ck, step, n);
        ld_adj_seed_kernel<<<g, kLdThreads, 0, st>>>(ck, sv, step, step == n_accepted - 1, t, Tg, grad_xs, a, n);
        for (int i = 6; i >= 1; --i) {
            if (int rc = gpode_vf_bwd_large(packed_bwd, D, M, S, a.Yi, sv.K[i], a.cot, a.Yb, acc_large, B, st)) return rc;
            ld_adj_stage_kernel<<<g, kLdThreads, 0, st>>>(ck, sv, step, i, t, Tg, a, n);
        }
        GPODE_LAUNCH_CHECK();
    }
    // the first step's k1 = f(y0) has no step before it to hand its cotangent to: one more VJP, at y0
    const LdBufs s0 = ld_step_view(ck, 0, n);
    if (int rc = gpode_vf_bwd_large(packed_bwd, D, M, S, s0.Y, s0.K[0], a.cot, a.Yb, acc_large, B, st)) return rc;
    ld_adj_x0_kernel<<<g, kLdThreads, 0, st>>>(a, grad_xs, grad_x0, n);
    GPODE_LAUNCH_CHECK();
    return 0;
}
