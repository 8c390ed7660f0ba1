// Multiple-shooting ELBO step for 8 < D <= 64 (gpode_shoot_fwd_large / gpode_shoot_bwd_large): the contract of
// gpode_shoot_fwd / gpode_shoot_bwd (shoot.cuh, integrate.cu) on the large-D kernels.
//
// Forward: the rows [row_lo, row_hi) of the (S_mc, N, T) segment batch take ONE 3/8-rule RK4 interval through
// gpode_rk4_fwd_large_dev (tcgen05 vector field + stage kernels), so the end point is bitwise the xs[1] of that call.
// Then ONE epilogue kernel evaluates, per end point, the decode pred W + bias, the Gaussian log-density of the
// observation and its derivative w.r.t. the likelihood variance, the shooting constraint against ss[row + 1] and the two
// seed vectors d(loglik sum)/d pred | d(constraint sum)/d pred. No (B, D_obs) tensor is written.
// Epilogue mapping: one warp per row (grid-stride). Lane l owns the observed dimensions d = l + 32 q (q < NQ) for the
// decode and the log-density, and the state dimensions j = l, l + 32 for the constraint and the seeds. W [D][DPW] sits
// in shared memory with an odd row stride DPW = 32 NQ + 1: the decode reads a row of W across the lanes, the seed
// contraction sl_j = -sum_d q_d W_jd a column (one bank per lane either way).
//
// Backward: one kernel forms grad_xs = [0, g_ll seed_ll + g_cons seed_c] (the two upstream scalars are read on the
// device), gpode_rk4_bwd_large runs the discrete adjoint straight into grad_ss[row_lo:row_hi] and adds the
// shared-parameter partial sums to acc_large, and a last kernel adds the constraint's pull on the next state,
// -g_cons seed_c[row - 1] (the rules of shoot.cuh shoot_store_grad, including the halo row row_hi).
//
// Sums are bitwise reproducible: per-lane float64 partials, warp shuffles, warps in warp order, one row of `work` per
// CTA, rows added in row order by the sum kernel of the D <= 8 step (gpode_shoot_sum_launch). Every launch size
// follows from the host shapes.
#include "common.cuh"
#include "shoot.cuh"

namespace {

constexpr int kLsThreads = 256, kLsWarps = kLsThreads / 32;
constexpr int kLsMaxCtas = 1024;                    // epilogue grid cap = rows of partial sums in `work`
constexpr int kLsCols = 2 + GPODE_SHOOT_MAX_DOBS;   // loglik, constraint, d loglik / d var_d

struct LsArgs {
    const float* xs1;         // [B, D] end points
    const float* ss;          // [S_mc N T, D] all sampled states
    const float* ys;          // [N, T, Dobs]
    const float* W;           // [D, Dobs]
    const float* bias;        // [Dobs] or NULL
    const float* lik_var;     // [Dobs]
    const float* cons_scale;  // 1 float
    int D, N, T, Dobs, laplace, halo;
    int64_t row_lo, B;
    float* pred_out;          // [B, D] or NULL
    float* seeds;             // [2, B, D] or NULL
    double* work;             // [gridDim.x][2 + Dobs]
};

__host__ __device__ inline int ls_dpw(int nq) { return 32 * nq + 1; }
// floats: W [D][DPW] | bias, 1/var, log(2 pi var) [32 NQ] each | per warp: end point [64], q [32 NQ]; then float64
// [warps][2 + Dobs]
__host__ __device__ inline size_t ls_smem_bytes(int D, int nq) {
    const size_t fl = (size_t)D * ls_dpw(nq) + 3 * 32 * nq + kLsWarps * (64 + 32 * nq);
    return ((fl * 4 + 15) & ~(size_t)15) + (size_t)kLsWarps * kLsCols * 8;
}

template <int NQ>
__global__ void __launch_bounds__(kLsThreads)
shoot_epilogue_large_kernel(const LsArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int DP = 32 * NQ, DPW = 32 * NQ + 1;
    const int D = a.D, Dobs = a.Dobs;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* sW = reinterpret_cast<float*>(smem_raw);
    float* sb = sW + D * DPW;
    float* siv = sb + DP;
    float* slv = siv + DP;
    float* spred = slv + DP + warp * (64 + DP);
    float* sq = spred + 64;
    double* wacc = reinterpret_cast<double*>(smem_raw + ls_smem_bytes(D, NQ) - (size_t)kLsWarps * kLsCols * 8);

    for (int i = threadIdx.x; i < D * DPW; i += kLsThreads) {
        const int l = i / DPW, d = i - l * DPW;
        sW[i] = d < Dobs ? a.W[l * Dobs + d] : 0.f;
    }
    for (int d = threadIdx.x; d < DP; d += kLsThreads) {
        const bool ok = d < Dobs;
        const float v = ok ? a.lik_var[d] : 1.f;
        sb[d] = (ok && a.bias) ? a.bias[d] : 0.f;
        siv[d] = ok ? 1.0f / v : 0.f;
        slv[d] = ok ? 1.8378770664093453f + logf(v) : 0.f;  // log(2 pi) + log var
    }
    const float scale = __ldg(a.cons_scale);
    const float inv = 1.0f / scale, inv2 = inv * inv;
    const float c0 = a.laplace ? -logf(2.0f * scale) : -logf(scale) - 0.9189385332046727f;  // -log s - 0.5 log 2 pi
    __syncthreads();

    double ll = 0.0, cs = 0.0, gv[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) gv[q] = 0.0;
    const int64_t NT = (int64_t)a.N * a.T;
    for (int64_t r = (int64_t)blockIdx.x * kLsWarps + warp; r < a.B; r += (int64_t)gridDim.x * kLsWarps) {
        const int64_t g = a.row_lo + r;
        const int t = (int)(g % a.T);
        const bool obs = !(a.halo && t == a.T - 1);   // this row carries an observation
        const bool has_next = t < a.T - 1;
        float p[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int j = lane + 32 * h;
            p[h] = j < D ? __ldg(a.xs1 + r * D + j) : 0.f;
            if (j < D) {
                spred[j] = p[h];
                if (a.pred_out != nullptr) a.pred_out[r * D + j] = p[h];
            }
        }
        __syncwarp();
        // decode and log-density of this lane's observed dimensions
        const float* __restrict__ y = a.ys + (g % NT) * Dobs;
        float yv[NQ], f[NQ];
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            const int d = lane + 32 * q;
            yv[q] = (obs && d < Dobs) ? __ldg(y + d) : 0.f;
            f[q] = sb[d];
        }
#pragma unroll 4
        for (int l = 0; l < D; ++l) {
            const float pl = spred[l];
#pragma unroll
            for (int q = 0; q < NQ; ++q) f[q] = fmaf(pl, sW[l * DPW + lane + 32 * q], f[q]);
        }
        float lsum = 0.f;
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            const int d = lane + 32 * q;
            const float iv = siv[d];
            const float diff = obs ? f[q] - yv[q] : 0.f;   // a padded dimension has f = y = 0
            const float qd = diff * iv;
            lsum += -0.5f * (slv[d] + diff * qd);
            gv[q] += obs ? (double)(-0.5f * (iv - qd * qd)) : 0.0;
            sq[d] = qd;
        }
        __syncwarp();
        // shooting constraint against the NEXT sampled state of the sequence, and the two seeds
        const float* __restrict__ nxt = a.ss + (g + (has_next ? 1 : 0)) * D;
        float csum = 0.f;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int j = lane + 32 * h;
            if (j >= D) continue;
            float sl = 0.f;
            const float* __restrict__ wr = sW + j * DPW;
#pragma unroll 4
            for (int d = 0; d < DP; ++d) sl = fmaf(-sq[d], wr[d], sl);
            const float diff = has_next ? __ldg(nxt + j) - p[h] : 0.f;
            float sc;
            if (a.laplace) {
                csum += has_next ? c0 - fabsf(diff) * inv : 0.f;
                sc = diff > 0.f ? inv : (diff < 0.f ? -inv : 0.f);   // d lp / d pred
            } else {
                csum += has_next ? c0 - 0.5f * diff * diff * inv2 : 0.f;
                sc = diff * inv2;
            }
            if (a.seeds != nullptr) {
                a.seeds[r * D + j] = sl;
                a.seeds[(a.B + r) * D + j] = sc;
            }
        }
        ll += obs ? (double)lsum : 0.0;
        cs += (double)csum;
        __syncwarp();   // spred / sq are rewritten by the next row
    }
    // lanes -> warp slots -> this CTA's row of `work`, in float64 and in a fixed order
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ll += __shfl_xor_sync(0xffffffffu, ll, o);
        cs += __shfl_xor_sync(0xffffffffu, cs, o);
    }
    double* wa = wacc + warp * kLsCols;
    if (lane == 0) {
        wa[0] = ll;
        wa[1] = cs;
    }
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
        const int d = lane + 32 * q;
        if (d < Dobs) wa[2 + d] = gv[q];
    }
    __syncthreads();
    double* __restrict__ row = a.work + (size_t)blockIdx.x * (2 + Dobs);
    for (int i = threadIdx.x; i < 2 + Dobs; i += kLsThreads) {
        double s = 0.0;
        for (int w = 0; w < kLsWarps; ++w) s += wacc[w * kLsCols + i];
        row[i] = s;
    }
}

// grad_xs [2, B, D] of the one-interval adjoint: [0 | g_ll seed_ll + g_cons seed_c]
__global__ void shoot_seed_large_kernel(const float* __restrict__ seeds, const float* __restrict__ g_ll,
                                        const float* __restrict__ g_cons, float* __restrict__ gxs, const int64_t n) {
    const float a = __ldg(g_ll), b = __ldg(g_cons);
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        gxs[e] = 0.f;
        gxs[n + e] = a * __ldg(seeds + e) + b * __ldg(seeds + n + e);
    }
}

// grad_ss[row_lo + row] (the adjoint's grad_x0, already in place) += the previous row's constraint pull; the state
// just past the last row receives the last row's pull when the range ends before the batch does
__global__ void shoot_pull_large_kernel(const float* __restrict__ seeds, const float* __restrict__ g_cons,
                                        float* __restrict__ grad_ss, const int D, const int64_t row_lo,
                                        const int64_t B, const int64_t n_total) {
    const float b = __ldg(g_cons);
    const float* __restrict__ sc = seeds + B * D;
    const int64_t n = B * D;
    float* __restrict__ gs = grad_ss + row_lo * D;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = e / D;
        const float pull = row >= 1 ? -b * __ldg(sc + e - D) : 0.f;
        gs[e] = gs[e] + pull;
        if (row == B - 1 && row_lo + B < n_total) gs[e + D] = -b * __ldg(sc + e);
    }
}

inline unsigned ls_ew_grid(int64_t n) {
    const int64_t g = (n + 255) / 256;
    return (unsigned)(g < 2368 ? (g < 1 ? 1 : g) : 2368);
}

int ls_check(const gpode_cache_t* c, const gpode_shoot_t* sh) {
    GPODE_CHECK_ARG(c != nullptr, "cache is NULL");
    GPODE_CHECK_ARG(c->D > GPODE_MAX_D && c->D <= GPODE_MAX_D_LARGE, "large-D shooting step needs %d < D <= %d, got %d",
                    GPODE_MAX_D, GPODE_MAX_D_LARGE, c->D);
    GPODE_CHECK_ARG(c->M >= 1 && c->S >= 1, "M=%d and S=%d must be positive", c->M, c->S);
    return gpode_check_shoot(sh);
}

// float64 words of `work` in front of the float scratch: the epilogue's per-CTA partial rows
constexpr int64_t kLsPartDoubles = (int64_t)kLsMaxCtas * kLsCols;

}  // namespace

extern "C" int64_t gpode_shoot_large_work_doubles(int D, int64_t n_rows) {
    if (D <= GPODE_MAX_D || D > GPODE_MAX_D_LARGE || n_rows < 0) return -1;
    // forward: xs [2,B,D] + the integrator's tmp (6 B D without checkpoints); backward: grad_xs [2,B,D] + 7 B D
    return kLsPartDoubles + (9 * n_rows * D + 1) / 2;
}

extern "C" int gpode_shoot_fwd_large(const float* packed_large, const gpode_cache_t* c, const gpode_shoot_t* sh,
                                     const float* ss, const float* t2, float* kstages, float* pred_out, float* seeds,
                                     double* sums_out, float* grad_lik_var, double* work, void* stream) {
    if (int rc = ls_check(c, sh)) return rc;
    GPODE_CHECK_ARG(packed_large && ss && t2 && sums_out && work, "NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int D = c->D;
    const int64_t B = sh->row_hi - sh->row_lo;
    if (B == 0) {
        GPODE_CUDA(cudaMemsetAsync(sums_out, 0, 2 * sizeof(double), st));
        if (grad_lik_var) GPODE_CUDA(cudaMemsetAsync(grad_lik_var, 0, sizeof(float) * sh->D_obs, st));
        return 0;
    }
    GPODE_CHECK_ARG((kstages == nullptr) == (seeds == nullptr), "kstages and seeds go together (both or neither)");
    float* xs = reinterpret_cast<float*>(work + kLsPartDoubles);   // [2, B, D]
    float* tmp = xs + 2 * B * D;
    if (int rc = gpode_rk4_fwd_large_dev(packed_large, c, ss + sh->row_lo * D, t2, 2, B, xs, kstages, tmp, stream))
        return rc;
    LsArgs a;
    a.xs1 = xs + B * D; a.ss = ss; a.ys = sh->ys; a.W = sh->W; a.bias = sh->bias; a.lik_var = sh->lik_var;
    a.cons_scale = sh->cons_scale;
    a.D = D; a.N = sh->N; a.T = sh->T; a.Dobs = sh->D_obs; a.laplace = sh->laplace & 1; a.halo = (sh->laplace >> 1) & 1;
    a.row_lo = sh->row_lo; a.B = B;
    a.pred_out = pred_out; a.seeds = seeds; a.work = work;
    const int nq = (sh->D_obs + 31) / 32;
    const size_t smem = ls_smem_bytes(D, nq);
    const int64_t want = (B + kLsWarps - 1) / kLsWarps;
    const int grid = (int)(want < kLsMaxCtas ? want : kLsMaxCtas);
    switch (nq) {
#define CASE(NQ_)                                                                                                  \
    case NQ_:                                                                                                      \
        GPODE_CUDA(cudaFuncSetAttribute(shoot_epilogue_large_kernel<NQ_>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                        (int)smem));                                                               \
        shoot_epilogue_large_kernel<NQ_><<<grid, kLsThreads, smem, st>>>(a);                                       \
        break;
        CASE(1) CASE(2) CASE(3) CASE(4)
#undef CASE
        default: break;
    }
    GPODE_LAUNCH_CHECK();
    return gpode_shoot_sum_launch(work, grid, 2 + sh->D_obs, sums_out, grad_lik_var, st);
}

extern "C" int gpode_shoot_bwd_large(const float* packed_bwd, const gpode_cache_t* c, const gpode_shoot_t* sh,
                                     const float* ss, const float* t2, const float* kstages, const float* seeds,
                                     const float* g_ll, const float* g_cons, float* grad_ss, float* acc_large,
                                     double* work, void* stream) {
    if (int rc = ls_check(c, sh)) return rc;
    const int64_t B = sh->row_hi - sh->row_lo;
    if (B == 0) return 0;
    GPODE_CHECK_ARG(packed_bwd && ss && t2 && kstages && seeds && g_ll && g_cons && grad_ss && acc_large && work,
                    "NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int D = c->D;
    const int64_t n = B * D, n_total = (int64_t)sh->S_mc * sh->N * sh->T;
    float* gxs = reinterpret_cast<float*>(work + kLsPartDoubles);   // [2, B, D]
    float* rk_work = gxs + 2 * n;                                   // 7 B D
    shoot_seed_large_kernel<<<ls_ew_grid(n), 256, 0, st>>>(seeds, g_ll, g_cons, gxs, n);
    GPODE_LAUNCH_CHECK();
    // xs: the adjoint of one interval reads only its start, xs[0] = the rows of ss; grad_x0 lands in grad_ss directly
    float* gx0 = grad_ss + sh->row_lo * D;
    if (int rc = gpode_rk4_bwd_large(packed_bwd, c, t2, 2, B, ss + sh->row_lo * D, kstages, gxs, gx0, acc_large,
                                     rk_work, stream))
        return rc;
    shoot_pull_large_kernel<<<ls_ew_grid(n), 256, 0, st>>>(seeds, g_cons, grad_ss, D, sh->row_lo, B, n_total);
    GPODE_LAUNCH_CHECK();
    return 0;
}
