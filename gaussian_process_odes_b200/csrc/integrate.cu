// C-ABI entry points of the integrator path; dispatch on the state dimension to the per-D translation units.
#include "common.cuh"
#include "shoot.cuh"

#define GPODE_FOR_EACH_D(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8)

#define GPODE_DECL(D_)                                                                                              \
    int gpode_vf_fwd_d##D_(const float*, int, int, const float*, float*, int64_t, cudaStream_t);                    \
    int gpode_rk4_fwd_d##D_(const float*, int, int, const float*, const float*, int, int64_t, float*, float*,       \
                            cudaStream_t);                                                                          \
    int gpode_rk4_bwd_d##D_(const float*, int, int, const float*, int, int64_t, const float*, const float*,         \
                            const float*, float*, float*, float*, float*, cudaStream_t);                            \
    int gpode_vf_bwd_d##D_(const float*, int, int, const float*, const float*, const float*, float*, int64_t,       \
                           float*, cudaStream_t);                                                                   \
    int gpode_fwd_sets_d##D_(const float*, int, int, int, int64_t, const float*, const float*, int, float*,         \
                             cudaStream_t);                                                                         \
    int gpode_shoot_fwd_d##D_(const float*, int, int, const float*, const float*, int64_t, float*, const ShootArgs*, \
                              int*, cudaStream_t);                                                                  \
    int gpode_shoot_bwd_d##D_(const float*, int, int, const float*, int64_t, const float*, const float*, float*,    \
                              float*, float*, const float*, const float*, const float*, float*, int64_t, int64_t,   \
                              cudaStream_t);                                                                        \
    bool gpode_shoot_row_sums_d##D_(int, int, int64_t);
GPODE_FOR_EACH_D(GPODE_DECL)
#undef GPODE_DECL

int gpode_param_grad_launch(const float* packed, int D, int M, int S, const float* ys, const float* kbs, int64_t VR,
                            float* acc, cudaStream_t stream, const int32_t* stats_dev = nullptr,
                            int64_t rows_per_step = 0);  // param_grad.cu

static int check_common(const float* packed, int D, int M, int S, int64_t B) {
    GPODE_CHECK_ARG(packed != nullptr, "packed parameter block is NULL");
    GPODE_CHECK_ARG(D >= 1 && D <= GPODE_MAX_D, "state dimension D=%d outside 1..%d", D, GPODE_MAX_D);
    GPODE_CHECK_ARG(M >= 1 && S >= 1, "M=%d and S=%d must be positive", M, S);
    GPODE_CHECK_ARG(B >= 0, "negative batch size %lld", (long long)B);
    return 0;
}

#define GPODE_SWITCH_D(D_, CALL)                                   \
    switch (D_) {                                                  \
        case 1: return CALL(1);                                    \
        case 2: return CALL(2);                                    \
        case 3: return CALL(3);                                    \
        case 4: return CALL(4);                                    \
        case 5: return CALL(5);                                    \
        case 6: return CALL(6);                                    \
        case 7: return CALL(7);                                    \
        case 8: return CALL(8);                                    \
        default: break;                                            \
    }                                                              \
    gpode_set_error("state dimension D=%d outside 1..%d", D_, GPODE_MAX_D); \
    return -1;

extern "C" int gpode_vf_fwd(const float* packed, int D, int M, int S, const float* x, float* f, int64_t B,
                            void* stream) {
    if (int rc = check_common(packed, D, M, S, B)) return rc;
    if (B == 0) return 0;
    GPODE_CHECK_ARG(x && f, "x / f is NULL");
#define CALL(D_) gpode_vf_fwd_d##D_(packed, M, S, x, f, B, (cudaStream_t)stream)
    GPODE_SWITCH_D(D, CALL)
#undef CALL
}

extern "C" int gpode_rk4_fwd(const float* packed, int D, int M, int S, const float* x0, const float* t, int Tg,
                             int64_t B, float* xs, float* kstages, void* stream) {
    if (int rc = check_common(packed, D, M, S, B)) return rc;
    GPODE_CHECK_ARG(Tg >= 1, "time grid needs at least one point, got %d", Tg);
    if (B == 0) return 0;
    GPODE_CHECK_ARG(x0 && t && xs, "x0 / t / xs is NULL");
#define CALL(D_) gpode_rk4_fwd_d##D_(packed, M, S, x0, t, Tg, B, xs, kstages, (cudaStream_t)stream)
    GPODE_SWITCH_D(D, CALL)
#undef CALL
}

static int fwd_sets_dispatch(const float* packed, int D, int M, int S, int n_sets, int64_t set_rows, const float* x0,
                             const float* t, int Tg, float* out, cudaStream_t st) {
#define CALL(D_) gpode_fwd_sets_d##D_(packed, M, S, n_sets, set_rows, x0, t, Tg, out, st)
    GPODE_SWITCH_D(D, CALL)
#undef CALL
}

static int check_sets(int n_sets, int64_t set_rows) {
    GPODE_CHECK_ARG(n_sets >= 1 && n_sets <= 65535, "n_sets=%d outside 1..65535", n_sets);
    GPODE_CHECK_ARG(set_rows >= 0, "negative rows per set %lld", (long long)set_rows);
    return 0;
}

extern "C" int gpode_vf_fwd_sets(const float* packed, int D, int M, int S, int n_sets, int64_t set_rows,
                                 const float* x, float* f, void* stream) {
    if (int rc = check_common(packed, D, M, S, set_rows)) return rc;
    if (int rc = check_sets(n_sets, set_rows)) return rc;
    if (set_rows == 0) return 0;
    GPODE_CHECK_ARG(x && f, "x / f is NULL");
    return fwd_sets_dispatch(packed, D, M, S, n_sets, set_rows, x, nullptr, 0, f, (cudaStream_t)stream);
}

extern "C" int gpode_rk4_fwd_sets(const float* packed, int D, int M, int S, int n_sets, int64_t set_rows,
                                  const float* x0, const float* t, int Tg, float* xs, void* stream) {
    if (int rc = check_common(packed, D, M, S, set_rows)) return rc;
    if (int rc = check_sets(n_sets, set_rows)) return rc;
    GPODE_CHECK_ARG(Tg >= 1, "time grid needs at least one point, got %d", Tg);
    if (set_rows == 0) return 0;
    GPODE_CHECK_ARG(x0 && t && xs, "x0 / t / xs is NULL");
    return fwd_sets_dispatch(packed, D, M, S, n_sets, set_rows, x0, t, Tg, xs, (cudaStream_t)stream);
}

static int rk4_bwd_dispatch(const float* packed, int D, int M, int S, const float* t, int Tg, int64_t B,
                            const float* xs, const float* kst, const float* gxs, float* gx0, float* vy, float* vk,
                            float* acc, cudaStream_t st) {
#define CALL(D_) gpode_rk4_bwd_d##D_(packed, M, S, t, Tg, B, xs, kst, gxs, gx0, vy, vk, acc, st)
    GPODE_SWITCH_D(D, CALL)
#undef CALL
}

extern "C" int gpode_rk4_bwd(const float* packed, int D, int M, int S, const float* t, int Tg, int64_t B,
                             const float* xs, const float* kstages, const float* grad_xs, float* grad_x0,
                             float* vrows, float* acc, void* stream) {
    if (int rc = check_common(packed, D, M, S, B)) return rc;
    GPODE_CHECK_ARG(Tg >= 1, "time grid needs at least one point, got %d", Tg);
    if (B == 0) return 0;
    GPODE_CHECK_ARG(t && xs && grad_xs && grad_x0 && acc, "NULL argument");
    if (Tg == 1) {
        GPODE_CUDA(cudaMemcpyAsync(grad_x0, grad_xs, sizeof(float) * B * D, cudaMemcpyDeviceToDevice,
                                   (cudaStream_t)stream));
        return 0;
    }
    GPODE_CHECK_ARG(kstages && vrows, "kstages / vrows is NULL");
    const int64_t VR = (int64_t)(Tg - 1) * 4 * B;
    float* vy = vrows;
    float* vk = vrows + VR * D;
    return rk4_bwd_dispatch(packed, D, M, S, t, Tg, B, xs, kstages, grad_xs, grad_x0, vy, vk, acc,
                            (cudaStream_t)stream);
}

static int vf_bwd_dispatch(const float* packed, int D, int M, int S, const float* x, const float* f, const float* gf,
                           float* gx, int64_t B, float* acc, cudaStream_t st) {
#define CALL(D_) gpode_vf_bwd_d##D_(packed, M, S, x, f, gf, gx, B, acc, st)
    GPODE_SWITCH_D(D, CALL)
#undef CALL
}

extern "C" int gpode_vf_bwd(const float* packed, int D, int M, int S, const float* x, const float* f,
                            const float* grad_f, float* grad_x, float* acc, int64_t B, void* stream) {
    if (int rc = check_common(packed, D, M, S, B)) return rc;
    if (B == 0) return 0;
    GPODE_CHECK_ARG(x && f && grad_f && grad_x && acc, "NULL argument");
    return vf_bwd_dispatch(packed, D, M, S, x, f, grad_f, grad_x, B, acc, (cudaStream_t)stream);
}

extern "C" int gpode_param_grad(const float* packed, int D, int M, int S, const float* ys, const float* kbs,
                                int64_t n_rows, float* acc, void* stream) {
    if (int rc = check_common(packed, D, M, S, n_rows)) return rc;
    if (n_rows == 0) return 0;
    GPODE_CHECK_ARG(ys && kbs && acc, "NULL argument");
    return gpode_param_grad_launch(packed, D, M, S, ys, kbs, n_rows, acc, (cudaStream_t)stream);
}

extern "C" int gpode_param_grad_dev(const float* packed, int D, int M, int S, const float* ys, const float* kbs,
                                    int64_t n_rows_max, const int32_t* stats_dev, int64_t rows_per_step, float* acc,
                                    void* stream) {
    if (int rc = check_common(packed, D, M, S, n_rows_max)) return rc;
    if (n_rows_max == 0) return 0;
    GPODE_CHECK_ARG(ys && kbs && acc && stats_dev, "NULL argument");
    return gpode_param_grad_launch(packed, D, M, S, ys, kbs, n_rows_max, acc, (cudaStream_t)stream, stats_dev,
                                   rows_per_step);
}

extern "C" int64_t gpode_vrow_floats(int D, int64_t n_virtual_rows) { return 2 * n_virtual_rows * (int64_t)D; }

// ------------------------------------------------------------------------------------------------------------------
// Fused multiple-shooting step (shoot.cuh): one RK4 interval per row of the (S_mc, N, T) segment batch with the ELBO's
// observation and constraint terms evaluated on the end point inside the integrator kernel.
// ------------------------------------------------------------------------------------------------------------------
namespace {
constexpr int kShootMaxCtas = GPODE_ACC_CAP_AV;  // every forward launch shape is clamped to this many CTAs
constexpr int kShootCols = 2 + GPODE_SHOOT_MAX_DOBS;

__global__ void __launch_bounds__(256)
shoot_sum_kernel(const double* __restrict__ work, const int n_rows, const int cols, double* __restrict__ sums,
                 float* __restrict__ g_var) {
    __shared__ double part[8 * kShootCols];
    __shared__ double tot[kShootCols];
    gpode_sum_rows_ordered<(kShootCols + 31) / 32>(work, (size_t)cols, n_rows, cols, kShootCols, part, tot);
    if (threadIdx.x < 2) sums[threadIdx.x] = tot[threadIdx.x];
    if (g_var != nullptr)
        for (int i = threadIdx.x; i + 2 < cols; i += blockDim.x) g_var[i] = (float)tot[2 + i];
}

int check_shoot(const gpode_shoot_t* sh, int D) {
    GPODE_CHECK_ARG(sh != nullptr, "shooting descriptor is NULL");
    GPODE_CHECK_ARG(sh->S_mc >= 1 && sh->N >= 1 && sh->T >= 1, "bad batch shape S_mc=%d N=%d T=%d", sh->S_mc, sh->N, sh->T);
    GPODE_CHECK_ARG(sh->D_obs >= 1 && sh->D_obs <= GPODE_SHOOT_MAX_DOBS, "observed dimension %d outside 1..%d", sh->D_obs,
                    GPODE_SHOOT_MAX_DOBS);
    GPODE_CHECK_ARG(sh->ys && sh->W && sh->lik_var && sh->cons_scale, "shooting descriptor holds a NULL tensor");
    const int64_t n_total = (int64_t)sh->S_mc * sh->N * sh->T;
    GPODE_CHECK_ARG(sh->row_lo >= 0 && sh->row_lo <= sh->row_hi && sh->row_hi <= n_total,
                    "row range [%lld,%lld) outside the %lld rows of the batch", (long long)sh->row_lo,
                    (long long)sh->row_hi, (long long)n_total);
    (void)D;
    return 0;
}
}  // namespace

extern "C" int64_t gpode_shoot_work_doubles(void) { return (int64_t)kShootMaxCtas * kShootCols; }

extern "C" int gpode_shoot_fwd(const float* packed, int D, int M, int S, const gpode_shoot_t* sh, const float* ss,
                               const float* t2, float* kstages, float* pred_out, float* seeds, double* sums_out,
                               float* grad_lik_var, double* work, void* stream) {
    if (int rc = check_shoot(sh, D)) return rc;
    const int64_t B = sh->row_hi - sh->row_lo;
    if (int rc = check_common(packed, D, M, S, B)) return rc;
    GPODE_CHECK_ARG(ss && t2 && sums_out && work, "NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (B == 0) {
        GPODE_CUDA(cudaMemsetAsync(sums_out, 0, 2 * sizeof(double), st));
        if (grad_lik_var) GPODE_CUDA(cudaMemsetAsync(grad_lik_var, 0, sizeof(float) * sh->D_obs, st));
        return 0;
    }
    ShootArgs a;
    a.ys = sh->ys; a.W = sh->W; a.bias = sh->bias; a.lik_var = sh->lik_var; a.cons_scale = sh->cons_scale; a.ss = ss;
    a.N = sh->N; a.T = sh->T; a.Dobs = sh->D_obs; a.laplace = sh->laplace & 1; a.halo = (sh->laplace >> 1) & 1; a.row_lo = sh->row_lo;
    a.n_total = (int64_t)sh->S_mc * sh->N * sh->T;
    a.pred_out = pred_out; a.seeds = seeds; a.work = work;
    int grid = 0;
    const float* x0 = ss + sh->row_lo * D;
    int rc = -1;
    switch (D) {
#define CASE(D_) case D_: rc = gpode_shoot_fwd_d##D_(packed, M, S, x0, t2, B, kstages, &a, &grid, st); break;
        GPODE_FOR_EACH_D(CASE)
#undef CASE
        default: break;
    }
    if (rc != 0) return rc;
    shoot_sum_kernel<<<1, 256, 0, st>>>(work, grid, 2 + sh->D_obs, sums_out, grad_lik_var);
    GPODE_LAUNCH_CHECK();
    return 0;
}

static bool shoot_row_sums(int D, int M, int S, int64_t B) {
    switch (D) {
#define CASE(D_) case D_: return gpode_shoot_row_sums_d##D_(M, S, B);
        GPODE_FOR_EACH_D(CASE)
#undef CASE
        default: return false;
    }
}

extern "C" int64_t gpode_shoot_bwd_vrows(int D, int M, int S, int64_t n_rows) {
    if (D < 1 || D > GPODE_MAX_D || M < 1 || S < 1 || n_rows < 0) return -1;
    return shoot_row_sums(D, M, S, n_rows) ? 0 : 4 * n_rows;
}

extern "C" int gpode_shoot_bwd(const float* packed, int D, int M, int S, const gpode_shoot_t* sh, const float* ss,
                               const float* t2, const float* kstages, const float* seeds, const float* g_ll,
                               const float* g_cons, float* grad_ss, float* vrows, float* acc, void* stream) {
    if (int rc = check_shoot(sh, D)) return rc;
    const int64_t B = sh->row_hi - sh->row_lo;
    if (int rc = check_common(packed, D, M, S, B)) return rc;
    if (B == 0) return 0;
    GPODE_CHECK_ARG(ss && t2 && kstages && seeds && g_ll && g_cons && grad_ss && acc, "NULL argument");
    GPODE_CHECK_ARG(vrows != nullptr || shoot_row_sums(D, M, S, B),
                    "vrows is NULL, but this configuration needs %lld virtual rows (gpode_shoot_bwd_vrows)",
                    (long long)(4 * B));
    const int64_t VR = 4 * B, n_total = (int64_t)sh->S_mc * sh->N * sh->T;
    const float* x0 = ss + sh->row_lo * D;
    cudaStream_t st = (cudaStream_t)stream;
    float* vk = vrows ? vrows + VR * D : nullptr;
    switch (D) {
#define CASE(D_)                                                                                                   \
    case D_:                                                                                                       \
        return gpode_shoot_bwd_d##D_(packed, M, S, t2, B, x0, kstages, vrows, vk, acc, seeds, g_ll, g_cons,         \
                                     grad_ss, sh->row_lo, n_total, st);
        GPODE_FOR_EACH_D(CASE)
#undef CASE
        default: break;
    }
    gpode_set_error("state dimension D=%d outside 1..%d", D, GPODE_MAX_D);
    return -1;
}
