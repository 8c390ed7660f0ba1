// One translation unit per state dimension (compiled with -DGPODE_D=<1..8>) so the eight sets of register-resident
// kernels build in parallel.
#include "integrate_impl.cuh"

#ifndef GPODE_D
#error "compile with -DGPODE_D=<state dimension>"
#endif

#define GPODE_CAT_(a, b) a##b
#define GPODE_CAT(a, b) GPODE_CAT_(a, b)

int GPODE_CAT(gpode_vf_fwd_d, GPODE_D)(const float* packed, int M, int S, const float* x, float* f, int64_t B,
                                       cudaStream_t st) {
    return launch_vf_fwd<GPODE_D>(packed, M, S, x, f, B, st);
}
int GPODE_CAT(gpode_rk4_fwd_d, GPODE_D)(const float* packed, int M, int S, const float* x0, const float* t, int Tg,
                                        int64_t B, float* xs, float* kst, cudaStream_t st) {
    return launch_rk4_fwd<GPODE_D>(packed, M, S, x0, t, Tg, B, xs, kst, st);
}
int GPODE_CAT(gpode_rk4_bwd_d, GPODE_D)(const float* packed, int M, int S, const float* t, int Tg, int64_t B,
                                        const float* xs, const float* kst, const float* gxs, float* gx0, float* vy,
                                        float* vk, float* acc, cudaStream_t st) {
    return launch_rk4_bwd<GPODE_D>(packed, M, S, t, Tg, B, xs, kst, gxs, gx0, vy, vk, acc, st);
}
int GPODE_CAT(gpode_vf_bwd_d, GPODE_D)(const float* packed, int M, int S, const float* x, const float* f,
                                       const float* gf, float* gx, int64_t B, float* acc, cudaStream_t st) {
    return launch_vf_bwd<GPODE_D>(packed, M, S, x, f, gf, gx, B, acc, st);
}
int GPODE_CAT(gpode_fwd_sets_d, GPODE_D)(const float* packed, int M, int S, int n_sets, int64_t set_rows,
                                         const float* x0, const float* t, int Tg, float* out, cudaStream_t st) {
    return launch_fwd_sets<GPODE_D>(packed, M, S, n_sets, set_rows, x0, t, Tg, out, st);
}
int GPODE_CAT(gpode_shoot_fwd_d, GPODE_D)(const float* packed, int M, int S, const float* x0, const float* t, int64_t B,
                                          float* kst, const ShootArgs* sh, int* grid_out, cudaStream_t st) {
    return launch_rk4_fwd<GPODE_D, true>(packed, M, S, x0, t, 2, B, nullptr, kst, st, *sh, grid_out);
}
int GPODE_CAT(gpode_shoot_bwd_d, GPODE_D)(const float* packed, int M, int S, const float* t, int64_t B,
                                          const float* x0, const float* kst, float* vy, float* vk, float* acc,
                                          const float* seeds, const float* g_ll, const float* g_cons, float* grad_ss,
                                          int64_t row_lo, int64_t n_total, cudaStream_t st) {
    ShootBwd sb;
    sb.seeds = seeds; sb.g_ll = g_ll; sb.g_cons = g_cons; sb.grad_ss = grad_ss; sb.row_lo = row_lo; sb.n_total = n_total;
    return launch_rk4_bwd<GPODE_D, true>(packed, M, S, t, 2, B, x0, kst, nullptr, nullptr, vy, vk, acc, st, sb);
}
bool GPODE_CAT(gpode_shoot_row_sums_d, GPODE_D)(int M, int S, int64_t B) { return use_mma_row_sums<GPODE_D>(M, S, B); }
