// Per-inducing-point gradient contraction ("phase B" of the backward).
//
// For the RBF pathwise-update term f_upd,k(x) = var_k sum_m nu_km K_km(x) the gradients w.r.t. nu and Z contract over
// ROWS, not over inducing points, so they cannot be reduced inside the row-per-thread adjoint kernel without M*D
// cross-thread reductions per row. Instead the adjoint kernel writes (stage input y, cotangent kb) pairs -- "virtual
// rows" -- and this kernel maps one thread to one (output dim k, inducing point m) pair and streams the virtual rows
// through shared memory (broadcast reads; round-1 revision: one thread per inducing point m covering all D outputs,
// so the squared differences are computed once per m instead of once per (k,m)), accumulating in registers
//     T[k][m]    += kb_k K_km                      -> grad nu_km = var_k T
//     W[k][m][j] += kb_k K_km (y_j - Z_mj)         -> grad Z_mj  = sum_k c_km W / ell_kj^2
// (SURVEY.md section 8a row A7, "kernel" VJP lines; reference arithmetic: autograd through src/core/kernels.py:53-99
// and src/core/dsvgp.py:192).
#include "vf.cuh"

namespace {

constexpr int kPgThreads = 256;

constexpr int kPgTile = 128;  // virtual rows staged per pass

// thread = one inducing point m (all D outputs k: the squared differences (y_j - Z_mj)^2 are shared by the D kernels);
// a CTA holds G = 256 / M row-groups that each take every G-th row of the staged tile.
template <int D>
__global__ void __launch_bounds__(kPgThreads)
param_grad_kernel(const float* __restrict__ packed, const int M, const int S, const float* __restrict__ ys,
                  const float* __restrict__ kbs, const int64_t VR_host, const int64_t rows_per_cta,
                  float* __restrict__ acc, const int32_t* __restrict__ stats_dev, const int64_t rows_per_step) {
    // row count: the host's, or (6 accepted_steps + 1) rows_per_step read from the dopri5 stats block on the device
    int64_t VR = VR_host;
    if (stats_dev != nullptr) {
        const int64_t live = ((int64_t)6 * stats_dev[1] + 1) * rows_per_step;
        VR = live < VR_host ? live : VR_host;
    }
    constexpr int RP = VfShape<D>::RP, KS = VfShape<D>::KS, WP = VfShape<D>::WP;
    constexpr int DP = (D + 3) & ~3;
    constexpr int RW = 2 * DP;  // floats per staged row: y padded to DP, cotangent padded to DP
    extern __shared__ __align__(16) float pg_smem[];  // [2][kPgTile * RW] double buffer: tile t+1 lands while tile t is
    float* const srow[2] = {pg_smem, pg_smem + kPgTile * RW};  // consumed; re-used for the group reduction at the end

    const float* __restrict__ kern = packed + D * ((((S + 1) >> 1) + 31) & ~31) * RP;
    const float* __restrict__ wnp = kern + M * KS;  // -w, [j][WP] with outputs k along the row
    int m, group, G;
    if (M >= kPgThreads) {
        m = blockIdx.y * kPgThreads + threadIdx.x;
        group = 0;
        G = 1;
    } else {  // the launch sizes the CTA to G*M threads rounded up to a warp: groups are packed back to back
        G = kPgThreads / M;
        group = threadIdx.x / M;
        m = threadIdx.x - group * M;
        if (group >= G) m = M;  // idle tail threads
    }
    const bool active = m < M;
    const int mm = active ? m : 0;

    // full output pairs ride in FFMA2, the odd last output in scalar FMAs (a half-empty pair costs the FMA pipe,
    // which bounds this kernel, as much as a full one)
    constexpr int KF = D / 2, KFA = KF > 0 ? KF : 1;
    constexpr bool kOdd = (D & 1) != 0;
    float z[D], wl[D];
    float2 wn[D][KFA];  // -w, output pairs (same packing as the integrator kernels)
#pragma unroll
    for (int j = 0; j < D; ++j) {
        z[j] = __ldg(kern + mm * KS + j);
#pragma unroll
        for (int kp = 0; kp < KF; ++kp)
            wn[j][kp] = make_float2(__ldg(wnp + j * WP + 2 * kp), __ldg(wnp + j * WP + 2 * kp + 1));
        wl[j] = __ldg(wnp + j * WP + D - 1);
    }
    float2 T2[KFA], W2[KFA][D];
    float Tl = 0.f, Wl[D];
#pragma unroll
    for (int j = 0; j < D; ++j) Wl[j] = 0.f;
#pragma unroll
    for (int kp = 0; kp < KF; ++kp) {
        T2[kp] = make_float2(0.f, 0.f);
#pragma unroll
        for (int j = 0; j < D; ++j) W2[kp][j] = make_float2(0.f, 0.f);
    }

    const int64_t r_begin = (int64_t)blockIdx.x * rows_per_cta;
    const int64_t r_end = r_begin + rows_per_cta < VR ? r_begin + rows_per_cta : VR;
    // each thread moves up to kPre (y, cotangent) element pairs of a tile: global -> registers (in flight during the
    // compute of the previous tile) -> shared memory; one barrier per tile
    constexpr int kPre = (kPgTile * D + 127) / 128;  // the CTA has at least 128 threads
    float py[kPre], pk[kPre];
    auto fetch = [&](const int64_t base, const int n) {
#pragma unroll
        for (int q = 0; q < kPre; ++q) {
            const int i = threadIdx.x + q * blockDim.x;
            const bool ok = i < n * D;
            py[q] = ok ? __ldg(ys + base * D + i) : 0.f;
            pk[q] = ok ? __ldg(kbs + base * D + i) : 0.f;
        }
    };
    auto stash = [&](float* __restrict__ dst, const int n) {
#pragma unroll
        for (int q = 0; q < kPre; ++q) {
            const int i = threadIdx.x + q * blockDim.x;
            if (i < n * D) {
                const int r = i / D, j = i - r * D;
                dst[r * RW + j] = py[q];
                dst[r * RW + DP + j] = pk[q];
            }
        }
    };
    auto tile_rows = [&](const int64_t base) { return (int)((r_end - base) < kPgTile ? (r_end - base) : kPgTile); };
    int buf = 0;
    if (r_begin < r_end) {
        fetch(r_begin, tile_rows(r_begin));
        stash(srow[0], tile_rows(r_begin));
    }
    __syncthreads();
    for (int64_t base = r_begin; base < r_end; base += kPgTile, buf ^= 1) {
        const int n = tile_rows(base);
        const int64_t next = base + kPgTile;
        const int n_next = next < r_end ? tile_rows(next) : 0;
        if (n_next) fetch(next, n_next);
        const float* __restrict__ cur = srow[buf];
        if (active) {
#pragma unroll 2
            for (int r = group; r < n; r += G) {
                float y[DP], kb[DP];
                lds_vec<DP>(y, cur + r * RW);
                lds_vec<DP>(kb, cur + r * RW + DP);
                float d[D], dd[D];
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    d[j] = y[j] - z[j];
                    dd[j] = d[j] * d[j];
                }
#pragma unroll
                for (int kp = 0; kp < KF; ++kp) {
                    float2 e = make_float2(0.f, 0.f);
#pragma unroll
                    for (int j = 0; j < D; ++j) e = ffma2(dd[j], wn[j][kp], e);
                    const float2 K = make_float2(gpode_ex2(e.x), gpode_ex2(e.y));
                    const float2 p = fmul2(make_float2(kb[2 * kp], kb[2 * kp + 1]), K);
                    T2[kp] = fadd2(T2[kp], p);
#pragma unroll
                    for (int j = 0; j < D; ++j) W2[kp][j] = ffma2(d[j], p, W2[kp][j]);
                }
                if constexpr (kOdd) {
                    float e = 0.f;
#pragma unroll
                    for (int j = 0; j < D; ++j) e = fmaf(dd[j], wl[j], e);
                    const float p = kb[D - 1] * gpode_ex2(e);
                    Tl += p;
#pragma unroll
                    for (int j = 0; j < D; ++j) Wl[j] = fmaf(d[j], p, Wl[j]);
                }
            }
        }
        if (n_next) stash(srow[buf ^ 1], n_next);  // the other buffer's readers finished before the previous barrier
        __syncthreads();
    }
    // ---- this CTA's partial sums -> its own row of the accumulator block (no atomics: the result must not depend on
    // scheduling). The G row-groups of the CTA are added in group order through shared memory.
    const GpodeAcc a = gpode_acc_layout(D, M);
    constexpr int NE = D + D * D;  // per inducing point: T[k] | W[j][k]
    float val[NE];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        const bool last = kOdd && k == D - 1;
        const int kp = (k >> 1) < KF ? (k >> 1) : 0;
        val[k] = last ? Tl : ((k & 1) ? T2[kp].y : T2[kp].x);
#pragma unroll
        for (int j = 0; j < D; ++j) val[D + j * D + k] = last ? Wl[j] : ((k & 1) ? W2[kp][j].y : W2[kp][j].x);
    }
    float* __restrict__ row = acc + a.off_tw + (size_t)blockIdx.x * M * NE;
    if (G == 1) {
        if (active) {
#pragma unroll
            for (int e = 0; e < NE; ++e) row[(size_t)m * NE + e] = val[e];
        }
    } else {
        // [M][NE] float64; the staged tiles are dead (barrier at the end of the loop)
        double* __restrict__ red = reinterpret_cast<double*>(pg_smem);
        for (int g = 0; g < G; ++g) {
            if (active && group == g) {
#pragma unroll
                for (int e = 0; e < NE; ++e) red[m * NE + e] = (g == 0 ? 0.0 : red[m * NE + e]) + (double)val[e];
            }
            __syncthreads();
        }
        for (int i = threadIdx.x; i < M * NE; i += blockDim.x) row[i] = (float)red[i];
    }
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) reinterpret_cast<int*>(acc)[1] = (int)gridDim.x;
}

// Accumulator rows -> parameter gradients. Rows are added in row order in float64 (fixed assignment of rows to warps,
// warps added in warp order), the contractions with nu / var / ell are done in float64 as well, and every output is
// rounded to float32 once. CTA b < ceil(M / kFinM) owns kFinM inducing points (grad_nu, grad_Z), the last CTA the
// lengthscale / variance sums (grad_ell, grad_var).
constexpr int kFinM = 4, kFinThreads = 256, kFinWarps = kFinThreads / 32;
constexpr int kFinMaxChunk = kFinM * (GPODE_MAX_D + GPODE_MAX_D * GPODE_MAX_D);  // 288
constexpr int kFinPerLane = (kFinMaxChunk + 31) / 32;                             // 9

__global__ void __launch_bounds__(kFinThreads)
grads_finalize_kernel(const int D, const int M, const float* __restrict__ nu, const float* __restrict__ ell,
                      const float* __restrict__ var, const float* __restrict__ acc, float* __restrict__ g_ell,
                      float* __restrict__ g_var, float* __restrict__ g_Z, float* __restrict__ g_nu) {
    __shared__ double part[kFinWarps][kFinMaxChunk];
    __shared__ double tot[kFinMaxChunk];
    const GpodeAcc a = gpode_acc_layout(D, M);
    const int* hdr = reinterpret_cast<const int*>(acc);
    const int n_mg = (M + kFinM - 1) / kFinM;
    const bool av = (int)blockIdx.x == n_mg;
    const int NE = a.n_tw_m;
    const int m0 = blockIdx.x * kFinM, cnt = av ? 0 : (M - m0 < kFinM ? M - m0 : kFinM);
    if (!av && hdr[2] > 0) {   // row sums of the tensor-core shooting adjoint (float64 rows, common.cuh)
        const int NR = a.n_rs_m;
        const double* __restrict__ rs = reinterpret_cast<const double*>(acc + a.off_rs) + (size_t)m0 * NR;
        gpode_sum_rows_ordered<kFinPerLane>(rs, (size_t)M * NR, hdr[2], cnt * NR, kFinMaxChunk, &part[0][0], tot);
        const double inv_2ln2 = 1.0 / (double)(-GPODE_NEG_2LN2);   // the kernel's float factor 2 ln2, exactly
        for (int i = threadIdx.x; i < cnt * D; i += blockDim.x) {
            const int mm = i / D, k = i - mm * D;
            g_nu[k * M + m0 + mm] = (float)((double)var[k] * tot[mm * NR + k] * inv_2ln2);   // var_k T[k][m]
            // grad_Z[m][j] = sum_k c_km W[k][m][j] / ell_kj^2 = -sum_rows d_j tq_j
            g_Z[(m0 + mm) * D + k] = (float)(-tot[mm * NR + D + k]);
        }
        return;
    }
    const int chunk = av ? a.n_av : cnt * NE;                       // contiguous floats of every row this CTA adds up
    const int n_rows = av ? hdr[0] : hdr[1];
    const size_t stride = av ? (size_t)a.n_av : (size_t)M * NE;
    const float* __restrict__ base = acc + (av ? a.off_av : a.off_tw + (size_t)m0 * NE);
    gpode_sum_rows_ordered<kFinPerLane>(base, stride, n_rows, chunk, kFinMaxChunk, &part[0][0], tot);
    if (av) {
        for (int i = threadIdx.x; i < D * D; i += blockDim.x) g_ell[i] = (float)(-tot[i] / (double)ell[i]);
        for (int k = threadIdx.x; k < D; k += blockDim.x) g_var[k] = (float)(0.5 * tot[D * D + k] / (double)var[k]);
        return;
    }
    for (int i = threadIdx.x; i < cnt * D; i += blockDim.x) {   // grad_nu[k][m] = var_k T[k][m]
        const int mm = i / D, k = i - mm * D;
        g_nu[k * M + m0 + mm] = (float)((double)var[k] * tot[mm * NE + k]);
    }
    for (int i = threadIdx.x; i < cnt * D; i += blockDim.x) {   // grad_Z[m][j] = sum_k var_k nu_km W[k][m][j] / ell_kj^2
        const int mm = i / D, j = i - mm * D;
        double sz = 0.0;
        for (int k = 0; k < D; ++k) {
            const double l = (double)ell[k * D + j];
            sz += (double)var[k] * (double)nu[k * M + m0 + mm] * tot[mm * NE + D + j * D + k] / (l * l);
        }
        g_Z[(m0 + mm) * D + j] = (float)sz;
    }
}

}  // namespace

static size_t pg_smem_bytes(int D, int M) {
    const int DP = (D + 3) & ~3;
    const size_t tiles = (size_t)2 * kPgTile * 2 * DP * sizeof(float);
    const size_t red = M < kPgThreads / 2 + 1 ? (size_t)M * (D + D * D) * sizeof(double) : 0;  // only when G >= 2
    return tiles > red ? tiles : red;
}

int gpode_param_grad_launch(const float* packed, int D, int M, int S, const float* ys, const float* kbs, int64_t VR,
                            float* acc, cudaStream_t stream, const int32_t* stats_dev, int64_t rows_per_step) {
    if (VR == 0) return 0;
    int sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // (more resident CTAs -- 80 or 64 registers instead of 124 -- were measured: 1.48 / 1.44 ms against 1.46: the kernel
    // is bound by the FP32 pipe, not by occupancy)
    const int gy = M >= kPgThreads ? (M + kPgThreads - 1) / kPgThreads : 1;
    // rows per CTA: enough CTAs to fill the machine (~4 per SM across gy), but at least one full tile each
    int64_t want_ctas = (int64_t)sms * 4 / gy;
    if (want_ctas < 1) want_ctas = 1;
    if (want_ctas > GPODE_ACC_CAP_TW) want_ctas = GPODE_ACC_CAP_TW;  // one accumulator row per blockIdx.x
    int64_t rows_per_cta = (VR + want_ctas - 1) / want_ctas;
    rows_per_cta = ((rows_per_cta + kPgTile - 1) / kPgTile) * kPgTile;
    const int64_t gx = (VR + rows_per_cta - 1) / rows_per_cta;
    dim3 grid((unsigned)gx, (unsigned)gy);
    const int threads = M >= kPgThreads ? kPgThreads : (((kPgThreads / M) * M + 31) / 32) * 32;
    switch (D) {
#define GPODE_PG_CASE(D_)                                                                                        \
    case D_:                                                                                                     \
        GPODE_CUDA(cudaFuncSetAttribute(param_grad_kernel<D_>, cudaFuncAttributeMaxDynamicSharedMemorySize,      \
                                        (int)pg_smem_bytes(D_, M)));                                             \
        param_grad_kernel<D_><<<grid, threads, pg_smem_bytes(D_, M), stream>>>(                                 \
            packed, M, S, ys, kbs, VR, rows_per_cta, acc, stats_dev, rows_per_step);                             \
        break;
        GPODE_PG_CASE(1) GPODE_PG_CASE(2) GPODE_PG_CASE(3) GPODE_PG_CASE(4)
        GPODE_PG_CASE(5) GPODE_PG_CASE(6) GPODE_PG_CASE(7) GPODE_PG_CASE(8)
#undef GPODE_PG_CASE
        default:
            gpode_set_error("state dimension D=%d outside 1..%d", D, GPODE_MAX_D);
            return -1;
    }
    GPODE_LAUNCH_CHECK();
    return 0;
}

extern "C" int64_t gpode_acc_floats(int D, int M) { return gpode_acc_layout(D, M).total; }
extern "C" int64_t gpode_acc_header_floats(void) { return GPODE_ACC_HDR; }

extern "C" int gpode_grads_finalize(const gpode_cache_t* c, const float* acc, float* grad_ell, float* grad_var,
                                    float* grad_Z, float* grad_nu, void* stream) {
    GPODE_CHECK_ARG(c != nullptr && acc != nullptr, "cache / acc is NULL");
    GPODE_CHECK_ARG(c->Z && c->nu && c->ell && c->var, "cache needs Z, nu, ell, var");
    GPODE_CHECK_ARG(grad_ell && grad_var && grad_Z && grad_nu, "NULL output");
    GPODE_CHECK_ARG(c->D >= 1 && c->D <= GPODE_MAX_D, "state dimension D=%d outside 1..%d", c->D, GPODE_MAX_D);
    const int n_mg = (c->M + kFinM - 1) / kFinM;
    grads_finalize_kernel<<<n_mg + 1, kFinThreads, 0, (cudaStream_t)stream>>>(c->D, c->M, c->nu, c->ell, c->var, acc,
                                                                             grad_ell, grad_var, grad_Z, grad_nu);
    GPODE_LAUNCH_CHECK();
    return 0;
}
