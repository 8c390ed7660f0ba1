// Batched in-shared-memory Cholesky / triangular solves for the per-output-dimension Kzz whitening of
// DSVGP_Layer.build_cache (reference src/core/dsvgp.py:110-122), its backward, and the whitened KL (dsvgp.py:199-230).
//
//   forward  (one CTA per output dim k):  K = K_k(Z,Z) + jitter I;  L = chol(K);  p = rff_forward(Z)_k;
//                                          s = L^-1 p;  nu_k = L^-T (u_k - s)
//   backward (given nub = dLoss/dnu_k):    rb = L^-1 nub;  ub = rb;  pb = -L^-T rb;
//                                          P  = -Phi(w rb^T - rb s^T), w = u_k - s   (= Phi(L^T Lbar), rank-2 form)
//                                          Kb = sym(L^-T P L^-1)  ->  Z, lengthscale, variance gradients through the
//                                          RBF; pb -> the RFF VJP evaluated at x = Z (SURVEY.md section 8a, "Derived
//                                          maths").
// The M x M tiles live in shared memory in float64 (M <= GPODE_MAX_M_F64) or float32 (M <= GPODE_MAX_M): Kzz + 1e-5 I
// has a condition number around 1e5, so float64 accumulation keeps nu at the float64-arbiter level instead of adding
// this kernel's round-off on top of the reference's (tests/ arbitrate with the float64 oracle).
#include "whiten.cuh"
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

namespace {

__device__ __forceinline__ int ld_for(int M) { return (M & 1) ? M : M + 1; }

// p_m = rff_forward(Z)_{m,k} for every inducing point: one warp per point (rff_at_point)
__device__ void rff_at_Z(const gpode_cache_t& c, int k, double* p_out) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const float ak = sqrtf(c.var[k] / (float)c.S);
    for (int m = warp; m < c.M; m += nwarps) {
        const double acc = rff_at_point(c, k, m, ak);
        if (lane == 0) p_out[m] = acc;
    }
}

// v <- L^-1 v (warp 0 only; caller syncs the CTA afterwards)
template <typename Real>
__device__ void trsv_lower(const Real* L, int M, int ld, Real* v, const Real* dinv) {
    if (threadIdx.x >= 32) return;
    const int lane = threadIdx.x;
    for (int c = 0; c < M; ++c) {
        __syncwarp();
        const Real rc = v[c] * dinv[c];
        __syncwarp();
        if (lane == 0) v[c] = rc;
        for (int i = c + 1 + lane; i < M; i += 32) v[i] -= L[i * ld + c] * rc;
    }
    __syncwarp();
}

// v <- L^-T v (warp 0 only)
template <typename Real>
__device__ void trsv_lower_t(const Real* L, int M, int ld, Real* v, const Real* dinv) {
    if (threadIdx.x >= 32) return;
    const int lane = threadIdx.x;
    for (int c = M - 1; c >= 0; --c) {
        __syncwarp();
        const Real rc = v[c] * dinv[c];
        __syncwarp();
        if (lane == 0) v[c] = rc;
        for (int i = lane; i < c; i += 32) v[i] -= L[c * ld + i] * rc;
    }
    __syncwarp();
}

template <typename Real>
__global__ void whiten_fwd_kernel(const gpode_cache_t c, const float* __restrict__ u, const float jitter,
                                  float* __restrict__ nu_out, double* __restrict__ L_out, double* __restrict__ sp_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int k = blockIdx.x, M = c.M, D = c.D, ld = ld_for(M);
    Real* A = reinterpret_cast<Real*>(smem_raw);  // (M+1) x ld: K then L, last row p^T -> s^T
    double* pvec = reinterpret_cast<double*>(A + (size_t)(M + 1) * ld + ((M + 1) * ld & 1));
    Real* wv = reinterpret_cast<Real*>(pvec + M);
    __shared__ Real dinv[GPODE_MAX_M];   // 1 / L_mm

    const float* ellk = c.ell + k * D;
    const double vark = (double)c.var[k];
    double inv_l[GPODE_MAX_D];
    for (int j = 0; j < D; ++j) inv_l[j] = 1.0 / (double)ellk[j];
    for (int i = threadIdx.x; i < M * M; i += blockDim.x) {
        const int m = i / M, n = i - m * M;
        if (n <= m) A[m * ld + n] = (Real)(rbf_entry(c.Z, inv_l, vark, D, m, n) + (m == n ? (double)jitter : 0.0));
    }
    rff_at_Z(c, k, pvec);
    __syncthreads();
    for (int m = threadIdx.x; m < M; m += blockDim.x) A[M * ld + m] = (Real)pvec[m];
    chol_inplace<Real>(A, M, M + 1, ld, dinv);
    // w = u_k - s ; nu = L^-T w
    for (int m = threadIdx.x; m < M; m += blockDim.x) {
        wv[m] = (Real)u[m * D + k] - A[M * ld + m];
        sp_out[((size_t)k * 2 + 0) * M + m] = (double)A[M * ld + m];
        sp_out[((size_t)k * 2 + 1) * M + m] = pvec[m];
    }
    for (int i = threadIdx.x; i < M * M; i += blockDim.x) {
        const int m = i / M, n = i - m * M;
        L_out[(size_t)k * M * M + i] = n <= m ? (double)A[m * ld + n] : 0.0;
    }
    __syncthreads();
    trsv_lower_t<Real>(A, M, ld, wv, dinv);
    __syncthreads();
    for (int m = threadIdx.x; m < M; m += blockDim.x) nu_out[k * M + m] = (float)wv[m];
}

// Batched Monte-Carlo prediction: n_sets function draws share Z and the hyper-parameters, hence ONE factor L per
// output dimension; a set only differs in p = rff_forward(Z) and u. One CTA per (output dim, set) reloads the float64
// factor from L2 and does the two triangular solves: nu = L^-T (u - L^-1 p).
template <typename Real>
__global__ void whiten_solve_sets_kernel(gpode_cache_t c, const float* __restrict__ u,
                                         const double* __restrict__ L_in, float* __restrict__ nu_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int k = blockIdx.x, M = c.M, D = c.D, S = c.S, ld = ld_for(M);
    {
        const size_t set = blockIdx.y;
        c.omega += set * D * S * D;
        c.phase += set * S * D;
        c.w += set * S * D;
        u += set * M * D;
        nu_out += set * D * M;
    }
    Real* L = reinterpret_cast<Real*>(smem_raw);
    double* pvec = reinterpret_cast<double*>(L + (size_t)M * ld + ((M * ld) & 1));
    Real* sv = reinterpret_cast<Real*>(pvec + M);
    __shared__ Real dinv[GPODE_MAX_M];
    for (int i = threadIdx.x; i < M * M; i += blockDim.x) {
        const int m = i / M, n = i - m * M;
        L[m * ld + n] = (Real)L_in[(size_t)k * M * M + i];
    }
    for (int m = threadIdx.x; m < M; m += blockDim.x) dinv[m] = (Real)(1.0 / L_in[(size_t)k * M * M + (size_t)m * M + m]);
    rff_at_Z(c, k, pvec);
    __syncthreads();
    for (int m = threadIdx.x; m < M; m += blockDim.x) sv[m] = (Real)pvec[m];
    __syncthreads();
    trsv_lower<Real>(L, M, ld, sv, dinv);
    __syncthreads();
    for (int m = threadIdx.x; m < M; m += blockDim.x) sv[m] = (Real)u[m * D + k] - sv[m];
    __syncthreads();
    trsv_lower_t<Real>(L, M, ld, sv, dinv);
    __syncthreads();
    for (int m = threadIdx.x; m < M; m += blockDim.x) nu_out[k * M + m] = (float)sv[m];
}

template <typename Real>
__global__ void whiten_bwd_kernel(const gpode_cache_t c, const float* __restrict__ u, const double* __restrict__ L_in,
                                  const double* __restrict__ sp_in, const float* __restrict__ gnu,
                                  float* __restrict__ g_u, float* __restrict__ g_Z, float* __restrict__ g_ell,
                                  float* __restrict__ g_var) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int k = blockIdx.x, M = c.M, D = c.D, S = c.S, ld = ld_for(M);
    Real* L = reinterpret_cast<Real*>(smem_raw);
    Real* P = L + (size_t)M * ld;
    Real* rb = P + (size_t)M * ld;  // M
    Real* pb = rb + M;              // M
    Real* wv = pb + M;              // M
    Real* sv = wv + M;              // M
    // float64 block-reduction scratch: [16 warps][D + 1] lengthscale / variance partials, then this CTA's share of
    // grad_Z, gzs[M][D] (read by cluster rank 0 through distributed shared memory)
    double* red = reinterpret_cast<double*>(sv + M + ((4 * M + 2 * M * ld) & 1));
    double* gzs = red + 16 * (D + 1);

    const float* ellk = c.ell + k * D;
    const double vark = (double)c.var[k];
    double inv_l[GPODE_MAX_D];
    for (int j = 0; j < D; ++j) inv_l[j] = 1.0 / (double)ellk[j];
    for (int i = threadIdx.x; i < M * M; i += blockDim.x) {
        const int m = i / M, n = i - m * M;
        L[m * ld + n] = (Real)L_in[(size_t)k * M * M + i];
    }
    __shared__ Real dinv[GPODE_MAX_M];
    for (int m = threadIdx.x; m < M; m += blockDim.x) {
        dinv[m] = (Real)(1.0 / L_in[(size_t)k * M * M + (size_t)m * M + m]);
        const Real s = (Real)sp_in[((size_t)k * 2 + 0) * M + m];
        sv[m] = s;
        wv[m] = (Real)u[m * D + k] - s;
        rb[m] = (Real)gnu[k * M + m];
    }
    __syncthreads();
    trsv_lower<Real>(L, M, ld, rb, dinv);  // rb = L^-1 nub  (= grad wrt u_k)
    __syncthreads();
    for (int m = threadIdx.x; m < M; m += blockDim.x) {
        pb[m] = -rb[m];
        g_u[m * D + k] = (float)rb[m];
    }
    __syncthreads();
    trsv_lower_t<Real>(L, M, ld, pb, dinv);  // pb = -L^-T rb
    // P = -Phi(w rb^T - rb s^T)
    for (int i = threadIdx.x; i < M * M; i += blockDim.x) {
        const int m = i / M, n = i - m * M;
        Real v = (Real)0;
        if (n <= m) {
            v = -(wv[m] * rb[n] - rb[m] * sv[n]);
            if (n == m) v *= (Real)0.5;
        }
        P[m * ld + n] = v;
    }
    __syncthreads();
    // Y = L^-T P, then X = Y L^-1: 2 M independent triangular solves -- every COLUMN of P in the first pass, every ROW
    // in the second -- each done by one thread from start to end, so neither pass needs a single barrier (round 1
    // eliminated row by row with the whole CTA: ~4 M barriers, which was most of this kernel's 0.4 ms at M = 100).
    // All threads read the same L entry at the same time (shared-memory broadcast); the leading dimension is odd, so
    // the per-thread columns / rows of P sit in different banks.
    // (Splitting every solve over four lanes of a warp -- 4 M busy threads, two xor shuffles and a __syncwarp per
    // substitution step -- was measured: 0.305 ms against 0.288 ms; the fixed cost per step outweighs the shorter dot
    // products at M = 100.)
    for (int n = threadIdx.x; n < M; n += blockDim.x) {          // column n:  L^T y = p  (back substitution)
        for (int i = M - 1; i >= 0; --i) {
            Real a0 = P[i * ld + n], a1 = (Real)0;
            int r = i + 1;
            for (; r + 1 < M; r += 2) {
                a0 -= L[r * ld + i] * P[r * ld + n];
                a1 -= L[(r + 1) * ld + i] * P[(r + 1) * ld + n];
            }
            if (r < M) a0 -= L[r * ld + i] * P[r * ld + n];
            P[i * ld + n] = (a0 + a1) * dinv[i];
        }
    }
    __syncthreads();
    for (int r = threadIdx.x; r < M; r += blockDim.x) {          // row r:  x L = y  (from the last column down)
        for (int cidx = M - 1; cidx >= 0; --cidx) {
            Real a0 = P[r * ld + cidx], a1 = (Real)0;
            int q = cidx + 1;
            for (; q + 1 < M; q += 2) {
                a0 -= P[r * ld + q] * L[q * ld + cidx];
                a1 -= P[r * ld + q + 1] * L[(q + 1) * ld + cidx];
            }
            if (q < M) a0 -= P[r * ld + q] * L[q * ld + cidx];
            P[r * ld + cidx] = (a0 + a1) * dinv[cidx];
        }
    }
    __syncthreads();
    // No floating-point atomics below: every sum is taken in a fixed order, so repeated calls are bitwise identical.
    // RBF backward with Kb = (X + X^T)/2: thread = (inducing point m, slice of the partner points n)
    double gvar = 0.0;           // this thread's share of the variance / lengthscale gradients (both parts)
    double gl[GPODE_MAX_D];
    for (int j = 0; j < D; ++j) gl[j] = 0.0;
    {
        const int parts = blockDim.x / M;  // launches use 128 threads for M < 64 and 512 for M <= 160: parts >= 1
        const int m = threadIdx.x % M, part = threadIdx.x / M;
        double gz[GPODE_MAX_D];
        for (int j = 0; j < D; ++j) gz[j] = 0.0;
        if (part < parts) {
            for (int n = part; n < M; n += parts) {
                const double kb = 0.5 * ((double)P[m * ld + n] + (double)P[n * ld + m]);
                const double E = kb * rbf_entry(c.Z, inv_l, vark, D, m, n);
                gvar += E;
                for (int j = 0; j < D; ++j) {
                    const double d = ((double)c.Z[m * D + j] - (double)c.Z[n * D + j]) * inv_l[j];
                    gz[j] -= 2.0 * E * d * inv_l[j];
                    gl[j] += E * d * d * inv_l[j];
                }
            }
        }
        gvar /= vark;
        for (int p = 0; p < parts; ++p) {  // the slices of one inducing point are added in slice order
            if (part == p)
                for (int j = 0; j < D; ++j) gzs[m * D + j] = (p == 0 ? 0.0 : gzs[m * D + j]) + gz[j];
            __syncthreads();
        }
    }
    // RFF VJP at x = Z with cotangent pb (only output dim k): one warp per inducing point, lanes over features
    {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
        const float ak = sqrtf(c.var[k] / (float)S);
        for (int m = warp; m < M; m += nwarps) {
            double G[GPODE_MAX_D];
            const double pbm = (double)pb[m];
            rff_vjp_at_point(c, k, m, pbm, ak, G);
            for (int j = 0; j < D; ++j) {
                double v = G[j];
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                if (lane == 0) {
                    gzs[m * D + j] += v;  // inducing point m belongs to this warp alone
                    gl[j] += -v * (double)c.Z[m * D + j] / (double)ellk[j];
                }
            }
            if (lane == 0) gvar += pbm * sp_in[((size_t)k * 2 + 1) * M + m] / (2.0 * vark);
        }
        // block sums of gvar, gl[j]: warp shuffles, then the warps in warp order
        for (int o = 16; o > 0; o >>= 1) gvar += __shfl_xor_sync(0xffffffffu, gvar, o);
        for (int j = 0; j < D; ++j)
            for (int o = 16; o > 0; o >>= 1) gl[j] += __shfl_xor_sync(0xffffffffu, gl[j], o);
        if (lane == 0) {
            red[warp * (D + 1) + D] = gvar;
            for (int j = 0; j < D; ++j) red[warp * (D + 1) + j] = gl[j];
        }
        __syncthreads();
        for (int j = threadIdx.x; j < D + 1; j += blockDim.x) {
            double t = 0.0;
            for (int w = 0; w < nwarps; ++w) t += red[w * (D + 1) + j];
            if (j < D) g_ell[k * D + j] = (float)t;
            else g_var[k] = (float)t;
        }
    }
    // grad_Z sums over the output dimensions = over the CTAs of this cluster: rank 0 adds them in rank order, reading
    // the other CTAs' gzs through distributed shared memory
    cg::cluster_group cluster = cg::this_cluster();
    cluster.sync();
    if (cluster.block_rank() == 0) {
        for (int i = threadIdx.x; i < M * D; i += blockDim.x) {
            double t = 0.0;
            for (int r = 0; r < D; ++r) t += cluster.map_shared_rank(gzs, r)[i];
            g_Z[i] = (float)t;
        }
    }
    cluster.sync();  // keep every CTA's shared memory alive until rank 0 has read it
}

// ---- whitened KL (dsvgp.py:199-230): one CTA, float64 accumulation ---------------------------------------------
__global__ void kl_fwd_kernel(const float* __restrict__ Um, const float* __restrict__ Ls, int D, int M,
                              float* __restrict__ out) {
    __shared__ double red[32];
    const int npk = M * (M + 1) / 2;
    double acc = 0.0;
    for (int i = threadIdx.x; i < M * D; i += blockDim.x) acc += (double)Um[i] * (double)Um[i];
    for (int i = threadIdx.x; i < D * npk; i += blockDim.x) acc += (double)Ls[i] * (double)Ls[i];
    // diagonal entries of row-major tril packing sit at index r(r+1)/2 + r
    for (int i = threadIdx.x; i < D * M; i += blockDim.x) {
        const int d = i / M, r = i - d * M;
        const double v = (double)Ls[(size_t)d * npk + (size_t)r * (r + 1) / 2 + r];
        acc -= log(v * v);
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
        out[0] = (float)(0.5 * (t - (double)M * (double)D));
    }
}

__global__ void kl_bwd_kernel(const float* __restrict__ Um, const float* __restrict__ Ls, int D, int M,
                              const float* __restrict__ gkl, float* __restrict__ gUm, float* __restrict__ gLs) {
    const int npk = M * (M + 1) / 2;
    const float g = gkl[0];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < M * D; i += gridDim.x * blockDim.x) gUm[i] = g * Um[i];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < D * npk; i += gridDim.x * blockDim.x) {
        const int p = i % npk;
        // is p a diagonal slot?  r = floor((sqrt(8p+1)-1)/2), diagonal iff p == r(r+1)/2 + r
        int r = (int)((sqrt(8.0 * (double)p + 1.0) - 1.0) * 0.5);
        while ((r + 1) * (r + 2) / 2 <= p) ++r;
        while (r * (r + 1) / 2 > p) --r;
        const bool diag = (p == r * (r + 1) / 2 + r);
        const float v = Ls[i];
        gLs[i] = g * (v - (diag ? 1.0f / v : 0.0f));
    }
}

// ---- inducing sample u = Um + Us_sqrt eps (dsvgp.py:78-90, full-rank branch) straight from the PACKED factor --------
// u[n][d] = Um[n][d] + sum_{m <= n} L_d[n][m] eps[m][d]; one thread per (n, d). Replaces the tril scatter of the
// (D, M, M) factor + a batched matrix product (and their backward: two products + an index-put) of the eager mirror.
__global__ void inducing_sample_fwd_kernel(const float* __restrict__ Um, const float* __restrict__ Ls,
                                           const float* __restrict__ eps, int D, int M, float* __restrict__ u) {
    const int npk = M * (M + 1) / 2;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < M * D; i += gridDim.x * blockDim.x) {
        const int n = i / D, d = i - n * D;
        const float* __restrict__ row = Ls + (size_t)d * npk + (size_t)n * (n + 1) / 2;
        float a0 = 0.f, a1 = 0.f;
        int m = 0;
        for (; m + 1 <= n; m += 2) {
            a0 = fmaf(row[m], eps[m * D + d], a0);
            a1 = fmaf(row[m + 1], eps[(m + 1) * D + d], a1);
        }
        if (m <= n) a0 = fmaf(row[m], eps[m * D + d], a0);
        u[i] = Um[i] + (a0 + a1);
    }
}
// grad_Ls[d][n][m] = g_u[n][d] eps[m][d]  (m <= n);  grad_Um = g_u is the caller's (identity)
__global__ void inducing_sample_bwd_kernel(const float* __restrict__ eps, const float* __restrict__ gu, int D, int M,
                                           float* __restrict__ gLs) {
    const int npk = M * (M + 1) / 2;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < D * npk; i += gridDim.x * blockDim.x) {
        const int d = i / npk, p = i - d * npk;
        int n = (int)((sqrt(8.0 * (double)p + 1.0) - 1.0) * 0.5);
        while ((n + 1) * (n + 2) / 2 <= p) ++n;
        while (n * (n + 1) / 2 > p) --n;
        const int m = p - n * (n + 1) / 2;
        gLs[i] = gu[n * D + d] * eps[m * D + d];
    }
}

template <typename Real>
size_t fwd_smem(int M) {
    const int ld = (M & 1) ? M : M + 1;
    return sizeof(Real) * ((size_t)(M + 1) * ld + 2) + sizeof(double) * M + sizeof(Real) * M + 16;
}
template <typename Real>
size_t solve_smem(int M) {
    const int ld = (M & 1) ? M : M + 1;
    return sizeof(Real) * ((size_t)M * ld + 2) + sizeof(double) * M + sizeof(Real) * M + 16;
}
template <typename Real>
size_t bwd_smem(int M, int D) {
    const int ld = (M & 1) ? M : M + 1;
    return sizeof(Real) * (2 * (size_t)M * ld + 4 * M + 2) + sizeof(double) * (16 * (D + 1) + (size_t)M * D + 1) + 16;
}

int check_cache(const gpode_cache_t* c, bool need_nu) {
    GPODE_CHECK_ARG(c != nullptr, "cache is NULL");
    GPODE_CHECK_ARG(c->D >= 1 && c->D <= GPODE_MAX_D, "state dimension D=%d outside 1..%d", c->D, GPODE_MAX_D);
    GPODE_CHECK_ARG(c->M >= 1 && c->M <= GPODE_MAX_M, "M=%d outside 1..%d (shared-memory Cholesky tile)", c->M,
                    GPODE_MAX_M);
    GPODE_CHECK_ARG(c->S >= 1, "S=%d must be positive", c->S);
    GPODE_CHECK_ARG(c->omega && c->phase && c->w && c->Z && c->ell && c->var, "cache tensor is NULL");
    GPODE_CHECK_ARG(!need_nu || c->nu, "cache.nu is NULL");
    return 0;
}

}  // namespace

extern "C" int gpode_whiten_fwd(const gpode_cache_t* c, const float* u, float jitter, float* nu_out, double* L_f64,
                                double* s_f64, void* stream) {
    if (int rc = check_cache(c, false)) return rc;
    GPODE_CHECK_ARG(u && nu_out && L_f64 && s_f64, "NULL argument");
    const int threads = c->M >= 64 ? 512 : 128;
    if (c->M <= GPODE_MAX_M_F64) {
        const size_t smem = fwd_smem<double>(c->M);
        GPODE_CUDA(cudaFuncSetAttribute(whiten_fwd_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        whiten_fwd_kernel<double><<<c->D, threads, smem, (cudaStream_t)stream>>>(*c, u, jitter, nu_out, L_f64, s_f64);
    } else {
        const size_t smem = fwd_smem<float>(c->M);
        GPODE_CUDA(cudaFuncSetAttribute(whiten_fwd_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        whiten_fwd_kernel<float><<<c->D, threads, smem, (cudaStream_t)stream>>>(*c, u, jitter, nu_out, L_f64, s_f64);
    }
    GPODE_LAUNCH_CHECK();
    return 0;
}

extern "C" int gpode_whiten_fwd_sets(const gpode_cache_t* c, const float* u, float jitter, int n_sets, float* nu_out,
                                     double* L_f64, double* s_f64, void* stream) {
    GPODE_CHECK_ARG(n_sets >= 1 && n_sets <= 65535, "n_sets=%d outside 1..65535", n_sets);
    // factor once (set 0 rides along), then the per-set solves
    if (int rc = gpode_whiten_fwd(c, u, jitter, nu_out, L_f64, s_f64, stream)) return rc;
    if (n_sets == 1) return 0;
    const int threads = c->M >= 64 ? 256 : 128;
    if (c->M <= GPODE_MAX_M_F64) {
        const size_t smem = solve_smem<double>(c->M);
        GPODE_CUDA(cudaFuncSetAttribute(whiten_solve_sets_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        whiten_solve_sets_kernel<double><<<dim3(c->D, n_sets), threads, smem, (cudaStream_t)stream>>>(*c, u, L_f64, nu_out);
    } else {
        const size_t smem = solve_smem<float>(c->M);
        GPODE_CUDA(cudaFuncSetAttribute(whiten_solve_sets_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        whiten_solve_sets_kernel<float><<<dim3(c->D, n_sets), threads, smem, (cudaStream_t)stream>>>(*c, u, L_f64, nu_out);
    }
    GPODE_LAUNCH_CHECK();
    return 0;
}

extern "C" int gpode_whiten_bwd(const gpode_cache_t* c, const float* u, const double* L_f64, const double* s_f64,
                                const float* grad_nu, float* grad_u, float* grad_Z, float* grad_ell, float* grad_var,
                                void* stream) {
    if (int rc = check_cache(c, false)) return rc;
    GPODE_CHECK_ARG(u && L_f64 && s_f64 && grad_nu && grad_u && grad_Z && grad_ell && grad_var, "NULL argument");
    const int threads = c->M >= 64 ? 512 : 128;
    // one CTA per output dimension, all D of them in ONE thread-block cluster (D <= 8 = the portable cluster size)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(c->D);
    cfg.blockDim = dim3(threads);
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = c->D;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (c->M <= GPODE_MAX_M_F64) {
        cfg.dynamicSmemBytes = bwd_smem<double>(c->M, c->D);
        GPODE_CUDA(cudaFuncSetAttribute(whiten_bwd_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)cfg.dynamicSmemBytes));
        GPODE_CUDA(cudaLaunchKernelEx(&cfg, whiten_bwd_kernel<double>, *c, u, L_f64, s_f64, grad_nu, grad_u, grad_Z,
                                      grad_ell, grad_var));
    } else {
        cfg.dynamicSmemBytes = bwd_smem<float>(c->M, c->D);
        GPODE_CUDA(cudaFuncSetAttribute(whiten_bwd_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)cfg.dynamicSmemBytes));
        GPODE_CUDA(cudaLaunchKernelEx(&cfg, whiten_bwd_kernel<float>, *c, u, L_f64, s_f64, grad_nu, grad_u, grad_Z,
                                      grad_ell, grad_var));
    }
    GPODE_LAUNCH_CHECK();
    return 0;
}

extern "C" int gpode_kl_fwd(const float* Um, const float* Ls_packed, int D, int M, float* kl_out, void* stream) {
    GPODE_CHECK_ARG(Um && Ls_packed && kl_out, "NULL argument");
    GPODE_CHECK_ARG(D >= 1 && M >= 1, "D=%d, M=%d must be positive", D, M);
    kl_fwd_kernel<<<1, 512, 0, (cudaStream_t)stream>>>(Um, Ls_packed, D, M, kl_out);
    GPODE_LAUNCH_CHECK();
    return 0;
}

extern "C" int gpode_kl_bwd(const float* Um, const float* Ls_packed, int D, int M, const float* grad_kl,
                            float* grad_Um, float* grad_Ls_packed, void* stream) {
    GPODE_CHECK_ARG(Um && Ls_packed && grad_kl && grad_Um && grad_Ls_packed, "NULL argument");
    GPODE_CHECK_ARG(D >= 1 && M >= 1, "D=%d, M=%d must be positive", D, M);
    const int n = D * (M * (M + 1) / 2);
    int grid = (n + 255) / 256;
    if (grid > 296) grid = 296;
    kl_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(Um, Ls_packed, D, M, grad_kl, grad_Um, grad_Ls_packed);
    GPODE_LAUNCH_CHECK();
    return 0;
}

extern "C" int gpode_inducing_sample_fwd(const float* Um, const float* Ls_packed, const float* eps, int D, int M,
                                         float* u_out, void* stream) {
    GPODE_CHECK_ARG(Um && Ls_packed && eps && u_out, "NULL argument");
    GPODE_CHECK_ARG(D >= 1 && M >= 1, "D=%d, M=%d must be positive", D, M);
    int grid = (M * D + 127) / 128;
    if (grid > 296) grid = 296;
    inducing_sample_fwd_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(Um, Ls_packed, eps, D, M, u_out);
    GPODE_LAUNCH_CHECK();
    return 0;
}

extern "C" int gpode_inducing_sample_bwd(const float* eps, const float* grad_u, int D, int M, float* grad_Ls_packed,
                                         void* stream) {
    GPODE_CHECK_ARG(eps && grad_u && grad_Ls_packed, "NULL argument");
    GPODE_CHECK_ARG(D >= 1 && M >= 1, "D=%d, M=%d must be positive", D, M);
    const int n = D * (M * (M + 1) / 2);
    int grid = (n + 255) / 256;
    if (grid > 296) grid = 296;
    inducing_sample_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(eps, grad_u, D, M, grad_Ls_packed);
    GPODE_LAUNCH_CHECK();
    return 0;
}
