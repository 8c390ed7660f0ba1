// Blocked float64 whitening for D <= GPODE_MAX_D and GPODE_MAX_M < M <= GPODE_MAX_M_BLOCKED: the same mathematics as
// whiten.cu (its header comment gives the forward and backward formulas), with the M x M matrices in global memory
// (the caller's L_f64 and workspace; 8 M^2 bytes per output dimension, L2-resident up to M ~ 1500 at D = 8) instead of
// one CTA's shared memory, so that every step spreads over many CTAs:
//   Kzz build          one launch over (element, k)
//   Cholesky           right-looking, panels of NB columns: per panel one launch factors the diagonal block and solves
//                      the panel below it (chol_inplace with the panel rows carried along, one CTA per 64 rows x k),
//                      one launch updates the trailing lower triangle (64 x 64 tiles x k, FP64 FMA) and writes the
//                      factored diagonal block
//   triangular solves  blocked TRSM, in place on an [M, N] right-hand side per k: per block of NB rows one launch
//                      solves the diagonal block (column sweep in shared memory), one launch updates the remaining rows
//                      (64 x 64 tiles). N = 1 for the vectors, n_sets for batched draws, M for the backward's Kbar.
// Every launch size follows from (D, M, n_sets) on the host: nothing reads the device, nothing allocates, so the whole
// path is stream-ordered and can be captured in a CUDA graph. No floating-point atomics: each output element is computed
// in a fixed order, and the cross-CTA sums of the backward go through per-CTA rows added in row order, so repeated
// calls are bitwise identical. Every column of a solve is computed by the same sequence of operations whatever N is, so
// a batched draw gets bitwise the nu of the single-draw call.
#include "whiten.cuh"

namespace {

constexpr int NB = 64;           // panel width of the Cholesky and block height of the triangular solves
constexpr int TB = 64;           // TB x TB output tile of the update kernels (256 threads x 4 x 4)
constexpr int kPanelRows = 64;   // panel rows below the diagonal block per CTA of the panel kernel
constexpr int kThreads = 256;
constexpr int kSolveCols = 32;   // right-hand sides per CTA of the diagonal-block solve
constexpr int kGradPts = 64;     // inducing points per CTA of the gradient contraction
constexpr int LDP = NB + 1;      // odd leading dimension of the shared-memory panels (conflict-free column reads)

constexpr size_t kPanelSmem = sizeof(double) * (NB + kPanelRows) * LDP;
constexpr size_t kUpdateSmem = sizeof(double) * 2 * TB * LDP;
constexpr size_t kSolveSmem = sizeof(double) * (NB * LDP + NB * kSolveCols);

inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }
// grid-stride launches: at most 8 CTAs of kThreads per SM (148 SMs)
inline int grid_for(int64_t n) { return n < kThreads ? 1 : (n > (int64_t)1184 * kThreads ? 1184 : cdiv(n, kThreads)); }

// ---- Kzz ---------------------------------------------------------------------------------------------------------
// L_k <- K_k(Z,Z) + jitter I in the lower triangle, zeros above (the factor is computed in place)
__global__ void kzz_build_kernel(const gpode_cache_t c, const float jitter, double* __restrict__ L) {
    const int k = blockIdx.y, M = c.M, D = c.D;
    const double vark = (double)c.var[k];
    double inv_l[GPODE_MAX_D];
    for (int j = 0; j < D; ++j) inv_l[j] = 1.0 / (double)c.ell[k * D + j];
    double* __restrict__ Lk = L + (size_t)k * M * M;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)M * M;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int m = (int)(i / M), n = (int)(i - (int64_t)m * M);
        Lk[i] = n <= m ? rbf_entry(c.Z, inv_l, vark, D, m, n) + (m == n ? (double)jitter : 0.0) : 0.0;
    }
}

// p = rff_forward(Z)_k of draw q = blockIdx.z (one warp per inducing point) into column q of B [D][M][N]; draw 0's
// prior also into sp[k][1]
__global__ void prior_kernel(gpode_cache_t c, const int N, double* __restrict__ B, double* __restrict__ sp) {
    const int k = blockIdx.y, q = blockIdx.z, M = c.M, D = c.D, S = c.S;
    c.omega += (size_t)q * D * S * D;
    c.phase += (size_t)q * S * D;
    c.w += (size_t)q * S * D;
    const int m = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (m >= M) return;
    const double p = rff_at_point(c, k, m, sqrtf(c.var[k] / (float)S));
    if ((threadIdx.x & 31) == 0) {
        B[((size_t)k * M + m) * N + q] = p;
        if (q == 0) sp[((size_t)k * 2 + 1) * M + m] = p;
    }
}

// ---- Cholesky ------------------------------------------------------------------------------------------------------
// Panel [j0, j0 + nb): every CTA loads the (already updated) diagonal block and its kPanelRows rows of the panel below
// it, factors the block with chol_inplace carrying those rows along (they end up holding L21 = A21 L11^-T) and writes
// its rows back. The block is factored redundantly by every CTA of the panel (NB^3 / 3 flops against the NB^2
// kPanelRows of its rows) and written by the next launch, chol_update_kernel: the other CTAs here still read it.
__global__ void __launch_bounds__(kThreads) chol_panel_kernel(double* __restrict__ L, const int M, const int j0) {
    extern __shared__ __align__(16) double A[];   // (nb + rows) x LDP
    __shared__ double dinv[NB];
    const int k = blockIdx.y, nb = min(NB, M - j0);
    const int r0 = j0 + nb + blockIdx.x * kPanelRows, rows = max(0, min(kPanelRows, M - r0));
    double* __restrict__ Lk = L + (size_t)k * M * M;
    for (int i = threadIdx.x; i < (nb + rows) * nb; i += blockDim.x) {
        const int r = i / nb, cc = i - r * nb;
        const int gr = r < nb ? j0 + r : r0 + r - nb;
        A[r * LDP + cc] = Lk[(size_t)gr * M + j0 + cc];
    }
    chol_inplace<double>(A, nb, nb + rows, LDP, dinv);
    for (int i = threadIdx.x; i < rows * nb; i += blockDim.x) {
        const int r = i / nb, cc = i - r * nb;
        Lk[(size_t)(r0 + r) * M + j0 + cc] = A[(nb + r) * LDP + cc];
    }
}

// Trailing update A22 -= L21 L21^T of panel [j0, j0 + nb) on the lower TB x TB tiles of rows / columns >= j0 + nb
// (CTA t < ntiles: linear tile index -> (ti >= tj)); entries above the diagonal are left alone (they stay zero).
// CTA ntiles factors the panel's diagonal block once more and writes it: a region no other CTA of this launch touches.
__global__ void __launch_bounds__(kThreads) chol_update_kernel(double* __restrict__ L, const int M, const int j0,
                                                               const int nb, const int ntiles) {
    extern __shared__ __align__(16) double sm[];
    double* As = sm;              // TB x LDP: rows of the tile's row block, panel columns
    double* Bs = sm + TB * LDP;   // TB x LDP: rows of the tile's column block
    const int k = blockIdx.y, t = blockIdx.x;
    if (t == ntiles) {
        __shared__ double dinv[NB];
        double* __restrict__ Lk = L + (size_t)k * M * M;
        for (int i = threadIdx.x; i < nb * nb; i += blockDim.x) {
            const int r = i / nb, cc = i - r * nb;
            As[r * LDP + cc] = Lk[(size_t)(j0 + r) * M + j0 + cc];
        }
        chol_inplace<double>(As, nb, nb, LDP, dinv);
        for (int i = threadIdx.x; i < nb * nb; i += blockDim.x) {
            const int r = i / nb, cc = i - r * nb;
            if (cc <= r) Lk[(size_t)(j0 + r) * M + j0 + cc] = As[r * LDP + cc];
        }
        return;
    }
    int ti = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
    while ((ti + 1) * (ti + 2) / 2 <= t) ++ti;
    while (ti * (ti + 1) / 2 > t) --ti;
    const int tj = t - ti * (ti + 1) / 2;
    const int j1 = j0 + nb, R0 = j1 + ti * TB, C0 = j1 + tj * TB;
    double* __restrict__ Lk = L + (size_t)k * M * M;
    for (int i = threadIdx.x; i < TB * nb; i += blockDim.x) {
        const int r = i / nb, p = i - r * nb;
        As[r * LDP + p] = R0 + r < M ? Lk[(size_t)(R0 + r) * M + j0 + p] : 0.0;
        Bs[r * LDP + p] = C0 + r < M ? Lk[(size_t)(C0 + r) * M + j0 + p] : 0.0;
    }
    __syncthreads();
    const int tr = threadIdx.x >> 4, tc = threadIdx.x & 15;
    double acc[4][4] = {};
    for (int p = 0; p < nb; ++p) {
        double a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = As[(tr + 16 * i) * LDP + p];
#pragma unroll
        for (int j = 0; j < 4; ++j) b[j] = Bs[(tc + 16 * j) * LDP + p];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = R0 + tr + 16 * i, cc = C0 + tc + 16 * j;
            if (r < M && cc <= r) Lk[(size_t)r * M + cc] -= acc[i][j];
        }
}

// ---- triangular solves, in place on B [D][M][N] ----------------------------------------------------------------------
// Diagonal block [i0, i0 + nb) of L X = B (UPPER: L^T X = B) for kSolveCols right-hand sides per CTA: column sweep in
// shared memory, x_r = (b_r - sum_c L_rc x_c) / L_rr with the sum taken in ascending (UPPER: descending) c.
template <bool UPPER>
__global__ void __launch_bounds__(kThreads) trsm_diag_kernel(const double* __restrict__ L, const int M, const int i0,
                                                             double* __restrict__ B, const int N) {
    extern __shared__ __align__(16) double sm[];
    double* Ls = sm;               // nb x LDP
    double* Xs = sm + NB * LDP;    // nb x cpc
    __shared__ double dinv[NB];
    const int k = blockIdx.y, nb = min(NB, M - i0);
    const int cpc = min(N, kSolveCols), c0 = blockIdx.x * cpc, ncols = min(cpc, N - c0);
    const double* __restrict__ Lk = L + (size_t)k * M * M;
    double* __restrict__ Bk = B + (size_t)k * M * N;
    for (int i = threadIdx.x; i < nb * nb; i += blockDim.x) {
        const int r = i / nb, cc = i - r * nb;
        Ls[r * LDP + cc] = Lk[(size_t)(i0 + r) * M + i0 + cc];
    }
    for (int r = threadIdx.x; r < nb; r += blockDim.x) dinv[r] = 1.0 / Lk[(size_t)(i0 + r) * M + i0 + r];
    for (int i = threadIdx.x; i < nb * cpc; i += blockDim.x) {
        const int r = i / cpc, q = i - r * cpc;
        if (q < ncols) Xs[i] = Bk[(size_t)(i0 + r) * N + c0 + q];
    }
    __syncthreads();
    const int q = threadIdx.x % cpc, rg = threadIdx.x / cpc, ngr = blockDim.x / cpc;
    for (int s = 0; s < nb; ++s) {
        const int c = UPPER ? nb - 1 - s : s;
        if (q < ncols && rg < ngr) {
            const double xc = Xs[c * cpc + q] * dinv[c];   // row c is final: no later step writes it
            if (UPPER) {
                for (int r = rg; r < c; r += ngr) Xs[r * cpc + q] = fma(-Ls[c * LDP + r], xc, Xs[r * cpc + q]);
            } else {
                for (int r = c + 1 + rg; r < nb; r += ngr) Xs[r * cpc + q] = fma(-Ls[r * LDP + c], xc, Xs[r * cpc + q]);
            }
        }
        __syncthreads();
    }
    for (int i = threadIdx.x; i < nb * cpc; i += blockDim.x) {
        const int r = i / cpc, qq = i - r * cpc;
        if (qq < ncols) Bk[(size_t)(i0 + r) * N + c0 + qq] = Xs[i] * dinv[r];
    }
}

// The rows the solved block feeds: lower, rows j >= i0 + nb: B_j -= L[j, block] X_block; upper, rows j < i0:
// B_j -= L[block, j]^T X_block. TB x TB tiles of (rows, right-hand sides); each element's sum runs over the block in
// ascending order.
template <bool UPPER>
__global__ void __launch_bounds__(kThreads) trsm_update_kernel(const double* __restrict__ L, const int M, const int i0,
                                                               double* __restrict__ B, const int N) {
    extern __shared__ __align__(16) double sm[];
    double* As = sm;              // TB x LDP: the L entries of the tile's rows
    double* Xs = sm + TB * LDP;   // nb x TB: the solved block, the tile's columns
    const int k = blockIdx.z, nb = min(NB, M - i0);
    const int rhi = UPPER ? i0 : M;
    const int R0 = (UPPER ? 0 : i0 + nb) + blockIdx.x * TB, C0 = blockIdx.y * TB;
    const double* __restrict__ Lk = L + (size_t)k * M * M;
    double* __restrict__ Bk = B + (size_t)k * M * N;
    for (int i = threadIdx.x; i < TB * nb; i += blockDim.x) {
        if (UPPER) {   // L[i0 + p][R0 + r]: consecutive threads read consecutive r
            const int p = i / TB, r = i - p * TB;
            As[r * LDP + p] = R0 + r < rhi ? Lk[(size_t)(i0 + p) * M + R0 + r] : 0.0;
        } else {
            const int r = i / nb, p = i - r * nb;
            As[r * LDP + p] = R0 + r < rhi ? Lk[(size_t)(R0 + r) * M + i0 + p] : 0.0;
        }
        const int p = i / TB, cc = i - p * TB;
        Xs[p * TB + cc] = C0 + cc < N ? Bk[(size_t)(i0 + p) * N + C0 + cc] : 0.0;
    }
    __syncthreads();
    const int tr = threadIdx.x >> 4, tc = threadIdx.x & 15;
    double acc[4][4] = {};
    for (int p = 0; p < nb; ++p) {
        double a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = As[(tr + 16 * i) * LDP + p];
#pragma unroll
        for (int j = 0; j < 4; ++j) b[j] = Xs[p * TB + tc + 16 * j];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = R0 + tr + 16 * i, cc = C0 + tc + 16 * j;
            if (r < rhi && cc < N) Bk[(size_t)r * N + cc] -= acc[i][j];
        }
}

// ---- forward element-wise steps ---------------------------------------------------------------------------------------
// B holds s = L^-1 p (column q = draw q): draw 0's s -> sp[k][0]; B <- w = u_q[:, k] - s
__global__ void fwd_rhs_kernel(const float* __restrict__ u, const int D, const int M, const int N,
                               double* __restrict__ B, double* __restrict__ sp) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)D * M * N;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int q = (int)(i % N), m = (int)((i / N) % M), k = (int)(i / ((int64_t)N * M));
        const double s = B[i];
        if (q == 0) sp[((size_t)k * 2 + 0) * M + m] = s;
        B[i] = (double)u[((size_t)q * M + m) * D + k] - s;
    }
}

// nu_out [N][D][M] <- B [D][M][N]
__global__ void fwd_out_kernel(const double* __restrict__ B, const int D, const int M, const int N,
                               float* __restrict__ nu_out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)D * M * N;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int m = (int)(i % M), k = (int)((i / M) % D), q = (int)(i / ((int64_t)M * D));
        nu_out[i] = (float)B[((size_t)k * M + m) * N + q];
    }
}

// ---- backward ------------------------------------------------------------------------------------------------------
__global__ void bwd_init_kernel(const float* __restrict__ gnu, const int n, double* __restrict__ rb) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) rb[i] = (double)gnu[i];
}

// rb = L^-1 nub is solved: grad_u = rb; pb <- -rb (solved next); P = -Phi(w rb^T - rb s^T), w = u_k - s, into Pw [D][M][M]
__global__ void bwd_form_kernel(const float* __restrict__ u, const int D, const int M, const double* __restrict__ sp,
                                const double* __restrict__ rb, double* __restrict__ pb, double* __restrict__ Pw,
                                float* __restrict__ g_u) {
    const int k = blockIdx.y;
    const double* __restrict__ s = sp + (size_t)k * 2 * M;
    const double* __restrict__ r = rb + (size_t)k * M;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)M * M;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int m = (int)(i / M), n = (int)(i - (int64_t)m * M);
        double v = 0.0;
        if (n <= m) {
            const double wm = (double)u[m * D + k] - s[m];
            v = -(wm * r[n] - r[m] * s[n]);
            if (n == m) v *= 0.5;
        }
        Pw[(size_t)k * M * M + i] = v;
        if (n == 0) {
            g_u[m * D + k] = (float)r[m];
            pb[(size_t)k * M + m] = -r[m];
        }
    }
}

// In-place transpose of every M x M matrix of A [D][M][M]
__global__ void transpose_kernel(double* __restrict__ A, const int M) {
    double* __restrict__ Ak = A + (size_t)blockIdx.y * M * M;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)M * M;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int m = (int)(i / M), n = (int)(i - (int64_t)m * M);
        if (n < m) {
            const double t = Ak[i];
            Ak[i] = Ak[(size_t)n * M + m];
            Ak[(size_t)n * M + m] = t;
        }
    }
}

// Kb = sym(X) contracted with the RBF derivative, plus the RFF VJP at x = Z with cotangent pb, for kGradPts inducing
// points of output dim k: thread = (point, quarter of the partner points, in order), quarters added in order; one
// warp per point for the VJP. gzK[k][m][:] = this output dimension's grad_Z row; rows[k][blockIdx.x][:] = the CTA's
// lengthscale / variance partial sums (D + 1 doubles).
__global__ void __launch_bounds__(kThreads) bwd_grad_kernel(const gpode_cache_t c, const double* __restrict__ Xw,
                                                            const double* __restrict__ pb,
                                                            const double* __restrict__ sp, double* __restrict__ gzK,
                                                            double* __restrict__ rows) {
    __shared__ double gzs[kGradPts * GPODE_MAX_D];
    __shared__ double red[(kThreads / 32) * (GPODE_MAX_D + 1)];
    const int k = blockIdx.y, M = c.M, D = c.D, S = c.S;
    const int parts = blockDim.x / kGradPts, ml = threadIdx.x % kGradPts, part = threadIdx.x / kGradPts;
    const int m0 = blockIdx.x * kGradPts, m = m0 + ml;
    const float* ellk = c.ell + k * D;
    const double vark = (double)c.var[k];
    const double* __restrict__ X = Xw + (size_t)k * M * M;
    double inv_l[GPODE_MAX_D], gl[GPODE_MAX_D], gz[GPODE_MAX_D];
    for (int j = 0; j < D; ++j) {
        inv_l[j] = 1.0 / (double)ellk[j];
        gl[j] = 0.0;
        gz[j] = 0.0;
    }
    double gvar = 0.0;
    if (m < M) {
        const int chunk = (M + parts - 1) / parts, n1 = min(M, (part + 1) * chunk);
        for (int n = part * chunk; n < n1; ++n) {
            const double kb = 0.5 * (X[(size_t)m * M + n] + X[(size_t)n * M + m]);
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
    for (int p = 0; p < parts; ++p) {   // the quarters of one inducing point are added in order
        if (part == p)
            for (int j = 0; j < D; ++j) gzs[ml * D + j] = (p == 0 ? 0.0 : gzs[ml * D + j]) + gz[j];
        __syncthreads();
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const float ak = sqrtf(c.var[k] / (float)S);
    for (int mm = warp; mm < kGradPts && m0 + mm < M; mm += nwarps) {
        double G[GPODE_MAX_D];
        const double pbm = pb[(size_t)k * M + m0 + mm];
        rff_vjp_at_point(c, k, m0 + mm, pbm, ak, G);
        for (int j = 0; j < D; ++j) {
            double v = G[j];
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) {
                gzs[mm * D + j] += v;   // inducing point mm belongs to this warp alone
                gl[j] += -v * (double)c.Z[(m0 + mm) * D + j] / (double)ellk[j];
            }
        }
        if (lane == 0) gvar += pbm * sp[((size_t)k * 2 + 1) * M + m0 + mm] / (2.0 * vark);
    }
    for (int o = 16; o > 0; o >>= 1) gvar += __shfl_xor_sync(0xffffffffu, gvar, o);
    for (int j = 0; j < D; ++j)
        for (int o = 16; o > 0; o >>= 1) gl[j] += __shfl_xor_sync(0xffffffffu, gl[j], o);
    if (lane == 0) {
        red[warp * (D + 1) + D] = gvar;
        for (int j = 0; j < D; ++j) red[warp * (D + 1) + j] = gl[j];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kGradPts * D; i += blockDim.x)
        if (m0 + i / D < M) gzK[((size_t)k * M + m0) * D + i] = gzs[i];
    for (int j = threadIdx.x; j < D + 1; j += blockDim.x) {
        double t = 0.0;
        for (int w = 0; w < nwarps; ++w) t += red[w * (D + 1) + j];
        rows[((size_t)k * gridDim.x + blockIdx.x) * (D + 1) + j] = t;
    }
}

// grad_Z = sum over k of gzK (k in order); grad_ell, grad_var = sums of the CTA rows (row order)
__global__ void bwd_finalize_kernel(const int D, const int M, const int nblk, const double* __restrict__ gzK,
                                    const double* __restrict__ rows, float* __restrict__ g_Z,
                                    float* __restrict__ g_ell, float* __restrict__ g_var) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < M * D + D * (D + 1); i += gridDim.x * blockDim.x) {
        double t = 0.0;
        if (i < M * D) {
            for (int k = 0; k < D; ++k) t += gzK[(size_t)k * M * D + i];
            g_Z[i] = (float)t;
        } else {
            const int e = i - M * D, k = e / (D + 1), j = e - k * (D + 1);
            for (int b = 0; b < nblk; ++b) t += rows[((size_t)k * nblk + b) * (D + 1) + j];
            if (j < D) g_ell[k * D + j] = (float)t;
            else g_var[k] = (float)t;
        }
    }
}

// ---- host side -------------------------------------------------------------------------------------------------------
int check_blocked(const gpode_cache_t* c) {
    GPODE_CHECK_ARG(c != nullptr, "cache is NULL");
    GPODE_CHECK_ARG(c->D >= 1 && c->D <= GPODE_MAX_D, "state dimension D=%d outside 1..%d", c->D, GPODE_MAX_D);
    GPODE_CHECK_ARG(c->M >= 1 && c->M <= GPODE_MAX_M_BLOCKED,
                    "M=%d outside 1..%d (GPODE_MAX_M_BLOCKED, the limit of the blocked whitening)", c->M,
                    GPODE_MAX_M_BLOCKED);
    GPODE_CHECK_ARG(c->S >= 1, "S=%d must be positive", c->S);
    GPODE_CHECK_ARG(c->omega && c->phase && c->w && c->Z && c->ell && c->var, "cache tensor is NULL");
    return 0;
}

int set_smem_attributes() {
    GPODE_CUDA(cudaFuncSetAttribute(chol_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPanelSmem));
    GPODE_CUDA(cudaFuncSetAttribute(chol_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kUpdateSmem));
    GPODE_CUDA(cudaFuncSetAttribute(trsm_diag_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSolveSmem));
    GPODE_CUDA(cudaFuncSetAttribute(trsm_diag_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSolveSmem));
    GPODE_CUDA(cudaFuncSetAttribute(trsm_update_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kUpdateSmem));
    GPODE_CUDA(cudaFuncSetAttribute(trsm_update_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kUpdateSmem));
    return 0;
}

// L_k = chol(L_k) in place for every k (lower triangle of the M x M row-major matrices)
void cholesky(double* L, int D, int M, cudaStream_t st) {
    for (int j0 = 0; j0 < M; j0 += NB) {
        const int nb = M - j0 < NB ? M - j0 : NB, below = M - j0 - nb;
        if (below > 0)
            chol_panel_kernel<<<dim3(cdiv(below, kPanelRows), D), kThreads, kPanelSmem, st>>>(L, M, j0);
        const int nt = cdiv(below, TB), ntiles = nt * (nt + 1) / 2;
        chol_update_kernel<<<dim3(ntiles + 1, D), kThreads, kUpdateSmem, st>>>(L, M, j0, nb, ntiles);
    }
}

// B [D][M][N] <- L^-1 B (upper: L^-T B), block by block
template <bool UPPER>
void trsm(const double* L, int D, int M, double* B, int N, cudaStream_t st) {
    const int nblk = cdiv(M, NB);
    for (int b = 0; b < nblk; ++b) {
        const int i0 = (UPPER ? nblk - 1 - b : b) * NB, nb = M - i0 < NB ? M - i0 : NB;
        trsm_diag_kernel<UPPER><<<dim3(cdiv(N, N < kSolveCols ? N : kSolveCols), D), kThreads, kSolveSmem, st>>>(
            L, M, i0, B, N);
        const int rest = UPPER ? i0 : M - i0 - nb;
        if (rest > 0)
            trsm_update_kernel<UPPER><<<dim3(cdiv(rest, TB), cdiv(N, TB), D), kThreads, kUpdateSmem, st>>>(L, M, i0, B,
                                                                                                         N);
    }
}

int64_t bwd_work_doubles(int D, int M) {
    return (int64_t)D * M * (2 + M + D) + (int64_t)D * cdiv(M, kGradPts) * (D + 1);
}

}  // namespace

extern "C" int64_t gpode_whiten_blocked_work_doubles(int D, int M, int n_sets) {
    if (D < 1 || D > GPODE_MAX_D || M < 1 || M > GPODE_MAX_M_BLOCKED || n_sets < 0 || n_sets > 65535) return -1;
    return n_sets == 0 ? bwd_work_doubles(D, M) : (int64_t)D * M * n_sets;
}

extern "C" int gpode_whiten_fwd_sets_blocked(const gpode_cache_t* c, const float* u, float jitter, int n_sets,
                                             float* nu_out, double* L_f64, double* s_f64, double* work,
                                             void* stream) {
    if (int rc = check_blocked(c)) return rc;
    GPODE_CHECK_ARG(n_sets >= 1 && n_sets <= 65535, "n_sets=%d outside 1..65535", n_sets);
    GPODE_CHECK_ARG(u && nu_out && L_f64 && s_f64 && work, "NULL argument");
    if (int rc = set_smem_attributes()) return rc;
    const cudaStream_t st = (cudaStream_t)stream;
    const int D = c->D, M = c->M, N = n_sets;
    kzz_build_kernel<<<dim3(grid_for((int64_t)M * M), D), kThreads, 0, st>>>(*c, jitter, L_f64);
    prior_kernel<<<dim3(cdiv(M, kThreads / 32), D, N), kThreads, 0, st>>>(*c, N, work, s_f64);
    cholesky(L_f64, D, M, st);
    trsm<false>(L_f64, D, M, work, N, st);                                      // s = L^-1 p
    fwd_rhs_kernel<<<grid_for((int64_t)D * M * N), kThreads, 0, st>>>(u, D, M, N, work, s_f64);   // w = u - s
    trsm<true>(L_f64, D, M, work, N, st);                                       // nu = L^-T w
    fwd_out_kernel<<<grid_for((int64_t)D * M * N), kThreads, 0, st>>>(work, D, M, N, nu_out);
    GPODE_LAUNCH_CHECK();
    return 0;
}

extern "C" int gpode_whiten_fwd_blocked(const gpode_cache_t* c, const float* u, float jitter, float* nu_out,
                                        double* L_f64, double* s_f64, double* work, void* stream) {
    return gpode_whiten_fwd_sets_blocked(c, u, jitter, 1, nu_out, L_f64, s_f64, work, stream);
}

extern "C" int gpode_whiten_bwd_blocked(const gpode_cache_t* c, const float* u, const double* L_f64,
                                        const double* s_f64, const float* grad_nu, float* grad_u, float* grad_Z,
                                        float* grad_ell, float* grad_var, double* work, void* stream) {
    if (int rc = check_blocked(c)) return rc;
    GPODE_CHECK_ARG(u && L_f64 && s_f64 && grad_nu && grad_u && grad_Z && grad_ell && grad_var && work,
                    "NULL argument");
    if (int rc = set_smem_attributes()) return rc;
    const cudaStream_t st = (cudaStream_t)stream;
    const int D = c->D, M = c->M, nblk = cdiv(M, kGradPts);
    // work: rb [D][M] | pb [D][M] | Kbar [D][M][M] | gzK [D][M][D] | rows [D][nblk][D + 1]
    double* rb = work;
    double* pb = rb + (size_t)D * M;
    double* Kw = pb + (size_t)D * M;
    double* gzK = Kw + (size_t)D * M * M;
    double* rows = gzK + (size_t)D * M * D;
    bwd_init_kernel<<<grid_for((int64_t)D * M), kThreads, 0, st>>>(grad_nu, D * M, rb);
    trsm<false>(L_f64, D, M, rb, 1, st);                                          // rb = L^-1 nub (= grad_u)
    bwd_form_kernel<<<dim3(grid_for((int64_t)M * M), D), kThreads, 0, st>>>(u, D, M, s_f64, rb, pb, Kw, grad_u);
    trsm<true>(L_f64, D, M, pb, 1, st);                                           // pb = -L^-T rb
    trsm<true>(L_f64, D, M, Kw, M, st);                                           // Y = L^-T P
    transpose_kernel<<<dim3(grid_for((int64_t)M * M), D), kThreads, 0, st>>>(Kw, M);
    trsm<true>(L_f64, D, M, Kw, M, st);                                           // X^T = L^-T Y^T  (X = Y L^-1)
    bwd_grad_kernel<<<dim3(nblk, D), kThreads, 0, st>>>(*c, Kw, pb, s_f64, gzK, rows);
    bwd_finalize_kernel<<<grid_for((int64_t)M * D + D * (D + 1)), kThreads, 0, st>>>(D, M, nblk, gzK, rows, grad_Z,
                                                                                     grad_ell, grad_var);
    GPODE_LAUNCH_CHECK();
    return 0;
}
