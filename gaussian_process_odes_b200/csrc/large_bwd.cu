// Backward (vector-Jacobian product) and device-side fixed-grid RK4 for 8 < D <= 64 -- the upper half of BASELINE.json
// configs[4] (state dimension 2-64). Round 1 had a forward-only tensor-core vector field driven by eager PyTorch host
// loops; this file adds
//   * vjp_large_kernel<DP>: xb = J(x)^T kb plus every shared-parameter partial sum (lengthscales, variances, nu, Z) of
//     one batch of (point, cotangent) rows -- what autograd does through DSVGP_Layer.forward (reference
//     src/core/dsvgp.py:172-197, rff_forward :124-137, RBF.K src/core/kernels.py:53-99); formulas: SURVEY.md 8(a) A7;
//   * gpode_rk4_fwd_large_dev / gpode_rk4_bwd_large: torchdiffeq's 3/8-rule RK4 (same operation order as
//     integrate_impl.cuh) and its discrete adjoint as a stream-ordered sequence of launches -- the tcgen05 vector-field
//     kernels of large_umma.cu for the forward evaluations, this VJP kernel for the adjoint, small element-wise kernels
//     for the stage algebra; step sizes are read from the device-side grid, nothing returns to the host;
//   * gpode_grads_finalize_large: per-CTA partial rows -> parameter gradients in float64, fixed order (no atomics).
//
// The RFF part of the VJP runs first, on the tcgen05 tensor cores (large_rffb.cu): it writes its share of the row
// cotangent to gx and its lengthscale partial sums to accumulator rows of its own. The kernels here add the RBF part.
// VJP mapping (FP32 CUDA cores). CTA = 128 threads = one tile of 128 rows, THREAD = ROW for everything that is per row:
//   RBF part, per inducing point m (CTA-uniform loop): dd_j = (x_j - Z_mj)^2 in registers; per k: e = sum_j dd_j w_kj,
//     K = 2^-e, p = kb_k K, t_j += 2 ln2 c_km p w_kj;  xb_j -= d_j t_j.
//   The sums over ROWS -- T[k][m] = sum_r p, A2[k][j] = sum_r p dd_j, Zb[m][j] = sum_r d_j t_j -- are taken by
//     re-mapping the CTA to (k, j-slice) / (j) over the staged [128 x D] tiles of p, dd and d t (no atomics, fixed
//     order), accumulated per CTA: A in shared memory, T and Zb in the CTA's own rows of a global scratch block.
#include "common.cuh"
#include "../../include/gpode_b200.h"

int gpode_vf_large_eval(const float* packed_large, const gpode_cache_t* c, const float* x, float* tmp, float* f,
                        const GpodeDraws& dr, cudaStream_t st);  // large_umma.cu: f = vf(x) on the tcgen05 tensor cores
// large_rffb.cu: the RFF part of the VJP on the tcgen05 tensor cores (both projections as 3xTF32 GEMMs)
int64_t gpode_rv_packed_floats(int D, int S);
int64_t gpode_rv_acc_floats(int D);
int gpode_rv_grid(int64_t B);
int gpode_rv_dn(int D);
int gpode_rv_pack(const gpode_cache_t* c, float* out, cudaStream_t st);
int gpode_rv_launch(const float* packed, int D, int S, const float* x, const float* kb, float* gx, int64_t B, float* acc,
                    cudaStream_t st);

namespace {

constexpr int kLbRows = 128, kLbThreads = 128;  // tile rows, threads
constexpr int kLbMaxCtas = 148 * 4;

__host__ __device__ inline int lb_dp(int D) { return D <= 16 ? 16 : (D <= 32 ? 32 : 64); }

struct LbLayout {
    int D, DP, M;
    int64_t off_w, off_z, off_c, total;  // floats
};
__host__ __device__ inline LbLayout lb_layout(int D, int M) {
    LbLayout L;
    L.D = D; L.DP = lb_dp(D); L.M = M;
    L.off_w = 0;                                      // [DP][DP] w_kj = 0.5 log2(e) / ell_kj^2
    L.off_z = L.off_w + (int64_t)L.DP * L.DP;         // [M][DP] Z
    L.off_c = L.off_z + (int64_t)M * L.DP;            // [M][DP] c_km = var_k nu_km, k contiguous
    L.total = L.off_c + (int64_t)M * L.DP;
    return L;
}

__global__ void pack_lb_kernel(const LbLayout L, const float* __restrict__ Z, const float* __restrict__ nu,
                               const float* __restrict__ ell, const float* __restrict__ var, float* __restrict__ out) {
    const int D = L.D, DP = L.DP, M = L.M;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int64_t i = i0; i < (int64_t)DP * DP; i += stride) {
        const int j = (int)(i % DP), k = (int)(i / DP);
        float v = 0.f;
        if (k < D && j < D) {
            const float l = ell[k * D + j];
            v = GPODE_HALF_LOG2E / (l * l);
        }
        out[L.off_w + i] = v;
    }
    for (int64_t i = i0; i < (int64_t)M * DP; i += stride) {
        const int j = (int)(i % DP), m = (int)(i / DP);
        out[L.off_z + i] = j < D ? Z[m * D + j] : 0.f;
        out[L.off_c + i] = j < D ? var[j] * nu[j * M + m] : 0.f;   // here j plays the role of k
    }
}

// shared memory (floats): xs | kbs | stA | stB | xbs (each [128][DP + 4]; xbs = the running row cotangent: kept out of
// the register file, which holds dd / t) | Ws [DP][DP] | As [DP][DP] | red [4][DP] | V1 [DP]
template <int DP>
struct LbSmem {
    static constexpr int LD = DP + 4;
    static constexpr int tile = kLbRows * LD;
    static constexpr int floats = 5 * tile + 2 * DP * DP + 4 * DP + DP;
    static constexpr size_t bytes = (size_t)floats * 4;
};

// RBF half of the VJP at DP = 16, 32 (DP = 64: rbf_vjp_large_kernel). gx holds the RFF half on entry (large_rffb.cu);
// this kernel adds the RBF half to it and writes the RBF and variance partial sums.
template <int DP>
__global__ void __launch_bounds__(kLbThreads, 2)
vjp_large_kernel(const float* __restrict__ pk, const LbLayout L, const float* __restrict__ x,
                 const float* __restrict__ f, const float* __restrict__ kb, float* __restrict__ gx, const int64_t B,
                 float* __restrict__ accA, float* __restrict__ accT, float* __restrict__ accZ) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int LD = LbSmem<DP>::LD, TILE = LbSmem<DP>::tile;
    float* xs = reinterpret_cast<float*>(smem_raw);
    float* kbs = xs + TILE;
    float* stA = kbs + TILE;
    float* stB = stA + TILE;
    float* xbs = stB + TILE;
    float* Ws = xbs + TILE;
    float* As = Ws + DP * DP;
    float* red = As + DP * DP;
    float* V1 = red + 4 * DP;
    const int D = L.D, M = L.M;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* __restrict__ z_g = pk + L.off_z;
    const float* __restrict__ c_g = pk + L.off_c;

    for (int i = tid; i < DP * DP; i += kLbThreads) {
        Ws[i] = pk[L.off_w + i];
        As[i] = 0.f;
    }
    for (int i = tid; i < DP; i += kLbThreads) V1[i] = 0.f;
    __syncthreads();
    float* __restrict__ Tg = accT + (size_t)blockIdx.x * D * M;
    float* __restrict__ Zg = accZ + (size_t)blockIdx.x * M * DP;

    const int64_t n_tiles = (B + kLbRows - 1) / kLbRows;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t r0 = tile * kLbRows;
        const int n = (int)((B - r0) < kLbRows ? (B - r0) : kLbRows);
        // ---- tiles of x and kb (coalesced), zero padded in both directions ----
        for (int i = tid; i < kLbRows * DP; i += kLbThreads) {
            const int r = i / DP, j = i - r * DP;
            const bool ok = r < n && j < D;
            xs[r * LD + j] = ok ? __ldg(x + (r0 + r) * D + j) : 0.f;
            kbs[r * LD + j] = ok ? __ldg(kb + (r0 + r) * D + j) : 0.f;
        }
        __syncthreads();
        float* __restrict__ xbr = xbs + tid * LD;   // this row's cotangent (only its own thread touches it)
#pragma unroll
        for (int j4 = 0; j4 < DP / 4; ++j4) {
            float4 init = make_float4(0.f, 0.f, 0.f, 0.f);
            if (tid < n) {
                const float* __restrict__ gr = gx + (r0 + tid) * D;
                init.x = 4 * j4 < D ? gr[4 * j4] : 0.f;
                init.y = 4 * j4 + 1 < D ? gr[4 * j4 + 1] : 0.f;
                init.z = 4 * j4 + 2 < D ? gr[4 * j4 + 2] : 0.f;
                init.w = 4 * j4 + 3 < D ? gr[4 * j4 + 3] : 0.f;
            }
            *reinterpret_cast<float4*>(xbr + 4 * j4) = init;
        }
        // variance partial sum, first half: V1[k] += sum_rows kb_k f_k
        for (int k = 0; k < D; ++k) {
            const float fv = tid < n ? __ldg(f + (r0 + tid) * D + k) : 0.f;
            const float v = gpode_warp_sum(kbs[tid * LD + k] * fv);
            if (lane == 0) red[warp * DP + k] = v;
        }
        __syncthreads();
        for (int k = tid; k < D; k += kLbThreads) V1[k] += (red[k] + red[DP + k]) + (red[2 * DP + k] + red[3 * DP + k]);

        // ================= RBF part =================
        constexpr int TK = DP / 16, TJ = DP / 8;   // row-contraction tile per thread: 16 x 8 tiles cover [DP][DP]
        static_assert(kLbThreads == 128 && (DP == 16 || DP == 32), "tile mapping assumes 128 threads");
        const int ck0 = (tid >> 3) * TK, cj0 = (tid & 7) * TJ;
        constexpr bool kTwoRows = DP >= 32;   // two rows x half the inputs per thread in the exponent / t phases
        constexpr int NC2 = DP / 8;           // float4 chunks of a lane's half row
        const int h2 = tid & 1, rA = tid >> 1, rB = rA + kLbRows / 2;
        auto off2 = [&](const int c) { return h2 * (DP / 2) + 4 * c; };
        for (int m = 0; m < M; ++m) {
            const float* __restrict__ zm = z_g + (size_t)m * DP;
            const float* __restrict__ cm = c_g + (size_t)m * DP;
            float2 dd[DP / 2], tt[DP / 2];   // one row x DP inputs, or two rows x DP / 2 inputs (kTwoRows)
            if constexpr (kTwoRows) {
            // Register tile: a thread owns TWO rows (rA, rB = rA + 64) x HALF of the input dimensions, so every W element
            // fetched from shared memory feeds both rows -- the one-row form below issues two broadcast LDS.128 (four
            // wavefronts each) per four packed FMAs and is bound by shared-memory wavefronts at DP >= 32. Chunk c of a
            // lane is floats off(c) .. off(c)+3 of the row. The exponent halves of the two lanes are added by one
            // shuffle (a + b in both lanes: bitwise the same value).
#pragma unroll
            for (int c = 0; c < NC2; ++c) {
                const int o = off2(c);
                const float4 zv = __ldg(reinterpret_cast<const float4*>(zm + o));
                const float4 xa = *reinterpret_cast<const float4*>(xs + rA * LD + o);
                const float4 xb4 = *reinterpret_cast<const float4*>(xs + rB * LD + o);
                const float a0 = xa.x - zv.x, a1 = xa.y - zv.y, a2 = xa.z - zv.z, a3 = xa.w - zv.w;
                const float b0 = xb4.x - zv.x, b1 = xb4.y - zv.y, b2 = xb4.z - zv.z, b3 = xb4.w - zv.w;
                dd[2 * c] = make_float2(a0 * a0, a1 * a1); dd[2 * c + 1] = make_float2(a2 * a2, a3 * a3);
                dd[2 * NC2 + 2 * c] = make_float2(b0 * b0, b1 * b1); dd[2 * NC2 + 2 * c + 1] = make_float2(b2 * b2, b3 * b3);
                tt[2 * c] = tt[2 * c + 1] = tt[2 * NC2 + 2 * c] = tt[2 * NC2 + 2 * c + 1] = make_float2(0.f, 0.f);
                *reinterpret_cast<float4*>(stB + rA * LD + o) = make_float4(a0 * a0, a1 * a1, a2 * a2, a3 * a3);
                *reinterpret_cast<float4*>(stB + rB * LD + o) = make_float4(b0 * b0, b1 * b1, b2 * b2, b3 * b3);
            }
#pragma unroll 2
            for (int k = 0; k < D; k += 2) {   // rows D .. DP-1 of Ws are zero padding; an odd D's last partner has q = 0
                const float* __restrict__ wa = Ws + k * DP;
                const float* __restrict__ wb = wa + DP;
                const float2 z2 = make_float2(0.f, 0.f);
                float2 eAa0 = z2, eAa1 = z2, eAb0 = z2, eAb1 = z2, eBa0 = z2, eBa1 = z2, eBb0 = z2, eBb1 = z2;
#pragma unroll
                for (int c = 0; c < NC2; ++c) {
                    const float4 a4 = *reinterpret_cast<const float4*>(wa + off2(c));
                    const float4 b4 = *reinterpret_cast<const float4*>(wb + off2(c));
                    const float2 al = make_float2(a4.x, a4.y), ah = make_float2(a4.z, a4.w);
                    const float2 bl = make_float2(b4.x, b4.y), bh = make_float2(b4.z, b4.w);
                    eAa0 = ffma2(dd[2 * c], al, eAa0); eAa1 = ffma2(dd[2 * c + 1], ah, eAa1);
                    eAb0 = ffma2(dd[2 * c], bl, eAb0); eAb1 = ffma2(dd[2 * c + 1], bh, eAb1);
                    eBa0 = ffma2(dd[2 * NC2 + 2 * c], al, eBa0); eBa1 = ffma2(dd[2 * NC2 + 2 * c + 1], ah, eBa1);
                    eBb0 = ffma2(dd[2 * NC2 + 2 * c], bl, eBb0); eBb1 = ffma2(dd[2 * NC2 + 2 * c + 1], bh, eBb1);
                }
                float sAa = (eAa0.x + eAa0.y) + (eAa1.x + eAa1.y), sAb = (eAb0.x + eAb0.y) + (eAb1.x + eAb1.y);
                float sBa = (eBa0.x + eBa0.y) + (eBa1.x + eBa1.y), sBb = (eBb0.x + eBb0.y) + (eBb1.x + eBb1.y);
                sAa += __shfl_xor_sync(0xffffffffu, sAa, 1); sAb += __shfl_xor_sync(0xffffffffu, sAb, 1);
                sBa += __shfl_xor_sync(0xffffffffu, sBa, 1); sBb += __shfl_xor_sync(0xffffffffu, sBb, 1);
                const bool two = k + 1 < D;
                const float pAa = kbs[rA * LD + k] * gpode_ex2(-sAa);
                const float pBa = kbs[rB * LD + k] * gpode_ex2(-sBa);
                const float pAb = two ? kbs[rA * LD + k + 1] * gpode_ex2(-sAb) : 0.f;
                const float pBb = two ? kbs[rB * LD + k + 1] * gpode_ex2(-sBb) : 0.f;
                {   // each lane of the pair stages one of the two rows
                    const int rs = h2 ? rB : rA;
                    stA[rs * LD + k] = h2 ? pBa : pAa;
                    if (two) stA[rs * LD + k + 1] = h2 ? pBb : pAb;
                }
                const float ca = -GPODE_NEG_2LN2 * __ldg(cm + k);             // q = 2 ln2 c_km kb_k K
                const float cb = two ? -GPODE_NEG_2LN2 * __ldg(cm + k + 1) : 0.f;
                const float qAa = ca * pAa, qAb = cb * pAb, qBa = ca * pBa, qBb = cb * pBb;
#pragma unroll
                for (int c = 0; c < NC2; ++c) {
                    const float4 a4 = *reinterpret_cast<const float4*>(wa + off2(c));
                    const float4 b4 = *reinterpret_cast<const float4*>(wb + off2(c));
                    const float2 al = make_float2(a4.x, a4.y), ah = make_float2(a4.z, a4.w);
                    const float2 bl = make_float2(b4.x, b4.y), bh = make_float2(b4.z, b4.w);
                    tt[2 * c] = ffma2(qAb, bl, ffma2(qAa, al, tt[2 * c]));
                    tt[2 * c + 1] = ffma2(qAb, bh, ffma2(qAa, ah, tt[2 * c + 1]));
                    tt[2 * NC2 + 2 * c] = ffma2(qBb, bl, ffma2(qBa, al, tt[2 * NC2 + 2 * c]));
                    tt[2 * NC2 + 2 * c + 1] = ffma2(qBb, bh, ffma2(qBa, ah, tt[2 * NC2 + 2 * c + 1]));
                }
            }
            } else {
                // dd / t as register pairs: every FMA below is the packed dual-FP32 form (SASS FFMA2), two outputs k per trip
                // (eight independent exponent chains, two MUFU exponentials in flight); summation order as the scalar form
#pragma unroll
                for (int j4 = 0; j4 < DP / 4; ++j4) {
                    const float4 xv = *reinterpret_cast<const float4*>(xs + tid * LD + 4 * j4);
                    const float4 zv = __ldg(reinterpret_cast<const float4*>(zm + 4 * j4));
                    const float d0 = xv.x - zv.x, d1 = xv.y - zv.y, d2 = xv.z - zv.z, d3 = xv.w - zv.w;
                    dd[2 * j4] = make_float2(d0 * d0, d1 * d1);
                    dd[2 * j4 + 1] = make_float2(d2 * d2, d3 * d3);
                    tt[2 * j4] = tt[2 * j4 + 1] = make_float2(0.f, 0.f);
                    *reinterpret_cast<float4*>(stB + tid * LD + 4 * j4) =
                        make_float4(dd[2 * j4].x, dd[2 * j4].y, dd[2 * j4 + 1].x, dd[2 * j4 + 1].y);
                }
#pragma unroll 1
                for (int k = 0; k < D; k += 2) {   // rows D .. DP-1 of Ws are zero padding; an odd D's last partner has q = 0
                    const float* __restrict__ wa = Ws + k * DP;
                    const float* __restrict__ wb = wa + DP;
                    float2 ea0 = make_float2(0.f, 0.f), ea1 = ea0, eb0 = ea0, eb1 = ea0;
#pragma unroll
                    for (int j4 = 0; j4 < DP / 4; ++j4) {
                        const float4 a4 = *reinterpret_cast<const float4*>(wa + 4 * j4);
                        const float4 b4 = *reinterpret_cast<const float4*>(wb + 4 * j4);
                        ea0 = ffma2(dd[2 * j4], make_float2(a4.x, a4.y), ea0);
                        ea1 = ffma2(dd[2 * j4 + 1], make_float2(a4.z, a4.w), ea1);
                        eb0 = ffma2(dd[2 * j4], make_float2(b4.x, b4.y), eb0);
                        eb1 = ffma2(dd[2 * j4 + 1], make_float2(b4.z, b4.w), eb1);
                    }
                    const bool two = k + 1 < D;
                    const float Ka = gpode_ex2(-((ea0.x + ea0.y) + (ea1.x + ea1.y)));
                    const float Kb = gpode_ex2(-((eb0.x + eb0.y) + (eb1.x + eb1.y)));
                    const float pa = kbs[tid * LD + k] * Ka;
                    const float pb = two ? kbs[tid * LD + k + 1] * Kb : 0.f;
                    stA[tid * LD + k] = pa;
                    if (two) stA[tid * LD + k + 1] = pb;
                    const float qa = -GPODE_NEG_2LN2 * __ldg(cm + k) * pa;   // 2 ln2 c_km kb_k K
                    const float qb = two ? -GPODE_NEG_2LN2 * __ldg(cm + k + 1) * pb : 0.f;
#pragma unroll
                    for (int j4 = 0; j4 < DP / 4; ++j4) {
                        const float4 a4 = *reinterpret_cast<const float4*>(wa + 4 * j4);
                        const float4 b4 = *reinterpret_cast<const float4*>(wb + 4 * j4);
                        tt[2 * j4] = ffma2(qb, make_float2(b4.x, b4.y), ffma2(qa, make_float2(a4.x, a4.y), tt[2 * j4]));
                        tt[2 * j4 + 1] = ffma2(qb, make_float2(b4.z, b4.w), ffma2(qa, make_float2(a4.z, a4.w), tt[2 * j4 + 1]));
                    }
                }
            }
            __syncthreads();  // p and dd of all 128 rows are staged
            // rows contracted by a (TK outputs k) x (TJ inputs j) register tile per thread: T[k][m] = sum_r p;
            // A[k][j] -= 2 ln2 w_kj c_km sum_r p dd_j. Per row one vector load of p and one or two of dd feed TK*TJ/2
            // packed FMAs (a broadcast LDS.128 costs four shared-memory wavefronts whatever its address pattern: the
            // first mapping, one k x DP/2 inputs per thread, spent 8 loads on 16 FMAs and ran at the wavefront peak).
            // Columns k >= D of the p tile are never written (stale bytes): their sums are computed and dropped.
            {
                float2 acc[TK][TJ / 2];
                float s1[TK];
#pragma unroll
                for (int a = 0; a < TK; ++a) {
                    s1[a] = 0.f;
#pragma unroll
                    for (int c = 0; c < TJ / 2; ++c) acc[a][c] = make_float2(0.f, 0.f);
                }
#pragma unroll 4
                for (int r = 0; r < kLbRows; ++r) {
                    float pv[TK];
                    float2 dv[TJ / 2];
                    if constexpr (TK == 2) {
                        const float2 p2 = *reinterpret_cast<const float2*>(stA + r * LD + ck0);
                        pv[0] = p2.x; pv[1] = p2.y;
                    } else {
                        pv[0] = stA[r * LD + ck0];
                    }
                    if constexpr (TJ >= 4) {
#pragma unroll
                        for (int c4 = 0; c4 < TJ / 4; ++c4) {
                            const float4 d4 = *reinterpret_cast<const float4*>(stB + r * LD + cj0 + 4 * c4);
                            dv[2 * c4] = make_float2(d4.x, d4.y);
                            dv[2 * c4 + 1] = make_float2(d4.z, d4.w);
                        }
                    } else {
                        dv[0] = *reinterpret_cast<const float2*>(stB + r * LD + cj0);
                    }
#pragma unroll
                    for (int a = 0; a < TK; ++a) {
                        s1[a] += pv[a];
#pragma unroll
                        for (int c = 0; c < TJ / 2; ++c) acc[a][c] = ffma2(pv[a], dv[c], acc[a][c]);
                    }
                }
#pragma unroll
                for (int a = 0; a < TK; ++a) {
                    const int k = ck0 + a;
                    if (k < D) {
                        if (cj0 == 0) Tg[(size_t)k * M + m] += s1[a];
                        const float cf = GPODE_NEG_2LN2 * __ldg(cm + k);   // -2 ln2 c_km
#pragma unroll
                        for (int c = 0; c < TJ / 2; ++c) {
                            const int j = cj0 + 2 * c;
                            As[k * DP + j] = fmaf(cf * Ws[k * DP + j], acc[a][c].x, As[k * DP + j]);
                            As[k * DP + j + 1] = fmaf(cf * Ws[k * DP + j + 1], acc[a][c].y, As[k * DP + j + 1]);
                        }
                    }
                }
            }
            __syncthreads();  // stB is free again
            // xb_j -= d_j t_j; the same products, summed over rows, are the Z gradient
            if constexpr (kTwoRows) {
#pragma unroll
                for (int c = 0; c < NC2; ++c) {
                    const int o = off2(c);
                    const float4 zv = __ldg(reinterpret_cast<const float4*>(zm + o));
#pragma unroll
                    for (int rr = 0; rr < 2; ++rr) {
                        const int r = rr ? rB : rA;
                        const float2 t0 = tt[2 * NC2 * rr + 2 * c], t1 = tt[2 * NC2 * rr + 2 * c + 1];
                        const float4 xv = *reinterpret_cast<const float4*>(xs + r * LD + o);
                        float4 dt;
                        dt.x = (xv.x - zv.x) * t0.x; dt.y = (xv.y - zv.y) * t0.y;
                        dt.z = (xv.z - zv.z) * t1.x; dt.w = (xv.w - zv.w) * t1.y;
                        float4 xv4 = *reinterpret_cast<const float4*>(xbs + r * LD + o);
                        xv4.x -= dt.x; xv4.y -= dt.y; xv4.z -= dt.z; xv4.w -= dt.w;
                        *reinterpret_cast<float4*>(xbs + r * LD + o) = xv4;
                        *reinterpret_cast<float4*>(stB + r * LD + o) = dt;
                    }
                }
            } else {
#pragma unroll
                for (int j4 = 0; j4 < DP / 4; ++j4) {
                    const float4 xv = *reinterpret_cast<const float4*>(xs + tid * LD + 4 * j4);
                    const float4 zv = __ldg(reinterpret_cast<const float4*>(zm + 4 * j4));
                    float4 dt;
                    dt.x = (xv.x - zv.x) * tt[2 * j4].x; dt.y = (xv.y - zv.y) * tt[2 * j4].y;
                    dt.z = (xv.z - zv.z) * tt[2 * j4 + 1].x; dt.w = (xv.w - zv.w) * tt[2 * j4 + 1].y;
                    float4 xv4 = *reinterpret_cast<const float4*>(xbr + 4 * j4);
                    xv4.x -= dt.x; xv4.y -= dt.y; xv4.z -= dt.z; xv4.w -= dt.w;
                    *reinterpret_cast<float4*>(xbr + 4 * j4) = xv4;
                    *reinterpret_cast<float4*>(stB + tid * LD + 4 * j4) = dt;
                }
            }
            __syncthreads();
            if (tid < D) {
                float zs0 = 0.f, zs1 = 0.f, zs2 = 0.f, zs3 = 0.f;
#pragma unroll 4
                for (int r = 0; r < kLbRows; r += 4) {
                    zs0 += stB[r * LD + tid]; zs1 += stB[(r + 1) * LD + tid];
                    zs2 += stB[(r + 2) * LD + tid]; zs3 += stB[(r + 3) * LD + tid];
                }
                Zg[(size_t)m * DP + tid] += (zs0 + zs1) + (zs2 + zs3);
            }
            __syncthreads();  // stA / stB are rewritten by the next inducing point
        }
        // ---- xb out (coalesced from its shared-memory tile) ----
        __syncthreads();
        for (int i = tid; i < n * D; i += kLbThreads) {
            const int r = i / D, j = i - r * D;
            gx[(r0 + r) * D + j] = xbs[r * LD + j];
        }
        __syncthreads();
    }
    // ---- this CTA's lengthscale / variance partial sums: accumulate into its own row (sequential launches add up) ----
    float* __restrict__ Ag = accA + (size_t)blockIdx.x * (DP * DP + DP);
    for (int i = tid; i < DP * DP; i += kLbThreads) Ag[i] += As[i];
    for (int i = tid; i < DP; i += kLbThreads) Ag[DP * DP + i] += V1[i];
}

// ---- RBF half of the VJP at DP = 64, on EIGHT warps ----------------------------------------------------------------
// Same tiles, arithmetic and accumulator rows as the RBF part of vjp_large_kernel, but two warpgroups share the 128-row
// tile, so every scheduler has two warps to interleave (ncu on the four-warp form at DP = 64: FMA pipe 24 %, issue 34 %,
// shared-memory wavefronts 59 % -- latency with one warp per scheduler). Both warpgroups build the same dd registers
// (thread = two rows x half the inputs); warpgroup w takes the output pairs k = 2w, 2w + 4, ... in the exponent / t
// phases and the rows 64w .. 64w + 63 in the row contraction (its partial tile meets warpgroup 0's through a scratch
// block), the two partial t's are applied to the cotangent tile one warpgroup after the other, and the Z column sums
// use four row classes per column (the same four interleaved partial sums, added in the same order).
constexpr int kRb2Threads = 256;
template <int DP>
struct Rb2Smem {
    static constexpr int LD = DP + 4;
    static constexpr int tile = kLbRows * LD;
    static constexpr int SCR = DP * DP / 128 + DP / 16;   // contraction accumulators + p sums per thread
    static constexpr int floats = 5 * tile + 2 * DP * DP + 4 * DP + DP + 128 * SCR;
    static constexpr size_t bytes = (size_t)floats * 4;
};

template <int DP>
__global__ void __launch_bounds__(kRb2Threads, 1)
rbf_vjp_large_kernel(const float* __restrict__ pk, const LbLayout L, const float* __restrict__ x,
                     const float* __restrict__ f, const float* __restrict__ kb, float* __restrict__ gx, const int64_t B,
                     float* __restrict__ accA, float* __restrict__ accT, float* __restrict__ accZ) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int LD = Rb2Smem<DP>::LD, TILE = Rb2Smem<DP>::tile, SCR = Rb2Smem<DP>::SCR;
    float* xs = reinterpret_cast<float*>(smem_raw);
    float* kbs = xs + TILE;
    float* stA = kbs + TILE;
    float* stB = stA + TILE;
    float* xbs = stB + TILE;
    float* Ws = xbs + TILE;
    float* As = Ws + DP * DP;
    float* red = As + DP * DP;
    float* V1 = red + 4 * DP;
    float* scr = V1 + DP;
    const int D = L.D, M = L.M;
    const int tid = threadIdx.x, lane = tid & 31, wg = tid >> 7, t = tid & 127;
    const float* __restrict__ z_g = pk + L.off_z;
    const float* __restrict__ c_g = pk + L.off_c;
    for (int i = tid; i < DP * DP; i += kRb2Threads) {
        Ws[i] = pk[L.off_w + i];
        As[i] = 0.f;
    }
    for (int i = tid; i < DP; i += kRb2Threads) V1[i] = 0.f;
    __syncthreads();
    float* __restrict__ Tg = accT + (size_t)blockIdx.x * D * M;
    float* __restrict__ Zg = accZ + (size_t)blockIdx.x * M * DP;
    constexpr int TK = DP / 16, TJ = DP / 8, NC2 = DP / 8;
    static_assert(DP == 32 || DP == 64, "two-row mapping");
    const int ck0 = (t >> 3) * TK, cj0 = (t & 7) * TJ;
    const int h2 = t & 1, rA = t >> 1, rB = rA + kLbRows / 2;
    auto off2 = [&](const int c) { return h2 * (DP / 2) + 4 * ((c + (DP == 64 ? h2 * (NC2 / 2) : 0)) & (NC2 - 1)); };

    const int64_t n_tiles = (B + kLbRows - 1) / kLbRows;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t r0 = tile * kLbRows;
        const int n = (int)((B - r0) < kLbRows ? (B - r0) : kLbRows);
        for (int i = tid; i < kLbRows * DP; i += kRb2Threads) {
            const int r = i / DP, j = i - r * DP;
            const bool ok = r < n && j < D;
            xs[r * LD + j] = ok ? __ldg(x + (r0 + r) * D + j) : 0.f;
            kbs[r * LD + j] = ok ? __ldg(kb + (r0 + r) * D + j) : 0.f;
            xbs[r * LD + j] = ok ? gx[(r0 + r) * D + j] : 0.f;   // the RFF half of the cotangent, written by the tensor-core kernel
        }
        __syncthreads();
        // variance partial sum, first half: V1[k] += sum_rows kb_k f_k (rows by warp shuffle, warps in warp order)
        if (wg == 0) {
            for (int k = 0; k < D; ++k) {
                const float fv = t < n ? __ldg(f + (r0 + t) * D + k) : 0.f;
                const float v = gpode_warp_sum(kbs[t * LD + k] * fv);
                if (lane == 0) red[(t >> 5) * DP + k] = v;
            }
        }
        __syncthreads();
        for (int k = tid; k < D; k += kRb2Threads) V1[k] += (red[k] + red[DP + k]) + (red[2 * DP + k] + red[3 * DP + k]);

        for (int m = 0; m < M; ++m) {
            const float* __restrict__ zm = z_g + (size_t)m * DP;
            const float* __restrict__ cm = c_g + (size_t)m * DP;
            float2 dd[DP / 2], tt[DP / 2];   // rows rA | rB, NC2 chunks of four inputs each
#pragma unroll
            for (int c = 0; c < NC2; ++c) {
                const int o = off2(c);
                const float4 zv = __ldg(reinterpret_cast<const float4*>(zm + o));
                const float4 xa = *reinterpret_cast<const float4*>(xs + rA * LD + o);
                const float4 xb4 = *reinterpret_cast<const float4*>(xs + rB * LD + o);
                const float a0 = xa.x - zv.x, a1 = xa.y - zv.y, a2 = xa.z - zv.z, a3 = xa.w - zv.w;
                const float b0 = xb4.x - zv.x, b1 = xb4.y - zv.y, b2 = xb4.z - zv.z, b3 = xb4.w - zv.w;
                dd[2 * c] = make_float2(a0 * a0, a1 * a1); dd[2 * c + 1] = make_float2(a2 * a2, a3 * a3);
                dd[2 * NC2 + 2 * c] = make_float2(b0 * b0, b1 * b1); dd[2 * NC2 + 2 * c + 1] = make_float2(b2 * b2, b3 * b3);
                tt[2 * c] = tt[2 * c + 1] = tt[2 * NC2 + 2 * c] = tt[2 * NC2 + 2 * c + 1] = make_float2(0.f, 0.f);
                if (wg == 0) {
                    *reinterpret_cast<float4*>(stB + rA * LD + o) = make_float4(a0 * a0, a1 * a1, a2 * a2, a3 * a3);
                    *reinterpret_cast<float4*>(stB + rB * LD + o) = make_float4(b0 * b0, b1 * b1, b2 * b2, b3 * b3);
                }
            }
#pragma unroll 2
            for (int k = 2 * wg; k < D; k += 4) {   // rows D .. DP-1 of Ws are zero padding; an odd D's last partner has q = 0
                const float* __restrict__ wa = Ws + k * DP;
                const float* __restrict__ wb = wa + DP;
                const float2 z2 = make_float2(0.f, 0.f);
                float2 eAa0 = z2, eAa1 = z2, eAb0 = z2, eAb1 = z2, eBa0 = z2, eBa1 = z2, eBb0 = z2, eBb1 = z2;
#pragma unroll
                for (int c = 0; c < NC2; ++c) {
                    const float4 a4 = *reinterpret_cast<const float4*>(wa + off2(c));
                    const float4 b4 = *reinterpret_cast<const float4*>(wb + off2(c));
                    const float2 al = make_float2(a4.x, a4.y), ah = make_float2(a4.z, a4.w);
                    const float2 bl = make_float2(b4.x, b4.y), bh = make_float2(b4.z, b4.w);
                    eAa0 = ffma2(dd[2 * c], al, eAa0); eAa1 = ffma2(dd[2 * c + 1], ah, eAa1);
                    eAb0 = ffma2(dd[2 * c], bl, eAb0); eAb1 = ffma2(dd[2 * c + 1], bh, eAb1);
                    eBa0 = ffma2(dd[2 * NC2 + 2 * c], al, eBa0); eBa1 = ffma2(dd[2 * NC2 + 2 * c + 1], ah, eBa1);
                    eBb0 = ffma2(dd[2 * NC2 + 2 * c], bl, eBb0); eBb1 = ffma2(dd[2 * NC2 + 2 * c + 1], bh, eBb1);
                }
                float sAa = (eAa0.x + eAa0.y) + (eAa1.x + eAa1.y), sAb = (eAb0.x + eAb0.y) + (eAb1.x + eAb1.y);
                float sBa = (eBa0.x + eBa0.y) + (eBa1.x + eBa1.y), sBb = (eBb0.x + eBb0.y) + (eBb1.x + eBb1.y);
                sAa += __shfl_xor_sync(0xffffffffu, sAa, 1); sAb += __shfl_xor_sync(0xffffffffu, sAb, 1);
                sBa += __shfl_xor_sync(0xffffffffu, sBa, 1); sBb += __shfl_xor_sync(0xffffffffu, sBb, 1);
                const bool two = k + 1 < D;
                const float pAa = kbs[rA * LD + k] * gpode_ex2(-sAa);
                const float pBa = kbs[rB * LD + k] * gpode_ex2(-sBa);
                const float pAb = two ? kbs[rA * LD + k + 1] * gpode_ex2(-sAb) : 0.f;
                const float pBb = two ? kbs[rB * LD + k + 1] * gpode_ex2(-sBb) : 0.f;
                {   // each lane of the pair stages one of the two rows
                    const int rs = h2 ? rB : rA;
                    stA[rs * LD + k] = h2 ? pBa : pAa;
                    if (two) stA[rs * LD + k + 1] = h2 ? pBb : pAb;
                }
                const float ca = -GPODE_NEG_2LN2 * __ldg(cm + k);             // q = 2 ln2 c_km kb_k K
                const float cb = two ? -GPODE_NEG_2LN2 * __ldg(cm + k + 1) : 0.f;
                const float qAa = ca * pAa, qAb = cb * pAb, qBa = ca * pBa, qBb = cb * pBb;
#pragma unroll
                for (int c = 0; c < NC2; ++c) {
                    const float4 a4 = *reinterpret_cast<const float4*>(wa + off2(c));
                    const float4 b4 = *reinterpret_cast<const float4*>(wb + off2(c));
                    const float2 al = make_float2(a4.x, a4.y), ah = make_float2(a4.z, a4.w);
                    const float2 bl = make_float2(b4.x, b4.y), bh = make_float2(b4.z, b4.w);
                    tt[2 * c] = ffma2(qAb, bl, ffma2(qAa, al, tt[2 * c]));
                    tt[2 * c + 1] = ffma2(qAb, bh, ffma2(qAa, ah, tt[2 * c + 1]));
                    tt[2 * NC2 + 2 * c] = ffma2(qBb, bl, ffma2(qBa, al, tt[2 * NC2 + 2 * c]));
                    tt[2 * NC2 + 2 * c + 1] = ffma2(qBb, bh, ffma2(qBa, ah, tt[2 * NC2 + 2 * c + 1]));
                }
            }
            __syncthreads();  // p and dd of all 128 rows are staged
            // rows contracted by a (TK outputs k) x (TJ inputs j) register tile per thread, 64 rows per warpgroup:
            // T[k][m] = sum_r p;  A[k][j] -= 2 ln2 w_kj c_km sum_r p dd_j.  Columns k >= D of the p tile are never
            // written (stale bytes): their sums are computed and dropped.
            {
                float2 acc[TK][TJ / 2];
                float s1[TK];
#pragma unroll
                for (int a = 0; a < TK; ++a) {
                    s1[a] = 0.f;
#pragma unroll
                    for (int c = 0; c < TJ / 2; ++c) acc[a][c] = make_float2(0.f, 0.f);
                }
#pragma unroll 4
                for (int r = wg * (kLbRows / 2); r < (wg + 1) * (kLbRows / 2); ++r) {
                    float pv[TK];
                    float2 dv[TJ / 2];
                    if constexpr (TK == 4) {
                        const float4 p4 = *reinterpret_cast<const float4*>(stA + r * LD + ck0);
                        pv[0] = p4.x; pv[1] = p4.y; pv[2] = p4.z; pv[3] = p4.w;
                    } else {
                        const float2 p2 = *reinterpret_cast<const float2*>(stA + r * LD + ck0);
                        pv[0] = p2.x; pv[1] = p2.y;
                    }
#pragma unroll
                    for (int c4 = 0; c4 < TJ / 4; ++c4) {
                        const float4 d4 = *reinterpret_cast<const float4*>(stB + r * LD + cj0 + 4 * c4);
                        dv[2 * c4] = make_float2(d4.x, d4.y);
                        dv[2 * c4 + 1] = make_float2(d4.z, d4.w);
                    }
#pragma unroll
                    for (int a = 0; a < TK; ++a) {
                        s1[a] += pv[a];
#pragma unroll
                        for (int c = 0; c < TJ / 2; ++c) acc[a][c] = ffma2(pv[a], dv[c], acc[a][c]);
                    }
                }
                float* __restrict__ mine = scr + t * SCR;
                if (wg == 1) {
#pragma unroll
                    for (int a = 0; a < TK; ++a) {
                        mine[TK * TJ + a] = s1[a];
#pragma unroll
                        for (int c = 0; c < TJ / 2; ++c)
                            *reinterpret_cast<float2*>(mine + a * TJ + 2 * c) = acc[a][c];
                    }
                }
                __syncthreads();
                if (wg == 0) {
#pragma unroll
                    for (int a = 0; a < TK; ++a) {
                        const int k = ck0 + a;
                        if (k < D) {
                            if (cj0 == 0) Tg[(size_t)k * M + m] += s1[a] + mine[TK * TJ + a];
                            const float cf = GPODE_NEG_2LN2 * __ldg(cm + k);   // -2 ln2 c_km
#pragma unroll
                            for (int c = 0; c < TJ / 2; ++c) {
                                const int j = cj0 + 2 * c;
                                const float2 o = *reinterpret_cast<const float2*>(mine + a * TJ + 2 * c);
                                As[k * DP + j] = fmaf(cf * Ws[k * DP + j], acc[a][c].x + o.x, As[k * DP + j]);
                                As[k * DP + j + 1] = fmaf(cf * Ws[k * DP + j + 1], acc[a][c].y + o.y, As[k * DP + j + 1]);
                            }
                        }
                    }
                }
            }
            // xb_j -= d_j t_j, warpgroup 0's half of the outputs first, then warpgroup 1's; the same products, summed
            // over rows, are the Z gradient
#pragma unroll
            for (int w = 0; w < 2; ++w) {
                if (wg == w) {
#pragma unroll
                    for (int c = 0; c < NC2; ++c) {
                        const int o = off2(c);
                        const float4 zv = __ldg(reinterpret_cast<const float4*>(zm + o));
#pragma unroll
                        for (int rr = 0; rr < 2; ++rr) {
                            const int r = rr ? rB : rA;
                            const float2 t0 = tt[2 * NC2 * rr + 2 * c], t1 = tt[2 * NC2 * rr + 2 * c + 1];
                            const float4 xv = *reinterpret_cast<const float4*>(xs + r * LD + o);
                            float4 dt;
                            dt.x = (xv.x - zv.x) * t0.x; dt.y = (xv.y - zv.y) * t0.y;
                            dt.z = (xv.z - zv.z) * t1.x; dt.w = (xv.w - zv.w) * t1.y;
                            float4 xv4 = *reinterpret_cast<const float4*>(xbs + r * LD + o);
                            xv4.x -= dt.x; xv4.y -= dt.y; xv4.z -= dt.z; xv4.w -= dt.w;
                            *reinterpret_cast<float4*>(xbs + r * LD + o) = xv4;
                            if (w == 1) {
                                const float4 d0 = *reinterpret_cast<const float4*>(stB + r * LD + o);
                                dt.x += d0.x; dt.y += d0.y; dt.z += d0.z; dt.w += d0.w;
                            }
                            *reinterpret_cast<float4*>(stB + r * LD + o) = dt;
                        }
                    }
                }
                __syncthreads();
            }
            if (tid < 4 * DP) {   // column j, row class y = r mod 4
                const int j = tid % DP, y = tid / DP;
                float zsum = 0.f;
#pragma unroll 8
                for (int r = y; r < kLbRows; r += 4) zsum += stB[r * LD + j];
                scr[y * DP + j] = zsum;
            }
            __syncthreads();
            if (tid < D)
                Zg[(size_t)m * DP + tid] += (scr[tid] + scr[DP + tid]) + (scr[2 * DP + tid] + scr[3 * DP + tid]);
        }
        // ---- xb out (coalesced from its shared-memory tile) ----
        __syncthreads();
        for (int i = tid; i < n * D; i += kRb2Threads) {
            const int r = i / D, j = i - r * D;
            gx[(r0 + r) * D + j] = xbs[r * LD + j];
        }
        __syncthreads();
    }
    float* __restrict__ Ag = accA + (size_t)blockIdx.x * (DP * DP + DP);
    for (int i = tid; i < DP * DP; i += kRb2Threads) Ag[i] += As[i];
    for (int i = tid; i < DP; i += kRb2Threads) Ag[DP * DP + i] += V1[i];
}

// ---- parameter gradients from the per-CTA rows (float64, rows in row order) ------------------------------------------
// grid.x covers the D*D + D*M + M*D outputs of the first kernel; acc = [accA rows | accT rows | accZ rows | accR rows].
// One thread per output, loads coalesced across outputs; the row loop runs eight independent partial sums (rows r,
// r + 8, ...) that are added in a fixed order, so the result is reproducible and the loads pipeline. The variance
// gradient needs sum_m c_km T[k][m]: it is taken from grad_nu = var_k T by a second kernel (one warp per output k) --
// round 2's first version looped over m x rows in one thread: 2.1 ms at D = 16 (592 rows).
// Block = 32 outputs x 8 row classes: thread (x, y) adds rows y, y + 8, ... of output x in row order, the eight partial
// sums meet in shared memory and are added in the fixed order ((0+1)+(2+3))+((4+5)+(6+7)) -- bitwise what one thread
// with eight interleaved partial sums gave (0.33-0.40 ms at 592-888 rows), at an eighth of the dependent chain.
__device__ __forceinline__ double lb_sum_rows(const float* __restrict__ base, const size_t stride, const size_t off,
                                              const int n_rows, const int y) {
    double s = 0.0;
#pragma unroll 4
    for (int r = y; r < n_rows; r += 8) s += (double)__ldcg(base + (size_t)r * stride + off);
    return s;
}

__global__ void __launch_bounds__(256)
finalize_large_kernel(const int D, const int DP, const int M, const int n_rows,
                      const float* __restrict__ accA, const float* __restrict__ accT,
                      const float* __restrict__ accZ, const float* __restrict__ accR, const int n_rows_r,
                      const int DN, const float* __restrict__ ell, const float* __restrict__ var,
                      float* __restrict__ g_ell, float* __restrict__ g_Z, float* __restrict__ g_nu) {
    __shared__ double part[2][8][32];
    const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + x;
    const int nA = D * D, nT = D * M, nZ = M * D;
    double p0 = 0.0, p1 = 0.0;
    if (i < nA) {
        const int k = i / D, j = i - k * D;
        p0 = lb_sum_rows(accA, (size_t)DP * DP + DP, (size_t)k * DP + j, n_rows, y);
        p1 = lb_sum_rows(accR, (size_t)DN * DN, (size_t)k * DN + j, n_rows_r, y);   // rows of the tensor-core RFF kernel
    } else if (i < nA + nT) {
        p0 = lb_sum_rows(accT, (size_t)D * M, (size_t)(i - nA), n_rows, y);
    } else if (i < nA + nT + nZ) {
        const int e = i - nA - nT, m = e / D, j = e - m * D;
        p0 = lb_sum_rows(accZ, (size_t)M * DP, (size_t)m * DP + j, n_rows, y);
    }
    part[0][y][x] = p0;
    part[1][y][x] = p1;
    __syncthreads();
    if (y != 0) return;
    double t[2];
#pragma unroll
    for (int q = 0; q < 2; ++q)
        t[q] = ((part[q][0][x] + part[q][1][x]) + (part[q][2][x] + part[q][3][x])) +
               ((part[q][4][x] + part[q][5][x]) + (part[q][6][x] + part[q][7][x]));
    if (i < nA) {
        g_ell[i] = (float)(-(t[0] + t[1]) / (double)ell[i]);
    } else if (i < nA + nT) {
        g_nu[i - nA] = (float)((double)var[(i - nA) / M] * t[0]);
    } else if (i < nA + nT + nZ) {
        g_Z[i - nA - nT] = (float)t[0];
    }
}

// grad_var[k] = (sum_rows kb_k f_k + sum_m c_km T[k][m]) / (2 var_k), with var_k T = grad_nu; one warp per k
__global__ void finalize_large_var_kernel(const int D, const int DP, const int M, const int n_rows,
                                          const float* __restrict__ accA, const float* __restrict__ nu,
                                          const float* __restrict__ var, const float* __restrict__ g_nu,
                                          float* __restrict__ g_var) {
    const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (k >= D) return;
    double v = 0.0;
    for (int r = lane; r < n_rows; r += 32) v += (double)__ldcg(accA + (size_t)r * (DP * DP + DP) + (size_t)DP * DP + k);
    for (int m = lane; m < M; m += 32) v += (double)nu[k * M + m] * (double)g_nu[k * M + m];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) g_var[k] = (float)(0.5 * v / (double)var[k]);
}

// ---- element-wise stage algebra of the 3/8-rule RK4 step and of its adjoint ------------------------------------------
#define LB_THIRD 0.3333333432674407958984375f
// mode 2..4: stage input of stage `mode`; mode 5: the step itself (out = y + (k1 + 3 (k2 + k3) + k4) dt / 8)
__global__ void rk4_stage_large_kernel(const int mode, const float* __restrict__ t, const int i,
                                       const float* __restrict__ y, const float* __restrict__ k1,
                                       const float* __restrict__ k2, const float* __restrict__ k3,
                                       const float* __restrict__ k4, float* __restrict__ out, const int64_t n) {
    const float dt = __fsub_rn(__ldg(t + i + 1), __ldg(t + i));
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        float v;
        if (mode == 2) v = __fadd_rn(y[e], __fmul_rn(__fmul_rn(dt, k1[e]), LB_THIRD));
        else if (mode == 3) v = __fadd_rn(y[e], __fmul_rn(dt, __fsub_rn(k2[e], __fmul_rn(k1[e], LB_THIRD))));
        else if (mode == 4) v = __fadd_rn(y[e], __fmul_rn(dt, __fadd_rn(__fsub_rn(k1[e], k2[e]), k3[e])));
        else {
            const float sum = __fadd_rn(__fadd_rn(k1[e], __fmul_rn(3.0f, __fadd_rn(k2[e], k3[e]))), k4[e]);
            v = __fadd_rn(y[e], __fmul_rn(__fmul_rn(sum, dt), 0.125f));
        }
        out[e] = v;
    }
}
// cotangent of stage `st` (4..1) from lambda and the VJPs already done (recursion of integrate_impl.cuh::rk4_bwd_kernel);
// st == 0: lambda <- grad_xs[i] + lambda + yb1 + yb2 + yb3 + yb4
__global__ void rk4_cot_large_kernel(const int st, const float* __restrict__ t, const int i,
                                     const float* lam, const float* __restrict__ yb4,
                                     const float* __restrict__ yb3, const float* __restrict__ yb2,
                                     const float* __restrict__ yb1, const float* __restrict__ gxi,
                                     float* out, const int64_t n) {  // st == 0 runs in place: out == lam
    const float h = __fsub_rn(__ldg(t + i + 1), __ldg(t + i));
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        float v;
        if (st == 4) v = 0.125f * h * lam[e];
        else if (st == 3) v = fmaf(0.375f * h, lam[e], h * yb4[e]);
        else if (st == 2) v = fmaf(0.375f * h, lam[e], h * (yb3[e] - yb4[e]));
        else if (st == 1) v = fmaf(0.125f * h, lam[e], fmaf(h * LB_THIRD, yb2[e] - yb3[e], h * yb4[e]));
        else v = gxi[e] + lam[e] + ((yb4[e] + yb3[e]) + (yb2[e] + yb1[e]));
        out[e] = v;
    }
}

int lb_check(const gpode_cache_t* c) {
    GPODE_CHECK_ARG(c != nullptr, "cache is NULL");
    GPODE_CHECK_ARG(c->D > GPODE_MAX_D && c->D <= GPODE_MAX_D_LARGE, "large-D path needs %d < D <= %d, got %d",
                    GPODE_MAX_D, GPODE_MAX_D_LARGE, c->D);
    GPODE_CHECK_ARG(c->S >= 1 && c->M >= 1 && c->omega && c->phase && c->w && c->Z && c->var && c->ell && c->nu,
                    "cache tensor is NULL");
    return 0;
}

// persistent grid: SMs x the CTAs per SM the launch bounds ask for -- two of vjp_large_kernel (DP = 16, 32), one of
// rbf_vjp_large_kernel (DP = 64). The accumulator rows are per CTA: every launch of one backward pass and the finalize
// kernel must agree on this number, and it fixes the order in which the parameter-gradient sums are added, so it is a
// constant rather than an occupancy query that would follow the compiler's register allocation.
int lb_grid(int64_t B, int DP) {
    int sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int64_t tiles = (B + kLbRows - 1) / kLbRows;
    int64_t g = (int64_t)sms * (DP == 64 ? 1 : 2);
    if (g > tiles) g = tiles;
    if (g > kLbMaxCtas) g = kLbMaxCtas;
    return (int)(g < 1 ? 1 : g);
}

template <int DP>
int launch_vjp(const float* pk, const LbLayout& L, const float* x, const float* f, const float* kb, float* gx,
               int64_t B, float* acc, cudaStream_t st) {
    const size_t smem = LbSmem<DP>::bytes;
    GPODE_CUDA(cudaFuncSetAttribute(vjp_large_kernel<DP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    float* accA = acc;
    float* accT = accA + (size_t)kLbMaxCtas * (DP * DP + DP);
    float* accZ = accT + (size_t)kLbMaxCtas * L.D * L.M;
    vjp_large_kernel<DP><<<lb_grid(B, DP), kLbThreads, smem, st>>>(pk, L, x, f, kb, gx, B, accA, accT, accZ);
    GPODE_LAUNCH_CHECK();
    return 0;
}

// floats of the RBF kernels' accumulator rows (the tensor-core RFF rows follow them in acc_large)
int64_t lb_acc_floats(int D, int M) {
    const int DP = lb_dp(D);
    return (int64_t)kLbMaxCtas * ((int64_t)DP * DP + DP + (int64_t)D * M + (int64_t)M * DP);
}
// the RFF half on the tcgen05 kernel of large_rffb.cu, then the RBF half on the CUDA cores
int vjp_dispatch(const float* pk, int D, int M, int S, const float* x, const float* f, const float* kb, float* gx,
                 int64_t B, float* acc, cudaStream_t st) {
    const LbLayout L = lb_layout(D, M);
    if (int rc = gpode_rv_launch(pk + L.total, D, S, x, kb, gx, B, acc + lb_acc_floats(D, M), st)) return rc;
    if (L.DP == 16) return launch_vjp<16>(pk, L, x, f, kb, gx, B, acc, st);
    if (L.DP == 32) return launch_vjp<32>(pk, L, x, f, kb, gx, B, acc, st);
    {
        constexpr int DP = 64;
        GPODE_CUDA(cudaFuncSetAttribute(rbf_vjp_large_kernel<DP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)Rb2Smem<DP>::bytes));
        float* accT = acc + (size_t)kLbMaxCtas * (DP * DP + DP);
        float* accZ = accT + (size_t)kLbMaxCtas * L.D * L.M;
        rbf_vjp_large_kernel<DP><<<lb_grid(B, DP), kRb2Threads, Rb2Smem<DP>::bytes, st>>>(pk, L, x, f, kb, gx, B, acc, accT,
                                                                                          accZ);
        GPODE_LAUNCH_CHECK();
        return 0;
    }
}

inline unsigned ew_grid(int64_t n) {
    const int64_t g = (n + 255) / 256;
    return (unsigned)(g < 2368 ? (g < 1 ? 1 : g) : 2368);
}

}  // namespace

extern "C" int64_t gpode_packed_large_bwd_floats(int D, int M, int S) {
    if (D <= GPODE_MAX_D || D > GPODE_MAX_D_LARGE || S < 1 || M < 1) return -1;
    return lb_layout(D, M).total + gpode_rv_packed_floats(D, S);   // RBF operands | tensor-core RFF operands
}

extern "C" int64_t gpode_acc_large_floats(int D, int M) {
    if (D <= GPODE_MAX_D || D > GPODE_MAX_D_LARGE || M < 1) return -1;
    return lb_acc_floats(D, M) + gpode_rv_acc_floats(D);
}

extern "C" int gpode_pack_cache_large_bwd(const gpode_cache_t* c, float* packed_bwd, void* stream) {
    if (int rc = lb_check(c)) return rc;
    GPODE_CHECK_ARG(packed_bwd != nullptr, "packed_bwd is NULL");
    const LbLayout L = lb_layout(c->D, c->M);
    pack_lb_kernel<<<592, 256, 0, (cudaStream_t)stream>>>(L, c->Z, c->nu, c->ell, c->var, packed_bwd);
    GPODE_LAUNCH_CHECK();
    return gpode_rv_pack(c, packed_bwd + L.total, (cudaStream_t)stream);
}

extern "C" int gpode_vf_bwd_large(const float* packed_bwd, int D, int M, int S, const float* x, const float* f,
                                  const float* grad_f, float* grad_x, float* acc_large, int64_t B, void* stream) {
    GPODE_CHECK_ARG(D > GPODE_MAX_D && D <= GPODE_MAX_D_LARGE && M >= 1 && S >= 1 && B >= 0, "bad sizes D=%d M=%d S=%d", D,
                    M, S);
    if (B == 0) return 0;
    GPODE_CHECK_ARG(packed_bwd && x && f && grad_f && grad_x && acc_large, "NULL argument");
    return vjp_dispatch(packed_bwd, D, M, S, x, f, grad_f, grad_x, B, acc_large, (cudaStream_t)stream);
}

extern "C" int gpode_grads_finalize_large(const gpode_cache_t* c, const float* acc_large, int64_t B, float* grad_ell,
                                          float* grad_var, float* grad_Z, float* grad_nu, void* stream) {
    if (int rc = lb_check(c)) return rc;
    GPODE_CHECK_ARG(acc_large && grad_ell && grad_var && grad_Z && grad_nu, "NULL argument");
    const int D = c->D, M = c->M, DP = lb_dp(D);
    const float* accA = acc_large;
    const float* accT = accA + (size_t)kLbMaxCtas * (DP * DP + DP);
    const float* accZ = accT + (size_t)kLbMaxCtas * D * M;
    const int n_out = D * D + 2 * D * M;
    const float* accR = acc_large + lb_acc_floats(D, M);
    const int n_rows_r = gpode_rv_grid(B) * 4;
    finalize_large_kernel<<<(n_out + 31) / 32, 256, 0, (cudaStream_t)stream>>>(
        D, DP, M, lb_grid(B, DP), accA, accT, accZ, accR, n_rows_r, gpode_rv_dn(D), c->ell, c->var, grad_ell, grad_Z,
        grad_nu);
    finalize_large_var_kernel<<<(D + 3) / 4, 128, 0, (cudaStream_t)stream>>>(D, DP, M, lb_grid(B, DP), accA, c->nu,
                                                                              c->var, grad_nu, grad_var);
    GPODE_LAUNCH_CHECK();
    return 0;
}

// xs [Tg,B,D] (xs[0] = x0), kstages [Tg-1,4,B,D] or NULL; tmp: 2 B D floats (6 B D when kstages is NULL);
// B = dr.n * dr.rows rows, draw q of the field integrating its own dr.rows of them
static int rk4_fwd_large(const float* packed_large, const gpode_cache_t* c, const float* x0, const float* t, int Tg,
                         float* xs, float* kstages, float* tmp, const GpodeDraws& dr, cudaStream_t st) {
    GPODE_CHECK_ARG(packed_large && x0 && t && xs && tmp, "NULL argument");
    const int64_t n = dr.n * dr.rows * c->D;
    GPODE_CUDA(cudaMemcpyAsync(xs, x0, sizeof(float) * n, cudaMemcpyDeviceToDevice, st));
    float* ys = tmp;
    float* frff = tmp + n;
    float* kloc = tmp + 2 * n;  // used only when the caller keeps no checkpoints
    const unsigned g = ew_grid(n);
    for (int i = 0; i + 1 < Tg; ++i) {
        const float* y = xs + (int64_t)i * n;
        float* k = kstages ? kstages + (int64_t)i * 4 * n : kloc;
        float *k1 = k, *k2 = k + n, *k3 = k + 2 * n, *k4 = k + 3 * n;
        if (int rc = gpode_vf_large_eval(packed_large, c, y, frff, k1, dr, st)) return rc;
        rk4_stage_large_kernel<<<g, 256, 0, st>>>(2, t, i, y, k1, k2, k3, k4, ys, n);
        if (int rc = gpode_vf_large_eval(packed_large, c, ys, frff, k2, dr, st)) return rc;
        rk4_stage_large_kernel<<<g, 256, 0, st>>>(3, t, i, y, k1, k2, k3, k4, ys, n);
        if (int rc = gpode_vf_large_eval(packed_large, c, ys, frff, k3, dr, st)) return rc;
        rk4_stage_large_kernel<<<g, 256, 0, st>>>(4, t, i, y, k1, k2, k3, k4, ys, n);
        if (int rc = gpode_vf_large_eval(packed_large, c, ys, frff, k4, dr, st)) return rc;
        rk4_stage_large_kernel<<<g, 256, 0, st>>>(5, t, i, y, k1, k2, k3, k4, xs + (int64_t)(i + 1) * n, n);
        GPODE_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" int gpode_rk4_fwd_large_dev(const float* packed_large, const gpode_cache_t* c, const float* x0, const float* t,
                                       int Tg, int64_t B, float* xs, float* kstages, float* tmp, void* stream) {
    if (int rc = lb_check(c)) return rc;
    GPODE_CHECK_ARG(Tg >= 1 && B >= 0, "bad sizes Tg=%d B=%lld", Tg, (long long)B);
    if (B == 0) return 0;
    return rk4_fwd_large(packed_large, c, x0, t, Tg, xs, kstages, tmp, gpode_one_draw(B), (cudaStream_t)stream);
}

// n_sets draws of the "sets" cache (packed by gpode_pack_cache_large_sets), each integrating its own set_rows rows;
// xs [Tg, n_sets set_rows, D], tmp 6 n_sets set_rows D floats
extern "C" int gpode_rk4_fwd_large_sets(const float* packed_large, const gpode_cache_t* c, int n_sets, int64_t set_rows,
                                        const float* x0, const float* t, int Tg, float* xs, float* tmp, void* stream) {
    if (int rc = lb_check(c)) return rc;
    GPODE_CHECK_ARG(n_sets >= 1 && n_sets <= 65535 && set_rows >= 0 && Tg >= 1, "bad sizes n_sets=%d Tg=%d", n_sets,
                    Tg);
    if (set_rows == 0) return 0;
    const GpodeDraws dr{n_sets, set_rows, gpode_packed_large_floats(c->D, c->M, c->S), nullptr, 0};
    return rk4_fwd_large(packed_large, c, x0, t, Tg, xs, nullptr, tmp, dr, (cudaStream_t)stream);
}

// Discrete adjoint of the above. work: 7 B D floats (lambda, stage input, cotangent, yb4, yb3, yb2, yb1).
extern "C" int gpode_rk4_bwd_large(const float* packed_bwd, const gpode_cache_t* c, const float* t, int Tg, int64_t B,
                                   const float* xs, const float* kstages, const float* grad_xs, float* grad_x0,
                                   float* acc_large, float* work, void* stream) {
    if (int rc = lb_check(c)) return rc;
    GPODE_CHECK_ARG(Tg >= 1 && B >= 0, "bad sizes Tg=%d B=%lld", Tg, (long long)B);
    if (B == 0) return 0;
    GPODE_CHECK_ARG(packed_bwd && t && xs && grad_xs && grad_x0 && acc_large && work, "NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int D = c->D, M = c->M, S = c->S;
    const int64_t n = B * D;
    if (Tg == 1) {
        GPODE_CUDA(cudaMemcpyAsync(grad_x0, grad_xs, sizeof(float) * n, cudaMemcpyDeviceToDevice, st));
        return 0;
    }
    GPODE_CHECK_ARG(kstages != nullptr, "kstages is NULL");
    float *lam = work, *ys = work + n, *kbar = work + 2 * n, *yb4 = work + 3 * n, *yb3 = work + 4 * n,
          *yb2 = work + 5 * n, *yb1 = work + 6 * n;
    GPODE_CUDA(cudaMemcpyAsync(lam, grad_xs + (int64_t)(Tg - 1) * n, sizeof(float) * n, cudaMemcpyDeviceToDevice, st));
    const unsigned g = ew_grid(n);
    for (int i = Tg - 2; i >= 0; --i) {
        const float* y = xs + (int64_t)i * n;
        const float* k = kstages + (int64_t)i * 4 * n;
        const float *k1 = k, *k2 = k + n, *k3 = k + 2 * n, *k4 = k + 3 * n;
        // stage 4
        rk4_stage_large_kernel<<<g, 256, 0, st>>>(4, t, i, y, k1, k2, k3, k4, ys, n);
        rk4_cot_large_kernel<<<g, 256, 0, st>>>(4, t, i, lam, yb4, yb3, yb2, yb1, nullptr, kbar, n);
        if (int rc = vjp_dispatch(packed_bwd, D, M, S, ys, k4, kbar, yb4, B, acc_large, st)) return rc;
        // stage 3
        rk4_stage_large_kernel<<<g, 256, 0, st>>>(3, t, i, y, k1, k2, k3, k4, ys, n);
        rk4_cot_large_kernel<<<g, 256, 0, st>>>(3, t, i, lam, yb4, yb3, yb2, yb1, nullptr, kbar, n);
        if (int rc = vjp_dispatch(packed_bwd, D, M, S, ys, k3, kbar, yb3, B, acc_large, st)) return rc;
        // stage 2
        rk4_stage_large_kernel<<<g, 256, 0, st>>>(2, t, i, y, k1, k2, k3, k4, ys, n);
        rk4_cot_large_kernel<<<g, 256, 0, st>>>(2, t, i, lam, yb4, yb3, yb2, yb1, nullptr, kbar, n);
        if (int rc = vjp_dispatch(packed_bwd, D, M, S, ys, k2, kbar, yb2, B, acc_large, st)) return rc;
        // stage 1
        rk4_cot_large_kernel<<<g, 256, 0, st>>>(1, t, i, lam, yb4, yb3, yb2, yb1, nullptr, kbar, n);
        if (int rc = vjp_dispatch(packed_bwd, D, M, S, y, k1, kbar, yb1, B, acc_large, st)) return rc;
        rk4_cot_large_kernel<<<g, 256, 0, st>>>(0, t, i, lam, yb4, yb3, yb2, yb1, grad_xs + (int64_t)i * n, lam, n);
        GPODE_LAUNCH_CHECK();
    }
    GPODE_CUDA(cudaMemcpyAsync(grad_x0, lam, sizeof(float) * n, cudaMemcpyDeviceToDevice, st));
    return 0;
}
