// Random-Fourier-feature part of the vector-Jacobian product for 8 < D <= 64 on the 5th-generation tensor cores.
//
// For one batch of (point x, cotangent kb) rows and every output dimension k
//     theta_ks = phase_sk + sum_j x_j Omega_jsk                  GEMM 1   [rows x (D+1)] x [(D+1) x S]
//     p_ks     = -kb_k a_sk sin(theta_ks)                        row threads (MUFU)
//     G_kj     = sum_s p_ks Omega_jsk                            GEMM 2   [rows x S] x [S x D]
//     xb_j    += G_kj ,   A[k][j] += sum_rows x_j G_kj           (lengthscale partial sums)
// -- what autograd does through DSVGP_Layer.rff_forward (reference src/core/dsvgp.py:124-137) inside
// DSVGP_Layer.forward (:172-197); formulas: SURVEY.md 8(a) A7. Both GEMMs are tcgen05.mma.cta_group::1.kind::tf32
// (M = 128 rows), error-compensated 3xTF32, fp32 accumulators in TMEM:
//   GEMM 1  SS form: A = [x | 1] tile (hi / lo, canonical K-major no-swizzle tiles in shared memory), B = the
//           (k, 64-feature) chunk of [Omega_k ; phase_k], N = 64;
//   GEMM 2  TS form: A = p, WRITTEN BACK TO TENSOR MEMORY by the row threads (tcgen05.st, hi and lo column blocks), B =
//           the same chunk of Omega_k re-tiled with the input dimension as N and the feature as K; the accumulator G_k
//           collects all chunks of output k.
// The FP32 CUDA-core loop this replaced (formerly the RFF part of vjp_large_kernel) spent 4 S D^2 FMAs per row on
// the two projections: the whole VJP took 80 ms per 1e5 rows at D = 64 (register spills); this kernel 5.7 ms (ncu: tensor
// pipe 26 % busy, bound by the L2 operand stream -- 14 GB per 1e5 rows, two tilings of Omega -- and by the single row
// warp per scheduler), the whole VJP 21.5 ms (profiles/r02_summary.md section 4).
//
// CTA = 192 threads, one 128-row tile at a time: warps 0-3 own the rows (thread = row = TMEM lane); lane 0 of warp 4
// streams the GEMM-1 operand chunks from L2 (cp.async.bulk + mbarrier, two-slot ring) and issues GEMM 1, lane 0 of warp 5
// does the same for GEMM 2 (its own two-slot ring: a GEMM-1 slot is free one GEMM earlier). The two issuers run
// independently -- GEMM 1 up to two chunks ahead of the rows, GEMM 2 right behind them -- so the tensor pipe always has
// work queued while the rows take the sines.
// TMEM (512 columns): theta 2 x 64 | p: 2 slots x (hi 64 | lo 64) | G 2 x 64.
#include "umma.cuh"
#include "../../include/gpode_b200.h"

namespace {

constexpr int kRvThreads = 192, kRvRows = 128, kRvNC = 64;
constexpr int kRvMaxCtas = 160;      // >= SM count: one accumulator row per (CTA, row warp)
constexpr int C_TH = 0, C_P = 128, C_G = 384;

__host__ __device__ inline int rv_kp(int D) { return (D + 1 + 7) & ~7; }   // padded K of GEMM 1 (inputs + phase slot)
__host__ __device__ inline int rv_dn(int D) { return (D + 15) & ~15; }     // padded N of GEMM 2
__host__ __device__ inline int rv_su(int S) { return (S + kRvNC - 1) / kRvNC * kRvNC; }
__host__ __device__ inline int64_t rv_b1(int D) { return 2 * (int64_t)rv_kp(D) * kRvNC; }  // floats: hi | lo
// GEMM-2 record: hi | lo | the chunk's feature weights a_sk (the row threads read them from the staged record instead of
// global memory: ncu showed the row warps -- one per scheduler -- waiting on those loads, long_scoreboard 2.8 per issue)
__host__ __device__ inline int64_t rv_b2(int D) { return 2 * (int64_t)rv_dn(D) * kRvNC + kRvNC; }
// canonical K-major no-swizzle tile of `rows` rows: [K/4 chunks][rows/8 groups][8 rows][4 floats]
__host__ __device__ inline int rv_off(int rows, int r, int q) {
    return (q >> 2) * (rows * 4) + (r >> 3) * 32 + (r & 7) * 4 + (q & 3);
}

// packed block: [k][chunk] B1 records | [k][chunk] B2 records | a[k][SU]
__global__ void rv_pack_kernel(const int D, const int S, const float* __restrict__ omega,
                               const float* __restrict__ phase, const float* __restrict__ w,
                               const float* __restrict__ var, float* __restrict__ out) {
    const int KP = rv_kp(D), DN = rv_dn(D), SU = rv_su(S), NCH = SU / kRvNC;
    const int64_t b1 = rv_b1(D), b2 = rv_b2(D);
    float* o1 = out;
    float* o2 = out + (int64_t)D * NCH * b1;
    float* oa = o2 + (int64_t)D * NCH * b2;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int64_t i = i0; i < (int64_t)D * SU * KP; i += stride) {
        const int q = (int)(i % KP), s = (int)((i / KP) % SU), k = (int)(i / ((int64_t)KP * SU));
        float v = 0.f;
        if (s < S) {
            if (q < D) v = omega[((size_t)q * S + s) * D + k];
            else if (q == D) v = phase[s * D + k];
        }
        float hi, lo;
        gpode_split_tf32_rn(v, hi, lo);
        float* r = o1 + ((int64_t)k * NCH + s / kRvNC) * b1;
        const int o = rv_off(kRvNC, s % kRvNC, q);
        r[o] = hi;
        r[(int64_t)KP * kRvNC + o] = lo;
    }
    for (int64_t i = i0; i < (int64_t)D * SU * DN; i += stride) {
        const int j = (int)(i % DN), s = (int)((i / DN) % SU), k = (int)(i / ((int64_t)DN * SU));
        const float v = (s < S && j < D) ? omega[((size_t)j * S + s) * D + k] : 0.f;
        float hi, lo;
        gpode_split_tf32_rn(v, hi, lo);
        float* r = o2 + ((int64_t)k * NCH + s / kRvNC) * b2;
        const int o = rv_off(DN, j, s % kRvNC);
        r[o] = hi;
        r[(int64_t)DN * kRvNC + o] = lo;
        if (j == 0) r[2 * (int64_t)DN * kRvNC + s % kRvNC] = s < S ? w[s * D + k] * sqrtf(var[k] / (float)S) : 0.f;
    }
    for (int64_t i = i0; i < (int64_t)D * SU; i += stride) {
        const int s = (int)(i % SU), k = (int)(i / SU);
        oa[i] = s < S ? w[s * D + k] * sqrtf(var[k] / (float)S) : 0.f;
    }
}

struct RvBars {
    uint64_t a_full, th_full[2], th_free[2], p_full[2], p_free[2], g_full[2], g_free[2], b1_full[2], b1_free[2],
        b2_full[2], b2_free[2];
    uint32_t tmem_ptr;
};
constexpr int kRvData = 256;  // byte offset of the tiles behind the barriers

__device__ __forceinline__ void rv_mma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void rv_tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n" ::"r"(taddr),
                 "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
                 "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
                 "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]),
                 "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
                 : "memory");
}
__device__ __forceinline__ void rv_tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void rv_tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
                 "tcgen05.wait::ld.sync.aligned;\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr)
                 : "memory");
}

// DN = padded input dimension (16 / 32 / 48 / 64): sizes the per-row cotangent registers
template <int DN>
__global__ void __launch_bounds__(kRvThreads, 1)
rff_vjp_large_kernel(const float* __restrict__ packed, const int D, const int S, const float* __restrict__ x,
                     const float* __restrict__ kb, float* __restrict__ gx, const int64_t B, float* __restrict__ acc) {
    extern __shared__ __align__(128) unsigned char smem[];
    RvBars* bar = reinterpret_cast<RvBars*>(smem);
    const int KP = rv_kp(D), SU = rv_su(S), NCH = SU / kRvNC;
    const int64_t b1f = rv_b1(D), b2f = rv_b2(D);
    const int a_floats = KP * kRvRows;
    float* a_hi = reinterpret_cast<float*>(smem + kRvData);
    float* a_lo = a_hi + a_floats;
    float* ring1 = a_lo + a_floats;          // [2][b1f]
    float* ring2 = ring1 + 2 * b1f;          // [2][b2f]
    const float* __restrict__ g1 = packed;
    const float* __restrict__ g2 = packed + (int64_t)D * NCH * b1f;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 128) {
        gpode_mbar_init(&bar->a_full, kRvRows);
        for (int i = 0; i < 2; ++i) {
            gpode_mbar_init(&bar->th_full[i], 1);
            gpode_mbar_init(&bar->th_free[i], kRvRows);
            gpode_mbar_init(&bar->p_full[i], kRvRows);
            gpode_mbar_init(&bar->p_free[i], 1);
            gpode_mbar_init(&bar->g_full[i], 1);
            gpode_mbar_init(&bar->g_free[i], kRvRows);
            gpode_mbar_init(&bar->b1_full[i], 1);
            gpode_mbar_init(&bar->b1_free[i], 1);
            gpode_mbar_init(&bar->b2_full[i], 1);
            gpode_mbar_init(&bar->b2_free[i], 1);
        }
    }
    if (warp == 4) {
        __syncwarp();
        tmem_alloc(&bar->tmem_ptr, 512u);
    }
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_base = bar->tmem_ptr;

    const int64_t n_tiles = (B + kRvRows - 1) / kRvRows;
    const int chunks_per_tile = D * NCH;
    const int k_rot = (int)(blockIdx.x % (unsigned)D);   // CTAs walk the outputs in different rotations (L2 lines)

    if (warp < 4) {
        const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
        float* __restrict__ accw = acc + ((size_t)blockIdx.x * 4 + warp) * (DN * DN);
        uint32_t q = 0, kc = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int64_t row0 = tile * kRvRows;
            // ---- state tile -> shared memory (coalesced global reads), pre-split into tf32 hi / lo ----
            for (int i = tid; i < kRvRows * D; i += kRvRows) {
                const int r = i / D, j = i - r * D;
                const float v = row0 + r < B ? __ldg(x + row0 * D + i) : 0.f;
                float hi, lo;
                gpode_split_tf32_rn(v, hi, lo);
                const int o = rv_off(kRvRows, r, j);
                a_hi[o] = hi;
                a_lo[o] = lo;
            }
            for (int c = D; c < KP; ++c) {  // slot D carries the constant 1 that picks up the phase row
                const int o = rv_off(kRvRows, tid, c);
                a_hi[o] = c == D ? 1.f : 0.f;
                a_lo[o] = 0.f;
            }
            fence_proxy_async_smem();
            mbar_arrive(&bar->a_full);
            const int64_t row = row0 + tid;
            float xb[DN];
#pragma unroll
            for (int j = 0; j < DN; ++j) xb[j] = 0.f;
#pragma unroll 1
            for (int kk = 0; kk < D; ++kk, ++kc) {
                const int k = kk + k_rot < D ? kk + k_rot : kk + k_rot - D;
                const float nkb = row < B ? -__ldg(kb + row * D + k) : 0.f;
#pragma unroll 1
                for (int c = 0; c < NCH; ++c, ++q) {
                    const int buf = q & 1;
                    mbar_wait_bounded(&bar->th_full[buf], (q >> 1) & 1);
                    tc_fence_after_sync();
                    uint32_t ra[32], rb[32];
                    tmem_ld32_issue(tmem_base + lane_base + (uint32_t)(C_TH + buf * kRvNC), ra);
                    tmem_ld32_issue(tmem_base + lane_base + (uint32_t)(C_TH + buf * kRvNC + 32), rb);
                    tmem_ld_wait(ra);
                    tmem_ld_wait(rb);
                    tc_fence_before_sync();
                    mbar_arrive(&bar->th_free[buf]);
                    // the chunk's feature weights ride in its GEMM-2 record (landed well before theta is ready; the slot
                    // is recycled only after GEMM 2, which waits for this thread's p_full arrival)
                    mbar_wait_bounded(&bar->b2_full[buf], (q >> 1) & 1);
                    const float* __restrict__ wg = ring2 + (size_t)buf * b2f + 2 * DN * kRvNC;
                    if (q >= 2) {   // GEMM 2 of chunk q - 2 has read this p slot
                        mbar_wait_bounded(&bar->p_free[buf], ((q >> 1) - 1) & 1);
                        tc_fence_after_sync();
                    }
                    const uint32_t p_hi = tmem_base + lane_base + (uint32_t)(C_P + buf * 2 * kRvNC);
                    const uint32_t p_lo = p_hi + kRvNC;
                    auto emit = [&](uint32_t (&r)[32], const int half) {
                        uint32_t lo[32];
#pragma unroll
                        for (int i = 0; i < 32; i += 4) {
                            const float4 w4 = *reinterpret_cast<const float4*>(wg + half * 32 + i);
                            const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const float p = (wv[u] * gpode_sin_red(__uint_as_float(r[i + u]))) * nkb;
                                float h, l;
                                gpode_split_tf32_rn(p, h, l);
                                r[i + u] = __float_as_uint(h);
                                lo[i + u] = __float_as_uint(l);
                            }
                        }
                        rv_tmem_st32(p_hi + (uint32_t)(half * 32), r);
                        rv_tmem_st32(p_lo + (uint32_t)(half * 32), lo);
                    };
                    emit(ra, 0);
                    emit(rb, 1);
                    rv_tmem_st_wait();
                    tc_fence_before_sync();
                    mbar_arrive(&bar->p_full[buf]);
                }
                // ---- output k complete: G_k -> row cotangent and the lengthscale partial sums ----
                const int kbuf = kc & 1;
                mbar_wait_bounded(&bar->g_full[kbuf], (kc >> 1) & 1);
                tc_fence_after_sync();
                float mine[(DN + 31) / 32];
#pragma unroll
                for (int i = 0; i < (DN + 31) / 32; ++i) mine[i] = 0.f;
#pragma unroll
                for (int j0 = 0; j0 < DN; j0 += 16) {
                    uint32_t gq[16];
                    rv_tmem_ld16(tmem_base + lane_base + (uint32_t)(C_G + kbuf * 64 + j0), gq);
#pragma unroll
                    for (int j4 = 0; j4 < 16; j4 += 4) {
                        const int o = rv_off(kRvRows, tid, j0 + j4);   // 4 consecutive input dimensions: one 16-byte chunk
                        float4 xh = make_float4(0.f, 0.f, 0.f, 0.f), xl = xh;
                        if (j0 + j4 < KP) {
                            xh = *reinterpret_cast<const float4*>(a_hi + o);
                            xl = *reinterpret_cast<const float4*>(a_lo + o);
                        }
                        const float xv[4] = {xh.x + xl.x, xh.y + xl.y, xh.z + xl.z, xh.w + xl.w};
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int j = j0 + j4 + u;
                            const float gv = __uint_as_float(gq[j4 + u]);
                            xb[j] += gv;
                            const float v = gpode_warp_sum(j < D ? xv[u] * gv : 0.f);
                            if ((j & 31) == lane) mine[j >> 5] = v;
                        }
                    }
                }
                tc_fence_before_sync();
                mbar_arrive(&bar->g_free[kbuf]);
#pragma unroll
                for (int i = 0; i < (DN + 31) / 32; ++i) {
                    const int j = lane + 32 * i;
                    if (j < D) accw[k * DN + j] += mine[i];   // this (CTA, warp, k, j) element has one owner: plain RMW
                }
            }
            if (row < B) {
#pragma unroll
                for (int j = 0; j < DN; ++j)
                    if (j < D) gx[row * D + j] = xb[j];
            }
        }
    } else if (tid == 128 || tid == 160) {
        // TWO issuing threads: A (warp 4) streams the GEMM-1 operands and issues GEMM 1, B (warp 5) streams the GEMM-2
        // operands and issues GEMM 2. A single issuer was the bound at small D: 36-60 K = 8 MMAs per chunk at ~75 cycles of
        // issue each (ncu at D = 64: tensor pipe 26 % busy, row warps waiting). tcgen05.commit tracks the MMAs of the
        // committing thread only, which is exactly what each barrier needs; the two GEMMs write different accumulators,
        // so their relative order in the tensor pipe does not matter.
        const bool is_a = tid == 128;
        const uint32_t idesc1 = umma_idesc_tf32(kRvRows, kRvNC);
        const uint32_t idesc2 = umma_idesc_tf32(kRvRows, DN);
        const uint32_t lbo_a = kRvRows * 16, lbo_b1 = kRvNC * 16, lbo_b2 = DN * 16;
        const uint64_t desc_a_hi = umma_smem_desc(gpode_smem_u32(a_hi), lbo_a, 128);
        const uint64_t desc_a_lo = umma_smem_desc(gpode_smem_u32(a_lo), lbo_a, 128);
        const uint64_t step_a = (2u * lbo_a) >> 4, step_b1 = (2u * lbo_b1) >> 4, step_b2 = (2u * lbo_b2) >> 4;
        const uint32_t bytes1 = (uint32_t)b1f * 4u, bytes2 = (uint32_t)b2f * 4u;
        int64_t my_tiles = 0;
        for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) ++my_tiles;
        const int64_t total = my_tiles * chunks_per_tile;
        auto chunk_src = [&](const int64_t gq, int& k, int& c) {   // (k, c) of this CTA's gq-th chunk
            const int64_t local = gq % chunks_per_tile;
            const int kk = (int)(local / NCH);
            c = (int)(local - (int64_t)kk * NCH);
            k = kk + k_rot < D ? kk + k_rot : kk + k_rot - D;
        };
        if (is_a) {
            auto load1 = [&](const int64_t gq) {
                const int slot = (int)(gq & 1);
                if (gq >= 2) mbar_wait_bounded(&bar->b1_free[slot], (uint32_t)(((gq >> 1) - 1) & 1));
                int k, c;
                chunk_src(gq, k, c);
                gpode_bulk_g2s(ring1 + (size_t)slot * b1f, g1 + ((int64_t)k * NCH + c) * b1f, bytes1,
                               &bar->b1_full[slot]);
            };
            int64_t gq = 0;
            uint32_t tile_it = 0;
            if (total > 0) load1(0);
            for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tile_it) {
                mbar_wait_bounded(&bar->a_full, tile_it & 1);
                tc_fence_after_sync();
                for (int ci = 0; ci < chunks_per_tile; ++ci, ++gq) {
                    const int slot = (int)(gq & 1);
                    if (gq + 1 < total) load1(gq + 1);
                    mbar_wait_bounded(&bar->b1_full[slot], (uint32_t)((gq >> 1) & 1));
                    if (gq >= 2) mbar_wait_bounded(&bar->th_free[slot], (uint32_t)(((gq >> 1) - 1) & 1));
                    tc_fence_after_sync();
                    // ---- GEMM 1: theta[slot] = [x | 1] [Omega_k ; phase_k] chunk ----
                    const uint32_t d = tmem_base + (uint32_t)(C_TH + slot * kRvNC);
                    const float* bh = ring1 + (size_t)slot * b1f;
                    uint64_t ah = desc_a_hi, al = desc_a_lo;
                    uint64_t bhd = umma_smem_desc(gpode_smem_u32(bh), lbo_b1, 128);
                    uint64_t bld = umma_smem_desc(gpode_smem_u32(bh + KP * kRvNC), lbo_b1, 128);
                    for (int ks = 0; ks < KP / 8; ++ks, ah += step_a, al += step_a, bhd += step_b1, bld += step_b1) {
                        umma_tf32_ss(d, ah, bhd, idesc1, ks > 0 ? 1u : 0u);
                        umma_tf32_ss(d, al, bhd, idesc1, 1u);
                        umma_tf32_ss(d, ah, bld, idesc1, 1u);
                        umma_tf32_ss(d, al, bld, idesc1, 1u);   // lo lo: see large_umma.cu (theta reaches tens of radians)
                    }
                    umma_commit(&bar->th_full[slot]);
                    umma_commit(&bar->b1_free[slot]);
                }
            }
        } else {
            auto load2 = [&](const int64_t gq) {
                const int slot = (int)(gq & 1);
                if (gq >= 2) mbar_wait_bounded(&bar->b2_free[slot], (uint32_t)(((gq >> 1) - 1) & 1));
                int k, c;
                chunk_src(gq, k, c);
                gpode_bulk_g2s(ring2 + (size_t)slot * b2f, g2 + ((int64_t)k * NCH + c) * b2f, bytes2,
                               &bar->b2_full[slot]);
            };
            uint32_t kc = 0;
            if (total > 0) load2(0);
            for (int64_t gq = 0; gq < total; ++gq) {
                const int c = (int)(gq % NCH);
                // the next chunk's operands (its feature weights are read by the rows as soon as its theta is ready)
                if (gq + 1 < total) load2(gq + 1);
                // ---- GEMM 2: G[kc & 1] (+)= p(gq) Omega^T chunk ----
                const int slot = (int)(gq & 1), kbuf = (int)(kc & 1);
                mbar_wait_bounded(&bar->b2_full[slot], (uint32_t)((gq >> 1) & 1));
                if (c == 0 && kc >= 2) mbar_wait_bounded(&bar->g_free[kbuf], ((kc >> 1) - 1) & 1);
                mbar_wait_bounded(&bar->p_full[slot], (uint32_t)((gq >> 1) & 1));
                tc_fence_after_sync();
                const uint32_t dG = tmem_base + (uint32_t)(C_G + kbuf * 64);
                const uint32_t pH = tmem_base + (uint32_t)(C_P + slot * 2 * kRvNC), pL = pH + kRvNC;
                const float* bh = ring2 + (size_t)slot * b2f;
                uint64_t bhd = umma_smem_desc(gpode_smem_u32(bh), lbo_b2, 128);
                uint64_t bld = umma_smem_desc(gpode_smem_u32(bh + DN * kRvNC), lbo_b2, 128);
#pragma unroll 1
                for (int ks = 0; ks < kRvNC / 8; ++ks, bhd += step_b2, bld += step_b2) {
                    rv_mma_ts(dG, pH + (uint32_t)(ks * 8), bhd, idesc2, (c > 0 || ks > 0) ? 1u : 0u);
                    rv_mma_ts(dG, pL + (uint32_t)(ks * 8), bhd, idesc2, 1u);
                    rv_mma_ts(dG, pH + (uint32_t)(ks * 8), bld, idesc2, 1u);
                }
                umma_commit(&bar->p_free[slot]);
                umma_commit(&bar->b2_free[slot]);
                if (c == NCH - 1) {
                    umma_commit(&bar->g_full[kbuf]);
                    ++kc;
                }
            }
        }
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 4) tmem_dealloc(tmem_base, 512u);
}

size_t rv_smem(int D) {
    const size_t need = kRvData + (size_t)(2 * rv_kp(D) * kRvRows + 2 * rv_b1(D) + 2 * rv_b2(D)) * 4;
    // every CTA allocates all 512 TMEM columns: ask for more than half of the SM's shared memory so that two CTAs of this
    // kernel can never share an SM (the second one would spin in tcgen05.alloc)
    return need > 116u * 1024u ? need : 116u * 1024u;
}

}  // namespace

// ---- internal interface used by large_bwd.cu ----------------------------------------------------------------------
int64_t gpode_rv_packed_floats(int D, int S) {
    const int NCH = rv_su(S) / kRvNC;
    return (int64_t)D * NCH * (rv_b1(D) + rv_b2(D)) + (int64_t)D * rv_su(S);
}
int64_t gpode_rv_acc_floats(int D) { return (int64_t)kRvMaxCtas * 4 * rv_dn(D) * rv_dn(D); }
int gpode_rv_grid(int64_t B) {
    int sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int64_t tiles = (B + kRvRows - 1) / kRvRows;
    int64_t g = tiles < sms ? tiles : sms;
    if (g > kRvMaxCtas) g = kRvMaxCtas;
    return (int)(g < 1 ? 1 : g);
}
int gpode_rv_dn(int D) { return rv_dn(D); }

int gpode_rv_pack(const gpode_cache_t* c, float* out, cudaStream_t st) {
    rv_pack_kernel<<<592, 256, 0, st>>>(c->D, c->S, c->omega, c->phase, c->w, c->var, out);
    GPODE_LAUNCH_CHECK();
    return 0;
}

// gx = RFF part of J(x)^T kb; acc: gpode_rv_acc_floats(D) floats, one [DN x DN] row per (CTA, row warp), accumulated into
int gpode_rv_launch(const float* packed, int D, int S, const float* x, const float* kb, float* gx, int64_t B, float* acc,
                    cudaStream_t st) {
    const size_t smem = rv_smem(D);
    GPODE_CHECK_ARG(smem <= 227u * 1024u, "large-D tensor-core VJP needs %zu bytes of shared memory at D=%d", smem, D);
    const int grid = gpode_rv_grid(B);
    const int DN = rv_dn(D);
#define GPODE_RV_CASE(DN_)                                                                                              \
    case DN_:                                                                                                           \
        GPODE_CUDA(cudaFuncSetAttribute(rff_vjp_large_kernel<DN_>, cudaFuncAttributeMaxDynamicSharedMemorySize,         \
                                        (int)smem));                                                                    \
        rff_vjp_large_kernel<DN_><<<grid, kRvThreads, smem, st>>>(packed, D, S, x, kb, gx, B, acc);                    \
        break;
    switch (DN) {
        GPODE_RV_CASE(16) GPODE_RV_CASE(32) GPODE_RV_CASE(48) GPODE_RV_CASE(64)
        default:
            gpode_set_error("large-D tensor-core VJP: unsupported padded dimension %d", DN);
            return -1;
    }
#undef GPODE_RV_CASE
    GPODE_LAUNCH_CHECK();
    return 0;
}
