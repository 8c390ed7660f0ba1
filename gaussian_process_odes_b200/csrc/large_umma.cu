// Random-Fourier-feature term of the vector field for 8 < D <= 64 on the 5th-generation tensor cores.
//
// At these state dimensions the projection theta_k = [x | 1] [Omega_k ; phase_k] (a [rows x (D+1)] x [(D+1) x S] GEMM per
// output dimension k) dominates everything: D * S * 2 (D+1) flops per row against D * S cosines. It runs as
// tcgen05.mma.cta_group::1.kind::tf32 (M = 128 rows, N = 64 features, K = 8 per instruction, (D+1)/8 K-steps),
// error-compensated 3xTF32, accumulators in TMEM. Omega does not fit in shared memory (4 MB at D = 64), so the
// pre-split, pre-tiled operand chunks of gpode_pack_cache_large stream from L2 through a two-slot shared-memory ring
// filled by bulk async copies (cp.async.bulk + mbarrier), one chunk = one (output k, 64 features) block.
//
// CTA = 160 threads: warps 0-3 own the 128 rows of a tile (thread = row = TMEM lane: tcgen05.ld, cos, weighted sum),
// warp 4 lane 0 is the producer: it issues the copies one chunk ahead and the MMAs. Ring slot i and TMEM buffer i are
// recycled together: "operands landed" (tx bytes) -> MMAs -> tcgen05.commit -> "theta ready" for the rows and
// "slot free" for the next copy; the rows' 128 arrivals -> "TMEM buffer free".
//
// Arithmetic replaced: DSVGP_Layer.rff_forward (reference src/core/dsvgp.py:124-137) for the upper sweep points of
// BASELINE.json configs[4]. Output: f_rff [B, D]; gpode_rbf_fwd_large (or gpode_vf_fwd_large_add_rbf) adds the RBF term.
// Batched prediction: both kernels take a draw index (GpodeDraws, common.cuh). The rows are those of n_sets draws, a
// tile belongs to one draw, and its operand chunks / c = var nu come from that draw's packed block.
#include "umma.cuh"

namespace {

constexpr int kLuThreads = 160;
constexpr int kLuRows = 128;
constexpr int kRbTmemCols = 128;  // RBF kernel: two buffers of up to 64 exponent columns
constexpr int kLuRing = 2;       // operand ring slots (4 was measured: no gain at D = 64, lower occupancy at D = 32)

__host__ __device__ inline int lu_kp(int D) { return (D + 1 + 7) & ~7; }          // padded K (input dims + phase slot)
// chunk width: every MMA re-reads the 128 x 8 state slice from shared memory whatever its N, so wide chunks pay once
// D is large (measured at D = 64: 2.67 -> 1.65 ms); at smaller D the smaller ring keeps more CTAs per SM
__host__ __device__ inline int lu_nc(int D) { return D > 40 ? 128 : 64; }
__host__ __device__ inline int lu_su(int D, int S) { return (S + lu_nc(D) - 1) / lu_nc(D) * lu_nc(D); }
__host__ __device__ inline int64_t lu_rec(int D) { return 2 * (int64_t)lu_kp(D) * lu_nc(D); }  // floats per chunk record

// canonical K-major no-swizzle tile of `rows` rows: [K/4 chunks][rows/8 groups][8 rows][4 floats]
__host__ __device__ inline int lu_off(int rows, int r, int q) {
    return (q >> 2) * (rows * 4) + (r >> 3) * 32 + (r & 7) * 4 + (q & 3);
}

// RBF-term operands: K_km = 2^(sum_j dd_j (-w_kj)) is a [rows x D] x [D x D] GEMM per inducing point m with A = the
// squared differences dd_j = (x_j - Z_mj)^2 (generated on the fly) and B = -W^T, w_kj = 0.5 log2(e) / ell_kj^2.
__host__ __device__ inline int lu_kd(int D) { return (D + 7) & ~7; }     // padded K of the RBF GEMM
__host__ __device__ inline int lu_nd(int D) { return (D + 15) & ~15; }   // padded N (outputs k)

// blockIdx.y = draw q: omega, phase, w, nu of draw q at their per-draw strides -> block q at out + q * stride
__global__ void pack_large_kernel(const int D, const int S, const int M, const float* __restrict__ omega,
                                  const float* __restrict__ phase, const float* __restrict__ w,
                                  const float* __restrict__ var, const float* __restrict__ ell,
                                  const float* __restrict__ nu, float* __restrict__ out, const int64_t stride) {
    omega += (int64_t)blockIdx.y * D * S * D;
    phase += (int64_t)blockIdx.y * S * D;
    w += (int64_t)blockIdx.y * S * D;
    nu += (int64_t)blockIdx.y * D * M;
    out += (int64_t)blockIdx.y * stride;
    const int NC = lu_nc(D);
    const int KP = lu_kp(D), SU = lu_su(D, S), NCH = SU / NC;
    const int64_t rec = lu_rec(D);
    const int64_t n_elem = (int64_t)D * SU * KP;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_elem; i += (int64_t)gridDim.x * blockDim.x) {
        const int q = (int)(i % KP);
        const int s = (int)((i / KP) % SU);
        const int k = (int)(i / ((int64_t)KP * SU));
        float v = 0.f;
        if (s < S) {
            if (q < D) v = omega[((size_t)q * S + s) * D + k];
            else if (q == D) v = phase[s * D + k];
        }
        float hi, lo;
        gpode_split_tf32_rn(v, hi, lo);
        float* r = out + ((int64_t)k * NCH + s / NC) * rec;
        const int o = lu_off(NC, s % NC, q);
        r[o] = hi;
        r[(int64_t)KP * NC + o] = lo;
    }
    float* aw = out + (int64_t)D * NCH * rec;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)D * SU;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int k = (int)(i / SU), s = (int)(i % SU);
        aw[i] = s < S ? w[s * D + k] * sqrtf(var[k] / (float)S) : 0.f;
    }
    // [-W^T hi | -W^T lo] (N rows = outputs k, K = input dims j, canonical tile layout) | c[m][N] = var_k nu_km
    const int KD = lu_kd(D), ND = lu_nd(D);
    float* wt = aw + (int64_t)D * SU;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < ND * KD; i += gridDim.x * blockDim.x) {
        const int k = i / KD, j = i - k * KD;
        float v = 0.f;
        if (k < D && j < D) {
            const float l = ell[k * D + j];
            v = -GPODE_HALF_LOG2E / (l * l);
        }
        float hi, lo;
        gpode_split_tf32_rn(v, hi, lo);
        const int o = lu_off(ND, k, j);
        wt[o] = hi;
        wt[ND * KD + o] = lo;
    }
    float* cp = wt + 2 * ND * KD;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < M * ND; i += gridDim.x * blockDim.x) {
        const int m = i / ND, k = i - m * ND;
        cp[i] = k < D ? var[k] * nu[k * M + m] : 0.f;
    }
}

struct LuSmem {  // byte offsets
    static constexpr int bar_afull = 0, bar_full = 8, bar_empty = 24, bar_bfull = 40, bar_bfree = 72, tmem_ptr = 104;
    static constexpr int tiles = 128;
};

__global__ void __launch_bounds__(kLuThreads)
rff_large_umma_kernel(const float* __restrict__ packed, const int D, const int S, const float* __restrict__ x,
                      float* __restrict__ f_rff, const GpodeDraws dr) {
    extern __shared__ __align__(128) unsigned char smem[];
    uint64_t* bar_afull = reinterpret_cast<uint64_t*>(smem + LuSmem::bar_afull);
    uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem + LuSmem::bar_full);
    uint64_t* bar_empty = reinterpret_cast<uint64_t*>(smem + LuSmem::bar_empty);
    uint64_t* bar_bfull = reinterpret_cast<uint64_t*>(smem + LuSmem::bar_bfull);
    uint64_t* bar_bfree = reinterpret_cast<uint64_t*>(smem + LuSmem::bar_bfree);
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + LuSmem::tmem_ptr);
    const int NC = lu_nc(D);
    const int KP = lu_kp(D), SU = lu_su(D, S), NCH = SU / NC;
    const int64_t rec = lu_rec(D);
    const int a_floats = KP * kLuRows;          // one of A_hi / A_lo
    const int b_floats = (int)rec;              // one ring slot: B_hi | B_lo
    float* a_hi = reinterpret_cast<float*>(smem + LuSmem::tiles);
    float* a_lo = a_hi + a_floats;
    float* ring = a_lo + a_floats;              // [kLuRing][b_floats]
    const int tid = threadIdx.x, warp = tid >> 5;

    if (tid == 128) {
        gpode_mbar_init(bar_afull, kLuRows);
        for (int i = 0; i < 2; ++i) {
            gpode_mbar_init(bar_full + i, 1);
            gpode_mbar_init(bar_empty + i, kLuRows);
        }
        for (int i = 0; i < kLuRing; ++i) {
            gpode_mbar_init(bar_bfull + i, 1);
            gpode_mbar_init(bar_bfree + i, 1);
        }
    }
    if (warp == 4) {
        __syncwarp();
        tmem_alloc(tmem_ptr, 2u * (uint32_t)NC);
    }
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_ptr;

    const int64_t tpd = (dr.rows + kLuRows - 1) / kLuRows;   // tiles per draw
    const int64_t n_tiles = tpd * dr.n;
    const int chunks_per_tile = D * NCH;
    // rows and producer skip the same tiles, so their chunk sequences still agree
    auto skip = [&](const int64_t tile) { return dr.done != nullptr && dr.done[(tile / tpd) * dr.done_stride] != 0; };
    // every CTA walks the output dimensions in its own rotation, so that the SMs do not all pull the same operand
    // chunk from the same L2 lines at the same moment
    const int k_rot = (int)(blockIdx.x % (unsigned)D);

    if (warp < 4) {
        uint32_t g = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            if (skip(tile)) continue;
            const int64_t q = tile / tpd, lr0 = (tile - q * tpd) * kLuRows;   // draw, its first row in this tile
            const int64_t row0 = q * dr.rows + lr0, nr = dr.rows - lr0;       // rows r < nr of the tile exist
            const float* __restrict__ aw = packed + q * dr.stride + (int64_t)D * NCH * rec;
            // ---- state tile -> shared memory (coalesced global reads), pre-split into tf32 hi / lo ----
            for (int i = tid; i < kLuRows * D; i += kLuRows) {
                const int r = i / D, j = i - r * D;
                const float v = r < nr ? __ldg(x + row0 * D + i) : 0.f;
                float hi, lo;
                gpode_split_tf32_rn(v, hi, lo);
                const int o = lu_off(kLuRows, r, j);
                a_hi[o] = hi;
                a_lo[o] = lo;
            }
            for (int q = D; q < KP; ++q) {  // slot D carries the constant 1 that picks up the phase row; the rest is 0
                const int o = lu_off(kLuRows, tid, q);
                a_hi[o] = q == D ? 1.f : 0.f;
                a_lo[o] = 0.f;
            }
            fence_proxy_async_smem();
            mbar_arrive(bar_afull);
            for (int kk = 0; kk < D; ++kk) {
                const int k = kk + k_rot < D ? kk + k_rot : kk + k_rot - D;
                float acc0 = 0.f, acc1 = 0.f;
                for (int c = 0; c < NCH; ++c, ++g) {
                    const int buf = g & 1;
                    mbar_wait_bounded(bar_full + buf, (g >> 1) & 1);
                    tc_fence_after_sync();
                    const uint32_t t0 = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * NC);
                    const float* __restrict__ wg = aw + (int64_t)k * SU + c * NC;
                    uint32_t ra[32], rb[32];
                    auto consume = [&](const uint32_t (&r)[32], const float* __restrict__ wgt) {
#pragma unroll
                        for (int i = 0; i < 32; i += 4) {
                            const float4 w4 = __ldg(reinterpret_cast<const float4*>(wgt + i));
                            acc0 = fmaf(w4.x, gpode_cos_red(__uint_as_float(r[i])), acc0);
                            acc1 = fmaf(w4.y, gpode_cos_red(__uint_as_float(r[i + 1])), acc1);
                            acc0 = fmaf(w4.z, gpode_cos_red(__uint_as_float(r[i + 2])), acc0);
                            acc1 = fmaf(w4.w, gpode_cos_red(__uint_as_float(r[i + 3])), acc1);
                        }
                    };
                    // 32-column blocks, the next block's TMEM load in flight while the current one is on the MUFU
                    tmem_ld32_issue(t0, ra);
                    for (int cc = 0; cc < NC; cc += 64) {
                        tmem_ld_wait(ra);
                        tmem_ld32_issue(t0 + cc + 32, rb);
                        consume(ra, wg + cc);
                        tmem_ld_wait(rb);
                        if (cc + 64 < NC) {
                            tmem_ld32_issue(t0 + cc + 64, ra);
                        } else {
                            tc_fence_before_sync();
                            mbar_arrive(bar_empty + buf);  // everything is in registers: the buffer may be overwritten
                        }
                        consume(rb, wg + cc + 32);
                    }
                }
                if (tid < nr) f_rff[(row0 + tid) * D + k] = acc0 + acc1;
            }
        }
    } else if (tid == 128) {
        // ---- producer: operand copies one chunk ahead, then the MMAs of the current chunk ----
        const uint32_t copy_bytes = (uint32_t)b_floats * 4u;
        // copy cursor: chunk ld_ci of tile ld_tile is the next one to copy
        int64_t ld_tile = blockIdx.x;
        while (ld_tile < n_tiles && skip(ld_tile)) ld_tile += gridDim.x;
        int ld_ci = 0;
        auto load = [&](const int64_t gq) {  // chunk gq of this CTA's sequence -> ring slot gq % kLuRing
            if (ld_tile >= n_tiles) return;
            const int slot = (int)(gq % kLuRing);
            if (gq >= kLuRing) mbar_wait_bounded(bar_bfree + slot, (uint32_t)((gq / kLuRing - 1) & 1));
            const int kk = ld_ci / NCH, c = ld_ci - kk * NCH;         // (kk, c) of the tile, kk rotated like the rows do
            const int k = kk + k_rot < D ? kk + k_rot : kk + k_rot - D;
            const float* src = packed + (ld_tile / tpd) * dr.stride + ((int64_t)k * NCH + c) * rec;
            if (++ld_ci == chunks_per_tile) {
                ld_ci = 0;
                do ld_tile += gridDim.x; while (ld_tile < n_tiles && skip(ld_tile));
            }
            float* dst = ring + (size_t)slot * b_floats;
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(gpode_smem_u32(bar_bfull + slot)),
                         "r"(copy_bytes)
                         : "memory");
            for (uint32_t off = 0; off < copy_bytes; off += 16384u) {
                const uint32_t n = copy_bytes - off < 16384u ? copy_bytes - off : 16384u;
                asm volatile(
                    "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                        gpode_smem_u32((const char*)dst + off)),
                    "l"((const char*)src + off), "r"(n), "r"(gpode_smem_u32(bar_bfull + slot))
                    : "memory");
            }
        };
        const uint32_t idesc = umma_idesc_tf32(kLuRows, NC);
        const uint32_t lbo_a = kLuRows * 16, lbo_b = (uint32_t)NC * 16;  // bytes between consecutive 16-byte K chunks
        const uint64_t desc_a_hi = umma_smem_desc(gpode_smem_u32(a_hi), lbo_a, 128);
        const uint64_t desc_a_lo = umma_smem_desc(gpode_smem_u32(a_lo), lbo_a, 128);
        const uint64_t step_a = (2u * lbo_a) >> 4, step_b = (2u * lbo_b) >> 4;  // one K-step = two K chunks
        int64_t gq = 0;
        uint32_t tile_it = 0;
        for (int64_t q = 0; q < kLuRing - 1; ++q) load(q);
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            if (skip(tile)) continue;
            mbar_wait_bounded(bar_afull, tile_it & 1);
            ++tile_it;
            tc_fence_after_sync();
            for (int ci = 0; ci < chunks_per_tile; ++ci, ++gq) {
                const int slot = (int)(gq % kLuRing), tb = (int)(gq & 1);
                load(gq + kLuRing - 1);
                mbar_wait_bounded(bar_bfull + slot, (uint32_t)((gq / kLuRing) & 1));
                if (gq >= 2) mbar_wait_bounded(bar_empty + tb, (uint32_t)(((gq >> 1) - 1) & 1));
                tc_fence_after_sync();
                const uint32_t d = tmem_base + (uint32_t)(tb * NC);
                const float* bh = ring + (size_t)slot * b_floats;
                const float* bl = bh + KP * NC;
                // descriptors are built once per chunk; a K-step only advances the 16-byte-granular start address
                // (the issuing thread's own instruction latency is what paces back-to-back MMAs)
                uint64_t ah = desc_a_hi, al = desc_a_lo;
                uint64_t bhd = umma_smem_desc(gpode_smem_u32(bh), lbo_b, 128);
                uint64_t bld = umma_smem_desc(gpode_smem_u32(bl), lbo_b, 128);
                // all FOUR products of the split (hi hi, lo hi, hi lo, lo lo): the angle theta reaches tens of radians, and
                // without the lo lo term (2^-22 of |x||Omega|) the gradients of a 30-step solve with whitened nu were
                // 3.3x further from float64 than the reference's own float32 run; the tensor pipe has the slack (the
                // kernel is bound by the L2 operand stream / the row threads)
                umma_tf32_ss(d, ah, bhd, idesc, 0u);
                umma_tf32_ss(d, al, bhd, idesc, 1u);
                umma_tf32_ss(d, ah, bld, idesc, 1u);
                umma_tf32_ss(d, al, bld, idesc, 1u);
                for (int ks = 1; ks < KP / 8; ++ks) {
                    ah += step_a; al += step_a; bhd += step_b; bld += step_b;
                    umma_tf32_ss(d, ah, bhd, idesc, 1u);
                    umma_tf32_ss(d, al, bhd, idesc, 1u);
                    umma_tf32_ss(d, ah, bld, idesc, 1u);
                    umma_tf32_ss(d, al, bld, idesc, 1u);
                }
                umma_commit(bar_full + tb);     // theta of this chunk is complete -> rows
                umma_commit(bar_bfree + slot);  // ... and the ring slot has been read -> a later copy
            }
        }
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 4) tmem_dealloc(tmem_base, 2u * (uint32_t)NC);
}


// ------------------------------------------------------------------------------------------------------------------
// RBF (pathwise update) term for 8 < D <= 64: f_k += sum_m c_km 2^(sum_j dd_mj (-w_kj)).  Per inducing point m one
// tcgen05 GEMM [128 rows x D] x [D x D]: warps 4-7 ("producers", thread = row) build the squared-difference tile of m
// in shared memory (pre-split 3xTF32, canonical layout), warp 8 lane 0 issues the MMAs against the resident -W^T, warps
// 0-3 ("consumers", thread = row = TMEM lane) read the exponents, take 2^e on the MUFU and accumulate c_km K_km in
// registers. Two A slots / two TMEM buffers keep the three stages running concurrently.
// Arithmetic replaced: RBF.K + the einsum of DSVGP_Layer.forward (reference src/core/kernels.py:53-99,
// src/core/dsvgp.py:188-195).
// ------------------------------------------------------------------------------------------------------------------
constexpr int kRbThreads = 288;

struct RbSmem {
    static constexpr int bar_afull = 0, bar_afree = 16, bar_full = 32, bar_empty = 48, tmem_ptr = 64;
    static constexpr int data = 128;
};

template <int NDT>   // NDT = lu_nd(D): sizes the per-row accumulators, so small D keeps several CTAs resident per SM
__global__ void __launch_bounds__(kRbThreads, NDT <= 16 ? 3 : (NDT <= 32 ? 2 : 1))
rbf_large_umma_kernel(const float* __restrict__ packed, const int D, const int S, const int M,
                      const float* __restrict__ Z, const float* __restrict__ x, const float* __restrict__ f_rff,
                      float* __restrict__ f_out, const GpodeDraws dr) {
    extern __shared__ __align__(128) unsigned char smem[];
    uint64_t* bar_afull = reinterpret_cast<uint64_t*>(smem + RbSmem::bar_afull);  // [2] 128 producer arrivals
    uint64_t* bar_afree = reinterpret_cast<uint64_t*>(smem + RbSmem::bar_afree);  // [2] commit
    uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem + RbSmem::bar_full);    // [2] commit
    uint64_t* bar_empty = reinterpret_cast<uint64_t*>(smem + RbSmem::bar_empty);  // [2] 128 consumer arrivals
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + RbSmem::tmem_ptr);
    const int KD = lu_kd(D), K4 = KD / 4;
    constexpr int ND = NDT;
    const int SU = lu_su(D, S), NCH = SU / lu_nc(D);
    const float* __restrict__ wt_g = packed + (int64_t)D * NCH * lu_rec(D) + (int64_t)D * SU;
    const int64_t cp_off = (int64_t)D * NCH * lu_rec(D) + (int64_t)D * SU + 2 * ND * KD;   // c = var nu: per draw
    float* wt = reinterpret_cast<float*>(smem + RbSmem::data);   // [-W^T hi | lo], 2 ND KD floats
    float* zs = wt + 2 * ND * KD;                                 // [M][KD], zero padded
    float* xs = zs + M * KD;                                      // [K4][128][4]
    float* at = xs + KD * kLuRows;                                // 2 slots x (A_hi | A_lo), each KD*128 floats
    const int a_floats = KD * kLuRows;
    const int tid = threadIdx.x, warp = tid >> 5;

    for (int i = tid; i < 2 * ND * KD; i += kRbThreads) wt[i] = __ldg(wt_g + i);
    for (int i = tid; i < M * KD; i += kRbThreads) {
        const int m = i / KD, j = i - m * KD;
        zs[i] = j < D ? __ldg(Z + m * D + j) : 0.f;
    }
    if (tid == 256) {
        for (int i = 0; i < 2; ++i) {
            gpode_mbar_init(bar_afull + i, kLuRows);
            gpode_mbar_init(bar_afree + i, 1);
            gpode_mbar_init(bar_full + i, 1);
            gpode_mbar_init(bar_empty + i, kLuRows);
        }
    }
    if (warp == 8) {
        __syncwarp();
        tmem_alloc(tmem_ptr, kRbTmemCols);
    }
    fence_proxy_async_smem();  // -W^T was written with ordinary stores and is read by the tensor core
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_ptr;
    const int64_t tpd = (dr.rows + kLuRows - 1) / kLuRows;   // tiles per draw; -W^T and Z are shared by all draws
    const int64_t n_tiles = tpd * dr.n;
    auto skip = [&](const int64_t tile) { return dr.done != nullptr && dr.done[(tile / tpd) * dr.done_stride] != 0; };

    if (warp < 4) {
        // ---- consumers: exponent -> 2^e -> weighted sum over the inducing points ----
        uint32_t g = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            if (skip(tile)) continue;
            const float* __restrict__ cp_g = packed + (tile / tpd) * dr.stride + cp_off;
            float f[ND];
#pragma unroll
            for (int k = 0; k < ND; ++k) f[k] = 0.f;
            for (int m = 0; m < M; ++m, ++g) {
                const int buf = g & 1;
                mbar_wait_bounded(bar_full + buf, (g >> 1) & 1);
                tc_fence_after_sync();
                const uint32_t t0 = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * 64);
                const float* __restrict__ cm = cp_g + (int64_t)m * ND;
                uint32_t ra[32], rb[ND > 32 ? 32 : 1];
                tmem_ld32_issue(t0, ra);
                if constexpr (ND > 32) tmem_ld32_issue(t0 + 32, rb);
                tmem_ld_wait(ra);
                if constexpr (ND > 32) tmem_ld_wait(rb);  // (one wait covers both loads; this pins rb's readers behind it)
                tc_fence_before_sync();
                mbar_arrive(bar_empty + buf);
#pragma unroll
                for (int q = 0; q < 2; ++q) {          // 16-column groups of the first 32 columns
                    if (q * 16 < ND) {
#pragma unroll
                        for (int i = 0; i < 16; i += 4) {
                            const float4 c4 = __ldg(reinterpret_cast<const float4*>(cm + q * 16 + i));
                            f[q * 16 + i] = fmaf(c4.x, gpode_ex2(__uint_as_float(ra[q * 16 + i])), f[q * 16 + i]);
                            f[q * 16 + i + 1] = fmaf(c4.y, gpode_ex2(__uint_as_float(ra[q * 16 + i + 1])), f[q * 16 + i + 1]);
                            f[q * 16 + i + 2] = fmaf(c4.z, gpode_ex2(__uint_as_float(ra[q * 16 + i + 2])), f[q * 16 + i + 2]);
                            f[q * 16 + i + 3] = fmaf(c4.w, gpode_ex2(__uint_as_float(ra[q * 16 + i + 3])), f[q * 16 + i + 3]);
                        }
                    }
                }
                if constexpr (ND > 32) {
#pragma unroll
                for (int q = 2; q < 4; ++q) {
                    if (q * 16 < ND) {
#pragma unroll
                        for (int i = 0; i < 16; i += 4) {
                            const int c = (q - 2) * 16 + i;
                            const float4 c4 = __ldg(reinterpret_cast<const float4*>(cm + q * 16 + i));
                            f[q * 16 + i] = fmaf(c4.x, gpode_ex2(__uint_as_float(rb[c])), f[q * 16 + i]);
                            f[q * 16 + i + 1] = fmaf(c4.y, gpode_ex2(__uint_as_float(rb[c + 1])), f[q * 16 + i + 1]);
                            f[q * 16 + i + 2] = fmaf(c4.z, gpode_ex2(__uint_as_float(rb[c + 2])), f[q * 16 + i + 2]);
                            f[q * 16 + i + 3] = fmaf(c4.w, gpode_ex2(__uint_as_float(rb[c + 3])), f[q * 16 + i + 3]);
                        }
                    }
                }
                }
            }
            const int64_t q = tile / tpd, lr = (tile - q * tpd) * kLuRows + tid, row = q * dr.rows + lr;
            if (lr < dr.rows) {
#pragma unroll
                for (int k = 0; k < ND; ++k)
                    if (k < D) f_out[row * D + k] = __ldg(f_rff + row * D + k) + f[k];
            }
        }
    } else if (warp < 8) {
        // ---- producers: dd tile of inducing point m, pre-split, canonical layout ----
        const int r = tid - 128;
        uint32_t g = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            if (skip(tile)) continue;
            const int64_t q = tile / tpd, lr0 = (tile - q * tpd) * kLuRows;
            const int64_t row0 = q * dr.rows + lr0, nr = dr.rows - lr0;
            asm volatile("bar.sync 1, 128;" ::: "memory");  // the previous tile's readers of xs are done
            for (int i = r; i < kLuRows * D; i += kLuRows) {
                const int rr = i / D, j = i - rr * D;
                xs[(j >> 2) * (kLuRows * 4) + rr * 4 + (j & 3)] = rr < nr ? __ldg(x + row0 * D + i) : 0.f;
            }
            for (int j = D; j < KD; ++j) xs[(j >> 2) * (kLuRows * 4) + r * 4 + (j & 3)] = 0.f;
            asm volatile("bar.sync 1, 128;" ::: "memory");
            for (int m = 0; m < M; ++m, ++g) {
                const int slot = g & 1;
                if (g >= 2) mbar_wait_bounded(bar_afree + slot, ((g >> 1) - 1) & 1);
                float* ah = at + (size_t)slot * 2 * a_floats;
                float* al = ah + a_floats;
                const int ro = (r >> 3) * 32 + (r & 7) * 4;
                for (int j4 = 0; j4 < K4; ++j4) {
                    const float4 x4 = *reinterpret_cast<const float4*>(xs + (j4 * kLuRows + r) * 4);
                    const float4 z4 = *reinterpret_cast<const float4*>(zs + m * KD + j4 * 4);
                    const float d0 = x4.x - z4.x, d1 = x4.y - z4.y, d2 = x4.z - z4.z, d3 = x4.w - z4.w;
                    float4 h, l;
                    gpode_split_tf32_rn(d0 * d0, h.x, l.x);
                    gpode_split_tf32_rn(d1 * d1, h.y, l.y);
                    gpode_split_tf32_rn(d2 * d2, h.z, l.z);
                    gpode_split_tf32_rn(d3 * d3, h.w, l.w);
                    *reinterpret_cast<float4*>(ah + j4 * (kLuRows * 4) + ro) = h;
                    *reinterpret_cast<float4*>(al + j4 * (kLuRows * 4) + ro) = l;
                }
                fence_proxy_async_smem();
                mbar_arrive(bar_afull + slot);
            }
        }
    } else if (tid == 256) {
        // ---- MMA issue ----
        const uint32_t idesc = umma_idesc_tf32(kLuRows, ND);
        const uint32_t lbo_a = kLuRows * 16, lbo_b = (uint32_t)ND * 16;
        // all descriptors up front; a K-step advances the 16-byte-granular start address by two K chunks
        const uint64_t desc_a[2] = {umma_smem_desc(gpode_smem_u32(at), lbo_a, 128),
                                    umma_smem_desc(gpode_smem_u32(at + 2 * a_floats), lbo_a, 128)};
        const uint64_t lo_a = ((uint32_t)a_floats * 4u) >> 4;
        const uint64_t desc_b_hi = umma_smem_desc(gpode_smem_u32(wt), lbo_b, 128);
        const uint64_t desc_b_lo = umma_smem_desc(gpode_smem_u32(wt + ND * KD), lbo_b, 128);
        const uint64_t step_a = (2u * lbo_a) >> 4, step_b = (2u * lbo_b) >> 4;
        uint32_t g = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            if (skip(tile)) continue;
            for (int m = 0; m < M; ++m, ++g) {
                const int slot = g & 1;
                mbar_wait_bounded(bar_afull + slot, (g >> 1) & 1);
                if (g >= 2) mbar_wait_bounded(bar_empty + slot, ((g >> 1) - 1) & 1);
                tc_fence_after_sync();
                const uint32_t d = tmem_base + (uint32_t)(slot * 64);
                uint64_t ahd = desc_a[slot], ald = desc_a[slot] + lo_a;
                uint64_t bhd = desc_b_hi, bld = desc_b_lo;
                umma_tf32_ss(d, ahd, bhd, idesc, 0u);
                umma_tf32_ss(d, ald, bhd, idesc, 1u);
                umma_tf32_ss(d, ahd, bld, idesc, 1u);
                for (int ks = 1; ks < KD / 8; ++ks) {
                    ahd += step_a; ald += step_a; bhd += step_b; bld += step_b;
                    umma_tf32_ss(d, ahd, bhd, idesc, 1u);
                    umma_tf32_ss(d, ald, bhd, idesc, 1u);
                    umma_tf32_ss(d, ahd, bld, idesc, 1u);
                }
                umma_commit(bar_full + slot);
                umma_commit(bar_afree + slot);
            }
        }
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 8) tmem_dealloc(tmem_base, kRbTmemCols);
}

}  // namespace

extern "C" int64_t gpode_packed_large_floats(int D, int M, int S) {
    if (D <= GPODE_MAX_D || D > GPODE_MAX_D_LARGE || S < 1 || M < 1) return -1;
    const int SU = lu_su(D, S);
    return (int64_t)D * (SU / lu_nc(D)) * lu_rec(D) + (int64_t)D * SU + 2 * (int64_t)lu_nd(D) * lu_kd(D) +
           (int64_t)M * lu_nd(D);
}

int gpode_vf_large_add_rbf_draws(const gpode_cache_t* c, const float* x, const float* f_rff, float* f,
                                 const GpodeDraws& dr, cudaStream_t st);  // large_d.cu

// n_sets blocks back to back, gpode_packed_large_floats(D,M,S) floats apart; omega / phase / w / nu of the cache carry
// the leading draw axis (a one-draw cache is the plain one)
static int pack_large(const gpode_cache_t* c, int n_sets, float* packed, void* stream) {
    GPODE_CHECK_ARG(c != nullptr && packed != nullptr, "cache / packed is NULL");
    GPODE_CHECK_ARG(c->D > GPODE_MAX_D && c->D <= GPODE_MAX_D_LARGE, "large-D path needs %d < D <= %d, got %d",
                    GPODE_MAX_D, GPODE_MAX_D_LARGE, c->D);
    GPODE_CHECK_ARG(n_sets >= 1 && n_sets <= 65535, "n_sets=%d outside 1..65535", n_sets);
    GPODE_CHECK_ARG(c->S >= 1 && c->M >= 1 && c->omega && c->phase && c->w && c->var && c->ell && c->nu,
                    "cache tensor is NULL");
    const unsigned gx = n_sets < 592 ? 592u / (unsigned)n_sets : 1u;
    pack_large_kernel<<<dim3(gx, n_sets), 256, 0, (cudaStream_t)stream>>>(
        c->D, c->S, c->M, c->omega, c->phase, c->w, c->var, c->ell, c->nu, packed,
        gpode_packed_large_floats(c->D, c->M, c->S));
    GPODE_LAUNCH_CHECK();
    return 0;
}

extern "C" int gpode_pack_cache_large(const gpode_cache_t* c, float* packed, void* stream) {
    return pack_large(c, 1, packed, stream);
}

extern "C" int gpode_pack_cache_large_sets(const gpode_cache_t* c, int n_sets, float* packed, void* stream) {
    return pack_large(c, n_sets, packed, stream);
}

static int rff_launch(const float* packed_large, int D, int S, const float* x, float* f_rff, const GpodeDraws& dr,
                      cudaStream_t st) {
    const int KP = lu_kp(D);
    const size_t smem = LuSmem::tiles + (size_t)(2 * KP * kLuRows + kLuRing * lu_rec(D)) * 4;
    GPODE_CUDA(cudaFuncSetAttribute(rff_large_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int sms = 148, dev = 0;
    GPODE_CUDA(cudaGetDevice(&dev));
    GPODE_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    int occ = (int)((227u * 1024u) / (smem + 1024u));   // shared memory and TMEM (512 columns) bound the residency
    if (occ > 512 / (2 * lu_nc(D))) occ = 512 / (2 * lu_nc(D));
    if (occ < 1) {
        gpode_set_error("large-D tensor-core kernel does not fit on an SM (smem %zu bytes)", smem);
        return -2;
    }
    const int64_t tiles = (dr.rows + kLuRows - 1) / kLuRows * dr.n, cap = (int64_t)sms * occ;
    rff_large_umma_kernel<<<(unsigned)(tiles < cap ? tiles : cap), kLuThreads, smem, st>>>(packed_large, D, S, x, f_rff,
                                                                                         dr);
    GPODE_LAUNCH_CHECK();
    return 0;
}

extern "C" int gpode_rff_fwd_large(const float* packed_large, int D, int S, const float* x, float* f_rff, int64_t B,
                                   void* stream) {
    GPODE_CHECK_ARG(packed_large && x && f_rff, "NULL argument");
    GPODE_CHECK_ARG(D > GPODE_MAX_D && D <= GPODE_MAX_D_LARGE && S >= 1 && B >= 0, "bad sizes D=%d S=%d", D, S);
    if (B == 0) return 0;
    return rff_launch(packed_large, D, S, x, f_rff, gpode_one_draw(B), (cudaStream_t)stream);
}

static size_t rbf_smem(int D, int M) {
    const int KD = lu_kd(D), ND = lu_nd(D);
    return RbSmem::data + (size_t)(2 * ND * KD + M * KD + KD * kLuRows + 4 * KD * kLuRows) * 4;
}

static int rbf_launch(const float* packed_large, int D, int M, int S, const float* Z, const float* x, const float* f_rff,
                      float* f, const GpodeDraws& dr, cudaStream_t st) {
    const int ND = lu_nd(D);
    const size_t smem = rbf_smem(D, M);
    GPODE_CHECK_ARG(smem <= 227u * 1024u, "M=%d too large for the shared-memory copy of Z (needs %zu bytes)", M, smem);
    void (*kern)(const float*, int, int, int, const float*, const float*, const float*, float*, GpodeDraws) =
        ND == 16 ? rbf_large_umma_kernel<16> : ND == 32 ? rbf_large_umma_kernel<32>
        : ND == 48 ? rbf_large_umma_kernel<48> : rbf_large_umma_kernel<64>;
    GPODE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int sms = 148, dev = 0;
    GPODE_CUDA(cudaGetDevice(&dev));
    GPODE_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    int occ = (int)((227u * 1024u) / (smem + 1024u));
    if (occ > 512 / kRbTmemCols) occ = 512 / kRbTmemCols;
    if (occ * kRbThreads > 2048) occ = 2048 / kRbThreads;
    // registers bound the residency below shared memory and TMEM for ND >= 32 (allocation: 8-register granules per thread)
    cudaFuncAttributes fa;
    GPODE_CUDA(cudaFuncGetAttributes(&fa, kern));
    GPODE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    const int reg_occ = 65536 / (((fa.numRegs + 7) & ~7) * kRbThreads);
    if (occ > reg_occ) occ = reg_occ;
    if (occ < 1) occ = 1;
    const int64_t tiles = (dr.rows + kLuRows - 1) / kLuRows * dr.n, cap = (int64_t)sms * occ;
    kern<<<(unsigned)(tiles < cap ? tiles : cap), kRbThreads, smem, st>>>(packed_large, D, S, M, Z, x, f_rff, f, dr);
    GPODE_LAUNCH_CHECK();
    return 0;
}

extern "C" int gpode_rbf_fwd_large(const float* packed_large, int D, int M, int S, const float* Z, const float* x,
                                   const float* f_rff, float* f, int64_t B, void* stream) {
    GPODE_CHECK_ARG(packed_large && Z && x && f_rff && f, "NULL argument");
    GPODE_CHECK_ARG(D > GPODE_MAX_D && D <= GPODE_MAX_D_LARGE && S >= 1 && M >= 1 && B >= 0, "bad sizes D=%d M=%d", D, M);
    if (B == 0) return 0;
    return rbf_launch(packed_large, D, M, S, Z, x, f_rff, f, gpode_one_draw(B), (cudaStream_t)stream);
}

// f = vf(x) for 8 < D <= 64: Fourier-feature term, then the RBF term added to it, both on the tcgen05 tensor cores (the
// RBF term falls back to the tiled FP32 kernel when Z does not fit its shared-memory copy). tmp: rows D floats.
// dr: the draws (gpode_one_draw(B) for one function); dr.stride must be gpode_packed_large_floats(D,M,S).
int gpode_vf_large_eval(const float* packed_large, const gpode_cache_t* c, const float* x, float* tmp, float* f,
                        const GpodeDraws& dr, cudaStream_t st) {
    if (int rc = rff_launch(packed_large, c->D, c->S, x, tmp, dr, st)) return rc;
    if (rbf_smem(c->D, c->M) <= 227u * 1024u) return rbf_launch(packed_large, c->D, c->M, c->S, c->Z, x, tmp, f, dr, st);
    return gpode_vf_large_add_rbf_draws(c, x, tmp, f, dr, st);
}

extern "C" int gpode_vf_fwd_large_sets(const float* packed_large, const gpode_cache_t* c, int n_sets, int64_t set_rows,
                                       const float* x, float* tmp, float* f, void* stream) {
    GPODE_CHECK_ARG(c != nullptr && c->D > GPODE_MAX_D && c->D <= GPODE_MAX_D_LARGE, "large-D path needs %d < D <= %d",
                    GPODE_MAX_D, GPODE_MAX_D_LARGE);
    GPODE_CHECK_ARG(n_sets >= 1 && n_sets <= 65535 && set_rows >= 0, "n_sets=%d outside 1..65535 or set_rows < 0",
                    n_sets);
    GPODE_CHECK_ARG(c->M >= 1 && c->S >= 1 && c->Z && c->nu && c->ell && c->var, "cache tensor is NULL");
    if (set_rows == 0) return 0;
    GPODE_CHECK_ARG(packed_large && x && tmp && f, "NULL argument");
    const GpodeDraws dr{n_sets, set_rows, gpode_packed_large_floats(c->D, c->M, c->S), nullptr, 0};
    return gpode_vf_large_eval(packed_large, c, x, tmp, f, dr, (cudaStream_t)stream);
}
