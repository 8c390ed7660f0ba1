// Shared helpers of the gpode_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/gpode_b200.h"

// ------------------------------------------------------------------------------------------------------------------
// error plumbing (per-thread last error string, int return codes as documented in include/gpode_b200.h)
// ------------------------------------------------------------------------------------------------------------------
void gpode_set_error(const char* fmt, ...);

#define GPODE_CHECK_ARG(cond, ...)                 \
    do {                                           \
        if (!(cond)) {                             \
            gpode_set_error(__VA_ARGS__);          \
            return -1;                             \
        }                                          \
    } while (0)

#define GPODE_CUDA(expr)                                                                          \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            gpode_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return (int)_e;                                                                       \
        }                                                                                         \
    } while (0)

#define GPODE_LAUNCH_CHECK()                                                                      \
    do {                                                                                          \
        cudaError_t _e = cudaGetLastError();                                                      \
        if (_e != cudaSuccess) {                                                                  \
            gpode_set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
            return (int)_e;                                                                       \
        }                                                                                         \
    } while (0)

// A packed block above the 227 KB a CTA can opt into (large M or S) is an argument error, reported before
// cudaFuncSetAttribute would fail on it and leave its error pending for the next launch check. static_bytes: the
// kernel's own __shared__ arrays, which count against the same 227 KB.
inline int check_smem_fits(size_t smem, size_t static_bytes = 0) {
    if (smem + static_bytes > 227 * 1024) {
        gpode_set_error("kernel does not fit on an SM (smem %zu bytes)", smem + static_bytes);
        return -2;
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------------------------
// process-wide kernel-selection options (gpode_set_option / gpode_get_option, include/gpode_b200.h): the library's only
// mutable global state. Defaults come from the environment ONCE, when the first option is read (GPODE_BWD_MMA,
// GPODE_FWD_MMA); after that only gpode_set_option changes them.
// ------------------------------------------------------------------------------------------------------------------
enum { GPODE_OPT_BWD_MMA = 0, GPODE_OPT_FWD_MMA, GPODE_OPT_COUNT };
int gpode_option(int which);  // pack.cu

// ------------------------------------------------------------------------------------------------------------------
// draw indexing of the large-D vector field (8 < D <= 64; batched Monte-Carlo prediction). n draws of `rows` rows each,
// laid out [n * rows, D]; draw q's packed block starts at packed + q * stride and its nu at nu + q * D * M. A tile never
// straddles two draws: draw q owns tiles [q * ceil(rows / TR), (q + 1) * ceil(rows / TR)) and its first tile starts at
// its row 0. done: NULL, or a per-draw flag (done[q * done_stride] != 0) read at the start of each tile -- a finished
// draw's tiles are skipped. One draw without flags ({1, B, 0, NULL, 0}) is the single-function evaluation.
// ------------------------------------------------------------------------------------------------------------------
struct GpodeDraws {
    int n;
    int64_t rows, stride;
    const int* done;
    int done_stride;
};
inline GpodeDraws gpode_one_draw(int64_t B) { return GpodeDraws{1, B, 0, nullptr, 0}; }

// ------------------------------------------------------------------------------------------------------------------
// packed parameter block (what every integrator CTA stages into shared memory with one bulk copy). Records are laid
// out for the packed dual-FP32 FMA of sm_100 (SASS FFMA2, PTX fma.rn.f32x2): two Fourier features / two output
// dimensions sit side by side so that one 64-bit register pair feeds one FFMA2.
//   rff  : one record of RP floats per (k, feature pair s2 = (2 s2, 2 s2 + 1)):
//            Omega_{0,s,k}, Omega_{0,s',k}, ..., Omega_{D-1,s,k}, Omega_{D-1,s',k}, phase_s, phase_s', a_s, a_s', pad
//            (a_{s,k} = w_{s,k} sqrt(var_k / S); an odd S is padded with a zero-weight feature).
//            Records are stored in groups of 32, 16-byte chunk-major inside a group: float offset
//              (k S2P + (s2 & ~31)) RP + c 128 + (s2 & 31) 4 + i     for chunk c, element i of the chunk,
//            so a warp whose lanes read 32 consecutive records (warp-per-row kernels) touches 512 contiguous bytes
//            per LDS.128 (conflict-free), while the row-per-thread kernels read one record by broadcast.
//   kern : [m][KS]     = Z_{m,0..D-1}, then output pairs c_{0,m}, c_{1,m}, ... (c_{k,m} = var_k nu_{k,m}; zero pad)
//   il   : [j][WP]     = output pairs -w_{0,j}, -w_{1,j}, ...  with w_{k,j} = 0.5 log2(e) / ell_{k,j}^2
//                        so that exp(-0.5 r_k^2) = 2^(sum_j d_j^2 (-w_kj))
// ------------------------------------------------------------------------------------------------------------------
struct GpodeLayout {
    int D, M, S, S2, S2P, RP, KS, WP;
    int off_rff, off_kern, off_il, total;  // in floats; every offset and `total` is a multiple of 4 (16 bytes)
    // tensor-core operand block, appended at `total` for D <= GPODE_MMAH_MAX_D:
    //  mmah : operands for mma.sync m16n8k16 f16 (vjp_mma.cuh: adjoint and forward), 152 words per (output k,
    //         tile of 8 features; tiles padded to an even count S8P with zero records):
    //           [0,64)    theta-B, lane-major (b0,b1) half2 pairs: contraction slots 0..D-1 = Omega_hi,
    //                     D..2D-1 = Omega_lo, 2D..3D-1 = Omega_hi (the state tile carries x_hi, x_hi, x_lo)
    //           [64,80)   per quad lane t: phase(2t), phase(2t+1), phase(2t), phase(2t+1)  (fp32, the MMA's C)
    //           [80,144)  G-B of the tile PAIR (2i, 2i+1), lane-major (b0,b1): the even record holds the hi
    //                     parts (tile 2i, tile 2i+1), the odd record the lo parts; one half2 =
    //                     (Bp[2t][g], Bp[2t+1][g]), Bp[s][j] = GPODE_MMAH_SCALE a_s Omega_{j,s,k}
    //           [144,152) a_s of the tile's 8 features (fp32; the forward's cosine weights)
    int S8P, off_mmah;
    int n_packed;  // floats of the whole packed block (gpode_packed_floats)
};
#define GPODE_MMAH_REC 152
#define GPODE_MMAH_MAX_D 5  // 3 D contraction slots (x_hi, x_hi, x_lo) must fit the 16 of one m16n8k16
#define GPODE_MMAH_SCALE 256.f  // keeps the fp16 low parts of a Omega out of the subnormal range

__host__ __device__ inline int gpode_round_up4(int x) { return (x + 3) & ~3; }

__host__ __device__ inline GpodeLayout gpode_layout(int D, int M, int S) {
    GpodeLayout L;
    L.D = D; L.M = M; L.S = S;
    L.S2 = (S + 1) / 2;
    L.S2P = (L.S2 + 31) & ~31;
    L.RP = gpode_round_up4(2 * D + 4);
    L.KS = gpode_round_up4(D + 2 * ((D + 1) / 2));
    L.WP = gpode_round_up4(2 * ((D + 1) / 2));
    L.off_rff = 0;
    L.off_kern = L.off_rff + D * L.S2P * L.RP;
    L.off_il = L.off_kern + M * L.KS;
    L.total = L.off_il + D * L.WP;
    L.S8P = ((S + 7) / 8 + 1) & ~1;
    L.off_mmah = L.total;
    L.n_packed = L.off_mmah + (D <= GPODE_MMAH_MAX_D ? D * L.S8P * GPODE_MMAH_REC : 0);
    return L;
}

// Accumulator block of the backward kernels. Shared-parameter gradients contract over every row of the batch; to keep
// them BITWISE REPRODUCIBLE (no floating-point atomics anywhere) each CTA writes its partial sums to a row of its own
// and gpode_grads_finalize adds the rows up in row order, in float64:
//   [0, 4)            header (int32): hdr[0] = AV rows written, hdr[1] = TW rows written, hdr[2] = RS rows written
//                                     (zeroed by the caller)
//   av rows           cap_av x (D*D + D):   A[k][j] | V[k]            one row per CTA of the adjoint / VJP kernel
//   tw rows           cap_tw x M*(D + D*D): per inducing point m:  T[k] (k < D) | W[j][k] (j, k < D)
//                                           one row per CTA (blockIdx.x) of param_grad_kernel
//   OR rs rows        float64, M*2D each:   per inducing point m:  2 ln2 T[k] (k < D) | sum d_j tq_j (j < D)
//                                           one row per CTA of the tensor-core shooting adjoint that sums the
//                                           inducing-point gradients itself (rk4_bwd_mma_kernel<D, true, true>);
//                                           they take the place of the tw rows (hdr[2] > 0 selects this form)
#define GPODE_ACC_HDR 4
#define GPODE_ACC_CAP_AV 4096
#define GPODE_ACC_CAP_TW 1024
struct GpodeAcc {
    int n_av, n_tw_m, n_rs_m;  // floats per AV row; floats per inducing point of a TW row; doubles per m of an RS row
    int64_t off_av, off_tw, off_rs, total;  // in floats; off_rs is even (8-byte aligned doubles)
};
__host__ __device__ inline GpodeAcc gpode_acc_layout(int D, int M) {
    GpodeAcc a;
    a.n_av = D * D + D;
    a.n_tw_m = D + D * D;
    a.n_rs_m = 2 * D;
    a.off_av = GPODE_ACC_HDR;
    a.off_tw = a.off_av + (int64_t)GPODE_ACC_CAP_AV * a.n_av;
    a.off_rs = a.off_tw;  // one row of 4 D M floats per SM at most: well inside the cap_tw x M (D + D^2) floats
    a.total = a.off_tw + (int64_t)GPODE_ACC_CAP_TW * M * a.n_tw_m;
    return a;
}

#define GPODE_HALF_LOG2E 0.72134752044448170368f  // 0.5 * log2(e)
#define GPODE_NEG_2LN2 (-1.3862943611198906f)          // -2 ln 2

// ------------------------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ float gpode_ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// ---- accurate sine / cosine for the latency-bound (warp-per-row) kernels ------------------------------------------
// Cody-Waite reduction by pi/2 in three float32 pieces (each product exact inside the FMA) + the Cephes minimax
// polynomials on [-pi/4, pi/4]: |error| <= 9.3e-8 for |x| <= 3e4 (checked against float64 over 1e7 points), no local
// memory (libm's cosf/sinf carry a Payne-Hanek slow path with a stack array). MUFU.COS / MUFU.SIN, which the wide
// kernels use, are ~1e-6 absolute at the |theta| ~ 10..30 rad this model produces.
__device__ __forceinline__ void gpode_trig_reduce(const float x, float& r, int& n) {
    const float q = rintf(x * 0.63661977236758138f);
    r = fmaf(q, -1.5707963705062866f, x);
    r = fmaf(q, 4.371138828673793e-08f, r);
    r = fmaf(q, 1.7151245100058819e-15f, r);
    n = (int)q;
}
__device__ __forceinline__ float gpode_sin_poly(const float r, const float z) {
    return fmaf(fmaf(fmaf(-1.9515295891e-4f, z, 8.3321608736e-3f), z, -1.6666654611e-1f), z * r, r);
}
__device__ __forceinline__ float gpode_cos_poly(const float z) {
    return fmaf(fmaf(fmaf(2.443315711809948e-5f, z, -1.388731625493765e-3f), z, 4.166664568298827e-2f), z * z,
                fmaf(-0.5f, z, 1.0f));
}
__device__ __forceinline__ float gpode_cos_cw(const float x) {
    float r;
    int n;
    gpode_trig_reduce(x, r, n);
    const float z = r * r;
    const float v = (n & 1) ? gpode_sin_poly(r, z) : gpode_cos_poly(z);
    return ((n + 1) & 2) ? -v : v;   // quadrants 0..3: cos, -sin, -cos, sin
}
__device__ __forceinline__ float gpode_sin_cw(const float x) {
    float r;
    int n;
    gpode_trig_reduce(x, r, n);
    const float z = r * r;
    const float v = (n & 1) ? gpode_cos_poly(z) : gpode_sin_poly(r, z);
    return (n & 2) ? -v : v;         // quadrants 0..3: sin, cos, -sin, -cos
}

// MUFU cosine / sine behind a two-piece Cody-Waite reduction by 2 pi (round-to-nearest by the 1.5 * 2^23 trick: four
// FP32-pipe operations, no conversion instruction). cos.approx first multiplies its argument by 1 / 2 pi in float32, so
// its absolute error grows like 1.2e-7 |theta|; with theta of tens of radians (large state dimensions: a sum over up to
// 64 inputs) that was the leading error of long solves. Reduced to [-pi, pi] it stays below ~5e-7 at any angle.
__device__ __forceinline__ float gpode_reduce_2pi(const float x) {
    const float q = fmaf(x, 0.15915494309189535f, 12582912.f) - 12582912.f;
    return fmaf(q, 1.7484555e-07f, fmaf(q, -6.2831854820251465f, x));   // 2 pi = 6.2831854820251465 - 1.7484555e-07
}
__device__ __forceinline__ float gpode_cos_red(const float x) { return __cosf(gpode_reduce_2pi(x)); }
__device__ __forceinline__ float gpode_sin_red(const float x) { return __sinf(gpode_reduce_2pi(x)); }

// ---- packed dual-FP32 arithmetic (sm_100: one issue slot, two FMAs) ---------------------------------------------
__device__ __forceinline__ unsigned long long gpode_pack2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ float2 gpode_unpack2(unsigned long long v) {
    float2 r;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
    return r;
}
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;"
        : "=l"(d)
        : "l"(gpode_pack2(a.x, a.y)), "l"(gpode_pack2(b.x, b.y)), "l"(gpode_pack2(c.x, c.y)));
    return gpode_unpack2(d);
}
__device__ __forceinline__ float2 ffma2(float a, float2 b, float2 c) { return ffma2(make_float2(a, a), b, c); }
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    unsigned long long d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(gpode_pack2(a.x, a.y)), "l"(gpode_pack2(b.x, b.y)));
    return gpode_unpack2(d);
}
__device__ __forceinline__ float2 fmul2(float a, float2 b) { return fmul2(make_float2(a, a), b); }
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(gpode_pack2(a.x, a.y)), "l"(gpode_pack2(b.x, b.y)));
    return gpode_unpack2(d);
}

// 3xTF32 split for the tcgen05 path, round-to-nearest: hi = tf32(v), lo = tf32(v - hi). Both parts have their 13 low
// mantissa bits clear, so the tensor core (which truncates) sees them exactly; the residual v - hi - lo is <= 2^-24 |v|
// and unbiased (a truncating split leaves a one-sided 2^-22 |v|, visible at D = 64 where 65 products add up).
__device__ __forceinline__ float gpode_round_tf32(float v) {
    return __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xffffe000u);
}
__device__ __forceinline__ void gpode_split_tf32_rn(float v, float& hi, float& lo) {
    hi = gpode_round_tf32(v);
    lo = gpode_round_tf32(v - hi);
}

__device__ __forceinline__ uint32_t gpode_smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}

// One thread: arm an mbarrier and pull `bytes` (multiple of 16, both sides 16B aligned) from global into shared
// memory with the bulk async-copy engine (TMA, non-tensor form: SASS UBLKCP).
__device__ __forceinline__ void gpode_mbar_init(uint64_t* mbar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(gpode_smem_u32(mbar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void gpode_bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* mbar) {
    const uint32_t kChunk = 32768;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(gpode_smem_u32(mbar)), "r"(bytes)
                 : "memory");
    for (uint32_t off = 0; off < bytes; off += kChunk) {
        uint32_t n = bytes - off < kChunk ? bytes - off : kChunk;
        asm volatile(
            "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                gpode_smem_u32((const char*)smem_dst + off)),
            "l"((const char*)gmem_src + off), "r"(n), "r"(gpode_smem_u32(mbar))
            : "memory");
    }
}

__device__ __forceinline__ void gpode_mbar_wait(uint64_t* mbar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(gpode_smem_u32(mbar)),
        "r"(parity)
        : "memory");
}

__device__ __forceinline__ float gpode_warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Deterministic second stage of every cross-CTA sum in this library: `n_rows` rows of `chunk` contiguous values (one
// row per producer CTA, `stride` values apart) are added up in float64 with a FIXED assignment -- warp w takes rows
// w, w + nwarps, ... in order, lanes take the columns, the warps' partial sums are then added in warp order -- so the
// result does not depend on how the producer CTAs were scheduled. tot[i], i < chunk, is valid after the call for the
// whole CTA. part: [nwarps][chunk_cap] float64 scratch in shared memory.
template <int PER_LANE, typename T>
__device__ __forceinline__ void gpode_sum_rows_ordered(const T* __restrict__ base, const size_t stride, const int n_rows,
                                                       const int chunk, const int chunk_cap, double* part, double* tot) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    double s[PER_LANE];
#pragma unroll
    for (int q = 0; q < PER_LANE; ++q) s[q] = 0.0;
    for (int r = warp; r < n_rows; r += nwarps) {
        const T* __restrict__ rowp = base + (size_t)r * stride;
#pragma unroll
        for (int q = 0; q < PER_LANE; ++q) {
            const int i = lane + 32 * q;
            if (i < chunk) s[q] += (double)__ldcg(rowp + i);  // written by other CTAs / an earlier kernel: bypass L1
        }
    }
#pragma unroll
    for (int q = 0; q < PER_LANE; ++q) {
        const int i = lane + 32 * q;
        if (i < chunk) part[warp * chunk_cap + i] = s[q];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < chunk; i += blockDim.x) {
        double t = 0.0;
        for (int w = 0; w < nwarps; ++w) t += part[w * chunk_cap + i];
        tot[i] = t;
    }
    __syncthreads();
}
#endif  // __CUDACC__
