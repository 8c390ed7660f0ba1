// Tensor-core adjoint of the vector field. In the VJP both random-Fourier-feature projections -- theta = x Omega and
// the back-projection G = (a sin theta) Omega^T -- run on the tensor cores as error-compensated split-fp16
// mma.sync m16n8k16 (SASS HMMA.16816.F32); sin, the RBF term, the stage algebra and every parameter-gradient partial
// sum stay FP32. Why the adjoint and not the forward kernel: ncu (profiles/r01_summary.md) shows the FFMA2 adjoint
// FMA-pipe bound (72 % busy, MUFU 36 %), and 10 of its 13 FMA-pipe cycles per (feature, output) are exactly these two
// projections; the forward kernel is MUFU-bound and gains nothing (measured with the 3xTF32 and tcgen05 forward experiments, DESIGN.md).
//
// Arithmetic replaced: autograd through DSVGP_Layer.forward (reference src/core/dsvgp.py:172-197, rff_forward
// :124-137, RBF.K src/core/kernels.py:53-99); formulas in SURVEY.md section 8(a) row A7.
//
// Split-fp16 ("3 x fp16"): v = hi + lo with hi = v & 0xffffe000 (11 significant bits, exact in fp16 while
// 6.1e-5 <= |v| < 65504) and lo = v - hi rounded to fp16; a product keeps hi hi + hi lo + lo hi, i.e. ~2^-21 relative,
// the same as the 3xTF32 split. One k = 16 MMA carries all three terms of theta because D <= 5 leaves room for the
// contraction slots (x_hi | x_hi | x_lo) . (Omega_hi ; Omega_lo ; Omega_hi); the phase enters as the accumulator
// input. Domain: |x_j| and |Omega| below 65504 (beyond that a float32 theta carries no phase information anyway).
//
// Layout. A warp owns 32 rows. Outside the tensor-core phase lane = row (state, cotangent, RBF term, RK4 algebra, no
// replication). For the tensor-core phase the warp re-reads its rows from a shared-memory stage in the MMA fragment
// layout, lane = (g = lane / 4, t = lane % 4), two 16-row tiles:
//   theta tile  C[16 x 8 features] = A[16 x 16 slots] B[16 x 8] + phase; lane (g,t) gets features 2t, 2t+1 of rows g, g+8.
//   G tile      C'[16 x 8 dims] += A'[16 x 16 features of a tile pair] B'[16 x 8], Bp = a Omega^T (pre-scaled, see
//               GPODE_MMAH_SCALE), once per split term (g_hi Bp_hi, g_lo Bp_hi, g_hi Bp_lo; three independent
//               accumulators): the fp32 accumulator pairs of theta ARE the half2 A' fragment after sin and split --
//               no shuffle, no register copy.
//               Lane (g,t) gets G for input dimensions 2t, 2t+1 of rows g, g+8 and hands the row cotangent back
//               through the stage.
#pragma once
#include <cuda_fp16.h>
#include "vf.cuh"

template <int D>
struct HShape {
    static constexpr int SXS = D | 1;                       // odd row stride: lane = row accesses are conflict-free
    static constexpr int kStageFloats = 2 * 32 * SXS + 32 * 8;  // x | 2 ln2 kb | RFF cotangent (8 dims per row)
};

// per-lane partial sums of the shared-parameter gradients, kept for the whole kernel
template <int D>
struct HAcc {
    static constexpr int KP = VfShape<D>::KP;
    float2 A2[KP][D];  // RBF: sum q'_k d_j^2 per output pair (the factor -w_kj is applied once, at the end)
    float2 Vq[KP];     // sum 2 ln2 kb_k (f_k + f_upd_k) per output pair
    float Aq[D][2];    // RFF (quad layout): sum x_j G_kj 2 ln2 kb_k SCALE for the lane's input dimensions j = 2t, 2t+1
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int k = 0; k < D; ++k) Aq[k][0] = Aq[k][1] = 0.f;
#pragma unroll
        for (int kp = 0; kp < KP; ++kp) {
            Vq[kp] = make_float2(0.f, 0.f);
#pragma unroll
            for (int j = 0; j < D; ++j) A2[kp][j] = make_float2(0.f, 0.f);
        }
    }
    // lane-partial A[k][j] | V[k] in the layout reduce_AV expects
    __device__ __forceinline__ void expand(const float* __restrict__ wnp, const int t, float (&A)[D][D],
                                           float (&Vo)[D]) const {
        constexpr int WP = VfShape<D>::WP;
        const float cG = 1.f / (GPODE_NEG_2LN2 * GPODE_MMAH_SCALE);
#pragma unroll
        for (int j = 0; j < D; ++j) {
            float w[WP];
            lds_vec<WP>(w, wnp + j * WP);
#pragma unroll
            for (int k = 0; k < D; ++k) {
                const float a2 = (k & 1) ? A2[k >> 1][j].y : A2[k >> 1][j].x;
                const float aq = ((j >> 1) == t) ? Aq[k][j & 1] : 0.f;
                A[k][j] = fmaf(w[k], a2, cG * aq);
            }
        }
#pragma unroll
        for (int k = 0; k < D; ++k) Vo[k] = ((k & 1) ? Vq[k >> 1].y : Vq[k >> 1].x) * (-1.f / GPODE_NEG_2LN2);
    }
};

__device__ __forceinline__ uint32_t gpode_pack_h2(const float lo, const float hi) {
    const __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ float gpode_trunc11(const float v) {
    return __uint_as_float(__float_as_uint(v) & 0xffffe000u);
}

// d = a b + c, m16n8k16, f16 operands, fp32 accumulate
__device__ __forceinline__ void gpode_mma_f16(float (&d)[4], const uint32_t (&a)[4], const uint32_t b0,
                                              const uint32_t b1, const float4 c) {
    asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%11,%12,%13};"
        : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1), "f"(c.x), "f"(c.y), "f"(c.z), "f"(c.w));
}
__device__ __forceinline__ void gpode_mma_f16_acc(float (&d)[4], const uint32_t (&a)[4], const uint32_t b0,
                                                  const uint32_t b1) {
    asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// Sum over the warp's lanes of v[i], returned on lane i for i < N (other lanes: unspecified). Each level halves the
// values a lane holds: the lane keeps the half its lane bit selects and adds the partner's copy of that half, so N = 32
// values cost 31 shuffles where a butterfly per value costs 160. A pair whose upper value no lane holds (i >= N) takes
// a plain butterfly; its upper lane ends with a copy that belongs to no i < N. Fixed order: bitwise reproducible.
template <int N>
__device__ __forceinline__ float gpode_warp_sum_transposed(float (&v)[32], const int lane) {
    static_assert(N >= 1 && N <= 32, "one value per lane at most");
#pragma unroll
    for (int h = 16; h >= 1; h >>= 1) {
        const bool up = (lane & h) != 0;
        float keep[16], recv[16];
#pragma unroll
        for (int r = 0; r < h && r < N; ++r) {
            if (r + h < N) {
                const float send = up ? v[r] : v[r + h];
                keep[r] = up ? v[r + h] : v[r];
                recv[r] = __shfl_xor_sync(0xffffffffu, send, h);
            } else {
                keep[r] = v[r];
                recv[r] = __shfl_xor_sync(0xffffffffu, v[r], h);
            }
        }
#pragma unroll
        for (int r = 0; r < h && r < N; r += 2) {
            if (r + 1 < h && r + 1 < N) {
                const float2 s = fadd2(make_float2(keep[r], keep[r + 1]), make_float2(recv[r], recv[r + 1]));
                v[r] = s.x;
                v[r + 1] = s.y;
            } else {
                v[r] = keep[r] + recv[r];
            }
        }
    }
    return v[0];
}

// xb = J(x)^T kb for the lane's row; parameter partial sums go to `acc`. fst = f(x) from the forward pass.
// small: staged [kern | il]; mmah: staged f16 operand records (GpodeLayout::mmah); stage: this warp's HShape stage.
// kRowSums: the per-inducing-point gradients are summed here as well, over the warp's 32 rows, into the warp's
// shared-memory accumulator rsum[m][2D] = {2 ln2 sum kb_k K_km (k < D), sum d_j tq_j (j < D)}: grad_nu and grad_Z
// without the virtual rows and the second kernel (gpode_grads_finalize applies the factors). W[k][m][j] of that kernel
// is only ever contracted with c_km / ell_kj^2, and sum_k c_km kb_k K_km d_j / ell_kj^2 = -d_j tq_j, the per-m term the
// cotangent takes anyway; so 2D sums per (row, m) replace its D + D^2 and nothing is recomputed.
template <int D, bool kRowSums = false>
__device__ __forceinline__ void vf_vjp_h(const float* __restrict__ small, const uint32_t* __restrict__ mmah,
                                         float* __restrict__ stage, const int M, const int S8P, const float (&x)[1][D],
                                         const float (&kb)[1][D], const float (&fst)[1][D], float (&xb)[1][D],
                                         HAcc<D>& acc, const int lane, float* __restrict__ rsum = nullptr) {
    static_assert(D <= GPODE_MMAH_MAX_D, "x_hi | x_hi | x_lo must fit the 16 contraction slots");
    constexpr int KS = VfShape<D>::KS, WP = VfShape<D>::WP, SXS = HShape<D>::SXS;
    const float* __restrict__ kern = small;
    const float* __restrict__ wnp = kern + M * KS;
    float* __restrict__ sx = stage;
    float* __restrict__ skb = stage + 32 * SXS;
    float* __restrict__ sxb = stage + 2 * 32 * SXS;
    const int g = lane >> 2, t = lane & 3;

    float kbn[D];  // 2 ln2 kb
#pragma unroll
    for (int j = 0; j < D; ++j) kbn[j] = -GPODE_NEG_2LN2 * kb[0][j];
    __syncwarp();  // the previous call's readers are done with the stage
#pragma unroll
    for (int j = 0; j < D; ++j) {
        sx[lane * SXS + j] = x[0][j];
        skb[lane * SXS + j] = kbn[j];
    }
    __syncwarp();

    // The two parts are independent and load different pipes (RFF: tensor + MUFU, RBF: FP32 FMA). Warps run the same
    // instruction stream in near lock-step, so half of the warps of every SM sub-partition (warp = 4 i + subpartition)
    // take the parts in the opposite order: at any time one group is in its MUFU-bound part, the other in its
    // FMA-bound part.
    const int warp_id = threadIdx.x >> 5;  // 2 + 2 per sub-partition whether warps map to it by id % 4 or by id / 4
    const bool rbf_first = ((warp_id ^ (warp_id >> 2)) & 1) != 0;
    float xbp[D];
#pragma unroll
    for (int j = 0; j < D; ++j) xbp[j] = 0.f;

    // ---- RFF part on the tensor cores (quad layout): state of one VJP ----
    uint32_t ax[2][4];
    float xsel[4][2], xbq[4][2];  // rows g + 8 r, input dimensions j = 2t, 2t+1
    auto rff_begin = [&]() {
        auto slotA = [&](const int row, const int s) -> float {  // x_hi | x_hi | x_lo | 0
            const int kind = s / D, j = s - kind * D;
            const float v = kind < 3 ? sx[row * SXS + j] : 0.f;
            const float hi = gpode_trunc11(v);
            return kind == 2 ? v - hi : hi;
        };
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
            const int r0 = 16 * mt + g, r1 = r0 + 8;
            ax[mt][0] = gpode_pack_h2(slotA(r0, 2 * t), slotA(r0, 2 * t + 1));
            ax[mt][1] = gpode_pack_h2(slotA(r1, 2 * t), slotA(r1, 2 * t + 1));
            ax[mt][2] = gpode_pack_h2(slotA(r0, 2 * t + 8), slotA(r0, 2 * t + 9));
            ax[mt][3] = gpode_pack_h2(slotA(r1, 2 * t + 8), slotA(r1, 2 * t + 9));
        }
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int jj = 0; jj < 2; ++jj) {
                xsel[r][jj] = (2 * t + jj < D) ? sx[(g + 8 * r) * SXS + 2 * t + jj] : 0.f;
                xbq[r][jj] = 0.f;
            }
    };
    // one feature-tile PAIR of output k: theta, sine, split, and the three G MMAs. The G MMAs contract over the 16
    // features of the pair (slots 0..7 = even tile, 8..15 = odd tile), so every A fragment is written in place by the
    // conversions and every B pair is one LDS.64.
    auto rff_pair = [&](const uint32_t* __restrict__ rec, float (&Ga)[2][4], float (&Gb)[2][4], float (&Gl)[2][4]) {
        uint32_t ah[2][4], al[2][4];  // [row tile][row g: even tile | row g+8: even | row g: odd | row g+8: odd]
        const uint2 bh = *reinterpret_cast<const uint2*>(rec + 80 + lane * 2);
        const uint2 bl = *reinterpret_cast<const uint2*>(rec + GPODE_MMAH_REC + 80 + lane * 2);
#pragma unroll
        for (int tl = 0; tl < 2; ++tl) {
            const uint32_t* __restrict__ rc = rec + tl * GPODE_MMAH_REC;
            const uint2 b = *reinterpret_cast<const uint2*>(rc + lane * 2);
            const float4 ph = *reinterpret_cast<const float4*>(rc + 64 + t * 4);
            float c[2][4];
            gpode_mma_f16(c[0], ax[0], b.x, b.y, ph);
            gpode_mma_f16(c[1], ax[1], b.x, b.y, ph);
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                float h[4], l[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float v = __sinf(c[mt][i]);
                    h[i] = gpode_trunc11(v);
                    l[i] = v - h[i];
                }
                ah[mt][2 * tl + 0] = gpode_pack_h2(h[0], h[1]);
                ah[mt][2 * tl + 1] = gpode_pack_h2(h[2], h[3]);
                al[mt][2 * tl + 0] = gpode_pack_h2(l[0], l[1]);
                al[mt][2 * tl + 1] = gpode_pack_h2(l[2], l[3]);
            }
        }
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
            gpode_mma_f16_acc(Ga[mt], ah[mt], bh.x, bh.y);
            gpode_mma_f16_acc(Gb[mt], al[mt], bh.x, bh.y);
            gpode_mma_f16_acc(Gl[mt], ah[mt], bl.x, bl.y);
        }
    };
    // the row's factor (2 ln2 kb_k; sign and scale are folded into cG) once per output, after the feature loop
    auto rff_output_done = [&](const int k, const float (&Ga)[2][4], const float (&Gb)[2][4], const float (&Gl)[2][4]) {
        float aq[2] = {0.f, 0.f};
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int r = 2 * mt + (i >> 1), jj = i & 1;
                const float tt = ((Ga[mt][i] + Gb[mt][i]) + Gl[mt][i]) * skb[(g + 8 * r) * SXS + k];
                xbq[r][jj] += tt;
                aq[jj] = fmaf(xsel[r][jj], tt, aq[jj]);
            }
#pragma unroll
        for (int kk = 0; kk < D; ++kk) {  // k is a run-time index here: predicated scatter keeps Aq in registers
            acc.Aq[kk][0] += (kk == k) ? aq[0] : 0.f;
            acc.Aq[kk][1] += (kk == k) ? aq[1] : 0.f;
        }
    };
    auto rff_end = [&]() {
#pragma unroll
        for (int r = 0; r < 4; ++r)
            *reinterpret_cast<float2*>(sxb + (g + 8 * r) * 8 + 2 * t) = make_float2(xbq[r][0], xbq[r][1]);
    };

    // ---- RBF part: lane = row, output pairs per FFMA2 ----
    // Full output pairs ride in FFMA2; the odd last output (D = 3, 5) goes through scalar FMAs instead of a
    // half-empty pair: the FMA pipe bounds this part (ncu: math_pipe_throttle) and a half-empty FFMA2 costs it as
    // much as a full one. (All-scalar was measured too: 0.47 ms per 1e6-row VJP against 0.43 for this split.)
    constexpr int KF = D / 2;
    constexpr bool kOdd = (D & 1) != 0;
    float2 wn[D][KF > 0 ? KF : 1];
    float wl[D];
    float2 kb2[KF > 0 ? KF : 1];
    auto rbf_begin = [&]() {
#pragma unroll
        for (int j = 0; j < D; ++j) {
            float w[WP];
            lds_vec<WP>(w, wnp + j * WP);
#pragma unroll
            for (int kp = 0; kp < KF; ++kp) wn[j][kp] = make_float2(w[2 * kp], w[2 * kp + 1]);
            wl[j] = w[D - 1];
        }
#pragma unroll
        for (int kp = 0; kp < KF; ++kp) {
            kb2[kp] = make_float2(kbn[2 * kp], kbn[2 * kp + 1]);
            acc.Vq[kp] = ffma2(kb2[kp], make_float2(fst[0][2 * kp], fst[0][2 * kp + 1]), acc.Vq[kp]);
        }
        if constexpr (kOdd) acc.Vq[KF].x = fmaf(kbn[D - 1], fst[0][D - 1], acc.Vq[KF].x);
    };
    // e0: start of the exponent sums, -inf for the padding steps of the last row-sum group (K = 0: adds nothing)
    // pz: the step's 2D row-sum values (kRowSums)
    auto rbf_step = [&](const int m, const float e0, float* __restrict__ pz) {
        float kp_[KS];
        lds_vec<KS>(kp_, kern + m * KS);
        float d[D], dd[D];
#pragma unroll
        for (int j = 0; j < D; ++j) {
            d[j] = x[0][j] - kp_[j];
            dd[j] = d[j] * d[j];
        }
        float2 tq[D];
        float tl[D];
#pragma unroll
        for (int j = 0; j < D; ++j) {
            tq[j] = make_float2(0.f, 0.f);
            tl[j] = 0.f;
        }
#pragma unroll
        for (int kp = 0; kp < KF; ++kp) {
            float2 e = make_float2(e0, e0);
#pragma unroll
            for (int j = 0; j < D; ++j) e = ffma2(dd[j], wn[j][kp], e);
            const float2 K = make_float2(gpode_ex2(e.x), gpode_ex2(e.y));
            const float2 p = fmul2(kb2[kp], K);    // 2 ln2 kb K
            const float2 q = fmul2(make_float2(kp_[D + 2 * kp], kp_[D + 2 * kp + 1]), p);   // q' = 2 ln2 kb c K
            if constexpr (kRowSums) {
                pz[2 * kp] = p.x;
                pz[2 * kp + 1] = p.y;
            }
            acc.Vq[kp] = fadd2(acc.Vq[kp], q);
#pragma unroll
            for (int j = 0; j < D; ++j) {
                tq[j] = ffma2(q, wn[j][kp], tq[j]);
                acc.A2[kp][j] = ffma2(dd[j], q, acc.A2[kp][j]);
            }
        }
        if constexpr (kOdd) {
            float e = e0;
#pragma unroll
            for (int j = 0; j < D; ++j) e = fmaf(dd[j], wl[j], e);
            const float p = kbn[D - 1] * gpode_ex2(e);
            const float q = kp_[2 * D - 1] * p;
            if constexpr (kRowSums) pz[D - 1] = p;
            acc.Vq[KF].x += q;
#pragma unroll
            for (int j = 0; j < D; ++j) {
                tl[j] = q * wl[j];
                acc.A2[KF][j].x = fmaf(dd[j], q, acc.A2[KF][j].x);
            }
        }
#pragma unroll
        for (int j = 0; j < D; ++j) {
            const float t = (tq[j].x + tq[j].y) + tl[j];
            if constexpr (kRowSums) pz[D + j] = d[j] * t;
            xbp[j] = fmaf(d[j], t, xbp[j]);
        }
    };

#pragma unroll 1
    for (int part = 0; part < 2; ++part) {
        if ((part == 0) != rbf_first) {
            rff_begin();
#pragma unroll 1   // one copy of the feature loop: the instruction cache is the scarce resource with 12 warps per SM
            for (int k = 0; k < D; ++k) {
                // three independent accumulation chains per row tile, one per split term: g_hi Bp_hi, g_lo Bp_hi, g_hi Bp_lo
                float Ga[2][4], Gb[2][4], Gl[2][4];
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                    for (int i = 0; i < 4; ++i) Ga[mt][i] = Gb[mt][i] = Gl[mt][i] = 0.f;
                const uint32_t* __restrict__ rec = mmah + (size_t)k * S8P * GPODE_MMAH_REC;
#pragma unroll 1
                for (int ft = 0; ft < S8P; ft += 2, rec += 2 * GPODE_MMAH_REC) rff_pair(rec, Ga, Gb, Gl);
                rff_output_done(k, Ga, Gb, Gl);
            }
            rff_end();
        } else {
            rbf_begin();
            if constexpr (kRowSums) {
                // G inducing points per group fill up to 32 values; one transposed warp sum per group leaves value i of
                // the group on lane i, which adds it to rsum[m0][i] (the group's values are contiguous there)
                constexpr int NV = 2 * D, G = 32 / NV;
#pragma unroll 1
                for (int m0 = 0; m0 < M; m0 += G) {
                    float v[32];
#pragma unroll
                    for (int g = 0; g < G; ++g) {
                        const bool real = m0 + g < M;
                        rbf_step(real ? m0 + g : M - 1, real ? 0.f : -INFINITY, v + g * NV);
                    }
                    const float s = gpode_warp_sum_transposed<G * NV>(v, lane);
                    const int i = m0 * NV + lane;
                    if (lane < G * NV && i < M * NV) rsum[i] += s;
                }
            } else {
#pragma unroll 2
                for (int m = 0; m < M; ++m) rbf_step(m, 0.f, nullptr);
            }
        }
    }
    __syncwarp();
    const float cG = 1.f / (GPODE_NEG_2LN2 * GPODE_MMAH_SCALE);
#pragma unroll
    for (int j = 0; j < D; ++j) xb[0][j] = fmaf(cG, sxb[lane * 8 + j], xbp[j]);
}

// f = vf(x) for the lane's row with the Fourier projection on the tensor cores: theta as in vf_vjp_h (one split-fp16
// MMA per 16 rows x 8 features), then per feature-output FMUL.RZ + MUFU.COS + one FMA on the weights a_s. The FFMA2
// forward spends D packed FMAs per feature pair on theta and is dispatch-bound next to the MUFU pipe (ncu: FMA pipe
// 64 %, XU 70 %); here theta costs the CUDA cores nothing. The RBF term is the FFMA2 one (lane = row).
template <int D>
__device__ __forceinline__ void vf_eval_h(const float* __restrict__ small, const uint32_t* __restrict__ mmah,
                                          float* __restrict__ stage, const int M, const int S8P, const float (&x)[1][D],
                                          float (&f)[1][D], const int lane) {
    static_assert(D <= GPODE_MMAH_MAX_D, "x_hi | x_hi | x_lo must fit the 16 contraction slots");
    constexpr int KS = VfShape<D>::KS, WP = VfShape<D>::WP, SXS = HShape<D>::SXS;
    const float* __restrict__ kern = small;
    const float* __restrict__ wnp = kern + M * KS;
    float* __restrict__ sx = stage;
    float* __restrict__ sxb = stage + 2 * 32 * SXS;
    const int g = lane >> 2, t = lane & 3;
    __syncwarp();  // the previous call's readers are done with the stage
#pragma unroll
    for (int j = 0; j < D; ++j) sx[lane * SXS + j] = x[0][j];
    __syncwarp();
    constexpr int KF = D / 2;
    constexpr bool kOdd = (D & 1) != 0;
    float2 wn[D][KF > 0 ? KF : 1];
    float wl[D];
#pragma unroll
    for (int j = 0; j < D; ++j) {
        float w[WP];
        lds_vec<WP>(w, wnp + j * WP);
#pragma unroll
        for (int kp = 0; kp < KF; ++kp) wn[j][kp] = make_float2(w[2 * kp], w[2 * kp + 1]);
        wl[j] = w[D - 1];
    }
    float2 fu[KF > 0 ? KF : 1];
    float fl = 0.f;
#pragma unroll
    for (int kp = 0; kp < KF; ++kp) fu[kp] = make_float2(0.f, 0.f);
    // One inducing point of the RBF term rides in every feature-tile trip of the RFF loop (a fused stream). Why fused:
    // the RFF loop alone saturates the MUFU pipe (ncu source view: 16 cosines per 129.7 cycles of a sub-partition =
    // 99 %), the RBF loop alone needs the FP32 pipe and the MUFU pipe for 40 cycles each per inducing point and reaches
    // 65 % of either, and a warp issues in order -- only a stream that carries MUFU work everywhere keeps that pipe fed
    // (tools/pipe_probe.cu: FFMA2 and MUFU do overlap when both are on offer). Measured against the two parts one after
    // the other, D = 5, M = 100, 1e6 rows: evaluation 0.528 -> 0.516 ms, RK4 step 2.123 -> 2.021 ms, bit-identical
    // results (the sums run in the same order); XU pipe 83 % of the active cycles (profiles/r02_summary.md).
    auto rbf_compute = [&](const float (&kp_)[KS]) {
        float dd[D];
#pragma unroll
        for (int j = 0; j < D; ++j) {
            const float d = x[0][j] - kp_[j];
            dd[j] = d * d;
        }
#pragma unroll
        for (int kp = 0; kp < KF; ++kp) {
            float2 e = make_float2(0.f, 0.f);
#pragma unroll
            for (int j = 0; j < D; ++j) e = ffma2(dd[j], wn[j][kp], e);
            const float2 K = make_float2(gpode_ex2(e.x), gpode_ex2(e.y));
            fu[kp] = ffma2(make_float2(kp_[D + 2 * kp], kp_[D + 2 * kp + 1]), K, fu[kp]);
        }
        if constexpr (kOdd) {
            float e = 0.f;
#pragma unroll
            for (int j = 0; j < D; ++j) e = fmaf(dd[j], wl[j], e);
            fl = fmaf(kp_[2 * D - 1], gpode_ex2(e), fl);
        }
    };
    auto rbf_step = [&](const int m) {
        float kp_[KS];
        lds_vec<KS>(kp_, kern + m * KS);
        rbf_compute(kp_);
    };
    uint32_t ax[2][4];
    auto slotA = [&](const int row, const int s) -> float {  // x_hi | x_hi | x_lo | 0
        const int kind = s / D, j = s - kind * D;
        const float v = kind < 3 ? sx[row * SXS + j] : 0.f;
        const float hi = gpode_trunc11(v);
        return kind == 2 ? v - hi : hi;
    };
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
        const int r0 = 16 * mt + g, r1 = r0 + 8;
        ax[mt][0] = gpode_pack_h2(slotA(r0, 2 * t), slotA(r0, 2 * t + 1));
        ax[mt][1] = gpode_pack_h2(slotA(r1, 2 * t), slotA(r1, 2 * t + 1));
        ax[mt][2] = gpode_pack_h2(slotA(r0, 2 * t + 8), slotA(r0, 2 * t + 9));
        ax[mt][3] = gpode_pack_h2(slotA(r1, 2 * t + 8), slotA(r1, 2 * t + 9));
    }
    int m = 0;
#pragma unroll 1
    for (int k = 0; k < D; ++k) {
        float fk[4] = {0.f, 0.f, 0.f, 0.f};
        const uint32_t* __restrict__ rc = mmah + (size_t)k * S8P * GPODE_MMAH_REC;
        const int n_fused = M - m < S8P ? M - m : S8P;   // tiles of this output that carry an inducing point
        int ft = 0;
#pragma unroll 2
        for (; ft < n_fused; ++ft, rc += GPODE_MMAH_REC, ++m) {   // branch-free body: one scheduling region
            const uint2 b = *reinterpret_cast<const uint2*>(rc + lane * 2);
            const float4 ph = *reinterpret_cast<const float4*>(rc + 64 + t * 4);
            const float2 a2 = *reinterpret_cast<const float2*>(rc + 144 + t * 2);
            float c[2][4];
            gpode_mma_f16(c[0], ax[0], b.x, b.y, ph);
            gpode_mma_f16(c[1], ax[1], b.x, b.y, ph);
            rbf_step(m);
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                fk[2 * mt] = fmaf(a2.x, __cosf(c[mt][0]), fk[2 * mt]);
                fk[2 * mt] = fmaf(a2.y, __cosf(c[mt][1]), fk[2 * mt]);
                fk[2 * mt + 1] = fmaf(a2.x, __cosf(c[mt][2]), fk[2 * mt + 1]);
                fk[2 * mt + 1] = fmaf(a2.y, __cosf(c[mt][3]), fk[2 * mt + 1]);
            }
        }
#pragma unroll 2
        for (; ft < S8P; ++ft, rc += GPODE_MMAH_REC) {
            const uint2 b = *reinterpret_cast<const uint2*>(rc + lane * 2);
            const float4 ph = *reinterpret_cast<const float4*>(rc + 64 + t * 4);
            const float2 a2 = *reinterpret_cast<const float2*>(rc + 144 + t * 2);
            float c[2][4];
            gpode_mma_f16(c[0], ax[0], b.x, b.y, ph);
            gpode_mma_f16(c[1], ax[1], b.x, b.y, ph);
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                fk[2 * mt] = fmaf(a2.x, __cosf(c[mt][0]), fk[2 * mt]);
                fk[2 * mt] = fmaf(a2.y, __cosf(c[mt][1]), fk[2 * mt]);
                fk[2 * mt + 1] = fmaf(a2.x, __cosf(c[mt][2]), fk[2 * mt + 1]);
                fk[2 * mt + 1] = fmaf(a2.y, __cosf(c[mt][3]), fk[2 * mt + 1]);
            }
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            float v = fk[r];
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            if (r == t) sxb[(g + 8 * r) * 8 + k] = v;
        }
    }
#pragma unroll 1
    for (; m < M; ++m) rbf_step(m);   // more inducing points than feature tiles
    __syncwarp();
#pragma unroll
    for (int k = 0; k < D; ++k) {
        const int kp = (k >> 1) < KF ? (k >> 1) : 0;
        const float u = (kOdd && k == D - 1) ? fl : ((k & 1) ? fu[kp].y : fu[kp].x);
        f[0][k] = sxb[lane * 8 + k] + u;
    }
}

// stage [kern | il] and the f16 operand records into shared memory (two bulk async copies, one mbarrier);
// dynamic shared memory layout: [0,16) mbarrier | small | mmah | ...
__device__ __forceinline__ void stage_params_h(unsigned char* smem_raw, const float* __restrict__ packed,
                                               const int off_kern, const int n_small, const int off_mmah,
                                               const int n_mmah) {
    uint64_t* mbar = reinterpret_cast<uint64_t*>(smem_raw);
    float* sp = reinterpret_cast<float*>(smem_raw + 16);
    if (threadIdx.x == 0) {
        gpode_mbar_init(mbar, 2);
        gpode_bulk_g2s(sp, packed + off_kern, (uint32_t)n_small * 4u, mbar);
        gpode_bulk_g2s(sp + n_small, packed + off_mmah, (uint32_t)n_mmah * 4u, mbar);
    }
    __syncthreads();
    gpode_mbar_wait(mbar, 0);
}
