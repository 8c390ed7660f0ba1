// Fused multiple-shooting ELBO epilogue (SURVEY.md section 8f item 2).
//
// In UniformSequenceModel.build_lowerbound_terms (reference src/gpode_shooting/models.py:108-146) every row of the
// (S_mc, N, T) segment batch is integrated over ONE interval and its end point x(t+1; s_t) is used twice:
//   * observation term   log N(ys[n,t] | decode(pred), var)                  (src/core/likelihoods.py:27-45,
//                                                                             decoder src/misc/mocap_utils.py:24-34)
//   * shooting constraint log p(ss[s,n,t+1] | loc = pred, scale), t < T-1    (src/core/constraints.py:26-36,56-66;
//                                                                             models.py:134-135)
// The reference (and round 1 of this library) writes the (B, 2, D) trajectory tensor, re-reads it in two more passes
// and again in their backward. Here the thread that owns a row in the RK4 kernel evaluates both terms on the end point
// while it is still in registers, and keeps two "seed" vectors per row -- d(loglik sum)/d pred and
// d(constraint sum)/d pred -- from which the adjoint kernel starts (lambda_T = g_ll seed_ll + g_cons seed_c with the
// two upstream scalar gradients read from device memory), so the trajectory tensor is never materialised.
//
// Sums are bitwise reproducible: per-thread float64 partials, warp shuffles, warps in warp order, one row of `work`
// per CTA, rows added in row order by shoot_sum_kernel (common.cuh gpode_sum_rows_ordered).
#pragma once
#include "common.cuh"

struct ShootArgs {
    const float* ys;          // [N, T, Dobs]
    const float* W;           // [D, Dobs]
    const float* bias;        // [Dobs] or NULL
    const float* lik_var;     // [Dobs]
    const float* cons_scale;  // 1 float
    const float* ss;          // [S_mc, N, T, D] all sampled states (rows of the segment batch)
    int N, T, Dobs, laplace;  // laplace: constraint family
    int halo;                 // 1: the LAST time index of every sequence is a neighbour state only (time sharding): no
                              // observation term for it (its seeds are zero, so its adjoint contributes nothing)
    int64_t row_lo;           // first row of this launch in the (S_mc, N, T) batch
    int64_t n_total;          // S_mc * N * T
    float* pred_out;          // [B_local, D] or NULL
    float* seeds;             // [2, B_local, D] or NULL (forward without gradients)
    double* work;             // [gridDim.x][2 + Dobs]
};

// shared-memory region of the epilogue (16-byte aligned): floats [W D x DP | bias DP | 1/var DP | log(2 pi var) DP] with
// the observed dimension padded to DP = roundup4(Dobs) (zero padding: a padded dimension contributes exactly 0), so that
// four observed dimensions are one LDS.128 per operand; then float64 [nwarps][2 + Dobs] accumulators (loglik,
// constraint, d loglik / d var_d)
__host__ __device__ inline int shoot_dp(int Dobs) { return (Dobs + 3) & ~3; }
__host__ __device__ inline size_t shoot_smem_floats(int D, int Dobs) { return (size_t)(D + 3) * shoot_dp(Dobs); }
__host__ __device__ inline size_t shoot_smem_bytes(int D, int Dobs, int nwarps) {
    return shoot_smem_floats(D, Dobs) * 4 + (size_t)nwarps * (2 + Dobs) * 8;
}
#define GPODE_SHOOT_MAX_DOBS 128

// integrate.cu, shared with the large-D step (large_shoot.cu): checks of the descriptor and its row range; the ordered
// float64 sum of the per-CTA partial rows [n_rows][cols] (cols = 2 + D_obs) into sums[2] and g_var[D_obs] (may be NULL)
int gpode_check_shoot(const gpode_shoot_t* sh);
int gpode_shoot_sum_launch(const double* work, int n_rows, int cols, double* sums, float* g_var, cudaStream_t st);

#ifdef __CUDACC__
template <int D>
struct ShootSmem {
    const float* W;
    const float* bias;
    const float* iv;
    const float* lv;
    double* wacc;  // this warp's [2 + Dobs]
    float inv, inv2, c0;

    // all threads of the CTA; `base` is 8-byte aligned. Ends with a __syncthreads().
    __device__ __forceinline__ void init(unsigned char* base, const ShootArgs& a) {
        float* f = reinterpret_cast<float*>(base);
        const int Dobs = a.Dobs, DP = shoot_dp(Dobs);
        float* sW = f;
        float* sb = f + D * DP;
        float* siv = sb + DP;
        float* slv = siv + DP;
        for (int i = threadIdx.x; i < D * DP; i += blockDim.x) {
            const int l = i / DP, d = i - l * DP;
            sW[i] = d < Dobs ? a.W[l * Dobs + d] : 0.f;
        }
        for (int d = threadIdx.x; d < DP; d += blockDim.x) {
            const bool ok = d < Dobs;
            const float v = ok ? a.lik_var[d] : 1.f;
            sb[d] = (ok && a.bias) ? a.bias[d] : 0.f;
            siv[d] = ok ? 1.0f / v : 0.f;
            slv[d] = ok ? 1.8378770664093453f + logf(v) : 0.f;  // log(2 pi) + log var
        }
        double* acc = reinterpret_cast<double*>(base + shoot_smem_floats(D, Dobs) * 4);
        const int nwarps = (blockDim.x + 31) >> 5;
        for (int i = threadIdx.x; i < nwarps * (2 + Dobs); i += blockDim.x) acc[i] = 0.0;
        W = sW; bias = sb; iv = siv; lv = slv;
        wacc = acc + (threadIdx.x >> 5) * (2 + Dobs);
        const float scale = a.cons_scale[0];
        inv = 1.0f / scale;
        inv2 = inv * inv;
        c0 = a.laplace ? -logf(2.0f * scale) : -logf(scale) - 0.9189385332046727f;  // -log s - 0.5 log 2 pi
        __syncthreads();
    }
};

// One row's contribution. kLanes: the 32 lanes of the warp hold 32 different rows (warp-collective: every lane must
// call it; `valid` masks rows past the end) -- otherwise exactly one lane of the warp calls it.
// ll / cs: the calling thread's float64 running sums.
template <int D, bool kLanes>
__device__ __forceinline__ void shoot_epilogue(const ShootArgs& a, const ShootSmem<D>& sm, const bool valid,
                                               const int64_t row_local, const int64_t n_local, const float (&pred)[D],
                                               double& ll, double& cs) {
    const int Dobs = a.Dobs;
    const int64_t g = a.row_lo + (valid ? row_local : 0);
    const int64_t NT = (int64_t)a.N * a.T;
    const float* __restrict__ y = a.ys + (g % NT) * Dobs;
    const int t = (int)(g % a.T);
    const bool obs = valid && !(a.halo && t == a.T - 1);   // this row carries an observation
    float sl[D];
#pragma unroll
    for (int l = 0; l < D; ++l) sl[l] = 0.f;
    float lsum = 0.f;
    const int DP = shoot_dp(Dobs);
    // four observed dimensions per trip (one LDS.128 per operand); the four observations are fetched before anything
    // depends on them and the loop is unrolled twice, so eight global loads are in flight per lane (the first version
    // went dimension by dimension and spent its time waiting on one 4-byte load at a time: ncu, stall_long_sb)
#pragma unroll 2
    for (int d0 = 0; d0 < DP; d0 += 4) {
        float yv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) yv[u] = (obs && d0 + u < Dobs) ? __ldg(y + d0 + u) : 0.f;
        const float4 b4 = *reinterpret_cast<const float4*>(sm.bias + d0);
        const float4 i4 = *reinterpret_cast<const float4*>(sm.iv + d0);
        const float4 l4 = *reinterpret_cast<const float4*>(sm.lv + d0);
        float f[4] = {b4.x, b4.y, b4.z, b4.w};
        const float iv[4] = {i4.x, i4.y, i4.z, i4.w}, lv[4] = {l4.x, l4.y, l4.z, l4.w};
        float4 w4[D];
#pragma unroll
        for (int l = 0; l < D; ++l) {
            w4[l] = *reinterpret_cast<const float4*>(sm.W + l * DP + d0);
            f[0] = fmaf(pred[l], w4[l].x, f[0]);
            f[1] = fmaf(pred[l], w4[l].y, f[1]);
            f[2] = fmaf(pred[l], w4[l].z, f[2]);
            f[3] = fmaf(pred[l], w4[l].w, f[3]);
        }
        float q[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const float diff = obs ? f[u] - yv[u] : 0.f;   // a padded dimension has f = y = 0
            q[u] = diff * iv[u];
            lsum += -0.5f * (lv[u] + diff * q[u]);
            float gvd = obs ? -0.5f * (iv[u] - q[u] * q[u]) : 0.f;
            if constexpr (kLanes) {
                gvd = gpode_warp_sum(gvd);
                if ((threadIdx.x & 31) == 0 && d0 + u < Dobs) sm.wacc[2 + d0 + u] += (double)gvd;
            } else {
                if (d0 + u < Dobs) sm.wacc[2 + d0 + u] += (double)gvd;
            }
        }
#pragma unroll
        for (int l = 0; l < D; ++l)
            sl[l] = fmaf(-q[0], w4[l].x, fmaf(-q[1], w4[l].y, fmaf(-q[2], w4[l].z, fmaf(-q[3], w4[l].w, sl[l]))));
    }
    // shooting constraint: this row's end point against the NEXT sampled state of the same sequence
    float sc[D];
    float csum = 0.f;
    const bool has_next = valid && t < a.T - 1;
    const float* __restrict__ nxt = a.ss + (g + (has_next ? 1 : 0)) * D;
#pragma unroll
    for (int l = 0; l < D; ++l) {
        const float diff = has_next ? __ldg(nxt + l) - pred[l] : 0.f;
        if (a.laplace) {
            csum += has_next ? sm.c0 - fabsf(diff) * sm.inv : 0.f;
            sc[l] = diff > 0.f ? sm.inv : (diff < 0.f ? -sm.inv : 0.f);   // d lp / d pred
        } else {
            csum += has_next ? sm.c0 - 0.5f * diff * diff * sm.inv2 : 0.f;
            sc[l] = diff * sm.inv2;
        }
    }
    if (valid) {
        ll += obs ? (double)lsum : 0.0;
        cs += (double)csum;
        if (a.seeds != nullptr) {
#pragma unroll
            for (int l = 0; l < D; ++l) {
                a.seeds[row_local * D + l] = sl[l];
                a.seeds[(n_local + row_local) * D + l] = sc[l];
            }
        }
        if (a.pred_out != nullptr) {
#pragma unroll
            for (int l = 0; l < D; ++l) a.pred_out[row_local * D + l] = pred[l];
        }
    }
}

// end of the kernel: thread sums -> warp slots -> this CTA's row of `work` (all in float64, fixed order)
template <int D>
__device__ __forceinline__ void shoot_finish(const ShootArgs& a, const ShootSmem<D>& sm, double ll, double cs) {
    const int lane = threadIdx.x & 31, nwarps = (blockDim.x + 31) >> 5, Dobs = a.Dobs;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ll += __shfl_xor_sync(0xffffffffu, ll, o);
        cs += __shfl_xor_sync(0xffffffffu, cs, o);
    }
    if (lane == 0) {
        sm.wacc[0] = ll;
        sm.wacc[1] = cs;
    }
    __syncthreads();
    const double* acc0 = sm.wacc - (threadIdx.x >> 5) * (2 + Dobs);
    double* __restrict__ row = a.work + (size_t)blockIdx.x * (2 + Dobs);
    for (int i = threadIdx.x; i < 2 + Dobs; i += blockDim.x) {
        double s = 0.0;
        for (int w = 0; w < nwarps; ++w) s += acc0[w * (2 + Dobs) + i];
        row[i] = s;
    }
}
#endif  // __CUDACC__
