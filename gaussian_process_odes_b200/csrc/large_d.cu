// RBF term of the vector field for 8 < D <= 64 on the FP32 CUDA cores, added to a Fourier-feature term computed by the
// tensor-core kernel (gpode_rff_fwd_large, large_umma.cu): f = f_rff + sum_m var_k nu_km exp(-0.5 r_km^2). This is the
// fallback of gpode_rbf_fwd_large when the inducing points do not fit its shared-memory copy of Z. Mapping:
//   * a CTA owns a tile of TR = 32 rows whose state lives in shared memory;
//   * thread = (output dim k, group of 8 rows): for every inducing point it reads Z through the read-only cache against
//     the tile's x in shared memory, every value reused for 8 rows from registers.
// Arithmetic replaced: the RBF half of DSVGP_Layer.forward (reference src/core/dsvgp.py:172-197). Takes the RAW cache
// tensors (no repacking needed).
#include "common.cuh"

namespace {

constexpr int kTR = 32;   // rows per CTA tile
constexpr int kRG = 8;    // rows per thread (register block)
constexpr int kNG = kTR / kRG;

struct LdArgs {
    int D, M;
    const float* Z;      // [M,D]
    const float* nu;     // [D,M]
    const float* ell;    // [D,D] (k,j)
    const float* var;    // [D]
};

// f[r][k] = frff[r][k] + RBF term for the tile; xs, fs: shared, TRANSPOSED [D][kTR] (a thread's 8 rows are two
// LDS.128); thread (k = tid % D, g = tid / D) handles rows g*8 .. g*8+7
__device__ void eval_tile(const LdArgs& a, const float* __restrict__ xs, float* __restrict__ fs, const float* wl,
                          const int k, const int g, const bool active, const float* __restrict__ frff,
                          const int64_t row0, const int64_t B) {
    const int D = a.D, M = a.M;
    if (active) {
        float acc[kRG];
#pragma unroll
        for (int r = 0; r < kRG; ++r) {
            const int64_t row = row0 + g * kRG + r;
            acc[r] = row < B ? __ldg(frff + row * D + k) : 0.f;
        }
        const float vk = __ldg(a.var + k);
        for (int m = 0; m < M; ++m) {
            float e[kRG];
#pragma unroll
            for (int r = 0; r < kRG; ++r) e[r] = 0.f;
            for (int j = 0; j < D; ++j) {
                const float z = __ldg(a.Z + m * D + j);
                const float wkj = wl[k * D + j];
                const float4 xa = *reinterpret_cast<const float4*>(xs + j * kTR + g * kRG);
                const float4 xb = *reinterpret_cast<const float4*>(xs + j * kTR + g * kRG + 4);
                const float xr[kRG] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
#pragma unroll
                for (int r = 0; r < kRG; ++r) {
                    const float d = xr[r] - z;
                    e[r] = fmaf(d * d, wkj, e[r]);
                }
            }
            const float c = vk * __ldg(a.nu + k * M + m);
#pragma unroll
            for (int r = 0; r < kRG; ++r) acc[r] = fmaf(c, gpode_ex2(-e[r]), acc[r]);
        }
#pragma unroll
        for (int r = 0; r < kRG; ++r) fs[k * kTR + g * kRG + r] = acc[r];
    }
    __syncthreads();
}

// smem: wl[D*D] | y[kTR*D] | f[kTR*D]. Draw q (GpodeDraws, common.cuh) owns ceil(rows / kTR) tiles and reads nu of draw q.
__global__ void large_d_rbf_kernel(LdArgs a, const float* __restrict__ x, const GpodeDraws dr,
                                   const float* __restrict__ frff, float* __restrict__ out) {
    extern __shared__ __align__(16) float sm[];
    const int D = a.D;
    float* wl = sm;
    float* y = wl + ((D * D + 3) & ~3);  // keep the tiles 16-byte aligned for the float4 reads
    float* fs = y + kTR * D;
    for (int i = threadIdx.x; i < D * D; i += blockDim.x) {
        const float l = __ldg(a.ell + i);
        wl[i] = GPODE_HALF_LOG2E / (l * l);
    }
    const int k = threadIdx.x % D, g = threadIdx.x / D;
    const bool active = g < kNG;
    const float* nu0 = a.nu;
    const int64_t tpd = (dr.rows + kTR - 1) / kTR;
    const int64_t ntiles = tpd * dr.n;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t q = tile / tpd;
        if (dr.done != nullptr && dr.done[q * dr.done_stride] != 0) continue;
        // rows of the tile past the draw's last row are out of range, as rows past B are for one draw
        const int64_t base = q * dr.rows, row0 = base + (tile - q * tpd) * kTR, B = base + dr.rows;
        a.nu = nu0 + q * D * a.M;
        __syncthreads();
        for (int i = threadIdx.x; i < kTR * D; i += blockDim.x) {
            const int r = i / D, j = i - r * D;
            y[j * kTR + r] = row0 + r < B ? __ldg(x + row0 * D + i) : 0.f;
        }
        __syncthreads();
        eval_tile(a, y, fs, wl, k, g, active, frff, row0, B);
        for (int i = threadIdx.x; i < kTR * D; i += blockDim.x) {
            const int r = i / D, j = i - r * D;
            if (row0 + r < B) out[row0 * D + i] = fs[j * kTR + r];
        }
    }
}

}  // namespace

int gpode_vf_large_add_rbf_draws(const gpode_cache_t* c, const float* x, const float* f_rff, float* f,
                                 const GpodeDraws& dr, cudaStream_t st) {
    const LdArgs a{c->D, c->M, c->Z, c->nu, c->ell, c->var};
    const int D = c->D;
    const int threads = ((kNG * D + 31) / 32) * 32;  // D=16 -> 64, D=32 -> 128, D=64 -> 256
    const size_t smem = sizeof(float) * ((size_t)((D * D + 3) & ~3) + 2 * (size_t)kTR * D);
    GPODE_CUDA(cudaFuncSetAttribute(large_d_rbf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0, sms = 148, dev = 0;
    GPODE_CUDA(cudaGetDevice(&dev));
    GPODE_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    GPODE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, large_d_rbf_kernel, threads, smem));
    if (occ < 1) {
        gpode_set_error("large-D kernel does not fit on an SM (smem %zu bytes)", smem);
        return -2;
    }
    const int64_t ntiles = (dr.rows + kTR - 1) / kTR * dr.n;
    const int64_t cap = (int64_t)sms * occ;
    large_d_rbf_kernel<<<(unsigned)(ntiles < cap ? ntiles : cap), threads, smem, st>>>(a, x, dr, f_rff, f);
    GPODE_LAUNCH_CHECK();
    return 0;
}

extern "C" int gpode_vf_fwd_large_add_rbf(const gpode_cache_t* c, const float* x, const float* f_rff, float* f,
                                          int64_t B, void* stream) {
    GPODE_CHECK_ARG(c != nullptr, "cache is NULL");
    GPODE_CHECK_ARG(c->D > GPODE_MAX_D && c->D <= GPODE_MAX_D_LARGE, "large-D path needs %d < D <= %d, got %d",
                    GPODE_MAX_D, GPODE_MAX_D_LARGE, c->D);
    GPODE_CHECK_ARG(c->M >= 1 && c->S >= 1 && B >= 0, "bad sizes");
    GPODE_CHECK_ARG(c->Z && c->nu && c->ell && c->var, "cache tensor is NULL");
    GPODE_CHECK_ARG(f_rff != nullptr, "f_rff is NULL");
    if (B == 0) return 0;
    GPODE_CHECK_ARG(x && f, "NULL argument");
    return gpode_vf_large_add_rbf_draws(c, x, f_rff, f, gpode_one_draw(B), (cudaStream_t)stream);
}
