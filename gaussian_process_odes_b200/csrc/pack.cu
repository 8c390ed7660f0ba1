// Error plumbing, ABI version, and the cache repacking kernel.
#include "common.cuh"
#include <string.h>
#include <cuda_fp16.h>

static thread_local char g_err[512] = "";

void gpode_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char* gpode_last_error(void) { return g_err; }
extern "C" int gpode_abi_version(void) { return GPODE_B200_ABI_VERSION; }

extern "C" int64_t gpode_packed_floats(int D, int M, int S) {
    if (D < 1 || M < 1 || S < 1) return -1;
    return gpode_layout(D, M, S).n_packed;
}

namespace {

// One thread per packed record. Source layouts are the reference's cache tensors (src/core/dsvgp.py:100-103,122):
// omega (j,s,k), phase (s,k), w (s,k), Z (m,j), nu (k,m), ell (k,j), var (k).
// blockIdx.y = parameter set (batched Monte-Carlo prediction): omega / phase / w / nu carry a leading set dimension,
// Z / ell / var are shared; the packed blocks follow each other at stride L.n_packed.
__global__ void pack_kernel(const GpodeLayout L, const float* __restrict__ omega, const float* __restrict__ phase,
                            const float* __restrict__ w, const float* __restrict__ Z, const float* __restrict__ nu,
                            const float* __restrict__ ell, const float* __restrict__ var, float* __restrict__ out) {
    const int D = L.D, M = L.M, S = L.S, S2 = L.S2;
    {
        const size_t set = blockIdx.y;
        omega += set * D * S * D;
        phase += set * S * D;
        w += set * S * D;
        if (nu) nu += set * D * M;
        out += set * L.n_packed;
    }
    const int n_rff = D * S2, n_kern = M, n_il = D;
    const int n_mmah = D <= GPODE_MMAH_MAX_D ? D * L.S8P * 32 : 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_rff + n_kern + n_il + n_mmah;
         i += gridDim.x * blockDim.x) {
        if (i >= n_rff + n_kern + n_il) {
            // f16 tensor-core operands of the adjoint (see GpodeLayout::mmah) for one lane of one (k, feature tile)
            const int q = i - (n_rff + n_kern + n_il);
            const int lane = q & 31, rec = q >> 5;          // rec = k * S8P + ft
            const int k = rec / L.S8P, ft = rec - k * L.S8P;
            const int g = lane >> 2, t = lane & 3;
            uint32_t* o = reinterpret_cast<uint32_t*>(out + L.off_mmah + (size_t)rec * GPODE_MMAH_REC);
            auto om = [&](int j, int sidx) -> float {
                return (j < D && sidx < S) ? omega[((size_t)j * S + sidx) * D + k] : 0.f;
            };
            auto split = [](float v, __half& hi, __half& lo) {
                hi = __float2half_rn(v);
                lo = __float2half_rn(v - __half2float(hi));
            };
            auto pack2 = [](__half a, __half b) -> uint32_t {
                return (uint32_t)__half_as_ushort(a) | ((uint32_t)__half_as_ushort(b) << 16);
            };
            auto slotB = [&](int slot, int sidx) -> __half {  // theta-B[slot][feature]
                __half hi = __float2half_rn(0.f), lo = hi;
                if (slot < 3 * D) split(om(slot % D, sidx), hi, lo);
                return (slot >= D && slot < 2 * D) ? lo : hi;
            };
            const int sg = 8 * ft + g;
            o[lane * 2 + 0] = pack2(slotB(2 * t, sg), slotB(2 * t + 1, sg));
            o[lane * 2 + 1] = pack2(slotB(2 * t + 8, sg), slotB(2 * t + 9, sg));
            const float ak = sqrtf(var[k] / (float)S) * GPODE_MMAH_SCALE;
            __half bh[2], bl[2];
            for (int h = 0; h < 2; ++h) {
                const int sidx = 8 * ft + 2 * t + h;
                const float a = sidx < S ? w[sidx * D + k] * ak : 0.f;
                split(a * om(g, sidx), bh[h], bl[h]);
                if (g == 0) {
                    const float ph = sidx < S ? phase[sidx * D + k] : 0.f;
                    reinterpret_cast<float*>(o)[64 + t * 4 + h] = ph;
                    reinterpret_cast<float*>(o)[64 + t * 4 + 2 + h] = ph;
                    reinterpret_cast<float*>(o)[144 + t * 2 + h] = a / GPODE_MMAH_SCALE;
                }
            }
            // G-B operands of a tile PAIR (2i, 2i+1) sit together so that each MMA's (b0, b1) comes out of one LDS.64:
            // even record [80,144): lane-major (hi of tile 2i, hi of tile 2i+1); odd record [80,144): (lo, lo)
            uint32_t* even = (ft & 1) ? o - GPODE_MMAH_REC : o;
            uint32_t* odd = even + GPODE_MMAH_REC;
            even[80 + lane * 2 + (ft & 1)] = pack2(bh[0], bh[1]);
            odd[80 + lane * 2 + (ft & 1)] = pack2(bl[0], bl[1]);
        } else if (i < n_rff) {
            const int k = i / S2, s2 = i - k * S2;
            // element e of the record lives at chunk e/4, slot e%4 of the chunk-major group layout
            float* base = out + L.off_rff + ((size_t)k * L.S2P + (s2 & ~31)) * L.RP + (s2 & 31) * 4;
#define GPODE_REC(e) base[((e) >> 2) * 128 + ((e) & 3)]
            for (int h = 0; h < 2; ++h) {
                const int s = 2 * s2 + h;
                const bool ok = s < S;
                for (int j = 0; j < D; ++j) GPODE_REC(2 * j + h) = ok ? omega[((size_t)j * S + s) * D + k] : 0.f;
                GPODE_REC(2 * D + h) = ok ? phase[s * D + k] : 0.f;
                GPODE_REC(2 * D + 2 + h) = ok ? w[s * D + k] * sqrtf(var[k] / (float)S) : 0.f;
            }
            for (int j = 2 * D + 4; j < L.RP; ++j) GPODE_REC(j) = 0.f;
#undef GPODE_REC
        } else if (i < n_rff + n_kern) {
            const int m = i - n_rff;
            float* o = out + L.off_kern + (size_t)m * L.KS;
            for (int j = 0; j < D; ++j) o[j] = Z[m * D + j];
            for (int k = 0; k < L.KS - D; ++k) o[D + k] = (nu && k < D) ? var[k] * nu[k * M + m] : 0.f;
        } else {
            const int j = i - n_rff - n_kern;
            float* o = out + L.off_il + (size_t)j * L.WP;
            for (int k = 0; k < L.WP; ++k)
                o[k] = k < D ? -GPODE_HALF_LOG2E / (ell[k * D + j] * ell[k * D + j]) : 0.f;
        }
    }
}

}  // namespace

static int pack_sets(const gpode_cache_t* c, int n_sets, float* packed, void* stream) {
    GPODE_CHECK_ARG(c != nullptr && packed != nullptr, "cache / packed is NULL");
    GPODE_CHECK_ARG(n_sets >= 1 && n_sets <= 65535, "n_sets=%d outside 1..65535", n_sets);
    GPODE_CHECK_ARG(c->D >= 1 && c->D <= GPODE_MAX_D, "state dimension D=%d outside 1..%d", c->D, GPODE_MAX_D);
    GPODE_CHECK_ARG(c->M >= 1 && c->S >= 1, "M=%d and S=%d must be positive", c->M, c->S);
    GPODE_CHECK_ARG(c->omega && c->phase && c->w && c->Z && c->ell && c->var, "cache tensor is NULL");
    const GpodeLayout L = gpode_layout(c->D, c->M, c->S);
    const int n = c->D * L.S2 + c->M + c->D + (c->D <= GPODE_MMAH_MAX_D ? c->D * L.S8P * 32 : 0);
    pack_kernel<<<dim3((n + 127) / 128, n_sets), 128, 0, (cudaStream_t)stream>>>(L, c->omega, c->phase, c->w, c->Z,
                                                                                 c->nu, c->ell, c->var, packed);
    GPODE_LAUNCH_CHECK();
    return 0;
}

extern "C" int gpode_pack_cache(const gpode_cache_t* c, float* packed, void* stream) {
    return pack_sets(c, 1, packed, stream);
}

extern "C" int gpode_pack_cache_sets(const gpode_cache_t* c, int n_sets, float* packed, void* stream) {
    return pack_sets(c, n_sets, packed, stream);
}

// ---- process-wide kernel-selection options (see common.cuh) ---------------------------------------------------------
#include <atomic>
#include <mutex>
#include <stdlib.h>
#include <string.h>
namespace {
std::atomic<int> g_opt[GPODE_OPT_COUNT];
std::once_flag g_opt_once;
const char* const kOptNames[GPODE_OPT_COUNT] = {"bwd_mma", "fwd_mma"};
void opt_init() {
    auto env_int = [](const char* n, int dflt) {
        const char* e = getenv(n);
        return e ? atoi(e) : dflt;
    };
    g_opt[GPODE_OPT_BWD_MMA] = env_int("GPODE_BWD_MMA", 1);
    g_opt[GPODE_OPT_FWD_MMA] = env_int("GPODE_FWD_MMA", 1);
}
}  // namespace
int gpode_option(int which) {
    std::call_once(g_opt_once, opt_init);
    return g_opt[which].load(std::memory_order_relaxed);
}
extern "C" int gpode_set_option(const char* name, int value) {
    std::call_once(g_opt_once, opt_init);
    GPODE_CHECK_ARG(name != nullptr, "option name is NULL");
    for (int i = 0; i < GPODE_OPT_COUNT; ++i)
        if (strcmp(name, kOptNames[i]) == 0) {
            g_opt[i].store(value, std::memory_order_relaxed);
            return 0;
        }
    gpode_set_error("unknown option %s (bwd_mma, fwd_mma)", name);
    return -1;
}
extern "C" int gpode_get_option(const char* name) {
    if (name == nullptr) return -1;
    for (int i = 0; i < GPODE_OPT_COUNT; ++i)
        if (strcmp(name, kOptNames[i]) == 0) return gpode_option(i);
    return -1;
}
