/*
 * gpode_b200 -- C ABI of the B200-native (sm_100a) GPODE hot path.
 *
 * The reference (hegdepashupati/gaussian-process-odes) is pure Python/PyTorch and has no FFI layer; the seams this
 * library replaces are Python call signatures. Each entry point below cites the reference code whose arithmetic it
 * replaces (paths relative to the reference repo root). INTEGRATION.md shows the ctypes binding a maintainer of the
 * reference would add.
 *
 * Conventions (SURVEY.md section 8b)
 *   - every pointer is a DEVICE pointer to float32 (row-major, contiguous) unless it is named *_f64 or says "host";
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*) and never synchronises the host;
 *   - return value: 0 = ok, <0 = argument/shape error, >0 = cudaError_t; gpode_last_error() gives the text;
 *   - no global mutable state except the per-thread last-error string; float32 arithmetic on the path
 *     (the Kzz factorisation accumulates in float64 in shared memory).
 *
 * Symbols: D = state dim (D_in == D_out), M = inducing points, S = Fourier features, B = rows of the integrated
 * batch, Tg = length of the time grid.
 */
#ifndef GPODE_B200_H
#define GPODE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPODE_B200_ABI_VERSION 2
#define GPODE_MAX_D 8          /* register-resident state kernels are instantiated for 1 <= D <= 8 */
#define GPODE_MAX_D_LARGE 64   /* the large-D kernels (tcgen05 forward, large-D VJP) cover 8 < D <= 64 */
#define GPODE_MAX_M_F64 112    /* whitening backward keeps two MxM float64 tiles in shared memory */
#define GPODE_MAX_M 160        /* ... and falls back to float32 tiles up to this M */
#define GPODE_MAX_M_BLOCKED 2048  /* blocked float64 whitening (matrices in global memory) for D <= GPODE_MAX_D */

/* One sampled GP function = the reference's "cache" (DSVGP_Layer.build_cache, src/core/dsvgp.py:92-122) plus the
 * kernel hyper-parameters it closes over (RBF, src/core/kernels.py:33-51). */
typedef struct gpode_cache {
    int32_t D, M, S;
    const float* omega;   /* [D,S,D]  rff_omega = eps/lengthscale, index (j,s,k)        dsvgp.py:101, kernels.py:101-112 */
    const float* phase;   /* [S,D]    rff_phase in radians                              dsvgp.py:102-103 */
    const float* w;       /* [S,D]    rff_weights                                       dsvgp.py:100 */
    const float* Z;       /* [M,D]    inducing locations                                dsvgp.py:66 */
    const float* nu;      /* [D,M]    nu = Kzz^-1 (u - f_prior(Z))                      dsvgp.py:119-122 */
    const float* ell;     /* [D,D]    lengthscales (k = output dim, j = input dim)      kernels.py:45-47 */
    const float* var;     /* [D]      signal variances                                  kernels.py:49-51 */
} gpode_cache_t;

int         gpode_abi_version(void);
const char* gpode_last_error(void);

/* Number of floats of the packed, kernel-friendly parameter block for (D,M,S). */
int64_t gpode_packed_floats(int D, int M, int S);

/* Repack one cache into the layout the integrator kernels stage into shared memory with one bulk (TMA) copy:
 * per (k,s) [Omega_0sk..Omega_{D-1}sk, phase_sk, w_sk*sqrt(var_k/S)], per m [Z_m, var_k*nu_km], scaled inverse
 * lengthscales. Replaces the per-call tensor prep of DSVGP_Layer.forward (src/core/dsvgp.py:172-197). */
int gpode_pack_cache(const gpode_cache_t* cache, float* packed, void* stream);

/* f = vector field at x. Replaces DSVGP_Layer.forward(t, x) (src/core/dsvgp.py:172-197 = rff_forward :124-137 +
 * RBF.K src/core/kernels.py:87-99 + einsum :192).  x, f: [B,D]. */
int gpode_vf_fwd(const float* packed, int D, int M, int S, const float* x, float* f, int64_t B, void* stream);

/* Vector-Jacobian product of the above (what autograd does through dsvgp.py:172-197), row part:
 *   grad_x [B,D]; every CTA writes its lengthscale / variance partial sums to a row of its own in `acc` (see
 *   gpode_acc_floats below); f [B,D] is the forward output (saved by the caller). Follow with gpode_param_grad(x, grad_f, B) for the
 *   per-inducing-point part and gpode_grads_finalize. */
int gpode_vf_bwd(const float* packed, int D, int M, int S, const float* x, const float* f, const float* grad_f,
                 float* grad_x, float* acc, int64_t B, void* stream);

/* Fixed-grid RK4 (3/8 rule) over the user's grid t[Tg] (float32, device), i.e. torchdiffeq 0.2.0
 * odeint(func, y0, t, method='rk4') as called by Flow.forward (src/core/flow.py:84-90) with func = ODEfunc
 * (flow.py:29-37). xs: [Tg,B,D] with xs[0] = x0 (torchdiffeq's own layout; Flow permutes it to [B,Tg,D]).
 * kstages: NULL, or [Tg-1,4,B,D] receiving the four stage derivatives of every step (the backward's checkpoints). */
int gpode_rk4_fwd(const float* packed, int D, int M, int S, const float* x0, const float* t, int Tg, int64_t B,
                  float* xs, float* kstages, void* stream);

/* Discrete adjoint of gpode_rk4_fwd == autograd through the unrolled solver (use_adjoint=False, the reference
 * default, train_vdp_gpode.py:52). grad_xs [Tg,B,D] -> grad_x0 [B,D]; lengthscale / variance partial sums go to this
 * call's rows of `acc`. vrows (gpode_vrow_floats(D, (Tg-1)*4*B) floats) receives, for every step and stage, the stage input
 * and its cotangent: rows [0, n) hold the stage inputs, rows [n, 2n) the cotangents, n = (Tg-1)*4*B. Follow with
 * gpode_param_grad(vrows, vrows + n*D, n) and gpode_grads_finalize. */
int gpode_rk4_bwd(const float* packed, int D, int M, int S, const float* t, int Tg, int64_t B, const float* xs,
                  const float* kstages, const float* grad_xs, float* grad_x0, float* vrows, float* acc,
                  void* stream);

/* Per-inducing-point gradient contraction over n_rows (point y, cotangent kb) pairs: partial sums
 * T[k,m] = sum kb_k K_km(y) and W[k,m,j] = sum kb_k K_km(y) (y_j - Z_mj), one row of `acc` per CTA (autograd through
 * src/core/kernels.py:53-99 and the einsum of src/core/dsvgp.py:192 w.r.t. nu and Z).  ys, kbs: [n_rows,D]. */
int gpode_param_grad(const float* packed, int D, int M, int S, const float* ys, const float* kbs, int64_t n_rows,
                     float* acc, void* stream);

/* Accumulator block shared by the *_bwd entry points and its conversion to parameter gradients.
 * Shared-parameter gradients contract over every row of the batch. To make them BITWISE REPRODUCIBLE the library uses
 * no floating-point atomics: each CTA of a *_bwd / param_grad kernel writes its partial sums to a row of its own
 * and gpode_grads_finalize adds the rows up in row order in float64 (and contracts with nu / var / ell in float64).
 *   acc layout (floats): header[gpode_acc_header_floats() = 4: int32 row counts, ZEROED BY THE CALLER before the
 *   first *_bwd call] | rows of A[D,D] | V[D] (one per adjoint CTA) | rows of {T[k], W[j,k]} per inducing point
 *   (one per param_grad CTA). One acc block serves ONE backward pass (one *_bwd call + one gpode_param_grad call).
 *   gpode_grads_finalize: grad_ell[D,D], grad_var[D], grad_Z[M,D], grad_nu[D,M] (overwritten). grad_ell already
 *   contains the path through omega = eps/ell (kernels.py:110-112). */
int64_t gpode_acc_header_floats(void);
int64_t gpode_acc_floats(int D, int M);
int64_t gpode_vrow_floats(int D, int64_t n_virtual_rows);
int gpode_grads_finalize(const gpode_cache_t* cache, const float* acc, float* grad_ell, float* grad_var,
                         float* grad_Z, float* grad_nu, void* stream);

/* Kzz whitening of build_cache (src/core/dsvgp.py:110-122): L = chol(K(Z,Z) + jitter I), nu = L^-T (u - L^-1 p),
 * p = rff_forward(Z) (dsvgp.py:112,124-137), batched over the D output dimensions (one CTA each, matrices in shared
 * memory).  u: [M,D]; nu_out: [D,M]; L_f64: [D,M,M] float64 and s_f64: [D,M] float64 are saved for the backward. */
int gpode_whiten_fwd(const gpode_cache_t* cache_without_nu, const float* u, float jitter, float* nu_out,
                     double* L_f64, double* s_f64, void* stream);
/* Backward of the above: grad_nu [D,M] -> grad_u [M,D], grad_Z [M,D], grad_ell [D,D], grad_var [D] (overwritten). */
int gpode_whiten_bwd(const gpode_cache_t* cache_with_nu, const float* u, const double* L_f64, const double* s_f64,
                     const float* grad_nu, float* grad_u, float* grad_Z, float* grad_ell, float* grad_var,
                     void* stream);
/* The same three operations (gpode_whiten_fwd, gpode_whiten_fwd_sets below, gpode_whiten_bwd) for 1 <= M <=
 * GPODE_MAX_M_BLOCKED at D <= GPODE_MAX_D, blocked: the M x M matrices live in global memory (L_f64 and the caller-owned
 * float64 workspace `work`), Cholesky in panels of 64 columns, blocked triangular solves, FP64 throughout. Arguments and
 * outputs mean what they mean for the tile kernels; the backward is bitwise reproducible and a draw of the sets form
 * gets bitwise the nu of the single-draw call. The launch sequence depends on (D, M, n_sets) only -- no host read, no
 * allocation -- so the calls can be captured in a CUDA graph. The library selects nothing itself: callers use these
 * above GPODE_MAX_M (ops.whiten / ops.whiten_sets do).
 *   gpode_whiten_blocked_work_doubles: float64 elements of `work` for the forward with n_sets >= 1 draws (D M n_sets),
 *     or, for n_sets = 0, for the backward (D M (M + D + 2) + D ceil(M/64) (D+1)); -1 for arguments out of range.
 *     Pure host arithmetic. */
int64_t gpode_whiten_blocked_work_doubles(int D, int M, int n_sets);
int gpode_whiten_fwd_blocked(const gpode_cache_t* cache_without_nu, const float* u, float jitter, float* nu_out,
                             double* L_f64, double* s_f64, double* work, void* stream);
int gpode_whiten_fwd_sets_blocked(const gpode_cache_t* cache_sets_without_nu, const float* u, float jitter, int n_sets,
                                  float* nu_out, double* L_f64, double* s_f64, double* work, void* stream);
int gpode_whiten_bwd_blocked(const gpode_cache_t* cache_with_nu, const float* u, const double* L_f64,
                             const double* s_f64, const float* grad_nu, float* grad_u, float* grad_Z, float* grad_ell,
                             float* grad_var, double* work, void* stream);

/* Whitened KL of DSVGP_Layer.kl (src/core/dsvgp.py:199-230), q_diag=False:
 *   kl = 0.5 * sum_k [ |Um_k|^2 + |tril(Ls_k)|_F^2 - sum_i log Ls_k,ii^2 - M ],  Ls given PACKED as the optvar of
 *   transforms.LowerTriangular (src/misc/transforms.py:70-76): [D, M(M+1)/2], row-major np.tril_indices order. */
int gpode_kl_fwd(const float* Um, const float* Ls_packed, int D, int M, float* kl_out, void* stream);
int gpode_kl_bwd(const float* Um, const float* Ls_packed, int D, int M, const float* grad_kl, float* grad_Um,
                 float* grad_Ls_packed, void* stream);
/* Inducing sample in whitened coordinates, u = Um + Us_sqrt eps (DSVGP_Layer.sample_inducing, src/core/dsvgp.py:78-90,
 * full-rank branch `einsum('dnm,md->nd', Us_sqrt, eps)`), straight from the packed lower-triangular factor Ls_packed
 * [D, M(M+1)/2] (row-major tril packing): u_out [M,D]. Backward: grad_Ls_packed = grad_u eps^T restricted to the lower
 * triangle (grad_Um = grad_u). */
int gpode_inducing_sample_fwd(const float* Um, const float* Ls_packed, const float* eps, int D, int M, float* u_out,
                              void* stream);
int gpode_inducing_sample_bwd(const float* eps, const float* grad_u, int D, int M, float* grad_Ls_packed, void* stream);

/* Adaptive Dormand-Prince 5(4) with torchdiffeq 0.2.0's controller (rtol/atol, whole-batch RMS norm, float64 time,
 * 4th-order dense output) -- odeint(..., method='dopri5'), the reference's default solver (src/core/flow.py:41).
 * Runs as ONE cooperative persistent kernel: accept/reject is decided on the device, one grid barrier per attempt.
 * t: the Tg output times, DEVICE float64, strictly monotone in either direction (a decreasing grid is integrated as
 * -f over -t, which is what torchdiffeq does). work: gpode_dopri5_work_floats(D,B) floats.
 * stats_out (device, 4 int32): nfe, accepted steps, rejected steps, status (0 ok, 1 attempt limit, 2 dt underflow,
 * 3 checkpoint capacity). */
int64_t gpode_dopri5_work_floats(int D, int64_t B);
/* ckpt / cap: NULL / 0 for inference. For training pass gpode_dopri5_ckpt_floats(D,B,Tg,cap) floats: the kernel
 * records, for every ACCEPTED step, the state at its start, its seven stage derivatives and its step size, and for
 * every output the step and abscissa it was interpolated at. status 3 = more than `cap` accepted steps (retry). */
int64_t gpode_dopri5_ckpt_floats(int D, int64_t B, int Tg, int cap);
int gpode_dopri5_fwd(const float* packed, int D, int M, int S, const float* x0, const double* t, int Tg, int64_t B,
                     double rtol, double atol, float* xs, float* work, int32_t* stats_out, float* ckpt, int cap,
                     void* stream);
/* Discrete adjoint through the accepted steps and the dense-output interpolation (step sizes are constants, as in
 * torchdiffeq where the controller runs under no_grad): grad_xs [Tg,B,D] -> grad_x0 [B,D]; lengthscale / variance
 * partial sums accumulate into `acc`; vrows = gpode_vrow_floats(D, (6 n_accepted + 1) B) floats in the layout of
 * gpode_rk4_bwd. Follow with gpode_param_grad over n = (6 n_accepted + 1) B rows and gpode_grads_finalize. */
int gpode_dopri5_bwd(const float* packed, int D, int M, int S, const double* t, int Tg, int64_t B,
                     const float* grad_xs, const float* ckpt, int cap, int n_accepted, float* grad_x0, float* vrows,
                     float* acc, void* stream);

/* The same two steps with the accepted-step count left ON THE DEVICE (stats_dev = the forward's stats_out), so that
 * nothing between forward and backward needs the host and the whole dopri5 training step can be captured in a CUDA
 * graph. vrows must hold the capacity, gpode_vrow_floats(D, (6 cap + 1) B) floats; the cotangent rows start at row
 * (6 cap + 1) B. gpode_param_grad_dev contracts the first (6 stats_dev[1] + 1) * rows_per_step of n_rows_max rows. */
int gpode_dopri5_bwd_dev(const float* packed, int D, int M, int S, const double* t, int Tg, int64_t B,
                         const float* grad_xs, const float* ckpt, int cap, const int32_t* stats_dev, float* grad_x0,
                         float* vrows, float* acc, void* stream);
int gpode_param_grad_dev(const float* packed, int D, int M, int S, const float* ys, const float* kbs,
                         int64_t n_rows_max, const int32_t* stats_dev, int64_t rows_per_step, float* acc,
                         void* stream);

/* Vector field for 8 < D <= GPODE_MAX_D_LARGE (the upper half of the scaling sweep): the Fourier-feature term as
 * tcgen05 kind::tf32 GEMMs (3xTF32, TMEM accumulators) over operand chunks pre-tiled by gpode_pack_cache_large
 * (gpode_packed_large_floats(D,M,S) floats) and streamed from L2 through a shared-memory ring;
 * gpode_vf_fwd_large_add_rbf adds the RBF term on the FP32 CUDA cores (state tiles in shared memory, RAW cache):
 * f = f_rff + K(x,Z) nu. */
int64_t gpode_packed_large_floats(int D, int M, int S);
int gpode_pack_cache_large(const gpode_cache_t* cache, float* packed_large, void* stream);
int gpode_rff_fwd_large(const float* packed_large, int D, int S, const float* x, float* f_rff, int64_t B, void* stream);
int gpode_vf_fwd_large_add_rbf(const gpode_cache_t* cache, const float* x, const float* f_rff, float* f, int64_t B,
                               void* stream);
/* ... and the RBF term on the tensor cores as well: per inducing point one [128 rows x D] x [D x D] GEMM of the
 * squared differences (built on the fly) against -W^T; f = f_rff + sum_m c_km 2^(...). Z: the raw [M,D] tensor. */
int gpode_rbf_fwd_large(const float* packed_large, int D, int M, int S, const float* Z, const float* x,
                        const float* f_rff, float* f, int64_t B, void* stream);

/* ---- Batched Monte-Carlo prediction: n_sets function draws in one launch (SURVEY.md section 8b item 1 "n_sets",
 * 8f item 3). Replaces the Python loop of compute_predictions / compute_test_predictions
 * (src/gpode/model_builder.py:60-96, src/gpode_shooting/mocap_model_builder.py:85-119), which rebuilds the cache
 * and integrates once per sample. A "sets" cache carries a leading n_sets dimension on the per-draw tensors
 * (omega [n,D,S,D], phase [n,S,D], w [n,S,D], nu [n,D,M]); Z, ell, var are shared. Set q owns rows
 * [q set_rows, (q+1) set_rows) of x / x0 / xs ([n_sets*set_rows, D] resp. [Tg, n_sets*set_rows, D]) and the packed
 * block at packed + q * gpode_packed_floats(D,M,S). Forward only (prediction runs under no_grad). */
int gpode_pack_cache_sets(const gpode_cache_t* cache_sets, int n_sets, float* packed, void* stream);
/* u [n_sets,M,D] -> nu_out [n_sets,D,M]: Kzz is factorised ONCE (it does not depend on the draw), then one CTA per
 * (output dim, set) does the two triangular solves. L_f64 [D,M,M], s_f64 [D,2,M]: float64 scratch. */
int gpode_whiten_fwd_sets(const gpode_cache_t* cache_sets_without_nu, const float* u, float jitter, int n_sets,
                          float* nu_out, double* L_f64, double* s_f64, void* stream);
int gpode_vf_fwd_sets(const float* packed, int D, int M, int S, int n_sets, int64_t set_rows, const float* x,
                      float* f, void* stream);
int gpode_rk4_fwd_sets(const float* packed, int D, int M, int S, int n_sets, int64_t set_rows, const float* x0,
                       const float* t, int Tg, float* xs, void* stream);
/* dopri5 with one controller PER SET (error norm over that set's rows: exactly the reference loop, which calls
 * odeint once per sample): one CTA per set, no grid barrier. work: gpode_dopri5_work_floats(D, n_sets*set_rows);
 * stats_out: 4 int32 per set. */
int gpode_dopri5_fwd_sets(const float* packed, int D, int M, int S, int n_sets, int64_t set_rows, const float* x0,
                          const double* t, int Tg, double rtol, double atol, float* xs, float* work,
                          int32_t* stats_out, void* stream);
/* The same for 8 < D <= GPODE_MAX_D_LARGE, on the large-D kernels with a draw index (forward only):
 *   gpode_pack_cache_large_sets: n_sets blocks of gpode_packed_large_floats(D,M,S) floats back to back (at M = 100,
 *     S = 256: 0.81 / 2.7 / 9.6 MB per draw for D = 16 / 32 / 64, so 128 draws at D = 64 take 1.2 GB).
 *   gpode_vf_fwd_large_sets: f = vf(x) of draw q on its set_rows rows; tmp: n_sets set_rows D floats. A 128-row tile
 *     never straddles two draws (a draw's last tile is ragged); f[q] is bitwise gpode_rff_fwd_large +
 *     gpode_rbf_fwd_large (or gpode_vf_fwd_large_add_rbf) on draw q alone.
 *   gpode_rk4_fwd_large_sets: gpode_rk4_fwd_large_dev over all n_sets set_rows rows with that field; xs
 *     [Tg, n_sets set_rows, D]; tmp: 6 n_sets set_rows D floats.
 *   gpode_dopri5_fwd_large_sets: gpode_dopri5_fwd_large with one controller per draw (element-wise kernels on a
 *     (blocks, draws) grid, one controller CTA per draw, the while loop runs until every draw is done; the tiles of a
 *     finished draw are skipped). Draw q's rows of xs and its stats_out[q] ([n_sets,4] int32) are bitwise those of
 *     gpode_dopri5_fwd_large on draw q alone. work: gpode_dopri5_large_sets_work_floats(D, n_sets, set_rows) floats.
 *     Cannot be called inside a stream capture. */
int gpode_pack_cache_large_sets(const gpode_cache_t* cache_sets, int n_sets, float* packed_large, void* stream);
int gpode_vf_fwd_large_sets(const float* packed_large, const gpode_cache_t* cache_sets, int n_sets, int64_t set_rows,
                            const float* x, float* tmp, float* f, void* stream);
int gpode_rk4_fwd_large_sets(const float* packed_large, const gpode_cache_t* cache_sets, int n_sets, int64_t set_rows,
                             const float* x0, const float* t, int Tg, float* xs, float* tmp, void* stream);
int64_t gpode_dopri5_large_sets_work_floats(int D, int n_sets, int64_t set_rows);
int gpode_dopri5_fwd_large_sets(const float* packed_large, const gpode_cache_t* cache_sets, int n_sets,
                                int64_t set_rows, const float* x0, const double* t, int Tg, double rtol, double atol,
                                float* xs, float* work, int32_t* stats_out, int max_attempts, void* stream);

/* ---- ELBO side terms either side of the integrator (SURVEY.md section 8f items 1-2) -------------------------------
 * Full-rank Gaussian state posteriors N(mean_r, L_r L_r^T + jitter I), r < R, L_r given as the PACKED lower triangle
 * (the optvar of transforms.LowerTriangular / StackedLowerTriangular, src/misc/transforms.py:70-76,105-112).
 * Replaces MultivariateNormal(...).rsample / .entropy of src/core/states.py:69-74,91-92,177-182,199-204:
 *   samples_out [S,R,D] = mean + chol(L L^T + jitter I) eps,  eps [S,R,D];   entropy_out [R] (either may be NULL). */
int gpode_state_fwd(const float* mean, const float* L_packed, const float* eps, int S, int64_t R, int D, float jitter,
                    float* samples_out, float* entropy_out, void* stream);
/* Backward: grad_samples [S,R,D] and/or grad_entropy [R] -> grad_mean [R,D] (may be NULL), grad_L_packed [R,D(D+1)/2]. */
int gpode_state_bwd(const float* L_packed, const float* eps, int S, int64_t R, int D, float jitter,
                    const float* grad_samples, const float* grad_entropy, float* grad_mean, float* grad_L_packed,
                    void* stream);

/* Sum over all elements of the Gaussian log-density of decoded predictions, with its gradients in the same pass
 * (Gaussian / ProjectedGaussian.log_prob, src/core/likelihoods.py:27-28,38-45, decoder = affine map as in
 * src/misc/mocap_utils.py:24-34): pred [S,R,D], ys [R,D_obs], W [D,D_obs], bias [D_obs] or NULL, var [D_obs].
 * sum_out (device float64) = sum log N(ys | pred W + bias, var); grad_pred [S,R,D] / grad_var [D_obs] (may be NULL)
 * are the derivatives of that SUM. work: gpode_side_work_doubles() float64 of scratch (per-CTA partial sums, added in
 * a fixed order by a second kernel: the result is bitwise reproducible, no atomics). */
int gpode_loglik_sum(const float* pred, const float* ys, const float* W, const float* bias, const float* var, int S,
                     int64_t R, int D, int D_obs, double* sum_out, float* grad_pred, float* grad_var, double* work,
                     void* stream);
int64_t gpode_side_work_doubles(void);

/* Shooting-constraint term of UniformSequenceModel (src/gpode_shooting/models.py:134-135,143 with
 * src/core/constraints.py:26-36 Gaussian / :56-66 Laplace): sum over sequences, t < T-1 and dims of
 * log p(ss[.,t+1,.] | loc = pred[.,t,.], scale). ss, pred: [SN,T,D]; scale: 1 float (device). grad_ss / grad_pred
 * ([SN,T,D], may be NULL) receive the derivatives of that SUM (untouched slots are zeroed). work: as for
 * gpode_loglik_sum. */
int gpode_constraint_sum(const float* ss, const float* pred, const float* scale, int64_t SN, int T, int D, int laplace,
                         double* sum_out, float* grad_ss, float* grad_pred, double* work, void* stream);

/* Differentiable path for 8 < D <= GPODE_MAX_D_LARGE (autograd through src/core/dsvgp.py:172-197 at the upper sweep
 * dimensions; round 1 was forward-only there). Everything is stream-ordered on the device -- no host loop reads a value.
 *   gpode_pack_cache_large_bwd: w_kj = 0.5 log2(e)/ell_kj^2, Z and c_km = var_k nu_km, padded to DP = 16 / 32 / 64,
 *     then the 3xTF32 operand chunks of the tensor-core Fourier-feature half (gpode_packed_large_bwd_floats(D,M,S)
 *     floats).
 *   gpode_vf_bwd_large: grad_x = J(x)^T grad_f (Fourier-feature half on the tcgen05 tensor cores, RBF half on the
 *     FP32 CUDA cores) and the partial sums of every shared-parameter gradient, ADDED to the
 *     calling launch's per-CTA rows of acc_large (gpode_acc_large_floats(D,M) floats, zeroed by the caller before the
 *     first launch of a backward pass; all launches of one pass must use the same B). f = the forward value at x.
 *   gpode_grads_finalize_large: rows -> grad_ell [D,D], grad_var [D], grad_Z [M,D], grad_nu [D,M] (float64, row order).
 *   gpode_rk4_fwd_large_dev: torchdiffeq's 3/8-rule RK4 on the float32 device grid t[Tg] as a sequence of launches (the
 *     tcgen05 vector-field kernels + element-wise stage kernels); xs [Tg,B,D], kstages [Tg-1,4,B,D] or NULL, tmp 2 B D
 *     floats of scratch (6 B D when kstages is NULL).
 *   gpode_rk4_bwd_large: its discrete adjoint (four gpode_vf_bwd_large launches per step); work: 7 B D floats. */
int64_t gpode_packed_large_bwd_floats(int D, int M, int S);
int64_t gpode_acc_large_floats(int D, int M);
int gpode_pack_cache_large_bwd(const gpode_cache_t* cache, float* packed_bwd, void* stream);
int gpode_vf_bwd_large(const float* packed_bwd, int D, int M, int S, const float* x, const float* f, const float* grad_f,
                       float* grad_x, float* acc_large, int64_t B, void* stream);
int gpode_grads_finalize_large(const gpode_cache_t* cache, const float* acc_large, int64_t B, float* grad_ell,
                               float* grad_var, float* grad_Z, float* grad_nu, void* stream);
int gpode_rk4_fwd_large_dev(const float* packed_large, const gpode_cache_t* cache, const float* x0, const float* t, int Tg,
                            int64_t B, float* xs, float* kstages, float* tmp, void* stream);
int gpode_rk4_bwd_large(const float* packed_bwd, const gpode_cache_t* cache, const float* t, int Tg, int64_t B,
                        const float* xs, const float* kstages, const float* grad_xs, float* grad_x0, float* acc_large,
                        float* work, void* stream);

/* Adaptive dopri5 for 8 < D <= GPODE_MAX_D_LARGE, controller on the device: torchdiffeq 0.2.0's
 * odeint(method='dopri5') as called from Flow.forward (src/core/flow.py:84-90). One attempt (six tcgen05 vector-field
 * evaluations, stage / error kernels, a one-CTA controller kernel, an accept kernel) is the body of a CUDA-graph WHILE
 * node; the controller sets the loop condition, so the host enqueues one graph launch and never synchronises (the
 * reference does once per attempt). t: float64 device grid (increasing or decreasing); xs [Tg,B,D]; stats_out (device,
 * 4 int32): nfe, accepted, rejected, status (0 ok, 1 attempt limit, 2 dt underflow, 3 checkpoint capacity); work:
 * gpode_dopri5_large_work_floats(D,B) floats. Cannot be called inside a stream capture (it builds its own graph).
 *   gpode_dopri5_fwd_large_ckpt: the same solve (bitwise the same xs and stats when it succeeds) that also records the
 *     accepted steps in ckpt, gpode_dopri5_ckpt_floats(D,B,Tg,cap) floats (layout at that function; k holds the RAW
 *     vector-field values here): 8 B D floats per accepted step. status 3 = more than `cap` accepted steps (retry with
 *     a larger cap).
 *   gpode_dopri5_bwd_large: the discrete adjoint of those steps (step sizes are constants, as in torchdiffeq; the two
 *     initial-step evaluations get no cotangent): grad_xs [Tg,B,D] -> grad_x0 [B,D], six gpode_vf_bwd_large launches
 *     per accepted step plus one at x0, all adding into acc_large (zeroed by the caller; follow with
 *     gpode_grads_finalize_large). n_accepted = stats_out[1] of the forward; work: 11 B D floats. Bitwise
 *     reproducible (no atomics). */
int64_t gpode_dopri5_large_work_floats(int D, int64_t B);
int gpode_dopri5_fwd_large(const float* packed_large, const gpode_cache_t* cache, const float* x0, const double* t, int Tg,
                           int64_t B, double rtol, double atol, float* xs, float* work, int32_t* stats_out,
                           int max_attempts, void* stream);
int gpode_dopri5_fwd_large_ckpt(const float* packed_large, const gpode_cache_t* cache, const float* x0, const double* t,
                                int Tg, int64_t B, double rtol, double atol, float* xs, float* work, int32_t* stats_out,
                                int max_attempts, float* ckpt, int cap, void* stream);
int gpode_dopri5_bwd_large(const float* packed_bwd, const gpode_cache_t* cache, const double* t, int Tg, int64_t B,
                           const float* grad_xs, const float* ckpt, int cap, int n_accepted, float* grad_x0,
                           float* acc_large, float* work, void* stream);

/* Fused multiple-shooting ELBO step (SURVEY.md section 8f item 2). Every row (s, n, t) of the (S_mc, N, T) batch of
 * sampled states `ss` is integrated over ONE interval t2[0] -> t2[1] with the 3/8-rule RK4 step (as gpode_rk4_fwd with
 * Tg = 2) and the two ELBO terms that use the end point are evaluated inside the integrator kernel, on the end point
 * while it is in registers (UniformSequenceModel.build_lowerbound_terms, src/gpode_shooting/models.py:119-135):
 *   sums_out[0] = sum_rows sum_d log N(ys[n,t,d] | (pred W + bias)_d, lik_var_d)    (src/core/likelihoods.py:27-45)
 *   sums_out[1] = sum_{rows, t < T-1} log p(ss[s,n,t+1] | loc = pred, scale)        (src/core/constraints.py:26-66)
 * for the rows [row_lo, row_hi) of the batch (row = (s N + n) T + t): a rank of a multi-GPU job passes its own range
 * and the FULL `ss`, so the constraint's neighbour state is local (the "halo" of the shard is one extra row of `ss`).
 * Outputs besides the two sums: grad_lik_var [D_obs] (d sums_out[0] / d lik_var, may be NULL), kstages [1,4,B,D] and
 * seeds [2,B,D] (d sums_out[0] / d pred | d sums_out[1] / d pred; both NULL for a forward without gradients),
 * pred_out [B,D] (may be NULL). work: gpode_shoot_work_doubles() float64 of scratch. Sums are taken in a fixed order
 * (bitwise reproducible).
 * `laplace` is a flag word: bit 0 = Laplace instead of Gaussian constraint density; bit 1 = TIME-SHARDED batch: `ss` /
 * `ys` hold a contiguous slice of the time axis plus ONE trailing halo index per sequence (the next rank's first state),
 * which is only the constraint's neighbour -- it gets no observation term and contributes nothing to any gradient except
 * the constraint's pull on it (distributed.enable_time_sharding: the state-distribution work shards with the rows). */
typedef struct {
    int32_t S_mc, N, T, D_obs, laplace;
    const float* ys;         /* [N, T, D_obs] */
    const float* W;          /* [D, D_obs] decoder (identity for the plain Gaussian likelihood) */
    const float* bias;       /* [D_obs] or NULL */
    const float* lik_var;    /* [D_obs] */
    const float* cons_scale; /* 1 float */
    int64_t row_lo, row_hi;
} gpode_shoot_t;
int64_t gpode_shoot_work_doubles(void);
int gpode_shoot_fwd(const float* packed, int D, int M, int S, const gpode_shoot_t* sh, const float* ss, const float* t2,
                    float* kstages, float* pred_out, float* seeds, double* sums_out, float* grad_lik_var, double* work,
                    void* stream);
/* Its adjoint: starts from lambda = g_ll seeds[0] + g_cons seeds[1] (g_ll, g_cons: upstream gradients of the two sums,
 * device scalars), writes grad_ss [S_mc,N,T,D] for rows [row_lo, row_hi) -- dynamics plus the constraint's pull on the
 * next state -- and for row row_hi when the range ends inside a sequence (the caller zeroes grad_ss first when the
 * range is not the whole batch); lengthscale / variance partial sums and virtual rows as gpode_rk4_bwd
 * (vrows: gpode_vrow_floats(D, 4 B) floats). Follow with gpode_param_grad over 4 B rows and gpode_grads_finalize.
 * vrows may be NULL when gpode_shoot_bwd_vrows(D, M, S, B) returns 0 (B = row_hi - row_lo): the tensor-core adjoint
 * (4 <= D <= 5, batches that fill the GPU) then sums the inducing-point gradients itself into `acc`, and only
 * gpode_grads_finalize follows. */
int64_t gpode_shoot_bwd_vrows(int D, int M, int S, int64_t n_rows);
int gpode_shoot_bwd(const float* packed, int D, int M, int S, const gpode_shoot_t* sh, const float* ss, const float* t2,
                    const float* kstages, const float* seeds, const float* g_ll, const float* g_cons, float* grad_ss,
                    float* vrows, float* acc, void* stream);

/* Kernel-selection options (the library's only process-wide mutable state). Defaults are read from the environment
 * once (GPODE_BWD_MMA, GPODE_FWD_MMA); names:
 *   "bwd_mma" / "fwd_mma" (1): tensor-core adjoint / forward at D = 4, 5 and B >= SMs x 384 rows; 0 = FFMA2 kernels.
 *       Domain of the split-fp16 operands: |x_j|, |Omega| < 65504 -- beyond it the kernels return NaN (fp16 overflow),
 *       never silently wrong numbers; a float32 angle of that size carries no phase information anyway.
 * Any other name is an error (-1). */
int gpode_set_option(const char* name, int value);
int gpode_get_option(const char* name);

/* Measurement utility (no reference counterpart): sustained FP32 FMA throughput of the current device in TFLOP/s
 * (best of 5 launches of a register-only FMA loop; synchronises the stream). scratch: >= 1 float (device). */
int gpode_probe_fp32_fma(double* tflops_out_host, double* ms_out_host, float* scratch, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GPODE_B200_H */
