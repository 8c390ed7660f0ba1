"""-m gpu: the persistent large-D (8 < D <= 64) kernels at batch sizes where every CTA runs two or more tiles.

Every large-D kernel walks its tiles as ``for (tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)`` and carries state
from one tile to the next: ring slots and mbarrier parities, TMEM buffers, the per-CTA accumulator rows of the VJP, the
per-thread partial sums of the grid-stride dopri5 kernels, the skipped tiles of finished draws. The oracle tests of
test_gpu_kernels / test_gpu_large_dopri5 / test_gpu_large_sets run at most one tile per CTA; here the batch sizes are
derived from the SM count and each kernel's grid rule, so that every CTA runs at least two tiles, most of them three,
the tile count is uneven across CTAs and the last tile is ragged. D, M and the operand chunks per tile are odd, so every
two-slot ring, double buffer and mbarrier parity starts a CTA's second tile on the other phase than its first.

The oracle is gpode_oracle evaluated over row chunks (row outputs and x-gradients concatenated, parameter gradients
summed). The large ones run on the device, as plain torch ops in float32 and float64: none of the product's kernels."""
import numpy as np
import pytest
import torch

import gpode_oracle as O
from util import (GRAD_KEYS, TOL_GRAD, TOL_TRAJ, TOL_VF, assert_grads, assert_parity, chunked_oracle, cuda_args,
                  cuda_grads, lazy, oracle_cache, oracle_dopri5, oracle_rk4, oracle_vf, time_grid)

pytestmark = pytest.mark.gpu

ROWS = 128                # rows per tile of the tcgen05 kernels, vjp_large_kernel and rbf_vjp_large_kernel
SMEM = 227 * 1024         # the launchers' shared-memory limit per CTA
LD_THREADS = 2368 * 256   # ld_grid (large_dopri5.cu): at most 2368 blocks x 256 threads, grid-stride over B * D


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- the grid rules of the launchers, restated ----------------------------------------------------------------------
def _lu_kp(D):
    return (D + 1 + 7) & ~7


def _lu_nc(D):
    return 128 if D > 40 else 64


def _lu_kd(D):
    return (D + 7) & ~7


def _lu_nd(D):
    return (D + 15) & ~15


def rff_fwd_ctas(D):
    """rff_launch (large_umma.cu): min(tiles, SMs * occ), occ = min(227 KB / (smem + 1 KB), 512 TMEM columns / 2 NC)."""
    KP, NC = _lu_kp(D), _lu_nc(D)
    smem = 128 + (2 * KP * ROWS + 2 * 2 * KP * NC) * 4
    return _sms() * min(SMEM // (smem + 1024), 512 // (2 * NC))


def rbf_smem(D, M):
    """rbf_smem (large_umma.cu): -W^T hi|lo, Z [M][KD], the state tile and two A slots (hi|lo)."""
    KD, ND = _lu_kd(D), _lu_nd(D)
    return 128 + (2 * ND * KD + M * KD + KD * ROWS + 4 * KD * ROWS) * 4


def rbf_fwd_ctas_max(D, M):
    """rbf_launch: occ = min(shared memory, 512 / 128 TMEM columns, 2048 / 288 threads, registers). The register bound
    depends on the compiler, so this is an upper bound of the grid: a batch that gives every CTA two tiles at this grid
    gives each at least as many at the real one."""
    return _sms() * min(SMEM // (rbf_smem(D, M) + 1024), 4, 2048 // 288)


def fallback_rbf_ctas_max(D):
    """large_d_rbf_kernel (large_d.cu, 32-row tiles): SMs x an occupancy query; bounded here by threads
    (((4 D + 31) / 32) 32 per CTA, 2048 per SM) and shared memory (D^2 + 2 * 32 D floats)."""
    threads = (4 * D + 31) // 32 * 32
    smem = 4 * (((D * D + 3) & ~3) + 2 * 32 * D)
    return _sms() * min(2048 // threads, SMEM // smem)


def m_star(D):
    """The largest M whose copy of Z fits the tcgen05 RBF forward's shared memory (rbf_smem <= 227 KB); at M* + 1 the
    forward takes the FP32 kernel gpode_vf_fwd_large_add_rbf."""
    return (SMEM - rbf_smem(D, 0)) // (4 * _lu_kd(D))


def rv_ctas(B):
    """gpode_rv_grid (large_rffb.cu): min(tiles, SMs, 160) CTAs of rff_vjp_large_kernel."""
    return min(-(-B // ROWS), _sms(), 160)


def lb_ctas(B, D):
    """lb_grid (large_bwd.cu): min(tiles, 2 SMs, 592) CTAs of vjp_large_kernel<16 / 32> (D <= 32), min(tiles, SMs) of
    rbf_vjp_large_kernel<64> (D > 32)."""
    return min(-(-B // ROWS), _sms() * (2 if D <= 32 else 1), 592)


def multi_tile_tiles(ctas):
    """3 tiles per CTA less a tenth of the CTAs: every CTA runs >= 2 tiles, most run 3, and the count is uneven."""
    n = 3 * ctas - max(1, ctas // 10)
    assert n >= 2 * ctas and n % ctas != 0
    return n


def multi_tile_batch(ctas, tail):
    """B rows in multi_tile_tiles(ctas) tiles of 128, the last one holding `tail` rows (1 <= tail < 128: ragged)."""
    assert 1 <= tail < ROWS
    return (multi_tile_tiles(ctas) - 1) * ROWS + tail


# ---- problem and oracle ---------------------------------------------------------------------------------------------
def _setup(D, M, S, B, seed, nu_scale=0.1):
    p, ys, ts, draws, _ = O.make_problem(D=D, M=M, S=S, N=1, T=4, seed=seed)
    gp, c = oracle_cache(p, draws, torch.float32)
    c['nu'] = torch.tensor(np.random.default_rng(seed + 1).normal(size=(D, M, 1)) * nu_scale, dtype=torch.float32)
    x = torch.tensor(np.random.default_rng(seed + 2).normal(size=(B, D)) * 1.5, dtype=torch.float32)
    return gp, c, x


def _tile_rows(tiles, B):
    return torch.cat([torch.arange(t * ROWS, min((t + 1) * ROWS, B)) for t in tiles])


# ---- forward ----------------------------------------------------------------------------------------------------------
# (D, M, S, tail). D * ceil(S / NC) operand chunks per tile (NC = 64 at D <= 40, 128 above): 17, 41 * 3, 63 -- all odd.
# B = multi_tile_batch(max(rff grid, rbf grid bound)): at D = 17 the Fourier kernel holds 4 CTAs per SM, above D = 40
# both kernels hold one; the D = 17 batch ends in a one-row tile.
@pytest.mark.parametrize("D,M,S,tail", [(17, 31, 64, 1), (41, 33, 384, 77), (63, 45, 128, 100)])
def test_forward_multi_tile_equals_single_tile_launches_and_oracle(D, M, S, tail):
    from gaussian_process_odes_b200 import ops
    ctas = max(rff_fwd_ctas(D), rbf_fwd_ctas_max(D, M))
    B = multi_tile_batch(ctas, tail)
    gp, c, x = _setup(D, M, S, B, seed=D + 5)
    args = cuda_args(gp, c)
    ts = time_grid(3, 0.05, D)
    xc = x.cuda()
    with torch.no_grad():
        f = ops.vector_field(xc, *args)
        xs = ops.rk4_integrate(xc, ts.cuda(), *args)
        # every row's sums run in an order fixed by the row alone: slices of <= 1000 rows (<= 8 tiles, one per CTA)
        # give the same bits
        for r0 in range(0, B, 1000):
            assert torch.equal(f[r0:r0 + 1000], ops.vector_field(xc[r0:r0 + 1000], *args)), ("vf", r0)
            assert torch.equal(xs[:, r0:r0 + 1000], ops.rk4_integrate(xc[r0:r0 + 1000], ts.cuda(), *args)), ("rk4", r0)
    # row-local: the oracle on the first, second and third tiles of CTAs 0, 1 and the last CTA, the last full tile and
    # the ragged one
    n = -(-B // ROWS)
    tiles = sorted({0, 1, ctas - 1, ctas, ctas + 1, 2 * ctas - 1, 2 * ctas, 2 * ctas + 1, n - 2, n - 1})
    rows = _tile_rows(tiles, B)
    xr = x[rows]
    f32 = O.vf_forward(xr, gp['Z'], gp['ell'], gp['var'], c)
    c64 = {k: v.double() for k, v in c.items()}
    f64 = O.vf_forward(xr.double(), gp['Z'].double(), gp['ell'].double(), gp['var'].double(), c64)
    assert_parity("multi-tile vf D=%d" % D, f.cpu()[rows], f32, f64, TOL_VF)
    r32 = O.odeint(lambda t, y: O.vf_forward(y, gp['Z'], gp['ell'], gp['var'], c), xr, ts, method='rk4')
    r64 = lambda: O.odeint(lambda t, y: O.vf_forward(y, gp['Z'].double(), gp['ell'].double(), gp['var'].double(), c64),
                           xr.double(), ts.double(), method='rk4')
    assert_parity("multi-tile rk4 D=%d" % D, xs.cpu()[:, rows], r32, r64, TOL_TRAJ)


# ---- VJP ------------------------------------------------------------------------------------------------------------
# (D, M, S, tail). D * ceil(S / 64) chunks per tile of the tensor-core Fourier half: 17, 33 * 3, 63. The RBF half is
# vjp_large_kernel<32> at D = 17 (2 CTAs per SM) and rbf_vjp_large_kernel<64> at D = 33, 63 (1 per SM); the Fourier
# half runs min(SMs, 160) CTAs. B = multi_tile_batch of the larger grid, so both halves and the finalize kernel (which
# reads one accumulator row per CTA) see >= 2 tiles per CTA.
VJP_SHAPES = [(17, 31, 64, 1), (33, 25, 192, 64), (63, 45, 64, 127)]


def _vjp_batch(D):
    ctas = max(rv_ctas(1 << 40), lb_ctas(1 << 40, D))
    return multi_tile_batch(ctas, dict((s[0], s[3]) for s in VJP_SHAPES)[D])


@pytest.mark.parametrize("D,M,S,tail", VJP_SHAPES)
def test_vjp_multi_tile_matches_chunked_oracle(D, M, S, tail):
    from gaussian_process_odes_b200 import ops
    B = _vjp_batch(D)
    assert rv_ctas(B) * 2 <= -(-B // ROWS) and lb_ctas(B, D) * 2 <= -(-B // ROWS)
    gp, c, x = _setup(D, M, S, B, seed=D + 11)
    cot = torch.tensor(np.random.default_rng(D).normal(size=(B, D)), dtype=torch.float32)
    fn = lambda xc, a: ops.vector_field(xc, *a)
    f, got = cuda_grads(fn, gp, c, x, cot)
    _, again = cuda_grads(fn, gp, c, x, cot)
    for k in GRAD_KEYS:
        assert torch.equal(got[k], again[k]), "two backward passes differ in grad " + k
    out32, ref32 = chunked_oracle(oracle_vf, gp, c, x, cot, torch.float32, 0)
    ref64 = lazy(lambda: chunked_oracle(oracle_vf, gp, c, x, cot, torch.float64, 0))
    assert_parity("multi-tile vf D=%d" % D, f.cpu(), out32, lambda: ref64()[0], TOL_VF)
    assert_grads("multi-tile vf D=%d" % D, got, ref32, lambda: ref64()[1], TOL_GRAD)


@pytest.mark.parametrize("D,M,S,tail", [VJP_SHAPES[0], VJP_SHAPES[2]])
def test_rk4_backward_multi_tile_matches_chunked_oracle(D, M, S, tail):
    """2 RK4 steps: eight VJPs add into the same accumulator rows before one finalize."""
    from gaussian_process_odes_b200 import ops
    B = _vjp_batch(D)
    gp, c, x = _setup(D, M, S, B, seed=D + 17)
    ts = time_grid(3, 0.05, 3)
    cot = torch.tensor(np.random.default_rng(D + 1).normal(size=(3, B, D)), dtype=torch.float32)
    xs, got = cuda_grads(lambda xc, a: ops.rk4_integrate(xc, ts.cuda(), *a), gp, c, x, cot)
    out32, ref32 = chunked_oracle(oracle_rk4(ts), gp, c, x, cot, torch.float32, 1)
    ref64 = lazy(lambda: chunked_oracle(oracle_rk4(ts), gp, c, x, cot, torch.float64, 1))
    assert_parity("multi-tile rk4 D=%d" % D, xs.cpu(), out32, lambda: ref64()[0], TOL_TRAJ)
    assert_grads("multi-tile rk4 D=%d" % D, got, ref32, lambda: ref64()[1], TOL_GRAD)


# ---- dopri5 -----------------------------------------------------------------------------------------------------------
def test_dopri5_grid_stride_kernels_run_several_passes():
    """D = 63, M = 9, S = 16 (one chunk that the features do not fill). B * D > 2 * 2368 * 256: every thread of the ld_*
    kernels (forward controller norms, stage algebra, adjoint stages) makes >= 2 grid-stride passes and its float64
    partial sums cover both."""
    from gaussian_process_odes_b200 import ops
    D, M, S = 63, 9, 16
    B = 2 * LD_THREADS // D + 257
    assert B * D > 2 * LD_THREADS
    gp, c, x = _setup(D, M, S, B, seed=63)
    ts = torch.tensor([0.0, 0.05, 0.32], dtype=torch.float32)
    cot = torch.tensor(np.random.default_rng(8).normal(size=(3, B, D)), dtype=torch.float32)
    args = cuda_args(gp, c, True)
    xc = x.cuda().requires_grad_(True)
    xs, stats = ops.dopri5_integrate(xc, ts.cuda(), *args)
    (xs * cot.cuda()).sum().backward()
    got = dict(x=xc.grad, Z=args[0].grad, ell=args[1].grad, var=args[2].grad, nu=args[3].grad)
    torch.cuda.reset_peak_memory_stats()
    out32, ref32, st = oracle_dopri5(gp, c, x, ts, cot, torch.float32)
    ref64 = lazy(lambda: oracle_dopri5(gp, c, x, ts, cot, torch.float64))
    nfe, acc, rej, status = [int(v) for v in stats.cpu()]
    assert status == 0 and nfe == 2 + 6 * (acc + rej)
    assert abs(acc - st['accepted']) <= 1 and abs(rej - st['rejected']) <= 1, (acc, rej, st)
    assert_parity("dopri5 B*D=%d" % (B * D), xs.detach().cpu(), out32, lambda: ref64()[0], TOL_TRAJ)
    # both are exact gradients of a discrete solve; they may differ by one accept/reject decision (as in
    # test_gpu_large_dopri5)
    assert_grads("dopri5 B*D=%d" % (B * D), got, ref32, lambda: ref64()[1], 2e-4)
    print("dopri5 oracle peak device memory: %.2f GB" % (torch.cuda.max_memory_allocated() / 2 ** 30))


# ---- batched prediction ---------------------------------------------------------------------------------------------
def _draw_sets(D, M, S, n, seed):
    """shared hyper-parameters + n draws; nu scaled per draw (1, 30, 100, 10, ...) so that the draws' dopri5 controllers
    finish at different attempts and the finished draws' tiles are skipped while the others still run"""
    p, ys, ts, _, _ = O.make_problem(D=D, M=M, S=S, N=1, T=4, seed=seed)
    gp = O.gp_params(O.cast(p, torch.float32))
    rng = np.random.default_rng(seed)
    t = lambda a: torch.tensor(np.asarray(a, dtype=np.float32))
    scale = torch.tensor([1.0, 30.0, 100.0, 10.0])[torch.arange(n) % 4].reshape(n, 1, 1)
    sets = dict(omega=t(rng.standard_normal(size=(n, D, S, D), dtype=np.float32)) / gp['ell'].T.unsqueeze(1),
                phase=t(rng.uniform(size=(n, S, D))) * 2 * np.pi, w=t(rng.normal(size=(n, S, D))),
                nu=t(rng.normal(size=(n, D, M))) * 0.1 * scale)
    return gp, sets


# (D, M, S, n, N): n * tiles-per-draw above every forward kernel's grid. Many draws x one row (the prediction shape,
# D = 45: both tcgen05 kernels hold one CTA per SM, one tile per draw); a few draws x many rows (D = 17: the Fourier
# kernel holds four CTAs per SM); M above m_star(63) = 139 at D = 63, where the RBF term runs on large_d_rbf_kernel
# (32-row tiles) and skips the finished draws' tiles itself.
def _sets_case(kind):
    """-> D, M, S, n, N and the tcgen05 Fourier kernel's grid"""
    if kind == "many_draws":
        ctas = max(rff_fwd_ctas(45), rbf_fwd_ctas_max(45, 33))
        return 45, 33, 128, multi_tile_tiles(ctas), 1, ctas
    if kind == "many_rows":
        n, ctas = 3, max(rff_fwd_ctas(17), rbf_fwd_ctas_max(17, 31))
        return 17, 31, 64, n, (multi_tile_tiles(ctas) // n - 1) * ROWS + 65, ctas
    # 32-row tiles: the Fourier kernel (128-row tiles, one CTA per SM at D = 63) runs more than 2 tiles per CTA too
    n, ctas = 5, fallback_rbf_ctas_max(63)
    return 63, m_star(63) + 2, 64, n, (multi_tile_tiles(ctas) // n - 1) * 32 + 17, rff_fwd_ctas(63)


@pytest.mark.parametrize("kind", ["many_draws", "many_rows", "rbf_fallback"])
def test_sets_multi_tile_with_skipped_draws_bitwise_per_draw(kind):
    from gaussian_process_odes_b200 import ops
    D, M, S, n, N, ctas = _sets_case(kind)
    gp, sets = _draw_sets(D, M, S, n, seed=D + n)
    assert (kind == "rbf_fallback") == (rbf_smem(D, M) > SMEM)
    noise = torch.tensor(np.random.default_rng(5).normal(size=(n, N, D)), dtype=torch.float32)
    x0 = (gp['Z'][torch.arange(n * N) % M].reshape(n, N, D) + 0.1 * noise).cuda()
    shared = [gp[k].cuda().contiguous() for k in ("Z", "ell", "var")]
    allsets = [sets[k].cuda() for k in ("nu", "omega", "phase", "w")]
    one = lambda q: [sets[k][q].cuda().contiguous() for k in ("nu", "omega", "phase", "w")]
    # the draws compared one by one: all of them for the vector field; for dopri5 the first four (every nu scale), the
    # last two and, with one tile per draw, those whose tile opens the second and third round of the Fourier kernel
    tpd = -(-N // ROWS)
    check = sorted({q for q in [0, 1, 2, 3, ctas // tpd - 1, ctas // tpd, 2 * ctas // tpd, n - 2, n - 1] if 0 <= q < n})
    ts = torch.tensor([0.0, 0.1, 0.35, 0.5]).cuda()
    with torch.no_grad():
        f = ops.vector_field_sets(x0, *shared, *allsets)
        for q in range(n):
            assert torch.equal(f[q], ops.vector_field(x0[q], *shared, *one(q))), "vf draw %d" % q
        xs, stats = ops.integrate_sets(x0, ts, *shared, *allsets, method="dopri5")
        counts = set()
        for q in range(n):
            nfe, acc, rej, status = stats[q].tolist()
            assert status == 0 and nfe == 2 + 6 * (acc + rej), (q, stats[q].tolist())
            counts.add(acc + rej)
        assert len(counts) >= 2, "every draw's controller took the same number of attempts: no tile was skipped"
        for q in check:
            ref, st = ops.dopri5_integrate(x0[q], ts, *shared, *one(q))
            assert torch.equal(xs[q], ref.permute(1, 0, 2)), "dopri5 draw %d differs from the single-draw call" % q
            assert torch.equal(stats[q], st), (q, stats[q].tolist(), st.tolist())
