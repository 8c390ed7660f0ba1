"""-m gpu: the blocked float64 whitening (csrc/whiten_blocked.cu) that ops.whiten / ops.whiten_sets use at D <= 8 above
M = 160 inducing points: against float64 torch.linalg differentiated by autograd, against the in-shared-memory tile
kernels where both exist, batched draws against single draws, repeatability, and end to end through the model classes
against the oracle port.

Inducing points sit on a unit lattice (jittered by 0.05) with lengthscales 0.7 (1 +- 5%), so Kzz + 1e-5 I is well
conditioned: cond <= 6.3e2 for every shape below (eigvalsh in float64; D = 8, M = 1024 is the largest). The float64
round-off of the two implementations then stays far below the float32 rounding of the outputs."""
import ctypes
import itertools
import math

import numpy as np
import pytest
import torch

import gpode_oracle as O
from util import TOL_GRAD, build_product_model, relerr

pytestmark = pytest.mark.gpu
JITTER = 1e-5


def _lattice(D, M, seed, spacing=1.0):
    side = math.ceil(M ** (1.0 / D) - 1e-9)
    pts = np.array(list(itertools.islice(itertools.product(range(side), repeat=D), M)), dtype=np.float64)
    return (pts + 0.05 * np.random.default_rng(seed).uniform(-1, 1, size=pts.shape)) * spacing


def _inputs(D, M, S, seed, n_sets=None):
    """Z, ell, var, u and the Fourier features of one draw (n_sets: a leading draw axis on u, omega, phase, w). Omega is
    scaled to the lattice's extent so that the float32 angles stay within a few radians."""
    rng = np.random.default_rng(seed)
    t = lambda a: torch.tensor(np.asarray(a), dtype=torch.float32, device="cuda")
    lead = () if n_sets is None else (n_sets,)
    Z = t(_lattice(D, M, seed))
    ell = t(0.7 * (1 + 0.05 * rng.uniform(-1, 1, size=(D, D))))
    var = t(0.5 + rng.uniform(size=D))
    u = t(rng.normal(size=lead + (M, D)))
    extent = float(Z.abs().max()) + 1.0
    omega = t(rng.normal(size=lead + (D, S, D)) / extent)
    phase = t(rng.uniform(size=lead + (S, D)) * 2 * np.pi)
    w = t(rng.normal(size=lead + (S, D)))
    return Z, ell, var, u, omega, phase, w


def _struct(Z, ell, var, omega, phase, w):
    from gaussian_process_odes_b200 import ops
    M, D = Z.shape
    S = w.shape[-2]
    return ops._cache_struct(D, M, S, omega, phase.contiguous(), w, Z, None, ell, var)


def _fwd(entry, Z, ell, var, u, omega, phase, w):
    """One C-ABI forward (tile or blocked) -> nu, L, sp."""
    from gaussian_process_odes_b200 import _lib
    from gaussian_process_odes_b200._lib import ptr, stream_ptr
    M, D = Z.shape
    st = _struct(Z, ell, var, omega, phase, w)
    nu = torch.empty(D, M, dtype=torch.float32, device="cuda")
    L = torch.empty(D, M, M, dtype=torch.float64, device="cuda")
    sp = torch.empty(D, 2, M, dtype=torch.float64, device="cuda")
    if entry == "blocked":
        work = torch.empty(_lib.load().gpode_whiten_blocked_work_doubles(D, M, 1), dtype=torch.float64, device="cuda")
        _lib.check(_lib.load().gpode_whiten_fwd_blocked(ctypes.byref(st), ptr(u), JITTER, ptr(nu), ptr(L), ptr(sp),
                                                        ptr(work), stream_ptr()))
    else:
        _lib.check(_lib.load().gpode_whiten_fwd(ctypes.byref(st), ptr(u), JITTER, ptr(nu), ptr(L), ptr(sp),
                                                stream_ptr()))
    return nu, L, sp


def _bwd(entry, Z, ell, var, u, omega, phase, w, L, sp, gnu):
    from gaussian_process_odes_b200 import _lib
    from gaussian_process_odes_b200._lib import ptr, stream_ptr
    M, D = Z.shape
    st = _struct(Z, ell, var, omega, phase, w)
    out = [torch.empty(M, D, device="cuda"), torch.empty(M, D, device="cuda"), torch.empty(D, D, device="cuda"),
           torch.empty(D, device="cuda")]   # grad_u, grad_Z, grad_ell, grad_var
    args = [ctypes.byref(st), ptr(u), ptr(L), ptr(sp), ptr(gnu)] + [ptr(o) for o in out]
    if entry == "blocked":
        work = torch.empty(_lib.load().gpode_whiten_blocked_work_doubles(D, M, 0), dtype=torch.float64, device="cuda")
        _lib.check(_lib.load().gpode_whiten_bwd_blocked(*args, ptr(work), stream_ptr()))
    else:
        _lib.check(_lib.load().gpode_whiten_bwd(*args, stream_ptr()))
    return out


def _prior(Z, ell, var, omega, phase, w, angles):
    """rff_forward(Z) (M, D), summed in float64, with omega = eps / ell (the library folds the omega path into
    grad_ell, as the reference's autograd does through kernels.py:110-112): differentiable in Z, ell and var. angles:
    the dtype the angles and feature weights are formed in (float32 is what the kernels and the reference do)."""
    S, D = w.shape
    eps = omega.double() * ell.detach().t().unsqueeze(1)
    om = (eps / ell.t().unsqueeze(1)).to(angles)
    theta = torch.einsum('mj,jsk->msk', Z.to(angles), om) + phase.to(angles).reshape(1, S, D)
    a = (w.double() * torch.sqrt(var / S)).to(angles)
    return (torch.cos(theta.double()) * a.double().unsqueeze(0)).sum(1)


def _reference(Z, ell, var, u, omega, phase, w, cot, p_kernel, angles):
    """nu and the gradients of <nu, cot> through float64 torch.linalg (ops._whiten_large's formulation). The prior
    enters with the kernel's value p_kernel; its derivative in Z and ell is that of _prior(..., angles), in var the
    exact p / (2 var) of p ~ sqrt(var) applied to p_kernel -- what the kernel does with its own prior."""
    from gaussian_process_odes_b200 import ops
    Zd, ed, vd, ud = [x.double().requires_grad_(True) for x in (Z, ell, var, u)]
    L = ops._kzz_cholesky_large(Zd, ed, vd, JITTER)
    p = _prior(Zd, ed, vd.detach(), omega, phase, w, angles)
    prior = p_kernel * torch.sqrt(vd / vd.detach()) + (p - p.detach())
    a = torch.linalg.solve_triangular(L, prior.t().unsqueeze(2), upper=False)
    ref = torch.linalg.solve_triangular(L.transpose(1, 2), ud.t().unsqueeze(2) - a, upper=True).squeeze(2)
    (ref * cot.double()).sum().backward()
    return L.detach(), a.detach().squeeze(2), p.detach(), dict(nu=ref.detach(), Z=Zd.grad, ell=ed.grad, var=vd.grad,
                                                                u=ud.grad)


SHAPES = [(D, M) for D in (1, 2, 5, 8) for M in (161, 200, 257, 511, 1024)] + [(2, 2048)]


@pytest.mark.parametrize("D,M", SHAPES)
def test_blocked_whitening_against_float64_linalg(D, M):
    """nu, L and the gradients of <nu, cot> w.r.t. u, Z, ell, var against the same function in float64 torch.linalg,
    differentiated by autograd (ops._whiten_large's formulation, omega = eps / ell). The kernel evaluates the prior at
    Z and its derivative with float32 angles, like the reference; the prior's value is checked against float64 on its
    own and enters the reference as a value (and through p ~ sqrt(var) into grad_var), so nu, grad_u and grad_var
    isolate the blocked factorisation and solves: 1e-6 of max-abs, the float32 rounding of the outputs. grad_Z and
    grad_ell also carry the derivative of the prior in Z and ell, whose float32 angles and weights leave ~1e-7..1e-6
    against float64: there the project's arbitration applies -- 1e-6, or 1.5x the deviation that float32 angles and
    weights alone cause in the same float64 reference."""
    from gaussian_process_odes_b200 import ops
    S = 64
    Z, ell, var, u, omega, phase, w = _inputs(D, M, S, seed=D * 7 + M)
    nu_b, L_b, sp_b = _fwd("blocked", Z, ell, var, u, omega, phase, w)
    cot = torch.tensor(np.random.default_rng(M).normal(size=(D, M)), dtype=torch.float32, device="cuda")
    leaves = [a.clone().requires_grad_(True) for a in (Z, ell, var, u)]
    nu = ops.whiten(*leaves, omega, phase, w, JITTER)
    (nu * cot).sum().backward()
    got = dict(nu=nu.detach(), Z=leaves[0].grad, ell=leaves[1].grad, var=leaves[2].grad, u=leaves[3].grad)
    assert torch.equal(got["nu"], nu_b)   # ops.whiten dispatches to the blocked entry point above M = 160

    p_kernel = sp_b[:, 1, :].t()
    L, s, p64, want = _reference(Z, ell, var, u, omega, phase, w, cot, p_kernel, torch.float64)
    want32 = _reference(Z, ell, var, u, omega, phase, w, cot, p_kernel, torch.float32)[3]
    assert relerr(L_b, L) <= 1e-9
    assert float(L_b.triu(1).abs().max()) == 0.0
    assert relerr(p_kernel, p64) <= 1e-6
    assert relerr(sp_b[:, 0, :], s) <= 1e-9
    for k in want:
        e, e_ref = relerr(got[k], want[k]), relerr(want32[k], want[k])
        assert e <= max(1e-6, 1.5 * e_ref), (k, e, e_ref)


@pytest.mark.parametrize("D", [2, 5, 8])
@pytest.mark.parametrize("M", [64, 112, 160])
def test_blocked_entry_points_match_tile_kernels(D, M):
    """Where both paths exist the blocked entry points reproduce gpode_whiten_fwd / _bwd. The tile kernels factor in
    float64 up to M = 112 (L and sp to 1e-12, the float32 outputs to 1e-6) and in float32 shared memory above: at
    M = 160 their own round-off, about cond(Kzz) 2^-24 (cond <= 6.3e2 here), bounds the agreement (1e-5)."""
    Z, ell, var, u, omega, phase, w = _inputs(D, M, 96, seed=100 + D + M)
    nu_t, L_t, sp_t = _fwd("tile", Z, ell, var, u, omega, phase, w)
    nu_b, L_b, sp_b = _fwd("blocked", Z, ell, var, u, omega, phase, w)
    tol64, tol32 = (1e-12, 1e-6) if M <= 112 else (1e-6, 1e-5)
    assert relerr(L_b, L_t) <= tol64
    assert relerr(sp_b, sp_t) <= tol64
    assert relerr(nu_b, nu_t) <= tol32
    gnu = torch.tensor(np.random.default_rng(M).normal(size=(D, M)), dtype=torch.float32, device="cuda")
    g_t = _bwd("tile", Z, ell, var, u, omega, phase, w, L_t, sp_t, gnu)
    g_b = _bwd("blocked", Z, ell, var, u, omega, phase, w, L_b, sp_b, gnu)
    for name, a, b in zip(("u", "Z", "ell", "var"), g_b, g_t):
        assert relerr(a, b) <= tol32, (name, relerr(a, b))


@pytest.mark.parametrize("n", [1, 7, 64])
def test_blocked_whiten_sets_bitwise_per_draw(n):
    """Every column of the blocked solves runs the same operations whatever the number of right-hand sides: a batched
    draw's nu is bitwise the single-draw call's."""
    from gaussian_process_odes_b200 import ops
    D, M, S = 5, 300, 64
    Z, ell, var, u, omega, phase, w = _inputs(D, M, S, seed=n, n_sets=n)
    with torch.no_grad():
        nu = ops.whiten_sets(Z, ell, var, u, omega, phase, w)
        assert nu.shape == (n, D, M)
        for q in range(n):
            nq = ops.whiten(Z, ell, var, u[q], omega[q], phase[q], w[q])
            assert torch.equal(nu[q], nq), "draw %d differs from the single-draw whitening" % q


def test_blocked_backward_is_bitwise_repeatable():
    D, M = 8, 600
    Z, ell, var, u, omega, phase, w = _inputs(D, M, 64, seed=5)
    _, L, sp = _fwd("blocked", Z, ell, var, u, omega, phase, w)
    gnu = torch.tensor(np.random.default_rng(1).normal(size=(D, M)), dtype=torch.float32, device="cuda")
    a = _bwd("blocked", Z, ell, var, u, omega, phase, w, L, sp, gnu)
    b = _bwd("blocked", Z, ell, var, u, omega, phase, w, L, sp, gnu)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def _lattice_problem(monkeypatch):
    """O.make_problem with the inducing points on a lattice of spacing 2 (lengthscales 1.3 +- 10%): the float32
    oracle's own Cholesky of Kzz stays well defined at M = 256 and 512."""
    make = O.make_problem

    def lattice_problem(D, M, *a, **k):
        p, ys, ts, draws, proj = make(D, M, *a, **k)
        p['inducing_loc'] = torch.tensor(_lattice(D, M, 3, spacing=2.0) - 2.0 * (math.ceil(M ** (1 / D)) - 1) / 2,
                                         dtype=p['inducing_loc'].dtype)
        return p, ys, ts, draws, proj

    monkeypatch.setattr(O, "make_problem", lattice_problem)


@pytest.mark.parametrize("kind,solver", [("gpode", "rk4"), ("gpode", "dopri5"), ("shooting", "rk4"),
                                         ("shooting", "dopri5")])
@pytest.mark.parametrize("D,M", [(2, 256), (2, 512), (5, 256), (5, 512)])
def test_models_with_many_inducing_points_match_oracle(kind, solver, D, M, monkeypatch):
    """SequenceModel (kind gpode) and UniformSequenceModel (kind shooting), rk4 and dopri5, above M = 160: ELBO loss
    and every parameter gradient against the oracle port, 1e-4 or float64-arbitrated."""
    from util import elbo_errors
    _lattice_problem(monkeypatch)
    kw = dict(D=D, M=M, S=64, N=2, T=5) if kind == "gpode" else dict(D=D, M=M, S=64, N=2, T=5, S_mc=2)
    rows = elbo_errors(kind, kw, solver, {}, 17 + D)
    for name, (e_cuda64, e_ref64, e_cuda32) in rows.items():
        assert e_cuda32 <= TOL_GRAD or e_cuda64 <= max(TOL_GRAD, 1.5 * e_ref64), (name, e_cuda64, e_ref64, e_cuda32)


def test_shooting_step_at_d8_m1024_matches_oracle(monkeypatch):
    """D = 8, M = 1024: the multiple-shooting step with the blocked whitening and the param_grad contraction."""
    from util import elbo_errors
    _lattice_problem(monkeypatch)
    rows = elbo_errors("shooting", dict(D=8, M=1024, S=64, N=1, T=4, S_mc=2), "rk4", {}, 8)
    for name, (e_cuda64, e_ref64, e_cuda32) in rows.items():
        assert e_cuda32 <= TOL_GRAD or e_cuda64 <= max(TOL_GRAD, 1.5 * e_ref64), (name, e_cuda64, e_ref64, e_cuda32)


def test_graphed_step_at_m512_equals_eager():
    """The blocked whitening inside a CUDA-graph captured training step: one replay gives the eager loss and
    gradients (state-sample noise pinned, same numpy seed)."""
    from gaussian_process_odes_b200 import builders, graphs
    from gaussian_process_odes_b200.core import states
    p, ys, ts, _, _ = O.make_problem(D=2, M=512, S=64, N=2, T=6, seed=4)
    p['inducing_loc'] = torch.tensor(_lattice(2, 512, 4, spacing=2.0) - 22.0, dtype=torch.float32)
    ys_c, ts_c = ys.cuda(), ts.cuda()
    fixed = {}

    def fixed_noise(shape, dtype, device):
        if tuple(shape) not in fixed:
            fixed[tuple(shape)] = torch.randn(shape, dtype=dtype, device=device)
        return fixed[tuple(shape)]

    saved = states._standard_normal
    states._standard_normal = fixed_noise
    try:
        m1 = build_product_model("gpode", p, ys, 64, "rk4")
        np.random.seed(9)
        l1 = builders.compute_loss_gpode(m1, ys_c, ts_c)[0]
        l1.backward()
        m2 = build_product_model("gpode", p, ys, 64, "rk4")
        step = graphs.GraphedStep(m2, lambda: builders.compute_loss_gpode(m2, ys_c, ts_c)[0])
        np.random.seed(9)
        l2 = step()
        torch.cuda.synchronize()
    finally:
        states._standard_normal = saved
    assert relerr(l2, l1) <= 1e-6
    for (n1, p1), (n2, p2) in zip(m1.named_parameters(), m2.named_parameters()):
        if p1.grad is not None:
            assert relerr(p2.grad, p1.grad) <= 1e-5, n1


@pytest.mark.parametrize("solver", ["rk4", "dopri5"])
def test_batched_predictions_at_m512_equal_loop(solver):
    from gaussian_process_odes_b200 import builders
    np.random.seed(3)
    torch.manual_seed(3)
    N, T, D, M = 2, 6, 2, 512
    model = builders.build_gpode(N=N, T=T, D=D, num_inducing=M, num_features=64, solver=solver,
                                 ts_dense_scale=3).cuda()
    with torch.no_grad():
        gp = model.flow.odefunc.diffeq
        gp.inducing_loc.optvar.copy_(torch.tensor(_lattice(D, M, 2, spacing=2.0) - 22.0, dtype=torch.float32))
        gp.Um.optvar.mul_(5.0)
    ts = torch.linspace(0.1, 2.0, T).cuda()
    x0 = torch.randn(N, D, device="cuda")
    np.random.seed(7)
    loop = builders.compute_test_predictions(model, x0, ts, eval_sample_size=5, batched=False)
    np.random.seed(7)
    bat = builders.compute_test_predictions(model, x0, ts, eval_sample_size=5, batched=True)
    assert bat.shape == loop.shape == (5, N, T, D)
    assert relerr(bat, loop) <= 1e-5
    assert relerr(bat[0], bat[1]) > 1e-3


def test_limits_raise_errors():
    """M above GPODE_MAX_M_BLOCKED is an argument error naming the limit; an M whose packed block does not fit the
    integrators' shared memory (D = 8, S = 512, M = 2048) raises the integrators' "does not fit" error."""
    from gaussian_process_odes_b200 import _lib, ops
    from gaussian_process_odes_b200._lib import GpodeError, ptr, stream_ptr
    Z, ell, var, u, omega, phase, w = _inputs(3, 2049, 32, seed=1)
    with pytest.raises(GpodeError, match="2048"):
        ops.whiten(Z, ell, var, u, omega, phase, w)
    st = _struct(Z, ell, var, omega, phase, w)
    nul = ctypes.c_void_p(16)
    assert _lib.load().gpode_whiten_fwd_blocked(ctypes.byref(st), ptr(u), JITTER, nul, nul, nul, nul,
                                                stream_ptr()) < 0
    assert b"GPODE_MAX_M_BLOCKED" in _lib.load().gpode_last_error()
    D, M, S = 8, 2048, 512
    Z, ell, var, u, omega, phase, w = _inputs(D, M, S, seed=2)
    with torch.no_grad():
        nu = ops.whiten(Z, ell, var, u, omega, phase, w)
        assert torch.isfinite(nu).all()
        x0 = torch.zeros(4, D, device="cuda")
        with pytest.raises(GpodeError, match="does not fit"):
            ops.rk4_integrate(x0, torch.linspace(0, 1, 3, device="cuda"), Z, ell, var, nu, omega, phase, w)
