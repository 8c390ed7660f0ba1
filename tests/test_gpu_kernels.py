"""-m gpu: the CUDA kernels, called through the C ABI (ctypes), against the oracle port on the same seeded inputs."""
import numpy as np
import pytest
import torch

import gpode_oracle as O
from util import TOL_GRAD, TOL_TRAJ, TOL_VF, assert_parity, oracle_cache, relerr, to_dev

pytestmark = pytest.mark.gpu

SHAPES = [  # D, M, S
    (2, 16, 256), (5, 100, 256), (1, 8, 32), (3, 24, 64), (4, 33, 100), (6, 20, 48), (7, 17, 40), (8, 100, 256)]


def _setup(D, M, S, B, seed=0, nu_scale=None):
    p, ys, ts, draws, _ = O.make_problem(D=D, M=M, S=S, N=1, T=4, seed=seed)
    gp32, c32 = oracle_cache(p, draws, torch.float32)
    gp64, c64 = oracle_cache(p, draws, torch.float64)
    if nu_scale is not None:  # SURVEY 8d config 5: nu ~ 0.1 N(0,1) supplied directly (skip the whitening)
        nu = torch.tensor(np.random.default_rng(seed + 1).normal(size=(D, M, 1)) * nu_scale, dtype=torch.float32)
        c32['nu'], c64['nu'] = nu, nu.double()
    x = torch.tensor(np.random.default_rng(seed + 2).normal(size=(B, D)) * 1.5, dtype=torch.float32)
    return gp32, c32, gp64, c64, x


def _cuda_args(gp, c):
    d = to_dev(dict(Z=gp['Z'], ell=gp['ell'], var=gp['var'], nu=c['nu'], omega=c['rff_omega'], phase=c['rff_phase'],
                    w=c['rff_weights']))
    return [d[k].float().contiguous() for k in ("Z", "ell", "var", "nu", "omega", "phase", "w")]


@pytest.mark.parametrize("D,M,S", SHAPES)
@pytest.mark.parametrize("B", [1, 37, 5000])
def test_vf_forward(D, M, S, B):
    from gaussian_process_odes_b200 import ops
    gp32, c32, gp64, c64, x = _setup(D, M, S, B, seed=D * 100 + B)
    f = ops.vector_field(x.cuda(), *_cuda_args(gp32, c32)).cpu()
    f32 = O.vf_forward(x, gp32['Z'], gp32['ell'], gp32['var'], c32)
    f64 = O.vf_closed_form(x.double(), gp64['Z'], gp64['ell'], gp64['var'], c32['rff_omega'].double(),
                           c32['rff_phase'].double(), c32['rff_weights'].double(), c32['nu'].double())
    # the reference's own float32 noise for this cache, measured on 4096 probe points
    xp = torch.tensor(np.random.default_rng(99).normal(size=(4096, D)) * 1.5, dtype=torch.float32)
    n32 = O.vf_forward(xp, gp32['Z'], gp32['ell'], gp32['var'], c32)
    n64 = O.vf_closed_form(xp.double(), gp64['Z'], gp64['ell'], gp64['var'], c32['rff_omega'].double(),
                           c32['rff_phase'].double(), c32['rff_weights'].double(), c32['nu'].double())
    # synthetic worst case: random Z and whitened nu give |var nu| ~ 1e2, so every K(x,Z_m) term's round-off (ex2.approx
    # here, the cancelling expanded distance in the reference) is amplified 100x; both sit at ~1e-5 of max|f|. The CUDA
    # value must be within 1e-5 of the float32 reference or at least as close to float64 as the reference's own float32
    # path is (x1.5, the arbiter rule of tests/util.py).
    assert_parity("vf D=%d" % D, f, f32, f64, TOL_VF,
                  ref_noise=relerr(n32, n64) * float(n64.abs().max() / f64.abs().max()))


BIG_SHAPES = [(2, 16, 256), (5, 100, 256), (3, 24, 64), (8, 20, 32)]


@pytest.mark.parametrize("D,M,S", BIG_SHAPES)
@pytest.mark.parametrize("B", [20000, 80000, 160000])
def test_vf_forward_row_per_thread_paths(D, M, S, B):
    """B > 16384 leaves the warp-per-row kernels: one row per thread, then R rows per thread (wide tiles)."""
    from gaussian_process_odes_b200 import ops
    gp32, c32, gp64, c64, x = _setup(D, M, S, B, seed=D + B, nu_scale=0.3)
    f = ops.vector_field(x.cuda(), *_cuda_args(gp32, c32)).cpu()
    f32 = O.vf_forward(x, gp32['Z'], gp32['ell'], gp32['var'], c32)
    assert relerr(f, f32) <= TOL_VF


@pytest.mark.parametrize("D,M,S", BIG_SHAPES)
@pytest.mark.parametrize("B,Tg", [(20000, 3), (80000, 2), (160000, 2)])
def test_rk4_row_per_thread_paths(D, M, S, B, Tg):
    from gaussian_process_odes_b200 import ops
    if D == 8 and B > 80000:
        pytest.skip("oracle memory")
    gp32, c32, gp64, c64, x = _setup(D, M, S, B, seed=D + B, nu_scale=0.3)
    ts = _grid(Tg, 0.1, Tg)
    cot = torch.tensor(np.random.default_rng(9).normal(size=(Tg, B, D)), dtype=torch.float32)
    args = [a.requires_grad_(i < 4) for i, a in enumerate(_cuda_args(gp32, c32))]
    xc = x.cuda().requires_grad_(True)
    xs = ops.rk4_integrate(xc, ts.cuda(), *args)
    xs.backward(cot.cuda())
    got = dict(x=xc.grad, Z=args[0].grad, ell=args[1].grad, var=args[2].grad, nu=args[3].grad)
    out, leaves = _grads_oracle(
        lambda l, cc: O.odeint(lambda t, y: O.vf_forward(y, l['Z'], l['ell'], l['var'], cc), l['x'],
                               ts.to(l['x'].dtype), method='rk4'), gp32, c32, x, torch.float32)
    assert relerr(xs.detach().cpu(), out.detach()) <= TOL_TRAJ
    out.backward(cot)
    g64 = _lazy_f64_grads(
        lambda l, cc: O.odeint(lambda t, y: O.vf_forward(y, l['Z'], l['ell'], l['var'], cc), l['x'],
                               ts.to(l['x'].dtype), method='rk4'), gp32, c32, x, cot)
    for k in got:
        assert_parity("rk4 grad " + k, got[k].cpu().reshape(leaves[k].grad.shape), leaves[k].grad, lambda k=k: g64()[k],
                      TOL_GRAD)


@pytest.mark.parametrize("D,M,S", SHAPES)
def test_vf_forward_moderate_nu_direct(D, M, S):
    """nu ~ 0.1 N(0,1): no cancellation, the CUDA value must match the float32 reference formula directly."""
    from gaussian_process_odes_b200 import ops
    gp32, c32, gp64, c64, x = _setup(D, M, S, 4096, seed=D, nu_scale=0.1)
    f = ops.vector_field(x.cuda(), *_cuda_args(gp32, c32)).cpu()
    f32 = O.vf_forward(x, gp32['Z'], gp32['ell'], gp32['var'], c32)
    assert relerr(f, f32) <= TOL_VF


def _lazy_f64_grads(fn, gp, c, x, cot):
    """-> callable returning the float64 oracle gradients of ``(fn(...) * cot).sum()``; evaluated at most once."""
    memo = {}

    def get():
        if not memo:
            out, leaves = _grads_oracle(fn, gp, c, x, torch.float64)
            out.backward(cot.double())
            memo.update({k: v.grad for k, v in leaves.items()})
        return memo
    return get


def _grads_oracle(fn, gp, c, x, dtype):
    leaves = dict(x=x.to(dtype).clone().requires_grad_(True), Z=gp['Z'].to(dtype).clone().requires_grad_(True),
                  ell=gp['ell'].to(dtype).clone().requires_grad_(True),
                  var=gp['var'].to(dtype).clone().requires_grad_(True),
                  nu=c['nu'].to(dtype).clone().requires_grad_(True))
    # omega = eps / ell must stay attached to ell (kernels.py:110-112): rebuild it from eps
    eps = (c['rff_omega'].double() * gp['ell'].double().T.unsqueeze(1)).to(dtype)
    cc = dict(rff_omega=eps / leaves['ell'].T.unsqueeze(1), rff_phase=c['rff_phase'].to(dtype),
              rff_weights=c['rff_weights'].to(dtype), nu=leaves['nu'])
    out = fn(leaves, cc)
    return out, leaves


@pytest.mark.parametrize("D,M,S", SHAPES)
@pytest.mark.parametrize("B", [3, 700])
def test_vf_backward(D, M, S, B):
    from gaussian_process_odes_b200 import ops
    gp32, c32, gp64, c64, x = _setup(D, M, S, B, seed=D * 7 + B, nu_scale=0.3)
    cot = torch.tensor(np.random.default_rng(5).normal(size=(B, D)), dtype=torch.float32)
    args = [a.requires_grad_(i < 4) for i, a in enumerate(_cuda_args(gp32, c32))]
    xc = x.cuda().requires_grad_(True)
    f = ops.vector_field(xc, *args)
    f.backward(cot.cuda())
    got = dict(x=xc.grad, Z=args[0].grad, ell=args[1].grad, var=args[2].grad, nu=args[3].grad)
    res = {}
    for dtype in (torch.float32, torch.float64):
        out, leaves = _grads_oracle(lambda l, cc: O.vf_forward(l['x'], l['Z'], l['ell'], l['var'], cc), gp32, c32, x,
                                    dtype)
        out.backward(cot.to(dtype))
        res[dtype] = {k: v.grad for k, v in leaves.items()}
    for k in got:
        assert_parity("vf grad %s D=%d" % (k, D), got[k].cpu().reshape(res[torch.float32][k].shape),
                      res[torch.float32][k], res[torch.float64][k], TOL_GRAD)


def _grid(Tg, h, seed):
    rng = np.random.default_rng(seed)
    steps = h * (1 + 0.3 * rng.uniform(-1, 1, size=Tg - 1))
    return torch.tensor(np.concatenate([[0.0], np.cumsum(steps)]), dtype=torch.float32)


@pytest.mark.parametrize("D,M,S", SHAPES)
@pytest.mark.parametrize("B,Tg,h", [(1, 20, 0.1), (130, 2, 0.29), (3000, 5, 0.05)])
def test_rk4_forward(D, M, S, B, Tg, h):
    from gaussian_process_odes_b200 import ops
    gp32, c32, gp64, c64, x = _setup(D, M, S, B, seed=D + Tg, nu_scale=0.3)
    ts = _grid(Tg, h, Tg)
    xs = ops.rk4_integrate(x.cuda(), ts.cuda(), *_cuda_args(gp32, c32)).cpu()
    ref32 = O.odeint(lambda t, y: O.vf_forward(y, gp32['Z'], gp32['ell'], gp32['var'], c32), x, ts, method='rk4')
    c64n = dict(c64, nu=c32['nu'].double())
    ref64 = O.odeint(lambda t, y: O.vf_forward(y, gp64['Z'], gp64['ell'], gp64['var'], c64n), x.double(),
                     ts.double(), method='rk4')
    assert xs.shape == ref32.shape
    assert torch.equal(xs[0], x)
    assert_parity("rk4 D=%d" % D, xs, ref32, ref64, TOL_TRAJ)


def _rbf_umma_m_star(D):
    """The largest M for which large_umma.cu's rbf_smem(D, M) = 128 + 4 (2 ND KD + M KD + 5 KD 128) bytes fits the
    227 KB a CTA may use (KD = D padded to 8, ND = D padded to 16): the tcgen05 RBF forward keeps all of Z in shared
    memory up to M*, and from M* + 1 on the vector field takes the FP32 kernel gpode_vf_fwd_large_add_rbf instead."""
    KD, ND = (D + 7) & ~7, (D + 15) & ~15
    return (227 * 1024 - 128 - 4 * (2 * ND * KD + 5 * KD * 128)) // (4 * KD)


# Shapes at the padding boundaries of the large-D kernels, small B: lb_dp 16|17, 32|33; rv_dn / lu_nd 16|17, 32|33,
# 48|49; lu_nc 40|41; lu_kp at D = 7 mod 8 (the phase slot fills the last K step: 15, 23, 31, 39, 47, 55, 63); S = 1
# and S = 65 above D = 40 (features that fill one chunk of 128 barely or not at all); M = 1; M* and M* + 1.
LARGE_EDGE_SHAPES = [(15, 9, 40, 77), (17, 11, 64, 129), (23, 5, 96, 200), (31, 13, 100, 131), (39, 7, 64, 150),
                     (40, 9, 130, 100), (47, 11, 65, 257), (48, 8, 129, 64), (49, 5, 200, 300), (55, 3, 1, 33),
                     (63, 1, 65, 255), (33, _rbf_umma_m_star(33), 64, 130), (33, _rbf_umma_m_star(33) + 1, 64, 130),
                     (64, _rbf_umma_m_star(64), 64, 129), (64, _rbf_umma_m_star(64) + 1, 64, 129)]


@pytest.mark.parametrize("D,M,S,B", [(16, 100, 256, 1000), (32, 40, 64, 77), (64, 100, 256, 300), (9, 10, 17, 5),
                                      (24, 7, 33, 64), (64, 150, 64, 130), (41, 30, 200, 257)] + LARGE_EDGE_SHAPES)
def test_large_state_dimension_forward(D, M, S, B):
    """8 < D <= 64 (upper half of the scaling sweep): tensor-core forward kernels, same parity bars."""
    from gaussian_process_odes_b200 import ops
    gp32, c32, gp64, c64, x = _setup(D, M, S, B, seed=D, nu_scale=0.1)
    args = _cuda_args(gp32, c32)
    with torch.no_grad():
        f = ops.vector_field(x.cuda(), *args).cpu()
        ts = _grid(4, 0.02, 2)
        xs = ops.rk4_integrate(x.cuda(), ts.cuda(), *args).cpu()
    f32 = O.vf_forward(x, gp32['Z'], gp32['ell'], gp32['var'], c32)
    c64n = dict(c64, nu=c32['nu'].double())
    f64 = O.vf_forward(x.double(), gp64['Z'], gp64['ell'], gp64['var'], c64n)
    # the reference's own float32 noise for this cache on 4096 probe points (the rule of test_vf_forward): a few dozen
    # rows underestimate it. At S = 1 nothing averages the one feature's cos(theta) round-off, |theta| reaches ~30, and
    # at D = 55, M = 3 the float32 reference is 3.1e-6 from float64 on the 33 test rows but 7.3e-6 on the probe points.
    xp = torch.tensor(np.random.default_rng(99).normal(size=(4096, D)) * 1.5, dtype=torch.float32)
    n32 = O.vf_forward(xp, gp32['Z'], gp32['ell'], gp32['var'], c32)
    n64 = O.vf_forward(xp.double(), gp64['Z'], gp64['ell'], gp64['var'], c64n)
    assert_parity("large-D vf", f, f32, f64, TOL_VF,
                  ref_noise=relerr(n32, n64) * float(n64.abs().max() / f64.abs().max()))
    ref32 = O.odeint(lambda t, y: O.vf_forward(y, gp32['Z'], gp32['ell'], gp32['var'], c32), x, ts, method='rk4')
    assert relerr(xs, ref32) <= TOL_TRAJ


@pytest.mark.parametrize("D,M,S,B", [(16, 100, 256, 1000), (32, 40, 64, 77), (64, 100, 256, 300), (9, 10, 17, 5),
                                      (24, 7, 33, 200), (64, 30, 64, 130), (41, 30, 200, 257)] + LARGE_EDGE_SHAPES)
def test_large_state_dimension_backward(D, M, S, B):
    """8 < D <= 64: gradients of the vector field and of a 2-step RK4 solve w.r.t. x, Z, lengthscales, variances and
    nu (gpode_vf_bwd_large / gpode_rk4_bwd_large: device-side adjoint, no host loop) against autograd through the
    oracle (reference src/core/dsvgp.py:124-137,172-197, kernels.py:53-99), float64-arbitrated."""
    from gaussian_process_odes_b200 import ops
    gp32, c32, gp64, c64, x = _setup(D, M, S, B, seed=D + 1, nu_scale=0.1)
    cot = torch.tensor(np.random.default_rng(5).normal(size=(B, D)), dtype=torch.float32)

    def cuda_grads(fn):
        args = [a.detach().clone().requires_grad_(i < 4) for i, a in enumerate(_cuda_args(gp32, c32))]
        xc = x.cuda().requires_grad_(True)
        out = fn(xc, args)
        return out, dict(x=xc.grad, Z=args[0].grad, ell=args[1].grad, var=args[2].grad, nu=args[3].grad), (xc, args)

    # ---- vector field
    args = [a.detach().clone().requires_grad_(i < 4) for i, a in enumerate(_cuda_args(gp32, c32))]
    xc = x.cuda().requires_grad_(True)
    ops.vector_field(xc, *args).backward(cot.cuda())
    got = dict(x=xc.grad, Z=args[0].grad, ell=args[1].grad, var=args[2].grad, nu=args[3].grad)
    fn = lambda l, cc: O.vf_forward(l['x'], l['Z'], l['ell'], l['var'], cc)
    out, leaves = _grads_oracle(fn, gp32, c32, x, torch.float32)
    out.backward(cot)
    g64 = _lazy_f64_grads(fn, gp32, c32, x, cot)
    for k in got:
        assert_parity("large-D vf grad " + k, got[k].cpu().reshape(leaves[k].grad.shape), leaves[k].grad,
                      lambda k=k: g64()[k], TOL_GRAD)
    # ---- RK4, 2 steps
    ts = _grid(3, 0.05, 3)
    cot3 = torch.tensor(np.random.default_rng(6).normal(size=(3, B, D)), dtype=torch.float32)
    args = [a.detach().clone().requires_grad_(i < 4) for i, a in enumerate(_cuda_args(gp32, c32))]
    xc = x.cuda().requires_grad_(True)
    xs = ops.rk4_integrate(xc, ts.cuda(), *args)
    xs.backward(cot3.cuda())
    got = dict(x=xc.grad, Z=args[0].grad, ell=args[1].grad, var=args[2].grad, nu=args[3].grad)
    fn = lambda l, cc: O.odeint(lambda t, y: O.vf_forward(y, l['Z'], l['ell'], l['var'], cc), l['x'],
                                ts.to(l['x'].dtype), method='rk4')
    out, leaves = _grads_oracle(fn, gp32, c32, x, torch.float32)
    assert relerr(xs.detach().cpu(), out.detach()) <= TOL_TRAJ
    out.backward(cot3)
    g64 = _lazy_f64_grads(fn, gp32, c32, x, cot3)
    for k in got:
        assert_parity("large-D rk4 grad " + k, got[k].cpu().reshape(leaves[k].grad.shape), leaves[k].grad,
                      lambda k=k: g64()[k], TOL_GRAD)
    # bitwise reproducible
    args2 = [a.detach().clone().requires_grad_(i < 4) for i, a in enumerate(_cuda_args(gp32, c32))]
    xc2 = x.cuda().requires_grad_(True)
    ops.rk4_integrate(xc2, ts.cuda(), *args2).backward(cot3.cuda())
    assert torch.equal(xc2.grad, xc.grad) and torch.equal(args2[0].grad, args[0].grad)
    assert torch.equal(args2[1].grad, args[1].grad) and torch.equal(args2[3].grad, args[3].grad)


@pytest.mark.parametrize("D,M,S,B", [(16, 100, 256, 300), (33, 20, 64, 40)])
def test_large_state_dimension_dopri5(D, M, S, B):
    """8 < D <= 64: the adaptive solver (device-side controller inside a CUDA-graph while loop around the tensor-core
    vector field, gpode_dopri5_fwd_large) against the restated dopri5; repeated calls are bitwise equal."""
    from gaussian_process_odes_b200 import ops
    gp32, c32, gp64, c64, x = _setup(D, M, S, B, seed=D, nu_scale=0.1)
    args = _cuda_args(gp32, c32)
    ts = torch.tensor([0.0, 0.05, 0.32], dtype=torch.float32)
    with torch.no_grad():
        xs, stats = ops.dopri5_integrate(x.cuda(), ts.cuda(), *args)
        back, _ = ops.dopri5_integrate(xs[-1].contiguous(), torch.flip(ts, [0]).cuda(), *args)
    st = {}
    ref32 = O.odeint(lambda t, y: O.vf_forward(y, gp32['Z'], gp32['ell'], gp32['var'], c32), x, ts, method='dopri5',
                     rtol=1e-6, atol=1e-6, stats=st)
    nfe, acc, rej, status = [int(v) for v in stats.cpu()]
    assert status == 0 and nfe == 2 + 6 * (acc + rej)
    assert abs(acc - st['accepted']) <= 1 and abs(rej - st['rejected']) <= 1
    assert torch.equal(xs[0].cpu(), x)
    assert relerr(xs.cpu(), ref32) <= TOL_TRAJ
    assert relerr(back[-1].cpu(), x) <= TOL_TRAJ  # decreasing grid: integrate back to the start


def test_rk4_decreasing_grid():
    """odeint accepts a decreasing grid (used by initialize_latents_with_data, model_initialization.py:70-73)."""
    from gaussian_process_odes_b200 import ops
    gp32, c32, gp64, c64, x = _setup(2, 16, 256, 10, seed=3, nu_scale=0.3)
    ts = -_grid(9, 0.1, 1)
    xs = ops.rk4_integrate(x.cuda(), ts.cuda(), *_cuda_args(gp32, c32)).cpu()
    ref32 = O.odeint(lambda t, y: O.vf_forward(y, gp32['Z'], gp32['ell'], gp32['var'], c32), x, ts, method='rk4')
    assert relerr(xs, ref32) <= TOL_TRAJ


@pytest.mark.parametrize("D,M,S", SHAPES)
@pytest.mark.parametrize("B,Tg,h", [(2, 12, 0.1), (300, 2, 0.29), (1100, 3, 0.05)])
def test_rk4_backward(D, M, S, B, Tg, h):
    from gaussian_process_odes_b200 import ops
    gp32, c32, gp64, c64, x = _setup(D, M, S, B, seed=D * 3 + Tg, nu_scale=0.3)
    ts = _grid(Tg, h, Tg + 1)
    cot = torch.tensor(np.random.default_rng(9).normal(size=(Tg, B, D)), dtype=torch.float32)
    args = [a.requires_grad_(i < 4) for i, a in enumerate(_cuda_args(gp32, c32))]
    xc = x.cuda().requires_grad_(True)
    xs = ops.rk4_integrate(xc, ts.cuda(), *args)
    xs.backward(cot.cuda())
    got = dict(x=xc.grad, Z=args[0].grad, ell=args[1].grad, var=args[2].grad, nu=args[3].grad)
    res = {}
    for dtype in (torch.float32, torch.float64):
        out, leaves = _grads_oracle(
            lambda l, cc: O.odeint(lambda t, y: O.vf_forward(y, l['Z'], l['ell'], l['var'], cc), l['x'],
                                   ts.to(l['x'].dtype), method='rk4'), gp32, c32, x, dtype)
        out.backward(cot.to(dtype))
        res[dtype] = {k: v.grad for k, v in leaves.items()}
    for k in got:
        assert_parity("rk4 grad %s D=%d" % (k, D), got[k].cpu().reshape(res[torch.float32][k].shape),
                      res[torch.float32][k], res[torch.float64][k], TOL_GRAD)


@pytest.mark.parametrize("D,M,S", [(2, 16, 256), (5, 100, 256), (3, 24, 64), (1, 7, 16), (4, 130, 64)])
def test_whiten_forward_backward(D, M, S):
    from gaussian_process_odes_b200 import ops
    p, ys, ts, draws, _ = O.make_problem(D=D, M=M, S=S, N=1, T=4, seed=40 + D)
    res = {}
    for dtype in (torch.float32, torch.float64):
        gp = O.gp_params(O.cast(p, dtype))
        d = O.cast(draws, dtype)
        leaves = dict(Z=gp['Z'].clone().requires_grad_(True), ell=gp['ell'].clone().requires_grad_(True),
                      var=gp['var'].clone().requires_grad_(True))
        u = O.sample_inducing(gp['Um'], gp['Us_sqrt'], d['eps_u']).clone().requires_grad_(True)
        # restate build_cache with u as a leaf
        omega = d['eps_omega'] / leaves['ell'].T.unsqueeze(1)
        phase = d['phase_u'] * 2 * np.pi
        Ku = O.rbf_K(leaves['Z'], None, leaves['ell'], leaves['var'])
        Lu = torch.linalg.cholesky(Ku + torch.eye(M, dtype=dtype) * O.JITTER)
        up = O.rff_forward(leaves['Z'], omega, phase, d['w'], leaves['var'])
        nu = torch.linalg.solve_triangular(Lu, up.T.unsqueeze(2), upper=False)
        nu = torch.linalg.solve_triangular(Lu.permute(0, 2, 1), u.T.unsqueeze(2) - nu, upper=True)
        # downstream functional that is well conditioned (what the ELBO sees): f at probe points
        xp = torch.tensor(np.random.default_rng(3).normal(size=(50, D)) * 1.5).to(dtype)
        cc = dict(rff_omega=omega, rff_phase=phase, rff_weights=d['w'], nu=nu)
        f = O.vf_forward(xp, leaves['Z'], leaves['ell'], leaves['var'], cc)
        cot = torch.tensor(np.random.default_rng(4).normal(size=(50, D))).to(dtype)
        (f * cot).sum().backward()
        res[dtype] = dict(f=f.detach(), nu=nu.detach(), u=u.grad, **{k: v.grad for k, v in leaves.items()})
        if dtype == torch.float32:
            u32, omega32, phase32 = u.detach(), omega.detach(), phase

    gp = O.gp_params(p)
    Zc, ec, vc = [gp[k].cuda().requires_grad_(True) for k in ("Z", "ell", "var")]
    uc = u32.cuda().requires_grad_(True)
    eps = draws['eps_omega'].cuda()
    omega_c = (eps / ec.T.unsqueeze(1)).detach()
    nu_c = ops.whiten(Zc, ec, vc, uc, omega_c, phase32.float().cuda(), draws['w'].cuda())
    xp = torch.tensor(np.random.default_rng(3).normal(size=(50, D)) * 1.5, dtype=torch.float32).cuda()
    f = ops.vector_field(xp, Zc, ec, vc, nu_c, omega_c, phase32.float().cuda(), draws['w'].cuda())
    cot = torch.tensor(np.random.default_rng(4).normal(size=(50, D)), dtype=torch.float32).cuda()
    (f * cot).sum().backward()
    assert_parity("whiten->f", f.cpu(), res[torch.float32]['f'], res[torch.float64]['f'], TOL_VF)
    got = dict(Z=Zc.grad, ell=ec.grad, var=vc.grad, u=uc.grad)
    for k in got:
        assert_parity("whiten grad " + k, got[k].cpu(), res[torch.float32][k], res[torch.float64][k], TOL_GRAD)
    # nu itself is ill-conditioned (cond(Kzz + 1e-5 I) ~ 1e5): only require float64-arbitrated agreement
    e_c, e_r = relerr(nu_c.cpu().reshape(D, M, 1), res[torch.float64]['nu']), relerr(res[torch.float32]['nu'],
                                                                                   res[torch.float64]['nu'])
    assert e_c <= max(1e-4, 1.5 * e_r), (e_c, e_r)


@pytest.mark.parametrize("D,M", [(2, 16), (5, 100), (3, 7)])
def test_whitened_kl(D, M):
    from gaussian_process_odes_b200 import ops
    p, *_ = O.make_problem(D=D, M=M, S=8, N=1, T=4, seed=60 + D)
    Um = p['Um'].clone().requires_grad_(True)
    Lp = p['Us_sqrt_packed'].clone().requires_grad_(True)
    kl = O.kl_whitened(Um, O.tril_from_packed(Lp, M))
    kl.backward()
    Uc, Lc = p['Um'].cuda().requires_grad_(True), p['Us_sqrt_packed'].cuda().requires_grad_(True)
    klc = ops.whitened_kl(Uc, Lc)
    klc.backward()
    assert relerr(klc.cpu(), kl.detach()) <= 1e-6
    assert relerr(Uc.grad.cpu(), Um.grad) <= 1e-6
    assert relerr(Lc.grad.cpu(), Lp.grad) <= 1e-6


def test_errors_are_loud():
    from gaussian_process_odes_b200 import ops, _lib
    gp32, c32, gp64, c64, x = _setup(2, 16, 32, 4)
    args = _cuda_args(gp32, c32)
    with pytest.raises(_lib.GpodeError):
        ops.vector_field(x, *args)  # CPU tensor: no CPU path
    with pytest.raises(_lib.GpodeError):
        ops.vector_field(x.cuda().double(), *args)
    with pytest.raises(_lib.GpodeError):
        ops.vector_field(torch.zeros(4, 3, device="cuda"), *args)
    # empty batch is legal
    assert ops.vector_field(torch.zeros(0, 2, device="cuda"), *args).shape == (0, 2)


# the tensor-core kernels take over at B >= SMs * 384 rows (56 832 on a B200)
@pytest.mark.parametrize("D,M,S,B", [(5, 100, 256, 60000), (4, 33, 100, 57001), (5, 17, 43, 58000)])
def test_rk4_backward_tensor_core_adjoint(D, M, S, B, monkeypatch):
    """D = 4, 5 and a batch that fills the machine: the adjoint's two Fourier projections run as split-fp16 mma.sync
    (csrc/vjp_mma.cuh). Checked against the oracle's autograd and against the FFMA2 adjoint (GPODE_BWD_MMA=0)."""
    from gaussian_process_odes_b200 import ops, _lib
    gp32, c32, gp64, c64, x = _setup(D, M, S, B, seed=D + B, nu_scale=0.3)
    Tg = 3
    ts = _grid(Tg, 0.1, Tg)
    cot = torch.tensor(np.random.default_rng(9).normal(size=(Tg, B, D)), dtype=torch.float32)

    def run(mode):
        _lib.set_option("bwd_mma", int(mode))
        _lib.set_option("fwd_mma", int(mode))
        args = [a.detach().clone().requires_grad_(i < 4) for i, a in enumerate(_cuda_args(gp32, c32))]
        xc = x.cuda().requires_grad_(True)
        xs = ops.rk4_integrate(xc, ts.cuda(), *args)
        xs.backward(cot.cuda())
        return dict(x=xc.grad, Z=args[0].grad, ell=args[1].grad, var=args[2].grad, nu=args[3].grad)

    try:
        got, base = run("1"), run("0")
    finally:
        _lib.set_option("bwd_mma", 1)
        _lib.set_option("fwd_mma", 1)
    out, leaves = _grads_oracle(
        lambda l, cc: O.odeint(lambda t, y: O.vf_forward(y, l['Z'], l['ell'], l['var'], cc), l['x'],
                               ts.to(l['x'].dtype), method='rk4'), gp32, c32, x, torch.float32)
    out.backward(cot)
    g64 = _lazy_f64_grads(
        lambda l, cc: O.odeint(lambda t, y: O.vf_forward(y, l['Z'], l['ell'], l['var'], cc), l['x'],
                               ts.to(l['x'].dtype), method='rk4'), gp32, c32, x, cot)
    for k in got:
        assert relerr(got[k], base[k]) <= TOL_GRAD, k
        assert_parity("tensor-core rk4 grad " + k, got[k].cpu().reshape(leaves[k].grad.shape), leaves[k].grad,
                      lambda k=k: g64()[k], TOL_GRAD)


@pytest.mark.parametrize("D,M,S,B", [(5, 100, 256, 58000), (4, 16, 40, 57011)])
def test_vf_backward_tensor_core_adjoint(D, M, S, B, monkeypatch):
    from gaussian_process_odes_b200 import ops, _lib
    gp32, c32, gp64, c64, x = _setup(D, M, S, B, seed=D * 7 + B, nu_scale=0.3)
    cot = torch.tensor(np.random.default_rng(5).normal(size=(B, D)), dtype=torch.float32)

    def run(mode):
        _lib.set_option("bwd_mma", int(mode))
        args = [a.detach().clone().requires_grad_(i < 4) for i, a in enumerate(_cuda_args(gp32, c32))]
        xc = x.cuda().requires_grad_(True)
        ops.vector_field(xc, *args).backward(cot.cuda())
        return dict(x=xc.grad, Z=args[0].grad, ell=args[1].grad, var=args[2].grad, nu=args[3].grad)

    try:
        got, base = run("1"), run("0")
    finally:
        _lib.set_option("bwd_mma", 1)
        _lib.set_option("fwd_mma", 1)
    out, leaves = _grads_oracle(lambda l, cc: O.vf_forward(l['x'], l['Z'], l['ell'], l['var'], cc), gp32, c32, x,
                                torch.float32)
    out.backward(cot)
    g64 = _lazy_f64_grads(lambda l, cc: O.vf_forward(l['x'], l['Z'], l['ell'], l['var'], cc), gp32, c32, x, cot)
    for k in got:
        assert relerr(got[k], base[k]) <= TOL_GRAD, k
        assert_parity("tensor-core vf grad " + k, got[k].cpu().reshape(leaves[k].grad.shape), leaves[k].grad,
                      lambda k=k: g64()[k], TOL_GRAD)


@pytest.mark.parametrize("D,M,S,B", [(5, 100, 256, 60000), (4, 33, 100, 57017), (5, 17, 43, 58000)])
def test_forward_tensor_core_path(D, M, S, B, monkeypatch):
    """D = 4, 5 and a batch that fills the machine: theta = x Omega of the forward pass as split-fp16 mma.sync
    (vf_eval_h). Vector field and a 3-step RK4 trajectory against the oracle and against the FFMA2 kernels
    (GPODE_FWD_MMA=0)."""
    from gaussian_process_odes_b200 import ops, _lib
    gp32, c32, gp64, c64, x = _setup(D, M, S, B, seed=D + B, nu_scale=0.3)
    ts = _grid(4, 0.1, 4)

    def run(mode):
        _lib.set_option("fwd_mma", int(mode))
        with torch.no_grad():
            args = _cuda_args(gp32, c32)
            return ops.vector_field(x.cuda(), *args).cpu(), ops.rk4_integrate(x.cuda(), ts.cuda(), *args).cpu()

    try:
        (f1, xs1), (f0, xs0) = run("1"), run("0")
    finally:
        _lib.set_option("fwd_mma", 1)
    f32 = O.vf_forward(x, gp32['Z'], gp32['ell'], gp32['var'], c32)
    out = O.odeint(lambda t, y: O.vf_forward(y, gp32['Z'], gp32['ell'], gp32['var'], c32), x, ts, method='rk4')
    assert relerr(f1, f0) <= TOL_VF and relerr(f1, f32) <= TOL_VF
    assert relerr(xs1, xs0) <= TOL_TRAJ and relerr(xs1, out) <= TOL_TRAJ
    assert torch.equal(xs1[0], x)
    # outside the split-fp16 domain (|x| >= 65504) the tensor-core kernels answer NaN, never a wrong finite number
    if D == 5 and B == 60000:
        xbad = x.clone()
        xbad[7, 2] = 1.0e5
        with torch.no_grad():
            fbad = ops.vector_field(xbad.cuda(), *_cuda_args(gp32, c32)).cpu()
        assert torch.isnan(fbad[7]).any() and torch.isfinite(fbad[:7]).all() and torch.isfinite(fbad[8:]).all()
