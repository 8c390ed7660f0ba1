"""-m gpu: differentiable dopri5 for 8 < D <= 64 (gpode_dopri5_fwd_large_ckpt records the accepted steps,
gpode_dopri5_bwd_large runs their discrete adjoint on the large-D VJP kernels) against autograd through the restated
torchdiffeq 0.2.0 dopri5, float64-arbitrated."""
import ctypes

import numpy as np
import pytest
import torch

import gpode_oracle as O
from util import TOL_GRAD, assert_parity, oracle_cache, to_dev

pytestmark = pytest.mark.gpu

SHAPES = [(9, 10, 17, 5), (16, 100, 256, 300), (33, 20, 64, 40), (64, 30, 64, 130)]
GRIDS = {"span": [0.0, 0.05, 0.32], "inside": [0.0, 0.01, 0.02, 0.05], "decreasing": [0.0, -0.2, -0.5]}


def _setup(D, M, S, B, seed):
    p, ys, ts, draws, _ = O.make_problem(D=D, M=M, S=S, N=1, T=4, seed=seed)
    gp, c = oracle_cache(p, draws, torch.float32)
    c['nu'] = torch.tensor(np.random.default_rng(seed + 1).normal(size=(D, M, 1)) * 0.1, dtype=torch.float32)
    x = torch.tensor(np.random.default_rng(seed + 2).normal(size=(B, D)) * 1.5, dtype=torch.float32)
    return gp, c, x


def _cuda_args(gp, c, grad):
    d = to_dev(dict(Z=gp['Z'], ell=gp['ell'], var=gp['var'], nu=c['nu'], omega=c['rff_omega'], phase=c['rff_phase'],
                    w=c['rff_weights']))
    return [d[k].float().contiguous().requires_grad_(grad and i < 4)
            for i, k in enumerate(("Z", "ell", "var", "nu", "omega", "phase", "w"))]


def _cuda_grads(gp, c, x, ts, cot, tol=1e-6):
    from gaussian_process_odes_b200 import ops
    args = _cuda_args(gp, c, True)
    xc = x.cuda().requires_grad_(True)
    xs, stats = ops.dopri5_integrate(xc, ts.cuda(), *args, rtol=tol, atol=tol)
    (xs * cot.cuda()).sum().backward()
    g = dict(x=xc.grad, Z=args[0].grad, ell=args[1].grad, var=args[2].grad, nu=args[3].grad)
    return xs.detach(), stats, {k: v.detach().cpu() for k, v in g.items()}


def _oracle_grads(gp, c, x, ts, cot, dtype, tol=1e-6):
    leaves = dict(x=x.to(dtype).clone().requires_grad_(True), Z=gp['Z'].to(dtype).clone().requires_grad_(True),
                  ell=gp['ell'].to(dtype).clone().requires_grad_(True),
                  var=gp['var'].to(dtype).clone().requires_grad_(True),
                  nu=c['nu'].to(dtype).clone().requires_grad_(True))
    # omega = eps / ell stays attached to ell (kernels.py:110-112): rebuild it from eps
    eps = (c['rff_omega'].double() * gp['ell'].double().T.unsqueeze(1)).to(dtype)
    cc = dict(rff_omega=eps / leaves['ell'].T.unsqueeze(1), rff_phase=c['rff_phase'].to(dtype),
              rff_weights=c['rff_weights'].to(dtype), nu=leaves['nu'])
    out = O.odeint(lambda t, y: O.vf_forward(y, leaves['Z'], leaves['ell'], leaves['var'], cc), leaves['x'],
                   ts.to(dtype), method='dopri5', rtol=tol, atol=tol)
    (out * cot.to(dtype)).sum().backward()
    return {k: v.grad.detach() for k, v in leaves.items()}


def _assert_grads_match(name, got, gp, c, x, ts, cot, tol=1e-6):
    ref32 = _oracle_grads(gp, c, x, ts, cot, torch.float32, tol)
    memo = {}

    def f64():
        if not memo:
            memo.update(_oracle_grads(gp, c, x, ts, cot, torch.float64, tol))
        return memo
    for k in got:
        # both are exact gradients of a discrete solve; they may differ by one accept/reject decision
        assert_parity("%s grad %s" % (name, k), got[k].reshape(ref32[k].shape), ref32[k], lambda k=k: f64()[k], 2e-4)


@pytest.mark.parametrize("grid", sorted(GRIDS))
@pytest.mark.parametrize("D,M,S,B", SHAPES)
def test_large_dopri5_gradients_match_oracle(D, M, S, B, grid):
    gp, c, x = _setup(D, M, S, B, seed=D + B)
    ts = torch.tensor(GRIDS[grid], dtype=torch.float32)
    cot = torch.tensor(np.random.default_rng(7).normal(size=(len(ts), B, D)), dtype=torch.float32)
    xs, stats, got = _cuda_grads(gp, c, x, ts, cot)
    assert int(stats[3]) == 0
    _assert_grads_match("D=%d %s" % (D, grid), got, gp, c, x, ts, cot)


def test_single_output_time_passes_the_cotangent_through():
    """Tg = 1: xs = x0, so grad_x0 is the incoming cotangent and every parameter gradient is zero."""
    gp, c, x = _setup(16, 100, 256, 300, seed=2)
    ts = torch.tensor([0.3], dtype=torch.float32)
    cot = torch.tensor(np.random.default_rng(1).normal(size=(1, 300, 16)), dtype=torch.float32)
    xs, stats, got = _cuda_grads(gp, c, x, ts, cot)
    assert torch.equal(xs[0].cpu(), x)
    assert torch.equal(got['x'], cot[0])
    for k in ("Z", "ell", "var", "nu"):
        assert bool((got[k] == 0).all()), k


@pytest.mark.parametrize("D,M,S,B", [(16, 100, 256, 300), (64, 30, 64, 130)])
def test_checkpointing_forward_is_bitwise_the_inference_forward_and_backward_is_deterministic(D, M, S, B):
    from gaussian_process_odes_b200 import ops
    gp, c, x = _setup(D, M, S, B, seed=D)
    ts = torch.tensor([0.0, 0.05, 0.32], dtype=torch.float32)
    cot = torch.tensor(np.random.default_rng(4).normal(size=(3, B, D)), dtype=torch.float32)
    with torch.no_grad():
        xs0, st0 = ops.dopri5_integrate(x.cuda(), ts.cuda(), *_cuda_args(gp, c, False))
    xs1, st1, g1 = _cuda_grads(gp, c, x, ts, cot)
    xs2, st2, g2 = _cuda_grads(gp, c, x, ts, cot)
    assert torch.equal(xs1, xs0) and torch.equal(st1, st0)
    assert torch.equal(xs2, xs0) and torch.equal(st2, st0)
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k


def _long_grid(gp, c, x, tol, min_steps):
    """The shortest of the horizons 0.5, 1, 2, ... whose solve needs more than ``min_steps`` accepted steps (counted by
    the float32 oracle). Short enough that the CUDA and oracle solves take the same steps up to one decision: over
    much longer horizons at tight tolerances a single extra rejection changes the step sequence, and with it the
    discrete solve whose gradient is compared."""
    T = 0.5
    while True:
        ts = torch.tensor([0.0, T / 3, T], dtype=torch.float32)
        st = {}
        with torch.no_grad():
            O.odeint(lambda t, y: O.vf_forward(y, gp['Z'], gp['ell'], gp['var'], c), x, ts, method='dopri5', rtol=tol,
                     atol=tol, stats=st)
        if st['accepted'] > min_steps or T >= 64:
            return ts, st['accepted']
        T *= 2


def test_checkpoint_capacity():
    """More accepted steps than the checkpoint capacity: the ckpt forward reports status 3 after `cap` accepted steps,
    and ops retries with a doubled capacity until the solve fits -- the gradients still match the oracle."""
    from gaussian_process_odes_b200 import ops, _lib
    from gaussian_process_odes_b200._lib import ptr, stream_ptr
    D, M, S, B, tol = 9, 10, 17, 5, 1e-8
    gp, c, x = _setup(D, M, S, B, seed=11)
    ts, n_oracle = _long_grid(gp, c, x, tol, 32)
    assert n_oracle > 32   # more than the initial capacity max(32, 4 Tg)
    # direct call, cap = 2
    lib = _lib.load()
    args = _cuda_args(gp, c, False)
    field = ops.LargeField(*args)
    xc, t64, xs, work, stats = ops._dopri5_large_setup(field, x.cuda(), ts.cuda())
    cap = 2
    ckpt = torch.empty(lib.gpode_dopri5_ckpt_floats(D, B, len(ts), cap), dtype=torch.float32, device="cuda")
    _lib.call("gpode_dopri5_fwd_large_ckpt", ptr(field.packed), ctypes.byref(field.struct), ptr(xc), ptr(t64), len(ts),
              B, tol, tol, ptr(xs), ptr(work), ptr(stats), 100000, ptr(ckpt), cap, stream_ptr())
    st = [int(v) for v in stats.cpu()]
    assert st[3] == 3 and st[1] == cap, st
    # through ops: the capacity grows until every accepted step is recorded
    cot = torch.tensor(np.random.default_rng(8).normal(size=(len(ts), B, D)), dtype=torch.float32)
    _, stats, got = _cuda_grads(gp, c, x, ts, cot, tol)
    st = [int(v) for v in stats.cpu()]
    assert st[3] == 0 and st[1] > 32, st
    _assert_grads_match("long horizon", got, gp, c, x, ts, cot, tol)


@pytest.mark.parametrize("kind,kw", [
    ("gpode", dict(D=12, M=20, S=64, N=2, T=8, D_obs=12)),
    ("shooting", dict(D=17, M=24, S=96, N=2, T=6, S_mc=3, D_obs=17)),
])
def test_models_above_eight_state_dimensions_train_with_dopri5(kind, kw):
    """SequenceModel / UniformSequenceModel with the reference's default solver at D = 12 / 17: ELBO loss and every
    parameter gradient against the oracle port, float64-arbitrated (the rule of the rk4 test of test_gpu_models)."""
    from util import elbo_errors
    rows = elbo_errors(kind, kw, "dopri5", {}, 31)
    for name, (e_cuda64, e_ref64, e_cuda32) in rows.items():
        assert e_cuda32 <= TOL_GRAD or e_cuda64 <= max(TOL_GRAD, 1.5 * e_ref64), (name, e_cuda64, e_ref64, e_cuda32)
