"""-m gpu: batched Monte-Carlo prediction (n_sets function draws per launch, SURVEY.md 8f item 3) against
(a) the single-draw product path called once per draw and (b) the oracle, draw by draw."""
import numpy as np
import pytest
import torch

import gpode_oracle as O
from util import TOL_TRAJ, TOL_VF, assert_parity, relerr, to_dev

pytestmark = pytest.mark.gpu


def _draw_sets(D, M, S, n, seed, nu_scale=0.3):
    """shared hyper-parameters + n independent draws; nu supplied directly (whitening is tested on its own)"""
    p, ys, ts, _, _ = O.make_problem(D=D, M=M, S=S, N=1, T=4, seed=seed)
    gp = O.gp_params(O.cast(p, torch.float32))
    rng = np.random.default_rng(seed)
    t = lambda a: torch.tensor(np.asarray(a), dtype=torch.float32)
    eps_omega = t(rng.normal(size=(n, D, S, D)))
    sets = dict(omega=eps_omega / gp['ell'].T.unsqueeze(1), phase=t(rng.uniform(size=(n, S, D))) * 2 * np.pi,
                w=t(rng.normal(size=(n, S, D))), nu=t(rng.normal(size=(n, D, M))) * nu_scale,
                eps_u=t(rng.normal(size=(n, M, D))))
    return gp, sets


def _one(sets, q):
    return [sets[k][q].cuda().contiguous() for k in ("nu", "omega", "phase", "w")]


def _shared(gp):
    return [gp[k].cuda().contiguous() for k in ("Z", "ell", "var")]


@pytest.mark.parametrize("D,M,S,n,N", [(2, 16, 256, 7, 1), (5, 100, 256, 5, 6), (3, 24, 63, 4, 37), (8, 30, 64, 3, 2),
                                       (1, 9, 33, 5, 3), (4, 33, 100, 3, 7), (6, 21, 47, 4, 5), (7, 17, 41, 3, 9)])
def test_vf_sets_matches_per_draw(D, M, S, n, N):
    from gaussian_process_odes_b200 import ops
    gp, sets = _draw_sets(D, M, S, n, seed=D + n)
    x = torch.tensor(np.random.default_rng(3).normal(size=(n, N, D)), dtype=torch.float32).cuda()
    with torch.no_grad():
        f = ops.vector_field_sets(x, *_shared(gp), *[sets[k].cuda() for k in ("nu", "omega", "phase", "w")])
        for q in range(n):
            fq = ops.vector_field(x[q], *_shared(gp), *_one(sets, q))
            assert torch.equal(f[q], fq), "set %d differs from the single-draw kernel" % q
    # and the oracle, for one draw
    c = dict(rff_omega=sets['omega'][1], rff_phase=sets['phase'][1].unsqueeze(0), rff_weights=sets['w'][1],
             nu=sets['nu'][1].unsqueeze(2))
    ref = O.vf_forward(x[1].cpu(), gp['Z'], gp['ell'], gp['var'], c)
    c64 = {k: v.double() for k, v in c.items()}
    ref64 = O.vf_forward(x[1].cpu().double(), gp['Z'].double(), gp['ell'].double(), gp['var'].double(), c64)
    assert_parity("vf_sets", f[1].cpu(), ref, ref64, TOL_VF)


@pytest.mark.parametrize("D,M,S,n", [(2, 16, 256, 9), (5, 100, 256, 4), (3, 130, 64, 3)])
def test_whiten_sets_matches_per_draw(D, M, S, n):
    from gaussian_process_odes_b200 import ops
    gp, sets = _draw_sets(D, M, S, n, seed=11 + D)
    u = (torch.einsum('dnm,smd->snd', gp['Us_sqrt'], sets['eps_u']) + gp['Um']).cuda().contiguous()
    shared = _shared(gp)
    with torch.no_grad():
        nu = ops.whiten_sets(*shared, u, sets['omega'].cuda(), sets['phase'].cuda(), sets['w'].cuda())
        for q in range(n):
            nq = ops.whiten(*shared, u[q], sets['omega'][q].cuda(), sets['phase'][q].cuda().unsqueeze(0),
                            sets['w'][q].cuda())
            # same float64 factor, two solve orders: agreement far below the float32 resolution of nu
            assert relerr(nu[q], nq) <= (1e-6 if M <= 112 else 2e-3), "set %d" % q


@pytest.mark.parametrize("method", ["rk4", "dopri5"])
@pytest.mark.parametrize("D,M,S,n,N", [(2, 16, 256, 6, 1), (5, 100, 256, 3, 6), (3, 24, 64, 4, 11), (1, 9, 33, 5, 3),
                                       (4, 33, 100, 3, 6), (6, 21, 47, 3, 5), (7, 17, 41, 4, 3), (8, 30, 64, 3, 2)])
def test_integrate_sets_matches_per_draw(method, D, M, S, n, N):
    from gaussian_process_odes_b200 import ops
    gp, sets = _draw_sets(D, M, S, n, seed=21 + D)
    x0 = torch.tensor(np.random.default_rng(4).normal(size=(n, N, D)), dtype=torch.float32).cuda()
    ts = torch.linspace(0, 1.0, 9).cuda()
    shared = _shared(gp)
    with torch.no_grad():
        xs, stats = ops.integrate_sets(x0, ts, *shared, *[sets[k].cuda() for k in ("nu", "omega", "phase", "w")],
                                       method=method)
        assert xs.shape == (n, N, 9, D)
        for q in range(n):
            if method == "rk4":
                ref = ops.rk4_integrate(x0[q], ts, *shared, *_one(sets, q)).permute(1, 0, 2)
                assert torch.equal(xs[q], ref), "set %d differs from the single-draw rk4 kernel" % q
            else:
                ref, st = ops.dopri5_integrate(x0[q], ts, *shared, *_one(sets, q))
                # one controller per draw == one odeint call per draw (only the summation order of the error norm differs)
                assert relerr(xs[q], ref.permute(1, 0, 2)) <= 1e-5, "set %d" % q
                a, b = [int(v) for v in stats[q].cpu()], [int(v) for v in st.cpu()]
                assert a[3] == 0 and b[3] == 0 and abs(a[1] - b[1]) <= 1 and a[0] == 2 + 6 * (a[1] + a[2])
    # oracle, one draw
    q = n - 1
    c = dict(rff_omega=sets['omega'][q], rff_phase=sets['phase'][q].unsqueeze(0), rff_weights=sets['w'][q],
             nu=sets['nu'][q].unsqueeze(2))
    f32 = lambda t, y: O.vf_forward(y, gp['Z'], gp['ell'], gp['var'], c)
    c64 = {k: v.double() for k, v in c.items()}
    f64 = lambda t, y: O.vf_forward(y, gp['Z'].double(), gp['ell'].double(), gp['var'].double(), c64)
    ref32 = O.odeint(f32, x0[q].cpu(), ts.cpu(), method=method)
    ref64 = O.odeint(f64, x0[q].cpu().double(), ts.cpu().double(), method=method, rtol=1e-9, atol=1e-9)
    assert_parity("integrate_sets", xs[q].permute(1, 0, 2).cpu(), ref32, ref64, max(TOL_TRAJ, 2e-5))


def test_sets_are_forward_only_and_validate_shapes():
    from gaussian_process_odes_b200 import ops
    from gaussian_process_odes_b200._lib import GpodeError
    gp, sets = _draw_sets(2, 16, 64, 3, seed=1)
    x0 = torch.zeros(3, 2, 2, device="cuda")
    args = _shared(gp) + [sets[k].cuda() for k in ("nu", "omega", "phase", "w")]
    with pytest.raises(GpodeError):
        ops.integrate_sets(x0.requires_grad_(), torch.linspace(0, 1, 3).cuda(), *args)
    with torch.no_grad():
        with pytest.raises(GpodeError):
            ops.integrate_sets(x0[:2].detach(), torch.linspace(0, 1, 3).cuda(), *args)
        with pytest.raises(GpodeError):
            ops.integrate_sets(x0.detach(), torch.linspace(0, 1, 3).cuda(), *args, method="euler")


@pytest.mark.parametrize("kind,solver", [("gpode", "dopri5"), ("gpode", "rk4"), ("shooting", "rk4")])
def test_compute_test_predictions_batched_equals_loop(kind, solver):
    """Same numpy seed -> the batched path consumes the host generator in the loop's order and returns the loop's
    trajectories (reference compute_test_predictions, src/gpode/model_builder.py:81-96)."""
    from gaussian_process_odes_b200 import builders
    np.random.seed(3)
    torch.manual_seed(3)
    N, T, D = 3, 8, 2
    build = builders.build_gpode if kind == "gpode" else builders.build_gpode_shooting
    model = build(N=N, T=T, D=D, num_inducing=16, num_features=64, solver=solver, ts_dense_scale=3).cuda()
    with torch.no_grad():
        model.flow.odefunc.diffeq.Um.optvar.mul_(5.0)
    ts = torch.linspace(0.1, 2.0, T).cuda()
    x0 = torch.randn(N, D, device="cuda")
    np.random.seed(7)
    loop = builders.compute_test_predictions(model, x0, ts, eval_sample_size=5, batched=False)
    np.random.seed(7)
    bat = builders.compute_test_predictions(model, x0, ts, eval_sample_size=5, batched=True)
    assert bat.shape == loop.shape == (5, N, T, D)
    assert relerr(bat, loop) <= 1e-5
    # different draws really are different functions
    assert relerr(bat[0], bat[1]) > 1e-3
    dev = builders.compute_test_predictions(model, x0, ts, eval_sample_size=4, rng="device")
    assert dev.shape == (4, N, T, D) and torch.isfinite(dev).all()
    pred = builders.compute_predictions(model, ts, eval_sample_size=6)
    assert pred.shape == (6, N, T, D) and torch.isfinite(pred).all()
