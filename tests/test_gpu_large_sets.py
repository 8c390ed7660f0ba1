"""-m gpu: batched Monte-Carlo prediction for 8 < D <= 64 (n_sets function draws per launch on the large-D kernels)
against the single-draw product path called once per draw -- bitwise, since every row sees the same arithmetic -- and
against the oracle for one draw."""
import numpy as np
import pytest
import torch

import gpode_oracle as O
from util import TOL_TRAJ, TOL_VF, assert_parity, relerr

pytestmark = pytest.mark.gpu

KEYS = ("nu", "omega", "phase", "w")


def _draw_sets(D, M, S, n, seed, nu_scale=0.1):
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
    return [sets[k][q].cuda().contiguous() for k in KEYS]


def _all(sets):
    return [sets[k].cuda() for k in KEYS]


def _shared(gp):
    return [gp[k].cuda().contiguous() for k in ("Z", "ell", "var")]


def _oracle_cache(sets, q):
    return dict(rff_omega=sets['omega'][q], rff_phase=sets['phase'][q].unsqueeze(0), rff_weights=sets['w'][q],
                nu=sets['nu'][q].unsqueeze(2))


# (16,100,256,5,129): a ragged second tile per draw; (64,150,64,2,5): Z does not fit the tcgen05 RBF kernel's shared
# memory, so the FP32 RBF kernel runs
@pytest.mark.parametrize("D,M,S,n,N", [(9, 16, 64, 3, 1), (16, 100, 256, 5, 129), (33, 40, 100, 4, 7),
                                       (64, 30, 256, 3, 2), (64, 150, 64, 2, 5)])
def test_vf_large_sets_matches_per_draw(D, M, S, n, N):
    from gaussian_process_odes_b200 import ops
    gp, sets = _draw_sets(D, M, S, n, seed=D + n)
    x = torch.tensor(np.random.default_rng(3).normal(size=(n, N, D)), dtype=torch.float32).cuda()
    with torch.no_grad():
        f = ops.vector_field_sets(x, *_shared(gp), *_all(sets))
        for q in range(n):
            fq = ops.vector_field(x[q], *_shared(gp), *_one(sets, q))
            assert torch.equal(f[q], fq), "draw %d differs from the single-draw kernels" % q
    c = _oracle_cache(sets, 1)
    ref = O.vf_forward(x[1].cpu(), gp['Z'], gp['ell'], gp['var'], c)
    c64 = {k: v.double() for k, v in c.items()}
    ref64 = O.vf_forward(x[1].cpu().double(), gp['Z'].double(), gp['ell'].double(), gp['var'].double(), c64)
    assert_parity("vf_large_sets", f[1].cpu(), ref, ref64, TOL_VF)


@pytest.mark.parametrize("D,M,S,n,N", [(12, 30, 64, 4, 3), (33, 40, 100, 3, 130), (64, 150, 64, 2, 5)])
def test_rk4_large_sets_matches_per_draw(D, M, S, n, N):
    from gaussian_process_odes_b200 import ops
    gp, sets = _draw_sets(D, M, S, n, seed=31 + D)
    x0 = torch.tensor(np.random.default_rng(4).normal(size=(n, N, D)), dtype=torch.float32).cuda()
    ts = torch.linspace(0, 0.5, 6).cuda()
    shared = _shared(gp)
    with torch.no_grad():
        xs, stats = ops.integrate_sets(x0, ts, *shared, *_all(sets), method="rk4")
        assert xs.shape == (n, N, 6, D) and stats is None
        for q in range(n):
            ref = ops.rk4_integrate(x0[q], ts, *shared, *_one(sets, q)).permute(1, 0, 2)
            assert torch.equal(xs[q], ref), "draw %d differs from the single-draw rk4" % q


@pytest.mark.parametrize("D,M,S,n,N", [(12, 30, 64, 4, 3), (33, 40, 100, 3, 130), (64, 150, 64, 2, 5)])
def test_dopri5_large_sets_bitwise_per_draw(D, M, S, n, N):
    """One controller per draw: draw q's trajectories and stats are bitwise those of the single-draw dopri5 -- on an
    increasing grid and on the decreasing grid of the initialisation's backward-in-time solve."""
    from gaussian_process_odes_b200 import ops
    gp, sets = _draw_sets(D, M, S, n, seed=41 + D)
    # states near the inducing points, where the RBF term is large, and nu scaled per draw: the controllers diverge
    sets['nu'] = sets['nu'] * torch.tensor([1.0, 30.0, 100.0, 10.0][:n]).reshape(n, 1, 1)
    noise = torch.tensor(np.random.default_rng(5).normal(size=(n, N, D)), dtype=torch.float32)
    x0 = (gp['Z'][torch.arange(n * N) % M].reshape(n, N, D) + 0.1 * noise).cuda()
    shared = _shared(gp)
    for ts in (torch.tensor([0.0, 0.1, 0.35, 0.5]).cuda(), torch.tensor([0.5, 0.2, 0.0]).cuda()):
        with torch.no_grad():
            xs, stats = ops.integrate_sets(x0, ts, *shared, *_all(sets), method="dopri5")
            counts = set()
            for q in range(n):
                ref, st = ops.dopri5_integrate(x0[q], ts, *shared, *_one(sets, q))
                assert torch.equal(xs[q], ref.permute(1, 0, 2)), "draw %d differs from the single-draw dopri5" % q
                assert torch.equal(stats[q], st), (q, stats[q].tolist(), st.tolist())
                nfe, acc, rej, status = stats[q].tolist()
                assert status == 0 and nfe == 2 + 6 * (acc + rej)
                counts.add((acc, rej))
        assert len(counts) >= 2, "the draws' controllers took the same steps: %s" % counts
    q = 0
    c = _oracle_cache(sets, q)
    ts = torch.tensor([0.0, 0.1, 0.35, 0.5])
    with torch.no_grad():
        xs, _ = ops.integrate_sets(x0, ts.cuda(), *shared, *_all(sets), method="dopri5")
    f32 = lambda t, y: O.vf_forward(y, gp['Z'], gp['ell'], gp['var'], c)
    c64 = {k: v.double() for k, v in c.items()}
    f64 = lambda t, y: O.vf_forward(y, gp['Z'].double(), gp['ell'].double(), gp['var'].double(), c64)
    ref32 = O.odeint(f32, x0[q].cpu(), ts, method="dopri5")
    ref64 = lambda: O.odeint(f64, x0[q].cpu().double(), ts.double(), method="dopri5", rtol=1e-9, atol=1e-9)
    assert_parity("dopri5_large_sets", xs[q].permute(1, 0, 2).cpu(), ref32, ref64, max(TOL_TRAJ, 2e-5))


@pytest.mark.parametrize("D,M,S,n", [(12, 30, 64, 5), (64, 100, 256, 3)])
def test_whiten_large_sets_matches_per_draw(D, M, S, n):
    from gaussian_process_odes_b200 import ops
    gp, sets = _draw_sets(D, M, S, n, seed=11 + D)
    u = (torch.einsum('dnm,smd->snd', gp['Us_sqrt'], sets['eps_u']) + gp['Um']).cuda().contiguous()
    shared = _shared(gp)
    with torch.no_grad():
        nu = ops.whiten_sets(*shared, u, sets['omega'].cuda(), sets['phase'].cuda(), sets['w'].cuda())
        assert nu.shape == (n, D, M)
        for q in range(n):
            nq = ops.whiten(*shared, u[q], sets['omega'][q].cuda(), sets['phase'][q].cuda().unsqueeze(0),
                            sets['w'][q].cuda())
            assert relerr(nu[q], nq) <= 1e-6, "draw %d" % q


@pytest.mark.parametrize("kind,D,solver", [("gpode", 12, "dopri5"), ("gpode", 12, "rk4"), ("shooting", 17, "rk4")])
def test_compute_test_predictions_large_d_batched_equals_loop(kind, D, solver):
    """Same numpy seed -> the batched path draws the loop's functions and returns the loop's trajectories."""
    from gaussian_process_odes_b200 import builders
    np.random.seed(3)
    torch.manual_seed(3)
    N, T = 3, 6
    build = builders.build_gpode if kind == "gpode" else builders.build_gpode_shooting
    model = build(N=N, T=T, D=D, num_inducing=16, num_features=64, solver=solver, ts_dense_scale=3).cuda()
    with torch.no_grad():
        model.flow.odefunc.diffeq.Um.optvar.mul_(5.0)
    ts = torch.linspace(0.1, 1.0, T).cuda()
    x0 = torch.randn(N, D, device="cuda")
    np.random.seed(7)
    loop = builders.compute_test_predictions(model, x0, ts, eval_sample_size=4, batched=False)
    np.random.seed(7)
    bat = builders.compute_test_predictions(model, x0, ts, eval_sample_size=4, batched=True)
    assert bat.shape == loop.shape == (4, N, T, D)
    assert relerr(bat, loop) <= 1e-5
    assert relerr(bat[0], bat[1]) > 1e-3


def test_predictions_and_initialisation_run_above_eight_dimensions():
    from gaussian_process_odes_b200 import builders, initialization
    np.random.seed(5)
    torch.manual_seed(5)
    N, T, D = 2, 5, 12
    model = builders.build_gpode(N=N, T=T, D=D, num_inducing=16, num_features=64).cuda()
    ts = np.linspace(0.1, 1.0, T).astype(np.float32)
    pred = builders.compute_predictions(model, torch.tensor(ts).cuda(), eval_sample_size=6)
    assert pred.shape == (6, N, T, D) and torch.isfinite(pred).all()
    ys = np.random.default_rng(2).normal(size=(N, T, D)).astype(np.float32)
    x0 = initialization.initial_state_from_data(model, ys[:, 0], ts, num_samples=8)
    assert x0.shape == (N, D) and torch.isfinite(x0).all()
    initialization.initialize_latents_with_data(model, ys, ts)
    assert torch.isfinite(model.x0_distribution.sample(num_samples=1)).all()


def test_large_sets_errors_and_empty_draws():
    from gaussian_process_odes_b200 import ops
    from gaussian_process_odes_b200._lib import GpodeError
    D, M, S, n = 65, 4, 8, 2
    big = [torch.rand(M, D), torch.rand(D, D) + 0.5, torch.rand(D), torch.rand(n, D, M), torch.rand(n, D, S, D),
           torch.rand(n, S, D), torch.rand(n, S, D)]
    with torch.no_grad(), pytest.raises(GpodeError):
        ops.vector_field_sets(torch.zeros(n, 1, D, device="cuda"), *[a.cuda() for a in big])
    gp, sets = _draw_sets(12, 16, 64, 3, seed=2)
    args = _shared(gp) + _all(sets)
    ts = torch.linspace(0, 0.2, 3).cuda()
    with pytest.raises(GpodeError):
        ops.integrate_sets(torch.zeros(3, 2, 12, device="cuda", requires_grad=True), ts, *args)
    with pytest.raises(GpodeError):
        ops.vector_field_sets(torch.zeros(3, 2, 12, device="cuda", requires_grad=True), *args)
    with torch.no_grad():
        x0 = torch.zeros(3, 0, 12, device="cuda")
        assert ops.vector_field_sets(x0, *args).shape == (3, 0, 12)
        xs, _ = ops.integrate_sets(x0, ts, *args, method="rk4")
        assert xs.shape == (3, 0, 3, 12)
        xs, stats = ops.integrate_sets(x0, ts, *args, method="dopri5")
        assert xs.shape == (3, 0, 3, 12) and torch.equal(stats.cpu(), torch.zeros(3, 4, dtype=torch.int32))
