"""-m gpu: the fused multiple-shooting step (ops.shooting_step: RK4 interval + observation log-likelihood + shooting
constraint in ONE kernel, adjoint seeded from the in-kernel gradients; SURVEY.md section 8f item 2) against the unfused
chain of launches (which the golden tests of round 1 pinned to the reference) and against the oracle, on every kernel
mapping (warp-per-row, row-per-thread, R rows per thread, tensor-core), with both constraint families, and under
segment-row sharding."""
import numpy as np
import pytest
import torch

import gpode_oracle as O
from util import TOL_GRAD, build_product_model, elbo_errors, injected_draws, product_grads, relerr

pytestmark = pytest.mark.gpu


def _run(p, ys, ts, draws, proj, kw, fuse, row_shard=None, world=1, constraint=None, time_shard=None):
    model = build_product_model("shooting", p, ys, kw['S'], "rk4", proj=None if proj is None else proj.components)
    if constraint is not None:
        from gaussian_process_odes_b200.core import constraints
        model.constraint = constraints.Laplace(d=1, scale=constraint, requires_grad=False).cuda()
    model.fuse_elbo = fuse
    model.row_shard = row_shard
    model.time_shard = time_shard
    with injected_draws(draws, mvn_order=("eps_x0", "eps_states")):
        ll, c, e, k0 = model.build_lowerbound_terms(ys.cuda(), ts.cuda(), num_samples=kw['S_mc'])
        kl = model.build_inducing_kl()
        if time_shard is not None:   # the entropy is this rank's share, only the two KL terms are replicated
            loss = -(ll + c + e - (k0 + kl) / float(world))
        else:
            loss = -(ll + c + (e - k0 - kl) / float(world))
    loss.backward()
    g = {k: (None if v is None else v.detach().clone()) for k, v in product_grads(model, "shooting").items()}
    return loss.detach(), dict(ll=ll.detach(), c=c.detach()), g, model


CASES = [
    # warp-per-row kernels
    dict(D=2, M=16, S=256, N=1, T=25, S_mc=5),
    dict(D=5, M=100, S=256, N=2, T=20, S_mc=3, D_obs=50, dt=0.01, ell0=1.25),
    dict(D=3, M=24, S=64, N=2, T=7, S_mc=2),
    # one row per thread (B = 18 000), R rows per thread (B = 160 000 at D = 2: R = 4)
    dict(D=3, M=24, S=64, N=3, T=3000, S_mc=2, D_obs=7, dt=0.01),
    dict(D=2, M=16, S=64, N=4, T=10000, S_mc=4, dt=0.01),
    # tensor-core kernels (D = 5, B >= 56 832)
    dict(D=5, M=100, S=256, N=2, T=6000, S_mc=5, D_obs=50, dt=0.01, ell0=1.25),
    # the other state dimensions, warp per row
    dict(D=1, M=9, S=33, N=2, T=9, S_mc=3),
    dict(D=4, M=33, S=100, N=2, T=13, S_mc=2),
    dict(D=6, M=21, S=47, N=1, T=17, S_mc=3),
    dict(D=7, M=17, S=41, N=2, T=6, S_mc=2, D_obs=9),
    dict(D=8, M=30, S=64, N=2, T=5, S_mc=3),
    # ... and one row per thread: just above 16 384 rows, below the wide and the tensor-core kernels
    dict(D=1, M=9, S=33, N=3, T=2731, S_mc=2, dt=0.01),
    dict(D=4, M=33, S=100, N=3, T=3001, S_mc=2, dt=0.01),
    dict(D=6, M=21, S=47, N=2, T=4201, S_mc=2, dt=0.01),
    dict(D=7, M=17, S=41, N=3, T=3001, S_mc=2, D_obs=9, dt=0.01),
    dict(D=8, M=30, S=64, N=3, T=3001, S_mc=2, dt=0.01),
]


@pytest.mark.parametrize("kw", CASES, ids=lambda k: "D%d_B%d" % (k['D'], k['S_mc'] * k['N'] * k['T']))
def test_fused_step_matches_unfused_chain(kw):
    p, ys, ts, draws, proj = O.make_problem(seed=5, **kw)
    l1, t1, g1, m1 = _run(p, ys, ts, draws, proj, kw, fuse=True)
    l0, t0, g0, m0 = _run(p, ys, ts, draws, proj, kw, fuse=False)
    assert m1.flow.num_evals() == m0.flow.num_evals() == 4
    assert relerr(l1, l0) <= 1e-5
    for k in t1:
        assert relerr(t1[k], t0[k]) <= 1e-5, k
    for k in g1:
        assert relerr(g1[k], g0[k]) <= TOL_GRAD, (k, relerr(g1[k], g0[k]))


def test_fused_step_with_laplace_constraint():
    kw = dict(D=2, M=16, S=64, N=2, T=30, S_mc=3)
    p, ys, ts, draws, proj = O.make_problem(seed=6, **kw)
    l1, t1, g1, _ = _run(p, ys, ts, draws, proj, kw, fuse=True, constraint=0.05)
    l0, t0, g0, _ = _run(p, ys, ts, draws, proj, kw, fuse=False, constraint=0.05)
    assert relerr(l1, l0) <= 1e-5 and relerr(t1['c'], t0['c']) <= 1e-5
    for k in g1:
        assert relerr(g1[k], g0[k]) <= TOL_GRAD, (k, relerr(g1[k], g0[k]))


@pytest.mark.parametrize("kw,world", [(CASES[0], 3), (CASES[1], 8), (CASES[3], 2)],
                         ids=["vdp_w3", "mocap09_w8", "rows18000_w2"])
def test_row_sharded_terms_and_gradients_add_up(kw, world):
    """Segment-row sharding (distributed.enable_row_sharding): the shares of ``world`` ranks -- run one after the other
    here -- add up to the unsharded loss and gradients. Blocks cut through Monte-Carlo samples, sequences and time; the
    constraint's neighbour state of a block's last row is the halo."""
    p, ys, ts, draws, proj = O.make_problem(seed=7, **kw)
    l_all, _, g_all, _ = _run(p, ys, ts, draws, proj, kw, fuse=True)
    l_sum, g_sum = 0.0, None
    for r in range(world):
        l, _, g, _ = _run(p, ys, ts, draws, proj, kw, fuse=True, row_shard=(r, world), world=world)
        l_sum = l_sum + l.double()
        g_sum = {k: v.double() for k, v in g.items()} if g_sum is None else {k: g_sum[k] + g[k].double() for k in g}
    assert relerr(l_sum, l_all) <= 1e-6
    for k in g_all:
        assert relerr(g_sum[k], g_all[k]) <= 2e-5, (k, relerr(g_sum[k], g_all[k]))


@pytest.mark.parametrize("kw,world", [(CASES[0], 3), (CASES[0], 8), (CASES[1], 4), (CASES[3], 2), (CASES[2], 16)],
                         ids=["vdp_w3", "vdp_w8", "mocap09_w4", "rows18000_w2", "more_ranks_than_times"])
def test_time_sharded_terms_and_gradients_add_up(kw, world):
    """Time sharding (distributed.enable_time_sharding): every rank -- run one after the other here -- samples and
    integrates only its slice of the time axis plus one halo state; losses and gradients add up to the unsharded ones
    (the halo state's gradient, the constraint's pull, lands on the neighbour's parameter rows). Includes slices of one
    index and more ranks than time indices."""
    p, ys, ts, draws, proj = O.make_problem(seed=7, **kw)
    l_all, _, g_all, _ = _run(p, ys, ts, draws, proj, kw, fuse=True)
    l_sum, g_sum = 0.0, None
    for r in range(world):
        l, _, g, _ = _run(p, ys, ts, draws, proj, kw, fuse=True, time_shard=(r, world), world=world)
        l_sum = l_sum + l.double()
        g = {k: (v if v is not None else torch.zeros_like(g_all[k])) for k, v in g.items()}
        g_sum = {k: v.double() for k, v in g.items()} if g_sum is None else {k: g_sum[k] + g[k].double() for k in g}
    assert relerr(l_sum, l_all) <= 1e-6
    for k in g_all:
        assert relerr(g_sum[k], g_all[k]) <= 2e-5, (k, relerr(g_sum[k], g_all[k]))


def _assert_matches_oracle(kw, seed):
    rows = elbo_errors("shooting", kw, "rk4", {}, seed)
    for k, (e_cuda64, e_ref64, e_cuda32) in rows.items():
        assert e_cuda32 <= TOL_GRAD or e_cuda64 <= max(TOL_GRAD, 1.5 * e_ref64), (k, e_cuda64, e_ref64, e_cuda32)


def test_fused_step_against_the_oracle_at_medium_batch():
    """18 000 segments (row-per-thread kernels) against the oracle port with the float64 arbiter."""
    _assert_matches_oracle(dict(D=3, M=24, S=64, N=3, T=3000, S_mc=2, D_obs=7, dt=0.01), 9)


@pytest.mark.parametrize("kw", [k for k in CASES if k['D'] in (4, 7) and k['S_mc'] * k['N'] * k['T'] > 16384],
                         ids=lambda k: "D%d_B%d" % (k['D'], k['S_mc'] * k['N'] * k['T']))
def test_fused_step_against_the_oracle_at_even_and_odd_d(kw):
    """rk4_fwd_kernel / rk4_bwd_kernel <D, 1, true> at D = 4 (output pairs only) and D = 7 (pairs and the scalar odd
    output) against the oracle port with the float64 arbiter."""
    _assert_matches_oracle(kw, 10 + kw['D'])


def test_end_points_on_request():
    from gaussian_process_odes_b200 import ops
    kw = dict(D=2, M=16, S=64, N=2, T=12, S_mc=3)
    p, ys, ts, draws, proj = O.make_problem(seed=8, **kw)
    model = build_product_model("shooting", p, ys, kw['S'], "rk4")
    with torch.no_grad(), injected_draws(draws, mvn_order=("eps_x0", "eps_states")):
        ss = model.state_distribution.sample(num_samples=kw['S_mc'])
        layer = model.flow.odefunc.diffeq
        layer.build_cache()
        W, b = model.likelihood._affine(ss)
        ll, c, pred = ops.shooting_step(ss, ts[:2].cuda(), *layer.cache_tensors(), ys.cuda(), W, b,
                                        model.likelihood.variance, model.constraint.scale, want_pred=True)
        xs = ops.rk4_integrate(ss.reshape(-1, 2), ts[:2].cuda(), *layer.cache_tensors())
    assert torch.equal(pred, xs[1])
    lp = model.likelihood.log_prob(pred.reshape(ss.shape), ys.cuda().unsqueeze(0)).sum()
    assert relerr(ll, lp) <= 1e-6
