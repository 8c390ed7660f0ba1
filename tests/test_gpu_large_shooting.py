"""The multiple-shooting ELBO step above eight state dimensions (ops.shooting_step at 8 < D <= 64: one RK4 interval on
the tcgen05 vector field, the observation log-likelihood, the shooting constraint and their seeds in one epilogue kernel,
the large-D adjoint seeded on the device; gpode_shoot_fwd_large / gpode_shoot_bwd_large) against the unfused chain of
launches (fuse_elbo = False), against the oracle, under segment-row and time sharding, and its refusals and fallbacks.
The state dimensions sit on both sides of the padded-dimension templates of the large-D kernels (16 / 32 / 64)."""
import ctypes

import numpy as np
import pytest
import torch

import gpode_oracle as O
from util import TOL_GRAD, build_product_model, elbo_errors, injected_draws, product_grads, relerr


def _decoder(D, Dobs, bias, seed):
    """(components (D, D_obs), scale, shift) of a LinearProjection; with ``bias`` the map has a per-dimension scale and
    an offset, i.e. pred W + b with b != 0"""
    rng = np.random.default_rng(seed)
    comp = rng.normal(size=(D, Dobs)) / np.sqrt(D)
    if not bias:
        return comp, None, None
    return comp, 1.0 + 0.2 * rng.uniform(-1, 1, size=D), 0.3 * rng.normal(size=D)


def _model(p, ys, kw, decoder=None, laplace=None, trainable_scale=False):
    model = build_product_model("shooting", p, ys, kw['S'], "rk4", proj=None if decoder is None else
                                torch.tensor(decoder[0], dtype=torch.float32))
    if decoder is not None and decoder[1] is not None:
        from gaussian_process_odes_b200.misc.mocap_utils import LinearProjection
        model.likelihood.projection = LinearProjection(*decoder)
    if laplace is not None:
        from gaussian_process_odes_b200.core import constraints
        model.constraint = constraints.Laplace(d=1, scale=laplace, requires_grad=False).cuda()
    if trainable_scale:
        model.constraint.unconstrained_scale.requires_grad_(True)
    return model


def _run(p, ys, ts, draws, kw, fuse, decoder=None, row_shard=None, time_shard=None, world=1, laplace=None,
         trainable_scale=False):
    from gaussian_process_odes_b200 import _lib
    model = _model(p, ys, kw, decoder, laplace, trainable_scale)
    model.fuse_elbo = fuse
    model.row_shard = row_shard
    model.time_shard = time_shard
    _lib.reset_launch_count()
    with injected_draws(draws, mvn_order=("eps_x0", "eps_states")):
        ll, c, e, k0 = model.build_lowerbound_terms(ys.cuda(), ts.cuda(), num_samples=kw['S_mc'])
        kl = model.build_inducing_kl()
        if time_shard is not None:   # the entropy is this rank's share, only the two KL terms are replicated
            loss = -(ll + c + e - (k0 + kl) / float(world))
        else:
            loss = -(ll + c + (e - k0 - kl) / float(world))
    loss.backward()
    fused_calls = _lib.LAUNCH_COUNT.get("gpode_shoot_fwd_large", 0) // _lib.KERNELS_PER_CALL["gpode_shoot_fwd_large"]
    g = {k: (None if v is None else v.detach().clone()) for k, v in product_grads(model, "shooting").items()}
    return loss.detach(), dict(ll=ll.detach(), c=c.detach()), g, fused_calls


def _problem(kw, seed):
    """O.make_problem plus the decoder of the case (None: the plain Gaussian likelihood, W = I)"""
    kw = dict(kw)
    Dobs, bias = kw.pop('D_obs', None), kw.pop('bias', False)
    p, ys, ts, draws, _ = O.make_problem(seed=seed, D_obs=Dobs, **kw)
    dec = None if Dobs is None else _decoder(kw['D'], Dobs, bias, seed + 1)
    return p, ys, ts, draws, dec


def _rows(k):
    return k['S_mc'] * k['N'] * k['T']


CASES = [
    # below one 128-row tile
    dict(D=9, M=24, S=96, N=2, T=6, S_mc=3, D_obs=1, bias=True),
    dict(D=12, M=20, S=64, N=2, T=8, S_mc=2),                                   # plain Gaussian likelihood (W = I)
    # ragged across tiles
    dict(D=16, M=32, S=128, N=3, T=47, S_mc=2, D_obs=16),
    dict(D=17, M=24, S=96, N=2, T=100, S_mc=5, D_obs=50, bias=True, dt=0.05),
    dict(D=32, M=40, S=128, N=4, T=51, S_mc=5, D_obs=128, dt=0.05),
    dict(D=64, M=30, S=64, N=2, T=13, S_mc=3, D_obs=50),
    # ~2e4 rows
    dict(D=33, M=100, S=256, N=4, T=1000, S_mc=5, D_obs=33, bias=True, dt=0.01),
    dict(D=64, M=100, S=256, N=4, T=1000, S_mc=5, D_obs=128, bias=True, dt=0.01),
]


@pytest.mark.gpu
@pytest.mark.parametrize("kw", CASES, ids=lambda k: "D%d_Dobs%s_B%d%s" % (k['D'], k.get('D_obs', k['D']), _rows(k),
                                                                         "_bias" if k.get('bias') else ""))
def test_large_step_matches_unfused_chain(kw):
    p, ys, ts, draws, dec = _problem(kw, 41)
    l1, t1, g1, n1 = _run(p, ys, ts, draws, kw, True, dec)
    l0, t0, g0, n0 = _run(p, ys, ts, draws, kw, False, dec)
    assert n1 == 1 and n0 == 0   # the fused arm ran the large-D step, the reference arm did not
    assert relerr(l1, l0) <= 1e-5
    for k in t1:
        assert relerr(t1[k], t0[k]) <= 1e-5, k
    for k in g1:
        assert relerr(g1[k], g0[k]) <= TOL_GRAD, (k, relerr(g1[k], g0[k]))


@pytest.mark.gpu
def test_large_step_with_laplace_constraint():
    kw = dict(D=17, M=24, S=96, N=2, T=30, S_mc=3, D_obs=20, bias=True)
    p, ys, ts, draws, dec = _problem(kw, 42)
    l1, t1, g1, n1 = _run(p, ys, ts, draws, kw, True, dec, laplace=0.05)
    l0, t0, g0, _ = _run(p, ys, ts, draws, kw, False, dec, laplace=0.05)
    assert n1 == 1
    assert relerr(l1, l0) <= 1e-5 and relerr(t1['c'], t0['c']) <= 1e-5
    for k in g1:
        assert relerr(g1[k], g0[k]) <= TOL_GRAD, (k, relerr(g1[k], g0[k]))


@pytest.mark.gpu
@pytest.mark.parametrize("kw,seed", [(dict(D=12, M=24, S=96, N=2, T=6, S_mc=3, D_obs=12), 43),
                                     (dict(D=33, M=24, S=96, N=2, T=6, S_mc=3, D_obs=50), 44)], ids=["D12", "D33_Dobs50"])
def test_large_step_against_the_oracle(kw, seed):
    """the whole ELBO through UniformSequenceModel (now on the large-D step) against the oracle port, judged by the
    float64 arbiter"""
    rows = elbo_errors("shooting", kw, "rk4", {}, seed)
    for k, (e_cuda64, e_ref64, e_cuda32) in rows.items():
        assert e_cuda32 <= TOL_GRAD or e_cuda64 <= max(TOL_GRAD, 1.5 * e_ref64), (k, e_cuda64, e_ref64, e_cuda32)


SHARD_CASES = [CASES[0], CASES[3], CASES[6]]


@pytest.mark.gpu
@pytest.mark.parametrize("kw,world", [(SHARD_CASES[0], 2), (SHARD_CASES[1], 3), (SHARD_CASES[2], 8)],
                         ids=["D9_w2", "D17_w3", "D33_w8"])
def test_large_row_sharded_terms_and_gradients_add_up(kw, world):
    """Segment-row sharding at D > 8: the shares of ``world`` ranks -- run one after the other -- add up to the
    unsharded loss and gradients. Blocks cut through Monte-Carlo samples, sequences and time."""
    p, ys, ts, draws, dec = _problem(kw, 45)
    l_all, _, g_all, _ = _run(p, ys, ts, draws, kw, True, dec)
    l_sum, g_sum = 0.0, None
    for r in range(world):
        l, _, g, n = _run(p, ys, ts, draws, kw, True, dec, row_shard=(r, world), world=world)
        assert n == 1
        l_sum = l_sum + l.double()
        g_sum = {k: v.double() for k, v in g.items()} if g_sum is None else {k: g_sum[k] + g[k].double() for k in g}
    assert relerr(l_sum, l_all) <= 1e-6
    for k in g_all:
        assert relerr(g_sum[k], g_all[k]) <= 2e-5, (k, relerr(g_sum[k], g_all[k]))


@pytest.mark.gpu
@pytest.mark.parametrize("kw,world", [(SHARD_CASES[1], 3), (SHARD_CASES[2], 4), (SHARD_CASES[0], 8)],
                         ids=["D17_w3", "D33_w4", "more_ranks_than_times"])
def test_large_time_sharded_terms_and_gradients_add_up(kw, world):
    """Time sharding at D > 8: every rank samples and integrates only its slice of the time axis plus one halo state;
    losses and gradients add up to the unsharded ones, with more ranks than time indices too (T = 6, 8 ranks)."""
    p, ys, ts, draws, dec = _problem(kw, 46)
    l_all, _, g_all, _ = _run(p, ys, ts, draws, kw, True, dec)
    l_sum, g_sum = 0.0, None
    for r in range(world):
        l, _, g, _ = _run(p, ys, ts, draws, kw, True, dec, time_shard=(r, world), world=world)
        l_sum = l_sum + l.double()
        g = {k: (v if v is not None else torch.zeros_like(g_all[k])) for k, v in g.items()}
        g_sum = {k: v.double() for k, v in g.items()} if g_sum is None else {k: g_sum[k] + g[k].double() for k in g}
    assert relerr(l_sum, l_all) <= 1e-6
    for k in g_all:
        assert relerr(g_sum[k], g_all[k]) <= 2e-5, (k, relerr(g_sum[k], g_all[k]))


def _step_inputs(kw, seed):
    """sampled states, the GP draw's cache tensors and the likelihood / constraint tensors of one step"""
    p, ys, ts, draws, dec = _problem(kw, seed)
    model = _model(p, ys, kw, dec)
    with torch.no_grad(), injected_draws(draws, mvn_order=("eps_x0", "eps_states")):
        ss = model.state_distribution.sample(num_samples=kw['S_mc'])
        layer = model.flow.odefunc.diffeq
        layer.build_cache()
        W, b = model.likelihood._affine(ss)
        cache = [t.detach().clone() for t in layer.cache_tensors()]
    return model, ss, ys.cuda(), ts[:2].cuda(), cache, W, b


@pytest.mark.gpu
def test_large_end_points_on_request():
    from gaussian_process_odes_b200 import ops
    kw = dict(D=33, M=24, S=96, N=2, T=40, S_mc=3, D_obs=40, bias=True)
    model, ss, ys, t2, cache, W, b = _step_inputs(kw, 47)
    with torch.no_grad():
        ll, c, pred = ops.shooting_step(ss, t2, *cache, ys, W, b, model.likelihood.variance, model.constraint.scale,
                                        want_pred=True)
        xs = ops.rk4_integrate(ss.reshape(-1, kw['D']), t2, *cache)
        lp = model.likelihood.log_prob(pred.reshape(ss.shape), ys.unsqueeze(0)).sum()
    assert torch.equal(pred, xs[1])
    assert relerr(ll, lp) <= 1e-6


@pytest.mark.gpu
def test_large_step_backward_is_bitwise_repeatable():
    """no floating-point atomics: two backward passes of the same step give the same bits"""
    from gaussian_process_odes_b200 import ops
    kw = dict(D=33, M=100, S=256, N=4, T=400, S_mc=5, D_obs=64, bias=True, dt=0.01)
    model, ss, ys, t2, cache, W, b = _step_inputs(kw, 48)
    var = model.likelihood.variance.detach()

    def once():
        leaves = [ss.clone().requires_grad_(True)] + [t.clone().requires_grad_(i < 4) for i, t in enumerate(cache)]
        lv = var.clone().requires_grad_(True)
        ll, c, _ = ops.shooting_step(leaves[0], t2, *leaves[1:], ys, W, b, lv, model.constraint.scale.detach())
        (0.7 * ll + 1.3 * c).backward()
        return [ll.detach(), c.detach(), lv.grad] + [x.grad for x in leaves[:5]]

    a, b2 = once(), once()
    for x, y in zip(a, b2):
        assert torch.equal(x, y)


@pytest.mark.gpu
def test_large_step_refuses_more_than_64_state_dimensions():
    from gaussian_process_odes_b200 import ops
    from gaussian_process_odes_b200._lib import GpodeError
    D, M, S, Dobs = 65, 4, 8, 3
    z = lambda *s: torch.zeros(*s, device="cuda")
    with pytest.raises(GpodeError, match="up to 64"):
        ops.shooting_step(z(1, 1, 2, D), z(2), z(M, D), z(D, D) + 1, z(D) + 1, z(D, M), z(D, S, D), z(S, D), z(S, D),
                          z(1, 2, Dobs), z(D, Dobs), None, z(Dobs) + 1, z(1) + 1)


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["dobs129", "trainable_scale"])
def test_large_configurations_without_the_step_take_the_unfused_chain(what):
    """D_obs = 129 (above GPODE_SHOOT_MAX_DOBS) or a trainable constraint scale: fuse_elbo = True takes the unfused chain
    and gives the same bits as fuse_elbo = False"""
    kw = dict(D=17, M=24, S=96, N=2, T=6, S_mc=3, D_obs=129 if what == "dobs129" else 20)
    p, ys, ts, draws, dec = _problem(kw, 49)
    ts_ = what == "trainable_scale"
    l1, t1, g1, n1 = _run(p, ys, ts, draws, kw, True, dec, trainable_scale=ts_)
    l0, t0, g0, _ = _run(p, ys, ts, draws, kw, False, dec, trainable_scale=ts_)
    assert n1 == 0
    assert torch.equal(l1, l0)
    for k in g1:
        assert torch.equal(g1[k], g0[k]), k


def test_large_work_size_and_argument_errors():
    """pure host entry points: the scratch size and the refusals before any CUDA call"""
    from gaussian_process_odes_b200 import _lib
    lib = _lib.load()
    part = 1024 * 130
    assert lib.gpode_shoot_large_work_doubles(9, 0) == part
    assert lib.gpode_shoot_large_work_doubles(64, 1000) == part + 9 * 1000 * 64 // 2
    assert lib.gpode_shoot_large_work_doubles(17, 3) == part + (9 * 3 * 17 + 1) // 2
    assert lib.gpode_shoot_large_work_doubles(8, 10) == -1 and lib.gpode_shoot_large_work_doubles(65, 10) == -1
    sh = _lib.GpodeShoot()
    sh.S_mc, sh.N, sh.T, sh.D_obs, sh.row_lo, sh.row_hi = 1, 1, 4, 3, 0, 4
    sh.ys = sh.W = sh.lik_var = sh.cons_scale = 16
    c = _lib.GpodeCache()
    c.D, c.M, c.S = 8, 4, 8
    args = (ctypes.byref(sh), None, None, None, None, None, None, None, None, None)
    assert lib.gpode_shoot_fwd_large(None, ctypes.byref(c), *args) < 0 and b"8 < D <= 64" in lib.gpode_last_error()
    c.D = 12
    sh.D_obs = 129
    assert lib.gpode_shoot_fwd_large(None, ctypes.byref(c), *args) < 0 and b"observed dimension" in lib.gpode_last_error()
    sh.D_obs, sh.row_hi = 3, 5
    assert lib.gpode_shoot_bwd_large(None, ctypes.byref(c), *args, None) < 0 and b"row range" in lib.gpode_last_error()
    sh.row_hi = 4
    assert lib.gpode_shoot_fwd_large(None, ctypes.byref(c), *args) < 0 and b"NULL" in lib.gpode_last_error()
