"""Shared helpers of the parity tests.

Tolerances are the ones BASELINE.json's north_star states: relative 1e-5 on vector-field values, 1e-4 on integrated
trajectories, 1e-4 on ELBO terms and gradients ("relative" = max-abs error over max-abs value of the tensor).
Where the reference's OWN float32 path is further than that from the float64 evaluation of the same formula
(|nu| ~ 1e2..4e2 makes sum_m var nu_m K_m cancel heavily; SURVEY.md section 7), the float64 oracle arbitrates:
the CUDA result must be at least as close to float64 as ARBITER_SLACK x the reference's float32 result is.
"""
import os

import numpy as np
import torch

import gpode_oracle as O

TOL_VF, TOL_TRAJ, TOL_GRAD = 1e-5, 1e-4, 1e-4
ARBITER_SLACK = 1.5
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def relerr(a, b):
    a = torch.as_tensor(a).detach().double().cpu()
    b = torch.as_tensor(b).detach().double().cpu()
    assert a.shape == b.shape, (a.shape, b.shape)
    return float((a - b).abs().max() / (b.abs().max() + 1e-300))


def assert_parity(name, cuda, ref32, f64, tol, ref_noise=None, slack=None):
    """cuda vs the float32 reference/oracle within tol, else arbitrated by float64. ``ref_noise``: the reference's
    float32-vs-float64 error measured on a larger sample of the same problem (a max over a handful of elements is
    too noisy a yardstick on its own)."""
    e_direct = relerr(cuda, ref32)
    if e_direct <= tol:
        return e_direct
    if callable(f64):
        f64 = f64()  # the float64 evaluation is only run when the direct comparison does not settle it
    e_cuda, e_ref = relerr(cuda, f64), relerr(ref32, f64)
    if ref_noise is not None:
        e_ref = max(e_ref, ref_noise)
    slack = ARBITER_SLACK if slack is None else slack
    assert e_cuda <= max(tol, slack * e_ref), (
        "%s: cuda-vs-ref32 %.3e > tol %.1e and cuda-vs-fp64 %.3e > %.1f x ref32-vs-fp64 %.3e"
        % (name, e_direct, tol, e_cuda, slack, e_ref))
    return e_cuda


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    t = lambda a: torch.tensor(a)
    out = dict(p={k[5:]: t(z[k]) for k in z.files if k.startswith("in_p_")},
               draws={k[8:]: t(z[k]) for k in z.files if k.startswith("in_draw_")},
               ys=t(z["in_ys"]), ts=t(z["in_ts"]),
               ref={k[4:]: t(z[k]) for k in z.files if k.startswith("ref_")},
               f64={k[4:]: t(z[k]) for k in z.files if k.startswith("f64_")},
               meta=[str(s) for s in z["meta"]])
    out["proj"] = t(z["in_proj_components"]) if "in_proj_components" in z.files else None
    return out


def to_dev(tree, dev="cuda"):
    if isinstance(tree, dict):
        return {k: to_dev(v, dev) for k, v in tree.items()}
    return tree.to(dev) if torch.is_tensor(tree) else tree


def oracle_cache(p, draws, dtype=torch.float32):
    """constrained GP parameters + cache from the oracle port, in ``dtype`` on CPU"""
    gp = O.gp_params(O.cast(p, dtype))
    d = O.cast(draws, dtype)
    c = O.build_cache(gp['Z'], gp['Um'], gp['Us_sqrt'], gp['ell'], gp['var'], d['w'], d['eps_omega'], d['phase_u'],
                      d['eps_u'])
    return gp, c


# ---- gradients of the CUDA ops and of the oracle evaluated over row chunks, on the device --------------------------
GRAD_KEYS = ("x", "Z", "ell", "var", "nu")


def cuda_args(gp, c, grad=False):
    """the seven cache tensors of the ops in their order, on the device; Z, ell, var and nu require grad if ``grad``"""
    d = to_dev(dict(Z=gp['Z'], ell=gp['ell'], var=gp['var'], nu=c['nu'], omega=c['rff_omega'], phase=c['rff_phase'],
                    w=c['rff_weights']))
    return [d[k].float().contiguous().requires_grad_(grad and i < 4)
            for i, k in enumerate(("Z", "ell", "var", "nu", "omega", "phase", "w"))]


def cuda_grads(fn, gp, c, x, cot):
    """fn(x, cache args) on the device -> (output, {x, Z, ell, var, nu: gradient of (output * cot).sum()})"""
    args = cuda_args(gp, c, True)
    xc = x.cuda().requires_grad_(True)
    out = fn(xc, args)
    out.backward(cot.cuda())
    return out.detach(), dict(x=xc.grad, Z=args[0].grad, ell=args[1].grad, var=args[2].grad, nu=args[3].grad)


def oracle_leaves(gp, c, x, dtype, dev):
    """x, Z, ell, var, nu as leaves in ``dtype`` on ``dev`` and the cache built on them"""
    leaves = dict(x=x.to(dev, dtype).clone().requires_grad_(True))
    for k in ("Z", "ell", "var"):
        leaves[k] = gp[k].to(dev, dtype).clone().requires_grad_(True)
    leaves['nu'] = c['nu'].to(dev, dtype).clone().requires_grad_(True)
    # omega = eps / ell stays attached to ell (kernels.py:110-112): rebuild it from eps
    eps = (c['rff_omega'].double() * gp['ell'].double().T.unsqueeze(1)).to(dev, dtype)
    cc = dict(rff_omega=eps / leaves['ell'].T.unsqueeze(1), rff_phase=c['rff_phase'].to(dev, dtype),
              rff_weights=c['rff_weights'].to(dev, dtype), nu=leaves['nu'])
    return leaves, cc


def oracle_vf(l, cc):
    return O.vf_forward(l['x'], l['Z'], l['ell'], l['var'], cc)


def oracle_rk4(ts):
    return lambda l, cc: O.odeint(lambda t, y: O.vf_forward(y, l['Z'], l['ell'], l['var'], cc), l['x'], ts.to(l['x']),
                                  method='rk4')


def chunked_oracle(fn, gp, c, x, cot, dtype, row_dim, dev="cuda", chunk=4096):
    """fn(leaves, cache) over row chunks of x: -> (output, {x, Z, ell, var, nu: gradient of (output * cot).sum()}) with
    the outputs and x-gradients concatenated and the parameter gradients summed over chunks (in float64). Exact for a
    row-separable fn (the vector field, fixed-grid RK4)."""
    outs, gx, gsum = [], [], {}
    for r0 in range(0, x.shape[0], chunk):
        l, cc = oracle_leaves(gp, c, x[r0:r0 + chunk], dtype, dev)
        out = fn(l, cc)
        out.backward(cot.narrow(row_dim, r0, l['x'].shape[0]).to(dev, dtype))
        outs.append(out.detach().cpu())
        gx.append(l['x'].grad.cpu())
        for k in GRAD_KEYS[1:]:
            g = l[k].grad.double().cpu()
            gsum[k] = gsum[k] + g if k in gsum else g
    grads = {k: v.to(dtype) for k, v in gsum.items()}
    grads['x'] = torch.cat(gx)
    return torch.cat(outs, row_dim), grads


def oracle_dopri5(gp, c, x, ts, cot, dtype, dev="cuda", rtol=1e-6, atol=1e-6):
    """autograd through the restated dopri5 -> (xs, {x, Z, ell, var, nu: gradient}, accept/reject counts). Every
    vector-field evaluation is checkpointed (recomputed in the backward pass), so the graph holds one state per
    evaluation instead of its [D, B, D] intermediates. The error norm spans the whole batch: this oracle is not
    chunked."""
    from torch.utils.checkpoint import checkpoint
    l, cc = oracle_leaves(gp, c, x, dtype, dev)
    st = {}
    f = lambda t, y: checkpoint(lambda yy: O.vf_forward(yy, l['Z'], l['ell'], l['var'], cc), y, use_reentrant=False)
    out = O.odeint(f, l['x'], ts.to(dev, dtype), method='dopri5', rtol=rtol, atol=atol, stats=st)
    (out * cot.to(dev, dtype)).sum().backward()
    return out.detach().cpu(), {k: v.grad.detach().cpu() for k, v in l.items()}, st


def lazy(fn):
    """fn() evaluated on the first call only"""
    memo = []

    def get():
        if not memo:
            memo.append(fn())
        return memo[0]
    return get


def assert_grads(name, got, ref32, ref64, tol, keys=GRAD_KEYS):
    """assert_parity of every gradient; ``ref64``: callable returning the float64 gradients"""
    for k in keys:
        assert_parity("%s grad %s" % (name, k), got[k].cpu().reshape(ref32[k].shape), ref32[k],
                      lambda k=k: ref64()[k], tol)


# ---- the fused shooting step (ops.shooting_step) and its oracle ----------------------------------------------------
def shoot_inputs(D, S_mc, N, T, seed, Dobs=None, bias=True, scale=0.3):
    """observations, decoder, likelihood variance and constraint scale of a shooting step (Dobs = D + 1 unless
    given); ``bias=False``: no decoder bias (the draws stay the same)"""
    rng = np.random.default_rng(seed)
    t = lambda a: torch.tensor(np.asarray(a), dtype=torch.float32)
    Dobs = D + 1 if Dobs is None else Dobs
    si = dict(t2=t([0.0, 0.07]), ys=t(rng.normal(size=(N, T, Dobs))), W=t(rng.normal(size=(D, Dobs)) * 0.5),
              bias=t(rng.normal(size=Dobs) * 0.1), lik_var=t(0.5 + rng.uniform(size=Dobs)), scale=t([scale]))
    if not bias:
        si['bias'] = None
    return si


def shoot_cuda(gp, c, ss, si, a_ll, a_c, laplace=False, rows=None, halo=False):
    """ops.shooting_step -> (ll, cons, {x: grad ss, Z, ell, var, nu, lik_var}) of a_ll ll + a_c cons"""
    from gaussian_process_odes_b200 import ops
    args = cuda_args(gp, c, True)
    sc = ss.cuda().requires_grad_(True)
    lv = si['lik_var'].cuda().requires_grad_(True)
    bias = si['bias'].cuda() if si['bias'] is not None else None
    ll, cons, _ = ops.shooting_step(sc, si['t2'].cuda(), *args, si['ys'].cuda(), si['W'].cuda(), bias, lv,
                                    si['scale'].cuda(), laplace=laplace, rows=rows, halo=halo)
    (a_ll * ll + a_c * cons).backward()
    return ll.detach().cpu(), cons.detach().cpu(), dict(x=sc.grad, Z=args[0].grad, ell=args[1].grad,
                                                        var=args[2].grad, nu=args[3].grad, lik_var=lv.grad)


def cons_logprob(y, loc, scale, laplace):
    """the shooting constraint's density (reference src/core/constraints.py:26-36, 56-66), elementwise"""
    dist = torch.distributions.Laplace if laplace else torch.distributions.Normal
    return dist(loc=loc, scale=scale).log_prob(y)


def shoot_oracle(gp, c, ss, si, a_ll, a_c, dtype, chunk, dev="cuda", laplace=False, rows=None, halo=False):
    """the same step through the oracle over row chunks of ``rows = (lo, hi)`` (all rows by default): pred = one RK4
    interval from every row, ll = sum of gauss_loglik(pred W + bias) over the rows that carry an observation (with
    ``halo`` not the last time index of a sequence), cons = sum over t < T-1 of the constraint's log-density of
    ss[t+1] given pred. The constraint's neighbour state is a leaf of its own per chunk; its gradient lands on the next
    row of ss (row hi included). -> (float64 [ll, cons], {x: grad of all of ss, Z, ell, var, nu, lik_var})"""
    S_mc, N, T, D = ss.shape
    x = ss.reshape(-1, D)
    B = x.shape[0]
    lo, hi = (0, B) if rows is None else rows
    tt = torch.arange(B) % T
    nxt = torch.cat([x[1:], x[:1]])     # row r's neighbour ss[s, n, t + 1] is row r + 1 (masked at t = T - 1)
    ys = si['ys'].unsqueeze(0).expand(S_mc, N, T, -1).reshape(B, -1)
    W, scale = [si[k].to(dev, dtype) for k in ("W", "scale")]
    bias = si['bias'].to(dev, dtype) if si['bias'] is not None else 0.0
    var = si['lik_var'].to(dev, dtype).requires_grad_(True)
    step = oracle_rk4(si['t2'])
    ll = cons = 0.0
    gx = torch.zeros(B + 1, D, dtype=dtype)
    gsum = {}
    for r0 in range(lo, hi, chunk):
        r1 = min(r0 + chunk, hi)
        l, cc = oracle_leaves(gp, c, x[r0:r1], dtype, dev)
        nb = nxt[r0:r1].to(dev, dtype).requires_grad_(True)
        pred = step(l, cc)[1]
        obs = torch.ones(r1 - r0) if not halo else (tt[r0:r1] < T - 1).to(torch.float32)
        lli = (O.gauss_loglik(pred @ W + bias, ys[r0:r1].to(dev, dtype), var)
               * obs.to(dev, dtype).unsqueeze(1)).sum()
        mask = (tt[r0:r1] < T - 1).to(dev, dtype).unsqueeze(1)
        ci = (cons_logprob(nb, pred, scale, laplace) * mask).sum()
        (a_ll * lli + a_c * ci).backward()
        ll, cons = ll + float(lli.detach()), cons + float(ci.detach())
        gx[r0:r1] += l['x'].grad.cpu()
        gx[r0 + 1:r1 + 1] += nb.grad.cpu()
        for k in ("Z", "ell", "var", "nu"):
            g = l[k].grad.double().cpu()
            gsum[k] = gsum[k] + g if k in gsum else g
    g = {k: v.to(dtype) for k, v in gsum.items()}
    g['x'] = gx[:B].reshape(S_mc, N, T, D)
    g['lik_var'] = var.grad.cpu() if var.grad is not None else torch.zeros(var.shape, dtype=dtype)
    return torch.tensor([ll, cons], dtype=torch.float64), g


def time_grid(Tg, h, seed):
    """Tg float32 points with steps h (1 +- 0.3 u)"""
    rng = np.random.default_rng(seed)
    steps = h * (1 + 0.3 * rng.uniform(-1, 1, size=Tg - 1))
    return torch.tensor(np.concatenate([[0.0], np.cumsum(steps)]), dtype=torch.float32)


# ---- building the product model from the shared unconstrained-parameter dict, and injecting random draws ----------
class _Queue:
    def __init__(self, items, what):
        self.items, self.what = list(items), what

    def __call__(self, shape, *a, **k):
        assert self.items, "more %s draws requested than injected" % self.what
        x = self.items.pop(0)
        assert tuple(x.shape) == tuple(shape), (self.what, tuple(x.shape), tuple(shape))
        return x.clone()


class injected_draws:
    """The next build_cache / rsample calls of the product modules consume ``draws`` (same protocol as
    oracle/reference_harness.injected_draws uses on the reference's modules)."""

    def __init__(self, draws, n_caches=1, mvn_order=()):
        self.d, self.n, self.mvn_order = draws, n_caches, mvn_order

    def __enter__(self):
        from gaussian_process_odes_b200.core import dsvgp, kernels, states
        d = {k: v.cpu() for k, v in self.d.items()}
        self.mods = (dsvgp, kernels, states)
        self.saved = (dsvgp.sample_normal, dsvgp.sample_uniform, kernels.sample_normal, states._standard_normal)
        dsvgp.sample_normal = _Queue([d['w'], d['eps_u']] * self.n, "dsvgp.normal")
        dsvgp.sample_uniform = _Queue([d['phase_u']] * self.n, "dsvgp.uniform")
        kernels.sample_normal = _Queue([d['eps_omega']] * self.n, "kernels.normal")
        q = _Queue([d[k] for k in self.mvn_order], "states.standard_normal")
        states._standard_normal = lambda shape, dtype, device: q(shape).to(device=device, dtype=dtype)
        return self

    def __exit__(self, *exc):
        dsvgp, kernels, states = self.mods
        dsvgp.sample_normal, dsvgp.sample_uniform, kernels.sample_normal, states._standard_normal = self.saved
        return False


def _set(param, value):
    with torch.no_grad():
        param.copy_(value.to(param))


def build_product_model(kind, p, ys, S, solver, ts_dense_scale=4, proj=None):
    from gaussian_process_odes_b200 import builders
    N, T, Dobs = ys.shape
    M, D = p['inducing_loc'].shape
    projection = None
    if proj is not None:
        from gaussian_process_odes_b200.misc.mocap_utils import LinearProjection
        projection = LinearProjection(proj.cpu().numpy())
    if kind == "gpode":
        model = builders.build_gpode(N, T, D, num_inducing=M, num_features=S, solver=solver,
                                     ts_dense_scale=ts_dense_scale, D_obs=Dobs, projection=projection)
        x0d = model.x0_distribution
    else:
        model = builders.build_gpode_shooting(N, T, D, num_inducing=M, num_features=S, solver=solver, D_obs=Dobs,
                                              projection=projection)
        x0d = model.state_distribution.x0
        _set(model.state_distribution.param_mean.optvar, p['state_mean'])
        _set(model.state_distribution.param_lchol.optvar, p['state_lchol_packed'])
        _set(model.constraint.unconstrained_scale, p['constraint_unconstrained_scale'])
    gp = model.flow.odefunc.diffeq
    _set(gp.inducing_loc.optvar, p['inducing_loc'])
    _set(gp.Um.optvar, p['Um'])
    _set(gp.Us_sqrt.optvar, p['Us_sqrt_packed'])
    _set(gp.kern.unconstrained_lengthscales, p['unconstrained_lengthscales'])
    _set(gp.kern.unconstrained_variance, p['unconstrained_variance'])
    _set(x0d.param_mean.optvar, p['x0_mean'])
    _set(x0d.param_lchol.optvar, p['x0_lchol_packed'])
    _set(model.likelihood.unconstrained_variance, p['lik_unconstrained_variance'])
    return model


def product_grads(model, kind):
    gp = model.flow.odefunc.diffeq
    g = dict(inducing_loc=gp.inducing_loc.optvar.grad, Um=gp.Um.optvar.grad, Us_sqrt_packed=gp.Us_sqrt.optvar.grad,
             unconstrained_lengthscales=gp.kern.unconstrained_lengthscales.grad,
             unconstrained_variance=gp.kern.unconstrained_variance.grad,
             lik_unconstrained_variance=model.likelihood.unconstrained_variance.grad)
    if kind == "gpode":
        g.update(x0_mean=model.x0_distribution.param_mean.optvar.grad,
                 x0_lchol_packed=model.x0_distribution.param_lchol.optvar.grad)
    else:
        sd = model.state_distribution
        g.update(x0_mean=sd.x0.param_mean.optvar.grad, x0_lchol_packed=sd.x0.param_lchol.optvar.grad,
                 state_mean=sd.param_mean.optvar.grad, state_lchol_packed=sd.param_lchol.optvar.grad)
    return g


def elbo_errors(kind, kw, solver, extra, seed):
    """One ELBO forward+backward of a seeded synthetic problem through the product (CUDA) path and through the oracle
    port in float32 and float64 (CPU). -> {name: (cuda-vs-fp64, port32-vs-fp64, cuda-vs-port32)} for the loss and every
    parameter gradient (relative = max-abs error / max-abs value)."""
    from gaussian_process_odes_b200 import builders
    p, ys, ts, draws, proj = O.make_problem(seed=seed, **kw)
    res = {}
    for dtype in (torch.float32, torch.float64):
        pp = {k: v.detach().clone().to(dtype).requires_grad_(True) for k, v in p.items()}
        pj = proj
        if proj is not None and dtype == torch.float64:
            comp = proj.components.double()
            pj = lambda x: torch.einsum('ntl,ld->ntd', x, comp)
        if kind == "gpode":
            r = O.elbo_gpode(pp, ys.to(dtype), ts.to(dtype), O.cast(draws, dtype), method=solver, project=pj, **extra)
        else:
            r = O.elbo_shooting(pp, ys.to(dtype), ts.to(dtype), O.cast(draws, dtype), method=solver, project=pj)
        r['loss'].backward()
        res[dtype] = (r['loss'].detach(), {k: v.grad for k, v in pp.items() if v.grad is not None})
    model = build_product_model(kind, p, ys, kw['S'], solver, ts_dense_scale=extra.get('ts_dense_scale', 4),
                                proj=proj.components if proj is not None else None)
    if kind == "gpode":
        with injected_draws(draws, mvn_order=("eps_x0",)):
            loss = builders.compute_loss_gpode(model, ys.cuda(), ts.cuda())[0]
    else:
        with injected_draws(draws, mvn_order=("eps_x0", "eps_states")):
            ll, c, e, k0 = model.build_lowerbound_terms(ys.cuda(), ts.cuda(), num_samples=kw['S_mc'])
            loss = -(ll + c + e - k0 - model.build_inducing_kl())
    loss.backward()
    g = product_grads(model, kind)
    (l32, g32), (l64, g64) = res[torch.float32], res[torch.float64]
    rows = {"loss": (relerr(loss.cpu(), l64), relerr(l32, l64), relerr(loss.cpu(), l32))}
    for k, v in g.items():
        rows[k] = (relerr(v.cpu(), g64[k]), relerr(g32[k], g64[k]), relerr(v.cpu(), g32[k]))
    return rows


# ---- shared memory of the D <= 8 integrator kernels, restated from their launchers ---------------------------------
# (csrc/common.cuh gpode_layout, csrc/integrate_impl.cuh launch_* / h_smem, csrc/dopri5_impl.cuh). Every CTA of these
# kernels stages the whole packed block, so its size grows with M (the kern records, KS floats per inducing point); a
# block above the 227 KB a CTA can opt into either hands the batch to the next kernel or is refused ("does not fit").
SMEM_OPTIN = 227 * 1024     # check_smem_fits
MAX_M_BLOCKED = 2048        # GPODE_MAX_M_BLOCKED: the largest M the whitening (and so training) accepts
TC_WARPS = 12               # kHWarps = kHFWarps: warps of the tensor-core kernels (D = 4, 5)
TC_ROW_FIELDS = 7           # kHRowFields
RED_WARPS = 16              # kRedWarps
DP_STATIC_SMEM = 96         # kDpStaticSmem: dopri5_kernel's own __shared__ arrays
ADJ_WARPS = 4               # kWarpsPerCta = kDpThreads / 32: warps of the warp-per-row adjoints


def packed_layout(D, M, S):
    """gpode_layout in floats: total (the block the FFMA2 kernels stage), n_small (kern + il records), n_mmah (the
    tensor-core operand records, D <= 5) and n_packed (gpode_packed_floats)"""
    r4 = lambda x: (x + 3) & ~3
    S2P = (((S + 1) // 2) + 31) & ~31
    RP, KS, WP = r4(2 * D + 4), r4(D + 2 * ((D + 1) // 2)), r4(2 * ((D + 1) // 2))
    n_small = M * KS + D * WP
    total = D * S2P * RP + n_small
    n_mmah = D * ((((S + 7) // 8) + 1) & ~1) * 152
    return dict(total=total, n_small=n_small, n_mmah=n_mmah, n_packed=total + (n_mmah if D <= 5 else 0))


def _red_floats(D):
    return (RED_WARPS * (D * D + D) + 3) & ~3


def _warp_acc_bytes(D, warps=ADJ_WARPS):
    return warps * 33 * (D * D + D) * 8     # kWarpAccDoubles<D>: a 32-lane slab and a row of D*D + D per warp


def _tc_smem(D, M, S, rk4, row_sums=False):
    """h_smem<D>(hp, rk4, kHWarps, row_sums)"""
    L = packed_layout(D, M, S)
    stage = 2 * 32 * (D | 1) + 32 * 8
    return 16 + 4 * (L['n_small'] + L['n_mmah'] + (0 if rk4 else _red_floats(D)) + TC_WARPS * stage
                     + (TC_WARPS * TC_ROW_FIELDS * D * 32 if rk4 else 0) + (TC_WARPS * M * 2 * D if row_sums else 0))


SHOOT_MAX_DOBS = 128        # GPODE_SHOOT_MAX_DOBS: the largest observed dimension the fused shooting step takes
THREAD_WARPS = 4            # kThreads / 32 = kWarpsPerCta: warps of the row-per-thread and warp-per-row kernels


def shoot_smem_bytes(D, Dobs, warps):
    """csrc/shoot.cuh shoot_smem_bytes: W, bias, 1/var and log(2 pi var) with Dobs padded to 4, then one float64 row of
    [2 + Dobs] accumulators per warp -- staged by the fused shooting forward on top of the integrator's block"""
    DP = (Dobs + 3) & ~3
    return (D + 3) * DP * 4 + warps * (2 + Dobs) * 8


def _shoot_tc_fwd(D, M, S):
    """launch_rk4_fwd<D, kShoot = true> on the tensor cores: the forward block rounded up to 16 bytes, then the
    epilogue's region for kHFWarps warps"""
    return ((_tc_smem(D, M, S, rk4=False) + 15) & ~15) + shoot_smem_bytes(D, SHOOT_MAX_DOBS, TC_WARPS)


# family -> (state dimensions, bytes(D, M, S), the kernels that stage that many bytes)
SMEM_FAMILIES = {
    "fwd": (range(1, 9), lambda D, M, S: 16 + 4 * packed_layout(D, M, S)['total'],
            "vf_fwd / rk4_fwd kernels (warp, row, wide) and the vf / rk4 *_sets kernels"),
    "dopri5_fwd": (range(1, 9), lambda D, M, S: 16 + 4 * packed_layout(D, M, S)['total'] + DP_STATIC_SMEM,
                   "dopri5_kernel, all three forms"),
    "bwd": (range(1, 9), lambda D, M, S: 16 + 4 * (packed_layout(D, M, S)['total'] + _red_floats(D)),
            "vf_bwd_kernel / rk4_bwd_kernel (row per thread, wide)"),
    "bwd_warp": (range(1, 9), lambda D, M, S: 16 + 4 * packed_layout(D, M, S)['total'] + _warp_acc_bytes(D),
                 "vf_bwd_warp_kernel / rk4_bwd_warp_kernel and dopri5_bwd_kernel"),
    "tc_fwd": ((4, 5), lambda D, M, S: _tc_smem(D, M, S, rk4=False), "vf_fwd_h_kernel / rk4_fwd_h_kernel"),
    "tc_bwd": ((4, 5), lambda D, M, S: _tc_smem(D, M, S, rk4=True),
               "rk4_bwd_mma_kernel; the bound on which vf_bwd_mma_kernel is chosen too"),
    "tc_row_sums": ((4, 5), lambda D, M, S: _tc_smem(D, M, S, rk4=True, row_sums=True),
                    "rk4_bwd_mma_kernel<D, true, true>: the shooting adjoint that sums the inducing-point gradients"),
    "shoot_fwd": (range(1, 9), lambda D, M, S: 16 + 4 * packed_layout(D, M, S)['total']
                  + shoot_smem_bytes(D, SHOOT_MAX_DOBS, THREAD_WARPS),
                  "rk4_fwd_warp_kernel / rk4_fwd_kernel <..., true> at Dobs = 128: the fused shooting forward"),
    "shoot_tc_fwd": ((4, 5), _shoot_tc_fwd,
                     "rk4_fwd_h_kernel<D, true> at Dobs = 128: the fused shooting forward on the tensor cores"),
}


def kernel_smem(family, D, M, S):
    return SMEM_FAMILIES[family][1](D, M, S)


def max_inducing(family, D, S):
    """M*: the largest M whose block fits (0 if not even M = 1 does), or None when M = MAX_M_BLOCKED fits -- that
    family cannot run out of shared memory at this S"""
    fits = lambda M: kernel_smem(family, D, M, S) <= SMEM_OPTIN
    if fits(MAX_M_BLOCKED):
        return None
    lo, hi = 0, MAX_M_BLOCKED          # fits(lo) or lo == 0; not fits(hi): the size grows with M
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if fits(mid) else (lo, mid)
    return lo
