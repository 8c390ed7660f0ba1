"""-m gpu: the fused ELBO side-term kernels against the reference's own formulation (torch.distributions on CPU)."""
import numpy as np
import pytest
import torch

import gpode_oracle as O
from util import relerr

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("D", range(1, 9))
@pytest.mark.parametrize("batch", [(1,), (6, 99), (3, 1)])
def test_state_sample_and_entropy(D, batch):
    from gaussian_process_odes_b200 import ops
    rng = np.random.default_rng(D + len(batch))
    P = D * (D + 1) // 2
    S = 4
    L = np.tril(rng.normal(size=batch + (D, D)) * 0.1) + np.eye(D) * 0.5  # well conditioned, like the model's 0.1 I init
    Lp = O.packed_from_tril(torch.tensor(L, dtype=torch.float32))
    mean = torch.tensor(rng.normal(size=batch + (D,)), dtype=torch.float32)
    eps = torch.tensor(rng.normal(size=(S,) + batch + (D,)), dtype=torch.float32)
    cot_s = torch.tensor(rng.normal(size=(S,) + batch + (D,)), dtype=torch.float32)
    cot_h = torch.tensor(rng.normal(size=batch), dtype=torch.float32)
    # reference formulation (src/core/states.py:69-74,91-92,203-204) in float64
    m64, l64 = mean.double().requires_grad_(True), Lp.double().requires_grad_(True)
    dist = O.mvn_from_lchol(m64, O.tril_from_packed(l64, D))
    smp = O.mvn_rsample(dist, eps.double())
    ent = dist.entropy()
    ((smp * cot_s.double()).sum() + (ent * cot_h.double()).sum()).backward()
    mc, lc = mean.cuda().requires_grad_(True), Lp.cuda().requires_grad_(True)
    smp_c = ops.state_sample(mc, lc, eps.cuda())
    ent_c = ops.state_entropy(lc, D)
    ((smp_c * cot_s.cuda()).sum() + (ent_c * cot_h.cuda()).sum()).backward()
    assert smp_c.shape == smp.shape and ent_c.shape == ent.shape
    assert relerr(smp_c, smp) <= 2e-5
    assert relerr(ent_c, ent) <= 2e-5
    assert relerr(mc.grad, m64.grad) <= 2e-5
    assert relerr(lc.grad, l64.grad) <= 2e-4


@pytest.mark.parametrize("D,Dobs,S,lead", [(5, 50, 3, (2, 20)), (2, 2, 5, (1, 25)), (5, 50, 1, (6, 100)), (3, 128, 2, (4, 7)),
                                           (1, 3, 2, (2, 11)), (4, 33, 4, (3, 9)), (6, 64, 5, (1, 40)),
                                           (7, 97, 9, (2, 5)), (8, 128, 3, (3, 8))])
@pytest.mark.parametrize("with_bias", [False, True])
def test_loglik_mean(D, Dobs, S, lead, with_bias):
    from gaussian_process_odes_b200 import ops
    rng = np.random.default_rng(D * Dobs + S)
    t = lambda a: torch.tensor(np.asarray(a), dtype=torch.float32)
    pred = t(rng.normal(size=(S,) + lead + (D,)))
    ys = t(rng.normal(size=(1,) + lead + (Dobs,)))
    W = t(rng.normal(size=(D, Dobs)))
    b = t(rng.normal(size=(Dobs,))) if with_bias else None
    var = t(rng.uniform(0.1, 2.0, size=(Dobs,)))
    p64, v64 = pred.double().requires_grad_(True), var.double().requires_grad_(True)
    f = p64 @ W.double() + (b.double() if b is not None else 0.0)
    ref = O.gauss_loglik(f, ys.double(), v64).mean()
    ref.backward()
    pc, vc = pred.cuda().requires_grad_(True), var.cuda().requires_grad_(True)
    got = ops.loglik_mean(pc, ys.cuda(), W.cuda(), None if b is None else b.cuda(), vc)
    (got * 1.7).backward()
    assert relerr(got, ref) <= 2e-6
    assert relerr(pc.grad, p64.grad * 1.7) <= 2e-5
    assert relerr(vc.grad, v64.grad * 1.7) <= 2e-5


def test_generic_projection_callable_still_works():
    """A likelihood whose decoder is an opaque callable takes the plain tensor path and gives the same ELBO."""
    from gaussian_process_odes_b200 import builders
    from util import build_product_model, injected_draws, load_golden
    g = load_golden("mocap_shooting_rk4")
    fused = build_product_model("shooting", g['p'], g['ys'], 256, "rk4", proj=g['proj'])
    generic = build_product_model("shooting", g['p'], g['ys'], 256, "rk4", proj=g['proj'])
    comp = g['proj'].cuda()
    generic.likelihood.projection = lambda x: torch.einsum('ntl,ld->ntd', x, comp)
    out = []
    for model in (fused, generic):
        with injected_draws(g['draws'], mvn_order=("eps_x0", "eps_states")):
            loss = builders.compute_loss_shooting(model, g['ys'].cuda(), g['ts'].cuda(), num_samples=3)[0]
        loss.backward()
        out.append((loss.detach().cpu(), model.likelihood.unconstrained_variance.grad.cpu(),
                    model.state_distribution.param_mean.optvar.grad.cpu()))
    assert relerr(out[0][0], out[1][0]) <= 1e-5
    assert relerr(out[0][1], out[1][1]) <= 1e-4
    assert relerr(out[0][2], out[1][2]) <= 1e-4


@pytest.mark.parametrize("laplace", [False, True])
@pytest.mark.parametrize("shape", [(3, 2, 7, 2), (5, 1, 25, 2), (2, 3, 4, 5), (1, 1, 2, 1)])
def test_constraint_sum(laplace, shape):
    """Fused shooting-constraint term against torch.distributions (reference src/core/constraints.py:26-36,56-66)."""
    from gaussian_process_odes_b200 import ops
    rng = np.random.default_rng(sum(shape))
    ss = torch.tensor(rng.normal(size=shape), dtype=torch.float32)
    pred = torch.tensor(rng.normal(size=shape), dtype=torch.float32)
    scale = torch.tensor([0.37], dtype=torch.float32)
    s64, p64 = ss.double().requires_grad_(True), pred.double().requires_grad_(True)
    dist = (torch.distributions.Laplace if laplace else torch.distributions.Normal)(loc=p64[:, :, :-1], scale=scale.double())
    ref = dist.log_prob(s64[:, :, 1:]).sum()
    (ref * 0.3).backward()
    sc, pc = ss.cuda().requires_grad_(True), pred.cuda().requires_grad_(True)
    got = ops.constraint_sum(sc, pc, scale.cuda(), laplace=laplace)
    (got * 0.3).backward()
    assert relerr(got, ref) <= 2e-6
    assert relerr(sc.grad, s64.grad) <= 2e-6
    assert relerr(pc.grad, p64.grad) <= 2e-6


def test_laplace_constraint_model_matches_tensor_path():
    """UniformSequenceModel with the Laplace prior: fused term == the reference formulation on plain tensors."""
    from gaussian_process_odes_b200 import builders
    from util import injected_draws, load_golden, build_product_model
    g = load_golden("vdp_shooting_rk4")
    out = []
    for fused in (True, False):
        m = builders.build_gpode_shooting(1, 25, 2, num_inducing=16, num_features=256, solver="rk4",
                                          constraint_type="laplace", constraint_initial_scale=1e-2)
        ref_m = build_product_model("shooting", g['p'], g['ys'], 256, "rk4")
        sd = ref_m.state_dict()
        sd["constraint.unconstrained_scale"] = m.state_dict()["constraint.unconstrained_scale"]
        m.load_state_dict(sd)
        if not fused:
            m.constraint.shooting_sum = None
        with injected_draws(g['draws'], mvn_order=("eps_x0", "eps_states")):
            loss = builders.compute_loss_shooting(m, g['ys'].cuda(), g['ts'].cuda(), num_samples=5)[0]
        loss.backward()
        out.append((loss.detach().cpu(), m.state_distribution.param_mean.optvar.grad.cpu()))
    assert relerr(out[0][0], out[1][0]) <= 1e-5
    assert relerr(out[0][1], out[1][1]) <= 1e-4


@pytest.mark.parametrize("D,M", [(2, 16), (5, 100), (3, 1), (1, 7)])
def test_inducing_sample_from_the_packed_factor(D, M):
    """u = Um + Us_sqrt eps (reference src/core/dsvgp.py:78-90, full-rank branch) through gpode_inducing_sample_fwd/_bwd
    straight from the packed lower-triangular parameter, against the reference's einsum over the scattered factor, and
    the x0 KL through the fused KL kernels against its spelled-out form."""
    from gaussian_process_odes_b200 import ops
    from gaussian_process_odes_b200.misc import transforms
    rng = np.random.default_rng(D * 100 + M)
    tr = transforms.LowerTriangular(M, D)
    packed = torch.tensor(rng.normal(size=(D, M * (M + 1) // 2)), dtype=torch.float32, device="cuda", requires_grad=True)
    Um = torch.tensor(rng.normal(size=(M, D)), dtype=torch.float32, device="cuda", requires_grad=True)
    eps = torch.tensor(rng.normal(size=(M, D)), dtype=torch.float32, device="cuda")
    cot = torch.tensor(rng.normal(size=(M, D)), dtype=torch.float32, device="cuda")
    u = ops.inducing_sample(Um, packed, eps)
    u.backward(cot)
    got = (u.detach().clone(), Um.grad.clone(), packed.grad.clone())
    Um.grad = packed.grad = None
    ref = torch.einsum('dnm, md->nd', tr.forward_tensor(packed), eps) + Um
    ref.backward(cot)
    assert relerr(got[0], ref.detach()) <= 1e-6
    assert relerr(got[1], Um.grad) <= 1e-6 and relerr(got[2], packed.grad) <= 1e-6


def test_initial_state_kl_through_the_fused_kernels():
    from gaussian_process_odes_b200.core import states
    torch.manual_seed(3)
    x0 = states.StateInitialVariationalGaussian(dim_n=6, dim_d=5).cuda()
    with torch.no_grad():
        x0.param_mean.optvar.normal_()
        x0.param_lchol.optvar.add_(0.05 * torch.randn_like(x0.param_lchol.optvar))
    kl = x0.kl()
    kl.backward()
    g = (x0.param_mean.optvar.grad.clone(), x0.param_lchol.optvar.grad.clone())
    x0.param_mean.optvar.grad = x0.param_lchol.optvar.grad = None
    alpha, Lq = x0.mean(), torch.tril(x0.lchol())
    d = torch.diagonal(Lq, dim1=1, dim2=2)
    ref = 0.5 * (-torch.log(d.pow(2)).sum(1) + alpha.pow(2).sum(1) + Lq.pow(2).sum(dim=(1, 2)) - 5.0).sum()
    ref.backward()
    assert relerr(kl.detach(), ref.detach()) <= 1e-6
    assert relerr(g[0], x0.param_mean.optvar.grad) <= 1e-6 and relerr(g[1], x0.param_lchol.optvar.grad) <= 1e-6
