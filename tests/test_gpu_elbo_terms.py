"""-m gpu: the ELBO terms around the integrator against float64 torch, at the shapes where their kernels change path.

- loglik_kernel (ops.loglik_mean, csrc/side_terms.cu): one warp per observation row on min(ceil(R / 8), 8 SMs, 2048)
  CTAs of 8 warps, lanes over the observed dimensions in passes of 32, samples in chunks of kSC = 4. Every D in 1..8,
  Dobs at the pass boundaries, S with and without a tail chunk, R = 1, 7, 8, 9 and past the grid cap (warps visit
  several rows), a problem whose variance gradient nearly cancels, and every gradient subset.
- constraint_kernel (ops.constraint_sum): one thread per (sequence, t < T-1, d) on a capped grid-stride loop whose
  per-CTA float64 partials side_sum_kernel adds. The bench shape (many CTAs, the loop iterates), T = 1 and 2, state
  dimensions 1, 9 and 64, the models' initial scale 1e-3 and exact Laplace ties (gradient 0).
- state_fwd/bwd_kernel (ops.state_sample / state_entropy): one thread per D x D factor. Every D, row counts at the CTA
  edges, factors with diagonals of both signs from 1e-3 to 3, and each one-sided backward on its own.
- the fused shooting epilogue (csrc/shoot.cuh, ops.shooting_step) on every forward mapping against util.shoot_oracle:
  Dobs up to 128, both constraint families, the halo flag, row ranges cut through samples and sequences and empty; the
  bench shape against a float64 epilogue on the kernel's end points; the epilogue's shared memory at the limits of
  util.SMEM_FAMILIES shoot_fwd / shoot_tc_fwd, and the model's unfused fallback past them.

float64 torch of the same formula is the reference; float32 torch arbitrates (util.assert_parity)."""
import math

import numpy as np
import pytest
import torch

import gpode_oracle as O
from test_gpu_many_inducing import _chunk, _problem
from test_gpu_small_d_mappings import (WARP_MAX_ROWS, grids_of, mma_min_rows, profiled, rows_per_thread,
                                       selected_mapping, tensor_cores, wide_min_rows)
from util import (GRAD_KEYS, SHOOT_MAX_DOBS, TOL_GRAD, assert_grads, assert_parity, cons_logprob, cuda_args, lazy,
                  max_inducing, oracle_leaves, oracle_rk4, relerr, shoot_cuda, shoot_inputs, shoot_oracle)

pytestmark = pytest.mark.gpu

TOL_VALUE, TOL_G = 2e-6, 2e-5
TOL_STATE = 2e-5    # samples and entropy: the bar of test_gpu_side_terms.py::test_state_sample_and_entropy
SHOOT_KEYS = GRAD_KEYS + ("lik_var",)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _randn(gen, *shape):
    return torch.randn(*shape, generator=gen, device="cuda", dtype=torch.float32)


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _leaf(t, dtype):
    """a fresh leaf copy of ``t`` in ``dtype`` (never ``t`` itself, which other evaluations reuse)"""
    return t.detach().to(dtype).clone().requires_grad_(True)


# ---- observation log-likelihood --------------------------------------------------------------------------------------
LL_PAIRS = [(1, 1), (2, 4), (3, 31), (4, 32), (5, 33), (6, 64), (7, 65), (8, 96), (1, 97), (2, 127), (3, 128),
            (8, 128), (4, 1), (6, 33), (7, 127), (5, 97)]
LL_CASES = [(D, Dobs, (1, 4, 5, 9)[i % 4], ("cap", 1, 7, 8, 9)[i % 5], i % 2 == 0, False)
            for i, (D, Dobs) in enumerate(LL_PAIRS)] + \
           [(8, 65, 9, "cap", False, False), (5, 50, 5, 200000, True, False), (5, 50, 5, 1000000, True, True)]


def _rows(R):
    """'cap': 13 rows more than the warps of the largest grid, so that some warps visit two rows"""
    return 8 * 8 * _sms() + 13 if R == "cap" else R


def _loglik_problem(D, Dobs, S, R, bias, cancel, seed):
    """pred (S, R, D), ys (1, R, Dobs), W, bias, var on the device; cancel: ys = (mean prediction) W + b + noise of
    variance var, so that the terms of the variance gradient nearly cancel"""
    g = _gen(seed)
    W = _randn(g, D, Dobs) / math.sqrt(D)
    b = _randn(g, Dobs) * 0.3 if bias else None
    var = torch.rand(Dobs, generator=g, device="cuda") * 1.9 + 0.1
    if cancel:
        base = _randn(g, 1, R, D)
        pred = base + 0.01 * _randn(g, S, R, D)
        ys = base @ W + (b if b is not None else 0.0) + var.sqrt() * _randn(g, 1, R, Dobs)
    else:
        pred = _randn(g, S, R, D)
        ys = _randn(g, 1, R, Dobs)
    return pred, ys, W, b, var


def _loglik_ref(pred, ys, W, b, var, dtype):
    """-> (mean, d/d pred, d/d var) of O.gauss_loglik in ``dtype`` on the device"""
    p, v = _leaf(pred, dtype), _leaf(var, dtype)
    f = p @ W.to(dtype) + (b.to(dtype) if b is not None else 0.0)
    val = O.gauss_loglik(f, ys.to(dtype), v).mean()
    val.backward()
    return val.detach(), p.grad, v.grad


@pytest.mark.parametrize("D,Dobs,S,R,bias,cancel", LL_CASES, ids=lambda v: str(v))
def test_loglik_against_float64(D, Dobs, S, R, bias, cancel):
    """value and both gradients of ops.loglik_mean; the value is bitwise the same whichever gradients are wanted"""
    from gaussian_process_odes_b200 import ops
    R = _rows(R)
    pred, ys, W, b, var = _loglik_problem(D, Dobs, S, R, bias, cancel, 7 * D + Dobs + S + R)
    r32 = _loglik_ref(pred, ys, W, b, var, torch.float32)
    r64 = lazy(lambda: _loglik_ref(pred, ys, W, b, var, torch.float64))
    values = []
    for need_p, need_v in ((True, True), (True, False), (False, True), (False, False)):
        pc, vc = pred.clone().requires_grad_(need_p), var.clone().requires_grad_(need_v)
        got = ops.loglik_mean(pc, ys, W, b, vc)
        values.append(got.detach())
        if need_p or need_v:
            got.backward()
        name = "loglik D=%d Dobs=%d S=%d R=%d grads=%d%d" % (D, Dobs, S, R, need_p, need_v)
        if need_p:
            assert_parity(name + " pred", pc.grad, r32[1], lambda: r64()[1], TOL_G)
        if need_v:
            assert_parity(name + " var", vc.grad, r32[2], lambda: r64()[2], TOL_G)
    assert_parity("loglik value D=%d Dobs=%d S=%d R=%d" % (D, Dobs, S, R), values[0], r32[0], lambda: r64()[0],
                  TOL_VALUE)
    for v in values[1:]:
        assert torch.equal(v, values[0]), "the value depends on which gradients are wanted"


def test_loglik_gaussian_ndim1_broadcast():
    """likelihoods.Gaussian(ndim=1) (one variance for every observed dimension) through log_prob_mean -- the fused
    kernel with the variance expanded -- against log_prob(...).mean() in float64"""
    import copy
    from gaussian_process_odes_b200.core import likelihoods
    g = _gen(11)
    F, Y = _randn(g, 3, 4, 50, 6), _randn(g, 1, 4, 50, 6)
    lik = likelihoods.Gaussian(ndim=1, init_val=0.37).cuda()
    Fc = F.clone().requires_grad_(True)
    got, kernels = profiled(lambda: lik.log_prob_mean(Fc, Y))
    grids_of(kernels, "loglik_kernel")
    got.backward()

    def ref(dtype):
        l = copy.deepcopy(lik).to(dtype)
        l.unconstrained_variance.grad = None
        Fr = _leaf(F, dtype)
        val = l.log_prob(Fr, Y.to(dtype)).mean()
        val.backward()
        return val.detach(), Fr.grad, l.unconstrained_variance.grad
    r32, r64 = ref(torch.float32), lazy(lambda: ref(torch.float64))
    assert_parity("ndim=1 value", got.detach(), r32[0], lambda: r64()[0], TOL_VALUE)
    assert_parity("ndim=1 grad F", Fc.grad, r32[1], lambda: r64()[1], TOL_G)
    assert_parity("ndim=1 grad variance", lik.unconstrained_variance.grad, r32[2], lambda: r64()[2], TOL_G)


# ---- shooting constraint ---------------------------------------------------------------------------------------------
CONS_SHAPES = [(5, 16, 12500, 5), (2, 3, 1, 4), (3, 2, 2, 3), (4, 5, 33, 1), (2, 3, 40, 9), (1, 2, 30, 64)]


@pytest.mark.parametrize("scale", [0.37, 1e-3])
@pytest.mark.parametrize("laplace", [False, True])
@pytest.mark.parametrize("shape", CONS_SHAPES, ids=lambda v: str(v))
def test_constraint_against_float64(shape, laplace, scale):
    """ops.constraint_sum: value and both gradients; every 7th pair an exact tie (gradient exactly 0), and the slots no
    pair reaches -- ss[:, :, 0] and pred[:, :, T-1] -- exactly 0"""
    from gaussian_process_odes_b200 import ops
    SM, N, T, D = shape
    g = _gen(sum(shape) + int(laplace))
    pred = _randn(g, *shape)
    ss = _randn(g, *shape)
    ss[:, :, 1:] = pred[:, :, :-1] + 2 * scale * _randn(g, SM, N, T - 1, D)
    tie = torch.zeros(SM, N, T - 1, D, dtype=torch.bool, device="cuda")
    tie.view(-1)[::7] = True
    ss[:, :, 1:][tie] = pred[:, :, :-1][tie]
    sk = torch.tensor([scale], dtype=torch.float32, device="cuda")
    sc, pc = ss.clone().requires_grad_(True), pred.clone().requires_grad_(True)
    got = ops.constraint_sum(sc, pc, sk, laplace=laplace)
    (got * 0.3).backward()

    def ref(dtype):
        s, p = _leaf(ss, dtype), _leaf(pred, dtype)
        val = cons_logprob(s[:, :, 1:], p[:, :, :-1], sk.to(dtype), laplace).sum()
        (val * 0.3).backward()
        return val.detach(), s.grad, p.grad
    name = "constraint %s %s scale=%g" % (shape, "laplace" if laplace else "gauss", scale)
    if T == 1:
        assert float(got) == 0.0
        assert not sc.grad.any() and not pc.grad.any()
        return
    r32, r64 = ref(torch.float32), lazy(lambda: ref(torch.float64))
    assert_parity(name + " value", got.detach(), r32[0], lambda: r64()[0], TOL_VALUE)
    assert_parity(name + " grad ss", sc.grad, r32[1], lambda: r64()[1], TOL_VALUE)
    assert_parity(name + " grad pred", pc.grad, r32[2], lambda: r64()[2], TOL_VALUE)
    assert not sc.grad[:, :, 0].any() and not pc.grad[:, :, T - 1].any()
    assert not sc.grad[:, :, 1:][tie].any() and not pc.grad[:, :, :-1][tie].any(), "a tie has a nonzero gradient"


# ---- state sampling and entropy --------------------------------------------------------------------------------------
STATE_CASES = [(1, 200003, 7), (2, 1, 1), (3, 127, 7), (4, 128, 0), (5, 129, 1), (6, 200003, 0), (7, 128, 7),
               (8, 200003, 1), (8, 129, 7), (1, 127, 0), (2, 129, 7), (3, 1, 0), (4, 200003, 7), (5, 128, 7),
               (6, 127, 1), (7, 1, 0)]


def _factors(D, R, seed):
    """packed lower-triangular factors whose diagonals have either sign and magnitudes 1e-3 .. 3; the off-diagonal
    entries of a row are 0.3 x its diagonal's magnitude, so chol(L L^T + 1e-5 I) stays well defined in float32"""
    rng = np.random.default_rng(seed)
    mag = 10.0 ** rng.uniform(-3.0, math.log10(3.0), size=(R, D))
    sign = np.where(rng.uniform(size=(R, D)) < 0.3, -1.0, 1.0)
    L = np.tril(rng.normal(size=(R, D, D)) * 0.3 * mag[:, :, None], -1)
    L[:, np.arange(D), np.arange(D)] = sign * mag
    return O.packed_from_tril(torch.tensor(L, dtype=torch.float32))


@pytest.mark.parametrize("D,R,S", STATE_CASES)
def test_state_sample_and_entropy_against_float64(D, R, S):
    """samples (gpode_state_bwd without the entropy gradient) and entropy (without the sample gradient) each with its
    own backward, against O.mvn_from_lchol (the reference's MultivariateNormal with the 1e-5 jitter)"""
    from gaussian_process_odes_b200 import ops
    rng = np.random.default_rng(D * 1000 + R + S)
    Lp = _factors(D, R, D + R + S)
    mean = torch.tensor(rng.normal(size=(R, D)), dtype=torch.float32)
    eps = torch.tensor(rng.normal(size=(S, R, D)), dtype=torch.float32)
    cot_s = torch.tensor(rng.normal(size=(S, R, D)), dtype=torch.float32)
    cot_h = torch.tensor(rng.normal(size=(R,)), dtype=torch.float32)

    def ref(dtype):
        out = {}
        m, l = _leaf(mean, dtype), _leaf(Lp, dtype)
        ent = O.mvn_from_lchol(m, O.tril_from_packed(l, D)).entropy()
        (ent * cot_h.to(dtype)).sum().backward()
        out.update(ent=ent.detach(), ent_L=l.grad)
        if S:
            m, l = _leaf(mean, dtype), _leaf(Lp, dtype)
            smp = O.mvn_rsample(O.mvn_from_lchol(m, O.tril_from_packed(l, D)), eps.to(dtype))
            (smp * cot_s.to(dtype)).sum().backward()
            out.update(smp=smp.detach(), smp_mean=m.grad, smp_L=l.grad)
        return out
    r32, r64 = ref(torch.float32), lazy(lambda: ref(torch.float64))
    got = {}
    lc = Lp.cuda().requires_grad_(True)
    ent = ops.state_entropy(lc, D)
    (ent * cot_h.cuda()).sum().backward()
    got.update(ent=ent.detach().cpu(), ent_L=lc.grad.cpu())
    if S:
        mc, lc = mean.cuda().requires_grad_(True), Lp.cuda().requires_grad_(True)
        smp = ops.state_sample(mc, lc, eps.cuda())
        (smp * cot_s.cuda()).sum().backward()
        got.update(smp=smp.detach().cpu(), smp_mean=mc.grad.cpu(), smp_L=lc.grad.cpu())
    assert got.keys() == r32.keys()
    for k in got:
        tol = TOL_STATE if k in ("ent", "smp") else TOL_G
        assert_parity("state D=%d R=%d S=%d %s" % (D, R, S, k), got[k], r32[k], lambda k=k: r64()[k], tol)


# ---- the fused shooting step -----------------------------------------------------------------------------------------
SHOOT_M, SHOOT_S = 37, 33    # odd: the last feature pair is half empty


def _zigzag_states(D, S_mc, N, T, lo, hi, seed):
    """sampled states: every sequence steps between two points c = +-(0.4 .. 0.8) apart per dimension (plus 0.02 noise),
    so that the end point of one interval (0.07 long) stays well away from the next state -- the Laplace constraint's
    gradient is the sign of their difference, which a near tie would leave to rounding. Spread over [lo, hi)."""
    rng = np.random.default_rng(seed)
    start = rng.uniform(lo, hi, size=(S_mc, N, 1, D))
    c = rng.uniform(0.4, 0.8, size=(S_mc, N, 1, D)) * np.where(rng.uniform(size=(S_mc, N, 1, D)) < 0.5, -1, 1)
    t = (np.arange(T) % 2).reshape(1, 1, T, 1)
    return torch.tensor(start + t * c + 0.02 * rng.normal(size=(S_mc, N, T, D)), dtype=torch.float32)


def _launch_shape(rows_launch, cut):
    """-> (S_mc, N, T, rows): a batch whose launch covers ``rows_launch`` rows, all of them or (cut) a range that starts
    inside a sequence of the first sample and ends inside a sequence of the second"""
    S_mc, N = 2, 3
    if not cut:
        T = -(-rows_launch // (S_mc * N))
        return S_mc, N, T, None
    T = rows_launch // 4 + 7
    lo = T + T // 2 + 1
    hi = lo + rows_launch
    assert lo % T and hi % T and lo < N * T < hi <= S_mc * N * T
    return S_mc, N, T, (lo, hi)


def _shoot_names(D, mapping):
    if mapping == "warp":
        return ["rk4_fwd_warp_kernel<%d, true>" % D, "rk4_bwd_warp_kernel<%d, true>" % D]
    if mapping == "tc":
        return ["rk4_fwd_h_kernel<%d, true>" % D, "rk4_bwd_mma_kernel<%d, true, true>" % D]
    R = rows_per_thread(D) if mapping == "wide" else 1
    return ["rk4_fwd_kernel<%d, %d, true>" % (D, R), "rk4_bwd_kernel<%d, %d, true>" % (D, R)]


def _laplace_margin(gp, c, ss, si, rows, T):
    """the smallest |ss[t+1] - pred[t]| over the pairs of the range (the kernel's end points)"""
    from gaussian_process_odes_b200 import ops
    S_mc, N, T, D = ss.shape
    lo, hi = (0, S_mc * N * T) if rows is None else rows
    with torch.no_grad():
        _, _, pred = ops.shooting_step(ss.cuda(), si['t2'].cuda(), *cuda_args(gp, c), si['ys'].cuda(), si['W'].cuda(),
                                       None, si['lik_var'].cuda(), si['scale'].cuda(), laplace=True, rows=rows,
                                       want_pred=True)
    x = ss.reshape(-1, D).cuda()
    r = torch.arange(lo, hi, device="cuda")
    keep = (r % T) < T - 1
    return float((x[(r + 1).clamp(max=x.shape[0] - 1)] - pred).abs()[keep].min())


def _shoot_case(D, M, S, S_mc, N, T, rows, Dobs, bias, laplace, halo, names, seed, absent=()):
    """ops.shooting_step once under the profiler against util.shoot_oracle: both sums and every gradient, lik_var's
    included"""
    B = S_mc * N * T
    gp, c, _ = _problem(D, M, S, 8, seed)
    side = math.ceil(M ** (1.0 / D) - 1e-9)
    ss = _zigzag_states(D, S_mc, N, T, -0.5, side - 0.5, seed)
    si = shoot_inputs(D, S_mc, N, T, seed, Dobs=Dobs, bias=bias)
    a_ll, a_c = 0.7, 1.3
    if laplace:
        assert _laplace_margin(gp, c, ss, si, rows, T) > 1e-2
    (ll, cons, got), kernels = profiled(lambda: shoot_cuda(gp, c, ss, si, a_ll, a_c, laplace=laplace, rows=rows,
                                                           halo=halo))
    for n in names:
        grids_of(kernels, n)
    for n in absent:
        with pytest.raises(AssertionError):
            grids_of(kernels, n)
    chunk = _chunk(D, M)
    kw = dict(laplace=laplace, rows=rows, halo=halo)
    sums32, ref32 = shoot_oracle(gp, c, ss, si, a_ll, a_c, torch.float32, chunk, **kw)
    ref64 = lazy(lambda: shoot_oracle(gp, c, ss, si, a_ll, a_c, torch.float64, chunk, **kw))
    name = "shoot D=%d M=%d S=%d B=%d rows=%s Dobs=%d bias=%d %s halo=%d" % (
        D, M, S, B, rows, Dobs, bias, "laplace" if laplace else "gauss", halo)
    assert_parity(name + " sums", torch.stack([ll, cons]).double(), sums32, lambda: ref64()[0], TOL_GRAD)
    assert_grads(name, got, ref32, lambda: ref64()[1], TOL_GRAD, keys=SHOOT_KEYS)
    if rows is not None:   # rows outside the range and past its neighbour get nothing
        g = got['x'].reshape(B, D)
        assert not g[:rows[0]].any() and not g[rows[1] + 1:].any()


# (D, mapping, Dobs, bias, laplace, halo, cut)
SHOOT_CASES = [(1, "warp", 1, False, False, False, False), (3, "warp", 128, True, True, True, True),
               (8, "warp", 127, False, False, True, False), (6, "warp", 5, True, True, False, True),
               (2, "thread", 5, True, True, False, True), (7, "thread", 128, False, False, True, False),
               (8, "thread", 1, True, True, True, True), (2, "wide", 127, False, True, True, True),
               (3, "wide", 1, True, False, False, False), (5, "wide", 128, True, False, True, True),
               (4, "tc", 128, True, False, True, True), (5, "tc", 1, False, True, False, False),
               (5, "tc", 127, True, False, True, True)]


@pytest.mark.parametrize("D,mapping,Dobs,bias,laplace,halo,cut", SHOOT_CASES, ids=lambda v: str(v))
def test_shooting_step_against_the_oracle(D, mapping, Dobs, bias, laplace, halo, cut):
    """the fused epilogue on the warp, row-per-thread, wide (tensor cores off at D = 4, 5) and tensor-core forward
    (with the row-sum adjoint) mappings"""
    sms = _sms()
    rows_launch = {"warp": 301, "thread": WARP_MAX_ROWS + 229, "wide": (wide_min_rows(D, sms) or 0) + 77,
                   "tc": (mma_min_rows(D, sms) or 0) + 77}[mapping]
    S_mc, N, T, rows = _launch_shape(rows_launch, cut)
    B_launch = S_mc * N * T if rows is None else rows[1] - rows[0]
    use_tc = mapping != "wide"
    assert selected_mapping(D, B_launch, sms, use_tc) == {"warp": 0, "thread": 1, "wide": rows_per_thread(D),
                                                          "tc": "mma"}[mapping]
    absent = ["param_grad_kernel<%d>" % D] if mapping == "tc" else []
    with tensor_cores(use_tc):
        _shoot_case(D, SHOOT_M, SHOOT_S, S_mc, N, T, rows, Dobs, bias, laplace, halo, _shoot_names(D, mapping),
                    17 * D + Dobs + int(laplace), absent=absent)


@pytest.mark.parametrize("D", [2, 5])
def test_shooting_step_empty_range(D):
    """rows = (k, k): zero sums, zero gradients everywhere (lik_var's included), no end points"""
    from gaussian_process_odes_b200 import ops
    S_mc, N, T = 2, 3, 40
    gp, c, _ = _problem(D, SHOOT_M, SHOOT_S, 8, 5 + D)
    ss = _zigzag_states(D, S_mc, N, T, 0.0, 2.0, D)
    si = shoot_inputs(D, S_mc, N, T, D, Dobs=7)
    for k in (0, N * T + 5, S_mc * N * T):
        args = cuda_args(gp, c, True)
        sc = ss.cuda().requires_grad_(True)
        lv = si['lik_var'].cuda().requires_grad_(True)
        ll, cons, pred = ops.shooting_step(sc, si['t2'].cuda(), *args, si['ys'].cuda(), si['W'].cuda(),
                                           si['bias'].cuda(), lv, si['scale'].cuda(), rows=(k, k), want_pred=True)
        (0.7 * ll + 1.3 * cons).backward()
        torch.cuda.synchronize()
        assert float(ll) == 0.0 and float(cons) == 0.0 and tuple(pred.shape) == (0, D)
        for name, g in (("ss", sc.grad), ("Z", args[0].grad), ("ell", args[1].grad), ("var", args[2].grad),
                        ("nu", args[3].grad), ("lik_var", lv.grad)):
            assert g is not None and not g.any(), (k, name)


# ---- the bench shape -------------------------------------------------------------------------------------------------
def _epilogue_ref(pred, ss, si, lo, T, a_ll, dtype):
    """the two sums and a_ll d(ll)/d var of the epilogue evaluated on given end points ``pred`` (rows lo..), float64 or
    float32 torch on the device"""
    B, D = pred.shape
    Dobs = si['W'].shape[1]
    x = ss.reshape(-1, D).cuda()
    S_mc, N = ss.shape[0], ss.shape[1]
    r = torch.arange(lo, lo + B, device="cuda")
    ys = si['ys'].cuda().reshape(N * T, Dobs)[r % (N * T)].to(dtype)
    var = si['lik_var'].cuda().to(dtype).requires_grad_(True)
    p = pred.to(dtype)
    ll = O.gauss_loglik(p @ si['W'].cuda().to(dtype) + si['bias'].cuda().to(dtype), ys, var).sum()
    keep = ((r % T) < T - 1).to(dtype).unsqueeze(1)
    nxt = x[(r + 1).clamp(max=x.shape[0] - 1)].cuda().to(dtype)
    cons = (cons_logprob(nxt, p, si['scale'].cuda().to(dtype), False) * keep).sum()
    (a_ll * ll).backward()
    return torch.stack([ll.detach(), cons]).double().cpu(), var.grad.cpu()


def _ss_rows_oracle(gp, c, ss, si, idx, T, a_ll, a_c, dtype):
    """the gradient of a_ll ll + a_c cons w.r.t. the sampled states of rows ``idx``: their own interval (observation and
    the constraint on the next state) and the constraint of the previous row's interval, for which they are the
    next state"""
    D = ss.shape[-1]
    x = ss.reshape(-1, D)
    B = x.shape[0]
    Dobs = si['W'].shape[1]
    step = oracle_rk4(si['t2'])
    l, cc = oracle_leaves(gp, c, x[idx], dtype, "cuda")
    pred = step(l, cc)[1]
    with torch.no_grad():
        lp, cp = oracle_leaves(gp, c, x[(idx - 1).clamp(min=0)], dtype, "cuda")
        pred_prev = step(lp, cp)[1]
    t = idx % T
    N = ss.shape[1]
    dev = lambda v: v.to("cuda", dtype)
    ys = dev(si['ys'].reshape(N * T, Dobs)[idx % (N * T)])
    ll = O.gauss_loglik(pred @ dev(si['W']) + dev(si['bias']), ys, dev(si['lik_var'])).sum()
    scale = dev(si['scale'])
    nxt = dev(x[(idx + 1).clamp(max=B - 1)])
    cons = (cons_logprob(nxt, pred, scale, False) * dev(t < T - 1).unsqueeze(1)).sum() + \
           (cons_logprob(l['x'], pred_prev, scale, False) * dev(t > 0).unsqueeze(1)).sum()
    (a_ll * ll + a_c * cons).backward()
    return l['x'].grad.cpu()


def test_shooting_step_at_the_bench_shape():
    """10^6 segments (D = 5, M = 100, S = 256, S_mc = 5, N = 16, T = 12 500, Dobs = 50): tensor-core forward, row-sum
    adjoint. Both sums and the lik_var gradient against a float64 epilogue on the kernel's own end points; the ss
    gradient of a few hundred rows (sequence and sample ends included) against the oracle"""
    from gaussian_process_odes_b200 import ops
    D, M, S, S_mc, N, T, Dobs = 5, 100, 256, 5, 16, 12500, 50
    B = S_mc * N * T
    seed = 2024
    gp, c, _ = _problem(D, M, S, 8, seed)
    side = math.ceil(M ** (1.0 / D) - 1e-9)
    ss = _zigzag_states(D, S_mc, N, T, -0.5, side - 0.5, seed)
    si = shoot_inputs(D, S_mc, N, T, seed, Dobs=Dobs)
    a_ll, a_c = 0.7, 1.3

    def run():
        args = cuda_args(gp, c, True)
        sc = ss.cuda().requires_grad_(True)
        lv = si['lik_var'].cuda().requires_grad_(True)
        ll, cons, pred = ops.shooting_step(sc, si['t2'].cuda(), *args, si['ys'].cuda(), si['W'].cuda(),
                                           si['bias'].cuda(), lv, si['scale'].cuda(), want_pred=True)
        (a_ll * ll + a_c * cons).backward()
        return torch.stack([ll.detach(), cons.detach()]).double().cpu(), pred, sc.grad, lv.grad.cpu()
    (sums, pred, g_ss, g_lv), kernels = profiled(run)
    for n in _shoot_names(D, "tc"):
        grids_of(kernels, n)
    r32 = _epilogue_ref(pred, ss, si, 0, T, a_ll, torch.float32)
    r64 = lazy(lambda: _epilogue_ref(pred, ss, si, 0, T, a_ll, torch.float64))
    assert_parity("bench sums", sums, r32[0], lambda: r64()[0], TOL_VALUE)
    assert_parity("bench grad lik_var", g_lv, r32[1], lambda: r64()[1], TOL_G)
    rng = np.random.default_rng(seed)
    idx = np.unique(np.concatenate([rng.choice(B, 300, replace=False),
                                    [0, 1, T - 1, T, N * T - 1, N * T, B - T, B - 1]]))
    idx = torch.as_tensor(idx)
    ref = lambda dt: _ss_rows_oracle(gp, c, ss, si, idx, T, a_ll, a_c, dt)
    assert_parity("bench grad ss rows", g_ss.reshape(B, D)[idx.cuda()].cpu(), ref(torch.float32),
                  lambda: ref(torch.float64), TOL_GRAD)


# ---- the epilogue at the shared-memory limit -------------------------------------------------------------------------
@pytest.mark.parametrize("dm", [0, 1])
def test_fused_tensor_core_forward_at_its_limit(dm):
    """D = 5, S = 256, Dobs = 128 on a tensor-core batch: at M* of shoot_tc_fwd the fused tensor-core forward runs, at
    M* + 1 the FFMA2 row-per-thread forward takes the batch; both match the oracle"""
    D, S = 5, 256
    M = max_inducing("shoot_tc_fwd", D, S) + dm
    assert max_inducing("fwd", D, S) is None and max_inducing("bwd", D, S) is None   # the FFMA2 kernels fit
    rows = mma_min_rows(D, _sms()) + 77
    S_mc, N, T, _ = _launch_shape(rows, False)
    assert rows <= S_mc * N * T < wide_min_rows(D, _sms())
    fwd_tc, fwd_thread = "rk4_fwd_h_kernel<%d, true>" % D, "rk4_fwd_kernel<%d, 1, true>" % D
    names = [fwd_thread if dm else fwd_tc, "rk4_bwd_kernel<%d, 1, true>" % D]
    _shoot_case(D, M, S, S_mc, N, T, None, SHOOT_MAX_DOBS, True, False, False, names, 500 + M,
                absent=[fwd_tc] if dm else [fwd_thread])


def test_fused_forward_at_its_limit_d8():
    """D = 8, S = 512, Dobs = 128, row per thread: at M* of shoot_fwd the fused step runs and matches the oracle"""
    D, S = 8, 512
    M = max_inducing("shoot_fwd", D, S)
    S_mc, N, T, _ = _launch_shape(WARP_MAX_ROWS + 229, False)
    _shoot_case(D, M, S, S_mc, N, T, None, SHOOT_MAX_DOBS, False, True, False,
                ["rk4_fwd_kernel<%d, 1, true>" % D, "rk4_bwd_kernel<%d, 1, true>" % D], 800 + M)


def test_fused_forward_past_its_limit_d8():
    """D = 8, S = 512, Dobs = 128, M = M* + 1 of shoot_fwd (the plain forward and the row-per-thread adjoint still
    fit): ops.shooting_step raises "does not fit" and leaves no pending CUDA error; UniformSequenceModel trains through
    the unfused chain on the same GP draw, its loss and gradients those of fuse_elbo = False; under row sharding the
    refusal propagates"""
    from gaussian_process_odes_b200 import builders, ops
    from gaussian_process_odes_b200._lib import GpodeError
    from gaussian_process_odes_b200.misc.mocap_utils import LinearProjection
    D, S, Dobs = 8, 512, SHOOT_MAX_DOBS
    M = max_inducing("shoot_fwd", D, S) + 1
    assert M <= max_inducing("fwd", D, S) and M <= max_inducing("bwd", D, S)
    S_mc, N, T, _ = _launch_shape(WARP_MAX_ROWS + 229, False)
    gp, c, _ = _problem(D, M, S, 8, 900)
    ss = _zigzag_states(D, S_mc, N, T, 0.0, 2.0, 900)
    si = shoot_inputs(D, S_mc, N, T, 900, Dobs=Dobs)
    with pytest.raises(GpodeError, match="does not fit"):
        ops.shooting_step(ss.cuda(), si['t2'].cuda(), *cuda_args(gp, c), si['ys'].cuda(), si['W'].cuda(),
                          si['bias'].cuda(), si['lik_var'].cuda(), si['scale'].cuda())
    small = _problem(2, 16, 17, 8, 3, "0.3")
    ts = torch.tensor([0.0, 0.1], dtype=torch.float32)
    xs = ops.rk4_integrate(small[2].cuda(), ts.cuda(), *cuda_args(*small[:2]))
    torch.cuda.synchronize()
    ref = oracle_rk4(ts)(*oracle_leaves(small[0], small[1], small[2], torch.float32, "cuda")).detach().cpu()
    assert relerr(xs.cpu(), ref) <= 1e-4

    ys = si['ys'].cuda()
    ts_model = torch.arange(T, dtype=torch.float32, device="cuda") * 0.07
    out = []
    for fuse in (True, False):   # the GP draws come from numpy's global generator, the states from torch's
        torch.manual_seed(5)
        np.random.seed(5)
        model = builders.build_gpode_shooting(N, T, D, num_inducing=M, num_features=S, solver="rk4", D_obs=Dobs,
                                              projection=LinearProjection(si['W'].numpy())).cuda()
        model.fuse_elbo = fuse
        torch.manual_seed(6)
        np.random.seed(6)
        loss = builders.compute_loss_shooting(model, ys, ts_model, num_samples=S_mc)[0]
        loss.backward()
        grads = {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}
        out.append((loss.detach(), grads, model))
    (l_f, g_f, model), (l_u, g_u, _) = out
    assert torch.isfinite(l_f) and relerr(l_f, l_u) <= 1e-6, (float(l_f), float(l_u))
    assert g_f.keys() == g_u.keys() and len(g_f) >= 8
    for k in g_f:
        assert relerr(g_f[k], g_u[k]) <= 1e-5, k
    model.row_shard = (0, 2)   # a sharded step has no unfused form: the refusal itself is reported
    with pytest.raises(GpodeError, match="does not fit"):
        builders.compute_loss_shooting(model, ys, ts_model, num_samples=S_mc)
