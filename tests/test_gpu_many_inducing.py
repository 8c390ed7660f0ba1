"""-m gpu: the D = 1..8 integrators, adjoints and gradient sums above 160 inducing points, against the oracle.

Since the blocked whitening, training and prediction at D <= 8 run up to M = 2048. Every integrator CTA stages the packed
block (KS floats per inducing point) in shared memory, param_grad_kernel gets a second grid dimension
ceil(M / 256) from M = 256 on, and the tensor-core shooting adjoint sums the inducing-point gradients itself only while
its row sums fit. This file runs each launch mapping at M = 257, 1024 and 2048, each kernel family at its
shared-memory limit M* and at M* + 1 (tests/util.py SMEM_FAMILIES, checked on the CPU by test_many_inducing_cpu.py),
the param_grad / finalize geometry at every ragged M, batched prediction, the KL and the inducing sample, and the
refusal of blocks that do not fit.

Inducing points sit on a unit lattice (jittered by 0.05, lengthscales 0.7 +- 5%), so K(Z,Z) is well conditioned and nu
is the whitened weight training feeds the kernels (ops.whiten, blocked above M = 160); one set of cases uses
nu = 0.3 N(0,1). S is odd, so the last feature pair is half empty. Every case asserts the kernel that ran
(torch.profiler) and holds the result to the project's bars (TOL_VF, TOL_TRAJ, TOL_GRAD, float64-arbitrated)."""
import ctypes
import math

import numpy as np
import pytest
import torch

import gpode_oracle as O
from test_gpu_small_d_mappings import (WARP_MAX_ROWS, grids_of, mma_min_rows, profiled, rows_per_thread,
                                       selected_mapping, tensor_cores, wide_min_rows)
from test_gpu_small_d_mappings import dopri5_kernel as dopri5_kernel_name
from test_gpu_whiten_blocked import _lattice
from test_many_inducing_cpu import oversized_calls
from util import (GRAD_KEYS, TOL_GRAD, TOL_TRAJ, TOL_VF, assert_grads, assert_parity, chunked_oracle, cuda_args, cuda_grads,
                  lazy, max_inducing, oracle_dopri5, oracle_leaves, oracle_rk4, oracle_vf, relerr, shoot_cuda,
                  shoot_inputs, shoot_oracle, time_grid)

pytestmark = pytest.mark.gpu

S_SMALL = 33        # odd: 17 feature pairs, the last one half empty
WARP_ROWS = 301     # warp-per-row batches (ragged)
DP_BATCH = {"one_cta": 13, "warp": 777, "thread": 1101}


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _chunk(D, M):
    """oracle rows per chunk: the [D, rows, M] kernel matrices stay near 2^25 elements"""
    return max(1024, min(16384, (1 << 25) // (D * M)))


def _problem(D, M, S, B, seed, nu="whitened", centred=False):
    """lattice inducing points, Fourier features with angles of a few radians, x spread over the lattice's box;
    nu: 'whitened' (ops.whiten of u ~ N(0,1), what training feeds the kernels) or '0.3' (0.3 N(0,1)). centred: the
    lattice centred on the origin and x ~ 1.5 N(0,1), so that |x| stays O(1) -- dopri5's error norm scales with |x|,
    and at |x| ~ 1e3 (D = 1, M = 2048) float32 rounding alone decides its accept / reject steps"""
    from gaussian_process_odes_b200 import ops
    rng = np.random.default_rng(seed)
    t = lambda a: torch.tensor(np.asarray(a), dtype=torch.float32)
    side = math.ceil(M ** (1.0 / D) - 1e-9)
    gp = dict(Z=t(_lattice(D, M, seed) - ((side - 1) / 2 if centred else 0.0)), ell=t(0.7 * (1 + 0.05 * rng.uniform(-1, 1, size=(D, D)))),
              var=t(0.5 + rng.uniform(size=D)))
    c = dict(rff_omega=t(rng.normal(size=(D, S, D)) / side), rff_phase=t(rng.uniform(size=(1, S, D)) * 2 * np.pi),
             rff_weights=t(rng.normal(size=(S, D))))
    if nu == "whitened":
        u = t(rng.normal(size=(M, D))).cuda()
        with torch.no_grad():
            c['nu'] = ops.whiten(gp['Z'].cuda(), gp['ell'].cuda(), gp['var'].cuda(), u, c['rff_omega'].cuda(),
                                 c['rff_phase'].cuda(), c['rff_weights'].cuda()).cpu().reshape(D, M, 1)
    else:
        c['nu'] = t(rng.normal(size=(D, M, 1)) * float(nu))
    x = t(rng.normal(size=(B, D)) * 1.5 if centred else rng.uniform(-0.5, side - 0.5, size=(B, D)))
    return gp, c, x


def _batch(D, mapping):
    sms = _sms()
    return {"warp": WARP_ROWS, "thread": WARP_MAX_ROWS + 229, "wide": (wide_min_rows(D, sms) or 0) + 77,
            "tc": (mma_min_rows(D, sms) or 0) + 77}[mapping]


def _names(entry, D, mapping):
    """(forward kernel, adjoint kernel) the launchers pick for this mapping"""
    R = rows_per_thread(D) if mapping == "wide" else 1
    if mapping == "tc":
        return (("vf_fwd_h_kernel<%d>" % D, "vf_bwd_mma_kernel<%d>" % D) if entry == "vf" else
                ("rk4_fwd_h_kernel<%d, false>" % D, "rk4_bwd_mma_kernel<%d, false, false>" % D))
    if mapping == "warp":
        return (("vf_fwd_warp_kernel<%d>" % D, "vf_bwd_warp_kernel<%d>" % D) if entry == "vf" else
                ("rk4_fwd_warp_kernel<%d, false>" % D, "rk4_bwd_warp_kernel<%d, false>" % D))
    return (("vf_fwd_kernel<%d, %d>" % (D, R), "vf_bwd_kernel<%d, %d>" % (D, R)) if entry == "vf" else
            ("rk4_fwd_kernel<%d, %d, false>" % (D, R), "rk4_bwd_kernel<%d, %d, false>" % (D, R)))


def _vf_rk4(entry, D, M, S, B, seed, nu, names, use_tc=True, grad=True):
    """the CUDA op (forward + all five gradients, or the forward alone) once under the profiler against the chunked
    oracle; ``names``: kernels that must have launched"""
    from gaussian_process_odes_b200 import ops
    gp, c, x = _problem(D, M, S, B, seed, nu)
    if entry == "vf":
        fn, ofn, tol, row_dim = (lambda xc, a: ops.vector_field(xc, *a)), oracle_vf, TOL_VF, 0
        cot = torch.tensor(np.random.default_rng(seed).normal(size=(B, D)), dtype=torch.float32)
    else:
        ts = time_grid(3, 0.1, seed)
        fn, ofn, tol, row_dim = (lambda xc, a: ops.rk4_integrate(xc, ts.cuda(), *a)), oracle_rk4(ts), TOL_TRAJ, 1
        cot = torch.tensor(np.random.default_rng(seed).normal(size=(3, B, D)), dtype=torch.float32)
    name = "%s D=%d M=%d S=%d B=%d nu=%s" % (entry, D, M, S, B, nu)
    with tensor_cores(use_tc):
        if grad:
            (out, got), kernels = profiled(lambda: cuda_grads(fn, gp, c, x, cot))
        else:
            with torch.no_grad():
                out, kernels = profiled(lambda: fn(x.cuda(), cuda_args(gp, c)))
    for n in names:
        grids_of(kernels, n)
    chunk = _chunk(D, M)
    if not grad:   # the oracle's forward alone
        ref = lambda dt: torch.cat([ofn(*oracle_leaves(gp, c, x[r:r + chunk], dt, "cuda")).detach().cpu()
                                    for r in range(0, B, chunk)], row_dim)
        assert_parity(name, out.cpu(), ref(torch.float32), lambda: ref(torch.float64), tol)
        return kernels
    out32, ref32 = chunked_oracle(ofn, gp, c, x, cot, torch.float32, row_dim, chunk=chunk)
    ref64 = lazy(lambda: chunked_oracle(ofn, gp, c, x, cot, torch.float64, row_dim, chunk=chunk))
    assert_parity(name, out.cpu(), out32, lambda: ref64()[0], tol)
    assert_grads(name, got, ref32, lambda: ref64()[1], TOL_GRAD)
    return kernels


# ---- every mapping at large M -------------------------------------------------------------------------------------
DIMS = (1, 2, 4, 5, 7, 8)


def _mappings(D):
    return ["warp", "thread"] + (["wide"] if rows_per_thread(D) > 1 else []) + (["tc"] if D in (4, 5) else [])


MAPPING_CASES = [(e, D, m, M, "whitened") for D in DIMS for m in _mappings(D)
                 for e, M in (("vf", 2048), ("rk4", 1024))] + \
                [(e, D, "warp", 257, nu) for D in DIMS for e in ("vf", "rk4") for nu in ("whitened", "0.3")]


@pytest.mark.parametrize("entry,D,mapping,M,nu", MAPPING_CASES, ids=lambda v: str(v))
def test_every_mapping_at_large_m(entry, D, mapping, M, nu):
    """vf and rk4 forward + adjoint on the warp, row-per-thread, wide and tensor-core mappings (the wide FFMA2 kernels
    at D = 4, 5 with the tensor cores switched off), at M = 2048 (vf) and 1024 (rk4), and on the warp mapping at
    M = 257 with both kinds of nu"""
    assert max_inducing("bwd_warp", D, S_SMALL) is None   # every kernel fits M = 2048 at this S
    B = _batch(D, mapping)
    use_tc = mapping == "tc" or mapping in ("warp", "thread")
    assert selected_mapping(D, B, _sms(), use_tc) == {"warp": 0, "thread": 1, "wide": rows_per_thread(D),
                                                      "tc": "mma"}[mapping]
    seed = 1000 * D + M + len(mapping) + (entry == "rk4") * 7 + (nu == "0.3") * 3
    _vf_rk4(entry, D, M, S_SMALL, B, seed, nu, _names(entry, D, mapping), use_tc=use_tc)


def _dopri5_case(D, M, S, B, seed, ts, rtol=1e-6, nu="whitened"):
    """dopri5 forward + discrete adjoint once under the profiler, against the oracle's solve"""
    from gaussian_process_odes_b200 import ops
    gp, c, x = _problem(D, M, S, B, seed, nu, centred=True)
    cot = torch.tensor(np.random.default_rng(seed).normal(size=(len(ts), B, D)), dtype=torch.float32)
    stats = []

    def run(xc, a):
        xs, st = ops.dopri5_integrate(xc, ts.cuda(), *a, rtol=rtol, atol=rtol)
        stats.append(st)
        return xs
    (xs, got), kernels = profiled(lambda: cuda_grads(run, gp, c, x, cot))
    out32, ref32, st = oracle_dopri5(gp, c, x, ts, cot, torch.float32, rtol=rtol, atol=rtol)
    ref64 = lazy(lambda: oracle_dopri5(gp, c, x, ts, cot, torch.float64, rtol=rtol, atol=rtol))
    nfe, acc, rej, status = [int(v) for v in stats[-1].cpu()]
    assert status == 0 and abs(acc - st['accepted']) <= 1 and abs(rej - st['rejected']) <= 1, (acc, rej, st)
    name = "dopri5 D=%d M=%d B=%d" % (D, M, B)
    assert_parity(name, xs.cpu(), out32, lambda: ref64()[0], TOL_TRAJ)
    assert_grads(name, got, ref32, lambda: ref64()[1], 2e-4)   # the dopri5 gradient bar of the mapping tests
    return kernels


DOPRI5_CASES = [(D, mapping, (1024, 2048)[(i + j) % 2]) for i, D in enumerate(DIMS)
                for j, mapping in enumerate(DP_BATCH)]


@pytest.mark.parametrize("D,mapping,M", DOPRI5_CASES)
def test_dopri5_forms_and_adjoint_at_large_m(D, mapping, M):
    """dopri5_kernel in one CTA, warp per row and row per thread, and dopri5_bwd_kernel after it, at M = 1024 / 2048"""
    B = DP_BATCH[mapping]
    ts = torch.tensor([0.0, 0.15, 0.4], dtype=torch.float32)
    kernels = _dopri5_case(D, M, S_SMALL, B, 31 * D + M + B, ts)
    grids_of(kernels, dopri5_kernel_name(D, B))
    grids_of(kernels, "dopri5_bwd_kernel<%d>" % D)
    grids_of(kernels, "param_grad_kernel<%d>" % D)


# ---- the fused shooting step (rk4_*_kernel<..., kShoot = true>) ----------------------------------------------------
def _shoot_case(D, M, S, S_mc, N, T, seed, names, absent=(), monkeypatch=None, vrows=False):
    """the fused step against the oracle; vrows: force the virtual-row adjoint (gpode_shoot_bwd with vrows +
    gpode_param_grad) where the tensor-core adjoint would sum the inducing-point gradients itself"""
    from gaussian_process_odes_b200 import _lib
    B = S_mc * N * T
    gp, c, x = _problem(D, M, S, B, seed)
    ss = x.reshape(S_mc, N, T, D)
    si = shoot_inputs(D, S_mc, N, T, seed)
    a_ll, a_c = 0.7, 1.3
    if vrows:
        monkeypatch.setattr(_lib.load(), "gpode_shoot_bwd_vrows", lambda D_, M_, S_, n: 4 * n)
    (ll, cons, got), kernels = profiled(lambda: shoot_cuda(gp, c, ss, si, a_ll, a_c))
    if vrows:
        monkeypatch.undo()
    for n in names:
        grids_of(kernels, n)
    for n in absent:
        with pytest.raises(AssertionError):
            grids_of(kernels, n)
    chunk = _chunk(D, M)
    sums32, ref32 = shoot_oracle(gp, c, ss, si, a_ll, a_c, torch.float32, chunk)
    ref64 = lazy(lambda: shoot_oracle(gp, c, ss, si, a_ll, a_c, torch.float64, chunk))
    name = "shoot D=%d M=%d S=%d B=%d%s" % (D, M, S, B, " vrows" if vrows else "")
    assert_parity(name + " sums", torch.stack([ll, cons]).double(), sums32, lambda: ref64()[0], TOL_GRAD)
    assert_grads(name, got, ref32, lambda: ref64()[1], TOL_GRAD, keys=GRAD_KEYS + ("lik_var",))
    return got


SHOOT_CASES = [(D, mapping) for D in DIMS for mapping in ("warp", "thread")]


@pytest.mark.parametrize("D,mapping", SHOOT_CASES)
def test_shooting_step_at_m1024(D, mapping):
    """rk4_fwd_*_kernel / rk4_bwd_*_kernel <..., kShoot = true> warp per row and row per thread at M = 1024"""
    S_mc, N, T = (2, 3, 50) if mapping == "warp" else (2, 3, 2769)
    B = S_mc * N * T
    assert selected_mapping(D, B, _sms()) == (0 if mapping == "warp" else 1)
    names = (["rk4_fwd_warp_kernel<%d, true>" % D, "rk4_bwd_warp_kernel<%d, true>" % D] if mapping == "warp" else
             ["rk4_fwd_kernel<%d, 1, true>" % D, "rk4_bwd_kernel<%d, 1, true>" % D])
    _shoot_case(D, 1024, S_SMALL, S_mc, N, T, 7 * D + B, names + ["param_grad_kernel<%d>" % D])


# ---- row sums against virtual rows at the row-sum limit (D = 4, 5) --------------------------------------------------
S_LIMIT = 129       # odd; the row-sum limit is M* = 283 (D = 4) and 182 (D = 5) here
ROW_SUM_CASES = [(D, dm) for D in (4, 5) for dm in (0, 1)]


@pytest.mark.parametrize("D,dm", ROW_SUM_CASES)
def test_row_sums_and_virtual_rows_at_the_limit(D, dm, monkeypatch):
    """the tensor-core shooting adjoint at M* of the row-sum family sums the inducing-point gradients itself (no
    param_grad_kernel); at M* + 1 it writes virtual rows for param_grad_kernel. Both match the oracle, and at M* the
    row sums match the same step with virtual rows forced"""
    from gaussian_process_odes_b200 import _lib
    M = max_inducing("tc_row_sums", D, S_LIMIT) + dm
    S_mc, N, T = 2, 3, 9500
    B = S_mc * N * T
    assert B >= mma_min_rows(D, _sms())
    assert (_lib.load().gpode_shoot_bwd_vrows(D, M, S_LIMIT, B) == 0) == (dm == 0)
    fwd = "rk4_fwd_h_kernel<%d, true>" % D
    if dm == 0:
        rs = _shoot_case(D, M, S_LIMIT, S_mc, N, T, 40 + D, [fwd, "rk4_bwd_mma_kernel<%d, true, true>" % D],
                         absent=["param_grad_kernel<%d>" % D])
        vr = _shoot_case(D, M, S_LIMIT, S_mc, N, T, 40 + D, [fwd, "rk4_bwd_mma_kernel<%d, true, false>" % D,
                                                               "param_grad_kernel<%d>" % D],
                         monkeypatch=monkeypatch, vrows=True)
        for k in ("x", "Z", "ell", "var", "nu"):
            assert relerr(rs[k], vr[k]) <= TOL_GRAD, k
    else:
        _shoot_case(D, M, S_LIMIT, S_mc, N, T, 40 + D, [fwd, "rk4_bwd_mma_kernel<%d, true, false>" % D,
                                                          "param_grad_kernel<%d>" % D])


# ---- each kernel family at its shared-memory limit ------------------------------------------------------------------
def _limit_cases():
    """(family, D, S, M*) for every family whose block can outgrow 227 KB at S = 129 or 512 (the row-sum family is
    test_row_sums_and_virtual_rows_at_the_limit's)"""
    out = []
    for S in (S_LIMIT, 512):
        for family, Ds in (("fwd", range(1, 9)), ("dopri5_fwd", range(1, 9)), ("bwd", range(1, 9)),
                           ("bwd_warp", range(1, 9)), ("tc_fwd", (4, 5)), ("tc_bwd", (4, 5))):
            for D in Ds:
                m = max_inducing(family, D, S)
                if m is not None and m >= 1:
                    out.append((family, D, S, m))
    return out


LIMIT_CASES = [c + (dm,) for c in _limit_cases() for dm in (0, 1)]


@pytest.mark.parametrize("family,D,S,M_star,dm", LIMIT_CASES, ids=lambda v: str(v))
def test_kernel_family_at_its_limit(family, D, S, M_star, dm):
    """At M* the family's kernel runs and matches the oracle; at M* + 1 the launcher hands the batch to the next
    mapping (tensor cores -> FFMA2) or refuses with "does not fit". Forward kernels whose adjoint cannot fit at this S
    are checked forward only."""
    from gaussian_process_odes_b200._lib import GpodeError
    M = M_star + dm
    seed = 97 * D + M + S
    fits = lambda f: max_inducing(f, D, S) is None or M <= max_inducing(f, D, S)
    if family == "dopri5_fwd":
        from gaussian_process_odes_b200 import ops
        B = DP_BATCH["one_cta"]
        gp, c, x = _problem(D, M, S, B, seed)
        ts = torch.tensor([0.0, 0.2, 0.3], dtype=torch.float32)
        with torch.no_grad():
            if dm:
                for b in DP_BATCH.values():   # one CTA, cooperative warp per row, row per thread
                    with pytest.raises(GpodeError, match="does not fit"):
                        ops.dopri5_integrate(x[:1].expand(b, D).contiguous().cuda(), ts.cuda(), *cuda_args(gp, c))
                return
            (xs, _), kernels = profiled(lambda: ops.dopri5_integrate(x.cuda(), ts.cuda(), *cuda_args(gp, c)))
        grids_of(kernels, dopri5_kernel_name(D, B))
        out32 = oracle_dopri5(gp, c, x, ts, torch.zeros(3, B, D), torch.float32)[0]
        assert_parity("dopri5 fwd D=%d M=%d S=%d" % (D, M, S), xs.cpu(), out32,
                      lambda: oracle_dopri5(gp, c, x, ts, torch.zeros(3, B, D), torch.float64)[0], TOL_TRAJ)
        return
    if family in ("fwd", "bwd_warp"):
        B, mapping, nxt = WARP_ROWS, "warp", None
    elif family == "bwd":
        B, mapping, nxt = _batch(D, "thread"), "thread", None
    else:
        B, mapping, nxt = _batch(D, "tc"), "tc", "thread"
    assert selected_mapping(D, B, _sms()) == {"warp": 0, "thread": 1, "tc": "mma"}[mapping]
    fwd_name, bwd_name = _names("vf", D, mapping)
    grad = fits("bwd_warp" if mapping == "warp" else "bwd")   # an adjoint exists for this batch at this M
    if family == "fwd":
        grad = False
    if dm == 0:
        names = [fwd_name] + ([bwd_name] if family != "fwd" else [])
        if family == "tc_fwd" and not fits("tc_bwd"):
            names = [fwd_name, _names("vf", D, "thread")[1]]
        _vf_rk4("vf", D, M, S, B, seed, "whitened", names, grad=grad or family != "fwd")
    elif nxt is None:   # no other kernel for this batch: an argument error, before any CUDA call
        with pytest.raises(GpodeError, match="does not fit"):
            _vf_rk4("vf", D, M, S, B, seed, "whitened", [], grad=family != "fwd")
    else:               # the tensor-core kernel hands over to the FFMA2 row-per-thread kernel
        f_next, b_next = _names("vf", D, nxt)
        names = [f_next, b_next] if family == "tc_fwd" else [fwd_name if fits("tc_fwd") else f_next, b_next]
        _vf_rk4("vf", D, M, S, B, seed, "whitened", names)


# ---- param_grad and finalize geometry --------------------------------------------------------------------------------
PG_M = (255, 256, 257, 511, 512, 513, 515)   # param_grad's gy = ceil(M / 256) boundaries; 515 = 3 mod 4 (kFinM)


@pytest.mark.parametrize("M", PG_M)
@pytest.mark.parametrize("D", [3, 8])
def test_param_grad_geometry(D, M):
    """the virtual-row adjoint of the vector field (every row one virtual row) on the warp mapping: param_grad_kernel
    on a ragged y-grid and grads_finalize on a partial last group of inducing points"""
    kernels = _vf_rk4("vf", D, M, S_SMALL, WARP_ROWS, 5 * D + M, "whitened",
                      ["vf_bwd_warp_kernel<%d>" % D, "param_grad_kernel<%d>" % D, "grads_finalize_kernel"])
    assert len(grids_of(kernels, "param_grad_kernel<%d>" % D)) == 1


@pytest.mark.parametrize("M", [257, 513])
def test_param_grad_dev_after_dopri5(M):
    """gpode_dopri5_bwd_dev + gpode_param_grad_dev (the accepted-step count read on the device) at a ragged M, against
    the oracle and the host-count path"""
    from gaussian_process_odes_b200 import ops
    D, B = 3, DP_BATCH["warp"]
    ts = torch.tensor([0.0, 0.2, 0.45], dtype=torch.float32)
    seed = 61 + M
    saved, n_stats = ops.DEVICE_COUNT_MODE, len(ops.DEVICE_COUNT_STATS)
    ops.DEVICE_COUNT_MODE = True
    try:
        kernels = _dopri5_case(D, M, S_SMALL, B, seed, ts)
        assert len(ops.DEVICE_COUNT_STATS) == n_stats + 1, "the device-count path did not run"
    finally:
        ops.DEVICE_COUNT_MODE = saved
        del ops.DEVICE_COUNT_STATS[n_stats:]
    grids_of(kernels, "dopri5_bwd_kernel<%d>" % D)
    grids_of(kernels, "param_grad_kernel<%d>" % D)
    _dopri5_case(D, M, S_SMALL, B, seed, ts)   # the host-count path on the same problem


# ---- batched prediction at large M ----------------------------------------------------------------------------------
@pytest.mark.parametrize("method", ["rk4", "dopri5"])
@pytest.mark.parametrize("D", [2, 8])
def test_integrate_sets_at_m1024(D, method):
    """five draws of N = 3 trajectories in one launch: each draw bitwise the single-draw call, draw 0 against the
    oracle"""
    from gaussian_process_odes_b200 import ops
    M, n, N = 1024, 5, 3
    ts = torch.tensor([0.0, 0.1, 0.25, 0.3], dtype=torch.float32)
    probs = [_problem(D, M, S_SMALL, N, 300 + 10 * D + q) for q in range(n)]
    gp = dict(probs[0][0])
    for q in range(1, n):   # shared Z, ell, var; per-draw features and nu
        probs[q] = (gp, probs[q][1], probs[q][2])
    st = lambda k: torch.stack([p[1][k] for p in probs]).cuda()
    x0 = torch.stack([p[2] for p in probs]).cuda()
    Z, ell, var = gp['Z'].cuda(), gp['ell'].cuda(), gp['var'].cuda()
    with torch.no_grad():
        xs, _ = ops.integrate_sets(x0, ts.cuda(), Z, ell, var, st('nu').squeeze(3), st('rff_omega'),
                                   st('rff_phase').squeeze(1), st('rff_weights'), method=method)
        for q in range(n):
            args = cuda_args(*probs[q][:2])
            if method == "rk4":
                single = ops.rk4_integrate(x0[q], ts.cuda(), *args)
            else:
                single = ops.dopri5_integrate(x0[q], ts.cuda(), *args)[0]
            assert torch.equal(xs[q], single.permute(1, 0, 2)), "draw %d differs from the single-draw call" % q
    gp0, c0, x = probs[0]
    if method == "rk4":
        ref = lambda dt: chunked_oracle(oracle_rk4(ts), gp0, c0, x, torch.zeros(4, N, D), dt, 1)[0]
    else:
        ref = lambda dt: oracle_dopri5(gp0, c0, x, ts, torch.zeros(4, N, D), dt)[0]
    assert_parity("sets %s D=%d" % (method, D), xs[0].permute(1, 0, 2).cpu(), ref(torch.float32),
                  lambda: ref(torch.float64), TOL_TRAJ)


# ---- KL and inducing sample -------------------------------------------------------------------------------------------
def _variational(D, M, seed):
    rng = np.random.default_rng(seed)
    Um = torch.tensor(rng.normal(size=(M, D)), dtype=torch.float32)
    L = np.tril(rng.normal(size=(D, M, M)) * 0.3 / math.sqrt(M), -1) + \
        np.eye(M)[None] * np.exp(rng.normal(size=(D, M, 1)) * 0.2)
    Lp = O.packed_from_tril(torch.tensor(L, dtype=torch.float32))
    return Um, Lp


def _diag_slots(M):
    i = np.arange(M)
    return torch.as_tensor(i * (i + 1) // 2 + i)


@pytest.mark.parametrize("M", [161, 1023, 2048])
@pytest.mark.parametrize("D", [1, 5, 8])
def test_whitened_kl_and_inducing_sample(D, M):
    """ops.whitened_kl and ops.inducing_sample, forward and backward, against float64 torch (float32 torch
    arbitrates); the KL gradient separately on every diagonal slot of the packed factor"""
    from gaussian_process_odes_b200 import ops
    Um, Lp = _variational(D, M, 13 * D + M)
    eps = torch.tensor(np.random.default_rng(M).normal(size=(M, D)), dtype=torch.float32)
    g_u = torch.tensor(np.random.default_rng(M + 1).normal(size=(M, D)), dtype=torch.float32)

    def ref(dt):
        U, L = Um.cuda().to(dt).requires_grad_(True), Lp.cuda().to(dt).requires_grad_(True)
        kl = O.kl_whitened(U, O.tril_from_packed(L, M))
        kl.backward()
        gk = (U.grad.cpu(), L.grad.cpu())
        U.grad = L.grad = None
        u = O.sample_inducing(U, O.tril_from_packed(L, M), eps.cuda().to(dt))
        u.backward(g_u.cuda().to(dt))
        return kl.detach().cpu(), gk, u.detach().cpu(), (U.grad.cpu(), L.grad.cpu())
    r32, r64 = ref(torch.float32), lazy(lambda: ref(torch.float64))
    U, L = Um.cuda().requires_grad_(True), Lp.cuda().requires_grad_(True)
    kl = ops.whitened_kl(U, L)
    kl.backward()
    got_kl = (kl.detach().cpu(), (U.grad.cpu(), L.grad.cpu()))
    U.grad = L.grad = None
    u = ops.inducing_sample(U, L, eps.cuda())
    u.backward(g_u.cuda())
    got_u = (u.detach().cpu(), (U.grad.cpu(), L.grad.cpu()))
    name = "D=%d M=%d" % (D, M)
    diag = _diag_slots(M)
    assert_parity("kl " + name, got_kl[0], r32[0], lambda: r64()[0], 1e-6)
    assert_parity("kl grad Um " + name, got_kl[1][0], r32[1][0], lambda: r64()[1][0], 1e-6)
    assert_parity("kl grad L " + name, got_kl[1][1], r32[1][1], lambda: r64()[1][1], 1e-6)
    assert_parity("kl grad diag " + name, got_kl[1][1][:, diag], r32[1][1][:, diag], lambda: r64()[1][1][:, diag],
                  1e-6)
    off = torch.ones(M * (M + 1) // 2, dtype=torch.bool)
    off[diag] = False
    assert float(got_kl[1][1][:, off].sub(r32[1][1][:, off]).abs().max()) <= 1e-6 * float(r32[1][1].abs().max())
    assert_parity("u " + name, got_u[0], r32[2], lambda: r64()[2], TOL_VF)
    assert_parity("u grad Um " + name, got_u[1][0], r32[3][0], lambda: r64()[3][0], TOL_VF)
    assert_parity("u grad L " + name, got_u[1][1], r32[3][1], lambda: r64()[3][1], TOL_VF)


# ---- oversized blocks: clean argument errors --------------------------------------------------------------------------
def test_oversized_blocks_raise_and_leave_no_pending_error():
    """D = 8, S = 512, M = M*(family) + 1: every entry point that can exceed 227 KB raises "does not fit" once; the
    next call on the thread, a small valid rk4, succeeds and the device synchronises cleanly"""
    from gaussian_process_odes_b200 import _lib, ops
    lib = _lib.load()
    gp, c, x = _problem(2, 16, 17, 8, 3, "0.3")
    ts = torch.tensor([0.0, 0.1, 0.2], dtype=torch.float32).cuda()
    want = lambda: oracle_rk4(ts.cpu())(*oracle_leaves(gp, c, x, torch.float32, "cuda")).detach().cpu()
    ref = want()
    for name, family, call in oversized_calls(lib, ctypes.c_void_p(16)):
        M = max_inducing(family, 8, 512) + 1
        with pytest.raises(_lib.GpodeError, match="does not fit"):
            _lib.check(call(M))
        xs = ops.rk4_integrate(x.cuda(), ts, *cuda_args(gp, c))
        torch.cuda.synchronize()
        assert relerr(xs.cpu(), ref) <= TOL_TRAJ, name
