"""The D = 1..8 kernels on every launch mapping, against the oracle.

For D <= 8 every entry point picks one of several kernels from D and the batch size B (csrc/integrate_impl.cuh,
csrc/dopri5_impl.cuh):
- vector field / RK4, forward and adjoint: one warp per row up to 16 384 rows, then one row per thread, then R rows per
  thread once B >= SMs * 256 R (R = 4 at D <= 2, 2 at D = 3..5, none above); at D = 4, 5 the tensor-core kernels take
  over from SMs * 384 rows unless the options fwd_mma / bwd_mma are 0.
- dopri5 forward: one CTA (one warp per row) up to 16 rows, one warp per row up to 1024, then one row per thread. Its
  adjoint is one warp per row on min(ceil(B / 4), SMs * occupancy, 4096) CTAs, grid-stride beyond that.

Every case here derives B from the SM count and these rules, just above the threshold of its mapping and ragged (not a
multiple of 32, of 128 R or of the CTA's rows), runs its CUDA calls once under torch.profiler and asserts that the
intended kernel launched: if a threshold moves, the test fails instead of checking another kernel. M and S are odd, so
the last Fourier-feature pair is half empty and the last group of 32 records partial. nu is either 0.3 N(0,1) or the
whitened weights of clustered inducing points (|var nu| ~ 30..120, terms that cancel across inducing points).

The oracle is gpode_oracle as plain torch ops on the device in float32 and float64 (arbiter, tests/util.py), over row
chunks for the row-separable vector field and RK4; dopri5 runs unchunked, its error norm spans the batch."""
import contextlib
import json
import os
import re
import tempfile

import numpy as np
import pytest
import torch

import gpode_oracle as O
from util import (TOL_GRAD, TOL_TRAJ, TOL_VF, assert_grads, assert_parity, chunked_oracle, cuda_args, cuda_grads, lazy,
                  oracle_cache, oracle_dopri5, oracle_rk4, oracle_vf, relerr, time_grid)

# ---- the launchers' rules, restated -----------------------------------------------------------------------------------
WARP_MAX_ROWS = 16384   # kWarpPathMaxRows: above it the row-per-thread kernels
THREADS = 128           # kThreads: a CTA of the row-per-thread kernels holds 128 R rows
H_THREADS = 384         # kHThreads = kHFThreads: the tensor-core kernels take over at SMs * 384 rows (D = 4, 5)
DP_ONE_CTA_ROWS = 16    # kDpOneCtaRows: dopri5 in one CTA
DP_WARP_MAX_ROWS = 1024  # dopri5 warp per row up to here, row per thread above
DP_BWD_WARPS = 4        # kDpThreads / 32: rows in flight per CTA of dopri5_bwd_kernel
DP_BWD_MAX_GRID = 4096  # GPODE_ACC_CAP_AV: one accumulator row per CTA
MAX_CTAS_PER_SM = 16    # 2048 threads / 128: an upper bound of the occupancy of a 128-thread kernel
CHUNK = 16384           # oracle rows per chunk


def rows_per_thread(D):
    """RowsFwd<D> = RowsBwd<D>: the R of the wide kernels"""
    return 4 if D <= 2 else (2 if D <= 5 else 1)


def wide_min_rows(D, sms):
    """use_wide<D, R>: B >= SMs * 2 * 128 * R (no wide kernel when R = 1)"""
    R = rows_per_thread(D)
    return sms * 2 * THREADS * R if R > 1 else None


def mma_min_rows(D, sms):
    """use_mma_fwd / use_mma_bwd at D = 4, 5 (kMmaBwd<D>)"""
    return sms * H_THREADS if D in (4, 5) else None


def mapping_batch(D, mapping, sms):
    """-> (B, R): just above the threshold of the mapping, with a ragged tail"""
    if mapping == "thread":
        return WARP_MAX_ROWS + 229, 1
    return wide_min_rows(D, sms) + 77, rows_per_thread(D)


def selected_mapping(D, B, sms, tensor_cores=True):
    """the rows per thread the launcher picks for B rows (0: warp per row, 'mma': tensor cores)"""
    mma = mma_min_rows(D, sms)
    if tensor_cores and mma is not None and B >= mma:
        return "mma"
    if B <= WARP_MAX_ROWS:
        return 0
    wide = wide_min_rows(D, sms)
    return rows_per_thread(D) if wide is not None and B >= wide else 1


def dopri5_kernel(D, B):
    """the forward kernel launch_dopri5 picks: dopri5_kernel<D, kWarp, kSets>"""
    if B <= DP_ONE_CTA_ROWS:
        return "dopri5_kernel<%d, true, true>" % D
    return "dopri5_kernel<%d, %s, false>" % (D, "true" if B <= DP_WARP_MAX_ROWS else "false")


def dopri5_two_pass_batch(sms, tail=77):
    """rows for which every warp of the dopri5 adjoint runs >= 2 rows at the largest grid the launcher may choose"""
    return 2 * DP_BWD_WARPS * min(sms * MAX_CTAS_PER_SM, DP_BWD_MAX_GRID) + tail


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- the kernels a call launched ------------------------------------------------------------------------------------
def profiled(fn):
    """fn() once under torch.profiler (CUDA activities) -> (fn's result, [(kernel name, grid x)] in launch order)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            events = json.load(fh)["traceEvents"]
    return out, [(e["name"], e["args"]["grid"][0]) for e in events if e.get("cat") == "kernel"]


def grids_of(kernels, name):
    """the grid sizes of every launch of kernel ``name`` (e.g. 'rk4_bwd_kernel<7, 1, false>'); asserts >= 1 launch.
    The trace holds demangled signatures: 'void (anonymous namespace)::rk4_bwd_kernel<7, 1, false>(float const*, ...)',
    'void dopri5_bwd_kernel<6>(Dopri5BwdArgs)'."""
    pat = re.compile(r"(?:^|[\s:])%s\(" % re.escape(name))
    grids = [g for n, g in kernels if pat.search(n)]
    assert grids, "%s did not launch; launched: %s" % (name, sorted({n[:80] for n, _ in kernels}))
    return grids


@contextlib.contextmanager
def tensor_cores(on):
    """options fwd_mma / bwd_mma for the block (the FFMA2 R = 2 kernels at D = 4, 5), restored afterwards"""
    from gaussian_process_odes_b200 import _lib
    saved = {k: _lib.get_option(k) for k in ("fwd_mma", "bwd_mma")}
    try:
        for k in saved:
            _lib.set_option(k, int(on))
        yield
    finally:
        for k, v in saved.items():
            _lib.set_option(k, v)


# ---- problems ---------------------------------------------------------------------------------------------------------
def _shape(D):
    """odd M and S: S / 2 feature pairs rounded up leave a partial group of 32 records at every D"""
    return 2 * D + 31, 16 * D + 61


def _setup(D, B, seed, nu):
    """nu = '0.3': 0.3 N(0,1); 'whitened': the cache's own whitened weights, inducing points at a tenth of the usual
    spread (ill-conditioned K(Z,Z): |var nu| ~ 30..120)"""
    M, S = _shape(D)
    p, ys, ts, draws, _ = O.make_problem(D=D, M=M, S=S, N=1, T=4, seed=seed)
    if nu == "whitened":
        p['inducing_loc'] = p['inducing_loc'] * 0.1
    gp, c = oracle_cache(p, draws, torch.float32)
    if nu != "whitened":
        c['nu'] = torch.tensor(np.random.default_rng(seed + 1).normal(size=(D, M, 1)) * float(nu), dtype=torch.float32)
    x = torch.tensor(np.random.default_rng(seed + 2).normal(size=(B, D)) * 1.5, dtype=torch.float32)
    return gp, c, x


# ---- vector field and RK4, forward and adjoint, above the warp-per-row batches ---------------------------------------
CELLS = [(D, m) for D in range(1, 9) for m in ("thread", "wide") if m == "thread" or rows_per_thread(D) > 1]


@pytest.mark.gpu
@pytest.mark.parametrize("nu", ["0.3", "whitened"])
@pytest.mark.parametrize("D,mapping", CELLS)
@pytest.mark.parametrize("entry", ["vf", "rk4"])
def test_row_per_thread_kernels_match_chunked_oracle(entry, D, mapping, nu):
    """vf_fwd_kernel / vf_bwd_kernel / rk4_fwd_kernel / rk4_bwd_kernel <D, R> for R = 1 and the wide R; at D = 4, 5 the
    wide ones are reached with the tensor-core kernels switched off."""
    from gaussian_process_odes_b200 import ops
    sms = _sms()
    B, R = mapping_batch(D, mapping, sms)
    use_tc = selected_mapping(D, B, sms) == R   # else the tensor-core kernels would take this batch (D = 4, 5)
    assert selected_mapping(D, B, sms, use_tc) == R and B % 32 and B % (THREADS * R)
    seed = 10 * D + (mapping == "wide") + 2 * (nu == "whitened") + 4 * (entry == "rk4")
    gp, c, x = _setup(D, B, seed, nu)
    if entry == "vf":
        fn, ofn, tol = (lambda xc, a: ops.vector_field(xc, *a)), oracle_vf, TOL_VF
        cot = torch.tensor(np.random.default_rng(seed).normal(size=(B, D)), dtype=torch.float32)
        fwd, bwd = "vf_fwd_kernel<%d, %d>" % (D, R), "vf_bwd_kernel<%d, %d>" % (D, R)
    else:
        ts = time_grid(3, 0.07, seed)
        fn, ofn, tol = (lambda xc, a: ops.rk4_integrate(xc, ts.cuda(), *a)), oracle_rk4(ts), TOL_TRAJ
        cot = torch.tensor(np.random.default_rng(seed).normal(size=(3, B, D)), dtype=torch.float32)
        fwd, bwd = "rk4_fwd_kernel<%d, %d, false>" % (D, R), "rk4_bwd_kernel<%d, %d, false>" % (D, R)
    with tensor_cores(use_tc):
        (out, got), kernels = profiled(lambda: cuda_grads(fn, gp, c, x, cot))
    grids_of(kernels, fwd)
    grids_of(kernels, bwd)
    row_dim = 0 if entry == "vf" else 1
    out32, ref32 = chunked_oracle(ofn, gp, c, x, cot, torch.float32, row_dim, chunk=CHUNK)
    ref64 = lazy(lambda: chunked_oracle(ofn, gp, c, x, cot, torch.float64, row_dim, chunk=CHUNK))
    name = "%s D=%d R=%d B=%d nu=%s" % (entry, D, R, B, nu)
    assert_parity(name, out.cpu(), out32, lambda: ref64()[0], tol)
    assert_grads(name, got, ref32, lambda: ref64()[1], TOL_GRAD)


# ---- dopri5 -------------------------------------------------------------------------------------------------------------
DP_BATCH = {"one_cta": 13, "warp": 777, "thread": 1101}


def _dopri5(ts, stats, rtol=1e-6):
    """(x0, cache args) -> xs of ops.dopri5_integrate; its stats are appended to ``stats``"""
    from gaussian_process_odes_b200 import ops

    def run(xc, a):
        xs, st = ops.dopri5_integrate(xc, ts.cuda(), *a, rtol=rtol, atol=rtol)
        stats.append(st)
        return xs
    return run


def _dopri5_case(D, B, seed, ts, rtol=1e-6):
    """the CUDA solve + its gradients once under the profiler, the oracle's solve in float32 (float64 lazily)"""
    gp, c, x = _setup(D, B, seed, "0.3")
    cot = torch.tensor(np.random.default_rng(seed).normal(size=(len(ts), B, D)), dtype=torch.float32)
    stats = []
    (xs, got), kernels = profiled(lambda: cuda_grads(_dopri5(ts, stats, rtol), gp, c, x, cot))
    out32, ref32, st = oracle_dopri5(gp, c, x, ts, cot, torch.float32, rtol=rtol, atol=rtol)
    ref64 = lazy(lambda: oracle_dopri5(gp, c, x, ts, cot, torch.float64, rtol=rtol, atol=rtol))
    nfe, acc, rej, status = [int(v) for v in stats[-1].cpu()]
    assert status == 0 and nfe == 2 + 6 * (acc + rej), (nfe, acc, rej, status)
    assert abs(acc - st['accepted']) <= 1 and abs(rej - st['rejected']) <= 1, (acc, rej, st)
    name = "dopri5 D=%d B=%d" % (D, B)
    assert torch.equal(xs[0].cpu(), x)
    assert_parity(name, xs.cpu(), out32, lambda: ref64()[0], TOL_TRAJ)
    # both are exact gradients of a discrete solve; they may differ by one accept / reject decision
    assert_grads(name, got, ref32, lambda: ref64()[1], 2e-4)
    return kernels, acc


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", ["one_cta", "warp", "thread"])
@pytest.mark.parametrize("D", range(1, 9))
def test_dopri5_forward_mappings_and_adjoint(D, mapping):
    """every D on each forward mapping; the grid decreases on every other (D, mapping), so each D and each mapping sees
    both directions"""
    B = DP_BATCH[mapping]
    decreasing = (D + list(DP_BATCH).index(mapping)) % 2 == 1
    ts = torch.tensor([0.0, 0.3, 0.35, 0.9], dtype=torch.float32) * (-1.0 if decreasing else 1.0)
    kernels, _ = _dopri5_case(D, B, 7 * D + len(mapping), ts)
    grids_of(kernels, dopri5_kernel(D, B))
    grids_of(kernels, "dopri5_bwd_kernel<%d>" % D)


@pytest.mark.gpu
def test_dopri5_adjoint_grid_stride():
    """B > 8 x the largest adjoint grid: every warp of dopri5_bwd_kernel carries two rows or more, in order; the forward
    runs one row per thread"""
    D = 5
    B = dopri5_two_pass_batch(_sms())
    ts = torch.tensor([0.0, 0.2, 0.45], dtype=torch.float32)
    kernels, _ = _dopri5_case(D, B, 55, ts)
    grids_of(kernels, dopri5_kernel(D, B))
    grid = grids_of(kernels, "dopri5_bwd_kernel<%d>" % D)[0]
    assert B >= 2 * DP_BWD_WARPS * grid, (B, grid)


@pytest.mark.gpu
def test_dopri5_checkpoint_capacity_retry():
    """more accepted steps than the first checkpoint capacity max(32, 4 Tg): the forward reports status 3 and
    _Dopri5.forward solves again with twice the capacity; the gradients come from the second solve"""
    from gaussian_process_odes_b200 import _lib
    D, B = 3, 40
    ts = torch.tensor([0.0, 0.4, 20.0], dtype=torch.float32)
    calls = _lib.LAUNCH_COUNT.get("gpode_dopri5_fwd", 0)
    kernels, acc = _dopri5_case(D, B, 31, ts)
    assert acc > max(32, 4 * len(ts)), acc
    assert _lib.LAUNCH_COUNT["gpode_dopri5_fwd"] - calls == 2, "the capacity retry did not run"
    assert len(grids_of(kernels, dopri5_kernel(D, B))) == 2


@pytest.mark.gpu
def test_dopri5_device_count_path_at_row_per_thread_batch():
    """gpode_dopri5_bwd_dev + gpode_param_grad_dev (the accepted-step count read on the device, as under CUDA-graph
    capture) against the host-count path, with the forward one row per thread"""
    from gaussian_process_odes_b200 import ops
    D, B = 6, DP_BATCH["thread"]
    gp, c, x = _setup(D, B, 66, "0.3")
    ts = torch.tensor([0.0, 0.25, 0.6], dtype=torch.float32)
    cot = torch.tensor(np.random.default_rng(66).normal(size=(3, B, D)), dtype=torch.float32)
    fn = _dopri5(ts, [])
    xs_h, g_h = cuda_grads(fn, gp, c, x, cot)
    saved, n_stats = ops.DEVICE_COUNT_MODE, len(ops.DEVICE_COUNT_STATS)
    ops.DEVICE_COUNT_MODE = True
    try:
        (xs_d, g_d), kernels = profiled(lambda: cuda_grads(fn, gp, c, x, cot))
        assert len(ops.DEVICE_COUNT_STATS) == n_stats + 1, "the device-count path did not run"
        st = [int(v) for v in ops.DEVICE_COUNT_STATS[-1].cpu()]
    finally:
        ops.DEVICE_COUNT_MODE = saved
        del ops.DEVICE_COUNT_STATS[n_stats:]
    grids_of(kernels, dopri5_kernel(D, B))
    grids_of(kernels, "dopri5_bwd_kernel<%d>" % D)
    assert st[3] == 0 and st[1] > 0, st
    # same forward kernel and adjoint grid: trajectory and x-gradient are bitwise equal; the parameter gradients sum the
    # virtual rows over the capacity instead of the count (other float32 partial-sum groups)
    assert torch.equal(xs_d, xs_h) and torch.equal(g_d['x'], g_h['x'])
    for k in ("Z", "ell", "var", "nu"):
        assert relerr(g_d[k], g_h[k]) <= TOL_GRAD, k


# ---- the rules and the oracle helpers themselves (no device) -----------------------------------------------------------
@pytest.mark.parametrize("sms", [148, 132, 40])
def test_batches_sit_just_above_their_thresholds_and_are_ragged(sms):
    if sms == 148:  # the B200's thresholds
        assert (wide_min_rows(2, sms), wide_min_rows(3, sms), mma_min_rows(4, sms)) == (151552, 75776, 56832)
        assert dopri5_two_pass_batch(sms) == 18944 + 77
    for D, mapping in CELLS:
        B, R = mapping_batch(D, mapping, sms)
        assert B % 32 and B % (THREADS * R), (D, mapping, B)
        lower = WARP_MAX_ROWS if mapping == "thread" else wide_min_rows(D, sms) - 1
        assert B - lower < 1024 and selected_mapping(D, B, sms, tensor_cores=False) == R
        assert selected_mapping(D, lower, sms, tensor_cores=False) != R
        if D in (4, 5) and sms == 148:  # the thread batch stays below the tensor-core kernels, the wide one not
            assert selected_mapping(D, B, sms) == (1 if mapping == "thread" else "mma")
    assert [dopri5_kernel(7, B) for B in (DP_ONE_CTA_ROWS, DP_ONE_CTA_ROWS + 1, DP_WARP_MAX_ROWS,
                                          DP_WARP_MAX_ROWS + 1)] == \
        ["dopri5_kernel<7, true, true>", "dopri5_kernel<7, true, false>", "dopri5_kernel<7, true, false>",
         "dopri5_kernel<7, false, false>"]
    assert [dopri5_kernel(1, B) for B in DP_BATCH.values()] == \
        ["dopri5_kernel<1, true, true>", "dopri5_kernel<1, true, false>", "dopri5_kernel<1, false, false>"]
    for B in DP_BATCH.values():
        assert B % DP_BWD_WARPS and B % THREADS


def test_kernel_name_match_is_exact():
    ks = [("void (anonymous namespace)::rk4_bwd_kernel<7, 1, false>(float const*, int)", 148),
          ("void (anonymous namespace)::vf_fwd_kernel<4, 2>(float const*, int)", 3),
          ("void dopri5_bwd_kernel<6>(Dopri5BwdArgs)", 40), ("dopri5_bwd_kernel<6>(Dopri5BwdArgs)", 41)]
    assert grids_of(ks, "rk4_bwd_kernel<7, 1, false>") == [148] and grids_of(ks, "vf_fwd_kernel<4, 2>") == [3]
    assert grids_of(ks, "dopri5_bwd_kernel<6>") == [40, 41]
    for wrong in ("rk4_bwd_kernel<7, 1, true>", "rk4_bwd_kernel<1, 1, false>", "vf_fwd_kernel<4, 1>",
                  "fwd_kernel<4, 2>", "dopri5_bwd_kernel<1>", "bwd_kernel<6>"):
        with pytest.raises(AssertionError):
            grids_of(ks, wrong)


@pytest.mark.parametrize("entry", ["vf", "rk4"])
@pytest.mark.parametrize("nu", ["0.3", "whitened"])
def test_chunked_oracle_equals_one_pass(entry, nu):
    """on the CPU at a tiny size: row chunks of 3 give the outputs and gradients of one autograd pass over all rows"""
    D, B = 3, 8
    gp, c, x = _setup(D, B, 4, nu)
    if entry == "vf":
        fn, cot, row_dim = oracle_vf, torch.randn(B, D, dtype=torch.float64), 0
    else:
        fn, cot, row_dim = oracle_rk4(time_grid(3, 0.1, 1)), torch.randn(3, B, D, dtype=torch.float64), 1
    out_c, g_c = chunked_oracle(fn, gp, c, x, cot, torch.float64, row_dim, dev="cpu", chunk=3)
    out_1, g_1 = chunked_oracle(fn, gp, c, x, cot, torch.float64, row_dim, dev="cpu", chunk=B)
    assert relerr(out_c, out_1) <= 1e-14
    for k in g_1:
        assert relerr(g_c[k], g_1[k]) <= 1e-12, k
    if nu == "whitened":
        assert float((c['nu'].squeeze(2) * gp['var'][:, None]).abs().max()) > 30


def test_dopri5_oracle_runs_on_cpu():
    D, B = 2, 5
    gp, c, x = _setup(D, B, 3, "0.3")
    ts = torch.tensor([0.0, -0.3, -0.5])
    cot = torch.ones(3, B, D)
    out, g, st = oracle_dopri5(gp, c, x, ts, cot, torch.float64, dev="cpu")
    assert out.shape == (3, B, D) and torch.equal(out[0], x.double()) and st['accepted'] >= 1
    assert set(g) == {"x", "Z", "ell", "var", "nu"} and all(torch.isfinite(v).all() for v in g.values())
