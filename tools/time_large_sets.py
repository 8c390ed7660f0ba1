"""Timing of batched Monte-Carlo prediction at 8 < D <= 64: n = 128 function draws, M = 100 inducing points, S = 256
Fourier features, D = 16 / 32 / 64, N = 1 and N = 128 initial states per draw.

For each shape and solver (rk4 on a 51-point grid, dopri5 at rtol = atol = 1e-6 on the same grid):
  * ``compute_test_predictions`` batched (one whitening, one pack, one integrator launch sequence for all draws)
    against ``batched=False`` (one full single-draw solve per draw), end to end, host clock around a device
    synchronise;
  * one ``gpode_vf_fwd_large_sets`` evaluation against n single-draw evaluations (``LargeField.__call__``) at the same
    states, CUDA events, operand blocks packed beforehand.
The card's name and power limit are read in the same run. At N < 128 every tile streams its draw's whole operand
block (9.6 MB per draw at D = 64: 1.2 GB per evaluation, more than the L2 holds).

    python tools/time_large_sets.py [--reps 3] [--out profiles/r04_large_sets.json]
"""
import argparse, json, os, subprocess, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]
from gaussian_process_odes_b200 import builders, ops, _lib


def gpu_info():
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                            text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:
        pl = "unknown"
    return dict(gpu=torch.cuda.get_device_name(), power_limit=pl)


def wall(fn, reps):
    fn()   # warm-up: module loads, graph reaper, allocator
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), [round(v, 2) for v in ts]


def events(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), [round(v, 3) for v in ts]


def predictions(D, N, solver, n, reps):
    np.random.seed(1)
    torch.manual_seed(1)
    model = builders.build_gpode(N=N, T=51, D=D, num_inducing=100, num_features=256, solver=solver,
                                 ts_dense_scale=2).cuda()   # scale 2: the solver grid is the 51-point grid itself
    ts = torch.linspace(0.0, 1.0, 51).cuda()
    x0 = torch.randn(N, D, device="cuda")
    out = {}
    for batched in (True, False):
        fn = lambda: builders.compute_test_predictions(model, x0, ts, eval_sample_size=n, batched=batched)
        out["batched_ms" if batched else "loop_ms"] = wall(fn, reps)
    np.random.seed(2)
    a = builders.compute_test_predictions(model, x0, ts, eval_sample_size=n, batched=True)
    np.random.seed(2)
    b = builders.compute_test_predictions(model, x0, ts, eval_sample_size=n, batched=False)
    out["relerr_batched_vs_loop"] = float((a - b).abs().max() / b.abs().max())
    if solver == "dopri5":
        st = model.flow.last_sets_stats.cpu()
        out["accepted_steps_min_max"] = [int(st[:, 1].min()), int(st[:, 1].max())]
    out["speedup"] = out["loop_ms"][0] / out["batched_ms"][0]
    return out


def vector_field(D, N, n, reps, M=100, S=256):
    g = torch.Generator().manual_seed(D)
    r = lambda *s: torch.randn(*s, generator=g)
    ell = torch.rand(D, D, generator=g) + 0.7
    Z, var = r(M, D).cuda(), (torch.rand(D, generator=g) + 0.5).cuda()
    omega = (r(n, D, S, D) / ell.T.unsqueeze(1)).cuda()
    phase, w, nu = (torch.rand(n, S, D, generator=g) * 6.283).cuda(), r(n, S, D).cuda(), (0.3 * r(n, D, M)).cuda()
    ell = ell.cuda()
    x = r(n, N, D).cuda()
    with torch.no_grad():
        pcs = ops.PackedCacheSets(Z, ell, var, nu, omega, phase, w)
        f, tmp = torch.empty_like(x), torch.empty_like(x)
        sets = lambda: _lib.call("gpode_vf_fwd_large_sets", _lib.ptr(pcs.packed), ops.ctypes.byref(pcs.struct), n, N,
                                 _lib.ptr(x), _lib.ptr(tmp), _lib.ptr(f), _lib.stream_ptr())
        fields = [ops.LargeField(Z, ell, var, nu[q], omega[q], phase[q], w[q]) for q in range(n)]
        xq = [x[q] for q in range(n)]
        loop = lambda: [fields[q](xq[q]) for q in range(n)]
        t_sets, t_loop = events(sets, reps), events(loop, reps)
        same = all(torch.equal(f[q], fields[q](xq[q])) for q in range(n))
    del fields, pcs
    torch.cuda.empty_cache()
    bytes_packed = _lib.load().gpode_packed_large_floats(D, M, S) * 4 * n
    return dict(sets_ms=t_sets, loop_ms=t_loop, speedup=t_loop[0] / t_sets[0], bitwise_equal=same,
                packed_bytes=bytes_packed, hbm_bound_ms_at_7_7_TBps=bytes_packed / 7.7e12 * 1e3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--n", type=int, default=128)
    ap.add_argument("--dims", default="16,32,64")
    ap.add_argument("--rows", default="1,128")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_large_sets.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_large_sets.py measures on the GPU; no CUDA device found")
    res = dict(gpu_info(), n_draws=a.n, M=100, S=256, grid_points=51, rtol=1e-6, atol=1e-6, shapes=[])
    for D in [int(v) for v in a.dims.split(",")]:
        for N in [int(v) for v in a.rows.split(",")]:
            row = dict(D=D, N=N, vf=vector_field(D, N, a.n, max(a.reps, 5)))
            for solver in ("rk4", "dopri5"):
                row[solver] = predictions(D, N, solver, a.n, a.reps)
            print(json.dumps(row), flush=True)
            res["shapes"].append(row)
    res["batched_not_faster"] = [dict(D=r["D"], N=r["N"], what=k) for r in res["shapes"] for k in ("vf", "rk4", "dopri5")
                                 if r[k]["speedup"] <= 1.0]
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
