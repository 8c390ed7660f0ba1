"""Timing of differentiable dopri5 at 8 < D <= 64 on the config-5 problem of SURVEY.md section 8d (M = 100, S = 256,
nu supplied directly, grid [0, 0.32], rtol = atol = 1e-6): the no-grad forward (gpode_dopri5_fwd_large), the
checkpointing forward (gpode_dopri5_fwd_large_ckpt, including its one host read of the stats), the backward
(gpode_dopri5_bwd_large + finalize), and one gpode_vf_bwd_large at the same shape. The backward runs 6 n_acc + 1 VJPs;
`bwd_over_vjps` is its time over that many single-VJP times (element-wise kernels and launches are the rest).
CUDA events, warm-up, median of the runs.

    python tools/time_large_dopri5.py [--reps 5] [--out profiles/r03_large_dopri5.json]
"""
import argparse, json, os, subprocess, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]
import gpode_oracle as O
from gaussian_process_odes_b200 import ops, _lib
from gaussian_process_odes_b200._lib import ptr, stream_ptr


def ev_time(fn, reps, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), [round(v, 3) for v in ts]


def gpu_info():
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                            text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:
        pl = "unknown"
    return dict(gpu=torch.cuda.get_device_name(), power_limit=pl)


def run(D, B, reps, M=100, S=256):
    p, ys, ts, draws, _ = O.make_problem(D=D, M=M, S=S, N=1, T=4, seed=5)
    gp = O.gp_params(p)
    omega = draws['eps_omega'] / gp['ell'].T.unsqueeze(1)
    nu = torch.tensor(np.random.default_rng(1).normal(size=(D, M)) * 0.1, dtype=torch.float32)
    const = [a.detach().cuda().contiguous() for a in (gp['Z'], gp['ell'], gp['var'], nu, omega,
                                                      draws['phase_u'] * 2 * np.pi, draws['w'])]
    args = [a.clone().requires_grad_(i < 4) for i, a in enumerate(const)]
    g = torch.Generator(device="cuda").manual_seed(D * 7 + B)
    x = torch.randn(B, D, device="cuda", generator=g)
    xg = x.clone().requires_grad_(True)
    t = torch.tensor([0.0, 0.32], dtype=torch.float32, device="cuda")
    cot = torch.randn(2, B, D, device="cuda", generator=g)
    out = dict(D=D, M=M, S=S, B=B, grid=[0.0, 0.32], rtol=1e-6, atol=1e-6)
    with torch.no_grad():
        out["fwd_nograd_ms"], out["fwd_nograd_runs"] = ev_time(lambda: ops.dopri5_integrate(x, t, *const), reps)
    out["fwd_ckpt_ms"], out["fwd_ckpt_runs"] = ev_time(lambda: ops.dopri5_integrate(xg, t, *args), reps)
    xs, stats = ops.dopri5_integrate(xg, t, *args)
    nfe, acc, rej, status = [int(v) for v in stats.cpu()]
    assert status == 0
    out.update(nfe=nfe, accepted=acc, rejected=rej)
    out["bwd_ms"], out["bwd_runs"] = ev_time(lambda: xs.backward(cot, retain_graph=True), reps)
    # one VJP at the same shape
    field = ops.LargeField(*const)
    pk, f, acc_buf, gx = field.packed_bwd, field(x), field.new_acc(), torch.empty_like(x)
    out["vjp_ms"], out["vjp_runs"] = ev_time(
        lambda: _lib.call("gpode_vf_bwd_large", ptr(pk), D, M, S, ptr(x), ptr(f), ptr(cot[1]), ptr(gx), ptr(acc_buf), B,
                          stream_ptr()), reps)
    out["n_vjp"] = 6 * acc + 1
    out["bwd_over_vjps"] = out["bwd_ms"] / (out["n_vjp"] * out["vjp_ms"])
    out["ckpt_bytes"] = 8 * B * D * 4 * max(32, 4 * 2)
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    info = gpu_info()
    print(json.dumps(info), flush=True)
    res = []
    for B in (10000, 100000):
        for D in (16, 32, 64):
            r = run(D, B, a.reps)
            print(json.dumps({k: v for k, v in r.items() if not k.endswith("_runs")}), flush=True)
            res.append(r)
            torch.cuda.empty_cache()
    if a.out:
        json.dump(dict(info, results=res), open(a.out, "w"), indent=1)
