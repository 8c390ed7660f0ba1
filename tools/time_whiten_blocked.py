"""Whitening forward + backward above M = 160 at D <= 8: the blocked float64 kernels (ops.whiten ->
gpode_whiten_{fwd,bwd}_blocked) against the float64 torch.linalg formulation (ops._whiten_large: batched cuSOLVER
Cholesky, cuBLAS triangular solves, autograd backward) on the same inputs, the two arms alternated in one process.
Then the whitening's share of one training step at M = 1024 (multiple-shooting model, rk4), per-call CUDA-event times
of every C-ABI call in the step (the whitened KL included).

    python tools/time_whiten_blocked.py [--reps 10] [--out profiles/r05_whiten_blocked.json]

Inputs of a few hundred MB at D = 8, M = 2048 stay partly L2-resident (126 MB) between passes, as they do in training,
where the same Kzz is factored and solved within one step."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def inputs(D, M, S, seed):
    import itertools
    import math
    rng = np.random.default_rng(seed)
    t = lambda a: torch.tensor(np.asarray(a), dtype=torch.float32, device="cuda")
    side = math.ceil(M ** (1.0 / D) - 1e-9)
    Z = np.array(list(itertools.islice(itertools.product(range(side), repeat=D), M)), dtype=np.float64)
    Z = t(Z + 0.05 * rng.uniform(-1, 1, size=Z.shape))
    ell = t(0.7 * (1 + 0.05 * rng.uniform(-1, 1, size=(D, D))))
    var = t(0.5 + rng.uniform(size=D))
    u = t(rng.normal(size=(M, D)))
    omega = t(rng.normal(size=(D, S, D)) / (float(Z.abs().max()) + 1.0))
    phase = t(rng.uniform(size=(S, D)) * 2 * np.pi)
    w = t(rng.normal(size=(S, D)))
    cot = t(rng.normal(size=(D, M)))
    return (Z, ell, var, u, omega, phase, w), cot


def arm_blocked(args, cot):
    from gaussian_process_odes_b200 import ops
    leaves = [a.clone().requires_grad_(True) for a in args[:4]]
    nu = ops.whiten(*leaves, *args[4:], 1e-5)
    nu.backward(cot)
    return [nu.detach()] + [x.grad for x in leaves]


def arm_linalg(args, cot):
    """omega = eps / ell inside autograd: the blocked kernels fold that path into grad_ell"""
    from gaussian_process_odes_b200 import ops
    leaves = [a.clone().requires_grad_(True) for a in args[:4]]
    eps = args[4] * args[1].t().unsqueeze(1)
    nu = ops._whiten_large(*leaves, eps / leaves[1].t().unsqueeze(1), *args[5:], 1e-5)
    nu.backward(cot)
    return [nu.detach()] + [x.grad for x in leaves]


def time_arm(fn, args, cot, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn(args, cot)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def step_share(D, M, reps):
    """Per-call times of one multiple-shooting training step at (D, M): which share is the whitening."""
    import gpode_oracle as O
    from gaussian_process_odes_b200 import _lib, builders
    from util import build_product_model
    import itertools
    import math
    p, ys, ts, _, _ = O.make_problem(D=D, M=M, S=256, N=4, T=50, seed=1)
    side = math.ceil(M ** (1.0 / D) - 1e-9)
    Zl = np.array(list(itertools.islice(itertools.product(range(side), repeat=D), M)), dtype=np.float64)
    p['inducing_loc'] = torch.tensor(2.0 * (Zl - (side - 1) / 2), dtype=torch.float32)
    model = build_product_model("shooting", p, ys, 256, "rk4")
    ys_c, ts_c = ys.cuda(), ts.cuda()

    def step():
        model.zero_grad(set_to_none=True)
        loss = builders.compute_loss_shooting(model, ys_c, ts_c, num_samples=5)[0]
        loss.backward()

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        step()
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / reps
    _lib.profile_start()
    for _ in range(reps):
        step()
    calls = {k: v / reps for k, (n, v) in _lib.profile_stop().items()}
    whiten = sum(v for k, v in calls.items() if k.startswith("gpode_whiten"))
    return dict(D=D, M=M, N=4, T=50, S=256, S_mc=5, step_ms=step_ms,
                calls_ms={k: round(v, 4) for k, v in sorted(calls.items(), key=lambda kv: -kv[1])},
                whiten_ms=whiten, whiten_share_of_step=whiten / step_ms)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_whiten_blocked.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_whiten_blocked.py measures on a CUDA device; none found")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    rows = []
    for D in (2, 5, 8):
        for M in (256, 512, 1024, 2048):
            args, cot = inputs(D, M, 256, seed=D + M)
            b, r = arm_blocked(args, cot), arm_linalg(args, cot)   # warm-up, and the outputs compared
            dev = [float((x - y).abs().max() / y.abs().max()) for x, y in zip(b, r)]
            tb, tl = [], []
            for _ in range(3):   # alternate the arms
                tb.append(time_arm(arm_blocked, args, cot, a.reps))
                tl.append(time_arm(arm_linalg, args, cot, a.reps))
            row = dict(D=D, M=M, S=256, blocked_ms=min(tb), linalg_ms=min(tl), blocked_ms_all=tb, linalg_ms_all=tl,
                       speedup=min(tl) / min(tb), max_rel_dev_nu_gZ_gell_gvar_gu=dev)
            print(json.dumps(row), flush=True)
            rows.append(row)
            del args, cot
            torch.cuda.empty_cache()
    shares = [step_share(D, 1024, a.reps) for D in (2, 5, 8)]
    for s in shares:
        print(json.dumps(s), flush=True)
    out = dict(gpu=smi, what="whitening forward + backward (ms per call pair, best of 3 alternated windows of "
               "%d calls); training-step share at M = 1024" % a.reps, rows=rows, step_share=shares)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
