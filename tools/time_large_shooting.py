"""The multiple-shooting training step above eight state dimensions: the large-D shooting step (gpode_shoot_fwd_large /
gpode_shoot_bwd_large, fuse_elbo = True) against the unfused chain (fuse_elbo = False: the large-D RK4 writes the
trajectory, torch ops decode it and evaluate the Gaussian log-density, gpode_constraint_sum runs as its own pass).
One step = UniformSequenceModel.build_lowerbound_terms + inducing KL, forward and backward, eager, on one model whose
fuse_elbo flag is toggled, so both arms train the same parameters.

Shapes: D = 16 / 32 / 64, M = 100, S = 256, S_mc = 5, N = 16, T = 1250 (1e5 segments), D_obs = 50 (a linear decoder
with bias) and D_obs = D (the plain Gaussian likelihood, W = I). After two warm-up steps per arm the arms run
alternately, `--rounds` times each, `--steps` steps per timed window (host clock around a device synchronise). Each arm's
torch.cuda.max_memory_allocated is taken over its own windows. Before timing, both arms evaluate one step from the same
seeds and their losses are compared.

    python tools/time_large_shooting.py [--rounds 5] [--steps 3] [--out profiles/r06_large_shooting.json]
"""
import argparse, json, os, subprocess, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
import gpode_oracle as O
from util import build_product_model


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[0].split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock, torch_device=torch.cuda.get_device_name())


def problem(D, Dobs, N, T, S_mc, M, S, seed):
    p, ys, ts, _, _ = O.make_problem(D=D, M=M, S=S, N=N, T=T, S_mc=S_mc, seed=seed, dt=0.01,
                                     D_obs=None if Dobs == D else Dobs)
    if Dobs == D:
        return build_product_model("shooting", p, ys, S, "rk4"), ys.cuda(), ts.cuda()
    from gaussian_process_odes_b200.misc.mocap_utils import LinearProjection
    rng = np.random.default_rng(seed + 1)
    comp = rng.normal(size=(D, Dobs)) / np.sqrt(D)
    model = build_product_model("shooting", p, ys, S, "rk4", proj=torch.tensor(comp, dtype=torch.float32))
    model.likelihood.projection = LinearProjection(comp, 1.0 + 0.2 * rng.uniform(-1, 1, size=D), 0.3 * rng.normal(size=D))
    return model, ys.cuda(), ts.cuda()


def step(model, ys, ts, S_mc):
    model.zero_grad(set_to_none=True)
    ll, c, e, k0 = model.build_lowerbound_terms(ys, ts, num_samples=S_mc)
    loss = -(ll + c + e - k0 - model.build_inducing_kl())
    loss.backward()
    return loss.detach()


def seeded_loss(model, ys, ts, S_mc, fuse, seed=11):
    model.fuse_elbo = fuse
    np.random.seed(seed)
    torch.manual_seed(seed)
    return float(step(model, ys, ts, S_mc))


def run(D, Dobs, rounds, steps, N=16, T=1250, S_mc=5, M=100, S=256):
    model, ys, ts = problem(D, Dobs, N, T, S_mc, M, S, seed=3 + D)
    out = dict(D=D, D_obs=Dobs, decoder="linear+bias" if Dobs != D else "identity", M=M, S=S, S_mc=S_mc, N=N, T=T,
               segments=S_mc * N * T, steps_per_window=steps)
    l1, l0 = seeded_loss(model, ys, ts, S_mc, True), seeded_loss(model, ys, ts, S_mc, False)
    out.update(loss_fused=l1, loss_unfused=l0, loss_relerr=abs(l1 - l0) / abs(l0))
    arms = {"fused": True, "unfused": False}
    for fuse in arms.values():
        model.fuse_elbo = fuse
        for _ in range(2):
            step(model, ys, ts, S_mc)
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    peak = {k: 0 for k in arms}
    for _ in range(rounds):
        for name, fuse in arms.items():
            model.fuse_elbo = fuse
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            t0 = time.perf_counter()
            for _ in range(steps):
                step(model, ys, ts, S_mc)
            torch.cuda.synchronize()
            times[name].append((time.perf_counter() - t0) * 1e3 / steps)
            peak[name] = max(peak[name], torch.cuda.max_memory_allocated())
    for name in arms:
        v = np.array(times[name])
        out[name + "_ms"] = float(np.median(v))
        out[name + "_ms_runs"] = [round(float(x), 3) for x in v]
        out[name + "_spread_ms"] = float(v.max() - v.min())
        out[name + "_peak_mib"] = round(peak[name] / 2 ** 20, 1)
    out["speedup_unfused_over_fused"] = out["unfused_ms"] / out["fused_ms"]
    # decision rule: the fused step is slower only when its fastest window is slower than the unfused arm's slowest
    out["fused_slower_beyond_spread"] = bool(min(times["fused"]) > max(times["unfused"]))
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--dims", default="16,32,64")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    info = gpu_info()
    print(json.dumps(info), flush=True)
    res = []
    for D in [int(s) for s in a.dims.split(",")]:
        for Dobs in (50, D):
            r = run(D, Dobs, a.rounds, a.steps)
            print(json.dumps({k: v for k, v in r.items() if not k.endswith("_runs")}), flush=True)
            res.append(r)
            torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(dict(info, results=res), open(a.out, "w"), indent=1)
