#!/usr/bin/env python
"""bench.py -- GP vector-field evals/s of the multiple-shooting ELBO forward+backward step (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scaling weak|strong]
                    [--rows-scale F] [--no-parity-check] [--no-cpu-baseline] [--dump-outputs DIR]

Workload (``config.workload``): BASELINE.json configs[3], "MoCap GPODE shooting variant on long synthetic
MoCap-shaped trajectories": latent D=5 -> D_obs=50 through a fixed orthonormal decoder, M=100 inducing points, S=256
Fourier features, S_mc=5 Monte-Carlo samples, N=16 sequences of T=12500 points per GPU -> 1,000,000 one-interval
shooting segments per GPU, one RK4 (3/8 rule) step of h=0.01 each. It is the largest single-GPU configuration, and
the one that shards (sequences across GPUs, weak scaling: N grows with the GPU count).

One "step" = one ELBO forward + backward (``build_lowerbound_terms`` + ``build_inducing_kl`` + ``loss.backward()``,
plus the shared-gradient all-reduce when N > 1) through the reference-facing API: GP cache build (whitening kernel),
fused RK4 forward kernel over all segments, the ELBO side terms, the discrete-adjoint kernel, the per-inducing-point
gradient kernel, whitening backward. The optimiser step is not part of the metric (BASELINE.md section 3).

``--scaling strong`` keeps the TOTAL at 16 sequences = 10^6 segments and splits them over the GPUs (16 / N sequences
each) instead of giving every GPU 16 sequences of its own. Before anything is timed, rank 0 checks the ELBO loss and
every parameter gradient of a 60 000-segment problem of the same shape -- the same kernels -- against the oracle port
(``tests/util.py::elbo_errors``; the oracle is the checker, never the thing measured).

value = segments x 4 vector-field evaluations (the reference's own NFE count for this step) / step time, aggregated
over all GPUs. ``e2e`` repeats the measurement with the observations copied from pinned host memory and the loss
read back to the host inside every timed step.

``--dump-outputs DIR`` writes what the last timed step returned to its caller on rank 0: ``loss.npy`` and one
``grad.<parameter name>.npy`` per parameter gradient. Inputs, initial parameters and the random draws are seeded, so
two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"  # NCCL's version banner goes to stdout and would break the one-JSON-line contract

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOAD = dict(name="mocap_shooting_long", D=5, D_obs=50, M=100, S=256, S_mc=5, N_per_gpu=16, T=12500, dt=0.01,
                solver="rk4")
METRIC = "gp_vector_field_evals_per_sec_elbo_fwd_bwd"
UNIT = "evals/s"


def f_vf(D, S, M):
    """Algorithmic flops of one vector-field evaluation of one row (SURVEY.md section 8d)."""
    return D * (S * (2 * D + 4) + M * (3 * D + 4))


DUMP_LIMIT_BYTES = 64 << 20


def step_outputs(model, loss):
    """What one ELBO step hands its caller, copied to the host: the loss and every parameter's gradient."""
    out = {"loss": loss.detach().cpu().numpy()}
    for name, p in model.named_parameters():
        if p.grad is not None:
            out["grad." + name] = p.grad.detach().cpu().numpy()
    return out


def write_outputs(out_dir, arrays, limit=DUMP_LIMIT_BYTES):
    """One float32 / float64 ``<name>.npy`` per array, at most ``limit`` bytes in all. If the arrays are larger, each
    one above its equal share of the limit is replaced by a fixed, seeded sample of its flattened elements (in index
    order), so that the files of two runs still correspond element for element."""
    os.makedirs(out_dir, exist_ok=True)
    share = limit // max(1, len(arrays)) - 4096   # 4 KB per file for the .npy header
    too_big = sum(a.nbytes + 4096 for a in arrays.values()) > limit
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64 if a.dtype == np.float64 else np.float32)
        if too_big and a.nbytes > share:
            idx = np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------------------------------------------------
# synthetic problem of the workload's shape
# ----------------------------------------------------------------------------------------------------------------------
def synthetic_sequences(N, T, D, D_obs, seed):
    """Smooth latent sequences (re-standardised cumulative sums) and their noisy decoded observations."""
    rng = np.random.default_rng(seed)
    lat = np.cumsum(rng.normal(size=(N, T, D)) * 0.05, axis=1)
    lat = (lat - lat.mean(axis=(0, 1), keepdims=True)) / (lat.std(axis=(0, 1), keepdims=True) + 1e-8)
    q, _ = np.linalg.qr(np.random.default_rng(1234).normal(size=(D_obs, D)))  # same decoder on every rank
    comp = q.T.astype(np.float32)  # (D, D_obs)
    ys = lat @ comp + rng.normal(size=(N, T, D_obs)) * 0.1
    return lat.astype(np.float32), ys.astype(np.float32), comp


def build_ours(w, rank, world, rows_scale, strong=False):
    from gaussian_process_odes_b200 import builders, distributed
    T = max(3, int(round(w["T"] * rows_scale)))
    if strong:
        if w["N_per_gpu"] % world:
            raise SystemExit("--scaling strong needs the GPU count to divide %d sequences" % w["N_per_gpu"])
        N_loc, N_glob = w["N_per_gpu"] // world, w["N_per_gpu"]
    else:
        N_loc, N_glob = w["N_per_gpu"], w["N_per_gpu"] * world
    lat, ys, comp = synthetic_sequences(N_loc, T, w["D"], w["D_obs"], seed=121 + rank)
    from gaussian_process_odes_b200.misc.mocap_utils import LinearProjection
    projection = LinearProjection(comp)
    np.random.seed(121)  # identical GP initialisation on every rank
    model = builders.build_gpode_shooting(N_loc, T, w["D"], num_inducing=w["M"], num_features=w["S"],
                                          solver=w["solver"], D_obs=w["D_obs"], projection=projection)
    model.num_observations = N_glob * T * w["D_obs"]
    gp = model.flow.odefunc.diffeq
    with torch.no_grad():
        gp.inducing_loc.optvar.copy_(torch.tensor(np.random.default_rng(5).normal(size=(w["M"], w["D"])),
                                                  dtype=torch.float32))
        model.state_distribution.x0.param_mean.optvar.copy_(torch.tensor(lat[:, 0]))
        model.state_distribution.param_mean.optvar.copy_(torch.tensor(lat[:, 1:]))
    distributed.broadcast_shared_parameters(model)
    ts = torch.arange(T, dtype=torch.float32) * w["dt"]
    return model, torch.tensor(ys), ts, N_glob, T


# ----------------------------------------------------------------------------------------------------------------------
# clocks during the timed region
# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        # NVML polled from a thread every ~5 ms (the timed region is a fraction of a second); nvidia-smi as fallback
        self.samples, self.halt, self.nv = [], threading.Event(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = (pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv, h = self.nv
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons",
                              getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None))
        while not self.halt.is_set():
            try:
                mask = int(get_reasons(h)) if get_reasons else 0
                self.samples.append((float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)),
                                     float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)),
                                     nv.nvmlDeviceGetPowerUsage(h) / 1000.0,
                                     [n for n, b in bits.items() if mask & b]))
            except Exception:
                pass
            time.sleep(0.005)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nv is not None:
            self.halt.set()
            self.thread.join(timeout=1)
            sm = [x[0] for x in self.samples]
            reasons = sorted({r for x in self.samples for r in x[3]})
            return dict(sm_mhz=float(np.median(sm)) if sm else None,
                        sm_max_mhz=max(x[1] for x in self.samples) if sm else None,
                        power_w_max=max(x[2] for x in self.samples) if sm else None, samples=len(sm),
                        source="nvml", reasons=reasons)
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smmax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smmax.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(smmax) if smmax else None,
                    power_w_max=max(power) if power else None, samples=len(sm), reasons=sorted(reasons))


# ----------------------------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port (reference algorithm restated op-for-op on torch CPU) on a bounded sample
# ----------------------------------------------------------------------------------------------------------------------
def cpu_elbo_timing(w, steps, warmup, T_sample=6000, N_sample=1, prefer_reference=True):
    """One ELBO forward+backward per step on the host cores. With the staged archive (or the checkout) present this is the
    UNMODIFIED reference -- its own DSVGP_Layer / Flow / UniformSequenceModel classes (oracle/reference_harness.py, the
    restated torchdiffeq 0.2.0 underneath, random draws injected so that every step sees the same numbers) --
    `kind: "reference"`; otherwise the oracle port (`kind: "port"`)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gpode_oracle as O
    import reference_harness as H
    torch.set_num_threads(os.cpu_count())
    p, ys, ts, draws, proj = O.make_problem(D=w["D"], M=w["M"], S=w["S"], N=N_sample, T=T_sample, S_mc=w["S_mc"],
                                            D_obs=w["D_obs"], dt=w["dt"], ell0=1.25, seed=121)
    rows = w["S_mc"] * N_sample * T_sample
    use_ref = prefer_reference and H.available()
    times = []
    if use_ref:
        try:
            mods = H._import_reference()
            model = H.build_reference_shooting(mods, p, ys, w["S"], solver=w["solver"], project=proj)
            params = [q for q in model.parameters() if q.requires_grad]
            for i in range(warmup + steps):
                for q in params:
                    q.grad = None
                t0 = time.perf_counter()
                with H.injected_draws(mods, draws, n_caches=1, mvn_order=("eps_x0", "eps_states")):
                    loss, _ = H.reference_shooting_loss(model, ys, ts, num_samples=w["S_mc"])
                loss.backward()
                t1 = time.perf_counter()
                if i >= warmup:
                    times.append(t1 - t0)
            what = "the UNMODIFIED reference modules (%s; restated torchdiffeq 0.2.0 rk4)" % (
                "/root/reference" if H.source() == "tree" else "oracle/_ref archive")
        except Exception as exc:  # the reference arm must never take the bench line down: fall back to the port, say so
            print("reference modules failed on this host (%s: %s); timing the oracle port instead" % (
                type(exc).__name__, exc), file=sys.stderr)
            use_ref, times = False, []
    if not use_ref:
        for i in range(warmup + steps):
            pp = {k: v.detach().clone().requires_grad_(True) for k, v in p.items()}
            t0 = time.perf_counter()
            r = O.elbo_shooting(pp, ys, ts, draws, method=w["solver"], project=proj)
            r["loss"].backward()
            t1 = time.perf_counter()
            if i >= warmup:
                times.append(t1 - t0)
        what = "the oracle port"
    sec = float(np.median(times))
    return dict(value=rows * 4 / sec, unit=UNIT, cores=torch.get_num_threads(), kind="reference" if use_ref else "port",
                sample="%d segments (S_mc=%d x N=%d x T=%d) of the same D=%d,M=%d,S=%d,D_obs=%d workload, median of %d "
                       "ELBO fwd+bwd steps of %s (torch CPU float32, %d threads)" % (
                           rows, w["S_mc"], N_sample, T_sample, w["D"], w["M"], w["S"], w["D_obs"], steps, what,
                           torch.get_num_threads()),
                ms_per_step=sec * 1e3, rows=rows)


# ----------------------------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = WORKLOAD
    cb = cpu_elbo_timing(w, steps=args.steps, warmup=args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": w["name"], "D": w["D"], "D_obs": w["D_obs"], "M": w["M"], "S": w["S"],
                       "S_mc": w["S_mc"], "solver": w["solver"], "segments_per_step": cb["rows"],
                       "note": ("the unmodified reference modules (archive staged by build(), restated torchdiffeq "
                                "underneath) on the host cores, bounded sample of the workload" if cb["kind"] == "reference"
                                else "reference algorithm (oracle port: no staged reference archive found) on the host "
                                     "cores, bounded sample of the workload")},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def pin_to_gpu_numa_node(index):
    """Bind this process to the CPU cores next to its GPU (NVML's ideal affinity) BEFORE any pinned buffer is allocated,
    so the staging memory of the end-to-end copies is first-touched on the GPU's own NUMA node (round 1: all ranks sat on
    cores 0-31 and shared one node's memory controller for 8 x 40 MB per step)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(index))
        return sorted(os.sched_getaffinity(0))
    except Exception:
        return None


def parity_precheck():
    """ELBO loss + every parameter gradient of a 60 000-segment MoCap-shaped shooting problem (whitened nu; the
    tensor-core forward / adjoint kernels and the row-per-thread gradient contraction -- the kernels timed below)
    against the oracle port in float32, arbitrated by float64. Raises on a mismatch."""
    for pth in (os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
        if pth not in sys.path:
            sys.path.insert(0, pth)
    from util import elbo_errors
    kw = dict(D=5, M=100, S=256, N=4, T=3000, S_mc=5, D_obs=50, dt=0.01, ell0=1.25)
    rows = elbo_errors("shooting", kw, "rk4", {}, 11)
    worst, bad = 0.0, []
    for k, (e_cuda64, e_ref64, e_cuda32) in rows.items():
        ok = e_cuda32 <= 1e-4 or e_cuda64 <= max(1e-4, 1.5 * e_ref64)
        worst = max(worst, min(e_cuda32, e_cuda64))
        if not ok:
            bad.append((k, e_cuda64, e_ref64, e_cuda32))
    if bad:
        raise SystemExit("parity pre-check FAILED against the oracle: %r" % (bad,))
    return {"segments": kw["S_mc"] * kw["N"] * kw["T"], "tensors": len(rows), "worst_rel_err": worst,
            "rule": "<= 1e-4 vs the float32 oracle port, or no further from float64 than 1.5x the port's own float32 error"}


def run_ours(args):
    from gaussian_process_odes_b200 import _lib, distributed
    rank, world, local_rank = distributed.init_from_env()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU path exists)"
    if world != args.gpus:
        if rank == 0:
            print("warning: --gpus %d but WORLD_SIZE=%d" % (args.gpus, world), file=sys.stderr)
    w = WORKLOAD
    dev = torch.device("cuda", local_rank)
    cpus = pin_to_gpu_numa_node(local_rank)
    _lib.load()
    parity = None
    if rank == 0 and not args.no_parity_check:
        parity = parity_precheck()
    strong = args.scaling == "strong"
    distributed.seed_ranks(121, rank)
    model, ys_host, ts_host, N_glob, T = build_ours(w, rank, world, args.rows_scale, strong)
    N_loc = ys_host.shape[0]
    ys_pinned = ys_host.pin_memory()
    ts_dev = ts_host.to(dev)
    ys_dev = ys_pinned.to(dev, non_blocking=True)
    rows_local = w["S_mc"] * N_loc * T
    rows_total = w["S_mc"] * N_glob * T
    evals_per_step = rows_total * 4

    def eager_step(ys):
        model.zero_grad(set_to_none=True)
        loss = distributed.sharded_shooting_loss(model, ys, ts_dev, w["S_mc"], N_glob, world)
        loss.backward()
        distributed.allreduce_shared_grads(model)
        return loss

    # The step is ~110 launches, and the host needs about as long to issue them (8.1 ms of CPU time per step, torch
    # profiler) as the GPU needs to run them, so the GPU idles ~0.4 ms per step behind the host. The library's own
    # answer for launch-bound steps is graphs.GraphedStep: ELBO forward + backward captured once into a CUDA graph and
    # replayed; per step the host only draws the GP function's random numbers (numpy, reference order) into static
    # buffers. The observations enter through a static device buffer; the gradient all-reduce stays outside the graph.
    gstep, ys_static = None, None
    if not args.no_graph:
        try:
            from gaussian_process_odes_b200 import graphs
            ys_static = ys_dev.clone()
            gstep = graphs.GraphedStep(
                model, lambda: distributed.sharded_shooting_loss(model, ys_static, ts_dev, w["S_mc"], N_glob, world))
        except Exception as e:  # capture is an optimisation: report and fall back to eager launches
            if rank == 0:
                print("warning: CUDA-graph capture failed (%r); timing eager launches" % (e,), file=sys.stderr)
            gstep = None

    def step(ys):
        if gstep is None:
            return eager_step(ys)
        if ys is not ys_static:
            ys_static.copy_(ys, non_blocking=True)   # device -> device, 40 MB, on the compute stream
        loss = gstep()
        distributed.allreduce_shared_grads(model)
        return loss

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(nsteps, body):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(nsteps):
            body()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        return float(ms.item())

    resident = ys_static if gstep is not None else ys_dev   # device-resident input of the `value` measurement
    for _ in range(args.warmup):
        step(resident)

    # ---- device-resident measurement ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    last = {}

    def timed_step():
        last["loss"] = step(resident)

    ms_total = timed(args.steps, timed_step)
    # copied now: the graph's loss and gradient buffers are overwritten by the passes below
    outputs = step_outputs(model, last["loss"]) if args.dump_outputs and rank == 0 else None
    _lib.reset_launch_count()
    for _ in range(args.steps):   # the kernels a step launches are counted on eager launches (a graph replay runs the same)
        eager_step(ys_dev)
    launches = _lib.total_launches()
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = ms_total / args.steps
    value = evals_per_step / (ms_per_step * 1e-3)

    # ---- end to end: pinned host observations in, loss out, every step ----
    # The observations of step i+1 travel host -> device on a copy stream (double-buffered) while step i computes;
    # every step's copy and its loss read-back happen inside the timed region.
    copy_stream = torch.cuda.Stream()
    y_bufs = [torch.empty_like(ys_dev) for _ in range(2)]
    t_bufs = [torch.empty(ts_host.shape, dtype=ts_host.dtype, device=dev) for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    loss_host = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ready = [torch.cuda.Event(), torch.cuda.Event()]
    state = {"i": 0, "left": 0}

    def prefetch(i):
        copy_stream.wait_stream(torch.cuda.current_stream())  # the buffer's previous reader has been enqueued
        with torch.cuda.stream(copy_stream):
            y_bufs[i % 2].copy_(ys_pinned, non_blocking=True)
            t_bufs[i % 2].copy_(ts_host, non_blocking=True)
            ready[i % 2].record(copy_stream)

    def e2e_body():
        i = state["i"]
        if state["left"] == state["total"]:
            prefetch(i)  # first step of a timed region: its own copy, not overlapped with anything
        torch.cuda.current_stream().wait_event(ready[i % 2])
        y, t = y_bufs[i % 2], t_bufs[i % 2]
        state["left"] -= 1
        if gstep is None:
            model.zero_grad(set_to_none=True)
            loss = distributed.sharded_shooting_loss(model, y, t, w["S_mc"], N_glob, world)
            if state["left"] > 0:
                prefetch(i + 1)  # next step's inputs: in flight during this step's backward
            loss.backward()
            distributed.allreduce_shared_grads(model)
        else:
            ys_static.copy_(y, non_blocking=True)   # staging buffer -> the graph's static input (device to device)
            ts_dev.copy_(t, non_blocking=True)
            if state["left"] > 0:
                prefetch(i + 1)  # enqueued BEFORE the replay: the next step's inputs travel while this step's graph runs
            loss = gstep()
            distributed.allreduce_shared_grads(model)
        # device -> host read of every step's loss: copied to pinned host memory on the compute stream right after the
        # step, consumed one step later (so the host keeps issuing the next step instead of idling the GPU behind a
        # blocking .item()); the last step's value is awaited inside the timed region
        loss_host[i % 2].copy_(loss.detach(), non_blocking=True)
        loss_ready[i % 2].record()
        if state["left"] < state["total"] - 1:
            loss_ready[(i - 1) % 2].synchronize()
            e2e_body.last = float(loss_host[(i - 1) % 2])
        if state["left"] == 0:
            loss_ready[i % 2].synchronize()
            e2e_body.last = float(loss_host[i % 2])
        state["i"] = i + 1

    def e2e_run(n):
        state["left"] = state["total"] = n
        return timed(n, e2e_body)

    e2e_run(2)
    ms_e2e = e2e_run(args.steps) / args.steps
    e2e = {"value": evals_per_step / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
           "h2d_bytes_per_step": int((ys_pinned.numel() + ts_host.numel()) * 4 * world), "d2h_bytes_per_step": 4 * world,
           "h2d": "pinned host -> device every step, double-buffered on a copy stream (step i+1's copy overlaps step i); "
                  "every rank is bound to the CPU cores of its GPU's NUMA node before the pinned buffers are allocated",
           "d2h": "every step's loss -> pinned host (async copy after the step), read by the host one step later; the "
                  "last one is awaited inside the timed region", "cpu_affinity_rank0": cpus}

    # ---- per-kernel breakdown (separate pass: CUDA events around every C-ABI call, MEDIAN over n_prof steps) ----
    n_prof = args.steps
    _lib.profile_start()
    for _ in range(n_prof):
        eager_step(ys_dev)   # eager launches: the events bracket the individual C-ABI calls
    raw = _lib.profile_stop(raw=True)
    kern = {}
    for k, v in raw.items():
        per = max(1, len(v) // n_prof)                       # calls of this entry point per step
        per_step = [sum(v[i * per:(i + 1) * per]) for i in range(n_prof)]
        kern[k] = {"calls_per_step": len(v) / n_prof, "ms_per_step": float(np.median(per_step)),
                   "ms_min": float(min(per_step)), "ms_max": float(max(per_step))}
    ours_ms = sum(v["ms_per_step"] for v in kern.values())

    roof = None
    if rank == 0:
        import ctypes
        tf, ms_probe = ctypes.c_double(), ctypes.c_double()
        scratch = torch.zeros(4, device=dev)
        _lib.check(_lib.load().gpode_probe_fp32_fma(ctypes.byref(tf), ctypes.byref(ms_probe),
                                                    _lib.ptr(scratch), _lib.stream_ptr()))
        fv = f_vf(w["D"], w["S"], w["M"])
        FWD, BWD, PG = "gpode_shoot_fwd", "gpode_shoot_bwd", "gpode_param_grad"
        flops = {FWD: rows_local * (4 * fv + 14 * w["D"]),   # SURVEY 8d: 4 F_vf + 14 D per row-step
                 BWD: rows_local * 8 * fv}                     # 4 VJPs ~ 2 F_vf each; nothing is recomputed
        # transcendentals (MUFU: cos / sin / ex2) per launch: D S + D M per evaluation or VJP, four of them per row
        mufu_ops = rows_local * 4 * w["D"] * (w["S"] + w["M"])
        sm_clock = (clocks or {}).get("sm_mhz") or 1965.0
        try:
            n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        except Exception:
            n_sm = 148
        mufu_peak = 16.0 * n_sm * sm_clock * 1e6             # 16 MUFU results / clk / SM (4 per sub-partition)
        dom = max(flops, key=lambda k: kern.get(k, {"ms_per_step": 0})["ms_per_step"])
        ms_dom = kern[dom]["ms_per_step"] / max(kern[dom]["calls_per_step"], 1)
        achieved = flops[dom] / (ms_dom * 1e-3) / 1e12
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):
            try:
                traffic = json.load(open(tpath)).get(dom)
            except Exception:
                traffic = None
        other = FWD if dom == BWD else BWD

        def entry(k):
            ms = kern[k]["ms_per_step"]
            return {"achieved": flops[k] / (ms * 1e-3) / 1e12, "frac": flops[k] / (ms * 1e-3) / 1e12 / tf.value,
                    "kernel_ms": ms,
                    "mufu": {"transcendentals_per_launch": mufu_ops, "floor_ms": mufu_ops / mufu_peak * 1e3,
                             "frac": (mufu_ops / mufu_peak * 1e3) / ms,
                             "peak": "16 / clk / SM x %d SMs x %.0f MHz (median SM clock of the timed region)" % (
                                 n_sm, sm_clock)}}
        comb_ms = kern[BWD]["ms_per_step"] + kern.get(PG, {"ms_per_step": 0.0})["ms_per_step"]
        roof = {"bound": "fp32_fma", "kernel": dom, "achieved": achieved, "peak": tf.value, "unit": "TFLOP/s",
                "frac": achieved / tf.value, "traffic": traffic,
                "peak_source": "measured here: gpode_probe_fp32_fma (register-only FMA loop, best of 5); "
                               "MEASURED_PEAKS.json has no FP32 entry",
                "algorithmic_flops_per_launch": flops[dom], "kernel_ms": ms_dom,
                "mufu": entry(dom)["mufu"],
                "combined_adjoint": {"kernels": [BWD, PG], "ms": comb_ms,
                                     "achieved": flops[BWD] / (comb_ms * 1e-3) / 1e12,
                                     "frac": flops[BWD] / (comb_ms * 1e-3) / 1e12 / tf.value,
                                     "note": "the Z / nu half of every VJP runs in the second kernel; same 8 F_vf credit "
                                             "over both durations"},
                "pipes": "at 4 <= D <= 5 the adjoint runs the two Fourier projections of every VJP (theta = x Omega, "
                         "G = g Omega^T: 10 of the 14 algorithmic FMAs per feature-output) and the forward the projection "
                         "theta as split-fp16 mma.sync on the tensor cores (csrc/vjp_mma.cuh); the flop count stays the "
                         "algorithmic FP32 one and the peak stays the FP32 FMA peak, so frac measures the whole kernel "
                         "against the CUDA-core roofline; 'mufu' is the transcendental (cos/sin/ex2) floor of the same "
                         "launch, which binds the forward kernel. Both kernels now include the fused ELBO epilogue "
                         "(likelihood + constraint on the end point; csrc/shoot.cuh) at no extra credit",
                "also": {other: entry(other)},
                "hbm_note": "FMA-bound path: algorithmic HBM bytes are %d per row forward (arithmetic intensity > 1e3 "
                            "flop/byte), so the HBM roofline (MEASURED_PEAKS.json hbm_gbs) is not the binding one" % (
                                4 * w["D"] * 3)}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_elbo_timing(w, steps=5, warmup=1)
        sat = {}
        for Ts in (1000, 3000):   # saturation: the port's throughput no longer depends on the sample size
            c2 = cpu_elbo_timing(w, steps=3, warmup=1, T_sample=Ts)
            sat["%d_segments" % c2["rows"]] = c2["value"]
        sat["%d_segments" % cpu["rows"]] = cpu["value"]
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
        cpu["saturation_evals_per_s"] = sat

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling,
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": w["name"], "D": w["D"], "D_obs": w["D_obs"], "M": w["M"], "S": w["S"],
                           "S_mc": w["S_mc"], "N_sequences_per_gpu": N_loc, "N_sequences_total": N_glob, "T": T,
                           "solver": w["solver"], "segments_per_gpu": rows_local, "segments_total": rows_total,
                           "evals_per_step": evals_per_step, "parallelism": "sequences sharded x%d" % world,
                           "cuda_graph": gstep is not None,
                           "l2": "working set per step (>= 0.4 GB of sampled states, stage checkpoints, adjoint seeds "
                                 "and virtual rows per 10^6 segments) exceeds the 126 MB L2; no explicit flush"},
                "elbo_fwd_bwd_ms": ms_per_step, "e2e": e2e, "gpu_launches": launches * world,
                "kernels_ms_per_step": kern, "own_kernels_share_of_step": ours_ms / ms_per_step,
                "roofline": roof, "cpu_baseline": cpu, "clocks": clocks, "parity_precheck": parity,
                "loss": getattr(e2e_body, "last", None)}
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows-scale", type=float, default=1.0, help="scale T (segments per GPU) for quick runs")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: 16 sequences (10^6 segments) per GPU; strong: 16 sequences in total")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of the captured CUDA graph")
    ap.add_argument("--no-parity-check", action="store_true", help="skip the oracle check before timing (profiling)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and parameter gradients of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup not negative")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the CUDA path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
