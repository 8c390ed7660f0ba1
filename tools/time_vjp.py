#!/usr/bin/env python
"""Time one vector-field VJP (B = 1e6) with the tensor-core and the FFMA2 adjoint (tuning helper)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import gpode_oracle as O  # noqa: E402
from gaussian_process_odes_b200 import _lib, ops  # noqa: E402

D, M = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (5, 100)
S, B = 256, int(os.environ.get("TB_ROWS", 1000000))
p, ys, ts, draws, _ = O.make_problem(D=D, M=M, S=S, N=1, T=4, seed=5)
gp = O.gp_params(p)
omega = draws["eps_omega"] / gp["ell"].T.unsqueeze(1)
nu = torch.tensor(np.random.default_rng(1).normal(size=(D, M)) * 0.1, dtype=torch.float32)
args = [t.cuda().contiguous() for t in (gp["Z"], gp["ell"], gp["var"], nu, omega, draws["phase_u"] * 2 * np.pi,
                                        draws["w"])]
x = torch.randn(B, D, device="cuda")
gf = torch.randn(B, D, device="cuda")
pc = ops.PackedCache(*args)
f = ops.vector_field(x, *args)
gx = torch.empty_like(x)
ptr = ops.ptr
for mode in os.environ.get("TV_VARIANTS", "0,1").split(","):
    _lib.set_option("bwd_mma", int(mode))
    acc = pc.new_acc()
    def run():
        _lib.call("gpode_vf_bwd", ptr(pc.packed), pc.D, pc.M, pc.S, ptr(x), ptr(f), ptr(gf), ptr(gx), ptr(acc),
                  B, ops.stream_ptr())
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        run()
    e1.record()
    torch.cuda.synchronize()
    print(json.dumps(dict(D=D, mma=mode, vjp_ms=round(e0.elapsed_time(e1) / 10, 4))), flush=True)
