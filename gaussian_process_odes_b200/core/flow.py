"""``ODEfunc`` / ``Flow``: the integrator boundary (mirror of reference ``src/core/flow.py``).

``Flow.forward(x0, ts)`` rebuilds the GP cache and integrates with the fused CUDA integrators through the
torchdiffeq-compatible ``odeint`` of ``gaussian_process_odes_b200.odeint`` (reference ``flow.py:60-90``). The NFE
counter buffer ``_num_evals`` is kept (``flow.py:18,26-27``) but is bumped once per integration by the number of
evaluations the kernel performed instead of by one tiny kernel launch per evaluation (``flow.py:30``)."""
import torch
import torch.nn as nn

from ..misc.settings import settings
from ..odeint import odeint as odeint_nonadjoint
from ..odeint import odeint_adjoint


class ODEfunc(nn.Module):
    def __init__(self, diffeq):
        super().__init__()
        self.diffeq = diffeq
        self.register_buffer("_num_evals", torch.tensor(0., device=settings.device))
        self.return_divergence = False

    def before_odeint(self, return_divergence, rebuild_cache):
        self.return_divergence = return_divergence
        self._num_evals.fill_(0)
        if rebuild_cache:
            self.diffeq.build_cache()

    def num_evals(self):
        return self._num_evals.item()

    def count_evals(self, n):
        self._num_evals += n

    def forward(self, t, states):
        self._num_evals += 1
        if self.return_divergence:
            # dead branch in the reference too: DSVGP_Layer has no forward_divergence (flow.py:31-34)
            raise NotImplementedError("divergence integration is not part of GPODE (no forward_divergence exists)")
        return self.diffeq(t, states)


class Flow(nn.Module):
    def __init__(self, diffeq, solver='dopri5', atol=1e-6, rtol=1e-6, use_adjoint=False):
        super().__init__()
        self.odefunc = ODEfunc(diffeq)
        self.solver = solver
        self.atol = atol
        self.rtol = rtol
        self.use_adjoint = use_adjoint

    def forward(self, x0, ts, return_divergence=False, rebuild_cache=True):
        """IVP solution ``(N,T,D)`` for initial states ``x0 (N,D)`` on the time sequence ``ts (T,)``. A new GP function
        is drawn per call unless ``rebuild_cache=False`` (the current draw is integrated)."""
        if return_divergence:
            raise NotImplementedError("divergence integration is not part of GPODE (dead branch, flow.py:70-80)")
        odeint = odeint_adjoint if self.use_adjoint else odeint_nonadjoint
        self.odefunc.before_odeint(return_divergence=False, rebuild_cache=rebuild_cache)
        xs = odeint(self.odefunc, x0, ts, atol=self.atol, rtol=self.rtol, method=self.solver)
        return xs.permute(1, 0, 2)

    def forward_sets(self, x0, ts, rng="numpy"):
        """Batched Monte-Carlo prediction: ``x0 (n,N,D)`` -> ``(n,N,T,D)``, draw q of the GP integrating ``x0[q]``.
        Equivalent to ``n`` calls of ``forward`` (cache rebuilt per call, ``flow.py:69``) under ``torch.no_grad()`` --
        the body of the reference's ``compute_predictions`` loop -- but one whitening, one pack and ONE integrator
        launch for all draws (dopri5 keeps one step-size controller per draw)."""
        from .. import ops
        layer = self.odefunc.diffeq
        with torch.no_grad():
            nu, omega, phase, w = layer.build_cache_sets(x0.shape[0], rng=rng)
            xs, stats = ops.integrate_sets(x0, ts, layer.inducing_loc(), layer.kern.lengthscales_dimwise(),
                                           layer.kern.variance_dimwise(), nu, omega, phase, w, method=self.solver,
                                           rtol=self.rtol, atol=self.atol)
        self.last_sets_stats = stats  # device int32 (n,4) for dopri5: nfe, accepted, rejected, status
        return xs

    def inverse(self, x0, ts, return_divergence=False):
        """Backward-in-time solve on the flipped grid, re-using the current cache (reference ``flow.py:92-115``)."""
        if return_divergence:
            raise NotImplementedError("divergence integration is not part of GPODE")
        odeint = odeint_adjoint if self.use_adjoint else odeint_nonadjoint
        self.odefunc.before_odeint(return_divergence=False, rebuild_cache=False)
        xs = odeint(self.odefunc, x0, torch.flip(ts, [0]), atol=self.atol, rtol=self.rtol, method=self.solver)
        return xs.permute(1, 0, 2)

    def num_evals(self):
        return self.odefunc.num_evals()

    def kl(self):
        return self.odefunc.diffeq.kl().sum()
