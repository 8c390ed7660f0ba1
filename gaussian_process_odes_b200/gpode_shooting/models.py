"""Multiple-shooting GPODE (mirror of reference ``src/gpode_shooting/models.py``): every one-interval segment of every
sampled state sequence is one row of a single wide batch that the fused integrator advances in one launch."""
from torch import nn

from ..misc.torch_utils import compute_ts_dense


def stack_segments(unstacked):
    return unstacked.reshape(-1, unstacked.shape[-1])


def unstack_segments(stacked, unstacked_shape):
    return stacked.reshape(unstacked_shape)


class BaseSequenceModel(nn.Module):
    def __init__(self, flow, num_observations, state_distribution, likelihood, constraint, ts_dense_scale=2):
        super().__init__()
        self.flow = flow
        self.num_observations = num_observations
        self.state_distribution = state_distribution
        self.likelihood = likelihood
        self.constraint = constraint
        self.ts_dense_scale = ts_dense_scale

    def build_flow(self, x0, ts):
        if self.ts_dense_scale < 2:
            raise ValueError("ts_dense_scale must be >= 2")
        dense = compute_ts_dense(ts, self.ts_dense_scale)
        ys = self.flow(x0, dense, return_divergence=False)
        return ys[:, ::self.ts_dense_scale - 1, :]

    def build_lowerbound_terms(self, ys, ts, **kwargs):
        raise NotImplementedError

    def build_objective(self, ys, ts):
        observ_loglik, state_constraint_loglik, state_entropy, initial_state_kl = self.build_lowerbound_terms(ys, ts)
        inducing_kl = self.build_inducing_kl()
        return -(observ_loglik + state_constraint_loglik + state_entropy - initial_state_kl - inducing_kl)

    def build_inducing_kl(self):
        return self.flow.kl() / self.num_observations

    def forward(self, x0, ts):
        return self.build_flow(x0, ts)

    def forward_sets(self, x0, ts, rng="numpy"):
        """``x0 (n,N,D)`` -> ``(n,N,T,D)``: ``forward`` for n independent GP draws in one launch (prediction only)."""
        if self.ts_dense_scale < 2:
            raise ValueError("ts_dense_scale must be >= 2")
        dense = compute_ts_dense(ts, self.ts_dense_scale)
        return self.flow.forward_sets(x0, dense, rng=rng)[:, :, ::self.ts_dense_scale - 1, :]


class _FusedDoesNotFit(Exception):
    """The fused shooting step refused its launch for shared memory; the cache of this step's GP draw is built."""


class UniformSequenceModel(BaseSequenceModel):
    """Observations on a uniform time grid: every segment spans ``ts[:2]`` (reference ``models.py:88-146``)."""

    # rows of the (S,N,T) segment batch this process integrates: None = all, or (rank, world) set by
    # ``distributed.enable_row_sharding`` (contiguous row blocks; every rank samples the same states)
    row_shard = None
    # a contiguous slice of the TIME axis per process, set by ``distributed.enable_time_sharding``: the state-distribution
    # work (Cholesky, sampling, entropy and their backward) shards together with the segment rows
    time_shard = None
    fuse_elbo = True   # False: the unfused path (separate integrator / likelihood / constraint launches)

    def _fused_terms(self, ss_samples, ys, ts, halo=False, T_global=None):
        """Observation log-likelihood mean and constraint total through ONE integrator launch with the two terms
        evaluated on the segment end points inside the kernel (``ops.shooting_step``), or None when the configuration
        has no fused kernel (solver other than rk4, D > 64, D_obs > 128, non-affine decoder, trainable constraint scale,
        CPU). Above D = 8 the step runs on the large-D kernels (tcgen05 vector field, one epilogue kernel). Raises
        _FusedDoesNotFit, with this step's GP cache already built, when the fused forward does not fit in shared
        memory."""
        from ..core.dsvgp import DSVGP_Layer
        from ..core.constraints import _ScaleFamily
        from ..ops import MAX_D_LARGE
        flow, lik, cons = self.flow, self.likelihood, self.constraint
        layer = flow.odefunc.diffeq
        S, N, T, D = ss_samples.shape
        affine = getattr(lik, "_affine", None)
        if not (self.fuse_elbo and ss_samples.is_cuda and flow.solver == "rk4" and isinstance(layer, DSVGP_Layer)
                and D <= MAX_D_LARGE and affine is not None and isinstance(cons, _ScaleFamily)
                and not cons.unconstrained_scale.requires_grad and cons.unconstrained_scale.numel() == 1):
            return None
        aff = affine(ss_samples)
        if aff is None:
            return None
        W, b = aff
        Dobs = W.shape[1]
        if W.shape[0] != D or Dobs > 128 or tuple(ys.shape) != (N, T, Dobs):
            return None
        from .. import ops
        from .._lib import GpodeError
        var = lik.variance
        if var.numel() != Dobs:
            var = var.expand(Dobs)
        rows = None
        if self.row_shard is not None and T_global is None:
            from ..distributed import shard_range
            rows = shard_range(S * N * T, *self.row_shard)
        flow.odefunc.before_odeint(return_divergence=False, rebuild_cache=True)
        try:
            ll_sum, cons_sum, _ = ops.shooting_step(ss_samples, ts[:2], *layer.cache_tensors(), ys, W, b, var,
                                                    cons.scale.detach(), laplace=cons._laplace, rows=rows, halo=halo)
        except GpodeError as e:
            # the epilogue's shared memory comes on top of the integrator's block: at many inducing points the fused
            # forward is refused (before any launch) where the separate integrator and side-term kernels still fit. A
            # sharded step has no unfused form: there the refusal is the error to report.
            if "does not fit" not in str(e) or self.row_shard is not None or T_global is not None:
                raise
            raise _FusedDoesNotFit() from e
        flow.odefunc.count_evals(4)
        return ll_sum / float(S * N * (T if T_global is None else T_global) * Dobs), cons_sum / S

    def _time_sharded_terms(self, ys, ts, num_samples):
        """This process's share of the four ELBO terms under time sharding: segments with time index in its slice
        ``[lo, hi)`` of the ``T`` indices of every sequence, for all Monte-Carlo samples. The sampled states of the slice
        plus ONE halo index (the next slice's first state: the constraint's neighbour, reference ``models.py:134-135``)
        are computed locally from the parameter rows of the slice, so sampling, entropy and their backward shard with the
        rows; the halo's gradient reaches its owner through the all-reduce. Observation and constraint terms and the
        entropy add up over the processes; the initial-state KL is replicated (weighted ``1/world`` by
        ``distributed.time_sharded_shooting_loss``)."""
        from ..distributed import shard_range
        sd = self.state_distribution
        rank, world = self.time_shard
        T = sd.dim_t + 1
        lo, hi = shard_range(T, rank, world)
        halo = hi < T
        zero = ys.new_zeros(())
        initial_state_kl = sd.x0.kl()
        if hi <= lo:   # more processes than time indices
            sd.sample_time_slice(num_samples, 0, 1)   # keep the random streams of all processes aligned
            self.flow.odefunc.before_odeint(return_divergence=False, rebuild_cache=True)
            return zero, zero, zero, initial_state_kl / self.num_observations
        ss_loc = sd.sample_time_slice(num_samples, lo, hi + int(halo))          # (S, N, hi - lo (+1), D)
        fused = self._fused_terms(ss_loc, ys[:, lo:hi + int(halo)].contiguous(), ts, halo=halo, T_global=T)
        if fused is None:
            raise RuntimeError("time sharding needs the fused shooting step (rk4, affine decoder with D_obs <= 128, "
                               "frozen constraint scale, D <= 64)")
        observation_loglik_mean, constraint_total = fused
        entropy = sd.entropy_time_slice(lo, hi).sum()
        return (observation_loglik_mean, constraint_total / self.num_observations, entropy / self.num_observations,
                initial_state_kl / self.num_observations)

    def build_lowerbound_terms(self, ys, ts, num_samples=1, **kwargs):
        """-> (observation log-lik mean, constraint log-lik, state entropy, initial-state KL), the last three scaled
        by ``1/num_observations`` (reference ``models.py:108-146``). With ``row_shard`` set the first two are this
        process's share (sums over its rows with the global normalisation): they add up over the ranks."""
        if self.time_shard is not None:
            return self._time_sharded_terms(ys, ts, num_samples)
        ss_samples = self.state_distribution.sample(num_samples=num_samples)  # (S,N,T,D)
        (S, N, T, D) = ss_samples.shape
        rebuild_cache = True
        try:
            fused = self._fused_terms(ss_samples, ys, ts)
        except _FusedDoesNotFit:
            fused, rebuild_cache = None, False   # integrate with the GP draw the fused attempt built
        if fused is not None:
            observation_loglik_mean, constraint_total = fused
            state_entropy = self.state_distribution.entropy()  # (N,T-1)
            initial_state_kl = self.state_distribution.x0.kl()
            assert state_entropy.shape == (N, T - 1)
            return (observation_loglik_mean, constraint_total / self.num_observations,
                    state_entropy.sum() / self.num_observations, initial_state_kl / self.num_observations)
        if self.row_shard is not None:
            raise RuntimeError("row sharding needs the fused shooting step (rk4, affine decoder with D_obs <= 128, "
                               "frozen constraint scale, D <= 64)")
        # one launch: S*N*T independent one-interval IVPs sharing one GP function draw
        predicted_xs = self.flow(x0=stack_segments(ss_samples), ts=ts[:2], rebuild_cache=rebuild_cache)  # (S*N*T, 2, D)
        predicted_xs = unstack_segments(predicted_xs[:, -1], (S, N, T, D))
        # mean log-likelihood: one fused decode + log-density kernel when the likelihood offers it
        mean_fn = getattr(self.likelihood, "log_prob_mean", None)
        if mean_fn is not None:
            observation_loglik_mean = mean_fn(predicted_xs, ys.unsqueeze(0))
        else:
            observation_loglik_mean = self.likelihood.log_prob(predicted_xs, ys.unsqueeze(0)).mean()
        state_entropy = self.state_distribution.entropy()  # (N,T-1)
        shooting_sum = getattr(self.constraint, "shooting_sum", None)
        if shooting_sum is not None:
            # mean over samples of the sum over (n, t, d): one fused kernel instead of a chain of (S,N,T-1,D) ops
            constraint_total = shooting_sum(ss_samples, predicted_xs) / S
        else:
            state_constraint_logprob = self.constraint.log_prob(ss_samples[:, :, 1:, :],
                                                                predicted_xs[:, :, :-1, :]).sum(3)  # (S,N,T-1)
            assert state_constraint_logprob.shape == (S, N, T - 1)
            constraint_total = state_constraint_logprob.mean(0).sum()
        initial_state_kl = self.state_distribution.x0.kl()
        assert state_entropy.shape == (N, T - 1)
        scaled_state_constraint_loglik = constraint_total / self.num_observations
        scaled_state_entropy = state_entropy.sum() / self.num_observations
        scaled_initial_state_kl = initial_state_kl / self.num_observations
        return observation_loglik_mean, scaled_state_constraint_loglik, scaled_state_entropy, scaled_initial_state_kl
