"""Multi-GPU data parallelism over independent sequences / shooting segments (SURVEY.md section 8e).

One process per GPU (``torch.distributed``, NCCL over NVLink). The multiple-shooting ELBO is a sum over sequences
(reference ``src/gpode_shooting/models.py:119-146``): each rank owns a contiguous block of sequences together with
their variational state parameters, every rank holds the same GP / likelihood parameters and draws the SAME GP
function sample (the reference draws it with numpy's global generator, so seeding numpy identically on all ranks is
enough), and the only exchange per step is ONE all-reduce(sum) of the small flattened shared-parameter gradient.
There is no data-path collective: segment rows never leave their GPU.
"""
import os

import numpy as np
import torch
import torch.distributed as dist


def init_from_env(backend=None):
    """Initialise the default process group from torchrun's environment; returns (rank, world, local_rank)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if torch.cuda.is_available():
        torch.cuda.set_device(local_rank)
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        kw = {}
        if backend == "nccl":
            kw["device_id"] = torch.device("cuda", local_rank)
        dist.init_process_group(backend=backend, rank=rank, world_size=world, **kw)
    return rank, world, local_rank


def shard_range(n_total, rank, world):
    """Contiguous, balanced block ``[lo, hi)`` of ``n_total`` sequences for ``rank`` (first ranks get the remainder)."""
    base, rem = divmod(n_total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def seed_ranks(seed, rank, same_states=False):
    """numpy (GP function draws: identical on every rank) vs torch (state samples: different per rank when the
    sequences are sharded, identical -- ``same_states=True`` -- when the rows of one replicated batch are sharded)."""
    np.random.seed(seed)
    tseed = seed + (0 if same_states else 1000003 * (rank + 1))
    torch.manual_seed(tseed)
    if torch.cuda.is_available():
        torch.cuda.manual_seed(tseed)


def shared_parameters(model):
    """Parameters replicated on every rank (GP, likelihood, constraint) -- everything but the per-sequence states."""
    local = set()
    for name in ("state_distribution", "x0_distribution"):
        mod = getattr(model, name, None)
        if mod is not None:
            local.update(id(p) for p in mod.parameters())
    return [p for p in model.parameters() if id(p) not in local]


def broadcast_shared_parameters(model, src=0):
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    params = shared_parameters(model)
    flat = torch.cat([p.data.reshape(-1) for p in params])
    dist.broadcast(flat, src=src)
    off = 0
    for p in params:
        n = p.numel()
        p.data.copy_(flat[off:off + n].view_as(p))
        off += n


def allreduce_shared_grads(model):
    """ONE all-reduce(sum) over the flattened gradients of the shared parameters (a few thousand floats)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return 0
    params = [p for p in shared_parameters(model) if p.requires_grad]
    flat = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in params])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    off = 0
    for p in params:
        n = p.numel()
        g = flat[off:off + n].view_as(p)
        if p.grad is None:
            p.grad = g.clone()
        else:
            p.grad.copy_(g)
        off += n
    return flat.numel()


def combine_shard_terms(observ_loglik_mean_local, scaled_constraint, scaled_entropy, scaled_init_kl, scaled_inducing_kl,
                        n_local, n_global, world):
    """Rank-local loss whose SUM over ranks is the global negative ELBO.

    The model on each rank is built with the GLOBAL ``num_observations``, so the constraint / entropy / initial-KL
    terms (sums over local sequences divided by the global count) just add up; the observation term is a mean over
    local observations and is re-weighted by ``n_local / n_global``; the inducing KL is counted once."""
    w = float(n_local) / float(n_global)
    return -(w * observ_loglik_mean_local + scaled_constraint + scaled_entropy - scaled_init_kl
             - scaled_inducing_kl / float(world))


def sharded_shooting_loss(model, ys_local, ts, num_samples, n_global, world):
    ll, cons, ent, k0 = model.build_lowerbound_terms(ys_local, ts, num_samples=num_samples)
    kl = model.build_inducing_kl()
    return combine_shard_terms(ll, cons, ent, k0, kl, ys_local.shape[0], n_global, world)


# ---- segment-row sharding: fewer sequences than GPUs (VDP: N = 1, MoCap-09: N = 6) -----------------------------------
# The (S_mc, N, T) segment batch of one ELBO evaluation (reference src/gpode_shooting/models.py:119-125) is cut into
# contiguous row blocks, one per rank, across Monte-Carlo samples, sequences AND time. Every rank keeps ALL variational
# parameters and draws the same state samples and the same GP function, so the constraint's neighbour state
# (models.py:134-135: the state one row past a block's end) is already local -- the halo of a block is one row of the
# replicated sample tensor, no exchange -- and the only collective is ONE all-reduce(sum) of the flattened gradient of
# every parameter: a rank's gradient w.r.t. the sampled states is non-zero only on its rows (+ the halo row).
def enable_row_sharding(model, rank=None, world=None):
    """Make ``model.build_lowerbound_terms`` integrate only this rank's block of segment rows (fused shooting step:
    rk4, an affine decoder with D_obs <= 128 and a frozen constraint scale, at every state dimension 1 <= D <= 64)."""
    if rank is None:
        rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
        world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    model.row_shard = (int(rank), int(world)) if world > 1 else None
    return model


def row_sharded_shooting_loss(model, ys, ts, num_samples, world=None):
    """Rank-local loss whose SUM over ranks is the global negative ELBO: the observation and constraint terms are this
    rank's share, the replicated terms (entropy, initial-state KL, inducing KL) are counted ``1/world`` times each."""
    if world is None:
        world = model.row_shard[1] if model.row_shard is not None else 1
    ll, cons, ent, k0 = model.build_lowerbound_terms(ys, ts, num_samples=num_samples)
    kl = model.build_inducing_kl()
    return -(ll + cons + (ent - k0 - kl) / float(world))


# ---- time sharding: ONE (or few) long sequence(s) -- VDP shooting, BASELINE configs[1] --------------------------------
# Row sharding keeps the whole variational state distribution on every rank: its Cholesky factors, samples, entropy and
# their backward (2e5 matrices for a 1e6-segment VDP problem) are replicated, and measured on 8 GPUs that is 2.5 of the
# 4 ms of a step -- no scaling. Time sharding gives each rank a contiguous slice [lo, hi) of the TIME axis of every
# sequence (all Monte-Carlo samples): it factorises / samples only the states of its slice plus one halo state (the
# next slice's first state, the constraint's neighbour), integrates the slice's segments, and owns their gradient rows.
# The halo state's gradient (the constraint's pull) lands on a parameter row owned by the next rank: the same single
# all-reduce(sum) of all gradients delivers it. Every rank draws the same noise (full shape, same order, then sliced),
# so the result equals the unsharded one.
def enable_time_sharding(model, rank=None, world=None):
    """Make ``model.build_lowerbound_terms`` evaluate only this rank's slice of the time axis (fused shooting step:
    rk4, an affine decoder with D_obs <= 128 and a frozen constraint scale, at every state dimension 1 <= D <= 64)."""
    if rank is None:
        rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
        world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    model.time_shard = (int(rank), int(world)) if world > 1 else None
    model.row_shard = None
    return model


def time_sharded_shooting_loss(model, ys, ts, num_samples, world=None):
    """Rank-local loss whose SUM over ranks is the global negative ELBO: observation, constraint and entropy terms are
    this rank's share; the replicated terms (initial-state KL, inducing KL) are counted ``1/world`` times each."""
    if world is None:
        world = model.time_shard[1] if model.time_shard is not None else 1
    ll, cons, ent, k0 = model.build_lowerbound_terms(ys, ts, num_samples=num_samples)
    kl = model.build_inducing_kl()
    return -(ll + cons + ent - (k0 + kl) / float(world))


def allreduce_all_grads(model):
    """ONE all-reduce(sum) over the flattened gradients of EVERY parameter (row sharding: all parameters are replicated)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return 0
    params = [p for p in model.parameters() if p.requires_grad]
    flat = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in params])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    off = 0
    for p in params:
        n = p.numel()
        g = flat[off:off + n].view_as(p)
        if p.grad is None:
            p.grad = g.clone()
        else:
            p.grad.copy_(g)
        off += n
    return flat.numel()


# ---- prediction: the Monte-Carlo draws are independent caches -> shard the draws (SURVEY.md section 8e) -------------
def gather_draws(local, n_total):
    """All-gather per-rank blocks of draws ``(n_local, ...)`` (block sizes from ``shard_range``) into the full
    ``(n_total, ...)`` tensor, in rank order, on every rank."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return local
    world = dist.get_world_size()
    sizes = [shard_range(n_total, r, world) for r in range(world)]
    biggest = max(hi - lo for lo, hi in sizes)
    pad = torch.zeros((biggest,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    pad[:local.shape[0]] = local
    parts = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(parts, pad)
    return torch.cat([parts[r][:hi - lo] for r, (lo, hi) in enumerate(sizes)], 0)


def sharded_predictions(model, ts, eval_sample_size, predict_fn=None, **kwargs):
    """``compute_predictions`` with the draws split across ranks: rank r computes draws ``shard_range(S, r, world)``
    through the batched n_sets path and every rank receives all ``(S,N,T,D)`` trajectories. Seed numpy / torch
    differently per rank (``seed_ranks`` keeps numpy identical on purpose -- for prediction offset it by the rank),
    otherwise every rank would integrate the same functions."""
    from . import builders
    rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    lo, hi = shard_range(eval_sample_size, rank, world)
    fn = builders.compute_predictions if predict_fn is None else predict_fn
    local = fn(model, ts, eval_sample_size=hi - lo, **kwargs)
    return gather_draws(local, eval_sample_size)
