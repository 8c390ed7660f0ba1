"""-m gpu: the tensor-core shooting adjoint that sums the inducing-point gradients itself (D = 4, 5, batches that fill
the GPU: no virtual rows, no gpode_param_grad) against the FFMA2 adjoint followed by gpode_param_grad (bwd_mma = 0),
for every parameter gradient, at inducing-point counts that leave a partial last group, batch sizes that are no
multiple of 32 or of a CTA's rows, and whitened weights |nu| ~ 1e2 whose terms cancel; repeated passes are bitwise
equal."""
import math

import pytest
import torch

from util import TOL_GRAD, relerr

pytestmark = pytest.mark.gpu


def _inputs(D, M, S, S_mc, N, T, nu_scale, seed, Dobs=3):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g)
    ell = 1.3 * (1 + 0.1 * r(D, D)).abs()
    cache = dict(Z=r(M, D) * 1.5, ell=ell, var=0.5 * (1 + 0.1 * r(D)).abs(), nu=r(D, M) * nu_scale,
                 omega=r(D, S, D) / ell[:, None, :], phase=torch.rand(S, D, generator=g) * 2 * math.pi, w=r(S, D))
    data = dict(ss=r(S_mc, N, T, D), ys=r(N, T, Dobs), W=r(D, Dobs) * 0.3, bias=r(Dobs) * 0.1,
                lik_var=0.5 + torch.rand(Dobs, generator=g), cons=torch.tensor([0.05]))
    return cache, data


def _grads(cache, data, bwd_mma):
    from gaussian_process_odes_b200 import ops, _lib
    _lib.set_option("bwd_mma", int(bwd_mma))
    try:
        leaves = {k: v.cuda().requires_grad_(k in ("Z", "ell", "var", "nu")) for k, v in cache.items()}
        ss = data["ss"].cuda().requires_grad_(True)
        ll, c, _ = ops.shooting_step(ss, torch.tensor([0.0, 0.01]).cuda(), leaves["Z"], leaves["ell"], leaves["var"],
                                     leaves["nu"], leaves["omega"], leaves["phase"], leaves["w"], data["ys"].cuda(),
                                     data["W"].cuda(), data["bias"].cuda(), data["lik_var"].cuda(),
                                     data["cons"].cuda())
        (ll + c).backward()
    finally:
        _lib.set_option("bwd_mma", 1)
    out = {k: leaves[k].grad for k in ("Z", "ell", "var", "nu")}
    out["ss"] = ss.grad
    return out


def _vrows(D, M, S, B, bwd_mma):
    from gaussian_process_odes_b200 import _lib
    _lib.set_option("bwd_mma", int(bwd_mma))
    try:
        return _lib.load().gpode_shoot_bwd_vrows(D, M, S, B)
    finally:
        _lib.set_option("bwd_mma", 1)


# B = S_mc N T >= 56 832 (148 SMs x 384 rows) selects the tensor-core adjoint on a B200
@pytest.mark.parametrize("D,M,S,S_mc,N,T,nu_scale", [
    (5, 100, 256, 3, 2, 9501, 0.3),     # the benchmark's field; B = 57 006
    (5, 37, 64, 3, 1, 19001, 0.3),      # 37 = 12 groups of 3 + 1
    (5, 1, 32, 2, 1, 28500, 0.3),
    (5, 128, 128, 3, 1, 19001, 0.3),
    (4, 37, 100, 3, 1, 19003, 0.3),     # 37 = 9 groups of 4 + 1
    (4, 128, 256, 1, 3, 19001, 0.3),
    (5, 100, 256, 3, 2, 9501, 100.0),   # whitened weights of a trained model: the per-row terms cancel
    (4, 37, 100, 3, 1, 19003, 100.0),
])
def test_row_sums_match_the_virtual_row_kernel(D, M, S, S_mc, N, T, nu_scale):
    B = S_mc * N * T
    if torch.cuda.get_device_properties(0).multi_processor_count * 384 > B:
        pytest.skip("the tensor-core adjoint needs a batch that fills this GPU")
    assert _vrows(D, M, S, B, 1) == 0 and _vrows(D, M, S, B, 0) == 4 * B
    cache, data = _inputs(D, M, S, S_mc, N, T, nu_scale, seed=D * 1000 + M)
    got, base = _grads(cache, data, 1), _grads(cache, data, 0)
    for k in got:
        assert torch.isfinite(got[k]).all(), k
        assert relerr(got[k], base[k]) <= TOL_GRAD, (k, relerr(got[k], base[k]))


def test_row_sums_are_bitwise_reproducible():
    cache, data = _inputs(5, 100, 256, 3, 2, 9501, 0.3, seed=11)
    a, b = _grads(cache, data, 1), _grads(cache, data, 1)
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_configurations_without_room_for_the_row_sums_keep_the_virtual_rows():
    """D = 5, S = 256: the per-warp row sums fit next to the operand records up to M = 101; above that (and below
    D = 4, or for small batches) the caller gets the virtual-row count and gpode_param_grad runs as before."""
    B = 60000
    assert _vrows(5, 102, 256, B, 1) == 4 * B
    assert _vrows(3, 24, 64, B, 1) == 4 * B
    assert _vrows(5, 100, 256, 1000, 1) == 4000
