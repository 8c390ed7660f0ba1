"""CPU: the shared-memory limits of the D <= 8 integrator kernels above 160 inducing points (tests/util.py restates
each launcher's block size as a function of D, M and S), checked against the library's host queries, and the
launchers' refusal of an oversized block before any CUDA call.

M*(family, D, S) is the largest M whose block fits the 227 KB a CTA can opt into; tests/test_gpu_many_inducing.py
takes its boundary cases from this table."""
import ctypes

import pytest

from util import MAX_M_BLOCKED, SMEM_FAMILIES, SMEM_OPTIN, kernel_smem, max_inducing, packed_layout

S_TABLE = (64, 256, 512)

# every (family, D) whose block can outgrow the 227 KB at M <= 2048, with M*; all others cannot run out of room there
LIMITS = {
    64: {("tc_row_sums", 4): 341, ("tc_row_sums", 5): 239},
    256: {("bwd_warp", 7): 1584, ("bwd_warp", 8): 1159, ("tc_bwd", 5): 1116, ("tc_row_sums", 4): 201,
          ("tc_row_sums", 5): 101, ("shoot_tc_fwd", 5): 1851},
    512: {("fwd", 7): 1388, ("fwd", 8): 1067, ("dopri5_fwd", 7): 1386, ("dopri5_fwd", 8): 1066, ("bwd", 7): 1332,
          ("bwd", 8): 995, ("bwd_warp", 6): 1866, ("bwd_warp", 7): 464, ("bwd_warp", 8): 0, ("tc_fwd", 4): 1493,
          ("tc_fwd", 5): 169, ("tc_bwd", 4): 189, ("tc_bwd", 5): 0, ("tc_row_sums", 4): 14, ("tc_row_sums", 5): 0,
          ("shoot_fwd", 7): 1243, ("shoot_fwd", 8): 914, ("shoot_tc_fwd", 4): 991, ("shoot_tc_fwd", 5): 0},
}


@pytest.mark.parametrize("S", S_TABLE)
def test_limit_table(S):
    got = {}
    for family, (Ds, _, _) in SMEM_FAMILIES.items():
        for D in Ds:
            m = max_inducing(family, D, S)
            if m is None:
                assert kernel_smem(family, D, MAX_M_BLOCKED, S) <= SMEM_OPTIN
                continue
            got[(family, D)] = m
            assert kernel_smem(family, D, m + 1, S) > SMEM_OPTIN
            assert m == 0 or kernel_smem(family, D, m, S) <= SMEM_OPTIN
    assert got == LIMITS[S]


def test_limit_table_orders_the_families():
    """a kernel that stages more than another runs out of room first: the row-sum adjoint before the tensor-core
    adjoint, the warp adjoints (float64 slabs) before the row-per-thread ones, dopri5 (its static arrays) and the fused
    shooting forward (its epilogue) before the other forward kernels"""
    big = MAX_M_BLOCKED + 1
    m = lambda f, D, S: big if max_inducing(f, D, S) is None else max_inducing(f, D, S)
    for S in (33, 64, 129, 256, 512):
        for D in range(1, 9):
            assert m("bwd_warp", D, S) <= m("bwd", D, S) <= m("fwd", D, S)
            assert m("dopri5_fwd", D, S) <= m("fwd", D, S)
            assert m("shoot_fwd", D, S) <= m("fwd", D, S)
        for D in (4, 5):
            assert m("tc_row_sums", D, S) <= m("tc_bwd", D, S) <= m("tc_fwd", D, S)
            assert m("shoot_tc_fwd", D, S) <= m("tc_fwd", D, S)


@pytest.mark.parametrize("S", [1, 33, 64, 129, 256, 512])
@pytest.mark.parametrize("D", range(1, 9))
def test_packed_floats_match_layout(D, S):
    from gaussian_process_odes_b200 import _lib
    lib = _lib.load()
    for M in (1, 160, 161, 257, 1023, 2048):
        assert lib.gpode_packed_floats(D, M, S) == packed_layout(D, M, S)['n_packed'], (D, M, S)


@pytest.mark.parametrize("S", [33, 64, 129, 256, 512])
@pytest.mark.parametrize("D", [4, 5])
def test_row_sums_switch_to_virtual_rows_at_the_table_limit(D, S):
    """gpode_shoot_bwd_vrows is 0 (the tensor-core adjoint sums the inducing-point gradients) up to M* of the
    row-sum family and 4 rows per segment from M* + 1: at S = 256 that is M = 101 at D = 5 and M = 201 at D = 4"""
    from gaussian_process_odes_b200 import _lib
    lib = _lib.load()
    rows = 10 ** 7      # above SMs * 384 on any device: the tensor-core adjoint is chosen
    m = max_inducing("tc_row_sums", D, S)
    if S == 256:
        assert m == {5: 101, 4: 201}[D]
    if m >= 1:
        assert lib.gpode_shoot_bwd_vrows(D, m, S, rows) == 0
    assert lib.gpode_shoot_bwd_vrows(D, m + 1, S, rows) == 4 * rows
    assert lib.gpode_shoot_bwd_vrows(D, 1, S, 1000) == 4000   # small batches: FFMA2 adjoint, virtual rows


@pytest.mark.parametrize("D", [1, 2, 3, 6, 7, 8])
def test_other_dimensions_always_need_virtual_rows(D):
    from gaussian_process_odes_b200 import _lib
    lib = _lib.load()
    for M in (1, 101, 2048):
        assert lib.gpode_shoot_bwd_vrows(D, M, 64, 10 ** 7) == 4 * 10 ** 7


def oversized_calls(lib, fake):
    """(entry point, family, thunk(M)) for every D <= 8 entry point whose block can exceed 227 KB, at D = 8, S = 512:
    thunk(M) calls it with M inducing points on the given pointers and returns its code"""
    D, S, Tg = 8, 512, 3
    p = fake
    return [
        ("gpode_vf_fwd", "fwd", lambda M: lib.gpode_vf_fwd(p, D, M, S, p, p, 4, None)),
        ("gpode_rk4_fwd", "fwd", lambda M: lib.gpode_rk4_fwd(p, D, M, S, p, p, Tg, 4, p, p, None)),
        ("gpode_vf_bwd", "bwd_warp", lambda M: lib.gpode_vf_bwd(p, D, M, S, p, p, p, p, p, 4, None)),
        ("gpode_rk4_bwd", "bwd_warp", lambda M: lib.gpode_rk4_bwd(p, D, M, S, p, Tg, 4, p, p, p, p, p, p, None)),
        ("gpode_dopri5_fwd", "dopri5_fwd",
         lambda M: lib.gpode_dopri5_fwd(p, D, M, S, p, p, Tg, 100, 1e-6, 1e-6, p, p, p, None, 0, None)),
        ("gpode_dopri5_fwd per draw", "dopri5_fwd",
         lambda M: lib.gpode_dopri5_fwd(p, D, M, S, p, p, Tg, 4, 1e-6, 1e-6, p, p, p, None, 0, None)),
        ("gpode_dopri5_bwd", "bwd_warp",
         lambda M: lib.gpode_dopri5_bwd(p, D, M, S, p, Tg, 4, p, p, 8, 2, p, p, p, None)),
        ("gpode_vf_fwd_sets", "fwd", lambda M: lib.gpode_vf_fwd_sets(p, D, M, S, 5, 3, p, p, None)),
        ("gpode_rk4_fwd_sets", "fwd", lambda M: lib.gpode_rk4_fwd_sets(p, D, M, S, 5, 3, p, p, Tg, p, None)),
        ("gpode_dopri5_fwd_sets", "dopri5_fwd",
         lambda M: lib.gpode_dopri5_fwd_sets(p, D, M, S, 5, 3, p, p, Tg, 1e-6, 1e-6, p, p, p, None)),
    ]


def test_oversized_blocks_are_refused_before_any_cuda_call():
    """At D = 8, S = 512 and M = M*(family) + 1 every entry point returns "does not fit" without touching its
    pointers (never dereferenced here) and without a CUDA call: a failed cudaFuncSetAttribute would leave its error
    pending for the next, unrelated launch check on the thread"""
    from gaussian_process_odes_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(16)
    for name, family, call in oversized_calls(lib, fake):
        M = max_inducing(family, 8, 512) + 1
        rc = call(M)
        err = lib.gpode_last_error().decode()
        assert rc != 0 and "does not fit" in err, (name, M, rc, err)
