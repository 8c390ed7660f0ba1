"""CPU: host-side contract of the blocked whitening entry points (workspace sizes, argument errors before any CUDA
call)."""
import ctypes


def test_blocked_workspace_sizes_and_limits():
    from gaussian_process_odes_b200 import _lib
    lib = _lib.load()
    # forward: the [D][M][n_sets] right-hand sides; backward (n_sets = 0): rb | pb | Kbar | grad_Z per output | rows
    assert lib.gpode_whiten_blocked_work_doubles(5, 300, 1) == 5 * 300
    assert lib.gpode_whiten_blocked_work_doubles(5, 300, 64) == 5 * 300 * 64
    assert lib.gpode_whiten_blocked_work_doubles(8, 1024, 0) == 8 * 1024 * (1024 + 8 + 2) + 8 * 16 * 9
    assert lib.gpode_whiten_blocked_work_doubles(2, 2048, 0) == 2 * 2048 * (2048 + 2 + 2) + 2 * 32 * 3
    for D, M, n in ((9, 300, 1), (0, 300, 1), (2, 2049, 1), (2, 0, 1), (2, 300, -1), (2, 300, 65536)):
        assert lib.gpode_whiten_blocked_work_doubles(D, M, n) == -1, (D, M, n)


def test_blocked_entry_points_reject_m_above_the_limit():
    from gaussian_process_odes_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(16)   # never dereferenced: the arguments are checked first
    c = _lib.GpodeCache()
    c.D, c.M, c.S = 3, 2049, 32
    c.omega = c.phase = c.w = c.Z = c.ell = c.var = fake.value
    rc = lib.gpode_whiten_fwd_blocked(ctypes.byref(c), fake, 1e-5, fake, fake, fake, fake, None)
    assert rc < 0 and b"2048" in lib.gpode_last_error() and b"GPODE_MAX_M_BLOCKED" in lib.gpode_last_error()
    rc = lib.gpode_whiten_fwd_sets_blocked(ctypes.byref(c), fake, 1e-5, 4, fake, fake, fake, fake, None)
    assert rc < 0 and b"GPODE_MAX_M_BLOCKED" in lib.gpode_last_error()
    rc = lib.gpode_whiten_bwd_blocked(ctypes.byref(c), fake, fake, fake, fake, fake, fake, fake, fake, fake, None)
    assert rc < 0 and b"GPODE_MAX_M_BLOCKED" in lib.gpode_last_error()
    c.M = 300
    rc = lib.gpode_whiten_fwd_blocked(ctypes.byref(c), fake, 1e-5, fake, fake, fake, None, None)
    assert rc < 0 and b"NULL" in lib.gpode_last_error()
    # the tile kernels keep their limit
    c.M = 161
    rc = lib.gpode_whiten_fwd(ctypes.byref(c), fake, 1e-5, fake, fake, fake, None)
    assert rc < 0 and b"1..160" in lib.gpode_last_error()


def test_blocked_launch_counts():
    from gaussian_process_odes_b200 import _lib
    # P = ceil(M / 64) panels: Cholesky and every solve 2 P - 1 launches
    assert _lib.whiten_blocked_launches(161) == 4 + 3 * 5
    assert _lib.whiten_blocked_launches(2048, bwd=True) == 5 + 4 * 63
