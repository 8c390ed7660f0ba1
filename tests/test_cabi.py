"""CPU: the C-ABI shared library loads and exports every symbol include/gpode_b200.h declares (no compute calls)."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "gpode_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gpode_[a-z0-9_]+)\s*\(", src)))


def test_library_builds_loads_and_exports_header_symbols():
    from gaussian_process_odes_b200 import _lib, build
    path = build.build()
    assert os.path.exists(path)
    lib = ctypes.CDLL(path)
    names = _declared()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), "libgpode_b200.so does not export %s" % n
    # the ctypes binding covers exactly the header
    assert sorted(_lib.SIGNATURES) == names
    assert _lib.load().gpode_abi_version() == 2


def test_pure_host_entry_points():
    from gaussian_process_odes_b200 import _lib
    lib = _lib.load()
    # layout arithmetic only: rff D*roundup32(S/2)*roundup4(2D+4) + kern M*roundup4(D+2*ceil(D/2)) + w D*roundup4(2*ceil(D/2))
    # + f16 tensor-core operand blocks D*roundup2(ceil(S/8))*152 (D <= 5)
    assert lib.gpode_packed_floats(2, 16, 256) == 2 * 128 * 8 + 16 * 4 + 2 * 4 + 2 * 32 * 152
    assert lib.gpode_packed_floats(5, 100, 256) == 5 * 128 * 16 + 100 * 12 + 5 * 8 + 5 * 32 * 152
    assert lib.gpode_packed_floats(3, 24, 64) == 3 * 32 * 12 + 24 * 8 + 3 * 4 + 3 * 8 * 152
    assert lib.gpode_packed_floats(8, 10, 40) == 8 * 32 * 20 + 10 * 16 + 8 * 8
    assert lib.gpode_packed_floats(0, 1, 1) == -1
    # header | 4096 adjoint-CTA rows of A[D,D] | V[D] | 1024 param-grad-CTA rows of M x {T[k], W[j,k]}
    assert lib.gpode_acc_header_floats() == 4
    assert lib.gpode_acc_floats(5, 100) == 4 + 4096 * (25 + 5) + 1024 * 100 * (5 + 25)
    assert lib.gpode_side_work_doubles() == 2048 * 129
    assert lib.gpode_vrow_floats(5, 1000) == 10000
    assert lib.gpode_dopri5_work_floats(2, 10) >= 5 * 20 + 8
    # argument errors are reported through the return code + gpode_last_error, before any CUDA call
    rc = lib.gpode_vf_fwd(None, 2, 16, 256, None, None, 4, None)
    assert rc < 0 and b"NULL" in lib.gpode_last_error()
    rc = lib.gpode_rk4_fwd(ctypes.c_void_p(16), 9, 16, 256, None, None, 2, 4, None, None, None)
    assert rc < 0 and b"dimension" in lib.gpode_last_error()
    # the kernel-selection options are bwd_mma and fwd_mma; any other name is rejected
    assert lib.gpode_set_option(b"use_mma", 1) == -1 and b"unknown option" in lib.gpode_last_error()
    assert lib.gpode_get_option(b"bwd_mma") in (0, 1) and lib.gpode_get_option(b"fwd_mma") in (0, 1)


def test_kernels_have_no_register_spills_on_the_config_shapes():
    """ptxas -v of the last build: the D=2 and D=5 integrator kernels (the BASELINE configs) stay in registers
    (a few L1-resident spill bytes in the 250-register adjoint kernels are tolerated, nothing more)."""
    from gaussian_process_odes_b200 import build
    build.build()
    rep = build.ptxas_report()
    if not rep:
        import pytest
        pytest.skip("no ptxas logs (library was prebuilt elsewhere)")
    for unit, name, regs, spill in rep:
        if unit in ("integrate_d2", "integrate_d5", "dopri5_d2", "dopri5_d5", "param_grad"):
            assert spill <= 256, (unit, name, regs, spill)
            assert regs <= 255
