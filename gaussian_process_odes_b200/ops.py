"""torch.autograd bindings of the CUDA hot path (one ``Function`` per C-ABI op pair).

Tensor conventions follow the reference's cache attributes (``DSVGP_Layer.build_cache``, reference
``src/core/dsvgp.py:92-122``): ``omega (D,S,D)``, ``phase (1,S,D)`` or ``(S,D)``, ``w (S,D)``, ``Z (M,D)``,
``nu (D,M,1)`` or ``(D,M)``, ``ell (D,D)``, ``var (D,)``. Gradients flow to ``x / x0``, ``Z``, ``ell``, ``var``, ``nu``
(and ``u`` for the whitening); ``omega`` is treated as ``eps/ell`` -- its gradient arrives folded into ``ell``
(reference ``src/core/kernels.py:110-112``), ``w`` and ``phase`` carry no gradient in the reference either.
"""
import ctypes

import torch

from . import _lib
from ._lib import GpodeCache, GpodeShoot, check, f32, ptr, stream_ptr


def _cache_struct(D, M, S, omega, phase, w, Z, nu, ell, var):
    c = GpodeCache()
    c.D, c.M, c.S = D, M, S
    c.omega, c.phase, c.w = ptr(omega).value, ptr(phase).value, ptr(w).value
    c.Z, c.nu = ptr(Z).value, (ptr(nu).value if nu is not None else None)
    c.ell, c.var = ptr(ell).value, ptr(var).value
    return c


class PackedCache:
    """One sampled GP function repacked for the integrator kernels (``gpode_pack_cache``)."""

    def __init__(self, Z, ell, var, nu, omega, phase, w):
        lib = _lib.load()
        self.Z, self.ell, self.var = f32(Z, "Z"), f32(ell, "ell"), f32(var, "var")
        self.omega, self.w = f32(omega, "omega"), f32(w, "w")
        self.M, self.D = self.Z.shape
        self.S = self.w.shape[0]
        self.phase = f32(phase, "phase").reshape(self.S, self.D)
        self.nu = f32(nu, "nu").reshape(self.D, self.M)
        if tuple(self.omega.shape) != (self.D, self.S, self.D) or tuple(self.ell.shape) != (self.D, self.D) \
                or tuple(self.var.shape) != (self.D,) or tuple(self.w.shape) != (self.S, self.D):
            raise _lib.GpodeError("inconsistent cache shapes: omega %s ell %s var %s w %s Z %s" % (
                tuple(self.omega.shape), tuple(self.ell.shape), tuple(self.var.shape), tuple(self.w.shape),
                tuple(self.Z.shape)))
        n = lib.gpode_packed_floats(self.D, self.M, self.S)
        self.packed = torch.empty(n, dtype=torch.float32, device=self.Z.device)
        self.struct = _cache_struct(self.D, self.M, self.S, self.omega, self.phase, self.w, self.Z, self.nu,
                                    self.ell, self.var)
        _lib.call("gpode_pack_cache", ctypes.byref(self.struct), ptr(self.packed), stream_ptr())

    def new_acc(self):
        """Accumulator block of ONE backward pass: per-CTA partial-sum rows (added in a fixed order by
        ``gpode_grads_finalize``: bitwise reproducible); only the 4-word header has to be zero."""
        lib = _lib.load()
        acc = torch.empty(lib.gpode_acc_floats(self.D, self.M), dtype=torch.float32, device=self.Z.device)
        acc[:lib.gpode_acc_header_floats()].zero_()
        return acc

    def finalize(self, acc):
        """acc -> (grad_Z, grad_ell, grad_var, grad_nu)"""
        dev = self.Z.device
        g_ell = torch.empty(self.D, self.D, dtype=torch.float32, device=dev)
        g_var = torch.empty(self.D, dtype=torch.float32, device=dev)
        g_Z = torch.empty(self.M, self.D, dtype=torch.float32, device=dev)
        g_nu = torch.empty(self.D, self.M, dtype=torch.float32, device=dev)
        _lib.call("gpode_grads_finalize", ctypes.byref(self.struct), ptr(acc), ptr(g_ell), ptr(g_var), ptr(g_Z),
                                               ptr(g_nu), stream_ptr())
        return g_Z, g_ell, g_var, g_nu


class _VectorField(torch.autograd.Function):
    """f = DSVGP_Layer.forward(t, x) (reference src/core/dsvgp.py:172-197) via gpode_vf_fwd / gpode_vf_bwd."""

    @staticmethod
    def forward(ctx, x, Z, ell, var, nu, omega, phase, w):
        pc = PackedCache(Z, ell, var, nu, omega, phase, w)
        xc = f32(x, "x")
        if xc.ndim != 2 or xc.shape[1] != pc.D:
            raise _lib.GpodeError("x must be (B,%d), got %s" % (pc.D, tuple(xc.shape)))
        f = torch.empty_like(xc)
        _lib.call("gpode_vf_fwd", ptr(pc.packed), pc.D, pc.M, pc.S, ptr(xc), ptr(f), xc.shape[0], stream_ptr())
        ctx.pc, ctx.nu_shape = pc, nu.shape
        ctx.save_for_backward(xc, f)
        return f

    @staticmethod
    def backward(ctx, gf):
        pc = ctx.pc
        xc, f = ctx.saved_tensors
        gf = f32(gf, "grad_f")
        gx = torch.empty_like(xc)
        acc = pc.new_acc()
        _lib.call("gpode_vf_bwd", ptr(pc.packed), pc.D, pc.M, pc.S, ptr(xc), ptr(f), ptr(gf), ptr(gx), ptr(acc),
                                       xc.shape[0], stream_ptr())
        _lib.call("gpode_param_grad", ptr(pc.packed), pc.D, pc.M, pc.S, ptr(xc), ptr(gf), xc.shape[0], ptr(acc),
                  stream_ptr())
        g_Z, g_ell, g_var, g_nu = pc.finalize(acc)
        return gx, g_Z, g_ell, g_var, g_nu.reshape(ctx.nu_shape), None, None, None


class _RK4(torch.autograd.Function):
    """xs = odeint(f, x0, t, method='rk4') (torchdiffeq 0.2.0 3/8 rule) via gpode_rk4_fwd / gpode_rk4_bwd."""

    @staticmethod
    def forward(ctx, x0, t, Z, ell, var, nu, omega, phase, w, want_grad):
        pc = PackedCache(Z, ell, var, nu, omega, phase, w)
        xc, tc = f32(x0, "x0"), f32(t, "t")
        if xc.ndim != 2 or xc.shape[1] != pc.D:
            raise _lib.GpodeError("x0 must be (B,%d), got %s" % (pc.D, tuple(xc.shape)))
        B, Tg = xc.shape[0], tc.shape[0]
        # ctx.needs_input_grad is True under torch.no_grad() too; the caller tells whether a graph is being recorded
        need_grad = want_grad and any(ctx.needs_input_grad)
        xs = torch.empty(Tg, B, pc.D, dtype=torch.float32, device=xc.device)
        kst = torch.empty(max(Tg - 1, 0), 4, B, pc.D, dtype=torch.float32, device=xc.device) if need_grad else None
        _lib.call("gpode_rk4_fwd", ptr(pc.packed), pc.D, pc.M, pc.S, ptr(xc), ptr(tc), Tg, B, ptr(xs),
                                        ptr(kst), stream_ptr())
        ctx.pc, ctx.nu_shape = pc, nu.shape
        if need_grad:
            ctx.save_for_backward(tc, xs, kst)
        return xs

    @staticmethod
    def backward(ctx, gxs):
        pc = ctx.pc
        tc, xs, kst = ctx.saved_tensors
        lib = _lib.load()
        Tg, B, D = xs.shape
        gxs = f32(gxs, "grad_xs")
        gx0 = torch.empty(B, D, dtype=torch.float32, device=xs.device)
        acc = pc.new_acc()
        n_vr = max(Tg - 1, 0) * 4 * B
        vrows = torch.empty(lib.gpode_vrow_floats(D, n_vr), dtype=torch.float32, device=xs.device)
        _lib.call("gpode_rk4_bwd", ptr(pc.packed), pc.D, pc.M, pc.S, ptr(tc), Tg, B, ptr(xs), ptr(kst), ptr(gxs),
                                ptr(gx0), ptr(vrows), ptr(acc), stream_ptr())
        if n_vr:
            _lib.call("gpode_param_grad", ptr(pc.packed), pc.D, pc.M, pc.S, ptr(vrows), ptr(vrows[n_vr * D:]), n_vr,
                      ptr(acc), stream_ptr())
        g_Z, g_ell, g_var, g_nu = pc.finalize(acc)
        return gx0, None, g_Z, g_ell, g_var, g_nu.reshape(ctx.nu_shape), None, None, None, None


MAX_M = 160           # GPODE_MAX_M: whitening in one CTA's shared memory (gpode_whiten_fwd / _bwd)
MAX_M_BLOCKED = 2048  # GPODE_MAX_M_BLOCKED: blocked float64 whitening above MAX_M (gpode_whiten_*_blocked)


def _whiten_work(D, M, n_sets, device):
    """float64 workspace of the blocked whitening (n_sets = 0: the backward's); a caching-allocator tensor, so the
    call stays capturable in a CUDA graph. Raises GpodeError naming the limit when M > MAX_M_BLOCKED."""
    n = _lib.load().gpode_whiten_blocked_work_doubles(D, M, n_sets)
    if n < 0:
        raise _lib.GpodeError("blocked whitening needs D <= 8 and 1 <= M <= %d (GPODE_MAX_M_BLOCKED), got D=%d, M=%d"
                              % (MAX_M_BLOCKED, D, M))
    return torch.empty(n, dtype=torch.float64, device=device)


class _Whiten(torch.autograd.Function):
    """nu = Kzz^-1-whitening of build_cache (reference src/core/dsvgp.py:110-122) via gpode_whiten_fwd / _bwd, or
    gpode_whiten_fwd_blocked / _bwd_blocked above MAX_M inducing points."""

    @staticmethod
    def forward(ctx, Z, ell, var, u, omega, phase, w, jitter):
        lib = _lib.load()
        Zc, ec, vc, uc = f32(Z, "Z"), f32(ell, "ell"), f32(var, "var"), f32(u, "u")
        oc, wc = f32(omega, "omega"), f32(w, "w")
        M, D = Zc.shape
        S = wc.shape[0]
        pc_ = f32(phase, "phase").reshape(S, D)
        st = _cache_struct(D, M, S, oc, pc_, wc, Zc, None, ec, vc)
        nu = torch.empty(D, M, dtype=torch.float32, device=Zc.device)
        L = torch.empty(D, M, M, dtype=torch.float64, device=Zc.device)
        sp = torch.empty(D, 2, M, dtype=torch.float64, device=Zc.device)
        if M > MAX_M:
            work = _whiten_work(D, M, 1, Zc.device)
            _lib.call("gpode_whiten_fwd_blocked", ctypes.byref(st), ptr(uc), float(jitter), ptr(nu), ptr(L), ptr(sp),
                      ptr(work), stream_ptr(), launches=_lib.whiten_blocked_launches(M))
        else:
            _lib.call("gpode_whiten_fwd", ctypes.byref(st), ptr(uc), float(jitter), ptr(nu), ptr(L), ptr(sp),
                      stream_ptr())
        ctx.keep = (st, Zc, ec, vc, uc, oc, pc_, wc)
        ctx.save_for_backward(L, sp)
        return nu

    @staticmethod
    def backward(ctx, gnu):
        lib = _lib.load()
        st, Zc, ec, vc, uc, oc, pc_, wc = ctx.keep
        L, sp = ctx.saved_tensors
        M, D = Zc.shape
        gnu = f32(gnu, "grad_nu").reshape(D, M)
        g_u = torch.empty(M, D, dtype=torch.float32, device=Zc.device)
        g_Z = torch.empty(M, D, dtype=torch.float32, device=Zc.device)
        g_ell = torch.empty(D, D, dtype=torch.float32, device=Zc.device)
        g_var = torch.empty(D, dtype=torch.float32, device=Zc.device)
        if M > MAX_M:
            work = _whiten_work(D, M, 0, Zc.device)
            _lib.call("gpode_whiten_bwd_blocked", ctypes.byref(st), ptr(uc), ptr(L), ptr(sp), ptr(gnu), ptr(g_u),
                      ptr(g_Z), ptr(g_ell), ptr(g_var), ptr(work), stream_ptr(),
                      launches=_lib.whiten_blocked_launches(M, bwd=True))
        else:
            _lib.call("gpode_whiten_bwd", ctypes.byref(st), ptr(uc), ptr(L), ptr(sp), ptr(gnu), ptr(g_u), ptr(g_Z),
                      ptr(g_ell), ptr(g_var), stream_ptr())
        return g_Z, g_ell, g_var, g_u, None, None, None, None


class _WhitenedKL(torch.autograd.Function):
    """DSVGP_Layer.kl (reference src/core/dsvgp.py:199-230) on the PACKED lower-triangular optvar."""

    @staticmethod
    def forward(ctx, Um, Ls_packed):
        Uc, Lc = f32(Um, "Um"), f32(Ls_packed, "Us_sqrt optvar")
        M, D = Uc.shape
        if tuple(Lc.shape) != (D, M * (M + 1) // 2):
            raise _lib.GpodeError("Us_sqrt optvar must be (%d,%d), got %s" % (D, M * (M + 1) // 2, tuple(Lc.shape)))
        out = torch.empty((), dtype=torch.float32, device=Uc.device)
        _lib.call("gpode_kl_fwd", ptr(Uc), ptr(Lc), D, M, ptr(out), stream_ptr())
        ctx.save_for_backward(Uc, Lc)
        return out

    @staticmethod
    def backward(ctx, g):
        Uc, Lc = ctx.saved_tensors
        M, D = Uc.shape
        gU, gL = torch.empty_like(Uc), torch.empty_like(Lc)
        _lib.call("gpode_kl_bwd", ptr(Uc), ptr(Lc), D, M, ptr(f32(g, "grad_kl")), ptr(gU), ptr(gL),
                                       stream_ptr())
        return gU, gL


class _InducingSample(torch.autograd.Function):
    """u = Um + Us_sqrt eps from the PACKED factor (gpode_inducing_sample_fwd/_bwd; reference dsvgp.py:78-90)."""

    @staticmethod
    def forward(ctx, Um, Ls_packed, eps):
        Uc, Lc, ec = f32(Um, "Um"), f32(Ls_packed, "Us_sqrt optvar"), f32(eps, "epsilon")
        M, D = Uc.shape
        if tuple(Lc.shape) != (D, M * (M + 1) // 2) or tuple(ec.shape) != (M, D):
            raise _lib.GpodeError("inducing sample: Us_sqrt optvar %s / epsilon %s do not match Um %s" % (
                tuple(Lc.shape), tuple(ec.shape), tuple(Uc.shape)))
        u = torch.empty_like(Uc)
        _lib.call("gpode_inducing_sample_fwd", ptr(Uc), ptr(Lc), ptr(ec), D, M, ptr(u), stream_ptr())
        ctx.save_for_backward(ec)
        ctx.dims = (D, M, Lc.shape)
        return u

    @staticmethod
    def backward(ctx, g):
        (ec,) = ctx.saved_tensors
        D, M, lshape = ctx.dims
        gc = f32(g, "grad_u")
        gL = torch.empty(lshape, dtype=torch.float32, device=ec.device)
        _lib.call("gpode_inducing_sample_bwd", ptr(ec), ptr(gc), D, M, ptr(gL), stream_ptr())
        return gc, gL, None


def inducing_sample(Um, Ls_packed, eps):
    """``Um (M,D) + einsum('dnm,md->nd', tril(Ls), eps)`` with ``Ls`` packed ``(D, M(M+1)/2)``."""
    return _InducingSample.apply(Um, Ls_packed, eps)


class _StateSample(torch.autograd.Function):
    """mean + chol(L L^T + jitter I) eps for a batch of packed lower-triangular factors (gpode_state_fwd/_bwd)."""

    @staticmethod
    def forward(ctx, mean, L_packed, eps, jitter):
        mc, lc, ec = f32(mean, "mean"), f32(L_packed, "L_packed"), f32(eps, "eps")
        D = mc.shape[-1]
        R = mc.numel() // D
        S = ec.numel() // (R * D) if R else 0
        out = torch.empty_like(ec)
        _lib.call("gpode_state_fwd", ptr(mc), ptr(lc), ptr(ec), S, R, D, float(jitter), ptr(out), ptr(None),
                  stream_ptr())
        ctx.save_for_backward(lc, ec)
        ctx.dims = (S, R, D, float(jitter), mean.shape, L_packed.shape)
        return out

    @staticmethod
    def backward(ctx, g):
        lc, ec = ctx.saved_tensors
        S, R, D, jitter, mshape, lshape = ctx.dims
        gm = torch.empty(mshape, dtype=torch.float32, device=lc.device)
        gl = torch.empty(lshape, dtype=torch.float32, device=lc.device)
        _lib.call("gpode_state_bwd", ptr(lc), ptr(ec), S, R, D, jitter, ptr(f32(g, "grad_samples")), ptr(None),
                  ptr(gm), ptr(gl), stream_ptr())
        return gm, gl, None, None


class _StateEntropy(torch.autograd.Function):
    """Entropy of N(., L L^T + jitter I) per matrix (gpode_state_fwd/_bwd with only the entropy output)."""

    @staticmethod
    def forward(ctx, L_packed, D, jitter):
        lc = f32(L_packed, "L_packed")
        R = lc.numel() // (D * (D + 1) // 2)
        out = torch.empty(L_packed.shape[:-1], dtype=torch.float32, device=lc.device)
        _lib.call("gpode_state_fwd", ptr(None), ptr(lc), ptr(None), 0, R, D, float(jitter), ptr(None), ptr(out),
                  stream_ptr())
        ctx.save_for_backward(lc)
        ctx.dims = (R, D, float(jitter), L_packed.shape)
        return out

    @staticmethod
    def backward(ctx, g):
        (lc,) = ctx.saved_tensors
        R, D, jitter, lshape = ctx.dims
        gl = torch.empty(lshape, dtype=torch.float32, device=lc.device)
        _lib.call("gpode_state_bwd", ptr(lc), ptr(None), 0, R, D, jitter, ptr(None), ptr(f32(g, "grad_entropy")),
                  ptr(None), ptr(gl), stream_ptr())
        return gl, None, None


def _side_work(device):
    """float64 scratch of the side-term sums (per-CTA partial rows, summed in a fixed order)."""
    return torch.empty(_lib.load().gpode_side_work_doubles(), dtype=torch.float64, device=device)


class _LoglikMean(torch.autograd.Function):
    """mean over all elements of log N(ys | pred W + b, var), value and gradients in one kernel (gpode_loglik_sum)."""

    @staticmethod
    def forward(ctx, pred, ys, W, bias, var):
        pc, yc, wc, vc = f32(pred, "pred"), f32(ys, "ys"), f32(W, "W"), f32(var, "var")
        bc = f32(bias, "bias") if bias is not None else None
        D, Dobs = wc.shape
        R = yc.numel() // Dobs
        S = pc.numel() // (R * D) if R else 1
        need_p, need_v = ctx.needs_input_grad[0], ctx.needs_input_grad[4]
        total = torch.empty((), dtype=torch.float64, device=pc.device)
        gp = torch.empty_like(pc) if need_p else None
        gv = torch.empty_like(vc) if need_v else None
        if vc.numel() != Dobs or (bc is not None and bc.numel() != Dobs):
            raise _lib.GpodeError("loglik_mean: var (and bias) must hold one value per observed dimension (%d), got %d"
                                  % (Dobs, vc.numel()))
        _lib.call("gpode_loglik_sum", ptr(pc), ptr(yc), ptr(wc), ptr(bc), ptr(vc), S, R, D, Dobs, ptr(total), ptr(gp),
                  ptr(gv), ptr(_side_work(pc.device)), stream_ptr())
        count = float(S * R * Dobs)
        ctx.count = count
        ctx.save_for_backward(*(t for t in (gp, gv) if t is not None))
        ctx.have = (need_p, need_v)
        return (total / count).to(torch.float32)

    @staticmethod
    def backward(ctx, g):
        saved = list(ctx.saved_tensors)
        need_p, need_v = ctx.have
        scale = g / ctx.count
        gp = saved.pop(0) * scale if need_p else None
        gv = saved.pop(0) * scale if need_v else None
        return gp, None, None, None, gv


class _ConstraintSum(torch.autograd.Function):
    """sum_{s,n,t<T-1,d} log p(ss[s,n,t+1,d] | pred[s,n,t,d], scale) in one kernel (gpode_constraint_sum)."""

    @staticmethod
    def forward(ctx, ss, pred, scale, laplace):
        sc, pc, kc = f32(ss, "ss"), f32(pred, "pred"), f32(scale, "scale")
        T, D = sc.shape[-2], sc.shape[-1]
        SN = sc.numel() // (T * D)
        need_s, need_p = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if ctx.needs_input_grad[2]:
            raise _lib.GpodeError("the fused constraint term treats the scale as a constant (requires_grad=False)")
        total = torch.empty((), dtype=torch.float64, device=sc.device)
        gs = torch.empty_like(sc) if need_s else None
        gp = torch.empty_like(pc) if need_p else None
        _lib.call("gpode_constraint_sum", ptr(sc), ptr(pc), ptr(kc), SN, T, D, int(bool(laplace)), ptr(total), ptr(gs),
                  ptr(gp), ptr(_side_work(sc.device)), stream_ptr())
        ctx.save_for_backward(*(t for t in (gs, gp) if t is not None))
        ctx.have = (need_s, need_p)
        return total.to(torch.float32)

    @staticmethod
    def backward(ctx, g):
        saved = list(ctx.saved_tensors)
        need_s, need_p = ctx.have
        gs = saved.pop(0) * g if need_s else None
        gp = saved.pop(0) * g if need_p else None
        return gs, gp, None, None


def constraint_sum(ss, pred, scale, laplace=False):
    """``ss``, ``pred``: (..., T, D). Sum over all leading axes, t < T-1 and D of log p(ss[t+1] | pred[t], scale)."""
    return _ConstraintSum.apply(ss, pred, scale, laplace)


def state_sample(mean, L_packed, eps, jitter=1e-5):
    """``eps (S, *batch, D)`` -> samples ``(S, *batch, D)`` of N(mean, L L^T + jitter I), L packed ``(*batch, P)``."""
    return _StateSample.apply(mean, L_packed, eps, jitter)


def state_entropy(L_packed, D, jitter=1e-5):
    return _StateEntropy.apply(L_packed, D, jitter)


def loglik_mean(pred, ys, W, bias, var):
    """pred ``(S?, ..., D)``, ys ``(..., D_obs)``: mean Gaussian log-density of ``ys`` under ``pred @ W + bias``."""
    return _LoglikMean.apply(pred, ys, W, bias, var)


def _shoot_descriptor(ss, t2, D, ys, W, bias, lik_var, cons_scale, flags, row_lo, row_hi):
    """Checked float32 views of the shooting-step inputs and their ``gpode_shoot_t`` -> (sh, tensors, row_lo, row_hi)"""
    sc, tc = f32(ss, "ss"), f32(t2, "ts[:2]")
    if sc.ndim != 4 or sc.shape[3] != D:
        raise _lib.GpodeError("ss must be (S_mc,N,T,%d), got %s" % (D, tuple(sc.shape)))
    if tc.numel() != 2:
        raise _lib.GpodeError("the fused shooting step integrates one interval: ts[:2], got %d points" % tc.numel())
    S_mc, N, T, _ = sc.shape
    yc, Wc, vc, kc = f32(ys, "ys"), f32(W, "W"), f32(lik_var, "likelihood variance"), f32(cons_scale, "scale")
    bc = f32(bias, "bias") if bias is not None else None
    Dobs = Wc.shape[1]
    if tuple(yc.shape) != (N, T, Dobs) or Wc.shape[0] != D or vc.numel() != Dobs or kc.numel() != 1 \
            or (bc is not None and bc.numel() != Dobs):
        raise _lib.GpodeError("inconsistent shooting shapes: ss %s ys %s W %s var %s scale %s" % (
            tuple(sc.shape), tuple(yc.shape), tuple(Wc.shape), tuple(vc.shape), tuple(kc.shape)))
    n_total = S_mc * N * T
    row_lo, row_hi = int(row_lo), int(n_total if row_hi is None else row_hi)
    sh = GpodeShoot()
    sh.S_mc, sh.N, sh.T, sh.D_obs, sh.laplace = S_mc, N, T, Dobs, int(flags)   # bit 0 Laplace, bit 1 halo
    sh.ys, sh.W, sh.bias = ptr(yc).value, ptr(Wc).value, (ptr(bc).value if bc is not None else None)
    sh.lik_var, sh.cons_scale = ptr(vc).value, ptr(kc).value
    sh.row_lo, sh.row_hi = row_lo, row_hi
    return sh, (sc, tc, yc, Wc, bc, vc, kc), row_lo, row_hi


class _ShootStep(torch.autograd.Function):
    """The integrator launch of the multiple-shooting ELBO with its two end-point terms fused in (``gpode_shoot_fwd`` /
    ``gpode_shoot_bwd``; reference ``src/gpode_shooting/models.py:119-135``): -> (log-likelihood SUM, constraint SUM,
    end points or None) over the rows ``[row_lo, row_hi)`` of the ``(S_mc, N, T)`` segment batch."""

    @staticmethod
    def forward(ctx, ss, t2, Z, ell, var, nu, omega, phase, w, ys, W, bias, lik_var, cons_scale, laplace, row_lo,
                row_hi, want_grad, want_pred):
        lib = _lib.load()
        pc = PackedCache(Z, ell, var, nu, omega, phase, w)
        D = pc.D
        sh, keep, row_lo, row_hi = _shoot_descriptor(ss, t2, D, ys, W, bias, lik_var, cons_scale, laplace, row_lo,
                                                     row_hi)
        sc, tc = keep[0], keep[1]
        if ctx.needs_input_grad[13]:
            raise _lib.GpodeError("the fused shooting step treats the constraint scale as a constant")
        B, Dobs = row_hi - row_lo, sh.D_obs
        need_grad = want_grad and any(ctx.needs_input_grad)
        dev = sc.device
        kst = torch.empty(1, 4, B, D, dtype=torch.float32, device=dev) if need_grad else None
        seeds = torch.empty(2, B, D, dtype=torch.float32, device=dev) if need_grad else None
        pred = torch.empty(B, D, dtype=torch.float32, device=dev) if want_pred else None
        sums = torch.empty(2, dtype=torch.float64, device=dev)
        gvar = torch.empty(Dobs, dtype=torch.float32, device=dev) if need_grad else None
        work = torch.empty(lib.gpode_shoot_work_doubles(), dtype=torch.float64, device=dev)
        _lib.call("gpode_shoot_fwd", ptr(pc.packed), pc.D, pc.M, pc.S, ctypes.byref(sh), ptr(sc), ptr(tc), ptr(kst),
                  ptr(pred), ptr(seeds), ptr(sums), ptr(gvar), ptr(work), stream_ptr())
        ctx.pc, ctx.nu_shape, ctx.sh, ctx.keep = pc, nu.shape, sh, keep
        ctx.full = (row_lo == 0 and row_hi == sc.shape[0] * sc.shape[1] * sc.shape[2])
        ctx.var_shape = lik_var.shape
        if need_grad:
            ctx.save_for_backward(sc, tc, kst, seeds, gvar)
        out32 = sums.to(torch.float32)
        if pred is not None:
            ctx.mark_non_differentiable(pred)
        return out32[0], out32[1], pred

    @staticmethod
    def backward(ctx, g_ll, g_cons, _g_pred):
        pc, sh = ctx.pc, ctx.sh
        sc, tc, kst, seeds, gvar = ctx.saved_tensors
        lib = _lib.load()
        B, D = seeds.shape[1], seeds.shape[2]
        dev = sc.device
        zero = lambda: torch.zeros((), dtype=torch.float32, device=dev)
        g_ll = f32(g_ll, "grad") if g_ll is not None else zero()
        g_cons = f32(g_cons, "grad") if g_cons is not None else zero()
        g_ss = torch.empty_like(sc) if ctx.full else torch.zeros_like(sc)
        acc = pc.new_acc()
        # 0 virtual rows: the tensor-core adjoint sums the inducing-point gradients itself (no gpode_param_grad)
        n_vr = lib.gpode_shoot_bwd_vrows(pc.D, pc.M, pc.S, B)
        vrows = torch.empty(lib.gpode_vrow_floats(D, n_vr), dtype=torch.float32, device=dev) if n_vr else None
        _lib.call("gpode_shoot_bwd", ptr(pc.packed), pc.D, pc.M, pc.S, ctypes.byref(sh), ptr(sc), ptr(tc), ptr(kst),
                  ptr(seeds), ptr(g_ll), ptr(g_cons), ptr(g_ss), ptr(vrows), ptr(acc), stream_ptr())
        if n_vr:
            _lib.call("gpode_param_grad", ptr(pc.packed), pc.D, pc.M, pc.S, ptr(vrows), ptr(vrows[n_vr * D:]), n_vr,
                      ptr(acc), stream_ptr())
        g_Z, g_ell, g_var, g_nu = pc.finalize(acc)
        g_lik = (gvar * g_ll).reshape(ctx.var_shape)
        return (g_ss, None, g_Z, g_ell, g_var, g_nu.reshape(ctx.nu_shape), None, None, None, None, None, None, g_lik,
                None, None, None, None, None, None)


def shooting_step(ss, t2, Z, ell, var, nu, omega, phase, w, ys, W, bias, lik_var, cons_scale, laplace=False,
                  rows=None, want_pred=False, halo=False):
    """One RK4 interval for every row of the sampled-state batch ``ss (S_mc,N,T,D)`` with the observation
    log-likelihood and the shooting constraint evaluated inside the integrator kernel. Returns
    ``(loglik_sum, constraint_sum, pred)``: sums over the rows ``rows = (lo, hi)`` of the flattened batch (all rows by
    default) -- ``loglik_sum`` over ``(row, d)`` of ``log N(ys[n,t,d] | (pred W + bias)_d, lik_var_d)`` and
    ``constraint_sum`` over ``(row with t < T-1, d)`` of ``log p(ss[s,n,t+1,d] | pred_d, cons_scale)`` -- and the end
    points ``pred (hi-lo, D)`` when ``want_pred`` (no gradient flows through them). Differentiable in ``ss``, ``Z``,
    ``ell``, ``var``, ``nu`` and ``lik_var``."""
    lo, hi = (0, None) if rows is None else rows
    # ``halo``: the last time index of every sequence of this (time-sharded) batch is the next rank's first state --
    # the constraint's neighbour only, no observation term (flag bit 1 of gpode_shoot_t.laplace)
    flags = int(bool(laplace)) | (2 if halo else 0)
    D = Z.shape[1]
    if D > MAX_D_REGISTER:
        if D > MAX_D_LARGE:
            raise _lib.GpodeError("the shooting step covers state dimensions up to %d, got D=%d" % (MAX_D_LARGE, D))
        fn = _ShootStepLarge
    else:
        fn = _ShootStep
    return fn.apply(ss, t2, Z, ell, var, nu, omega, phase, w, ys, W, bias, lik_var, cons_scale, flags, lo, hi,
                    torch.is_grad_enabled(), want_pred)


class _ShootStepLarge(torch.autograd.Function):
    """``_ShootStep`` for 8 < D <= 64 (``gpode_shoot_fwd_large`` / ``gpode_shoot_bwd_large``): one RK4 interval on the
    tcgen05 vector field, the two end-point terms and their seeds in one epilogue kernel, the large-D adjoint seeded
    on the device. Same arguments and results."""

    @staticmethod
    def forward(ctx, ss, t2, Z, ell, var, nu, omega, phase, w, ys, W, bias, lik_var, cons_scale, laplace, row_lo,
                row_hi, want_grad, want_pred):
        lib = _lib.load()
        field = LargeField(Z, ell, var, nu, omega, phase, w)
        D = field.D
        sh, keep, row_lo, row_hi = _shoot_descriptor(ss, t2, D, ys, W, bias, lik_var, cons_scale, laplace, row_lo,
                                                     row_hi)
        sc, tc = keep[0], keep[1]
        if ctx.needs_input_grad[13]:
            raise _lib.GpodeError("the fused shooting step treats the constraint scale as a constant")
        B, Dobs = row_hi - row_lo, sh.D_obs
        need_grad = want_grad and any(ctx.needs_input_grad)
        dev = sc.device
        kst = torch.empty(1, 4, B, D, dtype=torch.float32, device=dev) if need_grad else None
        seeds = torch.empty(2, B, D, dtype=torch.float32, device=dev) if need_grad else None
        pred = torch.empty(B, D, dtype=torch.float32, device=dev) if want_pred else None
        sums = torch.empty(2, dtype=torch.float64, device=dev)
        gvar = torch.empty(Dobs, dtype=torch.float32, device=dev) if need_grad else None
        work = torch.empty(lib.gpode_shoot_large_work_doubles(D, B), dtype=torch.float64, device=dev)
        _lib.call("gpode_shoot_fwd_large", ptr(field.packed), ctypes.byref(field.struct), ctypes.byref(sh), ptr(sc),
                  ptr(tc), ptr(kst), ptr(pred), ptr(seeds), ptr(sums), ptr(gvar), ptr(work), stream_ptr())
        ctx.field, ctx.nu_shape, ctx.sh, ctx.keep = field, nu.shape, sh, keep
        ctx.full = (row_lo == 0 and row_hi == sc.shape[0] * sc.shape[1] * sc.shape[2])
        ctx.var_shape = lik_var.shape
        if need_grad:
            ctx.save_for_backward(sc, tc, kst, seeds, gvar)
        out32 = sums.to(torch.float32)
        if pred is not None:
            ctx.mark_non_differentiable(pred)
        return out32[0], out32[1], pred

    @staticmethod
    def backward(ctx, g_ll, g_cons, _g_pred):
        field, sh = ctx.field, ctx.sh
        sc, tc, kst, seeds, gvar = ctx.saved_tensors
        B = seeds.shape[1]
        dev = sc.device
        zero = lambda: torch.zeros((), dtype=torch.float32, device=dev)
        g_ll = f32(g_ll, "grad") if g_ll is not None else zero()
        g_cons = f32(g_cons, "grad") if g_cons is not None else zero()
        g_ss = torch.empty_like(sc) if ctx.full else torch.zeros_like(sc)
        acc = field.new_acc()
        work = torch.empty(_lib.load().gpode_shoot_large_work_doubles(field.D, B), dtype=torch.float64, device=dev)
        _lib.call("gpode_shoot_bwd_large", ptr(field.packed_bwd), ctypes.byref(field.struct), ctypes.byref(sh),
                  ptr(sc), ptr(tc), ptr(kst), ptr(seeds), ptr(g_ll), ptr(g_cons), ptr(g_ss), ptr(acc), ptr(work),
                  stream_ptr())
        g_Z, g_ell, g_var, g_nu = field.finalize(acc, B)
        g_lik = (gvar * g_ll).reshape(ctx.var_shape)
        return (g_ss, None, g_Z, g_ell, g_var, g_nu.reshape(ctx.nu_shape), None, None, None, None, None, None, g_lik,
                None, None, None, None, None, None)


MAX_D_REGISTER = 8    # GPODE_MAX_D: differentiable register-resident kernels
MAX_D_LARGE = 64      # GPODE_MAX_D_LARGE: tcgen05 forward + large-D VJP kernels (rk4 and dopri5 differentiable)


class LargeField:
    """One sampled GP function for 8 < D <= 64: the Fourier-feature term runs on the tcgen05 tensor cores
    (``gpode_rff_fwd_large`` over the pre-tiled 3xTF32 operand chunks of ``gpode_pack_cache_large``), the RBF term as
    well (``gpode_rbf_fwd_large``; tiled FP32 kernel ``gpode_vf_fwd_large_add_rbf`` when Z does not fit its shared-
    memory copy). Pack once, evaluate many times. The backward operand block (``gpode_pack_cache_large_bwd``) is packed
    on first use."""

    def __init__(self, Z, ell, var, nu, omega, phase, w):
        lib = _lib.load()
        Zc, ec, vc, oc, wc = f32(Z, "Z"), f32(ell, "ell"), f32(var, "var"), f32(omega, "omega"), f32(w, "w")
        self.M, self.D = Zc.shape
        self.S = wc.shape[0]
        pc_, nc = f32(phase, "phase").reshape(self.S, self.D), f32(nu, "nu").reshape(self.D, self.M)
        self.keep = (Zc, ec, vc, oc, wc, pc_, nc)
        self.struct = _cache_struct(self.D, self.M, self.S, oc, pc_, wc, Zc, nc, ec, vc)
        n = lib.gpode_packed_large_floats(self.D, self.M, self.S)
        if n < 0:
            raise _lib.GpodeError("large-D path needs %d < D <= %d, got %d" % (MAX_D_REGISTER, MAX_D_LARGE, self.D))
        self.packed = torch.empty(n, dtype=torch.float32, device=Zc.device)
        self.rbf_on_tensor_cores = True
        self._packed_bwd = None
        _lib.call("gpode_pack_cache_large", ctypes.byref(self.struct), ptr(self.packed), stream_ptr())

    @property
    def packed_bwd(self):
        if self._packed_bwd is None:
            n = _lib.load().gpode_packed_large_bwd_floats(self.D, self.M, self.S)
            self._packed_bwd = torch.empty(n, dtype=torch.float32, device=self.packed.device)
            _lib.call("gpode_pack_cache_large_bwd", ctypes.byref(self.struct), ptr(self._packed_bwd), stream_ptr())
        return self._packed_bwd

    def new_acc(self):
        n = _lib.load().gpode_acc_large_floats(self.D, self.M)
        return torch.zeros(n, dtype=torch.float32, device=self.packed.device)

    def finalize(self, acc, B):
        """acc -> (grad_Z, grad_ell, grad_var, grad_nu)"""
        dev = self.packed.device
        g_ell = torch.empty(self.D, self.D, dtype=torch.float32, device=dev)
        g_var = torch.empty(self.D, dtype=torch.float32, device=dev)
        g_Z = torch.empty(self.M, self.D, dtype=torch.float32, device=dev)
        g_nu = torch.empty(self.D, self.M, dtype=torch.float32, device=dev)
        _lib.call("gpode_grads_finalize_large", ctypes.byref(self.struct), ptr(acc), B, ptr(g_ell), ptr(g_var),
                  ptr(g_Z), ptr(g_nu), stream_ptr())
        return g_Z, g_ell, g_var, g_nu

    def __call__(self, x):
        xc = f32(x, "x")
        if xc.ndim != 2 or xc.shape[1] != self.D:
            raise _lib.GpodeError("x must be (B,%d), got %s" % (self.D, tuple(xc.shape)))
        B = xc.shape[0]
        f_rff = torch.empty_like(xc)
        _lib.call("gpode_rff_fwd_large", ptr(self.packed), self.D, self.S, ptr(xc), ptr(f_rff), B, stream_ptr())
        f = torch.empty_like(xc)
        if self.rbf_on_tensor_cores:
            try:
                _lib.call("gpode_rbf_fwd_large", ptr(self.packed), self.D, self.M, self.S, ptr(self.keep[0]), ptr(xc),
                          ptr(f_rff), ptr(f), B, stream_ptr())
                return f
            except _lib.GpodeError as e:
                if "too large for the shared-memory copy of Z" not in str(e):
                    raise
                self.rbf_on_tensor_cores = False  # many inducing points at large D: the FP32 tiled CUDA kernel instead
        _lib.call("gpode_vf_fwd_large_add_rbf", ctypes.byref(self.struct), ptr(xc), ptr(f_rff), ptr(f), B,
                  stream_ptr())
        return f


class _VectorFieldLarge(torch.autograd.Function):
    """f = DSVGP_Layer.forward(t, x) for 8 < D <= 64: tcgen05 forward, ``gpode_vf_bwd_large`` backward."""

    @staticmethod
    def forward(ctx, x, Z, ell, var, nu, omega, phase, w):
        field = LargeField(Z, ell, var, nu, omega, phase, w)
        xc = f32(x, "x")
        f = field(xc)
        ctx.field, ctx.nu_shape = field, nu.shape
        ctx.save_for_backward(xc, f)
        return f

    @staticmethod
    def backward(ctx, gf):
        field = ctx.field
        xc, f = ctx.saved_tensors
        gf = f32(gf, "grad_f")
        B = xc.shape[0]
        gx = torch.empty_like(xc)
        acc = field.new_acc()
        _lib.call("gpode_vf_bwd_large", ptr(field.packed_bwd), field.D, field.M, field.S, ptr(xc), ptr(f), ptr(gf),
                  ptr(gx), ptr(acc), B, stream_ptr())
        g_Z, g_ell, g_var, g_nu = field.finalize(acc, B)
        return gx, g_Z, g_ell, g_var, g_nu.reshape(ctx.nu_shape), None, None, None


class _RK4Large(torch.autograd.Function):
    """``odeint(f, x0, t, method='rk4')`` for 8 < D <= 64 as a stream-ordered sequence of launches
    (``gpode_rk4_fwd_large_dev`` / ``gpode_rk4_bwd_large``): no host loop, no host read of the grid."""

    @staticmethod
    def forward(ctx, x0, t, Z, ell, var, nu, omega, phase, w, want_grad):
        field = LargeField(Z, ell, var, nu, omega, phase, w)
        xc, tc = f32(x0, "x0"), f32(t, "t")
        if xc.ndim != 2 or xc.shape[1] != field.D:
            raise _lib.GpodeError("x0 must be (B,%d), got %s" % (field.D, tuple(xc.shape)))
        B, D, Tg = xc.shape[0], field.D, tc.shape[0]
        need_grad = want_grad and any(ctx.needs_input_grad)
        dev = xc.device
        xs = torch.empty(Tg, B, D, dtype=torch.float32, device=dev)
        kst = torch.empty(max(Tg - 1, 0), 4, B, D, dtype=torch.float32, device=dev) if need_grad else None
        tmp = torch.empty((2 if need_grad else 6) * B * D, dtype=torch.float32, device=dev)
        _lib.call("gpode_rk4_fwd_large_dev", ptr(field.packed), ctypes.byref(field.struct), ptr(xc), ptr(tc), Tg, B,
                  ptr(xs), ptr(kst), ptr(tmp), stream_ptr())
        _lib.LAUNCH_COUNT["gpode_rk4_fwd_large_dev"] += 12 * max(Tg - 2, 0)   # counted once per call: add the other steps
        ctx.field, ctx.nu_shape = field, nu.shape
        if need_grad:
            ctx.save_for_backward(tc, xs, kst)
        return xs

    @staticmethod
    def backward(ctx, gxs):
        field = ctx.field
        tc, xs, kst = ctx.saved_tensors
        Tg, B, D = xs.shape
        gxs = f32(gxs, "grad_xs")
        gx0 = torch.empty(B, D, dtype=torch.float32, device=xs.device)
        acc = field.new_acc()
        work = torch.empty(7 * B * D, dtype=torch.float32, device=xs.device)
        _lib.call("gpode_rk4_bwd_large", ptr(field.packed_bwd), ctypes.byref(field.struct), ptr(tc), Tg, B, ptr(xs),
                  ptr(kst), ptr(gxs), ptr(gx0), ptr(acc), ptr(work), stream_ptr())
        _lib.LAUNCH_COUNT["gpode_rk4_bwd_large"] += 12 * max(Tg - 2, 0)
        g_Z, g_ell, g_var, g_nu = field.finalize(acc, B)
        return gx0, None, g_Z, g_ell, g_var, g_nu.reshape(ctx.nu_shape), None, None, None, None


def vector_field(x, Z, ell, var, nu, omega, phase, w):
    """f(x) of one sampled GP function; differentiable in x, Z, ell, var, nu (D <= 8: register-resident kernels;
    8 < D <= 64: tcgen05 forward + ``gpode_vf_bwd_large``)."""
    if Z.shape[1] > MAX_D_REGISTER:
        return _VectorFieldLarge.apply(x, Z, ell, var, nu, omega, phase, w)
    return _VectorField.apply(x, Z, ell, var, nu, omega, phase, w)


def rk4_integrate(x0, t, Z, ell, var, nu, omega, phase, w):
    """Fixed-grid RK4 (3/8 rule) over the float32 grid ``t``; returns ``(len(t), B, D)`` like torchdiffeq."""
    if Z.shape[1] > MAX_D_REGISTER:
        return _RK4Large.apply(x0, f32(t.to(device=x0.device, dtype=torch.float32), "t"), Z, ell, var, nu, omega, phase,
                               w, torch.is_grad_enabled())
    return _RK4.apply(x0, t, Z, ell, var, nu, omega, phase, w, torch.is_grad_enabled())


# dopri5 training without a host round trip (CUDA-graph capture): fixed checkpoint capacity, accepted-step count read on
# the device by the backward kernels. The stats blocks of such integrations are collected here so that a caller
# (graphs.GraphedStep.check) can verify status == 0 after the fact.
DEVICE_COUNT_MODE = False          # force the device-count path outside capture (tests)
DEVICE_COUNT_STATS = []


def _device_count_mode():
    return DEVICE_COUNT_MODE or torch.cuda.is_current_stream_capturing()


class _Dopri5(torch.autograd.Function):
    """xs = odeint(f, x0, t, method='dopri5') (torchdiffeq 0.2.0 controller) via gpode_dopri5_fwd / gpode_dopri5_bwd."""

    @staticmethod
    def forward(ctx, x0, t, Z, ell, var, nu, omega, phase, w, rtol, atol, want_grad):
        lib = _lib.load()
        pc = PackedCache(Z, ell, var, nu, omega, phase, w)
        xc = f32(x0, "x0")
        if xc.ndim != 2 or xc.shape[1] != pc.D:
            raise _lib.GpodeError("x0 must be (B,%d), got %s" % (pc.D, tuple(xc.shape)))
        B, Tg = xc.shape[0], t.shape[0]
        t64 = t.detach().to(device=xc.device, dtype=torch.float64).contiguous()
        need_grad = want_grad and any(ctx.needs_input_grad[:6])
        xs = torch.empty(Tg, B, pc.D, dtype=torch.float32, device=xc.device)
        work = torch.empty(lib.gpode_dopri5_work_floats(pc.D, B), dtype=torch.float32, device=xc.device)
        stats = torch.zeros(4, dtype=torch.int32, device=xc.device)
        cap = max(32, 4 * Tg) if need_grad else 0
        ckpt, n_acc = None, 0
        ctx.on_device = need_grad and _device_count_mode()
        if ctx.on_device:
            cap = max(64, 8 * Tg)  # no retry possible without the host: generous capacity, status 3 if exceeded
            ckpt = torch.empty(lib.gpode_dopri5_ckpt_floats(pc.D, B, Tg, cap), dtype=torch.float32, device=xc.device)
            _lib.call("gpode_dopri5_fwd", ptr(pc.packed), pc.D, pc.M, pc.S, ptr(xc), ptr(t64), Tg, B, float(rtol),
                      float(atol), ptr(xs), ptr(work), ptr(stats), ptr(ckpt), cap, stream_ptr())
            DEVICE_COUNT_STATS.append(stats)
            ctx.pc, ctx.nu_shape, ctx.cap, ctx.n_acc = pc, nu.shape, cap, -1
            ctx.save_for_backward(t64, ckpt, stats)
            ctx.mark_non_differentiable(stats)
            return xs, stats
        while True:
            if need_grad:
                ckpt = torch.empty(lib.gpode_dopri5_ckpt_floats(pc.D, B, Tg, cap), dtype=torch.float32,
                                   device=xc.device)
            _lib.call("gpode_dopri5_fwd", ptr(pc.packed), pc.D, pc.M, pc.S, ptr(xc), ptr(t64), Tg, B, float(rtol),
                      float(atol), ptr(xs), ptr(work), ptr(stats), ptr(ckpt), cap, stream_ptr())
            if not need_grad:
                break  # inference: no host synchronisation at all; `stats` stays on the device
            st = [int(v) for v in stats.cpu()]  # training: one sync per integration (the reference syncs per attempt)
            if st[3] == 3 and B > 0:
                cap *= 2
                continue
            if st[3] != 0:
                raise _lib.GpodeError("dopri5 failed: status %d (1 = attempt limit, 2 = step-size underflow)" % st[3])
            n_acc = st[1]
            break
        ctx.pc, ctx.nu_shape, ctx.cap, ctx.n_acc = pc, nu.shape, cap, n_acc
        if need_grad:
            ctx.save_for_backward(t64, ckpt)
        ctx.mark_non_differentiable(stats)
        return xs, stats

    @staticmethod
    def backward(ctx, gxs, _gstats):
        lib = _lib.load()
        pc = ctx.pc
        gxs = f32(gxs, "grad_xs")
        Tg, B, D = gxs.shape
        gx0 = torch.empty(B, D, dtype=torch.float32, device=gxs.device)
        acc = pc.new_acc()
        if ctx.on_device:
            t64, ckpt, stats = ctx.saved_tensors
            n_max = (6 * ctx.cap + 1) * B
            vrows = torch.empty(lib.gpode_vrow_floats(D, n_max), dtype=torch.float32, device=gxs.device)
            _lib.call("gpode_dopri5_bwd_dev", ptr(pc.packed), pc.D, pc.M, pc.S, ptr(t64), Tg, B, ptr(gxs), ptr(ckpt),
                      ctx.cap, ptr(stats), ptr(gx0), ptr(vrows), ptr(acc), stream_ptr())
            _lib.call("gpode_param_grad_dev", ptr(pc.packed), pc.D, pc.M, pc.S, ptr(vrows), ptr(vrows[n_max * D:]),
                      n_max, ptr(stats), B, ptr(acc), stream_ptr())
            g_Z, g_ell, g_var, g_nu = pc.finalize(acc)
            return gx0, None, g_Z, g_ell, g_var, g_nu.reshape(ctx.nu_shape), None, None, None, None, None, None
        t64, ckpt = ctx.saved_tensors
        n_vr = (6 * ctx.n_acc + 1) * B
        vrows = torch.empty(lib.gpode_vrow_floats(D, n_vr), dtype=torch.float32, device=gxs.device)
        _lib.call("gpode_dopri5_bwd", ptr(pc.packed), pc.D, pc.M, pc.S, ptr(t64), Tg, B, ptr(gxs), ptr(ckpt), ctx.cap,
                  ctx.n_acc, ptr(gx0), ptr(vrows), ptr(acc), stream_ptr())
        if n_vr:
            _lib.call("gpode_param_grad", ptr(pc.packed), pc.D, pc.M, pc.S, ptr(vrows), ptr(vrows[n_vr * D:]), n_vr,
                      ptr(acc), stream_ptr())
        g_Z, g_ell, g_var, g_nu = pc.finalize(acc)
        return gx0, None, g_Z, g_ell, g_var, g_nu.reshape(ctx.nu_shape), None, None, None, None, None, None


def _dopri5_large_setup(field, x0, t):
    xc = f32(x0, "x0")
    if xc.ndim != 2 or xc.shape[1] != field.D:
        raise _lib.GpodeError("x0 must be (B,%d), got %s" % (field.D, tuple(xc.shape)))
    B, Tg = xc.shape[0], t.shape[0]
    t64 = t.detach().to(device=xc.device, dtype=torch.float64).contiguous()
    xs = torch.empty(Tg, B, field.D, dtype=torch.float32, device=xc.device)
    work = torch.empty(_lib.load().gpode_dopri5_large_work_floats(field.D, B), dtype=torch.float32, device=xc.device)
    stats = torch.zeros(4, dtype=torch.int32, device=xc.device)
    return xc, t64, xs, work, stats


def _dopri5_large_d(x0, t, Z, ell, var, nu, omega, phase, w, rtol, atol, max_attempts=100000):
    """dopri5 for 8 < D <= 64 without gradients: torchdiffeq 0.2.0's controller (whole-batch RMS norm, float64 time,
    Hairer initial step with order 4, safety 0.9 / growth <= 10 / shrink >= 0.2, quartic dense output) ON THE DEVICE --
    ``gpode_dopri5_fwd_large``: one attempt = six evaluations on the tcgen05 vector-field kernels + element-wise stage /
    error kernels + a one-CTA controller kernel, looped by a CUDA-graph WHILE node whose condition the controller sets.
    The host enqueues one graph launch and reads nothing back (the reference synchronises once per attempt)."""
    field = LargeField(Z, ell, var, nu, omega, phase, w)
    xc, t64, xs, work, stats = _dopri5_large_setup(field, x0, t)
    _lib.call("gpode_dopri5_fwd_large", ptr(field.packed), ctypes.byref(field.struct), ptr(xc), ptr(t64), t64.shape[0],
              xc.shape[0], float(rtol), float(atol), ptr(xs), ptr(work), ptr(stats), int(max_attempts), stream_ptr())
    return xs, stats


class _Dopri5Large(torch.autograd.Function):
    """Differentiable dopri5 for 8 < D <= 64: ``gpode_dopri5_fwd_large_ckpt`` records the accepted steps (8 B D floats
    each), ``gpode_dopri5_bwd_large`` runs their discrete adjoint on the large-D VJP kernels. One host read of the stats
    per integration: the checkpoint capacity doubles until it holds every accepted step."""

    @staticmethod
    def forward(ctx, x0, t, Z, ell, var, nu, omega, phase, w, rtol, atol, max_attempts):
        lib = _lib.load()
        field = LargeField(Z, ell, var, nu, omega, phase, w)
        xc, t64, xs, work, stats = _dopri5_large_setup(field, x0, t)
        B, D, Tg = xc.shape[0], field.D, t64.shape[0]
        cap = max(32, 4 * Tg)
        while True:
            ckpt = torch.empty(lib.gpode_dopri5_ckpt_floats(D, B, Tg, cap), dtype=torch.float32, device=xc.device)
            _lib.call("gpode_dopri5_fwd_large_ckpt", ptr(field.packed), ctypes.byref(field.struct), ptr(xc), ptr(t64),
                      Tg, B, float(rtol), float(atol), ptr(xs), ptr(work), ptr(stats), int(max_attempts), ptr(ckpt), cap,
                      stream_ptr())
            st = [int(v) for v in stats.cpu()]
            if st[3] == 3:
                cap *= 2
                continue
            if st[3] != 0:
                raise _lib.GpodeError("dopri5 failed: status %d (1 = attempt limit, 2 = step-size underflow)" % st[3])
            break
        ctx.field, ctx.nu_shape, ctx.cap, ctx.n_acc = field, nu.shape, cap, st[1]
        ctx.save_for_backward(t64, ckpt)
        ctx.mark_non_differentiable(stats)
        return xs, stats

    @staticmethod
    def backward(ctx, gxs, _gstats):
        field = ctx.field
        t64, ckpt = ctx.saved_tensors
        gxs = f32(gxs, "grad_xs")
        Tg, B, D = gxs.shape
        gx0 = torch.empty(B, D, dtype=torch.float32, device=gxs.device)
        acc = field.new_acc()
        work = torch.empty(11 * B * D, dtype=torch.float32, device=gxs.device)
        _lib.call("gpode_dopri5_bwd_large", ptr(field.packed_bwd), ctypes.byref(field.struct), ptr(t64), Tg, B,
                  ptr(gxs), ptr(ckpt), ctx.cap, ctx.n_acc, ptr(gx0), ptr(acc), ptr(work), stream_ptr())
        _lib.LAUNCH_COUNT["gpode_dopri5_bwd_large"] += 19 * max(ctx.n_acc - 1, 0)   # counted for one step: the others
        g_Z, g_ell, g_var, g_nu = field.finalize(acc, B)
        return gx0, None, g_Z, g_ell, g_var, g_nu.reshape(ctx.nu_shape), None, None, None, None, None, None


def dopri5_integrate(x0, t, Z, ell, var, nu, omega, phase, w, rtol=1e-6, atol=1e-6):
    """Adaptive dopri5 with torchdiffeq 0.2.0's controller in one cooperative kernel. Returns ``(xs (len(t),B,D),
    stats)`` with ``stats`` a device int32 tensor [nfe, accepted, rejected, status]. Differentiable in x0, Z, ell,
    var, nu through the discrete adjoint of the accepted steps (step sizes are constants, as in torchdiffeq).
    For 8 < D <= 64 the same controller runs on the device inside a CUDA-graph while loop; without gradients that path
    never synchronises with the host, with gradients it reads the stats once per integration."""
    if Z.shape[1] > MAX_D_REGISTER:
        if torch.is_grad_enabled() and any(a.requires_grad for a in (x0, Z, ell, var, nu)):
            return _Dopri5Large.apply(x0, t, Z, ell, var, nu, omega, phase, w, rtol, atol, 100000)
        return _dopri5_large_d(x0, t, Z, ell, var, nu, omega, phase, w, rtol, atol)
    return _Dopri5.apply(x0, t, Z, ell, var, nu, omega, phase, w, rtol, atol, torch.is_grad_enabled())


def _kzz_cholesky_large(Zd, ed, vd, jitter):
    """float64 ``L (D,M,M) = chol(K(Z,Z) + jitter I)`` per output dimension for 8 < D <= 64 (``torch.linalg``)."""
    D, M = ed.shape[0], Zd.shape[0]
    Ks = []
    for k0 in range(0, D, 8):   # direct-form squared distance, eight output dimensions at a time ((8, M, M, J) temporary)
        d = (Zd[None, :, None, :] - Zd[None, None, :, :]) / ed[k0:k0 + 8, None, None, :]
        Ks.append(vd[k0:k0 + 8, None, None] * torch.exp(-0.5 * (d * d).sum(-1)))
    K = torch.cat(Ks, 0)
    return torch.linalg.cholesky(K + jitter * torch.eye(M, dtype=torch.float64, device=Zd.device))


def _whiten_large(Z, ell, var, u, omega, phase, w, jitter):
    """The same whitening for 8 < D <= 64, where the in-shared-memory Cholesky kernels (one CTA per output dimension, a
    cluster of D <= 8 CTAs in the backward) do not apply: D batched M x M factorisations and triangular solves through
    torch.linalg (cuSOLVER / cuBLAS -- library calls, once per ELBO step) in float64 like the kernels, squared distance in
    the direct form, differentiated by autograd. At these state dimensions the step time is in the integrator kernels
    (tcgen05 vector field and VJP); this keeps ``DSVGP_Layer.build_cache`` -- and with it ``Flow`` and the model classes --
    usable up to D = 64 (reference src/core/dsvgp.py:92-122 has no dimension limit)."""
    D = ell.shape[0]
    S = w.shape[0]
    Zd, ed, vd = Z.double(), ell.double(), var.double()
    L = _kzz_cholesky_large(Zd, ed, vd, jitter)
    theta = torch.einsum('mj,jsk->msk', Zd, omega.double()) + phase.double().reshape(1, S, D)
    prior = (torch.cos(theta) * (w.double() * torch.sqrt(vd / S)).unsqueeze(0)).sum(1)  # rff_forward(Z): (M, D)
    a = torch.linalg.solve_triangular(L, prior.t().unsqueeze(2), upper=False)
    nu = torch.linalg.solve_triangular(L.transpose(1, 2), u.double().t().unsqueeze(2) - a, upper=True)
    return nu.squeeze(2).float()


def whiten(Z, ell, var, u, omega, phase, w, jitter=1e-5):
    """nu (D,M) = L^-T (u - L^-1 rff_forward(Z)), L = chol(K(Z,Z) + jitter I), per output dimension."""
    if Z.shape[1] > MAX_D_REGISTER:
        if not Z.is_cuda:
            raise _lib.GpodeError("gpode_b200 has no CPU path: Z is on %s" % Z.device)
        if Z.shape[1] > MAX_D_LARGE:
            raise _lib.GpodeError("state dimension D=%d above %d" % (Z.shape[1], MAX_D_LARGE))
        return _whiten_large(Z, ell, var, u, omega, phase, w, jitter)
    return _Whiten.apply(Z, ell, var, u, omega, phase, w, jitter)


def whitened_kl(Um, Us_sqrt_packed):
    return _WhitenedKL.apply(Um, Us_sqrt_packed)


# ---- batched Monte-Carlo prediction: n_sets function draws per launch (forward only) ------------------------------
def _sets_common(Z, ell, var, omega, phase, w):
    Zc, ec, vc = f32(Z, "Z"), f32(ell, "ell"), f32(var, "var")
    oc, wc = f32(omega, "omega"), f32(w, "w")
    M, D = Zc.shape
    if oc.ndim != 4 or wc.ndim != 3:
        raise _lib.GpodeError("sets tensors need a leading n_sets axis: omega (n,D,S,D), w (n,S,D); got %s, %s"
                              % (tuple(oc.shape), tuple(wc.shape)))
    n, S = wc.shape[0], wc.shape[1]
    if D > MAX_D_LARGE:
        raise _lib.GpodeError("batched prediction needs D <= %d, got %d" % (MAX_D_LARGE, D))
    pc_ = f32(phase, "phase").reshape(n, S, D)
    if tuple(oc.shape) != (n, D, S, D) or tuple(wc.shape) != (n, S, D) or tuple(ec.shape) != (D, D):
        raise _lib.GpodeError("inconsistent sets shapes: omega %s w %s ell %s" % (
            tuple(oc.shape), tuple(wc.shape), tuple(ec.shape)))
    return Zc, ec, vc, oc, pc_, wc, n, D, M, S


def _whiten_large_sets(Zc, ec, vc, uc, oc, pc_, wc, jitter):
    """``whiten_sets`` for 8 < D <= 64: one float64 Kzz factorisation for all draws (``_kzz_cholesky_large``, as
    ``_whiten_large`` does for one draw), then the prior at Z and the two triangular solves per draw, a chunk of draws at
    a time (the float64 angles are (n, M, S, D): 1.7 GB for 128 draws at M = 100, S = 256, D = 64)."""
    n, S, D = wc.shape
    M = Zc.shape[0]
    Zd, ed, vd = Zc.double(), ec.double(), vc.double()
    L = _kzz_cholesky_large(Zd, ed, vd, jitter)
    a_scale = torch.sqrt(vd / S)
    nu = torch.empty(n, D, M, dtype=torch.float32, device=Zc.device)
    chunk = max(1, (1 << 25) // (M * S * D))   # draws per chunk: at most 256 MB of float64 angles
    for q0 in range(0, n, chunk):
        q1 = min(n, q0 + chunk)
        theta = torch.einsum('mj,njsk->nmsk', Zd, oc[q0:q1].double()) + pc_[q0:q1].double().unsqueeze(1)
        prior = (torch.cos(theta) * (wc[q0:q1].double() * a_scale).unsqueeze(1)).sum(2)   # rff_forward(Z): (c, M, D)
        a = torch.linalg.solve_triangular(L, prior.transpose(1, 2).unsqueeze(3), upper=False)
        nq = torch.linalg.solve_triangular(L.transpose(1, 2), uc[q0:q1].double().transpose(1, 2).unsqueeze(3) - a,
                                           upper=True)
        nu[q0:q1] = nq.squeeze(3).float()
    return nu


def whiten_sets(Z, ell, var, u, omega, phase, w, jitter=1e-5):
    """``u (n,M,D)`` and per-draw ``omega (n,D,S,D)``, ``phase (n,S,D)``, ``w (n,S,D)`` -> ``nu (n,D,M)``. One Kzz
    factorisation for all draws (``gpode_whiten_fwd_sets``, ``gpode_whiten_fwd_sets_blocked`` above MAX_M inducing
    points; float64 ``torch.linalg`` for 8 < D <= 64). No gradient."""
    Zc, ec, vc, oc, pc_, wc, n, D, M, S = _sets_common(Z, ell, var, omega, phase, w)
    uc = f32(u, "u")
    if tuple(uc.shape) != (n, M, D):
        raise _lib.GpodeError("u must be (%d,%d,%d), got %s" % (n, M, D, tuple(uc.shape)))
    if D > MAX_D_REGISTER:
        return _whiten_large_sets(Zc, ec, vc, uc, oc, pc_, wc, jitter)
    st = _cache_struct(D, M, S, oc, pc_, wc, Zc, None, ec, vc)
    nu = torch.empty(n, D, M, dtype=torch.float32, device=Zc.device)
    L = torch.empty(D, M, M, dtype=torch.float64, device=Zc.device)
    sp = torch.empty(D, 2, M, dtype=torch.float64, device=Zc.device)
    if M > MAX_M:
        work = _whiten_work(D, M, n, Zc.device)
        _lib.call("gpode_whiten_fwd_sets_blocked", ctypes.byref(st), ptr(uc), float(jitter), n, ptr(nu), ptr(L),
                  ptr(sp), ptr(work), stream_ptr(), launches=_lib.whiten_blocked_launches(M))
    else:
        _lib.call("gpode_whiten_fwd_sets", ctypes.byref(st), ptr(uc), float(jitter), n, ptr(nu), ptr(L), ptr(sp),
                  stream_ptr())
    return nu


class PackedCacheSets:
    """``n`` sampled GP functions sharing Z and the hyper-parameters, packed back to back (``gpode_pack_cache_sets``;
    ``gpode_pack_cache_large_sets`` for 8 < D <= 64, whose kernels also read the "sets" cache ``struct``)."""

    def __init__(self, Z, ell, var, nu, omega, phase, w):
        lib = _lib.load()
        self.keep = _sets_common(Z, ell, var, omega, phase, w)
        Zc, ec, vc, oc, pc_, wc, self.n, self.D, self.M, self.S = self.keep
        nc = f32(nu, "nu").reshape(self.n, self.D, self.M)
        self.keep = self.keep + (nc,)
        self.struct = _cache_struct(self.D, self.M, self.S, oc, pc_, wc, Zc, nc, ec, vc)
        self.large = self.D > MAX_D_REGISTER
        if self.large:
            stride, pack = lib.gpode_packed_large_floats(self.D, self.M, self.S), "gpode_pack_cache_large_sets"
        else:
            stride, pack = lib.gpode_packed_floats(self.D, self.M, self.S), "gpode_pack_cache_sets"
        self.packed = torch.empty(self.n * stride, dtype=torch.float32, device=Zc.device)
        _lib.call(pack, ctypes.byref(self.struct), self.n, ptr(self.packed), stream_ptr())


def _rows_of_sets(x, pcs, name):
    xc = f32(x, name)
    if xc.ndim != 3 or xc.shape[0] != pcs.n or xc.shape[2] != pcs.D:
        raise _lib.GpodeError("%s must be (%d,N,%d), got %s" % (name, pcs.n, pcs.D, tuple(xc.shape)))
    return xc, xc.shape[1]


def vector_field_sets(x, Z, ell, var, nu, omega, phase, w):
    """``x (n,N,D)`` -> ``f (n,N,D)``: draw q's vector field at its own N points, all draws in one launch."""
    if torch.is_grad_enabled() and any(a.requires_grad for a in (x, Z, ell, var, nu)):
        raise _lib.GpodeError("the batched (sets) path is forward only: call it under torch.no_grad()")
    pcs = PackedCacheSets(Z, ell, var, nu, omega, phase, w)
    xc, N = _rows_of_sets(x, pcs, "x")
    f = torch.empty_like(xc)
    if pcs.large:
        _lib.call("gpode_vf_fwd_large_sets", ptr(pcs.packed), ctypes.byref(pcs.struct), pcs.n, N, ptr(xc),
                  ptr(torch.empty_like(xc)), ptr(f), stream_ptr())
        return f
    _lib.call("gpode_vf_fwd_sets", ptr(pcs.packed), pcs.D, pcs.M, pcs.S, pcs.n, N, ptr(xc), ptr(f), stream_ptr())
    return f


def integrate_sets(x0, t, Z, ell, var, nu, omega, phase, w, method="dopri5", rtol=1e-6, atol=1e-6):
    """``x0 (n,N,D)``, shared grid ``t (Tg,)`` -> ``(xs (n,N,Tg,D), stats)``: draw q integrates its own N trajectories
    with its own function, exactly as n separate ``odeint`` calls would (dopri5: one controller per draw), in ONE
    launch (8 < D <= 64: one sequence of launches of the large-D kernels, every launch covering all draws; draw q's
    trajectories and stats are bitwise those of the single-draw call). ``stats``: device int32 ``(n,4)`` [nfe,
    accepted, rejected, status] for dopri5, ``None`` for rk4."""
    if torch.is_grad_enabled() and any(a.requires_grad for a in (x0, Z, ell, var, nu)):
        raise _lib.GpodeError("the batched (sets) path is forward only: call it under torch.no_grad()")
    lib = _lib.load()
    pcs = PackedCacheSets(Z, ell, var, nu, omega, phase, w)
    xc, N = _rows_of_sets(x0, pcs, "x0")
    Tg = t.shape[0]
    xs = torch.empty(Tg, pcs.n * N, pcs.D, dtype=torch.float32, device=xc.device)
    stats = None
    if method == "rk4" and pcs.large:
        tc = f32(t.to(device=xc.device, dtype=torch.float32), "t")
        tmp = torch.empty(6 * pcs.n * N * pcs.D, dtype=torch.float32, device=xc.device)
        _lib.call("gpode_rk4_fwd_large_sets", ptr(pcs.packed), ctypes.byref(pcs.struct), pcs.n, N, ptr(xc), ptr(tc), Tg,
                  ptr(xs), ptr(tmp), stream_ptr())
        _lib.LAUNCH_COUNT["gpode_rk4_fwd_large_sets"] += 12 * max(Tg - 2, 0)   # counted once per call: the other steps
    elif method == "rk4":
        tc = f32(t.to(device=xc.device, dtype=torch.float32), "t")
        _lib.call("gpode_rk4_fwd_sets", ptr(pcs.packed), pcs.D, pcs.M, pcs.S, pcs.n, N, ptr(xc), ptr(tc), Tg, ptr(xs),
                  stream_ptr())
    elif method == "dopri5" and pcs.large:
        t64 = t.detach().to(device=xc.device, dtype=torch.float64).contiguous()
        work = torch.empty(lib.gpode_dopri5_large_sets_work_floats(pcs.D, pcs.n, N), dtype=torch.float32,
                           device=xc.device)
        stats = torch.zeros(pcs.n, 4, dtype=torch.int32, device=xc.device)
        _lib.call("gpode_dopri5_fwd_large_sets", ptr(pcs.packed), ctypes.byref(pcs.struct), pcs.n, N, ptr(xc), ptr(t64),
                  Tg, float(rtol), float(atol), ptr(xs), ptr(work), ptr(stats), 100000, stream_ptr())
    elif method == "dopri5":
        t64 = t.detach().to(device=xc.device, dtype=torch.float64).contiguous()
        work = torch.empty(lib.gpode_dopri5_work_floats(pcs.D, pcs.n * N), dtype=torch.float32, device=xc.device)
        stats = torch.zeros(pcs.n, 4, dtype=torch.int32, device=xc.device)
        _lib.call("gpode_dopri5_fwd_sets", ptr(pcs.packed), pcs.D, pcs.M, pcs.S, pcs.n, N, ptr(xc), ptr(t64), Tg,
                  float(rtol), float(atol), ptr(xs), ptr(work), ptr(stats), stream_ptr())
    else:
        raise _lib.GpodeError("integrate_sets: method %r has no fused CUDA integrator (rk4, dopri5)" % (method,))
    return xs.view(Tg, pcs.n, N, pcs.D).permute(1, 2, 0, 3), stats

