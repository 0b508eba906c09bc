"""interp1 / interp2 — the host-side mirror of arma::interp1 / arma::interp2 for this path.

    arma::interp1(X, Y, XI, YI, "*linear", extrap)        -> YI = interp1(X, Y, XI, extrap)
    arma::interp2(X, Y, Z, XI, YI, ZI, "linear", extrap)  -> ZI = interp2(X, Y, Z, XI, YI, extrap)

Same argument order and meaning as Armadillo's free functions (fn_interp1.hpp / fn_interp2.hpp;
the reference links Armadillo, Makefile:5, but vendors none of it).  numpy arrays are host
buffers and go through the host entry points of the C-ABI (include/b200_interp.h); torch CUDA
tensors stay resident in HBM and go through the *_dev entry points on torch's current stream.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import B200_F32, B200_F64, check

_DT = {np.dtype(np.float64): B200_F64, np.dtype(np.float32): B200_F32}


def _np(a, dt=None):
    a = np.ascontiguousarray(a) if dt is None else np.ascontiguousarray(a, dtype=dt)
    if a.dtype not in _DT:
        raise TypeError(f"dtype {a.dtype} is not supported (float64 / float32 only)")
    return a


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


def _is_torch(t):
    return type(t).__module__.startswith("torch")


def _torch_stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev_operands(dtype, *ts):
    """Check device operands: contiguous CUDA tensors of the plan's dtype, on one device, of equal length."""
    import torch
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    for t in ts:
        if not (_is_torch(t) and t.is_cuda):
            raise TypeError("device operands must all be CUDA tensors")
        if t.dtype != tdt:
            raise TypeError(f"device operands must have the plan's dtype {dtype}, not {t.dtype}")
        if not t.is_contiguous():
            raise TypeError("device operands must be contiguous")
        if t.device != ts[0].device:
            raise ValueError("device operands must be on one device")
        if t.numel() != ts[0].numel():
            raise ValueError("device operands must have the same number of elements")


class Interp1Plan:
    """Grid (X, Y) resident in HBM; interpolate many query batches (b200_interp1_plan_*)."""

    def __init__(self, X, Y):
        X = _np(X)
        Y = _np(Y, X.dtype)
        if X.ndim != 1 or X.shape != Y.shape:
            raise ValueError("X and Y must be vectors of equal length")
        self.dtype = X.dtype
        self.n = X.size
        self._h = C.c_void_p()
        check(_lib.lib().b200_interp1_plan_create(_DT[X.dtype], _ptr(X), _ptr(Y), C.c_size_t(X.size), C.byref(self._h)))

    @property
    def lookup_mode(self):
        return _lib.lib().b200_interp1_plan_lookup_mode(self._h)

    def set_values(self, Y):
        """New values on the same knots.  A CUDA tensor (plan dtype, contiguous, Y.numel() == n) is read in place,
        ordered on torch's current stream; anything else is a host array (synchronous)."""
        if _is_torch(Y) and Y.is_cuda:
            import torch
            tdt = torch.float64 if self.dtype == np.float64 else torch.float32
            if Y.dtype != tdt or not Y.is_contiguous():
                raise TypeError("device values must be a contiguous CUDA tensor of the plan's dtype")
            if Y.numel() != self.n:
                raise ValueError("Y has the wrong length")
            check(_lib.lib().b200_interp1_plan_set_values_dev(self._h, C.c_void_p(Y.data_ptr()), _torch_stream()))
            return
        Y = _np(Y, self.dtype)
        if Y.size != self.n:
            raise ValueError("Y has the wrong length")
        check(_lib.lib().b200_interp1_plan_set_values(self._h, _ptr(Y)))

    def __call__(self, XI, extrap=np.nan, return_index=False, out=None):
        if _is_torch(XI):
            return self._call_dev(XI, extrap, return_index, out)
        XI = _np(XI, self.dtype)
        YI = np.empty(XI.shape, self.dtype) if out is None else out
        idx = np.empty(XI.shape, np.int32) if return_index else None
        check(_lib.lib().b200_interp1_exec(self._h, _ptr(XI), C.c_size_t(XI.size), _ptr(YI),
                                          _ptr(idx) if return_index else None, C.c_double(extrap)))
        return (YI, idx) if return_index else YI

    def _call_dev(self, XI, extrap, return_index, out):
        import torch
        _dev_operands(self.dtype, XI, *(() if out is None else (out,)))
        YI = torch.empty_like(XI) if out is None else out
        idx = torch.empty(XI.shape, dtype=torch.int32, device=XI.device) if return_index else None
        check(_lib.lib().b200_interp1_exec_dev(self._h, C.c_void_p(XI.data_ptr()), C.c_size_t(XI.numel()),
                                              C.c_void_p(YI.data_ptr()),
                                              C.c_void_p(idx.data_ptr()) if return_index else None,
                                              C.c_double(extrap), _torch_stream()))
        return (YI, idx) if return_index else YI

    def grad(self, XI, extrap=np.nan):
        """Queries with their gradient: returns (YI, DYDX).  YI has the bits of the value call; DYDX is the slope of the
        segment (NaN for a NaN query, 0 outside the grid, the last segment's slope on the last knot;
        include/b200_interp.h).  A CUDA tensor runs on torch's current stream; numpy arrays take the host path."""
        if _is_torch(XI):
            import torch
            _dev_operands(self.dtype, XI)
            YI, DY = torch.empty_like(XI), torch.empty_like(XI)
            check(_lib.lib().b200_interp1_grad_dev(self._h, C.c_void_p(XI.data_ptr()), C.c_size_t(XI.numel()),
                                                  C.c_void_p(YI.data_ptr()), C.c_void_p(DY.data_ptr()),
                                                  C.c_double(extrap), _torch_stream()))
            return YI, DY
        XI = _np(XI, self.dtype)
        YI, DY = np.empty(XI.shape, self.dtype), np.empty(XI.shape, self.dtype)
        check(_lib.lib().b200_interp1_grad(self._h, _ptr(XI), C.c_size_t(XI.size), _ptr(YI), _ptr(DY),
                                          C.c_double(extrap)))
        return YI, DY

    def adjoint(self, XI, G):
        """dY = W^T G (n values): the gradient of sum_k G[k] * YI[k] with respect to Y, bit-for-bit deterministic
        (include/b200_interp.h).  From CUDA tensors: a CUDA tensor written on torch's current stream, with the scratch
        taken from torch's allocator.  From numpy: a numpy array."""
        if _is_torch(XI) or _is_torch(G):
            import torch
            _dev_operands(self.dtype, XI, G)
            lib = _lib.lib()
            ni = XI.numel()
            need = C.c_size_t()
            check(lib.b200_interp1_adjoint_workspace(self._h, C.c_size_t(ni), C.byref(need)))
            ws = torch.empty(max(need.value, 1), dtype=torch.uint8, device=XI.device)
            dY = torch.empty(self.n, dtype=XI.dtype, device=XI.device)
            check(lib.b200_interp1_adjoint_dev(self._h, C.c_void_p(XI.data_ptr()), C.c_void_p(G.data_ptr()),
                                              C.c_size_t(ni), C.c_void_p(dY.data_ptr()), C.c_void_p(ws.data_ptr()),
                                              C.c_size_t(ws.numel()), _torch_stream()))
            return dY
        XI = _np(XI, self.dtype)
        G = _np(G, self.dtype)
        if XI.size != G.size:
            raise ValueError("XI and G must have the same number of elements")
        dY = np.empty(self.n, self.dtype)
        check(_lib.lib().b200_interp1_adjoint(self._h, _ptr(XI), _ptr(G), C.c_size_t(XI.size), _ptr(dY)))
        return dY

    def interp_torch(self, XI, Y=None, extrap=np.nan):
        """Differentiable interpolation of a CUDA tensor (a torch.autograd.Function): gradients flow to XI and Y.  With Y
        given, the plan first takes Y as its values (set_values, ordered on torch's current stream) and holds them
        afterwards.  The backward pass uses the slopes saved by the forward pass and the adjoint; it never reads the
        plan's values, so a set_values between forward and backward does not change the gradients.  Once
        differentiable; no gradient for extrap."""
        return _interp1_function().apply(XI, Y, self, float(extrap))

    def close(self):
        if self._h:
            _lib.lib().b200_interp1_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Interp2Plan:
    """Grid (X, Y, Z) resident in HBM.  Z is Y.size x X.size (rows follow Y), any memory order;
    it is stored column-major like arma::mat."""

    NO_CELLS, FORCE_CELLS, NO_BANDS, FORCE_BANDS, NO_TILES, FORCE_TILES, ORDER_YX = 1, 2, 4, 8, 16, 32, 64   # include/b200_interp.h flags

    def __init__(self, X, Y, Z, flags=0):
        X = _np(X)
        Y = _np(Y, X.dtype)
        Z = np.asarray(Z)
        if Z.shape != (Y.size, X.size):
            raise ValueError("Z must be Y.size x X.size (arma: X.n_elem == Z.n_cols, Y.n_elem == Z.n_rows)")
        Zf = np.asfortranarray(Z, dtype=X.dtype)
        self.dtype = X.dtype
        self.nx, self.ny = X.size, Y.size
        self._h = C.c_void_p()
        check(_lib.lib().b200_interp2_plan_create_ex(_DT[X.dtype], _ptr(X), C.c_size_t(X.size), _ptr(Y),
                                                    C.c_size_t(Y.size), _ptr(Zf), C.c_uint(flags), C.byref(self._h)))

    def set_values(self, Z):
        """New Z (Y.size x X.size) on the same axes; afterwards the plan gives what a plan created with Z gives.
        A CUDA tensor of the plan's dtype is read in place, ordered on torch's current stream: strides (1, ld) are
        passed column-major, (ld, 1) row-major, any other layout is made contiguous first.  Anything else is a host
        array in any memory order (synchronous)."""
        if _is_torch(Z) and Z.is_cuda:
            import torch
            if tuple(Z.shape) != (self.ny, self.nx):
                raise ValueError(f"Z must have shape {(self.ny, self.nx)} (Y.size x X.size), not {tuple(Z.shape)}")
            if Z.dtype != (torch.float64 if self.dtype == np.float64 else torch.float32):
                raise TypeError(f"device Z must have the plan's dtype {self.dtype}, not {Z.dtype}")
            s0, s1 = Z.stride()
            if s1 == 1 and s0 >= self.nx:
                ld, row_major = s0, 1
            elif s0 == 1 and s1 >= self.ny:
                ld, row_major = s1, 0
            else:
                Z = Z.contiguous()
                ld, row_major = self.nx, 1
            check(_lib.lib().b200_interp2_plan_set_values_dev(self._h, C.c_void_p(Z.data_ptr()), C.c_size_t(ld),
                                                             C.c_int(row_major), _torch_stream()))
            return
        Z = np.asarray(Z)
        if Z.shape != (self.ny, self.nx):
            raise ValueError(f"Z must have shape {(self.ny, self.nx)} (Y.size x X.size), not {Z.shape}")
        if Z.dtype.kind not in "fiu":
            raise TypeError(f"Z of dtype {Z.dtype} is not supported (real numbers only)")
        Zf = np.asfortranarray(Z, dtype=self.dtype)
        check(_lib.lib().b200_interp2_plan_set_values(self._h, _ptr(Zf)))

    def grid(self, XI, YI, extrap=np.nan):
        """Tensor-grid queries (Armadillo's interp2 shape): returns ZI of shape (YI.size, XI.size).  CUDA tensors run
        on torch's current stream; numpy arrays take the host path."""
        if _is_torch(XI) or _is_torch(YI):
            import torch
            self._grid_axes_dev(XI, YI)
            ZI = torch.empty((XI.numel(), YI.numel()), dtype=XI.dtype, device=XI.device)  # column-major ZI
            check(_lib.lib().b200_interp2_grid_dev(self._h, C.c_void_p(XI.data_ptr()), C.c_size_t(XI.numel()),
                                                  C.c_void_p(YI.data_ptr()), C.c_size_t(YI.numel()),
                                                  C.c_void_p(ZI.data_ptr()), C.c_double(extrap), _torch_stream()))
            return ZI.t()
        XI = _np(XI, self.dtype)
        YI = _np(YI, self.dtype)
        ZI = np.empty((YI.size, XI.size), self.dtype, order="F")
        check(_lib.lib().b200_interp2_grid(self._h, _ptr(XI), C.c_size_t(XI.size), _ptr(YI), C.c_size_t(YI.size),
                                          _ptr(ZI), C.c_double(extrap)))
        return ZI

    def _grid_axes_dev(self, XI, YI):
        _dev_operands(self.dtype, XI)
        _dev_operands(self.dtype, YI)   # checked on its own: XI and YI may differ in length
        if YI.device != XI.device:
            raise ValueError("device operands must be on one device")

    def grid_grad(self, XI, YI, extrap=np.nan):
        """Tensor-grid queries with their gradient: returns (ZI, DZDX, DZDY), each of shape (YI.size, XI.size).  ZI has
        the bits of grid(); the slopes are those scattered_grad gives at every (XI[j], YI[i]) (include/b200_interp.h).
        CUDA tensors run on torch's current stream and return column-major views; numpy arrays take the host path and
        return Fortran-ordered arrays."""
        if _is_torch(XI) or _is_torch(YI):
            import torch
            self._grid_axes_dev(XI, YI)
            out = [torch.empty((XI.numel(), YI.numel()), dtype=XI.dtype, device=XI.device) for _ in range(3)]
            check(_lib.lib().b200_interp2_grid_grad_dev(self._h, C.c_void_p(XI.data_ptr()), C.c_size_t(XI.numel()),
                                                       C.c_void_p(YI.data_ptr()), C.c_size_t(YI.numel()),
                                                       *(C.c_void_p(t.data_ptr()) for t in out), C.c_double(extrap),
                                                       _torch_stream()))
            return tuple(t.t() for t in out)
        XI = _np(XI, self.dtype)
        YI = _np(YI, self.dtype)
        out = [np.empty((YI.size, XI.size), self.dtype, order="F") for _ in range(3)]
        check(_lib.lib().b200_interp2_grid_grad(self._h, _ptr(XI), C.c_size_t(XI.size), _ptr(YI), C.c_size_t(YI.size),
                                               *(_ptr(a) for a in out), C.c_double(extrap)))
        return tuple(out)

    def grid_adjoint(self, XI, YI, G):
        """dZ = W^T G, shape (ny, nx), with G of shape (YI.size, XI.size): the gradient of sum_ij G[i, j] * ZI[i, j] with
        respect to Z; the bits of scattered_adjoint on the mesh (include/b200_interp.h).  From CUDA tensors: G with
        strides (1, ld) or (ld, 1) is read in place (anything else is made contiguous), the result is a contiguous
        (row-major) CUDA tensor written on torch's current stream, and the scratch comes from torch's allocator.  From
        numpy: a Fortran-ordered array."""
        if _is_torch(XI) or _is_torch(YI) or _is_torch(G):
            import torch
            self._grid_axes_dev(XI, YI)
            nxi, nyi = XI.numel(), YI.numel()
            if not (_is_torch(G) and G.is_cuda and G.device == XI.device):
                raise TypeError("G must be a CUDA tensor on the device of XI and YI")
            if G.dtype != XI.dtype:
                raise TypeError(f"G must have the plan's dtype {self.dtype}, not {G.dtype}")
            if tuple(G.shape) != (nyi, nxi):
                raise ValueError(f"G must have shape {(nyi, nxi)} (YI.size x XI.size), not {tuple(G.shape)}")
            s0, s1 = G.stride()
            if s0 == 1 and s1 >= max(nyi, 1):
                ldg, g_row_major = s1, 0
            elif s1 == 1 and s0 >= max(nxi, 1):
                ldg, g_row_major = s0, 1
            else:
                G = G.contiguous()
                ldg, g_row_major = max(nxi, 1), 1
            lib = _lib.lib()
            need = C.c_size_t()
            check(lib.b200_interp2_grid_adjoint_workspace(self._h, C.c_size_t(nxi), C.c_size_t(nyi), C.byref(need)))
            ws = torch.empty(max(need.value, 1), dtype=torch.uint8, device=XI.device)
            dZ = torch.empty((self.ny, self.nx), dtype=XI.dtype, device=XI.device)
            check(lib.b200_interp2_grid_adjoint_dev(
                self._h, C.c_void_p(XI.data_ptr()), C.c_size_t(nxi), C.c_void_p(YI.data_ptr()), C.c_size_t(nyi),
                C.c_void_p(G.data_ptr()), C.c_size_t(ldg), C.c_int(g_row_major), C.c_void_p(dZ.data_ptr()),
                C.c_size_t(self.nx), C.c_int(1), C.c_void_p(ws.data_ptr()), C.c_size_t(ws.numel()), _torch_stream()))
            return dZ
        XI = _np(XI, self.dtype)
        YI = _np(YI, self.dtype)
        G = np.asarray(G)
        if G.shape != (YI.size, XI.size):
            raise ValueError(f"G must have shape {(YI.size, XI.size)} (YI.size x XI.size), not {G.shape}")
        Gf = np.asfortranarray(G, dtype=self.dtype)
        dZ = np.empty((self.ny, self.nx), self.dtype, order="F")
        check(_lib.lib().b200_interp2_grid_adjoint(self._h, _ptr(XI), C.c_size_t(XI.size), _ptr(YI), C.c_size_t(YI.size),
                                                  _ptr(Gf), _ptr(dZ)))
        return dZ

    def grid_torch(self, XI, YI, Z=None, extrap=np.nan):
        """Differentiable tensor-grid interpolation of CUDA tensors (a torch.autograd.Function): returns ZI of shape
        (YI.size, XI.size), and gradients flow to XI, YI and Z.  With Z given, the plan first takes Z as its values
        (set_values, ordered on torch's current stream) and holds them afterwards.  The backward pass uses the slopes
        saved by the forward pass and grid_adjoint; it never reads the plan's values, so a set_values between forward and
        backward does not change the gradients.  Once differentiable; no gradient for extrap."""
        return _grid2_function().apply(XI, YI, Z, self, float(extrap))

    def scattered(self, XQ, YQ, extrap=np.nan, out=None):
        """Scattered queries (XQ[k], YQ[k]) -> ZQ[k].  CUDA tensors run on torch's current stream; numpy arrays take
        the host path."""
        if _is_torch(XQ) or _is_torch(YQ):
            import torch
            _dev_operands(self.dtype, XQ, YQ, *(() if out is None else (out,)))
            ZQ = torch.empty_like(XQ) if out is None else out
            check(_lib.lib().b200_interp2_scattered_dev(self._h, C.c_void_p(XQ.data_ptr()), C.c_void_p(YQ.data_ptr()),
                                                       C.c_size_t(XQ.numel()), C.c_void_p(ZQ.data_ptr()),
                                                       C.c_double(extrap), _torch_stream()))
            return ZQ
        XQ = _np(XQ, self.dtype)
        YQ = _np(YQ, self.dtype)
        if XQ.shape != YQ.shape:
            raise ValueError("XQ and YQ must have the same shape")
        ZQ = np.empty(XQ.shape, self.dtype) if out is None else out
        check(_lib.lib().b200_interp2_scattered(self._h, _ptr(XQ), _ptr(YQ), C.c_size_t(XQ.size), _ptr(ZQ),
                                               C.c_double(extrap)))
        return ZQ

    def scattered_grad(self, XQ, YQ, extrap=np.nan):
        """Scattered queries with their gradient: returns (ZQ, DZDX, DZDY).  ZQ has the bits of scattered(); the slopes
        are those of the bilinear cell (NaN for a NaN coordinate, 0 outside the grid, the last cell's slope on the
        last knot; include/b200_interp.h).  CUDA tensors run on torch's current stream; numpy arrays take the host
        path."""
        if _is_torch(XQ) or _is_torch(YQ):
            import torch
            _dev_operands(self.dtype, XQ, YQ)
            ZQ, DX, DY = torch.empty_like(XQ), torch.empty_like(XQ), torch.empty_like(XQ)
            check(_lib.lib().b200_interp2_scattered_grad_dev(
                self._h, C.c_void_p(XQ.data_ptr()), C.c_void_p(YQ.data_ptr()), C.c_size_t(XQ.numel()),
                C.c_void_p(ZQ.data_ptr()), C.c_void_p(DX.data_ptr()), C.c_void_p(DY.data_ptr()), C.c_double(extrap),
                _torch_stream()))
            return ZQ, DX, DY
        XQ = _np(XQ, self.dtype)
        YQ = _np(YQ, self.dtype)
        if XQ.shape != YQ.shape:
            raise ValueError("XQ and YQ must have the same shape")
        ZQ, DX, DY = (np.empty(XQ.shape, self.dtype) for _ in range(3))
        check(_lib.lib().b200_interp2_scattered_grad(self._h, _ptr(XQ), _ptr(YQ), C.c_size_t(XQ.size), _ptr(ZQ),
                                                    _ptr(DX), _ptr(DY), C.c_double(extrap)))
        return ZQ, DX, DY

    def scattered_adjoint(self, XQ, YQ, G):
        """dZ = W^T G, shape (ny, nx): the gradient of sum_k G[k] * ZQ[k] with respect to Z, bit-for-bit deterministic
        (include/b200_interp.h).  From CUDA tensors: a contiguous (row-major) CUDA tensor written on torch's current
        stream, with the scratch taken from torch's allocator.  From numpy: a Fortran-ordered array."""
        if _is_torch(XQ) or _is_torch(YQ) or _is_torch(G):
            import torch
            _dev_operands(self.dtype, XQ, YQ, G)
            lib = _lib.lib()
            nq = XQ.numel()
            need = C.c_size_t()
            check(lib.b200_interp2_scattered_adjoint_workspace(self._h, C.c_size_t(nq), C.byref(need)))
            ws = torch.empty(max(need.value, 1), dtype=torch.uint8, device=XQ.device)
            dZ = torch.empty((self.ny, self.nx), dtype=XQ.dtype, device=XQ.device)
            check(lib.b200_interp2_scattered_adjoint_dev(
                self._h, C.c_void_p(XQ.data_ptr()), C.c_void_p(YQ.data_ptr()), C.c_void_p(G.data_ptr()),
                C.c_size_t(nq), C.c_void_p(dZ.data_ptr()), C.c_size_t(self.nx), C.c_int(1),
                C.c_void_p(ws.data_ptr()), C.c_size_t(ws.numel()), _torch_stream()))
            return dZ
        XQ = _np(XQ, self.dtype)
        YQ = _np(YQ, self.dtype)
        G = _np(G, self.dtype)
        if not (XQ.size == YQ.size == G.size):
            raise ValueError("XQ, YQ and G must have the same number of elements")
        dZ = np.empty((self.ny, self.nx), self.dtype, order="F")
        check(_lib.lib().b200_interp2_scattered_adjoint(self._h, _ptr(XQ), _ptr(YQ), _ptr(G), C.c_size_t(XQ.size),
                                                       _ptr(dZ)))
        return dZ

    def scattered_torch(self, XQ, YQ, Z=None, extrap=np.nan):
        """Differentiable scattered interpolation of CUDA tensors (a torch.autograd.Function): gradients flow to XQ, YQ
        and Z.  With Z given, the plan first takes Z as its values (set_values, ordered on torch's current stream) and
        holds them afterwards.  The backward pass uses the slopes saved by the forward pass and the adjoint; it never
        reads the plan's values, so a set_values between forward and backward does not change the gradients.  Once
        differentiable; no gradient for extrap."""
        return _scattered2_function().apply(XQ, YQ, Z, self, float(extrap))

    def close(self):
        if self._h:
            _lib.lib().b200_interp2_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_INTERP1 = None


def _interp1_function():
    """The autograd.Function of Interp1Plan.interp_torch (built on first use: torch is imported only when needed)."""
    global _INTERP1
    if _INTERP1 is None:
        import torch
        from torch.autograd.function import once_differentiable

        class Interp1(torch.autograd.Function):
            @staticmethod
            def forward(ctx, XI, Y, plan, extrap):
                _dev_operands(plan.dtype, XI)
                if Y is not None:
                    plan.set_values(Y.detach())
                ctx.plan = plan
                if ctx.needs_input_grad[0]:
                    YI, DY = plan.grad(XI, extrap)
                    ctx.save_for_backward(XI, DY)
                else:
                    YI = plan(XI, extrap)
                    ctx.save_for_backward(XI)
                return YI

            @staticmethod
            @once_differentiable
            def backward(ctx, g):
                g = g.contiguous()
                saved = ctx.saved_tensors
                gx = g * saved[1] if ctx.needs_input_grad[0] else None
                gY = ctx.plan.adjoint(saved[0], g) if ctx.needs_input_grad[1] else None
                return gx, gY, None, None

        _INTERP1 = Interp1
    return _INTERP1


_SCATTERED2 = None


def _scattered2_function():
    """The autograd.Function of Interp2Plan.scattered_torch (built on first use: torch is imported only when needed)."""
    global _SCATTERED2
    if _SCATTERED2 is None:
        import torch
        from torch.autograd.function import once_differentiable

        class Scattered2(torch.autograd.Function):
            @staticmethod
            def forward(ctx, XQ, YQ, Z, plan, extrap):
                _dev_operands(plan.dtype, XQ, YQ)
                if Z is not None:
                    plan.set_values(Z.detach())
                ctx.plan = plan
                if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
                    ZQ, DX, DY = plan.scattered_grad(XQ, YQ, extrap)
                    ctx.save_for_backward(XQ, YQ, DX, DY)
                else:
                    ZQ = plan.scattered(XQ, YQ, extrap)
                    ctx.save_for_backward(XQ, YQ)
                return ZQ

            @staticmethod
            @once_differentiable
            def backward(ctx, g):
                g = g.contiguous()
                saved = ctx.saved_tensors
                XQ, YQ = saved[0], saved[1]
                gx = g * saved[2] if ctx.needs_input_grad[0] else None
                gy = g * saved[3] if ctx.needs_input_grad[1] else None
                gZ = ctx.plan.scattered_adjoint(XQ, YQ, g) if ctx.needs_input_grad[2] else None
                return gx, gy, gZ, None, None

        _SCATTERED2 = Scattered2
    return _SCATTERED2


_GRID2 = None


def _grid2_function():
    """The autograd.Function of Interp2Plan.grid_torch (built on first use: torch is imported only when needed)."""
    global _GRID2
    if _GRID2 is None:
        import torch
        from torch.autograd.function import once_differentiable

        class Grid2(torch.autograd.Function):
            @staticmethod
            def forward(ctx, XI, YI, Z, plan, extrap):
                plan._grid_axes_dev(XI, YI)
                if Z is not None:
                    plan.set_values(Z.detach())
                ctx.plan = plan
                if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
                    ZI, DX, DY = plan.grid_grad(XI, YI, extrap)
                    ctx.save_for_backward(XI, YI, DX, DY)
                else:
                    ZI = plan.grid(XI, YI, extrap)
                    ctx.save_for_backward(XI, YI)
                return ZI

            @staticmethod
            @once_differentiable
            def backward(ctx, g):
                saved = ctx.saved_tensors
                XI, YI = saved[0], saved[1]
                gx = (g * saved[2]).sum(0) if ctx.needs_input_grad[0] else None
                gy = (g * saved[3]).sum(1) if ctx.needs_input_grad[1] else None
                gZ = ctx.plan.grid_adjoint(XI, YI, g) if ctx.needs_input_grad[2] else None
                return gx, gy, gZ, None, None

        _GRID2 = Grid2
    return _GRID2


def interp1(X, Y, XI, extrap=np.nan, return_index=False):
    """arma::interp1(X, Y, XI, YI, "*linear", extrap) — one-shot call (b200_interp1_f64/_f32)."""
    X = _np(X)
    Y = _np(Y, X.dtype)
    XI = _np(XI, X.dtype)
    YI = np.empty(XI.shape, X.dtype)
    idx = np.empty(XI.shape, np.int32) if return_index else None
    fn = _lib.lib().b200_interp1_f64 if X.dtype == np.float64 else _lib.lib().b200_interp1_f32
    ex = C.c_double(extrap) if X.dtype == np.float64 else C.c_float(extrap)
    check(fn(_ptr(X), _ptr(Y), C.c_size_t(X.size), _ptr(XI), C.c_size_t(XI.size), _ptr(YI),
             _ptr(idx) if return_index else None, ex))
    return (YI, idx) if return_index else YI


def interp2(X, Y, Z, XI, YI, extrap=np.nan):
    """arma::interp2(X, Y, Z, XI, YI, ZI, "linear", extrap) — one-shot call (b200_interp2_f64/_f32)."""
    X = _np(X)
    Y = _np(Y, X.dtype)
    Z = np.asarray(Z)
    if Z.shape != (Y.size, X.size):
        raise ValueError("Z must be Y.size x X.size")
    Zf = np.asfortranarray(Z, dtype=X.dtype)
    XI = _np(XI, X.dtype)
    YI = _np(YI, X.dtype)
    ZI = np.empty((YI.size, XI.size), X.dtype, order="F")
    fn = _lib.lib().b200_interp2_f64 if X.dtype == np.float64 else _lib.lib().b200_interp2_f32
    ex = C.c_double(extrap) if X.dtype == np.float64 else C.c_float(extrap)
    check(fn(_ptr(X), C.c_size_t(X.size), _ptr(Y), C.c_size_t(Y.size), _ptr(Zf), _ptr(XI), C.c_size_t(XI.size),
             _ptr(YI), C.c_size_t(YI.size), _ptr(ZI), ex))
    return ZI
