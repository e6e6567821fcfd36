"""Rank-local dense operators: the role third-party ``pylops`` operators play
inside MPIBlockDiag / MPIVStack in the reference (BlockDiag.py:127-129,
VStack.py:129-131 call ``oper.matvec`` on a slice of the local array).

Any object with ``shape``, ``dtype``, ``matvec(x)``, ``rmatvec(x)`` acting on
1-D device tensors can be used; :class:`MatrixMult` is the dense block every
reference test / BASELINE config uses, applied by the b2_gemv kernels.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib

__all__ = ["MatrixMult", "LocalOperator", "apply_into"]

_REAL_OF = {torch.complex64: torch.float32, torch.complex128: torch.float64}
_CPLX_OF = {torch.float32: torch.complex64, torch.float64: torch.complex128, torch.bfloat16: torch.complex64}
_OUT_OK = {}


def _accepts_out(fn) -> bool:
    """does this bound method take an ``out=`` keyword?  (signature inspection, cached per function: catching
    TypeError around the call would mask genuine TypeErrors raised inside the operator and re-run it)"""
    import inspect
    key = getattr(fn, "__func__", fn)
    ok = _OUT_OK.get(key)
    if ok is None:
        try:
            params = inspect.signature(fn).parameters
            ok = "out" in params or any(p.kind is inspect.Parameter.VAR_KEYWORD for p in params.values())
        except (TypeError, ValueError):
            ok = False
        _OUT_OK[key] = ok
    return ok


def apply_into(oper, x: torch.Tensor, out: torch.Tensor, adjoint: bool) -> None:
    """``out[...] = oper(x)`` / ``oper^H(x)`` for a rank-local operator, writing in place when the operator
    supports ``out=`` (the b200 local operators), else through a temporary (cast to ``out``'s dtype)."""
    fn = oper.rmatvec if adjoint else oper.matvec
    if _accepts_out(fn):
        fn(x, out=out)
    else:
        _store(out, fn(x))


def _store(out: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    """out <- y with NumPy ``__setitem__`` casting, as the reference's ``y[a:b] = oper.matvec(...)``
    (BlockDiag.py:127-129): complex into real keeps the real part and warns"""
    if y.dtype.is_complex and not out.dtype.is_complex:
        import warnings
        warnings.warn("Casting complex values to real discards the imaginary part", np.exceptions.ComplexWarning,
                      stacklevel=3)
        y = y.real
    out.copy_(y.reshape(out.shape))
    return out


class LocalOperator:
    """minimal rank-local linear operator interface"""
    shape = (0, 0)
    dtype = np.float64

    def matvec(self, x: torch.Tensor) -> torch.Tensor:
        return self._matvec(x)

    def rmatvec(self, x: torch.Tensor) -> torch.Tensor:
        return self._rmatvec(x)

    # pylops-style aliases (MPILinearOperator(Op=...) calls Op._matvec)
    def _matvec(self, x):
        raise NotImplementedError

    def _rmatvec(self, x):
        raise NotImplementedError


class MatrixMult(LocalOperator):
    """Dense block ``y = A x`` / ``y = A^H x`` (pylops.MatrixMult for a single
    right-hand side).  ``A`` may be a NumPy array (uploaded once) or a device
    tensor; dtype float32/float64/complex64/complex128, or bfloat16 with
    float32 vectors.  HBM-bound GEMV kernels (csrc/gemv.cu)."""

    def __init__(self, A, dtype=None):
        if not isinstance(A, torch.Tensor):
            A = torch.as_tensor(np.asarray(A))
        if dtype is not None:
            A = A.to(_lib.torch_dtype(dtype))
        if A.dim() != 2:
            raise ValueError("MatrixMult expects a 2-D array")
        _lib.ctx()
        self.A = A.to("cuda").contiguous()
        self.shape = (int(A.shape[0]), int(A.shape[1]))
        self._tdtype = self.A.dtype
        self._xdtype = torch.float32 if self._tdtype is torch.bfloat16 else self._tdtype
        self.dtype = _lib.numpy_dtype(self._xdtype)

    def _apply(self, x: torch.Tensor, op: int, out=None) -> torch.Tensor:
        m, n = self.shape
        x = x.reshape(-1)
        nin, nout = (n, m) if op == _lib.OP_N else (m, n)
        if x.numel() != nin:
            raise ValueError(f"dimension mismatch: operator {self.shape}, vector {x.numel()}")
        if x.dtype.is_complex and not self._xdtype.is_complex:
            # real operator, complex data: result_type(op, x) is complex (the reference's NumPy promotion) --
            # apply to the real and imaginary parts instead of dropping the imaginary one
            rdt = torch.promote_types(self._xdtype, _REAL_OF[x.dtype])
            yr = self._apply(x.real.contiguous(), op).to(rdt)
            yi = self._apply(x.imag.contiguous(), op).to(rdt)
            y = torch.complex(yr, yi)
            return y if out is None else _store(out, y)
        if x.dtype != self._xdtype:
            x = x.to(self._xdtype)
        if not x.is_contiguous():
            x = x.contiguous()
        direct = out is not None and out.dtype == self._xdtype and out.is_contiguous() and out.numel() == nout
        if out is not None and out.numel() != nout:
            raise ValueError(f"dimension mismatch: operator {self.shape}, out {out.numel()}")
        y = out if direct else torch.empty(nout, dtype=self._xdtype, device=x.device)
        _lib.check(_lib.lib.b2_gemv(_lib.ctx(), self.A.data_ptr(), n, m, n, x.data_ptr(), y.data_ptr(),
                                    op, _lib.code(self._tdtype), _lib.code(self._xdtype), _lib.stream()),
                   "b2_gemv")
        if out is not None and not direct:       # caller's buffer has another dtype (e.g. mixed-dtype BlockDiag)
            return _store(out, y)
        return y

    def _matvec(self, x, out=None):
        return self._apply(x, _lib.OP_N, out)

    def _rmatvec(self, x, out=None):
        return self._apply(x, _lib.OP_H, out)

    def matvec(self, x, out=None):
        return self._apply(x, _lib.OP_N, out)

    def rmatvec(self, x, out=None):
        return self._apply(x, _lib.OP_H, out)


class _AxisDerivative(LocalOperator):
    """Rank-local derivative along one axis of a C-ordered ``dims`` block (the role of
    pylops.FirstDerivative / pylops.SecondDerivative inside MPIBlockDiag in MPILaplacian / MPIGradient,
    Laplacian.py:97-126, Gradient.py:101-119).  One batched stencil launch (b2_derivative_axis)."""
    _deriv = 1

    def __init__(self, dims, axis: int = 0, sampling: float = 1.0, kind: str = "centered", edge: bool = False,
                 order: int = 3, dtype=np.float64):
        self.dims = tuple(int(d) for d in (dims if np.ndim(dims) else (dims,)))
        self.axis = axis % len(self.dims)
        n = int(np.prod(self.dims))
        self.shape = (n, n)
        self.sampling, self.edge, self.order = float(sampling), bool(edge), int(order)
        kinds = {"forward": _lib.FD_FORWARD, "backward": _lib.FD_BACKWARD, "centered": _lib.FD_CENTERED}
        if kind not in kinds:
            raise NotImplementedError("'kind' must be 'forward', 'centered', or 'backward'")
        if self._deriv == 1 and kind == "centered" and order not in (3, 5):
            raise NotImplementedError("'order' must be '3, or '5'")
        self._kind = kinds[kind]
        self._tdtype = _lib.torch_dtype(dtype)
        self.dtype = _lib.numpy_dtype(self._tdtype)
        _lib.ctx()

    def _apply(self, x: torch.Tensor, adjoint: int, out=None) -> torch.Tensor:
        x = x.reshape(-1)
        tdt = self._tdtype
        if x.dtype.is_complex and not tdt.is_complex:
            tdt = _CPLX_OF[torch.promote_types(tdt, _REAL_OF[x.dtype])]     # real taps on complex data
        if x.dtype != tdt:
            x = x.to(tdt)
        if not x.is_contiguous():
            x = x.contiguous()
        direct = out is not None and out.dtype == tdt and out.is_contiguous() and out.numel() == x.numel()
        y = out if direct else torch.empty_like(x)
        n_outer = int(np.prod(self.dims[:self.axis])) if self.axis else 1
        n_axis = self.dims[self.axis]
        n_inner = int(np.prod(self.dims[self.axis + 1:])) if self.axis + 1 < len(self.dims) else 1
        cx = tdt.is_complex
        real = _REAL_OF.get(tdt, tdt)
        if cx and n_inner == 1:
            # complex along the innermost axis: the (re, im) pairs are the "inner" dimension
            n_inner = 2
        elif cx:
            n_inner *= 2
        _lib.check(_lib.lib.b2_derivative_axis(_lib.ctx(), x.data_ptr(), y.data_ptr(), n_outer, n_axis, n_inner,
                                               self._deriv, self._kind, self.order, int(self.edge), self.sampling,
                                               adjoint, _lib.code(real), _lib.stream()), "b2_derivative_axis")
        if out is not None and not direct:
            return _store(out, y)
        return y

    def _matvec(self, x, out=None):
        return self._apply(x, 0, out)

    def _rmatvec(self, x, out=None):
        return self._apply(x, 1, out)

    def matvec(self, x, out=None):
        return self._apply(x, 0, out)

    def rmatvec(self, x, out=None):
        return self._apply(x, 1, out)


class FirstDerivative(_AxisDerivative):
    _deriv = 1


class SecondDerivative(_AxisDerivative):
    _deriv = 2

    def __init__(self, dims, axis: int = 0, sampling: float = 1.0, kind: str = "centered", edge: bool = False,
                 dtype=np.float64):
        super().__init__(dims, axis=axis, sampling=sampling, kind=kind, edge=edge, order=3, dtype=dtype)


CONVOLVE_MAX_TAPS = 2048       # B2_CONV_MAX_TAPS (include/b200lops.h)


class Convolve1D(LocalOperator):
    """Rank-local 1-D convolution of a C-ordered ``dims`` block with a real filter ``h`` along ``axis`` -- the
    ``pylops.signalprocessing.Convolve1D(dims, h, offset, axis)`` that the seismic tutorials wrap in MPIBlockDiag
    (tutorials/reflectivity.py:75)::

        y[i] = sum_k h[k] x[i + offset - k]        (x = 0 outside the axis)

    and its exact transpose.  One batched launch per apply (b2_convolve1d); the taps are uploaded once, here.
    ``method`` is accepted for signature compatibility: "direct", "fft" and "overlapadd" all run the direct
    kernel.  Complex data is convolved with the real filter (real and imaginary parts alike)."""

    def __init__(self, dims, h, offset: int = 0, axis: int = -1, dtype="float64", method=None):
        if method not in (None, "direct", "fft", "overlapadd"):
            raise NotImplementedError("method must be None, 'direct', 'fft' or 'overlapadd'")
        if isinstance(h, torch.Tensor):
            h = h.detach().cpu().numpy()
        h = np.asarray(h)
        if np.iscomplexobj(h):
            raise NotImplementedError("complex filters are not supported")
        if h.ndim != 1:
            raise NotImplementedError("only a single 1-D filter is supported (no per-trace filters)")
        if not 1 <= h.size <= CONVOLVE_MAX_TAPS:
            raise NotImplementedError(f"filter length must be between 1 and {CONVOLVE_MAX_TAPS}, got {h.size}")
        self.dims = tuple(int(d) for d in (dims if np.ndim(dims) else (dims,)))
        self.axis = axis % len(self.dims)
        n = int(np.prod(self.dims))
        self.shape = (n, n)
        self.nh, self.offset = int(h.size), int(offset)
        self._tdtype = _lib.torch_dtype(dtype)
        if _REAL_OF.get(self._tdtype, self._tdtype) not in (torch.float32, torch.float64):
            raise NotImplementedError(f"dtype {dtype} is not supported (float32, float64, complex64, complex128)")
        self.dtype = _lib.numpy_dtype(self._tdtype)
        _lib.ctx()
        # taps in both precisions (data of either precision may arrive), so an apply never copies from the host
        self._taps = {t: torch.as_tensor(h.astype(_lib.numpy_dtype(t))).to("cuda") for t in (torch.float32, torch.float64)}
        self.n_outer = int(np.prod(self.dims[:self.axis])) if self.axis else 1
        self.n_axis = self.dims[self.axis]
        self.n_inner = int(np.prod(self.dims[self.axis + 1:])) if self.axis + 1 < len(self.dims) else 1

    def _apply(self, x: torch.Tensor, adjoint: int, out=None) -> torch.Tensor:
        x = x.reshape(-1)
        if x.numel() != self.shape[1]:
            raise ValueError(f"dimension mismatch: operator {self.shape}, vector {x.numel()}")
        tdt = self._tdtype
        if x.dtype.is_complex and not tdt.is_complex:
            tdt = _CPLX_OF[torch.promote_types(tdt, _REAL_OF[x.dtype])]     # real taps on complex data
        if x.dtype != tdt:
            x = x.to(tdt)
        if not x.is_contiguous():
            x = x.contiguous()
        direct = out is not None and out.dtype == tdt and out.is_contiguous() and out.numel() == x.numel()
        y = out if direct else torch.empty_like(x)
        real = _REAL_OF.get(tdt, tdt)
        # complex data: the (re, im) pairs are part of the inner dimension
        n_inner = 2 * self.n_inner if tdt.is_complex else self.n_inner
        taps = self._taps[real]
        _lib.check(_lib.lib.b2_convolve1d(_lib.ctx(), x.data_ptr(), y.data_ptr(), self.n_outer, self.n_axis, n_inner,
                                          taps.data_ptr(), self.nh, self.offset, adjoint, _lib.code(real),
                                          _lib.stream()), "b2_convolve1d")
        if out is not None and not direct:
            return _store(out, y)
        return y

    def _matvec(self, x, out=None):
        return self._apply(x, 0, out)

    def _rmatvec(self, x, out=None):
        return self._apply(x, 1, out)

    def matvec(self, x, out=None):
        return self._apply(x, 0, out)

    def rmatvec(self, x, out=None):
        return self._apply(x, 1, out)


class FFT(LocalOperator):
    """Rank-local real FFT along ``axis`` of a ``dims`` block -- the role of third-party
    ``pylops.signalprocessing.FFT(dims, axis, real=True, ifftshift_before=..., norm="ortho")`` inside
    MPIMDC (waveeqprocessing/MDC.py:55-58).  cuFFT through ``torch.fft`` (library plumbing, not a
    hot-path kernel: the FFTs are rank-replicated pre/post-processing around MPIFredholm1).
    pylops is absent from this image: the scaling convention restated here (orthonormal transform, positive
    frequencies scaled by sqrt(2) so that the adjoint of the one-sided transform is exact) follows pylops 2.x;
    it is checked through the MPIMDC fixtures (reference chain over the same restatement in NumPy)."""

    def __init__(self, dims, axis: int = 0, real: bool = True, ifftshift_before: bool = False, dtype=np.float64):
        if not real:
            raise NotImplementedError("only the real (one-sided) transform used by MDC is provided")
        self.dims = tuple(int(d) for d in dims)
        self.axis = axis % len(self.dims)
        self.nfft = self.dims[self.axis]
        self.nfo = self.nfft // 2 + 1
        self.dimsd = self.dims[:self.axis] + (self.nfo,) + self.dims[self.axis + 1:]
        self.shape = (int(np.prod(self.dimsd)), int(np.prod(self.dims)))
        self.ifftshift_before = ifftshift_before
        self.rdtype = _lib.torch_dtype(dtype)
        self.cdtype = {torch.float32: torch.complex64, torch.float64: torch.complex128}[self.rdtype]
        self.dtype = _lib.numpy_dtype(self.cdtype)
        self._npos = (self.nfft - 1) // 2          # bins 1 .. npos are "doubled" positive frequencies

    def _sl(self, lo, hi):
        s = [slice(None)] * len(self.dims)
        s[self.axis] = slice(lo, hi)
        return tuple(s)

    def _scale_band(self, out: torch.Tensor, src: torch.Tensor, a: float):
        """out = src with the positive-frequency band (bins 1 .. npos along ``axis``) scaled by ``a`` -- through
        b2_lincomb (copy + in-band scale: at most three launches, no eager torch elementwise pass)"""
        one = _lib.cpair(1.0)
        code = _lib.code(src.dtype)
        ctx, st = _lib.ctx(), _lib.stream()
        if self.axis == 0 and self._npos > 0 and src.is_contiguous():
            inner = int(np.prod(self.dimsd[1:])) if len(self.dimsd) > 1 else 1
            so, ss = out.reshape(-1), src.reshape(-1)
            lo, hi = inner, (1 + self._npos) * inner
            for b, e, coef in ((0, lo, 1.0), (lo, hi, a), (hi, ss.numel(), 1.0)):
                if e > b and (coef != 1.0 or so.data_ptr() != ss.data_ptr()):
                    _lib.check(_lib.lib.b2_lincomb(ctx, so[b:].data_ptr(), _lib.cpair(coef), ss[b:].data_ptr(), None, None,
                                                   e - b, code, 0, st), "b2_lincomb")
            return out
        if out.data_ptr() != src.data_ptr():
            out.copy_(src)
        out[self._sl(1, 1 + self._npos)] *= a
        return out

    def _matvec(self, x: torch.Tensor) -> torch.Tensor:
        x = x.reshape(self.dims)
        x = x.real if x.is_complex() else x
        x = x.to(self.rdtype)
        if self.ifftshift_before:
            x = torch.fft.ifftshift(x, dim=self.axis)
        y = torch.fft.rfft(x, n=self.nfft, dim=self.axis, norm="ortho")
        return self._scale_band(y, y, float(np.sqrt(2.0))).reshape(-1)

    def _rmatvec(self, x: torch.Tensor) -> torch.Tensor:
        x = x.reshape(self.dimsd)
        if x.dtype != self.cdtype:
            x = x.to(self.cdtype)
        xs = self._scale_band(torch.empty_like(x, memory_format=torch.contiguous_format), x.contiguous(),
                              float(1.0 / np.sqrt(2.0)))
        y = torch.fft.irfft(xs, n=self.nfft, dim=self.axis, norm="ortho")
        if self.ifftshift_before:
            y = torch.fft.fftshift(y, dim=self.axis)
        return y.reshape(-1)


class Identity(LocalOperator):
    """``pylops.Identity(N, M)``: keep the first N of M samples (adjoint: zero-pad) -- the frequency
    truncation of MDC (MDC.py:61-64)."""

    def __init__(self, N: int, M: int = None, dtype=np.float64):
        M = N if M is None else M
        self.shape = (int(N), int(M))
        self.dtype = _lib.numpy_dtype(_lib.torch_dtype(dtype))

    @staticmethod
    def _pad(x: torch.Tensor, n: int) -> torch.Tensor:
        """zero-padded copy of flat ``x`` to ``n`` elements: b2_lincomb (copy) + b2_fill (tail)"""
        x = x.reshape(-1).contiguous()
        y = torch.empty(n, dtype=x.dtype, device=x.device)
        code, ctx, st = _lib.code(x.dtype), _lib.ctx(), _lib.stream()
        if x.numel():
            _lib.check(_lib.lib.b2_lincomb(ctx, y.data_ptr(), _lib.cpair(1.0), x.data_ptr(), None, None, x.numel(), code, 0, st),
                       "b2_lincomb")
        if n > x.numel():
            _lib.check(_lib.lib.b2_fill(ctx, y[x.numel():].data_ptr(), _lib.cpair(0.0), n - x.numel(), code, st), "b2_fill")
        return y

    def _matvec(self, x: torch.Tensor) -> torch.Tensor:
        N, M = self.shape
        return x[:N] if N <= M else self._pad(x, N)

    def _rmatvec(self, x: torch.Tensor) -> torch.Tensor:
        N, M = self.shape
        return x[:M] if M <= N else self._pad(x, M)
