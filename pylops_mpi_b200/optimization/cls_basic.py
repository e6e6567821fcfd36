"""CG / CGLS solvers with the reference's recurrences, stopping rule and
outputs (pylops_mpi/optimization/cls_basic.py:12-531); the ``Solver`` base the
reference takes from pylops (callbacks, timing, banner) is restated minimally.

Two execution modes, same numbers:
  * generic: the reference's exact sequence of DistributedArray operations;
  * fused (default on device arrays): identical recurrences, but axpy-style
    updates run in place (no temporaries) and reductions that the reference
    issues back to back are computed in one launch + one Allreduce
    (q.q and c.c together; s.s and x.x together), cutting the five
    host-synchronised reductions per iteration (:389-401) to three.
"""
from __future__ import annotations

import os
import sys
import time
from typing import List, Optional, Sequence

import numpy as np
import torch

from .. import _lib
from ..Distributed import allreduce_
from ..DistributedArray import DistributedArray


class Solver:
    """subset of pylops.optimization.basesolver.Solver used by CG/CGLS"""

    def __init__(self, Op, callbacks: Optional[Sequence] = None):
        self.Op = Op
        self.callbacks = callbacks
        self.tstart = time.time()

    def callback(self, x, *args, **kwargs):
        pass

    def _print_solver(self, text: str = "", nbar: int = 80) -> None:
        print(f"{type(self).__name__}" + text)
        print("-" * nbar + "\n" + f"The Operator Op has {self.Op.shape[0]} rows and {self.Op.shape[1]} cols")

    def _print_finalize(self, nbar: int = 80) -> None:
        print(f"\nIterations = {self.iiter}        Total time (s) = {self.telapsed:.2f}")
        print("-" * nbar + "\n")


_GRAPH_SAFE_TYPES = ("MPIBlockDiag", "MPIVStack", "MPIHStack", "MPIFirstDerivative", "MPISecondDerivative",
                     "_MPISummaMatrixMult", "_MPIBlockMatrixMult", "_AdjointLinearOperator", "_TransposedLinearOperator",
                     "_ProductLinearOperator", "_ScaledLinearOperator", "_SumLinearOperator", "_ConjLinearOperator",
                     "MatrixMult", "FirstDerivative", "SecondDerivative", "Convolve1D")


_GRAPH_POOL = {}
_CAPTURE_MODE = os.environ.get("B2_CGLS_CAPTURE_MODE", "thread_local")   # diagnostics: "global" / "relaxed"


def _graph_pool():
    """process-wide (per device) memory pool shared by every solver capture.  torch only lets a capture join an
    existing pool while at least one live graph still references it (otherwise capture_begin trips
    'use_count > 0' in the caching allocator -- seen when one solver's graph had been freed before the next solver
    captured), so a tiny ANCHOR graph captured once per device owns the pool for the life of the process."""
    dev = torch.cuda.current_device()
    hit = _GRAPH_POOL.get(dev)
    if hit is None:
        torch.zeros(16, device="cuda")                   # load the fill kernel outside any capture
        g = torch.cuda.CUDAGraph()
        main = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(main)
        with torch.cuda.stream(side):
            g.capture_begin(capture_error_mode="thread_local")
            try:
                keep = torch.zeros(16, device="cuda")    # one allocation + one kernel node: the graph is not empty
            finally:
                g.capture_end()
        main.wait_stream(side)
        hit = _GRAPH_POOL[dev] = (g.pool(), g, keep)
    return hit[0]


def _reset_capture_state():
    """a capture that died half-way leaves torch's CUDA generator flagged as 'capturing' (every later RNG call then
    raises 'Offset increment outside graph capture'): one empty, successful capture clears the flag"""
    try:
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            g.capture_begin(capture_error_mode="thread_local")
            g.capture_end()
        torch.cuda.synchronize()
    except Exception:
        pass


def _graph_safe(Op) -> bool:
    """may an apply of ``Op`` be captured once in a CUDA graph and replayed?  Conservative whitelist: operators of
    this package whose apply is a fixed sequence of kernel launches / collectives with no host-side per-call state
    (MPIFredholm1's fused mode toggles double buffers on the host, third-party operators are unknown -> eager)"""
    name = type(Op).__name__
    if name not in _GRAPH_SAFE_TYPES:
        return False
    if name == "_MPISummaMatrixMult" and Op.base_comm.Get_size() > 1 and not getattr(Op, "_stationary", False):
        return False       # the pipelined SUMMA forks streams per round: keep it eager
    for child in list(getattr(Op, "args", ())) + list(getattr(Op, "ops", ())):
        if hasattr(child, "shape") and not isinstance(child, (int, float, complex, np.number)):
            if not _graph_safe(child):
                return False
    return True


def _generic(*arrs) -> bool:
    """True when any operand is not a plain DistributedArray (StackedDistributedArray models / data,
    test_solver.py:303+): the solvers then run the reference's own sequence of ``dot / + / *`` operations
    instead of the fused device-scalar step"""
    return any(not isinstance(a, DistributedArray) for a in arrs)


def _absdot(a: DistributedArray, b: DistributedArray) -> float:
    """|a . conj(b)| as the reference computes it (np.abs(a.dot(b.conj())).item())"""
    return float(np.abs(a.dot(b.conj())).item())


def _self_dots(arrs: Sequence[DistributedArray]) -> List[float]:
    """[|a . conj(a)| for a in arrs] in ONE kernel launch + ONE Allreduce + ONE host sync"""
    import ctypes as C
    k = len(arrs)
    a0 = arrs[0]
    views = [a._scatter_view() for a in arrs]
    n = views[0].numel()
    same = all(v.numel() == n and v.dtype == views[0].dtype for v in views) and \
        all(a.sub_comm is a0.sub_comm for a in arrs)
    if not same or k > 4:
        return [_absdot(a, a) for a in arrs]
    cx = views[0].dtype.is_complex
    out = torch.zeros(2 * k, dtype=torch.float64, device=views[0].device)
    ptrs = (C.c_void_p * k)(*[v.data_ptr() if n else None for v in views])
    _lib.check(_lib.lib.b2_dot_multi(_lib.ctx(), k, ptrs, ptrs, n, _lib.code(views[0].dtype), 1,
                                     out.data_ptr(), _lib.stream()), "b2_dot_multi")
    allreduce_(a0.sub_comm, out, "sum")
    res = out.cpu().numpy()
    if cx:
        return [float(np.abs(complex(res[2 * i], res[2 * i + 1]))) for i in range(k)]
    return [float(np.abs(res[i])) for i in range(k)]


def _dots_device(arrs: Sequence[DistributedArray], out: torch.Tensor, offset: int = 0) -> int:
    """out[offset + i*stride] = a_i . conj(a_i) (LOCAL partial sums, float64, no host sync);
    returns the number of doubles written.  One launch when all arrays share a length."""
    import ctypes as C
    views = [a._scatter_view() for a in arrs]
    stride = 2 if views[0].dtype.is_complex else 1
    n0 = views[0].numel()
    if all(v.numel() == n0 for v in views) and len(views) <= 4:
        groups = [views]
    else:
        groups = [[v] for v in views]
    off = offset
    for g in groups:
        k = len(g)
        n = g[0].numel()
        ptrs = (C.c_void_p * k)(*[v.data_ptr() if n else None for v in g])
        _lib.check(_lib.lib.b2_dot_multi(_lib.ctx(), k, ptrs, ptrs, n, _lib.code(g[0].dtype), 1,
                                         out.data_ptr() + 8 * off, _lib.stream()), "b2_dot_multi")
        off += k * stride
    return off - offset


def _scalar_div(out: torch.Tensor, oi: int, num: torch.Tensor, ni: int, den1: torch.Tensor, d1: int,
                den2: Optional[torch.Tensor] = None, d2: int = 0, alpha: float = 0.0):
    """out[oi] = |num[ni] / (den1[d1] + alpha * den2[d2])| on the device"""
    _lib.check(_lib.lib.b2_scalar_div(out.data_ptr() + 8 * oi, num.data_ptr() + 8 * ni, den1.data_ptr() + 8 * d1,
                                      (den2.data_ptr() + 8 * d2) if den2 is not None else None, float(alpha),
                                      _lib.stream()), "b2_scalar_div")


def _lincomb_dev(out: DistributedArray, a_dev: Optional[torch.Tensor], ai: int, a_scale: float,
                 x: DistributedArray, b_dev: Optional[torch.Tensor], bi: int, b_scale: float,
                 y: DistributedArray):
    """out = (a_scale * a_dev[ai]) * x + (b_scale * b_dev[bi]) * y with DEVICE scalars (NULL -> 1)"""
    o, xv, yv = out._cont(), out._as_mine(x), out._as_mine(y)   # one dtype for the kernel: the updated array's
    n = o.numel()
    if n:
        _lib.check(_lib.lib.b2_lincomb_dev(_lib.ctx(), o.data_ptr(),
                                           (a_dev.data_ptr() + 8 * ai) if a_dev is not None else None, float(a_scale),
                                           xv.data_ptr(),
                                           (b_dev.data_ptr() + 8 * bi) if b_dev is not None else None, float(b_scale),
                                           yv.data_ptr(), n, _lib.code(o.dtype), _lib.stream()), "b2_lincomb_dev")
    if o is not out.local_array:
        out.local_array.copy_(o)


def _lincomb_dev_norm2(out: DistributedArray, a_dev: Optional[torch.Tensor], ai: int, a_scale: float,
                       x: DistributedArray, b_dev: Optional[torch.Tensor], bi: int, b_scale: float,
                       y: DistributedArray, dev: torch.Tensor, slot: int) -> bool:
    """out = (a_scale a_dev[ai]) x + (b_scale b_dev[bi]) y AND dev[slot] = sum |out|^2 (local partial) in ONE kernel.
    Falls back (returns False after doing the plain update) for BROADCAST arrays -- their reduction runs on the
    re-scattered view -- and mixed dtypes."""
    from ..DistributedArray import Partition
    o = out._cont()
    fusable = out.partition is Partition.SCATTER and o is out.local_array and \
        x._tdtype == out._tdtype and y._tdtype == out._tdtype and out._tdtype in (torch.float32, torch.float64,
                                                                                 torch.complex64, torch.complex128)
    if not fusable:
        _lincomb_dev(out, a_dev, ai, a_scale, x, b_dev, bi, b_scale, y)
        return False
    _lib.check(_lib.lib.b2_lincomb_dev_norm2(_lib.ctx(), o.data_ptr(),
                                             (a_dev.data_ptr() + 8 * ai) if a_dev is not None else None, float(a_scale),
                                             x._cont().data_ptr(),
                                             (b_dev.data_ptr() + 8 * bi) if b_dev is not None else None, float(b_scale),
                                             y._cont().data_ptr(), o.numel(), _lib.code(o.dtype),
                                             dev.data_ptr() + 8 * slot, _lib.stream()), "b2_lincomb_dev_norm2")
    return True


class CG(Solver):
    """cls_basic.py:12-249"""

    def setup(self, y, x0, niter: Optional[int] = None, tol: float = 1e-4, show: bool = False):
        self.y = y
        self.niter = niter
        self.tol = tol
        x = x0.copy()
        self.r = self.y - self.Op.matvec(x)
        self.rank = x.rank
        self.c = self.r.copy()
        self._gen = _generic(x, self.r)
        self.kold = _absdot(self.r, self.r) if self._gen else _self_dots([self.r])[0]
        self.cost: List = [float(np.sqrt(self.kold))]
        self.iiter = 0
        return x

    def _step_generic(self, x):
        """cls_basic.py:127-141 verbatim in operations (stacked arrays)"""
        Opc = self.Op.matvec(self.c)
        cOpc = np.abs(self.c.dot(Opc.conj()))
        a = float((self.kold / cOpc).item())
        x += a * self.c
        self.r -= a * Opc
        k = _absdot(self.r, self.r)
        b = float(k / self.kold)
        self.c = self.r + b * self.c
        self.kold = k
        self.iiter += 1
        self.cost.append(float(np.sqrt(self.kold)))
        return x

    def step(self, x, show: bool = False):
        if self._gen:
            return self._step_generic(x)
        Opc = self.Op.matvec(self.c)
        cOpc = np.abs(self.c.dot(Opc.conj()))
        with np.errstate(divide="ignore", invalid="ignore"):      # the reference divides NumPy scalars: inf / nan, no raise
            a = float((np.float64(self.kold) / cOpc).item())
        x.axpy_(a, self.c)
        self.r.axpy_(-a, Opc)
        k = _self_dots([self.r])[0]
        b = float(k / self.kold)
        self.c.xpby_(self.r, b)
        self.kold = k
        self.iiter += 1
        self.cost.append(float(np.sqrt(self.kold)))
        return x

    def run(self, x, niter: Optional[int] = None, show: bool = False, itershow=(10, 10, 10)):
        niter = self.niter if niter is None else niter
        if niter is None:
            raise ValueError("niter must not be None")
        while self.iiter < niter and self.kold > self.tol:
            x = self.step(x, False)
            self.callback(x)
        return x

    def finalize(self, show: bool = False) -> None:
        self.tend = time.time()
        self.telapsed = self.tend - self.tstart
        self.cost = np.array(self.cost)

    def solve(self, y, x0, niter: int = 10, tol: float = 1e-4, show: bool = False,
              itershow=(10, 10, 10)):
        x = self.setup(y=y, x0=x0, niter=niter, tol=tol, show=show)
        x = self.run(x, niter, show=show, itershow=itershow)
        self.finalize(show)
        return x, self.iiter, self.cost


class CGLS(Solver):
    """cls_basic.py:252-531"""

    def _print_step(self, x) -> None:
        x0 = (x if isinstance(x, DistributedArray) else x[0]).local_array.reshape(-1)[0].item()
        strx = f"{x0:1.2e}   " if isinstance(x0, complex) else f"{x0:11.4e}        "
        print(f"{self.iiter:6g}       " + strx + f"{self.cost[self.iiter]:11.4e}    {self.cost1[self.iiter]:11.4e}")
        sys.stdout.flush()

    def setup(self, y, x0, niter: Optional[int] = None, damp: float = 0.0, tol: float = 1e-4,
              show: bool = False):
        self.y = y
        self.damp = damp ** 2
        self.tol = tol
        self.niter = niter
        x = x0.copy()
        self.s = self.y - self.Op.matvec(x)
        self._gen = _generic(x, self.s)
        if self._gen:
            return self._setup_generic(x, damp, show)
        r = self.Op.rmatvec(self.s)
        if damp != 0.0:
            r.axpy_(-damp, x)                       # r = Op^H s - damp * x   (:341-342)
        self.rank = x.rank
        self.c = r.copy()
        self.q = self.Op.matvec(self.c)
        self.kold = _self_dots([r])[0]
        # device-resident scalars for the fused step: [qq, cc | k, ss, xx | a, b | kold] (x2 if complex)
        # slot stride of the packed device scalars: (re, im) pairs as soon as ANY of the arrays is complex (a real
        # model with complex-typed data, as in MPIMDC, must not let a complex dot spill into its neighbour's slot)
        self._st = 2 if (x._tdtype.is_complex or self.s._tdtype.is_complex or self.c._tdtype.is_complex) else 1
        self._dev = torch.zeros(16, dtype=torch.float64, device=x.local_array.device)
        self._dev[14] = self.kold
        self.cost = []
        self.cost1 = []
        ss, xx = _self_dots([self.s, x]) if self.s.local_shape == x.local_shape else \
            (_self_dots([self.s])[0], _self_dots([x])[0])
        self.cost.append(float(np.sqrt(ss)))
        # note: un-squared damp here, squared in step(), as in the reference (:358 vs :401)
        self.cost1.append(np.sqrt(float(self.cost[0] ** 2 + damp * xx)))
        self.iiter = 0
        if show and self.rank == 0:
            self._print_solver(nbar=65)
            print(f"damp = {self.damp:10e}\ttol = {self.tol:10e}\tniter = {self.niter}")
            print("-" * 65 + "\n")
            print("    Itn          x[0]              r1norm         r2norm")
        return x

    def _setup_generic(self, x, damp, show):
        """cls_basic.py:339-366 in the reference's own operations (stacked arrays)"""
        r = self.Op.rmatvec(self.s) - x * damp
        self.rank = x.rank
        self.c = r.copy()
        self.q = self.Op.matvec(self.c)
        self.kold = _absdot(r, r)
        self.cost = [float(self.s.norm().item())]
        self.cost1 = [np.sqrt(float(self.cost[0] ** 2 + damp * _absdot(x, x)))]
        self.iiter = 0
        if show and self.rank == 0:
            self._print_solver(nbar=65)
            print(f"damp = {self.damp:10e}\ttol = {self.tol:10e}\tniter = {self.niter}")
            print("-" * 65 + "\n")
            print("    Itn          x[0]              r1norm         r2norm")
        return x

    def _step_generic(self, x, show):
        """cls_basic.py:389-404 verbatim in operations"""
        a = float(np.abs(self.kold / (self.q.dot(self.q.conj()) + self.damp * self.c.dot(self.c.conj()))).item())
        x += a * self.c
        self.s -= a * self.q
        r = self.Op.rmatvec(self.s) - self.damp * x
        k = _absdot(r, r)
        b = float(k / self.kold)
        self.c = r + b * self.c
        self.q = self.Op.matvec(self.c)
        self.kold = k
        self.iiter += 1
        self.cost.append(float(self.s.norm().item()))
        self.cost1.append(np.sqrt(float(self.cost[self.iiter] ** 2 + self.damp * _absdot(x, x))))
        if show and self.rank == 0:
            self._print_step(x)
        return x

    def step(self, x, show: bool = False):
        """One CGLS iteration (cls_basic.py:370-404) with the scalars a, b kept on the device:
        2 Allreduces and ONE host synchronisation per iteration (the reference: 5 and 5)."""
        if self._gen:
            return self._step_generic(x, show)
        dev, st = self._dev, self._st
        QQ, CC, K, SS, XX, A_, B_, KOLD = 0, st, 4, 4 + st, 4 + 2 * st, 12, 13, 14
        sub = self.c.sub_comm
        if getattr(self, "_q_stale", False):       # a block run (rotated order) left q one matvec behind
            self.q = self.Op.matvec(self.c)
            self._q_stale = False
        # a = |kold / (q.q + damp c.c)|                                                  (:389)
        _dots_device([self.q], dev, QQ)
        _dots_device([self.c], dev, CC)
        allreduce_(sub, dev[0:2 * st], "sum")
        _scalar_div(dev, A_, dev, KOLD, dev, QQ, dev, CC, self.damp)
        _lincomb_dev(x, dev, A_, 1.0, self.c, None, 0, 1.0, x)            # x += a c       (:390)
        _lincomb_dev(self.s, dev, A_, -1.0, self.q, None, 0, 1.0, self.s)  # s -= a q       (:391)
        r = self.Op.rmatvec(self.s)                                        # r = Op^H s - damp x
        if self.damp != 0.0:
            r.axpy_(-self.damp, x)
        _dots_device([r], dev, K)
        _dots_device([self.s], dev, SS)
        _dots_device([x], dev, XX)
        allreduce_(sub, dev[4:4 + 3 * st], "sum")
        _scalar_div(dev, B_, dev, K, dev, KOLD)                            # b = k / kold   (:395)
        _lincomb_dev(self.c, None, 0, 1.0, r, dev, B_, 1.0, self.c)        # c = r + b c    (:396)
        self.q = self.Op.matvec(self.c)
        host = dev[4:4 + 3 * st].cpu().numpy()                             # the one sync of the iteration
        dev[KOLD:KOLD + 1].copy_(dev[K:K + 1])
        k, ss, xx = (float(abs(host[i * st])) for i in range(3))
        self.kold = k
        self.iiter += 1
        self.cost.append(float(np.sqrt(ss)))
        self.cost1.append(np.sqrt(float(self.cost[self.iiter] ** 2 + self.damp * xx)))
        if show and self.rank == 0:
            self._print_step(x)
        return x

    # ---- block execution: iterations without host round trips, replayed as ONE CUDA graph per iteration -----------
    def _body(self, x, hist: torch.Tensor, it_dev: torch.Tensor):
        """one CGLS iteration in ROTATED order (q = Op c first): every array that crosses iterations (x, s, c) is
        updated in place and q, r live and die inside the body, so the captured graph can be replayed verbatim.
        Same recurrences and the same kernels as :meth:`step`; the three per-iteration scalars go to ``hist``."""
        dev, st = self._dev, self._st
        QQ, CC, K, SS, XX, A_, B_, KOLD = 0, st, 4, 4 + st, 4 + 2 * st, 12, 13, 14
        sub = self.c.sub_comm
        self.q = self.Op.matvec(self.c)
        _dots_device([self.q], dev, QQ)
        if not self._cc_ready:                      # c.c normally comes fused with the update of c (end of the body)
            _dots_device([self.c], dev, CC)
        allreduce_(sub, dev[0:2 * st], "sum")
        _scalar_div(dev, A_, dev, KOLD, dev, QQ, dev, CC, self.damp)
        # x += a c (+ x.x), s -= a q (+ s.s): update and the reduction the cost needs, one pass each
        if not _lincomb_dev_norm2(x, dev, A_, 1.0, self.c, None, 0, 1.0, x, dev, XX):
            _dots_device([x], dev, XX)
        if not _lincomb_dev_norm2(self.s, dev, A_, -1.0, self.q, None, 0, 1.0, self.s, dev, SS):
            _dots_device([self.s], dev, SS)
        r = self.Op.rmatvec(self.s)
        if self.damp != 0.0:
            r.axpy_(-self.damp, x)
        _dots_device([r], dev, K)
        allreduce_(sub, dev[4:4 + 3 * st], "sum")
        _scalar_div(dev, B_, dev, K, dev, KOLD)
        # c = r + b c (+ c.c for the next iteration's step length)
        self._cc_ready = _lincomb_dev_norm2(self.c, None, 0, 1.0, r, dev, B_, 1.0, self.c, dev, CC)
        _lib.check(_lib.lib.b2_history_push(dev.data_ptr() + 8 * K, 3, st, hist.data_ptr(), it_dev.data_ptr(),
                                            hist.shape[0], dev.data_ptr() + 8 * KOLD, dev.data_ptr() + 8 * K,
                                            _lib.stream()), "b2_history_push")

    def _run_blocks(self, x, niter: int):
        """remaining iterations in blocks: the body is captured ONCE in a CUDA graph (after one eager warm-up
        iteration) and replayed; the host reads the scalar history once per block.  With tol > 0 a block is at
        most 8 iterations and is re-run from a checkpoint up to the stopping iteration, so x, cost and the
        iteration count are exactly those of the reference's per-iteration test ``kold > tol`` (cls_basic.py:436)."""
        device = x.local_array.device
        total = niter - self.iiter
        hist = torch.zeros((total + 2, 3), dtype=torch.float64, device=device)
        it_dev = torch.zeros(1, dtype=torch.int64, device=device)
        done = [0]          # iterations whose scalars are in hist

        def absorb(upto: int):
            """move hist[done:upto] to the host-side cost arrays; returns the first stop index or None"""
            rows = hist[done[0]:upto].cpu().numpy()
            stop = None
            for i, (k, ss, xx) in enumerate(rows):
                self.kold = float(k)
                self.iiter += 1
                self.cost.append(float(np.sqrt(ss)))
                self.cost1.append(np.sqrt(float(self.cost[self.iiter] ** 2 + self.damp * xx)))
                if not (self.iiter < niter and self.kold > self.tol):
                    stop = done[0] + i + 1
                    break
            done[0] = upto if stop is None else stop
            return stop

        def rewind(ckpt, upto_it: int):
            xs, ss_, cs = ckpt
            for dst, src in ((x, xs), (self.s, ss_), (self.c, cs)):
                dst.local_array.copy_(src)
            self._dev[14] = self._kold_ckpt
            it_dev.fill_(upto_it)
            if self._cc_ready:                      # the fused c.c partial belongs to the restored c again
                _dots_device([self.c], self._dev, self._st)

        use_graph = os.environ.get("B2_CGLS_GRAPH", "1") != "0" and _graph_safe(self.Op)
        state = {"graph": None, "use": use_graph, "warm": 0}
        self.graph_replays, self.graph_error = 0, (None if use_graph else "operator not on the graph-safe list")
        self._cc_ready = False                      # first body computes c.c itself

        def one():
            """one iteration: the first runs eagerly (every kernel of the body gets loaded, lazy workspaces and
            communicators exist), then the body is captured once and replayed"""
            if state["graph"] is None and state["use"] and state["warm"] >= 1:
                t_cap = time.perf_counter()
                try:
                    # manual capture on a side stream (torch.cuda.graph() would add a device synchronise, a
                    # gc.collect() and an empty_cache() -- milliseconds, comparable to a whole 50-iteration solve)
                    pool = _graph_pool()
                    t_pool = time.perf_counter()
                    g = torch.cuda.CUDAGraph()
                    main = torch.cuda.current_stream()
                    if state.get("stream") is None:
                        state["stream"] = torch.cuda.Stream()
                    side = state["stream"]
                    side.wait_stream(main)
                    with torch.cuda.stream(side):
                        # one process-wide memory pool for all captures: the temporaries of the first capture are
                        # cudaMalloc'ed (slow when peers have this device mapped: measured 3.1 ms at 2 GPUs vs 0.65 ms
                        # at 1), later captures reuse the cached blocks
                        # thread_local error mode: NCCL's helper threads keep polling CUDA while we capture
                        # (observed at 8 ranks: a "global"-mode capture was invalidated and left torch's RNG state
                        # stuck in capture mode)
                        g.capture_begin(pool=pool, capture_error_mode=_CAPTURE_MODE)   # records only
                        t_begin = time.perf_counter()
                        try:
                            self._body(x, hist, it_dev)
                        finally:
                            t_body = time.perf_counter()
                            g.capture_end()
                    main.wait_stream(side)
                    state["graph"] = g
                    self.graph_replays = 0
                    t_end = time.perf_counter()
                    self.graph_capture_ms = (t_end - t_cap) * 1e3
                    self.graph_capture_breakdown_ms = {"pool": (t_pool - t_cap) * 1e3, "begin": (t_begin - t_pool) * 1e3,
                                                       "body": (t_body - t_begin) * 1e3, "end": (t_end - t_body) * 1e3}
                except Exception as exc:               # not capturable (host sync inside an operator ...): stay eager
                    state["use"] = False
                    self.graph_error = repr(exc)[:300]
                    print(f"[b200 cgls] CUDA-graph capture failed, running eagerly: {self.graph_error}", file=sys.stderr)
                    torch.cuda.synchronize()
                    _reset_capture_state()
            if state["graph"] is not None:
                state["graph"].replay()
                self.graph_replays += 1
            else:
                self._body(x, hist, it_dev)
                state["warm"] += 1

        block = total if self.tol <= 0.0 else min(total, 8)
        while self.iiter < niter and self.kold > self.tol:
            n = min(block, niter - self.iiter)
            start = done[0]
            ckpt = tuple(a.local_array.clone() for a in (x, self.s, self.c))
            self._kold_ckpt = float(self.kold)
            for _ in range(n):
                one()
            stop = absorb(start + n)
            if stop is not None and stop < start + n:
                # the stopping test fired inside the block: redo exactly the iterations up to it from the checkpoint
                rewind(ckpt, start)
                for _ in range(stop - start):
                    one()
            del ckpt
        self._q_stale = True        # rotated order: q is one matvec behind c (and lives in the graph's memory pool)
        self.q = None
        return x

    def run(self, x, niter: Optional[int] = None, show: bool = False, itershow=(10, 10, 10)):
        niter = self.niter if niter is None else niter
        if niter is None:
            raise ValueError("niter must not be None")
        plain_callback = type(self).callback is Solver.callback and not self.callbacks
        if not self._gen and not show and plain_callback and niter - self.iiter > 0:
            return self._run_blocks(x, niter)
        while self.iiter < niter and self.kold > self.tol:
            showstep = bool(show and (self.iiter < itershow[0] or niter - self.iiter < itershow[1]
                                      or self.iiter % itershow[2] == 0))
            x = self.step(x, showstep)
            self.callback(x)
        return x

    def finalize(self, show: bool = False, **kwargs) -> None:
        self.tend = time.time()
        self.telapsed = self.tend - self.tstart
        self.istop = 1 if self.kold < self.tol else 2
        self.r1norm = self.kold
        self.r2norm = self.cost1[self.iiter]
        if show and self.rank == 0:
            self._print_finalize(nbar=65)
        self.cost = np.array(self.cost)

    def solve(self, y, x0, niter: int = 10, damp: float = 0.0, tol: float = 1e-4, show: bool = False,
              itershow=(10, 10, 10)):
        x = self.setup(y=y, x0=x0, niter=niter, damp=damp, tol=tol, show=show)
        x = self.run(x, niter, show=show, itershow=itershow)
        self.finalize(show)
        return x, self.istop, self.iiter, self.r1norm, self.r2norm, self.cost
