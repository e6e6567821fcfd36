"""local.Convolve1D (b2_convolve1d): the NumPy oracle against the pylops restatement and the reference's fixtures
(tests/golden/convolve_golden.npz), then the CUDA operator inside MPIBlockDiag / ISTA / CGLS against both."""
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if HERE not in sys.path:
    sys.path.insert(0, HERE)
import golden_store  # noqa: E402
import convolve_oracle as co  # noqa: E402
import pylops_mpi_oracle as o  # noqa: E402

GOLD = golden_store.Golden(os.path.join(HERE, "golden", "convolve_golden.npz"))
GRID = [(P, dims, axis, nh, off, dt) for P in co.GRID_P for dims, axis in co.GRID_DIMS for nh in co.GRID_NH
        for off in co.grid_offsets(nh) for dt in co.GRID_DTYPES]


def _id(c):
    return co.grid_key(*c)[5:]


def oracle_blocks(x, P, dims, h, offset, axis, adjoint):
    n = int(np.prod(dims))
    return [co.convolve1d(x[r * n:(r + 1) * n], dims, h, offset, axis, adjoint) for r in range(P)]


def _close(dt):
    """tolerance against the reference's output: float32 data is rounded once to float32 there"""
    return dict(rtol=1e-5, atol=1e-5) if dt == "float32" else dict(rtol=1e-12, atol=1e-12)


# ---------------------------------------------------------------------------------------------------------------
# CPU: oracle vs restatement vs fixtures
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dims,axis", list(co.GRID_DIMS) + [((3,), 0), ((2, 50), 0)])
def test_oracle_matches_pylops_restatement(dims, axis):
    shim = os.path.join(HERE, "golden", "refshim")         # on sys.path only for this import (it has an mpi4py stand-in)
    sys.path.insert(0, shim)
    try:
        from pylops.signalprocessing.convolve1d import Convolve1D
    finally:
        sys.path.remove(shim)
    rng = np.random.default_rng(5)
    n = int(np.prod(dims))
    for nh in (1, 2, 4, 5, 6, 40, 41):
        for off in sorted({0, nh // 2, nh - 1}):
            h = rng.standard_normal(nh)
            x = rng.standard_normal(n) + 1j * rng.standard_normal(n)
            R = Convolve1D(dims, h, offset=off, axis=axis)
            for adj, ref in ((False, R._matvec), (True, R._rmatvec)):
                np.testing.assert_allclose(co.convolve1d(x, dims, h, off, axis, adj), ref(x), rtol=1e-12, atol=1e-12,
                                           err_msg=f"nh={nh} offset={off} adjoint={adj}")


@pytest.mark.parametrize("case", GRID, ids=_id)
def test_oracle_reproduces_fixture(case):
    P, dims, axis, nh, off, dt = case
    key = co.grid_key(*case)
    h, x = co.grid_inputs(key, P, dims, nh, dt)
    GOLD.record(key + "/h").check(h)
    GOLD.record(key + "/x").check(x)
    for name, adj in (("y", False), ("ya", True)):
        GOLD.record(key + "/" + name).check(oracle_blocks(x, P, dims, h, off, axis, adj), **_close(dt))


def test_oracle_adjoint_dottest():
    rng = np.random.default_rng(8)
    for dims, axis in co.GRID_DIMS:
        n = int(np.prod(dims))
        for nh in (1, 4, 41):
            for off in (-3, 0, nh // 2, nh - 1, nh + 7):
                h, u, v = rng.standard_normal(nh), rng.standard_normal(n), rng.standard_normal(n)
                lhs = np.dot(co.convolve1d(u, dims, h, off, axis), v)
                rhs = np.dot(u, co.convolve1d(v, dims, h, off, axis, adjoint=True))
                assert abs(lhs - rhs) <= 1e-12 * max(1.0, abs(lhs)), (dims, axis, nh, off)


class _BlockConv:
    """MPIBlockDiag([Convolve1D]) over P blocks, as the ``A`` of the oracle's ISTA (``A @ x``, ``A.conj().T @ r``)"""

    def __init__(self, P, dims, h, offset, adjoint=False):
        self.P, self.dims, self.h, self.offset, self.adjoint = P, dims, h, offset, adjoint

    def __matmul__(self, x):
        return np.concatenate(oracle_blocks(x, self.P, self.dims, self.h, self.offset, -1, self.adjoint))

    def conj(self):
        return self

    @property
    def T(self):
        return _BlockConv(self.P, self.dims, self.h, self.offset, not self.adjoint)


def refl_oracle(P):
    """the reflectivity chain in the oracle: r = D m, d = C r, ISTA and CGLS on C"""
    wav, m = co.refl_inputs(P)
    dims, wavc = co.REFL_DIMS, co.REFL_NT // 2
    n = int(np.prod(dims))
    D = o.first_derivative_dense(dims[-1])
    r = np.concatenate([o.derivative_along_axis(m[i * n:(i + 1) * n].reshape(dims), 2, D).ravel() for i in range(P)])
    C = _BlockConv(P, dims, wav, wavc)
    d = C @ r
    alpha = 1.0 / np.sum(np.abs(wav)) ** 2
    xi, iiter, cost = o.ista(C, d, np.zeros_like(d), 30, 1e-2, alpha, 1e-8, "soft")
    split = lambda v: o.SimArray([v[i * n:(i + 1) * n] for i in range(P)])                       # noqa: E731
    mv = lambda a: split(C @ a.asarray())                                                         # noqa: E731
    rmv = lambda a: split(C.T @ a.asarray())                                                      # noqa: E731
    xc, _s, iitc, _r1, _r2, costc = o.cgls(mv, rmv, split(d), split(np.zeros_like(d)), niter=20, tol=0.0)
    return dict(wav=wav, m=m, r=r, d=d, alpha=alpha, ista_x=xi, ista_iiter=iiter, ista_cost=cost,
                cgls_x=xc.asarray(), cgls_cost=costc, cgls_iit=iitc)


@pytest.mark.parametrize("P", co.GRID_P)
def test_oracle_reproduces_reflectivity_chain(P):
    ref = refl_oracle(P)
    g = f"refl/P{P}/"
    GOLD.record(g + "wav").check(ref["wav"])
    GOLD.record(g + "m").check(ref["m"])
    assert float(GOLD[g + "alpha"]) == ref["alpha"]
    for k in ("r", "d"):
        GOLD.record(g + k).check(ref[k], rtol=1e-12, atol=1e-12)
    assert int(GOLD[g + "ista_iiter"]) == ref["ista_iiter"]
    np.testing.assert_allclose(ref["ista_cost"], GOLD.record(g + "ista_cost").values, rtol=1e-10)
    GOLD.record(g + "ista_x").check(ref["ista_x"], rtol=1e-10, atol=1e-10)
    assert int(GOLD[g + "cgls_iit"]) == ref["cgls_iit"] == 20
    np.testing.assert_allclose(ref["cgls_cost"], GOLD.record(g + "cgls_cost").values, rtol=1e-9)
    GOLD.record(g + "cgls_x").check(ref["cgls_x"], rtol=1e-8, atol=1e-8)


# ---------------------------------------------------------------------------------------------------------------
# GPU: the CUDA operator
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pm():
    import pylops_mpi_b200 as pm
    return pm


def host(t):
    return t.cpu().numpy()


def block_op(pm, P, dims, h, offset, axis, dtype):
    """all P ranks' blocks on the one rank (world size 1)"""
    return pm.MPIBlockDiag([pm.local.Convolve1D(dims, h, offset=offset, axis=axis, dtype=dtype) for _ in range(P)])


@pytest.mark.gpu
@pytest.mark.parametrize("case", GRID, ids=_id)
def test_gpu_convolve_vs_reference(pm, case):
    P, dims, axis, nh, off, dt = case
    key = co.grid_key(*case)
    h, x = co.grid_inputs(key, P, dims, nh, dt)
    Op = block_op(pm, P, dims, h, off, axis, dt)
    xd = pm.DistributedArray.to_dist(x)
    for name, adj, got in (("y", False, Op @ xd), ("ya", True, Op.H @ xd)):
        got = host(got.asarray())
        assert got.dtype == np.dtype(dt)
        want = np.concatenate(oracle_blocks(x, P, dims, h, off, axis, adj))
        if dt == "float32":
            assert np.linalg.norm(got - want) <= 1e-6 * np.linalg.norm(want), name
            GOLD.record(key + "/" + name).check(got, rtol=1e-4, atol=1e-4)
        else:
            np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12, err_msg=name)
            GOLD.record(key + "/" + name).check(got, rtol=1e-12, atol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("dims,axis", list(co.GRID_DIMS) + [((3000,), 0), ((7, 2051), -1), ((600, 6), 0)])
@pytest.mark.parametrize("nh,off", [(1, 0), (5, 2), (41, 20), (40, 3), (41, -5), (12, 30)])
def test_gpu_dottest(pm, dims, axis, nh, off):
    rng = np.random.default_rng(11)
    n = int(np.prod(dims))
    h = rng.standard_normal(nh)
    Op = pm.MPIBlockDiag([pm.local.Convolve1D(dims, h, offset=off, axis=axis)])
    u = pm.DistributedArray.to_dist(rng.standard_normal(n))
    v = pm.DistributedArray.to_dist(rng.standard_normal(n))
    assert pm.dottest(Op, u, v, rtol=1e-12)
    # offsets outside [0, nh) too: the forward is still the direct formula
    np.testing.assert_allclose(host((Op @ u).asarray()), co.convolve1d(host(u.asarray()), dims, h, off, axis),
                               rtol=1e-12, atol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", ["float64", "float32"])
@pytest.mark.parametrize("dims,axis", [((1,), 0), ((2,), 0), ((3, 7), -1), ((7, 3), 0), ((5, 1030), -1),
                                       ((4, 1023), -1), ((9, 2049), -1), ((6, 13, 3), 1), ((11, 2, 5), 0),
                                       ((3, 257, 8), 1), ((2, 5, 6), 1)])
@pytest.mark.parametrize("nh", [1, 3, 8, 41, 300])
def test_gpu_edge_shapes(pm, dt, dims, axis, nh):
    """n_axis of 1, 2, below nh and odd; rows that are not a multiple of 4 samples; long halos"""
    rng = np.random.default_rng(nh)
    n = int(np.prod(dims))
    h = rng.standard_normal(nh)
    x = rng.standard_normal(n).astype(dt)
    for off in (0, nh // 2, nh - 1):
        C = pm.local.Convolve1D(dims, h, offset=off, axis=axis, dtype=dt)
        xt = pm.DistributedArray.to_dist(x).local_array
        for adj, got in ((False, C.matvec(xt)), (True, C.rmatvec(xt))):
            want = co.convolve1d(x, dims, h, off, axis, adj)
            got = host(got)
            tol = 1e-12 if dt == "float64" else 1e-6
            assert np.linalg.norm(got - want) <= tol * max(np.linalg.norm(want), 1e-30), (off, adj)


@pytest.mark.gpu
def test_gpu_unaligned_views(pm):
    """sub-blocks of MPIBlockDiag start at arbitrary element offsets: 16-byte loads / stores must not assume
    alignment"""
    rng = np.random.default_rng(4)
    h = rng.standard_normal(9)
    dims = [(3, 37), (1,), (2, 33), (5, 4, 3)]
    axes = [-1, 0, -1, 1]
    ops = [pm.local.Convolve1D(d, h, offset=3, axis=a) for d, a in zip(dims, axes)]
    sizes = [int(np.prod(d)) for d in dims]
    x = rng.standard_normal(sum(sizes))
    y = host((pm.MPIBlockDiag(ops) @ pm.DistributedArray.to_dist(x)).asarray())
    ends = np.cumsum([0] + sizes)
    want = np.concatenate([co.convolve1d(x[ends[i]:ends[i + 1]], d, h, 3, a) for i, (d, a) in enumerate(zip(dims, axes))])
    np.testing.assert_allclose(y, want, rtol=1e-12, atol=1e-12)


@pytest.mark.gpu
def test_gpu_empty_block(pm):
    import torch
    C = pm.local.Convolve1D((0, 5), np.ones(3), axis=-1)
    assert C.matvec(torch.zeros(0, device="cuda", dtype=torch.float64)).numel() == 0
    C = pm.local.Convolve1D((4, 0), np.ones(3), axis=0)
    assert C.rmatvec(torch.zeros(0, device="cuda", dtype=torch.float64)).numel() == 0


@pytest.mark.gpu
def test_gpu_out_dtype_cast_and_complex(pm):
    import torch
    rng = np.random.default_rng(2)
    dims, h = (4, 50), rng.standard_normal(7)
    C = pm.local.Convolve1D(dims, h, offset=2, axis=-1, dtype="float64")
    x = rng.standard_normal(200)
    xt = torch.as_tensor(x, device="cuda")
    out = torch.empty(200, dtype=torch.float32, device="cuda")
    r = C.matvec(xt, out=out)
    assert r.data_ptr() == out.data_ptr() and out.dtype == torch.float32
    np.testing.assert_allclose(host(out), co.convolve1d(x, dims, h, 2), rtol=1e-6, atol=1e-6)
    # out of the operator's own dtype is written in place
    out64 = torch.empty(200, dtype=torch.float64, device="cuda")
    assert C.rmatvec(xt, out=out64).data_ptr() == out64.data_ptr()
    np.testing.assert_allclose(host(out64), co.convolve1d(x, dims, h, 2, adjoint=True), rtol=1e-12, atol=1e-12)
    # complex data stays complex: real and imaginary parts convolved alike
    for cdt in (torch.complex128, torch.complex64):
        zt = torch.as_tensor(x + 1j * rng.standard_normal(200), device="cuda").to(cdt)
        got = C.matvec(zt)
        assert got.dtype == torch.complex128           # complex data with float64 taps
        np.testing.assert_allclose(host(got), co.convolve1d(host(zt), dims, h, 2), rtol=1e-12, atol=1e-12)
    C32 = pm.local.Convolve1D(dims, h, offset=2, axis=0, dtype="complex64")
    z = (x + 1j * rng.standard_normal(200)).astype(np.complex64)
    got = C32.rmatvec(torch.as_tensor(z, device="cuda"))
    assert got.dtype == torch.complex64
    want = co.convolve1d(z, dims, h, 2, axis=0, adjoint=True)
    assert np.linalg.norm(host(got) - want) <= 1e-6 * np.linalg.norm(want)


@pytest.mark.gpu
def test_gpu_broadcast_arrays(pm):
    """MPIVStack takes a BROADCAST model (MPIBlockDiag rejects one, as in the reference) and its adjoint returns one"""
    rng = np.random.default_rng(6)
    dims, h = (3, 40), rng.standard_normal(11)
    x = rng.standard_normal(120)
    Op = pm.MPIVStack([pm.local.Convolve1D(dims, h, offset=5)])
    y = Op @ pm.DistributedArray.to_dist(x, partition=pm.Partition.BROADCAST)
    np.testing.assert_allclose(host(y.asarray()), co.convolve1d(x, dims, h, 5), rtol=1e-12, atol=1e-12)
    xa = Op.H @ pm.DistributedArray.to_dist(x)
    assert xa.partition is pm.Partition.BROADCAST
    np.testing.assert_allclose(host(xa.asarray()), co.convolve1d(x, dims, h, 5, adjoint=True), rtol=1e-12, atol=1e-12)


@pytest.mark.gpu
def test_gpu_errors(pm):
    from pylops_mpi_b200 import _lib
    import torch
    with pytest.raises(NotImplementedError):
        pm.local.Convolve1D((10,), np.ones(3) * 1j)
    with pytest.raises(NotImplementedError):
        pm.local.Convolve1D((10, 4), np.ones((4, 3)))
    with pytest.raises(NotImplementedError):
        pm.local.Convolve1D((10,), np.ones(pm.local.CONVOLVE_MAX_TAPS + 1))
    with pytest.raises(NotImplementedError):
        pm.local.Convolve1D((10,), np.ones(3), method="spectral")
    for method in (None, "direct", "fft", "overlapadd"):
        pm.local.Convolve1D((10,), np.ones(3), method=method)
    # the C entry point: over the tap limit, bad dtype, in place
    x = torch.zeros(64, dtype=torch.float64, device="cuda")
    y = torch.zeros(64, dtype=torch.float64, device="cuda")
    taps = torch.ones(pm.local.CONVOLVE_MAX_TAPS + 1, dtype=torch.float64, device="cuda")
    call = lambda xp, yp, nh, code: _lib.lib.b2_convolve1d(_lib.ctx(), xp, yp, 1, 64, 1, taps.data_ptr(), nh, 0, 0,  # noqa: E731
                                                            code, _lib.stream())
    assert call(x.data_ptr(), y.data_ptr(), pm.local.CONVOLVE_MAX_TAPS + 1, _lib.F64) == 2005     # B2_ERR_UNSUPPORTED
    assert call(x.data_ptr(), y.data_ptr(), 0, _lib.F64) == 2002                                   # B2_ERR_ARG
    assert call(x.data_ptr(), y.data_ptr(), 3, _lib.C128) == 2001                                  # B2_ERR_DTYPE
    assert call(x.data_ptr(), x.data_ptr(), 3, _lib.F64) == 2002                                   # in place
    assert call(x.data_ptr(), y.data_ptr(), pm.local.CONVOLVE_MAX_TAPS, _lib.F64) == 0
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("P", co.GRID_P)
def test_gpu_reflectivity_ista_vs_reference(pm, P):
    wav, m = co.refl_inputs(P)
    dims, wavc = co.REFL_DIMS, co.REFL_NT // 2
    DDiag = pm.MPIBlockDiag([pm.local.FirstDerivative(dims, axis=-1) for _ in range(P)])
    CDiag = pm.MPIBlockDiag([pm.local.Convolve1D(dims, wav, offset=wavc, axis=-1) for _ in range(P)])
    r = DDiag @ pm.DistributedArray.to_dist(m)
    d = CDiag @ r
    g = f"refl/P{P}/"
    GOLD.record(g + "r").check(host(r.asarray()), rtol=1e-12, atol=1e-12)
    GOLD.record(g + "d").check(host(d.asarray()), rtol=1e-12, atol=1e-12)
    x0 = pm.DistributedArray.to_dist(np.zeros(m.size))
    x, iiter, cost = pm.ista(CDiag, d, x0=x0, niter=30, eps=1e-2, alpha=float(GOLD[g + "alpha"]), tol=1e-8)
    assert iiter == int(GOLD[g + "ista_iiter"])
    np.testing.assert_allclose(np.asarray(cost), GOLD.record(g + "ista_cost").values, rtol=1e-10, atol=1e-10)
    GOLD.record(g + "ista_x").check(host(x.asarray()), rtol=1e-10, atol=1e-10)


@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 3])
def test_gpu_reflectivity_cgls_graph_vs_eager(pm, P, monkeypatch):
    from pylops_mpi_b200.optimization.cls_basic import CGLS
    wav, m = co.refl_inputs(P)
    dims, wavc = co.REFL_DIMS, co.REFL_NT // 2
    g = f"refl/P{P}/"
    DDiag = pm.MPIBlockDiag([pm.local.FirstDerivative(dims, axis=-1) for _ in range(P)])
    CDiag = pm.MPIBlockDiag([pm.local.Convolve1D(dims, wav, offset=wavc, axis=-1) for _ in range(P)])
    d = CDiag @ (DDiag @ pm.DistributedArray.to_dist(m))
    res = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("B2_CGLS_GRAPH", mode)
        solver = CGLS(CDiag)
        x = solver.setup(y=d, x0=pm.DistributedArray.to_dist(np.zeros(m.size)), niter=20, damp=0.0, tol=0.0)
        x = solver.run(x, 20)
        solver.finalize()
        if mode == "1":
            assert solver.graph_error is None, solver.graph_error
            assert solver.graph_replays >= 18
        else:
            assert solver.graph_replays == 0
        res[mode] = (host(x.asarray()), np.asarray(solver.cost))
    np.testing.assert_allclose(res["1"][0], res["0"][0], rtol=1e-12, atol=1e-13)
    np.testing.assert_allclose(res["1"][1], res["0"][1], rtol=1e-12, atol=1e-13)
    GOLD.record(g + "cgls_x").check(res["1"][0], rtol=1e-8, atol=1e-8)
    np.testing.assert_allclose(res["1"][1], GOLD.record(g + "cgls_cost").values, rtol=1e-9)


@pytest.mark.gpu
def test_two_rank_reflectivity_chain():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip(f"needs 2 GPUs, box has {torch.cuda.device_count()}")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29731",
                        os.path.join(HERE, "convolve_worker.py")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-4000:] + r.stderr[-8000:])
    assert r.stdout.count("CONVOLVE_WORKER_OK") == 2
