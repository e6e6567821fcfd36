"""Golden-vector tests.  tests/golden/reference_golden.npz was produced by the
REAL reference code (pylops-mpi, imported unmodified under the in-process MPI shim,
tests/golden/make_golden.py) and is stored compactly (tests/golden_store.py): inputs
are redrawn here from their seeds and pinned by digest, larger outputs are kept as
digest + samples + weighted sum.  Here:
  * CPU (not gpu): the oracle must reproduce every fixture -> the oracle is pinned;
  * GPU: the CUDA path (world size 1) must reproduce the gathered fixtures, and every
    entry must match the oracle (pinned to the same fixtures by the CPU tests).
"""
import ast
import math
import os
import re

import numpy as np
import pytest

import golden_store
import pylops_mpi_oracle as o

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = golden_store.Golden(os.path.join(HERE, "golden", "reference_golden.npz"))
KEYS = GOLD.keys()


def cases(prefix, depth):
    """distinct key prefixes with `depth` components under `prefix`"""
    seen = []
    for k in KEYS:
        if k.startswith(prefix + "/"):
            c = "/".join(k.split("/")[:depth])
            if c not in seen:
                seen.append(c)
    return seen


def rec(case, name):
    return GOLD.record(f"{case}/{name}")


def normal_input(seed, n, dtype):
    """input of the stencil fixtures, drawn as make_golden draws it"""
    rng = np.random.default_rng(seed)
    x = rng.normal(0, 10, n).astype(dtype)
    if np.issubdtype(dtype, np.complexfloating):
        x = x + 1j * rng.normal(0, 10, n)
    return x


FD_CASES = cases("fd", 7)
KIND = re.compile(r"([a-z]+)(\d)")


def parse_fd(case):
    _, P, dims, h, ko, e, dt = case.split("/")
    kind, order = KIND.match(ko).groups()
    return int(P[1:]), ast.literal_eval(dims), float(h[1:]), kind, int(order), bool(int(e[1:])), np.dtype(dt)


def fd_oracle(case):
    """the fixture's input (checked against the reference's) and the oracle's per-rank outputs"""
    P, dims, h, kind, order, edge, dt = parse_fd(case)
    x = normal_input(7, int(np.prod(dims)), dt)
    rec(case, "x").check(x)
    y = o.first_derivative(o.to_dist(x, P), dims, h, kind, edge, order, False, dtype=dt)
    ya = o.first_derivative(o.to_dist(x, P), dims, h, kind, edge, order, True, dtype=dt)
    return x, y, ya


def test_fixture_inventory():
    assert len(FD_CASES) == 4 * 5 * 4 * 2 * 2
    assert len(cases("array", 4)) == 16 and len(cases("stack", 4)) == 12
    assert len(cases("mm", 5)) == 30 and len(cases("fredholm", 5)) == 24
    assert "config1/y" in GOLD
    assert "array/P1/(50, 51)/ax1/r0/dot" in GOLD and "array/P1/(50, 51)/ax1/r1/dot" not in GOLD


# ---------------------------------------------------------------------------------------------
# oracle vs the real reference (CPU)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", FD_CASES)
def test_oracle_first_derivative(case):
    P, dims, h, kind, order, edge, dt = parse_fd(case)
    if case + "/reference_raises" in GOLD:
        with pytest.raises((ValueError, IndexError)):
            x = np.zeros(int(np.prod(dims)), dtype=dt)
            o.first_derivative(o.to_dist(x, P), dims, h, kind, edge, order, False, dtype=dt)
            o.first_derivative(o.to_dist(x, P), dims, h, kind, edge, order, True, dtype=dt)
        return
    x, y, ya = fd_oracle(case)
    rec(case, "y").check(y)          # same NumPy ops -> bit-exact
    rec(case, "ya").check(ya)


def config1_oracle():
    x = np.zeros((11, 21))
    x[5, 10] = 1.0
    y = np.concatenate(o.first_derivative(o.to_dist(x.ravel(), 2), (11, 21)))
    mv = lambda a: o.SimArray(o.first_derivative(a.locs, (11, 21)))                   # noqa: E731
    rmv = lambda a: o.SimArray(o.first_derivative(a.locs, (11, 21), adjoint=True))    # noqa: E731
    xo, istop, iit, r1, r2, cost = o.cgls(mv, rmv, mv(o.SimArray(o.to_dist(x.ravel(), 2))),
                                          o.SimArray([np.zeros(126), np.zeros(105)]), niter=10, tol=0.0)
    return y, xo.asarray(), istop, iit, cost


def test_oracle_config1():
    y, xo, istop, iit, cost = config1_oracle()
    GOLD.record("config1/y").check(y.reshape(11, 21))
    assert iit == int(GOLD["config1/iit"]) and istop == int(GOLD["config1/istop"])
    np.testing.assert_allclose(cost, GOLD["config1/cost"], rtol=1e-12, atol=1e-30)
    GOLD.record("config1/xinv").check(xo, rtol=1e-12, atol=1e-30)


@pytest.mark.parametrize("case", cases("array", 4))
def test_oracle_distributed_array(case):
    _, P, shape, ax = case.split("/")
    P, shape, axis = int(P[1:]), ast.literal_eval(shape), int(ax[2:])
    rng = np.random.default_rng(42)
    a = rng.normal(100, 100, shape)
    b = rng.normal(300, 300, shape)
    al, bl = o.to_dist(a, P, axis=axis), o.to_dist(b, P, axis=axis)
    mask = [r % 2 for r in range(P)]
    for r in range(P):
        g = lambda n: GOLD[f"{case}/r{r}/{n}"]   # noqa: E731
        assert tuple(g("local_shape")) == o.local_split(shape, P, r, o.SCATTER, axis)
        assert [tuple(s) for s in g("local_shapes")] == o.local_shapes(shape, P, o.SCATTER, axis)
        np.testing.assert_allclose(o.dot(al, bl)[r], g("dot"), rtol=1e-14)
        np.testing.assert_allclose(o.dot(al, bl, vdot=True)[r], g("vdot"), rtol=1e-14)
        for o_ in (1, 2, np.inf, -np.inf, 0, 3):
            np.testing.assert_allclose(o.norm(al, o_)[r], g(f"norm{o_}"), rtol=1e-14)
        np.testing.assert_allclose(o.dot([a] * P, [a] * P, partition=o.BROADCAST)[r], g("bdot"), rtol=1e-14)
        if P >= 2:
            np.testing.assert_allclose(o.dot(al, al, mask=mask)[r], g("mdot"), rtol=1e-14)
            np.testing.assert_allclose(o.norm(al, 1, mask=mask)[r], g("mnorm"), rtol=1e-14)
    rec(case, "add").check([a + b] * P)
    if f"{case}/r0/ghost" in GOLD:
        rec(case, "ghost").check(o.add_ghost_cells(al, 0, [2] * P, [1] * P))


def stack_blocks(P, ny, nx, dtype):
    blocks = [np.random.default_rng(100 + r).standard_normal((ny - r, nx)).astype(dtype) for r in range(P)]
    if np.issubdtype(dtype, np.complexfloating):
        blocks = [b + 1j * np.random.default_rng(200 + r).standard_normal(b.shape) for r, b in enumerate(blocks)]
    xg = np.random.default_rng(1).standard_normal(P * nx).astype(dtype)
    yg = np.random.default_rng(2).standard_normal(sum(ny - r for r in range(P))).astype(dtype)
    return blocks, xg, yg


def stack_oracle(case):
    _, P, shp, dt = case.split("/")
    P, (ny, nx), dtype = int(P[1:]), tuple(int(v) for v in shp.split("x")), np.dtype(dt)
    blocks, xg, yg = stack_blocks(P, ny, nx, dtype)
    bl = [[b] for b in blocks]
    y = o.blockdiag(bl, o.to_dist(xg, P))
    xa = o.blockdiag(bl, o.to_dist(yg, P), adjoint=True)
    yv = o.vstack_matvec(bl, xg[:nx])
    xv = o.vstack_rmatvec(bl, o.to_dist(yg, P))
    sblocks = []
    for r in range(P):
        A = np.ones((ny, nx), dtype=dtype) * (r + 1)
        sblocks.append([A.conj().T @ A + 1e-5 * np.eye(nx, dtype=dtype)])
    xt = np.random.default_rng(42).normal(1, 10, P * nx).astype(dtype)
    mv = lambda v: o.SimArray(o.blockdiag(sblocks, v.locs))                  # noqa: E731
    rmv = lambda v: o.SimArray(o.blockdiag(sblocks, v.locs, adjoint=True))   # noqa: E731
    xo, istop, iit, r1, r2, cost = o.cgls(mv, rmv, mv(o.SimArray(o.to_dist(xt, P))),
                                          o.SimArray(o.to_dist(np.zeros(P * nx, dtype=dtype), P)), niter=nx, tol=1e-5)
    return P, y, xa, yv, xv, (xo.locs, istop, iit, r1, r2, np.asarray(cost))


@pytest.mark.parametrize("case", cases("stack", 4))
def test_oracle_blockdiag_vstack_cgls(case):
    P, y, xa, yv, xv, (xo, istop, iit, r1, r2, cost) = stack_oracle(case)
    rec(case, "bd_y").check(y, rtol=1e-13, atol=1e-13)
    rec(case, "bd_xa").check(xa, rtol=1e-13, atol=1e-13)
    rec(case, "vs_y").check(yv, rtol=1e-13, atol=1e-13)
    rec(case, "vs_x").check([xv] * P, rtol=1e-12, atol=1e-12)
    rec(case, "cgls_x").check(xo, rtol=1e-8, atol=1e-10)
    rec(case, "cgls_cost").check([cost] * P, rtol=1e-7, atol=1e-12)
    for r in range(P):
        g = lambda n: GOLD[f"{case}/r{r}/{n}"]   # noqa: E731
        assert (iit, istop) == (int(g("cgls_iit")), int(g("cgls_istop")))
        np.testing.assert_allclose([r1, r2], [g("cgls_r1"), g("cgls_r2")], rtol=1e-6, atol=1e-14)


def mm_inputs(N, K, M, dtype):
    A = np.arange(N * K, dtype=dtype).reshape(N, K)
    X = np.arange(K * M, dtype=dtype).reshape(K, M)
    if np.issubdtype(dtype, np.complexfloating):
        A, X = A + 0.5j * A, X + 0.7j * X
    return A, X


def mm_oracle(case):
    _, P, shp, dt, kind = case.split("/")
    P, (N, K, M), dtype = int(P[1:]), tuple(int(v) for v in shp.split("x")), np.dtype(dt)
    A, X = mm_inputs(N, K, M, dtype)
    Pp = math.isqrt(P)
    rtol = 1e-5 if dtype == np.float32 else 1e-13
    if kind == "summa":
        At = o.summa_tiles(A, P)
        y = o.summa_matvec(At, [t.flatten() for t in o.summa_tiles(X, P)], N, K, M, dtype=dtype)
        xa = o.summa_matvec(At, y, N, K, M, dtype=dtype, adjoint=True)
    else:
        blk, bc = int(math.ceil(N / Pp)), int(math.ceil(M / Pp))
        Arows = [A[(r % Pp) * blk:min(N, (r % Pp + 1) * blk)] for r in range(P)]
        Xc = [X[:, (r // Pp) * bc:min(M, (r // Pp + 1) * bc)].flatten() for r in range(P)]
        y = o.blockmm_matvec(Arows, Xc, N, K, M, dtype=dtype)
        xa = o.blockmm_matvec(Arows, y, N, K, M, dtype=dtype, adjoint=True)
    return y, xa, rtol


@pytest.mark.parametrize("case", cases("mm", 5))
def test_oracle_matrixmult(case):
    y, xa, rtol = mm_oracle(case)
    rec(case, "y").check(y, rtol=rtol)
    rec(case, "xa").check(xa, rtol=rtol * 10)


def fredholm_inputs(nz, dtype):
    nsl, nx, ny = 21, 4, 6
    rng = np.random.default_rng(5)
    G = rng.standard_normal((nsl, nx, ny))
    if np.issubdtype(dtype, np.complexfloating):
        G = G + 1j * rng.standard_normal((nsl, nx, ny))
    x = np.random.default_rng(6).standard_normal(nsl * ny * nz).astype(dtype)
    return G.astype(dtype), x


def fredholm_oracle(case):
    _, P, nz, dt, flags = case.split("/")
    P, nz, dtype = int(P[1:]), int(nz[2:]), np.dtype(dt)
    G, x = fredholm_inputs(nz, dtype)
    ext = [o.local_split((21,), P, r)[0] for r in range(P)]
    off = np.cumsum([0] + ext)
    G_loc = [G[off[r]:off[r + 1]] for r in range(P)]
    y = o.fredholm1(G_loc, x, nz)
    return y, o.fredholm1(G_loc, y, nz, adjoint=True)


@pytest.mark.parametrize("case", cases("fredholm", 5))
def test_oracle_fredholm(case):
    y, xa = fredholm_oracle(case)
    rec(case, "y").check(y, rtol=1e-13, atol=1e-13)
    rec(case, "xa").check(xa, rtol=1e-12, atol=1e-12)


# ---------------------------------------------------------------------------------------------
# CUDA path vs the real reference (GPU, world size 1: gathered fixtures)
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pm():
    import pylops_mpi_b200 as pm
    return pm


def host(t):
    return t.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in FD_CASES if c + "/reference_raises" not in KEYS])
def test_gpu_first_derivative_vs_reference(pm, case):
    P, dims, h, kind, order, edge, dt = parse_fd(case)
    x, oy, oya = fd_oracle(case)
    Fop = pm.MPIFirstDerivative(dims, sampling=h, kind=kind, edge=edge, order=order, dtype=dt)
    xd = pm.DistributedArray.to_dist(x)
    y, ya = host((Fop @ xd).asarray()), host((Fop.H @ xd).asarray())
    tol = dict(rtol=1e-12, atol=1e-12)
    rec(case, "y").check(y, **tol)
    rec(case, "ya").check(ya, **tol)
    np.testing.assert_allclose(y, np.concatenate(oy), **tol)
    np.testing.assert_allclose(ya, np.concatenate(oya), **tol)


@pytest.mark.gpu
def test_gpu_config1_vs_reference(pm):
    x = np.zeros((11, 21))
    x[5, 10] = 1.0
    Fop = pm.MPIFirstDerivative((11, 21), dtype=np.float64)
    y = Fop @ pm.DistributedArray.to_dist(x.ravel())
    GOLD.record("config1/y").check(host(y.asarray()).reshape(11, 21))
    xinv, istop, iit, r1, r2, cost = pm.cgls(Fop, y, x0=pm.DistributedArray.to_dist(np.zeros(231)), niter=10, tol=0.0)
    assert iit == int(GOLD["config1/iit"])
    np.testing.assert_allclose(cost, GOLD["config1/cost"], rtol=1e-6, atol=1e-12)
    GOLD.record("config1/xinv").check(host(xinv.asarray()), rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(host(xinv.asarray()), config1_oracle()[1], rtol=1e-6, atol=1e-9)


@pytest.mark.gpu
@pytest.mark.parametrize("case", cases("stack", 4))
def test_gpu_blockdiag_vstack_cgls_vs_reference(pm, case):
    _, P, shp, dt = case.split("/")
    P, (ny, nx), dtype = int(P[1:]), tuple(int(v) for v in shp.split("x")), np.dtype(dt)
    blocks, xg, yg = stack_blocks(P, ny, nx, dtype)
    ops = [pm.MatrixMult(b) for b in blocks]                     # all P blocks on the one rank
    BD = pm.MPIBlockDiag(ops)
    _, oy, oxa, oyv, oxv, (oxo, *_o) = stack_oracle(case)
    t12 = dict(rtol=1e-12, atol=1e-12)
    for name, got, want in (("bd_y", host((BD @ pm.DistributedArray.to_dist(xg)).asarray()), oy),
                            ("bd_xa", host((BD.H @ pm.DistributedArray.to_dist(yg)).asarray()), oxa)):
        rec(case, name).check(got, **t12)
        np.testing.assert_allclose(got, np.concatenate(want), **t12)
    VS = pm.MPIVStack(ops)
    xb = pm.DistributedArray.to_dist(xg[:nx], partition=pm.Partition.BROADCAST)
    got = host((VS @ xb).asarray())
    rec(case, "vs_y").check(got, **t12)
    np.testing.assert_allclose(got, np.concatenate(oyv), **t12)
    got = host((VS.H @ pm.DistributedArray.to_dist(yg)).asarray())
    rec(case, "vs_x").check([got] * P, rtol=1e-11, atol=1e-11)
    np.testing.assert_allclose(got, oxv, rtol=1e-11, atol=1e-11)
    sops = []
    for r in range(P):
        A = np.ones((ny, nx), dtype=dtype) * (r + 1)
        sops.append(pm.MatrixMult(A.conj().T @ A + 1e-5 * np.eye(nx, dtype=dtype)))
    Sop = pm.MPIBlockDiag(sops)
    xt = np.random.default_rng(42).normal(1, 10, P * nx).astype(dtype)
    yy = Sop @ pm.DistributedArray.to_dist(xt)
    xinv, istop, iit, r1, r2, cost = pm.cgls(Sop, yy, x0=pm.DistributedArray.to_dist(np.zeros(P * nx, dtype=dtype)),
                                             niter=nx, tol=1e-5)
    assert (iit, istop) == (int(GOLD[f"{case}/r0/cgls_iit"]), int(GOLD[f"{case}/r0/cgls_istop"]))
    rec(case, "cgls_x").check(host(xinv.asarray()), rtol=1e-6, atol=1e-8)
    np.testing.assert_allclose(host(xinv.asarray()), np.concatenate(oxo), rtol=1e-6, atol=1e-8)
    rec(case, "cgls_cost").check([np.asarray(cost)] * P, rtol=1e-5, atol=1e-8)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in cases("mm", 5) if c.split("/")[1] == "P1"])
def test_gpu_matrixmult_vs_reference(pm, case):
    _, P, shp, dt, kind = case.split("/")
    (N, K, M), dtype = tuple(int(v) for v in shp.split("x")), np.dtype(dt)
    A, X = mm_inputs(N, K, M, dtype)
    Aop = pm.MPIMatrixMult(A, M, kind=kind, dtype=dtype)
    y = Aop @ pm.DistributedArray.to_dist(X.ravel())
    oy, oxa, rtol = mm_oracle(case)
    got, gota = host(y.asarray()), host((Aop.H @ y).asarray())
    rec(case, "y").check(got, rtol=rtol)
    rec(case, "xa").check(gota, rtol=rtol * 10)
    np.testing.assert_allclose(got, oy[0], rtol=rtol)
    np.testing.assert_allclose(gota, oxa[0], rtol=rtol * 10)


@pytest.mark.gpu
@pytest.mark.parametrize("case", cases("fredholm", 5))
def test_gpu_fredholm_vs_reference(pm, case):
    _, P, nz, dt, flags = case.split("/")
    nz, dtype = int(nz[2:]), np.dtype(dt)
    G, x = fredholm_inputs(nz, dtype)
    Fop = pm.MPIFredholm1(G, nz=nz, dtype=dtype)
    y = Fop @ pm.DistributedArray.to_dist(x, partition=pm.Partition.BROADCAST)
    oy, oxa = fredholm_oracle(case)
    got, gota = host(y.asarray()), host((Fop.H @ y).asarray())
    rec(case, "y").check(got, rtol=1e-12, atol=1e-12)
    rec(case, "xa").check(gota, rtol=1e-11, atol=1e-11)
    np.testing.assert_allclose(got, oy, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(gota, oxa, rtol=1e-11, atol=1e-11)


# ---------------------------------------------------------------------------------------------
# "next" row f2: MPISecondDerivative -- oracle and CUDA path vs the real reference
# ---------------------------------------------------------------------------------------------
SD_CASES = cases("sd", 7)


def parse_sd(case):
    _, P, dims, h, kind, e, dt = case.split("/")
    return int(P[1:]), ast.literal_eval(dims), float(h[1:]), kind, bool(int(e[1:])), np.dtype(dt)


def sd_oracle(case):
    P, dims, h, kind, edge, dt = parse_sd(case)
    x = normal_input(9, int(np.prod(dims)), dt)
    rec(case, "x").check(x)
    y = o.second_derivative(o.to_dist(x, P), dims, h, kind, edge, False, dtype=dt)
    ya = o.second_derivative(o.to_dist(x, P), dims, h, kind, edge, True, dtype=dt)
    return x, y, ya


@pytest.mark.parametrize("case", SD_CASES)
def test_oracle_second_derivative(case):
    P, dims, h, kind, edge, dt = parse_sd(case)
    if case + "/reference_raises" in GOLD:
        with pytest.raises((ValueError, IndexError)):
            x = np.zeros(int(np.prod(dims)), dtype=dt)
            o.second_derivative(o.to_dist(x, P), dims, h, kind, edge, False, dtype=dt)
            o.second_derivative(o.to_dist(x, P), dims, h, kind, edge, True, dtype=dt)
        return
    x, y, ya = sd_oracle(case)
    rec(case, "y").check(y)
    rec(case, "ya").check(ya)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in SD_CASES if c + "/reference_raises" not in KEYS])
def test_gpu_second_derivative_vs_reference(pm, case):
    P, dims, h, kind, edge, dt = parse_sd(case)
    x, oy, oya = sd_oracle(case)
    Sop = pm.MPISecondDerivative(dims, sampling=h, kind=kind, edge=edge, dtype=dt)
    xd = pm.DistributedArray.to_dist(x)
    y, ya = host((Sop @ xd).asarray()), host((Sop.H @ xd).asarray())
    tol = dict(rtol=1e-12, atol=1e-11)
    rec(case, "y").check(y, **tol)
    rec(case, "ya").check(ya, **tol)
    np.testing.assert_allclose(y, np.concatenate(oy), **tol)
    np.testing.assert_allclose(ya, np.concatenate(oya), **tol)


@pytest.mark.gpu
@pytest.mark.parametrize("dims,axes", [((20, 17), (0, 1)), ((12, 9, 10), (0, 1, 2)), ((12, 9, 10), (-2, -1)), ((31,), (0,))])
@pytest.mark.parametrize("kind,edge", [("centered", False), ("centered", True), ("forward", False), ("backward", False)])
@pytest.mark.parametrize("dtype", [np.float64, np.complex128, np.float32])
def test_gpu_laplacian_and_local_derivatives(pm, dims, axes, kind, edge, dtype):
    rng = np.random.default_rng(5)
    n = int(np.prod(dims))
    x = rng.standard_normal(n).astype(dtype)
    if np.issubdtype(dtype, np.complexfloating):
        x = x + 1j * rng.standard_normal(n)
    weights = tuple(1.0 + 0.5 * i for i in range(len(axes)))
    sampling = tuple(1.0 + 0.25 * i for i in range(len(axes)))
    Lop = pm.MPILaplacian(dims, axes=axes, weights=weights, sampling=sampling, kind=kind, edge=edge, dtype=dtype)
    X = x.reshape(dims)
    ref = np.zeros(dims, dtype=np.complex128 if np.iscomplexobj(x) else np.float64)
    refa = np.zeros_like(ref)
    for ax, w, s in zip(axes, weights, sampling):
        D = o.second_derivative_dense(dims[ax], s, kind, edge)
        ref += w * o.derivative_along_axis(X, ax % len(dims), D)
        refa += w * o.derivative_along_axis(X, ax % len(dims), D.T)
    tol = dict(rtol=2e-4, atol=2e-4) if dtype == np.float32 else dict(rtol=1e-11, atol=1e-11)
    xd = pm.DistributedArray.to_dist(x)
    np.testing.assert_allclose(host((Lop @ xd).asarray()), ref.ravel(), **tol)
    np.testing.assert_allclose(host((Lop.H @ xd).asarray()), refa.ravel(), **tol)
    if dtype != np.float32:
        u = pm.DistributedArray.to_dist(rng.standard_normal(n).astype(dtype))
        v = pm.DistributedArray.to_dist(rng.standard_normal(n).astype(dtype))
        assert pm.dottest(Lop, u, v)
    # rank-local first derivatives along every axis (the MPIGradient building block)
    for ax in range(len(dims)):
        for k2, order in (("centered", 3), ("centered", 5), ("forward", 3)):
            if dims[ax] < 6:
                continue
            F = pm.local.FirstDerivative(dims, axis=ax, sampling=0.5, kind=k2, edge=edge, order=order, dtype=dtype)
            D1 = o.first_derivative_dense(dims[ax], 0.5, k2, edge, order)
            xt = torch_from(x)
            np.testing.assert_allclose(host(F.matvec(xt)), o.derivative_along_axis(X, ax, D1).ravel(), **tol)
            np.testing.assert_allclose(host(F.rmatvec(xt)), o.derivative_along_axis(X, ax, D1.T).ravel(), **tol)


def torch_from(a):
    import torch
    return torch.as_tensor(a).cuda()


# ---------------------------------------------------------------------------------------------
# "next" rows: MPIGradient / MPILaplacian -- the reference's glue (StackedDistributedArray, MPIStackedVStack,
# MPIBlockDiag re-partition, operator algebra) run over refshim's restated rank-local stencils
# ---------------------------------------------------------------------------------------------
GRAD_CASES = cases("grad", 5)
LAP_CASES = cases("lap", 8)


def parse_grad(case):
    _, P, dims, kind, e = case.split("/")
    dims = ast.literal_eval(dims)
    samp = {2: (1.0, 0.5), 3: (0.4, 1.0, 2.0)}[len(dims)]
    return int(P[1:]), dims, samp, kind, bool(int(e[1:]))


def parse_lap(case):
    _, P, dims, axes, weights, samp, kind, e = case.split("/")
    return (int(P[1:]), ast.literal_eval(dims), ast.literal_eval(axes), ast.literal_eval(weights),
            ast.literal_eval(samp), kind, bool(int(e[1:])))


def test_next_fixture_inventory():
    assert len(GRAD_CASES) == 3 * 2 * 4 and len(LAP_CASES) == 3 * 4 * 3


def grad_oracle(case):
    P, dims, samp, kind, edge = parse_grad(case)
    x = normal_input(13, int(np.prod(dims)), np.float64)
    rec(case, "x").check([x] * P)
    y = o.gradient(o.to_dist(x, P), dims, samp, kind, edge)
    return x, y, o.gradient_adjoint(y, dims, samp, kind, edge)


@pytest.mark.parametrize("case", GRAD_CASES)
def test_oracle_gradient(case):
    P, dims, samp, kind, edge = parse_grad(case)
    x, y, xa = grad_oracle(case)
    for ax in range(len(dims)):
        rec(case, f"y{ax}").check(y[ax], rtol=1e-13, atol=1e-12)
    rec(case, "xa").check(xa, rtol=1e-13, atol=1e-11)
    flat = np.concatenate([np.concatenate(a) for a in y])
    np.testing.assert_allclose(np.dot(flat, flat), GOLD[case + "/r0/dot"], rtol=1e-13)
    np.testing.assert_allclose(np.linalg.norm(flat), GOLD[case + "/r0/norm"], rtol=1e-13)


def lap_oracle(case):
    P, dims, axes, weights, samp, kind, edge = parse_lap(case)
    x = normal_input(14, int(np.prod(dims)), np.float64)
    rec(case, "x").check([x] * P)
    y = o.laplacian(o.to_dist(x, P), dims, axes, weights, samp, kind, edge, False)
    ya = o.laplacian(o.to_dist(x, P), dims, axes, weights, samp, kind, edge, True)
    return x, y, ya


@pytest.mark.parametrize("case", LAP_CASES)
def test_oracle_laplacian(case):
    x, y, ya = lap_oracle(case)
    rec(case, "y").check(y, rtol=1e-13, atol=1e-11)
    rec(case, "ya").check(ya, rtol=1e-13, atol=1e-11)


@pytest.mark.gpu
@pytest.mark.parametrize("case", GRAD_CASES)
def test_gpu_gradient_vs_reference(pm, case):
    P, dims, samp, kind, edge = parse_grad(case)
    x, oy, oxa = grad_oracle(case)
    Gop = pm.MPIGradient(dims, sampling=samp, kind=kind, edge=edge, dtype=np.float64)
    y = Gop.matvec(pm.DistributedArray.to_dist(x))
    for ax in range(len(dims)):
        got = host(y[ax].asarray())
        rec(case, f"y{ax}").check(got, rtol=1e-12, atol=1e-11)
        np.testing.assert_allclose(got, np.concatenate(oy[ax]), rtol=1e-12, atol=1e-11)
    got = host(Gop.rmatvec(y).asarray())
    rec(case, "xa").check(got, rtol=1e-12, atol=1e-10)
    np.testing.assert_allclose(got, np.concatenate(oxa), rtol=1e-12, atol=1e-10)
    np.testing.assert_allclose(y.dot(y), GOLD[case + "/r0/dot"], rtol=1e-12)
    np.testing.assert_allclose(y.norm(), GOLD[case + "/r0/norm"], rtol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("case", LAP_CASES)
def test_gpu_laplacian_vs_reference(pm, case):
    P, dims, axes, weights, samp, kind, edge = parse_lap(case)
    x, oy, oya = lap_oracle(case)
    Lop = pm.MPILaplacian(dims, axes=axes, weights=weights, sampling=samp, kind=kind, edge=edge, dtype=np.float64)
    xd = pm.DistributedArray.to_dist(x)
    tol = dict(rtol=1e-12, atol=1e-10)
    for name, got, want in (("y", host((Lop @ xd).asarray()), oy), ("ya", host((Lop.H @ xd).asarray()), oya)):
        rec(case, name).check(got, **tol)
        np.testing.assert_allclose(got, np.concatenate(want), **tol)


# ---------------------------------------------------------------------------------------------
# "next" row: ISTA / FISTA -- the reference's solver loops (cls_sparsity.py) over refshim's restated thresholds
# ---------------------------------------------------------------------------------------------
SPARSE_CASES = cases("sparse", 5)


def sparse_inputs(case):
    """same construction as make_golden.t_sparse"""
    _, P, solver, kind, dt = case.split("/")
    P, dtype = int(P[1:]), np.dtype(dt).type
    eps = {"soft": 0.5, "hard": 0.05, "half": 0.2}[kind]
    rng = np.random.default_rng(21)
    ny, nx = 13, 11
    blocks = []
    for r in range(P):
        A = rng.standard_normal((ny, nx))
        if np.issubdtype(dtype, np.complexfloating):
            A = A + 1j * rng.standard_normal((ny, nx))
        blocks.append(A.astype(dtype))
    xtrue = np.zeros(P * nx, dtype=dtype)
    k = max(2, P * nx // 5)
    xtrue[rng.permutation(P * nx)[:k]] = rng.standard_normal(k) * 3
    lam = max(np.linalg.norm(b, 2) ** 2 for b in blocks)
    return P, solver, kind, dtype, eps, blocks, xtrue, lam


def test_sparse_inventory():
    assert len(SPARSE_CASES) == 3 * 2 * 5


@pytest.mark.parametrize("case", SPARSE_CASES)
def test_oracle_ista_fista(case):
    import scipy.linalg
    P, solver, kind, dtype, eps, blocks, xtrue, lam = sparse_inputs(case)
    np.testing.assert_allclose(lam, GOLD[case + "/lam"], rtol=1e-6)
    A = scipy.linalg.block_diag(*blocks).astype(dtype)
    y = A @ xtrue
    x, iiter, cost = o.ista(A, y, np.zeros_like(xtrue), 40, eps, 1.0 / float(GOLD[case + "/lam"]), 1e-10, kind,
                            fista=(solver == "fista"))
    tol = 5e-4 if dtype == np.float32 else 1e-9
    assert iiter == int(GOLD[case + "/iiter"])
    np.testing.assert_allclose(cost, GOLD[case + "/cost"], rtol=tol)
    np.testing.assert_allclose(x, GOLD[case + "/x"], rtol=tol, atol=tol)
    eig = o.power_iteration(A.conj().T @ A, 300, 1e-13)[0]
    np.testing.assert_allclose(np.abs(eig), GOLD[case + "/maxeig"], rtol=1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("case", SPARSE_CASES)
def test_gpu_ista_fista_vs_reference(pm, case):
    P, solver, kind, dtype, eps, blocks, xtrue, lam = sparse_inputs(case)
    # one rank here: all P blocks stacked in this rank's MPIBlockDiag (same global operator, row-block layout)
    Op = pm.MPIBlockDiag([pm.local.MatrixMult(torch_from(b), dtype=dtype) for b in blocks])
    y = Op @ pm.DistributedArray.to_dist(xtrue)
    x0 = pm.DistributedArray.to_dist(np.zeros_like(xtrue))
    fn = pm.ista if solver == "ista" else pm.fista
    alpha = 1.0 / float(GOLD[case + "/lam"])
    x, iiter, cost = fn(Op, y, x0, niter=40, eps=eps, alpha=alpha, tol=1e-10, threshkind=kind)
    tol = 2e-3 if dtype == np.float32 else 1e-9
    assert iiter == int(GOLD[case + "/iiter"])
    np.testing.assert_allclose(cost, GOLD[case + "/cost"], rtol=tol)
    np.testing.assert_allclose(host(x.asarray()), GOLD[case + "/x"], rtol=tol, atol=tol)
    # generic (unfused) execution mode gives the same numbers: SOp = identity operator
    Iop = pm.MPIBlockDiag([pm.local.Identity(len(xtrue), dtype=dtype)])
    x2, iiter2, cost2 = fn(Op, y, x0, niter=40, SOp=Iop, eps=eps, alpha=alpha, tol=1e-10, threshkind=kind)
    assert iiter2 == iiter
    np.testing.assert_allclose(cost2, cost, rtol=tol)
    np.testing.assert_allclose(host(x2.asarray()), host(x.asarray()), rtol=tol, atol=tol)
    # step size from the power iteration (alpha=None)
    eig = pm.power_iteration(Op.H @ Op, niter=300, tol=1e-13, dtype=dtype,
                             b_k=pm.DistributedArray(global_shape=len(xtrue), dtype=dtype))[0]
    np.testing.assert_allclose(np.abs(eig), GOLD[case + "/maxeig"], rtol=1e-3)


# ---------------------------------------------------------------------------------------------
# "next" row f1: MPIMDC -- the reference's chain (MDC.py) over refshim's restated pylops FFT / Identity
# ---------------------------------------------------------------------------------------------
MDC_CASES = cases("mdc", 5)


def mdc_inputs(case):
    _, P, t, dt, cp = case.split("/")
    P, twosided, conj, prescaled = int(P[1:]), bool(int(t[1:])), bool(int(cp[1])), bool(int(cp[3]))
    dtype = np.dtype(dt)
    rng = np.random.default_rng(31)          # drawn as make_golden.t_mdc draws them
    ns, nr, nv, nt = 6, 5, 3, (31 if twosided else 32)
    nf = int(np.ceil((nt + 1) / 2)) - 3
    G = (rng.standard_normal((nf, ns, nr)) + 1j * rng.standard_normal((nf, ns, nr))).astype(dtype)
    rdt = np.real(np.ones(1, dtype)).dtype
    m = rng.standard_normal(nt * nr * nv).astype(rdt)
    d = rng.standard_normal(nt * ns * nv).astype(rdt)
    for name, a in (("G", G), ("m", m), ("d", d)):
        rec(case, name).check(a)
    off = np.cumsum([0] + [nf // P + (1 if r < nf % P else 0) for r in range(P)])
    return P, twosided, conj, prescaled, G, m, d, nt, off


def test_mdc_inventory():
    assert len(MDC_CASES) == 3 * 2 * 3


def mdc_oracle(case):
    P, twosided, conj, prescaled, G, m, d, nt, off = mdc_inputs(case)
    Gl = [G[off[r]:off[r + 1]].astype(np.complex128) for r in range(P)]
    kw = dict(dt=0.004, dr=2.0, prescaled=prescaled, conj=conj)
    return o.mdc(Gl, m.astype(np.float64), nt, 3, twosided, False, **kw), o.mdc(Gl, d.astype(np.float64), nt, 3, twosided, True, **kw)


@pytest.mark.parametrize("case", MDC_CASES)
def test_oracle_mdc(case):
    G = mdc_inputs(case)[4]
    y, xa = mdc_oracle(case)
    gy, gxa = rec(case, "y"), rec(case, "xa")
    assert gy.imag_zero and gxa.imag_zero
    tol = 2e-6 if G.dtype == np.complex64 else 1e-13
    gy.check(y, rtol=tol, atol=tol * gy.amax)
    gxa.check(xa, rtol=tol, atol=tol * gxa.amax)


@pytest.mark.gpu
@pytest.mark.parametrize("case", MDC_CASES)
def test_gpu_mdc_vs_reference(pm, case):
    P, twosided, conj, prescaled, G, m, d, nt, off = mdc_inputs(case)
    Mop = pm.MPIMDC(G, nt=nt, nv=3, nfreq=G.shape[0], dt=0.004, dr=2.0, twosided=twosided, conj=conj, prescaled=prescaled)
    y = Mop @ pm.DistributedArray.to_dist(m, partition=pm.Partition.BROADCAST)
    xa = Mop.H @ pm.DistributedArray.to_dist(d, partition=pm.Partition.BROADCAST)
    oy, oxa = mdc_oracle(case)
    tol = 2e-4 if G.dtype == np.complex64 else 1e-11
    for name, got, want in (("y", host(y.asarray()).real, oy), ("xa", host(xa.asarray()).real, oxa)):
        g = rec(case, name)
        g.check(got, rtol=tol, atol=tol * g.amax)
        np.testing.assert_allclose(got, want, rtol=tol, atol=tol * g.amax)
