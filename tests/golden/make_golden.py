"""Generate golden fixtures by running the REAL reference (a pylops-mpi source
checkout, imported unmodified) under the in-process MPI shim in tests/golden/refshim/.

    PYLOPS_MPI_REFERENCE=<pylops-mpi checkout> python tests/golden/make_golden.py
                                                  # writes tests/golden/reference_golden.npz

Needs the reference checkout; the tests do not.  The .npz it writes (in the compact
form of tests/golden_store.py) is committed and is what tests/test_golden.py checks
the oracle and the CUDA path against.  Third-party ``pylops`` is absent from the image.  On
the hot path its only arithmetic (the dense block ``A @ x``) is restated in
refshim/pylops; mpi4py is replaced by threads.  Everything else -- partition
bookkeeping, @reshaped, ghost cells, the stencils, BlockDiag/VStack/MatrixMult/
Fredholm1, dot/norm, CGLS, dottest -- is the reference's own code.
For the "next" rows more of pylops had to be restated (published formulas, marked
as such in refshim/pylops): the rank-local First/SecondDerivative used by
MPIGradient/MPILaplacian, the soft/hard/half thresholds used by ISTA/FISTA, and
the numpy FFT / Identity used by MPIMDC; the distributed glue and the solver
loops around them are still the reference's own code.
Not reproducible bit for bit: ``sparse/*/maxeig`` (the reference's power iteration
draws its start vector from the process-global NumPy RNG, which the rank threads
share); tests compare it with rtol 1e-3 only.
"""
import importlib
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("PYLOPS_MPI_REFERENCE", "")
sys.path.insert(0, os.path.join(HERE, "refshim"))
sys.path.insert(0, os.path.dirname(HERE))
import golden_store  # noqa: E402


def load_reference():
    pkg = types.ModuleType("pylops_mpi")
    pkg.__path__ = [os.path.join(REF, "pylops_mpi")]
    sys.modules["pylops_mpi"] = pkg
    da = importlib.import_module("pylops_mpi.DistributedArray")
    pkg.DistributedArray, pkg.Partition = da.DistributedArray, da.Partition
    pkg.StackedDistributedArray = da.StackedDistributedArray
    lo = importlib.import_module("pylops_mpi.LinearOperator")
    pkg.MPILinearOperator, pkg.asmpilinearoperator = lo.MPILinearOperator, lo.asmpilinearoperator
    slo = importlib.import_module("pylops_mpi.StackedLinearOperator")
    pkg.MPIStackedLinearOperator = slo.MPIStackedLinearOperator
    # sub-packages: register bare namespaces so their __init__ (which pulls in operators that need
    # more of third-party pylops than this path uses) is not executed
    for sub in ("basicoperators", "signalprocessing", "optimization", "waveeqprocessing"):
        m = types.ModuleType("pylops_mpi." + sub)
        m.__path__ = [os.path.join(REF, "pylops_mpi", sub)]
        sys.modules["pylops_mpi." + sub] = m
        setattr(pkg, sub, m)
    mods = {}
    for name in ("basicoperators.FirstDerivative", "basicoperators.SecondDerivative", "basicoperators.BlockDiag", "basicoperators.VStack",
                 "basicoperators.MatrixMult", "signalprocessing.Fredholm1", "optimization.cls_basic",
                 "utils.dottest"):
        mods[name.split(".")[-1]] = importlib.import_module("pylops_mpi." + name)
    bo = sys.modules["pylops_mpi.basicoperators"]
    bo.MPIBlockDiag, bo.MPISecondDerivative = mods["BlockDiag"].MPIBlockDiag, mods["SecondDerivative"].MPISecondDerivative
    for name in ("basicoperators.Gradient", "basicoperators.Laplacian", "optimization.eigs", "optimization.cls_sparsity",
                 "waveeqprocessing.MDC"):  # "next" rows: the reference's own glue over
        mods[name.split(".")[-1]] = importlib.import_module("pylops_mpi." + name)  # refshim/pylops/_derivatives.py
    return pkg, mods


def main():
    if not os.path.isdir(os.path.join(REF, "pylops_mpi")):
        raise SystemExit("set PYLOPS_MPI_REFERENCE to a pylops-mpi source checkout")
    from mpi4py import MPI
    import pylops
    pkg, mods = load_reference()
    DA, Partition = pkg.DistributedArray, pkg.Partition
    FD = mods["FirstDerivative"].MPIFirstDerivative
    SD = mods["SecondDerivative"].MPISecondDerivative
    BD = mods["BlockDiag"].MPIBlockDiag
    VS = mods["VStack"].MPIVStack
    MM = mods["MatrixMult"]
    FR = mods["Fredholm1"].MPIFredholm1
    CGLS = mods["cls_basic"].CGLS
    dottest = mods["dottest"].dottest
    out = {}

    def put(key, val):
        out[key] = np.asarray(val)

    # ---- DistributedArray: partition, dot, norm, masks, ghost cells -----------------------------
    def t_array(rank, P, shape, axis):
        rng = np.random.default_rng(42)
        a = rng.normal(100, 100, shape)
        b = rng.normal(300, 300, shape)
        A = DA.to_dist(a, axis=axis)
        B = DA.to_dist(b, axis=axis)
        res = {"local_shape": A.local_shape, "local_shapes": A.local_shapes, "dot": A.dot(B), "vdot": A.dot(B, vdot=True),
               "add": (A + B).asarray(), "mul": (A * B).asarray()}
        for o_ in (1, 2, np.inf, -np.inf, 0, 3):
            res[f"norm{o_}"] = A.norm(o_)
        Bc = DA.to_dist(a, partition=Partition.BROADCAST)
        res["bdot"] = Bc.dot(Bc)
        if P >= 2:
            mask = [r % 2 for r in range(P)]
            Am = DA.to_dist(a, axis=axis, mask=mask)
            res["mdot"] = Am.dot(Am)
            res["mnorm"] = Am.norm(1)
        if axis == 0 and min(A.local_shapes)[0] >= 2:
            res["ghost"] = A.add_ghost_cells(cells_front=2, cells_back=1)
        return res

    for P in (1, 2, 3, 4):
        for shape, axis in (((50, 51), 1), ((51, 50), 0), ((20, 21, 11), 1), ((600,), 0)):
            for r, res in enumerate(MPI.run_world(P, t_array, P, shape, axis)):
                for k, v in res.items():
                    put(f"array/P{P}/{shape}/ax{axis}/r{r}/{k}", v)

    # ---- MPIFirstDerivative ---------------------------------------------------------------------------
    def t_fd(rank, dims, h, kind, edge, order, dtype):
        rng = np.random.default_rng(7)
        n = int(np.prod(dims))
        x = rng.normal(0, 10, n).astype(dtype)
        if np.issubdtype(dtype, np.complexfloating):
            x = x + 1j * rng.normal(0, 10, n)
        Fop = FD(dims, sampling=h, kind=kind, edge=edge, order=order, dtype=dtype)
        xd = DA.to_dist(x)
        y = Fop @ xd
        ya = Fop.H @ xd
        u = DA.to_dist(rng.normal(0, 10, n).astype(dtype))
        v = DA.to_dist(rng.normal(0, 10, n).astype(dtype))
        return {"x": x, "y_local": y.local_array, "ya_local": ya.local_array, "dottest": dottest(Fop, u, v)}

    for P in (1, 2, 3, 4):
        for dims, h in (((11, 21), 1.0), ((13,), 1.0), ((30, 17), 0.4), ((29, 5, 3), 0.4), ((600,), 1.0)):
            for kind, order in (("forward", 3), ("backward", 3), ("centered", 3), ("centered", 5)):
                for edge in (False, True):
                    for dtype in (np.float64, np.complex128):
                        key = f"fd/P{P}/{dims}/h{h}/{kind}{order}/e{int(edge)}/{np.dtype(dtype).name}"
                        try:
                            res = MPI.run_world(P, t_fd, dims, h, kind, edge, order, dtype)
                        except (ValueError, IndexError) as exc:
                            put(key + "/reference_raises", type(exc).__name__)
                            continue
                        put(key + "/x", res[0]["x"])
                        for r, d in enumerate(res):
                            put(key + f"/r{r}/y", d["y_local"])
                            put(key + f"/r{r}/ya", d["ya_local"])
                            assert d["dottest"]

    # ---- MPISecondDerivative ("next" row f2) ---------------------------------------------------------------
    def t_sd(rank, dims, h, kind, edge, dtype):
        rng = np.random.default_rng(9)
        n = int(np.prod(dims))
        x = rng.normal(0, 10, n).astype(dtype)
        if np.issubdtype(dtype, np.complexfloating):
            x = x + 1j * rng.normal(0, 10, n)
        Sop = SD(dims, sampling=h, kind=kind, edge=edge, dtype=dtype)
        xd = DA.to_dist(x)
        y = Sop @ xd
        ya = Sop.H @ xd
        u = DA.to_dist(rng.normal(0, 10, n).astype(dtype))
        v = DA.to_dist(rng.normal(0, 10, n).astype(dtype))
        return {"x": x, "y_local": y.local_array, "ya_local": ya.local_array, "dottest": dottest(Sop, u, v)}

    for P in (1, 2, 3, 4):
        for dims, h in (((11, 21), 1.0), ((13,), 1.0), ((30, 17), 0.4), ((29, 5, 3), 0.4), ((600,), 1.0)):
            for kind in ("forward", "backward", "centered"):
                for edge in (False, True):
                    for dtype in (np.float64, np.complex128):
                        key = f"sd/P{P}/{dims}/h{h}/{kind}/e{int(edge)}/{np.dtype(dtype).name}"
                        try:
                            res = MPI.run_world(P, t_sd, dims, h, kind, edge, dtype)
                        except (ValueError, IndexError) as exc:
                            put(key + "/reference_raises", type(exc).__name__)
                            continue
                        put(key + "/x", res[0]["x"])
                        for r, d in enumerate(res):
                            put(key + f"/r{r}/y", d["y_local"])
                            put(key + f"/r{r}/ya", d["ya_local"])
                            assert d["dottest"]

    # config 1 (README.md:73-94) incl. dottest + cgls(niter=10)
    def t_config1(rank):
        x = np.zeros((11, 21))
        x[5, 10] = 1.0
        Fop = FD((11, 21), dtype=np.float64)
        xd = DA.to_dist(x.ravel())
        y = Fop @ xd
        x0 = DA(global_shape=231, local_shapes=y.local_shapes)
        x0[:] = 0
        solver = CGLS(Fop)
        xinv, istop, iit, r1, r2, cost = solver.solve(y, x0, niter=10, tol=0.0)
        return {"y": y.asarray().reshape(11, 21), "xinv": xinv.asarray(), "cost": cost, "iit": iit, "istop": istop}

    res = MPI.run_world(2, t_config1)[0]
    for k, v in res.items():
        put(f"config1/{k}", v)

    # ---- BlockDiag / VStack / CGLS (test_blockdiag.py, test_stack.py, test_solver.py) ----------------------
    def t_stack(rank, P, ny, nx, dtype):
        blocks = [np.random.default_rng(100 + r).standard_normal((ny - r, nx)).astype(dtype) for r in range(P)]
        if np.issubdtype(dtype, np.complexfloating):
            blocks = [b + 1j * np.random.default_rng(200 + r).standard_normal(b.shape) for r, b in enumerate(blocks)]
        Op = pylops.MatrixMult(blocks[rank], dtype=dtype)
        BDop = BD([Op])
        xg = np.random.default_rng(1).standard_normal(P * nx).astype(dtype)
        yg = np.random.default_rng(2).standard_normal(sum(ny - r for r in range(P))).astype(dtype)
        y = BDop @ DA.to_dist(xg)
        xa = BDop.H @ DA.to_dist(yg)
        VSop = VS([Op])
        xb = DA.to_dist(xg[:nx], partition=Partition.BROADCAST)
        yv = VSop @ xb
        xv = VSop.H @ DA.to_dist(yg)
        # cgls on the normal-equation style block of test_solver.py:150-196
        A = np.ones((ny, nx), dtype=dtype) * (rank + 1)
        blk = A.conj().T @ A + 1e-5 * np.eye(nx, dtype=dtype)
        Sop = BD([pylops.MatrixMult(blk, dtype=dtype)])
        xt = np.random.default_rng(42).normal(1, 10, P * nx).astype(dtype)
        yy = Sop @ DA.to_dist(xt)
        x0 = DA.to_dist(np.zeros(P * nx, dtype=dtype))
        xinv, istop, iit, r1, r2, cost = CGLS(Sop).solve(yy, x0, niter=nx, tol=1e-5)
        return {"bd_y": y.local_array, "bd_xa": xa.local_array, "vs_y": yv.local_array, "vs_x": xv.local_array,
                "cgls_x": xinv.local_array, "cgls_cost": cost, "cgls_iit": iit, "cgls_istop": istop,
                "cgls_r1": r1, "cgls_r2": r2}

    for P in (1, 2, 4):
        for ny, nx in ((11, 11), (31, 11)):
            for dtype in (np.float64, np.complex128):
                for r, res in enumerate(MPI.run_world(P, t_stack, P, ny, nx, dtype)):
                    for k, v in res.items():
                        put(f"stack/P{P}/{ny}x{nx}/{np.dtype(dtype).name}/r{r}/{k}", v)

    # ---- MPIMatrixMult block + summa (test_matrixmult.py) ---------------------------------------------------
    def t_mm(rank, P, N, K, M, dtype, kind):
        import math
        comm = MPI.COMM_WORLD
        A = np.arange(N * K, dtype=dtype).reshape(N, K)
        X = np.arange(K * M, dtype=dtype).reshape(K, M)
        if np.issubdtype(dtype, np.complexfloating):
            A, X = A + 0.5j * A, X + 0.7j * X
        Pp = math.isqrt(P)
        if kind == "summa":
            rs, cs = MM.local_block_split((N, K), rank, comm)
            Aop = MM.MPIMatrixMult(A[rs, cs].copy(), M, kind="summa", dtype=dtype)
            xs = MM.local_block_split((K, M), rank, comm)
            sizes = comm.allgather(int(np.prod(X[xs].shape)))
            xd = DA(global_shape=K * M, local_shapes=sizes, dtype=dtype)
            xd[:] = X[xs].ravel()
        else:
            blk, bc = int(math.ceil(N / Pp)), int(math.ceil(M / Pp))
            ci, ri = rank % Pp, rank // Pp
            Aop = MM.MPIMatrixMult(A[ci * blk:min(N, (ci + 1) * blk)].copy(), M, kind="block", dtype=dtype)
            Xc = X[:, ri * bc:min(M, (ri + 1) * bc)]
            ncs = comm.allgather(Xc.shape[1])
            xd = DA(global_shape=K * sum(ncs), local_shapes=[K * c for c in ncs], dtype=dtype)
            xd[:] = Xc.ravel()
        y = Aop @ xd
        xa = Aop.H @ y
        return {"y": y.local_array, "xa": xa.local_array}

    for P in (1, 4, 9):
        for (N, K, M, dtype) in ((64, 64, 64, np.float64), (37, 37, 37, np.float64), (50, 30, 40, np.float64),
                                 (22, 20, 16, np.complex128), (13, 14, 15, np.float32)):
            for kind in ("summa", "block"):
                for r, res in enumerate(MPI.run_world(P, t_mm, P, N, K, M, dtype, kind)):
                    for k, v in res.items():
                        put(f"mm/P{P}/{N}x{K}x{M}/{np.dtype(dtype).name}/{kind}/r{r}/{k}", v)

    # ---- MPIFredholm1 (test_fredholm.py) ------------------------------------------------------------------------
    def t_fr(rank, P, nz, dtype, saveGt, usematmul):
        nsl, nx, ny = 21, 4, 6
        rng = np.random.default_rng(5)
        G = rng.standard_normal((nsl, nx, ny))
        if np.issubdtype(dtype, np.complexfloating):
            G = G + 1j * rng.standard_normal((nsl, nx, ny))
        G = G.astype(dtype)
        x = np.random.default_rng(6).standard_normal(nsl * ny * nz).astype(dtype)
        ext = [nsl // P + (1 if r < nsl % P else 0) for r in range(P)]
        off = np.cumsum([0] + ext)
        Fop = FR(G[off[rank]:off[rank + 1]], nz=nz, saveGt=saveGt, usematmul=usematmul, dtype=dtype)
        y = Fop @ DA.to_dist(x, partition=Partition.BROADCAST)
        xa = Fop.H @ y
        return {"y": y.local_array, "xa": xa.local_array}

    for P in (1, 2, 3):
        for nz in (5, 1):
            for dtype in (np.float64, np.complex128):
                for saveGt, usematmul in ((True, True), (False, False)):
                    res = MPI.run_world(P, t_fr, P, nz, dtype, saveGt, usematmul)[0]
                    for k, v in res.items():
                        put(f"fredholm/P{P}/nz{nz}/{np.dtype(dtype).name}/s{int(saveGt)}m{int(usematmul)}/{k}", v)

    # ---- MPIGradient / MPILaplacian ("next" rows f2/f3; rank-local stencils restated in refshim/pylops) -------
    GR, LP = mods["Gradient"].MPIGradient, mods["Laplacian"].MPILaplacian

    def t_grad(rank, dims, samp, kind, edge, dtype):
        rng = np.random.default_rng(13)
        n = int(np.prod(dims))
        x = rng.normal(0, 10, n).astype(dtype)
        Gop = GR(dims, sampling=samp, kind=kind, edge=edge, dtype=dtype)
        y = Gop.matvec(DA.to_dist(x))
        xa = Gop.rmatvec(y)
        res = {"x": x, "xa": xa.local_array, "dot": y.dot(y), "norm": y.norm()}
        for i in range(y.narrays):
            res[f"y{i}"] = y[i].local_array
        return res

    def t_lap(rank, dims, axes, weights, samp, kind, edge, dtype):
        rng = np.random.default_rng(14)
        n = int(np.prod(dims))
        x = rng.normal(0, 10, n).astype(dtype)
        Lop = LP(dims, axes=axes, weights=weights, sampling=samp, kind=kind, edge=edge, dtype=dtype)
        xd = DA.to_dist(x)
        return {"x": x, "y": (Lop @ xd).local_array, "ya": (Lop.H @ xd).local_array}

    for P in (1, 2, 3):
        for dims, samp in (((21, 11), (1.0, 0.5)), ((13, 6, 7), (0.4, 1.0, 2.0))):
            for kind, edge in (("centered", True), ("centered", False), ("forward", False), ("backward", True)):
                for r, d in enumerate(MPI.run_world(P, t_grad, dims, samp, kind, edge, np.float64)):
                    for k, v in d.items():
                        put(f"grad/P{P}/{dims}/{kind}/e{int(edge)}/r{r}/{k}", v)
        for dims, axes, weights, samp in (((21, 11), (-2, -1), (1, 1), (1, 1)), ((21, 11), (0, 1), (2.0, 0.5), (0.4, 1.5)),
                                          ((13, 6, 7), (1, 2), (1, -2), (1.0, 0.5)), ((13, 6, 7), (2, 0), (1.5, 1), (1.0, 0.5))):
            for kind, edge in (("centered", True), ("forward", False), ("backward", False)):
                for r, d in enumerate(MPI.run_world(P, t_lap, dims, axes, weights, samp, kind, edge, np.float64)):
                    for k, v in d.items():
                        put(f"lap/P{P}/{dims}/{axes}/{weights}/{samp}/{kind}/e{int(edge)}/r{r}/{k}", v)

    # ---- ISTA / FISTA ("next" row: sparsity solvers; thresholds restated in refshim/pylops) ------------------
    ISTA, FISTA = mods["cls_sparsity"].ISTA, mods["cls_sparsity"].FISTA
    power_iteration = mods["eigs"].power_iteration

    def t_sparse(rank, P, solver, threshkind, dtype, niter, eps):
        rng = np.random.default_rng(21)
        ny, nx = 13, 11
        blocks = []
        for r in range(P):
            A = rng.standard_normal((ny, nx))
            if np.issubdtype(dtype, np.complexfloating):
                A = A + 1j * rng.standard_normal((ny, nx))
            blocks.append(A.astype(dtype))
        xtrue = np.zeros(P * nx, dtype=dtype)
        xtrue[rng.permutation(P * nx)[:max(2, P * nx // 5)]] = rng.standard_normal(max(2, P * nx // 5)) * 3
        Op = BD([pylops.MatrixMult(blocks[rank], dtype=dtype)])
        xt = DA.to_dist(xtrue)
        y = Op @ xt
        x0 = DA(global_shape=P * nx, dtype=dtype)
        x0[:] = 0
        lam = max(np.linalg.norm(b, 2) ** 2 for b in blocks)
        S = (ISTA if solver == "ista" else FISTA)(Op)
        x, iiter, cost = S.solve(y, x0, niter=niter, eps=eps, alpha=1.0 / lam, tol=1e-10, threshkind=threshkind)
        eig = power_iteration(Op.H @ Op, niter=200, tol=1e-12, dtype=dtype, backend="numpy",
                              b_k=DA(global_shape=P * nx, dtype=dtype))[0]
        return {"x": x.asarray(), "iiter": iiter, "cost": cost, "maxeig": np.abs(eig), "lam": lam}

    for P in (1, 2, 3):
        for solver in ("ista", "fista"):
            for threshkind, dtype, eps in (("soft", np.float64, 0.5), ("hard", np.float64, 0.05), ("half", np.float64, 0.2),
                                           ("soft", np.complex128, 0.5), ("soft", np.float32, 0.5)):
                res = MPI.run_world(P, t_sparse, P, solver, threshkind, dtype, 40, eps)[0]
                for k, v in res.items():
                    put(f"sparse/P{P}/{solver}/{threshkind}/{np.dtype(dtype).name}/{k}", v)

    # ---- MPIMDC ("next" row f1; the reference's chain F1^H I1^H MPIFredholm1 I F over refshim's restated FFT) ------
    MDC = mods["MDC"].MPIMDC

    def t_mdc(rank, P, twosided, dtype, conj, prescaled):
        rng = np.random.default_rng(31)
        ns, nr, nv, nt = 6, 5, 3, (31 if twosided else 32)
        nfmax = int(np.ceil((nt + 1) / 2)) - 3
        G = (rng.standard_normal((nfmax, ns, nr)) + 1j * rng.standard_normal((nfmax, ns, nr))).astype(dtype)
        rdt = np.real(np.ones(1, dtype)).dtype
        m = rng.standard_normal(nt * nr * nv).astype(rdt)
        d = rng.standard_normal(nt * ns * nv).astype(rdt)
        ext = [nfmax // P + (1 if r < nfmax % P else 0) for r in range(P)]
        off = np.cumsum([0] + ext)
        Mop = MDC(G[off[rank]:off[rank + 1]], nt=nt, nv=nv, nfreq=nfmax, dt=0.004, dr=2.0, twosided=twosided,
                  conj=conj, prescaled=prescaled)
        y = Mop @ DA.to_dist(m, partition=Partition.BROADCAST)
        xa = Mop.H @ DA.to_dist(d, partition=Partition.BROADCAST)
        return {"G": G, "m": m, "d": d, "y": y.local_array, "xa": xa.local_array}

    for P in (1, 2, 3):
        for twosided in (True, False):
            for dtype, conj, prescaled in ((np.complex128, False, False), (np.complex128, True, True), (np.complex64, False, False)):
                res = MPI.run_world(P, t_mdc, P, twosided, dtype, conj, prescaled)
                for k, v in res[0].items():
                    put(f"mdc/P{P}/t{int(twosided)}/{np.dtype(dtype).name}/c{int(conj)}p{int(prescaled)}/{k}", v)
                for r in range(1, P):      # BROADCAST outputs: identical on every rank
                    assert np.array_equal(res[r]["y"], res[0]["y"]) and np.array_equal(res[r]["xa"], res[0]["xa"])

    path = os.path.join(HERE, os.environ.get("GOLDEN_OUT", "reference_golden.npz"))
    golden_store.save(path, out)
    print(f"wrote {path}: {len(out)} arrays, {os.path.getsize(path) / 1e6:.2f} MB")


if __name__ == "__main__":
    main()
