"""Generate tests/golden/convolve_golden.npz by running the REAL reference (a pylops-mpi source checkout,
imported unmodified) over the restated pylops ``Convolve1D`` (refshim/pylops/signalprocessing/convolve1d.py):

    PYLOPS_MPI_REFERENCE=<pylops-mpi checkout> python tests/golden/make_golden_convolve.py

* ``conv/...``: MPIBlockDiag([Convolve1D(dims, h, offset, axis)]) forward and adjoint plus the reference's
  dottest, over the grid of tests/convolve_oracle.py (P = 1, 2, 3 ranks; inputs drawn from per-case seeds).
* ``refl/P<P>/...``: the chain of tutorials/reflectivity.py at a small size -- DDiag = MPIBlockDiag([FirstDerivative]),
  CDiag = MPIBlockDiag([Convolve1D(wav, offset=wavc)]), then ISTA (30 iterations, eps=1e-2, tol=1e-8) and CGLS
  (20 iterations) on CDiag.  ISTA gets an explicit ``alpha = 1 / (sum|h|)^2`` (a bound on 1 / ||C||^2): without
  it the reference estimates the step with a power iteration whose start vector is random.

The existing tests/golden/reference_golden.npz is not touched.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden  # noqa: E402  (puts refshim/ and tests/ on sys.path)
import golden_store  # noqa: E402
import convolve_oracle as co  # noqa: E402


def main():
    if not os.path.isdir(os.path.join(make_golden.REF, "pylops_mpi")):
        raise SystemExit("set PYLOPS_MPI_REFERENCE to a pylops-mpi source checkout")
    from mpi4py import MPI
    import pylops
    from pylops.signalprocessing.convolve1d import Convolve1D
    pkg, mods = make_golden.load_reference()
    DA = pkg.DistributedArray
    BD = mods["BlockDiag"].MPIBlockDiag
    CGLS = mods["cls_basic"].CGLS
    ISTA = mods["cls_sparsity"].ISTA
    dottest = mods["dottest"].dottest
    out = {}

    def put(key, val):
        out[key] = np.asarray(val)

    def t_conv(rank, key, P, dims, axis, nh, offset, dtype):
        h, x = co.grid_inputs(key, P, dims, nh, dtype)
        Op = BD([Convolve1D(dims, h, offset=offset, axis=axis, dtype=dtype)])
        xd = DA.to_dist(x)
        y = Op @ xd
        ya = Op.H @ xd
        rng = np.random.default_rng(3)
        u = DA.to_dist(rng.standard_normal(x.size).astype(dtype))
        v = DA.to_dist(rng.standard_normal(x.size).astype(dtype))
        ok = dottest(Op, u, v, rtol=1e-4 if dtype == "float32" else 1e-6)
        return {"h": h, "x": x, "y": y.local_array, "ya": ya.local_array, "dottest": ok}

    for P in co.GRID_P:
        for dims, axis in co.GRID_DIMS:
            for nh in co.GRID_NH:
                for offset in co.grid_offsets(nh):
                    for dtype in co.GRID_DTYPES:
                        key = co.grid_key(P, dims, axis, nh, offset, dtype)
                        res = MPI.run_world(P, t_conv, key, P, dims, axis, nh, offset, dtype)
                        put(key + "/h", res[0]["h"])
                        put(key + "/x", res[0]["x"])
                        for r, d in enumerate(res):
                            put(key + f"/r{r}/y", d["y"])
                            put(key + f"/r{r}/ya", d["ya"])
                            assert d["dottest"], key

    def t_refl(rank, P):
        wav, m = co.refl_inputs(P)
        wavc = co.REFL_NT // 2
        dims = co.REFL_DIMS
        n = int(np.prod(dims))
        DDiag = BD([pylops.FirstDerivative(dims, axis=-1)])
        CDiag = BD([Convolve1D(dims, wav, offset=wavc, axis=-1)])
        r = DDiag @ DA.to_dist(m)
        d = CDiag @ r
        x0 = DA(global_shape=P * n)
        x0[:] = 0.0
        alpha = 1.0 / np.sum(np.abs(wav)) ** 2
        xi, iiter, cost = ISTA(CDiag).solve(d, x0, niter=30, eps=1e-2, alpha=alpha, tol=1e-8)
        x0c = DA(global_shape=P * n)
        x0c[:] = 0.0
        xc, istop, iitc, r1, r2, costc = CGLS(CDiag).solve(d, x0c, niter=20, tol=0.0)
        return {"wav": wav, "m": m, "r": r.local_array, "d": d.local_array, "ista_x": xi.local_array,
                "ista_iiter": iiter, "ista_cost": cost, "alpha": alpha, "cgls_x": xc.local_array, "cgls_cost": costc,
                "cgls_iit": iitc}

    for P in co.GRID_P:
        res = MPI.run_world(P, t_refl, P)
        for k in ("wav", "m", "ista_iiter", "ista_cost", "alpha", "cgls_cost", "cgls_iit"):
            put(f"refl/P{P}/{k}", res[0][k])
        for r, d in enumerate(res):
            for k in ("r", "d", "ista_x", "cgls_x"):
                put(f"refl/P{P}/r{r}/{k}", d[k])

    path = os.path.join(HERE, os.environ.get("GOLDEN_OUT", "convolve_golden.npz"))
    golden_store.save(path, out)
    print(f"wrote {path}: {len(out)} arrays, {os.path.getsize(path) / 1e6:.2f} MB")


if __name__ == "__main__":
    main()
