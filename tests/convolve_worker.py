"""Two-rank reflectivity chain (tutorials/reflectivity.py at a small size): run under torchrun with one process per
GPU.  Each rank owns a (3, 8, 64) block; DDiag / CDiag are MPIBlockDiag over the rank-local FirstDerivative /
Convolve1D, then ISTA and CGLS on CDiag.  Every rank's output is compared with the NumPy oracle at the same P."""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (ROOT, os.path.join(ROOT, "oracle"), HERE):
    sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import convolve_oracle as co  # noqa: E402
import pylops_mpi_b200 as pm  # noqa: E402
from test_convolve import refl_oracle  # noqa: E402

comm = pm.get_comm_world()
rank, P = comm.Get_rank(), comm.Get_size()


def host(t):
    return t.cpu().numpy()


def check(name, got, ref, rtol=1e-12, atol=1e-12):
    np.testing.assert_allclose(got, ref, rtol=rtol, atol=atol, err_msg=f"[rank {rank}] {name}")


ref = refl_oracle(P)
wav, m = co.refl_inputs(P)
dims, wavc = co.REFL_DIMS, co.REFL_NT // 2
n = int(np.prod(dims))
mine = slice(rank * n, (rank + 1) * n)
DDiag = pm.MPIBlockDiag([pm.local.FirstDerivative(dims, axis=-1)])
CDiag = pm.MPIBlockDiag([pm.local.Convolve1D(dims, wav, offset=wavc, axis=-1)])
md = pm.DistributedArray.to_dist(m)
assert md.local_shape == (n,)
r = DDiag @ md
d = CDiag @ r
check("r", host(r.local_array), ref["r"][mine])
check("d", host(d.local_array), ref["d"][mine])
x0 = pm.DistributedArray(global_shape=P * n)
x0[:] = 0.0
x, iiter, cost = pm.ista(CDiag, d, x0=x0, niter=30, eps=1e-2, alpha=ref["alpha"], tol=1e-8)
assert iiter == ref["ista_iiter"], (iiter, ref["ista_iiter"])
check("ista cost", np.asarray(cost), ref["ista_cost"], 1e-10, 1e-10)
check("ista x", host(x.local_array), ref["ista_x"][mine], 1e-10, 1e-10)
x0c = pm.DistributedArray(global_shape=P * n)
x0c[:] = 0.0
xc, istop, iitc, r1, r2, costc = pm.cgls(CDiag, d, x0=x0c, niter=20, tol=0.0)
check("cgls cost", np.asarray(costc), ref["cgls_cost"], 1e-9, 1e-12)
check("cgls x", host(xc.local_array), ref["cgls_x"][mine], 1e-8, 1e-8)
comm.Barrier()
torch.cuda.synchronize()
print(f"CONVOLVE_WORKER_OK rank={rank} size={P}")
