"""NumPy oracle of the rank-local 1-D convolution (pylops_mpi_b200.local.Convolve1D), float64:

    forward: y[i] = sum_k h[k] x[i + offset - k]        (x = 0 outside [0, n_axis))
    adjoint: x[j] = sum_k h[k] y[j - offset + k]

the direct formula, written out sample by sample so that it shares no code with the pylops restatement
(tests/golden/refshim/pylops/signalprocessing/convolve1d.py) it is checked against.
"""
import numpy as np


def convolve1d(x, dims, h, offset=0, axis=-1, adjoint=False):
    """``Convolve1D(dims, h, offset, axis)`` applied to flat ``x`` (or its adjoint), in float64 / complex128"""
    dims = tuple(int(d) for d in (dims if np.ndim(dims) else (dims,)))
    h = np.asarray(h, dtype=np.float64)
    nh = h.size
    x = np.asarray(x)
    x = x.astype(np.complex128 if np.iscomplexobj(x) else np.float64).reshape(dims)
    xa = np.moveaxis(x, axis, -1)
    n = xa.shape[-1]
    y = np.zeros_like(xa)
    for i in range(n):
        for k in range(nh):
            s = i - offset + k if adjoint else i + offset - k
            if 0 <= s < n:
                y[..., i] += h[k] * xa[..., s]
    return np.moveaxis(y, -1, axis).ravel()


# the fixture grid of tests/golden/convolve_golden.npz (tests/golden/make_golden_convolve.py)
GRID_P = (1, 2, 3)
GRID_DIMS = (((37,), -1), ((5, 9, 37), -1), ((5, 9, 37), 0), ((5, 9, 37), 1), ((4, 3, 2, 19), 2))
GRID_NH = (1, 4, 5, 41)
GRID_DTYPES = ("float64", "float32", "complex128")
REFL_DIMS = (3, 8, 64)           # per rank
REFL_NT, REFL_DT, REFL_F0 = 41, 0.004, 20.0


def grid_offsets(nh):
    return sorted({0, nh // 2, nh - 1})


def grid_key(P, dims, axis, nh, offset, dtype):
    return f"conv/P{P}/{dims}/ax{axis}/nh{nh}/off{offset}/{dtype}"


def grid_inputs(key, P, dims, nh, dtype):
    """seeded filter ``h`` (float64) and global input ``x`` (P blocks of ``dims``) of one grid case"""
    import zlib
    rng = np.random.default_rng(zlib.crc32(key.encode()))
    h = rng.standard_normal(nh)
    n = P * int(np.prod(dims))
    x = rng.standard_normal(n)
    if dtype == "complex128":
        x = x + 1j * rng.standard_normal(n)
    return h, x.astype(dtype)


def refl_inputs(P):
    """the reflectivity chain's wavelet and blocky global model (P blocks of REFL_DIMS)"""
    rng = np.random.default_rng(77)
    ny, nx, nz = REFL_DIMS
    jumps = np.zeros((P * ny, nx, nz))
    jumps[..., rng.integers(4, nz - 4, 6)] = rng.normal(0, 1, (P * ny, nx, 6))
    return ricker(REFL_NT, REFL_DT, REFL_F0), np.cumsum(jumps, axis=-1).ravel()


def ricker(nt: int, dt: float, f0: float) -> np.ndarray:
    """centred Ricker wavelet with ``nt`` samples (nt odd) of peak frequency ``f0``: (1 - 2 a) exp(-a),
    a = (pi f0 t)^2, t = (k - nt // 2) dt"""
    t = (np.arange(nt) - nt // 2) * dt
    a = (np.pi * f0 * t) ** 2
    return (1.0 - 2.0 * a) * np.exp(-a)
