"""Restatement of third-party ``pylops.signalprocessing.Convolve1D`` (pylops 2.x ``_Convolve1D``, direct /
scipy path) -- TEST INFRASTRUCTURE so that tests/golden/make_golden_convolve.py can run the reference's
MPIBlockDiag / ISTA / CGLS over the operator of tutorials/reflectivity.py.  pylops shifts the filter by
zero-padding it by ``2 * (nh // 2 - offset)`` samples (one fewer for an even ``nh``) on the left (right when
negative) and then applies ``scipy.signal.convolve`` (forward) / ``scipy.signal.correlate`` (adjoint) with
``mode="same"`` along ``axis``."""
import numpy as np
from scipy.signal import convolve, correlate

from .. import LinearOperator


class Convolve1D(LinearOperator):
    def __init__(self, dims, h, offset=0, axis=-1, dtype="float64", method=None):
        dims = tuple(int(d) for d in (dims if np.ndim(dims) else (dims,)))
        h = np.asarray(h)
        if offset > h.size - 1:
            raise ValueError("offset must be smaller than len(h) - 1")
        self.dims, self.axis = dims, axis % len(dims)
        self.nh = h.size
        pad = 2 * (self.nh // 2 - int(offset))
        if self.nh % 2 == 0:
            pad -= 1
        if pad != 0:
            h = np.pad(h, (pad if pad > 0 else 0, -pad if pad < 0 else 0), mode="constant")
        shape = [1] * len(dims)
        shape[self.axis] = h.size
        self.h = h.reshape(shape)
        self.method = "direct" if method is None else method
        n = int(np.prod(dims))
        super().__init__(dtype=np.dtype(dtype), shape=(n, n))

    def _matvec(self, x):
        return convolve(np.reshape(x, self.dims), self.h, mode="same", method=self.method).ravel()

    def _rmatvec(self, x):
        return correlate(np.reshape(x, self.dims), self.h, mode="same", method=self.method).ravel()
