"""Compact storage of the reference's golden vectors (tests/golden/reference_golden.npz).

``save`` takes the flat ``{key: array}`` dictionary that tests/golden/make_golden.py collects from the
reference.  Keys of the form ``<group>/r<rank>/<name>`` (one array per simulated rank) are gathered into one
record ``<group>/<name>`` that keeps every rank's shape.  A record of at most ``FULL_MAX`` values is stored
whole.  A larger one is stored as a summary:

  * a SHA-256 digest of its bytes, for comparisons that must be bit-exact;
  * its values at the first and last position of every rank plus ``SAMPLES`` seeded positions in between;
  * one weighted sum ``s = sum(w * g)`` with fixed weights ``w`` in [-0.5, 0.5), with ``sum(|w| * |g|)``.

If ``allclose(actual, g, rtol, atol)`` holds elementwise, then
``|sum(w * actual) - s| <= atol * sum(|w|) + rtol * sum(|w| * |g|)``, so the weighted sum checks every entry
in aggregate (a shifted, permuted or mis-signed block moves it) without failing where the elementwise
comparison would pass.
"""
from __future__ import annotations

import hashlib
import json
import re
import zlib

import numpy as np

FULL_MAX = 64
SAMPLES = 4
_RANK_KEY = re.compile(r"^(.*)/r(\d+)/([^/]+)$")
_SLACK = 1e-14           # rounding of the two weighted sums themselves


def _weights(n: int) -> np.ndarray:
    """exact in float64 on every platform (integer hash, no libm)"""
    i = np.arange(n, dtype=np.uint64)
    return ((i * np.uint64(2654435761)) % np.uint64(1 << 32)).astype(np.float64) / float(1 << 32) - 0.5


def _digest(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def _as_float64(a: np.ndarray) -> np.ndarray:
    """values of a real / complex / integer array as a flat float64 array (complex: interleaved re, im)"""
    a = np.ascontiguousarray(a).ravel()
    if np.iscomplexobj(a):
        return a.astype(np.complex128).view(np.float64)
    return a.astype(np.float64)


def _from_float64(v: np.ndarray, dtype: np.dtype) -> np.ndarray:
    if np.issubdtype(dtype, np.complexfloating):
        return v.view(np.complex128).astype(dtype)
    return v.astype(dtype)


def save(path: str, arrays: dict) -> None:
    groups = {}
    for key, val in arrays.items():
        m = _RANK_KEY.match(key)
        name, rank = (f"{m.group(1)}/{m.group(3)}", int(m.group(2))) if m else (key, None)
        groups.setdefault(name, {})[rank] = np.asarray(val)
    meta, vals, idx = {}, [], []
    nvals = 0
    for name, per_rank in groups.items():
        ranks = sorted(per_rank, key=lambda r: -1 if r is None else r)
        assert ranks == [None] or ranks == list(range(len(ranks))), name
        parts = [per_rank[r] for r in ranks]
        if parts[0].dtype.kind == "U":
            meta[name] = {"str": str(parts[0])}
            continue
        dtype = np.result_type(*parts)
        flat = np.concatenate([p.astype(dtype).ravel() for p in parts])
        rec = {"dtype": dtype.str, "shapes": [list(p.shape) for p in parts], "per_rank": ranks != [None]}
        if flat.size <= FULL_MAX:
            sel = np.arange(flat.size)
        else:
            ends = np.cumsum([p.size for p in parts])
            fixed = set(np.concatenate([ends - np.array([p.size for p in parts]), ends - 1]).tolist())
            rng = np.random.default_rng(zlib.crc32(name.encode()))
            sel = np.array(sorted(fixed | set(rng.choice(flat.size, SAMPLES, replace=False).tolist())))
            w = _weights(flat.size)
            rec.update(digest=_digest(flat), wsum=[float(np.real(np.sum(w * flat))), float(np.imag(np.sum(w * flat)))],
                       wabs=float(np.sum(np.abs(w) * np.abs(flat))), wone=float(np.sum(np.abs(w))),
                       amax=float(np.max(np.abs(flat))))
            if np.iscomplexobj(flat):
                rec["imag_zero"] = bool(np.all(flat.imag == 0))
            idx.append(sel)
        v = _as_float64(flat[sel])
        rec.update(off=nvals, n=int(sel.size))
        vals.append(v)
        nvals += v.size
        meta[name] = rec
    np.savez_compressed(path, meta=np.array(json.dumps(meta)), vals=np.concatenate(vals),
                        idx=np.concatenate(idx).astype(np.int64))


class Record:
    """one stored array (or one gathered per-rank group); see the module docstring"""

    def __init__(self, name, rec, vals, idx, idx_off):
        self.name = name
        self.dtype = np.dtype(rec["dtype"])
        self.shapes = [tuple(s) for s in rec["shapes"]]
        self.size = sum(int(np.prod(s)) for s in self.shapes)
        self.full = "digest" not in rec
        self.rec = rec
        width = 2 if np.issubdtype(self.dtype, np.complexfloating) else 1
        self.values = _from_float64(vals[rec["off"]:rec["off"] + width * rec["n"]], self.dtype)
        self.index = np.arange(self.size) if self.full else idx[idx_off:idx_off + rec["n"]]

    @property
    def nranks(self):
        return len(self.shapes)

    def array(self, rank=None):
        """the stored array (of one rank); only records stored whole have one"""
        assert self.full, f"{self.name}: stored as a summary, compare with check()"
        ends = np.cumsum([0] + [int(np.prod(s)) for s in self.shapes])
        r = 0 if rank is None else rank
        return self.values[ends[r]:ends[r + 1]].reshape(self.shapes[r])

    @property
    def amax(self):
        return self.rec["amax"] if not self.full else float(np.max(np.abs(self.values)))

    @property
    def imag_zero(self):
        return self.rec["imag_zero"] if not self.full else bool(np.all(np.imag(self.values) == 0))

    def check(self, actual, rtol=0.0, atol=0.0):
        """compare ``actual`` with the record: a list holds one array per rank (rank count and per-rank sizes must
        match), a single array is the ranks' arrays gathered.  ``rtol == atol == 0`` asks for bit-exact equality
        (values cast to the stored dtype)."""
        parts = [np.asarray(p) for p in actual] if isinstance(actual, (list, tuple)) else [np.asarray(actual)]
        if isinstance(actual, (list, tuple)):
            assert len(parts) == self.nranks, f"{self.name}: {len(parts)} ranks, reference has {self.nranks}"
            assert [p.size for p in parts] == [int(np.prod(s)) for s in self.shapes], \
                f"{self.name}: per-rank sizes {[p.size for p in parts]} vs reference {self.shapes}"
        flat = np.concatenate([p.ravel() for p in parts])
        assert flat.size == self.size, f"{self.name}: {flat.size} values, reference has {self.size}"
        exact = rtol == 0.0 and atol == 0.0
        got = flat[self.index]
        if exact:
            np.testing.assert_array_equal(got, self.values, err_msg=self.name)
        else:
            np.testing.assert_allclose(got, self.values, rtol=rtol, atol=atol, err_msg=self.name)
        if self.full:
            return
        if exact:
            assert _digest(flat.astype(self.dtype)) == self.rec["digest"], f"{self.name}: bytes differ from the reference"
            return
        f = flat.astype(np.complex128 if np.iscomplexobj(flat) or np.issubdtype(self.dtype, np.complexfloating)
                        else np.float64)
        s = np.sum(_weights(f.size) * f)
        ref = complex(*self.rec["wsum"])
        bound = atol * self.rec["wone"] + (rtol + _SLACK) * self.rec["wabs"]
        assert abs(s - ref) <= bound, f"{self.name}: weighted sum {s} vs reference {ref} (bound {bound:.3e})"


class Golden:
    def __init__(self, path: str):
        with np.load(path, allow_pickle=False) as z:
            meta, vals, idx = json.loads(str(z["meta"])), z["vals"], z["idx"]
        self._strs = {k: r["str"] for k, r in meta.items() if "str" in r}
        self._recs = {}
        off = 0
        for k, r in meta.items():
            if "str" in r:
                continue
            self._recs[k] = Record(k, r, vals, idx, off)
            if "digest" in r:
                off += r["n"]

    def keys(self):
        """the original keys: ``<group>/r<rank>/<name>`` for a gathered per-rank record"""
        out = list(self._strs)
        for k, r in self._recs.items():
            if r.rec["per_rank"]:
                g, _, n = k.rpartition("/")
                out += [f"{g}/r{i}/{n}" for i in range(r.nranks)]
            else:
                out.append(k)
        return out

    def _split(self, key):
        m = _RANK_KEY.match(key)
        if m and f"{m.group(1)}/{m.group(3)}" in self._recs:
            rec = self._recs[f"{m.group(1)}/{m.group(3)}"]
            if rec.rec["per_rank"] and int(m.group(2)) < rec.nranks:
                return rec, int(m.group(2))
        return self._recs.get(key), None

    def __contains__(self, key):
        return key in self._strs or self._split(key)[0] is not None

    def record(self, key) -> Record:
        return self._recs[key]

    def __getitem__(self, key):
        """a string or an array stored whole (of one rank, for ``<group>/r<rank>/<name>``)"""
        if key in self._strs:
            return self._strs[key]
        rec, rank = self._split(key)
        if rec is None:
            raise KeyError(key)
        return rec.array(rank)
