"""Compact records of the original project's outputs, stored under tests/golden/ so that the parity tests run without a
build of the original.  Each array is kept as its SHA-256 (shape and dtype included), which stands in for a bit-exact
comparison, plus — for floating-point arrays — a seeded sample of its rows and its largest finite magnitude, which the
tolerance comparisons (relative error against max |ref|, mean / max image error) are evaluated on."""
import hashlib
import json
import os

import numpy as np

RASTER_RECORDS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "raster_ref_records.npz")
SAMPLE = 128  # sampled values per array (whole rows of per-point arrays, at least 8 rows)


def _np(x):
    if hasattr(x, "detach"):
        x = x.detach().cpu().numpy()
    return np.ascontiguousarray(np.asarray(x))


def _sha(a):
    h = hashlib.sha256(str((a.shape, a.dtype.str)).encode())
    h.update(a.tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def _rows(a):
    """Per-point arrays (P, ...) are sampled by whole rows; images and 1-D arrays by element."""
    return a.reshape(a.shape[0], -1) if a.ndim >= 2 and a.shape[0] > 16 else a.reshape(-1, 1)


def record(out, key, x, seed=0, extra_rows=(), sample=True):
    """Adds the record of array `x` under `key` to the dict `out` (later written with np.savez_compressed); sample=False
    keeps only what the bit-exact comparison needs."""
    a = _np(x)
    out[key + ".sha"], out[key + ".dtype"] = _sha(a), np.array(a.dtype.str)
    if a.dtype.kind != "f" or not sample:
        return
    out[key + ".finsha"] = _sha(np.isfinite(a))
    r = _rows(a)
    fin = np.isfinite(r)
    out[key + ".absmax"] = np.float64(np.abs(r[fin]).max()) if fin.any() else np.float64(0.0)
    if r.size == 0:
        out[key + ".idx"], out[key + ".val"] = np.zeros(0, np.int64), np.zeros((0, r.shape[1]), r.dtype)
        return
    n = max(8, SAMPLE // r.shape[1])
    rng = np.random.default_rng(seed)
    nz = np.flatnonzero((r != 0).any(1))
    pick = rng.choice(nz, min(n, len(nz)), replace=False) if len(nz) else np.zeros(0, np.int64)
    anywhere = rng.choice(len(r), min(max(2, n // 8), len(r)), replace=False)
    top = np.abs(np.where(fin, r, 0)).max(1).argmax()
    idx = np.union1d(np.union1d(pick, anywhere), np.r_[top, np.asarray(extra_rows, np.int64)]).astype(np.int64)
    out[key + ".idx"], out[key + ".val"] = idx, r[idx]


def save(path, out):
    """Writes the dict `out` as one compressed byte blob plus a JSON index (one .npz member per array would cost more in
    archive headers than the records themselves)."""
    index, parts, off = {}, [], 0
    for k in sorted(out):
        a = np.asarray(out[k], order="C")
        if a.dtype == np.int64 and k.endswith(".idx"):
            a = a.astype(np.int32)
        index[k] = [a.dtype.str, list(a.shape), off, a.nbytes]
        parts.append(a.tobytes())
        off += a.nbytes
    np.savez_compressed(path, index=np.array(json.dumps(index)), blob=np.frombuffer(b"".join(parts), np.uint8))


def load(path):
    z = np.load(path)
    blob = z["blob"].tobytes()
    return {k: np.frombuffer(blob, np.dtype(dt), count=int(np.prod(shape)), offset=off).reshape(tuple(shape))
            for k, (dt, shape, off, n) in json.loads(str(z["index"])).items()}


class Golden:
    """Reader of a record file written by save(); `key` names one recorded array."""

    def __init__(self, path):
        self.z = load(path)

    def has(self, key):
        return key + ".sha" in self.z

    def scalar(self, key):
        return self.z[key].item()

    def equal(self, key, x):
        """Bit-exact equality with the recorded array (shape included; integer and boolean arrays are compared by value)."""
        a, dt = _np(x), np.dtype(str(self.z[key + ".dtype"]))
        if a.dtype != dt and a.dtype.kind in "biu" and dt.kind in "biu":
            a = a.astype(dt)
        return np.array_equal(_sha(a), self.z[key + ".sha"])

    def finite_equal(self, key, x):
        return np.array_equal(_sha(np.isfinite(_np(x))), self.z[key + ".finsha"])

    def sample(self, key, x):
        """(ours, reference) on the recorded rows, as float64 arrays of shape (rows, values per row), and the reference's
        largest finite magnitude."""
        r = _rows(_np(x))
        idx = self.z[key + ".idx"]
        return r[idx].astype(np.float64), self.z[key + ".val"].astype(np.float64), float(self.z[key + ".absmax"])

    def rows(self, key):
        return self.z[key + ".idx"]

    def rel_err(self, key, x):
        """max |ours - ref| / (max |ref| + tiny) over the recorded rows (tests/util.py:rel_err on the sample)."""
        a, b, m = self.sample(key, x)
        return float(np.abs(a - b).max(initial=0.0) / (m + 1e-30))
