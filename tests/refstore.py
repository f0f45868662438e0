"""Stored outputs of the reference's own code, so that the tests comparing with it run where it cannot be compiled.

The reference's LIO sources, compiled over the stand-in headers of oracle/shim/ (oracle/Makefile, oracle/reference_py.py), only
build where the reference tree is present.  Each comparison with them is written as

    r = store("name", lambda: <call into the reference>, exact=("rows", ...))

With SRL_RECORD_REFERENCE=1 (and the reference libraries built) the call runs and its result is written to the module's
tests/golden/*.npz; otherwise the stored result is read back.  `fn` returns a flat dict of arrays and scalars.  Arrays named in
`exact` are large outputs the tests compare bit for bit: only their digest is stored, and the test compares it with the digest
of its own array.  Both modes return the same values, so a recording run also checks every assertion.
"""
from __future__ import annotations

import hashlib
import json
import os

import numpy as np

RECORD = os.environ.get("SRL_RECORD_REFERENCE") == "1"


def digest(*arrays) -> str:
    """Digest of the values and shapes of `arrays`: equal digests <=> np.array_equal for each pair (float -0.0 == 0.0)."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.asarray(a)
        a = a.astype(np.float64) + 0.0 if a.dtype.kind == "f" else a.astype(np.int64)
        h.update(repr(a.shape).encode())
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:32]


def map_digest(keys, counts, xyz) -> str:
    """Digest of a voxel map's content independent of the container's iteration order: voxels by key, points in voxel order."""
    keys, counts, xyz = np.asarray(keys), np.asarray(counts), np.asarray(xyz)
    order = np.lexsort(keys.T[::-1]) if keys.shape[0] else np.zeros(0, np.int64)
    return digest(keys[order], counts[order], *[xyz[i, :counts[i]] for i in order])


def eskf_fields(e) -> dict:
    return {f: np.asarray(getattr(e, f)) for f in ("p", "q", "v", "ba", "bg", "g", "cov")}


def near(name: str, a, approx) -> dict:
    """A large float array stored as the entries where it differs from `approx`, an array the test computes itself."""
    a, approx = np.asarray(a, np.float64), np.asarray(approx, np.float64)
    at = np.flatnonzero(a.ravel() != approx.ravel())
    return {f"{name}.at": at, f"{name}.val": a.ravel()[at], f"{name}.digest": digest(a)}


def from_near(r: dict, name: str, approx) -> np.ndarray:
    """Inverse of near(): the stored array, rebuilt from `approx` and checked against its digest."""
    a = np.array(approx, np.float64)
    a.ravel()[np.asarray(r[f"{name}.at"], np.int64)] = r[f"{name}.val"]
    assert digest(a) == r[f"{name}.digest"], f"{name}: the rebuilt array is not the stored one"
    return a


class Store:
    def __init__(self, filename: str):
        self.path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", filename)
        self.d = {}
        if os.path.exists(self.path) or not RECORD:
            with np.load(self.path) as z:                    # one index + one byte blob: far smaller than an npz entry per value
                blob = z["blob"].tobytes()
                for k, dtype, shape, at, n in json.loads(z["index"].item()):
                    self.d[k] = np.frombuffer(blob[at:at + n], dtype=dtype).reshape(shape)
        self.recorded = set()

    def __call__(self, name: str, fn, exact=()) -> dict:
        if RECORD:
            assert name not in self.recorded, f"{name} recorded twice"
            self.recorded.add(name)
            self.d = {k: v for k, v in self.d.items() if not k.startswith(name + ":")}
            for k, v in fn().items():
                self.d[f"{name}:{k}"] = np.asarray(digest(v) if k in exact else v)
        return self.get(name)

    def get(self, name: str) -> dict:
        """the stored output, also where another module's test records it"""
        out = {k.split(":", 1)[1]: v for k, v in self.d.items() if k.split(":", 1)[0] == name}
        assert out, f"no stored reference output named {name!r} in {self.path}"
        return {k: v.item() if v.ndim == 0 else v for k, v in out.items()}

    def save(self):
        if RECORD and self.recorded:
            index, parts, at = [], [], 0
            for k in sorted(self.d):
                a = np.ascontiguousarray(self.d[k])
                index.append((k, a.dtype.str, a.shape, at, a.nbytes))
                parts.append(a.tobytes())
                at += a.nbytes
            np.savez_compressed(self.path, index=np.array(json.dumps(index)), blob=np.frombuffer(b"".join(parts), np.uint8))
