"""What the reference project's own code returned, stored as golden data so the tests that compare against it run
anywhere.  A test asks for a value by key with the function that computes it from the reference:

    want = rec("vocoder[T=7]", lambda: <call into the reference>)

Normally the stored value is returned and the function is never called.  With XTTS_RECORD_REFERENCE=1 and the
reference tree present (oracle/ref_import.py), the function runs, and its value is returned and written to
tests/golden/<name>.npz.  Values may nest lists, tuples, dicts, str / int / float / bool / None, bytes, numpy arrays
and torch tensors (returned as numpy arrays)."""
from __future__ import annotations

import base64
import json
import os

import numpy as np

RECORD = os.environ.get("XTTS_RECORD_REFERENCE") == "1"
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class Records:
    def __init__(self, name: str):
        self.path = os.path.join(GOLDEN, name + ".npz")
        self._values = None
        self._arrays = None

    def _load(self):
        if self._values is None:
            self._values, self._arrays = {}, {}
            if os.path.exists(self.path):
                with np.load(self.path, allow_pickle=False) as z:
                    self._arrays = {k: z[k] for k in z.files if k != "__json__"}
                    self._values = json.loads(str(z["__json__"]))

    def __call__(self, key: str, compute):
        self._load()
        if RECORD:
            from oracle import ref_import
            if not ref_import.available():
                raise RuntimeError("XTTS_RECORD_REFERENCE=1 needs the reference tree (oracle/ref_import.py)")
            value = _plain(compute())
            self._arrays = {k: a for k, a in self._arrays.items() if not k.startswith(key + "#")}
            self._values[key] = self._encode(value, key)
            np.savez_compressed(self.path, __json__=np.array(json.dumps(self._values, sort_keys=True)), **self._arrays)
            return value
        if key not in self._values:
            raise KeyError(f"{key!r} is not recorded in {self.path}: record it with XTTS_RECORD_REFERENCE=1")
        return self._decode(self._values[key])

    def _encode(self, v, key):
        if isinstance(v, np.ndarray):
            name = f"{key}#{len([k for k in self._arrays if k.startswith(key + '#')])}"
            self._arrays[name] = v
            return {"__array__": name}
        if isinstance(v, bytes):
            return {"__bytes__": base64.b64encode(v).decode()}
        if isinstance(v, tuple):
            return {"__tuple__": [self._encode(x, key) for x in v]}
        if isinstance(v, list):
            return [self._encode(x, key) for x in v]
        if isinstance(v, dict):
            return {"__dict__": [[self._encode(k, key), self._encode(x, key)] for k, x in v.items()]}
        return v

    def _decode(self, v):
        if isinstance(v, list):
            return [self._decode(x) for x in v]
        if isinstance(v, dict):
            if "__array__" in v:
                return self._arrays[v["__array__"]]
            if "__bytes__" in v:
                return base64.b64decode(v["__bytes__"])
            if "__tuple__" in v:
                return tuple(self._decode(x) for x in v["__tuple__"])
            return {self._decode(k): self._decode(x) for k, x in v["__dict__"]}
        return v


def _plain(v):
    """torch tensors -> numpy arrays, numpy scalars -> Python scalars, recursively."""
    if hasattr(v, "detach") and hasattr(v, "numpy"):
        return v.detach().cpu().numpy()
    if isinstance(v, np.generic):
        return v.item()
    if isinstance(v, (list, tuple)):
        return type(v)(_plain(x) for x in v)
    if isinstance(v, dict):
        return {k: _plain(x) for k, x in v.items()}
    return v


def sample(a, n: int = 512):
    """(shape, a fixed seeded sample of at most n elements of the flattened array): how large outputs are stored."""
    a = np.asarray(a)
    idx = np.arange(a.size) if a.size <= n else np.sort(np.random.RandomState(a.size).choice(a.size, n, replace=False))
    return tuple(a.shape), a.reshape(-1)[idx]
