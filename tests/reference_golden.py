"""What the original RepSurf code returned, stored so that the comparisons with it run anywhere.

Outputs a test compares bit for bit are kept as SHA-256 digests (tests/golden/<name>.json); outputs it compares within a
tolerance are kept as small arrays, sampled where the full output is large (tests/golden/<name>.npz).

Recording: with REPSURF_RECORD_GOLDEN=<dir> set, every comparison computes the original's output live (the reference
Python through oracle/ref_loader.py, its CUDA kernels through tests/refcuda.py), checks against it as before and writes
<dir>/<name>.json / .npz; copy those into tests/golden/.
"""
import hashlib
import json
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RECORD_DIR = os.environ.get("REPSURF_RECORD_GOLDEN")


def digest(x):
    """Shape and values; integers widened to int64, and -0.0 counted as 0.0, as torch.equal does."""
    a = x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)
    if a.dtype.kind in "iub":
        a = a.astype(np.int64)
    elif a.dtype.kind == "f":
        a = a + a.dtype.type(0)
    h = hashlib.sha256(repr(a.shape).encode())
    h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def sample_rows(n, k, seed=0):
    """A fixed, sorted sample of k of n rows."""
    return np.sort(np.random.RandomState(seed).choice(n, min(n, k), replace=False))


class Reference:
    def __init__(self, name):
        self.name = name
        self.recording = bool(RECORD_DIR)
        self._digests = None
        self._arrays = None

    def _path(self, ext):
        return os.path.join(RECORD_DIR if self.recording else GOLDEN, f"{self.name}.{ext}")

    def _load(self):
        if self._digests is None:
            js, npz = self._path("json"), self._path("npz")
            self._digests = json.load(open(js)) if os.path.exists(js) or not self.recording else {}
            self._arrays = dict(np.load(npz)) if os.path.exists(npz) or not self.recording else {}

    def _save(self):
        os.makedirs(RECORD_DIR, exist_ok=True)
        with open(self._path("json"), "w") as f:
            json.dump(self._digests, f, indent=0, sort_keys=True)
        np.savez_compressed(self._path("npz"), **self._arrays)

    def same(self, key, got, ref):
        """whether `got` equals, bit for bit, what the original returned; `ref()` computes that (recording only)"""
        self._load()
        if self.recording:
            self._digests[key] = digest(ref())
            self._save()
        return digest(got) == self._digests[key]

    def equal(self, key, got, ref):
        assert self.same(key, got, ref), f"{self.name}: {key} differs from the original"

    def array(self, key, ref):
        """the original's output `ref()` (recorded; keep it small)"""
        self._load()
        if self.recording:
            a = ref()
            self._arrays[key] = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
            self._save()
        return self._arrays[key]
