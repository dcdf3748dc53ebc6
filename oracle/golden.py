"""TEST INFRASTRUCTURE ONLY (oracle/): fingerprints of reference outputs that are stored under tests/golden/ instead of the arrays.

A bit-exact comparison with an array too large to keep in the repository is a comparison of SHA-256 digests.  The digest is taken
of a canonical form that keeps exactly what the comparison looks at:
  * "bits"   -- every byte (torch.equal / == on integer views);
  * "values" -- floats compared as values with NaNs in the same places (np.array_equal(equal_nan=True)): -0.0 folds to +0.0, every
                NaN to one quiet NaN;
  * "map"    -- a (3 * rows, cols) vertex / normal map compared like tests/test_gpu_ops.py::same_map: the NaN mask of the x plane, and
                the bits of all three planes where x is valid (the y / z planes of an invalid pixel are not looked at).
"""
import hashlib

import numpy as np


def _np(a):
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(a)


def digest(a, mode="bits"):
    a = _np(a)
    if mode == "values":
        a = a.copy()
        a[a == 0] = 0
        a[np.isnan(a)] = np.nan
    elif mode == "map":
        a = a.reshape(3, -1).copy()
        a[:, np.isnan(a[0])] = np.nan
    elif mode != "bits":
        raise ValueError(mode)
    h = hashlib.sha256(a.dtype.str.encode())
    h.update(np.ascontiguousarray(a).view(np.uint8).tobytes())
    return h.hexdigest()


def canon_points(pts):
    """A point cloud of 32-byte records as a sorted (n, 4) uint64 array: extraction order is not part of the result."""
    a = np.ascontiguousarray(_np(pts)).view(np.uint64).reshape(-1, 4)
    return a[np.lexsort(a.T[::-1])] if len(a) else a


def sample_touched(weights, n, seed):
    """A fixed, seeded, sorted sample of the flat indices of touched voxels (weight != 0)."""
    idx = np.flatnonzero(_np(weights).reshape(-1))
    if len(idx) > n:
        idx = np.sort(np.random.default_rng(seed).choice(idx, n, replace=False))
    return idx.astype(np.int64)
