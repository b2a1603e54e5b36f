"""How tests/golden stores results of the reference's own code (tests/golden/make_ref_golden.py) and how tests read them back.

TEST INFRASTRUCTURE, NOT PRODUCT.  A result that a test compares bit for bit is stored as a SHA-256 digest (`digest`); a result compared
within a tolerance is stored whole, or, when it is large, as a fixed seeded sample of its entries (`put`, `pair`).
"""
import hashlib

import numpy as np

SAMPLE = 2048   # entries kept of an array with more than 2 * SAMPLE of them


def digest(*arrays):
    """SHA-256 over the dtype, shape and bytes of each array (numpy arrays or torch tensors)."""
    h = hashlib.sha256()
    for a in arrays:
        if hasattr(a, "detach"):
            a = a.detach().cpu().numpy()
        a = np.ascontiguousarray(a)
        h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def put(store, key, a):
    """store[key] = a as float32; above 2 * SAMPLE entries only a seeded sample of them, with their flat indices in store[key + '@']."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.size <= 2 * SAMPLE:
        store[key] = a
        return
    at = np.sort(np.random.default_rng(a.size).choice(a.size, SAMPLE, replace=False)).astype(np.int32)
    store[key] = a.reshape(-1)[at]
    store[key + "@"] = at


def pair(z, key, ours):
    """(ours, reference) over the entries the golden file keeps for `key`; `ours` is a numpy array or a torch tensor."""
    if hasattr(ours, "detach"):
        ours = ours.detach().cpu().numpy()
    if key + "@" in z:
        return ours.reshape(-1)[z[key + "@"]], z[key]
    return ours, z[key]
