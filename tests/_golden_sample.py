"""Large outputs in tests/golden/*.npz are stored as a seeded sample, to keep every file under 1 MB: `<key>` then holds
the values at the flat positions `<key>_at`.  Shared by the golden generators and the tests that read them."""
import numpy as np

LIMIT = 20000  # outputs up to this many elements are stored whole


def shrink(blob, keys):
    """replaces each output in `keys` that is larger than LIMIT by LIMIT values at seeded positions"""
    for key in keys:
        a = np.asarray(blob[key])
        if a.size > LIMIT:
            at = np.sort(np.random.default_rng(a.size).choice(a.size, LIMIT, replace=False)).astype(np.int32)
            blob[key], blob[key + "_at"] = a.reshape(-1)[at], at


def expect(z, key, got):
    """-> (the elements of `got` that the file holds, the stored values)"""
    if key + "_at" in z.files:
        return np.asarray(got).reshape(-1)[z[key + "_at"]], z[key]
    return np.asarray(got), z[key]
