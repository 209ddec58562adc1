"""What the reference's own code computed on the inputs of the tests that pin the oracle to it.

tests/golden/make_reference_vectors.py runs the reference's headers (compiled by oracle/ref_shim/build_ref.sh) over
the exact inputs of tests/test_oracle_vs_ref.py, tests/test_oracle_vs_ref_property.py and tests/test_n4_oracle.py and
stores the results under tests/golden/reference_*.npz, so those tests compare the oracle with the reference wherever
the repository is checked out.  Outputs compared exactly are stored as 64-bit digests of their bytes; values are kept where a
test compares with a tolerance."""
import hashlib
import os
import zlib

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_CACHE = {}


def digest(*arrays):
    """64-bit digest of the dtype, shape and bytes of each array."""
    h = hashlib.blake2b(digest_size=8)
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    return np.frombuffer(h.digest(), np.uint64)[0]


def point_digests(*arrays):
    """16-bit digest per row (first axis) of the arrays: per-keypoint comparison of flows and distances."""
    n = len(arrays[0])
    rows = np.concatenate([np.ascontiguousarray(a).reshape(n, -1).view(np.uint8) for a in arrays], axis=1)
    return np.array([int.from_bytes(hashlib.blake2b(r.tobytes(), digest_size=2).digest(), "little") for r in rows], np.uint16)


def cases(spaces, examples, name):
    """(index, parameters) of the examples[name] stored examples of spaces[name], a dict of parameter: (lo, hi) inclusive integer
    range, (lo, hi) of floats for a uniform draw, or a list of choices.  The first example takes every parameter's first value, the
    second its last, the others are drawn from a generator seeded with the name."""
    r = np.random.default_rng(zlib.crc32(name.encode()))
    count, cols = examples[name], {}
    for k, v in spaces[name].items():
        if isinstance(v, list):
            idx = r.integers(0, len(v), count)
            idx[:2] = 0, len(v) - 1
            cols[k] = [v[i] for i in idx]
        elif isinstance(v[0], float):
            cols[k] = r.uniform(v[0], v[1], count).tolist()
            cols[k][:2] = v
        else:
            cols[k] = r.integers(v[0], v[1] + 1, count).tolist()
            cols[k][:2] = v
    for i in range(count):
        yield i, {k: c[i] for k, c in cols.items()}


def load(name):
    """dict of the arrays of tests/golden/reference_<name>.npz"""
    if name not in _CACHE:
        with np.load(os.path.join(GOLD, "reference_%s.npz" % name)) as z:
            _CACHE[name] = {k: z[k] for k in z.files}
    return _CACHE[name]
