"""Recorded runs of the unmodified reference (tests/golden/reference_runs.npz, written by tests/golden/make_reference_runs.py).

The tests that hold the project against the reference read the reference's side from this file, so they run on every checkout,
with or without a reference build.  Integer structure (constraint types and bodies, colour groups) is stored as SHA-256 digests and
compared exactly; floating-point results are stored for a fixed, seeded sample of rows, together with the scale the full array
gives the relative error (max |x_ref|, max |x_ref - x_start|), so that the sampled error is measured against the same yardstick as
the full one."""
import hashlib
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_runs.npz")
SAMPLE_ROWS = 128
PARAM_ROWS = 32
_data = None


def load():
    global _data
    if _data is None:
        with np.load(PATH) as f:
            _data = {k: f[k] for k in f.files}
    return _data


def get(key):
    return load()[key]


def digest(a, dtype):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a, dtype=dtype).tobytes()).digest(), np.uint8)


STRUCTURE = ("constraint types", "constraint bodies", "group offsets", "group members")


def structure_digest(types, bodies, off, ids):
    """[4, 32]: digests of the constraint types, the constraint bodies and the colour groups (offsets, members)."""
    return np.stack([digest(types, np.int32), digest(bodies, np.uint32), digest(off, np.uint32), digest(ids, np.uint32)])


def assert_structure(prefix, types, bodies, off, ids):
    """Constraint types, bodies and colour groups bit for bit equal to the reference's."""
    d = structure_digest(types, bodies, off, ids) == get(prefix + "structure")
    assert d.all(), "%s: %s differ from the reference's" % (prefix, [n for n, ok in zip(STRUCTURE, d.all(axis=1)) if not ok])


def sampled(prefix, name, a, k=SAMPLE_ROWS):
    """(the reference's sample recorded as prefix + name, the same rows of `a`, the scale of the reference's full array)."""
    a = np.asarray(a)
    return get(prefix + name), a[sample_rows(len(a), k)], float(get(prefix + name + "_scale"))


def sample_rows(n, k=SAMPLE_ROWS, seed=0):
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.RandomState(seed).choice(n, k, replace=False))
