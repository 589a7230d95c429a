"""Stored results of the reference (quartiq/rayopt) for the tests that pin the
oracle, the table packer and the ray generator against it, so that those
tests run without the reference installed.  tests/golden/make_reference_pins.py
writes them from the live reference into tests/golden/pins/.

Arrays a test compares bit for bit are stored as a SHA-256 digest of their
canonical bytes (`digest`): equal digests <=> ``np.array_equal(a, b,
equal_nan=True)`` with equal shapes, at 64 bytes instead of the array.  Arrays
compared within a tolerance are stored as values (a fixed sample of rows
where the full array would be large, `sample_rows`).
"""
import hashlib
import json
import os
import types

import numpy as np

DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "pins")
SAMPLE_ROWS = 48


def digest(a):
    """SHA-256 of float64 `a` with every NaN made the same NaN and -0.0 made
    +0.0, and of its shape: two arrays have equal digests exactly when they
    have the same shape and are equal under ``np.array_equal(equal_nan=True)``"""
    a = np.asarray(a, np.float64)
    a = np.where(np.isnan(a), np.nan, a + 0.)
    h = hashlib.sha256(repr(a.shape).encode())
    h.update(np.ascontiguousarray(a, "<f8").tobytes())
    return h.hexdigest()


def sample_rows(n, k=SAMPLE_ROWS):
    """the fixed rows (along axis 0 of an n-row array) kept of a large array"""
    return np.unique(np.linspace(0, n - 1, min(n, k)).round().astype(np.int64))


def load(name):
    """(dict from <name>.json, dict of arrays from <name>.npz or {})"""
    with open(os.path.join(DIR, name + ".json")) as f:
        meta = json.load(f)
    path = os.path.join(DIR, name + ".npz")
    arrays = {}
    if os.path.exists(path):
        with np.load(path) as d:
            arrays = {k: d[k] for k in d.files}
    return meta, arrays


ATTRS = ("offset", "rotated", "rot_normal", "curvature", "conic", "alternate_intersection",
         "radius", "aspherics")


def element_attrs(e):
    """what the table packer reads of a reference element (JSON-able)"""
    out = {}
    for k in ATTRS:
        if hasattr(e, k):
            v = getattr(e, k)
            out[k] = None if v is None else (np.asarray(v, float).tolist() if np.ndim(v) else
                                             (bool(v) if isinstance(v, (bool, np.bool_)) else float(v)))
    return out


class PinnedElement:
    """an element of a reference System as the table packer reads it: the
    stored attributes and, for an element with a material, ``get_n_mu``
    answering with the reference's own (n, mu) for the index it is called
    with at each stored wavelength"""

    def __init__(self, attrs, n_mu=None):
        for k, v in attrs.items():
            setattr(self, k, np.asarray(v, float) if k in ("offset", "rot_normal") else v)
        if n_mu is not None:
            def get_n_mu(n0, l):
                n0_ref, n, mu = n_mu[repr(float(l))]
                assert n0 == n0_ref, (n0, n0_ref)
                return n, mu
            self.get_n_mu = get_n_mu


class PinnedSystem(list):
    """the element list of a reference System, as the table packer reads it"""

    def __init__(self, rec):
        super().__init__(PinnedElement(a, m) for a, m in zip(rec["elements"], rec["n_mu"]))
        self._n0 = rec["n0"]

    def refractive_index(self, l, i):
        assert i == 0
        return self._n0[repr(float(l))]


def conjugate(rec):
    """stand-in for a reference InfiniteConjugate / FiniteConjugate with the
    attributes rays.aim_record reads"""
    ns = types.SimpleNamespace(**rec)
    if "pupil" in rec:
        ns.pupil = types.SimpleNamespace(**rec["pupil"])
    return ns


def surface(rec):
    """stand-in for a reference Spheroid with the attributes rays.aim_record
    reads; ``surface_sag`` answers with the reference's sag at the one point
    it was evaluated at"""
    e = PinnedElement(rec["attrs"])
    if "sag" in rec:
        point, value = rec["sag"]

        def surface_sag(y):
            np.testing.assert_array_equal(y, point)
            return np.array([value])
        e.surface_sag = surface_sag
    return e
