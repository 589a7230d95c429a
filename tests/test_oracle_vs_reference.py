"""Pins the oracle AND the table packer against the reference: the packer
reads the reference's System as stored in tests/golden/pins/oracle.json, the
oracle traces the reference's launch rays, and the trace must equal the
reference's (tests/golden/make_reference_pins.py, pins.py)."""
import numpy as np
import pytest

import np_oracle
import pins
from rayopt_b200.rays import aim_infinite, disc
from rayopt_b200.surface_table import pack_system

META, ARRAYS = pins.load("oracle")


@pytest.mark.parametrize("name,n,clip", [
    ("cooke", 20000, False), ("double_gauss", 20000, True),
    ("zoom", 10000, True), ("cooke_asph", 400, True), ("mirror", 5000, False),
    ("singlet", 5000, True)])
def test_bitwise_vs_live_reference(name, n, clip):
    rec = META[name]
    assert rec["n"] == n and rec["clip"] == clip
    s = pins.PinnedSystem(rec)
    with np.errstate(all="ignore"):
        for li, w in enumerate(rec["wavelengths"]):
            y0, u0 = aim_infinite((0, .7), disc(n, 1), w["z"], w["p"], rec["angle"])
            assert pins.digest(y0) == w["y0"] and pins.digest(u0) == w["u0"]
            table, nn, rot0 = pack_system(s, w["l"])
            Y, U, I, T = np_oracle.trace(table, y0, u0, clip=clip, rot0=rot0)
            assert np.array_equal(nn, w["n"])
            exact = name != "cooke_asph"   # Newton fprime uses np.dot (BLAS)
            for k, a in zip("yuit", (Y, U, I, T)):
                if exact:
                    assert pins.digest(a) == w[k], k
                else:
                    assert pins.digest(np.isnan(a)) == w["nan_" + k], k
                    b = ARRAYS["%s_%d_%s" % (name, li, k)]
                    a = a[:, pins.sample_rows(n)]
                    assert np.array_equal(np.isnan(a), np.isnan(b))
                    np.testing.assert_allclose(a, b, rtol=1e-13, atol=1e-13)
