"""Host logic: table packer and the launch-ray generator (CPU)."""
import json

import numpy as np
import pytest

from conftest import load_golden
from rayopt_b200.rays import aim_infinite, disc
from rayopt_b200.surface_table import (SURFACE_DTYPE, pack_system, table_from_json,
                                       table_to_json, RTX_MAX_ASPH)


class FakeElement:
    def __init__(self, **kw):
        self.offset = np.array((0, 0, kw.pop("distance", 0.)))
        self.rotated = False
        self.radius = np.inf
        self.__dict__.update(kw)


class FakeSystem(list):
    wavelengths = [587e-9]

    def refractive_index(self, l, i):
        return 1.


def test_plain_element_is_a_non_refracting_plane():
    s = FakeSystem([FakeElement(), FakeElement(distance=3., radius=2.)])
    table, n, rot0 = pack_system(s, 587e-9)
    assert rot0 is None and len(table) == 1
    r = table[0]
    assert r["mu"] == 1 and r["c"] == 0 and r["n_asph"] == -1
    assert r["radius2"] == 4 and n[0] == 1 and r["offset"][2] == 3


def test_too_many_aspherics_rejected():
    s = FakeSystem([FakeElement(), FakeElement(aspherics=[0.]*(RTX_MAX_ASPH + 1))])
    with pytest.raises(ValueError):
        pack_system(s, 587e-9)


def test_json_roundtrip_is_lossless():
    c = load_golden("cooke_asph_f07_clip")
    t2 = table_from_json(json.loads(json.dumps(table_to_json(c["table"]))))
    assert t2.tobytes() == np.ascontiguousarray(c["table"], SURFACE_DTYPE).tobytes()


def test_aim_matches_reference_golden():
    c = load_golden("double_gauss_l0_clip")
    y, u = aim_infinite((0, .7), disc(256, 0), c["meta"]["z"], c["meta"]["p"],
                        np.deg2rad(14))
    assert np.array_equal(y, c["y0"]) and np.array_equal(u, c["u0"])


def test_aim_finite_restatement_vs_reference():
    """rays.aim_finite == FiniteConjugate.aim (rayopt/conjugates.py:137-166)
    bit for bit (the reference's results: tests/golden/pins/aim_finite.json)"""
    import pins
    from rayopt_b200.rays import aim_finite
    want, _ = pins.load("aim_finite")
    a = np.array(((-3., -2.5), (3., 2.5)))
    for z in (50., -40.):
        for yo in ((0, .7), (0., 0.), (.3, -.4)):
            hy, hu = aim_finite(yo, disc(500, 2), z, a, 5.)
            w = want["%g_%g_%g" % ((z,) + yo)]
            assert pins.digest(hy) == w["y"] and pins.digest(hu) == w["u"]
