"""Pins the ray-generator restatement (oracle/aim_oracle.py evaluating the
`rtx_aim` records of rayopt_b200/rays.py the way the CUDA kernels do) against
the LIVE reference: ``pupil_distribution`` (rayopt/utils.py:118-199),
``Pupil.map`` with and without its filter (rayopt/pupils.py:97-107),
``InfiniteConjugate.aim`` in all five projections with plane and curved object
surfaces, ``FiniteConjugate.aim`` with regular and telecentric pupils
(rayopt/conjugates.py:137-166, 208-255).  Bit-exact where no transcendental
function is evaluated per ray.  The reference's results are stored in
tests/golden/pins/aim.json/.npz (tests/golden/make_reference_pins.py): digests
of what is compared bit for bit, values (a fixed row sample of the larger
arrays) of what is compared within a tolerance."""
import numpy as np
import pytest

import aim_oracle
import pins
from rayopt_b200.rays import aim_record, grid_spec

P = np.array(((-3., -2.5), (2., 2.8)))          # pupil half-apertures [[-sag,-mer],[+sag,+mer]]
META, ARRAYS = pins.load("aim")
PLANE = pins.surface({"attrs": META["given"]["surface"]["attrs"]})


def infinite(angle, projection="rectilinear"):
    return pins.conjugate(dict(finite=False, angle=angle, projection=projection))


def assert_exact(got, want):
    assert list(np.shape(got)) == want["shape"], (np.shape(got), want["shape"])
    assert pins.digest(got) == want["digest"]


def assert_close(got, want, key, atol, sampled=True):
    assert list(np.shape(got)) == want["shape"], (np.shape(got), want["shape"])
    got = np.asarray(got)[pins.sample_rows(len(got))] if sampled else got
    np.testing.assert_allclose(got, ARRAYS[key], rtol=0, atol=atol, equal_nan=True)


@pytest.mark.parametrize("dist,n", [
    ("half-meridional", 7), ("meridional", 12), ("sagittal", 9), ("cross", 23), ("tee", 152),
    ("square", 500), ("triangular", 700), ("hexapolar", 400), ("meridional", 1)])
def test_grids_equal_pupil_distribution(dist, n):
    """the per-candidate formulas (k*step + start linspace / mgrid points, the
    unit-circle predicate, prepended centre ray) reproduce the reference grid
    bit for bit, in order, with the same `ref` index"""
    want = META["grids"]["%s-%d" % (dist, n)]
    r, grid = grid_spec(dist, n)
    assert r == want["ref"] and want["weight_is_none"]
    if grid is None:
        assert n == 1
        return
    rec = aim_record(infinite(.2), (0, .5), 30., P, grid)
    px, py, keep = aim_oracle.candidates(rec[0])
    got = np.c_[px[keep], py[keep]]
    if dist == "hexapolar":                       # sin/cos of the ring angles: last ulps
        assert_close(got, want["xy"], "grid_%s_%d" % (dist, n), 3e-16, sampled=False)
    else:
        assert_exact(got, want["xy"])


def test_quadrature_distributions_stay_on_the_host():
    for d in ("radau", "lobatto"):
        assert grid_spec(d, 13) == (0, None)


@pytest.mark.parametrize("filt", [False, True])
@pytest.mark.parametrize("projection", ["rectilinear", "stereographic", "equisolid",
                                        "orthographic", "equidistant"])
def test_infinite_conjugate_all_projections(projection, filt):
    obj = infinite(.35, projection)
    if projection == "orthographic":
        # the reference itself cannot aim this projection: conjugates.py:225-226
        # stacks a (n,1,1) array (``np.sqrt(1 - r)[:, None]`` with r already
        # (n,1)) and raises.  rays.project restates the evident intent
        # u = (y, sqrt(1 - |y|^2)); checked here for what it must satisfy.
        from rayopt_b200.rays import project
        u = project(np.array([[0, .7], [-.4, .9]]), .35, projection)
        np.testing.assert_allclose(np.square(u).sum(1), 1, rtol=0, atol=1e-15)
        np.testing.assert_allclose(u[:, :2], np.array([[0, .7], [-.4, .9]])*np.sin(.35))
        return
    for dist, n in (("square", 300), ("tee", 31), ("hexapolar", 200)):
        for yo in ((0., 0.), (0, .7), (-.4, .9)):
            key = "%s_%d_%s_%s_%g_%g" % (projection, filt, dist, n, yo[0], yo[1])
            want = META["infinite"][key]
            rec = aim_record(obj, yo, 25., P, grid_spec(dist, n)[1], filt, PLANE)
            with np.errstate(all="ignore"):
                y, u, pupil = aim_oracle.generate(rec)
            if dist == "hexapolar":
                assert_close(y, want["y"], key + "_y", 1e-14)
            else:
                assert_exact(y, want["y"])
            assert_exact(u, want["u"])


@pytest.mark.parametrize("kw", [dict(curvature=.02), dict(curvature=-.03, conic=-.6),
                                dict(curvature=.01, aspherics=[0, 2e-6, -1e-9])])
def test_infinite_conjugate_curved_object_surface(kw):
    """y += surface.intercept(y, u) u (conjugates.py:254) with a sphere, a conic
    and an asphere as system[0]"""
    i = [dict(curvature=.02), dict(curvature=-.03, conic=-.6),
         dict(curvature=.01, aspherics=[0, 2e-6, -1e-9])].index(kw)
    want = META["curved"]["kw%d" % i]
    surf = pins.surface(want["surface"])
    assert all(getattr(surf, k) == v for k, v in kw.items())
    rec = aim_record(infinite(.2), (0, .8), 20., P, grid_spec("square", 200)[1], True, surf)
    assert rec["curved"][0] == 1
    with np.errstate(all="ignore"):
        y, u, _ = aim_oracle.generate(rec)
    if "aspherics" in kw:                        # Newton: the reference's fprime is a BLAS dot
        assert_close(y, want["y"], "curved_%d_y" % i, 1e-13, sampled=False)
    else:
        assert_exact(y, want["y"])
    assert_exact(u, want["u"])


@pytest.mark.parametrize("telecentric", [False, True])
@pytest.mark.parametrize("z", [40., -35.])
def test_finite_conjugate(z, telecentric):
    """FiniteConjugate.aim: object point, pupil angles arctan2(a, z), tan() of
    the mapped coordinates (last ulps), telecentric pupils, curved object
    surfaces (y_z = -surface_sag), z < 0"""
    obj = pins.conjugate(dict(finite=True, radius=6., pupil=dict(telecentric=telecentric)))
    for j in range(2):
        for dist, n, filt in (("square", 300, True), ("cross", 21, False), ("triangular", 150, False)):
            key = "%d_%g_%d_%s" % (telecentric, z, j, dist)
            want = META["finite"][key]
            surf = pins.surface(want["surface"])
            rec = aim_record(obj, (.3, -.6), z, P, grid_spec(dist, n)[1], filt, surf)
            with np.errstate(all="ignore"):
                y, u, _ = aim_oracle.generate(rec)
            assert_exact(y, want["y"])
            assert_close(u, want["u"], "finite_%s_u" % key, 3e-16)


def test_given_pupil_coordinates_and_random():
    obj = infinite(.3)
    rng = np.random.default_rng(4)
    yp = rng.uniform(-1, 1, (500, 2))
    rec = aim_record(obj, (0, .5), 30., P, None, True, PLANE)
    y, u, pupil = aim_oracle.generate(rec, yp)
    assert 0 < len(y) < 500
    assert_exact(y, META["given"]["y"])
    assert_exact(u, META["given"]["u"])
    # "random": uniform in the unit disc, centre ray first, reproducible from the seed
    rec = aim_record(obj, (0, .5), 30., P, grid_spec("random", 4000)[1], False, None, seed=7)
    _, _, p1 = aim_oracle.generate(rec)
    _, _, p2 = aim_oracle.generate(rec)
    assert np.array_equal(p1, p2) and p1.shape == (4001, 2) and np.all(p1[0] == 0)
    r2 = np.square(p1[1:]).sum(1)
    assert r2.max() <= 1 and abs(r2.mean() - .5) < .02 and abs(p1[1:].mean()) < .02
    rec2 = aim_record(obj, (0, .5), 30., P, grid_spec("random", 4000)[1], False, None, seed=8)
    assert not np.array_equal(aim_oracle.generate(rec2)[2], p1)
