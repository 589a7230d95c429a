"""The device wavefront pipeline on hardware: rtx_opd_regrid against the numpy
restatement (oracle/psf_oracle.py), rtx_psf against the reference's numpy
expression (rayopt/geometric_trace.py:150-157), and the resident drop-in's
opd_map / psf_device against the reference's own opd() / psf()."""
import warnings

import numpy as np
import pytest
import yaml

import psf_oracle as po
import ref_shim
import systems_yaml
from test_psf_oracle import REGRID_VS_GRIDDATA

pytestmark = pytest.mark.gpu
needs_ref = pytest.mark.skipif(not ref_shim.available(), reason="no reference tree")


@pytest.fixture(scope="module")
def eng():
    from rayopt_b200.engine import Engine
    e = Engine(0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def R():
    warnings.simplefilter("ignore")
    np.seterr(all="ignore")
    return ref_shim.load()


def build(R, name):
    s = R.System(**yaml.safe_load(systems_yaml.SYSTEMS[name]))
    s.update()
    if name != "mirror":
        s.paraxial.refocus()
    return s


def resident(R, eng, name, field, nrays, clip=True, filter=None):
    from rayopt_b200 import bind
    t = bind(R.GeometricTrace, engine=eng, exact=True, resident=True)(build(R, name))
    t.rays_point((0, field), nrays=nrays, distribution="hexapolar", clip=clip, filter=filter)
    return t


@needs_ref
@pytest.mark.parametrize("name,field,nrays", [
    ("double_gauss", 0., 1000), ("double_gauss", .7, 1000), ("double_gauss", 1., 1000),
    ("double_gauss", 0., 100000), ("double_gauss", .7, 100000), ("double_gauss", 1., 100000),
    ("cooke_asph", .7, 5000), ("mirror", .5, 5000)])
def test_regrid_matches_oracle(R, eng, name, field, nrays):
    """clip=True: vignetted rays are NaN and their triangles are dropped"""
    t = resident(R, eng, name, field, nrays)
    rings = t._hex_rings
    assert rings is not None and t.nrays == 1 + 3*rings*(rings + 1)
    A, P, a_ref, p_ref, lscale = t._opd_device()
    x, y, o = po.ray_xyt(A.download(), P.download(), a_ref, p_ref, lscale)
    n = int(4*t.nrays**.5)
    h, count = po.bounds(x, y, o)
    want = po.regrid(x, y, o, rings, n, h)
    m1, h1, c1 = eng.opd_regrid(A, P, a_ref, p_ref, lscale, rings, n)
    m2, h2, c2 = eng.opd_regrid(A, P, a_ref, p_ref, lscale, rings, n)
    got, again = m1.download(), m2.download()
    for d in (A, P, m1, m2):
        d.free()
    assert (h1, c1) == (h, count) == (h2, c2)
    assert np.array_equal(got.view(np.int64), again.view(np.int64))      # run to run
    assert np.array_equal(np.isnan(got), np.isnan(want))
    assert np.nanmax(np.abs(got - want)) <= 1e-12
    assert np.isfinite(got).sum() > 0.2*n*n


def reference_psf(o, pad):
    good = np.isfinite(o)
    g = np.where(good, np.exp(-2j*np.pi*np.where(good, o, 0)), 0)/np.count_nonzero(good)**.5
    a = np.fft.fft2(g, (pad*o.shape[0],)*2)
    return (a*a.conj()).real/a.size


def smooth_map(n, seed):
    u, v = np.mgrid[-1:1:1j*n, -1:1:1j*n]
    rng = np.random.default_rng(seed)
    c = rng.standard_normal(6)
    o = c[0]*u + c[1]*v + c[2]*(u*u + v*v) + c[3]*u*v + .3*c[4]*(u*u + v*v)**2 + .1*c[5]*u**3
    o[u*u + v*v > 1] = np.nan
    return o


@pytest.mark.parametrize("n,pad", [(126, 4), (127, 4), (997, 4), (4000, 4)])
def test_psf_of_a_given_map(eng, n, pad):
    """M = pad n = 504, 508, 4*997 (prime) and 16000: Bluestein in one tile
    and in the four-step split"""
    o = smooth_map(n, n)
    d_o = eng.to_device(o)
    d_psf = eng.psf(d_o, pad)
    got = d_psf.download()
    d_o.free()
    d_psf.free()
    M = pad*n
    assert got.shape == (M, M)
    assert abs(got.sum() - 1) <= 1e-12                  # Parseval, the reference's normalisation
    if M <= 4000:
        want = reference_psf(o, pad)
    else:                                               # fft2 is separable: exact columns
        good = np.isfinite(o)
        g = np.where(good, np.exp(-2j*np.pi*np.where(good, o, 0)), 0)/np.count_nonzero(good)**.5
        cols = np.r_[0:8, M//2 - 4:M//2 + 4, np.random.default_rng(0).integers(0, M, 48)]
        rows = np.fft.fft(g, M, axis=1)[:, cols]
        a = np.fft.fft(rows, M, axis=0)
        want = (a*a.conj()).real/(M*M)
        got = got[:, cols]
        assert np.abs(want).max() > 0.5*got.max()
    assert np.abs(got - want).max() <= 1e-12*want.max()


@needs_ref
@pytest.mark.parametrize("name,field,nrays", [("double_gauss", .7, 2000), ("cooke", 1., 1500)])
def test_end_to_end_against_the_reference(R, eng, name, field, nrays):
    ref = R.GeometricTrace(build(R, name))
    kw = dict(nrays=nrays, distribution="hexapolar", clip=True)
    ref.rays_point((0, field), **kw)
    got = resident(R, eng, name, field, nrays)
    # opd_map with host regridding is today's opd()
    host = got.opd(radius=got.system[-1].distance)
    for a, b in zip(got.opd_map(regrid="host", radius=got.system[-1].distance), host):
        assert np.array_equal(a, b, equal_nan=True)
    # host regridding: the device FFT of that map is the reference's expression
    p0, q0, want = ref.psf()
    p1, q1, psf = got.psf_device(regrid="host")
    assert np.abs(psf - reference_psf(host[2], 4)).max() <= 1e-12*psf.max()
    # and the reference's psf() within what the per-ray OPD allows: the
    # resident per-ray OPD agrees with the reference's to 1e-8 waves at a node
    # (tests/test_gpu_dropin_reference.py), and sum |dpsf| <= 4 pi |do|
    t0 = ref.opd(radius=ref.system[-1].distance)[2]
    assert np.array_equal(np.isnan(t0), np.isnan(host[2]))
    assert np.nanmax(np.abs(t0 - host[2])) <= 1e-8
    assert np.abs(psf - want).sum() <= 4*np.pi*1e-8
    np.testing.assert_allclose(p1, p0, rtol=1e-12)
    np.testing.assert_allclose(q1, q0, rtol=1e-12)
    # device regridding: the same node grid; vignetted gaps stay NaN
    xs, ys, t = got.opd_map()
    x0, y0, _ = ref.opd()
    np.testing.assert_allclose(xs, x0, rtol=1e-12)
    np.testing.assert_allclose(ys, y0, rtol=1e-12)
    assert np.isnan(t).sum() >= np.isnan(ref.opd()[2]).sum()
    p2, q2, psf2 = got.psf_device()
    np.testing.assert_allclose(p2, p0, rtol=1e-12)
    assert abs(psf2.sum() - 1) <= 1e-12


@needs_ref
@pytest.mark.parametrize("name,field", [("double_gauss", 0.), ("double_gauss", 1.), ("cooke", .7)])
def test_device_regrid_psf_within_the_measured_bound(R, eng, name, field):
    """Unvignetted unfiltered bundles: the device map has griddata's NaN mask
    and differs at a node by at most tol = REGRID_VS_GRIDDATA ptp/N waves (the
    CPU measurement, tests/test_psf_oracle.py).  With |dg| <= 2 pi tol |g| per
    pupil sample and sum |g|^2 = 1, Parseval bounds sum |dpsf| <= 4 pi tol,
    which bounds the peak change and the centroid shift."""
    nrays = 2000
    ref = R.GeometricTrace(build(R, name))
    kw = dict(nrays=nrays, distribution="hexapolar", clip=False, filter=False)
    ref.rays_point((0, field), **kw)
    got = resident(R, eng, name, field, nrays, clip=False, filter=False)
    assert got._hex_rings is not None
    x, y, o = ref.opd(resample=False)
    ok = np.isfinite(o)
    assert ok.all()
    # plus the 1e-8 waves of the resident per-ray OPD
    tol = REGRID_VS_GRIDDATA*np.ptp(o)/len(o) + 1e-8
    _, _, t_ref = ref.opd()
    _, _, t_dev = got.opd_map(regrid="device")
    assert np.array_equal(np.isnan(t_ref), np.isnan(t_dev))
    assert np.nanmax(np.abs(t_ref - t_dev)) <= tol
    # psf() measures the OPD against a sphere of radius system[-1].distance
    o = ref.opd(radius=ref.system[-1].distance, resample=False)[2]
    tol = REGRID_VS_GRIDDATA*np.ptp(o)/len(o) + 1e-8
    p, q, want = ref.psf()
    p2, q2, psf = got.psf_device(regrid="device")
    np.testing.assert_allclose(p2, p, rtol=1e-12)
    np.testing.assert_allclose(q2, q, rtol=1e-12)
    tv = np.abs(psf - want).sum()
    assert tv <= 4*np.pi*tol
    assert abs(psf.max() - want.max()) <= 4*np.pi*tol
    for c in (p, q):
        assert abs((c*psf).sum() - (c*want).sum()) <= np.abs(c).max()*4*np.pi*tol
    assert abs(psf.sum() - 1) <= 1e-12 and abs(want.sum() - 1) <= 1e-12


@needs_ref
def test_regrid_choice(R, eng):
    from rayopt_b200 import bind
    t = bind(R.GeometricTrace, engine=eng, resident=True)(build(R, "double_gauss"))
    t.rays_point((0, .5), nrays=300, distribution="square", clip=True)
    assert t._hex_rings is None
    with pytest.raises(ValueError):
        t.opd_map(regrid="device")
    x, y, o = t.opd_map()                               # host path
    assert np.array_equal(o, t.opd()[2], equal_nan=True)
    t.rays_point((0, .5), nrays=300, distribution="hexapolar")   # filter = not clip = True
    assert t._hex_rings is None
    t.rays_point((0, .5), nrays=300, distribution="hexapolar", clip=True)
    assert t._hex_rings == 9
    t.rays_given(np.asarray(t.y[0]), np.asarray(t.u[0]))
    assert t._hex_rings is None
    with pytest.raises(ValueError):
        t.opd_map(regrid="sideways")


@needs_ref
def test_no_rays_made_it_through(R, eng):
    t = resident(R, eng, "double_gauss", .5, 300)
    t.system[1].radius = 1e-9                             # a closed first aperture
    t.propagate(clip=True)
    for fn in (lambda: t.opd_map(regrid="device"), lambda: t.psf_device()):
        with pytest.raises(ValueError, match="no rays made it through"):
            fn()
