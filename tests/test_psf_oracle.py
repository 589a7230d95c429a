"""CPU checks of the numpy restatement of the device wavefront pipeline
(oracle/psf_oracle.py): the hexapolar triangulation, the Bluestein FFT, and
the regridding against scipy's griddata on the reference's own bundles."""
import warnings

import numpy as np
import pytest

import psf_oracle as po
import ref_shim


@pytest.mark.parametrize("rings", [1, 2, 5, 16, 40])
def test_hex_triangulation(rings):
    from rayopt_b200.rays import hexapolar
    N = 1 + 3*rings*(rings + 1)
    R, xy = hexapolar(N)
    assert R == rings and po.rings_of(N) == rings
    tri = po.hex_triangles(rings)
    assert tri.shape == (6*rings*rings, 3)
    assert tri.min() == 0 and tri.max() == N - 1
    p = xy[tri]
    area2 = ((p[:, 1, 0] - p[:, 0, 0])*(p[:, 2, 1] - p[:, 0, 1])
             - (p[:, 2, 0] - p[:, 0, 0])*(p[:, 1, 1] - p[:, 0, 1]))
    # non-degenerate and consistently oriented in launch-pupil coordinates
    assert np.all(np.abs(area2) > 1e-3/rings**2)
    assert np.all(np.sign(area2) == np.sign(area2[0]))
    # they tile the outer-ring polygon (6R-gon of radius 1)
    outer = 0.5*6*rings*np.sin(2*np.pi/(6*rings))
    assert abs(np.abs(area2).sum()/2 - outer) < 1e-12
    # every interior edge is shared by exactly two triangles
    e = np.sort(np.concatenate([tri[:, [0, 1]], tri[:, [1, 2]], tri[:, [2, 0]]]), 1)
    _, cnt = np.unique(e, axis=0, return_counts=True)
    assert cnt.max() == 2 and (cnt == 1).sum() == 6*rings


@pytest.mark.parametrize("M", [504, 508, 4*997, 16000])
def test_bluestein_matches_numpy(M):
    rng = np.random.default_rng(M)
    x = rng.standard_normal((2, M)) + 1j*rng.standard_normal((2, M))
    want = np.fft.fft(x)
    scale = np.abs(want).max()
    assert np.abs(po.bluestein(x, M) - want).max() <= 1e-12*scale
    # the pruned first pass: a quarter of the input non-zero
    xq = x[:, :M//4]
    assert np.abs(po.bluestein(xq, M) - np.fft.fft(xq, M)).max() <= 1e-12*scale


def test_psf_restatement_matches_the_reference_expression():
    rng = np.random.default_rng(1)
    o = rng.standard_normal((37, 37))*.3
    o[np.hypot(*np.mgrid[-1:1:37j, -1:1:37j]) > 1] = np.nan
    good = np.isfinite(o)
    g = np.where(good, np.exp(-2j*np.pi*o), 0)/np.count_nonzero(good)**.5
    a = np.fft.fft2(g, (148, 148))                     # geometric_trace.py:150-157
    want = (a*a.conj()).real/a.size
    got = po.psf(o, 4)
    assert np.abs(got - want).max() <= 1e-12*want.max()
    assert abs(got.sum() - 1) < 1e-12


def test_nodes_are_numpy_mgrid():
    for n in (2, 121, 564, 4000):
        h = 18.61234
        xs, ys = np.mgrid[-1:1:1j*n, -1:1:1j*n]*h
        nd = po.nodes(n, h)
        assert np.array_equal(xs[:, 0], nd) and np.array_equal(ys[0], nd)


# Interpolation difference between the structured hexapolar triangulation and
# scipy's Delaunay triangulation (griddata), measured with the reference on
# the CPU over Double-Gauss, Cooke and Cooke + aspheres at fields 0 / 0.7 / 1
# with 919 and 19927 rays (unvignetted, unfiltered): the NaN masks are
# identical, and the largest difference at a node is 1.7e-3 waves (Cooke +
# aspheres, field 0.7, 19927 rays; 2.9e-2 at 919 rays).  The two
# triangulations differ only in nearly cocircular quads, where the difference
# is of order h^2 |grad^2 OPD| with h the ring spacing, i.e. ptp(OPD)/N: the
# measured worst case is 2.1 ptp/N.  The bound below is twice that.
REGRID_VS_GRIDDATA = 4.0


def reference_bundle(R, name, field, nrays, clip=False):
    import yaml
    import systems_yaml
    s = R.System(**yaml.safe_load(systems_yaml.SYSTEMS[name]))
    s.update()
    s.paraxial.refocus()
    t = R.GeometricTrace(s)
    t.rays_point((0, field), nrays=nrays, distribution="hexapolar", clip=clip, filter=False)
    return t


@pytest.mark.skipif(not ref_shim.available(), reason="no reference tree")
@pytest.mark.parametrize("name", ["double_gauss", "cooke"])
@pytest.mark.parametrize("field", [0., .7, 1.])
def test_regrid_matches_griddata(name, field):
    from scipy.interpolate import griddata
    warnings.simplefilter("ignore")
    with np.errstate(all="ignore"):
        R = ref_shim.load()
        t = reference_bundle(R, name, field, 2000)
        x, y, o = t.opd(resample=False)
        N = len(x)
        h, count = po.bounds(x, y, o)
        assert count == N
        n = int(4*N**.5)
        got = po.regrid(x, y, o, po.rings_of(N), n, h)
        ok = np.isfinite(x) & np.isfinite(y) & np.isfinite(o)
        xs, ys = np.mgrid[-1:1:1j*n, -1:1:1j*n]*h
        want = griddata((x[ok], y[ok]), o[ok], (xs, ys), method="linear", fill_value=np.nan)
        # the reference's own resampled opd() is the same griddata
        assert np.array_equal(want, t.opd()[2], equal_nan=True)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    tol = REGRID_VS_GRIDDATA*np.ptp(o[ok])/N
    assert np.nanmax(np.abs(got - want)) <= tol
