"""The PSF figures on hardware (rtx_psf_lines, rtx_psf_encircled, rtx_psf_mtf,
rtx_psf_window; Engine.psf_metrics, ResidentMixin.psf_metrics) against the
numpy definitions in oracle/psf_metrics_oracle.py and, end to end, against
Analysis.opds's figures (rayopt/analysis.py:319-346) of the reference's own
psf()."""
import warnings

import numpy as np
import pytest

import psf_metrics_oracle as po
import ref_shim
from test_gpu_psf import build, resident, smooth_map

pytestmark = pytest.mark.gpu
needs_ref = pytest.mark.skipif(not ref_shim.available(), reason="no reference tree")

# (n, pad): M = 504 (one FFT tile), 381 (odd), 3988 and 5056 (four-step)
SIZES = [(126, 4), (127, 3), (997, 4), (1264, 4)]


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


@pytest.fixture(scope="module", params=SIZES, ids=lambda s: "M%d" % (s[0]*s[1]))
def device_psf(request, eng):
    """(DEVICE psf, its download) of smooth_map at M = pad n"""
    n, pad = request.param
    d_o = eng.to_device(smooth_map(n, n))
    d_psf = eng.psf(d_o, pad)
    d_o.free()
    yield d_psf, d_psf.download()
    d_psf.free()


def test_lines_and_stats(eng, device_psf):
    d_psf, psf = device_psf
    M = psf.shape[0]
    lines, peak, total, bad = eng.psf_lines(d_psf)
    got = lines.download()
    again = eng.psf_lines(d_psf, out=lines)[0].download()
    lines.free()
    assert np.array_equal(got.view(np.int64), again.view(np.int64))   # run to run
    for a in (0, 1):
        want = psf.sum(a)
        assert np.all(np.abs(got[a] - want) <= M*2.**-53*want)
    assert peak == psf.max()
    assert bad == 0
    assert abs(total - psf.sum()) <= M*M*2.**-53*psf.sum()


def test_encircled_bit_identical_to_the_oracle(eng, device_psf):
    d_psf, psf = device_psf
    M = psf.shape[0]
    m = eng.psf_metrics(d_psf, 1.)
    c0, c1 = M/2 + m.x0/m.dx, M/2 + m.y0/m.dx
    want, _ = po.ee_bins(psf, c0, c1, len(m.ee))
    got = eng.psf_encircled(d_psf, c0, c1, len(m.ee))
    again = eng.psf_encircled(d_psf, c0, c1, len(m.ee))
    assert got.dtype == np.uint64
    assert np.array_equal(got, want)
    assert np.array_equal(got, again)
    assert np.array_equal(m.ee, np.cumsum(want)/2.**62)
    # an off-centre centre: tiles far from it, bins spread over the histogram
    c = (M/2 + 0.37*M, M/2 - 0.21*M)
    want, _ = po.ee_bins(psf, *c)
    assert np.array_equal(eng.psf_encircled(d_psf, *c, len(want)), want)
    with pytest.raises(ValueError):
        eng.psf_encircled(d_psf, *c, len(want) - 1)


def test_mtf(eng, device_psf):
    d_psf, psf = device_psf
    M = psf.shape[0]
    lines = eng.psf_lines(d_psf)[0]
    d_mtf = eng.psf_mtf(lines)
    got, host = d_mtf.download(), lines.download()
    lines.free()
    d_mtf.free()
    want = np.abs(np.fft.fft(host))[:, :M//2]
    assert got.shape == (2, M//2)
    assert np.abs(got - want).max() <= 1e-12


def test_window(eng, device_psf):
    d_psf, psf = device_psf
    M = psf.shape[0]
    s = np.fft.fftshift(psf)
    for i0, j0, w in ((M//2 - 10, M//2 - 3, 21), (M - 5, -4, 17), (0, 0, M)):
        d_w = eng.psf_window(d_psf, i0, j0, w)
        got = d_w.download()
        d_w.free()
        want = s[np.ix_((i0 + np.arange(w)) % M, (j0 + np.arange(w)) % M)]
        assert np.array_equal(got, want)


def test_psf_metrics_against_the_oracle(eng, device_psf):
    d_psf, psf = device_psf
    M = psf.shape[0]
    d = 1/(M*.7e-3)
    got = eng.psf_metrics(d_psf, d, window=12)
    want = po.psf_metrics(psf, d, window=12)
    fmax = np.abs(np.fft.fftfreq(M, d)).max()
    for k in ("x0", "y0"):       # line sums within M 2^-53 of numpy's
        assert abs(getattr(got, k) - want[k]) <= 2*M*2.**-53*fmax
    assert got.dx == want["dx"]
    assert got.peak == want["peak"]
    assert len(got.ee) == want["nbins"]
    # EE at the device's own centre (a centre a few ulps away may move an
    # element that lies within 1e-11 of an integer radius to the next bin)
    c0, c1 = M/2 + got.x0/got.dx, M/2 + got.y0/got.dx
    assert np.array_equal(got.ee, np.cumsum(po.ee_bins(psf, c0, c1, len(got.ee))[0])/2.**62)
    assert abs(got.ee[-1] - psf.sum()) <= M*M*2.**-63 + 1e-14
    assert np.array_equal(got.r, want["r"])
    assert np.array_equal(got.freq, want["freq"])
    assert np.abs(got.mtf - want["mtf"]).max() <= 1e-12
    # the window around the node of the device's own centroid
    ii = (int(np.floor(c0 + .5)) - 12 + np.arange(25)) % M
    jj = (int(np.floor(c1 + .5)) - 12 + np.arange(25)) % M
    fs = np.fft.fftshift(np.fft.fftfreq(M, d))
    x, y, w = got.window
    assert np.array_equal(w, np.fft.fftshift(psf)[np.ix_(ii, jj)])
    assert np.array_equal(x, np.broadcast_to((fs[ii] - got.x0)[:, None], (25, 25)))
    assert np.array_equal(y, np.broadcast_to((fs[jj] - got.y0)[None, :], (25, 25)))


def test_rejections(eng):
    psf = np.full((64, 64), 1/64**2)
    for bad in (-1e-3, np.nan, 2.5):
        p = psf.copy()
        p[3, 5] = bad
        d = eng.to_device(p)
        with pytest.raises(ValueError):
            eng.psf_metrics(d, 1.)
        d.free()
    d = eng.to_device(psf*3)              # every element in [0, 2], the sum 3
    with pytest.raises(ValueError):
        eng.psf_metrics(d, 1.)
    d.free()
    d = eng.to_device(psf)
    with pytest.raises(ValueError):
        eng.psf_metrics(d, 1., window=32)     # > (M - 1)//2 = 31
    assert eng.psf_metrics(d, 1., window=31).window[2].shape == (63, 63)
    d.free()


@needs_ref
@pytest.mark.parametrize("name,field,nrays", [("double_gauss", .7, 2000), ("cooke", 1., 2000)])
def test_end_to_end_against_analysis_opds(R, eng, name, field, nrays):
    """psf_metrics(regrid="host") against Analysis.opds's figures of the
    reference's own psf().  The two PSFs differ by sum |dpsf| <= 4 pi 1e-8
    (test_gpu_psf.test_end_to_end_against_the_reference); that bounds the
    change of the centroid (times max |x|), the peak, every EE value and every
    |DFT| of a line sum.  EE is compared at the device's centre: a centre a
    few ulps away can move an element within 1e-11 of an integer radius."""
    ref = R.GeometricTrace(build(R, name))
    ref.rays_point((0, field), nrays=nrays, distribution="hexapolar", clip=True)
    p, q, want_psf = ref.psf()
    got = resident(R, eng, name, field, nrays)
    m = got.psf_metrics(regrid="host", window=20)
    M = want_psf.shape[0]
    tv = 4*np.pi*1e-8
    want = po.analysis_opds(want_psf, p, q)
    assert abs(m.x0 - want["x0"]) <= np.abs(p).max()*tv
    assert abs(m.y0 - want["y0"]) <= np.abs(q).max()*tv
    assert abs(m.dx - want["dx"]) <= 1e-12*abs(want["dx"])
    assert abs(m.peak - want["peak"]) <= tv
    np.testing.assert_allclose(m.freq, want["freq"], rtol=1e-12)
    assert np.abs(m.mtf - want["mtf"]).max() <= tv + 1e-12
    center = (M/2 + m.x0/m.dx, M/2 + m.y0/m.dx)
    at = po.analysis_opds(want_psf, p, q, center=center)
    assert len(m.ee) == len(at["ee"])
    assert np.abs(m.ee - at["ee"]).max() <= tv + 1e-12
    np.testing.assert_allclose(m.r, at["r"], rtol=1e-12)
    # the window is the shifted PSF of psf_device around the centroid node
    p1, q1, psf = got.psf_device(regrid="host")
    x, y, w = m.window
    ii = (int(np.floor(center[0] + .5)) - 20 + np.arange(41)) % M
    jj = (int(np.floor(center[1] + .5)) - 20 + np.arange(41)) % M
    xs, ys, s = map(np.fft.fftshift, (p1, q1, psf))
    assert np.array_equal(w, s[np.ix_(ii, jj)])
    assert np.array_equal(x, xs[np.ix_(ii, jj)] - m.x0)
    assert np.array_equal(y, ys[np.ix_(ii, jj)] - m.y0)
    # the device regridding path gives the same kind of result
    m2 = got.psf_metrics()
    assert abs(m2.ee[-1] - 1) <= 1e-9
