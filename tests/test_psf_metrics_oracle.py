"""The PSF figures of Analysis.opds (rayopt/analysis.py:319-346) on the CPU:
the literal restatement (oracle/psf_metrics_oracle.py: analysis_opds) against the
reference's own special_sums.polar_sum, and the definitions the device
reproduces (psf_metrics) against that restatement."""
import importlib

import numpy as np
import pytest

import psf_metrics_oracle as po
import ref_shim
from test_gpu_psf import reference_psf, smooth_map

needs_ref = pytest.mark.skipif(not ref_shim.available(), reason="no reference tree")


def random_psf(M, seed):
    psf = np.random.default_rng(seed).random((M, M))**4
    return psf/psf.sum()


def smooth_psf(M):
    """the PSF of test_gpu_psf.smooth_map at pad 4 (pad 3 when 4 does not divide M)"""
    pad = 4 if M % 4 == 0 else 3
    return reference_psf(smooth_map(M//pad, M//pad), pad)


def grids(M, d):
    f = np.fft.fftfreq(M, d)
    return np.broadcast_arrays(f[:, None], f[None, :])


@needs_ref
@pytest.mark.parametrize("M", [64, 127, 504])
def test_analysis_opds_is_the_reference_polar_sum(monkeypatch, M):
    """bin index element for element, sums to 1e-15; the reference needs
    np.int and bincount(minlength=None), gone in numpy 2"""
    ref_shim.load()
    special_sums = importlib.import_module("rayopt.special_sums")
    psf = random_psf(M, M)
    p, q = grids(M, .013)
    got = po.analysis_opds(psf, p, q)
    seen = {}
    bincount = np.bincount

    def bincount_numpy1(x, weights=None, minlength=None):
        seen["k"] = np.array(x)
        return bincount(x, weights, 0 if minlength is None else minlength)
    monkeypatch.setattr(np, "int", np.int64, raising=False)
    monkeypatch.setattr(np, "bincount", bincount_numpy1)
    want = special_sums.polar_sum(np.fft.fftshift(psf), got["center"], "azimuthal")
    monkeypatch.undo()
    assert np.array_equal(seen["k"], got["k"].ravel())
    assert want.shape == got["ee"].shape
    assert np.abs(np.cumsum(want) - got["ee"]).max() <= 1e-15
    assert abs(got["ee"][-1] - 1) <= 1e-12


@pytest.mark.parametrize("kind", ["random", "smooth"])
@pytest.mark.parametrize("M", [504, 381, 3988])
def test_psf_metrics_agrees_with_analysis_opds(M, kind):
    psf = random_psf(M, M) if kind == "random" else smooth_psf(M)
    d = 1/(M*.7e-3)
    p, q = grids(M, d)
    got = po.psf_metrics(psf, d, window=7)
    want = po.analysis_opds(psf, p, q)
    fmax = np.abs(p).max()
    total = psf.sum()
    # centroid: two orders of one sum of M^2 non-negative terms
    for k in ("x0", "y0"):
        assert abs(got[k] - want[k]) <= 2*M*M*2**-53*fmax*total
    assert abs(got["dx"] - want["dx"]) <= 4*2**-53*abs(want["dx"])
    assert np.abs(np.array(got["center"]) - np.array(want["center"])).max() <= 1e-9
    assert got["peak"] == want["peak"]
    # encircled energy at the same center: the per-element bin is the same,
    # the sums differ by the fixed-point rounding and the FP64 bincount
    at = po.analysis_opds(psf, p, q, center=got["center"])
    assert got["nbins"] == at["ee"].size
    _, k = po.ee_bins(psf, *got["center"], got["nbins"])
    assert np.array_equal(k, at["k"])
    tol = M*M*2.**-63 + (M*M + got["nbins"])*2.**-53*total
    assert np.abs(got["ee"] - at["ee"]).max() <= tol
    assert abs(got["ee"][-1] - total) <= tol
    np.testing.assert_allclose(got["r"], at["r"], rtol=1e-12)
    # MTF along both axes, Analysis's order psf.sum(0), psf.sum(1)
    assert got["mtf"].shape == want["mtf"].shape == (2, M//2)
    assert np.abs(got["mtf"] - want["mtf"]).max() <= 1e-13
    np.testing.assert_allclose(got["freq"], want["freq"], rtol=1e-12)
    # the window: the shifted PSF around the centroid node, coordinates - x0
    x, y, w = got["window"]
    ic, jc = int(np.floor(got["center"][0] + .5)), int(np.floor(got["center"][1] + .5))
    xs, ys, s = map(np.fft.fftshift, (p, q, psf))
    rows, cols = np.arange(ic - 7, ic + 8) % M, np.arange(jc - 7, jc + 8) % M
    assert np.array_equal(w, s[np.ix_(rows, cols)])
    assert np.array_equal(x, xs[np.ix_(rows, cols)] - got["x0"])
    assert np.array_equal(y, ys[np.ix_(rows, cols)] - got["y0"])


def test_fixed_point_encircled_energy_is_exact_integer_arithmetic():
    """the bins are the rint(psf 2^62) summed exactly, whatever the order"""
    psf = random_psf(64, 1)
    c = (32.3, 31.9)
    bins, k = po.ee_bins(psf, *c)
    s = np.fft.fftshift(psf)
    q = np.rint(s*2.**62).astype(np.uint64)
    perm = np.random.default_rng(2).permutation(q.size)
    again = np.zeros_like(bins)
    np.add.at(again, k.ravel()[perm], q.ravel()[perm])
    assert np.array_equal(bins, again)
    assert abs(float(bins.sum())/2.**62 - psf.sum()) <= 64*64*2.**-63
    with pytest.raises(ValueError):
        po.psf_metrics(psf, 1., window=32)
