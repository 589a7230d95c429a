"""numpy restatement of the PSF figures (rtx_psf_lines, rtx_psf_encircled,
rtx_psf_mtf, rtx_psf_window in rayopt_b200/csrc/rtx_psf.cuh).

TEST INFRASTRUCTURE ONLY; never imported by rayopt_b200/.

* ``psf_metrics``: the figures of Engine.psf_metrics (line sums, centroid,
  fixed-point encircled energy, |DFT| of the line sums, the window) in numpy;
  ``ee_bins`` is its encircled-energy histogram, bit for bit the device's.
* ``analysis_opds``: the same figures as Analysis.opds (rayopt/analysis.py:
  319-346) computes them, restated literally for numpy 2.
"""
import math

import numpy as np

EE_ONE = 2.0**62


def ee_bins(psf, c0, c1, nbins=None):
    """rtx_psf_encircled on the UNSHIFTED psf: shifted node (I, J) adds
    rint(psf*2^62) (uint64) to bin trunc(sqrt((J - c1)^2 + (I - c0)^2));
    np.add.at makes the integer sums exact.  Returns (bins, per-element bin of
    the shifted array)"""
    s = np.fft.fftshift(psf)
    M0, M1 = s.shape
    I, J = np.ogrid[:M0, :M1]
    dj, di = J - c1, I - c0
    k = np.sqrt(dj*dj + di*di).astype(np.int64)
    if nbins is None:
        nbins = int(k.max()) + 1
    q = np.rint(s*EE_ONE).astype(np.uint64)
    bins = np.zeros(nbins, np.uint64)
    np.add.at(bins, k.ravel(), q.ravel())
    return bins, k


def psf_metrics(psf, d, window=0):
    """Engine.psf_metrics in numpy on the unshifted (M, M) psf with frequency
    spacing fftfreq(M, d): dict of x0, y0, dx, center, nbins, peak, bins, ee,
    r, freq, mtf, lines and window (None or (x, y, psf), 2w+1 nodes a side)"""
    M = psf.shape[0]
    cols, rows = psf.sum(0), psf.sum(1)
    f = np.fft.fftfreq(M, d)
    x0, y0 = math.fsum(f*rows), math.fsum(f*cols)
    fs = np.fft.fftshift(f)
    dx = fs[1] - fs[0]
    c0, c1 = M/2 + x0/dx, M/2 + y0/dx
    corner = np.array([0., M - 1.])
    rc = np.sqrt((corner[None, :] - c1)*(corner[None, :] - c1)
                 + (corner[:, None] - c0)*(corner[:, None] - c0))
    nbins = int(rc.max()) + 1
    bins, _ = ee_bins(psf, c0, c1, nbins)
    lines = np.stack([cols, rows])
    win = None
    if window:
        w = int(window)
        if w > (M - 1)//2:
            raise ValueError("window too large")
        side = 2*w + 1
        ii = (math.floor(c0 + .5) - w + np.arange(side)) % M
        jj = (math.floor(c1 + .5) - w + np.arange(side)) % M
        s = np.fft.fftshift(psf)
        win = tuple(np.broadcast_arrays((fs[ii] - x0)[:, None], (fs[jj] - y0)[None, :])) \
            + (s[np.ix_(ii, jj)],)
    return dict(x0=x0, y0=y0, dx=dx, center=(c0, c1), nbins=nbins, peak=psf.max(), bins=bins,
                ee=np.cumsum(bins)/EE_ONE, r=np.arange(nbins)*dx,
                freq=np.fft.fftfreq(M, dx)[:M//2], mtf=np.abs(np.fft.fft(lines))[:, :M//2],
                lines=lines, window=win)


def polar_sum_azimuthal(m, center):
    """special_sums.polar_sum(m, center, "azimuthal") (rayopt/special_sums.py:
    153-265, aspect=1, binsize=None) restated for numpy 2: int64 for np.int and
    bincount's default minlength.  Returns (sums, per-element bin)"""
    m = np.atleast_2d(m)
    i, j = np.ogrid[:m.shape[0], :m.shape[1]]
    i, j = i - center[0], j - center[1]
    aspect = 1.
    k = (j**2*aspect**2 + i**2)**.5
    binsize = min(1., aspect)
    k = (k/binsize).astype(np.int64)
    return np.bincount(k.ravel(), m.ravel()), k


def analysis_opds(psf, p, q, center=None):
    """the PSF figures of Analysis.opds (rayopt/analysis.py:319-346) restated
    literally on psf() = (p, q, psf); `center` overrides the polar_sum center.
    Returns a dict of x0, y0, dx, center, peak, ee, r, rm, freq, mtf (2, M//2)
    and the per-element bin k"""
    x, y, psf = map(np.fft.fftshift, (p, q, psf))
    x0 = (psf*x).sum()
    y0 = (psf*y).sum()
    x, y = x - x0, y - y0
    dx = x[1, 0] - x[0, 0]
    if center is None:
        center = (psf.shape[0]/2 + x0/dx, psf.shape[1]/2 + y0/dx)
    ee, k = polar_sum_azimuthal(psf, center)
    ee = np.cumsum(ee)
    rm = np.searchsorted(ee, .9)*1.5*dx
    xe = np.arange(ee.size)*dx
    mtf, freq = [], None
    for i in (0, 1):
        ot = np.fft.ifft(np.fft.ifftshift(psf.sum(i))*psf.size**.5)
        of = np.fft.fftfreq(ot.size, dx)
        ot, of = ot[:ot.size//2], of[:of.size//2]
        mtf.append(np.absolute(ot))
        freq = of
    return dict(x0=x0, y0=y0, dx=dx, center=center, peak=psf.max(), ee=ee, r=xe, rm=rm,
                freq=freq, mtf=np.array(mtf), k=k)
