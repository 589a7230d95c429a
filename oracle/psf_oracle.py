"""numpy restatement of the device wavefront pipeline (rayopt_b200/csrc/rtx_psf.cuh).

TEST INFRASTRUCTURE ONLY; never imported by rayopt_b200/.

* ``hex_triangles``: the structured triangulation of the hexapolar launch grid
  (pupil_distribution("hexapolar"), rayopt/utils.py:180-186) in the kernel's
  triangle order.
* ``regrid``: the OPD map of rtx_opd_regrid with the kernel's tie rule (a node
  takes the lowest-index triangle that contains it) and operation order, so
  that the device map equals it bit for bit.
* ``bluestein`` / ``psf``: the FFT algorithm of rtx_psf (radix-2 DIT in
  power-of-two tiles, four-step split above the tile size, chirp-z for every
  length) restated so that it can be validated against np.fft on the CPU.
"""
import numpy as np

BARY_EPS = 2.0**-40
FFT_TILE, FFT_L1 = 4096, 512


# ---- regridding -------------------------------------------------------------
def ring_ray(q, k):
    q, k = np.asarray(q, np.int64), np.asarray(k, np.int64)
    return np.where(q == 0, 0, 1 + 3*q*(q - 1) + k % np.maximum(6*q, 1))


def hex_triangles(rings):
    """(6 rings^2, 3) ray indices; triangles [6r^2, 6(r+1)^2) join ring r and
    ring r+1, 2r+1 per sector j: (i_m, o_m, o_m+1), (i_m, o_m+1, i_m+1) for
    m < r, then (i_r, o_r, o_r+1); i_m = r j + m, o_m = (r+1) j + m"""
    tid = np.arange(6*rings*rings, dtype=np.int64)
    r = np.floor(np.sqrt(tid/6.)).astype(np.int64)
    r = np.where(6*(r + 1)**2 <= tid, r + 1, r)
    r = np.where(6*r*r > tid, r - 1, r)
    w = tid - 6*r*r
    j = w//(2*r + 1)
    w = w - j*(2*r + 1)
    ib, ob, m = r*j, (r + 1)*j, w >> 1
    close, odd = w == 2*r, (w & 1) == 1
    v0 = ring_ray(r, np.where(close, ib + r, ib + m))
    v1 = ring_ray(r + 1, np.where(close, ob + r, np.where(odd, ob + m + 1, ob + m)))
    v2 = np.where(close, ring_ray(r + 1, ob + r + 1),
                  np.where(odd, ring_ray(r, ib + m + 1), ring_ray(r + 1, ob + m + 1)))
    return np.stack([v0, v1, v2], 1)


def rings_of(N):
    R = int(round((np.sqrt(12*N - 3) - 3)/6))
    if N != 1 + 3*R*(R + 1):
        raise ValueError("%d rays is not a hexapolar bundle" % N)
    return R


def ray_xyt(A, P, a_ref, p_ref, lscale):
    """per ray x, y = P - P[ref], t = -(A - A[ref])/(l/scale)"""
    return P[:, 0] - p_ref[0], P[:, 1] - p_ref[1], -(A - a_ref)/lscale


def bounds(x, y, t):
    """h and the number of rays with finite x, y, t (geometric_trace.py:135-139)"""
    ok = np.isfinite(x) & np.isfinite(y) & np.isfinite(t)
    if not ok.any():
        return 0., 0
    return float(np.fabs((x[ok], y[ok])).max()), int(ok.sum())


def nodes(n, h):
    """np.mgrid[-1:1:1j*n]*h as the kernel evaluates it: (k*step + -1)*h"""
    step = 2./(n - 1) if n > 1 else 1.
    return (np.arange(n, dtype=np.float64)*step + -1.)*h


def _tri_data(x, y, t, tri):
    X, Y, T = x[tri], y[tri], t[tri]
    ok = np.isfinite(X).all(1) & np.isfinite(Y).all(1) & np.isfinite(T).all(1)
    a = Y[:, 1] - Y[:, 2]
    b = X[:, 2] - X[:, 1]
    c = Y[:, 2] - Y[:, 0]
    e = X[:, 0] - X[:, 2]
    with np.errstate(invalid="ignore", over="ignore"):
        d = a*e + b*(Y[:, 0] - Y[:, 2])
    ok &= (d != 0) & np.isfinite(d)
    return X, Y, T, a, b, c, e, d, ok


def _bary(X, Y, a, b, c, e, d, px, py):
    dx, dy = px - X[:, 2], py - Y[:, 2]
    l0 = (a*dx + b*dy)/d
    l1 = (c*dx + e*dy)/d
    return l0, l1, (1. - l0) - l1


def regrid(x, y, t, rings, n, h=None):
    """rtx_opd_regrid on per-ray x, y, t: the (n, n) map, row i = x node"""
    if h is None:
        h = bounds(x, y, t)[0]
    step = 2./(n - 1) if n > 1 else 1.
    tri = hex_triangles(rings)
    X, Y, T, a, b, c, e, d, ok = _tri_data(x, y, t, tri)
    idx = np.nonzero(ok)[0]
    X, Y, T, a, b, c, e, d = (v[idx] for v in (X, Y, T, a, b, c, e, d))

    def krange(lo, hi):
        with np.errstate(invalid="ignore", divide="ignore"):
            u0 = np.floor((lo/h + 1.)/step) - 1.
            u1 = np.ceil((hi/h + 1.)/step) + 1.
        k0 = np.where(np.isnan(u0), 0, np.clip(u0, 0, n - 1)).astype(np.int64)
        k1 = np.where(np.isnan(u1), n - 1, np.clip(u1, 0, n - 1)).astype(np.int64)
        return k0, k1
    i0, i1 = krange(X.min(1), X.max(1))
    j0, j1 = krange(Y.min(1), Y.max(1))
    ni, nj = i1 - i0 + 1, j1 - j0 + 1
    owner = np.full(n*n, np.iinfo(np.int64).max, np.int64)
    node = nodes(n, h)
    # (triangle, candidate node) pairs, in chunks of triangles
    for s in range(0, len(idx), 1 << 16):
        sl = slice(s, s + (1 << 16))
        cnt = ni[sl]*nj[sl]
        k = np.repeat(np.arange(sl.start, sl.start + len(cnt)), cnt)
        off = np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt)
        ii = i0[k] + off//nj[k]
        jj = j0[k] + off % nj[k]
        with np.errstate(invalid="ignore", divide="ignore"):
            l0, l1, l2 = _bary(X[k], Y[k], a[k], b[k], c[k], e[k], d[k], node[ii], node[jj])
            inside = (l0 >= -BARY_EPS) & (l1 >= -BARY_EPS) & (l2 >= -BARY_EPS)
        np.minimum.at(owner, ii[inside]*n + jj[inside], idx[k[inside]])
    out = np.full(n*n, np.nan)
    hit = np.nonzero(owner != np.iinfo(np.int64).max)[0]
    o = owner[hit]
    X, Y, T, a, b, c, e, d, _ = _tri_data(x, y, t, tri[o])
    l0, l1, l2 = _bary(X, Y, a, b, c, e, d, node[hit//n], node[hit % n])
    out[hit] = (l0*T[:, 0] + l1*T[:, 1]) + l2*T[:, 2]
    return out.reshape(n, n)


# ---- FFT ----------------------------------------------------------------------
def _twiddles(L):
    return np.exp(-2j*np.pi*np.arange(L)/L)


def fft_tile(x, L, inv=False):
    """the kernel's in-place radix-2 DIT over the last axis (a power of two
    <= L), twiddles from the length-L table"""
    Ls = x.shape[-1]
    lg = Ls.bit_length() - 1
    rev = np.array([int(format(e, "0%db" % lg)[::-1], 2) if lg else 0 for e in range(Ls)])
    s = np.empty_like(x)
    s[..., rev] = x
    tw = _twiddles(L)
    if inv:
        tw = tw.conj()
    half = 1
    while half < Ls:
        s = s.reshape(x.shape[:-1] + (Ls//(2*half), 2, half))
        w = tw[np.arange(half)*(L//(2*half))]
        u, v = s[..., 0, :].copy(), s[..., 1, :]*w
        s[..., 0, :], s[..., 1, :] = u + v, u - v
        s = s.reshape(x.shape)
        half *= 2
    return s


def fft_pow2(x, inv=False):
    """length-L transform of the last axis as the device computes it: one tile
    when L <= FFT_TILE, otherwise four-step L = L1 x L2 (columns of L1 with
    stride L2, twiddle, rows of L2) with the result in the transposed order
    position L2 k1 + k2 <- X[k1 + L1 k2]; inv=True takes that order back"""
    L = x.shape[-1]
    if L <= FFT_TILE:
        return fft_tile(x, L, inv)
    L1, L2 = FFT_L1, L//FFT_L1
    tw = _twiddles(L)
    k1n2 = (np.arange(L1)[:, None]*np.arange(L2)) % L
    if not inv:
        a = x.reshape(x.shape[:-1] + (L1, L2))
        a = np.swapaxes(fft_tile(np.swapaxes(a, -1, -2), L), -1, -2)*tw[k1n2]
        return fft_tile(a, L).reshape(x.shape)
    a = fft_tile(x.reshape(x.shape[:-1] + (L1, L2)), L, inv=True)*tw[k1n2].conj()
    return np.swapaxes(fft_tile(np.swapaxes(a, -1, -2), L, inv=True), -1, -2).reshape(x.shape)


def bluestein(x, M):
    """length-M DFT of the rows of x (m_in <= M values each, zero-padded) by
    the chirp-z convolution of power-of-two length L >= M + m_in - 1"""
    x = np.atleast_2d(np.asarray(x, complex))
    m_in = x.shape[-1]
    L = 2
    while L < M + m_in - 1:
        L *= 2
    k = np.arange(M, dtype=np.int64)
    chirp = np.exp(-1j*np.pi*((k*k) % (2*M))/M)
    a = np.zeros(x.shape[:-1] + (L,), complex)
    a[..., :m_in] = x*chirp[:m_in]
    b = np.zeros(L, complex)
    b[:M] = chirp.conj()
    b[L - m_in + 1:] = chirp[1:m_in][::-1].conj()
    z = fft_pow2(fft_pow2(a)*fft_pow2(b), inv=True)
    return chirp*z[..., :M]/L


def psf(o, pad=4):
    """rtx_psf: |DFT2(pupil, pad n)|^2/(pad n)^2 by rows of the transposed
    pupil, transpose, rows"""
    n = o.shape[0]
    good = np.isfinite(o)
    g = np.where(good, np.exp(-2j*np.pi*np.where(good, o, 0)), 0)/np.sqrt(good.sum())
    M = pad*n
    rows = bluestein(g.T, M)          # n x M
    F = bluestein(rows.T, M)          # M x M
    return (F.real**2 + F.imag**2)/(M*M)
