"""Device-resident trace results with lazy host materialisation.

The full trace of 1e7 rays x 12 surfaces is 10 GB; PCIe moves it in 0.2 s while
the kernel needs 1.7 ms.  The consumers of ``GeometricTrace`` mostly read single
rows -- spot diagrams ``y[-1]``, ``i[-1]`` (rayopt/analysis.py:269-280), fans
``y[-1]``, ``y[0]``, ``u[0]`` (:231-245), ``rms`` ``y[i]``
(rayopt/geometric_trace.py:171-183), ``refocus`` ``y[at]``, ``i[at]`` (:82-99)
-- so the resident drop-in keeps ``y,u,i,t`` in HBM and hands out ``LazyRows``
objects that copy a surface row to the host the first time it is indexed (and
the whole array only for ``np.asarray``).

``ResidentMixin`` is the resident flavour of ``PropagateMixin``
(geometric_trace.py): ``bind(rayopt.GeometricTrace, resident=True)`` puts it in
front of the reference class; ``ResidentTrace`` is the standalone class with the
on-device ray generation on top.
"""
import numpy as np

from .engine import default_engine
from .surface_table import pack_system

# rows above this size live in page-locked host buffers (full-rate PCIe)
PINNED_ROW_BYTES = 1 << 20


class LazyRows:
    """numpy-like view of a device array (rows, ld, k...) restricted to the
    first `n` columns.  Indexing with a leading integer (or a slice of rows)
    downloads just those rows, once; like ``GeometricTrace.y[j]`` in the
    reference the result is a VIEW of the trace's storage: the host buffer of
    a row is reused, so a later ``propagate`` + access refreshes it in place.
    Item assignment writes through to the device."""

    def __init__(self, darray, n, dtype=np.float64):
        self._d = darray
        self._n = int(n)
        self.dtype = np.dtype(dtype)
        self.shape = (darray.shape[0], self._n) + tuple(darray.shape[2:])
        self.ndim = len(self.shape)
        self.size = int(np.prod(self.shape))
        self._rows = {}        # valid host copies
        self._bufs = {}        # host buffers (kept across invalidation)
        self.fetched_bytes = 0

    def __len__(self):
        return self.shape[0]

    def invalidate(self, rows=None):
        if rows is None:
            self._rows.clear()
        else:
            for r in rows:
                self._rows.pop(r, None)

    def _buffer(self, r):
        b = self._bufs.get(r)
        if b is None:
            shape = (self._n,) + self.shape[2:]
            nbytes = int(np.prod(shape))*self._d.dtype.itemsize
            eng = getattr(self._d, "engine", None)
            if nbytes >= PINNED_ROW_BYTES and hasattr(eng, "pinned_empty"):
                b = eng.pinned_empty(shape, self._d.dtype)
            else:
                b = np.empty(shape, self._d.dtype)
            self._bufs[r] = b
        return b

    def set_row(self, r, value):
        """host-side write of one row (e.g. launch rays), mirrored to the
        device; `value` broadcasts to (n, k) or to the padded (ld, k) row"""
        r = range(self.shape[0])[r]
        drow = self._d.rows(r)
        v = np.asarray(value)
        full = drow.shape[1:]
        if v.shape == full:                              # whole padded row
            v = np.ascontiguousarray(v, self._d.dtype)
            drow.upload(v)
            host = v[:self._n]
        else:
            host = np.ascontiguousarray(np.broadcast_to(v, (self._n,) + self.shape[2:]),
                                        self._d.dtype)
            drow.upload(host)                            # the first n columns are contiguous
        b = self._buffer(r)
        b[...] = host
        self._rows[r] = b if b.dtype == self.dtype else b.astype(self.dtype)

    def row(self, r):
        r = range(self.shape[0])[r]
        a = self._rows.get(r)
        if a is None:
            b = self._buffer(r)
            self._d.rows(r).download(out=b)              # first n columns of the row
            a = b if b.dtype == self.dtype else b.astype(self.dtype)
            self._rows[r] = a
            self.fetched_bytes += b.nbytes
        return a

    def __getitem__(self, idx):
        if not isinstance(idx, tuple):
            idx = (idx,)
        head, rest = idx[0], idx[1:]
        if isinstance(head, (int, np.integer)):
            a = self.row(int(head))
            return a[rest] if rest else a
        if isinstance(head, slice):
            rows = range(self.shape[0])[head]
            a = np.stack([self.row(r) for r in rows]) if len(rows) else \
                np.empty((0,) + self.shape[1:], self.dtype)
            return a[(slice(None),) + rest] if rest else a
        return np.asarray(self)[idx]

    def __setitem__(self, idx, value):
        if not isinstance(idx, tuple):
            idx = (idx,)
        head, rest = idx[0], idx[1:]
        rows = [range(self.shape[0])[int(head)]] if isinstance(head, (int, np.integer)) \
            else list(range(self.shape[0])[head])
        value = np.asarray(value)
        for k, r in enumerate(rows):
            v = value if isinstance(head, (int, np.integer)) or value.ndim < self.ndim else value[k]
            if rest:
                host = np.array(self.row(r))
                host[rest] = v
            else:
                host = v
            self.set_row(r, host)

    def __array__(self, dtype=None, copy=None):
        a = np.stack([self.row(r) for r in range(self.shape[0])])
        return a if dtype is None else a.astype(dtype)


class ResidentMixin:
    """``allocate / rays_given / propagate / rms / refocus`` of GeometricTrace
    (rayopt/geometric_trace.py:37-99,171-183) with the results resident in HBM.
    Same signatures and attribute names; ``y, u, i, t`` are ``LazyRows``.
    ``propagate`` moves no ray data over PCIe; ``rms`` and ``refocus`` reduce on
    the device (8 doubles come back)."""

    engine = None
    exact = False
    resident = True

    # the reference's default weights ones(N)/N (geometric_trace.py:57-58) are
    # materialised on first read: at 1e7 rays building them costs more than the
    # trace, and the device reductions never need them (w = None means 1/N)
    @property
    def w(self):
        if self._w is None and getattr(self, "_w_default", False):
            self._w = np.ones(self.nrays)/self.nrays
        return self._w

    @w.setter
    def w(self, value):
        self._w = value
        self._w_default = False
    _w = None
    # i[j] == u[j-1] bit for bit in unrotated systems (system.py:461-463): u and
    # i are then two row-shifted views of ONE (S+2, ld, 3) device buffer and the
    # kernel stores 56 instead of 80 bytes per ray-surface
    alias_incidence = True
    _dev = None

    def _engine(self):
        if self.engine is None:
            self.engine = default_engine()
        return self.engine

    # ---- a1
    def allocate(self, nrays):
        eng = self._engine()
        self.free()
        self.length = L = len(self.system)
        self.nrays = nrays
        self._ld = ld = (nrays + 63)//64*64
        d = {"y": eng.empty((L, ld, 3)), "t": eng.empty((L, ld))}
        if self.alias_incidence:
            d["uext"] = eng.empty((L + 1, ld, 3))
            d["u"], d["i"] = d["uext"].rows(1, L + 1), d["uext"].rows(0, L)
            self._i_alias = True
        else:
            d["u"], d["i"] = eng.empty((L, ld, 3)), eng.empty((L, ld, 3))
            self._i_alias = False
        self._dev = d
        self._wrap()
        self.n = np.empty(L)
        self.w = None
        self.ref = None
        self.l = 1.
        self._w_dev = None

    def _wrap(self):
        d, n = self._dev, self.nrays
        self.y, self.u = LazyRows(d["y"], n), LazyRows(d["u"], n)
        self.i, self.t = LazyRows(d["i"], n), LazyRows(d["t"], n)

    def _materialize_i(self):
        """a rotated element breaks i[j] == u[j-1]: give `i` its own array"""
        eng, d = self._engine(), self._dev
        own = eng.empty((self.length, self._ld, 3))
        own.copy_from(d["i"])
        eng.sync()
        d["i"] = own
        self._i_alias = False
        self.i = LazyRows(own, self.nrays)

    def free(self):
        """give the HBM back now (otherwise: when the object is collected)"""
        if self._dev:
            for a in self._dev.values():
                a.free()
        self._dev = None
        w = getattr(self, "_w_dev", None)
        if w is not None:
            w[1].free()
        self._w_dev = None

    # ---- a2
    def rays_given(self, y, u, l=None, w=None, ref=0):
        """rayopt/geometric_trace.py:49-70: launch rays into row 0 -- straight
        from the caller's arrays into HBM (one H2D per array when they are
        (N,3) float64; page-locked arrays copy at full PCIe rate)."""
        pos, dirn = np.broadcast_arrays(*np.atleast_2d(y, u))
        count, width = pos.shape
        if self._dev is None or self.nrays != count:
            self.allocate(count)
        self.l = self.system.wavelengths[0] if l is None else l
        self.w = w
        self._w_default = w is None
        self._w_dev = None
        self.ref = ref
        self._hex_rings = None
        if width != 3:
            y0 = np.zeros((count, 3))
            u0 = np.zeros((count, 3))
            y0[:, :width] = pos
            u0[:, :width] = dirn
            if width < 3:                                  # assumes forward rays, :65-67
                u0[:, 2] = np.sqrt(1 - np.square(u0[:, :2]).sum(-1))
            pos, dirn = y0, u0
        d = self._dev
        d["y"].rows(0).upload(pos)
        d["u"].rows(0).upload(dirn)
        d["i"].rows(0).copy_from(d["u"].rows(0), count*24)     # i[0] = u[0], :68
        self._zero_t0()                                        # t[0] = 0, :70
        for a in (self.y, self.u, self.i, self.t):
            a.invalidate()
        self.n[0] = self.system.refractive_index(self.l, 0)

    def _zero_t0(self):
        eng, row = self._engine(), self._dev["t"].rows(0)
        if hasattr(eng, "memset"):
            eng.memset(row, 0)
        else:
            row.upload(np.zeros(row.shape[1:]))

    def _cache_system(self):
        """Trace.propagate, rayopt/raytrace.py:32-36"""
        for name in ("path", "track", "origins", "mirrored"):
            try:
                setattr(self, name, getattr(self.system, name))
            except AttributeError:
                pass

    # ---- a3
    def propagate(self, start=1, stop=None, clip=False):
        """rayopt/geometric_trace.py:72-80 on the resident rows"""
        self._cache_system()
        init = start - 1
        table, n, rot0 = pack_system(self.system, self.l, start, stop, n0=self.n[init])
        rows = len(table)
        if rows == 0:
            return
        if self._i_alias and (rot0 is not None or (table["flags"] & 1).any()):
            self._materialize_i()
        d = self._dev
        sl = (start, start + rows)
        self._engine().trace_device(
            table, d["y"].rows(init), d["u"].rows(init),
            d["y"].rows(*sl), d["u"].rows(*sl),
            None if self._i_alias else d["i"].rows(*sl), d["t"].rows(*sl),
            N=self.nrays, ld=self._ld, clip=clip, rot0=rot0, exact=self.exact)
        self.n[start:start + rows] = n
        self._last_clip = bool(clip)
        touched = range(start, start + rows)
        for a in (self.y, self.u, self.t):
            a.invalidate(touched)
        # an aliased i[j] is u[j-1]: rows start+1 .. start+rows changed
        self.i.invalidate(range(start + 1, start + rows + 1) if self._i_alias else touched)

    # ---- reductions that never bring the rays to the host (SURVEY 8f-1)
    def _weights(self):
        """device copy of self.w, or None for the default 1/N weights"""
        if self._w is None or getattr(self, "_w_default", False):
            return None
        if self._w_dev is None or self._w_dev[0] is not self._w:
            if self._w_dev is not None:
                self._w_dev[1].free()
            self._w_dev = (self._w, self._engine().to_device(np.asarray(self._w, float)))
        return self._w_dev[1]

    def rms(self, i=-1, ref=None):
        """GeometricTrace.rms (rayopt/geometric_trace.py:171-183) on the
        resident intercepts (moment passes on the device, 64 bytes back)."""
        eng = self._engine()
        i = range(self.length)[i]
        ref_point = None if ref is None else \
            eng.download_rays(self._dev["y"].rows(i), [int(ref)])[0, :2]    # 24 bytes, not the row
        return eng.rms(self._dev["y"].rows(i), self._weights(), N=self.nrays,
                       ref_point=ref_point)

    def refocus(self, at=-1):
        """GeometricTrace.refocus (rayopt/geometric_trace.py:82-99): the
        least-squares focus shift from device moments of y[at], i[at]
        (rtx_focus_moments), then the re-trace."""
        eng = self._engine()
        at = range(self.length)[at]
        shift = eng.refocus_shift(self._dev["y"].rows(at), self._dev["i"].rows(at),
                                  self._weights(), N=self.nrays)
        self.system[at].distance += shift
        self.propagate()


    # ---- fused epilogues: the march itself reduces (no rows are stored or read)
    def _guess_center(self, table, rot0, clip):
        """(y_x, y_y, u_x, u_y) of the `ref` ray at the last surface of `table`
        (a 1-ray trace through the small-bundle path), zeros if it dies"""
        eng, d = self._engine(), self._dev
        ref = 0 if self.ref is None else int(self.ref)
        y0 = eng.download_rays(d["y"].rows(0), [ref])
        u0 = eng.download_rays(d["u"].rows(0), [ref])
        Y, _, I, _ = eng.trace(table, y0, u0, clip=clip, rot0=rot0, keep_last=True,
                               exact=self.exact, want=("y", "i"))
        c = np.r_[Y[0, 0, :2], I[0, 0, :2]/I[0, 0, 2]]
        return c if np.all(np.isfinite(c)) else np.zeros(4)

    def reduce(self, at=-1, clip=False):
        """ONE launch from the launch rays (row 0) to surface `at`: the trace
        kernel accumulates the rms / refocus moments of that surface in
        registers (rtx_trace_reduce) and stores nothing else.  Returns the 20
        moments (include/rtx.h) and the guess centre they refer to."""
        at = range(self.length)[at]
        table, _, rot0 = pack_system(self.system, self.l, 1, at + 1, n0=self.n[0])
        c = self._guess_center(table, rot0, clip)
        d = self._dev
        m = self._engine().trace_reduce(table, d["y"].rows(0), d["u"].rows(0), N=self.nrays,
                                        clip=clip, rot0=rot0, exact=self.exact,
                                        w=self._weights(), center=c)
        return m, c

    def rms_fused(self, at=-1, clip=False):
        """GeometricTrace.rms of surface `at` without a stored trace"""
        m, _ = self.reduce(at, clip)
        return self._engine().rms_from_moments(m, unit_weights=self._weights() is None)

    def refocus_fused(self, at=-1, clip=False):
        """GeometricTrace.refocus (geometric_trace.py:82-99) from one fused
        launch: the focus shift is applied to ``system[at].distance`` and
        returned; nothing is re-traced"""
        m, _ = self.reduce(at, clip)
        shift = self._engine().focus_shift_from_moments(m)
        self.system[at].distance += shift
        return shift

    def _opd_device(self, radius=None, after=-2, image=-1):
        """rtx_trace_opd into fresh DEVICE arrays A (N,), P (N,3); returns them
        with the reference ray's A[ref], P[ref] and l/scale"""
        eng, s, d = self._engine(), self.system, self._dev
        after, image = range(self.length)[after], range(self.length)[image]
        ref = int(self.ref)
        if radius is None:                                  # :110-114
            if s.image.pupil.telecentric:
                radius = self.track[image] - self.track[after]
            else:
                radius = -s.image.pupil.distance
        ea, ei = s[after], s[image]
        eye = np.eye(3)
        Ra = np.asarray(ea.rot_normal, float) if getattr(ea, "rotated", False) else eye
        Ri = np.asarray(ei.rot_normal, float) if getattr(ei, "rotated", False) else eye
        y_img_ref = eng.download_rays(d["y"].rows(image), [ref])[0]
        spec = dict(y0_ref=eng.download_rays(d["y"].rows(0), [ref])[0],
                    u0_ref=eng.download_rays(d["u"].rows(0), [ref])[0],
                    n0=self.n[0], n_after=self.n[after], M=Ra @ Ri.T,
                    d=(self.origins[after] - self.origins[image]) @ Ri.T - y_img_ref,
                    radius=radius, infinite=not s.object.finite)
        table, _, rot0 = pack_system(s, self.l, 1, after + 1, n0=self.n[0])
        A, P = eng.empty((self.nrays,)), eng.empty((self.nrays, 3))
        eng.trace_opd(table, d["y"].rows(0), d["u"].rows(0), spec, A, P, N=self.nrays,
                      clip=getattr(self, "_last_clip", False), rot0=rot0, exact=self.exact)
        a_ref = A.rows(ref).download()[0]
        p_ref = eng.download_rays(P, [ref])[0]
        return A, P, a_ref, p_ref, self.l/s.scale

    def opd_rays(self, radius=None, after=-2, image=-1):
        """per-ray part of GeometricTrace.opd (rayopt/geometric_trace.py:
        101-131) as the epilogue of a march from row 0 to surface `after`
        (rtx_trace_opd); the reference ray's terms are subtracted here.
        Returns (x, y, t): exit-pupil coordinates and the OPD in waves -- what
        ``opd(resample=False)`` returns in the reference.  Needs a propagated
        trace (the sphere is centred on ``y[image, ref]``)."""
        A, P, a_ref, p_ref, lscale = self._opd_device(radius, after, image)
        a, p = A.download(), P.download()
        A.free()
        P.free()
        t = -(a - a_ref)/lscale                             # :125-126
        p -= p_ref                                          # :131
        return p[:, 0], p[:, 1], t

    def opd(self, radius=None, after=-2, image=-1, resample=4):
        """GeometricTrace.opd with the per-ray part on the device; the
        regridding (scipy griddata, geometric_trace.py:133-144) stays on the host"""
        x, y, t = self.opd_rays(radius, after, image)
        if resample:
            from scipy.interpolate import griddata
            ok = np.isfinite(x) & np.isfinite(y) & np.isfinite(t)
            x, y, t = x[ok], y[ok], t[ok]
            if not t.size:
                raise ValueError("no rays made it through")
            n = int(resample*self.nrays**.5)
            h = np.fabs((x, y)).max()
            xs, ys = np.mgrid[-1:1:1j*n, -1:1:1j*n]*h
            t = griddata((x, y), t, (xs, ys), method="linear", fill_value=np.nan)
            x, y = xs, ys
        return x, y, t

    # ---- the OPD map and the PSF in HBM (rtx_opd_regrid, rtx_psf)
    # rings of the hexapolar launch grid when the launch rays are known to be
    # pupil_distribution("hexapolar") without a pupil filter, else None: the
    # ray index then gives the triangulation (rtx_opd_regrid)
    _hex_rings = None

    def rays_point(self, yo, wavelength=None, nrays=11, distribution="meridional", filter=None,
                   stop=None, clip=False):
        """GeometricTrace.rays_point (rayopt/geometric_trace.py:204-209) of the
        reference, recording whether the bundle is an unfiltered hexapolar
        grid (its `filter` defaults to ``not clip``)"""
        super().rays_point(yo, wavelength, nrays, distribution, filter, stop, clip)
        self._record_grid(distribution, nrays, (not clip) if filter is None else filter)

    def _record_grid(self, distribution, nrays, filter):
        rings = int(np.sqrt(nrays/3. - 1/12.) - 1/2.) if distribution == "hexapolar" else 0
        ok = int(nrays) > 1 and not filter and rings >= 1 and self.nrays == 1 + 3*rings*(rings + 1)
        self._hex_rings = rings if ok else None

    def _opd_grid(self, radius, after, image, resample, regrid):
        """(map, h, x): the (n, n) OPD map in HBM, h (None for the host path)
        and the x column of the node grid; regridded on the device, or by
        scipy griddata on the host (opd()) and uploaded"""
        if regrid is None:
            regrid = "host" if self._hex_rings is None else "device"
        if regrid == "host":
            xs, _, t = self.opd(radius, after, image, resample)
            return self._engine().to_device(t), None, xs[:, 0]
        if regrid != "device":
            raise ValueError("regrid must be 'device', 'host' or None, got %r" % (regrid,))
        if self._hex_rings is None:
            raise ValueError("device regridding needs a hexapolar bundle generated without "
                             "a pupil filter (rays_point(distribution='hexapolar', clip=True))")
        A, P, a_ref, p_ref, lscale = self._opd_device(radius, after, image)
        n = int(resample*self.nrays**.5)
        try:
            m, h, count = self._engine().opd_regrid(A, P, a_ref, p_ref, lscale, self._hex_rings, n)
        finally:
            A.free()
            P.free()
        if not count:
            m.free()
            raise ValueError("no rays made it through")
        return m, h, np.mgrid[-1:1:1j*n, -1:1:2j][0][:, 0]*h

    def opd_map(self, radius=None, after=-2, image=-1, resample=4, regrid=None):
        """GeometricTrace.opd(resample) (rayopt/geometric_trace.py:101-144):
        returns the reference's (x, y, t) node grids.  regrid="device"
        interpolates on the structured triangulation of a hexapolar launch
        grid in HBM (rtx_opd_regrid; vignetted gaps stay NaN, INTEGRATION.md
        section 5), "host" is opd(); None picks "device" when the bundle is
        known to be an unfiltered hexapolar grid."""
        if not resample or regrid == "host" or (regrid is None and self._hex_rings is None):
            return self.opd(radius, after, image, resample)
        m, h, _ = self._opd_grid(radius, after, image, resample, regrid)
        t = m.download()
        m.free()
        n = t.shape[0]
        xs, ys = np.mgrid[-1:1:1j*n, -1:1:1j*n]*h
        return xs, ys, t

    def psf_device(self, pad=4, resample=4, regrid=None, **kw):
        """GeometricTrace.psf (rayopt/geometric_trace.py:146-169) with the
        pupil function, the zero-padded 2-D DFT and |.|^2 in HBM (rtx_psf);
        the OPD map comes from opd_map's `regrid`.  Returns (p, q, psf)."""
        radius = self.system[-1].distance                   # :147
        m, _, x = self._opd_grid(radius, kw.pop("after", -2), kw.pop("image", -1), resample,
                                 regrid)
        if kw:
            raise TypeError("unexpected arguments %s" % sorted(kw))
        eng = self._engine()
        n = m.shape[0]
        try:
            d_psf = eng.psf(m, pad)
        finally:
            m.free()
        psf = eng.pinned_empty(d_psf.shape) if d_psf.nbytes >= PINNED_ROW_BYTES else None
        psf = d_psf.download(psf)
        d_psf.free()
        dx = x[1] - x[0]                                    # :158-161
        k = 1/(self.l/self.system.scale)
        f = np.fft.fftfreq(pad*n, dx*k/radius)
        p, q = np.broadcast_arrays(f[:, None], f)
        return p, q, psf

    def psf_metrics(self, pad=4, resample=4, regrid=None, window=0, **kw):
        """The figures Analysis.opds (rayopt/analysis.py:319-346) takes from
        psf() -- centroid, peak, encircled energy, MTF along both axes and
        optionally a (2 window + 1)^2 window around the centroid -- computed
        on the PSF in HBM (Engine.psf_metrics); the PSF itself never leaves
        the device.  The OPD map comes from opd_map's `regrid`, as in
        psf_device.  Returns an engine.PsfMetrics."""
        radius = self.system[-1].distance                   # geometric_trace.py:147
        m, _, x = self._opd_grid(radius, kw.pop("after", -2), kw.pop("image", -1), resample,
                                 regrid)
        if kw:
            m.free()
            raise TypeError("unexpected arguments %s" % sorted(kw))
        eng = self._engine()
        try:
            d_psf = eng.psf(m, pad)
        finally:
            m.free()
        try:
            k = 1/(self.l/self.system.scale)                # :158-161
            return eng.psf_metrics(d_psf, (x[1] - x[0])*k/radius, window)
        finally:
            d_psf.free()


class ResidentTrace(ResidentMixin):
    """Standalone resident drop-in (no rayopt import needed) with launch rays
    generated in HBM (SURVEY 8f-2)."""

    def __init__(self, system, engine=None, exact=False, alias_incidence=True):
        self.system = system
        self.engine = engine or default_engine()
        self.exact = exact
        self.alias_incidence = alias_incidence
        self._dev = None

    def rays_infinite(self, yo, z, p, angle, l=None, nrays=None, yp=None, ref=0):
        """Launch rays of an aimed bundle for an infinite conjugate generated
        directly in HBM (Engine.aim_infinite_device / rtx_aim_infinite): the
        hexapolar grid with about `nrays` rays, or the DEVICE pupil coordinates
        `yp` (N,2); (z, p) is the reference's pupil-aiming solution
        (System.pupil).  Nothing crosses PCIe."""
        from .rays import aim_frame
        eng = self.engine
        if yp is None:
            rings = int(np.sqrt(nrays/3. - 1/12.) - 1/2.)
            count = 1 + 3*rings*(rings + 1)
        else:
            rings, count = 0, yp.shape[0]
        if self._dev is None or self.nrays != count:
            self.allocate(count)
        self.l = self.system.wavelengths[0] if l is None else l
        self.w = None
        self._w_default, self._w_dev = True, None
        self.ref = ref
        frame = np.concatenate(aim_frame(yo, z, angle))
        pmax = float(np.fabs(np.asarray(p, float)).max())
        d = self._dev
        eng.aim_infinite_into(d["y"].rows(0), d["u"].rows(0), count, rings, frame, pmax, yp)
        self._hex_rings = rings if yp is None and rings >= 1 else None
        d["i"].rows(0).copy_from(d["u"].rows(0), count*24)   # i[0] = u[0] (geometric_trace.py:68)
        self._zero_t0()
        for a in (self.y, self.u, self.i, self.t):
            a.invalidate()
        self.n[0] = self.system.refractive_index(self.l, 0)

    def rays_device(self, yo, wavelength=None, nrays=11, distribution="hexapolar", filter=False,
                    stop=None, seed=0):
        """Launch rays of ``rays_point`` generated in HBM by the general
        generator (rtx_aim_plan / rtx_aim_rays): the pupil grid (hexapolar,
        square, triangular, random, meridional / sagittal / cross / tee lines),
        Pupil.map with its `filter`, Conjugate.aim for finite and infinite
        objects in every projection, telecentric pupils, curved object
        surfaces.  ``system.pupil`` (the aiming) stays host Python.  Returns
        False (nothing done) for the distributions that stay on the host."""
        from .rays import aim_record, grid_spec
        s, eng = self.system, self.engine
        ref, grid = grid_spec(distribution, nrays)
        if grid is None:
            return False
        l = s.wavelengths[0] if wavelength is None else wavelength
        z, p = s.pupil(yo, l=wavelength, stop=stop)
        spec = aim_record(s.object, yo, z, p, grid, filter, s[0], seed)
        count = eng.aim_count(spec)
        if self._dev is None or self.nrays != count:
            self.allocate(count)
        self.l = l
        self.w = None
        self._w_default, self._w_dev = True, None
        self.ref = ref
        d = self._dev
        eng.aim_rays_into(spec, d["y"].rows(0), d["u"].rows(0), count)
        self._record_grid(distribution, nrays, filter)
        d["i"].rows(0).copy_from(d["u"].rows(0), count*24)   # i[0] = u[0] (geometric_trace.py:68)
        self._zero_t0()
        for a in (self.y, self.u, self.i, self.t):
            a.invalidate()
        self.n[0] = s.refractive_index(self.l, 0)
        return True

    def rays_point(self, yo, wavelength=None, nrays=11, distribution="hexapolar",
                   filter=None, stop=None, clip=False):
        """GeometricTrace.rays_point (rayopt/geometric_trace.py:204-209) for a
        rayopt ``System``: the pupil is aimed by the reference on the host
        (``system.pupil``), the launch rays are generated in HBM
        (``rays_device``) -- or by ``system.aim`` on the host and uploaded for
        the quadrature distributions -- and traced with `clip`."""
        s = self.system
        filt = (not clip) if filter is None else filter
        if not self.rays_device(yo, wavelength, nrays, distribution, filt, stop):
            from rayopt.utils import pupil_distribution      # the reference's own helper
            l = s.wavelengths[0] if wavelength is None else wavelength
            z, p = s.pupil(yo, l=wavelength, stop=stop)
            ref, yp, weight = pupil_distribution(distribution, nrays)
            y, u = s.aim(yo, yp, z, p, filter=filt)
            self.rays_given(y, u, l, weight, ref)
        self.propagate(clip=clip)
