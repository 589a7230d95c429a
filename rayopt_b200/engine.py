"""Host-side handle of one GPU context of the ray-trace engine.

Thin, torch-free layer over the C ABI (include/rtx.h): device / pinned memory,
the trace call with host or device buffers, CUDA-event timing.  One `Engine`
per GPU (one process per GPU in multi-GPU runs).
"""
import ctypes as C
import math
import weakref
from collections import namedtuple

import numpy as np

from . import _lib
from ._lib import (RTX_F32, RTX_F64, RTX_KEEP_ALL, RTX_KEEP_LAST, RTX_EXACT,
                   RTX_STORE_DIRECT, RTX_RPT1, RTX_RPT2, RtxError, check, ptr)
from .surface_table import SURFACE_DTYPE

_DTYPES = {np.dtype(np.float64): RTX_F64, np.dtype(np.float32): RTX_F32}

# mirrors `struct rtx_opd` (include/rtx.h)
OPD_DTYPE = np.dtype([("y0_ref", "<f8", (3,)), ("u0_ref", "<f8", (3,)), ("n0", "<f8"),
                      ("n_after", "<f8"), ("M", "<f8", (9,)), ("d", "<f8", (3,)),
                      ("radius", "<f8"), ("infinite", "<i4"), ("reserved", "<i4")], align=True)

# the figures of a PSF (Engine.psf_metrics)
PsfMetrics = namedtuple("PsfMetrics", "x0 y0 dx peak ee r freq mtf window")


def _code(dtype):
    try:
        return _DTYPES[np.dtype(dtype)]
    except KeyError:
        raise TypeError("dtype must be float64 or float32, got %r" % (dtype,))


class DeviceArray:
    """A typed block of HBM owned by an Engine (freed with it or on .free())."""

    def __init__(self, engine, shape, dtype):
        self.engine = engine
        self.shape = tuple(int(s) for s in shape)
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape, dtype=np.int64))*self.dtype.itemsize
        p = C.c_void_p()
        check(engine.lib.rtx_malloc(engine.ctx, self.nbytes, C.byref(p)))
        self.ptr = p.value
        engine._live[id(self)] = self.ptr

    def free(self):
        eng = self.engine
        if self.ptr is not None and eng.ctx is not None and id(self) in eng._live:
            eng._live.pop(id(self), None)
            check(eng.lib.rtx_free_device(eng.ctx, self.ptr))
        self.ptr = None

    def __del__(self):              # dropped without free(): give the HBM back
        try:
            if self.ptr is not None and id(self) in self.engine._live:
                self.free()
        except Exception:
            pass

    def upload(self, a):
        a = np.ascontiguousarray(a, self.dtype)
        assert a.nbytes <= self.nbytes
        check(self.engine.lib.rtx_memcpy_h2d(self.engine.ctx, self.ptr, ptr(a), a.nbytes))
        self.engine.sync()          # `a` may be a temporary
        return self

    def download(self, out=None):
        if out is None:
            out = np.empty(self.shape, self.dtype)
        check(self.engine.lib.rtx_memcpy_d2h(self.engine.ctx, ptr(out), self.ptr, out.nbytes))
        self.engine.sync()
        return out

    def copy_from(self, other, nbytes=None):
        """device-to-device copy (asynchronous on the engine stream)"""
        n = min(self.nbytes, other.nbytes) if nbytes is None else int(nbytes)
        check(self.engine.lib.rtx_memcpy_d2d(self.engine.ctx, self.ptr, other.ptr, n))
        return self

    def rows(self, r0, r1=None):
        """byte-offset view of leading-axis rows (no copy)"""
        v = object.__new__(DeviceArray)
        r1 = r0 + 1 if r1 is None else r1
        row_bytes = self.nbytes//self.shape[0]
        v.engine, v.dtype = self.engine, self.dtype
        v.shape = (r1 - r0,) + self.shape[1:]
        v.nbytes = row_bytes*(r1 - r0)
        v.ptr = self.ptr + r0*row_bytes
        v.free = lambda: None
        v._parent = self            # keeps the allocation alive
        return v


class _PinnedBlock:
    """owner of one page-locked allocation: the numpy arrays handed out by
    Engine.pinned_empty are views of its buffer, so the memory is released
    (cudaFreeHost) only when the LAST view has died -- never under a live
    array, whatever happens to the trace object or the engine"""

    def __init__(self, lib, address, nbytes):
        self.address = address
        self.buf = (C.c_char*nbytes).from_address(address)
        weakref.finalize(self.buf, lib.rtx_host_free, None, address)


class Engine:
    def __init__(self, device=0, numa=None):
        """`numa`: pin this process to the CPUs / memory of the GPU's NUMA
        node (rtx_numa_bind) so that page-locked buffers are local to the
        GPU's PCIe root; default: only in one-process-per-GPU launches
        (LOCAL_RANK set)."""
        self.lib = _lib.load()
        self.ctx = None
        if self.lib.rtx_device_count() < 1:
            raise RtxError("no CUDA device visible: the rayopt_b200 engine has "
                           "no CPU fallback")
        ctx = C.c_void_p()
        check(self.lib.rtx_init(int(device), C.byref(ctx)))
        self.ctx = ctx
        self.device = int(device)
        self._live = {}
        self.numa_node = None
        import os
        if numa is None:
            numa = "LOCAL_RANK" in os.environ
        if numa:
            self.numa_bind(True)
        sm, fr, tot = C.c_int(), C.c_size_t(), C.c_size_t()
        name = C.create_string_buffer(128)
        check(self.lib.rtx_device_info(self.ctx, C.byref(sm), C.byref(fr), C.byref(tot), name, 128))
        self.sm_count, self.total_bytes = sm.value, tot.value
        self.name = name.value.decode()
        self._fin = weakref.finalize(self, Engine._finalize, self.lib, self.ctx, self._live)

    @staticmethod
    def _finalize(lib, ctx, live):
        # (also runs at interpreter exit) `live` is emptied first so that a
        # DeviceArray collected later sees "not mine any more" and never hands
        # the dangling context back to the library
        try:
            live.clear()
            lib.rtx_free(ctx)
        except Exception:
            pass

    def close(self):
        """Release the context and every DeviceArray still alive.  Page-locked
        arrays from pinned_empty stay valid: they are freed when their last
        numpy view dies."""
        if self.ctx is not None:
            for p in list(self._live.values()):     # device arrays still alive
                self.lib.rtx_free_device(self.ctx, p)
            self._live.clear()
            self._fin.detach()
            self.lib.rtx_free(self.ctx)
            self.ctx = None

    def numa_bind(self, enable=True):
        """rtx_numa_bind: returns the NUMA node (or -1 if not reported)"""
        node = C.c_int(-1)
        check(self.lib.rtx_numa_bind(self.ctx, int(bool(enable)), C.byref(node)))
        self.numa_node = node.value if enable else None
        return node.value

    # ---- memory -------------------------------------------------------
    def empty(self, shape, dtype=np.float64):
        return DeviceArray(self, shape, dtype)

    def to_device(self, a, dtype=None):
        a = np.ascontiguousarray(a, dtype)
        return DeviceArray(self, a.shape, a.dtype).upload(a)

    def pinned_empty(self, shape, dtype=np.float64):
        """numpy array backed by page-locked host memory (full-rate PCIe)"""
        dtype = np.dtype(dtype)
        n = int(np.prod(shape, dtype=np.int64))*dtype.itemsize
        p = C.c_void_p()
        check(self.lib.rtx_host_alloc(self.ctx, max(n, 16), C.byref(p)))
        block = _PinnedBlock(self.lib, p.value, max(n, 16))
        # the array's base chain holds block.buf: freed with the last view
        return np.frombuffer(block.buf, dtype=dtype, count=n//dtype.itemsize).reshape(shape)

    def memset(self, darray, value=0):
        check(self.lib.rtx_memset(self.ctx, darray.ptr, int(value), darray.nbytes))

    def free_bytes(self):
        fr = C.c_size_t()
        check(self.lib.rtx_device_info(self.ctx, None, C.byref(fr), None, None, 0))
        return fr.value

    def sync(self):
        check(self.lib.rtx_sync(self.ctx))

    # ---- timing -------------------------------------------------------
    def timer_start(self):
        check(self.lib.rtx_timer_start(self.ctx))

    def timer_stop(self):
        ms = C.c_float()
        check(self.lib.rtx_timer_stop(self.ctx, C.byref(ms)))
        return ms.value

    def last_kernel_ms(self):
        ms = C.c_float()
        check(self.lib.rtx_last_kernel_ms(self.ctx, C.byref(ms)))
        return ms.value

    def launch_count(self):
        return int(self.lib.rtx_launch_count(self.ctx))

    # ---- the hot path -------------------------------------------------
    @staticmethod
    def _table(table):
        table = np.ascontiguousarray(table, SURFACE_DTYPE)
        if table.ndim != 1 or len(table) < 1:
            raise ValueError("surface table must be a non-empty 1-d record array")
        return table

    @staticmethod
    def _flags(exact, direct, rpt=0):
        return ((RTX_EXACT if exact else 0) | (RTX_STORE_DIRECT if direct else 0)
                | {0: 0, 1: RTX_RPT1, 2: RTX_RPT2}[rpt])

    def trace_device(self, table, y0, u0, Y, U, I, T, N=None, ld=None, clip=False,
                     keep_last=False, rot0=None, exact=False, direct=False, rpt=0, mask=None,
                     path_sum=None, path_sum_upto=-1):
        """One launch on DEVICE arrays (DeviceArray or None for outputs).
        Asynchronous on the engine stream.  `mask`: optional uint32
        DeviceArray of ceil(N/32) words receiving the warp-ballot vignetting
        mask (bit set = the ray survives the last surface).  `path_sum`:
        optional (N,) DeviceArray receiving sum_{s <= path_sum_upto} t[s]."""
        table = self._table(table)
        dt = _code(y0.dtype)
        N = y0.shape[0] if N is None else int(N)
        first = next((a for a in (Y, U, I, T) if a is not None), None)
        if ld is None:
            ld = first.shape[1] if first is not None else (N + 63)//64*64
        r0 = None if rot0 is None else np.ascontiguousarray(rot0, np.float64).reshape(9)
        dp = lambda a: None if a is None else a.ptr  # noqa: E731
        if mask is None and path_sum is None and all(a is None for a in (Y, U, I, T)):
            raise ValueError("nothing to store: pass an output array, a mask or a path sum")
        check(self.lib.rtx_set_mask_output(self.ctx, dp(mask)))
        check(self.lib.rtx_set_path_sum_output(self.ctx, dp(path_sum), int(path_sum_upto)))
        check(self.lib.rtx_trace(
            self.ctx, ptr(table), len(table), ptr(r0), dt, N, y0.ptr, u0.ptr,
            int(bool(clip)), RTX_KEEP_LAST if keep_last else RTX_KEEP_ALL, ld,
            dp(Y), dp(U), dp(I), dp(T), self._flags(exact, direct, rpt)))

    def trace_device_batch(self, tables, y0s, u0s, Ys, Us, Is, Ts, Ns=None, ld=None, clip=False,
                           keep_last=False, rot0=None, exact=False):
        """rtx_trace_batch: several bundles of the same lens (one table each,
        e.g. one per wavelength) in ONE launch.  Lists of DeviceArrays (any of
        Ys/Us/Is/Ts may be None as a whole)."""
        nb = len(tables)
        tabs = [self._table(t) for t in tables]
        S = len(tabs[0])
        if any(len(t) != S for t in tabs):
            raise ValueError("all bundles of a batch must have the same number of surfaces")
        dt = _code(y0s[0].dtype)
        Ns = [a.shape[0] for a in y0s] if Ns is None else [int(n) for n in Ns]
        first = next(a for a in (Ys, Us, Is, Ts) if a is not None)[0]
        ld = first.shape[1] if ld is None else int(ld)
        vp = C.c_void_p

        def arr(items, get):
            if items is None:
                return None
            return (vp*nb)(*[vp(get(x)) for x in items])
        a_tab = arr(tabs, lambda t: t.ctypes.data)
        a_n = (C.c_int64*nb)(*Ns)
        r0 = None if rot0 is None else np.ascontiguousarray(rot0, np.float64).reshape(9)
        check(self.lib.rtx_trace_batch(
            self.ctx, nb, C.cast(a_tab, vp), S, ptr(r0), dt, C.cast(a_n, vp),
            C.cast(arr(y0s, lambda a: a.ptr), vp), C.cast(arr(u0s, lambda a: a.ptr), vp),
            int(bool(clip)), RTX_KEEP_LAST if keep_last else RTX_KEEP_ALL, ld,
            *[None if x is None else C.cast(arr(x, lambda a: a.ptr), vp) for x in (Ys, Us, Is, Ts)],
            self._flags(exact, False)))

    def trace(self, table, y0, u0, clip=False, keep_last=False, rot0=None,
              dtype=np.float64, exact=False, direct=False, rpt=0, out=None,
              want=("y", "u", "i", "t")):
        """Host arrays in, host arrays out (reference layout): returns
        Y,U,I (rows,N,3), T (rows,N); rows = S or 1.  H2D, kernel and D2H are
        pipelined over ray chunks inside the library."""
        table = self._table(table)
        dtype = np.dtype(dtype)
        dt = _code(dtype)
        y0 = np.ascontiguousarray(y0, dtype)
        u0 = np.ascontiguousarray(u0, dtype)
        if y0.ndim != 2 or y0.shape[1] != 3 or u0.shape != y0.shape:
            raise ValueError("y0, u0 must both be (N, 3)")
        N = y0.shape[0]
        rows = 1 if keep_last else len(table)
        if out is None:
            out = {}
        res = []
        for k, shape in (("y", (rows, N, 3)), ("u", (rows, N, 3)),
                         ("i", (rows, N, 3)), ("t", (rows, N))):
            if k not in want:
                res.append(None)
                continue
            a = out.get(k)
            if a is None:
                a = np.empty(shape, dtype)
            if a.shape != shape or a.dtype != dtype or not a.flags.c_contiguous:
                raise ValueError("output %r must be C-contiguous %s %r" % (k, dtype, shape))
            res.append(a)
        r0 = None if rot0 is None else np.ascontiguousarray(rot0, np.float64).reshape(9)
        check(self.lib.rtx_trace_host(
            self.ctx, ptr(table), len(table), ptr(r0), dt, N, ptr(y0), ptr(u0),
            int(bool(clip)), RTX_KEEP_LAST if keep_last else RTX_KEEP_ALL,
            ptr(res[0]), ptr(res[1]), ptr(res[2]), ptr(res[3]),
            self._flags(exact, direct, rpt)))
        return tuple(res)

    def trace_bundles(self, tables, y0s, u0s, clip=False, keep_last=False, rot0=None,
                      dtype=np.float64, exact=False, want=("y", "u", "i", "t")):
        """rtx_trace_batch_host: many (small) bundles of ONE lens, host arrays
        in and out, one H2D + launches of 8 bundles + one D2H.  `tables[b]`
        the table of bundle b (same number of surfaces), `y0s[b]`, `u0s[b]`
        its (N_b,3) launch rays.  Returns a list of (Y, U, I, T) per bundle
        (None for arrays not in `want`)."""
        nb = len(tables)
        tabs = [self._table(t) for t in tables]
        S = len(tabs[0])
        if any(len(t) != S for t in tabs):
            raise ValueError("all bundles of a batch must have the same number of surfaces")
        dtype = np.dtype(dtype)
        y0s = [np.ascontiguousarray(np.atleast_2d(a), dtype) for a in y0s]
        u0s = [np.ascontiguousarray(np.atleast_2d(a), dtype) for a in u0s]
        Ns = [a.shape[0] for a in y0s]
        rows = 1 if keep_last else S
        outs = {k: ([np.empty((rows, n, 3) if k != "t" else (rows, n), dtype) for n in Ns]
                    if k in want else None) for k in "yuit"}
        vp = C.c_void_p

        def arr(items):
            if items is None:
                return None
            return C.cast((vp*nb)(*[vp(a.ctypes.data) for a in items]), vp)
        keep = [arr(tabs), arr(y0s), arr(u0s)] + [arr(outs[k]) for k in "yuit"]
        r0 = None if rot0 is None else np.ascontiguousarray(rot0, np.float64).reshape(9)
        check(self.lib.rtx_trace_batch_host(
            self.ctx, nb, keep[0], S, ptr(r0), _code(dtype), C.cast((C.c_int64*nb)(*Ns), vp),
            keep[1], keep[2], int(bool(clip)), RTX_KEEP_LAST if keep_last else RTX_KEEP_ALL,
            keep[3], keep[4], keep[5], keep[6], self._flags(exact, False)))
        return [tuple(None if outs[k] is None else outs[k][b] for k in "yuit") for b in range(nb)]

    def trace_gather(self, table, y0, u0, dst_ptrs, dst_offset, N=None, clip=False,
                     rot0=None, exact=False, dst_i_ptrs=None, xy=False):
        """rtx_trace_gather: trace the local shard (DEVICE y0,u0) and store
        the last surface's intercepts into every buffer of `dst_ptrs` (raw
        device pointers: local or peer memory) at ray offset `dst_offset`;
        `dst_i_ptrs`: a second set of buffers for the incidence directions;
        `xy`: the intercept buffers are (Ntotal, 2) and receive x,y only."""
        table = self._table(table)
        N = y0.shape[0] if N is None else int(N)
        r0 = None if rot0 is None else np.ascontiguousarray(rot0, np.float64).reshape(9)
        arr = (C.c_void_p*len(dst_ptrs))(*[C.c_void_p(int(p)) for p in dst_ptrs])
        arr_i = None
        if dst_i_ptrs is not None:
            if len(dst_i_ptrs) != len(dst_ptrs):
                raise ValueError("dst_i_ptrs must match dst_ptrs")
            arr_i = C.cast((C.c_void_p*len(dst_ptrs))(*[C.c_void_p(int(p)) for p in dst_i_ptrs]),
                           C.c_void_p)
        check(self.lib.rtx_trace_gather(
            self.ctx, ptr(table), len(table), ptr(r0), _code(y0.dtype), N, y0.ptr, u0.ptr,
            int(bool(clip)), len(dst_ptrs), C.cast(arr, C.c_void_p), arr_i, int(dst_offset),
            self._flags(exact, False) | (_lib.RTX_GATHER_XY if xy else 0)))

    # ---- fused epilogues (no per-surface stores) -------------------------
    def trace_reduce(self, table, y0, u0, N=None, clip=False, rot0=None, exact=False, w=None,
                     center=None):
        """rtx_trace_reduce: march the DEVICE launch rays to the last surface
        of `table` and return the 20 rms / refocus moments of that surface
        (include/rtx.h) -- one launch, no intercept is stored.  `center`:
        (y_x, y_y, u_x, u_y) guess centres (e.g. the chief ray's)."""
        table = self._table(table)
        N = y0.shape[0] if N is None else int(N)
        r0 = None if rot0 is None else np.ascontiguousarray(rot0, np.float64).reshape(9)
        c = None if center is None else np.ascontiguousarray(center, np.float64).reshape(4)
        m = np.zeros(20)
        check(self.lib.rtx_trace_reduce(
            self.ctx, ptr(table), len(table), ptr(r0), _code(y0.dtype), N, y0.ptr, u0.ptr,
            int(bool(clip)), None if w is None else w.ptr, ptr(c), ptr(m),
            self._flags(exact, False)))
        return m

    @staticmethod
    def rms_from_moments(m, unit_weights=False, about_center=False):
        """GeometricTrace.rms (rayopt/geometric_trace.py:171-183) from the
        moments of ONE pass about a guess centre c: the spot is re-centred on
        the unweighted mean analytically, sum w |y - ybar|^2 = m3 - 2 ybar.(m1,
        m2) + |ybar|^2 m0 with ybar = (m6, m7)/N relative to c (cancellation
        free when c is within the spot).  Not NaN-masked, like the reference.
        `about_center`: rms about c itself (the reference's `ref` ray).
        `unit_weights`: the moments were taken with w = 1 -> default 1/N."""
        if m[4] != m[5] or m[5] == 0:
            return float("nan")
        if about_center:
            r2 = m[3]
        else:
            bx, by = m[6]/m[5], m[7]/m[5]
            r2 = m[3] - 2*(bx*m[1] + by*m[2]) + (bx*bx + by*by)*m[0]
        if unit_weights:
            r2 /= m[5]
        return float(np.sqrt(max(r2, 0.)))

    @staticmethod
    def focus_shift_from_moments(m):
        """the shift of GeometricTrace.refocus (rayopt/geometric_trace.py:82-99),
        t = -<w dy, du>/<w du, du> about the unweighted means of the rays
        with finite slope, from the one-pass sums m[8..19]"""
        G = m[8]
        if G == 0:
            return float("nan")
        by, bu = m[9:11]/G, m[11:13]/G
        W, Wy, Wu = m[13], m[14:16], m[16:18]
        num = m[18] - by.dot(Wu) - bu.dot(Wy) + by.dot(bu)*W
        den = m[19] - 2*bu.dot(Wu) + bu.dot(bu)*W
        return float(-num/den)

    def trace_opd(self, table, y0, u0, spec, A, P, N=None, clip=False, rot0=None, exact=False):
        """rtx_trace_opd: `spec` a dict with the members of `struct rtx_opd`
        (include/rtx.h); A (N,), P (N,3) DeviceArrays.  Asynchronous."""
        table = self._table(table)
        N = y0.shape[0] if N is None else int(N)
        r0 = None if rot0 is None else np.ascontiguousarray(rot0, np.float64).reshape(9)
        rec = np.zeros(1, OPD_DTYPE)
        for k in ("y0_ref", "u0_ref", "M", "d"):
            rec[k] = np.asarray(spec[k], float).reshape(rec[k].shape[1:])
        for k in ("n0", "n_after", "radius"):
            rec[k] = float(spec[k])
        rec["infinite"] = int(bool(spec["infinite"]))
        check(self.lib.rtx_trace_opd(
            self.ctx, ptr(table), len(table), ptr(r0), _code(y0.dtype), N, y0.ptr, u0.ptr,
            int(bool(clip)), ptr(rec), A.ptr, P.ptr, self._flags(exact, False)))

    def opd_regrid(self, A, P, a_ref, p_ref, lscale, rings, n, out=None):
        """rtx_opd_regrid: the n x n OPD map (waves) of a hexapolar bundle of
        `rings` rings from the DEVICE arrays A (N,), P (N,3) of trace_opd and
        the reference ray's A[ref], P[ref].  Returns (map DeviceArray, h,
        number of rays with finite x, y, t)."""
        out = self.empty((n, n)) if out is None else out
        h, count = C.c_double(), C.c_int64()
        p = np.ascontiguousarray(p_ref, np.float64).reshape(3)
        check(self.lib.rtx_opd_regrid(self.ctx, A.shape[0], A.ptr, P.ptr, float(a_ref), ptr(p),
                                      float(lscale), int(rings), int(n), out.ptr, C.byref(h),
                                      C.byref(count)))
        return out, h.value, count.value

    def psf(self, opd_map, pad=4, out=None):
        """rtx_psf: the (pad n)^2 PSF of the DEVICE n x n OPD map in waves
        (GeometricTrace.psf's definition).  Returns a DeviceArray.
        Asynchronous."""
        n = opd_map.shape[0]
        if opd_map.shape != (n, n) or opd_map.dtype != np.float64:
            raise ValueError("the OPD map must be a square float64 DeviceArray")
        out = self.empty((pad*n, pad*n)) if out is None else out
        check(self.lib.rtx_psf(self.ctx, n, opd_map.ptr, int(pad), out.ptr))
        return out

    @staticmethod
    def _square(d_psf):
        M = d_psf.shape[0]
        if d_psf.shape != (M, M) or d_psf.dtype != np.float64:
            raise ValueError("the PSF must be a square float64 DeviceArray")
        return M

    def psf_lines(self, d_psf, out=None):
        """rtx_psf_lines: one read of the DEVICE (M, M) PSF.  Returns (lines
        DeviceArray (2, M) = psf.sum(0), psf.sum(1); peak; total; number of
        elements that are non-finite or outside [0, 2])."""
        M = self._square(d_psf)
        out = self.empty((2, M)) if out is None else out
        stats = (C.c_double*3)()
        check(self.lib.rtx_psf_lines(self.ctx, M, d_psf.ptr, out.ptr, stats))
        return out, stats[0], stats[1], int(stats[2])

    def psf_encircled(self, d_psf, c0, c1, nbins):
        """rtx_psf_encircled: the radial histogram of fftshift(psf) about the
        shifted-frame center (c0, c1) in units of 2^-62 (uint64, nbins)"""
        M = self._square(d_psf)
        bins = np.empty(int(nbins), np.uint64)
        rc = self.lib.rtx_psf_encircled(self.ctx, M, d_psf.ptr, float(c0), float(c1), int(nbins),
                                        ptr(bins))
        if rc == -1:
            raise ValueError("an element's bin is beyond nbins = %d" % nbins)
        check(rc)
        return bins

    def psf_mtf(self, lines, out=None):
        """rtx_psf_mtf: |DFT| of the two DEVICE lines (2, M), the first M//2
        frequencies of each, into a DeviceArray (2, M//2).  Asynchronous."""
        M = lines.shape[1]
        if lines.shape != (2, M) or lines.dtype != np.float64:
            raise ValueError("the lines must be a (2, M) float64 DeviceArray")
        out = self.empty((2, M//2)) if out is None else out
        check(self.lib.rtx_psf_mtf(self.ctx, M, lines.ptr, out.ptr))
        return out

    def psf_window(self, d_psf, i0, j0, w, out=None):
        """rtx_psf_window: the (w, w) window of fftshift(psf) from shifted
        index (i0, j0), indices modulo M, into a DeviceArray.  Asynchronous."""
        M = self._square(d_psf)
        out = self.empty((w, w)) if out is None else out
        check(self.lib.rtx_psf_window(self.ctx, M, d_psf.ptr, int(i0), int(j0), int(w), out.ptr))
        return out

    def psf_metrics(self, d_psf, d, window=0):
        """The figures Analysis.opds (rayopt/analysis.py:319-346) takes from a
        PSF, computed on the DEVICE (M, M) FP64 PSF as rtx_psf writes it
        (unshifted) whose frequency spacing is np.fft.fftfreq(M, d).  Only
        O(M) bytes are transferred:

        * x0, y0: the centroid (psf*x).sum(), (psf*y).sum() of the shifted
          grids, from the line sums (math.fsum);
        * dx: the node spacing; peak: psf.max();
        * ee, r: the encircled energy cumsum(polar_sum(psf, (M/2 + x0/dx,
          M/2 + y0/dx), "azimuthal")) and its radii arange(len(ee))*dx, summed
          in 2^-62 fixed point (exact to M^2 2^-63);
        * freq, mtf: fftfreq(M, dx)[:M//2] and (2, M//2) |DFT| of psf.sum(0)
          and psf.sum(1), Analysis's order;
        * window: None, or (x, y, psf) of the (2w+1)^2 nodes of the shifted
          PSF around the centroid node, x and y relative to the centroid.

        ValueError when an element is non-finite or outside [0, 2], the sum
        exceeds 2 or w > (M-1)//2."""
        M = self._square(d_psf)
        w = int(window)
        if w < 0 or w > (M - 1)//2:
            raise ValueError("window %d is outside [0, %d] for M = %d" % (w, (M - 1)//2, M))
        lines, peak, total, bad = self.psf_lines(d_psf)
        try:
            if bad or not total <= 2:
                raise ValueError("the PSF has %d elements that are non-finite or outside [0, 2] "
                                 "and sums to %r (at most 2 is needed)" % (bad, total))
            cols, rows = lines.download()
            f = np.fft.fftfreq(M, d)
            x0, y0 = math.fsum(f*rows), math.fsum(f*cols)
            fs = np.fft.fftshift(f)
            dx = fs[1] - fs[0]
            c0, c1 = M/2 + x0/dx, M/2 + y0/dx
            corner = np.array([0., M - 1.])
            rc = np.sqrt((corner[None, :] - c1)*(corner[None, :] - c1)
                         + (corner[:, None] - c0)*(corner[:, None] - c0))
            nbins = int(rc.max()) + 1
            bins = self.psf_encircled(d_psf, c0, c1, nbins)
            d_mtf = self.psf_mtf(lines)
            try:
                mtf = d_mtf.download()
            finally:
                d_mtf.free()
        finally:
            lines.free()
        ee = np.cumsum(bins)/2.0**62
        win = None
        if w:
            side = 2*w + 1
            i0, j0 = math.floor(c0 + .5) - w, math.floor(c1 + .5) - w
            d_win = self.psf_window(d_psf, i0, j0, side)
            try:
                pw = d_win.download()
            finally:
                d_win.free()
            xw = fs[(i0 + np.arange(side)) % M] - x0
            yw = fs[(j0 + np.arange(side)) % M] - y0
            xw, yw = np.broadcast_arrays(xw[:, None], yw[None, :])
            win = (xw, yw, pw)
        return PsfMetrics(x0, y0, dx, peak, ee, np.arange(nbins)*dx,
                          np.fft.fftfreq(M, dx)[:M//2], mtf, win)

    def ipc_export(self, darray):
        h = (C.c_ubyte*64)()
        check(self.lib.rtx_ipc_export(self.ctx, darray.ptr, C.cast(h, C.c_void_p)))
        return bytes(h)

    def ipc_open(self, handle):
        h = (C.c_ubyte*64).from_buffer_copy(handle)
        p = C.c_void_p()
        check(self.lib.rtx_ipc_open(self.ctx, C.cast(h, C.c_void_p), C.byref(p)))
        return p.value

    def ipc_close(self, p):
        check(self.lib.rtx_ipc_close(self.ctx, p))

    def download_rays(self, darray, idx):
        """host copy of rays `idx` (1-d integer array) of a device array whose
        trailing axes are (rays, 3) -- a row view (1, ld, 3) or an (N, 3)
        array: one strided D2H when `idx` is an arithmetic progression, else one
        24-byte copy per ray (samples for parity checks)"""
        idx = np.asarray(idx, np.int64).reshape(-1)
        item = darray.dtype.itemsize*3
        out = np.empty((len(idx), 3), darray.dtype)
        if len(idx) == 0:
            return out
        step = int(idx[1] - idx[0]) if len(idx) > 1 else 1
        if len(idx) > 1 and step > 0 and np.all(np.diff(idx) == step):
            check(self.lib.rtx_memcpy2d_d2h(self.ctx, ptr(out), item, darray.ptr + int(idx[0])*item,
                                            step*item, item, len(idx)))
        else:
            for j, i in enumerate(idx):
                check(self.lib.rtx_memcpy_d2h(self.ctx, out[j].ctypes.data_as(C.c_void_p),
                                              darray.ptr + int(i)*item, item))
        self.sync()
        return out

    def aim_infinite_device(self, yo, z, p, angle, yp=None, nrays=None, dtype=np.float64,
                            rings=None):
        """Launch rays of an aimed bundle generated in HBM (rtx_aim_infinite):
        `yp` a DEVICE (N,2) array of pupil coordinates, or None for the
        hexapolar grid with about `nrays` rays (or exactly `rings` rings).
        Returns DeviceArrays (y0, u0)."""
        from .rays import aim_frame
        frame = np.ascontiguousarray(np.concatenate(aim_frame(yo, z, angle)), np.float64)
        pmax = float(np.fabs(np.asarray(p, float)).max())
        if yp is None:
            if rings is None:
                rings = int(np.sqrt(nrays/3. - 1/12.) - 1/2.)
            N = 1 + 3*rings*(rings + 1)
        else:
            rings, N = 0, yp.shape[0]
        y0, u0 = self.empty((N, 3), dtype), self.empty((N, 3), dtype)
        check(self.lib.rtx_aim_infinite(self.ctx, _code(dtype), N, None if yp is None else yp.ptr,
                                        rings, ptr(frame), pmax, y0.ptr, u0.ptr))
        return y0, u0

    def aim_finite_device(self, yo, z, p, radius, yp=None, nrays=None, dtype=np.float64):
        """Launch rays of an aimed bundle from a FINITE object generated in HBM
        (rtx_aim_finite; host restatement: rays.aim_finite).  Returns (y0, u0)."""
        from .rays import finite_frame
        frame = np.ascontiguousarray(np.concatenate(finite_frame(yo, z, radius)), np.float64)
        am = float(np.fabs(np.arctan2(np.asarray(p, float), z)).max())
        if yp is None:
            rings = int(np.sqrt(nrays/3. - 1/12.) - 1/2.)
            N = 1 + 3*rings*(rings + 1)
        else:
            rings, N = 0, yp.shape[0]
        y0, u0 = self.empty((N, 3), dtype), self.empty((N, 3), dtype)
        check(self.lib.rtx_aim_finite(self.ctx, _code(dtype), N, None if yp is None else yp.ptr,
                                      rings, ptr(frame), am, float(z), y0.ptr, u0.ptr))
        return y0, u0

    def aim_rays(self, spec, dtype=np.float64, first=0, count=None, yp=None, want_pupil=False):
        """rtx_aim_plan + rtx_aim_rays: launch rays `first .. first+count-1` of
        the bundle a `rtx_aim` record (rays.aim_record) describes, generated in
        HBM.  `yp`: DEVICE (n,2) FP64 pupil coordinates for GRID_GIVEN.
        Returns (y0, u0) DeviceArrays, plus the (count,2) pupil coordinates
        when `want_pupil`."""
        spec = np.ascontiguousarray(spec)
        n_given = 0 if yp is None else yp.shape[0]
        ypp = None if yp is None else yp.ptr
        total = C.c_int64()
        check(self.lib.rtx_aim_plan(self.ctx, ptr(spec), n_given, ypp, C.byref(total)))
        count = total.value - first if count is None else int(count)
        y0, u0 = self.empty((count, 3), dtype), self.empty((count, 3), dtype)
        po = self.empty((count, 2), np.float64) if want_pupil else None
        check(self.lib.rtx_aim_rays(self.ctx, ptr(spec), n_given, ypp, _code(dtype), int(first),
                                    count, y0.ptr, u0.ptr, None if po is None else po.ptr))
        return (y0, u0, po) if want_pupil else (y0, u0)

    def aim_rays_into(self, spec, y_dst, u_dst, count, first=0, yp=None):
        """rtx_aim_rays into existing device rows (DeviceArray views)"""
        spec = np.ascontiguousarray(spec)
        check(self.lib.rtx_aim_rays(self.ctx, ptr(spec), 0 if yp is None else yp.shape[0],
                                    None if yp is None else yp.ptr, _code(y_dst.dtype), int(first),
                                    int(count), y_dst.ptr, u_dst.ptr, None))

    def aim_count(self, spec, yp=None):
        """number of rays the record generates (after clipping / filtering)"""
        spec = np.ascontiguousarray(spec)
        total = C.c_int64()
        check(self.lib.rtx_aim_plan(self.ctx, ptr(spec), 0 if yp is None else yp.shape[0],
                                    None if yp is None else yp.ptr, C.byref(total)))
        return total.value

    def aim_infinite_into(self, y_dst, u_dst, count, rings, frame, pmax, yp=None):
        """rtx_aim_infinite into existing device rows (DeviceArray views)"""
        frame = np.ascontiguousarray(frame, np.float64)
        check(self.lib.rtx_aim_infinite(self.ctx, _code(y_dst.dtype), int(count),
                                        None if yp is None else yp.ptr, int(rings), ptr(frame),
                                        float(pmax), y_dst.ptr, u_dst.ptr))

    def selftest_math(self, a, b):
        """(6, n): engine a/b, IEEE a/b, engine sqrt(a), IEEE sqrt(a),
        engine 1/sqrt(a), IEEE 1/sqrt(a)"""
        a = np.ascontiguousarray(a, np.float64)
        b = np.ascontiguousarray(b, np.float64)
        out = np.empty((6, a.size))
        check(self.lib.rtx_selftest_math(self.ctx, a.size, ptr(a), ptr(b), ptr(out)))
        return out

    def moments(self, y, w=None, N=None, center=None):
        """Weighted moments of device intercepts about `center`
        (include/rtx.h rtx_moments): 8 doubles."""
        m = np.zeros(8)
        N = y.shape[-2] if N is None else int(N)
        c = None if center is None else np.ascontiguousarray(center, np.float64)
        check(self.lib.rtx_moments(self.ctx, _code(y.dtype), N, y.ptr,
                                   None if w is None else w.ptr, ptr(c), ptr(m)))
        return m

    def rms(self, y, w=None, N=None, ref_point=None, comm_sum=None):
        """GeometricTrace.rms (rayopt/geometric_trace.py:171-183) of device
        intercepts `y` (N,3) without a D2H of the rays: centre = unweighted
        mean (or `ref_point`), rms = sqrt(sum w |y - y0|^2) with the
        reference's default weights 1/N when `w` is None.  Like the
        reference it is NOT NaN-masked: any non-finite ray gives NaN.
        `comm_sum` (callable: 8-vector -> summed 8-vector) makes it the rms of
        a ray-sharded bundle (one all-reduce per pass)."""
        red = comm_sum or (lambda v: v)
        if ref_point is None:
            m = red(self.moments(y, w, N))
            if m[4] != m[5]:
                return float("nan")
            ref_point = (m[6]/m[5], m[7]/m[5])
        m = red(self.moments(y, w, N, center=ref_point))
        if m[4] != m[5]:
            return float("nan")
        return float(np.sqrt(m[3]/m[5] if w is None else m[3]))


    def refocus_shift(self, y, inc, w=None, N=None, comm_sum=None):
        """The focus shift of GeometricTrace.refocus (rayopt/geometric_trace.py:
        82-99), t = -<w y, u>/<w u, u> about the means of the finite rays, from
        DEVICE arrays y (N,3) and inc (N,3) of the surface -- no D2H of the rays.
        `comm_sum` all-reduces the 8 moments for ray-sharded bundles."""
        red = comm_sum or (lambda v: v)
        N = y.shape[-2] if N is None else int(N)

        def mom(center):
            m = np.zeros(8)
            c = None if center is None else np.ascontiguousarray(center, np.float64)
            check(self.lib.rtx_focus_moments(self.ctx, _code(y.dtype), N, y.ptr, inc.ptr,
                                             None if w is None else w.ptr, ptr(c), ptr(m)))
            return red(m)
        m = mom(None)
        if m[0] == 0:
            return float("nan")
        m = mom(m[2:6]/m[0])
        return float(-m[6]/m[7])


_default = {}


def default_engine(device=0):
    """process-wide engine for `device` (created on first use)"""
    e = _default.get(device)
    if e is None or e.ctx is None:
        e = _default[device] = Engine(device)
    return e
