/*
 * rtx.h -- C ABI of the B200-native sequential geometric ray-trace engine.
 *
 * This is the drop-in boundary for ONE hot path of quartiq/rayopt: the
 * per-surface  transfer -> intercept -> clip -> refract  loop
 *
 *     GeometricTrace.propagate      rayopt/geometric_trace.py:72-80
 *       System.propagate            rayopt/system.py:459-464
 *         TransformMixin.to_normal  rayopt/elements.py:174 (156-163)
 *         Interface.propagate       rayopt/elements.py:306-315
 *           Spheroid.intercept      rayopt/elements.py:477-501
 *           Interface.intercept     rayopt/elements.py:333-349 (Newton, aspheres)
 *           Element.clip            rayopt/elements.py:206-209
 *           Interface.refract       rayopt/elements.py:351-369
 *           Spheroid.surface_normal rayopt/elements.py:457-475
 *           Spheroid.surface_sag    rayopt/elements.py:440-455
 *         TransformMixin.from_normal rayopt/elements.py:171
 *
 * The reference has no FFI layer (pure numpy); the boundary it would bind is
 * "one call per GeometricTrace.propagate()": a table of per-surface POD
 * records (what System.propagate reads off each Element for one wavelength)
 * plus the launch rays, returning the (S, N, 3) / (S, N) result arrays the
 * reference stores into GeometricTrace.y/u/i/t (geometric_trace.py:80).
 *
 * Plain C, plain pointers and sizes.  No torch types.  Every function returns
 * 0 on success, a NEGATIVE rtx error (RTX_E_*) for argument errors, or a
 * POSITIVE cudaError_t for CUDA failures.  Numerical failure (missed surface,
 * total internal reflection, vignetting, Newton non-convergence) is NOT an
 * error: it is NaN in the data, exactly where the reference puts it
 * (elements.py:208, 347-348, 367, 496).
 *
 * A context is bound to one GPU and one CUDA stream and is not thread-safe;
 * use one context per GPU (one process per GPU in multi-GPU runs).
 */
#ifndef RTX_H
#define RTX_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTX_ABI_VERSION 2

/* maximum number of even-asphere coefficients per surface (Spheroid.aspherics,
 * elements.py:422-424).  Longer lists are rejected with RTX_E_UNSUPPORTED. */
#define RTX_MAX_ASPH 10
/* maximum number of surfaces in one trace call (bounded by the shared-memory
 * staging of the surface table) */
#define RTX_MAX_SURFACES 256

/* rtx_surface.flags */
#define RTX_F_ROTATED 1u /* apply rot (TransformMixin.rotated, elements.py:135) */
#define RTX_F_ALT     2u /* Spheroid.alternate_intersection, elements.py:497-498 */

/* dtype */
#define RTX_F64 0
#define RTX_F32 1

/* keep policy */
#define RTX_KEEP_ALL  0 /* store every surface: outputs have S rows   */
#define RTX_KEEP_LAST 1 /* store only the last surface: outputs have 1 row */

/* trace flags */
#define RTX_EXACT      1u /* FP64 only: unfused IEEE arithmetic in numpy's
                             evaluation order (bit-identical to the reference
                             on unrotated analytic surfaces) */
#define RTX_STORE_DIRECT 2u /* debug: force per-thread strided stores instead
                               of the shared-memory staged bulk (TMA) stores */
#define RTX_RPT1       4u /* tuning: one ray per thread  (default: library's choice) */
#define RTX_RPT2       8u /* tuning: two rays per thread */
#define RTX_GATHER_XY 16u /* rtx_trace_gather: the intercept buffers dst[k] are
                             (Ntotal, 2) arrays receiving x,y only -- what a spot
                             diagram reads (rayopt/analysis.py:274): 16 instead of
                             24 bytes per ray over NVLink */

/* errors */
#define RTX_OK              0
#define RTX_E_BADARG       -1
#define RTX_E_UNSUPPORTED  -2
#define RTX_E_NOMEM        -3

/*
 * One traced surface for one wavelength: everything System.propagate
 * (system.py:459-464) and Interface.propagate (elements.py:306-315) read off
 * the Element.  "Derived" members are scalars the reference computes in
 * Python per call; a caller that wants bit-identical results must compute
 * them with the same expressions (rayopt_b200/surface_table.py does);
 * rtx_surface_finalize() fills them the C way.
 */
typedef struct rtx_surface {
    double offset[3]; /* e.offset, subtracted in the incoming frame (system.py:461) */
    double rot[9];    /* e.rot_normal, row-major; to_normal is y @ rot.T,
                         from_normal is y @ rot (elements.py:156-175); used
                         only if RTX_F_ROTATED */
    double c;         /* Spheroid.curvature */
    double k;         /* Spheroid.conic */
    double kc2;       /* derived: (1 + k)*c**2          (elements.py:448,467) */
    double radius2;   /* derived: radius**2, +inf = no aperture (elements.py:207) */
    double mu;        /* 1 (no material), -1 (mirror) or n0/n (elements.py:283-289) */
    double muf;       /* derived: abs(mu)               (elements.py:360) */
    double sgn;       /* derived: sign(mu)              (elements.py:367) */
    double mu2m1;     /* derived: mu**2 - 1             (elements.py:366) */
    double n0;        /* index before the surface: t = s*n0 (elements.py:315) */
    double n;         /* index after the surface (fills GeometricTrace.n) */
    double asph[RTX_MAX_ASPH];  /* Spheroid.aspherics[j] multiplies r^(2(j+1)) */
    double dasph[RTX_MAX_ASPH]; /* derived: 2*(j+1)*asph[j] (elements.py:472) */
    int32_t n_asph;   /* -1: aspherics is None (analytic intercept);
                         >=0: len(aspherics), Newton intercept even if 0
                         (elements.py:478-479) */
    uint32_t flags;   /* RTX_F_* */
} rtx_surface;

typedef struct rtx_ctx rtx_ctx;

/* ---- library ---------------------------------------------------------- */
int rtx_abi_version(void);
/* sizeof(rtx_surface) / sizeof(rtx_aim) / sizeof(rtx_opd) as compiled, for
 * binding-side layout checks */
size_t rtx_sizeof_surface(void);
size_t rtx_sizeof_aim(void);
size_t rtx_sizeof_opd(void);
/* number of CUDA devices visible, or 0 */
int rtx_device_count(void);
/* static string for an rtx (negative) or CUDA (positive) error code */
const char *rtx_strerror(int code);
/* fill the derived members of n records from c,k,mu,asph and `radius` */
int rtx_surface_finalize(rtx_surface *surf, int n, const double *radius);

/* ---- context ---------------------------------------------------------- */
int rtx_init(int device, rtx_ctx **out);
int rtx_free(rtx_ctx *ctx);
int rtx_sync(rtx_ctx *ctx);
/* device properties: SM count, and bytes of free / total HBM */
int rtx_device_info(rtx_ctx *ctx, int *sm_count, size_t *free_bytes,
                    size_t *total_bytes, char *name, int name_len);

/* ---- memory (so that host code needs no other CUDA binding) ----------- */
int rtx_malloc(rtx_ctx *ctx, size_t bytes, void **dptr);
int rtx_free_device(rtx_ctx *ctx, void *dptr);
int rtx_host_alloc(rtx_ctx *ctx, size_t bytes, void **hptr); /* pinned */
/* ctx may be NULL (page-locked memory may outlive the context that made it) */
int rtx_host_free(rtx_ctx *ctx, void *hptr);
/*
 * NUMA placement of the calling thread (one process per GPU): enable = 1 pins
 * the thread to the CPUs of the NUMA node this context's GPU hangs off
 * (/sys/bus/pci/devices/<bus id>/numa_node) and makes that node the preferred
 * one for its allocations, so that page-locked buffers allocated afterwards
 * (rtx_host_alloc, the library's own bounce buffers) are local to the GPU's
 * PCIe root; enable = 0 restores the affinity and policy saved by the last
 * bind.  *node (may be NULL) receives the node, -1 when the platform does not
 * report one (nothing is changed then).
 */
int rtx_numa_bind(rtx_ctx *ctx, int enable, int *node);
/* asynchronous on the context stream; rtx_sync() to complete */
int rtx_memcpy_h2d(rtx_ctx *ctx, void *dst, const void *src, size_t bytes);
int rtx_memcpy_d2h(rtx_ctx *ctx, void *dst, const void *src, size_t bytes);
int rtx_memcpy_d2d(rtx_ctx *ctx, void *dst, const void *src, size_t bytes);
/* strided D2H: `height` rows of `width` bytes */
int rtx_memcpy2d_d2h(rtx_ctx *ctx, void *dst, size_t dpitch, const void *src,
                     size_t spitch, size_t width, size_t height);
int rtx_memset(rtx_ctx *ctx, void *dptr, int value, size_t bytes);

/* ---- timing on the context stream (CUDA events) ----------------------- */
int rtx_timer_start(rtx_ctx *ctx);
int rtx_timer_stop(rtx_ctx *ctx, float *ms); /* synchronises */
/* device time of the most recent trace kernel launch(es) of the last
 * rtx_trace call, measured with events around the launch */
int rtx_last_kernel_ms(rtx_ctx *ctx, float *ms);
/* number of kernels this context has launched so far */
int64_t rtx_launch_count(rtx_ctx *ctx);

/* ---- the hot path ------------------------------------------------------ */
/*
 * March N rays through S surfaces in one launch.  Replaces the loop
 * GeometricTrace.propagate -> System.propagate (geometric_trace.py:72-80,
 * system.py:459-464).
 *
 *  surf[S]  host pointer, surface records for system[start:stop]
 *  rot0     host pointer to 9 doubles or NULL: rot_normal of system[start-1]
 *           when that element is rotated; the launch rays are mapped with
 *           from_normal (y @ rot0) first (geometric_trace.py:76)
 *  dtype    RTX_F64 / RTX_F32: element type of ALL ray arrays
 *  y0,u0    DEVICE pointers, (N,3) C-contiguous: launch rays in the normal
 *           frame of system[start-1]
 *  clip     0/1: the `clip` argument of propagate (elements.py:309-310)
 *  keep     RTX_KEEP_ALL / RTX_KEEP_LAST
 *  ld       row pitch of the outputs in RAYS (>= N).  Outputs are DEVICE
 *           arrays Y,U,I: (rows, ld, 3), T: (rows, ld); rows = S or 1.
 *           With ld a multiple of 128 rays (64 suffices in FP64) the kernel
 *           uses staged bulk (TMA) stores and writes whole groups of 32 x
 *           rays-per-thread rays (columns N..ld-1 are padding and receive
 *           unspecified values); a multiple of 32 or 64 selects a kernel with
 *           fewer rays per thread; any other ld takes the per-thread store
 *           path and touches only columns < N.
 *           Y: intercepts, U: excidence, I: incidence directions (unclipped),
 *           T: optical path s*n0 -- all in the surface-normal frame, exactly
 *           the tuple System.propagate yields (system.py:463).
 *           Any of Y,U,I,T may be NULL to skip storing that array.
 */
int rtx_trace(rtx_ctx *ctx, const rtx_surface *surf, int S,
              const double *rot0, int dtype, int64_t N,
              const void *y0, const void *u0, int clip, int keep, int64_t ld,
              void *Y, void *U, void *I, void *T, unsigned flags);

/*
 * Batched bundles (SURVEY 8f-3): nb <= RTX_MAX_BATCH bundles of the SAME lens
 * (S surfaces each) -- typically one per wavelength or field: surf[b] its
 * table, N[b] its rays, y0[b], u0[b], Y[b].. its DEVICE arrays (rows x ld
 * pitch shared; Y, U, I, T may each be NULL as a whole) -- marched by ONE
 * launch: the persistent CTAs walk a launch-wide tile list and re-stage the
 * surface table (TMA) when they cross into the next bundle.  Removes the
 * kernel boundaries between the wavelength traces of one analysis step.
 */
#define RTX_MAX_BATCH 8
int rtx_trace_batch(rtx_ctx *ctx, int nb, const rtx_surface *const *surf, int S,
                    const double *rot0, int dtype, const int64_t *N,
                    const void *const *y0, const void *const *u0, int clip,
                    int keep, int64_t ld, void *const *Y, void *const *U,
                    void *const *I, void *const *T, unsigned flags);

/*
 * The same with HOST buffers in the reference layout, any number of bundles
 * (nb >= 1; per bundle y0,u0 (N[b],3) and Y,U,I (rows,N[b],3), T (rows,N[b])):
 * the front end for callers that issue many SMALL traces of one lens --
 * Analysis loops 3 fields x 3-5 wavelengths x 150-ray bundles
 * (rayopt/analysis.py:226-245, 266-280).  All launch rays go up in ONE H2D
 * from a page-locked bounce buffer, the bundles are marched 8 per launch
 * (rtx_trace_batch), all results come back in ONE D2H, one synchronisation.
 * Bundles too large for the bounce buffer are traced one by one through
 * rtx_trace_host.  Y, U, I, T may each be NULL as a whole.
 */
int rtx_trace_batch_host(rtx_ctx *ctx, int nb, const rtx_surface *const *surf,
                         int S, const double *rot0, int dtype, const int64_t *N,
                         const void *const *y0, const void *const *u0, int clip,
                         int keep, void *const *Y, void *const *U,
                         void *const *I, void *const *T, unsigned flags);

/*
 * Optional warp-ballot vignetting mask for the following rtx_trace /
 * rtx_trace_gather calls on device buffers: dmask (DEVICE, ceil(N/32) words,
 * or NULL to switch it off) receives bit (ray % 32) of word ray / 32 = 1 when
 * the ray leaves the last traced surface with a finite direction -- i.e. it
 * was not clipped (Element.clip, elements.py:206-209) and hit no NaN
 * condition on the way (elements.py:347-348, 367, 496).
 */
int rtx_set_mask_output(rtx_ctx *ctx, uint32_t *dmask);

/*
 * Optional per-ray optical path sum for the following rtx_trace calls on
 * device buffers: dsum (DEVICE, N values of the trace dtype, or NULL = off)
 * receives sum over traced surfaces 0..upto (inclusive; upto < 0: all) of
 * t -- the accumulation GeometricTrace.opd starts from
 * (rayopt/geometric_trace.py:102), without reading the (S,N) array again.
 */
int rtx_set_path_sum_output(rtx_ctx *ctx, void *dsum, int upto);

/*
 * Same call with HOST buffers in the reference layout: y0,u0 (N,3);
 * Y,U,I (rows,N,3), T (rows,N) C-contiguous (GeometricTrace.y/u/i/t rows
 * start..stop-1).  Synchronous.  Three regimes by size (rays + results):
 *   <= 16 KB  (ray aiming: 1-3 rays, hundreds of calls, rayopt/system.py:
 *             507-555) ZERO-COPY: the kernel reads the rays from and writes
 *             the results to a page-locked bounce buffer over PCIe -- one
 *             launch, one synchronisation;
 *   <= 4 MB   one H2D, one launch, one D2H through the bounce buffer;
 *   larger    rays are processed in ~256 MB chunks; H2D, kernel and D2H of
 *             consecutive chunks overlap on two streams.  Host buffers from
 *             rtx_host_alloc (pinned) copy at full PCIe rate; pageable ones
 *             work too.
 * The mask / path-sum side outputs do not apply to host-buffer calls.
 */
int rtx_trace_host(rtx_ctx *ctx, const rtx_surface *surf, int S,
                   const double *rot0, int dtype, int64_t N,
                   const void *y0, const void *u0, int clip, int keep,
                   void *Y, void *U, void *I, void *T, unsigned flags);

/* ---- fused trace + gather over peer memory (multi-GPU, SURVEY 8e) ------- */
/*
 * Cross-process device memory: export a buffer of this context's GPU as an
 * opaque 64-byte handle (cudaIpcGetMemHandle), open a handle exported by
 * another process of the same node (peer access over NVLink is enabled
 * lazily), close it again.
 */
#define RTX_IPC_HANDLE_BYTES 64
int rtx_ipc_export(rtx_ctx *ctx, void *dptr, unsigned char *handle);
int rtx_ipc_open(rtx_ctx *ctx, const unsigned char *handle, void **dptr);
int rtx_ipc_close(rtx_ctx *ctx, void *dptr);
/*
 * Trace this rank's shard (N rays, DEVICE y0,u0) and store the LAST surface's
 * intercepts straight into `npeers` (<= 8) gather buffers dst[k] -- (Ntotal_pad, 3)
 * arrays of `dtype` that are local or peer-GPU memory (rtx_ipc_open) -- at ray
 * offset dst_offset: the all-gather of GeometricTrace.y[-1] is done by the
 * trace kernel's own TMA bulk stores over NVLink instead of a separate
 * collective.  dst_i (may be NULL) is a second set of npeers buffers that
 * receive the last surface's INCIDENCE directions i[-1] the same way (the
 * through-focus spots of rayopt/analysis.py:274-280 read y[-1] and i[-1]).
 * Bulk stores need 16-byte aligned runs and write whole groups of 32 x
 * rays-per-thread rays: with dst_offset and N multiples of 64 rays (FP64;
 * 128 for the fastest FP32 kernel) exactly rays dst_offset .. dst_offset +
 * N - 1 are written by bulk stores; for any other N or offset the library
 * steps down to a kernel with smaller groups and finally to per-ray stores
 * that touch exactly N rays, so a shard can never spill into its
 * neighbour's range.  Asynchronous on
 * the context stream; after rtx_sync on every rank and a cross-rank barrier
 * all buffers hold the full spot.
 */
int rtx_trace_gather(rtx_ctx *ctx, const rtx_surface *surf, int S,
                     const double *rot0, int dtype, int64_t N, const void *y0,
                     const void *u0, int clip, int npeers, void *const *dst,
                     void *const *dst_i, int64_t dst_offset, unsigned flags);

/* ---- self-test --------------------------------------------------------- */
/*
 * The kernels use their own branch-free FP64 division / sqrt / rsqrt (the
 * library sequences minus the slow-path subroutine).  For n host operand
 * pairs (a, b) writes 6*n doubles to `out` (host): a/b (engine), a/b (IEEE
 * __ddiv_rn), sqrt(a) (engine), sqrt(a) (IEEE), 1/sqrt(a) (engine),
 * 1/sqrt(a) (IEEE).
 */
int rtx_selftest_math(rtx_ctx *ctx, int64_t n, const double *a, const double *b,
                      double *out);

/* ---- fused last-surface reductions (geometric_trace.py:171-183) ------- */
/*
 * Weighted moments of DEVICE intercepts y (N,3), dtype as given, about
 * `center` (host, 2 doubles, or NULL for the origin); dx = x - center[0]:
 * m[0]=sum w, m[1]=sum w*dx, m[2]=sum w*dy, m[3]=sum w*(dx^2+dy^2),
 * m[4]=count finite, m[5]=count total, m[6]=sum dx, m[7]=sum dy.
 * Rays with non-finite x or y are skipped (counted in m[5] only).
 * w (device, N values of dtype) may be NULL (w = 1).  m: host, 8 doubles.
 * Two calls (moments about 0, then about the mean) give the reference's
 * rms() without moving y to the host; per-rank moments add up
 * (all-reduce of 8 doubles) for ray-sharded multi-GPU runs.
 */
int rtx_moments(rtx_ctx *ctx, int dtype, int64_t N, const void *y,
                const void *w, const double *center, double *m);

/* ---- fused epilogues: the march with no per-surface stores (SURVEY 8f-1, 8f-4) */
/*
 * rms / centroid / refocus moments of surface S-1 in ONE launch from the
 * launch rays (DEVICE y0,u0; surf[S] = system[start:at+1]): the trace kernel
 * keeps the rays in registers, accumulates the moments there and writes 20
 * doubles -- GeometricTrace.rms (rayopt/geometric_trace.py:171-183) and the
 * focus shift of GeometricTrace.refocus (:82-99) of 1e9 rays without storing
 * a single intercept.  About the guess centres center[0..1] (intercept x,y)
 * and center[2..3] (slope i_x/i_z, i_y/i_z) -- e.g. the chief ray's, so that
 * the shift to the true means is cancellation-free (host, 4 doubles or NULL);
 * w: DEVICE weights (N values of dtype) or NULL (= 1).  m (host, 20 doubles):
 *   m[0..7]   as rtx_moments (sum w, sum w dx, sum w dy, sum w (dx^2+dy^2),
 *             #finite, #total, sum dx, sum dy)
 *   m[8..19]  over the rays with a finite slope: #good, sum dy (2), sum du (2),
 *             sum w, sum w dy (2), sum w du (2), sum w dy.du, sum w du.du
 * Per-rank moments add up (one all-reduce of 20 doubles) for ray-sharded runs.
 */
#define RTX_NMOMENTS 20
int rtx_trace_reduce(rtx_ctx *ctx, const rtx_surface *surf, int S,
                     const double *rot0, int dtype, int64_t N, const void *y0,
                     const void *u0, int clip, const void *w,
                     const double *center, double *m, unsigned flags);

/*
 * The per-ray part of GeometricTrace.opd (rayopt/geometric_trace.py:101-131)
 * as the epilogue of the march to surface `after` (surf[S] = system[1:after+1]):
 *   A = sum_s t[s] - tj*n0 + ti*n_after,   P = y' + ti*u' - (0, 0, radius)
 * with tj = u0_ref.(y0_ref - y0) for an object at infinity (`infinite`, :104-109),
 * y' = y[after] @ M + d, u' = u[after] @ M the change to the image frame
 * (:116-120; M = ea.rot_normal @ ei.rot_normal.T, d = (origins[after] -
 * origins[image]) @ ei.rot_normal.T - y[image, ref]) and ti the intercept with
 * the reference sphere Spheroid(curvature=1/radius) after y'_z += radius
 * (:123-124).  The caller finishes with the reference ray:
 *   t = -(A - A[ref])/(l/scale),  py = P - P[ref].
 * A: DEVICE (N,), P: DEVICE (N,3) of dtype.  Asynchronous.
 */
typedef struct rtx_opd {
    double y0_ref[3], u0_ref[3]; /* launch ray `ref` (row 0 of the trace) */
    double n0, n_after;
    double M[9], d[3];
    double radius;
    int32_t infinite;
    int32_t reserved;
} rtx_opd;
int rtx_trace_opd(rtx_ctx *ctx, const rtx_surface *surf, int S,
                  const double *rot0, int dtype, int64_t N, const void *y0,
                  const void *u0, int clip, const rtx_opd *opd, void *A,
                  void *P, unsigned flags);

/* ---- launch rays generated in HBM (SURVEY 8f-2) -------------------------- */
/*
 * Aimed bundle for an infinite conjugate (InfiniteConjugate.aim, rectilinear
 * projection, rayopt/conjugates.py:208-213,236-255; plane object surface) for
 * ONE field point: frame = {u[3], ybase[3], s[3], m[3]} (host, 12 doubles: the
 * common direction, yz - z*u, and the normalised sagittal / meridional
 * vectors of rayopt/utils.py:102-114), pmax = fabs(p).max() (Pupil.map,
 * rayopt/pupils.py:100).  Pupil coordinates: yp DEVICE (N,2) of `dtype`, or
 * NULL for the hexapolar grid of pupil_distribution (rayopt/utils.py:174-180)
 * with `hex_rings` rings, N = 1 + 3*hex_rings*(hex_rings+1).  Writes DEVICE
 * y0,u0 (N,3).  Asynchronous on the context stream.
 */
int rtx_aim_infinite(rtx_ctx *ctx, int dtype, int64_t N, const void *yp,
                     int hex_rings, const double *frame, double pmax, void *y0,
                     void *u0);

/*
 * Same for a finite conjugate (FiniteConjugate.aim, rayopt/conjugates.py:
 * 137-166; plane object surface, non-telecentric pupil, filter=False): frame =
 * {y[3] object point, u[3] = (0,0,z) - y, s[3], m[3]}, am = max |arctan2(p, z)|
 * (the pupil half-angle Pupil.map scales with), z the pupil distance.
 */
int rtx_aim_finite(rtx_ctx *ctx, int dtype, int64_t N, const void *yp,
                   int hex_rings, const double *frame, double am, double z,
                   void *y0, void *u0);

/*
 * General generator: the pupil grids of pupil_distribution (rayopt/utils.py:
 * 118-199), Pupil.map with its elliptical filter (rayopt/pupils.py:97-107) and
 * Conjugate.aim (rayopt/conjugates.py:137-166, 236-255) evaluated per ray on
 * the device.  Candidates rejected by a predicate (mesh points outside the
 * unit circle, rays outside the filter ellipse) are squeezed out in order
 * (two passes: block counts, host prefix sum, generation).
 *
 *  conjugate  0 infinite: frame = {u[3], ybase[3] = yz - z*u, s[3], m[3]}
 *             1 finite:   frame = {y[3] object point, u0[3], s[3], m[3]}
 *             (the projection, a telecentric pupil and a curved FINITE object
 *             surface only change these per-field constants: the host computes
 *             them with the reference's expressions, rayopt_b200/rays.py)
 *  grid       RTX_GRID_*; n = rings (hexapolar), mesh side (square,
 *             triangular: n x n points clipped to the unit circle + centre
 *             ray), number of random rays (+ centre ray); RTX_GRID_LINES: up to
 *             two np.linspace segments seg[k] = (x0, y0, x1, y1) of seg_m[k]
 *             points (meridional, sagittal, cross, tee, half-meridional);
 *             RTX_GRID_GIVEN: pupil coordinates yp, DEVICE (n_given, 2) FP64
 *  pmax       Pupil.map's scale fabs(a).max() (finite: of arctan2(a, z))
 *  filter     keep ((q - fc)^2 / fd2).sum() <= 1, q the scaled coordinates
 *  curved     infinite object only: intercept the rays with `surface`
 *             (system[0], in its own frame) instead of the plane z = 0
 */
#define RTX_GRID_GIVEN      0
#define RTX_GRID_HEXAPOLAR  1
#define RTX_GRID_SQUARE     2
#define RTX_GRID_TRIANGULAR 3
#define RTX_GRID_RANDOM     4
#define RTX_GRID_LINES      5
typedef struct rtx_aim {
    int32_t conjugate, grid, filter, curved;
    int64_t n;
    uint64_t seed;      /* RTX_GRID_RANDOM: counter-based generator */
    double seg[2][4];
    int64_t seg_m[2];
    double frame[12];
    double pmax, z;
    double fc[2], fd2[2];
    rtx_surface surface;
} rtx_aim;
/* number of rays the spec generates (runs the counting pass when a predicate
 * can reject candidates; the plan is cached in the context) */
int rtx_aim_plan(rtx_ctx *ctx, const rtx_aim *spec, int64_t n_given,
                 const void *yp, int64_t *n_rays);
/* rays first .. first+count-1 of the bundle into DEVICE y0,u0 (count,3) of
 * dtype; yp_out: optional DEVICE (count,2) FP64 receiving the fractional pupil
 * coordinates of those rays.  Asynchronous on the context stream. */
int rtx_aim_rays(rtx_ctx *ctx, const rtx_aim *spec, int64_t n_given,
                 const void *yp, int dtype, int64_t first, int64_t count,
                 void *y0, void *u0, void *yp_out);

/*
 * Moments for GeometricTrace.refocus (rayopt/geometric_trace.py:82-99) on
 * DEVICE arrays of one surface: y = intercepts (N,3), inc = incidence
 * directions (N,3); u = inc_xy/inc_z (tanarcsin); rays with non-finite u are
 * skipped.  About `center` = (y_x, y_y, u_x, u_y) (host, or NULL = 0):
 * m[0]=#good, m[1]=#total, m[2..3]=sum dy, m[4..5]=sum du,
 * m[6]=sum w (dy.du), m[7]=sum w (du.du).  The focus shift is
 * -m[6]/m[7] taken about the means of the good rays (two calls).
 */
int rtx_focus_moments(rtx_ctx *ctx, int dtype, int64_t N, const void *y,
                      const void *inc, const void *w, const double *center,
                      double *m);

/* ---- wavefront: OPD map and PSF (rayopt/geometric_trace.py:101-169) ------ */
/*
 * GeometricTrace.opd(resample) of a HEXAPOLAR launch bundle generated without
 * a pupil filter (pupil_distribution("hexapolar"), rayopt/utils.py:180-186:
 * N = 1 + 3*rings*(rings+1) rays, ring r of 6r rays starting at 1 + 3r(r-1)),
 * regridded on the device.  From the DEVICE arrays A (N,), P (N,3) of
 * rtx_trace_opd and the reference ray's A[ref] = a_ref and P[ref] = p_ref
 * (host, 3 doubles): per ray t = -(A - a_ref)/lscale (lscale = l/scale) and
 * (x, y) = P - p_ref; h = max |x|, |y| over rays whose x, y, t are finite
 * (:135-139).  DEVICE map (n,n) receives t linearly interpolated at the
 * nodes (x_i, y_j) = np.mgrid[-1:1:1j*n, -1:1:1j*n]*h, row i = x.  The
 * triangulation is the structured one of the launch grid (6*rings^2
 * triangles), not Delaunay: a triangle with a non-finite vertex is dropped,
 * so vignetted gaps stay NaN, and nodes outside every triangle are NaN.  A
 * node on a shared edge takes the value of the lowest-index triangle, so the
 * map is bit-identical run to run.  Host outputs: *h (may be NULL) and
 * *n_finite (may be NULL), the count of rays with finite x, y, t (0: no ray
 * made it through).  Synchronises.
 */
int rtx_opd_regrid(rtx_ctx *ctx, int64_t N, const double *A, const double *P,
                   double a_ref, const double *p_ref, double lscale, int rings,
                   int64_t n, double *map, double *h, int64_t *n_finite);

/*
 * GeometricTrace.psf (rayopt/geometric_trace.py:150-157) of an n x n OPD map
 * in waves (DEVICE, FP64, NaN outside the pupil): pupil function
 * where(finite, exp(-2 pi i o), 0)/sqrt(count), its zero-padded 2-D DFT of
 * size M x M, M = pad*n, and psf = |DFT|^2/M^2 into DEVICE psf (M,M) FP64.
 * Any M: every 1-D DFT is a Bluestein convolution computed with the library's
 * own power-of-two FFT; the first pass transforms only the n non-zero rows.
 * Scratch of about 32*n*M bytes plus up to 1 GB for large M is taken from the
 * stream-ordered allocator.  Asynchronous on the context stream.
 */
int rtx_psf(rtx_ctx *ctx, int64_t n, const double *map, int pad, double *psf);

/* ---- PSF figures (rayopt/analysis.py:319-346, Analysis.opds) ------------- */
/*
 * On the UNSHIFTED M x M FP64 PSF in DEVICE memory, as rtx_psf writes it
 * (1 <= M <= RTX_PSF_MAX_M).  fftshift maps unshifted index i to shifted
 * index (i + M/2) % M.  Every result is bit-identical run to run.
 */
#define RTX_PSF_MAX_M 1048576

/*
 * One read of psf: DEVICE lines (2, M) = psf.sum(0), then psf.sum(1), each
 * sum in a fixed order; HOST stats[3] = max element, sum of all elements,
 * and the count of elements that are non-finite or outside [0, 2].
 * Synchronises.
 */
int rtx_psf_lines(rtx_ctx *ctx, int64_t M, const double *psf, double *lines,
                  double *stats);

/*
 * special_sums.polar_sum(fftshift(psf), (c0, c1), "azimuthal") in fixed
 * point: shifted node (I, J) falls in bin trunc(sqrt((J - c1)^2 + (I - c0)^2))
 * (unfused IEEE in that order) and adds rint(psf * 2^62) to HOST bins
 * (nbins uint64).  Integer sums do not depend on the order of the atomics.
 * Needs every element in [0, 2] and their sum <= 2 (rtx_psf_lines checks
 * both).  RTX_E_BADARG when an element's bin is >= nbins.  Synchronises.
 */
int rtx_psf_encircled(rtx_ctx *ctx, int64_t M, const double *psf, double c0,
                      double c1, int64_t nbins, uint64_t *bins);

/*
 * |DFT_M| of the two DEVICE lines (2, M) into DEVICE mtf (2, M/2): the first
 * M/2 frequencies of each, with the library's Bluestein FFT (M >= 2).
 * Asynchronous on the context stream.
 */
int rtx_psf_mtf(rtx_ctx *ctx, int64_t M, const double *lines, double *mtf);

/*
 * DEVICE out (w, w) = fftshift(psf)[(i0 + a) % M, (j0 + b) % M], indices
 * taken modulo M (1 <= w <= M).  Asynchronous on the context stream.
 */
int rtx_psf_window(rtx_ctx *ctx, int64_t M, const double *psf, int64_t i0,
                   int64_t j0, int64_t w, double *out);

#ifdef __cplusplus
}
#endif
#endif /* RTX_H */
