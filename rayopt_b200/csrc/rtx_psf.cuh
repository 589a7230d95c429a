// rtx_psf.cuh -- device kernels of the wavefront pipeline behind
// GeometricTrace.opd(resample) and GeometricTrace.psf (rayopt/geometric_trace.py:
// 133-161): regridding of the per-ray OPD of a hexapolar bundle onto the n x n
// node grid (rtx_opd_regrid) and the zero-padded 2-D DFT of the pupil function
// (rtx_psf).  Included by rtx.cu; the entry points live there.
#pragma once
#include <cuda_runtime.h>

namespace rtx_wave {

// ---- regridding ------------------------------------------------------------
//
// Topology: the structured triangulation of the hexapolar launch grid (ring r
// holds 6r rays from index 1 + 3r(r-1)); triangles [6r^2, 6(r+1)^2) join ring r
// and ring r+1, 2r+1 per sector.  A node takes the value of the LOWEST-index
// triangle that contains it (barycentric coordinates >= -BARY_EPS), so nodes on
// shared edges and vertices are decided by a fixed rule and the map is
// bit-identical run to run.  All arithmetic that decides a node's triangle or
// value is unfused IEEE (the _rn intrinsics), in the operation order of
// oracle/psf_oracle.py.

constexpr unsigned NO_TRI = 0xffffffffu;
constexpr double BARY_EPS = 0x1p-40;

struct RegridArgs {
    const double* A;
    const double* P;
    long long N, ntri;
    double a_ref, px_ref, py_ref, lscale;
    int n;
    double step;  // np.mgrid[-1:1:1j*n] spacing, 2/(n-1)
    const unsigned long long* hbits;  // h as the bits of a non-negative double
};

// x, y, t of ray r: t = -(A - a_ref)/(l/scale), (x, y) = P - P[ref]
__device__ __forceinline__ bool ray_xyt(const RegridArgs& g, long long r, double& x, double& y,
                                        double& t) {
    x = __dsub_rn(g.P[3 * r], g.px_ref);
    y = __dsub_rn(g.P[3 * r + 1], g.py_ref);
    t = __ddiv_rn(-__dsub_rn(g.A[r], g.a_ref), g.lscale);
    return isfinite(x) && isfinite(y) && isfinite(t);
}

__device__ __forceinline__ long long ring_ray(long long q, long long k) {
    return q == 0 ? 0 : 1 + 3 * q * (q - 1) + k % (6 * q);
}

__device__ __forceinline__ void hex_triangle(long long tid, long long v[3]) {
    long long r = (long long)sqrt((double)tid / 6.0);
    while (6 * (r + 1) * (r + 1) <= tid) ++r;
    while (6 * r * r > tid) --r;
    long long w = tid - 6 * r * r;
    const long long j = w / (2 * r + 1);
    w -= j * (2 * r + 1);
    const long long ib = r * j, ob = (r + 1) * j;
    if (w == 2 * r) {  // the sector's closing triangle (i_r, o_r, o_{r+1})
        v[0] = ring_ray(r, ib + r);
        v[1] = ring_ray(r + 1, ob + r);
        v[2] = ring_ray(r + 1, ob + r + 1);
    } else if (w & 1) {  // (i_m, o_{m+1}, i_{m+1})
        const long long m = w >> 1;
        v[0] = ring_ray(r, ib + m);
        v[1] = ring_ray(r + 1, ob + m + 1);
        v[2] = ring_ray(r, ib + m + 1);
    } else {  // (i_m, o_m, o_{m+1})
        const long long m = w >> 1;
        v[0] = ring_ray(r, ib + m);
        v[1] = ring_ray(r + 1, ob + m);
        v[2] = ring_ray(r + 1, ob + m + 1);
    }
}

struct Tri {
    double x[3], y[3], t[3];
    double a, b, c, e, d;  // barycentric coefficients, d = twice the signed area
};

__device__ __forceinline__ bool load_tri(const RegridArgs& g, long long tid, Tri& T) {
    long long v[3];
    hex_triangle(tid, v);
    for (int k = 0; k < 3; ++k)
        if (!ray_xyt(g, v[k], T.x[k], T.y[k], T.t[k])) return false;
    T.a = __dsub_rn(T.y[1], T.y[2]);
    T.b = __dsub_rn(T.x[2], T.x[1]);
    T.c = __dsub_rn(T.y[2], T.y[0]);
    T.e = __dsub_rn(T.x[0], T.x[2]);
    T.d = __dadd_rn(__dmul_rn(T.a, T.e), __dmul_rn(T.b, __dsub_rn(T.y[0], T.y[2])));
    return T.d != 0.0 && isfinite(T.d);
}

__device__ __forceinline__ void bary(const Tri& T, double px, double py, double l[3]) {
    const double dx = __dsub_rn(px, T.x[2]), dy = __dsub_rn(py, T.y[2]);
    l[0] = __ddiv_rn(__dadd_rn(__dmul_rn(T.a, dx), __dmul_rn(T.b, dy)), T.d);
    l[1] = __ddiv_rn(__dadd_rn(__dmul_rn(T.c, dx), __dmul_rn(T.e, dy)), T.d);
    l[2] = __dsub_rn(__dsub_rn(1.0, l[0]), l[1]);
}

// node k of np.mgrid[-1:1:1j*n]*h: (k*step + -1)*h
__device__ __forceinline__ double node(long long k, double step, double h) {
    return __dmul_rn(__dadd_rn(__dmul_rn((double)k, step), -1.0), h);
}

__device__ __forceinline__ double hval(const RegridArgs& g) {
    return __longlong_as_double((long long)*g.hbits);
}

// h = max |x|, |y| over rays with finite x, y, t (geometric_trace.py:135-139)
// and the number of such rays
__global__ void regrid_bounds_kernel(RegridArgs g, unsigned long long* hbits,
                                     unsigned long long* count) {
    unsigned long long m = 0, c = 0;
    for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < g.N;
         r += (long long)gridDim.x * blockDim.x) {
        double x, y, t;
        if (ray_xyt(g, r, x, y, t)) {
            const unsigned long long b =
                (unsigned long long)__double_as_longlong(fmax(fabs(x), fabs(y)));
            m = b > m ? b : m;
            ++c;
        }
    }
    for (int o = 16; o; o >>= 1) {
        const unsigned long long mo = __shfl_xor_sync(0xffffffffu, m, o);
        m = mo > m ? mo : m;
        c += __shfl_xor_sync(0xffffffffu, c, o);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMax(hbits, m);
        atomicAdd(count, c);
    }
}

// candidate node range of [lo, hi] along one axis (one node of margin: the
// exact test below decides)
__device__ __forceinline__ void node_range(double lo, double hi, double step, double h, int n,
                                           int& k0, int& k1) {
    const double u0 = floor((lo / h + 1.0) / step) - 1.0, u1 = ceil((hi / h + 1.0) / step) + 1.0;
    k0 = (int)fmin(fmax(u0, 0.0), (double)(n - 1));  // NaN (h == 0): the whole axis
    k1 = (int)fmax(fmin(u1, (double)(n - 1)), 0.0);
}

__global__ void regrid_owner_kernel(RegridArgs g, unsigned* owner) {
    const double h = hval(g);
    for (long long tid = blockIdx.x * (long long)blockDim.x + threadIdx.x; tid < g.ntri;
         tid += (long long)gridDim.x * blockDim.x) {
        Tri T;
        if (!load_tri(g, tid, T)) continue;
        int i0, i1, j0, j1;
        node_range(fmin(fmin(T.x[0], T.x[1]), T.x[2]), fmax(fmax(T.x[0], T.x[1]), T.x[2]), g.step,
                   h, g.n, i0, i1);
        node_range(fmin(fmin(T.y[0], T.y[1]), T.y[2]), fmax(fmax(T.y[0], T.y[1]), T.y[2]), g.step,
                   h, g.n, j0, j1);
        for (int i = i0; i <= i1; ++i) {
            const double px = node(i, g.step, h);
            for (int j = j0; j <= j1; ++j) {
                double l[3];
                bary(T, px, node(j, g.step, h), l);
                if (l[0] >= -BARY_EPS && l[1] >= -BARY_EPS && l[2] >= -BARY_EPS)
                    atomicMin(&owner[(long long)i * g.n + j], (unsigned)tid);
            }
        }
    }
}

__global__ void regrid_eval_kernel(RegridArgs g, const unsigned* owner, double* map) {
    const double h = hval(g);
    const long long nn = (long long)g.n * g.n;
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < nn;
         k += (long long)gridDim.x * blockDim.x) {
        const unsigned o = owner[k];
        double v = __longlong_as_double(0x7ff8000000000000ll);  // NaN: outside every triangle
        if (o != NO_TRI) {
            Tri T;
            load_tri(g, o, T);
            double l[3];
            bary(T, node(k / g.n, g.step, h), node(k % g.n, g.step, h), l);
            v = __dadd_rn(__dadd_rn(__dmul_rn(l[0], T.t[0]), __dmul_rn(l[1], T.t[1])),
                          __dmul_rn(l[2], T.t[2]));
        }
        map[k] = v;
    }
}

// ---- PSF ---------------------------------------------------------------------
//
// psf = |DFT2(pupil, M x M)|^2 / M^2, pupil = where(finite, exp(-2 pi i o), 0)
// / sqrt(count) (geometric_trace.py:150-157), M = pad*n.  The 2-D transform is
// two batched 1-D passes over rows with a transpose between them; only the n
// non-zero input rows are transformed in the first pass.  Every 1-D DFT of
// length M is a Bluestein (chirp-z) convolution of power-of-two length
// L >= M + n - 1, computed with one shared-memory FFT kernel: in one tile when
// L <= FFT_TILE, otherwise as a four-step transform L = L1 x L2 (column pass,
// row pass, column pass) over a work buffer in HBM.

constexpr int FFT_TILE = 4096;   // complex doubles per CTA (64 KB of shared memory)
constexpr int FFT_THREADS = 512;
constexpr int FFT_L1 = 512;      // column length of the four-step split

enum : unsigned {
    F_LOAD_X = 1u,     // load chirp-modulated input rows (else the work buffer)
    F_LOAD_B = 2u,     // load the Bluestein kernel conj(chirp), wrapped
    F_FWD = 4u,        // forward FFT of the loaded data
    F_INV = 8u,        // inverse FFT of the loaded data
    F_CONV = 16u,      // after F_FWD: multiply by bhat, then inverse FFT
    F_TWIDDLE = 32u,   // four-step twiddle exp(-+2 pi i q e / L) after the transform
    F_OUT_C = 64u,     // epilogue: chirp * z / L into complex output rows
    F_OUT_ABS2 = 128u  // epilogue: |chirp * z / L|^2 * scale into real output rows
};

struct FftArgs {
    double2* work;         // L per sequence (or bhat when it is computed)
    const double2* x;      // input rows (F_LOAD_X): m_in values each
    long long x_stride;
    int m_in;
    const double2* chirp;  // exp(-pi i k^2 / M), k < M
    const double2* tw;     // exp(-2 pi i j / L), j < L
    const double2* bhat;   // FFT_L of the Bluestein kernel, in the work layout
    void* out;             // output rows (epilogues): M values each
    long long out_stride;
    double scale;
    long long nsub;        // sub-sequences in this launch
    int L, L1, L2, M;
    int Ls, logLs, C;      // transform length, log2, sub-sequences per CTA
    int col;               // 1: sub-sequence = column (stride L2), 0: row (contiguous)
    unsigned flags;
};

__device__ __forceinline__ double2 cmul(double2 a, double2 b) {
    return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}

__device__ __forceinline__ int brev(int e, int logn) {
    return logn ? (int)(__brev((unsigned)e) >> (32 - logn)) : 0;
}

// in-place radix-2 DIT over C sequences of Ls values (bit-reversed input,
// natural-order output)
__device__ void fft_stages(double2* s, const FftArgs& a, bool inv) {
    const int nb = a.C * (a.Ls >> 1);
    for (int half = 1, lg = 0; half < a.Ls; half <<= 1, ++lg) {
        const int tstride = a.L >> (lg + 1);
        for (int b = threadIdx.x; b < nb; b += blockDim.x) {
            const int c = b >> (a.logLs - 1), q = b & ((a.Ls >> 1) - 1);
            const int j = q & (half - 1);
            const int base = c * a.Ls + ((q >> lg) << (lg + 1)) + j;
            double2 w = __ldg(&a.tw[j * tstride]);
            if (inv) w.y = -w.y;
            const double2 u = s[base], v = cmul(s[base + half], w);
            s[base] = make_double2(u.x + v.x, u.y + v.y);
            s[base + half] = make_double2(u.x - v.x, u.y - v.y);
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(FFT_THREADS) fft_tile_kernel(FftArgs a) {
    extern __shared__ double2 sm[];
    const long long g0 = (long long)blockIdx.x * a.C;
    const int total = a.C * a.Ls;
    const bool cfast = a.col && a.L2 > 1;  // adjacent sub-sequences are adjacent in memory
    // element f of the tile -> (sub-sequence c, element e), its work index, its
    // natural (time or frequency) index
    auto locate = [&](int f, int& c, int& e, long long& s, long long& q, long long& widx) {
        if (cfast) {
            c = f % a.C;
            e = f / a.C;
        } else {
            e = f % a.Ls;
            c = f / a.Ls;
        }
        const long long g = g0 + c;
        if (a.col) {
            s = g / a.L2;
            q = g - s * a.L2;
            widx = s * a.L + (long long)a.L2 * e + q;
        } else {
            s = g / a.L1;
            q = g - s * a.L1;
            widx = s * a.L + (long long)a.L2 * q + e;
        }
        return g < a.nsub;
    };
    for (int f = threadIdx.x; f < total; f += blockDim.x) {
        int c, e;
        long long s, q, widx;
        double2 v = make_double2(0.0, 0.0);
        if (locate(f, c, e, s, q, widx)) {
            const long long nat = (long long)a.L2 * e + q;  // column passes
            if (a.flags & F_LOAD_X) {
                if (nat < a.m_in) v = cmul(a.x[s * a.x_stride + nat], __ldg(&a.chirp[nat]));
            } else if (a.flags & F_LOAD_B) {
                double2 w = make_double2(0.0, 0.0);
                if (nat < a.M)
                    w = __ldg(&a.chirp[nat]);
                else if (nat > a.L - a.m_in)
                    w = __ldg(&a.chirp[a.L - nat]);
                v = make_double2(w.x, -w.y);
            } else {
                v = a.work[widx];
            }
        }
        sm[c * a.Ls + brev(e, a.logLs)] = v;
    }
    __syncthreads();
    const bool inv_last = (a.flags & (F_INV | F_CONV)) != 0;
    fft_stages(sm, a, (a.flags & F_INV) != 0);
    if (a.flags & F_CONV) {
        // pointwise product with bhat, re-ordered bit-reversed for the inverse
        for (int f = threadIdx.x; f < total; f += blockDim.x) {
            const int c = f / a.Ls, e = f % a.Ls, r = brev(e, a.logLs);
            if (e > r) continue;
            const long long g = g0 + c;
            const long long q = a.col ? g % a.L2 : g % a.L1;
            const long long be = a.col ? (long long)a.L2 * e + q : (long long)a.L2 * q + e;
            const long long br = a.col ? (long long)a.L2 * r + q : (long long)a.L2 * q + r;
            const double2 ve = cmul(sm[c * a.Ls + e], __ldg(&a.bhat[be]));
            const double2 vr = cmul(sm[c * a.Ls + r], __ldg(&a.bhat[br]));
            sm[c * a.Ls + e] = vr;
            sm[c * a.Ls + r] = ve;
        }
        __syncthreads();
        fft_stages(sm, a, true);
    }
    const double invL = 1.0 / a.L;
    for (int f = threadIdx.x; f < total; f += blockDim.x) {
        int c, e;
        long long s, q, widx;
        if (!locate(f, c, e, s, q, widx)) continue;
        double2 v = sm[c * a.Ls + e];
        if (a.flags & F_TWIDDLE) {
            double2 w = __ldg(&a.tw[(q * e) % a.L]);
            if (inv_last) w.y = -w.y;
            v = cmul(v, w);
        }
        if (a.flags & (F_OUT_C | F_OUT_ABS2)) {
            const long long nat = (long long)a.L2 * e + q;
            if (nat >= a.M) continue;
            double2 X = cmul(__ldg(&a.chirp[nat]), v);
            X.x *= invL;
            X.y *= invL;
            if (a.flags & F_OUT_ABS2)
                ((double*)a.out)[s * a.out_stride + nat] = (X.x * X.x + X.y * X.y) * a.scale;
            else
                ((double2*)a.out)[s * a.out_stride + nat] = X;
        } else {
            a.work[widx] = v;
        }
    }
}

// chirp[k] = exp(-pi i k^2/M) (k < M), tw[j] = exp(-2 pi i j/L) (j < L)
__global__ void psf_tables_kernel(double2* chirp, int M, double2* tw, int L) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    double s, c;
    if (k < M) {
        const long long k2 = ((long long)k * k) % (2LL * M);
        sincospi(-(double)k2 / M, &s, &c);
        chirp[k] = make_double2(c, s);
    }
    if (k < L) {
        sincospi(-2.0 * k / L, &s, &c);
        tw[k] = make_double2(c, s);
    }
}

__global__ void finite_count_kernel(const double* o, long long nn, unsigned long long* count) {
    unsigned long long c = 0;
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < nn;
         k += (long long)gridDim.x * blockDim.x)
        c += isfinite(o[k]) ? 1 : 0;
    for (int o2 = 16; o2; o2 >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o2);
    if ((threadIdx.x & 31) == 0) atomicAdd(count, c);
}

// pupil function of the n x n map, written TRANSPOSED (gT[j][i] = g[i][j]) so
// that the row - transpose - row passes end in the natural order
__global__ void pupil_transpose_kernel(const double* o, int n, const unsigned long long* count,
                                       double2* gT) {
    __shared__ double2 tile[32][33];
    const int bj = blockIdx.x * 32, bi = blockIdx.y * 32;
    const double sq = sqrt((double)*count);
    for (int k = threadIdx.y; k < 32; k += blockDim.y) {
        const int i = bi + k, j = bj + threadIdx.x;
        if (i < n && j < n) {
            const double v = o[(long long)i * n + j];
            double2 p = make_double2(0.0, 0.0);
            if (isfinite(v)) {
                double s, c;
                sincospi(-2.0 * v, &s, &c);
                p = make_double2(c / sq, s / sq);
            }
            tile[k][threadIdx.x] = p;
        }
    }
    __syncthreads();
    for (int k = threadIdx.y; k < 32; k += blockDim.y) {
        const int j = bj + k, i = bi + threadIdx.x;
        if (i < n && j < n) gT[(long long)j * n + i] = tile[threadIdx.x][k];
    }
}

// out (cols x rows) = transpose of in (rows x cols)
__global__ void transpose_kernel(const double2* in, int rows, int cols, double2* out) {
    __shared__ double2 tile[32][33];
    const int bc = blockIdx.x * 32, br = blockIdx.y * 32;
    for (int k = threadIdx.y; k < 32; k += blockDim.y) {
        const int r = br + k, c = bc + threadIdx.x;
        if (r < rows && c < cols) tile[k][threadIdx.x] = in[(long long)r * cols + c];
    }
    __syncthreads();
    for (int k = threadIdx.y; k < 32; k += blockDim.y) {
        const int c = bc + k, r = br + threadIdx.x;
        if (r < rows && c < cols) out[(long long)c * rows + r] = tile[threadIdx.x][k];
    }
}

// ---- PSF figures (Analysis.opds, rayopt/analysis.py:319-346) -----------------
//
// All on the UNSHIFTED M x M PSF of rtx_psf.  Line sums: psf.sum(0) (per
// column) and psf.sum(1) (per row) from one read, in a fixed reduction order.
// Encircled energy: a radial histogram in the fftshifted frame (shifted index
// I = (i + M/2) % M), bin trunc(sqrt((J - c1)^2 + (I - c0)^2)) in unfused IEEE,
// accumulated in 2^-62 fixed point so that the sum is exact integer arithmetic
// and independent of the atomic order.

constexpr int LINES_THREADS = 256;
constexpr int LINES_PER_THREAD = 4;                            // columns per thread
constexpr int LINES_CW = LINES_THREADS * LINES_PER_THREAD;     // columns per tile
constexpr int LINES_RB = 128;                                  // rows per tile

// one RB x CW tile per CTA: column partials colp[band][j], row partials
// rowp[chunk][i], and per-CTA max and count of elements that are non-finite or
// outside [0, 2]
__global__ void __launch_bounds__(LINES_THREADS)
    psf_lines_tile_kernel(const double* psf, int M, double* colp, double* rowp, double* bmax,
                          unsigned long long* bbad) {
    __shared__ double wsum[LINES_RB][LINES_THREADS / 32];
    __shared__ double smax[LINES_THREADS / 32];
    __shared__ unsigned long long sbad[LINES_THREADS / 32];
    const int band = blockIdx.y, chunk = blockIdx.x;
    const int i0 = band * LINES_RB, j0 = chunk * LINES_CW;
    const int rows = min(LINES_RB, M - i0);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double col[LINES_PER_THREAD];
    for (int k = 0; k < LINES_PER_THREAD; ++k) col[k] = 0.0;
    double mx = 0.0;
    unsigned long long bad = 0;
#pragma unroll 4
    for (int r = 0; r < rows; ++r) {
        const double* row = psf + (long long)(i0 + r) * M;
        double v[LINES_PER_THREAD];
#pragma unroll
        for (int k = 0; k < LINES_PER_THREAD; ++k) {
            const int j = j0 + threadIdx.x + k * LINES_THREADS;
            v[k] = j < M ? __ldcs(row + j) : 0.0;
        }
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < LINES_PER_THREAD; ++k) {
            col[k] = __dadd_rn(col[k], v[k]);
            s = __dadd_rn(s, v[k]);
            mx = fmax(mx, v[k]);
            bad += (v[k] >= 0.0 && v[k] <= 2.0) ? 0 : 1;  // NaN fails both
        }
        for (int o = 16; o; o >>= 1) s = __dadd_rn(s, __shfl_xor_sync(0xffffffffu, s, o));
        if (lane == 0) wsum[r][warp] = s;
    }
#pragma unroll
    for (int k = 0; k < LINES_PER_THREAD; ++k) {
        const int j = j0 + threadIdx.x + k * LINES_THREADS;
        if (j < M) colp[(long long)band * M + j] = col[k];
    }
    for (int o = 16; o; o >>= 1) {
        mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        bad += __shfl_xor_sync(0xffffffffu, bad, o);
    }
    if (lane == 0) {
        smax[warp] = mx;
        sbad[warp] = bad;
    }
    __syncthreads();
    if (threadIdx.x < rows) {
        double s = 0.0;
        for (int w = 0; w < LINES_THREADS / 32; ++w) s = __dadd_rn(s, wsum[threadIdx.x][w]);
        rowp[(long long)chunk * M + i0 + threadIdx.x] = s;
    }
    if (threadIdx.x == 0) {
        for (int w = 0; w < LINES_THREADS / 32; ++w) {
            mx = fmax(mx, smax[w]);
            bad += w ? sbad[w] : 0;
        }
        const long long b = (long long)band * gridDim.x + chunk;
        bmax[b] = mx;
        bbad[b] = bad;
    }
}

// lines[j] = sum over bands of colp[band][j], lines[M + i] = sum over chunks of
// rowp[chunk][i], each in index order
__global__ void psf_lines_finish_kernel(const double* colp, const double* rowp, int M, int nband,
                                        int nchunk, double* lines) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= M) return;
    double c = 0.0, r = 0.0;
    for (int b = 0; b < nband; ++b) c = __dadd_rn(c, colp[(long long)b * M + j]);
    for (int b = 0; b < nchunk; ++b) r = __dadd_rn(r, rowp[(long long)b * M + j]);
    lines[j] = c;
    lines[M + j] = r;
}

// stats = (max over CTAs, sum of the row sums, count of bad elements); one CTA
// of LINES_THREADS threads, fixed strides and a fixed tree
__global__ void __launch_bounds__(LINES_THREADS)
    psf_stats_kernel(const double* rows, int M, const double* bmax,
                     const unsigned long long* bbad, long long nblocks, double* stats) {
    __shared__ double ssum[LINES_THREADS], smax[LINES_THREADS];
    __shared__ unsigned long long sbad[LINES_THREADS];
    double s = 0.0, mx = 0.0;
    unsigned long long bad = 0;
    for (int i = threadIdx.x; i < M; i += LINES_THREADS) s = __dadd_rn(s, rows[i]);
    for (long long b = threadIdx.x; b < nblocks; b += LINES_THREADS) {
        mx = fmax(mx, bmax[b]);
        bad += bbad[b];
    }
    ssum[threadIdx.x] = s;
    smax[threadIdx.x] = mx;
    sbad[threadIdx.x] = bad;
    __syncthreads();
    for (int h = LINES_THREADS / 2; h; h >>= 1) {
        if (threadIdx.x < h) {
            ssum[threadIdx.x] = __dadd_rn(ssum[threadIdx.x], ssum[threadIdx.x + h]);
            smax[threadIdx.x] = fmax(smax[threadIdx.x], smax[threadIdx.x + h]);
            sbad[threadIdx.x] += sbad[threadIdx.x + h];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        stats[0] = smax[0];
        stats[1] = ssum[0];
        stats[2] = (double)sbad[0];
    }
}

constexpr int EE_THREADS = 256;
constexpr int EE_T = 128;     // EE_T x EE_T shifted-frame tile per CTA
constexpr int EE_HB = 256;    // shared bins per CTA: a tile spans <= sqrt(2) EE_T + 2 bins
constexpr double EE_ONE = 0x1p62;

// the bin of shifted node (I, J): polar_sum's (j**2 + i**2)**.5, truncated
__device__ __forceinline__ long long ee_bin(int I, int J, double c0, double c1) {
    const double di = __dsub_rn((double)I, c0), dj = __dsub_rn((double)J, c1);
    return (long long)__dsqrt_rn(__dadd_rn(__dmul_rn(dj, dj), __dmul_rn(di, di)));
}

// distance from c to the nearest node of [lo, hi]
__device__ __forceinline__ double ee_near(int lo, int hi, double c) {
    return c < lo ? lo - c : (c > hi ? c - hi : 0.0);
}

__global__ void __launch_bounds__(EE_THREADS)
    psf_encircled_kernel(const double* psf, int M, double c0, double c1, long long nbins,
                         unsigned long long* bins, int* overflow) {
    __shared__ unsigned long long hist[EE_HB];
    const int I0 = blockIdx.y * EE_T, J0 = blockIdx.x * EE_T;
    const int I1 = min(I0 + EE_T, M) - 1, J1 = min(J0 + EE_T, M) - 1;
    // lowest bin of the tile, less a margin; elements outside the shared range
    // go straight to global memory
    const double di = ee_near(I0, I1, c0), dj = ee_near(J0, J1, c1);
    const long long lo = max(0LL, (long long)sqrt(dj * dj + di * di) - 2);
    for (int b = threadIdx.x; b < EE_HB; b += EE_THREADS) hist[b] = 0;
    __syncthreads();
    const int h = M / 2;
    const int J = J0 + (threadIdx.x % EE_T);
    const int j = J - h < 0 ? J - h + M : J - h;  // unshifted column
    constexpr int STEP = EE_THREADS / EE_T, U = 4;  // U rows loaded before any atomic
    if (J <= J1) {
        for (int Ib = I0 + threadIdx.x / EE_T; Ib <= I1; Ib += STEP * U) {
            double v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int I = Ib + u * STEP;
                const int i = I - h < 0 ? I - h + M : I - h;
                v[u] = I <= I1 ? __ldcs(psf + (long long)i * M + j) : 0.0;
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const unsigned long long q = __double2ull_rn(__dmul_rn(v[u], EE_ONE));
                if (!q) continue;
                const long long b = ee_bin(Ib + u * STEP, J, c0, c1);
                if (b >= nbins) {
                    atomicOr(overflow, 1);
                } else if (b >= lo && b < lo + EE_HB) {
                    atomicAdd(&hist[b - lo], q);
                } else {
                    atomicAdd(&bins[b], q);
                }
            }
        }
    }
    __syncthreads();
    for (int b = threadIdx.x; b < EE_HB; b += EE_THREADS)
        if (hist[b]) atomicAdd(&bins[lo + b], hist[b]);
}

// |X| = sqrt(|X|^2) of the first `half` of each of `nseq` rows of M values
__global__ void psf_abs_half_kernel(const double* abs2, int M, int half, int nseq, double* out) {
    const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (k >= (long long)half * nseq) return;
    const long long s = k / half, e = k - s * half;
    out[k] = sqrt(abs2[s * M + e]);
}

// real rows -> complex rows (imaginary part 0)
__global__ void real_to_complex_kernel(const double* x, long long n, double2* z) {
    const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (k < n) z[k] = make_double2(x[k], 0.0);
}

// out[a][b] = fftshift(psf)[(i0 + a) % M][(j0 + b) % M], 0 <= i0, j0 < M
__global__ void psf_window_kernel(const double* psf, int M, int i0, int j0, int w, double* out) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= w) return;
    const int h = M / 2;
    int J = j0 + b;
    J -= J >= M ? M : 0;
    const int j = J - h < 0 ? J - h + M : J - h;
    for (int a = blockIdx.y; a < w; a += gridDim.y) {
        int I = i0 + a;
        I -= I >= M ? M : 0;
        const int i = I - h < 0 ? I - h + M : I - h;
        out[(long long)a * w + b] = psf[(long long)i * M + j];
    }
}

}  // namespace rtx_wave
