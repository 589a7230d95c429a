// rtx.cu -- C ABI of the ray-trace engine (include/rtx.h): context, memory,
// the table conversion and the kernel launches.  Build:
//   nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared \
//        -Xcompiler -fPIC -o librtx.so rtx.cu
#include "../../include/rtx.h"
#include "rtx_device.cuh"
#include "rtx_psf.cuh"

#include <sched.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <cctype>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

using namespace rtx;

#define CK(call)                                \
    do {                                        \
        cudaError_t e_ = (call);                \
        if (e_ != cudaSuccess) return (int)e_;  \
    } while (0)

namespace {

constexpr int TABLE_SLOTS = 8;

struct TableSlot {
    void* host = nullptr;  // pinned
    void* dev = nullptr;
    cudaEvent_t done = nullptr;
    bool used = false;
    std::vector<unsigned char> key;  // the rtx_surface bytes + element size this slot holds
};

struct ChunkBuf {
    void* y0 = nullptr;
    void* u0 = nullptr;
    void* Y = nullptr;
    void* U = nullptr;
    void* I = nullptr;
    void* T = nullptr;
    size_t in_bytes = 0, out3_bytes = 0, out1_bytes = 0;
    cudaStream_t stream = nullptr;
};

}  // namespace

struct rtx_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t t0 = nullptr, t1 = nullptr;    // rtx_timer_*
    cudaEvent_t k0 = nullptr, k1 = nullptr;    // around the last trace launch
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> chunk_events;
    bool kernel_timed = false;
    TableSlot slots[TABLE_SLOTS];
    int next_slot = 0;
    size_t slot_bytes = 0;
    ChunkBuf chunk[2];
    double* d_moments = nullptr;
    double* d_epi = nullptr;  // rtx_trace_reduce
    // cached plan of the ray generator (rtx_aim_plan / rtx_aim_rays)
    std::vector<unsigned char> aim_key;
    std::vector<long long> aim_offsets;  // per block; empty: nothing is rejected
    long long* d_aim_offsets = nullptr;
    size_t d_aim_cap = 0;
    long long aim_total = 0, aim_M = 0;
    // small-bundle latency path (ray aiming: hundreds of 1-3 ray traces)
    void* small_host = nullptr;  // pinned: [y0|u0] in, [Y|U|I|T] out
    void* small_dev = nullptr;
    size_t small_bytes = 0;
    int64_t launches = 0;
    int max_smem_optin = 0;
    // kernel configuration (defaults = measured best, profiles/r1_sweep*.txt)
    int default_rpt = 2;      // rays per thread
    int store = 2;            // STORE_WARP / STORE_CTA
    int warps = 16;           // warps per CTA
    int nbuf = 1;             // staging buffers per CTA
    int lockstep = 1;         // CTA barrier per stored surface (STORE_WARP)
    int max_ctas_per_sm = 0;  // 0: whatever fits
    unsigned* mask = nullptr; // rtx_set_mask_output
    void* tsum = nullptr;     // rtx_set_path_sum_output
    int tsum_upto = 0;
    // rtx_numa_bind: what to restore
    bool numa_bound = false;
    cpu_set_t saved_affinity;
    bool tuned = false;       // an RTX_* environment knob overrides the heuristics
    int tune = 1;             // TraceParams::tune bits (RTX_TUNE); 1 = L2 evict_first stores
};

namespace {

template <typename T>
void convert_surface(const rtx_surface& s, DevSurf<T>& d) {
    memset(&d, 0, sizeof(d));
    for (int i = 0; i < 3; ++i) d.off[i] = (T)s.offset[i];
    for (int i = 0; i < 9; ++i) d.rot[i] = (T)s.rot[i];
    d.c = (T)s.c;
    d.k1 = (T)(1.0 + s.k);
    d.kc2 = (T)s.kc2;
    d.radius2 = (T)s.radius2;
    d.mu = (T)s.mu;
    d.muf = (T)s.muf;
    d.sgn = (T)s.sgn;
    d.mu2m1 = (T)s.mu2m1;
    d.n0 = (T)s.n0;
    d.inv_c = s.c != 0.0 ? (T)(1.0 / s.c) : (T)0;
    d.kc2k = (T)(s.k * s.c * s.c);
    for (int i = 0; i < RTX_MAX_ASPH; ++i) {
        d.asph[i] = (T)s.asph[i];
        d.dasph[i] = (T)s.dasph[i];
    }
    d.n_asph = s.n_asph;
    unsigned f = 0;
    if (s.flags & RTX_F_ROTATED) f |= DF_ROTATED;
    if (s.flags & RTX_F_ALT) f |= DF_ALT;
    if (s.c == 0.0 && s.n_asph < 0) f |= DF_FLATNORMAL;
    if (s.c != 0.0) f |= DF_CURVED;
    d.flags = f;
    // branch selection of Spheroid.intercept, elements.py:478-488
    if (s.n_asph >= 0)
        d.kind = KIND_NEWTON;
    else if (s.c == 0.0)
        d.kind = KIND_PLANE;
    else if (s.k == 0.0)
        d.kind = KIND_SPHERE;
    else
        d.kind = KIND_CONIC;
    // Interface.refract, elements.py:356,363
    if (s.mu == 1.0)
        d.refr = REFR_NONE;
    else if (s.mu == -1.0)
        d.refr = REFR_MIRROR;
    else
        d.refr = REFR_SNELL;
}

int ensure_slots(rtx_ctx* ctx, size_t bytes) {
    if (bytes <= ctx->slot_bytes) return 0;
    size_t nb = bytes < 16384 ? 16384 : bytes;
    for (auto& sl : ctx->slots) {
        if (sl.used) CK(cudaEventSynchronize(sl.done));
        if (sl.host) CK(cudaFreeHost(sl.host));
        if (sl.dev) CK(cudaFree(sl.dev));
        sl.host = sl.dev = nullptr;
        CK(cudaMallocHost(&sl.host, nb));
        CK(cudaMalloc(&sl.dev, nb));
        if (!sl.done) CK(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
        sl.used = false;
        sl.key.clear();
    }
    ctx->slot_bytes = nb;
    return 0;
}

template <typename T, bool EXACT, int RPT, int STORE, int WARPS, int NBUF>
int launch_one(rtx_ctx* ctx, const TraceParams<T>& p, cudaStream_t stream) {
    auto kern = trace_kernel<T, EXACT, RPT, STORE, WARPS, NBUF>;
    constexpr int threads = WARPS * 32;
    size_t smem = trace_smem_bytes<T, RPT>(p.S, STORE, WARPS, NBUF);
    if ((int)smem > ctx->max_smem_optin) return RTX_E_UNSUPPORTED;
    if (smem > 48 * 1024)
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem));
    if (occ < 1) occ = 1;
    if (ctx->max_ctas_per_sm > 0 && occ > ctx->max_ctas_per_sm) occ = ctx->max_ctas_per_sm;
    const long long per_cta = (long long)threads * RPT;
    TraceParams<T> q = p;  // launch-wide CTA-tile numbering over the bundles
    long long tiles = 0;
    for (int b = 0; b < q.nbatch; ++b) {
        q.item[b].tile0 = tiles;
        tiles += (q.item[b].N + per_cta - 1) / per_cta;
    }
    q.total_tiles = tiles;
    long long grid = (long long)ctx->sm_count * occ;  // persistent: one wave
    if (grid > tiles) grid = tiles;
    if (grid < 1) grid = 1;
    kern<<<(unsigned)grid, threads, smem, stream>>>(q);
    ctx->launches++;
    return (int)cudaGetLastError();
}

// the instantiated tuning space (rpt, store, warps, nbuf)
template <typename T, bool EXACT>
int launch_cfg(rtx_ctx* ctx, const TraceParams<T>& p, int rpt, int store, int warps, int nbuf,
               cudaStream_t stream) {
#define RTX_CASE(R, ST, W, NB)                                  \
    if (rpt == R && store == ST && warps == W && nbuf == NB)    \
        return launch_one<T, EXACT, R, ST, W, NB>(ctx, p, stream);
    if (store == STORE_DIRECT) return launch_one<T, EXACT, 1, STORE_DIRECT, 8, 1>(ctx, p, stream);
    RTX_CASE(1, STORE_WARP, 8, 2)
    RTX_CASE(2, STORE_WARP, 8, 2)
    RTX_CASE(2, STORE_CTA, 16, 1)
    RTX_CASE(1, STORE_CTA, 16, 1)
    RTX_CASE(2, STORE_CTA, 32, 1)
    RTX_CASE(2, STORE_CTA, 8, 1)
    RTX_CASE(2, STORE_WARP, 16, 2)
    if constexpr (sizeof(T) == 4) {  // FP32: four rays per thread (64 registers leave room)
        RTX_CASE(4, STORE_CTA, 16, 1)
        RTX_CASE(4, STORE_WARP, 16, 1)
    }
#ifdef RTX_TUNING_SPACE
    RTX_CASE(2, STORE_CTA, 8, 2)
    RTX_CASE(1, STORE_WARP, 16, 2)
    RTX_CASE(2, STORE_WARP, 8, 1)
    RTX_CASE(1, STORE_CTA, 8, 1)
    RTX_CASE(1, STORE_CTA, 8, 2)
    RTX_CASE(1, STORE_CTA, 16, 2)
    RTX_CASE(2, STORE_CTA, 16, 2)
    RTX_CASE(1, STORE_CTA, 32, 1)
    RTX_CASE(1, STORE_CTA, 32, 2)
    if constexpr (sizeof(T) == 4) {
        RTX_CASE(4, STORE_WARP, 8, 1)
        RTX_CASE(4, STORE_CTA, 8, 1)
        RTX_CASE(4, STORE_CTA, 32, 1)
    }
    RTX_CASE(2, STORE_WARP, 16, 1)
    if constexpr (sizeof(T) == 4) {
        RTX_CASE(4, STORE_WARP, 16, 2)
        RTX_CASE(4, STORE_WARP, 8, 2)
    }
#endif
#undef RTX_CASE
    return RTX_E_UNSUPPORTED;
}

template <typename T>
int launch_trace(rtx_ctx* ctx, const TraceParams<T>& p, bool exact, int rpt, int store, int warps,
                 int nbuf, cudaStream_t stream);

template <>
int launch_trace<double>(rtx_ctx* ctx, const TraceParams<double>& p, bool exact, int rpt,
                         int store, int warps, int nbuf, cudaStream_t stream) {
    if (exact) return launch_cfg<double, true>(ctx, p, rpt, store, warps, nbuf, stream);
    return launch_cfg<double, false>(ctx, p, rpt, store, warps, nbuf, stream);
}
template <>
int launch_trace<float>(rtx_ctx* ctx, const TraceParams<float>& p, bool exact, int rpt, int store,
                        int warps, int nbuf, cudaStream_t stream) {
    if (exact) return RTX_E_UNSUPPORTED;  // RTX_EXACT is FP64 only
    return launch_cfg<float, false>(ctx, p, rpt, store, warps, nbuf, stream);
}

// convert + upload the table; returns the device pointer.  The copy is
// ordered on `stream`; the pinned slot is recycled only after its copy ran.
template <typename T>
int upload_table(rtx_ctx* ctx, const rtx_surface* surf, int S, cudaStream_t stream,
                 const DevSurf<T>** out, const void* const* keep = nullptr, int nkeep = 0) {
    size_t bytes = (size_t)S * sizeof(DevSurf<T>);
    int rc = ensure_slots(ctx, bytes);
    if (rc) return rc;
    // a table that is already resident (same records, same arithmetic type) is
    // reused: repeated traces of the same lens / wavelength put no H2D copy
    // between their kernels
    const size_t raw = (size_t)S * sizeof(rtx_surface);
    const unsigned char* src = reinterpret_cast<const unsigned char*>(surf);
    for (auto& sl : ctx->slots) {
        if (sl.used && sl.key.size() == raw + 1 && sl.key[raw] == (unsigned char)sizeof(T) &&
            memcmp(sl.key.data(), src, raw) == 0) {
            *out = reinterpret_cast<const DevSurf<T>*>(sl.dev);
            return 0;
        }
    }
    // next slot in the ring that holds none of the tables the caller still
    // needs (the other bundles of a batched launch)
    int pick = ctx->next_slot;
    for (int tries = 0; tries < TABLE_SLOTS; ++tries) {
        bool busy = false;
        for (int k = 0; k < nkeep; ++k) busy = busy || keep[k] == ctx->slots[pick].dev;
        if (!busy) break;
        pick = (pick + 1) % TABLE_SLOTS;
    }
    TableSlot& sl = ctx->slots[pick];
    ctx->next_slot = (pick + 1) % TABLE_SLOTS;
    if (sl.used) CK(cudaEventSynchronize(sl.done));
    sl.used = false;
    DevSurf<T>* h = reinterpret_cast<DevSurf<T>*>(sl.host);
    for (int i = 0; i < S; ++i) convert_surface<T>(surf[i], h[i]);
    CK(cudaMemcpyAsync(sl.dev, sl.host, bytes, cudaMemcpyHostToDevice, stream));
    CK(cudaEventRecord(sl.done, stream));
    sl.key.assign(src, src + raw);
    sl.key.push_back((unsigned char)sizeof(T));
    sl.used = true;
    *out = reinterpret_cast<const DevSurf<T>*>(sl.dev);
    return 0;
}

int check_table(const rtx_surface* surf, int S) {
    if (!surf || S < 1 || S > RTX_MAX_SURFACES) return RTX_E_BADARG;
    for (int i = 0; i < S; ++i) {
        if (surf[i].n_asph > RTX_MAX_ASPH) return RTX_E_UNSUPPORTED;
        if (surf[i].n_asph < -1) return RTX_E_BADARG;
    }
    return 0;
}

template <typename T>
struct Batch {
    int n = 0;
    BatchItem<T> item[RTX_MAX_BATCH];
};

struct PeerDst {
    int n = 0;
    long long off = 0;
    void* ptr[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    void* ptr_i[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    bool has_i = false;
    bool xy = false;
};

template <typename T>
int trace_device(rtx_ctx* ctx, const rtx_surface* surf, int S, const double* rot0, long long N,
                 const void* y0, const void* u0, int clip, int keep, long long ld, void* Y,
                 void* U, void* I, void* Tt, unsigned flags, cudaStream_t stream,
                 const DevSurf<T>* table /* may be null: upload */,
                 const PeerDst* peers = nullptr, const Batch<T>* batch = nullptr) {
    if (!table) {
        int rc = upload_table<T>(ctx, surf, S, stream, &table);
        if (rc) return rc;
    }
    TraceParams<T> p;
    memset(&p, 0, sizeof(p));
    p.lockstep = 0;
    p.table = table;
    p.S = S;
    p.clip = clip ? 1 : 0;
    p.keep_last = keep == RTX_KEEP_LAST;
    p.has_rot0 = rot0 != nullptr;
    if (rot0)
        for (int i = 0; i < 9; ++i) p.rot0[i] = (T)rot0[i];
    p.N = N;
    p.ld = ld;
    p.y0 = (const T*)y0;
    p.u0 = (const T*)u0;
    p.Y = (T*)Y;
    p.U = (T*)U;
    p.I = (T*)I;
    p.Tt = (T*)Tt;
    bool peers_ok = true;
    if (peers && peers->n > 0) {
        p.npeer = peers->n;
        p.peer_off = peers->off;
        p.peer_has_i = peers->has_i ? 1 : 0;
        p.peer_xy = peers->xy ? 1 : 0;
        for (int k = 0; k < peers->n; ++k) {
            p.peer[k] = (T*)peers->ptr[k];
            p.peer_i[k] = (T*)peers->ptr_i[k];
        }
        // bulk stores need 16-byte aligned runs in every destination
        peers_ok = (peers->off * (peers->xy ? 2 : 3) * (long long)sizeof(T)) % 16 == 0 &&
                   (!peers->has_i || (peers->off * 3 * (long long)sizeof(T)) % 16 == 0);
        for (int k = 0; k < peers->n; ++k) {
            peers_ok = peers_ok && (reinterpret_cast<uintptr_t>(peers->ptr[k]) & 15u) == 0;
            peers_ok = peers_ok && (reinterpret_cast<uintptr_t>(peers->ptr_i[k]) & 15u) == 0;
        }
    }
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
    int rpt = ctx->default_rpt;
    if (flags & RTX_RPT1) rpt = 1;
    if (flags & RTX_RPT2) rpt = 2;
    int store = ctx->store, warps = ctx->warps, nbuf = ctx->nbuf;
    bool heavy = false;
    const bool explicit_rpt = (flags & (RTX_RPT1 | RTX_RPT2)) != 0;
    if (!ctx->tuned && !explicit_rpt) {
        // measured best configurations (profiles/r1_sweep8_defaults.txt,
        // r2b_sweep_newton_rewrite.txt; fractions of the measured HBM copy peak):
        //  FP64: 2 rays/thread x 16 warps, per-CTA bulk stores (24 KB runs)      0.93-0.95
        //  FP32: 4 rays/thread x 16 warps (2048-ray tiles, 24 KB runs again):
        //        half the per-thread overhead instructions of 2 rays/thread     0.92-0.94
        //  systems with >= 25 % Newton (aspheric) surfaces are bound by issue
        //  slots / the FP64 pipe, not by HBM: free-running 16-warp CTAs with
        //  per-warp stores (no lockstep barrier behind the long, divergent
        //  Newton chains) -- FP64 0.88, FP32 (4 rays per thread) 0.88
        //  (profiles/r2l_sweep_heavy_configs.txt)
        int newton = 0;
        for (int i = 0; i < S; ++i) newton += surf && surf[i].n_asph >= 0;
        // ... and so is a keep-LAST trace (one stored row: the stores are no
        // limit): free-running CTAs, 1e7 rays x 12 surfaces 0.94 -> 0.84 ms
        // (profiles/r2p_keep_last_configs.txt)
        // (a fused gather keeps the per-CTA 24 KB runs for its NVLink stores)
        heavy = newton * 4 >= S || (keep == RTX_KEEP_LAST && !(peers && peers->n > 0));
        if (sizeof(T) == 4) {
            rpt = 4;
            if (heavy) {
                store = STORE_WARP;
                warps = 16;
                nbuf = 1;
            } else {
                store = STORE_CTA;
                warps = 16;
                nbuf = 1;
            }
        } else if (heavy) {
            // free-running 16-warp CTAs with per-warp stores (fast 0.88, RTX_EXACT
            // 0.80; 8-warp CTAs: 0.855 with per-CTA stores / 0.77 exact on the
            // same box, profiles/r2l_sweep_heavy_configs.txt)
            rpt = 2;
            store = STORE_WARP;
            nbuf = 2;
            warps = 16;
        }
    }
    if (N <= 150 * 1000 && !ctx->tuned) {
        // small bundles: 256-ray warp tiles spread over all SMs (5e4 rays:
        // 0.35 vs 0.24 with 1024-ray tiles, profiles/r2n_midsize_configs.txt)
        rpt = 1;
        store = STORE_WARP;
        warps = 8;
        nbuf = 2;
    } else if (N <= 1500 * 1000 && !ctx->tuned && !explicit_rpt && !heavy && sizeof(T) == 8) {
        // mid-size FP64 bundles (what an analysis traces): 512-ray tiles, two
        // resident CTAs per SM -- twice the tiles to balance over the SMs
        // (3e5 rays 0.78 -> 0.88, 1e6 rays 0.81 -> 0.88)
        rpt = 1;
        store = STORE_CTA;
        warps = 16;
        nbuf = 1;
    } else if (N > 500 * 1000 && N <= 2500 * 1000 && !ctx->tuned && !explicit_rpt && !heavy &&
               sizeof(T) == 4) {
        // mid-size FP32 bundles: 512-ray tiles, three resident CTAs per SM
        // (1e6 rays 0.72 -> 0.92, 2e6 rays 0.81 -> 0.83)
        rpt = 2;
        store = STORE_CTA;
        warps = 8;
        nbuf = 1;
    } else if (N <= 32 * 1024) {  // (tuned contexts keep the old small-bundle rule)
        rpt = 1;
        store = STORE_WARP;
        warps = 8;
        nbuf = 2;
    } else if (explicit_rpt) {  // explicit RPT: its per-warp store kernel
        store = STORE_WARP;
        warps = 8;
        nbuf = 2;
    }
    const bool aligned = !(flags & RTX_STORE_DIRECT) && al16(Y) && al16(U) && al16(I) && al16(Tt) &&
                         peers_ok;
    // The staged paths write whole 32*rpt-ray groups: the pitch must be a
    // multiple of that, and so must the shard of a gather (into a gather buffer
    // a ragged tail would spill clamped copies of the last ray into the next
    // rank's range -- a race with that rank's own stores).
    auto fits = [&](int r) { return ld % (32 * r) == 0 && (p.npeer == 0 || N % (32 * r) == 0); };
    if (aligned && !ctx->tuned) {
        // step down to the kernel with fewer rays per thread that fits
        if (rpt == 4 && !fits(4)) {
            rpt = 2;
            if (heavy) {
                store = STORE_WARP;
                warps = 8;
                nbuf = 2;
            } else {
                store = STORE_CTA;
                warps = 32;
                nbuf = 1;
            }
        }
        if (rpt == 2 && !fits(2) && fits(1)) {
            rpt = 1;
            store = STORE_WARP;
            warps = 8;
            nbuf = 2;
        }
    }
    if (!(aligned && fits(rpt))) store = STORE_DIRECT;  // per-ray stores: exactly N rays
    if (batch && batch->n > 0) {
        p.nbatch = batch->n;
        for (int b = 0; b < batch->n; ++b) p.item[b] = batch->item[b];
    } else {
        p.nbatch = 1;
        p.item[0].table = table;
        p.item[0].y0 = p.y0;
        p.item[0].u0 = p.u0;
        p.item[0].Y = p.Y;
        p.item[0].U = p.U;
        p.item[0].I = p.I;
        p.item[0].Tt = p.Tt;
        p.item[0].N = N;
    }
    p.lockstep = heavy ? 0 : ctx->lockstep;
    p.tune = ctx->tune;
    p.mask = ctx->mask;
    p.tsum = (T*)ctx->tsum;
    p.tsum_upto = ctx->tsum_upto < 0 ? S - 1 : ctx->tsum_upto;
    return launch_trace<T>(ctx, p, (flags & RTX_EXACT) != 0, rpt, store, warps, nbuf, stream);
}

int ensure_chunk(rtx_ctx* ctx, ChunkBuf& cb, size_t in_bytes, size_t out3, size_t out1) {
    if (!cb.stream) CK(cudaStreamCreateWithFlags(&cb.stream, cudaStreamNonBlocking));
    if (in_bytes > cb.in_bytes) {
        if (cb.y0) CK(cudaFree(cb.y0));
        if (cb.u0) CK(cudaFree(cb.u0));
        cb.y0 = cb.u0 = nullptr;
        cb.in_bytes = 0;
        CK(cudaMalloc(&cb.y0, in_bytes));
        CK(cudaMalloc(&cb.u0, in_bytes));
        cb.in_bytes = in_bytes;
    }
    if (out3 > cb.out3_bytes) {
        if (cb.Y) CK(cudaFree(cb.Y));
        if (cb.U) CK(cudaFree(cb.U));
        if (cb.I) CK(cudaFree(cb.I));
        cb.Y = cb.U = cb.I = nullptr;
        cb.out3_bytes = 0;
        CK(cudaMalloc(&cb.Y, out3));
        CK(cudaMalloc(&cb.U, out3));
        CK(cudaMalloc(&cb.I, out3));
        cb.out3_bytes = out3;
    }
    if (out1 > cb.out1_bytes) {
        if (cb.T) CK(cudaFree(cb.T));
        cb.T = nullptr;
        cb.out1_bytes = 0;
        CK(cudaMalloc(&cb.T, out1));
        cb.out1_bytes = out1;
    }
    return 0;
}

void free_chunk(ChunkBuf& cb) {
    if (cb.y0) cudaFree(cb.y0);
    if (cb.u0) cudaFree(cb.u0);
    if (cb.Y) cudaFree(cb.Y);
    if (cb.U) cudaFree(cb.U);
    if (cb.I) cudaFree(cb.I);
    if (cb.T) cudaFree(cb.T);
    if (cb.stream) cudaStreamDestroy(cb.stream);
    cb = ChunkBuf();
}

void clear_chunk_events(rtx_ctx* ctx) {
    for (auto& pr : ctx->chunk_events) {
        cudaEventDestroy(pr.first);
        cudaEventDestroy(pr.second);
    }
    ctx->chunk_events.clear();
}

constexpr size_t SMALL_PATH_BYTES = 4u << 20;
constexpr size_t ZERO_COPY_BYTES = 16u << 10;  // rays + results of a zero-copy small trace

// Latency path for small bundles (aim_chief / aim_marginal issue hundreds of
// 1-3 ray traces, rayopt/system.py:507-555): one pinned bounce buffer, ONE
// H2D of [y0|u0], the kernel with ld = N (per-thread stores, reference
// layout on the device), ONE D2H of [Y|U|I|T], one synchronisation.
template <typename T>
int trace_host_small(rtx_ctx* ctx, const rtx_surface* surf, int S, const double* rot0,
                     long long N, const void* y0, const void* u0, int clip, int keep, void* Y,
                     void* U, void* I, void* Tt, unsigned flags, size_t in_bytes,
                     size_t out_bytes) {
    const int rows = keep == RTX_KEEP_LAST ? 1 : S;
    const size_t need = in_bytes + out_bytes;
    if (need > ctx->small_bytes) {
        if (ctx->small_host) CK(cudaFreeHost(ctx->small_host));
        if (ctx->small_dev) CK(cudaFree(ctx->small_dev));
        ctx->small_host = ctx->small_dev = nullptr;
        ctx->small_bytes = 0;
        size_t nb = need < (256u << 10) ? (256u << 10) : need;
        CK(cudaMallocHost(&ctx->small_host, nb));
        CK(cudaMalloc(&ctx->small_dev, nb));
        ctx->small_bytes = nb;
    }
    char* h = (char*)ctx->small_host;
    const size_t v3 = (size_t)N * 3 * sizeof(T), r3 = (size_t)rows * v3, r1 = r3 / 3;
    memcpy(h, y0, v3);
    memcpy(h + v3, u0, v3);
    // A handful of rays (ray aiming: 1-3): ZERO-COPY.  Page-locked memory is
    // mapped into the device's address space (UVA), so the kernel reads the
    // launch rays and writes its results straight over PCIe -- launch + one
    // synchronisation, no copy-engine round trips (2 x ~8 us).  Beyond
    // ZERO_COPY_BYTES the DMA engines win: one H2D, the kernel, one D2H.
    const bool zero_copy = need <= ZERO_COPY_BYTES && !getenv("RTX_NO_ZERO_COPY");
    char* d = zero_copy ? h : (char*)ctx->small_dev;
    if (!zero_copy) CK(cudaMemcpyAsync(d, h, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    char* dY = d + in_bytes;
    char *dU = dY + r3, *dI = dU + r3, *dT = dI + r3;
    int rc = trace_device<T>(ctx, surf, S, rot0, N, d, d + v3, clip, keep, N, Y ? dY : nullptr,
                             U ? dU : nullptr, I ? dI : nullptr, Tt ? dT : nullptr,
                             flags | RTX_STORE_DIRECT, ctx->stream, nullptr);
    if (rc) return rc;
    if (!zero_copy)
        CK(cudaMemcpyAsync(h + in_bytes, dY, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const char* o = h + in_bytes;
    if (Y) memcpy(Y, o, r3);
    if (U) memcpy(U, o + r3, r3);
    if (I) memcpy(I, o + 2 * r3, r3);
    if (Tt) memcpy(Tt, o + 3 * r3, r1);
    clear_chunk_events(ctx);
    ctx->kernel_timed = false;
    return 0;
}

template <typename T>
int trace_host(rtx_ctx* ctx, const rtx_surface* surf, int S, const double* rot0, long long N,
               const void* y0, const void* u0, int clip, int keep, void* Y, void* U, void* I,
               void* Tt, unsigned flags) {
    const int rows = keep == RTX_KEEP_LAST ? 1 : S;
    {
        const size_t in_b = (size_t)N * 6 * sizeof(T);
        const size_t out_b = (size_t)rows * N * 10 * sizeof(T);
        // (an explicit store-path / RPT request goes through the general path)
        if (in_b + out_b <= SMALL_PATH_BYTES && !(flags & (RTX_RPT1 | RTX_RPT2 | RTX_STORE_DIRECT)))
            return trace_host_small<T>(ctx, surf, S, rot0, N, y0, u0, clip, keep, Y, U, I, Tt,
                                       flags, in_b, out_b);
    }
    // chunk: ~256 MB of results, whole 128-ray groups
    long long per_ray = (long long)rows * 10 * sizeof(T) + 6 * sizeof(T);
    long long C = (256ll << 20) / per_ray;
    C = (C / 128) * 128;  // whole 128-ray groups: every staged kernel applies
    if (C < 4096) C = 4096;
    if (C > N) C = ((N + 127) / 128) * 128;
    const size_t in_bytes = (size_t)C * 3 * sizeof(T);
    const size_t out3 = (size_t)rows * C * 3 * sizeof(T);
    const size_t out1 = (size_t)rows * C * sizeof(T);
    for (int b = 0; b < 2; ++b) {
        int rc = ensure_chunk(ctx, ctx->chunk[b], in_bytes, out3, out1);
        if (rc) return rc;
    }
    // the table is uploaded once on the main stream; chunk streams wait for it
    const DevSurf<T>* table = nullptr;
    int rc = upload_table<T>(ctx, surf, S, ctx->stream, &table);
    if (rc) return rc;
    struct EventGuard {  // destroyed on every return path
        cudaEvent_t e = nullptr;
        ~EventGuard() {
            if (e) cudaEventDestroy(e);
        }
    } guard;
    CK(cudaEventCreateWithFlags(&guard.e, cudaEventDisableTiming));
    cudaEvent_t table_ready = guard.e;
    CK(cudaEventRecord(table_ready, ctx->stream));
    clear_chunk_events(ctx);
    int nchunk = 0;
    for (long long c0 = 0; c0 < N; c0 += C, ++nchunk) {
        ChunkBuf& cb = ctx->chunk[nchunk & 1];
        const long long n = (N - c0 < C) ? (N - c0) : C;
        if (nchunk < 2) CK(cudaStreamWaitEvent(cb.stream, table_ready, 0));
        CK(cudaMemcpyAsync(cb.y0, (const T*)y0 + c0 * 3, (size_t)n * 3 * sizeof(T),
                           cudaMemcpyHostToDevice, cb.stream));
        CK(cudaMemcpyAsync(cb.u0, (const T*)u0 + c0 * 3, (size_t)n * 3 * sizeof(T),
                           cudaMemcpyHostToDevice, cb.stream));
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        CK(cudaEventCreate(&e0));
        if (cudaError_t er = cudaEventCreate(&e1)) {
            cudaEventDestroy(e0);
            return (int)er;
        }
        ctx->chunk_events.emplace_back(e0, e1);  // owned by ctx from here on
        CK(cudaEventRecord(e0, cb.stream));
        rc = trace_device<T>(ctx, surf, S, rot0, n, cb.y0, cb.u0, clip, keep, C, Y ? cb.Y : nullptr,
                             U ? cb.U : nullptr, I ? cb.I : nullptr, Tt ? cb.T : nullptr, flags,
                             cb.stream, table);
        if (rc) {
            for (int b = 0; b < 2; ++b) cudaStreamSynchronize(ctx->chunk[b].stream);
            return rc;
        }
        CK(cudaEventRecord(e1, cb.stream));
        const size_t w3 = (size_t)n * 3 * sizeof(T), w1 = (size_t)n * sizeof(T);
        const size_t sp3 = (size_t)C * 3 * sizeof(T), sp1 = (size_t)C * sizeof(T);
        const size_t dp3 = (size_t)N * 3 * sizeof(T), dp1 = (size_t)N * sizeof(T);
        if (Y)
            CK(cudaMemcpy2DAsync((T*)Y + c0 * 3, dp3, cb.Y, sp3, w3, rows, cudaMemcpyDeviceToHost,
                                 cb.stream));
        if (U)
            CK(cudaMemcpy2DAsync((T*)U + c0 * 3, dp3, cb.U, sp3, w3, rows, cudaMemcpyDeviceToHost,
                                 cb.stream));
        if (I)
            CK(cudaMemcpy2DAsync((T*)I + c0 * 3, dp3, cb.I, sp3, w3, rows, cudaMemcpyDeviceToHost,
                                 cb.stream));
        if (Tt)
            CK(cudaMemcpy2DAsync((T*)Tt + c0, dp1, cb.T, sp1, w1, rows, cudaMemcpyDeviceToHost,
                                 cb.stream));
    }
    for (int b = 0; b < 2; ++b) CK(cudaStreamSynchronize(ctx->chunk[b].stream));
    ctx->kernel_timed = false;
    return 0;
}

}  // namespace

// =========================================================================
extern "C" {

int rtx_abi_version(void) { return RTX_ABI_VERSION; }

size_t rtx_sizeof_surface(void) { return sizeof(rtx_surface); }
size_t rtx_sizeof_aim(void) { return sizeof(rtx_aim); }
size_t rtx_sizeof_opd(void) { return sizeof(rtx_opd); }

int rtx_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

const char* rtx_strerror(int code) {
    switch (code) {
        case RTX_OK: return "ok";
        case RTX_E_BADARG: return "rtx: bad argument";
        case RTX_E_UNSUPPORTED: return "rtx: unsupported (too many aspheric coefficients / surfaces, or RTX_EXACT with FP32)";
        case RTX_E_NOMEM: return "rtx: out of memory";
        default: break;
    }
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "rtx: unknown error";
}

int rtx_surface_finalize(rtx_surface* surf, int n, const double* radius) {
    if (!surf || n < 0) return RTX_E_BADARG;
    for (int i = 0; i < n; ++i) {
        rtx_surface& s = surf[i];
        s.kc2 = (1.0 + s.k) * (s.c * s.c);
        if (radius) s.radius2 = radius[i] * radius[i];
        s.muf = fabs(s.mu);
        s.sgn = s.mu > 0 ? 1.0 : (s.mu < 0 ? -1.0 : 0.0);
        s.mu2m1 = s.mu * s.mu - 1.0;
        for (int j = 0; j < RTX_MAX_ASPH; ++j)
            s.dasph[j] = (j < s.n_asph) ? (double)(2 * (j + 1)) * s.asph[j] : 0.0;
    }
    return 0;
}

int rtx_init(int device, rtx_ctx** out) {
    if (!out) return RTX_E_BADARG;
    int n = 0;
    CK(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) return RTX_E_BADARG;
    CK(cudaSetDevice(device));
    rtx_ctx* ctx = new (std::nothrow) rtx_ctx();
    if (!ctx) return RTX_E_NOMEM;
    ctx->device = device;
    auto setup = [&]() -> int {
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, device));
        ctx->sm_count = prop.multiProcessorCount;
        ctx->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
        CK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        CK(cudaEventCreate(&ctx->t0));
        CK(cudaEventCreate(&ctx->t1));
        CK(cudaEventCreate(&ctx->k0));
        CK(cudaEventCreate(&ctx->k1));
        CK(cudaMalloc((void**)&ctx->d_moments, 8 * sizeof(double)));
        return 0;
    };
    if (int rc = setup()) {
        rtx_free(ctx);
        return rc;
    }
    // tuning knobs (experiments; the defaults above are the measured best)
    if (const char* e = getenv("RTX_RPT")) {
        int v = atoi(e);
        if (v == 1 || v == 2 || v == 4) ctx->default_rpt = v;
        ctx->tuned = true;
    }
    if (const char* e = getenv("RTX_WARPS")) {
        int v = atoi(e);
        if (v == 8 || v == 16 || v == 32) ctx->warps = v;
    }
    if (const char* e = getenv("RTX_STORE")) {
        int v = atoi(e);
        if (v == 1 || v == 2) ctx->store = v;
    }
    if (const char* e = getenv("RTX_NBUF")) {
        int v = atoi(e);
        if (v == 1 || v == 2) ctx->nbuf = v;
    }
    if (getenv("RTX_WARPS") || getenv("RTX_STORE") || getenv("RTX_NBUF")) ctx->tuned = true;
    if (const char* e = getenv("RTX_LOCK")) ctx->lockstep = atoi(e) != 0;
    if (const char* e = getenv("RTX_MAX_CTAS")) ctx->max_ctas_per_sm = atoi(e);
    if (const char* e = getenv("RTX_TUNE")) ctx->tune = atoi(e);
    *out = ctx;
    return 0;
}

int rtx_free(rtx_ctx* ctx) {
    if (!ctx) return 0;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    clear_chunk_events(ctx);
    for (auto& sl : ctx->slots) {
        if (sl.host) cudaFreeHost(sl.host);
        if (sl.dev) cudaFree(sl.dev);
        if (sl.done) cudaEventDestroy(sl.done);
    }
    free_chunk(ctx->chunk[0]);
    free_chunk(ctx->chunk[1]);
    if (ctx->d_moments) cudaFree(ctx->d_moments);
    if (ctx->d_epi) cudaFree(ctx->d_epi);
    if (ctx->d_aim_offsets) cudaFree(ctx->d_aim_offsets);
    if (ctx->small_host) cudaFreeHost(ctx->small_host);
    if (ctx->small_dev) cudaFree(ctx->small_dev);
    if (ctx->t0) cudaEventDestroy(ctx->t0);
    if (ctx->t1) cudaEventDestroy(ctx->t1);
    if (ctx->k0) cudaEventDestroy(ctx->k0);
    if (ctx->k1) cudaEventDestroy(ctx->k1);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return 0;
}

int rtx_sync(rtx_ctx* ctx) {
    if (!ctx) return RTX_E_BADARG;
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int rtx_device_info(rtx_ctx* ctx, int* sm_count, size_t* free_bytes, size_t* total_bytes,
                    char* name, int name_len) {
    if (!ctx) return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    if (sm_count) *sm_count = ctx->sm_count;
    size_t f = 0, t = 0;
    CK(cudaMemGetInfo(&f, &t));
    if (free_bytes) *free_bytes = f;
    if (total_bytes) *total_bytes = t;
    if (name && name_len > 0) {
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, ctx->device));
        snprintf(name, (size_t)name_len, "%s", prop.name);
    }
    return 0;
}

int rtx_malloc(rtx_ctx* ctx, size_t bytes, void** dptr) {
    if (!ctx || !dptr) return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMalloc(dptr, bytes ? bytes : 16));
    return 0;
}
int rtx_free_device(rtx_ctx* ctx, void* dptr) {
    if (!ctx) return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaFree(dptr));
    return 0;
}
int rtx_host_alloc(rtx_ctx* ctx, size_t bytes, void** hptr) {
    if (!ctx || !hptr) return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMallocHost(hptr, bytes ? bytes : 16));
    return 0;
}
int rtx_host_free(rtx_ctx* ctx, void* hptr) {
    (void)ctx;  // page-locked memory may outlive the context that allocated it
    CK(cudaFreeHost(hptr));
    return 0;
}

int rtx_numa_bind(rtx_ctx* ctx, int enable, int* node_out) {
    if (!ctx) return RTX_E_BADARG;
    if (node_out) *node_out = -1;
    if (!enable) {
        if (ctx->numa_bound) {
            sched_setaffinity(0, sizeof(cpu_set_t), &ctx->saved_affinity);
            syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0);
            ctx->numa_bound = false;
        }
        return 0;
    }
    char bus[32] = {0};
    CK(cudaDeviceGetPCIBusId(bus, (int)sizeof(bus), ctx->device));
    for (char* c = bus; *c; ++c) *c = (char)tolower((unsigned char)*c);
    char path[128];
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bus);
    int node = -1;
    if (FILE* f = fopen(path, "r")) {
        if (fscanf(f, "%d", &node) != 1) node = -1;
        fclose(f);
    }
    if (node < 0 || node >= 1024) return 0;  // not reported: leave everything alone
    snprintf(path, sizeof(path), "/sys/devices/system/node/node%d/cpulist", node);
    cpu_set_t set;
    CPU_ZERO(&set);
    int ncpu = 0;
    if (FILE* f = fopen(path, "r")) {  // "0-31,64-95"
        int a = 0, b = 0;
        while (fscanf(f, "%d", &a) == 1) {
            b = a;
            int ch = fgetc(f);
            if (ch == '-') {
                if (fscanf(f, "%d", &b) != 1) b = a;
                ch = fgetc(f);
            }
            for (int c = a; c <= b && c < CPU_SETSIZE; ++c) {
                CPU_SET(c, &set);
                ++ncpu;
            }
            if (ch != ',') break;
        }
        fclose(f);
    }
    if (ncpu == 0) return 0;
    if (!ctx->numa_bound) sched_getaffinity(0, sizeof(cpu_set_t), &ctx->saved_affinity);
    // only CPUs this process may use anyway (cgroup / taskset limits)
    cpu_set_t both;
    CPU_AND(&both, &set, &ctx->saved_affinity);
    if (CPU_COUNT(&both) > 0) sched_setaffinity(0, sizeof(cpu_set_t), &both);
    unsigned long mask[16] = {0};
    mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
    syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, 8 * sizeof(mask));
    ctx->numa_bound = true;
    if (node_out) *node_out = node;
    return 0;
}
int rtx_memcpy_h2d(rtx_ctx* ctx, void* dst, const void* src, size_t bytes) {
    if (!ctx) return RTX_E_BADARG;
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}
int rtx_memcpy_d2h(rtx_ctx* ctx, void* dst, const void* src, size_t bytes) {
    if (!ctx) return RTX_E_BADARG;
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return 0;
}
int rtx_memcpy_d2d(rtx_ctx* ctx, void* dst, const void* src, size_t bytes) {
    if (!ctx) return RTX_E_BADARG;
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    return 0;
}
int rtx_memcpy2d_d2h(rtx_ctx* ctx, void* dst, size_t dpitch, const void* src, size_t spitch,
                     size_t width, size_t height) {
    if (!ctx) return RTX_E_BADARG;
    CK(cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, height, cudaMemcpyDeviceToHost,
                         ctx->stream));
    return 0;
}
int rtx_memset(rtx_ctx* ctx, void* dptr, int value, size_t bytes) {
    if (!ctx) return RTX_E_BADARG;
    CK(cudaMemsetAsync(dptr, value, bytes, ctx->stream));
    return 0;
}

int rtx_timer_start(rtx_ctx* ctx) {
    if (!ctx) return RTX_E_BADARG;
    CK(cudaEventRecord(ctx->t0, ctx->stream));
    return 0;
}
int rtx_timer_stop(rtx_ctx* ctx, float* ms) {
    if (!ctx || !ms) return RTX_E_BADARG;
    CK(cudaEventRecord(ctx->t1, ctx->stream));
    CK(cudaEventSynchronize(ctx->t1));
    CK(cudaEventElapsedTime(ms, ctx->t0, ctx->t1));
    return 0;
}
int rtx_last_kernel_ms(rtx_ctx* ctx, float* ms) {
    if (!ctx || !ms) return RTX_E_BADARG;
    if (ctx->kernel_timed) {
        CK(cudaEventSynchronize(ctx->k1));
        CK(cudaEventElapsedTime(ms, ctx->k0, ctx->k1));
        return 0;
    }
    float tot = 0.f;
    for (auto& pr : ctx->chunk_events) {
        float t = 0.f;
        CK(cudaEventSynchronize(pr.second));
        CK(cudaEventElapsedTime(&t, pr.first, pr.second));
        tot += t;
    }
    *ms = tot;
    return 0;
}
int64_t rtx_launch_count(rtx_ctx* ctx) { return ctx ? ctx->launches : 0; }

int rtx_trace(rtx_ctx* ctx, const rtx_surface* surf, int S, const double* rot0, int dtype,
              int64_t N, const void* y0, const void* u0, int clip, int keep, int64_t ld, void* Y,
              void* U, void* I, void* T, unsigned flags) {
    if (!ctx) return RTX_E_BADARG;
    int rc = check_table(surf, S);
    if (rc) return rc;
    if (N < 0 || ld < N || !y0 || !u0) return RTX_E_BADARG;
    if (keep != RTX_KEEP_ALL && keep != RTX_KEEP_LAST) return RTX_E_BADARG;
    if (dtype != RTX_F64 && dtype != RTX_F32) return RTX_E_BADARG;
    if (N == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    CK(cudaEventRecord(ctx->k0, ctx->stream));
    if (dtype == RTX_F64)
        rc = trace_device<double>(ctx, surf, S, rot0, N, y0, u0, clip, keep, ld, Y, U, I, T, flags,
                                  ctx->stream, nullptr);
    else
        rc = trace_device<float>(ctx, surf, S, rot0, N, y0, u0, clip, keep, ld, Y, U, I, T, flags,
                                 ctx->stream, nullptr);
    if (rc) return rc;
    CK(cudaEventRecord(ctx->k1, ctx->stream));
    ctx->kernel_timed = true;
    return 0;
}

}  // extern "C"

namespace {
template <typename T>
int trace_batch(rtx_ctx* ctx, int nb, const rtx_surface* const* surf, int S, const double* rot0,
                const int64_t* N, const void* const* y0, const void* const* u0, int clip, int keep,
                long long ld, void* const* Y, void* const* U, void* const* I, void* const* Tt,
                unsigned flags) {
    Batch<T> bt;
    const void* tabs[RTX_MAX_BATCH];
    long long nmax = 0;
    for (int b = 0; b < nb; ++b) {
        const DevSurf<T>* tab = nullptr;
        int rc = upload_table<T>(ctx, surf[b], S, ctx->stream, &tab, tabs, bt.n);
        if (rc) return rc;
        tabs[bt.n] = tab;
        BatchItem<T>& it = bt.item[bt.n++];
        it.table = tab;
        it.y0 = (const T*)y0[b];
        it.u0 = (const T*)u0[b];
        it.Y = Y ? (T*)Y[b] : nullptr;
        it.U = U ? (T*)U[b] : nullptr;
        it.I = I ? (T*)I[b] : nullptr;
        it.Tt = Tt ? (T*)Tt[b] : nullptr;
        it.N = N[b];
        it.tile0 = 0;
        if (N[b] > nmax) nmax = N[b];
        // every bundle must satisfy the alignment the bulk-store path needs
        for (void* q : {(void*)it.Y, (void*)it.U, (void*)it.I, (void*)it.Tt})
            if (reinterpret_cast<uintptr_t>(q) & 15u) flags |= RTX_STORE_DIRECT;
    }
    // kernel configuration from the first bundle (same lens), N of the largest
    return trace_device<T>(ctx, surf[0], S, rot0, nmax, y0[0], u0[0], clip, keep, ld,
                           Y ? Y[0] : nullptr, U ? U[0] : nullptr, I ? I[0] : nullptr,
                           Tt ? Tt[0] : nullptr, flags, ctx->stream, bt.item[0].table, nullptr, &bt);
}
}  // namespace

extern "C" {

int rtx_trace_batch(rtx_ctx* ctx, int nb, const rtx_surface* const* surf, int S,
                    const double* rot0, int dtype, const int64_t* N, const void* const* y0,
                    const void* const* u0, int clip, int keep, int64_t ld, void* const* Y,
                    void* const* U, void* const* I, void* const* T, unsigned flags) {
    if (!ctx || nb < 1 || nb > RTX_MAX_BATCH || !surf || !N || !y0 || !u0) return RTX_E_BADARG;
    if (keep != RTX_KEEP_ALL && keep != RTX_KEEP_LAST) return RTX_E_BADARG;
    if (dtype != RTX_F64 && dtype != RTX_F32) return RTX_E_BADARG;
    for (int b = 0; b < nb; ++b) {
        int rc = check_table(surf[b], S);
        if (rc) return rc;
        if (N[b] < 1 || ld < N[b] || !y0[b] || !u0[b]) return RTX_E_BADARG;
    }
    CK(cudaSetDevice(ctx->device));
    unsigned* saved_mask = ctx->mask;  // per-ray side outputs are single-bundle features
    void* saved_tsum = ctx->tsum;
    ctx->mask = nullptr;
    ctx->tsum = nullptr;
    CK(cudaEventRecord(ctx->k0, ctx->stream));
    int rc = dtype == RTX_F64
                 ? trace_batch<double>(ctx, nb, surf, S, rot0, N, y0, u0, clip, keep, ld, Y, U, I,
                                       T, flags)
                 : trace_batch<float>(ctx, nb, surf, S, rot0, N, y0, u0, clip, keep, ld, Y, U, I, T,
                                      flags);
    ctx->mask = saved_mask;
    ctx->tsum = saved_tsum;
    if (rc) return rc;
    CK(cudaEventRecord(ctx->k1, ctx->stream));
    ctx->kernel_timed = true;
    return 0;
}

}  // extern "C"

namespace {
constexpr size_t BATCH_HOST_BYTES = 64u << 20;

template <typename T>
int trace_batch_host(rtx_ctx* ctx, int nb, const rtx_surface* const* surf, int S,
                     const double* rot0, const int64_t* N, const void* const* y0,
                     const void* const* u0, int clip, int keep, void* const* Y, void* const* U,
                     void* const* I, void* const* Tt, unsigned flags) {
    const int rows = keep == RTX_KEEP_LAST ? 1 : S;
    long long nmax = 0, nsum = 0;
    for (int b = 0; b < nb; ++b) {
        nmax = N[b] > nmax ? N[b] : nmax;
        nsum += N[b];
    }
    const long long ld = (nmax + 31) / 32 * 32;  // one pitch for all bundles: whole 32-ray groups
    std::vector<size_t> in_off((size_t)nb);
    size_t o = 0;
    for (int b = 0; b < nb; ++b) {  // [y0|u0] of every bundle, 16-byte aligned
        in_off[(size_t)b] = o;
        o += ((size_t)N[b] * 6 * sizeof(T) + 15) & ~size_t(15);
    }
    (void)nsum;
    const size_t per3 = (size_t)rows * ld * 3 * sizeof(T), per1 = (size_t)rows * ld * sizeof(T);
    const size_t per_bundle = (Y ? per3 : 0) + (U ? per3 : 0) + (I ? per3 : 0) + (Tt ? per1 : 0);
    const size_t in_pad = (o + 255) & ~size_t(255);
    const size_t need = in_pad + per_bundle * nb;
    if (need > BATCH_HOST_BYTES) {  // large bundles: one by one through the chunked pipeline
        for (int b = 0; b < nb; ++b) {
            if (N[b] == 0) continue;
            int rc = trace_host<T>(ctx, surf[b], S, rot0, N[b], y0[b], u0[b], clip, keep,
                                   Y ? Y[b] : nullptr, U ? U[b] : nullptr, I ? I[b] : nullptr,
                                   Tt ? Tt[b] : nullptr, flags);
            if (rc) return rc;
        }
        return 0;
    }
    if (need > ctx->small_bytes) {
        if (ctx->small_host) CK(cudaFreeHost(ctx->small_host));
        if (ctx->small_dev) CK(cudaFree(ctx->small_dev));
        ctx->small_host = ctx->small_dev = nullptr;
        ctx->small_bytes = 0;
        const size_t cap = need < (256u << 10) ? (256u << 10) : need;
        CK(cudaMallocHost(&ctx->small_host, cap));
        CK(cudaMalloc(&ctx->small_dev, cap));
        ctx->small_bytes = cap;
    }
    char* h = (char*)ctx->small_host;
    char* d = (char*)ctx->small_dev;
    for (int b = 0; b < nb; ++b) {
        const size_t v3 = (size_t)N[b] * 3 * sizeof(T);
        if (!v3) continue;
        memcpy(h + in_off[(size_t)b], y0[b], v3);
        memcpy(h + in_off[(size_t)b] + v3, u0[b], v3);
    }
    CK(cudaMemcpyAsync(d, h, o, cudaMemcpyHostToDevice, ctx->stream));
    for (int g0 = 0; g0 < nb; g0 += RTX_MAX_BATCH) {
        const int g = nb - g0 < RTX_MAX_BATCH ? nb - g0 : RTX_MAX_BATCH;
        const rtx_surface* gs[RTX_MAX_BATCH];
        int64_t gn[RTX_MAX_BATCH];
        const void *gy0[RTX_MAX_BATCH], *gu0[RTX_MAX_BATCH];
        void *gY[RTX_MAX_BATCH], *gU[RTX_MAX_BATCH], *gI[RTX_MAX_BATCH], *gT[RTX_MAX_BATCH];
        int m = 0;
        for (int k = 0; k < g; ++k) {
            const int b = g0 + k;
            if (N[b] == 0) continue;
            char* ob = d + in_pad + per_bundle * b;
            gs[m] = surf[b];
            gn[m] = N[b];
            gy0[m] = d + in_off[(size_t)b];
            gu0[m] = d + in_off[(size_t)b] + (size_t)N[b] * 3 * sizeof(T);
            gY[m] = Y ? ob : nullptr;
            ob += Y ? per3 : 0;
            gU[m] = U ? ob : nullptr;
            ob += U ? per3 : 0;
            gI[m] = I ? ob : nullptr;
            ob += I ? per3 : 0;
            gT[m] = Tt ? ob : nullptr;
            ++m;
        }
        if (m == 0) continue;
        int rc = trace_batch<T>(ctx, m, gs, S, rot0, gn, gy0, gu0, clip, keep, ld, Y ? gY : nullptr,
                                U ? gU : nullptr, I ? gI : nullptr, Tt ? gT : nullptr, flags);
        if (rc) return rc;
    }
    CK(cudaMemcpyAsync(h + in_pad, d + in_pad, per_bundle * nb, cudaMemcpyDeviceToHost,
                       ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int b = 0; b < nb; ++b) {  // (rows, ld, k) on the device -> (rows, N, k) of the caller
        const char* ob = h + in_pad + per_bundle * b;
        auto unpack = [&](void* dst, int k) {
            if (!dst) return;
            const size_t w = (size_t)N[b] * k * sizeof(T), pitch = (size_t)ld * k * sizeof(T);
            for (int r = 0; r < rows; ++r) memcpy((char*)dst + r * w, ob + r * pitch, w);
            ob += (size_t)rows * pitch;
        };
        unpack(Y ? Y[b] : nullptr, 3);
        unpack(U ? U[b] : nullptr, 3);
        unpack(I ? I[b] : nullptr, 3);
        unpack(Tt ? Tt[b] : nullptr, 1);
    }
    clear_chunk_events(ctx);
    ctx->kernel_timed = false;
    return 0;
}
}  // namespace

extern "C" {

int rtx_trace_batch_host(rtx_ctx* ctx, int nb, const rtx_surface* const* surf, int S,
                         const double* rot0, int dtype, const int64_t* N, const void* const* y0,
                         const void* const* u0, int clip, int keep, void* const* Y,
                         void* const* U, void* const* I, void* const* T, unsigned flags) {
    if (!ctx || nb < 1 || !surf || !N || !y0 || !u0) return RTX_E_BADARG;
    if (keep != RTX_KEEP_ALL && keep != RTX_KEEP_LAST) return RTX_E_BADARG;
    if (dtype != RTX_F64 && dtype != RTX_F32) return RTX_E_BADARG;
    for (int b = 0; b < nb; ++b) {
        int rc = check_table(surf[b], S);
        if (rc) return rc;
        if (N[b] < 0 || (N[b] > 0 && (!y0[b] || !u0[b]))) return RTX_E_BADARG;
    }
    CK(cudaSetDevice(ctx->device));
    unsigned* saved_mask = ctx->mask;
    void* saved_tsum = ctx->tsum;
    ctx->mask = nullptr;
    ctx->tsum = nullptr;
    int rc = dtype == RTX_F64
                 ? trace_batch_host<double>(ctx, nb, surf, S, rot0, N, y0, u0, clip, keep, Y, U, I,
                                            T, flags)
                 : trace_batch_host<float>(ctx, nb, surf, S, rot0, N, y0, u0, clip, keep, Y, U, I,
                                           T, flags);
    ctx->mask = saved_mask;
    ctx->tsum = saved_tsum;
    return rc;
}

int rtx_trace_host(rtx_ctx* ctx, const rtx_surface* surf, int S, const double* rot0, int dtype,
                   int64_t N, const void* y0, const void* u0, int clip, int keep, void* Y, void* U,
                   void* I, void* T, unsigned flags) {
    if (!ctx) return RTX_E_BADARG;
    int rc = check_table(surf, S);
    if (rc) return rc;
    if (N < 0 || !y0 || !u0) return RTX_E_BADARG;
    if (keep != RTX_KEEP_ALL && keep != RTX_KEEP_LAST) return RTX_E_BADARG;
    if (dtype != RTX_F64 && dtype != RTX_F32) return RTX_E_BADARG;
    if (N == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    unsigned* saved = ctx->mask;  // mask / path sum belong to device-buffer traces
    void* saved_tsum = ctx->tsum;
    ctx->mask = nullptr;
    ctx->tsum = nullptr;
    if (dtype == RTX_F64)
        rc = trace_host<double>(ctx, surf, S, rot0, N, y0, u0, clip, keep, Y, U, I, T, flags);
    else
        rc = trace_host<float>(ctx, surf, S, rot0, N, y0, u0, clip, keep, Y, U, I, T, flags);
    ctx->mask = saved;
    ctx->tsum = saved_tsum;
    return rc;
}

int rtx_set_mask_output(rtx_ctx* ctx, uint32_t* dmask) {
    if (!ctx) return RTX_E_BADARG;
    ctx->mask = dmask;
    return 0;
}

int rtx_set_path_sum_output(rtx_ctx* ctx, void* dsum, int upto) {
    if (!ctx) return RTX_E_BADARG;
    ctx->tsum = dsum;
    ctx->tsum_upto = upto;
    return 0;
}

int rtx_ipc_export(rtx_ctx* ctx, void* dptr, unsigned char* handle) {
    if (!ctx || !dptr || !handle) return RTX_E_BADARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == RTX_IPC_HANDLE_BYTES, "ipc handle size");
    CK(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, dptr));
    memcpy(handle, &h, sizeof(h));
    return 0;
}
int rtx_ipc_open(rtx_ctx* ctx, const unsigned char* handle, void** dptr) {
    if (!ctx || !dptr || !handle) return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    CK(cudaIpcOpenMemHandle(dptr, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}
int rtx_ipc_close(rtx_ctx* ctx, void* dptr) {
    if (!ctx) return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaIpcCloseMemHandle(dptr));
    return 0;
}

int rtx_trace_gather(rtx_ctx* ctx, const rtx_surface* surf, int S, const double* rot0, int dtype,
                     int64_t N, const void* y0, const void* u0, int clip, int npeers,
                     void* const* dst, void* const* dst_i, int64_t dst_offset, unsigned flags) {
    if (!ctx) return RTX_E_BADARG;
    int rc = check_table(surf, S);
    if (rc) return rc;
    if (N < 0 || !y0 || !u0 || npeers < 1 || npeers > 8 || !dst || dst_offset < 0)
        return RTX_E_BADARG;
    if (dtype != RTX_F64 && dtype != RTX_F32) return RTX_E_BADARG;
    if (N == 0) return 0;
    PeerDst pd;
    pd.n = npeers;
    pd.off = dst_offset;
    pd.has_i = dst_i != nullptr;
    pd.xy = (flags & RTX_GATHER_XY) != 0;
    for (int k = 0; k < npeers; ++k) {
        if (!dst[k] || (dst_i && !dst_i[k])) return RTX_E_BADARG;
        pd.ptr[k] = dst[k];
        if (dst_i) pd.ptr_i[k] = dst_i[k];
    }
    CK(cudaSetDevice(ctx->device));
    CK(cudaEventRecord(ctx->k0, ctx->stream));
    const long long ld = ((N + 127) / 128) * 128;  // only the gather destinations are written
    if (dtype == RTX_F64)
        rc = trace_device<double>(ctx, surf, S, rot0, N, y0, u0, clip, RTX_KEEP_LAST, ld, nullptr,
                                  nullptr, nullptr, nullptr, flags, ctx->stream, nullptr, &pd);
    else
        rc = trace_device<float>(ctx, surf, S, rot0, N, y0, u0, clip, RTX_KEEP_LAST, ld, nullptr,
                                 nullptr, nullptr, nullptr, flags, ctx->stream, nullptr, &pd);
    if (rc) return rc;
    CK(cudaEventRecord(ctx->k1, ctx->stream));
    ctx->kernel_timed = true;
    return 0;
}

int rtx_selftest_math(rtx_ctx* ctx, int64_t n, const double* a, const double* b, double* out) {
    if (!ctx || n < 1 || !a || !b || !out) return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    struct Bufs {  // freed on every return path
        double *a = nullptr, *b = nullptr, *o = nullptr;
        ~Bufs() {
            cudaFree(a);
            cudaFree(b);
            cudaFree(o);
        }
    } d;
    CK(cudaMalloc((void**)&d.a, n * sizeof(double)));
    CK(cudaMalloc((void**)&d.b, n * sizeof(double)));
    CK(cudaMalloc((void**)&d.o, 6 * n * sizeof(double)));
    CK(cudaMemcpyAsync(d.a, a, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d.b, b, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    selftest_math_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(d.a, d.b, d.o, n);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, d.o, 6 * n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int rtx_moments(rtx_ctx* ctx, int dtype, int64_t N, const void* y, const void* w,
                const double* center, double* m) {
    if (!ctx || !y || !m || N < 0) return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    const double cx = center ? center[0] : 0.0, cy = center ? center[1] : 0.0;
    CK(cudaMemsetAsync(ctx->d_moments, 0, 8 * sizeof(double), ctx->stream));
    if (N > 0) {
        long long blocks = (N + 255) / 256;
        long long cap = (long long)ctx->sm_count * 8;
        if (blocks > cap) blocks = cap;
        if (dtype == RTX_F64)
            moments_kernel<double><<<(unsigned)blocks, 256, 0, ctx->stream>>>(
                (const double*)y, (const double*)w, N, cx, cy, ctx->d_moments);
        else if (dtype == RTX_F32)
            moments_kernel<float><<<(unsigned)blocks, 256, 0, ctx->stream>>>(
                (const float*)y, (const float*)w, N, cx, cy, ctx->d_moments);
        else
            return RTX_E_BADARG;
        ctx->launches++;
        CK(cudaGetLastError());
    }
    CK(cudaMemcpyAsync(m, ctx->d_moments, 8 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

}  // extern "C"

namespace {
template <typename T, int MODE>
int launch_epi(rtx_ctx* ctx, const rtx_surface* surf, int S, const double* rot0, long long N,
               const void* y0, const void* u0, int clip, unsigned flags, EpiParams<T>& p) {
    const DevSurf<T>* table = nullptr;
    int rc = upload_table<T>(ctx, surf, S, ctx->stream, &table);
    if (rc) return rc;
    p.table = table;
    p.S = S;
    p.clip = clip ? 1 : 0;
    p.has_rot0 = rot0 != nullptr;
    if (rot0)
        for (int i = 0; i < 9; ++i) p.rot0[i] = (T)rot0[i];
    p.N = N;
    p.y0 = (const T*)y0;
    p.u0 = (const T*)u0;
    const bool exact = (flags & RTX_EXACT) != 0;
    if (exact && sizeof(T) == 4) return RTX_E_UNSUPPORTED;
    constexpr int RPT = 2, threads = 256;
    size_t smem = (((size_t)S * sizeof(DevSurf<T>) + 127) & ~size_t(127)) + 16;
    if ((int)smem > ctx->max_smem_optin) return RTX_E_UNSUPPORTED;
    auto go = [&](auto kern) -> int {
        if (smem > 48 * 1024)
            CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int occ = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem));
        if (occ < 1) occ = 1;
        const long long tiles = (N + threads * RPT - 1) / (threads * RPT);
        long long grid = (long long)ctx->sm_count * occ;
        if (grid > tiles) grid = tiles;
        if (grid < 1) grid = 1;
        kern<<<(unsigned)grid, threads, smem, ctx->stream>>>(p);
        ctx->launches++;
        return (int)cudaGetLastError();
    };
    if constexpr (sizeof(T) == 8) {
        if (exact) return go(epi_kernel<T, true, RPT, MODE>);
    }
    return go(epi_kernel<T, false, RPT, MODE>);
}
}  // namespace

extern "C" {

int rtx_trace_reduce(rtx_ctx* ctx, const rtx_surface* surf, int S, const double* rot0, int dtype,
                     int64_t N, const void* y0, const void* u0, int clip, const void* w,
                     const double* center, double* m, unsigned flags) {
    if (!ctx || !m) return RTX_E_BADARG;
    int rc = check_table(surf, S);
    if (rc) return rc;
    if (N < 0 || !y0 || !u0) return RTX_E_BADARG;
    if (dtype != RTX_F64 && dtype != RTX_F32) return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    if (!ctx->d_epi) CK(cudaMalloc((void**)&ctx->d_epi, RTX_NMOMENTS * sizeof(double)));
    CK(cudaMemsetAsync(ctx->d_epi, 0, RTX_NMOMENTS * sizeof(double), ctx->stream));
    if (N > 0) {
        CK(cudaEventRecord(ctx->k0, ctx->stream));
        if (dtype == RTX_F64) {
            EpiParams<double> p;
            memset(&p, 0, sizeof(p));
            p.w = (const double*)w;
            for (int k = 0; k < 2; ++k) {
                p.cy[k] = center ? center[k] : 0.0;
                p.cu[k] = center ? center[2 + k] : 0.0;
            }
            p.out = ctx->d_epi;
            rc = launch_epi<double, EPI_REDUCE>(ctx, surf, S, rot0, N, y0, u0, clip, flags, p);
        } else {
            EpiParams<float> p;
            memset(&p, 0, sizeof(p));
            p.w = (const float*)w;
            for (int k = 0; k < 2; ++k) {
                p.cy[k] = center ? center[k] : 0.0;
                p.cu[k] = center ? center[2 + k] : 0.0;
            }
            p.out = ctx->d_epi;
            rc = launch_epi<float, EPI_REDUCE>(ctx, surf, S, rot0, N, y0, u0, clip, flags, p);
        }
        if (rc) return rc;
        CK(cudaEventRecord(ctx->k1, ctx->stream));
        ctx->kernel_timed = true;
    }
    CK(cudaMemcpyAsync(m, ctx->d_epi, RTX_NMOMENTS * sizeof(double), cudaMemcpyDeviceToHost,
                       ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int rtx_trace_opd(rtx_ctx* ctx, const rtx_surface* surf, int S, const double* rot0, int dtype,
                  int64_t N, const void* y0, const void* u0, int clip, const rtx_opd* opd, void* A,
                  void* P, unsigned flags) {
    if (!ctx || !opd || !A || !P) return RTX_E_BADARG;
    int rc = check_table(surf, S);
    if (rc) return rc;
    if (N < 0 || !y0 || !u0 || opd->radius == 0.0) return RTX_E_BADARG;
    if (dtype != RTX_F64 && dtype != RTX_F32) return RTX_E_BADARG;
    if (N == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    auto fill = [&](auto& p) {
        memset(&p, 0, sizeof(p));
        p.infinite = opd->infinite;
        for (int k = 0; k < 3; ++k) {
            p.y0r[k] = opd->y0_ref[k];
            p.u0r[k] = opd->u0_ref[k];
            p.d[k] = opd->d[k];
        }
        for (int k = 0; k < 9; ++k) p.M[k] = opd->M[k];
        p.n0 = opd->n0;
        p.n_after = opd->n_after;
        p.radius = opd->radius;
    };
    CK(cudaEventRecord(ctx->k0, ctx->stream));
    if (dtype == RTX_F64) {
        EpiParams<double> p;
        fill(p);
        p.A = (double*)A;
        p.P = (double*)P;
        rc = launch_epi<double, EPI_OPD>(ctx, surf, S, rot0, N, y0, u0, clip, flags, p);
    } else {
        EpiParams<float> p;
        fill(p);
        p.A = (float*)A;
        p.P = (float*)P;
        rc = launch_epi<float, EPI_OPD>(ctx, surf, S, rot0, N, y0, u0, clip, flags, p);
    }
    if (rc) return rc;
    CK(cudaEventRecord(ctx->k1, ctx->stream));
    ctx->kernel_timed = true;
    return 0;
}

int rtx_aim_infinite(rtx_ctx* ctx, int dtype, int64_t N, const void* yp, int hex_rings,
                     const double* frame, double pmax, void* y0, void* u0) {
    if (!ctx || !frame || !y0 || !u0 || N < 0) return RTX_E_BADARG;
    if (!yp && (hex_rings < 0 || N != 1 + 3ll * hex_rings * (hex_rings + 1))) return RTX_E_BADARG;
    if (N == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    long long blocks = (N + 255) / 256;
    long long cap = (long long)ctx->sm_count * 16;
    if (blocks > cap) blocks = cap;
    const double* f = frame;
    if (dtype == RTX_F64)
        aim_infinite_kernel<double><<<(unsigned)blocks, 256, 0, ctx->stream>>>(
            (const double*)yp, hex_rings, N, pmax, f[0], f[1], f[2], f[3], f[4], f[5], f[6], f[7],
            f[8], f[9], f[10], f[11], (double*)y0, (double*)u0);
    else if (dtype == RTX_F32)
        aim_infinite_kernel<float><<<(unsigned)blocks, 256, 0, ctx->stream>>>(
            (const float*)yp, hex_rings, N, pmax, f[0], f[1], f[2], f[3], f[4], f[5], f[6], f[7],
            f[8], f[9], f[10], f[11], (float*)y0, (float*)u0);
    else
        return RTX_E_BADARG;
    ctx->launches++;
    return (int)cudaGetLastError();
}

int rtx_aim_finite(rtx_ctx* ctx, int dtype, int64_t N, const void* yp, int hex_rings,
                   const double* frame, double am, double z, void* y0, void* u0) {
    if (!ctx || !frame || !y0 || !u0 || N < 0) return RTX_E_BADARG;
    if (!yp && (hex_rings < 0 || N != 1 + 3ll * hex_rings * (hex_rings + 1))) return RTX_E_BADARG;
    if (N == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    long long blocks = (N + 255) / 256;
    long long cap = (long long)ctx->sm_count * 16;
    if (blocks > cap) blocks = cap;
    const double* f = frame;
    if (dtype == RTX_F64)
        aim_finite_kernel<double><<<(unsigned)blocks, 256, 0, ctx->stream>>>(
            (const double*)yp, hex_rings, N, am, z, f[0], f[1], f[2], f[3], f[4], f[5], f[6], f[7],
            f[8], f[9], f[10], f[11], (double*)y0, (double*)u0);
    else if (dtype == RTX_F32)
        aim_finite_kernel<float><<<(unsigned)blocks, 256, 0, ctx->stream>>>(
            (const float*)yp, hex_rings, N, am, z, f[0], f[1], f[2], f[3], f[4], f[5], f[6], f[7],
            f[8], f[9], f[10], f[11], (float*)y0, (float*)u0);
    else
        return RTX_E_BADARG;
    ctx->launches++;
    return (int)cudaGetLastError();
}

}  // extern "C"

namespace {
int aim_to_dev(const rtx_aim* a, long long n_given, AimDev& d) {
    memset(&d, 0, sizeof(d));
    d.conjugate = a->conjugate;
    d.grid = a->grid;
    d.filter = a->filter;
    d.curved = a->curved && a->conjugate == 0;
    d.n = a->n;
    d.seed = a->seed;
    memcpy(d.seg, a->seg, sizeof(d.seg));
    d.seg_m[0] = a->seg_m[0];
    d.seg_m[1] = a->seg_m[1];
    memcpy(d.frame, a->frame, sizeof(d.frame));
    d.pmax = a->pmax;
    d.z = a->z;
    for (int k = 0; k < 2; ++k) {
        d.fc[k] = a->fc[k];
        d.fd2[k] = a->fd2[k];
    }
    if (d.curved) {
        if (a->surface.n_asph > RTX_MAX_ASPH) return RTX_E_UNSUPPORTED;
        convert_surface<double>(a->surface, d.surf);
    }
    switch (a->grid) {
        case GRID_GIVEN: d.M = n_given; break;
        case GRID_HEXAPOLAR: d.M = 1 + 3 * a->n * (a->n + 1); break;
        case GRID_SQUARE:
        case GRID_TRIANGULAR:
            if (a->n < 2) return RTX_E_BADARG;
            d.M = 1 + a->n * a->n;
            break;
        case GRID_RANDOM: d.M = 1 + a->n; break;
        case GRID_LINES: d.M = a->seg_m[0] + a->seg_m[1]; break;
        default: return RTX_E_BADARG;
    }
    if (a->n < 0 || d.M < 0 || a->seg_m[0] < 0 || a->seg_m[1] < 0) return RTX_E_BADARG;
    if (a->conjugate != 0 && a->conjugate != 1) return RTX_E_BADARG;
    return 0;
}

// counting pass + prefix sum, cached per (spec, n_given, yp)
int aim_plan(rtx_ctx* ctx, const rtx_aim* spec, long long n_given, const void* yp, AimDev& d) {
    int rc = aim_to_dev(spec, n_given, d);
    if (rc) return rc;
    if (spec->grid == GRID_GIVEN && n_given > 0 && !yp) return RTX_E_BADARG;
    std::vector<unsigned char> key(sizeof(rtx_aim) + sizeof(long long) + sizeof(void*));
    memcpy(key.data(), spec, sizeof(rtx_aim));
    memcpy(key.data() + sizeof(rtx_aim), &n_given, sizeof(long long));
    memcpy(key.data() + sizeof(rtx_aim) + sizeof(long long), &yp, sizeof(void*));
    const bool rejects = spec->filter || spec->grid == GRID_SQUARE || spec->grid == GRID_TRIANGULAR;
    // (a GIVEN grid may have changed behind the same pointer: always recount it)
    if (key == ctx->aim_key && !(rejects && spec->grid == GRID_GIVEN)) return 0;
    ctx->aim_key.clear();
    ctx->aim_offsets.clear();
    ctx->aim_M = d.M;
    ctx->aim_total = d.M;
    if (rejects && d.M > 0) {
        const long long nb = (d.M + AIM_BLOCK - 1) / AIM_BLOCK;
        if ((size_t)(nb + 1) * sizeof(long long) > ctx->d_aim_cap) {
            if (ctx->d_aim_offsets) CK(cudaFree(ctx->d_aim_offsets));
            ctx->d_aim_offsets = nullptr;
            ctx->d_aim_cap = 0;
            CK(cudaMalloc((void**)&ctx->d_aim_offsets, (size_t)(nb + 1) * sizeof(long long)));
            ctx->d_aim_cap = (size_t)(nb + 1) * sizeof(long long);
        }
        int* d_counts = reinterpret_cast<int*>(ctx->d_aim_offsets);  // reused before the offsets
        long long grid = nb < (long long)ctx->sm_count * 8 ? nb : (long long)ctx->sm_count * 8;
        aim_count_kernel<<<(unsigned)grid, 256, 0, ctx->stream>>>(d, (const double*)yp, d_counts, nb);
        ctx->launches++;
        CK(cudaGetLastError());
        std::vector<int> counts((size_t)nb);
        CK(cudaMemcpyAsync(counts.data(), d_counts, (size_t)nb * sizeof(int), cudaMemcpyDeviceToHost,
                           ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->aim_offsets.resize((size_t)nb + 1);
        long long acc = 0;
        for (long long b = 0; b < nb; ++b) {
            ctx->aim_offsets[(size_t)b] = acc;
            acc += counts[(size_t)b];
        }
        ctx->aim_offsets[(size_t)nb] = acc;
        ctx->aim_total = acc;
        CK(cudaMemcpyAsync(ctx->d_aim_offsets, ctx->aim_offsets.data(),
                           (size_t)(nb + 1) * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    ctx->aim_key = key;
    return 0;
}
}  // namespace

extern "C" {

int rtx_aim_plan(rtx_ctx* ctx, const rtx_aim* spec, int64_t n_given, const void* yp,
                 int64_t* n_rays) {
    if (!ctx || !spec || !n_rays || n_given < 0) return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    AimDev d;
    int rc = aim_plan(ctx, spec, n_given, yp, d);
    if (rc) return rc;
    *n_rays = ctx->aim_total;
    return 0;
}

int rtx_aim_rays(rtx_ctx* ctx, const rtx_aim* spec, int64_t n_given, const void* yp, int dtype,
                 int64_t first, int64_t count, void* y0, void* u0, void* yp_out) {
    if (!ctx || !spec || !y0 || !u0 || n_given < 0 || first < 0 || count < 0) return RTX_E_BADARG;
    if (dtype != RTX_F64 && dtype != RTX_F32) return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    AimDev d;
    int rc = aim_plan(ctx, spec, n_given, yp, d);
    if (rc) return rc;
    if (first + count > ctx->aim_total) return RTX_E_BADARG;
    if (count == 0) return 0;
    long long b0, b1;
    const long long* d_off = nullptr;
    if (ctx->aim_offsets.empty()) {
        b0 = first / AIM_BLOCK;
        b1 = (first + count + AIM_BLOCK - 1) / AIM_BLOCK;
    } else {
        const auto& off = ctx->aim_offsets;  // off[b] = rank of block b's first kept ray
        const long long nb = (long long)off.size() - 1;
        long long lo = 0, hi = nb;  // last block with off[b] <= first
        while (lo + 1 < hi) {
            const long long mid = (lo + hi) / 2;
            if (off[(size_t)mid] <= first) lo = mid; else hi = mid;
        }
        b0 = lo;
        b1 = b0;
        while (b1 < nb && off[(size_t)b1] < first + count) ++b1;
        d_off = ctx->d_aim_offsets;
    }
    long long grid = b1 - b0;
    const long long cap = (long long)ctx->sm_count * 8;
    if (grid > cap) grid = cap;
    if (grid < 1) grid = 1;
    if (dtype == RTX_F64)
        aim_rays_kernel<double><<<(unsigned)grid, 256, 0, ctx->stream>>>(
            d, (const double*)yp, d_off, b0, b1, first, count, (double*)y0, (double*)u0,
            (double*)yp_out);
    else
        aim_rays_kernel<float><<<(unsigned)grid, 256, 0, ctx->stream>>>(
            d, (const double*)yp, d_off, b0, b1, first, count, (float*)y0, (float*)u0,
            (double*)yp_out);
    ctx->launches++;
    return (int)cudaGetLastError();
}

int rtx_focus_moments(rtx_ctx* ctx, int dtype, int64_t N, const void* y, const void* inc,
                      const void* w, const double* center, double* m) {
    if (!ctx || !y || !inc || !m || N < 0) return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    double c[4] = {0, 0, 0, 0};
    if (center)
        for (int k = 0; k < 4; ++k) c[k] = center[k];
    CK(cudaMemsetAsync(ctx->d_moments, 0, 8 * sizeof(double), ctx->stream));
    if (N > 0) {
        long long blocks = (N + 255) / 256;
        long long cap = (long long)ctx->sm_count * 8;
        if (blocks > cap) blocks = cap;
        if (dtype == RTX_F64)
            focus_moments_kernel<double><<<(unsigned)blocks, 256, 0, ctx->stream>>>(
                (const double*)y, (const double*)inc, (const double*)w, N, c[0], c[1], c[2], c[3],
                ctx->d_moments);
        else if (dtype == RTX_F32)
            focus_moments_kernel<float><<<(unsigned)blocks, 256, 0, ctx->stream>>>(
                (const float*)y, (const float*)inc, (const float*)w, N, c[0], c[1], c[2], c[3],
                ctx->d_moments);
        else
            return RTX_E_BADARG;
        ctx->launches++;
        CK(cudaGetLastError());
    }
    CK(cudaMemcpyAsync(m, ctx->d_moments, 8 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

}  // extern "C"

// ---- wavefront: OPD regridding and PSF (rtx_psf.cuh) ------------------------
namespace {

// stream-ordered scratch, released on every return path
struct Scratch {
    cudaStream_t stream;
    std::vector<void*> ptrs;
    explicit Scratch(cudaStream_t s) : stream(s) {}
    ~Scratch() {
        for (void* p : ptrs) cudaFreeAsync(p, stream);
    }
    template <typename T>
    int get(T** p, size_t count) {
        *p = nullptr;
        cudaError_t e = cudaMallocAsync((void**)p, count * sizeof(T), stream);
        if (e != cudaSuccess) return (int)e;
        ptrs.push_back(*p);
        return 0;
    }
};

int grid_for(rtx_ctx* ctx, long long work, int threads) {
    long long b = (work + threads - 1) / threads, cap = (long long)ctx->sm_count * 16;
    return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

int launch_fft(rtx_ctx* ctx, rtx_wave::FftArgs a, int col, long long nseq, unsigned flags) {
    a.col = col;
    a.flags = flags;
    a.Ls = col ? a.L1 : a.L2;
    a.logLs = 0;
    while ((1 << a.logLs) < a.Ls) ++a.logLs;
    a.C = rtx_wave::FFT_TILE / a.Ls;
    a.nsub = nseq * (col ? a.L2 : a.L1);
    const long long blocks = (a.nsub + a.C - 1) / a.C;
    rtx_wave::fft_tile_kernel<<<(unsigned)blocks, rtx_wave::FFT_THREADS,
                               rtx_wave::FFT_TILE * sizeof(double2), ctx->stream>>>(a);
    ctx->launches++;
    return (int)cudaGetLastError();
}

// one batch of nseq Bluestein DFTs of length M: rows of x (m_in values, stride
// x_stride) -> rows of out (stride out_stride), epilogue `epi`
int bluestein_rows(rtx_ctx* ctx, rtx_wave::FftArgs a, double2* work, long long work_seqs,
                   const double2* x, long long nseq, void* out, unsigned epi) {
    using namespace rtx_wave;
    a.x = x;
    if (a.L2 == 1) {  // the whole convolution in one tile
        a.out = out;
        return launch_fft(ctx, a, 1, nseq, F_LOAD_X | F_FWD | F_CONV | epi);
    }
    const size_t osz = (epi & F_OUT_ABS2) ? sizeof(double) : sizeof(double2);
    for (long long s0 = 0; s0 < nseq; s0 += work_seqs) {
        const long long cnt = nseq - s0 < work_seqs ? nseq - s0 : work_seqs;
        a.x = x + s0 * a.x_stride;
        a.work = work;
        a.out = (char*)out + (size_t)s0 * a.out_stride * osz;
        int rc = launch_fft(ctx, a, 1, cnt, F_LOAD_X | F_FWD | F_TWIDDLE);
        if (!rc) rc = launch_fft(ctx, a, 0, cnt, F_FWD | F_CONV | F_TWIDDLE);
        if (!rc) rc = launch_fft(ctx, a, 1, cnt, F_INV | epi);
        if (rc) return rc;
    }
    return 0;
}

// length-M DFTs of rows of m_in values as Bluestein convolutions: L, the
// four-step split and the lengths in `a` (zeroed first)
int bluestein_plan(long long M, long long m_in, rtx_wave::FftArgs& a) {
    using namespace rtx_wave;
    long long L = 1;
    while (L < M + m_in - 1) L <<= 1;
    if (L < 2) L = 2;
    memset(&a, 0, sizeof(a));
    a.L = (int)L;
    a.L1 = L <= FFT_TILE ? (int)L : FFT_L1;
    a.L2 = (int)(L / a.L1);
    if (a.L2 > FFT_TILE || M > (1LL << 30) / 2) return RTX_E_UNSUPPORTED;
    a.M = (int)M;
    a.m_in = (int)m_in;
    return 0;
}

// sequences the four-step work buffer holds (up to 1 GB); 0 in one tile
long long bluestein_work_seqs(const rtx_wave::FftArgs& a) {
    if (a.L2 == 1) return 0;
    const long long s = (1LL << 30) / ((long long)a.L * 16);
    return s > 0 ? s : 1;
}

// the chirp and twiddle tables and FFT_L of the Bluestein kernel, in the
// layout the convolution reads, into scratch of `sc`; enqueued on the stream
int bluestein_tables(rtx_ctx* ctx, Scratch& sc, rtx_wave::FftArgs& a) {
    using namespace rtx_wave;
    CK(cudaFuncSetAttribute(fft_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            FFT_TILE * (int)sizeof(double2)));
    double2 *chirp = nullptr, *tw = nullptr, *bhat = nullptr;
    int rc = sc.get(&chirp, (size_t)a.M);
    if (!rc) rc = sc.get(&tw, (size_t)a.L);
    if (!rc) rc = sc.get(&bhat, (size_t)a.L);
    if (rc) return rc;
    a.chirp = chirp;
    a.tw = tw;
    a.bhat = bhat;
    psf_tables_kernel<<<(unsigned)((a.L > a.M ? a.L : a.M) + 255) / 256, 256, 0, ctx->stream>>>(
        chirp, a.M, tw, a.L);
    ctx->launches++;
    CK(cudaGetLastError());
    FftArgs b = a;
    b.work = bhat;
    if (a.L2 == 1) return launch_fft(ctx, b, 1, 1, F_LOAD_B | F_FWD);
    rc = launch_fft(ctx, b, 1, 1, F_LOAD_B | F_FWD | F_TWIDDLE);
    if (!rc) rc = launch_fft(ctx, b, 0, 1, F_FWD);
    return rc;
}

}  // namespace

extern "C" {

int rtx_opd_regrid(rtx_ctx* ctx, int64_t N, const double* A, const double* P, double a_ref,
                   const double* p_ref, double lscale, int rings, int64_t n, double* map,
                   double* h, int64_t* n_finite) {
    if (!ctx || !A || !P || !p_ref || !map || rings < 1 || n < 1 || n > 46340 || lscale == 0.0)
        return RTX_E_BADARG;
    if (N != 1 + 3LL * rings * (rings + 1)) return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    Scratch sc(ctx->stream);
    unsigned long long* d_red = nullptr;  // [h bits, finite count]
    unsigned* owner = nullptr;
    int rc = sc.get(&d_red, 2);
    if (!rc) rc = sc.get(&owner, (size_t)(n * n));
    if (rc) return rc;
    CK(cudaMemsetAsync(d_red, 0, 2 * sizeof(unsigned long long), ctx->stream));
    CK(cudaMemsetAsync(owner, 0xff, (size_t)(n * n) * sizeof(unsigned), ctx->stream));
    rtx_wave::RegridArgs g;
    g.A = A;
    g.P = P;
    g.N = N;
    g.ntri = 6LL * rings * rings;
    g.a_ref = a_ref;
    g.px_ref = p_ref[0];
    g.py_ref = p_ref[1];
    g.lscale = lscale;
    g.n = (int)n;
    g.step = n > 1 ? 2.0 / (double)(n - 1) : 1.0;  // numpy's mgrid
    g.hbits = d_red;
    CK(cudaEventRecord(ctx->k0, ctx->stream));
    rtx_wave::regrid_bounds_kernel<<<grid_for(ctx, N, 256), 256, 0, ctx->stream>>>(g, d_red,
                                                                                 d_red + 1);
    rtx_wave::regrid_owner_kernel<<<grid_for(ctx, g.ntri, 128), 128, 0, ctx->stream>>>(g, owner);
    rtx_wave::regrid_eval_kernel<<<grid_for(ctx, n * n, 256), 256, 0, ctx->stream>>>(g, owner,
                                                                                   map);
    ctx->launches += 3;
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->k1, ctx->stream));
    ctx->kernel_timed = true;
    unsigned long long red[2];
    CK(cudaMemcpyAsync(red, d_red, sizeof(red), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (h) memcpy(h, &red[0], sizeof(double));
    if (n_finite) *n_finite = (int64_t)red[1];
    return 0;
}

int rtx_psf(rtx_ctx* ctx, int64_t n, const double* map, int pad, double* psf) {
    using namespace rtx_wave;
    if (!ctx || !map || !psf || n < 1 || pad < 1) return RTX_E_BADARG;
    const long long M = (long long)pad * n;
    FftArgs a;
    int rc = bluestein_plan(M, n, a);
    if (rc) return rc;
    a.x_stride = n;
    a.out_stride = M;
    CK(cudaSetDevice(ctx->device));
    Scratch sc(ctx->stream);
    unsigned long long* d_count = nullptr;
    double2 *gT = nullptr, *rows = nullptr, *rowsT = nullptr, *work = nullptr;
    const long long work_seqs = bluestein_work_seqs(a);
    rc = sc.get(&d_count, 1);
    if (!rc) rc = sc.get(&gT, (size_t)(n * n));
    if (!rc) rc = sc.get(&rows, (size_t)(n * M));
    if (!rc) rc = sc.get(&rowsT, (size_t)(n * M));
    if (!rc && work_seqs) rc = sc.get(&work, (size_t)(work_seqs * a.L));
    if (rc) return rc;
    a.scale = 1.0 / ((double)M * (double)M);
    CK(cudaEventRecord(ctx->k0, ctx->stream));
    CK(cudaMemsetAsync(d_count, 0, sizeof(unsigned long long), ctx->stream));
    rc = bluestein_tables(ctx, sc, a);
    if (rc) return rc;
    finite_count_kernel<<<grid_for(ctx, n * n, 256), 256, 0, ctx->stream>>>(map, n * n, d_count);
    const dim3 tgrid((unsigned)((n + 31) / 32), (unsigned)((n + 31) / 32)), tblock(32, 8);
    pupil_transpose_kernel<<<tgrid, tblock, 0, ctx->stream>>>(map, (int)n, d_count, gT);
    ctx->launches += 2;
    CK(cudaGetLastError());
    // pass 1: the n non-zero rows of the transposed pupil -> n x M
    rc = bluestein_rows(ctx, a, work, work_seqs, gT, n, rows, F_OUT_C);
    if (rc) return rc;
    transpose_kernel<<<dim3((unsigned)((M + 31) / 32), (unsigned)((n + 31) / 32)), tblock, 0,
                       ctx->stream>>>(rows, (int)n, (int)M, rowsT);
    ctx->launches++;
    CK(cudaGetLastError());
    // pass 2: M rows of n values -> |.|^2 / M^2 into the M x M PSF
    rc = bluestein_rows(ctx, a, work, work_seqs, rowsT, M, psf, F_OUT_ABS2);
    if (rc) return rc;
    CK(cudaEventRecord(ctx->k1, ctx->stream));
    ctx->kernel_timed = true;
    return 0;
}

int rtx_psf_lines(rtx_ctx* ctx, int64_t M, const double* psf, double* lines, double* stats) {
    using namespace rtx_wave;
    if (!ctx || !psf || !lines || !stats || M < 1 || M > RTX_PSF_MAX_M) return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    const int nchunk = (int)((M + LINES_CW - 1) / LINES_CW);
    const int nband = (int)((M + LINES_RB - 1) / LINES_RB);
    const long long nblocks = (long long)nchunk * nband;
    Scratch sc(ctx->stream);
    double *colp = nullptr, *rowp = nullptr, *bmax = nullptr, *d_stats = nullptr;
    unsigned long long* bbad = nullptr;
    int rc = sc.get(&colp, (size_t)(nband * M));
    if (!rc) rc = sc.get(&rowp, (size_t)(nchunk * M));
    if (!rc) rc = sc.get(&bmax, (size_t)nblocks);
    if (!rc) rc = sc.get(&bbad, (size_t)nblocks);
    if (!rc) rc = sc.get(&d_stats, 3);
    if (rc) return rc;
    CK(cudaEventRecord(ctx->k0, ctx->stream));
    psf_lines_tile_kernel<<<dim3((unsigned)nchunk, (unsigned)nband), LINES_THREADS, 0,
                            ctx->stream>>>(psf, (int)M, colp, rowp, bmax, bbad);
    psf_lines_finish_kernel<<<(unsigned)((M + 255) / 256), 256, 0, ctx->stream>>>(
        colp, rowp, (int)M, nband, nchunk, lines);
    psf_stats_kernel<<<1, LINES_THREADS, 0, ctx->stream>>>(lines + M, (int)M, bmax, bbad,
                                                          nblocks, d_stats);
    ctx->launches += 3;
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->k1, ctx->stream));
    ctx->kernel_timed = true;
    CK(cudaMemcpyAsync(stats, d_stats, 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int rtx_psf_encircled(rtx_ctx* ctx, int64_t M, const double* psf, double c0, double c1,
                      int64_t nbins, uint64_t* bins) {
    using namespace rtx_wave;
    if (!ctx || !psf || !bins || M < 1 || M > RTX_PSF_MAX_M || nbins < 1 || !std::isfinite(c0) ||
        !std::isfinite(c1))
        return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    Scratch sc(ctx->stream);
    unsigned long long* d_bins = nullptr;
    int* d_over = nullptr;
    int rc = sc.get(&d_bins, (size_t)nbins);
    if (!rc) rc = sc.get(&d_over, 1);
    if (rc) return rc;
    CK(cudaMemsetAsync(d_bins, 0, (size_t)nbins * sizeof(unsigned long long), ctx->stream));
    CK(cudaMemsetAsync(d_over, 0, sizeof(int), ctx->stream));
    const unsigned tiles = (unsigned)((M + EE_T - 1) / EE_T);
    CK(cudaEventRecord(ctx->k0, ctx->stream));
    psf_encircled_kernel<<<dim3(tiles, tiles), EE_THREADS, 0, ctx->stream>>>(
        psf, (int)M, c0, c1, nbins, d_bins, d_over);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->k1, ctx->stream));
    ctx->kernel_timed = true;
    int over = 0;
    CK(cudaMemcpyAsync(bins, d_bins, (size_t)nbins * sizeof(unsigned long long),
                       cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&over, d_over, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return over ? RTX_E_BADARG : 0;
}

int rtx_psf_mtf(rtx_ctx* ctx, int64_t M, const double* lines, double* mtf) {
    using namespace rtx_wave;
    if (!ctx || !lines || !mtf || M < 2 || M > RTX_PSF_MAX_M) return RTX_E_BADARG;
    FftArgs a;
    int rc = bluestein_plan(M, M, a);
    if (rc) return rc;
    a.x_stride = M;
    a.out_stride = M;
    a.scale = 1.0;
    CK(cudaSetDevice(ctx->device));
    Scratch sc(ctx->stream);
    double2 *z = nullptr, *work = nullptr;
    double* abs2 = nullptr;
    const long long work_seqs = bluestein_work_seqs(a);
    rc = sc.get(&z, (size_t)(2 * M));
    if (!rc) rc = sc.get(&abs2, (size_t)(2 * M));
    if (!rc && work_seqs) rc = sc.get(&work, (size_t)(work_seqs * a.L));
    if (rc) return rc;
    CK(cudaEventRecord(ctx->k0, ctx->stream));
    rc = bluestein_tables(ctx, sc, a);
    if (rc) return rc;
    real_to_complex_kernel<<<(unsigned)((2 * M + 255) / 256), 256, 0, ctx->stream>>>(lines, 2 * M,
                                                                                   z);
    ctx->launches++;
    CK(cudaGetLastError());
    rc = bluestein_rows(ctx, a, work, work_seqs, z, 2, abs2, F_OUT_ABS2);
    if (rc) return rc;
    const int half = (int)(M / 2);
    psf_abs_half_kernel<<<(unsigned)((2 * half + 255) / 256), 256, 0, ctx->stream>>>(
        abs2, (int)M, half, 2, mtf);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->k1, ctx->stream));
    ctx->kernel_timed = true;
    return 0;
}

int rtx_psf_window(rtx_ctx* ctx, int64_t M, const double* psf, int64_t i0, int64_t j0, int64_t w,
                   double* out) {
    using namespace rtx_wave;
    if (!ctx || !psf || !out || M < 1 || M > RTX_PSF_MAX_M || w < 1 || w > M) return RTX_E_BADARG;
    CK(cudaSetDevice(ctx->device));
    const int i = (int)(((i0 % M) + M) % M), j = (int)(((j0 % M) + M) % M);
    psf_window_kernel<<<dim3((unsigned)((w + 127) / 128), (unsigned)(w < 65535 ? w : 65535)), 128,
                        0, ctx->stream>>>(
        psf, (int)M, i, j, (int)w, out);
    ctx->launches++;
    CK(cudaGetLastError());
    return 0;
}

}  // extern "C"
