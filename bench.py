#!/usr/bin/env python
"""Benchmark of the geometric propagate hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--dump-outputs DIR]

Workload (N=1, and per rank for N>1 -- weak scaling): BASELINE.json configs[1],
"Double-Gauss 12-surface, 1e7 rays, 3 wavelengths, FP64, 1xB200": one STEP is
one pass of the hot path over the three wavelength bundles (3 launches of the
trace kernel, 1e7 aimed rays x 12 surfaces each, clip=True, full trace
y,u,i,t stored).  Metric: ray-surface intersections per second.

  value     device-resident inputs and outputs, CUDA events on the launching
            stream around exactly K steps (max over ranks)
  e2e       the same work through the call a user makes,
            GeometricTrace.propagate() on host arrays -> rtx_trace_host: H2D of
            the launch rays and D2H of the whole trace inside the timed region
            (page-locked host buffers, NUMA-local to the GPU);
            e2e.spot_consumer: the resident drop-in (what
            bind(rayopt.GeometricTrace, resident=True) runs): rays up,
            kernel, only y[-1] back -- what a spot-diagram consumer reads
  roofline  HBM: algorithmic bytes N*(6w + 10w*S) per launch / mean launch
            duration (CUDA events around every launch, separate pass)
  cpu_baseline  the REFERENCE itself (oracle/_ref, staged by oracle/make_ref.py)
            on all host cores: the whole workload ray-sharded over the cores;
            numpy port as fallback
  headline  (N=1, when the HBM is free) the north-star point: zoom S=20,
            1e8 rays, FP64, full trace resident, one launch
  c3        (N=1) BASELINE config C3: Cooke + aspheres, 1e8 rays, FP32
  multi_gpu (N>1) C4: every rank traces 1.25e8 rays generated in HBM and the
            SAME kernel stores y[-1] into the gather buffers of all ranks over
            NVLink (rtx_trace_gather); C5: the 25 zoom bundles split by rays
            so that every rank carries 25/N bundles' worth
  parity_ok samples of the timed results checked against the oracle (asserted)

`--impl reference` times the reference's own CPU path -- GeometricTrace.
rays_given + propagate of quartiq/rayopt -- on the same workload, ray-sharded
over all host cores (oracle/cpu_bench.py; one step = 1e7 rays x 3 wavelengths).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ray-surface intersections/sec"
UNIT = "ray-surfaces/s"
SYSTEM = "double_gauss"
FIELD_INDEX = 3            # field (0, 0.7) in tests/golden/systems.json
FIELD = (0., .7)
N_RAYS = 10_000_000        # per wavelength
WORKLOAD = ("C2: Double-Gauss 12-surface, 1e7 rays x 3 wavelengths, FP64, "
            "clip=True, field (0,0.7), full trace (y,u,i,t) stored")


def load_system(name):
    from rayopt_b200.surface_table import table_from_json
    with open(os.path.join(ROOT, "tests", "golden", "systems.json")) as f:
        ent = json.load(f)[name]
    ent["tables"] = [table_from_json(t) for t in ent["tables"]]
    return ent


def make_rays(ent, li, n, seed):
    from rayopt_b200.rays import aim_infinite, disc
    aim = ent["aim"][li][FIELD_INDEX]
    return aim_infinite(aim["field"], disc(n, seed), aim["z"], aim["p"],
                        ent["object_angle"])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def wait_first(self, timeout=5.0):
        """block until nvidia-smi has produced its first sample"""
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.01)

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        sm, smax, reasons, power = [], [], set(), []
        # samples inside the timed region; a region shorter than the sampling
        # period falls back to the samples nearest to it (still under load:
        # warm-up before, roofline pass after)
        rows = [r for t, r in self.rows if t0 <= t <= t1]
        if len(rows) < 2:
            near = sorted(self.rows, key=lambda tr: min(abs(tr[0] - t0), abs(tr[0] - t1)))
            rows = [r for _, r in near[:3]]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0]))
                smax.append(float(f[1]))
                power.append(float(f[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown",
                                "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def cpu_reference(steps, warmup):
    """The reference's CPU path on all host cores, in its own process
    (oracle/cpu_bench.py: no fork out of a CUDA process, no inherited NUMA
    binding): every step is the WHOLE C2 workload -- 1e7 rays per wavelength,
    ray-sharded over os.cpu_count() processes (78 125 rays per process on a
    128-thread host; with 4e5 rays per process the same host measured 3.0e7
    ray-surfaces/s, profiles/r2a_bench.json, so the natural sharding is also
    the reference's better case).  Returns cpu_bench's dict."""
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "cpu_bench.py"), "--system", SYSTEM,
           "--field", str(FIELD[0]), str(FIELD[1]), "--rays-total", str(N_RAYS),
           "--steps", str(steps), "--warmup", str(warmup)]
    out = subprocess.run(cmd, check=True, capture_output=True, text=True).stdout
    return json.loads(out.strip().splitlines()[-1])


def cpu_sample_text(r):
    return ("the whole workload per step: %d rays x %d wavelengths x %d surfaces, ray-sharded over "
            "%d processes x %d rays, quartiq/rayopt GeometricTrace.rays_given + "
            "propagate(clip=True), %.1f s per step" % (
                r["rays_per_step_and_wavelength"], r["wavelengths"], r["surfaces"], r["cores"],
                r["rays_per_proc"], statistics.mean(r["seconds"])))


def run_reference(args):
    """--impl reference: quartiq/rayopt's own GeometricTrace on all cores"""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    r = cpu_reference(args.steps, max(args.warmup, 1))
    sample = cpu_sample_text(r)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": statistics.mean(r["seconds"])*1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"],
                         "kind": r["kind"], "sample": sample},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


DUMP_RAYS = 12288          # rays per wavelength written by --dump-outputs


def dump_outputs(path, eng, dev, N):
    """--dump-outputs: the result arrays y, u, i, t of every wavelength bundle
    as the timed step left them, for rays 0, step, 2*step, ... (DUMP_RAYS of
    them, one strided D2H per surface row), float64, as <path>/<k>_l<li>.npy
    with the ray indices in <path>/ray_index.npy.  A ray clipped by an
    aperture or missing a surface is NaN in the trace from there on; every
    file is kept finite, so non-finite entries are written as 0 and
    <path>/<k>_l<li>_nonfinite.npy (float32, same shape) says what they were:
    1 for NaN, +2 / -2 for +inf / -inf, 0 for a finite value.  The launch rays depend only on the seed, so two builds
    given the same arguments can be compared array by array.
    3 bundles x 12 surfaces x 10 values x (8 + 4) B x 12288 rays = 53 MB."""
    from rayopt_b200._lib import check, ptr
    count = min(N, DUMP_RAYS)
    step = N//count
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "ray_index.npy"), np.arange(count, dtype=np.float64)*step)
    for li, d in enumerate(dev):
        for k in "YUIT":
            a = d[k]
            width = a.dtype.itemsize*(a.shape[2] if len(a.shape) == 3 else 1)
            out = np.empty((a.shape[0], count) + tuple(a.shape[2:]), a.dtype)
            for s in range(a.shape[0]):
                check(eng.lib.rtx_memcpy2d_d2h(eng.ctx, ptr(out[s]), width, a.rows(s).ptr,
                                               step*width, width, count))
            eng.sync()
            code = np.where(np.isnan(out), 1., np.where(np.isinf(out), 2.*np.sign(out), 0.))
            name = os.path.join(path, "%s_l%d" % (k.lower(), li))
            np.save(name + ".npy", np.where(np.isfinite(out), out, 0.))
            np.save(name + "_nonfinite.npy", code.astype(np.float32))


def rel_err(a, b):
    with np.errstate(invalid="ignore"):
        return float(np.nanmax(np.abs(a - b)/np.maximum(np.abs(b), 1.0)))


def check_sample(got, want, what, tol=1e-10):
    """parity of a sample of timed results: identical NaN mask, rel err <= tol"""
    ok = bool(np.array_equal(np.isnan(got), np.isnan(want)))
    err = rel_err(got, want) if ok else float("inf")
    return {"what": what, "nan_mask_equal": ok, "max_rel_err": err, "ok": ok and err <= tol}


# --------------------------------------------------------------------------
def leg_headline(eng, exact):
    """north-star point on one GPU: zoom S=20, ~1e8 rays (hexapolar grid
    generated in HBM), FP64, full trace resident, ONE launch per trace"""
    from rayopt_b200.rays import aim_infinite, hexapolar_xy
    ent = load_system("zoom")
    S, table, aim = ent["S"], ent["tables"][0], ent["aim"][0][FIELD_INDEX]
    rings = int(np.sqrt(1e8/3. - 1/12.) - 1/2.)
    N = 1 + 3*rings*(rings + 1)
    ld = (N + 63)//64*64
    need = N*48 + S*ld*80
    free = eng.free_bytes()
    if free < need + (2 << 30):
        return {"skipped": "needs %.1f GB of HBM, %.1f GB free" % (need/1e9, free/1e9)}
    y0, u0 = eng.aim_infinite_device(aim["field"], aim["z"], aim["p"], ent["object_angle"],
                                     nrays=10**8)
    out = [eng.empty((S, ld, 3)) for _ in range(3)] + [eng.empty((S, ld))]
    ms = []
    for _ in range(4):
        eng.trace_device(table, y0, u0, *out, N=N, ld=ld, clip=True, exact=exact)
        ms.append(eng.last_kernel_ms())
    k_ms = statistics.median(ms[1:])
    idx = np.unique(np.r_[0, np.random.default_rng(5).integers(1, N, 1500)])
    hy, hu = aim_infinite(aim["field"], hexapolar_xy(idx, rings), aim["z"], aim["p"],
                          ent["object_angle"])
    import np_oracle
    want = np_oracle.trace(table, hy, hu, clip=True)
    got = np.stack([np.stack([eng.download_rays(out[0].rows(j), idx) for j in range(S)]),
                    np.stack([eng.download_rays(out[1].rows(j), idx) for j in range(S)])])
    par = check_sample(got, np.stack([want[0], want[1]]), "headline y,u sample of %d rays" % len(idx))
    for a in [y0, u0] + out:
        a.free()
    alg = N*(48 + 80*S)
    peak, _ = peaks()
    return {"workload": "zoom S=20, %d rays (hexapolar grid generated in HBM), FP64, clip, full "
                        "trace resident, one launch" % N,
            "kernel_ms": k_ms, "all_ms": ms, "ray_surfaces_per_s": N*S/k_ms*1e3,
            "achieved_GBps": alg/k_ms/1e6, "frac": alg/k_ms/1e6/peak,
            "algorithmic_bytes": alg, "parity": par}


def maxr_t(torch, dist, x):
    t = torch.tensor([float(x)], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def leg_c3(eng):
    """BASELINE config C3 on one GPU: Cooke triplet with even aspheres (Newton
    intercept on 3 of 8 surfaces), ~1e8 rays generated in HBM, FP32, full
    trace resident (34 GB), one launch"""
    from rayopt_b200.rays import aim_infinite, hexapolar_xy
    import np_oracle
    ent = load_system("cooke_asph")
    S, table, aim = ent["S"], ent["tables"][0], ent["aim"][0][FIELD_INDEX]
    rings = int(np.sqrt(1e8/3. - 1/12.) - 1/2.)
    y0, u0 = eng.aim_infinite_device(aim["field"], aim["z"], aim["p"], ent["object_angle"],
                                     rings=rings, dtype=np.float32)
    N = y0.shape[0]//128*128
    need = S*N*40
    if eng.free_bytes() < need + (2 << 30):
        y0.free(), u0.free()
        return {"skipped": "needs %.1f GB of HBM" % (need/1e9)}
    out = [eng.empty((S, N, 3), np.float32) for _ in range(3)] + [eng.empty((S, N), np.float32)]
    ms = []
    for _ in range(4):
        eng.trace_device(table, y0, u0, *out, N=N, ld=N, clip=True)
        ms.append(eng.last_kernel_ms())
    k_ms = statistics.median(ms[1:])
    idx = np.unique(np.r_[0, np.random.default_rng(6).integers(1, N, 1500)])
    hy, hu = aim_infinite(aim["field"], hexapolar_xy(idx, rings), aim["z"], aim["p"],
                          ent["object_angle"])
    want = np_oracle.trace(table, hy, hu, clip=True)[0]
    got = np.stack([eng.download_rays(out[0].rows(j), idx) for j in range(S)]).astype(np.float64)
    flips = np.isnan(got) != np.isnan(want)         # rays within FP32 of an aperture edge
    both = ~np.isnan(got) & ~np.isnan(want)
    # SURVEY 8d comparator: per-surface scale for lengths (as tests/test_gpu_parity.py)
    scale = np.maximum(np.nanmax(np.abs(want), axis=(1, 2), keepdims=True), 1.0)
    rel = np.abs(got - want)/np.maximum(np.abs(want), scale)
    err = float(np.max(rel[both]))
    par = {"what": "C3 FP32 y sample of %d rays vs the FP64 oracle" % len(idx),
           "max_rel_err": err, "nan_mask_flips": int(flips.sum()), "entries": int(flips.size),
           "ok": bool(err <= 1e-5 and flips.mean() < 5e-3)}
    for a in [y0, u0] + out:
        a.free()
    alg = N*(24 + 40*S)
    peak, _ = peaks()
    return {"workload": "C3: Cooke + even aspheres S=8, %d rays generated in HBM, FP32, clip, full "
                        "trace resident, one launch" % N,
            "kernel_ms": k_ms, "all_ms": ms, "ray_surfaces_per_s": N*S/k_ms*1e3,
            "achieved_GBps": alg/k_ms/1e6, "frac": alg/k_ms/1e6/peak, "algorithmic_bytes": alg,
            "dtype": "f32", "parity": par}


def leg_c4(eng, dist, torch, exact, n_local=125_000_000):
    """C4: 1.25e8 rays per rank generated in HBM, trace + all-gather of y[-1]
    in one kernel per rank (TMA bulk stores into the IPC-mapped gather buffers
    of ALL ranks over NVLink)"""
    from rayopt_b200.rays import aim_infinite, hexapolar_xy
    from rayopt_b200.sharding import PeerGather
    import np_oracle
    rank, world = dist.get_rank(), dist.get_world_size()
    ent = load_system(SYSTEM)
    S, table = ent["S"], ent["tables"][0]
    n_local = n_local//64*64
    fields = [0, 3, 1, 2, 4, 3, 1, 2]                  # a field point per rank
    aim = ent["aim"][0][fields[rank % 8]]
    rings = int(np.sqrt((n_local + 4096)/3. - 1/12.) - 1/2.) + 1
    y0, u0 = eng.aim_infinite_device(aim["field"], aim["z"], aim["p"], ent["object_angle"],
                                     rings=rings)
    assert y0.shape[0] >= n_local
    pg = PeerGather(eng, dist, n_local*world)

    def run():
        eng.trace_gather(table, y0, u0, pg.ptrs, pg.b[rank], N=n_local, clip=True, exact=exact)
        eng.sync()
        dist.barrier()
    run()                                               # warm-up: IPC mappings, peer access
    kms, wall = [], []
    for _ in range(3):
        t0 = time.perf_counter()
        run()
        wall.append(time.perf_counter() - t0)
        kms.append(eng.last_kernel_ms())
    t = torch.tensor([statistics.median(kms), statistics.median(wall)*1e3], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    kms_max, wall_max = (float(x) for x in t)
    # a sample of the NEXT rank's segment as it arrived in THIS rank's buffer
    peer = (rank + 1) % world
    aim_p = ent["aim"][0][fields[peer % 8]]
    idx = np.unique(np.r_[0, np.random.default_rng(rank).integers(1, n_local, 400)])
    hy, hu = aim_infinite(aim_p["field"], hexapolar_xy(idx, rings), aim_p["z"], aim_p["p"],
                          ent["object_angle"])
    want = np_oracle.trace(table, hy, hu, clip=True)[0][-1]
    got = eng.download_rays(pg.buf, pg.b[peer] + idx)
    par = check_sample(got, want, "peer segment")
    # the statistics path (SURVEY 8e): every rank reduces its shard INSIDE the
    # trace kernel (rtx_trace_reduce, nothing stored), one NCCL all-reduce of 20
    # doubles; checked against rtx_moments over the full gathered spot
    center = np.zeros(4)
    eng.trace_reduce(table, y0, u0, N=n_local, clip=True, exact=exact, center=center)
    t0 = time.perf_counter()
    m_loc = eng.trace_reduce(table, y0, u0, N=n_local, clip=True, exact=exact, center=center)
    red_ms = eng.last_kernel_ms()
    m = torch.tensor(m_loc, device="cuda")
    dist.all_reduce(m, op=dist.ReduceOp.SUM)
    m = m.cpu().numpy()
    red_wall = maxr_t(torch, dist, (time.perf_counter() - t0)*1e3)
    m_full = eng.moments(pg.buf, N=n_local*world, center=center[:2])
    mom_err = float(np.max(np.abs(m[:8] - m_full)/np.maximum(np.abs(m_full), 1e-300)))
    mom_ok = bool(m[5] == n_local*world and m[4] == m_full[4] and mom_err < 1e-11)
    pg.close()
    # the same gather of (x, y) only (RTX_GATHER_XY): what a spot diagram reads,
    # 16 instead of 24 bytes per ray over NVLink (SURVEY 8e)
    pg2 = PeerGather(eng, dist, n_local*world, xy=True)

    def run_xy():
        eng.trace_gather(table, y0, u0, pg2.ptrs, pg2.b[rank], N=n_local, clip=True, exact=exact,
                         xy=True)
        eng.sync()
        dist.barrier()
    run_xy()
    kxy = []
    for _ in range(3):
        run_xy()
        kxy.append(eng.last_kernel_ms())
    kxy_max = maxr_t(torch, dist, statistics.median(kxy))
    got_xy = np.empty((len(idx), 2))
    for j, i in enumerate(pg2.b[peer] + idx):
        eng.lib.rtx_memcpy_d2h(eng.ctx, got_xy[j].ctypes.data, pg2.buf.ptr + int(i)*16, 16)
    eng.sync()
    par_xy = check_sample(got_xy, want[:, :2], "peer segment (x,y)")
    pg2.close()
    ok = torch.tensor([1.0 if (par["ok"] and mom_ok and par_xy["ok"]) else 0.0], device="cuda")
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    y0.free()
    u0.free()
    stats = {"api": "rtx_trace_reduce per rank + ONE NCCL all-reduce of 20 doubles",
             "kernel_ms_this_rank": red_ms, "wall_ms_max_over_ranks": red_wall,
             "rays_total": n_local*world, "rays_arrived": float(m[4]),
             "vs_rtx_moments_of_gathered_spot_rel_err": mom_err, "ok": mom_ok}
    return {"statistics_path": stats,
            "xy_only": {"kernel_ms_max_over_ranks": kxy_max,
                        "nvlink_bytes_sent_per_rank": (world - 1)*n_local*16,
                        "nvlink_GBps_per_rank": (world - 1)*n_local*16/(kxy_max*1e-3)/1e9,
                        "parity_this_rank": par_xy},
            "workload": "C4: Double-Gauss, %d rays per rank (%.3g total) generated in HBM, FP64, "
                        "trace + gather of y[-1] to all %d ranks in one kernel per rank"
                        % (n_local, n_local*world, world),
            "kernel_ms_max_over_ranks": kms_max, "wall_ms_max_over_ranks": wall_max,
            "ray_surfaces_per_s": world*n_local*S/(kms_max*1e-3),
            "nvlink_bytes_sent_per_rank": (world - 1)*n_local*24,
            "nvlink_GBps_per_rank": (world - 1)*n_local*24/(kms_max*1e-3)/1e9,
            "peer_segment_parity_ok": bool(ok.item() == 1.0), "parity_this_rank": par}


def leg_c5(eng, dist, torch, exact, NR=10_000_000):
    """C5: zoom S=20, 5 fields x 5 wavelengths x ~1e7 rays.  The 25 bundles
    form one ray space split evenly over the ranks (by rays: a rank carries
    25/world bundles' worth -- whole bundles plus at most two partial ones);
    launch rays generated in HBM, full trace (y,u,i,t) stored."""
    import np_oracle
    rank, world = dist.get_rank(), dist.get_world_size()
    ent = load_system("zoom")
    S = ent["S"]
    field_idx = [0, 1, 2, 4, 5]                        # fields 0, .25, .5, .75, 1
    bundles = [(fi, li) for fi in field_idx for li in range(5)]
    rings = int(np.sqrt(NR/3. - 1/12.) - 1/2.)
    N = 1 + 3*rings*(rings + 1)
    total = len(bundles)*N
    g0, g1 = rank*total//world//64*64, ((rank + 1)*total//world//64*64 if rank + 1 < world else total)
    segs = []                                           # (bundle, lo, hi) owned by this rank
    for b in range(len(bundles)):
        lo, hi = max(g0, b*N) - b*N, min(g1, (b + 1)*N) - b*N
        if hi > lo:
            segs.append((b, lo, hi))
    # one result set, sized for the longest segment and reused by every segment
    # of the rank (a throughput measurement: each launch stores its full trace;
    # 25 resident result sets would be 412 GB)
    ldmax = (max(hi - lo for _, lo, hi in segs) + 127)//128*128
    out = [eng.empty((S, ldmax, 3)) for _ in range(3)] + [eng.empty((S, ldmax))]
    work = []
    for b, lo, hi in segs:
        fi, li = bundles[b]
        aim = ent["aim"][li][fi]
        y0, u0 = eng.aim_infinite_device(aim["field"], aim["z"], aim["p"], ent["object_angle"],
                                         nrays=NR)
        work.append((ent["tables"][li], y0.rows(lo, hi), u0.rows(lo, hi), out, hi - lo, ldmax,
                     y0, u0))

    def step():
        for table, y0, u0, out, n, ld, _, _ in work:
            eng.trace_device(table, y0, u0, *out, N=n, ld=ld, clip=True, exact=exact)
    step()
    eng.sync()
    dist.barrier()
    reps = 3
    eng.timer_start()
    for _ in range(reps):
        step()
    ms = eng.timer_stop()/reps
    t = torch.tensor([ms], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    worst = float(t.item())
    table, y0, u0, out, n, ld, _, _ = work[-1]
    idx = np.arange(0, n, max(1, n//1500))
    hy, hu = eng.download_rays(y0, idx), eng.download_rays(u0, idx)
    want = np_oracle.trace(table, hy, hu, clip=True)
    got = np.stack([eng.download_rays(out[0].rows(j), idx) for j in range(S)])
    par = check_sample(got, want[0], "last segment y")
    ok = torch.tensor([1.0 if par["ok"] else 0.0], device="cuda")
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    mine = sum(w[4] for w in work)
    for w in work:
        w[6].free()
        w[7].free()
    for a in out:
        a.free()
    return {"workload": "C5: zoom S=20, 5 fields x 5 wavelengths x %d rays (25 bundles, split by "
                        "rays: %.3f bundles per rank), FP64, full trace stored" % (N, 25/world),
            "rays_this_rank": mine, "segments_this_rank": len(work),
            "step_ms_this_rank": ms, "step_ms_max_over_ranks": worst,
            "ray_surfaces_per_s": total*S/(worst*1e-3),
            "per_gpu_GBps": mine*(48 + 80*S)/(ms*1e-3)/1e9,
            "parity_ok": bool(ok.item() == 1.0), "parity_this_rank": par}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rays", type=int, default=N_RAYS)
    ap.add_argument("--exact", type=int, default=0, help="1: RTX_EXACT arithmetic")
    ap.add_argument("--direct", type=int, default=0, help="1: per-thread stores")
    ap.add_argument("--rpt", type=int, default=0, help="rays per thread (0: library default)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-headline", action="store_true")
    ap.add_argument("--no-multi", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of the last timed step's results as .npy files")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = torch = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from rayopt_b200.engine import Engine
    # this process and its page-locked buffers live on the GPU's NUMA node
    eng = Engine(local, numa=True)
    ent = load_system(SYSTEM)
    S, nl, N = ent["S"], len(ent["tables"]), args.rays
    ld = ((N + 63)//64)*64
    w = 8
    exact = bool(args.exact)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))   # the checker of the timed results
    import np_oracle
    checks = []

    def maxr(x):
        if dist is None:
            return float(x)
        t = torch.tensor([float(x)], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident workload: 3 bundles, 3 full result sets ----------
    host_rays = []
    dev = []
    # the launch rays are GENERATED IN HBM (rtx_aim_rays: pupil coordinates uniform
    # in the unit disc from the counter-based generator, seed per rank and
    # wavelength; InfiniteConjugate.aim from the reference's stored pupil-aiming
    # solution z, p); the e2e legs need them in page-locked host memory: one
    # D2H of the generated bundles before anything is timed
    import types
    from rayopt_b200.rays import GRID_RANDOM, aim_record
    obj = types.SimpleNamespace(finite=False, angle=ent["object_angle"], projection="rectilinear",
                                pupil=types.SimpleNamespace(telecentric=False))
    for li in range(nl):
        aim = ent["aim"][li][FIELD_INDEX]
        spec = aim_record(obj, aim["field"], aim["z"], aim["p"], dict(grid=GRID_RANDOM, n=N - 1),
                          False, None, seed=1000*rank + li)
        y0, u0 = eng.aim_rays(spec)                     # N - 1 random rays + the chief ray
        assert y0.shape[0] == N
        py, pu = eng.pinned_empty((N, 3)), eng.pinned_empty((N, 3))
        y0.download(out=py)
        u0.download(out=pu)
        host_rays.append((py, pu))
        d = {"y0": y0, "u0": u0,
             "Y": eng.empty((S, ld, 3)), "U": eng.empty((S, ld, 3)),
             "I": eng.empty((S, ld, 3)), "T": eng.empty((S, ld))}
        dev.append(d)

    def step():
        for li in range(nl):
            d = dev[li]
            eng.trace_device(ent["tables"][li], d["y0"], d["u0"], d["Y"], d["U"], d["I"],
                             d["T"], N=N, ld=ld, clip=True, exact=exact,
                             direct=bool(args.direct), rpt=args.rpt)

    def barrier():
        eng.sync()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        step()
    if sampler:
        sampler.wait_first()
        for _ in range(3):          # keep the GPU under load while the sampler spins up
            step()
    barrier()
    l0 = eng.launch_count()
    t_wall0 = time.time()
    eng.timer_start()
    for _ in range(args.steps):
        step()
    ms = eng.timer_stop()
    t_wall1 = time.time()
    launches = eng.launch_count() - l0
    for _ in range(3):              # samples right after the region are still under load
        step()
    barrier()
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    if args.dump_outputs and rank == 0:
        # the launches after the timed region repeat its step on the same
        # inputs, so the arrays hold what the last timed step wrote
        dump_outputs(args.dump_outputs, eng, dev, N)
    ms = maxr(ms)
    ms_per_step = ms/args.steps
    value = world*nl*N*S/(ms_per_step*1e-3)

    # ---- roofline of the dominant (only) kernel: events around each launch --
    per_launch = []
    for _ in range(2):
        for li in range(nl):
            d = dev[li]
            eng.trace_device(ent["tables"][li], d["y0"], d["u0"], d["Y"], d["U"], d["I"],
                             d["T"], N=N, ld=ld, clip=True, exact=exact,
                             direct=bool(args.direct), rpt=args.rpt)
            per_launch.append(eng.last_kernel_ms())
    k_ms = statistics.mean(per_launch)
    alg_bytes = N*(6*w + 10*w*S)
    achieved = alg_bytes/(k_ms*1e-3)/1e9
    peak, peak_src = peaks()
    # DRAM traffic per launch is NOT measurable from inside the process (it
    # needs ncu): the number below is carried over from the committed ncu
    # capture of this kernel at this size and labelled as such
    traffic = 10_017_400_000 if (N == N_RAYS and not args.direct) else None

    # ---- parity of the timed device-resident results (sample vs the oracle)
    idx = np.arange(0, N, max(1, N//2000))[:2000]
    want0 = np_oracle.trace(ent["tables"][0], host_rays[0][0][idx], host_rays[0][1][idx], clip=True)
    for k, j in (("Y", 0), ("U", 1), ("I", 2)):
        got = np.stack([eng.download_rays(dev[0][k].rows(s), idx) for s in range(S)])
        checks.append(check_sample(got, want0[j], "device-resident %s (bundle 0)" % k.lower()))
    for d in dev:
        for a in d.values():
            a.free()

    # ---- e2e: the call a user makes -- GeometricTrace.propagate() ----------
    # host (pinned) result arrays in the reference layout; inside the timed
    # region: H2D of the launch rays, the kernel, D2H of the whole trace.
    # The system is unrotated, so the drop-in stores u and i as two views of
    # one buffer (i[j] == u[j-1] bit for bit) and moves 56 B per ray-surface;
    # "full_copy" is the same through rtx_trace_host with all four arrays
    # (80 B per ray-surface).
    per_rank = {}

    def timed(fn, steps, tag=None):
        fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        own = time.perf_counter() - t0               # this rank's own work, before the barrier
        barrier()
        dt = maxr(time.perf_counter() - t0)
        if tag and dist is not None:                 # who is the slow one? (ms per step, by rank)
            t = torch.zeros(world, device="cuda", dtype=torch.float64)
            t[rank] = own/steps*1e3
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            per_rank[tag] = [round(float(x), 1) for x in t.cpu()]
        return dt

    def pcie_probe():
        """all ranks at once: one 1 GiB D2H and one 1 GiB H2D between HBM and this
        rank's page-locked (NUMA-local) memory, GB/s per rank -- the ceiling the
        host side leaves to the e2e pipeline when every GPU of the box copies"""
        from rayopt_b200._lib import check, ptr
        nb = 1 << 30
        h, d = eng.pinned_empty((nb,), np.uint8), eng.empty((nb,), np.uint8)
        out = {}
        for name, fn in (("d2h", lambda: check(eng.lib.rtx_memcpy_d2h(eng.ctx, ptr(h), d.ptr, nb))),
                         ("h2d", lambda: check(eng.lib.rtx_memcpy_h2d(eng.ctx, d.ptr, ptr(h), nb)))):
            fn()
            eng.sync()
            barrier()
            t0 = time.perf_counter()
            for _ in range(3):
                fn()
            eng.sync()
            gbs = 3*nb/(time.perf_counter() - t0)/1e9
            t = torch.zeros(world, device="cuda", dtype=torch.float64)
            t[rank] = gbs
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            out[name + "_GBps_per_rank"] = [round(float(x), 1) for x in t.cpu()]
            barrier()
        d.free()
        return out

    e2e = None
    if not args.no_e2e:
        from rayopt_b200 import GeometricTrace, PackedSystem, ResidentTrace
        ps = PackedSystem(ent["wavelengths"], ent["tables"], [n[0] for n in ent["n"]])
        # one trace object (7.5 GB of page-locked result arrays), propagated
        # once per wavelength and step: the launch rays of bundle 0, the
        # surface table of each wavelength
        g = GeometricTrace(ps, engine=eng, exact=exact)
        g.rays_given(host_rays[0][0], host_rays[0][1], l=ent["wavelengths"][0])

        def e2e_step():
            for l in ent["wavelengths"]:
                g.l = l
                g.propagate(clip=True)
        e2e_steps = max(1, min(args.steps, 3))
        dt = timed(e2e_step, e2e_steps, "e2e")
        # what came back to the host (last wavelength traced)
        wl = np_oracle.trace(ent["tables"][nl - 1], host_rays[0][0][idx], host_rays[0][1][idx],
                             clip=True)
        checks.append(check_sample(g.y[1:, idx], wl[0], "e2e host arrays y"))
        checks.append(check_sample(g.i[1:, idx], wl[2], "e2e host arrays i (view of u)"))
        checks.append(check_sample(g.t[1:, idx], wl[3], "e2e host arrays t"))
        e2e = {"value": world*nl*N*S*e2e_steps/dt, "unit": UNIT,
               "h2d_bytes_per_step": nl*N*6*w, "d2h_bytes_per_step": nl*N*S*7*w,
               "steps": e2e_steps, "ms_per_step": dt/e2e_steps*1e3,
               "api": "GeometricTrace.propagate(clip=True) -> rtx_trace_host: pinned host arrays, "
                      "chunked H2D/kernel/D2H pipeline; y,u,t copied back, i is a view of u"}
        if dist is not None:
            e2e["ms_per_step_by_rank"] = per_rank.get("e2e")
            e2e["pcie_probe_all_ranks_at_once"] = pcie_probe()
        del g
        import gc
        gc.collect()

        # ---- spot-diagram consumer (rayopt/analysis.py:269-280) on the resident
        # drop-in -- the class bind(rayopt.GeometricTrace, resident=True) puts in
        # front of the reference: rays_given (H2D), propagate (one launch, trace
        # stays in HBM), y[-1] (the only D2H)
        r = ResidentTrace(ps, engine=eng, exact=exact)
        spots = [None]*nl

        def spot_step():
            for li, l in enumerate(ent["wavelengths"]):
                r.rays_given(host_rays[li][0], host_rays[li][1], l=l)
                r.propagate(clip=True)
                spots[li] = r.y[-1]
        ssteps = max(1, min(args.steps, 5))
        dt = timed(spot_step, ssteps)
        wl = np_oracle.trace(ent["tables"][nl - 1], host_rays[nl - 1][0][idx],
                             host_rays[nl - 1][1][idx], clip=True)
        checks.append(check_sample(spots[nl - 1][idx], wl[0][-1], "resident spot y[-1]"))
        e2e["spot_consumer"] = {
            "value": world*nl*N*S*ssteps/dt, "unit": UNIT, "ms_per_step": dt/ssteps*1e3,
            "h2d_bytes_per_step": nl*N*6*w, "d2h_bytes_per_step": nl*N*3*w,
            "api": "ResidentTrace (the mixin behind bind(rayopt.GeometricTrace, resident=True)): "
                   "rays_given + propagate(clip=True) + y[-1]; the trace stays in HBM"}
        r.free()
        del r, spots
        gc.collect()

    if not args.no_e2e and world == 1:
        # all four arrays through the C ABI
        out = {"y": eng.pinned_empty((S, N, 3)), "u": eng.pinned_empty((S, N, 3)),
               "i": eng.pinned_empty((S, N, 3)), "t": eng.pinned_empty((S, N))}

        def full_step():
            for li in range(nl):
                eng.trace(ent["tables"][li], host_rays[li][0], host_rays[li][1], clip=True,
                          out=out, exact=exact, rpt=args.rpt)
        fsteps = max(1, min(args.steps, 2))
        dt = timed(full_step, fsteps)
        e2e["full_copy"] = {"value": world*nl*N*S*fsteps/dt, "ms_per_step": dt/fsteps*1e3,
                            "d2h_bytes_per_step": nl*N*S*10*w,
                            "api": "rtx_trace_host with y,u,i,t host outputs"}
        del out

    # ---- the multi-GPU design: fused trace + NVLink gather (C4), C5 by rays
    multi = None
    if world > 1 and not args.no_multi:
        multi = {"c4": leg_c4(eng, dist, torch, exact), "c5": leg_c5(eng, dist, torch, exact)}
        checks.append({"what": "C4 peer segments (all ranks)", "ok": multi["c4"]["peer_segment_parity_ok"]})
        checks.append({"what": "C5 samples (all ranks)", "ok": multi["c5"]["parity_ok"]})

    # ---- north-star point, driver-run when the GPU's memory allows ---------
    headline = c3 = None
    if world == 1 and not args.no_headline and N == N_RAYS:
        headline = leg_headline(eng, exact)
        if "parity" in headline:
            checks.append(headline["parity"])
        c3 = leg_c3(eng)
        if "parity" in c3:
            checks.append(c3["parity"])

    # ---- CPU baseline: the reference itself on the host cores ---------------
    cpu = None
    node = eng.numa_node
    eng.numa_bind(False)              # the CPU leg may use every core again
    if rank == 0 and world == 1 and not args.no_cpu:
        r = cpu_reference(steps=1, warmup=1)
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
               "sample": cpu_sample_text(r)}

    parity_ok = all(c["ok"] for c in checks)
    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "parity_ok": parity_ok,
            "config": {"workload": WORKLOAD, "rays_per_wavelength": N, "surfaces": S,
                       "wavelengths": nl, "parallelism": "rays sharded x%d" % world,
                       "arithmetic": "exact" if exact else "fast",
                       "stores": "direct" if args.direct else "tma-bulk",
                       "kernel_config": "rpt=%s store=%s warps=%s nbuf=%s (0/unset: library default rpt 2, per-CTA TMA bulk stores, 16 warps, 1 staging buffer)" % (args.rpt, os.environ.get("RTX_STORE", "-"), os.environ.get("RTX_WARPS", "-"), os.environ.get("RTX_NBUF", "-")),
                       "numa_node": node,
                       "rays": "aimed bundles generated in HBM (rtx_aim_rays, random disc, seed per "
                               "rank and wavelength)",
                       "l2": "outputs %.1f GB per launch >> 126 MB L2 (no flush needed)"
                             % (alg_bytes/1e9)},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved/peak, "traffic": traffic,
                         "traffic_source": "from profile, not measured in this run: ncu "
                                           "dram__bytes_read.sum+dram__bytes_write.sum per launch of "
                                           "this kernel at this size, profiles/r2c_dram_bytes_full_size.csv",
                         "peak_source": peak_src,
                         "kernel": "rtx::trace_kernel<double>", "kernel_ms": k_ms,
                         "algorithmic_bytes_per_launch": alg_bytes},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches,
            "clocks": clocks, "headline": headline, "c3": c3, "multi_gpu": multi,
            "parity_checks": checks,
        }))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()
    assert parity_ok, [c for c in checks if not c["ok"]]


if __name__ == "__main__":
    main()
