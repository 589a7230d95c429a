#!/usr/bin/env python
"""Device time of the PSF figures (Engine.psf_metrics: Analysis.opds,
rayopt/analysis.py:319-346) against the host alternative, on the 1e5- and
1e6-ray Double-Gauss hexapolar bundles of psf_timing.py.

    python scripts/psf_metrics_timing.py [--out profiles/psf_metrics_timing.txt]

Each pass (rtx_psf_lines, rtx_psf_encircled, rtx_psf_mtf, rtx_psf_window) is
timed with the CUDA events the library records around its kernels, as the mean
of `--reps` calls after a warm-up call of the same shape; the whole
psf_metrics call is timed with the host clock (it ends in a synchronise).  The
bytes a pass must read are computed from M and divided by its kernel time,
next to a 4 GB device-to-device copy measured in the same run.  The host
alternative is the D2H of the PSF into page-locked memory (CUDA events) plus
oracle/psf_metrics_oracle.analysis_opds, Analysis.opds's expressions, on this CPU.
"""
import argparse
import os
import platform
import subprocess
import sys
import time
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests", "golden")]

import numpy as np  # noqa: E402
import yaml  # noqa: E402

import psf_metrics_oracle  # noqa: E402
import ref_shim  # noqa: E402
import systems_yaml  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1e5,1e6")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--window", type=int, default=200)
    ap.add_argument("--out", default=None)
    ap.add_argument("--no-host", action="store_true")
    args = ap.parse_args()
    warnings.simplefilter("ignore")
    np.seterr(all="ignore")
    from rayopt_b200 import bind
    from rayopt_b200.engine import Engine
    eng = Engine(0)
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    except OSError:
        smi = eng.name
    say("device: %s | %s; host CPU: %s, %d cores" % (eng.name, smi, platform.processor() or
                                                      platform.machine(), os.cpu_count()))
    a = eng.empty((1 << 29,))                          # 4 GB
    b = eng.empty((1 << 29,))
    b.copy_from(a)
    eng.sync()
    eng.timer_start()
    for _ in range(10):
        b.copy_from(a)
    ms = eng.timer_stop()/10
    peak = 2*a.nbytes/ms/1e6
    say("HBM reference: D2D copy of 4 GB %.3f ms = %.0f GB/s (read + write)" % (ms, peak))
    a.free()
    b.free()

    R = ref_shim.load()
    for size in [int(float(s)) for s in args.sizes.split(",")]:
        s = R.System(**yaml.safe_load(systems_yaml.SYSTEMS["double_gauss"]))
        s.update()
        s.paraxial.refocus()
        t = bind(R.GeometricTrace, engine=eng, resident=True)(s)
        t.rays_point((0, .7), nrays=size, distribution="hexapolar", clip=True)
        N = t.nrays
        pad = 4
        radius = s[-1].distance
        m, _, x = t._opd_grid(radius, -2, -1, 4, "device")
        n = m.shape[0]
        M = pad*n
        d_psf = eng.psf(m, pad)
        m.free()
        d = (x[1] - x[0])*(1/(t.l/s.scale))/radius
        ktimes = {}

        def timed(name, fn):
            fn()                                       # warm-up, same shape
            eng.sync()
            acc = 0.
            for _ in range(args.reps):
                r = fn()
                eng.sync()
                acc += eng.last_kernel_ms()
            ktimes[name] = acc/args.reps
            return r
        d_lines = eng.empty((2, M))
        _, pk, total, _ = timed("lines", lambda: eng.psf_lines(d_psf, out=d_lines))
        res = eng.psf_metrics(d_psf, d, window=args.window)
        c0, c1 = M/2 + res.x0/res.dx, M/2 + res.y0/res.dx
        nbins = len(res.ee)
        timed("encircled", lambda: eng.psf_encircled(d_psf, c0, c1, nbins))
        d_mtf = eng.empty((2, M//2))
        timed("mtf", lambda: eng.psf_mtf(d_lines, out=d_mtf))
        w = 2*args.window + 1
        d_win = eng.empty((w, w))
        eng.psf_window(d_psf, 0, 0, w, out=d_win)
        eng.sync()
        eng.timer_start()
        for _ in range(args.reps):
            eng.psf_window(d_psf, 0, 0, w, out=d_win)
        ktimes["window"] = eng.timer_stop()/args.reps
        calls = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            eng.psf_metrics(d_psf, d, window=args.window)
            calls.append(time.perf_counter() - t0)
        call = 1e3*float(np.mean(calls))
        small = 8*2*M + 8*3 + 8*nbins + 8*2*(M//2) + 8*w*w
        say("N=%d rays, map %d^2, PSF %d^2 = %.2f GB FP64; clip=True, field 0.7; %d EE bins"
            % (N, n, M, M*M*8/1e9, nbins))
        reads = {"lines": 8*M*M, "encircled": 8*M*M, "mtf": 16*M, "window": 8*w*w}
        for k in ("lines", "encircled", "mtf", "window"):
            rate = reads[k]/ktimes[k]/1e6
            say("  %-10s %9.3f ms  reads %10.4f GB -> %6.0f GB/s = %.2f of the D2D copy rate"
                % (k, ktimes[k], reads[k]/1e9, rate, rate/peak))
        say("  psf_metrics(window=%d) call %.3f ms (host clock, mean of %d); %d bytes D2H "
            "(lines, stats, EE bins, MTF, window), no M^2-sized transfer"
            % (args.window, call, args.reps, small))
        say("  result: x0 %.6g y0 %.6g peak %.6g sum %.15f ee[-1] %.15f r90 %.4g"
            % (res.x0, res.y0, pk, total, res.ee[-1], res.r[min(np.searchsorted(res.ee, .9), nbins - 1)]))
        for dd in (d_lines, d_mtf, d_win):
            dd.free()
        if not args.no_host:
            host = eng.pinned_empty((M, M))
            d_psf.download(host)
            eng.sync()
            eng.timer_start()
            d_psf.download(host)
            d2h = eng.timer_stop()
            f = np.fft.fftfreq(M, d)
            p, q = np.broadcast_arrays(f[:, None], f)
            t0 = time.perf_counter()
            want = psf_metrics_oracle.analysis_opds(host, p, q)
            cpu = time.perf_counter() - t0
            say("  host alternative: D2H of the PSF %.3f ms (%.0f GB/s) + Analysis.opds's "
                "expressions (fftshift, ogrid radius, bincount, line-sum FFTs) %.2f s on the CPU "
                "= %.2f s -> device call %.0fx faster"
                % (d2h, M*M*8/d2h/1e6, cpu, cpu + d2h/1e3, (cpu + d2h/1e3)*1e3/call))
            say("  host result: x0 %.6g y0 %.6g peak %.6g, %d EE bins"
                % (want["x0"], want["y0"], want["peak"], len(want["ee"])))
            del host, want, p, q
        d_psf.free()
        t.free()
    eng.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
