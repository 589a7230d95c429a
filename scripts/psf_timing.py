#!/usr/bin/env python
"""Per-stage time of the device PSF (GeometricTrace.psf, rayopt/geometric_trace.py:
146-169) against the host pipeline (scipy griddata + numpy fft2) on hexapolar
bundles of the Double-Gauss fixture at 1e5 and 1e6 rays.

    python scripts/psf_timing.py [--out profiles/psf_timing.txt] [--sizes 1e5,1e6]

Device stages are timed with CUDA events on the engine stream, each over
`--reps` repetitions after a warm-up call of the same shape: trace_opd (the
march with the OPD epilogue), regrid (rtx_opd_regrid), PSF (rtx_psf) and the
D2H of the PSF into page-locked memory.  The FFT passes' bytes are counted
from the shapes (what each pass must read and write once) and divided by the
PSF time; the HBM reference is a device-to-device copy of 4 GB measured in the
same run.  The host path is timed once on this machine's CPU with the
reference's own code (resident opd() = griddata, then the psf expression).
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

import ref_shim  # noqa: E402
import systems_yaml  # noqa: E402


def fft_bytes(n, pad):
    """bytes rtx_psf's passes read and write once (complex = 16 B)"""
    M = pad*n
    L = 2
    while L < M + n - 1:
        L *= 2
    one_tile = L <= 4096

    def rows(nseq, out_item):
        if one_tile:
            return nseq*(16*n + out_item*M)
        return nseq*(16*n + 16*L + 2*16*L + 16*L + out_item*M)
    return (8*n*n + 8*n*n + 16*n*n                     # count, pupil read, transposed write
            + rows(n, 16) + 2*16*n*M + rows(M, 8))     # pass 1, transpose, pass 2


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1e5,1e6")
    ap.add_argument("--reps", type=int, default=5)
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
        N, rings = t.nrays, t._hex_rings
        n = int(4*N**.5)
        pad = 4
        M = pad*n
        radius = s[-1].distance
        times = {}

        def timed(name, fn):
            fn()                                       # warm-up, same shape
            eng.sync()
            eng.timer_start()
            for _ in range(args.reps):
                r = fn()
            times[name] = eng.timer_stop()/args.reps
            return r
        A, P, a_ref, p_ref, ls = t._opd_device(radius)

        def opd():
            A2, P2 = t._opd_device(radius)[:2]
            A2.free()
            P2.free()
        timed("trace_opd", opd)
        m = timed("regrid", lambda: eng.opd_regrid(A, P, a_ref, p_ref, ls, rings, n)[0])
        d_psf = eng.empty((M, M))
        timed("psf", lambda: eng.psf(m, pad, out=d_psf))
        host = eng.pinned_empty((M, M))
        timed("d2h", lambda: d_psf.download(host))
        fin = np.isfinite(m.download()).sum()
        tot = sum(times.values())
        gb = fft_bytes(n, pad)/1e9
        say("N=%d rays (%d rings), map %d^2 (%d finite), PSF %d^2 = %.2f GB FP64; clip=True, "
            "field 0.7" % (N, rings, n, fin, M, M*M*8/1e9))
        for k in ("trace_opd", "regrid", "psf", "d2h"):
            say("  %-10s %9.3f ms" % (k, times[k]))
        say("  device total %.3f ms (D2H included)" % tot)
        say("  FFT passes: %.2f GB moved once each -> %.0f GB/s = %.2f of the D2D copy rate"
            % (gb, gb/times["psf"]*1e3, gb/times["psf"]*1e3/peak))
        for d in (A, P, m, d_psf):
            d.free()
        if not args.no_host:
            t0 = time.perf_counter()
            xs, ys, o = t.opd(radius=radius)           # scipy griddata on the host
            t1 = time.perf_counter()
            good = np.isfinite(o)
            g = np.where(good, np.exp(-2j*np.pi*o), 0)/np.count_nonzero(good)**.5
            apsf = np.fft.fft2(g, (M, M))
            ref_psf = (apsf*apsf.conj()).real/apsf.size
            t2 = time.perf_counter()
            say("  host: griddata %.2f s, fft2 + |.|^2 %.2f s, total %.2f s -> device %.0fx faster"
                % (t1 - t0, t2 - t1, t2 - t0, (t2 - t0)*1e3/tot))
            del apsf, g, ref_psf
        del host
        t.free()
    eng.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
