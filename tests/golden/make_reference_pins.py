#!/usr/bin/env python
"""Generate tests/golden/pins/ FROM THE LIVE REFERENCE (see pins.py).

Needs the reference tree (oracle/ref_shim.py finds it):

    python tests/golden/make_reference_pins.py

oracle.json/.npz  test_oracle_vs_reference: per system and wavelength what
                  the packer reads of the reference's System, its pupil
                  solution (z, p) and the digests of its launch rays and of
                  its trace y,u,i,t (cooke_asph, compared within 1e-13: the
                  trace of a fixed sample of rays as values)
aim.json/.npz     test_aim_oracle: pupil_distribution, InfiniteConjugate.aim
                  and FiniteConjugate.aim results
aim_finite.json   test_packer: FiniteConjugate.aim results
elements.json/.npz  test_dropin_cpu: Spheroid.propagate / intercept / refract
                  results of four surfaces
"""
import json
import os
import sys
import warnings

import numpy as np
import yaml

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), HERE]

import pins  # noqa: E402
import ref_shim  # noqa: E402
import systems_yaml  # noqa: E402
from rayopt_b200.rays import disc  # noqa: E402
from rayopt_b200.surface_table import get_n_mu  # noqa: E402

warnings.simplefilter("ignore")
np.seterr(all="ignore")
R = ref_shim.load()
P = np.array(((-3., -2.5), (2., 2.8)))          # as tests/test_aim_oracle.py
ORACLE_CASES = [("cooke", 20000, False), ("double_gauss", 20000, True), ("zoom", 10000, True),
                ("cooke_asph", 400, True), ("mirror", 5000, False), ("singlet", 5000, True)]


def write(name, meta, arrays=None):
    os.makedirs(pins.DIR, exist_ok=True)
    with open(os.path.join(pins.DIR, name + ".json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)
    if arrays:
        np.savez_compressed(os.path.join(pins.DIR, name + ".npz"), **arrays)


def oracle_pins():
    meta, arrays = {}, {}
    for name, n, clip in ORACLE_CASES:
        s = R.System(**yaml.safe_load(systems_yaml.SYSTEMS[name]))
        s.update()
        s.paraxial.refocus()
        rec = {"n": n, "clip": clip, "angle": float(s.object.angle), "n0": {},
               "elements": [pins.element_attrs(e) for e in s],
               "n_mu": [{} if hasattr(e, "get_n_mu") else None for e in s], "wavelengths": []}
        for l in s.wavelengths[:2]:
            key = repr(float(l))
            g = R.GeometricTrace(s)
            z, p = s.pupil((0, .7), l=l)
            y, u = s.aim((0, .7), disc(n, 1), z, p, filter=False)
            g.rays_given(y, u, l)
            g.propagate(clip=clip)
            n0 = rec["n0"][key] = float(s.refractive_index(l, 0))
            for e, nm in zip(s[1:], rec["n_mu"][1:]):          # the packer's walk
                nn, mu = get_n_mu(e, n0, l)
                if nm is not None:
                    nm[key] = [n0, float(nn), None if mu is None else float(mu)]
                n0 = nn
            w = {"l": float(l), "z": float(z), "p": np.asarray(p, float).tolist(),
                 "n": g.n[1:].tolist(), "y0": pins.digest(g.y[0]), "u0": pins.digest(g.u[0])}
            for k in "yuit":
                w[k] = pins.digest(getattr(g, k)[1:])
            if name == "cooke_asph":
                idx = pins.sample_rows(n)
                for k in "yuit":
                    arrays["%s_%d_%s" % (name, len(rec["wavelengths"]), k)] = \
                        getattr(g, k)[1:, idx].copy()
                    w["nan_" + k] = pins.digest(np.isnan(getattr(g, k)[1:]))
            rec["wavelengths"].append(w)
        meta[name] = rec
    write("oracle", meta, arrays)


def aim_pins():
    meta, arrays = {"grids": {}, "infinite": {}, "curved": {}, "finite": {}}, {}

    def keep(key, a, exact, sample=True):
        """digest of `a`; with exact=False also the values (a fixed row sample)"""
        a = np.asarray(a, float)
        if not exact:
            arrays[key] = a[pins.sample_rows(len(a))] if sample else a
        return {"digest": pins.digest(a), "shape": list(a.shape)}

    for dist, n in (("half-meridional", 7), ("meridional", 12), ("sagittal", 9), ("cross", 23),
                    ("tee", 152), ("square", 500), ("triangular", 700), ("hexapolar", 400),
                    ("meridional", 1)):
        ref, xy, weight = R.utils.pupil_distribution(dist, n)
        meta["grids"]["%s-%d" % (dist, n)] = dict(
            ref=int(ref), weight_is_none=weight is None,
            xy=keep("grid_%s_%d" % (dist, n), xy, dist != "hexapolar", sample=False))
    for projection in ("rectilinear", "stereographic", "equisolid", "orthographic", "equidistant"):
        obj = R.conjugates.InfiniteConjugate(angle=.35, projection=projection)
        if projection == "orthographic":       # the reference raises (test_aim_oracle.py)
            try:
                obj.aim((0, .7), np.zeros((3, 2)), 25., P, surface=R.Spheroid(), filter=False)
                raise AssertionError("the reference aims orthographic projections now")
            except ValueError:
                continue
        for filt in (False, True):
            for dist, n in (("square", 300), ("tee", 31), ("hexapolar", 200)):
                ref, xy, _ = R.utils.pupil_distribution(dist, n)
                for yo in ((0., 0.), (0, .7), (-.4, .9)):
                    key = "%s_%d_%s_%s_%g_%g" % (projection, filt, dist, n, yo[0], yo[1])
                    want_y, want_u = obj.aim(yo, xy, 25., P, surface=R.Spheroid(), filter=filt)
                    meta["infinite"][key] = dict(y=keep(key + "_y", want_y, dist != "hexapolar"),
                                                 u=keep(key + "_u", want_u, True))
    for i, kw in enumerate([dict(curvature=.02), dict(curvature=-.03, conic=-.6),
                            dict(curvature=.01, aspherics=[0, 2e-6, -1e-9])]):
        obj = R.conjugates.InfiniteConjugate(angle=.2)
        surf = R.Spheroid(**kw)
        ref, xy, _ = R.utils.pupil_distribution("square", 200)
        want_y, want_u = obj.aim((0, .8), xy, 20., P, surface=surf, filter=True)
        meta["curved"]["kw%d" % i] = dict(surface={"attrs": pins.element_attrs(surf)},
                                          y=keep("curved_%d_y" % i, want_y, "aspherics" not in kw,
                                                 sample=False),
                                          u=keep("curved_%d_u" % i, want_u, True))
    for telecentric in (False, True):
        obj = R.conjugates.FiniteConjugate(radius=6., pupil=dict(type="radius", radius=3.,
                                                                 telecentric=telecentric))
        for z in (40., -35.):
            for j, surf in enumerate((R.Spheroid(), R.Spheroid(curvature=.02, conic=.3))):
                point = np.zeros((1, 3))
                point[..., :2] = -np.array([[.3, -.6]])*obj.radius
                srec = {"attrs": pins.element_attrs(surf),
                        "sag": [point.tolist(), float(np.asarray(surf.surface_sag(point)).reshape(-1)[0])]}
                for dist, n, filt in (("square", 300, True), ("cross", 21, False),
                                      ("triangular", 150, False)):
                    ref, xy, _ = R.utils.pupil_distribution(dist, n)
                    want_y, want_u = obj.aim((.3, -.6), xy, z, P, surface=surf, filter=filt)
                    key = "%d_%g_%d_%s" % (telecentric, z, j, dist)
                    meta["finite"][key] = dict(surface=srec, y=keep("finite_%s_y" % key, want_y, True),
                                               u=keep("finite_%s_u" % key, want_u, False))
    obj = R.conjugates.InfiniteConjugate(angle=.3)
    yp = np.random.default_rng(4).uniform(-1, 1, (500, 2))
    want_y, want_u = obj.aim((0, .5), yp, 30., P, surface=R.Spheroid(), filter=True)
    meta["given"] = dict(surface={"attrs": pins.element_attrs(R.Spheroid())},
                         y=keep("given_y", want_y, True), u=keep("given_u", want_u, True))
    write("aim", meta, arrays)


def aim_finite_pins():
    fc = R.conjugates.FiniteConjugate(radius=5., pupil=dict(type="radius", radius=3., distance=50.))
    a = np.array(((-3., -2.5), (3., 2.5)))
    meta = {}
    for z in (50., -40.):
        for yo in ((0, .7), (0., 0.), (.3, -.4)):
            y, u = fc.aim(np.array(yo), disc(500, 2), z=z, a=a.copy(), surface=None, filter=False)
            meta["%g_%g_%g" % ((z,) + yo)] = dict(y=pins.digest(y), u=pins.digest(u))
    write("aim_finite", meta)


def element_pins():
    """as tests/test_dropin_cpu.py::test_element_level_entry_points_match_reference"""
    rng = np.random.default_rng(5)
    n = 100
    y0 = np.c_[rng.normal(0, .5, (n, 2)), -np.ones(n)]
    u0 = rng.normal(0, .02, (n, 2))
    u0 = np.c_[u0, np.sqrt(1 - np.square(u0).sum(1))]
    meta, arrays = [], {}
    for j, kw in enumerate((dict(curvature=.1, material=1.5),
                            dict(curvature=-.05, conic=-.7, material="mirror"),
                            dict(curvature=.08, aspherics=[0, 1e-4, -2e-6], material=1.7),
                            dict(material=1.3))):
        kw = dict(kw)
        kw["material"] = R.Material.make(kw["material"])
        s = R.Spheroid(radius=1.2, **kw)
        want = s.propagate(y0, u0, 1.1, 550e-9, clip=True)
        nn, mu = s.get_n_mu(1.1, 550e-9)
        meta.append(dict(attrs=pins.element_attrs(s), n_mu=[1.1, float(nn), float(mu)],
                         mirror=bool(s.material.mirror), n=float(want[2])))
        mu = 1.1/want[2] if not s.material.mirror else -1.
        arrays.update({"%d_y" % j: want[0], "%d_u" % j: want[1], "%d_t" % j: want[3],
                       "%d_intercept" % j: s.intercept(y0, u0),
                       "%d_refract" % j: s.refract(want[0], u0, mu)})
    write("elements", {"surfaces": meta}, arrays)


if __name__ == "__main__":
    oracle_pins()
    aim_pins()
    aim_finite_pins()
    element_pins()
    for f in sorted(os.listdir(pins.DIR)):
        print("%-20s %7.1f kB" % (f, os.path.getsize(os.path.join(pins.DIR, f))/1e3))
