"""Host logic of the GeometricTrace drop-in on CPU: the engine is replaced by
a stand-in that runs the oracle through the same `Engine.trace` interface, so
that allocation, the u/i aliasing, sub-range propagate, rms/refocus and the
binding into the reference classes are exercised without a GPU."""
import warnings

import numpy as np
import pytest
import yaml

import np_oracle
import ref_shim
import systems_yaml
from conftest import load_golden, load_systems
from rayopt_b200 import GeometricTrace, PackedSystem, bind, system_propagate


class OracleEngine:
    """same call surface as rayopt_b200.engine.Engine.trace"""
    calls = 0

    def trace(self, table, y0, u0, clip=False, keep_last=False, rot0=None, dtype=np.float64,
              exact=False, direct=False, rpt=0, out=None, want=("y", "u", "i", "t")):
        OracleEngine.calls += 1
        Y, U, I, T = np_oracle.trace(table, y0, u0, clip=clip, rot0=rot0)
        res = dict(y=Y, u=U, i=I, t=T)
        if out is None:
            return tuple(res[k] if k in want else None for k in "yuit")
        for k in want:
            out[k][...] = res[k]
        return tuple(out.get(k) for k in "yuit")

    def pinned_empty(self, shape, dtype):
        return np.empty(shape, dtype)

    def trace_bundles(self, tables, y0s, u0s, clip=False, keep_last=False, rot0=None,
                      dtype=np.float64, exact=False, want=("y", "u", "i", "t")):
        OracleEngine.calls += 1
        return [np_oracle.trace(t, y, u, clip=clip) for t, y, u in zip(tables, y0s, u0s)]


def _packed(name):
    ent = load_systems()[name]
    return PackedSystem(ent["wavelengths"], ent["tables"], [n[0] for n in ent["n"]]), ent


def test_alias_incidence_full_and_subrange():
    ps, ent = _packed("double_gauss")
    c = load_golden("double_gauss_l1_clip")
    g = GeometricTrace(ps, engine=OracleEngine())
    g.rays_given(c["y0"], c["u0"], l=ent["wavelengths"][1])
    g.propagate(clip=True)
    assert g._i_alias and np.shares_memory(g.i, g.u)
    for a, b in ((g.y, c["Y"]), (g.u, c["U"]), (g.i, c["I"]), (g.t, c["T"])):
        assert np.array_equal(a[1:], b, equal_nan=True)
    assert np.array_equal(g.n[1:], c["n"]) and np.array_equal(g.i[0], g.u[0])
    # propagate(start, stop) on a sub-range (geometric_trace.py:72-80)
    c2 = load_golden("double_gauss_sub_4_9")
    g.rays_given(c2["y0"]*0 + c["y0"][:1], c["u0"][:1], l=ent["wavelengths"][0])
    g = GeometricTrace(ps, engine=OracleEngine())
    g.allocate(c2["y0"].shape[0])
    g.l, g.w, g.ref = ent["wavelengths"][0], None, 0
    g.y[3], g.u[3], g.n[3] = c2["y0"], c2["u0"], c2["table"]["n0"][0]
    g.propagate(start=4, stop=9, clip=True)
    for a, b in ((g.y, c2["Y"]), (g.u, c2["U"]), (g.i, c2["I"]), (g.t, c2["T"])):
        assert np.array_equal(a[4:9], b, equal_nan=True)


def test_rotated_system_materialises_incidence():
    c = load_golden("tilted_clip1")
    ps = PackedSystem([587.56e-9], [c["table"]], [c["table"]["n0"][0]])
    g = GeometricTrace(ps, engine=OracleEngine())
    g.rays_given(c["y0"], c["u0"], l=587.56e-9)
    g.propagate(clip=True)
    assert not g._i_alias and not np.shares_memory(g.i, g.u)
    for a, b in ((g.y, c["Y"]), (g.u, c["U"]), (g.i, c["I"]), (g.t, c["T"])):
        assert np.array_equal(a[1:], b, equal_nan=True)
    # without aliasing: same answer
    g2 = GeometricTrace(ps, engine=OracleEngine(), alias_incidence=False)
    g2.rays_given(c["y0"], c["u0"], l=587.56e-9)
    g2.propagate(clip=True)
    assert np.array_equal(g2.i, g.i, equal_nan=True)


def test_rays_given_pads_2d_input_and_rms_known_answer():
    """rays_given semantics (geometric_trace.py:49-70) and the reference's
    known answer rms = 0.052 (test_raytrace.py:192-195)"""
    ps, ent = _packed("cooke")
    c = load_golden("cooke_radau13")
    g = GeometricTrace(ps, engine=OracleEngine())
    g.rays_given(c["y0"][:, :2], c["u0"][:, :2], w=c["w"])
    assert g.l == ent["wavelengths"][0]
    np.testing.assert_allclose(g.u[0, :, 2], c["u0"][:, 2], rtol=1e-15)
    assert np.all(g.y[0, :, 2] == 0) and np.all(g.t[0] == 0)
    g.propagate()
    assert abs(g.rms() - 0.052)/0.052 < 1e-2


@pytest.mark.skipif(not ref_shim.available(), reason="reference tree not present")
def test_bound_reference_class_matches_reference():
    """rayopt_b200.bind(rayopt.GeometricTrace): rays_point / rays_clipping /
    refocus of the REFERENCE class run on the replaced allocate/propagate and
    give the reference's own results; System.propagate's replacement feeds
    the reference's ray aiming."""
    warnings.simplefilter("ignore")
    R = ref_shim.load()
    s = R.System(**yaml.safe_load(systems_yaml.COOKE))
    s.update()
    s.paraxial.refocus()
    GT = bind(R.GeometricTrace, engine=OracleEngine())
    ref = R.GeometricTrace(s)
    ref.rays_point((0, 1.), nrays=300, distribution="hexapolar", clip=True)
    got = GT(s)
    got.rays_point((0, 1.), nrays=300, distribution="hexapolar", clip=True)
    for k in "yuit":
        assert np.array_equal(getattr(got, k), getattr(ref, k), equal_nan=True), k
    assert np.array_equal(got.n, ref.n)
    assert np.array_equal(got.path, ref.path) and np.array_equal(got.origins, ref.origins)
    ref2, got2 = R.GeometricTrace(s), GT(s)
    ref2.rays_clipping((0, 1.))
    got2.rays_clipping((0, 1.))
    assert np.array_equal(got2.y, ref2.y, equal_nan=True)
    # the System.propagate cut used by aim_chief / aim_marginal (system.py:507-555)
    y, u = s.aim((0, .5), None, *s.pupil((0, .5)), filter=False)
    n0 = s.refractive_index(s.wavelengths[0], 0)
    a = list(s.propagate(y, u, n0, s.wavelengths[0], stop=6, clip=False))
    b = list(system_propagate(s, y, u, n0, s.wavelengths[0], stop=6, clip=False,
                              engine=OracleEngine()))
    assert len(a) == len(b) == 5
    for ya, yb in zip(a, b):
        for xa, xb in zip(ya, yb):
            assert np.array_equal(np.asarray(xa), np.asarray(xb), equal_nan=True)


def test_element_level_entry_points_match_reference():
    """rayopt_b200.elements.propagate / intercept / refract vs the reference's
    Spheroid methods (test_elements.py:109-134 style: a refracting sphere and
    an asphere hit by random near-axis rays); the surfaces and the reference's
    results are stored in tests/golden/pins/elements.json/.npz."""
    import pins
    from rayopt_b200 import elements as el
    meta, want = pins.load("elements")
    rng = np.random.default_rng(5)
    n = 100
    y0 = np.c_[rng.normal(0, .5, (n, 2)), -np.ones(n)]
    u0 = rng.normal(0, .02, (n, 2))
    u0 = np.c_[u0, np.sqrt(1 - np.square(u0).sum(1))]
    eng = OracleEngine()
    for j, rec in enumerate(meta["surfaces"]):
        l = 550e-9
        s = pins.PinnedElement(rec["attrs"], {repr(l): rec["n_mu"]})
        got = el.propagate(s, y0, u0, 1.1, l, clip=True, engine=eng)
        tol = dict(rtol=1e-13, atol=1e-14)
        np.testing.assert_allclose(got[0], want["%d_y" % j], **tol)
        np.testing.assert_allclose(got[1], want["%d_u" % j], **tol)
        assert got[2] == rec["n"]
        np.testing.assert_allclose(got[3], want["%d_t" % j], **tol)
        np.testing.assert_allclose(el.intercept(s, y0, u0, engine=eng), want["%d_intercept" % j], **tol)
        mu = 1.1/rec["n"] if not rec["mirror"] else -1.
        ys = want["%d_y" % j]
        np.testing.assert_allclose(el.refract(s, ys, u0, mu, engine=eng), want["%d_refract" % j],
                                   rtol=1e-12, atol=1e-13)


@pytest.mark.skipif(not ref_shim.available(), reason="reference tree not present")
def test_standalone_refocus_and_rms_match_reference():
    """the standalone class's own rays_given / rms / refocus (written against
    geometric_trace.py:49-99, 171-183) against the reference's"""
    warnings.simplefilter("ignore")
    R = ref_shim.load()

    def system():
        s = R.System(**yaml.safe_load(systems_yaml.DOUBLE_GAUSS))
        s.update()
        s.paraxial.refocus()
        s[-1].distance += .3          # defocus so that refocus has work to do
        return s
    s1, s2 = system(), system()
    ref = R.GeometricTrace(s1)
    ref.rays_point((0, .7), nrays=200, distribution="hexapolar", clip=True, filter=False)
    got = GeometricTrace(s2, engine=OracleEngine())
    got.rays_given(ref.y[0, :, :2] if False else ref.y[0], ref.u[0], ref.l, ref.w, ref.ref)
    got.propagate(clip=True)
    assert np.array_equal(got.y, ref.y, equal_nan=True)
    sub = np.isfinite(ref.y[-1, :, 0])
    d0 = s1[-1].distance
    ref.refocus()
    got.refocus()
    assert abs((s1[-1].distance - d0) - (s2[-1].distance - d0)) < 1e-12
    np.testing.assert_allclose(got.y[-1][sub], ref.y[-1][sub], rtol=0, atol=1e-11)
    # rms over the surviving rays (the reference's rms is not NaN-masked)
    g2 = GeometricTrace(s2, engine=OracleEngine())
    g2.rays_given(ref.y[0][sub], ref.u[0][sub], ref.l)
    g2.propagate()
    r2 = R.GeometricTrace(s2)
    r2.rays_given(ref.y[0][sub], ref.u[0][sub], ref.l)
    r2.propagate()
    assert abs(g2.rms() - r2.rms()) < 1e-14 and abs(g2.rms(ref=0) - r2.rms(ref=0)) < 1e-14


@pytest.mark.skipif(not ref_shim.available(), reason="reference tree not present")
def test_reference_own_raytrace_tests_through_the_dropin():
    """The reference's own integration tests for this path
    (rayopt/test/test_raytrace.py:151-199: test_aim_point, test_aim_point_more,
    test_quadrature) re-run with BOTH call sites replaced -- System.propagate
    (ray aiming) and GeometricTrace.allocate/propagate -- i.e. as the API
    conformance suite of the drop-in (engine: the oracle stand-in on CPU)."""
    warnings.simplefilter("ignore")
    R = ref_shim.load()
    import rayopt_b200

    class System(R.System):          # patched copies: leave the shared classes alone
        pass

    class Trace(R.GeometricTrace):
        pass
    rayopt_b200.install(System, Trace, engine=OracleEngine())
    s = System(**yaml.safe_load(systems_yaml.COOKE))
    s.update()
    s.paraxial.refocus()
    s.paraxial.update_conjugates()
    calls0 = OracleEngine.calls
    g = Trace(s)
    # test_aim_point
    g.rays_point((0, 1.))
    g.rays_clipping((0, 1.))
    g.rays_line((0, 1.))
    # test_aim_point_more
    i = s.stop
    r = np.array([el.radius for el in s[1:-1]])
    g.rays_clipping((0, 1.))
    np.testing.assert_allclose(g.u[0, :, :], g.u[0, (0,)*g.u.shape[1], :])
    np.testing.assert_allclose(g.y[i, 0, 1], 0, atol=5e-3)
    np.testing.assert_allclose(min(g.y[1:-1, 1, 1] + r), 0, atol=1e-3)
    np.testing.assert_allclose(max(g.y[1:-1, 2, 1] - r), 0, atol=1e-3)
    g.rays_point((0, 1.), distribution="cross", nrays=5, filter=False)
    np.testing.assert_allclose(g.y[i, :3, 1]/s[i].radius, [-1, 0, 1], atol=1e-3, rtol=3e-2)
    np.testing.assert_allclose(g.y[i, :, 0]/s[i].radius, [0, 0, 0, -1, 0, 1], atol=1e-1)
    # test_quadrature: the known answer of the path
    g.rays_point((0, 1.), nrays=13, distribution="radau", filter=False)
    a = g.rms()
    np.testing.assert_allclose(a, .052, rtol=1e-2)
    g.rays_point((0, 1.), nrays=500, distribution="square", clip=False, filter=True)
    np.testing.assert_allclose(a, g.rms(), rtol=5e-2)
    assert OracleEngine.calls - calls0 > 50          # aiming really went through the engine
    # and the aim solution equals the unpatched reference's
    s0 = R.System(**yaml.safe_load(systems_yaml.COOKE))
    s0.update()
    s0.paraxial.refocus()
    s0.paraxial.update_conjugates()
    z0, p0 = s0.pupil((0, 1.))
    z1, p1 = s.pupil((0, 1.))
    np.testing.assert_allclose(z1, z0, rtol=1e-12)
    np.testing.assert_allclose(p1, p0, rtol=1e-12)


class FakeDeviceArray:
    """numpy-backed stand-in for rayopt_b200.engine.DeviceArray"""

    def __init__(self, a):
        self.a = a
        self.shape, self.dtype, self.nbytes = a.shape, a.dtype, a.nbytes
        self.downloads = 0

    def rows(self, r0, r1=None):
        return FakeDeviceArray(self.a[r0:(r0 + 1 if r1 is None else r1)])

    def upload(self, v):
        v = np.asarray(v, self.a.dtype)
        self.a.reshape(-1)[:v.size] = v.reshape(-1)      # leading bytes, like the H2D copy
        return self

    def download(self, out=None):
        if out is None:
            return self.a.copy()
        out.reshape(-1)[:] = self.a.reshape(-1)[:out.size]
        return out

    def copy_from(self, other, nbytes=None):
        n = min(self.a.size, other.a.size) if nbytes is None else nbytes//self.a.itemsize
        self.a.reshape(-1)[:n] = other.a.reshape(-1)[:n]
        return self

    def free(self):
        pass


class FakeResidentEngine:
    def empty(self, shape, dtype=np.float64):
        return FakeDeviceArray(np.full(shape, np.nan, dtype))

    def to_device(self, a, dtype=None):
        return FakeDeviceArray(np.array(a, dtype))

    def trace_device(self, table, y0, u0, Y, U, I, T, N=None, ld=None, clip=False, rot0=None,
                     exact=False, **kw):
        res = np_oracle.trace(table, y0.a[0, :N], u0.a[0, :N], clip=clip, rot0=rot0)
        for dst, src in zip((Y, U, I, T), res):
            if dst is not None:
                dst.a[:, :N] = src

    def sync(self):
        pass

    def download_rays(self, d, idx):
        return d.a.reshape(-1, 3)[np.asarray(idx)].copy()

    def rms(self, y, w, N=None, ref_point=None):
        yy = y.a[0, :N, :2]
        c = yy.mean(0) if ref_point is None else np.asarray(ref_point)
        ww = np.ones(N)/N if w is None else w.a
        return float(np.sqrt((np.square(yy - c).sum(1)*ww).sum()))

    def refocus_shift(self, y, inc, w=None, N=None):
        yy, ii = y.a[0, :N, :2], inc.a[0, :N]
        uu = ii[:, :2]/ii[:, 2:]
        ok = np.isfinite(uu).all(1)
        yy, uu = yy[ok] - yy[ok].mean(0), uu[ok] - uu[ok].mean(0)
        ww = np.ones(len(yy)) if w is None else w.a[ok]
        return float(-(ww[:, None]*yy*uu).sum()/(ww[:, None]*uu*uu).sum())


def test_resident_trace_host_logic_on_cpu():
    """LazyRows / ResidentTrace bookkeeping (row cache, invalidation on
    re-propagate, sub-range traces from a resident row) without a GPU"""
    from rayopt_b200 import ResidentTrace
    ps, ent = _packed("double_gauss")
    c = load_golden("double_gauss_l0_clip")
    g = ResidentTrace(ps, engine=FakeResidentEngine())
    g.rays_given(c["y0"][:, :2] if False else c["y0"], c["u0"], l=ent["wavelengths"][0], w=c["w"])
    g.propagate(clip=True)
    assert g.y.shape == (13, 256, 3) and g.t.shape == (13, 256) and len(g.y) == 13
    assert np.array_equal(g.y[-1], c["Y"][-1], equal_nan=True)
    assert np.array_equal(g.y[5, :, :2], c["Y"][4, :, :2], equal_nan=True)
    assert np.array_equal(g.u[2:4], c["U"][1:3], equal_nan=True)
    assert np.array_equal(np.asarray(g.t)[1:], c["T"], equal_nan=True)
    assert np.array_equal(g.i[0], c["u0"]) and np.array_equal(g.n[1:], c["n"])
    first = g.y[-1]
    assert g.y[-1] is first                      # cached row
    g.propagate(start=4, stop=9, clip=False)     # rows 4..8 re-traced, cache dropped
    assert g.y[-1] is first and 5 not in g.y._rows
    want = np_oracle.trace(c["table"][3:8], g.y[3], g.u[3], clip=False)
    assert np.array_equal(g.y[4:9], want[0], equal_nan=True)
    assert abs(g.rms(3) - np_oracle.rms(g.y[3], c["w"])) < 1e-15


@pytest.mark.skipif(not ref_shim.available(), reason="reference tree not present")
def test_bound_resident_class_matches_reference():
    """bind(rayopt.GeometricTrace, resident=True) on the numpy stand-in of the
    device: the reference's rays_point / rays_clipping / rays_paraxial / opd
    run on LazyRows, rms / refocus on the (fake) device reductions"""
    warnings.simplefilter("ignore")
    R = ref_shim.load()

    def system():
        s = R.System(**yaml.safe_load(systems_yaml.DOUBLE_GAUSS))
        s.update()
        s.paraxial.refocus()
        s[-1].distance += .3
        return s
    s1, s2 = system(), system()
    GT = bind(R.GeometricTrace, engine=FakeResidentEngine(), resident=True)
    for fn, args, kw in (("rays_point", ((0, .7),), dict(nrays=150, distribution="hexapolar", clip=True)),
                         ("rays_point", ((0, 1.),), dict(nrays=31, distribution="tee", clip=True)),
                         ("rays_clipping", ((0, 1.),), {}), ("rays_paraxial", (), {})):
        ref, got = R.GeometricTrace(s1), GT(s2)
        getattr(ref, fn)(*args, **kw)
        getattr(got, fn)(*args, **kw)
        for k in "yuit":
            assert np.array_equal(np.asarray(getattr(got, k)), getattr(ref, k), equal_nan=True), (fn, k)
        assert np.array_equal(got.n, ref.n) and got.ref == ref.ref
        assert got._i_alias and got.y.shape == ref.y.shape
    ref, got = R.GeometricTrace(s1), GT(s2)
    for t in (ref, got):
        t.rays_point((0, .7), nrays=200, distribution="hexapolar", clip=True, filter=False)
    d0 = s1[-1].distance
    ref.refocus()
    got.refocus()
    assert abs(s1[-1].distance - d0) > 1e-3
    assert abs(s1[-1].distance - s2[-1].distance) < 1e-12
    for t in (ref, got):
        t.rays_point((0, 0.), nrays=100, distribution="hexapolar")
    assert abs(got.rms() - ref.rms()) < 1e-14 and abs(got.rms(ref=0) - ref.rms(ref=0)) < 1e-14
    # the reference's own opd() reads the LazyRows like arrays (the mixin's
    # device epilogue is exercised on the GPU, tests/test_gpu_dropin_reference.py)
    for a, b in zip(R.GeometricTrace.opd(got, resample=False), ref.opd(resample=False)):
        np.testing.assert_allclose(a, b, rtol=0, atol=1e-9)
    # the reference's report methods read the LazyRows like arrays
    small_r, small_g = R.GeometricTrace(s1), GT(s2)
    for t in (small_r, small_g):
        t.rays_point((0, .7), nrays=7, distribution="meridional")
    assert str(small_g) == str(small_r)
    # item assignment writes through (the reference's own rays_given would use it)
    got.y[0, :, 1] = 7.
    assert np.all(got.y[0][:, 1] == 7.) and np.all(got._dev["y"].a[0, :got.nrays, 1] == 7.)


@pytest.mark.skipif(not ref_shim.available(), reason="reference tree not present")
def test_resident_rays_point_matches_reference():
    """ResidentTrace.rays_point on a reference System: host aiming by the
    reference, hexapolar rays "generated on the device" (here: the host
    restatement behind the fake engine) -- same trace as the reference's
    rays_point; other distributions go through system.aim"""
    warnings.simplefilter("ignore")
    R = ref_shim.load()
    from rayopt_b200 import ResidentTrace

    import aim_oracle

    class Eng(FakeResidentEngine):
        """the device generator replaced by its numpy restatement"""
        generated = 0

        def aim_count(self, spec, yp=None):
            return len(aim_oracle.generate(spec)[0])

        def aim_rays_into(self, spec, y_dst, u_dst, count, first=0, yp=None):
            y, u, _ = aim_oracle.generate(spec)
            y_dst.a[0, :count], u_dst.a[0, :count] = y[first:first + count], u[first:first + count]
            Eng.generated += 1
    s = R.System(**yaml.safe_load(systems_yaml.DOUBLE_GAUSS))
    s.update()
    s.paraxial.refocus()
    ref = R.GeometricTrace(s)
    ref.rays_point((0, .7), nrays=500, distribution="hexapolar", clip=True)
    got = ResidentTrace(s, engine=Eng())
    got.rays_point((0, .7), nrays=500, distribution="hexapolar", clip=True)
    assert got.nrays == ref.y.shape[1]
    np.testing.assert_allclose(got.y[0], ref.y[0], rtol=0, atol=1e-13)
    np.testing.assert_allclose(np.asarray(got.y), ref.y, rtol=0, atol=1e-11)
    assert np.array_equal(np.isnan(np.asarray(got.u)), np.isnan(ref.u))
    for dist, n, clip in (("square", 60, False), ("tee", 31, True), ("triangular", 200, True),
                          ("cross", 21, False), ("radau", 13, False)):
        ref.rays_point((0, 1.), nrays=n, distribution=dist, clip=clip)
        got.rays_point((0, 1.), nrays=n, distribution=dist, clip=clip)
        assert got.ref == ref.ref and got.nrays == ref.y.shape[1], dist
        assert np.array_equal(np.asarray(got.y), ref.y, equal_nan=True), dist
        assert np.array_equal(np.asarray(got.u), ref.u, equal_nan=True), dist
        assert np.array_equal(got.w, ref.w), dist
    assert Eng.generated == 5                     # radau went through system.aim on the host


@pytest.mark.skipif(not ref_shim.available(), reason="reference tree not present")
def test_propagate_many_equals_individual_propagates():
    """propagate_many: the Analysis pattern (fields x wavelengths of small
    bundles, analysis.py:266-280) in one batched call leaves every bound trace
    exactly as its own propagate would"""
    import rayopt_b200
    warnings.simplefilter("ignore")
    R = ref_shim.load()
    s = R.System(**yaml.safe_load(systems_yaml.COOKE))
    s.update()
    s.paraxial.refocus()
    GT = bind(R.GeometricTrace, engine=OracleEngine())
    ref_, yp, weight = R.utils.pupil_distribution("hexapolar", 150)
    refs, traces = [], []
    for hi in (1., .707, 0.):
        for wi in s.wavelengths:
            r = R.GeometricTrace(s)
            r.rays_point((0, hi), wi, nrays=150, distribution="hexapolar", clip=True)
            refs.append(r)
            t = GT(s)
            z, p = s.pupil((0, hi), l=wi)
            y, u = s.aim((0, hi), yp, z, p, filter=False)
            t.rays_given(y, u, wi, weight, ref_)
            traces.append(t)
    calls0 = OracleEngine.calls
    rayopt_b200.propagate_many(traces, clip=True)
    assert OracleEngine.calls == calls0 + 1
    for r, t in zip(refs, traces):
        for k in "yuit":
            assert np.array_equal(getattr(t, k), getattr(r, k), equal_nan=True), k
        assert np.array_equal(t.n, r.n) and np.array_equal(t.path, r.path)
