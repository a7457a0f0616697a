"""GPU parity tests (run with -m gpu on a B200): backend='cuda' through the C ABI vs
 (a) the committed outputs of the imported reference (tests/golden/ref_cases.npz),
 (b) the reference's own golden vectors (tests/golden/reference_goldens.npz),
 (c) the CPU oracle on fresh seeded inputs, and size-independent properties at larger sizes.
Tolerance (BASELINE.json north_star / SURVEY.md §8d): rtol = 1e-5, atol = 1e-5*max|ref| for fp64.
"""
import numpy as np
import pytest
from numpy.testing import assert_allclose

import cases
from conftest import assert_parity

pytestmark = pytest.mark.gpu
R64 = 1e-5

GLOBAL_CASES = [c for c in cases.CASES if c["k"] is None and c["name"] != "ok2d_hole_effect_small"]   # incl. geographic
KNN_CASES = [c for c in cases.CASES if c["k"] is not None]


@pytest.fixture(scope="module")
def pk():
    import pykrige_b200
    return pykrige_b200


def _run(pk, case):
    inp = cases.build_inputs(case)
    model = cases.make_model(pk, case, inp)
    z, ss = cases.run_model(model, case, inp, "cuda")
    return inp, z, ss


@pytest.mark.parametrize("case", GLOBAL_CASES, ids=[c["name"] for c in GLOBAL_CASES])
def test_global_cases_match_reference(pk, case, ref_cases):
    inp, z, ss = _run(pk, case)
    zr, sr = ref_cases[case["name"] + "/z"], ref_cases[case["name"] + "/ss"]
    assert z.shape == zr.shape
    if case["style"] == "masked":
        assert np.ma.is_masked(z) and np.ma.is_masked(ss)
        assert np.array_equal(np.ma.getmaskarray(z), inp["mask"])
        keep = ~inp["mask"]
        z, ss, zr, sr = np.ma.getdata(z)[keep], np.ma.getdata(ss)[keep], zr[keep], sr[keep]
    assert_parity(z, zr, R64, case["name"] + " z")
    assert_parity(ss, sr, R64, case["name"] + " ss")


@pytest.mark.parametrize("case", KNN_CASES, ids=[c["name"] for c in KNN_CASES])
def test_moving_window_cases_match_reference(pk, case, ref_cases):
    inp, z, ss = _run(pk, case)
    assert_parity(z, ref_cases[case["name"] + "/z"], R64, case["name"] + " z")
    assert_parity(ss, ref_cases[case["name"] + "/ss"], R64, case["name"] + " ss")


def test_kt3d_ok_golden(pk, ref_goldens):
    """tests/test_core.py:490-507 through backend='cuda'."""
    g = ref_goldens
    d = g["data"]
    ok = pk.OrdinaryKriging(d[:, 0], d[:, 1], d[:, 2], variogram_model="exponential",
                            variogram_parameters=[500.0, 3000.0, 0.0])
    z, ss = ok.execute("grid", g["ok_gridx"], g["ok_gridy"], backend="cuda")
    assert_allclose(z, g["ok_answer"], rtol=1e-6)


def test_kt3d_uk_golden(pk, ref_goldens):
    """tests/test_core.py:707-725 through backend='cuda'."""
    g = ref_goldens
    d = g["data"]
    uk = pk.UniversalKriging(d[:, 0], d[:, 1], d[:, 2], variogram_model="exponential",
                             variogram_parameters=[500.0, 3000.0, 0.0], drift_terms=["regional_linear"])
    z, ss = uk.execute("grid", g["uk_gridx"], g["uk_gridy"], backend="cuda")
    assert_allclose(z, g["uk_answer"], rtol=1e-6)


def test_kt3d_3d_golden(pk, ref_goldens):
    """tests/test_core.py:1957-2017 through backend='cuda' (global and k=10 moving window)."""
    g = ref_goldens
    d = g["data3d"]
    ax = np.arange(10.0)
    k3 = pk.OrdinaryKriging3D(d[:, 0], d[:, 1], d[:, 2], d[:, 3], variogram_model="linear",
                              variogram_parameters=[1.0, 0.1])
    k, ss = k3.execute("grid", ax, ax, ax, backend="cuda")
    assert_allclose(k, g["answer3d"][:, 0].reshape(10, 10, 10), rtol=1e-3, atol=1e-8)
    assert_allclose(ss, g["answer3d"][:, 1].reshape(10, 10, 10), rtol=1e-3, atol=1e-8)


def test_meuk_external_drift_golden(pk, ref_goldens):
    """tests/test_core.py:1479-1507 through backend='cuda': universal kriging with the external-Z drift sampled
    from the DEM raster (test3_dem.asc) against the MEUK answer grid (test3_answer.asc), at the reference's own
    tolerance. The raster is sampled at the prediction points on the device (kb200_set_device_drift)."""
    g = ref_goldens
    d = g["data"]
    uk = pk.UniversalKriging(d[:, 0], d[:, 1], d[:, 2], variogram_model="spherical",
                             variogram_parameters=[500.0, 3000.0, 0.0], anisotropy_scaling=1.0, anisotropy_angle=0.0,
                             drift_terms=["external_Z"], external_drift=g["dem"], external_drift_x=g["dem_x"],
                             external_drift_y=g["dem_y"])
    z, ss = uk.execute("grid", g["ext_gridx"], g["ext_gridy"], backend="cuda")
    assert z.shape == g["ext_answer"].shape
    assert_allclose(z, g["ext_answer"], rtol=1e-5, atol=1e-8)
    # a raster that does not cover the prediction domain is refused like uk.py:545-551
    with pytest.raises(ValueError):
        uk.execute("grid", g["ext_gridx"] + 1.0e6, g["ext_gridy"], backend="cuda")


def test_ucla_uk_single_point(pk):
    """tests/test_core.py:856-895 (lecture notes by N. Christou, UCLA): universal kriging of one point, and an
    exact hit on a data point."""
    data = np.array([[61.0, 139.0, 477.0], [63.0, 140.0, 696.0], [64.0, 129.0, 227.0], [68.0, 128.0, 646.0],
                     [71.0, 140.0, 606.0], [73.0, 141.0, 791.0], [75.0, 128.0, 783.0]])
    uk = pk.UniversalKriging(data[:, 0], data[:, 1], data[:, 2], variogram_model="exponential",
                             variogram_parameters=[10.0, 9.99, 0.0], drift_terms=["regional_linear"])
    z, ss = uk.execute("points", np.array([65.0]), np.array([137.0]), backend="cuda")
    assert z[0] == pytest.approx(567.54, rel=0.1)
    assert ss[0] == pytest.approx(9.044, rel=0.1)
    z, ss = uk.execute("points", np.array([61.0]), np.array([139.0]), backend="cuda")
    assert z[0] == pytest.approx(477.0, rel=1e-3)
    assert abs(ss[0]) < 1e-3


def test_device_drift_equals_host_columns(pk):
    """point_log and external_Z evaluated at the prediction points BY THE KERNEL (kb200_set_device_drift) against
    the same terms evaluated by host numpy and shipped as 'specified' columns — two independent routes to the
    same system (uk.py:884-900 column order). Covers grid / points / masked styles, float32 and float64x, an
    on-node / on-line query of the bilinear sampler and a raster with a DESCENDING axis (the reference's
    first->= / last-<= node rule then brackets with nodes 0 and n-1)."""
    xyz, val = cases.synth_data(777, 400, 2)
    ex, ey = np.linspace(-100.0, 1100.0, 49), np.linspace(-50.0, 1050.0, 37)
    EX, EY = np.meshgrid(ex, ey)
    raster = 30.0 + 0.02 * EX - 0.01 * EY + 5.0 * np.sin(EX / 170.0) * np.cos(EY / 230.0)
    wells = np.array([[250.0, 300.0, 1.5], [700.0, 650.0, -0.8]])
    kw = dict(variogram_model="exponential", variogram_parameters=[1.0, 300.0, 0.05])
    for flip in (False, True):
        ry, rz = (ey[::-1].copy(), raster[::-1].copy()) if flip else (ey, raster)
        uk = pk.UniversalKriging(xyz[:, 0], xyz[:, 1], val, drift_terms=["regional_linear", "point_log", "external_Z"],
                                 point_drift=wells, external_drift=rz, external_drift_x=ex, external_drift_y=ry,
                                 anisotropy_scaling=1.7, anisotropy_angle=25.0, **kw)
        # host twin: the same columns as 'specified' drift
        cols_d = [uk._point_log_column(w, uk.X_ADJUSTED, uk.Y_ADJUSTED) for w in range(2)] + [np.asarray(uk.z_scalars)]
        us = pk.UniversalKriging(xyz[:, 0], xyz[:, 1], val, drift_terms=["regional_linear", "specified"],
                                 specified_drift=cols_d, anisotropy_scaling=1.7, anisotropy_angle=25.0, **kw)

        def host_cols(px, py):
            from pykrige_b200.core import _adjust_for_anisotropy
            xa, ya = _adjust_for_anisotropy(np.vstack((px, py)).T, [uk.XCENTER, uk.YCENTER], [1.7], [25.0]).T
            return [uk._point_log_column(w, xa, ya) for w in range(2)] + [uk._calculate_data_point_zscalars(px, py)]

        gx, gy = np.linspace(0.0, 1000.0, 41), np.linspace(0.0, 1000.0, 29)       # hits raster nodes and lines
        GX, GY = np.meshgrid(gx, gy)
        spec = [c.reshape(GX.shape) for c in host_cols(GX.ravel(), GY.ravel())]
        for dt, R in (("float64", 1e-9), ("float64x", 1e-7), ("float32", 1e-2)):
            zd, sd = uk.execute("grid", gx, gy, backend="cuda", dtype=dt)
            zh, sh = us.execute("grid", gx, gy, backend="cuda", specified_drift_arrays=spec, dtype=dt)
            assert_parity(zd, zh, R, "device drift grid z %s flip=%s" % (dt, flip))
            assert_parity(sd, sh, R, "device drift grid ss %s flip=%s" % (dt, flip))
        rng = np.random.default_rng(3)
        px = np.concatenate([rng.uniform(0, 1000, 500), [ex[7], ex[9], 333.3, wells[0, 0]]])
        py = np.concatenate([rng.uniform(0, 1000, 500), [ey[5], 444.4, ey[11], wells[0, 1]]])   # node, lines, a well
        zd, sd = uk.execute("points", px, py, backend="cuda")
        zh, sh = us.execute("points", px, py, backend="cuda", specified_drift_arrays=host_cols(px, py))
        assert_parity(zd, zh, 1e-9, "device drift points z flip=%s" % flip)
        assert_parity(sd, sh, 1e-9, "device drift points ss flip=%s" % flip)
        mask = rng.uniform(size=GX.shape) < 0.4
        zd, sd = uk.execute("masked", gx, gy, mask=mask, backend="cuda")
        zh, sh = us.execute("masked", gx, gy, mask=mask, backend="cuda", specified_drift_arrays=spec)
        assert np.array_equal(np.ma.getmaskarray(zd), mask)
        assert_parity(np.ma.getdata(zd)[~mask], np.ma.getdata(zh)[~mask], 1e-9, "device drift masked z")
        assert_parity(np.ma.getdata(sd)[~mask], np.ma.getdata(sh)[~mask], 1e-9, "device drift masked ss")


def test_large_outputs_are_staged_in_chunks(pk):
    """> 2^20 prediction points travel back through the pinned two-buffer pipeline in several launches; the
    result must equal the same points kriged in small direct calls, bit for bit (global and moving window)."""
    xyz, val = cases.synth_data(12, 300, 2)
    ok = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="spherical", variogram_parameters=[1.0, 400.0, 0.05])
    gx, gy = np.linspace(0, 1000, 1500), np.linspace(0, 1000, 1700)            # 2.55e6 points: 3 staged chunks
    z, ss = ok.execute("grid", gx, gy, backend="cuda")
    h = ok._ensure_problem()
    for first in (0, (1 << 20) - 100, 2 * (1 << 20) - 50, z.size - 1000):
        za, sa = h.execute_grid(gx, gy, None, None, first, 1000)
        assert np.array_equal(za, z.ravel()[first:first + 1000]) and np.array_equal(sa, ss.ravel()[first:first + 1000])
    zk, sk = ok.execute("grid", gx, gy, backend="cuda", n_closest_points=8)
    hk = ok._ensure_problem("float64", knn=True)
    for first in (0, (1 << 20) - 100, z.size - 1000):
        za, sa = hk.execute_knn_grid(8, gx, gy, None, first, 1000)
        assert np.array_equal(za, zk.ravel()[first:first + 1000]) and np.array_equal(sa, sk.ravel()[first:first + 1000])
    px, py = np.tile(gx, 900), np.repeat(gy[:900], gx.size)                    # 1.35e6 explicit points
    zp, sp = ok.execute("points", px, py, backend="cuda")
    assert np.array_equal(zp, z.ravel()[:zp.size]) and np.array_equal(sp, ss.ravel()[:sp.size])
    # host-supplied drift columns (functional + specified) travel with their chunk: 1.2e6 points in two staged launches
    uk = pk.UniversalKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="spherical", variogram_parameters=[1.0, 400.0, 0.05],
                             drift_terms=["regional_linear", "functional", "specified"],
                             functional_drift=[lambda x, y: np.sin(x / 300.0)], specified_drift=[0.002 * xyz[:, 0] * xyz[:, 1] / 1000.0])
    gxu, gyu = gx[:1200], gy[:1000]
    GX, GY = np.meshgrid(gxu, gyu)
    spec = [0.002 * GX * GY / 1000.0]
    zu, su = uk.execute("grid", gxu, gyu, backend="cuda", specified_drift_arrays=spec)
    rng = np.random.default_rng(2)
    for r0 in (0, 873, 999):                                                     # rows across the chunk boundary at 2^20
        zr, sr = uk.execute("points", gxu, np.full(gxu.size, gyu[r0]), backend="cuda",
                            specified_drift_arrays=[spec[0][r0].copy()])
        assert np.array_equal(zr, zu[r0]) and np.array_equal(sr, su[r0])


def test_ok3d_equals_ok2d_on_a_plane(pk, ref_goldens):
    """tests/test_core.py:1914-1956: 3-D kriging with z == 0 reproduces the 2-D KT3D_H2O answer."""
    g = ref_goldens
    d = g["data"]
    k3 = pk.OrdinaryKriging3D(d[:, 0], d[:, 1], np.zeros(d.shape[0]), d[:, 2], variogram_model="exponential",
                              variogram_parameters=[500.0, 3000.0, 0.0])
    k, ss = k3.execute("grid", g["ok_gridx"], g["ok_gridy"], np.array([0.0]), backend="cuda")
    assert_allclose(np.squeeze(k), g["ok_answer"], rtol=1e-6)


def test_exact_hits_interpolate(pk):
    """tests/test_core.py:1510-1836: at data locations z == data and sigma^2 == 0 when exact_values."""
    xyz, val = cases.synth_data(77, 300, 2)
    ok = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential",
                            variogram_parameters=[1.0, 300.0, 0.05])
    z, ss = ok.execute("points", xyz[:40, 0], xyz[:40, 1], backend="cuda")
    assert_allclose(z, val[:40], rtol=1e-9)
    assert np.max(np.abs(ss)) < 1e-9
    ok2 = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential",
                             variogram_parameters=[1.0, 300.0, 0.05], exact_values=False)
    z2, ss2 = ok2.execute("points", xyz[:40, 0], xyz[:40, 1], backend="cuda")
    assert np.all(ss2 > 1e-3)   # nugget smoothing: no longer exact (tests/test_core.py:430-487)


def test_full_size_properties_cfg2(pk):
    """BASELINE config 2 data size (N=5000, exponential) on a slab of the 1000x1000 grid:
    size-independent checks — linearity of z in the data values, invariance of sigma^2 to the values,
    shard concatenation == single call bit-for-bit, oracle agreement on a subsample."""
    from oracle import krige_oracle as ko
    xyz, val = cases.synth_data(1002, 5000, 2)
    gx = np.linspace(0.0, 1000.0, 1000)
    gy = np.linspace(0.0, 1000.0, 1000)[:8]           # 8000 points of the grid
    params = [1.0, 300.0, 0.05]
    ok = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential", variogram_parameters=params)
    z, ss = ok.execute("grid", gx, gy, backend="cuda")
    # linearity: krige(a*Z + b) == a*krige(Z) + b ; sigma^2 unchanged
    ok2 = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], 3.0 * val - 7.0, variogram_model="exponential",
                             variogram_parameters=params)
    z2, ss2 = ok2.execute("grid", gx, gy, backend="cuda")
    assert_allclose(z2, 3.0 * z - 7.0, rtol=1e-9)
    assert_allclose(ss2, ss, rtol=1e-12, atol=1e-14)
    # sharding determinism: two half slices concatenated == one call, bit for bit
    h = ok._ensure_problem()
    za, sa = h.execute_grid(gx, gy, None, None, 0, 3000)
    zb, sb = h.execute_grid(gx, gy, None, None, 3000, 5000)
    assert np.array_equal(np.concatenate([za, zb]), z.ravel())
    assert np.array_equal(np.concatenate([sa, sb]), ss.ravel())
    # oracle (5001^2 inverse, the reference's formulation) on 4096 grid points + 16 exact hits (SURVEY.md 8d)
    rng = np.random.default_rng(5)
    pick = rng.choice(z.size, 4096, replace=False)
    G = ko.grid_points([gx, gy])
    pts = np.vstack([G[pick], xyz[:16]])
    zo, so = ko.krige_chunked(xyz, val, "exponential", ko.stored_parameters("exponential", params), pts)
    zc, sc = ok.execute("points", pts[:, 0], pts[:, 1], backend="cuda")
    assert_parity(zc, zo, R64, "cfg2 z")
    assert_parity(sc, so, R64, "cfg2 ss")
    assert_allclose(z.ravel()[pick], zc[:4096], rtol=1e-12)
    # the tensor-core arithmetics against the ORACLE (not against the fp64 CUDA path)
    for dt, R in (("float64x", R64), ("float64x5", R64), ("float64x4", R64), ("float32", 1e-2)):
        zt, st = ok.execute("points", pts[:, 0], pts[:, 1], backend="cuda", dtype=dt)
        assert_parity(zt, zo, R, "cfg2 %s z vs oracle" % dt)
        assert_parity(st, so, R, "cfg2 %s ss vs oracle" % dt)


def test_indefinite_variogram_takes_general_path(pk, ref_cases):
    """hole-effect is not conditionally negative definite in 2-D on dense scatter: the covariance-form
    Cholesky fails and the general (Gauss-Jordan + quadratic form) path must reproduce the reference's
    LU-based numbers (the oracle inverts the same indefinite matrix, ok.py:663)."""
    from oracle import krige_oracle as ko
    xyz, val = cases.synth_data(9, 600, 2)
    params = [1.0, 300.0, 0.05]
    ok = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="hole-effect", variogram_parameters=params)
    pts = cases.synth_points(9, 300, 2, xyz)
    z, ss = ok.execute("points", pts[:, 0], pts[:, 1], backend="cuda")
    zo, so = ko.krige(xyz, val, "hole-effect", ko.stored_parameters("hole-effect", params), pts)
    assert_parity(z, zo, R64, "hole-effect z")
    assert_parity(ss, so, R64, "hole-effect ss")
    # universal kriging through the same fallback
    uk = pk.UniversalKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="hole-effect", variogram_parameters=params,
                             drift_terms=["regional_linear"])
    z, ss = uk.execute("points", pts[:, 0], pts[:, 1], backend="cuda")
    zo, so = ko.krige(xyz, val, "hole-effect", ko.stored_parameters("hole-effect", params), pts, regional_linear=True)
    assert_parity(z, zo, R64, "hole-effect uk z")
    assert_parity(ss, so, R64, "hole-effect uk ss")
    # the small committed reference case
    case = cases.CASE_BY_NAME["ok2d_hole_effect_small"]
    inp, z, ss = _run(pk, case)
    assert_parity(z, ref_cases[case["name"] + "/z"], R64, "hole small z")
    assert_parity(ss, ref_cases[case["name"] + "/ss"], R64, "hole small ss")
    with pytest.raises(NotImplementedError):
        ok.execute("points", pts[:4, 0], pts[:4, 1], backend="cuda", dtype="float32")


def test_blocked_general_inverse_matches_scalar_form_and_oracle(pk, monkeypatch):
    """The general path's inverse is a blocked Gauss-Jordan (cooperative panel kernel + DMMA rank-64 updates). At a
    size with many panels (N = 1900 -> 30 panels, rows dealt over the whole grid) it must reproduce the oracle's
    LU-based numbers (ok.py:663) and the column-at-a-time form of the same elimination (KB200_GJ=scalar), for OK
    and for UK; redundant points must still be reported as singular, not inverted into noise."""
    from oracle import krige_oracle as ko
    xyz, val = cases.synth_data(21, 1900, 2)
    params = [1.0, 250.0, 0.02]
    pts = cases.synth_points(21, 500, 2, xyz)
    sp = ko.stored_parameters("hole-effect", params)
    zo, so = ko.krige(xyz, val, "hole-effect", sp, pts)
    zu, su = ko.krige(xyz, val, "hole-effect", sp, pts, regional_linear=True)
    out, launches = {}, {}
    for mode in ("blocked", "scalar"):
        monkeypatch.setenv("KB200_GJ", mode)
        ok = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="hole-effect", variogram_parameters=params)
        z, ss = ok.execute("points", pts[:, 0], pts[:, 1], backend="cuda")
        launches[mode] = ok._kb_handle.timings()["launches"]
        assert_parity(z, zo, R64, "blocked GJ z (scalar=%s)" % mode)
        assert_parity(ss, so, R64, "blocked GJ ss (scalar=%s)" % mode)
        out[mode] = (z, ss)
        uk = pk.UniversalKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="hole-effect", variogram_parameters=params,
                                 drift_terms=["regional_linear"])
        z, ss = uk.execute("points", pts[:, 0], pts[:, 1], backend="cuda")
        assert_parity(z, zu, R64, "blocked GJ uk z (scalar=%s)" % mode)
        assert_parity(ss, su, R64, "blocked GJ uk ss (scalar=%s)" % mode)
    assert launches["blocked"] + 3000 < launches["scalar"]          # 3 launches per 64 columns instead of 2 per column
    assert_parity(out["blocked"][0], out["scalar"][0], 1e-7, "blocked vs scalar z")
    assert_parity(out["blocked"][1], out["scalar"][1], 1e-7, "blocked vs scalar ss")
    monkeypatch.setenv("KB200_GJ", "blocked")
    dup = np.vstack([xyz[:700], xyz[:4]])
    okd = pk.OrdinaryKriging(dup[:, 0], dup[:, 1], np.concatenate([val[:700], val[:4]]), variogram_model="hole-effect",
                             variogram_parameters=[1.0, 250.0, 0.0])
    with pytest.raises(np.linalg.LinAlgError):
        okd.execute("points", [10.0], [20.0], backend="cuda")


def test_singular_system_is_reported(pk):
    """Duplicate data points with a zero nugget make the kriging matrix exactly singular: the reference's
    scipy.linalg.inv raises LinAlgError; so must backend='cuda' (never silent numbers)."""
    xyz, val = cases.synth_data(10, 50, 2)
    xyz = np.vstack([xyz, xyz[:3]])
    val = np.concatenate([val, val[:3]])
    ok = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="spherical",
                            variogram_parameters=[1.0, 300.0, 0.0])
    with pytest.raises(np.linalg.LinAlgError):
        ok.execute("points", [10.0], [20.0], backend="cuda")


def test_edge_sizes(pk):
    """Empty and tiny inputs: zero prediction points, one prediction point, two data points."""
    xyz, val = cases.synth_data(12, 40, 2)
    ok = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="linear", variogram_parameters=[0.01, 0.1])
    z, ss = ok.execute("points", np.zeros(0), np.zeros(0), backend="cuda")
    assert z.shape == (0,) and ss.shape == (0,)
    z, ss = ok.execute("grid", [500.0], [500.0], backend="cuda")
    assert z.shape == (1, 1)
    from oracle import krige_oracle as ko
    two = pk.OrdinaryKriging([0.0, 10.0], [0.0, 5.0], [1.0, 3.0], variogram_model="linear", variogram_parameters=[0.5, 0.1])
    z, ss = two.execute("points", [2.0, 7.0], [1.0, 4.0], backend="cuda")
    zo, so = ko.krige(np.array([[0.0, 0.0], [10.0, 5.0]]), np.array([1.0, 3.0]), "linear", [0.5, 0.1],
                      np.array([[2.0, 1.0], [7.0, 4.0]]))
    assert_allclose(z, zo, rtol=1e-10)
    assert_allclose(ss, so, rtol=1e-10)


def test_custom_variogram_runs_on_device(pk):
    """A 'custom' callable (which the reference's native backend refuses, variogram_models.pyx:20-21) is
    tabulated by the host and interpolated on the device; a linear callable must agree with the built-in
    linear model, also far outside the data (the tabulated range follows the prediction points)."""
    xyz, val = cases.synth_data(3, 300, 2)
    fn = lambda m, d: m[0] * d + m[1]
    oc = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="custom", variogram_parameters=[0.004, 0.05],
                            variogram_function=fn)
    ob = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="linear", variogram_parameters=[0.004, 0.05])
    pts = cases.synth_points(3, 200, 2, xyz)
    far = np.array([[5000.0, -3000.0], [-20000.0, 40000.0]])
    for P in (pts, far, pts):                               # growing, then re-used tabulated range
        zc, sc = oc.execute("points", P[:, 0], P[:, 1], backend="cuda")
        zb, sb = ob.execute("points", P[:, 0], P[:, 1], backend="cuda")
        assert_parity(zc, zb, 1e-8, "custom linear z")
        assert_parity(sc, sb, 1e-8, "custom linear ss")
    with pytest.raises(ValueError):                         # not finite at d = 0
        bad = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="custom", variogram_parameters=[1.0],
                                 variogram_function=lambda m, d: m[0] * np.log(d))
        bad.execute("points", [1.0], [2.0], backend="cuda")


def test_intermediates_match_scipy(pk):
    """White-box: the device Cholesky factor and its inverse agree with scipy on the same matrix."""
    import scipy.linalg as sl
    from scipy.spatial.distance import cdist
    from oracle import krige_oracle as ko
    xyz, val = cases.synth_data(11, 700, 2)
    ok = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="spherical",
                            variogram_parameters=[1.0, 400.0, 0.05])
    h = ok._ensure_problem()
    n, n_pad = 700, 768
    L = h.debug_fetch(1, n_pad * n_pad).reshape(n_pad, n_pad)[:n, :n]
    W = h.debug_fetch(2, n_pad * n_pad).reshape(n_pad, n_pad)[:n, :n]
    c0 = 1.0
    C = c0 - ko.variogram("spherical", [0.95, 400.0, 0.05], cdist(xyz, xyz))
    np.fill_diagonal(C, c0)
    Lr = sl.cholesky(C, lower=True)
    assert_allclose(np.tril(L), Lr, rtol=1e-9, atol=1e-12)
    assert_allclose(np.tril(W), sl.solve_triangular(Lr, np.eye(n), lower=True), rtol=1e-7, atol=1e-10)


# ---- fp32 device math (tcgen05 kind::tf32, 3xTF32 split): tolerance rtol = 1e-2 (north_star) ----------
R32 = 1e-2
F32_CASES = [c for c in GLOBAL_CASES if c["name"] in (
    "cfg1_ok2d_n100_grid50", "ok2d_exponential_aniso", "ok2d_gaussian_aniso", "ok2d_spherical_aniso",
    "ok2d_linear_aniso", "ok2d_masked", "cfg2r_ok2d_n1000", "cfg3r_ok3d_n800", "cfg4r_uk2d_n1000",
    "uk2d_functional", "uk2d_all_grid", "uk3d_reglin", "ok3d_grid", "geo_ok_points")]


@pytest.mark.parametrize("case", F32_CASES, ids=[c["name"] for c in F32_CASES])
def test_fp32_cases_match_reference(pk, case, ref_cases):
    inp = cases.build_inputs(case)
    model = cases.make_model(pk, case, inp)
    style = case["style"]
    kw = dict(backend="cuda", dtype="float32")
    if case["n_specified"]:
        kw["specified_drift_arrays"] = [np.array(a) for a in inp["spec_pts"]]
    args = [inp["points"][:, c] for c in range(case["dim"])] if style == "points" else list(inp["axes"])
    if style == "masked":
        kw["mask"] = inp["mask"]
    z, ss = model.execute(style, *args, **kw)
    zr, sr = ref_cases[case["name"] + "/z"], ref_cases[case["name"] + "/ss"]
    if style == "masked":
        keep = ~inp["mask"]
        z, ss, zr, sr = np.ma.getdata(z)[keep], np.ma.getdata(ss)[keep], zr[keep], sr[keep]
    assert_parity(z, zr, R32, case["name"] + " z fp32")
    assert_parity(ss, sr, R32, case["name"] + " ss fp32")
    # 3xTF32 keeps fp32-class accuracy: far inside the 1e-2 budget
    assert np.max(np.abs(np.ravel(z) - np.ravel(zr))) <= 2e-4 * np.max(np.abs(zr))
    assert np.max(np.abs(np.ravel(ss) - np.ravel(sr))) <= 2e-4 * np.max(np.abs(sr))


def test_moving_window_goldens_and_fallback(pk, ref_goldens):
    """tests/test_core.py:1992-2017: OK3D moving window k=10 reproduces the KT3D answer; and a variogram
    that is not positive definite locally (hole-effect) goes through the pivoted-LU solver and still
    matches the oracle's scipy.linalg.solve."""
    from oracle import krige_oracle as ko
    g = ref_goldens
    d = g["data3d"]
    ax = np.arange(10.0)
    k3 = pk.OrdinaryKriging3D(d[:, 0], d[:, 1], d[:, 2], d[:, 3], variogram_model="linear",
                              variogram_parameters=[1.0, 0.1])
    k, ss = k3.execute("grid", ax, ax, ax, backend="cuda", n_closest_points=10)
    assert_allclose(k, g["answer3d"][:, 0].reshape(10, 10, 10), rtol=1e-3)
    assert_allclose(ss, g["answer3d"][:, 1].reshape(10, 10, 10), rtol=1e-3)
    xyz, val = cases.synth_data(21, 800, 2)
    params = [1.0, 120.0, 0.02]
    ok = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="hole-effect", variogram_parameters=params)
    pts = cases.synth_points(21, 200, 2, xyz)
    z, ss = ok.execute("points", pts[:, 0], pts[:, 1], backend="cuda", n_closest_points=24)
    zo, so = ko.krige(xyz, val, "hole-effect", ko.stored_parameters("hole-effect", params), pts, n_closest_points=24)
    assert_parity(z, zo, R64, "knn hole-effect z")
    assert_parity(ss, so, R64, "knn hole-effect ss")
    # k > 128 uses the LU solver directly
    z, ss = ok.execute("points", pts[:20, 0], pts[:20, 1], backend="cuda", n_closest_points=130)
    zo, so = ko.krige(xyz, val, "hole-effect", ko.stored_parameters("hole-effect", params), pts[:20], n_closest_points=130)
    assert_parity(z, zo, 1e-4, "knn k130 z")
    assert_parity(ss, so, 1e-4, "knn k130 ss")


def test_sklearn_krige_wrapper_routes_to_cuda(pk):
    """The caller side (compat.py:251-291): Krige.fit / predict / GridSearchCV drive execute(style='points',
    backend='cuda', n_closest_points=...) and reproduce the oracle's moving-window numbers."""
    pytest.importorskip("sklearn")
    from sklearn.model_selection import GridSearchCV
    from pykrige_b200.compat import Krige
    from oracle import krige_oracle as ko
    xyz, val = cases.synth_data(31, 160, 2)
    est = Krige(method="ordinary", variogram_model="exponential", variogram_parameters=[1.0, 300.0, 0.05],
                n_closest_points=12).fit(xyz[:120], val[:120])
    pred = est.predict(xyz[120:])
    zo, _ = ko.krige(xyz[:120], val[:120], "exponential", [0.95, 300.0, 0.05], xyz[120:], n_closest_points=12)
    assert_allclose(pred, zo, rtol=1e-8)
    search = GridSearchCV(Krige(variogram_parameters=None), {"method": ["ordinary", "universal"],
                                                             "variogram_model": ["linear", "spherical"]}, cv=3)
    search.fit(xyz, val)
    assert set(search.best_params_) == {"method", "variogram_model"}
    x3, v3 = cases.synth_data(32, 90, 3)
    est3 = Krige(method="universal3d", variogram_model="linear", variogram_parameters=[0.01, 0.1],
                 drift_terms=["regional_linear"]).fit(x3[:70], v3[:70])
    z3 = est3.predict(x3[70:])
    zo3, _ = ko.krige(x3[:70], v3[:70], "linear", [0.01, 0.1], x3[70:], regional_linear=True)
    assert_allclose(z3, zo3, rtol=1e-7)


# ---- dtype='float64x': fp64-class contraction on the INT8 tensor cores (exact slice products) ---------
F64X_CASES = [c for c in GLOBAL_CASES if c["name"] in (
    "cfg1_ok2d_n100_grid50", "ok2d_exponential_aniso", "ok2d_linear_aniso", "ok2d_power_aniso", "ok2d_masked",
    "cfg2r_ok2d_n1000", "cfg3r_ok3d_n800", "cfg4r_uk2d_n1000", "uk2d_all_grid", "uk3d_spec_func", "geo_ok_points")]


@pytest.mark.parametrize("case", F64X_CASES, ids=[c["name"] for c in F64X_CASES])
def test_float64x_cases_match_reference(pk, case, ref_cases):
    inp = cases.build_inputs(case)
    model = cases.make_model(pk, case, inp)
    style = case["style"]
    kw = dict(backend="cuda", dtype="float64x")
    if case["n_specified"]:
        kw["specified_drift_arrays"] = [np.array(a) for a in inp["spec_pts"]]
    args = [inp["points"][:, c] for c in range(case["dim"])] if style == "points" else list(inp["axes"])
    if style == "masked":
        kw["mask"] = inp["mask"]
    z, ss = model.execute(style, *args, **kw)
    zr, sr = ref_cases[case["name"] + "/z"], ref_cases[case["name"] + "/ss"]
    if style == "masked":
        keep = ~inp["mask"]
        z, ss, zr, sr = np.ma.getdata(z)[keep], np.ma.getdata(ss)[keep], zr[keep], sr[keep]
    assert_parity(z, zr, R64, case["name"] + " z float64x")        # the fp64 tolerance, 1e-5
    assert_parity(ss, sr, R64, case["name"] + " ss float64x")
    # and fp64-class in fact: within 1e-8 of the reference
    assert np.max(np.abs(np.ravel(z) - np.ravel(zr))) <= 1e-8 * np.max(np.abs(zr))
    assert np.max(np.abs(np.ravel(ss) - np.ravel(sr))) <= 1e-8 * np.max(np.abs(sr))


# ---- constructor side on the device (SURVEY.md §8f next-2): csrc/variogram.cu ----------------------
def _list_params(case):
    """stored -> list form of the constructors ([FULL sill, range, nugget], core.py:345-357)."""
    p = list(case["params"])
    if case["model"] in ("gaussian", "spherical", "exponential", "hole-effect"):
        return [p[0] + p[2], p[1], p[2]]
    return p


@pytest.mark.parametrize("case", cases.VARIOGRAM_CASES, ids=[c["name"] for c in cases.VARIOGRAM_CASES])
def test_device_experimental_variogram_matches_reference(pk, case, ref_ctor):
    """kb200_experimental_variogram vs core._initialize_variogram_model of the imported reference. The
    pair distances are computed in pdist's operation order, so bin assignment is identical; only the
    order of the per-bin sums differs (rtol 1e-10)."""
    from pykrige_b200 import core
    X, y = cases.build_ctor_inputs(case)
    lags, semi = core._experimental_variogram(X, y, case["nlags"], coordinates_type=case["coordinates_type"],
                                              device=True)
    assert lags.shape == ref_ctor[case["name"] + "/lags"].shape
    assert_allclose(lags, ref_ctor[case["name"] + "/lags"], rtol=1e-10)
    assert_allclose(semi, ref_ctor[case["name"] + "/semi"], rtol=1e-10)


def test_device_experimental_variogram_large_vs_host(pk):
    """N = 6000 (1.8e7 pairs): device vs the host mirror, counts exact, and run-to-run determinism of
    the private-bin kernel."""
    from pykrige_b200 import core, _cabi
    rng = np.random.default_rng(77)
    X = rng.uniform(0.0, 1000.0, (6000, 3))
    y = rng.normal(0.0, 1.0, 6000) + 0.01 * X[:, 0]
    h = _cabi.aux_handle()
    cnt, sd, sg, dmin, dmax = h.experimental_variogram(X, y, 12)
    cnt2, sd2, sg2, _, _ = h.experimental_variogram(X, y, 12)
    assert np.array_equal(sd, sd2) and np.array_equal(sg, sg2) and np.array_equal(cnt, cnt2)
    assert cnt.sum() == 6000 * 5999 // 2
    lags_h, semi_h = core._experimental_variogram(X, y, 12, device=False)
    keep = cnt > 0
    assert_allclose(sd[keep] / cnt[keep], lags_h, rtol=1e-10)
    assert_allclose(sg[keep] / cnt[keep], semi_h, rtol=1e-10)
    with pytest.raises(ValueError):
        h.experimental_variogram(X[:1], y[:1], 6)
    with pytest.raises(ValueError):
        h.experimental_variogram(X, y, 0)


def _stats_model(pk, case, X, y, **kw):
    params = _list_params(case)
    if case["dim"] == 3:
        return pk.OrdinaryKriging3D(X[:, 0], X[:, 1], X[:, 2], y, variogram_model=case["model"],
                                    variogram_parameters=params, **kw)
    return pk.OrdinaryKriging(X[:, 0], X[:, 1], y, variogram_model=case["model"], variogram_parameters=params,
                              coordinates_type=case["coordinates_type"], **kw)


@pytest.mark.parametrize("case", cases.STATS_CASES, ids=[c["name"] for c in cases.STATS_CASES])
def test_device_statistics_match_reference(pk, case, ref_ctor):
    """kb200_statistics (residuals from ONE Cholesky factor) vs core._find_statistics of the imported
    reference (N growing solves), through the class attributes delta / sigma / epsilon / Q1 / Q2 / cR."""
    from pykrige_b200 import core
    X, y = cases.build_ctor_inputs(case)
    m = _stats_model(pk, case, X, y)
    res = m._device_statistics()
    assert res is not None, "device route not taken"
    delta, sigma, epsilon = res
    dr, sr, er = (ref_ctor[case["name"] + "/" + k] for k in ("delta", "sigma", "epsilon"))
    assert delta.shape == dr.shape
    assert_allclose(delta, dr, rtol=1e-6, atol=1e-6 * np.abs(dr).max())
    assert_allclose(sigma, sr, rtol=1e-6)
    assert_allclose(epsilon, er, rtol=1e-6, atol=1e-6 * np.abs(er).max())
    if case["dim"] == 3:
        assert_allclose([m.Q1, m.Q2, m.cR], [core.calcQ1(er), core.calcQ2(er), core.calc_cR(core.calcQ2(er), sr)],
                        rtol=1e-6)


def test_device_statistics_reuse_factor_and_anisotropy(pk):
    """After a global execute() the statistics come from the factor already on the handle (no second
    factorisation); anisotropy goes through the adjusted coordinates like ok.py:361-368."""
    from oracle import krige_oracle as ko
    rng = np.random.default_rng(5)
    x, y = rng.uniform(0, 1000, 150), rng.uniform(0, 1000, 150)
    v = 3.0 + np.sin(x / 120.0) + rng.normal(0, 0.1, 150)
    m = pk.OrdinaryKriging(x, y, v, variogram_model="spherical", variogram_parameters=[1.2, 350.0, 0.1],
                           anisotropy_scaling=2.5, anisotropy_angle=35.0)
    m.execute("grid", np.linspace(0, 1000, 20), np.linspace(0, 1000, 20), backend="cuda")
    t0 = m._cuda_handle().timings()["launches"]
    res = m._device_statistics()
    assert m._cuda_handle().timings()["launches"] - t0 <= 2
    X = np.vstack((m.X_ADJUSTED, m.Y_ADJUSTED)).T
    d, s, e = ko.find_statistics(X, v, "spherical", [1.1, 350.0, 0.1])
    assert_allclose(res[0], d, rtol=1e-6, atol=1e-6 * np.abs(d).max())
    assert_allclose(res[1], s, rtol=1e-6)


def test_device_statistics_large_vs_oracle_subsample(pk):
    """N = 3000: the reference needs 3000 growing solves; check a few indices against core._krige's
    restatement and that UK (drift columns present) reads the same ordinary-kriging residuals."""
    from oracle import krige_oracle as ko
    xyz, val = cases.synth_data(808, 3000, 2)
    params = [1.0, 300.0, 0.05]
    ok = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential", variogram_parameters=params)
    h = ok._ensure_problem("float64")
    delta, sigma = h.statistics(3000)
    stored = ko.stored_parameters("exponential", params)
    for i in (1, 2, 17, 500, 1999, 2999):
        k, ss = ko.krige_one(xyz[:i], val[:i], xyz[i], "exponential", stored)
        assert_allclose(delta[i], val[i] - k, rtol=1e-6, atol=1e-8)
        assert_allclose(sigma[i], np.sqrt(ss), rtol=1e-6)
    assert delta[0] == 0.0 and sigma[0] == 0.0
    uk = pk.UniversalKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential", variogram_parameters=params,
                             drift_terms=["regional_linear"])
    d2, s2 = uk._ensure_problem("float64").statistics(3000)
    assert_allclose(d2, delta, rtol=1e-9, atol=1e-12)
    assert_allclose(s2, sigma, rtol=1e-9)


def test_device_statistics_unsupported_routes(pk):
    """Indefinite covariance form (general fallback) and kNN-only handles have no factor to read:
    the C ABI says so and the class falls back to the reference's host loop."""
    from pykrige_b200 import _cabi
    xyz, val = cases.synth_data(9, 600, 2)
    m = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="hole-effect",
                           variogram_parameters=[1.0, 300.0, 0.05])
    h = m._ensure_problem("float64")
    with pytest.raises(NotImplementedError):
        h.statistics(600)
    assert m._device_statistics() is None
    m._stats_state = "lazy"
    assert m.epsilon is not None and np.all(np.isfinite(m.epsilon))      # host loop of core.py:759-836
    hk = m._ensure_problem("float64", knn=True)
    with pytest.raises(_cabi.KrigeB200Error):
        hk.statistics(600)


# ---- pseudo_inv=True on the device (SURVEY.md §8f next-4): csrc/pinv.cu -------------------------------
@pytest.mark.parametrize("case", cases.PINV_CASES, ids=[c["name"] for c in cases.PINV_CASES])
def test_pseudo_inverse_cases_match_reference(pk, case, ref_pinv):
    """Redundant data points make the kriging matrix singular; the Jacobi-SVD pseudo-inverse must give the
    reference's scipy.linalg.pinv / pinvh numbers (both z and sigma^2)."""
    inp, z, ss = _run(pk, case)
    zr, sr = ref_pinv[case["name"] + "/z"], ref_pinv[case["name"] + "/ss"]
    assert z.shape == zr.shape
    assert_parity(np.asarray(z).ravel(), zr.ravel(), R64, "pinv z")
    assert_parity(np.asarray(ss).ravel(), sr.ravel(), R64, "pinv ss")


@pytest.mark.parametrize("ptype", ["pinv", "pinvh"])
def test_pseudo_inverse_known_answers(pk, ptype):
    """tests/test_core.py:2913-2949 (test_pseudo_2d / test_pseudo_3d) for all four classes."""
    data = np.array([[0.0, 0.0, 1.0], [0.0, 0.0, 3.0], [1.0, 0.0, 6.0]])
    for cls in (pk.OrdinaryKriging, pk.UniversalKriging):
        m = cls(data[:, 0], data[:, 1], data[:, 2], variogram_parameters=[1.0, 0.0], pseudo_inv=True,
                pseudo_inv_type=ptype)
        z1, ss1 = m.execute("points", 0.0, 0.0, backend="cuda")
        assert np.isclose(z1.item(), 2.0)
    d3 = np.array([[0.0, 0.0, 0.0, 1.0], [0.0, 0.0, 0.0, 3.0], [1.0, 0.0, 0.0, 6.0]])
    for cls in (pk.OrdinaryKriging3D, pk.UniversalKriging3D):
        m = cls(d3[:, 0], d3[:, 1], d3[:, 2], d3[:, 3], variogram_parameters=[1.0, 0.0], pseudo_inv=True,
                pseudo_inv_type=ptype)
        z1, ss1 = m.execute("points", 0.0, 0.0, 0.0, backend="cuda")
        assert np.isclose(z1.item(), 2.0)
    # without the pseudo-inverse the same data is singular (what scipy.linalg.inv raises)
    m = pk.OrdinaryKriging(data[:, 0], data[:, 1], data[:, 2], variogram_parameters=[1.0, 0.0])
    with pytest.raises(np.linalg.LinAlgError):
        m.execute("points", 0.0, 0.0, backend="cuda")


def test_pseudo_inverse_medium_size_and_routes(pk):
    """N = 700 with 20 redundant points vs the oracle; fp32 is refused; the moving window ignores the
    flag like the reference (ok.py:753)."""
    from oracle import krige_oracle as ko
    xyz, val = cases.synth_data(4242, 700, 2)
    for q in range(20):
        xyz[699 - q] = xyz[2 * q]
    params = [1.0, 250.0, 0.0]
    pts = cases.synth_points(4242, 500, 2, xyz)
    m = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential", variogram_parameters=params,
                           pseudo_inv=True)
    z, ss = m.execute("points", pts[:, 0], pts[:, 1], backend="cuda")
    zo, so = ko.krige(xyz, val, "exponential", ko.stored_parameters("exponential", params), pts, pseudo_inv="pinv")
    assert_parity(z, zo, R64, "pinv700 z")
    assert_parity(ss, so, R64, "pinv700 ss")
    with pytest.raises(NotImplementedError):
        m.execute("points", pts[:, 0], pts[:, 1], backend="cuda", dtype="float32")
    xyz2, val2 = cases.synth_data(4243, 400, 2)
    mk = pk.OrdinaryKriging(xyz2[:, 0], xyz2[:, 1], val2, variogram_model="exponential",
                            variogram_parameters=[1.0, 250.0, 0.05], pseudo_inv=True)
    zk, sk = mk.execute("points", pts[:, 0], pts[:, 1], backend="cuda", n_closest_points=8)
    zko, sko = ko.krige(xyz2, val2, "exponential", ko.stored_parameters("exponential", [1.0, 250.0, 0.05]), pts,
                        n_closest_points=8)
    assert_parity(zk, zko, R64, "pinv knn z")
    assert_parity(sk, sko, R64, "pinv knn ss")


# ---- whole-chain scenarios on the reference's own fixtures (fitted variograms) ------------------------
@pytest.mark.parametrize("sc", cases.SCENARIOS, ids=[s["name"] for s in cases.SCENARIOS])
def test_whole_chain_scenarios_match_reference(pk, sc, ref_scenarios, ref_goldens):
    """Constructor (device binning + least-squares fit) -> execute(backend='cuda') -> statistics against the
    imported reference run the same way (tests/test_core.py:565-666, 1020-1067, 1219-1255, 2205-2353 are the
    scenarios these replay). The three-drift case is exactly determined by its drift terms (5 points, 5
    constraints; the reference's own matrix has rcond 2e-33) — like the reference's test it is checked for
    shape and finiteness only."""
    data, args, kw = cases.scenario_inputs(sc, ref_goldens["data"])
    m = cases.scenario_model(pk, sc, data)
    z, ss = m.execute(sc["style"], *args, backend="cuda", **kw)
    zr, sr = ref_scenarios[sc["name"] + "/z"], ref_scenarios[sc["name"] + "/ss"]
    assert z.shape == zr.shape and ss.shape == sr.shape
    if sc["style"] == "masked":
        assert np.ma.is_masked(z)
        keep = ~np.ma.getmaskarray(z)
        z, ss, zr, sr = np.ma.getdata(z)[keep], np.ma.getdata(ss)[keep], zr[keep], sr[keep]
    if sc.get("three_drifts"):
        assert np.all(np.isfinite(z)) and np.all(np.isfinite(ss))
        return
    assert_parity(np.ravel(z), np.ravel(zr), R64, sc["name"] + " z")
    assert_parity(np.ravel(ss), np.ravel(sr), R64, sc["name"] + " ss")
    if sc.get("stats"):
        Q = ref_scenarios[sc["name"] + "/Q"]
        assert_allclose([m.Q1, m.Q2, m.cR], Q, rtol=1e-5)
        assert_allclose(m.epsilon, ref_scenarios[sc["name"] + "/epsilon"], rtol=1e-5,
                        atol=1e-5 * np.abs(ref_scenarios[sc["name"] + "/epsilon"]).max())


# ---- straight against the reference's compiled native code (outputs stored by golden/make_golden_native.py) ----
def test_cuda_matches_compiled_reference_twins(pk, ref_native):
    """backend='cuda' vs the reference's own `_c_exec_loop` / `_c_exec_loop_moving_window` (lib/cok.pyx) on
    seeded inputs."""
    xyz, val, pts = cases.native_inputs("cuda2d")
    assert_allclose([xyz.sum(), val.sum(), pts.sum()], ref_native["cuda2d/fp"], rtol=1e-12)
    for model in ("exponential", "spherical", "linear"):
        params = cases.MODELS[model]
        m = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model=model, variogram_parameters=list(params))
        z, ss = m.execute("points", pts[:, 0], pts[:, 1], backend="cuda")
        assert_parity(z, ref_native["cuda2d/%s/z" % model], R64, model + " z vs cok._c_exec_loop")
        assert_parity(ss, ref_native["cuda2d/%s/ss" % model], R64, model + " ss vs cok._c_exec_loop")
    m = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential",
                           variogram_parameters=[1.0, 150.0, 0.05])
    z, ss = m.execute("points", pts[:, 0], pts[:, 1], backend="cuda", n_closest_points=16)
    assert_parity(z, ref_native["cuda2d/k16/z"], R64, "knn z vs cok._c_exec_loop_moving_window")
    assert_parity(ss, ref_native["cuda2d/k16/ss"], R64, "knn ss vs cok._c_exec_loop_moving_window")


# ---- BASELINE configs 3, 4, 5 at their full data sizes: size-independent properties + oracle subsample ----
def test_full_size_properties_cfg3(pk):
    """Config 3 (OK3D, N=8000, gaussian [1, 300, 0.05]) on 4096 random points of the 200x200x50 grid + 16
    exact hits: linearity in the values, sigma^2 independent of the values, shard concatenation bit for bit,
    grid call == points call, oracle (full 8001^2 inverse) on a subsample."""
    from oracle import krige_oracle as ko
    xyz, val = cases.synth_data(1003, 8000, 3)
    params = [1.0, 300.0, 0.05]
    gx, gy, gz = np.linspace(0, 1000, 200), np.linspace(0, 1000, 200), np.linspace(0, 250, 50)
    mk = lambda v: pk.OrdinaryKriging3D(xyz[:, 0], xyz[:, 1], xyz[:, 2], v, variogram_model="gaussian",
                                        variogram_parameters=params)
    ok = mk(val)
    rng = np.random.default_rng(33)
    pts = np.column_stack([rng.choice(gx, 4096), rng.choice(gy, 4096), rng.choice(gz, 4096)])
    pts = np.vstack([pts, xyz[:16]])
    z, ss = ok.execute("points", pts[:, 0], pts[:, 1], pts[:, 2], backend="cuda")
    z2, ss2 = mk(-2.0 * val + 11.0).execute("points", pts[:, 0], pts[:, 1], pts[:, 2], backend="cuda")
    assert_allclose(z2, -2.0 * z + 11.0, rtol=1e-8)
    assert_allclose(ss2, ss, rtol=1e-12, atol=1e-14)
    assert_allclose(z[-16:], val[:16], rtol=1e-9)                       # exact hits interpolate
    assert np.all(np.abs(ss[-16:]) < 1e-9)
    h = ok._ensure_problem()
    zg, sg = h.execute_grid(gx, gy, gz, None, 777, 5000)               # a slice of the real grid
    za, sa = h.execute_grid(gx, gy, gz, None, 777, 1234)
    zb, sb = h.execute_grid(gx, gy, gz, None, 777 + 1234, 5000 - 1234)
    assert np.array_equal(np.concatenate([za, zb]), zg) and np.array_equal(np.concatenate([sa, sb]), sg)
    G = ko.grid_points([gx, gy, gz])[777:777 + 5000]
    zp, sp = ok.execute("points", G[:, 0], G[:, 1], G[:, 2], backend="cuda")
    assert_allclose(zg, zp, rtol=1e-12)
    assert_allclose(sg, sp, rtol=1e-10, atol=1e-13)
    zo, so = ko.krige_chunked(xyz, val, "gaussian", ko.stored_parameters("gaussian", params), pts)   # 4096 + 16
    assert_parity(z, zo, R64, "cfg3 z")
    assert_parity(ss, so, R64, "cfg3 ss")


def test_full_size_properties_cfg4(pk):
    """Config 4 (UK regional_linear, N=10000, exponential, fp32 device math): float32 and float64 device paths
    vs the oracle (10003^2 inverse) on 4096 + 16 points at their tolerances, drift reproduction
    (a field that IS a linear trend is returned exactly with zero-mean residual structure)."""
    from oracle import krige_oracle as ko
    xyz, val = cases.synth_data(1004, 10000, 2)
    params = [1.0, 300.0, 0.05]
    uk = pk.UniversalKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential", variogram_parameters=params,
                             drift_terms=["regional_linear"])
    rng = np.random.default_rng(44)
    pts = np.vstack([rng.uniform(0, 1000, (4096, 2)), xyz[:16]])
    z64, s64 = uk.execute("points", pts[:, 0], pts[:, 1], backend="cuda")
    z32, s32 = uk.execute("points", pts[:, 0], pts[:, 1], backend="cuda", dtype="float32")
    zo, so = ko.krige_chunked(xyz, val, "exponential", ko.stored_parameters("exponential", params), pts,
                              regional_linear=True)                       # 10003^2 inverse, 4096 + 16 points
    assert_parity(z64, zo, R64, "cfg4 z")
    assert_parity(s64, so, R64, "cfg4 ss")
    assert_parity(z32, zo, 1e-2, "cfg4 fp32 z vs oracle")
    assert_parity(s32, so, 1e-2, "cfg4 fp32 ss vs oracle")
    trend = 3.0 + 0.01 * xyz[:, 0] - 0.02 * xyz[:, 1]
    ut = pk.UniversalKriging(xyz[:, 0], xyz[:, 1], trend, variogram_model="exponential", variogram_parameters=params,
                             drift_terms=["regional_linear"])
    zt, _ = ut.execute("points", pts[:, 0], pts[:, 1], backend="cuda")
    assert_allclose(zt, 3.0 + 0.01 * pts[:, 0] - 0.02 * pts[:, 1], rtol=1e-8, atol=1e-8)


def test_full_size_properties_cfg5(pk):
    """Config 5 (OK 2-D, N=100000, k=64 moving window, exponential [1, 50, 0.05]): 4096 grid points + 16
    exact hits against the oracle's kd-tree + (k+1)^2 solves, shard concatenation bit for bit, linearity."""
    from oracle import krige_oracle as ko
    xyz, val = cases.synth_data(1005, 100000, 2)
    params = [1.0, 50.0, 0.05]
    ok = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential", variogram_parameters=params)
    g = np.linspace(0, 1000, 4000)
    rng = np.random.default_rng(55)
    pts = np.vstack([np.column_stack([rng.choice(g, 4096), rng.choice(g, 4096)]), xyz[:16]])
    z, ss = ok.execute("points", pts[:, 0], pts[:, 1], backend="cuda", n_closest_points=64)
    zo, so = ko.krige(xyz, val, "exponential", ko.stored_parameters("exponential", params), pts, n_closest_points=64)
    assert_parity(z, zo, R64, "cfg5 z")
    assert_parity(ss, so, R64, "cfg5 ss")
    h = ok._ensure_problem("float64", knn=True)
    zg, sg = h.execute_knn_grid(64, g, g, None, 123456, 6000)
    za, sa = h.execute_knn_grid(64, g, g, None, 123456, 2500)
    zb, sb = h.execute_knn_grid(64, g, g, None, 123456 + 2500, 3500)
    assert np.array_equal(np.concatenate([za, zb]), zg) and np.array_equal(np.concatenate([sa, sb]), sg)
    ok2 = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], 0.5 * val + 4.0, variogram_model="exponential",
                             variogram_parameters=params)
    z2, ss2 = ok2.execute("points", pts[:, 0], pts[:, 1], backend="cuda", n_closest_points=64)
    assert_allclose(z2, 0.5 * z + 4.0, rtol=1e-9)
    assert_allclose(ss2, ss, rtol=1e-12, atol=1e-14)


# ---- variogram_model='custom' on the device (KB200_VG_TABLE) ------------------------------------------------
CUSTOM_GLOBAL = [c for c in cases.CUSTOM_CASES]


@pytest.mark.parametrize("case", CUSTOM_GLOBAL, ids=[c["name"] for c in CUSTOM_GLOBAL])
def test_custom_variogram_cases_match_reference(pk, case, ref_custom):
    """User callables f(params, d) (ok.py:224-253) against the imported reference run with the same callable:
    global OK/UK 2-D/3-D, anisotropy, masked, non-exact, moving window, geographic."""
    inp, z, ss = _run(pk, case)
    zr, sr = ref_custom[case["name"] + "/z"], ref_custom[case["name"] + "/ss"]
    assert z.shape == zr.shape
    if case["style"] == "masked":
        keep = ~np.ma.getmaskarray(z)
        z, ss, zr, sr = np.ma.getdata(z)[keep], np.ma.getdata(ss)[keep], zr[keep], sr[keep]
    assert_parity(np.ravel(z), np.ravel(zr), R64, "custom z")
    assert_parity(np.ravel(ss), np.ravel(sr), R64, "custom ss")


def test_custom_variogram_other_dtypes(pk, ref_custom):
    """The tabulated model also feeds the tcgen05 kernels (float32 3xTF32, float64x INT8 slices)."""
    case = cases.CUSTOM_CASES[0]
    inp = cases.build_inputs(case)
    m = cases.make_model(pk, case, inp)
    P = inp["points"]
    zr, sr = ref_custom[case["name"] + "/z"], ref_custom[case["name"] + "/ss"]
    z, ss = m.execute("points", P[:, 0], P[:, 1], backend="cuda", dtype="float64x")
    assert_parity(z, zr, R64, "custom float64x z")
    assert_parity(ss, sr, R64, "custom float64x ss")
    z, ss = m.execute("points", P[:, 0], P[:, 1], backend="cuda", dtype="float32")
    assert_parity(z, zr, 1e-2, "custom float32 z")
    assert_parity(ss, sr, 1e-2, "custom float32 ss")


def test_gstools_model_through_cuda(pk):
    """The GSTools route (ok.py:224-239) end to end on the device with the stand-in package of tests/gstools_stub.py:
    the CovModel's pykrige_vario is tabulated (KB200_VG_TABLE) and the result agrees with the oracle run with the
    same callable and the model's anisotropy; global path, moving window and 3-D."""
    import gstools_stub
    from oracle import krige_oracle as ko
    xyz, val = cases.synth_data(88, 500, 2)
    pts = cases.synth_points(88, 400, 2, xyz)
    try:
        gstools_stub.install()
        m = gstools_stub.CovModel(dim=2, var=1.2, len_scale=120.0, nugget=0.05, anis=0.6, angle=35.0)
        ok = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, m)
        z, ss = ok.execute("points", pts[:, 0], pts[:, 1], backend="cuda")
        zo, so = ko.krige(xyz, val, m.pykrige_vario, [], pts, scaling=[m.pykrige_anis], angle=[m.pykrige_angle])
        assert_parity(z, zo, R64, "gstools z")
        assert_parity(ss, so, R64, "gstools ss")
        zk, sk = ok.execute("points", pts[:, 0], pts[:, 1], backend="cuda", n_closest_points=12)
        zo, so = ko.krige(xyz, val, m.pykrige_vario, [], pts, scaling=[m.pykrige_anis], angle=[m.pykrige_angle],
                          n_closest_points=12)
        assert_parity(zk, zo, R64, "gstools knn z")
        assert_parity(sk, so, R64, "gstools knn ss")
        x3, v3 = cases.synth_data(89, 300, 3)
        p3 = cases.synth_points(89, 200, 3, x3)
        m3 = gstools_stub.CovModel(dim=3, var=1.0, len_scale=200.0, nugget=0.02)
        k3 = pk.OrdinaryKriging3D(x3[:, 0], x3[:, 1], x3[:, 2], v3, m3)
        z, ss = k3.execute("points", p3[:, 0], p3[:, 1], p3[:, 2], backend="cuda")
        zo, so = ko.krige(x3, v3, m3.pykrige_vario, [], p3)
        assert_parity(z, zo, R64, "gstools 3d z")
        assert_parity(ss, so, R64, "gstools 3d ss")
    finally:
        gstools_stub.uninstall()


def test_tile_width_is_invisible(pk):
    """The fp64 solve kernel kriges the points left over after the last full round of 64-point tiles in a second launch
    with 32- or 16-point tiles (they spread over all SMs instead of keeping a few busy for a whole tile time: multi-GPU
    strong scaling). Per-point arithmetic must not depend on the tile width: slices whose tails fall on narrow tiles
    equal the same points of a call with a different split, bit for bit (OK and UK)."""
    xyz, val = cases.synth_data(77, 600, 2)
    gx, gy = np.linspace(0, 1000, 500), np.linspace(0, 1000, 500)
    for m in (pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential", variogram_parameters=[1.0, 300.0, 0.05]),
              pk.UniversalKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="spherical", variogram_parameters=[1.0, 400.0, 0.05],
                                  drift_terms=["regional_linear"])):
        z, ss = m.execute("grid", gx, gy, backend="cuda")              # 250 000 points: 26 full rounds + a narrow-tile tail
        h = m._ensure_problem()
        for first, count in ((0, 125000), (60000, 125000), (125000, 125000), (1000, 9472 * 2 + 100)):
            za, sa = h.execute_grid(gx, gy, None, None, first, count)   # different full-round / tail split
            assert np.array_equal(za, z.ravel()[first:first + count]) and np.array_equal(sa, ss.ravel()[first:first + count])
