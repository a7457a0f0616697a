"""CPU tests: the oracle (oracle/krige_oracle.py) is pinned against (a) the reference's own golden
vectors and (b) outputs of the imported reference for every seeded case (tests/golden/*.npz)."""
import numpy as np
import pytest
from numpy.testing import assert_allclose

import cases
from conftest import assert_parity
from oracle import krige_oracle as ko


def _oracle_case(case, inp):
    if case.get("geographic"):
        pts = inp["points"] if case["style"] == "points" else ko.grid_points(inp["axes"])
        return ko.krige_geographic(inp["data"], inp["values"], case["model"],
                                   ko.stored_parameters(case["model"], case["params"]), pts,
                                   exact_values=case["exact_values"], n_closest_points=case["k"])
    dim = case["dim"]
    ctor = case["ctor"]
    if dim == 2:
        scaling = [ctor.get("anisotropy_scaling", 1.0)]
        angle = [ctor.get("anisotropy_angle", 0.0)]
    else:
        scaling = [ctor.get("anisotropy_scaling_y", 1.0), ctor.get("anisotropy_scaling_z", 1.0)]
        angle = [ctor.get("anisotropy_angle_x", 0.0), ctor.get("anisotropy_angle_y", 0.0),
                 ctor.get("anisotropy_angle_z", 0.0)]
    stored = ko.stored_parameters(case["model"], case["params"])
    xyz = inp["data"]
    pts = inp["points"] if case["style"] == "points" else ko.grid_points(inp["axes"])
    center = (xyz.max(axis=0) + xyz.min(axis=0)) / 2.0
    P = ko.adjust_for_anisotropy(xyz, center, scaling, angle)
    Q = ko.adjust_for_anisotropy(pts, center, scaling, angle)
    dd, pd = [], []
    if case["point_log"] is not None:      # uk.py:884-896, 955-966 (wells in the adjusted frame)
        wells = np.array(case["point_log"], dtype=float)
        wxy = ko.adjust_for_anisotropy(wells[:, :2], center, scaling, angle)
        for w in range(wells.shape[0]):
            for X, lst in ((P, dd), (Q, pd)):
                with np.errstate(divide="ignore"):
                    ld = np.log(np.sqrt((X[:, 0] - wxy[w, 0]) ** 2 + (X[:, 1] - wxy[w, 1]) ** 2))
                ld[np.isinf(ld)] = -100.0
                lst.append(-wells[w, 2] * ld)
    if case["external_z"]:                 # bilinear sample at ORIGINAL coordinates (uk.py:512-628)
        from scipy.interpolate import RegularGridInterpolator
        f = RegularGridInterpolator((inp["ext_y"], inp["ext_x"]), inp["ext_z"])
        dd.append(f(np.column_stack((xyz[:, 1], xyz[:, 0]))))
        pd.append(f(np.column_stack((pts[:, 1], pts[:, 0]))))
    for j in range(case["n_specified"]):
        dd.append(np.asarray(inp["spec_data"][j]).ravel())
        pd.append(np.asarray(inp["spec_pts"][j]).ravel())
    for fn in case["functional"]:          # evaluated with adjusted coordinates (uk.py:906-910)
        f = cases.FUNCS[fn]
        dd.append(f(*[P[:, c] for c in range(dim)]))
        pd.append(f(*[Q[:, c] for c in range(dim)]))
    z, ss = ko.krige(xyz, inp["values"], case["model"], stored, pts, scaling=scaling, angle=angle,
                     regional_linear="regional_linear" in case["drift_terms"], data_drift=dd, point_drift=pd,
                     exact_values=case["exact_values"], n_closest_points=case["k"])
    return z, ss


@pytest.mark.parametrize("case", cases.CASES, ids=[c["name"] for c in cases.CASES])
def test_oracle_matches_reference_outputs(case, ref_cases):
    inp = cases.build_inputs(case)
    fp = ref_cases[case["name"] + "/fp"]
    assert_allclose([inp["data"].sum(), inp["values"].sum()], fp, rtol=1e-13)
    z, ss = _oracle_case(case, inp)
    zr = ref_cases[case["name"] + "/z"].ravel()
    sr = ref_cases[case["name"] + "/ss"].ravel()
    if case["style"] == "masked":
        keep = ~inp["mask"].ravel()
        z, ss, zr, sr = z[keep], ss[keep], zr[keep], sr[keep]
    # the oracle IS the reference's arithmetic: agreement to rounding of the dense inverse
    assert_parity(z, zr, 1e-9, case["name"] + " z")
    assert_parity(ss, sr, 1e-8, case["name"] + " ss")


def test_oracle_vs_kt3d_ok(ref_goldens):
    """tests/test_core.py:490-507: OK 2-D vs KT3D_H2O on the 100x100 grid."""
    g = ref_goldens
    d = g["data"]
    pts = ko.grid_points([g["ok_gridx"], g["ok_gridy"]])
    z, ss = ko.krige(d[:, :2], d[:, 2], "exponential", ko.stored_parameters("exponential", [500.0, 3000.0, 0.0]), pts)
    assert_allclose(z.reshape(g["ok_answer"].shape), g["ok_answer"], rtol=1e-7)


def test_oracle_vs_kt3d_uk(ref_goldens):
    """tests/test_core.py:707-725: UK regional-linear vs KT3D_H2O."""
    g = ref_goldens
    d = g["data"]
    pts = ko.grid_points([g["uk_gridx"], g["uk_gridy"]])
    z, ss = ko.krige(d[:, :2], d[:, 2], "exponential", ko.stored_parameters("exponential", [500.0, 3000.0, 0.0]),
                     pts, regional_linear=True)
    assert_allclose(z.reshape(g["uk_answer"].shape), g["uk_answer"], rtol=1e-7)


def test_oracle_vs_kt3d_3d(ref_goldens):
    """tests/test_core.py:1957-1989: OK3D vs KT3D, z and sigma^2, rtol 1e-3; and the moving window
    with k=10 equals the full answer (tests/test_core.py:1992-2017)."""
    g = ref_goldens
    d = g["data3d"]
    ax = np.arange(10.0)
    pts = ko.grid_points([ax, ax, ax])
    z, ss = ko.krige(d[:, :3], d[:, 3], "linear", [1.0, 0.1], pts)
    assert_allclose(z, g["answer3d"][:, 0], rtol=1e-3, atol=1e-8)
    assert_allclose(ss, g["answer3d"][:, 1], rtol=1e-3, atol=1e-8)
    z, ss = ko.krige(d[:, :3], d[:, 3], "linear", [1.0, 0.1], pts, n_closest_points=10)
    assert_allclose(z, g["answer3d"][:, 0], rtol=1e-3)
    assert_allclose(ss, g["answer3d"][:, 1], rtol=1e-3)


def test_oracle_kitanidis():
    """Kitanidis example 3.2 (tests/test_core.py:378-401): z = 1.6364, sigma^2 = 0.4201."""
    data = np.array([[9.7, 47.6, 1.22], [43.8, 24.6, 2.822]])
    z, ss = ko.krige(data[:, :2], data[:, 2], "linear", [0.006, 0.1], np.array([[18.8, 67.9]]))
    assert z[0] == pytest.approx(1.6364, rel=1e-4)
    assert ss[0] == pytest.approx(0.4201, rel=1e-4)


# ---- constructor side (SURVEY.md §8f next-2) ------------------------------------------------
def test_oracle_variogram_reference_known_answers():
    """tests/test_core.py:226-236 and :283-301 (the reference's own known answers)."""
    x = np.array([1.0 + n / np.sqrt(2) for n in range(4)])
    lags, semi = ko.experimental_variogram(np.vstack((x, x)).T, np.arange(1.0, 5.0, 1.0), 6)
    assert_allclose(lags, [1.0, 2.0, 3.0])
    assert_allclose(semi, [0.5, 2.0, 4.5])
    a = np.array([1.0, 2.0, 3.0, 4.0])
    lags, semi = ko.experimental_variogram(np.vstack((a, a, a)).T, a, 3)
    assert_allclose(lags, [np.sqrt(3.0), 2.0 * np.sqrt(3.0), 3.0 * np.sqrt(3.0)])
    assert_allclose(semi, [0.5, 2.0, 4.5])


@pytest.mark.parametrize("case", cases.VARIOGRAM_CASES, ids=[c["name"] for c in cases.VARIOGRAM_CASES])
def test_oracle_variogram_matches_reference(case, ref_ctor):
    X, y = cases.build_ctor_inputs(case)
    assert_allclose([X.sum(), y.sum()], ref_ctor[case["name"] + "/fp"], rtol=1e-12)
    lags, semi = ko.experimental_variogram(X, y, case["nlags"], case["coordinates_type"])
    assert_allclose(lags, ref_ctor[case["name"] + "/lags"], rtol=1e-12)
    assert_allclose(semi, ref_ctor[case["name"] + "/semi"], rtol=1e-12)


@pytest.mark.parametrize("case", cases.STATS_CASES, ids=[c["name"] for c in cases.STATS_CASES])
def test_oracle_statistics_match_reference(case, ref_ctor):
    X, y = cases.build_ctor_inputs(case)
    assert_allclose([X.sum(), y.sum()], ref_ctor[case["name"] + "/fp"], rtol=1e-12)
    delta, sigma, epsilon = ko.find_statistics(X, y, case["model"], case["params"], case["coordinates_type"])
    assert delta.shape == ref_ctor[case["name"] + "/delta"].shape
    assert_allclose(delta, ref_ctor[case["name"] + "/delta"], rtol=1e-8, atol=1e-10)
    assert_allclose(sigma, ref_ctor[case["name"] + "/sigma"], rtol=1e-8)
    assert_allclose(epsilon, ref_ctor[case["name"] + "/epsilon"], rtol=1e-8, atol=1e-10)


def test_oracle_krige_one_kitanidis():
    """tests/test_core.py:378-401: Kitanidis example 3.2 through core._krige."""
    data = np.array([[9.7, 47.6, 1.22], [43.8, 24.6, 2.822]])
    z, ss = ko.krige_one(data[:, :2], data[:, 2], np.array([18.8, 67.9]), "linear", [0.006, 0.1])
    assert z == pytest.approx(1.6364, rel=1e-4)
    assert ss == pytest.approx(0.4201, rel=1e-4)


# ---- pseudo_inv=True (SURVEY.md §8f next-4) ---------------------------------------------------------
@pytest.mark.parametrize("case", cases.PINV_CASES, ids=[c["name"] for c in cases.PINV_CASES])
def test_oracle_pseudo_inverse_matches_reference(case, ref_pinv):
    inp = cases.build_inputs(case)
    assert_allclose([inp["data"].sum(), inp["values"].sum()], ref_pinv[case["name"] + "/fp"], rtol=1e-12)
    pts = inp["points"] if case["style"] == "points" else ko.grid_points(inp["axes"])
    z, ss = ko.krige(inp["data"], inp["values"], case["model"], ko.stored_parameters(case["model"], case["params"]),
                     pts, regional_linear="regional_linear" in case["drift_terms"],
                     exact_values=case["exact_values"], pseudo_inv=case["ctor"]["pseudo_inv_type"])
    assert_parity(z, ref_pinv[case["name"] + "/z"].ravel(), 1e-9, "z")
    assert_parity(ss, ref_pinv[case["name"] + "/ss"].ravel(), 1e-9, "ss")


@pytest.mark.parametrize("ptype", ["pinv", "pinvh"])
def test_oracle_pseudo_inverse_known_answer(ptype):
    """tests/test_core.py:2913-2949: two redundant points (values 1 and 3) krige to their mean."""
    data = np.array([[0.0, 0.0, 1.0], [0.0, 0.0, 3.0], [1.0, 0.0, 6.0]])
    z, _ = ko.krige(data[:, :2], data[:, 2], "linear", [1.0, 0.0], np.array([[0.0, 0.0]]), pseudo_inv=ptype)
    assert np.isclose(z[0], 2.0)
    d3 = np.array([[0.0, 0.0, 0.0, 1.0], [0.0, 0.0, 0.0, 3.0], [1.0, 0.0, 0.0, 6.0]])
    z, _ = ko.krige(d3[:, :3], d3[:, 3], "linear", [1.0, 0.0], np.array([[0.0, 0.0, 0.0]]), pseudo_inv=ptype)
    assert np.isclose(z[0], 2.0)


# ---- the reference's compiled native twins (outputs stored by golden/make_golden_native.py) -----------
def _native_inputs(name, ref_native):
    xyz, val, pts = cases.native_inputs(name)
    assert_allclose([xyz.sum(), val.sum(), pts.sum()], ref_native[name + "/fp"], rtol=1e-12)
    return xyz, val, pts


@pytest.mark.parametrize("model", ["linear", "power", "gaussian", "exponential", "spherical"])
def test_oracle_matches_compiled_reference_twin(model, ref_native):
    """The numpy restatement vs the reference's own compiled `_c_exec_loop` (cok.pyx:14-96), same inputs."""
    xyz, val, pts = _native_inputs("global2d", ref_native)
    stored = ko.stored_parameters(model, cases.MODELS[model])
    for exact in (True, False):
        key = "global2d/%s/%s" % (model, "exact" if exact else "inexact")
        zo, so = ko.krige(xyz, val, model, stored, pts, exact_values=exact)
        assert_parity(zo, ref_native[key + "/z"], 1e-8, "z")
        assert_parity(so, ref_native[key + "/ss"], 1e-8, "ss")


def test_oracle_moving_window_matches_compiled_reference_twin(ref_native):
    """... and `_c_exec_loop_moving_window` (cok.pyx:98-193), 2-D and 3-D."""
    for name, k in (("window2d", 8), ("window3d", 12)):
        xyz, val, pts = _native_inputs(name, ref_native)
        stored = ko.stored_parameters("exponential", [1.0, 150.0, 0.05])
        zo, so = ko.krige(xyz, val, "exponential", stored, pts, n_closest_points=k)
        assert_parity(zo, ref_native["%s/k%d/z" % (name, k)], 1e-9, "z")
        assert_parity(so, ref_native["%s/k%d/ss" % (name, k)], 1e-9, "ss")


# ---- variogram_model='custom' ---------------------------------------------------------------------------
@pytest.mark.parametrize("case", cases.CUSTOM_CASES, ids=[c["name"] for c in cases.CUSTOM_CASES])
def test_oracle_custom_variogram_matches_reference(case, ref_custom):
    inp = cases.build_inputs(case)
    assert_allclose([inp["data"].sum(), inp["values"].sum()], ref_custom[case["name"] + "/fp"], rtol=1e-12)
    fn = cases.CUSTOM_VARIOGRAMS[case["custom"]][0]
    pts = inp["points"] if case["style"] == "points" else ko.grid_points(inp["axes"])
    if case.get("geographic"):
        z, ss = ko.krige_geographic(inp["data"], inp["values"], fn, case["params"], pts,
                                    exact_values=case["exact_values"], n_closest_points=case["k"])
    else:
        ctor, dim = case["ctor"], case["dim"]
        scaling = [ctor.get("anisotropy_scaling", 1.0)] if dim == 2 else [1.0, 1.0]
        angle = [ctor.get("anisotropy_angle", 0.0)] if dim == 2 else [0.0, 0.0, 0.0]
        z, ss = ko.krige(inp["data"], inp["values"], fn, case["params"], pts, scaling=scaling, angle=angle,
                         regional_linear="regional_linear" in case["drift_terms"],
                         exact_values=case["exact_values"], n_closest_points=case["k"])
    zr, sr = ref_custom[case["name"] + "/z"].ravel(), ref_custom[case["name"] + "/ss"].ravel()
    if case["style"] == "masked":
        keep = ~inp["mask"].ravel()
        z, ss, zr, sr = z[keep], ss[keep], zr[keep], sr[keep]
    assert_parity(z, zr, 1e-9, "z")
    assert_parity(ss, sr, 1e-9, "ss")
