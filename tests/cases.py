"""Seeded parity cases shared by tests/golden/make_golden.py (which runs the imported reference,
in the build container only) and the test-suite (which replays them through the oracle on CPU and
through backend='cuda' on the GPU). Synthetic inputs follow SURVEY.md §8(d): uniform random
scatter, values with a non-zero mean, list-form variogram parameters [FULL sill, range, nugget],
and the first 16 data coordinates appended as 'points' queries to exercise exact hits.
"""
import numpy as np


def synth_data(seed, n, dim, box=(1000.0, 1000.0, 250.0)):
    rng = np.random.default_rng(seed)
    xyz = np.column_stack([rng.uniform(0.0, box[c], n) for c in range(dim)])
    val = 50.0 + 10.0 * np.sin(xyz[:, 0] / 150.0) * np.cos(xyz[:, 1] / 200.0)
    if dim == 3:
        val = val + 5.0 * np.sin(xyz[:, 2] / 60.0)
    val = val + rng.normal(0.0, 1.0, n)
    return xyz, val


def synth_points(seed, m, dim, data_xyz, box=(1000.0, 1000.0, 250.0), n_hits=16):
    rng = np.random.default_rng(seed + 7919)
    pts = np.column_stack([rng.uniform(0.0, box[c], m) for c in range(dim)])
    hits = data_xyz[: min(n_hits, data_xyz.shape[0])]
    return np.vstack([pts, hits])


# seeded inputs of the comparisons with the reference's compiled twins (golden/make_golden_native.py -> ref_native.npz):
# name -> (seed, data points, query points, dim)
NATIVE_INPUTS = {"global2d": (11, 300, 200, 2), "window2d": (14, 400, 150, 2), "window3d": (15, 400, 150, 3),
                 "cuda2d": (2024, 1500, 2000, 2)}


def native_inputs(name):
    """(data coordinates, values, query points) of NATIVE_INPUTS[name]."""
    seed, n, m, dim = NATIVE_INPUTS[name]
    xyz, val = synth_data(seed, n, dim)
    return xyz, val, synth_points(seed, m, dim, xyz)


# functional drift terms by name (callables cannot be stored in fixtures)
FUNCS = {
    "fx": lambda x, y: x,
    "fy": lambda x, y: y,
    "fxy": lambda x, y: 1e-3 * x * y,
    "fx3": lambda x, y, z: x,
    "fy3": lambda x, y, z: y,
    "fz3": lambda x, y, z: z,
    "fr3": lambda x, y, z: np.sqrt(x * x + y * y + z * z),
}

MODELS = {
    "linear": [0.004, 0.05],
    "power": [0.002, 1.3, 0.05],
    "gaussian": [1.0, 300.0, 0.05],
    "exponential": [1.0, 300.0, 0.05],
    "spherical": [1.0, 400.0, 0.05],
    "hole-effect": [1.0, 300.0, 0.05],
}


def _c(name, cls, n, m, seed, model, params=None, **kw):
    d = dict(name=name, cls=cls, n=n, m=m, seed=seed, model=model,
             params=list(MODELS[model] if params is None else params),
             dim=3 if cls.endswith("3D") else 2, style="points", ctor={}, k=None,
             drift_terms=[], functional=[], n_specified=0, point_log=None, external_z=False,
             exact_values=True, box=(1000.0, 1000.0, 250.0), ref_backend="vectorized", geographic=False)
    d.update(kw)
    return d


CASES = []
# config 1 of BASELINE.json: OK 2-D, N=100, 50x50 grid, spherical
CASES.append(_c("cfg1_ok2d_n100_grid50", "OK", 100, 0, 1001, "spherical", style="grid",
                grid=(50, 50, 1)))
# every built-in variogram model, with anisotropy, points + exact hits
for i, mname in enumerate(["linear", "power", "gaussian", "exponential", "spherical"]):
    CASES.append(_c("ok2d_%s_aniso" % mname, "OK", 200, 300, 2000 + i, mname,
                    ctor=dict(anisotropy_scaling=1.7, anisotropy_angle=30.0)))
# hole-effect is not a valid (conditionally negative definite) model in 2-D for scattered data;
# the reference still returns LU numbers for it. Kept as a fixture for the singular-path test.
CASES.append(_c("ok2d_hole_effect_small", "OK", 12, 40, 2010, "hole-effect", params=[1.0, 900.0, 0.05]))
CASES.append(_c("ok2d_nonexact", "OK", 150, 200, 2020, "exponential", exact_values=False))
CASES.append(_c("ok2d_zero_nugget", "OK", 150, 200, 2021, "spherical", params=[2.0, 350.0, 0.0]))
CASES.append(_c("ok2d_masked", "OK", 120, 0, 2022, "exponential", style="masked", grid=(23, 17, 1)))
# reduced-size stand-ins for configs 2-4 that the reference can run in one call
CASES.append(_c("cfg2r_ok2d_n1000", "OK", 1000, 2000, 1002, "exponential"))
CASES.append(_c("cfg3r_ok3d_n800", "OK3D", 800, 1500, 1003, "gaussian"))
CASES.append(_c("cfg4r_uk2d_n1000", "UK", 1000, 2000, 1004, "exponential", drift_terms=["regional_linear"]))
# universal kriging drift kinds (uk.py:876-910)
CASES.append(_c("uk2d_reglin_aniso", "UK", 180, 260, 3001, "spherical", drift_terms=["regional_linear"],
                ctor=dict(anisotropy_scaling=0.6, anisotropy_angle=-20.0)))
CASES.append(_c("uk2d_pointlog", "UK", 120, 200, 3002, "exponential", drift_terms=["point_log"],
                point_log=[[300.0, 420.0, 1.0], [710.0, 150.0, -0.5]]))
CASES.append(_c("uk2d_externalz", "UK", 120, 200, 3003, "exponential", drift_terms=["external_Z"], external_z=True))
CASES.append(_c("uk2d_specified", "UK", 120, 200, 3004, "gaussian", drift_terms=["specified"], n_specified=2))
CASES.append(_c("uk2d_functional", "UK", 120, 200, 3005, "linear", drift_terms=["functional"],
                functional=["fx", "fy", "fxy"]))
CASES.append(_c("uk2d_all_grid", "UK", 90, 0, 3006, "exponential", style="grid", grid=(19, 13, 1),
                drift_terms=["regional_linear", "specified", "functional"], n_specified=1, functional=["fxy"]))
CASES.append(_c("uk2d_masked", "UK", 90, 0, 3007, "spherical", style="masked", grid=(15, 21, 1),
                drift_terms=["regional_linear"]))
# 3-D
CASES.append(_c("ok3d_linear_aniso", "OK3D", 200, 300, 4001, "linear",
                ctor=dict(anisotropy_scaling_y=1.4, anisotropy_scaling_z=3.0, anisotropy_angle_x=10.0,
                          anisotropy_angle_y=-25.0, anisotropy_angle_z=40.0)))
CASES.append(_c("ok3d_grid", "OK3D", 150, 0, 4002, "exponential", style="grid", grid=(9, 8, 7)))
CASES.append(_c("ok3d_masked", "OK3D", 100, 0, 4003, "spherical", style="masked", grid=(6, 7, 5)))
CASES.append(_c("uk3d_reglin", "UK3D", 200, 300, 4004, "gaussian", drift_terms=["regional_linear"]))
CASES.append(_c("uk3d_spec_func", "UK3D", 150, 200, 4005, "exponential", drift_terms=["specified", "functional"],
                n_specified=1, functional=["fx3", "fr3"]))
CASES.append(_c("uk3d_all_grid", "UK3D", 100, 0, 4006, "linear", style="grid", grid=(5, 6, 4),
                drift_terms=["regional_linear", "functional"], functional=["fr3"]))
# moving window (ok.py:722-758; reference backend 'loop')
CASES.append(_c("knn2d_k8", "OK", 500, 300, 5001, "exponential", params=[1.0, 150.0, 0.05], k=8, ref_backend="loop"))
CASES.append(_c("knn2d_k16_nonexact", "OK", 400, 200, 5002, "spherical", k=16, exact_values=False, ref_backend="loop"))
CASES.append(_c("knn2d_k64_grid", "OK", 3000, 0, 1005, "exponential", params=[1.0, 50.0, 0.05], k=64,
                style="grid", grid=(24, 20, 1), ref_backend="loop"))
CASES.append(_c("knn3d_k10", "OK3D", 300, 200, 5003, "linear", k=10, ref_backend="loop"))
CASES.append(_c("knn2d_k2", "OK", 60, 100, 5004, "linear", k=2, ref_backend="loop"))

# coordinates_type='geographic' (ok.py:292-306, 634-640, 930-996): lon in [0, 60), lat in [0, 45) shifted to a
# mid-latitude window; variogram ranges are in degrees
_GEO = dict(geographic=True, box=(60.0, 45.0, 1.0), ctor=dict(coordinates_type="geographic"))
CASES.append(_c("geo_ok_points", "OK", 250, 300, 6001, "exponential", params=[1.0, 25.0, 0.05], **_GEO))
CASES.append(_c("geo_ok_grid_spherical", "OK", 150, 0, 6002, "spherical", params=[1.0, 30.0, 0.02], style="grid",
                grid=(17, 12, 1), **_GEO))
CASES.append(_c("geo_ok_nonexact_linear", "OK", 120, 150, 6003, "linear", params=[0.05, 0.1], exact_values=False, **_GEO))
CASES.append(_c("geo_knn_k12", "OK", 400, 200, 6004, "exponential", params=[1.0, 20.0, 0.05], k=12, ref_backend="loop", **_GEO))

CASE_BY_NAME = {c["name"]: c for c in CASES}

# pseudo_inv=True (ok.py:156-165,660-661; tests/test_core.py:2913-2949): redundant data points (exact
# duplicates with different values, nugget 0 -> singular kriging matrix) are averaged. Kept out of CASES:
# their reference outputs live in tests/golden/ref_pinv.npz.
def _p(ptype="pinv"):
    return dict(pseudo_inv=True, pseudo_inv_type=ptype)


PINV_CASES = [
    _c("pinv_ok2d_dups", "OK", 80, 120, 7001, "exponential", params=[1.0, 300.0, 0.0], dups=4, ctor=_p()),
    _c("pinv_ok2d_dups_pinvh_linear", "OK", 60, 100, 7002, "linear", params=[0.004, 0.0], dups=3, ctor=_p("pinvh")),
    _c("pinv_uk2d_rl_dups", "UK", 90, 120, 7003, "spherical", params=[1.0, 400.0, 0.0], dups=3,
       drift_terms=["regional_linear"], ctor=_p()),
    _c("pinv_ok3d_dups", "OK3D", 70, 100, 7004, "exponential", params=[1.0, 300.0, 0.0], dups=3, ctor=_p()),
    _c("pinv_uk3d_rl_dups", "UK3D", 70, 100, 7005, "exponential", params=[1.0, 300.0, 0.0], dups=2,
       drift_terms=["regional_linear"], ctor=_p("pinvh")),
    _c("pinv_ok2d_regular_grid", "OK", 150, 0, 7006, "spherical", style="grid", grid=(19, 14, 1), ctor=_p()),
    _c("pinv_ok2d_nonexact", "OK", 50, 80, 7007, "exponential", params=[1.0, 300.0, 0.0], dups=2, exact_values=False,
       ctor=_p()),
]


def build_inputs(case):
    """Deterministic inputs of a case: data, values, prediction axes/points, mask, drift arrays."""
    dim = case["dim"]
    xyz, val = synth_data(case["seed"], case["n"], dim, case["box"])
    geo_shift = np.array([-20.0, 30.0]) if case.get("geographic") else None
    if geo_shift is not None:
        val = 50.0 + 10.0 * np.sin(xyz[:, 0] / 9.0) * np.cos(xyz[:, 1] / 7.0) + (val - np.round(val))
        xyz = xyz + geo_shift
    for q in range(case.get("dups", 0)):           # redundant data points (same place, different values)
        xyz[case["n"] - 1 - 2 * q] = xyz[3 * q]
    out = dict(data=xyz, values=val)
    rng = np.random.default_rng(case["seed"] + 31337)
    if case["style"] == "points":
        out["points"] = synth_points(case["seed"], case["m"], dim, xyz - (geo_shift if geo_shift is not None else 0.0),
                                     case["box"])
        if geo_shift is not None:
            out["points"] = out["points"] + geo_shift
        npt = out["points"].shape[0]
    else:
        nx, ny, nz = case["grid"]
        axes = [np.linspace(0.0, case["box"][0], nx), np.linspace(0.0, case["box"][1], ny)]
        if geo_shift is not None:
            axes = [axes[0] + geo_shift[0], axes[1] + geo_shift[1]]
        if dim == 3:
            axes.append(np.linspace(0.0, case["box"][2], nz))
        out["axes"] = axes
        npt = nx * ny * (nz if dim == 3 else 1)
        if case["style"] == "masked":
            shape = (ny, nx) if dim == 2 else (nz, ny, nx)
            out["mask"] = rng.uniform(size=shape) < 0.35
    if case["n_specified"]:
        # smooth specified drift fields evaluated at data and at prediction points
        def field(j, P):
            return np.cos(P[:, 0] / (180.0 + 40.0 * j)) + 0.5 * np.sin(P[:, 1] / (220.0 - 30.0 * j))
        out["spec_data"] = [field(j, xyz) for j in range(case["n_specified"])]
        if case["style"] == "points":
            out["spec_pts"] = [field(j, out["points"]) for j in range(case["n_specified"])]
        else:
            if dim == 2:
                gx, gy = np.meshgrid(out["axes"][0], out["axes"][1])
                P = np.column_stack((gx.ravel(), gy.ravel()))
                out["spec_pts"] = [field(j, P).reshape(gx.shape) for j in range(case["n_specified"])]
            else:
                gz, gy, gx = np.meshgrid(out["axes"][2], out["axes"][1], out["axes"][0], indexing="ij")
                P = np.column_stack((gx.ravel(), gy.ravel(), gz.ravel()))
                out["spec_pts"] = [field(j, P).reshape(gx.shape) for j in range(case["n_specified"])]
    if case["external_z"]:
        ex = np.linspace(-50.0, 1050.0, 45)
        ey = np.linspace(-50.0, 1050.0, 38)
        gx, gy = np.meshgrid(ex, ey)
        out["ext_x"], out["ext_y"] = ex, ey
        out["ext_z"] = 20.0 + 0.01 * gx + 5.0 * np.sin(gy / 170.0)
    return out


def make_model(module_ns, case, inp, reference=False):
    """Instantiate the kriging class named by the case from `module_ns` (the reference package or
    pykrige_b200)."""
    cls = {"OK": "OrdinaryKriging", "UK": "UniversalKriging", "OK3D": "OrdinaryKriging3D",
           "UK3D": "UniversalKriging3D"}[case["cls"]]
    K = getattr(module_ns, cls)
    xyz, val = inp["data"], inp["values"]
    kw = dict(variogram_model=case["model"], variogram_parameters=list(case["params"]),
              exact_values=case["exact_values"])
    if case.get("custom"):
        kw["variogram_function"] = CUSTOM_VARIOGRAMS[case["custom"]][0]
    kw.update(case["ctor"])
    if case["cls"] in ("UK", "UK3D"):
        kw["drift_terms"] = list(case["drift_terms"])
        if case["functional"]:
            kw["functional_drift"] = [FUNCS[f] for f in case["functional"]]
        if case["n_specified"]:
            kw["specified_drift"] = [np.array(a) for a in inp["spec_data"]]
        if case["point_log"] is not None:
            kw["point_drift"] = np.array(case["point_log"])
        if case["external_z"]:
            kw["external_drift"] = inp["ext_z"]
            kw["external_drift_x"] = inp["ext_x"]
            kw["external_drift_y"] = inp["ext_y"]
    if case["dim"] == 2:
        return K(xyz[:, 0], xyz[:, 1], val, **kw)
    return K(xyz[:, 0], xyz[:, 1], xyz[:, 2], val, **kw)


def run_model(model, case, inp, backend):
    """Call execute() the way a user would; returns (z, ss) as plain arrays + optional mask."""
    style = case["style"]
    kw = dict(backend=backend)
    if case["k"] is not None:
        kw["n_closest_points"] = case["k"]
    if case["n_specified"]:
        kw["specified_drift_arrays"] = [np.array(a) for a in inp["spec_pts"]]
    if style == "points":
        P = inp["points"]
        args = [P[:, c] for c in range(case["dim"])]
    else:
        args = list(inp["axes"])
    if style == "masked":
        kw["mask"] = inp["mask"]
    z, ss = model.execute(style, *args, **kw)
    return z, ss


# ---- constructor-side cases (SURVEY.md §8f next-2): experimental variogram + cross-validation ----
# X is what the reference hands to core._initialize_variogram_model / core._find_statistics: the
# anisotropy-ADJUSTED coordinates (lon/lat for geographic); parameters in stored form.
def _ctor_xy(case):
    rng = np.random.default_rng(case["seed"])
    kind, n, dim = case["layout"], case["n"], case["dim"]
    if kind == "lattice":                       # many pair distances coincide with lag edges
        side = int(round(n ** (1.0 / dim)))
        ax = [np.arange(side, dtype=float) * 10.0 for _ in range(dim)]
        X = np.column_stack([g.ravel() for g in np.meshgrid(*ax, indexing="ij")])
        X = X[rng.permutation(X.shape[0])]
    elif kind == "clusters":                    # two far clusters -> empty lags in between
        a = rng.normal(0.0, 5.0, (n // 2, dim))
        b = rng.normal(0.0, 5.0, (n - n // 2, dim)) + 1000.0
        X = np.vstack([a, b])
    elif kind == "geo":
        X = np.column_stack([rng.uniform(-170.0, 170.0, n), rng.uniform(-75.0, 75.0, n)])
    else:
        box = (1000.0, 1000.0, 250.0)
        X = np.column_stack([rng.uniform(0.0, box[c], n) for c in range(dim)])
    if case.get("dups"):                        # exact duplicates of earlier points (distinct values)
        for q in range(case["dups"]):
            X[n - 1 - 3 * q] = X[2 * q]
    s = 150.0 if kind != "geo" else 40.0
    y = 50.0 + 10.0 * np.sin(X[:, 0] / s) * np.cos(X[:, 1] / (1.3 * s)) + rng.normal(0.0, 1.0, X.shape[0])
    return X, y


def _e(name, layout, n, dim, nlags, seed):
    return dict(name=name, layout=layout, n=n, dim=dim, nlags=nlags, seed=seed,
                coordinates_type="geographic" if layout == "geo" else "euclidean")


VARIOGRAM_CASES = [
    _e("ev2d_n300_l6", "uniform", 300, 2, 6, 4001),
    _e("ev2d_n1500_l20", "uniform", 1500, 2, 20, 4002),
    _e("ev3d_n400_l6", "uniform", 400, 3, 6, 4003),
    _e("ev3d_n700_l50", "uniform", 700, 3, 50, 4004),       # more lags than the private-bin kernel holds
    _e("ev2d_lattice_l8", "lattice", 400, 2, 8, 4005),
    _e("ev3d_lattice_l5", "lattice", 343, 3, 5, 4006),
    _e("ev2d_clusters_l10", "clusters", 200, 2, 10, 4007),
    _e("ev2d_n2_l6", "uniform", 2, 2, 6, 4008),
    _e("ev2d_n3_l1", "uniform", 3, 2, 1, 4009),
    _e("evgeo_n250_l6", "geo", 250, 2, 6, 4010),
    _e("ev2d_n777_l37", "uniform", 777, 2, 37, 4011),       # row count not a tile multiple, max private lags
]


def _s(name, layout, n, dim, model, params, seed, **kw):
    d = dict(name=name, layout=layout, n=n, dim=dim, model=model, params=list(params), seed=seed,
             coordinates_type="geographic" if layout == "geo" else "euclidean")
    d.update(kw)
    return d


# parameters in STORED form ([psill, range, nugget] / [slope, nugget] / [scale, exponent, nugget])
STATS_CASES = [
    _s("st2d_exp_n120", "uniform", 120, 2, "exponential", [0.95, 100.0, 0.05], 5001),
    _s("st2d_gau_n80", "uniform", 80, 2, "gaussian", [0.9, 60.0, 0.1], 5002),
    _s("st3d_sph_n100", "uniform", 100, 3, "spherical", [1.0, 300.0, 0.0], 5003),
    _s("st2d_lin_n90", "uniform", 90, 2, "linear", [0.004, 0.05], 5004),
    _s("st2d_pow_n90", "uniform", 90, 2, "power", [0.002, 1.3, 0.05], 5005),
    _s("st2d_dups_n60", "uniform", 60, 2, "exponential", [0.9, 200.0, 0.1], 5006, dups=3),
    _s("stgeo_sph_n70", "geo", 70, 2, "spherical", [1.0, 60.0, 0.02], 5007),
    _s("st2d_exp_n257", "uniform", 257, 2, "exponential", [2.0, 150.0, 0.0], 5008),
]


def build_ctor_inputs(case):
    return _ctor_xy(case)


# ---- whole-chain scenarios on the reference's own small fixtures (tests/test_core.py:28-80): the
# variogram is FITTED (no parameters given), so constructor binning + least squares + execute() are all
# exercised. Reference outputs: tests/golden/ref_scenarios.npz (make_golden.py scenarios).
SAMPLE_2D = np.array([[0.3, 1.2, 0.47], [1.9, 0.6, 0.56], [1.1, 3.2, 0.74], [3.3, 4.4, 1.47], [4.7, 3.8, 1.74]])
SAMPLE_3D = np.array([[0.1, 0.1, 0.3, 0.9], [0.2, 0.1, 0.4, 0.8], [0.1, 0.3, 0.1, 0.9], [0.5, 0.4, 0.4, 0.5],
                      [0.3, 0.3, 0.2, 0.7]])


def _sc(name, cls, data, style, **kw):
    d = dict(name=name, cls=cls, data=data, style=style, ctor={}, exec={}, dim=3 if cls.endswith("3D") else 2)
    d.update(kw)
    return d


SCENARIOS = []
for _m in ("linear", "power", "gaussian", "spherical", "exponential"):
    SCENARIOS.append(_sc("val_ok_fit_" + _m, "OK", "validation", "grid", ctor=dict(variogram_model=_m)))
SCENARIOS.append(_sc("val_uk_fit_linear_rl", "UK", "validation", "grid",
                     ctor=dict(variogram_model="linear", drift_terms=["regional_linear"])))
SCENARIOS.append(_sc("val_ok_fit_spherical_weight_aniso", "OK", "validation", "grid",
                     ctor=dict(variogram_model="spherical", weight=True, nlags=8, anisotropy_scaling=2.0,
                               anisotropy_angle=30.0)))
SCENARIOS.append(_sc("val_ok_fit_exponential_stats", "OK", "validation", "grid",
                     ctor=dict(variogram_model="exponential", enable_statistics=True), stats=True))
SCENARIOS.append(_sc("s2d_ok_fit_linear_grid", "OK", "sample2d", "grid", ctor=dict(variogram_model="linear")))
SCENARIOS.append(_sc("s2d_ok_fit_linear_masked", "OK", "sample2d", "masked", ctor=dict(variogram_model="linear")))
SCENARIOS.append(_sc("s2d_ok_fit_linear_points", "OK", "sample2d", "points", ctor=dict(variogram_model="linear")))
SCENARIOS.append(_sc("s2d_uk_three_drifts", "UK", "sample2d", "grid",
                     ctor=dict(variogram_model="linear", drift_terms=["regional_linear", "external_Z", "point_log"]),
                     three_drifts=True))
SCENARIOS.append(_sc("s3d_ok_fit_linear_grid", "OK3D", "sample3d", "grid", ctor=dict(variogram_model="linear")))
SCENARIOS.append(_sc("s3d_uk_fit_linear_rl_masked", "UK3D", "sample3d", "masked",
                     ctor=dict(variogram_model="linear", drift_terms=["regional_linear"]), stats=True))
SCENARIOS.append(_sc("s3d_ok_fit_power_points", "OK3D", "sample3d", "points", ctor=dict(variogram_model="power"),
                     stats=True))


# ---- variogram_model='custom' (ok.py:224-253; tests/test_core.py:1837-1911): user callables f(params, d).
# Callables cannot live in fixtures, so they are named here; reference outputs: tests/golden/ref_custom.npz.
CUSTOM_VARIOGRAMS = {
    # the reference's own test function (tests/test_core.py:1840-1841)
    "log10": (lambda m, d: m[0] * np.log10(d + m[1]) + m[2], [1.0, 1.0, 1.0]),
    "log10_short": (lambda m, d: m[0] * np.log10(d + m[1]) + m[2], [0.5, 0.05, 1.0]),
    # nested structure: exponential + spherical + nugget
    "nested": (lambda m, d: m[0] * (1.0 - np.exp(-d / m[1])) + m[2] * np.where(
        d <= m[3], 1.5 * d / m[3] - 0.5 * (d / m[3]) ** 3, 1.0) + m[4], [0.6, 50.0, 0.4, 700.0, 0.02]),
    "sqrt": (lambda m, d: m[0] * np.sqrt(d) + m[1], [0.05, 0.1]),
    "cubic": (lambda m, d: m[0] * np.where(d < m[1], 7 * (d / m[1]) ** 2 - 8.75 * (d / m[1]) ** 3 + 3.5 * (d / m[1]) ** 5
                                           - 0.75 * (d / m[1]) ** 7, 1.0) + m[2], [1.0, 450.0, 0.05]),
}


def _cu(name, cls, n, m, seed, fn, **kw):
    c = _c(name, cls, n, m, seed, "linear", params=list(CUSTOM_VARIOGRAMS[fn][1]), **kw)
    c["model"] = "custom"
    c["custom"] = fn
    return c


CUSTOM_CASES = [
    _cu("custom_ok2d_log10", "OK", 150, 200, 8001, "log10"),
    _cu("custom_ok2d_log10_short_nonexact", "OK", 120, 150, 8002, "log10_short", exact_values=False),
    _cu("custom_ok2d_nested_grid_aniso", "OK", 200, 0, 8003, "nested", style="grid", grid=(21, 16, 1),
        ctor=dict(anisotropy_scaling=1.7, anisotropy_angle=25.0)),
    _cu("custom_uk2d_sqrt_rl", "UK", 140, 160, 8004, "sqrt", drift_terms=["regional_linear"]),
    _cu("custom_ok3d_cubic", "OK3D", 160, 150, 8005, "cubic"),
    _cu("custom_uk3d_nested_rl_masked", "UK3D", 120, 0, 8006, "nested", style="masked", grid=(9, 8, 5),
        drift_terms=["regional_linear"]),
    _cu("custom_knn2d_log10_k12", "OK", 400, 200, 8007, "log10", k=12, ref_backend="loop"),
    _cu("custom_geo_sqrt", "OK", 150, 120, 8008, "sqrt", geographic=True, box=(60.0, 45.0, 1.0),
        ctor=dict(coordinates_type="geographic")),
]


def scenario_inputs(sc, validation_data):
    """(data array, execute args, execute kwargs) of a scenario; `validation_data` is the 15-point KT3D_H2O
    set stored in reference_goldens.npz (tests/test_core.py:28-31)."""
    if sc["data"] == "validation":
        data = np.asarray(validation_data)
        args = [np.linspace(1067000.0, 1072000.0, 40), np.linspace(241500.0, 244000.0, 30)]
    elif sc["data"] == "sample2d":
        data = SAMPLE_2D
        args = [np.arange(0.0, 6.0, 1.0), np.arange(0.0, 5.5, 0.5)]
    else:
        data = SAMPLE_3D
        args = [np.arange(0.0, 0.6, 0.05), np.arange(0.0, 0.6, 0.01), np.arange(0.0, 0.6, 0.1)]
    kw = {}
    if sc["style"] == "masked":
        if sc["dim"] == 2:
            xi, yi = np.meshgrid(args[0], args[1])
            kw["mask"] = np.array(xi == yi)
        else:
            zi, yi, xi = np.meshgrid(args[2], args[1], args[0], indexing="ij")
            kw["mask"] = np.array((xi == yi) & (yi == zi))
    if sc["style"] == "points":
        rng = np.random.default_rng(99)
        lo, hi = data[:, :sc["dim"]].min(axis=0), data[:, :sc["dim"]].max(axis=0)
        P = rng.uniform(lo, hi, (25, sc["dim"]))
        P[:3] = data[:3, :sc["dim"]]                      # exact hits
        args = [P[:, c] for c in range(sc["dim"])]
    return data, args, kw


def scenario_model(module_ns, sc, data):
    cls = {"OK": "OrdinaryKriging", "UK": "UniversalKriging", "OK3D": "OrdinaryKriging3D",
           "UK3D": "UniversalKriging3D"}[sc["cls"]]
    kw = dict(sc["ctor"])
    if sc.get("three_drifts"):                            # tests/test_core.py:1222-1238
        dem = np.repeat(np.arange(0.0, 5.1, 0.1)[np.newaxis, :], 6, axis=0)
        kw.update(point_drift=np.array([[1.1, 1.1, -1.0]]), external_drift=dem,
                  external_drift_x=np.arange(0.0, 5.1, 0.1), external_drift_y=np.arange(0.0, 6.0, 1.0))
    cols = [data[:, c] for c in range(data.shape[1])]
    return getattr(module_ns, cls)(*cols, **kw)


# ---- automatic variogram fit (variogram_parameters=None) and bit patterns of the six model functions:
#      inputs shared by tests/golden/make_golden.py (vgfit) and tests/test_host.py -> tests/golden/ref_vgfit.npz
def vgfit_inputs(n, seed=77):
    """Seeded scatter for the automatic-fit cases."""
    rng = np.random.default_rng(seed + n)
    x = rng.uniform(0.0, 1000.0, n)
    y = rng.uniform(0.0, 1000.0, n)
    z = 50.0 + 10.0 * np.sin(x / 150.0) * np.cos(y / 200.0) + rng.normal(size=n)
    return x, y, z


VGFIT_MODELS = ("linear", "power", "gaussian", "spherical", "exponential", "hole-effect")
VGFIT_PARAMS = {"linear": [0.002, 0.1], "power": [0.05, 1.3, 0.1], "gaussian": [1.3, 420.0, 0.07],
                "spherical": [0.9, 510.0, 0.03], "exponential": [1.1, 333.0, 0.05], "hole-effect": [0.8, 270.0, 0.02]}


def vgfit_distances():
    rng = np.random.default_rng(4242)
    return np.concatenate([[0.0, 1e-12, 510.0, 509.99999999999994, 510.00000000000006], rng.uniform(0.0, 1500.0, 1019)])


def cpu_fingerprint():
    """numpy version + the SIMD features its ufunc loops dispatch on (exp / pow may differ in the last ulp between
    dispatch targets, so bit-for-bit comparisons are only meaningful on the same fingerprint)."""
    try:
        from numpy._core._multiarray_umath import __cpu_features__ as feats
    except ImportError:  # numpy < 2
        from numpy.core._multiarray_umath import __cpu_features__ as feats
    return np.__version__ + ":" + ",".join(sorted(k for k, v in feats.items() if v))


# ---- host-mirror API cases: constructor / update_variogram_model / execute()-argument validation of the four classes,
#      run against the imported reference by tests/golden/make_golden.py (api) -> tests/golden/ref_api.npz and against
#      pykrige_b200 by tests/test_host.py. Everything before the device call: attributes, stdout, warnings, exceptions.
API_FUNCS = {
    "f_xy": lambda x, y: x * y / 100.0,
    "f_sin": lambda x, y: np.sin(x / 30.0),
    "f_xyz": lambda x, y, z: x + y * z / 50.0,
    "vg_lin": lambda m, d: m[0] * d,
}


def api_inputs():
    """Named arrays the API cases refer to as '$name'."""
    rng = np.random.default_rng(20260923)
    n = 40
    x, y, zc = rng.uniform(0, 100, n), rng.uniform(0, 100, n), rng.uniform(0, 30, n)
    v = 10.0 + np.sin(x / 20.0) + 0.3 * rng.normal(size=n)
    d = dict(x=x, y=y, zc=zc, v=v, gx=np.linspace(0, 100, 7), gy=np.linspace(0, 100, 5), gz=np.linspace(0, 30, 3),
             dem=rng.uniform(0, 5, (12, 11)), demx=np.linspace(-5, 105, 11), demy=np.linspace(-5, 105, 12),
             wells=np.array([[10.0, 20.0, 1.0], [70.0, 80.0, -2.0]]), sx=0.1 * x, sy=0.2 * y, szc=zc.copy(),
             mask2=np.zeros((5, 7), bool), mask3=np.zeros((3, 5, 7), bool), z57=np.zeros((5, 7)), z75=np.zeros((7, 5)),
             z47=np.zeros((4, 7)), z7=np.zeros(7), z5=np.zeros(5), z4=np.zeros(4), z51=np.zeros((5, 1)),
             z357=np.zeros((3, 5, 7)), z753=np.zeros((7, 5, 3)), z3=np.zeros(3))
    d["mask2"][1, 2] = True
    d["wells2"] = d["wells"][:, :2]
    d["demx_short"] = d["demx"][:-1]
    d["sx_short"] = d["sx"][:-1]
    d["gx5"], d["gx3"], d["gy3"], d["gy4"] = d["gx"][:5], d["gx"][:3], d["gy"][:3], d["gy"][:4]
    d["mask2T"], d["mask2_rows3"], d["mask2_1d"] = d["mask2"].T, d["mask2"][:3], d["mask2"][0]
    d["mask3T"], d["mask3_2"], d["mask3_2d"] = d["mask3"].T, d["mask3"][:2], d["mask3"][0]
    d.update(API_FUNCS)
    return d


def _api(name, cls, kw=None, then=None):
    return dict(name=name, cls=cls, kw=dict(kw or {}), then=then)


_VP = {"linear": [0.01, 0.1], "power": [0.1, 1.2, 0.05]}
API_CASES = []
for _m in ("linear", "power", "gaussian", "spherical", "exponential", "hole-effect"):
    _lst = _VP.get(_m, [2.0, 40.0, 0.1])
    _dct = ({"slope": 1.0, "nugget": 0.1} if _m == "linear" else
            {"scale": 0.1, "exponent": 1.2, "nugget": 0.05} if _m == "power" else {"sill": 2.0, "range": 40.0, "nugget": 0.1})
    for _tag, _kw in (("fit", {}), ("fit_weight", dict(weight=True, nlags=4)),
                      ("aniso_verbose", dict(anisotropy_scaling=2.5, anisotropy_angle=33.0, verbose=True)),
                      ("stats_verbose", dict(enable_statistics=True, verbose=True)),
                      ("list", dict(variogram_parameters=_lst)), ("dict", dict(variogram_parameters=_dct)),
                      ("geographic", dict(coordinates_type="geographic", verbose=True))):
        API_CASES.append(_api("ok_%s_%s" % (_m, _tag), "OrdinaryKriging", dict(variogram_model=_m, **_kw)))
API_CASES += [
    _api("ok_psill_dict", "OrdinaryKriging", dict(variogram_model="gaussian", variogram_parameters={"psill": 1.0, "range": 40.0, "nugget": 0.1})),
    _api("ok_bad_list_len", "OrdinaryKriging", dict(variogram_model="gaussian", variogram_parameters=[1.0])),
    _api("ok_bad_param_type", "OrdinaryKriging", dict(variogram_model="gaussian", variogram_parameters="bad")),
    _api("ok_bad_dict_keys", "OrdinaryKriging", dict(variogram_model="power", variogram_parameters={"scale": 1.0})),
    _api("ok_bad_model", "OrdinaryKriging", dict(variogram_model="nomodel")),
    _api("ok_custom_no_function", "OrdinaryKriging", dict(variogram_model="custom", variogram_parameters=[1.0])),
    _api("ok_custom_no_parameters", "OrdinaryKriging", dict(variogram_model="custom", variogram_function="$vg_lin")),
    _api("ok_custom", "OrdinaryKriging", dict(variogram_model="custom", variogram_parameters=[0.02], variogram_function="$vg_lin", verbose=True)),
    _api("ok_pinvh", "OrdinaryKriging", dict(exact_values=False, pseudo_inv=True, pseudo_inv_type="pinvh", enable_statistics=True)),
    _api("ok_bad_pinv_type", "OrdinaryKriging", dict(pseudo_inv_type="zzz")),
    _api("ok_bad_coordinates", "OrdinaryKriging", dict(coordinates_type="nonsense")),
    _api("ok_bad_exact", "OrdinaryKriging", dict(exact_values="yes")),
    _api("ok_geo_aniso_warns", "OrdinaryKriging", dict(coordinates_type="geographic", anisotropy_scaling=2.0)),
]
_UKW = dict(variogram_model="linear", variogram_parameters=[0.01, 0.1])
_ALL5 = dict(drift_terms=["regional_linear", "point_log", "external_Z", "specified", "functional"], point_drift="$wells",
             external_drift="$dem", external_drift_x="$demx", external_drift_y="$demy", specified_drift=["$sx"],
             functional_drift=["$f_xy"], verbose=True, anisotropy_scaling=1.5, anisotropy_angle=20.0)
API_CASES += [
    _api("uk_plain_verbose", "UniversalKriging", dict(variogram_model="spherical", verbose=True)),
    _api("uk_rl_verbose", "UniversalKriging", dict(variogram_model="spherical", drift_terms=["regional_linear"], verbose=True)),
    _api("uk_external", "UniversalKriging", dict(drift_terms=["external_Z"], external_drift="$dem", external_drift_x="$demx", external_drift_y="$demy", verbose=True)),
    _api("uk_external_missing", "UniversalKriging", dict(drift_terms=["external_Z"])),
    _api("uk_external_bad_axis", "UniversalKriging", dict(drift_terms=["external_Z"], external_drift="$dem", external_drift_x="$demx_short", external_drift_y="$demy")),
    _api("uk_point_log", "UniversalKriging", dict(drift_terms=["point_log"], point_drift="$wells", verbose=True)),
    _api("uk_point_log_missing", "UniversalKriging", dict(drift_terms=["point_log"])),
    _api("uk_point_log_two_columns", "UniversalKriging", dict(drift_terms=["point_log"], point_drift="$wells2")),
    _api("uk_specified", "UniversalKriging", dict(drift_terms=["specified"], specified_drift=["$sx", "$sy"], verbose=True)),
    _api("uk_specified_missing", "UniversalKriging", dict(drift_terms=["specified"])),
    _api("uk_specified_not_list", "UniversalKriging", dict(drift_terms=["specified"], specified_drift="$sx")),
    _api("uk_specified_short", "UniversalKriging", dict(drift_terms=["specified"], specified_drift=["$sx_short"])),
    _api("uk_functional", "UniversalKriging", dict(drift_terms=["functional"], functional_drift=["$f_xy", "$f_sin"], verbose=True)),
    _api("uk_functional_missing", "UniversalKriging", dict(drift_terms=["functional"])),
    _api("uk_functional_not_list", "UniversalKriging", dict(drift_terms=["functional"], functional_drift="$f_xy")),
    _api("uk_bogus_term", "UniversalKriging", dict(drift_terms=["bogus"])),
    _api("uk_all_five", "UniversalKriging", _ALL5),
    _api("uk_pinv", "UniversalKriging", dict(exact_values=False, pseudo_inv=True)),
    _api("uk_bad_pinv_type", "UniversalKriging", dict(pseudo_inv_type="x")),
    _api("uk_bad_exact", "UniversalKriging", dict(exact_values=1)),
    _api("ok3d_fit_verbose", "OrdinaryKriging3D", dict(variogram_model="gaussian", verbose=True)),
    _api("ok3d_aniso_verbose", "OrdinaryKriging3D", dict(anisotropy_scaling_y=2.0, anisotropy_scaling_z=0.5, anisotropy_angle_x=10.0,
                                                         anisotropy_angle_y=20.0, anisotropy_angle_z=30.0, verbose=True)),
    _api("ok3d_list", "OrdinaryKriging3D", dict(variogram_model="gaussian", variogram_parameters=[2.0, 40.0, 0.1])),
    _api("ok3d_weight", "OrdinaryKriging3D", dict(nlags=3, weight=True)),
    _api("ok3d_pinvh", "OrdinaryKriging3D", dict(exact_values=False, pseudo_inv=True, pseudo_inv_type="pinvh")),
    _api("ok3d_bad_pinv_type", "OrdinaryKriging3D", dict(pseudo_inv_type="q")),
    _api("ok3d_bad_exact", "OrdinaryKriging3D", dict(exact_values=None)),
    _api("uk3d_rl_verbose", "UniversalKriging3D", dict(drift_terms=["regional_linear"], verbose=True)),
    _api("uk3d_specified", "UniversalKriging3D", dict(drift_terms=["specified"], specified_drift=["$sx", "$szc"])),
    _api("uk3d_specified_missing", "UniversalKriging3D", dict(drift_terms=["specified"])),
    _api("uk3d_specified_not_list", "UniversalKriging3D", dict(drift_terms=["specified"], specified_drift="$sx")),
    _api("uk3d_specified_short", "UniversalKriging3D", dict(drift_terms=["specified"], specified_drift=["$sx_short"])),
    _api("uk3d_functional", "UniversalKriging3D", dict(drift_terms=["functional"], functional_drift=["$f_xyz"], verbose=True)),
    _api("uk3d_functional_missing", "UniversalKriging3D", dict(drift_terms=["functional"])),
    _api("uk3d_functional_not_list", "UniversalKriging3D", dict(drift_terms=["functional"], functional_drift="$f_xyz")),
    _api("uk3d_bogus_term", "UniversalKriging3D", dict(drift_terms=["zzz"])),
    _api("uk3d_all", "UniversalKriging3D", dict(variogram_model="gaussian", anisotropy_scaling_y=2.0, anisotropy_angle_z=30.0,
                                                 drift_terms=["regional_linear", "specified", "functional"], specified_drift=["$sx"],
                                                 functional_drift=["$f_xyz"], verbose=True)),
]
# update_variogram_model on a verbose object (ok.py:379-553, uk.py:630-790, ok3d.py:354-520, uk3d.py)
for _cls, _base, _an in (("OrdinaryKriging", _UKW, dict(anisotropy_scaling=2.0, anisotropy_angle=10.0)),
                         ("UniversalKriging", dict(_UKW, drift_terms=["regional_linear"]), dict(anisotropy_scaling=2.0, anisotropy_angle=10.0)),
                         ("OrdinaryKriging3D", _UKW, dict(anisotropy_scaling_y=2.0, anisotropy_angle_z=10.0)),
                         ("UniversalKriging3D", dict(_UKW, drift_terms=["regional_linear"]), dict(anisotropy_scaling_y=2.0, anisotropy_angle_z=10.0))):
    _s = {"OrdinaryKriging": "ok", "UniversalKriging": "uk", "OrdinaryKriging3D": "ok3d", "UniversalKriging3D": "uk3d"}[_cls]
    for _tag, _a, _k in (("to_spherical_fit", ("spherical",), {}), ("to_gaussian_list", ("gaussian", [2.0, 30.0, 0.1]), {}),
                         ("new_anisotropy", ("linear",), _an), ("bad_model", ("nomodel",), {}), ("custom_missing", ("custom",), {}),
                         ("to_power_dict", ("power", {"scale": 1.0, "exponent": 1.1, "nugget": 0.0}), dict(nlags=4, weight=True))):
        API_CASES.append(_api("%s_update_%s" % (_s, _tag), _cls, dict(_base, verbose=True), ("update_variogram_model", _a, _k)))
    API_CASES.append(_api("%s_get_statistics" % _s, _cls, _base, ("get_statistics", (), {})))
    API_CASES.append(_api("%s_print_statistics" % _s, _cls, _base, ("print_statistics", (), {})))
# execute(): argument validation that precedes the backend dispatch (ok.py:834-874, uk.py:1169-1274, ok3d.py:833-876,
# uk3d.py:981-1098) — every case raises in the reference before any arithmetic
_US = dict(_UKW, drift_terms=["specified"], specified_drift=["$sx"])
for _s, _cls, _kw in (("ok", "OrdinaryKriging", _UKW), ("uk", "UniversalKriging", dict(_UKW, drift_terms=["regional_linear"]))):
    for _tag, _a, _k in (("bad_style", ("bogus", "$gx", "$gy"), {}), ("masked_no_mask", ("masked", "$gx", "$gy"), {}),
                         ("masked_bad_shape", ("masked", "$gx", "$gy"), dict(mask="$mask2_rows3")),
                         ("masked_1d", ("masked", "$gx", "$gy"), dict(mask="$mask2_1d")),
                         ("points_mismatch", ("points", "$gx", "$gy"), {})):
        API_CASES.append(_api("%s_execute_%s" % (_s, _tag), _cls, _kw, ("execute", _a, _k)))
API_CASES += [
    _api("ok_execute_k1", "OrdinaryKriging", _UKW, ("execute", ("grid", "$gx", "$gy"), dict(n_closest_points=1))),
    _api("ok_execute_k0", "OrdinaryKriging", _UKW, ("execute", ("grid", "$gx", "$gy"), dict(n_closest_points=0))),
    _api("uk_execute_spec_missing", "UniversalKriging", _US, ("execute", ("grid", "$gx", "$gy"), {})),
    _api("uk_execute_spec_not_list", "UniversalKriging", _US, ("execute", ("grid", "$gx", "$gy"), dict(specified_drift_arrays="$z57"))),
    _api("uk_execute_spec_bad_shape", "UniversalKriging", _US, ("execute", ("grid", "$gx", "$gy"), dict(specified_drift_arrays=["$z47"]))),
    _api("uk_execute_spec_1d_on_grid", "UniversalKriging", _US, ("execute", ("grid", "$gx", "$gy"), dict(specified_drift_arrays=["$z7"]))),
    _api("uk_execute_spec_points_len", "UniversalKriging", _US, ("execute", ("points", "$gx5", "$gy"), dict(specified_drift_arrays=["$z4"]))),
    _api("uk_execute_spec_points_2d", "UniversalKriging", _US, ("execute", ("points", "$gx5", "$gy"), dict(specified_drift_arrays=["$z51"]))),
    _api("uk_execute_spec_count", "UniversalKriging", _US, ("execute", ("grid", "$gx", "$gy"), dict(specified_drift_arrays=["$z57", "$z57"]))),
]
_U3S = dict(_UKW, drift_terms=["specified"], specified_drift=["$sx"])
for _s, _cls, _kw in (("ok3d", "OrdinaryKriging3D", _UKW), ("uk3d", "UniversalKriging3D", dict(_UKW, drift_terms=["regional_linear"]))):
    for _tag, _a, _k in (("bad_style", ("bogus", "$gx", "$gy", "$gz"), {}), ("masked_no_mask", ("masked", "$gx", "$gy", "$gz"), {}),
                         ("masked_bad_shape", ("masked", "$gx", "$gy", "$gz"), dict(mask="$mask3_2")),
                         ("masked_2d", ("masked", "$gx", "$gy", "$gz"), dict(mask="$mask3_2d")),
                         ("points_mismatch", ("points", "$gx3", "$gy4", "$gz"), {})):
        API_CASES.append(_api("%s_execute_%s" % (_s, _tag), _cls, _kw, ("execute", _a, _k)))
API_CASES += [
    _api("uk3d_execute_spec_missing", "UniversalKriging3D", _U3S, ("execute", ("grid", "$gx", "$gy", "$gz"), {})),
    _api("uk3d_execute_spec_not_list", "UniversalKriging3D", _U3S, ("execute", ("grid", "$gx", "$gy", "$gz"), dict(specified_drift_arrays="$z357"))),
    _api("uk3d_execute_spec_bad_shape", "UniversalKriging3D", _U3S, ("execute", ("grid", "$gx", "$gy", "$gz"), dict(specified_drift_arrays=["$z57"]))),
    _api("uk3d_execute_spec_points_len", "UniversalKriging3D", _U3S, ("execute", ("points", "$gx3", "$gy3", "$gz"), dict(specified_drift_arrays=["$z4"]))),
    _api("uk3d_execute_spec_count", "UniversalKriging3D", _U3S, ("execute", ("grid", "$gx", "$gy", "$gz"), dict(specified_drift_arrays=["$z357", "$z357"]))),
]

API_STAT_ATTRS = ("delta", "sigma", "epsilon", "Q1", "Q2", "cR")


def _api_resolve(v, named):
    if isinstance(v, str) and v.startswith("$"):
        return named[v[1:]]
    if isinstance(v, list):
        return [_api_resolve(q, named) for q in v]
    if isinstance(v, tuple):
        return tuple(_api_resolve(q, named) for q in v)
    if isinstance(v, dict):
        return {k: _api_resolve(q, named) for k, q in v.items()}
    return v


def api_run(module_ns, case, named, backend):
    """Run one API case against `module_ns` (the imported reference or pykrige_b200). Returns a record:
    kind 'ok' | 'exc', exception type and message, captured stdout, warning categories, and the public attributes of
    the object (numeric ones as float arrays, strings/bools/None as they are; callables by __name__)."""
    import contextlib
    import io
    import warnings
    is3 = case["cls"].endswith("3D")
    args = (named["x"], named["y"], named["zc"], named["v"]) if is3 else (named["x"], named["y"], named["v"])
    kw = _api_resolve(case["kw"], named)
    rec = dict(kind="ok", exc="", msg="", stdout="", warnings=[], attrs={}, ret=None)
    buf = io.StringIO()
    obj = None
    try:
        with contextlib.redirect_stdout(buf), warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            obj = getattr(module_ns, case["cls"])(*args, **kw)
            if case["then"] is not None:
                meth, a, k = case["then"]
                k = dict(_api_resolve(k, named))
                if meth == "execute":
                    k["backend"] = backend
                ret = getattr(obj, meth)(*_api_resolve(a, named), **k)
                if meth == "get_statistics":
                    rec["ret"] = np.asarray(ret, dtype=float)
        rec["warnings"] = [x.category.__name__ for x in w]
    except Exception as e:  # noqa: BLE001  (the exception IS the observation)
        rec.update(kind="exc", exc=type(e).__name__, msg=str(e))
    rec["stdout"] = buf.getvalue()
    if obj is not None and rec["kind"] == "ok":
        names = [k for k in vars(obj) if not k.startswith("_")]
        names += [k for k in ("lags", "semivariance") + API_STAT_ATTRS if k not in names]
        for k in names:
            try:
                val = getattr(obj, k)
            except AttributeError:
                continue
            if k == "variogram_dict" or isinstance(val, dict):
                continue
            if callable(val):
                rec["attrs"][k] = "callable:" + getattr(val, "__name__", "?")
            elif val is None or isinstance(val, (str, bool)):
                rec["attrs"][k] = val
            elif isinstance(val, (list, tuple)) and any(callable(q) for q in val):
                rec["attrs"][k] = "callables:" + ",".join(getattr(q, "__name__", "?") for q in val)
            else:
                try:
                    rec["attrs"][k] = np.asarray(val, dtype=float)
                except (TypeError, ValueError):
                    pass
    return rec


# ---- randomised whole-execute() configurations (tests/golden/make_golden.py fuzz -> ref_fuzz.npz; replayed through the
#      host wrappers on the C-ABI emulator by tests/test_host_execute_emulated.py): classes x styles x drift kinds x
#      anisotropy x exact_values x moving window, masks and specified-drift arrays also in the transposed orientation the
#      reference tolerates (ok.py:855-859, uk.py:1232-1240), rasters with a descending axis, exact hits ----
N_FUZZ = 240
_FUZZ_MODELS = ("linear", "power", "gaussian", "spherical", "exponential")


def _fuzz_f2(x, y):
    return np.sin(x / 40.0) * y / 50.0


def _fuzz_f3(x, y, z):
    return np.sin(x / 40.0) * y / 50.0 + z / 30.0


def fuzz_config(t):
    """Deterministic configuration number t, or None when the draw is over-determined (more drift terms than data)."""
    rng = np.random.default_rng(7_000_000 + t)
    dim = 3 if rng.uniform() < 0.4 else 2
    uk = rng.uniform() < 0.5
    n = int(rng.integers(8, 60))
    X = rng.uniform(0, 100, (n, dim))
    if dim == 3:
        X[:, 2] *= 0.3
    v = 5 + np.sin(X[:, 0] / 20) + 0.02 * X[:, 1] + rng.normal(size=n) * 0.3
    m = _FUZZ_MODELS[rng.integers(len(_FUZZ_MODELS))]
    if m == "linear":
        vp = [float(rng.uniform(0.001, 0.01)), float(rng.uniform(0, 0.2))]
    elif m == "power":
        vp = [float(rng.uniform(0.001, 0.01)), float(rng.uniform(0.5, 1.6)), float(rng.uniform(0, 0.2))]
    else:
        vp = [float(rng.uniform(0.8, 2.5)), float(rng.uniform(20.0, 90.0)), float(rng.uniform(0.01, 0.3))]
    kw = dict(variogram_model=m, variogram_parameters=vp)
    if rng.uniform() < 0.5:
        if dim == 2:
            kw.update(anisotropy_scaling=float(rng.uniform(0.3, 3)), anisotropy_angle=float(rng.uniform(-90, 90)))
        else:
            kw.update(anisotropy_scaling_y=float(rng.uniform(0.3, 3)), anisotropy_scaling_z=float(rng.uniform(0.3, 3)),
                      anisotropy_angle_x=float(rng.uniform(-90, 90)), anisotropy_angle_y=float(rng.uniform(-90, 90)),
                      anisotropy_angle_z=float(rng.uniform(-90, 90)))
    if rng.uniform() < 0.25:
        kw["exact_values"] = False
    ekw = {}
    nx, ny, nz = int(rng.integers(1, 7)), int(rng.integers(1, 7)), int(rng.integers(1, 5))
    gx, gy, gz = np.sort(rng.uniform(0, 100, nx)), np.sort(rng.uniform(0, 100, ny)), np.sort(rng.uniform(0, 30, nz))
    style = ("grid", "masked", "points")[rng.integers(3)]
    if style == "points":
        npnt = int(rng.integers(1, 12))
        gx, gy, gz = rng.uniform(0, 100, npnt), rng.uniform(0, 100, npnt), rng.uniform(0, 30, npnt)
        if npnt > 1 and rng.uniform() < 0.5:          # an exact hit on a data point (not as the only point: sigma^2 = 0)
            gx[0], gy[0] = X[0, 0], X[0, 1]
            if dim == 3:
                gz[0] = X[0, 2]
        nx = ny = nz = npnt
    shape = (ny, nx) if dim == 2 else (nz, ny, nx)
    distinct = len(set(shape)) == len(shape)
    if style == "masked":
        mask = rng.uniform(size=shape) < 0.4
        if rng.uniform() < 0.3 and distinct:
            mask = mask.T if dim == 2 else mask.swapaxes(0, 2)
        ekw["mask"] = mask
    cls = ("Universal" if uk else "Ordinary") + "Kriging" + ("3D" if dim == 3 else "")
    terms = []
    if uk:
        if rng.uniform() < 0.6:
            terms.append("regional_linear")
        if dim == 2 and rng.uniform() < 0.4:
            terms.append("point_log")
            kw["point_drift"] = np.column_stack([rng.uniform(0, 100, 2), rng.uniform(0, 100, 2), rng.uniform(-2, 2, 2)])
        if dim == 2 and rng.uniform() < 0.4:
            terms.append("external_Z")
            ex = np.linspace(-10, 110, int(rng.integers(3, 9)))
            ey = np.linspace(-10, 110, int(rng.integers(3, 9)))
            if rng.uniform() < 0.3:
                ey = ey[::-1].copy()
            kw.update(external_drift=rng.uniform(0, 5, (ey.size, ex.size)), external_drift_x=ex, external_drift_y=ey)
        if rng.uniform() < 0.4:
            terms.append("specified")
            kw["specified_drift"] = [1e-3 * X[:, 0] * X[:, 1]]
            if style == "points":
                ekw["specified_drift_arrays"] = [1e-3 * gx * gy]
            else:
                g = 1e-3 * gx[None, :] * gy[:, None]
                if dim == 3:
                    g = np.broadcast_to(g, (nz, ny, nx)).copy()
                if rng.uniform() < 0.3 and distinct:
                    g = g.T if dim == 2 else g.swapaxes(0, 2)
                ekw["specified_drift_arrays"] = [g]
        if rng.uniform() < 0.4:
            terms.append("functional")
            kw["functional_drift"] = [_fuzz_f2] if dim == 2 else [_fuzz_f3]
        kw["drift_terms"] = terms
        n_terms = ((dim if "regional_linear" in terms else 0) + (2 if "point_log" in terms else 0)
                   + sum(q in terms for q in ("external_Z", "specified", "functional")))
        if n < n_terms + 3:
            return None
    knn = None
    if not uk and rng.uniform() < 0.3:
        knn = int(rng.integers(2, min(n, 9)))
        ekw["n_closest_points"] = knn
    data = (X[:, 0], X[:, 1], v) if dim == 2 else (X[:, 0], X[:, 1], X[:, 2], v)
    pts = (gx, gy) if dim == 2 else (gx, gy, gz)
    return dict(t=t, cls=cls, data=data, kw=kw, style=style, pts=pts, ekw=ekw, knn=knn,
                text="%s n=%d %s %s %s terms=%s knn=%s" % (cls, n, m, style, shape, terms, knn))


# ---- stateful sequences: execute / update_variogram_model (also with a new anisotropy) / execute on ONE object
#      (tests/golden/make_golden.py fuzz -> ref_fuzz.npz keys 'seq<t>/<step>/z|ss'): the problem cache must follow the
#      variogram and the re-adjusted data, functional drift sees the new frame, point_log wells keep the frame they were
#      adjusted in at construction (the reference does not re-adjust them, uk.py:630-790) ----
N_SEQ = 60


def seq_config(t):
    rng = np.random.default_rng(8_000_000 + t)
    dim = 3 if rng.uniform() < 0.4 else 2
    uk = rng.uniform() < 0.6
    n = int(rng.integers(12, 40))
    X = rng.uniform(0, 100, (n, dim))
    v = 5 + np.sin(X[:, 0] / 20) + rng.normal(size=n) * 0.3
    cls = ("Universal" if uk else "Ordinary") + "Kriging" + ("3D" if dim == 3 else "")
    kw = dict(variogram_model="exponential", variogram_parameters=[1.5, 40.0, 0.1])
    if uk:
        terms = ["regional_linear"] if rng.uniform() < 0.5 else []
        if dim == 2 and rng.uniform() < 0.5:
            terms.append("point_log")
            kw["point_drift"] = np.array([[30.0, 40.0, 1.0], [70.0, 20.0, -1.5]])
        if rng.uniform() < 0.5:
            terms.append("functional")
            kw["functional_drift"] = [_fuzz_f2 if dim == 2 else _fuzz_f3]
        kw["drift_terms"] = terms
    data = (X[:, 0], X[:, 1], v) if dim == 2 else (X[:, 0], X[:, 1], X[:, 2], v)
    pts = (np.sort(rng.uniform(0, 100, 4)), np.sort(rng.uniform(0, 100, 3)), np.sort(rng.uniform(0, 100, 2)))[:dim]
    steps = []
    for _ in range(int(rng.integers(2, 5))):
        if rng.uniform() < 0.45:
            steps.append(("exec",))
            continue
        m = ("linear", "gaussian", "spherical", "power")[rng.integers(4)]
        p = {"linear": [0.01, 0.1], "power": [0.01, 1.2, 0.1]}.get(m) or [float(rng.uniform(1, 2)), float(rng.uniform(20, 80)), 0.1]
        an = {}
        if rng.uniform() < 0.6:
            an = (dict(anisotropy_scaling=float(rng.uniform(0.5, 2)), anisotropy_angle=float(rng.uniform(-60, 60))) if dim == 2
                  else dict(anisotropy_scaling_y=float(rng.uniform(0.5, 2)), anisotropy_angle_z=float(rng.uniform(-60, 60))))
        steps.append(("upd", m, p, an))
    steps.append(("exec",))
    return dict(cls=cls, data=data, kw=kw, pts=pts, steps=steps, text="%s %s %s" % (cls, kw.get("drift_terms"), steps))


def seq_run(module_ns, c, backend):
    """Replay the sequence; returns the (z, ss) of every 'exec' step."""
    obj = getattr(module_ns, c["cls"])(*c["data"], **c["kw"])
    outs = []
    for st in c["steps"]:
        if st[0] == "upd":
            obj.update_variogram_model(st[1], st[2], **st[3])
        else:
            z, ss = obj.execute("grid", *c["pts"], backend=backend)
            outs.append((np.asarray(z), np.asarray(ss)))
    return outs


# ---- more randomised draws, CPU replay only (the device side of these kinds is covered by the seeded GPU cases):
#      geographic coordinates, pseudo_inv with redundant points, exact duplicates WITHOUT pseudo_inv (the reference's
#      scipy.linalg.inv raises LinAlgError), custom variogram callables incl. UK and anisotropy, all with and without the
#      moving window -> ref_fuzz.npz keys 'kind<t>/...' ----
N_KIND = 160
_KIND_CUSTOMS = ((lambda m, d: m[0] * np.log10(d + m[1]) + m[2], [1.0, 1.0, 1.0]), (lambda m, d: m[0] * np.sqrt(d) + m[1], [0.05, 0.1]))


def kind_config(t):
    rng = np.random.default_rng(9_000_000 + t)
    kind = ("geo", "pinv", "custom", "dups")[t % 4]
    n = int(rng.integers(10, 50))
    dim = 2
    if kind == "geo":
        X = np.column_stack([rng.uniform(-170, 170, n), rng.uniform(-80, 80, n)])
    else:
        dim = 3 if rng.uniform() < 0.3 else 2
        X = rng.uniform(0, 100, (n, dim))
    v = 5 + np.sin(X[:, 0] / 20) + rng.normal(size=n) * 0.3
    kw = dict(variogram_model="exponential", variogram_parameters=[1.5, 40.0, 0.1])
    cls = "OrdinaryKriging" + ("3D" if dim == 3 else "")
    if kind == "geo":
        kw["coordinates_type"] = "geographic"
    if kind in ("pinv", "dups"):
        X = np.vstack([X, X[:3]])
        v = np.concatenate([v, v[:3] + (0.0 if rng.uniform() < 0.5 else 0.1)])
        n += 3
    if kind == "pinv":
        kw.update(pseudo_inv=True, pseudo_inv_type=("pinv", "pinvh")[(t // 4) % 2])
    if kind == "custom":
        f, p = _KIND_CUSTOMS[rng.integers(2)]
        kw = dict(variogram_model="custom", variogram_function=f, variogram_parameters=list(p))
        if rng.uniform() < 0.5 and dim == 2:
            kw.update(anisotropy_scaling=2.0, anisotropy_angle=30.0)
        if rng.uniform() < 0.4:
            cls = "UniversalKriging" + ("3D" if dim == 3 else "")
            kw["drift_terms"] = ["regional_linear"]
    ekw = {}
    style = ("grid", "points", "masked")[rng.integers(3)]
    lo, hi = X.min(0), X.max(0)
    nx, ny, nz = int(rng.integers(1, 6)), int(rng.integers(1, 6)), int(rng.integers(1, 4))
    gx = np.sort(rng.uniform(lo[0] - 5, hi[0] + 5, nx))
    gy = np.sort(rng.uniform(-85, 85, ny) if kind == "geo" else rng.uniform(lo[1] - 5, hi[1] + 5, ny))
    gz = np.sort(rng.uniform(0, 100, nz))
    if style == "points":
        m = int(rng.integers(1, 9))
        gx, gy, gz = rng.uniform(lo[0], hi[0], m), rng.uniform(lo[1], hi[1], m), rng.uniform(0, 100, m)
        nx = ny = nz = m
    shape = (ny, nx) if dim == 2 else (nz, ny, nx)
    if style == "masked":
        ekw["mask"] = rng.uniform(size=shape) < 0.4
    knn = None
    if cls.startswith("Ordinary") and rng.uniform() < 0.35 and kind != "dups":
        knn = int(rng.integers(2, 8))
        ekw["n_closest_points"] = knn
    data = (X[:, 0], X[:, 1], v) if dim == 2 else (X[:, 0], X[:, 1], X[:, 2], v)
    pts = (gx, gy) if dim == 2 else (gx, gy, gz)
    return dict(t=t, kind=kind, cls=cls, data=data, kw=kw, style=style, pts=pts, ekw=ekw, knn=knn,
                text="%s %s n=%d %s %s knn=%s" % (kind, cls, n, style, shape, knn))
