"""dtype='float64' on the INT8 tensor cores (csrc/solve_i8.cu with S = 8 slices, routed in csrc/api.cu: describe()).

On the Cholesky path with KB_F64_I8_NMIN <= n <= KB_F64_I8_NMAX the fp64 contraction q = ||W c||^2 runs as 8 exact
signed 7-bit slices of W and c (55 bits), exact int32 accumulation per slice-pair diagonal d = s + t < 8, and an exact
two-half recombination V = H * 2^28 + L converted to fp64 once. The host tests check that arithmetic in numpy; the GPU
tests check the route choice and that both routes compute the same numbers.
"""
import os
import re

import numpy as np
import pytest
import scipy.linalg

import cases
from conftest import ROOT, assert_parity
from oracle import krige_oracle as ko
from test_device_algebra_model import i8_slices

S = 8
N_MAX = 65535                       # int32 accumulators: n * 8 * 64^2 < 2^31


def _api_define(name):
    src = open(os.path.join(ROOT, "pykrige_b200", "csrc", "api.cu")).read()
    return int(re.search(r"#define %s (\d+)" % name, src).group(1))


def s8_recombine(acc):
    """The kernel's epilogue on the 8 diagonal sums acc[d] (int64 arrays): H = sum_{d<4} acc_d 2^(7 (3-d)),
    L = sum_{d>=4} acc_d 2^(7 (7-d)) in int64, then (double)H * 2^28 + (double)L."""
    H = np.zeros_like(acc[0])
    L = np.zeros_like(acc[0])
    for d in range(4):
        H = H * 128 + acc[d]
    for d in range(4, 8):
        L = L * 128 + acc[d]
    return H.astype(np.float64) * 2.0 ** 28 + L.astype(np.float64), H, L


def s8_matvec_rows(W, c):
    """(W c)_r through the S = 8 slice scheme, with the kernel's per-row / per-column exponents."""
    ew = np.floor(np.log2(np.max(np.abs(W), axis=1))).astype(int) + 1
    ec = int(np.floor(np.log2(np.max(np.abs(c))))) + 1
    ws = np.stack([i8_slices(W[r], int(ew[r]), S) for r in range(W.shape[0])], axis=1)     # [S, rows, n]
    cs = i8_slices(c, ec, S)
    assert np.abs(ws).max() <= 64 and np.abs(cs).max() <= 64
    acc = []
    for d in range(S):
        a = sum(ws[s] @ cs[d - s] for s in range(d + 1))
        assert np.abs(a).max() < 2 ** 31, "int32 TMEM accumulator would overflow"
        acc.append(a)
    v, _, _ = s8_recombine(acc)
    return np.ldexp(v, ew + ec - 12 - 7 * (S - 1))


@pytest.mark.parametrize("n", [600, 2000])
def test_s8_slice_model_is_as_accurate_as_fp64(n):
    """q = ||W c||^2 of an exponential kriging problem, W = chol(C)^-1: the S = 8 scheme stays within 4x of the plain
    fp64 product's error against an 80-bit long double reference (S = 7 would be ~100x worse)."""
    xyz, val = cases.synth_data(5, n, 2)
    m = ko.stored_parameters("exponential", [1.0, 300.0, 0.05])
    gam = ko.variogram("exponential", m, ko.cdist(xyz, xyz))
    np.fill_diagonal(gam, 0.0)
    c0 = m[0] + m[2]
    W = scipy.linalg.solve_triangular(np.linalg.cholesky(c0 - gam), np.eye(n), lower=True)
    Wl = W.astype(np.longdouble)
    err64 = err8 = 0.0
    for q in cases.synth_points(5, 6, 2, xyz, n_hits=1):
        c = c0 - ko.variogram("exponential", m, np.sqrt(np.sum((xyz - q) ** 2, axis=1)))
        ref = np.sum((Wl @ c.astype(np.longdouble)) ** 2)
        err64 = max(err64, float(abs(np.sum((W @ c) ** 2) - ref) / ref))
        err8 = max(err8, float(abs(np.sum(s8_matvec_rows(W, c) ** 2) - ref) / ref))
    assert err8 <= 4.0 * max(err64, 2.0 ** -53), (err8, err64)


def test_s8_recombination_is_exact_at_the_worst_case_bound():
    """|acc_d| <= n (d+1) 64^2 for n <= 65535: one int64 V = sum_d acc_d 2^(7 (7-d)) can overflow, the two halves cannot,
    both are exact in fp64, and the final sum rounds the exact V once (== float(V) of the Python integer)."""
    n = N_MAX
    bound = [n * (d + 1) * 64 * 64 for d in range(S)]
    assert sum(b * 2 ** (7 * (7 - d)) for d, b in enumerate(bound)) >= 2 ** 63         # a single int64 would overflow
    rng = np.random.default_rng(8)
    rows = [np.array(bound), -np.array(bound), np.array([(-1) ** d * b for d, b in enumerate(bound)])]
    rows += [np.array([int(rng.integers(-b, b + 1)) for b in bound]) for _ in range(2000)]
    rows += [np.array([int(rng.integers(-b, b + 1)) if d >= 4 else 0 for d, b in enumerate(bound)]) for _ in range(100)]
    A = np.stack(rows).astype(np.int64)                                                # [cases, 8]
    v, H, L = s8_recombine([A[:, d] for d in range(S)])
    for i in range(A.shape[0]):
        Hx = sum(int(A[i, d]) * 2 ** (7 * (3 - d)) for d in range(4))
        Lx = sum(int(A[i, d]) * 2 ** (7 * (7 - d)) for d in range(4, 8))
        assert int(H[i]) == Hx and int(L[i]) == Lx
        assert abs(Hx) < 2 ** 53 and abs(Lx) < 2 ** 53                                  # exact in fp64
        assert v[i] == float(Hx * 2 ** 28 + Lx)                                         # one correct rounding


def test_s8_int32_accumulators_cannot_overflow():
    """Worst case of the largest diagonal sum (d = 7: 8 slice pairs of |64 * 64| per k) stays below 2^31 for every n the
    route accepts, and the route's limit in api.cu is that bound."""
    assert _api_define("KB_F64_I8_NMAX") == N_MAX
    assert _api_define("KB_F64_I8_SLICES") == S
    assert N_MAX * S * 64 * 64 < 2 ** 31 <= (N_MAX + 1) * S * 64 * 64
    assert 1 <= _api_define("KB_F64_I8_NMIN") <= N_MAX
    # balanced digits: slice 0 in [-64, 64], the others in [-64, 63]
    x = np.array([1 - 2.0 ** -60, -(1 - 2.0 ** -60), 0.5, -0.5, 2.0 ** -50])
    sl = i8_slices(x, 0, S)
    assert np.abs(sl).max() <= 64 and sl[1:].max() <= 63


# ---------------------------------------------------------------------------------------------------------------- GPU
N_TEST = 2048           # >= KB_F64_I8_NMIN: problems on the int8 route


@pytest.fixture(scope="module")
def pk():
    import pykrige_b200
    return pykrige_b200


def _slices(model):
    return int(model._kb_handle.timings()["solve_slices"])


def _both_routes(model, monkeypatch, style, *args):
    out = {}
    for route in ("default", "dmma"):
        if route == "dmma":
            monkeypatch.setenv("KB200_F64_SOLVE", "dmma")
        else:
            monkeypatch.delenv("KB200_F64_SOLVE", raising=False)
        model._kb_key = None
        z, ss = model.execute(style, *args, backend="cuda")
        out[route] = (np.asarray(z).ravel(), np.asarray(ss).ravel(), _slices(model))
    monkeypatch.delenv("KB200_F64_SOLVE", raising=False)
    return out


def _assert_routes_agree(out, what, hits=0):
    """z and sigma^2 of both routes agree to 1e-12 of their maximum; sigma^2 at the trailing `hits` exact hits <= 1e-9."""
    (z8, s8, k8), (zd, sd, kd) = out["default"], out["dmma"]
    assert (k8, kd) == (S, 0), (what, k8, kd)
    assert np.abs(z8 - zd).max() <= 1e-12 * np.abs(zd).max(), (what, np.abs(z8 - zd).max())
    assert np.abs(s8 - sd).max() <= 1e-12 * np.abs(sd).max(), (what, np.abs(s8 - sd).max())
    if hits:
        assert np.abs(s8[-hits:]).max() <= 1e-9 and np.abs(sd[-hits:]).max() <= 1e-9, what


@pytest.mark.gpu
def test_route_choice(pk, monkeypatch):
    """Config-2 data (N=5000) takes the int8 route, a config-1-sized problem (N=100) and KB200_F64_SOLVE=dmma the DMMA
    kernel; the non-default dtypes keep their own kernels."""
    monkeypatch.delenv("KB200_F64_SOLVE", raising=False)
    xyz, val = cases.synth_data(1002, 5000, 2)
    ok = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential", variogram_parameters=[1.0, 300.0, 0.05])
    ok.execute("points", [1.0, 2.0], [3.0, 4.0], backend="cuda")
    assert _slices(ok) == S
    for dt, k in (("float64x", 6), ("float64x4", 4), ("float32", 0)):
        ok.execute("points", [1.0], [3.0], backend="cuda", dtype=dt)
        assert _slices(ok) == k, dt
    small = pk.OrdinaryKriging(xyz[:100, 0], xyz[:100, 1], val[:100], variogram_model="spherical",
                               variogram_parameters=[1.0, 400.0, 0.05])
    small.execute("points", [1.0], [3.0], backend="cuda")
    assert _slices(small) == 0
    monkeypatch.setenv("KB200_F64_SOLVE", "dmma")
    ok._kb_key = None
    ok.execute("points", [1.0], [3.0], backend="cuda")
    assert _slices(ok) == 0


@pytest.mark.gpu
def test_int8_route_matches_dmma_cfg2(pk, monkeypatch):
    """Config 2 (N=5000, exponential): a slab of the 1000x1000 grid plus 16 exact hits, int8 route vs DMMA kernel."""
    xyz, val = cases.synth_data(1002, 5000, 2)
    ok = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential", variogram_parameters=[1.0, 300.0, 0.05])
    gx = np.linspace(0.0, 1000.0, 1000)
    gy = np.linspace(0.0, 1000.0, 1000)[:8]
    _assert_routes_agree(_both_routes(ok, monkeypatch, "grid", gx, gy), "cfg2 grid slab")
    G = ko.grid_points([gx, gy])
    pts = np.vstack([G, xyz[:16]])
    _assert_routes_agree(_both_routes(ok, monkeypatch, "points", pts[:, 0], pts[:, 1]), "cfg2 slab + hits", hits=16)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["ok3d", "uk_drift", "geographic", "custom_table"])
def test_int8_route_matches_dmma_other_problems(pk, monkeypatch, kind):
    n = N_TEST
    if kind == "ok3d":
        xyz, val = cases.synth_data(31, n, 3)
        m = pk.OrdinaryKriging3D(xyz[:, 0], xyz[:, 1], xyz[:, 2], val, variogram_model="gaussian",
                                 variogram_parameters=[1.0, 300.0, 0.05])
        pts = cases.synth_points(31, 3000, 3, xyz)
        out = _both_routes(m, monkeypatch, "points", pts[:, 0], pts[:, 1], pts[:, 2])
    else:
        if kind == "geographic":
            rng = np.random.default_rng(32)
            xyz = np.column_stack([rng.uniform(-20.0, 40.0, n), rng.uniform(30.0, 75.0, n)])
            val = 10.0 + np.sin(np.radians(xyz[:, 0]) * 3.0) + rng.normal(0.0, 0.1, n)
            m = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential",
                                   variogram_parameters=[1.0, 20.0, 0.05], coordinates_type="geographic")
            pts = np.vstack([np.column_stack([rng.uniform(-20.0, 40.0, 3000), rng.uniform(30.0, 75.0, 3000)]), xyz[:16]])
        else:
            xyz, val = cases.synth_data(33, n, 2)
            if kind == "uk_drift":
                m = pk.UniversalKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential",
                                        variogram_parameters=[1.0, 300.0, 0.05], drift_terms=["regional_linear"])
            else:
                fn = lambda p, d: p[0] * (1.0 - np.exp(-d / (p[1] / 3.0))) + p[2]      # noqa: E731
                m = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="custom",
                                       variogram_parameters=[1.0, 300.0, 0.05], variogram_function=fn)
            pts = cases.synth_points(33, 3000, 2, xyz)
        out = _both_routes(m, monkeypatch, "points", pts[:, 0], pts[:, 1])
    _assert_routes_agree(out, kind, hits=16)


@pytest.mark.gpu
def test_indefinite_problem_falls_back_to_dmma(pk, monkeypatch):
    """hole-effect at N >= KB_F64_I8_NMIN: the Cholesky fails, the general path packs fp64 tiles and runs the DMMA
    kernel (solve_slices 0), matching the oracle."""
    monkeypatch.delenv("KB200_F64_SOLVE", raising=False)
    xyz, val = cases.synth_data(34, N_TEST, 2)
    params = [1.0, 250.0, 0.02]
    ok = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="hole-effect", variogram_parameters=params)
    pts = cases.synth_points(34, 300, 2, xyz)
    z, ss = ok.execute("points", pts[:, 0], pts[:, 1], backend="cuda")
    assert _slices(ok) == 0
    zo, so = ko.krige(xyz, val, "hole-effect", ko.stored_parameters("hole-effect", params), pts)
    assert_parity(z, zo, 1e-5, "hole-effect z")
    assert_parity(ss, so, 1e-5, "hole-effect ss")


def _second_handle(pk, make, style, args, monkeypatch, describe_env=None):
    """Factor on one handle; describe the same problem on a second handle of the same device, copy the blob over,
    commit it, and execute there (the non-root rank's path)."""
    import torch
    from pykrige_b200 import multigpu
    a = make()
    z1, s1 = a.execute(style, *args, backend="cuda")
    k1 = _slices(a)
    b = make()
    if describe_env:
        monkeypatch.setenv("KB200_F64_SOLVE", describe_env)
    hb = multigpu._describe_only(b, "float64")
    monkeypatch.delenv("KB200_F64_SOLVE", raising=False)
    dev = torch.device("cuda", torch.cuda.current_device())
    ta, tb = multigpu.blob_as_tensor(a._kb_handle, dev), multigpu.blob_as_tensor(hb, dev)
    assert ta.numel() == tb.numel()
    tb.copy_(ta)
    torch.cuda.synchronize()
    hb.blob_commit()
    b._kb_key = b._problem_signature(multigpu._dtype_code("float64"), False)
    z2, s2 = b.execute(style, *args, backend="cuda")
    assert b._kb_handle is hb and _slices(b) == k1
    assert np.array_equal(np.asarray(z1), np.asarray(z2)) and np.array_equal(np.asarray(s1), np.asarray(s2))
    return k1


@pytest.mark.gpu
def test_second_handle_reproduces_the_factoring_handle(pk, monkeypatch):
    """The route travels in the blob header: a describe-only handle (even one described under KB200_F64_SOLVE=dmma)
    runs the kernel the factoring handle packed for, bit for bit; once on the int8 route, once on the fallback."""
    monkeypatch.delenv("KB200_F64_SOLVE", raising=False)
    xyz, val = cases.synth_data(1002, 5000, 2)
    gx, gy = np.linspace(0.0, 1000.0, 1000), np.linspace(0.0, 1000.0, 1000)[:4]
    k = _second_handle(pk, lambda: pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential",
                                                      variogram_parameters=[1.0, 300.0, 0.05]),
                       "grid", (gx, gy), monkeypatch, describe_env="dmma")
    assert k == S
    xh, vh = cases.synth_data(34, N_TEST, 2)
    pts = cases.synth_points(34, 500, 2, xh)
    k = _second_handle(pk, lambda: pk.OrdinaryKriging(xh[:, 0], xh[:, 1], vh, variogram_model="hole-effect",
                                                      variogram_parameters=[1.0, 250.0, 0.02]),
                       "points", (pts[:, 0], pts[:, 1]), monkeypatch)
    assert k == 0
