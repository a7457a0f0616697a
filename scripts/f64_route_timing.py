"""dtype='float64': the INT8 8-slice contraction (solve_kernel_i8<8, .>) against the fp64 DMMA kernel (solve_kernel_pt).

Both routes run in one process, alternating, --reps repetitions each, selected per problem with KB200_F64_SOLVE=int8 |
dmma (read when the problem is described). Prints one JSON line per measurement:

  gpu      name, power limit and SM clocks (nvidia-smi, same process)
  cfg2     OK 2-D N=5000, 1000x1000 grid: solve-kernel points/s, whole-step ms (factor + grid execute), agreement,
           the route the default (no override) takes, and the int8 accounting: MMAs x MACs over the solve time,
           against the kind::i8 rate measured in profiles/README.md (~3700 MAC/clk/SM)
  sweep    n in {256, 512, 1024, 2048, 5000} at 2^18 and 10^6 random points: solve ms of both routes (places N_MIN)
  cfg3     OK3D N=8000, 200x200x50 grid, gaussian

    python scripts/f64_route_timing.py [--reps 3] [--skip-cfg3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cases  # noqa: E402
import pykrige_b200 as pk  # noqa: E402

ROUTES = ("int8", "dmma")
S, BN, BK, TM = 8, 64, 32, 128
MAC_PER_CLK_SM_I8 = 3700.0      # measured kind::i8 rate (profiles/README.md, int8-slice section)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks_throttle_reasons.active"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        return {"error": str(e)}
    return {"query": q, "gpus": out}


def sm_clock_mhz():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except (OSError, subprocess.SubprocessError, ValueError, IndexError):
        return float("nan")


def i8_macs(n, na, m):
    """MACs the S=8 kernel issues for m points: per 128-point tile, 36 MMAs of 128 x 64 x 32 per (row block, k-stage)."""
    nk = (n + BK - 1) // BK
    nrb = (n + na + BN - 1) // BN
    stages = sum(nk if (j + 1) * BN > n else min(nk, ((j + 1) * BN + BK - 1) // BK) for j in range(nrb))
    return ((m + TM - 1) // TM) * stages * (S * (S + 1) // 2) * TM * BN * BK


def run(model, route, style, args):
    """Factor + execute on one route; returns (z, ss, step_ms, solve_ms, slices)."""
    os.environ["KB200_F64_SOLVE"] = route
    model._kb_key = None
    h = model._cuda_handle()
    h.reset_counters()
    t0 = time.perf_counter()
    z, ss = model.execute(style, *args, backend="cuda", dtype="float64")
    step_ms = (time.perf_counter() - t0) * 1e3
    tm = model._kb_handle.timings()
    return np.asarray(z).ravel(), np.asarray(ss).ravel(), step_ms, tm["solve_ms"], int(tm["solve_slices"])


def default_slices(model, style, args):
    os.environ.pop("KB200_F64_SOLVE", None)
    model._kb_key = None
    model.execute(style, *[a[:64] if style == "points" else a for a in args], backend="cuda", dtype="float64")
    return int(model._kb_handle.timings()["solve_slices"])


def compare(model, style, args, m, reps, tag, extra=None):
    res = {r: [] for r in ROUTES}
    out = {}
    run(model, "int8", style, args); run(model, "dmma", style, args)          # warm both routes
    for _ in range(reps):
        for r in ROUTES:
            z, ss, step, solve, sl = run(model, r, style, args)
            res[r].append((step, solve, sl))
            out[r] = (z, ss)
    clk = sm_clock_mhz()
    line = {"what": tag, "points": m, "reps": reps, "default_slices": default_slices(model, style, args)}
    for r in ROUTES:
        steps = [s for s, _, _ in res[r]]
        solves = [s for _, s, _ in res[r]]
        line[r] = {"slices": res[r][0][2], "step_ms": steps, "solve_ms": solves,
                   "solve_points_per_s_median": m / (float(np.median(solves)) * 1e-3)}
    line["solve_speedup_median"] = float(np.median([s for _, s, _ in res["dmma"]]) /
                                         np.median([s for _, s, _ in res["int8"]]))
    (z8, s8), (zd, sd) = out["int8"], out["dmma"]
    line["max_rel_z"] = float(np.abs(z8 - zd).max() / np.abs(zd).max())
    line["max_rel_ss"] = float(np.abs(s8 - sd).max() / np.abs(sd).max())
    if extra:
        line.update(extra(res, clk))
    print(json.dumps(line), flush=True)
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--skip-cfg3", action="store_true")
    a = ap.parse_args()
    print(json.dumps({"what": "gpu", **gpu_info()}), flush=True)

    # ---- config 2 ----
    xyz, val = cases.synth_data(1002, 5000, 2)
    model = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential",
                               variogram_parameters=[1.0, 300.0, 0.05])
    axes = (np.linspace(0.0, 1000.0, 1000), np.linspace(0.0, 1000.0, 1000))
    m = 1000 * 1000

    def i8_accounting(res, clk):
        macs = i8_macs(5000, 2, m)
        s = float(np.median([x for _, x, _ in res["int8"]])) * 1e-3
        rate = macs / s / (clk * 1e6) / 148.0
        return {"int8_accounting": {"macs": macs, "sm_clock_mhz": clk, "mac_per_clk_per_sm": rate,
                                    "frac_of_measured_i8_rate": rate / MAC_PER_CLK_SM_I8}}

    compare(model, "grid", axes, m, a.reps, "cfg2", i8_accounting)

    # ---- n sweep ----
    rng = np.random.default_rng(7)
    for n in (256, 512, 1024, 2048, 5000):
        xyz, val = cases.synth_data(2000 + n, n, 2)
        model = pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, variogram_model="exponential",
                                   variogram_parameters=[1.0, 300.0, 0.05])
        for mp in (1 << 18, 1000000):
            px, py = rng.uniform(0.0, 1000.0, mp), rng.uniform(0.0, 1000.0, mp)
            compare(model, "points", (px, py), mp, a.reps, "sweep n=%d" % n)

    # ---- config 3 ----
    if not a.skip_cfg3:
        xyz, val = cases.synth_data(1003, 8000, 3)
        model = pk.OrdinaryKriging3D(xyz[:, 0], xyz[:, 1], xyz[:, 2], val, variogram_model="gaussian",
                                     variogram_parameters=[1.0, 300.0, 0.05])
        axes = (np.linspace(0, 1000, 200), np.linspace(0, 1000, 200), np.linspace(0, 250, 50))
        compare(model, "grid", axes, 200 * 200 * 50, a.reps, "cfg3")
    print(json.dumps({"what": "gpu_after", **gpu_info()}), flush=True)


if __name__ == "__main__":
    main()
