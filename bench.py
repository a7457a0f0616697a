#!/usr/bin/env python
"""bench.py — kriged grid points / second of the B200 backend='cuda' execute() path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--configs cfg1,cfg3,...|none]
                    [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1], SURVEY.md §8d cfg2): OrdinaryKriging 2-D, N=5000 random-scatter
data (seed 1002), 1000x1000 grid, exponential variogram [1.0, 300, 0.05], fp64 (DMMA kernel).
One step = one full execute(): assemble + factor + krige every grid point (the reference re-assembles
and re-inverts on every call, ok.py:847,663 — so does every timed step here; nothing is cached).

  value : whole-step throughput with the point generation on device and outputs left in HBM
          (kb200_set_problem + kb200_execute_grid_dev); timed with CUDA events on the launching stream.
  e2e   : the same step through the public class API (OrdinaryKriging.execute('grid', ..., backend='cuda'))
          with host buffers: H2D of data/axes and D2H of (z, sigma^2) inside the region.
  roofline : the fused solve kernel against the MEASURED fp64 GEMM rate of this GPU (torch.matmul 8192^3 taken
          in this run; MEASURED_PEAKS.json holds no fp64 entry). `frac` uses the algorithmic 2*(N+1)^2 flop per
          grid point of SURVEY.md §8(d) (the reference's inverse GEMV); `frac_executed` uses the flops the
          covariance-form triangular kernel actually issues (~ n^2 (1 + 256/n) per point).
  cpu_baseline : the oracle port of the reference's inverse x RHS path (oracle/krige_oracle.py) on the box's
          host cores (BLAS threads pinned to the core count), on a bounded sample of the same grid.

--dump-outputs DIR writes what the last timed headline step computed, the whole 1000x1000 grid of kriged values
and kriging variances, to DIR/zvalues.npy and DIR/sigmasq.npy (float64, shape (ny, nx) as execute('grid') returns
them; 16 MB in all). The inputs are seeded, so two builds run with the same arguments can be compared output for
output.

N>1 (torchrun, one rank per GPU): rank 0 factors, one NCCL broadcast ships the factor blob, every rank kriges a
contiguous slice of the SAME 1000x1000 grid (strong scaling: the headline `value`); the weak-scaling variant
(1000 x 1000*N points) is reported under config.weak.

config.configs holds the other BASELINE configs — cfg1 (N=100, 50x50, spherical), cfg3 (OK3D N=8000, 200x200x50,
gaussian, fp64), cfg4 (UK regional-linear N=10000, 2000x2000, fp32 device math), cfg5 (moving window k=64,
N=100000, 4000x4000) — each run on the N GPUs of this launch (their named GPU counts are 1 / 8 / 4 / 8), timed the
same way, with 4096+16-point parity against the CPU oracle checked in the run. A failed check of the HEADLINE aborts the
bench (no number without parity); a side config that fails its check, or raises, stays in the line flagged
`"invalid"` / `"error"` instead of taking the measured headline down with it.
"""
import os
import sys

# BLAS threads of the CPU legs: torchrun exports OMP_NUM_THREADS=1 to its children, which would throttle the
# oracle (and inflate every GPU/CPU ratio); pin them to the core count before numpy loads OpenBLAS.
_RANK0 = int(os.environ.get("RANK", "0")) == 0
for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ[_v] = str(os.cpu_count() or 1) if _RANK0 else "1"

import argparse  # noqa: E402
import json  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "kriged grid points/sec (N data -> M grid)"
UNIT = "points/s"
R64, R32 = 1e-5, 1e-2          # parity tolerances of BASELINE.json north_star (fp64 / fp32 device math)

CONFIGS = {
    "cfg1": dict(cls="OK", dim=2, n=100, seed=1001, grid=(50, 50), box=(1000.0, 1000.0), model="spherical",
                 params=[1.0, 400.0, 0.05], dtype="float64", named_gpus=1,
                 text="OrdinaryKriging 2D, N=100 data, 50x50 grid, spherical variogram (BASELINE configs[0])"),
    "cfg2": dict(cls="OK", dim=2, n=5000, seed=1002, grid=(1000, 1000), box=(1000.0, 1000.0), model="exponential",
                 params=[1.0, 300.0, 0.05], dtype="float64", named_gpus=1,
                 text="OrdinaryKriging 2D, N=5000 data, 1000x1000 grid, exponential variogram, fp64 (BASELINE configs[1])"),
    "cfg3": dict(cls="OK3D", dim=3, n=8000, seed=1003, grid=(200, 200, 50), box=(1000.0, 1000.0, 250.0),
                 model="gaussian", params=[1.0, 300.0, 0.05], dtype="float64", named_gpus=8,
                 text="OrdinaryKriging3D, N=8000 data, 200x200x50 grid, gaussian variogram, fp64 (BASELINE configs[2])"),
    "cfg4": dict(cls="UK", dim=2, n=10000, seed=1004, grid=(2000, 2000), box=(1000.0, 1000.0), model="exponential",
                 params=[1.0, 300.0, 0.05], dtype="float32", named_gpus=4,
                 text="UniversalKriging 2D regional-linear drift, N=10000 data, 2000x2000 grid, fp32 device math "
                      "(tcgen05 3xTF32) (BASELINE configs[3])"),
    "cfg5": dict(cls="OK", dim=2, n=100000, seed=1005, grid=(4000, 4000), box=(1000.0, 1000.0), model="exponential",
                 params=[1.0, 50.0, 0.05], dtype="float64", k=64, named_gpus=8,
                 text="OrdinaryKriging 2D moving window n_closest_points=64, N=100000 data, 4000x4000 grid "
                      "(BASELINE configs[4])"),
}


def cfg_data(cfg):
    import cases
    return cases.synth_data(cfg["seed"], cfg["n"], cfg["dim"])


def cfg_axes(cfg, scale_last=1):
    ax = [np.linspace(0.0, cfg["box"][c], cfg["grid"][c]) for c in range(cfg["dim"])]
    if scale_last > 1:      # weak scaling: the slowest axis grows with the GPU count
        c = cfg["dim"] - 1
        ax[c] = np.linspace(0.0, cfg["box"][c] * scale_last, cfg["grid"][c] * scale_last)
    return ax


def make_model(cfg, xyz, val):
    import pykrige_b200 as pk
    kw = dict(variogram_model=cfg["model"], variogram_parameters=cfg["params"])
    if cfg["cls"] == "OK":
        return pk.OrdinaryKriging(xyz[:, 0], xyz[:, 1], val, **kw)
    if cfg["cls"] == "UK":
        return pk.UniversalKriging(xyz[:, 0], xyz[:, 1], val, drift_terms=["regional_linear"], **kw)
    return pk.OrdinaryKriging3D(xyz[:, 0], xyz[:, 1], xyz[:, 2], val, **kw)


def flop_per_point(cfg):
    """Algorithmic work per prediction point, SURVEY.md §8(d)."""
    if cfg.get("k"):
        k1 = cfg["k"] + 1
        return (2.0 / 3.0) * k1**3 + 2.0 * k1**2
    K = {"OK": 0, "OK3D": 0, "UK": 2}[cfg["cls"]]
    return 2.0 * (cfg["n"] + K + 1) ** 2


def executed_flop_per_point(cfg):
    """What the covariance-form kernels issue: the lower-triangular product in 256-row blocks (rows of a block run
    to the block's diagonal end) plus the K+2 dense dual rows: ~ n^2 (1 + 256/n) + 2 (K+2) n."""
    if cfg.get("k"):
        k = cfg["k"]
        return k**3 / 3.0 + 4.0 * k**2          # Cholesky + two right-hand sides, forward + back
    n = cfg["n"]
    K = {"OK": 0, "OK3D": 0, "UK": 2}[cfg["cls"]]
    return float(n) * n * (1.0 + 256.0 / n) + 2.0 * (K + 2) * n


# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi style clock / throttle-reason samples during the timed region (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons, self.stop_flag = [], set(), False
        self.max_mhz = None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            }
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.1)
        except Exception as e:  # noqa: BLE001
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "samples": len(s), "reasons": sorted(self.reasons)}


def measure_gemm_peak(torch, dtype, tf32=False):
    n = 8192
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = bool(tf32)
    try:
        a = torch.randn(n, n, device="cuda", dtype=dtype)
        b = torch.randn(n, n, device="cuda", dtype=dtype)
        a @ b
        torch.cuda.synchronize()
        best = 1e30
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a @ b
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        del a, b
        torch.cuda.empty_cache()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    return 2.0 * n**3 / (best * 1e-3) / 1e12


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([d.get("num_threads", 1) for d in threadpool_info()] or [1])
    except Exception:  # noqa: BLE001
        return None


# ---------------------------------------------------------------------------------------------
def cpu_arm(steps, warmup):
    """The reference's own CPU arithmetic for the headline path on the host cores: the oracle port of
    backend='vectorized' (_get_kriging_matrix + scipy.linalg.inv once, then inverse x RHS per slab,
    ok.py:626-683; oracle.PreparedKriging / krige_chunked) with the BLAS threads pinned to the core count, and,
    when oracle/_ref is built, the reference's compiled backend='C' twin (cok.pyx:_c_exec_loop).
    One step = a 10000-point slab (10 rows) of the same 1000x1000 grid; the set-up is timed separately
    (SURVEY.md §8d) — at 1e6 points it is < 2 % of the reference's job."""
    from oracle import krige_oracle as ko
    from threadpoolctl import threadpool_limits
    cfg = CONFIGS["cfg2"]
    xyz, val = cfg_data(cfg)
    gx, gy = cfg_axes(cfg)
    stored = ko.stored_parameters(cfg["model"], cfg["params"])
    cores = os.cpu_count() or 1
    slab = 10 * gx.size
    with threadpool_limits(limits=cores):
        t0 = time.perf_counter()
        prep = ko.PreparedKriging(xyz, val, cfg["model"], stored)
        setup_s = time.perf_counter() - t0

        def step(i):
            rows = np.arange(10) + 10 * (i % (gy.size // 10))
            return prep.krige(ko.grid_points([gx, gy[rows]]))

        for i in range(warmup):
            step(i)
        t0 = time.perf_counter()
        for i in range(max(1, steps)):
            step(warmup + i)
        dt = (time.perf_counter() - t0) / max(1, steps)
        threads = blas_threads()
    value = slab / dt
    kind = "port"
    sample = ("oracle.PreparedKriging (inverse x RHS, ok.py:665-681) on 10 grid rows (%d points) per step, "
              "%s BLAS threads; set-up (matrix + scipy.linalg.inv) %.2f s timed separately; whole 1e6-point job "
              "incl. set-up: %.0f points/s" % (slab, threads, setup_s, 1e6 / (setup_s + 1e6 * dt / slab)))
    other = None
    try:
        from oracle import ref_native as rn
        if rn.available():
            G = ko.grid_points([gx, gy[:1]])
            t1 = time.perf_counter(); rn.exec_loop(xyz, G[:100], val, cfg["model"], stored); t1 = time.perf_counter() - t1
            t2 = time.perf_counter(); rn.exec_loop(xyz, G[:600], val, cfg["model"], stored); t2 = time.perf_counter() - t2
            nat = 500.0 / max(1e-9, t2 - t1)
            other = {"value": nat, "unit": UNIT, "kind": "reference",
                     "sample": "oracle/_ref cok._c_exec_loop (the reference's backend='C'): 600 vs 100 grid points, "
                               "steady per-point rate (its internal matrix inverse excluded)"}
            if nat > value:          # report the FASTER CPU implementation of the path as the reference arm
                other, value, kind, sample = (
                    {"value": value, "unit": UNIT, "kind": "port", "sample": sample}, nat, "reference", other["sample"])
                dt = slab / value
    except Exception as e:  # noqa: BLE001
        other = {"unavailable": "%s: %s" % (type(e).__name__, e)}
    return {"value": value, "unit": UNIT, "cores": cores, "blas_threads": threads, "kind": kind, "sample": sample,
            "setup_s": setup_s, "other_cpu_implementation": other}, dt, slab


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cpu, dt, slab = cpu_arm(args.steps, args.warmup)
    cfg = CONFIGS["cfg2"]
    line = {
        "impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": cfg["text"], "n_data": cfg["n"], "grid": list(cfg["grid"]), "variogram": cfg["model"],
                   "variogram_parameters": cfg["params"], "seed": cfg["seed"],
                   "sample": "%d-point slabs of the grid per step" % slab},
        "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------
class Ctx:
    pass


def timed(ctx, fn, steps):
    torch, dist = ctx.torch, ctx.dist
    if ctx.world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ctx.stream)
    for _ in range(steps):
        fn()
    e1.record(ctx.stream)
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=ctx.dev)
    if ctx.world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)     # max over ranks
        dist.barrier()
    return float(ms.item()) / steps


def oracle_parity(ctx, cfg, model, xyz, val, axes, z_loc, ss_loc, first, count, n_sample=4096, n_hits=16, fatal=True):
    """4096 random cells of the kriged grid (taken from every rank's slice of the LAST timed e2e step) + the first
    16 data coordinates as 'points' queries (exact hits), against the CPU oracle on rank 0. SURVEY.md §8(d)."""
    from pykrige_b200 import multigpu  # noqa: F401
    from oracle import krige_oracle as ko
    from threadpoolctl import threadpool_limits
    npt = int(np.prod([a.size for a in axes]))
    rng = np.random.default_rng(7)
    pick = np.sort(rng.choice(npt, size=min(n_sample, npt), replace=False))
    mine = pick[(pick >= first) & (pick < first + count)]
    part = (mine, z_loc[mine - first], ss_loc[mine - first])
    parts = [part]
    if ctx.world > 1:
        parts = [None] * ctx.world
        ctx.dist.all_gather_object(parts, part)
    if ctx.rank != 0:
        return None
    idx = np.concatenate([p[0] for p in parts])
    zg = np.concatenate([p[1] for p in parts])
    sg = np.concatenate([p[2] for p in parts])
    order = np.argsort(idx)
    idx, zg, sg = idx[order], zg[order], sg[order]
    assert np.array_equal(idx, pick)
    sizes = [a.size for a in axes]
    cols = [axes[0][idx % sizes[0]], axes[1][(idx // sizes[0]) % sizes[1]]]
    if cfg["dim"] == 3:
        cols.append(axes[2][idx // (sizes[0] * sizes[1])])
    G = np.column_stack(cols)
    hits = xyz[:n_hits]
    k = cfg.get("k")
    kw = dict(n_closest_points=k) if k else {}
    if cfg["dim"] == 3:
        zh, sh = model.execute("points", hits[:, 0], hits[:, 1], hits[:, 2], backend="cuda", dtype=cfg["dtype"], **kw)
    elif cfg["cls"] == "UK":
        zh, sh = model.execute("points", hits[:, 0], hits[:, 1], backend="cuda", dtype=cfg["dtype"])
    else:
        zh, sh = model.execute("points", hits[:, 0], hits[:, 1], backend="cuda", dtype=cfg["dtype"], **kw)
    Q = np.vstack([G, hits])
    stored = ko.stored_parameters(cfg["model"], cfg["params"])
    t0 = time.perf_counter()
    with threadpool_limits(limits=os.cpu_count() or 1):
        if k:
            zo, so = ko.krige(xyz, val, cfg["model"], stored, Q, n_closest_points=k)
        else:
            zo, so = ko.krige_chunked(xyz, val, cfg["model"], stored, Q, regional_linear=(cfg["cls"] == "UK"))
    t_oracle = time.perf_counter() - t0
    z = np.concatenate([zg, zh])
    ss = np.concatenate([sg, sh])
    R = R32 if cfg["dtype"] == "float32" else R64
    ok = bool(np.allclose(z, zo, rtol=R, atol=R * np.abs(zo).max()) and np.allclose(ss, so, rtol=R, atol=R * np.abs(so).max()))
    out = {"points_checked": int(Q.shape[0]), "rtol": R,
           "max_rel_z": float(np.max(np.abs(z - zo)) / np.max(np.abs(zo))),
           "max_rel_ss": float(np.max(np.abs(ss - so)) / np.max(np.abs(so))),
           "max_abs_ss_at_exact_hits": float(np.max(np.abs(sh))), "pass": ok, "oracle_s": t_oracle,
           "against": "oracle/krige_oracle.py (reference formulation: inverse x RHS%s)" % (" per point, k+1 system" if k else "")}
    if not ok and fatal:
        raise SystemExit("bench.py: parity against the oracle FAILED for %s: %s" % (cfg["text"], json.dumps(out)))
    return out


def gather_grid(ctx, d_out, count, sizes):
    """(z, sigma^2) of every rank's slice of the grid, as host arrays of the grid's shape (slowest axis first) on
    rank 0; (None, None) on the other ranks."""
    part = d_out[:2 * count].view(2, count).cpu().numpy()
    parts = [part]
    if ctx.world > 1:
        parts = [None] * ctx.world
        ctx.dist.all_gather_object(parts, part)
    if ctx.rank != 0:
        return None, None
    zs = np.concatenate(parts, axis=1)
    return zs[0].reshape(sizes[::-1]), zs[1].reshape(sizes[::-1])


def bench_config(ctx, name, steps, warmup, e2e_steps, weak=False, dtype=None, parity=True, fatal_parity=False,
                 outputs=None):
    """Time one BASELINE config on the ranks of this launch. Device-resident step (factor + krige this rank's
    contiguous slice, outputs left in HBM) and end-to-end step (public API, host buffers). Max over ranks.
    `outputs` (a dict) receives the grid the last timed device-resident step computed (gather_grid)."""
    import pykrige_b200 as pk  # noqa: F401
    from pykrige_b200 import multigpu
    torch, dist = ctx.torch, ctx.dist
    cfg = dict(CONFIGS[name])
    if dtype:
        cfg["dtype"] = dtype
    xyz, val = cfg_data(cfg)
    axes = cfg_axes(cfg, ctx.world if weak else 1)
    sizes = [a.size for a in axes]
    nx, ny = sizes[0], sizes[1]
    nz = sizes[2] if cfg["dim"] == 3 else 1
    npt = nx * ny * nz
    k = cfg.get("k")
    model = make_model(cfg, xyz, val)
    h = model._cuda_handle()
    h.set_stream(ctx.stream.cuda_stream)
    first, count = multigpu.shard_range(npt, ctx.rank, ctx.world)
    d_ax = [torch.from_numpy(a).to(ctx.dev) for a in axes]
    d_out = torch.empty(2 * max(count, 1), dtype=torch.float64, device=ctx.dev)
    ptr = [t.data_ptr() for t in d_ax] + ([0] if cfg["dim"] == 2 else [])

    def factor():
        model._kb_key = None            # full re-assembly + re-factorisation every step (nothing cached)
        if k:
            return model._ensure_problem("float64", knn=True)
        return multigpu.prepare_sharded(model, dist if ctx.world > 1 else None, dtype=cfg["dtype"])

    def step_dev():
        with torch.cuda.stream(ctx.stream):
            ctx.flush.zero_()
        factor()
        if k:
            h.execute_knn_grid_dev(k, nx, ny, nz, ptr[0], ptr[1], ptr[2], first, count,
                                   d_out.data_ptr(), d_out.data_ptr() + 8 * count)
        else:
            h.execute_grid_dev(nx, ny, nz, ptr[0], ptr[1], ptr[2], 0, first, count,
                               d_out.data_ptr(), d_out.data_ptr() + 8 * count)

    last = {}

    def step_e2e():
        with torch.cuda.stream(ctx.stream):
            ctx.flush.zero_()
        model._kb_key = None
        if ctx.world == 1:
            kw = dict(n_closest_points=k) if k else {}
            if cfg["cls"] == "UK":
                z, ss = model.execute("grid", *axes, backend="cuda", dtype=cfg["dtype"])
            else:
                z, ss = model.execute("grid", *axes, backend="cuda", dtype=cfg["dtype"], **kw)
            last["z"], last["ss"] = np.ravel(z), np.ravel(ss)
        else:
            z, ss, f, c = multigpu.execute_sharded(model, "grid", axes, dist, n_closest_points=k, dtype=cfg["dtype"])
            last["z"], last["ss"] = z, ss

    for _ in range(warmup):
        step_dev()
    h.reset_counters()
    ms_dev = timed(ctx, step_dev, steps)
    if outputs is not None:
        outputs["zvalues"], outputs["sigmasq"] = gather_grid(ctx, d_out, count, sizes)
    tm = h.timings()
    launches = torch.tensor([tm["launches"]], dtype=torch.float64, device=ctx.dev)
    if ctx.world > 1:
        dist.all_reduce(launches)
    step_e2e()
    ms_e2e = timed(ctx, step_e2e, e2e_steps)
    par = None
    if parity:
        par = oracle_parity(ctx, cfg, model, xyz, val, axes, last["z"], last["ss"], first, count, fatal=fatal_parity)
    kernel_ms = (tm["knn_solve_ms"] if k else tm["solve_ms"]) / steps
    n_launch = max(1.0, tm["solve_launches"] / steps)
    res = {
        "workload": cfg["text"] + (" [weak: slowest axis x %d]" % ctx.world if weak and ctx.world > 1 else ""),
        "n_gpus": ctx.world, "named_gpus": cfg["named_gpus"], "dtype": cfg["dtype"], "grid_points": npt,
        "steps": steps, "warmup": warmup,
        "value": npt / (ms_dev * 1e-3), "unit": UNIT, "ms_per_step": ms_dev,
        "e2e": {"value": npt / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e, "steps": e2e_steps,
                "h2d_bytes_per_step": 8 * ((cfg["dim"] + 1) * cfg["n"] + sum(sizes)), "d2h_bytes_per_step": 16 * npt},
        "phases_ms_per_step_rank0": {kk: tm[kk] / steps for kk in
                                     ("assemble_ms", "cholesky_ms", "trtri_ms", "pack_dual_ms", "solve_ms", "h2d_ms",
                                      "knn_search_ms", "knn_solve_ms") if tm.get(kk)},
        "kernel_points_per_s_rank0": count / (kernel_ms * 1e-3) if kernel_ms > 0 else None,
        "kernel_ms_rank0": kernel_ms, "kernel_launches_per_step": n_launch, "points_rank0": count,
        "gpu_launches": int(launches.item()),
        "parity_vs_oracle": par,
    }
    if par is not None and not par["pass"]:      # a side config whose numbers differ from the reference's is reported as such
        res["invalid"] = "parity against the oracle failed: the throughput of this config must not be used"
    return res, cfg


def roofline_for(cfg, res, peaks):
    """Roofline of the dominant kernel of a config from this run's own CUDA-event kernel time (rank 0)."""
    k = cfg.get("k")
    if res["kernel_ms_rank0"] <= 0:
        return None
    pts, sec = res["points_rank0"], res["kernel_ms_rank0"] * 1e-3
    alg, exe = flop_per_point(cfg), executed_flop_per_point(cfg)
    if cfg["dtype"] == "float32":
        peak, src, kern = peaks["tf32"], "torch.matmul fp32 8192^3 with TF32 allowed (cuBLAS), this run", \
            "solve_kernel_tf32 (tcgen05.mma kind::tf32, 3xTF32 split: 3 tensor MACs per algorithmic MAC)"
        exe *= 3.0
    else:
        peak, src = peaks["fp64"], "torch.matmul fp64 8192^3 (cuBLAS DGEMM), best of 3, this run"
        kern = ("knn_solve_kernel (exact kNN + k x k Cholesky per point, fp64 FMA pipe)" if k else
                "solve_kernel_pt (persistent point-tile kernel, fp64 DMMA mma.sync.m8n8k4; RHS generation and finalize fused)")
    ach = pts * alg / sec / 1e12
    return {"bound": "tensor" if not k else "fp64-fma", "kernel": kern, "achieved": ach, "peak": peak, "unit": "TFLOP/s",
            "frac": ach / peak, "achieved_executed": pts * exe / sec / 1e12, "frac_executed": pts * exe / sec / 1e12 / peak,
            "peak_source": src, "algorithmic_flop_per_point": alg, "executed_flop_per_point": exe,
            "points_per_launch": pts / res["kernel_launches_per_step"],
            "avg_launch_ms": res["kernel_ms_rank0"] / res["kernel_launches_per_step"]}


def static_traffic():
    """DRAM bytes per launch of the headline kernel from the committed ncu --set full capture (NOT measured in
    this run: ncu cannot run inside a timed bench)."""
    for rel in ("profiles/r02/solve_kernel_summary.json", "profiles/solve_kernel_summary.json"):
        p = os.path.join(ROOT, rel)
        if os.path.exists(p):
            try:
                d = json.load(open(p))
                return d.get("dram_bytes_per_launch"), "static: %s (ncu --set full, 1e6-point launch)" % rel
            except Exception:  # noqa: BLE001
                pass
    return None, "no committed ncu capture"


def run_ours(args):
    import torch
    import pykrige_b200 as pk  # noqa: F401

    ctx = Ctx()
    ctx.torch = torch
    ctx.world = int(os.environ.get("WORLD_SIZE", "1"))
    ctx.rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # libraries (NCCL prints its version) must not write to stdout: rank 0 prints exactly ONE JSON line
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: backend='cuda' has no CPU fallback")
    torch.cuda.set_device(local)
    ctx.dist = None
    if ctx.world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        ctx.dist = dist
    ctx.dev = torch.device("cuda", local)
    ctx.stream = torch.cuda.Stream(device=ctx.dev)
    ctx.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=ctx.dev)

    peaks = {"fp64": None, "tf32": None}
    if ctx.rank == 0:
        peaks["fp64"] = measure_gemm_peak(torch, torch.float64)
        peaks["tf32"] = measure_gemm_peak(torch, torch.float32, tf32=True)

    # ---- headline: cfg2, fixed 1000x1000 grid split over the ranks (strong scaling) ----
    sampler = ClockSampler(local)
    sampler.start()
    outputs = {} if args.dump_outputs else None
    head, cfg2 = bench_config(ctx, "cfg2", args.steps, args.warmup, args.steps, parity=True, fatal_parity=True,
                              outputs=outputs)
    sampler.stop_flag = True
    sampler.join(timeout=2.0)
    if outputs is not None and ctx.rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    extra = {}
    wanted = [] if args.configs == "none" else [c for c in args.configs.split(",") if c]
    osteps, owarm = min(args.steps, 3), min(args.warmup, 3)
    for name in wanted:
        if name not in CONFIGS or name == "cfg2":
            continue
        try:
            res, cfg = bench_config(ctx, name, osteps, owarm, min(2, osteps))
            if ctx.rank == 0:
                res["roofline"] = roofline_for(cfg, res, peaks)
        except Exception as e:  # noqa: BLE001  (a side config must not take the measured headline down with it)
            res = {"workload": CONFIGS[name]["text"], "error": "%s: %s" % (type(e).__name__, e)}
        extra[name] = res
    # the same grid through the fp64-class int8-slice tensor-core kernels (own driver-timed arm, dtype f64x)
    f64x = {}
    if args.configs != "none":
        for dt in ("float64x", "float64x4"):
            try:
                res, cfg = bench_config(ctx, "cfg2", osteps, owarm, min(2, osteps), dtype=dt)
            except Exception as e:  # noqa: BLE001
                res = {"workload": CONFIGS["cfg2"]["text"], "dtype": dt, "error": "%s: %s" % (type(e).__name__, e)}
            res["kernel"] = ("solve_kernel_i8: tcgen05.mma kind::i8, %s error-free slices, exact int32 accumulation in "
                             "TMEM, exact int64 recombination" % ("6 (41-bit)" if dt == "float64x" else "4 (27-bit)"))
            f64x[dt] = res
    weak = None
    if ctx.world > 1:
        try:
            w, _ = bench_config(ctx, "cfg2", osteps, owarm, min(2, osteps), weak=True, parity=False)
            weak = {kk: w[kk] for kk in ("workload", "grid_points", "value", "unit", "ms_per_step", "e2e")}
        except Exception as e:  # noqa: BLE001
            weak = {"error": "%s: %s" % (type(e).__name__, e)}

    if ctx.rank == 0:
        roof = roofline_for(cfg2, head, peaks)
        traffic, tsrc = static_traffic()
        roof["traffic"] = traffic
        roof["traffic_source"] = tsrc
        roof["note"] = ("frac = algorithmic 2(N+1)^2 flop/point (the reference's inverse GEMV, SURVEY.md 8d) over the measured "
                        "DGEMM rate; the kernel executes the covariance-form triangular product (about half of that), so frac "
                        "can exceed 1; frac_executed is the utilisation of the fp64 tensor pipe")
        cpu = cpu_arm(3, 1)[0] if ctx.world == 1 else None
        line = {
            "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": ctx.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": cfg2["text"], "n_data": cfg2["n"], "grid": list(cfg2["grid"]), "variogram": cfg2["model"],
                "variogram_parameters": cfg2["params"], "seed": cfg2["seed"],
                "l2": "flush: a 256 MiB buffer is rewritten between timed steps; each step also rewrites the 3x210 MB "
                      "factor workspaces",
                "parallelism": "grid-point sharding of the fixed grid over %d GPU(s) (strong scaling), one NCCL broadcast "
                               "of the factor blob" % ctx.world,
                "phases_ms_per_step_rank0": head["phases_ms_per_step_rank0"],
                "solve_only_points_per_s_rank0": head["kernel_points_per_s_rank0"],
                "parity_vs_oracle": head["parity_vs_oracle"],
                "weak": weak,
                "configs": extra,
                "f64x_int8_slices": f64x,
                "peaks_tflops_this_run": peaks,
            },
            "roofline": roof,
            "cpu_baseline": cpu,
            "e2e": dict(head["e2e"], api="OrdinaryKriging.execute('grid', gx, gy, backend='cuda') -> kb200_set_problem + "
                                         "kb200_execute_grid (host buffers), factorisation not cached"
                        if ctx.world == 1 else "multigpu.execute_sharded(model, 'grid', [gx, gy], dist): rank 0 factors, "
                                               "one broadcast, every rank returns its host slice"),
            "gpu_launches": head["gpu_launches"],
            "clocks": sampler.result(),
        }
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if ctx.world > 1:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--configs", default="cfg1,cfg3,cfg4,cfg5",
                    help="other BASELINE configs to run after the headline (comma list, or 'none')")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the grid the last timed headline step computed to DIR/{zvalues,sigmasq}.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
