"""Generate tests/golden/ref_native.npz from the reference's own compiled twins of the hot path
(`_c_exec_loop` / `_c_exec_loop_moving_window` of lib/cok.pyx, built into oracle/_ref by oracle/build_ref.py).

    python oracle/build_ref.py && python tests/golden/make_golden_native.py

A script of its own because make_golden.py imports the reference's pure-Python package as `pykrige`, and the compiled
twins have to be imported under that same package name. Inputs are tests/cases.py NATIVE_INPUTS; each entry stores
(z, sigmasq) as <input>/<variant>/z and .../ss, plus <input>/fp, a fingerprint of the inputs that lets the tests
detect a drifting RNG.
"""
import os
import sys
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cases  # noqa: E402
from oracle import krige_oracle as ko, ref_native as rn  # noqa: E402

# variogram of the moving-window comparisons
WINDOW_MODEL, WINDOW_PARAMS = "exponential", [1.0, 150.0, 0.05]


def fingerprint(xyz, val, pts):
    return np.array([xyz.sum(), val.sum(), pts.sum()])


def main():
    if not rn.available():
        raise SystemExit("oracle/_ref is not built: run python oracle/build_ref.py first")
    out = {}

    def put(key, zs):
        out[key + "/z"], out[key + "/ss"] = (np.asarray(a, dtype=np.float64) for a in zs)

    xyz, val, pts = cases.native_inputs("global2d")
    out["global2d/fp"] = fingerprint(xyz, val, pts)
    for model in ("linear", "power", "gaussian", "exponential", "spherical"):
        stored = ko.stored_parameters(model, cases.MODELS[model])
        for exact in (True, False):
            put("global2d/%s/%s" % (model, "exact" if exact else "inexact"),
                rn.exec_loop(xyz, pts, val, model, stored, exact_values=exact))
    stored = ko.stored_parameters(WINDOW_MODEL, WINDOW_PARAMS)
    for name, k in (("window2d", 8), ("window3d", 12)):
        xyz, val, pts = cases.native_inputs(name)
        out[name + "/fp"] = fingerprint(xyz, val, pts)
        put("%s/k%d" % (name, k), rn.exec_loop_moving_window(xyz, pts, val, WINDOW_MODEL, stored, k))
    xyz, val, pts = cases.native_inputs("cuda2d")
    out["cuda2d/fp"] = fingerprint(xyz, val, pts)
    for model in ("exponential", "spherical", "linear"):
        put("cuda2d/" + model, rn.exec_loop(xyz, pts, val, model, ko.stored_parameters(model, cases.MODELS[model])))
    put("cuda2d/k16", rn.exec_loop_moving_window(xyz, pts, val, WINDOW_MODEL, stored, 16))
    np.savez_compressed(os.path.join(HERE, "ref_native.npz"), **out)
    for key in sorted(out):
        print("%-32s %s mean=%.6f" % (key, out[key].shape, float(np.mean(out[key]))))


if __name__ == "__main__":
    main()
