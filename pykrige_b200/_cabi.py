"""ctypes binding of libkrige_b200.so (include/krige_b200.h).

This is the thin shim named in BASELINE.json's north_star: Python host code calling
hand-written sm_100a CUDA through a C ABI. There is no CPU fallback — if the shared
library is missing, or no CUDA device is present, the backend raises.
"""
import ctypes
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libkrige_b200.so")

KB200_OK = 0
KB200_EBADARG = -1
KB200_EUNSUPPORTED = -2
KB200_ESINGULAR = -3
KB200_ECUDA = -4
KB200_ENOMEM = -5
KB200_ESTATE = -6

KB200_F64 = 0
KB200_F32 = 1
KB200_F64X = 2   # fp64-class contraction on the INT8 tensor cores (exact slice products), 6 slices = 41 bits
KB200_F64X5 = 3  # 5 slices = 34 bits
KB200_F64X4 = 4  # 4 slices = 27 bits
DTYPES = {"float64": KB200_F64, "float32": KB200_F32, "float64x": KB200_F64X, "float64x5": KB200_F64X5,
          "float64x4": KB200_F64X4}
MAX_DRIFT = 15

# every symbol include/krige_b200.h declares (checked by tests/test_cabi.py)
EXPORTS = [
    "kb200_create", "kb200_destroy", "kb200_last_error", "kb200_version",
    "kb200_set_problem", "kb200_execute_points", "kb200_execute_grid",
    "kb200_execute_points_dev", "kb200_execute_grid_dev",
    "kb200_execute_knn_points", "kb200_execute_knn_grid", "kb200_execute_knn_grid_dev",
    "kb200_set_problem_knn",
    "kb200_blob_bytes", "kb200_blob_ptr", "kb200_describe_problem", "kb200_blob_commit",
    "kb200_set_coordinates", "kb200_set_stream", "kb200_last_timings", "kb200_reset_counters", "kb200_debug_fetch",
    "kb200_experimental_variogram", "kb200_statistics", "kb200_set_pseudo_inverse",
    "kb200_set_variogram_table", "kb200_set_device_drift",
    "kb200_group_create", "kb200_group_destroy", "kb200_group_last_error", "kb200_group_size", "kb200_group_member",
    "kb200_group_set_problem", "kb200_group_set_problem_knn", "kb200_group_execute_points",
    "kb200_group_execute_grid", "kb200_group_execute_knn_points", "kb200_group_execute_knn_grid",
]

_c_double_p = ctypes.POINTER(ctypes.c_double)
_lib = None


class KrigeB200Error(RuntimeError):
    pass


def load_library():
    """dlopen libkrige_b200.so (built by __graft_entry__.build() / make -C pykrige_b200/csrc)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise KrigeB200Error(
            "libkrige_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C pykrige_b200/csrc`. backend='cuda' has no CPU fallback." % LIB_PATH
        )
    lib = ctypes.CDLL(LIB_PATH)
    h = ctypes.c_void_p
    i64 = ctypes.c_int64
    i32 = ctypes.c_int
    dp = ctypes.c_void_p  # double* (host or device), passed as raw addresses
    lib.kb200_create.argtypes = [ctypes.POINTER(h), i32]
    lib.kb200_destroy.argtypes = [h]
    lib.kb200_destroy.restype = None
    lib.kb200_last_error.argtypes = [h]
    lib.kb200_last_error.restype = ctypes.c_char_p
    lib.kb200_version.restype = i32
    prob = [h, i32, i32, i64, dp, dp, dp, dp, dp, dp, i32, dp, i32, i32, ctypes.c_double, i32, i32, dp]
    lib.kb200_set_problem.argtypes = prob
    lib.kb200_describe_problem.argtypes = prob
    lib.kb200_set_problem_knn.argtypes = [h, i32, i64, dp, dp, dp, dp, dp, dp, i32, dp, i32, i32, ctypes.c_double]
    lib.kb200_execute_points.argtypes = [h, i64, dp, dp, dp, dp, dp, dp]
    lib.kb200_execute_points_dev.argtypes = [h, i64, dp, dp, dp, dp, dp, dp]
    grid = [h, i64, i64, i64, dp, dp, dp, dp, i64, i64, dp, dp]
    lib.kb200_execute_grid.argtypes = grid
    lib.kb200_execute_grid_dev.argtypes = grid
    lib.kb200_execute_knn_points.argtypes = [h, i32, i64, dp, dp, dp, dp, dp]
    kgrid = [h, i32, i64, i64, i64, dp, dp, dp, i64, i64, dp, dp]
    lib.kb200_execute_knn_grid.argtypes = kgrid
    lib.kb200_execute_knn_grid_dev.argtypes = kgrid
    lib.kb200_blob_bytes.argtypes = [h]
    lib.kb200_blob_bytes.restype = i64
    lib.kb200_blob_ptr.argtypes = [h]
    lib.kb200_blob_ptr.restype = ctypes.c_void_p
    lib.kb200_blob_commit.argtypes = [h]
    lib.kb200_set_coordinates.argtypes = [h, i32]
    lib.kb200_set_stream.argtypes = [h, ctypes.c_void_p]
    lib.kb200_last_timings.argtypes = [h, _c_double_p, i32]
    lib.kb200_reset_counters.argtypes = [h]
    lib.kb200_reset_counters.restype = None
    lib.kb200_debug_fetch.argtypes = [h, i32, dp, i64]
    lib.kb200_debug_fetch.restype = i64
    lib.kb200_experimental_variogram.argtypes = [h, i32, i64, dp, dp, dp, dp, i32, dp, dp, dp, dp]
    lib.kb200_statistics.argtypes = [h, dp, dp]
    lib.kb200_set_pseudo_inverse.argtypes = [h, i32]
    lib.kb200_set_variogram_table.argtypes = [h, i64, ctypes.c_double, dp]
    lib.kb200_set_device_drift.argtypes = [h, i32, dp, i64, i64, dp, dp, dp]
    lib.kb200_group_create.argtypes = [ctypes.POINTER(h), i32, ctypes.POINTER(i32)]
    lib.kb200_group_destroy.argtypes = [h]
    lib.kb200_group_destroy.restype = None
    lib.kb200_group_last_error.argtypes = [h]
    lib.kb200_group_last_error.restype = ctypes.c_char_p
    lib.kb200_group_size.argtypes = [h]
    lib.kb200_group_member.argtypes = [h, i32]
    lib.kb200_group_member.restype = ctypes.c_void_p
    lib.kb200_group_set_problem.argtypes = prob
    lib.kb200_group_set_problem_knn.argtypes = lib.kb200_set_problem_knn.argtypes
    lib.kb200_group_execute_points.argtypes = lib.kb200_execute_points.argtypes
    lib.kb200_group_execute_grid.argtypes = grid
    lib.kb200_group_execute_knn_points.argtypes = lib.kb200_execute_knn_points.argtypes
    lib.kb200_group_execute_knn_grid.argtypes = kgrid
    _lib = lib
    return lib


_aux = None
_aux_error = None


def aux_handle():
    """One shared Handle for the constructor-side device helpers (experimental variogram). Raises
    KrigeB200Error when the library or a CUDA device is missing (the failure is cached)."""
    global _aux, _aux_error
    if _aux is not None:
        return _aux
    if _aux_error is not None:
        raise KrigeB200Error(_aux_error)
    try:
        _aux = Handle()
    except KrigeB200Error as e:
        _aux_error = str(e)
        raise
    return _aux


def device_available():
    try:
        aux_handle()
        return True
    except KrigeB200Error:
        return False


def _ptr(a):
    return None if a is None else a.ctypes.data


def _f64(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


TIMING_KEYS = ["assemble_ms", "cholesky_ms", "trtri_ms", "pack_dual_ms", "solve_ms", "finalize_ms",
               "h2d_ms", "d2h_ms", "knn_search_ms", "knn_solve_ms", "solve_launches", "launches", "solve_slices"]


class Handle:
    """Owns one kb200_handle. Error codes are mapped to the exception types the reference
    raises at the same places (SURVEY.md §8b)."""

    _PREFIX = "kb200_"
    _owned = True

    @classmethod
    def _borrowed(cls, lib, raw):
        """A view of a handle owned by someone else (a group member): never destroyed from here."""
        self = cls.__new__(cls)
        self.lib = lib
        self._h = ctypes.c_void_p(raw)
        self._owned = False
        return self

    def __init__(self, device=-1):
        self.lib = load_library()
        self._h = ctypes.c_void_p()
        rc = self.lib.kb200_create(ctypes.byref(self._h), int(device))
        if rc != KB200_OK:
            self._h = None
            raise KrigeB200Error(
                "kb200_create failed (code %d): no usable CUDA device. backend='cuda' has no CPU fallback." % rc
            )

    def close(self):
        if getattr(self, "_h", None):
            if self._owned:
                self.lib.kb200_destroy(self._h)
            self._h = None

    def _fn(self, name):
        return getattr(self.lib, self._PREFIX + name)

    def _errmsg(self):
        msg = self.lib.kb200_last_error(self._h)
        return msg.decode() if msg else ""

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, knn=False):
        if rc == KB200_OK:
            return
        msg = self._errmsg()
        if rc == KB200_EBADARG:
            raise ValueError(msg)
        if rc == KB200_EUNSUPPORTED:
            raise NotImplementedError(msg)
        if rc == KB200_ESINGULAR:
            if knn:
                raise ValueError("Singular matrix")  # cok.pyx:176-179
            raise np.linalg.LinAlgError(msg or "singular matrix")  # scipy.linalg.inv behaviour
        if rc == KB200_ENOMEM:
            raise MemoryError(msg)
        raise KrigeB200Error("libkrige_b200 error %d: %s" % (rc, msg))

    # -- problem description ---------------------------------------------------------
    def _problem_args(self, dim, dtype, x, y, z, values, center, aniso, model, vparams, exact_values, eps,
                      n_rl, drift_data):
        x, y, values = _f64(x), _f64(y), _f64(values)
        z = _f64(z) if dim == 3 else None
        center = _f64(center)
        aniso = _f64(np.asarray(aniso).reshape(-1))
        vparams = _f64(vparams)
        n_hd = 0
        if drift_data is not None and len(drift_data):
            drift_data = _f64(np.asarray(drift_data, dtype=np.float64).reshape(len(drift_data), -1))
            n_hd = drift_data.shape[0]
        else:
            drift_data = None
        keep = (x, y, z, values, center, aniso, vparams, drift_data)
        args = [self._h, int(dim), int(dtype), int(x.size), _ptr(x), _ptr(y), _ptr(z), _ptr(values),
                _ptr(center), _ptr(aniso), int(model), _ptr(vparams), int(vparams.size),
                int(bool(exact_values)), float(eps), int(n_rl), int(n_hd), _ptr(drift_data)]
        return args, keep

    def set_problem(self, dim, dtype, x, y, z, values, center, aniso, model, vparams, exact_values, eps,
                    n_rl=0, drift_data=None):
        args, keep = self._problem_args(dim, dtype, x, y, z, values, center, aniso, model, vparams,
                                        exact_values, eps, n_rl, drift_data)
        self._check(self._fn("set_problem")(*args))

    def describe_problem(self, dim, dtype, x, y, z, values, center, aniso, model, vparams, exact_values, eps,
                         n_rl=0, drift_data=None):
        args, keep = self._problem_args(dim, dtype, x, y, z, values, center, aniso, model, vparams,
                                        exact_values, eps, n_rl, drift_data)
        self._check(self.lib.kb200_describe_problem(*args))

    def set_problem_knn(self, dim, x, y, z, values, center, aniso, model, vparams, exact_values, eps):
        x, y, values = _f64(x), _f64(y), _f64(values)
        z = _f64(z) if dim == 3 else None
        center = _f64(center)
        aniso = _f64(np.asarray(aniso).reshape(-1))
        vparams = _f64(vparams)
        self._check(self._fn("set_problem_knn")(
            self._h, int(dim), int(x.size), _ptr(x), _ptr(y), _ptr(z), _ptr(values), _ptr(center), _ptr(aniso),
            int(model), _ptr(vparams), int(vparams.size), int(bool(exact_values)), float(eps)))

    # -- execute (host buffers) --------------------------------------------------------
    def execute_points(self, px, py, pz=None, drift_pts=None):
        px, py, pz = _f64(px), _f64(py), _f64(pz)
        m = px.size
        z = np.empty(m, dtype=np.float64)
        ss = np.empty(m, dtype=np.float64)
        dpts = _f64(drift_pts)
        self._check(self._fn("execute_points")(self._h, m, _ptr(px), _ptr(py), _ptr(pz), _ptr(dpts),
                                                  _ptr(z), _ptr(ss)))
        return z, ss

    def execute_grid(self, gx, gy, gz=None, drift_pts=None, first=0, count=None):
        gx, gy, gz = _f64(gx), _f64(gy), _f64(gz)
        nx, ny, nz = gx.size, gy.size, (gz.size if gz is not None else 1)
        if count is None:
            count = nx * ny * nz - first
        z = np.empty(count, dtype=np.float64)
        ss = np.empty(count, dtype=np.float64)
        dpts = _f64(drift_pts)
        self._check(self._fn("execute_grid")(self._h, nx, ny, nz, _ptr(gx), _ptr(gy), _ptr(gz), _ptr(dpts),
                                                int(first), int(count), _ptr(z), _ptr(ss)))
        return z, ss

    def execute_knn_points(self, k, px, py, pz=None):
        px, py, pz = _f64(px), _f64(py), _f64(pz)
        m = px.size
        z = np.empty(m, dtype=np.float64)
        ss = np.empty(m, dtype=np.float64)
        self._check(self._fn("execute_knn_points")(self._h, int(k), m, _ptr(px), _ptr(py), _ptr(pz),
                                                      _ptr(z), _ptr(ss)), knn=True)
        return z, ss

    def execute_knn_grid(self, k, gx, gy, gz=None, first=0, count=None):
        gx, gy, gz = _f64(gx), _f64(gy), _f64(gz)
        nx, ny, nz = gx.size, gy.size, (gz.size if gz is not None else 1)
        if count is None:
            count = nx * ny * nz - first
        z = np.empty(count, dtype=np.float64)
        ss = np.empty(count, dtype=np.float64)
        self._check(self._fn("execute_knn_grid")(self._h, int(k), nx, ny, nz, _ptr(gx), _ptr(gy), _ptr(gz),
                                                    int(first), int(count), _ptr(z), _ptr(ss)), knn=True)
        return z, ss

    # -- execute (device pointers: raw addresses, e.g. torch_tensor.data_ptr()) -----------
    def execute_grid_dev(self, nx, ny, nz, d_gx, d_gy, d_gz, d_drift, first, count, d_z, d_ss):
        self._check(self.lib.kb200_execute_grid_dev(self._h, int(nx), int(ny), int(nz), d_gx, d_gy, d_gz, d_drift,
                                                    int(first), int(count), d_z, d_ss))

    def execute_points_dev(self, m, d_px, d_py, d_pz, d_drift, d_z, d_ss):
        self._check(self.lib.kb200_execute_points_dev(self._h, int(m), d_px, d_py, d_pz, d_drift, d_z, d_ss))

    def execute_knn_grid_dev(self, k, nx, ny, nz, d_gx, d_gy, d_gz, first, count, d_z, d_ss):
        self._check(self.lib.kb200_execute_knn_grid_dev(self._h, int(k), int(nx), int(ny), int(nz), d_gx, d_gy, d_gz,
                                                        int(first), int(count), d_z, d_ss), knn=True)

    # -- multi-GPU factor blob -----------------------------------------------------------
    def blob(self):
        return int(self.lib.kb200_blob_ptr(self._h) or 0), int(self.lib.kb200_blob_bytes(self._h))

    def blob_commit(self):
        self._check(self.lib.kb200_blob_commit(self._h))

    def set_coordinates(self, geographic):
        self._check(self.lib.kb200_set_coordinates(self._h, 1 if geographic else 0))

    def set_stream(self, cuda_stream):
        self._check(self.lib.kb200_set_stream(self._h, ctypes.c_void_p(int(cuda_stream))))

    # -- instrumentation ------------------------------------------------------------------
    def timings(self):
        buf = (ctypes.c_double * len(TIMING_KEYS))()
        n = self.lib.kb200_last_timings(self._h, buf, len(TIMING_KEYS))
        return {TIMING_KEYS[i]: buf[i] for i in range(n)}

    def reset_counters(self):
        self.lib.kb200_reset_counters(self._h)

    def set_variogram_table(self, nodes, dmax):
        """nodes[i] = gamma at d_i = dmax * (i / (len - 1))**2 (KB200_VG_TABLE, 'custom' callables)."""
        nodes = _f64(nodes)
        self._check(self.lib.kb200_set_variogram_table(self._h, nodes.size, float(dmax), _ptr(nodes)))

    def set_pseudo_inverse(self, enable):
        self._check(self.lib.kb200_set_pseudo_inverse(self._h, 1 if enable else 0))

    def set_device_drift(self, wells, ext):
        """Drift terms the solve kernels evaluate at the prediction points themselves (kb200_set_device_drift):
        wells = [n_wells, 3] (adjusted x, adjusted y, strength) or None; ext = (axis_x, axis_y, raster[ny, nx])
        or None."""
        w = _f64(np.asarray(wells, dtype=np.float64).reshape(-1, 3)) if wells is not None and len(wells) else None
        if ext is not None:
            ex, ey, ez = _f64(np.ravel(ext[0])), _f64(np.ravel(ext[1])), _f64(ext[2])
            if ez.shape != (ey.size, ex.size):
                raise ValueError("external drift raster must be shaped (len(y), len(x))")
            args = (ex.size, ey.size, _ptr(ex), _ptr(ey), _ptr(ez))
        else:
            args = (0, 0, None, None, None)
        self._check(self.lib.kb200_set_device_drift(self._h, 0 if w is None else w.shape[0], _ptr(w), *args))

    def experimental_variogram(self, X, values, nlags, geographic=False):
        """Device twin of the pdist binning (core.py:432-505): X = (n, 2|3) ADJUSTED coordinates (or
        lon/lat when geographic). Returns (counts, lag_sum, semi_sum, dmin, dmax)."""
        X = np.asarray(X, dtype=np.float64)
        dim = X.shape[1]
        cols = [_f64(X[:, c]) for c in range(dim)]
        v = _f64(values)
        nl = int(nlags)
        cnt, sd, sg, mm = (np.zeros(max(nl, 0)), np.zeros(max(nl, 0)), np.zeros(max(nl, 0)), np.zeros(2))
        self._check(self.lib.kb200_set_coordinates(self._h, 1 if geographic else 0))
        self._check(self.lib.kb200_experimental_variogram(
            self._h, dim, X.shape[0], _ptr(cols[0]), _ptr(cols[1]), _ptr(cols[2]) if dim > 2 else None,
            _ptr(v), nl, _ptr(cnt), _ptr(sd), _ptr(sg), _ptr(mm)))
        return cnt, sd, sg, float(mm[0]), float(mm[1])

    def statistics(self, n):
        """(delta, sigma) of core._find_statistics (core.py:759-836) from the factor of the current
        problem; skipped points are 0."""
        delta = np.zeros(int(n))
        sigma = np.zeros(int(n))
        self._check(self.lib.kb200_statistics(self._h, _ptr(delta), _ptr(sigma)))
        return delta, sigma

    def debug_fetch(self, what, count):
        out = np.empty(int(count), dtype=np.float64)
        got = self.lib.kb200_debug_fetch(self._h, int(what), _ptr(out), int(count))
        if got < 0:
            self._check(int(got))
        return out[:got]


class Group(Handle):
    """kb200_group: n_gpus handles behind one call from one host thread (single-process multi-GPU). Same
    execute / set_problem methods as Handle; configuration calls fan out to the members."""

    _PREFIX = "kb200_group_"

    def __init__(self, n_gpus, devices=None):
        self.lib = load_library()
        self._h = ctypes.c_void_p()
        dev = None
        if devices is not None:
            dev = (ctypes.c_int * int(n_gpus))(*[int(d) for d in devices])
        rc = self.lib.kb200_group_create(ctypes.byref(self._h), int(n_gpus), dev)
        if rc != KB200_OK:
            self._h = None
            if rc == KB200_EBADARG:
                raise ValueError("n_gpus=%d: this box does not have that many CUDA devices" % int(n_gpus))
            raise KrigeB200Error("kb200_group_create failed (code %d): no usable CUDA device" % rc)
        self.size = int(self.lib.kb200_group_size(self._h))
        self.members = [Handle._borrowed(self.lib, self.lib.kb200_group_member(self._h, i)) for i in range(self.size)]

    def close(self):
        if getattr(self, "_h", None):
            for m in self.members:
                m._h = None
            self.lib.kb200_group_destroy(self._h)
            self._h = None

    def _errmsg(self):
        msg = self.lib.kb200_group_last_error(self._h)
        return msg.decode() if msg else ""

    def describe_problem(self, *a, **k):
        raise NotImplementedError("a group factors on its first device and copies the blob itself")

    # configuration: per member
    def set_coordinates(self, geographic):
        for m in self.members:
            m.set_coordinates(geographic)

    def set_pseudo_inverse(self, enable):
        for m in self.members:
            m.set_pseudo_inverse(enable)

    def set_variogram_table(self, nodes, dmax):
        for m in self.members:
            m.set_variogram_table(nodes, dmax)

    def set_device_drift(self, wells, ext):
        for m in self.members:
            m.set_device_drift(wells, ext)

    # instrumentation / constructor-side helpers: the factoring member
    def timings(self):
        return self.members[0].timings()

    def reset_counters(self):
        for m in self.members:
            m.reset_counters()

    def statistics(self, n):
        return self.members[0].statistics(n)

    def blob(self):
        return self.members[0].blob()
