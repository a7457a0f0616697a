// api.cu — C ABI of libkrige_b200.so (include/krige_b200.h): handle, problem set-up,
// orchestration of the factor kernels (factor.cu), the fused solve (solve.cu) and the
// moving window (knn.cu). Host code only; no torch types, no CPU compute path.
#include <cuda_runtime.h>
#include <string>
#include <vector>
#include <cstring>
#include <cstdio>
#include <cmath>
#include <cstdlib>
#include <algorithm>
#include <thread>
#include "kernels.h"

#define KB_VERSION 2000
static const int64_t KB_STAGE_PTS = 1 << 20;   // prediction points per staged output chunk (2 x 8 MB through pinned memory)
#define KB_TILE_COST_32 0.532     // one round of 32-point tiles relative to one round of 64-point tiles (fp64 kernel, N=5000:
#define KB_TILE_COST_16 0.301     // 7.34 / 3.91 / 2.21 ms per round; scripts/tile_timing.py, profiles/r02/tile_width_timing_run21.log)
static const int64_t KB_STAGE_MIN = 1 << 18;   // below this the outputs go straight to the caller's buffers

struct Src {
    bool grid; int64_t nx, ny, nz;
    const double *a, *b, *c;      // points (px,py,pz) or axes (gx,gy,gz), device pointers
    int64_t first, count;
    const double* d_drift; int64_t drift_stride, drift_first;
};

// general (indefinite) path: blocked Gauss-Jordan unless KB200_GJ=scalar
#define KB_GJ_DEFAULT_BLOCKED 1

// dtype='float64' contraction: on the Cholesky path with KB_F64_I8_NMIN <= n <= KB_F64_I8_NMAX the INT8 slice kernel with
// 8 exact slices (55 bits, as accurate as the fp64 product; solve_i8.cu), else the DMMA kernel (solve.cu). The int32
// accumulators bound n (n * 8 * 64^2 < 2^31). Solve kernel, int8 over DMMA on a B200: 1.00x at n=256, 1.17x at 512,
// 1.42x at 1024, 1.73x at 2048 (profiles/README.md, scripts/f64_route_timing.py).
#define KB_F64_I8_SLICES 8
#define KB_F64_I8_NMIN 512
#define KB_F64_I8_NMAX 65535

// Slice count of the contraction of a dtype='float64' problem (0 = DMMA). A function of the problem alone, never of the
// prediction points, so that shards, chunks and devices all run the same kernel. KB200_F64_SOLVE=dmma | int8 overrides
// the size rule; it is the cross-check and profiling switch of the tests and scripts, read when a problem is described.
static int f64_route_slices(int64_t n, bool pinv) {
    if (pinv || n > KB_F64_I8_NMAX) return 0;
    if (const char* e = std::getenv("KB200_F64_SOLVE")) {
        if (std::strcmp(e, "dmma") == 0) return 0;
        if (std::strcmp(e, "int8") == 0) return KB_F64_I8_SLICES;
    }
    return n >= KB_F64_I8_NMIN ? KB_F64_I8_SLICES : 0;
}

struct DevBuf {
    void* p = nullptr; size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct kb200_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;

    // description
    bool described = false, ready = false, knn_ready = false;
    bool factor_live = false;  // L (wC) and the forward solves (wF) of the ready problem are still in the workspace
    int slices = 0;           // contraction on the INT8 slice kernel: number of slices (float64: 8; float64x*: 6 / 5 / 4), else 0
    int gform = 0;            // 1: general (indefinite) fallback, tiles hold the symmetric inverse
    int geo = 0;              // 1: coordinates_type='geographic' for the next problem description
    int pinv = 0;             // 1: pseudo_inv=True for the next problem description (global path only)
    int pinv_sweeps = 0, pinv_rank = 0;
    int dim = 2, dtype = KB200_F64, n = 0, n_pad = 0, ld = 0, n_rl = 0, n_hd = 0, K1 = 1, na = 2, nrb = 0;
    VgParams vg{};
    Aniso an{};
    DriftScale ds{};
    PackMap pm{};
    std::vector<double> hx, hy, hz, hval, hdrift;
    double bb_lo[3] = {0, 0, 0}, bb_hi[3] = {0, 0, 0};   // adjusted bounding box of the data

    // blob (one allocation): header | consts | ax | ay | az | tiles
    DevBuf blob;
    size_t off_consts = 0, off_ax = 0, off_ay = 0, off_az = 0, off_tiles = 0, off_rowscale = 0, blob_bytes = 0;

    // factor workspace
    DevBuf wC, wW, wT, wF, wRaw, wFlag;
    // execute workspace
    DevBuf wPart, wAux, wPts, wOut, wAxes, wDrift, wScratch;
    int num_sms = 148;
    // device-evaluated drift terms (kb200_set_device_drift): configuration + the count used by the described problem
    DeviceDrift dd{};
    DevBuf wWells, wExt;
    int n_dev = 0;
    // pinned staging of the outputs (two chunks in flight) and the stream that drains them
    void* pin[2] = {nullptr, nullptr};
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t evk[2] = {}, evc[2] = {};
    // look-ahead Cholesky: high-priority side stream for the panel chain + ordering events
    cudaStream_t hi_stream = nullptr;
    std::vector<cudaEvent_t> fev;
    // knn workspace
    DevBuf kSorted, kCells;
    DevBuf wVario;            // constructor-side helpers (experimental variogram, statistics)
    DevBuf wTab;              // KB200_VG_TABLE: (value, slope) pairs on the device
    std::vector<double> htab; // ... and on the host (value, slope interleaved), for the covariance shift
    double tab_dmax = 0.0; int tab_n = 0;
    KnnParams kp{};
    int k_ncells = 0;

    cudaEvent_t ev[16] = {};
    double tm[13] = {};
    long long launches = 0, solve_launches = 0;
};

static int fail(kb200_ctx* h, int code, const std::string& msg) {
    if (h) h->err = msg;
    return code;
}
#define CU(h, expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { \
    return fail(h, _e == cudaErrorMemoryAllocation ? KB200_ENOMEM : KB200_ECUDA, \
                std::string(#expr) + ": " + cudaGetErrorString(_e)); } } while (0)

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

extern "C" int kb200_version(void) { return KB_VERSION; }

extern "C" int kb200_create(kb200_handle* out, int device) {
    if (!out) return KB200_EBADARG;
    *out = nullptr;
    int cnt = 0;
    cudaError_t e = cudaGetDeviceCount(&cnt);
    if (e != cudaSuccess || cnt == 0) return KB200_ECUDA;   // no CPU fallback by design
    kb200_ctx* h = new kb200_ctx();
    if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) device = 0; }
    if (device >= cnt) { delete h; return KB200_EBADARG; }
    h->device = device;
    if (cudaSetDevice(device) != cudaSuccess) { delete h; return KB200_ECUDA; }
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { delete h; return KB200_ECUDA; }
    h->own_stream = true;
    for (auto& ev : h->ev) if (cudaEventCreate(&ev) != cudaSuccess) { delete h; return KB200_ECUDA; }
    if (kbk_factor_init() != cudaSuccess || kbk_solve_init() != cudaSuccess || kbk_solve_tf32_init() != cudaSuccess ||
        kbk_solve_i8_init() != cudaSuccess || kbk_ev_init() != cudaSuccess || kbk_pinv_init() != cudaSuccess) { delete h; return KB200_ECUDA; }
    if (cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || h->num_sms < 1) h->num_sms = 148;
    *out = h;
    return KB200_OK;
}

extern "C" void kb200_destroy(kb200_handle h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    for (DevBuf* b : {&h->blob, &h->wC, &h->wW, &h->wT, &h->wF, &h->wRaw, &h->wFlag, &h->wPart, &h->wAux,
                      &h->wPts, &h->wOut, &h->wAxes, &h->wDrift, &h->wScratch, &h->kSorted, &h->kCells, &h->wVario, &h->wTab,
                      &h->wWells, &h->wExt}) b->release();
    for (int i = 0; i < 2; ++i) {
        if (h->pin[i]) cudaFreeHost(h->pin[i]);
        if (h->evk[i]) cudaEventDestroy(h->evk[i]);
        if (h->evc[i]) cudaEventDestroy(h->evc[i]);
    }
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->hi_stream) cudaStreamDestroy(h->hi_stream);
    for (auto& e : h->fev) cudaEventDestroy(e);
    for (auto& ev : h->ev) if (ev) cudaEventDestroy(ev);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

extern "C" const char* kb200_last_error(kb200_handle h) { return h ? h->err.c_str() : "null handle"; }

extern "C" int kb200_set_stream(kb200_handle h, void* s) {
    if (!h) return KB200_EBADARG;
    if (h->own_stream && h->stream) { cudaStreamSynchronize(h->stream); cudaStreamDestroy(h->stream); }
    h->stream = reinterpret_cast<cudaStream_t>(s);
    h->own_stream = false;
    return KB200_OK;
}

extern "C" int kb200_set_coordinates(kb200_handle h, int coordinates_type) {
    if (!h) return KB200_EBADARG;
    if (coordinates_type != KB200_EUCLIDEAN && coordinates_type != KB200_GEOGRAPHIC)
        return fail(h, KB200_EBADARG, "coordinates_type must be KB200_EUCLIDEAN or KB200_GEOGRAPHIC");
    h->geo = coordinates_type == KB200_GEOGRAPHIC ? 1 : 0;
    h->described = false; h->ready = false; h->knn_ready = false; h->factor_live = false;
    return KB200_OK;
}

extern "C" int kb200_set_pseudo_inverse(kb200_handle h, int enable) {
    if (!h) return KB200_EBADARG;
    h->pinv = enable ? 1 : 0;
    h->described = false; h->ready = false; h->knn_ready = false; h->factor_live = false;
    return KB200_OK;
}

extern "C" void kb200_reset_counters(kb200_handle h) {
    if (!h) return;
    h->launches = 0; h->solve_launches = 0;
    for (double& t : h->tm) t = 0.0;
}

extern "C" int kb200_last_timings(kb200_handle h, double* ms, int n) {
    if (!h || !ms) return KB200_EBADARG;
    h->tm[10] = (double)h->solve_launches;
    h->tm[11] = (double)h->launches;
    h->tm[12] = (double)h->slices;
    int m = std::min(n, 13);
    for (int i = 0; i < m; ++i) ms[i] = h->tm[i];
    return m;
}

// gamma on the host (only to choose the covariance shift c0)
static double host_gamma(const kb200_ctx* h, const VgParams& v, double d) {
    switch (v.model) {
        case KB200_VG_LINEAR: return v.p0 * d + v.p1;
        case KB200_VG_POWER: return v.p0 * std::pow(d, v.p1) + v.p2;
        case KB200_VG_TABLE: {
            // same cubic Hermite as kb_gamma<KB200_VG_TABLE>; the largest tabulated value up to d, so that the
            // shift also covers non-monotone callables
            if (h->tab_n < 2) return 1.0;
            const double inv_h = (h->tab_n - 1) / std::sqrt(h->tab_dmax);
            int last = (int)std::min<double>(h->tab_n - 1, std::ceil(std::sqrt(std::max(d, 0.0)) * inv_h));
            double g = h->htab[0];
            for (int i = 0; i <= last; ++i) g = std::max(g, h->htab[2 * (size_t)i]);
            return g;
        }
        default: return v.p0 + v.p2;
    }
}

extern "C" int kb200_set_variogram_table(kb200_handle h, int64_t n_nodes, double dmax, const double* gamma_nodes) {
    if (!h) return KB200_EBADARG;
    if (n_nodes < 16 || n_nodes > (1LL << 26) || !gamma_nodes || !(dmax > 0.0) || !std::isfinite(dmax))
        return fail(h, KB200_EBADARG, "variogram table: 16 <= n_nodes <= 2^26, dmax > 0");
    const int n = (int)n_nodes;
    for (int i = 0; i < n; ++i)
        if (!std::isfinite(gamma_nodes[i])) return fail(h, KB200_EBADARG, "variogram table: the callable must be finite on [0, dmax] (node " + std::to_string(i) + ")");
    h->described = false; h->ready = false; h->knn_ready = false; h->factor_live = false;
    // slopes per unit node index: centred differences, second-order one-sided at the two ends
    h->htab.resize(2 * (size_t)n);
    for (int i = 0; i < n; ++i) {
        double m;
        if (i == 0) m = -1.5 * gamma_nodes[0] + 2.0 * gamma_nodes[1] - 0.5 * gamma_nodes[2];
        else if (i == n - 1) m = 1.5 * gamma_nodes[n - 1] - 2.0 * gamma_nodes[n - 2] + 0.5 * gamma_nodes[n - 3];
        else m = 0.5 * (gamma_nodes[i + 1] - gamma_nodes[i - 1]);
        h->htab[2 * (size_t)i] = gamma_nodes[i];
        h->htab[2 * (size_t)i + 1] = m;
    }
    h->tab_n = n; h->tab_dmax = dmax;
    cudaSetDevice(h->device);
    CU(h, h->wTab.reserve(h->htab.size() * sizeof(double)));
    CU(h, cudaMemcpyAsync(h->wTab.p, h->htab.data(), h->htab.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    return KB200_OK;
}

// ---- description (shared by set_problem / describe_problem / set_problem_knn) ----
static int describe(kb200_ctx* h, bool knn_only, int dim, int dtype, int64_t n,
                    const double* x, const double* y, const double* z, const double* values,
                    const double* center, const double* aniso, int model, const double* vparams, int n_vparams,
                    int exact_values, double eps, int n_rl, int n_hd, const double* drift_data) {
    if (!h) return KB200_EBADARG;
    h->described = false; h->ready = false; h->knn_ready = false; h->factor_live = false;
    if (dim != 2 && dim != 3) return fail(h, KB200_EBADARG, "dim must be 2 or 3");
    if (h->geo && dim != 2) return fail(h, KB200_EBADARG, "geographic coordinates are two-dimensional (lon, lat)");
    if (h->geo && (n_rl || n_hd)) return fail(h, KB200_EUNSUPPORTED, "universal kriging has no geographic mode (uk.py:337)");
    if (dtype < KB200_F64 || dtype > KB200_F64X4)
        return fail(h, KB200_EBADARG, "dtype must be KB200_F64, KB200_F32, KB200_F64X, KB200_F64X5 or KB200_F64X4");
    if (n < 1 || (!knn_only && n > (int64_t)(KB_MAXRB - 1) * KB_BM) || n > (1LL << 30)) return fail(h, KB200_EBADARG, "n out of range");
    if (!x || !y || (dim == 3 && !z) || !values || !center || !aniso || (!vparams && model != KB200_VG_TABLE))
        return fail(h, KB200_EBADARG, "null input array");
    if (model < KB200_VG_LINEAR || model > KB200_VG_TABLE)
        return fail(h, KB200_EUNSUPPORTED, "variogram model has no device implementation");
    int need = (model == KB200_VG_TABLE) ? 0 : (model == KB200_VG_LINEAR) ? 2 : 3;
    if (model == KB200_VG_TABLE) {
        if (h->tab_n < 16) return fail(h, KB200_ESTATE, "KB200_VG_TABLE: call kb200_set_variogram_table first");
        if (n_vparams != 0 && !vparams) return fail(h, KB200_EBADARG, "null input array");
    } else if (n_vparams != need) return fail(h, KB200_EBADARG, "wrong number of variogram parameters");
    if (!(n_rl == 0 || n_rl == dim)) return fail(h, KB200_EBADARG, "n_rl must be 0 or dim");
    if (n_hd < 0 || n_rl + n_hd > KB200_MAX_DRIFT) return fail(h, KB200_EBADARG, "too many drift terms");
    if (n_hd > 0 && !drift_data) return fail(h, KB200_EBADARG, "drift_data is null");
    if (knn_only && (n_rl || n_hd)) return fail(h, KB200_EUNSUPPORTED, "moving window supports ordinary kriging only");
    const int n_dev = h->dd.n_wells + h->dd.ext;
    if (n_dev > n_hd) return fail(h, KB200_EBADARG, "device drift terms (kb200_set_device_drift) exceed the n_hd described drift columns");
    if (n_dev && dim != 2) return fail(h, KB200_EUNSUPPORTED, "point_log / external_Z drift terms are two-dimensional (uk.py)");
    h->n_dev = n_dev;
    h->slices = dtype == KB200_F64X ? 6 : dtype == KB200_F64X5 ? 5 : dtype == KB200_F64X4 ? 4 : 0;
    if (dtype == KB200_F64 && !knn_only) h->slices = f64_route_slices(n, h->pinv != 0);

    const int user_dim = dim;
    h->dim = h->geo ? KB_GEO : dim; h->dtype = dtype; h->n = (int)n; h->n_rl = n_rl; h->n_hd = n_hd;
    h->K1 = n_rl + n_hd + 1; h->na = h->K1 + 1;
    h->vg.model = model;
    h->vg.p0 = need > 0 ? vparams[0] : 0.0; h->vg.p1 = need > 1 ? vparams[1] : 0.0; h->vg.p2 = (need == 3) ? vparams[2] : 0.0;
    h->vg.inv_a = 0.0;
    if (model == KB200_VG_EXPONENTIAL || model == KB200_VG_HOLE_EFFECT) h->vg.inv_a = 1.0 / (h->vg.p1 / 3.0);
    else if (model == KB200_VG_GAUSSIAN) { const double r = h->vg.p1 * (4.0 / 7.0); h->vg.inv_a = 1.0 / (r * r); }
    else if (model == KB200_VG_SPHERICAL) h->vg.inv_a = 1.0 / h->vg.p1;
    h->vg.tab = h->wTab.as<double2>(); h->vg.tab_n = h->tab_n;
    h->vg.tab_inv_h = h->tab_n > 1 ? (h->tab_n - 1) / std::sqrt(h->tab_dmax) : 0.0;
    h->vg.eps = eps; h->vg.exact = exact_values ? 1 : 0;
    for (int i = 0; i < 9; ++i) h->an.m[i] = 0.0;
    for (int i = 0; i < dim * dim; ++i) h->an.m[i] = aniso[i];
    for (int i = 0; i < 3; ++i) h->an.c[i] = i < dim ? center[i] : 0.0;
    h->hx.assign(x, x + n); h->hy.assign(y, y + n);
    if (dim == 3) h->hz.assign(z, z + n); else h->hz.assign(n, 0.0);
    h->hval.assign(values, values + n);
    if (n_hd) h->hdrift.assign(drift_data, drift_data + (size_t)n_hd * n); else h->hdrift.clear();

    // adjusted bounding box on the host (drift rescale + c0 for unbounded models)
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    (void)user_dim;
    const int sdim = h->geo ? 3 : dim;            // spatial dimensions of the device coordinates
    for (int64_t i = 0; i < n; ++i) {
        if (h->geo) {
            const double rad = 0.017453292519943295;
            double u[3] = {std::cos(x[i] * rad) * std::cos(y[i] * rad), std::sin(x[i] * rad) * std::cos(y[i] * rad),
                           std::sin(y[i] * rad)};
            for (int r = 0; r < 3; ++r) { lo[r] = std::min(lo[r], u[r]); hi[r] = std::max(hi[r], u[r]); }
            continue;
        }
        double d[3] = {x[i] - h->an.c[0], y[i] - h->an.c[1], dim == 3 ? z[i] - h->an.c[2] : 0.0};
        for (int r = 0; r < dim; ++r) {
            double v = h->an.c[r];
            for (int c = 0; c < dim; ++c) v += h->an.m[r * dim + c] * d[c];
            lo[r] = std::min(lo[r], v); hi[r] = std::max(hi[r], v);
        }
    }
    if (h->geo) for (int r = 0; r < 3; ++r) { lo[r] -= 1e-9; hi[r] += 1e-9; }   // device sincos may differ in the last ulp
    for (int r = 0; r < 3; ++r) { h->bb_lo[r] = r < sdim ? lo[r] : 0.0; h->bb_hi[r] = r < sdim ? hi[r] : 0.0; }
    double diag2 = 0.0;
    for (int r = 0; r < sdim; ++r) diag2 += (hi[r] - lo[r]) * (hi[r] - lo[r]);
    if (model == KB200_VG_TABLE && h->tab_dmax < (h->geo ? 180.0 : std::sqrt(diag2)))
        return fail(h, KB200_EBADARG, "variogram table: dmax is smaller than the extent of the data");
    double c0 = host_gamma(h, h->vg, h->geo ? 180.0 : std::sqrt(diag2));
    if (!(c0 > 0.0) || !std::isfinite(c0)) c0 = 1.0;
    h->vg.c0 = c0;
    for (int c = 0; c <= KB200_MAX_DRIFT; ++c) { h->ds.shift[c] = 0.0; h->ds.scale[c] = 1.0; }
    for (int c = 0; c < n_rl; ++c) {
        h->ds.shift[c] = 0.5 * (hi[c] + lo[c]);
        double half = 0.5 * (hi[c] - lo[c]);
        h->ds.scale[c] = half > 0.0 ? 1.0 / half : 1.0;
    }
    for (int c = 0; c < n_hd; ++c) {
        const double* col = drift_data + (size_t)c * n;
        double mean = 0.0;
        for (int64_t i = 0; i < n; ++i) mean += col[i];
        mean /= (double)n;
        double amax = 0.0;
        for (int64_t i = 0; i < n; ++i) amax = std::max(amax, std::fabs(col[i] - mean));
        h->ds.shift[n_rl + c] = mean;
        h->ds.scale[n_rl + c] = amax > 0.0 ? 1.0 / amax : 1.0;
    }

    if (h->pinv && !knn_only) {
        // pseudo-inverse of the reference's own matrix: gamma form (c0 = 0), raw drift columns (pinv.cu)
        if (dtype != KB200_F64) return fail(h, KB200_EUNSUPPORTED, "pseudo_inv=True runs in float64 only");
        if (n + h->K1 > kbk_pinv_max_nt())
            return fail(h, KB200_EUNSUPPORTED, "pseudo_inv=True supports at most " + std::to_string(kbk_pinv_max_nt() - h->K1) + " data points");
        h->vg.c0 = 0.0;
        for (int c = 0; c <= KB200_MAX_DRIFT; ++c) { h->ds.shift[c] = 0.0; h->ds.scale[c] = 1.0; }
    }

    // tile stream map
    h->n_pad = (int)align_up((size_t)n, KB_BM);
    h->ld = h->n_pad;
    h->nrb = knn_only ? 0 : (int)((n + h->na + KB_BM - 1) / KB_BM);
    int nk = (int)((n + KB_BK - 1) / KB_BK);
    h->pm.nrb = h->nrb;
    long long off = 0;
    for (int I = 0; I < h->nrb; ++I) {
        bool has_dual = (I + 1) * KB_BM > n;     // block holds rows >= n (dual rows live there)
        int kt = has_dual ? nk : std::min(nk, (I + 1) * KB_BM / KB_BK);
        h->pm.ktiles[I] = kt;
        h->pm.tile_off[I] = off;
        off += kt;
    }
    size_t esz = 8;   // fp64 value, or TF32 hi + lo pair: both 8 bytes per element
    size_t o = 0;
    o += align_up(64 * sizeof(double), 256);
    h->off_consts = o; o += align_up(512 * sizeof(double), 256);
    h->off_ax = o; o += align_up((size_t)h->n_pad * 8, 256);
    h->off_ay = o; o += align_up((size_t)h->n_pad * 8, 256);
    h->off_az = o; o += align_up((size_t)h->n_pad * 8, 256);
    h->off_tiles = o;
    // a float64 problem that may take the int8 route reserves room for both layouts: whether the Cholesky succeeds (else
    // the general path packs fp64 tiles) is known only after the factorisation, and every rank sizes the blob alike
    const int i8s = (dtype == KB200_F64) ? ((h->pinv || n > KB_F64_I8_NMAX) ? 0 : KB_F64_I8_SLICES) : h->slices;
    size_t o8 = o;
    if (i8s) {
        o8 += (size_t)kbk_i8_total_tiles(i8s, (int)n, h->na, nullptr) * kbk_i8_tile_bytes(i8s);
        o8 = align_up(o8, 256);
        h->off_rowscale = o8; o8 += align_up((size_t)kbk_i8_rows(i8s, (int)n, h->na) * sizeof(double), 256);
    }
    if (dtype == KB200_F64 || dtype == KB200_F32) o += (size_t)off * KB_BM * KB_BK * esz;
    o = std::max(o, o8);
    h->blob_bytes = knn_only ? h->off_tiles : o;
    cudaSetDevice(h->device);
    CU(h, h->blob.reserve(h->blob_bytes));
    h->described = true;
    return KB200_OK;
}

extern "C" int kb200_describe_problem(kb200_handle h, int dim, int dtype, int64_t n,
                                      const double* x, const double* y, const double* z, const double* values,
                                      const double* center, const double* aniso,
                                      int model, const double* vparams, int n_vparams,
                                      int exact_values, double eps, int n_rl, int n_hd, const double* drift_data) {
    return describe(h, false, dim, dtype, n, x, y, z, values, center, aniso, model, vparams, n_vparams,
                    exact_values, eps, n_rl, n_hd, drift_data);
}

extern "C" int64_t kb200_blob_bytes(kb200_handle h) { return (h && h->described) ? (int64_t)h->blob_bytes : 0; }
extern "C" void* kb200_blob_ptr(kb200_handle h) { return (h && h->described) ? h->blob.p : nullptr; }

// header layout (doubles): [0] magic, [1] c0, [2..18) shift, [18..34) scale, [34] gform, [35] slices
static const double KB_MAGIC = 20260922.0;

extern "C" int kb200_blob_commit(kb200_handle h) {
    if (!h || !h->described) return fail(h, KB200_ESTATE, "describe the problem first");
    cudaSetDevice(h->device);
    double hdr[64];
    CU(h, cudaMemcpyAsync(hdr, h->blob.p, sizeof(hdr), cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    if (hdr[0] != KB_MAGIC) return fail(h, KB200_ESTATE, "blob does not hold a factored problem");
    h->vg.c0 = hdr[1];
    h->gform = (int)hdr[34];
    h->slices = (int)hdr[35];        // the kernel the factoring handle packed for
    for (int c = 0; c <= KB200_MAX_DRIFT; ++c) { h->ds.shift[c] = hdr[2 + c]; h->ds.scale[c] = hdr[18 + c]; }
    h->ready = true;
    return KB200_OK;
}

static float ev_ms(cudaEvent_t a, cudaEvent_t b) { float t = 0.f; cudaEventElapsedTime(&t, a, b); return t; }

extern "C" int kb200_set_problem(kb200_handle h, int dim, int dtype, int64_t n,
                                 const double* x, const double* y, const double* z, const double* values,
                                 const double* center, const double* aniso,
                                 int model, const double* vparams, int n_vparams,
                                 int exact_values, double eps, int n_rl, int n_hd, const double* drift_data) {
    int rc = describe(h, false, dim, dtype, n, x, y, z, values, center, aniso, model, vparams, n_vparams,
                      exact_values, eps, n_rl, n_hd, drift_data);
    if (rc != KB200_OK) return rc;
    cudaStream_t st = h->stream;
    const int np = h->n_pad, ld = h->ld, nn = h->n;
    const size_t mat = (size_t)np * ld * sizeof(double);
    CU(h, h->wC.reserve(mat)); CU(h, h->wW.reserve(mat)); CU(h, h->wT.reserve(mat));
    CU(h, h->wF.reserve((size_t)3 * KB_MAXAUX * np * sizeof(double)));
    CU(h, h->wRaw.reserve((size_t)(4 + h->n_hd) * nn * sizeof(double)));
    CU(h, h->wFlag.reserve(256));
    double* raw = h->wRaw.as<double>();
    double *rx = raw, *ry = raw + nn, *rz = raw + 2 * (size_t)nn, *rv = raw + 3 * (size_t)nn, *rh = raw + 4 * (size_t)nn;
    char* blob = h->blob.as<char>();
    double* ax = reinterpret_cast<double*>(blob + h->off_ax);
    double* ay = reinterpret_cast<double*>(blob + h->off_ay);
    double* az = reinterpret_cast<double*>(blob + h->off_az);
    double* consts = reinterpret_cast<double*>(blob + h->off_consts);
    int* flag = h->wFlag.as<int>();
    int launches = 0;

    CU(h, cudaEventRecord(h->ev[0], st));
    CU(h, cudaMemcpyAsync(rx, h->hx.data(), nn * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaMemcpyAsync(ry, h->hy.data(), nn * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaMemcpyAsync(rz, h->hz.data(), nn * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaMemcpyAsync(rv, h->hval.data(), nn * 8, cudaMemcpyHostToDevice, st));
    if (h->n_hd) CU(h, cudaMemcpyAsync(rh, h->hdrift.data(), (size_t)h->n_hd * nn * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaMemsetAsync(ax, 0, (size_t)np * 8, st));
    CU(h, cudaMemsetAsync(ay, 0, (size_t)np * 8, st));
    CU(h, cudaMemsetAsync(az, 0, (size_t)np * 8, st));
    CU(h, kbk_adjust_data(h->dim, h->an, nn, rx, ry, rz, ax, ay, az, st)); ++launches;
    CU(h, cudaEventRecord(h->ev[1], st));

    // covariance shift: c0 = sill for bounded models; for linear/power grow c0 until C is
    // positive definite (DESIGN.md §3). A model that is not a valid variogram in this
    // dimension (e.g. hole-effect in 2-D/3-D) never becomes positive definite.
    const bool unbounded = (h->vg.model == KB200_VG_LINEAR || h->vg.model == KB200_VG_POWER || h->vg.model == KB200_VG_TABLE);
    const int max_try = unbounded ? 5 : 1;
    const double c0_first = h->vg.c0;
    int hflag = 0;
    float t_asm = 0.f, t_chol = 0.f;
    for (int attempt = 0; attempt < max_try; ++attempt) {
        CU(h, cudaMemsetAsync(flag, 0, sizeof(int), st));
        CU(h, cudaEventRecord(h->ev[2], st));
        CU(h, kbk_assemble(h->dim, h->vg, nn, np, ld, ax, ay, az, h->wC.as<double>(), st)); ++launches;
        CU(h, cudaEventRecord(h->ev[3], st));
        if (h->pinv) {                                  // no factorisation: the pseudo-inverse works on -Gamma itself
            CU(h, cudaEventRecord(h->ev[4], st));
            CU(h, cudaStreamSynchronize(st));
            t_asm += ev_ms(h->ev[2], h->ev[3]);
            break;
        }
        {
            if (!h->hi_stream) {
                int lo = 0, hi = 0;
                CU(h, cudaDeviceGetStreamPriorityRange(&lo, &hi));
                CU(h, cudaStreamCreateWithPriority(&h->hi_stream, cudaStreamNonBlocking, hi));
            }
            const size_t need = 2 * (size_t)((np / 64 + 3) / 4) + 1;
            while (h->fev.size() < need) {
                cudaEvent_t e;
                CU(h, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                h->fev.push_back(e);
            }
        }
        CU(h, kbk_cholesky(h->wC.as<double>(), h->wW.as<double>(), h->wT.as<double>(), ld, np, flag, 3.6e-15 * h->vg.c0, st, h->hi_stream,
                           h->fev.data(), (int)h->fev.size(), &launches));
        CU(h, cudaEventRecord(h->ev[4], st));
        CU(h, cudaMemcpyAsync(&hflag, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(h, cudaStreamSynchronize(st));
        t_asm += ev_ms(h->ev[2], h->ev[3]); t_chol += ev_ms(h->ev[3], h->ev[4]);
        if (hflag != 0 && std::getenv("KB200_DEBUG")) std::fprintf(stderr, "[kb200] cholesky flag %d (attempt %d, c0 %g)\n", hflag, attempt, h->vg.c0);
        if (hflag == 0) break;
        h->vg.c0 *= 2.0;
    }
    h->gform = 0;
    double* Fz = h->wF.as<double>();
    double* Hz = Fz + (size_t)KB_MAXAUX * np;
    double* Uz = Hz + (size_t)KB_MAXAUX * np;
    CU(h, cudaMemsetAsync(consts, 0, 512 * sizeof(double), st));
    if (h->pinv) {
        // pseudo_inv=True: A^+ of the bordered gamma-form matrix (pinv.cu), then the quadratic-form solve
        const int nt = nn + h->K1;
        CU(h, h->wVario.reserve(kbk_pinv_workspace_doubles(nt) * sizeof(double)));
        CU(h, cudaEventRecord(h->ev[4], st));
        CU(h, kbk_build_fz(nn, np, h->n_rl, h->n_hd, ax, ay, az, h->ds, rh, rv, Fz, st)); ++launches;
        CU(h, kbk_pinv(nn, h->K1, np, h->wC.as<double>(), ld, Fz, rv, Uz, consts, h->wVario.as<double>(), flag, st,
                       &launches, &h->pinv_sweeps, &h->pinv_rank));
        if (h->pinv_sweeps < 0) { h->launches += launches; return fail(h, KB200_ESINGULAR, "pseudo-inverse: the Jacobi SVD did not converge"); }
        CU(h, cudaMemsetAsync(flag, 0, sizeof(int), st));
        CU(h, cudaEventRecord(h->ev[5], st));
        CU(h, kbk_pack_gform(h->wC.as<double>(), ld, nn, np, h->na, Uz, h->pm, blob + h->off_tiles, st)); ++launches;
        h->gform = 2;
    } else if (hflag != 0) {
        // C is not positive definite: the variogram is not conditionally negative definite in this
        // dimension (e.g. hole-effect on dense scatter). General fallback: blocked Gauss-Jordan inverse with
        // partial pivoting + quadratic-form solve (DESIGN.md §3b). fp64 only.
        if (h->dtype != KB200_F64) {
            h->launches += launches;
            return fail(h, KB200_EUNSUPPORTED, "dtype float32 / float64x need a positive definite covariance form "
                        "(the variogram is not valid in this dimension); use float64");
        }
        h->vg.c0 = c0_first;
        h->slices = 0;                                  // fp64 quadratic-form tiles, DMMA kernel
        CU(h, cudaMemsetAsync(flag, 0, sizeof(int), st));
        CU(h, cudaEventRecord(h->ev[3], st));
        CU(h, kbk_assemble(h->dim, h->vg, nn, np, ld, ax, ay, az, h->wC.as<double>(), st)); ++launches;
        CU(h, h->wVario.reserve(kbk_general_inverse_workspace_bytes(np)));
        const char* gj_env = std::getenv("KB200_GJ");            // "blocked" | "scalar": cross-check switch of the tests
        const bool gj_scalar = gj_env ? gj_env[0] == 's' : !KB_GJ_DEFAULT_BLOCKED;
        CU(h, kbk_general_inverse(h->wC.as<double>(), ld, nn, np, h->wVario.p, flag, 3.6e-15 * h->vg.c0, st, &launches,
                                  gj_scalar));
        CU(h, cudaEventRecord(h->ev[4], st));
        CU(h, cudaMemcpyAsync(&hflag, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(h, cudaStreamSynchronize(st));
        t_chol += ev_ms(h->ev[3], h->ev[4]);
        if (hflag != 0) {
            h->launches += launches;
            return fail(h, KB200_ESINGULAR, "kriging matrix is singular (zero pivot in column " +
                        std::to_string(hflag - 1) + ")");
        }
        h->gform = 1;
        CU(h, cudaEventRecord(h->ev[5], st));
        CU(h, kbk_dual_gform(h->wC.as<double>(), ld, nn, np, h->n_rl, h->n_hd, ax, ay, az, h->ds, rh, rv,
                             Fz, Uz, consts, flag, st, &launches));
        CU(h, kbk_pack_gform(h->wC.as<double>(), ld, nn, np, h->na, Uz, h->pm, blob + h->off_tiles, st)); ++launches;
    } else {
    CU(h, kbk_trtri(h->wC.as<double>(), h->wW.as<double>(), h->wT.as<double>(), ld, np, st, &launches));
    CU(h, cudaEventRecord(h->ev[5], st));
    CU(h, kbk_dual(h->wW.as<double>(), ld, nn, np, h->n_rl, h->n_hd, ax, ay, az, h->ds, rh, rv,
                   Fz, Hz, Uz, consts, flag, st, &launches));
    if (h->dtype == KB200_F32) {
        CU(h, kbk_pack_tf32(h->wW.as<double>(), ld, nn, np, h->na, Uz, h->pm, blob + h->off_tiles, st));
    } else if (h->slices) {
        const int nrb8 = kbk_i8_nrb(h->slices, nn, h->na);
        std::vector<long long> toff(nrb8 + 1);
        kbk_i8_total_tiles(h->slices, nn, h->na, toff.data());
        // workspace (T1 scratch is free now): tile offsets | row exponents
        long long* d_toff = reinterpret_cast<long long*>(h->wT.as<char>());
        int* d_rowexp = reinterpret_cast<int*>(h->wT.as<char>() + align_up((size_t)(nrb8 + 1) * sizeof(long long), 256));   // kbk_i8_rows ints
        CU(h, cudaMemcpyAsync(d_toff, toff.data(), (size_t)(nrb8 + 1) * sizeof(long long), cudaMemcpyHostToDevice, st));
        CU(h, kbk_pack_i8(h->slices, h->wW.as<double>(), ld, nn, np, h->na, Uz, d_rowexp,
                          reinterpret_cast<double*>(blob + h->off_rowscale), d_toff, blob + h->off_tiles, st));
        CU(h, cudaStreamSynchronize(st));      // toff is a host temporary
        ++launches;
    } else {
        CU(h, kbk_pack(h->dtype, h->wW.as<double>(), ld, nn, np, h->na, Uz, h->pm, blob + h->off_tiles, st));
    }
    ++launches;
    }
    double hdr[64] = {0};
    hdr[0] = KB_MAGIC; hdr[1] = h->vg.c0; hdr[34] = (double)h->gform; hdr[35] = (double)h->slices;
    for (int c = 0; c <= KB200_MAX_DRIFT; ++c) { hdr[2 + c] = h->ds.shift[c]; hdr[18 + c] = h->ds.scale[c]; }
    CU(h, cudaMemcpyAsync(blob, hdr, sizeof(hdr), cudaMemcpyHostToDevice, st));
    CU(h, cudaEventRecord(h->ev[6], st));
    CU(h, cudaMemcpyAsync(&hflag, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(h, cudaStreamSynchronize(st));
    h->tm[6] += ev_ms(h->ev[0], h->ev[1]);
    h->tm[0] += t_asm; h->tm[1] += t_chol;
    h->tm[2] += ev_ms(h->ev[4], h->ev[5]);
    h->tm[3] += ev_ms(h->ev[5], h->ev[6]);
    h->launches += launches;
    if (hflag != 0) return fail(h, KB200_ESINGULAR, "drift/unbiasedness block F^T C^-1 F is singular");
    h->ready = true;
    h->factor_live = !h->gform;
    return KB200_OK;
}

// ---- device-evaluated drift terms -----------------------------------------------------------------------
extern "C" int kb200_set_device_drift(kb200_handle h, int n_wells, const double* wells,
                                      int64_t ext_nx, int64_t ext_ny, const double* ext_x, const double* ext_y,
                                      const double* ext_z) {
    if (!h) return KB200_EBADARG;
    if (n_wells < 0 || n_wells > KB200_MAX_DRIFT || (n_wells > 0 && !wells))
        return fail(h, KB200_EBADARG, "device drift: bad point_log description");
    const bool ext = ext_nx > 0 || ext_ny > 0;
    if (ext && (ext_nx < 1 || ext_ny < 1 || ext_nx > (1 << 30) || ext_ny > (1 << 30) || !ext_x || !ext_y || !ext_z))
        return fail(h, KB200_EBADARG, "device drift: bad external_Z raster description");
    h->described = false; h->ready = false; h->factor_live = false;
    cudaSetDevice(h->device);
    h->dd = DeviceDrift{};
    if (n_wells) {
        CU(h, h->wWells.reserve((size_t)3 * n_wells * 8));
        CU(h, cudaMemcpyAsync(h->wWells.p, wells, (size_t)3 * n_wells * 8, cudaMemcpyHostToDevice, h->stream));
        h->dd.n_wells = n_wells; h->dd.wells = h->wWells.as<double>();
    }
    if (ext) {
        const size_t nx = (size_t)ext_nx, ny = (size_t)ext_ny;
        CU(h, h->wExt.reserve((nx + ny + nx * ny) * 8));
        double* d = h->wExt.as<double>();
        CU(h, cudaMemcpyAsync(d, ext_x, nx * 8, cudaMemcpyHostToDevice, h->stream));
        CU(h, cudaMemcpyAsync(d + nx, ext_y, ny * 8, cudaMemcpyHostToDevice, h->stream));
        CU(h, cudaMemcpyAsync(d + nx + ny, ext_z, nx * ny * 8, cudaMemcpyHostToDevice, h->stream));
        bool sorted = true;
        for (size_t i = 1; i < nx && sorted; ++i) sorted = ext_x[i] >= ext_x[i - 1];
        for (size_t i = 1; i < ny && sorted; ++i) sorted = ext_y[i] >= ext_y[i - 1];
        h->dd.ext = 1; h->dd.ext_nx = (int)ext_nx; h->dd.ext_ny = (int)ext_ny; h->dd.ext_sorted = sorted ? 1 : 0;
        h->dd.ext_x = d; h->dd.ext_y = d + nx; h->dd.ext_z = d + nx + ny;
    }
    CU(h, cudaStreamSynchronize(h->stream));     // the caller's arrays may go away
    return KB200_OK;
}

// ---- execute --------------------------------------------------------------
// One persistent launch of the solve kernel of the handle's dtype over points [s.first, s.first + s.count).
// NOTE: one kernel for every point count: the summation order per point must not depend on how the points are
// sharded or chunked (concatenated shards == single call, bit for bit; SURVEY.md §4 (iii)).
// One persistent launch of the solve kernel of the handle's dtype over points [s.first, s.first + s.count) with point
// tiles of `tp` points.
static int launch_solve(kb200_ctx* h, const Src& s, double* d_z, double* d_ss, int tp) {
    cudaStream_t st = h->stream;
    char* blob = h->blob.as<char>();
    PointSource ps{};
    ps.grid = s.grid ? 1 : 0;
    ps.px = s.a; ps.py = s.b; ps.pz = s.c; ps.gx = s.a; ps.gy = s.b; ps.gz = s.c;
    ps.nx = s.nx; ps.ny = s.ny; ps.nz = s.nz;
    const bool i8 = h->slices != 0;
    const bool f32 = h->dtype == KB200_F32;
    long long ntiles = (s.count + tp - 1) / tp;
    int grid = (int)std::min<long long>(ntiles, h->num_sms);
    CU(h, h->wScratch.reserve(i8 ? kbk_solve_i8_scratch_bytes(h->slices, h->n, grid) : f32 ? kbk_solve_tf32_scratch_bytes(h->n, grid)
                                  : kbk_solve_pt_scratch_doubles(h->n, grid) * sizeof(double)));
    SolvePtParams pp{};
    pp.vg = h->vg; pp.an = h->an; ps.first = s.first; pp.ps = ps;
    pp.n = h->n; pp.na = h->na; pp.nrb = h->nrb; pp.n_rl = h->n_rl; pp.n_hd = h->n_hd;
    pp.ax = reinterpret_cast<double*>(blob + h->off_ax);
    pp.ay = reinterpret_cast<double*>(blob + h->off_ay);
    pp.az = reinterpret_cast<double*>(blob + h->off_az);
    pp.tiles = blob + h->off_tiles; pp.pm = h->pm; pp.ds = h->ds;
    pp.consts = reinterpret_cast<double*>(blob + h->off_consts);
    pp.dd = h->dd; pp.n_dev = h->n_dev;
    pp.drift_pts = s.d_drift; pp.drift_stride = s.drift_stride; pp.drift_first = s.drift_first;
    pp.m = s.count; pp.scratch = h->wScratch.as<double>(); pp.gform = h->gform;
    pp.z_out = d_z; pp.ss_out = d_ss;
    pp.rowscale = reinterpret_cast<const double*>(blob + h->off_rowscale);
    if (i8) CU(h, kbk_solve_i8(h->slices, h->dim, pp, grid, st));
    else if (f32) CU(h, kbk_solve_tf32(h->dim, pp, grid, st));
    else CU(h, kbk_solve_pt(h->dim, pp, grid, tp, st));
    h->launches += 1; h->solve_launches += 1;
    return KB200_OK;
}

// Relative cost of one round of the fp64 kernel with 64 / 32 / 16-point tiles (a tile streams all of W once whatever its
// width; the DMMA work is proportional to the width). Measured at N=5000 (profiles/r02/tile_width_timing_*.log).
static double tile_cost(int tp) { return tp == 64 ? 1.0 : (tp == 32 ? KB_TILE_COST_32 : KB_TILE_COST_16); }

// NOTE: the summation order per point does not depend on the tile width, on how the points are sharded or chunked, or on
// the number of launches (concatenated shards == single call, bit for bit; SURVEY.md §4 (iii)).
static int run_solve(kb200_ctx* h, const Src& s, double* d_z, double* d_ss) {
    const bool i8 = h->slices != 0;
    const bool f32 = h->dtype == KB200_F32;
    if (i8 || f32) return launch_solve(h, s, d_z, d_ss, i8 ? kbk_solve_i8_tile_points() : kbk_solve_tf32_tile_points());
    // fp64 DMMA kernel: full rounds of 64-point tiles over all SMs, then the leftover points as ONE more launch whose tile
    // width minimises rounds x cost: a partial round of 64-point tiles keeps a few SMs busy for a whole tile time
    const long long S = h->num_sms;
    if (const char* e = std::getenv("KB200_TILE")) {           // profiling override: one launch, fixed width
        const int t = std::atoi(e);
        if (t == 64 || t == 32 || t == 16) return launch_solve(h, s, d_z, d_ss, t);
    }
    const long long nt64 = (s.count + KB_TN - 1) / KB_TN;
    const long long main_pts = std::min<long long>(s.count, (nt64 / S) * S * KB_TN);
    const long long rem = s.count - main_pts;
    if (main_pts > 0) {
        Src m = s; m.count = main_pts;
        int rc = launch_solve(h, m, d_z, d_ss, KB_TN); if (rc) return rc;
    }
    if (rem > 0) {
        int best = KB_TN; double bc = 1e300;
        for (int tp : {64, 32, 16}) {
            const long long nt = (rem + tp - 1) / tp;
            const double c = (double)((nt + S - 1) / S) * tile_cost(tp);
            if (c < bc * 0.999) { bc = c; best = tp; }
        }
        Src t = s; t.first = s.first + main_pts; t.count = rem; t.drift_first = s.drift_first + main_pts;
        int rc = launch_solve(h, t, d_z + main_pts, d_ss + main_pts, best); if (rc) return rc;
    }
    return KB200_OK;
}

static int run_knn(kb200_ctx* h, int k, const Src& s, double* d_z, double* d_ss, int chol);

// Launch `total` points in chunks and bring (z, ss) to the caller's HOST buffers. Large outputs travel through two
// pinned staging buffers on a second stream while the next chunk computes; the host drains a buffer into the
// caller's (pageable) memory while the GPU works. launch(o, m, d_z, d_ss) enqueues points [o, o+m) of the call.
template <class Launch>
static int run_to_host(kb200_ctx* h, int64_t total, double* z_out, double* ss_out, Launch launch) {
    cudaStream_t st = h->stream;
    CU(h, h->wOut.reserve((size_t)2 * total * 8));
    double* dz = h->wOut.as<double>();
    double* dss = dz + total;
    CU(h, cudaEventRecord(h->ev[7], st));
    if (total < KB_STAGE_MIN) {
        int rc = launch((int64_t)0, total, dz, dss); if (rc) return rc;
        CU(h, cudaEventRecord(h->ev[8], st));
        CU(h, cudaMemcpyAsync(z_out, dz, total * 8, cudaMemcpyDeviceToHost, st));
        CU(h, cudaMemcpyAsync(ss_out, dss, total * 8, cudaMemcpyDeviceToHost, st));
        CU(h, cudaEventRecord(h->ev[11], st));
        CU(h, cudaStreamSynchronize(st));
        h->tm[7] += ev_ms(h->ev[8], h->ev[11]);
        return KB200_OK;
    }
    if (!h->copy_stream) {
        CU(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            CU(h, cudaHostAlloc(&h->pin[i], (size_t)2 * KB_STAGE_PTS * 8, cudaHostAllocDefault));
            CU(h, cudaEventCreateWithFlags(&h->evk[i], cudaEventDisableTiming));
            CU(h, cudaEventCreate(&h->evc[i]));
        }
    }
    const int64_t nch = (total + KB_STAGE_PTS - 1) / KB_STAGE_PTS;
    auto chunk_len = [&](int64_t c) { return std::min<int64_t>(KB_STAGE_PTS, total - c * KB_STAGE_PTS); };
    auto drain = [&](int64_t c) -> int {          // staged chunk c -> the caller's buffers
        const int b = (int)(c & 1);
        CU(h, cudaEventSynchronize(h->evc[b]));
        const double* p = reinterpret_cast<const double*>(h->pin[b]);
        const int64_t m = chunk_len(c);
        std::memcpy(z_out + c * KB_STAGE_PTS, p, (size_t)m * 8);
        std::memcpy(ss_out + c * KB_STAGE_PTS, p + KB_STAGE_PTS, (size_t)m * 8);
        return KB200_OK;
    };
    for (int64_t c = 0; c < nch; ++c) {
        const int b = (int)(c & 1);
        const int64_t o = c * KB_STAGE_PTS, m = chunk_len(c);
        int rc = launch(o, m, dz + o, dss + o); if (rc) return rc;
        CU(h, cudaEventRecord(h->evk[b], st));
        if (c == nch - 1) CU(h, cudaEventRecord(h->ev[8], st));
        if (c >= 2) { rc = drain(c - 2); if (rc) return rc; }
        double* p = reinterpret_cast<double*>(h->pin[b]);
        CU(h, cudaStreamWaitEvent(h->copy_stream, h->evk[b], 0));
        CU(h, cudaMemcpyAsync(p, dz + o, (size_t)m * 8, cudaMemcpyDeviceToHost, h->copy_stream));
        CU(h, cudaMemcpyAsync(p + KB_STAGE_PTS, dss + o, (size_t)m * 8, cudaMemcpyDeviceToHost, h->copy_stream));
        CU(h, cudaEventRecord(h->evc[b], h->copy_stream));
    }
    for (int64_t c = std::max<int64_t>(0, nch - 2); c < nch; ++c) { int rc = drain(c); if (rc) return rc; }
    CU(h, cudaStreamSynchronize(st));
    h->tm[7] += ev_ms(h->ev[8], h->evc[(nch - 1) & 1]);
    return KB200_OK;
}

static int check_ready(kb200_ctx* h) {
    if (!h) return KB200_EBADARG;
    if (!h->ready) return fail(h, KB200_ESTATE, "no factored problem: call kb200_set_problem (or blob_commit) first");
    cudaSetDevice(h->device);
    return KB200_OK;
}
static int n_host_drift(const kb200_ctx* h) { return h->n_hd - h->n_dev; }

extern "C" int kb200_execute_points_dev(kb200_handle h, int64_t m,
                                        const double* d_px, const double* d_py, const double* d_pz,
                                        const double* d_drift_pts, double* d_z, double* d_ss) {
    int rc = check_ready(h); if (rc) return rc;
    if (m <= 0) return KB200_OK;
    if (!d_px || !d_py || (h->dim == 3 && !d_pz) || !d_z || !d_ss) return fail(h, KB200_EBADARG, "null pointer");
    if (n_host_drift(h) && !d_drift_pts) return fail(h, KB200_EBADARG, "drift values at the points are required");
    Src s{false, 0, 0, 0, d_px, d_py, d_pz, 0, m, d_drift_pts, m, 0};
    CU(h, cudaEventRecord(h->ev[7], h->stream));
    rc = run_solve(h, s, d_z, d_ss); if (rc) return rc;
    CU(h, cudaEventRecord(h->ev[8], h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    h->tm[4] += ev_ms(h->ev[7], h->ev[8]);
    return KB200_OK;
}

static int check_grid(kb200_ctx* h, int64_t nx, int64_t ny, int64_t nz, int64_t first, int64_t count) {
    if (nx < 1 || ny < 1 || nz < 1 || first < 0 || count < 0 || first + count > nx * ny * nz)
        return fail(h, KB200_EBADARG, "bad grid slice");
    if (h->dim != 3 && nz != 1) return fail(h, KB200_EBADARG, "nz must be 1 for 2-D");
    return KB200_OK;
}

extern "C" int kb200_execute_grid_dev(kb200_handle h, int64_t nx, int64_t ny, int64_t nz,
                                      const double* d_gx, const double* d_gy, const double* d_gz,
                                      const double* d_drift_pts, int64_t first, int64_t count,
                                      double* d_z, double* d_ss) {
    int rc = check_ready(h); if (rc) return rc;
    rc = check_grid(h, nx, ny, nz, first, count); if (rc) return rc;
    if (count == 0) return KB200_OK;
    if (!d_gx || !d_gy || (h->dim == 3 && !d_gz) || !d_z || !d_ss) return fail(h, KB200_EBADARG, "null pointer");
    if (n_host_drift(h) && !d_drift_pts) return fail(h, KB200_EBADARG, "drift values at the points are required");
    Src s{true, nx, ny, nz, d_gx, d_gy, d_gz, first, count, d_drift_pts, count, 0};
    CU(h, cudaEventRecord(h->ev[7], h->stream));
    rc = run_solve(h, s, d_z, d_ss); if (rc) return rc;
    CU(h, cudaEventRecord(h->ev[8], h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    h->tm[4] += ev_ms(h->ev[7], h->ev[8]);
    return KB200_OK;
}

// host drift columns [n_host][stride] -> device columns [n_host][m] holding items [off, off + m) of each column
static int upload_drift(kb200_ctx* h, const double* drift_pts, int64_t stride, int64_t off, int64_t m, const double** dd) {
    *dd = nullptr;
    const int nh = n_host_drift(h);
    if (!nh) return KB200_OK;
    CU(h, h->wDrift.reserve((size_t)nh * m * 8));
    for (int c = 0; c < nh; ++c)
        CU(h, cudaMemcpyAsync(h->wDrift.as<double>() + (size_t)c * m, drift_pts + (size_t)c * stride + off, (size_t)m * 8,
                              cudaMemcpyHostToDevice, h->stream));
    *dd = h->wDrift.as<double>();
    return KB200_OK;
}

// points [off, off + m) of the caller's arrays (drift columns have `stride` items each)
static int exec_points_impl(kb200_ctx* h, int64_t off, int64_t m, const double* px, const double* py, const double* pz,
                            const double* drift_pts, int64_t stride, double* z_out, double* ss_out) {
    int rc = check_ready(h); if (rc) return rc;
    if (m <= 0) return KB200_OK;
    if (!px || !py || (h->dim == 3 && !pz) || !z_out || !ss_out) return fail(h, KB200_EBADARG, "null pointer");
    if (n_host_drift(h) && !drift_pts) return fail(h, KB200_EBADARG, "drift values at the points are required");
    cudaStream_t st = h->stream;
    CU(h, h->wPts.reserve((size_t)3 * m * 8));
    double* dp = h->wPts.as<double>();
    CU(h, cudaEventRecord(h->ev[9], st));
    CU(h, cudaMemcpyAsync(dp, px + off, m * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaMemcpyAsync(dp + m, py + off, m * 8, cudaMemcpyHostToDevice, st));
    if (h->dim == 3) CU(h, cudaMemcpyAsync(dp + 2 * m, pz + off, m * 8, cudaMemcpyHostToDevice, st));
    const double* dd = nullptr;
    rc = upload_drift(h, drift_pts, stride, off, m, &dd); if (rc) return rc;
    CU(h, cudaEventRecord(h->ev[10], st));
    rc = run_to_host(h, m, z_out + off, ss_out + off, [&](int64_t o, int64_t c, double* dz, double* dss) {
        Src s{false, 0, 0, 0, dp, dp + m, dp + 2 * m, o, c, dd, m, o};
        return run_solve(h, s, dz, dss);
    });
    if (rc) return rc;
    h->tm[6] += ev_ms(h->ev[9], h->ev[10]);
    h->tm[4] += ev_ms(h->ev[7], h->ev[8]);
    return KB200_OK;
}

extern "C" int kb200_execute_points(kb200_handle h, int64_t m,
                                    const double* px, const double* py, const double* pz,
                                    const double* drift_pts, double* z_out, double* ss_out) {
    if (!h) return KB200_EBADARG;
    return exec_points_impl(h, 0, m, px, py, pz, drift_pts, m, z_out, ss_out);
}

// grid points [first, first + count); drift columns cover the caller's slice [cfirst, cfirst + ccount) and
// z_out / ss_out are indexed relative to cfirst
static int exec_grid_impl(kb200_ctx* h, int64_t nx, int64_t ny, int64_t nz,
                          const double* gx, const double* gy, const double* gz,
                          const double* drift_pts, int64_t cfirst, int64_t ccount, int64_t first, int64_t count,
                          double* z_out, double* ss_out) {
    int rc = check_ready(h); if (rc) return rc;
    rc = check_grid(h, nx, ny, nz, first, count); if (rc) return rc;
    if (count == 0) return KB200_OK;
    if (!gx || !gy || (h->dim == 3 && !gz) || !z_out || !ss_out) return fail(h, KB200_EBADARG, "null pointer");
    if (n_host_drift(h) && !drift_pts) return fail(h, KB200_EBADARG, "drift values at the points are required");
    cudaStream_t st = h->stream;
    CU(h, h->wAxes.reserve((size_t)(nx + ny + nz) * 8));
    double* da = h->wAxes.as<double>();
    CU(h, cudaEventRecord(h->ev[9], st));
    CU(h, cudaMemcpyAsync(da, gx, nx * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaMemcpyAsync(da + nx, gy, ny * 8, cudaMemcpyHostToDevice, st));
    if (h->dim == 3) CU(h, cudaMemcpyAsync(da + nx + ny, gz, nz * 8, cudaMemcpyHostToDevice, st));
    const double* dd = nullptr;
    rc = upload_drift(h, drift_pts, ccount, first - cfirst, count, &dd); if (rc) return rc;
    CU(h, cudaEventRecord(h->ev[10], st));
    rc = run_to_host(h, count, z_out + (first - cfirst), ss_out + (first - cfirst),
                     [&](int64_t o, int64_t c, double* dz, double* dss) {
        Src s{true, nx, ny, nz, da, da + nx, da + nx + ny, first + o, c, dd, count, o};
        return run_solve(h, s, dz, dss);
    });
    if (rc) return rc;
    h->tm[6] += ev_ms(h->ev[9], h->ev[10]);
    h->tm[4] += ev_ms(h->ev[7], h->ev[8]);
    return KB200_OK;
}

extern "C" int kb200_execute_grid(kb200_handle h, int64_t nx, int64_t ny, int64_t nz,
                                  const double* gx, const double* gy, const double* gz,
                                  const double* drift_pts, int64_t first, int64_t count,
                                  double* z_out, double* ss_out) {
    if (!h) return KB200_EBADARG;
    return exec_grid_impl(h, nx, ny, nz, gx, gy, gz, drift_pts, first, count, first, count, z_out, ss_out);
}

// ---- moving window ----------------------------------------------------------
extern "C" int kb200_set_problem_knn(kb200_handle h, int dim, int64_t n,
                                     const double* x, const double* y, const double* z, const double* values,
                                     const double* center, const double* aniso,
                                     int model, const double* vparams, int n_vparams, int exact_values, double eps) {
    int rc = describe(h, true, dim, KB200_F64, n, x, y, z, values, center, aniso, model, vparams, n_vparams,
                      exact_values, eps, 0, 0, nullptr);
    if (rc != KB200_OK) return rc;
    cudaStream_t st = h->stream;
    const int nn = h->n, np = h->n_pad;
    CU(h, h->wRaw.reserve((size_t)4 * nn * sizeof(double)));
    double* raw = h->wRaw.as<double>();
    double *rx = raw, *ry = raw + nn, *rz = raw + 2 * (size_t)nn, *rv = raw + 3 * (size_t)nn;
    char* blob = h->blob.as<char>();
    double* ax = reinterpret_cast<double*>(blob + h->off_ax);
    double* ay = reinterpret_cast<double*>(blob + h->off_ay);
    double* az = reinterpret_cast<double*>(blob + h->off_az);
    int launches = 0;
    CU(h, cudaEventRecord(h->ev[0], st));
    CU(h, cudaMemcpyAsync(rx, h->hx.data(), nn * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaMemcpyAsync(ry, h->hy.data(), nn * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaMemcpyAsync(rz, h->hz.data(), nn * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaMemcpyAsync(rv, h->hval.data(), nn * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaMemsetAsync(ax, 0, (size_t)np * 8, st));
    CU(h, cudaMemsetAsync(ay, 0, (size_t)np * 8, st));
    CU(h, cudaMemsetAsync(az, 0, (size_t)np * 8, st));
    CU(h, kbk_adjust_data(h->dim, h->an, nn, rx, ry, rz, ax, ay, az, st)); ++launches;
    CU(h, cudaEventRecord(h->ev[1], st));
    // uniform cell grid with ~2 points per cell over the adjusted bounding box
    KnnParams& kp = h->kp;
    kp = KnnParams{};
    double ext[3] = {0, 0, 0}, vol = 1.0; int live = 0;
    const int sdim = h->dim == KB_GEO ? 3 : h->dim;
    for (int r = 0; r < sdim; ++r) { ext[r] = h->bb_hi[r] - h->bb_lo[r]; if (ext[r] > 0.0) { vol *= ext[r]; ++live; } }
    double cell = live ? std::pow(vol * 2.0 / (double)nn, 1.0 / live) : 1.0;
    if (!(cell > 0.0) || !std::isfinite(cell)) cell = 1.0;
    int g[3] = {1, 1, 1};
    for (;;) {
        long long tot = 1;
        for (int r = 0; r < sdim; ++r) {
            double cnt = std::floor(ext[r] / cell) + 1.0;
            g[r] = (int)std::min(cnt, 4096.0);
            tot *= g[r];
        }
        if (tot <= (1LL << 22)) break;
        cell *= 1.5;
    }
    // a cell edge slightly larger than ext/g keeps every data point inside the grid after clamping
    for (int r = 0; r < sdim; ++r) if (g[r] == 4096) cell = std::max(cell, ext[r] / 4095.0);
    kp.dim = h->dim; kp.n = nn; kp.gx = g[0]; kp.gy = g[1]; kp.gz = g[2];
    kp.ox = h->bb_lo[0]; kp.oy = h->bb_lo[1]; kp.oz = h->bb_lo[2];
    kp.cell = cell; kp.inv_cell = 1.0 / cell;
    int ncells = g[0] * g[1] * g[2];
    h->k_ncells = ncells;
    CU(h, h->kSorted.reserve((size_t)nn * (4 * sizeof(double) + 2 * sizeof(int))));
    CU(h, h->kCells.reserve((size_t)2 * (ncells + 1) * sizeof(int)));
    CU(h, h->wFlag.reserve(256));
    double* sx = h->kSorted.as<double>();
    double *sy = sx + nn, *sz = sy + nn, *sv = sz + nn;
    int* sorig = reinterpret_cast<int*>(sv + nn);
    int* cell_of = sorig + nn;
    int* cell_start = h->kCells.as<int>();
    int* cursor = cell_start + (ncells + 1);
    CU(h, kbk_knn_build(h->dim, nn, ax, ay, az, rv, kp, sx, sy, sz, sv, sorig, cell_of, cell_start, cursor,
                        ncells, st, &launches));
    CU(h, cudaEventRecord(h->ev[2], st));
    CU(h, cudaStreamSynchronize(st));
    h->tm[6] += ev_ms(h->ev[0], h->ev[1]);
    h->tm[8] += ev_ms(h->ev[1], h->ev[2]);
    h->launches += launches;
    h->knn_ready = true;
    return KB200_OK;
}


// ---- moving window: execute ---------------------------------------------------------------------------------
static int run_knn(kb200_ctx* h, int k, const Src& s, double* d_z, double* d_ss, int chol) {
    cudaStream_t st = h->stream;
    KnnParams kp = h->kp;
    kp.vg = h->vg; kp.an = h->an; kp.k = k;
    {   // radius (in cells) of the ball expected to hold k points at the mean density
        double ppc = (double)h->n / (double)std::max(1, h->k_ncells);
        int live = 0;
        if (kp.gx > 1) ++live; if (kp.gy > 1) ++live; if (kp.gz > 1) ++live;
        double cells = (double)k / std::max(ppc, 1e-9);
        double R = live >= 3 ? std::cbrt(cells * 3.0 / (4.0 * 3.14159265358979)) : (live == 2 ? std::sqrt(cells / 3.14159265358979) : 0.5 * cells);
        kp.r0 = (int)std::min(64.0, std::max(1.0, std::ceil(R)));
    }
    PointSource ps{};
    ps.grid = s.grid ? 1 : 0;
    ps.px = s.a; ps.py = s.b; ps.pz = s.c; ps.gx = s.a; ps.gy = s.b; ps.gz = s.c;
    ps.nx = s.nx; ps.ny = s.ny; ps.nz = s.nz; ps.first = s.first;
    kp.ps = ps; kp.m = s.count; kp.z_out = d_z; kp.ss_out = d_ss; kp.flag = h->wFlag.as<int>();
    CU(h, kbk_knn_solve(kp, chol, st));
    h->launches += 1; h->solve_launches += 1;
    return KB200_OK;
}

static int check_knn(kb200_ctx* h, int k) {
    if (!h) return KB200_EBADARG;
    if (!h->knn_ready) return fail(h, KB200_ESTATE, "call kb200_set_problem_knn first");
    cudaSetDevice(h->device);
    if (k < 2) return fail(h, KB200_EBADARG, "n_closest_points has to be at least two!");
    if (k > h->n) return fail(h, KB200_EBADARG, "n_closest_points exceeds the number of data points");
    if (kbk_knn_smem_per_warp(k, 0, 1) > 200 * 1024) return fail(h, KB200_EUNSUPPORTED, "n_closest_points too large for the shared-memory local solver");
    return KB200_OK;
}

// Run the moving window to HOST buffers and handle the solver flag: 2 = a local covariance block was not positive
// definite (variogram not valid in this dimension) -> repeat with the pivoted-LU solver (dgesv semantics);
// 1 = exactly singular local system -> ValueError('Singular matrix') (cok.pyx:176-179).
template <class MakeSrc>
static int knn_to_host(kb200_ctx* h, int k, int64_t total, double* z_out, double* ss_out, MakeSrc make_src) {
    int* flag = h->wFlag.as<int>();
    for (int chol = 1; chol >= 0; --chol) {
        CU(h, cudaMemsetAsync(flag, 0, sizeof(int), h->stream));
        int rc = run_to_host(h, total, z_out, ss_out, [&](int64_t o, int64_t c, double* dz, double* dss) {
            return run_knn(h, k, make_src(o, c), dz, dss, chol);
        });
        if (rc) return rc;
        int hflag = 0;
        CU(h, cudaMemcpy(&hflag, flag, sizeof(int), cudaMemcpyDeviceToHost));
        h->tm[9] += ev_ms(h->ev[7], h->ev[8]);
        if (hflag == 0) return KB200_OK;
        if (hflag != 2 || chol == 0) return fail(h, KB200_ESINGULAR, "Singular matrix");
    }
    return KB200_OK;
}

extern "C" int kb200_execute_knn_grid_dev(kb200_handle h, int k, int64_t nx, int64_t ny, int64_t nz,
                                          const double* d_gx, const double* d_gy, const double* d_gz,
                                          int64_t first, int64_t count, double* d_z, double* d_ss) {
    int rc = check_knn(h, k); if (rc) return rc;
    rc = check_grid(h, nx, ny, nz, first, count); if (rc) return rc;
    if (count == 0) return KB200_OK;
    if (!d_gx || !d_gy || (h->dim == 3 && !d_gz) || !d_z || !d_ss) return fail(h, KB200_EBADARG, "null pointer");
    Src s{true, nx, ny, nz, d_gx, d_gy, d_gz, first, count, nullptr, 0, 0};
    int* flag = h->wFlag.as<int>();
    for (int chol = 1; chol >= 0; --chol) {
        CU(h, cudaMemsetAsync(flag, 0, sizeof(int), h->stream));
        CU(h, cudaEventRecord(h->ev[7], h->stream));
        rc = run_knn(h, k, s, d_z, d_ss, chol); if (rc) return rc;
        CU(h, cudaEventRecord(h->ev[8], h->stream));
        int hflag = 0;
        CU(h, cudaMemcpyAsync(&hflag, flag, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CU(h, cudaStreamSynchronize(h->stream));
        h->tm[9] += ev_ms(h->ev[7], h->ev[8]);
        if (hflag == 0) return KB200_OK;
        if (hflag != 2 || chol == 0) return fail(h, KB200_ESINGULAR, "Singular matrix");
    }
    return KB200_OK;
}

static int exec_knn_grid_impl(kb200_ctx* h, int k, int64_t nx, int64_t ny, int64_t nz,
                              const double* gx, const double* gy, const double* gz,
                              int64_t cfirst, int64_t first, int64_t count, double* z_out, double* ss_out) {
    int rc = check_knn(h, k); if (rc) return rc;
    rc = check_grid(h, nx, ny, nz, first, count); if (rc) return rc;
    if (count == 0) return KB200_OK;
    if (!gx || !gy || (h->dim == 3 && !gz) || !z_out || !ss_out) return fail(h, KB200_EBADARG, "null pointer");
    cudaStream_t st = h->stream;
    CU(h, h->wAxes.reserve((size_t)(nx + ny + nz) * 8));
    double* da = h->wAxes.as<double>();
    CU(h, cudaEventRecord(h->ev[9], st));
    CU(h, cudaMemcpyAsync(da, gx, nx * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaMemcpyAsync(da + nx, gy, ny * 8, cudaMemcpyHostToDevice, st));
    if (h->dim == 3) CU(h, cudaMemcpyAsync(da + nx + ny, gz, nz * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaEventRecord(h->ev[10], st));
    rc = knn_to_host(h, k, count, z_out + (first - cfirst), ss_out + (first - cfirst), [&](int64_t o, int64_t c) {
        return Src{true, nx, ny, nz, da, da + nx, da + nx + ny, first + o, c, nullptr, 0, 0};
    });
    if (rc) return rc;
    h->tm[6] += ev_ms(h->ev[9], h->ev[10]);
    return KB200_OK;
}

extern "C" int kb200_execute_knn_grid(kb200_handle h, int k, int64_t nx, int64_t ny, int64_t nz,
                                      const double* gx, const double* gy, const double* gz,
                                      int64_t first, int64_t count, double* z_out, double* ss_out) {
    if (!h) return KB200_EBADARG;
    return exec_knn_grid_impl(h, k, nx, ny, nz, gx, gy, gz, first, first, count, z_out, ss_out);
}

static int exec_knn_points_impl(kb200_ctx* h, int k, int64_t off, int64_t m,
                                const double* px, const double* py, const double* pz, double* z_out, double* ss_out) {
    int rc = check_knn(h, k); if (rc) return rc;
    if (m <= 0) return KB200_OK;
    if (!px || !py || (h->dim == 3 && !pz) || !z_out || !ss_out) return fail(h, KB200_EBADARG, "null pointer");
    cudaStream_t st = h->stream;
    CU(h, h->wPts.reserve((size_t)3 * m * 8));
    double* dp = h->wPts.as<double>();
    CU(h, cudaEventRecord(h->ev[9], st));
    CU(h, cudaMemcpyAsync(dp, px + off, m * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaMemcpyAsync(dp + m, py + off, m * 8, cudaMemcpyHostToDevice, st));
    if (h->dim == 3) CU(h, cudaMemcpyAsync(dp + 2 * m, pz + off, m * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaEventRecord(h->ev[10], st));
    rc = knn_to_host(h, k, m, z_out + off, ss_out + off, [&](int64_t o, int64_t c) {
        return Src{false, 0, 0, 0, dp, dp + m, dp + 2 * m, o, c, nullptr, 0, 0};
    });
    if (rc) return rc;
    h->tm[6] += ev_ms(h->ev[9], h->ev[10]);
    return KB200_OK;
}

extern "C" int kb200_execute_knn_points(kb200_handle h, int k, int64_t m,
                                        const double* px, const double* py, const double* pz,
                                        double* z_out, double* ss_out) {
    if (!h) return KB200_EBADARG;
    return exec_knn_points_impl(h, k, 0, m, px, py, pz, z_out, ss_out);
}

// ---- single-process multi-GPU: a group of handles driven by one caller thread --------------------------------
// SURVEY.md §8(b)/(e): the caller makes ONE call from one host thread; inside, one worker thread per device runs
// the per-device call on that device's handle (CUDA work of different devices overlaps, and so do the host-side
// drains of the staged outputs). Device 0 factors; the factor blob goes to the peers by cudaMemcpyPeerAsync over
// NVLink (the single transfer of the path); prediction points are cut into contiguous blocks in the reference's
// flattened order (ok.py:864-866), so the gathered result equals the single-GPU result bit for bit.
struct kb200_group_ctx {
    std::vector<kb200_ctx*> m;
    bool peers = false;
    std::string err;
};

static int gfail(kb200_group_ctx* g, int code, const std::string& msg) { if (g) g->err = msg; return code; }

template <class F>
static int group_parallel(kb200_group_ctx* g, F f) {
    const int G = (int)g->m.size();
    std::vector<int> rc(G, KB200_OK);
    std::vector<std::thread> th;
    th.reserve(G);
    for (int i = 1; i < G; ++i) th.emplace_back([&, i]() { rc[i] = f(i); });
    rc[0] = f(0);
    for (auto& t : th) t.join();
    for (int i = 0; i < G; ++i)
        if (rc[i] != KB200_OK) return gfail(g, rc[i], "device " + std::to_string(g->m[i]->device) + ": " + g->m[i]->err);
    return KB200_OK;
}

static void shard_block(int64_t count, int rank, int world, int64_t* first, int64_t* n) {
    const int64_t base = count / world, rem = count % world;
    *first = rank * base + std::min<int64_t>(rank, rem);
    *n = base + (rank < rem ? 1 : 0);
}

extern "C" int kb200_group_create(kb200_group* out, int n_gpus, const int* devices) {
    if (!out) return KB200_EBADARG;
    *out = nullptr;
    int cnt = 0;
    if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt == 0) return KB200_ECUDA;
    if (n_gpus < 1 || n_gpus > cnt) return KB200_EBADARG;
    kb200_group_ctx* g = new kb200_group_ctx();
    for (int i = 0; i < n_gpus; ++i) {
        kb200_handle h = nullptr;
        int rc = kb200_create(&h, devices ? devices[i] : i);
        if (rc != KB200_OK) { for (auto* m : g->m) kb200_destroy(m); delete g; return rc; }
        g->m.push_back(h);
    }
    *out = g;
    return KB200_OK;
}

extern "C" void kb200_group_destroy(kb200_group g) {
    if (!g) return;
    for (auto* m : g->m) kb200_destroy(m);
    delete g;
}

extern "C" const char* kb200_group_last_error(kb200_group g) { return g ? g->err.c_str() : "null group"; }
extern "C" int kb200_group_size(kb200_group g) { return g ? (int)g->m.size() : 0; }
extern "C" kb200_handle kb200_group_member(kb200_group g, int i) {
    return (g && i >= 0 && i < (int)g->m.size()) ? g->m[i] : nullptr;
}

extern "C" int kb200_group_set_problem(kb200_group g, int dim, int dtype, int64_t n,
                                       const double* x, const double* y, const double* z, const double* values,
                                       const double* center, const double* aniso,
                                       int model, const double* vparams, int n_vparams,
                                       int exact_values, double eps, int n_rl, int n_hd, const double* drift_data) {
    if (!g || g->m.empty()) return KB200_EBADARG;
    // member 0 assembles + factors while the peers describe the problem (allocating their blobs)
    int rc = group_parallel(g, [&](int i) {
        if (i == 0) return kb200_set_problem(g->m[0], dim, dtype, n, x, y, z, values, center, aniso, model, vparams,
                                             n_vparams, exact_values, eps, n_rl, n_hd, drift_data);
        return kb200_describe_problem(g->m[i], dim, dtype, n, x, y, z, values, center, aniso, model, vparams,
                                      n_vparams, exact_values, eps, n_rl, n_hd, drift_data);
    });
    if (rc) return rc;
    const int G = (int)g->m.size();
    kb200_ctx* h0 = g->m[0];
    if (G > 1 && !g->peers) {
        for (int i = 1; i < G; ++i) {
            int can = 0;
            cudaDeviceCanAccessPeer(&can, g->m[i]->device, h0->device);
            if (can) { cudaSetDevice(g->m[i]->device); cudaDeviceEnablePeerAccess(h0->device, 0); cudaGetLastError(); }
        }
        g->peers = true;
    }
    cudaSetDevice(h0->device);
    for (int i = 1; i < G; ++i) {
        if (g->m[i]->blob_bytes != h0->blob_bytes) return gfail(g, KB200_ESTATE, "group: blob size mismatch");
        cudaError_t e = cudaMemcpyPeerAsync(g->m[i]->blob.p, g->m[i]->device, h0->blob.p, h0->device, h0->blob_bytes, h0->stream);
        if (e != cudaSuccess) return gfail(g, KB200_ECUDA, std::string("cudaMemcpyPeerAsync: ") + cudaGetErrorString(e));
    }
    if (cudaStreamSynchronize(h0->stream) != cudaSuccess) return gfail(g, KB200_ECUDA, "group: blob copy failed");
    for (int i = 1; i < G; ++i) {
        rc = kb200_blob_commit(g->m[i]);
        if (rc) return gfail(g, rc, g->m[i]->err);
    }
    return KB200_OK;
}

extern "C" int kb200_group_set_problem_knn(kb200_group g, int dim, int64_t n,
                                           const double* x, const double* y, const double* z, const double* values,
                                           const double* center, const double* aniso,
                                           int model, const double* vparams, int n_vparams, int exact_values, double eps) {
    if (!g || g->m.empty()) return KB200_EBADARG;
    // every device builds its own cell grid from the coordinates (1.6-2.4 MB of input; nothing to broadcast)
    return group_parallel(g, [&](int i) {
        return kb200_set_problem_knn(g->m[i], dim, n, x, y, z, values, center, aniso, model, vparams, n_vparams,
                                     exact_values, eps);
    });
}

extern "C" int kb200_group_execute_grid(kb200_group g, int64_t nx, int64_t ny, int64_t nz,
                                        const double* gx, const double* gy, const double* gz,
                                        const double* drift_pts, int64_t first, int64_t count,
                                        double* z_out, double* ss_out) {
    if (!g || g->m.empty()) return KB200_EBADARG;
    const int G = (int)g->m.size();
    return group_parallel(g, [&](int i) {
        int64_t f, c; shard_block(count, i, G, &f, &c);
        return exec_grid_impl(g->m[i], nx, ny, nz, gx, gy, gz, drift_pts, first, count, first + f, c, z_out, ss_out);
    });
}

extern "C" int kb200_group_execute_points(kb200_group g, int64_t m,
                                          const double* px, const double* py, const double* pz,
                                          const double* drift_pts, double* z_out, double* ss_out) {
    if (!g || g->m.empty()) return KB200_EBADARG;
    const int G = (int)g->m.size();
    return group_parallel(g, [&](int i) {
        int64_t f, c; shard_block(m, i, G, &f, &c);
        return exec_points_impl(g->m[i], f, c, px, py, pz, drift_pts, m, z_out, ss_out);
    });
}

extern "C" int kb200_group_execute_knn_grid(kb200_group g, int k, int64_t nx, int64_t ny, int64_t nz,
                                            const double* gx, const double* gy, const double* gz,
                                            int64_t first, int64_t count, double* z_out, double* ss_out) {
    if (!g || g->m.empty()) return KB200_EBADARG;
    const int G = (int)g->m.size();
    return group_parallel(g, [&](int i) {
        int64_t f, c; shard_block(count, i, G, &f, &c);
        return exec_knn_grid_impl(g->m[i], k, nx, ny, nz, gx, gy, gz, first, first + f, c, z_out, ss_out);
    });
}

extern "C" int kb200_group_execute_knn_points(kb200_group g, int k, int64_t m,
                                              const double* px, const double* py, const double* pz,
                                              double* z_out, double* ss_out) {
    if (!g || g->m.empty()) return KB200_EBADARG;
    const int G = (int)g->m.size();
    return group_parallel(g, [&](int i) {
        int64_t f, c; shard_block(m, i, G, &f, &c);
        return exec_knn_points_impl(g->m[i], k, f, c, px, py, pz, z_out, ss_out);
    });
}

// ---- debug taps (tests only) ------------------------------------------------
// ---- constructor-side helpers (SURVEY.md 8f next-2) -----------------------------------------------
extern "C" int kb200_experimental_variogram(kb200_handle h, int dim, int64_t n,
                                            const double* x, const double* y, const double* z, const double* values,
                                            int nlags, double* counts, double* lag_sum, double* semi_sum,
                                            double* dminmax) {
    if (!h) return KB200_EBADARG;
    if (dim != 2 && dim != 3) return fail(h, KB200_EBADARG, "dim must be 2 or 3");
    if (h->geo && dim != 2) return fail(h, KB200_EBADARG, "Geographic coordinate type only supported for 2D datasets.");
    if (n < 2 || n > 2000000000LL) return fail(h, KB200_EBADARG, "the experimental variogram needs 2 <= n < 2^31 points");
    if (nlags < 1 || nlags > 4096) return fail(h, KB200_EBADARG, "nlags must be in [1, 4096]");
    if (!x || !y || (dim == 3 && !z) || !values || !counts || !lag_sum || !semi_sum)
        return fail(h, KB200_EBADARG, "null array");
    cudaSetDevice(h->device);
    cudaStream_t st = h->stream;
    const int nn = (int)n, kdim = h->geo ? KB_GEO : dim;
    // persistent CTAs: as many per SM as the (private-bin) shared memory allows, up to 8 — the pair loop is a
    // chain of shared-memory read-modify-writes and square roots, so it needs warps to hide latency
    const size_t ev_sm = kbk_ev_smem(nlags, nlags <= kbk_ev_priv_max_lags() ? 1 : 0) + 1024;
    const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (size_t)(220 * 1024) / ev_sm));
    const int grid = kbk_ev_grid(nn, per_sm * h->num_sms);
    // workspace: x | y | z | v | edges | bmin | bmax | part | out
    const size_t o_edges = 4 * (size_t)nn, o_bmin = o_edges + nlags + 1, o_bmax = o_bmin + grid,
                 o_part = o_bmax + grid, o_out = o_part + (size_t)grid * 3 * nlags, total = o_out + 3 * (size_t)nlags;
    CU(h, h->wVario.reserve(total * sizeof(double)));
    double* w = h->wVario.as<double>();
    double *dx = w, *dy = w + nn, *dz = w + 2 * (size_t)nn, *dv = w + 3 * (size_t)nn;
    CU(h, cudaMemcpyAsync(dx, x, (size_t)nn * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaMemcpyAsync(dy, y, (size_t)nn * 8, cudaMemcpyHostToDevice, st));
    if (dim == 3) CU(h, cudaMemcpyAsync(dz, z, (size_t)nn * 8, cudaMemcpyHostToDevice, st));
    CU(h, cudaMemcpyAsync(dv, values, (size_t)nn * 8, cudaMemcpyHostToDevice, st));
    CU(h, kbk_ev_minmax(kdim, nn, dx, dy, dz, grid, w + o_bmin, w + o_bmax, st));
    std::vector<double> mm(2 * (size_t)grid);
    CU(h, cudaMemcpyAsync(mm.data(), w + o_bmin, 2 * (size_t)grid * 8, cudaMemcpyDeviceToHost, st));
    CU(h, cudaStreamSynchronize(st));
    double dmin = mm[0], dmax = mm[grid];
    for (int b = 1; b < grid; ++b) { dmin = std::min(dmin, mm[b]); dmax = std::max(dmax, mm[grid + b]); }
    if (!(dmax >= dmin)) return fail(h, KB200_EBADARG, "pair distances are not finite");
    // equal-width lag edges exactly as core.py:471-476 (same fp64 expression, evaluated on the host)
    const double dd = (dmax - dmin) / nlags;
    std::vector<double> edges(nlags + 1);
    for (int k = 0; k < nlags; ++k) edges[k] = dmin + k * dd;
    edges[nlags] = dmax + 0.001;
    CU(h, cudaMemcpyAsync(w + o_edges, edges.data(), (size_t)(nlags + 1) * 8, cudaMemcpyHostToDevice, st));
    CU(h, kbk_ev_bin(kdim, nn, dx, dy, dz, dv, nlags, w + o_edges, dd > 0.0 ? 1.0 / dd : 0.0, grid,
                     w + o_part, w + o_out, st));
    std::vector<double> out(3 * (size_t)nlags);
    CU(h, cudaMemcpyAsync(out.data(), w + o_out, out.size() * 8, cudaMemcpyDeviceToHost, st));
    CU(h, cudaStreamSynchronize(st));
    for (int k = 0; k < nlags; ++k) { counts[k] = out[k]; lag_sum[k] = out[nlags + k]; semi_sum[k] = out[2 * (size_t)nlags + k]; }
    if (dminmax) { dminmax[0] = dmin; dminmax[1] = dmax; }
    h->launches += 3;
    return KB200_OK;
}

extern "C" int kb200_statistics(kb200_handle h, double* delta, double* sigma) {
    if (!h || !delta || !sigma) return KB200_EBADARG;
    if (!h->ready) return fail(h, KB200_ESTATE, "no factored problem: call kb200_set_problem first");
    if (h->gform) return fail(h, KB200_EUNSUPPORTED, "cross-validation statistics need the positive definite "
                              "covariance form (this problem runs on the general fallback)");
    if (!h->factor_live) return fail(h, KB200_ESTATE, "the Cholesky factor is not on this handle "
                                     "(problem received through kb200_blob_commit)");
    cudaSetDevice(h->device);
    cudaStream_t st = h->stream;
    const int nn = h->n, np = h->n_pad;
    char* blob = h->blob.as<char>();
    const double* ax = reinterpret_cast<double*>(blob + h->off_ax);
    const double* ay = reinterpret_cast<double*>(blob + h->off_ay);
    const double* az = reinterpret_cast<double*>(blob + h->off_az);
    const double* Hz = h->wF.as<double>() + (size_t)KB_MAXAUX * np;
    const int K = h->n_rl + h->n_hd;                       // Hz row K = L^-1 1, row K+1 = L^-1 Z
    CU(h, h->wVario.reserve((size_t)nn * (2 * sizeof(double) + sizeof(int)) + 256));
    double* d_delta = h->wVario.as<double>();
    double* d_sigma = d_delta + nn;
    int* d_dup = reinterpret_cast<int*>(d_sigma + nn);
    CU(h, kbk_statistics(h->dim, nn, ax, ay, az, h->wC.as<double>(), h->ld,
                         Hz + (size_t)K * np, Hz + (size_t)(K + 1) * np, d_dup, d_delta, d_sigma, st));
    CU(h, cudaMemcpyAsync(delta, d_delta, (size_t)nn * 8, cudaMemcpyDeviceToHost, st));
    CU(h, cudaMemcpyAsync(sigma, d_sigma, (size_t)nn * 8, cudaMemcpyDeviceToHost, st));
    CU(h, cudaStreamSynchronize(st));
    h->launches += 2;
    return KB200_OK;
}

extern "C" int64_t kb200_debug_fetch(kb200_handle h, int what, double* out, int64_t cap) {
    if (!h || !out) return KB200_EBADARG;
    if (!h->described) return KB200_ESTATE;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    const size_t mat = (size_t)h->n_pad * h->ld;
    const void* src = nullptr; size_t cnt = 0;
    if (what == 1) { src = h->wC.p; cnt = mat; }
    else if (what == 2) { src = h->wW.p; cnt = mat; }
    else if (what == 3) {
        size_t nU = (size_t)h->na * h->n_pad;
        size_t total = nU + (size_t)h->K1 * h->K1 + h->K1 + 1;
        if ((int64_t)total > cap) return KB200_EBADARG;
        const double* Uz = h->wF.as<double>() + (size_t)2 * KB_MAXAUX * h->n_pad;
        if (cudaMemcpy(out, Uz, nU * 8, cudaMemcpyDeviceToHost) != cudaSuccess) return KB200_ECUDA;
        if (cudaMemcpy(out + nU, h->blob.as<char>() + h->off_consts, ((size_t)h->K1 * h->K1 + h->K1) * 8,
                       cudaMemcpyDeviceToHost) != cudaSuccess) return KB200_ECUDA;
        out[total - 1] = h->vg.c0;
        return (int64_t)total;
    } else return KB200_EBADARG;
    if (!src) return KB200_ESTATE;
    if ((int64_t)cnt > cap) return KB200_EBADARG;
    if (cudaMemcpy(out, src, cnt * 8, cudaMemcpyDeviceToHost) != cudaSuccess) return KB200_ECUDA;
    return (int64_t)cnt;
}
