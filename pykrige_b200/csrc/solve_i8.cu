// solve_i8.cu — K3 on the INT8 path of the 5th-generation tensor cores (tcgen05.mma kind::i8, exact int32 accumulation
// in TMEM): q_j = ||W c_j||^2 (DESIGN.md §3) for dtype = KB200_F64 (S = 8, the default fp64 route for
// KB_F64_I8_NMIN <= n <= 65535 on the Cholesky path, api.cu) and KB200_F64X / F64X5 / F64X4 (S = 6 / 5 / 4).
//
// Error-free slicing (the "Ozaki scheme"): every row of W and every RHS column is scaled by a power of two
// into (-1, 1) and cut into S signed slices of 6+7+...+7 bits (S = 8: 55 bits, 6: 41, 5: 34, 4: 27),
//      x = 2^e * sum_s slice_s * 2^(-6-7s),   |slice_s| <= 64,
// so that  W_rk c_k = 2^(ew_r + ec_j) * sum_{s,t} w_s c_t 2^(-12-7(s+t)).  All slice products with the
// same d = s + t are summed EXACTLY in one int32 TMEM accumulator (|sum| <= n * (d+1) * 64^2 < 2^31 for
// n <= 65535 at S = 8); pairs with d >= S are dropped (relative 2^-(7S+6) per term). The S accumulators are combined
// exactly in int64 in the epilogue and converted to fp64 once. S = 8 is as accurate as the fp64 product it replaces
// (tests/test_f64_int8_route.py); S = 6 agrees with the fp64 DMMA kernel to ~1e-10; fewer slices trade bits for MMAs
// (S(S+1)/2 per k-stage: 36 / 21 / 15 / 10) and operand bytes.
//
// Orientation as in solve_tf32.cu: D[point][W row], M = 128 points (TMEM lanes), N = BN W rows per row block
// with S * BN <= 512 TMEM columns (BN = 64 / 80 / 96 / 128: the RHS slices are re-read once per row block, so fewer
// slices also mean fewer re-reads), K = 32 per MMA; operands in the canonical no-swizzle K-major UMMA layout
// (8-row x 16-byte core matrices, k-chunks 128 B apart, 8-row groups 256 B apart), one stage = 32 k = one MMA
// k-step. The variogram model is a run-time switch here (phase G is < 10 % of the kernel), so that the slice
// count and the dimension are the only template parameters.
#include "common.cuh"
#include "kernels.h"

#define I8_THREADS 512
#define I8_GEN_THREADS 256                 // warps 8..15: two generator threads per prediction point
#define I8_TM 128
#define I8_BK 32
#define I8_C_SLICE (I8_TM * I8_BK)            // 4 KB

template <int S> struct I8Cfg {
    static constexpr int BN = (S == 8) ? 64 : (S == 6) ? 80 : (S == 5) ? 96 : 128;   // S * BN <= 512 TMEM columns, BN % 16 == 0
    static constexpr int STAGES = (S == 8) ? 4 : (S == 4) ? 6 : 5;                 // S = 8: 4 x 48 KB stages
    static constexpr int W_SLICE = BN * I8_BK;
    static constexpr int W_BYTES = S * W_SLICE;
    static constexpr int C_BYTES = S * I8_C_SLICE;
    static constexpr int STAGE_BYTES = W_BYTES + C_BYTES;
    // D = S32 (bits 4-5 = 2), A = B = signed 8 bit (bits 7-9, 10-12 = 1), K-major, N = BN, M = 128
    static constexpr uint32_t IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(I8_TM >> 4) << 24);
};

__device__ __forceinline__ uint32_t i8_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void i8_mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" :: "r"(i8_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void i8_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" :: "r"(i8_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void i8_mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" :: "r"(i8_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void i8_mbar_wait(uint64_t* bar, uint32_t parity) {
    for (uint32_t it = 0; it < (1u << 26); ++it) {
        uint32_t ok;
        asm volatile("{\n\t.reg .pred p;\n\t"
                     "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(ok) : "r"(i8_smem_u32(bar)), "r"(parity) : "memory");
        if (ok) return;
    }
    __trap();
}
__device__ __forceinline__ void i8_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 :: "r"(i8_smem_u32(dst)), "l"(src), "r"(bytes), "r"(i8_smem_u32(bar)) : "memory");
}
// K-major, no swizzle: LBO (k-chunk stride) = 128 B, SBO (8-row group stride) = 256 B, version 1
__device__ __forceinline__ uint64_t i8_desc(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3fffu) | ((uint64_t)(128u >> 4) << 16) | ((uint64_t)(256u >> 4) << 32) |
           (1ull << 46);
}
__device__ __forceinline__ void i8_mma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "setp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}\n"
                 :: "r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void i8_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n"
                 :: "r"(i8_smem_u32(bar)) : "memory");
}

// CW consecutive 32-bit TMEM columns of this thread's lane (CW = 8 or 16), waited for
template <int CW>
__device__ __forceinline__ void i8_tmem_ld(uint32_t taddr, uint32_t (&u)[CW]) {
    if constexpr (CW == 16) {
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
            : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
              "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
            : "r"(taddr));
    } else {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
                     : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7])
                     : "r"(taddr));
    }
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
}

// S signed 7-bit digits of y = x * 2^-e (|y| < 1): x = 2^e * sum_s out[s] * 2^(-6-7s) + O(2^(e-7S)), out[s] in [-64, 64].
// One fp64 multiply + one round-to-nearest conversion to a 6+7(S-1)-bit integer, then balanced base-128 digits with
// integer ops (the digit loop used to be 4 fp64 instructions per slice on the pipe the RHS generators are bound by).
template <int S>
__device__ __forceinline__ void i8_slice(double x, int e, signed char (&out)[S]) {
    long long v = __double2ll_rn(scalbn(x, 6 + 7 * (S - 1) - e));      // |v| <= 2^(6+7(S-1))
#pragma unroll
    for (int s = S - 1; s >= 1; --s) {
        const int d = (int)((v + 64) & 127) - 64;                        // balanced digit in [-64, 63]
        out[s] = (signed char)d;
        v = (v - d) >> 7;                                                // exact: v - d is a multiple of 128
    }
    out[0] = (signed char)v;                                             // |v| <= 64
}
// the same with the scale 2^(6+7(S-1)-e) precomputed by the caller (one per prediction point)
template <int S>
__device__ __forceinline__ void i8_slice_scaled(double x, double scale, signed char (&out)[S]) {
    if (S <= 4) {                                                        // 27 bits + sign: 32-bit integer digits
        int v = __double2int_rn(x * scale);
#pragma unroll
        for (int s = S - 1; s >= 1; --s) {
            const int d = ((v + 64) & 127) - 64;
            out[s] = (signed char)d;
            v = (v - d) >> 7;
        }
        out[0] = (signed char)v;
    } else {
        long long v = __double2ll_rn(x * scale);
#pragma unroll
        for (int s = S - 1; s >= 1; --s) {
            const int d = (int)((v + 64) & 127) - 64;
            out[s] = (signed char)d;
            v = (v - d) >> 7;
        }
        out[0] = (signed char)v;
    }
}
// byte offset of element (r, k) inside one slice tile with `rows` rows (k in [0, 32))
__device__ __forceinline__ int i8_off(int r, int k) { return (r >> 3) * 256 + (k >> 4) * 128 + (r & 7) * 16 + (k & 15); }

__host__ __device__ __forceinline__ int i8_ktiles(int J, int n, int nk, int BN) {
    return ((J + 1) * BN > n) ? nk : min(nk, ((J + 1) * BN + I8_BK - 1) / I8_BK);
}

// ---- pack ---------------------------------------------------------------------------------------------
// rowscale[r] = 2^(ew_r - 12) with ew_r = exponent such that max_k |row_r[k]| * 2^-ew_r < 1
__global__ void __launch_bounds__(256) i8_rowscale_kernel(const double* __restrict__ W, int ld, int n, int n_pad, int na,
                                                           const double* __restrict__ Uz, int nrows,
                                                           int* __restrict__ rowexp, double* __restrict__ rowscale) {
    int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (row >= nrows) return;
    double m = 0.0;
    if (row < n) { for (int k = lane; k <= row; k += 32) m = fmax(m, fabs(W[(size_t)row * ld + k])); }
    else if (row < n + na) { for (int k = lane; k < n; k += 32) m = fmax(m, fabs(Uz[(size_t)(row - n) * n_pad + k])); }
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) {
        int e = 0;
        if (m > 0.0) { (void)frexp(m, &e); }        // m = f * 2^e, f in [0.5, 1)
        rowexp[row] = e;
        rowscale[row] = scalbn(1.0, e - 12);
    }
}

// tile (row block J, k stage t): S slices x (BN rows x 32 k) int8 in UMMA layout
template <int S>
__global__ void __launch_bounds__(256) i8_pack_kernel(const double* __restrict__ W, int ld, int n, int n_pad, int na,
                                                       const double* __restrict__ Uz, const int* __restrict__ rowexp,
                                                       int nk, const long long* __restrict__ tile_off,
                                                       signed char* __restrict__ out) {
    typedef I8Cfg<S> C;
    const int J = blockIdx.y, t = blockIdx.x;
    if (t >= i8_ktiles(J, n, nk, C::BN)) return;
    signed char* o = out + (size_t)(tile_off[J] + t) * C::W_BYTES;
    for (int e = threadIdx.x; e < C::BN * I8_BK; e += 256) {
        const int rl = e >> 5, kl = e & 31;
        const int r = J * C::BN + rl, k = t * I8_BK + kl;
        double v = 0.0;
        if (r < n) { if (k <= r) v = W[(size_t)r * ld + k]; }
        else if (r < n + na) { if (k < n) v = Uz[(size_t)(r - n) * n_pad + k]; }
        signed char sl[S];
        i8_slice<S>(v, (r < n + na) ? rowexp[r] : 0, sl);
        const int off = i8_off(rl, kl);
#pragma unroll
        for (int s = 0; s < S; ++s) o[s * C::W_SLICE + off] = sl[s];
    }
}

// shifted covariance with the model as a run-time switch (uniform across the grid)
__device__ __forceinline__ double i8_cov_rhs(const VgParams& v, double d) {
    switch (v.model) {
        case KB200_VG_LINEAR: return kb_cov_rhs<KB200_VG_LINEAR>(v, d);
        case KB200_VG_POWER: return kb_cov_rhs<KB200_VG_POWER>(v, d);
        case KB200_VG_GAUSSIAN: return kb_cov_rhs<KB200_VG_GAUSSIAN>(v, d);
        case KB200_VG_EXPONENTIAL: return kb_cov_rhs<KB200_VG_EXPONENTIAL>(v, d);
        case KB200_VG_SPHERICAL: return kb_cov_rhs<KB200_VG_SPHERICAL>(v, d);
        case KB200_VG_TABLE: return kb_cov_rhs<KB200_VG_TABLE>(v, d);
        default: return kb_cov_rhs<KB200_VG_HOLE_EFFECT>(v, d);
    }
}

// Warp roles (512 threads): warp 0 lane 0 = bulk-copy producer, warp 1 lane 0 = MMA issuer, warp 2 = TMEM allocator,
// warps 4-7 = epilogue (thread = TMEM lane = prediction point), warps 8-15 = RHS generators (two threads per point,
// alternating k-stages: the fp64 sqrt/exp chains are latency-bound, eight warps keep the pipe fed; twelve gave +2 % at
// S = 4 and -8 % at S = 6 through register spills).
// The generators work one point tile AHEAD of the tensor pipe: they evaluate and slice the RHS column block of
// tile i+1 into the other half of the double-buffered scratch ring while the MMAs of tile i run (the fp64 pipe
// and the tensor pipe do not compete); gfull / gempty mbarriers hand the buffers over.
template <int S, int DIM>
__global__ void __launch_bounds__(I8_THREADS, 1) solve_kernel_i8(const __grid_constant__ SolvePtParams P) {
    typedef I8Cfg<S> C;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* stage_base = smem_raw;                                                    // STAGES * STAGE_BYTES
    double* auxs = reinterpret_cast<double*>(smem_raw + (size_t)C::STAGES * C::STAGE_BYTES);  // KB_MAXAUX * 128
    int* pexp = reinterpret_cast<int*>(auxs + KB_MAXAUX * I8_TM);                            // 2 x 128 point exponents
    uint64_t* full = reinterpret_cast<uint64_t*>(pexp + 2 * I8_TM);                          // STAGES
    uint64_t* empty = full + C::STAGES;
    uint64_t* tfull = empty + C::STAGES;                                                     // 1
    uint64_t* tempty = tfull + 1;                                                            // 1
    uint64_t* gfull = tempty + 1;                                                            // 2
    uint64_t* gempty = gfull + 2;                                                            // 2
    uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(gempty + 2);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nk = (P.n + I8_BK - 1) / I8_BK;
    const int nrb = (P.n + P.na + C::BN - 1) / C::BN;
    const size_t sbuf = (size_t)nk * C::C_BYTES;                                             // one RHS column block
    unsigned char* scratch = reinterpret_cast<unsigned char*>(P.scratch) + (size_t)blockIdx.x * 2 * sbuf;
    const unsigned char* gt = reinterpret_cast<const unsigned char*>(P.tiles);
    const long long ntiles = (P.m + I8_TM - 1) / I8_TM;
    const int model = P.vg.model;

    if (tid == 0) {
        for (int s = 0; s < C::STAGES; ++s) { i8_mbar_init(&full[s], 1); i8_mbar_init(&empty[s], 1); }
        i8_mbar_init(tfull, 1); i8_mbar_init(tempty, 4);
        for (int b = 0; b < 2; ++b) { i8_mbar_init(&gfull[b], I8_GEN_THREADS); i8_mbar_init(&gempty[b], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n"
                     :: "r"(i8_smem_u32(tmem_base_smem)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem_base = *tmem_base_smem;

    if (warp >= 8) {
        // ---------------- generators: RHS column block -> S int8 slices per value, UMMA layout ----------------
        const int pl = (tid - 8 * 32) & (I8_TM - 1);       // 0..127: point within the tile
        const int ks = (tid - 8 * 32) >> 7;                // 0..1: k-stage parity handled by this thread
        constexpr int KW = (S == 8) ? 8 : 16;              // k values sliced per store (S = 8: fewer live slice bytes)
        uint32_t it = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
            const int b = (int)(it & 1);
            i8_mbar_wait(&gempty[b], ((it >> 1) & 1) ^ 1);         // the tile that used this buffer is finished
            unsigned char* sc = scratch + (size_t)b * sbuf;
            const long long pj = tile * I8_TM + pl;
            const bool pvalid = pj < P.m;
            double px = 0.0, py = 0.0, pz = 0.0;
            if (pvalid) kb_load_point<DIM>(P.ps, P.an, pj, px, py, pz);
            // scale of this point's column: |c| <= c0 for the bounded models (gamma <= sill); for linear / power /
            // tabulated models a first pass finds the maximum
            int ec;
            {
                double cmax = fabs(P.vg.c0);
                if (model == KB200_VG_LINEAR || model == KB200_VG_POWER || model == KB200_VG_TABLE) {
                    if (pvalid)
                        for (int k = 0; k < P.n; ++k) {
                            double d = kb_dist<DIM>(__ldg(P.ax + k), __ldg(P.ay + k), KB_HASZ(DIM) ? __ldg(P.az + k) : 0.0, px, py, pz);
                            cmax = fmax(cmax, fabs(i8_cov_rhs(P.vg, d)));
                        }
                }
                (void)frexp(cmax * 1.0000001, &ec);        // cmax * 2^-ec < 1
            }
            if (ks == 0) pexp[b * I8_TM + pl] = ec;
            const double cscale = scalbn(1.0, 6 + 7 * (S - 1) - ec);
            for (int t = ks; t < nk; t += I8_GEN_THREADS / I8_TM) {
                unsigned char* ct = sc + (size_t)t * C::C_BYTES;
#pragma unroll 1
                for (int kc = 0; kc < I8_BK / KW; ++kc) {  // KW-byte k-chunks per stage
                    signed char sl[KW][S];
#pragma unroll
                    for (int kk = 0; kk < KW; ++kk) {
                        const int k = t * I8_BK + kc * KW + kk;
                        double c = 0.0;
                        if (pvalid && k < P.n) {
                            double d = kb_dist<DIM>(__ldg(P.ax + k), __ldg(P.ay + k), KB_HASZ(DIM) ? __ldg(P.az + k) : 0.0, px, py, pz);
                            c = i8_cov_rhs(P.vg, d);
                        }
                        i8_slice_scaled<S>(c, cscale, sl[kk]);
                    }
                    const int off = i8_off(pl, kc * KW);
#pragma unroll
                    for (int s = 0; s < S; ++s) {
                        uint32_t w[KW / 4];
#pragma unroll
                        for (int q = 0; q < KW / 4; ++q)
                            w[q] = (uint32_t)(uint8_t)sl[4 * q][s] | ((uint32_t)(uint8_t)sl[4 * q + 1][s] << 8) |
                                   ((uint32_t)(uint8_t)sl[4 * q + 2][s] << 16) | ((uint32_t)(uint8_t)sl[4 * q + 3][s] << 24);
                        if constexpr (KW == 16) *reinterpret_cast<uint4*>(ct + s * I8_C_SLICE + off) = make_uint4(w[0], w[1], w[2], w[3]);
                        else *reinterpret_cast<uint2*>(ct + s * I8_C_SLICE + off) = make_uint2(w[0], w[1]);
                    }
                }
            }
            // generic-proxy global writes -> read by the async proxy (bulk copies) of this CTA
            __threadfence();
            asm volatile("fence.proxy.async.global;\n" ::: "memory");
            i8_mbar_arrive(&gfull[b]);
        }
    } else if (warp == 0) {
        // ---------------- producer: W tiles + RHS tiles -> smem ring ----------------
        if (lane == 0) {
            const uint64_t pol_w = kb_policy_evict_last(), pol_c = kb_policy_evict_first();
            uint32_t gg = 0, it = 0;
            for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
                const int b = (int)(it & 1);
                const unsigned char* sc = scratch + (size_t)b * sbuf;
                i8_mbar_wait(&gfull[b], (it >> 1) & 1);
                long long tau = 0;
                for (int J = 0; J < nrb; ++J) {
                    const int kt = i8_ktiles(J, P.n, nk, C::BN);
                    for (int t = 0; t < kt; ++t, ++tau, ++gg) {
                        const int s = gg % C::STAGES;
                        i8_mbar_wait(&empty[s], (uint32_t)(((gg / C::STAGES) & 1) ^ 1));
                        i8_mbar_expect_tx(&full[s], C::STAGE_BYTES);
                        unsigned char* sb = stage_base + (size_t)s * C::STAGE_BYTES;
                        kb_bulk_g2s_hint(sb, gt + (size_t)tau * C::W_BYTES, C::W_BYTES, &full[s], pol_w);
                        kb_bulk_g2s_hint(sb + C::W_BYTES, sc + (size_t)t * C::C_BYTES, C::C_BYTES, &full[s], pol_c);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ---------------- MMA issuer ----------------
        if (lane == 0) {
            uint32_t gg = 0, gb = 0;
            for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                for (int J = 0; J < nrb; ++J, ++gb) {
                    const int kt = i8_ktiles(J, P.n, nk, C::BN);
                    i8_mbar_wait(tempty, (uint32_t)((gb & 1) ^ 1));
                    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                    for (int t = 0; t < kt; ++t, ++gg) {
                        const int s = gg % C::STAGES;
                        i8_mbar_wait(&full[s], (uint32_t)((gg / C::STAGES) & 1));
                        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                        const uint32_t wb = i8_smem_u32(stage_base + (size_t)s * C::STAGE_BYTES);
                        const uint32_t cb = wb + C::W_BYTES;
#pragma unroll
                        for (int d = 0; d < S; ++d) {
#pragma unroll
                            for (int sw = 0; sw <= d; ++sw) {
                                const int sc = d - sw;                                     // slice of c
                                const uint32_t acc = (t == 0 && sw == 0) ? 0u : 1u;
                                i8_mma(tmem_base + (uint32_t)d * C::BN, i8_desc(cb + sc * I8_C_SLICE),
                                       i8_desc(wb + sw * C::W_SLICE), C::IDESC, acc);
                            }
                        }
                        i8_commit(&empty[s]);
                    }
                    i8_commit(tfull);
                }
            }
        }
    } else if (warp >= 4) {
        // ---------------- epilogue: thread = TMEM lane = prediction point ----------------
        constexpr int CW = (S == 8) ? 8 : 16;               // TMEM columns per load (S = 8: H and L both live)
        const int pl = (warp & 3) * 32 + lane;
        const uint32_t t_addr = tmem_base + (((uint32_t)(warp & 3) * 32u) << 16);
        uint32_t gb = 0, it = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
            const int b = (int)(it & 1);
            i8_mbar_wait(&gfull[b], (it >> 1) & 1);            // acquire the generators' pexp[b]
            const double pscale = scalbn(1.0, pexp[b * I8_TM + pl] - 7 * (S - 1));
            double q = 0.0;
            for (int J = 0; J < nrb; ++J, ++gb) {
                i8_mbar_wait(tfull, (uint32_t)(gb & 1));
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
#pragma unroll 1
                for (int ch = 0; ch < C::BN / CW; ++ch) {
                    // exact recombination: V = sum_d acc_d * 2^(7 (S-1-d)).  S <= 6: V fits in int64 (|acc_d| < 2^30, d = 0
                    // has one slice pair: < 2^27 * 2^35).  S = 8: |acc_0| <= n * 2^12 shifted by 2^49 can exceed int64, so
                    // V = H * 2^28 + L with H = sum_{d<4} acc_d 2^(7 (3-d)), L = sum_{d>=4} acc_d 2^(7 (7-d)); for
                    // n <= 65535 (|acc_d| < (d+1) 2^28) |H| < 2^50 and |L| < 2^52 are exact in int64 and in fp64, and
                    // (double)H * 2^28 + (double)L rounds V once
                    long long V[CW];
                    double X[CW];
#pragma unroll
                    for (int j = 0; j < CW; ++j) V[j] = 0;
#pragma unroll
                    for (int d = 0; d < S; ++d) {
                        uint32_t u[CW];
                        i8_tmem_ld<CW>(t_addr + (uint32_t)d * C::BN + (uint32_t)(ch * CW), u);
#pragma unroll
                        for (int j = 0; j < CW; ++j) V[j] = V[j] * 128 + (long long)(int)u[j];
                        if (S == 8 && d == 3) {
#pragma unroll
                            for (int j = 0; j < CW; ++j) { X[j] = (double)V[j] * 268435456.0; V[j] = 0; }   // H * 2^28
                        }
                    }
                    const int r0 = J * C::BN + ch * CW;
#pragma unroll
                    for (int j = 0; j < CW; ++j) {
                        const int r = r0 + j;
                        if (r < P.n + P.na) {
                            const double v = (S == 8) ? X[j] + (double)V[j] : (double)V[j];
                            const double x = v * (__ldg(P.rowscale + r) * pscale);
                            if (r < P.n) q += x * x;
                            else auxs[(r - P.n) * I8_TM + pl] = x;
                        }
                    }
                }
                asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
                __syncwarp();
                if (lane == 0) i8_mbar_arrive(tempty);
            }
            // ---------------- phase F: finalize (DESIGN.md §3), thread = point ----------------
            const long long pj = tile * I8_TM + pl;
            if (pj < P.m) kb_finalize_point<DIM, double>(P, pj, q, auxs + pl, I8_TM);
            __syncwarp();
            if (lane == 0) i8_mbar_arrive(&gempty[b]);       // scratch half b and pexp[b] may be rewritten
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" :: "r"(tmem_base), "r"(512u) : "memory");
    }
}

// ---- host side ---------------------------------------------------------------------------------------
template <int S> static size_t i8_smem_s() {
    return (size_t)I8Cfg<S>::STAGES * I8Cfg<S>::STAGE_BYTES + (size_t)KB_MAXAUX * I8_TM * sizeof(double) + 2 * I8_TM * sizeof(int) +
           (2 * I8Cfg<S>::STAGES + 6) * sizeof(uint64_t) + 64;
}
static int i8_bn(int S) { return S == 8 ? I8Cfg<8>::BN : S == 6 ? I8Cfg<6>::BN : S == 5 ? I8Cfg<5>::BN : I8Cfg<4>::BN; }
bool kbk_i8_valid_slices(int S) { return (S >= 4 && S <= 6) || S == 8; }
int kbk_i8_nrb(int S, int n, int na) { return (n + na + i8_bn(S) - 1) / i8_bn(S); }
int kbk_i8_rows(int S, int n, int na) { return kbk_i8_nrb(S, n, na) * i8_bn(S); }
long long kbk_i8_total_tiles(int S, int n, int na, long long* tile_off /* [nrb+1] or null */) {
    int nk = (n + I8_BK - 1) / I8_BK, nrb = kbk_i8_nrb(S, n, na);
    long long off = 0;
    for (int J = 0; J < nrb; ++J) { if (tile_off) tile_off[J] = off; off += i8_ktiles(J, n, nk, i8_bn(S)); }
    if (tile_off) tile_off[nrb] = off;
    return off;
}
size_t kbk_i8_tile_bytes(int S) { return (size_t)S * i8_bn(S) * I8_BK; }
size_t kbk_solve_i8_scratch_bytes(int S, int n, int grid) { return (size_t)grid * 2 * ((n + I8_BK - 1) / I8_BK) * S * I8_C_SLICE; }   // double-buffered
int kbk_solve_i8_tile_points() { return I8_TM; }

template <int S, int DIM>
static cudaError_t i8_attr() {
    return cudaFuncSetAttribute(solve_kernel_i8<S, DIM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)i8_smem_s<S>());
}
cudaError_t kbk_solve_i8_init() {
#define KB_ATTR(S) KB_CUDA_OK((i8_attr<S, 2>())); KB_CUDA_OK((i8_attr<S, 3>())); KB_CUDA_OK((i8_attr<S, KB_GEO>()));
    KB_ATTR(4) KB_ATTR(5) KB_ATTR(6) KB_ATTR(8)
#undef KB_ATTR
    return cudaSuccess;
}

template <int S>
static cudaError_t i8_launch(int dim, const SolvePtParams& p, int grid, cudaStream_t st) {
    const size_t sm = i8_smem_s<S>();
    if (dim == KB_GEO) solve_kernel_i8<S, KB_GEO><<<grid, I8_THREADS, sm, st>>>(p);
    else if (dim == 2) solve_kernel_i8<S, 2><<<grid, I8_THREADS, sm, st>>>(p);
    else solve_kernel_i8<S, 3><<<grid, I8_THREADS, sm, st>>>(p);
    return cudaGetLastError();
}
cudaError_t kbk_solve_i8(int S, int dim, const SolvePtParams& p, int grid, cudaStream_t st) {
    if (p.vg.model < KB200_VG_LINEAR || p.vg.model > KB200_VG_TABLE) return cudaErrorInvalidValue;
    return S == 8 ? i8_launch<8>(dim, p, grid, st) : S == 6 ? i8_launch<6>(dim, p, grid, st)
         : S == 5 ? i8_launch<5>(dim, p, grid, st) : i8_launch<4>(dim, p, grid, st);
}

// W (+ dual rows) -> row scales + int8 slice tiles. tile_off_dev: device copy of the per-row-block tile offsets.
cudaError_t kbk_pack_i8(int S, const double* W, int ld, int n, int n_pad, int na, const double* Uz,
                        int* rowexp, double* rowscale, const long long* tile_off_dev, void* out, cudaStream_t st) {
    int nrb = kbk_i8_nrb(S, n, na), nk = (n + I8_BK - 1) / I8_BK;
    int nrows = nrb * i8_bn(S);
    i8_rowscale_kernel<<<(nrows + 7) / 8, 256, 0, st>>>(W, ld, n, n_pad, na, Uz, nrows, rowexp, rowscale);
    dim3 grid(nk, nrb);
    if (S == 8) i8_pack_kernel<8><<<grid, 256, 0, st>>>(W, ld, n, n_pad, na, Uz, rowexp, nk, tile_off_dev, (signed char*)out);
    else if (S == 6) i8_pack_kernel<6><<<grid, 256, 0, st>>>(W, ld, n, n_pad, na, Uz, rowexp, nk, tile_off_dev, (signed char*)out);
    else if (S == 5) i8_pack_kernel<5><<<grid, 256, 0, st>>>(W, ld, n, n_pad, na, Uz, rowexp, nk, tile_off_dev, (signed char*)out);
    else i8_pack_kernel<4><<<grid, 256, 0, st>>>(W, ld, n, n_pad, na, Uz, rowexp, nk, tile_off_dev, (signed char*)out);
    return cudaGetLastError();
}
