// score.cu -- K4 RobustScaler -> PCA projection, K5 RBF one-class SVM decision for
// both detectors (GEMM form on the fp64 tensor pipe with the RBF/dual-coef reduction fused into
// the tile epilogue; the direct-difference fp64 kernel stays as the wide-D fallback), K6
// per-strain accumulators.
//
// Replaces improved_detection.py:134-135 (scaler.transform, pca.transform), :138-142
// (predict + decision_function of the two OneClassSVMs; libsvm k_function RBF,
// sklearn/svm/src/libsvm/svm.cpp:461-472, decision sum - rho, sign rule sum > 0) and
// the reductions behind :151-152 and :202-211.
#include <algorithm>
#include <type_traits>
#include "common.cuh"

namespace {

// ---- fp64 tensor-core form of the projection (mma.sync m8n8k4 f64), software pipelined ----
// Measured on this B200 (profiles/fp64_peak_test.cu): DFMA 36 TFLOP/s, DMMA 37 TFLOP/s; a
// register-tiled CUDA-core fp64 kernel (removed) reached ~9 because every 32-feature stage first
// waited for its global loads.  Here the components come through cp.async into a second buffer and the raw
// features of the next stage are prefetched into registers while the current stage computes.
// Block = 16 warps = 64 cells x 104 components (13 n8 tiles; blockIdx.y tiles wider PCAs);
// warp = 16 cells x 3-4 n8 tiles (4 cell groups x 4 component groups).  A call scores ~15k cells =
// 236 blocks on 148 SMs, so the warps have to come from inside the block: with 4 warps per SM the
// DMMA pipe was 21 % active (ncu), latency bound.  Shared-memory pitches put the 64-bit
// fragment loads of a half-warp on 16 distinct bank pairs (x: 36 doubles per cell row, w: 108
// per feature row).  comp_pad is the [F rounded to 32][C rounded to 104] zero-padded copy.
constexpr int DT = 512;          // threads
constexpr int DM = 64;           // cells per block
constexpr int DK = 32;           // features per stage
constexpr int DN = 104;          // components per block tile
constexpr int DXP = DK + 4;      // x pitch (doubles)
constexpr int DWP = DN + 4;      // w pitch (doubles)
constexpr int DXR = DM / (DT / 32);   // cell rows per warp in the x tile

__device__ __forceinline__ void dmma884(double (&d)[2], double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d[0]), "+d"(d[1]) : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(DT, 2)
scaler_pca_dmma_kernel(const float* __restrict__ feat, int n_cells, const int32_t* __restrict__ n_dev,
                       int F, int C, int CP, const double* __restrict__ center, const double* __restrict__ scale,
                       const double* __restrict__ rscale, int center_is_f32, const double* __restrict__ comp_pad,
                       const double* __restrict__ offset, int f32_flow, double* __restrict__ z_out) {
    extern __shared__ __align__(16) unsigned char pca_smem[];
    double* xs = reinterpret_cast<double*>(pca_smem);                 // [2][DM][DXP]
    double* ws = xs + 2 * DM * DXP;                                   // [2][DK][DWP]
    const int n = dev_count(n_cells, n_dev);
    const int cell0 = blockIdx.x * DM;
    if (cell0 >= n) return;
    const int c_tile0 = blockIdx.y * DN;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int gid = lane >> 2, tig = lane & 3;
    const int n_stages = (F + DK - 1) / DK;
    // component group of this warp: n8 tiles [nt0, nt0 + ntc) = {0-3, 4-6, 7-9, 10-12}
    const int mg = warp & 3, ng = warp >> 2;
    const int nt0 = ng == 0 ? 0 : 1 + 3 * ng, ntc = ng == 0 ? 4 : 3;
    static_assert(DN / 8 == 13 && DT == 512, "warp tiling below assumes 13 n8 tiles over 4 component groups");
    double acc[2][4][2];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;

    auto issue_w = [&](int stage, int buf) {          // DK x DN doubles as 16-byte chunks
        const double* src = comp_pad + (size_t)stage * DK * CP + c_tile0;
        double* dst = ws + buf * DK * DWP;
        // 64 chunk slots per feature row (52 used): row / chunk from shifts, no division by 52
        for (int idx = tid; idx < DK * 64; idx += DT) {
            const int ff = idx >> 6, c2 = idx & 63;
            if (c2 < DN / 2) {
                const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst + ff * DWP + 2 * c2);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src + (size_t)ff * CP + 2 * c2) : "memory");
            }
        }
    };
    float xr[DXR];
    auto load_x = [&](int stage) {                    // raw features: one cell row per warp iteration
        const int f = stage * DK + lane;
#pragma unroll
        for (int j = 0; j < DXR; ++j) {
            const int cell = cell0 + warp + j * (DT / 32);
            xr[j] = (cell < n && f < F) ? __ldg(feat + (size_t)cell * F + f) : 0.f;
        }
    };
    auto store_x = [&](int stage, int buf) {          // scaler applied on the way (sklearn's float32 flow)
        const int f = stage * DK + lane;
        double cen = 0.0, sc = 1.0, rsc = 1.0;
        if (f < F) {
            if (center) cen = center[f];
            if (scale) { sc = scale[f]; if (rscale) rsc = rscale[f]; }
        }
        double* dst = xs + buf * DM * DXP;
#pragma unroll
        for (int j = 0; j < DXR; ++j) {
            float v = xr[j];
            if (f < F) {
                if (center) {
                    if (center_is_f32) v = __fsub_rn(v, (float)cen);
                    else v = (float)__dsub_rn((double)v, cen);
                }
                if (scale) {
                    // RN(v / sc) without the division sequence: q = RN(v * RN(1/sc)) is within one
                    // ulp, the remainder v - q*sc is exact in one FMA, and q + rem * RN(1/sc) rounds
                    // to the correctly rounded quotient (Markstein); the fp32 rounding follows as in
                    // sklearn's in-place float32 division
                    const double a = (double)v;
                    if (rscale) {
                        const double q = __dmul_rn(a, rsc);
                        const double rem = __fma_rn(-q, sc, a);
                        v = (float)__fma_rn(rem, rsc, q);
                    } else {                      // a scale whose reciprocal is not a normal number
                        v = (float)__ddiv_rn(a, sc);
                    }
                }
            }
            dst[(warp + j * (DT / 32)) * DXP + lane] = (double)v;
        }
    };

    issue_w(0, 0);
    load_x(0);
    store_x(0, 0);
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();
    for (int st = 0; st < n_stages; ++st) {
        const int buf = st & 1;
        const bool more = st + 1 < n_stages;
        if (more) {
            issue_w(st + 1, buf ^ 1);
            load_x(st + 1);
        }
        const double* xb = xs + buf * DM * DXP + (mg * 16 + gid) * DXP + tig;
        const double* wb = ws + buf * DK * DWP + tig * DWP + nt0 * 8 + gid;
        // the tile count of a warp (4 or 3) is a compile-time constant inside each branch: no
        // predicate, branch or WARPSYNC in front of the MMAs
        auto mma_stage = [&](auto ntc_c) {
            constexpr int NTC = decltype(ntc_c)::value;
#pragma unroll
            for (int k4 = 0; k4 < DK / 4; ++k4) {
                const double a0 = xb[k4 * 4];
                const double a1 = xb[8 * DXP + k4 * 4];
#pragma unroll
                for (int nt = 0; nt < NTC; ++nt) {
                    const double b = wb[k4 * 4 * DWP + nt * 8];
                    dmma884(acc[0][nt], a0, b);
                    dmma884(acc[1][nt], a1, b);
                }
            }
        };
        if (ng == 0) mma_stage(std::integral_constant<int, 4>{});
        else mma_stage(std::integral_constant<int, 3>{});
        if (more) {
            store_x(st + 1, buf ^ 1);
            asm volatile("cp.async.wait_all;" ::: "memory");
        }
        __syncthreads();
    }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
        const int cell = cell0 + mg * 16 + mt * 8 + gid;
        if (cell >= n) continue;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int c = c_tile0 + (nt0 + nt) * 8 + 2 * tig + j;
                if (nt >= ntc || c >= C) continue;
                const double off = offset[c];
                double z;
                if (f32_flow) z = (double)__fsub_rn((float)acc[mt][nt][j], (float)off);
                else z = __dsub_rn(acc[mt][nt][j], off);
                z_out[(size_t)cell * C + c] = z;
            }
    }
}

constexpr int PT = 256;     // threads of the direct-difference SVM kernel
constexpr int SCELLS = 8;   // cells per block in the SVM kernel

// dec = sum_i coef_i * exp(-gamma * ||z - sv_i||^2) - rho  (fp64, direct difference).
__global__ void __launch_bounds__(PT)
svm_rbf_kernel(const double* __restrict__ z, int n_cells, const int32_t* __restrict__ n_dev, int D,
               const double* __restrict__ sv_t, const double* __restrict__ coef, int n_sv,
               int n_sv_pad, double gamma, double rho, double* __restrict__ dec,
               int8_t* __restrict__ pred) {
    extern __shared__ double zs[];  // [SCELLS][D]
    __shared__ double red[SCELLS][PT / 32];
    const int n = dev_count(n_cells, n_dev);
    const int cell0 = blockIdx.x * SCELLS;
    if (cell0 >= n) return;
    const int nc = min(SCELLS, n - cell0);
    for (int i = threadIdx.x; i < SCELLS * D; i += PT) {
        const int k = i / D;
        zs[i] = k < nc ? z[(size_t)cell0 * D + i] : 0.0;
    }
    __syncthreads();
    double part[SCELLS];
#pragma unroll
    for (int k = 0; k < SCELLS; ++k) part[k] = 0.0;
    for (int i = threadIdx.x; i < n_sv; i += PT) {
        double d2[SCELLS];
#pragma unroll
        for (int k = 0; k < SCELLS; ++k) d2[k] = 0.0;
        for (int d = 0; d < D; ++d) {
            const double s = __ldg(sv_t + (size_t)d * n_sv_pad + i);
#pragma unroll
            for (int k = 0; k < SCELLS; ++k) {
                const double df = zs[k * D + d] - s;
                d2[k] = fma(df, df, d2[k]);
            }
        }
        const double a = coef[i];
#pragma unroll
        for (int k = 0; k < SCELLS; ++k) part[k] = fma(a, exp(-gamma * d2[k]), part[k]);
    }
#pragma unroll
    for (int k = 0; k < SCELLS; ++k) {
        const double v = warp_sum(part[k]);
        if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = v;
    }
    __syncthreads();
    if (threadIdx.x < nc) {
        double s = 0.0;
        for (int w = 0; w < PT / 32; ++w) s += red[threadIdx.x][w];
        s -= rho;
        dec[cell0 + threadIdx.x] = s;
        pred[cell0 + threadIdx.x] = s > 0.0 ? 1 : -1;     // svm.cpp:2841
    }
}

// ---- K5 in GEMM form on the fp64 tensor pipe ------------------------------------------------
// ||z - s||^2 = ||z||^2 + ||s||^2 - 2 z.s : the z.s^T products of a 64-cell x 128-SV tile run as
// mma.sync m8n8k4 f64 (same fragment layout as the projection kernel above), and the epilogue of
// every tile is the fused RBF: arg = -gamma||z||^2 - gamma||s||^2 + 2 gamma z.s (clamped to <= 0),
// part += coef * exp(arg), kept per thread for its two cell rows.  In fp64 the cancellation costs
// ~1e-16 * (||z||^2 + ||s||^2) * gamma in the exponent, i.e. ~1e-13 in the decision (gate: 1e-9
// against libsvm on the same input, tests/test_gpu_parity.py).  The direct-difference kernel above
// issues a DADD and a DFMA per (cell, SV, dim) on the same fp64 pipe; this form needs one
// multiply-add, so it halves the fp64 work (north_star: "one GEMM-form kernel with a fused
// exp/dual-coef reduction").
// Block = 16 warps: 4 cell groups (16 cells = 2 m8 tiles) x 4 SV groups (32 SVs = 4 n8 tiles).
// The block's 64 z rows stay in shared memory for the whole launch ([64][DPAD+4], pitch = 4 mod 16
// doubles -> a half-warp's 64-bit fragment loads hit 16 distinct bank pairs); the support vectors
// stream through a cp.async double buffer in stages of 128 SVs x 16 dims (pitch 20 doubles).
// sv_pad is the zero-padded row-major copy [n_sv rounded to 128][D rounded to 16]; gsn[i] =
// -gamma * ||s_i||^2; padded rows have coef 0.
// min(x, 0) that lets a NaN through (fmin would turn a non-finite row into "kernel value 1" = an inlier)
__device__ __forceinline__ double neg_part(double x) { return x > 0.0 ? 0.0 : x; }

constexpr int GT = 512;            // threads
constexpr int GM = 64;             // cells per block
constexpr int GN = 128;            // support vectors per tile
constexpr int GK = 16;             // dims per stage
constexpr int GSP = GK + 4;        // pitch of a staged SV row (doubles)

__global__ void __launch_bounds__(GT, 2)
svm_rbf_dmma_kernel(const double* __restrict__ z, int n_cells, const int32_t* __restrict__ n_dev, int D,
                    int DPAD, const double* __restrict__ sv_pad, const double* __restrict__ coef,
                    const double* __restrict__ gsn, int n_tiles, double gamma, double rho,
                    double* __restrict__ dec, int8_t* __restrict__ pred, double* __restrict__ partial,
                    int partial_pitch) {
    extern __shared__ __align__(16) unsigned char svm_smem[];
    const int ZP = DPAD + 4;
    double* zs = reinterpret_cast<double*>(svm_smem);       // [GM][ZP]
    double* sb = zs + GM * ZP;                              // [2][GN][GSP]
    double* gzn = sb + 2 * GN * GSP;                        // [GM]  -gamma * ||z||^2
    double* red = gzn + GM;                                 // [4][GM]
    const int n = dev_count(n_cells, n_dev);
    const int cell0 = blockIdx.x * GM;
    if (cell0 >= n) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int gid = lane >> 2, tig = lane & 3;
    const int mg = warp & 3, ng = warp >> 2;
    const int nk = DPAD / GK;
    // blockIdx.y owns a contiguous range of SV tiles (gridDim.y > 1 when a call has too few cell
    // blocks to fill the SMs; the partial sums are added in a fixed order by svm_finalize_kernel)
    const int tiles_per = (n_tiles + gridDim.y - 1) / gridDim.y;
    const int tile_begin = blockIdx.y * tiles_per;
    const int my_tiles = max(0, min(n_tiles, tile_begin + tiles_per) - tile_begin);
    const int n_stages = my_tiles * nk;

    auto issue_sv = [&](int stage, int buf) {               // GN rows x GK doubles as 16-byte chunks
        const int tile = tile_begin + stage / nk, ks = stage % nk;
        const double* src = sv_pad + (size_t)tile * GN * DPAD + ks * GK;
        double* dst = sb + buf * GN * GSP;
        for (int idx = tid; idx < GN * (GK / 2); idx += GT) {
            const int r = idx / (GK / 2), c2 = idx - r * (GK / 2);
            const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst + r * GSP + 2 * c2);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src + (size_t)r * DPAD + 2 * c2) : "memory");
        }
    };
    if (n_stages > 0) issue_sv(0, 0);
    // the block's z rows (zero padded) and their scaled squared norms: 4 rows per warp
    for (int r = warp; r < GM; r += GT / 32) {
        const int cell = cell0 + r;
        double ss = 0.0;
        for (int d = lane; d < DPAD; d += 32) {
            const double v = (cell < n && d < D) ? z[(size_t)cell * D + d] : 0.0;
            zs[r * ZP + d] = v;
            ss = fma(v, v, ss);
        }
        ss = warp_sum(ss);
        if (lane == 0) gzn[r] = -gamma * ss;
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();

    const double g2 = 2.0 * gamma;
    const double* za0 = zs + (mg * 16 + gid) * ZP + tig;
    const double* za1 = za0 + 8 * ZP;
    const double gz0 = gzn[mg * 16 + gid], gz1 = gzn[mg * 16 + 8 + gid];
    double part0 = 0.0, part1 = 0.0;
    double acc[2][4][2];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;

    int tile = tile_begin, ks = 0;
    for (int st = 0; st < n_stages; ++st) {
        const int buf = st & 1;
        if (st + 1 < n_stages) issue_sv(st + 1, buf ^ 1);
        const double* bb = sb + buf * GN * GSP + (ng * 32 + gid) * GSP + tig;
        const double* a0p = za0 + ks * GK;
        const double* a1p = za1 + ks * GK;
#pragma unroll
        for (int k4 = 0; k4 < GK / 4; ++k4) {
            const double a0 = a0p[k4 * 4];
            const double a1 = a1p[k4 * 4];
#pragma unroll
            for (int nt = 0; nt < 4; ++nt) {
                const double b = bb[nt * 8 * GSP + k4 * 4];
                dmma884(acc[0][nt], a0, b);
                dmma884(acc[1][nt], a1, b);
            }
        }
        if (++ks == nk) {
            // fused RBF epilogue of this tile: acc[mt][nt][j] = z_cell . s_sv
            const int sv0 = tile * GN + ng * 32 + 2 * tig;
#pragma unroll
            for (int nt = 0; nt < 4; ++nt) {
                const double2 cf = __ldg(reinterpret_cast<const double2*>(coef + sv0 + nt * 8));
                const double2 gs = __ldg(reinterpret_cast<const double2*>(gsn + sv0 + nt * 8));
                part0 = fma(cf.x, exp(neg_part(fma(g2, acc[0][nt][0], gz0 + gs.x))), part0);
                part0 = fma(cf.y, exp(neg_part(fma(g2, acc[0][nt][1], gz0 + gs.y))), part0);
                part1 = fma(cf.x, exp(neg_part(fma(g2, acc[1][nt][0], gz1 + gs.x))), part1);
                part1 = fma(cf.y, exp(neg_part(fma(g2, acc[1][nt][1], gz1 + gs.y))), part1);
                acc[0][nt][0] = acc[0][nt][1] = acc[1][nt][0] = acc[1][nt][1] = 0.0;
            }
            ks = 0;
            ++tile;
        }
        asm volatile("cp.async.wait_all;" ::: "memory");
        __syncthreads();
    }
    // the 4 lanes of a quad hold different SV columns of the same two cells; then the 4 SV groups
    part0 += __shfl_xor_sync(0xffffffffu, part0, 1);
    part0 += __shfl_xor_sync(0xffffffffu, part0, 2);
    part1 += __shfl_xor_sync(0xffffffffu, part1, 1);
    part1 += __shfl_xor_sync(0xffffffffu, part1, 2);
    if (tig == 0) {
        red[ng * GM + mg * 16 + gid] = part0;
        red[ng * GM + mg * 16 + 8 + gid] = part1;
    }
    __syncthreads();
    if (tid < GM && cell0 + tid < n) {
        const double s = (red[tid] + red[GM + tid]) + (red[2 * GM + tid] + red[3 * GM + tid]);
        if (partial) {
            partial[(size_t)blockIdx.y * partial_pitch + cell0 + tid] = s;
        } else {
            dec[cell0 + tid] = s - rho;
            pred[cell0 + tid] = s - rho > 0.0 ? 1 : -1;     // svm.cpp:2841
        }
    }
}

// dec = (sum of the SV-range partial sums, in range order) - rho
__global__ void __launch_bounds__(256)
svm_finalize_kernel(const double* __restrict__ partial, int partial_pitch, int splits, int n_cells,
                    const int32_t* __restrict__ n_dev, double rho, double* __restrict__ dec,
                    int8_t* __restrict__ pred) {
    const int n = dev_count(n_cells, n_dev);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double s = 0.0;
    for (int k = 0; k < splits; ++k) s += partial[(size_t)k * partial_pitch + i];
    s -= rho;
    dec[i] = s;
    pred[i] = s > 0.0 ? 1 : -1;
}

// K6: acc[strain] += {1, cons anomalous, mod anomalous, mse, mse^2, mae, mae^2, 0}
__global__ void __launch_bounds__(256)
strain_accumulate_kernel(const cia_cell* __restrict__ cells, int n_cells,
                         const int32_t* __restrict__ n_dev, const float* __restrict__ mse,
                         const float* __restrict__ mae, const int8_t* __restrict__ pc,
                         const int8_t* __restrict__ pm, const int32_t* __restrict__ field_strain,
                         double* __restrict__ acc, int n_strains) {
    const int n = dev_count(n_cells, n_dev);
    const int lane = threadIdx.x & 31;
    for (int base = (blockIdx.x * blockDim.x + threadIdx.x) - lane; base < n; base += gridDim.x * blockDim.x) {
        const int i = base + lane;
        const bool valid = i < n;
        int strain = -1;
        double v[7] = {0, 0, 0, 0, 0, 0, 0};
        if (valid) {
            strain = field_strain ? field_strain[cells[i].field] : 0;
            if (strain < 0 || strain >= n_strains) strain = -1;
            const double a = (double)mse[i], b = (double)mae[i];
            v[0] = 1.0; v[1] = pc[i] == -1 ? 1.0 : 0.0; v[2] = pm[i] == -1 ? 1.0 : 0.0;
            v[3] = a; v[4] = a * a; v[5] = b; v[6] = b * b;
        }
        const unsigned act = __ballot_sync(0xffffffffu, strain >= 0);
        if (strain >= 0) {
            const unsigned m = __match_any_sync(act, strain);
            const int leader = __ffs(m) - 1;
#pragma unroll
            for (int k = 0; k < 7; ++k) {
                // fixed-order reduction over the group's lanes
                double s = 0.0;
                for (unsigned mm = m; mm; mm &= mm - 1) {
                    const int src = __ffs(mm) - 1;
                    s += __shfl_sync(m, v[k], src);
                }
                if (lane == leader) atomicAdd(&acc[(size_t)strain * 8 + k], s);
            }
        }
    }
}

}  // namespace

int k_svm_decision(cia_ctx* h, const float* features, int n, const int32_t* n_dev,
                   double* dec_cons, double* dec_mod, int8_t* pred_cons, int8_t* pred_mod,
                   double* pca_out, cudaStream_t s) {
    if (n <= 0) return CIA_OK;
    if (!h->sp.loaded || !h->svm[0].loaded || !h->svm[1].loaded) {
        h->err = "cia_svm_decision: scaler/pca/svm artifacts not loaded";
        return CIA_E_STATE;
    }
    const ScalerPca& sp = h->sp;
    double* z = pca_out;
    if (!z) {
        int rc = ws_reserve(h, h->ws_feat, (size_t)n * sp.C * sizeof(double));
        if (rc) return rc;
        z = (double*)h->ws_feat.p;
    }
    if (first_use(h, (const void*)svm_rbf_kernel)) {
        CIA_CUDA(cudaFuncSetAttribute(svm_rbf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        CIA_CUDA(cudaFuncSetAttribute(scaler_pca_dmma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    }
    bool pca_done = false;
    if (h->pca_kernel == 1) {                         // tensor-core projection (score_tc.cu)
        int rc = k_pca_tc(h, features, n, n_dev, z, &pca_done, s);
        if (rc) return rc;
    }
    if (!pca_done) {
        const size_t sm1 = sizeof(double) * 2 * (DM * DXP + DK * DWP);
        scaler_pca_dmma_kernel<<<dim3((n + DM - 1) / DM, sp.CP / DN), DT, sm1, s>>>(
            features, n, n_dev, sp.F, sp.C, sp.CP, sp.has_center ? sp.center : nullptr,
            sp.has_scale ? sp.scale : nullptr, sp.has_scale && sp.rscale_ok ? sp.rscale : nullptr, sp.center_is_f32, sp.comp_pad,
            sp.offset, sp.f32_flow, z);
        CIA_LAUNCH_CHECK();
    }
    for (int which = 0; which < 2; ++which) {
        const SvmModel& m = h->svm[which];
        if (m.dim != sp.C) { h->err = "svm dimension != pca components"; return CIA_E_STATE; }
        if (h->svm_kernel == 1) {
            // tensor-core GEMM form (score_tc.cu); falls through when the model is not served by it
            bool done = false;
            int rc = k_svm_tc(h, m, z, n, n_dev, which == 0 ? dec_cons : dec_mod, which == 0 ? pred_cons : pred_mod, &done, s);
            if (rc) return rc;
            if (done) continue;
        }
        const size_t sm3 = sizeof(double) * ((size_t)GM * (m.dim_pad + 4) + 2 * GN * GSP + GM + 4 * GM);
        if (sm3 <= (size_t)h->max_smem_optin) {
            if (first_use(h, (const void*)svm_rbf_dmma_kernel))
                CIA_CUDA(cudaFuncSetAttribute(svm_rbf_dmma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem_optin));
            // fill the SMs: when the call has few cell blocks, split the SV tiles over blockIdx.y
            const int bx = (n + GM - 1) / GM, n_tiles = (m.n_sv + GN - 1) / GN;
            const int per_sm = sm3 * 2 + 4096 <= (size_t)h->max_smem_optin ? 2 : 1;
            int splits = (h->num_sms * per_sm + bx - 1) / bx;
            splits = std::max(1, std::min(splits, n_tiles / 4));     // at least 4 tiles per block
            double* partial = nullptr;
            if (splits > 1) {
                int rc = ws_reserve(h, h->ws_svm, (size_t)splits * n * sizeof(double));
                if (rc) return rc;
                partial = (double*)h->ws_svm.p;
            }
            double* dec = which == 0 ? dec_cons : dec_mod;
            int8_t* pred = which == 0 ? pred_cons : pred_mod;
            svm_rbf_dmma_kernel<<<dim3(bx, splits), GT, sm3, s>>>(
                z, n, n_dev, m.dim, m.dim_pad, m.sv_pad, m.coef, m.gsn, n_tiles, m.gamma, m.rho,
                dec, pred, partial, n);
            if (splits > 1) {
                CIA_LAUNCH_CHECK();
                svm_finalize_kernel<<<(n + 255) / 256, 256, 0, s>>>(partial, n, splits, n, n_dev, m.rho, dec, pred);
            }
        } else {   // very wide feature spaces: the z tile does not fit in shared memory
            const size_t sm2 = (size_t)SCELLS * m.dim * sizeof(double);
            svm_rbf_kernel<<<(n + SCELLS - 1) / SCELLS, PT, sm2, s>>>(
                z, n, n_dev, m.dim, m.sv_t, m.coef, m.n_sv, m.n_sv_pad, m.gamma, m.rho,
                which == 0 ? dec_cons : dec_mod, which == 0 ? pred_cons : pred_mod);
        }
        CIA_LAUNCH_CHECK();
    }
    return CIA_OK;
}

int k_strain_accumulate(cia_ctx* h, const cia_cell* cells, int n, const int32_t* n_dev,
                        const cia_scores* sc, const int32_t* field_strain, double* acc,
                        int n_strains, cudaStream_t s) {
    if (n <= 0 || !acc) return CIA_OK;
    int blocks = (n + 255) / 256;
    if (blocks > h->num_sms * 8) blocks = h->num_sms * 8;
    strain_accumulate_kernel<<<blocks, 256, 0, s>>>(cells, n, n_dev, sc->mse, sc->mae,
                                                    sc->pred_conservative, sc->pred_moderate,
                                                    field_strain, acc, n_strains);
    CIA_LAUNCH_CHECK();
    return CIA_OK;
}
