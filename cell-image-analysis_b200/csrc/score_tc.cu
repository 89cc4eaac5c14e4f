// score_tc.cu -- K4 + K5 on the 5th-generation tensor cores (tcgen05, accumulators in TMEM):
// RobustScaler -> PCA projection (scaler_pca_tc_kernel, further down) and both one-class RBF SVM
// decision functions in GEMM form, ||z - s||^2 = ||z||^2 + ||s||^2 - 2 z.s^T, with the z.s^T products
// of a 128-cell x 128-SV tile as tcgen05.mma (fp16 operands split hi + lo, three MMAs per k-step) and
// the exp / dual-coefficient reduction fused into the tile epilogue (svm_rbf_tc_kernel).
//
// Replaces scaler.transform / pca.transform (improved_detection.py:134-135) and detector.predict +
// detector.decision_function (:138-142; libsvm k_function RBF, sklearn/svm/src/libsvm/svm.cpp:461-472,
// sum - rho and the sign rule :2832-2841).  The fp64 DMMA kernels in score.cu stay as the exact anchors
// (cia_set_option "svm_kernel" / "pca_kernel" = 0) and serve what these kernels do not (more than 256
// dimensions, negative dual coefficients, float64 scaler centres, feature counts not divisible by 32).
//
// Why fp16 x 3 is accurate enough for the SVM (DESIGN.md section 4.1): only the CROSS term z.s goes
// through the tensor cores; gamma||z||^2 (per cell, in the prologue) and gamma||s||^2 (per SV, at load
// time) are exact fp64.  Every row (cell) and the SV matrix are scaled by a power of two so that their
// largest element sits in [2^13, 2^14): x = hi + lo carries 22 significant bits, the dropped lo*lo term
// is 2^-22 of |z||s|.  What would err systematically is kept out of fp32:
//   * tcgen05 adds every MMA into its fp32 accumulator with round-toward-zero
//     (profiles/umma_rounding_test.cu): a 16-k-step chain under-estimates z.s by ~6e-7 relative, always in
//     the same direction for the near SVs that dominate a decision (measured: 3e-5 on the golden detectors).
//     So a TMEM accumulator only ever holds ONE pipeline stage (32 dims: the four cross-term MMAs first, the
//     two hi*hi MMAs last); the epilogue warps add the stage partials in fp32 registers with
//     round-to-nearest while the other three TMEM stage buffers fill, and the mean deficit of the two
//     remaining truncations (1.5 * 2^-25) rides on the row factor, which is an fp32 PAIR (a single fp32's
//     own rounding would be an error of the same size, common to all pairs of a detector);
//   * the per-cell term log2(e) * gamma||z||^2 is split into an integer (added to the exponent field as an
//     integer) and a fraction that multiplies the finished row sum in fp64;
//   * 2^t is a Cody-Waite reduction + degree-6 minimax polynomial in packed FFMA2 (max rel. error 1e-7,
//     mean 4e-10; ex2.approx measured 1.3e-4 in the decision at 5 000 SVs);
//   * row sums: fp32 over 32 terms, then 64-bit fixed point -- integer addition is associative, so a cell's
//     decision does not depend on how its SV tiles were cut over CTAs, i.e. on its position in the call;
//   * decisions within the kernel's error of zero are recomputed in fp64 (svm_refine_kernel).
//
// Work distribution: the (cell tile, SV tile) pairs are one flat list cut into equal contiguous
// ranges, one per CTA (one CTA per SM); a cell tile whose SV range spans several CTAs gets one
// partial sum per CTA, added by svm_tc_finalize_kernel.
//   warps 0..15 build the A operand (z tile: scale, split, K-major core matrices), then run the
//               epilogue: TMEM quadrant = warp & 3, column quarter = warp >> 2
//   warp 16     lane 0 streams the SV tiles (hi | lo images, 32 dims per stage) with cp.async.bulk
//   warps 17,18 lane 0 of each issues the MMAs of every second stage (one thread sustains ~one tcgen05.mma per
//               60 cycles plus ~90 per barrier wait; a stage is six 64-cycle MMAs); TMEM holds four stage accumulators
#include "common.cuh"
#include "tc_ptx.cuh"

#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <vector>

using namespace tcptx;

namespace {
namespace svmtc {
constexpr int EPI_WARPS = 16;
constexpr int PROD_WARP = 16, MMA_WARP = 17;     // MMA_WARP and MMA_WARP + 1 issue alternate stages
constexpr int NT = 19 * 32;
constexpr int TM = 128, TN = 128;
constexpr int KC = 32;                       // dims per pipeline stage = 2 k-steps
constexpr int K8_B = TN * 16;                // one 8-dim core-matrix column of a 128-row operand: 2 KB
constexpr int HALF_B = (KC / 8) * K8_B;      // hi (or lo) part of a stage: 8 KB
constexpr int STAGE_B = 2 * HALF_B;
constexpr int MAX_STAGES = 8;
constexpr int NBUF = 4;                      // TMEM accumulators (128 columns each), one flush group each
constexpr int FL = 2;                        // stages (of 32 dims) accumulated in TMEM between flushes
constexpr int TMEM_COLS = NBUF * TN;
constexpr int STATIC_SMEM_EST = 8 * 1024;    // barriers + per-row arrays below (host-side budget)
constexpr double LOG2E = 1.4426950408889634074;
}  // namespace svmtc

#define TMEM_LD32(taddr, v)                                                                               \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                \
                 "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"                                 \
                 "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"                \
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),     \
                   "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), \
                   "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]),           \
                   "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]),           \
                   "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])            \
                 : "r"(taddr))
#define TMEM_WAIT32(v)                                                                                    \
    asm volatile("tcgen05.wait::ld.sync.aligned;"                                                         \
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]),     \
                   "+r"(v[7]), "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), \
                   "+r"(v[14]), "+r"(v[15]), "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]),           \
                   "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]), "+r"(v[24]), "+r"(v[25]),           \
                   "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31]) :: "memory")

__device__ __forceinline__ unsigned long long add2(unsigned long long a, unsigned long long b) {
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}

// (2^(t0 + nrow), 2^(t1 + nrow)) for an integer nrow: n = rint(t) by the magic-number add, f = t - n in
// [-0.5, 0.5], degree-6 minimax polynomial in packed fp32x2 FMAs; n and nrow (pre-shifted into the
// exponent field, nsh = nrow << 23) are added to the exponent as integers.  t is clamped to
// tmin = -126 - nrow (the result underflows to ~1e-38 instead of wrapping).  Relative error <= 1.0e-7
// (fp32 Horner), mean 4e-10 (fit and figures: DESIGN.md section 4).
template <bool SLOW>
__device__ __forceinline__ void exp2x2(unsigned long long t, float tmin, float tmax, uint32_t nsh, float& r0f, float& r1f) {
    float t0, t1;
    unpack2(t, t0, t1);
    t0 = fmaxf(t0, tmin);                     // fmaxf also drops a NaN (0 * inf of a degenerate row)
    t1 = fmaxf(t1, tmin);
    if (SLOW) { t0 = fminf(t0, tmax); t1 = fminf(t1, tmax); }
    const unsigned long long tt = pack2(t0, t1);
    const unsigned long long m = add2(tt, pack2(12582912.f, 12582912.f));          // 1.5 * 2^23: n in the low mantissa bits
    const unsigned long long nf = add2(m, pack2(-12582912.f, -12582912.f));
    const unsigned long long f = fma2(nf, pack2(-1.f, -1.f), tt);                  // exact
    unsigned long long p = pack2(0.00015337577497120947f, 0.00015337577497120947f);
    p = fma2(p, f, pack2(0.0013399859890341759f, 0.0013399859890341759f));
    p = fma2(p, f, pack2(0.009618519805371761f, 0.009618519805371761f));
    p = fma2(p, f, pack2(0.05550329014658928f, 0.05550329014658928f));
    p = fma2(p, f, pack2(0.24022646248340607f, 0.24022646248340607f));
    p = fma2(p, f, pack2(0.6931471824645996f, 0.6931471824645996f));
    p = fma2(p, f, pack2(1.0f, 1.0f));
    r0f = __uint_as_float((uint32_t)p + ((uint32_t)m << 23) + nsh);
    r1f = __uint_as_float((uint32_t)(p >> 32) + ((uint32_t)(m >> 32) << 23) + nsh);
}

#ifdef CIA_SVM_TIMING
__device__ unsigned long long g_svm_dbg[16];
#define SDBG_T(var) const long long var = clock64()
#define SDBG_ADD(acc, a, b) acc += (b) - (a)
#else
#define SDBG_T(var)
#define SDBG_ADD(acc, a, b)
#endif

__global__ void __launch_bounds__(svmtc::NT, 1)
svm_rbf_tc_kernel(const double* __restrict__ z, int n_cells, const int32_t* __restrict__ n_dev, int D, int Dpad,
                  const __half* __restrict__ sv_hi, const __half* __restrict__ sv_lo,
                  const float* __restrict__ gcol, int n_svt, double fac_base, double gamma, int per_cta,
                  int stages, double fx_scale, long long* __restrict__ partial, int pitch,
                  double* __restrict__ rowmul_out) {
    using namespace svmtc;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES], tfull_bar[NBUF], tempty_bar[NBUF];
    __shared__ uint32_t tmem_base_s;
    __shared__ float s_rowfac[TM], s_rowfac_lo[TM], s_nrow[TM];
    __shared__ int s_erow[TM];
    __shared__ double s_rowmul[TM];
    __shared__ long long s_red[4][TM];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n = dev_count(n_cells, n_dev);
    const int n_ct = (n + TM - 1) / TM;
    const long long W = (long long)n_ct * n_svt;
    const long long w0 = (long long)blockIdx.x * per_cta;
    const long long w1 = W < w0 + per_cta ? W : w0 + per_cta;
    if (w0 >= W) return;                          // uniform per CTA, nothing allocated yet

    const int nk8 = Dpad >> 3;
    const int n_kc = (Dpad + KC - 1) / KC;
    const uint32_t a_half_b = (uint32_t)Dpad * 256u;          // hi (or lo) image of the z tile
    unsigned char* const a_hi = smem;
    unsigned char* const a_lo = smem + a_half_b;
    const uint32_t a_addr = smem_u32(smem);
    const uint32_t st_addr = a_addr + 2 * a_half_b;

    if (warp == MMA_WARP) tmem_alloc(&tmem_base_s, TMEM_COLS);
    if (tid == 0) {
        for (int i = 0; i < MAX_STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
        for (int i = 0; i < NBUF; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], EPI_WARPS); }
        fence_barrier_init();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    constexpr uint32_t IDESC = make_idesc(TM, TN);

    uint32_t p_st = 0, p_ph = 0;                  // producer: stage, parity of its round
    uint32_t m_st = 0, m_ph = 0, m_grp = 0;       // MMA issuers: stage ring position / parity, running flush-group count
    uint32_t e_buf = 0;                           // epilogue: running flush-group count

    for (long long w = w0; w < w1;) {
        const int ct = (int)(w / n_svt), t0 = (int)(w - (long long)ct * n_svt);
        const int nt = (int)((long long)(n_svt - t0) < w1 - w ? (long long)(n_svt - t0) : w1 - w);

        // ---------------- A operand of this cell tile ----------------
        if (warp < EPI_WARPS) {
            // (the previous segment's MMAs have completed: every epilogue warp waited on its last tile)
            asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");      // per-row arrays free
            for (int r = warp; r < TM; r += EPI_WARPS) {
                const int cell = ct * TM + r;
                double mx = 0.0, ss = 0.0;
                if (cell < n)
                    for (int d = lane; d < D; d += 32) {
                        const double v = z[(size_t)cell * D + d];
                        mx = fmax(mx, fabs(v));
                        ss = fma(v, v, ss);
                    }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                ss = warp_sum(ss);
                if (lane == 0) {
                    int e = 0;
                    if (mx > 0.0 && mx < 1e300) e = 13 - ilogb(mx);
                    e = max(-100, min(100, e));
                    const double growl = -gamma * ss * LOG2E;
                    double nr = rint(growl);
                    if (!(nr > -1048576.0)) nr = -1048576.0;            // also catches NaN / -inf rows
                    s_erow[r] = e;
                    const double fac = ldexp(fac_base, -e);         // fac_base carries the truncation compensation
                    const float fh = (float)fac;
                    s_rowfac[r] = fh;
                    s_rowfac_lo[r] = (float)(fac - (double)fh);
                    s_nrow[r] = (float)nr;
                    s_rowmul[r] = exp2(growl - nr);
                }
            }
            asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
            for (int idx = tid; idx < TM * nk8; idx += EPI_WARPS * 32) {
                const int r = idx & (TM - 1), k8 = idx >> 7;
                const int cell = ct * TM + r;
                const double sc = __hiloint2double((1023 + s_erow[r]) << 20, 0);   // 2^e, exact
                __align__(16) __half hh[8];
                __align__(16) __half ll[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int d = k8 * 8 + j;
                    const double v = (cell < n && d < D) ? z[(size_t)cell * D + d] * sc : 0.0;
                    hh[j] = __double2half(v);
                    ll[j] = __double2half(v - (double)__half2float(hh[j]));
                }
                *reinterpret_cast<uint4*>(a_hi + (size_t)idx * 16) = *reinterpret_cast<const uint4*>(hh);
                *reinterpret_cast<uint4*>(a_lo + (size_t)idx * 16) = *reinterpret_cast<const uint4*>(ll);
            }
            fence_async_smem();
        }
        __syncthreads();

        if (warp == PROD_WARP) {
            // ================= SV tile stream =================
            if (lane == 0) {
                for (int t = t0; t < t0 + nt; ++t)
                    for (int kc = 0; kc < n_kc; ++kc) {
                        mbar_wait_sleep(&empty_bar[p_st], p_ph ^ 1);
                        const int k8n = min(KC / 8, nk8 - kc * (KC / 8));
                        const uint32_t bytes = (uint32_t)k8n * K8_B;
                        const size_t off = ((size_t)t * nk8 + (size_t)kc * (KC / 8)) * (TN * 8);   // halves
                        mbar_expect_tx(&full_bar[p_st], 2 * bytes);
                        bulk_load(st_addr + p_st * STAGE_B, sv_hi + off, bytes, &full_bar[p_st]);
                        bulk_load(st_addr + p_st * STAGE_B + HALF_B, sv_lo + off, bytes, &full_bar[p_st]);
                        if (++p_st == (uint32_t)stages) { p_st = 0; p_ph ^= 1; }
                    }
            }
            __syncwarp();
        } else if (warp >= MMA_WARP) {
            // ================= MMA issuers (the whole warp runs the loop, one elected lane issues) =================
            {
                const uint32_t me = (uint32_t)(warp - MMA_WARP);
#ifdef CIA_SVM_TIMING
                long long m_tempty = 0, m_full = 0, m_issue = 0;
#endif
                const uint64_t ah0 = make_smem_desc(a_addr, K8_B, 128), al0 = make_smem_desc(a_addr + a_half_b, K8_B, 128);
                const uint64_t bh0 = make_smem_desc(st_addr, K8_B, 128), bl0 = make_smem_desc(st_addr + HALF_B, K8_B, 128);
                for (int t = t0; t < t0 + nt; ++t) {
                    // a flush group = FL consecutive stages accumulated in one TMEM buffer; the two issuing threads
                    // take alternate groups (m_st / m_ph: shared-memory stage and round parity of the group's first stage)
                    for (int g0 = 0; g0 < n_kc; g0 += FL, ++m_grp) {
                        const int gn = min(FL, n_kc - g0);
                        const uint32_t st0 = m_st, ph0 = m_ph;
                        m_st += (uint32_t)gn;
                        if (m_st >= (uint32_t)stages) { m_st -= (uint32_t)stages; m_ph ^= 1; }
                        if ((m_grp & 1) != me) continue;
                        const uint32_t buf = m_grp & (NBUF - 1);
                        uint32_t stv[FL];
                        SDBG_T(q0);
                        mbar_wait_sleep(&tempty_bar[buf], ((m_grp / NBUF) & 1) ^ 1);   // the epilogue has drained this buffer
                        SDBG_T(q1);
#pragma unroll
                        for (int u = 0; u < FL; ++u) {
                            uint32_t st = st0 + (uint32_t)u, ph = ph0;
                            if (st >= (uint32_t)stages) { st -= (uint32_t)stages; ph ^= 1; }
                            stv[u] = st;
                            if (u < gn) mbar_wait_sleep(&full_bar[st], ph);
                        }
                        SDBG_T(q2);
                        SDBG_ADD(m_tempty, q0, q1); SDBG_ADD(m_full, q1, q2);
                        tc_fence_after();
                        if (elect_one()) {
                        const uint32_t d = tmem_base + buf * TN;
                        // all cross terms (2^-11 of the product) of the group first into the fresh accumulator, the
                        // hi*hi k-steps last: only those are truncated at the sum's full magnitude
#pragma unroll
                        for (int pass = 0; pass < 2; ++pass)
#pragma unroll
                            for (int u = 0; u < FL; ++u) {
                                if (u < gn) {
                                    const int kc = g0 + u;
                                    const int ksn = min(KC / 16, (nk8 - kc * (KC / 8)) >> 1);
                                    const uint64_t ao = (uint64_t)((uint32_t)(kc * (KC / 16)) * ((2 * K8_B) >> 4));
                                    const uint64_t bo = (uint64_t)(stv[u] * (STAGE_B >> 4));
#pragma unroll
                                    for (int s = 0; s < KC / 16; ++s) {
                                        if (s < ksn) {
                                            const uint64_t so = (uint64_t)(s * ((2 * K8_B) >> 4));
                                            if (pass == 0) {
                                                umma_f16(d, ah0 + ao + so, bl0 + bo + so, IDESC, (u == 0 && s == 0) ? 0u : 1u);
                                                umma_f16(d, al0 + ao + so, bh0 + bo + so, IDESC, 1u);
                                            } else {
                                                umma_f16(d, ah0 + ao + so, bh0 + bo + so, IDESC, 1u);
                                            }
                                        }
                                    }
                                }
                            }
#pragma unroll
                        for (int u = 0; u < FL; ++u)
                            if (u < gn) umma_commit(&empty_bar[stv[u]]);
                        umma_commit(&tfull_bar[buf]);
                        }
                        __syncwarp();
                        SDBG_T(q3);
                        SDBG_ADD(m_issue, q2, q3);
                    }
                }
#ifdef CIA_SVM_TIMING
                if (me == 0 && lane == 0) {
                    atomicAdd(&g_svm_dbg[0], (unsigned long long)m_tempty); atomicAdd(&g_svm_dbg[1], (unsigned long long)m_full);
                    atomicAdd(&g_svm_dbg[2], (unsigned long long)m_issue);
                }
#endif
            }
            __syncwarp();
        } else {
            // ================= epilogue: fused RBF + dual-coefficient reduction =================
            const int q = warp & 3, cq = warp >> 2, row = 32 * q + lane;
            const float rf = s_rowfac[row], rfl = s_rowfac_lo[row], nrw = s_nrow[row];
            const unsigned long long rf2 = pack2(rf, rf), rfl2 = pack2(rfl, rfl);
            // 2^(t + nrow): nrow goes into the exponent field as an integer; rows whose nrow is beyond the
            // fp32 exponent range contribute 2^-126-ish terms (their kernel values are < 1e-38 anyway)
            const float nrc = fminf(fmaxf(nrw, -250.f), 120.f);
            const float tmin = -126.f - nrc, tmax = 126.f - nrc;
            const uint32_t nsh = (uint32_t)((int)nrc) << 23;
            // far outliers (log2e * gamma||z||^2 beyond the fp32 exponent range): the rest of n_row is added to t
            // in fp32 and t is clamped on both sides -- a warp-uniform slow path, one more FADD2 per pair
            const float rem = nrw - nrc;
            const unsigned long long rem2 = pack2(rem, rem);
            const bool slow = __any_sync(0xffffffffu, rem != 0.f);
            const uint32_t taddr0 = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(cq * 32);
#ifdef CIA_SVM_TIMING
            long long e_wait = 0, e_flush = 0, e_exp = 0, e_tiles = 0;
#endif
            // row sums in 64-bit FIXED POINT (2^-S, S from the model): integer addition is associative, so a cell's
            // decision does not depend on how its SV tiles were cut over CTAs, i.e. on its position in the call
            long long rowsum = 0;
            for (int t = t0; t < t0 + nt; ++t) {
                // ---- z.s of this tile: the stage partials added in fp32 registers, round to nearest ----
                float acc[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[j] = 0.f;
#pragma unroll 1
                for (int g0 = 0; g0 < n_kc; g0 += FL, ++e_buf) {
                    const uint32_t buf = e_buf & (NBUF - 1);
                    SDBG_T(w0);
                    mbar_wait_sleep(&tfull_bar[buf], (e_buf / NBUF) & 1);
                    SDBG_T(w1);
                    SDBG_ADD(e_wait, w0, w1);
                    tc_fence_after();
                    uint32_t v[32];
                    TMEM_LD32(taddr0 + buf * TN, v);
                    TMEM_WAIT32(v);
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&tempty_bar[buf]);
#pragma unroll
                    for (int j = 0; j < 32; j += 2) fadd2(acc[j], acc[j + 1], v[j], v[j + 1]);
                    SDBG_T(w2);
                    SDBG_ADD(e_flush, w1, w2);
                }
                SDBG_T(x0);
                // ---- fused RBF + dual-coefficient reduction ----
                // t = acc * (2 gamma log2e 2^-(e_row + e_s)) + (log2e * -gamma||s||^2 + log2 coef)  [+ n_row]
                const float4* gc = reinterpret_cast<const float4*>(gcol + (size_t)t * TN + cq * 32);
                float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
                if (!slow) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const float4 g = __ldg(gc + (j >> 2));
                        const unsigned long long a01 = pack2(acc[j], acc[j + 1]), a23 = pack2(acc[j + 2], acc[j + 3]);
                        const unsigned long long ta = fma2(a01, rf2, fma2(a01, rfl2, pack2(g.x, g.y)));
                        const unsigned long long tb = fma2(a23, rf2, fma2(a23, rfl2, pack2(g.z, g.w)));
                        float e0, e1, e2, e3;
                        exp2x2<false>(ta, tmin, tmax, nsh, e0, e1);
                        exp2x2<false>(tb, tmin, tmax, nsh, e2, e3);
                        s0 += e0; s1 += e1; s2 += e2; s3 += e3;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const float4 g = __ldg(gc + (j >> 2));
                        const unsigned long long a01 = pack2(acc[j], acc[j + 1]), a23 = pack2(acc[j + 2], acc[j + 3]);
                        const unsigned long long ta = add2(fma2(a01, rf2, fma2(a01, rfl2, pack2(g.x, g.y))), rem2);
                        const unsigned long long tb = add2(fma2(a23, rf2, fma2(a23, rfl2, pack2(g.z, g.w))), rem2);
                        float e0, e1, e2, e3;
                        exp2x2<true>(ta, tmin, tmax, nsh, e0, e1);
                        exp2x2<true>(tb, tmin, tmax, nsh, e2, e3);
                        s0 += e0; s1 += e1; s2 += e2; s3 += e3;
                    }
                }
                rowsum += __double2ll_rn((double)((s0 + s1) + (s2 + s3)) * fx_scale);
                SDBG_T(x1);
                SDBG_ADD(e_exp, x0, x1);
#ifdef CIA_SVM_TIMING
                ++e_tiles;
#endif
            }
#ifdef CIA_SVM_TIMING
            if (tid == 0) {
                atomicAdd(&g_svm_dbg[4], (unsigned long long)e_wait); atomicAdd(&g_svm_dbg[5], (unsigned long long)e_flush);
                atomicAdd(&g_svm_dbg[6], (unsigned long long)e_exp); atomicAdd(&g_svm_dbg[7], (unsigned long long)e_tiles);
            }
#endif
            s_red[cq][row] = rowsum;
            asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
            if (cq == 0) {
                const int cell = ct * TM + row;
                if (cell < n) {
                    const int first_cta = (int)(((long long)ct * n_svt) / per_cta);
                    partial[(size_t)((int)blockIdx.x - first_cta) * pitch + cell] =
                        (s_red[0][row] + s_red[1][row]) + (s_red[2][row] + s_red[3][row]);
                    rowmul_out[cell] = s_rowmul[row];          // the same value from every CTA that shares the cell tile
                }
            }
        }
        w += nt;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == svmtc::MMA_WARP) tmem_dealloc(tmem_base, svmtc::TMEM_COLS);
}

// dec = (partial sums of the CTAs that shared this cell tile, in CTA order) - rho
__global__ void __launch_bounds__(256)
svm_tc_finalize_kernel(const long long* __restrict__ partial, int pitch, int n_svt, int per_cta, int n_cells,
                       const int32_t* __restrict__ n_dev, const double* __restrict__ rowmul, double fx_inv, double rho,
                       double* __restrict__ dec, int8_t* __restrict__ pred) {
    const int n = dev_count(n_cells, n_dev);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long ct = i / svmtc::TM;
    const int first = (int)((ct * n_svt) / per_cta), last = (int)(((ct + 1) * n_svt - 1) / per_cta);
    long long t = 0;
    for (int k = 0; k <= last - first; ++k) t += partial[(size_t)k * pitch + i];
    const double s = (double)t * fx_inv * rowmul[i] - rho;
    dec[i] = s;
    pred[i] = s > 0.0 ? 1 : -1;                    // svm.cpp:2841
}

// ---------------------------------------------------------------------------------------------
// K4 on the tensor cores: RobustScaler -> PCA projection, z = x2 @ components^T - offset.
//
// M = 128 cells, N = 128 components (blockIdx.y walks wider PCAs), K = the 2048 encoder features in
// stages of 32.  The A operand cannot be copied, it has to be COMPUTED: four producer warps (one
// thread per cell row) read the raw float32 features, apply the scaler exactly as sklearn's in-place
// float32 flow does (x1 = f32(x - center), x2 = f32(f64(x1) / scale), the division as reciprocal +
// exact-remainder FMA, bit-identical to the DMMA kernel in score.cu), scale the row's 32 values by a
// power of two so that the largest sits in [2^13, 2^14), split them into fp16 hi + lo and store them
// as K-major core matrices; the power of two goes to the epilogue through a small ring.  The
// components arrive pre-split ([stage][hi | lo][4][128][8]) by cp.async.bulk.  Per stage six MMAs
// (cross terms first, hi*hi last) fill one of four TMEM accumulators; eight epilogue warps add the
// stage partial, times the row's power of two, into fp32 registers with round-to-nearest (FFMA2) --
// tcgen05's own accumulation truncates (see above) -- and finish with sklearn's float32 subtraction
// of the offset.  Error against the exactly rounded projection: ~2e-7 of |z| (the oracle's own
// float32 sgemm is at 7e-7), tests/test_gpu_svm_tc.py.
// ---------------------------------------------------------------------------------------------
namespace pcatc {
constexpr int PROD_WARPS = 8, EPI_WARPS = 8;            // producers: two groups of four warps, alternate stages
constexpr int EPI_WARP0 = PROD_WARPS;
constexpr int MMA_WARP = PROD_WARPS + EPI_WARPS;        // and MMA_WARP + 1: alternate stages
constexpr int BULK_WARP = MMA_WARP + 2;
constexpr int NT = (BULK_WARP + 1) * 32;
constexpr int TM = 128, TN = 128, KC = 32;
constexpr int K8_B = 128 * 16;
constexpr int HALF_B = (KC / 8) * K8_B;                 // 8 KB: hi (or lo) of one operand stage
constexpr int STAGE_B = 4 * HALF_B;                     // A hi | A lo | B hi | B lo
constexpr int STAGES = 4;
constexpr int NBUF = 4;
constexpr int RING = 16;                                // row-scale ring (>= STAGES + NBUF stages in flight)
constexpr int PAR_F = 2048;                             // scaler constants of up to this many features live in shared memory
constexpr int SMEM_B = STAGES * STAGE_B + RING * TM * 4 + PAR_F * 16;
}  // namespace pcatc

__global__ void __launch_bounds__(pcatc::NT, 1)
scaler_pca_tc_kernel(const float* __restrict__ feat, int n_cells, const int32_t* __restrict__ n_dev, int F, int C,
                     const float4* __restrict__ par_g /* {center, RN(1/scale), scale hi, scale lo} per feature */,
                     const __half* __restrict__ comp_img,
                     float w_unscale, const double* __restrict__ offset, int f32_flow, double* __restrict__ z_out) {
    using namespace pcatc;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t full_bar[STAGES], empty_bar[STAGES], tfull_bar[NBUF], tempty_bar[NBUF];
    __shared__ uint32_t tmem_base_s;
    float* const ring = reinterpret_cast<float*>(smem + STAGES * STAGE_B);      // [RING][TM]
    float4* const par = reinterpret_cast<float4*>(smem + STAGES * STAGE_B + RING * TM * 4);   // scaler constants

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n = dev_count(n_cells, n_dev);
    const int n_ct = (n + TM - 1) / TM;
    if ((int)blockIdx.x >= n_ct) return;
    const int n_kc = F / KC;                                  // F is a multiple of 32 (host checks)
    const int cb = blockIdx.y;                                // component block of 128
    const uint32_t s_addr = smem_u32(smem);
    const bool par_s = F <= PAR_F;                            // scaler constants staged in shared memory

    if (warp == MMA_WARP) tmem_alloc(&tmem_base_s, NBUF * TN);
    if (tid == 0) {
        for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], PROD_WARPS / 2 + 1); mbar_init(&empty_bar[i], 1); }
        for (int i = 0; i < NBUF; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], EPI_WARPS); }
        fence_barrier_init();
    }
    if (par_s)
        for (int i = tid; i < F; i += NT) par[i] = __ldg(par_g + i);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    constexpr uint32_t IDESC = make_idesc(TM, TN);

    uint32_t cnt = 0;                                         // running stage count of this CTA (every role keeps its own copy)
    if (warp < PROD_WARPS) {
        // ================= A producers: scaler + power-of-two scaling + hi/lo split =================
        // a warp owns 32 cell rows of the tile, 32 features per stage.  Loads are coalesced: instruction i of a lane
        // reads row 4i + lane/8, features 4(lane%8)..+3 (8 lanes = one 128-byte line; a thread-per-row layout costs
        // 32 L1 wavefronts per instruction and bound the kernel at ~1000 cycles a stage).  The two groups of four
        // warps take alternate stages and every thread fetches its NEXT stage before it works on the current one.
        const int grp = warp >> 2, r0 = 32 * (warp & 3) + (lane >> 3), ch = lane & 7;
        const long long total = (long long)((n_ct - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x) * n_kc;   // stages of this CTA
        auto fetch = [&](long long sidx, float4 (&x)[8]) {
            const int ct = (int)blockIdx.x + (int)(sidx / n_kc) * (int)gridDim.x, kc = (int)(sidx % n_kc);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int cell = ct * TM + r0 + 4 * i;
                x[i] = (sidx < total && cell < n)
                           ? __ldg(reinterpret_cast<const float4*>(feat + (size_t)cell * F + kc * KC) + ch)
                           : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        };
        float4 xn[8];
        fetch(grp, xn);
        for (long long sidx = grp; sidx < total; sidx += 2) {
            const uint32_t c = (uint32_t)sidx, st = c % STAGES;
            const int kc = (int)(sidx % n_kc);
            float4 x[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) x[i] = xn[i];
            fetch(sidx + 2, xn);
            // RobustScaler in fp32 only (fp64 conversions run at a fraction of the fp32 rate and bound this kernel
            // otherwise): x1 = RN(x - center) as sklearn's float32 subtraction; x2 = RN(x1 / scale) with the float64
            // scale as an fp32 pair: q = RN(x1 * RN(1/scale)) is within an ulp, x1 - q * scale_hi is exact in one FMA,
            // the scale_lo part and the final fma(rem, 1/scale, q) follow -- the correctly rounded quotient except
            // within 2^-49 of a rounding boundary (1 element in ~10^7 differs by an ulp from the float64 division)
            float4 pf[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) pf[k] = par_s ? par[kc * KC + 4 * ch + k] : __ldg(par_g + kc * KC + 4 * ch + k);
            auto scaler = [](float xv, const float4& p) {
                const float x1 = __fsub_rn(xv, p.x);
                const float q = __fmul_rn(x1, p.y);
                const float rem = __fmaf_rn(-q, p.w, __fmaf_rn(-q, p.z, x1));
                return __fmaf_rn(rem, p.y, q);
            };
            float up[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                x[i].x = scaler(x[i].x, pf[0]); x[i].y = scaler(x[i].y, pf[1]);
                x[i].z = scaler(x[i].z, pf[2]); x[i].w = scaler(x[i].w, pf[3]);
                // (a NaN feature is dropped by fmaxf here and comes back through hi)
                float mx = fmaxf(fmaxf(fabsf(x[i].x), fabsf(x[i].y)), fmaxf(fabsf(x[i].z), fabsf(x[i].w)));
                mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
                mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
                mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 4));
                // 2^e with the largest |x2| of the row's stage in [2^13, 2^14); e in [-100, 100]
                int e = 0;
                if (mx > 0.f && mx < 3e38f) e = 13 - (int)((__float_as_uint(mx) >> 23) & 0xFF) + 127;
                e = max(-100, min(100, e));
                up[i] = __uint_as_float((uint32_t)(127 + e) << 23);
            }
            mbar_wait_sleep(&empty_bar[st], ((c / STAGES) & 1) ^ 1);
            unsigned char* a_hi = smem + st * STAGE_B + ((ch >> 1) * TM) * 16 + (ch & 1) * 8;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int r = r0 + 4 * i;
                const float v0 = x[i].x * up[i], v1 = x[i].y * up[i], v2 = x[i].z * up[i], v3 = x[i].w * up[i];   // exact
                const __half2 h01 = __floats2half2_rn(v0, v1), h23 = __floats2half2_rn(v2, v3);
                const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
                const __half2 l01 = __floats2half2_rn(v0 - f01.x, v1 - f01.y), l23 = __floats2half2_rn(v2 - f23.x, v3 - f23.y);
                *reinterpret_cast<uint2*>(a_hi + r * 16) = make_uint2(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23));
                *reinterpret_cast<uint2*>(a_hi + HALF_B + r * 16) = make_uint2(*reinterpret_cast<const uint32_t*>(&l01), *reinterpret_cast<const uint32_t*>(&l23));
                if (ch == 0) ring[(c % RING) * TM + r] = __uint_as_float(0x7F000000u - __float_as_uint(up[i])) * w_unscale;   // 2^-e, exact
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&full_bar[st]);
        }
    } else
    for (int ct = blockIdx.x; ct < n_ct; ct += gridDim.x) {
        if (warp == BULK_WARP) {
            // ================= component stream =================
            if (lane == 0) {
                for (int kc = 0; kc < n_kc; ++kc, ++cnt) {
                    const uint32_t st = cnt % STAGES;
                    mbar_wait_sleep(&empty_bar[st], ((cnt / STAGES) & 1) ^ 1);
                    mbar_expect_tx(&full_bar[st], 2 * HALF_B);
                    bulk_load(s_addr + st * STAGE_B + 2 * HALF_B, comp_img + ((size_t)cb * n_kc + kc) * (2 * HALF_B / 2),
                              2 * HALF_B, &full_bar[st]);
                }
            }
            __syncwarp();
        } else if (warp >= MMA_WARP) {
            // ================= MMA issuers (alternate stages; the whole warp runs the loop, one elected lane issues) =================
            {
                const uint32_t me = (uint32_t)(warp - MMA_WARP);
                const uint64_t d0 = make_smem_desc(s_addr, K8_B, 128);
                for (int kc = 0; kc < n_kc; ++kc, ++cnt) {
                    if ((cnt & 1) != me) continue;
                    const uint32_t st = cnt % STAGES, buf = cnt % NBUF;
                    mbar_wait_sleep(&tempty_bar[buf], ((cnt / NBUF) & 1) ^ 1);
                    mbar_wait_sleep(&full_bar[st], (cnt / STAGES) & 1);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t d = tmem_base + buf * TN;
                        const uint64_t ah = d0 + (uint64_t)((st * STAGE_B) >> 4), al = ah + (HALF_B >> 4);
                        const uint64_t bh = ah + (2 * HALF_B >> 4), bl = ah + (3 * HALF_B >> 4);
#pragma unroll
                        for (int s = 0; s < KC / 16; ++s) {
                            const uint64_t so = (uint64_t)(s * ((2 * K8_B) >> 4));
                            umma_f16(d, ah + so, bl + so, IDESC, s == 0 ? 0u : 1u);
                            umma_f16(d, al + so, bh + so, IDESC, 1u);
                        }
#pragma unroll
                        for (int s = 0; s < KC / 16; ++s) {
                            const uint64_t so = (uint64_t)(s * ((2 * K8_B) >> 4));
                            umma_f16(d, ah + so, bh + so, IDESC, 1u);
                        }
                        umma_commit(&empty_bar[st]);
                        umma_commit(&tfull_bar[buf]);
                    }
                    __syncwarp();
                }
            }
        } else {
            // ================= epilogue: fp32 round-to-nearest accumulation of the stage partials =================
            const int ew = warp - EPI_WARP0, q = ew & 3, hf = ew >> 2, row = 32 * q + lane;
            const uint32_t taddr0 = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(hf * 64);
            unsigned long long acc[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[j] = 0ull;
#pragma unroll 1
            for (int kc = 0; kc < n_kc; ++kc, ++cnt) {
                const uint32_t buf = cnt % NBUF;
                mbar_wait_sleep(&tfull_bar[buf], (cnt / NBUF) & 1);
                tc_fence_after();
                const float sc = ring[(cnt % RING) * TM + row];
                const unsigned long long sc2 = pack2(sc, sc);
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    uint32_t v[16];
                    TMEM_LD16(taddr0 + buf * TN + (uint32_t)(b * 16), v);
                    TMEM_WAIT16(v);
                    if (b == 3) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&tempty_bar[buf]);
                    }
#pragma unroll
                    for (int j = 0; j < 16; j += 2)
                        acc[b * 8 + (j >> 1)] = fma2(pack2(__uint_as_float(v[j]), __uint_as_float(v[j + 1])), sc2, acc[b * 8 + (j >> 1)]);
                }
            }
            const int cell = ct * TM + row;
            if (cell < n) {
                // the two full-magnitude truncations of a stage's hi*hi MMAs: mean deficit 1.5 * 2^-25
                constexpr double DEBIAS = 1.0 + 1.5 * 2.9802322387695312e-8;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    float a0, a1;
                    unpack2(acc[j], a0, a1);
                    const int c = cb * TN + hf * 64 + 2 * j;
                    if (c < C) {
                        const double off = __ldg(offset + c), v = (double)a0 * DEBIAS;
                        z_out[(size_t)cell * C + c] = f32_flow ? (double)__fsub_rn((float)v, (float)off) : __dsub_rn(v, off);
                    }
                    if (c + 1 < C) {
                        const double off = __ldg(offset + c + 1), v = (double)a1 * DEBIAS;
                        z_out[(size_t)cell * C + c + 1] = f32_flow ? (double)__fsub_rn((float)v, (float)off) : __dsub_rn(v, off);
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == pcatc::MMA_WARP) tmem_dealloc(tmem_base, pcatc::NBUF * pcatc::TN);
}

// Exact re-evaluation of the decisions the fp16 x 3 kernel cannot sign with certainty.  Its error is a
// few 2^-24 of the kernel sum (the z tile keeps 22 of the 24 significand bits of the float32 PCA scores,
// and that rounding is common to all SVs of a row: measured 6e-5 at 20 000 SVs with sum(coef) = 2e4, 1e-6
// at the golden detectors), so a decision with |dec| < thr_abs + thr_rel * (dec + rho) is recomputed in
// fp64 with direct differences -- libsvm's own arithmetic, svm.cpp:461-472 -- by a whole block, its SV
// partial sums added in a fixed order.  Such cells are rare (~1e-5 of a screen); the scan costs 8 bytes a cell.
__global__ void __launch_bounds__(256)
svm_refine_kernel(const double* __restrict__ z, int n_cells, const int32_t* __restrict__ n_dev, int D,
                  const double* __restrict__ sv_t, const double* __restrict__ coef, int n_sv, int n_sv_pad,
                  double gamma, double rho, double thr_abs, double thr_rel, double* __restrict__ dec,
                  int8_t* __restrict__ pred) {
    extern __shared__ double zrow[];             // [D]
    __shared__ int s_list[256];
    __shared__ int s_count;
    __shared__ double s_part[8];
    const int n = dev_count(n_cells, n_dev);
    const int tid = threadIdx.x;
    for (int base = blockIdx.x * 256; base < n; base += gridDim.x * 256) {
        if (tid == 0) s_count = 0;
        __syncthreads();
        const int c = base + tid;
        if (c < n) {
            const double d = dec[c];
            if (fabs(d) < thr_abs + thr_rel * fabs(d + rho)) s_list[atomicAdd(&s_count, 1)] = c;
        }
        __syncthreads();
        const int cnt = s_count;
        for (int k = 0; k < cnt; ++k) {
            const int cell = s_list[k];          // (the order of the list does not matter: cells are independent)
            for (int d = tid; d < D; d += 256) zrow[d] = z[(size_t)cell * D + d];
            __syncthreads();
            double part = 0.0;
            for (int i = tid; i < n_sv; i += 256) {
                double d2 = 0.0;
                for (int d = 0; d < D; ++d) {
                    const double df = zrow[d] - __ldg(sv_t + (size_t)d * n_sv_pad + i);
                    d2 = fma(df, df, d2);
                }
                part = fma(coef[i], exp(-gamma * d2), part);
            }
            part = warp_sum(part);
            if ((tid & 31) == 0) s_part[tid >> 5] = part;
            __syncthreads();
            if (tid == 0) {
                double sum = 0.0;
                for (int w = 0; w < 8; ++w) sum += s_part[w];
                sum -= rho;
                dec[cell] = sum;
                pred[cell] = sum > 0.0 ? 1 : -1;
            }
            __syncthreads();
        }
    }
}

}  // namespace

// Operand images of one detector for svm_rbf_tc_kernel (called from cia_load_svm): support vectors
// scaled by 2^e_s and split hi + lo, as [SV tile of 128][dim / 8][128][8 halves] (the K-major
// core-matrix order a tile's bulk copy lands in); gcol[i] = log2(e) * -gamma||s_i||^2 + log2(coef_i).
int k_svm_tc_prepare(cia_ctx* h, SvmModel& m, const double* sv, const double* coef) {
    m.tc_ok = false;
    cudaFree(m.tc_hi); cudaFree(m.tc_lo); cudaFree(m.tc_gcol);
    m.tc_hi = m.tc_lo = nullptr; m.tc_gcol = nullptr;
    if (m.dim_pad > 256) return CIA_OK;              // the z tile (hi + lo) would not fit in shared memory
    double mx = 0.0;
    for (size_t i = 0; i < (size_t)m.n_sv * m.dim; ++i) {
        if (!std::isfinite(sv[i])) return CIA_OK;
        mx = std::fmax(mx, std::fabs(sv[i]));
    }
    for (int i = 0; i < m.n_sv; ++i)
        if (!(coef[i] >= 0.0) || !std::isfinite(coef[i])) return CIA_OK;   // one-class duals are >= 0; anything else: DMMA path
    const int es = mx > 0.0 ? 13 - std::ilogb(mx) : 0;
    if (es < -100 || es > 100) return CIA_OK;
    const int n_svt = (m.n_sv + svmtc::TN - 1) / svmtc::TN, nk8 = m.dim_pad / 8;
    std::vector<__half> hi((size_t)n_svt * nk8 * svmtc::TN * 8, __float2half_rn(0.f)), lo = hi;
    std::vector<float> g((size_t)n_svt * svmtc::TN, -1e30f);
    for (int i = 0; i < m.n_sv; ++i) {
        const int t = i / svmtc::TN, r = i % svmtc::TN;
        double ss = 0.0;
        for (int d = 0; d < m.dim; ++d) {
            const double v0 = sv[(size_t)i * m.dim + d];
            ss += v0 * v0;
            const double v = std::ldexp(v0, es);
            const __half hv = __double2half(v);
            const size_t idx = (((size_t)t * nk8 + d / 8) * svmtc::TN + r) * 8 + (d % 8);
            hi[idx] = hv;
            lo[idx] = __double2half(v - (double)__half2float(hv));
        }
        if (coef[i] > 0.0) g[i] = (float)(svmtc::LOG2E * (-m.gamma * ss) + std::log2(coef[i]));
    }
    CIA_CUDA(cudaMalloc(&m.tc_hi, hi.size() * sizeof(__half)));
    CIA_CUDA(cudaMalloc(&m.tc_lo, lo.size() * sizeof(__half)));
    CIA_CUDA(cudaMalloc(&m.tc_gcol, g.size() * sizeof(float)));
    CIA_CUDA(cudaMemcpy(m.tc_hi, hi.data(), hi.size() * sizeof(__half), cudaMemcpyHostToDevice));
    CIA_CUDA(cudaMemcpy(m.tc_lo, lo.data(), lo.size() * sizeof(__half), cudaMemcpyHostToDevice));
    CIA_CUDA(cudaMemcpy(m.tc_gcol, g.data(), g.size() * sizeof(float), cudaMemcpyHostToDevice));
    // fixed-point exponent of the row sums: sum_i coef_i K_i <= n_sv * max coef, kept below 2^61
    double amax = 1.0;
    for (int i = 0; i < m.n_sv; ++i) amax = std::fmax(amax, coef[i]);
    m.tc_fx = std::max(0, std::min(50, 60 - (int)std::ceil(std::log2((double)n_svt * svmtc::TN * amax))));
    m.tc_es = es;
    m.tc_svt = n_svt;
    m.tc_ok = true;
    return CIA_OK;
}

// returns CIA_OK and sets *done = false when this model / size is not served by the tensor-core kernel
int k_svm_tc(cia_ctx* h, const SvmModel& m, const double* z, int n, const int32_t* n_dev, double* dec,
             int8_t* pred, bool* done, cudaStream_t s) {
    using namespace svmtc;
    *done = false;
    if (!m.tc_ok) return CIA_OK;
    const int a_bytes = 2 * m.dim_pad * 256;
    int stages = (h->max_smem_optin - STATIC_SMEM_EST - a_bytes) / STAGE_B;
    if (stages < 3) return CIA_OK;
    stages = std::min(stages, MAX_STAGES);
    const int smem_b = a_bytes + stages * STAGE_B;
    auto kern = svm_rbf_tc_kernel;
    if (first_use(h, (const void*)kern))
        CIA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem_optin - STATIC_SMEM_EST));
    const int n_ct = (n + TM - 1) / TM;
    const long long W = (long long)n_ct * m.tc_svt;
    // equal contiguous ranges of (cell tile, SV tile) pairs, one CTA per SM; a range never shorter than 2
    // pairs (each range pays one A-operand build)
    int per_cta = (int)((W + h->num_sms - 1) / h->num_sms);
    per_cta = std::max(per_cta, std::min(2, m.tc_svt));
    const int grid = (int)((W + per_cta - 1) / per_cta);
    const int slots = (m.tc_svt + per_cta - 1) / per_cta + 1;
    int rc = ws_reserve(h, h->ws_svm, (size_t)(slots + 1) * n * sizeof(double));
    if (rc) return rc;
    long long* partial = (long long*)h->ws_svm.p;
    double* rowmul = (double*)h->ws_svm.p + (size_t)slots * n;
    // mean deficit of the full-magnitude round-toward-zero accumulations of a flush group, in units of 2^-25
    // (a flush group is FL = 2 stages = four hi*hi k-steps whose running sum is truncated four times:
    // (1/4 + 2/4 + 3/4 + 1) = 2.5 mean truncations of the group sum)
    constexpr double debias = 2.5;
    const double fac_base = std::ldexp(2.0 * m.gamma * LOG2E, -m.tc_es) * (1.0 + debias * 2.9802322387695312e-8);
    kern<<<grid, NT, smem_b, s>>>(z, n, n_dev, m.dim, m.dim_pad, (const __half*)m.tc_hi, (const __half*)m.tc_lo, m.tc_gcol, m.tc_svt, fac_base,
                                  m.gamma, per_cta, stages, std::ldexp(1.0, m.tc_fx), partial, n, rowmul);
    CIA_LAUNCH_CHECK();
#ifdef CIA_SVM_TIMING
    if (getenv("CIA_SVM_DUMP")) {
        unsigned long long d[16];
        cudaStreamSynchronize(s);
        cudaMemcpyFromSymbol(d, g_svm_dbg, sizeof(d));
        const double u = d[7] ? (double)d[7] : 1.0;      // tiles seen by thread 0 of every CTA
        fprintf(stderr, "svm_tc per tile (cycles): mma thread 0 {wait tmem-empty %.0f, wait smem-full %.0f, issue %.0f} x2 threads; "
                        "epilogue warp 0 {wait tmem-full %.0f, flush %.0f, exp %.0f}; tiles %llu\n",
                d[0] / u, d[1] / u, d[2] / u, d[4] / u, d[5] / u, d[6] / u, d[7]);
        memset(d, 0, sizeof(d));
        cudaMemcpyToSymbol(g_svm_dbg, d, sizeof(d));
    }
#endif
    svm_tc_finalize_kernel<<<(n + 255) / 256, 256, 0, s>>>(partial, n, m.tc_svt, per_cta, n, n_dev, rowmul,
                                                             std::ldexp(1.0, -m.tc_fx), m.rho, dec, pred);
    CIA_LAUNCH_CHECK();
    if (h->svm_refine) {
        int blocks = std::min((n + 255) / 256, h->num_sms * 4);
        svm_refine_kernel<<<blocks, 256, m.dim * sizeof(double), s>>>(z, n, n_dev, m.dim, m.sv_t, m.coef, m.n_sv, m.n_sv_pad, m.gamma,
                                                                     m.rho, 2e-4, 4e-7, dec, pred);
        CIA_LAUNCH_CHECK();
    }
    *done = true;
    return CIA_OK;
}

// Operand image of the PCA components for scaler_pca_tc_kernel (called from cia_load_scaler_pca): scaled by
// 2^e_w, split hi + lo, as [component block of 128][stage of 32 features][hi | lo][feature / 8][128][8].
int k_pca_tc_prepare(cia_ctx* h, ScalerPca& sp, const double* components /* [C][F] */) {
    sp.tc_ok = false;
    cudaFree(sp.tc_img); sp.tc_img = nullptr;
    cudaFree(sp.tc_par); sp.tc_par = nullptr;
    if (sp.F % pcatc::KC != 0) return CIA_OK;
    // the kernel's fp32 scaler: float32 centre (sklearn fit on float32 features) and scale / 1/scale as fp32 pairs
    if (sp.has_center && !sp.center_is_f32) return CIA_OK;
    if (sp.has_scale && !sp.rscale_ok) return CIA_OK;
    double mx = 0.0;
    for (size_t i = 0; i < (size_t)sp.C * sp.F; ++i) {
        if (!std::isfinite(components[i])) return CIA_OK;
        mx = std::fmax(mx, std::fabs(components[i]));
    }
    const int ew = mx > 0.0 ? 13 - std::ilogb(mx) : 0;
    if (ew < -20 || ew > 20) return CIA_OK;
    const int ncb = (sp.C + pcatc::TN - 1) / pcatc::TN, n_kc = sp.F / pcatc::KC;
    std::vector<__half> img((size_t)ncb * n_kc * 2 * (pcatc::KC / 8) * pcatc::TN * 8, __float2half_rn(0.f));
    for (int c = 0; c < sp.C; ++c)
        for (int f = 0; f < sp.F; ++f) {
            const double v = std::ldexp(components[(size_t)c * sp.F + f], ew);
            const __half hv = __double2half(v);
            const int cbk = c / pcatc::TN, cr = c % pcatc::TN, kc = f / pcatc::KC, k8 = (f % pcatc::KC) / 8;
            const size_t base = ((size_t)cbk * n_kc + kc) * 2 * (pcatc::KC / 8) * pcatc::TN * 8;
            const size_t idx = ((size_t)k8 * pcatc::TN + cr) * 8 + (f % 8);
            img[base + idx] = hv;
            img[base + (size_t)(pcatc::KC / 8) * pcatc::TN * 8 + idx] = __double2half(v - (double)__half2float(hv));
        }
    CIA_CUDA(cudaMalloc(&sp.tc_img, img.size() * sizeof(__half)));
    CIA_CUDA(cudaMemcpy(sp.tc_img, img.data(), img.size() * sizeof(__half), cudaMemcpyHostToDevice));
    {
        std::vector<double> cen((size_t)sp.F, 0.0), sc((size_t)sp.F, 1.0);
        if (sp.has_center) CIA_CUDA(cudaMemcpy(cen.data(), sp.center, sp.F * sizeof(double), cudaMemcpyDeviceToHost));
        if (sp.has_scale) CIA_CUDA(cudaMemcpy(sc.data(), sp.scale, sp.F * sizeof(double), cudaMemcpyDeviceToHost));
        std::vector<float> par((size_t)sp.F * 4);
        for (int f = 0; f < sp.F; ++f) {
            const float shi = (float)sc[f];
            par[4 * f + 0] = (float)cen[f];
            par[4 * f + 1] = (float)(1.0 / sc[f]);
            par[4 * f + 2] = shi;
            par[4 * f + 3] = (float)(sc[f] - (double)shi);
            if (!std::isnormal(shi) || !std::isnormal(par[4 * f + 1])) { cudaFree(sp.tc_img); sp.tc_img = nullptr; return CIA_OK; }
        }
        CIA_CUDA(cudaMalloc(&sp.tc_par, par.size() * sizeof(float)));
        CIA_CUDA(cudaMemcpy(sp.tc_par, par.data(), par.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    sp.tc_ew = ew;
    sp.tc_ok = true;
    return CIA_OK;
}

int k_pca_tc(cia_ctx* h, const float* features, int n, const int32_t* n_dev, double* z, bool* done, cudaStream_t s) {
    using namespace pcatc;
    const ScalerPca& sp = h->sp;
    *done = false;
    if (!sp.tc_ok) return CIA_OK;
    if (first_use(h, (const void*)scaler_pca_tc_kernel))
        CIA_CUDA(cudaFuncSetAttribute(scaler_pca_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_B));
    const int n_ct = (n + TM - 1) / TM, ncb = (sp.C + TN - 1) / TN;
    const int gx = std::min(n_ct, std::max(1, h->num_sms / ncb));
    scaler_pca_tc_kernel<<<dim3(gx, ncb), NT, SMEM_B, s>>>(
        features, n, n_dev, sp.F, sp.C, (const float4*)sp.tc_par, (const __half*)sp.tc_img,
        std::ldexp(1.f, -sp.tc_ew), sp.offset, sp.f32_flow, z);
    CIA_LAUNCH_CHECK();
    *done = true;
    return CIA_OK;
}
