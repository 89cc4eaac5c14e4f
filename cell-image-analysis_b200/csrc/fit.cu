// fit.cu -- the fits of create_anomaly_detector (CAE_improved_modeltrain.py:404-423) on the device:
//   RobustScaler().fit            train:408      exact column sorts, numpy's percentile arithmetic
//   PCA covariance                train:412-414  fp64 centred Gram X_c^T X_c / (n - 1) (the eigh runs in the caller)
//   OneClassSVM(kernel="rbf").fit train:420-423  libsvm's SMO (svm.cpp Solver::Solve, solve_one_class), one
//                                                persistent cooperative kernel for all iterations
#include "common.cuh"

#include <cooperative_groups.h>
#include <cub/cub.cuh>
#include <climits>
#include <cmath>

namespace cg = cooperative_groups;

// ---------------------------------------------------------------------------------------------------------------
// RobustScaler
// ---------------------------------------------------------------------------------------------------------------

// [n, F] -> [F, n]; NaN is refused (the encoder never produces one; np.nanmedian would skip it)
__global__ void fit_transpose_f32_kernel(const float* __restrict__ x, int n, int F, float* __restrict__ xt,
                                         int32_t* status) {
    __shared__ float tile[32][33];
    const int f0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    for (int k = threadIdx.y; k < 32; k += 8) {
        const int r = r0 + k, f = f0 + threadIdx.x;
        float v = 0.f;
        if (r < n && f < F) {
            v = x[(size_t)r * F + f];
            if (v != v) raise_status(status, CIA_E_ARG);
        }
        tile[k][threadIdx.x] = v;
    }
    __syncthreads();
    for (int k = threadIdx.y; k < 32; k += 8) {
        const int f = f0 + k, r = r0 + threadIdx.x;
        if (r < n && f < F) xt[(size_t)f * n + r] = tile[threadIdx.x][k];
    }
}

__global__ void fit_offsets_kernel(int* off, int F, int n) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f <= F) off[f] = f * n;
}

// np.percentile(col, 100 q), method "linear", of a sorted float32 column: numpy's virtual index
// n q + (1 - q) - 1, and _lerp with the difference taken in float32 (b - a of two float32 values) and the
// interpolation in float64 (seg_percentile_kernel, segment.cu, restates the same arithmetic)
__device__ double np_percentile_sorted(const float* s, int n, double q) {
    const double virt = __dsub_rn(__dadd_rn(__dmul_rn((double)n, q), __dadd_rn(1.0, __dmul_rn(q, -1.0))), 1.0);
    long long prev = (long long)floor(virt), next = prev + 1;
    if (virt >= (double)(n - 1)) { prev = n - 1; next = prev; }
    if (virt < 0) { prev = 0; next = 0; }
    const double g = __dsub_rn(virt, floor(virt));
    const float a = s[prev], b = s[next];
    const double d = (double)__fsub_rn(b, a);
    if (g >= 0.5) return __dsub_rn((double)b, __dmul_rn(d, __dsub_rn(1.0, g)));
    return __dadd_rn((double)a, __dmul_rn(d, g));
}

// center_ = np.nanmedian (float32), scale_ = q75 - q25 (float64) with _handle_zeros_in_scale
__global__ void fit_scaler_quantiles_kernel(const float* __restrict__ sorted, int n, int F, float* __restrict__ center,
                                            double* __restrict__ scale) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    const float* s = sorted + (size_t)f * n;
    // the mean of the two middle elements: exact in float64, one rounding to float32 (np.median of float32)
    center[f] = (n & 1) ? s[n / 2] : (float)__dmul_rn(__dadd_rn((double)s[n / 2 - 1], (double)s[n / 2]), 0.5);
    const double sc = __dsub_rn(np_percentile_sorted(s, n, 0.75), np_percentile_sorted(s, n, 0.25));
    scale[f] = sc < 10.0 * 2.220446049250313e-16 ? 1.0 : sc;   // scale < 10 * finfo(float64).eps -> 1.0
}

// RobustScaler.transform of float32 X: X -= center_ (float32), X /= scale_ (float64 division, stored as float32)
__global__ void fit_scaler_apply_kernel(const float* __restrict__ x, size_t total, int F, const float* __restrict__ center,
                                        const double* __restrict__ scale, float* __restrict__ out) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int f = (int)(i % F);
        out[i] = (float)__ddiv_rn((double)__fsub_rn(x[i], center[f]), scale[f]);
    }
}

int k_fit_robust_scaler(cia_ctx* h, const float* x, int n, int F, float* center, double* scale, float* scaled,
                        cudaStream_t s) {
    if ((long long)n * F > INT_MAX) { h->err = "cia_fit_robust_scaler: n * F must be below 2^31"; return CIA_E_UNSUPPORTED; }
    const size_t total = (size_t)n * F;
    size_t tmp_bytes = 0;
    CIA_CUDA(cub::DeviceSegmentedRadixSort::SortKeys(nullptr, tmp_bytes, (const float*)nullptr, (float*)nullptr, (int)total,
                                                      F, (const int*)nullptr, (const int*)nullptr, 0, 32, s));
    const size_t a_bytes = (total * sizeof(float) + 255) & ~(size_t)255;
    const size_t o_bytes = ((size_t)(F + 1) * sizeof(int) + 255) & ~(size_t)255;
    int rc = ws_reserve(h, h->ws_fit, 2 * a_bytes + o_bytes + tmp_bytes);
    if (rc) return rc;
    unsigned char* base = (unsigned char*)h->ws_fit.p;
    float* xt = (float*)base;
    float* sorted = (float*)(base + a_bytes);
    int* off = (int*)(base + 2 * a_bytes);
    void* tmp = base + 2 * a_bytes + o_bytes;
    fit_transpose_f32_kernel<<<dim3((F + 31) / 32, (n + 31) / 32), dim3(32, 8), 0, s>>>(x, n, F, xt, h->status_dev);
    CIA_LAUNCH_CHECK();
    fit_offsets_kernel<<<(F + 256) / 256, 256, 0, s>>>(off, F, n);
    CIA_LAUNCH_CHECK();
    CIA_CUDA(cub::DeviceSegmentedRadixSort::SortKeys(tmp, tmp_bytes, xt, sorted, (int)total, F, off, off + 1, 0, 32, s));
    h->launches++;
    fit_scaler_quantiles_kernel<<<(F + 127) / 128, 128, 0, s>>>(sorted, n, F, center, scale);
    CIA_LAUNCH_CHECK();
    if (scaled) {
        fit_scaler_apply_kernel<<<h->num_sms * 8, 256, 0, s>>>(x, total, F, center, scale, scaled);
        CIA_LAUNCH_CHECK();
    }
    return CIA_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// PCA: column means and the centred covariance in fp64
// ---------------------------------------------------------------------------------------------------------------

#define FIT_MEAN_CHUNKS 64

// partial[c][f] = sum of rows [c * rows, (c + 1) * rows) of column f, rows in order
__global__ void fit_colsum_kernel(const float* __restrict__ x, int n, int F, int rows, double* __restrict__ partial) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    const int r0 = blockIdx.y * rows, r1 = min(n, r0 + rows);
    double acc = 0.0;
    for (int r = r0; r < r1; ++r) acc = __dadd_rn(acc, (double)x[(size_t)r * F + f]);
    partial[(size_t)blockIdx.y * F + f] = acc;
}

__global__ void fit_mean_kernel(const double* __restrict__ partial, int chunks, int n, int F, double* __restrict__ mean) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    double acc = 0.0;
    for (int c = 0; c < chunks; ++c) acc = __dadd_rn(acc, partial[(size_t)c * F + f]);
    mean[f] = __ddiv_rn(acc, (double)n);
}

// One 64 x 64 tile of the upper triangle per CTA: cov[a][b] = sum_r (x_ra - m_a)(x_rb - m_b) / (n - 1), rows in
// order with fp64 FMAs (each of the 256 threads owns a 4 x 4 block); the tile is mirrored into the lower triangle.
#define GRAM_T 64
#define GRAM_K 16
__global__ void __launch_bounds__(256) fit_gram_kernel(const float* __restrict__ x, int n, int F,
                                                       const double* __restrict__ mean, double* __restrict__ cov) {
    __shared__ double sa[GRAM_K][GRAM_T], sb[GRAM_K][GRAM_T];
    const int T = (F + GRAM_T - 1) / GRAM_T;
    int p = blockIdx.x, bi = 0;
    while (p >= T - bi) { p -= T - bi; ++bi; }
    const int bj = bi + p;
    const int a0 = bi * GRAM_T, b0 = bj * GRAM_T;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    double acc[4][4] = {};
    for (int r0 = 0; r0 < n; r0 += GRAM_K) {
        for (int e = threadIdx.x; e < GRAM_K * GRAM_T; e += 256) {
            const int k = e / GRAM_T, c = e % GRAM_T, r = r0 + k;
            const int fa = a0 + c, fb = b0 + c;
            sa[k][c] = (r < n && fa < F) ? __dsub_rn((double)x[(size_t)r * F + fa], mean[fa]) : 0.0;
            sb[k][c] = (r < n && fb < F) ? __dsub_rn((double)x[(size_t)r * F + fb], mean[fb]) : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < GRAM_K; ++k) {
            double va[4], vb[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) { va[u] = sa[k][ty * 4 + u]; vb[u] = sb[k][tx * 4 + u]; }
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int v = 0; v < 4; ++v) acc[u][v] = __fma_rn(va[u], vb[v], acc[u][v]);
        }
        __syncthreads();
    }
    const double den = (double)(n - 1);
    for (int u = 0; u < 4; ++u)
        for (int v = 0; v < 4; ++v) {
            const int fa = a0 + ty * 4 + u, fb = b0 + tx * 4 + v;
            if (fa < F && fb < F && fa <= fb) {
                const double c = __ddiv_rn(acc[u][v], den);
                cov[(size_t)fa * F + fb] = c;
                cov[(size_t)fb * F + fa] = c;
            }
        }
}

int k_fit_pca_gram(cia_ctx* h, const float* x, int n, int F, double* mean, double* cov, cudaStream_t s) {
    const int chunks = n < FIT_MEAN_CHUNKS ? n : FIT_MEAN_CHUNKS;
    const int rows = (n + chunks - 1) / chunks;
    int rc = ws_reserve(h, h->ws_fit, (size_t)chunks * F * sizeof(double));
    if (rc) return rc;
    double* partial = (double*)h->ws_fit.p;
    fit_colsum_kernel<<<dim3((F + 127) / 128, chunks), 128, 0, s>>>(x, n, F, rows, partial);
    CIA_LAUNCH_CHECK();
    fit_mean_kernel<<<(F + 127) / 128, 128, 0, s>>>(partial, chunks, n, F, mean);
    CIA_LAUNCH_CHECK();
    const int T = (F + GRAM_T - 1) / GRAM_T;
    fit_gram_kernel<<<T * (T + 1) / 2, 256, 0, s>>>(x, n, F, mean, cov);
    CIA_LAUNCH_CHECK();
    return CIA_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// One-class SVM: libsvm's SMO, step for step
// ---------------------------------------------------------------------------------------------------------------
// Problem of solve_one_class (svm.cpp): C_i = 1, y_i = +1, p = 0, Q_ij = (float)exp(-gamma (xsq_i + xsq_j - 2 x_i.x_j))
// (Qfloat), QD_i = 1.  Every dot product, xsq included, is one fp64 FMA chain over the dimensions in order, so
// Q is symmetric and exactly 1 on the diagonal and for duplicated points, as in libsvm.  No shrinking: libsvm
// reaches the same alpha with and without it.  The gradient update uses explicit round-to-nearest multiplies and
// adds because libsvm's own loop is compiled without FMA contraction.

#define SMO_THREADS 256
#define SMO_CH 8           // rows per pass of the gradient initialisation
#define SMO_MAX_DIM 512

struct SmoSel1 { double v, a; int idx; };            // -G_t, alpha_t, t       (select i)
struct SmoSel2 { double obj, g, a, gmax2; int idx; }; // obj_diff, G_t, alpha_t (select j) and max G over alpha > 0

// libsvm keeps the LAST index among equal values (`>=` / `<=` over ascending t): with that tie rule the winner
// is a total order, so the grid-wide reduction gives it whatever the combination order
__device__ __forceinline__ void sel1_merge(SmoSel1& a, const SmoSel1& b) {
    if (b.idx >= 0 && (a.idx < 0 || b.v > a.v || (b.v == a.v && b.idx > a.idx))) a = b;
}
__device__ __forceinline__ void sel2_merge(SmoSel2& a, const SmoSel2& b) {
    const double m = fmax(a.gmax2, b.gmax2);
    if (b.idx >= 0 && (a.idx < 0 || b.obj < a.obj || (b.obj == a.obj && b.idx > a.idx))) { a.obj = b.obj; a.g = b.g; a.a = b.a; a.idx = b.idx; }
    a.gmax2 = m;
}
__device__ __forceinline__ SmoSel1 sel1_shfl(const SmoSel1& x, int o) {
    SmoSel1 y;
    y.v = __shfl_xor_sync(0xffffffffu, x.v, o); y.a = __shfl_xor_sync(0xffffffffu, x.a, o);
    y.idx = __shfl_xor_sync(0xffffffffu, x.idx, o);
    return y;
}
__device__ __forceinline__ SmoSel2 sel2_shfl(const SmoSel2& x, int o) {
    SmoSel2 y;
    y.obj = __shfl_xor_sync(0xffffffffu, x.obj, o); y.g = __shfl_xor_sync(0xffffffffu, x.g, o);
    y.a = __shfl_xor_sync(0xffffffffu, x.a, o); y.gmax2 = __shfl_xor_sync(0xffffffffu, x.gmax2, o);
    y.idx = __shfl_xor_sync(0xffffffffu, x.idx, o);
    return y;
}

// reduce over the CTA; thread 0 gets the result
template <class T, class Sh, class Mg>
__device__ __forceinline__ T block_reduce(T v, T* sh, Sh shfl, Mg merge) {
    for (int o = 16; o > 0; o >>= 1) { T w = shfl(v, o); merge(v, w); }
    const int warp = threadIdx.x >> 5;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[warp] = v;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) merge(v, sh[w]);
    return v;
}

__device__ __forceinline__ float smo_q(double xsq_i, double xsq_t, double dot, double gamma) {
    const double arg = __dmul_rn(-gamma, __dsub_rn(__dadd_rn(xsq_i, xsq_t), __dmul_rn(2.0, dot)));
    return (float)exp(arg);
}

// X [l, d] -> XT [d, l] (coalesced columns for the row passes), xsq, and the start of solve_one_class:
// alpha = 1 for the first npos - 1 indices, `last` at npos - 1, 0 after
__global__ void smo_prepare_kernel(const double* __restrict__ X, int l, int d, int npos, double last,
                                   double* __restrict__ XT, double* __restrict__ xsq, double* __restrict__ alpha) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= l) return;
    double s = 0.0;
    for (int k = 0; k < d; ++k) {
        const double v = X[(size_t)t * d + k];
        XT[(size_t)k * l + t] = v;
        s = __fma_rn(v, v, s);
    }
    xsq[t] = s;
    alpha[t] = t < npos - 1 ? 1.0 : (t == npos - 1 ? last : 0.0);
}

// G_t = sum over i ascending with alpha_i > 0 of alpha_i * Q_it (Solver::Solve, "initialize gradient")
__global__ void __launch_bounds__(128) smo_grad_init_kernel(const double* __restrict__ X, const double* __restrict__ XT,
                                                            const double* __restrict__ xsq, int l, int d, int npos, double last,
                                                            double gamma, double* __restrict__ G) {
    extern __shared__ double sx[];   // [SMO_CH][d]
    __shared__ double sxsq[SMO_CH];
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const double xsq_t = t < l ? xsq[t] : 0.0;
    double g = 0.0;
    for (int i0 = 0; i0 < npos; i0 += SMO_CH) {
        const int nc = min(SMO_CH, npos - i0);
        __syncthreads();
        for (int e = threadIdx.x; e < nc * d; e += blockDim.x) sx[e] = X[(size_t)i0 * d + e];
        if (threadIdx.x < nc) sxsq[threadIdx.x] = xsq[i0 + threadIdx.x];
        __syncthreads();
        if (t < l) {
            double acc[SMO_CH];
#pragma unroll
            for (int c = 0; c < SMO_CH; ++c) acc[c] = 0.0;
            for (int k = 0; k < d; ++k) {
                const double xt = XT[(size_t)k * l + t];
#pragma unroll
                for (int c = 0; c < SMO_CH; ++c)
                    if (c < nc) acc[c] = __fma_rn(sx[c * d + k], xt, acc[c]);
            }
#pragma unroll
            for (int c = 0; c < SMO_CH; ++c)
                if (c < nc) {
                    const double a = i0 + c < npos - 1 ? 1.0 : last;
                    g = __dadd_rn(g, __dmul_rn(a, (double)smo_q(sxsq[c], xsq_t, acc[c], gamma)));
                }
        }
    }
    if (t < l) G[t] = g;
}

struct SmoArgs {
    const double* XT;
    const double* xsq;
    double* alpha;
    double* G;
    float* Qi;            // row i of Q, kept between the two phases of an iteration
    SmoSel1* part1;       // per-CTA candidates
    SmoSel2* part2;
    double* result;       // rho, obj, n_iter, status
    int l, d, max_iter;
    double gamma, tol;
};

// The iterations of Solver::Solve.  Per iteration two grid-wide barriers:
//   phase A (fused with the previous update): candidates for i (arg max of -G over alpha < 1)      | barrier
//   phase B: row Q_i, candidates for j (second-order rule over alpha > 0) and Gmax2 = max G        | barrier
//   every CTA computes the same alpha update from the selected records, then phase A again with row Q_j
// Each thread owns the same indices t in every phase, so alpha / G / Q_i[t] need no exchange except
// through the two selected records (and Q_i[j], written before the second barrier).
__global__ void __launch_bounds__(SMO_THREADS) ocsvm_smo_kernel(SmoArgs a) {
    cg::grid_group grid = cg::this_grid();
    extern __shared__ double xs[];   // [d]: the row of the pass
    __shared__ SmoSel1 sh1[SMO_THREADS / 32];
    __shared__ SmoSel2 sh2[SMO_THREADS / 32];
    __shared__ SmoSel1 best1;
    __shared__ SmoSel2 best2;
    __shared__ double xsq_row;
    const int l = a.l, d = a.d;
    const int tid0 = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
    auto m1 = [](SmoSel1& x, const SmoSel1& y) { sel1_merge(x, y); };
    auto m2 = [](SmoSel2& x, const SmoSel2& y) { sel2_merge(x, y); };
    auto s1 = [](const SmoSel1& x, int o) { return sel1_shfl(x, o); };
    auto s2 = [](const SmoSel2& x, int o) { return sel2_shfl(x, o); };

    SmoSel1 c1{0.0, 0.0, -1};
    for (int t = tid0; t < l; t += stride) {
        const double at = a.alpha[t];
        if (at < 1.0) sel1_merge(c1, SmoSel1{-a.G[t], at, t});
    }
    c1 = block_reduce(c1, sh1, s1, m1);
    if (threadIdx.x == 0) a.part1[blockIdx.x] = c1;

    int iter = 0, status = 0;
    for (;;) {
        grid.sync();
        if (a.max_iter != -1 && iter >= a.max_iter) { status = 1; break; }
        SmoSel1 r1{0.0, 0.0, -1};
        for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) sel1_merge(r1, a.part1[b]);
        r1 = block_reduce(r1, sh1, s1, m1);
        if (threadIdx.x == 0) best1 = r1;
        __syncthreads();
        const SmoSel1 bi = best1;
        if (bi.idx < 0) break;        // every alpha at the upper bound: Gmax = -INF, no j
        const int i = bi.idx;
        const double Gmax = bi.v;
        for (int k = threadIdx.x; k < d; k += blockDim.x) xs[k] = a.XT[(size_t)k * l + i];
        if (threadIdx.x == 0) xsq_row = a.xsq[i];
        __syncthreads();
        const double xsq_i = xsq_row;
        SmoSel2 c2{INFINITY, 0.0, 0.0, -INFINITY, -1};
        for (int t = tid0; t < l; t += stride) {
            double dot = 0.0;
            for (int k = 0; k < d; ++k) dot = __fma_rn(xs[k], a.XT[(size_t)k * l + t], dot);
            const float q = smo_q(xsq_i, a.xsq[t], dot, a.gamma);
            a.Qi[t] = q;
            const double at = a.alpha[t];
            if (at > 0.0) {
                const double gt = a.G[t];
                if (gt >= c2.gmax2) c2.gmax2 = gt;
                const double gd = __dadd_rn(Gmax, gt);
                if (gd > 0) {
                    const double quad = __dsub_rn(__dadd_rn(1.0, 1.0), __dmul_rn(2.0, (double)q));
                    const double num = -__dmul_rn(gd, gd);
                    const double obj = quad > 0 ? __ddiv_rn(num, quad) : __ddiv_rn(num, 1e-12);
                    SmoSel2 c{obj, gt, at, -INFINITY, t};
                    sel2_merge(c2, c);
                }
            }
        }
        c2 = block_reduce(c2, sh2, s2, m2);
        if (threadIdx.x == 0) a.part2[blockIdx.x] = c2;
        grid.sync();
        SmoSel2 r2{INFINITY, 0.0, 0.0, -INFINITY, -1};
        for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) sel2_merge(r2, a.part2[b]);
        r2 = block_reduce(r2, sh2, s2, m2);
        if (threadIdx.x == 0) best2 = r2;
        __syncthreads();
        const SmoSel2 bj = best2;
        if (__dadd_rn(Gmax, bj.gmax2) < a.tol || bj.idx < 0) break;
        ++iter;
        const int j = bj.idx;

        // the same-sign branch of the update (y_i = y_j = +1, C_i = C_j = 1)
        const double Gi = -bi.v, Gj = bj.g, old_ai = bi.a, old_aj = bj.a;
        double quad = __dsub_rn(__dadd_rn(1.0, 1.0), __dmul_rn(2.0, (double)a.Qi[j]));
        if (quad <= 0) quad = 1e-12;
        const double delta = __ddiv_rn(__dsub_rn(Gi, Gj), quad);
        const double sum = __dadd_rn(old_ai, old_aj);
        double ai = __dsub_rn(old_ai, delta), aj = __dadd_rn(old_aj, delta);
        if (sum > 1.0) { if (ai > 1.0) { ai = 1.0; aj = __dsub_rn(sum, 1.0); } }
        else           { if (aj < 0)   { aj = 0;   ai = sum; } }
        if (sum > 1.0) { if (aj > 1.0) { aj = 1.0; ai = __dsub_rn(sum, 1.0); } }
        else           { if (ai < 0)   { ai = 0;   aj = sum; } }
        const double dai = __dsub_rn(ai, old_ai), daj = __dsub_rn(aj, old_aj);

        for (int k = threadIdx.x; k < d; k += blockDim.x) xs[k] = a.XT[(size_t)k * l + j];
        if (threadIdx.x == 0) xsq_row = a.xsq[j];
        __syncthreads();
        const double xsq_j = xsq_row;
        c1 = SmoSel1{0.0, 0.0, -1};
        for (int t = tid0; t < l; t += stride) {
            double dot = 0.0;
            for (int k = 0; k < d; ++k) dot = __fma_rn(xs[k], a.XT[(size_t)k * l + t], dot);
            const float qj = smo_q(xsq_j, a.xsq[t], dot, a.gamma);
            const double g = __dadd_rn(a.G[t], __dadd_rn(__dmul_rn((double)a.Qi[t], dai), __dmul_rn((double)qj, daj)));
            a.G[t] = g;
            double at = a.alpha[t];
            if (t == i) { at = ai; a.alpha[t] = ai; }
            if (t == j) { at = aj; a.alpha[t] = aj; }
            if (at < 1.0) sel1_merge(c1, SmoSel1{-g, at, t});
        }
        c1 = block_reduce(c1, sh1, s1, m1);
        if (threadIdx.x == 0) a.part1[blockIdx.x] = c1;
    }

    // calculate_rho and the objective, by one warp: min / max in any order, the two sums in index order
    // (every CTA left the loop after the same barrier, so alpha and G are final and visible)
    if (blockIdx.x != 0 || threadIdx.x >= 32) return;
    const int lane = threadIdx.x;
    double ub = INFINITY, lb = -INFINITY, sum_free = 0.0, v = 0.0;
    int nr_free = 0;
    for (int base = 0; base < l; base += 32) {
        const int t = base + lane;
        double at = 0.0, gt = 0.0;
        if (t < l) {
            at = a.alpha[t]; gt = a.G[t];
            if (at >= 1.0) lb = fmax(lb, gt);
            else if (at <= 0.0) ub = fmin(ub, gt);
        }
        // alpha = 0 adds a signed zero to v, which changes nothing: only nonzero alpha are summed
        unsigned nz = __ballot_sync(0xffffffffu, t < l && at != 0.0);
        while (nz) {
            const int k = __ffs(nz) - 1;
            nz &= nz - 1;
            const double ak = __shfl_sync(0xffffffffu, at, k), gk = __shfl_sync(0xffffffffu, gt, k);
            v = __dadd_rn(v, __dmul_rn(ak, __dadd_rn(gk, 0.0)));
            if (ak < 1.0) { sum_free = __dadd_rn(sum_free, gk); ++nr_free; }
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        ub = fmin(ub, __shfl_xor_sync(0xffffffffu, ub, o));
        lb = fmax(lb, __shfl_xor_sync(0xffffffffu, lb, o));
    }
    if (lane == 0) {
        a.result[0] = nr_free > 0 ? __ddiv_rn(sum_free, (double)nr_free) : __dmul_rn(__dadd_rn(ub, lb), 0.5);
        a.result[1] = __ddiv_rn(v, 2.0);
        a.result[2] = (double)iter;
        a.result[3] = (double)status;
    }
}

int k_ocsvm_fit(cia_ctx* h, const double* X, int l, int d, double nu, double gamma, double tol, int max_iter,
                double* alpha, double* result, cudaStream_t s) {
    if (d > SMO_MAX_DIM) {
        h->err = "cia_ocsvm_fit: at most " + std::to_string(SMO_MAX_DIM) + " dimensions";
        return CIA_E_UNSUPPORTED;
    }
    // solve_one_class: nu_l is the sequential sum of C_i * nu, then alpha_i = min(C_i, nu_l) while nu_l > 0
    double nu_l = 0;
    for (int i = 0; i < l; ++i) nu_l += 1.0 * nu;
    int npos = 0;
    double last = 0;
    while (nu_l > 0 && npos < l) {
        last = nu_l < 1.0 ? nu_l : 1.0;
        nu_l -= last;
        ++npos;
    }
    int per_sm = 0;
    const size_t smem = (size_t)d * sizeof(double);
    CIA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ocsvm_smo_kernel, SMO_THREADS, smem));
    if (per_sm < 1) { h->err = "cia_ocsvm_fit: SMO kernel does not fit on an SM"; return CIA_E_CUDA; }
    // no more CTAs than rows to give them: fewer CTAs make each barrier cheaper
    const int want = (l + SMO_THREADS - 1) / SMO_THREADS;
    int nb = h->num_sms * per_sm;
    if (nb > want) nb = want;
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t o_xt = 0, o_xsq = o_xt + al((size_t)l * d * 8), o_g = o_xsq + al((size_t)l * 8),
                 o_q = o_g + al((size_t)l * 8), o_p1 = o_q + al((size_t)l * 4), o_p2 = o_p1 + al((size_t)nb * sizeof(SmoSel1)),
                 total = o_p2 + al((size_t)nb * sizeof(SmoSel2));
    int rc = ws_reserve(h, h->ws_fit, total);
    if (rc) return rc;
    unsigned char* base = (unsigned char*)h->ws_fit.p;
    SmoArgs a{};
    a.XT = (const double*)(base + o_xt); a.xsq = (const double*)(base + o_xsq); a.alpha = alpha;
    a.G = (double*)(base + o_g); a.Qi = (float*)(base + o_q);
    a.part1 = (SmoSel1*)(base + o_p1); a.part2 = (SmoSel2*)(base + o_p2);
    a.result = result; a.l = l; a.d = d; a.max_iter = max_iter; a.gamma = gamma; a.tol = tol;
    smo_prepare_kernel<<<(l + 127) / 128, 128, 0, s>>>(X, l, d, npos, last, (double*)a.XT, (double*)a.xsq, alpha);
    CIA_LAUNCH_CHECK();
    smo_grad_init_kernel<<<(l + 127) / 128, 128, SMO_CH * smem, s>>>(X, a.XT, a.xsq, l, d, npos, last, gamma, a.G);
    CIA_LAUNCH_CHECK();
    void* args[] = {(void*)&a};
    CIA_CUDA(cudaLaunchCooperativeKernel((void*)ocsvm_smo_kernel, dim3(nb), dim3(SMO_THREADS), args, smem, s));
    CIA_LAUNCH_CHECK();
    return CIA_OK;
}
