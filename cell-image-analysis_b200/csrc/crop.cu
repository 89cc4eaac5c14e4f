// crop.cu -- K2: bbox crop + CLAHE + anti-aliased resize to 64x64 + float32 cast,
// one CTA per cell, everything between the uint16 bbox read and the 64x64 write
// staying in shared memory.
//
// Replaces improved_detection.py:88 (crop), :98 exposure.equalize_adapthist(cell,
// clip_limit=0.02), :99 resize(..., (64, 64), anti_aliasing=True) and the float32
// cast of :122 (training twin CAE_improved_modeltrain.py:80, 92-93, 332).
// The operation order of scikit-image's CLAHE is replicated step for step
// (SURVEY.md A.2): the integer core (14-bit quantise, 256-bin tile histograms,
// clip + serial redistribution, cumulative mapping) is exact, and the float steps use
// the same precision and rounding (fp64 products rounded to fp32 and accumulated in
// fp32, truncation to uint16), so the uint16 levels are bit-identical.  The resize
// (A.3) runs in fp64 and is rounded to fp32 once, like det:122.
//
// Algorithmic HBM traffic per cell: 2*h*w bytes read + 16 KiB written.
#include "common.cuh"

namespace {

constexpr int K2_THREADS = 512;
constexpr int K2_WARPS = K2_THREADS / 32;
constexpr int NBINS = 256;
constexpr int BIN_SIZE = 65;           // 1 + 16384 / 256
constexpr int MAX_RADIUS = 31;         // gaussian radius for bbox sides <= 1024
constexpr int MAX_SIDE = 1024;

struct Geom {
    int h, w, kh, kw, ntr, ntc, npix, clim;
};

// ceil(2^32 / s) for s = 2..256: floor(n / s) == umulhi(n, magic[s]) exactly for n < 2^16
// (the error term n * (magic * s - 2^32) stays below 2^32).  Replaces the generic integer
// divisions of the redistribution loop, whose operands are warp-uniform and <= 256.
constexpr int MAGIC_N = 256;
struct MagicTab { uint32_t v[MAGIC_N + 1]; };
constexpr MagicTab make_magic() {
    MagicTab t{};
    t.v[0] = 0; t.v[1] = 0;
    for (int s = 2; s <= MAGIC_N; ++s) t.v[s] = 0xFFFFFFFFu / (uint32_t)s + 1u;
    return t;
}
__constant__ MagicTab k_magic = make_magic();
constexpr int MAPTAB_N = 1024;         // entries of the per-cell count -> level table (2 KB)

__device__ __forceinline__ int reflect_idx(int i, int n) {   // numpy 'reflect'
    if (n == 1) return 0;
    while (i < 0 || i >= n) i = i < 0 ? -i : 2 * (n - 1) - i;
    return i;
}
__device__ __forceinline__ int mirror_idx(int i, int n) {    // ndimage 'mirror'
    if (n == 1) return 0;
    const int p = 2 * n - 2;
    i = i < 0 ? -i : i;
    i %= p;
    return i >= n ? p - i : i;
}

// ndimage 'mirror' for an index at most one period out of range (all the resize taps are:
// |offset| <= gaussian radius + 1 << n whenever blurring is on); anything else takes the
// general path.  No integer modulo on the hot path.
__device__ __forceinline__ int mirror_near(int i, int n) {
    int j = i < 0 ? -i : i;
    if (j >= n) j = 2 * n - 2 - j;
    if ((unsigned)j >= (unsigned)n) j = mirror_idx(i, n);
    return j;
}

__host__ __device__ inline size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }
__host__ __device__ inline size_t cell_bytes(int h, int w, int ntr, int ntc) {
    const size_t hw = (size_t)h * w;
    size_t maps = (size_t)ntr * ntc * NBINS * sizeof(uint16_t);
    size_t t = (size_t)CIA_CROP * w * sizeof(double);
    return align16(hw) + align16(2 * hw) + align16(maps > t ? maps : t);
}

// One warp: clip + redistribute a 256-bin histogram held 8 CONSECUTIVE bins per lane
// (bin = 8*lane + m), then cumulative mapping.  skimage clip_histogram / map_histogram.
// Instruction diet (the kernel is issue-bound): the strided selection `(b - index) % step`
// uses one reciprocal per iteration (exact for b < 256), the prefix sum is 7 local adds + one
// warp scan, the 8 uint16 map entries of a lane leave as one 16-byte store.
__device__ __forceinline__ void clip_and_map(int (&hv)[8], int clim, double scale, int lane,
                                             uint16_t* __restrict__ map_out,
                                             const uint16_t* __restrict__ level_tab) {
    int ex = 0;
#pragma unroll
    for (int m = 0; m < 8; ++m) {
        const int c = min(hv[m], clim);
        ex += hv[m] - c; hv[m] = c;
    }
    ex = __reduce_add_sync(0xffffffffu, ex);          // REDUX: one instruction instead of a 5-step shuffle tree
    if (ex > 0) {
        const int incr = ex / NBINS;
        if (incr > 0) {     // with incr == 0 (small tiles: excess < 256) both passes below change nothing
            const int upper = clim - incr;
            int nlow = 0;
#pragma unroll
            for (int m = 0; m < 8; ++m)
                if (hv[m] < upper) { hv[m] += incr; ++nlow; }
            int midsum = 0, nmid = 0;
#pragma unroll
            for (int m = 0; m < 8; ++m)
                if (hv[m] >= upper && hv[m] < clim) { midsum += hv[m]; ++nmid; hv[m] = clim; }
            // nlow, nmid <= 256 each and midsum <= 256 * clim < 2^17 fit one 32-bit REDUX each way
            const unsigned cnts = __reduce_add_sync(0xffffffffu, (unsigned)nlow | ((unsigned)nmid << 16));
            const int msum = __reduce_add_sync(0xffffffffu, midsum);
            ex -= (int)(cnts & 0xFFFFu) * incr;
            ex += msum - (int)(cnts >> 16) * clim;
        }

        while (ex > 0) {
            const int prev = ex;
            bool stuck = false;
            for (int index = 0; index < NBINS; ++index) {
                unsigned under = 0;
#pragma unroll
                for (int m = 0; m < 8; ++m) under |= (hv[m] < clim ? 1u : 0u) << m;
                // count of under-limit bins over the warp
                const int cnt = __reduce_add_sync(0xffffffffu, __popc(under));
                if (cnt == 0) { stuck = true; break; }   // nothing can move any more
                // step = max(cnt / ex, 1) with cnt <= 256: table reciprocal instead of a division
                int step = 1;
                if (ex <= cnt) step = ex == 1 ? cnt : (int)__umulhi((unsigned)cnt, k_magic.v[ex]);
                const unsigned magic = k_magic.v[step];                     // ceil(2^32 / step), step <= 256
                int moved = 0;
#pragma unroll
                for (int m = 0; m < 8; ++m) {
                    const int d = 8 * lane + m - index;
                    bool sel = d >= 0 && ((under >> m) & 1u);
                    if (sel && step > 1) {
                        const unsigned qd = __umulhi((unsigned)d, magic);    // floor(d / step), exact for d < 2^16
                        sel = (unsigned)d - qd * (unsigned)step == 0u;
                    }
                    if (sel) { ++hv[m]; ++moved; }
                }
                ex -= __reduce_add_sync(0xffffffffu, moved);
                if (ex <= 0) break;
            }
            if (stuck || prev == ex) break;
        }
    }

    // cumulative sum in bin order, scale, clip, truncate
    int pre[8];
    pre[0] = hv[0];
#pragma unroll
    for (int m = 1; m < 8; ++m) pre[m] = pre[m - 1] + hv[m];
    int run = pre[7];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, run, o);
        if (lane >= o) run += t;
    }
    const int base = run - pre[7];
    __align__(16) uint16_t mv16[8];
    if (level_tab) {
        // the level depends on the cumulative count only: looked up in the per-cell table built
        // with the very expression of the other branch
#pragma unroll
        for (int m = 0; m < 8; ++m) mv16[m] = level_tab[base + pre[m]];
    } else {
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            // clip after the truncation (same result: both are monotone; the product stays far below 2^31)
            const int mv = (int)__dmul_rn((double)(base + pre[m]), scale);
            mv16[m] = (uint16_t)min(mv, 16383);
        }
    }
    *reinterpret_cast<uint4*>(map_out + 8 * lane) = *reinterpret_cast<const uint4*>(mv16);
}

__device__ __forceinline__ void block_minmax(int& mn, int& mx, int* sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) { sh[wid] = mn; sh[K2_WARPS + wid] = mx; }
    __syncthreads();
    mn = sh[0]; mx = sh[K2_WARPS];
#pragma unroll
    for (int i = 1; i < K2_WARPS; ++i) { mn = min(mn, sh[i]); mx = max(mx, sh[K2_WARPS + i]); }
}

__device__ __forceinline__ int cell_class(const cia_cell& C, size_t lo_bytes, size_t hi_bytes) {
    const int h = C.maxr - C.minr, w = C.maxc - C.minc;
    if (h > MAX_SIDE || w > MAX_SIDE) return 2;       // refused inside the class-2 launch
    const int kh = max(h / 8, 1), kw = max(w / 8, 1);
    const size_t need = cell_bytes(h, w, (h + kh - 1) / kh, (w + kw - 1) / kw);
    return need <= lo_bytes ? 0 : (need <= hi_bytes ? 1 : 2);
}

// cls: 0/1 = shared-memory classes (dynamic smem = smem_bytes), 2 = global-scratch class.
// Walks cls_list[0 .. *cls_count) (cls_list == nullptr: every cell, skipping the other classes).
__global__ void __launch_bounds__(K2_THREADS)
crop_clahe_resize_kernel(const uint16_t* __restrict__ images, int H, int W,
                         const cia_cell* __restrict__ cells, int n_cells,
                         const int32_t* __restrict__ n_cells_dev, double clip_limit, double intensity_inv,
                         float* __restrict__ crops32, double* __restrict__ crops64,
                         int cls, size_t lo_bytes, size_t hi_bytes,
                         unsigned char* __restrict__ gscratch, size_t gscratch_per_cta,
                         int32_t* status, uint16_t* __restrict__ levels_out,
                         const int64_t* __restrict__ level_offsets,
                         const int32_t* __restrict__ cls_list, const int32_t* __restrict__ cls_count) {
    extern __shared__ __align__(16) unsigned char dyn[];
    __shared__ __align__(16) uint32_t hist_s[K2_WARPS][NBINS];
    __shared__ double ctab_s[2][MAX_SIDE / 8];      // a/kh and b/kw interpolation coefficients
    __shared__ int red_s[2 * K2_WARPS];
    __shared__ double gw_s[2][2 * MAX_RADIUS + 2];

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int n = cls_list ? min(*cls_count, n_cells) : dev_count(n_cells, n_cells_dev);

    for (int it = blockIdx.x; it < n; it += gridDim.x) {
        const int cell = cls_list ? cls_list[it] : it;
        const cia_cell C = cells[cell];
        Geom g;
        g.h = C.maxr - C.minr; g.w = C.maxc - C.minc;
        g.kh = max(g.h / 8, 1); g.kw = max(g.w / 8, 1);
        g.ntr = (g.h + g.kh - 1) / g.kh; g.ntc = (g.w + g.kw - 1) / g.kw;
        g.npix = g.kh * g.kw;
        {
            double cl = __dmul_rn(clip_limit, (double)g.npix);
            if (!(cl >= 1.0)) cl = 1.0;
            g.clim = clip_limit > 0.0 ? (int)cl : 16384;
        }
        const size_t need = cell_bytes(g.h, g.w, g.ntr, g.ntc);
        int my_cls;
        if (g.h > MAX_SIDE || g.w > MAX_SIDE) {
            if (cls == 2 && tid == 0) raise_status(status, CIA_E_UNSUPPORTED);
            if (cls == 2) {
                // defined output for the unsupported cell: zeros
                for (int i = tid; i < CIA_CROP * CIA_CROP; i += K2_THREADS) {
                    crops32[(size_t)cell * 4096 + i] = 0.f;
                    if (crops64) crops64[(size_t)cell * 4096 + i] = 0.0;
                }
            }
            continue;
        }
        my_cls = need <= lo_bytes ? 0 : (need <= hi_bytes ? 1 : 2);
        if (my_cls != cls) continue;

        unsigned char* base = cls == 2 ? gscratch + (size_t)blockIdx.x * gscratch_per_cta : dyn;
        const int hw = g.h * g.w;
        uint8_t* bins = base;
        uint16_t* rimg = reinterpret_cast<uint16_t*>(base + align16(hw));
        uint16_t* maps = reinterpret_cast<uint16_t*>(base + align16(hw) + align16(2 * (size_t)hw));
        double* T = reinterpret_cast<double*>(maps);

        const uint16_t* img = images + ((size_t)C.field * H + C.minr) * (size_t)W + C.minc;

        // ---- A: load bbox, min / max ----
        const unsigned w_magic = 0xFFFFFFFFu / (unsigned)g.w + 1u;      // i / w for i * w < 2^32 (hw <= 2^20, w <= 2^10)
        int mn = 65535, mx = 0;
        for (int i = tid; i < hw; i += K2_THREADS) {
            const int y = (g.w == 1) ? i : (int)__umulhi((unsigned)i, w_magic), x = i - y * g.w;
            const int v = __ldg(img + (size_t)y * W + x);
            rimg[i] = (uint16_t)v;
            mn = min(mn, v); mx = max(mx, v);
        }
        block_minmax(mn, mx, red_s);

        // ---- B: 14-bit quantise (round half even) and bin ----
        {
            const double inv = intensity_inv;
            const double vmin = __dmul_rn((double)mn, inv), vmax = __dmul_rn((double)mx, inv);
            const double den = __dsub_rn(vmax, vmin);
            for (int i = tid; i < hw; i += K2_THREADS) {
                const double v = __dmul_rn((double)rimg[i], inv);
                int q;
                if (mn != mx) {
                    const double t = __dmul_rn(__ddiv_rn(__dsub_rn(v, vmin), den), 16383.0);
                    q = __double2int_rn(t);
                } else {
                    q = __double2int_rn(fmin(fmax(v, 0.0), 16383.0));
                }
                bins[i] = (uint8_t)(q / BIN_SIZE);
            }
        }

        // ---- C: per-tile histogram -> clipped mapping ----
        const int ntiles = g.ntr * g.ntc;
        const double map_scale = __ddiv_rn(16383.0, (double)g.npix);
        const unsigned kw_magic = 0xFFFFFFFFu / (unsigned)g.kw + 1u;       // p / kw for p < 2^16 (npix <= 128*128)
        // count -> level table (ctab_s is free until stage D).  A tile's counts sum to npix plus at
        // most one redistribution pass of overshoot (< 256), so npix + 256 entries cover every
        // cumulative count; larger tiles convert per bin.
        uint16_t* level_tab = nullptr;
        if (g.npix + NBINS <= MAPTAB_N) {
            level_tab = reinterpret_cast<uint16_t*>(&ctab_s[0][0]);
            for (int c = tid; c < g.npix + NBINS; c += K2_THREADS)
                level_tab[c] = (uint16_t)min((int)__dmul_rn((double)c, map_scale), 16383);
        }
        __syncthreads();
        for (int t = wid; t < ntiles; t += K2_WARPS) {
            // ntr, ntc <= 16 here only matters for speed: t / ntc via the reciprocal table
            const int ti = g.ntc == 1 ? t : (g.ntc <= MAGIC_N ? (int)__umulhi((unsigned)t, k_magic.v[g.ntc]) : t / g.ntc);
            const int tj = t - ti * g.ntc;
            uint32_t* hs = hist_s[wid];
            reinterpret_cast<uint4*>(hs)[2 * lane] = make_uint4(0, 0, 0, 0);
            reinterpret_cast<uint4*>(hs)[2 * lane + 1] = make_uint4(0, 0, 0, 0);
            __syncwarp();
            const int y0 = ti * g.kh, x0 = tj * g.kw;
            if (y0 + g.kh <= g.h && x0 + g.kw <= g.w) {
                // interior tile: no padding, no reflection
                const uint8_t* bt = bins + y0 * g.w + x0;
                for (int p = lane; p < g.npix; p += 32) {
                    const int a = (g.kw == 1) ? p : (int)__umulhi((unsigned)p, kw_magic), b = p - a * g.kw;
                    atomicAdd(&hs[bt[a * g.w + b]], 1u);
                }
            } else {
                for (int p = lane; p < g.npix; p += 32) {
                    const int a = (g.kw == 1) ? p : (int)__umulhi((unsigned)p, kw_magic), b = p - a * g.kw;
                    const int y = reflect_idx(y0 + a, g.h);
                    const int x = reflect_idx(x0 + b, g.w);
                    atomicAdd(&hs[bins[y * g.w + x]], 1u);
                }
            }
            __syncwarp();
            int hv[8];
            {
                const uint4 h0 = reinterpret_cast<const uint4*>(hs)[2 * lane];
                const uint4 h1 = reinterpret_cast<const uint4*>(hs)[2 * lane + 1];
                hv[0] = (int)h0.x; hv[1] = (int)h0.y; hv[2] = (int)h0.z; hv[3] = (int)h0.w;
                hv[4] = (int)h1.x; hv[5] = (int)h1.y; hv[6] = (int)h1.z; hv[7] = (int)h1.w;
            }
            __syncwarp();
            clip_and_map(hv, g.clim, map_scale, lane, maps + (size_t)t * NBINS, level_tab);
        }
        __syncthreads();

        // ---- D: 4-corner interpolation, fp32 accumulation, truncate to uint16 ----
        int rmn = 65535, rmx = 0;
        {
            const int pr = g.kh / 2, pc = g.kw / 2;
            // np.arange(k) / k tables (fp64 divisions once per cell instead of twice per pixel)
            for (int a = tid; a < g.kh; a += K2_THREADS) ctab_s[0][a] = __ddiv_rn((double)a, (double)g.kh);
            for (int b = tid; b < g.kw; b += K2_THREADS) ctab_s[1][b] = __ddiv_rn((double)b, (double)g.kw);
            __syncthreads();
            const unsigned kh_magic = 0xFFFFFFFFu / (unsigned)g.kh + 1u;
            for (int i = tid; i < hw; i += K2_THREADS) {
                const int y = (g.w == 1) ? i : (int)__umulhi((unsigned)i, w_magic), x = i - y * g.w;
                const int Y = y + pr, X = x + pc;
                const int I = (g.kh == 1) ? Y : (int)__umulhi((unsigned)Y, kh_magic), a = Y - I * g.kh;
                const int J = (g.kw == 1) ? X : (int)__umulhi((unsigned)X, kw_magic), b = X - J * g.kw;
                const double cr = ctab_s[0][a];
                const double cc = ctab_s[1][b];
                const double icr = __dsub_rn(1.0, cr), icc = __dsub_rn(1.0, cc);
                const int t0 = min(max(I - 1, 0), g.ntr - 1), t1 = min(max(I, 0), g.ntr - 1);
                const int u0 = min(max(J - 1, 0), g.ntc - 1), u1 = min(max(J, 0), g.ntc - 1);
                const int bin = bins[i];
                const double m00 = (double)maps[((size_t)t0 * g.ntc + u0) * NBINS + bin];
                const double m01 = (double)maps[((size_t)t0 * g.ntc + u1) * NBINS + bin];
                const double m10 = (double)maps[((size_t)t1 * g.ntc + u0) * NBINS + bin];
                const double m11 = (double)maps[((size_t)t1 * g.ntc + u1) * NBINS + bin];
                float res = 0.f;
                res = __fadd_rn(res, __double2float_rn(__dmul_rn(m00, __dmul_rn(icc, icr))));
                res = __fadd_rn(res, __double2float_rn(__dmul_rn(m01, __dmul_rn(cc, icr))));
                res = __fadd_rn(res, __double2float_rn(__dmul_rn(m10, __dmul_rn(icc, cr))));
                res = __fadd_rn(res, __double2float_rn(__dmul_rn(m11, __dmul_rn(cc, cr))));
                const int r = (int)res;
                rimg[i] = (uint16_t)r;
                rmn = min(rmn, r); rmx = max(rmx, r);
            }
        }
        block_minmax(rmn, rmx, red_s);   // also orders the rimg writes / maps reads
        if (levels_out) {                // test tap: the bit-exact integer core
            uint16_t* dst = levels_out + level_offsets[cell];
            for (int i = tid; i < hw; i += K2_THREADS) dst[i] = rimg[i];
        }

        // ---- E: gaussian weights for the axes that shrink ----
        const double fr = __ddiv_rn((double)g.h, 64.0), fc = __ddiv_rn((double)g.w, 64.0);
        double sig_r = __dmul_rn(__dsub_rn(fr, 1.0), 0.5), sig_c = __dmul_rn(__dsub_rn(fc, 1.0), 0.5);
        if (sig_r < 0.0) sig_r = 0.0;
        if (sig_c < 0.0) sig_c = 0.0;
        const bool blur_r = sig_r > 1e-15, blur_c = sig_c > 1e-15;
        const int rad_r = blur_r ? (int)(4.0 * sig_r + 0.5) : 0;
        const int rad_c = blur_c ? (int)(4.0 * sig_c + 0.5) : 0;
        // source coordinate of each of the 64 output rows / columns: integer part and weight, once
        // per cell (ctab_s and hist_s are free after stage D / C)
        int* coord_i = reinterpret_cast<int*>(&hist_s[0][0]);
        if (tid >= 64 && tid < 64 + 2 * CIA_CROP) {
            const int k = tid - 64, axis = k >> 6, o = k & 63;
            const double cc = ((double)o + 0.5) * (axis == 0 ? fr : fc) - 0.5;
            const double fl = floor(cc);
            ctab_s[axis][o] = cc - fl;
            coord_i[axis * CIA_CROP + o] = (int)fl;
        }
        if (wid < 2) {
            const bool on = wid == 0 ? blur_r : blur_c;
            const int rad = wid == 0 ? rad_r : rad_c;
            const double sg = wid == 0 ? sig_r : sig_c;
            if (on) {
                double s = 0.0;
                const double cf = -0.5 / (sg * sg);
                for (int j = lane; j <= 2 * rad; j += 32) {
                    const double xx = (double)(j - rad);
                    const double e = exp(cf * xx * xx);
                    gw_s[wid][j] = e;
                    s += e;
                }
                s = warp_sum(s);
                __syncwarp();
                for (int j = lane; j <= 2 * rad; j += 32) gw_s[wid][j] = gw_s[wid][j] / s;
            }
        }
        __syncthreads();

        const bool degenerate = rmn == rmx;
        const double den = (double)(rmx - rmn);
        const double lo = degenerate ? fmin(fmax((double)rmn, 0.0), 1.0) : 0.0;
        const double hi = degenerate ? lo : 1.0;
        // (r - rmn) / den with both operands integers <= 16383: reciprocal, product and one FMA
        // correction give the correctly rounded quotient (Markstein); exhaustively checked against
        // IEEE division over the whole domain by tests/test_exact_division.py
        const double den_rcp = degenerate ? 0.0 : __drcp_rn(den);
        auto value = [&](int y, int x) -> double {
            const double r = (double)rimg[y * g.w + x];
            // degenerate (constant) image: every pixel equals rmn, i.e. clip(rmn, 0, 1) = lo
            const double a = r - (double)rmn;
            const double q0 = __dmul_rn(a, den_rcp);
            const double q = __fma_rn(__fma_rn(-q0, den, a), den_rcp, q0);
            return degenerate ? lo : q;
        };

        // ---- F: rows: (zoom o gaussian) along axis 0 -> T[64][w] ----
        for (int i = tid; i < CIA_CROP * g.w; i += K2_THREADS) {
            const int oy = (g.w == 1) ? i : (int)__umulhi((unsigned)i, w_magic), x = i - oy * g.w;
            const double t = ctab_s[0][oy];
            const int i0 = coord_i[oy];
            double v[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int yy = i0 + e;
                if (!blur_r) {
                    v[e] = value(mirror_near(yy, g.h), x);
                } else {
                    double acc = 0.0;
                    for (int j = 0; j <= 2 * rad_r; ++j)
                        acc += gw_s[0][j] * value(mirror_near(mirror_near(yy, g.h) + j - rad_r, g.h), x);
                    v[e] = acc;
                }
            }
            T[i] = (1.0 - t) * v[0] + t * v[1];
        }
        __syncthreads();

        // ---- G: columns -> 64x64, clip, store ----
        for (int i = tid; i < CIA_CROP * CIA_CROP; i += K2_THREADS) {
            const int oy = i >> 6, ox = i & 63;
            const double t = ctab_s[1][ox];
            const int j0 = coord_i[CIA_CROP + ox];
            const double* Trow = T + (size_t)oy * g.w;
            double v[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int xx = j0 + e;
                if (!blur_c) {
                    v[e] = Trow[mirror_near(xx, g.w)];
                } else {
                    double acc = 0.0;
                    for (int j = 0; j <= 2 * rad_c; ++j)
                        acc += gw_s[1][j] * Trow[mirror_near(mirror_near(xx, g.w) + j - rad_c, g.w)];
                    v[e] = acc;
                }
            }
            double o = (1.0 - t) * v[0] + t * v[1];
            if (crops64) {
                o = fmin(fmax(o, lo), hi);
                crops64[(size_t)cell * 4096 + i] = o;
            }
            // det:122 rounding; lo and hi are 0 or 1, exact in fp32, and rounding is monotone, so
            // clipping after the conversion equals converting the clipped value
            crops32[(size_t)cell * 4096 + i] = fminf(fmaxf((float)o, (float)lo), (float)hi);
        }
        __syncthreads();
    }
}


// ---------------------------------------------------------------------------------------
// Fast path: cells whose CLAHE clip limit is 1 (tiles of < 100 pixels at clip_limit 0.02 --
// every cell with sides up to ~80 px, i.e. all of BASELINE config 2).
//
// ncu on the general kernel above (profiles/r1j_crop_full.txt): 57k warp instructions per ~34x34
// cell, half of them in the per-tile stage -- a warp clips, redistributes and prefix-sums a dense
// 256-bin histogram for a tile that holds 16 pixels.  With clip limit 1 the clipped histogram is
// an OCCUPANCY SET: every bin is 0 or 1, the excess is npix - popcount, `excess // 256` is 0 (so
// the two bulk passes of clip_histogram change nothing) and the serial redistribution only ever
// turns zero bins into ones.  A tile is therefore a 256-bit mask: ONE THREAD per tile builds it
// with shared-memory ORs, runs skimage's redistribution loop on the bits, and stores per 32-bin
// word the number of bits set below it; the mapping of a bin is then
//     level_tab[ bits_below(word) + popc(word & mask_up_to(bin)) ]
// evaluated where the interpolation needs it -- 72 bytes per tile instead of a 512-byte table,
// ~10 KB of shared memory per typical cell, 13-16 resident CTAs of 128 threads per SM.
// The bbox is fetched with aligned 16-byte loads (8 pixels each) straight into shared memory,
// the two resize passes stream through a per-warp row block (no 64 x w intermediate, no block
// barrier), and cells are handed out by an atomic work counter (bbox areas vary 20x).
// Arithmetic is the general kernel's, operation for operation: same uint16 levels, bit for bit.
// ---------------------------------------------------------------------------------------
constexpr int KF_THREADS = 128;
constexpr int KF_WARPS = KF_THREADS / 32;
constexpr int KF_TILE_WORDS = 18;      // 8 x (mask word, bits set below it) + 2 pad words (bank spread, 8-byte aligned)
constexpr int KF_TBUF = 176;           // doubles per warp: the row block of the resize passes
constexpr int KF_MAX_SIDE = 96;        // gaussian radius <= 1 up to here
constexpr int KF_MAX_NPIX = 256;       // excess < 256 => the bulk passes of clip_histogram are no-ops
constexpr int KF_CLASSES = 2;

struct FastLayout {
    int pitch;                          // uint16 elements per staged row (multiple of 8)
    int o_bins, o_tiles, o_coef, o_ltab, o_rinfo, o_cinfo, total;
};
__host__ __device__ inline FastLayout fast_layout(int h, int w, int ntiles, int npix) {
    FastLayout L;
    L.pitch = ((w + 14) >> 3) << 3;
    int o = (int)align16((size_t)h * L.pitch * 2);       // raw pixels, later the dense uint16 levels
    const int u0 = o;                                    // everything below is dead after stage D ...
    L.o_bins = o;  o += (int)align16((size_t)h * w);
    L.o_tiles = o; o += (int)align16((size_t)ntiles * KF_TILE_WORDS * 4);
    L.o_coef = o;  o += npix * 32;
    L.o_ltab = o;  o += (int)align16((KF_MAX_NPIX + 1) * 2);
    L.o_rinfo = o; o += (int)align16((size_t)h * 4);
    L.o_cinfo = o; o += (int)align16((size_t)w * 4);
    const int tb = u0 + KF_WARPS * KF_TBUF * 8;          // ... and shares its space with the row blocks
    L.total = o > tb ? o : tb;
    return L;
}

// class of a cell: 0..KF_CLASSES-1 fast (by shared-memory need), KF_CLASSES + {0,1,2} general
__device__ __forceinline__ int cell_class_all(const cia_cell& C, double clip_limit, const int* fast_bytes,
                                              size_t lo_bytes, size_t hi_bytes) {
    const int h = C.maxr - C.minr, w = C.maxc - C.minc;
    if (h >= 1 && w >= 1 && h <= KF_MAX_SIDE && w <= KF_MAX_SIDE) {
        const int kh = max(h / 8, 1), kw = max(w / 8, 1), npix = kh * kw;
        double cl = __dmul_rn(clip_limit, (double)npix);
        if (!(cl >= 1.0)) cl = 1.0;
        if (clip_limit > 0.0 && (int)cl == 1 && npix <= KF_MAX_NPIX) {
            const int need = fast_layout(h, w, ((h + kh - 1) / kh) * ((w + kw - 1) / kw), npix).total;
            for (int c = 0; c < KF_CLASSES; ++c)
                if (need <= fast_bytes[c]) return c;
        }
    }
    return KF_CLASSES + cell_class(C, lo_bytes, hi_bytes);
}

struct FastBytes { int v[KF_CLASSES]; };

// Work lists of all classes.  cls_counts[c] = entries of list c (zeroed by the caller).
__global__ void __launch_bounds__(256)
crop_classify_all_kernel(const cia_cell* __restrict__ cells, int n_cells,
                         const int32_t* __restrict__ n_cells_dev, double clip_limit, FastBytes fb,
                         size_t lo_bytes, size_t hi_bytes, int32_t* __restrict__ cls_counts,
                         int32_t* __restrict__ lists, size_t list_stride) {
    const int n = dev_count(n_cells, n_cells_dev);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int c = cell_class_all(cells[i], clip_limit, fb.v, lo_bytes, hi_bytes);
        lists[(size_t)c * list_stride + atomicAdd(cls_counts + c, 1)] = i;
    }
}

template <bool WANT64>
__global__ void __launch_bounds__(KF_THREADS, 8)
crop_fast_kernel(const uint16_t* __restrict__ images, int H, int W, const cia_cell* __restrict__ cells,
                 double intensity_inv, float* __restrict__ crops32, double* __restrict__ crops64,
                 const int32_t* __restrict__ list, const int32_t* __restrict__ count,
                 int32_t* __restrict__ work_counter, uint16_t* __restrict__ levels_out,
                 const int64_t* __restrict__ level_offsets) {
    extern __shared__ __align__(16) unsigned char dyn[];
    __shared__ double ctab_s[2][CIA_CROP];        // interpolation weight of each output row / column
    __shared__ int coord_s[2][CIA_CROP];          // integer source coordinate
    __shared__ int src0_s[2][CIA_CROP], src1_s[2][CIA_CROP];   // unblurred axis: mirrored source line offsets
    __shared__ double gw_s[2][4];                 // gaussian taps (radius <= 1)
    __shared__ double scale_s[2];
    __shared__ int rad_s[2];                      // gaussian radius per axis, -1 = not blurred
    __shared__ int red_s[2 * KF_WARPS];
    __shared__ int work_s;

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int n = *count;

    for (;;) {
        __syncthreads();                          // the previous cell's shared memory is free
        if (tid == 0) work_s = atomicAdd(work_counter, 1);
        __syncthreads();
        const int it = work_s;
        if (it >= n) break;
        const int cell = list[it];
        const cia_cell C = cells[cell];
        const int h = C.maxr - C.minr, w = C.maxc - C.minc;
        const int kh = max(h / 8, 1), kw = max(w / 8, 1);
        const int ntr = (h + kh - 1) / kh, ntc = (w + kw - 1) / kw;
        const int npix = kh * kw, ntiles = ntr * ntc, hw = h * w;
        const FastLayout L = fast_layout(h, w, ntiles, npix);
        uint16_t* raw = reinterpret_cast<uint16_t*>(dyn);        // staged rows; from stage D on: dense levels
        uint8_t* bins = dyn + L.o_bins;
        uint32_t* tiles = reinterpret_cast<uint32_t*>(dyn + L.o_tiles);
        double* coef = reinterpret_cast<double*>(dyn + L.o_coef);
        uint16_t* level_tab = reinterpret_cast<uint16_t*>(dyn + L.o_ltab);
        uint32_t* rinfo = reinterpret_cast<uint32_t*>(dyn + L.o_rinfo);
        uint32_t* cinfo = reinterpret_cast<uint32_t*>(dyn + L.o_cinfo);
        double* tbuf = reinterpret_cast<double*>(dyn + L.o_bins) + wid * KF_TBUF;

        const unsigned w_magic = 0xFFFFFFFFu / (unsigned)w + 1u;         // i / w for i < 2^16
        const long long base_elem = ((long long)C.field * H + C.minr) * (long long)W + C.minc;
        const long long end_elem = (long long)(C.field + 1) * H * (long long)W;
        // element alignment (mod 8) of the first pixel of bbox row 0 / increment per row
        const int e00 = (int)((((unsigned long long)(uintptr_t)images >> 1) + (unsigned long long)base_elem) & 7ull);
        const int wlow = W & 7;

        // ---- A: bbox -> shared memory with aligned 16-byte loads; min / max ----
        int mn = 65535, mx = 0;
        {
            const int chunks = L.pitch >> 3;
            const unsigned c_magic = k_magic.v[chunks];                  // chunks in 1..13 (1: w == 1, no magic)
            for (int i = tid; i < h * chunks; i += KF_THREADS) {
                const int y = (chunks == 1) ? i : (int)__umulhi((unsigned)i, c_magic), c = i - y * chunks;
                const int e0 = (e00 + y * wlow) & 7;
                const int first = 8 * c - e0;                            // bbox column of the chunk's first pixel
                if (first >= w) continue;
                const long long g0 = base_elem + (long long)y * W + first;
                uint4 v;
                if (g0 >= 0 && g0 + 8 <= end_elem) {
                    v = __ldg(reinterpret_cast<const uint4*>(images + g0));
                } else {                                                 // chunk straddles the buffer's ends
                    uint16_t t[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        t[k] = (first + k >= 0 && first + k < w) ? __ldg(images + g0 + k) : (uint16_t)0;
                    v = make_uint4(t[0] | ((uint32_t)t[1] << 16), t[2] | ((uint32_t)t[3] << 16),
                                   t[4] | ((uint32_t)t[5] << 16), t[6] | ((uint32_t)t[7] << 16));
                }
                *reinterpret_cast<uint4*>(raw + y * L.pitch + 8 * c) = v;
                const uint32_t vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int px = (int)((vv[k >> 1] >> (16 * (k & 1))) & 0xFFFFu);
                    if ((unsigned)(first + k) < (unsigned)w) { mn = min(mn, px); mx = max(mx, px); }
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        }
        if (lane == 0) { red_s[wid] = mn; red_s[KF_WARPS + wid] = mx; }
        // per-cell tables (independent of the pixels): count -> level, interpolation coefficients,
        // row / column -> (tile pair, in-tile offset)
        {
            const double map_scale = __ddiv_rn(16383.0, (double)npix);
            for (int c = tid; c <= KF_MAX_NPIX; c += KF_THREADS)
                level_tab[c] = (uint16_t)min((int)__dmul_rn((double)c, map_scale), 16383);
            for (int p = tid; p < npix; p += KF_THREADS) {
                const int a = p / kw, b = p - a * kw;
                const double cr = __ddiv_rn((double)a, (double)kh), cc = __ddiv_rn((double)b, (double)kw);
                const double icr = __dsub_rn(1.0, cr), icc = __dsub_rn(1.0, cc);
                coef[4 * p + 0] = __dmul_rn(icc, icr);
                coef[4 * p + 1] = __dmul_rn(cc, icr);
                coef[4 * p + 2] = __dmul_rn(icc, cr);
                coef[4 * p + 3] = __dmul_rn(cc, cr);
            }
            const int pr = kh / 2, pc = kw / 2;
            for (int y = tid; y < h; y += KF_THREADS) {
                const int Y = y + pr, I = Y / kh, a = Y - I * kh;
                const int t0 = min(max(I - 1, 0), ntr - 1), t1 = min(I, ntr - 1);
                rinfo[y] = (uint32_t)(t0 * ntc) | ((uint32_t)(t1 * ntc) << 8) | ((uint32_t)(a * kw) << 16);
            }
            for (int x = tid; x < w; x += KF_THREADS) {
                const int X = x + pc, J = X / kw, b = X - J * kw;
                const int u0 = min(max(J - 1, 0), ntc - 1), u1 = min(J, ntc - 1);
                cinfo[x] = (uint32_t)u0 | ((uint32_t)u1 << 8) | ((uint32_t)b << 16);
            }
        }
        __syncthreads();
        mn = red_s[0]; mx = red_s[KF_WARPS];
#pragma unroll
        for (int i = 1; i < KF_WARPS; ++i) { mn = min(mn, red_s[i]); mx = max(mx, red_s[KF_WARPS + i]); }

        // ---- B: 14-bit quantise (round half even) and bin ----
        {
            const double vmin = __dmul_rn((double)mn, intensity_inv), vmax = __dmul_rn((double)mx, intensity_inv);
            const double den = __dsub_rn(vmax, vmin);
            for (int i = tid; i < hw; i += KF_THREADS) {
                const int y = (w == 1) ? i : (int)__umulhi((unsigned)i, w_magic), x = i - y * w;
                const double v = __dmul_rn((double)raw[y * L.pitch + ((e00 + y * wlow) & 7) + x], intensity_inv);
                int q;
                if (mn != mx) q = __double2int_rn(__dmul_rn(__ddiv_rn(__dsub_rn(v, vmin), den), 16383.0));
                else q = __double2int_rn(fmin(fmax(v, 0.0), 16383.0));
                bins[i] = (uint8_t)(q / BIN_SIZE);
            }
        }
        __syncthreads();

        // ---- C: one thread per tile: occupancy mask, redistribution on the bits, prefix counts ----
        for (int t = tid; t < ntiles; t += KF_THREADS) {
            const int ti = ntc == 1 ? t : (int)__umulhi((unsigned)t, k_magic.v[ntc]), tj = t - ti * ntc;
            uint32_t* tw = tiles + t * KF_TILE_WORDS;
#pragma unroll
            for (int k = 0; k < 8; ++k) tw[2 * k] = 0u;
            const int y0 = ti * kh, x0 = tj * kw;
            for (int a = 0; a < kh; ++a) {
                const int y = reflect_idx(y0 + a, h);
                const uint8_t* brow = bins + y * w;
                for (int b = 0; b < kw; ++b) {
                    const int bin = brow[reflect_idx(x0 + b, w)];
                    tw[2 * (bin >> 5)] |= 1u << (bin & 31);
                }
            }
            int set = 0;
#pragma unroll
            for (int k = 0; k < 8; ++k) set += __popc(tw[2 * k]);
            int ex = npix - set;                  // clip at 1: every bin above the limit gives up its surplus
            while (ex > 0) {                      // skimage clip_histogram's redistribution loop, on bits
                const int prev = ex;
                for (int index = 0; index < NBINS; ++index) {
                    const int under = NBINS - set;
                    if (under == 0) break;
                    int step = 1;
                    if (ex <= under) step = ex == 1 ? under : (int)__umulhi((unsigned)under, k_magic.v[ex]);
                    int moved = 0;
                    for (int p = index; p < NBINS; p += step) {
                        uint32_t* wp = tw + 2 * (p >> 5);
                        const uint32_t m = 1u << (p & 31), v = *wp;
                        if (!(v & m)) { *wp = v | m; ++moved; }
                    }
                    ex -= moved; set += moved;
                    if (ex <= 0) break;
                }
                if (prev == ex) break;
            }
            int run = 0;
#pragma unroll
            for (int k = 0; k < 8; ++k) { tw[2 * k + 1] = (uint32_t)run; run += __popc(tw[2 * k]); }
        }
        __syncthreads();

        // ---- D: 4-corner interpolation, fp32 accumulation, truncate to uint16 (dense, over `raw`) ----
        // (the raw pixels are dead: stage B was their last reader)
        int rmn = 65535, rmx = 0;
        for (int i = tid; i < hw; i += KF_THREADS) {
            const int y = (w == 1) ? i : (int)__umulhi((unsigned)i, w_magic), x = i - y * w;
            const uint32_t ri = rinfo[y], ci = cinfo[x];
            const int bin = bins[i];
            const int wsel = 2 * (bin >> 5);
            const uint32_t below = 0xFFFFFFFFu >> (31 - (bin & 31));
            const double* cf = coef + 4 * ((ri >> 16) + (ci >> 16));
            const int tr[2] = {(int)(ri & 255u), (int)((ri >> 8) & 255u)};
            const int tc[2] = {(int)(ci & 255u), (int)((ci >> 8) & 255u)};
            float res = 0.f;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const uint2 mw = *reinterpret_cast<const uint2*>(tiles + (tr[e >> 1] + tc[e & 1]) * KF_TILE_WORDS + wsel);
                const double m = (double)level_tab[mw.y + __popc(mw.x & below)];
                res = __fadd_rn(res, __double2float_rn(__dmul_rn(m, cf[e])));
            }
            const int r = (int)res;
            rmn = min(rmn, r); rmx = max(rmx, r);
            // `raw` still holds staged pixels that OTHER threads may be reading?  No: stage B finished
            // before the barrier above, and stage C / D read bins only.
            raw[i] = (uint16_t)r;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            rmn = min(rmn, __shfl_xor_sync(0xffffffffu, rmn, o));
            rmx = max(rmx, __shfl_xor_sync(0xffffffffu, rmx, o));
        }
        if (lane == 0) { red_s[wid] = rmn; red_s[KF_WARPS + wid] = rmx; }

        // ---- E: per-cell resize tables: source rows / columns, weights, gaussian taps ----
        // (one thread does the scalar fp64 set-up; the loops below read plain integers)
        if (tid == 0) {
            const double fr = __ddiv_rn((double)h, 64.0), fc = __ddiv_rn((double)w, 64.0);
            for (int axis = 0; axis < 2; ++axis) {
                double sg = __dmul_rn(__dsub_rn(axis == 0 ? fr : fc, 1.0), 0.5);
                if (sg < 0.0) sg = 0.0;
                const bool on = sg > 1e-15;
                const int rad = on ? (int)(4.0 * sg + 0.5) : 0;
                rad_s[axis] = on ? rad : -1;                           // -1: this axis is not blurred
                if (on) {
                    // same sums as the general kernel's warp_sum for <= 3 taps: (e0 + e1) + (e2 + 0)
                    const double cf = -0.5 / (sg * sg);
                    double e[3] = {0.0, 0.0, 0.0};
                    for (int k = 0; k <= 2 * rad; ++k) { const double xx = (double)(k - rad); e[k] = exp(cf * xx * xx); }
                    const double ssum = (e[0] + e[1]) + e[2];
                    for (int k = 0; k <= 2 * rad; ++k) gw_s[axis][k] = e[k] / ssum;
                }
            }
            scale_s[0] = fr; scale_s[1] = fc;
        }
        __syncthreads();
        rmn = red_s[0]; rmx = red_s[KF_WARPS];
#pragma unroll
        for (int i = 1; i < KF_WARPS; ++i) { rmn = min(rmn, red_s[i]); rmx = max(rmx, red_s[KF_WARPS + i]); }
        {
            const int axis = tid >> 6, o = tid & 63;                   // 128 threads = 2 axes x 64 outputs
            const int nn = axis == 0 ? h : w;
            const double cc = ((double)o + 0.5) * scale_s[axis] - 0.5;
            const double fl = floor(cc);
            const int i0 = (int)fl;
            ctab_s[axis][o] = cc - fl;
            coord_s[axis][o] = i0;
            // unblurred axis: the two (mirrored) source lines of this output line, as element offsets
            src0_s[axis][o] = mirror_near(i0, nn) * (axis == 0 ? w : 1);
            src1_s[axis][o] = mirror_near(i0 + 1, nn) * (axis == 0 ? w : 1);
        }
        if (levels_out) {                          // test tap: the bit-exact integer core
            uint16_t* dst = levels_out + level_offsets[cell];
            for (int i = tid; i < hw; i += KF_THREADS) dst[i] = raw[i];
        }
        __syncthreads();
        const int rad_r = rad_s[0], rad_c = rad_s[1];

        // The interpolation weights of every output sum to one, so (r - rmn) / den commutes with
        // them: the passes run on the integer levels and the affine map is applied once per output
        // pixel (the general kernel normalises first; the difference is ~1e-16, the gate 1e-5).
        const bool degenerate = rmn == rmx;
        const double lo = degenerate ? fmin(fmax((double)rmn, 0.0), 1.0) : 0.0;
        const double hi = degenerate ? lo : 1.0;
        const double den_rcp = degenerate ? 0.0 : __drcp_rn((double)(rmx - rmn));
        const double nrm_off = degenerate ? lo : -(double)rmn * den_rcp;      // o = raw * den_rcp + nrm_off

        // ---- F + G: a warp takes a block of RB output rows: zoom(+blur) along axis 0 into its row
        // block, then along axis 1, normalise, clip, store ----
        const int RB = w <= 11 ? 16 : (w <= 22 ? 8 : (w <= 44 ? 4 : (w <= 88 ? 2 : 1)));
        double sx[2]; int c0[2], c1[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            sx[e] = ctab_s[1][lane + 32 * e];
            c0[e] = rad_c < 0 ? src0_s[1][lane + 32 * e] : coord_s[1][lane + 32 * e];
            c1[e] = src1_s[1][lane + 32 * e];
        }
        for (int oy0 = wid * RB; oy0 < CIA_CROP; oy0 += KF_WARPS * RB) {
            if (rad_r < 0) {
                for (int i = lane; i < RB * w; i += 32) {
                    const int r = (w == 1) ? i : (int)__umulhi((unsigned)i, w_magic), x = i - r * w;
                    const double t = ctab_s[0][oy0 + r];
                    const double v0 = (double)raw[src0_s[0][oy0 + r] + x], v1 = (double)raw[src1_s[0][oy0 + r] + x];
                    tbuf[i] = (1.0 - t) * v0 + t * v1;
                }
            } else {
                for (int i = lane; i < RB * w; i += 32) {
                    const int r = (w == 1) ? i : (int)__umulhi((unsigned)i, w_magic), x = i - r * w;
                    const double t = ctab_s[0][oy0 + r];
                    const int i0 = coord_s[0][oy0 + r];
                    double v[2];
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int yc = mirror_near(i0 + e, h);
                        double acc = 0.0;
                        for (int k = 0; k <= 2 * rad_r; ++k)
                            acc += gw_s[0][k] * (double)raw[mirror_near(yc + k - rad_r, h) * w + x];
                        v[e] = acc;
                    }
                    tbuf[i] = (1.0 - t) * v[0] + t * v[1];
                }
            }
            __syncwarp();
            for (int r = 0; r < RB; ++r) {
                const double* Trow = tbuf + r * w;
                float* dst32 = crops32 + (size_t)cell * 4096 + (size_t)(oy0 + r) * 64 + lane;
#pragma unroll
                for (int e2 = 0; e2 < 2; ++e2) {
                    double v0, v1;
                    if (rad_c < 0) {
                        v0 = Trow[c0[e2]]; v1 = Trow[c1[e2]];
                    } else {
                        double v[2];
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int xc = mirror_near(c0[e2] + e, w);
                            double acc = 0.0;
                            for (int k = 0; k <= 2 * rad_c; ++k)
                                acc += gw_s[1][k] * Trow[mirror_near(xc + k - rad_c, w)];
                            v[e] = acc;
                        }
                        v0 = v[0]; v1 = v[1];
                    }
                    double o = (1.0 - sx[e2]) * v0 + sx[e2] * v1;
                    o = degenerate ? lo : __fma_rn(o, den_rcp, nrm_off);
                    if (WANT64) {
                        o = fmin(fmax(o, lo), hi);
                        crops64[(size_t)cell * 4096 + (size_t)(oy0 + r) * 64 + lane + 32 * e2] = o;
                    }
                    dst32[32 * e2] = fminf(fmaxf((float)o, (float)lo), (float)hi);
                }
            }
            __syncwarp();
        }
    }
}

}  // namespace

int k_crop_resize(cia_ctx* h, const uint16_t* images, int H, int W, const cia_cell* cells,
                  int n_cells, const int32_t* n_cells_dev, const cia_params* p, float* crops32,
                  double* crops64, cudaStream_t s, uint16_t* levels_out,
                  const int64_t* level_offsets) {
    if (n_cells <= 0) return CIA_OK;
    const size_t lo_bytes = 92 * 1024, hi_bytes = 206 * 1024;   // 2 CTAs/SM and 1 CTA/SM with the 19.5 KB static part
    // fast-path classes by shared-memory need: 8 (the register limit at 64 per thread) / 5 resident CTAs per SM
    const FastBytes fb = {{26 * 1024, 42 * 1024}};
    const int fast_ctas[KF_CLASSES] = {8, 5};
    if (first_use(h, (const void*)crop_clahe_resize_kernel))
        CIA_CUDA(cudaFuncSetAttribute(crop_clahe_resize_kernel,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hi_bytes));
    auto fast = crops64 ? crop_fast_kernel<true> : crop_fast_kernel<false>;
    if (first_use(h, (const void*)fast)) {
        CIA_CUDA(cudaFuncSetAttribute(fast, cudaFuncAttributeMaxDynamicSharedMemorySize, fb.v[KF_CLASSES - 1]));
        CIA_CUDA(cudaFuncSetAttribute(fast, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    }
    const int huge_ctas = 32;
    const size_t per_cta = cell_bytes(MAX_SIDE, MAX_SIDE, 15, 15);
    // [class counters + work counters (256 B)] [6 lists of n ints] [global scratch of the class-2 CTAs]
    constexpr int NCLS = KF_CLASSES + 3;
    const size_t list_stride = (((size_t)n_cells + 63) / 64) * 64;
    const size_t list_bytes = list_stride * sizeof(int32_t);
    int rc = ws_reserve(h, h->ws_crop_scratch, 256 + NCLS * list_bytes + per_cta * huge_ctas);
    if (rc) return rc;
    unsigned char* wsb = (unsigned char*)h->ws_crop_scratch.p;
    int32_t* cls_counts = (int32_t*)wsb;                 // [0..NCLS): list lengths, [16..16+KF_CLASSES): work counters
    int32_t* work = cls_counts + 16;
    int32_t* lists = (int32_t*)(wsb + 256);
    unsigned char* gscratch = wsb + 256 + NCLS * list_bytes;
    CIA_CUDA(cudaMemsetAsync(cls_counts, 0, 256, s));
    {
        int cb = (n_cells + 255) / 256;
        if (cb > h->num_sms * 4) cb = h->num_sms * 4;
        crop_classify_all_kernel<<<cb, 256, 0, s>>>(cells, n_cells, n_cells_dev, p->clip_limit, fb, lo_bytes,
                                                    hi_bytes, cls_counts, lists, list_stride);
        CIA_LAUNCH_CHECK();
    }
    for (int c = 0; c < KF_CLASSES; ++c) {
        int g = h->num_sms * fast_ctas[c];
        if (g > n_cells) g = n_cells;
        fast<<<g, KF_THREADS, fb.v[c], s>>>(images, H, W, cells, p->intensity_inv, crops32, crops64,
                                                        lists + c * list_stride, cls_counts + c, work + c,
                                                        levels_out, level_offsets);
        CIA_LAUNCH_CHECK();
    }
    int g0 = h->num_sms * 2; if (g0 > n_cells) g0 = n_cells;
    int g1 = h->num_sms;     if (g1 > n_cells) g1 = n_cells;
    int g2 = huge_ctas;      if (g2 > n_cells) g2 = n_cells;
    const int gg[3] = {g0, g1, g2};
    const size_t gsm[3] = {lo_bytes, hi_bytes, 0};
    for (int c = 0; c < 3; ++c) {
        crop_clahe_resize_kernel<<<gg[c], K2_THREADS, gsm[c], s>>>(
            images, H, W, cells, n_cells, n_cells_dev, p->clip_limit, p->intensity_inv, crops32, crops64, c,
            lo_bytes, hi_bytes, c == 2 ? gscratch : nullptr, c == 2 ? per_cta : 0, h->status_dev, levels_out,
            level_offsets, lists + (KF_CLASSES + c) * list_stride, cls_counts + KF_CLASSES + c);
        CIA_LAUNCH_CHECK();
    }
    return CIA_OK;
}
