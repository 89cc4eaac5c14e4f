// segment.cu -- N2: StarDist2D inference on the GPU, the producer of the int32 label field of the hot path
// (improved_detection.py:44, 62-63; CAE_improved_modeltrain.py:53-55):
//
//     normalized = csbdeep.utils.normalize(seg_channel)              -> seg_hist / seg_percentile / seg_normalize
//     labels, _  = stardist_model.predict_instances(normalized)      -> U-Net (seg_first / seg_conv), candidates,
//                                                                       polygon NMS, label rendering
//
// stardist / csbdeep are third-party packages absent from /root/reference and from this image; the algorithm is
// restated from their published description (oracle/stardist.py + oracle/stardist_post.c: "parity unpinned").
//
// U-Net (csbdeep unet_block behind StarDist2D._build): every 3x3 convolution except the first (Cin = 1) is a
// tcgen05 implicit GEMM over fp16 activations in chunk-planar order [C/8][y][x][8] (16 bytes = one pixel's 8
// channels = one row of a K-major UMMA core matrix, the layout of cae_tc.cu).  A unit is a 16-row x 8*TILES-column
// output tile: its zero-padded (18 x 8*TILES+2) input block of 32 channels sits in shared memory ONCE per
// 32-channel chunk and serves all nine taps through shifted descriptor start addresses (no im2col); max-pooling
// and "nearest up-sampling + concatenate with the skip" are folded into the staging, so neither is a kernel or a
// trip through HBM.  Accumulators (TILES x N fp32 columns) live in TMEM.  Three forms of the same arithmetic,
// chosen per layer (launch_seg_layer):
//   seg_conv_tma_kernel  Cin = 32 layers that read their producer directly: a cp.async.bulk.tensor box per unit into a
//                        3-stage ring (out-of-bounds zero fill = the padding), producer / MMA / epilogue warps, two
//                        TMEM accumulator sets: the epilogue of unit u runs under the MMAs of unit u + 1
//   seg_conv_ws_kernel   the same pipeline with eight SOFTWARE producer warps (pooled / up-sampled + concatenated /
//                        multi-chunk inputs with their weight blocks): layers with long MMA phases per step
//   seg_conv_kernel      stage -> MMA -> epilogue in sequence, up to four CTAs per SM interleaving: the rest
// The 1x1 heads (prob: sigmoid, dist: linear, floor 1e-3) are seg_heads_tma_kernel (all feature channels of a
// 16 x 16 tile per box, N = 48).
//
// Post-processing: candidates (prob > threshold, 2-pixel border excluded) are sorted by probability (cub radix
// sort), binned on a 32-px lattice (counting sort), and suppressed greedily IN PARALLEL with the sequential algorithm's
// exact result: a candidate becomes a winner once every better candidate whose bounding circle reaches it is decided;
// the winners of a round then suppress their undecided neighbours by the polygon overlap (intersection / smaller
// area > threshold; the intersection of two star-convex polygons as the sum over their triangle fans' pairwise
// clipped areas: a float32 partial sum as a rigorous lower bound first, the exact fp64 sum where that does not
// decide, one warp per pair).  One cooperative kernel runs all rounds.  Kept polygons are rendered with
// skimage.draw.polygon's point-in-polygon rule, the better polygon winning a pixel (atomicMin).
#include "common.cuh"
#include "tc_ptx.cuh"

#include <cooperative_groups.h>
#include <cub/cub.cuh>
#include <cuda.h>          // CUtensorMap (types only; the encoder is fetched through the runtime)
#include <cuda_fp16.h>

#include <cmath>

namespace cg = cooperative_groups;

namespace {
using namespace tcptx;

constexpr int SEG_RAYS = 32;         // n_rays of the tensor-core head kernel (2D_versatile_fluo, StarDist's default)
constexpr int SEG_BIN = 32;          // lattice pitch of the candidate bins in pixels
constexpr int SEG_KC = 32;           // input channels per shared-memory chunk

struct SegConv {
    int cin = 0, cout = 0, taps = 9;
    int n_tile = 0, groups = 0, chunks = 0;     // Cout columns per CTA, Cout / n_tile, Cin / 32
    __half* w_img = nullptr;                    // [group][chunk][tap][4][n_tile][8] fp16
    float* bias = nullptr;                      // [groups * n_tile]
    float* w32 = nullptr;                       // first layer only: [9][cout] fp32
};
struct SegOp {
    int layer, mode;             // mode -1: first layer (fp32 image in); 0 direct; 1 2x2 max-pool of src0; 2 up(src0) ++ src1
    int src0, src1, dst;         // activation buffer ids
    int c0, c1;                  // channels of src0 / src1
    int shift;                   // output resolution = field >> shift
    int pool_dst;                // >= 0: buffer for the 2x2 max-pooled copy of the output (the next layer pools this one)
    int full_needed;             // the full-resolution output is read as well (a skip connection)
};

}  // namespace

struct SegModel {
    int grid = 2, depth = 3, n_conv = 2, base = 32, after = 128, n_rays = 32;
    std::vector<SegConv> conv;
    std::vector<SegOp> ops;
    std::vector<int> buf_ch, buf_shift;
    double* ray_sin = nullptr;   // [n_rays] np.sin(np.linspace(0, 2 pi, n_rays, endpoint=False)), from the host
    double* ray_cos = nullptr;
    Workspace act, post, cubtmp;
    Workspace screen;            // cia_screen_images: normalized padded fields, labels when the caller keeps none
    // pointers into `post` of the last cia_seg_instances call (details of the kept polygons)
    int last_cap = 0;
    float *vy = nullptr, *vx = nullptr, *pprob = nullptr;
    int *pyx = nullptr, *kept_rank = nullptr, *n_kept = nullptr;
    float* prob_map = nullptr;   // heads' outputs of the last cia_seg_predict (inside `act`)
    float* dist_map = nullptr;
    int last_hg = 0, last_wg = 0;
};

namespace {

// ---------------------------------------------------------------------------------------
// csbdeep.utils.normalize: np.percentile (linear interpolation) of a uint16 image from its exact histogram
// ---------------------------------------------------------------------------------------
// Every kernel of the normalisation takes the field from blockIdx.y (blockIdx.x for the one-CTA percentile): csbdeep
// normalizes each image by its own percentiles, so each field has its own histogram copies, wsum and (mi, ma).
constexpr int SEG_HIST_COPIES = 16;   // copies of the histogram (by CTA): the background's few grey levels are hot addresses
constexpr size_t SEG_HIST_FIELD = (size_t)SEG_HIST_COPIES * 65536;   // histogram words per field

__global__ void seg_hist_kernel(const uint16_t* __restrict__ img, size_t n, uint32_t* __restrict__ hist) {
    img += (size_t)blockIdx.y * n;
    hist += (size_t)blockIdx.y * SEG_HIST_FIELD + (size_t)(blockIdx.x % SEG_HIST_COPIES) * 65536;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31;
    for (size_t i0 = (size_t)blockIdx.x * blockDim.x; i0 < n; i0 += stride) {     // warp-uniform trip count
        const size_t i = i0 + threadIdx.x;
        const bool ok = i < n;
        const unsigned v = ok ? img[i] : 0x10000u;
        const unsigned peers = __match_any_sync(0xffffffffu, v);
        if (ok && lane == __ffs(peers) - 1) atomicAdd(hist + v, (uint32_t)__popc(peers));
    }
}

// copy 0 += copies 1..15; wsum[b / 32] = population of 32 consecutive bins (what the selection kernel scans)
__global__ void seg_hist_reduce_kernel(uint32_t* __restrict__ hist, uint32_t* __restrict__ wsum) {
    hist += (size_t)blockIdx.y * SEG_HIST_FIELD;
    wsum += (size_t)blockIdx.y * 2048;
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t c = 0;
    for (int cp = 0; cp < SEG_HIST_COPIES; ++cp) c += hist[(size_t)cp * 65536 + b];
    hist[b] = c;
    const uint32_t w = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0) wsum[b >> 5] = w;
}

// numpy's percentile for the default method: virtual index n q + (1 + q (1 - 1 - 1)) - 1, the two neighbouring order
// statistics a <= b and _lerp(a, b, t) = a + (b - a) t, or b - (b - a)(1 - t) where t >= 0.5 (numpy/lib/_function_base_impl.py)
__global__ void __launch_bounds__(1024) seg_percentile_kernel(const uint32_t* __restrict__ hist, const uint32_t* __restrict__ wsum,
                                                              size_t n, double q_lo, double q_hi, float* __restrict__ mi_ma) {
    hist += (size_t)blockIdx.x * SEG_HIST_FIELD;
    wsum += (size_t)blockIdx.x * 2048;
    mi_ma += 2 * blockIdx.x;
    typedef cub::BlockScan<unsigned long long, 1024> Scan;
    __shared__ typename Scan::TempStorage tmp;
    __shared__ unsigned s_val[4];
    const int t = threadIdx.x;
    unsigned long long local = 0;
    local = (unsigned long long)wsum[2 * t] + wsum[2 * t + 1];      // bins [64 t, 64 t + 64)
    unsigned long long before;
    Scan(tmp).ExclusiveSum(local, before);
    long long want[4];
    double gam[2];
    for (int p = 0; p < 2; ++p) {
        const double q = p ? q_hi : q_lo;
        const double virt = __dsub_rn(__dadd_rn(__dmul_rn((double)n, q), __dadd_rn(1.0, __dmul_rn(q, -1.0))), 1.0);
        long long prev = (long long)floor(virt), next = prev + 1;
        if (virt >= (double)(n - 1)) { prev = (long long)n - 1; next = prev; }
        if (virt < 0) { prev = 0; next = 0; }          // numpy clips negative indexes to the first element
        want[2 * p] = prev; want[2 * p + 1] = next;
        gam[p] = __dsub_rn(virt, floor(virt));
    }
    for (int w = 0; w < 4; ++w) {
        if ((unsigned long long)want[w] >= before && (unsigned long long)want[w] < before + local) {
            unsigned long long c = before;
            for (int k = 0; k < 64; ++k) {
                c += hist[t * 64 + k];
                if ((unsigned long long)want[w] < c) { s_val[w] = (unsigned)(t * 64 + k); break; }
            }
        }
    }
    __syncthreads();
    if (t == 0) {
        for (int p = 0; p < 2; ++p) {
            const double a = (double)s_val[2 * p], b = (double)s_val[2 * p + 1], g = gam[p];
            const double d = __dsub_rn(b, a);
            double r = __dadd_rn(a, __dmul_rn(d, g));
            if (g >= 0.5) r = __dsub_rn(b, __dmul_rn(d, __dsub_rn(1.0, g)));
            mi_ma[p] = (float)r;
        }
    }
}

// np.pad(mode='reflect') source index of padded position i along a side of n pixels (the reflection is periodic
// with period 2 (n - 1), as numpy's repeated reflection of pads wider than the image)
__device__ __forceinline__ int seg_reflect(int i, int n) {
    if (i < n) return i;
    if (n == 1) return 0;
    const int p = 2 * (n - 1), k = i % p;
    return k < n ? k : p - k;
}

// normalize_mi_ma(x, mi, ma, clip=False, eps=1e-20, dtype=float32): (x - mi) / (ma - mi + eps) in float32, written
// straight into the field's reflect-padded [Hp][Wp] frame (a pointwise map commutes with the padding)
__global__ void seg_normalize_kernel(const uint16_t* __restrict__ img, int H, int W, int Hp, int Wp,
                                     const float* __restrict__ mi_ma, float eps, float* __restrict__ out) {
    img += (size_t)blockIdx.y * H * W;
    out += (size_t)blockIdx.y * Hp * Wp;
    mi_ma += 2 * blockIdx.y;
    const float mi = mi_ma[0], den = __fadd_rn(__fsub_rn(mi_ma[1], mi), eps);
    const size_t stride = (size_t)gridDim.x * blockDim.x, n = (size_t)Hp * Wp;
    if (Hp == H && Wp == W) {
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
            out[i] = __fdiv_rn(__fsub_rn((float)img[i], mi), den);
        return;
    }
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int y = (int)(i / Wp), x = (int)(i - (size_t)y * Wp);
        const size_t src = (size_t)seg_reflect(y, H) * W + seg_reflect(x, W);
        out[i] = __fdiv_rn(__fsub_rn((float)img[src], mi), den);
    }
}

// ---------------------------------------------------------------------------------------
// U-Net
// ---------------------------------------------------------------------------------------
// First layer, Cin = 1 (K = 9: no tensor-core shape): one thread per PAIR of horizontally adjacent pixels (W is even:
// field sides are multiples of 16), packed fp32x2 FMAs (the pixel value in both lanes, two output channels per
// instruction, each lane an IEEE fma: bias first, taps in order), every 128-bit weight read from shared memory serves
// both pixels, fp16 chunk-planar output.
__global__ void __launch_bounds__(256) seg_first_kernel(const float* __restrict__ img, const float* __restrict__ w,
                                                        const float* __restrict__ bias, __half* __restrict__ out, int H,
                                                        int W, int cout, int F) {
    extern __shared__ __align__(16) float sw[];   // [9][cout] weights, [cout] bias
    for (int i = threadIdx.x; i < 10 * cout; i += blockDim.x) sw[i] = i < 9 * cout ? w[i] : bias[i - 9 * cout];
    __syncthreads();
    const int Wp = (W + 1) >> 1;
    const size_t idx0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx0 >= (size_t)F * H * Wp) return;
    const int f = (int)(idx0 / ((size_t)H * Wp));      // fields [F][H][W] in, [F][cout/8][H][W][8] out
    const size_t idx = idx0 - (size_t)f * H * Wp;
    img += (size_t)f * H * W;
    out += (size_t)f * cout * H * W;
    const int y = (int)(idx / Wp), x = 2 * (int)(idx - (size_t)y * Wp);
    const bool two = x + 1 < W;
    float win[3][4];                               // rows y-1..y+1, columns x-1..x+2
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int yy = y + r - 1, xx = x + c - 1;
            win[r][c] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? __ldg(img + (size_t)yy * W + xx) : 0.f;
        }
    unsigned long long va[9], vb[9];
#pragma unroll
    for (int t = 0; t < 9; ++t) {
        va[t] = pack2(win[t / 3][t % 3], win[t / 3][t % 3]);
        vb[t] = pack2(win[t / 3][t % 3 + 1], win[t / 3][t % 3 + 1]);
    }
    const ulonglong2* sw2 = reinterpret_cast<const ulonglong2*>(sw);
    for (int cgp = 0; cgp < cout / 8; ++cgp) {
        unsigned long long aa[4], ab[4];
        {
            const ulonglong2 b0 = sw2[(9 * cout + cgp * 8) / 4], b1 = sw2[(9 * cout + cgp * 8) / 4 + 1];
            aa[0] = ab[0] = b0.x; aa[1] = ab[1] = b0.y; aa[2] = ab[2] = b1.x; aa[3] = ab[3] = b1.y;
        }
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const ulonglong2 w0 = sw2[(t * cout + cgp * 8) / 4], w1 = sw2[(t * cout + cgp * 8) / 4 + 1];
            aa[0] = fma2(va[t], w0.x, aa[0]); aa[1] = fma2(va[t], w0.y, aa[1]);
            aa[2] = fma2(va[t], w1.x, aa[2]); aa[3] = fma2(va[t], w1.y, aa[3]);
            ab[0] = fma2(vb[t], w0.x, ab[0]); ab[1] = fma2(vb[t], w0.y, ab[1]);
            ab[2] = fma2(vb[t], w1.x, ab[2]); ab[3] = fma2(vb[t], w1.y, ab[3]);
        }
        __align__(16) __half oa[8], ob[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float lo, hi;
            unpack2(aa[k], lo, hi);
            oa[2 * k] = __float2half_rn(fmaxf(lo, 0.f)); oa[2 * k + 1] = __float2half_rn(fmaxf(hi, 0.f));
            unpack2(ab[k], lo, hi);
            ob[2 * k] = __float2half_rn(fmaxf(lo, 0.f)); ob[2 * k + 1] = __float2half_rn(fmaxf(hi, 0.f));
        }
        __half* dst = out + (((size_t)cgp * H + y) * W + x) * 8;
        *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(oa);
        if (two) *reinterpret_cast<uint4*>(dst + 8) = *reinterpret_cast<const uint4*>(ob);
    }
}

struct SegConvArgs {
    const __half* src0;
    const __half* src1;
    const uint4* w;
    const float* bias;
    __half* out;
    float* prob;
    float* dist;
    int H, W;            // output resolution
    int F;               // fields: every map is [F][...] with the field outermost, units are decomposed per field
    int c0, c1, mode, ntaps, groups, chunks;
    // seg_conv_tma_kernel: POOL 1 / 2 also writes (only writes) MaxPooling2D((2, 2)) of the output for the next layer
    __half* out_pool;
};

template <int N, int TILES>
struct SegCfg {
    static constexpr int COLS = 8 * TILES + 2;
    static constexpr int ROW_B = COLS * 16;
    static constexpr int PLANE_B = 18 * ROW_B;            // = LBO of A (next 8 channels)
    static constexpr int A_B = (SEG_KC / 8) * PLANE_B;
    static constexpr int WT_B = (SEG_KC / 8) * N * 16;    // one tap of one 32-channel chunk
    static constexpr int W_B = 9 * WT_B;
    static constexpr int SMEM_B = A_B + W_B;
    static constexpr int TMEM_COLS = pow2_cols(TILES * N);
    static constexpr int NU = (SEG_KC / 8) * 18 * COLS;   // 16-byte units of one staged block
    // CTAs that share an SM (512 TMEM columns, 227 KB of shared memory): their stage -> MMA -> epilogue chains interleave
    static constexpr int BY_TMEM = 512 / TMEM_COLS, BY_SMEM = (227 * 1024) / (SMEM_B + 2048);
    static constexpr int CTAS_PER_SM = (BY_TMEM < BY_SMEM ? BY_TMEM : BY_SMEM) > 4 ? 4 : (BY_TMEM < BY_SMEM ? BY_TMEM : BY_SMEM);
};

__device__ __forceinline__ uint4 hmax8(uint4 a, uint4 b) {
    uint4 r;
    const __half2* pa = reinterpret_cast<const __half2*>(&a);
    const __half2* pb = reinterpret_cast<const __half2*>(&b);
    __half2* pr = reinterpret_cast<__half2*>(&r);
#pragma unroll
    for (int k = 0; k < 4; ++k) pr[k] = __hmax2(pa[k], pb[k]);
    return r;
}

// One 16-byte unit (8 channels of plane `pl` of the layer's input at output-resolution pixel (y, x)), with the
// pooling / up-sampling / concatenation of the U-Net folded in.
// s0 / s1: the unit's field of src0 / src1 (seg_src).
__device__ __forceinline__ uint4 seg_load(const SegConvArgs& a, const uint4* s0, const uint4* s1, int pl, int y, int x) {
    if (a.mode == 0) return __ldg(s0 + ((size_t)pl * a.H + y) * a.W + x);
    if (a.mode == 1) {                                   // MaxPooling2D((2, 2)) of the producer's 2H x 2W map
        const size_t Ws = 2 * (size_t)a.W;
        const uint4* p = s0 + ((size_t)pl * 2 * a.H + 2 * y) * Ws + 2 * x;
        return hmax8(hmax8(__ldg(p), __ldg(p + 1)), hmax8(__ldg(p + Ws), __ldg(p + Ws + 1)));
    }
    const int p0 = a.c0 >> 3;                            // Concatenate([UpSampling2D((2, 2))(low), skip])
    if (pl < p0) return __ldg(s0 + ((size_t)pl * (a.H >> 1) + (y >> 1)) * (a.W >> 1) + (x >> 1));
    return __ldg(s1 + ((size_t)(pl - p0) * a.H + y) * a.W + x);
}

// field f of the layer's inputs: src0 holds c0 channels at the resolution its mode implies, src1 c1 at the output's
__device__ __forceinline__ void seg_src(const SegConvArgs& a, int f, const uint4*& s0, const uint4*& s1) {
    const size_t px = (size_t)a.H * a.W;
    const size_t px0 = a.mode == 1 ? 4 * px : a.mode == 2 ? (size_t)(a.H >> 1) * (a.W >> 1) : px;
    s0 = reinterpret_cast<const uint4*>(a.src0) + (size_t)f * (a.c0 >> 3) * px0;
    s1 = reinterpret_cast<const uint4*>(a.src1) + (size_t)f * (a.c1 >> 3) * px;
}

// EPI 0: bias + ReLU -> fp16 chunk-planar;  EPI 1: heads (columns 0..31 dist = max(1e-3, .), column 32 prob = sigmoid)
template <int N, int TILES, int EPI>
__global__ void __launch_bounds__(256, SegCfg<N, TILES>::CTAS_PER_SM) seg_conv_kernel(const SegConvArgs a) {
    using C = SegCfg<N, TILES>;
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_base_s;
    unsigned char* sa = smem;
    unsigned char* sw = smem + C::A_B;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    const int tiles_x = (a.W + 8 * TILES - 1) / (8 * TILES), tiles_y = (a.H + 15) / 16;
    const int per_field = tiles_x * tiles_y;
    const int n_units = per_field * a.F * a.groups;
    if ((int)blockIdx.x >= n_units) return;               // uniform: nothing allocated yet

    if (warp == 0) tmem_alloc(&tmem_base_s, C::TMEM_COLS);
    if (tid == 32) { mbar_init(&bar, TILES); fence_barrier_init(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    constexpr uint32_t IDESC = make_idesc(128, N);
    const int w_units = a.ntaps * (C::WT_B / 16);        // 16-byte units of one (group, chunk) weight block
    const bool resident = a.chunks == 1 && a.groups == 1;
    bool w_loaded = false;
    uint32_t phase = 0;

    for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
        const int g = unit / (per_field * a.F);               // unit = (group, field, tile)
        const int fu = unit - g * (per_field * a.F);
        const int f = fu / per_field, t2 = fu - f * per_field;
        const int ty = t2 / tiles_x, tx = t2 - ty * tiles_x;
        const int y0 = 16 * ty, x0 = 8 * TILES * tx;
        const uint4 *s0, *s1;
        seg_src(a, f, s0, s1);
        const size_t fpx = (size_t)f * a.H * a.W;

        for (int kc = 0; kc < a.chunks; ++kc) {
            if (!(resident && w_loaded)) {
                const uint4* wsrc = a.w + (size_t)(g * a.chunks + kc) * w_units;
                for (int i = tid; i < w_units; i += 256) reinterpret_cast<uint4*>(sw)[i] = __ldg(wsrc + i);
            }
            // input block: two batches of independent 16-byte requests per thread, all of a batch in flight before
            // any store (a block costs two memory round trips)
            constexpr int SB = ((C::NU + 255) / 256 + 1) / 2;
#pragma unroll 1
            for (int i0 = tid; i0 < C::NU; i0 += SB * 256) {
                uint4 v[SB];
                uint32_t d[SB];
#pragma unroll
                for (int j = 0; j < SB; ++j) {
                    const int idx = i0 + j * 256;
                    d[j] = 0xFFFFFFFFu;
                    v[j] = make_uint4(0, 0, 0, 0);
                    if (idx < C::NU) {
                        const int c = idx / (18 * C::COLS);
                        const int rem = idx - c * (18 * C::COLS);
                        const int ry = rem / C::COLS, rc = rem - ry * C::COLS;
                        const int y = y0 + ry - 1, x = x0 + rc - 1;
                        d[j] = (uint32_t)idx * 16u;
                        // a one-tap layer (the heads) never reads the halo ring
                        const bool halo = a.ntaps == 1 && (ry == 0 || ry == 17 || rc == 0 || rc == C::COLS - 1);
                        if (!halo && y >= 0 && y < a.H && x >= 0 && x < a.W) v[j] = seg_load(a, s0, s1, kc * (SEG_KC / 8) + c, y, x);
                    }
                }
#pragma unroll
                for (int j = 0; j < SB; ++j)
                    if (d[j] != 0xFFFFFFFFu) *reinterpret_cast<uint4*>(sa + d[j]) = v[j];
            }
            fence_async_smem();
            tc_fence_before();
            __syncthreads();
            tc_fence_after();
            if (warp < TILES && lane == 0) {              // one issuing lane per tile (independent accumulators)
                const uint64_t ad0 = make_smem_desc(smem_u32(sa) + (uint32_t)(warp * 8 * 16), C::PLANE_B, C::ROW_B);
                const uint64_t bd0 = make_smem_desc(smem_u32(sw), N * 16, 128);
                const uint32_t d_tmem = tmem_base + (uint32_t)(warp * N);
                for (int tap = 0; tap < a.ntaps; ++tap) {
                    const int dy = a.ntaps == 1 ? 1 : tap / 3, dx = a.ntaps == 1 ? 1 : tap % 3;
#pragma unroll
                    for (int s = 0; s < SEG_KC / 16; ++s) {
                        const uint64_t ad = ad0 + (uint64_t)((dx * 16 + dy * C::ROW_B + 2 * s * C::PLANE_B) >> 4);
                        const uint64_t bd = bd0 + (uint64_t)(((tap * (SEG_KC / 8) + 2 * s) * N * 16) >> 4);
                        umma_f16(d_tmem, ad, bd, IDESC, (kc == 0 && tap == 0 && s == 0) ? 0u : 1u);
                    }
                }
                umma_commit(&bar);
            }
            __syncwarp();
            mbar_wait(&bar, phase);                        // MMAs done: the blocks may be overwritten, TMEM read
            phase ^= 1u;
            tc_fence_after();
        }
        w_loaded = true;

        // ---- epilogue: TMEM lane r = output pixel (row r >> 3, column 8 t + (r & 7)) of tile t ----
        const int q = warp & 3, half_sel = warp >> 2;
        const int r = 32 * q + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * q) << 16);
        const int y = y0 + (r >> 3);
        if (EPI == 0) {
            constexpr int SL = N / 8;
#pragma unroll 1
            for (int p = half_sel; p < TILES * SL; p += 2) {
                const int t = p / SL, sl = p - t * SL;
                const int x = x0 + 8 * t + (r & 7);
                uint32_t v[8];
                TMEM_LD8(lane_addr + (uint32_t)(t * N + sl * 8), v);
                TMEM_WAIT8(v);
                const int c0 = g * N + sl * 8;
                __align__(16) __half o[8];
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    o[k] = __float2half_rn(fmaxf(__fadd_rn(__uint_as_float(v[k]), __ldg(a.bias + c0 + k)), 0.f));
                if (y < a.H && x < a.W)
                    *reinterpret_cast<uint4*>(a.out + fpx * a.groups * N + (((size_t)(c0 >> 3) * a.H + y) * a.W + x) * 8) =
                        *reinterpret_cast<const uint4*>(o);
            }
        } else {
            constexpr int SL = SEG_RAYS / 8 + 1;           // four dist slices + the slice whose first column is prob
#pragma unroll 1
            for (int p = half_sel; p < TILES * SL; p += 2) {
                const int t = p / SL, sl = p - t * SL;
                const int x = x0 + 8 * t + (r & 7);
                uint32_t v[8];
                TMEM_LD8(lane_addr + (uint32_t)(t * N + sl * 8), v);
                TMEM_WAIT8(v);
                if (y < a.H && x < a.W) {
                    const size_t px = fpx + (size_t)y * a.W + x;
                    if (sl < SEG_RAYS / 8) {
                        float o[8];
#pragma unroll
                        for (int k = 0; k < 8; ++k)       // dist = np.maximum(1e-3, dist) (StarDist2D.predict)
                            o[k] = fmaxf(1e-3f, __fadd_rn(__uint_as_float(v[k]), __ldg(a.bias + sl * 8 + k)));
                        float4* dd = reinterpret_cast<float4*>(a.dist + px * SEG_RAYS + sl * 8);
                        dd[0] = make_float4(o[0], o[1], o[2], o[3]);
                        dd[1] = make_float4(o[4], o[5], o[6], o[7]);
                    } else {
                        const float z = __fadd_rn(__uint_as_float(v[0]), __ldg(a.bias + SEG_RAYS));
                        a.prob[px] = 1.f / (1.f + expf(-z));
                    }
                }
            }
        }
        // the next unit's MMAs overwrite these accumulators: ordered by the fence + barrier before their issue
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, C::TMEM_COLS);
}

// ---------------------------------------------------------------------------------------
// The same convolution for layers that read their producer directly with Cin = 32 (one chunk, weights resident:
// the two full-resolution layers, `features`, the second layer of a level): TMA-fed and warp-specialised.
//   warp 8  : one lane issues a cp.async.bulk.tensor.4d box (8 halves, 8 TILES + 2 columns, 18 rows, 4 planes) per
//             unit into a 3-stage ring; out-of-bounds coordinates zero-fill the halo ('same' padding for free)
//   warp 9  : one elected lane issues the unit's 18 TILES MMAs into one of two TMEM accumulator sets and commits to the
//             stage's `empty` barrier (the block is free) and the set's `full` barrier
//   warps 0-7: epilogue of unit u (tcgen05.ld, bias, ReLU, fp16, 16-byte stores) under the MMAs of unit u + 1
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2,%3,%4,%5}], [%6];"
        ::"r"(dst), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(bar)) : "memory");
}

template <int N, int TILES>
struct SegTmaCfg {
    using B = SegCfg<N, TILES>;
    static constexpr int STAGES = 3;
    static constexpr int A_STRIDE = (B::A_B + 1023) / 1024 * 1024;
    static constexpr int SMEM_B = STAGES * A_STRIDE + B::W_B;
    static constexpr int TMEM_COLS = pow2_cols(2 * TILES * N);
    static constexpr int THREADS = 320;
    static_assert(TMEM_COLS <= 512 && SMEM_B <= 225 * 1024, "does not fit");
};

// POOL 0: the layer's output; 1: only its 2x2 max-pooled copy (the full-resolution map is read by nobody else: it never
// exists in HBM); 2: both (a skip connection).  The four pool partners of a pixel are lanes l, l ^ 1 (column), l ^ 8 (row)
// of one warp; max of the rounded halves = rounding of the max, so the consumer sees what pooling the stored map gives.
template <int N, int TILES, int POOL>
__global__ void __launch_bounds__(320, 1) seg_conv_tma_kernel(const __grid_constant__ CUtensorMap tm, const uint4* __restrict__ w,
                                                              const float* __restrict__ bias, __half* __restrict__ out,
                                                              __half* __restrict__ out_pool, int H, int W, int F) {
    using C = SegCfg<N, TILES>;
    using T = SegTmaCfg<N, TILES>;
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ __align__(8) uint64_t full[T::STAGES], empty[T::STAGES], tfull[2], tempty[2];
    __shared__ uint32_t tmem_base_s;
    unsigned char* sw = smem + T::STAGES * T::A_STRIDE;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // unit = (field, tile); the tensor map's outermost dimension is field * 4 + plane, so a box at plane 4 f reads
    // field f only and the y / x out-of-bounds zero fill is that field's own padding
    const int tiles_x = (W + 8 * TILES - 1) / (8 * TILES), tiles_y = (H + 15) / 16;
    const int per_field = tiles_x * tiles_y;
    const int n_units = per_field * F;
    if ((int)blockIdx.x >= n_units) return;

    if (warp == 0) tmem_alloc(&tmem_base_s, T::TMEM_COLS);
    if (tid == 32) {
        for (int s = 0; s < T::STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(&tfull[0], 1); mbar_init(&tfull[1], 1);
        mbar_init(&tempty[0], 8); mbar_init(&tempty[1], 8);
        fence_barrier_init();
    }
    for (int i = tid; i < C::W_B / 16; i += T::THREADS) reinterpret_cast<uint4*>(sw)[i] = __ldg(w + i);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    constexpr uint32_t IDESC = make_idesc(128, N);

    if (warp == 8) {
        if (lane == 0) {
            int j = 0;
            for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++j) {
                const int s = j % T::STAGES;
                mbar_wait(&empty[s], (uint32_t)(((j / T::STAGES) & 1) ^ 1));
                const int f = unit / per_field, t2 = unit - f * per_field;
                const int ty = t2 / tiles_x, tx = t2 - ty * tiles_x;
                mbar_expect_tx(&full[s], C::A_B);
                tma_load_4d(smem_u32(smem + s * T::A_STRIDE), &tm, 0, 8 * TILES * tx - 1, 16 * ty - 1, 4 * f, &full[s]);
            }
        }
    } else if (warp == 9) {
        int j = 0;
        for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++j) {
            const int s = j % T::STAGES, t = j & 1;
            mbar_wait(&full[s], (uint32_t)((j / T::STAGES) & 1));
            mbar_wait(&tempty[t], (uint32_t)(((j >> 1) & 1) ^ 1));
            tc_fence_after();
            if (elect_one()) {
                const uint64_t ad0 = make_smem_desc(smem_u32(smem + s * T::A_STRIDE), C::PLANE_B, C::ROW_B);
                const uint64_t bd0 = make_smem_desc(smem_u32(sw), N * 16, 128);
                const uint32_t d0 = tmem_base + (uint32_t)(t * TILES * N);
#pragma unroll
                for (int tap = 0; tap < 9; ++tap) {
                    const int dy = tap / 3, dx = tap % 3;
#pragma unroll
                    for (int ks = 0; ks < SEG_KC / 16; ++ks)
#pragma unroll
                        for (int tile = 0; tile < TILES; ++tile) {
                            const uint64_t ad = ad0 + (uint64_t)((tile * 128 + dx * 16 + dy * C::ROW_B + 2 * ks * C::PLANE_B) >> 4);
                            const uint64_t bd = bd0 + (uint64_t)(((tap * (SEG_KC / 8) + 2 * ks) * N * 16) >> 4);
                            umma_f16(d0 + (uint32_t)(tile * N), ad, bd, IDESC, (tap == 0 && ks == 0) ? 0u : 1u);
                        }
                }
                umma_commit(&empty[s]);
                umma_commit(&tfull[t]);
            }
            __syncwarp();
        }
    } else {
        const int q = warp & 3, half_sel = warp >> 2;
        const int r = 32 * q + lane;
        constexpr int SL = N / 8;
        int j = 0;
        for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++j) {
            const int t = j & 1;
            const int f = unit / per_field, t2 = unit - f * per_field;
            const int ty = t2 / tiles_x, tx = t2 - ty * tiles_x;
            const int y = 16 * ty + (r >> 3), x0 = 8 * TILES * tx;
            __half* fout = out + (size_t)f * N * H * W;
            __half* fpool = out_pool + (size_t)f * N * (H >> 1) * (W >> 1);
            mbar_wait(&tfull[t], (uint32_t)((j >> 1) & 1));
            tc_fence_after();
            const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(t * TILES * N);
#pragma unroll 1
            for (int p = half_sel; p < TILES * SL; p += 2) {
                const int tile = p / SL, sl = p - tile * SL;
                const int x = x0 + 8 * tile + (r & 7);
                uint32_t v[8];
                TMEM_LD8(lane_addr + (uint32_t)(tile * N + sl * 8), v);
                TMEM_WAIT8(v);
                __align__(16) __half o[8];
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    o[k] = __float2half_rn(fmaxf(__fadd_rn(__uint_as_float(v[k]), __ldg(bias + sl * 8 + k)), 0.f));
                if (POOL != 1 && y < H && x < W)
                    *reinterpret_cast<uint4*>(fout + (((size_t)sl * H + y) * W + x) * 8) = *reinterpret_cast<const uint4*>(o);
                if (POOL != 0) {
                    uint4 u = *reinterpret_cast<const uint4*>(o), p1;
                    p1.x = __shfl_xor_sync(0xffffffffu, u.x, 1); p1.y = __shfl_xor_sync(0xffffffffu, u.y, 1);
                    p1.z = __shfl_xor_sync(0xffffffffu, u.z, 1); p1.w = __shfl_xor_sync(0xffffffffu, u.w, 1);
                    u = hmax8(u, p1);
                    p1.x = __shfl_xor_sync(0xffffffffu, u.x, 8); p1.y = __shfl_xor_sync(0xffffffffu, u.y, 8);
                    p1.z = __shfl_xor_sync(0xffffffffu, u.z, 8); p1.w = __shfl_xor_sync(0xffffffffu, u.w, 8);
                    u = hmax8(u, p1);
                    if (((r & 1) | ((r >> 3) & 1)) == 0 && y < H && x < W)
                        *reinterpret_cast<uint4*>(fpool + (((size_t)sl * (H >> 1) + (y >> 1)) * (W >> 1) + (x >> 1)) * 8) = u;
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[t]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, T::TMEM_COLS);
}

// ---------------------------------------------------------------------------------------
// The 1x1 heads (`prob`, `dist`) in the TMA-fed form: one box per unit brings ALL `features` channels of a 16 x 16
// pixel tile (no halo for one tap), the unit is Cin / 16 k-steps x 2 tiles of N = 48 MMAs, the epilogue writes
// dist = max(1e-3, .) and prob = sigmoid(.) in fp32.  The layer is bandwidth bound (268 MB in, 138 MB out).
// ---------------------------------------------------------------------------------------
template <int CIN>
struct SegHeadsCfg {
    static constexpr int N = 48, TILES = 2, PLANES = CIN / 8;
    static constexpr int ROW_B = 16 * 16, PLANE_B = 16 * ROW_B;        // 16 x 16 pixels, 16 bytes each
    static constexpr int A_B = PLANES * PLANE_B;
    static constexpr int W_B = PLANES * N * 16;
    static constexpr int STAGES = (215 * 1024 - W_B) / A_B >= 3 ? 3 : 2;
    static constexpr int SMEM_B = STAGES * A_B + W_B;
    static constexpr int TMEM_COLS = 256;                               // two sets of 2 x 48 columns
    static constexpr int SET_COLS = 128;
    static constexpr int THREADS = 320;
    static_assert(SMEM_B <= 225 * 1024 && A_B % 1024 == 0, "does not fit");
};

template <int CIN>
__global__ void __launch_bounds__(320, 1) seg_heads_tma_kernel(const __grid_constant__ CUtensorMap tm, const uint4* __restrict__ w,
                                                               const float* __restrict__ bias, float* __restrict__ prob,
                                                               float* __restrict__ dist, int H, int W, int F) {
    using T = SegHeadsCfg<CIN>;
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ __align__(8) uint64_t full[T::STAGES], empty[T::STAGES], tfull[2], tempty[2];
    __shared__ uint32_t tmem_base_s;
    unsigned char* sw = smem + T::STAGES * T::A_B;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tiles_x = (W + 15) / 16, tiles_y = (H + 15) / 16;
    const int per_field = tiles_x * tiles_y;               // unit = (field, tile), as seg_conv_tma_kernel
    const int n_units = per_field * F;
    if ((int)blockIdx.x >= n_units) return;

    if (warp == 0) tmem_alloc(&tmem_base_s, T::TMEM_COLS);
    if (tid == 32) {
        for (int s = 0; s < T::STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(&tfull[0], 1); mbar_init(&tfull[1], 1);
        mbar_init(&tempty[0], 8); mbar_init(&tempty[1], 8);
        fence_barrier_init();
    }
    for (int i = tid; i < T::W_B / 16; i += T::THREADS) reinterpret_cast<uint4*>(sw)[i] = __ldg(w + i);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    constexpr uint32_t IDESC = make_idesc(128, T::N);

    if (warp == 8) {
        if (lane == 0) {
            int j = 0;
            for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++j) {
                const int s = j % T::STAGES;
                mbar_wait(&empty[s], (uint32_t)(((j / T::STAGES) & 1) ^ 1));
                const int f = unit / per_field, t2 = unit - f * per_field;
                const int ty = t2 / tiles_x, tx = t2 - ty * tiles_x;
                mbar_expect_tx(&full[s], T::A_B);
                tma_load_4d(smem_u32(smem + s * T::A_B), &tm, 0, 16 * tx, 16 * ty, T::PLANES * f, &full[s]);
            }
        }
    } else if (warp == 9) {
        int j = 0;
        for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++j) {
            const int s = j % T::STAGES, t = j & 1;
            mbar_wait(&full[s], (uint32_t)((j / T::STAGES) & 1));
            mbar_wait(&tempty[t], (uint32_t)(((j >> 1) & 1) ^ 1));
            tc_fence_after();
            if (elect_one()) {
                const uint64_t ad0 = make_smem_desc(smem_u32(smem + s * T::A_B), T::PLANE_B, T::ROW_B);
                const uint64_t bd0 = make_smem_desc(smem_u32(sw), T::N * 16, 128);
                const uint32_t d0 = tmem_base + (uint32_t)(t * T::SET_COLS);
#pragma unroll
                for (int ks = 0; ks < CIN / 16; ++ks)
#pragma unroll
                    for (int tile = 0; tile < T::TILES; ++tile) {
                        const uint64_t ad = ad0 + (uint64_t)((tile * 128 + 2 * ks * T::PLANE_B) >> 4);
                        const uint64_t bd = bd0 + (uint64_t)((2 * ks * T::N * 16) >> 4);
                        umma_f16(d0 + (uint32_t)(tile * T::N), ad, bd, IDESC, ks == 0 ? 0u : 1u);
                    }
                umma_commit(&empty[s]);
                umma_commit(&tfull[t]);
            }
            __syncwarp();
        }
    } else {
        const int q = warp & 3, half_sel = warp >> 2;
        const int r = 32 * q + lane;
        constexpr int SL = SEG_RAYS / 8 + 1;
        int j = 0;
        for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++j) {
            const int t = j & 1;
            const int f = unit / per_field, t2 = unit - f * per_field;
            const int ty = t2 / tiles_x, tx = t2 - ty * tiles_x;
            const int y = 16 * ty + (r >> 3), x0 = 16 * tx;
            mbar_wait(&tfull[t], (uint32_t)((j >> 1) & 1));
            tc_fence_after();
            const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(t * T::SET_COLS);
#pragma unroll 1
            for (int p = half_sel; p < T::TILES * SL; p += 2) {
                const int tile = p / SL, sl = p - tile * SL;
                const int x = x0 + 8 * tile + (r & 7);
                uint32_t v[8];
                TMEM_LD8(lane_addr + (uint32_t)(tile * T::N + sl * 8), v);
                TMEM_WAIT8(v);
                if (y < H && x < W) {
                    const size_t px = ((size_t)f * H + y) * W + x;
                    if (sl < SEG_RAYS / 8) {
                        float o[8];
#pragma unroll
                        for (int k = 0; k < 8; ++k)
                            o[k] = fmaxf(1e-3f, __fadd_rn(__uint_as_float(v[k]), __ldg(bias + sl * 8 + k)));
                        float4* dd = reinterpret_cast<float4*>(dist + px * SEG_RAYS + sl * 8);
                        dd[0] = make_float4(o[0], o[1], o[2], o[3]);
                        dd[1] = make_float4(o[4], o[5], o[6], o[7]);
                    } else {
                        const float z = __fadd_rn(__uint_as_float(v[0]), __ldg(bias + SEG_RAYS));
                        prob[px] = 1.f / (1.f + expf(-z));
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[t]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, T::TMEM_COLS);
}

// ---------------------------------------------------------------------------------------
// The general layer in the same warp-specialised form: the producer is SOFTWARE (eight warps run the staging of
// seg_conv_kernel -- pooled, up-sampled + concatenated or direct inputs, any number of 32-channel chunks, each with
// its weight block -- into a 2-3 stage ring and arrive on the stage's `full` barrier), one warp issues the MMAs of a
// (unit, chunk) step as soon as its stage is full, eight warps run the epilogue of unit u under the MMAs of unit u + 1.
// Staging, tensor math and epilogue of DIFFERENT units overlap inside one CTA instead of across co-resident CTAs.
// ---------------------------------------------------------------------------------------
template <int N, int TILES>
struct SegWsCfg {
    using B = SegCfg<N, TILES>;
    static constexpr int STAGE_B = (B::A_B + B::W_B + 1023) / 1024 * 1024;
    static constexpr int STAGES = (220 * 1024) / STAGE_B >= 3 ? 3 : 2;
    static constexpr int SMEM_B = STAGES * STAGE_B;
    static constexpr int TMEM_COLS = pow2_cols(2 * TILES * N);
    static constexpr int PROD = 256;                       // producer threads (warps 8..15)
    static constexpr int THREADS = 256 + PROD + 32;        // epilogue warps 0..7, producers, MMA warp 16
    static_assert(TMEM_COLS <= 512 && SMEM_B <= 225 * 1024, "does not fit");
};

template <int N, int TILES>
__global__ void __launch_bounds__(SegWsCfg<N, TILES>::THREADS, 1) seg_conv_ws_kernel(const SegConvArgs a) {
    using C = SegCfg<N, TILES>;
    using T = SegWsCfg<N, TILES>;
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ __align__(8) uint64_t full[T::STAGES], empty[T::STAGES], tfull[2], tempty[2];
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tiles_x = (a.W + 8 * TILES - 1) / (8 * TILES), tiles_y = (a.H + 15) / 16;
    const int per_field = tiles_x * tiles_y, per_group = per_field * a.F;    // unit = (group, field, tile)
    const int n_units = per_group * a.groups;
    if ((int)blockIdx.x >= n_units) return;

    if (warp == 0) tmem_alloc(&tmem_base_s, T::TMEM_COLS);
    if (tid == 32) {
        for (int s = 0; s < T::STAGES; ++s) { mbar_init(&full[s], T::PROD); mbar_init(&empty[s], 1); }
        mbar_init(&tfull[0], 1); mbar_init(&tfull[1], 1);
        mbar_init(&tempty[0], 8); mbar_init(&tempty[1], 8);
        fence_barrier_init();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    constexpr uint32_t IDESC = make_idesc(128, N);
    const int w_units = a.ntaps * (C::WT_B / 16);

    if (warp >= 8 && warp < 16) {
        // ---- producers ----
        const int pt = tid - 256;
        int step = 0;
        for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
            const int g = unit / per_group, fu = unit - g * per_group;
            const int f = fu / per_field, t2 = fu - f * per_field;
            const int ty = t2 / tiles_x, tx = t2 - ty * tiles_x;
            const int y0 = 16 * ty, x0 = 8 * TILES * tx;
            const uint4 *s0, *s1;
            seg_src(a, f, s0, s1);
            for (int kc = 0; kc < a.chunks; ++kc, ++step) {
                const int s = step % T::STAGES;
                mbar_wait(&empty[s], (uint32_t)(((step / T::STAGES) & 1) ^ 1));
                unsigned char* sa = smem + s * T::STAGE_B;
                unsigned char* sw = sa + C::A_B;
                const uint4* wsrc = a.w + (size_t)(g * a.chunks + kc) * w_units;
                for (int i = pt; i < w_units; i += T::PROD) reinterpret_cast<uint4*>(sw)[i] = __ldg(wsrc + i);
                constexpr int SB = ((C::NU + T::PROD - 1) / T::PROD + 1) / 2;
#pragma unroll 1
                for (int i0 = pt; i0 < C::NU; i0 += SB * T::PROD) {
                    uint4 v[SB];
                    uint32_t d[SB];
#pragma unroll
                    for (int j = 0; j < SB; ++j) {
                        const int idx = i0 + j * T::PROD;
                        d[j] = 0xFFFFFFFFu;
                        v[j] = make_uint4(0, 0, 0, 0);
                        if (idx < C::NU) {
                            const int c = idx / (18 * C::COLS);
                            const int rem = idx - c * (18 * C::COLS);
                            const int ry = rem / C::COLS, rc = rem - ry * C::COLS;
                            const int y = y0 + ry - 1, x = x0 + rc - 1;
                            d[j] = (uint32_t)idx * 16u;
                            if (y >= 0 && y < a.H && x >= 0 && x < a.W) v[j] = seg_load(a, s0, s1, kc * (SEG_KC / 8) + c, y, x);
                        }
                    }
#pragma unroll
                    for (int j = 0; j < SB; ++j)
                        if (d[j] != 0xFFFFFFFFu) *reinterpret_cast<uint4*>(sa + d[j]) = v[j];
                }
                fence_async_smem();
                mbar_arrive(&full[s]);
            }
        }
    } else if (warp == 16) {
        // ---- MMA issue ----
        int step = 0, j = 0;
        for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++j) {
            const int t = j & 1;
            for (int kc = 0; kc < a.chunks; ++kc, ++step) {
                const int s = step % T::STAGES;
                mbar_wait(&full[s], (uint32_t)((step / T::STAGES) & 1));
                if (kc == 0) mbar_wait(&tempty[t], (uint32_t)(((j >> 1) & 1) ^ 1));
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t sa = smem_u32(smem + s * T::STAGE_B);
                    const uint64_t ad0 = make_smem_desc(sa, C::PLANE_B, C::ROW_B);
                    const uint64_t bd0 = make_smem_desc(sa + C::A_B, N * 16, 128);
                    const uint32_t d0 = tmem_base + (uint32_t)(t * TILES * N);
                    for (int tap = 0; tap < a.ntaps; ++tap) {
                        const int dy = a.ntaps == 1 ? 1 : tap / 3, dx = a.ntaps == 1 ? 1 : tap % 3;
#pragma unroll
                        for (int ks = 0; ks < SEG_KC / 16; ++ks)
#pragma unroll
                            for (int tile = 0; tile < TILES; ++tile) {
                                const uint64_t ad = ad0 + (uint64_t)((tile * 128 + dx * 16 + dy * C::ROW_B + 2 * ks * C::PLANE_B) >> 4);
                                const uint64_t bd = bd0 + (uint64_t)(((tap * (SEG_KC / 8) + 2 * ks) * N * 16) >> 4);
                                umma_f16(d0 + (uint32_t)(tile * N), ad, bd, IDESC, (kc == 0 && tap == 0 && ks == 0) ? 0u : 1u);
                            }
                    }
                    umma_commit(&empty[s]);
                    if (kc == a.chunks - 1) umma_commit(&tfull[t]);
                }
                __syncwarp();
            }
        }
    } else if (warp < 8) {
        // ---- epilogue ----
        const int q = warp & 3, half_sel = warp >> 2;
        const int r = 32 * q + lane;
        constexpr int SL = N / 8;
        int j = 0;
        for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++j) {
            const int t = j & 1;
            const int g = unit / per_group, fu = unit - g * per_group;
            const int f = fu / per_field, t2 = fu - f * per_field;
            const int ty = t2 / tiles_x, tx = t2 - ty * tiles_x;
            const int y = 16 * ty + (r >> 3), x0 = 8 * TILES * tx;
            __half* fout = a.out + (size_t)f * a.groups * N * a.H * a.W;
            mbar_wait(&tfull[t], (uint32_t)((j >> 1) & 1));
            tc_fence_after();
            const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(t * TILES * N);
#pragma unroll 1
            for (int p = half_sel; p < TILES * SL; p += 2) {
                const int tile = p / SL, sl = p - tile * SL;
                const int x = x0 + 8 * tile + (r & 7);
                uint32_t v[8];
                TMEM_LD8(lane_addr + (uint32_t)(tile * N + sl * 8), v);
                TMEM_WAIT8(v);
                const int c0 = g * N + sl * 8;
                __align__(16) __half o[8];
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    o[k] = __float2half_rn(fmaxf(__fadd_rn(__uint_as_float(v[k]), __ldg(a.bias + c0 + k)), 0.f));
                if (y < a.H && x < a.W)
                    *reinterpret_cast<uint4*>(fout + (((size_t)(c0 >> 3) * a.H + y) * a.W + x) * 8) = *reinterpret_cast<const uint4*>(o);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[t]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, T::TMEM_COLS);
}

// ---------------------------------------------------------------------------------------
// Instances from (prob, dist): candidates, polygons, bins, greedy NMS, rendering
// ---------------------------------------------------------------------------------------
// Candidates in descending probability, ties: the larger flat index first (np.argsort(prob, stable)[::-1]):
// flags -> exclusive scan -> compaction in DESCENDING index order -> stable radix sort of the inverted probability
// bits (32-bit keys, the index as the value: half the passes of a 64-bit key sort).
// F fields [F][Hgp][Wgp] (maps padded to Hgp x Wgp, candidates only in the logical hg x wg part): the flat index runs
// over all fields and the key carries the field above bit 32, so the sort over 32 + ceil(log2 F) bits orders by
// field, then exactly as a one-field call; one field keeps 32-bit keys.
__global__ void seg_cand_flags_kernel(const float* __restrict__ prob, int F, int Hgp, int Wgp, int hg, int wg, float thr,
                                      int border, int* __restrict__ flags) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= F * Hgp * Wgp) return;
    const int rem = idx % (Hgp * Wgp);
    const int i = rem / Wgp, j = rem - i * Wgp;
    flags[idx] = (prob[idx] > thr && i >= border && i < hg - border && j >= border && j < wg - border) ? 1 : 0;
}

template <typename K>
__global__ void seg_cand_scatter_kernel(const float* __restrict__ prob, const int* __restrict__ flags, const int* __restrict__ excl,
                                        int cap, int field_px, K* __restrict__ keys, unsigned* __restrict__ vals,
                                        int* __restrict__ count) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= cap) return;
    const int total = excl[cap - 1] + flags[cap - 1];
    if (idx == 0) *count = total;
    if (flags[idx]) {
        const int pos = total - 1 - excl[idx];
        K key = (K)~__float_as_uint(prob[idx]);
        if constexpr (sizeof(K) == 8) key |= (K)(idx / field_px) << 32;
        keys[pos] = key;
        vals[pos] = (unsigned)idx;
    }
}

// dist_to_coord: coord = (dist * [sin, cos]).astype(float32); coord += points  (float32 += int: added in fp64, stored fp32)
// rank r (sorted order over all fields) -> its field's polygon; rfield[r] = field.  Bins are per field: field f owns
// bins [f nby nbx, (f + 1) nby nbx), so no reach ever crosses into another field.
__global__ void seg_polygons_kernel(const unsigned* __restrict__ sorted_idx, const int* __restrict__ count, int cap,
                                    const float* __restrict__ prob, const float* __restrict__ dist, int Hgp, int Wgp, int grid,
                                    const double* __restrict__ rsin, const double* __restrict__ rcos, int H, int W,
                                    float* __restrict__ vy, float* __restrict__ vx, int* __restrict__ pyx,
                                    float* __restrict__ pprob, float* __restrict__ rmax, double* __restrict__ area,
                                    int* __restrict__ bin_of, int* __restrict__ bin_count, unsigned* __restrict__ rmax_all,
                                    int* __restrict__ rfield) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = min(*count, cap);
    if (r >= n) return;
    const unsigned idx = sorted_idx[r];
    const int f = (int)(idx / (unsigned)(Hgp * Wgp));
    const unsigned rem = idx - (unsigned)f * (unsigned)(Hgp * Wgp);
    const int i = (int)(rem / (unsigned)Wgp), j = (int)(rem - (unsigned)i * Wgp);
    const int py = i * grid, px = j * grid;
    const float* d = dist + (size_t)idx * SEG_RAYS;
    float ys[SEG_RAYS], xs[SEG_RAYS];
    float rm = 0.f;
#pragma unroll
    for (int k = 0; k < SEG_RAYS; ++k) {
        const float dk = d[k];
        rm = fmaxf(rm, dk);
        const float ty = (float)__dmul_rn((double)dk, rsin[k]), tx = (float)__dmul_rn((double)dk, rcos[k]);
        ys[k] = (float)__dadd_rn((double)ty, (double)py);
        xs[k] = (float)__dadd_rn((double)tx, (double)px);
        vy[(size_t)r * SEG_RAYS + k] = ys[k];
        vx[(size_t)r * SEG_RAYS + k] = xs[k];
    }
    double s = 0.0;                                      // shoelace, sequential, no contraction
#pragma unroll
    for (int k = 0; k < SEG_RAYS; ++k) {
        const int k1 = (k + 1) & (SEG_RAYS - 1);
        s = __dadd_rn(s, __dsub_rn(__dmul_rn((double)xs[k], (double)ys[k1]), __dmul_rn((double)xs[k1], (double)ys[k])));
    }
    area[r] = __dmul_rn(0.5, fabs(s));
    pyx[2 * r] = py; pyx[2 * r + 1] = px;
    pprob[r] = prob[idx];
    rmax[r] = rm;
    atomicMax(rmax_all, __float_as_uint(rm));            // rm >= 1e-3 > 0: the bit pattern orders like the value
    const int nbx = (W + SEG_BIN - 1) / SEG_BIN, nby = (H + SEG_BIN - 1) / SEG_BIN;
    const int bin = (f * nby + min(py / SEG_BIN, nby - 1)) * nbx + min(px / SEG_BIN, nbx - 1);
    rfield[r] = f;
    bin_of[r] = bin;
    atomicAdd(bin_count + bin, 1);
}

// counting sort of the candidates by bin: exclusive scan of the bin populations (one CTA), then seg_binorder_kernel
// hands out positions with one atomic per candidate (the order INSIDE a bin is irrelevant to the suppression's result)
__global__ void __launch_bounds__(1024) seg_bins_kernel(const int* __restrict__ bin_count, int nbins, int* __restrict__ bin_start,
                                                        int* __restrict__ bin_cursor) {
    typedef cub::BlockScan<int, 1024> Scan;
    __shared__ typename Scan::TempStorage tmp;
    __shared__ int carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int b0 = 0; b0 < nbins; b0 += 1024) {
        const int b = b0 + threadIdx.x;
        const int c = b < nbins ? bin_count[b] : 0;
        int ex, total;
        Scan(tmp).ExclusiveSum(c, ex, total);
        const int carry = carry_s;
        if (b < nbins) { bin_start[b] = carry + ex; bin_cursor[b] = carry + ex; }
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + total;
        __syncthreads();
    }
    if (threadIdx.x == 0) bin_start[nbins] = carry_s;
}

__device__ __forceinline__ double cross_rn(double ax, double ay, double bx, double by, double px, double py) {
    return __dsub_rn(__dmul_rn(__dsub_rn(bx, ax), __dsub_rn(py, ay)), __dmul_rn(__dsub_rn(by, ay), __dsub_rn(px, ax)));
}

// Two counter-clockwise triangles: do their bounding boxes miss, or does an edge of one have all three vertices of
// the other strictly outside?  (the same statements, in the same order, as oracle/stardist_post.c::tri_tri_area)
__device__ __forceinline__ bool tri_separated(const double* sx, const double* sy, const double* cx, const double* cy) {
    double mn1 = fmin(fmin(sx[0], sx[1]), sx[2]), mx1 = fmax(fmax(sx[0], sx[1]), sx[2]);
    double mn2 = fmin(fmin(cx[0], cx[1]), cx[2]), mx2 = fmax(fmax(cx[0], cx[1]), cx[2]);
    if (mx1 < mn2 || mx2 < mn1) return true;
    mn1 = fmin(fmin(sy[0], sy[1]), sy[2]); mx1 = fmax(fmax(sy[0], sy[1]), sy[2]);
    mn2 = fmin(fmin(cy[0], cy[1]), cy[2]); mx2 = fmax(fmax(cy[0], cy[1]), cy[2]);
    if (mx1 < mn2 || mx2 < mn1) return true;
#pragma unroll
    for (int e = 0; e < 3; ++e) {
        const int e1 = e == 2 ? 0 : e + 1;
        if (cross_rn(cx[e], cy[e], cx[e1], cy[e1], sx[0], sy[0]) < 0.0 && cross_rn(cx[e], cy[e], cx[e1], cy[e1], sx[1], sy[1]) < 0.0 &&
            cross_rn(cx[e], cy[e], cx[e1], cy[e1], sx[2], sy[2]) < 0.0) return true;
        if (cross_rn(sx[e], sy[e], sx[e1], sy[e1], cx[0], cy[0]) < 0.0 && cross_rn(sx[e], sy[e], sx[e1], sy[e1], cx[1], cy[1]) < 0.0 &&
            cross_rn(sx[e], sy[e], sx[e1], sy[e1], cx[2], cy[2]) < 0.0) return true;
    }
    return false;
}

// area of the intersection of two triangles that are not separated: Sutherland-Hodgman, then the shoelace sum
__device__ double tri_clip_area(const double* sx, const double* sy, const double* cx, const double* cy) {
    double px[8], py[8], qx[8], qy[8];
    int n = 3;
    for (int k = 0; k < 3; ++k) { px[k] = sx[k]; py[k] = sy[k]; }
    for (int e = 0; e < 3; ++e) {
        const double ax = cx[e], ay = cy[e], bx = cx[(e + 1) % 3], by = cy[(e + 1) % 3];
        int m = 0;
        for (int k = 0; k < n; ++k) {
            const int k1 = k + 1 == n ? 0 : k + 1;
            const double dc = cross_rn(ax, ay, bx, by, px[k], py[k]);
            const double dn = cross_rn(ax, ay, bx, by, px[k1], py[k1]);
            if (dc >= 0.0) { qx[m] = px[k]; qy[m] = py[k]; ++m; }
            if ((dc >= 0.0) != (dn >= 0.0)) {
                const double t = __ddiv_rn(dc, __dsub_rn(dc, dn));
                qx[m] = __dadd_rn(px[k], __dmul_rn(t, __dsub_rn(px[k1], px[k])));
                qy[m] = __dadd_rn(py[k], __dmul_rn(t, __dsub_rn(py[k1], py[k])));
                ++m;
            }
        }
        n = m;
        if (n == 0) return 0.0;
        for (int k = 0; k < n; ++k) { px[k] = qx[k]; py[k] = qy[k]; }
    }
    double s = 0.0;
    for (int k = 0; k < n; ++k) {
        const int k1 = k + 1 == n ? 0 : k + 1;
        s = __dadd_rn(s, __dsub_rn(__dmul_rn(px[k], py[k1]), __dmul_rn(px[k1], py[k])));
    }
    return __dmul_rn(0.5, fabs(s));
}

// The same clipping in float32 on coordinates relative to the winner's centre: only used for the LOWER BOUND of the
// overlap (relative error ~1e-5 against a 1 % safety margin), never for a value that is compared exactly.
__device__ float tri_clip_area_f32(const float* sx, const float* sy, const float* cx, const float* cy) {
    float bx0[8], by0[8], bx1[8], by1[8];
    int n = 3;
#pragma unroll
    for (int k = 0; k < 3; ++k) { bx0[k] = sx[k]; by0[k] = sy[k]; }
#pragma unroll
    for (int e = 0; e < 3; ++e) {
        const float* px = (e & 1) ? bx1 : bx0;
        const float* py = (e & 1) ? by1 : by0;
        float* qx = (e & 1) ? bx0 : bx1;
        float* qy = (e & 1) ? by0 : by1;
        const float ax = cx[e], ay = cy[e], ex = cx[e == 2 ? 0 : e + 1] - ax, ey = cy[e == 2 ? 0 : e + 1] - ay;
        int m = 0;
        float dc = ex * (py[0] - ay) - ey * (px[0] - ax);
        for (int k = 0; k < n; ++k) {
            const int k1 = k + 1 == n ? 0 : k + 1;
            const float dn = ex * (py[k1] - ay) - ey * (px[k1] - ax);
            if (dc >= 0.f) { qx[m] = px[k]; qy[m] = py[k]; ++m; }
            if ((dc >= 0.f) != (dn >= 0.f)) {
                const float t = __fdividef(dc, dc - dn);
                qx[m] = fmaf(t, px[k1] - px[k], px[k]);
                qy[m] = fmaf(t, py[k1] - py[k], py[k]);
                ++m;
            }
            dc = dn;
        }
        n = m;
        if (n == 0) return 0.f;
    }
    // three clips: the result is in buffer 1
    float s2 = 0.f;
    for (int k = 0; k < n; ++k) {
        const int k1 = k + 1 == n ? 0 : k + 1;
        s2 += bx1[k] * by1[k1] - bx1[k1] * by1[k];
    }
    return 0.5f * fabsf(s2);
}

#ifndef SEG_NMS_CTAS
#define SEG_NMS_CTAS 4     // CTAs per SM of the suppression kernel (64 registers: latency-bound fp64 chains want warps)
#endif
struct NmsArgs {
    const float *vy, *vx;        // [rank][32]
    const int* pyx;              // [rank][2]
    const double* area;          // [rank]
    const int* b_rank;           // candidates in BIN order (position k): rank,
    const float4* b_yxr;         //   (y, x, rmax, field as int bits)
    const int* bin_start;
    const int* count;
    const unsigned* rmax_all;
    int* state;          // by bin position: 0 undecided, 2 suppressed, 4 + round: kept (winner of that round)
    int* cnt;            // [3] undecided counters of rounds r, r + 1, r + 2 (mod 3)
    int nbx, nby, cap;           // bins of ONE field; field f's bins start at f nby nbx
    double thr;
};

// polygons w (the winner) and i: intersection area over the smaller area.  One warp: lane a clips fan triangle a
// of w against the 32 fan triangles of i (starting at its own index); the lane sums are added in lane order
// (the oracle's order).
__device__ double seg_overlap_warp(const NmsArgs& a, int w, int i, float (*sp)[2][SEG_RAYS], int lane) {
    __syncwarp();
    sp[0][0][lane] = a.vy[(size_t)w * SEG_RAYS + lane]; sp[0][1][lane] = a.vx[(size_t)w * SEG_RAYS + lane];
    sp[1][0][lane] = a.vy[(size_t)i * SEG_RAYS + lane]; sp[1][1][lane] = a.vx[(size_t)i * SEG_RAYS + lane];
    __syncwarp();
    const int l1 = (lane + 1) & (SEG_RAYS - 1);
    const double cwx = (double)a.pyx[2 * w + 1], cwy = (double)a.pyx[2 * w];
    const double cix = (double)a.pyx[2 * i + 1], ciy = (double)a.pyx[2 * i];
    // step 0, a rigorous shortcut: every term of the fan sum is >= 0, so the sum over ANY subset of pairs is a lower
    // bound of the intersection.  Candidates of the same nucleus (nearly all tests) overlap far above the threshold:
    // the same-index pairs and their neighbours at index distance 1 and 2 prove "suppressed" after three or five clipped
    // batches (measured on ellipse fields: 80 % after three, all after five) instead of 1024 separation tests + the full list.  The exact sum is only needed near the threshold.
    {
        const double denom = __dadd_rn(fmin(a.area[w], a.area[i]), 1e-10);
        const float need = (float)(a.thr * denom * (1.0 + 1e-2));     // float32 clipping: 1 % covers its rounding many times over
        const float ox = (float)a.pyx[2 * w + 1], oy = (float)a.pyx[2 * w];
        const float sx[3] = {0.f, sp[0][1][lane] - ox, sp[0][1][l1] - ox};
        const float sy[3] = {0.f, sp[0][0][lane] - oy, sp[0][0][l1] - oy};
        const float fix = (float)a.pyx[2 * i + 1] - ox, fiy = (float)a.pyx[2 * i] - oy;
        float lb = 0.f;
#pragma unroll 1
        for (int q = 0; q < 5; ++q) {                    // index offsets 0, +1, -1, +2, -2
            const int b = (lane + (q == 0 ? 0 : q == 1 ? 1 : q == 2 ? SEG_RAYS - 1 : q == 3 ? 2 : SEG_RAYS - 2)) & (SEG_RAYS - 1);
            const int b1 = (b + 1) & (SEG_RAYS - 1);
            const float cx[3] = {fix, sp[1][1][b] - ox, sp[1][1][b1] - ox};
            const float cy[3] = {fiy, sp[1][0][b] - oy, sp[1][0][b1] - oy};
            lb += tri_clip_area_f32(sx, sy, cx, cy);
            if (q == 0 || q == 1 || q == 3) continue;    // test after both neighbours of each distance
            float tot = lb;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
            if (tot > need) return (double)tot / denom;  // > thr: the full sum can only be larger
        }
    }
    // bounding boxes (the vertices' extent, as the oracle): only reached by pairs the lower bound did not decide
    float y0 = sp[0][0][lane], y1 = y0, x0 = sp[0][1][lane], x1 = x0;
    float u0 = sp[1][0][lane], u1 = u0, v0 = sp[1][1][lane], v1 = v0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        y0 = fminf(y0, __shfl_xor_sync(0xffffffffu, y0, o)); y1 = fmaxf(y1, __shfl_xor_sync(0xffffffffu, y1, o));
        x0 = fminf(x0, __shfl_xor_sync(0xffffffffu, x0, o)); x1 = fmaxf(x1, __shfl_xor_sync(0xffffffffu, x1, o));
        u0 = fminf(u0, __shfl_xor_sync(0xffffffffu, u0, o)); u1 = fmaxf(u1, __shfl_xor_sync(0xffffffffu, u1, o));
        v0 = fminf(v0, __shfl_xor_sync(0xffffffffu, v0, o)); v1 = fmaxf(v1, __shfl_xor_sync(0xffffffffu, v1, o));
    }
    if (y1 < u0 || u1 < y0 || x1 < v0 || v1 < x0) return 0.0;
    // step 1: lane = fan triangle of w; bit st of `mask` = its pair with triangle (lane + st) of i needs clipping
    unsigned mask = 0;
    {
        const double sx[3] = {cwx, (double)sp[0][1][lane], (double)sp[0][1][l1]};
        const double sy[3] = {cwy, (double)sp[0][0][lane], (double)sp[0][0][l1]};
        for (int st = 0; st < SEG_RAYS; ++st) {
            const int b = (lane + st) & (SEG_RAYS - 1), b1 = (b + 1) & (SEG_RAYS - 1);
            const double cx[3] = {cix, (double)sp[1][1][b], (double)sp[1][1][b1]};
            const double cy[3] = {ciy, (double)sp[1][0][b], (double)sp[1][0][b1]};
            if (!tri_separated(sx, sy, cx, cy)) mask |= 1u << st;
        }
    }
    // step 2: the pairs of all lanes form one list (lane-major, ascending st), clipped 32 at a time with every lane
    // busy; a lane then adds ITS pairs' areas in list order = the oracle's order (separated pairs contribute +0.0)
    const int cnt = __popc(mask);
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    const int off = incl - cnt, total = __shfl_sync(0xffffffffu, incl, 31);
    double part = 0.0;
    for (int g0 = 0; g0 < total; g0 += 32) {
        const int g = min(g0 + lane, total - 1);
        int own = 0;                                     // largest lane whose first pair is at or before g
#pragma unroll
        for (int step = 16; step > 0; step >>= 1) {
            const int oc = __shfl_sync(0xffffffffu, off, own + step);
            if (oc <= g) own += step;
        }
        const int oo = __shfl_sync(0xffffffffu, off, own);
        const unsigned om = __shfl_sync(0xffffffffu, mask, own);
        const int st = (int)__fns(om, 0, g - oo + 1);   // the (g - oo + 1)-th set bit
        double ar = 0.0;
        if (g0 + lane < total) {
            const int a1 = (own + 1) & (SEG_RAYS - 1);
            const int b = (own + st) & (SEG_RAYS - 1), b1 = (b + 1) & (SEG_RAYS - 1);
            const double sx[3] = {cwx, (double)sp[0][1][own], (double)sp[0][1][a1]};
            const double sy[3] = {cwy, (double)sp[0][0][own], (double)sp[0][0][a1]};
            const double cx[3] = {cix, (double)sp[1][1][b], (double)sp[1][1][b1]};
            const double cy[3] = {ciy, (double)sp[1][0][b], (double)sp[1][0][b1]};
            ar = tri_clip_area(sx, sy, cx, cy);
        }
        const int lo_g = max(off, g0), hi_g = min(off + cnt, g0 + 32);
        const int mine = max(0, hi_g - lo_g);
        const int most = __reduce_max_sync(0xffffffffu, mine);
        for (int t = 0; t < most; ++t) {
            const double v = __shfl_sync(0xffffffffu, ar, (lo_g + t - g0) & 31);
            if (t < mine) part = __dadd_rn(part, v);
        }
    }
    double inter = 0.0;
    for (int l = 0; l < 32; ++l) inter = __dadd_rn(inter, __shfl_sync(0xffffffffu, part, l));
    return __ddiv_rn(inter, __dadd_rn(fmin(a.area[w], a.area[i]), 1e-10));
}

__device__ __forceinline__ int ld_volatile(const int* p) { return *reinterpret_cast<const volatile int*>(p); }

// A candidate's neighbours are the candidates of the bins its reach touches; a row of bins is one contiguous range
// of bin positions, read 32 at a time (coalesced: rank, state, centre and radius all live in bin order).
__global__ void __launch_bounds__(256, SEG_NMS_CTAS) seg_nms_kernel(const NmsArgs a) {
    cg::grid_group grid = cg::this_grid();
    __shared__ float s_poly[8][2][2][SEG_RAYS];
    const int n = min(*a.count, a.cap);
    const float RM = __uint_as_float(*a.rmax_all);
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gthreads = gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int gwarp = gtid >> 5, gwarps = gthreads >> 5;
    const float inv_bin = 1.f / SEG_BIN;

    for (int round = 0;; ++round) {
        const int mark = 4 + round;
        if (gtid == 0) a.cnt[(round + 1) % 3] = 0;
        for (int phase = 0; phase < 2; ++phase) {
            // phase 0: an open candidate none of whose better candidates in reach is still open wins the round
            // phase 1: the round's winners suppress their open neighbours by the exact overlap
            for (int k = gwarp; k < n; k += gwarps) {
                if (ld_volatile(a.state + k) != 0) continue;                 // warp-uniform
                const int rank = a.b_rank[k];
                const float4 me = a.b_yxr[k];
                const int* fbins = a.bin_start + __float_as_int(me.w) * a.nby * a.nbx;   // the candidate's field
                const float reach = me.z + RM + 0.01f;
                const int by0 = max(0, (int)floorf((me.x - reach) * inv_bin)), by1 = min(a.nby - 1, (int)floorf((me.x + reach) * inv_bin));
                const int bx0 = max(0, (int)floorf((me.y - reach) * inv_bin)), bx1 = min(a.nbx - 1, (int)floorf((me.y + reach) * inv_bin));
                bool done = false;                                           // phase 0: blocked, phase 1: suppressed
                // rows of bins from the candidate's own row outwards: what blocks or suppresses it is usually a
                // candidate of the same nucleus, found in the first rows
                const int byc = min(max((int)floorf(me.x * inv_bin), by0), by1);
                const int nrows = by1 - by0 + 1;
                for (int j = 0, up = 0, dn = 1; j < nrows && !done; ++j) {
                    int by;
                    if ((byc - up >= by0) && (up < dn || byc + dn > by1)) { by = byc - up; ++up; }
                    else { by = byc + dn; ++dn; }
                    const int ke = fbins[by * a.nbx + bx1 + 1];
                    for (int k0 = fbins[by * a.nbx + bx0]; k0 < ke && !done; k0 += 32) {
                        const int kk = k0 + lane;
                        bool hit = false;
                        int rj = -1;
                        if (kk < ke) {
                            rj = a.b_rank[kk];
                            if (rj < rank) {
                                const int st = ld_volatile(a.state + kk);
                                if (phase == 0 ? (st == 0 || st == mark) : (st == mark)) {
                                    const float4 o = a.b_yxr[kk];
                                    const float dy = me.x - o.x, dx = me.y - o.y, rr = me.z + o.z + 0.01f;
                                    hit = dy * dy + dx * dx < rr * rr;
                                }
                            }
                        }
                        unsigned m = __ballot_sync(0xffffffffu, hit);
                        if (phase == 0) { done = m != 0; continue; }
                        while (m && !done) {
                            const int src = __ffs(m) - 1;
                            m &= m - 1;
                            const int w = __shfl_sync(0xffffffffu, rj, src);
                            done = seg_overlap_warp(a, w, rank, s_poly[wib], lane) > a.thr;
                        }
                    }
                }
                if (lane == 0) {
                    if (phase == 0) { if (!done) *reinterpret_cast<volatile int*>(a.state + k) = mark; }
                    else if (done) *reinterpret_cast<volatile int*>(a.state + k) = 2;
                    else atomicAdd(a.cnt + round % 3, 1);
                }
            }
            grid.sync();
        }
        if (ld_volatile(a.cnt + round % 3) == 0) break;              // the same value for every thread
    }
}

// bin-order copies of what the suppression reads per neighbour
__global__ void seg_binorder_kernel(const int* __restrict__ bin_of, int* __restrict__ bin_cursor, const int* __restrict__ count,
                                    int cap, const int* __restrict__ pyx, const float* __restrict__ rmax,
                                    const int* __restrict__ rfield, int* __restrict__ b_rank, float4* __restrict__ b_yxr,
                                    int* __restrict__ pos) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= min(*count, cap)) return;
    const int k = atomicAdd(bin_cursor + bin_of[r], 1);
    b_rank[k] = r;
    b_yxr[k] = make_float4((float)pyx[2 * r], (float)pyx[2 * r + 1], rmax[r], __int_as_float(rfield[r]));
    pos[r] = k;
}

__global__ void seg_flags_kernel(const int* __restrict__ state, const int* __restrict__ pos, const int* __restrict__ count,
                                 int cap, int* __restrict__ flags) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= cap) return;
    flags[r] = (r < min(*count, cap) && state[pos[r]] >= 4) ? 1 : 0;
}

// kept polygons in rank order; ranks are grouped by field, so kstart[f] (kept polygons of the fields before f,
// [F + 1]) is excl at the first rank of field f: written by that rank for f and the empty fields before it
__global__ void seg_compact_kernel(const int* __restrict__ flags, const int* __restrict__ excl, int cap,
                                   const int* __restrict__ count, const int* __restrict__ rfield, int F,
                                   int* __restrict__ kept_rank, int* __restrict__ n_kept, int* __restrict__ kstart) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= cap) return;
    if (flags[r]) kept_rank[excl[r]] = r;
    if (r == cap - 1) *n_kept = excl[r] + flags[r];
    const int n = min(*count, cap);
    if (r < n) {
        const int fr = rfield[r], fp = r == 0 ? -1 : rfield[r - 1];
        for (int f = fp + 1; f <= fr; ++f) kstart[f] = excl[r];
        if (r == n - 1)
            for (int f = fr + 1; f <= F; ++f) kstart[f] = excl[r] + flags[r];
    } else if (r == 0) {
        for (int f = 0; f <= F; ++f) kstart[f] = 0;
    }
}

// skimage.draw.polygon's test (skimage/_shared/_geometry / _pnpoly.h point_in_polygon): crossings of the edges
// with the rays to the right and to the left of the point; vertex and edge points count as inside
__device__ __forceinline__ int seg_pnpoly(const float* vxs, const float* vys, double x, double y) {
    int l_cross = 0, r_cross = 0;
    const double eps = 1e-12;
    double x1 = __dsub_rn((double)vxs[SEG_RAYS - 1], x), y1 = __dsub_rn((double)vys[SEG_RAYS - 1], y);
    for (int i = 0; i < SEG_RAYS; ++i) {
        const double x0 = __dsub_rn((double)vxs[i], x), y0 = __dsub_rn((double)vys[i], y);
        if (-eps < x0 && x0 < eps && -eps < y0 && y0 < eps) return 3;
        if ((y0 > 0) != (y1 > 0)) {
            if (__ddiv_rn(__dsub_rn(__dmul_rn(x0, y1), __dmul_rn(x1, y0)), __dsub_rn(y1, y0)) > 0) ++r_cross;
        }
        if ((y0 < 0) != (y1 < 0)) {
            if (__ddiv_rn(__dsub_rn(__dmul_rn(x0, y1), __dmul_rn(x1, y0)), __dsub_rn(y1, y0)) < 0) ++l_cross;
        }
        x1 = x0; y1 = y0;
    }
    if ((r_cross & 1) != (l_cross & 1)) return 2;
    return r_cross & 1;
}

constexpr int SEG_RENDER_SPLIT = 16;   // warps that share one polygon's bounding box
constexpr int SEG_EMPTY = 0x7F7F7F7F;   // cudaMemset(0x7F) background of the atomicMin target

// polygons_to_label: polygons drawn in ascending probability, label = NMS output index + 1  ==  every pixel takes
// the smallest index among the polygons that cover it
__global__ void __launch_bounds__(256) seg_render_kernel(const float* __restrict__ vy, const float* __restrict__ vx,
                                                         const int* __restrict__ pyx, const int* __restrict__ kept_rank,
                                                         const int* __restrict__ n_kept, const int* __restrict__ rfield,
                                                         int H, int W, int32_t* __restrict__ labels) {
    __shared__ float s_v[8][2][SEG_RAYS];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, gwarps = (gridDim.x * blockDim.x) >> 5;
    const int nk = *n_kept;
    for (int job = gwarp; job < nk * SEG_RENDER_SPLIT; job += gwarps) {
        const int k = job / SEG_RENDER_SPLIT, part = job - k * SEG_RENDER_SPLIT;    // rows part, part + 16, ... of polygon k
        const int r = kept_rank[k];
        int32_t* flabels = labels + (size_t)rfield[r] * H * W;     // global kept index k + 1; seg_finalize_kernel rebases it
        __syncwarp();
        const float yv = vy[(size_t)r * SEG_RAYS + lane], xv = vx[(size_t)r * SEG_RAYS + lane];
        s_v[wib][0][lane] = yv; s_v[wib][1][lane] = xv;
        __syncwarp();
        float y0 = yv, y1 = yv, x0 = xv, x1 = xv;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            y0 = fminf(y0, __shfl_xor_sync(0xffffffffu, y0, o)); y1 = fmaxf(y1, __shfl_xor_sync(0xffffffffu, y1, o));
            x0 = fminf(x0, __shfl_xor_sync(0xffffffffu, x0, o)); x1 = fmaxf(x1, __shfl_xor_sync(0xffffffffu, x1, o));
        }
        // pixels within the fan's inscribed circle are inside, pixels beyond its largest vertex distance outside,
        // whatever the crossing test would say (margins of 0.1 % and 0.01 px: nothing near the boundary is decided here)
        const float cyf = (float)pyx[2 * r], cxf = (float)pyx[2 * r + 1];
        float d2 = (yv - cyf) * (yv - cyf) + (xv - cxf) * (xv - cxf), d2min = d2, d2max = d2;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            d2min = fminf(d2min, __shfl_xor_sync(0xffffffffu, d2min, o));
            d2max = fmaxf(d2max, __shfl_xor_sync(0xffffffffu, d2max, o));
        }
        const float rin = fmaxf(sqrtf(d2min) * 0.9942f - 0.01f, 0.f);     // cos(pi / 32) = 0.99518: the chords' distance
        const float rout = sqrtf(d2max) * 1.001f + 0.01f;
        const float rin2 = rin * rin, rout2 = rout * rout;
        // minr = int(max(0, r.min())), maxr = min(shape[0] - 1, int(ceil(r.max())))
        const int minr = (int)fmaxf(0.f, y0), maxr = min(H - 1, (int)ceilf(y1));
        const int minc = (int)fmaxf(0.f, x0), maxc = min(W - 1, (int)ceilf(x1));
        if (maxr < minr || maxc < minc) continue;
        const int bw = maxc - minc + 1;
        for (int yy = minr + part; yy <= maxr; yy += SEG_RENDER_SPLIT)
            for (int xx = minc + lane; xx <= maxc; xx += 32) {
                const float q2 = ((float)yy - cyf) * ((float)yy - cyf) + ((float)xx - cxf) * ((float)xx - cxf);
                if (q2 > rout2) continue;
                if (q2 < rin2 || seg_pnpoly(s_v[wib][1], s_v[wib][0], (double)xx, (double)yy))
                    atomicMin(flabels + (size_t)yy * W + xx, k + 1);
            }
        (void)bw;
    }
}

// field blockIdx.y: background -> 0, label k + 1 of the global kept order -> rank within the field + 1; n_inst [F]
__global__ void seg_finalize_kernel(int32_t* __restrict__ labels, size_t n, const int* __restrict__ kstart,
                                    int32_t* __restrict__ n_inst) {
    const int f = blockIdx.y;
    labels += (size_t)f * n;
    const int base = kstart[f];
    if (n_inst && blockIdx.x == 0 && threadIdx.x == 0) n_inst[f] = kstart[f + 1] - base;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int32_t v = labels[i];
        if (v == SEG_EMPTY) labels[i] = 0;
        else if (base) labels[i] = v - base;
    }
}

__global__ void seg_details_kernel(const float* __restrict__ vy, const float* __restrict__ vx, const int* __restrict__ pyx,
                                   const float* __restrict__ pprob, const int* __restrict__ kept_rank,
                                   const int* __restrict__ n_kept, int cap, int32_t* __restrict__ points,
                                   float* __restrict__ prob, float* __restrict__ coord) {
    const int k = blockIdx.x, lane = threadIdx.x;
    if (k >= min(*n_kept, cap)) return;
    const int r = kept_rank[k];
    coord[((size_t)k * 2 + 0) * SEG_RAYS + lane] = vy[(size_t)r * SEG_RAYS + lane];
    coord[((size_t)k * 2 + 1) * SEG_RAYS + lane] = vx[(size_t)r * SEG_RAYS + lane];
    if (lane == 0) { points[2 * k] = pyx[2 * r]; points[2 * k + 1] = pyx[2 * r + 1]; prob[k] = pprob[r]; }
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
template <int N, int TILES, int EPI>
int launch_seg_conv(cia_ctx* h, const SegConvArgs& a, cudaStream_t s) {
    using C = SegCfg<N, TILES>;
    auto kern = seg_conv_kernel<N, TILES, EPI>;
    if (first_use(h, (const void*)kern))
        CIA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_B));
    const int tiles_x = (a.W + 8 * TILES - 1) / (8 * TILES), tiles_y = (a.H + 15) / 16;
    int grid = tiles_x * tiles_y * a.F * a.groups;
    if (grid > C::CTAS_PER_SM * h->num_sms) grid = C::CTAS_PER_SM * h->num_sms;
    kern<<<grid, 256, C::SMEM_B, s>>>(a);
    CIA_LAUNCH_CHECK();
    return CIA_OK;
}

typedef CUresult (*SegTensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                         const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                         CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

template <int N, int TILES, int POOL = 0>
int launch_seg_conv_tma(cia_ctx* h, const SegConvArgs& a, cudaStream_t s) {
    using C = SegCfg<N, TILES>;
    using T = SegTmaCfg<N, TILES>;
    static SegTensorMapEncodeFn encode = [] {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess) fn = nullptr;
        return (SegTensorMapEncodeFn)fn;
    }();
    if (!encode) { h->err = "cuTensorMapEncodeTiled is not available from this driver"; return CIA_E_UNSUPPORTED; }
    // chunk-planar fp16 activations [F][4 planes][H][W][8]: dims (8, x, y, field * 4 + plane); out-of-bounds reads give zeros
    CUtensorMap tm;
    const cuuint64_t dims[4] = {8, (cuuint64_t)a.W, (cuuint64_t)a.H, (cuuint64_t)4 * a.F};
    const cuuint64_t strides[3] = {16, (cuuint64_t)16 * a.W, (cuuint64_t)16 * a.W * a.H};
    const cuuint32_t box[4] = {8, (cuuint32_t)C::COLS, 18, 4};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    if (encode(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, (void*)a.src0, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) {
        h->err = "cuTensorMapEncodeTiled failed (segmentation activations)";
        return CIA_E_CUDA;
    }
    auto kern = seg_conv_tma_kernel<N, TILES, POOL>;
    if (first_use(h, (const void*)kern))
        CIA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, T::SMEM_B));
    const int tiles_x = (a.W + 8 * TILES - 1) / (8 * TILES), tiles_y = (a.H + 15) / 16;
    int grid = tiles_x * tiles_y * a.F;
    if (grid > h->num_sms) grid = h->num_sms;
    kern<<<grid, T::THREADS, T::SMEM_B, s>>>(tm, a.w, a.bias, a.out, a.out_pool, a.H, a.W, a.F);
    CIA_LAUNCH_CHECK();
    return CIA_OK;
}

template <int N, int TILES>
int launch_seg_conv_ws(cia_ctx* h, const SegConvArgs& a, cudaStream_t s) {
    using T = SegWsCfg<N, TILES>;
    auto kern = seg_conv_ws_kernel<N, TILES>;
    if (first_use(h, (const void*)kern))
        CIA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, T::SMEM_B));
    const int tiles_x = (a.W + 8 * TILES - 1) / (8 * TILES), tiles_y = (a.H + 15) / 16;
    int grid = tiles_x * tiles_y * a.F * a.groups;
    if (grid > h->num_sms) grid = h->num_sms;
    kern<<<grid, T::THREADS, T::SMEM_B, s>>>(a);
    CIA_LAUNCH_CHECK();
    return CIA_OK;
}

// heads over a CIN = 128 `features` map: weights as one linear image [plane][48][8] (the chunks of the staged layout
// are consecutive planes, so the same upload serves both kernels)
int launch_seg_heads_tma(cia_ctx* h, const SegConvArgs& a, cudaStream_t s) {
    using T = SegHeadsCfg<128>;
    static SegTensorMapEncodeFn encode = [] {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess) fn = nullptr;
        return (SegTensorMapEncodeFn)fn;
    }();
    if (!encode) { h->err = "cuTensorMapEncodeTiled is not available from this driver"; return CIA_E_UNSUPPORTED; }
    CUtensorMap tm;
    const cuuint64_t dims[4] = {8, (cuuint64_t)a.W, (cuuint64_t)a.H, (cuuint64_t)T::PLANES * a.F};   // field * PLANES + plane
    const cuuint64_t strides[3] = {16, (cuuint64_t)16 * a.W, (cuuint64_t)16 * a.W * a.H};
    const cuuint32_t box[4] = {8, 16, 16, (cuuint32_t)T::PLANES};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    if (encode(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, (void*)a.src0, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) {
        h->err = "cuTensorMapEncodeTiled failed (segmentation features)";
        return CIA_E_CUDA;
    }
    auto kern = seg_heads_tma_kernel<128>;
    if (first_use(h, (const void*)kern))
        CIA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, T::SMEM_B));
    int grid = ((a.W + 15) / 16) * ((a.H + 15) / 16) * a.F;
    if (grid > h->num_sms) grid = h->num_sms;
    kern<<<grid, T::THREADS, T::SMEM_B, s>>>(tm, a.w, a.bias, a.prob, a.dist, a.H, a.W, a.F);
    CIA_LAUNCH_CHECK();
    return CIA_OK;
}

int launch_seg_heads(cia_ctx* h, const SegConv& c, const SegConvArgs& a, cudaStream_t s) {
    if (h->seg_conv_tma && c.cin == 128 && ((size_t)a.src0 % 16) == 0) return launch_seg_heads_tma(h, a, s);
    return launch_seg_conv<48, 2, 1>(h, a, s);
}

// does this layer run in the TMA-fed kernel (and can therefore hand a pooled copy of its output to the next layer)?
bool seg_tma_eligible(const cia_ctx* h, const SegConv& c, int mode) {
    return h->seg_conv_tma && mode == 0 && c.chunks == 1 && c.groups == 1;
}

// one 3x3 layer of the plan: the TMA-fed kernel where the layer reads its producer directly with one 32-channel chunk
int launch_seg_layer(cia_ctx* h, const SegConv& c, const SegConvArgs& a, cudaStream_t s) {
    const bool tma = h->seg_conv_tma && a.mode == 0 && c.chunks == 1 && c.groups == 1 && ((size_t)a.src0 % 16) == 0;
    if (tma && a.out_pool && (a.H & 1) == 0 && (a.W & 1) == 0) {       // pooled copy for the next layer (see seg_tma_eligible)
        const bool both = a.out != nullptr;
        if (c.n_tile == 32) return both ? launch_seg_conv_tma<32, 4, 2>(h, a, s) : launch_seg_conv_tma<32, 4, 1>(h, a, s);
        if (c.n_tile == 64) return both ? launch_seg_conv_tma<64, 4, 2>(h, a, s) : launch_seg_conv_tma<64, 4, 1>(h, a, s);
        return both ? launch_seg_conv_tma<128, 2, 2>(h, a, s) : launch_seg_conv_tma<128, 2, 1>(h, a, s);
    }
    if (tma && c.n_tile == 32) return launch_seg_conv_tma<32, 4>(h, a, s);
    if (tma && c.n_tile == 64) return launch_seg_conv_tma<64, 4>(h, a, s);
    if (tma && c.n_tile == 128) return launch_seg_conv_tma<128, 2>(h, a, s);
    // measured per layer on B200 (profiles/r2u_seg_launches.txt): the software producer pays for layers with two or more
    // chunks and 64+ output channels per CTA (long MMA phases per step); short steps (N = 32) and pooled single- or
    // double-chunk inputs are faster with three co-resident staged CTAs.  seg_conv_ws = 2 forces it everywhere (tests).
    const bool ws = h->seg_conv_ws == 2 ||
                    (h->seg_conv_ws == 1 && c.n_tile >= 64 && c.chunks >= 2 && !(a.mode == 1 && c.chunks == 2));
    if (ws) {
        if (c.n_tile == 128) return launch_seg_conv_ws<128, 2>(h, a, s);
        if (c.n_tile == 64) return launch_seg_conv_ws<64, 4>(h, a, s);
        return launch_seg_conv_ws<32, 4>(h, a, s);
    }
    if (c.n_tile == 128) return launch_seg_conv<128, 2, 0>(h, a, s);
    if (c.n_tile == 64) return launch_seg_conv<64, 4, 0>(h, a, s);
    return launch_seg_conv<32, 4, 0>(h, a, s);
}

int free_model(SegModel* m) {
    if (!m) return 0;
    for (auto& c : m->conv) { cudaFree(c.w_img); cudaFree(c.bias); cudaFree(c.w32); }
    cudaFree(m->ray_sin); cudaFree(m->ray_cos);
    cudaFree(m->act.p); cudaFree(m->post.p); cudaFree(m->cubtmp.p); cudaFree(m->screen.p);
    delete m;
    return 0;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace

void k_seg_free(cia_ctx* h) {
    free_model(h->seg);
    h->seg = nullptr;
}

// Builds the execution plan of StarDist2D._build + csbdeep unet_block for the given configuration and uploads the
// weights as UMMA operand images.  kernels[l]: HWIO float32 [kh][kw][cin][cout] in the order the model applies them
// (grid blocks, down levels, middle, up levels, `features`, `prob`, `dist`).
int k_seg_load(cia_ctx* h, const cia_seg_config* cfg, int n_layers, const float* const* kernels,
               const float* const* biases, const int64_t* shapes, const double* ray_sin, const double* ray_cos) {
    k_seg_free(h);
    if (cfg->n_rays != SEG_RAYS) { h->err = "segmentation: n_rays must be 32"; return CIA_E_UNSUPPORTED; }
    if (cfg->n_channel_in != 1) { h->err = "segmentation: n_channel_in must be 1"; return CIA_E_UNSUPPORTED; }
    if (cfg->grid != 1 && cfg->grid != 2 && cfg->grid != 4) { h->err = "segmentation: grid must be 1, 2 or 4 (square)"; return CIA_E_UNSUPPORTED; }
    if (cfg->unet_n_depth < 1 || cfg->unet_n_depth > 5 || cfg->unet_n_conv_per_depth < 1 || cfg->net_conv_after_unet <= 0) {
        h->err = "segmentation: unsupported U-Net configuration"; return CIA_E_UNSUPPORTED;
    }
    SegModel* m = new SegModel();
    m->grid = cfg->grid; m->depth = cfg->unet_n_depth; m->n_conv = cfg->unet_n_conv_per_depth;
    m->base = cfg->unet_n_filter_base; m->after = cfg->net_conv_after_unet; m->n_rays = cfg->n_rays;

    // ---- plan ----
    std::vector<int> plan_cout;
    int cur = -1, cur_ch = 1, shift = 0;
    bool pend_pool = false;
    int up_low = -1, up_low_ch = 0, up_skip = -1, up_skip_ch = 0;
    auto new_buf = [&](int ch, int sh) { m->buf_ch.push_back(ch); m->buf_shift.push_back(sh); return (int)m->buf_ch.size() - 1; };
    auto emit = [&](int cout) {
        SegOp op{};
        op.layer = (int)plan_cout.size();
        op.shift = shift;
        if (cur < 0) { op.mode = -1; op.src0 = op.src1 = -1; op.c0 = 1; op.c1 = 0; }
        else if (up_low >= 0) { op.mode = 2; op.src0 = up_low; op.src1 = up_skip; op.c0 = up_low_ch; op.c1 = up_skip_ch; up_low = -1; }
        else { op.mode = pend_pool ? 1 : 0; op.src0 = cur; op.src1 = -1; op.c0 = cur_ch; op.c1 = 0; }
        pend_pool = false;
        op.pool_dst = -1; op.full_needed = 1;
        op.dst = new_buf(cout, shift);
        cur = op.dst; cur_ch = cout;
        plan_cout.push_back(cout);
        m->ops.push_back(op);
    };
    for (int pooled = 1; pooled < m->grid; pooled *= 2) {
        for (int k = 0; k < m->n_conv; ++k) emit(m->base);
        pend_pool = true; ++shift;
    }
    std::vector<int> skip(m->depth), skip_ch(m->depth);
    for (int n = 0; n < m->depth; ++n) {
        for (int k = 0; k < m->n_conv; ++k) emit(m->base << n);
        skip[n] = cur; skip_ch[n] = cur_ch;
        pend_pool = true; ++shift;
    }
    for (int k = 0; k < m->n_conv - 1; ++k) emit(m->base << m->depth);
    emit(m->base << std::max(0, m->depth - 1));
    for (int n = m->depth - 1; n >= 0; --n) {
        --shift;
        up_low = cur; up_low_ch = cur_ch; up_skip = skip[n]; up_skip_ch = skip_ch[n];
        for (int k = 0; k < m->n_conv - 1; ++k) emit(m->base << n);
        emit(m->base << std::max(0, n - 1));
    }
    emit(m->after);
    // a layer whose output is max-pooled by the next one gets a buffer for the pooled copy (written by the producer's
    // epilogue when it runs in the TMA-fed kernel); the full-resolution map is only needed where something else reads it
    for (size_t l = 0; l + 1 < m->ops.size(); ++l) {
        if (m->ops[l + 1].mode != 1 || m->ops[l + 1].src0 != m->ops[l].dst) continue;
        m->ops[l].pool_dst = new_buf(m->buf_ch[m->ops[l].dst], m->ops[l].shift + 1);
        bool other_reader = false;
        for (size_t k = l + 2; k < m->ops.size(); ++k)
            other_reader |= m->ops[k].src0 == m->ops[l].dst || m->ops[k].src1 == m->ops[l].dst;
        m->ops[l].full_needed = other_reader ? 1 : 0;
    }
    const int n_body = (int)plan_cout.size();
    if (n_layers != n_body + 2) {
        h->err = "segmentation: expected " + std::to_string(n_body + 2) + " conv layers, got " + std::to_string(n_layers);
        free_model(m); return CIA_E_ARG;
    }

    // ---- weights ----
    m->conv.resize(n_body + 1);
    auto fail = [&](const std::string& why) { h->err = "segmentation: " + why; free_model(m); return CIA_E_UNSUPPORTED; };
    for (int l = 0; l < n_body; ++l) {
        const SegOp& op = m->ops[l];
        const int64_t* sh = shapes + 4 * l;
        const int cin = op.c0 + op.c1, cout = plan_cout[l];
        if (sh[0] != 3 || sh[1] != 3 || sh[2] != cin || sh[3] != cout)
            return fail("layer " + std::to_string(l) + " has shape [" + std::to_string(sh[0]) + "," + std::to_string(sh[1]) + "," +
                        std::to_string(sh[2]) + "," + std::to_string(sh[3]) + "], the configuration implies [3,3," +
                        std::to_string(cin) + "," + std::to_string(cout) + "]");
        SegConv& c = m->conv[l];
        c.cin = cin; c.cout = cout; c.taps = 9;
        if (op.mode == -1) {
            if (cout % 8 || cout > 128) return fail("first layer needs Cout % 8 == 0 and <= 128");
            CIA_CUDA(cudaMalloc((void**)&c.w32, (size_t)9 * cout * sizeof(float)));
            CIA_CUDA(cudaMemcpy(c.w32, kernels[l], (size_t)9 * cout * sizeof(float), cudaMemcpyHostToDevice));
            CIA_CUDA(cudaMalloc((void**)&c.bias, cout * sizeof(float)));
            CIA_CUDA(cudaMemcpy(c.bias, biases[l], cout * sizeof(float), cudaMemcpyHostToDevice));
            continue;
        }
        if (cin % SEG_KC || cout % 32 || op.c0 % SEG_KC) return fail("channel counts must be multiples of 32");
        c.n_tile = cout % 128 == 0 ? 128 : cout % 64 == 0 ? 64 : 32;
        c.groups = cout / c.n_tile; c.chunks = cin / SEG_KC;
        std::vector<__half> img((size_t)c.groups * c.chunks * 9 * (SEG_KC / 8) * c.n_tile * 8);
        const float* w = kernels[l];
        for (int g = 0; g < c.groups; ++g)
            for (int kc = 0; kc < c.chunks; ++kc)
                for (int tap = 0; tap < 9; ++tap)
                    for (int p = 0; p < SEG_KC / 8; ++p)
                        for (int nn = 0; nn < c.n_tile; ++nn)
                            for (int j = 0; j < 8; ++j) {
                                const int ci = kc * SEG_KC + p * 8 + j, co = g * c.n_tile + nn;
                                img[(((((size_t)g * c.chunks + kc) * 9 + tap) * (SEG_KC / 8) + p) * c.n_tile + nn) * 8 + j] =
                                    __float2half_rn(w[((size_t)tap * cin + ci) * cout + co]);
                            }
        CIA_CUDA(cudaMalloc((void**)&c.w_img, img.size() * sizeof(__half)));
        CIA_CUDA(cudaMemcpy(c.w_img, img.data(), img.size() * sizeof(__half), cudaMemcpyHostToDevice));
        CIA_CUDA(cudaMalloc((void**)&c.bias, cout * sizeof(float)));
        CIA_CUDA(cudaMemcpy(c.bias, biases[l], cout * sizeof(float), cudaMemcpyHostToDevice));
    }
    {   // heads: `prob` [1,1,after,1] and `dist` [1,1,after,n_rays] as one 1-tap image, columns 0..31 dist, 32 prob
        const int64_t* sp = shapes + 4 * n_body;
        const int64_t* sd = shapes + 4 * (n_body + 1);
        if (sp[0] != 1 || sp[1] != 1 || sp[2] != m->after || sp[3] != 1 || sd[0] != 1 || sd[1] != 1 || sd[2] != m->after ||
            sd[3] != SEG_RAYS)
            return fail("prob / dist heads must be 1x1 convolutions over the `features` layer");
        if (m->after % SEG_KC) return fail("net_conv_after_unet must be a multiple of 32");
        SegConv& c = m->conv[n_body];
        c.cin = m->after; c.cout = 48; c.taps = 1; c.n_tile = 48; c.groups = 1; c.chunks = m->after / SEG_KC;
        std::vector<__half> img((size_t)c.chunks * (SEG_KC / 8) * 48 * 8, __float2half_rn(0.f));
        std::vector<float> b(48, 0.f);
        const float* wp = kernels[n_body];
        const float* wd = kernels[n_body + 1];
        for (int kc = 0; kc < c.chunks; ++kc)
            for (int p = 0; p < SEG_KC / 8; ++p)
                for (int nn = 0; nn <= SEG_RAYS; ++nn)
                    for (int j = 0; j < 8; ++j) {
                        const int ci = kc * SEG_KC + p * 8 + j;
                        const float v = nn < SEG_RAYS ? wd[(size_t)ci * SEG_RAYS + nn] : wp[ci];
                        img[((((size_t)kc * (SEG_KC / 8)) + p) * 48 + nn) * 8 + j] = __float2half_rn(v);
                    }
        for (int nn = 0; nn < SEG_RAYS; ++nn) b[nn] = biases[n_body + 1][nn];
        b[SEG_RAYS] = biases[n_body][0];
        CIA_CUDA(cudaMalloc((void**)&c.w_img, img.size() * sizeof(__half)));
        CIA_CUDA(cudaMemcpy(c.w_img, img.data(), img.size() * sizeof(__half), cudaMemcpyHostToDevice));
        CIA_CUDA(cudaMalloc((void**)&c.bias, 48 * sizeof(float)));
        CIA_CUDA(cudaMemcpy(c.bias, b.data(), 48 * sizeof(float), cudaMemcpyHostToDevice));
    }
    CIA_CUDA(cudaMalloc((void**)&m->ray_sin, SEG_RAYS * sizeof(double)));
    CIA_CUDA(cudaMalloc((void**)&m->ray_cos, SEG_RAYS * sizeof(double)));
    CIA_CUDA(cudaMemcpy(m->ray_sin, ray_sin, SEG_RAYS * sizeof(double), cudaMemcpyHostToDevice));
    CIA_CUDA(cudaMemcpy(m->ray_cos, ray_cos, SEG_RAYS * sizeof(double), cudaMemcpyHostToDevice));
    h->seg = m;
    return CIA_OK;
}

// n_fields uint16 fields [F][H][W] -> float32 [F][Hp][Wp] (Hp >= H, Wp >= W: reflect-padded); mi_ma_out [F][2] or null
int k_seg_normalize(cia_ctx* h, const uint16_t* img, int n_fields, int H, int W, int Hp, int Wp, double pmin, double pmax,
                    float* out, float* mi_ma_out, cudaStream_t s) {
    if (n_fields > 65535) { h->err = "segmentation: at most 65535 fields per call"; return CIA_E_ARG; }
    // scratch of the handle's own (not ws_misc, which the autoencoder uses): [F] histogram copies (4 MB per field),
    // [F][2048] sums of 32 bins, [F][2] percentiles
    const size_t words = (size_t)n_fields * (SEG_HIST_FIELD + 2048 + 2);
    int rc = ws_reserve(h, h->ws_seg_norm, words * sizeof(uint32_t));
    if (rc) return rc;
    uint32_t* hist = (uint32_t*)h->ws_seg_norm.p;
    uint32_t* wsum = hist + (size_t)n_fields * SEG_HIST_FIELD;
    float* mima = mi_ma_out ? mi_ma_out : (float*)(wsum + (size_t)n_fields * 2048);
    const size_t n = (size_t)H * W;
    CIA_CUDA(cudaMemsetAsync(hist, 0, (size_t)n_fields * SEG_HIST_FIELD * sizeof(uint32_t), s));
    const int gx = std::max(SEG_HIST_COPIES, h->num_sms * 8 / n_fields);
    seg_hist_kernel<<<dim3(gx, n_fields), 256, 0, s>>>(img, n, hist);
    CIA_LAUNCH_CHECK();
    seg_hist_reduce_kernel<<<dim3(65536 / 256, n_fields), 256, 0, s>>>(hist, wsum);
    CIA_LAUNCH_CHECK();
    seg_percentile_kernel<<<n_fields, 1024, 0, s>>>(hist, wsum, n, pmin / 100.0, pmax / 100.0, mima);   // np.true_divide(q, 100)
    CIA_LAUNCH_CHECK();
    seg_normalize_kernel<<<dim3(gx, n_fields), 256, 0, s>>>(img, H, W, Hp, Wp, mima, 1e-20f, out);
    CIA_LAUNCH_CHECK();
    return CIA_OK;
}

int k_seg_div(cia_ctx* h) { return h->seg ? h->seg->grid << h->seg->depth : 0; }
int k_seg_grid(cia_ctx* h) { return h->seg ? h->seg->grid : 0; }

// The network: F normalized float32 fields [F][H][W] (device) -> prob [F][H/grid][W/grid], dist [F][H/grid][W/grid][32].
// Every layer is one launch for all F fields; per field the arithmetic is that of a one-field call.
int k_seg_predict(cia_ctx* h, const float* img, int F, int H, int W, float* prob_out, float* dist_out, cudaStream_t s) {
    SegModel* m = h->seg;
    if (!m) { h->err = "segmentation model not loaded (cia_seg_load)"; return CIA_E_STATE; }
    if (F < 1) { h->err = "segmentation: n_fields must be >= 1"; return CIA_E_ARG; }
    const int div = m->grid << m->depth;
    if (H % div || W % div || H <= 0 || W <= 0) {
        h->err = "segmentation: field sides must be multiples of " + std::to_string(div) +
                 " (StarDist pads with np.pad(mode='reflect') otherwise: pad on the host)";
        return CIA_E_UNSUPPORTED;
    }
    // activation buffers [F][C/8][y][x][8] (bump allocation; no reuse: 1.4 GB per 2048 x 2048 field)
    std::vector<size_t> off(m->buf_ch.size());
    size_t total = 0;
    for (size_t b = 0; b < off.size(); ++b) {
        off[b] = total;
        total += align_up((size_t)F * m->buf_ch[b] * (H >> m->buf_shift[b]) * (W >> m->buf_shift[b]) * sizeof(__half), 256);
    }
    const int gs = m->grid == 1 ? 0 : (m->grid == 2 ? 1 : 2);
    const int Hg = H >> gs, Wg = W >> gs;
    const size_t prob_off = total; total += align_up((size_t)F * Hg * Wg * sizeof(float), 256);
    const size_t dist_off = total; total += align_up((size_t)F * Hg * Wg * SEG_RAYS * sizeof(float), 256);
    int rc = ws_reserve(h, m->act, total);
    if (rc) return rc;
    unsigned char* base = (unsigned char*)m->act.p;
    m->prob_map = (float*)(base + prob_off); m->dist_map = (float*)(base + dist_off);
    m->last_hg = Hg; m->last_wg = Wg;

    std::vector<char> pooled_by_producer(m->ops.size(), 0);
    for (size_t l = 0; l < m->ops.size(); ++l) {
        const SegOp& op = m->ops[l];
        const SegConv& c = m->conv[l];
        const int Ho = H >> op.shift, Wo = W >> op.shift;
        __half* out = (__half*)(base + off[op.dst]);
        if (op.mode == -1) {
            const size_t n = (size_t)F * Ho * ((Wo + 1) / 2);
            seg_first_kernel<<<(unsigned)((n + 255) / 256), 256, 10 * c.cout * sizeof(float), s>>>(img, c.w32, c.bias, out, Ho, Wo, c.cout, F);
            CIA_LAUNCH_CHECK();
            continue;
        }
        SegConvArgs a{};
        a.src0 = (const __half*)(base + off[op.src0]);
        a.src1 = op.src1 >= 0 ? (const __half*)(base + off[op.src1]) : nullptr;
        a.w = (const uint4*)c.w_img; a.bias = c.bias; a.out = out;
        a.H = Ho; a.W = Wo; a.F = F; a.c0 = op.c0; a.c1 = op.c1; a.mode = op.mode; a.ntaps = 9; a.groups = c.groups; a.chunks = c.chunks;
        // pooled input already written by the producer's epilogue: read it directly (a Cin = 32 layer then runs TMA-fed too)
        if (op.mode == 1 && l > 0 && pooled_by_producer[l - 1]) {
            a.mode = 0;
            a.src0 = (const __half*)(base + off[m->ops[l - 1].pool_dst]);
        }
        // and this layer's own pooled copy, when the next layer pools it and this one runs in the TMA-fed kernel
        pooled_by_producer[l] = h->seg_pool_out && op.pool_dst >= 0 && seg_tma_eligible(h, c, a.mode) && !(Ho & 1) && !(Wo & 1);
        if (pooled_by_producer[l]) {
            a.out_pool = (__half*)(base + off[op.pool_dst]);
            if (!op.full_needed) a.out = nullptr;
        }
        rc = launch_seg_layer(h, c, a, s);
        if (rc) return rc;
    }
    {
        const SegConv& c = m->conv.back();
        const SegOp& last = m->ops.back();
        SegConvArgs a{};
        a.src0 = (const __half*)(base + off[last.dst]);
        a.w = (const uint4*)c.w_img; a.bias = c.bias;
        a.prob = m->prob_map; a.dist = m->dist_map;
        a.H = Hg; a.W = Wg; a.F = F; a.c0 = c.cin; a.c1 = 0; a.mode = 0; a.ntaps = 1; a.groups = 1; a.chunks = c.chunks;
        rc = launch_seg_heads(h, c, a, s);
        if (rc) return rc;
    }
    if (prob_out) CIA_CUDA(cudaMemcpyAsync(prob_out, m->prob_map, (size_t)F * Hg * Wg * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (dist_out) CIA_CUDA(cudaMemcpyAsync(dist_out, m->dist_map, (size_t)F * Hg * Wg * SEG_RAYS * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return CIA_OK;
}

// One layer of the plan on caller-provided activations (tests: every staging mode / tile shape against a
// float32 convolution of the same fp16 operands).  layer = index into the plan, or -2 for the heads.
int k_seg_debug_layer(cia_ctx* h, int layer, const void* src0, const void* src1, const float* img, int Ho, int Wo,
                      void* out, float* prob, float* dist, cudaStream_t s) {
    SegModel* m = h->seg;
    if (!m) { h->err = "segmentation model not loaded"; return CIA_E_STATE; }
    if (layer == -2) {
        const SegConv& c = m->conv.back();
        SegConvArgs a{};
        a.src0 = (const __half*)src0; a.w = (const uint4*)c.w_img; a.bias = c.bias; a.prob = prob; a.dist = dist;
        a.H = Ho; a.W = Wo; a.F = 1; a.c0 = c.cin; a.mode = 0; a.ntaps = 1; a.groups = 1; a.chunks = c.chunks;
        return launch_seg_heads(h, c, a, s);
    }
    if (layer < 0 || layer >= (int)m->ops.size()) { h->err = "segmentation: no such layer"; return CIA_E_ARG; }
    const SegOp& op = m->ops[layer];
    const SegConv& c = m->conv[layer];
    if (op.mode == -1) {
        const size_t n = (size_t)Ho * ((Wo + 1) / 2);
        seg_first_kernel<<<(unsigned)((n + 255) / 256), 256, 10 * c.cout * sizeof(float), s>>>(img, c.w32, c.bias, (__half*)out, Ho, Wo, c.cout, 1);
        CIA_LAUNCH_CHECK();
        return CIA_OK;
    }
    SegConvArgs a{};
    a.src0 = (const __half*)src0; a.src1 = (const __half*)src1; a.w = (const uint4*)c.w_img; a.bias = c.bias; a.out = (__half*)out;
    a.H = Ho; a.W = Wo; a.F = 1; a.c0 = op.c0; a.c1 = op.c1; a.mode = op.mode; a.ntaps = 9; a.groups = c.groups; a.chunks = c.chunks;
    return launch_seg_layer(h, c, a, s);
}

int k_seg_layer_info(cia_ctx* h, int layer, int* info /* [6]: mode, c0, c1, cout, shift, n_layers */) {
    SegModel* m = h->seg;
    if (!m) { h->err = "segmentation model not loaded"; return CIA_E_STATE; }
    if (layer < 0 || layer >= (int)m->ops.size()) { h->err = "segmentation: no such layer"; return CIA_E_ARG; }
    const SegOp& op = m->ops[layer];
    info[0] = op.mode; info[1] = op.c0; info[2] = op.c1; info[3] = m->conv[layer].cout; info[4] = op.shift;
    info[5] = (int)m->ops.size();
    return CIA_OK;
}

// _instances_from_prediction for F fields: prob [F][Hgp][Wgp], dist [F][Hgp][Wgp][32] (device; null = the last
// cia_seg_predict's), candidates inside the logical hg x wg part of each map -> labels int32 [F][H][W] (rank within the
// field + 1), n_inst_dev [F].  One launch sequence for all fields: the suppression runs every field's rounds together.
int k_seg_instances(cia_ctx* h, const float* prob, const float* dist, int F, int Hgp, int Wgp, int hg, int wg, int grid,
                    int H, int W, double prob_thresh, double nms_thresh, int32_t* labels, int32_t* n_inst_dev, cudaStream_t s) {
    SegModel* m = h->seg;
    if (!m) { h->err = "segmentation model not loaded (cia_seg_load)"; return CIA_E_STATE; }
    if (!prob) prob = m->prob_map;
    if (!dist) dist = m->dist_map;
    if (!prob || !dist) { h->err = "segmentation: no prob / dist maps"; return CIA_E_ARG; }
    if (F < 1 || F > 65535 || hg > Hgp || wg > Wgp) { h->err = "segmentation: bad field count or map size"; return CIA_E_ARG; }
    if ((size_t)F * Hgp * Wgp >= 0x7fffffffull) { h->err = "segmentation: grid too large"; return CIA_E_UNSUPPORTED; }
    const int cap = F * Hgp * Wgp;
    const int nbx = (W + SEG_BIN - 1) / SEG_BIN, nby = (H + SEG_BIN - 1) / SEG_BIN, nbins = F * nbx * nby;
    const bool wide = F > 1;                        // 64-bit keys with the field above bit 32
    int key_bits = 32;
    while ((1 << (key_bits - 32)) < F) ++key_bits;   // 32 + ceil(log2 F)
    const size_t kb = wide ? 8 : 4;

    // workspace carve-up
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o += align_up(bytes, 256); return at; };
    const size_t o_keys0 = take((size_t)cap * kb), o_keys1 = take((size_t)cap * kb), o_vals0 = take((size_t)cap * 4), o_vals1 = take((size_t)cap * 4);
    const size_t o_binof = take((size_t)cap * 4), o_bcnt = take((size_t)(nbins + 1) * 4), o_bcur = take((size_t)(nbins + 1) * 4);
    const size_t o_vy = take((size_t)cap * SEG_RAYS * 4), o_vx = take((size_t)cap * SEG_RAYS * 4);
    const size_t o_pyx = take((size_t)cap * 8), o_pp = take((size_t)cap * 4), o_rm = take((size_t)cap * 4);
    const size_t o_area = take((size_t)cap * 8), o_state = take((size_t)cap * 4), o_flags = take((size_t)cap * 4);
    const size_t o_excl = take((size_t)cap * 4), o_kept = take((size_t)cap * 4);
    const size_t o_bins = take((size_t)(nbins + 1) * 4), o_small = take(64);
    const size_t o_brank = take((size_t)cap * 4), o_byxr = take((size_t)cap * 16), o_pos = take((size_t)cap * 4);
    const size_t o_rfield = take((size_t)cap * 4), o_kstart = take((size_t)(F + 1) * 4);
    int rc = ws_reserve(h, m->post, o);
    if (rc) return rc;
    unsigned char* b = (unsigned char*)m->post.p;
    void* keys0 = b + o_keys0; void* keys1 = b + o_keys1;
    unsigned* vals0 = (unsigned*)(b + o_vals0); unsigned* vals1 = (unsigned*)(b + o_vals1);
    int* bin_of = (int*)(b + o_binof); int* bin_count = (int*)(b + o_bcnt); int* bin_cursor = (int*)(b + o_bcur);
    float* vy = (float*)(b + o_vy); float* vx = (float*)(b + o_vx);
    int* pyx = (int*)(b + o_pyx); float* pp = (float*)(b + o_pp); float* rm = (float*)(b + o_rm);
    double* area = (double*)(b + o_area);
    int* state = (int*)(b + o_state); int* flags = (int*)(b + o_flags); int* excl = (int*)(b + o_excl);
    int* kept = (int*)(b + o_kept); int* bins = (int*)(b + o_bins);
    int* b_rank = (int*)(b + o_brank); float4* b_yxr = (float4*)(b + o_byxr); int* pos = (int*)(b + o_pos);
    int* rfield = (int*)(b + o_rfield); int* kstart = (int*)(b + o_kstart);
    int* small = (int*)(b + o_small);         // [0] count, [1] rmax bits, [2..4] nms counters, [5] n_kept
    m->last_cap = cap; m->vy = vy; m->vx = vx; m->pprob = pp; m->pyx = pyx; m->kept_rank = kept; m->n_kept = small + 5;

    typedef unsigned long long K64;
    size_t tmp_sort = 0, tmp_scan = 0;
    if (wide) cub::DeviceRadixSort::SortPairs(nullptr, tmp_sort, (K64*)keys0, (K64*)keys1, vals0, vals1, cap, 0, key_bits, s);
    else cub::DeviceRadixSort::SortPairs(nullptr, tmp_sort, (unsigned*)keys0, (unsigned*)keys1, vals0, vals1, cap, 0, 32, s);
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_scan, flags, excl, cap, s);
    rc = ws_reserve(h, m->cubtmp, std::max(tmp_sort, tmp_scan));
    if (rc) return rc;
    size_t tmp_bytes = m->cubtmp.cap;

    CIA_CUDA(cudaMemsetAsync(keys0, 0xFF, (size_t)cap * kb, s));
    CIA_CUDA(cudaMemsetAsync(bin_count, 0, (size_t)(nbins + 1) * 4, s));
    CIA_CUDA(cudaMemsetAsync(state, 0, (size_t)cap * 4, s));
    CIA_CUDA(cudaMemsetAsync(small, 0, 64, s));
    CIA_CUDA(cudaMemsetAsync(labels, 0x7F, (size_t)F * H * W * sizeof(int32_t), s));
    seg_cand_flags_kernel<<<(cap + 255) / 256, 256, 0, s>>>(prob, F, Hgp, Wgp, hg, wg, (float)prob_thresh, 2, flags);
    CIA_LAUNCH_CHECK();
    tmp_bytes = m->cubtmp.cap;
    CIA_CUDA(cub::DeviceScan::ExclusiveSum(m->cubtmp.p, tmp_bytes, flags, excl, cap, s));
    h->launches++;
    tmp_bytes = m->cubtmp.cap;
    if (wide) {
        seg_cand_scatter_kernel<K64><<<(cap + 255) / 256, 256, 0, s>>>(prob, flags, excl, cap, Hgp * Wgp, (K64*)keys0, vals0, small);
        CIA_LAUNCH_CHECK();
        CIA_CUDA(cub::DeviceRadixSort::SortPairs(m->cubtmp.p, tmp_bytes, (K64*)keys0, (K64*)keys1, vals0, vals1, cap, 0, key_bits, s));
    } else {
        seg_cand_scatter_kernel<unsigned><<<(cap + 255) / 256, 256, 0, s>>>(prob, flags, excl, cap, Hgp * Wgp, (unsigned*)keys0, vals0, small);
        CIA_LAUNCH_CHECK();
        CIA_CUDA(cub::DeviceRadixSort::SortPairs(m->cubtmp.p, tmp_bytes, (unsigned*)keys0, (unsigned*)keys1, vals0, vals1, cap, 0, 32, s));
    }
    h->launches++;
    seg_polygons_kernel<<<(cap + 127) / 128, 128, 0, s>>>(vals1, small, cap, prob, dist, Hgp, Wgp, grid, m->ray_sin, m->ray_cos, H, W,
                                                         vy, vx, pyx, pp, rm, area, bin_of, bin_count, (unsigned*)(small + 1), rfield);
    CIA_LAUNCH_CHECK();
    seg_bins_kernel<<<1, 1024, 0, s>>>(bin_count, nbins, bins, bin_cursor);
    CIA_LAUNCH_CHECK();
    seg_binorder_kernel<<<(cap + 255) / 256, 256, 0, s>>>(bin_of, bin_cursor, small, cap, pyx, rm, rfield, b_rank, b_yxr, pos);
    CIA_LAUNCH_CHECK();
    {
        NmsArgs a{};
        a.vy = vy; a.vx = vx; a.pyx = pyx; a.area = area; a.b_rank = b_rank; a.b_yxr = b_yxr; a.bin_start = bins; a.count = small;
        a.rmax_all = (const unsigned*)(small + 1); a.state = state; a.cnt = small + 2; a.nbx = nbx; a.nby = nby; a.cap = cap;
        a.thr = nms_thresh;
        int per_sm = 0;
        CIA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, seg_nms_kernel, 256, 0));
        if (per_sm < 1) { h->err = "segmentation: NMS kernel does not fit"; return CIA_E_CUDA; }
        if (per_sm > 4) per_sm = 4;
        void* args[] = {(void*)&a};
        CIA_CUDA(cudaLaunchCooperativeKernel((void*)seg_nms_kernel, dim3(h->num_sms * per_sm), dim3(256), args, 0, s));
        CIA_LAUNCH_CHECK();
    }
    seg_flags_kernel<<<(cap + 255) / 256, 256, 0, s>>>(state, pos, small, cap, flags);
    CIA_LAUNCH_CHECK();
    tmp_bytes = m->cubtmp.cap;
    CIA_CUDA(cub::DeviceScan::ExclusiveSum(m->cubtmp.p, tmp_bytes, flags, excl, cap, s));
    h->launches++;
    seg_compact_kernel<<<(cap + 255) / 256, 256, 0, s>>>(flags, excl, cap, small, rfield, F, kept, small + 5, kstart);
    CIA_LAUNCH_CHECK();
    seg_render_kernel<<<h->num_sms * 8, 256, 0, s>>>(vy, vx, pyx, kept, small + 5, rfield, H, W, labels);
    CIA_LAUNCH_CHECK();
    seg_finalize_kernel<<<dim3(std::max(1, h->num_sms * 8 / F), F), 256, 0, s>>>(labels, (size_t)H * W, kstart, n_inst_dev);
    CIA_LAUNCH_CHECK();
    return CIA_OK;
}

int k_seg_screen_buffers(cia_ctx* h, size_t norm_bytes, size_t label_bytes, float** norm, int32_t** labels) {
    SegModel* m = h->seg;
    if (!m) { h->err = "segmentation model not loaded (cia_seg_load)"; return CIA_E_STATE; }
    const size_t lo = align_up(norm_bytes, 256);
    const int rc = ws_reserve(h, m->screen, lo + label_bytes);
    if (rc) return rc;
    *norm = (float*)m->screen.p;
    *labels = (int32_t*)((unsigned char*)m->screen.p + lo);
    return CIA_OK;
}

int k_seg_details(cia_ctx* h, int cap, int32_t* points, float* prob, float* coord, cudaStream_t s) {
    SegModel* m = h->seg;
    if (!m || !m->vy) { h->err = "segmentation: no instances computed yet"; return CIA_E_STATE; }
    if (cap <= 0) return CIA_OK;
    seg_details_kernel<<<cap, SEG_RAYS, 0, s>>>(m->vy, m->vx, m->pyx, m->pprob, m->kept_rank, m->n_kept, cap, points, prob, coord);
    CIA_LAUNCH_CHECK();
    return CIA_OK;
}
