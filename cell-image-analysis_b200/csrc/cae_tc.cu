// cae_tc.cu -- K3 tensor-core path: the convolutional autoencoder as tcgen05 implicit
// GEMMs (UMMA, accumulators in TMEM), one kernel per layer, activations as fp16 in
// "chunk-planar" order [cell][C/8][y][x][8] so that every 16-byte unit is one pixel's 8
// channels -- exactly one row of a K-major UMMA core matrix.
//
// Replaces autoencoder.predict + MSE/MAE (improved_detection.py:125-127) and, in
// precision mode 1, encoder.predict (det:130); architecture CAE_improved_modeltrain.py:188-216.
//
// Implicit GEMM without im2col: a padded input block lives in shared memory; for filter
// tap (dy,dx) the A operand of the MMA is the SAME block addressed with a shifted start
// address (descriptor start += (dy*pitch+dx)*16 B).  An MMA tile is M=128 output pixels =
// 16 rows x 8 columns: 8 consecutive pixels are the 8 rows of a core matrix (16 B apart),
// the 16 image rows are the 16 core-matrix groups (stride-byte-offset = row pitch).
// N = Cout, K = 16 input channels per instruction, 9 taps x Cin/16 instructions per tile.
// Pooling layers use four "phase" tiles (py,px) over de-interleaved even/odd columns so
// that the 2x2 max-pool partners of a pooled pixel sit in the SAME TMEM lane (no shuffles).
// fp32-grade encoder features: operands are split x = hi + lo (two fp16), weights scaled by
// a power of two; three MMAs (hi*hi, hi*lo, lo*hi) accumulate into one fp32 TMEM tile.
//
// One kernel per layer and path, one launch per layer over up to cae_pass_cells (18944) cells.
// Split-precision encoder (precision 1 and 3 unless a separate encoder is loaded; precision 3 runs L3 as below):
//   L1  1->32 @64  conv1_tc_split_kernel         K = 9 im2col rows built by byte permutes, 3 MMAs per phase, writes hi/lo fp16
//   L2 32->64 @32  conv_tc_acc2_kernel<..,32,3>  TMA-fed double-buffered half-cell blocks, 3 taps per flush
//   L3 64->32 @16  conv_tc_acc_kernel<..,16,1>   row-pair tiles, N-stacked weights, register-staged, 1 tap per flush -> features
// Single-pass encoder (precision 2, a separately loaded encoder; precision 3's L3, its features from an exact fp32 L3):
//   L1  1->32 @64  conv1_fp32_planar_kernel      exact fp32 on the CUDA cores, writes hi fp16
//   L2, L3         conv_tc_kernel<EPI_POOL>      four pooling-phase tiles
// Decoder (every path):
//   L4 32->32 @8   conv_tc_kernel<EPI_PLAIN>     single pass, TMEM double-buffered
//   L5 32->64 @16  conv_tc_kernel<EPI_PLAIN,UPSIN> up-sampling folded into the staging
//   L6 64->32 @32  conv_tc_kernel<EPI_PHASE>     phase form at 16x16, N = 128
//   L7 32->1  @64  final_tapsum_kernel           one tap, (phase, neighbour) pairs on N, shifted tap sum + sigmoid + MSE/MAE
#include "common.cuh"
#include "tc_ptx.cuh"

#include <cuda.h>          // CUtensorMap (types only; the encoder is fetched through the runtime)
#include <cuda_fp16.h>

#include <cmath>

namespace {

constexpr int TCT = 256;   // 8 warps: warp&3 = TMEM lane quadrant, warp>>2 = column-slice parity
// EPI_PHASE: the layer runs at its INPUT's (pre-upsampling) resolution R with the four output phases
// (py,px) of the 2x nearest up-sampled grid as column groups: N = 4 * Cout, output is 2R x 2R
enum { EPI_POOL = 0, EPI_PLAIN = 2, EPI_PHASE = 4 };

using namespace tcptx;

// MMA issue loops of the accumulating encoder kernels (L2, L3): the whole warp runs the loop and one elected lane
// executes the tcgen05 instructions, so that descriptors stay in uniform registers (tc_ptx.cuh, elect_one):
// ~3 instead of ~20 instructions per MMA.  Measured (bench.py cae_layers, 486k cells): L2 52.4 -> 45.6 ms,
// L3 23.4 -> 22.1 ms (the form with lane 0 running the loop was removed).  The single-pass kernels (L1, L4-L7)
// measured 2-5 % SLOWER in the elected form and keep `if (lane == 0) { loop }`.
#define ISSUE_BEGIN if (elect_one()) {
#define ISSUE_END } __syncwarp();
// The accumulating kernels wait with the suspend-time hint (mbar_wait_sleep): a waiting warp sleeps in hardware
// instead of re-issuing try_wait + branch next to the issuing warp of its scheduler.  The plain loop for these
// kernels, and the hint for the single-pass kernels' waits, were measured and removed.

// Pooling layers: value of a pooled pixel from the max over its 2x2 window of the SIGN-FOLDED conv
// accumulators (weight columns carry sign(bn scale), see k_cae_tc_prepare).  bias -> ReLU -> BN is
// monotone in the conv output, so max-pool(f(c)) == f(max c) for a scale >= 0 and f(min c) otherwise;
// with the fold both are sign * max(sign * c): one XOR puts the sign back, f is evaluated once.
// invd = inv_scale * (mean relative deficit of the round-toward-zero accumulation): the truncations of
// the tensor core always shrink a partial sum, by an amount proportional to it on average, so the mean
// deficit of the whole sum is a fixed fraction of the sum and is added back here with the bias.
__device__ __forceinline__ float pooled_act(float folded_max, float inv_scale, float invd, float b, float s, float t) {
    const float m = __uint_as_float(__float_as_uint(folded_max) ^ (__float_as_uint(s) & 0x80000000u));
    // BatchNormalization as Keras evaluates it: x * inv + offset, a product and a sum rounded
    // separately (not one FMA) -- the oracle and the exact-fp32 path do the same
    return __fadd_rn(__fmul_rn(fmaxf(fmaf(m, inv_scale, fmaf(m, invd, b)), 0.f), s), t);
}

// Every tensor-core activation is stored here, as fp16 (hi, and the fp16 remainder lo for the split
// layers).  A value outside the fp16 range (|x| > 65504 after rounding, e.g. a BatchNorm with a large
// gamma over a small moving variance) or a NaN would reach the next layer as inf / NaN and turn MSE / MAE
// into inf or NaN -- or, masked by a later ReLU, into a wrong finite score -- without a word.  Such a
// store raises CIA_E_UNSUPPORTED on the handle's status word (cia_check_status).
__device__ __forceinline__ void split_store8(const float (&o)[8], __half* hi_dst, __half* lo_dst, bool& range_ok) {
    __align__(16) __half hh[8];
    __align__(16) __half ll[8];
    // |x| < 65520 rounds to a finite fp16 (65504 is the largest; 65520 ties to even, to inf); NaN fails the
    // comparison.  Tested on the fp32 values (one predicate-accumulating compare per element); the kernel
    // raises the status once, at its end, if any of its stores failed
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        hh[k] = __float2half_rn(o[k]);
        ll[k] = __float2half_rn(o[k] - __half2float(hh[k]));
        range_ok = range_ok && fabsf(o[k]) < 65520.f;
    }
    *reinterpret_cast<uint4*>(hi_dst) = *reinterpret_cast<const uint4*>(hh);
    if (lo_dst) *reinterpret_cast<uint4*>(lo_dst) = *reinterpret_cast<const uint4*>(ll);
}

// ---------------------------------------------------------------------------------------
// Layers 2..7 (Cin >= 32)
// ---------------------------------------------------------------------------------------
template <int CIN, int COUT, int R, int EPI, int NPASS>
struct Cfg {
    static constexpr bool POOL = EPI == EPI_POOL;
    static constexpr int NCH = CIN / 8;
    static constexpr int FILL_ROWS = POOL ? R + 2 : 18;              // rows actually staged
    // non-pool units: a 16-row band x UNIT_COLS columns (16 instead of 32 for the 64-channel 32x32
    // layer, so that two CTAs fit per SM and one's staging/epilogue overlaps the other's MMAs)
    static constexpr int UNIT_COLS = (R >= 32 && CIN >= 64) ? 16 : R;
    static constexpr int COL_BLOCKS = R / UNIT_COLS;
    static constexpr int ROW_UNITS = POOL ? 9 : UNIT_COLS + 2;        // 16-byte units per staged row
    static constexpr int ROW_B = ROW_UNITS * 16;
    static constexpr int PLANE_B = FILL_ROWS * ROW_B;
    static constexpr int CHUNK_B = (POOL ? 2 : 1) * PLANE_B;          // = LBO of A
    static constexpr int REGION_B = NCH * CHUNK_B;
    static constexpr int SBO_A = POOL ? 2 * ROW_B : ROW_B;
    static constexpr int TILES = POOL ? 4 : (UNIT_COLS >= 8 ? UNIT_COLS / 8 : 1);
    static constexpr int UNITS_PER_CELL = POOL ? (R >= 32 ? 2 : 1) : (R >= 32 ? 2 : 1) * COL_BLOCKS;
    static constexpr int TBUF_COLS = TILES * COUT;                    // one accumulator set
    // single-pass layers double-buffer the accumulators: the MMAs of unit u+1 run under the epilogue of u
    static constexpr int TMEM_COLS = pow2_cols((NPASS == 1 ? 2 : 1) * TBUF_COLS);
    static constexpr int W_B = 9 * NCH * COUT * 16;
    static constexpr int PARTS = NPASS > 1 ? 2 : 1;
    static constexpr int SMEM_B = PARTS * (REGION_B + W_B);
    // one CTA per SM, single pass, no pooling phases: a ninth warp issues the MMAs
    static constexpr bool DED_ISSUER = NPASS == 1 && !POOL && SMEM_B > 100 * 1024;
    static constexpr int THREADS = TCT + (DED_ISSUER ? 32 : 0);
};

// Stage the zero-padded input block of one unit into shared memory (pool layers: columns
// de-interleaved by parity).  Loads are issued in batches of BATCH independent 16-byte
// requests per thread before any store, so a unit pays ~one L2 latency instead of one per element.
template <class C, int R, int NPASS, int NT, int BATCH, bool UPSIN = false>
__device__ __forceinline__ void stage_block(const __half* __restrict__ in_hi, const __half* __restrict__ in_lo,
                                            unsigned char* a0, unsigned char* a1, int cell, int sub, int tid) {
    constexpr int COLS = C::POOL ? 18 : C::ROW_UNITS;
    constexpr int N_UNITS16 = C::NCH * C::FILL_ROWS * COLS;
    constexpr int ITERS = (N_UNITS16 + NT - 1) / NT;
#pragma unroll 1
    for (int i0 = 0; i0 < ITERS; i0 += BATCH) {
        uint4 vh[BATCH], vl[BATCH];
        uint32_t dst[BATCH];
#pragma unroll
        for (int j = 0; j < BATCH; ++j) {
            const int idx = tid + (i0 + j) * NT;
            vh[j] = make_uint4(0, 0, 0, 0); vl[j] = make_uint4(0, 0, 0, 0);
            dst[j] = 0xFFFFFFFFu;
            if (i0 + j < ITERS && idx < N_UNITS16) {
                const int c = idx / (C::FILL_ROWS * COLS);
                const int rem = idx - c * (C::FILL_ROWS * COLS);
                const int ry = rem / COLS, rc = rem - ry * COLS;
                int y, x;
                if (C::POOL) {
                    y = ry - 1; x = 16 * sub - 1 + rc;
                    dst[j] = (uint32_t)(((c * 2 + (rc & 1)) * C::FILL_ROWS + ry) * 9 + (rc >> 1)) * 16u;
                } else {
                    y = 16 * (sub / C::COL_BLOCKS) + ry - 1;
                    x = C::UNIT_COLS * (sub % C::COL_BLOCKS) + rc - 1;
                    dst[j] = (uint32_t)((c * C::FILL_ROWS + ry) * C::ROW_UNITS + rc) * 16u;
                }
                if (y >= 0 && y < R && x >= 0 && x < R) {
                    // UPSIN: the producer stored the low-res activation; nearest up-sampling happens here
                    constexpr int RS = UPSIN ? R / 2 : R;
                    const int ys = UPSIN ? (y >> 1) : y, xs = UPSIN ? (x >> 1) : x;
                    const size_t src = ((((size_t)cell * C::NCH + c) * RS + ys) * RS + xs);
                    vh[j] = __ldg(reinterpret_cast<const uint4*>(in_hi) + src);
                    if (NPASS > 1) vl[j] = __ldg(reinterpret_cast<const uint4*>(in_lo) + src);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < BATCH; ++j) {
            if (dst[j] != 0xFFFFFFFFu) {
                *reinterpret_cast<uint4*>(a0 + dst[j]) = vh[j];
                if (NPASS > 1) *reinterpret_cast<uint4*>(a1 + dst[j]) = vl[j];
            }
        }
    }
}

template <int CIN, int COUT, int R, int EPI, int NPASS, bool UPSIN>
__global__ void __launch_bounds__(Cfg<CIN, COUT, R, EPI, NPASS>::THREADS, (Cfg<CIN, COUT, R, EPI, NPASS>::SMEM_B > 100 * 1024) ? 1 : 2)
conv_tc_kernel(const __half* __restrict__ in_hi, const __half* __restrict__ in_lo,
               const uint4* __restrict__ w_hi, const uint4* __restrict__ w_lo, float inv_scale,
               const float* __restrict__ bias, const float* __restrict__ bn_s,
               const float* __restrict__ bn_t, __half* __restrict__ out_hi, __half* __restrict__ out_lo,
               float* __restrict__ feat, int n_cells, const int32_t* __restrict__ n_dev, int cell0,
               int chunk_cells,
               int32_t* __restrict__ status) {
    bool range_ok = true;             // every fp16 activation store of this thread was finite
    using C = Cfg<CIN, COUT, R, EPI, NPASS>;
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ __align__(8) uint64_t bar[2];
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    unsigned char* a_part[2] = {smem, smem + C::REGION_B};
    unsigned char* w_part[2] = {smem + C::PARTS * C::REGION_B, smem + C::PARTS * C::REGION_B + C::W_B};

    int n = dev_count(n_cells, n_dev) - cell0;
    if (n > chunk_cells) n = chunk_cells;
    if (n <= 0) return;                       // uniform: nothing allocated yet
    const int n_units = n * C::UNITS_PER_CELL;

    if (warp == 0) tmem_alloc(&tmem_base_s, C::TMEM_COLS);
    constexpr int NISS = C::DED_ISSUER ? 1 : C::TILES;           // issuing warps (TILES <= 4 <= warps)
    if (tid == 32) { mbar_init(&bar[0], NISS); mbar_init(&bar[1], NISS); fence_barrier_init(); }
    // weights: linear copy of the prepared UMMA images
    for (int i = tid; i < C::W_B / 16; i += TCT) {
        reinterpret_cast<uint4*>(w_part[0])[i] = __ldg(w_hi + i);
        if (NPASS > 1) reinterpret_cast<uint4*>(w_part[1])[i] = __ldg(w_lo + i);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    constexpr uint32_t IDESC = make_idesc(128, COUT);

    // ---- input staging as a software pipeline (single-pass layers): the 16-byte loads of unit
    // u+1 are issued into registers right after the MMAs of unit u and parked in shared memory
    // once the block has been consumed; element -> (chunk, row, col, smem offset) is unit-invariant.
    constexpr int S_COLS = C::POOL ? 18 : C::ROW_UNITS;
    constexpr int S_N = C::NCH * C::FILL_ROWS * S_COLS;
    constexpr int S_IT = (S_N + TCT - 1) / TCT;
    constexpr bool PIPE = NPASS == 1;
    uint32_t s_dst[S_IT], s_crc[S_IT];
    uint4 s_val[S_IT];
    if (PIPE) {
#pragma unroll
        for (int j = 0; j < S_IT; ++j) {
            const int idx = tid + j * TCT;
            s_dst[j] = 0xFFFFFFFFu; s_crc[j] = 0;
            if (idx < S_N && tid < TCT) {
                const int c = idx / (C::FILL_ROWS * S_COLS);
                const int rem = idx - c * (C::FILL_ROWS * S_COLS);
                const int ry = rem / S_COLS, rc = rem - ry * S_COLS;
                s_crc[j] = (uint32_t)((c << 16) | (ry << 8) | rc);
                s_dst[j] = C::POOL ? (uint32_t)(((c * 2 + (rc & 1)) * C::FILL_ROWS + ry) * 9 + (rc >> 1)) * 16u
                                   : (uint32_t)((c * C::FILL_ROWS + ry) * C::ROW_UNITS + rc) * 16u;
            }
        }
    }
    auto prefetch = [&](int unit) {
        const int cell = cell0 + unit / C::UNITS_PER_CELL;
        const int sub = unit % C::UNITS_PER_CELL;
        const int y0 = C::POOL ? -1 : 16 * (sub / C::COL_BLOCKS) - 1;
        const int x0 = C::POOL ? 16 * sub - 1 : C::UNIT_COLS * (sub % C::COL_BLOCKS) - 1;
        constexpr int RS = UPSIN ? R / 2 : R;
        const uint4* base = reinterpret_cast<const uint4*>(in_hi) + (size_t)cell * C::NCH * RS * RS;
#pragma unroll
        for (int j = 0; j < S_IT; ++j) {
            const int c = (int)(s_crc[j] >> 16), y = y0 + (int)((s_crc[j] >> 8) & 255u), x = x0 + (int)(s_crc[j] & 255u);
            s_val[j] = make_uint4(0, 0, 0, 0);
            if (s_dst[j] != 0xFFFFFFFFu && y >= 0 && y < R && x >= 0 && x < R) {
                const int ys = UPSIN ? (y >> 1) : y, xs = UPSIN ? (x >> 1) : x;
                s_val[j] = __ldg(base + ((size_t)c * RS + ys) * RS + xs);
            }
        }
    };
    auto park = [&]() {              // prefetched registers -> the shared-memory input block
#pragma unroll
        for (int j = 0; j < S_IT; ++j)
            if (s_dst[j] != 0xFFFFFFFFu) *reinterpret_cast<uint4*>(a_part[0] + s_dst[j]) = s_val[j];
    };
    // MMA issue: one lane of one warp PER TILE (a single thread sustains only ~one tcgen05.mma per
    // 60 cycles; the tiles' accumulators are independent); each commits to the buffer's barrier
    auto issue_mmas = [&](uint32_t tbuf) {
        if (C::DED_ISSUER) {
            // one extra warp issues for all tiles (an N = 128 MMA takes longer than the ~60 cycles a single
            // thread needs per issue; two issuing warps measured slower): the eight worker warps go straight
            // to their epilogue instead of two of them first spending the whole MMA time inside the issue loop
            if (lane == 0 && warp == TCT / 32) {
                tc_fence_after();
                const uint64_t ad0 = make_smem_desc(smem_u32(a_part[0]), C::CHUNK_B, C::SBO_A);
                const uint64_t bd0 = make_smem_desc(smem_u32(w_part[0]), COUT * 16, 128);
#pragma unroll
                for (int tap = 0; tap < 9; ++tap) {
                    const int dy = tap / 3, dx = tap % 3;
#pragma unroll
                    for (int s = 0; s < CIN / 16; ++s)
#pragma unroll
                        for (int t = 0; t < C::TILES; ++t) {
                            const uint64_t ad = ad0 + (uint64_t)((t * 8 * 16 + dx * 16 + dy * C::ROW_B + 2 * s * C::CHUNK_B) >> 4);
                            const uint64_t bd = bd0 + (uint64_t)(((tap * C::NCH + 2 * s) * COUT * 16) >> 4);
                            umma_f16(tmem_base + tbuf * C::TBUF_COLS + (uint32_t)(t * COUT), ad, bd, IDESC,
                                     (tap == 0 && s == 0) ? 0u : 1u);
                        }
                }
                umma_commit(&bar[tbuf]);
            }
            return;
        }
        if (lane == 0 && warp < NISS) {
            tc_fence_after();
            const int t = warp, py = t >> 1, px = t & 1;
            uint64_t dxo[3];          // tap-column offset in 16-byte units (pool: parity plane + half-column)
#pragma unroll
            for (int dx = 0; dx < 3; ++dx)
                dxo[dx] = C::POOL ? (uint64_t)((((px + dx) & 1) * C::PLANE_B + ((px + dx) >> 1) * 16) >> 4)
                                  : (uint64_t)dx;
            const uint32_t tile_off = C::POOL ? (uint32_t)(py * C::ROW_B) : (uint32_t)(t * 8 * 16);
            const uint32_t d_tmem = tmem_base + tbuf * C::TBUF_COLS + (uint32_t)(t * COUT);
#pragma unroll 1
            for (int pass = 0; pass < NPASS; ++pass) {
                const uint64_t ad0 = make_smem_desc(smem_u32(a_part[pass == 2 ? 1 : 0]) + tile_off, C::CHUNK_B, C::SBO_A);
                const uint64_t bd0 = make_smem_desc(smem_u32(w_part[pass == 1 ? 1 : 0]), COUT * 16, 128);
                const uint32_t acc0 = pass > 0 ? 1u : 0u;
#pragma unroll
                for (int tap = 0; tap < 9; ++tap) {
                    const int dy = tap / 3, dx = tap % 3;
#pragma unroll
                    for (int s = 0; s < CIN / 16; ++s) {
                        const uint64_t ad = ad0 + dxo[dx] + (uint64_t)((dy * C::ROW_B + 2 * s * C::CHUNK_B) >> 4);
                        const uint64_t bd = bd0 + (uint64_t)(((tap * C::NCH + 2 * s) * COUT * 16) >> 4);
                        umma_f16(d_tmem, ad, bd, IDESC, (tap == 0 && s == 0) ? acc0 : 1u);
                    }
                }
            }
            umma_commit(&bar[tbuf]);
        }
    };

    if (PIPE && (int)blockIdx.x < n_units) {
        // prologue: first unit staged and its MMAs in flight, second unit's loads in registers
        prefetch(blockIdx.x);
        park();
        fence_async_smem();
        __syncthreads();
        issue_mmas(0);
        if ((int)(blockIdx.x + gridDim.x) < n_units) prefetch(blockIdx.x + gridDim.x);
    }

    uint32_t it = 0;
    for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++it) {
        const int cell = cell0 + unit / C::UNITS_PER_CELL;
        const int sub = unit % C::UNITS_PER_CELL;   // POOL: pooled X half; else: 16-row band
        const uint32_t tbuf = PIPE ? (it & 1) : 0u;

        if (PIPE) {
            // MMAs of this unit done -> the input block is free: park the next unit, start its MMAs into
            // the other accumulator set, fetch the unit after that; all of it runs under this unit's epilogue.
            // The barrier also orders the previous epilogue's TMEM reads before the MMAs that overwrite them.
            mbar_wait(&bar[tbuf], (it >> 1) & 1);
            tc_fence_after();
            if (unit + (int)gridDim.x < n_units) {
                park();
                fence_async_smem();
                tc_fence_before();
                __syncthreads();
                issue_mmas(tbuf ^ 1);
                if (unit + 2 * (int)gridDim.x < n_units) prefetch(unit + 2 * gridDim.x);
            }
        } else {
            stage_block<C, R, NPASS, TCT, 8, UPSIN>(in_hi, in_lo, a_part[0], a_part[1], cell, sub, tid);
            fence_async_smem();
            __syncthreads();
            issue_mmas(0);
            mbar_wait(&bar[0], it & 1);
            tc_fence_after();
        }

        // ---- epilogue: TMEM -> registers -> bias/ReLU/BN (-> pool) -> global ----
        if (C::DED_ISSUER && warp >= TCT / 32) continue;     // the issuing warp has no epilogue share
        const int q = warp & 3, half_sel = warp >> 2;
        const int r = 32 * q + lane;                   // MMA row = TMEM lane
        const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * q) << 16) + tbuf * C::TBUF_COLS;
        if (EPI == EPI_POOL) {
            constexpr int RO = R / 2;
            const int Y = r >> 3, X = 8 * sub + (r & 7);
#pragma unroll 1
            for (int sl = half_sel; sl < COUT / 8; sl += 2) {
                const int c0 = sl * 8;
                uint32_t v[4][8];
#pragma unroll
                for (int ph = 0; ph < 4; ++ph) TMEM_LD8(lane_addr + (uint32_t)(ph * COUT + c0), v[ph]);
#pragma unroll
                for (int ph = 0; ph < 4; ++ph) TMEM_WAIT8(v[ph]);
                float o[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const float b = __ldg(bias + c0 + k), s = __ldg(bn_s + c0 + k), t = __ldg(bn_t + c0 + k);
                    o[k] = pooled_act(fmaxf(fmaxf(__uint_as_float(v[0][k]), __uint_as_float(v[1][k])),
                                            fmaxf(__uint_as_float(v[2][k]), __uint_as_float(v[3][k]))),
                                      inv_scale, 0.f, b, s, t);
                }
                if (Y < RO) {
                    const size_t off = ((((size_t)cell * (COUT / 8) + sl) * RO + Y) * RO + X) * 8;
                    split_store8(o, out_hi + off, out_lo ? out_lo + off : nullptr, range_ok);
                    if (feat) {
                        float4* f = reinterpret_cast<float4*>(feat + (size_t)cell * (RO * RO * COUT) +
                                                             (size_t)(Y * RO + X) * COUT + c0);
                        f[0] = make_float4(o[0], o[1], o[2], o[3]);
                        f[1] = make_float4(o[4], o[5], o[6], o[7]);
                    }
                }
            }
        } else if (EPI == EPI_PHASE) {
            // N = 4 phases x CREAL channels: a thread serves the channel slices of its warp-half for all
            // tiles and phases, so the bias / BN constants of a slice are fetched once
            constexpr int CREAL = COUT / 4, RO = 2 * R;
            const int y = 16 * (sub / C::COL_BLOCKS) + (r >> 3);
            const int xblk = C::UNIT_COLS * (sub % C::COL_BLOCKS);
#pragma unroll 1
            for (int cs = half_sel; cs < CREAL / 8; cs += 2) {
                float b8[8], s8[8], t8[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    b8[k] = __ldg(bias + cs * 8 + k); s8[k] = __ldg(bn_s + cs * 8 + k); t8[k] = __ldg(bn_t + cs * 8 + k);
                }
#pragma unroll 1
                for (int t = 0; t < C::TILES; ++t) {
                    const int x = xblk + 8 * t + (r & 7);
                    uint32_t v[4][8];
#pragma unroll
                    for (int ph = 0; ph < 4; ++ph) TMEM_LD8(lane_addr + (uint32_t)(t * COUT + ph * CREAL + cs * 8), v[ph]);
#pragma unroll
                    for (int ph = 0; ph < 4; ++ph) TMEM_WAIT8(v[ph]);
                    if (y < R) {
#pragma unroll
                        for (int ph = 0; ph < 4; ++ph) {
                            float o[8];
#pragma unroll
                            for (int k = 0; k < 8; ++k) {
                                const float a = fmaxf(fmaf(__uint_as_float(v[ph][k]), inv_scale, b8[k]), 0.f);
                                o[k] = __fadd_rn(__fmul_rn(a, s8[k]), t8[k]);
                            }
                            const size_t off = ((((size_t)cell * (CREAL / 8) + cs) * RO + 2 * y + (ph >> 1)) * RO +
                                                2 * x + (ph & 1)) * 8;
                            split_store8(o, out_hi + off, nullptr, range_ok);
                        }
                    }
                }
            }
        } else {
            const int y = 16 * (sub / C::COL_BLOCKS) + (r >> 3);
            const int xblk = C::UNIT_COLS * (sub % C::COL_BLOCKS);
            constexpr int SL = COUT / 8;
#pragma unroll 1
            for (int p = half_sel; p < C::TILES * SL; p += 2) {
                const int t = p / SL, sl = p - t * SL;
                const int c0 = sl * 8;
                const int x = xblk + 8 * t + (r & 7);
                uint32_t v[8];
                TMEM_LD8(lane_addr + (uint32_t)(t * COUT + c0), v);
                TMEM_WAIT8(v);
                float o[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    float a = fmaf(__uint_as_float(v[k]), inv_scale, __ldg(bias + c0 + k));
                    a = fmaxf(a, 0.f);
                    o[k] = __fadd_rn(__fmul_rn(a, __ldg(bn_s + c0 + k)), __ldg(bn_t + c0 + k));
                }
                if (y < R) {
                    const size_t off = ((((size_t)cell * (COUT / 8) + sl) * R + y) * R + x) * 8;
                    split_store8(o, out_hi + off, nullptr, range_ok);
                }
            }
        }
        // single-pass layers need no barrier here (the one before the next MMA issue orders the TMEM reads)
        if (!PIPE) {
            tc_fence_before();
            __syncthreads();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, C::TMEM_COLS);
    if (!range_ok) raise_status(status, CIA_E_UNSUPPORTED);
}

// ---------------------------------------------------------------------------------------
// Split-precision pooling layers with ACCURATE accumulation (encoder layers 2 and 3).
//
// tcgen05.mma adds every k-step into its fp32 TMEM accumulator with round-toward-zero
// (profiles/umma_rounding_test.cu): a K = 288..576 chain picks up a ~1e-6 relative bias, too
// much for the one-class SVM downstream.  Here a TMEM accumulator only ever holds ONE filter
// tap: the cross terms (hi*lo, lo*hi; 2^-11 of the magnitude) are issued first into the fresh
// accumulator, the hi*hi k-steps last, so only Cin/16 truncations happen at a third of the
// final magnitude.  The nine per-tap partial sums are added in fp32 registers (round to
// nearest) by the epilogue warps while the MMA warp already fills the other TMEM stage.
//   warps 0..15: stage input block, per tap tcgen05.ld the partial and add, final epilogue
//   warps 16-19: one lane each issues the MMAs of one pooling-phase tile (a single thread
//                cannot issue faster than ~60 cycles per tcgen05.mma)
// ---------------------------------------------------------------------------------------
constexpr int ACC_EPI_WARPS = 16;
constexpr int ACC_MMA_WARPS = 4;
constexpr int ACC_THREADS = (ACC_EPI_WARPS + ACC_MMA_WARPS) * 32;

// Geometry of the accurate-accumulation kernel: ONE unit = one whole cell.  The zero-padded
// (R+2) x (R+2) input is staged once, column-parity de-interleaved.
template <int CIN, int COUT, int R>
struct AccCfg {
    static constexpr int NCH = CIN / 8;
    static constexpr int FILL_ROWS = R + 2;
    static constexpr int COLS = R + 2;                    // staged columns
    static constexpr int ROW_UNITS = COLS / 2;            // 16-byte units per parity-plane row
    static constexpr int ROW_B = ROW_UNITS * 16;
    static constexpr int PLANE_B = FILL_ROWS * ROW_B;
    static constexpr int CHUNK_B = 2 * PLANE_B;           // = LBO of A
    static constexpr int REGION_B = NCH * CHUNK_B;
    static constexpr int W_B = 9 * NCH * COUT * 16;
    static constexpr int SMEM_B = 2 * (REGION_B + W_B);
};

template <class A, int R, int NT, int BATCH>
__device__ __forceinline__ void stage_pool_cell(const __half* __restrict__ in_hi, const __half* __restrict__ in_lo,
                                                unsigned char* a0, unsigned char* a1, int cell, int tid) {
    constexpr int N_UNITS16 = A::NCH * A::FILL_ROWS * A::COLS;
    constexpr int ITERS = (N_UNITS16 + NT - 1) / NT;
#pragma unroll 1
    for (int i0 = 0; i0 < ITERS; i0 += BATCH) {
        uint4 vh[BATCH], vl[BATCH];
        uint32_t dst[BATCH];
#pragma unroll
        for (int j = 0; j < BATCH; ++j) {
            const int idx = tid + (i0 + j) * NT;
            vh[j] = make_uint4(0, 0, 0, 0); vl[j] = make_uint4(0, 0, 0, 0);
            dst[j] = 0xFFFFFFFFu;
            if (i0 + j < ITERS && idx < N_UNITS16) {
                const int c = idx / (A::FILL_ROWS * A::COLS);
                const int rem = idx - c * (A::FILL_ROWS * A::COLS);
                const int ry = rem / A::COLS, rc = rem - ry * A::COLS;
                const int y = ry - 1, x = rc - 1;
                dst[j] = (uint32_t)(((c * 2 + (rc & 1)) * A::FILL_ROWS + ry) * A::ROW_UNITS + (rc >> 1)) * 16u;
                if (y >= 0 && y < R && x >= 0 && x < R) {
                    const size_t src = ((((size_t)cell * A::NCH + c) * R + y) * R + x);
                    vh[j] = __ldg(reinterpret_cast<const uint4*>(in_hi) + src);
                    vl[j] = __ldg(reinterpret_cast<const uint4*>(in_lo) + src);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < BATCH; ++j) {
            if (dst[j] != 0xFFFFFFFFu) {
                *reinterpret_cast<uint4*>(a0 + dst[j]) = vh[j];
                *reinterpret_cast<uint4*>(a1 + dst[j]) = vl[j];
            }
        }
    }
}

#ifdef CIA_ACC_TIMING
__device__ unsigned long long g_acc_dbg[16];
#define DBG_T(var) const long long var = clock64()
#define DBG_ADD(acc, a, b) acc += (b) - (a)
#else
#define DBG_T(var)
#define DBG_ADD(acc, a, b)
#endif

template <int CIN, int COUT, int R, int G>
__global__ void __launch_bounds__(ACC_THREADS, 1)
conv_tc_acc_kernel(const __half* __restrict__ in_hi, const __half* __restrict__ in_lo,
                   const uint4* __restrict__ w_hi, const uint4* __restrict__ w_lo, float inv_scale, float invd,
                   const float* __restrict__ bias, const float* __restrict__ bn_s,
                   const float* __restrict__ bn_t, __half* __restrict__ out_hi, __half* __restrict__ out_lo,
                   float* __restrict__ feat, int n_cells, const int32_t* __restrict__ n_dev, int cell0,
                   int chunk_cells,
                   int32_t* __restrict__ status) {
    bool range_ok = true;             // every fp16 activation store of this thread was finite
    using C = AccCfg<CIN, COUT, R>;
    static_assert(CIN == 64 && COUT == 32 && R == 16, "the L3 geometry: row-pair tiles, N-stacked weights");
    // The pooled output is only 8 x 8, so a 16-row-group tile takes BOTH row phases (row group g = conv
    // row g, stride one staged row) and there are two tiles (px = 0, 1) instead of four half-empty ones;
    // the 2x2 pool then pairs lanes r and r^8 with one shuffle per value.
    constexpr int NT = 2;                        // accumulator tiles per stage = issuing warps
    // N-stacked weights (N <= 32, where an MMA costs its 4 KB A-operand read whatever N is): the B operand
    // of the hi activations is the weight image's hi and lo rows stacked along N, so hi*hi and hi*lo come out
    // of ONE N = 2*COUT instruction in adjacent column groups and lo*hi is added to the cross group by a
    // second one -- two A reads per k-step instead of three.  The cross group is flushed with the hi*hi
    // group (its truncations are 2^-11 of the sum's).
    constexpr int TILE_COLS = 2 * COUT;
    constexpr int STAGE_COLS = NT * TILE_COLS;
    constexpr int TMEM_COLS = pow2_cols(2 * STAGE_COLS);
    constexpr int CW = COUT / 4;                 // columns per epilogue warp
    constexpr int NGRP = (9 + G - 1) / G;        // TMEM flushes per pooled tile (G filter taps each)
    constexpr int EPT = ACC_EPI_WARPS * 32;
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ __align__(8) uint64_t full_bar[2], empty_bar[2], ready_bar;
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    unsigned char* a_part[2] = {smem, smem + C::REGION_B};
    unsigned char* w_part[2] = {smem + 2 * C::REGION_B, smem + 2 * C::REGION_B + C::W_B};

    int n = dev_count(n_cells, n_dev) - cell0;
    if (n > chunk_cells) n = chunk_cells;
    if (n <= 0) return;
    const int n_units = n;                       // one unit = one cell

    if (warp == 0) tmem_alloc(&tmem_base_s, TMEM_COLS);
    if (tid == 32) {
        mbar_init(&full_bar[0], NT); mbar_init(&full_bar[1], NT);
        mbar_init(&empty_bar[0], ACC_EPI_WARPS); mbar_init(&empty_bar[1], ACC_EPI_WARPS);
        mbar_init(&ready_bar, ACC_EPI_WARPS);
        fence_barrier_init();
    }
    // stacked image [(tap, chunk)][hi rows 0..COUT-1 | lo rows][8 halves] over both weight regions
    for (int i = tid; i < 2 * C::W_B / 16; i += ACC_THREADS) {
        const int tc = i / (2 * COUT), row = i - tc * (2 * COUT);
        reinterpret_cast<uint4*>(w_part[0])[i] = row < COUT ? __ldg(w_hi + tc * COUT + row) : __ldg(w_lo + tc * COUT + row - COUT);
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    constexpr uint32_t IDESC = make_idesc(128, COUT);

    if (warp >= ACC_EPI_WARPS) {
        // ================= MMA issuers: one warp per phase tile =================
        // A single thread sustains only one tcgen05.mma per ~60 cycles (elect loop, R2UR moves,
        // dependent uniform-register adds), more than the 45-48 cycles an M128 x N<=64 MMA takes;
        // issuing warps, each owning the accumulator tile of one pooling phase, keep the tensor pipe
        // fed.  Each commits to the stage's full barrier (count NT).
        if (warp - ACC_EPI_WARPS < NT) {
            const int t = warp - ACC_EPI_WARPS, px = t & 1;
            const uint64_t a_hi0 = make_smem_desc(smem_u32(a_part[0]), C::CHUNK_B, C::ROW_B);
            const uint64_t a_lo0 = make_smem_desc(smem_u32(a_part[1]), C::CHUNK_B, C::ROW_B);
            const uint64_t b_hi0 = make_smem_desc(smem_u32(w_part[0]), TILE_COLS * 16, 128);   // the stacked operand
            constexpr uint32_t IDESC2 = make_idesc(128, TILE_COLS);
            uint64_t dxo[3];                   // (parity plane, half-column shift) of tap column dx, in 16-byte units
#pragma unroll
            for (int dx = 0; dx < 3; ++dx) dxo[dx] = (uint64_t)((((px + dx) & 1) * C::PLANE_B + ((px + dx) >> 1) * 16) >> 4);
            uint32_t it = 0, uphase = 0;
#ifdef CIA_ACC_TIMING
            long long m_ready = 0, m_empty = 0, m_issue = 0;
#endif
            for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
                DBG_T(m0);
                mbar_wait_sleep(&ready_bar, uphase);
                DBG_T(m1);
                DBG_ADD(m_ready, m0, m1);
                uphase ^= 1;
                tc_fence_after();
#pragma unroll
                for (int grp = 0; grp < NGRP; ++grp) {
                    const uint32_t st = it & 1;
                    DBG_T(m2);
                    mbar_wait_sleep(&empty_bar[st], ((it >> 1) & 1) ^ 1);
                    DBG_T(m3);
                    DBG_ADD(m_empty, m2, m3);
                    tc_fence_after();
                    const uint32_t d = tmem_base + st * STAGE_COLS + (uint32_t)(t * TILE_COLS);
                    ISSUE_BEGIN
                    // hi x [hi | lo] (N = 2*COUT, zero-initialising both column groups), then lo x hi into the cross group
#pragma unroll
                    for (int pass = 0; pass < 2; ++pass) {
#pragma unroll
                        for (int tg = 0; tg < G; ++tg) {
                            const int tap = grp * G + tg;
                            if (tap < 9) {
                                const int dy = tap / 3, dx = tap % 3;
                                const uint64_t a0 = (pass == 1 ? a_lo0 : a_hi0) + dxo[dx];
#pragma unroll
                                for (int s = 0; s < CIN / 16; ++s) {
                                    const uint64_t ad = a0 + (uint64_t)((dy * C::ROW_UNITS * 16 + 2 * s * C::CHUNK_B) >> 4);
                                    const uint64_t bd = b_hi0 + (uint64_t)(((tap * C::NCH + 2 * s) * TILE_COLS * 16) >> 4);
                                    if (pass == 0) umma_f16(d, ad, bd, IDESC2, (tg == 0 && s == 0) ? 0u : 1u);
                                    else umma_f16(d + COUT, ad, bd, IDESC, 1u);
                                }
                            }
                        }
                    }
                    umma_commit(&full_bar[st]);
                    ISSUE_END
                    DBG_T(m4);
                    DBG_ADD(m_issue, m3, m4);
                    ++it;
                }
            }
#ifdef CIA_ACC_TIMING
            if (warp == ACC_EPI_WARPS && lane == 0) {
                atomicAdd(&g_acc_dbg[8], (unsigned long long)m_ready);
                atomicAdd(&g_acc_dbg[9], (unsigned long long)m_empty);
                atomicAdd(&g_acc_dbg[10], (unsigned long long)m_issue);
            }
#endif
        }
    } else {
        // ================= loaders / accumulating epilogue =================
        const int q = warp & 3, cq = warp >> 2;
        const int r = 32 * q + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(cq * CW);
        uint32_t it = 0;
#ifdef CIA_ACC_TIMING
        long long e_stage = 0, e_full = 0, e_ld = 0, e_add = 0, e_final = 0, e_units = 0;
#endif
        for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
            const int cell = cell0 + unit;
            DBG_T(e0);
            // stage the zero-padded, column-parity de-interleaved input block (hi and lo); only the CTA's
            // first cell is staged here, the others right after the previous cell's last flush (below)
            if (unit == (int)blockIdx.x) {
                stage_pool_cell<C, R, EPT, 6>(in_hi, in_lo, a_part[0], a_part[1], cell, tid);
                fence_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&ready_bar);
            }
            DBG_T(e1);
            DBG_ADD(e_stage, e0, e1);
#ifdef CIA_ACC_TIMING
            ++e_units;
#endif

            float acc[NT][CW];
#pragma unroll
            for (int ph = 0; ph < NT; ++ph)
#pragma unroll
                for (int k = 0; k < CW; ++k) acc[ph][k] = 0.f;
#pragma unroll 1
            for (int grp = 0; grp < NGRP; ++grp) {
                const uint32_t st = it & 1;
                DBG_T(e2);
                mbar_wait_sleep(&full_bar[st], (it >> 1) & 1);
                DBG_T(e3);
                DBG_ADD(e_full, e2, e3);
                tc_fence_after();
#pragma unroll
                for (int hp = 0; hp < NT / 2; ++hp) {
                    uint32_t v[2][CW / 8][8];
                    uint32_t vc[2][CW / 8][8];     // cross-term group of the stacked tiles
#pragma unroll
                    for (int p2 = 0; p2 < 2; ++p2)
#pragma unroll
                        for (int k8 = 0; k8 < CW / 8; ++k8) {
                            TMEM_LD8(lane_addr + st * STAGE_COLS + (uint32_t)((2 * hp + p2) * TILE_COLS + k8 * 8), v[p2][k8]);
                            TMEM_LD8(lane_addr + st * STAGE_COLS + (uint32_t)((2 * hp + p2) * TILE_COLS + COUT + k8 * 8), vc[p2][k8]);
                        }
#pragma unroll
                    for (int p2 = 0; p2 < 2; ++p2)
#pragma unroll
                        for (int k8 = 0; k8 < CW / 8; ++k8) {
                            TMEM_WAIT8(v[p2][k8]);
                            TMEM_WAIT8(vc[p2][k8]);
                        }
                    if (hp == NT / 2 - 1) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&empty_bar[st]);
                        DBG_T(e4);
                        DBG_ADD(e_ld, e3, e4);
                    }
#pragma unroll
                    for (int p2 = 0; p2 < 2; ++p2)
#pragma unroll
                        for (int k8 = 0; k8 < CW / 8; ++k8)
#pragma unroll
                            for (int k = 0; k < 8; k += 2) {  // packed fp32x2 add (FADD2), round to nearest
                                fadd2(acc[2 * hp + p2][k8 * 8 + k], acc[2 * hp + p2][k8 * 8 + k + 1],
                                      vc[p2][k8][k], vc[p2][k8][k + 1]);
                                fadd2(acc[2 * hp + p2][k8 * 8 + k], acc[2 * hp + p2][k8 * 8 + k + 1],
                                      v[p2][k8][k], v[p2][k8][k + 1]);
                            }
                }
                DBG_T(e5);
                DBG_ADD(e_add, e3, e5);
                ++it;
            }
            DBG_T(e6);
            // the cell's last MMAs have completed (its last full barrier): the input block is free, so the
            // next cell is staged NOW and its MMAs run under the final epilogue below
            if (unit + (int)gridDim.x < n_units) {
                stage_pool_cell<C, R, EPT, 6>(in_hi, in_lo, a_part[0], a_part[1], cell + (int)gridDim.x, tid);
                fence_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&ready_bar);
            }
            // final epilogue from registers: bias -> ReLU -> BN -> 2x2 max -> hi/lo fp16 (+ fp32 tap)
            constexpr int RO = R / 2;
            const int Y = r >> 4, X = r & 7;
#pragma unroll
            for (int k8 = 0; k8 < CW / 8; ++k8) {
                const int c0 = cq * CW + k8 * 8;
                float o[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const float b = __ldg(bias + c0 + k), s = __ldg(bn_s + c0 + k), t = __ldg(bn_t + c0 + k);
                    float m = acc[0][k8 * 8 + k];
#pragma unroll
                    for (int ph = 1; ph < NT; ++ph) m = fmaxf(m, acc[ph][k8 * 8 + k]);
                    m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 8));   // conv rows 2Y, 2Y+1
                    o[k] = pooled_act(m, inv_scale, invd, b, s, t);
                }
                if (r & 8) continue;      // the even conv row's lane stores the pooled pixel
                const size_t off = ((((size_t)cell * (COUT / 8) + c0 / 8) * RO + Y) * RO + X) * 8;
                split_store8(o, out_hi + off, out_lo ? out_lo + off : nullptr, range_ok);
                if (feat) {
                    float4* f = reinterpret_cast<float4*>(feat + (size_t)cell * (RO * RO * COUT) +
                                                         (size_t)(Y * RO + X) * COUT + c0);
                    f[0] = make_float4(o[0], o[1], o[2], o[3]);
                    f[1] = make_float4(o[4], o[5], o[6], o[7]);
                }
            }
            DBG_T(e7);
            DBG_ADD(e_final, e6, e7);
        }
#ifdef CIA_ACC_TIMING
        if (tid == 0) {
            atomicAdd(&g_acc_dbg[0], (unsigned long long)e_stage);
            atomicAdd(&g_acc_dbg[1], (unsigned long long)e_full);
            atomicAdd(&g_acc_dbg[2], (unsigned long long)e_ld);
            atomicAdd(&g_acc_dbg[3], (unsigned long long)e_add);
            atomicAdd(&g_acc_dbg[4], (unsigned long long)e_final);
            atomicAdd(&g_acc_dbg[5], (unsigned long long)e_units);
        }
#endif
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, TMEM_COLS);
    if (!range_ok) raise_status(status, CIA_E_UNSUPPORTED);
}

// ---------------------------------------------------------------------------------------
// Accurate accumulation for the R = 32 pooling layer (L2): TMA-fed, double-buffered blocks.
// In-kernel clocks on a whole-cell form of the kernel above at R = 32 (since removed;
// profiles/r1_acc_phase_cycles.txt) showed its phases running back to back per cell: staging 7.7k cycles -> MMAs 22k (issue-bound at ~51
// cycles per M128xN64xK16 instruction) -> final epilogue 3.7k, with per-tap flushes keeping
// the epilogue warps busier (27k) than the tensor pipe.  Here one unit = one pooled X-half
// (16 input columns + halo, 2 x 39 KB hi/lo) and the two halves of a cell alternate between
// two shared-memory buffers.  A block is four TMA boxes (hi/lo x column parity): the tensor
// map walks x with element stride 2, which de-interleaves the columns by parity on the fly,
// and out-of-bounds coordinates (x = -1 / 32, y = -1 / 32) zero-fill the halo.  The copy of
// half-unit k+2 is issued by one thread the moment the last MMAs of half-unit k (same buffer)
// have completed, i.e. a whole half-unit ahead of its use; no warp stages anything.
// ---------------------------------------------------------------------------------------
template <int CIN, int COUT, int R_>
struct Acc2Cfg {
    static constexpr int R = R_;
    static constexpr int NCH = CIN / 8;
    static constexpr int FILL_ROWS = R + 2;
    static constexpr int HALVES = R / 16;                 // 16-column blocks per cell = shared-memory buffers
    static constexpr int BOX_X = 16 + 2;                  // columns a box spans (every second one is read)
    static constexpr int ROW_UNITS = BOX_X / 2;           // 16-byte units per parity-plane row
    static constexpr int ROW_B = ROW_UNITS * 16;
    static constexpr int PLANE_B = FILL_ROWS * ROW_B;     // one (parity, chunk) plane = LBO of A
    static constexpr int PAR_B = NCH * PLANE_B;           // one TMA box: all chunks of one column parity
    static constexpr int REGION_B = 2 * PAR_B;            // hi or lo part of a block
    static constexpr int SBO_A = 2 * ROW_B;
    static constexpr int BUF_B = 2 * REGION_B;            // hi + lo of one block
    static constexpr int W_B = 9 * NCH * COUT * 16;
    static constexpr int SMEM_B = HALVES * BUF_B + 2 * W_B;
    static_assert(PAR_B % 128 == 0, "TMA destinations must be 128-byte aligned");
};

__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3,
                                            int c4, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2,%3,%4,%5,%6}], [%7];"
        ::"r"(dst), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(smem_u32(bar)) : "memory");
}
// one half block = 4 boxes over the [cell][chunk][y][x][8] fp16 activations (tensor-map dims 8, x, y, chunk, cell)
template <class A>
__device__ __forceinline__ void tma_load_half_block(const CUtensorMap* tm_hi, const CUtensorMap* tm_lo, uint32_t buf,
                                                    int cell_rel, int half, uint64_t* bar) {
    mbar_expect_tx(bar, A::BUF_B);
#pragma unroll
    for (int par = 0; par < 2; ++par) {
        const int x0 = half * 16 - 1 + par;
        tma_load_5d(buf + par * A::PAR_B, tm_hi, 0, x0, -1, 0, cell_rel, bar);
        tma_load_5d(buf + A::REGION_B + par * A::PAR_B, tm_lo, 0, x0, -1, 0, cell_rel, bar);
    }
}

template <int CIN, int COUT, int R, int G>
__global__ void __launch_bounds__(ACC_THREADS, 1)
conv_tc_acc2_kernel(const __grid_constant__ CUtensorMap tm_hi, const __grid_constant__ CUtensorMap tm_lo,
                    const uint4* __restrict__ w_hi, const uint4* __restrict__ w_lo, float inv_scale, float invd,
                    const float* __restrict__ bias, const float* __restrict__ bn_s,
                    const float* __restrict__ bn_t, __half* __restrict__ out_hi, __half* __restrict__ out_lo,
                    float* __restrict__ feat, int n_cells, const int32_t* __restrict__ n_dev, int cell0,
                    int chunk_cells,
                    int32_t* __restrict__ status) {
    bool range_ok = true;             // every fp16 activation store of this thread was finite
    using C = Acc2Cfg<CIN, COUT, R>;
    static_assert(CIN == 32 && COUT == 64 && R == 32, "the L2 geometry: two half-cell blocks, four pooling-phase tiles");
    constexpr int NT = 4;                        // accumulator tiles per stage = issuing warps
    constexpr int STAGE_COLS = NT * COUT;
    constexpr int TMEM_COLS = pow2_cols(2 * STAGE_COLS);
    constexpr int CW = COUT / 4;                 // columns per epilogue warp
    constexpr int NGRP = (9 + G - 1) / G;        // TMEM flushes per pooled tile (G filter taps each)
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ __align__(8) uint64_t full_bar[2], empty_bar[2], ready_bar[2];
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    unsigned char* w_part[2] = {smem + C::HALVES * C::BUF_B, smem + C::HALVES * C::BUF_B + C::W_B};

    int n = dev_count(n_cells, n_dev) - cell0;
    if (n > chunk_cells) n = chunk_cells;
    if (n <= 0) return;
    const int n_units = n;                       // CTA-level unit = one cell = two half blocks

    if (warp == 0) tmem_alloc(&tmem_base_s, TMEM_COLS);
    if (tid == 32) {
        mbar_init(&full_bar[0], NT); mbar_init(&full_bar[1], NT);
        mbar_init(&empty_bar[0], ACC_EPI_WARPS); mbar_init(&empty_bar[1], ACC_EPI_WARPS);
        mbar_init(&ready_bar[0], 1); mbar_init(&ready_bar[1], 1);
        fence_barrier_init();
    }
    for (int i = tid; i < C::W_B / 16; i += ACC_THREADS) {
        reinterpret_cast<uint4*>(w_part[0])[i] = __ldg(w_hi + i);
        reinterpret_cast<uint4*>(w_part[1])[i] = __ldg(w_lo + i);
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    const uint32_t sbase = smem_u32(smem);
    constexpr uint32_t IDESC = make_idesc(128, COUT);

    if (warp >= ACC_EPI_WARPS) {
        // ================= MMA issuers: one warp per phase tile =================
        if (warp - ACC_EPI_WARPS < NT) {
            const int t = warp - ACC_EPI_WARPS, py = t >> 1, px = t & 1;
            const uint64_t b_hi0 = make_smem_desc(smem_u32(w_part[0]), COUT * 16, 128);
            const uint64_t b_lo0 = make_smem_desc(smem_u32(w_part[1]), COUT * 16, 128);
            uint64_t dxo[3];                   // (parity plane, half-column shift) of tap column dx, in 16-byte units
#pragma unroll
            for (int dx = 0; dx < 3; ++dx) dxo[dx] = (uint64_t)((((px + dx) & 1) * C::PAR_B + ((px + dx) >> 1) * 16) >> 4);
            uint32_t it = 0, cphase = 0;
#ifdef CIA_ACC_TIMING
            long long m_ready = 0, m_empty = 0, m_issue = 0;
#endif
            for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
#pragma unroll
                for (int half = 0; half < C::HALVES; ++half) {
                    const uint32_t abase = sbase + half * C::BUF_B + py * C::ROW_B;
                    const uint64_t a_hi0 = make_smem_desc(abase, C::PLANE_B, C::SBO_A);
                    const uint64_t a_lo0 = make_smem_desc(abase + C::REGION_B, C::PLANE_B, C::SBO_A);
                    DBG_T(m0);
                    mbar_wait_sleep(&ready_bar[half], cphase);
                    DBG_T(m1);
                    DBG_ADD(m_ready, m0, m1);
                    tc_fence_after();
#pragma unroll
                    for (int grp = 0; grp < NGRP; ++grp) {
                        const uint32_t st = it & 1;
                        DBG_T(m2);
                        mbar_wait_sleep(&empty_bar[st], ((it >> 1) & 1) ^ 1);
                        DBG_T(m3);
                        DBG_ADD(m_empty, m2, m3);
                        tc_fence_after();
                        const uint32_t d = tmem_base + st * STAGE_COLS + (uint32_t)(t * COUT);
                        ISSUE_BEGIN
                        // within a flush group: all cross terms (hi*lo, lo*hi; tiny) first, hi*hi last
#pragma unroll
                        for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
                            for (int tg = 0; tg < G; ++tg) {
                                const int tap = grp * G + tg;
                                if (tap < 9) {
                                    const int dy = tap / 3, dx = tap % 3;
                                    const uint64_t a0 = (pass == 1 ? a_lo0 : a_hi0) + dxo[dx];
                                    const uint64_t b0 = pass == 0 ? b_lo0 : b_hi0;
#pragma unroll
                                    for (int s = 0; s < CIN / 16; ++s) {
                                        const uint64_t ad = a0 + (uint64_t)((dy * C::ROW_B + 2 * s * C::PLANE_B) >> 4);
                                        const uint64_t bd = b0 + (uint64_t)(((tap * C::NCH + 2 * s) * COUT * 16) >> 4);
                                        umma_f16(d, ad, bd, IDESC, (pass == 0 && tg == 0 && s == 0) ? 0u : 1u);
                                    }
                                }
                            }
                        }
                        umma_commit(&full_bar[st]);
                        ISSUE_END
                        DBG_T(m4);
                        DBG_ADD(m_issue, m3, m4);
                        ++it;
                    }
                }
                cphase ^= 1;
            }
#ifdef CIA_ACC_TIMING
            if (warp == ACC_EPI_WARPS && lane == 0) {
                atomicAdd(&g_acc_dbg[8], (unsigned long long)m_ready);
                atomicAdd(&g_acc_dbg[9], (unsigned long long)m_empty);
                atomicAdd(&g_acc_dbg[10], (unsigned long long)m_issue);
            }
#endif
        }
    } else {
        // ================= copy issuers / accumulating epilogue =================
        const int q = warp & 3, cq = warp >> 2;
        const int r = 32 * q + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(cq * CW);
        uint32_t it = 0;
#ifdef CIA_ACC_TIMING
        long long e_stage = 0, e_full = 0, e_ld = 0, e_add = 0, e_final = 0, e_units = 0;
#endif
        if (tid == 0 && (int)blockIdx.x < n_units) {          // prologue: all blocks of the first cell
            for (int hb = 0; hb < C::HALVES; ++hb)
                tma_load_half_block<C>(&tm_hi, &tm_lo, sbase + hb * C::BUF_B, blockIdx.x, hb, &ready_bar[hb]);
        }
        for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
            const int cell = cell0 + unit;
#ifdef CIA_ACC_TIMING
            ++e_units;
#endif
#pragma unroll 1
            for (int sub = 0; sub < C::HALVES; ++sub) {
                float acc[NT][CW];
#pragma unroll
                for (int ph = 0; ph < NT; ++ph)
#pragma unroll
                    for (int k = 0; k < CW; ++k) acc[ph][k] = 0.f;
#pragma unroll 1
                for (int grp = 0; grp < NGRP; ++grp) {
                    const uint32_t st = it & 1;
                    DBG_T(e2);
                    mbar_wait_sleep(&full_bar[st], (it >> 1) & 1);
                    DBG_T(e3);
                    DBG_ADD(e_full, e2, e3);
                    tc_fence_after();
                    // the last MMAs reading this buffer are done: refill it with the same half of the next cell
                    if (grp == NGRP - 1 && tid == 0 && unit + (int)gridDim.x < n_units)
                        tma_load_half_block<C>(&tm_hi, &tm_lo, sbase + sub * C::BUF_B, unit + (int)gridDim.x, sub,
                                               &ready_bar[sub]);
                    // two phases at a time keeps the live registers under the 102-per-thread budget
#pragma unroll
                    for (int hp = 0; hp < NT / 2; ++hp) {
                        uint32_t v[2][CW / 8][8];
#pragma unroll
                        for (int p2 = 0; p2 < 2; ++p2)
#pragma unroll
                            for (int k8 = 0; k8 < CW / 8; ++k8)
                                TMEM_LD8(lane_addr + st * STAGE_COLS + (uint32_t)((2 * hp + p2) * COUT + k8 * 8), v[p2][k8]);
#pragma unroll
                        for (int p2 = 0; p2 < 2; ++p2)
#pragma unroll
                            for (int k8 = 0; k8 < CW / 8; ++k8) TMEM_WAIT8(v[p2][k8]);
                        if (hp == NT / 2 - 1) {
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(&empty_bar[st]);
                            DBG_T(e4);
                            DBG_ADD(e_ld, e3, e4);
                        }
#pragma unroll
                        for (int p2 = 0; p2 < 2; ++p2)
#pragma unroll
                            for (int k8 = 0; k8 < CW / 8; ++k8)
#pragma unroll
                                for (int k = 0; k < 8; k += 2)   // packed fp32x2 add (FADD2), round to nearest
                                    fadd2(acc[2 * hp + p2][k8 * 8 + k], acc[2 * hp + p2][k8 * 8 + k + 1],
                                          v[p2][k8][k], v[p2][k8][k + 1]);
                    }
                    DBG_T(e5);
                    DBG_ADD(e_add, e3, e5);
                    ++it;
                }
                DBG_T(e6);
                // final epilogue from registers: bias -> ReLU -> BN -> 2x2 max -> hi/lo fp16 (+ fp32 tap)
                constexpr int RO = R / 2;
                const int Y = r >> 3, X = 8 * sub + (r & 7);
#pragma unroll
                for (int k8 = 0; k8 < CW / 8; ++k8) {
                    const int c0 = cq * CW + k8 * 8;
                    float o[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const float b = __ldg(bias + c0 + k), sc = __ldg(bn_s + c0 + k), sh = __ldg(bn_t + c0 + k);
                        float m = acc[0][k8 * 8 + k];
#pragma unroll
                        for (int ph = 1; ph < NT; ++ph) m = fmaxf(m, acc[ph][k8 * 8 + k]);
                        o[k] = pooled_act(m, inv_scale, invd, b, sc, sh);
                    }
                    const size_t off = ((((size_t)cell * (COUT / 8) + c0 / 8) * RO + Y) * RO + X) * 8;
                    split_store8(o, out_hi + off, out_lo ? out_lo + off : nullptr, range_ok);
                    if (feat) {
                        float4* f = reinterpret_cast<float4*>(feat + (size_t)cell * (RO * RO * COUT) +
                                                             (size_t)(Y * RO + X) * COUT + c0);
                        f[0] = make_float4(o[0], o[1], o[2], o[3]);
                        f[1] = make_float4(o[4], o[5], o[6], o[7]);
                    }
                }
                DBG_T(e7);
                DBG_ADD(e_final, e6, e7);
            }   // sub (pooled X half)
        }
#ifdef CIA_ACC_TIMING
        if (tid == 0) {
            atomicAdd(&g_acc_dbg[0], (unsigned long long)e_stage);
            atomicAdd(&g_acc_dbg[1], (unsigned long long)e_full);
            atomicAdd(&g_acc_dbg[2], (unsigned long long)e_ld);
            atomicAdd(&g_acc_dbg[3], (unsigned long long)e_add);
            atomicAdd(&g_acc_dbg[4], (unsigned long long)e_final);
            atomicAdd(&g_acc_dbg[5], (unsigned long long)e_units);
        }
#endif
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, TMEM_COLS);
    if (!range_ok) raise_status(status, CIA_E_UNSUPPORTED);
}

// ---------------------------------------------------------------------------------------
// Layer 1 (Cin = 1, K = 9)
// ---------------------------------------------------------------------------------------
// Layer 1 of the single-pass path on the CUDA cores, exact fp32 FMAs (with K = 9 the layer is
// epilogue-bound, not MMA-bound).  One block = one quadrant of a cell (pooled 16x16 = conv 32x32);
// thread = (channel group of 8, pooled pixel), 4 conv pixels x 8 channels in registers; output =
// the chunk-planar fp16 plane.
__global__ void __launch_bounds__(256, 2)
conv1_fp32_planar_kernel(const float* __restrict__ crops, const float* __restrict__ wgt /* [9][32] */,
                         const float* __restrict__ bias, const float* __restrict__ bn_s,
                         const float* __restrict__ bn_t, __half* __restrict__ out_hi,
                         int n_cells, const int32_t* __restrict__ n_dev, int cell0, int chunk_cells,
                         int32_t* __restrict__ status) {
    bool range_ok = true;             // every fp16 activation store of this thread was finite
    __shared__ __align__(16) float xs[34][36];
    __shared__ __align__(16) float ws[9][32];
    int n = dev_count(n_cells, n_dev) - cell0;
    if (n > chunk_cells) n = chunk_cells;
    const int tid = threadIdx.x, cg = tid >> 6, p = tid & 63;
    for (int i = tid; i < 9 * 32; i += 256) ws[i >> 5][i & 31] = __ldg(wgt + i);
    float b8[8], s8[8], t8[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        b8[k] = __ldg(bias + cg * 8 + k); s8[k] = __ldg(bn_s + cg * 8 + k); t8[k] = __ldg(bn_t + cg * 8 + k);
    }
    // BN after ReLU is monotone in the conv output when its scale is >= 0, so the 2x2 max can be taken
    // first and ReLU + BN applied once (bit-identical); a negative scale keeps the per-pixel form
    bool scale_pos = true;
#pragma unroll
    for (int k = 0; k < 8; ++k) scale_pos = scale_pos && s8[k] >= 0.f;
    for (int unit = blockIdx.x; unit < n * 4; unit += gridDim.x) {
        const int cell = cell0 + (unit >> 2), qy = (unit >> 1) & 1, qx = unit & 1;
        const float* xr = crops + (size_t)cell * 4096;
        __syncthreads();
        {   // all five loads of a thread in flight before the first store (one latency, not five)
            float v[5];
#pragma unroll
            for (int j = 0; j < 5; ++j) {
                const int i = tid + j * 256;
                const int ry = i / 34, rc = i - ry * 34;
                const int y = 32 * qy + ry - 1, x = 32 * qx + rc - 1;
                v[j] = (i < 34 * 34 && y >= 0 && y < 64 && x >= 0 && x < 64) ? __ldg(xr + y * 64 + x) : 0.f;
            }
#pragma unroll
            for (int j = 0; j < 5; ++j) {
                const int i = tid + j * 256;
                if (i < 34 * 34) xs[i / 34][i % 34] = v[j];
            }
        }
        __syncthreads();
#pragma unroll 1
        for (int it = 0; it < 4; ++it) {
            const int P = it * 64 + p, Y = P >> 4, X = P & 15;
            float win[4][4];
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                const float2 v0 = *reinterpret_cast<const float2*>(&xs[2 * Y + a][2 * X]);
                const float2 v1 = *reinterpret_cast<const float2*>(&xs[2 * Y + a][2 * X + 2]);
                win[a][0] = v0.x; win[a][1] = v0.y; win[a][2] = v1.x; win[a][3] = v1.y;
            }
            // packed fp32x2 FMAs (FFMA2): two output channels per instruction, IEEE RN per lane;
            // accumulators start from the bias so that (bias + sum) is one FMA chain
            unsigned long long acc2[4][4], win2[4][4];
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) win2[a][b] = pack2(win[a][b], win[a][b]);
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) acc2[q][kk] = pack2(b8[2 * kk], b8[2 * kk + 1]);
#pragma unroll
            for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                for (int dx = 0; dx < 3; ++dx) {
                    const ulonglong2 w0 = *reinterpret_cast<const ulonglong2*>(&ws[dy * 3 + dx][cg * 8]);
                    const ulonglong2 w1 = *reinterpret_cast<const ulonglong2*>(&ws[dy * 3 + dx][cg * 8 + 4]);
                    const unsigned long long wp[4] = {w0.x, w0.y, w1.x, w1.y};
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        acc2[0][kk] = fma2(win2[dy][dx], wp[kk], acc2[0][kk]);
                        acc2[1][kk] = fma2(win2[dy][dx + 1], wp[kk], acc2[1][kk]);
                        acc2[2][kk] = fma2(win2[dy + 1][dx], wp[kk], acc2[2][kk]);
                        acc2[3][kk] = fma2(win2[dy + 1][dx + 1], wp[kk], acc2[3][kk]);
                    }
                }
            float acc[4][8];
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) unpack2(acc2[q][kk], acc[q][2 * kk], acc[q][2 * kk + 1]);
            float o[8];
            if (scale_pos) {
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const float m = fmaxf(fmaxf(acc[0][k], acc[1][k]), fmaxf(acc[2][k], acc[3][k]));
                    o[k] = __fadd_rn(__fmul_rn(fmaxf(m, 0.f), s8[k]), t8[k]);
                }
            } else {
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    float m = -INFINITY;
#pragma unroll
                    for (int q = 0; q < 4; ++q) m = fmaxf(m, __fadd_rn(__fmul_rn(fmaxf(acc[q][k], 0.f), s8[k]), t8[k]));
                    o[k] = m;
                }
            }
            const size_t off = ((((size_t)cell * 4 + cg) * 32 + (16 * qy + Y)) * 32 + (16 * qx + X)) * 8;
            split_store8(o, out_hi + off, nullptr, range_ok);
        }
    }
    if (!range_ok) raise_status(status, CIA_E_UNSUPPORTED);
}

// ---------------------------------------------------------------------------------------
// Layer 1 on the tensor cores (default for the split-precision pass).
//
// With K = 9 the MMAs are almost free (12 per 128 pooled pixels); the cost is building the A
// operand and the epilogue.  One unit = a band of 8 conv rows x 64 columns = 4 x 32 pooled
// pixels = the 128 rows of an MMA tile; the four pooling phases (py,px) are four tiles, so the
// pool partners of a pooled pixel share a TMEM lane.  Per unit:
//   1. the 10 x 64 input window (one float4 per loading thread, fetched one unit ahead) is scaled
//      by 2^6, split ONCE per input pixel into fp16 hi + lo and parked in shared memory with one
//      8-byte store per part (the zero halo columns are written once in the prologue);
//   2. the explicit im2col rows are assembled by byte permutes only: the window of a pooled pixel
//      is 3 rows x 3 words, the K order is chosen per column phase so that three of the five
//      words of an A row are the loaded words themselves (k8 sits in the second k-chunk, whose
//      other seven columns stay zero from the kernel prologue);
//   3. three MMAs per phase (hi*lo, lo*hi, then hi*hi) accumulate in one TMEM tile: within an
//      instruction the products are summed exactly and added with ONE round-toward-zero
//      (profiles/umma_rounding_test.cu), the cross terms are 2^-11 of the result;
//   4. epilogue: ReLU and BN are monotone in the conv output -- increasing for a BN scale >= 0,
//      decreasing otherwise -- so the 2x2 max of the reference equals ONE evaluation at the max
//      (resp. min) over the phases, bit for bit.  The weight image carries the sign of the BN
//      scale per output channel, so the extremum is always a max and the sign is put back with
//      one XOR; the mean half-ulp deficit of the truncation is added back together with the
//      bias, then ReLU, BN, hi/lo split, 16-byte stores (512 contiguous bytes per warp).
// Double-buffered windows, A blocks and TMEM stages; a ninth warp issues the MMAs (one thread), so the
// MMAs of unit u+1 run under the epilogue of u and the eight worker warps meet at ONE barrier per unit.
// Inputs must satisfy |x| < 1023 (crops are CLAHE output in [0,1]).
// ---------------------------------------------------------------------------------------
namespace l1tc {
constexpr int WORKER_WARPS = 8;
constexpr int NT = (WORKER_WARPS + 1) * 32;       // + one MMA-issuing warp
constexpr int XS_PITCH = 72;                      // halves per staged window row: column x sits at x + 4
constexpr int XS_PART_B = 10 * XS_PITCH * 2;
constexpr int XS_LOADERS = 10 * 16;               // one float4 (4 columns of one window row) per loading thread
constexpr int A_PH_B = 2 * 128 * 16;              // one phase: [k-chunk][row][8 halves]
constexpr int A_PART_B = 4 * A_PH_B;              // hi or lo part of a block
constexpr int A_BUF_B = 2 * A_PART_B;
constexpr int W_IMG_B = 2 * 32 * 16;              // [k-chunk][n][8 halves]
constexpr int W_B = 4 * W_IMG_B;                  // [px][hi | lo]
constexpr int SMEM_B = 2 * A_BUF_B + W_B + 4 * XS_PART_B;   // two A blocks, weights, two windows
constexpr int TBUF_COLS = 4 * 32;
constexpr int TMEM_COLS = 2 * TBUF_COLS;
constexpr int XSCALE_EXP = 6;
// tap (dy*3+dx) held by K column k of the A rows of column phase px (see build below)
__host__ __device__ constexpr int tap_of(int px, int k) {
    return px == 1 ? (k < 6 ? (k >> 1) * 3 + (k & 1) : (k - 6) * 3 + 2)
                   : (k < 6 ? (k >> 1) * 3 + (k & 1) + 1 : (k - 6) * 3);
}
}  // namespace l1tc

__global__ void __launch_bounds__(l1tc::NT, 2)
conv1_tc_split_kernel(const float* __restrict__ crops, const uint4* __restrict__ w_img, float inv_scale,
                      float debias, const float* __restrict__ bias, const float* __restrict__ bn_s,
                      const float* __restrict__ bn_t, __half* __restrict__ out_hi, __half* __restrict__ out_lo,
                      int n_cells, const int32_t* __restrict__ n_dev, int cell0, int chunk_cells,
                      int32_t* __restrict__ status) {
    bool range_ok = true;             // every fp16 activation store of this thread was finite
    using namespace l1tc;
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ __align__(8) uint64_t done_bar[2], afull_bar[2];
    __shared__ uint32_t tmem_base_s;
    unsigned char* const w_s = smem + 2 * A_BUF_B;
    unsigned char* const xs0 = w_s + W_B;          // two windows of [hi | lo] parts

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int n = dev_count(n_cells, n_dev) - cell0;
    if (n > chunk_cells) n = chunk_cells;
    if (n <= 0) return;
    const int n_units = n * 8;
    const int stride = (int)gridDim.x;

    if (warp == 0) tmem_alloc(&tmem_base_s, TMEM_COLS);
    if (tid == 32) {
        mbar_init(&done_bar[0], 1); mbar_init(&done_bar[1], 1);
        mbar_init(&afull_bar[0], WORKER_WARPS); mbar_init(&afull_bar[1], WORKER_WARPS);
        fence_barrier_init();
    }
    for (int i = tid; i < 2 * A_BUF_B / 16; i += NT) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    for (int i = tid; i < 4 * XS_PART_B / 16; i += NT) reinterpret_cast<uint4*>(xs0)[i] = make_uint4(0, 0, 0, 0);
    for (int i = tid; i < W_B / 16; i += NT) reinterpret_cast<uint4*>(w_s)[i] = __ldg(w_img + i);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    constexpr uint32_t IDESC = make_idesc(128, 32);

    if (warp == WORKER_WARPS) {
        // ================= MMA issuer: one thread, 12 MMAs per unit =================
        // (the workers never run issue code: with the issue inside four of the worker warps the
        // other four waited for them at every block barrier)
        if (lane == 0) {
            uint64_t d_ahi[4], d_alo[4], d_whi[2], d_wlo[2];
#pragma unroll
            for (int ph = 0; ph < 4; ++ph) {
                d_ahi[ph] = make_smem_desc(smem_u32(smem) + (uint32_t)(ph * A_PH_B), 128 * 16, 128);
                d_alo[ph] = make_smem_desc(smem_u32(smem) + (uint32_t)(A_PART_B + ph * A_PH_B), 128 * 16, 128);
            }
#pragma unroll
            for (int px = 0; px < 2; ++px) {
                d_whi[px] = make_smem_desc(smem_u32(w_s) + (uint32_t)((px * 2) * W_IMG_B), 32 * 16, 128);
                d_wlo[px] = make_smem_desc(smem_u32(w_s) + (uint32_t)((px * 2 + 1) * W_IMG_B), 32 * 16, 128);
            }
            uint32_t it = 0;
            for (int unit = blockIdx.x; unit < n_units; unit += stride, ++it) {
                const uint32_t buf = it & 1;
                mbar_wait(&afull_bar[buf], (it >> 1) & 1);      // A block written AND the TMEM stage drained
                tc_fence_after();
                const uint64_t bo = (uint64_t)(buf * (A_BUF_B >> 4));
#pragma unroll
                for (int ph = 0; ph < 4; ++ph) {
                    const uint32_t d = tmem_base + buf * TBUF_COLS + (uint32_t)(ph * 32);
                    umma_f16(d, d_ahi[ph] + bo, d_wlo[ph & 1], IDESC, 0u);
                    umma_f16(d, d_alo[ph] + bo, d_whi[ph & 1], IDESC, 1u);
                    umma_f16(d, d_ahi[ph] + bo, d_whi[ph & 1], IDESC, 1u);
                }
                umma_commit(&done_bar[buf]);
            }
        }
    } else {
        // ================= workers: window split, A rows, epilogue =================
        // epilogue role: TMEM lane quadrant q (= pooled row of the band), 16 channels per warp half
        const int q = warp & 3, hs = warp >> 2;
        float b16[16], s16[16], t16[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            b16[k] = __ldg(bias + 16 * hs + k); s16[k] = __ldg(bn_s + 16 * hs + k); t16[k] = __ldg(bn_t + 16 * hs + k);
        }
        const float invd = inv_scale * debias;
        // loading role (threads 0..159): window row lrow, columns 4*lc4 .. 4*lc4+3
        const int lrow = tid >> 4, lc4 = tid & 15;
        float4 pv = make_float4(0.f, 0.f, 0.f, 0.f);
        auto prefetch = [&](int unit) {
            const int y = 8 * (unit & 7) - 1 + lrow;
            pv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (tid < XS_LOADERS && y >= 0 && y < 64)
                pv = __ldg(reinterpret_cast<const float4*>(crops + (size_t)(cell0 + (unit >> 3)) * 4096 + y * 64) + lc4);
        };
        auto split_park = [&](unsigned char* xs) {
            if (tid < XS_LOADERS) {
                constexpr float SC = (float)(1 << XSCALE_EXP);
                const float v0 = pv.x * SC, v1 = pv.y * SC, v2 = pv.z * SC, v3 = pv.w * SC;
                const __half2 h01 = __floats2half2_rn(v0, v1), h23 = __floats2half2_rn(v2, v3);
                const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
                const __half2 l01 = __floats2half2_rn(v0 - f01.x, v1 - f01.y), l23 = __floats2half2_rn(v2 - f23.x, v3 - f23.y);
                const int o = (lrow * XS_PITCH + 4 * lc4 + 4) * 2;
                *reinterpret_cast<uint2*>(xs + o) = make_uint2(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23));
                *reinterpret_cast<uint2*>(xs + XS_PART_B + o) = make_uint2(*reinterpret_cast<const uint32_t*>(&l01), *reinterpret_cast<const uint32_t*>(&l23));
            }
        };
        // thread -> (MMA row r = pooled pixel (Y,X) of the band, row phase py); both column phases.
        // Window columns c0..c3 (x = 2X-1 .. 2X+2) sit in three words: (.,c0) (c1,c2) (c3,.)
        auto build = [&](const unsigned char* xs, unsigned char* ab) {
            const int r = tid & 127, py = tid >> 7, Y = r >> 5, X = r & 31;
#pragma unroll
            for (int part = 0; part < 2; ++part) {
                const uint32_t* xw = reinterpret_cast<const uint32_t*>(xs + part * XS_PART_B) +
                                     (2 * Y + py) * (XS_PITCH / 2) + X + 1;
                uint32_t wa[3], wb[3], wc[3];
#pragma unroll
                for (int a = 0; a < 3; ++a) {
                    wa[a] = xw[a * (XS_PITCH / 2)]; wb[a] = xw[a * (XS_PITCH / 2) + 1]; wc[a] = xw[a * (XS_PITCH / 2) + 2];
                }
                unsigned char* dst = ab + part * A_PART_B + (py * 2) * A_PH_B + r * 16;
                // px = 0: columns c0,c1,c2;  K = (0,1)(0,2)(1,1)(1,2)(2,1)(2,2)(0,0)(1,0) | (2,0)
                *reinterpret_cast<uint4*>(dst) = make_uint4(wb[0], wb[1], wb[2], __byte_perm(wa[0], wa[1], 0x7632));
                *reinterpret_cast<uint32_t*>(dst + 128 * 16) = wa[2] >> 16;
                // px = 1: columns c1,c2,c3;  K = (0,0)(0,1)(1,0)(1,1)(2,0)(2,1)(0,2)(1,2) | (2,2)
                *reinterpret_cast<uint4*>(dst + A_PH_B) = make_uint4(wb[0], wb[1], wb[2], __byte_perm(wc[0], wc[1], 0x5410));
                *reinterpret_cast<uint32_t*>(dst + A_PH_B + 128 * 16) = wc[2] & 0xFFFFu;
            }
        };
        // window (kk & 1) and A block (kk & 1) of the CTA's kk-th unit: split, worker barrier, A rows, signal.
        // The window is double-buffered because a fast warp may split unit kk+1 while a slow one still
        // builds unit kk; by unit kk+2 every warp has passed the worker barrier of kk+1, i.e. finished kk.
        auto produce = [&](uint32_t kk) {
            unsigned char* xs = xs0 + (kk & 1) * 2 * XS_PART_B;
            split_park(xs);
            asm volatile("bar.sync 1, %0;" ::"n"(WORKER_WARPS * 32) : "memory");
            build(xs, smem + (kk & 1) * A_BUF_B);
            fence_async_smem();
            tc_fence_before();      // orders this thread's TMEM reads of the stage's previous unit
            __syncwarp();
            if (lane == 0) mbar_arrive(&afull_bar[kk & 1]);
        };

        if ((int)blockIdx.x < n_units) {
            prefetch(blockIdx.x);
            produce(0);
            if ((int)blockIdx.x + stride < n_units) prefetch(blockIdx.x + stride);
        }
        uint32_t it = 0;
        for (int unit = blockIdx.x; unit < n_units; unit += stride, ++it) {
            const uint32_t tbuf = it & 1;
            if (unit + stride < n_units) {
                // the other A block was consumed by the MMAs of unit-stride (their barrier was waited on one
                // iteration ago); its TMEM stage was drained by this thread's epilogue of that unit
                produce(it + 1);
                if (unit + 2 * stride < n_units) prefetch(unit + 2 * stride);
            }
            mbar_wait(&done_bar[tbuf], (it >> 1) & 1);
            tc_fence_after();

            const int cell = cell0 + (unit >> 3), Yp = 4 * (unit & 7) + q;
            const uint32_t taddr = tmem_base + ((uint32_t)(32 * q) << 16) + tbuf * TBUF_COLS + (uint32_t)(16 * hs);
#pragma unroll
            for (int sl = 0; sl < 2; ++sl) {
                uint32_t v[4][8];
#pragma unroll
                for (int ph = 0; ph < 4; ++ph) TMEM_LD8(taddr + (uint32_t)(ph * 32 + sl * 8), v[ph]);
#pragma unroll
                for (int ph = 0; ph < 4; ++ph) TMEM_WAIT8(v[ph]);
                float o[8];
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    o[k] = pooled_act(fmaxf(fmaxf(__uint_as_float(v[0][k]), __uint_as_float(v[1][k])),
                                            fmaxf(__uint_as_float(v[2][k]), __uint_as_float(v[3][k]))),
                                      inv_scale, invd, b16[sl * 8 + k], s16[sl * 8 + k], t16[sl * 8 + k]);
                const size_t off = ((((size_t)cell * 4 + (2 * hs + sl)) * 32 + Yp) * 32 + lane) * 8;
                split_store8(o, out_hi + off, out_lo + off, range_ok);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, TMEM_COLS);
    if (!range_ok) raise_status(status, CIA_E_UNSUPPORTED);
}

// ---------------------------------------------------------------------------------------
// Layer 7 (32 -> 1 channel on the 2x up-sampled 64x64 map) with the filter taps on the N axis.
//
// In phase form the layer is a 3x3 conv on the 32x32 low-resolution map with four outputs
// (py,px) per pixel, and each output only sees a 2x2 block of low-resolution neighbours (the
// nine high-resolution taps collapse onto them).  As an implicit GEMM that is N = 16 with four
// real columns and K = 9 taps x 32 channels: 144 MMAs per cell whose cost is the 4 KB A-operand
// fetch (ncu: tensor-core pipe 87 % busy for 18 % math, profiles/r1j_cae_full.txt).  Here the
// contraction over channels and the sum over taps swap places:
//     P[pixel][(py,px),(ty,tx)] = sum_c A6[pixel][c] * Weff[c][(py,px),(ty,tx)]      (16 columns)
//     out[2Y+py][2X+px] = sum_{ty,tx} P[(Y+py-1+ty, X+px-1+tx)][(py,px),(ty,tx)] + bias
// -- ONE tap, K = 32: 16 MMAs per cell, no halo, and the A operand of a cell is its 64 KB of
// activations exactly as they lie in HBM ([chunk][y][x][8] = K-major core matrices), fetched by
// one bulk copy (TMA) into one of two buffers.  The weights ride as [hi | lo] fp16 pairs on 32
// columns (the A fetch bounds an MMA whatever N is), so this layer's weights are exact.  The
// shifted tap sum runs on the CUDA cores through shared-memory planes [column][pixel], fused
// with sigmoid, (x - y)^2, |x - y| and the per-cell reduction.
//   warps 0..15: epilogue (TMEM lane quadrant = warp & 3, tiles (warp >> 2) and (warp >> 2) + 4)
//   warp 16:     lane 0 issues the bulk copies and the MMAs
// ---------------------------------------------------------------------------------------
namespace l7 {
constexpr int EPI_WARPS = 16;
constexpr int NT = (EPI_WARPS + 1) * 32;
constexpr int A_B = 1024 * 32 * 2;                 // one cell: 4 chunks x 1024 pixels x 8 halves
constexpr int W_B = 4 * 32 * 16;                   // [chunk][32 columns][8 halves]
constexpr int PL_B = 16 * 1024 * 4;                // tap-sum planes [column][pixel] fp32
constexpr int SMEM_B = 2 * A_B + W_B + PL_B;
constexpr int STAGE_COLS = 8 * 32;                 // 8 tiles x (16 hi + 16 lo columns)
}  // namespace l7

__global__ void __launch_bounds__(l7::NT, 1)
final_tapsum_kernel(const __half* __restrict__ a6, const uint4* __restrict__ w_img, float inv_scale,
                    const float* __restrict__ bias, const float* __restrict__ crops,
                    float* __restrict__ mse, float* __restrict__ mae, int n_cells,
                    const int32_t* __restrict__ n_dev, int cell0, int chunk_cells) {
    using namespace l7;
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ __align__(8) uint64_t a_full[2], d_full[2], d_empty[2];
    __shared__ uint32_t tmem_base_s;
    __shared__ float red_s[2][2][EPI_WARPS];
    unsigned char* const w_s = smem + 2 * A_B;
    float* const planes = reinterpret_cast<float*>(smem + 2 * A_B + W_B);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int n = dev_count(n_cells, n_dev) - cell0;
    if (n > chunk_cells) n = chunk_cells;
    if (n <= 0) return;
    const int stride = (int)gridDim.x;

    if (warp == 0) tmem_alloc(&tmem_base_s, 2 * STAGE_COLS);
    if (tid == 32) {
        for (int i = 0; i < 2; ++i) { mbar_init(&a_full[i], 1); mbar_init(&d_full[i], 1); mbar_init(&d_empty[i], EPI_WARPS); }
        fence_barrier_init();
    }
    for (int i = tid; i < W_B / 16; i += NT) reinterpret_cast<uint4*>(w_s)[i] = __ldg(w_img + i);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    if (warp == EPI_WARPS) {
        if (lane == 0) {
            constexpr uint32_t IDESC = make_idesc(128, 32);
            const uint64_t bd0 = make_smem_desc(smem_u32(w_s), 32 * 16, 128);
            const __half* src0 = a6 + (size_t)cell0 * (A_B / 2);
            // prologue: the first two cells' activations
            for (int k = 0; k < 2; ++k) {
                const int unit = (int)blockIdx.x + k * stride;
                if (unit < n) {
                    mbar_expect_tx(&a_full[k], A_B);
                    bulk_load(smem_u32(smem) + k * A_B, src0 + (size_t)unit * (A_B / 2), A_B, &a_full[k]);
                }
            }
            uint32_t it = 0;
            for (int unit = blockIdx.x; unit < n; unit += stride, ++it) {
                const uint32_t st = it & 1, ph = (it >> 1) & 1;
                mbar_wait(&a_full[st], ph);
                mbar_wait(&d_empty[st], ph ^ 1);            // the epilogue of two cells ago has drained this stage
                tc_fence_after();
                const uint64_t ad0 = make_smem_desc(smem_u32(smem) + st * A_B, 1024 * 16, 128);
#pragma unroll
                for (int t = 0; t < 8; ++t)
#pragma unroll
                    for (int ks = 0; ks < 2; ++ks)
                        umma_f16(tmem_base + st * STAGE_COLS + (uint32_t)(t * 32),
                                 ad0 + (uint64_t)((t * 128 * 16 + 2 * ks * 1024 * 16) >> 4),
                                 bd0 + (uint64_t)((2 * ks * 32 * 16) >> 4), IDESC, ks);
                umma_commit(&d_full[st]);
                // the MMAs have read the buffer: refill it with the cell after next
                mbar_wait(&d_full[st], ph);
                if (unit + 2 * stride < n) {
                    mbar_expect_tx(&a_full[st], A_B);
                    bulk_load(smem_u32(smem) + st * A_B, src0 + (size_t)(unit + 2 * stride) * (A_B / 2), A_B, &a_full[st]);
                }
            }
        }
    } else {
        const int q = warp & 3, g = warp >> 2;
        const float b = __ldg(bias);
        uint32_t it = 0;
        for (int unit = blockIdx.x; unit < n; unit += stride, ++it) {
            const uint32_t st = it & 1, ph = (it >> 1) & 1;
            const int cell = cell0 + unit;
            mbar_wait(&d_full[st], ph);
            tc_fence_after();
            // planes of the previous cell have been consumed (barrier 2 of the previous iteration)
#pragma unroll
            for (int tt = 0; tt < 2; ++tt) {
                const int t = g + 4 * tt;
                const int p = 128 * t + 32 * q + lane;
                const uint32_t taddr = tmem_base + ((uint32_t)(32 * q) << 16) + st * STAGE_COLS + (uint32_t)(t * 32);
                uint32_t v[4][8];
#pragma unroll
                for (int k = 0; k < 4; ++k) TMEM_LD8(taddr + 8 * k, v[k]);
#pragma unroll
                for (int k = 0; k < 4; ++k) TMEM_WAIT8(v[k]);
#pragma unroll
                for (int c = 0; c < 16; ++c)
                    planes[c * 1024 + p] = __uint_as_float(v[c >> 3][c & 7]) + __uint_as_float(v[2 + (c >> 3)][c & 7]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&d_empty[st]);
            asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");      // planes complete
            float se = 0.f, ae = 0.f;
            const float* xr = crops + (size_t)cell * 4096;
#pragma unroll
            for (int tt = 0; tt < 2; ++tt) {
                const int p = 128 * (g + 4 * tt) + 32 * q + lane;
                const int Y = p >> 5, X = p & 31;
#pragma unroll
                for (int py = 0; py < 2; ++py) {
                    const float2 xv = __ldg(reinterpret_cast<const float2*>(xr + (2 * Y + py) * 64 + 2 * X));
#pragma unroll
                    for (int px = 0; px < 2; ++px) {
                        float sum = 0.f;
#pragma unroll
                        for (int ty = 0; ty < 2; ++ty)
#pragma unroll
                            for (int tx = 0; tx < 2; ++tx) {
                                const int yy = Y + py - 1 + ty, xx = X + px - 1 + tx;
                                if ((unsigned)yy < 32u && (unsigned)xx < 32u)
                                    sum += planes[(4 * (2 * py + px) + 2 * ty + tx) * 1024 + yy * 32 + xx];
                            }
                        const float a = fmaf(sum, inv_scale, b);
                        const float rec = __fdividef(1.f, 1.f + __expf(-a));   // |err| ~1e-6, MSE gate is 1e-3
                        const float d = (px ? xv.y : xv.x) - rec;
                        se = fmaf(d, d, se);
                        ae += fabsf(d);
                    }
                }
            }
            se = warp_sum(se); ae = warp_sum(ae);
            if (lane == 0) { red_s[it & 1][0][warp] = se; red_s[it & 1][1][warp] = ae; }
            asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");      // planes free, partial sums visible
            if (tid == 0) {
                float s = 0.f, a = 0.f;
#pragma unroll
                for (int w = 0; w < EPI_WARPS; ++w) { s += red_s[it & 1][0][w]; a += red_s[it & 1][1][w]; }
                mse[cell] = s * (1.f / 4096.f);
                mae[cell] = a * (1.f / 4096.f);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 2 * l7::STAGE_COLS);
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
template <int CIN, int COUT, int R, int EPI, int NPASS, bool UPSIN = false>
int launch_tc(cia_ctx* h, const CaeWeights& w, int layer, const __half* in_hi, const __half* in_lo,
              __half* out_hi, __half* out_lo, float* feat, int n, const int32_t* n_dev, int cell0, int chunk,
              cudaStream_t s) {
    using C = Cfg<CIN, COUT, R, EPI, NPASS>;
    auto kern = conv_tc_kernel<CIN, COUT, R, EPI, NPASS, UPSIN>;
    if (first_use(h, (const void*)kern))
        CIA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_B));
    int grid = chunk * C::UNITS_PER_CELL;
    const int cap = h->num_sms * (C::SMEM_B > 100 * 1024 ? 1 : 2);
    if (grid > cap) grid = cap;
    kern<<<grid, C::THREADS, C::SMEM_B, s>>>(in_hi, in_lo, (const uint4*)w.tc_w[layer][0], (const uint4*)w.tc_w[layer][1],
                                      w.tc_inv_scale[layer], w.bias[layer], w.bn_scale[layer], w.bn_shift[layer],
                                      out_hi, out_lo, feat, n, n_dev, cell0, chunk, h->status_dev);
    CIA_LAUNCH_CHECK();
    return CIA_OK;
}

#ifdef CIA_ACC_TIMING
// per-phase cycle sums of one launch (thread 0 / first MMA warp of every CTA), averaged per cell
static void acc_timing_dump(const char* name, int cin, int cout, int r, int g, cudaStream_t s) {
    if (!getenv("CIA_ACC_DUMP")) return;
    unsigned long long d[16];
    cudaStreamSynchronize(s);
    cudaMemcpyFromSymbol(d, g_acc_dbg, sizeof(d));
    const double u = d[5] ? (double)d[5] : 1.0;
    fprintf(stderr, "%s<%d,%d,%d,G%d> cells %llu per-cell cycles: stage %.0f wait_full %.0f ld %.0f ld+add %.0f "
                    "final %.0f | mma: wait_ready %.0f wait_empty %.0f issue %.0f\n", name, cin, cout, r, g, d[5],
            d[0] / u, d[1] / u, d[2] / u, d[3] / u, d[4] / u, d[8] / u, d[9] / u, d[10] / u);
    memset(d, 0, sizeof(d));
    cudaMemcpyToSymbol(g_acc_dbg, d, sizeof(d));
}
#else
static inline void acc_timing_dump(const char*, int, int, int, int, cudaStream_t) {}
#endif

// mean relative deficit of the accumulating kernels' truncated sums, in units of 2^-24
// (cia_set_option "cae_l2_debias" / "cae_l3_debias", 0 = off; derivation in DESIGN.md section 5)
static float acc_debias(const cia_ctx* h, int layer) { return h->cae_debias[layer == 1 ? 1 : 2] * 5.9604645e-8f; }

template <int CIN, int COUT, int R, int G = 1>
int launch_tc_acc(cia_ctx* h, const CaeWeights& w, int layer, const __half* in_hi, const __half* in_lo,
                  __half* out_hi, __half* out_lo, float* feat, int n, const int32_t* n_dev, int cell0,
                  int chunk, cudaStream_t s) {
    using C = AccCfg<CIN, COUT, R>;
    auto kern = conv_tc_acc_kernel<CIN, COUT, R, G>;
    if (first_use(h, (const void*)kern))
        CIA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_B));
    int grid = chunk;
    if (grid > h->num_sms) grid = h->num_sms;
    kern<<<grid, ACC_THREADS, C::SMEM_B, s>>>(in_hi, in_lo, (const uint4*)w.tc_w[layer][0],
                                              (const uint4*)w.tc_w[layer][1], w.tc_inv_scale[layer],
                                              w.tc_inv_scale[layer] * acc_debias(h, layer), w.bias[layer],
                                              w.bn_scale[layer], w.bn_shift[layer], out_hi, out_lo, feat, n, n_dev,
                                              cell0, chunk, h->status_dev);
    CIA_LAUNCH_CHECK();
    acc_timing_dump("acc", CIN, COUT, R, G, s);
    return CIA_OK;
}

// Tensor map over one chunk buffer of chunk-planar fp16 activations [cells][C/8][R][R][8]:
// dims (8, x, y, chunk, cell); the box reads every second column (element stride 2 along x).
typedef CUresult (*TensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                      const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                      CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int encode_act_map(cia_ctx* h, CUtensorMap* tm, const __half* base, int nch, int r, int cells, int box_x,
                          int box_y) {
    static TensorMapEncodeFn encode = [] {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess) fn = nullptr;
        return (TensorMapEncodeFn)fn;
    }();
    if (!encode) { h->err = "cuTensorMapEncodeTiled is not available from this driver"; return CIA_E_UNSUPPORTED; }
    const cuuint64_t dims[5] = {8, (cuuint64_t)r, (cuuint64_t)r, (cuuint64_t)nch, (cuuint64_t)cells};
    const cuuint64_t strides[4] = {16, (cuuint64_t)16 * r, (cuuint64_t)16 * r * r, (cuuint64_t)16 * r * r * nch};
    const cuuint32_t box[5] = {8, (cuuint32_t)box_x, (cuuint32_t)box_y, (cuuint32_t)nch, 1};
    const cuuint32_t estr[5] = {1, 2, 1, 1, 1};
    const CUresult rc = encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, (void*)base, dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS) { h->err = "cuTensorMapEncodeTiled failed"; return CIA_E_CUDA; }
    return CIA_OK;
}

// R = 32 pooling layer with TMA-fed double-buffered half-cell blocks (conv_tc_acc2_kernel).
// in_hi / in_lo are the chunk buffers' own base addresses (cell 0 of the chunk).
template <int CIN, int COUT, int R, int G>
int launch_tc_acc2(cia_ctx* h, const CaeWeights& w, int layer, const __half* in_hi, const __half* in_lo,
                   int buf_cells, __half* out_hi, __half* out_lo, float* feat, int n, const int32_t* n_dev,
                   int cell0, int chunk, cudaStream_t s) {
    using C = Acc2Cfg<CIN, COUT, R>;
    static_assert(C::SMEM_B + 1280 <= 227 * 1024, "double-buffered blocks do not fit in shared memory");
    auto kern = conv_tc_acc2_kernel<CIN, COUT, R, G>;
    if (first_use(h, (const void*)kern))
        CIA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_B));
    CUtensorMap tm_hi, tm_lo;
    int rc;
    if ((rc = encode_act_map(h, &tm_hi, in_hi, C::NCH, C::R, buf_cells, C::BOX_X, C::FILL_ROWS))) return rc;
    if ((rc = encode_act_map(h, &tm_lo, in_lo, C::NCH, C::R, buf_cells, C::BOX_X, C::FILL_ROWS))) return rc;
    int grid = chunk;
    if (grid > h->num_sms) grid = h->num_sms;
    kern<<<grid, ACC_THREADS, C::SMEM_B, s>>>(tm_hi, tm_lo, (const uint4*)w.tc_w[layer][0],
                                              (const uint4*)w.tc_w[layer][1], w.tc_inv_scale[layer],
                                              w.tc_inv_scale[layer] * acc_debias(h, layer), w.bias[layer],
                                              w.bn_scale[layer], w.bn_shift[layer], out_hi, out_lo, feat, n, n_dev,
                                              cell0, chunk, h->status_dev);
    CIA_LAUNCH_CHECK();
    acc_timing_dump("acc2", CIN, COUT, R, G, s);
    return CIA_OK;
}

// One B image: [(tap*NCH + chunk)*N + n][8] halves = w[tap][chunk*8 + j][n] * 2^sw, hi and lo parts.
static void pack_image(const std::vector<float>& w /* [taps][cin][n] */, int taps, int cin, int N,
                       int n_real, int sw, std::vector<__half>& hi, std::vector<__half>& lo,
                       const float* colsign = nullptr) {
    const int nch = cin / 8;
    hi.assign((size_t)taps * nch * N * 8, __float2half_rn(0.f));
    lo = hi;
    const float sc = std::ldexp(1.f, sw);
    for (int tap = 0; tap < taps; ++tap)
        for (int c = 0; c < cin; ++c)
            for (int nn = 0; nn < n_real; ++nn) {
                const float v = w[((size_t)tap * cin + c) * n_real + nn] * sc * (colsign ? colsign[nn] : 1.f);
                const __half hv = __float2half_rn(v);
                const size_t idx = (((size_t)tap * nch + c / 8) * N + nn) * 8 + (c % 8);
                hi[idx] = hv;
                lo[idx] = __float2half_rn(v - __half2float(hv));
            }
}

static int scale_exp(const std::vector<float>& w) {
    float m = 0.f;
    for (float v : w) m = std::fmax(m, std::fabs(v));
    if (!(m > 0.f)) return 0;
    int e;
    std::frexp(m, &e);          // m = f * 2^e, f in [0.5, 1)
    return 2 - e;               // m * 2^sw in [2, 4)
}

}  // namespace

int k_cae_tc_prepare(cia_ctx* h, int which) {
    CaeWeights& w = h->cae[which];
    w.tc_ready = false;
    for (int L = 0; L < w.n_conv; ++L) {
        const int cin = kCaeCin[L], cout = kCaeCout[L];
        std::vector<float> k((size_t)9 * cin * cout);
        CIA_CUDA(cudaMemcpy(k.data(), w.kernel[L], k.size() * sizeof(float), cudaMemcpyDeviceToHost));
        std::vector<__half> hi, lo;
        int sw;
        // pooling layers: ReLU + BN is monotone in the conv output, decreasing where the BN scale is
        // negative; the images carry that sign per output channel so that the pooled value is always
        // f(max over the 2x2 window) and the epilogues put the sign back with one XOR (bit-identical)
        std::vector<float> colsign(cout, 1.f);
        if (L < 3) {
            std::vector<float> sc_h(cout);
            CIA_CUDA(cudaMemcpy(sc_h.data(), w.bn_scale[L], cout * sizeof(float), cudaMemcpyDeviceToHost));
            for (int c = 0; c < cout; ++c) colsign[c] = std::signbit(sc_h[c]) ? -1.f : 1.f;
        }
        if (L == 0) {
            // layer 1 (K = 9): one image [px][hi | lo][k-chunk][n][8 halves] for conv1_tc_split_kernel, K columns
            // in the order its A rows are assembled in (l1tc::tap_of); K columns 9..15 are zero
            sw = scale_exp(k);
            const float sc = std::ldexp(1.f, sw);
            std::vector<__half> img((size_t)4 * 2 * 32 * 8, __float2half_rn(0.f));
            for (int px = 0; px < 2; ++px)
                for (int kk = 0; kk < 9; ++kk)
                    for (int nn = 0; nn < 32; ++nn) {
                        const float v = k[(size_t)l1tc::tap_of(px, kk) * 32 + nn] * sc * colsign[nn];
                        const __half hv = __float2half_rn(v);
                        const size_t idx = ((size_t)(kk >> 3) * 32 + nn) * 8 + (kk & 7);
                        img[(size_t)(px * 2 + 0) * 512 + idx] = hv;
                        img[(size_t)(px * 2 + 1) * 512 + idx] = __float2half_rn(v - __half2float(hv));
                    }
            w.tc_inv_scale[L] = std::ldexp(1.f, -sw - l1tc::XSCALE_EXP);
            cudaFree(w.tc_w[L][0]); w.tc_w[L][0] = nullptr;
            CIA_CUDA(cudaMalloc(&w.tc_w[L][0], img.size() * sizeof(__half)));
            CIA_CUDA(cudaMemcpy(w.tc_w[L][0], img.data(), img.size() * sizeof(__half), cudaMemcpyHostToDevice));
            continue;
        }
        if (L == 6) {
            // phase form: conv on the nearest-up-sampled input == 3x3 conv on the low-res input
            // with 4 outputs (py,px); weights of hi-res taps that fall on the same low-res pixel add up
            std::vector<float> kp((size_t)9 * cin * 4, 0.f);
            for (int py = 0; py < 2; ++py)
                for (int px = 0; px < 2; ++px)
                    for (int dy = 0; dy < 3; ++dy)
                        for (int dx = 0; dx < 3; ++dx) {
                            const int oy = (int)std::floor((py + dy - 1) / 2.0), ox = (int)std::floor((px + dx - 1) / 2.0);
                            const int tl = (oy + 1) * 3 + (ox + 1);
                            for (int c = 0; c < cin; ++c)
                                kp[((size_t)tl * cin + c) * 4 + py * 2 + px] += k[((size_t)(dy * 3 + dx) * cin + c)];
                        }
            // the scale of the phase form's weights; final_tapsum_kernel's image (below) and tc_inv_scale[6] use it
            sw = scale_exp(kp);
            // final_tapsum_kernel's image: ONE tap, the (phase, low-resolution neighbour) pairs on 16 columns
            // + their fp16 remainders on 16 more: [chunk][32][8]
            {
                std::vector<float> kt((size_t)cin * 16, 0.f);
                for (int py = 0; py < 2; ++py)
                    for (int px = 0; px < 2; ++px)
                        for (int dy = 0; dy < 3; ++dy)
                            for (int dx = 0; dx < 3; ++dx) {
                                const int oy = (int)std::floor((py + dy - 1) / 2.0), ox = (int)std::floor((px + dx - 1) / 2.0);
                                const int ty = oy - (py - 1), tx = ox - (px - 1);
                                for (int c = 0; c < cin; ++c)
                                    kt[(size_t)c * 16 + 4 * (2 * py + px) + 2 * ty + tx] += k[((size_t)(dy * 3 + dx) * cin + c)];
                            }
                std::vector<__half> img((size_t)(cin / 8) * 32 * 8, __float2half_rn(0.f));
                const float sc = std::ldexp(1.f, sw);        // the same scale: kt's entries are kp's (sums of the same taps)
                for (int c = 0; c < cin; ++c)
                    for (int col = 0; col < 16; ++col) {
                        const float v = kt[(size_t)c * 16 + col] * sc;
                        const __half hv = __float2half_rn(v);
                        img[((size_t)(c / 8) * 32 + col) * 8 + (c % 8)] = hv;
                        img[((size_t)(c / 8) * 32 + 16 + col) * 8 + (c % 8)] = __float2half_rn(v - __half2float(hv));
                    }
                cudaFree(w.tc_w7); w.tc_w7 = nullptr;
                CIA_CUDA(cudaMalloc(&w.tc_w7, img.size() * sizeof(__half)));
                CIA_CUDA(cudaMemcpy(w.tc_w7, img.data(), img.size() * sizeof(__half), cudaMemcpyHostToDevice));
            }
            w.tc_inv_scale[L] = std::ldexp(1.f, -sw);
            continue;
        } else if (L == 5) {
            // same phase form with all Cout channels: N = 4 phases x Cout, run at the low (input) resolution --
            // 2 tiles x 9 taps instead of 8 tiles x 9 taps of MMAs per cell
            const int N = 4 * cout;
            std::vector<float> kp((size_t)9 * cin * N, 0.f);
            for (int py = 0; py < 2; ++py)
                for (int px = 0; px < 2; ++px)
                    for (int dy = 0; dy < 3; ++dy)
                        for (int dx = 0; dx < 3; ++dx) {
                            const int oy = (int)std::floor((py + dy - 1) / 2.0), ox = (int)std::floor((px + dx - 1) / 2.0);
                            const int tl = (oy + 1) * 3 + (ox + 1);
                            for (int c = 0; c < cin; ++c)
                                for (int co = 0; co < cout; ++co)
                                    kp[((size_t)tl * cin + c) * N + (py * 2 + px) * cout + co] +=
                                        k[((size_t)(dy * 3 + dx) * cin + c) * cout + co];
                        }
            sw = scale_exp(kp);
            pack_image(kp, 9, cin, N, N, sw, hi, lo);
        } else {
            sw = scale_exp(k);
            pack_image(k, 9, cin, cout, cout, sw, hi, lo, L < 3 ? colsign.data() : nullptr);
        }
        w.tc_inv_scale[L] = std::ldexp(1.f, -sw);
        for (int j = 0; j < 2; ++j) {
            cudaFree(w.tc_w[L][j]); w.tc_w[L][j] = nullptr;
            const std::vector<__half>& src = j == 0 ? hi : lo;
            CIA_CUDA(cudaMalloc(&w.tc_w[L][j], src.size() * sizeof(__half)));
            CIA_CUDA(cudaMemcpy(w.tc_w[L][j], src.data(), src.size() * sizeof(__half), cudaMemcpyHostToDevice));
        }
    }
    w.tc_ready = true;
    return CIA_OK;
}

// precision 1: split-precision (3 MMAs) encoder, features tapped from the tensor-core pass.
// precision 2: single-pass tensor-core autoencoder for MSE/MAE; features from the exact fp32
//              encoder (the reference itself runs encoder.predict as a second pass, det:130).
int k_cae_forward_tc(cia_ctx* h, const float* crops, int n, const int32_t* n_dev, float* mse,
                     float* mae, float* features, int mode, cudaStream_t s) {
    if (n <= 0) return CIA_OK;
    const CaeWeights& ae = h->cae[0];
    if (!ae.loaded || ae.n_conv != 7 || !ae.tc_ready) { h->err = "cia_cae_forward: autoencoder not loaded"; return CIA_E_STATE; }
    const bool sep = h->cae[1].loaded;
    const bool tc_feat = mode == 1 && !sep;
    // mode 3: L1 + L2 on tensor cores with split operands, fp32 tap of the 16x16x64 activation,
    // L3 (the layer whose long RZ-accumulated K=576 chains dominate the feature error) in exact fp32
    const bool l3_exact = mode == 3 && !sep;
    // cells per pass over the seven layers.  Measured (profiles/r1_cae_chunk_sweep.txt): every launch
    // pays a fixed prologue (37-147 KB of weights into each CTA's shared memory, TMEM allocation,
    // pipeline fill, a ragged last wave), and keeping a chunk's activations L2-resident buys nothing
    // because the layers are tensor-pipe / issue bound, not DRAM bound: 296 cells/pass -> 67 ms,
    // 1024 -> 49 ms, 16576 (112 per SM) -> 39.6 ms for the same 121k cells.  303 KB of workspace per cell.
    // The cap is 128 cells per SM so that a 32-field chunk (capacity 32 x ~520 labels = 16640 cells) is ONE
    // pass: with 16576 every chunk launched a second, empty pass of all seven kernels.
    const int CH_MAX = h->cae_pass_cells;
    const int CH = n < CH_MAX ? (n + 147) / 148 * 148 : CH_MAX;
    // halves per cell; A4 / A5 are stored at their own (pre-upsampling) resolution
    const size_t a1 = 4 * 32 * 32 * 8, a2 = 8 * 16 * 16 * 8, a3 = 4 * 8 * 8 * 8, a4u = 4 * 8 * 8 * 8,
                 a5u = 8 * 16 * 16 * 8, a6 = 4 * 32 * 32 * 8;
    const size_t per_cell = 2 * a1 + 2 * a2 + a3 + a4u + a5u + a6;     // halves
    int rc = ws_reserve(h, h->ws_misc, (size_t)CH * per_cell * sizeof(__half));
    if (rc) return rc;
    float* A2f = nullptr;
    if (l3_exact) {
        if ((rc = ws_reserve(h, h->ws_act, (size_t)CH * 16 * 16 * 64 * sizeof(float)))) return rc;
        A2f = (float*)h->ws_act.p;
    }
    __half* A1h = (__half*)h->ws_misc.p;
    __half* A1l = A1h + CH * a1;
    __half* A2h = A1l + CH * a1;
    __half* A2l = A2h + CH * a2;
    __half* A3h = A2l + CH * a2;
    __half* A4u = A3h + CH * a3;
    __half* A5u = A4u + CH * a4u;
    __half* A6 = A5u + CH * a5u;
    CIA_CUDA(cudaMemsetAsync(mse, 0, (size_t)n * sizeof(float), s));
    CIA_CUDA(cudaMemsetAsync(mae, 0, (size_t)n * sizeof(float), s));
    const bool side_encoder = features && !tc_feat && !l3_exact;
    if (side_encoder) {
        // fork: encoder.predict (det:130) in exact fp32 on the side stream, concurrently with
        // autoencoder.predict (det:125) on the tensor cores
        CIA_CUDA(cudaEventRecord(h->ev_fork, s));
        CIA_CUDA(cudaStreamWaitEvent(h->side, h->ev_fork, 0));
        rc = k_encoder_fp32(h, sep ? h->cae[1] : h->cae[0], crops, n, n_dev, features, h->side);
        if (rc) return rc;
        CIA_CUDA(cudaEventRecord(h->ev_join, h->side));
    }
    for (int c0 = 0; c0 < n; c0 += CH) {
        const int chunk = (n - c0) < CH ? (n - c0) : CH;
        // activation buffers are chunk-relative; kernels index by absolute cell
        __half* a1h = A1h - (size_t)c0 * a1; __half* a1l = A1l - (size_t)c0 * a1;
        __half* a2h = A2h - (size_t)c0 * a2; __half* a2l = A2l - (size_t)c0 * a2;
        __half* a3h = A3h - (size_t)c0 * a3; __half* a4 = A4u - (size_t)c0 * a4u;
        __half* a5 = A5u - (size_t)c0 * a5u; __half* a6p = A6 - (size_t)c0 * a6;
        float* feat = tc_feat ? features : nullptr;
        int grid1 = chunk * 4;
        if (grid1 > h->num_sms * 8) grid1 = h->num_sms * 8;
        // per-layer event marks of every pass (cia_profile_layers): L1..L7 boundaries
        const int pass = c0 / CH;
        if (h->layer_ev && pass < CIA_LAYER_PASSES) h->layer_passes = pass + 1;
#define CIA_LMARK(i) do { if (h->layer_ev && pass < CIA_LAYER_PASSES) CIA_CUDA(cudaEventRecord(h->layer_ev[pass * CIA_LAYER_MARKS + (i)], s)); } while (0)
        CIA_LMARK(0);
        if (tc_feat || l3_exact) {
            // the half-ulp truncation compensation of layer 1's single accumulation: cia_set_option "cae_l1_debias"
            const float l1_debias = h->cae_debias[0] * 5.9604645e-8f;
            if (first_use(h, (const void*)conv1_tc_split_kernel))
                CIA_CUDA(cudaFuncSetAttribute(conv1_tc_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, l1tc::SMEM_B));
            int gridt = chunk * 8;
            if (gridt > h->num_sms * 2) gridt = h->num_sms * 2;
            conv1_tc_split_kernel<<<gridt, l1tc::NT, l1tc::SMEM_B, s>>>(crops, (const uint4*)ae.tc_w[0][0], ae.tc_inv_scale[0],
                                                                        l1_debias, ae.bias[0], ae.bn_scale[0], ae.bn_shift[0],
                                                                        a1h, a1l, n, n_dev, c0, chunk, h->status_dev);
            CIA_LAUNCH_CHECK();
            CIA_LMARK(1);
            float* a2f = l3_exact ? A2f - (size_t)c0 * (16 * 16 * 64) : nullptr;
            // three taps per TMEM flush of layer 2 keep the epilogue warps below the tensor pipe's time.  An N-stacked
            // variant (hi x [hi|lo] as one N = 128 instruction: 112 instead of 145 pipe cycles per k-step by
            // profiles/umma_microbench.cu) was built and measured in round 2: 53.3 vs 51.5 ms -- its flushes double
            // (main + cross column groups) and the drain of a two-tile stage no longer hides under the other stage's
            // MMAs (DESIGN.md 5)
            if ((rc = launch_tc_acc2<32, 64, 32, 3>(h, ae, 1, A1h, A1l, CH, a2h, a2l, a2f, n, n_dev, c0, chunk, s))) return rc;
            CIA_LMARK(2);
            if (l3_exact) {
                if ((rc = launch_tc<64, 32, 16, EPI_POOL, 1>(h, ae, 2, a2h, nullptr, a3h, nullptr, nullptr, n, n_dev, c0, chunk, s))) return rc;
                if (features && (rc = k_conv3_fp32(h, ae, a2f, n, n_dev, features, c0, chunk, s))) return rc;
            } else {
                // Measured and dropped (DESIGN.md section 5): a TMA-fed L3 with one input buffer refilled the moment the
                // cell's last MMAs complete (cae 75.6 vs 74.0 ms per 242k cells), three taps per flush (no gain), the
                // input block through cp.async (27.3 vs 23.7 ms), four TMEM stages with the MMAs of two flush groups
                // interleaved (23.8 vs 22.1 ms)
                if ((rc = launch_tc_acc<64, 32, 16, 1>(h, ae, 2, a2h, a2l, a3h, nullptr, feat, n, n_dev, c0, chunk, s))) return rc;
            }
        } else {
            conv1_fp32_planar_kernel<<<grid1, 256, 0, s>>>(crops, ae.kernel[0], ae.bias[0], ae.bn_scale[0],
                                                           ae.bn_shift[0], a1h, n, n_dev, c0, chunk, h->status_dev);
            CIA_LAUNCH_CHECK();
            CIA_LMARK(1);
            if ((rc = launch_tc<32, 64, 32, EPI_POOL, 1>(h, ae, 1, a1h, nullptr, a2h, nullptr, nullptr, n, n_dev, c0, chunk, s))) return rc;
            CIA_LMARK(2);
            if ((rc = launch_tc<64, 32, 16, EPI_POOL, 1>(h, ae, 2, a2h, nullptr, a3h, nullptr, nullptr, n, n_dev, c0, chunk, s))) return rc;
        }
        CIA_LMARK(3);
        if ((rc = launch_tc<32, 32, 8, EPI_PLAIN, 1>(h, ae, 3, a3h, nullptr, a4, nullptr, nullptr, n, n_dev, c0, chunk, s))) return rc;
        CIA_LMARK(4);
        if ((rc = launch_tc<32, 64, 16, EPI_PLAIN, 1, true>(h, ae, 4, a4, nullptr, a5, nullptr, nullptr, n, n_dev, c0, chunk, s))) return rc;
        CIA_LMARK(5);
        if ((rc = launch_tc<64, 128, 16, EPI_PHASE, 1>(h, ae, 5, a5, nullptr, a6p, nullptr, nullptr, n, n_dev, c0, chunk, s))) return rc;
        CIA_LMARK(6);
        if (first_use(h, (const void*)final_tapsum_kernel))
            CIA_CUDA(cudaFuncSetAttribute(final_tapsum_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, l7::SMEM_B));
        int g7 = chunk < h->num_sms ? chunk : h->num_sms;
        final_tapsum_kernel<<<g7, l7::NT, l7::SMEM_B, s>>>(a6p, (const uint4*)ae.tc_w7, ae.tc_inv_scale[6], ae.bias[6],
                                                          crops, mse, mae, n, n_dev, c0, chunk);
        CIA_LAUNCH_CHECK();
        CIA_LMARK(7);
#undef CIA_LMARK
    }
    if (side_encoder) CIA_CUDA(cudaStreamWaitEvent(s, h->ev_join, 0));
    return CIA_OK;
}
