// tiff_dev.cu -- device decode of compressed TIFF fields (SURVEY 8f row N1): the strips / tiles of a chunk of
// fields are independent streams, so one launch decodes all of them, one warp per segment.  Lane 0 runs the serial
// decoder of tiff_decode.h (Deflate, LZW, PackBits or Zstandard) into the caller's scratch with its tables and the
// Deflate window in shared memory; then the warp undoes horizontal differencing along each row with a shuffle scan,
// swaps big-endian samples, widens 8-bit samples and writes the segment's rectangle (cropped at the field's edges)
// into the uint16 planes that cia_screen_images reads.
#include "common.cuh"
#include "tiff_decode.h"

namespace {

constexpr int kStatusCorrupt = 1, kStatusShort = 2, kStatusBadSegment = 4;
constexpr int kMaxSide = 1 << 20, kMaxSamples = 16;   // per segment: rows, cols / interleaved samples

__device__ __forceinline__ uint32_t load_sample(const uint8_t* row, int x, int samples, int s, int bps, int big) {
    if (bps == 1) return row[(size_t)x * samples + s];
    const uint8_t* p = row + ((size_t)x * samples + s) * 2;
    return big ? ((uint32_t)p[0] << 8 | p[1]) : ((uint32_t)p[1] << 8 | p[0]);
}

__global__ void __launch_bounds__(32) tiff_decode_kernel(const uint8_t* __restrict__ src, size_t src_bytes,
                                                         const cia_tiff_segment* __restrict__ segs, int n_fields,
                                                         int H, int W, uint8_t* __restrict__ scratch,
                                                         size_t scratch_bytes, uint16_t* __restrict__ seg_out,
                                                         uint16_t* __restrict__ img_out, int32_t* status) {
    __shared__ union {
        TdInflateWork inflate;
        TdLzwWork lzw;
        TdZstdWork zstd;
    } work;
    __shared__ long long produced;
    const int lane = threadIdx.x;
    const cia_tiff_segment g = segs[blockIdx.x];
    const bool field_ok = g.field >= 0 && g.field < n_fields;
    const int bps = g.bytes_per_sample;
    // sides and samples are bounded before they are multiplied, so `need` cannot wrap
    bool ok = field_ok && g.rows > 0 && g.rows <= kMaxSide && g.cols > 0 && g.cols <= kMaxSide && g.samples > 0 &&
              g.samples <= kMaxSamples && (bps == 1 || bps == 2) &&
              g.seg_sample < g.samples && g.img_sample < g.samples && (g.predictor == 1 || g.predictor == 2) &&
              g.y0 >= 0 && g.x0 >= 0;
    const size_t need = (size_t)g.rows * (size_t)g.cols * (size_t)g.samples * (size_t)bps;
    ok = ok && g.src_off <= src_bytes && g.src_len <= src_bytes - g.src_off && g.dst_off <= scratch_bytes &&
         need <= scratch_bytes - g.dst_off;
    if (!ok) {
        if (lane == 0 && field_ok) atomicOr(status + g.field, kStatusBadSegment);   // no field to flag otherwise
        return;
    }
    uint8_t* d = scratch + g.dst_off;
    if (lane == 0) {
        const uint8_t* s = src + g.src_off;
        long long n;
        switch (g.compression) {
            case 1: n = td_copy(s, g.src_len, d, need); break;
            case 5: n = td_lzw(s, g.src_len, d, need, &work.lzw); break;
            case 8: case 32946: n = td_inflate(s, g.src_len, d, need, &work.inflate); break;
            case 32773: n = td_packbits(s, g.src_len, d, need); break;
            case 50000: case 34926: n = td_zstd(s, g.src_len, d, need, &work.zstd); break;
            default: n = -1;
        }
        produced = n;
        if (n < 0 || (size_t)n < need) atomicOr(status + g.field, n < 0 ? kStatusCorrupt : kStatusShort);
    }
    __syncwarp();
    const long long n = produced;
    for (size_t i = (size_t)(n > 0 ? n : 0) + lane; i < need; i += 32) d[i] = 0;   // nothing stale survives
    __syncwarp();
    if (g.y0 >= H || g.x0 >= W) return;
    const int ys = min(g.rows, H - g.y0), xs = min(g.cols, W - g.x0);
    const size_t row_bytes = (size_t)g.cols * g.samples * bps;
    const uint32_t mask = bps == 1 ? 0xffu : 0xffffu;
    const size_t plane = (size_t)g.field * H * W;
    for (int pass = 0; pass < 2; ++pass) {
        // pass 0: the analysis sample (and the segmentation sample when it is the same one), pass 1: the other
        const int s = pass == 0 ? g.img_sample : g.seg_sample;
        uint16_t* o0 = pass == 0 ? img_out : seg_out;
        uint16_t* o1 = pass == 0 && seg_out && g.seg_sample == g.img_sample ? seg_out : nullptr;
        if (s < 0 || !o0 || (pass == 1 && g.seg_sample == g.img_sample)) continue;
        for (int r = 0; r < ys; ++r) {
            const uint8_t* row = d + (size_t)r * row_bytes;
            const size_t orow = plane + (size_t)(g.y0 + r) * W + g.x0;
            uint32_t carry = 0;
            for (int x0 = 0; x0 < xs; x0 += 32) {
                const int x = x0 + lane;
                uint32_t v = x < xs ? load_sample(row, x, g.samples, s, bps, g.big_endian) : 0;
                if (g.predictor == 2) {
#pragma unroll
                    for (int k = 1; k < 32; k <<= 1) {
                        const uint32_t t = __shfl_up_sync(0xffffffffu, v, k);
                        if (lane >= k) v += t;
                    }
                    v = (v + carry) & mask;
                    carry = __shfl_sync(0xffffffffu, v, 31);
                }
                if (x < xs) {
                    o0[orow + x] = (uint16_t)v;
                    if (o1) o1[orow + x] = (uint16_t)v;
                }
            }
        }
    }
}

}  // namespace

extern "C" {

int cia_tiff_decode_fields(cia_handle h, const uint8_t* src, size_t src_bytes, const cia_tiff_segment* segs,
                           int n_segs, int n_fields, int H, int W, uint8_t* scratch, size_t scratch_bytes,
                           uint16_t* seg_out, uint16_t* img_out, int32_t* field_status, void* stream) {
    if (!h) return CIA_E_ARG;
    if (n_segs < 0 || n_fields <= 0 || H <= 0 || W <= 0 || !img_out || !field_status ||
        (n_segs > 0 && (!src || !segs || !scratch))) {
        h->err = "cia_tiff_decode_fields: bad argument";
        return CIA_E_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    CIA_CUDA(cudaMemsetAsync(field_status, 0, sizeof(int32_t) * (size_t)n_fields, s));
    if (n_segs == 0) return CIA_OK;
    tiff_decode_kernel<<<n_segs, 32, 0, s>>>(src, src_bytes, segs, n_fields, H, W, scratch, scratch_bytes, seg_out,
                                             img_out, field_status);
    CIA_LAUNCH_CHECK();
    return CIA_OK;
}

}  // extern "C"
