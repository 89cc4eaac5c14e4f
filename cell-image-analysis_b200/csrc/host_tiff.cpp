// host_tiff.cpp -- host-side TIFF strip / tile decompressors behind tiff_min.read_tiff (the reader
// standing in for tiff.imread, improved_detection.py:51): LZW (TIFF 6.0 section 13, MSB-first codes,
// "early change") and PackBits.  Plain C++, no CUDA; exported through the C-ABI so that the Python
// reader does not decode 8 MB fields byte by byte in the interpreter.  Deflate is zlib's (Python).  Zstandard is
// td_zstd of tiff_decode.h, the decoder the device runs, compiled for the host.
#include <stddef.h>
#include <stdint.h>
#include <memory>
#include <vector>

#include "tiff_decode.h"

extern "C" {

// Returns the number of bytes written to dst (<= cap), or -1 on a corrupt stream.
long long cia_tiff_lzw_decode(const uint8_t* src, size_t n, uint8_t* dst, size_t cap) {
    if (!src || !dst) return -1;
    struct Entry { int32_t prev; uint8_t ch; uint8_t first; uint16_t len; };
    std::vector<Entry> tab(4096 + 2);
    for (int i = 0; i < 256; ++i) tab[i] = {-1, (uint8_t)i, (uint8_t)i, 1};
    const int CLEAR = 256, EOI = 257;
    int next = 258, bits = 9, old = -1;
    uint64_t acc = 0;
    int have = 0;
    size_t ip = 0, op = 0;
    for (;;) {
        while (have < bits && ip < n) { acc = (acc << 8) | src[ip++]; have += 8; }
        if (have < bits) break;                               // stream ended without EOI: accept what we have
        const int code = (int)((acc >> (have - bits)) & ((1u << bits) - 1));
        have -= bits;
        if (code == EOI) break;
        if (code == CLEAR) { next = 258; bits = 9; old = -1; continue; }
        if (old < 0) {                                        // first code after a clear: a literal
            if (code >= 256) return -1;
            if (op < cap) dst[op] = (uint8_t)code;
            ++op; old = code;
            continue;
        }
        int emit = code;
        uint8_t tail_ch = 0;
        bool kwk = false;
        if (code >= next) {                                   // KwKwK: string(old) + first(string(old))
            if (code != next) return -1;
            emit = old; kwk = true; tail_ch = tab[old].first;
        }
        const int len = tab[emit].len + (kwk ? 1 : 0);
        if (op + (size_t)len <= cap) {
            size_t w = op + (size_t)tab[emit].len;
            for (int c = emit; c >= 0; c = tab[c].prev) dst[--w] = tab[c].ch;
            if (kwk) dst[op + (size_t)len - 1] = tail_ch;
        } else {                                              // partial tail: slow path with bounds checks
            std::vector<uint8_t> tmp((size_t)len);
            size_t w = (size_t)tab[emit].len;
            for (int c = emit; c >= 0; c = tab[c].prev) tmp[--w] = tab[c].ch;
            if (kwk) tmp[(size_t)len - 1] = tail_ch;
            for (int i = 0; i < len && op + (size_t)i < cap; ++i) dst[op + (size_t)i] = tmp[(size_t)i];
        }
        op += (size_t)len;
        if (next < 4096) {
            tab[next] = {old, kwk ? tail_ch : tab[code].first, tab[old].first, (uint16_t)(tab[old].len + 1)};
            ++next;
            if (next + 1 >= (1 << bits) && bits < 12) ++bits;   // "early change": widen one code early
        }
        old = code;
        if (op >= cap) break;
    }
    return (long long)(op < cap ? op : cap);
}

long long cia_tiff_packbits_decode(const uint8_t* src, size_t n, uint8_t* dst, size_t cap) {
    if (!src || !dst) return -1;
    size_t ip = 0, op = 0;
    while (ip < n && op < cap) {
        const int8_t h = (int8_t)src[ip++];
        if (h >= 0) {
            const size_t k = (size_t)h + 1;
            for (size_t i = 0; i < k && ip < n && op < cap; ++i) dst[op++] = src[ip++];
        } else if (h != -128) {
            if (ip >= n) return -1;
            const uint8_t v = src[ip++];
            for (size_t i = 0, k = (size_t)(1 - h); i < k && op < cap; ++i) dst[op++] = v;
        }
    }
    return (long long)op;
}

// Zstandard frames (RFC 8878) with the contract of cia_tiff_lzw_decode: output clipped at cap, -1 on a corrupt stream.
long long cia_tiff_zstd_decode(const uint8_t* src, size_t n, uint8_t* dst, size_t cap) {
    if (!src || !dst) return -1;
    std::unique_ptr<TdZstdWork> w(new TdZstdWork);
    return td_zstd(src, n, dst, cap, w.get());
}

}  // extern "C"
