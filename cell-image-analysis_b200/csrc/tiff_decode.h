// tiff_decode.h -- TIFF strip / tile decompressors as __host__ __device__ functions: zlib-wrapped Deflate
// (RFC 1950 / 1951), TIFF LZW and PackBits.  csrc/tiff_dev.cu runs them on the device, one segment per warp;
// tests/host_fuzz/fuzz_tiff_decode.cpp compiles the same code for the host under AddressSanitizer + UBSan.
//
// Every decoder reads only src[0, n) and writes only dst[0, cap).  Each returns the bytes written (<= cap) or -1
// on a stream the host reader refuses:
//   td_inflate  accepts and refuses exactly what Python's zlib.decompress (wbits 15) does: bad header, preset
//               dictionary, invalid block type / stored length / code sets / codes, a distance before the first
//               output byte, a truncated stream and a wrong Adler-32 are refused; bytes after the Adler-32 are
//               ignored.  Output past cap is decoded into a 32 KB window (back references and the checksum need it)
//               and dropped, like zlib.decompress(data)[:cap].
//   td_lzw      MSB-first codes with early change; clipping and refusals exactly as cia_tiff_lzw_decode
//               (csrc/host_tiff.cpp).  Table entries are (offset, length) of a substring of the output already
//               written, so the table is 24 KB and a string is one forward copy.
//   td_packbits exactly cia_tiff_packbits_decode.
#pragma once
#include <stddef.h>
#include <stdint.h>

#ifdef __CUDACC__
#define TD_FN __host__ __device__ inline
#else
#define TD_FN inline
#endif

#define TD_FAST 10               // bits of the one-lookup Huffman table; longer codes take the canonical walk
#define TD_WINDOW 32768

struct TdHuff {
    uint16_t fast[1 << TD_FAST];  // (length << 9) | symbol, 0: no code of <= TD_FAST bits has these bits
    int16_t count[16];            // codes per length
    int16_t sym[288];             // symbols in canonical order
};

struct TdInflateWork {            // 38 KB: shared memory of one warp on the device
    TdHuff lit, dist;
    uint8_t lens[320];
    uint8_t win[TD_WINDOW];       // output bytes at positions >= cap
};

struct TdLzwWork {                // 24 KB
    uint32_t pos[4096];
    uint16_t len[4096];
};

struct TdBits {
    const uint8_t* p;
    size_t n, i;
    uint64_t buf;
    int cnt;
};

TD_FN void td_fill(TdBits& s) {
    while (s.cnt <= 56 && s.i < s.n) { s.buf |= (uint64_t)s.p[s.i++] << s.cnt; s.cnt += 8; }
}

// k <= 16 bits, LSB first; false when the stream ends first
TD_FN bool td_get(TdBits& s, int k, uint32_t& v) {
    if (s.cnt < k) td_fill(s);
    if (s.cnt < k) return false;
    v = (uint32_t)(s.buf & ((1u << k) - 1));
    s.buf >>= k;
    s.cnt -= k;
    return true;
}

// zlib's inflate_table rules: over-subscribed sets are refused; incomplete sets only as a single one-bit code of a
// literal / length or distance set.  A set with no codes at all is accepted (any use of it is an invalid code),
// except for the code-length code, where zlib's outcome is always an error and it is refused here at once.
TD_FN bool td_build(TdHuff& h, const uint8_t* lens, int n, bool code_lengths) {
    for (int l = 0; l < 16; ++l) h.count[l] = 0;
    for (int s = 0; s < n; ++s) h.count[lens[s]]++;
    for (int i = 0; i < (1 << TD_FAST); ++i) h.fast[i] = 0;
    int max = 0;
    for (int l = 1; l < 16; ++l) if (h.count[l]) max = l;
    h.count[0] = 0;
    if (max == 0) return !code_lengths;
    int left = 1;
    for (int l = 1; l < 16; ++l) {
        left <<= 1;
        left -= h.count[l];
        if (left < 0) return false;
    }
    if (left > 0 && (code_lengths || max != 1)) return false;
    int16_t offs[16];
    offs[1] = 0;
    for (int l = 1; l < 15; ++l) offs[l + 1] = (int16_t)(offs[l] + h.count[l]);
    for (int s = 0; s < n; ++s) if (lens[s]) h.sym[offs[lens[s]]++] = (int16_t)s;
    int code = 0, k = 0;
    for (int l = 1; l <= TD_FAST; ++l) {
        for (int j = 0; j < h.count[l]; ++j, ++k, ++code) {
            int rev = 0;
            for (int b = 0; b < l; ++b) rev |= ((code >> b) & 1) << (l - 1 - b);
            for (int e = rev; e < (1 << TD_FAST); e += 1 << l) h.fast[e] = (uint16_t)((l << 9) | h.sym[k]);
        }
        code <<= 1;
    }
    return true;
}

// one symbol, -1 on an invalid code or the end of the stream
TD_FN int td_decode(TdBits& s, const TdHuff& h) {
    if (s.cnt < 15) td_fill(s);
    const uint32_t e = h.fast[s.buf & ((1u << TD_FAST) - 1)];
    if (e && (int)(e >> 9) <= s.cnt) {
        s.buf >>= e >> 9;
        s.cnt -= (int)(e >> 9);
        return (int)(e & 511);
    }
    int code = 0, first = 0, index = 0;           // canonical walk (puff)
    for (int l = 1; l < 16; ++l) {
        if (l > s.cnt) return -1;
        code |= (int)((s.buf >> (l - 1)) & 1);
        const int count = h.count[l];
        if (code - count < first) {
            s.buf >>= l;
            s.cnt -= l;
            return h.sym[index + (code - first)];
        }
        index += count;
        first += count;
        first <<= 1;
        code <<= 1;
    }
    return -1;
}

struct TdOut {
    uint8_t* dst;
    size_t cap, op;
    uint8_t* win;
    uint32_t a, b, run;           // Adler-32 with the modulo deferred over 5552 bytes
};

TD_FN void td_put(TdOut& o, uint8_t v) {
    if (o.op < o.cap) o.dst[o.op] = v;
    else o.win[o.op & (TD_WINDOW - 1)] = v;
    ++o.op;
    o.a += v;
    o.b += o.a;
    if (++o.run == 5552) { o.a %= 65521u; o.b %= 65521u; o.run = 0; }
}

TD_FN uint8_t td_at(const TdOut& o, size_t q) { return q < o.cap ? o.dst[q] : o.win[q & (TD_WINDOW - 1)]; }

TD_FN long long td_inflate(const uint8_t* src, size_t n, uint8_t* dst, size_t cap, TdInflateWork* w) {
    TdBits s{src, n, 0, 0, 0};
    TdOut o{dst, cap, 0, w->win, 1, 0, 0};
    uint32_t cmf, flg;
    if (!td_get(s, 8, cmf) || !td_get(s, 8, flg)) return -1;
    if (((cmf << 8) | flg) % 31 || (cmf & 15) != 8 || (cmf >> 4) + 8 > 15 || (flg & 0x20)) return -1;
    const char* order = "\x10\x11\x12\x00\x08\x07\x09\x06\x0a\x05\x0b\x04\x0c\x03\x0d\x02\x0e\x01\x0f";
    uint32_t last = 0;
    do {
        uint32_t type;
        if (!td_get(s, 1, last) || !td_get(s, 2, type)) return -1;
        if (type == 0) {                          // stored
            const int drop = s.cnt & 7;
            s.buf >>= drop;
            s.cnt -= drop;
            uint32_t len, nlen;
            if (!td_get(s, 16, len) || !td_get(s, 16, nlen) || len != (nlen ^ 0xffffu)) return -1;
            for (uint32_t i = 0; i < len; ++i) {
                uint32_t v;
                if (!td_get(s, 8, v)) return -1;
                td_put(o, (uint8_t)v);
            }
            continue;
        }
        if (type == 3) return -1;
        if (type == 1) {                          // fixed codes (286, 287, 30 and 31 decode but are invalid)
            for (int i = 0; i < 288; ++i) w->lens[i] = (uint8_t)(i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8);
            td_build(w->lit, w->lens, 288, false);
            for (int i = 0; i < 32; ++i) w->lens[i] = 5;
            td_build(w->dist, w->lens, 32, false);
        } else {                                  // dynamic codes
            uint32_t hlit, hdist, hclen;
            if (!td_get(s, 5, hlit) || !td_get(s, 5, hdist) || !td_get(s, 4, hclen)) return -1;
            const int nlen = (int)hlit + 257, ndist = (int)hdist + 1, ncode = (int)hclen + 4;
            if (nlen > 286 || ndist > 30) return -1;
            for (int i = 0; i < 19; ++i) w->lens[(int)order[i]] = 0;
            for (int i = 0; i < ncode; ++i) {
                uint32_t v;
                if (!td_get(s, 3, v)) return -1;
                w->lens[(int)order[i]] = (uint8_t)v;
            }
            if (!td_build(w->lit, w->lens, 19, true)) return -1;
            int have = 0;
            while (have < nlen + ndist) {
                const int sym = td_decode(s, w->lit);
                if (sym < 0) return -1;
                if (sym < 16) { w->lens[have++] = (uint8_t)sym; continue; }
                uint32_t rep, v = 0;
                if (sym == 16) {
                    if (have == 0 || !td_get(s, 2, rep)) return -1;
                    v = w->lens[have - 1];
                    rep += 3;
                } else if (sym == 17) {
                    if (!td_get(s, 3, rep)) return -1;
                    rep += 3;
                } else {
                    if (!td_get(s, 7, rep)) return -1;
                    rep += 11;
                }
                if (have + (int)rep > nlen + ndist) return -1;
                for (uint32_t r = 0; r < rep; ++r) w->lens[have++] = (uint8_t)v;
            }
            if (w->lens[256] == 0) return -1;
            if (!td_build(w->lit, w->lens, nlen, false)) return -1;
            if (!td_build(w->dist, w->lens + nlen, ndist, false)) return -1;
        }
        for (;;) {
            const int sym = td_decode(s, w->lit);
            if (sym < 0) return -1;
            if (sym < 256) { td_put(o, (uint8_t)sym); continue; }
            if (sym == 256) break;
            const int li = sym - 257;
            if (li > 28) return -1;
            uint32_t len, extra;
            if (li < 8) { len = 3 + li; extra = 0; }
            else if (li == 28) { len = 258; extra = 0; }
            else { extra = (uint32_t)(li - 4) >> 2; len = ((4u + (li & 3)) << extra) + 3; }
            uint32_t v;
            if (extra) { if (!td_get(s, (int)extra, v)) return -1; len += v; }
            const int ds = td_decode(s, w->dist);
            if (ds < 0 || ds > 29) return -1;
            uint32_t dist;
            if (ds < 4) { dist = 1 + ds; extra = 0; }
            else { extra = ((uint32_t)ds >> 1) - 1; dist = ((2u + (ds & 1)) << extra) + 1; }
            if (extra) { if (!td_get(s, (int)extra, v)) return -1; dist += v; }
            if (dist > o.op) return -1;
            if (o.op + len <= o.cap) {            // the common case: source and destination inside dst
                uint8_t* d = o.dst + o.op;
                const uint8_t* q = d - dist;
                for (uint32_t i = 0; i < len; ++i) {
                    const uint8_t c = q[i];
                    d[i] = c;
                    o.a += c;
                    o.b += o.a;
                    if (++o.run == 5552) { o.a %= 65521u; o.b %= 65521u; o.run = 0; }
                }
                o.op += len;
            } else {
                for (uint32_t i = 0; i < len; ++i) td_put(o, td_at(o, o.op - dist));
            }
        }
    } while (!last);
    const int drop = s.cnt & 7;                    // the Adler-32 starts on a byte boundary, big endian
    s.buf >>= drop;
    s.cnt -= drop;
    uint32_t adler = 0;
    for (int i = 0; i < 4; ++i) {
        uint32_t v;
        if (!td_get(s, 8, v)) return -1;
        adler = (adler << 8) | v;
    }
    if (adler != (((o.b % 65521u) << 16) | (o.a % 65521u))) return -1;
    return (long long)(o.op < cap ? o.op : cap);
}

TD_FN long long td_lzw(const uint8_t* src, size_t n, uint8_t* dst, size_t cap, TdLzwWork* t) {
    const int CLEAR = 256, EOI = 257;
    int next = 258, bits = 9, old = -1;
    uint64_t acc = 0;
    int have = 0;
    size_t ip = 0, op = 0, prev_pos = 0, prev_len = 0;   // the previous code's string is dst[prev_pos, +prev_len)
    for (;;) {
        while (have < bits && ip < n) { acc = (acc << 8) | src[ip++]; have += 8; }
        if (have < bits) break;
        const int code = (int)((acc >> (have - bits)) & ((1u << bits) - 1));
        have -= bits;
        if (code == EOI) break;
        if (code == CLEAR) { next = 258; bits = 9; old = -1; continue; }
        if (old < 0) {
            if (code >= 256) return -1;
            if (op < cap) dst[op] = (uint8_t)code;
            prev_pos = op; prev_len = 1;
            ++op; old = code;
            continue;
        }
        size_t len;
        if (code >= next) {                        // KwKwK: string(old) + its first byte, one overlapping copy
            if (code != next) return -1;
            len = prev_len + 1;
            for (size_t i = 0; i < len && op + i < cap; ++i) dst[op + i] = dst[prev_pos + i];
        } else if (code < 256) {
            len = 1;
            if (op < cap) dst[op] = (uint8_t)code;
        } else {
            len = t->len[code];
            const size_t p = t->pos[code];
            for (size_t i = 0; i < len && op + i < cap; ++i) dst[op + i] = dst[p + i];
        }
        if (next < 4096) {                         // string(old) + first byte of this string
            t->pos[next] = (uint32_t)prev_pos;
            t->len[next] = (uint16_t)(prev_len + 1);
            ++next;
            if (next + 1 >= (1 << bits) && bits < 12) ++bits;
        }
        prev_pos = op; prev_len = len;
        op += len;
        old = code;
        if (op >= cap) break;
    }
    return (long long)(op < cap ? op : cap);
}

TD_FN long long td_packbits(const uint8_t* src, size_t n, uint8_t* dst, size_t cap) {
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

// compression 1 (none): the first cap bytes
TD_FN long long td_copy(const uint8_t* src, size_t n, uint8_t* dst, size_t cap) {
    const size_t k = n < cap ? n : cap;
    for (size_t i = 0; i < k; ++i) dst[i] = src[i];
    return (long long)k;
}
