// tiff_decode.h -- TIFF strip / tile decompressors as __host__ __device__ functions: zlib-wrapped Deflate
// (RFC 1950 / 1951), TIFF LZW, PackBits and Zstandard (RFC 8878).  csrc/tiff_dev.cu runs them on the device, one
// segment per warp; csrc/host_tiff.cpp runs td_zstd for the host reader; tests/host_fuzz/fuzz_tiff_decode.cpp and
// fuzz_tiff_zstd.cpp compile the same code for the host under AddressSanitizer + UBSan.
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
//   td_zstd     Zstandard frames (concatenated, skippable ones skipped); a dictionary ID other than 0, a malformed
//               or truncated frame (cut inside a frame: refused, as libzstd does; cut between frames: short), a
//               frame content size or an XXH64 content checksum that does not match are refused.  A frame that
//               declares a content size within cap is decoded and checked completely, and writing past that size
//               refuses it; a frame without one, or with one past cap, stops at cap unchecked, and what follows is
//               ignored.  Stricter than libzstd 1.5 on streams no conforming encoder writes: a non-zero reserved
//               field in the sequence modes byte, bits left over at the end of a sequence or Huffman bitstream and
//               Huffman codes longer than 11 bits (RFC 8878's maximum) are refused.  Matches are copied out of dst
//               itself, so no window is kept.
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

// ---- Zstandard (RFC 8878) ----

struct TdFse {                    // FSE decoding table entry: the symbol; the next state is base + nb bits
    uint16_t base;
    uint8_t nb, sym;
};

struct TdZstdWork {               // 11 KB
    TdFse ll[512], ml[512], of[256];   // sequence tables, kept for the next block's repeat mode
    TdFse wt[64];                 // Huffman weights
    uint16_t huf[2048];           // (bits << 8) | literal, indexed by the next huf_log bits; kept for treeless blocks
    int16_t norm[256];
    uint16_t next[256];
    uint8_t wts[256];
    uint32_t ll_base[36], ml_base[53];
    uint8_t ll_bits[36], ml_bits[53];
};

TD_FN int td_hb(uint32_t x) {     // index of the highest set bit, x > 0
#ifdef __CUDA_ARCH__
    return 31 - __clz(x);
#else
    return 31 - __builtin_clz(x);
#endif
}

TD_FN uint32_t td_le32(const uint8_t* p) {
    return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24;
}

TD_FN uint64_t td_le64(const uint8_t* p) { return td_le32(p) | (uint64_t)td_le32(p + 4) << 32; }

TD_FN uint64_t td_rotl(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }

TD_FN uint64_t td_xxh64(const uint8_t* p, size_t n) {     // seed 0
    const uint64_t P1 = 0x9E3779B185EBCA87ull, P2 = 0xC2B2AE3D27D4EB4Full, P3 = 0x165667B19E3779F9ull,
                   P4 = 0x85EBCA77C2B2AE63ull, P5 = 0x27D4EB2F165667C5ull;
    size_t i = 0;
    uint64_t h;
    if (n >= 32) {
        uint64_t v0 = P1 + P2, v1 = P2, v2 = 0, v3 = 0 - P1;
        for (; i + 32 <= n; i += 32) {
            v0 = td_rotl(v0 + td_le64(p + i) * P2, 31) * P1;
            v1 = td_rotl(v1 + td_le64(p + i + 8) * P2, 31) * P1;
            v2 = td_rotl(v2 + td_le64(p + i + 16) * P2, 31) * P1;
            v3 = td_rotl(v3 + td_le64(p + i + 24) * P2, 31) * P1;
        }
        h = td_rotl(v0, 1) + td_rotl(v1, 7) + td_rotl(v2, 12) + td_rotl(v3, 18);
        h = (h ^ td_rotl(v0 * P2, 31) * P1) * P1 + P4;
        h = (h ^ td_rotl(v1 * P2, 31) * P1) * P1 + P4;
        h = (h ^ td_rotl(v2 * P2, 31) * P1) * P1 + P4;
        h = (h ^ td_rotl(v3 * P2, 31) * P1) * P1 + P4;
    } else {
        h = P5;
    }
    h += n;
    for (; i + 8 <= n; i += 8) h = td_rotl(h ^ td_rotl(td_le64(p + i) * P2, 31) * P1, 27) * P1 + P4;
    if (i + 4 <= n) {
        h = td_rotl(h ^ td_le32(p + i) * P1, 23) * P2 + P3;
        i += 4;
    }
    for (; i < n; ++i) h = td_rotl(h ^ p[i] * P5, 11) * P1;
    h ^= h >> 33;
    h *= P2;
    h ^= h >> 29;
    h *= P3;
    return h ^ (h >> 32);
}

// at least 25 bits from bit `bit` on, LSB first; bytes past n read as 0
TD_FN uint32_t td_peek_fwd(const uint8_t* p, size_t n, size_t bit) {
    uint32_t v = 0;
    const size_t b = bit >> 3;
    for (int k = 0; k < 4; ++k) if (b + k < n) v |= (uint32_t)p[b + k] << (8 * k);
    return v >> (bit & 7);
}

// FSE table description (RFC 8878 4.1.1) -> norm[0, nsym), log.  Returns the bytes it takes or -1.
TD_FN long long td_fse_header(const uint8_t* p, size_t n, int max_sym, int max_log, int16_t* norm, int& nsym,
                              int& log) {
    log = (int)(td_peek_fwd(p, n, 0) & 15) + 5;
    if (n == 0 || log > max_log) return -1;
    size_t bit = 4;
    int remaining = (1 << log) + 1, threshold = 1 << log, nb = log + 1, s = 0;
    bool prev0 = false;
    for (;;) {
        if (prev0) {                               // 2-bit repeat flags of zero counts, 3 means another flag
            uint32_t r;
            do {
                r = td_peek_fwd(p, n, bit) & 3;
                bit += 2;
                for (uint32_t k = 0; k < r; ++k) {
                    if (s > max_sym) return -1;
                    norm[s++] = 0;
                }
            } while (r == 3);
            if (s > max_sym) return -1;
        }
        const uint32_t v = td_peek_fwd(p, n, bit);
        const int mx = 2 * threshold - 1 - remaining;
        int count;
        if ((int)(v & (uint32_t)(threshold - 1)) < mx) {
            count = (int)(v & (uint32_t)(threshold - 1));
            bit += nb - 1;
        } else {
            count = (int)(v & (uint32_t)(2 * threshold - 1));
            if (count >= threshold) count -= mx;
            bit += nb;
        }
        --count;                                   // -1: a "less than 1" probability
        remaining -= count < 0 ? -count : count;
        norm[s++] = (int16_t)count;
        prev0 = count == 0;
        if (remaining <= 1) break;
        while (remaining < threshold) { --nb; threshold >>= 1; }
        if (s > max_sym) break;
    }
    if (remaining != 1 || bit > 8 * n) return -1;
    nsym = s;
    return (long long)((bit + 7) >> 3);
}

TD_FN bool td_fse_build(TdFse* t, const int16_t* norm, int nsym, int log, uint16_t* next) {
    const int size = 1 << log, mask = size - 1, step = (size >> 1) + (size >> 3) + 3;
    int high = size - 1;
    for (int s = 0; s < nsym; ++s) {
        if (norm[s] == -1) {
            t[high--].sym = (uint8_t)s;
            next[s] = 1;
        } else {
            next[s] = (uint16_t)norm[s];
        }
    }
    int pos = 0;
    for (int s = 0; s < nsym; ++s) {
        for (int i = 0; i < norm[s]; ++i) {
            t[pos].sym = (uint8_t)s;
            do pos = (pos + step) & mask; while (pos > high);
        }
    }
    if (pos != 0) return false;
    for (int u = 0; u < size; ++u) {
        const uint32_t x = next[t[u].sym]++;
        const int nb = log - td_hb(x);
        t[u].nb = (uint8_t)nb;
        t[u].base = (uint16_t)((x << nb) - (uint32_t)size);
    }
    return true;
}

// Backward bitstream: read from the end towards the start, the last byte's highest set bit marks the end.
struct TdRev {
    const uint8_t* p;
    size_t n;
    long long pos;                // bits [0, pos) are unread; < 0: read past the start
    long long base;               // c holds bits [base, base + 64)
    uint64_t c;
};

TD_FN void td_rev_load(TdRev& r) {
    long long lo = ((r.pos + 7) >> 3) - 8;
    if (lo < 0) lo = 0;
    uint64_t c = 0;
    for (int k = 7; k >= 0; --k) {
        c <<= 8;
        if ((size_t)lo + k < r.n) c |= r.p[lo + k];
    }
    r.c = c;
    r.base = lo * 8;
}

TD_FN bool td_rev_init(TdRev& r, const uint8_t* p, size_t n) {
    if (n == 0 || p[n - 1] == 0) return false;
    r.p = p;
    r.n = n;
    r.pos = (long long)(n - 1) * 8 + td_hb(p[n - 1]);
    td_rev_load(r);
    return true;
}

// the next k <= 32 bits, bits before the start read as 0
TD_FN uint32_t td_rev_peek(TdRev& r, int k) {
    if (k == 0) return 0;                          // (c >> 64 when 64 bits are left)
    if (r.pos - r.base < k && r.base > 0) td_rev_load(r);
    const long long sh = r.pos - k - r.base;
    const uint64_t v = sh >= 0 ? r.c >> sh : (sh <= -64 ? 0 : r.c << -sh);
    return (uint32_t)(v & ((1ull << k) - 1));
}

TD_FN uint32_t td_rev_get(TdRev& r, int k) {
    const uint32_t v = td_rev_peek(r, k);
    r.pos -= k;
    return v;
}

// Huffman tree description (RFC 8878 4.2.1) -> w->huf.  Returns the bytes it takes or -1.
TD_FN long long td_huf_header(const uint8_t* p, size_t n, TdZstdWork* w, int& huf_log) {
    if (n == 0) return -1;
    int nw = 0;
    size_t used;
    if (p[0] < 128) {                              // FSE-compressed weights, two interleaved states
        used = 1 + (size_t)p[0];
        if (p[0] == 0 || used > n) return -1;
        int nsym, log;
        const long long h = td_fse_header(p + 1, p[0], 255, 6, w->norm, nsym, log);
        if (h < 0 || !td_fse_build(w->wt, w->norm, nsym, log, w->next)) return -1;
        TdRev r;
        if (!td_rev_init(r, p + 1 + h, (size_t)p[0] - (size_t)h)) return -1;
        uint32_t s1 = td_rev_get(r, log), s2 = td_rev_get(r, log);
        for (;;) {                                 // until a state update reads past the start
            if (nw > 253) return -1;
            w->wts[nw++] = w->wt[s1].sym;
            s1 = w->wt[s1].base + td_rev_get(r, w->wt[s1].nb);
            if (r.pos < 0) { w->wts[nw++] = w->wt[s2].sym; break; }
            if (nw > 253) return -1;
            w->wts[nw++] = w->wt[s2].sym;
            s2 = w->wt[s2].base + td_rev_get(r, w->wt[s2].nb);
            if (r.pos < 0) { w->wts[nw++] = w->wt[s1].sym; break; }
        }
    } else {                                       // 4-bit weights
        nw = p[0] - 127;
        used = 1 + (size_t)(nw + 1) / 2;
        if (used > n) return -1;
        for (int i = 0; i < nw; ++i) w->wts[i] = (uint8_t)(i & 1 ? p[1 + i / 2] & 15 : p[1 + i / 2] >> 4);
    }
    uint32_t total = 0;
    for (int i = 0; i < nw; ++i) {
        if (w->wts[i] > 11) return -1;
        if (w->wts[i]) total += 1u << (w->wts[i] - 1);
    }
    if (total == 0) return -1;
    const int L = td_hb(total) + 1;                // the last weight completes the code to 2^L
    const uint32_t rest = (1u << L) - total;
    if (L > 11 || (rest & (rest - 1))) return -1;
    w->wts[nw++] = (uint8_t)(td_hb(rest) + 1);
    int ones = 0;
    for (int i = 0; i < nw; ++i) ones += w->wts[i] == 1;
    if (ones < 2 || (ones & 1)) return -1;
    uint32_t pos = 0;                              // codes by increasing weight, then by literal
    for (int wv = 1; wv <= L; ++wv) {
        for (int s = 0; s < nw; ++s) {
            if (w->wts[s] != wv) continue;
            const uint16_t e = (uint16_t)(((L + 1 - wv) << 8) | s);
            for (uint32_t k = 0; k < (1u << (wv - 1)); ++k) w->huf[pos++] = e;
        }
    }
    huf_log = L;
    return (long long)used;
}

// the literals of one compressed block: raw bytes, one repeated byte, or 1 / 4 Huffman streams decoded as used
struct TdLit {
    const uint8_t* p;
    uint32_t size, done;          // literals of the block, literals used
    int type;                     // 0 raw, 1 RLE, 2 Huffman
    int streams, cur, log;
    uint32_t seg, end;            // literals per stream (the last takes the rest); `done` at the current stream's end
    size_t off[5];                // the streams are p[off[k], off[k + 1])
    TdRev r;
};

TD_FN bool td_lit_open(TdLit& L) {
    L.end = L.cur == L.streams - 1 ? L.size : (uint32_t)(L.cur + 1) * L.seg;
    return td_rev_init(L.r, L.p + L.off[L.cur], L.off[L.cur + 1] - L.off[L.cur]);
}

// the current stream must end exactly with its literals
TD_FN bool td_lit_advance(TdLit& L) {
    if (L.r.pos != 0 || L.cur + 1 >= L.streams) return false;
    ++L.cur;
    return td_lit_open(L);
}

// k literals to d (the caller keeps done + k <= size)
TD_FN bool td_lit_copy(TdLit& L, const TdZstdWork* w, uint8_t* d, uint32_t k) {
    if (L.type == 0) {
        for (uint32_t i = 0; i < k; ++i) d[i] = L.p[L.done + i];
        L.done += k;
    } else if (L.type == 1) {
        for (uint32_t i = 0; i < k; ++i) d[i] = L.p[0];
        L.done += k;
    } else {
        for (uint32_t i = 0; i < k; ++i) {
            while (L.done == L.end) if (!td_lit_advance(L)) return false;
            const uint32_t e = w->huf[td_rev_peek(L.r, L.log)];
            L.r.pos -= e >> 8;
            if (L.r.pos < 0) return false;
            d[i] = (uint8_t)e;
            ++L.done;
        }
    }
    return true;
}

struct TdZFrame {
    uint8_t* dst;
    size_t cap, op, start;        // start: the frame's first output byte
    size_t lim;                   // writes stop here: cap, or the frame's end when its declared content size fits
    int over;                     // what reaching lim early means: 1 the output is full, -1 corrupt (past the size)
    size_t block_max;
    uint32_t rep[3];
    int ll_log, of_log, ml_log, huf_log;   // -1: no table yet in this frame
};

// k bytes of literals to the output, clipped at lim: 0, f.over when lim comes first, -1 corrupt
TD_FN int td_zlits(TdLit& L, const TdZstdWork* w, TdZFrame& f, uint32_t k) {
    const size_t room = f.lim - f.op;
    const uint32_t m = k < room ? k : (uint32_t)room;
    if (!td_lit_copy(L, w, f.dst + f.op, m)) return -1;
    f.op += m;
    return m < k ? f.over : 0;
}

// one sequence table (RFC 8878 3.1.1.3.2.1): predefined, RLE, FSE-compressed or repeat.  Returns bytes used or -1.
TD_FN long long td_seq_table(int mode, const uint8_t* p, size_t n, TdFse* t, int& log, int max_sym, int max_log,
                             const char* predef, int predef_log, TdZstdWork* w) {
    if (mode == 0) {
        int nsym = 0;
        for (; predef[nsym]; ++nsym) w->norm[nsym] = (int16_t)(predef[nsym] - '1');
        td_fse_build(t, w->norm, nsym, predef_log, w->next);
        log = predef_log;
        return 0;
    }
    if (mode == 1) {
        if (n == 0 || p[0] > max_sym) return -1;
        t[0].sym = p[0];
        t[0].nb = 0;
        t[0].base = 0;
        log = 0;
        return 1;
    }
    if (mode == 2) {
        int nsym, lg;
        const long long h = td_fse_header(p, n, max_sym, max_log, w->norm, nsym, lg);
        if (h < 0 || !td_fse_build(t, w->norm, nsym, lg, w->next)) return -1;
        log = lg;
        return h;
    }
    return log < 0 ? -1 : 0;
}

// one compressed block p[0, n): 0, 1 when the output is full first, -1 corrupt (also: output past the frame's
// declared content size)
TD_FN int td_zblock(const uint8_t* p, size_t n, TdZFrame& f, TdZstdWork* w) {
    if (n == 0) return -1;
    TdLit L;
    L.done = 0;
    L.type = p[0] & 3;
    const int sf = (p[0] >> 2) & 3;
    size_t ip;
    if (L.type < 2) {                              // raw or RLE literals
        if (sf == 1) {
            if (n < 2) return -1;
            L.size = (uint32_t)(p[0] >> 4) | (uint32_t)p[1] << 4;
            ip = 2;
        } else if (sf == 3) {
            if (n < 3) return -1;
            L.size = (uint32_t)(p[0] >> 4) | (uint32_t)p[1] << 4 | (uint32_t)p[2] << 12;
            ip = 3;
        } else {
            L.size = p[0] >> 3;
            ip = 1;
        }
        L.p = p + ip;
        const size_t len = L.type == 0 ? L.size : 1;
        if (L.size > f.block_max || len > n - ip) return -1;
        ip += len;
    } else {                                       // Huffman literals, with a new tree or the previous one
        const int hl = sf < 2 ? 3 : sf + 2, bits = sf < 2 ? 10 : sf == 2 ? 14 : 18;
        if (n < (size_t)hl) return -1;
        uint64_t h = 0;
        for (int k = 0; k < hl; ++k) h |= (uint64_t)p[k] << (8 * k);
        L.size = (uint32_t)(h >> 4) & ((1u << bits) - 1);
        size_t cs = (size_t)(h >> (4 + bits)) & ((1u << bits) - 1);
        L.streams = sf == 0 ? 1 : 4;
        if (L.size == 0 || L.size > f.block_max || (L.streams == 4 && L.size < 6) || cs > n - hl) return -1;
        const uint8_t* q = p + hl;
        ip = hl + cs;
        if (L.type == 2) {
            const long long t = td_huf_header(q, cs, w, f.huf_log);
            if (t < 0) return -1;
            q += t;
            cs -= (size_t)t;
        } else if (f.huf_log < 0) {
            return -1;
        }
        L.type = 2;
        L.p = q;
        L.log = f.huf_log;
        L.off[0] = 0;
        L.off[1] = L.off[4] = cs;
        if (L.streams == 4) {                      // jump table: the sizes of the first three streams
            if (cs < 6) return -1;
            const size_t s1 = q[0] | q[1] << 8, s2 = q[2] | q[3] << 8, s3 = q[4] | q[5] << 8;
            if (s1 + s2 + s3 > cs - 6) return -1;
            L.off[0] = 6;
            L.off[1] = 6 + s1;
            L.off[2] = 6 + s1 + s2;
            L.off[3] = 6 + s1 + s2 + s3;
        }
        L.seg = (L.size + 3) / 4;
        L.cur = 0;
        if (!td_lit_open(L)) return -1;
    }
    if (ip >= n) return -1;                        // sequences section
    uint32_t nseq = p[ip++];
    if (nseq == 255) {
        if (n - ip < 2) return -1;
        nseq = (p[ip] | (uint32_t)p[ip + 1] << 8) + 0x7F00;
        ip += 2;
    } else if (nseq >= 128) {
        if (ip >= n) return -1;
        nseq = ((nseq - 128) << 8) + p[ip++];
    }
    size_t blk = 0;                                // bytes this block has produced
    if (nseq > 0) {
        if (ip >= n) return -1;
        const int modes = p[ip++];
        if (modes & 3) return -1;
        long long t = td_seq_table(modes >> 6, p + ip, n - ip, w->ll, f.ll_log, 35, 9,
                                   "543333333333322233333333343222220000", 6, w);
        if (t < 0) return -1;
        ip += (size_t)t;
        t = td_seq_table((modes >> 4) & 3, p + ip, n - ip, w->of, f.of_log, 31, 8, "22222233322222222222222200000", 5,
                         w);
        if (t < 0) return -1;
        ip += (size_t)t;
        t = td_seq_table((modes >> 2) & 3, p + ip, n - ip, w->ml, f.ml_log, 52, 9,
                         "25433333322222222222222222222222222222222222220000000", 6, w);
        if (t < 0) return -1;
        ip += (size_t)t;
        TdRev r;
        if (!td_rev_init(r, p + ip, n - ip)) return -1;
        uint32_t sll = td_rev_get(r, f.ll_log), sof = td_rev_get(r, f.of_log), sml = td_rev_get(r, f.ml_log);
        for (uint32_t i = 0; i < nseq; ++i) {
            const int ofc = w->of[sof].sym, mlc = w->ml[sml].sym, llc = w->ll[sll].sym;
            const uint32_t ofv = (1u << ofc) + td_rev_get(r, ofc);
            const uint32_t ml = w->ml_base[mlc] + td_rev_get(r, w->ml_bits[mlc]);
            const uint32_t ll = w->ll_base[llc] + td_rev_get(r, w->ll_bits[llc]);
            if (i + 1 < nseq) {
                sll = w->ll[sll].base + td_rev_get(r, w->ll[sll].nb);
                sml = w->ml[sml].base + td_rev_get(r, w->ml[sml].nb);
                sof = w->of[sof].base + td_rev_get(r, w->of[sof].nb);
            }
            if (r.pos < 0) return -1;
            uint32_t off;                          // offset value 1-3: a repeat offset (shifted by one when ll == 0)
            if (ofv > 3) {
                off = ofv - 3;
                f.rep[2] = f.rep[1];
                f.rep[1] = f.rep[0];
                f.rep[0] = off;
            } else {
                const uint32_t idx = ofv - 1 + (ll == 0);
                if (idx == 0) {
                    off = f.rep[0];
                } else {
                    off = idx == 3 ? f.rep[0] - 1 : f.rep[idx];
                    if (idx != 1) f.rep[2] = f.rep[1];
                    f.rep[1] = f.rep[0];
                    f.rep[0] = off;
                }
            }
            if (ll > L.size - L.done) return -1;
            blk += (size_t)ll + ml;
            if (blk > f.block_max) return -1;
            const int q = td_zlits(L, w, f, ll);
            if (q) return q;
            if (off == 0 || off > f.op - f.start) return -1;   // a match starts inside its own frame
            const size_t room = f.lim - f.op;
            const uint32_t m = ml < room ? ml : (uint32_t)room;
            uint8_t* d = f.dst + f.op;
            const uint8_t* s = d - off;
            for (uint32_t k = 0; k < m; ++k) d[k] = s[k];
            f.op += m;
            if (m < ml) return f.over;
        }
        if (r.pos != 0) return -1;
    } else if (ip != n) {
        return -1;
    }
    const uint32_t rest = L.size - L.done;
    if (blk + rest > f.block_max) return -1;
    const int q = td_zlits(L, w, f, rest);
    if (q) return q;
    if (L.type == 2) {                             // every Huffman stream used up exactly
        while (L.cur + 1 < L.streams) if (!td_lit_advance(L)) return -1;
        if (L.r.pos != 0) return -1;
    }
    return 0;
}

// one frame p[0, n) (its magic checked by the caller) to f.dst from f.op; `used`: its bytes.
// 0, 1 when the output is full first, -1 corrupt
TD_FN int td_zframe(const uint8_t* p, size_t n, TdZFrame& f, TdZstdWork* w, size_t& used) {
    if (n < 5) return -1;
    const int fhd = p[4], fcs_flag = fhd >> 6, single = (fhd >> 5) & 1, did_flag = fhd & 3;
    if (fhd & 8) return -1;                        // reserved bit
    size_t ip = 5;
    uint64_t window = 0;
    if (!single) {
        if (ip >= n) return -1;
        const int wd = p[ip++];
        window = 1ull << (10 + (wd >> 3));
        window += (window >> 3) * (uint64_t)(wd & 7);
    }
    const size_t did_bytes = did_flag == 3 ? 4 : (size_t)did_flag;
    const size_t fcs_bytes = fcs_flag == 0 ? (size_t)single : (size_t)1 << fcs_flag;
    if (n - ip < did_bytes + fcs_bytes) return -1;
    uint32_t did = 0;
    for (size_t k = 0; k < did_bytes; ++k) did |= (uint32_t)p[ip + k] << (8 * k);
    if (did) return -1;                            // dictionaries are not supported
    ip += did_bytes;
    uint64_t fcs = 0;
    for (size_t k = 0; k < fcs_bytes; ++k) fcs |= (uint64_t)p[ip + k] << (8 * k);
    if (fcs_bytes == 2) fcs += 256;
    ip += fcs_bytes;
    if (single) window = fcs;
    f.block_max = window < 131072 ? (size_t)window : 131072;
    f.start = f.op;
    f.rep[0] = 1;
    f.rep[1] = 4;
    f.rep[2] = 8;
    f.ll_log = f.of_log = f.ml_log = f.huf_log = -1;
    // A declared content size that fits in the output bounds the frame: a frame that writes past it is corrupt, so
    // such a frame is decoded completely and its checksum verified.  Otherwise output stops at cap, unchecked.
    const bool bounded = fcs_bytes && fcs <= f.cap - f.start;
    f.lim = bounded ? f.start + (size_t)fcs : f.cap;
    f.over = bounded ? -1 : 1;
    for (;;) {
        if (n - ip < 3) return -1;
        const uint32_t bh = (uint32_t)p[ip] | (uint32_t)p[ip + 1] << 8 | (uint32_t)p[ip + 2] << 16;
        ip += 3;
        const uint32_t type = (bh >> 1) & 3, bs = bh >> 3;
        if (type == 3 || bs > f.block_max) return -1;
        int q;
        if (type == 2) {
            if (bs > n - ip) return -1;
            q = td_zblock(p + ip, bs, f, w);
            ip += bs;
        } else {                                   // raw or RLE block
            const size_t len = type == 0 ? bs : 1;
            if (len > n - ip) return -1;
            const size_t room = f.lim - f.op, m = bs < room ? bs : room;
            uint8_t* d = f.dst + f.op;
            for (size_t k = 0; k < m; ++k) d[k] = p[ip + (type == 0 ? k : 0)];
            f.op += m;
            ip += len;
            q = m < bs ? f.over : 0;
        }
        if (q) return q;
        if (bh & 1) break;
    }
    const size_t got = f.op - f.start;
    if (fcs_bytes && got != fcs) return -1;
    if ((fhd >> 2) & 1) {                          // content checksum: low 32 bits of XXH64
        if (n - ip < 4) return -1;
        if ((uint32_t)td_xxh64(f.dst + f.start, got) != td_le32(p + ip)) return -1;
        ip += 4;
    }
    used = ip;
    return 0;
}

TD_FN long long td_zstd(const uint8_t* src, size_t n, uint8_t* dst, size_t cap, TdZstdWork* w) {
    const char* llb = "\1\1\1\1\2\2\3\3\4\6\7\10\11\12\13\14\15\16\17\20";        // extra bits of codes 16..35
    const char* mlb = "\1\1\1\1\2\2\3\3\4\4\5\7\10\11\12\13\14\15\16\17\20";    // extra bits of codes 32..52
    for (int c = 0; c < 36; ++c) {
        w->ll_bits[c] = (uint8_t)(c < 16 ? 0 : llb[c - 16]);
        w->ll_base[c] = c <= 16 ? (uint32_t)c : w->ll_base[c - 1] + (1u << w->ll_bits[c - 1]);
    }
    for (int c = 0; c < 53; ++c) {
        w->ml_bits[c] = (uint8_t)(c < 32 ? 0 : mlb[c - 32]);
        w->ml_base[c] = c <= 32 ? (uint32_t)c + 3 : w->ml_base[c - 1] + (1u << w->ml_bits[c - 1]);
    }
    TdZFrame f;
    f.dst = dst;
    f.cap = cap;
    f.op = 0;
    size_t ip = 0;
    while (ip < n && f.op < cap) {
        if (n - ip < 4) return -1;
        const uint32_t magic = td_le32(src + ip);
        if ((magic & 0xFFFFFFF0u) == 0x184D2A50u) {      // skippable frame
            if (n - ip < 8 || td_le32(src + ip + 4) > n - ip - 8) return -1;
            ip += 8 + (size_t)td_le32(src + ip + 4);
            continue;
        }
        if (magic != 0xFD2FB528u) return -1;
        size_t used = 0;
        const int q = td_zframe(src + ip, n - ip, f, w, used);
        if (q < 0) return -1;
        if (q > 0) return (long long)cap;
        ip += used;
    }
    return (long long)f.op;
}
