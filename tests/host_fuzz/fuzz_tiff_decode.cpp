// ASan/UBSan harness for the device TIFF decoders (csrc/tiff_decode.h), compiled for the host.  Every buffer is an
// exact-size heap block, so AddressSanitizer traps the first byte read or written outside a stream or a capacity.
// Built and run by tests/test_tiff_decode_host.py:
//     fuzz_tiff_decode records <in> <out>   decode each record of <in> (u8 kind 0 Deflate / 1 LZW / 2 PackBits,
//                                            u64 cap, u32 n, n bytes); write i64 result + the bytes to <out>.
//                                            LZW and PackBits must equal cia_tiff_lzw_decode / _packbits_decode.
//     fuzz_tiff_decode random <iters>       random and bit-flipped streams of all three kinds at random capacities
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <random>
#include <vector>

#include "../../cell-image-analysis_b200/csrc/tiff_decode.h"

extern "C" long long cia_tiff_lzw_decode(const uint8_t*, size_t, uint8_t*, size_t);
extern "C" long long cia_tiff_packbits_decode(const uint8_t*, size_t, uint8_t*, size_t);

static std::unique_ptr<TdInflateWork> g_inflate(new TdInflateWork);
static std::unique_ptr<TdLzwWork> g_lzw(new TdLzwWork);
static long long g_mismatch = 0;

// decodes src into an exact-size block; for LZW / PackBits also with the host decoder, which must agree
static long long run(int kind, const std::vector<uint8_t>& in, size_t cap, std::vector<uint8_t>& got) {
    uint8_t* s = (uint8_t*)malloc(in.size() ? in.size() : 1);
    if (!in.empty()) memcpy(s, in.data(), in.size());
    uint8_t* d = (uint8_t*)malloc(cap ? cap : 1);
    long long r;
    if (kind == 0) {
        r = td_inflate(s, in.size(), d, cap, g_inflate.get());
    } else {
        r = kind == 1 ? td_lzw(s, in.size(), d, cap, g_lzw.get()) : td_packbits(s, in.size(), d, cap);
        uint8_t* e = (uint8_t*)malloc(cap ? cap : 1);
        const long long q = kind == 1 ? cia_tiff_lzw_decode(s, in.size(), e, cap)
                                      : cia_tiff_packbits_decode(s, in.size(), e, cap);
        if (q != r || (r > 0 && memcmp(d, e, (size_t)r))) {
            if (g_mismatch++ < 5) fprintf(stderr, "mismatch kind %d n %zu cap %zu: %lld vs host %lld\n", kind, in.size(), cap, r, q);
        }
        free(e);
    }
    got.assign(d, d + (r > 0 ? r : 0));
    free(d);
    free(s);
    return r;
}

int main(int argc, char** argv) {
    if (argc >= 4 && !strcmp(argv[1], "records")) {
        FILE* f = fopen(argv[2], "rb");
        FILE* o = fopen(argv[3], "wb");
        if (!f || !o) return 2;
        long long n_rec = 0;
        for (;;) {
            uint8_t kind;
            uint64_t cap;
            uint32_t n;
            if (fread(&kind, 1, 1, f) != 1) break;
            if (fread(&cap, 8, 1, f) != 1 || fread(&n, 4, 1, f) != 1) return 2;
            std::vector<uint8_t> in(n), got;
            if (n && fread(in.data(), 1, n, f) != n) return 2;
            const long long r = run(kind, in, (size_t)cap, got);
            fwrite(&r, 8, 1, o);
            if (!got.empty()) fwrite(got.data(), 1, got.size(), o);
            ++n_rec;
        }
        fclose(f);
        fclose(o);
        printf("ok: %lld records %lld mismatches\n", n_rec, g_mismatch);
        return g_mismatch ? 1 : 0;
    }
    if (argc >= 3 && !strcmp(argv[1], "random")) {
        const int iters = atoi(argv[2]);
        std::mt19937_64 rng(1234);
        long long refused[3] = {0, 0, 0};
        for (int it = 0; it < iters; ++it) {
            const int kind = it % 3;
            std::vector<uint8_t> in(rng() % 4096), got;
            for (auto& b : in) b = (uint8_t)rng();
            if (kind == 0 && in.size() >= 2 && (it & 4)) {          // a valid header, so the block decoders run
                in[0] = 0x78;
                in[1] = 0x9c;
            }
            const size_t cap = rng() % 3 == 0 ? 0 : rng() % 65536;
            if (run(kind, in, cap, got) < 0) refused[kind]++;
        }
        printf("ok: %d iterations, refused %lld %lld %lld, %lld mismatches\n", iters, refused[0], refused[1],
               refused[2], g_mismatch);
        return g_mismatch ? 1 : 0;
    }
    fprintf(stderr, "usage: fuzz_tiff_decode records <in> <out> | random <iters>\n");
    return 2;
}
