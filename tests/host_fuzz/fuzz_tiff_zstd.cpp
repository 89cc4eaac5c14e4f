// ASan/UBSan harness for the Zstandard decoder (td_zstd of csrc/tiff_decode.h), compiled for the host.  Every buffer
// is an exact-size heap block, so AddressSanitizer traps the first byte read or written outside a stream or a
// capacity.  Built and run by tests/test_tiff_zstd_fuzz.py:
//     fuzz_tiff_zstd records <in> <out>   decode each record of <in> (u64 cap, u32 n, n bytes); write the i64 result
//                                          and the bytes to <out>.  cia_tiff_zstd_decode must agree with td_zstd.
//     fuzz_tiff_zstd random <iters>       random frames: random bytes behind a valid magic and frame header
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <random>
#include <vector>

#include "../../cell-image-analysis_b200/csrc/tiff_decode.h"

extern "C" long long cia_tiff_zstd_decode(const uint8_t*, size_t, uint8_t*, size_t);

static std::unique_ptr<TdZstdWork> g_work(new TdZstdWork);
static long long g_mismatch = 0;

static long long run(const std::vector<uint8_t>& in, size_t cap, std::vector<uint8_t>& got) {
    uint8_t* s = (uint8_t*)malloc(in.size() ? in.size() : 1);
    if (!in.empty()) memcpy(s, in.data(), in.size());
    uint8_t* d = (uint8_t*)malloc(cap ? cap : 1);
    uint8_t* e = (uint8_t*)malloc(cap ? cap : 1);
    const long long r = td_zstd(s, in.size(), d, cap, g_work.get());
    const long long q = cia_tiff_zstd_decode(s, in.size(), e, cap);
    if (q != r || (r > 0 && memcmp(d, e, (size_t)r))) {
        if (g_mismatch++ < 5) fprintf(stderr, "mismatch n %zu cap %zu: %lld vs %lld\n", in.size(), cap, r, q);
    }
    got.assign(d, d + (r > 0 ? r : 0));
    free(e);
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
            uint64_t cap;
            uint32_t n;
            if (fread(&cap, 8, 1, f) != 1) break;
            if (fread(&n, 4, 1, f) != 1) return 2;
            std::vector<uint8_t> in(n), got;
            if (n && fread(in.data(), 1, n, f) != n) return 2;
            const long long r = run(in, (size_t)cap, got);
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
        std::mt19937_64 rng(4321);
        long long refused = 0;
        for (int it = 0; it < iters; ++it) {
            std::vector<uint8_t> in(6 + rng() % 4096), got;
            for (auto& b : in) b = (uint8_t)rng();
            const uint8_t magic[4] = {0x28, 0xB5, 0x2F, 0xFD};
            memcpy(in.data(), magic, 4);
            in[4] &= 0xF4;                                   // no dictionary, reserved bit clear
            in[5] = (uint8_t)(0x50 + rng() % 8);             // a 1 MB-class window when there is a descriptor
            const size_t cap = rng() % 3 == 0 ? 0 : rng() % 65536;
            if (run(in, cap, got) < 0) refused++;
        }
        printf("ok: %d iterations, refused %lld, %lld mismatches\n", iters, refused, g_mismatch);
        return g_mismatch ? 1 : 0;
    }
    fprintf(stderr, "usage: fuzz_tiff_zstd records <in> <out> | random <iters>\n");
    return 2;
}
