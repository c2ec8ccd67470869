// Gpu::verify_grouped of the C++ mirror (include/jubjub_schnorr.hpp) on one part read from a file; built and run by
// tests/test_verify_grouped.py.  Usage: test_grouped <in> <out>.  <in>: kind (int32), n (uint64), then pk, sig and msg of the
// n items of that kind; <out>: the n statuses, the n challenges and the fallback count (uint64).
#include <cstdio>
#include <vector>

#include "jubjub_schnorr.hpp"

int main(int argc, char** argv) {
    if (argc != 3) return 2;
    FILE* f = std::fopen(argv[1], "rb");
    if (!f) return 2;
    int32_t kind = 0;
    uint64_t n = 0;
    if (std::fread(&kind, 4, 1, f) != 1 || std::fread(&n, 8, 1, f) != 1) return 2;
    const size_t pkw = kind == JJS_KIND_SINGLE ? 32 : 64, sgw = kind == JJS_KIND_DOUBLE ? 96 : 64;
    std::vector<uint8_t> pk(pkw * n), sig(sgw * n), msg(32 * n), status(n), c(32 * n);
    if (std::fread(pk.data(), 1, pk.size(), f) != pk.size() || std::fread(sig.data(), 1, sig.size(), f) != sig.size() ||
        std::fread(msg.data(), 1, msg.size(), f) != msg.size())
        return 2;
    std::fclose(f);
    jubjub_schnorr::Gpu gpu;
    jjs_part part{kind, pk.data(), nullptr, sig.data(), msg.data(), (size_t)n, status.data(), c.data(), nullptr, nullptr};
    const uint64_t fallback = gpu.verify_grouped(&part, 1);
    f = std::fopen(argv[2], "wb");
    if (!f) return 2;
    std::fwrite(status.data(), 1, n, f);
    std::fwrite(c.data(), 1, c.size(), f);
    std::fwrite(&fallback, 8, 1, f);
    std::fclose(f);
    std::printf("cpp grouped ok\n");
    return 0;
}
