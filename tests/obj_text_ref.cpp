// obj_text_ref.cpp -- an independent statement of the float text Mesh.WriteObj prints (.NET Core `float.ToString()`):
// the shortest round-trip digits from std::to_chars(float, chars_format::scientific), laid out by the .NET rule
// (scientific when the decimal exponent is below -4 or at least max(#digits, 7), exponent with at least two digits;
// "-0", "NaN", "Infinity", "-Infinity").  Built by tests/test_gpu_obj.py with g++ -std=c++17.
//
//   obj_text_ref texts                 little-endian uint32 bit patterns on stdin -> one text per line on stdout
//   obj_text_ref digests FIRST N       FNV-1a-64 of the concatenated text + '\n' of every bit pattern of the 2^20-pattern
//                                      blocks FIRST .. FIRST+N-1 in increasing order, one hex digest per line (threaded)
#include <atomic>
#include <charconv>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

static int net_text(uint32_t bits, char* out)
{
    float x;
    std::memcpy(&x, &bits, 4);
    const bool neg = (bits >> 31) != 0;
    if (std::isnan(x)) { std::memcpy(out, "NaN", 3); return 3; }
    if (std::isinf(x)) {
        if (neg) { std::memcpy(out, "-Infinity", 9); return 9; }
        std::memcpy(out, "Infinity", 8);
        return 8;
    }
    if (x == 0.0f) {
        if (neg) { std::memcpy(out, "-0", 2); return 2; }
        out[0] = '0';
        return 1;
    }
    char buf[48];
    const auto r = std::to_chars(buf, buf + sizeof(buf), x, std::chars_format::scientific);
    *r.ptr = 0;
    // buf = [-]d[.ddd]e(+|-)XX
    std::string digits;
    const char* p = buf + (neg ? 1 : 0);
    for (; *p != 'e'; p++)
        if (*p != '.') digits += *p;
    const int E = std::atoi(p + 1);
    const int nd = (int)digits.size();
    std::string s = neg ? "-" : "";
    if (E < -4 || E >= std::max(nd, 7)) {
        s += digits[0];
        if (nd > 1) s += "." + digits.substr(1);
        char e[16];
        std::snprintf(e, sizeof(e), "E%c%02d", E < 0 ? '-' : '+', E < 0 ? -E : E);
        s += e;
    } else if (E < 0) {
        s += "0." + std::string(-E - 1, '0') + digits;
    } else if (nd <= E + 1) {
        s += digits + std::string(E + 1 - nd, '0');
    } else {
        s += digits.substr(0, E + 1) + "." + digits.substr(E + 1);
    }
    std::memcpy(out, s.data(), s.size());
    return (int)s.size();
}

static uint64_t block_digest(uint32_t block)
{
    uint64_t h = 14695981039346656037ull;
    char t[64];
    for (uint32_t i = 0; i < (1u << 20); i++) {
        const int n = net_text((block << 20) | i, t);
        t[n] = '\n';
        for (int k = 0; k <= n; k++) { h ^= (unsigned char)t[k]; h *= 1099511628211ull; }
    }
    return h;
}

int main(int argc, char** argv)
{
    if (argc >= 2 && std::strcmp(argv[1], "texts") == 0) {
        uint32_t bits;
        char t[64];
        while (std::fread(&bits, 4, 1, stdin) == 1) {
            const int n = net_text(bits, t);
            t[n] = '\n';
            std::fwrite(t, 1, n + 1, stdout);
        }
        return 0;
    }
    if (argc >= 4 && std::strcmp(argv[1], "digests") == 0) {
        const uint32_t first = (uint32_t)std::strtoul(argv[2], nullptr, 10), n = (uint32_t)std::strtoul(argv[3], nullptr, 10);
        if ((uint64_t)first + n > 4096) { std::fprintf(stderr, "blocks out of range\n"); return 2; }
        std::vector<uint64_t> d(n);
        std::atomic<uint32_t> next{0};
        const unsigned nt = std::max(1u, std::thread::hardware_concurrency());
        std::vector<std::thread> pool;
        for (unsigned k = 0; k < nt; k++)
            pool.emplace_back([&] {
                for (uint32_t i; (i = next++) < n;) d[i] = block_digest(first + i);
            });
        for (auto& th : pool) th.join();
        for (uint64_t v : d) std::printf("%016llx\n", (unsigned long long)v);
        return 0;
    }
    std::fprintf(stderr, "usage: obj_text_ref texts < bits | obj_text_ref digests FIRST N\n");
    return 2;
}
