// Hash-to-curve over messages of different lengths through the C++ mirror (host/secp256k1_voi.hpp): for the DST and
// messages given on the command line (hex, "-" for an empty message), h2c::HashToCurveBatch must give, row by row and
// in both suites, the bytes of the per-item Secp256k1_XMD_SHA256_SSWU_RO / _NU calls; an empty DST must throw.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "../../secp256k1-voi_b200/host/secp256k1_voi.hpp"

static std::vector<uint8_t> unhex(const std::string &h) {
    if (h == "-") return {};
    std::vector<uint8_t> o(h.size() / 2);
    for (size_t i = 0; i < o.size(); i++) o[i] = (uint8_t)strtoul(h.substr(2 * i, 2).c_str(), nullptr, 16);
    return o;
}

int main(int argc, char **argv) {
    if (argc < 3) return 2;
    namespace h2c = secp256k1::secec::h2c;
    const std::string d = argv[1];
    const std::vector<uint8_t> dst(d.begin(), d.end());
    std::vector<std::vector<uint8_t>> msgs;
    for (int i = 2; i < argc; i++) msgs.push_back(unhex(argv[i]));
    const size_t n = msgs.size();
    for (bool ro : {true, false}) {
        std::vector<uint8_t> out(65 * n), st(n);
        h2c::HashToCurveBatch(dst, msgs, ro, out.data(), st.data());
        for (size_t i = 0; i < n; i++) {
            auto p = ro ? h2c::Secp256k1_XMD_SHA256_SSWU_RO(dst.data(), dst.size(), msgs[i].data(), msgs[i].size())
                        : h2c::Secp256k1_XMD_SHA256_SSWU_NU(dst.data(), dst.size(), msgs[i].data(), msgs[i].size());
            auto want = p.UncompressedBytes();
            if (st[i] != S256_ST_OK || want.size() != 65 || !std::equal(want.begin(), want.end(), out.begin() + 65 * i)) {
                fprintf(stderr, "FAILED: row %zu (ro=%d) differs from the per-item call\n", i, (int)ro);
                return 1;
            }
        }
    }
    bool threw = false;
    try {
        std::vector<uint8_t> out(65 * n), st(n);
        h2c::HashToCurveBatch({}, msgs, true, out.data(), st.data());
    } catch (const secp256k1::Error &) {
        threw = true;
    }
    if (!threw) {
        fprintf(stderr, "FAILED: an empty DST was accepted\n");
        return 1;
    }
    printf("h2c varlen mirror ok\n");
    return 0;
}
