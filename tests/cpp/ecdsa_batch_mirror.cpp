// Recoverable ECDSA batch verification through the C++ mirror (host/secp256k1_voi.hpp): rows given on the command
// line as pk65, digest32, r||s||v triples must pass as one batch, also with RejectMalleable (the rows are low-s); the
// same batch with one bit of the last s flipped must not.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "../../secp256k1-voi_b200/host/secp256k1_voi.hpp"

static std::vector<uint8_t> unhex(const std::string &h) {
    std::vector<uint8_t> o(h.size() / 2);
    for (size_t i = 0; i < o.size(); i++) o[i] = (uint8_t)strtoul(h.substr(2 * i, 2).c_str(), nullptr, 16);
    return o;
}

int main(int argc, char **argv) {
    if (argc < 4 || (argc - 1) % 3 != 0) return 2;
    std::vector<uint8_t> pk, dg, sig;
    size_t n = (size_t)(argc - 1) / 3;
    for (size_t i = 0; i < n; i++) {
        auto p = unhex(argv[1 + 3 * i]), d = unhex(argv[2 + 3 * i]), s = unhex(argv[3 + 3 * i]);
        if (p.size() != 65 || d.size() != 32 || s.size() != 65) return 2;
        pk.insert(pk.end(), p.begin(), p.end());
        dg.insert(dg.end(), d.begin(), d.end());
        sig.insert(sig.end(), s.begin(), s.end());
    }
    namespace secec = secp256k1::secec;
    if (!secec::RecoverableBatchVerify(pk.data(), dg.data(), sig.data(), n) ||
        !secec::RecoverableBatchVerify(pk.data(), dg.data(), sig.data(), n, true)) {
        fprintf(stderr, "FAILED: valid batch rejected\n");
        return 1;
    }
    sig[65 * (n - 1) + 63] ^= 1;
    if (secec::RecoverableBatchVerify(pk.data(), dg.data(), sig.data(), n)) {
        fprintf(stderr, "FAILED: corrupted batch accepted\n");
        return 1;
    }
    printf("ecdsa batch mirror ok\n");
    return 0;
}
