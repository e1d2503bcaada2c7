// BIP-340 batch verification through the C++ mirror (host/secp256k1_voi.hpp): the valid 32-byte-message rows of
// the BIP-340 vectors, given on the command line as pk, msg, sig triples, must pass as one batch; the same batch with
// one bit of the last s flipped must not.
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
    std::vector<uint8_t> pk, msg, sig;
    size_t n = (size_t)(argc - 1) / 3;
    for (size_t i = 0; i < n; i++) {
        auto p = unhex(argv[1 + 3 * i]), m = unhex(argv[2 + 3 * i]), s = unhex(argv[3 + 3 * i]);
        if (p.size() != 32 || m.size() != 32 || s.size() != 64) return 2;
        pk.insert(pk.end(), p.begin(), p.end());
        msg.insert(msg.end(), m.begin(), m.end());
        sig.insert(sig.end(), s.begin(), s.end());
    }
    namespace btc = secp256k1::secec::bitcoin;
    if (!btc::SchnorrBatchVerify(pk.data(), msg.data(), 32, sig.data(), n)) {
        fprintf(stderr, "FAILED: valid batch rejected\n");
        return 1;
    }
    sig[64 * (n - 1) + 63] ^= 1;
    if (btc::SchnorrBatchVerify(pk.data(), msg.data(), 32, sig.data(), n)) {
        fprintf(stderr, "FAILED: corrupted batch accepted\n");
        return 1;
    }
    printf("batch mirror ok\n");
    return 0;
}
