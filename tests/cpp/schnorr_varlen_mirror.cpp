// BIP-340 over messages of different lengths through the C++ mirror (host/secp256k1_voi.hpp): the valid rows of the
// BIP-340 vectors, given on the command line as pk, msg, sig triples ("-" for an empty message), must verify row by row
// and as one batch; the same batch with one bit of the last s flipped must fail both ways; SchnorrSignBatch over the
// rows must give signatures that verify.
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
    if (argc < 4 || (argc - 1) % 3 != 0) return 2;
    std::vector<uint8_t> pk, sig;
    std::vector<std::vector<uint8_t>> msgs;
    size_t n = (size_t)(argc - 1) / 3;
    for (size_t i = 0; i < n; i++) {
        auto p = unhex(argv[1 + 3 * i]), s = unhex(argv[3 + 3 * i]);
        if (p.size() != 32 || s.size() != 64) return 2;
        pk.insert(pk.end(), p.begin(), p.end());
        msgs.push_back(unhex(argv[2 + 3 * i]));
        sig.insert(sig.end(), s.begin(), s.end());
    }
    namespace btc = secp256k1::secec::bitcoin;
    std::vector<uint8_t> ok(n);
    btc::SchnorrVerifyBatch(pk.data(), msgs, sig.data(), ok.data());
    for (size_t i = 0; i < n; i++)
        if (ok[i] != 1) {
            fprintf(stderr, "FAILED: valid row %zu rejected\n", i);
            return 1;
        }
    if (!btc::SchnorrBatchVerify(pk.data(), msgs, sig.data())) {
        fprintf(stderr, "FAILED: valid batch rejected\n");
        return 1;
    }
    sig[64 * (n - 1) + 63] ^= 1;
    btc::SchnorrVerifyBatch(pk.data(), msgs, sig.data(), ok.data());
    if (ok[n - 1] != 0 || btc::SchnorrBatchVerify(pk.data(), msgs, sig.data())) {
        fprintf(stderr, "FAILED: corrupted row accepted\n");
        return 1;
    }
    // sign every message under one key, then verify the batch
    std::vector<uint8_t> priv(32 * n, 0), aux(32 * n, 0x5a), sig2(64 * n), st(n);
    for (size_t i = 0; i < n; i++) priv[32 * i + 31] = 3;
    btc::SchnorrSignBatch(priv.data(), msgs, aux.data(), sig2.data(), st.data());
    auto key = btc::SchnorrPrivateKey::NewSchnorrPrivateKey(priv.data(), 32);
    std::vector<uint8_t> pk2;
    for (size_t i = 0; i < n; i++) {
        if (st[i] != S256_ST_OK) return 1;
        auto x = key.PublicKeyRef().Bytes();
        pk2.insert(pk2.end(), x.begin(), x.end());
    }
    if (!btc::SchnorrBatchVerify(pk2.data(), msgs, sig2.data())) {
        fprintf(stderr, "FAILED: signed batch rejected\n");
        return 1;
    }
    printf("varlen mirror ok\n");
    return 0;
}
