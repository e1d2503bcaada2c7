// der_sim.cpp -- TEST INFRASTRUCTURE ONLY: the device DER parser (der.cuh) on the CPU.
//
// Runs the item functions of k_parse_der and k_check_bip66 one row at a time, with the rows read through the same
// msg_offsets accessor the kernels are instantiated with: row i is der[offsets[i], offsets[i + 1]), and a row with
// decreasing offsets is unreadable (rejected, no byte read).
#include "../../secp256k1-voi_b200/csrc/der.cuh"

using namespace s256;
#define EXPORT extern "C" __attribute__((visibility("default")))

// k_parse_der<msg_offsets, BIP66>: r||s rows (zeros when rejected) and ok bytes
EXPORT void sim_parse_der(const uint8_t *der, const size_t *offsets, size_t n, int bip66, uint8_t *sig64, uint8_t *ok) {
    const msg_offsets rows{der, offsets, 0};
    for (size_t i = 0; i < n; i++) {
        uint32_t rs[16];
        ok[i] = (uint8_t)(bip66 ? item_parse_der<true>(i, rows, rs) : item_parse_der<false>(i, rows, rs));
        der_store_sig64(sig64 + 64 * i, rs);
    }
}

// k_check_bip66<msg_offsets>
EXPORT void sim_check_bip66(const uint8_t *der, const size_t *offsets, size_t n, uint8_t *ok) {
    const msg_offsets rows{der, offsets, 0};
    for (size_t i = 0; i < n; i++) ok[i] = (uint8_t)item_check_bip66(i, rows);
}
