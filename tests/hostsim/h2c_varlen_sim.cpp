// h2c_varlen_sim.cpp -- TEST INFRASTRUCTURE ONLY: s256_hash_to_curve_varlen_dev on the CPU.
//
// Builds on hostsim.cpp (included whole) and drives what api_h2c.cu's chunk_hash_to_curve runs for the msg_offsets
// instantiation of k_hash_to_curve: each row is read through the same accessor (row i is msg[offsets[i], offsets[i + 1]),
// and a row with decreasing offsets is unreadable: no byte of it is read and its validity byte is 0), hashed by
// item_hash_to_curve, and converted by the shared batched-affine conversion with the validity bytes as pvalid.  The
// DST is used as given (1..255 bytes): the library hashes a longer one on the host before any kernel sees it.
#include "hostsim.cpp"

EXPORT void sim_hash_to_curve_varlen(const uint8_t *dst, size_t dst_len, const uint8_t *msg, const size_t *offsets, size_t n,
                                     int ro, uint8_t *out65, uint8_t *status) {
    scratch s(n ? n : 1);
    const msg_offsets rows{msg, offsets, 0};
    for (size_t i = 0; i < n; i++) {
        const uint8_t *m;
        size_t len;
        s.pvalid[i] = (uint8_t)rows.row(i, m, len);
        item_hash_to_curve(s.res[i], dst, (int)dst_len, m, len, ro);
    }
    run_finish(s, n, true, false, 0, out65, status, nullptr);
}
