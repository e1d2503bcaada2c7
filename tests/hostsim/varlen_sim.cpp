// varlen_sim.cpp -- TEST INFRASTRUCTURE ONLY: the BIP-340 entry points over messages of different lengths
// (s256_schnorr_verify_varlen, s256_schnorr_sign_varlen, s256_schnorr_batch_verify_varlen) on the CPU.
//
// Builds on batch_sim.cpp (included whole, with hostsim.cpp under it) and drives the item functions the kernels run,
// with the message rows read through the same msg_offsets accessor the *_varlen kernels are instantiated with: row i
// is msg[offsets[i], offsets[i + 1]), and a row with decreasing offsets is unreadable (invalid, no byte read).
#include "batch_sim.cpp"

static msg_offsets rows_of(const uint8_t *msg, const size_t *offsets) { return msg_offsets{msg, offsets, 0}; }

// api.cu's chunk_schnorr_verify with k_schnorr_scalars<msg_offsets>
EXPORT void sim_schnorr_verify_varlen(const uint8_t *pkx, const uint8_t *msg, const size_t *offsets, const uint8_t *sig,
                                      size_t n, uint8_t *ok) {
    scratch s(n);
    const msg_offsets rows = rows_of(msg, offsets);
    for (size_t i = 0; i < n; i++) s.pvalid[i] = item_decode_xonly(s.aff[i], pkx + 32 * i);
    for (size_t i = 0; i < n; i++)
        item_schnorr_scalars(i, n, pkx, rows, sig, s.u1.data(), s.dig1.data(), s.dig2.data(), s.sfl.data());
    run_dsm(s, n);
    run_finish(s, n, true, true, 2, nullptr, ok, sig);
}

// api_sign.cu's chunk_schnorr_sign with k_schnorr_nonce<msg_offsets> and k_schnorr_sign_finish<msg_offsets>
EXPORT void sim_schnorr_sign_varlen(const uint8_t *priv32, const uint8_t *msg, const size_t *offsets, const uint8_t *aux32,
                                    size_t n, uint8_t *sig64, uint8_t *status) {
    ensure_tables();
    scratch s(n);
    const msg_offsets rows = rows_of(msg, offsets);
    std::vector<uint8_t> p65(65 * n), r65(65 * n), kbuf(32 * n), valid(n), st(n);
    for (size_t i = 0; i < n; i++) {
        sc k;
        sc_from_be32(k, priv32 + 32 * i);
        item_base_mult_ct(s.res[i], k, g_ct.data());
    }
    run_finish(s, n, false, false, 0, p65.data(), st.data(), nullptr);
    for (size_t i = 0; i < n; i++) {
        const uint8_t *m;
        size_t len;
        const uint32_t row_ok = rows.row(i, m, len);
        valid[i] = (uint8_t)(row_ok & item_schnorr_nonce(kbuf.data() + 32 * i, priv32 + 32 * i, p65.data() + 65 * i, m, len,
                                                         aux32 + 32 * i));
    }
    for (size_t i = 0; i < n; i++) {
        sc k;
        sc_from_be32(k, kbuf.data() + 32 * i);
        item_base_mult_ct(s.res[i], k, g_ct.data());
    }
    run_finish(s, n, false, false, 0, r65.data(), st.data(), nullptr);
    for (size_t i = 0; i < n; i++) {
        const uint8_t *m;
        size_t len;
        rows.row(i, m, len);
        item_schnorr_sign_finish(sig64 + 64 * i, status + i, priv32 + 32 * i, p65.data() + 65 * i, r65.data() + 65 * i,
                                 kbuf.data() + 32 * i, m, len, valid[i]);
    }
}

// Pass 1 of the batch (k_batch_leaves<msg_offsets>, then the tree) with chunks of `chunk` rows
static void sim_batch_seed_varlen(uint32_t seed[8], const uint8_t *pkx, const msg_offsets &rows, const uint8_t *sig, size_t n,
                                  size_t chunk) {
    size_t chunks = (n + chunk - 1) / chunk;
    std::vector<uint32_t> roots(8 * chunks), leaves(8 * chunk);
    for (size_t k = 0; k < chunks; k++) {
        size_t off = k * chunk, c = std::min(chunk, n - off);
        for (size_t i = 0; i < c; i++) {
            const uint8_t *m;
            size_t len;
            rows.row(off + i, m, len);
            batch_leaf(leaves.data() + 8 * i, pkx + 32 * (off + i), sig + 64 * (off + i), m, len);
        }
        batch_tree_fold(leaves.data(), c);
        std::copy(leaves.begin(), leaves.begin() + 8, roots.begin() + 8 * k);
    }
    batch_tree_fold(roots.data(), chunks);
    batch_seed(seed, roots.data(), (uint64_t)n);
}
EXPORT void sim_schnorr_batch_randomizers_varlen(const uint8_t *pkx, const uint8_t *msg, const size_t *offsets, const uint8_t *sig,
                                                 size_t n, size_t chunk, uint8_t *seed32, uint8_t *a32) {
    uint32_t seed[8];
    sim_batch_seed_varlen(seed, pkx, rows_of(msg, offsets), sig, n, chunk);
    words_be32(seed32, seed);
    for (size_t i = 0; i < n; i++) {
        sc a;
        batch_randomizer(a, seed, (uint64_t)i);
        sc_to_be32(a32 + 32 * i, a);
    }
}
// sim_schnorr_batch_verify of batch_sim.cpp with the rows of k_batch_prepare<msg_offsets>
EXPORT void sim_schnorr_batch_verify_varlen(const uint8_t *pkx, const uint8_t *msg, const size_t *offsets, const uint8_t *sig,
                                            size_t n, size_t chunk, uint8_t *ok) {
    if (n == 0) {
        *ok = 1;
        return;
    }
    ensure_tables();
    const msg_offsets rows = rows_of(msg, offsets);
    uint32_t seed[8];
    sim_batch_seed_varlen(seed, pkx, rows, sig, n, chunk);
    bool bad = false;
    sc sum = sc_zero();
    pt acc;
    pt_set_identity(acc);
    for (size_t off = 0; off < n; off += chunk) {
        size_t c = std::min(chunk, n - off);
        std::vector<apt> aff2(2 * c);
        std::vector<uint8_t> k2(64 * c), pt65(65 * 2 * c);
        for (size_t i = 0; i < c; i++) {
            size_t g = off + i;
            const uint8_t *m;
            size_t len;
            const uint32_t row_ok = rows.row(g, m, len);
            sc as;
            bad |= !item_batch_prepare(aff2.data() + 2 * i, k2.data() + 64 * i, as, pkx + 32 * g, m, len, sig + 64 * g, seed,
                                       (uint64_t)g, row_ok);
            sc_add(sum, sum, as);
        }
        for (size_t v = 0; v < 2 * c; v++) {
            pt65[65 * v] = 4;
            fe_to_be32(pt65.data() + 65 * v + 1, aff2[v].x);
            fe_to_be32(pt65.data() + 65 * v + 33, aff2[v].y);
        }
        uint8_t out65[65], st = 0, part96[96];
        sim_msm(k2.data(), pt65.data(), 2 * c, 1, 0, out65, &st, part96);
        pt part;
        pt_from_be96(part, part96);
        pt_add(acc, acc, part);
    }
    pt sg;
    item_base_mult_ct(sg, sum, g_ct.data());
    pt_add(acc, acc, sg);
    *ok = (uint8_t)(!bad && fe_is_zero(acc.z));
}
