// batch_sim.cpp -- TEST INFRASTRUCTURE ONLY: the BIP-340 batch verification of api_msm.cu
// (s256_schnorr_batch_verify) on the CPU.
//
// Builds on hostsim.cpp (included whole, so this library carries its own copy of the simulation) and runs the
// item functions of csrc/batch.cuh in the order the kernels run them, one "thread" at a time.  Each chunk's MSM
// rows go through hostsim.cpp's sim_msm, the same Pippenger flow chunk_msm_body runs on the device.
#include "hostsim.cpp"
#include "../../secp256k1-voi_b200/csrc/batch.cuh"

// Pass 1 with chunks of `chunk` rows: leaves, one root per chunk, the tree of the roots, the seed.
static void sim_batch_seed(uint32_t seed[8], const uint8_t *pkx, const uint8_t *msg, size_t msg_len, const uint8_t *sig,
                           size_t n, size_t chunk) {
    size_t chunks = (n + chunk - 1) / chunk;
    std::vector<uint32_t> roots(8 * chunks), leaves(8 * chunk);
    for (size_t k = 0; k < chunks; k++) {
        size_t off = k * chunk, c = std::min(chunk, n - off);
        for (size_t i = 0; i < c; i++)
            batch_leaf(leaves.data() + 8 * i, pkx + 32 * (off + i), sig + 64 * (off + i), msg + msg_len * (off + i), msg_len);
        batch_tree_fold(leaves.data(), c);
        std::copy(leaves.begin(), leaves.begin() + 8, roots.begin() + 8 * k);
    }
    batch_tree_fold(roots.data(), chunks);
    batch_seed(seed, roots.data(), (uint64_t)n);
}
// the seed (32 B) and every a_i (32 B big-endian) for chunks of `chunk` rows
EXPORT void sim_schnorr_batch_randomizers(const uint8_t *pkx, const uint8_t *msg, size_t msg_len, const uint8_t *sig, size_t n,
                                          size_t chunk, uint8_t *seed32, uint8_t *a32) {
    uint32_t seed[8];
    sim_batch_seed(seed, pkx, msg, msg_len, sig, n, chunk);
    words_be32(seed32, seed);
    for (size_t i = 0; i < n; i++) {
        sc a;
        batch_randomizer(a, seed, (uint64_t)i);
        sc_to_be32(a32 + 32 * i, a);
    }
}
// The api_msm.cu flow of s256_schnorr_batch_verify, sequentially: seed, then per chunk the MSM rows and the scalar sum,
// the rows through sim_msm (projective partial), then + (sum a_i s_i) G and the identity test.
EXPORT void sim_schnorr_batch_verify(const uint8_t *pkx, const uint8_t *msg, size_t msg_len, const uint8_t *sig, size_t n,
                                     size_t chunk, uint8_t *ok) {
    if (n == 0) {
        *ok = 1;
        return;
    }
    ensure_tables();
    uint32_t seed[8];
    sim_batch_seed(seed, pkx, msg, msg_len, sig, n, chunk);
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
            sc as;
            bad |= !item_batch_prepare(aff2.data() + 2 * i, k2.data() + 64 * i, as, pkx + 32 * g, msg + msg_len * g, msg_len,
                                       sig + 64 * g, seed, (uint64_t)g);
            sc_add(sum, sum, as);
        }
        for (size_t v = 0; v < 2 * c; v++) {  // canonical affine rows, as sim_msm decodes them into its own scratch
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
