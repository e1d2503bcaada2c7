// ecdsa_batch_sim.cpp -- TEST INFRASTRUCTURE ONLY: the recoverable ECDSA batch verification of api_msm.cu
// (s256_ecdsa_recoverable_batch_verify) on the CPU.
//
// Builds on hostsim.cpp (included whole, so this library carries its own copy of the simulation) and runs the
// item functions of csrc/batch.cuh in the order the kernels run them, one "thread" at a time: per chunk the points one
// row at a time (k_ecdsa_batch_points), then the scalars in groups of K rows sharing one inversion
// (k_ecdsa_batch_prepare<K>, with the device's strided layout).  Each chunk's MSM rows go through hostsim.cpp's sim_msm,
// the same Pippenger flow chunk_msm_body runs on the device.
#include "hostsim.cpp"
#include "../../secp256k1-voi_b200/csrc/batch.cuh"

// Pass 1 with chunks of `chunk` rows: leaves, one root per chunk, the tree of the roots, the seed.
static void sim_ecdsa_seed(uint32_t seed[8], const uint8_t *pk, const uint8_t *dg, const uint8_t *sig, size_t n,
                           size_t chunk) {
    size_t chunks = (n + chunk - 1) / chunk;
    std::vector<uint32_t> roots(8 * chunks), leaves(8 * chunk);
    for (size_t k = 0; k < chunks; k++) {
        size_t off = k * chunk, c = std::min(chunk, n - off);
        for (size_t i = 0; i < c; i++)
            batch_leaf_ecdsa(leaves.data() + 8 * i, pk + 65 * (off + i), dg + 32 * (off + i), sig + 65 * (off + i));
        batch_tree_fold(leaves.data(), c);
        std::copy(leaves.begin(), leaves.begin() + 8, roots.begin() + 8 * k);
    }
    batch_tree_fold(roots.data(), chunks);
    batch_seed(seed, roots.data(), (uint64_t)n, S256_BATCH_TAG_ECDSA);
}
// the seed (32 B) and every a_i (32 B big-endian) for chunks of `chunk` rows
EXPORT void sim_ecdsa_batch_randomizers(const uint8_t *pk, const uint8_t *dg, const uint8_t *sig, size_t n, size_t chunk,
                                        uint8_t *seed32, uint8_t *a32) {
    uint32_t seed[8];
    sim_ecdsa_seed(seed, pk, dg, sig, n, chunk);
    words_be32(seed32, seed);
    for (size_t i = 0; i < n; i++) {
        sc a;
        batch_randomizer(a, seed, (uint64_t)i);
        sc_to_be32(a32 + 32 * i, a);
    }
}

// every group of one chunk of c rows; returns 1 if all rows are valid
template <int K>
static uint32_t sim_groups(size_t c, size_t off, const uint8_t *dg, const uint8_t *sig, uint32_t flags, const uint8_t *pvalid,
                           const uint32_t seed[8], apt *aff2, uint8_t *k2, sc &sum) {
    const size_t stride = (c + K - 1) / K;
    uint32_t ok = 1;
    for (size_t t = 0; t < stride; t++) {
        sc part;
        ok &= group_ecdsa_batch_prepare<K>(t, stride, c, off, dg, sig, flags, pvalid, seed, aff2, k2, part);
        sc_add(sum, sum, part);
    }
    return ok;
}
// The api_msm.cu flow of s256_ecdsa_recoverable_batch_verify, sequentially, with chunks of `chunk` rows and inversion
// groups of k rows (0: as the device picks them for the chunk size, inv_k_for).  Writes what
// s256_debug_ecdsa_batch_rows returns (seed32, k64, pts128, sum32, rejected; all optional) and the verdict.
EXPORT void sim_ecdsa_batch(const uint8_t *pk, const uint8_t *dg, const uint8_t *sig, uint32_t flags, size_t n, size_t chunk,
                            int k, uint8_t *seed32, uint8_t *k64, uint8_t *pts128, uint8_t *sum32, uint8_t *rejected,
                            uint8_t *ok) {
    if (n == 0) {
        *ok = 1;
        return;
    }
    ensure_tables();
    uint32_t seed[8];
    sim_ecdsa_seed(seed, pk, dg, sig, n, chunk);
    uint32_t good = 1;
    sc sum = sc_zero();
    pt acc;
    pt_set_identity(acc);
    for (size_t off = 0; off < n; off += chunk) {
        size_t c = std::min(chunk, n - off);
        const uint8_t *cpk = pk + 65 * off, *cdg = dg + 32 * off, *csig = sig + 65 * off;
        std::vector<apt> aff2(2 * c);
        std::vector<uint8_t> pvalid(c), k2(64 * c), pt65(65 * 2 * c);
        for (size_t i = 0; i < c; i++) pvalid[i] = (uint8_t)item_ecdsa_batch_points(aff2.data() + 2 * i, cpk + 65 * i, csig + 65 * i);
        int kk = k ? k : (c >= ((size_t)1 << 19) ? 32 : (c >= ((size_t)1 << 16) ? 4 : 1));
        if (kk == 1)
            good &= sim_groups<1>(c, off, cdg, csig, flags, pvalid.data(), seed, aff2.data(), k2.data(), sum);
        else if (kk == 4)
            good &= sim_groups<4>(c, off, cdg, csig, flags, pvalid.data(), seed, aff2.data(), k2.data(), sum);
        else
            good &= sim_groups<32>(c, off, cdg, csig, flags, pvalid.data(), seed, aff2.data(), k2.data(), sum);
        for (size_t v = 0; v < 2 * c; v++) {  // canonical affine rows, as sim_msm decodes them into its own scratch
            pt65[65 * v] = 4;
            fe_to_be32(pt65.data() + 65 * v + 1, aff2[v].x);
            fe_to_be32(pt65.data() + 65 * v + 33, aff2[v].y);
            if (pts128) std::memcpy(pts128 + 64 * (2 * off + v), pt65.data() + 65 * v + 1, 64);
        }
        if (k64) std::memcpy(k64 + 64 * off, k2.data(), 64 * c);
        uint8_t out65[65], st = 0, part96[96];
        sim_msm(k2.data(), pt65.data(), 2 * c, 1, 0, out65, &st, part96);
        pt part;
        pt_from_be96(part, part96);
        pt_add(acc, acc, part);
    }
    if (seed32) words_be32(seed32, seed);
    if (sum32) sc_to_be32(sum32, sum);
    if (rejected) *rejected = (uint8_t)(good == 0);
    pt sg;
    item_base_mult_ct(sg, sum, g_ct.data());
    pt_add(acc, acc, sg);
    *ok = (uint8_t)(good && fe_is_zero(acc.z));
}
