// batch.cuh -- BIP-340 batch verification (BIP-340 "Batch Verification"): the per-row item functions of
// s256_schnorr_batch_verify (api_msm.cu).  A batch of u signatures is accepted when
//
//     (sum a_i s_i) G  -  sum a_i R_i  -  sum (a_i e_i) P_i  =  O        (a_0 = 1, the other a_i random, 128-bit)
//
// with R_i = lift_x(r_i), P_i = lift_x(pkx_i), e_i the BIP-340 challenge.  The randomizers are derived from a hash
// tree over all the inputs, so that the batch can be hashed in parallel and in chunks:
//
//     leaf_i = SHA-256(pkx_i || sig_i || msg_i)
//     node   = SHA-256(left || right); level 0 = leaves, pairs (2j, 2j + 1) upward, an unpaired last node moves up
//              unchanged; root = the last node
//     seed   = tagged_hash("S256/BIP0340/batch", root || be64(u))
//     a_i    = int(SHA-256(seed || be64(i))[0:16]), 1 if that is 0;  a_0 = 1
//
// Node j of level L covers the leaves [j 2^L, (j + 1) 2^L), so the roots of chunks of 2^k rows are the nodes of
// level k and their tree is the rest of the full tree: the seed does not depend on the chunk size.
#pragma once
#include "kernels.cuh"

namespace s256 {

// leaf = SHA-256(pkx32 || sig64 || msg[0, msg_len)) as big-endian words
S256_HD void batch_leaf(uint32_t out[8], const uint8_t *pkx32, const uint8_t *sig64, const uint8_t *msg, size_t msg_len) {
    if (msg_len == 32) {  // 128 bytes: two data blocks and the padding block, all in words
        uint32_t w[16];
        sha_iv(out);
        be32_words(w, pkx32);
        be32_words(w + 8, sig64);
        sha256_compress(out, w);
        be32_words(w, sig64 + 32);
        be32_words(w + 8, msg);
        sha256_compress(out, w);
        w[0] = 0x80000000u;
#pragma unroll
        for (int i = 1; i < 15; i++) w[i] = 0;
        w[15] = 128 * 8;
        sha256_compress(out, w);
        return;
    }
    sha_stream c;
    uint8_t d[32];
    sha_init(c);
    sha_update(c, pkx32, 32);
    sha_update(c, sig64, 64);
    sha_update(c, msg, msg_len);
    sha_final(c, d);
    be32_words(out, d);
}
// out = SHA-256(l || r), 64 bytes; out may alias l or r
S256_HD void batch_node(uint32_t out[8], const uint32_t l[8], const uint32_t r[8]) {
    uint32_t h[8], w[16];
    sha_iv(h);
#pragma unroll
    for (int i = 0; i < 8; i++) {
        w[i] = l[i];
        w[8 + i] = r[i];
    }
    sha256_compress(h, w);
    w[0] = 0x80000000u;
#pragma unroll
    for (int i = 1; i < 15; i++) w[i] = 0;
    w[15] = 64 * 8;
    sha256_compress(h, w);
#pragma unroll
    for (int i = 0; i < 8; i++) out[i] = h[i];
}
// The tree rule over m >= 1 nodes of 8 words, level by level in place: the root ends up in nodes[0..8).
S256_HD void batch_tree_fold(uint32_t *nodes, size_t m) {
    while (m > 1) {
        size_t up = (m + 1) / 2;
        for (size_t j = 0; j < up; j++) {
            if (2 * j + 1 < m) {
                batch_node(nodes + 8 * j, nodes + 16 * j, nodes + 16 * j + 8);
            } else {
                for (int k = 0; k < 8; k++) nodes[8 * j + k] = nodes[16 * j + k];
            }
        }
        m = up;
    }
}
// seed = tagged_hash("S256/BIP0340/batch", root || be64(n))
S256_HD void batch_seed(uint32_t seed[8], const uint32_t root[8], uint64_t n) {
    const char tag[] = "S256/BIP0340/batch";
    uint8_t th[32], tail[40], d[32];
    sha_stream c;
    sha_init(c);
    sha_update(c, reinterpret_cast<const uint8_t *>(tag), sizeof(tag) - 1);
    sha_final(c, th);
    words_be32(tail, root);
    for (int k = 0; k < 8; k++) tail[32 + k] = (uint8_t)(n >> (56 - 8 * k));
    sha_init(c);
    sha_update(c, th, 32);
    sha_update(c, th, 32);
    sha_update(c, tail, 40);
    sha_final(c, d);
    be32_words(seed, d);
}
// a_i: 1 for i = 0, else the first 16 bytes of SHA-256(seed || be64(i)) as a big-endian integer (1 if that is 0)
S256_HD void batch_randomizer(sc &a, const uint32_t seed[8], uint64_t i) {
    a = sc_one();
    if (i == 0) return;
    uint32_t h[8], w[16];
    sha_iv(h);
#pragma unroll
    for (int k = 0; k < 8; k++) w[k] = seed[k];
    w[8] = (uint32_t)(i >> 32);
    w[9] = (uint32_t)i;
    w[10] = 0x80000000u;
#pragma unroll
    for (int k = 11; k < 15; k++) w[k] = 0;
    w[15] = 40 * 8;
    sha256_compress(h, w);
    if ((h[0] | h[1] | h[2] | h[3]) == 0) return;
    a.v[0] = h[3];
    a.v[1] = h[2];
    a.v[2] = h[1];
    a.v[3] = h[0];
}

// Row gi of the batch: the MSM rows -R (scalar a) and -P (scalar a e) at aff2[0..2) and k2[0..64), and as = a s for
// the G side.  Negating the points keeps the R scalar at 128 bits, so its second endomorphism half is (almost) all
// zero digits.  The same rejections as item_decode_xonly and item_schnorr_scalars: the key does not lift, r >= p or
// not an x-coordinate of the curve, s >= n.  A rejected row gets G with the scalar 0 and as = 0.  Returns 1 if valid.
S256_HD uint32_t item_batch_prepare(apt *aff2, uint8_t *k2, sc &as, const uint8_t *pkx32, const uint8_t *msg, size_t msg_len,
                                    const uint8_t *sig64, const uint32_t seed[8], uint64_t gi) {
    apt P, R;
    sc s, e, a, ae;
    uint32_t ok = item_decode_xonly(P, pkx32);
    ok &= item_decode_xonly(R, sig64);  // R = lift_x(r): r < p, and r^3 + 7 a square
    ok &= 1u - sc_from_be32(s, sig64 + 32);
    item_schnorr_challenge(e, sig64, pkx32, msg, msg_len);
    batch_randomizer(a, seed, gi);
    sc_mul(ae, a, e);
    sc_mul(as, a, s);
    fe_neg(R.y, R.y);
    fe_normalize(R.y, R.y);
    fe_neg(P.y, P.y);
    fe_normalize(P.y, P.y);
    if (!ok) {
        R = P = apt_generator();
        a = ae = as = sc_zero();
    }
    aff2[0] = R;
    aff2[1] = P;
    sc_to_be32(k2, a);
    sc_to_be32(k2 + 32, ae);
    return ok;
}

}  // namespace s256
