// batch.cuh -- batch verification: the per-row item functions of s256_schnorr_batch_verify (BIP-340 "Batch
// Verification") and s256_ecdsa_recoverable_batch_verify (api_msm.cu).  A batch of u BIP-340 signatures is accepted when
//
//     (sum a_i s_i) G  -  sum a_i R_i  -  sum (a_i e_i) P_i  =  O        (a_0 = 1, the other a_i random, 128-bit)
//
// with R_i = lift_x(r_i), P_i = lift_x(pkx_i), e_i the BIP-340 challenge.  A batch of u recoverable ECDSA signatures
// r||s||v is accepted when
//
//     (sum a_i u1_i) G  +  sum (a_i u2_i) Q_i  -  sum a_i R_i  =  O       (the same a_i)
//
// with R_i = RecoverPoint(r_i, v_i), u1_i = e_i / s_i, u2_i = r_i / s_i.  The randomizers are derived from a hash tree
// over all the inputs, so that the batch can be hashed in parallel and in chunks:
//
//     leaf_i = SHA-256(pkx_i || sig_i || msg_i)              (BIP-340; msg_i of any length, >= 96 bytes hashed)
//              SHA-256(pk65_i || digest32_i || sig65_i)      (ECDSA)
//     node   = SHA-256(left || right); level 0 = leaves, pairs (2j, 2j + 1) upward, an unpaired last node moves up
//              unchanged; root = the last node
//     seed   = tagged_hash(tag, root || be64(u)),  tag = "S256/BIP0340/batch" or "S256/ECDSA/batch"
//     a_i    = int(SHA-256(seed || be64(i))[0:16]), 1 if that is 0;  a_0 = 1
//
// Node j of level L covers the leaves [j 2^L, (j + 1) 2^L), so the roots of chunks of 2^k rows are the nodes of
// level k and their tree is the rest of the full tree: the seed does not depend on the chunk size.
#pragma once
#include "kernels.cuh"

namespace s256 {

#define S256_BATCH_TAG_BIP340 "S256/BIP0340/batch"
#define S256_BATCH_TAG_ECDSA "S256/ECDSA/batch"

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
// leaf = SHA-256(pk65 || digest32 || sig65), 162 bytes: three blocks, the padding in the last one
S256_HD uint8_t ecdsa_leaf_byte(const uint8_t *pk65, const uint8_t *digest32, const uint8_t *sig65, int k) {
    if (k < 65) return pk65[k];
    if (k < 97) return digest32[k - 65];
    if (k < 162) return sig65[k - 97];
    return k == 162 ? 0x80 : 0;
}
S256_HD void batch_leaf_ecdsa(uint32_t out[8], const uint8_t *pk65, const uint8_t *digest32, const uint8_t *sig65) {
    uint32_t w[16];
    sha_iv(out);
#pragma unroll
    for (int b = 0; b < 3; b++) {
#pragma unroll
        for (int j = 0; j < 16; j++) {
            const int k = 64 * b + 4 * j;
            w[j] = ((uint32_t)ecdsa_leaf_byte(pk65, digest32, sig65, k) << 24) |
                   ((uint32_t)ecdsa_leaf_byte(pk65, digest32, sig65, k + 1) << 16) |
                   ((uint32_t)ecdsa_leaf_byte(pk65, digest32, sig65, k + 2) << 8) | ecdsa_leaf_byte(pk65, digest32, sig65, k + 3);
        }
        if (b == 2) w[15] = 162 * 8;
        sha256_compress(out, w);
    }
}
// seed = tagged_hash(tag, root || be64(n)); tag is NUL-terminated
S256_HD void batch_seed(uint32_t seed[8], const uint32_t root[8], uint64_t n, const char *tag = S256_BATCH_TAG_BIP340) {
    size_t tag_len = 0;
    while (tag[tag_len]) tag_len++;
    uint8_t th[32], tail[40], d[32];
    sha_stream c;
    sha_init(c);
    sha_update(c, reinterpret_cast<const uint8_t *>(tag), tag_len);
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
// not an x-coordinate of the curve, s >= n, and a message row that cannot be read (row_ok = 0, msg_offsets).  A
// rejected row gets G with the scalar 0 and as = 0.  Returns 1 if valid.
S256_HD uint32_t item_batch_prepare(apt *aff2, uint8_t *k2, sc &as, const uint8_t *pkx32, const uint8_t *msg, size_t msg_len,
                                    const uint8_t *sig64, const uint32_t seed[8], uint64_t gi, uint32_t row_ok = 1u) {
    apt P, R;
    sc s, e, a, ae;
    uint32_t ok = row_ok & item_decode_xonly(P, pkx32);
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

// ECDSA row gi, first half (one row per thread: the square root wants every thread the GPU has): -R at aff2[0] with
// R = RecoverPoint(r, v) (v < 4, r < n, r + n < p if v & 2, x on the curve; point_s11n.go:245-282) and Q at aff2[1],
// decoded like secec.NewPublicKey (04 || X || Y, canonical, on the curve).  Returns 1 if both decode.
S256_HD uint32_t item_ecdsa_batch_points(apt *aff2, const uint8_t *pk65, const uint8_t *sig65) {
    apt Q, R;
    uint32_t ok = item_decode_uncompressed(Q, pk65);
    ok &= item_decode_recover(R, sig65);
    fe_neg(R.y, R.y);
    fe_normalize(R.y, R.y);
    aff2[0] = R;
    aff2[1] = Q;
    return ok;
}
// ECDSA row gi, second half, given p = item_ecdsa_parse of the row (r, s in [1, n), low-s with
// FLAG_REJECT_MALLEABLE, e = the leftmost 32 digest bytes mod n), w = 1 / p.s and points_ok from
// item_ecdsa_batch_points: the MSM scalars a (for -R) and a u2 (for Q) at k2[0..64), and au1 = a u1 for the G side.
// The row holds iff u1 G + u2 Q - R = O, which is r^-1 (s R - e G) = Q, the key recoverable Verify compares
// (secec/ecdsa.go:221-227).  A rejected row gets G twice with the scalar 0 and au1 = 0.  Returns 1 if valid.
S256_HD uint32_t item_ecdsa_batch_prepare(apt *aff2, uint8_t *k2, sc &au1, const ecdsa_parsed &p, const sc &w,
                                          uint32_t points_ok, const uint32_t seed[8], uint64_t gi) {
    const uint32_t ok = p.valid & points_ok;
    sc a, u1, u2, au2;
    batch_randomizer(a, seed, gi);
    sc_mul(u1, p.e, w);
    sc_mul(u2, p.r, w);
    sc_mul(au1, a, u1);
    sc_mul(au2, a, u2);
    if (!ok) {
        aff2[0] = aff2[1] = apt_generator();
        a = au1 = au2 = sc_zero();
    }
    sc_to_be32(k2, a);
    sc_to_be32(k2 + 32, au2);
    return ok;
}
// Rows t, t + stride, ..., t + (K - 1) stride of a chunk of n rows starting at batch row off: one s^-1 chain shared by
// the K rows (Montgomery's trick, as group_ecdsa_scalars), sum = their sum of a u1.  pvalid[i] is the result of
// item_ecdsa_batch_points for row i, whose points are already at aff2[2i, 2i + 2).  Returns 1 if all K rows are valid.
template <int K>
S256_HD uint32_t group_ecdsa_batch_prepare(size_t t, size_t stride, size_t n, size_t off, const uint8_t *digest32,
                                           const uint8_t *sig65, uint32_t flags, const uint8_t *pvalid,
                                           const uint32_t seed[8], apt *aff2, uint8_t *k2, sc &sum) {
    sc pre[K];
    sc run = sc_one();
    ecdsa_parsed p;
    for (int m = 0; m < K; m++) {
        size_t i = t + (size_t)m * stride;
        pre[m] = run;
        if (i < n) {
            item_ecdsa_parse(p, digest32 + 32 * i, sig65 + 65 * i, flags);
            sc_mul(run, run, p.s);
        }
    }
    sc inv;
    sc_invert(inv, run);
    uint32_t ok = 1;
    sum = sc_zero();
    for (int m = K - 1; m >= 0; m--) {
        size_t i = t + (size_t)m * stride;
        if (i >= n) continue;
        item_ecdsa_parse(p, digest32 + 32 * i, sig65 + 65 * i, flags);
        sc w, au1;
        sc_mul(w, inv, pre[m]);
        sc_mul(inv, inv, p.s);
        ok &= item_ecdsa_batch_prepare(aff2 + 2 * i, k2 + 64 * i, au1, p, w, pvalid[i], seed, (uint64_t)(off + i));
        sc_add(sum, sum, au1);
    }
    return ok;
}

}  // namespace s256
