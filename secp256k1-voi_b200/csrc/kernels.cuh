// kernels.cuh -- the batched secp256k1 kernels (sm_100a).
//
// One item per thread for the curve work; K items per thread where a
// Montgomery-trick batched inversion amortises a Fermat chain.  Every kernel
// body is a plain S256_HD "item" function plus a thin __global__ wrapper, so
// tests/hostsim can run the identical logic on a CPU-only box.
//
// Device scratch (all per item, SoA, see api.cu):
//   aff   apt   decoded / validated affine input point           64 B
//   u1    sc    G-side scalar                                    32 B
//   dig1/2 int8 [ND][n] signed window digits of the GLV halves   2*ND B
//   sfl   u8    bit0 scalars-valid, bit1 negate P, bit2 negate lambda*P
//   tbl   pt    multiples 1..TS of P (see item_dsm_table)        96*DSM_TSTRIDE B
//   res   pt    projective result                                96 B
#pragma once
#include "fe.cuh"
#include "point.cuh"
#include "jac.cuh"
#include "sc.cuh"
#include "sha256.cuh"

namespace s256 {

// per-item window for the variable-base half of u1*G + u2*P
#ifndef S256_W
#define S256_W 5
#endif
constexpr int DSM_W = S256_W;
constexpr int DSM_ND = glv_recode<DSM_W>::ND;  // digits per 128-bit half
constexpr int DSM_TS = 1 << (DSM_W - 1);       // table entries 1..TS
// The verification ladder runs in Jacobian coordinates over an AFFINE per-item table (jac.cuh) unless S256_DSM_RCB
// asks for the round-1 form (complete projective formulas, projective table).  Per-item table scratch in units of
// sizeof(pt): the Jacobian build keeps the TS affine rows the ladder reads (64 B each), then the TS - 2 Z ratios of
// the co-Z chain that built them (32 B each; the first slot holds the common denominator once the rows are scaled).
#ifndef S256_DSM_RCB
#define S256_DSM_JAC 1
static_assert(DSM_TS >= 4, "the co-Z table needs at least two chain steps (item_dsm_table)");
constexpr int DSM_TSTRIDE = (64 * DSM_TS + 32 * (DSM_TS - 2) + 95) / 96;
#else
constexpr int DSM_TSTRIDE = DSM_TS;
#endif
// fixed-base comb for the G half of the verification ladder: COMB_NW windows of COMB_WB bits, SIGNED
// digits in [-(2^(WB-1) - 1), 2^(WB-1)], entries (j + 1) * 2^(WB*w) * G for j = 0 .. 2^(WB-1) - 1.
// No doublings, one mixed addition per window, so wider windows are fewer additions and the only
// price is table memory -- which this GPU has: WB = 22 is 12 windows of 2^21 entries = 1.5 GiB of the
// 180 GB (WB = 16: 16 windows, 32 MiB), one 64-byte gather per window, public data.
#ifndef S256_COMB_WB
#define S256_COMB_WB 22
#endif
constexpr int COMB_WB = S256_COMB_WB;
constexpr int COMB_NW = (257 + COMB_WB - 1) / COMB_WB;  // 256 scalar bits + the recoding carry
constexpr int COMB_SZ = 1 << (COMB_WB - 1);
// signed digit w of u1 (carry in / out); the top window absorbs the last carry
S256_HD int32_t comb_digit(const sc &u1, int w, uint32_t &carry) {
    int bit = w * COMB_WB;
    uint32_t v = 0;
    if (bit < 256) {
        v = u1.v[bit >> 5] >> (bit & 31);
        if ((bit & 31) + COMB_WB > 32 && (bit >> 5) + 1 < 8) v |= u1.v[(bit >> 5) + 1] << (32 - (bit & 31));
        v &= (1u << COMB_WB) - 1u;
    }
    v += carry;                                         // 0 .. 2^WB
    carry = (v + (uint32_t)COMB_SZ - 1u) >> COMB_WB;    // 1 iff v > 2^(WB-1)
    return (int32_t)v - (int32_t)(carry << COMB_WB);
}
// constant-time fixed-base tables: signed WB-bit digits in [-(2^(WB-1) - 1), 2^(WB-1)]; entries
// (j + 1) * 2^(WB*w) * G for j = 0 .. 2^(WB-1) - 1.  Two window sizes are resident: WB = 6
// (43 windows x 32 entries = 88 064 bytes, twice per SM) for the throughput kernel, and WB = 5
// (52 x 16 = 53 248 bytes) for the lane-split small-batch kernels, where every CTA stages its own copy
// of the table and a smaller one starts sooner.  WB = 7 is 3 % faster at 2^20 and 2x slower at 4096.
template <int WB>
struct ct_cfg {
    static constexpr int NW = (257 + WB - 1) / WB;  // 256 scalar bits + the recoding carry
    static constexpr int SZ = 1 << (WB - 1);
};
#ifndef S256_CT_WB
#define S256_CT_WB 6
#endif
#ifndef S256_CT_WB_SMALL
#define S256_CT_WB_SMALL 5
#endif
constexpr int CT_WB = S256_CT_WB, CT_WB_SMALL = S256_CT_WB_SMALL;
constexpr int CT_NW = ct_cfg<CT_WB>::NW;  // for the work model (s256_mac32_per_item)
// digit w of the recoding: bits [WB*w, WB*w + WB) of k plus the incoming carry
template <int CT_WB>
S256_HD uint32_t ct_window_bits(const sc &k, int w) {
    int bit = w * CT_WB;
    if (bit >= 256) return 0u;
    int limb = bit >> 5, sh = bit & 31;
    uint32_t v = k.v[limb] >> sh;
    if (sh + CT_WB > 32 && limb + 1 < 8) v |= k.v[limb + 1] << (32 - sh);
    return v & ((1u << CT_WB) - 1u);
}
// constant-time variable-base ladder (ScalarMult / ECDH): signed window
#ifndef S256_CTW
#define S256_CTW 4
#endif
constexpr int CTM_W = S256_CTW;
constexpr int CTM_ND = glv_recode<CTM_W>::ND;
constexpr int CTM_TS = 1 << (CTM_W - 1);
static_assert(CTM_TS * (96 + 64 + 32) <= DSM_TSTRIDE * 96, "the ct ladder shares the per-item table scratch of the vartime ladder");

enum : uint8_t { ST_INVALID = 0, ST_OK = 1, ST_IDENTITY = 2 };
enum : uint32_t { FLAG_REJECT_MALLEABLE = 1u };
enum : uint8_t { SFL_VALID = 1, SFL_NEG1 = 2, SFL_NEG2 = 4 };

// ---------------------------------------------------------------------------
// table generation: out[w * 2^wb + d] = d * 2^(wb*w) * G, affine; d = 0 unused.
// Plain double-and-add from G with a per-thread Fermat inversion: init only.
// (internal/gentable/point_mul_table.go:16-49 produces the same multiples.)
// ---------------------------------------------------------------------------
S256_HD void item_gen_multiple(apt &out, uint32_t w, uint32_t d, int wb) {
    // d * 2^(wb*w) * G; d may use up to wb + 1 bits (the signed ct table needs d = 2^(wb-1) = 8 with wb = 4)
    if (d == 0) {
        out.x = fe_zero();
        out.y = fe_zero();
        return;
    }
    apt g = apt_generator();
    pt acc;
    pt_set_identity(acc);
    for (int b = wb; b >= 0; b--) {
        pt_double(acc, acc);
        if ((d >> b) & 1u) pt_add_mixed(acc, acc, g.x, g.y);
    }
    int nd = wb * (int)w;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int k = 0; k < nd; k++) pt_double(acc, acc);
    fe zi;
    fe_invert(zi, acc.z);
    fe_mul(out.x, acc.x, zi);
    fe_mul(out.y, acc.y, zi);
    fe_normalize(out.x, out.x);
    fe_normalize(out.y, out.y);
}

// ---------------------------------------------------------------------------
// point decoding (SEC 1).  Invalid inputs are replaced by G so that the curve
// kernels run on sane data; the valid byte carries the verdict.
// ---------------------------------------------------------------------------
// point_s11n.go:178-213 -- 04 || X || Y, canonical coordinates, on curve
S256_HD uint8_t item_decode_uncompressed(apt &out, const uint8_t *b) {
    apt a;
    fe_from_be32(a.x, b + 1);
    fe_from_be32(a.y, b + 33);
    uint32_t ok = (uint32_t)(b[0] == 0x04) & fe_limbs_are_canonical(a.x) & fe_limbs_are_canonical(a.y);
    ok &= apt_on_curve(a);
    apt g = apt_generator();
    fe_cmov(out.x, g.x, a.x, ok);
    fe_cmov(out.y, g.y, a.y, ok);
    return (uint8_t)ok;
}
// point_s11n.go:140-172 -- x canonical, y = sqrt(x^3 + 7) with the requested
// parity.  Used for BIP-340 lift_x (parity 0, schnorr.go:257-275) and
// RecoverPoint (point_s11n.go:245-282).
S256_HD uint8_t item_decompress(apt &out, const fe &x, uint32_t x_ok, uint32_t want_odd) {
    fe yy, y, yn;
    fe_curve_rhs(yy, x);
    uint32_t ok = x_ok & fe_sqrt(y, yy);
    fe_normalize(y, y);
    fe_neg(yn, y);
    fe_normalize(yn, yn);
    uint32_t flip = (y.v[0] & 1u) ^ (want_odd & 1u);
    fe_cmov(y, y, yn, flip);
    apt g = apt_generator();
    fe_cmov(out.x, g.x, x, ok);
    fe_cmov(out.y, g.y, y, ok);
    return (uint8_t)ok;
}

// ---------------------------------------------------------------------------
// scalar preparation for R = u1*G + u2*P: GLV-split u2, sign-normalise,
// recode both halves into signed W-bit digits.
// ---------------------------------------------------------------------------
S256_HD void item_store_scalars(const sc &u1, const sc &u2, uint32_t valid, size_t i, size_t n, sc *u1_out,
                                int8_t *dig1, int8_t *dig2, uint8_t *sfl) {
    uint32_t m1[4], m2[4], neg1, neg2;
    sc_split_glv_abs(m1, neg1, m2, neg2, u2);
    int8_t d1[DSM_ND], d2[DSM_ND];
    glv_recode<DSM_W>::run(d1, m1);
    glv_recode<DSM_W>::run(d2, m2);
#pragma unroll
    for (int s = 0; s < DSM_ND; s++) {
        dig1[(size_t)s * n + i] = d1[s];
        dig2[(size_t)s * n + i] = d2[s];
    }
    u1_out[i] = u1;
    sfl[i] = (uint8_t)((valid ? SFL_VALID : 0) | (neg1 ? SFL_NEG1 : 0) | (neg2 ? SFL_NEG2 : 0));
}

// secec/ecdsa.go:392-470 steps 1-4 and secec/s11n.go:129-145: r, s canonical
// and non-zero, optional low-s rule (ecdsa.go:212), e = leftmost 32 digest
// bytes mod n (ecdsa.go:477-486).  s is replaced by 1 when invalid so the
// shared inversion stays well defined.
struct ecdsa_parsed {
    sc r, s, e;
    uint32_t valid;
};
S256_HD void item_ecdsa_parse(ecdsa_parsed &o, const uint8_t *digest32, const uint8_t *sig64, uint32_t flags) {
    uint32_t rr = sc_from_be32(o.r, sig64);
    uint32_t sr = sc_from_be32(o.s, sig64 + 32);
    uint32_t ok = (1u - rr) & (1u - sr) & (1u - sc_is_zero(o.r)) & (1u - sc_is_zero(o.s));
    if (flags & FLAG_REJECT_MALLEABLE) ok &= 1u - sc_is_gt_half_n(o.s);
    sc_from_be32(o.e, digest32);
    sc one = sc_one();
    sc_cmov(o.s, one, o.s, ok);
    o.valid = ok;
}

// K items per thread, strided by `stride` so that a warp touches consecutive
// items: Montgomery's trick shares one x^(n-2) chain between K inversions.
template <int K>
S256_HD void group_ecdsa_scalars(size_t t, size_t stride, size_t n, const uint8_t *digest32, const uint8_t *sig64,
                                 uint32_t flags, sc *u1_out, int8_t *dig1, int8_t *dig2, uint8_t *sfl) {
    sc pre[K];
    sc run = sc_one();
    ecdsa_parsed p;
    for (int m = 0; m < K; m++) {
        size_t i = t + (size_t)m * stride;
        pre[m] = run;
        if (i < n) {
            item_ecdsa_parse(p, digest32 + 32 * i, sig64 + 64 * i, flags);
            sc_mul(run, run, p.s);
        }
    }
    sc inv;
    sc_invert(inv, run);
    for (int m = K - 1; m >= 0; m--) {
        size_t i = t + (size_t)m * stride;
        if (i >= n) continue;
        item_ecdsa_parse(p, digest32 + 32 * i, sig64 + 64 * i, flags);
        sc sinv, u1, u2;
        sc_mul(sinv, inv, pre[m]);
        sc_mul(inv, inv, p.s);
        sc_mul(u1, p.e, sinv);  // ecdsa.go:429
        sc_mul(u2, p.r, sinv);  // ecdsa.go:430
        item_store_scalars(u1, u2, p.valid, i, n, u1_out, dig1, dig2, sfl);
    }
}

// raw u1, u2 (DoubleScalarMultBasepointVartime called directly): reduce like
// NewScalarFromBytes.
S256_HD void item_plain_scalars(size_t i, size_t n, const uint8_t *u1b, const uint8_t *u2b, sc *u1_out, int8_t *dig1,
                                int8_t *dig2, uint8_t *sfl) {
    sc u1, u2;
    sc_from_be32(u1, u1b + 32 * i);
    sc_from_be32(u2, u2b + 32 * i);
    item_store_scalars(u1, u2, 1u, i, n, u1_out, dig1, dig2, sfl);
}

// BIP-340 lift_x: x-only key, even y (secec/bitcoin/schnorr.go:257-275)
S256_HD uint8_t item_decode_xonly(apt &out, const uint8_t *pkx32) {
    fe x;
    fe_from_be32(x, pkx32);
    return item_decompress(out, x, fe_limbs_are_canonical(x), 0u);
}
// RecoverPoint (point_s11n.go:245-282): x = r (+ n if v & 2), parity v & 1.
// r + n must stay below p -- the reference's round-trip sanity check.
S256_HD uint8_t item_decode_recover(apt &out, const uint8_t *sig65) {
    uint32_t v = sig65[64];
    sc r;
    uint32_t ok = 1u - sc_from_be32(r, sig65);
    ok &= (uint32_t)(v < 4);
    fe x;
#pragma unroll
    for (int k = 0; k < 8; k++) x.v[k] = r.v[k];
    if (v & 2u) {
        fe nn = fe_group_order();
        uint64_t acc = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            acc = (acc >> 32) + x.v[k] + nn.v[k];
            x.v[k] = (uint32_t)acc;
        }
        ok &= (1u - (uint32_t)(acc >> 32)) & fe_limbs_are_canonical(x);
    }
    return item_decompress(out, x, ok, v & 1u);
}

// secec/ecdsa.go:244-282: u1 = -e / r, u2 = s / r over r||s||v rows (65 B),
// K items per thread sharing one inversion.
template <int K>
S256_HD void group_recover_scalars(size_t t, size_t stride, size_t n, const uint8_t *digest32, const uint8_t *sig65,
                                   sc *u1_out, int8_t *dig1, int8_t *dig2, uint8_t *sfl) {
    sc pre[K];
    sc run = sc_one();
    const sc one = sc_one();
    ecdsa_parsed p;
    for (int m = 0; m < K; m++) {
        size_t i = t + (size_t)m * stride;
        pre[m] = run;
        if (i < n) {
            item_ecdsa_parse(p, digest32 + 32 * i, sig65 + 65 * i, 0u);
            sc_cmov(p.r, one, p.r, p.valid);
            sc_mul(run, run, p.r);
        }
    }
    sc inv;
    sc_invert(inv, run);
    for (int m = K - 1; m >= 0; m--) {
        size_t i = t + (size_t)m * stride;
        if (i >= n) continue;
        item_ecdsa_parse(p, digest32 + 32 * i, sig65 + 65 * i, 0u);
        sc_cmov(p.r, one, p.r, p.valid);
        sc rinv, ne, a, b2;
        sc_mul(rinv, inv, pre[m]);
        sc_mul(inv, inv, p.r);
        sc_neg(ne, p.e);
        sc_mul(a, ne, rinv);
        sc_mul(b2, p.s, rinv);
        item_store_scalars(a, b2, p.valid, i, n, u1_out, dig1, dig2, sfl);
    }
}

// e = H_challenge(r || P || m) mod n (secec/bitcoin/schnorr.go:445-446) for one row: sg = r || s, pkx = x(P)
S256_HD void item_schnorr_challenge(sc &e, const uint8_t *sg, const uint8_t *pkx, const uint8_t *m, size_t msg_len) {
    uint8_t eb[32];
    if (msg_len == 32) {  // fixed layout: the tag midstate plus two compressions, all in words
        uint32_t rw[8], pw[8], mw[8], ew[8];
        be32_words(rw, sg);
        be32_words(pw, pkx);
        be32_words(mw, m);
        bip340_tagged_96(ew, TAG_CHALLENGE, rw, pw, mw);
        words_be32(eb, ew);
    } else {
        bip340_challenge(eb, sg, pkx, m, msg_len);
    }
    sc_from_be32(e, eb);
}
// secec/bitcoin/schnorr.go:420-449: r < p, s < n (zero allowed),
// e = H(r||P||m) mod n; R = s*G + (-e)*P (:244-245)
S256_HD void item_schnorr_scalars(size_t i, size_t n, const uint8_t *pkx32, const uint8_t *msg, size_t msg_len,
                                  const uint8_t *sig64, sc *u1_out, int8_t *dig1, int8_t *dig2, uint8_t *sfl) {
    const uint8_t *sg = sig64 + 64 * i;
    fe r;
    fe_from_be32(r, sg);
    sc s, e, ne;
    uint32_t ok = fe_limbs_are_canonical(r) & (1u - sc_from_be32(s, sg + 32));
    item_schnorr_challenge(e, sg, pkx32 + 32 * i, msg + msg_len * i, msg_len);
    sc_neg(ne, e);
    item_store_scalars(s, ne, ok, i, n, u1_out, dig1, dig2, sfl);
}

// ---------------------------------------------------------------------------
// R = u1*G + u2*P, variable time (point_mul_glv.go:307-317 and everything
// under it).  Signed fixed windows with uniform control flow replace the
// reference's zero-digit skipping (a warp only skips when all 32 lanes do).
//   table : [1..TS]P by doublings and mixed additions (P is affine)
//   ladder: ND steps of W doublings + two complete additions, the lambda half
//           reusing the same table through x -> beta*x
//   G half: COMB_NW mixed additions from the precomputed comb, no doublings
// Public data, variable time as in the reference: the group law runs on fe_ops<true> (fe_vt.cuh).
// ---------------------------------------------------------------------------
// a table row as twelve 64-bit loads (register pairs are what the multiplier wants anyway; 128-bit loads would force
// 4-register alignment, which cost more in moves than it saved -- DESIGN.md section 5)
S256_HD void pt_fetch64(pt &r, const pt *p) {
#if defined(__CUDA_ARCH__) && !defined(S256_DSM_LD32)
    const uint2 *q = reinterpret_cast<const uint2 *>(p);
#pragma unroll
    for (int k = 0; k < 4; k++) {
        uint2 a = q[k], b = q[4 + k], c = q[8 + k];
        r.x.v[2 * k] = a.x; r.x.v[2 * k + 1] = a.y;
        r.y.v[2 * k] = b.x; r.y.v[2 * k + 1] = b.y;
        r.z.v[2 * k] = c.x; r.z.v[2 * k + 1] = c.y;
    }
#else
    r = *p;
#endif
}
// public data, variable time as in the reference: the short-ripple field operations of fe_vt.cuh.  (The branch-free
// set in this ladder: 22.74 ms against 21.55, k_dsm at 2^20 -- profiles/r02_variants.json.)
constexpr bool DSM_VT = true;
// (Tried and measured, k_dsm at 2^20: the two table rows of a step copied to shared memory with cp.async during the
// doublings, the digits loaded one step ahead and the comb entry of the next window requested before the current
// addition -- the long-scoreboard waits they remove are 6.9 % of the stall samples, but the extra live values spill
// (236 -> 400 bytes of spill stores under the 128-register cap): 21.34 ms against 21.22-21.39 without.  Not kept.)
#if defined(S256_DSM_JAC)
// an affine table row as eight 64-bit loads
S256_HD void apt_fetch64(apt &r, const apt *p) {
#if defined(__CUDA_ARCH__) && !defined(S256_DSM_LD32)
    const uint2 *q = reinterpret_cast<const uint2 *>(p);
#pragma unroll
    for (int k = 0; k < 4; k++) {
        uint2 a = q[k], b = q[4 + k];
        r.x.v[2 * k] = a.x; r.x.v[2 * k + 1] = a.y;
        r.y.v[2 * k] = b.x; r.y.v[2 * k + 1] = b.y;
    }
#else
    r = *p;
#endif
}
// Jacobian form (jac.cuh).  Table: the multiples [1..TS]P as AFFINE points of an isomorphic curve, all over the COMMON
// denominator Z_all (no inversion), so that every ladder addition is a mixed one.  They are built as a co-Z chain
// (Meloni's ZADDU; libsecp256k1's odd-multiples table with its "global Z" is the same construction):
//   * DBLU from the affine key P gives 2P at Z_2 = 2y and P at that same Z;
//   * for k = 2 .. TS - 1, ZADDU(P, kP) gives (k + 1)P and P again, both at Z_(k+1) = Z_k u_k, u_k = X(P) - X(kP).
// No Z is ever formed: the rows are stored as they come, row k at Z_k, with the ratio u_k.  A backward pass then scales
// row k by (r^2, r^3), r = u_k ... u_(TS-1) = Z_TS / Z_k (row TS and the last copy of P are at Z_TS already), and
// Z_all = Z_TS = 2y r_2.  (X_k r^2, Y_k r^3) are the affine coordinates of kP on y^2 = x^3 + 7 Z_all^6; neither the
// a = 0 doubling nor the mixed addition nor x -> beta x involves b, so the ladder runs there unchanged, and its result
// (X', Y', Z') is (X', Y', Z' Z_all) on secp256k1.
// No step is exceptional: u_k = 0 would mean kP = +-P, i.e. (k -+ 1)P = O with 1 <= k -+ 1 <= TS, impossible on a
// curve of prime order; P itself is never O (every decoder substitutes G for an invalid row) and y != 0.
// Layout of the item's scratch (bytes): [0, 64 TS) rows 1..TS; then u_2 .. u_(TS-1), 32 B each, whose first slot
// holds Z_all once the rows are scaled.  item_dsm_table builds the rows, item_dsm_ladder runs the ladder over them;
// item_dsm is the composition.
// (Round 2 first divided every row by its own Z -- one safegcd inversion per item through Montgomery's trick, 20.01 ms
// at 2^20; then one inversion per CTA, 19.14 ms, with 6 % of the warp time spent at the barrier around it; then
// doublings and mixed additions with prefix / suffix products of their Z's for the common denominator, 18.14 ms.)
constexpr int DSM_U_OFF = 64 * DSM_TS;  // byte offset of the ratios (and of Z_all) in the item's scratch
template <class F>
S256_HD void item_dsm_table(F &f, size_t i, const apt *aff, pt *tbl) {
    char *base = reinterpret_cast<char *>(tbl + i * (size_t)DSM_TSTRIDE);
    apt *A = reinterpret_cast<apt *>(base);            // A[k - 1] = row k
    fe *U = reinterpret_cast<fe *>(base + DSM_U_OFF);  // U[k - 2] = u_k
    apt P = aff[i];
    apt p, q;  // P and kP at Z_k
    jac_dblu(f, q.x, q.y, p.x, p.y, P.x, P.y);
    A[1] = q;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int k = 2; k < DSM_TS; k++) {
        fe u;
        jac_zaddu(f, p.x, p.y, q.x, q.y, u);
        A[k] = q;
        U[k - 2] = u;
    }
    A[0] = p;
    fe r = U[DSM_TS - 3];
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int k = DSM_TS - 1; k >= 2; k--) {
        if (k < DSM_TS - 1) {
            fe uk = U[k - 2];
            f.mul(r, r, uk);
        }
        apt a = A[k - 1];
        fe rr;
        f.sqr(rr, r);
        f.mul(a.x, a.x, rr);
        f.mul(rr, rr, r);
        f.mul(a.y, a.y, rr);
        A[k - 1] = a;
    }
    fe zall;
    f.mul2(zall, P.y);
    f.mul(zall, zall, r);
    U[0] = zall;  // for the way back
}
template <class F>
S256_HD void item_dsm_ladder(F &f, size_t i, size_t n, const sc *u1s, const int8_t *dig1, const int8_t *dig2,
                             const uint8_t *sfl, pt *tbl, pt *res, const apt *comb) {
    char *base = reinterpret_cast<char *>(tbl + i * (size_t)DSM_TSTRIDE);
    const apt *A = reinterpret_cast<const apt *>(base);
    uint32_t fl = sfl[i];
    // the identity is the flag; the coordinates underneath are all zero, which every doubling maps to all zero (with
    // (0 : 1 : 0) they become small negative numbers, i.e. values next to 2^256, whose products take the folds' rare path)
    pt acc;
    acc.x = fe_zero();
    acc.y = fe_zero();
    acc.z = fe_zero();
    uint32_t inf = 1u;
    const fe beta = fe_beta();
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int s = DSM_ND - 1; s >= 0; s--) {
        // digits first: their loads and the table rows' trip from L2 overlap the doublings
        int da = dig1[(size_t)s * n + i];
        int db = dig2[(size_t)s * n + i];
#if defined(__CUDA_ARCH__) && !defined(S256_DSM_NO_PREFETCH)
        {
            int ma = da < 0 ? -da : da, mb = db < 0 ? -db : db;
            if (ma) asm volatile("prefetch.global.L1 [%0];" ::"l"(A + (ma - 1)));
            if (mb) asm volatile("prefetch.global.L1 [%0];" ::"l"(A + (mb - 1)));
        }
#endif
        if (s != DSM_ND - 1) {
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
            for (int k = 0; k < DSM_W; k++) jac_double(f, acc, acc);
        }
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int h = 0; h < 2; h++) {
            int d = h ? db : da;
            if (d != 0) {
                uint32_t neg = (uint32_t)(d < 0) ^ ((fl >> (1 + h)) & 1u);
                int mag = d < 0 ? -d : d;
                apt q;
                apt_fetch64(q, A + (mag - 1));
                if (h) f.mul(q.x, q.x, beta);
                if (neg) {
                    fe z = fe_zero();
                    f.sub(q.y, z, q.y);
                }
                jac_add_mixed_var(f, acc, inf, q.x, q.y);
            }
        }
    }
    if (!inf) {  // back from the isomorphic curve before the G half, whose rows are points of secp256k1 itself
        fe zall = reinterpret_cast<const fe *>(base + DSM_U_OFF)[0];
        f.mul(acc.z, acc.z, zall);
    }
    sc u1 = u1s[i];
    uint32_t carry = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int w = 0; w < COMB_NW; w++) {
        int32_t d = comb_digit(u1, w, carry);
        if (d != 0) {
            uint32_t mag = (uint32_t)(d < 0 ? -d : d);
            apt g = comb[(size_t)w * COMB_SZ + (mag - 1u)];
            if (d < 0) {
                fe z = fe_zero();
                f.sub(g.y, z, g.y);
            }
            jac_add_mixed_var(f, acc, inf, g.x, g.y);
        }
    }
    pt out;
    jac_to_projective(f, out, acc, inf);
    res[i] = out;
}
S256_HD void item_dsm(size_t i, size_t n, const apt *aff, const sc *u1s, const int8_t *dig1, const int8_t *dig2,
                      const uint8_t *sfl, pt *tbl, pt *res, const apt *comb) {
    fe_ops<DSM_VT> f;
    item_dsm_table(f, i, aff, tbl);
    item_dsm_ladder(f, i, n, u1s, dig1, dig2, sfl, tbl, res, comb);
}
#else
S256_HD void item_dsm(size_t i, size_t n, const apt *aff, const sc *u1s, const int8_t *dig1, const int8_t *dig2,
                      const uint8_t *sfl, pt *tbl, pt *res, const apt *comb) {
    pt *T = tbl + i * (size_t)DSM_TS;
    {
        apt P = aff[i];
        pt cur;
        pt_from_affine(cur, P);
        T[0] = cur;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int k = 2; k <= DSM_TS; k += 2) {
            pt h = T[k / 2 - 1];
            pt_double<DSM_VT>(cur, h);
            T[k - 1] = cur;
            if (k < DSM_TS) {
                pt_add_mixed<DSM_VT>(cur, cur, P.x, P.y);
                T[k] = cur;
            }
        }
    }
    uint32_t fl = sfl[i];
    pt acc;
    pt_set_identity(acc);
    const fe beta = fe_beta();
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int s = DSM_ND - 1; s >= 0; s--) {
        // digits first: their loads and the table rows' trip from L2 overlap the doublings
        int da = dig1[(size_t)s * n + i];
        int db = dig2[(size_t)s * n + i];
#if defined(__CUDA_ARCH__) && !defined(S256_DSM_NO_PREFETCH)
        {
            int ma = da < 0 ? -da : da, mb = db < 0 ? -db : db;
            if (ma) {
                const char *r = reinterpret_cast<const char *>(T + (ma - 1));
                asm volatile("prefetch.global.L1 [%0];" ::"l"(r));
                asm volatile("prefetch.global.L1 [%0];" ::"l"(r + 64));
            }
            if (mb) {
                const char *r = reinterpret_cast<const char *>(T + (mb - 1));
                asm volatile("prefetch.global.L1 [%0];" ::"l"(r));
                asm volatile("prefetch.global.L1 [%0];" ::"l"(r + 64));
            }
        }
#endif
        if (s != DSM_ND - 1) {
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
            for (int k = 0; k < DSM_W; k++) pt_double<DSM_VT>(acc, acc);
        }
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int h = 0; h < 2; h++) {
            int d = h ? db : da;
            if (d != 0) {
                uint32_t neg = (uint32_t)(d < 0) ^ ((fl >> (1 + h)) & 1u);
                int mag = d < 0 ? -d : d;
                pt q;
                pt_fetch64(q, T + (mag - 1));
                if (h) fe_ops<DSM_VT>::mul(q.x, q.x, beta);
                if (neg) {
                    fe z = fe_zero();
                    fe_ops<DSM_VT>::sub(q.y, z, q.y);
                }
                if (s == DSM_ND - 1 && h == 0)
                    acc = q;  // the accumulator is still the identity: the first addition is an assignment
                else
                    pt_add<DSM_VT>(acc, acc, q);
            }
        }
    }
    sc u1 = u1s[i];
    uint32_t carry = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int w = 0; w < COMB_NW; w++) {
        int32_t d = comb_digit(u1, w, carry);
        if (d != 0) {
            uint32_t mag = (uint32_t)(d < 0 ? -d : d);
            apt g = comb[(size_t)w * COMB_SZ + (mag - 1u)];
            if (d < 0) {
                fe z = fe_zero();
                fe_ops<DSM_VT>::sub(g.y, z, g.y);
            }
            pt_add_mixed<DSM_VT>(acc, acc, g.x, g.y);
        }
    }
    res[i] = acc;
}

#endif

// ---------------------------------------------------------------------------
// ECDSA finish (secec/ecdsa.go:450-467) without leaving projective space:
// x(R) mod n == r  <=>  X == r*Z  or  (r + n < p and X == (r + n)*Z).
// ---------------------------------------------------------------------------
S256_HD uint8_t item_ecdsa_finish(const pt &R, const uint8_t *sig64, uint32_t valid) {
    fe r, rn, t;
    fe_from_be32(r, sig64);
    uint32_t ok = valid & (1u - pt_is_identity(R));
    fe_mul(t, r, R.z);
    uint32_t m1 = fe_equal(t, R.x);
    // r + n as an integer; usable iff it does not wrap and is < p
    fe nn = fe_group_order();
    uint64_t acc = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        acc = (acc >> 32) + r.v[k] + nn.v[k];
        rn.v[k] = (uint32_t)acc;
    }
    uint32_t fits = (1u - (uint32_t)(acc >> 32)) & fe_limbs_are_canonical(rn);
    fe_mul(t, rn, R.z);
    uint32_t m2 = fits & fe_equal(t, R.x);
    return (uint8_t)(ok & (m1 | m2));
}

// ---------------------------------------------------------------------------
// projective -> affine for K results per thread with one shared Fermat chain
// (replaces the per-point inversion of point_projective.go:278-302), then the
// SEC 1 encodings of point_s11n.go:66-134.  Branch-free on the point value
// (identity handled by select), so the constant-time paths can use it.
// mode 0: 65-byte uncompressed + status; mode 1: 32-byte x + status (ECDH,
// secec/secec.go:53-56: identity is an error); mode 2: BIP-340 acceptance
// (schnorr.go:451-478): not identity, y even, x == sig[0:32].
// ---------------------------------------------------------------------------
// Row access for the conversion kernel.  On the device a point is fetched with six 128-bit loads
// (the rows are 96 bytes apart, 16-byte aligned) instead of 24 word loads.
S256_HD void pt_fetch(pt &r, const pt *p) {
#if defined(__CUDA_ARCH__)
    const uint4 *q = reinterpret_cast<const uint4 *>(p);
    uint4 a0 = q[0], a1 = q[1], a2 = q[2], a3 = q[3], a4 = q[4], a5 = q[5];
    r.x.v[0] = a0.x; r.x.v[1] = a0.y; r.x.v[2] = a0.z; r.x.v[3] = a0.w;
    r.x.v[4] = a1.x; r.x.v[5] = a1.y; r.x.v[6] = a1.z; r.x.v[7] = a1.w;
    r.y.v[0] = a2.x; r.y.v[1] = a2.y; r.y.v[2] = a2.z; r.y.v[3] = a2.w;
    r.y.v[4] = a3.x; r.y.v[5] = a3.y; r.y.v[6] = a3.z; r.y.v[7] = a3.w;
    r.z.v[0] = a4.x; r.z.v[1] = a4.y; r.z.v[2] = a4.z; r.z.v[3] = a4.w;
    r.z.v[4] = a5.x; r.z.v[5] = a5.y; r.z.v[6] = a5.z; r.z.v[7] = a5.w;
#else
    r = *p;
#endif
}
S256_HD void fe_fetch(fe &r, const fe *p) {
#if defined(__CUDA_ARCH__)
    const uint4 *q = reinterpret_cast<const uint4 *>(p);
    uint4 a0 = q[0], a1 = q[1];
    r.v[0] = a0.x; r.v[1] = a0.y; r.v[2] = a0.z; r.v[3] = a0.w;
    r.v[4] = a1.x; r.v[5] = a1.y; r.v[6] = a1.z; r.v[7] = a1.w;
#else
    r = *p;
#endif
}

// Batched projective -> affine + encode.  `stage` (device only, may be null): 2080 bytes of shared
// memory per warp.  The 65-byte rows of the 32 consecutive items a warp converts at a time form one
// contiguous, 16-byte aligned 2080-byte block; written row by row they are byte stores 65 bytes apart
// (every store instruction touches 32 sectors), so they are assembled in shared memory and leave as
// 130 coalesced 128-bit stores.
template <int K>
S256_HD void group_finish_affine(size_t t, size_t stride, size_t n, const pt *res, const uint8_t *in_status, int mode,
                                 uint8_t *out, uint8_t *status, const uint8_t *sig64, uint8_t *stage = nullptr) {
    fe pre[K];
    fe run = fe_one();
    const fe one = fe_one();
    for (int m = 0; m < K; m++) {
        size_t i = t + (size_t)m * stride;
        pre[m] = run;
        if (i < n) {
            fe z;
            fe_fetch(z, &res[i].z);
            fe_cmov(z, z, one, fe_is_zero(z));
            fe_mul(run, run, z);
        }
    }
    fe inv;
    fe_invert(inv, run);
#if defined(__CUDA_ARCH__)
    const unsigned lane = threadIdx.x & 31u;
    const bool full_warp = stage != nullptr && (t - lane) + 32 <= stride;  // every lane of the warp is alive
#endif
    for (int m = K - 1; m >= 0; m--) {
        size_t i = t + (size_t)m * stride;
        if (i >= n) continue;
        pt R;
        pt_fetch(R, &res[i]);
        uint32_t ident = fe_is_zero(R.z);
        fe z;
        fe_cmov(z, R.z, one, ident);
        fe zi, x, y;
        fe_mul(zi, inv, pre[m]);
        fe_mul(inv, inv, z);
        fe_mul(x, R.x, zi);
        fe_mul(y, R.y, zi);
        fe_normalize(x, x);
        fe_normalize(y, y);
        uint32_t in_ok = in_status ? (uint32_t)(in_status[i] != 0) : 1u;
        uint32_t keep = in_ok & (1u - ident);
        uint32_t km = 0u - keep;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            x.v[k] &= km;
            y.v[k] &= km;
        }
        uint8_t st = (uint8_t)(in_ok ? (ident ? ST_IDENTITY : ST_OK) : ST_INVALID);
        if (mode == 0) {
#if defined(__CUDA_ARCH__)
            const size_t i0 = i - lane;  // first item of this warp's block of rows
            if (full_warp && i0 + 32 <= n && (((size_t)(out + 65 * i0)) & 15u) == 0) {
                uint8_t *o = stage + 65 * lane;
                o[0] = (uint8_t)(keep ? 0x04 : 0x00);
                fe_to_be32(o + 1, x);
                fe_to_be32(o + 33, y);
                __syncwarp();
                const uint4 *src = reinterpret_cast<const uint4 *>(stage);
                uint4 *dst = reinterpret_cast<uint4 *>(out + 65 * i0);
                for (unsigned j = lane; j < 130; j += 32) dst[j] = src[j];
                __syncwarp();
                status[i] = st;
                continue;
            }
#endif
            uint8_t *o = out + 65 * i;
            o[0] = (uint8_t)(keep ? 0x04 : 0x00);
            fe_to_be32(o + 1, x);
            fe_to_be32(o + 33, y);
            status[i] = st;
        } else if (mode == 1) {
            fe_to_be32(out + 32 * i, x);
            status[i] = st;
        } else {
            fe r;
            fe_from_be32(r, sig64 + 64 * i);
            uint32_t same = 1;
#pragma unroll
            for (int k = 0; k < 8; k++) same &= (uint32_t)(r.v[k] == x.v[k]);
            status[i] = (uint8_t)(keep & same & (1u - (y.v[0] & 1u)));
        }
    }
}

// k_finish_affine body: fold the validity sources (decoded point, scalar
// parse) into cstat, convert, and for mode 3 (RecoverPublicKey) turn an
// identity result into an error (secec/secec.go:206-209).
template <int K>
S256_HD void group_finish(size_t t, size_t stride, size_t n, const pt *res, const uint8_t *pvalid, const uint8_t *sfl,
                          uint8_t *cstat, int mode, uint8_t *out, uint8_t *status, const uint8_t *sig64,
                          uint8_t *stage = nullptr) {
    for (int m = 0; m < K; m++) {
        size_t i = t + (size_t)m * stride;
        if (i < n) {
            uint32_t v = 1;
            if (pvalid) v &= (uint32_t)(pvalid[i] != 0);
            if (sfl) v &= (uint32_t)(sfl[i] & SFL_VALID);
            cstat[i] = (uint8_t)v;
        }
    }
    group_finish_affine<K>(t, stride, n, res, cstat, mode == 3 ? 0 : mode, out, status, sig64, stage);
    if (mode == 3) {
        for (int m = 0; m < K; m++) {
            size_t i = t + (size_t)m * stride;
            if (i < n && status[i] == ST_IDENTITY) status[i] = ST_INVALID;
        }
    }
}

// ---------------------------------------------------------------------------
// constant-time fixed-base multiplication (point_mul_table.go:168-194): no
// doublings, one mixed addition per WB-bit window.  The scalar is recoded
// branch-free into signed digits d_w in [-(2^(WB-1) - 1), 2^(WB-1)], every window
// reads all 2^(WB-1) table entries and keeps one by register select (the GPU
// counterpart of point_mul_table_amd64.s:81-130) -- the table is staged in shared memory and
// every lane reads the same address, so neither the address stream nor the
// bank pattern depends on the scalar -- the sign is applied by select, and
// digit 0 is resolved by select after a dummy add (point_mul_table.go:118-129).
// ---------------------------------------------------------------------------
template <int CT_WB = S256_CT_WB>
S256_HD void item_base_mult_ct(pt &acc, const sc &k, const apt *tab /* [NW][SZ] */) {
    constexpr int CT_NW = ct_cfg<CT_WB>::NW, CT_SZ = ct_cfg<CT_WB>::SZ;
    pt_set_identity(acc);
    uint32_t carry = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int w = 0; w < CT_NW; w++) {
        uint32_t v = ct_window_bits<CT_WB>(k, w) + carry;                       // 0 .. 2^WB
        carry = (v + (uint32_t)CT_SZ - 1u) >> CT_WB;                      // 1 iff v > 2^(WB-1)
        int32_t d = (int32_t)v - (int32_t)(carry << CT_WB);               // -(2^(WB-1) - 1) .. 2^(WB-1)
        uint32_t sign = (uint32_t)d >> 31;
        uint32_t mag = (uint32_t)((d ^ -(int32_t)sign) + (int32_t)sign);
        apt sel;
        sel.x = fe_zero();
        sel.y = fe_zero();
        const apt *row = tab + w * CT_SZ;
#if defined(__CUDA_ARCH__)
#pragma unroll 2
#endif
        for (uint32_t j = 1; j <= (uint32_t)CT_SZ; j++) {
            // a register select per word (SEL on the device: no branch, no address depends on mag)
            const bool hit = j == mag;
            apt e = row[j - 1];
#pragma unroll
            for (int q = 0; q < 8; q++) {
                sel.x.v[q] = hit ? e.x.v[q] : sel.x.v[q];
                sel.y.v[q] = hit ? e.y.v[q] : sel.y.v[q];
            }
        }
        // mag == 0 selected nothing: add a well-formed dummy (entry 1) and discard the sum
        uint32_t zero = (uint32_t)(mag == 0);
        apt e1 = row[0];
        fe_cmov(sel.x, sel.x, e1.x, zero);
        fe_cmov(sel.y, sel.y, e1.y, zero);
        fe_cneg(sel.y, sel.y, sign);
        pt sum;
        pt_add_mixed(sum, acc, sel.x, sel.y);
        pt_cmov(acc, sum, acc, zero);
    }
}

// The throughput kernels run the same multiplication with a JACOBIAN accumulator and the mixed Jacobian addition
// (jac.cuh) in its constant-time flavour: 8 M + 3 S = 719 MAC32 per window instead of 11 M = 805 for the complete mixed
// addition, fewer additions / subtractions, still no branch and no address that depends on the scalar
// (2^20 scalars: 6.55 -> 6.08 ms).  The formula is incomplete; here its exceptional cases CANNOT occur, and the only
// special value, the identity the accumulator starts as, is a flag resolved by select:
//   * Windows are taken in ascending order.  With B = 2^WB and digits |d_v| <= B/2, the accumulator before window w is
//     A = sum_{v<w} d_v B^v, |A| <= (B/2)(B^w - 1)/(B - 1) < 0.51 B^w, and the entry added is E = d_w B^w with
//     |E| >= B^w > |A| (a zero digit adds a dummy whose sum is discarded).  The formula fails iff A = +-E (mod n).
//   * Below the top window |A -+ E| < (B/2 + 0.51) B^w < 2^252 < n, and A -+ E != 0 as integers: not congruent.
//   * Top window (bits from 252 up): A + E = k, the scalar itself, reduced mod n by sc_from_be32: 0 <= k < n.
//     A + E = 0 (mod n) would need k = 0, i.e. no non-zero digit at all.  A - E = 2A - k lies in (-n - 2^252.02,
//     2^252.02); it is not 0 (|E| > |A|), and 2A - k = -n would need E = n + A to be a multiple of 2^252 with
//     -0.51 * 2^252 < A < 0: A = (2^256 - n) - m 2^252 has no such value (m = 0 gives A > 0, m = 1 gives A < -0.9 * 2^252).
//   * A = 0 (mod n) with |A| < n means A = 0, and then every lower digit is zero (the lowest non-zero digit d_v would
//     have to satisfy B | d_v): the flag "all digits so far were zero" is exactly "the accumulator is the identity".
// The lane-split small-batch kernels sum the windows in another order (partial sums per lane, folded by a tree) and
// keep the complete formulas, as do their folds; -DS256_BM_RCB restores them here as well.
#ifndef S256_BM_RCB
template <int CT_WB = S256_CT_WB>
S256_HD void item_base_mult_ct_jac(pt &out, const sc &k, const apt *tab) {
    constexpr int CT_NW = ct_cfg<CT_WB>::NW, CT_SZ = ct_cfg<CT_WB>::SZ;
    fe_ops<false> f;
    pt acc;
    acc.x = acc.y = acc.z = fe_zero();
    uint32_t inf = 1u, carry = 0;
    const fe one = fe_one();
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int w = 0; w < CT_NW; w++) {
        uint32_t v = ct_window_bits<CT_WB>(k, w) + carry;
        carry = (v + (uint32_t)CT_SZ - 1u) >> CT_WB;
        int32_t d = (int32_t)v - (int32_t)(carry << CT_WB);
        uint32_t sign = (uint32_t)d >> 31;
        uint32_t mag = (uint32_t)((d ^ -(int32_t)sign) + (int32_t)sign);
        apt sel;
        sel.x = fe_zero();
        sel.y = fe_zero();
        const apt *row = tab + w * CT_SZ;
#if defined(__CUDA_ARCH__)
#pragma unroll 2
#endif
        for (uint32_t j = 1; j <= (uint32_t)CT_SZ; j++) {
            const bool hit = j == mag;
            apt e = row[j - 1];
#pragma unroll
            for (int q = 0; q < 8; q++) {
                sel.x.v[q] = hit ? e.x.v[q] : sel.x.v[q];
                sel.y.v[q] = hit ? e.y.v[q] : sel.y.v[q];
            }
        }
        uint32_t zero = (uint32_t)(mag == 0);
        apt e1 = row[0];
        fe_cmov(sel.x, sel.x, e1.x, zero);
        fe_cmov(sel.y, sel.y, e1.y, zero);
        fe_cneg(sel.y, sel.y, sign);
        pt sum;
        jac_add_mixed_nocheck(f, sum, acc, sel.x, sel.y);
        // the accumulator is still the identity: the sum is the addend itself
        fe_cmov(sum.x, sum.x, sel.x, inf);
        fe_cmov(sum.y, sum.y, sel.y, inf);
        fe_cmov(sum.z, sum.z, one, inf);
        pt_cmov(acc, sum, acc, zero);
        inf &= zero;
    }
    pt hom, id;
    fe zz;
    fe_sqr(zz, acc.z);
    fe_mul(hom.x, acc.x, acc.z);
    hom.y = acc.y;
    fe_mul(hom.z, zz, acc.z);
    pt_set_identity(id);
    pt_cmov(out, hom, id, inf);
}
#endif

// Small batches: the windows of one scalar are dealt round-robin to T lanes (window j*T + part in
// iteration j, so the whole warp stays in lockstep); the caller folds the T partial points with
// complete additions.  Digits are recoded first (carry chain) into a local array that is then read
// at an index depending only on the lane number.  Same selects as above, over the 5-bit table.
// `row_bytes`: distance between the rows of two consecutive windows.  The lanes of a group read the SAME entry index of
// DIFFERENT windows at the same time; with the natural stride (16 entries x 64 B = 1024 B) all of them hit the same
// four banks -- an 8-way conflict on every shared load of the kernel (ncu: 12.8 M of 14.8 M wavefronts were conflicts,
// profiles/r02_ct_counters.txt).  The kernel stages the table with 16 bytes of padding per row, which spreads the
// eight lanes over the eight 16-byte bank groups.  (Public addressing either way: lane number and loop counters.)
template <int CT_WB = S256_CT_WB_SMALL>
S256_HD void item_base_mult_ct_part(pt &acc, const sc &k, const apt *tab, int part, int T,
                                    size_t row_bytes = (size_t)ct_cfg<CT_WB>::SZ * sizeof(apt)) {
    constexpr int CT_NW = ct_cfg<CT_WB>::NW, CT_SZ = ct_cfg<CT_WB>::SZ;
    int8_t dig[CT_NW];
    uint32_t carry = 0;
#pragma unroll 1
    for (int w = 0; w < CT_NW; w++) {
        uint32_t v = ct_window_bits<CT_WB>(k, w) + carry;
        carry = (v + (uint32_t)CT_SZ - 1u) >> CT_WB;
        dig[w] = (int8_t)((int32_t)v - (int32_t)(carry << CT_WB));
    }
    pt_set_identity(acc);
    const int iters = (CT_NW + T - 1) / T;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int j = 0; j < iters; j++) {
        int w = j * T + part;
        uint32_t inrange = (uint32_t)(w < CT_NW);
        int wc = inrange ? w : 0;
        int32_t d = inrange ? (int32_t)dig[wc] : 0;
        uint32_t sign = (uint32_t)d >> 31;
        uint32_t mag = (uint32_t)((d ^ -(int32_t)sign) + (int32_t)sign);
        apt sel;
        sel.x = fe_zero();
        sel.y = fe_zero();
        const apt *row = reinterpret_cast<const apt *>(reinterpret_cast<const char *>(tab) + (size_t)wc * row_bytes);
#if defined(__CUDA_ARCH__)
#pragma unroll 2
#endif
        for (uint32_t e = 1; e <= (uint32_t)CT_SZ; e++) {
            const bool hit = e == mag;
            apt t = row[e - 1];
#pragma unroll
            for (int q = 0; q < 8; q++) {
                sel.x.v[q] = hit ? t.x.v[q] : sel.x.v[q];
                sel.y.v[q] = hit ? t.y.v[q] : sel.y.v[q];
            }
        }
        uint32_t zero = (uint32_t)(mag == 0);
        apt e1 = row[0];
        fe_cmov(sel.x, sel.x, e1.x, zero);
        fe_cmov(sel.y, sel.y, e1.y, zero);
        fe_cneg(sel.y, sel.y, sign);
        pt sum;
        pt_add_mixed(sum, acc, sel.x, sel.y);
        pt_cmov(acc, sum, acc, zero);
    }
}

// Table storage policies for the ct ladder's affine table: per-item rows in global memory (host
// simulation, or when shared memory is not used) and per-thread columns in shared memory
// ([entry][limb group][thread], LDS.128 / STS.128 conflict-free).  Either way the address stream depends
// only on public values.
struct CtTableGlobal {
    pt *T;
    // affine entries live behind the projective scratch rows of the same per-item region
    S256_HD void store_affine(int j, const apt &a) const { reinterpret_cast<apt *>(T + CTM_TS)[j] = a; }
    S256_HD apt load_affine(int j) const { return reinterpret_cast<const apt *>(T + CTM_TS)[j]; }
};
#if defined(__CUDACC__)
// Entry 1 (the point itself) is not kept in shared memory: it is read back from the item's input row `p0` (a public
// address; 64 bytes that stay in L1), so that the columns of entries 2..TS take (TS - 1) x 64 x TPB bytes -- 56 KB for
// TS = 8, which lets FOUR 128-thread CTAs share an SM's 228 KB instead of three.
template <int TPB>
struct CtTableShared {
    uint32_t t;
    const apt *p0;
    // affine entries: 16 words = 4 x uint4 per entry, same conflict-free column layout
    __device__ __forceinline__ void store_affine(int j, const apt &a) const {
        extern __shared__ uint4 ct_smem[];
        if (j == 0) return;
        const uint32_t *w = a.x.v;  // x, y are contiguous
#pragma unroll
        for (int g = 0; g < 4; g++)
            ct_smem[(uint32_t)((j - 1) * 4 + g) * TPB + t] = make_uint4(w[4 * g], w[4 * g + 1], w[4 * g + 2], w[4 * g + 3]);
    }
    __device__ __forceinline__ apt load_affine(int j) const {
        extern __shared__ uint4 ct_smem[];
        apt a;
        uint32_t *w = a.x.v;
        if (j == 0) {
            const uint4 *q = reinterpret_cast<const uint4 *>(p0);
#pragma unroll
            for (int g = 0; g < 4; g++) {
                uint4 v = q[g];
                w[4 * g] = v.x; w[4 * g + 1] = v.y; w[4 * g + 2] = v.z; w[4 * g + 3] = v.w;
            }
            return a;
        }
#pragma unroll
        for (int g = 0; g < 4; g++) {
            uint4 q = ct_smem[(uint32_t)((j - 1) * 4 + g) * TPB + t];
            w[4 * g] = q.x; w[4 * g + 1] = q.y; w[4 * g + 2] = q.z; w[4 * g + 3] = q.w;
        }
        return a;
    }
};
#endif

// The constant-time GLV ladder over an AFFINE per-item table: [1..TS]P are built in projective form in the
// per-item global scratch `G`, brought to affine with ONE shared inversion (Montgomery's trick over
// their Z's; none is zero because P has prime order n and TS < n), and kept in the fast table `T`.
// Every window then costs a mixed addition (11 M) instead of a complete one (12 M) and the entries are
// a third smaller.  Digit 0 adds entry 1 and discards the sum (the mixed formula needs a finite addend),
// as the fixed-base ladder does.  No branch and no address depends on the scalar.
// The table holds multiples of the PUBLIC point: it is built with the variable-time field operations (fe_vt.cuh); the
// secret scalar first appears in the recoding below, and everything from there on is the constant-time flavour.
#ifndef S256_CTM_TAB_CT
constexpr bool CTM_TAB_VT = true;
#else
constexpr bool CTM_TAB_VT = false;
#endif
// Phase 1 (public data): [1..TS]P in projective form in the item's scratch G, the prefix products of Z_2..Z_TS behind
// them and the affine rows of CtTableGlobal, and their total, which the caller inverts -- alone (item_scalar_mult_ct_affine) or once
// for the whole CTA (api.cu k_scalar_mult_ct).
S256_HD void item_ctm_table(size_t i, const apt *aff, pt *G, fe &zprod) {
    const apt P = aff[i];
    pt cur;
    pt_from_affine(cur, P);
    G[0] = cur;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int k = 2; k <= CTM_TS; k += 2) {
        pt h = G[k / 2 - 1];
        pt_double<CTM_TAB_VT>(cur, h);
        G[k - 1] = cur;
        if (k < CTM_TS) {
            pt_add_mixed<CTM_TAB_VT>(cur, cur, P.x, P.y);
            G[k] = cur;
        }
    }
    // Z_1 = 1; the products Z_2 .. Z_j for the shared inversion
    fe *pre = reinterpret_cast<fe *>(reinterpret_cast<char *>(G) + CTM_TS * (96 + 64));
    fe run = fe_one();
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int j = 1; j < CTM_TS; j++) {
        pre[j] = run;
        fe z = G[j].z;
        fe_ops<CTM_TAB_VT>::mul(run, run, z);
    }
    zprod = run;
}
// Phase 2: inv = (Z_2 ... Z_TS)^-1; the affine table into T, then the constant-time ladder.
template <class TAB>
S256_HD void item_ctm_ladder(size_t i, const apt *aff, const uint8_t *k32, const TAB &T, pt *G, fe inv, pt *res) {
    {
        const fe *pre = reinterpret_cast<const fe *>(reinterpret_cast<const char *>(G) + CTM_TS * (96 + 64));
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int j = CTM_TS - 1; j >= 1; j--) {
            pt e = G[j];
            fe zi, pj = pre[j];
            apt a;
            fe_ops<CTM_TAB_VT>::mul(zi, inv, pj);
            fe_ops<CTM_TAB_VT>::mul(inv, inv, e.z);
            fe_ops<CTM_TAB_VT>::mul(a.x, e.x, zi);
            fe_ops<CTM_TAB_VT>::mul(a.y, e.y, zi);
            T.store_affine(j, a);
        }
        T.store_affine(0, aff[i]);
    }
    sc k;
    sc_from_be32(k, k32 + 32 * i);
    uint32_t m1[4], m2[4], neg1, neg2;
    sc_split_glv_abs(m1, neg1, m2, neg2, k);
    int8_t d1[CTM_ND], d2[CTM_ND];
    glv_recode<CTM_W>::run(d1, m1);
    glv_recode<CTM_W>::run(d2, m2);
    pt acc;
    pt_set_identity(acc);
    const fe beta = fe_beta();
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int s = CTM_ND - 1; s >= 0; s--) {
        if (s != CTM_ND - 1) {
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
            for (int q = 0; q < CTM_W; q++) pt_double(acc, acc);
        }
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int h = 0; h < 2; h++) {
            int32_t d = h ? (int32_t)d2[s] : (int32_t)d1[s];
            uint32_t sign = (uint32_t)d >> 31;                                // 1 iff d < 0
            uint32_t mag = (uint32_t)((d ^ -(int32_t)sign) + (int32_t)sign);  // |d|, branch-free
            uint32_t neg = sign ^ (h ? neg2 : neg1);
            uint32_t zero = (uint32_t)(mag == 0);
            apt q = T.load_affine(0);  // the dummy addend of digit 0, replaced below otherwise
#if defined(__CUDA_ARCH__)
#pragma unroll 2
#endif
            for (uint32_t j = 2; j <= (uint32_t)CTM_TS; j++) {
                const bool hit = j == mag;
                apt e = T.load_affine((int)j - 1);
#pragma unroll
                for (int w = 0; w < 8; w++) {
                    q.x.v[w] = hit ? e.x.v[w] : q.x.v[w];
                    q.y.v[w] = hit ? e.y.v[w] : q.y.v[w];
                }
            }
            if (h) fe_mul(q.x, q.x, beta);  // h is the (public) half index, not a secret
            fe_cneg(q.y, q.y, neg);
            pt sum;
            pt_add_mixed(sum, acc, q.x, q.y);
            pt_cmov(acc, sum, acc, zero);
        }
    }
    res[i] = acc;
}
template <class TAB>
S256_HD void item_scalar_mult_ct_affine(size_t i, const apt *aff, const uint8_t *k32, const TAB &T, pt *G, pt *res) {
    fe zprod, inv;
    item_ctm_table(i, aff, G, zprod);
    fe_invert(inv, zprod);
    item_ctm_ladder(i, aff, k32, T, G, inv, res);
}

// point_s11n.go:140-172 -- SetCompressedBytes: 02/03 || X
S256_HD uint8_t item_decode_compressed(apt &out, const uint8_t *b) {
    fe x;
    fe_from_be32(x, b + 1);
    uint32_t ok = (uint32_t)((b[0] == 0x02) | (b[0] == 0x03)) & fe_limbs_are_canonical(x);
    return item_decompress(out, x, ok, (uint32_t)(b[0] & 1u));
}

// ---------------------------------------------------------------------------
// Deterministic ECDSA signing: PrivateKey.Sign(RFC6979SHA256(), digest)
// (secec/ecdsa.go:284-390 with the DRBG of secec/ecdsa_k_rfc6979.go).  Everything
// here handles secrets: no branch or address depends on d or k, except the
// rejection of an out-of-range DRBG output (probability 2^-128, the reference
// short-circuits there too, ecdsa.go:537-540).
//   nonce kernel : d canonical & non-zero (NewPrivateKey, secec/secec.go:141-160),
//                  e = digest mod n, k = first DRBG output in [1, n)
//   R = k*G      : the constant-time fixed-base kernel + batched affine conversion
//   finish       : r = x(R) mod n, s = (r*d + e)/k with one shared k^-1 chain per group,
//                  low-s normalisation, recovery id = (didReduce << 1 | yOdd) ^ negated
// An item whose r or s comes out zero (the reference would draw another k; not reachable in
// practice) is reported as S256_ST_INVALID rather than retried.
// ---------------------------------------------------------------------------
S256_HD uint8_t item_rfc6979_nonce(uint8_t kout[32], const uint8_t *priv32, const uint8_t *digest32) {
    sc d, e;
    uint32_t d_ok = (1u - sc_from_be32(d, priv32)) & (1u - sc_is_zero(d));
    sc_from_be32(e, digest32);
    // K, V, int2octets(x) and bits2octets(h) as big-endian words (ecdsa_k_rfc6979.go:108-145)
    uint32_t K[8], V[8], xw[8], hw[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        V[i] = 0x01010101u;
        K[i] = 0;
        xw[i] = d.v[7 - i];
        hw[i] = e.v[7 - i];
    }
    // every HMAC under one key shares the key's two pad states; those of the initial all-zero K are constants
    uint32_t ist[8], ost[8];
    hmac_zero_key_states(ist, ost);
    for (uint32_t oct = 0; oct < 2; oct++) {
        hmac_st_m97(K, ist, ost, V, oct, xw, hw);
        hmac_pad_state(ist, K, 0x36363636u);
        hmac_pad_state(ost, K, 0x5c5c5c5cu);
        hmac_st_m32(V, ist, ost, V);
    }
    uint32_t ok = 0;
    sc k;
    for (int attempt = 0; attempt < 8 && !ok; attempt++) {
        if (attempt) {  // out-of-range candidate (probability 2^-128): K = HMAC(K, V || 00), byte-stream form
            uint8_t m[33], Kb[32], Vb[32];
            for (int i = 0; i < 8; i++)
                for (int b = 0; b < 4; b++) {
                    m[4 * i + b] = Vb[4 * i + b] = (uint8_t)(V[i] >> (24 - 8 * b));
                    Kb[4 * i + b] = (uint8_t)(K[i] >> (24 - 8 * b));
                }
            m[32] = 0x00;
            hmac_sha256_k32(Kb, Kb, m, 33);
            for (int i = 0; i < 8; i++)
                K[i] = ((uint32_t)Kb[4 * i] << 24) | ((uint32_t)Kb[4 * i + 1] << 16) | ((uint32_t)Kb[4 * i + 2] << 8) | Kb[4 * i + 3];
            hmac_pad_state(ist, K, 0x36363636u);
            hmac_pad_state(ost, K, 0x5c5c5c5cu);
            hmac_st_m32(V, ist, ost, V);
        }
        hmac_st_m32(V, ist, ost, V);
        uint32_t l[8];
#pragma unroll
        for (int i = 0; i < 8; i++) l[i] = V[7 - i];
        ok = (1u - sc_reduce_once(k, l, 0)) & (1u - sc_is_zero(k));
    }
    // an invalid key still runs the pipeline on a harmless nonce (k = 1)
    uint32_t good = ok & d_ok;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        uint32_t wv = good ? V[i] : (uint32_t)(i == 7);
        kout[4 * i] = (uint8_t)(wv >> 24);
        kout[4 * i + 1] = (uint8_t)(wv >> 16);
        kout[4 * i + 2] = (uint8_t)(wv >> 8);
        kout[4 * i + 3] = (uint8_t)wv;
    }
    return (uint8_t)good;
}

template <int K>
S256_HD void group_sign_finish(size_t t, size_t stride, size_t n, const uint8_t *priv32, const uint8_t *digest32,
                               const uint8_t *kbuf, const uint8_t *valid, const uint8_t *r65, uint8_t *sig64,
                               uint8_t *recid, uint8_t *status) {
    sc pre[K];
    sc run = sc_one();
    for (int m = 0; m < K; m++) {
        size_t i = t + (size_t)m * stride;
        pre[m] = run;
        if (i < n) {
            sc k;
            sc_from_be32(k, kbuf + 32 * i);  // in [1, n) by construction
            sc_mul(run, run, k);
        }
    }
    sc inv;
    sc_invert(inv, run);
    for (int m = K - 1; m >= 0; m--) {
        size_t i = t + (size_t)m * stride;
        if (i >= n) continue;
        sc k, kinv, d, e, r, s, ns;
        sc_from_be32(k, kbuf + 32 * i);
        sc_mul(kinv, inv, pre[m]);
        sc_mul(inv, inv, k);
        sc_from_be32(d, priv32 + 32 * i);
        sc_from_be32(e, digest32 + 32 * i);
        const uint8_t *R = r65 + 65 * i;
        uint32_t did_reduce = sc_from_be32(r, R + 1);
        uint32_t y_odd = R[64] & 1u;
        sc_mul(s, r, d);
        sc_add(s, s, e);
        sc_mul(s, s, kinv);
        uint32_t neg = sc_is_gt_half_n(s);
        sc_neg(ns, s);
        sc_cmov(s, s, ns, neg);
        uint32_t ok = (uint32_t)(valid[i] != 0) & (1u - sc_is_zero(r)) & (1u - sc_is_zero(s));
        uint32_t km = 0u - ok;
#pragma unroll
        for (int q = 0; q < 8; q++) {
            r.v[q] &= km;
            s.v[q] &= km;
        }
        sc_to_be32(sig64 + 64 * i, r);
        sc_to_be32(sig64 + 64 * i + 32, s);
        recid[i] = (uint8_t)((((did_reduce << 1) | y_odd) ^ neg) & km);
        status[i] = (uint8_t)(ok ? ST_OK : ST_INVALID);
    }
}

// ---------------------------------------------------------------------------
// BIP-340 signing: SchnorrPrivateKey.Sign (secec/bitcoin/schnorr.go:322-400), keys
// built like NewSchnorrPrivateKeyFromECDSA (:161-180).  Secrets throughout: branch-free.
//   P = d'*G (ct fixed-base kernel) -> nonce kernel: d = d' or n - d' (even y(P)),
//   t = d xor H_aux(aux), k' = H_nonce(t || Px || m) mod n  ->  R = k'*G  ->
//   finish: k = k' or n - k' (even y(R)), e = H_challenge(Rx || Px || m) mod n, sig = Rx || k + e*d.
// The reference's post-signing self-check (:393, :402-418) recomputes R from (s - d*e)*G; with
// deterministic arithmetic it cannot fail, and the parity tests verify every signature instead.
// ---------------------------------------------------------------------------
S256_HD uint8_t item_schnorr_nonce(uint8_t kout[32], const uint8_t *priv32, const uint8_t *p65, const uint8_t *msg,
                                   size_t msg_len, const uint8_t *aux32) {
    sc dp, d, nd;
    uint32_t ok = (1u - sc_from_be32(dp, priv32)) & (1u - sc_is_zero(dp));
    sc_neg(nd, dp);
    sc_cmov(d, dp, nd, (uint32_t)(p65[64] & 1u));
    uint8_t rnd[32];
    uint32_t tw[8], aw[8], pw[8], rw[8];
    be32_words(aw, aux32);
    bip340_tagged_32(tw, TAG_AUX, aw);
#pragma unroll
    for (int i = 0; i < 8; i++) tw[i] ^= d.v[7 - i];  // t = bytes(d) xor hash_aux(a)
    be32_words(pw, p65 + 1);
    if (msg_len == 32) {  // fixed layout: two compressions from the tag midstate
        uint32_t mw[8];
        be32_words(mw, msg);
        bip340_tagged_96(rw, TAG_NONCE, tw, pw, mw);
        words_be32(rnd, rw);
    } else {
        uint8_t t[32];
        words_be32(t, tw);
        sha_stream c;
        sha_init_tagged(c, TAG_NONCE);
        sha_update(c, t, 32);
        sha_update(c, p65 + 1, 32);
        sha_update(c, msg, msg_len);
        sha_final(c, rnd);
    }
    sc kp;
    sc_from_be32(kp, rnd);
    ok &= 1u - sc_is_zero(kp);  // errKPrimeIsZero
    sc one = sc_one();
    sc_cmov(kp, one, kp, ok);   // a harmless nonce keeps the pipeline well defined
    sc_to_be32(kout, kp);
    return (uint8_t)ok;
}
S256_HD void item_schnorr_sign_finish(uint8_t *sig64, uint8_t *status, const uint8_t *priv32, const uint8_t *p65,
                                      const uint8_t *r65, const uint8_t *kbuf, const uint8_t *msg, size_t msg_len,
                                      uint32_t valid) {
    sc dp, d, nd, kp, k, nk, e, sum;
    sc_from_be32(dp, priv32);
    sc_neg(nd, dp);
    sc_cmov(d, dp, nd, (uint32_t)(p65[64] & 1u));
    sc_from_be32(kp, kbuf);
    sc_neg(nk, kp);
    sc_cmov(k, kp, nk, (uint32_t)(r65[64] & 1u));
    uint8_t eb[32];
    if (msg_len == 32) {
        uint32_t rw[8], pw[8], mw[8], ew[8];
        be32_words(rw, r65 + 1);
        be32_words(pw, p65 + 1);
        be32_words(mw, msg);
        bip340_tagged_96(ew, TAG_CHALLENGE, rw, pw, mw);
        words_be32(eb, ew);
    } else {
        sha_stream c;
        sha_init_tagged(c, TAG_CHALLENGE);
        sha_update(c, r65 + 1, 32);
        sha_update(c, p65 + 1, 32);
        sha_update(c, msg, msg_len);
        sha_final(c, eb);
    }
    sc_from_be32(e, eb);
    sc_mul(sum, e, d);
    sc_add(sum, k, sum);
    uint8_t m = (uint8_t)(0u - (valid & 1u));
    uint8_t sb[32];
    sc_to_be32(sb, sum);
    for (int i = 0; i < 32; i++) {
        sig64[i] = r65[1 + i] & m;
        sig64[32 + i] = sb[i] & m;
    }
    *status = (uint8_t)(valid ? ST_OK : ST_INVALID);
}

}  // namespace s256
