// group_sim.cpp -- TEST INFRASTRUCTURE ONLY: the entry points whose kernels share one inversion between K rows
// (k_finish_affine<K>, k_ecdsa_scalars<K, RECOVER>, k_sign_finish<K>), on the CPU, with K chosen per call.
//
// The device picks K by chunk size (ctx.h inv_k_for: 1 below 2^16 rows, 4 below 2^19, 32 above); hostsim.cpp always
// runs K = 32.  This file builds on hostsim.cpp (included whole, like batch_sim.cpp) and runs the same item and group
// functions in the order api.cu / api_sign.cu launch them, with the device's strides:
//   k_ecdsa_scalars, k_sign_finish: thread t owns rows t + m * stride, stride = ceil(n / K);
//   k_finish_affine:                the same stride rounded up to a multiple of 32.
#include "hostsim.cpp"

static size_t group_stride(size_t n, int k) { return (n + k - 1) / k; }
static size_t finish_stride(size_t n, int k) { return (group_stride(n, k) + 31) & ~(size_t)31; }

// DISPATCH_K of ctx.h with a run-time K; any other value is refused
#define GSIM_DISPATCH(k, CALL)                              \
    switch (k) {                                            \
        case 1: { constexpr int KK = 1; CALL; } return 0;   \
        case 4: { constexpr int KK = 4; CALL; } return 0;   \
        case 32: { constexpr int KK = 32; CALL; } return 0; \
        default: return -1;                                 \
    }

template <int KK>
static void finish_k(scratch &s, size_t n, bool use_pvalid, bool use_sfl, int mode, uint8_t *out, uint8_t *status) {
    size_t stride = finish_stride(n, KK);
    for (size_t t = 0; t < stride; t++)
        group_finish<KK>(t, stride, n, s.res.data(), use_pvalid ? s.pvalid.data() : nullptr,
                         use_sfl ? s.sfl.data() : nullptr, s.cstat.data(), mode, out, status, nullptr);
}

template <int KK>
static void ecdsa_verify_k(const uint8_t *pk, const uint8_t *dg, const uint8_t *sig, uint32_t flags, size_t n, uint8_t *ok) {
    scratch s(n);
    for (size_t i = 0; i < n; i++) s.pvalid[i] = item_decode_uncompressed(s.aff[i], pk + 65 * i);
    size_t stride = group_stride(n, KK);
    for (size_t t = 0; t < stride; t++)
        group_ecdsa_scalars<KK>(t, stride, n, dg, sig, flags, s.u1.data(), s.dig1.data(), s.dig2.data(), s.sfl.data());
    run_dsm(s, n);
    for (size_t i = 0; i < n; i++) {
        uint32_t valid = (uint32_t)(s.pvalid[i] != 0) & (uint32_t)(s.sfl[i] & SFL_VALID);
        ok[i] = item_ecdsa_finish(s.res[i], sig + 64 * i, valid);
    }
}
template <int KK>
static void ecdsa_recover_k(const uint8_t *dg, const uint8_t *sig65, size_t n, uint8_t *pk65, uint8_t *status) {
    scratch s(n);
    for (size_t i = 0; i < n; i++) s.pvalid[i] = item_decode_recover(s.aff[i], sig65 + 65 * i);
    size_t stride = group_stride(n, KK);
    for (size_t t = 0; t < stride; t++)
        group_recover_scalars<KK>(t, stride, n, dg, sig65, s.u1.data(), s.dig1.data(), s.dig2.data(), s.sfl.data());
    run_dsm(s, n);
    finish_k<KK>(s, n, true, true, 3, pk65, status);
}
template <int KK>
static void double_scalar_mult_k(const uint8_t *u1, const uint8_t *u2, const uint8_t *pt65, size_t n, uint8_t *out65,
                                 uint8_t *status) {
    scratch s(n);
    for (size_t i = 0; i < n; i++) s.pvalid[i] = item_decode_uncompressed(s.aff[i], pt65 + 65 * i);
    for (size_t i = 0; i < n; i++) item_plain_scalars(i, n, u1, u2, s.u1.data(), s.dig1.data(), s.dig2.data(), s.sfl.data());
    run_dsm(s, n);
    finish_k<KK>(s, n, true, false, 0, out65, status);
}
// k G for every row, alternating the complete and the Jacobian-accumulator forms by index as sim_scalar_base_mult does
static void base_mult_rows(scratch &s, const uint8_t *k32, size_t n) {
    ensure_tables();
    for (size_t i = 0; i < n; i++) {
        sc k;
        sc_from_be32(k, k32 + 32 * i);
        if (i & 1)
            item_base_mult_ct(s.res[i], k, g_ct.data());
        else
            item_base_mult_ct_jac(s.res[i], k, g_ct.data());
    }
}
template <int KK>
static void scalar_base_mult_k(const uint8_t *k32, size_t n, uint8_t *out65, uint8_t *status) {
    scratch s(n);
    base_mult_rows(s, k32, n);
    finish_k<KK>(s, n, false, false, 0, out65, status);
}
template <int KK>
static void scalar_mult_k(const uint8_t *k32, const uint8_t *pt65, size_t n, int mode, uint8_t *out, uint8_t *status) {
    scratch s(n);
    for (size_t i = 0; i < n; i++) s.pvalid[i] = item_decode_uncompressed(s.aff[i], pt65 + 65 * i);
    for (size_t i = 0; i < n; i++) {
        CtTableGlobal T{s.tbl.data() + i * (size_t)DSM_TSTRIDE};
        item_scalar_mult_ct_affine(i, s.aff.data(), k32, T, s.tbl.data() + i * (size_t)DSM_TSTRIDE, s.res.data());
    }
    finish_k<KK>(s, n, true, false, mode, out, status);
}
// api_sign.cu chunk_sign: nonce -> R = k G -> finish (mode 0) -> k_sign_finish
template <int KK>
static void ecdsa_sign_k(const uint8_t *priv32, const uint8_t *digest32, size_t n, uint8_t *sig64, uint8_t *recid,
                         uint8_t *status) {
    scratch s(n);
    std::vector<uint8_t> kbuf(32 * n), valid(n), r65(65 * n), rst(n);
    for (size_t i = 0; i < n; i++) valid[i] = item_rfc6979_nonce(kbuf.data() + 32 * i, priv32 + 32 * i, digest32 + 32 * i);
    base_mult_rows(s, kbuf.data(), n);
    finish_k<KK>(s, n, false, false, 0, r65.data(), rst.data());
    size_t stride = group_stride(n, KK);
    for (size_t t = 0; t < stride; t++)
        group_sign_finish<KK>(t, stride, n, priv32, digest32, kbuf.data(), valid.data(), r65.data(), sig64, recid, status);
}
// api_sign.cu chunk_schnorr_sign: P = d'G -> finish -> nonce -> R = k'G -> finish -> per-row signature
template <int KK>
static void schnorr_sign_k(const uint8_t *priv32, const uint8_t *msg, size_t msg_len, const uint8_t *aux32, size_t n,
                           uint8_t *sig64, uint8_t *status) {
    scratch s(n);
    std::vector<uint8_t> p65(65 * n), r65(65 * n), kbuf(32 * n), valid(n), st(n);
    base_mult_rows(s, priv32, n);
    finish_k<KK>(s, n, false, false, 0, p65.data(), st.data());
    for (size_t i = 0; i < n; i++)
        valid[i] = item_schnorr_nonce(kbuf.data() + 32 * i, priv32 + 32 * i, p65.data() + 65 * i, msg + msg_len * i, msg_len,
                                      aux32 + 32 * i);
    base_mult_rows(s, kbuf.data(), n);
    finish_k<KK>(s, n, false, false, 0, r65.data(), st.data());
    for (size_t i = 0; i < n; i++)
        item_schnorr_sign_finish(sig64 + 64 * i, status + i, priv32 + 32 * i, p65.data() + 65 * i, r65.data() + 65 * i,
                                 kbuf.data() + 32 * i, msg + msg_len * i, msg_len, valid[i]);
}

// Exported forms: the first argument is K (1, 4 or 32); the return value is 0, or -1 for any other K.
EXPORT int gsim_ecdsa_verify(int k, const uint8_t *pk, const uint8_t *dg, const uint8_t *sig, uint32_t flags, size_t n,
                             uint8_t *ok) {
    GSIM_DISPATCH(k, ecdsa_verify_k<KK>(pk, dg, sig, flags, n, ok));
}
EXPORT int gsim_ecdsa_recover(int k, const uint8_t *dg, const uint8_t *sig65, size_t n, uint8_t *pk65, uint8_t *status) {
    GSIM_DISPATCH(k, ecdsa_recover_k<KK>(dg, sig65, n, pk65, status));
}
EXPORT int gsim_double_scalar_mult(int k, const uint8_t *u1, const uint8_t *u2, const uint8_t *pt65, size_t n, uint8_t *out65,
                                   uint8_t *status) {
    GSIM_DISPATCH(k, double_scalar_mult_k<KK>(u1, u2, pt65, n, out65, status));
}
EXPORT int gsim_scalar_base_mult(int k, const uint8_t *k32, size_t n, uint8_t *out65, uint8_t *status) {
    GSIM_DISPATCH(k, scalar_base_mult_k<KK>(k32, n, out65, status));
}
EXPORT int gsim_scalar_mult(int k, const uint8_t *k32, const uint8_t *pt65, size_t n, int mode, uint8_t *out, uint8_t *status) {
    GSIM_DISPATCH(k, scalar_mult_k<KK>(k32, pt65, n, mode, out, status));
}
EXPORT int gsim_ecdsa_sign_rfc6979(int k, const uint8_t *priv32, const uint8_t *digest32, size_t n, uint8_t *sig64,
                                   uint8_t *recid, uint8_t *status) {
    GSIM_DISPATCH(k, ecdsa_sign_k<KK>(priv32, digest32, n, sig64, recid, status));
}
EXPORT int gsim_schnorr_sign(int k, const uint8_t *priv32, const uint8_t *msg, size_t msg_len, const uint8_t *aux32, size_t n,
                             uint8_t *sig64, uint8_t *status) {
    GSIM_DISPATCH(k, schnorr_sign_k<KK>(priv32, msg, msg_len, aux32, n, sig64, status));
}
