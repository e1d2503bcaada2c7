// api_sign.cu -- deterministic ECDSA signing (RFC 6979 nonces) and BIP-340 signing: kernels and entry points.
#include "ctx.h"

// ---- deterministic signing (kernels.cuh) ----
__global__ void __launch_bounds__(S256_TPB) k_rfc6979_nonce(const uint8_t *priv32, const uint8_t *digest32, size_t n,
                                                            uint8_t *kbuf, uint8_t *valid) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    valid[i] = item_rfc6979_nonce(kbuf + 32 * i, priv32 + 32 * i, digest32 + 32 * i);
}
template <int K>
__global__ void __launch_bounds__(S256_TPB) k_sign_finish(size_t n, const uint8_t *priv32, const uint8_t *digest32,
                                                          const uint8_t *kbuf, const uint8_t *valid, const uint8_t *r65,
                                                          uint8_t *sig64, uint8_t *recid, uint8_t *status) {
    size_t stride = (n + K - 1) / K;
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= stride) return;
    group_sign_finish<K>(t, stride, n, priv32, digest32, kbuf, valid, r65, sig64, recid, status);
}

// M: msg_uniform or msg_offsets (kernels.cuh); a row that cannot be read signs nothing (status S256_ST_INVALID)
template <class M>
__global__ void __launch_bounds__(S256_TPB) k_schnorr_nonce(const uint8_t *priv32, const uint8_t *p65, M rows,
                                                            const uint8_t *aux32, size_t n, uint8_t *kbuf, uint8_t *valid) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t *m;
    size_t len;
    const uint32_t row_ok = rows.row(i, m, len);
    valid[i] = (uint8_t)(row_ok & item_schnorr_nonce(kbuf + 32 * i, priv32 + 32 * i, p65 + 65 * i, m, len, aux32 + 32 * i));
}
template <class M>
__global__ void __launch_bounds__(S256_TPB) k_schnorr_sign_finish(const uint8_t *priv32, const uint8_t *p65,
                                                                  const uint8_t *r65, const uint8_t *kbuf, M rows,
                                                                  const uint8_t *valid, size_t n, uint8_t *sig64,
                                                                  uint8_t *status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t *m;
    size_t len;
    rows.row(i, m, len);
    item_schnorr_sign_finish(sig64 + 64 * i, status + i, priv32 + 32 * i, p65 + 65 * i, r65 + 65 * i, kbuf + 32 * i, m, len,
                             valid[i]);
}


// PrivateKey.Sign(RFC6979SHA256(), digest): nonce -> k*G (ct) -> affine -> (r, s, v).  Scratch use: k in
// v.u1 (32 B/item), R in v.out (65 B/item), validity in v.pvalid; the nonce buffer is wiped afterwards.
static int chunk_sign(s256_ctx *ctx, const view &v, const uint8_t *priv32, const uint8_t *digest32, size_t n,
                      uint8_t *sig64, uint8_t *recid, uint8_t *status, cudaStream_t s) {
    uint8_t *kbuf = reinterpret_cast<uint8_t *>(v.u1);
    LAUNCH(ctx, k_rfc6979_nonce, grid_for(n), 0, s, priv32, digest32, n, kbuf, v.pvalid);
    s256_launch_base_mult_ct(kbuf, n, ctx->ct_tab, ctx->ct_tab_small, ctx->ct_tab_huge, v.res, s);
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
    s256_launch_finish_affine(ctx, n, v.res, nullptr, nullptr, v.cstat, 0, v.out, v.sfl, nullptr, s);
    DISPATCH_K(n, LAUNCH(ctx, k_sign_finish<KK>, grid_for_groups(n, KK), 0, s, n, priv32, digest32, kbuf, v.pvalid, v.out,
                         sig64, recid, status));
    CK(cudaMemsetAsync(kbuf, 0, 32 * n, s));
    CK(cudaMemsetAsync(v.res, 0, sizeof(pt) * n, s));
    return S256_SUCCESS;
}

// SchnorrPrivateKey.Sign: P = d'G -> nonce -> R = k'G -> finish.  Byte scratch: P in v.out, R and k' in the
// per-item table area (1536 B/item, unused by this path); both secret buffers are wiped afterwards.
template <class M>
static int chunk_schnorr_sign(s256_ctx *ctx, const view &v, const uint8_t *priv32, const M &rows, const uint8_t *aux32,
                              size_t n, uint8_t *sig64, uint8_t *status, cudaStream_t s) {
    uint8_t *arena = reinterpret_cast<uint8_t *>(v.tbl);
    uint8_t *r65 = arena, *kbuf = arena + 65 * n;
    s256_launch_base_mult_ct(priv32, n, ctx->ct_tab, ctx->ct_tab_small, ctx->ct_tab_huge, v.res, s);
    s256_launch_finish_affine(ctx, n, v.res, nullptr, nullptr, v.cstat, 0, v.out, v.sfl, nullptr, s);
    LAUNCH(ctx, k_schnorr_nonce<M>, grid_for(n), 0, s, priv32, v.out, rows, aux32, n, kbuf, v.pvalid);
    s256_launch_base_mult_ct(kbuf, n, ctx->ct_tab, ctx->ct_tab_small, ctx->ct_tab_huge, v.res, s);
    ctx->launches.fetch_add(2, std::memory_order_relaxed);
    s256_launch_finish_affine(ctx, n, v.res, nullptr, nullptr, v.cstat, 0, r65, v.sfl, nullptr, s);
    LAUNCH(ctx, k_schnorr_sign_finish<M>, grid_for(n), 0, s, priv32, v.out, r65, kbuf, rows, v.pvalid, n, sig64, status);
    CK(cudaMemsetAsync(kbuf, 0, 32 * n, s));
    CK(cudaMemsetAsync(v.res, 0, sizeof(pt) * n, s));
    return S256_SUCCESS;
}


extern "C" int s256_ecdsa_sign_rfc6979_dev(s256_ctx *ctx, const uint8_t *priv32, const uint8_t *digest32, size_t n,
                                           uint8_t *sig64, uint8_t *recid, uint8_t *status, void *stream) {
    ENTER(ctx);
    if (n && (!priv32 || !digest32 || !sig64 || !recid || !status)) return S256_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    int rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        return chunk_sign(ctx, view_at(ctx, 0), priv32 + 32 * off, digest32 + 32 * off, c, sig64 + 64 * off, recid + off,
                          status + off, s);
    });
    if (rc != S256_SUCCESS) wipe_secret_scratch(ctx);  // the chunk code returned before its own wipes
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}
extern "C" int s256_ecdsa_sign_rfc6979(s256_ctx *ctx, const uint8_t *priv32, const uint8_t *digest32, size_t n,
                                       uint8_t *sig64, uint8_t *recid, uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && (!priv32 || !digest32 || !sig64 || !recid || !status)) return S256_ERR_ARG;
    int rc = pipelined(ctx, n, [&](const view &v, size_t off, size_t c, cudaStream_t s) {
        CK(cudaMemcpyAsync(v.in_a, priv32 + 32 * off, 32 * c, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(v.in_b, digest32 + 32 * off, 32 * c, cudaMemcpyHostToDevice, s));
        // outputs staged in v.in_c (sig64), v.cstat is busy inside finish_affine -> recid in v.in_a + 32*cap? use tail of in_c
        uint8_t *d_sig = v.in_c, *d_rec = v.in_c + 64 * c, *d_st = v.st;
        int r = chunk_sign(ctx, v, v.in_a, v.in_b, c, d_sig, d_rec, d_st, s);
        if (r != S256_SUCCESS) return r;
        CK(cudaMemcpyAsync(sig64 + 64 * off, d_sig, 64 * c, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(recid + off, d_rec, c, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(status + off, d_st, c, cudaMemcpyDeviceToHost, s));
        CK(cudaMemsetAsync(v.in_a, 0, 32 * c, s));  // wipe the staged private keys
        return S256_SUCCESS;
    });
    if (rc != S256_SUCCESS) wipe_secret_scratch(ctx);  // the chunk code returned before its own wipes
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}

extern "C" int s256_schnorr_sign_dev(s256_ctx *ctx, const uint8_t *priv32, const uint8_t *msg, size_t msg_len,
                                     const uint8_t *aux32, size_t n, uint8_t *sig64, uint8_t *status, void *stream) {
    ENTER(ctx);
    if (n && (!priv32 || (!msg && msg_len) || !aux32 || !sig64 || !status)) return S256_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    int rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        return chunk_schnorr_sign(ctx, view_at(ctx, 0), priv32 + 32 * off, msg_uniform{msg + msg_len * off, msg_len},
                                  aux32 + 32 * off, c, sig64 + 64 * off, status + off, s);
    });
    if (rc != S256_SUCCESS) wipe_secret_scratch(ctx);  // the chunk code returned before its own wipes
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}
extern "C" int s256_schnorr_sign(s256_ctx *ctx, const uint8_t *priv32, const uint8_t *msg, size_t msg_len,
                                 const uint8_t *aux32, size_t n, uint8_t *sig64, uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && (!priv32 || (!msg && msg_len) || !aux32 || !sig64 || !status)) return S256_ERR_ARG;
    size_t need = (msg_len ? msg_len : 1) * (n < ctx->cap ? n : ctx->cap);
    if (int grc = grow_in_b(ctx, need)) return grc;
    int rc = pipelined(ctx, n, [&](const view &v, size_t off, size_t c, cudaStream_t ps) {
        uint8_t *dmsg = ctx->in_b + msg_len * (size_t)(v.st - ctx->st);  // messages are msg_len apart, not 32
        CK(cudaMemcpyAsync(v.in_a, priv32 + 32 * off, 32 * c, cudaMemcpyHostToDevice, ps));
        if (msg_len) CK(cudaMemcpyAsync(dmsg, msg + msg_len * off, msg_len * c, cudaMemcpyHostToDevice, ps));
        CK(cudaMemcpyAsync(v.in_c, aux32 + 32 * off, 32 * c, cudaMemcpyHostToDevice, ps));
        uint8_t *d_sig = reinterpret_cast<uint8_t *>(v.aff);  // 64 B per item, unused by this path
        int r = chunk_schnorr_sign(ctx, v, v.in_a, msg_uniform{dmsg, msg_len}, v.in_c, c, d_sig, v.st, ps);
        if (r != S256_SUCCESS) return r;
        CK(cudaMemcpyAsync(sig64 + 64 * off, d_sig, 64 * c, cudaMemcpyDeviceToHost, ps));
        CK(cudaMemcpyAsync(status + off, v.st, c, cudaMemcpyDeviceToHost, ps));
        CK(cudaMemsetAsync(v.in_a, 0, 32 * c, ps));  // wipe the staged private keys
        return S256_SUCCESS;
    });
    if (rc != S256_SUCCESS) wipe_secret_scratch(ctx);  // the chunk code returned before its own wipes
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}

extern "C" int s256_schnorr_sign_varlen_dev(s256_ctx *ctx, const uint8_t *priv32, const uint8_t *msg, const size_t *offsets,
                                            const uint8_t *aux32, size_t n, uint8_t *sig64, uint8_t *status, void *stream) {
    ENTER(ctx);
    if (n && (!priv32 || !msg || !offsets || !aux32 || !sig64 || !status)) return S256_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    int rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        return chunk_schnorr_sign(ctx, view_at(ctx, 0), priv32 + 32 * off, msg_offsets{msg, offsets + off, 0}, aux32 + 32 * off,
                                  c, sig64 + 64 * off, status + off, s);
    });
    if (rc != S256_SUCCESS) wipe_secret_scratch(ctx);  // the chunk code returned before its own wipes
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}
extern "C" int s256_schnorr_sign_varlen(s256_ctx *ctx, const uint8_t *priv32, const uint8_t *msg, const size_t *offsets,
                                        const uint8_t *aux32, size_t n, uint8_t *sig64, uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && (!priv32 || !offsets || !aux32 || !sig64 || !status)) return S256_ERR_ARG;
    if (int grc = n ? varlen_staging(ctx, msg, offsets, n, ctx->cap) : S256_SUCCESS) return grc;
    int rc = pipelined(ctx, n, [&](const view &v, size_t off, size_t c, cudaStream_t ps) {
        msg_offsets rows;
        CK(cudaMemcpyAsync(v.in_a, priv32 + 32 * off, 32 * c, cudaMemcpyHostToDevice, ps));
        if (int r = varlen_stage_part(ctx, msg, offsets, off, (size_t)(v.st - ctx->st), c, ps, rows)) return r;
        CK(cudaMemcpyAsync(v.in_c, aux32 + 32 * off, 32 * c, cudaMemcpyHostToDevice, ps));
        uint8_t *d_sig = reinterpret_cast<uint8_t *>(v.aff);  // 64 B per item, unused by this path
        int r = chunk_schnorr_sign(ctx, v, v.in_a, rows, v.in_c, c, d_sig, v.st, ps);
        if (r != S256_SUCCESS) return r;
        CK(cudaMemcpyAsync(sig64 + 64 * off, d_sig, 64 * c, cudaMemcpyDeviceToHost, ps));
        CK(cudaMemcpyAsync(status + off, v.st, c, cudaMemcpyDeviceToHost, ps));
        CK(cudaMemsetAsync(v.in_a, 0, 32 * c, ps));  // wipe the staged private keys
        return S256_SUCCESS;
    });
    if (rc != S256_SUCCESS) wipe_secret_scratch(ctx);  // the chunk code returned before its own wipes
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}
