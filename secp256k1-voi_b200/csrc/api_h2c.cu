// api_h2c.cu -- hash to curve (RFC 9380): kernels (h2c.cuh) and entry points.
#include <type_traits>

#include "ctx.h"
#include "h2c.cuh"

// M: msg_uniform or msg_offsets (kernels.cuh).  The msg_offsets instantiation also writes each row's validity byte to
// `valid`; a row that cannot be read hashes nothing of it, and k_finish_affine turns it into S256_ST_INVALID.
template <class M>
__global__ void __launch_bounds__(S256_TPB) k_hash_to_curve(const uint8_t *dst, int dst_len, M rows, size_t n, int ro,
                                                            pt *res, uint8_t *valid) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t *m;
    size_t len;
    const uint32_t ok = rows.row(i, m, len);
    pt r;
    item_hash_to_curve(r, dst, dst_len, m, len, ro);
    res[i] = r;
    if constexpr (std::is_same<M, msg_offsets>::value) valid[i] = (uint8_t)ok;
}
__global__ void __launch_bounds__(S256_TPB) k_expand_xmd(const uint8_t *dst, int dst_len, const uint8_t *msg,
                                                         size_t msg_len, size_t n, int len, uint8_t *out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    h2c_expand_xmd(out + (size_t)len * i, len, dst, dst_len, msg + msg_len * i, msg_len);
}

// RFC 9380 section 5.3.3 / h2c_expand_message.go:52-62: an oversize DST is replaced by its hash (host side:
// public bytes, one hash per call)
static int prepare_dst(const uint8_t *dst, size_t dst_len, uint8_t buf[H2C_MAX_DST], int *out_len) {
    if (!dst || dst_len == 0) return S256_ERR_ARG;  // errInvalidDomainSep
    if (dst_len > (size_t)H2C_MAX_DST) {
        sha_stream c;
        sha_init(c);
        sha_update(c, (const uint8_t *)"H2C-OVERSIZE-DST-", 17);
        sha_update(c, dst, dst_len);
        sha_final(c, buf);
        *out_len = 32;
    } else {
        memcpy(buf, dst, dst_len);
        *out_len = (int)dst_len;
    }
    return S256_SUCCESS;
}
// grows the message staging buffer (ctx->in_b) like the Schnorr entry points do
static int ensure_msg_staging(s256_ctx *ctx, size_t msg_len, size_t n) {
    size_t need = (msg_len ? msg_len : 1) * (n < ctx->cap ? n : ctx->cap);
    if (int grc = grow_in_b(ctx, need)) return grc;
    return S256_SUCCESS;
}

// One chunk: hash n rows to projective points in v.res, then the shared batched conversion into out (65 bytes per
// row) and status.  Rows of msg_offsets carry their validity in v.pvalid.
template <class M>
static void chunk_hash_to_curve(s256_ctx *ctx, const view &v, const uint8_t *dst, int dst_len, const M &rows, size_t n, int ro,
                                uint8_t *out, uint8_t *status, cudaStream_t s) {
    const bool ragged = std::is_same<M, msg_offsets>::value;
    LAUNCH(ctx, k_hash_to_curve<M>, grid_for(n), 0, s, dst, dst_len, rows, n, ro, v.res, ragged ? v.pvalid : nullptr);
    s256_launch_finish_affine(ctx, n, v.res, ragged ? v.pvalid : nullptr, nullptr, v.cstat, 0, out, status, nullptr, s);
}

extern "C" int s256_hash_to_curve(s256_ctx *ctx, const uint8_t *dst, size_t dst_len, const uint8_t *msg, size_t msg_len,
                                  size_t n, int random_oracle, uint8_t *out65, uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && ((!msg && msg_len) || !out65 || !status)) return S256_ERR_ARG;
    uint8_t dbuf[H2C_MAX_DST];
    int dl = 0;
    int rc = prepare_dst(dst, dst_len, dbuf, &dl);
    if (rc != S256_SUCCESS) return rc;
    rc = ensure_msg_staging(ctx, msg_len, n);
    if (rc != S256_SUCCESS) return rc;
    cudaStream_t s = ctx->stream;
    CK(cudaMemcpyAsync(ctx->in_c, dbuf, (size_t)dl, cudaMemcpyHostToDevice, s));
    rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        view v = view_at(ctx, 0);
        if (msg_len) CK(cudaMemcpyAsync(ctx->in_b, msg + msg_len * off, msg_len * c, cudaMemcpyHostToDevice, s));
        chunk_hash_to_curve(ctx, v, ctx->in_c, dl, msg_uniform{ctx->in_b, msg_len}, c, random_oracle ? 1 : 0, v.out, v.st, s);
        CK(cudaMemcpyAsync(out65 + 65 * off, v.out, 65 * c, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(status + off, v.st, c, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        return S256_SUCCESS;
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}

// The DST of a call travels as a kernel parameter to ctx->h2c_dst: it is on the device as soon as the launch is
// enqueued, so the forms below neither synchronise for it nor read the caller's host memory after they return.
struct h2c_dst_words {
    uint32_t w[64];
};
__global__ void k_put_dst(h2c_dst_words d, uint32_t *out) {
#pragma unroll
    for (int k = 0; k < 64; k++) out[k] = d.w[k];
}
static void put_dst(s256_ctx *ctx, const h2c_dst_words &d, cudaStream_t s) {
    k_put_dst<<<1, 1, 0, s>>>(d, reinterpret_cast<uint32_t *>(ctx->h2c_dst));
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
}

extern "C" int s256_hash_to_curve_dev(s256_ctx *ctx, const uint8_t *dst, size_t dst_len, const uint8_t *msg, size_t msg_len,
                                      size_t n, int random_oracle, uint8_t *out65, uint8_t *status, void *stream) {
    ENTER(ctx);
    if (n && ((!msg && msg_len) || !out65 || !status)) return S256_ERR_ARG;
    h2c_dst_words d{};
    int dl = 0;
    if (int rc = prepare_dst(dst, dst_len, reinterpret_cast<uint8_t *>(d.w), &dl)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    put_dst(ctx, d, s);
    int rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        chunk_hash_to_curve(ctx, view_at(ctx, 0), ctx->h2c_dst, dl, msg_uniform{msg + msg_len * off, msg_len}, c,
                            random_oracle ? 1 : 0, out65 + 65 * off, status + off, s);
        return S256_SUCCESS;
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}

extern "C" int s256_hash_to_curve_varlen_dev(s256_ctx *ctx, const uint8_t *dst, size_t dst_len, const uint8_t *msg,
                                             const size_t *offsets, size_t n, int random_oracle, uint8_t *out65,
                                             uint8_t *status, void *stream) {
    ENTER(ctx);
    if (n && (!msg || !offsets || !out65 || !status)) return S256_ERR_ARG;
    h2c_dst_words d{};
    int dl = 0;
    if (int rc = prepare_dst(dst, dst_len, reinterpret_cast<uint8_t *>(d.w), &dl)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    put_dst(ctx, d, s);
    int rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        chunk_hash_to_curve(ctx, view_at(ctx, 0), ctx->h2c_dst, dl, msg_offsets{msg, offsets + off, 0}, c, random_oracle ? 1 : 0,
                            out65 + 65 * off, status + off, s);
        return S256_SUCCESS;
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}

// The host form stages rows as the *_varlen host forms of api.cu do.  The DST goes to ctx->h2c_dst on ctx->stream,
// and stream2, which runs every other pipeline part, waits for it.
extern "C" int s256_hash_to_curve_varlen(s256_ctx *ctx, const uint8_t *dst, size_t dst_len, const uint8_t *msg,
                                         const size_t *offsets, size_t n, int random_oracle, uint8_t *out65, uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && (!offsets || !out65 || !status)) return S256_ERR_ARG;
    h2c_dst_words d{};
    int dl = 0;
    if (int rc = prepare_dst(dst, dst_len, reinterpret_cast<uint8_t *>(d.w), &dl)) return rc;
    if (int grc = n ? varlen_staging(ctx, msg, offsets, n, ctx->cap) : S256_SUCCESS) return grc;
    put_dst(ctx, d, ctx->stream);
    CK(cudaEventRecord(ctx->ev_decode, ctx->stream));
    CK(cudaStreamWaitEvent(ctx->stream2, ctx->ev_decode, 0));
    int rc = pipelined(ctx, n, [&](const view &v, size_t off, size_t c, cudaStream_t ps) {
        msg_offsets rows;
        if (int r = varlen_stage_part(ctx, msg, offsets, off, (size_t)(v.st - ctx->st), c, ps, rows)) return r;
        chunk_hash_to_curve(ctx, v, ctx->h2c_dst, dl, rows, c, random_oracle ? 1 : 0, v.out, v.st, ps);
        CK(cudaMemcpyAsync(out65 + 65 * off, v.out, 65 * c, cudaMemcpyDeviceToHost, ps));
        CK(cudaMemcpyAsync(status + off, v.st, c, cudaMemcpyDeviceToHost, ps));
        return S256_SUCCESS;
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}

extern "C" int s256_expand_message_xmd(s256_ctx *ctx, const uint8_t *dst, size_t dst_len, const uint8_t *msg,
                                       size_t msg_len, size_t n, size_t len_in_bytes, uint8_t *out) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && ((!msg && msg_len) || !out)) return S256_ERR_ARG;
    if (len_in_bytes == 0 || len_in_bytes > 96) return S256_ERR_ARG;  // the suites here need 48 or 96
    uint8_t dbuf[H2C_MAX_DST];
    int dl = 0;
    int rc = prepare_dst(dst, dst_len, dbuf, &dl);
    if (rc != S256_SUCCESS) return rc;
    rc = ensure_msg_staging(ctx, msg_len, n);
    if (rc != S256_SUCCESS) return rc;
    cudaStream_t s = ctx->stream;
    CK(cudaMemcpyAsync(ctx->in_c, dbuf, (size_t)dl, cudaMemcpyHostToDevice, s));
    uint8_t *d_out = reinterpret_cast<uint8_t *>(ctx->res);  // 96 B per item
    rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        if (msg_len) CK(cudaMemcpyAsync(ctx->in_b, msg + msg_len * off, msg_len * c, cudaMemcpyHostToDevice, s));
        LAUNCH(ctx, k_expand_xmd, grid_for(c), 0, s, ctx->in_c, dl, ctx->in_b, msg_len, c, (int)len_in_bytes, d_out);
        CK(cudaMemcpyAsync(out + len_in_bytes * off, d_out, len_in_bytes * c, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        return S256_SUCCESS;
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}
