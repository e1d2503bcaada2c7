// ctx.h -- private to csrc/: the context object, launch / error macros and the chunking helpers
// shared by the translation units of the library (api.cu, api_msm.cu, api_sign.cu).  The split exists
// for build time only (each unit is compiled in parallel).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "../../include/secp256k1_b200.h"
#include "kernels.cuh"
#include "launchers.h"

using namespace s256;

#define S256_TPB 128

struct s256_ctx {
    int device = -1;
    size_t cap = 0;
    std::mutex mu;
    cudaStream_t stream = nullptr, stream2 = nullptr, stream3 = nullptr;
    std::string last_err;
    std::atomic<uint64_t> launches{0};
    // constant tables
    apt *comb = nullptr;    // [COMB_NW][COMB_SZ]
    apt *ct_tab = nullptr, *ct_tab_small = nullptr, *ct_tab_huge = nullptr;  // signed-window tables of G: 6-, 5- and 7-bit (kernels.cuh)
    // per-chunk scratch
    apt *aff = nullptr;
    sc *u1 = nullptr;
    int8_t *dig1 = nullptr, *dig2 = nullptr;
    uint8_t *sfl = nullptr, *pvalid = nullptr, *cstat = nullptr;
    pt *tbl = nullptr, *res = nullptr;
    // staging for the host-pointer entry points
    uint8_t *in_a = nullptr, *in_b = nullptr, *in_c = nullptr, *out = nullptr, *st = nullptr;
    size_t in_b_bytes = 0;
    size_t *in_off = nullptr;  // the message offsets of the *_varlen host forms (allocated on first use)
    size_t in_off_count = 0;
    uint8_t *h2c_dst = nullptr;  // the hash-to-curve DST of the current call (256 bytes, api_h2c.cu)
    unsigned long long *sink = nullptr;
    // MSM scratch (allocated on first use)
    size_t msm_cap = 0;
    uint32_t *msm_counts = nullptr, *msm_offsets = nullptr, *msm_cursor = nullptr, *msm_entries = nullptr;
    uint32_t *msm_flag = nullptr;
    uint32_t *msm_nsl = nullptr, *msm_sloff = nullptr, *msm_perm = nullptr, *msm_hist = nullptr, *msm_sbkt = nullptr;
    void *msm_range = nullptr;
    size_t msm_max_slices = 0;
    pt *msm_buckets = nullptr, *msm_win = nullptr, *msm_part = nullptr, *msm_acc = nullptr, *msm_tmp = nullptr;
    apt *msm_aff2 = nullptr;  // the 2n virtual points of the endomorphism form
    pt *msm_bsum = nullptr;   // dense per-bucket sums (short-slice plans)
    void *msm_half = nullptr; // the 2n 128-bit scalar halves
    void *msm_cub = nullptr;
    size_t msm_cub_bytes = 0;
    // BIP-340 batch verification (api_msm.cu): seed, the scalar sum and its bytes, then one root per chunk
    uint32_t *bat = nullptr;
    size_t bat_chunks = 0;
    // optional per-kernel timing of the dominant kernel (bench.py roofline)
    bool profiling = false;
    // sub-chunks per host-pointer call (S256_PIPE_PARTS).  Measured (scripts/e2e_parts.py): splitting does not
    // pay -- the batched-inversion kernel is latency bound, so its cost multiplies with the part count.
    int pipe_parts = 1;
    cudaEvent_t ev_decode = nullptr, ev_pipe[10] = {};
    // recorded when a call has enqueued its last work; the next call's streams wait on it (scratch_guard below)
    cudaEvent_t ev_idle = nullptr;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> dsm_events;
    // multi-GPU MSM (api_msm.cu): an ncclComm_t built by s256_comm_init, and the 112-byte rows of the gather
    void *comm = nullptr;
    int comm_rank = 0, comm_size = 0;
    void *comm_buf = nullptr;
};
#define S256_COMM_MAX_RANKS 72

#define CK(call)                                                                     \
    do {                                                                             \
        cudaError_t e_ = (call);                                                     \
        if (e_ != cudaSuccess) {                                                     \
            ctx->last_err = std::string(#call) + ": " + cudaGetErrorString(e_);      \
            return S256_ERR_CUDA;                                                    \
        }                                                                            \
    } while (0)

static inline unsigned grid_for(size_t n) { return (unsigned)((n + S256_TPB - 1) / S256_TPB); }
#define LAUNCH(ctx, kern, grid, smem, strm, ...)                  \
    do {                                                          \
        kern<<<(grid), S256_TPB, (smem), (strm)>>>(__VA_ARGS__);  \
        (ctx)->launches.fetch_add(1, std::memory_order_relaxed);  \
    } while (0)

struct dev_guard {
    int prev = -1;
    explicit dev_guard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
    }
    ~dev_guard() {
        int cur = -1;
        cudaGetDevice(&cur);
        if (prev >= 0 && cur != prev) cudaSetDevice(prev);
    }
};


// A window into the per-item scratch arrays starting at item `off`: sub-chunks of one call work on
// disjoint windows, so they can be in flight on different streams at the same time.
struct view {
    apt *aff;
    sc *u1;
    int8_t *dig1, *dig2;
    uint8_t *sfl, *pvalid, *cstat;
    pt *tbl, *res;
    uint8_t *in_a, *in_b, *in_c, *out, *st;
};
static inline view view_at(const s256_ctx *ctx, size_t off) {
    view v;
    v.aff = ctx->aff + off;
    v.u1 = ctx->u1 + off;
    v.dig1 = ctx->dig1 + (size_t)DSM_ND * off;  // [digit][item] inside the window
    v.dig2 = ctx->dig2 + (size_t)DSM_ND * off;
    v.sfl = ctx->sfl + off;
    v.pvalid = ctx->pvalid + off;
    v.cstat = ctx->cstat + off;
    v.tbl = ctx->tbl + (size_t)DSM_TSTRIDE * off;
    v.res = ctx->res + off;
    v.in_a = ctx->in_a + 65 * off;
    v.in_b = ctx->in_b + 32 * off;
    v.in_c = ctx->in_c + 65 * off;
    v.out = ctx->out + 65 * off;
    v.st = ctx->st + off;
    return v;
}


#ifndef S256_INV_K
#define S256_INV_K 32
#endif
constexpr int INV_K = S256_INV_K;
// Inversion group size by batch size: K items share one Fermat chain but are processed serially by
// one thread, so small batches use small groups (n = 4096 with K = 32 would run on 128 threads).
static inline int inv_k_for(size_t n) { return n >= ((size_t)1 << 19) ? INV_K : (n >= ((size_t)1 << 16) ? 4 : 1); }
#define DISPATCH_K(n, CALL)               \
    do {                                  \
        switch (inv_k_for(n)) {           \
            case 1: { constexpr int KK = 1; CALL; } break;  \
            case 4: { constexpr int KK = 4; CALL; } break;  \
            default: { constexpr int KK = INV_K; CALL; } break; \
        }                                 \
    } while (0)
constexpr int MSM_MAX_PARTS = 64;  // (2^16 buckets) / (128 threads * 8 buckets)
static inline unsigned grid_for_groups(size_t n, int k) { return grid_for((n + k - 1) / k); }

// Runs `body(offset, count)` over chunks of at most cap items.
template <typename F>
static int for_chunks(s256_ctx *ctx, size_t n, F body) {
    for (size_t off = 0; off < n; off += ctx->cap) {
        size_t c = n - off < ctx->cap ? n - off : ctx->cap;
        int rc = body(off, c);
        if (rc != S256_SUCCESS) return rc;
    }
    return S256_SUCCESS;
}
// Host-pointer calls: the chunk is cut into sub-chunks that alternate between two streams, each
// doing its own H2D -> kernels -> D2H on a disjoint scratch window, so the copies of one sub-chunk
// overlap the kernels of the other.  body(view, global offset, count, stream).
// Default (pipe_parts == 1, "auto"): chunks of >= 2^18 items are cut at 6/64, 24/64 and 44/64 -- a small
// first part so that the main kernel starts early, growing parts so that the copies and the short
// latency-bound preparation kernels of part k+1 hide under the main kernel of part k, and a last part
// small enough that its trailing D2H stays short; entry points that return one byte per item use two
// parts (1/8, 7/8).  Measured in DESIGN.md section 5; S256_PIPE_CUTS overrides the cut points.  S256_PIPE_PARTS=n > 1 forces n equal parts
// (measured slower, DESIGN.md section 5); S256_PIPE_PARTS=0 disables the split.
template <typename F>
static int pipelined(s256_ctx *ctx, size_t n, F body, bool small_output = false) {
    const size_t min_sub = 65536;
    for (size_t off = 0; off < n; off += ctx->cap) {
        size_t c = n - off < ctx->cap ? n - off : ctx->cap;
        size_t cut[17];
        int np = 1;
        cut[0] = 0;
        if (ctx->pipe_parts == 1 && c >= ((size_t)1 << 18)) {
            if (small_output) {  // one byte per item comes back: no trailing D2H to keep short
                np = 2;
                cut[1] = (c / 8 + 127) & ~(size_t)127;
            } else {
                np = 4;
                cut[1] = (c / 64 * 6 + 127) & ~(size_t)127;
                cut[2] = (c / 64 * 24 + 127) & ~(size_t)127;
                cut[3] = (c / 64 * 44 + 127) & ~(size_t)127;
            }
            if (const char *cs = getenv("S256_PIPE_CUTS")) {  // tuning knob: cut points in 64ths, increasing
                int k = 1, prev = 0;
                for (const char *q = cs; *q && k < 8;) {
                    int v = atoi(q);
                    if (v <= prev || v >= 64) break;
                    cut[k++] = (c / 64 * (size_t)v + 127) & ~(size_t)127;
                    prev = v;
                    while (*q && *q != ',') q++;
                    if (*q == ',') q++;
                }
                np = k;
            }
        } else if (ctx->pipe_parts > 1) {
            size_t parts = c / min_sub;
            if (parts > (size_t)ctx->pipe_parts) parts = (size_t)ctx->pipe_parts;
            if (parts < 1) parts = 1;
            size_t sub = (c + parts - 1) / parts;
            sub = (sub + 127) & ~(size_t)127;
            np = 0;
            for (size_t so = 0; so < c; so += sub) cut[np++] = so;
        }
        cut[np] = c;
        for (int k = 0; k < np; k++) {
            size_t so = cut[k], sc_ = cut[k + 1] - cut[k];
            int rc = body(view_at(ctx, so), off + so, sc_, (k & 1) ? ctx->stream2 : ctx->stream);
            if (rc != S256_SUCCESS) return rc;
        }
        CK(cudaStreamSynchronize(ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream2));
    }
    return S256_SUCCESS;
}
static inline int check_launch(s256_ctx *ctx) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        ctx->last_err = std::string("kernel launch: ") + cudaGetErrorString(e);
        return S256_ERR_CUDA;
    }
    return S256_SUCCESS;
}


// Grows the variable-width staging buffer in_b: the new buffer is allocated FIRST and swapped in only on success, so a
// failed allocation leaves the context exactly as it was (never with in_b == NULL).
static inline int grow_in_b(s256_ctx *ctx, size_t need) {
    if (need <= ctx->in_b_bytes) return S256_SUCCESS;
    uint8_t *fresh = nullptr;
    if (cudaMalloc(&fresh, need) != cudaSuccess) {
        cudaGetLastError();
        ctx->last_err = "cudaMalloc(staging buffer)";
        return S256_ERR_NOMEM;
    }
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->stream2);
    cudaStreamSynchronize(ctx->stream3);
    if (ctx->in_b) cudaFree(ctx->in_b);
    ctx->in_b = fresh;
    ctx->in_b_bytes = need;
    return S256_SUCCESS;
}

// The host forms of the *_varlen entry points: message row i is msg[offsets[i], offsets[i + 1]), n + 1 offsets, and the
// rows are staged by chunks of at most `chunk` rows.  Rejects decreasing offsets (S256_ERR_ARG, before anything is
// enqueued) and a NULL msg under non-empty rows, then grows the staging: in_b to the bytes of the longest chunk, in_off
// to 2 chunk + 2 offsets.  A part starting at row `so` of its chunk takes its c + 1 offsets at in_off + 2 so, so that
// the parts of a pipelined chunk (on two streams) never write the same entry.  S256_ERR_NOMEM if that does not fit.
static inline int varlen_staging(s256_ctx *ctx, const uint8_t *msg, const size_t *offsets, size_t n, size_t chunk) {
    for (size_t i = 0; i < n; i++)
        if (offsets[i + 1] < offsets[i]) return S256_ERR_ARG;
    if (!msg && offsets[n] != offsets[0]) return S256_ERR_ARG;
    size_t span = 1;
    for (size_t off = 0; off < n; off += chunk) {
        const size_t c = n - off < chunk ? n - off : chunk;
        if (offsets[off + c] - offsets[off] > span) span = offsets[off + c] - offsets[off];
    }
    if (int rc = grow_in_b(ctx, span)) return rc;
    const size_t count = 2 * (n < chunk ? n : chunk) + 2;
    if (count <= ctx->in_off_count) return S256_SUCCESS;
    size_t *fresh = nullptr;
    if (cudaMalloc(&fresh, count * sizeof(size_t)) != cudaSuccess) {
        cudaGetLastError();
        ctx->last_err = "cudaMalloc(offset staging)";
        return S256_ERR_NOMEM;
    }
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->stream2);
    cudaStreamSynchronize(ctx->stream3);
    if (ctx->in_off) cudaFree(ctx->in_off);
    ctx->in_off = fresh;
    ctx->in_off_count = count;
    return S256_SUCCESS;
}
// Stages rows [off, off + c) of a *_varlen host call whose chunk starts at row off - so: the bytes go to their place in
// in_b (relative to the chunk's first byte), the offsets as they are to in_off + 2 so.  The rows' accessor on `s`.
static inline int varlen_stage_part(s256_ctx *ctx, const uint8_t *msg, const size_t *offsets, size_t off, size_t so, size_t c,
                                    cudaStream_t s, msg_offsets &rows) {
    uint8_t *dmsg = ctx->in_b + (offsets[off] - offsets[off - so]);
    size_t *doff = ctx->in_off + 2 * so;
    const size_t bytes = offsets[off + c] - offsets[off];
    if (bytes) CK(cudaMemcpyAsync(dmsg, msg + offsets[off], bytes, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(doff, offsets + off, (c + 1) * sizeof(size_t), cudaMemcpyHostToDevice, s));
    rows = msg_offsets{dmsg, doff, offsets[off]};
    return S256_SUCCESS;
}

// Error-path hygiene for the entry points that handle secrets (signing, ScalarMult / ECDH): a CUDA failure makes the
// normal code return before its own targeted wipes, so the caller of this helper clears every scratch array that can
// hold a private scalar, a nonce, k*P in projective form or a shared x, for the whole context capacity.
static inline void wipe_secret_scratch(s256_ctx *ctx) {
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->stream2);
    cudaStreamSynchronize(ctx->stream3);
    cudaGetLastError();
    const size_t m = ctx->cap;
    cudaMemsetAsync(ctx->u1, 0, sizeof(sc) * m, ctx->stream);
    cudaMemsetAsync(ctx->res, 0, sizeof(pt) * m, ctx->stream);
    cudaMemsetAsync(ctx->tbl, 0, 97 * m, ctx->stream);  // BIP-340 signing keeps R and k' at the start of this area
    cudaMemsetAsync(ctx->in_a, 0, 65 * m, ctx->stream);
    cudaMemsetAsync(ctx->in_b, 0, ctx->in_b_bytes, ctx->stream);
    cudaMemsetAsync(ctx->in_c, 0, 65 * m, ctx->stream);
    cudaMemsetAsync(ctx->out, 0, 65 * m, ctx->stream);
    cudaStreamSynchronize(ctx->stream);
}

#define ENTER(ctx)                       \
    if (!(ctx)) return S256_ERR_ARG;     \
    std::lock_guard<std::mutex> lk_((ctx)->mu); \
    dev_guard dg_((ctx)->device)


// Device-side ordering between calls.  Every entry point works in the one per-context scratch, and a *_dev call returns
// as soon as its kernels are enqueued on the CALLER's stream; the mutex (ENTER) only orders the enqueueing.  Without more,
// a second call on another stream -- or a host-pointer call on the context's own streams -- could overwrite scratch the
// first one is still using (verdicts silently wrong; in the signing path the nonce k shares a buffer with u1, so a clash
// between k*G and the finishing kernel would sign with a different k than the one behind r and leak the key).  So the
// streams a call uses first wait on ev_idle, and the call records ev_idle on its stream when it is done enqueueing.
// (Waiting on an event that was never recorded is a no-op.)
struct scratch_guard {
    s256_ctx *c;
    cudaStream_t s;
    scratch_guard(s256_ctx *c_, cudaStream_t s_, bool internal_streams) : c(c_), s(s_) {
        cudaStreamWaitEvent(s, c->ev_idle, 0);
        if (internal_streams) {
            if (c->stream != s) cudaStreamWaitEvent(c->stream, c->ev_idle, 0);
            cudaStreamWaitEvent(c->stream2, c->ev_idle, 0);
            cudaStreamWaitEvent(c->stream3, c->ev_idle, 0);
        }
    }
    ~scratch_guard() { cudaEventRecord(c->ev_idle, s); }
    scratch_guard(const scratch_guard &) = delete;
    scratch_guard &operator=(const scratch_guard &) = delete;
};

// launchers of kernels that live in api.cu but are needed by the other units
void s256_launch_decode_uncompressed(s256_ctx *ctx, const uint8_t *pt65, size_t n, apt *aff, uint8_t *pvalid, cudaStream_t s);
void s256_launch_finish_affine(s256_ctx *ctx, size_t n, const pt *res, const uint8_t *pvalid, const uint8_t *sfl,
                               uint8_t *cstat, int mode, uint8_t *out, uint8_t *status, const uint8_t *sig64,
                               cudaStream_t s);
void s256_internal_comm_release(s256_ctx *ctx);  // api_msm.cu: destroys the NCCL communicator, if any
void s256_launch_scalar_mult_ct(size_t n, const apt *aff, const uint8_t *k32, pt *tbl, pt *res, cudaStream_t s);
