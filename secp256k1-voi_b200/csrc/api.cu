// api.cu -- C ABI (include/secp256k1_b200.h) over the sm_100a kernels: lifecycle, the verification /
// multiplication entry points and their kernels.  MSM lives in api_msm.cu, signing in api_sign.cu.
//
// Host side only orchestrates: device buffers, copies, launches.  There is no
// CPU implementation of any curve operation in this library: without a CUDA
// device every entry point fails with S256_ERR_NO_DEVICE.
#include "ctx.h"
#include "microbench.cuh"

// ---------------------------------------------------------------------------
// __global__ wrappers
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(S256_TPB) k_gen_table(apt *out, int wb, size_t total) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    uint32_t w = (uint32_t)(idx >> wb), d = (uint32_t)(idx & ((1u << wb) - 1u));
    apt a;
    item_gen_multiple(a, w, d, wb);
    out[idx] = a;
}
// The signed comb of the verification ladder (kernels.cuh): out[w][j] = (j + 1) * B_w, B_w = 2^(COMB_WB*w) * G.
// 25 M entries, so not one bit-serial multiple and one inversion each (k_gen_table): a thread owns COMB_RUN
// consecutive entries of one window, reaches the first by double-and-add over B_w, walks the rest with
// mixed additions of B_w, and converts all of them with one shared inversion.
__global__ void k_comb_bases(apt *bases) {
    uint32_t w = threadIdx.x;
    if (w < (uint32_t)COMB_NW) item_gen_multiple(bases[w], w, 1u, COMB_WB);
}
constexpr int COMB_RUN = 32;
static_assert(COMB_SZ % COMB_RUN == 0, "a run never straddles two windows");
__global__ void __launch_bounds__(S256_TPB) k_gen_comb(const apt *bases, size_t total, apt *out) {
    size_t e0 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * COMB_RUN;
    if (e0 >= total) return;
    const apt B = bases[e0 / COMB_SZ];
    const uint32_t m = (uint32_t)(e0 % COMB_SZ) + 1u;  // first multiplier of the run, <= 2^(WB-1)
    pt buf[COMB_RUN];
    pt acc;
    pt_set_identity(acc);
#pragma unroll 1
    for (int b = COMB_WB - 1; b >= 0; b--) {
        pt_double(acc, acc);
        if ((m >> b) & 1u) pt_add_mixed(acc, acc, B.x, B.y);
    }
    buf[0] = acc;
#pragma unroll 1
    for (int i = 1; i < COMB_RUN; i++) {
        pt_add_mixed(acc, acc, B.x, B.y);
        buf[i] = acc;
    }
    fe pre[COMB_RUN], run = fe_one(), inv;
#pragma unroll 1
    for (int i = 0; i < COMB_RUN; i++) {
        pre[i] = run;
        fe_mul(run, run, buf[i].z);  // never zero: (j + 1) * 2^(WB*w) < n
    }
    fe_invert(inv, run);
#pragma unroll 1
    for (int i = COMB_RUN - 1; i >= 0; i--) {
        fe zi;
        apt a;
        fe_mul(zi, inv, pre[i]);
        fe_mul(inv, inv, buf[i].z);
        fe_mul(a.x, buf[i].x, zi);
        fe_mul(a.y, buf[i].y, zi);
        fe_normalize(a.x, a.x);
        fe_normalize(a.y, a.y);
        out[e0 + i] = a;
    }
}
// the signed constant-time table: out[w][j] = (j + 1) * 2^(CT_WB*w) * G
template <int WB>
__global__ void __launch_bounds__(S256_TPB) k_gen_ct_table(apt *out) {
    constexpr int CT_SZ = ct_cfg<WB>::SZ, CT_NW = ct_cfg<WB>::NW, CT_WB = WB;
    uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (uint32_t)(CT_NW * CT_SZ)) return;
    apt a;
    item_gen_multiple(a, idx / CT_SZ, idx % CT_SZ + 1u, CT_WB);
    out[idx] = a;
}

__global__ void __launch_bounds__(S256_TPB) k_decode_uncompressed(const uint8_t *pt65, size_t n, apt *aff,
                                                                  uint8_t *pvalid) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    apt a;
    pvalid[i] = item_decode_uncompressed(a, pt65 + 65 * i);
    aff[i] = a;
}

__global__ void __launch_bounds__(S256_TPB) k_decode_compressed(const uint8_t *pt33, size_t n, apt *aff,
                                                                uint8_t *pvalid) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    apt a;
    pvalid[i] = item_decode_compressed(a, pt33 + 33 * i);
    aff[i] = a;
}
// secec.NewPublicKey (secec/secec.go:183-199) over rows of mixed SEC 1 encodings (stride 65, len[i] bytes
// used): Point.SetBytes (point_s11n.go:209-228) dispatches on the length; the identity encoding is a
// valid point but not a public key (errAIsInfinity).  pvalid: 1 ok, 0 invalid, 2 identity.
__global__ void __launch_bounds__(S256_TPB) k_decode_sec1(const uint8_t *enc65, const uint8_t *len, size_t n, apt *aff,
                                                          uint8_t *pvalid) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t *e = enc65 + 65 * i;
    apt a;
    a.x = fe_zero();
    a.y = fe_zero();
    uint8_t st = ST_INVALID;
    if (len[i] == 65)
        st = item_decode_uncompressed(a, e) ? ST_OK : ST_INVALID;
    else if (len[i] == 33)
        st = item_decode_compressed(a, e) ? ST_OK : ST_INVALID;
    else if (len[i] == 1 && e[0] == 0x00)
        st = ST_IDENTITY;
    pvalid[i] = st;
    aff[i] = a;
}
// affine (validated) -> 65-byte encoding; invalid -> zeros, status = the decoder's code
__global__ void __launch_bounds__(S256_TPB) k_encode_affine(const apt *aff, const uint8_t *pvalid, size_t n,
                                                            uint8_t *out65, uint8_t *status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    apt a = aff[i];
    uint32_t ok = pvalid[i] != 0;
    uint8_t *o = out65 + 65 * i;
    if (ok) {
        o[0] = 0x04;
        fe_to_be32(o + 1, a.x);
        fe_to_be32(o + 33, a.y);
    } else {
        for (int b = 0; b < 65; b++) o[b] = 0;
    }
    status[i] = ok ? ST_OK : ST_INVALID;
}
// affine (validated) -> 33-byte compressed encoding (point_s11n.go:90-117); invalid -> zeros
__global__ void __launch_bounds__(S256_TPB) k_encode_compressed(const apt *aff, const uint8_t *pvalid, size_t n,
                                                                uint8_t *out33, uint8_t *status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    apt a = aff[i];
    uint32_t ok = pvalid[i] != 0;
    uint8_t *o = out33 + 33 * i;
    if (ok) {
        o[0] = (uint8_t)(0x02u | fe_is_odd(a.y));
        fe_to_be32(o + 1, a.x);
    } else {
        for (int b = 0; b < 33; b++) o[b] = 0;
    }
    status[i] = ok ? ST_OK : ST_INVALID;
}
__global__ void __launch_bounds__(S256_TPB) k_encode_public_key(const apt *aff, const uint8_t *pvalid, size_t n,
                                                                uint8_t *out65, uint8_t *status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    apt a = aff[i];
    uint8_t *o = out65 + 65 * i;
    if (pvalid[i] == ST_OK) {
        o[0] = 0x04;
        fe_to_be32(o + 1, a.x);
        fe_to_be32(o + 33, a.y);
    } else {
        for (int b = 0; b < 65; b++) o[b] = 0;
    }
    status[i] = pvalid[i];
}

// BIP-340 lift_x: x-only key, even y (secec/bitcoin/schnorr.go:257-275)
__global__ void __launch_bounds__(S256_TPB) k_decode_xonly(const uint8_t *pkx32, size_t n, apt *aff, uint8_t *pvalid) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    apt a;
    pvalid[i] = item_decode_xonly(a, pkx32 + 32 * i);
    aff[i] = a;
}

// RecoverPoint (point_s11n.go:245-282): x = r (+ n if v & 2), parity v & 1
__global__ void __launch_bounds__(S256_TPB) k_decode_recover(const uint8_t *sig65, size_t n, apt *aff,
                                                             uint8_t *pvalid) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    apt a;
    pvalid[i] = item_decode_recover(a, sig65 + 65 * i);
    aff[i] = a;
}

template <int K, bool RECOVER>
__global__ void __launch_bounds__(S256_TPB, 4) k_ecdsa_scalars(const uint8_t *digest32, const uint8_t *sig, size_t n,
                                                            uint32_t flags, sc *u1, int8_t *dig1, int8_t *dig2,
                                                            uint8_t *sfl) {
    size_t stride = (n + K - 1) / K;
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= stride) return;
    if (!RECOVER)
        group_ecdsa_scalars<K>(t, stride, n, digest32, sig, flags, u1, dig1, dig2, sfl);
    else
        group_recover_scalars<K>(t, stride, n, digest32, sig, u1, dig1, dig2, sfl);
}

__global__ void __launch_bounds__(S256_TPB) k_plain_scalars(const uint8_t *u1b, const uint8_t *u2b, size_t n, sc *u1,
                                                            int8_t *dig1, int8_t *dig2, uint8_t *sfl) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    item_plain_scalars(i, n, u1b, u2b, u1, dig1, dig2, sfl);
}

// secec/bitcoin/schnorr.go:420-449: r < p, s < n (zero allowed), e = H(r||P||m) mod n;
// R = s*G + (-e)*P (:244-245)
__global__ void __launch_bounds__(S256_TPB) k_schnorr_scalars(const uint8_t *pkx32, const uint8_t *msg, size_t msg_len,
                                                              const uint8_t *sig64, size_t n, sc *u1, int8_t *dig1,
                                                              int8_t *dig2, uint8_t *sfl) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    item_schnorr_scalars(i, n, pkx32, msg, msg_len, sig64, u1, dig1, dig2, sfl);
}

#ifndef S256_DSM_MINB
#define S256_DSM_MINB 4
#endif
#ifndef S256_DSM_TPB
#define S256_DSM_TPB S256_TPB
#endif
// One inversion per CTA instead of one per item (Montgomery's trick across the CTA; used by the constant-time ladder
// for its public table -- the verification ladder needs no inversion any more): every thread leaves the product
// of its table's Z's in shared memory, warp 0 takes TPB / 32 of them per lane, multiplies them up, forms the
// product of all OTHER lanes' values with an xor butterfly (9 products), inverts the CTA's total once (safegcd: 23 k
// instructions, which each of the four warps used to spend) and walks back to the individual inverses.  Public data.
__device__ __forceinline__ void fe_shfl_xor(fe &r, const fe &a, int m) {
#pragma unroll
    for (int k = 0; k < 8; k++) r.v[k] = __shfl_xor_sync(0xFFFFFFFFu, a.v[k], m);
}
template <int TPB, class F>
__device__ __forceinline__ void cta_invert(F &f, fe &inv, const fe &c, fe *sh) {
    constexpr int PER = TPB / 32;
    sh[threadIdx.x] = c;
    __syncthreads();
    // (warp 0 always: rotating the inverting warp over the SM's four schedulers measured 0.5 % slower)
    if (threadIdx.x < 32) {
        fe *mine = sh + threadIdx.x * PER;
        fe pre[PER];
        pre[0] = mine[0];
#pragma unroll
        for (int k = 1; k < PER; k++) f.mul(pre[k], pre[k - 1], mine[k]);
        fe all = pre[PER - 1], others, got;
        fe_shfl_xor(others, all, 1);
        f.mul(all, all, others);
#pragma unroll 1
        for (int m = 2; m < 32; m <<= 1) {
            fe_shfl_xor(got, all, m);
            f.mul(others, others, got);
            f.mul(all, all, got);
        }
        fe o;
        fe_invert(o, all);
        f.mul(o, o, others);  // (this lane's product)^-1
#pragma unroll
        for (int k = PER - 1; k >= 1; k--) {
            fe ck = mine[k], t;
            f.mul(t, o, pre[k - 1]);
            f.mul(o, o, ck);
            mine[k] = t;
        }
        mine[0] = o;
    }
    __syncthreads();
    inv = sh[threadIdx.x];
}
__global__ void __launch_bounds__(S256_DSM_TPB, S256_DSM_MINB)
    k_dsm(size_t n, const apt *aff, const sc *u1, const int8_t *dig1, const int8_t *dig2, const uint8_t *sfl, pt *tbl,
          pt *res, const apt *comb) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    item_dsm(i, n, aff, u1, dig1, dig2, sfl, tbl, res, comb);
}

// 4-bit windows over an affine table: entries 2..8 x 64 bytes per thread = 56 KB of shared memory per CTA, four CTAs per SM
#ifndef S256_SM_MINB
#define S256_SM_MINB 4
#endif
__global__ void __launch_bounds__(S256_TPB, S256_SM_MINB)
    k_scalar_mult_ct(size_t n, const apt *aff, const uint8_t *k32, pt *tbl, pt *res) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
#ifdef S256_CT_TABLE_GLOBAL
    if (i >= n) return;
    CtTableGlobal T{tbl + i * (size_t)DSM_TSTRIDE};
    item_scalar_mult_ct_affine(i, aff, k32, T, tbl + i * (size_t)DSM_TSTRIDE, res);
#else
    // the table is public (multiples of the peer's point): one inversion for the CTA, as in k_dsm.  The exchange area
    // is the front of the (not yet written) table columns: a static array would cost the fourth CTA of the SM.
    extern __shared__ uint4 ct_smem[];
    fe *sh = reinterpret_cast<fe *>(ct_smem);
    const bool live = i < n;
    fe_ops<true> f;
    fe zprod = fe_one(), inv;
    if (live) item_ctm_table(i, aff, tbl + i * (size_t)DSM_TSTRIDE, zprod);
    cta_invert<S256_TPB>(f, inv, zprod, sh);
    __syncthreads();  // every inverse has been read before the first table column lands on the exchange area
    if (!live) return;
    CtTableShared<S256_TPB> T{threadIdx.x, aff + i};
    item_ctm_ladder(i, aff, k32, T, tbl + i * (size_t)DSM_TSTRIDE, inv, res);
#endif
}
#ifdef S256_CT_TABLE_GLOBAL
constexpr size_t CT_SMEM_BYTES = 0;
#else
constexpr size_t CT_SMEM_BYTES = (size_t)(CTM_TS - 1) * 4 * S256_TPB * sizeof(uint4);
#endif
void s256_launch_scalar_mult_ct(size_t n, const apt *aff, const uint8_t *k32, pt *tbl, pt *res, cudaStream_t s) {
    if (n == 0) return;
    k_scalar_mult_ct<<<(unsigned)((n + S256_TPB - 1) / S256_TPB), S256_TPB, CT_SMEM_BYTES, s>>>(n, aff, k32, tbl, res);
}


__global__ void __launch_bounds__(S256_TPB) k_ecdsa_finish(size_t n, const pt *res, const uint8_t *sig64,
                                                           const uint8_t *pvalid, const uint8_t *sfl, uint8_t *ok) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    pt R = res[i];
    uint32_t valid = (uint32_t)(pvalid[i] != 0) & (uint32_t)(sfl[i] & SFL_VALID);
    ok[i] = item_ecdsa_finish(R, sig64 + 64 * i, valid);
}

// in-status = pvalid (may be null) AND sfl valid bit (may be null)
template <int K>
__global__ void __launch_bounds__(S256_TPB) k_finish_affine(size_t n, const pt *res, const uint8_t *pvalid,
                                                            const uint8_t *sfl, uint8_t *comb_status, int mode,
                                                            uint8_t *out, uint8_t *status, const uint8_t *sig64) {
    __shared__ uint4 stage[S256_TPB / 32][130];  // 2080 bytes per warp: 32 rows of 65 bytes (kernels.cuh)
    // a multiple of 32, so that the items a warp converts together start at a multiple of 32 (the
    // staged 2080-byte block is then 16-byte aligned in `out`)
    size_t stride = (((n + K - 1) / K) + 31) & ~(size_t)31;
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= stride) return;
    group_finish<K>(t, stride, n, res, pvalid, sfl, comb_status, mode, out, status, sig64,
                    reinterpret_cast<uint8_t *>(stage[threadIdx.x / 32]));
}

__global__ void __launch_bounds__(S256_TPB) k_field_op(int op, const uint8_t *a32, const uint8_t *b32, size_t n,
                                                       uint8_t *out32) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (op < 16 || op >= 20) {
        fe a, b, r;
        fe_from_be32(a, a32 + 32 * i);
        fe_from_be32(b, b32 + 32 * i);
        switch (op) {
            case 0: fe_mul(r, a, b); break;
            case 1: fe_add(r, a, b); break;
            case 2: fe_sub(r, a, b); break;
            case 3: fe_invert(r, a); break;
            case 4: fe_sqrt(r, a); break;
            case 5: fe_mul_small(r, a, 21u); break;
            case 6: fe_sqr(r, a); break;
            case 7: fe_invert_fermat(r, a); break;
            // 8 + op: the variable-time flavour (fe_vt.cuh) of the same operation
            case 8: fe_mul_vt(r, a, b); break;
            case 9: fe_add_vt(r, a, b); break;
            case 10: fe_sub_vt(r, a, b); break;
            case 13: fe_mul_small_vt(r, a, 21u); break;
            case 14: fe_sqr_vt(r, a); break;
            case 15: fe_mul8_vt(r, a); break;
            case 20: fe_mul2_vt(r, a); break;
            case 21: fe_mul3_vt(r, a); break;
            case 22: fe_sub2_vt(r, a, b); break;
            case 23: fe_submul8_vt(r, a, b); break;
            case 24: fe_ops<false>::mul2add(r, a, b, b, a); break;  // the constant-time fused a b + c d (device)
            case 25: fe_ops<false>::mul2sub(r, a, a, b, b); break;
            default: r = fe_zero();
        }
        fe_normalize(r, r);
        fe_to_be32(out32 + 32 * i, r);
    } else {
        sc a, b, r;
        sc_from_be32(a, a32 + 32 * i);
        sc_from_be32(b, b32 + 32 * i);
        switch (op) {
            case 16: sc_mul(r, a, b); break;
            case 17: sc_add(r, a, b); break;
            case 18: sc_invert(r, a); break;
            case 19: sc_invert_fermat(r, a); break;
            default: r = sc_zero();
        }
        sc_to_be32(out32 + 32 * i, r);
    }
}

// page-locked host memory for callers that want full-speed copies (cudaHostAllocPortable: any device)
extern "C" void *s256_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
extern "C" void s256_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

extern "C" const char *s256_strerror(int code) {
    switch (code) {
        case S256_SUCCESS: return "success";
        case S256_ERR_NO_DEVICE: return "no usable CUDA device (sm_100 required; there is no CPU fallback)";
        case S256_ERR_CUDA: return "CUDA runtime error";
        case S256_ERR_ARG: return "invalid argument";
        case S256_ERR_NOMEM: return "out of memory";
        case S256_ERR_UNIMPLEMENTED: return "not implemented";
        case S256_ERR_NCCL: return "NCCL error";
        default: return "unknown error";
    }
}
extern "C" const char *s256_last_cuda_error(const s256_ctx *ctx) { return ctx ? ctx->last_err.c_str() : ""; }
extern "C" int s256_device(const s256_ctx *ctx) { return ctx ? ctx->device : -1; }
extern "C" uint64_t s256_launch_count(const s256_ctx *ctx) { return ctx ? ctx->launches.load() : 0; }

extern "C" void s256_free(s256_ctx *ctx) {
    if (!ctx) return;
    {
        dev_guard g(ctx->device);
        s256_internal_comm_release(ctx);
        void *ptrs[] = {ctx->comb, ctx->ct_tab, ctx->ct_tab_small, ctx->ct_tab_huge, ctx->aff, ctx->u1,   ctx->dig1, ctx->dig2, ctx->sfl, ctx->pvalid,
                        ctx->cstat, ctx->tbl,   ctx->res, ctx->in_a, ctx->in_b, ctx->in_c, ctx->out, ctx->st,
                        ctx->sink, ctx->msm_counts, ctx->msm_offsets, ctx->msm_cursor, ctx->msm_entries, ctx->msm_flag,
                        ctx->msm_buckets, ctx->msm_win, ctx->msm_acc, ctx->msm_tmp, ctx->msm_cub, ctx->msm_nsl, ctx->msm_sloff,
                        ctx->msm_perm, ctx->msm_hist, ctx->msm_range, ctx->msm_part, ctx->msm_sbkt, ctx->comm_buf, ctx->msm_aff2, ctx->msm_half, ctx->msm_bsum,
                        ctx->bat};
        for (void *p : ptrs)
            if (p) cudaFree(p);
        if (ctx->stream) cudaStreamDestroy(ctx->stream);
        if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
        if (ctx->ev_decode) cudaEventDestroy(ctx->ev_decode);
        if (ctx->ev_idle) cudaEventDestroy(ctx->ev_idle);
        for (cudaEvent_t e : ctx->ev_pipe)
            if (e) cudaEventDestroy(e);
        if (ctx->stream3) cudaStreamDestroy(ctx->stream3);
    }
    delete ctx;
}

static int ctx_alloc(s256_ctx *ctx) {
    size_t cap = ctx->cap;
    CK(cudaMalloc(&ctx->comb, sizeof(apt) * ((size_t)COMB_NW * COMB_SZ + COMB_NW)));  // + the window bases B_w
    CK(cudaMalloc(&ctx->ct_tab, sizeof(apt) * ct_cfg<CT_WB>::NW * ct_cfg<CT_WB>::SZ));
    CK(cudaMalloc(&ctx->ct_tab_small, sizeof(apt) * ct_cfg<CT_WB_SMALL>::NW * ct_cfg<CT_WB_SMALL>::SZ));
    CK(cudaMalloc(&ctx->ct_tab_huge, sizeof(apt) * ct_cfg<7>::NW * ct_cfg<7>::SZ));
    CK(cudaMalloc(&ctx->aff, sizeof(apt) * cap));
    CK(cudaMalloc(&ctx->u1, sizeof(sc) * cap));
    CK(cudaMalloc(&ctx->dig1, (size_t)DSM_ND * cap));
    CK(cudaMalloc(&ctx->dig2, (size_t)DSM_ND * cap));
    CK(cudaMalloc(&ctx->sfl, cap));
    CK(cudaMalloc(&ctx->pvalid, cap));
    CK(cudaMalloc(&ctx->cstat, cap));
    CK(cudaMalloc(&ctx->tbl, sizeof(pt) * DSM_TSTRIDE * cap));
    CK(cudaMalloc(&ctx->res, sizeof(pt) * cap));
    CK(cudaMalloc(&ctx->in_a, 65 * cap));
    CK(cudaMalloc(&ctx->in_c, 65 * cap));
    CK(cudaMalloc(&ctx->in_b, 32 * cap));
    ctx->in_b_bytes = 32 * cap;
    CK(cudaMalloc(&ctx->out, 65 * cap));
    CK(cudaMalloc(&ctx->st, cap));
    CK(cudaMalloc(&ctx->sink, 16));
    return S256_SUCCESS;
}

extern "C" int s256_init(s256_ctx **out, int device, size_t max_batch) {
    if (!out) return S256_ERR_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return S256_ERR_NO_DEVICE;
    if (device < 0 && cudaGetDevice(&device) != cudaSuccess) return S256_ERR_NO_DEVICE;
    if (device >= count) return S256_ERR_ARG;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return S256_ERR_NO_DEVICE;
    if (prop.major != 10) return S256_ERR_NO_DEVICE;  // sm_100a code only
    s256_ctx *ctx = new (std::nothrow) s256_ctx;
    if (!ctx) return S256_ERR_NOMEM;
    ctx->device = device;
    ctx->cap = max_batch ? max_batch : ((size_t)1 << 20);
    dev_guard g(device);
    int rc = ctx_alloc(ctx);
    if (rc != S256_SUCCESS && cudaGetLastError() == cudaErrorMemoryAllocation) rc = S256_ERR_NOMEM;  // also clears the error
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);  // stream2 feeds stream: its short kernels go first
    if (rc == S256_SUCCESS && (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
                               cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
                               cudaStreamCreateWithPriority(&ctx->stream3, cudaStreamNonBlocking, prio_hi) != cudaSuccess))
        rc = S256_ERR_CUDA;
    if (rc == S256_SUCCESS && (cudaEventCreateWithFlags(&ctx->ev_decode, cudaEventDisableTiming) != cudaSuccess ||
                               cudaEventCreateWithFlags(&ctx->ev_idle, cudaEventDisableTiming) != cudaSuccess))
        rc = S256_ERR_CUDA;
    for (cudaEvent_t &e : ctx->ev_pipe)
        if (rc == S256_SUCCESS && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) rc = S256_ERR_CUDA;
    if (rc == S256_SUCCESS) {
        // generator tables (reference: package init, point_mul_table.go:75-100,147-160)
        size_t total = (size_t)COMB_NW * COMB_SZ;
        apt *bases = ctx->comb + total;
        k_comb_bases<<<1, 32, 0, ctx->stream>>>(bases);
        LAUNCH(ctx, k_gen_comb, grid_for(total / COMB_RUN), 0, ctx->stream, bases, total, ctx->comb);
        LAUNCH(ctx, k_gen_ct_table<CT_WB>, grid_for((size_t)ct_cfg<CT_WB>::NW * ct_cfg<CT_WB>::SZ), 0, ctx->stream,
               ctx->ct_tab);
        LAUNCH(ctx, k_gen_ct_table<CT_WB_SMALL>, grid_for((size_t)ct_cfg<CT_WB_SMALL>::NW * ct_cfg<CT_WB_SMALL>::SZ), 0,
               ctx->stream, ctx->ct_tab_small);
        LAUNCH(ctx, k_gen_ct_table<7>, grid_for((size_t)ct_cfg<7>::NW * ct_cfg<7>::SZ), 0, ctx->stream, ctx->ct_tab_huge);
        s256_ct_kernels_init();
        if (CT_SMEM_BYTES)
            cudaFuncSetAttribute(k_scalar_mult_ct, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CT_SMEM_BYTES);
        cudaFuncSetAttribute(k_scalar_mult_ct, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        const char *pp = getenv("S256_PIPE_PARTS");
        if (pp && atoi(pp) >= 0 && atoi(pp) <= 16) ctx->pipe_parts = atoi(pp);
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) {
            fprintf(stderr, "s256_init: table generation failed: %s\n", cudaGetErrorString(e));
            rc = S256_ERR_CUDA;
        }
    }
    if (rc != S256_SUCCESS) {
        s256_free(ctx);
        return rc;
    }
    *out = ctx;
    return S256_SUCCESS;
}

// ---------------------------------------------------------------------------
// device-pointer pipelines (one chunk <= cap)
// ---------------------------------------------------------------------------
void s256_launch_decode_uncompressed(s256_ctx *ctx, const uint8_t *pt65, size_t n, apt *aff, uint8_t *pvalid,
                                     cudaStream_t s) {
    LAUNCH(ctx, k_decode_uncompressed, grid_for(n), 0, s, pt65, n, aff, pvalid);
}
void s256_launch_finish_affine(s256_ctx *ctx, size_t n, const pt *res, const uint8_t *pvalid, const uint8_t *sfl,
                               uint8_t *cstat, int mode, uint8_t *out, uint8_t *status, const uint8_t *sig64,
                               cudaStream_t s) {
    DISPATCH_K(n, LAUNCH(ctx, k_finish_affine<KK>, grid_for_groups(n, KK), 0, s, n, res, pvalid, sfl, cstat, mode, out,
                         status, sig64));
}

static void enqueue_dsm(s256_ctx *ctx, const view &v, size_t n, cudaStream_t s) {
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (ctx->profiling) {
        cudaEventCreate(&e0);
        cudaEventCreate(&e1);
        cudaEventRecord(e0, s);
    }
    k_dsm<<<(unsigned)((n + S256_DSM_TPB - 1) / S256_DSM_TPB), S256_DSM_TPB, 0, s>>>(n, v.aff, v.u1, v.dig1, v.dig2, v.sfl, v.tbl,
                                                                                         v.res, ctx->comb);
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
    if (ctx->profiling) {
        cudaEventRecord(e1, s);
        ctx->dsm_events.emplace_back(e0, e1);
    }
}


// The scalar kernel needs digest + signature only and the decode kernel the public keys only: when the
// caller passes a second stream, decode runs there (behind the key copy) and joins through an event.
static int chunk_ecdsa_verify(s256_ctx *ctx, const view &v, const uint8_t *pk, const uint8_t *dg, const uint8_t *sig, uint32_t flags,
                              size_t n, uint8_t *ok, cudaStream_t s, cudaStream_t s_decode = nullptr) {
    DISPATCH_K(n, LAUNCH(ctx, (k_ecdsa_scalars<KK, false>), grid_for_groups(n, KK), 0, s, dg, sig, n, flags, v.u1,
                         v.dig1, v.dig2, v.sfl));
    if (s_decode && s_decode != s) {
        LAUNCH(ctx, k_decode_uncompressed, grid_for(n), 0, s_decode, pk, n, v.aff, v.pvalid);
        cudaEventRecord(ctx->ev_decode, s_decode);
        cudaStreamWaitEvent(s, ctx->ev_decode, 0);
    } else {
        LAUNCH(ctx, k_decode_uncompressed, grid_for(n), 0, s, pk, n, v.aff, v.pvalid);
    }
    enqueue_dsm(ctx, v, n, s);
    LAUNCH(ctx, k_ecdsa_finish, grid_for(n), 0, s, n, v.res, sig, v.pvalid, v.sfl, ok);
    return S256_SUCCESS;
}
static int chunk_ecdsa_recover(s256_ctx *ctx, const view &v, const uint8_t *dg, const uint8_t *sig65, size_t n, uint8_t *pk65,
                               uint8_t *status, cudaStream_t s) {
    LAUNCH(ctx, k_decode_recover, grid_for(n), 0, s, sig65, n, v.aff, v.pvalid);
    DISPATCH_K(n, LAUNCH(ctx, (k_ecdsa_scalars<KK, true>), grid_for_groups(n, KK), 0, s, dg, sig65, n, 0u, v.u1,
                         v.dig1, v.dig2, v.sfl));
    enqueue_dsm(ctx, v, n, s);
    DISPATCH_K(n, LAUNCH(ctx, k_finish_affine<KK>, grid_for_groups(n, KK), 0, s, n, v.res, v.pvalid, v.sfl, v.cstat,
           3, pk65, status, (const uint8_t *)nullptr));
    return S256_SUCCESS;
}
static int chunk_schnorr_verify(s256_ctx *ctx, const view &v, const uint8_t *pkx, const uint8_t *msg, size_t msg_len,
                                const uint8_t *sig, size_t n, uint8_t *ok, cudaStream_t s) {
    LAUNCH(ctx, k_decode_xonly, grid_for(n), 0, s, pkx, n, v.aff, v.pvalid);
    LAUNCH(ctx, k_schnorr_scalars, grid_for(n), 0, s, pkx, msg, msg_len, sig, n, v.u1, v.dig1, v.dig2,
           v.sfl);
    enqueue_dsm(ctx, v, n, s);
    DISPATCH_K(n, LAUNCH(ctx, k_finish_affine<KK>, grid_for_groups(n, KK), 0, s, n, v.res, v.pvalid, v.sfl, v.cstat,
           2, (uint8_t *)nullptr, ok, sig));
    return S256_SUCCESS;
}
static int chunk_dsm(s256_ctx *ctx, const view &v, const uint8_t *u1, const uint8_t *u2, const uint8_t *pt65, size_t n,
                     uint8_t *out65, uint8_t *status, cudaStream_t s) {
    LAUNCH(ctx, k_decode_uncompressed, grid_for(n), 0, s, pt65, n, v.aff, v.pvalid);
    LAUNCH(ctx, k_plain_scalars, grid_for(n), 0, s, u1, u2, n, v.u1, v.dig1, v.dig2, v.sfl);
    enqueue_dsm(ctx, v, n, s);
    DISPATCH_K(n, LAUNCH(ctx, k_finish_affine<KK>, grid_for_groups(n, KK), 0, s, n, v.res, v.pvalid,
           (const uint8_t *)nullptr, v.cstat, 0, out65, status, (const uint8_t *)nullptr));
    return S256_SUCCESS;
}
static int chunk_base_mult(s256_ctx *ctx, const view &v, const uint8_t *k32, size_t n, uint8_t *out65, uint8_t *status,
                           cudaStream_t s) {
    s256_launch_base_mult_ct(k32, n, ctx->ct_tab, ctx->ct_tab_small, ctx->ct_tab_huge, v.res, s);
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
    DISPATCH_K(n, LAUNCH(ctx, k_finish_affine<KK>, grid_for_groups(n, KK), 0, s, n, v.res, (const uint8_t *)nullptr,
           (const uint8_t *)nullptr, v.cstat, 0, out65, status, (const uint8_t *)nullptr));
    return S256_SUCCESS;
}

// Point.ScalarMult / PrivateKey.ECDH: decode (public) -> ct ladder -> batched affine
static int chunk_scalar_mult(s256_ctx *ctx, const view &v, const uint8_t *k32, const uint8_t *pt65, size_t n, int mode, uint8_t *out,
                             uint8_t *status, cudaStream_t s) {
    LAUNCH(ctx, k_decode_uncompressed, grid_for(n), 0, s, pt65, n, v.aff, v.pvalid);
    s256_launch_scalar_mult_ct(n, v.aff, k32, v.tbl, v.res, s);
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
    DISPATCH_K(n, LAUNCH(ctx, k_finish_affine<KK>, grid_for_groups(n, KK), 0, s, n, v.res, v.pvalid,
           (const uint8_t *)nullptr, v.cstat, mode, out, status, (const uint8_t *)nullptr));
    return S256_SUCCESS;
}

// ---------------------------------------------------------------------------
// exported entry points
// ---------------------------------------------------------------------------

extern "C" int s256_ecdsa_verify_dev(s256_ctx *ctx, const uint8_t *pk, const uint8_t *dg, const uint8_t *sig,
                                     uint32_t flags, size_t n, uint8_t *ok, void *stream) {
    ENTER(ctx);
    if (n && (!pk || !dg || !sig || !ok)) return S256_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    int rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        return chunk_ecdsa_verify(ctx, view_at(ctx, 0), pk + 65 * off, dg + 32 * off, sig + 64 * off, flags, c, ok + off, s);
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}
// Host-pointer verification as a pipeline over two sub-chunks, 3/16 and 13/16 of the chunk.
// Two feeder streams (high priority) carry the inputs in -- digests + signatures then the scalar kernel
// on one, public keys then the decode kernel on the other -- and the main stream runs the ladder and
// the final check of each sub-chunk as soon as both of its events have fired.  The ladder therefore
// starts after 3/16 of the copy, and the rest of the PCIe traffic and the second scalar kernel hide
// under the first ladder as long as the link sustains ~32 GB/s (a ladder consumes its 161 B/item at
// 7.5 GB/s).  Measured schedules (ms per 2^20 call on one GPU, S256_VERIFY_CUTS in 64ths): 6 -> 23.86,
// 8 -> 24.10, 12 -> 23.98, 16 -> 24.29, 4 -> 24.31, 4,16 -> 24.27, 2,8,32 -> 24.56, 2,6,16,36 -> 25.33:
// every extra part costs a latency-bound scalar kernel that takes SM slots from a ladder.  With eight
// GPUs copying at once each link gave ~34 GB/s and the 6/64 cut left a 2 ms bubble (26.1 ms per call),
// hence 12/64.
// S256_TRACE=1: device timestamps of the pipeline stages, printed per call (debug aid, off by default)
struct stage_trace {
    bool on;
    std::vector<std::pair<const char *, cudaEvent_t>> ev;
    cudaEvent_t t0 = nullptr;
    explicit stage_trace(cudaStream_t s) : on(getenv("S256_TRACE") != nullptr) {
        if (on) {
            cudaEventCreate(&t0);
            cudaEventRecord(t0, s);
        }
    }
    void mark(const char *what, cudaStream_t s) {
        if (!on) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, s);
        ev.emplace_back(what, e);
    }
    void dump() {
        if (!on) return;
        for (auto &p : ev) {
            float ms = 0;
            cudaEventSynchronize(p.second);
            cudaEventElapsedTime(&ms, t0, p.second);
            fprintf(stderr, "[s256 trace] %-12s %8.3f ms\n", p.first, ms);
            cudaEventDestroy(p.second);
        }
        cudaEventDestroy(t0);
    }
};
static int verify_pipelined(s256_ctx *ctx, const uint8_t *pk, const uint8_t *dg, const uint8_t *sig, uint32_t flags,
                            size_t off, size_t c, uint8_t *ok) {
    cudaStream_t feed = ctx->stream2, feed_pk = ctx->stream3, mainst = ctx->stream;
    // cut points in 64ths of the chunk; S256_VERIFY_CUTS="a,b,.." (each in 1..63, increasing) overrides them
    int P = 2;
    size_t cut[6] = {0, (c / 64 * 12 + 127) & ~(size_t)127, c, c, c, c};
    if (const char *cs = getenv("S256_VERIFY_CUTS")) {
        int k = 1, prev = 0;
        for (const char *q = cs; *q && k < 5;) {
            int v = atoi(q);
            if (v <= prev || v >= 64) break;
            cut[k++] = (c / 64 * (size_t)v + 127) & ~(size_t)127;
            prev = v;
            while (*q && *q != ',') q++;
            if (*q == ',') q++;
        }
        cut[k] = c;
        P = k;
    }
    stage_trace tr(feed);
    static const char *const names[5][4] = {{"sig+dg A", "scalars A", "decode A", "ladder A"},
                                            {"sig+dg B", "scalars B", "decode B", "ladder B"},
                                            {"sig+dg C", "scalars C", "decode C", "ladder C"},
                                            {"sig+dg D", "scalars D", "decode D", "ladder D"},
                                            {"sig+dg E", "scalars E", "decode E", "ladder E"}};
    for (int k = 0; k < P; k++) {
        size_t so = cut[k], n = cut[k + 1] - cut[k];
        view v = view_at(ctx, so);
        size_t g = off + so;
        CK(cudaMemcpyAsync(v.in_b, dg + 32 * g, 32 * n, cudaMemcpyHostToDevice, feed));
        CK(cudaMemcpyAsync(v.in_c, sig + 64 * g, 64 * n, cudaMemcpyHostToDevice, feed));
        tr.mark(names[k][0], feed);
        CK(cudaMemcpyAsync(v.in_a, pk + 65 * g, 65 * n, cudaMemcpyHostToDevice, feed_pk));
        DISPATCH_K(n, LAUNCH(ctx, (k_ecdsa_scalars<KK, false>), grid_for_groups(n, KK), 0, feed, v.in_b, v.in_c, n, flags, v.u1,
                             v.dig1, v.dig2, v.sfl));
        tr.mark(names[k][1], feed);
        CK(cudaEventRecord(ctx->ev_pipe[2 * k], feed));
        LAUNCH(ctx, k_decode_uncompressed, grid_for(n), 0, feed_pk, v.in_a, n, v.aff, v.pvalid);
        tr.mark(names[k][2], feed_pk);
        CK(cudaEventRecord(ctx->ev_pipe[2 * k + 1], feed_pk));
    }
    for (int k = 0; k < P; k++) {
        size_t so = cut[k], n = cut[k + 1] - cut[k];
        view v = view_at(ctx, so);
        CK(cudaStreamWaitEvent(mainst, ctx->ev_pipe[2 * k], 0));
        CK(cudaStreamWaitEvent(mainst, ctx->ev_pipe[2 * k + 1], 0));
        enqueue_dsm(ctx, v, n, mainst);
        tr.mark(names[k][3], mainst);
        LAUNCH(ctx, k_ecdsa_finish, grid_for(n), 0, mainst, n, v.res, v.in_c, v.pvalid, v.sfl, v.st);
    }
    CK(cudaMemcpyAsync(ok + off, ctx->st, c, cudaMemcpyDeviceToHost, mainst));
    tr.mark("d2h", mainst);
    CK(cudaStreamSynchronize(mainst));
    tr.dump();
    return S256_SUCCESS;
}
extern "C" int s256_ecdsa_verify(s256_ctx *ctx, const uint8_t *pk, const uint8_t *dg, const uint8_t *sig,
                                 uint32_t flags, size_t n, uint8_t *ok) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && (!pk || !dg || !sig || !ok)) return S256_ERR_ARG;
    if (ctx->pipe_parts == 1 && n >= ((size_t)1 << 18)) {
        int rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
            if (c < ((size_t)1 << 16)) {  // a short tail chunk: plain path
                view v = view_at(ctx, 0);
                cudaStream_t s = ctx->stream;
                CK(cudaMemcpyAsync(v.in_b, dg + 32 * off, 32 * c, cudaMemcpyHostToDevice, s));
                CK(cudaMemcpyAsync(v.in_c, sig + 64 * off, 64 * c, cudaMemcpyHostToDevice, s));
                CK(cudaMemcpyAsync(v.in_a, pk + 65 * off, 65 * c, cudaMemcpyHostToDevice, s));
                int r = chunk_ecdsa_verify(ctx, v, v.in_a, v.in_b, v.in_c, flags, c, v.st, s);
                if (r != S256_SUCCESS) return r;
                CK(cudaMemcpyAsync(ok + off, v.st, c, cudaMemcpyDeviceToHost, s));
                CK(cudaStreamSynchronize(s));
                return S256_SUCCESS;
            }
            return verify_pipelined(ctx, pk, dg, sig, flags, off, c, ok);
        });
        return rc != S256_SUCCESS ? rc : check_launch(ctx);
    }
    int rc = pipelined(ctx, n, [&](const view &v, size_t off, size_t c, cudaStream_t s) {
        // digest + signature first: the batched inversion starts while the keys are still in flight
        cudaStream_t s2 = (s == ctx->stream) ? ctx->stream2 : ctx->stream;
        CK(cudaMemcpyAsync(v.in_b, dg + 32 * off, 32 * c, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(v.in_c, sig + 64 * off, 64 * c, cudaMemcpyHostToDevice, s));
        bool split = ctx->pipe_parts == 1;
        CK(cudaMemcpyAsync(v.in_a, pk + 65 * off, 65 * c, cudaMemcpyHostToDevice, split ? s2 : s));
        int r = chunk_ecdsa_verify(ctx, v, v.in_a, v.in_b, v.in_c, flags, c, v.st, s, split ? s2 : s);
        if (r != S256_SUCCESS) return r;
        CK(cudaMemcpyAsync(ok + off, v.st, c, cudaMemcpyDeviceToHost, s));
        return S256_SUCCESS;
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}

extern "C" int s256_ecdsa_recover_dev(s256_ctx *ctx, const uint8_t *dg, const uint8_t *sig65, size_t n, uint8_t *pk65,
                                      uint8_t *status, void *stream) {
    ENTER(ctx);
    if (n && (!dg || !sig65 || !pk65 || !status)) return S256_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    int rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        return chunk_ecdsa_recover(ctx, view_at(ctx, 0), dg + 32 * off, sig65 + 65 * off, c, pk65 + 65 * off, status + off, s);
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}
extern "C" int s256_ecdsa_recover(s256_ctx *ctx, const uint8_t *dg, const uint8_t *sig65, size_t n, uint8_t *pk65,
                                  uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && (!dg || !sig65 || !pk65 || !status)) return S256_ERR_ARG;
    int rc = pipelined(ctx, n, [&](const view &v, size_t off, size_t c, cudaStream_t s) {
        CK(cudaMemcpyAsync(v.in_b, dg + 32 * off, 32 * c, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(v.in_c, sig65 + 65 * off, 65 * c, cudaMemcpyHostToDevice, s));
        int r = chunk_ecdsa_recover(ctx, v, v.in_b, v.in_c, c, v.out, v.st, s);
        if (r != S256_SUCCESS) return r;
        CK(cudaMemcpyAsync(pk65 + 65 * off, v.out, 65 * c, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(status + off, v.st, c, cudaMemcpyDeviceToHost, s));
        return S256_SUCCESS;
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}

extern "C" int s256_schnorr_verify_dev(s256_ctx *ctx, const uint8_t *pkx, const uint8_t *msg, size_t msg_len,
                                       const uint8_t *sig, size_t n, uint8_t *ok, void *stream) {
    ENTER(ctx);
    if (n && (!pkx || (!msg && msg_len) || !sig || !ok)) return S256_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    int rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        return chunk_schnorr_verify(ctx, view_at(ctx, 0), pkx + 32 * off, msg + msg_len * off, msg_len, sig + 64 * off, c, ok + off, s);
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}
extern "C" int s256_schnorr_verify(s256_ctx *ctx, const uint8_t *pkx, const uint8_t *msg, size_t msg_len,
                                   const uint8_t *sig, size_t n, uint8_t *ok) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && (!pkx || (!msg && msg_len) || !sig || !ok)) return S256_ERR_ARG;
    size_t need = (msg_len ? msg_len : 1) * (n < ctx->cap ? n : ctx->cap);
    if (int grc = grow_in_b(ctx, need)) return grc;
    int rc = pipelined(ctx, n, [&](const view &v, size_t off, size_t c, cudaStream_t ps) {
        uint8_t *dmsg = ctx->in_b + msg_len * (size_t)(v.st - ctx->st);  // messages are msg_len apart, not 32
        CK(cudaMemcpyAsync(v.in_a, pkx + 32 * off, 32 * c, cudaMemcpyHostToDevice, ps));
        if (msg_len) CK(cudaMemcpyAsync(dmsg, msg + msg_len * off, msg_len * c, cudaMemcpyHostToDevice, ps));
        CK(cudaMemcpyAsync(v.in_c, sig + 64 * off, 64 * c, cudaMemcpyHostToDevice, ps));
        int r = chunk_schnorr_verify(ctx, v, v.in_a, dmsg, msg_len, v.in_c, c, v.st, ps);
        if (r != S256_SUCCESS) return r;
        CK(cudaMemcpyAsync(ok + off, v.st, c, cudaMemcpyDeviceToHost, ps));
        return S256_SUCCESS;
    }, /*small_output=*/true);
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}

extern "C" int s256_double_scalar_mult_basepoint_vartime_dev(s256_ctx *ctx, const uint8_t *u1, const uint8_t *u2,
                                                             const uint8_t *pt65, size_t n, uint8_t *out65,
                                                             uint8_t *status, void *stream) {
    ENTER(ctx);
    if (n && (!u1 || !u2 || !pt65 || !out65 || !status)) return S256_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    int rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        return chunk_dsm(ctx, view_at(ctx, 0), u1 + 32 * off, u2 + 32 * off, pt65 + 65 * off, c, out65 + 65 * off, status + off, s);
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}
extern "C" int s256_double_scalar_mult_basepoint_vartime(s256_ctx *ctx, const uint8_t *u1, const uint8_t *u2,
                                                         const uint8_t *pt65, size_t n, uint8_t *out65,
                                                         uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && (!u1 || !u2 || !pt65 || !out65 || !status)) return S256_ERR_ARG;
    int rc = pipelined(ctx, n, [&](const view &v, size_t off, size_t c, cudaStream_t s) {
        CK(cudaMemcpyAsync(v.in_a, pt65 + 65 * off, 65 * c, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(v.in_b, u1 + 32 * off, 32 * c, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(v.in_c, u2 + 32 * off, 32 * c, cudaMemcpyHostToDevice, s));
        int r = chunk_dsm(ctx, v, v.in_b, v.in_c, v.in_a, c, v.out, v.st, s);
        if (r != S256_SUCCESS) return r;
        CK(cudaMemcpyAsync(out65 + 65 * off, v.out, 65 * c, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(status + off, v.st, c, cudaMemcpyDeviceToHost, s));
        return S256_SUCCESS;
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}

extern "C" int s256_scalar_base_mult_dev(s256_ctx *ctx, const uint8_t *k32, size_t n, uint8_t *out65, uint8_t *status,
                                         void *stream) {
    ENTER(ctx);
    if (n && (!k32 || !out65 || !status)) return S256_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    int rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        return chunk_base_mult(ctx, view_at(ctx, 0), k32 + 32 * off, c, out65 + 65 * off, status + off, s);
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}
extern "C" int s256_scalar_base_mult(s256_ctx *ctx, const uint8_t *k32, size_t n, uint8_t *out65, uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && (!k32 || !out65 || !status)) return S256_ERR_ARG;
    int rc = pipelined(ctx, n, [&](const view &v, size_t off, size_t c, cudaStream_t s) {
        CK(cudaMemcpyAsync(v.in_b, k32 + 32 * off, 32 * c, cudaMemcpyHostToDevice, s));
        int r = chunk_base_mult(ctx, v, v.in_b, c, v.out, v.st, s);
        if (r != S256_SUCCESS) return r;
        CK(cudaMemcpyAsync(out65 + 65 * off, v.out, 65 * c, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(status + off, v.st, c, cudaMemcpyDeviceToHost, s));
        return S256_SUCCESS;
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}

static int scalar_mult_common_dev(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, int mode,
                                  uint8_t *out, uint8_t *status, void *stream) {
    ENTER(ctx);
    if (n && (!k32 || !pt65 || !out || !status)) return S256_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    size_t w = mode == 1 ? 32 : 65;
    int rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        int r = chunk_scalar_mult(ctx, view_at(ctx, 0), k32 + 32 * off, pt65 + 65 * off, c, mode, out + w * off, status + off, s);
        if (r == S256_SUCCESS) CK(cudaMemsetAsync(ctx->res, 0, sizeof(pt) * c, s));  // k*P in projective form
        return r;
    });
    if (rc != S256_SUCCESS) wipe_secret_scratch(ctx);
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}
static int scalar_mult_common_host(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, int mode,
                                   uint8_t *out, uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && (!k32 || !pt65 || !out || !status)) return S256_ERR_ARG;
    size_t w = mode == 1 ? 32 : 65;
    int rc = pipelined(ctx, n, [&](const view &v, size_t off, size_t c, cudaStream_t s) {
        CK(cudaMemcpyAsync(v.in_a, pt65 + 65 * off, 65 * c, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(v.in_b, k32 + 32 * off, 32 * c, cudaMemcpyHostToDevice, s));
        int r = chunk_scalar_mult(ctx, v, v.in_b, v.in_a, c, mode, v.out, v.st, s);
        if (r != S256_SUCCESS) return r;
        CK(cudaMemcpyAsync(out + w * off, v.out, w * c, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(status + off, v.st, c, cudaMemcpyDeviceToHost, s));
        // the staged private scalars, k*P in projective form and the shared x do not outlive the call
        CK(cudaMemsetAsync(v.in_b, 0, 32 * c, s));
        CK(cudaMemsetAsync(v.res, 0, sizeof(pt) * c, s));
        CK(cudaMemsetAsync(v.out, 0, w * c, s));
        return S256_SUCCESS;
    });
    if (rc != S256_SUCCESS) wipe_secret_scratch(ctx);
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}
extern "C" int s256_scalar_mult(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, uint8_t *out65,
                                uint8_t *status) {
    return scalar_mult_common_host(ctx, k32, pt65, n, 0, out65, status);
}
extern "C" int s256_scalar_mult_dev(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, uint8_t *out65,
                                    uint8_t *status, void *stream) {
    return scalar_mult_common_dev(ctx, k32, pt65, n, 0, out65, status, stream);
}
extern "C" int s256_ecdh(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, uint8_t *x32,
                         uint8_t *status) {
    return scalar_mult_common_host(ctx, k32, pt65, n, 1, x32, status);
}
extern "C" int s256_ecdh_dev(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, uint8_t *x32,
                             uint8_t *status, void *stream) {
    return scalar_mult_common_dev(ctx, k32, pt65, n, 1, x32, status, stream);
}
// NewPointFromBytes on compressed encodings (point_s11n.go:140): 33 B -> 65 B + status
extern "C" int s256_point_decompress(s256_ctx *ctx, const uint8_t *pt33, size_t n, uint8_t *out65, uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && (!pt33 || !out65 || !status)) return S256_ERR_ARG;
    cudaStream_t s = ctx->stream;
    int rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        CK(cudaMemcpyAsync(ctx->in_a, pt33 + 33 * off, 33 * c, cudaMemcpyHostToDevice, s));
        LAUNCH(ctx, k_decode_compressed, grid_for(c), 0, s, ctx->in_a, c, ctx->aff, ctx->pvalid);
        LAUNCH(ctx, k_encode_affine, grid_for(c), 0, s, ctx->aff, ctx->pvalid, c, ctx->out, ctx->st);
        CK(cudaMemcpyAsync(out65 + 65 * off, ctx->out, 65 * c, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(status + off, ctx->st, c, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        return S256_SUCCESS;
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}
extern "C" int s256_point_compress(s256_ctx *ctx, const uint8_t *pt65, size_t n, uint8_t *out33, uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && (!pt65 || !out33 || !status)) return S256_ERR_ARG;
    cudaStream_t s = ctx->stream;
    int rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        CK(cudaMemcpyAsync(ctx->in_a, pt65 + 65 * off, 65 * c, cudaMemcpyHostToDevice, s));
        LAUNCH(ctx, k_decode_uncompressed, grid_for(c), 0, s, ctx->in_a, c, ctx->aff, ctx->pvalid);
        LAUNCH(ctx, k_encode_compressed, grid_for(c), 0, s, ctx->aff, ctx->pvalid, c, ctx->out, ctx->st);
        CK(cudaMemcpyAsync(out33 + 33 * off, ctx->out, 33 * c, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(status + off, ctx->st, c, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        return S256_SUCCESS;
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}
// secec.NewPublicKey over mixed SEC 1 encodings -> the uncompressed bytes PublicKey caches (secec/secec.go:84)
extern "C" int s256_new_public_keys(s256_ctx *ctx, const uint8_t *enc65, const uint8_t *enc_len, size_t n, uint8_t *out65,
                                    uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && (!enc65 || !enc_len || !out65 || !status)) return S256_ERR_ARG;
    cudaStream_t s = ctx->stream;
    int rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        CK(cudaMemcpyAsync(ctx->in_a, enc65 + 65 * off, 65 * c, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(ctx->in_b, enc_len + off, c, cudaMemcpyHostToDevice, s));
        LAUNCH(ctx, k_decode_sec1, grid_for(c), 0, s, ctx->in_a, ctx->in_b, c, ctx->aff, ctx->pvalid);
        LAUNCH(ctx, k_encode_public_key, grid_for(c), 0, s, ctx->aff, ctx->pvalid, c, ctx->out, ctx->st);
        CK(cudaMemcpyAsync(out65 + 65 * off, ctx->out, 65 * c, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(status + off, ctx->st, c, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        return S256_SUCCESS;
    });
    return rc != S256_SUCCESS ? rc : check_launch(ctx);
}
// secec.ParseASN1PublicKey (secec/s11n.go:38-76): SubjectPublicKeyInfo on the host (codecs.cpp), NewPublicKey
// on the device.  status: the parser's code, else the decoder's.
extern "C" int s256_parse_asn1_public_keys_checked(s256_ctx *ctx, const uint8_t *der, const size_t *offsets, size_t n,
                                                   uint8_t *out65, uint8_t *status) {
    if (!ctx || (n && (!der || !offsets || !out65 || !status))) return S256_ERR_ARG;
    if (n == 0) return S256_SUCCESS;
    try {  // no exception may cross the C ABI (and cgo): a failed host allocation is an error code
        std::vector<uint8_t> enc(65 * n), len(n), pst(n);
        int rc = s256_parse_asn1_public_keys(der, offsets, n, enc.data(), len.data(), pst.data());
        if (rc != S256_SUCCESS) return rc;
        rc = s256_new_public_keys(ctx, enc.data(), len.data(), n, out65, status);
        if (rc != S256_SUCCESS) return rc;
        for (size_t i = 0; i < n; i++)
            if (pst[i] != S256_ST_OK) {
                status[i] = pst[i];
                memset(out65 + 65 * i, 0, 65);
            }
        return S256_SUCCESS;
    } catch (const std::bad_alloc &) {
        return S256_ERR_NOMEM;
    }
}

// PublicKey.Verify with EncodingASN1 (secec/ecdsa.go:171-228): parse on the host (codecs.cpp), then the
// same batch as the compact path; rows the parser rejects come back false.
extern "C" int s256_ecdsa_verify_asn1(s256_ctx *ctx, const uint8_t *pk65, const uint8_t *digest32, const uint8_t *der,
                                      const size_t *offsets, uint32_t flags, size_t n, uint8_t *ok) {
    if (!ctx || (n && (!pk65 || !digest32 || !der || !offsets || !ok))) return S256_ERR_ARG;
    if (n == 0) return S256_SUCCESS;
    try {
        std::vector<uint8_t> sig(64 * n), parsed(n);
        int rc = s256_parse_asn1_signatures(der, offsets, n, sig.data(), parsed.data());
        if (rc != S256_SUCCESS) return rc;
        rc = s256_ecdsa_verify(ctx, pk65, digest32, sig.data(), flags, n, ok);
        if (rc != S256_SUCCESS) return rc;
        for (size_t i = 0; i < n; i++) ok[i] &= parsed[i];
        return S256_SUCCESS;
    } catch (const std::bad_alloc &) {
        return S256_ERR_NOMEM;
    }
}
// bitcoin.VerifyASN1 (secec/bitcoin/ecdsa_shitcoin.go:29-35)
extern "C" int s256_bitcoin_verify_asn1(s256_ctx *ctx, const uint8_t *pk65, const uint8_t *digest32, const uint8_t *der,
                                        const size_t *offsets, size_t n, uint8_t *ok) {
    if (!ctx || (n && (!pk65 || !digest32 || !der || !offsets || !ok))) return S256_ERR_ARG;
    if (n == 0) return S256_SUCCESS;  // (offsets may be NULL then)
    try {
        std::vector<uint8_t> bip(n);
        int rc = s256_is_valid_signature_encoding_bip0066(der, offsets, n, bip.data());
        if (rc != S256_SUCCESS) return rc;
        // strip the sighash byte of the rows that passed; rejected rows become empty (and fail to parse)
        std::vector<size_t> off2(n + 1);
        std::vector<uint8_t> der2;
        der2.reserve(offsets[n] - offsets[0]);
        for (size_t i = 0; i < n; i++) {
            off2[i] = der2.size();
            if (bip[i]) der2.insert(der2.end(), der + offsets[i], der + offsets[i + 1] - 1);
        }
        off2[n] = der2.size();
        if (der2.empty()) der2.push_back(0);
        rc = s256_ecdsa_verify_asn1(ctx, pk65, digest32, der2.data(), off2.data(), S256_FLAG_REJECT_MALLEABLE, n, ok);
        if (rc != S256_SUCCESS) return rc;
        for (size_t i = 0; i < n; i++) ok[i] &= bip[i];
        return S256_SUCCESS;
    } catch (const std::bad_alloc &) {
        return S256_ERR_NOMEM;
    }
}

// ---------------------------------------------------------------------------
// debug / measurement
// ---------------------------------------------------------------------------
extern "C" int s256_debug_gen_table(s256_ctx *ctx, int wbits, int nwin, uint8_t *out) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (!out || wbits < 1 || wbits > 16 || nwin < 1 || wbits * nwin > 256) return S256_ERR_ARG;
    size_t total = (size_t)nwin << wbits;
    apt *d = nullptr;
    CK(cudaMalloc(&d, total * sizeof(apt)));
    LAUNCH(ctx, k_gen_table, grid_for(total), 0, ctx->stream, d, wbits, total);
    apt *h = (apt *)malloc(total * sizeof(apt));
    cudaError_t e = cudaMemcpyAsync(h, d, total * sizeof(apt), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d);
    if (e != cudaSuccess) {
        free(h);
        ctx->last_err = cudaGetErrorString(e);
        return S256_ERR_CUDA;
    }
    // byte serialisation only (BE X || Y per entry, d = 0 skipped)
    for (int w = 0; w < nwin; w++)
        for (size_t dgt = 1; dgt < ((size_t)1 << wbits); dgt++) {
            const apt &a = h[((size_t)w << wbits) + dgt];
            fe_to_be32(out, a.x);
            fe_to_be32(out + 32, a.y);
            out += 64;
        }
    free(h);
    return S256_SUCCESS;
}

extern "C" int s256_debug_field_op(s256_ctx *ctx, int op, const uint8_t *a32, const uint8_t *b32, size_t n,
                                   uint8_t *out32) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n && (!a32 || !b32 || !out32)) return S256_ERR_ARG;
    if (n > ctx->cap) return S256_ERR_ARG;
    cudaStream_t s = ctx->stream;
    CK(cudaMemcpyAsync(ctx->in_a, a32, 32 * n, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(ctx->in_c, b32, 32 * n, cudaMemcpyHostToDevice, s));
    LAUNCH(ctx, k_field_op, grid_for(n), 0, s, op, ctx->in_a, ctx->in_c, n, ctx->out);
    CK(cudaMemcpyAsync(out32, ctx->out, 32 * n, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return check_launch(ctx);
}

// Per-kernel timing of k_dsm with CUDA events on the launching stream: enable, run
// steps, then read (synchronises on the recorded events and clears them).
extern "C" int s256_profile_enable(s256_ctx *ctx, int enable) {
    ENTER(ctx);
    for (auto &pr : ctx->dsm_events) {
        cudaEventDestroy(pr.first);
        cudaEventDestroy(pr.second);
    }
    ctx->dsm_events.clear();
    ctx->profiling = enable != 0;
    return S256_SUCCESS;
}
extern "C" int s256_profile_read(s256_ctx *ctx, double *dsm_ms_total, uint64_t *dsm_launches) {
    ENTER(ctx);
    double total = 0;
    uint64_t cnt = 0;
    for (auto &pr : ctx->dsm_events) {
        CK(cudaEventSynchronize(pr.second));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, pr.first, pr.second));
        total += ms;
        cnt++;
        cudaEventDestroy(pr.first);
        cudaEventDestroy(pr.second);
    }
    ctx->dsm_events.clear();
    if (dsm_ms_total) *dsm_ms_total = total;
    if (dsm_launches) *dsm_launches = cnt;
    return S256_SUCCESS;
}

// Integer-pipe probes (microbench.cuh): operations per second for one variant.
template <int V>
static void launch_probe(int blocks, int iters, cudaStream_t s, unsigned long long *sink) {
    k_int_probe<V><<<blocks, 256, 0, s>>>(12345u, iters, sink);
}
extern "C" int s256_microbench_variant(s256_ctx *ctx, int variant, int iters, double *ops_per_s, double *ms_out) {
    ENTER(ctx);
    if (iters < 1 || variant < 0 || variant >= MB_NVARIANTS) return S256_ERR_ARG;
    typedef void (*fn_t)(int, int, cudaStream_t, unsigned long long *);
    static const fn_t fns[MB_NVARIANTS] = {launch_probe<0>, launch_probe<1>, launch_probe<2>, launch_probe<3>,
                                           launch_probe<4>, launch_probe<5>, launch_probe<6>, launch_probe<7>,
                                           launch_probe<8>, launch_probe<9>, launch_probe<10>};
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    const int blocks = 148 * 8;
    fns[variant](blocks, 16, ctx->stream, ctx->sink);
    CK(cudaEventRecord(e0, ctx->stream));
    fns[variant](blocks, iters, ctx->stream, ctx->sink);
    CK(cudaEventRecord(e1, ctx->stream));
    ctx->launches.fetch_add(2);
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (ops_per_s) *ops_per_s = (double)blocks * 256 * (double)iters * mb_ops_per_trip(variant) / (ms * 1e-3);
    if (ms_out) *ms_out = ms;
    return check_launch(ctx);
}

extern "C" int s256_microbench_imad(s256_ctx *ctx, int iters, double *mac32_per_s, double *ms) {
    // the carry-chained form is the one the field multiplier issues, and the fastest MAC32 form measured
    return s256_microbench_variant(ctx, MB_MADC_CHAIN, iters, mac32_per_s, ms);
}

// Field-multiplication probes (DESIGN.md section 10): dependent products in two interleaved chains, the
// instruction-level parallelism a point formula offers.  form 0: fe_mul as the ladders call it (8x32 limbs,
// IMAD.WIDE carry chains, out of line); 1: the same inlined.  (Form 2 was the 5x52-limb FP64-pipe experiment of round 1:
// parity with the integer multiplier, not adopted, removed in round 2 -- DESIGN.md section 5.)
template <int FORM>
__global__ void __launch_bounds__(128, 4) k_femul_probe(uint32_t seed, int iters, unsigned long long *sink) {
    uint32_t a = seed ^ (threadIdx.x * 2654435761u), b = seed + blockIdx.x * 40503u + 1u;
    unsigned long long acc = 0;
    {
        fe x1, y1, x2, y2;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            x1.v[k] = a + 7u * k;
            y1.v[k] = b + 11u * k;
            x2.v[k] = a ^ (0x9e3779b9u * (k + 1));
            y2.v[k] = b ^ (0x85ebca6bu * (k + 1));
        }
#pragma unroll 1
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int k = 0; k < 2; k++) {
                if (FORM == 0) {
                    fe_mul(x1, x1, y1);
                    fe_mul(x2, x2, y2);
                    fe_mul(y1, y1, x2);
                    fe_mul(y2, y2, x1);
                } else {
                    fe_mul_inline(x1, x1, y1);
                    fe_mul_inline(x2, x2, y2);
                    fe_mul_inline(y1, y1, x2);
                    fe_mul_inline(y2, y2, x1);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 8; k++) acc ^= (unsigned long long)(x1.v[k] ^ y1.v[k]) << 32 | (x2.v[k] ^ y2.v[k]);
    }
    if (acc == 0x123456789abcdefull) sink[0] = acc;
}
template <int FORM>
static void launch_femul_probe(int blocks, int iters, cudaStream_t s, unsigned long long *sink) {
    k_femul_probe<FORM><<<blocks, 128, 0, s>>>(12345u, iters, sink);
}
extern "C" int s256_microbench_fe_mul(s256_ctx *ctx, int form, int iters, double *muls_per_s, double *ms_out) {
    ENTER(ctx);
    if (iters < 1 || form < 0 || form > 1) return S256_ERR_ARG;
    typedef void (*fn_t)(int, int, cudaStream_t, unsigned long long *);
    static const fn_t fns[2] = {launch_femul_probe<0>, launch_femul_probe<1>};
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    const int blocks = 148 * 16;
    fns[form](blocks, 4, ctx->stream, ctx->sink);
    CK(cudaEventRecord(e0, ctx->stream));
    fns[form](blocks, iters, ctx->stream, ctx->sink);
    CK(cudaEventRecord(e1, ctx->stream));
    ctx->launches.fetch_add(2);
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (muls_per_s) *muls_per_s = (double)blocks * 128 * (double)iters * 8.0 / (ms * 1e-3);
    if (ms_out) *ms_out = ms;
    return check_launch(ctx);
}

// Measured, not modelled: the number of ladder additions the last verification-type call on this context really
// executed (non-zero digits of its two recoded halves), for the first `n` items of its last chunk.  bench.py turns it
// into the executed MAC32 of that k_dsm launch: additions with a zero digit are skipped, and the lambda half costs one
// more multiplication (x -> beta x) per executed addition.
__global__ void __launch_bounds__(S256_TPB) k_count_nonzero_digits(const int8_t *d1, const int8_t *d2, size_t total1,
                                                                  size_t total2, unsigned long long *out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
    unsigned a = 0, b = 0;
    for (; i < total2; i += stride) {
        a += (i < total1) && d1[i] != 0;   // digits are stored [digit][item]: the top digit of the first half is the
        b += d2[i] != 0;                   // assignment that starts the ladder, not an addition
    }
    a = __reduce_add_sync(0xffffffffu, a);
    b = __reduce_add_sync(0xffffffffu, b);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(out, (unsigned long long)a);
        atomicAdd(out + 1, (unsigned long long)b);
    }
}
extern "C" int s256_debug_ladder_add_count(s256_ctx *ctx, size_t n, uint64_t *adds_g_half, uint64_t *adds_lambda_half) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (!adds_g_half || !adds_lambda_half || n > ctx->cap) return S256_ERR_ARG;
    cudaStream_t s = ctx->stream;
    CK(cudaMemsetAsync(ctx->sink, 0, 16, s));
    if (n) LAUNCH(ctx, k_count_nonzero_digits, 148 * 8, 0, s, ctx->dig1, ctx->dig2, (size_t)(DSM_ND - 1) * n, (size_t)DSM_ND * n, ctx->sink);
    unsigned long long h[2] = {0, 0};
    CK(cudaMemcpyAsync(h, ctx->sink, 16, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    *adds_g_half = h[0];
    *adds_lambda_half = h[1];
    return check_launch(ctx);
}
// executed MAC32 of one k_dsm item given its measured number of ladder additions (both halves) and beta multiplications
// The Jacobian ladder (jac.cuh): doubling 2 M + 5 S (or 3 M + 4 S), mixed addition 6 M + 3 S + one fused pair, the table's
// co-Z chain and its scaling to a common denominator (kernels.cuh) and the conversion of the result.
struct dsm_costs {
    double dbl, add, mix, table, tail;
};
static dsm_costs dsm_cost_model() {
    const double M = 73, S = 45;
#ifndef S256_NO_FUSED
    const double F2 = 137;  // a b + c d with one reduction: 128 + 8 + 1
#else
    const double F2 = 2 * M;
#endif
    dsm_costs c;
#if defined(S256_DSM_JAC)
#ifndef S256_JDBL_3M4S
    c.dbl = 2 * M + 5 * S;
#else
    c.dbl = 3 * M + 4 * S;
#endif
    c.mix = 6 * M + 3 * S + F2;
    c.add = c.mix;  // the ladder adds affine rows
    // co-Z chain (kernels.cuh): DBLU M + 5 S, TS - 2 ZADDU of 4 M + 2 S; the backward pass TS - 3 ratio products and
    // 3 M + S for each of the TS - 2 rows not yet at Z_all; Z_all = 2y r_2, and one product to come back from the
    // isomorphic curve -- no inversion
    c.table = (M + 5 * S) + (DSM_TS - 2) * (4 * M + 2 * S) + (DSM_TS - 3) * M + (DSM_TS - 2) * (3 * M + S) + 2 * M;
    c.tail = 2 * M + S;
#else
#ifndef S256_NO_FUSED
    c.dbl = 4 * M + 2 * S + F2, c.add = 6 * M + 3 * F2, c.mix = 5 * M + 3 * F2;
#else
    c.dbl = 6 * M + 2 * S, c.add = 12 * M, c.mix = 11 * M;
#endif
    c.table = (DSM_TS / 2) * c.dbl + (DSM_TS / 2 - 1) * c.mix;
    c.tail = 0;
#endif
    return c;
}
extern "C" double s256_mac32_k_dsm(double adds_per_item, double beta_muls_per_item) {
    const dsm_costs c = dsm_cost_model();
    // (the very first addition of the ladder is an assignment; bench.py subtracts it from the measured count)
    return c.table + (DSM_ND - 1) * DSM_W * c.dbl + adds_per_item * c.add + beta_muls_per_item * 73 + COMB_NW * c.mix + c.tail;
}

// MAC32 (32x32->64 multiply-accumulates, i.e. IMAD.WIDE issues) per item as EXECUTED (DESIGN.md section 5):
// F_p mul = 73 (64 + 8 + the fold's one), F_p square = 45 (28 + 8 + 8 + 1), Z_n modmul = 133.  Multiplication by
// b3 = 21 and by 8 are shifts and adds now (fe_vt.cuh): no multiplier work in the variable-time flavour, one
// product (the fold) in the constant-time one.  Ladder steps with a zero digit are skipped, so the model charges the
// EXPECTED number of executed additions for uniformly random scalars: a signed 5-bit digit is zero with probability
// 2^-5, the top digit of a 128-bit half (3 bits + carry) with probability 1/8.
extern "C" double s256_mac32_per_item(const char *name) {
    const double M = 73, S = 45, ZN = 133;
#ifndef S256_NO_FUSED
    const double F2 = 137;  // a b + c d with one reduction (variable-time flavour only)
    const double dbl = 4 * M + 2 * S + F2, add = 6 * M + 3 * F2, mix = 5 * M + 3 * F2;   // k_dsm, MSM
#else
    const double dbl = 6 * M + 2 * S, add = 12 * M, mix = 11 * M;
#endif
#if !defined(S256_NO_FUSED) && !defined(S256_NO_FUSED_CT)
    const double dbl_ct = 4 * M + 2 * S + F2 + 2, mix_ct = 5 * M + 3 * F2 + 2;    // fused pairs in the constant-time flavour too
    const double jmix_ct = 6 * M + 3 * S + F2;
#else
    const double dbl_ct = 6 * M + 2 * S + 2, mix_ct = 11 * M + 2;                 // + the folds of 21a and 8a / 21a twice
    const double jmix_ct = 8 * M + 3 * S;
#endif
    // inversions are safegcd (modinv.cuh): 20 batches x (54 + 36) 32x32->64 products, whatever the modulus
    const double inv_fe = 20 * 90, sqrt_fe = 254 * S + 13 * M + 2 * S + M, inv_sc = 20 * 90;
    const double oncurve = 2 * S + M;
    const dsm_costs dc = dsm_cost_model();
    const double adds_per_half = (DSM_ND - 1) * (1.0 - 1.0 / (1 << DSM_W)) + 15.0 / 16.0;
    // (the first addition of the first half is an assignment: the accumulator is still the identity)
    const double ladder = (DSM_ND - 1) * DSM_W * dc.dbl + (2 * adds_per_half - 15.0 / 16.0) * dc.add + adds_per_half * M;
    const double comb = COMB_NW * dc.mix;
    const double dsm = dc.table + ladder + comb + dc.tail;
    const double split = 3 * ZN + 2 * 64;
    const double affine = (3 + 2) * M + inv_fe / INV_K;
    std::string s(name ? name : "");
    if (s == "k_dsm") return dsm;  // the ladder kernel alone
    if (s == "ecdsa_verify") return oncurve + (5 * ZN + inv_sc / INV_K + split) + dsm + 2 * M;
    if (s == "ecdsa_recover") return sqrt_fe + (6 * ZN + inv_sc / INV_K + split) + dsm + affine;
    if (s == "schnorr_verify") return sqrt_fe + (ZN + split) + dsm + affine;
    if (s == "double_scalar_mult_basepoint_vartime") return oncurve + split + dsm + affine;
#ifndef S256_BM_RCB
    const double bm = ct_cfg<7>::NW * jmix_ct + 2 * M + S;  // large batches: 7-bit windows, Jacobian accumulator (kernels.cuh)
#else
    const double bm = ct_cfg<7>::NW * mix_ct;
#endif
    if (s == "scalar_base_mult") return bm + affine;
    if (s == "schnorr_sign") return 2 * (bm + affine) + 2 * ZN;  // + ~9 SHA-256 blocks
    if (s == "ecdsa_sign_rfc6979") return bm + affine + (5 * ZN + inv_sc / INV_K);  // + 22 SHA-256 blocks
    if (s == "scalar_mult" || s == "ecdh") {
        const double tab = (CTM_TS / 2) * dbl_ct + (CTM_TS / 2 - 1) * mix_ct + 5 * (CTM_TS - 1) * M + inv_fe;  // + normalisation
        const double lad = (CTM_ND - 1) * CTM_W * dbl_ct + 2 * CTM_ND * mix_ct + CTM_ND * M;
        return oncurve + split + tab + lad + affine;
    }
#ifndef S256_MSM_RCB
    if (s == "msm_mixed_add") return dc.mix;  // one bucket accumulation step of the Pippenger MSM (k_msm_slices): Jacobian mixed
#else
    if (s == "msm_mixed_add") return mix;
#endif
    return 0.0;
}
