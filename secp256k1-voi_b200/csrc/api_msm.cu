// api_msm.cu -- Point.MultiScalarMult[Vartime]: the Pippenger kernels (msm.cuh) and their entry points, and the
// BIP-340 batch verification built on them (batch.cuh).
#include "ctx.h"
#include "msm.cuh"
#include "batch.cuh"
#include "coop.cuh"
#include <cub/device/device_scan.cuh>
#include <dlfcn.h>
#include <functional>
#include <nccl.h>  // types only: the library is resolved at run time (no link-time dependency on NCCL)

// ---- Pippenger MSM (msm.cuh) -------------------------------------------------
// Pass 1, one thread per point: split the scalar with the endomorphism (once: the halves are kept for pass 2), write the
// two virtual points (x, y), (beta x, y), count the digits of both halves into their buckets.
__global__ void __launch_bounds__(S256_TPB) k_msm_prepare(const uint8_t *k32, const apt *aff, size_t n, msm_plan plan,
                                                          uint4 *half, uint8_t *hsign, apt *aff2, uint32_t *counts) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    sc k, m[2];
    sc_from_be32(k, k32 + 32 * i);
    uint32_t neg[2];
    msm_glv_halves(m[0], neg[0], m[1], neg[1], k);
    half[2 * i] = make_uint4(m[0].v[0], m[0].v[1], m[0].v[2], m[0].v[3]);
    half[2 * i + 1] = make_uint4(m[1].v[0], m[1].v[1], m[1].v[2], m[1].v[3]);
    hsign[i] = (uint8_t)(neg[0] | (neg[1] << 1));
    apt p = aff[i], p0, p1;
    msm_glv_points(p0, p1, p);
    aff2[2 * i] = p0;
    aff2[2 * i + 1] = p1;
    for (int h = 0; h < 2; h++) {
        int32_t d[MSM_MAX_WIN];
        msm_digits(d, m[h], plan);
        for (int w = 0; w < plan.nwin; w++)
            if (d[w] != 0) atomicAdd(&counts[(uint32_t)w * (uint32_t)plan.nb + ((uint32_t)(d[w] < 0 ? -d[w] : d[w]) - 1u)], 1u);
    }
}
// Pass 2: the same digits again, scattered into the bucket-sorted entry list as (virtual point << 1) | negate
__global__ void __launch_bounds__(S256_TPB) k_msm_scatter(size_t n, msm_plan plan, const uint4 *half, const uint8_t *hsign,
                                                          uint32_t *cursor, uint32_t *entries) {
    size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x;  // virtual point
    if (v >= 2 * n) return;
    uint4 q = half[v];
    sc m;
    m.v[0] = q.x; m.v[1] = q.y; m.v[2] = q.z; m.v[3] = q.w;
    m.v[4] = m.v[5] = m.v[6] = m.v[7] = 0u;
    uint32_t hneg = (hsign[v >> 1] >> (v & 1)) & 1u;
    int32_t d[MSM_MAX_WIN];
    msm_digits(d, m, plan);
    for (int w = 0; w < plan.nwin; w++) {
        int32_t dw = d[w];
        if (dw == 0) continue;
        uint32_t mag = (uint32_t)(dw < 0 ? -dw : dw);
        uint32_t pos = atomicAdd(&cursor[(uint32_t)w * (uint32_t)plan.nb + (mag - 1u)], 1u);
        entries[pos] = ((uint32_t)v << 1) | ((uint32_t)(dw < 0) ^ hneg);
    }
}
// nsl[b] = slices of bucket b (counts -> slice counts), then scanned into sl_off
__global__ void __launch_bounds__(S256_TPB) k_msm_slice_counts(uint32_t total, const uint32_t *counts, uint32_t *nsl, int slice) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < total) nsl[b] = msm_slices_of(counts[b], slice);
    if (b == total) nsl[b] = 0;
}
// Slice schedule: range[s] = entry range of slice s, hist[MSM_SLICE - len] = slices of that length.
#define S256_MSM_ST 256
constexpr int MSM_BINS = MSM_SLICE + 1;
__global__ void __launch_bounds__(S256_MSM_ST) k_msm_slice_ranges(uint32_t max_slices, uint32_t total, const uint32_t *sl_off,
                                                                  const uint32_t *offsets, uint2 *range, uint32_t *bucket_of,
                                                                  uint32_t *hist, int slice) {
    __shared__ uint32_t sh[MSM_BINS];
    for (int i = threadIdx.x; i < MSM_BINS; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < max_slices && s < sl_off[total]) {
        uint32_t st, en;
        bucket_of[s] = msm_slice_range(st, en, s, sl_off, offsets, total, slice);
        range[s] = make_uint2(st, en);
        atomicAdd(&sh[MSM_SLICE - (en - st)], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < MSM_BINS; i += blockDim.x)
        if (sh[i]) atomicAdd(&hist[i], sh[i]);
}
// perm = slice ids ordered by decreasing length (order inside a length class is arbitrary)
__global__ void __launch_bounds__(S256_MSM_ST) k_msm_slice_perm(uint32_t max_slices, uint32_t total, const uint32_t *sl_off,
                                                                const uint2 *range, const uint32_t *hist, uint32_t *cursor,
                                                                uint32_t *perm) {
    __shared__ uint32_t cnt[MSM_BINS], base[MSM_BINS];
    for (int i = threadIdx.x; i < MSM_BINS; i += blockDim.x) cnt[i] = 0;
    __syncthreads();
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    bool live = s < max_slices && s < sl_off[total];
    uint32_t bin = 0, rank = 0;
    if (live) {
        uint2 r = range[s];
        bin = MSM_SLICE - (r.y - r.x);
        rank = atomicAdd(&cnt[bin], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < MSM_BINS; i += blockDim.x) {
        uint32_t c = cnt[i], before = 0;
        if (c) {
            for (int k = 0; k < i; k++) before += hist[k];
            base[i] = before + atomicAdd(&cursor[i], c);
        }
    }
    __syncthreads();
    if (live) perm[base[bin] + rank] = s;
}
#ifndef S256_MSM_SLICES_MINB
#define S256_MSM_SLICES_MINB 4   // 128 registers: four CTAs per SM instead of the three that 130 registers allowed
#endif
__global__ void __launch_bounds__(S256_TPB, S256_MSM_SLICES_MINB) k_msm_slices(uint32_t max_slices, uint32_t total, const uint32_t *sl_off,
                                                         const uint32_t *perm, const uint2 *range, const uint32_t *entries,
                                                         const apt *aff, pt *slice_sum) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= max_slices || t >= sl_off[total]) return;
    uint32_t s = perm[t];
    uint2 r = range[s];
    pt acc;
    msm_bucket_sum(acc, entries, r.x, r.y, aff);
    slice_sum[s] = acc;
}
// second level for buckets of more than MSM_SUPER slices (msm.cuh); a no-op thread otherwise
__global__ void __launch_bounds__(S256_TPB) k_msm_superslices(uint32_t max_slices, uint32_t total, const uint32_t *sl_off,
                                                              const uint32_t *bucket_of, pt *slice_sum) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= max_slices || s >= sl_off[total]) return;
    uint32_t b = bucket_of[s];
    msm_superslice_fold(slice_sum, s, sl_off[b], sl_off[b + 1]);
}

// bucket b = the sum of its slice sums, one thread per bucket, written densely (bsum[b]) together with the identity
// slice map the window stage then reads it through: with short slices a bucket has several slice sums, and folding
// them inside the window stage would put those additions on its serial chains (measured: k_msm_windows 0.20 -> 0.50 ms
// at n = 2^17 with 16-entry slices).
__global__ void __launch_bounds__(S256_TPB) k_msm_fold_buckets(uint32_t total, const pt *slice_sum, const uint32_t *sl_off,
                                                               pt *bsum, uint32_t *ident) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b <= total) ident[b] = b;
    if (b >= total) return;
    pt acc;
    msm_bucket_from_slices(acc, slice_sum, sl_off, b);
    bsum[b] = acc;
}

// One CTA of MSM_WT threads, thread t holding (run_t, sum_t) with sum_t weighted relative to its own
// first element: returns (in thread 0)  R = sum_t run_t  and  A = sum_t (sum_t + t * 2^lg * run_t).
// sum_t t * run_t is the sum over t >= 1 of the suffix sums S_t = sum_{u >= t} run_u.
__device__ __forceinline__ void msm_cta_weighted(pt &R, pt &A, const pt &run, const pt &sum, int lg, pt *sh) {
    int t = threadIdx.x;
    sh[t] = run;
    __syncthreads();
    for (int d = 1; d < MSM_WT; d <<= 1) {
        pt v = sh[t];
        if (t + d < MSM_WT) {
            pt o = sh[t + d];
            pt_add<true>(v, v, o);
        }
        __syncthreads();
        sh[t] = v;
        __syncthreads();
    }
    R = sh[0];
    pt v = sum;
    if (t >= 1) {
        pt st = sh[t];
        msm_weigh(v, sum, st, lg);
    }
    __syncthreads();
    sh[t] = v;
    __syncthreads();
    for (int stride = MSM_WT / 2; stride >= 1; stride >>= 1) {
        if (t < stride) {
            pt a = sh[t], b = sh[t + stride];
            pt_add<true>(a, a, b);
            sh[t] = a;
        }
        __syncthreads();
    }
    A = sh[0];
}
// level 1, grid (parts, nwin): part[(w * parts + blk) * 2 + {0, 1}] = (R, A) of the CTA's MSM_WT * seg buckets
__global__ void __launch_bounds__(MSM_WT) k_msm_windows(msm_plan plan, const pt *slice_sum, const uint32_t *sl_off, pt *part,
                                                        int parts) {
    __shared__ pt sh[MSM_WT];
    int w = blockIdx.y, t = threadIdx.x;
    int nbw = msm_window_buckets(plan, w);
    if ((int)blockIdx.x >= msm_parts_for(nbw)) return;
    int seg = msm_seg_for(nbw);
    int lo = (blockIdx.x * MSM_WT + t) * seg, hi = lo + seg;
    if (hi > nbw) hi = nbw;
    pt run, sum;
    if (lo < hi) {
        msm_segment_pair(run, sum, slice_sum, sl_off, (uint32_t)w * (uint32_t)plan.nb, lo, hi);
    } else {
        pt_set_identity(run);
        pt_set_identity(sum);
    }
    pt R, A;
    msm_cta_weighted(R, A, run, sum, msm_log2(seg), sh);
    if (t == 0) {
        part[((size_t)w * parts + blockIdx.x) * 2] = R;
        part[((size_t)w * parts + blockIdx.x) * 2 + 1] = A;
    }
}
// level 2, one CTA per window: win[w] = sum over the window's CTAs q of (A_q + q * MSM_WT * seg * R_q)
__global__ void __launch_bounds__(MSM_WT) k_msm_windows2(msm_plan plan, const pt *part, int parts, pt *win) {
    __shared__ pt sh[MSM_WT];
    int w = blockIdx.x, t = threadIdx.x;
    int nbw = msm_window_buckets(plan, w);
    pt run, sum;
    if (t < msm_parts_for(nbw)) {
        run = part[((size_t)w * parts + t) * 2];
        sum = part[((size_t)w * parts + t) * 2 + 1];
    } else {
        pt_set_identity(run);
        pt_set_identity(sum);
    }
    pt R, A;
    msm_cta_weighted(R, A, run, sum, msm_log2(MSM_WT * msm_seg_for(nbw)), sh);
    if (t == 0) win[w] = A;
}
// acc (device, projective) += Horner(windows); first = overwrite.  One warp, 8-lane cooperative group law.
__global__ void __launch_bounds__(32) k_msm_final(msm_plan plan, const pt *win, pt *acc, int first) {
    int j = threadIdx.x & 7;
    pt r;
    pt_set_identity(r);
    for (int w = plan.nwin - 1; w >= 0; w--) {
        if (w != plan.nwin - 1)
            for (int k = 0; k < plan.c; k++) pt_double_coop(r, j);
        pt t = win[w];
        pt_add_coop(r, t, j);
    }
    if (!first) {
        pt a = *acc;
        pt_add_coop(r, a, j);
    }
    __syncwarp();
    if (threadIdx.x == 0) *acc = r;
}
// out[t] = sum of in[t], in[t + nout], ...   (tree levels of the constant-time MSM)
__global__ void __launch_bounds__(S256_TPB) k_reduce_points(const pt *in, size_t n, pt *out, size_t nout) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nout) return;
    pt acc;
    pt_set_identity(acc);
    for (size_t i = t; i < n; i += nout) {
        pt q = in[i];
        pt_add(acc, acc, q);
    }
    out[t] = acc;
}
__global__ void k_acc_point(const pt *in, pt *acc, int first) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    pt r = *in;
    if (!first) {
        pt a = *acc;
        pt_add(r, r, a);
    }
    *acc = r;
}
__global__ void __launch_bounds__(S256_TPB) k_any_invalid(const uint8_t *pvalid, size_t n, uint32_t *flag) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && pvalid[i] == 0) atomicOr(flag, 1u);
}
// partial96 rows -> one projective sum; rows must be points on the curve (or the identity)
__global__ void k_combine_partials(const uint8_t *partials96, size_t m, pt *out, uint32_t *flag) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    pt acc;
    pt_set_identity(acc);
    for (size_t j = 0; j < m; j++) {
        pt q;
        pt_from_be96(q, partials96 + 96 * j);
        uint32_t ok = fe_limbs_are_canonical(q.x) & fe_limbs_are_canonical(q.y) & fe_limbs_are_canonical(q.z) &
                      pt_on_curve(q);
        if (!ok) {
            atomicOr(flag, 1u);
            continue;
        }
        pt_add(acc, acc, q);
    }
    *out = acc;
}
__global__ void k_export_partial(const pt *acc, uint8_t *out96) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    pt a = *acc;
    pt_to_be96(out96, a);
}


// ---------------------------------------------------------------------------
// MSM
// ---------------------------------------------------------------------------
static size_t msm_entries_capacity(const s256_ctx *ctx) {
    // nwin * 2n entries (two 128-bit halves per scalar): c = 4 gives 32 windows, i.e. 64 n; the planner is at
    // c >= 10 (26 n) once n >= 2^14 and chunk_msm widens the windows until the entries fit
    size_t cap = ctx->cap;
    size_t small = (size_t)MSM_MAX_WIN * (cap < 65536 ? cap : 65536), large = (size_t)26 * cap;
    return small > large ? small : large;
}
static int msm_ensure(s256_ctx *ctx) {
    if (ctx->msm_cap) return S256_SUCCESS;
    size_t total = 0;
    for (int c = 4; c <= MSM_MAX_C; c++) {
        size_t t = (size_t)msm_plan_for_c(c, 128).total;
        if (t > total) total = t;
    }
    CK(cudaMalloc(&ctx->msm_bsum, (total + 1) * sizeof(pt)));
    CK(cudaMalloc(&ctx->msm_aff2, 2 * ctx->cap * sizeof(apt)));
    CK(cudaMalloc(&ctx->msm_half, 2 * ctx->cap * sizeof(uint4)));
    CK(cudaMalloc(&ctx->msm_counts, (total + 1) * 4));
    CK(cudaMalloc(&ctx->msm_offsets, (total + 1) * 4));
    CK(cudaMalloc(&ctx->msm_cursor, (total + 1) * 4));
    CK(cudaMalloc(&ctx->msm_entries, msm_entries_capacity(ctx) * 4));
    // slice sums: one per bucket at least, plus one per MSM_SLICE entries
    ctx->msm_max_slices = total + msm_entries_capacity(ctx) / (MSM_SLICE / 4) + 1;  // the shortest slice length (msm.cuh)
    CK(cudaMalloc(&ctx->msm_buckets, ctx->msm_max_slices * sizeof(pt)));
    CK(cudaMalloc(&ctx->msm_nsl, (total + 1) * 4));
    CK(cudaMalloc(&ctx->msm_sloff, (total + 1) * 4));
    CK(cudaMalloc(&ctx->msm_range, ctx->msm_max_slices * sizeof(uint2)));
    CK(cudaMalloc(&ctx->msm_perm, ctx->msm_max_slices * 4));
    CK(cudaMalloc(&ctx->msm_sbkt, ctx->msm_max_slices * 4));
    CK(cudaMalloc(&ctx->msm_hist, 2 * MSM_BINS * 4));
    CK(cudaMalloc(&ctx->msm_part, (size_t)MSM_MAX_WIN * MSM_MAX_PARTS * 2 * sizeof(pt)));
    CK(cudaMalloc(&ctx->msm_win, (size_t)MSM_MAX_WIN * sizeof(pt)));
    CK(cudaMalloc(&ctx->msm_acc, sizeof(pt)));
    CK(cudaMalloc(&ctx->msm_tmp, 4096 * sizeof(pt)));
    CK(cudaMalloc(&ctx->msm_flag, 4));
    size_t bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, bytes, ctx->msm_counts, ctx->msm_offsets, (int)(total + 1));
    ctx->msm_cub_bytes = bytes;
    CK(cudaMalloc(&ctx->msm_cub, bytes));
    ctx->msm_cap = ctx->cap;
    return S256_SUCCESS;
}

// one chunk of points already in ctx->aff (device pointers): msm_acc (+)= sum k_i P_i
static int chunk_msm_body(s256_ctx *ctx, const uint8_t *k32, size_t n, int vartime, int first, cudaStream_t s) {
    if (!vartime || n < 32) {
        // constant-time flavour (and tiny inputs): ct ladder per item, then a sum tree
        s256_launch_scalar_mult_ct(n, ctx->aff, k32, ctx->tbl, ctx->res, s);
        ctx->launches.fetch_add(1, std::memory_order_relaxed);
        size_t m = n < 2048 ? (n < 32 ? 1 : 32) : 2048;
        LAUNCH(ctx, k_reduce_points, grid_for(m), 0, s, ctx->res, n, ctx->msm_tmp, m);
        if (m > 32) {
            LAUNCH(ctx, k_reduce_points, grid_for(32), 0, s, ctx->msm_tmp, m, ctx->msm_tmp + 2048, (size_t)32);
            LAUNCH(ctx, k_reduce_points, 1, 0, s, ctx->msm_tmp + 2048, (size_t)32, ctx->msm_tmp + 2048 + 32, (size_t)1);
            k_acc_point<<<1, 1, 0, s>>>(ctx->msm_tmp + 2048 + 32, ctx->msm_acc, first);
        } else if (m > 1) {
            LAUNCH(ctx, k_reduce_points, 1, 0, s, ctx->msm_tmp, m, ctx->msm_tmp + 2048, (size_t)1);
            k_acc_point<<<1, 1, 0, s>>>(ctx->msm_tmp + 2048, ctx->msm_acc, first);
        } else {
            k_acc_point<<<1, 1, 0, s>>>(ctx->msm_tmp, ctx->msm_acc, first);
        }
        ctx->launches.fetch_add(1, std::memory_order_relaxed);
        return S256_SUCCESS;
    }
    // endomorphism form: 2n virtual points with 128-bit scalars (msm.cuh)
    const size_t nv = 2 * n;
    msm_plan pl = msm_make_plan(nv, 128);
    while (pl.c < MSM_MAX_C && (size_t)pl.nwin * nv > msm_entries_capacity(ctx)) pl = msm_plan_for_c(pl.c + 1, 128);
    uint32_t total = (uint32_t)pl.total;
    CK(cudaMemsetAsync(ctx->msm_counts, 0, ((size_t)total + 1) * 4, s));
    LAUNCH(ctx, k_msm_prepare, grid_for(n), 0, s, k32, ctx->aff, n, pl, (uint4 *)ctx->msm_half, ctx->sfl, ctx->msm_aff2,
           ctx->msm_counts);
    size_t bytes = ctx->msm_cub_bytes;
    CK(cub::DeviceScan::ExclusiveSum(ctx->msm_cub, bytes, ctx->msm_counts, ctx->msm_offsets, (int)(total + 1), s));
    CK(cudaMemcpyAsync(ctx->msm_cursor, ctx->msm_offsets, (size_t)total * 4, cudaMemcpyDeviceToDevice, s));
    LAUNCH(ctx, k_msm_scatter, grid_for(nv), 0, s, n, pl, (const uint4 *)ctx->msm_half, ctx->sfl, ctx->msm_cursor,
           ctx->msm_entries);
    // buckets -> slices of <= MSM_SLICE entries
    LAUNCH(ctx, k_msm_slice_counts, grid_for((size_t)total + 1), 0, s, total, ctx->msm_counts, ctx->msm_nsl, pl.slice);
    CK(cub::DeviceScan::ExclusiveSum(ctx->msm_cub, bytes, ctx->msm_nsl, ctx->msm_sloff, (int)(total + 1), s));
    size_t max_slices = (size_t)total + ((size_t)pl.nwin * nv) / (size_t)pl.slice + 1;
    if (max_slices > ctx->msm_max_slices) max_slices = ctx->msm_max_slices;
    // hand the slices out longest first: every warp then runs (almost) equally long threads
    CK(cudaMemsetAsync(ctx->msm_hist, 0, 2 * MSM_BINS * 4, s));
    unsigned sgrid = (unsigned)((max_slices + S256_MSM_ST - 1) / S256_MSM_ST);
    k_msm_slice_ranges<<<sgrid, S256_MSM_ST, 0, s>>>((uint32_t)max_slices, total, ctx->msm_sloff, ctx->msm_offsets,
                                                     (uint2 *)ctx->msm_range, ctx->msm_sbkt, ctx->msm_hist, pl.slice);
    k_msm_slice_perm<<<sgrid, S256_MSM_ST, 0, s>>>((uint32_t)max_slices, total, ctx->msm_sloff, (const uint2 *)ctx->msm_range,
                                                   ctx->msm_hist, ctx->msm_hist + MSM_BINS, ctx->msm_perm);
    LAUNCH(ctx, k_msm_slices, grid_for(max_slices), 0, s, (uint32_t)max_slices, total, ctx->msm_sloff, ctx->msm_perm,
           (const uint2 *)ctx->msm_range, ctx->msm_entries, ctx->msm_aff2, ctx->msm_buckets);
    LAUNCH(ctx, k_msm_superslices, grid_for(max_slices), 0, s, (uint32_t)max_slices, total, ctx->msm_sloff, ctx->msm_sbkt,
           ctx->msm_buckets);
    int parts = msm_parts_for(pl.nb);
    if (msm_parts_for(pl.nb_top) > parts) parts = msm_parts_for(pl.nb_top);
    const pt *bucket_sums = ctx->msm_buckets;
    const uint32_t *bucket_map = ctx->msm_sloff;
    if (pl.slice < MSM_SLICE) {  // several slices per bucket: fold them first, all buckets in parallel
        LAUNCH(ctx, k_msm_fold_buckets, grid_for((size_t)total + 1), 0, s, total, ctx->msm_buckets, ctx->msm_sloff,
               ctx->msm_bsum, ctx->msm_nsl);  // msm_nsl (the per-bucket slice counts) is free again: reused as the map
        bucket_sums = ctx->msm_bsum;
        bucket_map = ctx->msm_nsl;
    }
    k_msm_windows<<<dim3(parts, pl.nwin), MSM_WT, 0, s>>>(pl, bucket_sums, bucket_map, ctx->msm_part, parts);
    k_msm_windows2<<<pl.nwin, MSM_WT, 0, s>>>(pl, ctx->msm_part, parts, ctx->msm_win);
    k_msm_final<<<1, 32, 0, s>>>(pl, ctx->msm_win, ctx->msm_acc, first);
    ctx->launches.fetch_add(5, std::memory_order_relaxed);
    return S256_SUCCESS;
}
// one chunk of encoded points: decode into ctx->aff (a failed decode sets msm_flag), then the sum
static int chunk_msm(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, int vartime, int first,
                     cudaStream_t s) {
    s256_launch_decode_uncompressed(ctx, pt65, n, ctx->aff, ctx->pvalid, s);
    LAUNCH(ctx, k_any_invalid, grid_for(n), 0, s, ctx->pvalid, n, ctx->msm_flag);
    return chunk_msm_body(ctx, k32, n, vartime, first, s);
}

// host pointers -> msm_acc holds the projective sum; *invalid = 1 if a point failed to decode
static int msm_run(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, int vartime, uint32_t *invalid) {
    int rc = msm_ensure(ctx);
    if (rc != S256_SUCCESS) return rc;
    cudaStream_t s = ctx->stream;
    CK(cudaMemsetAsync(ctx->msm_flag, 0, 4, s));
    if (n == 0) {
        pt id;
        pt_set_identity(id);
        CK(cudaMemcpyAsync(ctx->msm_acc, &id, sizeof(pt), cudaMemcpyHostToDevice, s));
        CK(cudaStreamSynchronize(s));
    }
    int first = 1;
    rc = for_chunks(ctx, n, [&](size_t off, size_t c) {
        CK(cudaMemcpyAsync(ctx->in_a, pt65 + 65 * off, 65 * c, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(ctx->in_b, k32 + 32 * off, 32 * c, cudaMemcpyHostToDevice, s));
        int r = chunk_msm(ctx, ctx->in_b, ctx->in_a, c, vartime, first, s);
        first = 0;
        return r;
    });
    if (rc != S256_SUCCESS) return rc;
    CK(cudaMemcpyAsync(invalid, ctx->msm_flag, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return check_launch(ctx);
}
// msm_acc -> 65-byte encoding + status
static int msm_finish(s256_ctx *ctx, uint8_t *out65, uint8_t *status) {
    cudaStream_t s = ctx->stream;
    s256_launch_finish_affine(ctx, 1, ctx->msm_acc, nullptr, nullptr, ctx->cstat, 0, ctx->out, ctx->st, nullptr, s);
    CK(cudaMemcpyAsync(out65, ctx->out, 65, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(status, ctx->st, 1, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return check_launch(ctx);
}
extern "C" int s256_msm(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, int vartime, uint8_t *out65,
                        uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (!out65 || !status || (n && (!k32 || !pt65))) return S256_ERR_ARG;
    uint32_t invalid = 0;
    int rc = msm_run(ctx, k32, pt65, n, vartime, &invalid);
    if (rc != S256_SUCCESS) return rc;
    if (invalid) {
        memset(out65, 0, 65);
        *status = S256_ST_INVALID;
        return S256_SUCCESS;
    }
    return msm_finish(ctx, out65, status);
}
extern "C" int s256_msm_partial(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, int vartime,
                                uint8_t *partial96, uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (!partial96 || !status || (n && (!k32 || !pt65))) return S256_ERR_ARG;
    uint32_t invalid = 0;
    int rc = msm_run(ctx, k32, pt65, n, vartime, &invalid);
    if (rc != S256_SUCCESS) return rc;
    if (invalid) {
        memset(partial96, 0, 96);
        *status = S256_ST_INVALID;
        return S256_SUCCESS;
    }
    cudaStream_t s = ctx->stream;
    k_export_partial<<<1, 1, 0, s>>>(ctx->msm_acc, ctx->out);
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
    CK(cudaMemcpyAsync(partial96, ctx->out, 96, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    *status = S256_ST_OK;
    return check_launch(ctx);
}
extern "C" int s256_msm_combine(s256_ctx *ctx, const uint8_t *partials96, size_t m, uint8_t *out65, uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (!out65 || !status || (m && !partials96)) return S256_ERR_ARG;
    if (96 * m > 65 * ctx->cap) return S256_ERR_ARG;
    int rc = msm_ensure(ctx);
    if (rc != S256_SUCCESS) return rc;
    cudaStream_t s = ctx->stream;
    CK(cudaMemsetAsync(ctx->msm_flag, 0, 4, s));
    if (m) CK(cudaMemcpyAsync(ctx->in_a, partials96, 96 * m, cudaMemcpyHostToDevice, s));
    k_combine_partials<<<1, 1, 0, s>>>(ctx->in_a, m, ctx->msm_acc, ctx->msm_flag);
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
    uint32_t invalid = 0;
    CK(cudaMemcpyAsync(&invalid, ctx->msm_flag, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (invalid) {
        memset(out65, 0, 65);
        *status = S256_ST_INVALID;
        return S256_SUCCESS;
    }
    return msm_finish(ctx, out65, status);
}


// ---------------------------------------------------------------------------
// Batch verification (batch.cuh): one verdict for a whole batch of BIP-340 signatures or of recoverable ECDSA
// signatures, from one randomized multi-scalar multiplication.
//
// Rows go in chunks of C = the largest power of two <= cap / 2, so that a chunk's 2C MSM points fit the per-chunk
// scratch and the chunk roots are nodes of the batch's hash tree.  Pass 1 hashes the rows into leaves (ctx->u1) and
// folds each chunk to its root (k_batch_tree); k_batch_seed folds the roots into the seed.  Pass 2 turns each chunk into
// its 2c MSM rows in ctx->aff / ctx->out plus per-CTA sums of the G-side scalars (ctx->u1, folded into one scalar by
// k_batch_fold) and runs them through the Pippenger body.  The finish adds (the scalar sum) G and tests the sum for the
// identity.  What differs between the two row kinds -- the leaf kernel, the prepare kernels and the seed's tag -- is a
// kind struct (batch_schnorr, batch_ecdsa) the shared driver batch_verify_run is instantiated with.
// ---------------------------------------------------------------------------
constexpr int BATCH_SEG = 2 * S256_TPB;  // nodes one CTA of k_batch_tree folds into one
// ctx->bat, in 32-bit words: the seed, the scalar sum (limbs), the scalar sum (big-endian bytes), one root per chunk
constexpr size_t BAT_SEED = 0, BAT_SUM = 8, BAT_SUM_BE = 16, BAT_ROOTS = 24;

// the sum of v over the CTA, valid in thread 0
__device__ sc cta_sc_sum(sc v) {
    __shared__ sc sh[S256_TPB];
    const int t = threadIdx.x;
    sh[t] = v;
    __syncthreads();
    for (int stride = S256_TPB / 2; stride >= 1; stride >>= 1) {
        if (t < stride) {
            sc a = sh[t], b = sh[t + stride];
            sc_add(a, a, b);
            sh[t] = a;
        }
        __syncthreads();
    }
    return sh[0];
}

// M: msg_uniform or msg_offsets (kernels.cuh)
template <class M>
__global__ void __launch_bounds__(S256_TPB) k_batch_leaves(const uint8_t *pkx32, M rows, const uint8_t *sig64, size_t n,
                                                           uint32_t *leaves) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t h[8];
    const uint8_t *m;
    size_t len;
    rows.row(i, m, len);  // an unreadable row hashes as empty; k_batch_prepare rejects it
    batch_leaf(h, pkx32 + 32 * i, sig64 + 64 * i, m, len);
    uint4 *o = reinterpret_cast<uint4 *>(leaves + 8 * i);
    o[0] = make_uint4(h[0], h[1], h[2], h[3]);
    o[1] = make_uint4(h[4], h[5], h[6], h[7]);
}
__global__ void __launch_bounds__(S256_TPB) k_ecdsa_batch_leaves(const uint8_t *pk65, const uint8_t *digest32,
                                                                 const uint8_t *sig65, size_t n, uint32_t *leaves) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t h[8];
    batch_leaf_ecdsa(h, pk65 + 65 * i, digest32 + 32 * i, sig65 + 65 * i);
    uint4 *o = reinterpret_cast<uint4 *>(leaves + 8 * i);
    o[0] = make_uint4(h[0], h[1], h[2], h[3]);
    o[1] = make_uint4(h[4], h[5], h[6], h[7]);
}
// out[b] = the node over in[b * BATCH_SEG, ...) by the tree rule: the first level from global memory, the rest in
// shared memory.  Segments start at multiples of 2^8, so out[] is a level of the whole tree.
__global__ void __launch_bounds__(S256_TPB) k_batch_tree(const uint32_t *in, size_t m, uint32_t *out) {
    __shared__ uint32_t sh[S256_TPB][8];
    const size_t base = (size_t)blockIdx.x * BATCH_SEG;
    const uint32_t t = threadIdx.x;
    uint32_t cnt = (uint32_t)(m - base < (size_t)BATCH_SEG ? m - base : (size_t)BATCH_SEG);
    uint32_t h[8] = {};
    if (2 * t + 1 < cnt) {
        batch_node(h, in + 8 * (base + 2 * t), in + 8 * (base + 2 * t + 1));
    } else if (2 * t < cnt) {
        for (int k = 0; k < 8; k++) h[k] = in[8 * (base + 2 * t) + k];
    }
    for (int k = 0; k < 8; k++) sh[t][k] = h[k];
    cnt = (cnt + 1) / 2;
    __syncthreads();
    while (cnt > 1) {
        uint32_t up = (cnt + 1) / 2;
        if (t < up) {
            if (2 * t + 1 < cnt) {
                batch_node(h, sh[2 * t], sh[2 * t + 1]);
            } else {
                for (int k = 0; k < 8; k++) h[k] = sh[2 * t][k];
            }
        }
        __syncthreads();
        if (t < up)
            for (int k = 0; k < 8; k++) sh[t][k] = h[k];
        __syncthreads();
        cnt = up;
    }
    if (t < 8) out[8 * (size_t)blockIdx.x + t] = sh[0][t];
}
// chunk roots -> seed (one thread; a batch has few chunks)
template <class Kind>
__global__ void k_batch_seed(uint32_t *bat, size_t chunks, uint64_t n) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    batch_tree_fold(bat + BAT_ROOTS, chunks);
    batch_seed(bat + BAT_SEED, bat + BAT_ROOTS, n, Kind::tag());
}
// rows [off, off + n) of the batch -> MSM rows 2i, 2i + 1 of the chunk, part[CTA] = the CTA's sum of a_i s_i,
// flag |= a rejected row
template <class M>
__global__ void __launch_bounds__(S256_TPB) k_batch_prepare(const uint8_t *pkx32, M rows, const uint8_t *sig64, size_t n,
                                                            size_t off, const uint32_t *seed_in, apt *aff2, uint8_t *k2,
                                                            sc *part, uint32_t *flag) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    sc as = sc_zero();
    if (i < n) {
        uint32_t seed[8];
        for (int k = 0; k < 8; k++) seed[k] = seed_in[k];
        const uint8_t *m;
        size_t len;
        const uint32_t row_ok = rows.row(i, m, len);
        uint32_t ok = item_batch_prepare(aff2 + 2 * i, k2 + 64 * i, as, pkx32 + 32 * i, m, len, sig64 + 64 * i, seed,
                                         (uint64_t)(off + i), row_ok);
        if (!ok) atomicOr(flag, 1u);
    }
    sc sum = cta_sc_sum(as);
    if (threadIdx.x == 0) part[blockIdx.x] = sum;
}
// ECDSA rows [0, n) of the chunk -> the points -R_i, Q_i of MSM rows 2i, 2i + 1 and pvalid[i], one row per thread
__global__ void __launch_bounds__(S256_TPB) k_ecdsa_batch_points(const uint8_t *pk65, const uint8_t *sig65, size_t n,
                                                                 apt *aff2, uint8_t *pvalid) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    pvalid[i] = (uint8_t)item_ecdsa_batch_points(aff2 + 2 * i, pk65 + 65 * i, sig65 + 65 * i);
}
// ECDSA rows [off, off + n) of the batch, K per thread sharing one inversion -> the scalars of MSM rows 2i, 2i + 1
// (G with scalar 0 for a rejected row), part[CTA] = the CTA's sum of a_i u1_i, flag |= a rejected row
template <int K>
__global__ void __launch_bounds__(S256_TPB) k_ecdsa_batch_prepare(const uint8_t *digest32, const uint8_t *sig65,
                                                                  uint32_t flags, const uint8_t *pvalid, size_t n, size_t off,
                                                                  const uint32_t *seed_in, apt *aff2, uint8_t *k2, sc *part,
                                                                  uint32_t *flag) {
    const size_t stride = (n + K - 1) / K;
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    sc au1 = sc_zero();
    if (t < stride) {
        uint32_t seed[8];
        for (int k = 0; k < 8; k++) seed[k] = seed_in[k];
        uint32_t ok = group_ecdsa_batch_prepare<K>(t, stride, n, off, digest32, sig65, flags, pvalid, seed, aff2, k2, au1);
        if (!ok) atomicOr(flag, 1u);
    }
    sc sum = cta_sc_sum(au1);
    if (threadIdx.x == 0) part[blockIdx.x] = sum;
}
// the scalar sum (+)= the m CTA sums (first = overwrite), kept as limbs and as big-endian bytes.  One CTA.
__global__ void __launch_bounds__(S256_TPB) k_batch_fold(const sc *part, size_t m, uint32_t *bat, int first) {
    sc acc = sc_zero();
    for (size_t j = threadIdx.x; j < m; j += S256_TPB) {
        sc q = part[j];
        sc_add(acc, acc, q);
    }
    sc r = cta_sc_sum(acc);
    if (threadIdx.x == 0) {
        sc *sum = reinterpret_cast<sc *>(bat + BAT_SUM);
        if (!first) {
            sc a = *sum;
            sc_add(r, r, a);
        }
        *sum = r;
        sc_to_be32(reinterpret_cast<uint8_t *>(bat + BAT_SUM_BE), r);
    }
}
// ok = no row was rejected and the sum is the identity
__global__ void k_batch_verdict(const uint32_t *flag, const pt *acc, uint8_t *ok) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    pt a = *acc;
    *ok = (uint8_t)((uint32_t)(*flag == 0) & fe_is_zero(a.z));
}

static size_t batch_chunk(const s256_ctx *ctx) {  // the largest power of two <= cap / 2
    size_t c = 1;
    while (4 * c <= ctx->cap) c *= 2;
    return c;
}
static int batch_ensure(s256_ctx *ctx, size_t chunks) {
    if (chunks <= ctx->bat_chunks) return S256_SUCCESS;
    if (chunks < 16) chunks = 16;
    uint32_t *fresh = nullptr;
    CK(cudaMalloc(&fresh, (BAT_ROOTS + 8 * chunks) * 4));
    if (ctx->bat) cudaFree(ctx->bat);  // synchronises the device: no call still reads the old array
    ctx->bat = fresh;
    ctx->bat_chunks = chunks;
    return S256_SUCCESS;
}
// A batch's rows: three arrays of fixed-width rows (width 0: no bytes) and the flags of the call.
//   BIP-340: a = x-only keys (32), b = messages (msg_len), c = r||s (64)
//   ECDSA:   a = keys (65),        b = digests (32),       c = r||s||v (65)
// BIP-340 messages of any length (the *_varlen calls) have wb = 0 and offsets: row i of b is
// b[boff[i] - bbase, boff[i + 1] - bbase) (msg_offsets).
struct batch_rows {
    const uint8_t *a, *b, *c;
    size_t wa, wb, wc;
    uint32_t flags;
    const size_t *boff = nullptr;
    size_t bbase = 0;
    batch_rows at(size_t off) const {
        return {a + wa * off, wb ? b + wb * off : b, c + wc * off, wa, wb, wc, flags, boff ? boff + off : boff, bbase};
    }
};
// The row kinds: the seed's tag, pass 1 (leaves of c rows into `leaves`) and pass 2 (the chunk's MSM rows and per-CTA
// G-side sums in ctx->u1; returns the number of CTA sums).
struct batch_schnorr {
    static __host__ __device__ const char *tag() { return S256_BATCH_TAG_BIP340; }
    static void leaves(s256_ctx *ctx, const batch_rows &r, size_t c, uint32_t *leaves, cudaStream_t s) {
        if (r.boff)
            LAUNCH(ctx, k_batch_leaves<msg_offsets>, grid_for(c), 0, s, r.a, msg_offsets{r.b, r.boff, r.bbase}, r.c, c, leaves);
        else
            LAUNCH(ctx, k_batch_leaves<msg_uniform>, grid_for(c), 0, s, r.a, msg_uniform{r.b, r.wb}, r.c, c, leaves);
    }
    static size_t prepare(s256_ctx *ctx, const batch_rows &r, size_t c, size_t off, cudaStream_t s) {
        if (r.boff)
            LAUNCH(ctx, k_batch_prepare<msg_offsets>, grid_for(c), 0, s, r.a, msg_offsets{r.b, r.boff, r.bbase}, r.c, c, off,
                   ctx->bat + BAT_SEED, ctx->aff, ctx->out, ctx->u1, ctx->msm_flag);
        else
            LAUNCH(ctx, k_batch_prepare<msg_uniform>, grid_for(c), 0, s, r.a, msg_uniform{r.b, r.wb}, r.c, c, off,
                   ctx->bat + BAT_SEED, ctx->aff, ctx->out, ctx->u1, ctx->msm_flag);
        return grid_for(c);
    }
};
struct batch_ecdsa {
    static __host__ __device__ const char *tag() { return S256_BATCH_TAG_ECDSA; }
    static void leaves(s256_ctx *ctx, const batch_rows &r, size_t c, uint32_t *leaves, cudaStream_t s) {
        LAUNCH(ctx, k_ecdsa_batch_leaves, grid_for(c), 0, s, r.a, r.b, r.c, c, leaves);
    }
    // The points go one row per thread; the scalars K rows per thread (inv_k_for), so that K rows share the inversion
    // of s without running the square root of RecoverPoint on c / K threads.
    static size_t prepare(s256_ctx *ctx, const batch_rows &r, size_t c, size_t off, cudaStream_t s) {
        LAUNCH(ctx, k_ecdsa_batch_points, grid_for(c), 0, s, r.a, r.c, c, ctx->aff, ctx->pvalid);
        size_t parts = 0;
        DISPATCH_K(c, {
            LAUNCH(ctx, k_ecdsa_batch_prepare<KK>, grid_for_groups(c, KK), 0, s, r.b, r.c, r.flags, ctx->pvalid, c, off,
                   ctx->bat + BAT_SEED, ctx->aff, ctx->out, ctx->u1, ctx->msm_flag);
            parts = grid_for_groups(c, KK);
        });
        return parts;
    }
};
// chunk_done(off, c): called once per chunk while its MSM rows are in ctx->out / ctx->aff (the debug hooks)
using batch_chunk_fn = std::function<int(size_t, size_t)>;
// n >= 1 rows; rows(off, c, pass, r) gives the device rows of a chunk (the host form copies them in first).
// The verdict byte goes to d_ok; nothing is synchronised unless chunk_done does.
template <class Kind, typename F>
static int batch_verify_run(s256_ctx *ctx, size_t n, F rows, uint8_t *d_ok, cudaStream_t s,
                            const batch_chunk_fn &chunk_done = nullptr) {
    int rc = msm_ensure(ctx);
    if (rc != S256_SUCCESS) return rc;
    const size_t C = batch_chunk(ctx), chunks = (n + C - 1) / C;
    rc = batch_ensure(ctx, chunks);
    if (rc != S256_SUCCESS) return rc;
    uint32_t *leaves = reinterpret_cast<uint32_t *>(ctx->u1);
    uint32_t *level[2] = {reinterpret_cast<uint32_t *>(ctx->res),
                          reinterpret_cast<uint32_t *>(ctx->res) + 8 * ((C + BATCH_SEG - 1) / BATCH_SEG)};
    batch_rows r;
    // pass 1: leaves -> chunk roots -> seed
    for (size_t k = 0; k < chunks; k++) {
        const size_t off = k * C, c = n - off < C ? n - off : C;
        rc = rows(off, c, 0, r);
        if (rc != S256_SUCCESS) return rc;
        Kind::leaves(ctx, r, c, leaves, s);
        const uint32_t *src = leaves;
        size_t m = c;
        int side = 0;
        do {
            size_t g = (m + BATCH_SEG - 1) / BATCH_SEG;
            uint32_t *dst = g == 1 ? ctx->bat + BAT_ROOTS + 8 * k : level[side];
            LAUNCH(ctx, k_batch_tree, (unsigned)g, 0, s, src, m, dst);
            src = dst;
            side ^= 1;
            m = g;
        } while (m > 1);
    }
    k_batch_seed<Kind><<<1, 1, 0, s>>>(ctx->bat, chunks, (uint64_t)n);
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
    // pass 2: per chunk, the MSM rows and the scalar sum, then the Pippenger body
    CK(cudaMemsetAsync(ctx->msm_flag, 0, 4, s));
    for (size_t k = 0; k < chunks; k++) {
        const size_t off = k * C, c = n - off < C ? n - off : C;
        rc = rows(off, c, 1, r);
        if (rc != S256_SUCCESS) return rc;
        const size_t parts = Kind::prepare(ctx, r, c, off, s);
        k_batch_fold<<<1, S256_TPB, 0, s>>>(ctx->u1, parts, ctx->bat, k == 0);
        ctx->launches.fetch_add(1, std::memory_order_relaxed);
        if (chunk_done && (rc = chunk_done(off, c)) != S256_SUCCESS) return rc;
        rc = chunk_msm_body(ctx, ctx->out, 2 * c, 1, k == 0, s);
        if (rc != S256_SUCCESS) return rc;
    }
    // finish: + (the scalar sum) G, then the verdict
    s256_launch_base_mult_ct(reinterpret_cast<const uint8_t *>(ctx->bat + BAT_SUM_BE), 1, ctx->ct_tab, ctx->ct_tab_small,
                             ctx->ct_tab_huge, ctx->res, s);
    k_acc_point<<<1, 1, 0, s>>>(ctx->res, ctx->msm_acc, 0);
    k_batch_verdict<<<1, 1, 0, s>>>(ctx->msm_flag, ctx->msm_acc, d_ok);
    ctx->launches.fetch_add(3, std::memory_order_relaxed);
    return check_launch(ctx);
}
// The device form: rows in device memory, the verdict byte to d_ok, nothing synchronised.
template <class Kind>
static int batch_verify_dev(s256_ctx *ctx, const batch_rows &dev, size_t n, uint8_t *d_ok, cudaStream_t s) {
    if (n == 0) {
        CK(cudaMemsetAsync(d_ok, 1, 1, s));
        return S256_SUCCESS;
    }
    return batch_verify_run<Kind>(ctx, n, [&](size_t off, size_t, int, batch_rows &r) {
        r = dev.at(off);
        return S256_SUCCESS;
    }, d_ok, s);
}
// The host form's rows: a batch of one chunk is copied in once and read by both passes, a longer one chunk by chunk in
// each pass.  Ragged messages go with their offsets (varlen_staging checks them first).  The verdict byte goes to ctx->st.
template <class Kind>
static int batch_verify_host(s256_ctx *ctx, const batch_rows &host, size_t n, const batch_chunk_fn &chunk_done = nullptr) {
    const size_t C = batch_chunk(ctx);
    if (int grc = host.boff ? varlen_staging(ctx, host.b, host.boff, n, C) : grow_in_b(ctx, (host.wb ? host.wb : 1) * C))
        return grc;
    cudaStream_t s = ctx->stream;
    const bool resident = n <= C;
    const batch_rows staged{ctx->in_a, ctx->in_b, ctx->in_c, host.wa, host.wb, host.wc, host.flags,
                            host.boff ? ctx->in_off : nullptr};
    return batch_verify_run<Kind>(ctx, n, [&](size_t off, size_t c, int pass, batch_rows &r) {
        if (pass == 0 || !resident) {
            const batch_rows h = host.at(off);
            CK(cudaMemcpyAsync(ctx->in_a, h.a, h.wa * c, cudaMemcpyHostToDevice, s));
            msg_offsets unused;
            if (h.boff) {
                if (int rc = varlen_stage_part(ctx, host.b, host.boff, off, 0, c, s, unused)) return rc;
            } else if (h.wb) {
                CK(cudaMemcpyAsync(ctx->in_b, h.b, h.wb * c, cudaMemcpyHostToDevice, s));
            }
            CK(cudaMemcpyAsync(ctx->in_c, h.c, h.wc * c, cudaMemcpyHostToDevice, s));
        }
        r = staged;
        if (host.boff) r.bbase = host.boff[off];
        return S256_SUCCESS;
    }, ctx->st, s, chunk_done);
}
// host rows -> *ok, the one host synchronisation of the call
template <class Kind>
static int batch_verify_host_sync(s256_ctx *ctx, const batch_rows &host, size_t n, uint8_t *ok) {
    if (n == 0) {
        *ok = 1;
        return S256_SUCCESS;
    }
    cudaStream_t s = ctx->stream;
    int rc = batch_verify_host<Kind>(ctx, host, n);
    if (rc != S256_SUCCESS) return rc;
    CK(cudaMemcpyAsync(ok, ctx->st, 1, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return check_launch(ctx);
}
// The batch equation as the kernels build it, copied back chunk by chunk (the s256_debug_*_batch_rows hooks).
template <class Kind>
static int batch_debug_rows(s256_ctx *ctx, const batch_rows &host, size_t n, uint8_t *seed32, uint8_t *k64,
                            uint8_t *pts128, uint8_t *sum32, uint8_t *rejected) {
    cudaStream_t s = ctx->stream;
    std::vector<apt> aff;
    int rc = batch_verify_host<Kind>(ctx, host, n, [&](size_t off, size_t c) {
        aff.resize(2 * c);
        CK(cudaMemcpyAsync(k64 + 64 * off, ctx->out, 64 * c, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(aff.data(), ctx->aff, 2 * c * sizeof(apt), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        for (size_t v = 0; v < 2 * c; v++) {
            fe_to_be32(pts128 + 64 * (2 * off + v), aff[v].x);
            fe_to_be32(pts128 + 64 * (2 * off + v) + 32, aff[v].y);
        }
        return S256_SUCCESS;
    });
    if (rc != S256_SUCCESS) return rc;
    uint32_t seed[8], flag = 0;
    CK(cudaMemcpyAsync(seed, ctx->bat + BAT_SEED, 32, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(sum32, ctx->bat + BAT_SUM_BE, 32, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(&flag, ctx->msm_flag, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    words_be32(seed32, seed);
    *rejected = (uint8_t)(flag != 0);
    return check_launch(ctx);
}

static batch_rows schnorr_rows(const uint8_t *pkx, const uint8_t *msg, size_t msg_len, const uint8_t *sig) {
    return {pkx, msg, sig, 32, msg_len, 64, 0u};
}
extern "C" int s256_schnorr_batch_verify_dev(s256_ctx *ctx, const uint8_t *pkx, const uint8_t *msg, size_t msg_len,
                                             const uint8_t *sig, size_t n, uint8_t *ok, void *stream) {
    ENTER(ctx);
    if (!ok || (n && (!pkx || (!msg && msg_len) || !sig))) return S256_ERR_ARG;
    if (ctx->cap < 2) return S256_ERR_ARG;  // a chunk needs two MSM rows per signature
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    return batch_verify_dev<batch_schnorr>(ctx, schnorr_rows(pkx, msg, msg_len, sig), n, ok, s);
}
extern "C" int s256_schnorr_batch_verify(s256_ctx *ctx, const uint8_t *pkx, const uint8_t *msg, size_t msg_len,
                                         const uint8_t *sig, size_t n, uint8_t *ok) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (!ok || (n && (!pkx || (!msg && msg_len) || !sig))) return S256_ERR_ARG;
    if (ctx->cap < 2) return S256_ERR_ARG;
    return batch_verify_host_sync<batch_schnorr>(ctx, schnorr_rows(pkx, msg, msg_len, sig), n, ok);
}
extern "C" int s256_debug_schnorr_batch_rows(s256_ctx *ctx, const uint8_t *pkx, const uint8_t *msg, size_t msg_len,
                                             const uint8_t *sig, size_t n, uint8_t *seed32, uint8_t *k64, uint8_t *pts128,
                                             uint8_t *sum32, uint8_t *rejected) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n == 0 || !pkx || (!msg && msg_len) || !sig || !seed32 || !k64 || !pts128 || !sum32 || !rejected)
        return S256_ERR_ARG;
    if (ctx->cap < 2) return S256_ERR_ARG;
    return batch_debug_rows<batch_schnorr>(ctx, schnorr_rows(pkx, msg, msg_len, sig), n, seed32, k64, pts128, sum32, rejected);
}

static batch_rows schnorr_varlen_rows(const uint8_t *pkx, const uint8_t *msg, const size_t *offsets, const uint8_t *sig) {
    return {pkx, msg, sig, 32, 0, 64, 0u, offsets};
}
extern "C" int s256_schnorr_batch_verify_varlen_dev(s256_ctx *ctx, const uint8_t *pkx, const uint8_t *msg, const size_t *offsets,
                                                    const uint8_t *sig, size_t n, uint8_t *ok, void *stream) {
    ENTER(ctx);
    if (!ok || (n && (!pkx || !msg || !offsets || !sig))) return S256_ERR_ARG;
    if (ctx->cap < 2) return S256_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    return batch_verify_dev<batch_schnorr>(ctx, schnorr_varlen_rows(pkx, msg, offsets, sig), n, ok, s);
}
extern "C" int s256_schnorr_batch_verify_varlen(s256_ctx *ctx, const uint8_t *pkx, const uint8_t *msg, const size_t *offsets,
                                                const uint8_t *sig, size_t n, uint8_t *ok) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (!ok || (n && (!pkx || !offsets || !sig))) return S256_ERR_ARG;
    if (ctx->cap < 2) return S256_ERR_ARG;
    return batch_verify_host_sync<batch_schnorr>(ctx, schnorr_varlen_rows(pkx, msg, offsets, sig), n, ok);
}
extern "C" int s256_debug_schnorr_batch_rows_varlen(s256_ctx *ctx, const uint8_t *pkx, const uint8_t *msg,
                                                    const size_t *offsets, const uint8_t *sig, size_t n, uint8_t *seed32,
                                                    uint8_t *k64, uint8_t *pts128, uint8_t *sum32, uint8_t *rejected) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n == 0 || !pkx || !offsets || !sig || !seed32 || !k64 || !pts128 || !sum32 || !rejected) return S256_ERR_ARG;
    if (ctx->cap < 2) return S256_ERR_ARG;
    return batch_debug_rows<batch_schnorr>(ctx, schnorr_varlen_rows(pkx, msg, offsets, sig), n, seed32, k64, pts128, sum32,
                                           rejected);
}

static batch_rows ecdsa_rows(const uint8_t *pk65, const uint8_t *digest32, const uint8_t *sig65, uint32_t flags) {
    return {pk65, digest32, sig65, 65, 32, 65, flags};
}
extern "C" int s256_ecdsa_recoverable_batch_verify_dev(s256_ctx *ctx, const uint8_t *pk65, const uint8_t *digest32,
                                                       const uint8_t *sig65, uint32_t flags, size_t n, uint8_t *ok,
                                                       void *stream) {
    ENTER(ctx);
    if (!ok || (n && (!pk65 || !digest32 || !sig65))) return S256_ERR_ARG;
    if (ctx->cap < 2) return S256_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    return batch_verify_dev<batch_ecdsa>(ctx, ecdsa_rows(pk65, digest32, sig65, flags), n, ok, s);
}
extern "C" int s256_ecdsa_recoverable_batch_verify(s256_ctx *ctx, const uint8_t *pk65, const uint8_t *digest32,
                                                   const uint8_t *sig65, uint32_t flags, size_t n, uint8_t *ok) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (!ok || (n && (!pk65 || !digest32 || !sig65))) return S256_ERR_ARG;
    if (ctx->cap < 2) return S256_ERR_ARG;
    return batch_verify_host_sync<batch_ecdsa>(ctx, ecdsa_rows(pk65, digest32, sig65, flags), n, ok);
}
extern "C" int s256_debug_ecdsa_batch_rows(s256_ctx *ctx, const uint8_t *pk65, const uint8_t *digest32, const uint8_t *sig65,
                                           uint32_t flags, size_t n, uint8_t *seed32, uint8_t *k64, uint8_t *pts128,
                                           uint8_t *sum32, uint8_t *rejected) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (n == 0 || !pk65 || !digest32 || !sig65 || !seed32 || !k64 || !pts128 || !sum32 || !rejected) return S256_ERR_ARG;
    if (ctx->cap < 2) return S256_ERR_ARG;
    return batch_debug_rows<batch_ecdsa>(ctx, ecdsa_rows(pk65, digest32, sig65, flags), n, seed32, k64, pts128, sum32,
                                         rejected);
}



// ---------------------------------------------------------------------------
// Device-resident and multi-GPU MSM.
//
// s256_msm_dev: inputs and outputs in HBM, everything enqueued on the caller's stream, no host synchronisation.
//
// s256_msm_sharded[_dev]: config 5 of BASELINE.json.  One process per GPU; rank g passes ITS contiguous slice of the
// batch.  Each rank reduces its slice to a projective partial (Pippenger), ONE ncclAllGather of 112 bytes per rank
// brings the partials together on every GPU, one warp folds them (8-lane cooperative additions) and the shared
// batched-affine kernel encodes the sum.  The partials never leave the device; the host-pointer form synchronises once,
// to read 66 bytes.  NCCL is resolved with dlopen at the first s256_comm_* call: in a process that already uses NCCL
// (torch.distributed) that is the copy already loaded, otherwise libnccl.so.2 from the loader path; a context that
// never shards never touches it.  The communicator is built from an ncclUniqueId that rank 0 obtains with
// s256_comm_unique_id and the application hands to the other ranks (any channel: MPI, torch.distributed, a file).
// ---------------------------------------------------------------------------
namespace {
struct nccl_api {
    void *h = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};
nccl_api &nccl() {
    static nccl_api api;
    static std::once_flag once;
    std::call_once(once, [] {
        void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);   // the copy the process already uses, if any
        if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return;
        api.h = h;
        api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(dlsym(h, "ncclGetUniqueId"));
        api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(dlsym(h, "ncclCommInitRank"));
        api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(dlsym(h, "ncclCommDestroy"));
        api.AllGather = reinterpret_cast<decltype(api.AllGather)>(dlsym(h, "ncclAllGather"));
        api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(dlsym(h, "ncclGetErrorString"));
        api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllGather && api.GetErrorString;
    });
    return api;
}
#define NCCLCK(call)                                                                             \
    do {                                                                                         \
        ncclResult_t r_ = (call);                                                                \
        if (r_ != ncclSuccess) {                                                                 \
            ctx->last_err = std::string(#call) + ": " + nccl().GetErrorString(r_);               \
            return S256_ERR_NCCL;                                                                \
        }                                                                                        \
    } while (0)

// what one rank contributes to the gather: its projective partial in limb form and its "a point failed to decode" flag
struct msm_wire {
    pt p;
    uint32_t invalid, pad[3];
};
static_assert(sizeof(msm_wire) == 112, "wire format");
}  // namespace

__global__ void k_msm_pack(const pt *acc, const uint32_t *flag, msm_wire *out) {
    if (threadIdx.x == 0) {
        out->p = *acc;
        out->invalid = *flag;
        out->pad[0] = out->pad[1] = out->pad[2] = 0;
    }
}
// acc = sum of the m gathered partials (one warp, 8-lane cooperative additions); flag |= any rank's flag
__global__ void __launch_bounds__(32) k_msm_fold_wire(const msm_wire *in, int m, pt *acc, uint32_t *flag) {
    int j = threadIdx.x & 7;
    pt r;
    pt_set_identity(r);
    uint32_t bad = 0;
    for (int g = 0; g < m; g++) {
        pt q = in[g].p;
        bad |= in[g].invalid;
        pt_add_coop(r, q, j);
    }
    __syncwarp();
    if (threadIdx.x == 0) {
        *acc = r;
        if (bad) atomicOr(flag, 1u);
    }
}
// after the encode: a failed decode anywhere turns the result into (all zero, S256_ST_INVALID), on the device
__global__ void k_msm_publish(const uint32_t *flag, uint8_t *out65, uint8_t *status) {
    if (*flag) {
        for (int i = threadIdx.x; i < 65; i += blockDim.x) out65[i] = 0;
        if (threadIdx.x == 0) *status = S256_ST_INVALID;
    }
}

// device pointers, any n: msm_acc / msm_flag hold the local sum afterwards (nothing synchronised)
static int msm_run_dev(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, int vartime, cudaStream_t s) {
    int rc = msm_ensure(ctx);
    if (rc != S256_SUCCESS) return rc;
    CK(cudaMemsetAsync(ctx->msm_flag, 0, 4, s));
    if (n == 0) {
        static const pt id = [] { pt p; pt_set_identity(p); return p; }();
        CK(cudaMemcpyAsync(ctx->msm_acc, &id, sizeof(pt), cudaMemcpyHostToDevice, s));
    }
    int first = 1;
    return for_chunks(ctx, n, [&](size_t off, size_t c) {
        int r = chunk_msm(ctx, k32 + 32 * off, pt65 + 65 * off, c, vartime, first, s);
        first = 0;
        return r;
    });
}
// msm_acc -> out65 / status (device pointers), flag honoured, nothing synchronised
static int msm_finish_dev(s256_ctx *ctx, uint8_t *out65, uint8_t *status, cudaStream_t s) {
    s256_launch_finish_affine(ctx, 1, ctx->msm_acc, nullptr, nullptr, ctx->cstat, 0, out65, status, nullptr, s);
    k_msm_publish<<<1, 96, 0, s>>>(ctx->msm_flag, out65, status);
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
    return check_launch(ctx);
}
extern "C" int s256_msm_dev(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, int vartime, uint8_t *out65,
                            uint8_t *status, void *stream) {
    ENTER(ctx);
    if (!out65 || !status || (n && (!k32 || !pt65))) return S256_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    int rc = msm_run_dev(ctx, k32, pt65, n, vartime, s);
    if (rc != S256_SUCCESS) return rc;
    return msm_finish_dev(ctx, out65, status, s);
}

// the Pippenger plan for n points on one GPU (window bits, windows): what bench.py's work model needs
extern "C" int s256_msm_plan(size_t n, int *window_bits, int *windows) {
    if (!window_bits || !windows) return S256_ERR_ARG;
    msm_plan pl = msm_make_plan(2 * n, 128);
    *window_bits = pl.c;
    *windows = pl.nwin;
    return S256_SUCCESS;
}
extern "C" int s256_comm_unique_id(uint8_t id128[128]) {
    if (!id128) return S256_ERR_ARG;
    if (!nccl().ok) return S256_ERR_NCCL;
    ncclUniqueId id;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId");
    if (nccl().GetUniqueId(&id) != ncclSuccess) return S256_ERR_NCCL;
    memcpy(id128, &id, 128);
    return S256_SUCCESS;
}
extern "C" int s256_comm_init(s256_ctx *ctx, const uint8_t id128[128], int rank, int nranks) {
    ENTER(ctx);
    if (!id128 || nranks < 1 || rank < 0 || rank >= nranks || nranks > S256_COMM_MAX_RANKS) return S256_ERR_ARG;
    if (!nccl().ok) {
        ctx->last_err = "libnccl.so.2 not found (dlopen)";
        return S256_ERR_NCCL;
    }
    if (ctx->comm) {
        nccl().CommDestroy((ncclComm_t)ctx->comm);
        ctx->comm = nullptr;
    }
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    ncclComm_t comm = nullptr;
    NCCLCK(nccl().CommInitRank(&comm, nranks, id, rank));
    ctx->comm = comm;
    ctx->comm_rank = rank;
    ctx->comm_size = nranks;
    if (!ctx->comm_buf) CK(cudaMalloc(&ctx->comm_buf, sizeof(msm_wire) * (S256_COMM_MAX_RANKS + 1)));
    return S256_SUCCESS;
}
void s256_internal_comm_release(s256_ctx *ctx) {
    if (ctx->comm && nccl().ok) nccl().CommDestroy((ncclComm_t)ctx->comm);
    ctx->comm = nullptr;
    ctx->comm_size = 0;
}
extern "C" int s256_comm_free(s256_ctx *ctx) {
    ENTER(ctx);
    s256_internal_comm_release(ctx);
    return S256_SUCCESS;
}
// local partial (already in msm_acc / msm_flag) -> gathered and folded on every rank
static int msm_exchange(s256_ctx *ctx, cudaStream_t s) {
    if (!ctx->comm) return S256_SUCCESS;  // no communicator: the partial is the sum
    msm_wire *send = reinterpret_cast<msm_wire *>(ctx->comm_buf), *recv = send + 1;
    k_msm_pack<<<1, 32, 0, s>>>(ctx->msm_acc, ctx->msm_flag, send);
    NCCLCK(nccl().AllGather(send, recv, sizeof(msm_wire), ncclUint8, (ncclComm_t)ctx->comm, s));
    k_msm_fold_wire<<<1, 32, 0, s>>>(recv, ctx->comm_size, ctx->msm_acc, ctx->msm_flag);
    ctx->launches.fetch_add(2, std::memory_order_relaxed);
    return S256_SUCCESS;
}
extern "C" int s256_msm_sharded_dev(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n_local, int vartime,
                                    uint8_t *out65, uint8_t *status, void *stream) {
    ENTER(ctx);
    if (!out65 || !status || (n_local && (!k32 || !pt65))) return S256_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    scratch_guard sg_(ctx, s, false);
    int rc = msm_run_dev(ctx, k32, pt65, n_local, vartime, s);
    if (rc != S256_SUCCESS) return rc;
    rc = msm_exchange(ctx, s);
    if (rc != S256_SUCCESS) return rc;
    return msm_finish_dev(ctx, out65, status, s);
}
extern "C" int s256_msm_sharded(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n_local, int vartime,
                                uint8_t *out65, uint8_t *status) {
    ENTER(ctx);
    scratch_guard sg_(ctx, ctx->stream, true);
    if (!out65 || !status || (n_local && (!k32 || !pt65))) return S256_ERR_ARG;
    cudaStream_t s = ctx->stream;
    int rc = msm_ensure(ctx);
    if (rc != S256_SUCCESS) return rc;
    CK(cudaMemsetAsync(ctx->msm_flag, 0, 4, s));
    if (n_local == 0) {
        static const pt id = [] { pt p; pt_set_identity(p); return p; }();
        CK(cudaMemcpyAsync(ctx->msm_acc, &id, sizeof(pt), cudaMemcpyHostToDevice, s));
    }
    int first = 1;
    rc = for_chunks(ctx, n_local, [&](size_t off, size_t c) {
        CK(cudaMemcpyAsync(ctx->in_a, pt65 + 65 * off, 65 * c, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(ctx->in_b, k32 + 32 * off, 32 * c, cudaMemcpyHostToDevice, s));
        int r = chunk_msm(ctx, ctx->in_b, ctx->in_a, c, vartime, first, s);
        first = 0;
        return r;
    });
    if (rc != S256_SUCCESS) return rc;
    rc = msm_exchange(ctx, s);
    if (rc != S256_SUCCESS) return rc;
    rc = msm_finish_dev(ctx, ctx->out, ctx->st, s);
    if (rc != S256_SUCCESS) return rc;
    CK(cudaMemcpyAsync(out65, ctx->out, 65, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(status, ctx->st, 1, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));  // the one host synchronisation of the call
    return check_launch(ctx);
}
