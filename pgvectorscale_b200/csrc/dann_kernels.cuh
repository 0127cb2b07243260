// dann_kernels.cuh — the non-graph kernels of the scan path (sm_100a):
//   prepare_queries  : amrescan's vector preparation (cosine normalise + SBQ quantize)
//   sbq_distance     : stand-alone batched SBQ XOR+popcount gather (the roofline kernel)
//   full_distance    : exact f32 L2 / cosine / inner product, AVX2 summation order
//   rerank_resort    : get_full_distance_for_resort + the sliding rerank window
//   normalize_rows / pad_rows : index load helpers
// Reference paths are relative to /root/reference/pgvectorscale/src/access_method/.
// Every f32 operation that decides a result is spelled with an explicit-rounding
// intrinsic (__fadd_rn, __fmul_rn, __fmaf_rn, __fdiv_rn, __fsqrt_rn): nvcc never
// contracts or reorders those, so the arithmetic is the reference's op for op.
#pragma once
#include <math_constants.h>

#include "dann_device.cuh"
#include "dann_distance.cuh"
#include "dann_heap.cuh"

/* f32::NAN (0x7fc00000): the "no distance" value of padded / unrescored rows */
#define DANN_NAN_F __int_as_float(0x7fc00000)

/* ------------------------------------------------------------------------------------ */
/* preprocess_cosine (distance/mod.rs:225-253): norm = sequential f32 sum of v*v;        */
/* returns the divisor (sqrt(norm)) or 0 when the vector is left untouched.              */
__device__ __forceinline__ float cosine_divisor_from_norm(float norm, uint32_t len) {
    const float eps = 1.1920929e-07f; /* f32::EPSILON */
    float adj = __fmul_rn(eps, (float)len);
    if (norm < eps) return 0.0f;
    if (norm >= __fsub_rn(1.0f, adj) && norm <= __fadd_rn(1.0f, adj)) return 0.0f;
    return __fsqrt_rn(norm);
}

/* SbqQuantizer::quantize, one dimension (sbq/quantize.rs:52-102): number of leading ones */
__device__ __forceinline__ uint32_t sbq_count_ones(float v, float mean, float m2, float count_f,
                                                   uint32_t bits) {
    if (bits == 1) return v > mean ? 1u : 0u;
    float variance = __fdiv_rn(m2, count_f);
    float std_dev = __fsqrt_rn(variance);
    float z = __fdiv_rn(__fsub_rn(v, mean), std_dev);
    float ranges = (float)(bits + 1);
    float index = __fdiv_rn(__fadd_rn(z, 2.0f), __fdiv_rn(4.0f, ranges));
    if (index < 1.0f) return 0u;
    float fl = floorf(index); /* `index.floor() as usize`: saturating, NaN -> 0 */
    uint32_t as_u;
    if (!(fl == fl)) as_u = 0u;
    else if (fl >= 4294967040.0f) as_u = 0xFFFFFFFFu;
    else if (fl <= 0.0f) as_u = 0u;
    else as_u = (uint32_t)fl;
    return as_u < bits ? as_u : bits;
}

/* One CTA per query.  q_full_out [B][dim] (optional), q_codes_out [B][cw].
 * labels/mod.rs:209-238 (from_scan_key_data) -> pg_vector.rs:125-157 (create_inner: the
 * index copy is truncated to dim_index, each copy normalised on its own) ->
 * sbq/mod.rs:145-148 (quantize the index copy). */
__global__ void __launch_bounds__(128) dann_prepare_kernel(IndexView ix, const float *queries, int B,
                                                           float *q_full_out, uint64_t *q_codes_out) {
    DANN_DYN_SMEM(dann_smem);
    float *qi = reinterpret_cast<float *>(dann_smem); /* [dim_index] normalised index copy */
    DANN_STATIC_SMEM float s_div[2];
    const int q = blockIdx.x;
    const float *src = queries + (size_t)q * ix.dim;
    const bool cosine = ix.distance_type == DANN_COSINE;
    if (cosine) {
        /* Iterator::sum over v*v in index order: a sequential dependent chain; two warps
         * run the two chains (full copy / truncated copy) side by side. */
        if (threadIdx.x == 0 || threadIdx.x == 32) {
            const uint32_t len = threadIdx.x == 0 ? ix.dim : ix.dim_index;
            float norm = 0.0f;
            for (uint32_t i = 0; i < len; i++) {
                float v = src[i];
                norm = __fadd_rn(norm, __fmul_rn(v, v));
            }
            s_div[threadIdx.x >> 5] = cosine_divisor_from_norm(norm, len);
        }
    } else if (threadIdx.x == 0) {
        s_div[0] = 0.0f;
        s_div[1] = 0.0f;
    }
    __syncthreads();
    const float dfull = s_div[0], dindex = s_div[1];
    for (uint32_t i = threadIdx.x; i < ix.dim; i += blockDim.x) {
        float v = src[i];
        if (q_full_out) q_full_out[(size_t)q * ix.dim + i] = dfull != 0.0f ? __fdiv_rn(v, dfull) : v;
        if (i < ix.dim_index) qi[i] = dindex != 0.0f ? __fdiv_rn(v, dindex) : v;
    }
    __syncthreads();
    const float count_f = __ull2float_rn(ix.count); /* `self.count as f32` */
    for (uint32_t w = threadIdx.x; w < ix.cw; w += blockDim.x) {
        uint64_t word = 0;
        if (w < ix.words) {
            for (uint32_t b = 0; b < 64; b++) {
                uint32_t p = w * 64 + b;
                uint32_t i = p / ix.bits, j = p - i * ix.bits;
                if (i >= ix.dim_index) break;
                uint32_t ones = sbq_count_ones(qi[i], ix.mean[i], ix.bits > 1 ? ix.m2[i] : 0.0f,
                                               count_f, ix.bits);
                if (j < ones) word |= 1ull << b;
            }
        }
        q_codes_out[(size_t)q * ix.cw + w] = word;
    }
}

/* Plain storage layout: amrescan's vector preparation without a quantizer (pg_vector.rs:125-157): the full copy and
 * the copy truncated to dim_index, each cosine-normalised on its own.  One CTA per query. */
__global__ void __launch_bounds__(128) dann_prepare_plain_kernel(uint32_t dim, uint32_t dim_index, int cosine,
                                                                 const float *queries, float *q_full_out,
                                                                 float *q_index_out) {
    DANN_STATIC_SMEM float s_div[2];
    const int q = blockIdx.x;
    const float *src = queries + (size_t)q * dim;
    if (cosine) {
        if (threadIdx.x == 0 || threadIdx.x == 32) {
            const uint32_t len = threadIdx.x == 0 ? dim : dim_index;
            float norm = 0.0f;
            for (uint32_t i = 0; i < len; i++) {
                float v = src[i];
                norm = __fadd_rn(norm, __fmul_rn(v, v));
            }
            s_div[threadIdx.x >> 5] = cosine_divisor_from_norm(norm, len);
        }
    } else if (threadIdx.x == 0) {
        s_div[0] = 0.0f;
        s_div[1] = 0.0f;
    }
    __syncthreads();
    const float dfull = s_div[0], dindex = s_div[1];
    for (uint32_t i = threadIdx.x; i < dim; i += blockDim.x) {
        float v = src[i];
        q_full_out[(size_t)q * dim + i] = dfull != 0.0f ? __fdiv_rn(v, dfull) : v;
        if (i < dim_index) q_index_out[(size_t)q * dim_index + i] = dindex != 0.0f ? __fdiv_rn(v, dindex) : v;
    }
}

/* Plain storage layout, after the rerank kernel: every comparison of the beam search was a full-distance comparison
 * (plain/storage.rs:238,288), so d_full = candidates + reranked rows and d_quantized = 0.  Only launched when the
 * rerank ran (num_dimensions_to_index < num_dimensions, scan.rs:392-403). */
__global__ void dann_plain_stats_kernel(dann_query_stats *stats, int B) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= B) return;
    dann_query_stats st = stats[q];
    st.d_full = st.candidates + st.d_full; /* the rerank kernel left the number of reranked rows here */
    st.d_quantized = 0;
    stats[q] = st;
}

/* ------------------------------------------------------------------------------------ */
/* Stand-alone SBQ distance: out[i] = popcount(code[pair_node[i]] ^ qcode[pair_q[i]])     */
/* (distance_xor_optimized, distance/mod.rs:265-323).  G lanes share one code row with    */
/* 128-bit no-allocate loads; UNR pairs are in flight per lane group.                     */
template <int NCH, int UNR>
__global__ void __launch_bounds__(512) dann_sbq_distance_kernel(const uint64_t *__restrict__ codes,
                                                                uint32_t cw,
                                                                const uint64_t *__restrict__ qcodes,
                                                                const uint32_t *__restrict__ pair_q,
                                                                const uint32_t *__restrict__ pair_node,
                                                                size_t npairs, uint32_t *__restrict__ out,
                                                                uint32_t G, uint32_t Gshift) {
    const uint32_t lane = threadIdx.x & 31, gl = lane & (G - 1);
    const uint32_t nchunks = cw >> 1;
    const size_t groups_per_block = blockDim.x >> Gshift;
    const size_t gid = (size_t)blockIdx.x * groups_per_block + (threadIdx.x >> Gshift);
    const size_t ngroups = (size_t)gridDim.x * groups_per_block;
    for (size_t p0 = gid * UNR; p0 < npairs; p0 += ngroups * UNR) {
        uint32_t nq[UNR], nn[UNR];
#pragma unroll
        for (int u = 0; u < UNR; u++) {
            size_t p = p0 + u;
            bool ok = p < npairs;
            nq[u] = ok ? ldg_stream_u32(pair_q + p) : 0u;
            nn[u] = ok ? ldg_stream_u32(pair_node + p) : 0u;
        }
        ulonglong2 v[UNR][NCH];
#pragma unroll
        for (int u = 0; u < UNR; u++) {
            const ulonglong2 *row = reinterpret_cast<const ulonglong2 *>(codes + (size_t)nn[u] * cw);
#pragma unroll
            for (int i = 0; i < NCH; i++) {
                uint32_t c = gl + i * G;
                v[u][i] = (c < nchunks && p0 + u < npairs) ? ldg_stream_u128(row + c) : make_ulonglong2(0, 0);
            }
        }
#pragma unroll
        for (int u = 0; u < UNR; u++) {
            const ulonglong2 *qrow = reinterpret_cast<const ulonglong2 *>(qcodes + (size_t)nq[u] * cw);
            uint32_t s = 0;
#pragma unroll
            for (int i = 0; i < NCH; i++) {
                uint32_t c = gl + i * G;
                if (c < nchunks) {
                    ulonglong2 qv = __ldg(qrow + c);
                    s += __popcll(v[u][i].x ^ qv.x) + __popcll(v[u][i].y ^ qv.y);
                }
            }
            for (uint32_t o = G >> 1; o > 0; o >>= 1) s += __shfl_xor_sync(DANN_FULL, s, o);
            if (gl == 0 && p0 + u < npairs) out[p0 + u] = s;
        }
    }
}

/* ---- 1-D TMA bulk copy (cp.async.bulk) of one query row into shared memory ---------- */
#ifndef DANN_SIMT_EMU
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void tma_load_1d(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t phase) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(phase)
        : "memory");
}

#endif /* !DANN_SIMT_EMU */

/* Stage query row `src` [n floats] into shared `dst`: TMA bulk copy when the row is a
 * multiple of 16 B and 16-B aligned, plain loads otherwise.  Block-wide. */
__device__ __forceinline__ void stage_query_row(float *dst, const float *src, uint32_t n, uint64_t *bar) {
#ifndef DANN_SIMT_EMU
    const bool tma_ok = (n & 3u) == 0 && ((reinterpret_cast<uintptr_t>(src) & 15u) == 0);
    if (tma_ok) {
        if (threadIdx.x == 0) mbar_init(bar, 1);
        __syncthreads();
        if (threadIdx.x == 0) tma_load_1d(dst, src, n * 4u, bar);
        mbar_wait(bar, 0);
    } else
#else
    (void)bar; /* no TMA under the CPU emulator: the plain-copy branch below */
#endif
    {
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
        __syncthreads();
    }
}

/* out[b*m+i] = distance_fn(vectors[nodes[b*m+i]], q_full[b]) ; one CTA per query */
__global__ void __launch_bounds__(128) dann_full_distance_kernel(IndexView ix, const float *q_full,
                                                                 const uint32_t *nodes, int m, float *out) {
    DANN_DYN_SMEM(dann_smem);
    float *qs = reinterpret_cast<float *>(dann_smem);
    DANN_STATIC_SMEM uint64_t bar;
    const int q = blockIdx.x;
    stage_query_row(qs, q_full + (size_t)q * ix.dim, ix.dim, &bar);
    const uint32_t lane = threadIdx.x & 31, mm = lane & 7, gbase = lane & 24;
    const uint32_t group = threadIdx.x >> 3, ngroups = blockDim.x >> 3;
    const bool vec4 = (ix.dim & 3u) == 0;
    const uint32_t rounds = ((uint32_t)m + ngroups - 1) / ngroups;
    for (uint32_t r = 0; r < rounds; r++) {
        uint32_t it = r * ngroups + group;
        uint32_t node = it < (uint32_t)m ? nodes[(size_t)q * m + it] : DANN_INVALID_NODE;
        const float *x = ix.vectors + (size_t)(node == DANN_INVALID_NODE ? 0 : node) * ix.dim;
        float d = vec4 ? full_distance_group8<true>(ix.distance_type, x, qs, ix.dim, mm, gbase)
                       : full_distance_group8<false>(ix.distance_type, x, qs, ix.dim, mm, gbase);
        if (mm == 0 && it < (uint32_t)m) out[(size_t)q * m + it] = node == DANN_INVALID_NODE ? DANN_NAN_F : d;
    }
}

/* ------------------------------------------------------------------------------------ */
/* next_with_resort (scan.rs:244-305) for the first k rows of one query per CTA:          */
/*   phase 1  get_full_distance_for_resort (sbq/storage.rs:304-328) of every streamed     */
/*            node — 8 lanes per 3-KB row, 128-bit loads, query row staged by TMA;        */
/*   phase 2  the sliding window: a BinaryHeap<ResortData> (min on total_cmp distance,    */
/*            scan.rs:111-117) filled to `rescore`, pop one, refill one, ...              */
/* rescore == 0 bypasses phase 1 and returns the stream order (scan.rs:251-253).          */
struct RerankArgs {
    IndexView ix;
    const float *q_full;        /* [B][dim] */
    const uint32_t *stream;     /* [B][c_target] */
    const uint32_t *stream_len; /* [B] */
    uint32_t c_target, k, rescore;
    uint64_t *out_tid;          /* [B][k] */
    float *out_dist;            /* [B][k] or NULL */
    uint32_t *out_node;         /* [B][k] or NULL */
    uint32_t *out_count;        /* [B] or NULL */
    dann_query_stats *stats;    /* [B] or NULL : d_full is filled here */
};

__global__ void __launch_bounds__(128) dann_rerank_kernel(const RerankArgs a) {
    DANN_DYN_SMEM(dann_smem);
    const IndexView &ix = a.ix;
    float *qs = reinterpret_cast<float *>(dann_smem);                    /* [dim rounded to 4] */
    const uint32_t dim4 = (ix.dim + 3u) & ~3u;
    float *ds = qs + dim4;                                              /* [c_target] */
    uint64_t *hp = reinterpret_cast<uint64_t *>(ds + ((a.c_target + 1u) & ~1u)); /* [rescore] */
    /* the TMA barrier lives in the dynamic window too: with no static shared memory the host's check of a request
     * against the opt-in limit (rerank_smem_bytes) is exact */
    uint64_t *bar = hp + a.rescore;
    const int q = blockIdx.x;
    const uint32_t sl = a.stream_len[q];
    const uint32_t *st = a.stream + (size_t)q * a.c_target;
    uint64_t *otid = a.out_tid + (size_t)q * a.k;

    if (a.rescore == 0) {
        for (uint32_t i = threadIdx.x; i < a.k; i += blockDim.x) {
            bool ok = i < sl;
            uint32_t node = ok ? st[i] : DANN_INVALID_NODE;
            otid[i] = ok ? ix.tids[node] : DANN_INVALID_TID;
            if (a.out_dist) a.out_dist[(size_t)q * a.k + i] = DANN_NAN_F;
            if (a.out_node) a.out_node[(size_t)q * a.k + i] = node;
        }
        if (threadIdx.x == 0 && a.out_count) a.out_count[q] = sl < a.k ? sl : a.k;
        return;
    }

    stage_query_row(qs, a.q_full + (size_t)q * ix.dim, ix.dim, bar);
    {
        const uint32_t lane = threadIdx.x & 31, mm = lane & 7, gbase = lane & 24;
        const uint32_t group = threadIdx.x >> 3, ngroups = blockDim.x >> 3;
        const bool vec4 = (ix.dim & 3u) == 0;
        const uint32_t rounds = (sl + ngroups - 1) / ngroups;
        for (uint32_t r = 0; r < rounds; r++) {
            uint32_t it = r * ngroups + group;
            uint32_t node = it < sl ? st[it] : 0u;
            const float *x = ix.vectors + (size_t)node * ix.dim;
            float d = vec4 ? full_distance_group8<true>(ix.distance_type, x, qs, ix.dim, mm, gbase)
                           : full_distance_group8<false>(ix.distance_type, x, qs, ix.dim, mm, gbase);
            if (mm == 0 && it < sl) ds[it] = d;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        using H = RustHeap<uint64_t, 32>;
        ArrayStore<uint64_t> store{hp};
        uint32_t len = 0, si = 0, rows = 0;
        for (; rows < a.k; rows++) {
            while (len < a.rescore && si < sl) { /* refill: resort_buffer.push(ResortData{..}) */
                H::push(store, len, ((uint64_t)total_ukey(ds[si]) << 32) | si);
                si++;
            }
            if (len == 0) break;
            uint64_t e = H::pop(store, len);
            uint32_t idx = (uint32_t)e, node = st[idx];
            otid[rows] = ix.tids[node];
            if (a.out_dist) a.out_dist[(size_t)q * a.k + rows] = ds[idx];
            if (a.out_node) a.out_node[(size_t)q * a.k + rows] = node;
        }
        if (a.out_count) a.out_count[q] = rows;
        if (a.stats) a.stats[q].d_full = si; /* full_distance_comparisons, scan.rs:258 */
        for (uint32_t i = rows; i < a.k; i++) {
            otid[i] = DANN_INVALID_TID;
            if (a.out_dist) a.out_dist[(size_t)q * a.k + i] = DANN_NAN_F;
            if (a.out_node) a.out_node[(size_t)q * a.k + i] = DANN_INVALID_NODE;
        }
    }
}

/* ------------------------------------------------------------------------------------ */
/* Index load: cosine rows are normalised ONCE with preprocess_cosine's arithmetic        */
/* (sequential sum per row).  Each warp takes 32 rows: coalesced 128-B row segments go     */
/* through a padded shared tile so that every lane runs the sequential chain of one row.  */
__global__ void __launch_bounds__(256) dann_normalize_rows_kernel(float *vectors, uint32_t n, uint32_t dim) {
    DANN_STATIC_SMEM float tile[8][32][33];
    DANN_STATIC_SMEM float divs[8][32];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t nblocks32 = (n + 31) / 32;
    for (uint32_t blk = blockIdx.x * 8 + warp; blk < nblocks32; blk += gridDim.x * 8) {
        const uint32_t row0 = blk * 32;
        float norm = 0.0f;
        for (uint32_t c0 = 0; c0 < dim; c0 += 32) {
            for (uint32_t r = 0; r < 32; r++) {
                uint32_t row = row0 + r, col = c0 + lane;
                tile[warp][r][lane] = (row < n && col < dim) ? vectors[(size_t)row * dim + col] : 0.0f;
            }
            __syncwarp();
            uint32_t lim = dim - c0 < 32 ? dim - c0 : 32;
            for (uint32_t j = 0; j < lim; j++) {
                float v = tile[warp][lane][j];
                norm = __fadd_rn(norm, __fmul_rn(v, v));
            }
            __syncwarp();
        }
        divs[warp][lane] = cosine_divisor_from_norm(norm, dim);
        __syncwarp();
        for (uint32_t r = 0; r < 32; r++) {
            uint32_t row = row0 + r;
            float dv = divs[warp][r];
            if (row < n && dv != 0.0f)
                for (uint32_t col = lane; col < dim; col += 32) {
                    size_t o = (size_t)row * dim + col;
                    vectors[o] = __fdiv_rn(vectors[o], dv);
                }
        }
        __syncwarp();
    }
}

/* dst[n][dst_w] <- src[n][src_w] padded with `fill` (u32 rows: neighbour lists; u64: codes) */
template <typename Tp>
__global__ void dann_pad_rows_kernel(Tp *dst, const Tp *src, size_t n, uint32_t src_w, uint32_t dst_w,
                                     Tp fill) {
    size_t total = n * dst_w;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (size_t)gridDim.x * blockDim.x) {
        size_t r = i / dst_w;
        uint32_t c = (uint32_t)(i - r * dst_w);
        dst[i] = c < src_w ? src[r * src_w + c] : fill;
    }
}

/* Index load: does any neighbour list repeat an id?  (The reference's builder never produces
 * one — add_neighbors dedupes through a HashSet, graph/mod.rs:212-266 — but the scan must not
 * depend on that: when a list does, the search kernel stages the list 32 ids at a time so the
 * FIRST occurrence is the one that inserts.)  One warp per row, lists up to 64 ids. */
__global__ void dann_check_unique_kernel(const uint32_t *nbrs, uint32_t n, uint32_t R, uint32_t Rp,
                                         uint32_t *flag) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < n; row += warps) {
        const uint32_t *r = nbrs + (size_t)row * Rp;
        uint32_t n0 = lane < R ? r[lane] : DANN_INVALID_NODE;
        uint32_t n1 = lane + 32 < R ? r[lane + 32] : DANN_INVALID_NODE;
        unsigned i0 = __ballot_sync(DANN_FULL, n0 == DANN_INVALID_NODE);
        unsigned i1 = __ballot_sync(DANN_FULL, n1 == DANN_INVALID_NODE);
        uint32_t cut0 = i0 ? (uint32_t)(__ffs(i0) - 1) : 32u;
        uint32_t cut1 = i0 ? 0u : (i1 ? (uint32_t)(__ffs(i1) - 1) : 32u);
        bool v0 = lane < cut0, v1 = lane < cut1;
        if (!v0) n0 = DANN_INVALID_NODE;
        if (!v1) n1 = DANN_INVALID_NODE;
        const unsigned mm0 = __match_any_sync(DANN_FULL, n0), mm1 = __match_any_sync(DANN_FULL, n1);
        bool dup = (v0 && __popc(mm0) > 1) || (v1 && __popc(mm1) > 1);
        for (int k = 0; k < 32; k++) {
            uint32_t x = __shfl_sync(DANN_FULL, n1, k);
            dup |= v0 && x != DANN_INVALID_NODE && x == n0;
        }
        if (__any_sync(DANN_FULL, dup) && lane == 0) atomicOr(flag, 1u);
    }
}

/* ------------------------------------------------------------------------------------ */
/* Streaming scan (dann_scan_gettuple): one step of next_with_resort (scan.rs:244-305).       */
/* The rerank window lives in HBM between calls: win[] is the BinaryHeap<ResortData> array,   */
/* entries (total_cmp key of the exact distance << 32) | node.  One thread: push the rows that */
/* just came off the approximate stream, then pop one row for the executor.                  */
struct ScanWindow {
    uint32_t len, d_full;
};
struct ScanRow {
    uint64_t tid;
    uint32_t node, have;
    float dist;
    uint32_t pad;
};
__global__ void dann_scan_resort_kernel(IndexView ix, ScanWindow *w, uint64_t *win, uint32_t rescore,
                                        const uint32_t *new_nodes, const float *new_dist, uint32_t skip,
                                        uint32_t nnew, ScanRow *out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    ScanRow r;
    r.tid = DANN_INVALID_TID;
    r.node = DANN_INVALID_NODE;
    r.have = 0;
    r.dist = DANN_NAN_F;
    r.pad = 0;
    if (rescore == 0) { /* resort_buffer.capacity() == 0: the stream order is the result (scan.rs:251-253) */
        if (nnew > skip) {
            r.node = new_nodes[skip];
            r.tid = ix.tids[r.node];
            r.have = 1;
        }
        *out = r;
        return;
    }
    using H = RustHeap<uint64_t, 32>;
    ArrayStore<uint64_t> store{win};
    uint32_t len = w->len;
    for (uint32_t i = skip; i < nnew; i++) { /* full_distance_comparisons += 1; resort_buffer.push(..) */
        H::push(store, len, ((uint64_t)total_ukey(new_dist[i]) << 32) | new_nodes[i]);
        w->d_full++;
    }
    if (len > 0) {
        uint64_t e = H::pop(store, len);
        uint32_t uk = (uint32_t)(e >> 32) ^ 0x80000000u; /* undo total_ukey: the transform is an involution */
        int32_t b = (int32_t)uk;
        b ^= (int32_t)(((uint32_t)(b >> 31)) >> 1);
        r.node = (uint32_t)e;
        r.dist = __int_as_float(b);
        r.tid = ix.tids[r.node];
        r.have = 1;
    }
    w->len = len;
    *out = r;
}

/* ---- one-synchronisation amgettuple (DANN_SCAN_FUSED=1): the search launch, the exact distances of the rows it
 * appended and the window step are enqueued back to back; the two kernels below read the search's outcome (rows
 * produced, overflow bits) from device memory instead of the host doing so in between, and the last one gathers
 * everything the host needs into one ScanStepOut.  A search that overflowed its workspace leaves the window alone. */
struct ScanStepOut {
    uint32_t overflow, slen;
    dann_query_stats stats;
    ScanRow row;
    ScanWindow win;
};

__global__ void __launch_bounds__(128) dann_scan_distance_kernel(IndexView ix, const float *q_full, const uint32_t *stream,
                                                                 const uint32_t *slen_p, const uint32_t *overflow_p,
                                                                 uint32_t skip, float *out) {
    DANN_DYN_SMEM(dann_smem);
    float *qs = reinterpret_cast<float *>(dann_smem);
    DANN_STATIC_SMEM uint64_t bar;
    if (*overflow_p) return;
    const uint32_t slen = *slen_p;
    if (slen <= skip) return;
    stage_query_row(qs, q_full, ix.dim, &bar);
    const uint32_t lane = threadIdx.x & 31, mm = lane & 7, gbase = lane & 24;
    const uint32_t group = threadIdx.x >> 3, ngroups = blockDim.x >> 3;
    const bool vec4 = (ix.dim & 3u) == 0;
    const uint32_t m = slen - skip, rounds = (m + ngroups - 1) / ngroups;
    for (uint32_t r = 0; r < rounds; r++) {
        const uint32_t it = skip + r * ngroups + group;
        const uint32_t node = it < slen ? stream[it] : 0u;
        const float *x = ix.vectors + (size_t)node * ix.dim;
        const float d = vec4 ? full_distance_group8<true>(ix.distance_type, x, qs, ix.dim, mm, gbase)
                             : full_distance_group8<false>(ix.distance_type, x, qs, ix.dim, mm, gbase);
        if (mm == 0 && it < slen) out[it] = d;
    }
}

__global__ void dann_scan_finish_kernel(IndexView ix, ScanWindow *w, uint64_t *win, uint32_t rescore, const uint32_t *stream,
                                        const float *dist, uint32_t skip, const uint32_t *slen_p, uint32_t slen_fixed,
                                        const uint32_t *overflow_p, const dann_query_stats *stats_p, ScanStepOut *out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    ScanStepOut o;
    o.overflow = overflow_p ? *overflow_p : 0u;
    o.slen = slen_p ? *slen_p : slen_fixed; /* no search this call: nothing new beyond `skip` */
    o.stats = *stats_p;
    o.row.tid = DANN_INVALID_TID;
    o.row.node = DANN_INVALID_NODE;
    o.row.have = 0;
    o.row.dist = DANN_NAN_F;
    o.row.pad = 0;
    if (o.overflow) { /* the host regrows the workspace and replays: the window must not move */
        o.win = *w;
        *out = o;
        return;
    }
    const uint32_t nnew = o.slen;
    if (rescore == 0) {
        if (nnew > skip) {
            o.row.node = stream[skip];
            o.row.tid = ix.tids[o.row.node];
            o.row.have = 1;
        }
        o.win = *w;
        *out = o;
        return;
    }
    using H = RustHeap<uint64_t, 32>;
    ArrayStore<uint64_t> store{win};
    uint32_t len = w->len, dfull = w->d_full;
    for (uint32_t i = skip; i < nnew; i++) {
        H::push(store, len, ((uint64_t)total_ukey(dist[i]) << 32) | stream[i]);
        dfull++;
    }
    if (len > 0) {
        uint64_t e = H::pop(store, len);
        uint32_t uk = (uint32_t)(e >> 32) ^ 0x80000000u;
        int32_t b = (int32_t)uk;
        b ^= (int32_t)(((uint32_t)(b >> 31)) >> 1);
        o.row.node = (uint32_t)e;
        o.row.dist = __int_as_float(b);
        o.row.tid = ix.tids[o.row.node];
        o.row.have = 1;
    }
    w->len = len;
    w->d_full = dfull;
    o.win.len = len;
    o.win.d_full = dfull;
    *out = o;
}

