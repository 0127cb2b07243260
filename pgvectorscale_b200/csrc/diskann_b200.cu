// diskann_b200.cu — C ABI (include/diskann_b200.h) over the sm_100a kernels.
//
// There is NO CPU fallback anywhere in this file: without a CUDA device every entry
// point that computes returns DANN_ERR_NO_DEVICE.  The CPU oracle under oracle/ is
// test infrastructure and is never linked or called from here.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "dann_device.cuh"
#include "dann_kernels.cuh"
#include "dann_search.cuh"
#include "dann_search2.cuh"
#include "dann_search3.cuh"
#include "dann_build.cuh"
#include "dann_plan.h"

#include <cub/device/device_radix_sort.cuh>

/* ------------------------------------------------------------------------------------ */
#define DANN_SMEM_SLACK 128u /* bytes behind every dynamic shared-memory window (see launch_prepare) */

static thread_local std::string g_err;

static int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    try {
        g_err = buf;
    } catch (...) { /* out of memory while recording the message: the code still goes back */
    }
    return code;
}

extern "C" const char *dann_last_error(void) { return g_err.c_str(); }

/* Nothing may propagate out of an extern "C" entry point into the Rust / pgrx caller: every int-returning entry
 * point is a function-try-block that ends with this handler (std::bad_alloc from a host-side vector -> DANN_ERR_OOM). */
#define DANN_CATCH                                                                               \
    catch (const std::bad_alloc &) { return fail(DANN_ERR_OOM, "host allocation failed"); }      \
    catch (...) { return fail(DANN_ERR_STATE, "unexpected C++ exception in the host code"); }

extern "C" int dann_device_count(void) try {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
} DANN_CATCH

#define CK(call)                                                                               \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess) {                                                               \
            if (ix) ix->poisoned = (e_ != cudaErrorMemoryAllocation);                          \
            cudaGetLastError();                                                                \
            return fail(e_ == cudaErrorMemoryAllocation ? DANN_ERR_OOM : DANN_ERR_CUDA,        \
                        "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));    \
        }                                                                                      \
    } while (0)

/* The stream a call that takes DEVICE buffers from its caller runs on.  A caller that names a stream gets exactly that
 * (its buffers must be ready in that stream's order).  A caller that passes NULL gets the index's own
 * cudaStreamNonBlocking stream - which is ordered behind NOTHING the caller did, so the library first makes it wait for
 * everything already submitted to the legacy default stream: what a default-stream kernel or a plain cudaMemcpy of the
 * caller's would have been ordered after.  (Found on B200 in round 2: the fixture quantized rows that torch was still
 * generating on its default stream; until e0113f2 the index load's blocking cudaMemcpy calls had been the accidental
 * barrier.  Work a caller runs on other non-blocking streams needs that stream passed in, or a synchronisation.) */
struct dann_index;
static cudaError_t order_after_default_stream(dann_index *ix, cudaStream_t st);
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    bool fresh = false; /* set when reserve() had to allocate new (uninitialised) memory */
    cudaError_t reserve(size_t bytes) {
        fresh = false;
        if (bytes <= cap) return cudaSuccess;
        fresh = true;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T>
    T *as() const { return reinterpret_cast<T *>(p); }
};

struct dann_index {
    int device = 0;
    IndexView v{};
    std::vector<void *> owned;
    uint64_t hbm_bytes = 0;
    cudaStream_t stream = nullptr;
    std::mutex mu;
    int sm_count = 0;
    size_t smem_optin = 0;
    std::atomic<uint64_t> launches{0}; /* bumped by entry points that do not take `mu` too */
    bool poisoned = false;
    /* per-warp-slot search workspace */
    DevBuf ws_hash, ws_cand, ws_heap, ws_bitmap, ws_ins;
    /* per-batch scratch */
    DevBuf sc_qfull, sc_qcodes, sc_stream, sc_stream_len, sc_stats, sc_qlist, sc_ctl, sc_node;
    /* staging for the host-buffer entry point */
    DevBuf st_queries, st_labels, st_label_off, st_tid, st_dist, st_count, st_stats;
    dann_batch_timing timing{};
    dann_search_plan_info last_plan{};
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_order = nullptr; /* see DANN_DEVICE_INPUT_STREAM */
    uint32_t G = 1, Gshift = 0, NCH = 1;
    uint32_t lists_unique = 0;
    /* plain storage layout (experimental): nodes carry their f32 index vector, no SBQ codes */
    bool plain = false;
    const float *index_vectors = nullptr; /* [n][dim_index] in HBM */
    DevBuf sc_qindex;
};


static cudaError_t order_after_default_stream(dann_index *ix, cudaStream_t st) {
    cudaError_t e = cudaEventRecord(ix->ev_order, cudaStreamLegacy);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(st, ix->ev_order, 0);
    return e;
}
#define DANN_DEVICE_INPUT_STREAM(st, stream)                         \
    cudaStream_t st = (stream) ? (cudaStream_t)(stream) : ix->stream; \
    if (!(stream)) CK(order_after_default_stream(ix, st))

struct dann_scan {
    dann_index *ix = nullptr;
    std::vector<float> query;
    std::vector<int16_t> labels;
    int nlabels = -1;
    int L = 100, rescore = 50;
    bool active = false;
    /* suspended search state in HBM (see SavedScan / dann_search.cuh) */
    DevBuf d_qindex; /* plain layout: the prepared index slice */
    DevBuf d_step;   /* DANN_SCAN_FUSED: one ScanStepOut per amgettuple */
    DevBuf d_query, d_qfull, d_qcodes, d_labels, d_label_off, d_saved, d_heap_sm, d_vis, d_heap_tail, d_cnode, d_set,
        d_ins, d_stream, d_slen, d_stats, d_dist, d_win, d_winst, d_row, d_ctl;
    SearchPlan plan{};
    uint32_t grow = 1;
    uint32_t streamed = 0;  /* rows taken off the approximate stream so far */
    uint32_t win_len = 0;   /* rows sitting in the rerank window */
    bool exhausted = false; /* next() returned None */
    dann_query_stats stats{};
};

/* ------------------------------------------------------------------------------------ */
template <typename Tp>
static cudaError_t upload(dann_index *ix, const Tp *host, size_t count, Tp **out) {
    void *p = nullptr;
    size_t bytes = std::max<size_t>(count * sizeof(Tp), 16);
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return e;
    ix->owned.push_back(p);
    ix->hbm_bytes += bytes;
    /* Every copy of the index goes through ix->stream, the cudaStreamNonBlocking stream its kernels run on.  A plain
     * cudaMemcpy from pageable memory runs on the legacy stream and may return once the data is STAGED, before the DMA
     * has landed; a kernel on a non-blocking stream is not ordered behind it and can read the stale destination
     * (found in round 2: dann_pad_rows_kernel padded rows of whatever the buffer held before - garbage neighbour ids,
     * wrong rows or an illegal access, depending on the process's allocation history). */
    if (host && count) e = cudaMemcpyAsync(p, host, count * sizeof(Tp), cudaMemcpyHostToDevice, ix->stream);
    else e = cudaMemsetAsync(p, 0, bytes, ix->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ix->stream); /* the caller's buffer is borrowed for the call only */
    *out = reinterpret_cast<Tp *>(p);
    return e;
}

/* rows of width src_w -> device rows of width dst_w (padded with `fill`), in row chunks so
 * the temporary never exceeds ~256 MB */
template <typename Tp>
static cudaError_t upload_padded(dann_index *ix, const Tp *host, size_t n, uint32_t src_w, uint32_t dst_w,
                                 Tp fill, Tp **out) {
    void *p = nullptr;
    size_t bytes = std::max<size_t>(n * dst_w * sizeof(Tp), 16);
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return e;
    ix->owned.push_back(p);
    ix->hbm_bytes += bytes;
    *out = reinterpret_cast<Tp *>(p);
    if (n == 0) return cudaSuccess;
    if (src_w == dst_w) {
        e = cudaMemcpyAsync(p, host, n * src_w * sizeof(Tp), cudaMemcpyHostToDevice, ix->stream);
        return e == cudaSuccess ? cudaStreamSynchronize(ix->stream) : e;
    }
    size_t chunk = std::max<size_t>(1, (256ull << 20) / (src_w * sizeof(Tp)));
    void *tmp = nullptr;
    e = cudaMalloc(&tmp, std::min(chunk, n) * src_w * sizeof(Tp));
    if (e != cudaSuccess) return e;
    for (size_t r0 = 0; r0 < n && e == cudaSuccess; r0 += chunk) {
        size_t rows = std::min(chunk, n - r0);
        e = cudaMemcpyAsync(tmp, host + r0 * src_w, rows * src_w * sizeof(Tp), cudaMemcpyHostToDevice, ix->stream);
        if (e != cudaSuccess) break; /* same stream as the kernel below: ordered */
        dann_pad_rows_kernel<Tp><<<1024, 256, 0, ix->stream>>>(reinterpret_cast<Tp *>(p) + r0 * dst_w,
                                                             reinterpret_cast<Tp *>(tmp), rows, src_w,
                                                             dst_w, fill);
        ix->launches++;
        e = cudaStreamSynchronize(ix->stream);
    }
    cudaFree(tmp);
    return e;
}

extern "C" void dann_index_free(dann_index *ix) {
    if (!ix) return;
    cudaSetDevice(ix->device);
    for (void *p : ix->owned) cudaFree(p);
    DevBuf *bufs[] = {&ix->ws_hash, &ix->ws_cand, &ix->ws_heap, &ix->ws_bitmap, &ix->ws_ins, &ix->sc_qfull, &ix->sc_qcodes,
                      &ix->sc_stream, &ix->sc_stream_len, &ix->sc_stats, &ix->sc_qlist, &ix->sc_ctl,
                      &ix->sc_node, &ix->sc_qindex, &ix->st_queries, &ix->st_labels, &ix->st_label_off, &ix->st_tid,
                      &ix->st_dist, &ix->st_count, &ix->st_stats};
    for (DevBuf *b : bufs) b->release();
    for (auto &e : ix->ev)
        if (e) cudaEventDestroy(e);
    if (ix->ev_order) cudaEventDestroy(ix->ev_order);
    if (ix->stream) cudaStreamDestroy(ix->stream);
    cudaGetLastError();
    delete ix;
}

/* Everything the kernels index with comes from the snapshot: reject ids and offsets that would send a
 * gather out of bounds here, on the host, before anything is copied (the reference gets the same guarantee
 * from Postgres' page/item bounds checks, util/page.rs:254-290). */
static int validate_snapshot(const dann_snapshot_desc *s, uint32_t *words_out, bool plain) {
    if (s->dim == 0 || s->dim_index == 0 || s->dim_index > s->dim || s->R == 0 || (!plain && s->bits == 0))
        return fail(DANN_ERR_INVALID_ARG, "bad snapshot geometry");
    uint32_t words = 0;
    if (!plain) {
        uint64_t nb = (uint64_t)s->dim_index * s->bits;
        words = (uint32_t)(nb % 64 == 0 ? nb / 64 : nb / 64 + 1); /* quantize.rs:38-46 */
        if (words != s->words) return fail(DANN_ERR_INVALID_ARG, "words=%u but dim_index*bits needs %u", s->words, words);
    }
    *words_out = words;
    if (s->distance_type < DANN_COSINE || s->distance_type > DANN_IP)
        return fail(DANN_ERR_INVALID_ARG, "unknown distance type %d", s->distance_type);
    if (s->n == DANN_INVALID_NODE) return fail(DANN_ERR_INVALID_ARG, "n collides with the invalid-node sentinel");
    if (plain) { /* build.rs:264-290: what CREATE INDEX rejects for storage_layout = plain */
        if (s->distance_type == DANN_IP) return fail(DANN_ERR_INVALID_ARG, "inner product distance is not supported with plain storage");
        if (s->has_labels) return fail(DANN_ERR_INVALID_ARG, "labeled filtering is not supported with plain storage");
        if (s->dim_index > 2000) return fail(DANN_ERR_INVALID_ARG, "too many dimensions to index with plain storage (max is 2000)");
        if (s->n && (!s->nbrs || !s->heap_tid)) return fail(DANN_ERR_INVALID_ARG, "snapshot arrays missing");
    } else {
        if (s->n && (!s->codes || !s->nbrs || !s->heap_tid || !s->mean))
            return fail(DANN_ERR_INVALID_ARG, "snapshot arrays missing");
        if (s->bits > 1 && s->n && !s->m2) return fail(DANN_ERR_INVALID_ARG, "m2 is required when bits > 1 (sbq/quantize.rs:73-101)");
    }
    if (s->has_labels && s->n && (!s->label_off || (s->label_off[s->n] && !s->labels)))
        return fail(DANN_ERR_INVALID_ARG, "has_labels set but label arrays missing");
    if (s->start_default != DANN_INVALID_NODE && s->start_default >= s->n)
        return fail(DANN_ERR_INVALID_ARG, "start_default out of range");
    if (s->n_start_labels && s->start_labels && s->start_label_nodes) {
        for (uint32_t i = 0; i < s->n_start_labels; i++) {
            if (s->start_label_nodes[i] >= s->n) return fail(DANN_ERR_INVALID_ARG, "start node of label %d out of range", (int)s->start_labels[i]);
            if (i && s->start_labels[i] <= s->start_labels[i - 1]) return fail(DANN_ERR_INVALID_ARG, "start_labels must be strictly ascending");
        }
    }
    for (size_t r = 0; r < s->n; r++) { /* a list ends at its first invalid id (sbq/node.rs:260-273) */
        const uint32_t *row = s->nbrs + r * s->R;
        for (uint32_t j = 0; j < s->R && row[j] != DANN_INVALID_NODE; j++)
            if (row[j] >= s->n) return fail(DANN_ERR_INVALID_ARG, "neighbour %u of node %zu is %u, outside the index (n=%u)", j, r, row[j], s->n);
    }
    if (s->has_labels && s->n) {
        if (s->label_off[0] != 0) return fail(DANN_ERR_INVALID_ARG, "label_off[0] must be 0");
        for (size_t r = 0; r < s->n; r++)
            if (s->label_off[r + 1] < s->label_off[r]) return fail(DANN_ERR_INVALID_ARG, "label_off is not monotone at node %zu", r);
    }
    return DANN_OK;
}

static int index_load_impl(const dann_snapshot_desc *s, const float *index_vectors, int device, dann_index **out) {
    dann_index *ix = nullptr;
    if (!s || !out) return fail(DANN_ERR_INVALID_ARG, "dann_index_load: NULL argument");
    *out = nullptr;
    const bool plain = index_vectors != nullptr;
    uint32_t words = 0;
    int vrc = validate_snapshot(s, &words, plain);
    if (vrc) return vrc;
    int ndev = dann_device_count();
    if (ndev <= 0) return fail(DANN_ERR_NO_DEVICE, "no CUDA device visible (this library has no CPU path)");
    if (device < 0 || device >= ndev) return fail(DANN_ERR_INVALID_ARG, "device %d out of range (%d devices)", device, ndev);

    ix = new (std::nothrow) dann_index();
    if (!ix) return fail(DANN_ERR_OOM, "host allocation failed");
    ix->device = device;
    struct Guard {
        dann_index *&p;
        bool keep = false;
        ~Guard() {
            if (!keep && p) {
                dann_index_free(p);
                p = nullptr;
            }
        }
    } guard{ix};

    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    ix->sm_count = prop.multiProcessorCount;
    ix->smem_optin = prop.sharedMemPerBlockOptin;
    CK(cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking));
    for (auto &e : ix->ev) CK(cudaEventCreate(&e));
    CK(cudaEventCreateWithFlags(&ix->ev_order, cudaEventDisableTiming));

    IndexView &v = ix->v;
    v.n = s->n;
    v.dim = s->dim;
    v.dim_index = s->dim_index;
    v.bits = s->bits;
    v.words = words;
    v.cw = (words + 1u) & ~1u;
    v.R = s->R;
    v.Rp = (s->R + 7u) & ~7u;
    v.distance_type = s->distance_type;
    v.has_labels = s->has_labels ? 1 : 0;
    v.count = s->count;
    v.start_default = s->n ? s->start_default : DANN_INVALID_NODE;
    v.n_start_labels = s->start_labels && s->start_label_nodes ? s->n_start_labels : 0;
    if (!plain && pick_code_mapping(v.cw, &ix->G, &ix->Gshift, &ix->NCH) != 0)
        return fail(DANN_ERR_INVALID_ARG, "SBQ code of %u words is wider than this build supports", words);
    ix->plain = plain;

    float *mean = nullptr, *m2 = nullptr, *vectors = nullptr;
    uint64_t *codes = nullptr, *tids = nullptr;
    uint32_t *nbrs = nullptr, *sln = nullptr, *loff = nullptr;
    int16_t *sl = nullptr, *labs = nullptr;
    if (plain) { /* nodes carry their f32 index vector instead of an SBQ code (plain/node.rs:17-22) */
        float *iv = nullptr;
        CK(upload(ix, index_vectors, (size_t)s->n * s->dim_index, &iv));
        ix->index_vectors = iv;
    } else {
        CK(upload(ix, s->mean, (size_t)s->dim_index, &mean));
        CK(upload(ix, s->bits > 1 ? s->m2 : nullptr, (size_t)s->dim_index, &m2));
        CK(upload_padded<uint64_t>(ix, s->codes, s->n, words, v.cw, 0ull, &codes));
    }
    CK(upload_padded<uint32_t>(ix, s->nbrs, s->n, v.R, v.Rp, DANN_INVALID_NODE, &nbrs));
    CK(upload(ix, s->heap_tid, (size_t)s->n, &tids));
    if (s->vectors) CK(upload(ix, s->vectors, (size_t)s->n * s->dim, &vectors)); /* NULL: supplied later (dann_index_set_vectors) */
    CK(upload(ix, v.n_start_labels ? s->start_labels : nullptr, (size_t)v.n_start_labels, &sl));
    CK(upload(ix, v.n_start_labels ? s->start_label_nodes : nullptr, (size_t)v.n_start_labels, &sln));
    if (v.has_labels && s->n) {
        CK(upload(ix, s->label_off, (size_t)s->n + 1, &loff));
        CK(upload(ix, s->labels, (size_t)s->label_off[s->n], &labs));
    } else {
        v.has_labels = 0;
    }
    v.mean = mean;
    v.m2 = m2;
    v.codes = codes;
    v.nbrs = nbrs;
    v.tids = tids;
    v.vectors = vectors;
    v.start_labels = sl;
    v.start_label_nodes = sln;
    v.label_off = loff;
    v.labels = labs;
    if (s->n && s->R <= 64) {
        uint32_t *flag = nullptr;
        CK(cudaMalloc(&flag, 4));
        ix->owned.push_back(flag);
        CK(cudaMemsetAsync(flag, 0, 4, ix->stream));
        dann_check_unique_kernel<<<ix->sm_count * 8, 256, 0, ix->stream>>>(nbrs, s->n, v.R, v.Rp, flag);
        ix->launches++;
        uint32_t h = 1;
        CK(cudaMemcpyAsync(&h, flag, 4, cudaMemcpyDeviceToHost, ix->stream));
        CK(cudaStreamSynchronize(ix->stream));
        ix->lists_unique = h == 0;
    }
    if (s->distance_type == DANN_COSINE && s->n && vectors) {
        /* rerank reads the heap vector through PgVector::from_datum -> preprocess_cosine
         * (sbq/storage.rs:304-328, pg_vector.rs:153-155); the result only depends on the row,
         * so it is computed once here with the same arithmetic. */
        int blocks = std::min<long long>((s->n + 255) / 256, (long long)ix->sm_count * 8);
        dann_normalize_rows_kernel<<<std::max(blocks, 1), 256, 0, ix->stream>>>(vectors, s->n, s->dim);
        ix->launches++;
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(ix->stream));
    }
    guard.keep = true;
    *out = ix;
    return DANN_OK;
}

extern "C" int dann_index_load(const dann_snapshot_desc *s, int device, dann_index **out) try {
    return index_load_impl(s, nullptr, device, out);
} DANN_CATCH

extern "C" int dann_index_load_plain(const dann_snapshot_desc *s, const float *index_vectors, int device, dann_index **out) try {
    if (!index_vectors && s && s->n) return fail(DANN_ERR_INVALID_ARG, "dann_index_load_plain: NULL index_vectors");
    /* Bit-exact against the oracle under the CPU SIMT emulator, not yet run on hardware: opt-in until it has been. */
    static const float dummy = 0.0f;
    return index_load_impl(s, index_vectors ? index_vectors : &dummy, device, out);
} DANN_CATCH

extern "C" uint64_t dann_index_hbm_bytes(const dann_index *ix) { return ix ? ix->hbm_bytes : 0; }
extern "C" uint64_t dann_kernel_launches(const dann_index *ix) { return ix ? ix->launches.load() : 0; }
extern "C" uint32_t dann_code_stride(const dann_index *ix) { return ix ? ix->v.cw : 0; }

extern "C" int dann_last_search_plan(dann_index *ix, dann_search_plan_info *out) try {
    if (!ix || !out) return fail(DANN_ERR_INVALID_ARG, "dann_last_search_plan: NULL argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    *out = ix->last_plan;
    return DANN_OK;
} DANN_CATCH

extern "C" int dann_last_batch_timing(dann_index *ix, dann_batch_timing *out) try {
    if (!ix || !out) return fail(DANN_ERR_INVALID_ARG, "NULL argument");
    *out = ix->timing;
    return DANN_OK;
} DANN_CATCH

/* ------------------------------------------------------------------------------------ */
static int check_live(dann_index *ix) {
    if (!ix) return fail(DANN_ERR_INVALID_ARG, "NULL index");
    if (ix->poisoned) return fail(DANN_ERR_CUDA, "index handle is poisoned by an earlier CUDA error");
    cudaError_t e = cudaSetDevice(ix->device);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(DANN_ERR_CUDA, "cudaSetDevice(%d): %s", ix->device, cudaGetErrorString(e));
    }
    return DANN_OK;
}

static int launch_prepare(dann_index *ix, const float *d_queries, int B, float *d_q_full, uint64_t *d_q_codes,
                          cudaStream_t st) {
    /* DANN_SMEM_SLACK: ptxas may turn neighbouring shared-memory loads of a loop into one 16-byte load issued BEFORE the
     * loop's bounds test (compute-sanitizer caught dann_prepare_kernel reading 16 bytes past a 28-byte window; on
     * hardware that is a fault whenever it crosses the CTA's allocation), so no dynamic window ends where its data ends */
    size_t smem = (size_t)((ix->v.dim_index + 3u) & ~3u) * sizeof(float) + DANN_SMEM_SLACK;
    if (smem > 48 * 1024)
        CK(cudaFuncSetAttribute(dann_prepare_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dann_prepare_kernel<<<B, 128, smem, st>>>(ix->v, d_queries, B, d_q_full, d_q_codes);
    ix->launches++;
    CK(cudaGetLastError());
    return DANN_OK;
}

extern "C" int dann_prepare_queries(dann_index *ix, const float *d_queries, int B, float *d_q_full,
                                    uint64_t *d_q_codes, void *stream) try {
    int rc = check_live(ix);
    if (rc) return rc;
    if (!d_queries || !d_q_codes || B <= 0) return fail(DANN_ERR_INVALID_ARG, "dann_prepare_queries: bad argument");
    if (ix->plain) return fail(DANN_ERR_STATE, "dann_prepare_queries: a plain-storage index has no quantizer");
    std::lock_guard<std::mutex> lk(ix->mu);
    DANN_DEVICE_INPUT_STREAM(st, stream);
    rc = launch_prepare(ix, d_queries, B, d_q_full, d_q_codes, st);
    if (rc) return rc;
    CK(cudaStreamSynchronize(st));
    return DANN_OK;
} DANN_CATCH

template <int NCH, int UNR>
static void launch_sbq_u(dann_index *ix, const uint64_t *q, const uint32_t *pq, const uint32_t *pn, size_t np,
                         uint32_t *out, cudaStream_t st) {
    const int threads = (int)env_u32("DANN_SBQ_THREADS", 256);
    /* one full wave of resident CTAs (grid-stride loop inside): no partial last wave */
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, dann_sbq_distance_kernel<NCH, UNR>, threads, 0) != cudaSuccess || occ < 1)
        occ = 4;
    int blocks = ix->sm_count * (int)env_u32("DANN_SBQ_BLOCKS_PER_SM", (uint32_t)occ);
    dann_sbq_distance_kernel<NCH, UNR><<<blocks, threads, 0, st>>>(ix->v.codes, ix->v.cw, q, pq, pn, np, out, ix->G,
                                                                  ix->Gshift);
}

template <int NCH>
static void launch_sbq(dann_index *ix, const uint64_t *q, const uint32_t *pq, const uint32_t *pn, size_t np,
                       uint32_t *out, cudaStream_t st) {
    /* pairs in flight per lane group.  Measured on B200 (tools/bench_sbq.py, 192-B codes): UNR=2 -> 40
     * registers, 5.04 TB/s; UNR=4 -> 64 registers, 4.36 TB/s; UNR=8 -> 128 registers, 3.79 TB/s:
     * occupancy beats per-thread memory-level parallelism for these random row gathers. */
    constexpr int UNR = NCH <= 4 ? 2 : 1;
    if (NCH <= 3) {
        switch (env_u32("DANN_SBQ_UNR", UNR)) {
            case 1: return launch_sbq_u<NCH, 1>(ix, q, pq, pn, np, out, st);
            case 4: return launch_sbq_u<NCH, 4>(ix, q, pq, pn, np, out, st);
            case 8: return launch_sbq_u<NCH, 8>(ix, q, pq, pn, np, out, st);
            default: break;
        }
    }
    launch_sbq_u<NCH, UNR>(ix, q, pq, pn, np, out, st);
}

extern "C" int dann_sbq_distance(dann_index *ix, const uint64_t *d_qcodes, const uint32_t *d_pair_q,
                                 const uint32_t *d_pair_node, size_t npairs, uint32_t *d_out, void *stream) try {
    int rc = check_live(ix);
    if (rc) return rc;
    if (!d_qcodes || !d_pair_q || !d_pair_node || !d_out) return fail(DANN_ERR_INVALID_ARG, "dann_sbq_distance: NULL buffer");
    if (ix->plain) return fail(DANN_ERR_STATE, "dann_sbq_distance: a plain-storage index has no SBQ codes");
    if (npairs == 0) return DANN_OK;
    DANN_DEVICE_INPUT_STREAM(st, stream);
    switch (ix->NCH) {
        case 1: launch_sbq<1>(ix, d_qcodes, d_pair_q, d_pair_node, npairs, d_out, st); break;
        case 2: launch_sbq<2>(ix, d_qcodes, d_pair_q, d_pair_node, npairs, d_out, st); break;
        case 3: launch_sbq<3>(ix, d_qcodes, d_pair_q, d_pair_node, npairs, d_out, st); break;
        case 4: launch_sbq<4>(ix, d_qcodes, d_pair_q, d_pair_node, npairs, d_out, st); break;
        default: launch_sbq<8>(ix, d_qcodes, d_pair_q, d_pair_node, npairs, d_out, st); break;
    }
    ix->launches++;
    CK(cudaGetLastError());
    if (!stream) CK(cudaStreamSynchronize(st));
    return DANN_OK;
} DANN_CATCH

extern "C" int dann_full_distance(dann_index *ix, const float *d_q_full, const uint32_t *d_nodes, int B, int m,
                                  float *d_out, void *stream) try {
    int rc = check_live(ix);
    if (rc) return rc;
    if (!d_q_full || !d_nodes || !d_out || B <= 0 || m <= 0) return fail(DANN_ERR_INVALID_ARG, "dann_full_distance: bad argument");
    DANN_DEVICE_INPUT_STREAM(st, stream);
    size_t smem = (size_t)((ix->v.dim + 3u) & ~3u) * sizeof(float) + DANN_SMEM_SLACK;
    if (smem > 48 * 1024)
        CK(cudaFuncSetAttribute(dann_full_distance_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dann_full_distance_kernel<<<B, 128, smem, st>>>(ix->v, d_q_full, d_nodes, m, d_out);
    ix->launches++;
    CK(cudaGetLastError());
    if (!stream) CK(cudaStreamSynchronize(st));
    return DANN_OK;
} DANN_CATCH

/* ------------------------------------------------------------------------------------ */
/* search kernel dispatch                                                                */
typedef void (*search_fn)(const SearchArgs);
template <typename T>
static search_fn pick_search(uint32_t nch) {
    switch (nch) {
        case 1: return dann_search_kernel<T, 1>;
        case 2: return dann_search_kernel<T, 2>;
        case 3: return dann_search_kernel<T, 3>;
        case 4: return dann_search_kernel<T, 4>;
        default: return dann_search_kernel<T, 8>;
    }
}
template <typename T>
static search_fn pick_search2(uint32_t nch) {
    switch (nch) {
        case 1: return dann_search2_kernel<T, 1>;
        case 2: return dann_search2_kernel<T, 2>;
        case 3: return dann_search2_kernel<T, 3>;
        case 4: return dann_search2_kernel<T, 4>;
        default: return dann_search2_kernel<T, 8>;
    }
}
static search_fn pick_kernel(bool pairs, int entry, uint32_t nch, bool plain = false) {
    if (plain) return dann_search_kernel<Ent64, 1, 1>;
    if (pairs) return entry == 0 ? pick_search2<Ent32x21>(nch) : entry == 1 ? pick_search2<Ent32x16>(nch) : pick_search2<Ent64>(nch);
    return entry == 0 ? pick_search<Ent32x21>(nch) : entry == 1 ? pick_search<Ent32x16>(nch) : pick_search<Ent64>(nch);
}

template <typename T, int MAXW>
static search_fn pick_lean_t(uint32_t nch) {
    switch (nch) {
        case 1: return dann_search3_kernel<T, 1, MAXW>;
        case 2: return dann_search3_kernel<T, 2, MAXW>;
        default: return dann_search3_kernel<T, 3, MAXW>; /* the plan offers the lean kernel up to 96 16-byte chunks */
    }
}
/* dann_search3.cuh: 4-byte (key11 | node-or-hash-slot21) or 8-byte (key32 | node32) entries; 32 or 16 resident warps */
static search_fn pick_lean(int entry, uint32_t nch, int maxw) {
    if (maxw <= 16) return entry == 0 ? pick_lean_t<Ent32x21, 16>(nch) : pick_lean_t<Ent64, 16>(nch);
    return entry == 0 ? pick_lean_t<Ent32x21, 32>(nch) : pick_lean_t<Ent64, 32>(nch);
}

static int make_plan(dann_index *ix, uint32_t nq, uint32_t L, uint32_t c_target, uint32_t grow, bool keyed,
                     SearchPlan *p, bool force_single = false, bool allow_lean = false) {
    PlanInputs in;
    in.n = ix->v.n;
    in.R = ix->v.R;
    in.words = ix->v.words;
    in.smem_optin = ix->smem_optin;
    in.sm_count = ix->sm_count;
    in.plain_dim = ix->plain ? ix->v.dim_index : 0;
    in.allow_lean = allow_lean;
    in.ws_budget = 0;
    char err[256];
    int rc = dann_make_plan(in, nq, L, c_target, grow, keyed, p, force_single, err, sizeof err);
    if (rc) return fail(rc, "%s", err);
    if (p->lean) {
        /* the lean plan takes as many query slots as the batch fills; only when that needs more HBM than the
         * workspaces already hold is free memory looked at (cudaMemGetInfo costs about half a millisecond - more than
         * a small batch's other host work) and the slot count cut to what fits: free HBM now plus what the
         * workspaces hold, less a reserve for the batch scratch that is sized after the plan */
        const uint64_t slots = (uint64_t)p->grid * p->W;
        const uint64_t need_heap = slots * p->cand_cap * (uint64_t)p->esize;
        const uint64_t need_set = slots * (p->bitmap_words ? (uint64_t)p->bitmap_words * 4u : (uint64_t)p->hash_cap * 4u);
        const uint64_t held_set = p->bitmap_words ? ix->ws_bitmap.cap : ix->ws_hash.cap;
        if (need_heap > ix->ws_heap.cap || need_set > held_set) {
            size_t fr = 0, tot = 0;
            if (cudaMemGetInfo(&fr, &tot) == cudaSuccess) {
                const uint64_t held = (uint64_t)ix->ws_hash.cap + ix->ws_heap.cap + ix->ws_bitmap.cap + ix->ws_cand.cap + ix->ws_ins.cap;
                const uint64_t reserve = 768ull << 20;
                const uint64_t avail = (uint64_t)fr + held;
                in.ws_budget = avail > reserve ? avail - reserve : 1;
                /* DevBuf::reserve over-allocates by a quarter: plan against 4/5 of the budget */
                in.ws_budget = in.ws_budget / 5 * 4;
                rc = dann_make_plan(in, nq, L, c_target, grow, keyed, p, force_single, err, sizeof err);
                if (rc) return fail(rc, "%s", err);
            }
        }
    }
    return DANN_OK;
}

/* The beam search over B prepared query codes, with the invisible workspace-growth reruns.
 * vis_out != NULL selects build mode (dann_build.cuh). */
static int run_search(dann_index *ix, const uint64_t *d_q_codes, const int16_t *d_labels, const int32_t *d_label_off,
                      int B, uint32_t L, uint32_t c_target, dann_query_stats *d_stats, uint64_t *vis_out,
                      uint32_t *vis_out_len, uint32_t vis_out_cap, cudaStream_t st, const float *d_q_index = nullptr) {
    const IndexView &v = ix->v;
    uint32_t *d_ctl = ix->sc_ctl.as<uint32_t>(); /* [0]=work counter, [1]=overflow bits */
    int rc;
    std::vector<uint32_t> qlist;
    std::vector<dann_query_stats> hstats;
    uint32_t grow = 1;
    uint32_t nq = (uint32_t)B;
    for (int attempt = 0;; attempt++) {
        SearchPlan p;
        rc = make_plan(ix, nq, L, c_target, grow, d_label_off != nullptr, &p, false, vis_out == nullptr);
        if (rc) return rc;
        const size_t slots = (size_t)p.grid * p.W;
        if (!p.bitmap_words) CK(ix->ws_hash.reserve(slots * p.hash_cap * sizeof(uint32_t)));
        if (!p.lean) CK(ix->ws_cand.reserve(slots * p.cand_cap * sizeof(uint32_t))); /* lean entries carry their node */
        CK(ix->ws_heap.reserve(slots * p.cand_cap * (size_t)p.esize));
        if (p.bitmap_words) {
            CK(ix->ws_bitmap.reserve(slots * (size_t)p.bitmap_words * 4));
            if (ix->ws_bitmap.fresh) CK(cudaMemsetAsync(ix->ws_bitmap.p, 0, ix->ws_bitmap.cap, st));
            if (!p.lean) CK(ix->ws_ins.reserve(slots * (size_t)p.ins_cap * 4));
        }
        CK(cudaMemsetAsync(d_ctl, 0, 8, st));
        SearchArgs a;
        a.ix = v;
        a.q_codes = d_q_codes;
        a.q_labels = d_labels;
        a.q_label_off = d_label_off;
        a.qlist = attempt == 0 ? nullptr : ix->sc_qlist.as<uint32_t>();
        a.nq = nq;
        a.L = L;
        a.c_target = c_target;
        a.stream = ix->sc_stream.as<uint32_t>();
        a.stream_len = ix->sc_stream_len.as<uint32_t>();
        a.stats = d_stats;
        a.overflow = d_ctl + 1;
        a.counter = d_ctl;
        a.hash = ix->ws_hash.as<uint32_t>();
        a.hash_cap = p.hash_cap;
        a.bitmap = ix->ws_bitmap.as<uint32_t>();
        a.bitmap_words = p.bitmap_words;
        a.ins_list = ix->ws_ins.as<uint32_t>();
        a.ins_cap = p.ins_cap;
        a.lists_unique = ix->lists_unique;
        a.cand_node = ix->ws_cand.as<uint32_t>();
        a.cand_cap = p.cand_cap;
        a.heap_tail = ix->ws_heap.p;
        a.hs = p.hs;
        a.vcap = p.vcap;
        a.G = ix->G;
        a.Gshift = ix->Gshift;
        a.per_warp_smem = p.per_warp;
        a.saved = nullptr;
        a.saved_heap_sm = nullptr;
        a.saved_vis = nullptr;
        a.build_mode = vis_out ? 1u : 0u;
        a.vis_out = vis_out;
        a.vis_out_len = vis_out_len;
        a.vis_out_cap = vis_out_cap;
        a.hv_flags = env_u32("DANN_HV_FLAGS", 4095);
        a.plain_vectors = ix->index_vectors;
        a.q_index = d_q_index;
        a.plain_dim = ix->plain ? v.dim_index : 0;
        if (attempt == 0) {
            dann_search_plan_info &pi = ix->last_plan;
            pi.kernel = p.lean ? 3u : p.pairs ? 2u : 1u;
            pi.slots_per_sm = p.W;
            pi.grid = p.grid;
            pi.heap_smem = p.hs;
            pi.visited_cap = p.vcap;
            pi.cand_cap = p.cand_cap;
            pi.entry_bytes = p.esize;
            pi.bitmap = p.bitmap_words ? 1u : 0u;
            pi.slot_hbm_bytes = (uint64_t)p.cand_cap * p.esize + (p.bitmap_words ? (uint64_t)p.bitmap_words * 4u : (uint64_t)p.hash_cap * 4u) +
                                (p.lean ? 0u : (uint64_t)p.cand_cap * 4u + (p.bitmap_words ? (uint64_t)p.ins_cap * 4u : 0u));
            pi.smem_per_slot = p.per_warp;
            pi.retries = 0;
        } else {
            ix->last_plan.retries = (uint32_t)attempt;
        }
        search_fn fn = p.lean ? pick_lean(p.entry, ix->NCH, p.maxw) : pick_kernel(p.pairs, p.entry, ix->NCH, ix->plain);
        size_t smem = (size_t)p.per_warp * p.W + DANN_SMEM_SLACK;
        CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        fn<<<p.grid, p.W * (p.pairs ? 64 : 32), smem, st>>>(a);
        ix->launches++;
        CK(cudaGetLastError());
        uint32_t ctl[2] = {0, 0};
        {
            cudaError_t e_ = cudaMemcpyAsync(ctl, d_ctl, 8, cudaMemcpyDeviceToHost, st);
            if (e_ == cudaSuccess) e_ = cudaStreamSynchronize(st);
            if (e_ != cudaSuccess) { /* a faulting search kernel: say which one and how it was planned */
                ix->poisoned = true;
                return fail(DANN_ERR_CUDA, "search kernel %s failed: %s [attempt %d nq %u L %u c_target %u | n %u R %u Rp %u cw %u "
                            "keyed %d | grid %u W %u smem %zu per_warp %u hs %u vcap %u cand_cap %u hash_cap %u bitmap_words %u ins_cap %u entry %d]",
                            p.lean ? "lean" : p.pairs ? "two-warp" : "single-warp", cudaGetErrorString(e_), attempt, nq, L, c_target,
                            v.n, v.R, v.Rp, v.cw, d_label_off != nullptr, p.grid, p.W, smem, p.per_warp, p.hs, p.vcap, p.cand_cap,
                            p.hash_cap, p.bitmap_words, p.ins_cap, p.entry);
            }
        }
        if (ctl[1] == 0) break;
        if (getenv("DANN_DEBUG_STATUS")) fprintf(stderr, "[diskann_b200] search overflow bits 0x%x (attempt %d, plan need=%u vcap=%u)\n", ctl[1], attempt, p.need, p.vcap);
        if (ctl[1] & DANN_ST_INTERNAL) return fail(DANN_ERR_STATE, "internal error: next-node prediction mismatch in the two-warp search kernel");
        /* some queries outgrew their workspace: rerun exactly those with a larger one */
        if (attempt >= 8) return fail(DANN_ERR_CAPACITY, "search workspace still too small after %d growth steps", attempt);
        hstats.resize(B);
        CK(cudaMemcpy(hstats.data(), d_stats, (size_t)B * sizeof(dann_query_stats), cudaMemcpyDeviceToHost));
        qlist.clear();
        for (int b = 0; b < B; b++)
            if (hstats[b].status) qlist.push_back((uint32_t)b);
        nq = (uint32_t)qlist.size();
        CK(cudaMemcpyAsync(ix->sc_qlist.p, qlist.data(), nq * sizeof(uint32_t), cudaMemcpyHostToDevice, st)); /* ordered before the rerun on st */
        CK(cudaStreamSynchronize(st));
        grow *= 2;
        ix->timing.retries++;
    }
    return DANN_OK;
}

/* dann_rerank_kernel's dynamic shared memory: the query row, one f32 per streamed row (even count, so that the window
 * is 8-byte aligned), the rescore window, the TMA barrier (16 B), and the slack.  Both the request check and the launch
 * use it, so that a request the check accepts always launches. */
static size_t rerank_smem_bytes(uint32_t dim, uint32_t c_target, uint32_t rescore) {
    return (size_t)((dim + 3u) & ~3u) * 4 + (size_t)((c_target + 1u) & ~1u) * 4 + (size_t)rescore * 8 + 16 + DANN_SMEM_SLACK;
}

/* B queries, first k rows each.  All pointers are device pointers. */
static int search_batch_device_locked(dann_index *ix, const float *d_queries, const int16_t *d_labels,
                                      const int32_t *d_label_off, int B, int k, int L, int rescore,
                                      uint64_t *d_out_tid, float *d_out_dist, uint32_t *d_out_node,
                                      uint32_t *d_out_count, dann_query_stats *d_out_stats, cudaStream_t st) {
    const IndexView &v = ix->v;
    if (B <= 0 || k <= 0) return fail(DANN_ERR_INVALID_ARG, "B and k must be positive");
    if (L < 1 || L > 10000) return fail(DANN_ERR_INVALID_ARG, "search_list_size %d outside 1..10000 (guc.rs:11-26)", L);
    if (rescore < 0 || rescore > 1000) return fail(DANN_ERR_INVALID_ARG, "rescore %d outside 0..1000 (guc.rs:28-43)", rescore);
    if (!d_queries || !d_out_tid) return fail(DANN_ERR_INVALID_ARG, "NULL query or output buffer");
    if (ix->plain) {
        if (d_label_off) return fail(DANN_ERR_INVALID_ARG, "plain storage does not support label filters (plain/storage.rs:260)");
        /* scan.rs:392-403: a plain index only resorts when it holds fewer dimensions than the heap column */
        if (v.dim == v.dim_index) rescore = 0;
    }
    if (rescore > 0 && v.n && !v.vectors) return fail(DANN_ERR_STATE, "index has no heap vectors yet (dann_index_set_vectors): rescore must be 0");
    /* rows needed from the approximate stream: scan.rs:255-305 */
    const uint32_t c_target = rescore == 0 ? (uint32_t)k : (uint32_t)rescore + (uint32_t)k - 1u;
    const size_t rerank_smem = rerank_smem_bytes(v.dim, c_target, (uint32_t)rescore);
    if (rerank_smem > ix->smem_optin) /* the rerank kernel keeps one f32 per streamed row + the window in shared memory */
        return fail(DANN_ERR_INVALID_ARG, "k=%d rows with rescore=%d need %zu B of shared memory per scan (limit %zu): "
                    "fetch fewer rows per scan", k, rescore, rerank_smem, ix->smem_optin);

    CK(ix->sc_qfull.reserve((size_t)B * v.dim * sizeof(float)));
    CK(ix->sc_qcodes.reserve((size_t)B * v.cw * sizeof(uint64_t)));
    CK(ix->sc_stream.reserve((size_t)B * c_target * sizeof(uint32_t)));
    CK(ix->sc_stream_len.reserve((size_t)B * sizeof(uint32_t)));
    CK(ix->sc_stats.reserve((size_t)B * sizeof(dann_query_stats)));
    CK(ix->sc_qlist.reserve((size_t)B * sizeof(uint32_t)));
    CK(ix->sc_ctl.reserve(64));
    dann_query_stats *d_stats = d_out_stats ? d_out_stats : ix->sc_stats.as<dann_query_stats>();

    ix->timing = dann_batch_timing{};
    CK(cudaEventRecord(ix->ev[0], st));
    int rc;
    if (ix->plain) {
        CK(ix->sc_qindex.reserve((size_t)B * v.dim_index * sizeof(float)));
        dann_prepare_plain_kernel<<<B, 128, 0, st>>>(v.dim, v.dim_index, v.distance_type == DANN_COSINE, d_queries,
                                                    ix->sc_qfull.as<float>(), ix->sc_qindex.as<float>());
        ix->launches++;
        CK(cudaGetLastError());
    } else {
        rc = launch_prepare(ix, d_queries, B, ix->sc_qfull.as<float>(), ix->sc_qcodes.as<uint64_t>(), st);
        if (rc) return rc;
    }
    CK(cudaEventRecord(ix->ev[1], st));

    rc = run_search(ix, ix->sc_qcodes.as<uint64_t>(), d_labels, d_label_off, B, (uint32_t)L, c_target, d_stats, nullptr,
                    nullptr, 0, st, ix->sc_qindex.as<float>());
    if (rc) return rc;
    CK(cudaEventRecord(ix->ev[2], st));

    RerankArgs r;
    r.ix = v;
    r.q_full = ix->sc_qfull.as<float>();
    r.stream = ix->sc_stream.as<uint32_t>();
    r.stream_len = ix->sc_stream_len.as<uint32_t>();
    r.c_target = c_target;
    r.k = (uint32_t)k;
    r.rescore = (uint32_t)rescore;
    r.out_tid = d_out_tid;
    r.out_dist = d_out_dist;
    r.out_node = d_out_node;
    r.out_count = d_out_count;
    r.stats = d_stats;
    if (rerank_smem > 48 * 1024)
        CK(cudaFuncSetAttribute(dann_rerank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rerank_smem));
    dann_rerank_kernel<<<B, 128, rerank_smem, st>>>(r);
    ix->launches++;
    CK(cudaGetLastError());
    if (ix->plain && rescore > 0) {
        dann_plain_stats_kernel<<<(B + 127) / 128, 128, 0, st>>>(d_stats, B);
        ix->launches++;
        CK(cudaGetLastError());
    }
    CK(cudaEventRecord(ix->ev[3], st));
    CK(cudaStreamSynchronize(st));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, ix->ev[0], ix->ev[1]));
    ix->timing.prepare_ms = ms;
    CK(cudaEventElapsedTime(&ms, ix->ev[1], ix->ev[2]));
    ix->timing.search_ms = ms;
    CK(cudaEventElapsedTime(&ms, ix->ev[2], ix->ev[3]));
    ix->timing.rerank_ms = ms;
    ix->timing.resort_ms = 0.0f; /* the rerank window runs inside the rerank kernel */
    CK(cudaEventElapsedTime(&ms, ix->ev[0], ix->ev[3]));
    ix->timing.total_ms = ms;
    return DANN_OK;
}

extern "C" int dann_search_batch_device(dann_index *ix, const float *d_queries, const int16_t *d_labels,
                                        const int32_t *d_label_off, int B, int k, int search_list_size,
                                        int rescore, uint64_t *d_out_tid, float *d_out_dist,
                                        uint32_t *d_out_count, dann_query_stats *d_out_stats, void *stream) try {
    int rc = check_live(ix);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ix->mu);
    DANN_DEVICE_INPUT_STREAM(st, stream);
    return search_batch_device_locked(ix, d_queries, d_labels, d_label_off, B, k, search_list_size, rescore,
                                      d_out_tid, d_out_dist, nullptr, d_out_count, d_out_stats, st);
} DANN_CATCH

/* host-buffer batch with optional node ids (used by the scan operator too) */
static int search_batch_host(dann_index *ix, const float *queries, const int16_t *labels,
                             const int32_t *label_off, int B, int k, int L, int rescore, uint64_t *out_tid,
                             float *out_dist, uint32_t *out_node, uint32_t *out_count,
                             dann_query_stats *out_stats) {
    int rc = check_live(ix);
    if (rc) return rc;
    if (B <= 0 || k <= 0 || !queries || !out_tid) return fail(DANN_ERR_INVALID_ARG, "dann_search_batch: bad argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    cudaStream_t st = ix->stream;
    const IndexView &v = ix->v;
    const size_t nk = (size_t)B * k;
    CK(ix->st_queries.reserve((size_t)B * v.dim * sizeof(float)));
    CK(ix->st_tid.reserve(nk * sizeof(uint64_t)));
    CK(ix->st_dist.reserve(nk * sizeof(float)));
    CK(ix->sc_node.reserve(nk * sizeof(uint32_t)));
    CK(ix->st_count.reserve((size_t)B * sizeof(uint32_t)));
    CK(ix->st_stats.reserve((size_t)B * sizeof(dann_query_stats)));
    CK(cudaMemcpyAsync(ix->st_queries.p, queries, (size_t)B * v.dim * sizeof(float), cudaMemcpyHostToDevice, st));
    const int16_t *d_lab = nullptr;
    const int32_t *d_off = nullptr;
    std::vector<int16_t> nl;
    std::vector<int32_t> no;
    if (label_off) {
        /* LabelSet::from(Vec): sort_unstable + dedup per query (labels/mod.rs:30-37) */
        no.resize((size_t)B + 1);
        no[0] = 0;
        if (label_off[0] < 0) return fail(DANN_ERR_INVALID_ARG, "label_off[0] is negative");
        if (label_off[B] > label_off[0] && !labels) return fail(DANN_ERR_INVALID_ARG, "labels is NULL but label_off describes a non-empty key");
        for (int b = 0; b < B; b++) {
            int32_t o0 = label_off[b], o1 = label_off[b + 1];
            if (o1 < o0) return fail(DANN_ERR_INVALID_ARG, "label_off is not monotone");
            size_t s0 = nl.size();
            if (o1 > o0) nl.insert(nl.end(), labels + o0, labels + o1);
            std::sort(nl.begin() + s0, nl.end());
            nl.erase(std::unique(nl.begin() + s0, nl.end()), nl.end());
            no[b + 1] = (int32_t)nl.size();
        }
        CK(ix->st_labels.reserve(std::max<size_t>(nl.size(), 1) * sizeof(int16_t)));
        CK(ix->st_label_off.reserve(no.size() * sizeof(int32_t)));
        if (!nl.empty()) CK(cudaMemcpyAsync(ix->st_labels.p, nl.data(), nl.size() * sizeof(int16_t), cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ix->st_label_off.p, no.data(), no.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        d_lab = ix->st_labels.as<int16_t>();
        d_off = ix->st_label_off.as<int32_t>();
    }
    rc = search_batch_device_locked(ix, ix->st_queries.as<float>(), d_lab, d_off, B, k, L, rescore,
                                    ix->st_tid.as<uint64_t>(), ix->st_dist.as<float>(), ix->sc_node.as<uint32_t>(),
                                    ix->st_count.as<uint32_t>(), ix->st_stats.as<dann_query_stats>(), st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out_tid, ix->st_tid.p, nk * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    if (out_dist) CK(cudaMemcpyAsync(out_dist, ix->st_dist.p, nk * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (out_node) CK(cudaMemcpyAsync(out_node, ix->sc_node.p, nk * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    if (out_count) CK(cudaMemcpyAsync(out_count, ix->st_count.p, (size_t)B * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    if (out_stats) CK(cudaMemcpyAsync(out_stats, ix->st_stats.p, (size_t)B * sizeof(dann_query_stats), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return DANN_OK;
}

extern "C" int dann_search_batch(dann_index *ix, const float *queries, const int16_t *labels,
                                 const int32_t *label_off, int B, int k, int search_list_size, int rescore,
                                 uint64_t *out_tid, float *out_dist, uint32_t *out_count,
                                 dann_query_stats *out_stats) try {
    return search_batch_host(ix, queries, labels, label_off, B, k, search_list_size, rescore, out_tid, out_dist,
                             nullptr, out_count, out_stats);
} DANN_CATCH

/* ------------------------------------------------------------------------------------ */
/* index construction (SURVEY.md §8f row 1) — see dann_build.cuh                            */

extern "C" int dann_index_set_vectors(dann_index *ix, const float *vectors) try {
    int rc = check_live(ix);
    if (rc) return rc;
    if (!vectors) return fail(DANN_ERR_INVALID_ARG, "dann_index_set_vectors: NULL vectors");
    std::lock_guard<std::mutex> lk(ix->mu);
    IndexView &v = ix->v;
    if (!v.n) return DANN_OK;
    float *d = const_cast<float *>(v.vectors);
    if (!d) {
        void *p = nullptr;
        size_t bytes = (size_t)v.n * v.dim * sizeof(float);
        CK(cudaMalloc(&p, bytes));
        ix->owned.push_back(p);
        ix->hbm_bytes += bytes;
        d = reinterpret_cast<float *>(p);
        v.vectors = d;
    }
    CK(cudaMemcpyAsync(d, vectors, (size_t)v.n * v.dim * sizeof(float), cudaMemcpyHostToDevice, ix->stream)); /* ordered before the normalisation */
    CK(cudaStreamSynchronize(ix->stream));
    if (v.distance_type == DANN_COSINE) {
        int blocks = std::min<long long>((v.n + 255) / 256, (long long)ix->sm_count * 8);
        dann_normalize_rows_kernel<<<std::max(blocks, 1), 256, 0, ix->stream>>>(d, v.n, v.dim);
        ix->launches++;
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(ix->stream));
    }
    return DANN_OK;
} DANN_CATCH

extern "C" int dann_index_set_vectors_device(dann_index *ix, float *d_vectors) try {
    int rc = check_live(ix);
    if (rc) return rc;
    if (!d_vectors) return fail(DANN_ERR_INVALID_ARG, "dann_index_set_vectors_device: NULL vectors");
    std::lock_guard<std::mutex> lk(ix->mu);
    IndexView &v = ix->v;
    if (!v.n) return DANN_OK;
    if (v.vectors) return fail(DANN_ERR_STATE, "dann_index_set_vectors_device: the index already owns a vector array");
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, d_vectors) != cudaSuccess || at.type != cudaMemoryTypeDevice || at.device != ix->device) {
        cudaGetLastError();
        return fail(DANN_ERR_INVALID_ARG, "dann_index_set_vectors_device: not a device pointer on device %d", ix->device);
    }
    v.vectors = d_vectors; /* borrowed: not in ix->owned */
    ix->hbm_bytes += (uint64_t)v.n * v.dim * sizeof(float);
    CK(order_after_default_stream(ix, ix->stream)); /* the caller's rows: see DANN_DEVICE_INPUT_STREAM */
    if (v.distance_type == DANN_COSINE) {
        int blocks = std::min<long long>((v.n + 255) / 256, (long long)ix->sm_count * 8);
        dann_normalize_rows_kernel<<<std::max(blocks, 1), 256, 0, ix->stream>>>(d_vectors, v.n, v.dim);
        ix->launches++;
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(ix->stream));
    }
    return DANN_OK;
} DANN_CATCH

extern "C" int dann_index_download_nbrs(dann_index *ix, uint32_t *out) try {
    int rc = check_live(ix);
    if (rc) return rc;
    if (!out) return fail(DANN_ERR_INVALID_ARG, "dann_index_download_nbrs: NULL buffer");
    std::lock_guard<std::mutex> lk(ix->mu);
    const IndexView &v = ix->v;
    if (!v.n) return DANN_OK;
    CK(cudaMemcpy2D(out, (size_t)v.R * 4, v.nbrs, (size_t)v.Rp * 4, (size_t)v.R * 4, v.n, cudaMemcpyDeviceToHost));
    return DANN_OK;
} DANN_CATCH

extern "C" int dann_build_graph(dann_index *ix, int num_neighbors, int search_list_size, float max_alpha,
                                uint32_t max_batch, dann_build_stats *out) try {
    int rc = check_live(ix);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ix->mu);
    IndexView &v = ix->v;
    if (ix->plain) return fail(DANN_ERR_STATE, "dann_build_graph builds over SBQ codes: not available for a plain-storage index");
    if (v.R != DANN_BUILD_SLACK || v.Rp != DANN_BUILD_SLACK)
        return fail(DANN_ERR_INVALID_ARG, "dann_build_graph needs an index loaded with R == %u neighbour slots", DANN_BUILD_SLACK);
    if (num_neighbors < 1 || num_neighbors > (int)DANN_BUILD_SLACK) return fail(DANN_ERR_INVALID_ARG, "num_neighbors must be 1..%u", DANN_BUILD_SLACK);
    if (search_list_size < 1 || search_list_size > 1000) return fail(DANN_ERR_INVALID_ARG, "build search_list_size must be 1..1000");
    if (v.has_labels && v.n_start_labels == 0)
        return fail(DANN_ERR_INVALID_ARG, "a labeled build needs the per-label start nodes (first node carrying each label)");
    if (v.n == 0) return DANN_OK;
    if (v.start_default != 0) return fail(DANN_ERR_INVALID_ARG, "dann_build_graph inserts in id order: start_default must be 0");
    if (max_batch == 0) max_batch = 1u << 20;
    cudaStream_t st = ix->stream;
    const uint32_t n = v.n;
    const uint32_t vis_cap = 2 * DANN_BUILD_CMAX;
    const uint32_t mb = std::min<uint32_t>(max_batch, n);
    /* the prune kernel stages DANN_BUILD_CMAX candidate codes per warp in shared memory: a code too wide for one warp is
     * refused here, before the neighbour lists are cleared, so that a refused build leaves the index as it was */
    const uint32_t cws = v.cw | 1u;
    const size_t pw = ((size_t)DANN_BUILD_CMAX * 8 + (size_t)DANN_BUILD_CMAX * cws * 8 + DANN_BUILD_CMAX * 4 +
                       DANN_BUILD_SLACK * 4 + DANN_BUILD_SLACK * 2 + 15) & ~(size_t)15;
    const size_t budget = ix->smem_optin > 1024 ? ix->smem_optin - 1024 : ix->smem_optin;
    const int bw = (int)std::min<size_t>(8, budget / pw);
    if (bw < 1) return fail(DANN_ERR_CAPACITY, "SBQ code of %u words is too wide for the prune kernel's shared memory", v.words);

    DevBuf b_dist, b_deg, b_vis, b_vlen, b_k0, b_k1, b_v0, b_v1, b_heads, b_tmp, b_stream, b_slen, b_stats;
    struct Cleanup {
        std::vector<DevBuf *> v;
        ~Cleanup() {
            for (DevBuf *b : v) b->release();
        }
    } cleanup{{&b_dist, &b_deg, &b_vis, &b_vlen, &b_k0, &b_k1, &b_v0, &b_v1, &b_heads, &b_tmp, &b_stream, &b_slen, &b_stats}};
    const size_t ntrip = (size_t)mb * DANN_BUILD_SLACK;
    CK(b_dist.reserve((size_t)n * DANN_BUILD_SLACK * sizeof(uint16_t)));
    CK(b_deg.reserve((size_t)n));
    CK(b_vis.reserve((size_t)mb * vis_cap * sizeof(uint64_t)));
    CK(b_vlen.reserve((size_t)mb * 4));
    CK(b_k0.reserve(ntrip * 8));
    CK(b_k1.reserve(ntrip * 8));
    CK(b_v0.reserve(ntrip * 4));
    CK(b_v1.reserve(ntrip * 4));
    CK(b_heads.reserve(ntrip * 4 + 64));
    CK(ix->sc_stream.reserve((size_t)mb * 4)); /* run_search writes stream_len / stats even in build mode */
    CK(ix->sc_stream_len.reserve((size_t)mb * 4));
    CK(b_stats.reserve((size_t)mb * sizeof(dann_query_stats)));
    CK(ix->sc_qlist.reserve((size_t)mb * sizeof(uint32_t)));
    CK(ix->sc_ctl.reserve(64));
    size_t tmp_bytes = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, b_k0.as<uint64_t>(), b_k1.as<uint64_t>(), b_v0.as<uint32_t>(),
                                       b_v1.as<uint32_t>(), ntrip, 16, 64, st));
    CK(b_tmp.reserve(tmp_bytes));
    uint32_t *nbrs = const_cast<uint32_t *>(v.nbrs);
    CK(cudaMemsetAsync(nbrs, 0xFF, (size_t)n * DANN_BUILD_SLACK * 4, st));
    CK(cudaMemsetAsync(b_deg.p, 0, n, st));

    BuildArgs ba;
    ba.codes = v.codes;
    ba.cw = v.cw;
    ba.cws = cws;
    ba.n = n;
    ba.nbrs = nbrs;
    ba.nbr_dist = b_dist.as<uint16_t>();
    ba.deg = b_deg.as<uint8_t>();
    ba.R = (uint32_t)num_neighbors;
    ba.limit = std::min<uint32_t>(DANN_BUILD_SLACK, (uint32_t)std::ceil((double)num_neighbors * 1.3));
    ba.max_alpha = max_alpha;
    ba.label_off = v.has_labels ? v.label_off : nullptr;
    ba.labels = v.has_labels ? v.labels : nullptr;
    ba.per_warp_smem = (uint32_t)pw;
    const size_t bsmem = pw * bw + DANN_SMEM_SLACK;
    CK(cudaFuncSetAttribute(dann_build_prune_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem));
    CK(cudaFuncSetAttribute(dann_build_backlink_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem));
    CK(cudaFuncSetAttribute(dann_build_finalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem));
    const int bgrid = ix->sm_count * std::max<int>(1, (int)(budget / bsmem));

    dann_build_stats bs{};
    cudaEvent_t e[5];
    for (auto &x : e) CK(cudaEventCreate(&x));
    struct EvGuard {
        cudaEvent_t *e;
        ~EvGuard() {
            for (int i = 0; i < 5; i++) cudaEventDestroy(e[i]);
        }
    } evg{e};
    const uint32_t lists_unique_saved = ix->lists_unique;
    ix->lists_unique = 1; /* the builder never repeats an id within a list */
    const bool verbose = getenv("DANN_BUILD_VERBOSE") != nullptr;
    /* node 0 is the entry point (the reference's first inserted node); everything else arrives in
     * batches that grow with the graph (at most 1/16 of it) up to max_batch */
    for (uint32_t lo = 1; lo < n;) {
        uint32_t m = std::max<uint32_t>(1, lo / 16);
        m = std::min(std::min(m, mb), n - lo);
        /* graph/mod.rs:637-660: a labeled node is inserted twice — first from the label start nodes with the
         * label filter on, then from the default start node without it; the second pass merges with the
         * neighbours the first one left (add_neighbors) */
        uint32_t nheads = 0;
        for (int pass = v.has_labels ? 0 : 1; pass < 2; pass++) {
            const int16_t *qlab = pass == 0 ? v.labels : nullptr;
            const int32_t *qoff = pass == 0 ? reinterpret_cast<const int32_t *>(v.label_off + lo) : nullptr;
            CK(cudaEventRecord(e[0], st));
            rc = run_search(ix, v.codes + (size_t)lo * v.cw, qlab, qoff, (int)m, (uint32_t)search_list_size, 1u,
                            b_stats.as<dann_query_stats>(), b_vis.as<uint64_t>(), b_vlen.as<uint32_t>(), vis_cap, st);
            if (rc) {
                ix->lists_unique = lists_unique_saved;
                return rc;
            }
            CK(cudaEventRecord(e[1], st));
            dann_build_prune_kernel<<<bgrid, bw * 32, bsmem, st>>>(ba, lo, m, b_vis.as<uint64_t>(), b_vlen.as<uint32_t>(),
                                                                  vis_cap, b_k0.as<uint64_t>(), b_v0.as<uint32_t>());
            ix->launches++;
            CK(cudaGetLastError());
            CK(cudaEventRecord(e[2], st));
            const size_t cnt = (size_t)m * DANN_BUILD_SLACK;
            size_t tb = b_tmp.cap;
            CK(cub::DeviceRadixSort::SortPairs(b_tmp.p, tb, b_k0.as<uint64_t>(), b_k1.as<uint64_t>(), b_v0.as<uint32_t>(),
                                               b_v1.as<uint32_t>(), cnt, 16, 64, st));
            uint32_t *d_nheads = b_heads.as<uint32_t>() + ntrip;
            CK(cudaMemsetAsync(d_nheads, 0, 4, st));
            dann_build_heads_kernel<<<ix->sm_count * 4, 256, 0, st>>>(b_k1.as<uint64_t>(), cnt, b_heads.as<uint32_t>(), d_nheads);
            ix->launches += 2;
            CK(cudaMemcpyAsync(&nheads, d_nheads, 4, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            CK(cudaEventRecord(e[3], st));
            if (nheads) {
                dann_build_backlink_kernel<<<bgrid, bw * 32, bsmem, st>>>(ba, b_k1.as<uint64_t>(), b_v1.as<uint32_t>(), cnt,
                                                                         b_heads.as<uint32_t>(), nheads);
                ix->launches++;
                CK(cudaGetLastError());
            }
            CK(cudaEventRecord(e[4], st));
            CK(cudaStreamSynchronize(st));
            float ms;
            CK(cudaEventElapsedTime(&ms, e[0], e[1]));
            bs.search_ms += ms;
            CK(cudaEventElapsedTime(&ms, e[1], e[2]));
            bs.prune_ms += ms;
            CK(cudaEventElapsedTime(&ms, e[2], e[3]));
            bs.sort_ms += ms;
            CK(cudaEventElapsedTime(&ms, e[3], e[4]));
            bs.backlink_ms += ms;
        }
        bs.batches++;
        if (verbose && (bs.batches % 16 == 0 || lo + m >= n))
            fprintf(stderr, "[dann_build] batch %u: nodes %u..%u (m=%u, %u destinations) search %.0f prune %.0f sort %.0f backlink %.0f ms\n",
                    bs.batches, lo, lo + m, m, nheads, bs.search_ms, bs.prune_ms, bs.sort_ms, bs.backlink_ms);
        lo += m;
    }
    dann_build_finalize_kernel<<<bgrid, bw * 32, bsmem, st>>>(ba);
    ix->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    if (env_u32("DANN_BUILD_RESCUE", 0) == 1 && !v.has_labels) { /* opt-in: see dann_build.cuh "in-edge rescue" */
        DevBuf b_in, b_claim;
        struct Rel {
            DevBuf *a, *b;
            ~Rel() {
                a->release();
                b->release();
            }
        } rel{&b_in, &b_claim};
        CK(b_in.reserve((size_t)n * 4));
        CK(b_claim.reserve((size_t)n * 4 + 4));
        uint32_t *d_claim = b_claim.as<uint32_t>(), *d_resc = d_claim + n;
        for (int round = 0; round < 16; round++) {
            CK(cudaMemsetAsync(b_in.p, 0, (size_t)n * 4, st));
            CK(cudaMemsetAsync(d_claim, 0, (size_t)n * 4 + 4, st));
            dann_build_mark_indegree_kernel<<<ix->sm_count * 8, 256, 0, st>>>(nbrs, b_deg.as<uint8_t>(), n, b_in.as<uint32_t>());
            dann_build_rescue_kernel<<<ix->sm_count * 4, 256, 0, st>>>(nbrs, b_deg.as<uint8_t>(), n, (uint32_t)num_neighbors,
                                                                      b_in.as<uint32_t>(), d_claim, d_resc);
            dann_build_rescue_degrees_kernel<<<ix->sm_count * 4, 256, 0, st>>>(b_deg.as<uint8_t>(), d_claim, n, (uint32_t)num_neighbors);
            ix->launches += 3;
            CK(cudaGetLastError());
            uint32_t resc = 0;
            CK(cudaMemcpyAsync(&resc, d_resc, 4, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            if (verbose) fprintf(stderr, "[dann_build] rescue round %d: %u nodes had no in-edge\n", round, resc);
            if (!resc) break;
        }
    }
    bs.total_ms = bs.search_ms + bs.prune_ms + bs.sort_ms + bs.backlink_ms;
    /* average degree */
    {
        std::vector<uint8_t> hdeg(std::min<uint32_t>(n, 1u << 20));
        CK(cudaMemcpy(hdeg.data(), b_deg.p, hdeg.size(), cudaMemcpyDeviceToHost));
        double sdeg = 0;
        for (uint8_t d : hdeg) sdeg += d;
        bs.avg_degree = sdeg / (double)hdeg.size();
    }
    if (out) *out = bs;
    return DANN_OK;
} DANN_CATCH

/* ------------------------------------------------------------------------------------ */
/* scan operator: ambeginscan / amrescan / amgettuple / amendscan (scan.rs:309-476)       */

extern "C" int dann_scan_begin(dann_index *ix, dann_scan **out) try {
    if (!ix || !out) return fail(DANN_ERR_INVALID_ARG, "dann_scan_begin: NULL argument");
    dann_scan *sc = new (std::nothrow) dann_scan();
    if (!sc) return fail(DANN_ERR_OOM, "host allocation failed");
    sc->ix = ix;
    *out = sc;
    return DANN_OK;
} DANN_CATCH

static void scan_release(dann_scan *sc) {
    DevBuf *bufs[] = {&sc->d_qindex, &sc->d_step, &sc->d_query, &sc->d_qfull, &sc->d_qcodes, &sc->d_labels, &sc->d_label_off, &sc->d_saved,
                      &sc->d_heap_sm, &sc->d_vis, &sc->d_heap_tail, &sc->d_cnode, &sc->d_set, &sc->d_ins, &sc->d_stream,
                      &sc->d_slen, &sc->d_stats, &sc->d_dist, &sc->d_win, &sc->d_winst, &sc->d_row, &sc->d_ctl};
    for (DevBuf *b : bufs) b->release();
}

/* (re)allocate the scan's private workspace for the current plan and reset the search state */
static int scan_reset_search(dann_scan *sc) {
    dann_index *ix = sc->ix;
    cudaStream_t st = ix->stream;
    SearchPlan &p = sc->plan;
    int rc = make_plan(ix, 1, (uint32_t)sc->L, (uint32_t)sc->rescore + 64u, sc->grow, sc->nlabels >= 0, &p, true);
    if (rc) return rc;
    CK(sc->d_saved.reserve(sizeof(SavedScan)));
    CK(sc->d_heap_sm.reserve((size_t)p.hs * p.esize + 16));
    CK(sc->d_vis.reserve((size_t)p.vcap * 8));
    CK(sc->d_heap_tail.reserve((size_t)p.cand_cap * p.esize));
    CK(sc->d_cnode.reserve((size_t)p.cand_cap * 4));
    CK(sc->d_ins.reserve((size_t)p.ins_cap * 4));
    if (p.bitmap_words) {
        CK(sc->d_set.reserve((size_t)p.bitmap_words * 4));
        CK(cudaMemsetAsync(sc->d_set.p, 0, (size_t)p.bitmap_words * 4, st));
    } else {
        CK(sc->d_set.reserve((size_t)p.hash_cap * 4));
    }
    CK(cudaMemsetAsync(sc->d_saved.p, 0, sizeof(SavedScan), st));
    return DANN_OK;
}

extern "C" int dann_scan_rescan(dann_scan *sc, const float *query, const int16_t *labels, int nlabels,
                                int search_list_size, int rescore) try {
    if (!sc) return fail(DANN_ERR_INVALID_ARG, "dann_scan_rescan: NULL scan");
    if (search_list_size < 1 || search_list_size > 10000) return fail(DANN_ERR_INVALID_ARG, "search_list_size %d outside 1..10000", search_list_size);
    if (rescore < 0 || rescore > 1000) return fail(DANN_ERR_INVALID_ARG, "rescore %d outside 0..1000", rescore);
    if (nlabels > 0 && !labels) return fail(DANN_ERR_INVALID_ARG, "labels is NULL but nlabels > 0");
    dann_index *ix = sc->ix;
    int rc = check_live(ix);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ix->mu);
    const IndexView &v = ix->v;
    if (ix->plain) {
        if (query && nlabels >= 0) return fail(DANN_ERR_INVALID_ARG, "plain storage does not support label filters (plain/storage.rs:260)");
        if (v.dim == v.dim_index) rescore = 0; /* scan.rs:392-403: next() instead of next_with_resort */
    }
    if (rescore > 0 && v.n && !v.vectors) return fail(DANN_ERR_STATE, "index has no heap vectors yet: rescore must be 0");
    cudaStream_t st = ix->stream;
    const uint32_t dim = v.dim;
    if (query) sc->query.assign(query, query + dim);
    else sc->query.assign(dim, 0.0f); /* NULL order-by argument: zero vector, no labels (labels/mod.rs:214-216) */
    sc->nlabels = query ? nlabels : -1;
    sc->labels.clear();
    if (sc->nlabels > 0) { /* LabelSet::from(Vec): sort_unstable + dedup (labels/mod.rs:30-37) */
        sc->labels.assign(labels, labels + nlabels);
        std::sort(sc->labels.begin(), sc->labels.end());
        sc->labels.erase(std::unique(sc->labels.begin(), sc->labels.end()), sc->labels.end());
    }
    sc->L = search_list_size;
    sc->rescore = rescore;
    sc->grow = 1;
    sc->streamed = sc->win_len = 0;
    sc->exhausted = false;
    sc->stats = dann_query_stats{};
    /* amrescan's vector preparation runs once, here */
    CK(sc->d_query.reserve((size_t)dim * 4));
    CK(sc->d_qfull.reserve((size_t)dim * 4));
    CK(sc->d_qcodes.reserve((size_t)v.cw * 8));
    CK(sc->d_slen.reserve(16));
    CK(sc->d_stats.reserve(sizeof(dann_query_stats)));
    CK(sc->d_win.reserve((size_t)std::max(rescore, 1) * 8));
    CK(sc->d_winst.reserve(sizeof(ScanWindow)));
    CK(sc->d_row.reserve(sizeof(ScanRow)));
    CK(sc->d_ctl.reserve(64));
    CK(cudaMemcpyAsync(sc->d_query.p, sc->query.data(), (size_t)dim * 4, cudaMemcpyHostToDevice, st));
    if (sc->nlabels >= 0) {
        int32_t off[2] = {0, (int32_t)sc->labels.size()};
        CK(sc->d_labels.reserve(std::max<size_t>(sc->labels.size(), 1) * 2));
        CK(sc->d_label_off.reserve(8));
        if (!sc->labels.empty()) CK(cudaMemcpyAsync(sc->d_labels.p, sc->labels.data(), sc->labels.size() * 2, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(sc->d_label_off.p, off, 8, cudaMemcpyHostToDevice, st));
    }
    CK(cudaMemsetAsync(sc->d_winst.p, 0, sizeof(ScanWindow), st));
    if (ix->plain) {
        CK(sc->d_qindex.reserve((size_t)v.dim_index * 4));
        dann_prepare_plain_kernel<<<1, 128, 0, st>>>(v.dim, v.dim_index, v.distance_type == DANN_COSINE, sc->d_query.as<float>(),
                                                    sc->d_qfull.as<float>(), sc->d_qindex.as<float>());
        ix->launches++;
        CK(cudaGetLastError());
    } else {
        rc = launch_prepare(ix, sc->d_query.as<float>(), 1, sc->d_qfull.as<float>(), sc->d_qcodes.as<uint64_t>(), st);
        if (rc) return rc;
    }
    rc = scan_reset_search(sc);
    if (rc) return rc;
    CK(cudaStreamSynchronize(st));
    sc->active = true;
    return DANN_OK;
} DANN_CATCH

/* Enqueue the resumable search for rows [0, want) of this launch (d_ctl[1] receives the overflow bits). */
static int scan_launch_search(dann_scan *sc, uint32_t want) {
    dann_index *ix = sc->ix;
    const IndexView &v = ix->v;
    cudaStream_t st = ix->stream;
    {
        const SearchPlan &p = sc->plan;
        CK(sc->d_stream.reserve((size_t)want * 4));
        uint32_t *d_ctl = sc->d_ctl.as<uint32_t>();
        CK(cudaMemsetAsync(d_ctl, 0, 8, st));
        SearchArgs a;
        a.ix = v;
        a.q_codes = sc->d_qcodes.as<uint64_t>();
        a.q_labels = sc->nlabels >= 0 ? sc->d_labels.as<int16_t>() : nullptr;
        a.q_label_off = sc->nlabels >= 0 ? sc->d_label_off.as<int32_t>() : nullptr;
        a.qlist = nullptr;
        a.nq = 1;
        a.L = (uint32_t)sc->L;
        a.c_target = want;
        a.stream = sc->d_stream.as<uint32_t>();
        a.stream_len = sc->d_slen.as<uint32_t>();
        a.stats = sc->d_stats.as<dann_query_stats>();
        a.overflow = d_ctl + 1;
        a.counter = d_ctl;
        a.hash = sc->d_set.as<uint32_t>();
        a.hash_cap = p.hash_cap;
        a.bitmap = sc->d_set.as<uint32_t>();
        a.bitmap_words = p.bitmap_words;
        a.ins_list = sc->d_ins.as<uint32_t>();
        a.ins_cap = p.ins_cap;
        a.lists_unique = ix->lists_unique;
        a.cand_node = sc->d_cnode.as<uint32_t>();
        a.cand_cap = p.cand_cap;
        a.heap_tail = sc->d_heap_tail.p;
        a.hs = p.hs;
        a.vcap = p.vcap;
        a.G = ix->G;
        a.Gshift = ix->Gshift;
        a.per_warp_smem = p.per_warp;
        a.saved = sc->d_saved.as<SavedScan>();
        a.saved_heap_sm = sc->d_heap_sm.p;
        a.saved_vis = sc->d_vis.as<uint64_t>();
        a.build_mode = 0;
        a.vis_out = nullptr;
        a.vis_out_len = nullptr;
        a.vis_out_cap = 0;
        a.hv_flags = 0;
        a.plain_vectors = ix->index_vectors;
        a.q_index = sc->d_qindex.as<float>();
        a.plain_dim = ix->plain ? v.dim_index : 0;
        search_fn fn = pick_kernel(false, p.entry, ix->NCH, ix->plain);
        CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(p.per_warp + DANN_SMEM_SLACK)));
        fn<<<1, 32, p.per_warp + DANN_SMEM_SLACK, st>>>(a);
        ix->launches++;
        CK(cudaGetLastError());
    }
    return DANN_OK;
}

/* Pull `need` more rows off the approximate stream into d_stream[skip ..]; returns how many came. */
static int scan_pull(dann_scan *sc, uint32_t need, uint32_t *got, uint32_t *skip_out) {
    dann_index *ix = sc->ix;
    cudaStream_t st = ix->stream;
    uint32_t skip = 0; /* rows that are only re-generated because the workspace had to grow */
    for (int attempt = 0;; attempt++) {
        const uint32_t want = skip + need;
        int lrc = scan_launch_search(sc, want);
        if (lrc) return lrc;
        uint32_t *d_ctl = sc->d_ctl.as<uint32_t>();
        struct {
            uint32_t ctl[2];
        } h;
        CK(cudaMemcpyAsync(h.ctl, d_ctl, 8, cudaMemcpyDeviceToHost, st));
        uint32_t slen = 0;
        CK(cudaMemcpyAsync(&slen, sc->d_slen.p, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&sc->stats, sc->d_stats.p, sizeof(dann_query_stats), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (h.ctl[1] == 0) {
            if (slen < want) sc->exhausted = true;
            *got = slen > skip ? slen - skip : 0;
            *skip_out = skip;
            return DANN_OK;
        }
        /* the scan outgrew its workspace: rebuild it twice as large and replay the stream up to here */
        if (attempt >= 8) return fail(DANN_ERR_CAPACITY, "scan workspace still too small after %d growth steps", attempt);
        sc->grow *= 2;
        int rc = scan_reset_search(sc);
        if (rc) return rc;
        skip = sc->streamed;
    }
}

/* DANN_SCAN_FUSED=1: the same amgettuple with ONE host synchronisation: search, exact distances of the new rows and the
 * window step are enqueued back to back (the kernels read the search's outcome from device memory) and a single
 * ScanStepOut comes back.  Same rows, same counters after every call; opt-in until it has been timed on hardware. */
static int gettuple_fused(dann_scan *sc, uint32_t *block, uint16_t *offset, uint32_t *node_id, float *dist) {
    dann_index *ix = sc->ix;
    const IndexView &v = ix->v;
    cudaStream_t st = ix->stream;
    const uint32_t rescore = (uint32_t)sc->rescore;
    const uint32_t need = rescore == 0 ? 1u : (sc->win_len < rescore ? rescore - sc->win_len : 0u);
    const bool searching = need && !sc->exhausted;
    CK(sc->d_step.reserve(sizeof(ScanStepOut)));
    ScanStepOut o;
    uint32_t skip = 0;
    for (int attempt = 0;; attempt++) {
        const uint32_t want = skip + need;
        if (searching) {
            int lrc = scan_launch_search(sc, want);
            if (lrc) return lrc;
            if (rescore > 0) {
                CK(sc->d_dist.reserve((size_t)want * 4));
                size_t smem = (size_t)((v.dim + 3u) & ~3u) * sizeof(float) + DANN_SMEM_SLACK;
                if (smem > 48 * 1024)
                    CK(cudaFuncSetAttribute(dann_scan_distance_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                dann_scan_distance_kernel<<<1, 128, smem, st>>>(v, sc->d_qfull.as<float>(), sc->d_stream.as<uint32_t>(),
                                                               sc->d_slen.as<uint32_t>(), sc->d_ctl.as<uint32_t>() + 1, skip,
                                                               sc->d_dist.as<float>());
                ix->launches++;
                CK(cudaGetLastError());
            }
        }
        dann_scan_finish_kernel<<<1, 32, 0, st>>>(v, sc->d_winst.as<ScanWindow>(), sc->d_win.as<uint64_t>(), rescore,
                                                 sc->d_stream.as<uint32_t>(), sc->d_dist.as<float>(), skip,
                                                 searching ? sc->d_slen.as<uint32_t>() : nullptr, skip,
                                                 searching ? sc->d_ctl.as<uint32_t>() + 1 : nullptr,
                                                 sc->d_stats.as<dann_query_stats>(), sc->d_step.as<ScanStepOut>());
        ix->launches++;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(&o, sc->d_step.p, sizeof o, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (!o.overflow) {
            if (searching) {
                if (o.slen < want) sc->exhausted = true;
                sc->streamed += o.slen > skip ? o.slen - skip : 0;
                sc->stats = o.stats;
            }
            break;
        }
        /* the scan outgrew its workspace: rebuild it twice as large and replay the stream up to here */
        if (attempt >= 8) return fail(DANN_ERR_CAPACITY, "scan workspace still too small after %d growth steps", attempt);
        sc->grow *= 2;
        int rrc = scan_reset_search(sc);
        if (rrc) return rrc;
        skip = sc->streamed;
    }
    sc->win_len = o.win.len;
    sc->stats.d_full = o.win.d_full;
    if (ix->plain) {
        sc->stats.d_full += sc->stats.candidates;
        sc->stats.d_quantized = 0;
    }
    sc->stats.stream_len = sc->streamed;
    if (!o.row.have) return 0;
    if (block) *block = (uint32_t)(o.row.tid >> 16);
    if (offset) *offset = (uint16_t)(o.row.tid & 0xFFFFu);
    if (node_id) *node_id = o.row.node;
    if (dist) *dist = o.row.dist;
    return 1;
}

extern "C" int dann_scan_gettuple(dann_scan *sc, uint32_t *block, uint16_t *offset, uint32_t *node_id, float *dist) try {
    if (!sc) return fail(DANN_ERR_INVALID_ARG, "dann_scan_gettuple: NULL scan");
    if (!sc->active) return fail(DANN_ERR_STATE, "dann_scan_gettuple before dann_scan_rescan");
    dann_index *ix = sc->ix;
    int rc = check_live(ix);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ix->mu);
    /* one host synchronisation per row is the default since it was timed on B200 (4.1 vs 4.6 ms per 10-row scan at
     * 1M x 768, bench.py --mode scan); DANN_SCAN_FUSED=0 selects the step-by-step path below */
    if (env_u32("DANN_SCAN_FUSED", 1) == 1) return gettuple_fused(sc, block, offset, node_id, dist);
    const IndexView &v = ix->v;
    cudaStream_t st = ix->stream;
    /* next_with_resort (scan.rs:244-305): `while resort_buffer.len() < resort_size { next() ... }` then pop;
     * with resort_size == 0 it is a plain next() */
    const uint32_t rescore = (uint32_t)sc->rescore;
    uint32_t need = rescore == 0 ? 1u : (sc->win_len < rescore ? rescore - sc->win_len : 0u);
    uint32_t got = 0, skip = 0;
    if (need && !sc->exhausted) {
        rc = scan_pull(sc, need, &got, &skip);
        if (rc) return rc;
        sc->streamed += got;
    }
    if (rescore > 0 && got > 0) { /* get_full_distance_for_resort for the rows that just arrived */
        CK(sc->d_dist.reserve((size_t)(skip + got) * 4));
        size_t smem = (size_t)((v.dim + 3u) & ~3u) * sizeof(float) + DANN_SMEM_SLACK;
        if (smem > 48 * 1024)
            CK(cudaFuncSetAttribute(dann_full_distance_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        dann_full_distance_kernel<<<1, 128, smem, st>>>(v, sc->d_qfull.as<float>(), sc->d_stream.as<uint32_t>(),
                                                       (int)(skip + got), sc->d_dist.as<float>());
        ix->launches++;
        CK(cudaGetLastError());
    }
    dann_scan_resort_kernel<<<1, 32, 0, st>>>(v, sc->d_winst.as<ScanWindow>(), sc->d_win.as<uint64_t>(), rescore,
                                             sc->d_stream.as<uint32_t>(), sc->d_dist.as<float>(), skip, skip + got,
                                             sc->d_row.as<ScanRow>());
    ix->launches++;
    CK(cudaGetLastError());
    ScanRow row;
    ScanWindow ws;
    CK(cudaMemcpyAsync(&row, sc->d_row.p, sizeof(ScanRow), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&ws, sc->d_winst.p, sizeof(ScanWindow), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    sc->win_len = ws.len;
    sc->stats.d_full = ws.d_full;
    if (ix->plain) { /* every comparison of the beam search was a full-distance comparison (plain/storage.rs:238,288) */
        sc->stats.d_full += sc->stats.candidates;
        sc->stats.d_quantized = 0;
    }
    sc->stats.stream_len = sc->streamed;
    if (!row.have) return 0;
    if (block) *block = (uint32_t)(row.tid >> 16);
    if (offset) *offset = (uint16_t)(row.tid & 0xFFFFu);
    if (node_id) *node_id = row.node;
    if (dist) *dist = row.dist;
    return 1;
} DANN_CATCH

extern "C" int dann_scan_stats(dann_scan *sc, dann_query_stats *out) try {
    if (!sc || !out) return fail(DANN_ERR_INVALID_ARG, "dann_scan_stats: NULL argument");
    *out = sc->stats;
    return DANN_OK;
} DANN_CATCH

extern "C" void dann_scan_end(dann_scan *sc) {
    if (!sc) return;
    cudaSetDevice(sc->ix->device);
    scan_release(sc);
    cudaGetLastError();
    delete sc;
}

/* ------------------------------------------------------------------------------------ */
/* query coalescing for process-per-connection hosts (SURVEY.md §8f row 4)                */
#include "dann_coalescer.h"
#include "dann_group.h"

/* ------------------------------------------------------------------------------------ */
/* reading an index relation file (SURVEY.md §8f row 2): host only                       */
#include "dann_pgreader.h"

struct dann_pg_relation {
    dannpg::Relation rel;
};

extern "C" int dann_pg_relation_open(const char *path, dann_pg_relation **out) try {
    if (!path || !out) return fail(DANN_ERR_INVALID_ARG, "dann_pg_relation_open: NULL argument");
    *out = nullptr;
    dann_pg_relation *r = new dann_pg_relation();
    const int rc = dannpg::open_relation(path, &r->rel);
    if (rc != DANN_OK) {
        const std::string msg = r->rel.err;
        delete r;
        return fail(rc, "dann_pg_relation_open: %s", msg.c_str());
    }
    *out = r;
    return DANN_OK;
} DANN_CATCH

extern "C" void dann_pg_relation_close(dann_pg_relation *rel) { delete rel; }

extern "C" int dann_pg_relation_stat(const dann_pg_relation *rel, dann_pg_relation_info *out) try {
    if (!rel || !out) return fail(DANN_ERR_INVALID_ARG, "dann_pg_relation_stat: NULL argument");
    dannpg::stat_relation(rel->rel, out);
    return DANN_OK;
} DANN_CATCH

extern "C" int dann_pg_read_chain(const dann_pg_relation *rel, uint32_t block, uint16_t offset, int page_type, void *buf,
                                  size_t cap, size_t *len) try {
    if (!rel || !len || (cap && !buf)) return fail(DANN_ERR_INVALID_ARG, "dann_pg_read_chain: NULL argument");
    std::vector<unsigned char> bytes;
    std::string err;
    const int rc = dannpg::read_chain(rel->rel, block, offset, page_type, bytes, err);
    if (rc != DANN_OK) return fail(rc, "dann_pg_read_chain (%u,%u): %s", block, (unsigned)offset, err.c_str());
    *len = bytes.size();
    if (cap) memcpy(buf, bytes.data(), std::min(cap, bytes.size()));
    return DANN_OK;
} DANN_CATCH

static int pg_extract(const dann_pg_relation *rel, const dann_pg_meta *meta, bool plain, dann_pg_snapshot **out, const char *who) {
    if (!rel || !meta || !out) return fail(DANN_ERR_INVALID_ARG, "%s: NULL argument", who);
    *out = nullptr;
    dannpg::SbqOut *o = new dannpg::SbqOut();
    memset(&o->pub, 0, sizeof o->pub);
    std::string err;
    int rc;
    try {
        rc = dannpg::extract_nodes(rel->rel, meta, plain, o, err);
    } catch (...) {
        delete o;
        throw;
    }
    if (rc != DANN_OK) {
        delete o;
        return fail(rc, "%s: %s", who, err.c_str());
    }
    o->pub.self = o;
    *out = &o->pub;
    return DANN_OK;
}

extern "C" int dann_pg_extract_sbq(const dann_pg_relation *rel, const dann_pg_meta *meta, dann_pg_snapshot **out) try {
    return pg_extract(rel, meta, false, out, "dann_pg_extract_sbq");
} DANN_CATCH

extern "C" int dann_pg_extract_plain(const dann_pg_relation *rel, const dann_pg_meta *meta, dann_pg_snapshot **out) try {
    return pg_extract(rel, meta, true, out, "dann_pg_extract_plain");
} DANN_CATCH

extern "C" void dann_pg_snapshot_free(dann_pg_snapshot *s) {
    if (s) delete static_cast<dannpg::SbqOut *>(s->self);
}

extern "C" int dann_pg_heap_fetch_vectors(const dann_pg_relation *heap, const dann_pg_relation *toast, const dann_pg_heap_layout *layout,
                                          const uint64_t *heap_tid, uint32_t n, float *out, uint32_t *n_missing) try {
    if (!heap || !layout || (n && (!heap_tid || !out)) || !layout->dim || (layout->natts_before && (!layout->attlen || !layout->attalign)))
        return fail(DANN_ERR_INVALID_ARG, "dann_pg_heap_fetch_vectors: bad argument");
    uint32_t missing = 0;
    std::string err;
    const int rc = dannpg::fetch_vectors(heap->rel, toast ? &toast->rel : nullptr, layout, heap_tid, n, out, &missing, err);
    if (rc != DANN_OK) return fail(rc, "dann_pg_heap_fetch_vectors: %s", err.c_str());
    if (n_missing) *n_missing = missing;
    return DANN_OK;
} DANN_CATCH
