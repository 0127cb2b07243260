/*
 * diskann_b200.h — C ABI of the B200-native StreamingDiskANN index-scan engine.
 *
 * This is the drop-in boundary for pgvectorscale's `diskann` index *scan* path: the
 * Rust/pgrx access-method callbacks stay host code and call these entry points where
 * they used to run `TSVScanState::initialize` and `TSVResponseIterator::next_with_resort`.
 * Reference citations are relative to /root/reference/pgvectorscale/src/access_method/.
 *
 *   reference interface                              replaced by
 *   ------------------------------------------------ -----------------------------------
 *   ambeginscan            scan.rs:309-333           dann_scan_begin
 *   amrescan               scan.rs:336-367           dann_scan_rescan
 *     TSVScanState::initialize      scan.rs:57-88
 *     LabeledVector::from_scan_key_data labels/mod.rs:209-238
 *     Graph::greedy_search_streaming_init graph/mod.rs:331-354
 *   amgettuple             scan.rs:370-436           dann_scan_gettuple
 *     TSVResponseIterator::next_with_resort scan.rs:244-305
 *     Graph::greedy_search_iterate  graph/mod.rs:357-385
 *     SbqSpeedupStorage::visit_lsn  sbq/storage.rs:125-190
 *     get_full_distance_for_resort  sbq/storage.rs:304-328
 *   amendscan              scan.rs:439-476           dann_scan_end (+ dann_scan_stats)
 *   MetaPage::fetch / SbqMeans::load (index -> RAM)  dann_index_load (index -> HBM)
 *   PlainStorage::load_for_search plain/storage.rs   dann_index_load_plain
 *   distance_xor_optimized distance/mod.rs:265-323   dann_sbq_distance (micro-kernel)
 *   distance_l2 / _cosine / _inner_product :88-209   dann_full_distance (micro-kernel)
 *   SbqQuantizer::quantize sbq/quantize.rs:52-102    dann_prepare_queries
 *
 * Conventions: every function returns DANN_OK (0) or a negative dann_status; nothing
 * throws, longjmps or aborts (the Rust shim turns a non-zero code into pgrx::error!).
 * dann_last_error() gives a thread-local message.  Host pointers are borrowed for the
 * duration of the call only.  A dann_index is immutable after load and may be shared
 * by host threads (calls on one index are serialised internally); a dann_scan is
 * single-threaded, like a Postgres backend.
 */
#ifndef DISKANN_B200_H
#define DISKANN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DANN_INVALID_NODE 0xFFFFFFFFu          /* InvalidBlockNumber, sbq/node.rs:261-273 */
#define DANN_INVALID_TID 0xFFFFFFFFFFFFFFFFull /* "no row" in batch outputs */

typedef enum {
    DANN_OK = 0,
    DANN_ERR_INVALID_ARG = -1,
    DANN_ERR_CUDA = -2,      /* sticky: the handle is poisoned */
    DANN_ERR_NO_DEVICE = -3, /* no CUDA device / driver: there is NO CPU fallback */
    DANN_ERR_OOM = -4,
    DANN_ERR_CAPACITY = -5,  /* per-query state outgrew the largest workspace we may allocate */
    DANN_ERR_STATE = -6,
    DANN_ERR_FORMAT = -7     /* dann_pg_*: the relation file is not what the reader can vouch for; nothing is guessed */
} dann_status;

typedef enum { DANN_COSINE = 0, DANN_L2 = 1, DANN_IP = 2 } dann_distance; /* distance/mod.rs:11-15 */

/* Flat snapshot of one diskann index (host memory, row-major). See
 * pgvectorscale_b200/snapshot.py for the field-by-field provenance. */
typedef struct {
    uint32_t n;             /* nodes */
    uint32_t dim;           /* heap vector dimensions */
    uint32_t dim_index;     /* num_dimensions_to_index, pg_vector.rs:143-148 */
    uint32_t bits;          /* SBQ bits per dimension, meta_page.rs:312-323 */
    uint32_t words;         /* u64 per code = ceil(dim_index*bits/64), quantize.rs:38-46 */
    uint32_t R;             /* num_neighbors, meta_page.rs:284-294 */
    int32_t distance_type;  /* dann_distance */
    int32_t has_labels;
    uint64_t count;         /* SbqMeans.count */
    const float *mean;      /* [dim_index] */
    const float *m2;        /* [dim_index], may be NULL when bits == 1 */
    const uint64_t *codes;  /* [n*words] */
    const uint32_t *nbrs;   /* [n*R], list ends at first DANN_INVALID_NODE */
    const uint64_t *heap_tid; /* [n] (block<<16)|offset, offset 0 = deleted */
    const float *vectors;   /* [n*dim] raw heap vectors */
    uint32_t start_default; /* DANN_INVALID_NODE = empty graph */
    uint32_t n_start_labels;
    const int16_t *start_labels;       /* ascending */
    const uint32_t *start_label_nodes;
    const uint32_t *label_off;         /* [n+1] if has_labels */
    const int16_t *labels;             /* sorted, dedup per node */
} dann_snapshot_desc;

/* Per-query counters: the ones the reference logs at amendscan (scan.rs:461-472). */
typedef struct {
    uint32_t visits;      /* visits=      */
    uint32_t d_quantized; /* d_quantized= */
    uint32_t candidates;  /* candidate=   */
    uint32_t d_full;      /* d_full=      */
    uint32_t stream_len;  /* non-deleted items consumed from the ListSearchResult */
    uint32_t status;      /* 0 ok; internal overflow bits are retried and never surface */
} dann_query_stats;

typedef struct dann_index dann_index;
typedef struct dann_scan dann_scan;

const char *dann_last_error(void);
int dann_device_count(void);

/* ---- index lifetime ----------------------------------------------------------- */
/* Copies the snapshot into HBM of `device` (vectors cosine-normalised once, with the
 * reference's preprocess_cosine arithmetic, distance/mod.rs:225-253). */
int dann_index_load(const dann_snapshot_desc *snap, int device, dann_index **out);
/* storage_layout = plain (storage.rs:144-169; PlainStorage, plain/storage.rs:223-307): every node carries the f32
 * vector it was indexed with - index_vectors [n*dim_index], i.e. truncated to num_dimensions_to_index and, for cosine,
 * normalised after truncation (pg_vector.rs:143-155) - and the beam search compares the query with it directly; the
 * snapshot's SBQ fields (bits, words, count, mean, m2, codes) are ignored.  As in the reference (build.rs:264-290)
 * inner product, label filters and more than 2000 indexed dimensions are rejected.  Scans rerank from `vectors` only
 * when dim_index < dim (scan.rs:392-403), otherwise rows come back in beam-search order with dist = NaN.
 * Verified bit-exact against the oracle on B200 (tests/test_zz_plain_gpu.py) and under CPU emulation of the kernel. */
int dann_index_load_plain(const dann_snapshot_desc *snap, const float *index_vectors, int device, dann_index **out);
void dann_index_free(dann_index *ix);
/* `vectors` may be NULL in the snapshot (see dann_index_set_vectors); scans then need rescore == 0.
 * Bytes of HBM held by the index arrays (codes, nbrs, tids, vectors, labels, means): */
uint64_t dann_index_hbm_bytes(const dann_index *ix);

/* ---- scan operator: one row at a time, amgettuple order ------------------------ */
int dann_scan_begin(dann_index *ix, dann_scan **out);
/* query: [dim] raw floats, NULL = SQL NULL order-by argument (zero vector, no labels,
 * labels/mod.rs:214-216). nlabels < 0 = no scan key; >= 0 = `labels && ARRAY[...]`
 * (sorted+dedup is done here, labels/mod.rs:30-37). search_list_size / rescore are the
 * GUCs diskann.query_search_list_size / diskann.query_rescore (guc.rs:3-4). */
int dann_scan_rescan(dann_scan *sc, const float *query, const int16_t *labels, int nlabels,
                     int search_list_size, int rescore);
/* How far a scan may stream: the suspended search's workspace is planned for rescore + 64 streamed rows; a scan that
 * runs past it (a selective post-filter without LIMIT) has its workspace rebuilt twice as large and the stream
 * replayed from row 0 - invisible to the caller except in time (the k-th doubling replays 2^k x the first plan) - up
 * to eight doublings or 2^30 candidates per query, then DANN_ERR_CAPACITY.  The reference can stream the whole index
 * through amgettuple; this operator is built for top-k scans (k ~ rescore) and says so.
 * One amgettuple: resumes the scan's suspended search (its state lives in HBM between calls), pulls
 * exactly the rows TSVResponseIterator::next_with_resort would (scan.rs:244-305), pops one.
 * Returns 1 and fills the outputs for the next row, 0 at end of scan, <0 on error.
 * dist is the exact rerank distance (NaN when rescore == 0). Any output may be NULL. */
int dann_scan_gettuple(dann_scan *sc, uint32_t *block, uint16_t *offset, uint32_t *node_id,
                       float *dist);
int dann_scan_stats(dann_scan *sc, dann_query_stats *out);
void dann_scan_end(dann_scan *sc);

/* ---- entry points that take DEVICE buffers (dann_search_batch_device, dann_prepare_queries, dann_sbq_distance,
 * dann_full_distance, dann_index_set_vectors_device): `stream` is the CUDA stream the call runs on and the order in
 * which the caller's buffers must be ready.  stream == NULL: the call runs on the index's own non-blocking stream,
 * after everything the caller has already submitted to the legacy default stream (the order a default-stream kernel
 * or a plain cudaMemcpy would have had); buffers produced on OTHER non-blocking streams need that stream passed here,
 * or a synchronisation by the caller.  Outputs are complete when the call returns. */

/* ---- batch: B independent scans, first k rows of each ---------------------------- */
/* Host buffers; H2D/D2H copies are part of the call (this is the end-to-end path).
 * labels/label_off: CSR of each query's scan-key labels, label_off == NULL = no key.
 * out_tid [B*k] (block<<16|offset, DANN_INVALID_TID past out_count[b]), out_dist [B*k],
 * out_count [B] rows produced, out_stats [B] (each may be NULL except out_tid).
 * rescore + k is bounded by the rerank kernel's shared memory (on a B200 about 57 000 rows at 768 dimensions,
 * 42 000 at 16 000): larger requests return DANN_ERR_INVALID_ARG and leave the handle usable (the streaming
 * scan operator is not bound by the rerank window). */
int dann_search_batch(dann_index *ix, const float *queries, const int16_t *labels,
                      const int32_t *label_off, int B, int k, int search_list_size,
                      int rescore, uint64_t *out_tid, float *out_dist, uint32_t *out_count,
                      dann_query_stats *out_stats);
/* Same with every buffer already resident in HBM of the index's device; work is
 * enqueued on `stream` (a cudaStream_t; NULL = the index's own stream, see the note on device buffers above) and
 * the call returns after the stream has drained (it must read back a 4-byte overflow flag). Query labels
 * must already be sorted+dedup per query. */
int dann_search_batch_device(dann_index *ix, const float *d_queries, const int16_t *d_labels,
                             const int32_t *d_label_off, int B, int k, int search_list_size,
                             int rescore, uint64_t *d_out_tid, float *d_out_dist,
                             uint32_t *d_out_count, dann_query_stats *d_out_stats,
                             void *stream);

/* ---- stand-alone kernels (roofline metric + per-kernel parity tests), device buffers -- */
/* amrescan's vector preparation: cosine-normalise + SBQ-quantize B queries.
 * d_q_full [B*dim] (may be NULL), d_q_codes [B*dann_code_stride(ix)]. */
int dann_prepare_queries(dann_index *ix, const float *d_queries, int B, float *d_q_full,
                         uint64_t *d_q_codes, void *stream);
uint32_t dann_code_stride(const dann_index *ix); /* u64 per code row in HBM (words rounded up to even) */
/* SBQ distance: out[i] = popcount(code[pair_node[i]] ^ qcode[pair_q[i]]). */
int dann_sbq_distance(dann_index *ix, const uint64_t *d_qcodes, const uint32_t *d_pair_q,
                      const uint32_t *d_pair_node, size_t npairs, uint32_t *d_out, void *stream);
/* Exact rerank distance: out[b*m+i] = distance_fn(vectors[nodes[b*m+i]], q_full[b]);
 * nodes == DANN_INVALID_NODE are skipped (out = NaN). */
int dann_full_distance(dann_index *ix, const float *d_q_full, const uint32_t *d_nodes, int B,
                       int m, float *d_out, void *stream);

/* ---- index construction (SURVEY.md §8f row 1; NOT the scan hot path) -----------------------------
 * GPU batch Vamana over SBQ codes built from the scan kernels: greedy_search_for_build
 * (graph/mod.rs:285-327) + prune_neighbors (:392-488) + back-pointers (:212-266,720-737), nodes
 * inserted in batches.  The index must have been loaded with R == 64 neighbour slots per node
 * (contents ignored) and start_default == 0; `vectors` may be NULL at load and supplied later.  A labeled
 * index (has_labels, with start_labels/start_label_nodes = the first node carrying each label) is built
 * the reference's way: a label-filtered insertion pass from the label start nodes, then the unfiltered
 * one (graph/mod.rs:637-660), with the label-aware prune (:445-455).  On return every list holds
 * <= num_neighbors ids.  The graph is a valid diskann graph but not the reference's serial insertion
 * order, so it serves bulk builds, fixtures and benchmarks.  The prune step stages 128 candidate codes per
 * warp in shared memory, which on a B200 holds codes of up to 222 words (14 208 dimensions at 1 bit); a wider
 * code returns DANN_ERR_CAPACITY before anything is written, and the index keeps its neighbour lists. */
typedef struct {
    uint32_t batches;
    float search_ms, prune_ms, sort_ms, backlink_ms, total_ms;
    double avg_degree;
} dann_build_stats;
int dann_build_graph(dann_index *ix, int num_neighbors, int search_list_size, float max_alpha, uint32_t max_batch,
                     dann_build_stats *out);
/* Copy the neighbour lists back to the host: out [n][R] with R = the snapshot's R. */
int dann_index_download_nbrs(dann_index *ix, uint32_t *out);
/* Supply (or replace) the heap vectors of an index loaded with vectors == NULL; [n][dim] host floats. */
int dann_index_set_vectors(dann_index *ix, const float *vectors);
/* The same with the rows already in HBM on the index's device: d_vectors [n][dim] is BORROWED - the index reads it in
 * place (no second copy: 50M x 768-d rows are 153.6 GB of the 180) and, for cosine, normalises it in place once like
 * dann_index_load does; the caller keeps it allocated until dann_index_free. */
int dann_index_set_vectors_device(dann_index *ix, float *d_vectors);

/* ---- query-batch data parallelism over replicated indexes (SURVEY.md §8b / §8e) ------------------------------
 * One host process, one full replica of the index per GPU.  dann_group_search_batch cuts the batch into contiguous
 * slices (the first devices take the remainder), every device runs the whole hot path on its slice concurrently,
 * and each device's result copy lands directly in the caller's arrays at its slice's offset: rows come back in
 * query order, identical to a single-device dann_search_batch.  The graph is never sharded (every hop would cross
 * NVLink).  Separate PROCESSES per GPU (torchrun) gather with one NCCL collective instead: pgvectorscale_b200/group.py.
 * devices == NULL means devices 0..ndev-1.  Host pointers, borrowed for the call. */
typedef struct dann_group dann_group;
int dann_group_create(const dann_snapshot_desc *snap, int ndev, const int *devices, dann_group **out);
int dann_group_size(const dann_group *g);
dann_index *dann_group_replica(dann_group *g, int i); /* replica i (e.g. to attach vectors or read timings); NULL if out of range */
int dann_group_search_batch(dann_group *g, const float *queries, const int16_t *labels, const int32_t *label_offsets,
                            int B, int k, int search_list_size, int rescore, uint64_t *out_tid, float *out_dist,
                            uint32_t *out_count, dann_query_stats *out_stats);
void dann_group_free(dann_group *g);

/* ---- reading an index RELATION FILE (SURVEY.md §8f row 2; pgvectorscale_b200/csrc/dann_pgreader.h) -------------------
 * Host-only, no GPU involved.  Replaces, for an external loader (the sidecar after a CHECKPOINT, an offline exporter):
 *   ReadablePage::read / get_type / get_item_unchecked   util/page.rs:254-290   dann_pg_relation_open / _info
 *   TsvPageOpaqueData::read_from_page / verify            util/page.rs:59-97     (every page is checked the same way)
 *   ChainItemReader::read                                 util/chain.rs:125-183  dann_pg_read_chain
 *   MetaPage::fetch: magic + version of MetaPageHeader    meta_page.rs:386-419   dann_pg_relation_info.meta_*
 *   ArchivedSbqNode accessors + SbqMeans::load            sbq/node.rs:236-330, sbq/mod.rs:88-122   dann_pg_extract_sbq
 *   ArchivedPlainNode accessors                           plain/node.rs:15-120   dann_pg_extract_plain
 *   TableSlot::from_index_heap_pointer + PgVector::from_datum  util/table_slot.rs:13-53, pg_vector.rs:125-199   dann_pg_heap_fetch_vectors
 * The MetaPage BODY is an rkyv archive of a repr(Rust) struct whose field order cannot be pinned offline: the caller
 * supplies its scalars (dann_pg_meta; a Rust host fills them from MetaPage's getters) and the reader cross-checks them
 * against the node items; the node items' own field order is inferred and verified, never assumed (see the header of
 * dann_pgreader.h).  Anything unexpected is DANN_ERR_FORMAT with a message, not a best effort.
 * Staleness: a snapshot is valid for exactly the `fingerprint` it was extracted under - a hash over every page's
 * (block, pd_lsn, pd_checksum, pd_lower, pd_upper); every WAL-logged change of a page moves its pd_lsn. */
typedef struct dann_pg_relation dann_pg_relation;
typedef struct {
    uint32_t nblocks;
    uint32_t pages_by_type[9]; /* PageType histogram, util/page.rs:28-38 (5 = SbqNode, 7 = SbqMeans, 8 = Meta) */
    uint32_t new_pages;        /* all-zero pages (PageIsNew) */
    uint32_t foreign_pages;    /* pages that fail the extension's page checks */
    uint32_t meta_magic;       /* 768756476 when block 0 is a Meta page whose header item parses, else 0 */
    uint32_t meta_version;     /* TSV_VERSION (3 in the reference at hand) */
    uint64_t node_items;       /* LP_NORMAL line pointers on SbqNode pages */
    uint64_t max_lsn;
    uint64_t fingerprint;
} dann_pg_relation_info;
/* path = the relation's first segment file (base/<db>/<relfilenode>); "<path>.1", ".2", ... are picked up */
int dann_pg_relation_open(const char *path, dann_pg_relation **out);
void dann_pg_relation_close(dann_pg_relation *rel);
int dann_pg_relation_stat(const dann_pg_relation *rel, dann_pg_relation_info *out);
/* Reassembles the chained item that starts at (block, offset): *len = its size; copies min(*len, cap) bytes into buf
 * (buf may be NULL with cap == 0 to ask for the size).  page_type < 0 = do not check the pages' PageType. */
int dann_pg_read_chain(const dann_pg_relation *rel, uint32_t block, uint16_t offset, int page_type, void *buf, size_t cap,
                       size_t *len);
typedef struct { /* MetaPage scalars (meta_page.rs:212-282) and the pointers it holds */
    uint32_t num_dimensions, num_dimensions_to_index, bq_bits, num_neighbors;
    int32_t distance_type; /* dann_distance */
    int32_t has_labels;
    uint32_t start_block;  /* start_nodes.default_node; DANN_INVALID_NODE (InvalidBlockNumber) = empty graph */
    uint16_t start_offset;
    uint32_t n_start_labels; /* start_nodes.labeled_nodes */
    const int16_t *start_labels;
    const uint32_t *start_label_block;
    const uint16_t *start_label_offset;
    uint32_t means_block;  /* quantizer_metadata; DANN_INVALID_NODE = the quantizer uses no means */
    uint16_t means_offset;
} dann_pg_meta;
typedef struct { /* owned by the library until dann_pg_snapshot_free */
    dann_snapshot_desc snap;   /* ready for dann_index_load (dann_index_load_plain with index_vectors below) except
                                  vectors == NULL: heap rows live in the TABLE; fetch heap_tid[i] in order and attach
                                  them with dann_index_set_vectors */
    const float *index_vectors; /* plain layout: [n * dim_index] the vector each node stores (plain/node.rs:17-22); else NULL */
    const uint64_t *index_tid; /* [n] (block<<16)|offset of node i inside the index relation, ascending: the
                                  IndexPointer -> dense node id map */
    uint64_t fingerprint;      /* of the relation as extracted */
    uint32_t layout[4];        /* which 8-byte cell of the archived root held: heap pointer, code (or f32 vector),
                                  neighbour vector, fourth vector */
    void *self;                /* the library's owner object (dann_pg_snapshot_free) */
} dann_pg_snapshot;
/* storage_layout = memory_optimized: SbqNode pages (sbq/node.rs:26-42) + the SbqMeans chain */
int dann_pg_extract_sbq(const dann_pg_relation *rel, const dann_pg_meta *meta, dann_pg_snapshot **out);
/* storage_layout = plain: Node pages (plain/node.rs:15-22); bq_bits, has_labels and the means pointer of `meta` are ignored */
int dann_pg_extract_plain(const dann_pg_relation *rel, const dann_pg_meta *meta, dann_pg_snapshot **out);
void dann_pg_snapshot_free(dann_pg_snapshot *s);

/* The heap rows of a snapshot: the vector column of the TABLE's relation file(s), read the way the rerank reads it
 * (sbq/storage.rs:304-328 -> util/table_slot.rs:13-53 -> pg_vector.rs:125-199: tuple by TID, detoast, f32[dim]).
 * Postgres' documented heap / varlena / TOAST formats and pgvector's value layout only (no rkyv).  `heap` and `toast`
 * are opened with dann_pg_relation_open on the table's and its TOAST table's files (toast may be NULL when every value
 * is inline).  The caller describes the attributes IN FRONT of the vector column (pg_attribute.attlen: > 0 fixed, -1
 * varlena; attalign 'c' 's' 'i' 'd').  Rows that are gone - heap_tid offset 0, dead or unused line pointer, NULL value -
 * come back as zeros and are counted in *n_missing; HOT redirects are followed; there is no visibility test (the
 * index names the tuples, the executor re-checks each row).  Compressed values are refused (the type is STORAGE external). */
typedef struct {
    uint32_t natts_before;  /* attributes in front of the vector column */
    const int16_t *attlen;  /* [natts_before] */
    const char *attalign;   /* [natts_before] */
    uint32_t dim;           /* vector(dim) */
    char vector_align;      /* 0 = 'i' (what CREATE TYPE vector declares) */
} dann_pg_heap_layout;
int dann_pg_heap_fetch_vectors(const dann_pg_relation *heap, const dann_pg_relation *toast, const dann_pg_heap_layout *layout,
                               const uint64_t *heap_tid, uint32_t n, float *out, uint32_t *n_missing);

/* How the last batch search of this index was planned (diagnostics for benchmarks and profiles). */
typedef struct {
    uint32_t kernel;         /* 1 = single-warp, 2 = two-warp (round 1), 3 = lean warp-per-query (dann_search3.cuh) */
    uint32_t slots_per_sm;   /* resident queries per SM */
    uint32_t grid;           /* CTAs (one per SM) */
    uint32_t heap_smem;      /* heap entries kept in shared memory per query */
    uint32_t visited_cap, cand_cap;
    uint32_t entry_bytes;    /* 4 or 8 */
    uint32_t bitmap;         /* 1 = bitmap inserted-set, 0 = hash set */
    uint64_t slot_hbm_bytes; /* per-slot HBM workspace (heap tail + inserted-set [+ side tables]) */
    uint32_t smem_per_slot;
    uint32_t retries;        /* workspace-growth reruns of the last call */
} dann_search_plan_info;
int dann_last_search_plan(dann_index *ix, dann_search_plan_info *out);

/* ---- query coalescing (SURVEY.md §8f row 4: multi-process serving, the in-process half) ----------------------
 * Postgres is process-per-connection with amcanparallel = false (mod.rs:63): one scan per backend at a time, while
 * the engine's throughput comes from batches.  A coalescer owns a dispatcher thread; any number of host threads (one
 * per connected backend in a sidecar that holds the HBM-resident index) call dann_coalescer_search with ONE query and
 * block; requests that arrive within max_wait_us of the first one (at most max_batch, same k / search_list_size /
 * rescore, all keyed or all unkeyed) become one dann_search_batch call.  Each caller receives exactly the rows,
 * distances and counters a private dann_search_batch of its query returns.  nlabels < 0 = no scan key.
 * The socket / shared-memory transport between backends and the sidecar is not part of this library. */
typedef struct dann_coalescer dann_coalescer;
int dann_coalescer_create(dann_index *ix, int max_batch, int max_wait_us, dann_coalescer **out);
int dann_coalescer_search(dann_coalescer *c, const float *query, const int16_t *labels, int nlabels, int k,
                          int search_list_size, int rescore, uint64_t *out_tid, float *out_dist,
                          uint32_t *out_count, dann_query_stats *out_stats);
int dann_coalescer_stats(dann_coalescer *c, uint64_t *batches, uint64_t *queries, uint64_t *largest_batch);
void dann_coalescer_destroy(dann_coalescer *c); /* drains what is queued, then stops; destroy before dann_index_free */

/* Number of this library's kernel launches since load (bench.py "gpu_launches"). */
uint64_t dann_kernel_launches(const dann_index *ix);

/* ---- device-timed leg of the last batch call (CUDA events on the launch stream) ---- */
typedef struct {
    float prepare_ms, search_ms, rerank_ms, resort_ms, total_ms;
    uint32_t retries; /* workspace-growth retries of the search kernel */
} dann_batch_timing;
int dann_last_batch_timing(dann_index *ix, dann_batch_timing *out);

#ifdef __cplusplus
}
#endif
#endif
