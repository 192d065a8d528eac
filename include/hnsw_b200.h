/*
 * hnsw_b200.h -- C ABI of the B200-native HNSW hot path (libhnsw_b200.so).
 *
 * Drop-in boundary for ONE path of dhwodnjs/pgvector-hnsw-partitioning: distance evaluation for
 * the vector_l2_ops / vector_ip_ops / vector_cosine_ops (and halfvec_*) operator classes inside
 * HNSW search and index build, the hnswbuild insert path, the hnswgettuple scan path, and
 * partition routing / top-k merge.
 *
 * Citations: the reference mount contains no source (/root/reference/README.md:1, "# pg", is the
 * whole tree), so no reference file:line can be given.  Each entry point names the PostgreSQL
 * index-AM callback or upstream-pgvector function [RECALL] whose role it takes; INTEGRATION.md
 * shows the Postgres-side glue a maintainer would add.
 *
 * Conventions: plain pointers and sizes, no C++/torch types.  "host" pointers are ordinary CPU
 * memory owned by the caller; "dev" pointers are CUDA device memory on the index's GPU.  Every
 * function returning int returns 0 (or a count) on success and a negative HB_E* code on failure;
 * hb_last_error() gives the message (Postgres glue turns it into ereport(ERROR)).  One handle is
 * not thread-safe; distinct handles are.  There is no CPU fallback: without a CUDA device every
 * call fails with HB_ECUDA.
 */
#ifndef HNSW_B200_H
#define HNSW_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* operator classes: FUNCTION 1 (HNSW_DISTANCE_PROC) of the opclass */
enum {
    HB_L2 = 0,     /* vector_l2_ops / halfvec_l2_ops         : vector_l2_squared_distance       */
    HB_IP = 1,     /* vector_ip_ops / halfvec_ip_ops         : vector_negative_inner_product    */
    HB_COSINE = 2, /* vector_cosine_ops / halfvec_cosine_ops : normalise (FUNCTION 2) + neg. ip */
    HB_L1 = 3      /* vector_l1_ops / halfvec_l1_ops (0.7+)  : l1_distance (no exact scan)       */
};
enum { HB_F32 = 0 /* vector */, HB_F16 = 1 /* halfvec */ };

enum {
    HB_OK = 0,
    HB_EINVAL = -1,    /* bad argument (dimension, m, ef_construction range, NULL pointer ...) */
    HB_ECUDA = -2,     /* CUDA runtime failure or no device */
    HB_ENOMEM = -3,    /* capacity exceeded / allocation failed */
    HB_ESTATE = -4,    /* call order (gettuple before rescan ...) */
    HB_ELIMIT = -5     /* more than HB_TIE_LIMIT exactly-equal distances at the ef boundary */
};

#define HB_HEAPTIDS 10     /* HNSW_HEAPTIDS: duplicate heap TIDs kept per element */
#define HB_MAX_DIM 2000        /* HNSW_MAX_DIM: "column cannot have more than 2000 dimensions for hnsw index" (vector) */
#define HB_MAX_DIM_HALF 4000   /* the same limit for halfvec (HNSW_MAX_DIM * 2) */
#define HB_TIE_LIMIT 4096

typedef struct hb_index hb_index;   /* one HNSW index = one partition, resident on one GPU  */
typedef struct hb_scan hb_scan;     /* IndexScanDesc->opaque (HnswScanOpaque)               */

typedef struct {
    int64_t n_dist;    /* query<->element distance evaluations */
    int64_t n_hop0;    /* elements expanded on layer 0         */
    int64_t n_hopu;    /* elements expanded on layers >= 1     */
    int64_t n_pair;    /* element<->element evaluations in neighbour selection (build) */
    int64_t n_slow;    /* queries re-run on the large-visited-set path */
} hb_counters;

const char *hb_last_error(void);
const char *hb_version(void);
/* number of CUDA devices, or HB_ECUDA */
int hb_device_count(void);

/* ---- index lifetime: hnswhandler reloptions (m, ef_construction) + opclass ---------------- */
/* m in [2,100], ef_construction in [4,1000] and >= 2m (hnsw.c reloption checks).  capacity = number of
 * elements to reserve room for (inserts beyond it grow the index, see hb_index_reserve); seed drives the
 * level draw of HnswInitElement. */
hb_index *hb_index_create(int device, int dim, int m, int ef_construction, int metric, int dtype,
                          int64_t capacity, uint64_t seed);
void hb_index_free(hb_index *ix);
int64_t hb_index_size(const hb_index *ix);          /* elements */
int hb_index_entry(const hb_index *ix, int32_t *entry, int *entry_level);

/* ---- ambuild (hnswbuild) / aminsert (hnswinsert) -------------------------------------------- */
/* Insert n tuples (vecs: n x dim of the index dtype, host; heap_tids NULL = row number).
 * hb_build on an empty index is the CREATE INDEX heap scan; hb_insert appends to a live index.
 * NULL vectors are the caller's to skip (as pgvector's BuildCallback does); zero-norm vectors are
 * skipped under HB_COSINE.  Returns the number of tuples indexed, or a negative error. */
int64_t hb_build(hb_index *ix, const void *host_vecs, int64_t n, const int64_t *heap_tids);
int64_t hb_insert(hb_index *ix, const void *host_vecs, int64_t n, const int64_t *heap_tids);
/* Grow the index to hold `capacity` elements (never shrinks).  hb_build / hb_insert call it themselves
 * when rows arrive beyond the capacity (a pgvector index has none), unless the option "auto_grow" is 0. */
int hb_index_reserve(hb_index *ix, int64_t capacity);
/* ambulkdelete, first pass (hnswvacuum.c RemoveHeapTids): the given heap TIDs leave the index; an
 * element left without TIDs keeps routing searches and returns nothing.  Returns the number of TIDs
 * removed. */
int64_t hb_bulk_delete(hb_index *ix, const int64_t *dead_tids, int64_t n_dead);
/* ambulkdelete, second and third pass (hnswvacuum.c RepairGraph + MarkDeleted): every element that points at an
 * emptied element (or whose layer-0 list is not full) gets its neighbours recomputed -- a search in which
 * emptied elements are walked through but do not count towards ef_construction (+1, it finds itself) -- and is
 * re-linked (HnswUpdateNeighborsOnDisk with checkExisting); the entry point is repaired first, or replaced by
 * the highest live element when it was emptied; then the emptied elements lose their lists and their vector.
 * Returns the number of elements marked deleted; *repaired (may be NULL) = elements re-linked.  Option
 * "vacuum_batch": elements repaired concurrently (default 2048; 1 = one after the other, the graph is then the
 * sequential algorithm's).  Slots of deleted elements are not reused by later inserts. */
int64_t hb_vacuum_repair(hb_index *ix, int64_t *repaired);
/* Free the memory only inserts use (cached neighbour distances, the pair-distance cache -- 2 kB per
 * element at m = 16 --, batch workspaces), as pgvector frees its in-memory build state when CREATE
 * INDEX ends.  Scans are unaffected; a later hb_insert allocates what it needs again. */
int hb_index_trim(hb_index *ix);
/* largest batch of the GPU insert pipeline (0 = automatic: n/16, at most 8192; 1 = the sequential
 * algorithm, graph identical to one-at-a-time insertion) */
int hb_set_build_batch(hb_index *ix, int max_batch);
/* HnswInitElement's level draw for the seq-th initialised element: (int)(-ln(U) / ln(m)), capped */
int hb_level_for(uint64_t seed, int64_t seq, int m);
/* tuning knobs: "slots" (visited-table size), "grid" (CTA cap of the persistent scans and of the exact scan;
 * the exact scan splits its work the same way under any cap, so a cap only makes each CTA run more work items and
 * the answer does not change), "build_batch",
 * "per_query_counters" (0/1), "variant" (scan kernel forced for tests: 0 automatic; 6 never the
 * four-warps-per-query kernels of small batches; 7 / 17 / 27 those kernels for every row length: default form /
 * list in shared memory / no row staging; 9 the shared-memory-list warp kernel instead of the register-list one;
 * all give identical results; any other value is refused with HB_EINVAL), "link_kernel" (reverse-link
 * kernel: 0 automatic, 1 warp per list, 2 pipelined TMA-staged, 3 memoised pair distances; all give
 * the same graph), "pair_cache" (0 = do not allocate the pair-distance cache), "pair_fill" (0 = fill
 * the cache in place instead of with the pre-pass), "eval_table" (0 = the recomputing form of the
 * reverse-link kernels), "build_fraction" (a batch is at most 1/value of the graph,
 * default 16).  0 restores the automatic choice. */
int hb_set_option(hb_index *ix, const char *name, int value);

/* ---- flat graph image (the layout in HBM; DESIGN.md "Data layout") ------------------------- */
/* Load a graph built elsewhere (e.g. by the CPU oracle, or converted from pgvector index pages).
 * vecs n x dim (normalised already when cosine); level n; nbr0 n x 2m (-1 pad); uoff n (row into
 * nbru or -1); nbru upper_rows x m; ntids n (NULL = all 1); tids n x HB_HEAPTIDS (NULL = id).
 * entry -1 with n > 0 (no entry point) is accepted only when no element holds a heap TID: the state vacuum
 * leaves after removing every element; the next insert becomes the entry point. */
int hb_index_load(hb_index *ix, int64_t n, int64_t upper_rows, int32_t entry, const void *vecs,
                  const uint8_t *level, const int32_t *nbr0, const int32_t *uoff,
                  const int32_t *nbru, const uint8_t *ntids, const int64_t *tids);
/* Load the graph from the pages of a pgvector HNSW index relation as PostgreSQL stores them (n_pages
 * x 8192 bytes: block 0 = metapage, then element / neighbour tuples; pgvector 0.7-0.8 layout AS
 * RECALLED -- see csrc/pgpages.cu).  The handle's dim, m and dtype must match the index; vectors of
 * a cosine index are stored normalised already.  Deleted elements keep their place in the graph
 * and return no tuples; a metapage without an entry point loads as hb_index_load's entry -1. */
int hb_index_load_pgvector_pages(hb_index *ix, const void *pages, int64_t n_pages);
/* what the pages hold (metapage fields, element and upper-layer row counts) -- to size hb_index_create;
 * host only, needs no device; any out pointer may be NULL */
int hb_pgvector_pages_info(const void *pages, int64_t n_pages, int *dim, int *m, int *ef_construction,
                           int64_t *n_elements, int64_t *upper_rows);
int64_t hb_index_upper_rows(const hb_index *ix);
/* any pointer may be NULL */
int hb_index_export(const hb_index *ix, void *vecs, uint8_t *level, int32_t *nbr0, int32_t *uoff,
                    int32_t *nbru, uint8_t *ntids, int64_t *tids);

/* ---- ambeginscan / amrescan / amgettuple / amendscan (hnswscan.c) -------------------------- */
hb_scan *hb_beginscan(hb_index *ix);
/* bind the ORDER BY query vector (dim components of the index dtype) and hnsw.ef_search */
int hb_rescan(hb_scan *scan, const void *host_query, int ef_search);
/* next-nearest heap TID: 1 = produced, 0 = exhausted, <0 = error.  Forward scans only. */
int hb_gettuple(hb_scan *scan, int64_t *heap_tid, float *distance);
void hb_endscan(hb_scan *scan);
/* hnsw.iterative_scan (pgvector 0.8): HB_ITER_OFF = amgettuple stops after the ef_search results;
 * HB_ITER_RELAXED / HB_ITER_STRICT = when they are consumed the scan resumes from the candidates it
 * discarded (ResumeScanItems) until the index is exhausted; after max_scan_tuples visited tuples
 * the remaining discarded candidates are returned without further search.  STRICT drops tuples
 * that are nearer than one already returned.  Call between hb_beginscan and the first hb_gettuple
 * (it applies to every later hb_rescan of this scan). */
enum { HB_ITER_OFF = 0, HB_ITER_RELAXED = 1, HB_ITER_STRICT = 2 };
int hb_scan_set_iterative(hb_scan *scan, int mode, int64_t max_scan_tuples);

/* ---- resumable scans, batched ---------------------------------------------------------------- */
/* The same thing for nq queries at once.  hb_iter_next returns each query's next batch of elements
 * nearest-first (elem/dist: nq x ef_search host arrays, padded with -1 / +inf; cnt: nq): first the
 * GetScanItems result, then one ResumeScanItems batch per call, then -- past max_scan_tuples --
 * the leftover candidates one per call.  Return value: total elements produced (0 = every scan is
 * exhausted), negative on error.  State per query lives in HBM (visited bitmap of n bits and the
 * discarded list); hb_iter_begin fails with HB_ENOMEM when nq of them do not fit. */
typedef struct hb_iter hb_iter;
hb_iter *hb_iter_begin(hb_index *ix, const void *host_queries, int64_t nq, int ef_search, int64_t max_scan_tuples);
int64_t hb_iter_next(hb_iter *it, int32_t *elem, float *dist, int32_t *cnt);
int hb_iter_tuples(hb_iter *it, int64_t *tuples /* nq: upstream's `tuples` counter */);
void hb_iter_end(hb_iter *it);
/* Filtered top-k on top of the resumable scans (what hnsw.iterative_scan is for): scans continue
 * until k heap TIDs whose bit is set in allowed_bits (bit t = TID t, n_bits bits) were found, the
 * index is exhausted or max_scan_tuples was reached.  relaxed_order.  out_tids/out_dist nq x k
 * (-1 / +inf padded), out_cnt nq. */
int hb_search_batch_filtered(hb_index *ix, const void *host_queries, int64_t nq, int ef_search, int k,
                             const uint8_t *allowed_bits, int64_t n_bits, int64_t max_scan_tuples,
                             int64_t *out_tids, float *out_dist, int32_t *out_cnt);

/* ---- batched scan (the extension a GPU needs: many amrescan+amgettuple at once) ------------ */
/* host buffers in, host buffers out; H2D and D2H copies happen inside.  For each of nq queries
 * writes the first k heap TIDs nearest-first (pad: -1 / +inf) and the count. */
int hb_search_batch(hb_index *ix, const void *host_queries, int64_t nq, int ef_search, int k,
                    int64_t *out_tids, float *out_dist, int32_t *out_cnt);
/* asynchronous form: the H2D copy, scan, TID mapping and D2H copy are queued on the stream of
 * `slot` (0..3) and the call returns; hb_search_batch_wait(slot) completes it.  Batches in
 * different slots overlap (copies under scans, one batch's tail under the next one's ramp).  Host
 * buffers must stay valid -- and be pinned for the copies to overlap -- until the wait. */
int hb_search_batch_async(hb_index *ix, int slot, const void *host_queries, int64_t nq, int ef_search,
                          int k, int64_t *out_tids, float *out_dist, int32_t *out_cnt);
int hb_search_batch_wait(hb_index *ix, int slot);
/* as above but returns elements (graph node ids), ef per query: out_elem/out_dist nq x ef */
int hb_search_batch_elements(hb_index *ix, const void *host_queries, int64_t nq, int ef_search,
                             int32_t *out_elem, float *out_dist, int32_t *out_cnt);
/* device-resident: queries already in HBM (nq x dim, index dtype), results left in HBM;
 * asynchronous on `stream` (a cudaStream_t passed as void*; NULL = default stream).  Calls on
 * different streams may be in flight together (each stream gets its own workspace).
 * dev_out_elem / dev_out_dist: nq x ef; dev_out_cnt: nq. */
int hb_search_batch_dev(hb_index *ix, const void *dev_queries, int64_t nq, int ef_search,
                        int32_t *dev_out_elem, float *dev_out_dist, int32_t *dev_out_cnt,
                        void *stream);
/* waits for `stream` and returns the status of the last hb_search_batch_dev queued on it: HB_ELIMIT when a query
 * of that batch had more than HB_TIE_LIMIT candidates tying at the ef boundary (its result count is 0) */
int hb_search_batch_status(hb_index *ix, void *stream);
/* one HnswSearchLayer call from explicit entry points (unit-test surface of the layer kernel):
 * ep nq x nep element ids; out nq x max(ef,nep) */
int hb_search_layer(hb_index *ix, const void *host_queries, int64_t nq, const int32_t *ep, int nep,
                    int ef, int layer, int32_t *out_elem, float *out_dist, int32_t *out_cnt);
/* counters accumulated since the last reset (algorithmic bytes for the roofline come from these) */
int hb_get_counters(hb_index *ix, hb_counters *out, int reset);
/* per-query counters of the last batch (needs option per_query_counters = 1): nq x 4 int32 =
 * n_dist, n_hop0, n_hopu, 1 if the query ran on the large-visited-set path */
int hb_get_per_query_counters(hb_index *ix, int64_t nq, int32_t *out);
/* device time (ms) of the most recent search kernel launch sequence on the index's own events */
float hb_last_search_ms(const hb_index *ix);

/* ---- opclass support functions, batched --------------------------------------------------- */
/* FUNCTION 1: distances from each of nq queries to its own list of nc candidate elements
 * (cand nq x nc, ids < 0 give +inf).  The query-vs-neighbour-list kernel on its own. */
int hb_distance_batch(hb_index *ix, const void *host_queries, int64_t nq, const int32_t *cand,
                      int nc, float *out_dist);
/* device-resident form (queries nq x dim, cand nq x nc, out nq x nc all in HBM; queries must be
 * normalised already under the cosine opclass); asynchronous on stream */
int hb_distance_batch_dev(hb_index *ix, const void *dev_queries, int64_t nq, const int32_t *dev_cand,
                          int nc, float *dev_out, void *stream);
/* FUNCTION 2 + l2_normalize: n x dim in, n x dim out (index dtype), ok[i] = 0 for zero norm */
int hb_normalize(hb_index *ix, const void *host_in, int64_t n, void *host_out, uint8_t *ok);

/* ---- exact scan of a partition (recall ground truth; bf16 tcgen05 GEMM + fp32 re-rank) ------ */
int hb_bruteforce(hb_index *ix, const void *host_queries, int64_t nq, int k, int32_t *out_elem,
                  float *out_dist);
/* same, with diagnostics: dbg_scores (optional, host, nq x n) receives the raw bf16 GEMM scores;
 * stats (optional, 3 floats): queries certified exact by the bf16 error bound, queries re-scanned
 * exhaustively in fp32, GEMM kernel milliseconds.  1 <= k <= 128.  Either way the answer is the exact top-k
 * of the canonical fp32 distance (FUNCTION 1) by (distance, element id), padded with -1 / +inf when n < k.
 * hb_set_option(ix, "grid", g) caps the GEMM kernel's CTAs at g. */
int hb_bruteforce_ex(hb_index *ix, const void *host_queries, int64_t nq, int k, int32_t *out_elem,
                     float *out_dist, float *dbg_scores, float *stats);

/* ---- partition routing / merge -------------------------------------------------------------- */
/* partition of a heap TID / row id: splitmix64(id) mod n_partitions */
int hb_partition_of(int64_t id, int n_partitions);
void hb_partition_route(const int64_t *ids, int64_t n, int n_partitions, int32_t *out_part);
/* merge P per-partition top-k lists (dev_tids / dev_dist: P x nq x k, nearest-first, pad -1/+inf)
 * into nq x k on the device; asynchronous on stream. */
int hb_merge_topk_dev(int device, const int64_t *dev_tids, const float *dev_dist, int n_parts,
                      int64_t nq, int k, int64_t *dev_out_tids, float *dev_out_dist, void *stream);
/* map element ids to the first k heap TIDs on the device (nq x ef elements -> nq x k tids) */
int hb_elements_to_tids_dev(hb_index *ix, const int32_t *dev_elem, const float *dev_dist,
                            int64_t nq, int ef, int k, int64_t *dev_out_tids, float *dev_out_dist,
                            void *stream);

/* ---- the partitioned index (the fork's feature): P hash partitions over `world` GPUs -------------- */
/* One process per GPU.  A row belongs to partition splitmix64(heap_tid) mod P; rank r owns the partitions
 * {p : p mod world == r}, each an ordinary hb_index on the rank's GPU.  A search sends the same query batch
 * to every partition, merges the owned partitions' top-k on the device, exchanges the per-rank lists (12 bytes
 * per result) and merges again: every rank ends with the same nq x k answer, ordered by (distance, heap TID).
 * The exchange is an all-gather done with stores into the peers' memory over NVLink (buffers mapped through CUDA
 * IPC, epoch flags instead of a collective kernel) or, with hb_part_set_option("exchange", 0) or when peer mapping
 * is not possible, ONE ncclAllGather.  The handle owns the NCCL communicator (NCCL is dlopen'ed when world > 1);
 * all ranks must make the same sequence of hb_part_search_* calls, as in any NCCL program.  No CPU fallback. */
typedef struct hb_part hb_part;
#define HB_PART_ID_BYTES 128   /* sizeof(ncclUniqueId) */
#define HB_PART_SLOTS 4        /* search batches that can be in flight */
/* rank 0 obtains the communicator id and hands it to the other ranks by whatever means the host has
 * (Postgres shared memory, a file, torch.distributed ...) */
int hb_part_unique_id(void *id_out /* HB_PART_ID_BYTES */);
/* collective when world > 1 (ncclCommInitRank); unique_id may be NULL when world == 1.  Partition p draws
 * its levels from seed + p, whichever rank builds it. */
hb_part *hb_part_create(int device, int dim, int m, int ef_construction, int metric, int dtype, int n_partitions,
                        int64_t capacity_per_partition, uint64_t seed, int rank, int world, const void *unique_id);
void hb_part_free(hb_part *pt);
/* partitions this rank owns (ascending) -> count; partitions may be NULL */
int hb_part_owned(const hb_part *pt, int32_t *partitions);
/* the hb_index of an owned partition (owned by the hb_part; NULL when another rank owns it) */
hb_index *hb_part_index(hb_part *pt, int partition);
int64_t hb_part_size(const hb_part *pt);            /* elements over the owned partitions */
int hb_part_set_option(hb_part *pt, const char *name, int value);   /* "exchange" (see above), else hb_set_option on every owned partition */
int hb_part_get_counters(hb_part *pt, hb_counters *out, int reset); /* summed over the owned partitions */
/* ambuild / aminsert: every rank passes the same tuples (or any superset of those it owns); each tuple is
 * indexed by the owner of its partition, owned partitions are built concurrently, no collective.  Returns the
 * number of tuples this rank indexed. */
int64_t hb_part_build(hb_part *pt, const void *host_vecs, int64_t n, const int64_t *heap_tids);
/* Batched ORDER BY ... LIMIT k over all partitions, asynchronous: queued on slot `slot` (0..HB_PART_SLOTS-1),
 * completed by hb_part_search_wait.  root < 0: `queries` (nq x dim, index dtype) holds the batch on every
 * rank already; root >= 0: only rank `root` passes queries and they are ncclBroadcast to the others first.
 * queries_on_device / out_on_device: the buffers are device memory of this rank's GPU (ready when the call is
 * made) instead of host memory (pinned for the copies to overlap).  out_tids / out_dist: nq x k, padded with
 * -1 / +inf; every rank receives the full answer.  Buffers must stay valid until the wait. */
int hb_part_search_async(hb_part *pt, int slot, const void *queries, int queries_on_device, int root, int64_t nq,
                         int ef_search, int k, int64_t *out_tids, float *out_dist, int out_on_device);
int hb_part_search_wait(hb_part *pt, int slot);
/* synchronous, host buffers: slot 0 + wait */
int hb_part_search(hb_part *pt, const void *host_queries, int root, int64_t nq, int ef_search, int k,
                   int64_t *out_tids, float *out_dist);

#ifdef __cplusplus
}
#endif
#endif
