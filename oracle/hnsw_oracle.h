/*
 * hnsw_oracle.h -- CPU oracle for the HNSW hot path.  TEST INFRASTRUCTURE ONLY.
 *
 * PARITY UNPINNED: /root/reference holds a single 5-byte README (README.md:1, "# pg") and no
 * source, tests or golden vectors, and there is no PostgreSQL in the image.  This oracle therefore
 * restates the HNSW semantics of upstream pgvector (hnswutils.c / hnswbuild.c / hnswscan.c /
 * vector.c / halfutils.c, v0.7-0.8) from memory plus Malkov & Yashunin (arXiv:1603.09320,
 * Alg. 1/2/4/5).  No reference file:line can be cited beyond README.md:1; each function below
 * names the upstream function it restates instead.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
 * load this library.  The product path (pgvector-hnsw-partitioning_b200/) never links or calls it.
 */
#ifndef HNSW_ORACLE_H
#define HNSW_ORACLE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { ORC_L2 = 0, ORC_IP = 1, ORC_COSINE = 2, ORC_L1 = 3 };   /* vector_l2_ops / vector_ip_ops / vector_cosine_ops / vector_l1_ops */
enum { ORC_F32 = 0, ORC_F16 = 1 };                 /* vector / halfvec storage */
/* distance summation order:
 *   ORC_DIST_CANON   = the fixed 32-lane x VEC-accumulator FMA order + butterfly tree the CUDA
 *                      kernels use, so distances (and hence ids) can be compared bit-exactly;
 *   ORC_DIST_NATURAL = pgvector's plain scalar loop, compiled with its Makefile's flags
 *                      (-ftree-vectorize -fassociative-math ...), used for CPU timing and for the
 *                      tolerance-based comparison. */
enum { ORC_DIST_CANON = 0, ORC_DIST_NATURAL = 1 };

#define ORC_HEAPTIDS 10   /* HNSW_HEAPTIDS: heap TIDs (duplicates) per element */

typedef struct OrcIndex OrcIndex;

typedef struct {
    int64_t n_dist;    /* distance evaluations query<->element (incl. the entry point)      */
    int64_t n_hop0;    /* nodes expanded at layer 0                                         */
    int64_t n_hopu;    /* nodes expanded at layers >= 1                                     */
    int64_t n_pair;    /* element<->element evaluations (CheckElementCloser), build only    */
} OrcCounters;

OrcIndex *orc_create(int dim, int m, int ef_construction, int metric, int dtype, int dist_mode,
                     uint64_t seed);
void orc_free(OrcIndex *ix);
void orc_set_dist_mode(OrcIndex *ix, int dist_mode);

/* level of the seq-th initialised element: (int)(-log(U) * 1/ln(m)), capped (HnswInitElement) */
int orc_level_for(uint64_t seed, int64_t seq, int m);
int orc_max_level(int m);
/* partition routing used by the fork-level spec: splitmix64(id) mod P */
uint64_t orc_splitmix64(uint64_t x);

/* hnswbuild.c InsertTuple (in-memory build phase).  vec: dim floats (ORC_F32) or dim IEEE halfs.
 * Returns the element id the tuple landed in (a new one, or an existing duplicate's), -1 if the
 * tuple was skipped (cosine opclass and zero norm), -2 on error. */
int64_t orc_insert(OrcIndex *ix, const void *vec, int64_t heap_tid);
int64_t orc_build(OrcIndex *ix, const void *vecs, int64_t n, const int64_t *heap_tids);

/* hnswvacuum.c [RECALL]: ambulkdelete = RemoveHeapTids (orc_bulk_delete: returns the TIDs removed), then
 * RepairGraph + MarkDeleted (orc_vacuum_repair: elements without heap TIDs stop counting towards ef, every element
 * that points at one -- or whose layer 0 is not full -- gets its neighbours recomputed (HnswFindElementNeighbors with
 * existing = true) and re-linked, the entry point moves if it was deleted; then the emptied elements are unlinked
 * and zeroed.  Returns the number of elements marked deleted; *repaired = elements re-linked). */
int64_t orc_bulk_delete(OrcIndex *ix, const int64_t *dead_tids, int64_t n_dead);
int64_t orc_vacuum_repair(OrcIndex *ix, int64_t *repaired);

/* hnswscan.c GetScanItems: entry -> greedy descent (ef=1) -> layer-0 search (ef_search).
 * Writes up to ef (element, distance) pairs nearest-first; returns the count. */
int orc_search_elements(const OrcIndex *ix, const void *query, int ef, int32_t *out_elem,
                        float *out_dist, OrcCounters *ctr);
/* hnswgettuple streaming: heap TIDs nearest-first, first k of them. Returns count. */
int orc_search_tids(const OrcIndex *ix, const void *query, int ef, int k, int64_t *out_tids,
                    float *out_dist, OrcCounters *ctr);
/* many queries, `threads` OpenMP threads over disjoint queries (N concurrent backends).
 * out_elem/out_dist are nq x ef (padded with -1 / +inf); out_cnt nq. ctr (nullable) is summed. */
void orc_search_batch(const OrcIndex *ix, const void *queries, int64_t nq, int ef, int32_t *out_elem,
                      float *out_dist, int32_t *out_cnt, OrcCounters *ctr, int threads);

/* hnsw.iterative_scan (pgvector 0.8 hnswscan.c GetScanItems with `discarded` + ResumeScanItems):
 * orc_iter_next returns the next batch of elements nearest-first -- first the ef results of
 * GetScanItems, then one ResumeScanItems batch per call; after `tuples` reached max_scan_tuples the
 * remaining discarded candidates come one per call.  0 = exhausted.  out_* hold ef entries. */
typedef struct OrcIter OrcIter;
OrcIter *orc_iter_begin(const OrcIndex *ix, const void *query, int ef, int64_t max_scan_tuples);
int orc_iter_next(OrcIter *it, int32_t *out_elem, float *out_dist);
int64_t orc_iter_tuples(const OrcIter *it);
int64_t orc_iter_discarded(const OrcIter *it);
void orc_iter_counters(const OrcIter *it, OrcCounters *out);
void orc_iter_end(OrcIter *it);

/* one HnswSearchLayer call on an explicit entry list (for unit tests of the layer kernel) */
int orc_search_layer(const OrcIndex *ix, const void *query, const int32_t *ep, int nep, int ef,
                     int lc, int32_t *out_elem, float *out_dist, OrcCounters *ctr);

/* exact top-k by the opclass distance accumulated in double (recall ground truth) over the stored
 * (normalised for cosine) vectors; ties by element id. out: nq x k. */
void orc_bruteforce(const OrcIndex *ix, const void *queries, int64_t nq, int k, int32_t *out_elem,
                    double *out_dist, int threads);
/* exact top-k in the library's own arithmetic (the exact scan's contract): every row's canonical fp32
 * FUNCTION 1 distance (dist_q_row; cosine queries normalised as by the scans), the k smallest by
 * (distance, element id), padded with -1 / +inf when n < k.  out: nq x k. */
void orc_exact_topk(const OrcIndex *ix, const void *queries, int64_t nq, int k, int32_t *out_elem,
                    float *out_dist, int threads);

/* scalar entry points (vector.c / halfutils.c support functions); metric_is_ip: 0 = squared l2,
 * 1 = negative inner product, ORC_L1 = l1 */
float orc_distance(int metric_is_ip, int dtype, int dist_mode, int dim, const void *a, const void *b);
/* l2_normalize; returns 0 if the norm is zero (HnswCheckNorm fails) */
int orc_normalize(int dtype, int dist_mode, int dim, const void *in, void *out);

/* flat graph image (same layout the CUDA library loads) */
int64_t orc_n(const OrcIndex *ix);
int64_t orc_upper_rows(const OrcIndex *ix);
int32_t orc_entry(const OrcIndex *ix);
int orc_entry_level(const OrcIndex *ix);
void orc_counters(const OrcIndex *ix, OrcCounters *out);   /* build-side totals */
/* vecs: n x dim (stored dtype); level: n; nbr0: n x 2m (-1 pad); uoff: n (row into nbru or -1);
 * nbru: upper_rows x m; ntids: n; tids: n x ORC_HEAPTIDS.  Any pointer may be NULL. */
void orc_export(const OrcIndex *ix, void *vecs, uint8_t *level, int32_t *nbr0, int32_t *uoff,
                int32_t *nbru, uint8_t *ntids, int64_t *tids);
/* build an index object around an existing graph (e.g. one built on the GPU) */
OrcIndex *orc_import(int dim, int m, int ef_construction, int metric, int dtype, int dist_mode,
                     int64_t n, int64_t upper_rows, int32_t entry, const void *vecs,
                     const uint8_t *level, const int32_t *nbr0, const int32_t *uoff,
                     const int32_t *nbru, const uint8_t *ntids, const int64_t *tids);

#ifdef __cplusplus
}
#endif
#endif
