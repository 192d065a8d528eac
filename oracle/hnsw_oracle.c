/*
 * hnsw_oracle.c -- CPU restatement of pgvector's HNSW hot path.  TEST INFRASTRUCTURE ONLY
 * (see hnsw_oracle.h: parity unpinned, /root/reference/README.md:1 is the entire reference).
 *
 * Upstream functions restated here [RECALL = from memory of pgvector v0.7-0.8, unverifiable in
 * this container] and [PAPER = arXiv:1603.09320]:
 *   search_layer()            <- hnswutils.c HnswSearchLayer            [PAPER Alg. 2]
 *   find_element_neighbors()  <- hnswutils.c HnswFindElementNeighbors   [PAPER Alg. 1]
 *   select_neighbors()        <- hnswutils.c SelectNeighbors + CheckElementCloser [PAPER Alg. 4,
 *                                keepPrunedConnections]
 *   update_connection()       <- hnswutils.c HnswUpdateConnection
 *   orc_insert()              <- hnswbuild.c InsertTupleInMemory / UpdateGraphInMemory /
 *                                FindDuplicateInMemory
 *   orc_search_elements()     <- hnswscan.c GetScanItems                [PAPER Alg. 5]
 *   orc_search_tids()         <- hnswscan.c hnswgettuple
 *   orc_level_for()           <- hnswutils.c HnswInitElement, HnswGetMaxLevel
 *   canonical/natural dist    <- vector.c / halfutils.c support functions
 *
 * Choices pgvector leaves to its pairing heap (order among equal distances) are made
 * deterministic here: every ordering is by the key (distance, element id).  The admission and
 * termination tests compare distances only, exactly as upstream does
 * (`eDistance < f->distance || alwaysAdd`, `c->distance > f->distance`).
 */
#include "hnsw_oracle.h"

#include <immintrin.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* ---- dist_natural.c ---- */
float orc_nat_l2_f32(int dim, const float *ax, const float *bx);
float orc_nat_ip_f32(int dim, const float *ax, const float *bx);
float orc_nat_l2_f16(int dim, const float *ax, const uint16_t *bx);
float orc_nat_ip_f16(int dim, const float *ax, const uint16_t *bx);
float orc_nat_l1_f32(int dim, const float *ax, const float *bx);
float orc_nat_l1_f16(int dim, const float *ax, const uint16_t *bx);
double orc_nat_sqnorm_f32(int dim, const float *ax);

typedef struct { float d; int32_t id; } Cand;

struct OrcIndex {
    int dim, m, efc, metric, dtype, dist_mode;
    int esize;                 /* bytes per stored component */
    uint64_t seed;
    int64_t n, cap, seq;
    char *vecs;                /* n x dim, stored dtype, normalised when cosine */
    uint8_t *level;
    int32_t *nbr0; float *nbr0d; uint8_t *cnt0;        /* n x 2m, cached distances, lengths */
    int32_t *uoff;                                      /* n: first row in the upper table or -1 */
    int32_t *nbru; float *nbrud; uint8_t *cntu;         /* urows x m */
    int64_t urows, ucap;
    uint8_t *ntids; int64_t *tids;                      /* n x ORC_HEAPTIDS */
    uint8_t *deleted;                                   /* HnswElementTupleData.deleted (set by vacuum's MarkDeleted) */
    int32_t entry; int entry_level;
    int stale_d;               /* cached distances unknown (imported graph): recomputed before the next insert */
    OrcCounters ctr;
};

/* ------------------------------------------------------------------ distances */

static inline int key_lt(Cand a, Cand b) { return a.d < b.d || (a.d == b.d && a.id < b.id); }

/* Canonical order (shared with the CUDA kernels, csrc/distance.cuh): component e of a row goes
 * to accumulator e mod (32*VEC), VEC = components per 16 bytes (4 fp32, 8 fp16); accumulators
 * are FMA chains in increasing e; a lane's VEC accumulators fold pairwise; the 32 lane partials
 * fold by the xor-butterfly 16,8,4,2,1. */
static float canon_fold(const float *acc, int vec)
{
    float p[32];
    if (vec == 4)
        for (int l = 0; l < 32; l++)
            p[l] = (acc[4 * l] + acc[4 * l + 1]) + (acc[4 * l + 2] + acc[4 * l + 3]);
    else
        for (int l = 0; l < 32; l++)
            p[l] = ((acc[8 * l] + acc[8 * l + 1]) + (acc[8 * l + 2] + acc[8 * l + 3])) +
                   ((acc[8 * l + 4] + acc[8 * l + 5]) + (acc[8 * l + 6] + acc[8 * l + 7]));
    for (int s = 16; s >= 1; s >>= 1)
        for (int l = 0; l < s; l++)
            p[l] = p[l] + p[l + s];
    return p[0];
}

static float canon_l2(int dim, const float *a, const float *b, int vec)
{
    float acc[256];
    int w = 32 * vec;
    memset(acc, 0, sizeof(float) * w);
    int full = dim / w * w;
    for (int base = 0; base < full; base += w)
        for (int j = 0; j < w; j++) {
            float t = a[base + j] - b[base + j];
            acc[j] = fmaf(t, t, acc[j]);
        }
    for (int j = 0; full + j < dim; j++) {
        float t = a[full + j] - b[full + j];
        acc[j] = fmaf(t, t, acc[j]);
    }
    return canon_fold(acc, vec);
}

static float canon_ip(int dim, const float *a, const float *b, int vec)
{
    float acc[256];
    int w = 32 * vec;
    memset(acc, 0, sizeof(float) * w);
    int full = dim / w * w;
    for (int base = 0; base < full; base += w)
        for (int j = 0; j < w; j++)
            acc[j] = fmaf(a[base + j], b[base + j], acc[j]);
    for (int j = 0; full + j < dim; j++)
        acc[j] = fmaf(a[full + j], b[full + j], acc[j]);
    return canon_fold(acc, vec);
}

/* vector_l1_distance (pgvector 0.7 VectorL1Distance): sum of |a - b|, canonical order, plain adds */
static float canon_l1(int dim, const float *a, const float *b, int vec)
{
    float acc[256];
    int w = 32 * vec;
    memset(acc, 0, sizeof(float) * w);
    for (int e = 0; e < dim; e++)
        acc[e % w] = acc[e % w] + fabsf(a[e] - b[e]);
    return canon_fold(acc, vec);
}

/* squared norm in double, canonical order (products of two floats are exact in double, so only
 * the addition order matters) */
static double canon_sqnorm(int dim, const float *a, int vec)
{
    double acc[256];
    int w = 32 * vec;
    for (int j = 0; j < w; j++) acc[j] = 0.0;
    for (int e = 0; e < dim; e++)
        acc[e % w] += (double) a[e] * (double) a[e];
    double p[32];
    for (int l = 0; l < 32; l++) {
        const double *c = acc + vec * l;
        if (vec == 4) p[l] = (c[0] + c[1]) + (c[2] + c[3]);
        else p[l] = ((c[0] + c[1]) + (c[2] + c[3])) + ((c[4] + c[5]) + (c[6] + c[7]));
    }
    for (int s = 16; s >= 1; s >>= 1)
        for (int l = 0; l < s; l++) p[l] = p[l] + p[l + s];
    return p[0];
}

static void half_to_float(int dim, const uint16_t *h, float *f)
{
    int i = 0;
    for (; i + 8 <= dim; i += 8)
        _mm256_storeu_ps(f + i, _mm256_cvtph_ps(_mm_loadu_si128((const __m128i *) (h + i))));
    for (; i < dim; i++) f[i] = _cvtsh_ss(h[i]);
}

/* distance between a float query and a stored row (the opclass's FUNCTION 1:
 * vector_l2_squared_distance / vector_negative_inner_product and halfvec equivalents) */
static float dist_q_row(const OrcIndex *ix, const float *q, const void *row)
{
    int ip = ix->metric == ORC_IP || ix->metric == ORC_COSINE;
    float r;
    if (ix->metric == ORC_L1) {
        if (ix->dist_mode == ORC_DIST_NATURAL)
            return ix->dtype == ORC_F32 ? orc_nat_l1_f32(ix->dim, q, (const float *) row)
                                        : orc_nat_l1_f16(ix->dim, q, (const uint16_t *) row);
        if (ix->dtype == ORC_F32) return canon_l1(ix->dim, q, (const float *) row, 4);
        float tmp[ix->dim];
        half_to_float(ix->dim, (const uint16_t *) row, tmp);
        return canon_l1(ix->dim, q, tmp, 8);
    }
    if (ix->dist_mode == ORC_DIST_NATURAL) {
        if (ix->dtype == ORC_F32)
            r = ip ? orc_nat_ip_f32(ix->dim, q, (const float *) row)
                   : orc_nat_l2_f32(ix->dim, q, (const float *) row);
        else
            r = ip ? orc_nat_ip_f16(ix->dim, q, (const uint16_t *) row)
                   : orc_nat_l2_f16(ix->dim, q, (const uint16_t *) row);
    } else if (ix->dtype == ORC_F32) {
        r = ip ? canon_ip(ix->dim, q, (const float *) row, 4)
               : canon_l2(ix->dim, q, (const float *) row, 4);
    } else {
        float tmp[ix->dim];
        half_to_float(ix->dim, (const uint16_t *) row, tmp);
        r = ip ? canon_ip(ix->dim, q, tmp, 8) : canon_l2(ix->dim, q, tmp, 8);
    }
    return ip ? -r : r;
}

static inline const void *row_of(const OrcIndex *ix, int64_t e)
{
    return ix->vecs + (size_t) e * ix->dim * ix->esize;
}

static void row_as_float(const OrcIndex *ix, int64_t e, float *out)
{
    if (ix->dtype == ORC_F32) memcpy(out, row_of(ix, e), sizeof(float) * ix->dim);
    else half_to_float(ix->dim, (const uint16_t *) row_of(ix, e), out);
}

float orc_distance(int metric_is_ip, int dtype, int dist_mode, int dim, const void *a, const void *b)
{
    OrcIndex t;
    memset(&t, 0, sizeof t);
    /* 0 = l2, 1 = negative inner product, ORC_L1 = l1 */
    t.dim = dim; t.metric = metric_is_ip == ORC_L1 ? ORC_L1 : (metric_is_ip ? ORC_IP : ORC_L2); t.dtype = dtype; t.dist_mode = dist_mode;
    float qa[dim];
    if (dtype == ORC_F32) memcpy(qa, a, sizeof(float) * dim);
    else half_to_float(dim, (const uint16_t *) a, qa);
    return dist_q_row(&t, qa, b);
}

/* l2_normalize (vector.c / halfvec.c): norm in double, x / norm rounded to the stored type */
int orc_normalize(int dtype, int dist_mode, int dim, const void *in, void *out)
{
    float f[dim];
    if (dtype == ORC_F32) memcpy(f, in, sizeof(float) * dim);
    else half_to_float(dim, (const uint16_t *) in, f);
    double sq = dist_mode == ORC_DIST_NATURAL ? orc_nat_sqnorm_f32(dim, f)
                                               : canon_sqnorm(dim, f, dtype == ORC_F32 ? 4 : 8);
    double norm = sqrt(sq);
    if (!(norm > 0.0)) {
        memcpy(out, in, (size_t) dim * (dtype == ORC_F32 ? 4 : 2));
        return 0;
    }
    if (dtype == ORC_F32) {
        float *o = (float *) out;
        for (int i = 0; i < dim; i++) o[i] = (float) ((double) f[i] / norm);
    } else {
        uint16_t *o = (uint16_t *) out;
        for (int i = 0; i < dim; i++)
            o[i] = _cvtss_sh((float) ((double) f[i] / norm), _MM_FROUND_TO_NEAREST_INT);
    }
    return 1;
}

/* ------------------------------------------------------------------ helpers */

uint64_t orc_splitmix64(uint64_t x)
{
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}

/* HnswGetMaxLevel: what fits the neighbour tuple on an 8 kB page, capped at 255 */
int orc_max_level(int m)
{
    int v = (8192 - 24 - 8 - 8 - 4) / 6 / m - 2;
    return v > 255 ? 255 : (v < 0 ? 0 : v);
}

int orc_level_for(uint64_t seed, int64_t seq, int m)
{
    uint64_t r = orc_splitmix64(seed ^ orc_splitmix64((uint64_t) seq));
    double u = ((double) (r >> 11) + 1.0) * (1.0 / 9007199254740992.0);   /* (0,1] */
    double ml = 1.0 / log((double) m);
    int level = (int) (-log(u) * ml);
    int mx = orc_max_level(m);
    return level > mx ? mx : level;
}

static inline int layer_m(const OrcIndex *ix, int lc) { return lc == 0 ? 2 * ix->m : ix->m; }

static inline int32_t *nbrs(const OrcIndex *ix, int64_t e, int lc, float **d, uint8_t **cnt)
{
    if (lc == 0) {
        if (d) *d = ix->nbr0d + e * 2 * ix->m;
        *cnt = ix->cnt0 + e;
        return ix->nbr0 + e * 2 * ix->m;
    }
    int64_t row = (int64_t) ix->uoff[e] + (lc - 1);
    if (d) *d = ix->nbrud + row * ix->m;
    *cnt = ix->cntu + row;
    return ix->nbru + row * ix->m;
}

/* ------------------------------------------------------------------ scratch */

typedef struct {
    uint32_t *stamp; int64_t stamp_n; uint32_t epoch;     /* visited set */
    Cand *C; int nC, capC;                                /* min-heap of candidates */
    Cand *W; int nW, capW;                                /* max-heap of results */
} Scratch;

static void scratch_init(Scratch *s) { memset(s, 0, sizeof *s); }
static void scratch_free(Scratch *s) { free(s->stamp); free(s->C); free(s->W); }
static void scratch_begin(Scratch *s, int64_t n, int ef)
{
    if (s->stamp_n < n) {
        free(s->stamp);
        s->stamp_n = n + n / 2 + 1024;
        s->stamp = (uint32_t *) calloc((size_t) s->stamp_n, sizeof(uint32_t));
        s->epoch = 0;
    }
    if (++s->epoch == 0) { memset(s->stamp, 0, sizeof(uint32_t) * s->stamp_n); s->epoch = 1; }
    if (s->capW < ef + 2) { s->capW = ef + 2; s->W = (Cand *) realloc(s->W, sizeof(Cand) * s->capW); }
    s->nC = s->nW = 0;
}
static void c_push(Scratch *s, Cand c)
{
    if (s->nC == s->capC) { s->capC = s->capC ? 2 * s->capC : 256; s->C = (Cand *) realloc(s->C, sizeof(Cand) * s->capC); }
    int i = s->nC++;
    while (i > 0) { int p = (i - 1) / 2; if (!key_lt(c, s->C[p])) break; s->C[i] = s->C[p]; i = p; }
    s->C[i] = c;
}
static Cand c_pop(Scratch *s)
{
    Cand top = s->C[0], last = s->C[--s->nC];
    int i = 0;
    for (;;) {
        int l = 2 * i + 1, r = l + 1, b = i; Cand bv = last;
        if (l < s->nC && key_lt(s->C[l], bv)) { b = l; bv = s->C[l]; }
        if (r < s->nC && key_lt(s->C[r], bv)) { b = r; bv = s->C[r]; }
        if (b == i) break;
        s->C[i] = s->C[b]; i = b;
    }
    if (s->nC > 0) s->C[i] = last;
    return top;
}
static void w_push(Scratch *s, Cand c)
{
    int i = s->nW++;
    while (i > 0) { int p = (i - 1) / 2; if (!key_lt(s->W[p], c)) break; s->W[i] = s->W[p]; i = p; }
    s->W[i] = c;
}
static Cand w_pop(Scratch *s)
{
    Cand top = s->W[0], last = s->W[--s->nW];
    int i = 0;
    for (;;) {
        int l = 2 * i + 1, r = l + 1, b = i; Cand bv = last;
        if (l < s->nW && key_lt(bv, s->W[l])) { b = l; bv = s->W[l]; }
        if (r < s->nW && key_lt(bv, s->W[r])) { b = r; bv = s->W[r]; }
        if (b == i) break;
        s->W[i] = s->W[b]; i = b;
    }
    if (s->nW > 0) s->W[i] = last;
    return top;
}

/* ------------------------------------------------------------------ HnswSearchLayer */

/* ep: entry candidates with distances already computed.  out: up to ef results, NEAREST first
 * (upstream returns the list furthest-first and consumes it from the tail; callers here index
 * from the front).  Returns the count. */
/* discarded candidates of an iterative scan (pgvector 0.8 HnswSearchLayer `discarded`): a min-heap
 * on (distance, id) of everything that was visited but is not in W */
typedef struct { Cand *a; int n, cap; } Disc;
static void disc_push(Disc *h, Cand c)
{
    if (h->n == h->cap) { h->cap = h->cap ? 2 * h->cap : 1024; h->a = (Cand *) realloc(h->a, sizeof(Cand) * h->cap); }
    int i = h->n++;
    while (i > 0) { int p = (i - 1) / 2; if (!key_lt(c, h->a[p])) break; h->a[i] = h->a[p]; i = p; }
    h->a[i] = c;
}
static Cand disc_pop(Disc *h)
{
    Cand top = h->a[0], last = h->a[--h->n];
    int i = 0;
    for (;;) {
        int l = 2 * i + 1, r = l + 1, b = i; Cand bv = last;
        if (l < h->n && key_lt(h->a[l], bv)) { b = l; bv = h->a[l]; }
        if (r < h->n && key_lt(h->a[r], bv)) { b = r; bv = h->a[r]; }
        if (b == i) break;
        h->a[i] = h->a[b]; i = b;
    }
    if (h->n > 0) h->a[i] = last;
    return top;
}

/* disc (nullable): evicted and not-admitted candidates are kept.  init_visited = 0: the visited set
 * of the previous call stays and the entry points are not re-marked (ResumeScanItems).  tuples
 * (nullable) counts visited elements as upstream's `tuples` does. */
static int search_layer_ex(const OrcIndex *ix, const float *q, const Cand *ep, int nep, int ef, int lc,
                           Cand *out, Scratch *s, OrcCounters *ctr, Disc *disc, int init_visited, int64_t *tuples)
{
    if (init_visited) scratch_begin(s, ix->n, ef > nep ? ef : nep);
    else {
        int need = (ef > nep ? ef : nep) + 2;
        if (s->capW < need) { s->capW = need; s->W = (Cand *) realloc(s->W, sizeof(Cand) * s->capW); }
        s->nC = s->nW = 0;
    }
    int wlen = 0;
    for (int i = 0; i < nep; i++) {
        if (init_visited) {
            s->stamp[ep[i].id] = s->epoch;
            if (tuples) (*tuples)++;
        }
        c_push(s, ep[i]);
        w_push(s, ep[i]);
        wlen++;
    }
    while (s->nC > 0) {
        Cand c = c_pop(s);
        Cand f = s->W[0];
        if (c.d > f.d) break;
        if (ctr) { if (lc == 0) ctr->n_hop0++; else ctr->n_hopu++; }
        uint8_t *cnt;
        const int32_t *nb = nbrs(ix, c.id, lc, NULL, &cnt);
        for (int i = 0; i < *cnt; i++) {
            int32_t e = nb[i];
            if (s->stamp[e] == s->epoch) continue;
            s->stamp[e] = s->epoch;
            if (tuples) (*tuples)++;
            int always = wlen < ef;
            f = s->W[0];
            float ed = dist_q_row(ix, q, row_of(ix, e));
            if (ctr) ctr->n_dist++;
            Cand ec = { ed, e };
            if (ed < f.d || always) {
                c_push(s, ec);
                w_push(s, ec);
                wlen++;
                if (wlen > ef) {                       /* upstream leaves wlen > ef; same effect */
                    Cand d = w_pop(s); wlen--;
                    if (disc) disc_push(disc, d);
                }
            } else if (disc) disc_push(disc, ec);
        }
    }
    int cnt = s->nW;
    for (int i = cnt - 1; i >= 0; i--) out[i] = w_pop(s);
    return cnt;
}

static int search_layer(const OrcIndex *ix, const float *q, const Cand *ep, int nep, int ef, int lc,
                        Cand *out, Scratch *s, OrcCounters *ctr)
{
    return search_layer_ex(ix, q, ep, nep, ef, lc, out, s, ctr, NULL, 1, NULL);
}

/* ------------------------------------------------------------------ SelectNeighbors */

static float dist_elems(const OrcIndex *ix, int64_t a, int64_t b, OrcCounters *ctr)
{
    float fa[ix->dim];
    row_as_float(ix, a, fa);
    if (ctr) ctr->n_pair++;
    return dist_q_row(ix, fa, row_of(ix, b));
}

/* c: candidates NEAREST first (key order).  r_out: selected, in upstream's list order.
 * *pruned (nullable) receives the candidate upstream reports as pruned.  Returns |r|. */
static int select_neighbors(const OrcIndex *ix, const Cand *c, int nc, int lm, Cand *r_out,
                            Cand *pruned, OrcCounters *ctr)
{
    if (nc <= lm) {
        /* `if (list_length(w) <= lm) return w;` -- w is furthest-first upstream */
        for (int i = 0; i < nc; i++) r_out[i] = c[nc - 1 - i];
        return nc;
    }
    Cand wd[nc];
    int nr = 0, nwd = 0, i = 0;
    while (i < nc && nr < lm) {
        Cand e = c[i++];
        int closer = 1;
        for (int j = 0; j < nr; j++) {
            float d = dist_elems(ix, e.id, r_out[j].id, ctr);
            if (d <= e.d) { closer = 0; break; }
        }
        if (closer) r_out[nr++] = e; else wd[nwd++] = e;
    }
    int wdoff = 0;
    while (wdoff < nwd && nr < lm) r_out[nr++] = wd[wdoff++];
    if (pruned) *pruned = wdoff < nwd ? wd[wdoff] : c[nc - 1];
    return nr;
}

/* ------------------------------------------------------------------ HnswFindElementNeighbors */

typedef struct { Cand *items; int *len; } NeighborPlan;   /* per layer, lm slots each */

static void find_element_neighbors(OrcIndex *ix, int64_t e, int level, const float *q, Cand **sel,
                                   int *nsel, Scratch *s, OrcCounters *ctr)
{
    int efc = ix->efc;
    int epcap = efc > 1 ? efc : 1;
    Cand *ep = (Cand *) malloc(sizeof(Cand) * (epcap + 1));
    Cand *w = (Cand *) malloc(sizeof(Cand) * (epcap + 1));
    int nep = 1;
    ep[0].id = ix->entry;
    ep[0].d = dist_q_row(ix, q, row_of(ix, ix->entry));
    if (ctr) ctr->n_dist++;
    int entry_level = ix->entry_level;
    for (int lc = entry_level; lc >= level + 1; lc--) {
        int nw = search_layer(ix, q, ep, nep, 1, lc, w, s, ctr);
        memcpy(ep, w, sizeof(Cand) * nw); nep = nw;
    }
    if (level > entry_level) level = entry_level;
    for (int lc = level; lc >= 0; lc--) {
        int lm = layer_m(ix, lc);
        int nw = search_layer(ix, q, ep, nep, efc, lc, w, s, ctr);
        nsel[lc] = select_neighbors(ix, w, nw, lm, sel[lc], NULL, ctr);
        memcpy(ep, w, sizeof(Cand) * nw); nep = nw;
    }
    (void) e;
    free(ep); free(w);
}

/* ------------------------------------------------------------------ HnswUpdateConnection */

static int cmp_cand(const void *a, const void *b)
{
    Cand x = *(const Cand *) a, y = *(const Cand *) b;
    return key_lt(x, y) ? -1 : (key_lt(y, x) ? 1 : 0);
}

/* add `e` (distance d) to the layer-lc list of element n, shrinking by the heuristic if full */
static void update_connection(OrcIndex *ix, int32_t e, float d, int32_t n, int lm, int lc,
                              OrcCounters *ctr)
{
    float *nd; uint8_t *cnt;
    int32_t *nb = nbrs(ix, n, lc, &nd, &cnt);
    if (*cnt < lm) {
        nb[*cnt] = e; nd[*cnt] = d; (*cnt)++;
        return;
    }
    Cand c[lm + 1], r[lm + 1], pruned;
    for (int i = 0; i < lm; i++) { c[i].id = nb[i]; c[i].d = nd[i]; }
    c[lm].id = e; c[lm].d = d;
    qsort(c, lm + 1, sizeof(Cand), cmp_cand);     /* sortCandidates = true: (distance, address) */
    select_neighbors(ix, c, lm + 1, lm, r, &pruned, ctr);
    for (int i = 0; i < lm; i++)
        if (nb[i] == pruned.id) { nb[i] = e; nd[i] = d; break; }
}

/* ------------------------------------------------------------------ create / grow */

OrcIndex *orc_create(int dim, int m, int efc, int metric, int dtype, int dist_mode, uint64_t seed)
{
    if (dim < 1 || m < 2 || m > 100 || efc < 4 || efc > 1000 || efc < 2 * m) return NULL;
    OrcIndex *ix = (OrcIndex *) calloc(1, sizeof *ix);
    ix->dim = dim; ix->m = m; ix->efc = efc; ix->metric = metric; ix->dtype = dtype;
    ix->dist_mode = dist_mode; ix->seed = seed; ix->esize = dtype == ORC_F32 ? 4 : 2;
    ix->entry = -1; ix->entry_level = -1;
    return ix;
}

void orc_set_dist_mode(OrcIndex *ix, int dist_mode) { ix->dist_mode = dist_mode; }

void orc_free(OrcIndex *ix)
{
    if (!ix) return;
    free(ix->vecs); free(ix->level); free(ix->nbr0); free(ix->nbr0d); free(ix->cnt0);
    free(ix->uoff); free(ix->nbru); free(ix->nbrud); free(ix->cntu); free(ix->ntids); free(ix->tids); free(ix->deleted);
    free(ix);
}

static void grow_elems(OrcIndex *ix, int64_t need)
{
    if (need <= ix->cap) return;
    int64_t cap = ix->cap ? ix->cap * 2 : 1024;
    while (cap < need) cap *= 2;
    int m2 = 2 * ix->m;
    ix->vecs = (char *) realloc(ix->vecs, (size_t) cap * ix->dim * ix->esize);
    ix->level = (uint8_t *) realloc(ix->level, cap);
    ix->nbr0 = (int32_t *) realloc(ix->nbr0, sizeof(int32_t) * cap * m2);
    ix->nbr0d = (float *) realloc(ix->nbr0d, sizeof(float) * cap * m2);
    ix->cnt0 = (uint8_t *) realloc(ix->cnt0, cap);
    ix->uoff = (int32_t *) realloc(ix->uoff, sizeof(int32_t) * cap);
    ix->ntids = (uint8_t *) realloc(ix->ntids, cap);
    ix->deleted = (uint8_t *) realloc(ix->deleted, cap);
    memset(ix->deleted + ix->cap, 0, (size_t) (cap - ix->cap));
    ix->tids = (int64_t *) realloc(ix->tids, sizeof(int64_t) * cap * ORC_HEAPTIDS);
    ix->cap = cap;
}

static void grow_upper(OrcIndex *ix, int64_t need)
{
    if (need <= ix->ucap) return;
    int64_t cap = ix->ucap ? ix->ucap * 2 : 256;
    while (cap < need) cap *= 2;
    ix->nbru = (int32_t *) realloc(ix->nbru, sizeof(int32_t) * cap * ix->m);
    ix->nbrud = (float *) realloc(ix->nbrud, sizeof(float) * cap * ix->m);
    ix->cntu = (uint8_t *) realloc(ix->cntu, cap);
    ix->ucap = cap;
}

/* ------------------------------------------------------------------ insert (in-memory build) */

/* an imported graph carries no owner->neighbour distances: compute them as the first insert needs them (the GPU
 * library does the same for a loaded graph) */
static void refresh_cached_distances(OrcIndex *ix)
{
    int m2 = 2 * ix->m, m = ix->m;
    for (int64_t e = 0; e < ix->n; e++) {
        for (int i = 0; i < ix->cnt0[e]; i++) ix->nbr0d[e * m2 + i] = dist_elems(ix, e, ix->nbr0[e * m2 + i], NULL);
        for (int l = 1; l <= ix->level[e]; l++) {
            int64_t r = (int64_t) ix->uoff[e] + l - 1;
            for (int i = 0; i < ix->cntu[r]; i++) ix->nbrud[r * m + i] = dist_elems(ix, e, ix->nbru[r * m + i], NULL);
        }
    }
    ix->stale_d = 0;
}

int64_t orc_insert(OrcIndex *ix, const void *vec, int64_t heap_tid)
{
    int dim = ix->dim;
    if (ix->stale_d) refresh_cached_distances(ix);
    size_t rowb = (size_t) dim * ix->esize;
    grow_elems(ix, ix->n + 1);
    int64_t e = ix->n;
    char *row = ix->vecs + (size_t) e * rowb;
    if (ix->metric == ORC_COSINE) {
        /* HnswCheckNorm + HnswNormValue */
        if (!orc_normalize(ix->dtype, ix->dist_mode, dim, vec, row)) return -1;
    } else {
        memcpy(row, vec, rowb);
    }
    int level = orc_level_for(ix->seed, ix->seq++, ix->m);
    ix->level[e] = (uint8_t) level;
    ix->cnt0[e] = 0;
    for (int i = 0; i < 2 * ix->m; i++) ix->nbr0[e * 2 * ix->m + i] = -1;
    ix->ntids[e] = 1;
    ix->tids[e * ORC_HEAPTIDS] = heap_tid;
    ix->uoff[e] = -1;

    if (ix->entry < 0) {
        if (level > 0) {
            grow_upper(ix, ix->urows + level);
            ix->uoff[e] = (int32_t) ix->urows;
            for (int r = 0; r < level; r++) {
                ix->cntu[ix->urows + r] = 0;
                for (int i = 0; i < ix->m; i++) ix->nbru[(ix->urows + r) * ix->m + i] = -1;
            }
            ix->urows += level;
        }
        ix->n++;
        ix->entry = (int32_t) e; ix->entry_level = level;
        return e;
    }

    float q[dim];
    row_as_float(ix, e, q);
    int nl = level + 1;
    Cand *sel[nl]; int nsel[nl];
    for (int lc = 0; lc < nl; lc++) { sel[lc] = (Cand *) malloc(sizeof(Cand) * (2 * ix->m + 1)); nsel[lc] = 0; }
    Scratch s; scratch_init(&s);
    find_element_neighbors(ix, e, level, q, sel, nsel, &s, &ix->ctr);
    scratch_free(&s);

    /* FindDuplicateInMemory: walk layer-0 neighbours in stored order, stop at the first that is
     * not byte-identical; attach the heap TID to the first identical one with room */
    int64_t dup = -1;
    for (int i = 0; i < nsel[0]; i++) {
        int32_t nbr = sel[0][i].id;
        if (memcmp(row_of(ix, nbr), row, rowb) != 0) break;
        if (ix->ntids[nbr] < ORC_HEAPTIDS) { dup = nbr; break; }
    }
    if (dup >= 0) {
        ix->tids[dup * ORC_HEAPTIDS + ix->ntids[dup]++] = heap_tid;
        for (int lc = 0; lc < nl; lc++) free(sel[lc]);
        return dup;
    }

    /* AddElementInMemory + AddConnections */
    if (level > 0) {
        grow_upper(ix, ix->urows + level);
        ix->uoff[e] = (int32_t) ix->urows;
        for (int r = 0; r < level; r++) {
            ix->cntu[ix->urows + r] = 0;
            for (int i = 0; i < ix->m; i++) ix->nbru[(ix->urows + r) * ix->m + i] = -1;
        }
        ix->urows += level;
    }
    ix->n++;
    for (int lc = 0; lc < nl; lc++) {
        float *nd; uint8_t *cnt;
        int32_t *nb = nbrs(ix, e, lc, &nd, &cnt);
        for (int i = 0; i < nsel[lc]; i++) { nb[i] = sel[lc][i].id; nd[i] = sel[lc][i].d; }
        *cnt = (uint8_t) nsel[lc];
    }
    /* UpdateNeighborsInMemory */
    for (int lc = level; lc >= 0; lc--) {
        int lm = layer_m(ix, lc);
        for (int i = 0; i < nsel[lc]; i++)
            update_connection(ix, (int32_t) e, sel[lc][i].d, sel[lc][i].id, lm, lc, &ix->ctr);
    }
    if (level > ix->entry_level) { ix->entry = (int32_t) e; ix->entry_level = level; }
    for (int lc = 0; lc < nl; lc++) free(sel[lc]);
    return e;
}

int64_t orc_build(OrcIndex *ix, const void *vecs, int64_t n, const int64_t *heap_tids)
{
    size_t rowb = (size_t) ix->dim * ix->esize;
    for (int64_t i = 0; i < n; i++) {
        int64_t r = orc_insert(ix, (const char *) vecs + (size_t) i * rowb, heap_tids ? heap_tids[i] : i);
        if (r == -2) return -2;
    }
    return ix->n;
}


/* ------------------------------------------------------------------ vacuum (hnswvacuum.c) */
/* ambulkdelete upstream = RemoveHeapTids, RepairGraph, MarkDeleted [RECALL].  orc_bulk_delete is the first pass,
 * orc_vacuum_repair the second and third. */

static int cmp_i64(const void *a, const void *b)
{
    int64_t x = *(const int64_t *) a, y = *(const int64_t *) b;
    return x < y ? -1 : (x > y ? 1 : 0);
}

/* RemoveHeapTids: dead heap TIDs leave their elements (the remaining TIDs keep their order); returns how many left */
int64_t orc_bulk_delete(OrcIndex *ix, const int64_t *dead_tids, int64_t n_dead)
{
    if (n_dead <= 0) return 0;
    int64_t *dead = (int64_t *) malloc(sizeof(int64_t) * n_dead);
    memcpy(dead, dead_tids, sizeof(int64_t) * n_dead);
    qsort(dead, n_dead, sizeof(int64_t), cmp_i64);
    int64_t removed = 0;
    for (int64_t e = 0; e < ix->n; e++) {
        int64_t *t = ix->tids + e * ORC_HEAPTIDS;
        int nt = ix->ntids[e], w = 0;
        for (int k = 0; k < nt; k++)
            if (!bsearch(&t[k], dead, n_dead, sizeof(int64_t), cmp_i64)) t[w++] = t[k];
        for (int k = w; k < nt; k++) t[k] = 0;
        removed += nt - w;
        ix->ntids[e] = (uint8_t) w;
    }
    free(dead);
    return removed;
}

/* HnswSearchLayer as vacuum calls it (skipElement != NULL): elements left without heap TIDs are traversed and
 * kept in W but do not count towards ef (CountElement); wlen is never decremented ("No need to decrement wlen"),
 * so from the first overflow on every counted admission evicts the furthest entry, whatever it is. */
static int search_layer_vacuum(const OrcIndex *ix, const float *q, const Cand *ep, int nep, int ef, int lc, Cand **out,
                               int *out_cap, Scratch *s, OrcCounters *ctr)
{
    scratch_begin(s, ix->n, ef > nep ? ef : nep);
    int wlen = 0;
    for (int i = 0; i < nep; i++) {
        s->stamp[ep[i].id] = s->epoch;
        c_push(s, ep[i]);
        if (s->nW + 2 > s->capW) { s->capW = 2 * s->capW + 2; s->W = (Cand *) realloc(s->W, sizeof(Cand) * s->capW); }
        w_push(s, ep[i]);
        if (ix->ntids[ep[i].id] != 0) wlen++;
    }
    while (s->nC > 0) {
        Cand c = c_pop(s);
        Cand f = s->W[0];
        if (c.d > f.d) break;
        if (ctr) { if (lc == 0) ctr->n_hop0++; else ctr->n_hopu++; }
        uint8_t *cnt;
        const int32_t *nb = nbrs(ix, c.id, lc, NULL, &cnt);
        for (int i = 0; i < *cnt; i++) {
            int32_t e = nb[i];
            if (s->stamp[e] == s->epoch) continue;
            s->stamp[e] = s->epoch;
            int always = wlen < ef;
            f = s->W[0];
            float ed = dist_q_row(ix, q, row_of(ix, e));
            if (ctr) ctr->n_dist++;
            Cand ec = { ed, e };
            if (ed < f.d || always) {
                c_push(s, ec);
                if (s->nW + 2 > s->capW) { s->capW = 2 * s->capW + 2; s->W = (Cand *) realloc(s->W, sizeof(Cand) * s->capW); }
                w_push(s, ec);
                if (ix->ntids[e] != 0) {
                    wlen++;
                    if (wlen > ef) (void) w_pop(s);
                }
            }
        }
    }
    int cnt = s->nW;
    if (*out_cap < cnt + 1) { *out_cap = cnt + 64; *out = (Cand *) realloc(*out, sizeof(Cand) * *out_cap); }
    for (int i = cnt - 1; i >= 0; i--) (*out)[i] = w_pop(s);
    return cnt;
}

/* NeedsUpdated: a neighbour is being deleted, or layer 0 is not full */
static int needs_updated(const OrcIndex *ix, int64_t e)
{
    for (int lc = ix->level[e]; lc >= 0; lc--) {
        uint8_t *cnt;
        const int32_t *nb = nbrs(ix, e, lc, NULL, &cnt);
        for (int i = 0; i < *cnt; i++)
            if (ix->ntids[nb[i]] == 0) return 1;
    }
    return ix->cnt0[e] < 2 * ix->m;
}

/* HnswUpdateNeighborsOnDisk (checkExisting = true) for one neighbour: HnswUpdateConnection on the list as stored,
 * distances recomputed, a neighbour that is being deleted is replaced before any heuristic selection */
static void update_connection_vacuum(OrcIndex *ix, int32_t e, float d, int32_t n, int lm, int lc, OrcCounters *ctr)
{
    float *nd; uint8_t *cnt;
    int32_t *nb = nbrs(ix, n, lc, &nd, &cnt);
    for (int i = 0; i < *cnt; i++) if (nb[i] == e) return;           /* existing connection */
    if (*cnt < lm) { nb[*cnt] = e; nd[*cnt] = d; (*cnt)++; return; }
    Cand c[lm + 1], r[lm + 1], pruned;
    int have = 0;
    for (int i = 0; i < lm; i++) {
        c[i].id = nb[i];
        c[i].d = dist_elems(ix, n, nb[i], ctr);
        nd[i] = c[i].d;
        if (ix->ntids[nb[i]] == 0) { pruned = c[i]; have = 1; break; }      /* prune element if being deleted */
    }
    if (!have) {
        c[lm].id = e; c[lm].d = d;
        qsort(c, lm + 1, sizeof(Cand), cmp_cand);
        select_neighbors(ix, c, lm + 1, lm, r, &pruned, ctr);
    }
    for (int i = 0; i < lm; i++)
        if (nb[i] == pruned.id) { nb[i] = e; nd[i] = d; break; }
}

/* RepairGraphElement */
static void repair_element(OrcIndex *ix, int64_t e, int32_t entry, Scratch *s, OrcCounters *ctr)
{
    if (entry >= 0 && e == entry) return;
    int m = ix->m, level = ix->level[e];
    int nl = level + 1;
    Cand *sel[nl]; int nsel[nl];
    for (int lc = 0; lc < nl; lc++) { sel[lc] = (Cand *) malloc(sizeof(Cand) * (2 * m + 1)); nsel[lc] = 0; }
    if (entry >= 0) {
        /* HnswFindElementNeighbors(existing = true): the element's stored lists are still in the graph while it searches */
        float q[ix->dim];
        row_as_float(ix, e, q);
        int cap_ep = 64, cap_w = 64, nep = 1;
        Cand *ep = (Cand *) malloc(sizeof(Cand) * cap_ep), *w = (Cand *) malloc(sizeof(Cand) * cap_w);
        ep[0].id = entry;
        ep[0].d = dist_q_row(ix, q, row_of(ix, entry));
        if (ctr) ctr->n_dist++;
        int entry_level = ix->level[entry];
        for (int lc = entry_level; lc >= level + 1; lc--) {
            int nw = search_layer_vacuum(ix, q, ep, nep, 1, lc, &w, &cap_w, s, ctr);
            if (cap_ep < nw + 1) { cap_ep = nw + 64; ep = (Cand *) realloc(ep, sizeof(Cand) * cap_ep); }
            memcpy(ep, w, sizeof(Cand) * nw); nep = nw;
        }
        int top = level > entry_level ? entry_level : level;
        for (int lc = top; lc >= 0; lc--) {
            int lm = layer_m(ix, lc);
            int nw = search_layer_vacuum(ix, q, ep, nep, ix->efc + 1, lc, &w, &cap_w, s, ctr);   /* "Add one for existing element" */
            /* RemoveElements: the element itself and elements being deleted help the search but are not candidates */
            Cand lw[nw + 1];
            int nlw = 0;
            for (int i = 0; i < nw; i++)
                if (w[i].id != e && ix->ntids[w[i].id] != 0) lw[nlw++] = w[i];
            nsel[lc] = select_neighbors(ix, lw, nlw, lm, sel[lc], NULL, ctr);
            if (cap_ep < nw + 1) { cap_ep = nw + 64; ep = (Cand *) realloc(ep, sizeof(Cand) * cap_ep); }
            memcpy(ep, w, sizeof(Cand) * nw); nep = nw;
        }
        free(ep); free(w);
    }
    /* overwrite the neighbour tuple (HnswInitNeighbors emptied every layer first) */
    for (int lc = 0; lc < nl; lc++) {
        float *nd; uint8_t *cnt;
        int32_t *nb = nbrs(ix, e, lc, &nd, &cnt);
        int lm = layer_m(ix, lc);
        for (int i = 0; i < lm; i++) { nb[i] = i < nsel[lc] ? sel[lc][i].id : -1; nd[i] = i < nsel[lc] ? sel[lc][i].d : 0.0f; }
        *cnt = (uint8_t) nsel[lc];
    }
    for (int lc = level; lc >= 0; lc--) {
        int lm = layer_m(ix, lc);
        for (int i = 0; i < nsel[lc]; i++)
            update_connection_vacuum(ix, (int32_t) e, sel[lc][i].d, sel[lc][i].id, lm, lc, ctr);
    }
    for (int lc = 0; lc < nl; lc++) free(sel[lc]);
}

/* RepairGraph (entry point first, then every element in page order) + MarkDeleted.  Returns the number of
 * elements marked deleted by this call; *repaired (nullable) = elements whose neighbours were recomputed. */
int64_t orc_vacuum_repair(OrcIndex *ix, int64_t *repaired)
{
    Scratch s; scratch_init(&s);
    OrcCounters *ctr = &ix->ctr;
    int64_t nrep = 0;
    /* the highest live element that is not the entry point (RemoveHeapTids remembers it; first one in page order) */
    int32_t highest = -1; int hl = -1;
    for (int64_t e = 0; e < ix->n; e++)
        if (ix->ntids[e] != 0 && e != ix->entry && ix->level[e] > hl) { highest = (int32_t) e; hl = ix->level[e]; }
    /* RepairGraphEntryPoint */
    if (highest >= 0 && needs_updated(ix, highest)) { repair_element(ix, highest, ix->entry, &s, ctr); nrep++; }
    if (ix->entry >= 0) {
        if (ix->ntids[ix->entry] == 0) {
            ix->entry = highest;
            ix->entry_level = highest >= 0 ? ix->level[highest] : -1;
        } else if (needs_updated(ix, ix->entry)) { repair_element(ix, ix->entry, highest, &s, ctr); nrep++; }
    }
    for (int64_t e = 0; e < ix->n; e++) {
        if (ix->ntids[e] == 0) continue;
        if (!needs_updated(ix, e)) continue;
        if (e == ix->entry) continue;
        repair_element(ix, e, ix->entry, &s, ctr);
        nrep++;
    }
    /* MarkDeleted: the emptied elements leave the graph for good */
    int64_t marked = 0;
    size_t rowb = (size_t) ix->dim * ix->esize;
    for (int64_t e = 0; e < ix->n; e++) {
        if (ix->ntids[e] != 0 || ix->deleted[e]) continue;
        ix->deleted[e] = 1;
        marked++;
        memset(ix->vecs + (size_t) e * rowb, 0, rowb);
        for (int lc = ix->level[e]; lc >= 0; lc--) {
            float *nd; uint8_t *cnt;
            int32_t *nb = nbrs(ix, e, lc, &nd, &cnt);
            int lm = layer_m(ix, lc);
            for (int i = 0; i < lm; i++) { nb[i] = -1; nd[i] = 0.0f; }
            *cnt = 0;
        }
    }
    scratch_free(&s);
    if (repaired) *repaired = nrep;
    return marked;
}

/* ------------------------------------------------------------------ scan */

static void query_as_float(const OrcIndex *ix, const void *query, float *q)
{
    int dim = ix->dim;
    if (ix->metric == ORC_COSINE) {
        char tmp[(size_t) dim * ix->esize];
        orc_normalize(ix->dtype, ix->dist_mode, dim, query, tmp);
        if (ix->dtype == ORC_F32) memcpy(q, tmp, sizeof(float) * dim);
        else half_to_float(dim, (const uint16_t *) tmp, q);
    } else if (ix->dtype == ORC_F32) {
        memcpy(q, query, sizeof(float) * dim);
    } else {
        half_to_float(dim, (const uint16_t *) query, q);
    }
}

static int scan_items(const OrcIndex *ix, const void *query, int ef, Cand *out, Scratch *s,
                      OrcCounters *ctr)
{
    if (ix->entry < 0) return 0;
    float q[ix->dim];
    query_as_float(ix, query, q);
    Cand ep[1], w[2];
    ep[0].id = ix->entry;
    ep[0].d = dist_q_row(ix, q, row_of(ix, ix->entry));
    if (ctr) ctr->n_dist++;
    for (int lc = ix->entry_level; lc >= 1; lc--) {
        search_layer(ix, q, ep, 1, 1, lc, w, s, ctr);
        ep[0] = w[0];
    }
    return search_layer(ix, q, ep, 1, ef, 0, out, s, ctr);
}

int orc_search_elements(const OrcIndex *ix, const void *query, int ef, int32_t *out_elem,
                        float *out_dist, OrcCounters *ctr)
{
    Scratch s; scratch_init(&s);
    Cand *w = (Cand *) malloc(sizeof(Cand) * (ef + 2));
    int n = scan_items(ix, query, ef, w, &s, ctr);
    for (int i = 0; i < n; i++) { out_elem[i] = w[i].id; out_dist[i] = w[i].d; }
    free(w); scratch_free(&s);
    return n;
}

int orc_search_tids(const OrcIndex *ix, const void *query, int ef, int k, int64_t *out_tids,
                    float *out_dist, OrcCounters *ctr)
{
    Scratch s; scratch_init(&s);
    Cand *w = (Cand *) malloc(sizeof(Cand) * (ef + 2));
    int n = scan_items(ix, query, ef, w, &s, ctr);
    int o = 0;
    for (int i = 0; i < n && o < k; i++)
        for (int t = ix->ntids[w[i].id] - 1; t >= 0 && o < k; t--) {   /* heaptids[--heaptidsLength] */
            out_tids[o] = ix->tids[(int64_t) w[i].id * ORC_HEAPTIDS + t];
            out_dist[o] = w[i].d;
            o++;
        }
    free(w); scratch_free(&s);
    return o;
}

void orc_search_batch(const OrcIndex *ix, const void *queries, int64_t nq, int ef, int32_t *out_elem,
                      float *out_dist, int32_t *out_cnt, OrcCounters *ctr, int threads)
{
    size_t rowb = (size_t) ix->dim * ix->esize;
    int64_t nd = 0, h0 = 0, hu = 0;
    if (threads < 1) threads = 1;
#pragma omp parallel num_threads(threads) reduction(+ : nd, h0, hu)
    {
        Scratch s; scratch_init(&s);
        Cand *w = (Cand *) malloc(sizeof(Cand) * (ef + 2));
        OrcCounters c;
#pragma omp for schedule(dynamic, 16)
        for (int64_t i = 0; i < nq; i++) {
            memset(&c, 0, sizeof c);
            int n = scan_items(ix, (const char *) queries + (size_t) i * rowb, ef, w, &s, &c);
            for (int j = 0; j < ef; j++) {
                out_elem[i * ef + j] = j < n ? w[j].id : -1;
                out_dist[i * ef + j] = j < n ? w[j].d : INFINITY;
            }
            if (out_cnt) out_cnt[i] = n;
            nd += c.n_dist; h0 += c.n_hop0; hu += c.n_hopu;
        }
        free(w); scratch_free(&s);
    }
    if (ctr) { ctr->n_dist += nd; ctr->n_hop0 += h0; ctr->n_hopu += hu; }
}

/* ------------------------------------------------------------------ iterative scan (pgvector 0.8) */
/* hnswscan.c with hnsw.iterative_scan on: GetScanItems keeps the discarded candidates and the
 * visited set; when the ef_search results are consumed, ResumeScanItems seeds another layer-0
 * search with the ef_search nearest discarded candidates.  Once `tuples` reaches
 * hnsw.max_scan_tuples the remaining discarded candidates are handed out one per call. */
struct OrcIter {
    const OrcIndex *ix;
    float *q;
    int ef;
    int64_t max_tuples, tuples;
    Scratch s;
    Disc disc;
    int started;
    OrcCounters ctr;
};

OrcIter *orc_iter_begin(const OrcIndex *ix, const void *query, int ef, int64_t max_scan_tuples)
{
    OrcIter *it = (OrcIter *) calloc(1, sizeof *it);
    it->ix = ix; it->ef = ef; it->max_tuples = max_scan_tuples;
    it->q = (float *) malloc(sizeof(float) * ix->dim);
    query_as_float(ix, query, it->q);
    scratch_init(&it->s);
    return it;
}

int orc_iter_next(OrcIter *it, int32_t *out_elem, float *out_dist)
{
    const OrcIndex *ix = it->ix;
    int ef = it->ef, n = 0;
    Cand *w = (Cand *) malloc(sizeof(Cand) * (ef + 2));
    if (!it->started) {
        it->started = 1;
        if (ix->entry >= 0) {
            Cand ep[1], u[2];
            ep[0].id = ix->entry;
            ep[0].d = dist_q_row(ix, it->q, row_of(ix, ix->entry));
            it->ctr.n_dist++;
            for (int lc = ix->entry_level; lc >= 1; lc--) {
                search_layer(ix, it->q, ep, 1, 1, lc, u, &it->s, &it->ctr);
                ep[0] = u[0];
            }
            n = search_layer_ex(ix, it->q, ep, 1, ef, 0, w, &it->s, &it->ctr, &it->disc, 1, &it->tuples);
        }
    } else if (it->disc.n > 0) {
        if (it->tuples >= it->max_tuples) {
            w[0] = disc_pop(&it->disc);          /* return remaining tuples */
            n = 1;
        } else {
            Cand *ep = (Cand *) malloc(sizeof(Cand) * ef);
            int nep = 0;
            while (nep < ef && it->disc.n > 0) ep[nep++] = disc_pop(&it->disc);
            n = search_layer_ex(ix, it->q, ep, nep, ef, 0, w, &it->s, &it->ctr, &it->disc, 0, &it->tuples);
            free(ep);
        }
    }
    for (int i = 0; i < n; i++) { out_elem[i] = w[i].id; out_dist[i] = w[i].d; }
    free(w);
    return n;
}

int64_t orc_iter_tuples(const OrcIter *it) { return it->tuples; }
int64_t orc_iter_discarded(const OrcIter *it) { return it->disc.n; }
void orc_iter_counters(const OrcIter *it, OrcCounters *out) { *out = it->ctr; }

void orc_iter_end(OrcIter *it)
{
    if (!it) return;
    scratch_free(&it->s); free(it->disc.a); free(it->q); free(it);
}

int orc_search_layer(const OrcIndex *ix, const void *query, const int32_t *ep, int nep, int ef,
                     int lc, int32_t *out_elem, float *out_dist, OrcCounters *ctr)
{
    float q[ix->dim];
    query_as_float(ix, query, q);
    Cand epc[nep];
    for (int i = 0; i < nep; i++) {
        epc[i].id = ep[i];
        epc[i].d = dist_q_row(ix, q, row_of(ix, ep[i]));
        if (ctr) ctr->n_dist++;
    }
    Scratch s; scratch_init(&s);
    int cap = (ef > nep ? ef : nep) + 2;
    Cand *w = (Cand *) malloc(sizeof(Cand) * cap);
    int n = search_layer(ix, q, epc, nep, ef, lc, w, &s, ctr);
    for (int i = 0; i < n; i++) { out_elem[i] = w[i].id; out_dist[i] = w[i].d; }
    free(w); scratch_free(&s);
    return n;
}

/* ------------------------------------------------------------------ brute force (ground truth) */

typedef struct { double d; int32_t id; } DCand;
static inline int dkey_lt(DCand a, DCand b) { return a.d < b.d || (a.d == b.d && a.id < b.id); }

void orc_bruteforce(const OrcIndex *ix, const void *queries, int64_t nq, int k, int32_t *out_elem,
                    double *out_dist, int threads)
{
    int dim = ix->dim;
    size_t rowb = (size_t) dim * ix->esize;
    if (threads < 1) threads = 1;
#pragma omp parallel for num_threads(threads) schedule(dynamic, 4)
    for (int64_t qi = 0; qi < nq; qi++) {
        float q[dim], r[dim];
        query_as_float(ix, (const char *) queries + (size_t) qi * rowb, q);
        DCand top[k + 1];
        int nt = 0;
        for (int64_t e = 0; e < ix->n; e++) {
            row_as_float(ix, e, r);
            double acc = 0.0;
            if (ix->metric == ORC_L2)
                for (int i = 0; i < dim; i++) { double t = (double) q[i] - (double) r[i]; acc += t * t; }
            else if (ix->metric == ORC_L1)
                for (int i = 0; i < dim; i++) acc += fabs((double) q[i] - (double) r[i]);
            else {
                for (int i = 0; i < dim; i++) acc += (double) q[i] * (double) r[i];
                acc = -acc;
            }
            DCand c = { acc, (int32_t) e };
            if (nt == k && !dkey_lt(c, top[k - 1])) continue;
            int p = nt < k ? nt++ : k - 1;
            while (p > 0 && dkey_lt(c, top[p - 1])) { top[p] = top[p - 1]; p--; }
            top[p] = c;
        }
        for (int j = 0; j < k; j++) {
            out_elem[qi * k + j] = j < nt ? top[j].id : -1;
            out_dist[qi * k + j] = j < nt ? top[j].d : INFINITY;
        }
    }
}

void orc_exact_topk(const OrcIndex *ix, const void *queries, int64_t nq, int k, int32_t *out_elem,
                    float *out_dist, int threads)
{
    int dim = ix->dim;
    size_t rowb = (size_t) dim * ix->esize;
    if (threads < 1) threads = 1;
#pragma omp parallel for num_threads(threads) schedule(dynamic, 4)
    for (int64_t qi = 0; qi < nq; qi++) {
        float q[dim];
        query_as_float(ix, (const char *) queries + (size_t) qi * rowb, q);
        Cand *top = malloc(sizeof(Cand) * (size_t) k);
        int nt = 0;
        for (int64_t e = 0; e < ix->n; e++) {
            Cand c = { dist_q_row(ix, q, row_of(ix, e)), (int32_t) e };
            if (nt == k && !key_lt(c, top[k - 1])) continue;
            int p = nt < k ? nt++ : k - 1;
            while (p > 0 && key_lt(c, top[p - 1])) { top[p] = top[p - 1]; p--; }
            top[p] = c;
        }
        for (int j = 0; j < k; j++) {
            out_elem[qi * k + j] = j < nt ? top[j].id : -1;
            out_dist[qi * k + j] = j < nt ? top[j].d : INFINITY;
        }
        free(top);
    }
}

/* ------------------------------------------------------------------ flat image */

int64_t orc_n(const OrcIndex *ix) { return ix->n; }
int64_t orc_upper_rows(const OrcIndex *ix) { return ix->urows; }
int32_t orc_entry(const OrcIndex *ix) { return ix->entry; }
int orc_entry_level(const OrcIndex *ix) { return ix->entry_level; }
void orc_counters(const OrcIndex *ix, OrcCounters *out) { *out = ix->ctr; }

void orc_export(const OrcIndex *ix, void *vecs, uint8_t *level, int32_t *nbr0, int32_t *uoff,
                int32_t *nbru, uint8_t *ntids, int64_t *tids)
{
    int64_t n = ix->n;
    int m2 = 2 * ix->m, m = ix->m;
    if (vecs) memcpy(vecs, ix->vecs, (size_t) n * ix->dim * ix->esize);
    if (level) memcpy(level, ix->level, n);
    if (nbr0)
        for (int64_t e = 0; e < n; e++)
            for (int i = 0; i < m2; i++)
                nbr0[e * m2 + i] = i < ix->cnt0[e] ? ix->nbr0[e * m2 + i] : -1;
    if (uoff) memcpy(uoff, ix->uoff, sizeof(int32_t) * n);
    if (nbru)
        for (int64_t r = 0; r < ix->urows; r++)
            for (int i = 0; i < m; i++)
                nbru[r * m + i] = i < ix->cntu[r] ? ix->nbru[r * m + i] : -1;
    if (ntids) memcpy(ntids, ix->ntids, n);
    if (tids) memcpy(tids, ix->tids, sizeof(int64_t) * n * ORC_HEAPTIDS);
}

OrcIndex *orc_import(int dim, int m, int efc, int metric, int dtype, int dist_mode, int64_t n,
                     int64_t upper_rows, int32_t entry, const void *vecs, const uint8_t *level,
                     const int32_t *nbr0, const int32_t *uoff, const int32_t *nbru,
                     const uint8_t *ntids, const int64_t *tids)
{
    OrcIndex *ix = orc_create(dim, m, efc, metric, dtype, dist_mode, 0);
    if (!ix) return NULL;
    grow_elems(ix, n > 0 ? n : 1);
    grow_upper(ix, upper_rows > 0 ? upper_rows : 1);
    int m2 = 2 * m;
    memcpy(ix->vecs, vecs, (size_t) n * dim * ix->esize);
    memcpy(ix->level, level, n);
    memcpy(ix->uoff, uoff, sizeof(int32_t) * n);
    for (int64_t e = 0; e < n; e++) {
        int c = 0;
        for (int i = 0; i < m2; i++) {
            ix->nbr0[e * m2 + i] = nbr0[e * m2 + i];
            ix->nbr0d[e * m2 + i] = 0.0f;
            if (nbr0[e * m2 + i] >= 0) c = i + 1;
        }
        ix->cnt0[e] = (uint8_t) c;
        ix->ntids[e] = ntids ? ntids[e] : 1;
        if (tids) memcpy(ix->tids + e * ORC_HEAPTIDS, tids + e * ORC_HEAPTIDS, sizeof(int64_t) * ORC_HEAPTIDS);
        else ix->tids[e * ORC_HEAPTIDS] = e;
    }
    for (int64_t r = 0; r < upper_rows; r++) {
        int c = 0;
        for (int i = 0; i < m; i++) {
            ix->nbru[r * m + i] = nbru[r * m + i];
            ix->nbrud[r * m + i] = 0.0f;
            if (nbru[r * m + i] >= 0) c = i + 1;
        }
        ix->cntu[r] = (uint8_t) c;
    }
    ix->n = n; ix->urows = upper_rows; ix->seq = n;
    ix->entry = entry; ix->entry_level = entry >= 0 ? level[entry] : -1;
    ix->stale_d = 1;
    return ix;
}
