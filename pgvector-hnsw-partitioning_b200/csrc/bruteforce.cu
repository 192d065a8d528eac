// bruteforce.cu -- exact scan of one partition (config 5): recall ground truth and the tensor-pipe
// roofline check.  Upstream's own recall tests compare the index scan with a sequential scan
// (`SET enable_indexscan = off`) [RECALL; reference mount empty, /root/reference/README.md:1]; this
// is that sequential scan for a batch of queries.
//
//   1. candidate generation: S = Q * X^T on the 5th-gen tensor cores -- bf16 operands (TMA, 128-byte
//      swizzle, 4-stage mbarrier ring) -> tcgen05.mma, fp32 accumulators in TMEM (two 128x256 buffers)
//      -> eight epilogue warps read TMEM with tcgen05.ld and keep, per query row and column half, the
//      K1 best columns of the slice of X this CTA streams.  The selection is arranged so that it hides
//      under the MMAs: one max + one branch per 32 columns; a hit computes its rank with independent
//      compares and shifts a register-resident sorted list with selects; thresholds are seeded from
//      slices of the same query that already finished (global per-query K1-th score), which cuts the
//      insertions ~4x.
//   2. fp32 re-rank: the exact canonical-order distance (distance.cuh) of every candidate.
//   3. certification: bf16 rounding perturbs a dot product by at most (2^-8 + 2^-11)*|q|*|x|, so any
//      row that was NOT kept has a true distance above a bound computed from the slice threshold; if
//      that bound exceeds the k-th exact distance the result is provably the exact top-k.  Queries
//      that cannot be certified are re-scanned exhaustively in fp32.
//
// Warp roles (320 threads, one CTA per SM, persistent over (query tile, X slice) work items ordered
// slice-major so the CTAs of a wave stream the same rows of X through L2 together):
//   warp 0 lane 0: TMA producer;  warp 1 lane 0: MMA issuer (warp 1 owns the TMEM allocation);
//   warps 2-9: epilogue, two per TMEM lane quarter.
// cta_group::1, M=128 N=256 K=16 per instruction.  Measured on B200 at 10k x 1M x 768: the MMA/TMA
// pipeline alone runs at 1.59 PFLOP/s; with the TMEM reads of the epilogue 1.13 PFLOP/s (0.80 of the
// measured sustained cuBLAS peak), the selection itself no longer shows.
#include "index.h"
#include "scan_kernel.cuh"

#include <cuda.h>
#include <cuda_bf16.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

namespace hb {

constexpr int BF_BM = 128, BF_BN = 256, BF_BK = 64, BF_STAGES = 4, BF_K1 = 16;
constexpr int BF_EPI_WARPS = 8;                 // two per TMEM lane quarter, each takes half of the columns
constexpr int BF_THREADS = 64 + 32 * BF_EPI_WARPS;
constexpr uint32_t BF_A_BYTES = BF_BM * BF_BK * 2, BF_B_BYTES = BF_BN * BF_BK * 2;
constexpr uint32_t BF_STAGE_BYTES = BF_A_BYTES + BF_B_BYTES;
constexpr size_t BF_SMEM = (size_t) BF_STAGES * BF_STAGE_BYTES + 2 * BF_BN * 4 + 256;

struct BfParams {
    int nq, N, kchunks, n_mtiles, S, ntiles, tiles_per_split;   // candidate lists: nq x (2*S) x K1 (two column halves per slice)
    const float *xnh;        // 0.5 * |x|^2 per row for L2, nullptr for inner product / cosine
    float *cand_score;       // nq x S x K1 (bf16-GEMM scores, best first)
    int32_t *cand_id;        // nq x S x K1 (-1 padded)
    float *cand_thr;         // nq x S: score of the K1-th kept row, -inf when the slice kept everything
    float *dbg;              // optional nq x N raw scores (tests)
    float *gthr;             // nq_pad: best K1-th score any finished slice reported for the query (threshold seed)
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t) __cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *b, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *b, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *b)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *b, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "LAB_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra LAB_WAIT;\n\t"
        "DONE:\n\t"
        "}" ::"r"(smem_u32(b)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
// K-major, 128-byte swizzle: rows at 128-byte pitch, 8-row groups 1024 bytes apart
__device__ __forceinline__ uint64_t umma_desc(const void *smem_tile)
{
    uint64_t d = 0;
    d |= (uint64_t) ((smem_u32(smem_tile) & 0x3FFFF) >> 4);   // start address
    d |= (uint64_t) 1 << 16;                                  // leading byte offset (unused with swizzle)
    d |= (uint64_t) (1024 >> 4) << 32;                        // stride byte offset
    d |= (uint64_t) 1 << 46;                                  // descriptor version (Blackwell)
    d |= (uint64_t) 2 << 61;                                  // SWIZZLE_128B
    return d;
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void atomic_max_float(float *addr, float v)
{
    int old = __float_as_int(*addr);
    while (__int_as_float(old) < v) {
        const int assumed = old;
        old = atomicCAS(reinterpret_cast<int *>(addr), assumed, __float_as_int(v));
        if (old == assumed) break;
    }
}

template <bool DBG, bool L2>
__global__ void __launch_bounds__(BF_THREADS, 1)
bf_gemm_topk_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const BfParams p)
{
    extern __shared__ __align__(1024) uint8_t bf_smem[];
    uint8_t *smem = bf_smem;
    float *xnh = reinterpret_cast<float *>(smem + (size_t) BF_STAGES * BF_STAGE_BYTES);   // [2][BF_BN]
    uint64_t *full = reinterpret_cast<uint64_t *>(xnh + 2 * BF_BN);
    uint64_t *empty = full + BF_STAGES;
    uint64_t *tfull = empty + BF_STAGES;
    uint64_t *tempty = tfull + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < BF_STAGES; s++) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
        for (int a = 0; a < 2; a++) { mbar_init(tfull + a, 1); mbar_init(tempty + a, BF_EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    const int items = p.n_mtiles * p.S;
    // instruction descriptor: D=f32, A=B=bf16, both K-major, N=256, M=128
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t) (BF_BN >> 3) << 17) | ((uint32_t) (BF_BM >> 4) << 24);

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int item = blockIdx.x; item < items; item += gridDim.x) {
                const int split = item / p.n_mtiles, m = item % p.n_mtiles;
                const int nt0 = split * p.tiles_per_split, nt1 = min(nt0 + p.tiles_per_split, p.ntiles);
                for (int nt = nt0; nt < nt1; nt++)
                    for (int kc = 0; kc < p.kchunks; kc++) {
                        mbar_wait(empty + stage, phase ^ 1);
                        mbar_expect_tx(full + stage, BF_STAGE_BYTES);
                        uint8_t *a = smem + (size_t) stage * BF_STAGE_BYTES;
                        tma_load_2d(a, &tmA, full + stage, kc * BF_BK, m * BF_BM);
                        tma_load_2d(a + BF_A_BYTES, &tmB, full + stage, kc * BF_BK, nt * BF_BN);
                        if (++stage == BF_STAGES) { stage = 0; phase ^= 1; }
                    }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int item = blockIdx.x; item < items; item += gridDim.x) {
                const int split = item / p.n_mtiles;
                const int nt0 = split * p.tiles_per_split, nt1 = min(nt0 + p.tiles_per_split, p.ntiles);
                for (int nt = nt0; nt < nt1; nt++) {
                    mbar_wait(tempty + acc, acc_phase ^ 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t d_tmem = tmem_base + (uint32_t) acc * BF_BN;
                    for (int kc = 0; kc < p.kchunks; kc++) {
                        mbar_wait(full + stage, phase);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint8_t *a = smem + (size_t) stage * BF_STAGE_BYTES;
                        const uint64_t adesc = umma_desc(a), bdesc = umma_desc(a + BF_A_BYTES);
#pragma unroll
                        for (int k = 0; k < BF_BK / 16; k++)
                            umma_f16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kc | k) != 0 ? 1u : 0u);
                        umma_commit(empty + stage);          // frees the stage when these MMAs retire
                        if (++stage == BF_STAGES) { stage = 0; phase ^= 1; }
                    }
                    umma_commit(tfull + acc);                // accumulator complete
                    acc ^= 1;
                    if (acc == 0) acc_phase ^= 1;
                }
            }
        }
    } else {
        const int quarter = warp & 3;                         // TMEM lanes this warp may read
        const int half = (warp - 2) >> 2;                     // which 128 of the 256 columns
        const int row = quarter * 32 + lane;
        const int et = threadIdx.x - 64;                      // 0..255 among the epilogue threads
        int acc = 0; uint32_t acc_phase = 0;
        const float NEG_INF = __int_as_float(0xff800000);
        for (int item = blockIdx.x; item < items; item += gridDim.x) {
            const int split = item / p.n_mtiles, m = item % p.n_mtiles;
            const int nt0 = split * p.tiles_per_split, nt1 = min(nt0 + p.tiles_per_split, p.ntiles);
            const int q = m * BF_BM + row;
            const bool valid_q = q < p.nq;
            // the K1 best (score, column) of this query row so far: sorted, in registers.  A hit
            // computes its rank with independent compares and shifts the tail with selects, so the
            // rare path is ~K1 independent instructions deep instead of a K1-long dependent chain.
            float ts[BF_K1];
            int32_t ti[BF_K1];
#pragma unroll
            for (int j = 0; j < BF_K1; j++) { ts[j] = NEG_INF; ti[j] = -1; }
            // seed: a slice that already finished for this query kept K1 rows scoring >= gthr, so rows
            // at or below it can never reach the query's top K1 -- skip them from the start
            const float seed = valid_q ? *reinterpret_cast<volatile float *>(p.gthr + q) : NEG_INF;
            float thr = seed;
            for (int nt = nt0; nt < nt1; nt++) {
                const int n0 = nt * BF_BN;
                float *xn = xnh + (nt & 1) * BF_BN;
                if constexpr (L2) {
                    for (int c = et; c < BF_BN; c += 32 * BF_EPI_WARPS) xn[c] = (n0 + c) < p.N ? p.xnh[n0 + c] : 0.f;
                    asm volatile("bar.sync 1, %0;" ::"n"(32 * BF_EPI_WARPS) : "memory");
                }
                mbar_wait(tfull + acc, acc_phase);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t taddr = tmem_base + ((uint32_t) (quarter * 32) << 16) + (uint32_t) acc * BF_BN + half * (BF_BN / 2);
                const int ncols = min(BF_BN, p.N - n0);       // columns past N are TMA zero fill
#pragma unroll 1
                for (int c = 0; c < BF_BN / 64; c++) {
                    uint32_t v[32];
                    tmem_ld32(taddr + c * 32, v);
                    const int col0 = half * (BF_BN / 2) + c * 32;
                    if constexpr (DBG) {
                        if (valid_q)
                            for (int i = 0; i < 32; i++)
                                if (col0 + i < ncols) p.dbg[(size_t) q * p.N + n0 + col0 + i] = __uint_as_float(v[i]);
                    }
                    float sv[32];
#pragma unroll
                    for (int i = 0; i < 32; i++) {
                        sv[i] = __uint_as_float(v[i]);
                        if constexpr (L2) sv[i] -= xn[col0 + i];
                        if (col0 + i >= ncols) sv[i] = NEG_INF;           // only the last tile of X has such columns
                    }
                    // one branch per 32 columns: the best of the chunk against the threshold
                    float mx = sv[0];
#pragma unroll
                    for (int i = 1; i < 32; i++) mx = fmaxf(mx, sv[i]);
                    if (valid_q && mx > thr) {
                        unsigned hits = 0;
#pragma unroll
                        for (int i = 0; i < 32; i++) hits |= sv[i] > thr ? (1u << i) : 0u;
                        while (hits) {
                            const int i = __ffs(hits) - 1;
                            hits &= hits - 1;
                            // sv[i] for a run-time i: five levels of selects keep sv in registers
                            float m16[16], m8[8], m4[4], m2[2];
#pragma unroll
                            for (int t = 0; t < 16; t++) m16[t] = (i & 16) ? sv[t + 16] : sv[t];
#pragma unroll
                            for (int t = 0; t < 8; t++) m8[t] = (i & 8) ? m16[t + 8] : m16[t];
#pragma unroll
                            for (int t = 0; t < 4; t++) m4[t] = (i & 4) ? m8[t + 4] : m8[t];
#pragma unroll
                            for (int t = 0; t < 2; t++) m2[t] = (i & 2) ? m4[t + 2] : m4[t];
                            const float sc = (i & 1) ? m2[1] : m2[0];
                            if (!(sc > thr)) continue;                    // the threshold rose inside this chunk
                            const int32_t id = n0 + col0 + i;
                            int r0 = 0, r1 = 0, r2 = 0, r3 = 0;           // rank = entries that stay ahead (ties keep earlier columns first)
#pragma unroll
                            for (int j = 0; j < BF_K1; j += 4) {
                                r0 += ts[j] >= sc ? 1 : 0;
                                r1 += ts[j + 1] >= sc ? 1 : 0;
                                r2 += ts[j + 2] >= sc ? 1 : 0;
                                r3 += ts[j + 3] >= sc ? 1 : 0;
                            }
                            const int r = (r0 + r1) + (r2 + r3);
#pragma unroll
                            for (int j = BF_K1 - 1; j >= 1; j--) {
                                ts[j] = j > r ? ts[j - 1] : (j == r ? sc : ts[j]);
                                ti[j] = j > r ? ti[j - 1] : (j == r ? id : ti[j]);
                            }
                            ts[0] = r == 0 ? sc : ts[0];
                            ti[0] = r == 0 ? id : ti[0];
                            thr = fmaxf(seed, ts[BF_K1 - 1]);
                        }
                    }
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty + acc);
                acc ^= 1;
                if (acc == 0) acc_phase ^= 1;
            }
            if (valid_q) {
                const size_t slot = (size_t) q * (2 * p.S) + 2 * split + half;
#pragma unroll
                for (int j = 0; j < BF_K1; j++) { p.cand_score[slot * BF_K1 + j] = ts[j]; p.cand_id[slot * BF_K1 + j] = ti[j]; }
                p.cand_thr[slot] = thr;                        // every row this slice dropped scored <= thr
                if (ti[BF_K1 - 1] >= 0) atomic_max_float(p.gthr + q, ts[BF_K1 - 1]);
            }
        }
    }
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    }
}

// rows of the index (padded fp32 / fp16 rows) -> bf16 [n x kpad], plus 0.5|x|^2 and max |x|
template <typename T>
__global__ void to_bf16_kernel(const char *__restrict__ rows, size_t row_bytes, int dim, int kpad, int64_t n,
                               __nv_bfloat16 *__restrict__ out, float *__restrict__ xnh, unsigned int *__restrict__ max_norm_bits)
{
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t) blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= n) return;
    const T *src = reinterpret_cast<const T *>(rows + r * row_bytes);
    float s = 0.f;
    for (int e = lane; e < kpad; e += 32) {
        const float v = e < dim ? (float) src[e] : 0.f;
        s += v * v;
        out[r * kpad + e] = __float2bfloat16_rn(v);
    }
    for (int b = 16; b >= 1; b >>= 1) s += __shfl_xor_sync(FULL, s, b);
    if (lane == 0) {
        if (xnh) xnh[r] = 0.5f * s;
        if (max_norm_bits) atomicMax(max_norm_bits, __float_as_uint(sqrtf(s) * 1.000001f));
    }
}

// exact fp32 re-rank results -> top-k by (distance, id) and the certificate
__global__ void bf_select_kernel(const int32_t *__restrict__ cand_id, const float *__restrict__ cand_dist,
                                 const float *__restrict__ cand_thr, const float *__restrict__ qnorm2h,
                                 const unsigned int *__restrict__ max_norm_bits, int nq, int S, int k, int l2,
                                 int32_t *__restrict__ out_elem, float *__restrict__ out_dist, int32_t *__restrict__ uncertain)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const int C = S * BF_K1;
    constexpr int KMAX = 128;
    float bd[KMAX]; int32_t bi[KMAX];
    int cnt = 0;
    for (int c = 0; c < C; c++) {
        const int32_t id = cand_id[(size_t) q * C + c];
        if (id < 0) continue;
        const float d = cand_dist[(size_t) q * C + c];
        if (cnt == k && !(d < bd[k - 1] || (d == bd[k - 1] && id < bi[k - 1]))) continue;
        int j = cnt < k ? cnt++ : k - 1;
        while (j > 0 && (d < bd[j - 1] || (d == bd[j - 1] && id < bi[j - 1]))) { bd[j] = bd[j - 1]; bi[j] = bi[j - 1]; j--; }
        bd[j] = d; bi[j] = id;
    }
    for (int j = 0; j < k; j++) {
        out_elem[(size_t) q * k + j] = j < cnt ? bi[j] : -1;
        out_dist[(size_t) q * k + j] = j < cnt ? bd[j] : __int_as_float(0x7f800000);
    }
    // certificate: every row a slice did not keep has bf16 score <= thr, so its true score is at most
    // thr + E with E = (2^-8 + 2^-11) |q| |x|max
    const float qn = sqrtf(2.f * qnorm2h[q]);
    const float E = (1.f / 256.f + 1.f / 2048.f) * qn * __uint_as_float(*max_norm_bits);
    bool ok = true;
    if (cnt == k) {
        const float tau = bd[k - 1];
        for (int s = 0; s < S && ok; s++) {
            const float thr = cand_thr[(size_t) q * S + s];
            if (thr == __int_as_float(0xff800000)) continue;
            const float lb = l2 ? (2.f * qnorm2h[q] - 2.f * (thr + E)) : -(thr + E);
            ok = lb > tau;
        }
    } else {
        for (int s = 0; s < S; s++) ok = ok && cand_thr[(size_t) q * S + s] == __int_as_float(0xff800000);
    }
    uncertain[q] = ok ? 0 : 1;
}

// exhaustive fp32 path for queries the certificate rejected: distances to every row are computed by
// the canonical distance kernel (dist_batch), then selected here.  One block per query.
__global__ void bf_full_select_kernel(const float *__restrict__ dist, int64_t n, int k, int32_t *__restrict__ out_elem,
                                      float *__restrict__ out_dist)
{
    // every round extracts the next (distance, id) minimum with a block-wide arg-min over n: n*k work,
    // used only for the rare query the certificate rejected.
    __shared__ float prev_d;
    __shared__ int32_t prev_i;
    if (threadIdx.x == 0) { prev_d = __int_as_float(0xff800000); prev_i = -1; }
    __syncthreads();
    __shared__ float rd[256];
    __shared__ int32_t ri[256];
    for (int j = 0; j < k; j++) {
        float bd = __int_as_float(0x7f800000);
        int32_t bi = -1;
        const float pd = prev_d; const int32_t pi = prev_i;
        for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
            const float d = dist[i];
            const bool after = d > pd || (d == pd && (int32_t) i > pi);
            if (after && (bi < 0 || d < bd || (d == bd && (int32_t) i < bi))) { bd = d; bi = (int32_t) i; }
        }
        rd[threadIdx.x] = bd; ri[threadIdx.x] = bi;
        __syncthreads();
        for (int s = blockDim.x / 2; s > 0; s >>= 1) {
            if (threadIdx.x < s) {
                const float d2 = rd[threadIdx.x + s]; const int32_t i2 = ri[threadIdx.x + s];
                if (i2 >= 0 && (ri[threadIdx.x] < 0 || d2 < rd[threadIdx.x] || (d2 == rd[threadIdx.x] && i2 < ri[threadIdx.x]))) {
                    rd[threadIdx.x] = d2; ri[threadIdx.x] = i2;
                }
            }
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            out_elem[j] = ri[0];
            out_dist[j] = ri[0] >= 0 ? rd[0] : __int_as_float(0x7f800000);
            prev_d = rd[0]; prev_i = ri[0];
        }
        __syncthreads();
    }
}

__global__ void iota_kernel(int32_t *a, int64_t n)
{
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = (int32_t) i;
}

typedef CUresult (*encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                              const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                              CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static encode_fn get_encode()
{
    static encode_fn fn = nullptr;
    if (fn) return fn;
    void *p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || !p) return nullptr;
    fn = (encode_fn) p;
    return fn;
}

static int make_map(CUtensorMap *map, void *base, uint64_t rows, uint64_t kpad, uint32_t box_rows)
{
    encode_fn enc = get_encode();
    if (!enc) { set_error("cuTensorMapEncodeTiled is not available from the driver"); return HB_ECUDA; }
    cuuint64_t gdim[2] = { kpad, rows };
    cuuint64_t gstr[1] = { kpad * 2 };
    cuuint32_t box[2] = { (cuuint32_t) BF_BK, box_rows };
    cuuint32_t estr[2] = { 1, 1 };
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d)", (int) r); return HB_ECUDA; }
    return HB_OK;
}

struct BfState {
    DevBuf gthr, xb, xnh, misc, qraw, qn, qb, qnh, cand_score, cand_id, cand_thr, cand_dist, out_elem, out_dist, uncertain, iota, full_dist, dbg;
    int64_t built_n = -1;
    uint64_t built_gen = 0;      // hb_index::generation the bf16 image was made from
    int kpad = 0;
};

// the exact scan's state belongs to the handle (hb_index::bf): distinct handles share nothing
static BfState *bf_state(hb_index *ix)
{
    if (!ix->bf) ix->bf = new BfState();
    return static_cast<BfState *>(ix->bf);
}

void bruteforce_release(hb_index *ix)
{
    if (!ix->bf) return;
    BfState *s = static_cast<BfState *>(ix->bf);
    ix->bf = nullptr;
    DevBuf *b[] = { &s->gthr, &s->xb, &s->xnh, &s->misc, &s->qraw, &s->qn, &s->qb, &s->qnh, &s->cand_score, &s->cand_id, &s->cand_thr,
                    &s->cand_dist, &s->out_elem, &s->out_dist, &s->uncertain, &s->iota, &s->full_dist, &s->dbg };
    for (auto x : b) x->release();
    delete s;
}

}   // namespace hb

using namespace hb;

extern "C" {

// dbg_scores: optional host buffer nq x n receiving the raw bf16-GEMM scores (tests); stats (optional):
// [0] queries certified exact by the bf16 bound, [1] queries re-scanned in fp32, [2] GEMM kernel ms
int hb_bruteforce_ex(hb_index *ix, const void *host_queries, int64_t nq, int k, int32_t *out_elem, float *out_dist,
                     float *dbg_scores, float *stats)
{
    if (!ix || !host_queries || !out_elem || !out_dist || k < 1 || k > 128) { set_error("hb_bruteforce: bad argument (1 <= k <= 128)"); return HB_EINVAL; }
    if (nq <= 0) return HB_OK;
    if (ix->metric == HB_L1) {
        // the exact scan is a q.x contraction (bf16 GEMM + fp32 re-rank): squared L2, inner product and cosine only
        set_error("hb_bruteforce: the exact scan supports the l2, ip and cosine operator classes, not l1");
        return HB_EINVAL;
    }
    HB_CK(cudaSetDevice(ix->device));
    cudaStream_t s = ix->stream;
    const int64_t n = ix->n;
    if (n == 0) {
        for (int64_t i = 0; i < nq * k; i++) { out_elem[i] = -1; out_dist[i] = INFINITY; }
        return HB_OK;
    }
    BfState &st = *bf_state(ix);
    const int kpad = ((ix->dim + BF_BK - 1) / BF_BK) * BF_BK;
    const bool l2 = ix->metric == HB_L2;
    HB_CK(st.misc.ensure(64));
    unsigned int *max_bits = st.misc.as<unsigned int>();

    // bf16 image of the partition (rebuilt whenever the index changed: every mutation bumps the generation)
    if (st.built_n != n || st.kpad != kpad || st.built_gen != ix->generation) {
        HB_CK(st.xb.ensure((size_t) n * kpad * 2));
        HB_CK(st.xnh.ensure(sizeof(float) * n));
        HB_CK(cudaMemsetAsync(max_bits, 0, 4, s));
        const int wpb = 8, grid = (int) ((n + wpb - 1) / wpb);
        if (ix->dtype == HB_F32)
            to_bf16_kernel<float><<<grid, wpb * 32, 0, s>>>(ix->d_vecs, ix->row_bytes, ix->dim, kpad, n, st.xb.as<__nv_bfloat16>(), st.xnh.as<float>(), max_bits);
        else
            to_bf16_kernel<__half><<<grid, wpb * 32, 0, s>>>(ix->d_vecs, ix->row_bytes, ix->dim, kpad, n, st.xb.as<__nv_bfloat16>(), st.xnh.as<float>(), max_bits);
        HB_CK(cudaGetLastError());
        st.built_n = n; st.kpad = kpad; st.built_gen = ix->generation;
    }

    // queries: H2D, normalise for cosine (exact path), bf16 copy padded to a whole tile
    const size_t qbytes = (size_t) nq * ix->dim * ix->esize;
    const int n_mtiles = (int) ((nq + BF_BM - 1) / BF_BM);
    const int64_t nq_pad = (int64_t) n_mtiles * BF_BM;
    HB_CK(st.qraw.ensure(qbytes));
    HB_CK(st.qn.ensure(qbytes));
    HB_CK(st.qb.ensure((size_t) nq_pad * kpad * 2));
    HB_CK(st.qnh.ensure(sizeof(float) * nq_pad));
    HB_CK(cudaMemcpyAsync(st.qraw.p, host_queries, qbytes, cudaMemcpyHostToDevice, s));
    const void *qexact = st.qraw.p;
    if (ix->metric == HB_COSINE) {
        int rc = normalize_dev(ix, st.qraw.p, nq, st.qn.p, s);   // the canonical l2_normalize
        if (rc) return rc;
        qexact = st.qn.p;
    }
    HB_CK(cudaMemsetAsync(st.qb.p, 0, (size_t) nq_pad * kpad * 2, s));
    {
        const int wpb = 8, grid = (int) ((nq + wpb - 1) / wpb);
        const size_t qrow = (size_t) ix->dim * ix->esize;
        if (ix->dtype == HB_F32)
            to_bf16_kernel<float><<<grid, wpb * 32, 0, s>>>((const char *) qexact, qrow, ix->dim, kpad, nq, st.qb.as<__nv_bfloat16>(), st.qnh.as<float>(), nullptr);
        else
            to_bf16_kernel<__half><<<grid, wpb * 32, 0, s>>>((const char *) qexact, qrow, ix->dim, kpad, nq, st.qb.as<__nv_bfloat16>(), st.qnh.as<float>(), nullptr);
        HB_CK(cudaGetLastError());
    }

    // work decomposition: (query tile, slice of X); slices sized so the grid fills whole waves
    const int ntiles = (int) ((n + BF_BN - 1) / BF_BN);
    int best_S = 1; double best_eff = -1;
    for (int S = 1; S <= 16 && S <= ntiles; S++) {
        const int64_t items = (int64_t) n_mtiles * S;
        const double eff = (double) items / (double) (((items + ix->num_sms - 1) / ix->num_sms) * ix->num_sms);
        if (eff > best_eff + 1e-9 || (std::fabs(eff - best_eff) <= 1e-9 && S > best_S && S <= 8)) { best_eff = eff; best_S = S; }
    }
    BfParams p;
    memset(&p, 0, sizeof p);
    p.nq = (int) nq; p.N = (int) n; p.kchunks = kpad / BF_BK; p.n_mtiles = n_mtiles;
    p.tiles_per_split = (ntiles + best_S - 1) / best_S;
    p.S = (ntiles + p.tiles_per_split - 1) / p.tiles_per_split;
    p.ntiles = ntiles;
    p.xnh = l2 ? st.xnh.as<float>() : nullptr;
    const int S2 = 2 * p.S;                      // two column halves per slice
    const size_t C = (size_t) S2 * BF_K1;
    HB_CK(st.cand_score.ensure(sizeof(float) * nq * C));
    HB_CK(st.cand_id.ensure(sizeof(int32_t) * nq * C));
    HB_CK(st.cand_thr.ensure(sizeof(float) * nq * S2));
    HB_CK(st.cand_dist.ensure(sizeof(float) * nq * C));
    HB_CK(st.out_elem.ensure(sizeof(int32_t) * nq * k));
    HB_CK(st.out_dist.ensure(sizeof(float) * nq * k));
    HB_CK(st.uncertain.ensure(sizeof(int32_t) * nq));
    p.cand_score = st.cand_score.as<float>(); p.cand_id = st.cand_id.as<int32_t>(); p.cand_thr = st.cand_thr.as<float>();
    if (dbg_scores) {
        HB_CK(st.dbg.ensure(sizeof(float) * nq * n));
        p.dbg = st.dbg.as<float>();
    }
    HB_CK(st.gthr.ensure(sizeof(float) * nq_pad));
    {
        std::vector<float> ninf((size_t) nq_pad, -INFINITY);
        HB_CK(cudaMemcpyAsync(st.gthr.p, ninf.data(), sizeof(float) * nq_pad, cudaMemcpyHostToDevice, s));
        HB_CK(cudaStreamSynchronize(s));
    }
    p.gthr = st.gthr.as<float>();
    CUtensorMap tmA, tmB;
    int rc = make_map(&tmA, st.qb.p, (uint64_t) nq_pad, (uint64_t) kpad, BF_BM);
    if (rc) return rc;
    rc = make_map(&tmB, st.xb.p, (uint64_t) n, (uint64_t) kpad, BF_BN);
    if (rc) return rc;
    const int items = p.n_mtiles * p.S;
    const int grid = std::min(items, ix->num_sms);
    auto kern = dbg_scores ? (l2 ? bf_gemm_topk_kernel<true, true> : bf_gemm_topk_kernel<true, false>)
                           : (l2 ? bf_gemm_topk_kernel<false, true> : bf_gemm_topk_kernel<false, false>);
    HB_CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) BF_SMEM));
    HB_CK(cudaEventRecord(ix->ev0, s));
    kern<<<grid, BF_THREADS, BF_SMEM, s>>>(tmA, tmB, p);
    HB_CK(cudaGetLastError());
    HB_CK(cudaEventRecord(ix->ev1, s));

    // fp32 re-rank of every candidate in the canonical order, then select + certify
    DistBatchParams dp;
    dp.g = ix->view(); dp.queries = qexact; dp.nq = nq; dp.cand = st.cand_id.as<int32_t>(); dp.nc = (int) C; dp.out = st.cand_dist.as<float>();
    HB_CK(get_dist_launcher(ix->dtype, metric_kind(ix->metric))(dp, s));
    bf_select_kernel<<<(int) ((nq + 63) / 64), 64, 0, s>>>(st.cand_id.as<int32_t>(), st.cand_dist.as<float>(), st.cand_thr.as<float>(),
                                                          st.qnh.as<float>(), max_bits, (int) nq, S2, k, l2 ? 1 : 0,
                                                          st.out_elem.as<int32_t>(), st.out_dist.as<float>(), st.uncertain.as<int32_t>());
    HB_CK(cudaGetLastError());
    std::vector<int32_t> unc(nq);
    HB_CK(cudaMemcpyAsync(out_elem, st.out_elem.p, sizeof(int32_t) * nq * k, cudaMemcpyDeviceToHost, s));
    HB_CK(cudaMemcpyAsync(out_dist, st.out_dist.p, sizeof(float) * nq * k, cudaMemcpyDeviceToHost, s));
    HB_CK(cudaMemcpyAsync(unc.data(), st.uncertain.p, sizeof(int32_t) * nq, cudaMemcpyDeviceToHost, s));
    if (dbg_scores) HB_CK(cudaMemcpyAsync(dbg_scores, st.dbg.p, sizeof(float) * nq * n, cudaMemcpyDeviceToHost, s));
    HB_CK(cudaStreamSynchronize(s));
    float gemm_ms = 0.f;
    cudaEventElapsedTime(&gemm_ms, ix->ev0, ix->ev1);

    // exhaustive fp32 re-scan of the queries the certificate rejected
    int64_t n_unc = 0;
    for (int64_t q = 0; q < nq; q++) n_unc += unc[q] ? 1 : 0;
    if (n_unc > 0) {
        HB_CK(st.iota.ensure(sizeof(int32_t) * n));
        HB_CK(st.full_dist.ensure(sizeof(float) * n));
        iota_kernel<<<(int) ((n + 255) / 256), 256, 0, s>>>(st.iota.as<int32_t>(), n);
        const size_t qrow = (size_t) ix->dim * ix->esize;
        for (int64_t q = 0; q < nq; q++) {
            if (!unc[q]) continue;
            DistBatchParams fp;
            fp.g = ix->view(); fp.queries = (const char *) qexact + q * qrow; fp.nq = 1; fp.cand = st.iota.as<int32_t>();
            fp.nc = (int) n; fp.out = st.full_dist.as<float>();
            HB_CK(get_dist_launcher(ix->dtype, metric_kind(ix->metric))(fp, s));
            bf_full_select_kernel<<<1, 256, 0, s>>>(st.full_dist.as<float>(), n, k, st.out_elem.as<int32_t>() + q * k, st.out_dist.as<float>() + q * k);
            HB_CK(cudaGetLastError());
            HB_CK(cudaMemcpyAsync(out_elem + q * k, st.out_elem.as<int32_t>() + q * k, sizeof(int32_t) * k, cudaMemcpyDeviceToHost, s));
            HB_CK(cudaMemcpyAsync(out_dist + q * k, st.out_dist.as<float>() + q * k, sizeof(float) * k, cudaMemcpyDeviceToHost, s));
        }
        HB_CK(cudaStreamSynchronize(s));
    }
    if (stats) { stats[0] = (float) (nq - n_unc); stats[1] = (float) n_unc; stats[2] = gemm_ms; }
    return HB_OK;
}

int hb_bruteforce(hb_index *ix, const void *host_queries, int64_t nq, int k, int32_t *out_elem, float *out_dist)
{
    return hb_bruteforce_ex(ix, host_queries, nq, k, out_elem, out_dist, nullptr, nullptr);
}

}   // extern "C"
