// search.cu — GraphSearcher.search, device resident: one CTA walks one query through the whole traversal
// (base:graph/GraphSearcher.java:263-282 internalSearch, :334-353 initializeInternal, :355-370 stopSearch,
//  :406-457 searchOneLayer, :471-507 reranking; neighbour loop base:graph/OnHeapGraphIndex.java:475-483).
//
// State per query, all in shared memory (the kernel's own header comment, further down, has the exactness argument):
//   * ONE list sorted by the reference's 64-bit key holding the nodes SEEN so far that can still matter, each with an
//     "expanded" and an "accepted" flag; its unexpanded entries are the reference's candidate max-heap in pop order;
//   * a shadow copy of the reference's bounded result heap (same array, same sift procedures): stopSearch's strict <, the
//     "tie with the worst result is expanded but not added" rule and NodeQueue.rerank's array order come from it;
//   * upper levels run with a 1-entry result heap over the same list; moving down a level clears the expanded flags
//     (setEntryPointsFromPreviousLayer);
//   * visited = an exact set of node ids, never cleared between levels (GraphSearcher keeps `visited` across levels):
//     16-bit region-tagged slots in shared memory (visited_insert_smem), or — for graphs / beams the shared-memory table
//     does not take, and for the re-run of a query that outgrew it — an open-addressing table of 32-bit ids in a per-CTA slice
//     of global scratch (visited_insert).
// Every hop is: read one adjacency row (FusedPQ: one record) -> filter through visited, requesting every new row from DRAM
// with one bulk L2 prefetch -> score the survivors with the row scorers of scorers.cuh -> parallel rank-merge into the list.
#include <limits.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>

#include "kernels.h"

namespace jv {

struct SearchParams {
    GraphDesc g;
    DataDesc approx;
    DataDesc rerank;
    int has_rerank;
    int metric;
    const float *queries;
    int query_stride;
    int nq, topK, rerankK;
    int list_cap;    // entries the candidate list retains (>= rerankK; the slack holds the tie tail)
    int list_alloc;  // entries per list buffer (>= list_cap and >= sort_pow2)
    int sort_pow2;   // next power of two >= rerankK (bitonic sort of the result heap)
    int visited_cap;
    int visited_shift;
    int32_t *visited_tables;
    int *work_counter;
    int32_t *nodes_out;
    float *scores_out;
    SearchCounters *counters;
    uint8_t *overflow;
    const int32_t *query_index;
    int blobA_floats, blobR_floats, smemA_floats;  // smemA_floats: what the walking scorer's prepared query takes of shared memory
    float *blob_global;  // PQ: per-CTA slices of global scratch (L2 resident) hold the LUT rows of the sub-spaces >= pq_smem_m
    int pq_smem_m;       // PQ: sub-spaces [0, pq_smem_m) keep their LUT rows in shared memory (multiple of 4; M = all, 0 = none)
    // acceptOrds / threshold / rerankFloor of GraphSearcher.search(sp, topK, rerankK, threshold, rerankFloor, acceptOrds)
    const uint32_t *accept_bits;  // bit (node & 31) of word (node >> 5); nullptr = Bits.ALL
    long long accept_stride;      // words between two queries' bitsets (0 = one bitset shared by the batch)
    float threshold, rerank_floor;
    int filtered;                 // accept_bits != nullptr || threshold > 0
    const int *arrived;           // nullptr, or: query i may be read only once *arrived > i (the H2D copy is still running)
    int lenient;                  // insert searches of the builder: a full visited table ends the walk with what it has, a tie tail
                                  // that does not fit is dropped — counted in counters->overflowed, never an error (build.cu)
    // visited set in shared memory (plan_search decides): 2^vis_slots_log 16-bit slots split into 2^(vis_bits-15) regions; 0 = the
    // per-CTA global table
    int vis_slots_log, vis_rlog;
    unsigned vis_idmask;
    int early_pf;      // request the adjacency / FusedPQ record of a new candidate that lands among the next two pops at score time
    int pq_rows;       // PQ walk: lane = candidate, warp = partial sum (score_pq_partial) instead of an 8-lane group per candidate
    int row_prefetch;  // fp32 / NVQ walks: 1 = a bulk L2 prefetch of every newly visited row is issued by the thread that discovered it
    int sketch;        // fp32 DOT_PRODUCT walks: `sk` bounds a candidate's score before its row is read (see SKETCH_MARGIN)
    F32Sketch sk;
    unsigned long long *dbg;  // JV_SEARCH_PROFILE builds only: per-phase cycle totals
};

// Slack of the sketch bound, relative to ||q|| ||x||. A candidate is dropped unread when
//     score_map(fp32(P q) . fp32(P x) + ||q_perp|| ||r|| + SKETCH_MARGIN ||q|| ||x||) < score of the list's last entry,
// which is sound when the margin covers every gap between that sum and the fp32 score the row scorer would have produced:
//   * the row scorer's 768-term fp32 dot: at most gamma_768 = 768 * 2^-24 = 4.6e-5 of ||q|| ||x|| (sum |q_i x_i| <= ||q|| ||x||);
//   * the 32-term fp32 dot of the sketch, with P q and P x each rounded once from double: ~(32 + 2) * 2^-24 = 2e-6;
//   * P rounded to fp32 is orthonormal only to ~32 * 2^-23 = 3.8e-6, which P^T r != 0 costs at most ~4e-6 (||q_perp|| itself is
//     exact: it is measured against the Gram matrix of the rounded basis);
//   * ||q_perp||, ||q||, ||r||, ||x|| are rounded UP from double, and the three fp32 additions of the bound cost a few 2^-24.
// Total below 6e-5; 1e-3 keeps a factor of 15 in hand and drops ~0.1 % fewer candidates than the exact test would.
constexpr float SKETCH_MARGIN = 1e-3f;

// whole CTA: out[0..SKETCH_K) = fp32(P q), out[SKETCH_K] = ||q - P^T P q||, out[SKETCH_K + 1] = ||q||, from the prepared fp32 query
// in shared memory. In double: with a = P q, ||q - P^T a||^2 = ||q||^2 - 2 a.a + a^T G a, G the Gram matrix of the stored basis.
__device__ __forceinline__ void sketch_prepare(const F32Sketch &sk, int stride, const float *q, float *out, double *dred)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    for (int j = warp; j < SKETCH_K; j += nw) {
        const float *b = sk.basis + (size_t)j * stride;
        double a = 0.0;
        for (int i = lane; i < stride; i += 32) a = fma((double)__ldg(b + i), (double)q[i], a);
        a = warp_sum_d(a);
        if (lane == 0) dred[j] = a;
    }
    double qq = 0.0;
    for (int i = tid; i < stride; i += blockDim.x) qq = fma((double)q[i], (double)q[i], qq);
    qq = warp_sum_d(qq);
    if (lane == 0) dred[SKETCH_K + warp] = qq;
    __syncthreads();
    if (warp == 0) {
        const double a = dred[lane];
        double t = 0.0;
        for (int k = 0; k < SKETCH_K; k++) t = fma(__ldg(sk.gram + lane * SKETCH_K + k), dred[k], t);
        const double aa = warp_sum_d(a * a), aga = warp_sum_d(a * t);
        double q2 = 0.0;
        for (int w = 0; w < nw; w++) q2 += dred[SKETCH_K + w];
        out[lane] = (float)a;
        if (lane == 0) {
            out[SKETCH_K] = __double2float_ru(sqrt(fmax(0.0, q2 - 2.0 * aa + aga)));
            out[SKETCH_K + 1] = __double2float_ru(sqrt(q2));
        }
    }
    __syncthreads();
}

__device__ __forceinline__ bool visited_insert(int32_t *t, unsigned mask, int shift, int32_t v)
{
    unsigned h = ((unsigned)v * 2654435761u) >> shift;
    for (unsigned probes = 0; probes <= mask; ++probes) {
        const int old = atomicCAS(&t[h], -1, v);
        if (old == -1) return true;
        if (old == v) return false;
        h = (h + 1) & mask;
    }
    return false;
}

// The same set in shared memory, 16 bits per slot. x = id * odd mod 2^bits is a bijection on [0, 2^bits) (bits = ceil(log2 n) >= 15);
// its top (bits - 15) bits choose a REGION of the table, its low 15 bits are the tag stored there (bit 15 = occupied), and a probe
// sequence never leaves its region — so (region, tag) identifies the id exactly and the set has no false positives. A full region
// reports through *fail (the query is re-run on the global table, like any visited-table overflow).
__device__ __forceinline__ bool visited_insert_smem(unsigned short *t, unsigned idmask, int rlog, int32_t v, int *fail)
{
    const unsigned x = ((unsigned)v * 0x9E3779B1u) & idmask;
    const unsigned tag = x & 0x7fffu;
    const unsigned short val = (unsigned short)(tag | 0x8000u);
    const unsigned rmask = (1u << rlog) - 1u;
    unsigned short *base = t + ((size_t)(x >> 15) << rlog);
    unsigned h = (tag * 0x9E3779B1u) >> (32 - rlog);
    for (unsigned probes = 0; probes <= rmask; ++probes) {
#ifdef JV_VIS_CAS_GENERIC
        const unsigned short old = atomicCAS(&base[h], (unsigned short)0, val);
#else
        // explicit .shared state space: a 16-bit CAS is an LDS + 32-bit ATOMS.CAS loop on the containing word; through a generic
        // pointer (atomicCAS on unsigned short *) the compiler emits the slower generic ATOM.E.CAS
        unsigned short old;
        asm volatile("atom.shared.cas.b16 %0, [%1], %2, %3;" : "=h"(old) : "r"(smem_u32(base + h)), "h"((unsigned short)0), "h"(val) : "memory");
#endif
        if (old == 0) return true;
        if (old == val) return false;
        h = (h + 1) & rmask;
    }
    *fail = 1;
    return false;
}

// number of keys in the descending-sorted array a[0..n) that are greater than k
__device__ __forceinline__ int count_greater_desc(const long long *a, int n, long long k)
{
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a[mid] > k) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ void bitonic_sort_desc_block(long long *keys, int n_pow2)
{
    for (int k = 2; k <= n_pow2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n_pow2; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const long long a = keys[i], b = keys[ixj];
                    const bool desc = (i & k) == 0;
                    if (desc ? (a < b) : (a > b)) { keys[i] = b; keys[ixj] = a; }
                }
            }
            __syncthreads();
        }
    }
}

// The reference's result queue is a BoundedLongHeap (min-heap of keys, 1-based array): its ARRAY ORDER decides which of two
// equal exact scores survives NodeQueue.rerank, so the device keeps the same array with the same sift procedures
// (base:util/AbstractLongHeap.java:158-187 upHeap / downHeap, base:util/BoundedLongHeap.java:60-70,100-104 push / updateTop).
__device__ __forceinline__ void heap_up(long long *h, int pos)
{
    int i = pos;
    const long long v = h[i];
    int j = i >> 1;
    while (j > 0 && v < h[j]) {
        h[i] = h[j];
        i = j;
        j >>= 1;
    }
    h[i] = v;
}
__device__ __forceinline__ void heap_down(long long *h, int size, int pos)
{
    int i = pos;
    const long long v = h[i];
    int j = i << 1, k = j + 1;
    if (k <= size && h[k] < h[j]) j = k;
    while (j <= size && h[j] < v) {
        h[i] = h[j];
        i = j;
        j = i << 1;
        k = j + 1;
        if (k <= size && h[k] < h[j]) j = k;
    }
    h[i] = v;
}

#ifndef JV_SEARCH_THREADS
#define JV_SEARCH_THREADS 256
#endif
#ifndef JV_SEARCH_MINB
#define JV_SEARCH_MINB 5
#endif
#ifndef JV_SEARCH_MINB_PQ
#define JV_SEARCH_MINB_PQ 6  // tools/sweep_pq_minb.sh: 5 -> 777k q/s, 6 -> 817k, 8 -> 592k (c3, LUT in L2)
#endif
// CTA width per walking scorer. fp32 / NVQ rows are scored a warp per row and, with every new row already on its way to L2
// (bulk prefetch), the walk gains from MORE queries in flight rather than more warps per query: 128 threads, 10 CTAs per SM
// (c2: 14.7 -> 14.2 ms). PQ / BQ score a hop's ~28 candidates in one pass over 8 warps (PQ: one warp per partial sum): 256 threads.
#ifndef JV_SEARCH_THREADS_ROWS
#define JV_SEARCH_THREADS_ROWS 128
#endif
template <int KIND>
struct SearchThreads {
    static constexpr int value = (KIND == KIND_F32 || KIND == KIND_NVQ) ? JV_SEARCH_THREADS_ROWS : JV_SEARCH_THREADS;
};
static int search_threads_of(int kind) { return (kind == KIND_F32 || kind == KIND_NVQ) ? JV_SEARCH_THREADS_ROWS : JV_SEARCH_THREADS; }

// optional phase timers (tools/: build with JV_NVCC_EXTRA=-DJV_SEARCH_PROFILE); compiled out of the product build
#ifdef JV_SEARCH_PROFILE
#define JV_T(var) const long long var = clock64()
#define JV_ACC(slot, a, b) do { if (threadIdx.x == 0) dbg_local[slot] += (unsigned long long)((b) - (a)); } while (0)
#else
#define JV_T(var)
#define JV_ACC(slot, a, b)
#endif

// flags of a list entry
constexpr uint8_t F_EXPANDED = 1;  // popped from the candidate queue at this level
constexpr uint8_t F_ACCEPTED = 2;  // acceptOrds.get(node) && score >= threshold (what addTopCandidate requires at level 0)

// State per query (see the file header). The traversal is EXACTLY the reference's, ties included:
//   candidates  = the unexpanded entries of ONE list sorted by the reference key (pop order = the max-heap's pop order);
//   results     = `heap`, the reference's BoundedLongHeap of the best rerankK (1 on upper levels) popped nodes, same array order;
//   stopSearch  = results full && score(best candidate) < score(worst result)  (GraphSearcher.java:355-361, strict);
//   addTopCandidate = push while not full, replace the worst when strictly better, otherwise (tie with the worst) expand the
//                 node without adding it (GraphSearcher.java:520-530);
//   a list entry may be dropped when at least rerankK accepted entries score STRICTLY higher (it can never be popped before
//   stopSearch fires); the list keeps `list_cap` >= rerankK entries so a tie tail survives, and a query whose tail does not fit
//   is re-run by the host with a larger list (overflow code 2), never answered approximately;
//   upper levels: a node refused by addTopCandidate is neither a result nor evicted, so it is removed from the list at once
//   (setEntryPointsFromPreviousLayer re-queues results + evicted only, GraphSearcher.java:316-323).
// MINB: resident CTAs per SM the register allocation is capped for. PQ is compiled twice: 6 (40 registers; the L2-LUT mode, where
// nothing else limits residency) and 4 (64 registers; the modes whose shared-memory LUT part allows at most 4-5 CTAs anyway).
// VSM: the visited set lives in shared memory (a template parameter, not a run-time flag: the two forms must not cost each other
// registers — the fp32 walk lost 15 % when they shared one instantiation).
template <int KIND, int METRIC, int MINB, bool VSM>
__global__ void __launch_bounds__(SearchThreads<KIND>::value, MINB) graph_search_kernel(SearchParams P)
{
    constexpr int SEARCH_THREADS = SearchThreads<KIND>::value;
    constexpr int HEAP_TID = SEARCH_THREADS - 32;  // the thread that maintains the result heap (lane 0 of the last warp)
    constexpr int G = GroupOf<KIND>::value;
    constexpr int NG = SEARCH_THREADS / G;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // prepared query of the walking scorer. PQ: the LUT may be split, rows of sub-spaces < pq_smem_m in shared memory (blobA), the
    // others in this CTA's global slice (blobH); every other kind: all of it in shared memory
    float *blobA = reinterpret_cast<float *>(smem_raw);
    float *blobH = P.blob_global ? P.blob_global + (size_t)blockIdx.x * P.blobA_floats : blobA;
    const int splitm = (KIND == KIND_PQ && P.blob_global) ? P.pq_smem_m : (1 << 30);
    float *blobR = reinterpret_cast<float *>(smem_raw) + P.smemA_floats;
    long long *keys0 = reinterpret_cast<long long *>(blobR + P.blobR_floats);
    long long *keys1 = keys0 + P.list_alloc;
    long long *cand_keys = keys1 + P.list_alloc;
    long long *heap = cand_keys + MAX_DEGREE;  // 1-based, rerankK entries
    int32_t *cand_ids = reinterpret_cast<int32_t *>(heap + ((P.rerankK + 2) & ~1));
    uint8_t *cand_acc = reinterpret_cast<uint8_t *>(cand_ids + MAX_DEGREE);
    uint8_t *cand_slot = cand_acc + MAX_DEGREE;  // fused PQ: position of the candidate inside the expanded node's record
    uint8_t *flags0 = cand_slot + MAX_DEGREE;
    uint8_t *flags1 = flags0 + P.list_alloc;
    unsigned short *vis = reinterpret_cast<unsigned short *>((reinterpret_cast<uintptr_t>(flags1 + P.list_alloc) + 15) & ~(uintptr_t)15);
    constexpr bool vsm = VSM;  // visited set in shared memory (16-bit slots) instead of the per-CTA global table
    uint32_t *pq_stage = reinterpret_cast<uint32_t *>(vis + (VSM ? (1 << P.vis_slots_log) : 0));  // PQ row mode: the hop's code rows
    float *pq_part = reinterpret_cast<float *>(pq_stage + P.g.degree * ((P.approx.code_stride >> 2) + 1));  // and its partial sums
    __shared__ int s_vfail;
    __shared__ long long s_nk;  // key of the second unexpanded entry behind the one being expanded (see JV_EMIT)
    __shared__ float red[36];
    __shared__ int s_q, s_n, s_m, s_hsize, s_cnt;
    __shared__ int s_drop[2];  // best sortable score that fell off the list, double-buffered like s_posv
    __shared__ int s_posv[2];
    // fp32 sketch: P q, ||q_perp||, ||q|| (sketch_prepare) and the count of a hop's candidates the bound did not drop. The survivors'
    // ids go to the idle list buffer `nxt` (written only by the merge; launch_search checks that it holds a whole hop), and
    // sketch_prepare's scratch to cand_keys (idle before the walk): 9 CTAs per SM leave no room for more static shared memory.
    __shared__ __align__(16) float s_sk[KIND == KIND_F32 ? SKETCH_K + 4 : 4];
    __shared__ int s_ns;

    const int tid = threadIdx.x;
    const int group = tid / G, lane = tid % G;
    const int L = P.rerankK, LC = P.list_cap;
    const unsigned vmask = (unsigned)P.visited_cap - 1u;
    const int vis_limit = 3 << (P.vis_slots_log > 2 ? P.vis_slots_log - 2 : 0);  // shared-memory table: at most 3/4 full
    int32_t *table = P.visited_tables + (size_t)blockIdx.x * P.visited_cap;
    const int degree = P.g.degree;

    for (;;) {
        if (tid == 0) {
            const int w = atomicAdd(P.work_counter, 1);
            if (P.arrived && w < P.nq) {
                // the batch is still being copied in (api.cu jv_graph_search_batch_ex): wait until the watermark has passed this query
                const int need = P.query_index ? P.query_index[w] : w;
                // (bounded: ~10 s of waiting for a copy that takes milliseconds means the copy stream died — trap, never hang the GPU)
                unsigned spins = 0;
                while (*reinterpret_cast<const volatile int *>(P.arrived) <= need) {
                    __nanosleep(200);
                    if (++spins > 50000000u) __trap();
                }
            }
            s_q = w;
        }
        __syncthreads();
        const int wq = s_q;
        if (wq >= P.nq) break;
        const int qi = P.query_index ? P.query_index[wq] : wq;
        const float *q = P.queries + (size_t)qi * P.query_stride;
        const uint32_t *acc = P.accept_bits ? P.accept_bits + (size_t)qi * P.accept_stride : nullptr;
#ifdef JV_SEARCH_PROFILE
        unsigned long long dbg_local[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#endif
        JV_T(t_q0);
        prepare_blob(P.approx, P.metric, q, blobA, red, blobH, splitm);
        if (KIND == KIND_F32 && P.sketch) sketch_prepare(P.sk, P.approx.stride, blobA, s_sk, reinterpret_cast<double *>(cand_keys));
        if (P.has_rerank) prepare_blob(P.rerank, P.metric, q, blobR, red);
        if (vsm) {
            int4 *t4 = reinterpret_cast<int4 *>(vis);
            const int4 z = make_int4(0, 0, 0, 0);
            for (int i = tid; i < (1 << (P.vis_slots_log - 3)); i += SEARCH_THREADS) t4[i] = z;
            if (tid == 0) s_vfail = 0;
        } else {
            int4 *t4 = reinterpret_cast<int4 *>(table);
            const int4 m1 = make_int4(-1, -1, -1, -1);
            for (int i = tid; i < (P.visited_cap >> 2); i += SEARCH_THREADS) t4[i] = m1;
        }
        __syncthreads();
        JV_T(t_q1);
        JV_ACC(0, t_q0, t_q1);

        long long *cur = keys0, *nxt = keys1;
        uint8_t *fcur = flags0, *fnxt = flags1;
        // initializeInternal: score the entry node, mark it visited (GraphSearcher.java:346-348)
        if (group == 0) {
            const float sc = KIND == KIND_PQ ? score_pq<METRIC>(P.approx, blobA, P.g.entry_node, lane, blobH, splitm) : score_row<KIND, METRIC>(P.approx, blobA, P.g.entry_node, lane);
            if (lane == 0) {
                const int32_t en = P.g.entry_node;
                cur[0] = topk_key(sc, en);
                fcur[0] = ((!acc || ((acc[en >> 5] >> (en & 31)) & 1u)) && sc >= P.threshold) ? F_ACCEPTED : 0;
                if (vsm) visited_insert_smem(vis, P.vis_idmask, P.vis_rlog, en, &s_vfail);
                else visited_insert(table, vmask, P.visited_shift, en);
            }
        }
        int size = 1;
        int table_cnt = 1;
        unsigned visited = 0, expanded = 0, expanded_base = 0, rows_read = 0;
        int failed = 0;  // 1: visited table full, 2: candidate list too short for a tie tail
        bool truncated = false, inexact = false;  // lenient mode: the walk was cut short / a tie tail was dropped
        __syncthreads();

        for (int lvl = P.g.entry_level; lvl >= 0 && !failed && !truncated; --lvl) {
            const int K = lvl > 0 ? 1 : L;
            // a new level: results + evicted are candidates again (setEntryPointsFromPreviousLayer), the result heap is empty
            for (int i = tid; i < size; i += SEARCH_THREADS) fcur[i] &= F_ACCEPTED;
            int sel = 0;
            if (tid == 0) { s_posv[0] = 0; s_posv[1] = INT_MAX; s_n = 0; s_m = 0; s_hsize = 0; s_drop[0] = INT_MIN; s_drop[1] = INT_MIN; s_cnt = 0; s_ns = 0; }
            __syncthreads();
            for (;;) {
                const int p = s_posv[sel];  // first unexpanded entry = the top of the candidate queue
                if (p == INT_MAX) break;    // candidates.size() == 0
                JV_T(t_i0);
                const long long ckey = cur[p];
                const int hs = s_hsize;
                const float csc = key_score(ckey);
                const float wsc = hs > 0 ? key_score(heap[1]) : 0.f;
                if (hs >= K && csc < wsc) break;  // stopSearch (strict <: a tie with the worst result is still expanded)
                const int node = key_node(ckey);
                // addTopCandidate: 1 push, 2 replace the worst, 3 tie with the worst: not added, 0 not acceptable (level 0 only)
                int action = 0;
                if (lvl > 0 || (fcur[p] & F_ACCEPTED)) action = hs < K ? 1 : (csc > wsc ? 2 : 3);
                const int dead = (lvl > 0 && action == 3) ? p : -1;
                // a full list at level 0: a candidate can only enter it by beating the last entry, which the sketch bound tests first
                const bool skh = KIND == KIND_F32 && P.sketch && lvl == 0 && size == LC;
                if (tid == 0) { fcur[p] |= F_EXPANDED; s_posv[sel ^ 1] = INT_MAX; s_m = 0; }
                expanded++;
                if (lvl == 0) expanded_base++;
                const int32_t *nb;
                if (lvl == 0) nb = P.g.adj0 + (size_t)node * degree;
                else {
                    const int32_t row = P.g.upper_row[(size_t)(lvl - 1) * P.g.n + node];
                    nb = row >= 0 ? P.g.upper_adj + ((size_t)P.g.upper_off[lvl - 1] + row) * degree : nullptr;
                }
                // FusedPQ (OnDiskGraphIndex.java:639-651, "useEdgeLoading && level == 0"): ids and the neighbours' codes come from the
                // expanded node's own record
                const bool fused = KIND == KIND_PQ && lvl == 0 && P.g.fused != nullptr;
                const uint8_t *rec = fused ? P.g.fused + (size_t)node * P.g.fused_rec : nullptr;
                if (fused) {
                    nb = reinterpret_cast<const int32_t *>(rec);
                    if (P.pq_rows) {
                        // the record's code rows do not depend on which neighbours turn out to be new: the warps that have no
                        // neighbour to test copy ALL of them (degree x code_stride contiguous bytes) into shared memory while
                        // warp 0 runs visited.add(); the scoring phase then finds candidate i's codes at slot cand_slot[i]
                        const int cw = P.approx.code_stride >> 2, cws = cw + 1;
                        const uint32_t *src = reinterpret_cast<const uint32_t *>(rec + 4 * degree);
                        for (int t = tid - 64; t >= 0 && t < degree * cw; t += SEARCH_THREADS - 64) {
                            const int i = t / cw;
                            pq_stage[i * cws + (t - i * cw)] = __ldg(src + t);
                        }
                    } else if (tid >= 64) {
                        // the code rows of this record are needed one barrier from now: pull the whole record towards L2 at once
                        const int o = (tid - 64) * 128;
                        if (o < P.g.fused_rec) prefetch_l2(rec + o);
                    }
                }
                // processNeighbors: score a neighbour only if visited.add() says it is new (OnHeapGraphIndex.java:478)
                if (nb)
                    for (int t = tid; t < degree; t += SEARCH_THREADS) {
                        const int32_t f = __ldg(nb + t);
                        if (f >= 0 && (vsm ? visited_insert_smem(vis, P.vis_idmask, P.vis_rlog, f, &s_vfail) : visited_insert(table, vmask, P.visited_shift, f))) {
                            const int slot = atomicAdd(&s_n, 1);
                            cand_ids[slot] = f;
                            if (KIND == KIND_PQ) cand_slot[slot] = (uint8_t)t;
                            // the row is needed one barrier from now: start the DRAM -> L2 transfer of all of it at once (one
                            // UBLKPF per row; bytes in flight that occupy no registers and no shared memory)
                            if (KIND == KIND_F32 && skh) {
                                // the bound needs the 128-byte sketch line and the norms; the row only if the candidate survives
                                prefetch_l2(P.sk.proj + (size_t)f * (SKETCH_K / 4));
                                prefetch_l2(P.sk.norms + f);
                            } else if (KIND == KIND_F32 && P.row_prefetch == 1) bulk_prefetch_l2(P.approx.rows + (size_t)f * P.approx.stride, (unsigned)P.approx.stride * 4u);
                            if (KIND == KIND_NVQ && P.row_prefetch == 1) {
                                bulk_prefetch_l2(P.approx.bytes + (size_t)f * P.approx.byte_stride, (unsigned)P.approx.byte_stride);
                                prefetch_l2(P.approx.params + (size_t)f * 4 * P.approx.nsub);  // {min, max, growthRate, midpoint} per sub-vector
                            }
                        }
                    }
                // Speculation by the otherwise idle warps (PQ / BQ only: their traversal is a latency chain and HBM is idle, while
                // the fp32 / NVQ paths are bandwidth-bound and must not waste it): the entries right behind p are the likeliest to
                // be expanded next, so touch their adjacency rows and prefetch their neighbours' code rows into L2.
                // Reads only; results unchanged.
                if (lvl == 0 && (KIND == KIND_F32 || KIND == KIND_NVQ)) {
                    // bandwidth-bound kinds speculate on the ADJACENCY rows only (128 B each, nothing next to the 3 KB rows): the next
                    // pops are most likely the unexpanded entries right behind p, and their rows then come from L2 instead of DRAM
                    if (tid >= 32 && tid < 36) {
                        const int pp = p + (tid - 31);
                        if (pp < size && !(fcur[pp] & F_EXPANDED)) prefetch_l2(P.g.adj0 + (size_t)key_node(cur[pp]) * degree);
                    }
                }
                if (lvl == 0 && P.early_pf && tid == 36) {
                    // the next pop is the best of {unexpanded old entries, this hop's new candidates}: a new candidate that beats the
                    // SECOND unexpanded old entry is among the next two pops, so its adjacency (or FusedPQ record) is requested the
                    // moment its score is known (JV_EMIT) instead of after the merge
                    int found = 0;
                    const int end = min(size, p + 17);
                    long long nk = end > p + 1 ? cur[end - 1] : KEY_MIN;
                    for (int i = p + 1; i < end; i++)
                        if (!(fcur[i] & F_EXPANDED) && ++found == 2) { nk = cur[i]; break; }
                    if (found < 2 && end == size) nk = KEY_MIN;
                    s_nk = nk;
                }
                if (lvl == 0 && (KIND == KIND_PQ || KIND == KIND_BQ)) {
                    const int w = tid >> 5;
                    if (w >= 1 && w <= 3) {
                        const int pp = p + w;
                        if (pp < size && !(fcur[pp] & F_EXPANDED) && KIND == KIND_PQ && P.g.fused) {
                            // one record = ids + codes: pull its lines towards L2 (25 x 128 B at degree 32, M = 96)
                            const char *r2 = reinterpret_cast<const char *>(P.g.fused + (size_t)key_node(cur[pp]) * P.g.fused_rec);
                            for (int o = (tid & 31) * 128; o < P.g.fused_rec; o += 32 * 128) prefetch_l2(r2 + o);
                        } else if (pp < size && !(fcur[pp] & F_EXPANDED)) {
                            const int32_t *nb2 = P.g.adj0 + (size_t)key_node(cur[pp]) * degree;
                            for (int t = tid & 31; t < degree; t += 32) {
                                const int32_t f = __ldg(nb2 + t);
                                if (KIND == KIND_PQ && f >= 0) {
                                    const char *a = reinterpret_cast<const char *>(P.approx.codes + (size_t)f * P.approx.code_stride);
                                    prefetch_l2(a);
                                    prefetch_l2(a + P.approx.M - 1);
                                } else if (KIND == KIND_BQ && f >= 0) {
                                    const char *a = reinterpret_cast<const char *>(P.approx.words + (size_t)f * P.approx.W);
                                    for (int o = 0; o < P.approx.W * 8; o += 128) prefetch_l2(a + o);
                                    prefetch_l2(a + P.approx.W * 8 - 1);
                                }
                            }
                        }
                    }
                }
                __syncthreads();
                JV_T(t_i1);
                JV_ACC(1, t_i0, t_i1);
                // every thread has read the heap top by now: apply addTopCandidate to the result heap
                if (tid == HEAP_TID) {
                    if (action == 1) {
                        heap[hs + 1] = ckey;
                        heap_up(heap, hs + 1);
                        s_hsize = hs + 1;
                    } else if (action == 2) {
                        heap[1] = ckey;
                        heap_down(heap, hs, 1);
                    }
                }
                if (tid == 0) { s_drop[sel ^ 1] = INT_MIN; s_cnt = 0; }
                const int n = s_n;
                table_cnt += n;
                if (vsm ? (table_cnt > vis_limit || s_vfail) : (table_cnt * 2 > P.visited_cap)) {
                    if (P.lenient) truncated = true;
                    else failed = 1;
                    break;
                }
                // A candidate that scores under the last entry of a FULL list is dropped by the merge whatever the other candidates do, so
                // it is dropped here and the merge only ranks the survivors (late in a walk that is most of them).
                // (the list's last key is re-read from shared memory by the one lane that needs it: nothing extra lives in registers
                // across the scoring loop)
#define JV_EMIT(sc_, f_)                                                                                                            \
    do {                                                                                                                            \
        const long long key_ = topk_key((sc_), (f_));                                                                               \
        if (lvl == 0 && P.early_pf && key_ > s_nk) {                                                                                \
            if (KIND == KIND_PQ && P.g.fused) bulk_prefetch_l2(P.g.fused + (size_t)(f_) * P.g.fused_rec, (unsigned)P.g.fused_rec);  \
            else prefetch_l2(P.g.adj0 + (size_t)(f_) * degree);                                                                     \
        }                                                                                                                           \
        if (dead < 0 && size == LC && key_ < cur[LC - 1]) atomicMax(&s_drop[sel], float_to_sortable(sc_));                          \
        else {                                                                                                                      \
            const int m_ = atomicAdd(&s_m, 1);                                                                                      \
            cand_keys[m_] = key_;                                                                                                   \
            if (P.filtered) cand_acc[m_] = ((!acc || ((acc[(f_) >> 5] >> ((f_) & 31)) & 1u)) && (sc_) >= P.threshold) ? F_ACCEPTED : 0; \
        }                                                                                                                           \
    } while (0)
                if (KIND == KIND_F32) {
                    const int32_t *ids = cand_ids;
                    int ns = n;
                    if (skh) {
                        // bound pass: 8 lanes per candidate, one 16-byte piece of its sketch line each. A candidate whose bound is under
                        // the last entry is dropped here exactly as JV_EMIT would drop it after reading the row; the bound, not the
                        // unread exact score, goes into s_drop (>= the exact score, so the exactness test below stays sound). The rows
                        // of the survivors are requested at once and scored by the unchanged loop below.
                        const float tail = key_score(cur[LC - 1]);
                        const int sl = tid & 7;
                        int32_t *surv = reinterpret_cast<int32_t *>(nxt);
                        for (int i = tid >> 3; i < n; i += SEARCH_THREADS / 8) {
                            const int32_t f = cand_ids[i];
                            const float4 u = __ldg(P.sk.proj + (size_t)f * (SKETCH_K / 4) + sl);
                            const float4 a = reinterpret_cast<const float4 *>(s_sk)[sl];
                            const float d = group_sum<8>(fmaf(a.x, u.x, fmaf(a.y, u.y, fmaf(a.z, u.z, __fmul_rn(a.w, u.w)))));
                            if (sl == 0) {
                                const float2 nm = __ldg(P.sk.norms + f);
                                const float ub = score_map(METRIC, d + s_sk[SKETCH_K] * nm.x + SKETCH_MARGIN * s_sk[SKETCH_K + 1] * nm.y);
                                if (ub < tail) atomicMax(&s_drop[sel], float_to_sortable(ub));
                                else {
                                    surv[atomicAdd(&s_ns, 1)] = f;
                                    bulk_prefetch_l2(P.approx.rows + (size_t)f * P.approx.stride, (unsigned)P.approx.stride * 4u);
                                }
                            }
                        }
                        __syncthreads();
                        ids = surv;
                        ns = s_ns;
                    }
                    rows_read += ns;
                    // two rows per warp at a time: twice the loads in flight, query fragment read once
                    for (int i = group; i < ns; i += 2 * NG) {
                        const int32_t fa = ids[i];
                        const bool two = i + NG < ns;
                        const int32_t fb = two ? ids[i + NG] : fa;
                        float sa, sb;
                        score_f32_pair<METRIC>(P.approx, blobA, fa, fb, lane, sa, sb);
                        if (lane == 0) {
                            JV_EMIT(sa, fa);
                            if (two) JV_EMIT(sb, fb);
                        }
                    }
                } else if (KIND == KIND_PQ && P.pq_rows) {
                    // lane = candidate, warp = one of the 8 partial sums of the ADC score (score_pq_partial): the code rows of the
                    // hop are staged in shared memory by one coalesced pass, then every gather instruction of a warp reads ONE LUT row
                    const int cw = P.approx.code_stride >> 2, cws = cw + 1;  // odd word stride: no bank conflicts across candidates
                    if (!fused) {
                        for (int t = tid; t < n * cw; t += SEARCH_THREADS) {
                            const int i = t / cw, wd = t - i * cw;
                            pq_stage[i * cws + wd] = __ldg(reinterpret_cast<const uint32_t *>(P.approx.codes + (size_t)cand_ids[i] * P.approx.code_stride) + wd);
                        }
                        __syncthreads();
                    }
                    const int pstride = (degree + 31) & ~31;
                    for (int g = tid >> 5; g < 8; g += SEARCH_THREADS / 32)
                        for (int i = tid & 31; i < n; i += 32) {
                            float ps, pa;
                            score_pq_partial<METRIC>(P.approx, blobA, blobH, splitm, reinterpret_cast<const uint8_t *>(pq_stage + (fused ? (int)cand_slot[i] : i) * cws), g, ps, pa);
                            pq_part[g * pstride + i] = ps;
                            if (METRIC == JV_METRIC_COSINE) pq_part[(8 + g) * pstride + i] = pa;
                        }
                    __syncthreads();
                    for (int i = tid; i < n; i += SEARCH_THREADS) {
                        float sraw = pq_fold8(pq_part + i, pstride);
                        if (METRIC == JV_METRIC_COSINE)
                            sraw = __fdiv_rn(sraw, __fsqrt_rn(__fmul_rn(pq_fold8(pq_part + 8 * pstride + i, pstride), blobH[P.approx.M * P.approx.k])));
                        const float sc = score_map(METRIC, sraw);
                        const int32_t f = cand_ids[i];
                        JV_EMIT(sc, f);
                    }
                } else if (KIND == KIND_PQ && fused) {
                    // FusedPQDecoder.similarityToNeighbor (FusedPQDecoder.java:107-114): the code row sits inside the record just read
                    const uint8_t *codes0 = rec + 4 * degree;
                    for (int i = group; i < n; i += NG) {
                        const int32_t f = cand_ids[i];
                        const float sc = score_pq_codes<METRIC>(P.approx, blobA, codes0 + (size_t)cand_slot[i] * P.g.fused_code_stride, lane, blobH, splitm);
                        if (lane == 0) JV_EMIT(sc, f);
                    }
                } else {
                    for (int i = group; i < n; i += NG) {
                        const int32_t f = cand_ids[i];
                        const float sc = KIND == KIND_PQ ? score_pq<METRIC>(P.approx, blobA, f, lane, blobH, splitm) : score_row<KIND, METRIC>(P.approx, blobA, f, lane);
                        if (lane == 0) JV_EMIT(sc, f);
                    }
                }
#undef JV_EMIT
                __syncthreads();
                JV_T(t_i2);
                JV_ACC(2, t_i1, t_i2);
                visited += n;
                const int nm = s_m;  // candidates that survived the pre-filter
                // rank-merge (old list is sorted; candidates are few): every element computes its slot directly and the
                // first unexpanded slot of the next list falls out of the same pass. The entry at `dead` (refused on an
                // upper level) leaves the list.
                const int live = size - (dead >= 0 ? 1 : 0);
                const int newsize = min(LC, live + nm);
                const long long dead_key = dead >= 0 ? cur[dead] : KEY_MIN;
                int mypos = INT_MAX, mydrop = INT_MIN;
                // one work item per thread: items [0, size) are old entries, [size, size + n) the new candidates, so the
                // two kinds run on different warps instead of back to back on warp 0
                for (int it = tid; it < size + nm; it += SEARCH_THREADS) {
                    if (it < size) {
                        if (it == dead) continue;
                        const long long k = cur[it];
                        int c = 0;
#pragma unroll 8
                        for (int j = 0; j < nm; j++) c += (cand_keys[j] > k);
                        const int np = it + c - ((dead >= 0 && it > dead) ? 1 : 0);
                        const uint8_t fl = fcur[it];
                        if (np < LC) {
                            nxt[np] = k;
                            fnxt[np] = fl;
                            if (!(fl & F_EXPANDED)) mypos = min(mypos, np);
                        } else if (!(fl & F_EXPANDED) || lvl > 0) mydrop = max(mydrop, float_to_sortable(key_score(k)));
                    } else {
                        const long long k = cand_keys[it - size];
                        int c = count_greater_desc(cur, size, k) - ((dead >= 0 && dead_key > k) ? 1 : 0);
#pragma unroll 8
                        for (int jj = 0; jj < nm; jj++) c += (cand_keys[jj] > k);
                        if (c < LC) {
                            nxt[c] = k;
                            fnxt[c] = P.filtered ? cand_acc[it - size] : F_ACCEPTED;
                            mypos = min(mypos, c);
                            // a new candidate that lands at the very front is the likeliest next expansion: start pulling
                            // its adjacency row towards L2 now (128 B; reads only)
                            if (c < 2 && lvl == 0) {
                                if (KIND == KIND_PQ && P.g.fused) prefetch_l2(P.g.fused + (size_t)key_node(k) * P.g.fused_rec);
                                else prefetch_l2(P.g.adj0 + (size_t)key_node(k) * degree);
                            }
                        } else mydrop = max(mydrop, float_to_sortable(key_score(k)));
                    }
                }
                if (mypos != INT_MAX) atomicMin(&s_posv[sel ^ 1], mypos);
                if (mydrop != INT_MIN) atomicMax(&s_drop[sel], mydrop);
                if (tid == 0) { s_n = 0; s_ns = 0; }
                __syncthreads();
                JV_T(t_i3);
                JV_ACC(3, t_i2, t_i3);
#ifdef JV_SEARCH_PROFILE
                if (tid == 0) { dbg_local[5] += 1; dbg_local[6] += (unsigned long long)n; }
#endif
                // something fell off the end of the list: that is exact only if at least rerankK accepted entries score strictly
                // higher than everything dropped (then none of it can be popped before stopSearch fires). For a candidate the sketch
                // dropped unread, dm holds its bound: the test may fail where the exact score would have passed, never the reverse.
                const int dm = s_drop[sel];
                if (dm != INT_MIN) {
                    bool ok;
                    if (!P.filtered) ok = float_to_sortable(key_score(nxt[L - 1])) > dm;  // newsize == LC >= L here
                    else {
                        int c = 0;
                        for (int i = tid; i < newsize; i += SEARCH_THREADS)
                            c += ((fnxt[i] & F_ACCEPTED) && float_to_sortable(key_score(nxt[i])) > dm) ? 1 : 0;
                        if (c) atomicAdd(&s_cnt, c);
                        __syncthreads();
                        ok = s_cnt >= L;
                    }
                    if (!ok) {
                        if (P.lenient) inexact = true;  // keep walking: only the exactness of tie handling is lost
                        else { failed = 2; break; }
                    }
                }
                { long long *t = cur; cur = nxt; nxt = t; }
                { uint8_t *t = fcur; fcur = fnxt; fnxt = t; }
                size = newsize;
                sel ^= 1;
            }
            __syncthreads();
        }

        JV_T(t_r0);
        int32_t *no = P.nodes_out + (size_t)qi * P.topK;
        float *so = P.scores_out + (size_t)qi * P.topK;
        unsigned reranked = 0;
        if (failed) {
            for (int i = tid; i < P.topK; i += SEARCH_THREADS) { no[i] = -1; so[i] = 0.f; }
            if (tid == 0) { P.overflow[qi] = (uint8_t)failed; atomicAdd(&P.counters->overflowed, 1ull); }
        } else {
            if (tid == 0) {
                P.overflow[qi] = 0;
                if (truncated || inexact) atomicAdd(&P.counters->overflowed, 1ull);
            }
            const int hs = s_hsize;  // the results: heap[1 .. hs]
            if (P.has_rerank) {
                // NodeQueue.rerank (NodeQueue.java:168-230): rescore, in HEAP-ARRAY order, the results whose approximate score
                // is >= rerankFloor (or the single best one if none is), keep the topK best exact scores; on an exact-score
                // tie at the topK boundary the entry met first in array order stays.
                constexpr int NGR = SEARCH_THREADS / 32;
                const int wgroup = tid >> 5, wlane = tid & 31;
                if (tid == 0) s_cnt = 0;
                __syncthreads();
                {
                    int c = 0;
                    for (int i = tid; i < hs; i += SEARCH_THREADS) {
                        const bool above = key_score(heap[1 + i]) >= P.rerank_floor;
                        fcur[i] = above ? 1 : 0;
                        c += above ? 1 : 0;
                    }
                    if (c) atomicAdd(&s_cnt, c);
                }
                __syncthreads();
                int nrr = s_cnt;
                if (nrr == 0 && hs > 0) {
                    // nothing above the floor: the best approximate score is reranked alone (first maximum in array order)
                    if (tid == 0) {
                        int bi = 0;
                        float bs = key_score(heap[1]);
                        for (int i = 1; i < hs; i++) {
                            const float s = key_score(heap[1 + i]);
                            if (s > bs) { bs = s; bi = i; }
                        }
                        fcur[bi] = 1;
                    }
                    nrr = 1;
                    __syncthreads();
                }
                if (KIND == KIND_PQ || KIND == KIND_BQ) {
                    // the approximate walk left HBM idle: pull every survivor's exact row towards L2 before the rescoring loop
                    const int lines = P.rerank.kind == KIND_F32 ? (P.rerank.stride * 4 + 127) / 128 : (P.rerank.byte_stride + 127) / 128;
                    for (int t = tid; t < hs * lines; t += SEARCH_THREADS) {
                        const int i = t / lines, l = t - i * lines;
                        if (!fcur[i]) continue;
                        const int32_t f = key_node(heap[1 + i]);
                        const char *a = P.rerank.kind == KIND_F32 ? reinterpret_cast<const char *>(P.rerank.rows + (size_t)f * P.rerank.stride)
                                                                  : reinterpret_cast<const char *>(P.rerank.bytes + (size_t)f * P.rerank.byte_stride);
                        prefetch_l2(a + (size_t)l * 128);
                    }
                }
                // exact keys in array order -> cur[0 .. hs) (KEY_MIN = not reranked)
                if (P.rerank.kind == KIND_F32) {
                    for (int i = wgroup; i < hs; i += 2 * NGR) {
                        const int32_t fa = key_node(heap[1 + i]);
                        const bool two = i + NGR < hs;
                        const int32_t fb = two ? key_node(heap[1 + i + NGR]) : fa;
                        const bool da = fcur[i] != 0, db = two && fcur[i + NGR] != 0;
                        float sa = 0.f, sb = 0.f;
                        if (da || db) score_f32_pair<METRIC>(P.rerank, blobR, da ? fa : fb, db ? fb : fa, wlane, sa, sb);
                        if (wlane == 0) {
                            cur[i] = da ? topk_key(sa, fa) : KEY_MIN;
                            if (two) cur[i + NGR] = db ? topk_key(sb, fb) : KEY_MIN;
                        }
                    }
                } else {
                    for (int i = wgroup; i < hs; i += NGR) {
                        const int32_t f = key_node(heap[1 + i]);
                        float sc = 0.f;
                        const bool d = fcur[i] != 0;
                        if (d) sc = score_row<KIND_NVQ, METRIC>(P.rerank, blobR, f, wlane);
                        if (wlane == 0) cur[i] = d ? topk_key(sc, f) : KEY_MIN;
                    }
                }
                __syncthreads();
                for (int i = tid; i < P.sort_pow2; i += SEARCH_THREADS) nxt[i] = i < hs ? cur[i] : KEY_MIN;
                __syncthreads();
                bitonic_sort_desc_block(nxt, P.sort_pow2);
                reranked = (unsigned)nrr;
                const bool boundary_tie = nrr > P.topK && key_score(nxt[P.topK - 1]) == key_score(nxt[P.topK]);
                if (!boundary_tie) {
                    for (int i = tid; i < P.topK; i += SEARCH_THREADS) {
                        if (i < nrr) { no[i] = key_node(nxt[i]); so[i] = key_score(nxt[i]); }
                        else { no[i] = -1; so[i] = 0.f; }
                    }
                } else if (tid == 0) {
                    // replay the reference loop (NodeQueue.java:199-215) over the array order; `heap` is free to be reused
                    long long *rh = heap;
                    int rs = 0;
                    for (int i = 0; i < hs; i++) {
                        const long long v = cur[i];
                        if (v == KEY_MIN) continue;
                        if (rs < P.topK) { rh[++rs] = v; heap_up(rh, rs); }
                        else if (key_score(v) > key_score(rh[1])) { rh[1] = v; heap_down(rh, rs, 1); }
                    }
                    for (int i = rs - 1; i >= 0; i--) {  // pop: worst first
                        const long long v = rh[1];
                        rh[1] = rh[rs--];
                        if (rs > 0) heap_down(rh, rs, 1);
                        no[i] = key_node(v);
                        so[i] = key_score(v);
                    }
                }
            } else {
                // no reranker: the best topK of the results by approximate key (GraphSearcher.java:478-486, :494-500)
                for (int i = tid; i < P.sort_pow2; i += SEARCH_THREADS) nxt[i] = i < hs ? heap[1 + i] : KEY_MIN;
                __syncthreads();
                bitonic_sort_desc_block(nxt, P.sort_pow2);
                for (int i = tid; i < P.topK; i += SEARCH_THREADS) {
                    if (i < hs) { no[i] = key_node(nxt[i]); so[i] = key_score(nxt[i]); }
                    else { no[i] = -1; so[i] = 0.f; }
                }
            }
            if (tid == 0) {
                atomicAdd(&P.counters->visited, (unsigned long long)visited);
                atomicAdd(&P.counters->expanded, (unsigned long long)expanded);
                atomicAdd(&P.counters->expanded_base, (unsigned long long)expanded_base);
                atomicAdd(&P.counters->reranked, (unsigned long long)reranked);
                if (KIND == KIND_F32) atomicAdd(&P.counters->rows_read, (unsigned long long)rows_read);
            }
        }
        __syncthreads();
#ifdef JV_SEARCH_PROFILE
        {
            JV_T(t_r1);
            JV_ACC(4, t_r0, t_r1);
            JV_ACC(7, t_q0, t_r1);
            if (tid == 0 && P.dbg)
                for (int i = 0; i < 8; i++) atomicAdd(&P.dbg[i], dbg_local[i]);
        }
#endif
    }
}

static int next_pow2i(int v)
{
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

// shared-memory floats of the walking scorer's prepared query: everything, except for a PQ LUT of which only the rows of the
// first pq_smem_m sub-spaces stay in shared memory
static int search_smemA_floats(const DataDesc &approx, int pq_smem_m)
{
    if (approx.kind != KIND_PQ || pq_smem_m >= approx.M) return blob_floats(approx);
    return (pq_smem_m * approx.k + 3) & ~3;
}

static size_t search_smem_bytes(const DataDesc &approx, const DataDesc *rerank, int rerankK, int list_alloc, int pq_smem_m, int vis_slots_log = 0, int pq_rows_degree = 0)
{
    size_t b = (size_t)search_smemA_floats(approx, pq_smem_m) * 4;
    if (rerank) b += (size_t)blob_floats(*rerank) * 4;
    b += (size_t)list_alloc * 8 * 2;                  // the two list buffers
    b += (size_t)MAX_DEGREE * 8;                      // candidate keys of one hop
    b += (size_t)((rerankK + 2) & ~1) * 8;            // result heap (1-based)
    b += (size_t)MAX_DEGREE * 4 + (size_t)MAX_DEGREE * 2; // candidate ids + accept flags + record slots
    b += (size_t)list_alloc * 2;                      // entry flags of the two buffers
    b = (b + 15) & ~(size_t)15;
    if (vis_slots_log) b += (size_t)2 << vis_slots_log;  // visited set, 16 bits per slot
    if (pq_rows_degree) b += (size_t)pq_rows_degree * ((approx.code_stride >> 2) + 1) * 4 + (size_t)16 * ((pq_rows_degree + 31) & ~31) * 4;  // staged codes + partial sums
    return (b + 15) & ~(size_t)15;
}

#ifndef JV_VISITED_SMEM_DEFAULT
#define JV_VISITED_SMEM_DEFAULT true
#endif
#ifndef JV_PQ_ROWS_DEFAULT
#define JV_PQ_ROWS_DEFAULT 1
#endif
#ifndef JV_SEARCH_MINB_PQ_WIDE
#define JV_SEARCH_MINB_PQ_WIDE 4
#endif
#ifndef JV_ROW_PREFETCH_DEFAULT
#define JV_ROW_PREFETCH_DEFAULT 1
#endif
#ifndef JV_SEARCH_MINB_ROWS
#define JV_SEARCH_MINB_ROWS 9
#endif
#ifndef JV_SEARCH_MINB_ROWS_WIDE
#define JV_SEARCH_MINB_ROWS_WIDE 8
#endif
constexpr int MINB_DEFAULT = JV_SEARCH_MINB, MINB_PQ_LITE = JV_SEARCH_MINB_PQ, MINB_PQ_WIDE = JV_SEARCH_MINB_PQ_WIDE;
constexpr int MINB_ROWS = JV_SEARCH_MINB_ROWS, MINB_ROWS_WIDE = JV_SEARCH_MINB_ROWS_WIDE;  // fp32 / NVQ walks (56 registers at 128 threads, 9 CTAs per SM. c2, burst: 9 x 56 registers 14.24 ms, 8 x 64 registers 13.84 ms; sustained under the 1000 W cap — what bench.py times — 14.2 ms vs 14.8 ms: 9 x 56 ships)

template <int KIND, int METRIC, int MINB, bool VSM>
static cudaError_t occupancy_of(size_t smem, int *blocks_per_sm)
{
    cudaError_t e = cudaFuncSetAttribute(graph_search_kernel<KIND, METRIC, MINB, VSM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, graph_search_kernel<KIND, METRIC, MINB, VSM>, SearchThreads<KIND>::value, smem);
}

#define JV_SEARCH_DISPATCH_V(kind, metric, pq_wide, V, CALL)                                                  \
    do {                                                                                        \
        if ((kind) == KIND_F32 && (pq_wide)) {                                                  \
            if ((metric) == JV_METRIC_EUCLIDEAN) { CALL(KIND_F32, JV_METRIC_EUCLIDEAN, MINB_ROWS_WIDE, V); } \
            else if ((metric) == JV_METRIC_DOT) { CALL(KIND_F32, JV_METRIC_DOT, MINB_ROWS_WIDE, V); } \
            else { CALL(KIND_F32, JV_METRIC_COSINE, MINB_ROWS_WIDE, V); }                            \
        } else if ((kind) == KIND_F32) {                                                        \
            if ((metric) == JV_METRIC_EUCLIDEAN) { CALL(KIND_F32, JV_METRIC_EUCLIDEAN, MINB_ROWS, V); }       \
            else if ((metric) == JV_METRIC_DOT) { CALL(KIND_F32, JV_METRIC_DOT, MINB_ROWS, V); }              \
            else { CALL(KIND_F32, JV_METRIC_COSINE, MINB_ROWS, V); }                                          \
        } else if ((kind) == KIND_PQ && (pq_wide)) {                                            \
            if ((metric) == JV_METRIC_EUCLIDEAN) { CALL(KIND_PQ, JV_METRIC_EUCLIDEAN, MINB_PQ_WIDE, V); } \
            else if ((metric) == JV_METRIC_DOT) { CALL(KIND_PQ, JV_METRIC_DOT, MINB_PQ_WIDE, V); } \
            else { CALL(KIND_PQ, JV_METRIC_COSINE, MINB_PQ_WIDE, V); }                             \
        } else if ((kind) == KIND_PQ) {                                                         \
            if ((metric) == JV_METRIC_EUCLIDEAN) { CALL(KIND_PQ, JV_METRIC_EUCLIDEAN, MINB_PQ_LITE, V); } \
            else if ((metric) == JV_METRIC_DOT) { CALL(KIND_PQ, JV_METRIC_DOT, MINB_PQ_LITE, V); } \
            else { CALL(KIND_PQ, JV_METRIC_COSINE, MINB_PQ_LITE, V); }                             \
        } else if ((kind) == KIND_BQ) {                                                         \
            if ((metric) == JV_METRIC_EUCLIDEAN) { CALL(KIND_BQ, JV_METRIC_EUCLIDEAN, MINB_DEFAULT, V); }        \
            else if ((metric) == JV_METRIC_DOT) { CALL(KIND_BQ, JV_METRIC_DOT, MINB_DEFAULT, V); }               \
            else { CALL(KIND_BQ, JV_METRIC_COSINE, MINB_DEFAULT, V); }                                           \
        } else {                                                                                \
            if ((metric) == JV_METRIC_EUCLIDEAN) { CALL(KIND_NVQ, JV_METRIC_EUCLIDEAN, MINB_ROWS, V); }       \
            else if ((metric) == JV_METRIC_DOT) { CALL(KIND_NVQ, JV_METRIC_DOT, MINB_ROWS, V); }              \
            else { CALL(KIND_NVQ, JV_METRIC_COSINE, MINB_ROWS, V); }                                          \
        }                                                                                       \
    } while (0)
#define JV_SEARCH_DISPATCH(kind, metric, pq_wide, vsm, CALL)                    \
    do {                                                                       \
        if (vsm) JV_SEARCH_DISPATCH_V(kind, metric, pq_wide, true, CALL);      \
        else JV_SEARCH_DISPATCH_V(kind, metric, pq_wide, false, CALL);         \
    } while (0)

cudaError_t plan_search(const DataDesc &approx, const DataDesc *rerank, const GraphDesc &g, int topK, int rerankK, int nq,
                        int visited_cap_hint, int list_cap_hint, int sm_count, SearchPlan *plan)
{
    if (g.degree > MAX_DEGREE || rerankK < 1 || topK < 1 || topK > rerankK) return cudaErrorInvalidValue;
    plan->threads = search_threads_of(approx.kind);
    plan->sort_pow2 = next_pow2i(rerankK);
    // The list keeps rerankK entries plus a tie tail (see the kernel header). Continuous scores tie rarely: the slack that
    // rounds rerankK up to a multiple of 32 is enough; BQ scores take at most dim + 1 values, so whole groups tie at the
    // boundary. A query whose tail does not fit reports overflow code 2 and is re-run with list_cap_hint = 4x.
    int cap = list_cap_hint > 0 ? list_cap_hint : (approx.kind == KIND_BQ ? 2 * rerankK + 64 : rerankK + 28);
    if (cap < rerankK) cap = rerankK;
    cap = (cap + 3) & ~3;
    if (cap > MAX_LIST_CAP) cap = MAX_LIST_CAP;
    if (cap < rerankK) return cudaErrorInvalidValue;
    plan->list_cap = cap;
    plan->list_alloc = cap > plan->sort_pow2 ? cap : plan->sort_pow2;
    // PQ: a LUT of M*k fp32 (96 KB at M=96) in shared memory limits residency to 2 CTAs per SM, and the walk is a latency chain
    // (profiles/r1_search_phase_cycles.md). When five LUTs do not fit an SM's shared memory the LUT lives in an L2-resident
    // global slice per CTA instead: residency becomes register-limited (5 CTAs per SM) and the gathers are served by L2.
    // Measured on c3: 19.25 ms -> 13.1 ms per 10 000 queries. JV_PQ_LUT=smem|l2 overrides.
    // Round 2: the LUT may be SPLIT — rows of the first pq_smem_m sub-spaces in shared memory, the rest in the L2 slice — which
    // trades L2 gather traffic against residency continuously (JV_PQ_LUT=smem|l2 or JV_PQ_LUT_SMEM_M=<sub-spaces> override).
    plan->blob_in_global = 0;
    plan->pq_smem_m = approx.kind == KIND_PQ ? approx.M : 0;
    if (approx.kind == KIND_PQ) {
        const char *mode = getenv("JV_PQ_LUT");
        const char *msub = getenv("JV_PQ_LUT_SMEM_M");
        if (msub) plan->pq_smem_m = std::max(0, std::min(approx.M, atoi(msub))) & ~3;
        else if (mode && mode[0] == 'l') plan->pq_smem_m = 0;
        else if (mode && mode[0] == 's') plan->pq_smem_m = approx.M;
        else plan->pq_smem_m = (size_t)blob_floats(approx) * 4 * 5 > 200 * 1024 ? 0 : approx.M;
        plan->blob_in_global = plan->pq_smem_m < approx.M ? 1 : 0;
    }
    plan->blob_floats = blob_floats(approx);
    // PQ scoring layout of a hop: JV_PQ_SCORE=rows (lane = candidate, warp = partial sum) | group (8 lanes per candidate)
    plan->pq_rows = 0;
    if (approx.kind == KIND_PQ) {
        const char *pt = getenv("JV_PQ_SCORE");
        plan->pq_rows = pt ? (pt[0] == 'r') : JV_PQ_ROWS_DEFAULT;
    }
    const int prd = plan->pq_rows ? g.degree : 0;
    plan->smem_bytes = search_smem_bytes(approx, rerank, rerankK, plan->list_alloc, plan->pq_smem_m, 0, prd);
    if (plan->smem_bytes > 227 * 1024 && approx.kind == KIND_PQ && plan->pq_smem_m > 0) {
        plan->pq_smem_m = 0;  // a long list next to a LUT: keep the list in shared memory, move the whole LUT to L2
        plan->blob_in_global = 1;
        plan->smem_bytes = search_smem_bytes(approx, rerank, rerankK, plan->list_alloc, 0, 0, prd);
    }
    if (plan->smem_bytes > 227 * 1024) return cudaErrorInvalidValue;
    int vcap = visited_cap_hint > 0 ? visited_cap_hint : next_pow2i(4 * rerankK * (g.degree > 16 ? g.degree : 16));
    if (vcap < 2048) vcap = 2048;
    if (vcap > (1 << 22)) vcap = 1 << 22;
    plan->visited_cap = next_pow2i(vcap);
    // Visited set in shared memory (16-bit slots, see visited_insert_smem): no L2 round trip per neighbour, no 64 KB table to clear
    // per query, nothing of it in L2. Taken on the first attempt when the table a walk of this effort needs fits 32 KB and every
    // region keeps at least 32 slots; a query that outgrows it (or fills one region) is re-run on the global table
    // (visited_cap_hint > 0).
    // JV_VISITED=global|smem overrides, JV_VISITED_SMEM_SLOTS sets the slot count.
    plan->vis_slots_log = 0;
    plan->vis_rlog = 0;
    plan->vis_idmask = 0;
    {
        const char *vm = getenv("JV_VISITED");
        const char *vs = getenv("JV_VISITED_SMEM_SLOTS");
        int bits = 15;
        while ((1ll << bits) < g.n) bits++;
        int slots = vs ? next_pow2i(atoi(vs)) : plan->visited_cap / 2;
        int slog = 0;
        while ((1 << slog) < slots) slog++;
        // many regions (large n) want more slots each: grow the table up to 32 KB (10M nodes: 512 regions of 32 slots, ~6 expected
        // entries each for a 3 200-node walk)
        while (!vs && slog - (bits - 15) < 7 && slog < 14) slog++;
        const int rlog = slog - (bits - 15);
        const bool want = vm ? vm[0] == 's' : JV_VISITED_SMEM_DEFAULT;
        if (want && visited_cap_hint <= 0 && slog >= 10 && slog <= 14 && rlog >= 5) {
            const size_t sb = search_smem_bytes(approx, rerank, rerankK, plan->list_alloc, plan->pq_smem_m, slog, prd);
            if (sb <= 227 * 1024) {
                plan->vis_slots_log = slog;
                plan->vis_rlog = rlog;
                plan->vis_idmask = (unsigned)((1ull << bits) - 1ull);
                plan->smem_bytes = sb;
            }
        }
    }
    // JV_ROW_PREFETCH=0|1|2: L2 prefetch of the newly visited rows (fp32 / NVQ walks)
    {
        const char *rp = getenv("JV_ROW_PREFETCH");
        plan->row_prefetch = rp ? atoi(rp) : JV_ROW_PREFETCH_DEFAULT;
        if (approx.kind == KIND_NVQ && ((approx.byte_stride & 15) || plan->row_prefetch != 1)) plan->row_prefetch = 0;
        if (approx.kind != KIND_F32 && approx.kind != KIND_NVQ) plan->row_prefetch = 0;
    }
    int bps = 0;
    cudaError_t e = cudaSuccess;
    const int metric_for_occ = JV_METRIC_DOT;
#define CALL(K, M, B, V) e = occupancy_of<K, M, B, V>(plan->smem_bytes, &bps)
    JV_SEARCH_DISPATCH(approx.kind, metric_for_occ, false, plan->vis_slots_log != 0, CALL);
    plan->pq_wide = 0;
    if (e == cudaSuccess && approx.kind == KIND_PQ) {
        // the 64-register build wherever shared memory (not registers) is what limits residency
        int bw = 0;
        const int lite = bps;
        JV_SEARCH_DISPATCH(approx.kind, metric_for_occ, true, plan->vis_slots_log != 0, CALL);
        bw = bps;
        const char *pw = getenv("JV_PQ_WIDE");  // 0 | 1: force the register build (tuning)
        if (e == cudaSuccess && (pw ? pw[0] == '1' : bw >= lite)) plan->pq_wide = 1;
        else bps = lite;
    }
    if (e == cudaSuccess && approx.kind == KIND_F32) {
        // JV_SEARCH_WIDE=1: the 64-register build of the fp32 walk (4 resident CTAs per SM instead of 5, no spills) — a tuning knob
        const char *w = getenv("JV_SEARCH_WIDE");
        if (w && w[0] == '1') {
            plan->pq_wide = 1;
            JV_SEARCH_DISPATCH(approx.kind, metric_for_occ, true, plan->vis_slots_log != 0, CALL);
        }
    }
#undef CALL
    if (e != cudaSuccess) return e;
    if (bps < 1) return cudaErrorInvalidValue;
    long long ctas = (long long)bps * sm_count;
    if (ctas > nq) ctas = nq;
    if (ctas < 1) ctas = 1;
    plan->ctas = (int)ctas;
    return cudaSuccess;
}

size_t search_scratch_bytes(const SearchPlan &p)
{
    size_t b = p.vis_slots_log ? 256 : (size_t)p.ctas * p.visited_cap * sizeof(int32_t);
    if (p.blob_in_global) b += (size_t)p.ctas * p.blob_floats * sizeof(float) + 256;
    return b;
}

cudaError_t launch_search(const GraphDesc &g, const DataDesc &approx, const DataDesc *rerank, int metric, const float *queries_dev,
                          int nq, int topK, int rerankK, const SearchPlan &plan, void *scratch_dev, int *work_counter_dev,
                          int32_t *nodes_out_dev, float *scores_out_dev, SearchCounters *counters_dev, uint8_t *overflow_flags_dev,
                          const int32_t *query_index_dev, int query_stride, const SearchFilter *filter, cudaStream_t s,
                          const F32Sketch *sketch)
{
    if (nq <= 0) return cudaSuccess;
    SearchParams P;
    // (the survivors of a hop, up to `degree` ids, are staged in one idle list buffer of list_alloc 64-bit entries)
    P.sketch = (sketch && approx.kind == KIND_F32 && metric == JV_METRIC_DOT && 2 * plan.list_alloc >= g.degree) ? 1 : 0;
    P.sk = P.sketch ? *sketch : F32Sketch{};
    P.accept_bits = filter ? filter->accept_bits : nullptr;
    P.accept_stride = filter ? filter->accept_stride_words : 0;
    P.threshold = filter ? filter->threshold : 0.f;
    P.rerank_floor = filter ? filter->rerank_floor : 0.f;
    P.filtered = (P.accept_bits != nullptr || P.threshold > 0.f) ? 1 : 0;
    P.lenient = filter ? filter->lenient : 0;
    P.arrived = filter ? filter->arrived : nullptr;
    P.query_stride = query_stride > 0 ? query_stride : approx.dim;
    P.g = g;
    if (!(approx.kind == KIND_PQ && g.fused && g.fused_codes_of == approx.codes && g.fused_code_stride == approx.code_stride)) P.g.fused = nullptr;
    {
        const char *fe = getenv("JV_FUSED_PQ");
        if (fe && fe[0] == '0') P.g.fused = nullptr;
    }
    P.approx = approx;
    P.has_rerank = rerank ? 1 : 0;
    P.rerank = rerank ? *rerank : approx;
    P.metric = metric;
    P.queries = queries_dev;
    P.nq = nq;
    P.topK = topK;
    P.rerankK = rerankK;
    P.list_cap = plan.list_cap;
    P.list_alloc = plan.list_alloc;
    P.sort_pow2 = plan.sort_pow2;
    P.visited_cap = plan.visited_cap;
    int lg = 0;
    while ((1 << lg) < plan.visited_cap) lg++;
    P.visited_shift = 32 - lg;
    P.visited_tables = reinterpret_cast<int32_t *>(scratch_dev);
    P.work_counter = work_counter_dev;
    P.nodes_out = nodes_out_dev;
    P.scores_out = scores_out_dev;
    P.counters = counters_dev;
    P.overflow = overflow_flags_dev;
    P.query_index = query_index_dev;
    P.blobA_floats = blob_floats(approx);
    P.pq_smem_m = plan.pq_smem_m;
    P.smemA_floats = search_smemA_floats(approx, plan.pq_smem_m);
    P.blobR_floats = rerank ? blob_floats(*rerank) : 0;
    P.blob_global = nullptr;
    P.vis_slots_log = plan.vis_slots_log;
    P.vis_rlog = plan.vis_rlog;
    P.vis_idmask = plan.vis_idmask;
    P.row_prefetch = plan.row_prefetch;
    P.pq_rows = plan.pq_rows;
    {
        // on for the latency-bound walks (PQ / BQ: c3 12.0 -> 11.5 ms); off where HBM is already saturated and a wasted adjacency
        // line costs more than an early one saves (fp32 / NVQ: c2 13.8 vs 14.0 ms). JV_EARLY_PREFETCH=0|1 overrides.
        const char *ep = getenv("JV_EARLY_PREFETCH");
        // (a batch that does not fill the GPU is latency bound whatever the scorer: on as well)
        P.early_pf = ep ? atoi(ep) : ((approx.kind == KIND_PQ || approx.kind == KIND_BQ || nq <= plan.ctas) ? 1 : 0);
    }
    if (plan.blob_in_global) {
        size_t off = ((plan.vis_slots_log ? 256 : (size_t)plan.ctas * plan.visited_cap * sizeof(int32_t)) + 255) & ~(size_t)255;
        P.blob_global = reinterpret_cast<float *>(reinterpret_cast<char *>(scratch_dev) + off);
    }
    P.dbg = nullptr;
#ifdef JV_SEARCH_PROFILE
    static unsigned long long *dbg_dev = nullptr;
    if (!dbg_dev) cudaMalloc(&dbg_dev, 8 * sizeof(unsigned long long));
    cudaMemsetAsync(dbg_dev, 0, 8 * sizeof(unsigned long long), s);
    P.dbg = dbg_dev;
#endif
    cudaError_t e = cudaMemsetAsync(work_counter_dev, 0, sizeof(int), s);
    if (e != cudaSuccess) return e;
#define CALL(K, M, B, V)                                                                                                              \
    do {                                                                                                                              \
        e = cudaFuncSetAttribute(graph_search_kernel<K, M, B, V>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem_bytes); \
        if (e == cudaSuccess) graph_search_kernel<K, M, B, V><<<plan.ctas, SearchThreads<K>::value, plan.smem_bytes, s>>>(P);               \
    } while (0)
    JV_SEARCH_DISPATCH(approx.kind, metric, plan.pq_wide != 0, plan.vis_slots_log != 0, CALL);
#undef CALL
    if (e != cudaSuccess) return e;
    g_launches++;
#ifdef JV_SEARCH_PROFILE
    {
        unsigned long long h[8];
        cudaStreamSynchronize(s);
        cudaMemcpy(h, P.dbg, sizeof(h), cudaMemcpyDeviceToHost);
        const double it = h[5] ? (double)h[5] : 1.0, nqd = (double)nq;
        fprintf(stderr, "[search profile] kind=%d nq=%d iterations/q=%.1f scored/it=%.1f cycles/it: gather=%.0f score=%.0f merge=%.0f | per query: prepare+clear=%.0f rerank+out=%.0f total=%.0f\n",
                approx.kind, nq, it / nqd, (double)h[6] / it, (double)h[1] / it, (double)h[2] / it, (double)h[3] / it, (double)h[0] / nqd, (double)h[4] / nqd, (double)h[7] / nqd);
    }
#endif
    return cudaGetLastError();
}

}  // namespace jv
