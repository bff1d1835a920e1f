// kernels.h — host-callable launchers of the sm_100a kernels (internal; the public surface is include/jvector_b200.h)
#pragma once
#include <atomic>
#include <cuda_runtime.h>
#include <stdint.h>

#include "scorers.cuh"

namespace jv {

extern std::atomic<long long> g_launches;  // kernels launched by this library (jv_kernel_launch_count)
constexpr int MAX_DEGREE = 128;            // widest adjacency row the search kernel accepts

struct GraphDesc {
    int32_t n;
    int degree;
    int levels;  // >= 1
    int32_t entry_node;
    int entry_level;
    const int32_t *adj0;       // [n][degree]
    const int32_t *upper_row;  // [(levels-1)][n] row index or -1 (nullptr when levels == 1)
    const int32_t *upper_adj;  // rows of all upper levels, concatenated
    const long long *upper_off;  // [(levels-1)] first row of each level in upper_adj (device)
    // FusedPQ feature (base:graph/disk/feature/FusedPQ.java): per node ONE record = [degree int32 neighbour ids][degree code rows
    // of fused_code_stride bytes, zero padded], so a level-0 hop of a PQ walk is one contiguous read. nullptr = not fused.
    const uint8_t *fused;
    const uint8_t *fused_codes_of;  // the PQ code array the records were packed from (identity of the data set they belong to)
    int fused_rec;                  // bytes per record (multiple of 16)
    int fused_code_stride;
};

struct SearchCounters {  // device-side totals
    unsigned long long visited, expanded, expanded_base, reranked, overflowed;
    unsigned long long rows_read;  // fp32 walks: full rows the walking scorer read (visited minus the sketch's drops)
};

// ---- sketch.cu: projection sketch of an fp32 data set (DOT_PRODUCT walks skip rows it proves cannot enter the list) ----
// For an orthonormal basis P (SKETCH_K rows of `stride` floats) and r = x - P^T (P x):  q.x = (P q).(P x) + q.r  and
// q.r <= ||q - P^T P q|| ||r||, so (P q).(P x) + ||q_perp|| ||r|| bounds the score from above for 128 + 8 bytes of reads per row.
constexpr int SKETCH_K = 32;
struct F32Sketch {
    const float *basis;   // [SKETCH_K][stride] fp32 rows of P (orthonormal in double, then rounded)
    const double *gram;   // [SKETCH_K][SKETCH_K] basis . basis^T of the ROUNDED rows (what the query side's ||q_perp|| uses)
    const float4 *proj;   // [n][SKETCH_K / 4] fp32(P x): one 128-byte line per row
    const float2 *norms;  // [n] {||x - P^T fp32(P x)||, ||x||}, both rounded up
};
size_t f32_sketch_bytes(const DataDesc &d);
// builds the sketch of `d` into `mem` (f32_sketch_bytes long) and synchronises `s`. *captured = the share of the sample rows'
// energy (sum of squares) the basis captures; the caller discards a sketch that captures too little to drop anything.
cudaError_t build_f32_sketch(const DataDesc &d, void *mem, F32Sketch *sk, double *captured, cudaStream_t s);

// ---- kernels_batch.cu ----
cudaError_t launch_prepare(const DataDesc &d, int metric, const float *queries_dev, int nq, float *blobs_dev, cudaStream_t s);
// ragged: query qi scores ids[offsets[qi]..offsets[qi+1]); offsets == nullptr: every query scores ids[0..n) -> scores[qi*n + i]
constexpr int HOP_MAX_IDS = 64;
struct HopIds { int32_t ids[HOP_MAX_IDS]; };
// one hop of one search with the ids in the kernel parameters and the scores stored to mapped host memory (latency path)
cudaError_t launch_score_hop(const DataDesc &d, int metric, const float *blob_dev, const int32_t *ids_host, int n, float *scores_mapped, cudaStream_t s);
cudaError_t launch_score_ragged(const DataDesc &d, int metric, const float *blobs_dev, int nq, const int32_t *ids_dev,
                                const int32_t *offsets_dev, int n_shared, int max_per_query, float *scores_dev, cudaStream_t s, int chunk = 0,
                                int *done_counter = nullptr, int *host_flag = nullptr, int seq = 0);
cudaError_t launch_score_pairs(const DataDesc &d, int metric, const int32_t *a_dev, const int32_t *b_dev, int n, float *out_dev, cudaStream_t s);

struct TopkScratch {
    int32_t *sample_ids;   // [S]
    float *sample_scores;  // [nq][S]
    long long *thr;        // [nq]
    long long *thr_safe;   // [nq]
    long long *buf;        // [nq][cap]
    int *cnt;              // [nq]
    int *qlist_a, *qlist_b;  // [nq] each: queries still unresolved after a pass
    int S, cap;
};
cudaError_t launch_topk_bruteforce(const DataDesc &d, int metric, const float *blobs_dev, int nq, int k, const TopkScratch &ts,
                                   long long *keys_out_dev, int *overflow_flag_dev, cudaStream_t s);

cudaError_t launch_add_int(int *dst_dev, const int *src_dev, cudaStream_t s);
// keys[i] -> same score, node id + id_base (KEY_MIN pads untouched)
cudaError_t launch_key_rebase(long long *keys_dev, long long count, long long id_base, cudaStream_t s);
// per query: the k best of parts*k keys (the NCCL-gathered per-shard top-k), descending
cudaError_t launch_topk_merge(const long long *keys_in_dev, int nq, int parts, int k, long long *keys_out_dev, cudaStream_t s);
// the same for keys laid out [parts][nq][k] (shard-major, what peer copies / all_gather produce)
cudaError_t launch_topk_merge_strided(const long long *keys_in_dev, int nq, int parts, int k, long long *keys_out_dev, cudaStream_t s);

cudaError_t launch_bq_encode(const float *rows_dev, long long n, int dim, int row_stride, unsigned long long *words_dev, cudaStream_t s);
cudaError_t launch_pq_encode(const DataDesc &pq, const float *rows_dev, long long n, int row_stride, uint8_t *codes_dev, cudaStream_t s);
cudaError_t launch_pq_self_magnitudes(const DataDesc &pq, float *mag_dev, cudaStream_t s);
cudaError_t launch_pq_pair_table(const DataDesc &pq, int euclidean, float *table_dev, cudaStream_t s);
cudaError_t launch_kmeans_assign(const float *points_dev, long long n, int dim, int point_stride, const float *centroids_dev, int k, int32_t *assign_dev, cudaStream_t s);
cudaError_t launch_nvq_encode(const float *rows_dev, long long n, int row_stride, int nsub, const int *sizes_dev, const int *offsets_dev,
                              const float *mean_dev, int learn, float *params_dev, uint8_t *bytes_dev, int byte_stride, cudaStream_t s);

// ---- bq_imma.cu: BQ Hamming top-k as an exact u8 contraction on the tensor cores (IMMA.16832) ----
constexpr int BQ_IMMA_CAP = 8192;  // captured keys per query in the filter pass
bool bq_imma_supported(const DataDesc &d, int k);
size_t bq_imma_scratch_bytes(long long n, int nq, int W);
// fully asynchronous on `s`: keys_out_dev [nq][k] best first with GLOBAL ids (row + id_base); *unresolved_dev = number of queries
// the integer-threshold path could not resolve (a Hamming bin wider than the buffer) — the caller falls back for those batches
cudaError_t launch_bq_topk_imma(const DataDesc &d, const float *queries_dev, int nq, int k, long long id_base, void *scratch_dev,
                                long long *keys_out_dev, int *unresolved_dev, int sm_count, cudaStream_t s);
// ---- bq_umma.cu: the filter pass of the same pipeline on tcgen05 (kind::i8, TMEM accumulators) ----
bool bq_umma_supported(const DataDesc &d);
size_t bq_umma_image_bytes(int nq, int W);
cudaError_t launch_bq_umma_filter(const DataDesc &d, const uint32_t *qbits_dev, int nq, int nq_pad, const int *t2_dev, const int *pb_dev, long long *buf_dev,
                                  int *cnt_dev, int cap, long long id_base, uint8_t *images_dev, int sm_count, cudaStream_t s);

// FusedPQ.writeInline (FusedPQ.java:122-141) for every node: records[node] = ids + the neighbours' code rows in neighbour order
cudaError_t launch_fuse_pq(const GraphDesc &g, const DataDesc &pq, uint8_t *records_dev, int rec_bytes, cudaStream_t s);

// ---- search.cu ----
constexpr int MAX_LIST_CAP = 8192;  // longest candidate list (entries) the search kernel keeps in shared memory
struct SearchPlan {
    int threads;
    size_t smem_bytes;
    int ctas;
    int list_cap;     // entries the candidate list retains: rerankK + room for a tie tail
    int list_alloc;   // entries per list buffer (>= list_cap, >= sort_pow2)
    int sort_pow2;    // next power of two >= rerankK
    int visited_cap;  // power of two
    int blob_in_global;  // PQ: (part of) the LUT lives in an L2-resident global slice per CTA
    int pq_smem_m;       // PQ: LUT rows of sub-spaces [0, pq_smem_m) stay in shared memory
    int pq_wide;         // PQ: the 64-register build of the kernel (residency is limited by shared memory anyway)
    int blob_floats;
    int vis_slots_log, vis_rlog;  // visited set in shared memory: log2(slots), log2(slots per region); 0 = per-CTA global table
    unsigned vis_idmask;
    int row_prefetch;             // fp32 / NVQ walks: bulk L2 prefetch of newly visited rows
    int pq_rows;                  // PQ walk: lane = candidate, warp = partial sum
};
// acceptOrds / threshold / rerankFloor of GraphSearcher.search (base:graph/GraphSearcher.java:166-181,427-431, NodeQueue.java:168-230)
struct SearchFilter {
    const uint32_t *accept_bits;    // device; bit (node & 31) of word (node >> 5) set = acceptable; nullptr = Bits.ALL
    long long accept_stride_words;  // words between the bitsets of two queries; 0 = one bitset shared by the whole batch
    float threshold;                // minimum approximate score of a result; 0 = none
    float rerank_floor;             // NodeQueue.rerank's rerankFloor; 0 = none
    int lenient;                    // builder only: overflowing walks are cut short and counted instead of failing
    const int *arrived;             // device int or nullptr: queries [0, *arrived) are in place (host-pointer searches overlap the H2D copy)
};
cudaError_t plan_search(const DataDesc &approx, const DataDesc *rerank, const GraphDesc &g, int topK, int rerankK, int nq,
                        int visited_cap_hint, int list_cap_hint, int sm_count, SearchPlan *plan);
size_t search_scratch_bytes(const SearchPlan &p);
cudaError_t launch_search(const GraphDesc &g, const DataDesc &approx, const DataDesc *rerank, int metric, const float *queries_dev,
                          int nq, int topK, int rerankK, const SearchPlan &plan, void *scratch_dev, int *work_counter_dev,
                          int32_t *nodes_out_dev, float *scores_out_dev, SearchCounters *counters_dev, uint8_t *overflow_flags_dev,
                          const int32_t *query_index_dev, int query_stride, const SearchFilter *filter, cudaStream_t s,
                          const F32Sketch *sketch = nullptr);

// ---- build.cu ----
struct BuildParams {
    int degree, beam;
    float overflow, alpha;
    int max_batch;
    int window;  // in-progress peers every insert sees besides its beam (-1 = default: what fits the 128-candidate tile, at most 32)
};
struct BuildStats {
    long long searched, pruned, dropped_backlinks, batches;
    long long truncated_searches;  // insert searches cut short by a full visited table / an oversized tie tail (pathological inputs)
};
// flat Vamana graph over rows [0, n) of an f32 data set; adj_out_dev [n][degree] (-1 padded); entry node is 0
cudaError_t build_graph_flat(const DataDesc &f32, int metric, const BuildParams &bp, int32_t *adj_out_dev, int sm_count,
                             BuildStats *stats, cudaStream_t s);
// the same build advanced batch by batch; a sharded build calls the *_slice functions for its part of each batch and moves the
// rows between the replicas itself (see build.cu)
struct GraphBuilder;
cudaError_t builder_create(const DataDesc &d, int metric, const BuildParams &bp, int sm_count, GraphBuilder **out, cudaStream_t s);
void builder_destroy(GraphBuilder *B);
bool builder_next_batch(GraphBuilder *B, int *first, int *count);
cudaError_t builder_insert_slice(GraphBuilder *B, int first, int count, int lo, int hi, int32_t *rows_out, int *deg_out, cudaStream_t s);
cudaError_t builder_apply_new(GraphBuilder *B, int first, int count, const int32_t *rows, const int *rdeg, cudaStream_t s);
cudaError_t builder_reprune_slice(GraphBuilder *B, int lo, int hi, int32_t *rows_out, int *deg_out, cudaStream_t s);
cudaError_t builder_apply_repruned(GraphBuilder *B, int count, const int32_t *rows, const int *rdeg, cudaStream_t s);
cudaError_t builder_collect_over_degree(GraphBuilder *B, cudaStream_t s);
cudaError_t builder_list_count(GraphBuilder *B, int *count_host, cudaStream_t s);
cudaError_t builder_finish(GraphBuilder *B, int32_t *adj_out_dev, BuildStats *stats, cudaStream_t s);
int builder_row_cap(const GraphBuilder *B);
int builder_degree(const GraphBuilder *B);
int builder_max_batch(const GraphBuilder *B);
cudaError_t launch_gather_rows(const DataDesc &f32, const int32_t *ids_dev, int count, float *out_dev, cudaStream_t s);

}  // namespace jv
