/*
 * jvector_b200.h — C ABI of libjvector_b200.so, the B200 (sm_100a) replacement for JVector's libjvector.so.
 *
 * Two groups of entry points:
 *
 *  (1) The 24 symbols of the reference's native library, with identical C signatures, so the library can be
 *      installed as `libjvector.so` under jvector-native unchanged. They replace
 *      /root/reference/jvector-native/src/main/native/src/jvector_simd_kernel_list.h:35-61 and
 *      src/jvector_simd.h:47,53. The reference binds them with Linker.Option.critical(true) on on-heap segments
 *      (jvector-native/src/main/java/.../cnative/NativeSimdOps.java:1164,1226,...), i.e. they must be short,
 *      synchronous, host-memory functions; they are the n = 1 case and stay on the host by contract.
 *
 *  (2) The batched GPU entry points (prefix jv_) that the GPU-backed VectorizationProvider / ScoreFunction
 *      implementations bind with ordinary (non-critical) downcall handles: data sets are registered once and
 *      live in HBM; each hop / rerank list / multi-query step / whole search batch is ONE call.
 *      They replace the per-candidate call sites
 *        base:graph/OnHeapGraphIndex.java:475-483, base:graph/disk/OnDiskGraphIndex.java:639-661 (neighbour loop),
 *        base:graph/NodeQueue.java:168-188 (rerank loop), base:quantization/PQDecoder.java:48-53 (LUT build),
 *        base:graph/GraphIndexBuilder.java:830-835, base:graph/diversity/VamanaDiversityProvider.java:56-95,
 *        base:graph/GraphSearcher.java:263-282,406-457 (whole traversal, device resident).
 *      (`base:` = jvector-base/src/main/java/io/github/jbellis/jvector/)
 *
 * Conventions for group (2): every function returns an int status (0 = JV_OK, negative = error) and never throws
 * or aborts across the ABI; jv_last_error() returns a thread-local message. All pointer arguments are HOST
 * pointers borrowed for the duration of the call unless the name ends in _device. Scores are the reference's
 * similarity scores (base:vector/VectorSimilarityFunction.java:37-69), higher = closer. Top-k keys are the
 * reference's 64-bit ordering key (base:graph/NodeQueue.java:125-137). No CPU fallback exists: without an
 * sm_100 device jv_gpu_init() fails and every other jv_ call returns JV_ERR_NO_DEVICE.
 */
#ifndef JVECTOR_B200_H
#define JVECTOR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define JV_API __attribute__((visibility("default")))

/* ------------------------------------------------------------------------------------------------
 * (1) legacy libjvector.so ABI — jvector_simd_kernel_list.h:35-61
 * ---------------------------------------------------------------------------------------------- */
JV_API float cosine_f32(const float *a, size_t aoffset, const float *b, size_t boffset, size_t length);
JV_API float dot_product_f32(const float *a, size_t aoffset, const float *b, size_t boffset, size_t length);
JV_API float euclidean_f32(const float *a, size_t aoffset, const float *b, size_t boffset, size_t length);
JV_API void add_in_place_f32(float *v1, const float *v2, size_t length);
JV_API void add_scalar_in_place_f32(float *v1, float value, size_t length);
JV_API void sub_in_place_f32(float *v1, const float *v2, size_t length);
JV_API void sub_scalar_in_place_f32(float *v1, float value, size_t length);
JV_API float max_f32(const float *v, size_t length);
JV_API void min_in_place_f32(float *v1, const float *v2, size_t length);
JV_API float assemble_and_sum_f32(const float *data, int dataBase, const unsigned char *baseOffsets, int baseOffsetsOffset, size_t baseOffsetsLength);
JV_API float assemble_and_sum_pq_f32(const float *data, size_t subspaceCount, const unsigned char *baseOffsets1, int baseOffsetsOffset1, const unsigned char *baseOffsets2, int baseOffsetsOffset2, int clusterCount);
JV_API float pq_decoded_cosine_similarity_f32(const unsigned char *baseOffsets, int baseOffsetsOffset, size_t baseOffsetsLength, int clusterCount, const float *partialSums, const float *aMagnitude, float bMagnitude);
JV_API void calculate_partial_sums_dot_f32(const float *codebook, int codebookIndex, size_t size, int clusterCount, const float *query, int queryOffset, float *partialSums);
JV_API void calculate_partial_sums_euclidean_f32(const float *codebook, int codebookIndex, size_t size, int clusterCount, const float *query, int queryOffset, float *partialSums);
JV_API void calculate_partial_sums_self_magnitude_f32(const float *codebook, int codebookIndex, size_t size, int clusterCount, float *partialSums);
JV_API void nvq_quantize_8bit(const float *vector, size_t length, float alpha, float x0, float minValue, float maxValue, unsigned char *destination);
JV_API float nvq_loss(const float *vector, size_t length, float alpha, float x0, float minValue, float maxValue, int nBits);
JV_API float nvq_uniform_loss(const float *vector, size_t length, float minValue, float maxValue, int nBits);
JV_API float nvq_square_l2_distance_8bit(const float *vector, const unsigned char *quantized, size_t length, float alpha, float x0, float minValue, float maxValue);
JV_API float nvq_dot_product_8bit(const float *vector, const unsigned char *quantized, size_t length, float alpha, float x0, float minValue, float maxValue);
JV_API int64_t nvq_cosine_8bit_packed(const float *vector, const unsigned char *quantized, size_t length, float alpha, float x0, float minValue, float maxValue, const float *centroid);
/* no-op here: this library reads NVQ bytes in natural order (as base:vector/DefaultVectorUtilSupport.java:454) */
JV_API void nvq_shuffle_query_in_place_8bit(float *vector, size_t length);
/* jvector_simd.h:47,53 — reflected on by base:vector/VectorizationProvider.java:132-136 */
JV_API const char *jvector_simd_get_active_isa(void);
JV_API const char *jvector_simd_get_max_isa_env(void);

/* ------------------------------------------------------------------------------------------------
 * (2) batched GPU ABI
 * ---------------------------------------------------------------------------------------------- */
enum { JV_EUCLIDEAN = 0, JV_DOT_PRODUCT = 1, JV_COSINE = 2 }; /* VectorSimilarityFunction ordinal order */

enum {
    JV_OK = 0,
    JV_ERR_NO_DEVICE = -1,   /* no CUDA device / not sm_100 / jv_gpu_init not called */
    JV_ERR_INVALID = -2,     /* bad argument */
    JV_ERR_CUDA = -3,        /* CUDA runtime error, see jv_last_error() */
    JV_ERR_OOM = -4,
    JV_ERR_UNSUPPORTED = -5, /* combination not implemented (e.g. metric for BQ other than Hamming score) */
    JV_ERR_OVERFLOW = -6     /* device scratch (visited table, candidate list) too small even after retry */
};

typedef struct jv_dataset_s *jv_dataset; /* vectors / codes resident in HBM */
typedef struct jv_query_s *jv_query;     /* one query prepared against one data set (LUT / bits / shifted copy) */
typedef struct jv_graph_s *jv_graph;     /* adjacency resident in HBM */

/* Bind CUDA device `device` and make it the device on which the CALLING THREAD creates data sets and graphs. Idempotent. Every
 * handle remembers its device, so binding another device later never invalidates existing handles. */
JV_API int jv_gpu_init(int device);
/* One process driving several GPUs (the reference host is one JVM: base:vector/VectorizationProvider.java:79-177): bind every
 * device of the mask (bit d = CUDA device d) and enable peer access between them (NVLink / NVSwitch). SURVEY §8(b). */
JV_API int jv_gpu_init_mask(uint32_t device_mask);
JV_API uint32_t jv_gpu_bound_mask(void);
/* the device on which the calling thread's next register / create calls place their data (a bound device) */
JV_API int jv_gpu_set_device(int device);
JV_API int jv_gpu_device_count(void);
JV_API const char *jv_last_error(void);
JV_API const char *jv_version(void);
JV_API int jv_gpu_sm_count(void);

/* ---- data sets (the RandomAccessVectorValues / CompressedVectors a ScoreFunction reads) ---- */
/* rows: [n][dim] fp32 row-major (base:graph/RandomAccessVectorValues.java) */
JV_API int jv_dataset_register_f32(const float *rows, int64_t n, int dim, jv_dataset *out);
/* PQVectors: codes [n][M] u8 (base:quantization/PQVectors.java:377-395), codebooks concatenated in sub-space order,
 * codebook m = k * size_m floats [k][size_m] (ProductQuantization.java:66), sub-vector sizes per
 * ProductQuantization.java:535-550, centroid = globalCentroid or NULL */
JV_API int jv_dataset_register_pq(const uint8_t *codes, int64_t n, int dim, int M, int k, const float *codebooks,
                                  const float *centroid, jv_dataset *out);
/* BQVectors: words [n][ceil(dim/64)] u64, bit j of word i = (v[64 i + j] > 0) (BinaryQuantization.java:96-109) */
JV_API int jv_dataset_register_bq(const uint64_t *words, int64_t n, int dim, jv_dataset *out);
/* NVQVectors, 8 bit: bytes [n][dim] u8 (sub-vectors concatenated), params [n][nsub][4] = {min,max,growthRate,midpoint}
 * (NVQuantization.java:489-498), mean = globalMean */
JV_API int jv_dataset_register_nvq(const uint8_t *bytes, const float *params, int64_t n, int dim, int nsub,
                                   const float *mean, jv_dataset *out);
/* rows already in HBM on the calling thread's device (e.g. produced by another kernel): BORROWED, not copied — the caller keeps
 * them alive until jv_dataset_free. 16-byte aligned, row_stride = dim rounded up to 4 floats, padding floats zero. */
JV_API int jv_dataset_adopt_f32_device(const float *rows_device, int64_t n, int dim, int row_stride, jv_dataset *out);
/* fp32 data sets searched with DOT_PRODUCT (dim >= 256, rows >= 252 MB) carry a projection sketch: 32 fp32 projections and two
 * norms per row (136 bytes per row, in HBM), built by the first such graph search, with which the walk proves most candidates
 * cannot enter its list without reading their rows. Results are the same with and without it. The sketch describes the rows as
 * they were when it was built: rows must not change while a data set is in use (adopted rows are the caller's memory) unless
 * jv_dataset_invalidate_sketch is called after the change and before the next search. JV_F32_SKETCH=0 turns the sketch off. */
JV_API int jv_dataset_invalidate_sketch(jv_dataset ds);
/* state: 1 built, 0 not built (yet), -1 skipped because the basis captured < 50 % of the rows' energy (nothing would be dropped);
 * captured: that share. Any output may be NULL; basis_out [32][row_stride], proj_out [n][32], norms_out [n][2] need state 1. */
JV_API int jv_dataset_f32_sketch(jv_dataset ds, int *state, double *captured, float *basis_out, float *proj_out, float *norms_out);
JV_API int jv_dataset_device(jv_dataset ds);
/* ImmutablePQVectors' code-vs-code scoring (base:quantization/ImmutablePQVectors.java:63-105): build the triangular
 * centroid-vs-centroid table of ProductQuantization.createCodebookPartialSums (ProductQuantization.java:609-628; 12.6 MB at M = 96,
 * k = 256) in HBM; jv_score_pairs on this data set then sums table entries — assembleAndSumPQ, native-c:
 * src/jvector_simd_kernels.cpp:729-815 — instead of recomputing centroid distances. EUCLIDEAN and DOT_PRODUCT have their own
 * tables, COSINE uses the dot-product one. */
JV_API int jv_dataset_pq_pair_table(jv_dataset pq, int metric);
JV_API int jv_dataset_pq_pair_table_download(jv_dataset pq, int metric, float *table_out /* [M][k (k + 1) / 2] */);
JV_API int jv_dataset_free(jv_dataset ds);
JV_API int64_t jv_dataset_size(jv_dataset ds);
JV_API int jv_dataset_dim(jv_dataset ds);
JV_API int64_t jv_dataset_device_bytes(jv_dataset ds);

/* ---- ScoreFunction for one query: CompressedVectors.precomputedScoreFunctionFor / DefaultSearchScoreProvider.exact ---- */
JV_API int jv_query_begin(jv_dataset ds, const float *q, int metric, jv_query *out);
/* the neighbour loop of one processNeighbors call / one rerank list: ids[n] -> scores[n], ONE kernel launch */
JV_API int jv_score_batch(jv_query q, const int32_t *ids, int n, float *scores_out);
JV_API int jv_query_end(jv_query q);
/* PQ only: copy the query's partial-sums table (PQDecoder.java:41-54) back, lut_out[M*k] */
JV_API int jv_query_get_lut(jv_query q, float *lut_out);

/* ---- query batches: the host-driven seam with persistent state ----
 * A batch of searches that the HOST drives hop by hop (GraphSearcher on the JVM, base:graph/GraphSearcher.java:406-457): the
 * prepared queries (LUTs / bit packs / shifted copies) are built once and stay in HBM until jv_query_batch_end; a step uploads
 * only ids + offsets through pinned staging owned by the batch and brings the scores back. */
typedef struct jv_query_batch_s *jv_query_batch;
JV_API int jv_query_batch_begin(jv_dataset ds, int metric, const float *queries, int nq, jv_query_batch *out);
/* one step of all nq searches: query i scores ids[offsets[i] .. offsets[i+1]) -> scores_out in the same order; ONE launch.
 * device_ms (optional): CUDA-event time of the scoring kernel alone */
JV_API int jv_query_batch_score(jv_query_batch b, const int32_t *ids, const int32_t *offsets, float *scores_out, double *device_ms);
/* one hop of search `query_index`: ids[n] -> scores_out[n]; the kernel reads / writes mapped pinned memory (no separate copies) */
JV_API int jv_query_batch_score_one(jv_query_batch b, int query_index, const int32_t *ids, int n, float *scores_out);
JV_API int jv_query_batch_end(jv_query_batch b);

/* one step of many searches: query qi scores ids[offsets[qi] .. offsets[qi+1]) ; one launch for the whole step */
JV_API int jv_score_multi(jv_dataset ds, int metric, const float *queries, int nq, const int32_t *ids,
                          const int32_t *offsets, float *scores_out);
/* diversity scoring (BuildScoreProvider.diversityProviderFor): score(a[i], b[i]) for n pairs, one launch.
 * f32: exact; PQ: codebook-vs-codebook (PQVectors.java:284-350); BQ: BQVectors.java:98-105 */
JV_API int jv_score_pairs(jv_dataset ds, int metric, const int32_t *a, const int32_t *b, int n, float *scores_out);
/* exhaustive scoring of every row for nq queries with a fused device-side top-k; keys_out[nq][k] best first,
 * padded with INT64_MIN */
JV_API int jv_topk_bruteforce(jv_dataset ds, int metric, const float *queries, int nq, int k, int64_t *keys_out);
/* multi-GPU form (SURVEY §8e): the base is range-sharded, this rank holds rows [id_base, id_base + n); queries and keys stay in
 * HBM so the keys can be the NCCL send buffer. Node ids inside the keys are global (local id + id_base). */
JV_API int jv_topk_bruteforce_device(jv_dataset ds, int metric, const float *queries_device, int nq, int k, int64_t id_base,
                                     int64_t *keys_out_device);
/* the merge after the all-gather: keys_in [nq][parts * k] (any order) -> keys_out [nq][k] best first */
JV_API int jv_topk_merge_device(const int64_t *keys_in_device, int nq, int parts, int k, int64_t *keys_out_device);

/* Stream-ordered forms for callers that own a CUDA stream (the multi-process bench puts the local top-k, the NCCL all-gather and
 * the merge on ONE stream with no host synchronisation in between). BQ data sets only (the tensor-core contraction of
 * csrc/bq_imma.cu); *status_device receives the number of queries left unresolved (0 normally; non-zero = call the synchronous
 * form, which falls back to the key-threshold kernels). cuda_stream: a cudaStream_t. */
JV_API int jv_topk_bruteforce_device_async(jv_dataset ds, int metric, const float *queries_device, int nq, int k, int64_t id_base,
                                           int64_t *keys_out_device, int32_t *status_device, void *cuda_stream);
/* keys_in: SHARD-MAJOR [parts][nq][k], exactly what an all-gather of the per-rank [nq][k] arrays produces */
JV_API int jv_topk_merge_device_async(const int64_t *keys_in_device, int nq, int parts, int k, int64_t *keys_out_device, void *cuda_stream);

/* ---- several GPUs driven by ONE process (SURVEY §8b last row, §8e) ----
 * jv_multi: a base RANGE-SHARDED by contiguous node id over the devices bound by jv_gpu_init_mask (shard i holds rows
 * [first_row_i, first_row_i + rows_i)). jv_multi_topk_bruteforce: every shard scores all queries on its own stream (one worker
 * thread per device inside the call), the per-shard top-k keys (global node ids) go to the first device by NVLink peer copies
 * and are merged there by the reference key — the same exchange the multi-process path does with an NCCL all-gather. */
typedef struct jv_multi_s *jv_multi;
JV_API int jv_multi_register_bq(const uint64_t *words, int64_t n, int dim, jv_multi *out);
JV_API int jv_multi_register_f32(const float *rows, int64_t n, int dim, jv_multi *out);
JV_API int jv_multi_free(jv_multi m);
JV_API int jv_multi_shard_count(jv_multi m);
JV_API int jv_multi_shard_info(jv_multi m, int shard, int *device, int64_t *first_row, int64_t *rows);
JV_API int jv_multi_topk_bruteforce(jv_multi m, int metric, const float *queries, int nq, int k, int64_t *keys_out);

/* ---- bulk encoders (next to the scoring path: ProductQuantization.encodeAll, BinaryQuantization.encodeAll,
 *      NVQuantization.encodeAll) ---- */
JV_API int jv_bq_encode_batch(const float *rows, int64_t n, int dim, uint64_t *words_out);
JV_API int jv_pq_encode_batch(const float *rows, int64_t n, int dim, int M, int k, const float *codebooks,
                              const float *centroid, uint8_t *codes_out);
JV_API int jv_nvq_encode_batch(const float *rows, int64_t n, int dim, int nsub, const float *mean, int learn,
                               float *params_out, uint8_t *bytes_out);
/* the assignment step of k-means (KMeansPlusPlusClusterer.getNearestCluster, base:quantization/KMeansPlusPlusClusterer.java:329-342)
 * for a batch of points [n][dim] against centroids [k][dim]: index of the nearest centroid, first minimum wins */
JV_API int jv_kmeans_assign_batch(const float *points, int64_t n, int dim, const float *centroids, int k, int32_t *assignments_out);
/* the same encoders over rows that are already resident in HBM (a registered fp32 data set): no host->device copy */
JV_API int jv_bq_encode_dataset(jv_dataset f32, uint64_t *words_out);
JV_API int jv_pq_encode_dataset(jv_dataset f32, int M, int k, const float *codebooks, const float *centroid, uint8_t *codes_out);
JV_API int jv_nvq_encode_dataset(jv_dataset f32, int nsub, const float *mean, int learn, float *params_out, uint8_t *bytes_out);

/* NVQ inline vectors without a host round trip: encode the resident fp32 rows into a NEW resident NVQ data set */
JV_API int jv_nvq_encode_dataset_resident(jv_dataset f32, int nsub, const float *mean, int learn, jv_dataset *out);

/* ---- graph: ImmutableGraphIndex adjacency in HBM + GraphSearcher traversal on the device ---- */
/* adj0: [n][degree] int32, -1 padded (level 0). */
JV_API int jv_graph_create(int32_t n, int degree, const int32_t *adj0, int32_t entry_node, jv_graph *out);
/* add level 1, 2, ... in order; node_ids[count] are the members, adj [count][degree] their lists at that level.
 * The entry node must be a member of the last level added. */
JV_API int jv_graph_add_level(jv_graph g, int32_t count, const int32_t *node_ids, const int32_t *adj);
/* FusedPQ feature (base:graph/disk/feature/FusedPQ.java:99-101,122-141,215-241): pack, for every node, its level-0 neighbour ids
 * and the neighbours' PQ codes into ONE record [degree int32 ids][degree code rows, zero padded] (built on the device from the
 * resident adjacency and codes). A later search whose `approx` is this PQ data set then scores neighbours from the expanded
 * node's record — FusedPQDecoder.similarityToNeighbor (base:quantization/FusedPQDecoder.java:84-114), the
 * "useEdgeLoading && level == 0" branch of OnDiskGraphIndex.java:639-651 — one contiguous read per hop; upper levels and the
 * entry node use the plain code rows (the hierarchy's cached source features, FusedPQDecoder.java:96-105). Scores are those of
 * the plain PQ walk. JV_FUSED_PQ=0 in the environment ignores the records (A/B timing). */
JV_API int jv_graph_fuse_pq(jv_graph g, jv_dataset pq);
/* records_out [n][*record_bytes] (query the size with records_out = NULL first) */
JV_API int jv_graph_fused_download(jv_graph g, uint8_t *records_out, int *record_bytes);
JV_API int jv_graph_free(jv_graph g);
JV_API int jv_graph_info(jv_graph g, int32_t *n, int *degree, int *levels, int32_t *entry_node);
JV_API int jv_graph_download(jv_graph g, int level, int32_t *node_ids_out, int32_t *adj_out, int32_t *count_out);

typedef struct {
    int64_t visited;       /* sum over queries of SearchResult.visitedCount (GraphSearcher.java:445-449) */
    int64_t expanded;      /* expandedCount */
    int64_t expanded_base; /* expandedCountBaseLayer */
    int64_t reranked;      /* reranked */
    int64_t retried;       /* queries re-run with a larger visited table */
    double device_ms;      /* CUDA-event time of the device work of this call */
} jv_search_stats;

/* GraphSearcher.search for nq queries at once: traversal scored by `approx`, optional exact rerank by `reranker`
 * (NULL = none, then rerankK survivors are cut to topK by approximate score as GraphSearcher.java:478-486).
 * nodes_out/scores_out [nq][topK], best first, padded with -1 / 0.
 * Host buffers: a batch of >= 1 MB of queries is copied in chunks on a second stream while the search kernel already runs (each
 * query is read only after its chunk has arrived), so with pinned (jv_host_register / cudaHostRegister) buffers the H2D copy is
 * hidden behind the first wave of queries; pageable buffers work and simply copy first. device_ms then includes that overlap. */
JV_API int jv_graph_search_batch(jv_graph g, jv_dataset approx, jv_dataset reranker, int metric,
                                 const float *queries, int nq, int topK, int rerankK,
                                 int32_t *nodes_out, float *scores_out, jv_search_stats *stats);
/* GraphSearcher.search(scoreProvider, topK, rerankK, threshold, rerankFloor, acceptOrds) — base:graph/GraphSearcher.java:166-181.
 * accept_bits: bit (node & 31) of 32-bit word (node >> 5) set = the node may be a RESULT (it is still traversed), applied on
 * level 0 only as searchOneLayer does (:427-431); accept_stride_words = 0 shares one bitset between all queries of the batch,
 * otherwise query i uses accept_bits + i * accept_stride_words. threshold: minimum approximate score of a result (the
 * TwoPhaseTracker early-termination heuristic of ScoreTracker.java is NOT run: a threshold search here visits at least what
 * the reference visits). rerank_floor: NodeQueue.rerank's rerankFloor (NodeQueue.java:168-230). NULL = {NULL, 0, 0, 0}.
 * A filter that rejects most nodes needs a long candidate list; beyond 8192 live candidates the call fails with JV_ERR_OVERFLOW. */
typedef struct {
    const uint32_t *accept_bits;
    int64_t accept_stride_words;
    float threshold;
    float rerank_floor;
} jv_search_options;
JV_API int jv_graph_search_batch_ex(jv_graph g, jv_dataset approx, jv_dataset reranker, int metric,
                                    const float *queries, int nq, int topK, int rerankK, const jv_search_options *opts,
                                    int32_t *nodes_out, float *scores_out, jv_search_stats *stats);
/* same with queries / outputs already in HBM (no host copies in the call) */
JV_API int jv_graph_search_batch_device(jv_graph g, jv_dataset approx, jv_dataset reranker, int metric,
                                        const float *queries_device, int nq, int topK, int rerankK,
                                        int32_t *nodes_out_device, float *scores_out_device, jv_search_stats *stats);

/* _ex form with everything in HBM; opts->accept_bits is a DEVICE pointer here */
JV_API int jv_graph_search_batch_device_ex(jv_graph g, jv_dataset approx, jv_dataset reranker, int metric,
                                           const float *queries_device, int nq, int topK, int rerankK,
                                           const jv_search_options *opts_device_bits, int32_t *nodes_out_device,
                                           float *scores_out_device, jv_search_stats *stats);

/* Replicas: graph + data sets registered once per device (jv_gpu_set_device(d), then the ordinary create / register calls); the
 * batch is split into contiguous slices, one per replica, searched concurrently (no data-path exchange). stats sums the counters,
 * device_ms is the slowest replica. */
JV_API int jv_multi_graph_search_batch(int replicas, const jv_graph *graphs, const jv_dataset *approx, const jv_dataset *rerankers,
                                       int metric, const float *queries, int nq, int topK, int rerankK, const jv_search_options *opts,
                                       int32_t *nodes_out, float *scores_out, jv_search_stats *stats);

/* GraphIndexBuilder.build over an f32 data set with exact scoring (BuildScoreProvider.randomAccessScoreProvider):
 * batched inserts, device-side beam search + Vamana robust prune + back-links. */
typedef struct {
    int degree;        /* M */
    int beam_width;    /* efConstruction */
    float overflow;    /* neighborOverflow, e.g. 1.2 */
    float alpha;       /* 1.2 */
    int add_hierarchy; /* HNSW-style upper levels (GraphIndexBuilder.java:562-575) */
    uint64_t seed;
    int max_batch;     /* 0 = default (16384): nodes inserted per round; they play the reference's concurrently inserting threads */
    int concurrent_window; /* in-progress peers each insert sees besides its beam (getConcurrentCandidates,
                              GraphIndexBuilder.java:823-837): -1 = default (what fits the 128-candidate prune tile, <= 32), 0 = none */
} jv_build_params;
JV_API int jv_graph_build(jv_dataset f32, int metric, const jv_build_params *params, jv_graph *out, double *device_ms);
/* The same build advanced batch by batch, for a build SHARDED over several GPUs (BASELINE config 5): every participant holds a
 * replica of the rows and of the adjacency; per batch each one searches + prunes ITS slice (jv_builder_insert_slice), the caller
 * all-gathers the slices (NCCL; jvector_b200/parallel.py sharded_build), every participant applies the whole batch — back-links in
 * sorted order, so all replicas stay bit-identical — and the rows that passed overflow * M are re-pruned slice-wise and exchanged
 * the same way. All *_device pointers are device buffers of the caller (the collective's send / receive buffers); work is
 * enqueued on `cuda_stream`. Slices are positions [lo, hi) of the batch (insert) or of the sorted overflow list (re-prune). */
typedef struct jv_builder_s *jv_builder;
JV_API int jv_builder_create(jv_dataset f32, int metric, const jv_build_params *params, void *cuda_stream, jv_builder *out);
JV_API int jv_builder_info(jv_builder b, int *degree, int *row_cap, int *max_batch);
JV_API int jv_builder_next_batch(jv_builder b, int32_t *first, int32_t *count); /* count = 0: every node is inserted */
JV_API int jv_builder_insert_slice(jv_builder b, int32_t first, int32_t count, int32_t lo, int32_t hi,
                                   int32_t *rows_out_device /* [count][degree], rows lo..hi-1 written */, int32_t *deg_out_device /* [count] */);
/* rows of the WHOLE batch; overflow_rows (optional, forces a stream sync): length of the sorted list of rows to re-prune */
JV_API int jv_builder_apply_new(jv_builder b, int32_t first, int32_t count, const int32_t *rows_device, const int32_t *deg_device, int32_t *overflow_rows);
JV_API int jv_builder_reprune_slice(jv_builder b, int32_t lo, int32_t hi, int32_t *rows_out_device /* [.][row_cap] */, int32_t *deg_out_device);
JV_API int jv_builder_apply_repruned(jv_builder b, int32_t count, const int32_t *rows_device, const int32_t *deg_device);
/* cleanup(): the sorted list of rows longer than M (enforceDegree), to be re-pruned with the two calls above */
JV_API int jv_builder_collect_over_degree(jv_builder b, int32_t *rows);
JV_API int jv_builder_finish(jv_builder b, jv_graph *out, double *device_ms);
JV_API int jv_builder_free(jv_builder b);
/* counters of this thread's last jv_graph_build (level 0): vectors scored by the insert searches, batches, back-links dropped */
JV_API int jv_graph_build_stats(int64_t *scored_vectors, int64_t *batches, int64_t *dropped_backlinks);

/* device-memory helpers for callers that keep queries/results in HBM (bench `value` leg) */
JV_API int jv_device_malloc(void **out, size_t bytes);
JV_API int jv_device_free(void *p);
JV_API int jv_memcpy_h2d(void *dst_device, const void *src_host, size_t bytes);
JV_API int jv_memcpy_d2h(void *dst_host, const void *src_device, size_t bytes);
JV_API int jv_host_register(void *p, size_t bytes); /* pin a host buffer for faster copies */
JV_API int jv_host_unregister(void *p);
JV_API int jv_device_synchronize(void);
JV_API int64_t jv_kernel_launch_count(void); /* kernels this library has launched since load */
JV_API int64_t jv_search_rows_read(void);    /* fp32 rows the graph searches' walks have read since load (< visited with a sketch) */

#ifdef __cplusplus
}
#endif
#endif /* JVECTOR_B200_H */
