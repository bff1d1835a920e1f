// jvector_b200.hpp — header-only C++ host mirror of the reference's scoring interface over the C ABI (jvector_b200.h).
//
// The reference host is Java; no JDK exists in this image, so the host-side mirror the tests can COMPILE is C++ (and the
// ctypes layer in jvector_b200/api.py). Names and argument meaning follow the reference:
//   VectorSimilarityFunction                       base:vector/VectorSimilarityFunction.java:34-80
//   ScoreFunction::similarityTo / similarityToBatch base:graph/similarity/ScoreFunction.java:30-80 (+ the batch form)
//   F32Vectors / PQVectors / BQVectors / NVQVectors  RandomAccessVectorValues / CompressedVectors, resident in HBM
//   GraphSearcher::search(topK, rerankK)            base:graph/GraphSearcher.java:222-243, for a batch of queries
//   GraphIndexBuilder(M, beamWidth, neighborOverflow, alpha, addHierarchy)::build   base:graph/GraphIndexBuilder.java:436-448
// Errors: the reference throws (UnsupportedOperationException at provider load, IllegalArgumentException on bad arguments);
// here every non-zero status becomes a jv::Error carrying jv_last_error(). No CPU fallback.
#ifndef JVECTOR_B200_HPP
#define JVECTOR_B200_HPP

#include <cstdint>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "jvector_b200.h"

namespace jv {

enum class VectorSimilarityFunction : int { EUCLIDEAN = JV_EUCLIDEAN, DOT_PRODUCT = JV_DOT_PRODUCT, COSINE = JV_COSINE };

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string &m) : std::runtime_error("jvector_b200 error " + std::to_string(c) + ": " + m), code(c) {}
};
inline void check(int rc)
{
    if (rc != JV_OK) throw Error(rc, jv_last_error());
}
/// NativeVectorizationProvider's constructor: throws when no sm_100 device can be bound (caller falls back to Panama)
inline void init(int device = 0) { check(jv_gpu_init(device)); }

class Vectors {
public:
    Vectors(const Vectors &) = delete;
    Vectors &operator=(const Vectors &) = delete;
    Vectors(Vectors &&o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    ~Vectors() { if (h_) jv_dataset_free(h_); }
    int64_t size() const { return jv_dataset_size(h_); }
    int dimension() const { return jv_dataset_dim(h_); }
    jv_dataset handle() const { return h_; }
    // fp32 rows changed in place (adopted device rows): the projection sketch no longer describes them (jv_dataset_invalidate_sketch)
    void invalidate_sketch() { jv_dataset_invalidate_sketch(h_); }
    /// BuildScoreProvider.diversityProviderFor: score(a[i], b[i]) for every pair, one launch
    std::vector<float> diversityScores(const std::vector<int32_t> &a, const std::vector<int32_t> &b, VectorSimilarityFunction vsf) const
    {
        std::vector<float> out(a.size());
        check(jv_score_pairs(h_, (int)vsf, a.data(), b.data(), (int)a.size(), out.data()));
        return out;
    }

protected:
    Vectors() = default;
    jv_dataset h_ = nullptr;
};

struct F32Vectors : Vectors {
    F32Vectors(const float *rows, int64_t n, int dim) { check(jv_dataset_register_f32(rows, n, dim, &h_)); }
};
struct PQVectors : Vectors {
    PQVectors(const uint8_t *codes, int64_t n, int dim, int M, int k, const float *codebooks, const float *centroid = nullptr)
    {
        check(jv_dataset_register_pq(codes, n, dim, M, k, codebooks, centroid, &h_));
    }
};
struct BQVectors : Vectors {
    BQVectors(const uint64_t *words, int64_t n, int dim) { check(jv_dataset_register_bq(words, n, dim, &h_)); }
};
struct NVQVectors : Vectors {
    NVQVectors(const uint8_t *bytes, const float *params, int64_t n, int dim, int nsub, const float *mean)
    {
        check(jv_dataset_register_nvq(bytes, params, n, dim, nsub, mean, &h_));
    }
};

/// ScoreFunction for one query (CompressedVectors.precomputedScoreFunctionFor / DefaultSearchScoreProvider.exact)
class ScoreFunction {
public:
    ScoreFunction(const Vectors &v, const float *query, VectorSimilarityFunction vsf) { check(jv_query_begin(v.handle(), query, (int)vsf, &q_)); }
    ScoreFunction(const ScoreFunction &) = delete;
    ScoreFunction &operator=(const ScoreFunction &) = delete;
    ~ScoreFunction() { if (q_) jv_query_end(q_); }
    /// the neighbour loop of one processNeighbors call / one rerank list: ONE kernel launch
    void similarityToBatch(const int32_t *ids, int n, float *out) const { check(jv_score_batch(q_, ids, n, out)); }
    std::vector<float> similarityToBatch(const std::vector<int32_t> &ids) const
    {
        std::vector<float> out(ids.size());
        similarityToBatch(ids.data(), (int)ids.size(), out.data());
        return out;
    }
    float similarityTo(int32_t node2) const
    {
        float s;
        similarityToBatch(&node2, 1, &s);
        return s;
    }

private:
    jv_query q_ = nullptr;
};

class GraphIndex {
public:
    GraphIndex(int32_t n, int degree, const int32_t *adj0, int32_t entryNode) { check(jv_graph_create(n, degree, adj0, entryNode, &g_)); }
    explicit GraphIndex(jv_graph g) : g_(g) {}
    GraphIndex(const GraphIndex &) = delete;
    GraphIndex &operator=(const GraphIndex &) = delete;
    GraphIndex(GraphIndex &&o) noexcept : g_(o.g_) { o.g_ = nullptr; }
    ~GraphIndex() { if (g_) jv_graph_free(g_); }
    void addLevel(const std::vector<int32_t> &nodeIds, const std::vector<int32_t> &adj) { check(jv_graph_add_level(g_, (int32_t)nodeIds.size(), nodeIds.data(), adj.data())); }
    jv_graph handle() const { return g_; }
    int32_t size() const { int32_t n = 0; check(jv_graph_info(g_, &n, nullptr, nullptr, nullptr)); return n; }
    int maxDegree() const { int d = 0; check(jv_graph_info(g_, nullptr, &d, nullptr, nullptr)); return d; }
    std::vector<int32_t> adjacency(int level = 0) const
    {
        int32_t cnt = 0;
        check(jv_graph_download(g_, level, nullptr, nullptr, &cnt));
        std::vector<int32_t> adj((size_t)cnt * maxDegree());
        check(jv_graph_download(g_, level, nullptr, adj.data(), &cnt));
        return adj;
    }

private:
    jv_graph g_ = nullptr;
};

/// SearchResult (base:graph/SearchResult.java) for a batch: nodes/scores [nq][topK] best first, -1 padded
struct SearchResult {
    std::vector<int32_t> nodes;
    std::vector<float> scores;
    int topK = 0;
    int64_t visitedCount = 0, expandedCount = 0, expandedCountBaseLayer = 0, rerankedCount = 0;
    double deviceMs = 0;
};

class GraphSearcher {
public:
    explicit GraphSearcher(const GraphIndex &g) : g_(g) {}
    SearchResult search(const Vectors &approx, const float *queries, int nq, VectorSimilarityFunction vsf, int topK, int rerankK, const Vectors *reranker = nullptr) const
    {
        SearchResult r;
        r.topK = topK;
        r.nodes.resize((size_t)nq * topK);
        r.scores.resize((size_t)nq * topK);
        jv_search_stats st;
        check(jv_graph_search_batch(g_.handle(), approx.handle(), reranker ? reranker->handle() : nullptr, (int)vsf, queries, nq, topK, rerankK, r.nodes.data(),
                                    r.scores.data(), &st));
        r.visitedCount = st.visited; r.expandedCount = st.expanded; r.expandedCountBaseLayer = st.expanded_base; r.rerankedCount = st.reranked; r.deviceMs = st.device_ms;
        return r;
    }

private:
    const GraphIndex &g_;
};

class GraphIndexBuilder {
public:
    GraphIndexBuilder(VectorSimilarityFunction vsf, int M, int beamWidth, float neighborOverflow, float alpha, bool addHierarchy, uint64_t seed = 0)
        : vsf_(vsf), p_{M, beamWidth, neighborOverflow, alpha, addHierarchy ? 1 : 0, seed, 0, -1} {}
    GraphIndex build(const F32Vectors &v)
    {
        jv_graph g = nullptr;
        check(jv_graph_build(v.handle(), (int)vsf_, &p_, &g, &deviceMs));
        return GraphIndex(g);
    }
    double deviceMs = 0;

private:
    VectorSimilarityFunction vsf_;
    jv_build_params p_;
};

}  // namespace jv
#endif
