"""The projection sketch of fp32 DOT_PRODUCT walks (sketch.cu, search.cu): its bound never undercuts the exact score, searches give
the same bits with and without it while reading fewer rows, and data it cannot help (i.i.d. rows) keeps the plain walk.
Data sets are 300k x 256 fp32 (307 MB): the sketch is built only for rows that do not fit twice in L2."""
import ctypes as C
import os

import numpy as np
import pytest

N, DIM, LAT = 300_000, 256, 32
DOT = None


def _jv():
    import jvector_b200 as jv
    global DOT
    jv.init(0)
    DOT = jv.VectorSimilarityFunction.DOT_PRODUCT
    return jv


def latent_rows(rng, n, dim, noise=0.25):
    """the shape of bench.py's latent rows: a 32-factor Gaussian model plus isotropic noise, normalised"""
    a = rng.standard_normal((LAT, dim), dtype=np.float32) / np.float32(np.sqrt(LAT))
    x = rng.standard_normal((n, LAT), dtype=np.float32) @ a
    x += noise * rng.standard_normal((n, dim), dtype=np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    return x


def iid_rows(rng, n, dim):
    x = rng.standard_normal((n, dim), dtype=np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    return x


def sketch_of(vec):
    from jvector_b200 import _native as nat
    lib = nat.load()
    st, cap = C.c_int(), C.c_double()
    nat.check(lib.jv_dataset_f32_sketch(vec._h, C.byref(st), C.byref(cap), None, None, None))
    if st.value != 1:
        return st.value, cap.value, None
    n, stride = vec.size(), (vec.dimension() + 3) & ~3
    basis = np.empty((32, stride), np.float32)
    proj = np.empty((n, 32), np.float32)
    norms = np.empty((n, 2), np.float32)
    nat.check(lib.jv_dataset_f32_sketch(vec._h, None, None, nat.fp(basis), nat.fp(proj), nat.fp(norms)))
    return st.value, cap.value, (basis, proj, norms)


def ring_graph(n, degree=8):
    """any graph triggers the sketch build: neighbours i +- 1..degree/2"""
    jv = _jv()
    off = np.concatenate([np.arange(1, degree // 2 + 1), -np.arange(1, degree // 2 + 1)])
    adj = (np.arange(n)[:, None] + off[None, :]) % n
    return jv.GraphIndex(adj.astype(np.int32), 0)


def search(jv, graph, vec, queries, sketch, topK=10, rerankK=100):
    old = os.environ.get("JV_F32_SKETCH")
    os.environ["JV_F32_SKETCH"] = "1" if sketch else "0"
    try:
        return jv.GraphSearcher(graph).search(vec, queries, DOT, topK, rerankK)
    finally:
        if old is None:
            del os.environ["JV_F32_SKETCH"]
        else:
            os.environ["JV_F32_SKETCH"] = old


@pytest.fixture(scope="module")
def latent_world():
    jv = _jv()
    rng = np.random.default_rng(7)
    x = latent_rows(rng, N + 200, DIM)
    data, queries = np.ascontiguousarray(x[:N]), np.ascontiguousarray(x[N:])
    vec = jv.F32Vectors(data)
    gi = jv.GraphIndexBuilder(DOT, M=16, beamWidth=100).build(vec)
    return jv, data, queries, vec, gi


def sketch_bound(basis, proj, norms, q, ids):
    """the kernel's bound (search.cu: sketch_prepare + the bound pass), mapped like a DOT_PRODUCT score"""
    b = basis.astype(np.float64)
    qd = np.zeros(basis.shape[1], np.float64)
    qd[:len(q)] = q
    a = b @ qd
    g = b @ b.T
    qq = qd @ qd
    qperp = np.float32(np.sqrt(max(0.0, qq - 2 * (a @ a) + a @ g @ a)))
    d = proj[ids] @ a.astype(np.float32)
    raw = d + qperp * norms[ids, 0] + np.float32(1e-3) * np.float32(np.sqrt(qq)) * norms[ids, 1]
    return (np.float32(1) + raw.astype(np.float32)) / np.float32(2)


def check_bound(jv, data, vec, queries, pairs_per_query, rng):
    st, _, sk = sketch_of(vec)
    assert st == 1
    basis, proj, norms = sk
    checked = 0
    for q in queries:
        exact_all = data @ q
        top = np.argpartition(-exact_all, 200)[:200]
        ids = np.unique(np.concatenate([top, rng.integers(0, len(data), pairs_per_query - 200)])).astype(np.int32)
        exact = vec.score_function_for(q, DOT).similarityToBatch(ids)  # the device row scorer the walk uses
        ub = sketch_bound(basis, proj, norms, q, ids)
        bad = np.nonzero(ub < exact)[0]
        assert len(bad) == 0, "bound below the exact score for rows %s: %s < %s" % (ids[bad[:5]], ub[bad[:5]], exact[bad[:5]])
        checked += len(ids)
    return checked


@pytest.mark.gpu
def test_sketch_bound_never_below_exact_score(latent_world):
    jv, data, queries, vec, gi = latent_world
    rng = np.random.default_rng(11)
    search(jv, gi, vec, queries[:4], True)  # builds the sketch
    checked = check_bound(jv, data, vec, queries[:100], 5000, rng)
    # a quarter i.i.d. rows (far from the basis) and row norms spread over two decades, in one data set whose sketch is still built
    x = np.concatenate([latent_rows(rng, 3 * N // 4, DIM), iid_rows(rng, N - 3 * N // 4, DIM)])
    x *= np.exp(rng.uniform(np.log(0.1), np.log(10.0), (N, 1))).astype(np.float32)
    q = np.concatenate([latent_rows(rng, 50, DIM), iid_rows(rng, 50, DIM)]) * np.float32(3.0)
    v2 = jv.F32Vectors(np.ascontiguousarray(x))
    search(jv, ring_graph(N), v2, q[:2], True)
    checked += check_bound(jv, x, v2, q, 5000, rng)
    assert checked >= 900_000


@pytest.mark.gpu
def test_sketch_search_results_identical(latent_world):
    import oracle_lib as o
    from oracle_lib import fp, ip
    jv, data, queries, vec, gi = latent_world
    off = search(jv, gi, vec, queries, False)
    on = search(jv, gi, vec, queries, True)
    assert sketch_of(vec)[0] == 1
    assert np.array_equal(off.nodes, on.nodes)
    assert np.array_equal(off.scores.view(np.int32), on.scores.view(np.int32))
    assert (off.visitedCount, off.expandedCount) == (on.visitedCount, on.expandedCount)
    # and the traversal is still the reference's, in the kernels' summation order
    L = o.load()
    _, adj = gi.level(0)
    g = o.make_graph(adj, gi.info()["entry_node"])
    nodes, scores = np.empty(10, np.int32), np.empty(10, np.float32)
    for i in range(8):
        sf = L.jvo_scorer_f32(o.DOT_PRODUCT, fp(data), N, DIM, fp(queries[i]))
        L.jvo_scorer_set_order(sf, 1)
        L.jvo_graph_search(C.byref(g), sf, None, 10, 100, ip(nodes), fp(scores), None)
        L.jvo_scorer_free(sf)
        assert np.array_equal(nodes, on.nodes[i]) and np.array_equal(scores.view(np.int32), on.scores[i].view(np.int32)), i


@pytest.mark.gpu
def test_sketch_reads_fewer_rows_than_visited(latent_world):
    from jvector_b200 import _native as nat
    jv, data, queries, vec, gi = latent_world
    lib = nat.load()
    r0 = lib.jv_search_rows_read()
    off = search(jv, gi, vec, queries, False)
    r1 = lib.jv_search_rows_read()
    on = search(jv, gi, vec, queries, True)
    r2 = lib.jv_search_rows_read()
    assert r1 - r0 == off.visitedCount  # without the sketch every visited row is read
    assert r2 - r1 < 0.8 * on.visitedCount, (r2 - r1, on.visitedCount)


@pytest.mark.gpu
def test_sketch_skipped_on_iid_rows():
    from jvector_b200 import _native as nat
    jv = _jv()
    rng = np.random.default_rng(5)
    x = iid_rows(rng, N + 20, DIM)
    vec = jv.F32Vectors(np.ascontiguousarray(x[:N]))
    lib = nat.load()
    r0 = lib.jv_search_rows_read()
    res = search(jv, ring_graph(N), vec, x[N:], True)
    st, cap, _ = sketch_of(vec)
    assert st == -1 and cap < 0.5, (st, cap)
    assert lib.jv_search_rows_read() - r0 == res.visitedCount
    # invalidating forgets the decision; the next search decides again
    nat.check(lib.jv_dataset_invalidate_sketch(vec._h))
    assert sketch_of(vec)[0] == 0
    search(jv, ring_graph(N), vec, x[N:N + 2], True)
    assert sketch_of(vec)[0] == -1
