"""Pins the CPU oracle (oracle/jv_oracle.c) before anything trusts it:
  (a) against the reference's own compiled kernels oracle/_ref/libjvector.so (SURVEY §8c),
  (b) against the siftsmall ground truth shipped with the reference,
  (c) against the known answers / tolerances of the reference's unit tests.
No GPU needed."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as o
from oracle_lib import bp, fp, ip, lp, wp
from recorded_ref import where_recorded

REL = 1e-4  # native-c:tests/test_similarity.cpp:101,140,172


@pytest.mark.parametrize("n", o.KERNEL_TEST_SIZES)
def test_similarity_vs_ref_make_vec(oracle, ref, n):
    a, b = o.make_vec(n, 0.7), o.make_vec(n, 1.3)
    for mine, theirs in ((oracle.jvo_dot_f32, ref.dot_product_f32), (oracle.jvo_l2_f32, ref.euclidean_f32),
                         (oracle.jvo_cosine_f32, ref.cosine_f32), (oracle.jvo_cosine_native_f32, ref.cosine_f32)):
        want = theirs(fp(a), 0, fp(b), 0, n)
        got = mine(fp(a), fp(b), n)
        assert abs(got - want) <= REL * abs(want) + 1e-30
    # offsets path (test_similarity.cpp:110-128) and the identities of :150-219
    ap, bpad = np.concatenate([np.ones(3, np.float32), a]), np.concatenate([np.ones(3, np.float32), b])
    assert abs(ref.dot_product_f32(fp(ap), 3, fp(bpad), 3, n) - oracle.jvo_dot_f32(fp(a), fp(b), n)) <= REL * abs(oracle.jvo_dot_f32(fp(a), fp(b), n))
    assert oracle.jvo_l2_f32(fp(a), fp(a), n) <= 1e-6 * n
    a2 = (2 * a).astype(np.float32)
    assert abs(oracle.jvo_cosine_f32(fp(a), fp(a2), n) - 1.0) <= 1e-5


def test_similarity_unit_1021(oracle, ref):
    # tests:vector/TestVectorizationProvider.java:37-61 — unit-norm 1021-dim, abs 1e-4
    rng = np.random.default_rng(7)
    for _ in range(20):
        v = o.random_unit_vectors(rng, 2, 1021)
        assert abs(oracle.jvo_dot_f32(fp(v[0]), fp(v[1]), 1021) - ref.dot_product_f32(fp(v[0]), 0, fp(v[1]), 0, 1021)) <= 1e-4
        assert abs(oracle.jvo_l2_f32(fp(v[0]), fp(v[1]), 1021) - ref.euclidean_f32(fp(v[0]), 0, fp(v[1]), 0, 1021)) <= 1e-4
        assert abs(oracle.jvo_cosine_f32(fp(v[0]), fp(v[1]), 1021) - ref.cosine_f32(fp(v[0]), 0, fp(v[1]), 0, 1021)) <= 1e-4


def test_score_map_and_key(oracle):
    assert oracle.jvo_score_from_raw(o.EUCLIDEAN, 3.0) == np.float32(0.25)
    assert oracle.jvo_score_from_raw(o.DOT_PRODUCT, 0.5) == np.float32(0.75)
    # NumericUtils.floatToSortableInt is monotone; ties go to the smaller node id (NodeQueue.java:125-137)
    xs = np.array([-np.inf, -3.5, -1e-30, -0.0, 0.0, 1e-30, 0.25, 1.0, np.inf], dtype=np.float32)
    ks = [oracle.jvo_topk_key(float(x), 5) for x in xs]
    assert all(ks[i] <= ks[i + 1] for i in range(len(ks) - 1))
    assert oracle.jvo_topk_key(0.5, 3) > oracle.jvo_topk_key(0.5, 4)
    for x in xs:
        k = oracle.jvo_topk_key(float(x), 123456)
        assert oracle.jvo_key_node(k) == 123456
        assert np.float32(oracle.jvo_key_score(k)).tobytes() == np.float32(x).tobytes()
    got = o.keys_of(xs, np.full(len(xs), 5))
    assert [int(g) for g in got] == ks


def test_siftsmall_ground_truth(oracle, sift):
    # C1 golden fixture: exact-L2 top-100 of the brute-force scorer + key must reproduce the shipped ivecs
    base, queries, gt = sift
    keys = np.empty(100, dtype=np.int64)
    mism = 0
    for qi in range(0, 100, 5):
        oracle.jvo_bruteforce_topk_f32(o.EUCLIDEAN, fp(base), base.shape[0], 128, fp(queries[qi]), 100, lp(keys))
        nodes = np.array([oracle.jvo_key_node(int(k)) for k in keys])
        if not np.array_equal(nodes, gt[qi]):
            # ties in integer-valued SIFT distances may be ordered differently in the shipped file: compare as sets
            # of (distance) and require identical distance sequences
            d_mine = ((base[nodes] - queries[qi]) ** 2).sum(1)
            d_gt = ((base[gt[qi]] - queries[qi]) ** 2).sum(1)
            assert np.array_equal(d_mine, d_gt)
            mism += 1
    assert mism <= 10


def _pq_setup(rng, n, dim, M, k=256):
    data = o.random_unit_vectors(rng, n, dim)
    cb, sizes, offsets = o.train_pq_numpy(rng, data[: min(n, 2000)], M, k, iters=2)
    return data, cb, sizes, offsets


def test_pq_layout_known(oracle):
    sizes = np.zeros(5, np.int32)
    offs = np.zeros(5, np.int32)
    oracle.jvo_pq_layout(13, 5, ip(sizes), ip(offs))
    assert sizes.tolist() == [3, 3, 3, 2, 2] and offs.tolist() == [0, 3, 6, 9, 11]


@pytest.mark.parametrize("dim,M", [(64, 8), (100, 7), (768, 96), (33, 33)])
def test_pq_vs_ref(oracle, ref, dim, M):
    rng = np.random.default_rng(dim * 131 + M)
    k = 256
    data, cb, sizes, offsets = _pq_setup(rng, 300, dim, M, k)
    q = o.random_unit_vectors(rng, 1, dim)[0]
    codes = o.encode_pq(oracle, cb, sizes, offsets, M, k, None, data)
    # codes are argmin of L2 with first-min-wins (ProductQuantization.java:507-520)
    for i in (0, 17):
        for m in (0, M - 1):
            cbm = cb[k * offsets[m]: k * (offsets[m] + sizes[m])].reshape(k, sizes[m])
            d = ((cbm - data[i, offsets[m]:offsets[m] + sizes[m]]) ** 2).sum(1)
            assert abs(d[codes[i, m]] - d.min()) <= 1e-6
    for metric, fn in ((o.DOT_PRODUCT, ref.calculate_partial_sums_dot_f32), (o.EUCLIDEAN, ref.calculate_partial_sums_euclidean_f32)):
        lut = np.empty(M * k, np.float32)
        oracle.jvo_pq_lut(fp(cb), ip(sizes), ip(offsets), M, k, None, fp(q), dim, metric, fp(lut))
        rl = np.empty(M * k, np.float32)
        for m in range(M):
            cbm = np.ascontiguousarray(cb[k * offsets[m]: k * (offsets[m] + sizes[m])])
            fn(fp(cbm), m, int(sizes[m]), k, fp(q), int(offsets[m]), fp(rl))
        w = where_recorded(rl)
        np.testing.assert_allclose(lut[w], rl[w], rtol=1e-5, atol=1e-6)
        for i in range(0, 300, 13):
            want = ref.assemble_and_sum_f32(fp(rl), k, bp(codes), i * M, M)
            got = oracle.jvo_pq_adc(fp(lut), k, bp(codes[i]), M)
            assert abs(got - want) <= 1e-5 * max(1.0, abs(want))
    # self magnitudes + decoded cosine
    mag = np.empty(M * k, np.float32)
    oracle.jvo_pq_self_magnitudes(fp(cb), ip(sizes), ip(offsets), M, k, fp(mag))
    rmag = np.empty(M * k, np.float32)
    for m in range(M):
        cbm = np.ascontiguousarray(cb[k * offsets[m]: k * (offsets[m] + sizes[m])])
        ref.calculate_partial_sums_self_magnitude_f32(fp(cbm), m, int(sizes[m]), k, fp(rmag))
    w = where_recorded(rmag)
    np.testing.assert_allclose(mag[w], rmag[w], rtol=1e-5, atol=1e-7)
    lut = np.empty(M * k, np.float32)
    oracle.jvo_pq_lut(fp(cb), ip(sizes), ip(offsets), M, k, None, fp(q), dim, o.DOT_PRODUCT, fp(lut))
    bmag = oracle.jvo_dot_f32(fp(q), fp(q), dim)
    for i in range(0, 300, 29):
        want = ref.pq_decoded_cosine_similarity_f32(bp(codes), i * M, M, k, fp(lut), fp(mag), bmag)
        got = oracle.jvo_pq_decoded_cosine(bp(codes[i]), M, k, fp(lut), fp(mag), bmag)
        assert abs(got - want) <= 1e-5
    # pair table (assemble_and_sum_pq_f32)
    if M * k * (k + 1) // 2 <= 4_000_000:
        table = np.empty(M * k * (k + 1) // 2, np.float32)
        oracle.jvo_pq_pair_table(fp(cb), ip(sizes), ip(offsets), M, k, o.EUCLIDEAN, fp(table))
        for i, j in ((0, 1), (5, 5), (7, 250)):
            want = ref.assemble_and_sum_pq_f32(fp(table), M, bp(codes), i * M, bp(codes), j * M, k)
            got = oracle.jvo_pq_pair_sum(fp(table), M, k, bp(codes[i]), bp(codes[j]))
            assert abs(got - want) <= 1e-5 * max(1.0, abs(want))
            direct = oracle.jvo_pq_diversity_direct(fp(cb), ip(sizes), ip(offsets), M, k, o.EUCLIDEAN, bp(codes[i]), bp(codes[j]))
            assert abs(1.0 / (1.0 + got) - direct) <= 1e-6


def test_pq_raw_equals_precomputed(oracle):
    # tests:quantization/TestCompressedVectors.java:230-256 — LUT path == direct path, abs 1e-6, centered or not
    rng = np.random.default_rng(11)
    for dim, M, centered in ((64, 4, False), (200, 13, True), (768, 96, False), (17, 8, True)):
        k = 256
        data, cb, sizes, offsets = _pq_setup(rng, 64, dim, M, k)
        cen = data.mean(0).astype(np.float32) if centered else None
        codes = o.encode_pq(oracle, cb, sizes, offsets, M, k, cen, data)
        q = o.random_unit_vectors(rng, 1, dim)[0]
        for metric in (o.EUCLIDEAN, o.DOT_PRODUCT, o.COSINE):
            lm = o.EUCLIDEAN if metric == o.EUCLIDEAN else o.DOT_PRODUCT
            lut = np.empty(M * k, np.float32)
            mag = np.empty(M * k, np.float32)
            oracle.jvo_pq_lut(fp(cb), ip(sizes), ip(offsets), M, k, fp(cen), fp(q), dim, lm, fp(lut))
            oracle.jvo_pq_self_magnitudes(fp(cb), ip(sizes), ip(offsets), M, k, fp(mag))
            cq = (q - cen).astype(np.float32) if centered else q
            bmag = oracle.jvo_dot_f32(fp(cq), fp(cq), dim)
            for i in range(0, 64, 7):
                a = oracle.jvo_pq_score_lut(metric, fp(lut), fp(mag), bmag, k, bp(codes[i]), M)
                b = oracle.jvo_pq_score_direct(fp(cb), ip(sizes), ip(offsets), M, k, fp(cen), fp(q), dim, metric, bp(codes[i]))
                assert abs(a - b) <= 2e-6, (dim, M, metric, a, b)


def test_assemble_and_sum_1000_trials(oracle, ref):
    # tests:vector/TestVectorizationProvider.java:64-91 (dataBase = 0, 32 offsets into a 256-vector, abs 1e-4)
    rng = np.random.default_rng(3)
    for _ in range(1000):
        v2 = rng.random(256, dtype=np.float32)
        offs = rng.integers(0, 256, 32).astype(np.uint8)
        want = float(v2[offs].astype(np.float64).sum())
        assert abs(oracle.jvo_pq_adc(fp(v2), 0, bp(offs), 32) - want) <= 1e-4
        assert abs(ref.assemble_and_sum_f32(fp(v2), 0, bp(offs), 0, 32) - want) <= 1e-4


def test_bq(oracle):
    rng = np.random.default_rng(5)
    for dim in (1, 63, 64, 65, 128, 1536, 1000):
        v = rng.standard_normal((2, dim)).astype(np.float32)
        v[0, 0] = 0.0  # strict > 0: zeros encode to 0 (BinaryQuantization.java:104)
        W = (dim + 63) // 64
        a = np.zeros(W, np.uint64)
        b = np.zeros(W, np.uint64)
        oracle.jvo_bq_encode(fp(v[0]), dim, wp(a))
        oracle.jvo_bq_encode(fp(v[1]), dim, wp(b))
        bits_a = np.unpackbits(a.view(np.uint8), bitorder="little")[:dim]
        assert np.array_equal(bits_a, (v[0] > 0).astype(np.uint8))
        hd = int(((v[0] > 0) != (v[1] > 0)).sum())
        assert oracle.jvo_hamming(wp(a), wp(b), W) == hd
        assert oracle.jvo_bq_score(wp(a), wp(b), W, dim) == np.float32(1) - np.float32(hd) / np.float32(dim)
    # tests:quantization/TestCompressedVectors.java:77 — BQ compressed size is 8 bytes at d = 64
    assert (64 + 63) // 64 * 8 == 8


def _shuffled(ref, q):
    s = q.copy()
    ref.nvq_shuffle_query_in_place_8bit(fp(s), len(s))
    return s


@pytest.mark.parametrize("n", [1, 5, 16, 63, 64, 65, 128, 384, 385, 1000])
def test_nvq_vs_ref(oracle, ref, n):
    rng = np.random.default_rng(100 + n)
    v = (rng.standard_normal(n) * 0.05).astype(np.float32)
    q = (rng.standard_normal(n) * 0.05).astype(np.float32)
    cen = (rng.standard_normal(n) * 0.01).astype(np.float32)
    minv, maxv = float(v.min()), float(v.max())
    if n == 1:
        minv, maxv = float(v[0]) - 0.01, float(v[0]) + 0.01
    for alpha in (1e-2, 1e-6, 3.0, 7.3, 19.0):
        by = np.empty(n, np.uint8)
        rby = np.empty(n, np.uint8)
        oracle.jvo_nvq_quantize_8bit(fp(v), n, alpha, 0.0, minv, maxv, bp(by))
        ref.nvq_quantize_8bit(fp(v), n, alpha, 0.0, minv, maxv, bp(rby))
        assert np.array_equal(by, rby), (n, alpha, np.flatnonzero(by != rby))
        lo, rlo = oracle.jvo_nvq_loss(fp(v), n, alpha, 0.0, minv, maxv, 8), ref.nvq_loss(fp(v), n, alpha, 0.0, minv, maxv, 8)
        assert abs(lo - rlo) <= 1e-5 * abs(rlo) + 1e-12
        # distances: the reference kernels want their private lane order (SURVEY Appendix B)
        want = ref.nvq_dot_product_8bit(fp(_shuffled(ref, q)), bp(by), n, alpha, 0.0, minv, maxv)
        got = oracle.jvo_nvq_dot_8bit(fp(q), bp(by), n, alpha, 0.0, minv, maxv)
        scale = float(np.abs(q).sum() * max(abs(minv), abs(maxv))) + 1e-12
        assert abs(got - want) <= 1e-5 * scale
        want = ref.nvq_square_l2_distance_8bit(fp(_shuffled(ref, q)), bp(by), n, alpha, 0.0, minv, maxv)
        got = oracle.jvo_nvq_l2_8bit(fp(q), bp(by), n, alpha, 0.0, minv, maxv)
        assert abs(got - want) <= 1e-5 * abs(want) + 1e-12
        pk = ref.nvq_cosine_8bit_packed(fp(_shuffled(ref, q)), bp(by), n, alpha, 0.0, minv, maxv, fp(_shuffled(ref, cen)))
        w0 = np.array([pk & 0xffffffff], dtype=np.uint32).view(np.float32)[0]
        w1 = np.array([(pk >> 32) & 0xffffffff], dtype=np.uint32).view(np.float32)[0]
        out = np.empty(2, np.float32)
        oracle.jvo_nvq_cosine_8bit(fp(q), bp(by), n, alpha, 0.0, minv, maxv, fp(cen), fp(out))
        assert abs(out[0] - w0) <= 1e-5 * scale and abs(out[1] - w1) <= 1e-5 * abs(w1) + 1e-12
    ul, rul = oracle.jvo_nvq_uniform_loss(fp(v), n, minv, maxv, 8), ref.nvq_uniform_loss(fp(v), n, minv, maxv, 8)
    assert abs(ul - rul) <= 1e-5 * abs(rul) + 1e-12


@pytest.mark.parametrize("n", [5, 31, 32, 33, 64, 384, 1000])
def test_nvq_loss_lane_orders_vs_ref(oracle, ref, n):
    # the loss sums are defined up to summation order (scalar provider: sequential; Panama / native: lane accumulators); the
    # 32-lane order the device uses stays inside the reference's own agreement band and the search it drives picks the same
    # growth rate as the sequential order except on near-ties
    rng = np.random.default_rng(300 + n)
    v = (rng.standard_normal(n) * 0.05).astype(np.float32)
    minv, maxv = float(v.min()), float(v.max())
    for alpha in (1e-6, 1e-2, 3.000001, 7.3, 19.000001):
        rlo = ref.nvq_loss(fp(v), n, alpha, 0.0, minv, maxv, 8)
        for lanes in (1, 8, 16, 32):
            lo = oracle.jvo_nvq_loss_lanes(fp(v), n, alpha, 0.0, minv, maxv, 8, lanes)
            assert abs(lo - rlo) <= 1e-5 * abs(rlo) + 1e-12, (lanes, alpha)
    rul = ref.nvq_uniform_loss(fp(v), n, minv, maxv, 8)
    for lanes in (1, 8, 16, 32):
        assert abs(oracle.jvo_nvq_uniform_loss_lanes(fp(v), n, minv, maxv, 8, lanes) - rul) <= 1e-5 * abs(rul) + 1e-12
    assert oracle.jvo_nvq_loss_lanes(fp(v), n, 2.5, 0.0, minv, maxv, 8, 1) == oracle.jvo_nvq_loss(fp(v), n, 2.5, 0.0, minv, maxv, 8)
    p1, p32 = np.empty(4, np.float32), np.empty(4, np.float32)
    b1, b32 = np.empty(n, np.uint8), np.empty(n, np.uint8)
    oracle.jvo_nvq_encode_subvector_lanes(fp(v), n, 1, 1, fp(p1), bp(b1))
    oracle.jvo_nvq_encode_subvector_lanes(fp(v), n, 1, 32, fp(p32), bp(b32))
    assert np.array_equal(p1[[0, 1, 3]], p32[[0, 1, 3]]) and abs(p1[2] - p32[2]) <= 0.11  # at most one grid step apart


def test_nvq_dequant_elementwise_exact(oracle, ref):
    # per-element dequantisation is bit-reproducible: n = 1 calls of the reference kernel isolate one element
    rng = np.random.default_rng(9)
    one = np.ones(1, np.float32)
    for _ in range(200):
        minv, maxv = -abs(rng.standard_normal()) * 0.1 - 1e-3, abs(rng.standard_normal()) * 0.1 + 1e-3
        alpha = float(rng.choice([1e-2, 1e-6, 2.0, 9.1]))
        b = np.array([rng.integers(0, 256)], dtype=np.uint8)
        want = ref.nvq_dot_product_8bit(fp(one), bp(b), 1, alpha, 0.0, minv, maxv)
        got = oracle.jvo_nvq_dequant(int(b[0]), alpha, 0.0, minv, maxv)
        assert np.float32(got).tobytes() == np.float32(want).tobytes()


def test_nvq_known_sizes_and_error_bounds(oracle):
    # tests:quantization/TestCompressedVectors.java:92-128 — compressed sizes 4 + sum(dims + 28)
    def size(d, nsub):
        sizes, _ = o.pq_layout(d, nsub)
        return 4 + int(sum(s + 28 for s in sizes))
    assert (size(64, 1), size(64, 2), size(65, 1)) == (96, 124, 97)
    # :171-228 testNVQEncodings — mean |NVQ score - exact| bounds
    rng = np.random.default_rng(21)
    for dim in (256, 512):
        for nsub in (1, 2, 4):
            for learn in (0, 1):
                n = 40
                data = o.random_unit_vectors(rng, n, dim)
                mean = data.mean(0).astype(np.float32)
                params = np.empty((n, nsub, 4), np.float32)
                bys = np.empty((n, dim), np.uint8)
                for i in range(n):
                    oracle.jvo_nvq_encode(fp(data[i]), fp(mean), dim, nsub, learn, fp(params[i]), bp(bys[i]))
                q = o.random_unit_vectors(rng, 1, dim)[0]
                for metric, tol in ((o.EUCLIDEAN, 1.0), (o.DOT_PRODUCT, 4.0), (o.COSINE, 10.0)):
                    err = 0.0
                    for i in range(n):
                        a = oracle.jvo_nvq_score(metric, fp(q), fp(mean), dim, nsub, fp(params[i]), bp(bys[i]))
                        e = oracle.jvo_compare_f32(metric, fp(q), fp(data[i]), dim)
                        err += abs(a - e)
                    assert err / n <= 0.0005 * (dim / 256.0) * tol, (dim, nsub, learn, metric, err / n)


def test_scorer_contexts_port_equals_ref(oracle, ref):
    rng = np.random.default_rng(33)
    n, dim, M, k, nsub = 200, 96, 12, 256, 2
    data, cb, sizes, offsets = _pq_setup(rng, n, dim, M, k)
    codes = o.encode_pq(oracle, cb, sizes, offsets, M, k, None, data)
    mean = data.mean(0).astype(np.float32)
    params = np.empty((n, nsub, 4), np.float32)
    bys = np.empty((n, dim), np.uint8)
    for i in range(n):
        oracle.jvo_nvq_encode(fp(data[i]), fp(mean), dim, nsub, 1, fp(params[i]), bp(bys[i]))
    q = o.random_unit_vectors(rng, 1, dim)[0]
    metrics, kinds = (o.EUCLIDEAN, o.DOT_PRODUCT, o.COSINE), ("f32", "pq", "nvq")

    def scores(ref_so):
        """[metric][kind][node] scores of the oracle's scorers, their arithmetic routed through ref_so (None: the oracle's own)"""
        assert oracle.jvo_use_ref(ref_so) == 0
        out = np.empty((len(metrics), len(kinds), n), np.float32)
        for a, metric in enumerate(metrics):
            ctxs = [oracle.jvo_scorer_f32(metric, fp(data), n, dim, fp(q)),
                    oracle.jvo_scorer_pq(metric, fp(cb), M, k, dim, None, bp(codes), n, fp(q)),
                    oracle.jvo_scorer_nvq(metric, fp(mean), dim, nsub, fp(params), bp(bys), n, fp(q))]
            for b, c in enumerate(ctxs):
                out[a, b] = [oracle.jvo_scorer_score(c, i) for i in range(n)]
                oracle.jvo_scorer_free(c)
        oracle.jvo_use_ref(None)
        return out
    port = scores(None)
    via_ref = ref.capture(lambda: scores(o.REF_SO.encode()))
    for a in range(len(metrics)):
        for b in range(len(kinds)):
            np.testing.assert_allclose(port[a, b], via_ref[a, b], rtol=1e-5, atol=1e-6)
    # the f32 scorer equals jvo_compare
    assert port[metrics.index(o.DOT_PRODUCT), kinds.index("f32")][3] == oracle.jvo_compare_f32(o.DOT_PRODUCT, fp(q), fp(data[3]), dim)


def test_retain_diverse_known_answer(oracle):
    # tests:graph/TestVectorGraph.java:457-526 testDiversity: 7 unit-circle vectors, DOT_PRODUCT, M=4(degree 2*... ),
    # restated at the level of retainDiverse: with alpha = 1.0 a candidate closer to a selected neighbour than to the
    # base node is dropped.
    ang = np.array([0.5, 0.75, 0.2, 0.9, 0.8, 0.77, 0.6]) * np.pi
    vec = np.stack([np.cos(ang), np.sin(ang)], 1).astype(np.float32)
    basei = 1  # node 1 (0.75π): candidates are the others, sorted by score desc
    others = [i for i in range(7) if i != basei]
    sc = np.array([oracle.jvo_compare_f32(o.DOT_PRODUCT, fp(vec[basei]), fp(vec[i]), 2) for i in others], np.float32)
    order = np.argsort(-sc, kind="stable")
    nodes = np.array(others, np.int32)[order]
    scores = np.ascontiguousarray(sc[order])
    nc = len(nodes)
    pair = np.empty((nc, nc), np.float32)
    for i in range(nc):
        for j in range(nc):
            pair[i, j] = oracle.jvo_compare_f32(o.DOT_PRODUCT, fp(vec[nodes[i]]), fp(vec[nodes[j]]), 2)
    sel = np.zeros(nc, np.uint8)
    cnt = oracle.jvo_retain_diverse(fp(scores), ip(nodes), nc, fp(pair), 4, 1.0, bp(sel))
    kept = nodes[sel.astype(bool)].tolist()
    # nearest on each side survive; nodes shadowed by a closer selected neighbour do not
    assert kept == [5, 6] and cnt == 2


def test_graph_build_and_search_siftsmall(oracle, sift):
    # C1: graph search over siftsmall (M=16, ef=100, overflow 1.2, alpha 1.2, no hierarchy: SiftSmall.java:86-93)
    base, queries, gt = sift
    n = 2000  # a slice keeps the CPU suite fast; ground truth recomputed for the slice
    b = np.ascontiguousarray(base[:n])
    adj = np.empty((n, 16), np.int32)
    entry = oracle.jvo_graph_build_f32(o.EUCLIDEAN, fp(b), n, 128, 16, 100, 1.2, 1.2, ip(adj))
    assert (adj < n).all() and (adj >= -1).all()
    deg = (adj >= 0).sum(1)
    assert deg.max() <= 16 and deg.mean() > 8
    g = o.make_graph(adj, entry)
    hits = 0
    nodes = np.empty(10, np.int32)
    scores = np.empty(10, np.float32)
    st = o.Stats()
    for qi in range(50):
        sf = oracle.jvo_scorer_f32(o.EUCLIDEAN, fp(b), n, 128, fp(queries[qi]))
        c = oracle.jvo_graph_search(C.byref(g), sf, None, 10, 100, ip(nodes), fp(scores), C.byref(st))
        oracle.jvo_scorer_free(sf)
        assert c == 10 and st.visited > 100
        assert all(scores[i] >= scores[i + 1] for i in range(9))
        d = ((b - queries[qi]) ** 2).sum(1)
        truth = set(np.argsort(d, kind="stable")[:10].tolist())
        hits += len(truth & set(nodes.tolist()))
    assert hits / 500.0 > 0.9  # tests:graph/TestVectorGraph.java:672


def test_builder_known_answer_diversity(oracle):
    # tests:graph/TestVectorGraph.java:457-526 testDiversity — golden neighbour lists of GraphIndexBuilder(DOT_PRODUCT, M=4, beamWidth=10,
    # neighborOverflow=1.0, alpha=1.0) over 7 unit-circle vectors, checked after each insert. The oracle builder inserts sequentially, so
    # building the first n vectors reproduces the state after addGraphNode(n-1).
    ang = np.array([0.5, 0.75, 0.2, 0.9, 0.8, 0.77, 0.6]) * np.pi
    vec = np.ascontiguousarray(np.stack([np.cos(ang), np.sin(ang)], 1), dtype=np.float32)
    expected = {
        3: {0: [1, 2], 1: [0], 2: [0]},
        4: {0: [1, 2], 1: [0, 3], 2: [0], 3: [1]},
        5: {0: [1, 2], 1: [0, 3, 4], 2: [0], 3: [1, 4], 4: [1, 3]},
        6: {0: [1, 2], 1: [0, 3, 4, 5], 2: [0], 3: [1, 4], 4: [1, 3, 5], 5: [1, 4]},
    }
    for n, want in expected.items():
        adj = np.empty((n, 4), np.int32)
        oracle.jvo_graph_build_f32(o.DOT_PRODUCT, fp(vec), n, 2, 4, 10, 1.0, 1.0, ip(adj))
        for node, nbrs in want.items():
            got = sorted(int(x) for x in adj[node] if x >= 0)
            assert got == nbrs, (n, node, got, nbrs)


def test_builder_known_answer_fallback_and_3d(oracle):
    # tests:graph/TestVectorGraph.java:533-611 — EUCLIDEAN, M=2, beamWidth=10, overflow 1.0, alpha 1.0
    # testDiversityFallback: a new closer neighbour displaces the farthest one although every neighbour stays diverse
    v = np.array([[0, 0, 0], [0, 10, 0], [0, 0, 20], [10, 0, 0], [0, 4, 0]], np.float32)
    for n, want in ((3, {0: [1, 2], 1: [0], 2: [0]}), (4, {0: [1, 3], 1: [0], 2: [0], 3: [0]})):
        adj = np.empty((n, 2), np.int32)
        oracle.jvo_graph_build_f32(o.EUCLIDEAN, fp(np.ascontiguousarray(v[:n])), n, 3, 2, 10, 1.0, 1.0, ip(adj))
        for node, nbrs in want.items():
            assert sorted(int(x) for x in adj[node] if x >= 0) == nbrs, ("fallback", n, node, adj[node].tolist())
    # testDiversity3d: a neighbour BECOMES non-diverse when a newer, better neighbour arrives
    v = np.array([[0, 0, 0], [0, 10, 0], [0, 0, 20], [0, 9, 0]], np.float32)
    for n, want in ((3, {0: [1, 2], 1: [0], 2: [0]}), (4, {0: [2, 3], 1: [0, 3], 2: [0], 3: [0, 1]})):
        adj = np.empty((n, 2), np.int32)
        oracle.jvo_graph_build_f32(o.EUCLIDEAN, fp(np.ascontiguousarray(v[:n])), n, 3, 2, 10, 1.0, 1.0, ip(adj))
        for node, nbrs in want.items():
            assert sorted(int(x) for x in adj[node] if x >= 0) == nbrs, ("3d", n, node, adj[node].tolist())


def test_warp_order_scorers_agree_with_sequential_order(oracle):
    # order 1 (the kernels' summation order) is the same arithmetic as order 0: every score within 1e-5 relative, BQ identical
    rng = np.random.default_rng(91)
    for dim, M, nsub in ((64, 16, 2), (100, 7, 3), (768, 96, 2), (33, 33, 1)):
        n = 120
        data = o.random_unit_vectors(rng, n, dim)
        q = o.random_unit_vectors(rng, 1, dim)[0]
        cb, sizes, offsets = o.train_pq_numpy(rng, data, M, 256, iters=1)
        cen = data.mean(0).astype(np.float32)
        codes = o.encode_pq(oracle, cb, sizes, offsets, M, 256, cen, data)
        params = np.empty((n, nsub, 4), np.float32)
        bys = np.empty((n, dim), np.uint8)
        for i in range(n):
            oracle.jvo_nvq_encode(fp(data[i]), fp(cen), dim, nsub, 1, fp(params[i]), bp(bys[i]))
        words = np.zeros((n, (dim + 63) // 64), np.uint64)
        for i in range(n):
            oracle.jvo_bq_encode(fp(data[i]), dim, wp(words[i]))
        for metric in (o.EUCLIDEAN, o.DOT_PRODUCT, o.COSINE):
            for mk in (lambda: oracle.jvo_scorer_f32(metric, fp(data), n, dim, fp(q)),
                       lambda: oracle.jvo_scorer_pq(metric, fp(cb), M, 256, dim, fp(cen), bp(codes), n, fp(q)),
                       lambda: oracle.jvo_scorer_nvq(metric, fp(cen), dim, nsub, fp(params), bp(bys), n, fp(q)),
                       lambda: oracle.jvo_scorer_bq(wp(words), n, dim, fp(q))):
                sf = mk()
                a = np.array([oracle.jvo_scorer_score(sf, i) for i in range(n)], np.float32)
                oracle.jvo_scorer_set_order(sf, 1)
                b = np.array([oracle.jvo_scorer_score(sf, i) for i in range(n)], np.float32)
                oracle.jvo_scorer_free(sf)
                assert np.abs(a - b).max() <= 1e-5 * max(1e-2, float(np.abs(a).max())), (dim, metric)
        assert oracle.jvo_compare_f32_warp(o.DOT_PRODUCT, fp(q), fp(data[3]), dim) == pytest.approx(oracle.jvo_compare_f32(o.DOT_PRODUCT, fp(q), fp(data[3]), dim), rel=1e-5)
