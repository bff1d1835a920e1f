"""CPU-side checks of the C-ABI library: it loads without a GPU, exports every symbol include/jvector_b200.h declares,
the 24 legacy libjvector.so symbols compute what the reference's own kernels compute, and the GPU group fails loudly
(no CPU fallback) when no device is present."""
import os
import re
import subprocess

import numpy as np
import pytest

import oracle_lib as o
from oracle_lib import bp, fp
from recorded_ref import where_recorded

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from jvector_b200 import _native as nat
    if not os.path.exists(nat.SO):
        from jvector_b200 import build
        build.build()
    return nat.load()


def test_header_symbols_exported(lib):
    from jvector_b200 import _native as nat
    hdr = open(os.path.join(ROOT, "include", "jvector_b200.h")).read()
    declared = set(re.findall(r"JV_API\s+[\w\s\*]+?\b(\w+)\s*\(", hdr))
    assert len(declared) >= 24 + 30
    out = subprocess.check_output(["nm", "-D", "--defined-only", nat.SO], text=True)
    # " i " = GNU indirect function: the multi-versioned similarity symbols (legacy_simd.cpp) resolve through dlsym like any other
    exported = {line.split()[-1] for line in out.splitlines() if " T " in line or " i " in line}
    missing = declared - exported
    assert not missing, missing
    bound = {name for name, _, _ in nat.SYMBOLS}
    assert declared == bound, declared ^ bound
    # the 24 symbols of the reference ABI (native-c:src/jvector_simd_kernel_list.h:35-61 + jvector_simd.h:47,53)
    legacy = ["cosine_f32", "dot_product_f32", "euclidean_f32", "add_in_place_f32", "add_scalar_in_place_f32", "sub_in_place_f32",
              "sub_scalar_in_place_f32", "max_f32", "min_in_place_f32", "assemble_and_sum_f32", "assemble_and_sum_pq_f32",
              "pq_decoded_cosine_similarity_f32", "calculate_partial_sums_dot_f32", "calculate_partial_sums_euclidean_f32",
              "calculate_partial_sums_self_magnitude_f32", "nvq_quantize_8bit", "nvq_loss", "nvq_uniform_loss",
              "nvq_square_l2_distance_8bit", "nvq_dot_product_8bit", "nvq_cosine_8bit_packed", "nvq_shuffle_query_in_place_8bit",
              "jvector_simd_get_active_isa", "jvector_simd_get_max_isa_env"]
    assert set(legacy) <= exported


def test_same_symbols_as_reference_library(lib, ref):
    from jvector_b200 import _native as nat
    theirs = ref.capture(lambda: sorted(subprocess.check_output(["nm", "-D", "--defined-only", o.REF_SO], text=True).splitlines()))
    ours = subprocess.check_output(["nm", "-D", "--defined-only", nat.SO], text=True)
    t = {l.split()[-1] for l in theirs if " T " in l}
    u = {l.split()[-1] for l in ours.splitlines() if " T " in l or " i " in l}
    assert t <= u, t - u


def test_diagnostics(lib):
    assert lib.jvector_simd_get_active_isa() == b"sm_100a"
    assert lib.jv_version().startswith(b"jvector-b200")


@pytest.mark.parametrize("n", o.KERNEL_TEST_SIZES)
def test_legacy_similarity_and_elementwise(lib, ref, n):
    a, b = o.make_vec(n, 0.7), o.make_vec(n, 1.3)
    for name in ("dot_product_f32", "euclidean_f32", "cosine_f32"):
        want = getattr(ref, name)(fp(a), 0, fp(b), 0, n)
        got = getattr(lib, name)(fp(a), 0, fp(b), 0, n)
        assert abs(got - want) <= 1e-4 * abs(want) + 1e-30
    ap = np.concatenate([np.full(3, 9.0, np.float32), a])
    bpad = np.concatenate([np.full(3, 9.0, np.float32), b])
    assert abs(lib.dot_product_f32(fp(ap), 3, fp(bpad), 3, n) - lib.dot_product_f32(fp(a), 0, fp(b), 0, n)) == 0
    # element-wise (native-c:tests/test_elementwise.cpp:49-187)
    for name in ("add_in_place_f32", "sub_in_place_f32", "min_in_place_f32"):
        x, y = a.copy(), a.copy()
        getattr(lib, name)(fp(x), fp(b), n)
        getattr(ref, name)(fp(y), fp(b), n)
        assert np.array_equal(x, y)
    for name in ("add_scalar_in_place_f32", "sub_scalar_in_place_f32"):
        x, y = a.copy(), a.copy()
        getattr(lib, name)(fp(x), 2.5, n)
        getattr(ref, name)(fp(y), 2.5, n)
        assert np.array_equal(x, y)
    assert lib.max_f32(fp(a), n) == ref.max_f32(fp(a), n) == a.max()


def test_legacy_pq(lib, ref, oracle):
    rng = np.random.default_rng(1)
    dim, M, k = 96, 12, 256
    data = o.random_unit_vectors(rng, 300, dim)
    cb, sizes, offsets = o.train_pq_numpy(rng, data, M, k, iters=1)
    codes = o.encode_pq(oracle, cb, sizes, offsets, M, k, None, data[:50])
    q = o.random_unit_vectors(rng, 1, dim)[0]
    for name in ("calculate_partial_sums_dot_f32", "calculate_partial_sums_euclidean_f32"):
        x, y = np.zeros(M * k, np.float32), np.zeros(M * k, np.float32)
        for m in range(M):
            cbm = np.ascontiguousarray(cb[k * offsets[m]: k * (offsets[m] + sizes[m])])
            getattr(lib, name)(fp(cbm), m, int(sizes[m]), k, fp(q), int(offsets[m]), fp(x))
            getattr(ref, name)(fp(cbm), m, int(sizes[m]), k, fp(q), int(offsets[m]), fp(y))
        w = where_recorded(y)
        np.testing.assert_allclose(x[w], y[w], rtol=1e-5, atol=1e-6)
        for i in range(50):
            assert abs(lib.assemble_and_sum_f32(fp(x), k, bp(codes), i * M, M) - ref.assemble_and_sum_f32(fp(y), k, bp(codes), i * M, M)) <= 1e-5
    mag, rmag = np.zeros(M * k, np.float32), np.zeros(M * k, np.float32)
    for m in range(M):
        cbm = np.ascontiguousarray(cb[k * offsets[m]: k * (offsets[m] + sizes[m])])
        lib.calculate_partial_sums_self_magnitude_f32(fp(cbm), m, int(sizes[m]), k, fp(mag))
        ref.calculate_partial_sums_self_magnitude_f32(fp(cbm), m, int(sizes[m]), k, fp(rmag))
    w = where_recorded(rmag)
    np.testing.assert_allclose(mag[w], rmag[w], rtol=1e-5)
    for i in range(50):
        assert abs(lib.pq_decoded_cosine_similarity_f32(bp(codes), i * M, M, k, fp(x), fp(mag), 1.0) -
                   ref.pq_decoded_cosine_similarity_f32(bp(codes), i * M, M, k, fp(x), fp(mag), 1.0)) <= 1e-5
    table = np.empty(M * k * (k + 1) // 2, np.float32)
    oracle.jvo_pq_pair_table(fp(cb), o.ip(sizes), o.ip(offsets), M, k, o.EUCLIDEAN, fp(table))
    for i, j in ((0, 1), (3, 3), (10, 49)):
        assert abs(lib.assemble_and_sum_pq_f32(fp(table), M, bp(codes), i * M, bp(codes), j * M, k) -
                   ref.assemble_and_sum_pq_f32(fp(table), M, bp(codes), i * M, bp(codes), j * M, k)) <= 1e-5


@pytest.mark.parametrize("n", [1, 7, 64, 65, 384, 1000])
def test_legacy_nvq(lib, ref, n):
    rng = np.random.default_rng(n)
    v = (rng.standard_normal(n) * 0.05).astype(np.float32)
    q = (rng.standard_normal(n) * 0.05).astype(np.float32)
    cen = (rng.standard_normal(n) * 0.01).astype(np.float32)
    minv, maxv = (float(v.min()), float(v.max())) if n > 1 else (float(v[0]) - 0.01, float(v[0]) + 0.01)
    for alpha in (1e-2, 2.0, 11.5):
        x, y = np.empty(n, np.uint8), np.empty(n, np.uint8)
        lib.nvq_quantize_8bit(fp(v), n, alpha, 0.0, minv, maxv, bp(x))
        ref.nvq_quantize_8bit(fp(v), n, alpha, 0.0, minv, maxv, bp(y))
        assert np.array_equal(x, y)
        assert abs(lib.nvq_loss(fp(v), n, alpha, 0.0, minv, maxv, 8) - ref.nvq_loss(fp(v), n, alpha, 0.0, minv, maxv, 8)) <= 1e-5 * ref.nvq_loss(fp(v), n, alpha, 0.0, minv, maxv, 8) + 1e-12
        qs, cs = q.copy(), cen.copy()
        ref.nvq_shuffle_query_in_place_8bit(fp(qs), n)
        ref.nvq_shuffle_query_in_place_8bit(fp(cs), n)
        q2 = q.copy()
        lib.nvq_shuffle_query_in_place_8bit(fp(q2), n)
        assert np.array_equal(q2, q)  # natural order: identity, as the scalar provider
        scale = float(np.abs(q).sum() * max(abs(minv), abs(maxv))) + 1e-12
        assert abs(lib.nvq_dot_product_8bit(fp(q), bp(x), n, alpha, 0.0, minv, maxv) - ref.nvq_dot_product_8bit(fp(qs), bp(x), n, alpha, 0.0, minv, maxv)) <= 1e-5 * scale
        w = ref.nvq_square_l2_distance_8bit(fp(qs), bp(x), n, alpha, 0.0, minv, maxv)
        assert abs(lib.nvq_square_l2_distance_8bit(fp(q), bp(x), n, alpha, 0.0, minv, maxv) - w) <= 1e-5 * abs(w) + 1e-12
        a = lib.nvq_cosine_8bit_packed(fp(q), bp(x), n, alpha, 0.0, minv, maxv, fp(cen))
        b = ref.nvq_cosine_8bit_packed(fp(qs), bp(x), n, alpha, 0.0, minv, maxv, fp(cs))
        for sh in (0, 32):
            fa = np.array([(a >> sh) & 0xffffffff], dtype=np.uint32).view(np.float32)[0]
            fb = np.array([(b >> sh) & 0xffffffff], dtype=np.uint32).view(np.float32)[0]
            assert abs(fa - fb) <= 1e-5 * max(scale, abs(fb))
    assert abs(lib.nvq_uniform_loss(fp(v), n, minv, maxv, 8) - ref.nvq_uniform_loss(fp(v), n, minv, maxv, 8)) <= 1e-5 * ref.nvq_uniform_loss(fp(v), n, minv, maxv, 8) + 1e-12


def test_gpu_group_fails_loudly_without_device(lib):
    """No CPU fallback: on a box without an sm_100 device every jv_ call reports JV_ERR_NO_DEVICE."""
    import ctypes as C
    if lib.jv_gpu_device_count() > 0:
        pytest.skip("a GPU is present")
    assert lib.jv_gpu_init(0) == -1
    h = C.c_void_p()
    rows = np.zeros((4, 8), np.float32)
    assert lib.jv_dataset_register_f32(fp(rows), 4, 8, C.byref(h)) == -1
    assert b"jv_gpu_init" in lib.jv_last_error()
    from jvector_b200 import F32Vectors, JVectorB200Error
    with pytest.raises(JVectorB200Error):
        F32Vectors(rows)
