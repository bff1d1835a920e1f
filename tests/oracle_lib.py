"""ctypes access to the CPU oracle (oracle/libjv_oracle.so) and to the reference's own compiled kernels
(oracle/_ref/libjvector.so). TEST INFRASTRUCTURE: imported only by tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs."""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libjvector.so")
GOLDEN = os.path.join(ROOT, "tests", "golden")

EUCLIDEAN, DOT_PRODUCT, COSINE = 0, 1, 2

f32p = C.POINTER(C.c_float)
u8p = C.POINTER(C.c_uint8)
i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_int64)
u64p = C.POINTER(C.c_uint64)


def fp(a):
    return a.ctypes.data_as(f32p) if a is not None else None


def bp(a):
    return a.ctypes.data_as(u8p) if a is not None else None


def ip(a):
    return a.ctypes.data_as(i32p) if a is not None else None


def lp(a):
    return a.ctypes.data_as(i64p) if a is not None else None


def wp(a):
    return a.ctypes.data_as(u64p) if a is not None else None


class Graph(C.Structure):
    _fields_ = [("n", C.c_int32), ("levels", C.c_int32), ("degree", C.c_int32), ("entry_node", C.c_int32),
                ("entry_level", C.c_int32), ("adj0", i32p), ("upper_row", i32p), ("upper_adj", i32p),
                ("upper_off", i64p)]


class Stats(C.Structure):
    _fields_ = [("visited", C.c_int32), ("expanded", C.c_int32), ("expanded_base", C.c_int32), ("reranked", C.c_int32)]


class Dataset(C.Structure):
    _fields_ = [("kind", C.c_int), ("metric", C.c_int), ("dim", C.c_int), ("base", f32p), ("n", C.c_int64),
                ("codebooks", f32p), ("M", C.c_int), ("k", C.c_int), ("centroid", f32p), ("codes", u8p), ("order", C.c_int)]


_lib = None


def build():
    subprocess.check_call(["make", "-C", ORACLE_DIR, "libjv_oracle.so"], stdout=subprocess.DEVNULL)
    if os.path.isdir("/root/reference/jvector-native"):
        subprocess.check_call([os.path.join(ORACLE_DIR, "build_ref.sh")], stdout=subprocess.DEVNULL)


def load():
    global _lib
    if _lib is not None:
        return _lib
    so = os.path.join(ORACLE_DIR, "libjv_oracle.so")
    src = os.path.join(ORACLE_DIR, "jv_oracle.c")
    if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        build()
    L = C.CDLL(so)
    F, I, P = C.c_float, C.c_int, C.c_void_p

    def sig(name, res, *args):
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = list(args)

    for n in ("jvo_dot_f32", "jvo_l2_f32", "jvo_cosine_f32", "jvo_cosine_native_f32"):
        sig(n, F, f32p, f32p, I)
    sig("jvo_score_from_raw", F, I, F)
    sig("jvo_compare_f32", F, I, f32p, f32p, I)
    sig("jvo_float_to_sortable_int", C.c_int32, F)
    sig("jvo_topk_key", C.c_int64, F, C.c_int32)
    sig("jvo_key_score", F, C.c_int64)
    sig("jvo_key_node", C.c_int32, C.c_int64)
    sig("jvo_bruteforce_topk_f32", None, I, f32p, C.c_int64, I, f32p, I, i64p)
    sig("jvo_pq_layout", None, I, I, i32p, i32p)
    sig("jvo_pq_encode", None, f32p, i32p, i32p, I, I, f32p, f32p, I, u8p)
    sig("jvo_pq_lut", None, f32p, i32p, i32p, I, I, f32p, f32p, I, I, f32p)
    sig("jvo_pq_self_magnitudes", None, f32p, i32p, i32p, I, I, f32p)
    sig("jvo_pq_adc", F, f32p, I, u8p, I)
    sig("jvo_pq_decoded_cosine", F, u8p, I, I, f32p, f32p, F)
    sig("jvo_pq_score_lut", F, I, f32p, f32p, F, I, u8p, I)
    sig("jvo_pq_score_direct", F, f32p, i32p, i32p, I, I, f32p, f32p, I, I, u8p)
    sig("jvo_pq_diversity_direct", F, f32p, i32p, i32p, I, I, I, u8p, u8p)
    sig("jvo_pq_pair_table", None, f32p, i32p, i32p, I, I, I, f32p)
    sig("jvo_pq_pair_sum", F, f32p, I, I, u8p, u8p)
    sig("jvo_pq_diversity_table", F, I, f32p, I, I, u8p, u8p)
    sig("jvo_kmeans_assign", None, f32p, C.c_int64, I, f32p, I, i32p)
    sig("jvo_bq_encode", None, f32p, I, u64p)
    sig("jvo_hamming", I, u64p, u64p, I)
    sig("jvo_bq_score", F, u64p, u64p, I, I)
    sig("jvo_nvq_logistic", F, F, F, F)
    sig("jvo_nvq_logit", F, F, F, F)
    sig("jvo_nvq_dequant", F, C.c_uint8, F, F, F, F)
    sig("jvo_nvq_quantize_8bit", None, f32p, I, F, F, F, F, u8p)
    sig("jvo_nvq_loss", F, f32p, I, F, F, F, F, I)
    sig("jvo_nvq_uniform_loss", F, f32p, I, F, F, I)
    sig("jvo_nvq_dot_8bit", F, f32p, u8p, I, F, F, F, F)
    sig("jvo_nvq_l2_8bit", F, f32p, u8p, I, F, F, F, F)
    sig("jvo_nvq_cosine_8bit", None, f32p, u8p, I, F, F, F, F, f32p, f32p)
    sig("jvo_nvq_encode_subvector", None, f32p, I, I, f32p, u8p)
    sig("jvo_nvq_encode", None, f32p, f32p, I, I, I, f32p, u8p)
    sig("jvo_nvq_loss_lanes", F, f32p, I, F, F, F, F, I, I)
    sig("jvo_nvq_uniform_loss_lanes", F, f32p, I, F, F, I, I)
    sig("jvo_nvq_encode_subvector_lanes", None, f32p, I, I, I, f32p, u8p)
    sig("jvo_nvq_encode_lanes", None, f32p, f32p, I, I, I, I, f32p, u8p)
    sig("jvo_nvq_score", F, I, f32p, f32p, I, I, f32p, u8p)
    sig("jvo_use_ref", I, C.c_char_p)
    sig("jvo_ref_isa", C.c_char_p)
    sig("jvo_scorer_f32", P, I, f32p, C.c_int64, I, f32p)
    sig("jvo_scorer_pq", P, I, f32p, I, I, I, f32p, u8p, C.c_int64, f32p)
    sig("jvo_scorer_bq", P, u64p, C.c_int64, I, f32p)
    sig("jvo_scorer_nvq", P, I, f32p, I, I, f32p, u8p, C.c_int64, f32p)
    sig("jvo_scorer_score", F, P, C.c_int32)
    sig("jvo_scorer_set_order", None, P, I)
    sig("jvo_fused_pq_pack", None, i32p, C.c_int32, I, u8p, I, u8p)
    sig("jvo_scorer_set_packed_neighbors", None, P, u8p, I)
    sig("jvo_scorer_score_neighbor", F, P, C.c_int32, I)
    sig("jvo_compare_f32_warp", F, I, f32p, f32p, I)
    sig("jvo_scorer_free", None, P)
    sig("jvo_graph_search", I, C.POINTER(Graph), P, P, I, I, i32p, f32p, C.POINTER(Stats))
    sig("jvo_graph_search_ex", I, C.POINTER(Graph), P, P, I, I, F, F, C.POINTER(C.c_uint32), i32p, f32p, C.POINTER(Stats))
    sig("jvo_graph_search_batch", C.c_double, C.POINTER(Graph), C.POINTER(Dataset), f32p, I, I, I, I, i32p, f32p, i64p)
    sig("jvo_numa_nodes", I)
    sig("jvo_alloc_interleaved", C.c_void_p, C.c_size_t)
    sig("jvo_free_interleaved", None, C.c_void_p, C.c_size_t)
    sig("jvo_nvq_encode_batch", C.c_double, f32p, C.c_int64, I, I, f32p, I, I, f32p, u8p)
    sig("jvo_bq_bruteforce_batch", C.c_double, u64p, C.c_int64, I, u64p, I, I, I, i64p)
    sig("jvo_graph_build_f32", C.c_int32, I, f32p, C.c_int32, I, I, I, F, F, i32p)
    sig("jvo_retain_diverse", I, f32p, i32p, I, f32p, I, F, u8p)
    _lib = L
    return L


_F, _I, _Z = C.c_float, C.c_int, C.c_size_t
# the 24-symbol ABI of native-c:src/jvector_simd_kernel_list.h: name -> (restype, argtypes)
REF_SIGNATURES = {
    "cosine_f32": (_F, [f32p, _Z, f32p, _Z, _Z]), "dot_product_f32": (_F, [f32p, _Z, f32p, _Z, _Z]),
    "euclidean_f32": (_F, [f32p, _Z, f32p, _Z, _Z]),
    "assemble_and_sum_f32": (_F, [f32p, _I, u8p, _I, _Z]), "assemble_and_sum_pq_f32": (_F, [f32p, _Z, u8p, _I, u8p, _I, _I]),
    "pq_decoded_cosine_similarity_f32": (_F, [u8p, _I, _Z, _I, f32p, f32p, _F]),
    "calculate_partial_sums_dot_f32": (None, [f32p, _I, _Z, _I, f32p, _I, f32p]),
    "calculate_partial_sums_euclidean_f32": (None, [f32p, _I, _Z, _I, f32p, _I, f32p]),
    "calculate_partial_sums_self_magnitude_f32": (None, [f32p, _I, _Z, _I, f32p]),
    "nvq_quantize_8bit": (None, [f32p, _Z, _F, _F, _F, _F, u8p]), "nvq_loss": (_F, [f32p, _Z, _F, _F, _F, _F, _I]),
    "nvq_uniform_loss": (_F, [f32p, _Z, _F, _F, _I]),
    "nvq_square_l2_distance_8bit": (_F, [f32p, u8p, _Z, _F, _F, _F, _F]), "nvq_dot_product_8bit": (_F, [f32p, u8p, _Z, _F, _F, _F, _F]),
    "nvq_cosine_8bit_packed": (C.c_int64, [f32p, u8p, _Z, _F, _F, _F, _F, f32p]),
    "nvq_shuffle_query_in_place_8bit": (None, [f32p, _Z]),
    "add_in_place_f32": (None, [f32p, f32p, _Z]), "sub_in_place_f32": (None, [f32p, f32p, _Z]), "min_in_place_f32": (None, [f32p, f32p, _Z]),
    "add_scalar_in_place_f32": (None, [f32p, _F, _Z]), "sub_scalar_in_place_f32": (None, [f32p, _F, _Z]),
    "max_f32": (_F, [f32p, _Z]),
    "jvector_simd_get_active_isa": (C.c_char_p, []), "jvector_simd_get_max_isa_env": (C.c_char_p, []),
}


def load_ref():
    """The reference's own libjvector.so (built by build() where the reference's sources are present), or None."""
    if not os.path.exists(REF_SO):
        build()
        if not os.path.exists(REF_SO):
            return None
    L = C.CDLL(REF_SO)
    for name, (res, args) in REF_SIGNATURES.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    return L


def interleaved_array(shape, dtype=np.float32):
    """numpy array over a buffer whose pages are interleaved across the NUMA nodes (CPU-baseline inputs)"""
    L = load()
    count = int(np.prod(shape))
    nbytes = count * np.dtype(dtype).itemsize
    p = L.jvo_alloc_interleaved(nbytes)
    if not p:
        return np.empty(shape, dtype)
    buf = (C.c_char * nbytes).from_address(p)
    return np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)  # lives for the process (bench inputs)


# ---------------------------------------------------------------------------------------------
# fixtures and generators
# ---------------------------------------------------------------------------------------------
def read_fvecs(path):
    raw = np.fromfile(path, dtype=np.int32)
    dim = int(raw[0])
    return raw.reshape(-1, dim + 1)[:, 1:].copy().view(np.float32)


def read_ivecs(path):
    raw = np.fromfile(path, dtype=np.int32)
    dim = int(raw[0])
    return raw.reshape(-1, dim + 1)[:, 1:].copy()


def load_siftsmall():
    d = os.path.join(GOLDEN, "siftsmall")
    return (read_fvecs(os.path.join(d, "siftsmall_base.fvecs")), read_fvecs(os.path.join(d, "siftsmall_query.fvecs")),
            read_ivecs(os.path.join(d, "siftsmall_groundtruth.ivecs")))


KERNEL_TEST_SIZES = [1, 3, 4, 5, 7, 8, 9, 15, 16, 17, 19, 32, 33, 37, 64, 71, 100, 128, 255]  # native-c:tests/test_helpers.cpp:49-76


def make_vec(n, seed):
    """native-c:tests/test_helpers.cpp:78-87"""
    i = np.arange(n)
    v = np.float32(seed) * (np.float32(1.0) + (i % 7).astype(np.float32) * np.float32(0.13))
    v = np.where(i % 3 == 0, -v, v).astype(np.float32)
    return (v + np.float32(0.5)).astype(np.float32)


def random_unit_vectors(rng, n, dim):
    v = rng.standard_normal((n, dim)).astype(np.float32)
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    return np.ascontiguousarray(v, dtype=np.float32)


def pq_layout(dim, M):
    base, rem = divmod(dim, M)
    sizes = np.array([base + (1 if m < rem else 0) for m in range(M)], dtype=np.int32)
    offsets = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int32)
    return sizes, offsets


def train_pq_numpy(rng, data, M, k=256, iters=6):
    """Lloyd k-means per subspace (test/bench helper; PQ training itself is out of scope: SURVEY §2.1).
    Returns codebooks concatenated: codebook m = k*size_m floats at k*offsets[m]."""
    n, dim = data.shape
    sizes, offsets = pq_layout(dim, M)
    out = np.empty(k * dim, dtype=np.float32)
    for m in range(M):
        sub = data[:, offsets[m]:offsets[m] + sizes[m]]
        kk = min(k, n)
        cent = sub[rng.choice(n, kk, replace=False)].copy()
        if kk < k:
            cent = np.concatenate([cent, rng.standard_normal((k - kk, sizes[m])).astype(np.float32)])
        for _ in range(iters):
            d = (sub * sub).sum(1)[:, None] - 2 * sub @ cent.T + (cent * cent).sum(1)[None, :]
            a = d.argmin(1)
            cnt = np.bincount(a, minlength=k).astype(np.float32)
            sums = np.zeros((k, sizes[m]), dtype=np.float32)
            np.add.at(sums, a, sub)
            nz = cnt > 0
            cent[nz] = sums[nz] / cnt[nz, None]
        out[k * offsets[m]: k * (offsets[m] + sizes[m])] = cent.reshape(-1)
    return out, sizes, offsets


def encode_pq(L, codebooks, sizes, offsets, M, k, centroid, data):
    codes = np.empty((data.shape[0], M), dtype=np.uint8)
    for i in range(data.shape[0]):
        L.jvo_pq_encode(fp(codebooks), ip(sizes), ip(offsets), M, k, fp(centroid), fp(data[i]), data.shape[1], bp(codes[i]))
    return codes


def keys_of(scores, nodes):
    """top-k key (base:graph/NodeQueue.java:125-137) vectorised in numpy, for cross-checks."""
    bits = np.asarray(scores, dtype=np.float32).view(np.int32).astype(np.int64)
    sortable = bits ^ ((bits >> 31) & 0x7fffffff)
    return (sortable << 32) | ((~np.asarray(nodes, dtype=np.int64)) & 0xffffffff)


def make_graph(adj0, entry_node=0, upper=None):
    """Build a ctypes Graph. upper: list (level 1..) of (node_ids int32[], adj int32[count][degree])."""
    n, degree = adj0.shape
    g = Graph()
    keep = [adj0]
    g.n, g.degree, g.entry_node = n, degree, entry_node
    g.adj0 = ip(adj0)
    if upper:
        rows = np.full((len(upper), n), -1, dtype=np.int32)
        offs = np.zeros(len(upper), dtype=np.int64)
        blocks = []
        o = 0
        for l, (ids, adj) in enumerate(upper):
            rows[l, ids] = np.arange(len(ids), dtype=np.int32)
            offs[l] = o
            o += len(ids)
            blocks.append(adj.astype(np.int32))
        ua = np.ascontiguousarray(np.concatenate(blocks, axis=0))
        keep += [rows, offs, ua]
        g.levels = len(upper) + 1
        g.entry_level = len(upper)
        g.upper_row, g.upper_adj, g.upper_off = ip(rows), ip(ua), lp(offs)
    else:
        g.levels, g.entry_level = 1, 0
    g._keep = keep
    return g
