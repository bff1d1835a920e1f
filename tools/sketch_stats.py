"""c2's fp32 walk with and without the projection sketch: sketch build time, the share of visited rows the walk still reads, the
queries re-run for a candidate-list overflow, and device time. Same data, graph and queries as bench.py c2 (single GPU).

    python tools/sketch_stats.py [--n 1000000] [--nq 10000] [--reps 3]"""
import argparse
import ctypes as C
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
import jvector_b200 as jv  # noqa: E402
from jvector_b200 import _native as nat  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--nq", type=int, default=10_000)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    lib = jv.init(0)
    DOT = jv.VectorSimilarityFunction.DOT_PRODUCT
    base = bench.gen_unit_rows_device(torch, bench.SEED, a.n, a.dim, "latent")
    qd = bench.gen_unit_rows_device(torch, bench.SEED + 1, a.nq, a.dim, "latent")
    h = C.c_void_p()
    nat.check(lib.jv_dataset_adopt_f32_device(C.c_void_p(base.data_ptr()), a.n, a.dim, a.dim, C.byref(h)))
    vec = jv.api._Vectors(h, base)
    gi = jv.GraphIndexBuilder(DOT, M=32, beamWidth=100, neighborOverflow=1.2, alpha=1.2, addHierarchy=True, seed=bench.SEED).build(vec)
    dn, ds = C.c_void_p(), C.c_void_p()
    nat.check(lib.jv_device_malloc(C.byref(dn), a.nq * 40))
    nat.check(lib.jv_device_malloc(C.byref(ds), a.nq * 40))
    st = nat.SearchStats()

    def run(sketch):
        os.environ["JV_F32_SKETCH"] = "1" if sketch else "0"
        r0 = lib.jv_search_rows_read()
        t0 = time.perf_counter()
        nat.check(lib.jv_graph_search_batch_device(gi._h, vec._h, None, int(DOT), C.c_void_p(qd.data_ptr()), a.nq, 10, 100, dn, ds, C.byref(st)))
        wall = (time.perf_counter() - t0) * 1e3
        return {"device_ms": round(st.device_ms, 3), "wall_ms": round(wall, 1), "visited": st.visited, "rows_read": lib.jv_search_rows_read() - r0,
                "retried": st.retried}

    print("off (first call):", run(False))
    first = run(True)
    state, cap = C.c_int(), C.c_double()
    nat.check(lib.jv_dataset_f32_sketch(vec._h, C.byref(state), C.byref(cap), None, None, None))
    print("on (first call, includes the sketch build):", first, "state", state.value, "captured %.4f" % cap.value)
    print("sketch build ~ %.1f ms (first-call wall minus device time)" % (first["wall_ms"] - first["device_ms"]))
    for _ in range(a.reps):
        for sk in (False, True):
            r = run(sk)
            r["rows_read/visited"] = round(r["rows_read"] / max(1, r["visited"]), 4)
            print("sketch=%d" % sk, r, flush=True)
    lib.jv_device_free(dn)
    lib.jv_device_free(ds)


if __name__ == "__main__":
    main()
