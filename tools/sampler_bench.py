"""Host-side timing of the exact pairwise epoch sampler at the synthetic scale (no GPU needed).

    RECAD_SAMPLER_TRACE=1 python tools/sampler_bench.py [--epochs 3] [--cache /tmp/sb/allpos.npz]
"""
import argparse
import ctypes as C
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from recad_b200 import _lib, ops  # noqa: E402


def allpos(w, cache):
    if cache and os.path.exists(cache):
        z = np.load(cache)
        return z["ptr"], z["col"]
    eu, ei = bench.synth_edges(w, torch.device("cpu"))
    U = w["n_users"]
    ptr = np.zeros(U + 1, dtype=np.int64)
    np.cumsum(np.bincount(eu.numpy(), minlength=U), out=ptr[1:])
    col = ei.numpy().astype(np.int32)          # keys were unique-sorted: ascending per user
    if cache:
        np.savez(cache, ptr=ptr, col=col)
    return ptr, col


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--epochs", type=int, default=3)
    ap.add_argument("--workload", default="synthetic")
    ap.add_argument("--cache", default="")
    ap.add_argument("--compare", action="store_true",
                    help="also run the plain sampler + shuffle draws (recad_mt19937_pairwise) and compare every output")
    a = ap.parse_args()
    w = bench.WORKLOADS[a.workload]
    t0 = time.time()
    ptr, col = allpos(w, a.cache)
    hp, hc = ops.host_empty(ptr.shape, np.int64), ops.host_empty(col.shape, np.int32)
    hp[:], hc[:] = ptr, col
    print(f"positives ready in {time.time() - t0:.1f} s: {len(col)} pairs", flush=True)
    n = len(col)
    np.random.seed(2023)
    st, key, pos = ops._np_state()
    out = ops.host_empty((n, 3), np.int64)
    j = ops.host_empty(n, np.uint32)
    perm = ops.host_empty(n, np.int64)
    key2, pos2 = key.copy(), [pos[0]]
    users, rel, negs, j2 = (ops.host_empty(n, np.uint32) for _ in range(4))
    perm32 = ops.host_empty(n, np.int32)
    for e in range(a.epochs):
        t0 = time.time()
        m = ops.mt_pairwise_soa_raw(key2, pos2, w["n_users"], w["n_items"], n, hp, hc, users, rel, negs, j2)
        t1 = time.time()
        ops.permutation_apply32(j2[:m], perm32)
        t2 = time.time()
        print(f"epoch {e} [soa]: sampler+draws {t1 - t0:.3f} s, swaps {t2 - t1:.3f} s", flush=True)
        if a.compare:
            t0 = time.time()
            n_out, cpos = C.c_int64(), C.c_int32(pos[0])
            _lib.check(_lib.lib().recad_mt19937_pairwise(key.ctypes.data, C.byref(cpos), w["n_users"], w["n_items"], n, hp.ctypes.data,
                                                         hc.ctypes.data, out.ctypes.data, C.byref(n_out)), "recad_mt19937_pairwise")
            pos[0] = cpos.value
            S = out[:n_out.value]
            jj = ops.mt_permutation_draw_raw(key, pos, len(S), j)
            t1 = time.time()
            ops.permutation_apply(jj, perm)
            t2 = time.time()
            same = (m == len(S) and np.array_equal(users[:m], S[:, 0]) and np.array_equal(hc[hp[users[:m]] + rel[:m]], S[:, 1])
                    and np.array_equal(negs[:m], S[:, 2]) and np.array_equal(j2[:m], jj) and np.array_equal(perm32[:m], perm[:m])
                    and np.array_equal(key, key2) and pos[0] == pos2[0])
            print(f"epoch {e} [plain]: sampler+draws {t1 - t0:.3f} s, swaps {t2 - t1:.3f} s; identical: {same}", flush=True)


if __name__ == "__main__":
    main()
