#!/usr/bin/env python
"""Generates tests/golden/anms_rangetree.npz from the reference's own anms::RangeTree on seeded lists.

    python tests/golden/make_anms_golden.py     # needs oracle/_ref/libanms_ref.so (oracle/anms_ref/Makefile)

Unlike the other fixtures these are the REFERENCE's outputs: oracle/anms_ref/Makefile compiles DynOSAM's
dynosam/src/frontend/anms/anms.cc with a stub OpenCV header.  The file stores the lists, their cv::sortIdx walk order, K,
the tolerance, the image size and the reference's selection as indices into each list, so the pin travels without the
DynOSAM checkout (tests/test_sample_dynamic.py).
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import anms_oracle as AO                # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def anms_lists(seed=17, n_lists=48):
    """Seeded ANMS inputs: (xy float32 [n][2], K, tolerance, cols, rows) per list; integer and float coordinates,
    n log-uniform in [1, 4000], K from 1 to 400 (some K > n)."""
    rng = np.random.default_rng(seed)
    out = []
    for t in range(n_lists):
        cols, rows = [(1242, 375), (160, 120), (640, 480)][t % 3]
        n = int(np.exp(rng.uniform(0, np.log(4000))))
        K = [1, 2, int(rng.integers(3, 401)), int(rng.integers(3, 401)), int(rng.integers(3, 401)), n + int(rng.integers(1, 50))][t % 6]
        if t % 2 == 0:
            xy = np.stack([rng.integers(0, cols, n), rng.integers(0, rows, n)], 1).astype(np.float32)
        else:
            xy = np.stack([rng.uniform(0, cols, n), rng.uniform(0, rows, n)], 1).astype(np.float32)
        out.append((xy, K, [0.01, 0.001][(t//2) % 2], cols, rows))
    return out


def ref_anms():
    """anms_ref_range_tree of oracle/_ref/libanms_ref.so: (xy in walk order, K, tol, cols, rows) -> positions"""
    path = os.path.join(ROOT, "oracle", "_ref", "libanms_ref.so")
    if not os.path.exists(path):
        raise SystemExit(f"{path} is missing: build() compiles it from a DynOSAM checkout (oracle/anms_ref/Makefile)")
    L = C.CDLL(path)
    L.anms_ref_range_tree.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_void_p]

    def run(xy, K, tol, cols, rows):
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2); out = np.zeros(max(len(xy), 1), np.int32)
        m = L.anms_ref_range_tree(xy.ctypes.data, len(xy), int(K), float(tol), int(cols), int(rows), out.ctypes.data)
        return [int(v) for v in out[:m]]
    return run


def anms_fixture(ref_range_tree):
    xy, counts, K, tol, cols, rows, order, sel, nsel = [], [], [], [], [], [], [], [], []
    for a, k, t, c, r in anms_lists():
        o = AO.anms_priority_order(len(a))
        s = [int(o[i]) for i in ref_range_tree(a[o], k, t, c, r)]
        xy.append(a); counts.append(len(a)); K.append(k); tol.append(t); cols.append(c); rows.append(r); order.append(o); sel += s; nsel.append(len(s))
    return {"xy": np.concatenate(xy).astype(np.float32), "counts": np.array(counts, np.int32), "K": np.array(K, np.int32),
            "tolerance": np.array(tol, np.float32), "cols": np.array(cols, np.int32), "rows": np.array(rows, np.int32),
            "order": np.concatenate(order).astype(np.int32), "selected": np.array(sel, np.int32), "n_selected": np.array(nsel, np.int32)}


def main():
    path = os.path.join(HERE, "anms_rangetree.npz")
    np.savez_compressed(path, **anms_fixture(ref_anms()))
    print(os.path.basename(path), os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
