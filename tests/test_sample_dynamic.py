"""sampleDynamic on the device (DESIGN.md section 8f-4): the cv::sortIdx tie order, anms::RangeTree and the feature
construction after the candidate scan.

Bar: bit-exact.  The Python restatement (oracle/anms_oracle.py) is pinned against the reference's own RangeTree,
compiled from the DynOSAM sources into oracle/_ref/libanms_ref.so (oracle/anms_ref/Makefile; those cases skip where it
was not built) and against tests/golden/anms_rangetree.npz (the same compiled reference's selections, always).  The
kernels are pinned against the restatement and the fixture: same indices, same order, same counts.
"""
import ctypes as C
import os

import numpy as np
import pytest

from dynosam_b200.synth_frames import SyntheticStream

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libanms_ref.so")
GOLDEN = os.path.join(ROOT, "tests", "golden", "anms_rangetree.npz")
W, H = 1242, 375


def _lib_built():
    import __graft_entry__ as g
    if not os.path.exists(os.path.join(ROOT, "dynosam_b200", "libdynofront.so")):
        g.build()


def _ref():
    if not os.path.exists(REF_SO):
        pytest.skip("compiled reference RangeTree (oracle/_ref/libanms_ref.so) not built: no DynOSAM checkout")
    L = C.CDLL(REF_SO)
    L.anms_ref_range_tree.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_void_p]

    def run(xy, K, tol, cols, rows):
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2); out = np.zeros(max(len(xy), 1), np.int32)
        m = L.anms_ref_range_tree(xy.ctypes.data, len(xy), int(K), float(tol), int(cols), int(rows), out.ctypes.data)
        return [int(v) for v in out[:m]]
    return run


def _suppress(xy, K, tol, cols, rows):
    """suppressNonMax(RangeTree) on equal responses, oracle side: cv2.sortIdx ranking, then the restatement; returns
    indices into xy in selection order"""
    from oracle import anms_oracle as AO, frontend_oracle as FO
    order = AO.anms_priority_order(len(xy))
    return [int(order[i]) for i in AO.anms_range_tree(np.asarray(xy, np.float32).reshape(-1, 2)[order], K, tol, cols, rows)]


def _lists(seed, count, n_max, small=False):
    """seeded lists: integer / float coordinates, n log-uniform in [1, n_max], K in [1, 400] (K > n included)"""
    rng = np.random.default_rng(seed)
    out = []
    for t in range(count):
        cols, rows = (W, H) if not small or t % 2 == 0 else (96, 64)
        n = int(np.exp(rng.uniform(0, np.log(n_max))))
        K = int(rng.integers(1, 401)) if t % 5 else n + int(rng.integers(0, 30))
        K = max(K, 1)
        if t % 2 == 0:
            xy = np.stack([rng.integers(0, cols, n), rng.integers(0, rows, n)], 1).astype(np.float32)
        else:
            xy = np.stack([rng.uniform(0, cols, n), rng.uniform(0, rows, n)], 1).astype(np.float32)
        out.append((xy, K, [0.01, 0.001][(t//2) % 2], cols, rows))
    return out


# ------------------------------------------------------------------------------------------------ CPU
def test_tie_order_matches_cv2_sortidx():
    import cv2
    _lib_built()
    from dynosam_b200.frontend import anms_tie_order
    for n in list(range(1, 5001)) + [65536, 232875, 465750]:
        ref = cv2.sortIdx(np.zeros((1, n), np.int32), cv2.SORT_EVERY_ROW | cv2.SORT_DESCENDING).ravel()
        assert np.array_equal(anms_tie_order(n), ref), n
    assert len(anms_tie_order(0)) == 0


def test_restatement_matches_compiled_reference():
    ref = _ref()
    lists = _lists(101, 200, 20000, small=True) + _lists(7, 12, 3000)
    lists[0] = (lists[0][0][:1], 5, 0.01, W, H)                                   # n = 1
    assert len(lists) >= 200 and max(len(x[0]) for x in lists) > 10000 and any(K > len(xy) for xy, K, *_ in lists)
    from oracle import anms_oracle as AO, frontend_oracle as FO
    for xy, K, tol, cols, rows in lists:
        order = AO.anms_priority_order(len(xy))
        assert AO.anms_range_tree(xy[order], K, tol, cols, rows) == ref(xy[order], K, tol, cols, rows), (len(xy), K, tol, cols, rows)


def test_restatement_matches_golden():
    from oracle import anms_oracle as AO, frontend_oracle as FO
    z = np.load(GOLDEN)
    off = 0; soff = 0
    for l, n in enumerate(z["counts"]):
        xy = z["xy"][off:off + n]; order = z["order"][off:off + n]
        assert np.array_equal(AO.anms_priority_order(n), order)
        sel = z["selected"][soff:soff + z["n_selected"][l]]
        assert _suppress(xy, int(z["K"][l]), float(z["tolerance"][l]), int(z["cols"][l]), int(z["rows"][l])) == list(sel), l
        off += n; soff += z["n_selected"][l]
    assert 0 < z["n_selected"].sum() and (z["n_selected"] == 0).any()


def test_k1_selects_nothing():
    from oracle import anms_oracle as AO, frontend_oracle as FO
    rng = np.random.default_rng(3)
    xy = np.stack([rng.uniform(0, W, 500), rng.uniform(0, H, 500)], 1).astype(np.float32)
    assert AO.anms_range_tree(xy, 1, 0.01, W, H) == []
    assert AO.anms_search_range(500, 1, 0.01, W, H)[0] == -2**31              # NaN -> INT_MIN, the search never starts
    if os.path.exists(REF_SO):
        assert _ref()(xy, 1, 0.01, W, H) == []


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_anms_range_tree_matches_oracle():
    from dynosam_b200.frontend import FeatureTrackerGPU
    t = FeatureTrackerGPU(W, H)
    one = np.array([[7.5, 3.25]], np.float32)
    for cols, rows, seed in [(W, H, 11), (96, 64, 12)]:
        rng = np.random.default_rng(seed)
        lists = [(xy, K) for xy, K, *_ in _lists(seed, 60, 12000)]
        if cols != W:
            lists = [(np.stack([rng.uniform(0, cols, len(xy)), rng.uniform(0, rows, len(xy))], 1).astype(np.float32), K) for xy, K in lists[:30]]
        lists += [(np.zeros((0, 2), np.float32), 10), (one, 5), (one, 1), (lists[0][0], 0), (lists[0][0], 1)]   # n = 0, n = 1, K = 0, K = 1
        for tol in (0.01, 0.001):
            got = t.anms_range_tree([xy for xy, _ in lists], [K for _, K in lists], tol, cols, rows)          # one launch for all lists
            for (xy, K), g in zip(lists, got):
                assert list(g) == (_suppress(xy, K, tol, cols, rows) if K > 0 else []), (len(xy), K, tol, cols, rows)
            assert [len(g) for g in got[-5:]] == [0, 1, 0, 0, 0]


@pytest.mark.gpu
def test_anms_global_memory_paths():
    """lists whose points and / or cell bitmap do not fit in shared memory (4000 x 4000 cells = 2 MB of bitmap;
    30000 points = 240 KB) take the global-memory fallbacks"""
    from dynosam_b200.frontend import FeatureTrackerGPU
    t = FeatureTrackerGPU(W, H)
    rng = np.random.default_rng(9)
    big = np.stack([rng.uniform(0, 4000, 30000), rng.uniform(0, 4000, 30000)], 1).astype(np.float32)
    mid = np.stack([rng.integers(0, 4000, 2000), rng.integers(0, 4000, 2000)], 1).astype(np.float32)
    got = t.anms_range_tree([big, mid], [200, 150], 0.01, 4000, 4000)
    for xy, K, g in zip([big, mid], [200, 150], got):
        assert list(g) == _suppress(xy, K, 0.01, 4000, 4000)
    dense = np.stack([rng.integers(0, W, 28000), rng.integers(0, H, 28000)], 1).astype(np.float32)   # bitmap shared, points global
    g, = t.anms_range_tree([dense], [200], 0.01, W, H)
    assert list(g) == _suppress(dense, 200, 0.01, W, H)


@pytest.mark.gpu
def test_anms_range_tree_reproduces_golden():
    from dynosam_b200.frontend import FeatureTrackerGPU
    z = np.load(GOLDEN)
    t = FeatureTrackerGPU(W, H)
    off = 0; soff = 0
    for l, n in enumerate(z["counts"]):
        g, = t.anms_range_tree([z["xy"][off:off + n]], [int(z["K"][l])], float(z["tolerance"][l]), int(z["cols"][l]), int(z["rows"][l]))
        assert np.array_equal(g, z["selected"][soff:soff + z["n_selected"][l]]), l
        off += n; soff += z["n_selected"][l]


def _c4_frame(k, seed=42):
    """frame k of the C4 stream with the detection mask that trackDynamic leaves (previous features, min distance 2)"""
    from oracle import anms_oracle as AO, frontend_oracle as FO
    rng = np.random.default_rng(seed + k)
    st = SyntheticStream(n_objects=10, seed=seed)
    _, m0, f0 = st.frame(k - 1); _, m1, f1 = st.frame(k)
    kps, labs = [], []
    for lab in range(1, 11):
        ys, xs = np.nonzero(m0 == lab)
        if len(ys) == 0:
            continue
        sel = rng.choice(len(ys), size=min(150, len(ys)), replace=False)
        kps.append(np.stack([xs[sel] + 0.5 + f0[ys[sel], xs[sel], 0], ys[sel] + 0.5 + f0[ys[sel], xs[sel], 1]], 1)); labs.append(np.full(len(sel), lab, np.int32))
    kp = np.concatenate(kps); lab = np.concatenate(labs)
    ok = (kp[:, 0] > 1) & (kp[:, 0] < W - 1) & (kp[:, 1] > 1) & (kp[:, 1] < H - 1)
    kp, lab = kp[ok], lab[ok]
    age = rng.integers(0, 21, len(lab)).astype(np.int32); tid = np.arange(len(lab), dtype=np.int64)
    det = FO.track_dynamic(kp, lab, age, tid, f1, m1, None, FO.TrackParams(), 10**6)[7]
    return m1, f1, (kp, lab, age, tid), det


@pytest.mark.gpu
@pytest.mark.parametrize("frame", [3, 40])
def test_sample_dynamic_bit_exact(frame):
    from dynosam_b200.frontend import FeatureTrackerGPU, TrackParams
    from oracle import anms_oracle as AO, frontend_oracle as FO
    m1, f1, (kp, lab, age, tid), det = _c4_frame(frame)
    objects = list(range(1, 11))
    num_track = [0, 200, 199, 198, 250, 0, 120, 0, 10, 0]                          # K = 200, 0, 1, 2, 0, 200, 80, 200, 190, 200
    prm = TrackParams()
    t = FeatureTrackerGPU(W, H); t.set_frame(f1, m1, None)
    acc, *_ , det_gpu, _trk = t.track_dynamic(kp, lab, age, tid, prm, 10**6)
    assert np.array_equal(det_gpu, det)
    got = t.sample_dynamic(objects, num_track, prm, 5000, max_features=200)
    want = AO.sample_dynamic(f1, m1, det, objects, num_track, 200, FO.TrackParams(), 5000)
    for key in ("candidates", "zero_flow", "selected"):
        assert np.array_equal(got[key], want[key]), key
    assert np.array_equal(got["offset"], np.concatenate([[0], np.cumsum(want["selected"])[:-1]]))
    for key in ("keypoint", "flow", "predicted", "tracklet", "object"):
        assert got[key].shape == want[key].shape and np.array_equal(got[key], want[key]), key
    assert got["next_tracklet_id"] == want["next_tracklet_id"] == 5000 + int(want["selected"].sum())
    assert want["candidates"].min() > 0 and want["selected"][1] == 0 and want["selected"][2] == 0 and want["selected"][4] == 0
    assert want["selected"][0] > 100 and want["selected"][3] > 0
    again = t.sample_dynamic(objects, num_track, prm, 5000, max_features=200)       # the same call again: the same outputs
    for key in got:
        assert np.array_equal(np.asarray(got[key]), np.asarray(again[key])), key


@pytest.mark.gpu
def test_sample_dynamic_capacity_and_arguments():
    from dynosam_b200.frontend import FeatureTrackerGPU, FrontendError, TrackParams
    m1, f1, feats, det = _c4_frame(5)
    t = FeatureTrackerGPU(W, H); t.set_frame(f1, m1, det)
    with pytest.raises(FrontendError):
        t.sample_dynamic(list(range(1, 11)), [0]*10, TrackParams(), 100, capacity=10)
    full = t.sample_dynamic(list(range(1, 11)), [0]*10, TrackParams(), 100)
    assert len(full["tracklet"]) > 10 and full["tracklet"][0] == 100
    none = t.sample_dynamic([], [], TrackParams(), 7)
    assert none["next_tracklet_id"] == 7 and len(none["keypoint"]) == 0
