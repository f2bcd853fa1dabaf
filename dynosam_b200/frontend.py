"""ctypes binding of libdynofront.so (include/dynofront.h): dense-flow tracking / mask propagation / pyramidal KLT.
Mirrors the reference's FeatureTracker entry points (dynosam/src/frontend/vision/FeatureTracker.cc).  No CPU fallback."""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdynofront.so")
EXPORTS = ["dynofront_create", "dynofront_destroy", "dynofront_last_error", "dynofront_set_frame", "dynofront_track_dynamic",
           "dynofront_sample_candidates", "dynofront_propagate_mask", "dynofront_klt_track", "dynofront_klt_track_fb",
           "dynofront_klt_last_min_eig", "dynofront_stereo_track", "dynofront_track_static_flow", "dynofront_next_frame", "dynofront_pin_host", "dynofront_unpin_host",
           "dynofront_get_motion_mask", "dynofront_get_pyramid_level", "dynofront_sample_dynamic", "dynofront_anms_range_tree",
           "dynofront_anms_tie_order"]


class TrackParamsC(C.Structure):
    _fields_ = [("max_dynamic_feature_age", C.c_int32), ("min_distance", C.c_int32), ("shrink_row", C.c_int32), ("shrink_col", C.c_int32)]


@dataclass
class TrackParams:
    max_dynamic_feature_age: int = 20
    min_distance: int = 2
    shrink_row: int = 0
    shrink_col: int = 0

    def c(self):
        return TrackParamsC(self.max_dynamic_feature_age, self.min_distance, self.shrink_row, self.shrink_col)


class KltFbParamsC(C.Structure):
    _fields_ = [("win", C.c_int32), ("max_level", C.c_int32), ("max_count", C.c_int32), ("epsilon", C.c_double),
                ("win_back", C.c_int32), ("max_level_back", C.c_int32), ("max_count_back", C.c_int32), ("epsilon_back", C.c_double),
                ("use_initial_flow", C.c_int32), ("min_eig_threshold", C.c_double), ("max_fb_distance", C.c_double),
                ("check_static", C.c_int32), ("max_feature_track_age", C.c_int32), ("track", TrackParamsC)]


_LIB = None


def load():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it first (__graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        L.dynofront_last_error.restype = C.c_char_p
        L.dynofront_last_error.argtypes = [C.c_void_p]
        L.dynofront_create.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.dynofront_destroy.argtypes = [C.c_void_p]
        L.dynofront_set_frame.argtypes = [C.c_void_p] + [C.c_void_p]*3
        L.dynofront_track_dynamic.argtypes = [C.c_void_p, C.c_int32] + [C.c_void_p]*4 + [C.POINTER(TrackParamsC), C.POINTER(C.c_int64)] + [C.c_void_p]*8
        L.dynofront_sample_candidates.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.POINTER(TrackParamsC)] + [C.c_void_p]*4 + [C.c_int64]
        L.dynofront_propagate_mask.argtypes = [C.c_void_p, C.c_int32] + [C.c_void_p]*4 + [C.POINTER(TrackParamsC), C.c_int32, C.c_void_p]
        L.dynofront_klt_track.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_int32, C.c_double, C.POINTER(C.c_float)]
        L.dynofront_klt_track_fb.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.POINTER(KltFbParamsC), C.c_void_p, C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_float)]
        L.dynofront_stereo_track.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                                             C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]
        L.dynofront_klt_last_min_eig.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.dynofront_track_static_flow.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32,
                                                  C.POINTER(C.c_int64)] + [C.c_void_p]*8 + [C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.dynofront_next_frame.argtypes = [C.c_void_p] + [C.c_void_p]*4
        L.dynofront_pin_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.dynofront_unpin_host.argtypes = [C.c_void_p, C.c_void_p]
        L.dynofront_get_motion_mask.argtypes = [C.c_void_p, C.c_void_p]
        L.dynofront_sample_dynamic.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.POINTER(TrackParamsC),
                                               C.POINTER(C.c_int64)] + [C.c_void_p]*8 + [C.c_int64, C.POINTER(C.c_float)]
        L.dynofront_anms_range_tree.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int32, C.c_int32,
                                                C.c_void_p, C.c_void_p]
        L.dynofront_anms_tie_order.argtypes = [C.c_int32, C.c_void_p]
        L.dynofront_get_pyramid_level.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_void_p, C.c_void_p]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class FrontendError(RuntimeError):
    pass


def anms_tie_order(n):
    """Walk order of n equal responses (cv::sortIdx(zeros(1, n), SORT_EVERY_ROW | SORT_DESCENDING)); host only."""
    out = np.zeros(int(n), np.int32)
    if load().dynofront_anms_tie_order(int(n), _p(out)) != 0:
        raise FrontendError(f"dynofront_anms_tie_order({n}) failed")
    return out


class FeatureTrackerGPU:
    """One handle per camera stream (image size fixed at construction)."""

    def __init__(self, width, height, device=0):
        self.lib = load(); self.W, self.H = int(width), int(height)
        self.h = C.c_void_p()
        st = self.lib.dynofront_create(device, self.W, self.H, C.byref(self.h))
        if st != 0:
            raise FrontendError(f"dynofront_create failed ({st}): no sm_100 CUDA device; libdynofront has no CPU path")

    def _ck(self, st):
        if st != 0:
            raise FrontendError(f"libdynofront status {st}: {self.lib.dynofront_last_error(self.h).decode()}")

    def close(self):
        if self.h:
            self.lib.dynofront_destroy(self.h); self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_frame(self, flow, motion_mask, detection_mask=None):
        flow = np.ascontiguousarray(flow, dtype=np.float32); motion_mask = np.ascontiguousarray(motion_mask, dtype=np.int32)
        det = None if detection_mask is None else np.ascontiguousarray(detection_mask, dtype=np.uint8)
        self._ck(self.lib.dynofront_set_frame(self.h, _p(flow), _p(motion_mask), _p(det)))

    # ---- streaming mode (resident frames)
    def pin(self, arr):
        """register a C-contiguous numpy array as pinned host memory (asynchronous uploads); keep it alive until unpin"""
        self._ck(self.lib.dynofront_pin_host(self.h, _p(arr), arr.nbytes))

    def unpin(self, arr):
        self._ck(self.lib.dynofront_unpin_host(self.h, _p(arr)))

    def next_frame(self, gray, flow, motion_mask, detection_mask=None):
        """arrays must already be C-contiguous uint8 / float32 / int32 (no conversion copies on the streaming path)"""
        assert gray.dtype == np.uint8 and flow.dtype == np.float32 and motion_mask.dtype == np.int32
        assert gray.flags.c_contiguous and flow.flags.c_contiguous and motion_mask.flags.c_contiguous
        self._ck(self.lib.dynofront_next_frame(self.h, _p(gray), _p(flow), _p(motion_mask), _p(detection_mask)))

    def propagate_mask_resident(self, prev_pred_kp, prev_label, prm: TrackParams, min_votes=150):
        kp = np.ascontiguousarray(prev_pred_kp, dtype=np.float64).reshape(-1, 2); lab = np.ascontiguousarray(prev_label, dtype=np.int32)
        pc = prm.c()
        self._ck(self.lib.dynofront_propagate_mask(self.h, kp.shape[0], _p(kp), _p(lab), None, None, C.byref(pc), int(min_votes), None))

    def motion_mask(self):
        out = np.zeros((self.H, self.W), np.int32)
        self._ck(self.lib.dynofront_get_motion_mask(self.h, _p(out)))
        return out

    def track_dynamic(self, prev_pred_kp, prev_label, prev_age, prev_tracklet, prm: TrackParams, next_tracklet_id: int, want_masks=True):
        kp = np.ascontiguousarray(prev_pred_kp, dtype=np.float64).reshape(-1, 2); n = kp.shape[0]
        lab = np.ascontiguousarray(prev_label, dtype=np.int32); age = np.ascontiguousarray(prev_age, dtype=np.int32)
        tid = np.ascontiguousarray(prev_tracklet, dtype=np.int64)
        acc = np.zeros(n, np.uint8); pk = np.zeros((n, 2)); fl = np.zeros((n, 2)); oage = np.zeros(n, np.int32)
        otid = np.zeros(n, np.int64); olab = np.zeros(n, np.int32)
        det = np.zeros((self.H, self.W), np.uint8) if want_masks else None
        trk = np.zeros((self.H, self.W), np.uint8) if want_masks else None
        nid = C.c_int64(int(next_tracklet_id)); pc = prm.c()
        self._ck(self.lib.dynofront_track_dynamic(self.h, n, _p(kp), _p(lab), _p(age), _p(tid), C.byref(pc), C.byref(nid), _p(acc), _p(pk), _p(fl),
                                                  _p(oage), _p(otid), _p(olab), _p(det), _p(trk)))
        return acc, pk, fl, oage, otid, olab, nid.value, det, trk

    def sample_candidates(self, objects, prm: TrackParams, capacity=None):
        objs = np.ascontiguousarray(objects, dtype=np.int32); n = objs.shape[0]
        cap = int(capacity if capacity is not None else self.W*self.H)
        counts = np.zeros(n, np.int32); offs = np.zeros(n, np.int32); zero = np.zeros(n, np.int32); idx = np.empty(cap, np.int32)
        pc = prm.c()
        self._ck(self.lib.dynofront_sample_candidates(self.h, n, _p(objs), C.byref(pc), _p(counts), _p(offs), _p(zero), _p(idx), cap))
        return {int(o): idx[offs[i]:offs[i] + counts[i]].copy() for i, o in enumerate(objs)}, {int(o): int(zero[i]) for i, o in enumerate(objs)}

    def sample_dynamic(self, objects, num_track, prm: TrackParams, next_tracklet_id: int, max_features=200, tolerance=0.01, capacity=None):
        """FeatureTracker::sampleDynamic in one call: candidate scan, RangeTree ANMS with K = max(max_features - num_track, 0)
        per object, new features.  Returns a dict: per object (order of `objects`) candidates / zero_flow / selected /
        offset, per feature keypoint / flow / predicted (n, 2) float64, tracklet int64, object int32, and next_tracklet_id."""
        objs = np.ascontiguousarray(objects, dtype=np.int32); n = objs.shape[0]
        nt = np.ascontiguousarray(num_track, dtype=np.int32)
        assert nt.shape == (n,)
        cap = int(capacity if capacity is not None else max(int(max_features), 0)*n + 64)
        cand = np.zeros(n, np.int32); zero = np.zeros(n, np.int32); sel = np.zeros(n, np.int32); off = np.zeros(n, np.int32)
        kp = np.zeros((cap, 2)); fl = np.zeros((cap, 2)); pk = np.zeros((cap, 2)); tid = np.zeros(cap, np.int64)
        nid = C.c_int64(int(next_tracklet_id)); pc = prm.c(); ms = C.c_float()
        st = self.lib.dynofront_sample_dynamic(self.h, n, _p(objs), _p(nt), int(max_features), float(tolerance), C.byref(pc), C.byref(nid),
                                               _p(cand), _p(zero), _p(sel), _p(off), _p(kp), _p(fl), _p(pk), _p(tid), cap, C.byref(ms))
        if st == -1 and int(sel.sum()) > cap and capacity is None:          # more features than the default room: once more, large enough
            return self.sample_dynamic(objects, num_track, prm, next_tracklet_id, max_features, tolerance, capacity=int(sel.sum()))
        self._ck(st)
        self.last_ms = ms.value
        m = int(sel.sum())
        return dict(candidates=cand, zero_flow=zero, selected=sel, offset=off, keypoint=kp[:m], flow=fl[:m], predicted=pk[:m], tracklet=tid[:m],
                    object=np.repeat(objs, sel), next_tracklet_id=nid.value)

    def anms_range_tree(self, lists, num_ret_points, tolerance=0.01, cols=None, rows=None):
        """AdaptiveNonMaximumSuppression(RangeTree) on several lists of float (x, y) in one launch (the trackDynamicKLT call
        site).  lists: sequence of (n_l, 2) arrays in the caller's order; num_ret_points: K per list.  Returns a list of
        int32 arrays: the selected indices into each list, in selection order."""
        arrs = [np.ascontiguousarray(a, dtype=np.float32).reshape(-1, 2) for a in lists]
        counts = np.array([len(a) for a in arrs], np.int32)
        xy = np.ascontiguousarray(np.concatenate(arrs) if arrs else np.zeros((0, 2), np.float32), dtype=np.float32)
        K = np.ascontiguousarray(num_ret_points, dtype=np.int32).reshape(-1)
        assert K.shape == counts.shape
        idx = np.zeros(max(len(xy), 1), np.int32); nsel = np.zeros(len(arrs), np.int32)
        self._ck(self.lib.dynofront_anms_range_tree(self.h, len(arrs), _p(counts), _p(xy), _p(K), float(tolerance), int(cols or self.W),
                                                    int(rows or self.H), _p(idx), _p(nsel)))
        offs = np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.int64) if len(arrs) else []
        return [idx[o:o + k].copy() for o, k in zip(offs, nsel)]

    def propagate_mask(self, prev_pred_kp, prev_label, prev_mask, prev_flow, current_mask, prm: TrackParams, min_votes=150):
        kp = np.ascontiguousarray(prev_pred_kp, dtype=np.float64).reshape(-1, 2)
        lab = np.ascontiguousarray(prev_label, dtype=np.int32)
        pm = np.ascontiguousarray(prev_mask, dtype=np.int32); pf = np.ascontiguousarray(prev_flow, dtype=np.float32)
        cur = np.ascontiguousarray(current_mask, dtype=np.int32).copy(); pc = prm.c()
        self._ck(self.lib.dynofront_propagate_mask(self.h, kp.shape[0], _p(kp), _p(lab), _p(pm), _p(pf), C.byref(pc), int(min_votes), _p(cur)))
        return cur

    def klt_track(self, prev_gray, cur_gray, prev_pts, win=21, max_level=3, max_count=30, eps=0.03, initial=None, min_eig=1e-4):
        """cv::calcOpticalFlowPyrLK(prev, cur, prevPts, nextPts, status, err, (win,win), maxLevel, (EPS|COUNT, max_count, eps))."""
        pg = np.ascontiguousarray(prev_gray, dtype=np.uint8); cg = np.ascontiguousarray(cur_gray, dtype=np.uint8)
        p0 = np.ascontiguousarray(prev_pts, dtype=np.float32).reshape(-1, 2); n = p0.shape[0]
        nxt = np.ascontiguousarray(initial, dtype=np.float32).reshape(-1, 2).copy() if initial is not None else np.zeros((n, 2), np.float32)
        st = np.zeros(n, np.uint8); err = np.zeros(n, np.float32); ms = C.c_float()
        self._ck(self.lib.dynofront_klt_track(self.h, _p(pg), _p(cg), n, _p(p0), _p(nxt), _p(st), _p(err), win, max_level, max_count, float(eps),
                                              1 if initial is not None else 0, float(min_eig), C.byref(ms)))
        self.last_ms = ms.value
        return nxt, st, err

    def klt_track_fb(self, prev_gray, cur_gray, prev_pts, prm: TrackParams | None = None, prev_age=None, max_feature_track_age=25,
                     win=21, max_level=3, max_count=30, eps=0.03, initial=None, min_eig=1e-4, max_fb_distance=0.5):
        """KltFeatureTracker::trackPoints in one call: forward LK, backward LK (21x21, 5 levels, OpenCV default criteria), the
        round-trip test and -- when prev_age is given -- the label / border / age checks.  Returns (next, status, back, keep)."""
        pg = None if prev_gray is None else np.ascontiguousarray(prev_gray, dtype=np.uint8)     # None, None: the resident frame pair
        cg = None if cur_gray is None else np.ascontiguousarray(cur_gray, dtype=np.uint8)
        p0 = np.ascontiguousarray(prev_pts, dtype=np.float32).reshape(-1, 2); n = p0.shape[0]
        nxt = np.ascontiguousarray(initial, dtype=np.float32).reshape(-1, 2).copy() if initial is not None else np.zeros((n, 2), np.float32)
        st = np.zeros(n, np.uint8); back = np.zeros((n, 2), np.float32); keep = np.zeros(n, np.uint8); ms = C.c_float()
        check = prev_age is not None
        age = np.ascontiguousarray(prev_age, dtype=np.int32) if check else None
        pc = KltFbParamsC(win, max_level, max_count, float(eps), 21, 5, 30, 0.01, 1 if initial is not None else 0, float(min_eig), float(max_fb_distance),
                          1 if check else 0, int(max_feature_track_age), (prm or TrackParams()).c())
        ns = C.c_int32(); nk = C.c_int32()
        self._ck(self.lib.dynofront_klt_track_fb(self.h, _p(pg), _p(cg), n, _p(p0), _p(nxt), _p(st), _p(back), C.byref(pc), _p(age), _p(keep),
                                                 C.byref(ns), C.byref(nk), C.byref(ms)))
        self.last_ms = ms.value; self.last_counts = (ns.value, nk.value)
        return nxt, st, back, (keep if check else None)

    def stereo_track(self, left_gray, right_gray, left_pts, fx, baseline):
        """FeatureTracker::stereoTrack without its RANSAC: (right_pts, status, depth, valid)"""
        lg = np.ascontiguousarray(left_gray, dtype=np.uint8); rg = np.ascontiguousarray(right_gray, dtype=np.uint8)
        p0 = np.ascontiguousarray(left_pts, dtype=np.float32).reshape(-1, 2); n = p0.shape[0]
        rp = np.zeros((n, 2), np.float32); st = np.zeros(n, np.uint8); depth = np.zeros(n); valid = np.zeros(n, np.uint8); ms = C.c_float()
        self._ck(self.lib.dynofront_stereo_track(self.h, _p(lg), _p(rg), n, _p(p0), _p(rp), _p(st), float(fx), float(baseline), _p(depth), _p(valid), C.byref(ms)))
        self.last_ms = ms.value
        return rp, st, depth, valid

    def klt_last_min_eig(self, n):
        out = np.zeros((n, 2), np.float32)
        self._ck(self.lib.dynofront_klt_last_min_eig(self.h, n, _p(out)))
        return out

    def track_static_flow(self, prev_pred_kp, prev_age, prev_usable, det_xy, cell_size, max_features, next_tracklet_id):
        """ExternalFlowFeatureTracker::trackStatic on the frame given to set_frame.  Returns a dict of per-feature arrays."""
        kp = np.ascontiguousarray(prev_pred_kp, dtype=np.float64).reshape(-1, 2); n = kp.shape[0]
        age = np.ascontiguousarray(prev_age, dtype=np.int32); use = np.ascontiguousarray(prev_usable, dtype=np.uint8)
        det = np.ascontiguousarray(det_xy, dtype=np.int32).reshape(-1, 2); m = det.shape[0]
        acc = np.zeros(n, np.uint8); fl = np.zeros((n, 2)); pk = np.zeros((n, 2)); oage = np.zeros(n, np.int32)
        dacc = np.zeros(m, np.uint8); dfl = np.zeros((m, 2)); dpk = np.zeros((m, 2)); dtid = np.zeros(m, np.int64)
        nid = C.c_int64(int(next_tracklet_id)); nt = C.c_int32(); nd = C.c_int32()
        self._ck(self.lib.dynofront_track_static_flow(self.h, n, _p(kp), _p(age), _p(use), m, _p(det), int(cell_size), int(max_features), C.byref(nid),
                                                      _p(acc), _p(fl), _p(pk), _p(oage), _p(dacc), _p(dfl), _p(dpk), _p(dtid), C.byref(nt), C.byref(nd)))
        return dict(acc=acc, flow=fl, pred=pk, age=oage, det_acc=dacc, det_flow=dfl, det_pred=dpk, det_tracklet=dtid,
                    next_tracklet_id=nid.value, n_tracked=nt.value, n_detected=nd.value)

    def pyramid_level(self, which, level):
        w = C.c_int32(); h = C.c_int32()
        self._ck(self.lib.dynofront_get_pyramid_level(self.h, which, level, C.byref(w), C.byref(h), None, None))
        img = np.zeros((h.value, w.value), np.uint8); der = np.zeros((h.value, w.value, 2), np.int16)
        self._ck(self.lib.dynofront_get_pyramid_level(self.h, which, level, C.byref(w), C.byref(h), _p(img), _p(der)))
        return img, der
