"""CPU ORACLE (TEST INFRASTRUCTURE, NOT PRODUCT) for sampleDynamic after the candidate scan (DESIGN.md section 8f-4).

Literal Python restatement of
  * AdaptiveNonMaximumSuppression::suppressNonMax(RangeTree)   dynosam/src/frontend/anms/NonMaximumSupression.cc:45-93,
    with the ranking taken from cv2.sortIdx itself
  * anms::RangeTree                                            dynosam/src/frontend/anms/anms.cc:278-362, C semantics
  * the tail of FeatureTracker::sampleDynamic                  dynosam/src/frontend/vision/FeatureTracker.cc:955-1015
The candidate scan is oracle/frontend_oracle.py's.  RangeTree is pinned against the reference's own anms.cc, compiled by
oracle/anms_ref/Makefile, and against tests/golden/anms_rangetree.npz (tests/test_sample_dynamic.py).
"""
from __future__ import annotations

import numpy as np

from oracle.frontend_oracle import TrackParams, sample_dynamic_candidates


def _c_int(v: float) -> int:
    """double -> int as x86-64 cvttsd2si: truncation; NaN and out-of-range give INT_MIN."""
    import math
    if math.isnan(v) or v >= 2.0**31 or v < -2.0**31:
        return -2**31
    return int(v)


def _round_half_away(v) -> float:
    """C round(): halves away from zero, exact."""
    import math
    if not math.isfinite(v):
        return float(v)
    a = abs(v); t = math.floor(a)
    if a - t >= 0.5:
        t += 1
    return math.copysign(float(t), v)


def anms_search_range(n: int, K: int, tolerance: float, cols: int, rows: int):
    """The binary-search set-up of anms::RangeTree (anms.cc:281-310) with C semantics: (high, low, Kmin, Kmax)."""
    import math
    exp1 = rows + cols + 2*K                                                    # int
    exp2 = 4*cols + 4*K + 4*rows*K + rows*rows + cols*cols - 2*rows*cols + 4*rows*cols*K    # long long
    exp3 = math.sqrt(exp2) if exp2 >= 0 else float("nan")
    exp4 = float(K - 1)
    with np.errstate(divide="ignore", invalid="ignore"):
        q1 = np.float64(exp1 + exp3)/np.float64(exp4); q2 = np.float64(exp1 - exp3)/np.float64(exp4)
    sol1 = -_round_half_away(float(q1)); sol2 = -_round_half_away(float(q2))
    high = _c_int(sol1 if sol1 > sol2 else sol2)
    low = _c_int(math.floor(math.sqrt(n/K))) if K > 0 else -2**31              # (K = 0: sqrt(+inf) -> INT_MIN)
    f = np.float32
    kt = f(K)*f(tolerance)                                                      # float: tolerance is float
    kmin = int(_round_half_away(float(f(f(K) - kt)))); kmax = int(_round_half_away(float(f(f(K) + kt))))
    return high, low, kmin, kmax


def anms_range_tree(xy, K: int, tolerance: float, cols: int, rows: int):
    """anms::RangeTree (anms.cc:278-362), literal: xy[n][2] float32 in the order the reference walks them (after the
    cv::sortIdx ranking).  Returns the positions (into xy) of the selected points, in selection order.  K <= 0 returns
    nothing (the reference's K = 0 is undefined behaviour; see DESIGN.md)."""
    xy = np.asarray(xy, dtype=np.float32).reshape(-1, 2)
    n = len(xy)
    if n == 0 or K <= 0:
        return []
    high, low, kmin, kmax = anms_search_range(n, K, tolerance, cols, rows)
    cx = xy[:, 0].astype(np.int64); cy = xy[:, 1].astype(np.int64)           # rangetree<u16, u16> stores truncated cells
    result, prevwidth = [], -1
    while True:
        d = high - low
        width = low + (d//2 if d >= 0 else -((-d)//2))                          # C division truncates toward zero
        if width == prevwidth or low > high:
            return result                                                       # the previous iteration's selection
        included = np.ones(n, bool)
        result = []
        w = np.float32(width)
        for i in range(n):
            if not included[i]:
                continue
            included[i] = False
            result.append(i)
            minx = int(xy[i, 0] - w); maxx = int(xy[i, 0] + w)                  # float arithmetic, then int truncation
            miny = int(xy[i, 1] - w); maxy = int(xy[i, 1] + w)
            minx = max(minx, 0); miny = max(miny, 0)
            included[(cx >= minx) & (cx <= maxx) & (cy >= miny) & (cy <= maxy)] = False     # treeANMS.search: inclusive box
        if kmin <= len(result) <= kmax:
            return result
        if len(result) < kmin:
            high = width - 1
        else:
            low = width + 1
        prevwidth = width


def anms_priority_order(n: int):
    """cv::sortIdx over n equal int responses, SORT_DESCENDING (NonMaximumSupression.cc:45-57): the walk order."""
    import cv2
    if n == 0:
        return np.zeros(0, np.int64)
    return cv2.sortIdx(np.zeros((1, n), np.int32), cv2.SORT_EVERY_ROW | cv2.SORT_DESCENDING).ravel().astype(np.int64)


def sample_dynamic(flow, motion_mask, detection_mask, objects, num_track, max_features, prm: TrackParams, next_tracklet_id: int,
                   tolerance=0.01):
    """FeatureTracker::sampleDynamic (FeatureTracker.cc:864-1015): candidate scan, suppressNonMax(RangeTree) per object
    with K = max(max_features - num_track, 0), then the new features (age 0, key-point (j, i), measured flow, predicted
    key-point) with tracklet ids handed out in the order of `objects`.  Returns a dict of per-object lists and per-feature
    arrays, the same layout as FeatureTrackerGPU.sample_dynamic."""
    rows, cols = motion_mask.shape
    cand, zero = sample_dynamic_candidates(flow, motion_mask, detection_mask, objects, prm)
    kp, fl, pred, tid, obj, n_sel = [], [], [], [], [], []
    for o, nt in zip(objects, num_track):
        c = cand[int(o)]
        order = anms_priority_order(len(c))
        ranked = [c[k] for k in order]
        xy = np.array([(p % cols, p//cols) for p in ranked], np.float32).reshape(-1, 2)
        sel = anms_range_tree(xy, max(int(max_features) - int(nt), 0), tolerance, cols, rows)
        n_sel.append(len(sel))
        for s in sel:
            p = ranked[s]; i, j = p//cols, p % cols
            fx = float(flow[i, j, 0]); fy = float(flow[i, j, 1])
            kp.append((float(j), float(i))); fl.append((fx, fy)); pred.append((float(j) + fx, float(i) + fy))
            tid.append(next_tracklet_id); next_tracklet_id += 1; obj.append(int(o))
    return dict(candidates=np.array([len(cand[int(o)]) for o in objects], np.int32), zero_flow=np.array([zero[int(o)] for o in objects], np.int32),
                selected=np.array(n_sel, np.int32), keypoint=np.array(kp, np.float64).reshape(-1, 2), flow=np.array(fl, np.float64).reshape(-1, 2),
                predicted=np.array(pred, np.float64).reshape(-1, 2), tracklet=np.array(tid, np.int64), object=np.array(obj, np.int32),
                next_tracklet_id=next_tracklet_id)
