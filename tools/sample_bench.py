#!/usr/bin/env python
"""sample_bench.py -- sampleDynamic after the candidate scan: dynofront_sample_dynamic against the path it replaces.

Per C4 frame (1242x375 synthetic stream, 10 objects, K = max_dynamic_features_per_frame = 200 per object, tolerance
0.01), after trackDynamic has left its detection mask on the device:
  device   dynofront_sample_dynamic: scan -> RangeTree ANMS -> new features, one call, one synchronisation;
           its device time (CUDA events) and the host time per call;
  replaced dynofront_sample_candidates (device scan, every candidate index copied to the host), then per object the
           cv::sortIdx ranking and the reference's own anms::RangeTree (oracle/_ref/libanms_ref.so, compiled from the
           DynOSAM sources) and the feature construction on the host: on one core, and with the objects spread over all
           cores (a thread per object; the ctypes call releases the GIL).
Both paths are checked to select the same features on every frame.  Prints one JSON line.
    python tools/sample_bench.py [--frames 200] [--warmup 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from dynosam_b200.synth_frames import SyntheticStream, W, H  # noqa: E402

N_OBJ, K, TOL = 10, 200, 0.01


def ref_lib():
    path = os.path.join(ROOT, "oracle", "_ref", "libanms_ref.so")
    if not os.path.exists(path):
        raise SystemExit(f"{path} is missing: build() compiles it from a DynOSAM checkout (oracle/anms_ref/Makefile)")
    L = C.CDLL(path)
    L.anms_ref_range_tree.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_void_p]
    return L


def frame_inputs(st, k, rng):
    """flow / mask of frame k and the previous dynamic features (predicted into frame k) that trackDynamic consumes"""
    _, m0, f0 = st.frame(k - 1); _, m1, f1 = st.frame(k)
    kps, labs = [], []
    for lab in range(1, N_OBJ + 1):
        ys, xs = np.nonzero(m0 == lab)
        if len(ys) == 0:
            continue
        sel = rng.choice(len(ys), size=min(150, len(ys)), replace=False)
        kps.append(np.stack([xs[sel] + 0.5 + f0[ys[sel], xs[sel], 0], ys[sel] + 0.5 + f0[ys[sel], xs[sel], 1]], 1)); labs.append(np.full(len(sel), lab, np.int32))
    kp = np.concatenate(kps); lab = np.concatenate(labs)
    ok = (kp[:, 0] > 1) & (kp[:, 0] < W - 1) & (kp[:, 1] > 1) & (kp[:, 1] < H - 1)
    n = int(ok.sum())
    return np.ascontiguousarray(m1, np.int32), np.ascontiguousarray(f1, np.float32), (kp[ok], lab[ok], rng.integers(0, 21, n).astype(np.int32), np.arange(n, dtype=np.int64))


def host_path(t, prm, objects, flow, L, pool, next_id):
    """the replaced path: device scan + candidate D2H, then ranking, RangeTree and construction on the host"""
    import cv2
    t0 = time.perf_counter()
    cand, _ = t.sample_candidates(objects, prm, capacity=W*H//2)
    t1 = time.perf_counter()

    def one(o):
        c = cand[o]
        if len(c) == 0:
            return np.zeros(0, np.int64)
        order = cv2.sortIdx(np.zeros((1, len(c)), np.int32), cv2.SORT_EVERY_ROW | cv2.SORT_DESCENDING).ravel()
        ranked = c[order]
        xy = np.ascontiguousarray(np.stack([ranked % W, ranked//W], 1), np.float32); out = np.zeros(len(c), np.int32)
        m = L.anms_ref_range_tree(xy.ctypes.data, len(c), K, TOL, W, H, out.ctypes.data)
        return ranked[out[:m]].astype(np.int64)
    sel = list(pool.map(one, objects)) if pool is not None else [one(o) for o in objects]
    p = np.concatenate(sel)
    kp = np.stack([p % W, p//W], 1).astype(np.float64)
    fl = flow.reshape(-1, 2)[p].astype(np.float64)
    feats = dict(keypoint=kp, flow=fl, predicted=kp + fl, tracklet=next_id + np.arange(len(p), dtype=np.int64))
    t2 = time.perf_counter()
    return feats, t1 - t0, t2 - t1


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                            timeout=30).stdout.strip()
    except Exception as e:                                        # noqa: BLE001
        pl = f"not read ({e.__class__.__name__})"
    return name, pl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=200); ap.add_argument("--warmup", type=int, default=5); ap.add_argument("--out")
    args = ap.parse_args()
    from dynosam_b200.frontend import FeatureTrackerGPU, TrackParams
    L = ref_lib()
    name, power = gpu_info()
    st = SyntheticStream(n_objects=N_OBJ, seed=42); rng = np.random.default_rng(42)
    t = FeatureTrackerGPU(W, H); prm = TrackParams()
    objects = list(range(1, N_OBJ + 1)); num_track = [0]*N_OBJ
    ncores = os.cpu_count() or 1
    pool = ThreadPoolExecutor(max_workers=min(ncores, N_OBJ))
    rec = {k: [] for k in ("dev_ms", "e2e_ms", "scan_d2h_ms", "host_1core_ms", "host_allcores_ms", "candidates", "selected")}
    for k in range(1, args.frames + args.warmup + 1):
        m1, f1, (kp, lab, age, tid) = frame_inputs(st, k, rng)
        t.set_frame(f1, m1, None)
        t.track_dynamic(kp, lab, age, tid, prm, 10**6, want_masks=False)       # leaves the detection mask on the device
        t0 = time.perf_counter()
        r = t.sample_dynamic(objects, num_track, prm, 10**6, max_features=K, tolerance=TOL)
        e2e = time.perf_counter() - t0
        dev = t.last_ms
        f_one, scan1, host1 = host_path(t, prm, objects, f1, L, None, 10**6)
        f_all, scan2, host2 = host_path(t, prm, objects, f1, L, pool, 10**6)
        for f in (f_one, f_all):
            for key in f:
                assert np.array_equal(f[key], r[key]), (k, key)
        if k > args.warmup:
            rec["dev_ms"].append(dev); rec["e2e_ms"].append(1e3*e2e); rec["scan_d2h_ms"].append(1e3*(scan1 + scan2)/2)
            rec["host_1core_ms"].append(1e3*host1); rec["host_allcores_ms"].append(1e3*host2)
            rec["candidates"].append(int(r["candidates"].sum())); rec["selected"].append(int(r["selected"].sum()))
    pool.shutdown()
    mean = {k: float(np.mean(v)) for k, v in rec.items()}
    med = {k: float(np.median(v)) for k, v in rec.items()}
    out = {"metric": "sampleDynamic after the scan, ms per C4 frame", "frames": args.frames, "gpu": name, "power_limit": power, "host_cores": ncores,
           "workload": f"C4 1242x375 synthetic stream, {N_OBJ} objects, K = {K} per object, tolerance {TOL}, detection mask from trackDynamic",
           "device_sample_dynamic_ms": {"mean": mean["dev_ms"], "median": med["dev_ms"]},
           "device_sample_dynamic_end_to_end_ms": {"mean": mean["e2e_ms"], "median": med["e2e_ms"]},
           "replaced_scan_and_candidate_d2h_ms": {"mean": mean["scan_d2h_ms"], "median": med["scan_d2h_ms"]},
           "replaced_host_anms_1core_ms": {"mean": mean["host_1core_ms"], "median": med["host_1core_ms"]},
           "replaced_host_anms_allcores_ms": {"mean": mean["host_allcores_ms"], "median": med["host_allcores_ms"]},
           "replaced_total_1core_ms": mean["scan_d2h_ms"] + mean["host_1core_ms"],
           "replaced_total_allcores_ms": mean["scan_d2h_ms"] + mean["host_allcores_ms"],
           "candidates_per_frame": mean["candidates"], "selected_per_frame": mean["selected"], "outputs_equal": True}
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
