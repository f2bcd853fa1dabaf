#!/usr/bin/env python
"""bench.py -- LM iterations/s of the B200-native DynOSAM batch solver (BASELINE.json metric).

One "step" = one outer Levenberg-Marquardt iteration (1 materialising linearize + >= 1 damped Schur solve +
>= 1 chi^2 sweep) on the synthetic 10k-key-frame / 100-object / 2M-landmark dynamic graph (BASELINE.json
configs[4]; it fits one B200, so it is also the N=1 workload).  N > 1: landmarks are sharded in time over the ranks and
the reduced solve is distributed (one cell of the banded system per rank: a reduce per cell, an all-reduce of the small
boundary-separator system and of the pose update); strong scaling: total work fixed.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C5|C3|C2|C1] [--scale s] [--dump-outputs DIR]
    python bench.py --impl reference ...    # CPU arm: the oracle port on the host cores, same config at full size

--dump-outputs DIR writes what the last timed LM iteration left in the solver, as a caller reads it back, to DIR/*.npy
(float64): pose [n_pose, 12], point [n_point, 3], flow [n_flow, 2] (only when the graph has optical-flow variables) and
lm_stats = [chi^2 initial, chi^2 final, lambda final, iterations, inner iterations].  An empty array is not written.  Above
64 MB in all, each array keeps a fixed seeded sample of its rows.  The inputs depend on the arguments alone, so two builds
can be compared output for output.

The JSON line carries `roofline` (Jacobian-build kernel vs measured HBM bandwidth), `reduced_solve` (vs the fp64 rate
measured on the box), `e2e` (through the C ABI from host arrays), `cpu_baseline` + `parity_check` (one full-size LM
iteration of the oracle port, compared with the GPU's first iteration) and `configs` (C2, C3, front-end C4).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from dynosam_b200 import synth  # noqa: E402
from dynosam_b200.problem import Problem, FactorBlock, ARITY, SLOT_CLASS  # noqa: E402

METRIC = "LM iters/sec on 10k-pose/2M-landmark dynamic BA"
UNIT = "LM iterations/s"


def _solver_positions(p: Problem) -> np.ndarray:
    order = np.argsort(p.pose_order, kind="stable") if p.pose_order is not None else np.arange(p.n_pose)
    pos = np.empty(p.n_pose, dtype=np.int64); pos[order] = np.arange(p.n_pose)
    return pos


def _point_groups(p: Problem) -> np.ndarray:
    """Landmark groups as libdynoba's symbolic phase forms them: points joined by a factor with more than one point
    slot (the points of a WCME / WCPE tracklet chain) are eliminated together.  Returns the group id of every point."""
    npt = p.n_point
    edges = []
    for b in p.blocks:
        ls = [k for k, c in enumerate(SLOT_CLASS[b.type]) if c == 1]
        for k in ls[1:]:
            edges.append(np.stack([b.idx[:, ls[0]], b.idx[:, k]], 1))
    if not edges or not npt:
        return np.arange(npt, dtype=np.int64)
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    e = np.concatenate(edges).astype(np.int64)
    _, group = connected_components(coo_matrix((np.ones(e.shape[0], dtype=np.int8), (e[:, 0], e[:, 1])), shape=(npt, npt)), directed=False)
    return group.astype(np.int64)


def problem_bandwidth(p: Problem) -> int:
    """Scalar half-bandwidth of the reduced system in the solver ordering (same rule as libdynoba's finalize): the
    widest spread of pose positions over one landmark group, or over one pose-only factor."""
    pos = _solver_positions(p)
    group = _point_groups(p)
    ng = int(group.max(initial=-1)) + 1
    gmin = np.full(ng, np.iinfo(np.int64).max); gmax = np.full(ng, -1)
    spread = 0
    for b in p.blocks:
        cls = SLOT_CLASS[b.type]
        pslots = [k for k, c in enumerate(cls) if c == 0]
        lslots = [k for k, c in enumerate(cls) if c == 1]
        if not pslots or not b.n:
            continue
        pp = pos[b.idx[:, pslots]]
        lo, hi = pp.min(1), pp.max(1)
        spread = max(spread, int((hi - lo).max(initial=0)))        # (also the single-factor spread of flow-variable factors)
        if lslots:
            g = group[b.idx[:, lslots[0]]]
            np.minimum.at(gmin, g, lo); np.maximum.at(gmax, g, hi)
    ok = gmax >= 0
    if ok.any():
        spread = max(spread, int((gmax[ok] - gmin[ok]).max()))
    return 6*spread + 5


def shard_problem(p: Problem, rank: int, world: int) -> Problem:
    """Time shard of rank `rank`.  Landmarks that share a factor (the points of a WCME / WCPE tracklet chain) form one
    group; a group, with all its factors, goes to the rank whose slice of the (frame-ordered) pose axis holds the
    group's first pose, and a pose-only factor to the rank of its first pose.  Poses are replicated.  Contiguous time
    slices keep a rank's contribution to the reduced system inside the cells it owns (plus a halo one co-visibility
    window wide), which is what the library's per-cell reduce moves.  q.meta["kept_points"] = mask of the kept points."""
    if world == 1:
        return p
    pos = _solver_positions(p)
    group = _point_groups(p)
    ngroup = int(group.max(initial=-1)) + 1
    first = np.full(ngroup, np.iinfo(np.int64).max)
    for b in p.blocks:
        cls = SLOT_CLASS[b.type]
        ls = [k for k, c in enumerate(cls) if c == 1]; ps = [k for k, c in enumerate(cls) if c == 0]
        if ls and ps:
            np.minimum.at(first, group[b.idx[:, ls[0]]], pos[b.idx[:, ps]].min(1))
    first[first == np.iinfo(np.int64).max] = 0
    # slices of the pose axis: the library's own cut of the reduced system into per-rank cells when it is there (so that a
    # rank's landmarks contribute to the cells it owns), else uniform
    try:
        from dynosam_b200.binding import plan_partition
        bounds = plan_partition(p.n_pose, problem_bandwidth(p), world).astype(np.int64)
    except Exception:
        bounds = None
    if bounds is not None and (np.diff(bounds) > 0).all():
        owner_of_pos = lambda q: np.clip(np.searchsorted(bounds, q, side="right") - 1, 0, world - 1)
    else:
        owner_of_pos = lambda q: np.minimum(q*world//max(p.n_pose, 1), world - 1)
    keep_pt = owner_of_pos(first)[group] == rank
    new_idx = np.cumsum(keep_pt) - 1
    blocks = []
    for b in p.blocks:
        cls = SLOT_CLASS[b.type]
        ls = [k for k, c in enumerate(cls) if c == 1]; ps = [k for k, c in enumerate(cls) if c == 0]
        if any(c == 2 for c in cls):          # optical-flow variables are not sharded: such blocks stay on rank 0
            if rank == 0:
                blocks.append(b)
            continue
        if ls:
            sel = keep_pt[b.idx[:, ls[0]]]
            assert all(np.array_equal(keep_pt[b.idx[:, k]], sel) for k in ls[1:]), "a factor straddles two landmark shards"
        else:
            sel = owner_of_pos(pos[b.idx[:, ps]].min(1)) == rank
        idx = b.idx[sel].copy()
        for k in ls:
            idx[:, k] = new_idx[idx[:, k]]
        blocks.append(FactorBlock(b.type, idx, None if b.meas is None else b.meas[sel],
                                  b.sigma if b.sigma_bcast else b.sigma[sel], b.robust_k,
                                  None if b.aux_idx is None else b.aux_idx[sel]))
    q = Problem(p.pose, p.point[keep_pt], flow=p.flow, aux_pose=p.aux_pose, calib=p.calib, blocks=blocks, pose_order=p.pose_order,
                pose_keys=p.pose_keys, point_keys=None if p.point_keys is None else p.point_keys[keep_pt], meta=dict(p.meta))
    q.meta["kept_points"] = keep_pt
    return q


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index; self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill(); out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def dump_outputs(directory, arrays, budget=64 << 20):
    """the non-empty arrays as float64 DIR/<name>.npy; above `budget` bytes in all, every 2-D array keeps the same fraction
    of its rows, a sample drawn from a fixed seed (the same rows on every run with the same arguments)."""
    os.makedirs(directory, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    arrays = {k: a for k, a in arrays.items() if a.size}
    total = sum(a.nbytes for a in arrays.values())
    frac = min(1.0, (budget - 4096*len(arrays))/total) if total else 1.0     # (4 KB per file covers the .npy header)
    for name, a in arrays.items():
        if frac < 1.0 and a.ndim == 2:
            keep = np.random.default_rng(0).choice(a.shape[0], max(1, int(a.shape[0]*frac)), replace=False)
            a = a[np.sort(keep)]
        np.save(os.path.join(directory, name + ".npy"), a)


def cpu_oracle_rate(cfg_name, formulation, seed, scale, iters, threads):
    """`iters` LM iterations of the CPU oracle (port of the reference's GTSAM-4.2 path) on the named config at `scale`
    (1.0 = the stated workload, no extrapolation).  Returns the measured rate and the chi^2 trace ends."""
    from oracle import oracle as O
    os.environ["OMP_NUM_THREADS"] = str(threads)
    ps = synth.make_config(cfg_name, formulation=formulation, seed=seed, scale=scale)
    o = O.OracleProblem(ps)
    t0 = time.perf_counter()
    st = o.optimize(max_iterations=iters, rel_tol=0.0, abs_tol=0.0)
    dt = time.perf_counter() - t0
    return dict(rate=max(st["iterations"], 1)/dt, seconds=dt, iterations=st["iterations"], inner=st["inner_iterations"],
                error_initial=st["error_initial"], error_final=st["error_final"], n_factors=ps.n_factors, frames=ps.meta["n_frames"],
                stats={k: st[k] for k in ("t_linearize", "t_schur", "t_solve", "t_backsub", "t_error")})


def _cpu_run(cfg_name, formulation, seed, scale, iters, threads, timeout):
    """cpu_oracle_rate in a clean process (own OpenMP runtime, no CUDA context)."""
    code = ("import json,sys; sys.path.insert(0, %r); import bench; "
            "print(json.dumps(bench.cpu_oracle_rate(%r, %r, %d, %r, %d, %d)))" % (ROOT, cfg_name, formulation, seed, scale, iters, threads))
    env = dict(os.environ, OMP_NUM_THREADS=str(threads)); env.pop("OMP_PROC_BIND", None)
    try:
        pr = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=timeout)
        return json.loads(pr.stdout.strip().splitlines()[-1])
    except Exception:
        return None


_THREADS_FILE = os.path.join("/tmp", "dynoba_cpu_threads.json")


def cpu_threads(cfg_name, formulation, seed):
    """Thread count of the CPU legs: the fastest of {8, 16, 32, all} on a 1/50 time slice of the workload (the box's
    OpenMP scaling depends on what the container is really allowed to use).  Chosen once per box and reused by both CPU
    legs (`--impl reference` and the cpu_baseline of the product arm) through a file in /tmp."""
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        d = json.load(open(_THREADS_FILE))
        if d.get("ncpu") == ncpu and d.get("config") == [cfg_name, formulation]:
            return int(d["threads"]), d["probed"]
    except Exception:
        pass
    cands = sorted({t for t in (8, 16, 32, ncpu) if t <= ncpu} or {ncpu})
    best_t, best_rate = cands[0], -1.0
    for t in cands:
        r = _cpu_run(cfg_name, formulation, seed, 0.02, 1, t, 120)
        if r and r["rate"] > best_rate:
            best_t, best_rate = t, r["rate"]
    try:
        json.dump({"ncpu": ncpu, "config": [cfg_name, formulation], "threads": best_t, "probed": cands}, open(_THREADS_FILE, "w"))
    except Exception:
        pass
    return best_t, cands


def cpu_oracle_leg(cfg_name, formulation, seed, scale, iters):
    threads, probed = cpu_threads(cfg_name, formulation, seed)
    r = _cpu_run(cfg_name, formulation, seed, scale, iters, threads, 1500 + 120*iters)
    if r is None:
        r = dict(rate=float("nan"), seconds=float("nan"), iterations=0, inner=0, error_initial=float("nan"), error_final=float("nan"),
                 n_factors=0, frames=0, stats={})
    r["threads"] = threads; r["probed"] = probed
    r["sample"] = (f"{cfg_name}{'' if scale == 1.0 else f' at {scale:g} scale'} ({r['frames']} key-frames, {r['n_factors']} factors): "
                   f"{r['iterations']} LM iteration(s), {r['inner']} damped solves, in {r['seconds']:.1f} s on {threads} threads "
                   f"(fastest of {probed} on a 1/50 slice); no extrapolation")
    return r


# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant Jacobian-build kernel, from an `ncu --set full`
# capture of this very launch (a counter value cannot be measured inside a timed run); the capture is named next to it.
# Only valid for the exact launch that was profiled: C5 at full scale on one GPU; anything else reports null.
NCU_TRAFFIC = {("C5", "hybrid", 5, 11376204): (576.973e6 + 4550.677e6, "profiles/r02_final.md section 3 (ncu --set full of the same launch)")}


def ncu_traffic(args, world, blk):
    if world != 1 or args.scale != 1.0:
        return None, None
    v = NCU_TRAFFIC.get((args.config, args.formulation, int(blk.type), int(blk.n)))
    return (float(v[0]), v[1]) if v else (None, None)


def quick_config_rate(cfg_name, formulation, seed, device, steps=3):
    """LM iterations/s of another BASELINE config on one GPU (graph resident, device-timed), for the `configs` object."""
    from dynosam_b200.binding import Solver, default_params
    p = synth.make_config(cfg_name, formulation=formulation, seed=seed)
    s = Solver(p, device=device)
    prm = dict(relative_error_tol=0.0, absolute_error_tol=0.0)
    s.optimize(default_params(max_iterations=1, **prm)); s.reset_values()
    st = s.optimize(default_params(max_iterations=steps, **prm))
    info = s.info()
    s.close()
    return {"workload": f"{cfg_name}: {p.meta['n_frames']} key-frames / {p.meta['n_objects']} objects / {p.n_point} landmarks, {p.n_factors} factors",
            "value": st["iterations"]/(st["ms_total"]*1e-3), "unit": UNIT, "steps": st["iterations"], "inner_iterations": st["inner_iterations"],
            "ms_per_step": st["ms_total"]/max(st["iterations"], 1), "chi2": [st["error_initial"], st["error_final"]],
            "reduced_dim": info["reduced_dim"], "bandwidth": info["bandwidth"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="dynoba", choices=["dynoba", "reference"])
    ap.add_argument("--config", default="C5")
    ap.add_argument("--formulation", default="hybrid")
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true", help="skip the C2 / C3 / front-end lines of the `configs` object")
    ap.add_argument("--cells", type=int, default=0, help="cells of the reduced solve (0 automatic, -1 plain band)")
    ap.add_argument("--replicated-solve", action="store_true", help="N > 1: all-reduce the reduced system and solve it on every rank")
    ap.add_argument("--tune", default="", help="name=value,... performance parameters (dynoba_set_tuning)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="", help="write the values and LM statistics of the last timed "
                    "iteration to DIR/*.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    K, W = args.steps, max(args.warmup, 0)
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = synth.CONFIGS[args.config]
    config = {"workload": f"{args.config}: synthetic {cfg['n_frames']} key-frames / {cfg['n_objects']} objects / "
                          f"{cfg['n_static']} static + {cfg['n_dynamic']} dynamic landmarks, {args.formulation} formulation"
                          + (f", scale {args.scale}" if args.scale != 1.0 else ""),
              "parallelism": (f"landmarks sharded in time x{world}; reduced solve " + ("replicated" if args.replicated_solve else "distributed: one cell of the band per rank, "
                              "reduce per cell + all-reduce of the boundary system")) if world > 1 else "1 GPU",
              "seed": args.seed,
              "l2_policy": "working set (Jacobian tiles, GBs) >> 126 MB L2; no explicit flush",
              "noise": "sigma_point 0.2, Huber k 1e-4, LM defaults with rel/abs tol 0 so that exactly K iterations run",
              "timed_region": "LM iterations 1..K from the initial values (after W warm-up iterations and a value reset)"}

    if args.impl == "reference":
        # CPU arm: the reference's own toolchain (GTSAM) is absent, so this is the oracle port (cpu_baseline.kind "port"),
        # on the stated workload at full size; a step = one LM iteration (at full size ~20 s of CPU work each)
        if rank != 0:
            return
        r = cpu_oracle_leg(args.config, args.formulation, args.seed, args.scale, K)
        config["timed_region"] = f"LM iterations 1..{K} from the initial values on the host cores"
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": r["rate"], "unit": UNIT, "n_gpus": args.gpus, "steps": r["iterations"],
                          "warmup": 0, "ms_per_step": 1e3/r["rate"], "higher_is_better": True, "scaling": "strong",
                          "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                          "inner_iterations": r["inner"], "chi2": [r["error_initial"], r["error_final"]],
                          "cpu_baseline": {"value": r["rate"], "unit": UNIT, "cores": r["threads"], "kind": "port", "sample": r["sample"], "breakdown_s": r["stats"]},
                          "e2e": {"value": r["rate"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (libdynoba has no CPU path)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from dynosam_b200.binding import Solver, default_params

    full = synth.make_config(args.config, formulation=args.formulation, seed=args.seed, scale=args.scale)
    bw = problem_bandwidth(full) if world > 1 else 0
    prob = shard_problem(full, rank, world)

    def _tensor(dev, n):
        class _A:  # noqa
            __cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (dev, False), "version": 3, "strides": None}
        return torch.as_tensor(_A(), device=f"cuda:{local}")

    def allreduce_cb(dev, n, stream):
        with torch.cuda.stream(torch.cuda.ExternalStream(stream)):
            dist.all_reduce(_tensor(dev, n))

    def reduce_cb(dev, n, root, stream):
        with torch.cuda.stream(torch.cuda.ExternalStream(stream)):
            dist.reduce(_tensor(dev, n), dst=root)

    def new_solver(p):
        s = Solver(p, device=local)
        s.set_partition(args.cells)
        for kv in filter(None, args.tune.split(",")):
            k, v = kv.split("="); s.set_tuning(k, float(v))
        if world > 1:
            s.set_shard(rank, world, allreduce_cb, bw)
            if not args.replicated_solve:
                s.set_reduce(reduce_cb)
        return s

    prm = dict(relative_error_tol=0.0, absolute_error_tol=0.0)
    s = new_solver(prob)
    s.finalize()
    info = s.info()
    # ---- parity at the stated size (outside the timed region): chi^2 at the initial values and after the first LM
    # iteration, to be compared with the CPU oracle's first iteration below
    first = s.optimize(default_params(max_iterations=1, **prm))
    s.reset_values()
    if W:
        s.optimize(default_params(max_iterations=W, **prm))
        s.reset_values()      # the timed region is LM iterations 1..K from the initial values, like the CPU arm
    lin_ms = [s.linearize() for _ in range(3)]                      # whole Jacobian-build pass (after warm-up)
    # the dominant Jacobian-build kernel alone: the factor block with the most algorithmic bytes
    blk_stats = [s.linearize_block(bi) for bi in range(len(prob.blocks))]
    dom = int(np.argmax([b for _, b in blk_stats])) if blk_stats else 0
    dom_ms = [s.linearize_block(dom)[0] for _ in range(7)] if blk_stats else [0.0]
    dom_bytes = blk_stats[dom][1] if blk_stats else 0
    fp64_peak = s.fp64_rate()
    # ---- timed region: exactly K LM iterations, device-timed (CUDA events on the solver's stream), max over ranks
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    t0 = time.perf_counter()
    st = s.optimize(default_params(max_iterations=K, **prm))
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    if world > 1:
        dist.barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:          # (N > 1: rank 0's landmark shard)
        pose, point, flow = s.values()
        dump_outputs(args.dump_outputs, {"pose": pose, "point": point, "flow": flow, "lm_stats": [
            st["error_initial"], st["error_final"], st["lambda_final"], st["iterations"], st["inner_iterations"]]})
    ms = torch.tensor([st["ms_total"], wall*1e3], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms[0]); steps_done = st["iterations"]
    value = steps_done/(ms_total*1e-3) if ms_total > 0 else 0.0

    # ---- end-to-end through the C-ABI with host buffers: ingest (H2D) + K iterations + read-back (D2H)
    e2e = None
    if not args.no_e2e:
        s.close(); del s
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        s2 = new_solver(prob)
        s2.finalize()
        st2 = s2.optimize(default_params(max_iterations=K, **prm))
        pose, point, _ = s2.values()
        torch.cuda.synchronize()
        t_e2e = time.perf_counter() - t0
        tt = torch.tensor([t_e2e], dtype=torch.float64, device=f"cuda:{local}")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        h2d = prob.pose.nbytes + prob.point.nbytes + prob.aux_pose.nbytes + sum(
            b.idx.nbytes + (b.meas.nbytes if b.meas is not None else 0) + 8*b.sigma_dim*b.n + (b.aux_idx.nbytes if b.aux_idx is not None else 0)
            for b in prob.blocks)
        d2h = pose.nbytes + point.nbytes
        e2e = {"value": st2["iterations"]/float(tt[0]), "unit": UNIT, "h2d_bytes_per_step": int(h2d/max(K, 1)),
               "d2h_bytes_per_step": int(d2h/max(K, 1)), "note": "one ingest + read-back per optimize() call, amortised over K steps; "
               "includes the host-side symbolic phase (sorting / band layout)", "seconds": float(tt[0])}
        s2.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6650.0); peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback"
    lin = float(np.median(lin_ms))
    pass_ach = info["jacobian_bytes"]/(lin*1e-3)/1e9 if lin > 0 else 0.0
    dms = float(np.median(dom_ms))
    ach = dom_bytes/(dms*1e-3)/1e9 if dms > 0 else 0.0
    traffic, traffic_src = ncu_traffic(args, world, prob.blocks[dom])
    from dynosam_b200.problem import TYPE_NAMES
    solves = max(st["inner_iterations"], 1)
    chol_flops = float(info["reduced_dim"])*float(info["bandwidth"])**2
    solve_ms = st["ms_factor"]/solves
    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps_done, "warmup": W,
           "ms_per_step": ms_total/max(steps_done, 1), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f64", "data": "synthetic", "config": config, "clocks": clocks, "gpu_launches": int(st["kernel_launches"]),
           "inner_iterations": st["inner_iterations"], "chi2": [st["error_initial"], st["error_final"]],
           "reduced_dim": info["reduced_dim"], "bandwidth": info["bandwidth"], "n_factors_rank0": prob.n_factors,
           "phases_ms": {k: st[k] for k in ("ms_linearize", "ms_schur", "ms_factor", "ms_error", "ms_total")},
           "roofline": {"kernel": f"linearize_kernel<{TYPE_NAMES[prob.blocks[dom].type]}> (materialising Jacobian build of the largest factor block, "
                                  f"{prob.blocks[dom].n} factors)",
                        "bound": "hbm", "achieved": ach, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                        "frac": ach/peak if peak else None, "traffic": traffic, "traffic_source": traffic_src,
                        "algorithmic_bytes": int(dom_bytes), "ms_per_launch": dms,
                        "whole_pass": {"algorithmic_bytes": info["jacobian_bytes"], "ms": lin, "achieved": pass_ach,
                                       "frac": pass_ach/peak if peak else None,
                                       "note": "all factor blocks of one linearize() incl. the numerically differentiated smoothing factors and the final reduction"}},
           "reduced_solve": {"kernel": "band_cholesky_dataflow_kernel_v3 + band_backward_cluster_kernel (this rank's share)", "bound": "fp64 latency chain / DMMA",
                             "flops_per_solve": chol_flops, "note": "n*bw^2 of the plain band Cholesky, whole system; spiked chains do up to 4x that per column",
                             "ms_per_solve": solve_ms, "achieved_tflops": chol_flops/(solve_ms*1e-3)/1e12 if solve_ms > 0 else None,
                             "fp64_peak_tflops": fp64_peak, "fp64_peak_source": "dynoba_fp64_rate: register-only DFMA kernel on this GPU (MEASURED_PEAKS.json has no fp64 entry)",
                             "frac": chol_flops/(solve_ms*1e-3)/1e12/fp64_peak if solve_ms > 0 and fp64_peak > 0 else None}}
    if e2e:
        out["e2e"] = e2e
    if not args.no_cpu_baseline:
        # one LM iteration of the oracle port on the SAME workload at full size: the CPU baseline and, from the same run, the
        # parity check at the stated size (chi^2 at the initial values and after the first accepted step, 1e-6 relative)
        r = cpu_oracle_leg(args.config, args.formulation, args.seed, args.scale, 1)
        out["cpu_baseline"] = {"value": r["rate"], "unit": UNIT, "cores": r["threads"], "kind": "port", "sample": r["sample"], "breakdown_s": r["stats"]}
        rel0 = abs(first["error_initial"] - r["error_initial"])/max(abs(r["error_initial"]), 1e-300)
        rel1 = abs(first["error_final"] - r["error_final"])/max(abs(r["error_final"]), 1e-300)
        out["parity_check"] = {"workload": config["workload"], "against": "oracle port, same seeded graph, first LM iteration",
                               "chi2_initial": [first["error_initial"], r["error_initial"], rel0],
                               "chi2_after_first_iteration": [first["error_final"], r["error_final"], rel1],
                               "inner_iterations": [first["inner_iterations"], r["inner"]], "tolerance": 1e-6,
                               "ok": bool(rel0 <= 1e-6 and rel1 <= 1e-6 and first["inner_iterations"] == r["inner"])}
    if world == 1 and not args.no_extra_configs and args.scale == 1.0:
        # the other BASELINE configs, short runs (not the headline; the parity of these shapes is covered by tests/)
        extra = {}
        for name in ("C2", "C3"):
            if name != args.config:
                try:
                    extra[name] = quick_config_rate(name, args.formulation, args.seed, local)
                except Exception as e:  # pragma: no cover
                    extra[name] = {"error": str(e)}
        try:
            import bench_frontend
            extra["C4"] = bench_frontend.run_dynoba(200, 5)
        except Exception as e:  # pragma: no cover
            extra["C4"] = {"error": str(e)}
        out["configs"] = extra
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
