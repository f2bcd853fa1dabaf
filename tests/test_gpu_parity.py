"""GPU parity tests: the CUDA hot path (through the C-ABI) against the CPU oracle on the same seeded inputs.

Tolerances: north_star asks for <= 1e-6 relative on residuals / chi^2; element-wise Jacobians and rhs are
checked much tighter (1e-9 relative to the block's largest element) because both sides are fp64.
"""
import numpy as np
import pytest

from dynosam_b200 import synth
from dynosam_b200.problem import (BETWEEN6, FLOWPROJ2, HYBRID3, HYBRID_STEREO3, MOTIONPOSE3, POSE2POINT3, PRIOR6,
                                  SMOOTH_HYBRID6, SMOOTH_POSE6, STEREO3, TERNARY3, TYPE_NAMES, FactorBlock, Problem)

pytestmark = pytest.mark.gpu

REL_CHI2 = 1e-6


def _solver(p):
    from dynosam_b200.binding import Solver
    return Solver(p)


def _oracle(p):
    from oracle import oracle as O
    return O.OracleProblem(p)


_all_types_problem = synth.make_all_types_problem


def _check_linearization(p):
    s = _solver(p); o = _oracle(p)
    ms = s.linearize()
    assert ms > 0
    for bi, b in enumerate(p.blocks):
        A, bv = s.linearization(bi)
        Ao, bo = o.linearize_block(bi)
        sa = max(np.abs(Ao).max(), 1e-300); sb = max(np.abs(bo).max(), 1e-300)
        # numerically differentiated factors: both sides run the same central differences; rounding differs
        tol = 1e-6 if b.type in (MOTIONPOSE3, SMOOTH_HYBRID6, SMOOTH_POSE6) else 1e-9
        assert np.abs(A - Ao).max() <= tol*sa, (TYPE_NAMES[b.type], np.abs(A - Ao).max(), sa)
        assert np.abs(bv - bo).max() <= 1e-9*sb + 1e-12, TYPE_NAMES[b.type]
        e = s.factor_errors(bi); eo = o.error_block(bi)
        assert np.abs(e - eo).max() <= REL_CHI2*max(np.abs(eo).max(), 1e-300), TYPE_NAMES[b.type]
    assert abs(s.error() - o.error()) <= REL_CHI2*abs(o.error())
    s.close()


def test_linearize_every_factor_type():
    _check_linearization(_all_types_problem())


@pytest.mark.parametrize("formulation", ["hybrid", "wcme", "wcpe"])
def test_linearize_c1(formulation):
    _check_linearization(synth.make_config("C1", formulation=formulation))


def test_stereo_cheirality_on_device():
    from dynosam_b200 import lie
    I = lie.identity()[0]
    blk = FactorBlock(STEREO3, np.array([[0, 0], [0, 1]]), np.array([[300, 290, 170.0], [300, 290, 170.0]]), np.array([1.0]))
    p = Problem(I[None], np.array([[0.5, 0.2, 8.0], [0.5, 0.2, -8.0]]), blocks=[blk])
    s = _solver(p); s.linearize()
    A, bv = s.linearization(0)
    assert np.all(A[1] == 0) and np.allclose(bv[1], -2*p.calib[0])      # behind the camera: zero J, e = 2 fx
    Ao, bo = _oracle(p).linearize_block(0)
    assert np.allclose(A, Ao, rtol=1e-12, atol=1e-9) and np.allclose(bv, bo, rtol=1e-12, atol=1e-9)


def test_reduced_system_and_damped_solve_c1():
    p = synth.make_config("C1", formulation="hybrid")
    s = _solver(p); o = _oracle(p)
    lam = 1e-5
    S, g = s.reduced_system(lam)
    So, go, pos = o.reduced_dense(lam)
    perm = np.concatenate([6*pos[i] + np.arange(6) for i in range(p.n_pose)])
    So = So[np.ix_(perm, perm)]; go = go[perm]
    assert np.abs(S - So).max() <= 1e-9*np.abs(So).max()
    assert np.abs(g - go).max() <= 1e-9*np.abs(go).max()
    d = s.solve(lam)
    rc, do = o.schur_solve(lam)
    assert rc == 0
    assert np.linalg.norm(d - do) <= 1e-6*np.linalg.norm(do)
    # against the dense normal equations as well (independent of the Schur organisation)
    H, gg = o.dense_normal()
    dd = np.linalg.solve(H + lam*np.eye(H.shape[0]), gg)
    assert np.linalg.norm(d - dd) <= 1e-6*np.linalg.norm(dd)


def test_retract_matches_oracle():
    p = synth.make_config("C1", formulation="hybrid")
    s = _solver(p); o = _oracle(p)
    rng = np.random.default_rng(0)
    d = rng.normal(0, 0.05, 6*p.n_pose + 3*p.n_point)
    s.retract(d); o.retract(d)
    pose, point, _ = s.values()
    assert np.abs(pose - o.pose).max() < 1e-12 and np.abs(point - o.point).max() < 1e-12
    assert abs(s.error() - o.error()) <= REL_CHI2*o.error()


@pytest.mark.parametrize("robust", [True, False])
def test_lm_c1_matches_oracle(robust):
    p = synth.make_config("C1", formulation="hybrid", robust=robust)
    s = _solver(p); o = _oracle(p)
    st = s.optimize()
    so = o.optimize()
    assert abs(st["error_initial"] - so["error_initial"]) <= REL_CHI2*so["error_initial"]
    assert st["iterations"] == so["iterations"] and st["inner_iterations"] == so["inner_iterations"]
    assert abs(st["error_final"] - so["error_final"]) <= REL_CHI2*so["error_final"]
    pose, point, _ = s.values()
    assert np.abs(pose - o.pose).max() < 1e-6 and np.abs(point - o.point).max() < 1e-5
    assert st["kernel_launches"] > 0


def test_lm_static_only_medium():
    """configs[1] topology (static BA) at 1/50 scale: 40 key-frames, 10k landmarks."""
    p = synth.make_config("C2", scale=0.02)
    s = _solver(p); o = _oracle(p)
    st = s.optimize(max_iterations=6)
    so = o.optimize(max_iterations=6)
    assert st["iterations"] == so["iterations"]
    assert abs(st["error_final"] - so["error_final"]) <= REL_CHI2*so["error_final"]


def test_lm_hybrid_medium_properties():
    """configs[2] topology at 1/20 scale: chi^2 decreases monotonically over accepted steps, variables move
    towards the ground truth, and the result agrees with the oracle."""
    p = synth.make_config("C3", scale=0.05)
    s = _solver(p); o = _oracle(p)
    e0 = s.error()
    st = s.optimize(max_iterations=5)
    assert st["error_final"] < e0 and st["error_initial"] == pytest.approx(e0, rel=1e-12)
    so = o.optimize(max_iterations=5)
    assert st["iterations"] == so["iterations"]
    assert abs(st["error_final"] - so["error_final"]) <= REL_CHI2*so["error_final"]


def test_lm_wcme_c1_matches_oracle():
    """World-centric motion formulation: one point per (tracklet, frame) chained by LandmarkMotionTernaryFactor;
    the landmark block is block-tridiagonal per tracklet (general landmark-group kernels)."""
    p = synth.make_config("C1", formulation="wcme")
    s = _solver(p); o = _oracle(p)
    lam = 1e-4
    d = s.solve(lam)
    rc, do = o.schur_solve(lam)
    assert rc == 0 and np.linalg.norm(d - do) <= 1e-6*np.linalg.norm(do)
    st = s.optimize(); so = o.optimize()
    assert st["iterations"] == so["iterations"] and st["inner_iterations"] == so["inner_iterations"]
    assert abs(st["error_final"] - so["error_final"]) <= REL_CHI2*so["error_final"]
    pose, point, _ = s.values()
    assert np.abs(pose - o.pose).max() < 1e-6 and np.abs(point - o.point).max() < 1e-5


def test_lm_wcpe_c1_matches_oracle():
    """World-centric POSE formulation end to end (WorldPoseEstimator.cc:89-315): object pose variables L_k, one point
    per (tracklet, frame) chained by the four-key LandmarkMotionPoseFactor (numerical Jacobians, as the reference), and
    the three-pose LandmarkPoseSmoothingFactor.  Numerical differentiation leaves ~1e-6 of rounding in the Jacobians, so
    the trajectories are compared a little looser than the analytic formulations."""
    p = synth.make_config("C1", formulation="wcpe")
    assert any(b.type == MOTIONPOSE3 for b in p.blocks) and any(b.type == SMOOTH_POSE6 for b in p.blocks)
    s = _solver(p); o = _oracle(p)
    assert abs(s.error() - o.error()) <= REL_CHI2*o.error()
    lam = 1e-4
    d = s.solve(lam)
    rc, do = o.schur_solve(lam)
    assert rc == 0 and np.linalg.norm(d - do) <= 1e-5*np.linalg.norm(do)
    # The formulation has a gauge freedom (the reference puts no prior on the object poses: L_k only enters through
    # L_k L_k-1^-1 and the body-frame smoothing), so the reduced system is singular up to lambda*I: as LM drives lambda below
    # ~1e-10 the Cholesky pivots of both implementations sit at rounding level and accept / reject trial steps differently
    # (tools/wcpe_trace.py).  Compared while the damped system is well posed: the first five iterations.
    st = s.optimize(max_iterations=5); so = o.optimize(max_iterations=5)
    assert st["iterations"] == so["iterations"] == 5 and st["inner_iterations"] == so["inner_iterations"]
    assert st["error_final"] < 2e-3*st["error_initial"]
    # Both sides accumulate the reduced system with atomics, so each run differs from the next in the last bits, and along
    # the gauge direction a step amplifies that by ~1/lambda: after five chained steps two runs of the SAME implementation
    # differ by up to ~1e-3 in chi^2, so a comparison of the two trajectories' ends fails at random.  The five iterations
    # are compared one at a time instead, the oracle taking each step from the GPU's iterate at the GPU's lambda.  Measured
    # on a B200, GPU against oracle from equal inputs: <= 1.1e-5 relative while lambda >= 1e-8 (steps 1-4), <= 2.5e-4 for
    # the fifth step (lambda 1e-9); the oracle against itself on 1 and 8 threads: <= 6e-6.
    from dynosam_b200.binding import default_params
    s = _solver(p); o = _oracle(p)
    lam = default_params().lambda_initial
    for it in range(5):
        pose, point, _ = s.values()
        o.pose[:] = pose; o.point[:] = point
        st = s.optimize(max_iterations=1, lambda_initial=lam); so = o.optimize(max_iterations=1, lambda_initial=lam)
        assert st["iterations"] == so["iterations"] == 1 and st["inner_iterations"] == so["inner_iterations"], it
        assert abs(st["error_initial"] - so["error_initial"]) <= REL_CHI2*so["error_initial"], it
        tol = 1e-4 if lam > 5e-9 else 1e-3          # lambda 1e-5 ... 1e-8, then 1e-9
        assert abs(st["error_final"] - so["error_final"]) <= tol*so["error_final"], (it, st["error_final"], so["error_final"])
        lam = st["lambda_final"]


def test_damped_solve_every_factor_type():
    """One damped Schur solve on the graph that holds every factor type (chains of MOTIONPOSE3 / TERNARY3, points
    with factors in several blocks, optical-flow variables) against the dense normal equations of the oracle."""
    p = _all_types_problem()
    s = _solver(p); o = _oracle(p)
    lam = 1e-2
    d = s.solve(lam)
    H, g = o.dense_normal()
    dd = np.linalg.solve(H + lam*np.eye(H.shape[0]), g)
    assert np.linalg.norm(d - dd) <= 1e-6*np.linalg.norm(dd)


def test_flow_projection_star_lm():
    """Row a15: Pose3FlowProjectionFactor star graph (1 pose, N flow variables), as in
    OpticalFlowAndPoseOptimizer::optimize (MotionSolver-inl.hpp:88-260) with max 10 iterations."""
    from dynosam_b200 import lie
    rng = np.random.default_rng(5)
    n = 200
    X_prev = lie.identity()[0]
    X_cur_gt = lie.se3_exp(np.array([[0.01, -0.02, 0.005, 0.05, -0.02, 0.9]]))[0]
    K = np.array([721.5377, 721.5377, 0.0, 609.5593, 172.854, 0.0])
    kp = np.stack([rng.uniform(50, 1190, n), rng.uniform(30, 340, n)], 1); depth = rng.uniform(5, 40, n)
    pc = np.stack([(kp[:, 0] - K[3])/K[0]*depth, (kp[:, 1] - K[4])/K[1]*depth, depth], 1)
    q = lie.transform_to(np.tile(X_cur_gt, (n, 1)), pc)
    proj = np.stack([K[0]*q[:, 0]/q[:, 2] + K[3], K[1]*q[:, 1]/q[:, 2] + K[4]], 1)
    flow_gt = proj - kp
    meas = np.concatenate([kp, depth[:, None], np.tile(X_prev, (n, 1))], 1)
    blocks = [FactorBlock(FLOWPROJ2, np.stack([np.arange(n), np.zeros(n, dtype=int)], 1), meas, np.array([0.5]), 0.0),
              FactorBlock(PRIOR6, np.array([[0]]), lie.identity(), np.full(6, 1.0))]
    p = Problem(lie.identity(), np.zeros((0, 3)), flow=flow_gt + rng.normal(0, 0.5, (n, 2)), calib=K, blocks=blocks)
    s = _solver(p); o = _oracle(p)
    st = s.optimize(max_iterations=10); so = o.optimize(max_iterations=10)
    assert st["iterations"] == so["iterations"]
    assert abs(st["error_final"] - so["error_final"]) <= REL_CHI2*max(so["error_final"], 1e-12) + 1e-12
    pose, _, flow = s.values()
    assert np.abs(pose - o.pose).max() < 1e-6 and np.abs(flow - o.flow).max() < 1e-5


def test_two_directional_factorisation_long_trajectory():
    """A trajectory long enough for the two-directional (twisted) band factorisation: forward and backward halves
    meeting at a middle separator must give the same step and the same LM run as the oracle's plain band Cholesky."""
    p = synth.make_problem(n_frames=400, n_objects=4, n_static=4000, n_dynamic=2000, formulation="hybrid", seed=13,
                           object_span=(120, 200))
    s = _solver(p); o = _oracle(p)
    info = s.info()
    assert info["reduced_dim"] >= 32*(4*((info["bandwidth"] + 31)//32) + 4)      # the twisted path is active
    lam = 1e-4
    d = s.solve(lam)
    rc, do = o.schur_solve(lam)
    assert rc == 0 and np.linalg.norm(d - do) <= 1e-6*np.linalg.norm(do)
    S, g = s.reduced_system(lam)
    So, go, pos = o.reduced_dense(lam)
    perm = np.concatenate([6*pos[i] + np.arange(6) for i in range(p.n_pose)])
    assert np.abs(S - So[np.ix_(perm, perm)]).max() <= 1e-9*np.abs(So).max()
    st = s.optimize(max_iterations=6); so = o.optimize(max_iterations=6)
    assert st["iterations"] == so["iterations"] and st["inner_iterations"] == so["inner_iterations"]
    # six chained LM steps on a 6.4k-dim system whose damped step is only reproducible to ~1e-7 (both sides are 8e-8
    # from the dense solve, tools/twist_check.py): the two trajectories agree to ~2e-6, with or without the twist
    assert abs(st["error_final"] - so["error_final"]) <= 1e-5*so["error_final"]


def test_lm_full_c2_matches_oracle():
    """BASELINE config C2 at full size (2 k key-frames / 500 k static landmarks, 4.2 M factors): chi^2 at the initial
    values and three LM iterations against the oracle."""
    p = synth.make_config("C2")
    assert p.meta["n_frames"] == 2000 and p.n_point == 500_000
    s = _solver(p); o = _oracle(p)
    e, eo = s.error(), o.error()
    assert abs(e - eo) <= REL_CHI2*eo
    st = s.optimize(max_iterations=3); so = o.optimize(max_iterations=3)
    assert st["iterations"] == so["iterations"] and st["inner_iterations"] == so["inner_iterations"]
    assert abs(st["error_final"] - so["error_final"]) <= REL_CHI2*so["error_final"]
    s.close()


def test_cell_partition_matches_plain_band():
    """Nested dissection in time of the reduced solve: P = 2, 4, 8, 16 concurrent chains (1, 2, 4, 8 cells, with spike
    fill-in next to the boundary separators) against the oracle's plain band Cholesky and against the one-chain kernel."""
    p = synth.make_problem(n_frames=1200, n_objects=3, n_static=6000, n_dynamic=1500, formulation="hybrid", seed=5,
                           object_span=(200, 300), max_static_age=6, max_dynamic_age=6)
    o = _oracle(p)
    lam = 1e-4
    rc, do = o.schur_solve(lam)
    assert rc == 0
    steps = {}
    for cells in (-1, 1, 2, 4, 8):
        s = _solver(p); s.set_partition(cells)
        info = s.info()
        wb = (info["bandwidth"] + 31)//32
        assert info["reduced_dim"]//32 >= (4*8 - 1)*max(wb, 2), "graph too short for 8 cells"
        d = s.solve(lam)
        assert np.linalg.norm(d - do) <= 1e-6*np.linalg.norm(do), cells
        steps[cells] = d
        s.close()
    for cells in (1, 2, 4, 8):
        assert np.linalg.norm(steps[cells] - steps[-1]) <= 1e-7*np.linalg.norm(steps[-1]), cells
    so = o.optimize(max_iterations=5)
    for cells in (2, 8):
        s = _solver(p); s.set_partition(cells)
        st = s.optimize(max_iterations=5)
        assert st["iterations"] == so["iterations"] and st["inner_iterations"] == so["inner_iterations"], cells
        assert abs(st["error_final"] - so["error_final"]) <= 1e-5*so["error_final"], cells
        s.close()


def _permuted(p, seed, landmark_runs):
    """The same graph with its factors listed in another order: whole landmark runs shuffled (the order DynOSAM's
    formulations produce up to the order of the landmarks -- the run-based sort of the symbolic phase) or every factor
    shuffled individually (the general stable sort)."""
    import dataclasses
    rng = np.random.default_rng(seed)
    blocks = []
    for b in p.blocks:
        n = b.idx.shape[0]
        if landmark_runs and b.type in (POSE2POINT3, HYBRID3):
            lm = b.idx[:, -1]
            starts = np.flatnonzero(np.r_[True, lm[1:] != lm[:-1]])
            runs = np.split(np.arange(n), starts[1:])
            perm = np.concatenate([runs[i] for i in rng.permutation(len(runs))])
        else:
            perm = rng.permutation(n)
        sig = b.sigma if b.sigma.ndim == 1 else b.sigma[perm]
        blocks.append(FactorBlock(b.type, b.idx[perm], None if b.meas is None else b.meas[perm], sig, b.robust_k,
                                  aux_idx=None if b.aux_idx is None else b.aux_idx[perm]))
    return dataclasses.replace(p, blocks=blocks)


@pytest.mark.parametrize("landmark_runs", [True, False])
def test_factor_order_does_not_matter(landmark_runs):
    """Both sorting paths of the symbolic phase lead to the same damped step and the same LM result."""
    p = synth.make_config("C1")
    q = _permuted(p, 11, landmark_runs)
    lam = 1e-3
    d0 = _solver(p).solve(lam); d1 = _solver(q).solve(lam)
    assert np.linalg.norm(d0 - d1) <= 1e-9*np.linalg.norm(d0)
    s0 = _solver(p).optimize(); s1 = _solver(q).optimize()
    assert s0["iterations"] == s1["iterations"] and s0["inner_iterations"] == s1["inner_iterations"]
    assert abs(s0["error_final"] - s1["error_final"]) <= 1e-9*s0["error_final"]


def test_recycled_device_blocks_are_clean():
    """Solvers created one after the other reuse cached device allocations; results must not depend on what the
    previous owner left behind (a world-centric graph first, then the hybrid one twice)."""
    w = synth.make_config("C1", formulation="wcme")
    _solver(w).optimize()
    p = synth.make_config("C1")
    a = _solver(p); sa = a.optimize(); va = a.values()
    del a
    _solver(w).optimize()
    b = _solver(p); sb = b.optimize(); vb = b.values()
    # (atomic flushes make the sums order-dependent at the last bits, hence tolerances instead of equality)
    assert sa["iterations"] == sb["iterations"] and abs(sa["error_final"] - sb["error_final"]) <= 1e-9*sa["error_final"]
    assert np.abs(va[0] - vb[0]).max() < 1e-8 and np.abs(va[1] - vb[1]).max() < 1e-8


def test_unsupported_topology_reports_status():
    """A tracklet chained over more than 21 frames is outside the general-group kernel: status, not garbage."""
    from dynosam_b200.binding import DynobaError, ERR_UNSUPPORTED
    p = synth.make_problem(n_frames=40, n_objects=1, n_static=50, n_dynamic=20, formulation="wcme", seed=2,
                           max_dynamic_age=35, object_span=(40, 40))
    s = _solver(p)
    assert s.error() > 0         # linearize / chi^2 work for every factor type
    with pytest.raises(DynobaError) as ei:
        s.optimize()
    assert ei.value.status == ERR_UNSUPPORTED


def test_plain_c_program_runs_on_the_gpu(tmp_path):
    """tests/capi/capi_smoke.c through include/dynoba.h: a C consumer of the ABI optimises a small graph on the device."""
    import os, subprocess, sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_host import _build_capi_smoke
    exe = _build_capi_smoke(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
