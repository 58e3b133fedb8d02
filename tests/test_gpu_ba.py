"""HP2 parity on the GPU, through the C ABI, against the CPU oracle."""
import numpy as np
import pytest

import oracle
from particlesfm_b200 import _abi, ba, synthetic as syn

pytestmark = pytest.mark.gpu


def _opts(rot, focal, solver, pp=False):
    o = oracle.ba_global_options(refine_rotation=rot, refine_focal_length=focal)
    o.refine_principal_point = int(pp)
    o.linear_solver = solver
    return o


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


PASSES = [(False, False), (True, True), (True, False)]


@pytest.mark.parametrize("rot,focal", PASSES)
def test_evaluate_matches_oracle(gpu, rot, focal):
    prob, _ = syn.make_ba_problem(12, 900, 6, seed=3, track_len_range=(2, 9))
    o = _opts(rot, focal, _abi.SOLVER_EXACT_SCHUR)
    c0, r0, gc0, gp0 = oracle.ba_evaluate(prob, o)
    S = ba.ResidentSolver(prob)
    c1, r1, gc1, gp1 = S.evaluate(o)
    assert abs(c1 - c0) <= 1e-12 * abs(c0)
    assert _rel(r1, r0) < 1e-12
    assert _rel(gc1, gc0) < 1e-10
    assert _rel(gp1, gp0) < 1e-10


def test_evaluate_principal_point_and_losses(gpu):
    prob, _ = syn.make_ba_problem(8, 400, 5, seed=4)
    for loss in (_abi.LOSS_TRIVIAL, _abi.LOSS_SOFT_L1, _abi.LOSS_CAUCHY):
        o = _opts(True, True, _abi.SOLVER_EXACT_SCHUR, pp=True)
        o.loss_function_type = loss
        c0, r0, gc0, gp0 = oracle.ba_evaluate(prob, o)
        c1, r1, gc1, gp1 = ba.ResidentSolver(prob).evaluate(o)
        assert abs(c1 - c0) <= 1e-12 * abs(c0)
        assert _rel(r1, r0) < 1e-12 and _rel(gc1, gc0) < 1e-10 and _rel(gp1, gp0) < 1e-10


@pytest.mark.parametrize("rot,focal", PASSES)
def test_linear_step_matches_cholesky(gpu, rot, focal):
    prob, _ = syn.make_ba_problem(10, 600, 6, seed=5)
    o = _opts(rot, focal, _abi.SOLVER_EXACT_SCHUR)
    for radius in (1e4, 1e1):
        sc0, sp0, _ = oracle.ba_linear_step(prob, o, radius, _abi.SOLVER_EXACT_SCHUR)
        sc1, sp1, it = ba.ResidentSolver(prob).linear_step(o, radius)
        assert it > 0
        # the same algorithm on both sides: equal to the rounding of two well-conditioned solves
        # (tests/test_schur_step.py checks every reduced-system path against an extended-precision reference)
        assert _rel(sc1, sc0) < 1e-10, (rot, focal, radius, _rel(sc1, sc0))
        assert _rel(sp1, sp0) < 1e-10


def test_iterative_linear_step_matches_oracle_pcg(gpu):
    # same algorithm (ConjugateGradientsSolver + SCHUR_JACOBI, eta = 0.1) on both sides
    prob, _ = syn.make_ba_problem(10, 600, 6, seed=6)
    o = _opts(True, True, _abi.SOLVER_ITERATIVE_SCHUR)
    sc0, sp0, it0 = oracle.ba_linear_step(prob, o, 1e4, _abi.SOLVER_ITERATIVE_SCHUR)
    sc1, sp1, it1 = ba.ResidentSolver(prob).linear_step(o, 1e4)
    assert it1 == it0
    assert _rel(sc1, sc0) < 1e-7 and _rel(sp1, sp0) < 1e-7


@pytest.mark.parametrize("rot,focal", PASSES)
def test_full_solve_exact_mode(gpu, rot, focal):
    """Final poses / points within 1e-5 relative of the oracle (north-star tolerance),
    same iteration counts, gauge parameters bit-identical to the input."""
    prob, truth = syn.make_ba_problem(16, 1500, 7, seed=7)
    o = _opts(rot, focal, _abi.SOLVER_EXACT_SCHUR)
    p0, p1 = prob.copy(), prob.copy()
    s0 = oracle.ba_solve(p0, o)
    s1 = ba.solve_problem(p1, o)
    assert s1.termination == s0.termination
    assert s1.num_iterations == s0.num_iterations
    assert s1.num_successful_steps == s0.num_successful_steps
    assert abs(s1.final_cost - s0.final_cost) <= 1e-5 * s0.final_cost
    assert abs(s1.initial_cost - s0.initial_cost) <= 1e-10 * s0.initial_cost
    for a, b in ((p1.qvec, p0.qvec), (p1.tvec, p0.tvec), (p1.xyz, p0.xyz), (p1.cam_params, p0.cam_params)):
        assert _rel(a, b) < 1e-5
    # gauge: constant pose of image 0 and tvec[0] of image 1
    q0 = prob.qvec[0] / np.linalg.norm(prob.qvec[0])
    assert np.array_equal(p1.qvec[0], q0) and np.array_equal(p1.tvec[0], prob.tvec[0])
    assert p1.tvec[1, 0] == prob.tvec[1, 0]
    if not rot:
        qn = prob.qvec / np.linalg.norm(prob.qvec, axis=1, keepdims=True)
        assert np.array_equal(p1.qvec, qn)
    if not focal:
        assert np.array_equal(p1.cam_params, prob.cam_params)


def test_full_solve_iterative_mode(gpu):
    prob, truth = syn.make_ba_problem(24, 3000, 8, seed=8)
    o = _opts(True, True, _abi.SOLVER_ITERATIVE_SCHUR)
    p0, p1 = prob.copy(), prob.copy()
    s0 = oracle.ba_solve(p0, o)
    s1 = ba.solve_problem(p1, o)
    assert s1.final_cost < 0.2 * s1.initial_cost
    assert abs(s1.final_cost - s0.final_cost) <= 1e-3 * s0.final_cost
    ate = syn.umeyama_ate(syn.camera_centres(p1.qvec, p1.tvec), truth["centres"])
    ate0 = syn.umeyama_ate(syn.camera_centres(p0.qvec, p0.tvec), truth["centres"])
    assert abs(ate - ate0) < 1e-3      # "Sintel ATE within 1e-3 m of reference" stand-in


def test_zero_noise_recovers_truth(gpu):
    prob, truth = syn.make_ba_problem(12, 800, 6, seed=9, noise_px=0.0)
    o = _opts(True, False, _abi.SOLVER_EXACT_SCHUR)
    o.function_tolerance = 1e-14; o.gradient_tolerance = 1e-12; o.parameter_tolerance = 1e-14
    o.max_num_iterations = 60
    s = ba.solve_problem(prob, o)
    assert s.final_cost < 1e-6 * s.initial_cost
    assert syn.umeyama_ate(syn.camera_centres(prob.qvec, prob.tvec), truth["centres"]) < 1e-4


def test_long_tracks_and_unobserved_points(gpu):
    # tracks longer than 256 observations select the 512-wide tiles; points without
    # observations and images without observations are left untouched
    prob, _ = syn.make_ba_problem(300, 40, 300, seed=10)
    prob2, _ = syn.make_ba_problem(300, 400, 9, seed=11)
    obs_image = np.concatenate([prob.obs_image, prob2.obs_image])
    obs_point = np.concatenate([prob.obs_point, prob2.obs_point + 40])
    keep = obs_image != 17                       # image 17 has no observation
    xyz = np.concatenate([prob.xyz, prob2.xyz, np.full((5, 3), 123.0)])
    p = _abi.BAProblem(prob.qvec, prob.tvec, xyz, prob.cam_params, obs_image[keep], obs_point[keep],
                       np.concatenate([prob.obs_xy, prob2.obs_xy])[keep], prob.image_camera,
                       prob.pose_constant, prob.tvec_constant_mask, prob.camera_constant)
    o = _opts(True, True, _abi.SOLVER_ITERATIVE_SCHUR)
    o.max_num_iterations = 6
    p0, p1 = p.copy(), p.copy()
    s0 = oracle.ba_solve(p0, o)
    s1 = ba.solve_problem(p1, o)
    assert np.array_equal(p1.xyz[-5:], xyz[-5:])
    assert np.array_equal(p1.tvec[17], p.tvec[17])
    assert abs(s1.initial_cost - s0.initial_cost) <= 1e-10 * s0.initial_cost
    assert abs(s1.final_cost - s0.final_cost) <= 1e-2 * s0.final_cost


def test_zero_residuals_and_errors(gpu):
    prob, _ = syn.make_ba_problem(4, 10, 3, seed=12)
    empty = _abi.BAProblem(prob.qvec, prob.tvec, prob.xyz, prob.cam_params, np.zeros(0, np.int32),
                           np.zeros(0, np.int32), np.zeros((0, 2)), prob.image_camera)
    import ctypes as C
    from particlesfm_b200 import _lib
    o = _opts(True, True, _abi.SOLVER_AUTO)
    s = _abi.BASummary()
    st = empty.struct()
    assert _lib.lib().psfm_ba_solve(C.byref(st), C.byref(o), C.byref(s)) == _abi.PSFM_ZERO_RESIDUALS
    bad = prob.copy()
    bad.obs_image = bad.obs_image.copy(); bad.obs_image[0] = 99
    st = bad.struct()
    assert _lib.lib().psfm_ba_solve(C.byref(st), C.byref(o), C.byref(s)) == _abi.PSFM_ERR_INVALID


def test_exact_mode_long_tracks_dense_reduced_system(gpu):
    """Tracks spanning (almost) the whole sequence make the reduced camera system dense
    (Sintel-like: ~50 frames, tracks of 3..50 frames): the band-aware Cholesky must take the
    dense route and still match the oracle's dense Cholesky path."""
    prob, truth = syn.make_ba_problem(50, 3000, 12, seed=14, track_len_range=(3, 50))
    o = _opts(True, True, _abi.SOLVER_AUTO)          # <= 1000 images -> exact Schur
    p0, p1 = prob.copy(), prob.copy()
    s0 = oracle.ba_solve(p0, o)
    s1 = ba.solve_problem(p1, o)
    assert s1.linear_solver_used == _abi.SOLVER_EXACT_SCHUR and s1.num_explicit_solves == s1.num_iterations
    assert s1.num_iterations == s0.num_iterations and s1.termination == s0.termination
    assert abs(s1.final_cost - s0.final_cost) <= 1e-8 * s0.final_cost
    for a, b in ((p1.qvec, p0.qvec), (p1.tvec, p0.tvec), (p1.xyz, p0.xyz), (p1.cam_params, p0.cam_params)):
        assert _rel(a, b) < 1e-7


def test_exact_mode_duplicate_observations_and_dynamic_dropouts(gpu):
    """A point observed twice in the same image (both orders enter the diagonal block) and
    tracks with holes (30 % of the observations dropped, as after motion segmentation)."""
    prob, _ = syn.make_ba_problem(30, 2500, 10, seed=15, dynamic_fraction=0.3)
    rng = np.random.default_rng(0)
    dup = rng.choice(prob.num_observations, 200, replace=False)
    xy = np.concatenate([prob.obs_xy, prob.obs_xy[dup] + rng.normal(0, 0.3, (200, 2))])
    p = _abi.BAProblem(prob.qvec, prob.tvec, prob.xyz, prob.cam_params, np.concatenate([prob.obs_image, prob.obs_image[dup]]),
                       np.concatenate([prob.obs_point, prob.obs_point[dup]]), xy, prob.image_camera,
                       prob.pose_constant, prob.tvec_constant_mask, prob.camera_constant)
    for rot, focal in ((True, True), (False, False)):
        o = _opts(rot, focal, _abi.SOLVER_EXACT_SCHUR)
        p0, p1 = p.copy(), p.copy()
        s0 = oracle.ba_solve(p0, o)
        s1 = ba.solve_problem(p1, o)
        assert s1.num_iterations == s0.num_iterations
        assert abs(s1.final_cost - s0.final_cost) <= 1e-8 * s0.final_cost
        assert _rel(p1.xyz, p0.xyz) < 1e-6 and _rel(p1.tvec, p0.tvec) < 1e-6


def test_exact_mode_principal_point_falls_back_to_tight_pcg(gpu):
    prob, _ = syn.make_ba_problem(10, 600, 6, seed=16)
    o = _opts(True, True, _abi.SOLVER_EXACT_SCHUR, pp=True)
    p0, p1 = prob.copy(), prob.copy()
    s0 = oracle.ba_solve(p0, o)
    s1 = ba.solve_problem(p1, o)
    assert s1.num_explicit_solves == 0 and s1.num_schur_products > 0
    assert s1.num_iterations == s0.num_iterations
    assert abs(s1.final_cost - s0.final_cost) <= 1e-6 * s0.final_cost


def _mixed_track_problem(frames, long_len, seed):
    """A few tracks of `long_len` observations (select the 512-wide tiles) plus short ones."""
    a, _ = syn.make_ba_problem(frames, 24, long_len, seed=seed)
    b, _ = syn.make_ba_problem(frames, 600, 8, seed=seed + 1)
    return _abi.BAProblem(a.qvec, a.tvec, np.concatenate([a.xyz, b.xyz]), a.cam_params,
                          np.concatenate([a.obs_image, b.obs_image]),
                          np.concatenate([a.obs_point, b.obs_point + a.num_points]),
                          np.concatenate([a.obs_xy, b.obs_xy]), a.image_camera,
                          a.pose_constant, a.tvec_constant_mask, a.camera_constant)


@pytest.mark.parametrize("frames,long_len,fused", [(320, 300, 1), (520, 500, 1)])
def test_exact_mode_wide_tiles(gpu, frames, long_len, fused):
    """Tracks of 300 / 500 observations run the fused Schur kernel on 512-wide tiles (per-image
    staging for up to 520 images next to the per-observation records in shared memory); the
    unfused k_schur_w + k_schur_pairs path is covered by test_code_paths_agree.  Both sizes
    must reproduce the oracle's exact step."""
    p = _mixed_track_problem(frames, long_len, seed=30)
    o = _opts(True, True, _abi.SOLVER_EXACT_SCHUR)
    o.max_num_iterations = 3
    p0, p1 = p.copy(), p.copy()
    s0 = oracle.ba_solve(p0, o)
    s1 = ba.solve_problem(p1, o)
    assert s1.explicit_fused == fused and s1.num_pair_entries > 0
    assert s1.num_iterations == s0.num_iterations
    assert abs(s1.initial_cost - s0.initial_cost) <= 1e-10 * s0.initial_cost
    assert abs(s1.final_cost - s0.final_cost) <= 1e-8 * s0.final_cost
    assert _rel(p1.tvec, p0.tvec) < 1e-7 and _rel(p1.xyz, p0.xyz) < 1e-7


def test_code_paths_agree(gpu, monkeypatch):
    """The persistent cp.async-pipelined kernels, the one-CTA-per-tile kernels, the fused and
    the unfused Schur paths and both Cholesky dispatches are the same arithmetic in a different
    schedule: identical LM trajectories, parameters equal to ~1e-12."""
    prob, _ = syn.make_ba_problem(40, 6000, 9, seed=31, dynamic_fraction=0.1)
    o = _opts(True, True, _abi.SOLVER_EXACT_SCHUR)
    ref = prob.copy()
    s_ref = ba.solve_problem(ref, o)
    assert s_ref.explicit_fused == 1
    for env in ("PSFM_NO_PIPE", "PSFM_SCHUR_UNFUSED", "PSFM_NO_PIPE_SCHUR"):
        monkeypatch.setenv(env, "1")
        p = prob.copy()
        s = ba.solve_problem(p, o)
        monkeypatch.delenv(env)
        assert s.num_iterations == s_ref.num_iterations and s.termination == s_ref.termination, env
        assert abs(s.final_cost - s_ref.final_cost) <= 1e-11 * s_ref.final_cost, env
        assert _rel(p.xyz, ref.xyz) < 1e-9 and _rel(p.qvec, ref.qvec) < 1e-9, env
        if env == "PSFM_SCHUR_UNFUSED":
            assert s.explicit_fused == 0


def test_tracks_longer_than_a_tile_are_rejected(gpu):
    p = _mixed_track_problem(620, 600, seed=32)
    with pytest.raises(Exception, match="512 observations"):
        ba.solve_problem(p, _opts(True, True, _abi.SOLVER_AUTO))


def test_run_to_run_drift_is_bounded(gpu):
    """HP2 is NOT bit-reproducible run to run: per-image sums and band blocks are accumulated with
    fp64 atomics (RED) whose order depends on the tile schedule (DESIGN.md §3.2).  This bounds the
    drift: same iteration counts, costs to 1e-12, parameters to 1e-9 relative over repeated solves —
    four orders of magnitude inside the 1e-5 parity tolerance."""
    prob, _ = syn.make_ba_problem(30, 20000, 8, seed=13)
    o = _opts(True, True, _abi.SOLVER_EXACT_SCHUR)
    runs = []
    for _ in range(4):
        p = prob.copy()
        s = ba.solve_problem(p, o)
        runs.append((s, p))
    s0, p0 = runs[0]
    for s, p in runs[1:]:
        assert s.num_iterations == s0.num_iterations and s.termination == s0.termination
        assert abs(s.final_cost - s0.final_cost) <= 1e-12 * s0.final_cost
        for a, b in ((p.qvec, p0.qvec), (p.tvec, p0.tvec), (p.xyz, p0.xyz), (p.cam_params, p0.cam_params)):
            assert _rel(a, b) < 1e-9
