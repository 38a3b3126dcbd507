"""GPU parity tier for the bundle-adjustment path: b200ba_solve (CUDA, fp64) against the CPU oracle on the same
inputs.  Bar (BASELINE.json north_star): final cost / residual and parameters within 1e-5 relative; residual
counts exact; constant blocks bit-identical."""
import os

import numpy as np
import pytest

import oracle_ba
from colmap_b200.bundle_adjustment import (CAUCHY, DENSE_SCHUR, HUBER, ITERATIVE_SCHUR, PINHOLE, RADIAL, RADIAL_FISHEYE,
                                           SIMPLE_PINHOLE, SIMPLE_RADIAL_FISHEYE,
                                           SIMPLE_RADIAL, SOFT_L1, TWO_CAMS_FROM_WORLD, BundleAdjustmentConfig,
                                           BundleAdjustmentOptions, CreateDefaultBundleAdjuster, solve_flat)
from colmap_b200.synthetic import flat_to_reconstruction, synthesize_ba_problem

pytestmark = pytest.mark.gpu
REL = 1e-5


def _gauge(flat):
    flat.pose_constant = flat.pose_constant.copy(); flat.pose_fixed_dim = flat.pose_fixed_dim.copy()
    flat.pose_constant[0] = 1
    base = flat.poses[1, 4:] - flat.poses[0, 4:]
    flat.pose_fixed_dim[1] = int(np.argmax(np.abs(base)))
    return flat


def _both(options, noisy):
    a, b = noisy.copy(), noisy.copy()
    for f in (a, b):
        f.pose_constant, f.pose_fixed_dim, f.point_constant, f.cam_constant = (noisy.pose_constant, noisy.pose_fixed_dim,
                                                                                noisy.point_constant, noisy.cam_constant)
    s_gpu = solve_flat(options, a)
    s_ref = oracle_ba.solve(options, b)
    return a, s_gpu, b, s_ref


def _assert_parity(a, s_gpu, b, s_ref, param_rel=REL):
    assert s_gpu.num_residuals == s_ref.num_residuals
    assert s_gpu.num_effective_parameters == s_ref.num_effective_parameters
    # COLMAP runs Ceres with function_tolerance = 0: the last LM steps sit at the rounding noise of the cost, so
    # CONVERGENCE (gradient tolerance) vs NO_CONVERGENCE (100 iterations) can legitimately differ between two
    # correct implementations; both must be usable and agree on the solution.
    assert s_gpu.termination_type in (0, 1) and s_ref.termination_type in (0, 1)
    assert abs(s_gpu.initial_cost - s_ref.initial_cost) <= 1e-9 * s_ref.initial_cost
    assert abs(s_gpu.final_cost - s_ref.final_cost) <= REL * s_ref.final_cost
    for u, v in ((a.poses, b.poses), (a.cam_params, b.cam_params), (a.points, b.points)):
        assert np.allclose(u, v, rtol=param_rel, atol=param_rel * max(1.0, np.abs(v).max()))


def test_b1_config_dense_schur():
    """BASELINE config B1: 10 pinhole cameras (one shared PINHOLE), 1k points, 5k observations."""
    gt, noisy = synthesize_ba_problem(10, 1000, 5, models=(PINHOLE,), shared_camera=True, seed=42)
    _gauge(noisy)
    a, sg, b, sr = _both(BundleAdjustmentOptions(), noisy)
    assert sg.linear_solver_type_used == DENSE_SCHUR and sg.num_residuals == 10000
    _assert_parity(a, sg, b, sr)


@pytest.mark.parametrize("models,shared,lst", [
    ((SIMPLE_RADIAL,), False, ITERATIVE_SCHUR),
    ((PINHOLE, SIMPLE_RADIAL), False, ITERATIVE_SCHUR),          # mixed models (config B5 style)
    ((SIMPLE_PINHOLE, RADIAL, PINHOLE, SIMPLE_RADIAL), False, DENSE_SCHUR),
    ((RADIAL,), True, ITERATIVE_SCHUR),                          # shared intrinsics block: exact SCHUR_JACOBI cross terms
    ((SIMPLE_RADIAL_FISHEYE, RADIAL_FISHEYE, SIMPLE_RADIAL), False, ITERATIVE_SCHUR),   # equidistant-fisheye models
    ((RADIAL_FISHEYE,), True, DENSE_SCHUR),
])
def test_model_grid_parity(models, shared, lst):
    gt, noisy = synthesize_ba_problem(24, 1500, 6, models=models, shared_camera=shared, seed=7)
    _gauge(noisy)
    a, sg, b, sr = _both(BundleAdjustmentOptions(linear_solver_type=lst), noisy)
    _assert_parity(a, sg, b, sr)


@pytest.mark.parametrize("kw", [
    dict(refine_principal_point=True),
    dict(refine_focal_length=False),
    dict(refine_extra_params=False, refine_focal_length=False),   # constant cameras
    dict(constant_rig_from_world_rotation=True),
    dict(refine_points3D=False),
    dict(loss_function_type=SOFT_L1), dict(loss_function_type=CAUCHY, loss_function_scale=2.0),
    dict(loss_function_type=HUBER, loss_function_scale=1.5),
])
def test_option_grid_parity(kw):
    gt, noisy = synthesize_ba_problem(12, 400, 6, models=(SIMPLE_RADIAL,), seed=11)
    _gauge(noisy)
    a, sg, b, sr = _both(BundleAdjustmentOptions(**kw), noisy)
    # refining the principal point of 12 single-image cameras leaves a nearly flat valley (principal point vs
    # rotation): the cost is pinned to 1e-5 but the position along the valley is only determined to ~1e-3
    _assert_parity(a, sg, b, sr, param_rel=1e-3 if kw.get("refine_principal_point") else REL)


def test_constant_blocks_bit_identical_and_residual_counts():
    gt, noisy = synthesize_ba_problem(8, 200, 5, models=(PINHOLE,), shared_camera=True, seed=3)
    _gauge(noisy)
    noisy.point_constant = noisy.point_constant.copy(); noisy.point_constant[:25] = 1
    noisy.pose_constant[5] = 1
    before = noisy.copy()
    a, sg, b, sr = _both(BundleAdjustmentOptions(), noisy)
    _assert_parity(a, sg, b, sr)
    assert np.array_equal(a.points[:25], before.points[:25])
    assert np.array_equal(a.poses[0], before.poses[0]) and np.array_equal(a.poses[5], before.poses[5])
    assert a.cam_params[2] == before.cam_params[2] and a.cam_params[3] == before.cam_params[3]
    # the gauge-fixed translation coordinate of frame 2 does not move
    d = int(noisy.pose_fixed_dim[1])
    assert a.poses[1, 4 + d] == before.poses[1, 4 + d]
    # only points variable: residuals of constant points vanish from the count
    o = BundleAdjustmentOptions(refine_rig_from_world=False, refine_focal_length=False, refine_extra_params=False)
    a2, sg2, b2, sr2 = _both(o, noisy)
    assert sg2.num_residuals == sr2.num_residuals == 2 * 175 * 5


def test_reconstruction_level_api_mirrors_reference_tests():
    """bundle_adjustment_test.cc:303-411 through the BundleAdjuster mirror: Nominal (everything variable, two-cams
    gauge), ConstantPoints3D (explicitly constant points keep their coordinates bit-identically and only add
    residuals), images outside the config become constant-pose observations."""
    gt, noisy = synthesize_ba_problem(10, 200, 10, models=(SIMPLE_RADIAL,), shared_camera=True, seed=1,
                                      point2D_stddev=0.5, point3D_stddev=0.1, translation_stddev=0.1, rotation_stddev_deg=0.5)
    rec = flat_to_reconstruction(noisy)
    cfg = BundleAdjustmentConfig()
    for i in rec.images:
        cfg.AddImage(i)
    cfg.FixGauge(TWO_CAMS_FROM_WORLD)
    summary = CreateDefaultBundleAdjuster(BundleAdjustmentOptions(), cfg, rec).Solve()
    assert summary.termination_type == 0 and summary.num_residuals == 2 * 2000
    rmse = np.sqrt(2 * summary.final_cost / 2000)
    assert rmse < 0.5 * np.sqrt(2) * 1.05
    # first image untouched (gauge)
    assert np.array_equal(rec.images[1].cam_from_world, noisy.poses[0] / np.r_[np.ones(4) * np.linalg.norm(noisy.poses[0, :4]), 1, 1, 1]) or \
        np.allclose(rec.images[1].cam_from_world, noisy.poses[0], atol=0)

    # ConstantPoints3D: two images in the config, points 1 and 2 constant, everything else from those images variable
    rec2 = flat_to_reconstruction(noisy)
    cfg2 = BundleAdjustmentConfig()
    cfg2.AddImage(1); cfg2.AddImage(2)
    cfg2.AddConstantPoint(1); cfg2.AddConstantPoint(2)
    xyz1, xyz2 = rec2.points3D[1].xyz.copy(), rec2.points3D[2].xyz.copy()
    s2 = CreateDefaultBundleAdjuster(BundleAdjustmentOptions(), cfg2, rec2).Solve()
    assert np.array_equal(rec2.points3D[1].xyz, xyz1) and np.array_equal(rec2.points3D[2].xyz, xyz2)
    n_in = sum(1 for im in (rec2.images[1], rec2.images[2]) for _ in im.points2D)
    n_extra = sum(1 for pid in (1, 2) for (iid, _) in rec2.points3D[pid].track if iid not in (1, 2))
    assert s2.num_residuals == 2 * (n_in + n_extra)
    # images outside the config keep their poses
    assert np.array_equal(rec2.images[5].cam_from_world, noisy.poses[4])


def test_medium_iterative_problem_converges_like_the_oracle():
    gt, noisy = synthesize_ba_problem(60, 12000, 6, models=(SIMPLE_RADIAL,), seed=21)
    _gauge(noisy)
    a, sg, b, sr = _both(BundleAdjustmentOptions(linear_solver_type=ITERATIVE_SCHUR), noisy)
    # both runs stop at 100 inexact-Newton iterations (gradient tolerance 1e-4 on the unscaled gradient is not reached):
    # the cost agrees to 1e-5 (actually ~1e-10) while the weakest directions are only pinned to ~1e-4
    _assert_parity(a, sg, b, sr, param_rel=1e-4)
    assert sg.num_linear_solver_iterations > 0 and sg.spmv_launches > 0 and sg.kernel_launches > 0


def test_long_tracks_use_the_generic_path():
    """Tracks of every size class in one problem: <= 32 observations (warp-packed), 33..256 (block-packed) and > 256
    (generic two-kernel path with global atomics) must all reproduce the oracle."""
    lens = np.concatenate([np.full(600, 6), np.full(30, 40), np.full(12, 200), np.full(6, 300), np.full(3, 330)])
    gt, noisy = synthesize_ba_problem(340, len(lens), 0, models=(SIMPLE_RADIAL,), shared_camera=True, seed=17,
                                      track_lengths=lens)
    _gauge(noisy)
    a, sg, b, sr = _both(BundleAdjustmentOptions(linear_solver_type=ITERATIVE_SCHUR, max_num_iterations=15), noisy)
    assert sg.num_residuals == 2 * int(lens.sum())
    _assert_parity(a, sg, b, sr, param_rel=1e-4)


def test_golden_fixture_solution():
    """tests/golden/ba_case_small.npz (problem + the oracle's frozen solution): the GPU solver lands on the stored
    solution within the 1e-5 relative tolerance, without the oracle being run."""
    from test_golden_cpu import ba_case
    z, o, flat = ba_case()
    s = solve_flat(o, flat)
    assert s.num_residuals == int(z["num_residuals"]) and s.num_effective_parameters == int(z["num_effective_parameters"])
    assert abs(s.initial_cost - float(z["initial_cost"])) <= 1e-9 * float(z["initial_cost"])
    assert abs(s.final_cost - float(z["final_cost"])) <= 1e-5 * float(z["final_cost"])
    assert np.allclose(flat.poses, z["sol_poses"], rtol=1e-5, atol=1e-5)
    assert np.allclose(flat.points, z["sol_points"], rtol=1e-5, atol=1e-5)
    assert np.allclose(flat.cam_params, z["sol_cam_params"], rtol=1e-5, atol=1e-5)


# ---------------------------------------------------------------- BASELINE sizes
def test_b3_full_size_parity_vs_oracle():
    """BASELINE config B3 at FULL size (500 SIMPLE_RADIAL cameras with their own intrinsics, 300k points, 2M
    observations, ITERATIVE_SCHUR + SCHUR_JACOBI): the first 12 LM iterations of both implementations - cost 1e-5,
    parameters 1e-4 (inexact Newton steps: the PCG forcing term leaves the weakest directions pinned to ~1e-4)."""
    gt, noisy = synthesize_ba_problem(500, 300000, 7, models=(SIMPLE_RADIAL,), seed=42, num_obs=2000000)
    _gauge(noisy)
    a, sg, b, sr = _both(BundleAdjustmentOptions(linear_solver_type=ITERATIVE_SCHUR, max_num_iterations=12), noisy)
    assert sg.num_residuals == 4000000
    assert sg.num_successful_steps + sg.num_unsuccessful_steps == sr.num_successful_steps + sr.num_unsuccessful_steps
    _assert_parity(a, sg, b, sr, param_rel=1e-4)


def test_b5_shaped_mixed_models_parity_vs_oracle():
    """B5-shaped (mixed camera models, > 1M observations): 400 cameras cycling over four models, 180k points, 1.1M
    observations, ITERATIVE_SCHUR; 8 LM iterations against the oracle."""
    gt, noisy = synthesize_ba_problem(400, 180000, 6, models=(PINHOLE, SIMPLE_RADIAL, RADIAL, SIMPLE_RADIAL_FISHEYE),
                                      seed=5, num_obs=1100000)
    _gauge(noisy)
    a, sg, b, sr = _both(BundleAdjustmentOptions(linear_solver_type=ITERATIVE_SCHUR, max_num_iterations=8), noisy)
    assert sg.num_residuals == 2200000
    _assert_parity(a, sg, b, sr, param_rel=1e-4)


def test_assemble_then_solve_on_the_gpu():
    """SURVEY 8(a) DefaultBundleAdjuster ctor + 8(f-3): the C++ assembly (b200ba_assemble: observations, constancy rules,
    two-cams gauge, config.NumImages() for the solver choice) feeding b200ba_solve on the GPU, against the oracle run on
    the Python mirror's flattening of the same reconstruction: a LOCAL bundle adjustment (6 of 40 images in the config,
    constant-pose observations from outside images through explicit variable points)."""
    from colmap_b200.bundle_adjustment import assemble_reconstruction, flatten_reconstruction, BundleAdjuster
    gt, noisy = synthesize_ba_problem(40, 1500, 8, models=(SIMPLE_RADIAL,), seed=2)
    rec = flat_to_reconstruction(noisy)
    cfg = BundleAdjustmentConfig()
    for i in (3, 4, 5, 9, 10, 11):
        cfg.AddImage(i)
    for pid in list(rec.points3D)[:200]:
        cfg.AddVariablePoint(pid)
    cfg.FixGauge(TWO_CAMS_FROM_WORLD)
    o = BundleAdjustmentOptions()
    flat_c, image_ids, camera_ids, point_ids = assemble_reconstruction(o, cfg, rec)
    assert flat_c.num_config_images == 6
    sg = solve_flat(o, flat_c)
    assert sg.linear_solver_type_used == DENSE_SCHUR          # 6 config images, although the model has 40 (ADVICE r1)
    # oracle on the Python mirror's flattening + the same gauge the adapter applies
    rec2 = flat_to_reconstruction(noisy)
    adj = BundleAdjuster(o, cfg, rec2)
    flat_p, *_ = flatten_reconstruction(o, cfg, rec2)
    flat_p.pose_constant, flat_p.pose_fixed_dim = flat_c.pose_constant.copy(), flat_c.pose_fixed_dim.copy()
    sr = oracle_ba.solve(o, flat_p)
    assert sg.num_residuals == sr.num_residuals and sg.num_effective_parameters == sr.num_effective_parameters
    assert abs(sg.final_cost - sr.final_cost) <= REL * sr.final_cost
    assert np.allclose(flat_c.poses, flat_p.poses, rtol=REL, atol=REL) and np.allclose(flat_c.points, flat_p.points, rtol=REL, atol=REL)
    outside = [k for k, i in enumerate(image_ids) if i not in cfg.Images()]
    assert np.array_equal(flat_c.poses[outside], noisy.poses[outside])       # constant blocks bit-identical


def test_cross_backend_with_the_reference_caspar_solver():
    """The reference's own GPU backend (generated Caspar solver, fp32) on the same problem, as stored in
    tests/golden/ba_reference_caspar.npz (tests/golden/make_golden.py --reference) - the cross-backend check of
    bundle_adjustment_caspar_test.cc:957-1022 (MergedCalibMatchesCeres: one shared SIMPLE_RADIAL camera, principal point
    refined; focal within 20, principal point within 10, extra within 1.5e-2 in fp32) with our solver in the role of
    Ceres, plus the final cost.  Caspar fixes one frame only (scale left free), so costs and intrinsics are compared,
    poses are not."""
    import make_golden
    a, o = make_golden.caspar_case()
    sg = solve_flat(o, a)
    rc = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ba_reference_caspar.npz"))
    msg = f"ours {sg.final_cost} ({a.cam_params}) caspar {float(rc['final_cost'])} ({rc['cam_params']})"
    assert int(rc["num_residuals"]) == sg.num_residuals, msg
    assert abs(float(rc["final_cost"]) - sg.final_cost) <= 2e-2 * sg.final_cost, msg
    pa, pb = a.cam_params.reshape(-1, 4), rc["cam_params"].reshape(-1, 4)
    assert np.abs(pa[:, 0] - pb[:, 0]).max() < 20.0 and np.abs(pa[:, 1:3] - pb[:, 1:3]).max() < 10.0, msg
    assert np.abs(pa[:, 3] - pb[:, 3]).max() < 1.5e-2, msg


# ---------------------------------------------------------------- the twelve wide camera models + rigs on the solve path
from colmap_b200.bundle_adjustment import (DIVISION, EQUIRECTANGULAR, EUCM, FISHEYE, FOV, FULL_OPENCV, OPENCV, OPENCV_FISHEYE,
                                           RAD_TAN_THIN_PRISM_FISHEYE, SIMPLE_DIVISION, SIMPLE_FISHEYE, THIN_PRISM_FISHEYE)


@pytest.mark.parametrize("models,shared,kw", [
    ((OPENCV,), False, {}),
    ((OPENCV,), True, dict(refine_principal_point=True)),                       # 8-wide intrinsics block, shared: cross terms
    ((OPENCV_FISHEYE, FISHEYE, SIMPLE_RADIAL), False, {}),                      # wide + narrow mixed
    ((FULL_OPENCV,), True, dict(refine_principal_point=True)),                  # 12-wide block: two 6-ranges + their pair
    ((RAD_TAN_THIN_PRISM_FISHEYE,), True, dict(refine_principal_point=True)),   # 16-wide block
    ((FOV, EUCM, DIVISION, SIMPLE_DIVISION), False, {}),
    ((SIMPLE_FISHEYE, THIN_PRISM_FISHEYE), True, dict(linear_solver_type=ITERATIVE_SCHUR)),
    ((EQUIRECTANGULAR, PINHOLE), False, {}),                                    # metadata parameters are never refined
    ((OPENCV_FISHEYE, FULL_OPENCV), False, dict(linear_solver_type=ITERATIVE_SCHUR)),   # own wide cameras, PCG: SCHUR_JACOBI blocks
                                                                                        # of 6 and 10 columns from the 6-range pairs
])
def test_wide_model_grid_parity(models, shared, kw):
    """models_jacobian.h:322-1565 on the solve path: every model beyond the <= 5-parameter family through the wide kernel
    instantiations, against the oracle (whose wide Jacobians come from the complex-step method).  High-order distortion
    models converge slowly along nearly flat directions (k5, k6, s-terms): when a run stops at the iteration limit instead
    of the gradient tolerance the two trajectories (fp32-stored vs fp64 Jacobians) are compared at 1e-4 in the cost."""
    n_img = 12 if shared else 16
    gt, noisy = synthesize_ba_problem(n_img, 1200, 8, models=models, shared_camera=shared, seed=19, point2D_stddev=0.3,
                                      point3D_stddev=0.02, rotation_stddev_deg=0.3)
    _gauge(noisy)
    # (1) the arithmetic: three LM iterations from the same start must agree tightly (same gradient, damping, reduced system)
    a, sg, b, sr = _both(BundleAdjustmentOptions(max_num_iterations=3, **kw), noisy)
    assert sg.num_residuals == sr.num_residuals and sg.num_effective_parameters == sr.num_effective_parameters
    assert abs(sg.initial_cost - sr.initial_cost) <= 1e-9 * sr.initial_cost
    assert abs(sg.final_cost - sr.final_cost) <= 1e-6 * sr.final_cost
    for u, v in ((a.poses, b.poses), (a.points, b.points), (a.cam_params, b.cam_params)):
        assert np.allclose(u, v, rtol=1e-5, atol=1e-5 * max(1.0, np.abs(v).max()))
    # (2) the full run: back at the noise floor; the cost agrees to 1e-5 where both runs reach the gradient tolerance and
    # to 1e-3 where they stop at the iteration limit inside the flat valley of a high-order model
    a, sg, b, sr = _both(BundleAdjustmentOptions(**kw), noisy)
    converged = sg.termination_type == 0 and sr.termination_type == 0
    msg = (f"ours {sg.final_cost!r} (type {sg.termination_type}, {sg.num_successful_steps}+{sg.num_unsuccessful_steps} steps) "
           f"oracle {sr.final_cost!r} (type {sr.termination_type}, {sr.num_successful_steps}+{sr.num_unsuccessful_steps} steps)")
    assert abs(sg.final_cost - sr.final_cost) <= (REL if converged else 1e-3) * sr.final_cost, msg
    rmse = np.sqrt(2 * sg.final_cost / (sg.num_residuals / 2))
    assert rmse < 0.3 * np.sqrt(2) * 1.1
    if converged and not kw.get("refine_principal_point"):
        for u, v in ((a.poses, b.poses), (a.points, b.points)):
            assert np.allclose(u, v, rtol=1e-4, atol=1e-4 * max(1.0, np.abs(v).max()))


@pytest.mark.parametrize("kw,sensor_const,models", [
    ({}, None, (SIMPLE_RADIAL,)),                                               # everything variable
    (dict(refine_sensor_from_rig=False), None, (SIMPLE_RADIAL, PINHOLE)),       # RigReprojErrorConstantRigCostFunctor
    ({}, [1, 0], (OPENCV, SIMPLE_RADIAL, FISHEYE)),                             # one sensor constant, wide models in the rig
    (dict(refine_rig_from_world=False), None, (SIMPLE_RADIAL,)),                # frames fixed, sensors + intrinsics + points move
    (dict(linear_solver_type=ITERATIVE_SCHUR, refine_principal_point=True), None, (PINHOLE, SIMPLE_RADIAL, RADIAL)),
])
def test_rig_parity(kw, sensor_const, models):
    """Non-trivial frames (reprojection_error.h:344-420, bundle_adjustment_ceres.cc:753-827): cam_from_world =
    sensor_from_rig * rig_from_world, the sensor_from_rig poses as camera-side blocks of their own."""
    from colmap_b200.synthetic import synthesize_rig_problem
    gt, noisy = synthesize_rig_problem(10, 3, 800, 8, models=models, seed=23, point2D_stddev=0.5)
    _gauge(noisy)
    if sensor_const is not None:
        noisy.sensor_constant = np.array(sensor_const, np.uint8)
    before = noisy.copy()
    a, sg, b, sr = _both(BundleAdjustmentOptions(**kw), noisy)
    _assert_parity(a, sg, b, sr, param_rel=1e-4)
    assert np.allclose(a.sensors, b.sensors, rtol=1e-4, atol=1e-4)
    if kw.get("refine_sensor_from_rig") is False:
        assert np.array_equal(a.sensors, before.sensors)                        # constant blocks bit-identical
    if sensor_const is not None:
        assert np.array_equal(a.sensors[0], before.sensors[0]) and not np.array_equal(a.sensors[1], before.sensors[1])
    if kw.get("refine_rig_from_world") is False:
        assert np.array_equal(a.poses, before.poses)


def test_reconstruction_level_api_with_rigs_recovers_ground_truth():
    """NominalMultiCameraRig (bundle_adjustment_ceres_test.cc:183-220) through the BundleAdjuster mirror on the GPU: 2 rigs x
    3 cameras x 5 frames, 200 points, noisy points and rig poses, two-cams gauge; every frame, sensor_from_rig, camera and
    point variable.  The solve returns to the noise floor, recovers the sensor_from_rig poses and the relative geometry
    (the reference asks 0.1 deg / 0.1 units after alignment), and agrees with the oracle on the same flat problem."""
    import copy
    from test_ba_cpu import _noisy_rig_reconstruction
    from colmap_b200.bundle_adjustment import flatten_reconstruction
    gt, rec = _noisy_rig_reconstruction()
    cfg = BundleAdjustmentConfig()
    for i in rec.images:
        cfg.AddImage(i)
    cfg.FixGauge(TWO_CAMS_FROM_WORLD)
    o = BundleAdjustmentOptions()
    rec_o = copy.deepcopy(rec)
    summary = CreateDefaultBundleAdjuster(o, cfg, rec).Solve()
    n_obs = 200 * len(rec.images)
    assert summary.termination_type in (0, 1) and summary.num_residuals == 2 * n_obs
    # 200 x 3 points + 10 x 6 frames - 7 (gauge) + 4 x 6 sensors + 6 x 2 intrinsics
    assert summary.num_effective_parameters == 600 + 60 - 7 + 24 + 12
    rmse = np.sqrt(2 * summary.final_cost / n_obs)
    assert rmse < 0.5 * np.sqrt(2) * 1.05
    for r in rec.rigs:
        for c, sfr in rec.rigs[r].sensors.items():
            g = gt.rigs[r].sensors[c]
            assert abs(np.dot(sfr[:4], g[:4])) > np.cos(np.deg2rad(0.1) / 2), (r, c)
            assert np.abs(sfr[4:] - g[4:]).max() < 0.02, (r, c, sfr[4:] - g[4:])
    P = np.stack([rec.points3D[k].xyz for k in sorted(rec.points3D)][:60]); G = np.stack([gt.points3D[k].xyz for k in sorted(gt.points3D)][:60])
    dp = np.linalg.norm(P[:, None] - P[None], axis=-1); dg = np.linalg.norm(G[:, None] - G[None], axis=-1)
    assert np.abs(dp / (dp.sum() / dg.sum()) - dg).max() < 0.1
    # the oracle on the same problem
    flat = flatten_reconstruction(o, cfg, rec_o)[0]
    so = oracle_ba.solve(o, flat)
    assert so.num_effective_parameters == summary.num_effective_parameters
    assert abs(so.final_cost - summary.final_cost) <= REL * so.final_cost
    assert np.allclose(np.stack([rec.frames[f].rig_from_world for f in sorted(rec.frames)]), flat.poses, rtol=REL, atol=REL)
