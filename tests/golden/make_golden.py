"""Generator of the committed golden fixtures in tests/golden/ (test infrastructure).

  python tests/golden/make_golden.py              # oracle fixtures (CPU, anywhere)
  python tests/golden/make_golden.py --reference  # + the fixtures produced by the UNMODIFIED reference GPU code
                                                  #   (oracle/_ref/libpm_ref.so, oracle/_ref/libcaspar_ref.so; needs a GPU)
  --out DIR                                       # write the fixtures to DIR instead of tests/golden/

Fixtures
  reference_known_answers.json   vectors transcribed from the reference's own tests (file:line in every entry); this
                                 file is hand-written, the script only validates that it parses.
  pm_case_96x64.npz              a seeded 1 ref + 4 src PatchMatch problem (bitmaps, K/R/T, depth range, options) and
                                 the oracle's depth / normal / selection-probability maps for it.  The CUDA path must
                                 reproduce them bit for bit (tests/test_pm_gpu.py) and the oracle must keep producing
                                 them (tests/test_pm_cpu.py) - the fp32 contract is frozen by this file.
  pm_reference_cuda_160x120.npz  depth / normal maps the reference's own CUDA implementation produced for a seeded
                                 problem on a B200 (written by --reference).  Not bit-defined (texture filtering,
                                 --use_fast_math): tests compare statistics (tests/test_pm_gpu.py).
  pm_reference_cuda_480x270_grid.npz, pm_reference_cuda_1920x1080_grid.npz
                                 the reference PatchMatchCuda on the seeded scenes of the statistical-parity tests
                                 (written by --reference): its depth / normal maps on a regular pixel grid (every
                                 `step`-th row and column) and the whole-map statistics of its depth against the ground
                                 truth.  The scenes are regenerated from their seed by the tests.
  ba_reference_caspar.npz        the reference's Caspar bundle adjuster on the seeded problem of the cross-backend test
                                 (written by --reference): residual count, final cost, refined intrinsics.
  ba_case_small.npz              a seeded BA problem (8 images, 120 points) and the oracle's solution / summary.
"""
import argparse
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def pm_problem_arrays(sc):
    imgs = sc["images"]
    return dict(bitmaps=np.stack([im.bitmap for im in imgs]), K=np.stack([im.K for im in imgs]),
                R=np.stack([im.R for im in imgs]), T=np.stack([im.T for im in imgs]),
                depth_min=np.float64(sc["depth_min"]), depth_max=np.float64(sc["depth_max"]),
                depth_gt=sc["depth_gt"].astype(np.float32))


def pm_problem_from_arrays(z):
    from colmap_b200.patch_match import Image, Problem
    images = [Image(bitmap=np.ascontiguousarray(z["bitmaps"][i]), K=z["K"][i], R=z["R"][i], T=z["T"][i])
              for i in range(len(z["bitmaps"]))]
    return Problem(ref_image_idx=0, src_image_idxs=list(range(1, len(images))), images=images)


# statistical parity with the reference PatchMatchCuda: scene size -> grid step of the stored maps (3600 and 8160 pixels)
REFERENCE_PARITY = {(480, 270): 6, (1920, 1080): 16}


def reference_parity_case(w, h):
    """The seeded 8-source scene and the default options (5 iterations, photometric + filter) of the parity tests."""
    from colmap_b200.patch_match import PatchMatchOptions
    from colmap_b200.synthetic import make_patch_match_scene
    sc = make_patch_match_scene(w, h, 8, seed=0)
    o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], geom_consistency=False, gpu_index="0")
    return sc, o


def reference_parity_name(w, h):
    return f"pm_reference_cuda_{w}x{h}_grid.npz"


def depth_stats(depth, gt):
    """(valid fraction, median relative error, fraction within 1e-3 relative) of a depth map against the ground truth."""
    v = depth > 0
    rel = np.abs(depth - gt)[v] / gt[v]
    return float(v.mean()), float(np.median(rel)), float((rel < 1e-3).mean())


def caspar_case():
    """The seeded problem and options of the cross-backend test: 12 images sharing one SIMPLE_RADIAL camera, principal
    point refined, two-cams gauge."""
    from colmap_b200.bundle_adjustment import BundleAdjustmentOptions, SIMPLE_RADIAL
    from colmap_b200.synthetic import synthesize_ba_problem
    gt, noisy = synthesize_ba_problem(12, 2000, 8, models=(SIMPLE_RADIAL,), shared_camera=True, seed=13,
                                      point2D_stddev=0.5, point3D_stddev=0.1, translation_stddev=0.05, rotation_stddev_deg=0.3)
    noisy.pose_constant = noisy.pose_constant.copy(); noisy.pose_fixed_dim = noisy.pose_fixed_dim.copy()
    noisy.pose_constant[0] = 1
    noisy.pose_fixed_dim[1] = int(np.argmax(np.abs(noisy.poses[1, 4:] - noisy.poses[0, 4:])))
    return noisy, BundleAdjustmentOptions(refine_principal_point=True)


def make_pm_oracle_case(dst):
    import oracle_pm
    from colmap_b200.patch_match import PatchMatchOptions
    from colmap_b200.synthetic import make_patch_match_scene
    sc = make_patch_match_scene(96, 64, 4, seed=3)
    opts = dict(geom_consistency=False, num_iterations=2, filter=True)
    o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], **opts)
    out = oracle_pm.run(o, sc["problem"])
    np.savez_compressed(os.path.join(dst, "pm_case_96x64.npz"), **pm_problem_arrays(sc),
                        options=json.dumps(opts), depth=out["depth"], normal=out["normal"], sel_prob=out["sel_prob"],
                        mask=out["mask"])
    print("pm_case_96x64.npz: valid", float((out["depth"] > 0).mean()))


def make_pm_reference_case(dst):
    import ref_pm
    from colmap_b200.patch_match import PatchMatchOptions
    from colmap_b200.synthetic import make_patch_match_scene
    sc = make_patch_match_scene(160, 120, 4, seed=5)
    opts = dict(geom_consistency=False, num_iterations=5, filter=True)
    o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], **opts)
    out = ref_pm.run(o, sc["problem"])
    np.savez_compressed(os.path.join(dst, "pm_reference_cuda_160x120.npz"), **pm_problem_arrays(sc),
                        options=json.dumps(opts), depth=out["depth"], normal=out["normal"])
    print("pm_reference_cuda_160x120.npz ->", dst, "valid", float((out["depth"] > 0).mean()))


def make_pm_reference_parity_cases(dst):
    import ref_pm
    for (w, h), step in REFERENCE_PARITY.items():
        sc, o = reference_parity_case(w, h)
        out = ref_pm.run(o, sc["problem"])
        valid_frac, median_rel_err, frac_rel_err_lt_1e_3 = depth_stats(out["depth"], sc["depth_gt"])
        path = os.path.join(dst, reference_parity_name(w, h))
        np.savez_compressed(path, step=np.int64(step), depth=out["depth"][::step, ::step],
                            normal=out["normal"][:, ::step, ::step], valid_frac=np.float64(valid_frac),
                            median_rel_err=np.float64(median_rel_err), frac_rel_err_lt_1e_3=np.float64(frac_rel_err_lt_1e_3))
        print(os.path.basename(path), "->", dst, "valid", valid_frac, "median rel err", median_rel_err)


def make_caspar_reference_case(dst):
    import ref_caspar
    flat, o = caspar_case()
    r = ref_caspar.solve(flat, o)
    # no initial cost: the generated solver never writes caspar::SolveResult::initial_score (solver.cc:2408-2410)
    np.savez_compressed(os.path.join(dst, "ba_reference_caspar.npz"), num_residuals=np.int64(r["num_residuals"]),
                        final_cost=np.float64(r["final_cost"]), cam_params=flat.cam_params)
    print("ba_reference_caspar.npz ->", dst, "final cost", r["final_cost"], "intrinsics", flat.cam_params)


def make_ba_case(dst):
    import oracle_ba
    from colmap_b200.bundle_adjustment import BundleAdjustmentOptions, ITERATIVE_SCHUR, SIMPLE_RADIAL, PINHOLE
    from colmap_b200.synthetic import synthesize_ba_problem
    gt, noisy = synthesize_ba_problem(8, 120, 4, models=(SIMPLE_RADIAL, PINHOLE), seed=11)
    noisy.pose_constant = noisy.pose_constant.copy(); noisy.pose_fixed_dim = noisy.pose_fixed_dim.copy()
    noisy.pose_constant[0] = 1
    noisy.pose_fixed_dim[1] = int(np.argmax(np.abs(noisy.poses[1, 4:] - noisy.poses[0, 4:])))
    o = BundleAdjustmentOptions(linear_solver_type=ITERATIVE_SCHUR, max_num_iterations=30)
    sol = noisy.copy(); sol.pose_constant, sol.pose_fixed_dim = noisy.pose_constant, noisy.pose_fixed_dim
    s = oracle_ba.solve(o, sol)
    np.savez_compressed(
        os.path.join(dst, "ba_case_small.npz"),
        poses=noisy.poses, pose_constant=noisy.pose_constant, pose_fixed_dim=noisy.pose_fixed_dim,
        cam_model=noisy.cam_model, cam_off=noisy.cam_off, cam_params=noisy.cam_params, cam_constant=noisy.cam_constant,
        points=noisy.points, point_constant=noisy.point_constant, obs_pose=noisy.obs_pose, obs_cam=noisy.obs_cam,
        obs_point=noisy.obs_point, obs_xy=noisy.obs_xy,
        sol_poses=sol.poses, sol_cam_params=sol.cam_params, sol_points=sol.points,
        initial_cost=np.float64(s.initial_cost), final_cost=np.float64(s.final_cost),
        num_residuals=np.int64(s.num_residuals), num_effective_parameters=np.int64(s.num_effective_parameters),
        max_num_iterations=np.int64(30))
    print("ba_case_small.npz: cost", s.initial_cost, "->", s.final_cost, "steps", s.num_successful_steps, s.num_unsuccessful_steps)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", action="store_true")
    ap.add_argument("--out", default=HERE)
    a = ap.parse_args()
    json.load(open(os.path.join(HERE, "reference_known_answers.json")))
    os.makedirs(a.out, exist_ok=True)
    if a.reference:
        import ref_caspar
        import ref_pm
        if not (ref_pm.available() and ref_caspar.available()):
            raise SystemExit("oracle/_ref/libpm_ref.so or libcaspar_ref.so missing: build() makes them where the "
                             "reference sources are")
        make_pm_reference_case(a.out)
        make_pm_reference_parity_cases(a.out)
        make_caspar_reference_case(a.out)
    else:
        make_pm_oracle_case(a.out)
        make_ba_case(a.out)
