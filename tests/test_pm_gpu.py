"""GPU parity tier for the PatchMatch path: the CUDA kernels, called through the C-ABI, against the
CPU oracle on the same inputs.  Bar: bit-exact depth / normal / selection-probability / consistency
outputs (the oracle's fp32 contract is the spec the kernels implement)."""
import os

import numpy as np
import pytest

import oracle_pm
from colmap_b200.patch_match import PatchMatch, PatchMatchOptions, consistency_list_from_mask
from colmap_b200.synthetic import make_patch_match_scene

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _run_cuda(o, problem, wpc=None, fused=False, env=None):
    for k, v in (env or {}).items():
        os.environ[k] = str(v)
    if wpc is not None:
        os.environ["B200PM_WPC"] = str(wpc)
    os.environ.pop("B200PM_MAX_SWEEPS", None)
    os.environ["B200PM_FUSED"] = "1" if fused else "0"
    pm = PatchMatch(o, problem)
    pm.Run()
    out = dict(depth=pm.GetDepthMap(), normal=pm.GetNormalMap(), sel_prob=pm.GetSelProbMap())
    if o.filter:
        out["mask"] = pm.GetConsistencyMask()
        out["list"] = pm.GetConsistentImageIdxs()
    pm.close()
    os.environ.pop("B200PM_WPC", None)
    os.environ.pop("B200PM_FUSED", None)
    for k in (env or {}):
        os.environ.pop(k, None)
    return out


def _assert_bit_exact(got, ref, keys=("depth", "normal", "sel_prob")):
    for k in keys:
        eq = _bits(got[k]) == _bits(ref[k])
        assert eq.all(), f"{k}: {(~eq).sum()} of {eq.size} values differ"


def test_fast_reciprocal_is_ieee_over_all_floats():
    """The per-tap reciprocal (MUFU.RCP + one Newton step after clamping to [1e-30, 1e30]) must equal the
    correctly rounded division the oracle uses, for every one of the 2^32 float bit patterns."""
    import ctypes
    from colmap_b200 import load_library
    lib = load_library()
    lib.b200pm_test_rcp_exhaustive.restype = ctypes.c_longlong
    assert lib.b200pm_test_rcp_exhaustive() == 0


@pytest.mark.parametrize("wpc,fused", [(1, False), (2, False), (4, False), (1, True), (2, True), (4, True)])
def test_photometric_bit_exact_vs_oracle(wpc, fused):
    """Both schedules (split rand/pixel/serial passes = default, and the single fused sweep kernel) for every
    warps-per-column setting must reproduce the oracle bit for bit."""
    sc = make_patch_match_scene(96, 72, 4, seed=0)
    o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], geom_consistency=False,
                          num_iterations=2)
    got = _run_cuda(o, sc["problem"], wpc, fused)
    ref = oracle_pm.run(o, sc["problem"])
    _assert_bit_exact(got, ref)
    assert np.array_equal(got["mask"], ref["mask"])
    assert np.array_equal(got["list"], consistency_list_from_mask(ref["mask"], sc["problem"].src_image_idxs))


@pytest.mark.parametrize("prune,prune_from,chunks,geom", [
    (0, 0, 1, False),     # the pixel pass evaluates every (hypothesis, image) pair, one chunk: the round-1 schedule
    (1, 0, 3, False),     # prediction + exact early-out from the very first sweep (poor prediction: many late evaluations)
    (1, 1, 4, False),     # the default schedule
    (2, 0, 2, False),     # adversarial: the pixel pass evaluates NOTHING, the serial pass must fill every entry it needs
    (1, 0, 2, True), (2, 0, 1, True),
])
def test_early_out_schedules_are_exact(prune, prune_from, chunks, geom):
    """The pixel pass may skip (hypothesis, image) pairs - predicted unsampled, or ruled out because the partial cost sum
    already exceeds the current hypothesis' - and the serial pass re-checks / fills in with the true samples.  Whatever the
    pixel pass chose to evaluate, the result must be the oracle's, bit for bit."""
    sc = make_patch_match_scene(96, 72, 5, seed=3, with_gt_maps=geom)
    prob = sc["problem"]
    if geom:
        rng = np.random.default_rng(1)
        prob.depth_maps = [(d * (1 + 0.002 * rng.standard_normal(d.shape))).astype(np.float32) for d in sc["depth_maps"]]
        prob.normal_maps = [n.copy() for n in sc["normal_maps"]]
    o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], geom_consistency=geom, num_iterations=2,
                          num_samples=15 if not geom else 37)
    ref = oracle_pm.run(o, prob)
    for wpc in (1, 2):
        got = _run_cuda(o, prob, wpc=wpc, env=dict(B200PM_PRUNE=prune, B200PM_PRUNE_FROM=prune_from, B200PM_CHUNKS=chunks))
        _assert_bit_exact(got, ref)
        assert np.array_equal(got["mask"], ref["mask"])


@pytest.mark.parametrize("w,h,n,radius,step,samples", [
    (70, 50, 3, 3, 1, 7),      # ragged sizes, small window
    (64, 80, 8, 5, 2, 15),     # window_step 2, portrait, 8 sources
    (33, 17, 1, 2, 1, 4),      # single source image: filter_min_num_consistent=2 zeroes everything
    (50, 40, 5, 7, 1, 20),     # big window
    (36, 28, 2, 20, 2, 5),     # kMaxPatchMatchWindowRadius = 20 (41x41 window, step 2)
    (30, 24, 2, 14, 1, 3),     # 29x29 window: 841 taps, > 48 KB of dynamic shared memory in the pixel pass
    (40, 30, 3, 4, 1, 40),     # more than 32 Monte-Carlo samples
])
def test_option_grid_bit_exact(w, h, n, radius, step, samples):
    sc = make_patch_match_scene(w, h, n, seed=11)
    o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], geom_consistency=False,
                          num_iterations=1, window_radius=radius, window_step=step, num_samples=samples)
    got = _run_cuda(o, sc["problem"])
    ref = oracle_pm.run(o, sc["problem"])
    _assert_bit_exact(got, ref)
    assert np.array_equal(got["mask"], ref["mask"])


def test_no_filter_and_mixed_source_sizes():
    sc = make_patch_match_scene(80, 60, 3, seed=2)
    # crop one source image (different size than the reference; principal point unchanged)
    img = sc["images"][2]
    img.bitmap = np.ascontiguousarray(img.bitmap[:50, :70])
    o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], geom_consistency=False,
                          num_iterations=1, filter=False)
    got = _run_cuda(o, sc["problem"])
    ref = oracle_pm.run(o, sc["problem"])
    _assert_bit_exact(got, ref)
    assert (got["depth"] > 0).all()


def test_geometric_consistency_bit_exact():
    sc = make_patch_match_scene(80, 60, 4, seed=4, with_gt_maps=True)
    prob = sc["problem"]
    # photometric maps stand in: ground truth + noise for the sources, for the reference
    rng = np.random.default_rng(0)
    prob.depth_maps = [(d * (1 + 0.002 * rng.standard_normal(d.shape))).astype(np.float32) for d in sc["depth_maps"]]
    prob.depth_maps[2][10:20, 10:30] = 0.0          # holes -> max cost
    prob.normal_maps = [n.copy() for n in sc["normal_maps"]]
    o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], geom_consistency=True,
                          num_iterations=1)
    ref = oracle_pm.run(o, prob)
    for fused in (False, True):
        got = _run_cuda(o, prob, fused=fused)
        _assert_bit_exact(got, ref)
        assert np.array_equal(got["mask"], ref["mask"])


def test_rerun_on_resident_inputs_is_reproducible():
    sc = make_patch_match_scene(64, 48, 3, seed=9)
    o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], geom_consistency=False,
                          num_iterations=1)
    pm = PatchMatch(o, sc["problem"])
    pm.Run()
    a = pm.GetDepthMap()
    pm.RunOnly()
    b = pm.GetDepthMap()
    pm.close()
    assert np.array_equal(_bits(a), _bits(b))


def test_full_hd_properties():
    """BASELINE config C2 size (1 ref + 8 src, 1920x1080, window 11) with fewer iterations: properties
    that do not need the oracle."""
    sc = make_patch_match_scene(1920, 1080, 8, seed=0)
    o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], geom_consistency=False,
                          num_iterations=2)
    got = _run_cuda(o, sc["problem"])
    d = got["depth"]
    valid = d > 0
    assert valid.mean() > 0.85
    inside = (d[valid] >= sc["depth_min"]) & (d[valid] <= sc["depth_max"])
    assert inside.mean() > 0.999
    rel = np.abs(d - sc["depth_gt"])[valid] / sc["depth_gt"][valid]
    assert np.median(rel) < 5e-3
    nn = np.linalg.norm(got["normal"][:, valid], axis=0)
    assert np.allclose(nn, 1, atol=1e-4)
    assert (got["normal"][:, ~valid] == 0).all() and (got["mask"][:, ~valid] == 0).all()
    assert (got["mask"][:, valid].sum(axis=0) >= 2).all()
    assert np.isfinite(got["sel_prob"]).all() and (got["sel_prob"] >= 0).all() and (got["sel_prob"] <= 1).all()


def _reference_parity(w, h):
    """Runs the CUDA path on the scene of make_golden.reference_parity_case and loads what COLMAP's own
    patch_match_cuda.cu (unmodified, built against stub headers, PTX JIT) produced for it: whole-map statistics of its
    depth against the ground truth, and its depth / normal maps on a regular pixel grid.  Returns (stored fixture,
    whole-map statistics of our depth, our depth and normal on the same grid)."""
    import make_golden
    sc, o = make_golden.reference_parity_case(w, h)
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", make_golden.reference_parity_name(w, h)))
    got = _run_cuda(o, sc["problem"])
    s = int(z["step"])
    return z, make_golden.depth_stats(got["depth"], sc["depth_gt"]), got["depth"][::s, ::s], got["normal"][:, ::s, ::s]


def test_statistical_parity_with_the_real_reference_cuda():
    """tests/golden/pm_reference_cuda_480x270_grid.npz: the reference PatchMatchCuda on a 480x270 scene.  It is
    stochastic and numerically different (fast-math, texture filtering), so the comparison is statistical: same
    completeness and accuracy against the analytic ground truth over the whole map, and per-pixel agreement of the two
    depth maps on the stored grid (3600 pixels)."""
    ref, (vb, mb, fb), depth, normal = _reference_parity(480, 270)
    va, ma, fa = float(ref["valid_frac"]), float(ref["median_rel_err"]), float(ref["frac_rel_err_lt_1e_3"])
    assert abs(va - vb) < 0.01 and abs(fa - fb) < 0.02 and mb < 2 * ma + 1e-5
    both = (ref["depth"] > 0) & (depth > 0)
    dd = np.abs(ref["depth"] - depth)[both]
    assert both.mean() > 0.97
    assert (dd < 1e-3).mean() > 0.8          # depth ~ 5 m: 1e-3 m = 2e-4 relative
    assert (dd < 1e-4).mean() > 0.25         # north_star: within 1e-4 m where both converge
    nn = (ref["normal"] * normal).sum(0)[both]
    assert np.median(nn) > 0.999


# ---------------------------------------------------------------- committed golden fixtures (tests/golden/)
def test_golden_fixture_bit_exact():
    """tests/golden/pm_case_96x64.npz (inputs + the oracle's frozen outputs): the CUDA path reproduces the stored maps
    bit for bit without the oracle being run."""
    import json
    import make_golden
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pm_case_96x64.npz"))
    o = PatchMatchOptions(depth_min=float(z["depth_min"]), depth_max=float(z["depth_max"]), **json.loads(str(z["options"])))
    got = _run_cuda(o, make_golden.pm_problem_from_arrays(z))
    _assert_bit_exact(got, {k: z[k] for k in ("depth", "normal", "sel_prob")})
    assert np.array_equal(got["mask"], z["mask"])


def test_golden_reference_cuda_fixture_statistics():
    """tests/golden/pm_reference_cuda_160x120.npz: maps produced by the UNMODIFIED reference PatchMatchCuda on a B200
    (tests/golden/make_golden.py --reference).  The reference is not bit-defined (texture filtering, fast-math), so the
    comparison is statistical: completeness, accuracy against the analytic ground truth, per-pixel agreement.
    Tolerance: 1e-4 m median / 1e-3 relative per pixel where both converge (BASELINE north_star)."""
    import json
    import make_golden
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pm_reference_cuda_160x120.npz")
    if not os.path.exists(path):
        pytest.skip("reference fixture not generated yet")
    z = np.load(path)
    o = PatchMatchOptions(depth_min=float(z["depth_min"]), depth_max=float(z["depth_max"]), **json.loads(str(z["options"])))
    got = _run_cuda(o, make_golden.pm_problem_from_arrays(z))
    ours, ref, gt = got["depth"], z["depth"], z["depth_gt"]
    v_ours, v_ref = ours > 0, ref > 0
    assert abs(v_ours.mean() - v_ref.mean()) < 0.03
    both = v_ours & v_ref
    assert both.mean() > 0.8
    err_ours = np.median(np.abs(ours[both] - gt[both]) / gt[both])
    err_ref = np.median(np.abs(ref[both] - gt[both]) / gt[both])
    assert err_ours < 1e-3 and err_ours < 1.5 * err_ref + 1e-5   # 160x120: both sit at ~3.5e-4 (pixel footprint)
    rel = np.abs(ours[both] - ref[both]) / ref[both]
    assert np.median(rel) < 1e-4                    # 5 m scene: 1e-4 relative = 0.5 mm
    assert (rel < 1e-3).mean() > 0.9
    n_dot = (got["normal"] * z["normal"]).sum(0)[both]
    assert np.median(n_dot) > 0.999


# ---------------------------------------------------------------- BASELINE sizes
def test_c2_full_size_bit_exact_vs_oracle():
    """BASELINE config C2 at FULL size (1 ref + 8 src, 1920x1080, window 11, 15 samples), one iteration = all four
    sweep directions + the filter: depth / normal / selection probabilities / consistency mask bit for bit against the
    oracle (which needs ~35 s on the box's host threads for this)."""
    sc = make_patch_match_scene(1920, 1080, 8, seed=0)
    o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], geom_consistency=False,
                          window_radius=5, window_step=1, num_samples=15, num_iterations=1)
    got = _run_cuda(o, sc["problem"])
    ref = oracle_pm.run(o, sc["problem"])
    _assert_bit_exact(got, ref)
    assert np.array_equal(got["mask"], ref["mask"])


def test_c2_full_size_statistical_parity_with_the_real_reference_cuda():
    """C2 (all 5 iterations) against COLMAP's own PatchMatchCuda (tests/golden/pm_reference_cuda_1920x1080_grid.npz).
    STATISTICAL parity (the reference is stochastic in its float details: fast-math, 9-bit texture weights): the figures
    of profiles/pm_ref_compare_1920x1080.json (61 % of pixels within 1e-4 m, 98.7 % within 1e-3 m, 5 m scene) pinned
    with a margin; whole-map completeness and accuracy, per-pixel agreement on the stored grid (8160 pixels)."""
    ref, (vb, eb, _), depth, normal = _reference_parity(1920, 1080)
    va, ea = float(ref["valid_frac"]), float(ref["median_rel_err"])
    assert abs(va - vb) < 0.005 and vb > 0.99
    assert eb < 1.5 * ea + 1e-6 and eb < 5e-5
    both = (ref["depth"] > 0) & (depth > 0)
    dd = np.abs(ref["depth"] - depth)[both]
    assert (dd < 1e-4).mean() > 0.55          # north_star: within 1e-4 m where both converge
    assert (dd < 1e-3).mean() > 0.97
    assert np.median((ref["normal"] * normal).sum(0)[both]) > 0.9999


def test_two_phase_with_device_resident_maps_equals_the_host_round_trip():
    """SURVEY 8(e) geometric exchange: the photometric maps exported device-to-device (b200pm_get_*_device) and handed to
    the geometric problems as device pointers (b200pm_problem::maps_on_device) give bit-identical results to the
    reference's contract (host maps in, host maps out)."""
    import torch
    from colmap_b200.workspace import run_two_phase
    sc = make_patch_match_scene(96, 72, 3, seed=6)
    images = sc["images"]
    srcs = [[j for j in range(4) if j != i] for i in range(4)]
    o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], num_iterations=1, gpu_index="0")
    host = run_two_phase(images, srcs, o, 0, 1)
    dev = run_two_phase(images, srcs, o, 0, 1, device=torch.device("cuda", 0))
    for i in range(4):
        assert np.array_equal(_bits(host[i][0]), _bits(dev[i][0])) and np.array_equal(_bits(host[i][1]), _bits(dev[i][1]))
        assert (dev[i][0] > 0).mean() > 0.5
