#!/usr/bin/env python
"""bench.py — headline benchmark of the two hot paths (BASELINE.json).

Primary line (one JSON object on stdout, rank 0): PatchMatch Mpixels/s on config C2
("PatchMatch: 1 ref + 8 src views, 1920x1080, window 11, 5 iters, 1 GPU"); one reference image per
GPU (weak scaling, no data-path collective in photometric mode).  The BA metric (LM iterations/s on
B3) rides along under the "ba" key when the BA path is built.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

value  : device-resident (inputs already in HBM), CUDA-event time of b200pm_run, max over ranks.
e2e    : the same metric through the public API with HOST (pinned) buffers: create (H2D + prefilter +
         init) + run + depth/normal read-back (D2H) + destroy, wall clock around synchronous calls.
roofline / cpu_baseline: see DESIGN.md §5.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C2 = dict(width=1920, height=1080, num_src=8, window_radius=5, window_step=1, num_samples=15, num_iterations=5)
# one string for both arms (the driver compares config.workload of the two lines)
C2_WORKLOAD = ("PatchMatch C2: 1 ref + 8 src views, 1920x1080, window 11, 15 samples, 5 iters, photometric + filter; "
               "one reference image per GPU")
B3_WORKLOAD = ("BA B3: 500 cameras (SIMPLE_RADIAL, own intrinsics), 300k points, 2M observations, ITERATIVE_SCHUR + "
               "SCHUR_JACOBI, two-cams gauge, trivial loss, 100 LM iterations max")


def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for k, nm in enumerate(names):
                if len(r) > 5 + k and r[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=(max(mx) if mx else None),
                    reasons=sorted(reasons), samples=len(sm))


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def _ncu_traffic(name):
    """per-launch DRAM traffic of the dominant kernel from the committed ncu summary, or None."""
    path = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(path):
        with open(path) as f:
            v = json.load(f).get(name)
            return v.get("bytes") if isinstance(v, dict) else v
    return None


def _use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU legs (rank 0 only) are meant to use every host core.  The
    oracles are OpenMP code on the process' libgomp, so the team size is raised there.  Returns the thread count in use."""
    import ctypes
    n = os.cpu_count() or 1
    try:
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(n)
    except OSError:
        n = int(os.environ.get("OMP_NUM_THREADS", n))
    return n


def _oracle_pm_sample(threads=None):
    """Bounded CPU sample of the same workload with the oracle: a 240x136 crop-scale scene (1/63.5 of the
    pixels of C2), 8 sources, the full 5 iterations; Mpixels/s is per reference pixel so it is comparable."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_pm
    from colmap_b200.patch_match import PatchMatchOptions
    from colmap_b200.synthetic import make_patch_match_scene
    w, h = 240, 136
    sc = make_patch_match_scene(w, h, C2["num_src"], seed=0)
    o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], geom_consistency=False,
                          window_radius=C2["window_radius"], num_iterations=C2["num_iterations"])
    _use_all_host_threads()
    t = time.time()
    oracle_pm.run(o, sc["problem"])
    dt = time.time() - t
    return w * h / 1e6 / dt, dt, f"{w}x{h} scene, {C2['num_src']} src, window 11, 5 iterations (all sweeps), oracle port"


B3 = dict(num_images=500, num_points=300000, num_obs=2000000)


def _b3_problem():
    import numpy as np
    from colmap_b200.bundle_adjustment import SIMPLE_RADIAL
    from colmap_b200.synthetic import synthesize_ba_problem
    gt, noisy = synthesize_ba_problem(B3["num_images"], B3["num_points"], 7, models=(SIMPLE_RADIAL,), seed=42,
                                      num_obs=B3["num_obs"])
    noisy.pose_constant = noisy.pose_constant.copy(); noisy.pose_fixed_dim = noisy.pose_fixed_dim.copy()
    noisy.pose_constant[0] = 1                                   # TWO_CAMS_FROM_WORLD gauge
    noisy.pose_fixed_dim[1] = int(np.argmax(np.abs(noisy.poses[1, 4:] - noisy.poses[0, 4:])))
    return noisy


def _fresh(noisy):
    f = noisy.copy()
    f.pose_constant, f.pose_fixed_dim = noisy.pose_constant, noisy.pose_fixed_dim
    return f


def _oracle_ba_sample(noisy, max_iters=100):
    """CPU leg: the same B3 problem and the SAME iteration limit as the GPU arm (100 LM iterations), oracle port, all
    host threads (about 10-30 s)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_ba
    from colmap_b200.bundle_adjustment import ITERATIVE_SCHUR, BundleAdjustmentOptions
    o = BundleAdjustmentOptions(linear_solver_type=ITERATIVE_SCHUR, max_num_iterations=max_iters)
    _use_all_host_threads()
    t = time.time()
    s = oracle_ba.solve(o, _fresh(noisy))
    dt = time.time() - t
    steps = s.num_successful_steps + s.num_unsuccessful_steps
    return steps / dt, dt, f"B3 problem (500 cams, 300k pts, 2M obs), full solve ({steps} LM iterations, limit {max_iters}), ITERATIVE_SCHUR, oracle port"


DUMP_LIMIT = 64 << 20      # bytes that --dump-outputs may write in all
DUMP_SAMPLE = 1 << 17      # rows kept of an output too large to store whole


def _fixed_sample(n, k=DUMP_SAMPLE):
    """Sorted indices of a seeded sample of k of range(n) (all of them when n <= k): the same rows in every run."""
    import numpy as np
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, k, replace=False))


def _ba_outputs(prefix, flat, summary, sample_points=False):
    """What a caller of solve_flat receives: the refined blocks of `flat` and the summary's costs."""
    import numpy as np
    pts = flat.points[_fixed_sample(len(flat.points))] if sample_points else flat.points
    return {f"{prefix}_poses": flat.poses, f"{prefix}_cam_params": flat.cam_params, f"{prefix}_points": pts,
            f"{prefix}_cost": np.array([summary.initial_cost, summary.final_cost], np.float64)}


def dump_outputs(directory, outputs):
    """Writes every array of `outputs` as DIR/<name>.npy in float32 / float64 (integer and mask arrays as float32)."""
    import numpy as np
    arrays = {k: np.ascontiguousarray(v if v.dtype in (np.float32, np.float64) else v.astype(np.float32))
              for k, v in outputs.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(directory, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), a)


def bench_ba(steps, warmup, peak, peak_src, with_cpu, outputs=None):
    """BA leg: LM iterations/s on config B3 (500 SIMPLE_RADIAL cameras, 300k points, 2M observations, Schur-PCG).
    `outputs`, when given, receives the solution of the last timed solve."""
    from colmap_b200.bundle_adjustment import ITERATIVE_SCHUR, BundleAdjustmentOptions, solve_flat
    noisy = _b3_problem()
    o = BundleAdjustmentOptions(linear_solver_type=ITERATIVE_SCHUR)
    for _ in range(max(warmup, 1)):
        solve_flat(o, _fresh(noisy))
    lm, dev_ms, wall_ms, spmv_ms, spmv_n, launches = 0, 0.0, 0.0, 0.0, 0, 0
    for _ in range(steps):
        f = _fresh(noisy)
        t = time.time()
        s = solve_flat(o, f)                       # host arrays in, host arrays out (H2D/D2H inside)
        wall_ms += (time.time() - t) * 1e3
        lm += s.num_successful_steps + s.num_unsuccessful_steps
        dev_ms += s.solve_ms; spmv_ms += s.spmv_ms_total; spmv_n += s.spmv_launches; launches += s.kernel_launches
    nobs = B3["num_obs"]
    spmv_launch_ms = spmv_ms / max(spmv_n, 1)
    alg = 192 * nobs                                # SURVEY.md §8(d): 2*(8*dc+24+8) B per observation per PCG iteration, dc = 8
    achieved = alg / (spmv_launch_ms * 1e-3) / 1e9
    h2d = f.poses.nbytes + f.cam_params.nbytes + f.points.nbytes + f.obs_xy.nbytes + 3 * f.obs_pose.nbytes
    d2h = f.poses.nbytes + f.cam_params.nbytes + f.points.nbytes
    out = {"metric": "ba_lm_iterations_per_s", "value": lm / (dev_ms * 1e-3), "unit": "LM iterations/s", "dtype": "f64",
           "ms_per_step": dev_ms / steps, "lm_iterations_per_solve": lm / steps,
           "config": {"workload": B3_WORKLOAD},
           "e2e": {"value": lm / (wall_ms * 1e-3), "unit": "LM iterations/s", "h2d_bytes_per_step": int(h2d),
                   "d2h_bytes_per_step": int(d2h), "ms_per_step": wall_ms / steps},
           "final_cost": s.final_cost, "termination_type": s.termination_type, "gpu_launches": int(launches),
           "roofline": {"bound": "hbm", "kernel": "ba_schur_spmv_warp_smem_kernel + ba_cam_stream_loop_kernel (one implicit-Schur product)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                        "frac": achieved / peak, "traffic": _ncu_traffic("ba_schur_spmv_kernel"), "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": alg, "launch_ms": spmv_launch_ms}}
    if outputs is not None:
        outputs.update(_ba_outputs("ba_b3", f, s))
    if with_cpu:
        v, dt, sample = _oracle_ba_sample(noisy)
        out["cpu_baseline"] = {"value": v, "unit": "LM iterations/s", "cores": os.cpu_count(), "kind": "port",
                               "sample": sample, "seconds": dt}
    return out



C4 = dict(width=3840, height=2160, num_src=20, images_total=200, images_per_gpu_default=3)
C4_WORKLOAD = ("PatchMatch C4: 200-image workspace, 4K frames (3840x2160), 20 source images per reference image, window 11, "
               "5 iters, geometric consistency (photometric pass, NCCL all-gather of the depth maps, geometric pass + "
               "filter), 8 GPUs")
B5 = dict(num_images=2000, num_points=2000000, num_obs=12000000)
B5_WORKLOAD = ("BA B5: 2000 cameras (PINHOLE / SIMPLE_RADIAL 50/50, own intrinsics), 2M points, 12M observations, "
               "ITERATIVE_SCHUR + SCHUR_JACOBI, points sharded over the ranks")


def bench_c4(rank, world, local_rank, images_total):
    """C4-shaped leg: `images_total` 4K views of one scene, every view a reference image with its 20 nearest views as
    sources, the reference's two-phase schedule (patch_match.cc:176-204) sharded over the ranks; the photometric depth
    maps stay in HBM and cross the ranks in ONE NCCL all-gather (colmap_b200/workspace.py).  Mpixels/s = reference
    pixels of FINAL (geometric, filtered) maps per second of the whole two-phase run, host bitmaps in, host maps out."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from colmap_b200.patch_match import PatchMatchOptions
    from colmap_b200.sharding import max_over_ranks
    from colmap_b200.synthetic import make_workspace_scene
    from colmap_b200.workspace import run_two_phase
    dev = torch.device("cuda", local_rank)
    sc = make_workspace_scene(C4["width"], C4["height"], images_total, seed=7, device=dev)
    n = images_total
    cen = sc["centers"]
    nsrc = min(C4["num_src"], n - 1)
    srcs = []
    for i in range(n):
        order = np.argsort(np.linalg.norm(cen - cen[i], axis=1), kind="stable")
        srcs.append([int(j) for j in order if j != i][:nsrc])
    o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], geom_consistency=True, window_radius=5,
                          num_samples=15, num_iterations=5, gpu_index=str(local_rank))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.time()
    out = run_two_phase(sc["images"], srcs, o, rank, world, device=dev)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    dt = max_over_ranks(time.time() - t0, "cuda") if world > 1 else time.time() - t0
    mine = sorted(out)
    valid = float(np.mean([(out[i][0] > 0).mean() for i in mine])) if mine else 0.0
    rel = [np.median(np.abs(out[i][0] - sc["depth_gt"][i])[out[i][0] > 0] / sc["depth_gt"][i][out[i][0] > 0]) for i in mine]
    mpix = n * C4["width"] * C4["height"] / 1e6
    return {"metric": "patchmatch_mpixels_per_s", "value": mpix / dt, "unit": "Mpixels/s", "n_gpus": world, "seconds": dt,
            "config": {"workload": C4_WORKLOAD, "images_run": n, "images_of_config": C4["images_total"],
                       "sources_per_image": nsrc,
                       "note": ("the full 200-image configuration" if n == C4["images_total"] else
                                f"bounded sample of the configuration: {n} of its 200 images (same frames, sources, options, "
                                "schedule and exchange), so that the default bench run ends within minutes")},
            "exchange": "NCCL all-gather of device-resident depth maps (no host round trip)",
            "quality": {"valid_frac": valid, "median_rel_depth_err": float(np.median(rel)) if rel else None}}


def bench_b5(steps, warmup, rank, world, local_rank, comm, outputs=None):
    """BA leg on config B5 (2000 cameras, 2M points, 12M observations, mixed models), points sharded over the ranks.
    `outputs`, when given, receives the solution of the last timed solve (a fixed sample of the points)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from colmap_b200.bundle_adjustment import (ITERATIVE_SCHUR, PINHOLE, SIMPLE_RADIAL, BundleAdjustmentOptions, shard_flat_problem,
                                               solve_flat, solve_flat_sharded)
    from colmap_b200.sharding import max_over_ranks
    from colmap_b200.synthetic import synthesize_ba_problem
    gt, noisy = synthesize_ba_problem(B5["num_images"], B5["num_points"], 6, models=(PINHOLE, SIMPLE_RADIAL), seed=42,
                                      num_obs=B5["num_obs"])
    noisy.pose_constant = noisy.pose_constant.copy(); noisy.pose_fixed_dim = noisy.pose_fixed_dim.copy()
    noisy.pose_constant[0] = 1
    noisy.pose_fixed_dim[1] = int(np.argmax(np.abs(noisy.poses[1, 4:] - noisy.poses[0, 4:])))
    o = BundleAdjustmentOptions(linear_solver_type=ITERATIVE_SCHUR, gpu_index=local_rank)
    lm, dev_ms, wall_ms, s = 0, 0.0, 0.0, None
    for i in range(max(warmup, 1) + steps):
        if world > 1:
            local = shard_flat_problem(noisy, rank, world)
            torch.cuda.synchronize(); dist.barrier()
            t = time.time()
            s = solve_flat_sharded(o, local, comm)
            torch.cuda.synchronize(); dist.barrier()
        else:
            local = _fresh(noisy)
            t = time.time()
            s = solve_flat(o, local)
        if i >= max(warmup, 1):
            wall_ms += (time.time() - t) * 1e3
            lm += s.num_successful_steps + s.num_unsuccessful_steps
            dev_ms += s.solve_ms
    if world > 1:
        dev_ms = max_over_ranks(dev_ms, "cuda"); wall_ms = max_over_ranks(wall_ms, "cuda")
    elif outputs is not None:
        outputs.update(_ba_outputs("ba_b5", local, s, sample_points=True))
    return {"metric": "ba_lm_iterations_per_s", "value": lm / (dev_ms * 1e-3), "unit": "LM iterations/s", "dtype": "f64",
            "n_gpus": world, "scaling": "strong", "ms_per_step": dev_ms / steps, "lm_iterations_per_solve": lm / steps,
            "config": {"workload": B5_WORKLOAD},
            "e2e": {"value": lm / (wall_ms * 1e-3), "unit": "LM iterations/s", "ms_per_step": wall_ms / steps},
            "final_cost": s.final_cost, "initial_cost": s.initial_cost, "termination_type": s.termination_type,
            "pcg_iterations_per_solve": s.num_linear_solver_iterations}


def bench_ba_sharded(steps, warmup, rank, world, local_rank, with_b5=False):
    """BA leg at N > 1: the same B3 problem, points sharded over the ranks (strong scaling), one all-reduce of the
    camera-side vector per PCG iteration inside b200ba_solve_sharded (the library's peer-memory kernel; NCCL only for
    the set-up exchanges and as the fallback when peers cannot map each other)."""
    import torch
    import torch.distributed as dist
    from colmap_b200.bundle_adjustment import (ITERATIVE_SCHUR, BAComm, BundleAdjustmentOptions, shard_flat_problem,
                                               solve_flat_sharded)
    noisy = _b3_problem()
    idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        idt.copy_(torch.tensor(list(BAComm.unique_id()), dtype=torch.uint8))
    dist.broadcast(idt, src=0)
    comm = BAComm(bytes(idt.cpu().tolist()), rank, world)
    o = BundleAdjustmentOptions(linear_solver_type=ITERATIVE_SCHUR, gpu_index=local_rank)
    lm, dev_ms, wall_ms = 0, 0.0, 0.0
    for i in range(max(warmup, 1) + steps):
        local = shard_flat_problem(noisy, rank, world)
        torch.cuda.synchronize(); dist.barrier()
        t = time.time()
        s = solve_flat_sharded(o, local, comm)
        torch.cuda.synchronize(); dist.barrier()
        if i >= max(warmup, 1):
            wall_ms += (time.time() - t) * 1e3
            lm += s.num_successful_steps + s.num_unsuccessful_steps
            dev_ms += s.solve_ms
    b5 = None
    if with_b5:
        try:
            b5 = bench_b5(steps, 1, rank, world, local_rank, comm)
        except Exception as e:
            b5 = {"error": repr(e)}
    collective = ("one-shot all-reduce kernel over NVLink peer memory (cudaIpc symmetric buffers), one launch per collective"
                  if comm.peer_memory() else "ncclAllReduce")
    comm.close()
    from colmap_b200.sharding import max_over_ranks
    dev_ms = max_over_ranks(dev_ms, "cuda"); wall_ms = max_over_ranks(wall_ms, "cuda")
    out = {"metric": "ba_lm_iterations_per_s", "value": lm / (dev_ms * 1e-3), "unit": "LM iterations/s", "dtype": "f64",
           "n_gpus": world, "scaling": "strong", "ms_per_step": dev_ms / steps, "lm_iterations_per_solve": lm / steps,
           "config": {"workload": B3_WORKLOAD + "; points sharded over the ranks", "collective": collective},
           "e2e": {"value": lm / (wall_ms * 1e-3), "unit": "LM iterations/s", "ms_per_step": wall_ms / steps},
           "final_cost": s.final_cost, "termination_type": s.termination_type,
           "pcg_iterations_per_solve": s.num_linear_solver_iterations}
    if b5 is not None:
        out["b5"] = b5
    return out


def run_reference(args, rank, world, local_rank):
    """Reference arm.  COLMAP has no CPU implementation of PatchMatch (exe/mvs.cc:260 aborts without CUDA): its
    implementation of this path IS mvs/patch_match_cuda.cu.  When oracle/_ref/libpm_ref.so exists (the reference's
    own CUDA sources compiled in place against stub headers, oracle/build_ref.sh, as compute_90 PTX that the driver
    JITs - upstream's Blackwell configuration) this arm times it on the full C2 workload through the same host-buffer
    entry (constructor + Run + GetDepthMap/GetNormalMap), on EVERY rank (one reference image per GPU, like our arm),
    max over ranks.  Otherwise it falls back to the CPU oracle port on a bounded sample (rank 0).  The BA leg times
    (a) the reference's own GPU backend, Caspar (oracle/_ref/libcaspar_ref.so, when built) and (b) the fp64 oracle
    port on the host threads (Ceres is not installed in this image)."""
    cores = os.cpu_count()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    line = None
    try:
        import ref_pm
        have_ref = ref_pm.available()
    except Exception:
        have_ref = False
    torch = None
    if have_ref:
        try:
            import torch
            have_ref = torch.cuda.is_available()
        except Exception:
            have_ref = False
    if not have_ref and rank != 0:
        return
    distributed = have_ref and world > 1
    if distributed:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if have_ref:
        from colmap_b200.patch_match import PatchMatchOptions
        from colmap_b200.synthetic import make_patch_match_scene
        sc = make_patch_match_scene(C2["width"], C2["height"], C2["num_src"], seed=rank)
        o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], geom_consistency=False,
                              window_radius=C2["window_radius"], window_step=C2["window_step"],
                              num_samples=C2["num_samples"], num_iterations=C2["num_iterations"], gpu_index=str(local_rank))
        for _ in range(args.warmup):              # the first call also pays the PTX JIT (~1 min)
            ref_pm.run(o, sc["problem"])
        if distributed:
            torch.cuda.synchronize(); dist.barrier()
        t0 = time.time()
        for _ in range(args.steps):
            ref_pm.run(o, sc["problem"])
        if distributed:
            torch.cuda.synchronize(); dist.barrier()
        t = (time.time() - t0) * 1e3 / args.steps
        if distributed:
            from colmap_b200.sharding import max_over_ranks
            t = max_over_ranks(t, "cuda")
        v = world * C2["width"] * C2["height"] / 1e6 / (t * 1e-3)
        sample = "full C2 workload; reference PatchMatchCuda (unmodified sources, compute_90 PTX JIT) on the same GPU(s)"
        line = {"impl": "reference", "metric": "patchmatch_mpixels_per_s", "value": v, "unit": "Mpixels/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": t, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": C2_WORKLOAD,
                           "l2": "inputs larger than L2: cost/sel-prob maps 3 x 66 MB + 66 MB source footprints vs 126 MB L2",
                           "parallelism": f"problems x{world} (no collective)",
                           "note": "the reference implementation of this path is CUDA (no CPU PatchMatch exists in "
                                   "COLMAP); timed end to end with host buffers"},
                "cpu_baseline": {"value": v, "unit": "Mpixels/s", "cores": 0, "kind": "reference", "sample": sample},
                "e2e": {"value": v, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
    else:
        vals = []
        for i in range(args.warmup + args.steps):
            v, dt, sample = _oracle_pm_sample()
            if i >= args.warmup:
                vals.append((v, dt))
        v = sum(x[0] for x in vals) / len(vals)
        ms = 1e3 * sum(x[1] for x in vals) / len(vals)
        line = {"impl": "reference", "metric": "patchmatch_mpixels_per_s", "value": v, "unit": "Mpixels/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": C2_WORKLOAD, "sample": sample},
                "cpu_baseline": {"value": v, "unit": "Mpixels/s", "cores": cores, "kind": "port", "sample": sample},
                "e2e": {"value": v, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
    if rank == 0 and not args.no_ba:
        ba = {"impl": "reference", "metric": "ba_lm_iterations_per_s", "unit": "LM iterations/s",
              "config": {"workload": B3_WORKLOAD}}
        try:
            noisy = _b3_problem()
            try:
                ba["caspar"] = _caspar_ba(noisy, args.steps, args.warmup)
                ba["value"] = ba["caspar"]["value"]
            except Exception as e:
                ba["caspar"] = {"unavailable": repr(e)}
            v, dt, sample = _oracle_ba_sample(noisy)
            ba["cpu_baseline"] = {"value": v, "unit": "LM iterations/s", "cores": cores, "kind": "port", "sample": sample,
                                  "seconds": dt}
            ba.setdefault("value", v)
            ba["note"] = ("Ceres is not installed in this image; `caspar` is the reference's own GPU backend (fp32), "
                          "`cpu_baseline` the fp64 oracle port that restates Ceres' algorithm")
        except Exception as e:
            ba["error"] = repr(e)
        line["ba"] = ba
    if rank == 0:
        print(json.dumps(line), flush=True)
    if distributed:
        dist.destroy_process_group()


def _caspar_ba(noisy, steps, warmup):
    """The reference's CasparBundleAdjuster core (thirdparty Symforce-Caspar generated solver, compiled in place into
    oracle/_ref/libcaspar_ref.so by oracle/build_ref.sh) on the same flat problem."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import ref_caspar
    if not ref_caspar.available():
        raise RuntimeError("oracle/_ref/libcaspar_ref.so not built")
    out = None
    for i in range(max(warmup, 1) + steps):
        r = ref_caspar.solve(_fresh(noisy))
        if i == max(warmup, 1):
            out = dict(lm=0, ms=0.0)
        if out is not None:
            out["lm"] += r["iterations"]; out["ms"] += r["solve_ms"]
    return {"value": out["lm"] / (out["ms"] * 1e-3), "unit": "LM iterations/s", "kind": "reference (Caspar, fp32, GPU)",
            "lm_iterations_per_solve": out["lm"] / steps, "ms_per_step": out["ms"] / steps, "final_cost": r["final_cost"],
            "setup_ms": r["setup_ms"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ba", action="store_true")
    ap.add_argument("--c4-images", type=int, default=-1,
                    help="images of the C4-shaped workspace leg: -1 = 3 per GPU when 8 GPUs run (the configuration's GPU count), "
                         "else skipped; 0 = skip; 200 = the full configuration")
    ap.add_argument("--b5", type=int, default=1, help="BA config B5 leg (2000 cameras, 2M points, 12M observations; strong scaling over the ranks): 1 = run, 0 = skip")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of each single-GPU leg returned (rank 0) as DIR/<name>.npy, so that "
                         "two builds can be compared output for output; the inputs are seeded")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")

    rank = _env_int("RANK", 0)
    world = _env_int("WORLD_SIZE", 1)
    local_rank = _env_int("LOCAL_RANK", 0)

    if args.impl == "reference":
        run_reference(args, rank, world, local_rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: colmap_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from colmap_b200.patch_match import PatchMatch, PatchMatchOptions
    from colmap_b200.synthetic import make_patch_match_scene

    # one reference image (problem) per GPU: the reference's own multi-GPU mode (patch_match.cc:176-205)
    sc = make_patch_match_scene(C2["width"], C2["height"], C2["num_src"], seed=rank)
    # pinned host copies of the inputs (the e2e leg uploads from these)
    for im in sc["images"]:
        t = torch.empty(im.bitmap.shape, dtype=torch.uint8, pin_memory=True)
        t.numpy()[...] = im.bitmap
        im._pinned = t
        im.bitmap = t.numpy()
    o = PatchMatchOptions(depth_min=sc["depth_min"], depth_max=sc["depth_max"], geom_consistency=False,
                          window_radius=C2["window_radius"], window_step=C2["window_step"],
                          num_samples=C2["num_samples"], num_iterations=C2["num_iterations"], gpu_index=str(local_rank))
    W, H, N = C2["width"], C2["height"], C2["num_src"]
    mpix = W * H / 1e6

    def barrier():
        torch.cuda.synchronize()
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident leg
    pm = PatchMatch(o, sc["problem"])
    pm.Run()
    for _ in range(max(args.warmup - 1, 0)):
        pm.RunOnly()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    t0 = time.time()
    dev_ms, sweep_ms, launches = 0.0, 0.0, 0
    pass_ms = [0.0, 0.0, 0.0]
    for _ in range(args.steps):
        pm.RunOnly()
        dev_ms += pm.last_run_ms()
        sweep_ms += pm.last_sweep_ms()
        launches += pm.last_num_launches()
        for k in range(3):
            pass_ms[k] += pm.last_pass_ms(k)
    barrier()
    wall_ms = (time.time() - t0) * 1e3
    clocks = sampler.stop()
    depth = pm.GetDepthMap()
    valid = depth > 0
    rel = np.abs(depth - sc["depth_gt"])[valid] / sc["depth_gt"][valid]
    quality = dict(valid_frac=float(valid.mean()), median_rel_depth_err=float(np.median(rel)))
    outputs = {} if args.dump_outputs and rank == 0 else None
    if outputs is not None:
        # the per-source maps (N x H x W) are kept at a fixed sample of pixels
        px = _fixed_sample(W * H)
        outputs.update(pm_depth=depth, pm_normal=pm.GetNormalMap(), pm_sel_prob=pm.GetSelProbMap().reshape(N, -1)[:, px],
                       pm_consistency_mask=pm.GetConsistencyMask().reshape(N, -1)[:, px])
    pm.close()

    # ---------------- end-to-end leg through the public API with host buffers
    def one_e2e():
        p = PatchMatch(o, sc["problem"])
        p.Run()                      # Check + create (H2D, prefilter, init) + run
        d = p.GetDepthMap()          # D2H
        n = p.GetNormalMap()         # D2H
        p.close()
        return d, n
    one_e2e()
    barrier()
    t0 = time.time()
    for _ in range(args.steps):
        one_e2e()
    barrier()
    e2e_ms = (time.time() - t0) * 1e3 / args.steps
    h2d = W * H + sum(im.bitmap.size for im in sc["images"][1:]) + 4 * N * 43 * 4
    d2h = 16 * W * H

    from colmap_b200.sharding import max_over_ranks
    ms_per_step = max_over_ranks(dev_ms / args.steps, "cuda")
    e2e_ms = max_over_ranks(e2e_ms, "cuda")
    wall_per_step = max_over_ranks(wall_ms / args.steps, "cuda")

    ba_sharded = None
    want_b5 = args.b5 == 1
    if distributed and not args.no_ba:
        try:
            ba_sharded = bench_ba_sharded(args.steps, args.warmup, rank, world, local_rank, with_b5=want_b5)
        except Exception as e:
            ba_sharded = {"error": repr(e)}
    c4 = None
    c4_images = args.c4_images if args.c4_images >= 0 else (C4["images_per_gpu_default"] * world if world == 8 else 0)
    if c4_images > 0:
        try:
            c4 = bench_c4(rank, world, local_rank, c4_images)
        except Exception as e:
            c4 = {"error": repr(e)}
    if rank == 0:
        n_sweeps = 4 * C2["num_iterations"]
        # one sweep = rand (+ msg on a second stream) + pixel + serial pass; pm_pixel_kernel (NCC of 3 of the 4 alternative
        # hypotheses, one warp per pixel, exact early-out) and pm_serial_kernel (column-serial) take about half each
        pixel_launch_ms = pass_ms[1] / args.steps / n_sweeps
        sweep_launch_ms = sweep_ms / args.steps / n_sweeps
        alg_bytes = (41 + 17 * N) * W * H            # SURVEY.md §8(d): per pixel per sweep, photometric (whole sweep)
        peak, peak_src = _peaks()
        achieved = alg_bytes / (sweep_launch_ms * 1e-3) / 1e9
        taps_per_sweep = W * H * 4 * N * 121          # 4 hypotheses x N images x 121 bilinear taps per pixel
        roofline = {"bound": "hbm", "kernel": "pm_pixel_kernel (+ pm_rand_kernel | pm_msg_kernel, pm_serial_kernel = one sweep)",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": _ncu_traffic("pm_sweep"), "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": sweep_launch_ms,
                    "pass_ms_per_sweep": {"rand_and_msg": pass_ms[0] / args.steps / n_sweeps, "pixel": pixel_launch_ms,
                                          "serial": pass_ms[2] / args.steps / n_sweeps},
                    "taps_per_s": taps_per_sweep / (sweep_launch_ms * 1e-3),
                    "note": "the faithful sweep is instruction-issue bound, not HBM bound (DESIGN.md §2): 177 algorithmic "
                            "bytes per pixel per sweep against up to 3872 bilinear taps (~45 instructions each; the exact "
                            "early-out of the pixel pass skips about half of them, taps_per_s counts all 3872); ncu: 67% "
                            "issue-slot utilisation in pm_pixel_kernel, 51-53% in the column-serial pm_serial_kernel"}
        line = {"metric": "patchmatch_mpixels_per_s", "value": world * mpix / (ms_per_step * 1e-3), "unit": "Mpixels/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": C2_WORKLOAD,
                           "l2": "inputs larger than L2: cost/sel-prob maps 3 x 66 MB + 66 MB source footprints vs 126 MB L2",
                           "parallelism": f"problems x{world} (no collective)"},
                "e2e": {"value": world * mpix / (e2e_ms * 1e-3), "unit": "Mpixels/s", "h2d_bytes_per_step": int(h2d),
                        "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms},
                "gpu_launches": int(launches), "wall_ms_per_step": wall_per_step, "clocks": clocks,
                "roofline": roofline, "quality": quality}
        if not args.no_cpu_baseline and world == 1:
            v, dt, sample = _oracle_pm_sample()
            line["cpu_baseline"] = {"value": v, "unit": "Mpixels/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": sample, "seconds": dt}
        if not args.no_ba and world == 1:
            try:
                line["ba"] = bench_ba(args.steps, args.warmup, peak, peak_src, not args.no_cpu_baseline, outputs)
            except Exception as e:  # the primary metric must still be reported
                line["ba"] = {"error": repr(e)}
        if ba_sharded is not None:
            line["ba"] = ba_sharded
        if want_b5 and not distributed and not args.no_ba:
            try:
                line.setdefault("ba", {})["b5"] = bench_b5(args.steps, 1, rank, world, local_rank, None, outputs)
            except Exception as e:
                line.setdefault("ba", {})["b5"] = {"error": repr(e)}
        if c4 is not None:
            line["c4"] = c4
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if distributed:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
