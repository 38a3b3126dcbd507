"""Host-side MVS workspace pieces (include/b200_mvs_workspace.h, colmap_b200/mvs_workspace.py): the reference's own
known answers (mvs/model_test.cc, mvs/consistency_graph_test.cc, mvs/mat_test.cc, util/misc_test.cc), parity with the
independent oracle (oracle/ws_oracle.py) on random models, file-format bytes, the patch-match.cfg reader, and the
controller schedule with an injected (CPU) runner."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ws_oracle  # noqa: E402

from colmap_b200.mvs_workspace import (ConsistencyGraph, Model, ModelPoint, PatchMatchController, WorkspaceError,  # noqa: E402
                                       read_depth_map, read_mat, read_normal_map, read_problems, write_mat,
                                       write_model_binary)
from colmap_b200.patch_match import PatchMatchOptions  # noqa: E402

K = [100, 0, 50, 0, 100, 50, 0, 0, 1]
I3 = [1, 0, 0, 0, 1, 0, 0, 0, 1]


def _model(Ts, points):
    m = Model()
    for i, T in enumerate(Ts):
        m.add_image(f"img{i}.jpg", 100, 100, K, I3, T)
    for xyz, track in points:
        m.points.append(ModelPoint(*[float(v) for v in xyz], list(track)))
    return m


# ---------------------------------------------------------------- reference known answers (mvs/model_test.cc:84-196)
def test_compute_shared_points_known_answer():
    m = _model([[0, 0, 0], [-1, 0, 0], [-2, 0, 0]], [((5, 0, 10), (0, 1)), ((6, 0, 10), (0, 1, 2))])
    s = m.ComputeSharedPoints()
    assert len(s) == 3
    assert s[0][1] == 2 and s[1][0] == 2 and s[0][2] == 1 and s[2][0] == 1 and s[1][2] == 1 and s[2][1] == 1


def test_compute_depth_ranges_known_answers():
    m = _model([[0, 0, 0]], [((0, 0, float(i)), (0,)) for i in range(1, 101)])
    (lo, hi), = m.ComputeDepthRanges()
    assert lo == np.float32(1.5) and hi == np.float32(125.0)       # 1 % / 99 % percentiles, stretched by 25 %
    (lo, hi), = _model([[0, 0, 0]], []).ComputeDepthRanges()
    assert lo == -1.0 and hi == -1.0


def test_compute_triangulation_angles_known_answer():
    m = _model([[0, 0, 0], [-1, 0, 0]], [((0.5, 0, 10), (0, 1))])
    a = m.ComputeTriangulationAngles(50)
    assert len(a) == 2
    assert abs(a[0][1] - 2.0 * np.arctan(0.5 / 10.0)) < 1e-5
    assert a[0][1] == a[1][0]


def test_get_max_overlapping_images_known_answer():
    pts = [((0.5, 0, 5.0 + i), (0, 1)) for i in range(10)] + [((1.0, 0, 10.0), (0, 2))]
    m = _model([[0, 0, 0], [-1, 0, 0], [-2, 0, 0]], pts)
    o = m.GetMaxOverlappingImages(2, 0.0)
    assert len(o) == 3 and o[0] and o[0][0] == 1


def test_image_name_lookup():
    m = _model([[0, 0, 0]], [])
    assert m.GetImageIdx(m.GetImageName(0)) == 0
    with pytest.raises(WorkspaceError):
        m.GetImageIdx("nonexistent")
    with pytest.raises(WorkspaceError):
        m.GetImageName(-1)
    with pytest.raises(WorkspaceError):
        m.GetImageName(1)


# ---------------------------------------------------------------- consistency graph (mvs/consistency_graph_test.cc:40-138)
def test_consistency_graph_known_answers(tmp_path):
    g = ConsistencyGraph(2, 2, [])
    assert all(len(g.GetImageIdxs(r, c)) == 0 for r in range(2) for c in range(2)) and g.GetNumBytes() == 16
    g = ConsistencyGraph(2, 1, [0, 0, 3, 5, 7, 33])
    assert list(g.GetImageIdxs(0, 0)) == [5, 7, 33] and len(g.GetImageIdxs(0, 1)) == 0 and g.GetNumBytes() == 32
    g = ConsistencyGraph(2, 1, [0, 0, 0])
    assert len(g.GetImageIdxs(0, 0)) == 0 and len(g.GetImageIdxs(0, 1)) == 0 and g.GetNumBytes() == 20
    g = ConsistencyGraph(1, 2, [0, 0, 3, 5, 7, 33, 0, 1, 1, 100])
    assert list(g.GetImageIdxs(0, 0)) == [5, 7, 33] and list(g.GetImageIdxs(1, 0)) == [100] and g.GetNumBytes() == 48
    assert ConsistencyGraph().GetNumBytes() == 0
    path = str(tmp_path / "consistency_graph.bin")
    g.Write(path)
    assert open(path, "rb").read() == ws_oracle.graph_bytes(1, 2, [0, 0, 3, 5, 7, 33, 0, 1, 1, 100])
    h = ConsistencyGraph()
    h.Read(path)
    assert h.GetNumBytes() == g.GetNumBytes() and list(h.GetImageIdxs(0, 0)) == [5, 7, 33] and list(h.GetImageIdxs(1, 0)) == [100]
    for bad in ([0, 0], [0, 0, -1], [2, 0, 0], [0, 0, 3, 1]):      # truncated / negative count / outside / overrun
        with pytest.raises(WorkspaceError):
            ConsistencyGraph(1, 2, bad)


# ---------------------------------------------------------------- map files (mvs/mat.cc:41-66)
def test_mat_files_round_trip_and_bytes(tmp_path):
    rng = np.random.default_rng(0)
    depth = rng.random((7, 5)).astype(np.float32)
    normal = rng.random((3, 7, 5)).astype(np.float32)
    pd, pn = str(tmp_path / "d.bin"), str(tmp_path / "n.bin")
    write_mat(pd, depth); write_mat(pn, normal)
    assert open(pd, "rb").read() == ws_oracle.mat_bytes(depth)        # "5&7&1&" + row-major floats
    assert open(pn, "rb").read() == ws_oracle.mat_bytes(normal)       # slice-major
    assert np.array_equal(read_depth_map(pd), depth) and np.array_equal(read_normal_map(pn), normal)
    assert read_mat(pn).shape == (3, 7, 5)
    with pytest.raises(WorkspaceError):
        read_depth_map(pn)
    with pytest.raises(WorkspaceError):
        read_mat(str(tmp_path / "missing.bin"))
    open(str(tmp_path / "t.bin"), "wb").write(b"5&7&1&" + b"\x00" * 10)
    with pytest.raises(WorkspaceError):
        read_mat(str(tmp_path / "t.bin"))


# ---------------------------------------------------------------- parity with the oracle on random models
def _random_model(seed, n_img=9, n_pts=400):
    rng = np.random.default_rng(seed)
    m, imgs = Model(), []
    for i in range(n_img):
        a = rng.uniform(-0.3, 0.3)
        R = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]], np.float32)
        T = np.array([rng.uniform(-2, 2), rng.uniform(-0.3, 0.3), rng.uniform(-0.5, 0.5)], np.float32)
        m.add_image(f"im_{i:03d}.png", 64, 48, K, R, T)
        imgs.append((R, T))
    pts = []
    for _ in range(n_pts):
        xyz = np.array([rng.uniform(-3, 3), rng.uniform(-2, 2), rng.uniform(4, 12)], np.float32)
        track = list(rng.choice(n_img, size=int(rng.integers(1, 6)), replace=True))     # duplicates allowed, like real tracks
        pts.append((xyz, [int(t) for t in track]))
        m.points.append(ModelPoint(float(xyz[0]), float(xyz[1]), float(xyz[2]), [int(t) for t in track]))
    return m, imgs, pts


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_model_statistics_match_the_oracle(seed):
    m, imgs, pts = _random_model(seed)
    assert m.ComputeSharedPoints() == ws_oracle.shared_points(len(imgs), pts)
    got, ref = m.ComputeDepthRanges(), ws_oracle.depth_ranges(imgs, pts)
    assert np.allclose(got, ref, rtol=2e-7, atol=0)
    for p in (0.0, 50.0, 75.0, 100.0):
        got, ref = m.ComputeTriangulationAngles(p), ws_oracle.triangulation_angles(imgs, pts, p)
        assert [sorted(d) for d in got] == [sorted(d) for d in ref]
        for dg, dr in zip(got, ref):
            assert np.allclose([dg[k] for k in sorted(dg)], [dr[k] for k in sorted(dr)], rtol=1e-6, atol=1e-7)
    for num, ang in ((3, 0.0), (20, 2.0), (1, 5.0)):
        assert m.GetMaxOverlappingImages(num, ang) == ws_oracle.max_overlapping_images(imgs, pts, num, ang)


# ---------------------------------------------------------------- patch-match.cfg (patch_match.cc:240-372, util/misc_test.cc:58-84)
def test_read_problems_all_auto_and_lists():
    m, imgs, pts = _random_model(3)
    names = [m.GetImageName(i) for i in range(len(imgs))]
    cfg = "\n".join([
        "# comment line", "", f"  {names[0]}  ", "__all__",
        names[1], "__auto__, 3",
        names[2], f"{names[3]}, {names[4]} ;{names[5]},,",
        "# another comment", names[6], "__auto__, 0",          # no source images -> dropped
    ]) + "\n"
    pr = read_problems(cfg, m, 1.0)
    assert pr[0] == (0, [i for i in range(len(imgs)) if i != 0])
    assert pr[1] == (1, ws_oracle.max_overlapping_images(imgs, pts, 3, 1.0)[1])
    assert pr[2] == (2, [3, 4, 5])
    assert len(pr) == 3
    with pytest.raises(WorkspaceError):
        read_problems("unknown.png\n__all__\n", m, 1.0)
    with pytest.raises(WorkspaceError):
        read_problems(f"{names[0]}\nunknown.png\n", m, 1.0)
    assert read_problems("", m, 1.0) == []
    assert read_problems(f"{names[0]}\n", m, 1.0) == []        # a reference line without a source line


# ---------------------------------------------------------------- COLMAP sparse model reader + controller schedule
def _write_workspace(tmp, n_img=4, w=48, h=36):
    from PIL import Image as PILImage
    rng = np.random.default_rng(5)
    cams = {1: dict(model_id=1, width=w, height=h, params=[40.0, 41.0, w / 2, h / 2])}
    images, points = {}, {}
    os.makedirs(os.path.join(tmp, "images"), exist_ok=True)
    for i in range(n_img):
        name = f"view{i}.png"
        images[i + 1] = dict(qvec=[1.0, 0.0, 0.0, 0.0], tvec=[-0.2 * i, 0.0, 0.0], camera_id=1, name=name)
        PILImage.fromarray(rng.integers(0, 255, (h, w), dtype=np.uint8)).save(os.path.join(tmp, "images", name))
    for p in range(60):
        xyz = [rng.uniform(-1, 1), rng.uniform(-1, 1), rng.uniform(4, 6)]
        points[p + 1] = dict(xyz=xyz, track=[(i + 1, p) for i in range(n_img)])
    write_model_binary(os.path.join(tmp, "sparse"), cams, images, points)
    os.makedirs(os.path.join(tmp, "stereo"), exist_ok=True)
    with open(os.path.join(tmp, "stereo", "patch-match.cfg"), "w") as f:
        for i in range(n_img):
            f.write(f"view{i}.png\n__auto__, 2\n")
    return cams, images, points


def test_read_from_colmap_and_controller_schedule(tmp_path):
    tmp = str(tmp_path)
    cams, images, points = _write_workspace(tmp)
    m = Model.ReadFromCOLMAP(tmp)
    assert len(m.images) == 4 and len(m.points) == 60 and m.GetImageName(2) == "view2.png"
    assert np.allclose(m.images[1].K, [[40, 0, 24], [0, 41, 18], [0, 0, 1]]) and np.allclose(m.images[3].T, [-0.6, 0, 0])
    assert all(sorted(p.track) == [0, 1, 2, 3] for p in m.points)

    calls = []

    def runner(o, problem):            # CPU stand-in for the sweep: records the schedule, returns recognisable maps
        hh, ww = problem.images[0].bitmap.shape
        calls.append((o.geom_consistency, o.filter, len(problem.src_image_idxs), o.depth_min, o.depth_max,
                      problem.depth_maps is not None))
        tag = 2.0 if o.geom_consistency else 1.0
        out = dict(depth=np.full((hh, ww), tag, np.float32), normal=np.full((3, hh, ww), tag, np.float32))
        if o.write_consistency_graph:
            out["consistency"] = np.array([0, 0, 2, 1, 2], np.int32)   # pixel (col 0, row 0): local sources 1 and 2
        return out

    o = PatchMatchOptions(geom_consistency=True, write_consistency_graph=True)
    c = PatchMatchController(o, tmp)
    assert c.Run(runner) == 8                                   # 4 photometric + 4 geometric problems
    assert [x[0] for x in calls] == [False] * 4 + [True] * 4    # all photometric problems first
    assert all(x[1] is False for x in calls[:4]) and all(x[1] is True for x in calls[4:])   # first phase without filter
    assert all(x[2] == 2 for x in calls) and all(x[5] for x in calls[4:]) and not any(x[5] for x in calls[:4])
    lo, hi = m.ComputeDepthRanges()[0]
    assert calls[0][3] == lo and calls[0][4] == hi             # depth range from the sparse model
    d = read_depth_map(os.path.join(tmp, "stereo", "depth_maps", "view0.png.geometric.bin"))
    n = read_normal_map(os.path.join(tmp, "stereo", "normal_maps", "view0.png.photometric.bin"))
    assert d.shape == (36, 48) and np.all(d == 2.0) and n.shape == (3, 36, 48) and np.all(n == 1.0)
    g = ConsistencyGraph()
    g.Read(os.path.join(tmp, "stereo", "consistency_graphs", "view0.png.geometric.bin"))
    srcs = c.problems[0][1]
    assert list(g.GetImageIdxs(0, 0)) == srcs                   # local source indices mapped back to model indices
    assert PatchMatchController(o, tmp).Run(runner) == 0        # existing outputs are skipped


def test_library_exports_every_declared_workspace_symbol():
    import re
    from colmap_b200 import load_library
    lib = load_library()
    hdr = open(os.path.join(ROOT, "include", "b200_mvs_workspace.h")).read()
    names = set(re.findall(r"\b(b200ws_[a-z_0-9]+)\s*\(", hdr))
    assert len(names) >= 12
    for n in names:
        assert hasattr(lib, n), n


# ---------------------------------------------------------------- two ranks (gloo) share one workspace
def _controller_worker(rank, world, port, tmp, q):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from colmap_b200.mvs_workspace import PatchMatchController as C
    from colmap_b200.patch_match import PatchMatchOptions as O
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    seen = []

    def runner(o, problem):
        hh, ww = problem.images[0].bitmap.shape
        if o.geom_consistency:      # the photometric maps of ALL source images must be on disk by now, whoever wrote them
            assert problem.depth_maps is not None and all(float(d[0, 0]) >= 100.0 for d in problem.depth_maps)
        seen.append(o.geom_consistency)
        v = float(np.float32(100 + rank)) if not o.geom_consistency else float(np.float32(200 + rank))
        return dict(depth=np.full((hh, ww), v, np.float32), normal=np.full((3, hh, ww), v, np.float32))

    n = C(O(geom_consistency=True), tmp).Run(runner, rank=rank, world=world)
    dist.destroy_process_group()
    q.put((rank, n, seen))


def test_controller_two_ranks_share_a_workspace(tmp_path):
    import socket
    import torch.multiprocessing as mp
    tmp = str(tmp_path)
    _write_workspace(tmp, n_img=5)
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_controller_worker, args=(r, 2, port, tmp, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=180) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert res[0][1] + res[1][1] == 10 and {res[0][1], res[1][1]} == {4, 6}          # 5 photometric + 5 geometric, split 3 / 2
    for _, n, seen in res:
        assert seen == [False] * (n // 2) + [True] * (n // 2)                        # phase order on every rank
    for i in range(5):
        d = read_depth_map(os.path.join(tmp, "stereo", "depth_maps", f"view{i}.png.geometric.bin"))
        assert d.shape == (36, 48) and float(d[0, 0]) in (200.0, 201.0)


def test_controller_thread_pool_follows_gpu_index_list(tmp_path):
    """`gpu_index = "0,0"`: two worker threads on device 0 (patch_match.cc:375-384 + the thread pool of :176-205); every
    problem carries the device of its worker; the photometric phase still completes before the geometric one starts."""
    import threading
    import time
    tmp = str(tmp_path)
    _write_workspace(tmp, n_img=6)
    lock, state = threading.Lock(), dict(active=0, peak=0, log=[])

    def runner(o, problem):
        with lock:
            state["active"] += 1; state["peak"] = max(state["peak"], state["active"])
            state["log"].append((o.geom_consistency, o.gpu_index, threading.get_ident()))
        time.sleep(0.05)
        with lock:
            state["active"] -= 1
        hh, ww = problem.images[0].bitmap.shape
        return dict(depth=np.ones((hh, ww), np.float32), normal=np.ones((3, hh, ww), np.float32))

    c = PatchMatchController(PatchMatchOptions(geom_consistency=True, gpu_index="0,0"), tmp)
    assert c.ReadGpuIndices() == [0, 0]
    assert c.Run(runner) == 12
    assert state["peak"] == 2
    assert [g for g, _, _ in state["log"]] == [False] * 6 + [True] * 6
    assert {i for _, i, _ in state["log"]} == {"0"}
    assert len({t for _, _, t in state["log"][:6]}) == 2
    c2 = PatchMatchController(PatchMatchOptions(gpu_index="-1"), tmp)
    assert c2.ReadGpuIndices(num_devices=4) == [0, 1, 2, 3] and PatchMatchController(PatchMatchOptions(gpu_index="1, 3"), tmp).ReadGpuIndices() == [1, 3]


def test_run_workspace_fails_loudly_without_a_workspace_or_a_gpu(tmp_path):
    """b200pm_run_workspace (the controller in C++) has no CPU path: a missing sparse model, a corrupt one and - with a valid
    workspace - the absence of a CUDA device are all reported as errors, nothing is written."""
    from colmap_b200.mvs_workspace import WorkspaceError, run_workspace
    from colmap_b200.patch_match import PatchMatchOptions
    o = PatchMatchOptions()
    with pytest.raises(WorkspaceError, match="cannot open"):
        run_workspace(o, str(tmp_path / "nowhere"))
    ws = tmp_path / "ws"
    (ws / "sparse").mkdir(parents=True)
    (ws / "sparse" / "cameras.bin").write_bytes(np.array([1], np.uint64).tobytes() + b"\x01\x00")          # count 1, then truncated
    with pytest.raises(WorkspaceError, match="truncated"):
        run_workspace(o, str(ws))
    # a structurally valid (tiny) workspace: without a device the call must refuse, not fall back.  The call runs in a
    # child process that sees no CUDA device, so that this holds on a machine with a GPU as well.
    import re
    import struct
    import subprocess
    cam = struct.pack("<Q", 1) + struct.pack("<IiQQ", 1, 1, 64, 48) + struct.pack("<4d", 50.0, 50.0, 32.0, 24.0)
    (ws / "sparse" / "cameras.bin").write_bytes(cam)
    imgs = struct.pack("<Q", 2)
    for i in (1, 2):
        imgs += struct.pack("<I", i) + struct.pack("<4d", 1.0, 0.0, 0.0, 0.0) + struct.pack("<3d", 0.1 * i, 0.0, 0.0) + struct.pack("<I", 1)
        imgs += f"im{i}.pgm".encode() + b"\x00" + struct.pack("<Q", 0)
    (ws / "sparse" / "images.bin").write_bytes(imgs)
    pts = struct.pack("<Q", 1) + struct.pack("<Q", 1) + struct.pack("<3d", 0.0, 0.0, 3.0) + bytes([1, 2, 3]) + struct.pack("<d", 0.5)
    pts += struct.pack("<Q", 2) + struct.pack("<II", 1, 0) + struct.pack("<II", 2, 0)
    (ws / "sparse" / "points3D.bin").write_bytes(pts)
    (ws / "stereo").mkdir()
    (ws / "stereo" / "patch-match.cfg").write_text("im1.pgm\n__all__\nim2.pgm\n__all__\n")
    (ws / "images").mkdir()
    for i in (1, 2):
        (ws / "images" / f"im{i}.pgm").write_bytes(b"P5\n64 48\n255\n" + bytes(64 * 48))
    child = ("import sys\n"
             "from colmap_b200.mvs_workspace import WorkspaceError, run_workspace\n"
             "from colmap_b200.patch_match import PatchMatchOptions\n"
             "try:\n"
             "    run_workspace(PatchMatchOptions(), sys.argv[1], gpu_indices=[0])\n"
             "except WorkspaceError as e:\n"
             "    print(e)\n"
             "    sys.exit(3)\n")
    r = subprocess.run([sys.executable, "-c", child, str(ws)], capture_output=True, text=True, timeout=300, cwd=ROOT,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 3, r.stdout + r.stderr
    assert re.search("CUDA|device|GPU", r.stdout), r.stdout
    assert not (ws / "stereo" / "depth_maps").exists() or not any((ws / "stereo" / "depth_maps").iterdir())
