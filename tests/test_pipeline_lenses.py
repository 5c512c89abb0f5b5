"""CapturePipeline(lens="per_camera"): every camera's frames undistorted with its own calibration, end to end against the CPU
restatement of the reference run with each camera's own K / dist; the default "camera0" mode visibly differs on such a rig; the
per-camera drop-in call _find_dot(img, camera_number=c)."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from mocapv2_b200 import engine as E
from mocapv2_b200 import synth as S
from mocapv2_b200.pipeline import CapturePipeline, StepsInFlight
from oracle import restate as R

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# two lenses that bend differently enough that camera 0's model moves camera 1's centroids
TWO_LENSES = [(np.array([[620.0, 0, 321.0], [0, 618.0, 242.0], [0, 0, 1]]), np.array([-0.28, 0.09, 0.001, -0.001, 0.0])),
              (np.array([[575.0, 0, 334.0], [0, 580.0, 231.0], [0, 0, 1]]), np.array([0.06, 0.01, -0.002, 0.002, 0.0]))]


def scene(rig, n_sets, n_markers, seed, spread, min_sep=60.0, margin=40.0):
    rng = np.random.default_rng(seed)
    X0 = S.sample_markers(rig, n_markers, rng, spread=spread, min_sep_px=min_sep, margin=margin, tries=400)
    frames = []
    for _ in range(n_sets):
        X = X0 + rng.uniform(-0.01, 0.01, X0.shape)
        radii = rng.integers(14, 23, (len(rig["poses"]), len(X)))
        frames.append(S.render_frameset(rig, X, radii, rng))
    return np.stack(frames)


def two_lens_rig():
    return S.ring_rig(2, 640, 480, radius=3.0, lenses=TWO_LENSES)


def check(engine, rig, frames, n_markers, max_groups, **kw):
    """The per-camera pipeline step against the reference with each camera's own lens (tolerances of test_pipeline_e2e.py)."""
    pipe = CapturePipeline(engine, rig, max_blobs=64, obj_count=n_markers, max_groups=max_groups, lens="per_camera", **kw)
    res = pipe.step(torch.from_numpy(frames).to(engine.device))
    n_sets, C = frames.shape[:2]
    total = 0
    for s in range(n_sets):
        pts = [R.find_dot(frames[s, c], *S.camera_lens(rig, c)) for c in range(C)]
        for c in range(C):
            assert res.det.points(s * C + c) == pts[c], f"centroids of frame-set {s} camera {c}"
        trace = {}
        obj, ipa = R.correspond(pts, rig["poses"], rig["camera_params"], rig["Fs"], n_markers, trace=trace, max_cand=8, max_groups=max_groups)
        nv, no = int(res.corr.n_valid[s]), int(res.corr.n_obj[s])
        assert nv == (len(ipa) if ipa.size else 0) and no == (len(obj) if obj.size else 0)
        if nv:
            assert np.array_equal(res.corr.img[s, :nv].cpu().numpy(), ipa)
            got = res.corr.obj[s, :no].cpu().numpy()
            assert (np.abs(got - obj).max(axis=1) / np.linalg.norm(obj, axis=1)).max() < 1e-4
            e = res.corr.err[s, :nv].cpu().numpy()
            assert np.abs(np.sqrt(e) - np.sqrt(np.array(trace["errors"]))).max() < 1e-3
        total += no
    return pipe, res, total


def test_per_camera_lenses_two_cameras(engine):
    rig = two_lens_rig()
    assert rig["per_camera_lens"] and not np.allclose(rig["camera_params"][0]["intrinsic_matrix"], rig["camera_params"][1]["intrinsic_matrix"])
    frames = scene(rig, 2, 4, 501, 0.5)
    pipe, res, total = check(engine, rig, frames, 4, 64)
    assert total > 0 and pipe.lenses.n == 2
    # the default mode undistorts camera 1 with camera 0's lens: some centroid moves (a lens set that is ignored fails here)
    plain = CapturePipeline(engine, rig, max_blobs=64, obj_count=4, max_groups=64)
    base = plain.step(torch.from_numpy(frames).to(engine.device))
    assert any(base.det.points(f) != res.det.points(f) for f in range(4))
    assert all(base.det.points(f) == res.det.points(f) for f in (0, 2))          # camera 0: the same lens either way


def test_per_camera_steps_in_flight_equal_step(engine):
    rig = two_lens_rig()
    frames = scene(rig, 2, 4, 502, 0.5)
    batches = [torch.from_numpy(np.roll(frames, k, axis=0).copy()).to(engine.device) for k in range(2)]
    pipe = CapturePipeline(engine, rig, max_blobs=64, obj_count=4, max_groups=64, lens="per_camera")
    pipe.pipelined_min_frames = 1
    want = []
    for k in range(2):                                             # (a step's results live in the pipeline's buffers)
        w = pipe.step(batches[k])
        want.append((w.det.count.clone(), w.det.xy.clone(), w.corr.n_obj.clone(), w.corr.obj.clone()))
    flight = StepsInFlight(pipe, depth=2)
    assert all(l.lens == "per_camera" and l.lenses.tables.data_ptr() == pipe.lenses.tables.data_ptr() for l in flight.lanes)
    flight.fork()
    got = [flight.submit(batches[i % 2]) for i in range(4)]
    flight.join()
    if engine.device.type == "cuda":
        torch.cuda.synchronize()
    for i in (2, 3):
        r, w = got[i], want[i % 2]
        assert torch.equal(r.det.count, w[0]) and torch.equal(r.corr.n_obj, w[2])
        for f in range(len(w[0])):
            assert torch.equal(r.det.xy[f, :int(w[0][f])], w[1][f, :int(w[0][f])])
        for s in range(len(w[2])):
            assert torch.equal(r.corr.obj[s, :int(w[2][s])], w[3][s, :int(w[2][s])])


def test_default_rig_is_unchanged():
    """Rigs without lenses= project every camera with camera 0's lens, as before (the bench's workloads)."""
    rig = S.ring_rig(3, 640, 480, radius=3.0)
    assert "per_camera_lens" not in rig
    X = np.array([[0.05, 0.02, 0.0]]) + rig["centre"]
    K, D = rig["camera_params"][0]["intrinsic_matrix"], rig["camera_params"][0]["distortion_coef"]
    assert np.array_equal(S.marker_pixels(rig, X), np.stack([S.project_distorted(X, p, K, D) for p in rig["poses"]]))


@pytest.mark.gpu
def test_per_camera_lenses_config3(gpu_engine):
    rig = S.ring_rig(6, 1440, 1080, radius=6.0, lenses=S.per_camera_lenses(6, seed=603))
    frames = scene(rig, 3, 32, 603, 0.42, min_sep=70.0)
    assert check(gpu_engine, rig, frames, 32, 256)[2] > 0


@pytest.mark.gpu
def test_per_camera_lenses_config4_few_markers(gpu_engine):
    rig = S.ring_rig(16, 2048, 2048, radius=6.0, lenses=S.per_camera_lenses(16, seed=104))
    frames = scene(rig, 2, 12, 104, 0.9, min_sep=70.0)
    assert check(gpu_engine, rig, frames, 12, 4096)[2] > 0


# ---- two ranks over gloo on the emulation build, per-camera lenses ---------------------------------------------------------------
def _ring4():
    lenses = [(np.array([[600.0 + 15 * c, 0, 240.0 + 3 * c], [0, 600.0 - 10 * c, 180.0 - 2 * c], [0, 0, 1]]),
               np.array([-0.25 + 0.05 * c, 0.06, 0.0, 0.001 * c, 0.0])) for c in range(4)]
    rig = S.ring_rig(4, 480, 360, radius=3.0, lenses=lenses)
    return rig, scene(rig, 2, 3, 405, 0.12, min_sep=75.0, margin=36.0)


def _run(rank, world, port, out_dir):
    sys.path.insert(0, REPO)
    sys.path.insert(0, os.path.join(REPO, "tests", "emu"))
    import torch.distributed as dist
    import build_emu
    from emu_engine import EmuEngine
    if world > 1:
        dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    eng = EmuEngine(build_emu.build())
    rig, fr = _ring4()
    pipe = CapturePipeline(eng, rig, max_blobs=8, obj_count=4, max_groups=16, lens="per_camera")
    local = torch.from_numpy(fr[:, pipe.cam_begin:pipe.cam_begin + pipe.cams_local].copy())
    res = pipe.step(local)
    torch.save({"b": res.fs_begin, "e": res.fs_end, "obj": res.corr.obj, "n_obj": res.corr.n_obj, "img": res.corr.img,
                "n_valid": res.corr.n_valid, "err": res.corr.err, "count": res.det.count, "xy": res.det.xy,
                "n_lenses": pipe.lenses.n, "tables_bytes": pipe.lenses.tables.numel()},
               os.path.join(out_dir, f"rank{rank}_of{world}.pt"))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def test_two_ranks_per_camera_equal_one_rank(tmp_path):
    sys.path.insert(0, os.path.join(REPO, "tests", "emu"))
    import build_emu
    build_emu.build()
    out = str(tmp_path)
    _run(0, 1, 0, out)
    port = 35500 + os.getpid() % 2000
    mp.spawn(_run, args=(2, port, out), nprocs=2, join=True)
    one = torch.load(os.path.join(out, "rank0_of1.pt"))
    assert int(one["n_obj"].min()) >= 1 and one["n_lenses"] == 4
    for r in range(2):
        two = torch.load(os.path.join(out, f"rank{r}_of2.pt"))
        b, e = two["b"], two["e"]
        assert two["n_lenses"] == 2 and two["tables_bytes"] * 2 == one["tables_bytes"]       # only its own cameras' tables
        for k in ("n_valid", "n_obj", "img", "obj", "err"):
            assert torch.equal(two[k], one[k][b:e]), k
        # each rank detected its own cameras with their own lenses
        assert torch.equal(two["count"].view(2, 2), one["count"].view(2, 4)[:, 2 * r:2 * r + 2])
        mine = one["xy"].view(2, 4, *one["xy"].shape[1:])[:, 2 * r:2 * r + 2].reshape(two["xy"].shape)
        for f in range(4):
            c = int(two["count"][f])
            assert torch.equal(two["xy"][f, :c], mine[f, :c])


# ---- drop-in: _find_dot(img, camera_number=c) --------------------------------------------------------------------------------
def test_find_dot_with_camera_number(engine):
    from mocapv2_b200.lib import ImageOperations as IO
    rig = two_lens_rig()
    frames = scene(rig, 1, 4, 506, 0.5)[0]
    saved = IO.camera_params
    E.set_default_engine(engine)
    IO.camera_params = rig["camera_params"]
    try:
        img = frames[1]
        _, pts = IO._find_dot(img, camera_number=1)
        assert pts == R.find_dot(img, *TWO_LENSES[1]) and pts != [[None, None]]
        _, pts0 = IO._find_dot(img)
        assert pts0 == R.find_dot(img, *TWO_LENSES[0]) and pts0 != pts
        assert IO._find_dot(img, camera_number=0)[1] == pts0
        with pytest.raises(IndexError):
            IO._find_dot(img, camera_number=2)
    finally:
        IO.camera_params = saved
        E.set_default_engine(None)
