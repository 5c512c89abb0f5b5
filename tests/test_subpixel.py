"""Sub-pixel centroids: the float32 nearest to cv.moments' m10/m00, m01/m00 in place of the reference's int() (lib/ImageOperations.py:
59-62), from the detection kernels through the correspondence, the multi-rank pipeline and the drop-in functions.

Each mode is checked against its own oracle: int(q) and float32(q) of the same FP64 quotient q (trunc(float32(q)) may differ from
trunc(q) when q lies within half a float32 ulp below an integer, so one mode is never derived from the other).  Contours, filter,
order, counts and flags are those of the integer mode.  The `engine` tests run on the CPU emulation build and on the GPU.
"""
import copy
import json
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from mocapv2_b200 import engine as E
from mocapv2_b200 import synth as S
from mocapv2_b200.lib import Helpers as H
from mocapv2_b200.lib import ImageOperations as IO
from oracle import restate as R
from util import GOLDEN, K, D

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALL = ("bits", "labels", "blob_sums", "contours")
REL_XYZ = 1e-4        # the tolerances of test_geometry_parity.py
TOL_PX = 1e-3


def dev(engine, a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(engine.device)


def is_gpu(engine):
    return engine.device.type == "cuda"


# ---- the float32 oracle -----------------------------------------------------------------------------------------------------
def centroid_f32(a00, a10, a01):
    """float32(m10/m00), float32(m01/m00) with cv.moments' scaling (oracle.restate.centroid without the int()); None if m00 == 0."""
    if a00 == 0:
        return None
    if a00 > 0:
        m00, m10, m01 = a00 * 0.5, a10 * 0.16666666666666666, a01 * 0.16666666666666666
    else:
        m00, m10, m01 = a00 * -0.5, a10 * -0.16666666666666666, a01 * -0.16666666666666666
    return [float(np.float32(m10 / m00)), float(np.float32(m01 / m00))]


def oracle_points(binimg, min_area=R.MIN_AREA, min_circ=R.MIN_CIRC, subpixel=False):
    """Kept centroids of a filtered binary image in the reference's output order: [[int, int], ...] or [[float, float], ...]."""
    contours, _ = R.find_contours(binimg)
    pts = []
    for c in contours:
        a00, a10, a01, per = R.contour_stats(c)
        area = abs(a00) * 0.5
        if a00 != 0 and per and 4 * np.pi * area / (per * per) > min_circ and area > min_area:
            pts.append(centroid_f32(a00, a10, a01) if subpixel else R.centroid(a00, a10, a01))
    return pts


def check_modes(res_int, res_sub, i, binimg, min_area=R.MIN_AREA):
    """Frame i of an int call and a sub-pixel call on the same frames: each equals its oracle; counts and flags agree."""
    want_i = oracle_points(binimg, min_area)
    want_f = oracle_points(binimg, min_area, subpixel=True)
    assert res_int.xy.dtype == torch.int32 and res_sub.xy.dtype == torch.float32
    assert int(res_int.count[i]) == int(res_sub.count[i]) == len(want_f)
    assert int(res_int.flags[i]) == int(res_sub.flags[i])
    assert res_int.points(i) == (want_i if want_i else [[None, None]])
    n = len(want_f)
    got = res_sub.xy[i, :n].cpu().numpy()
    assert np.array_equal(got, np.array(want_f, dtype=np.float32).reshape(-1, 2)), "sub-pixel centroids differ from the oracle"
    pts = res_sub.points(i)
    assert pts == (want_f if want_f else [[None, None]]) and all(type(v) is float for p in pts if p[0] is not None for v in p)


# ---- scenes ---------------------------------------------------------------------------------------------------------------------
def fuzz_scenes(seed, n, H, W):
    """fuzz_detect-style frames: discs, rings (hole borders), bars, blobs cut by the frame edges, flat ellipses."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[:H, :W]
    out = []
    for _ in range(n):
        img = rng.integers(0, 40, (H, W)).astype(np.uint8)
        for k in range(9):
            cx, cy = int(rng.integers(0, W)), int(rng.integers(0, H))
            if k < 2:                                                      # on a frame edge
                cx, cy = [(0, cy), (W - 1, cy), (cx, 0), (cx, H - 1)][int(rng.integers(0, 4))]
            kind = k % 4
            if kind == 0:
                r = int(rng.integers(5, 22)); img[(xx - cx) ** 2 + (yy - cy) ** 2 <= r * r] = 255
            elif kind == 1:
                r = int(rng.integers(8, 24)); d2 = (xx - cx) ** 2 + (yy - cy) ** 2
                img[(d2 <= r * r) & (d2 >= (r // 2) ** 2)] = 255
            elif kind == 2:
                w, h = int(rng.integers(4, 40)), int(rng.integers(4, 30)); img[cy:cy + h, cx:cx + w] = 255
            else:
                ax, ay = float(rng.uniform(10, 40)), float(rng.uniform(4, 14))
                img[((xx - cx) / ax) ** 2 + ((yy - cy) / ay) ** 2 <= 1.0] = 255
        out.append(img)
    return np.stack(out)


LENSES = [
    (np.array([[300.0, 0, 112.0], [0, 300.0, 80.0], [0, 0, 1]]), np.array([-0.20, 0.01, 0.001, -0.001, 0.0])),
    (np.eye(3), np.zeros(5)),
]


# ---- detection ------------------------------------------------------------------------------------------------------------------
def test_shapes_golden_both_modes(engine):
    """Rings, holes, nested and edge-touching blobs at odd frame sizes: one-shot call and parity-output call (general path)."""
    z = np.load(os.path.join(GOLDEN, "shapes.npz"))
    for i in ((0, 1, 3, 4, 5) if not is_gpu(engine) else range(6)):
        img = z[f"frame_{i}"]
        _, binimg = R.filter_frame(img, K, D)
        for outputs in ((), ALL):
            a = engine.detect(dev(engine, img[None]), K, D, outputs=outputs)
            b = engine.detect(dev(engine, img[None]), K, D, outputs=outputs, subpixel=True)
            check_modes(a, b, 0, binimg)
            if outputs:
                assert int(b.flags[0]) & 64                                 # parity outputs: the general path finished the frame
                assert torch.equal(a.extras["contours"], b.extras["contours"])


@pytest.mark.parametrize("outputs", [(), ("contours",), ALL])
def test_random_scenes_with_a_lens_set(engine, outputs):
    """Random scenes, two lenses mixed frame by frame: one-shot call (cluster path, or the general path with the parity outputs)."""
    H, W = 160, 224
    n = 8 if is_gpu(engine) else 4
    frames = fuzz_scenes(7, n, H, W)
    order = [i % 2 for i in range(n)]
    ls = engine.lens_set([{"intrinsic_matrix": k.tolist(), "distortion_coef": d.tolist()} for k, d in LENSES], H, W)
    a = engine.detect(dev(engine, frames), lenses=ls, frame_lens=order, min_area=30.0, outputs=outputs)
    b = engine.detect(dev(engine, frames), lenses=ls, frame_lens=order, min_area=30.0, outputs=outputs, subpixel=True)
    for i in range(n):
        _, binimg = R.filter_frame(frames[i], *LENSES[order[i]])
        check_modes(a, b, i, binimg, 30.0)


def test_overlapped_call_both_modes(engine):
    """The overlapped call (chunks, the general path for the frames the cluster units hand over) equals the one-shot call in either mode
    and leaves the integer results as they were."""
    H, W = 160, 224
    n = 8 if is_gpu(engine) else 5
    frames = fuzz_scenes(11, n, H, W)
    one_i = engine.detect(dev(engine, frames), K, D, min_area=30.0)
    one_f = engine.detect(dev(engine, frames), K, D, min_area=30.0, subpixel=True)
    over_i = engine.detect_pipelined(dev(engine, frames), K, D, min_area=30.0, chunk_frames=2, outputs=("contours",))
    over_f = engine.detect_pipelined(dev(engine, frames), K, D, min_area=30.0, chunk_frames=2, outputs=("contours",), subpixel=True)
    for i in range(n):
        _, binimg = R.filter_frame(frames[i], K, D)
        check_modes(over_i, over_f, i, binimg, 30.0)
        m = int(one_f.count[i])
        assert torch.equal(one_f.xy[i, :m], over_f.xy[i, :m]) and torch.equal(one_i.xy[i, :m], over_i.xy[i, :m])
    assert torch.equal(over_i.extras["contours"], over_f.extras["contours"])


def test_out_buffers_are_checked_for_the_centroid_format(engine):
    frames = dev(engine, np.zeros((1, 64, 96), np.uint8))
    res = engine.detect(frames, K, D)
    with pytest.raises(ValueError):
        engine.detect(frames, K, D, out=res, subpixel=True)
    res = engine.detect(frames, K, D, subpixel=True)
    with pytest.raises(ValueError):
        engine.detect_pipelined(frames, K, D, out=res)


def test_float32_oracle_equals_live_cv2_moments():
    cv2 = pytest.importorskip("cv2")
    z = np.load(os.path.join(GOLDEN, "shapes.npz"))
    n = 0
    for i in range(6):
        _, binimg = R.filter_frame(z[f"frame_{i}"], K, D)
        contours, _ = R.find_contours(binimg)
        for c in contours:
            m = cv2.moments(c.reshape(-1, 1, 2).astype(np.int32))
            a00, a10, a01, _ = R.contour_stats(c)
            if m["m00"] == 0:
                assert centroid_f32(a00, a10, a01) is None
                continue
            assert centroid_f32(a00, a10, a01) == [float(np.float32(m["m10"] / m["m00"])), float(np.float32(m["m01"] / m["m00"]))]
            n += 1
    assert n > 10


# ---- correspondence ---------------------------------------------------------------------------------------------------------------
def subpixel_lists(rig, rng, n_markers=5, decoys=3):
    """Per-camera float32 centroid lists: ideal projections plus in-band decoys, shuffled; Python floats holding float32 values."""
    X = S.config_markers("c3", rig, rng)[:n_markers]
    uv = S.marker_pixels(rig, X)
    pts = []
    for c in range(len(rig["poses"])):
        p = [list(q) for q in uv[c]]
        for _ in range(decoys):
            u, v = uv[c][rng.integers(0, n_markers)]
            p.append([u + rng.uniform(-6, 6), v + rng.uniform(-6, 6)])
        order = rng.permutation(len(p))
        pts.append([[float(np.float32(p[k][0])), float(np.float32(p[k][1]))] for k in order])
    return pts


@pytest.mark.parametrize("blocked", [False, True])
@pytest.mark.parametrize("fp64", [True, False])
def test_correspondence_on_float32_lists(engine, fp64, blocked):
    rig = S.config_rig("c3")
    rng = np.random.default_rng(23)
    cams = engine.cameras(rig["poses"], rig["camera_params"])
    Fs = dev(engine, np.array(rig["Fs"], dtype=np.float64))
    for case in range(4 if is_gpu(engine) else 2):
        pts = subpixel_lists(rig, rng)
        obj_count = int(rng.integers(0, 6))
        trace = {}
        o, ipa = R.correspond(pts, rig["poses"], rig["camera_params"], rig["Fs"], obj_count, trace=trace)
        mp_ = max(len(p) for p in pts)
        xy = np.zeros((1, 6, mp_, 2), np.float32)
        cnt = np.array([[len(p) for p in pts]], np.int32)
        for c, p in enumerate(pts):
            xy[0, c, :len(p)] = np.array(p, np.float32)
        if blocked:                                                     # two source ranks of three cameras: [B, S, C/B, max_pts, 2]
            xy, cnt = xy.reshape(2, 1, 3, mp_, 2), cnt.reshape(2, 1, 3)
        r = engine.correspond(dev(engine, xy), dev(engine, cnt), Fs, cams, obj_count=obj_count, fp64=fp64, want_cand=True)
        assert r.img.dtype == torch.float32
        nv, no = int(r.n_valid[0]), int(r.n_obj[0])
        assert nv == len(ipa) > 0 and no == len(o)
        cand = r.cand[0].cpu().numpy()
        for j, per_cam in enumerate(trace["candidates"]):
            for i in range(1, 6):
                assert [int(k) for k in cand[j, i] if k >= 0] == [k for k, _ in per_cam[i]][:8]
        assert np.array_equal(r.img[0, :nv].cpu().numpy().astype(np.float64), ipa)
        assert float((np.abs(r.obj[0, :no].cpu().numpy() - o).max(axis=1) / np.linalg.norm(o, axis=1)).max()) < (1e-10 if fp64 else REL_XYZ)
        got_e = r.err[0, :nv].cpu().numpy()
        assert np.abs(np.sqrt(got_e) - np.sqrt(np.array(trace["errors"]))).max() < (1e-9 if fp64 else TOL_PX)
        assert int(r.flags[0]) & 3 == 0


def test_correspondence_rejects_other_dtypes(engine):
    rig = S.config_rig("c1")
    cams = engine.cameras(rig["poses"], rig["camera_params"])
    Fs = dev(engine, np.array(rig["Fs"], dtype=np.float64))
    cnt = dev(engine, np.ones((1, 2), np.int32))
    with pytest.raises(ValueError):
        engine.correspond(dev(engine, np.zeros((1, 2, 1, 2), np.float64)), cnt, Fs, cams)
    res = engine.correspond(dev(engine, np.zeros((1, 2, 1, 2), np.int32)), cnt, Fs, cams)
    with pytest.raises(ValueError):
        engine.correspond(dev(engine, np.zeros((1, 2, 1, 2), np.float32)), cnt, Fs, cams, out=res)


# ---- drop-in ----------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def dropin(engine):
    E.set_default_engine(engine)
    saved = (H.camera_params, H.Fs, IO.camera_params, H.precision)
    H.camera_params = np.array(S.shipped_camera_params(2))
    H.Fs = [S.SHIPPED_F, S.SHIPPED_F]
    IO.camera_params = S.shipped_camera_params(2)
    yield engine
    H.camera_params, H.Fs, IO.camera_params, H.precision = saved
    E.set_default_engine(None)


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_dropin_subpixel_find_dot_and_matching(dropin, precision):
    H.precision = precision
    z = np.load(os.path.join(GOLDEN, "c1_frames.npz"))
    rig = S.config_rig("c1")
    pts = []
    for c in range(2):
        img = z["frames"][0, c]
        _, p = IO._find_dot(img, subpixel=True)
        _, binimg = R.filter_frame(img, K, D)
        assert p == oracle_points(binimg, subpixel=True) and all(type(v) is float for q in p for v in q)
        _, pi = IO._find_dot(img)
        assert pi == oracle_points(binimg) and all(type(v) is int for q in pi for v in q)
        pts.append(p)
    o_ref, ipa_ref = R.correspond(pts, rig["poses"], rig["camera_params"], rig["Fs"], 4)
    arg = copy.deepcopy(pts)
    arg[0].append([None, None])
    obj, ipa = H.find_point_correspondance_and_object_points(arg, S.shipped_poses(), 4)
    assert [None, None] not in arg[0]
    assert ipa.dtype == np.float64 and np.array_equal(ipa, ipa_ref)
    assert obj.shape == o_ref.shape and len(obj) > 0
    assert (np.abs(obj - o_ref).max(axis=1) / np.linalg.norm(o_ref, axis=1)).max() < (1e-11 if precision == "fp64" else REL_XYZ)


def test_dropin_point_forms(dropin):
    poses = S.shipped_poses()
    meta = json.load(open(os.path.join(GOLDEN, "c1.json")))
    rec = meta["corr"][0]
    _, ipa = H.find_point_correspondance_and_object_points(copy.deepcopy(rec["points"]), poses, 4)
    assert ipa.dtype == np.int64 and np.array_equal(ipa, np.array(rec["image_points_all"]))
    as_float = [[[float(x), float(y)] for x, y in cam] for cam in rec["points"]]    # integer-valued floats: the int path
    _, ipa = H.find_point_correspondance_and_object_points(as_float, poses, 4)
    assert ipa.dtype == np.int64
    bad = copy.deepcopy(rec["points"])
    bad[1][0] = [bad[1][0][0] + 0.1, bad[1][0][1]]                                  # 0.1 is no float32 value
    with pytest.raises(ValueError, match="float32"):
        H.find_point_correspondance_and_object_points(bad, poses, 4)


# ---- pipeline ---------------------------------------------------------------------------------------------------------------------
def _ring4_scene():
    rig = S.ring_rig(4, 480, 360, radius=6.0)
    rng = np.random.default_rng(404)
    frames = []
    for _ in range(2):
        X = S.sample_markers(rig, 3, rng, spread=0.10, min_sep_px=75.0, margin=36.0, tries=400)
        radii = rng.integers(17, 21, (4, len(X)))
        frames.append(S.render_frameset(rig, X, radii, rng))
    return rig, np.stack(frames)                                 # [FS=2, C=4, 360, 480]


def _run(rank, world, port, out_dir, backend="gloo", overlapped=False):
    sys.path.insert(0, REPO)
    sys.path.insert(0, os.path.join(REPO, "tests", "emu"))
    from mocapv2_b200.engine import CaptureEngine
    from mocapv2_b200.pipeline import CapturePipeline
    if backend == "nccl":
        torch.cuda.set_device(rank)
        if world > 1:
            dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                                    device_id=torch.device(f"cuda:{rank}"))
        eng = CaptureEngine(f"cuda:{rank}")
    else:
        import build_emu
        if world > 1:
            dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
        from emu_engine import EmuEngine
        eng = EmuEngine(build_emu.build())
    rig, fr = _ring4_scene()
    pipe = CapturePipeline(eng, rig, max_blobs=8, obj_count=4, max_groups=16, fp64=False, centroids="subpixel")
    local = torch.from_numpy(fr)[:, pipe.cam_begin:pipe.cam_begin + pipe.cams_local].contiguous().to(eng.device)
    if overlapped:                                               # overlapped detection + store-to-peer exchange, three steps
        pipe.pipelined_min_frames = 1
        for _ in range(3):
            res = pipe.step(local)
        assert world == 1 or pipe._peer, "the store-to-peer exchange was not set up"
    else:
        res = pipe.step(local)
    cpu = lambda t: t.cpu()
    torch.save({"b": res.fs_begin, "e": res.fs_end, "obj": cpu(res.corr.obj), "n_obj": cpu(res.corr.n_obj), "img": cpu(res.corr.img),
                "n_valid": cpu(res.corr.n_valid), "err": cpu(res.corr.err), "xy": cpu(res.det.xy), "count": cpu(res.det.count)},
               os.path.join(out_dir, f"rank{rank}_of{world}.pt"))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _compare(out):
    one = torch.load(os.path.join(out, "rank0_of1.pt"))
    assert one["img"].dtype == torch.float32 and one["xy"].dtype == torch.float32 and int(one["n_valid"].sum()) > 0
    assert bool((one["img"] != one["img"].floor()).any())        # sub-pixel values reached the matching
    for r in range(2):
        two = torch.load(os.path.join(out, f"rank{r}_of2.pt"))
        b, e = two["b"], two["e"]
        assert torch.equal(two["n_valid"], one["n_valid"][b:e]) and torch.equal(two["n_obj"], one["n_obj"][b:e])
        for s in range(e - b):
            nv, no = int(two["n_valid"][s]), int(two["n_obj"][s])
            assert torch.equal(two["img"][s, :nv], one["img"][b + s, :nv])
            assert torch.equal(two["obj"][s, :no], one["obj"][b + s, :no])
            assert torch.equal(two["err"][s, :nv], one["err"][b + s, :nv])
        assert torch.equal(two["count"].view(2, 2), one["count"].view(2, 4)[:, 2 * r:2 * r + 2])
        assert torch.equal(two["xy"].view(2, 2, -1, 2), one["xy"].view(2, 4, -1, 2)[:, 2 * r:2 * r + 2])


def test_pipeline_rejects_an_unknown_centroid_mode(emu_engine):
    with pytest.raises(ValueError):
        from mocapv2_b200.pipeline import CapturePipeline
        CapturePipeline(emu_engine, S.config_rig("c1"), centroids="float")


def test_subpixel_pipeline_two_ranks_equal_one_rank(tmp_path):
    sys.path.insert(0, os.path.join(REPO, "tests", "emu"))
    import build_emu
    build_emu.build()
    out = str(tmp_path)
    _run(0, 1, 0, out)
    port = 35500 + os.getpid() % 2000
    mp.spawn(_run, args=(2, port, out), nprocs=2, join=True)
    _compare(out)


@pytest.mark.gpu
def test_subpixel_two_gpus_store_to_peer_equal_one_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    out = str(tmp_path)
    port = 36500 + os.getpid() % 2000
    mp.spawn(_run, args=(1, port, out, "nccl", True), nprocs=1, join=True)
    mp.spawn(_run, args=(2, port, out, "nccl", True), nprocs=2, join=True)
    _compare(out)


# ---- accuracy ---------------------------------------------------------------------------------------------------------------------
def ideal_pixels(rig, X):
    """(C, M, 2) undistorted pinhole projections K0 [R|t] X: where the detection's undistorted image shows the markers."""
    K0 = np.asarray(rig["camera_params"][0]["intrinsic_matrix"], dtype=np.float64)
    out = []
    for p in rig["poses"]:
        Y = X @ np.asarray(p["R"]).T + np.asarray(p["t"]).reshape(3)
        h = Y @ K0.T
        out.append(h[:, :2] / h[:, 2:3])
    return np.stack(out)


def test_subpixel_accuracy_small_rig(engine):
    """Three cameras at 640x480, seeded scenes: sub-pixel centroids are unbiased to 0.05 px with an rms below 0.2 px per axis, and
    the matched 3-D points are at least four times closer to the markers than with whole-pixel centroids."""
    from mocapv2_b200.pipeline import CapturePipeline
    rig = S.ring_rig(3, 640, 480, radius=6.0)
    rng = np.random.default_rng(S.SEED0 + 77)
    n_sets = 8 if is_gpu(engine) else 4
    frames, markers = [], []
    for _ in range(n_sets):
        X = S.sample_markers(rig, 8, rng, spread=0.22, min_sep_px=90.0, margin=40.0, tries=400)
        frames.append(S.render_frameset(rig, X, rng.integers(14, 23, (3, len(X))), rng))
        markers.append(X)
    frames = np.stack(frames)
    dxy, err3 = [], {}
    for mode in ("int", "subpixel"):
        pipe = CapturePipeline(engine, rig, max_blobs=32, obj_count=32, max_groups=64, fp64=True, centroids=mode)
        res = pipe.step(dev(engine, frames))
        e3 = []
        for s in range(n_sets):
            truth = ideal_pixels(rig, markers[s])
            for c in range(3):
                i = s * 3 + c
                n = int(res.det.count[i])
                got = res.det.xy[i, :n].cpu().numpy().astype(np.float64)
                _, binimg = R.filter_frame(frames[s, c], rig["camera_params"][0]["intrinsic_matrix"], rig["camera_params"][0]["distortion_coef"])
                assert np.array_equal(got, np.array(oracle_points(binimg, subpixel=mode == "subpixel"), np.float64).reshape(-1, 2))
                if mode == "subpixel":
                    for q in got:
                        d = truth[c] - q
                        k = int(np.argmin((d * d).sum(axis=1)))
                        if np.abs(d[k]).max() < 3.0:
                            dxy.append(q - truth[c][k])
            no = int(res.corr.n_obj[s])
            for P in res.corr.obj[s, :no].cpu().numpy():
                d = float(np.linalg.norm(markers[s] - P, axis=1).min())
                if d < 0.01:                                            # a marker, not a ghost match
                    e3.append(d)
        assert len(e3) >= n_sets
        err3[mode] = float(np.mean(e3))
    dxy = np.array(dxy)
    assert len(dxy) >= 10 * n_sets
    assert np.all(np.abs(dxy.mean(axis=0)) <= 0.05), dxy.mean(axis=0)
    assert np.all(np.sqrt((dxy ** 2).mean(axis=0)) <= 0.2), np.sqrt((dxy ** 2).mean(axis=0))
    assert err3["subpixel"] <= 0.25 * err3["int"], err3
