"""Correspondence with a root's candidate groups spread over a whole CTA: against the capped restatement of the reference on a
bench-shaped 16-camera frame-set and at the edges of the group rounds, and bit-identical whatever the batch, layout or call."""
import numpy as np
import pytest
import torch

from mocapv2_b200 import synth as S
from oracle import restate as R

MAX_CAND = 8
REL_XYZ = 1e-4
TOL_PX = 1e-3


def dev(engine, a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(engine.device)


def to_lists(xy, cnt):
    """xy [C, max_pts, 2], cnt [C] -> the reference's per-camera lists"""
    return [[[x.item(), y.item()] for x, y in xy[c, :cnt[c]]] for c in range(xy.shape[0])]


def check_against_oracle(r, s, xy, cnt, rig, obj_count, fp64, max_groups):
    trace = {}
    o, ipa = R.correspond(to_lists(xy, cnt), rig["poses"], rig["camera_params"], rig["Fs"], obj_count, trace=trace,
                          max_cand=MAX_CAND, max_groups=max_groups)
    C = xy.shape[0]
    cand = r.cand[s].cpu().numpy()
    for j in range(int(cnt[0])):
        for i in range(1, C):
            want = [k for k, _ in trace["candidates"][j][i]]
            assert list(cand[j, i, :len(want)]) == want and (cand[j, i, len(want):] == -1).all()
    nv, no = int(r.n_valid[s]), int(r.n_obj[s])
    assert nv == len(ipa) and no == len(o)
    if nv:
        assert np.array_equal(r.img[s, :nv].cpu().numpy(), np.asarray(ipa, dtype=xy.dtype))
        got = r.obj[s, :no].cpu().numpy()
        assert (np.abs(got - o).max(axis=1) / np.linalg.norm(o, axis=1)).max() < (1e-10 if fp64 else REL_XYZ)
        e = r.err[s, :nv].cpu().numpy()
        assert np.abs(np.sqrt(e) - np.sqrt(np.array(trace["errors"]))).max() < (1e-9 if fp64 else TOL_PX)
    capped = any(n > max_groups for n, p in zip(trace["n_groups"], trace["per_root"]) if p is not None)
    assert bool(int(r.flags[s]) & 1) == capped


@pytest.mark.parametrize("fp64", [False, True])
def test_bench_shaped_frame_set(engine, fp64):
    """16 cameras, the marker pixels of one bench frame-set (128 markers; a view keeps the pixels inside the frame, about 97 per
    camera), candidates capped at 8 and groups at 64 as in the bench: candidates and image points exact, points and errors within
    the parity tolerances, the group-cap flag as the restatement's group counts say."""
    import bench
    rig, cen, _ = bench.make_scene(1)
    C = cen.shape[1]
    max_pts = 160
    xy = np.zeros((C, max_pts, 2), np.int32)
    cnt = np.zeros((C,), np.int32)
    for c in range(C):
        p = cen[0, c]
        p = p[(p[:, 0] >= 0) & (p[:, 0] < rig["W"]) & (p[:, 1] >= 0) & (p[:, 1] < rig["H"])]
        cnt[c] = len(p)
        xy[c, :len(p)] = p
    cams = engine.cameras(rig["poses"], rig["camera_params"])
    Fs = dev(engine, np.array(rig["Fs"], dtype=np.float64))
    r = engine.correspond(dev(engine, xy[None]), dev(engine, cnt[None]), Fs, cams, obj_count=128, max_groups=64, fp64=fp64,
                          want_cand=True)
    assert int(r.n_valid[0]) > 8
    check_against_oracle(r, 0, xy, cnt, rig, 128, fp64, 64)


# (candidates in cameras 1, 2, 3) per frame-set with one root: 1, 6, 9, 32, 35, 64, 70 and 512 groups
ONE_ROOT = [(1, 1, 1), (2, 3, 1), (3, 3, 1), (4, 8, 1), (5, 7, 1), (8, 8, 1), (5, 7, 2), (8, 8, 8)]


def edge_frame_sets(pt_dtype):
    """One marker per frame-set seen by 4 cameras; camera c > 0 holds its projection and n_c - 1 points a few pixels away, so every
    group is a well-posed triangulation.  The last two frame-sets: ten roots (neighbouring pixels of one marker) sharing 3 x 8 x 2
    candidates, and one with no point in camera 0; the one before them has no point in camera 2 (no complete root)."""
    rig = S.config_rig("c4")
    C = 4
    poses, params = rig["poses"][:C], rig["camera_params"][:C]
    rng = np.random.default_rng(7)
    offs = np.array([[0, 0], [2, 1], [-1, 3], [3, -2], [-3, -1], [1, -3], [4, 2], [-2, 4], [0, 5], [5, 0]], np.float64)
    shapes = [(1,) + n for n in ONE_ROOT] + [(1, 3, 0, 2), (10, 3, 8, 2), (0, 3, 3, 3)]
    max_pts = 12
    xy = np.zeros((len(shapes), C, max_pts, 2), pt_dtype)
    cnt = np.zeros((len(shapes), C), np.int32)
    for s, ns in enumerate(shapes):
        X = rig["centre"] + rng.uniform(-0.4, 0.4, (1, 3))
        for c in range(C):
            p = S.project_distorted(X, poses[c], params[c]["intrinsic_matrix"], params[c]["distortion_coef"])[0]
            p = p + offs[:ns[c]] + (rng.uniform(0, 1, (ns[c], 2)) if pt_dtype == np.float32 else 0.0)
            xy[s, c, :ns[c]] = np.floor(p) if pt_dtype == np.int32 else p
            cnt[s, c] = ns[c]
    sub = {"poses": poses, "camera_params": params, "Fs": rig["Fs"][:C - 1]}
    return sub, xy, cnt


@pytest.mark.parametrize("pt_dtype", [np.int32, np.float32])
@pytest.mark.parametrize("fp64", [False, True])
@pytest.mark.parametrize("max_groups", [31, 33, 64, 65, 4096])
def test_group_round_edges(engine, monkeypatch, max_groups, fp64, pt_dtype):
    """Evaluated group counts on both sides of 32 and 64 (capped counts 31, 33, 65 through max_groups), several complete roots
    splitting one CTA's groups, a frame-set without a complete root and one without a camera-0 point."""
    monkeypatch.setattr(R, "EPI_CUTOFF", 1e9)                    # every point is a candidate: the counts are the shapes above
    rig, xy, cnt = edge_frame_sets(pt_dtype)
    cams = engine.cameras(rig["poses"], rig["camera_params"])
    Fs = dev(engine, np.array(rig["Fs"], dtype=np.float64))
    r = engine.correspond(dev(engine, xy), dev(engine, cnt), Fs, cams, obj_count=4, cutoff=1e9, max_groups=max_groups, fp64=fp64,
                          want_cand=True)
    for s in range(xy.shape[0]):
        check_against_oracle(r, s, xy[s], cnt[s], rig, 4, fp64, max_groups)
    assert int(r.n_valid[-3]) == 0 and int(r.n_valid[-1]) == 0 and int(r.n_valid[-2]) == 10


def same(a, b, cnt):
    """every output the call defines: cand rows of the roots, cameras >= 1 (the rest of cand is left as the caller allocated it)"""
    for name in ("obj", "n_obj", "img", "n_valid", "err", "flags"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    for s, n in enumerate(cnt[:, 0]):
        assert torch.equal(a.cand[s, :n, 1:], b.cand[s, :n, 1:])


@pytest.mark.parametrize("pt_dtype", [np.int32, np.float32])
@pytest.mark.parametrize("fp64", [False, True])
def test_bit_identical_across_calls_batches_and_layouts(engine, fp64, pt_dtype):
    """Two calls on the same input, the batch against each frame-set alone, and the camera-blocked layout against the plain one
    agree bit for bit (the error sums keep one order whatever the CTA that evaluates a group)."""
    rig, xy, cnt = edge_frame_sets(pt_dtype)
    cams = engine.cameras(rig["poses"], rig["camera_params"])
    Fs = dev(engine, np.array(rig["Fs"], dtype=np.float64))
    kw = dict(obj_count=4, cutoff=1e9, max_groups=64, fp64=fp64, want_cand=True)
    a = engine.correspond(dev(engine, xy), dev(engine, cnt), Fs, cams, **kw)
    b = engine.correspond(dev(engine, xy), dev(engine, cnt), Fs, cams, **kw)
    same(a, b, cnt)
    for s in range(xy.shape[0]):
        one = engine.correspond(dev(engine, xy[s:s + 1]), dev(engine, cnt[s:s + 1]), Fs, cams, **kw)
        part = type(a)(**{k: (v[s:s + 1] if v is not None else None) for k, v in vars(a).items()})
        same(one, part, cnt[s:s + 1])
    # two camera blocks of two cameras: xy [B, S, C/B, max_pts, 2], count [B, S, C/B]
    S_, C, mp, _ = xy.shape
    xb = xy.reshape(S_, 2, 2, mp, 2).transpose(1, 0, 2, 3, 4)
    cb = cnt.reshape(S_, 2, 2).transpose(1, 0, 2)
    blk = engine.correspond(dev(engine, xb), dev(engine, cb), Fs, cams, **kw)
    same(a, blk, cnt)
