"""Geometry parity: DLT triangulation, reprojection error and epipolar correspondence through the C-ABI against
the reference-generated fixtures and the oracle.  Tolerances (BASELINE.json north_star): correspondence pairs
bit-exact (ties within 1e-5 of the cutoff are flagged), 3-D points within 1e-4 relative, reprojection error within
1e-3 px (compared as RMS pixels: the reference's value is a mean of SQUARED residuals, px^2)."""
import json
import os

import numpy as np
import pytest
import torch

from mocapv2_b200 import synth as S
from oracle import restate as R
from util import GOLDEN, lists_to_arrays

REL_XYZ = 1e-4        # north_star: 3-D points within 1e-4 relative error
TOL_PX = 1e-3         # north_star: reprojection error within 1e-3 px


def dev(engine, a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(engine.device)


def rel_err(X, ref):
    return float((np.abs(X - ref).max(axis=1) / np.linalg.norm(ref, axis=1)).max())


def kat():
    z = np.load(os.path.join(GOLDEN, "kat_triangulate.npz"))
    poses = [{"R": z["R"][i], "t": z["t"][i]} for i in range(2)]
    cp = [{"intrinsic_matrix": z["K"][i], "distortion_coef": z["dist"][i]} for i in range(2)]
    return z, poses, cp


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_kat_reference_golden_vector(engine, dtype):
    """jsons/image_points.json -> jsons/after_ba_objects.json, the reference's own known-answer pair."""
    z, poses, cp = kat()
    cams = engine.cameras(poses, cp)
    xyz, err = engine.triangulate(dev(engine, z["image_points"]).to(dtype), cams)
    X = xyz.double().cpu().numpy()
    e = err.double().cpu().numpy()
    tol = 1e-12 if dtype == torch.float64 else REL_XYZ
    assert rel_err(X, z["objects_json"]) < tol
    assert np.abs(np.sqrt(e) - np.sqrt(z["errors_ref"])).max() < (1e-9 if dtype == torch.float64 else TOL_PX)
    if dtype == torch.float64:                       # check mode reproduces cv.projectPoints' float32 roundings exactly
        assert np.allclose(e, z["errors_ref"], rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_eight_view_groups(engine, dtype):
    z = np.load(os.path.join(GOLDEN, "c5_groups.npz"))
    rig = S.config_rig("c5")
    cams = engine.cameras(rig["poses"], rig["camera_params"])
    pts = dev(engine, z["groups"]).to(dtype)
    xyz, err = engine.triangulate(pts, cams)
    assert rel_err(xyz.double().cpu().numpy(), z["objects_ref"]) < (1e-11 if dtype == torch.float64 else REL_XYZ)
    assert np.abs(np.sqrt(err.double().cpu().numpy()) - np.sqrt(z["errors_ref"])).max() < (1e-9 if dtype == torch.float64 else TOL_PX)
    # calculate_reprojection_errors on given object points (Helpers.py:102-143)
    e2 = engine.reproject(pts, dev(engine, z["objects_ref"]).to(dtype), cams)
    assert np.abs(np.sqrt(e2.double().cpu().numpy()) - np.sqrt(z["errors_ref"])).max() < (1e-9 if dtype == torch.float64 else TOL_PX)


def test_empty_batch(engine):
    rig = S.config_rig("c1")
    cams = engine.cameras(rig["poses"], rig["camera_params"])
    xyz, err = engine.triangulate(torch.zeros((0, 2, 2), dtype=torch.float32, device=engine.device), cams)
    assert xyz.shape == (0, 3) and err.shape == (0,)


def run_correspond(engine, points, rig, obj_count, fp64, **kw):
    xy, cnt = lists_to_arrays(points)
    cams = engine.cameras(rig["poses"], rig["camera_params"])
    Fs = dev(engine, np.array(rig["Fs"], dtype=np.float64))
    return engine.correspond(dev(engine, xy), dev(engine, cnt), Fs, cams, obj_count=obj_count, fp64=fp64, want_cand=True, **kw)


@pytest.mark.parametrize("fp64", [True, False])
def test_correspondence_reference_cases(engine, fp64):
    """find_point_correspondance_and_object_points on 2/6/8/16-camera frame-sets produced by the reference itself."""
    geo = json.load(open(os.path.join(GOLDEN, "geometry.json")))
    if engine.device.type != "cuda":
        geo = geo[::3]
    rigs = {}
    for rec in geo:
        rig = rigs.setdefault(rec["config"], S.config_rig(rec["config"]))
        r = run_correspond(engine, rec["points"], rig, rec["obj_count"], fp64)
        nv, no = int(r.n_valid[0]), int(r.n_obj[0])
        ref_ipa = np.array(rec["image_points_all"])
        ref_o = np.array(rec["object_points"])
        assert nv == (ref_ipa.shape[0] if ref_ipa.size else 0)
        if nv:
            assert np.array_equal(r.img[0, :nv].cpu().numpy(), ref_ipa)            # matched pairs: bit-exact
            assert no == ref_o.shape[0]
            assert rel_err(r.obj[0, :no].cpu().numpy(), ref_o) < (1e-11 if fp64 else REL_XYZ)
        else:
            assert no == 0                                                          # the reference returns shape (0,)
        # candidate lists and per-root mean errors against the oracle's trace
        trace = {}
        R.correspond(rec["points"], rig["poses"], rig["camera_params"], rig["Fs"], rec["obj_count"], trace=trace)
        cand = r.cand[0].cpu().numpy()
        for j, per_cam in enumerate(trace["candidates"]):
            for i in range(1, len(rig["poses"])):
                want = [k for k, _ in per_cam[i]]
                got = [int(k) for k in cand[j, i] if k >= 0]
                assert got == want[:8]
        errs = [e for e in trace["errors"]]
        got_e = r.err[0, :nv].cpu().numpy()
        assert np.abs(np.sqrt(got_e) - np.sqrt(np.array(errs))).max(initial=0.0) < (1e-9 if fp64 else TOL_PX)
        assert bool(int(r.flags[0]) & 4) == bool(trace["ties"])


@pytest.mark.parametrize("fp64", [True, False])
def test_correspondence_ambiguous_candidates(engine, fp64):
    """Several points inside the 10 px epipolar band: candidate order, the cartesian group enumeration, the
    first-group point and the mean-over-all-groups ranking (Helpers.py:219-273), incl. obj_count+1 slicing."""
    rig = S.config_rig("c3")
    rng = np.random.default_rng(21)
    n_cases = 6 if engine.device.type == "cuda" else 2
    for case in range(n_cases):
        X = S.config_markers("c3", rig, rng)[:5] * 1.0
        uv = S.marker_pixels(rig, X)
        pts = []
        for c in range(6):
            p = [[int(u), int(v)] for u, v in uv[c]]
            for k in range(3):                        # decoys close to true points -> extra in-band candidates
                u, v = uv[c][rng.integers(0, 5)]
                p.append([int(u + rng.uniform(-6, 6)), int(v + rng.uniform(-6, 6))])
            order = rng.permutation(len(p))
            pts.append([p[k] for k in order])
        if case == 1:
            pts[2] = [[None, None]]
        obj_count = int(rng.integers(0, 7))
        trace = {}
        o, ipa = R.correspond(pts, rig["poses"], rig["camera_params"], rig["Fs"], obj_count, trace=trace)
        r = run_correspond(engine, pts, rig, obj_count, fp64)
        nv, no = int(r.n_valid[0]), int(r.n_obj[0])
        assert nv == (ipa.shape[0] if ipa.size else 0) and no == (o.shape[0] if o.size else 0)
        if nv:
            assert max(trace["n_groups"]) > 1                                      # the case really is ambiguous
            assert np.array_equal(r.img[0, :nv].cpu().numpy(), ipa)
            assert rel_err(r.obj[0, :no].cpu().numpy(), o) < (1e-10 if fp64 else REL_XYZ)
            got_e = r.err[0, :nv].cpu().numpy()
            assert np.abs(np.sqrt(got_e) - np.sqrt(np.array(trace["errors"]))).max() < (1e-9 if fp64 else TOL_PX)
        assert int(r.flags[0]) & 3 == 0                                            # no cap was hit


def test_correspondence_caps_are_flagged(engine):
    """More in-band candidates than MOCAP_MAX_CAND / more groups than max_groups: flagged, never silent."""
    rig = S.config_rig("c1")
    root = [320, 240]
    line = R.epiline_f32(root, np.array(rig["Fs"][0]))
    a, b, c = line
    pts1 = []
    for k in range(12):                                # 12 points on the epipolar line of the root
        x = 100 + 30 * k
        pts1.append([x, int(round(-(a * x + c) / b))])
    r = run_correspond(engine, [[root], pts1], rig, 0, True, max_groups=4)
    assert int(r.flags[0]) & 2 and int(r.flags[0]) & 1
    r = run_correspond(engine, [[root], pts1[:6]], rig, 0, True, max_groups=4)
    assert int(r.flags[0]) & 1 and not int(r.flags[0]) & 2


def test_batch_of_frame_sets_equals_one_by_one(engine):
    geo = [g for g in json.load(open(os.path.join(GOLDEN, "geometry.json"))) if g["config"] == "c3" and g["obj_count"] == 10]
    rig = S.config_rig("c3")
    mp = 16
    arrays = [lists_to_arrays(g["points"], mp) for g in geo]
    xy = np.concatenate([a[0] for a in arrays])
    cnt = np.concatenate([a[1] for a in arrays])
    cams = engine.cameras(rig["poses"], rig["camera_params"])
    Fs = dev(engine, np.array(rig["Fs"], dtype=np.float64))
    r = engine.correspond(dev(engine, xy), dev(engine, cnt), Fs, cams, obj_count=10)
    for s, g in enumerate(geo):
        one = engine.correspond(dev(engine, xy[s:s + 1]), dev(engine, cnt[s:s + 1]), Fs, cams, obj_count=10)
        assert int(one.n_valid[0]) == int(r.n_valid[s]) and int(one.n_obj[0]) == int(r.n_obj[s])
        no = int(one.n_obj[0])
        assert torch.equal(one.obj[0, :no], r.obj[s, :no])                          # bit-identical (fixed-order reductions)


# ---------------------------------------------------------------------------------------------------------------------------
# GPU only: C5 sizes through size-independent properties
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_c5_million_points_properties(gpu_engine):
    """1e6 eight-view correspondences: exact projections triangulate back to the marker (round trip), FP32 main mode
    stays within 1e-4 of the FP64 check mode on the whole batch, the oracle agrees on a sample, and the result does
    not depend on the batch split."""
    eng = gpu_engine
    rig = S.config_rig("c5")
    cams = eng.cameras(rig["poses"], rig["camera_params"])
    P = 1_000_000
    g = torch.Generator(device=eng.device).manual_seed(5)
    centre = torch.tensor(np.asarray(rig["centre"]), device=eng.device)
    X = centre + (torch.rand((P, 3), generator=g, device=eng.device, dtype=torch.float64) - 0.5) * 1.0
    cam_np = cams.cpu().numpy()
    Pm = torch.tensor(cam_np[:, :12].reshape(8, 3, 4), device=eng.device)
    Xh = torch.cat([X, torch.ones((P, 1), device=eng.device, dtype=torch.float64)], dim=1)
    proj = torch.einsum("cij,pj->pci", Pm, Xh)
    uv = proj[..., :2] / proj[..., 2:3]                                             # ideal pinhole pixels (no distortion)
    xyz64, _ = eng.triangulate(uv.contiguous(), cams)
    assert float(((xyz64 - X).abs().amax(dim=1) / X.norm(dim=1)).max()) < 1e-8      # round trip
    uvi = torch.floor(uv + (torch.rand(uv.shape, generator=g, device=eng.device, dtype=torch.float64) - 0.5) * 4).contiguous()
    xyz64, err64 = eng.triangulate(uvi, cams)
    xyz32, err32 = eng.triangulate(uvi.float().contiguous(), cams)
    rel = ((xyz32.double() - xyz64).abs().amax(dim=1) / xyz64.norm(dim=1)).max()
    assert float(rel) < REL_XYZ
    assert float((err32.double().sqrt() - err64.sqrt()).abs().max()) < TOL_PX
    idx = torch.randint(0, P, (64,), generator=torch.Generator().manual_seed(1))
    ref = R.triangulate_points(uvi[idx.to(eng.device)].cpu().numpy(), rig["poses"], rig["camera_params"])
    assert rel_err(xyz64[idx.to(eng.device)].cpu().numpy(), ref) < 1e-10
    ref_e = R.reprojection_errors(uvi[idx.to(eng.device)].cpu().numpy(), ref, rig["poses"], rig["camera_params"])
    assert np.abs(err64[idx.to(eng.device)].cpu().numpy() - ref_e).max() < 1e-7
    half, _ = eng.triangulate(uvi[: P // 2].float().contiguous(), cams)
    assert torch.equal(half, xyz32[: P // 2])
