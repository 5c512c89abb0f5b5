"""Triangulation and reprojection against an FP64 DLT over the volume each rig sees, for every kernel variant.

The oracle here is a batched restatement of oracle.restate.triangulate_point / reprojection_error (cross-checked against them on a
sample), so thousands of points per case stay cheap.  Bounds are split by the conditioning of the DLT, kappa = lam_max / (lam_2 - lam_1)
of B = A^T A (lam_1 the smallest eigenvalue):
  - well-posed points (kappa < K0): FP32 meets BASELINE.json's contract (1e-4 relative, 1e-3 px), FP64 the check mode's tight bounds;
  - every point with at least two views: a finite result whose error stays below C_KAPPA * kappa * u (u the unit round-off), which a
    broken solve misses even where the input itself is ill-posed (two nearly opposite cameras: kappa up to ~1e8).
"""
import numpy as np
import pytest
import torch

from mocapv2_b200 import synth as S
from oracle import restate as R

REL_XYZ = 1e-4            # BASELINE.json: 3-D points within 1e-4 relative error
TOL_PX = 1e-3             # BASELINE.json: reprojection error within 1e-3 px (compared as RMS pixels)
F64_REL, F64_PX = 1e-11, 1e-9
U = {torch.float32: 2.0 ** -24, torch.float64: 2.0 ** -53}
# K0: every all-view point of the cases below has kappa 4 .. 79; pairs of the 6-camera ring two apart (120 degrees) reach ~140; nearly
# opposite pairs (1.6e3 .. 2.5e6) and 2-view rows of the masked cases (up to ~3e4) lie beyond.  tools/triangulation_volume_probe.py.
K0 = 1e3
# C_KAPPA: largest relative X error / (kappa * u) over every case of this file: FP32 0.78 on a B200 (1000 W) and 1.0 on the CPU
# emulation build, FP64 18.5 / 18.8 (a pair of the ring at kappa 18; X = v[:3] / v[3] with |X| ~ 6 m, so kappa * u is not the
# whole constant).  Set at about 4 and 5 times that.
C_KAPPA = {torch.float32: 4.0, torch.float64: 100.0}
MARGIN = 8.0              # px a point keeps from the frame edge in every used view


def dev(engine, a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(engine.device)


# ---- oracle -----------------------------------------------------------------------------------------------------------------
def rig_arrays(poses, params):
    Rt = np.stack([np.c_[np.asarray(p["R"], np.float64), np.asarray(p["t"], np.float64).reshape(3)] for p in poses])
    K = np.stack([np.asarray(c["intrinsic_matrix"], np.float64) for c in params])
    D = np.zeros((len(params), 5))
    for i, c in enumerate(params):
        d = np.asarray(c["distortion_coef"], np.float64).ravel()[:5]
        D[i, :d.size] = d
    return Rt, K, D


def view_rank(valid):
    """K (and distortion) of a view is taken by its rank among the point's valid views (Helpers.py:58-62)."""
    return np.clip(np.cumsum(valid, axis=1) - 1, 0, None)


def dlt64(pts, valid, Rt, K):
    """Batched FP64 DLT: pts [N, C, 2], valid [N, C] bool -> X [N, 3], kappa [N] (NaN rows where fewer than two views are valid)."""
    P = K[view_rank(valid)] @ Rt[None]                                            # [N, C, 3, 4]
    x, y = pts[..., 0:1], pts[..., 1:2]
    A = np.stack([y * P[:, :, 2] - P[:, :, 1], P[:, :, 0] - x * P[:, :, 2]], axis=2) * valid[:, :, None, None]
    A = A.reshape(len(pts), -1, 4)
    w, V = np.linalg.eigh(np.einsum("nri,nrj->nij", A, A))
    with np.errstate(divide="ignore", invalid="ignore"):                        # rows of fewer than two views, set to NaN below
        X = V[:, :3, 0] / V[:, 3:4, 0]
        kappa = w[:, 3] / (w[:, 1] - w[:, 0])
    few = valid.sum(1) < 2
    X[few] = np.nan
    kappa[few] = np.nan
    return X, kappa


def project_f32(X, Rt, K, D):
    """project_point_f32 for X [N, 3] through per-point cameras Rt [N, C, 3, 4], K [N, C, 3, 3], D [N, C, 5] -> (u, v) [N, C]."""
    X32 = X.astype(np.float32).astype(np.float64)[:, None, :]
    Y = [Rt[..., r, 0] * X32[..., 0] + Rt[..., r, 1] * X32[..., 1] + Rt[..., r, 2] * X32[..., 2] + Rt[..., r, 3] for r in range(3)]
    with np.errstate(divide="ignore"):
        z = np.where(Y[2] != 0, 1.0 / Y[2], 1.0)
    x, y = Y[0] * z, Y[1] * z
    k1, k2, p1, p2, k3 = (D[..., i] for i in range(5))
    r2 = x * x + y * y
    r4 = r2 * r2
    r6 = r4 * r2
    a1 = 2 * x * y
    a2 = r2 + 2 * x * x
    a3 = r2 + 2 * y * y
    cdist = 1 + k1 * r2 + k2 * r4 + k3 * r6
    xd = x * cdist + p1 * a1 + p2 * a2
    yd = y * cdist + p1 * a3 + p2 * a1
    return (xd * K[..., 0, 0] + K[..., 0, 2]).astype(np.float32), (yd * K[..., 1, 1] + K[..., 1, 2]).astype(np.float32)


def reproj64(pts, valid, X, Rt, K, D):
    """Mean squared x / y residual (px^2) over the valid views, pose by camera, lens by rank; NaN where fewer than two are valid."""
    rk = view_rank(valid)
    u, v = project_f32(X, np.broadcast_to(Rt[None], (len(pts),) + Rt.shape), K[rk], D[rk])
    sq = ((pts[..., 0] - u) ** 2 + (pts[..., 1] - v) ** 2) * valid
    nv = valid.sum(1)
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(nv >= 2, sq.sum(1) / (2 * nv), np.nan)


def cross_check(pts, valid, X, kappa, err, poses, params, rng, n=12):
    """The batched oracle agrees with oracle.restate on a sample of the points."""
    Ks = [np.asarray(c["intrinsic_matrix"], np.float64) for c in params]
    for i in rng.choice(len(pts), size=min(n, len(pts)), replace=False):
        idx = np.nonzero(valid[i])[0]
        if len(idx) < 2:
            continue
        Ps = [Ks[r] @ np.c_[np.asarray(poses[k]["R"]), np.asarray(poses[k]["t"]).reshape(3)] for r, k in enumerate(idx)]
        ref = R.triangulate_point(pts[i, idx], Ps)
        assert np.abs(ref - X[i]).max() / np.linalg.norm(ref) < 64 * kappa[i] * U[torch.float64]
        e = R.reprojection_error(pts[i, idx], X[i], [poses[k] for k in idx], params)
        assert abs(e - err[i]) <= 1e-12 * e


# ---- inputs -----------------------------------------------------------------------------------------------------------------
RIGS = {
    "c1": lambda: S.config_rig("c1"),
    "c3": lambda: S.config_rig("c3"),
    "c4": lambda: S.config_rig("c4"),
    "c5": lambda: S.config_rig("c5"),
    "ring6_lenses": lambda: S.ring_rig(6, 1440, 1080, lenses=S.per_camera_lenses(6)),
    "ring16_lenses": lambda: S.ring_rig(16, 2048, 2048, lenses=S.per_camera_lenses(16)),
}
_rig_cache = {}
HALF = {"c1": 0.5}        # m either side of the rig centre that points are drawn from (c1's 640x480 frames see a small volume)


def rig_views(name, views):
    rig = _rig_cache.setdefault(name, RIGS[name]())
    sub = dict(rig, poses=[rig["poses"][k] for k in views], camera_params=[rig["camera_params"][k] for k in views])
    return rig, sub


def visible_points(rig, sub, n, rng, half=1.5):
    """n seeded points of centre +- half (m) that every view of `sub` sees at least MARGIN px inside the frame -> X, pixels [n, C, 2]."""
    Xs, uvs, got = [], [], 0
    for _ in range(200):
        X = rig["centre"] + rng.uniform(-half, half, (2 * n + 1000, 3))
        uv = S.marker_pixels(sub, X)                                              # [C, M, 2]
        ok = ((uv[..., 0] > MARGIN) & (uv[..., 0] < rig["W"] - MARGIN) & (uv[..., 1] > MARGIN) & (uv[..., 1] < rig["H"] - MARGIN)).all(0)
        Xs.append(X[ok])
        uvs.append(uv[:, ok].transpose(1, 0, 2))
        got += int(ok.sum())
        if got >= n:
            break
    assert got >= n, "the rig does not see the volume"
    return np.concatenate(Xs)[:n], np.concatenate(uvs)[:n]


def centroids(uv, kind, rng):
    if kind == "int":
        return np.floor(uv)
    return (uv + rng.normal(0.0, 0.3, uv.shape)).astype(np.float32).astype(np.float64)


# ---- checks -----------------------------------------------------------------------------------------------------------------
def check_points(X, err, Xref, kappa, eref, eown, dtype, need_well_posed=True):
    """Bounds of the module docstring.  X / err from the kernel; Xref / kappa / eref from the oracle, eown the oracle's error at the
    kernel's X (rows with < 2 views NaN).  FP32 is held to the contract against the oracle's error at its own point; FP64 gets X within
    F64_REL and its error exact at its own X (against eref, a last-bit difference of X can move the float32 rounding of X by an ulp)."""
    has = np.isfinite(kappa)
    assert np.isnan(X[~has]).all() and np.isnan(err[~has]).all()
    assert np.isfinite(X[has]).all() and np.isfinite(err[has]).all()
    rel = np.abs(X[has] - Xref[has]).max(1) / np.linalg.norm(Xref[has], axis=1)
    k = kappa[has]
    ratio = rel / (k * U[dtype])
    assert ratio.max() < C_KAPPA[dtype], f"error {rel[ratio.argmax()]:.2e} at kappa {k[ratio.argmax()]:.2e}"
    wp = k < K0
    if need_well_posed:
        assert wp.any()
    dpx = np.abs(np.sqrt(err[has]) - np.sqrt((eref if dtype == torch.float32 else eown)[has]))
    rel_tol, px_tol = (REL_XYZ, TOL_PX) if dtype == torch.float32 else (F64_REL, F64_PX)
    assert rel[wp].max(initial=0.0) < rel_tol, f"well-posed rel X {rel[wp].max():.2e}"
    assert dpx[wp].max(initial=0.0) < px_tol, f"well-posed |d rms px| {dpx[wp].max():.2e}"
    return rel, dpx, k


def run_case(engine, rig_name, views, n, seed, kind, dtype, valid=None, half=None, need_well_posed=True):
    """Triangulate n visible points in both the kernel and the oracle; also reproject the oracle's and the kernel's points."""
    rng = np.random.default_rng(seed)
    rig, sub = rig_views(rig_name, views)
    _, uv = visible_points(rig, sub, n, rng, HALF.get(rig_name, 1.5) if half is None else half)
    pts = centroids(uv, kind, rng)
    C = len(views)
    vmask = np.ones((n, C), bool) if valid is None else valid.astype(bool)
    Rt, K, D = rig_arrays(sub["poses"], sub["camera_params"])
    Xref, kappa = dlt64(pts, vmask, Rt, K)
    eref = reproj64(pts, vmask, Xref, Rt, K, D)
    cross_check(pts, vmask, Xref, kappa, eref, sub["poses"], sub["camera_params"], rng)
    cams = engine.cameras(sub["poses"], sub["camera_params"])
    tp = dev(engine, pts).to(dtype)
    tv = None if valid is None else dev(engine, valid.astype(np.uint8))
    xyz, err = engine.triangulate(tp, cams, tv)
    X = xyz.double().cpu().numpy()
    check_points(X, err.double().cpu().numpy(), Xref, kappa, eref, reproj64(pts, vmask, X, Rt, K, D), dtype, need_well_posed)
    # reproject: the oracle's points, and the kernel's own points against the oracle's projection of them
    px_tol = TOL_PX if dtype == torch.float32 else F64_PX
    has = np.isfinite(kappa)
    for Xin in (Xref, X):
        e = engine.reproject(tp, dev(engine, np.nan_to_num(Xin)).to(dtype), cams, tv).double().cpu().numpy()
        ewant = reproj64(pts, vmask, Xin, Rt, K, D)
        assert np.isnan(e[~has]).all()
        assert np.abs(np.sqrt(e[has]) - np.sqrt(ewant[has])).max() < px_tol
    return kappa


# ---- cases ------------------------------------------------------------------------------------------------------------------
ALL_VIEW_CASES = [                     # (rig, first C views): FP32 runs triangulate_dense_f32_kernel<C> at C = 2, 4, 6, 8, 16
    ("c1", 2), ("c3", 3), ("c3", 6), ("c4", 2), ("c4", 4), ("c4", 7), ("c4", 8), ("c4", 16),
    ("c5", 5), ("c5", 8), ("ring6_lenses", 6), ("ring16_lenses", 16),
]


@pytest.mark.parametrize("kind", ["int", "sub"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])
@pytest.mark.parametrize("rig_name,C", ALL_VIEW_CASES, ids=[f"{r}-C{c}" for r, c in ALL_VIEW_CASES])
def test_all_views_over_volume(engine, rig_name, C, dtype, kind):
    """Every view valid, points over the whole commonly visible volume, 333 points (not a multiple of the 128-thread CTA)."""
    kappa = run_case(engine, rig_name, list(range(C)), 333, 1000 + 17 * C + len(rig_name), kind, dtype)
    assert kappa.max() < K0                                           # all-view points of every rig are well-posed


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])
@pytest.mark.parametrize("rig_name", ["ring6_lenses", "ring16_lenses", "c5"])
def test_masked_views_rank_lenses(engine, rig_name, dtype):
    """Random masks (40 % of views dropped) plus rows with 0, 1 and 2 valid views: P and the residual take K and the distortion of the
    view's rank among the valid views, so with a lens per camera a kernel that indexed them by camera fails; < 2 views give NaN."""
    rig = _rig_cache.setdefault(rig_name, RIGS[rig_name]())
    C = len(rig["poses"])
    n = 301
    rng = np.random.default_rng(77 + C)
    valid = (rng.random((n, C)) >= 0.4).astype(np.uint8)
    valid[0] = 0
    valid[1] = 0
    valid[1, C - 1] = 1
    valid[2] = 0
    valid[2, [1, C - 2]] = 1
    valid[3] = 1
    run_case(engine, rig_name, list(range(C)), n, 31 + C, "sub", dtype, valid=valid, half=0.6)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])
def test_every_pair_of_the_ring(engine, dtype):
    """All 15 camera pairs of the 6-camera ring: neighbours are well-posed, nearly opposite cameras have nearly collinear rays
    (kappa beyond 1e6), where only the kappa * u bound applies."""
    ks = []
    for a in range(6):
        for b in range(a + 1, 6):
            ks.append(run_case(engine, "c3", [a, b], 130, 500 + 6 * a + b, "int", dtype, half=0.4, need_well_posed=False))
    ks = np.concatenate(ks)
    assert ks.min() < 100 and ks.max() > 1e6                                     # the sweep spans well- to ill-posed


def test_ba_residuals_per_hypothesis(engine):
    """mocap_ba_residuals_batch: 9 pose hypotheses in one launch (blockIdx.y), each against its own oracle."""
    rng = np.random.default_rng(9)
    rig, sub = rig_views("c3", list(range(6)))
    _, uv = visible_points(rig, sub, 257, rng)
    pts = np.floor(uv)
    sets, want = [], []
    for s in range(9):
        poses = [dict(R=p["R"], t=np.asarray(p["t"]).reshape(3) + (rng.normal(0, 2e-3, 3) if s else 0.0)) for p in sub["poses"]]
        Rt, K, D = rig_arrays(poses, sub["camera_params"])
        valid = np.ones(pts.shape[:2], bool)
        X, _ = dlt64(pts, valid, Rt, K)
        want.append(reproj64(pts, valid, X, Rt, K, D))
        sets.append(engine.cameras(poses, sub["camera_params"]))
    e = engine.ba_residuals(dev(engine, pts), torch.stack(sets)).cpu().numpy()
    for s in range(9):
        assert np.abs(np.sqrt(e[s]) - np.sqrt(want[s])).max() < F64_PX, f"hypothesis {s}"


# ---- GPU only: more points than one grid of triangulate_kernel ----------------------------------------------------------------
def grid_points(engine):
    """Points one launch covers before its grid-stride loop wraps: SMs * 16 CTAs * 128 threads (launch_tri)."""
    return torch.cuda.get_device_properties(engine.device).multi_processor_count * 16 * 128


def sample_rows(P, G, rng):
    """A seeded sample plus the first and last point of every grid pass."""
    edges = [i for k in range(0, P, G) for i in (k, min(k + G, P) - 1)]
    return np.unique(np.r_[rng.choice(P, 2000, replace=False), edges])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])
@pytest.mark.parametrize("masked", [False, True], ids=["all-views", "masked"])
def test_grid_stride_beyond_one_grid(gpu_engine, dtype, masked):
    """2.4 grids of points through the generic (C = 5) and the masked (per-camera lenses) triangulation and through reproject."""
    eng = gpu_engine
    G = grid_points(eng)
    P = 2 * G + 2 * G // 5 + 77
    rng = np.random.default_rng(41 + masked)
    name = "ring6_lenses" if masked else "c5"
    views = list(range(6)) if masked else list(range(5))
    rig, sub = rig_views(name, views)
    _, uv = visible_points(rig, sub, P, rng, half=0.6)
    pts = centroids(uv, "sub", rng)
    valid = (rng.random((P, len(views))) >= 0.3).astype(np.uint8) if masked else None
    cams = eng.cameras(sub["poses"], sub["camera_params"])
    tp = dev(eng, pts).to(dtype)
    tv = None if valid is None else dev(eng, valid)
    xyz, err = eng.triangulate(tp, cams, tv)
    e_rep = eng.reproject(tp, xyz, cams, tv)
    rows = sample_rows(P, G, rng)
    vm = np.ones((len(rows), len(views)), bool) if valid is None else valid[rows].astype(bool)
    Rt, K, D = rig_arrays(sub["poses"], sub["camera_params"])
    Xref, kappa = dlt64(pts[rows], vm, Rt, K)
    eref = reproj64(pts[rows], vm, Xref, Rt, K, D)
    X = xyz.double().cpu().numpy()[rows]
    ewant = reproj64(pts[rows], vm, X, Rt, K, D)
    check_points(X, err.double().cpu().numpy()[rows], Xref, kappa, eref, ewant, dtype)
    has = np.isfinite(kappa)
    e2 = e_rep.double().cpu().numpy()[rows]
    assert np.isnan(e2[~has]).all()
    assert np.abs(np.sqrt(e2[has]) - np.sqrt(ewant[has])).max() < (TOL_PX if dtype == torch.float32 else F64_PX)


@pytest.mark.gpu
def test_ba_residuals_beyond_one_grid(gpu_engine):
    """mocap_ba_residuals_batch with 4 hypotheses over 2.2 grids of points."""
    eng = gpu_engine
    G = grid_points(eng)
    P = 2 * G + G // 5 + 3
    rng = np.random.default_rng(43)
    rig, sub = rig_views("c3", list(range(6)))
    _, uv = visible_points(rig, sub, P, rng, half=0.6)
    pts = np.floor(uv)
    rows = sample_rows(P, G, rng)
    sets, want = [], []
    for s in range(4):
        poses = [dict(R=p["R"], t=np.asarray(p["t"]).reshape(3) + (rng.normal(0, 2e-3, 3) if s else 0.0)) for p in sub["poses"]]
        Rt, K, D = rig_arrays(poses, sub["camera_params"])
        valid = np.ones((len(rows), 6), bool)
        X, _ = dlt64(pts[rows], valid, Rt, K)
        want.append(reproj64(pts[rows], valid, X, Rt, K, D))
        sets.append(eng.cameras(poses, sub["camera_params"]))
    e = eng.ba_residuals(dev(eng, pts), torch.stack(sets)).cpu().numpy()
    for s in range(4):
        assert np.abs(np.sqrt(e[s, rows]) - np.sqrt(want[s])).max() < F64_PX, f"hypothesis {s}"
