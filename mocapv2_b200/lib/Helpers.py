"""B200 drop-in for the hot-path functions of the reference's lib/Helpers.py.

Same names, arguments, return conventions and module globals as the reference:
  triangulate_point / triangulate_points                     lib/Helpers.py:43-99
  calculate_reprojection_error / calculate_reprojection_errors   lib/Helpers.py:102-143
  find_point_correspondance_and_object_points                lib/Helpers.py:178-280
  bundle_adjustment, params_to_camera_poses                  lib/Helpers.py:145-176 (caller of the path, SURVEY 8f row 1)
  get_extrinsics, read_camera_params, read_fundamental_matrix lib/Helpers.py:282-291, 30-40, 22-28
  globals camera_params, camera_params_path, Fs (assignable: >2-camera rigs inject them, like with the reference)
The arithmetic runs in libmocap_b200.so (sm_100a).  These list-in / ndarray-out calls handle one frame-set and are
latency bound, so they use the kernels' FP64 check mode (`precision = "fp64"`; scipy's finite-difference bundle
adjustment, Helpers.py:158-176, needs it); set `precision = "fp32"` for the throughput mode the batch API uses.
"""
import json
import warnings

import numpy as np
import torch

from .. import _cabi
from .. import engine as _engine

camera_params = None
camera_params_path = "./jsons/camera-params-in.json"
Fs = []
precision = "fp64"
max_groups = 1 << 16        # candidate groups evaluated per root before MOCAP_CFLAG_GROUP_CAP is raised


def get_extrinsics(path="./jsons/after_ba_extrinsics.json"):
    global global_camera_poses
    global camera_count
    with open(path) as file:
        global_camera_poses = json.load(file)
    for pose in global_camera_poses:
        pose["R"] = np.array(pose["R"])
        pose["t"] = np.array(pose["t"])
    camera_count = len(global_camera_poses)
    return global_camera_poses, camera_count


def read_fundamental_matrix():
    global Fs
    if len(Fs) == 0:
        with open("./jsons/fundamentals.json") as file:
            Fs = json.load(file)
            print("Fundamental matrix loaded")


def read_camera_params():
    global camera_params
    if camera_params is None:
        with open(camera_params_path, "r") as file:
            camera_params = np.array(json.load(file))
            print("Camera params loaded")
            return camera_params


def _dtype():
    return torch.float64 if precision == "fp64" else torch.float32


def _is_none(p):
    return p is None or (len(p) == 2 and p[0] is None and p[1] is None)


def _group_arrays(groups, n_cams):
    """list of groups ([C][2], None allowed) -> pts (P, C, 2) float64, valid (P, C) uint8."""
    P = len(groups)
    pts = np.zeros((P, n_cams, 2), dtype=np.float64)
    valid = np.zeros((P, n_cams), dtype=np.uint8)
    for g, group in enumerate(groups):
        for c, p in enumerate(group):
            if not _is_none(p):
                pts[g, c] = (float(p[0]), float(p[1]))
                valid[g, c] = 1
    return pts, valid


def _run_triangulate(groups, camera_poses, want_err=False, xyz=None):
    eng = _engine.default_engine()
    read_camera_params()
    C = len(camera_poses)
    pts, valid = _group_arrays(groups, C)
    cams = eng.cameras(camera_poses, camera_params)
    dt = _dtype()
    tp = torch.from_numpy(pts).to(eng.device, dt)
    tv = None if valid.all() else torch.from_numpy(valid).to(eng.device)
    if xyz is None:
        X, e = eng.triangulate(tp, cams, tv, want_err=want_err)
        return X.double().cpu().numpy(), (e.double().cpu().numpy() if want_err else None), valid
    tx = torch.from_numpy(np.asarray(xyz, dtype=np.float64).reshape(-1, 3)).to(eng.device, dt)
    e = eng.reproject(tp, tx, cams, tv)
    return None, e.double().cpu().numpy(), valid


def triangulate_point(image_points, camera_poses):
    """image_points shape = [camera_count,2]; views equal to [None, None] are dropped; <= 1 view -> [None, None, None]."""
    image_points = list(image_points)
    if sum(0 if _is_none(p) else 1 for p in image_points) <= 1:
        return [None, None, None]
    X, _, _ = _run_triangulate([image_points], camera_poses)
    return X[0]


def triangulate_points(image_points, camera_poses):
    """image_points shape = [obj points,camera_count,2]; groups holding a [None, None] view are skipped (Helpers.py:93)."""
    groups = [g for g in image_points if not any(_is_none(p) for p in g)]
    if len(groups) == 0:
        return np.array([])
    X, _, _ = _run_triangulate(groups, camera_poses)
    return X


def calculate_reprojection_error(image_points, object_point, camera_poses):
    """mean of squared x/y pixel residuals over the cameras that saw the point (px^2); None if <= 1 view."""
    image_points = list(image_points)
    if sum(0 if _is_none(p) else 1 for p in image_points) <= 1:
        return None
    _, e, _ = _run_triangulate([image_points], camera_poses, xyz=[object_point])
    return float(e[0])


def calculate_reprojection_errors(image_points, object_points, camera_poses):
    groups, xyz = [], []
    for g, X in zip(image_points, object_points):
        if sum(0 if _is_none(p) else 1 for p in g) <= 1:
            continue
        groups.append(list(g))
        xyz.append(X)
    if not groups:
        return np.array([])
    _, e, _ = _run_triangulate(groups, camera_poses, xyz=np.asarray(xyz, dtype=np.float64))
    return e


def params_to_camera_poses(params, num_cameras=2):
    """rotation vector + translation per camera after the first -> pose dicts (lib/Helpers.py:145-156)."""
    from scipy.spatial.transform import Rotation
    camera_poses = [{"R": np.eye(3), "t": np.array([0, 0, 0], dtype=np.float32)}]
    for i in range(0, num_cameras - 1):
        camera_poses.append({"R": Rotation.as_matrix(Rotation.from_rotvec(params[i * 6: i * 6 + 3])),
                             "t": params[i * 6 + 3: i * 6 + 6]})
    return camera_poses


def bundle_adjustment(image_points, camera_poses):
    """Refine the second camera's pose (lib/Helpers.py:158-176): scipy least_squares (TRF, 2-point finite differences) over the
    mean squared reprojection errors, cast to float32 like the reference.  Same quirks: two cameras hard-coded (:162, :174).

    The residual -- triangulate_points + calculate_reprojection_errors on all points (:160-167) -- runs on the GPU in FP64 with the
    reference's roundings, and an optimiser iteration costs ONE launch: scipy hands the perturbed parameter vectors of its
    finite-difference Jacobian to `workers`, here a map that evaluates all of them as pose hypotheses of a single
    mocap_ba_residuals_batch call (x and the six x + h e_i).  The optimiser itself, its step sizes and its arithmetic on the
    residuals are scipy's, exactly as in the reference, so jsons/before_ba_extrinsics.json still gives after_ba_extrinsics.json."""
    from scipy import optimize
    from scipy.spatial.transform import Rotation
    eng = _engine.default_engine()
    read_camera_params()
    groups = [list(g) for g in image_points]
    fused = len(groups) > 0 and all(len(g) == 2 and not any(_is_none(p) for p in g) for g in groups)
    stats = {"launches": 0, "hypotheses": 0}

    if fused:
        pts_dev = torch.from_numpy(np.asarray(groups, dtype=np.float64).reshape(len(groups), 2, 2)).to(eng.device)

        def residuals_of(params_list):
            cams = np.stack([_engine.pack_cameras(params_to_camera_poses(np.asarray(p), 2), camera_params) for p in params_list])
            err = eng.ba_residuals(pts_dev, torch.from_numpy(cams).to(eng.device))
            stats["launches"] += 1
            stats["hypotheses"] += len(params_list)
            return [e.astype(np.float32) for e in err.cpu().numpy()]

        def residual_function(params):
            return residuals_of([params])[0]

        def hypotheses_map(fun, xs):                       # scipy's `workers`: all finite-difference points of an iteration at once
            return [np.atleast_1d(r) for r in residuals_of(list(xs))]
    else:                                                  # groups with missing views: the reference's per-call path (:93, :125)
        global precision
        saved = precision

        def residual_function(params):
            global precision
            precision = "fp64"
            try:
                poses = params_to_camera_poses(params, 2)
                object_points = triangulate_points(image_points, poses)
                errors = calculate_reprojection_errors(image_points, object_points, poses)
            finally:
                precision = saved
            return errors.astype(np.float32)
        hypotheses_map = None

    init_params = np.array([])
    for camera_pose in camera_poses[1:]:
        init_params = np.concatenate([init_params, Rotation.from_matrix(camera_pose["R"]).as_rotvec(),
                                      np.asarray(camera_pose["t"]).flatten()])
    result = optimize.least_squares(residual_function, init_params, verbose=0, loss="linear", method="trf", ftol=1E-5, xtol=1E-15,
                                    workers=hypotheses_map)
    bundle_adjustment.last_stats = dict(stats, nfev=int(result.nfev), njev=int(result.njev) if result.njev is not None else None)
    return params_to_camera_poses(result.x)


def find_point_correspondance_and_object_points(image_points, camera_poses, obj_count=0, debug=False):
    """image_points shape = [camera_count, obj points, 2] -> (object_points sorted by error, image_points_all).

    Mutates the per-camera lists like the reference (one [None, None] removed from each, Helpers.py:184-188).
    The points are whole pixels (the output of _find_dot; image_points_all int64) or sub-pixel centroids whose every coordinate is a
    float32 value (the output of _find_dot(..., subpixel=True); image_points_all float64, as the reference returns float lists)."""
    read_camera_params()
    for image_points_i in image_points:
        try:
            image_points_i.remove([None, None])
        except Exception:
            pass
    read_fundamental_matrix()
    eng = _engine.default_engine()
    C = len(camera_poses)
    if len(image_points) < C:
        raise IndexError("list index out of range")              # image_points[i], Helpers.py:203-216
    if C > 1 and len(Fs) < C - 1:
        raise IndexError("list index out of range")              # Fs[i-1], Helpers.py:206
    lists = []
    for cam in list(image_points)[:C]:
        pts = [p for p in np.asarray(cam, dtype=object).reshape(-1, 2).tolist() if not _is_none(p)] if len(cam) else []
        lists.append(np.asarray(pts, dtype=np.float64).reshape(-1, 2))
    if all(np.array_equal(a, np.rint(a)) for a in lists):
        dtype = np.int32
    elif all(np.array_equal(a, a.astype(np.float32)) for a in lists):
        dtype = np.float32                                       # sub-pixel centroids: every coordinate exactly a float32 value
    else:
        raise ValueError("image points must be integer pixel coordinates (the output of _find_dot) or float32 values "
                         "(the output of _find_dot(..., subpixel=True))")
    lists = [a.astype(dtype) for a in lists]
    max_pts = max(1, max(len(a) for a in lists))
    xy = np.zeros((1, C, max_pts, 2), dtype=dtype)
    cnt = np.zeros((1, C), dtype=np.int32)
    for c, a in enumerate(lists):
        cnt[0, c] = len(a)
        xy[0, c, :len(a)] = a
    cams = eng.cameras(camera_poses, camera_params)
    F = torch.from_numpy(np.asarray(Fs, dtype=np.float64)[: max(C - 1, 0)].reshape(-1, 3, 3).copy()).to(eng.device)
    res = eng.correspond(torch.from_numpy(xy).to(eng.device), torch.from_numpy(cnt).to(eng.device), F, cams,
                         obj_count=int(obj_count), fp64=(precision == "fp64"), max_groups=max_groups)
    flags = int(res.flags[0])
    if flags & (_cabi.CFLAG_GROUP_CAP | _cabi.CFLAG_CAND_CAP):
        warnings.warn("candidate cap reached (MOCAP_MAX_CAND / max_groups): ranking used a truncated group set")
    if debug and flags & _cabi.CFLAG_TIE:
        print("epipolar distance within 1e-5 of the cutoff (tie)")
    nv, no = int(res.n_valid[0]), int(res.n_obj[0])
    if nv == 0:
        return np.array([]), np.array([])
    return res.obj[0, :no].cpu().numpy(), res.img[0, :nv].cpu().numpy().astype(np.int64 if dtype == np.int32 else np.float64)
