"""Synthetic rigs and IR frames for the BASELINE.json configs (C1..C5).  Data plumbing, no hot-path code.

The frame recipe follows SURVEY.md section 8(d): background uint8 ~ U[0,40), every visible marker a filled
disc of value 255 with radius U{14..22} px, then a sigma=1.2 Gaussian blur.  Marker centres are the pinhole
projection of the 3-D marker through K[R|t] followed by the forward distortion model of camera 0, because
the reference's ``_find_dot`` always undistorts with camera 0's coefficients (lib/ImageOperations.py:37-38).
A rig built with one lens per camera (``ring_rig(..., lenses=...)``, ``per_camera_lenses``) records that
(``rig["per_camera_lens"]``); its markers are then projected with every camera's own K and distortion.

``fundamental_from_poses`` restates CalculateCameraPoses.py:26-78 (F = K2^-T [t]x R K1^-1 for the relative
pose cam1 -> cam2); it is how jsons/fundamentals.json is produced, needed for rigs with more than 2 cameras.
"""
from __future__ import annotations

import json
import os

import numpy as np

# jsons/camera-params-in.json[0] of the reference (calibration data, identical for both shipped cameras).
SHIPPED_K = [[4425.2825371191575, 0.0, 1002.8525938875283],
             [0.0, 4384.8283962019805, 937.7284647311761],
             [0.0, 0.0, 1.0]]
SHIPPED_DIST = [-0.10851162502101634, -0.3633831473519663, -0.004334575904059801,
                -0.0133267085440563, 3.760714860334118]
# jsons/after_ba_extrinsics.json
SHIPPED_POSES = [
    {"R": [[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.0, 0.0, 1.0]], "t": [0.0, 0.0, 0.0]},
    {"R": [[0.8777073023572017, 0.1320083201977881, -0.4606557226252616],
           [-0.14209968061844094, 0.989768481237702, 0.012885430398314857],
           [0.4576434989781684, 0.05414939470549039, 0.8874853637644106]],
     "t": [-0.9981776218123374, -0.05336798347158354, -0.026297869475077427]},
]
# jsons/fundamentals.json (the same matrix is stored twice there)
SHIPPED_F = [[4.8347798791554796e-08, -3.8809070512419274e-08, 0.0003468916292637166],
             [-7.428990458578177e-07, -1.001621415010475e-07, -0.005991563036692725],
             [-0.0007711268620280697, 0.0074991896444215975, 1.0]]
# SURVEY 8(d) C1: four markers visible in both 640x480 views of the shipped rig
C1_MARKERS = [(0.2102, 0.4108, -2.10), (0.2687, 0.3246, -2.04), (0.3737, 0.3560, -2.06), (0.3056, 0.3991, -2.04)]

SEED0 = 20261018


def shipped_camera_params(n=2):
    return [{"intrinsic_matrix": [list(r) for r in SHIPPED_K], "distortion_coef": list(SHIPPED_DIST)}
            for _ in range(n)]


def shipped_poses():
    return [{"R": np.array(p["R"], dtype=np.float64), "t": np.array(p["t"], dtype=np.float64)} for p in SHIPPED_POSES]


def fundamental_from_poses(pose1, pose2, K1, K2):
    """F with x2^T F x1 = 0 (CalculateCameraPoses.py:26-78), normalised so F[2][2] = 1 when possible."""
    R1 = np.asarray(pose1["R"], dtype=np.float64)
    t1 = np.asarray(pose1["t"], dtype=np.float64).reshape(3, 1)
    R2 = np.asarray(pose2["R"], dtype=np.float64)
    t2 = np.asarray(pose2["t"], dtype=np.float64).reshape(3, 1)
    R_rel = R2 @ R1.T
    t_rel = (t2 - R_rel @ t1).ravel()
    tx = np.array([[0.0, -t_rel[2], t_rel[1]], [t_rel[2], 0.0, -t_rel[0]], [-t_rel[1], t_rel[0], 0.0]])
    E = tx @ R_rel
    F = np.linalg.inv(np.asarray(K2, dtype=np.float64)).T @ E @ np.linalg.inv(np.asarray(K1, dtype=np.float64))
    if abs(F[2, 2]) > 1e-300:
        F = F / F[2, 2]
    return F


def project_distorted(X, pose, K, dist):
    """Pinhole + forward Brown distortion (k1,k2,p1,p2,k3): world points (n,3) -> pixels (n,2), FP64."""
    X = np.asarray(X, dtype=np.float64).reshape(-1, 3)
    R = np.asarray(pose["R"], dtype=np.float64)
    t = np.asarray(pose["t"], dtype=np.float64).reshape(3)
    K = np.asarray(K, dtype=np.float64)
    k1, k2, p1, p2, k3 = (list(dist) + [0, 0, 0, 0, 0])[:5]
    Y = X @ R.T + t
    x = Y[:, 0] / Y[:, 2]
    y = Y[:, 1] / Y[:, 2]
    r2 = x * x + y * y
    cd = 1 + k1 * r2 + k2 * r2 * r2 + k3 * r2 * r2 * r2
    xd = x * cd + 2 * p1 * x * y + p2 * (r2 + 2 * x * x)
    yd = y * cd + p1 * (r2 + 2 * y * y) + 2 * p2 * x * y
    return np.stack([K[0, 0] * xd + K[0, 2], K[1, 1] * yd + K[1, 2]], axis=1)


def _rot_a_to_b(a, b):
    """Rotation matrix taking unit vector a to unit vector b."""
    a = a / np.linalg.norm(a)
    b = b / np.linalg.norm(b)
    v = np.cross(a, b)
    c = float(a @ b)
    if np.linalg.norm(v) < 1e-15:
        return np.eye(3)
    vx = np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])
    return np.eye(3) + vx + vx @ vx / (1 + c)


def per_camera_lenses(n_cams, seed=SEED0, scale=1.0):
    """n_cams distinct lenses around the shipped one, [(K, dist), ...]: focal lengths within +-3 %, principal point within +-2 %
    of the frame size of the shipped calibration (2048 px), distortion coefficients within +-15 % (times `scale`).  Camera 0 keeps
    the shipped lens."""
    rng = np.random.default_rng(seed)
    out = [(np.array(SHIPPED_K, dtype=np.float64), np.array(SHIPPED_DIST, dtype=np.float64))]
    for _ in range(1, n_cams):
        K = np.array(SHIPPED_K, dtype=np.float64)
        K[0, 0] *= 1 + scale * rng.uniform(-0.03, 0.03)
        K[1, 1] *= 1 + scale * rng.uniform(-0.03, 0.03)
        K[0, 2] += scale * rng.uniform(-40.0, 40.0)
        K[1, 2] += scale * rng.uniform(-40.0, 40.0)
        d = np.array(SHIPPED_DIST, dtype=np.float64) * (1 + scale * rng.uniform(-0.15, 0.15, 5))
        out.append((K, d))
    return out


def camera_lens(rig, c):
    """(K, dist) the frames of camera c are distorted with: its own with per-camera lenses, camera 0's otherwise."""
    cp = rig["camera_params"][c if rig.get("per_camera_lens") else 0]
    return cp["intrinsic_matrix"], cp["distortion_coef"]


def ring_rig(n_cams, W, H, radius=6.0, K=None, dist=None, height=0.8, lenses=None):
    """n_cams cameras on a ring looking at the origin so that the origin projects to the image centre.

    Camera 0 is re-based to R = I, t = 0 like the reference's calibration (CalculateCameraPoses.py) does, i.e.
    world coordinates are camera-0 coordinates.  Returns dict(camera_params, poses, Fs, W, H, centre).
    lenses: [(K_i, dist_i)] one per camera (in place of K / dist): the rig's frames are distorted per camera.
    """
    if lenses is not None:
        if len(lenses) != n_cams:
            raise ValueError("one lens per camera")
        K, dist = lenses[0]
    K = np.array(SHIPPED_K if K is None else K, dtype=np.float64)
    dist = list(SHIPPED_DIST if dist is None else dist)
    ray_c = np.linalg.inv(K) @ np.array([W / 2.0, H / 2.0, 1.0])
    poses_w = []
    for c in range(n_cams):
        ang = 2 * np.pi * c / n_cams + 0.13
        pos = np.array([radius * np.cos(ang), height * (1 if c % 2 == 0 else -0.6), radius * np.sin(ang)])
        fwd = -pos / np.linalg.norm(pos)
        up = np.array([0.0, 1.0, 0.0])
        right = np.cross(up, fwd)
        right /= np.linalg.norm(right)
        down = np.cross(fwd, right)
        R0 = np.stack([right, down, fwd], axis=0)          # world -> camera, z forward, y down
        Rw = _rot_a_to_b(np.array([0.0, 0.0, 1.0]), ray_c) @ R0
        tw = -Rw @ pos
        poses_w.append((Rw, tw))
    # re-base on camera 0
    R0w, t0w = poses_w[0]
    poses = []
    for Rw, tw in poses_w:
        R = Rw @ R0w.T
        t = tw - R @ t0w
        poses.append({"R": R, "t": t})
    centre = R0w @ np.zeros(3) + t0w                        # the ring centre in camera-0 coordinates
    if lenses is None:
        cams = [{"intrinsic_matrix": K.tolist(), "distortion_coef": dist} for _ in range(n_cams)]
        Fs = [fundamental_from_poses(poses[0], poses[i], K, K).tolist() for i in range(1, n_cams)]
        return {"camera_params": cams, "poses": poses, "Fs": Fs, "W": W, "H": H, "centre": centre}
    Ks = [np.asarray(k, dtype=np.float64) for k, _ in lenses]
    cams = [{"intrinsic_matrix": k.tolist(), "distortion_coef": list(np.asarray(d, dtype=np.float64))} for k, (_, d) in zip(Ks, lenses)]
    Fs = [fundamental_from_poses(poses[0], poses[i], Ks[0], Ks[i]).tolist() for i in range(1, n_cams)]
    return {"camera_params": cams, "poses": poses, "Fs": Fs, "W": W, "H": H, "centre": centre, "per_camera_lens": True}


def shipped_rig(W=640, H=480):
    """C1: the reference's own 2-camera calibration, as-is."""
    return {"camera_params": shipped_camera_params(2), "poses": shipped_poses(),
            "Fs": [[list(r) for r in SHIPPED_F], [list(r) for r in SHIPPED_F]], "W": W, "H": H,
            "centre": np.array([0.29, 0.37, -2.06])}


def sample_markers(rig, n_markers, rng, spread=0.45, min_sep_px=56.0, margin=40.0, tries=200):
    """3-D marker positions (camera-0 coordinates) visible in every view; best-effort pixel separation."""
    lens = [camera_lens(rig, c) for c in range(len(rig["poses"]))]
    W, H = rig["W"], rig["H"]
    out = []
    proj = []
    for _ in range(n_markers):
        best = None
        for k in range(tries):
            X = rig["centre"] + rng.uniform(-spread, spread, 3)
            uv = np.stack([project_distorted(X, p, *lens[c])[0] for c, p in enumerate(rig["poses"])])
            if (uv[:, 0] < margin).any() or (uv[:, 0] > W - margin).any() or \
               (uv[:, 1] < margin).any() or (uv[:, 1] > H - margin).any():
                continue
            if best is None:
                best = (X, uv)
            if proj:
                d = np.sqrt(((np.stack(proj) - uv[None]) ** 2).sum(-1))
                if d.min() < min_sep_px and k < tries - 1:
                    continue
            best = (X, uv)
            break
        if best is None:
            raise RuntimeError("rig cannot see the marker volume")
        out.append(best[0])
        proj.append(best[1])
    return np.array(out)


def marker_pixels(rig, X):
    """(C, M, 2) float64 ideal (distorted) pixel centres of markers X (M,3)."""
    return np.stack([project_distorted(X, p, *camera_lens(rig, c)) for c, p in enumerate(rig["poses"])])


def gaussian_kernel1d(sigma=1.2):
    ks = int(round(sigma * 6 + 1)) | 1
    x = np.arange(ks) - ks // 2
    k = np.exp(-(x * x) / (2 * sigma * sigma))
    return (k / k.sum()).astype(np.float64)


def render_frame(H, W, centres, radii, rng, sigma=1.2):
    """One uint8 frame: U[0,40) background, discs of 255, Gaussian blur (numpy, reflect-101 border)."""
    img = rng.integers(0, 40, (H, W)).astype(np.float64)
    for (cx, cy), r in zip(centres, radii):
        x0, x1 = int(max(0, np.floor(cx - r - 1))), int(min(W, np.ceil(cx + r + 2)))
        y0, y1 = int(max(0, np.floor(cy - r - 1))), int(min(H, np.ceil(cy + r + 2)))
        if x1 <= x0 or y1 <= y0:
            continue
        yy, xx = np.mgrid[y0:y1, x0:x1]
        m = (xx - cx) ** 2 + (yy - cy) ** 2 <= r * r
        img[y0:y1, x0:x1][m] = 255.0
    k = gaussian_kernel1d(sigma)
    h = len(k) // 2
    p = np.pad(img, h, mode="reflect")
    tmp = sum(k[i] * p[:, i:i + W] for i in range(len(k)))
    out = sum(k[i] * tmp[i:i + H, :] for i in range(len(k)))
    return np.clip(np.rint(out), 0, 255).astype(np.uint8)


def render_frameset(rig, X, radii, rng):
    """One synchronized frame-set: (C,H,W) uint8 for markers X with per-camera disc radii (C,M)."""
    uv = marker_pixels(rig, X)
    return np.stack([render_frame(rig["H"], rig["W"], uv[c], radii[c], rng) for c in range(len(rig["poses"]))])


def config_rig(name):
    """The rig of a BASELINE.json config: 'c1' (shipped 2-cam 640x480), 'c3' (6 x 1440x1080), 'c4' (16 x 2048^2)."""
    if name == "c1":
        return shipped_rig(640, 480)
    if name == "c3":
        return ring_rig(6, 1440, 1080, radius=6.0)
    if name == "c4":
        return ring_rig(16, 2048, 2048, radius=6.0)
    if name == "c5":
        return ring_rig(8, 2048, 2048, radius=6.0)
    raise ValueError(name)


def config_markers(name, rig, rng):
    if name == "c1":
        return np.array(C1_MARKERS, dtype=np.float64)
    n = {"c3": 32, "c4": 128, "c5": 128}[name]
    return sample_markers(rig, n, rng, spread={"c3": 0.42, "c4": 0.55, "c5": 0.55}[name])


# ----------------------------------------------------------------------------------------------
# Device-side generator for the bench (torch tensors; data plumbing only)
# ----------------------------------------------------------------------------------------------
def disc_stamps(radii=range(14, 23), sigma=1.2, side=57):
    """Pre-blurred disc patches [len(radii), side, side] uint8 (centre at side//2)."""
    k = gaussian_kernel1d(sigma)
    h = len(k) // 2
    out = []
    c = side // 2
    yy, xx = np.mgrid[0:side, 0:side]
    for r in radii:
        img = np.where((xx - c) ** 2 + (yy - c) ** 2 <= r * r, 255.0, 0.0)
        p = np.pad(img, h, mode="constant")
        tmp = sum(k[i] * p[:, i:i + side] for i in range(len(k)))
        o = sum(k[i] * tmp[i:i + side, :] for i in range(len(k)))
        out.append(np.clip(np.rint(o), 0, 255).astype(np.uint8))
    return np.stack(out)


def render_batch_torch(H, W, centres_px, radius_idx, seed, device, stamps=None, out=None):
    """Frames [n,H,W] uint8 on `device`: U[0,40) background, max-composited pre-blurred disc stamps.

    centres_px: int64 tensor [n, M, 2] (x, y) integer disc centres; radius_idx: int64 [n, M] index into stamps;
    seed: one int for the batch or a list of n ints (per-frame background noise).
    A cheaper on-device variant of render_frame (the blur is applied to the discs only); every arm of the
    bench consumes the same frames, so only determinism matters here.
    """
    import torch
    if stamps is None:
        stamps = torch.from_numpy(disc_stamps()).to(device)
    n, M, _ = centres_px.shape
    side = stamps.shape[-1]
    g = torch.Generator(device=device)
    if out is None:
        out = torch.empty((n, H, W), dtype=torch.uint8, device=device)
    if isinstance(seed, (list, tuple)):                      # one seed per frame: a frame does not depend on its batch
        for i, sd in enumerate(seed):
            g.manual_seed(int(sd))
            out[i].copy_(torch.randint(0, 40, (H, W), dtype=torch.uint8, device=device, generator=g))
    else:
        g.manual_seed(int(seed))
        out.copy_(torch.randint(0, 40, (n, H, W), dtype=torch.uint8, device=device, generator=g))
    d = torch.arange(side, device=device) - side // 2
    ys = centres_px[:, :, 1, None, None] + d[None, None, :, None]           # [n,M,side,1]
    xs = centres_px[:, :, 0, None, None] + d[None, None, None, :]           # [n,M,1,side]
    ok = (ys >= 0) & (ys < H) & (xs >= 0) & (xs < W)
    lin = (torch.arange(n, device=device)[:, None, None, None] * H + ys.clamp(0, H - 1)) * W + xs.clamp(0, W - 1)
    val = stamps[radius_idx]                                                 # [n,M,side,side]
    sel = ok & (val > 40)
    flat = out.view(-1)
    # amax handles overlapping stamps deterministically
    flat.scatter_reduce_(0, lin[sel], val[sel], reduce="amax", include_self=True)
    return out


def save_rig_json(rig, path):
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        json.dump({"camera_params": rig["camera_params"],
                   "poses": [{"R": np.asarray(p["R"]).tolist(), "t": np.asarray(p["t"]).tolist()} for p in rig["poses"]],
                   "Fs": [np.asarray(F).tolist() for F in rig["Fs"]], "W": rig["W"], "H": rig["H"],
                   "centre": np.asarray(rig["centre"]).tolist()}, f)
