#!/usr/bin/env python
"""Contract benchmark of the capture hot path (see BASELINE.json / SURVEY.md section 8d).

    python bench.py [--gpus N --steps K --warmup W]             this repo (libmocap_b200.so, sm_100a)
    python bench.py --impl reference [...]                       the reference's CPU path (OpenCV/NumPy) on the host cores

Workload (config.workload): BASELINE config 4 -- 16-camera 2048x2048 rig, 128 markers, full detect + match +
triangulate.  One step = one batch of F0*N synchronized frame-sets: every rank detects its 16/N cameras of all
frame-sets, ONE all-gather moves the centroid records, every rank matches + triangulates its F0 frame-sets.
Per-GPU work is constant in N (weak scaling).  value = frames/s over all ranks, inputs resident in HBM; e2e = the
same through the public API from pinned host memory (H2D of the frames and D2H of the results inside the timed region).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

from mocapv2_b200 import synth as S  # noqa: E402

CONFIG = "c4"
N_MARKERS = 128
MAX_BLOBS = 160
MAX_GROUPS = 64            # candidate groups evaluated per root (cap policy, flagged per frame-set)
MAX_CAND = 8               # MOCAP_MAX_CAND
JITTER = 0.01              # metres, per frame-set (SURVEY 8d)
SPREAD = 0.95              # half-extent (m) of the marker volume around the rig centre: fills the 2048x2048 views


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 300 = more than 0.5 s of device time; reference arm: 20)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frame-sets", type=int, default=64, help="frame-sets per GPU per step (F0)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-sample", type=int, default=1, help="frame-sets timed for cpu_baseline (0 = skip)")
    ap.add_argument("--in-flight", type=int, default=2, help="steps in flight in the timed loop (each on its own lane: stream, detection pipe, buffers)")
    ap.add_argument("--no-scan-token", action="store_true", help="let the scans of the lanes run side by side (A/B of StepsInFlight.scan_token)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-geometry", action="store_true", help="skip the config-5 geometry sweep")
    ap.add_argument("--no-extra", action="store_true", help="skip front step, _find_dot latency and the C1 / C3 configs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to DIR/<name>.npy (float64; rank 0's frame-sets and cameras)")
    a = ap.parse_args()
    if a.steps is None:
        a.steps = 300 if a.impl == "b200" else 20
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


# ---------------------------------------------------------------------------------------------------------------------
# synthetic rig + frames (data plumbing)
# ---------------------------------------------------------------------------------------------------------------------
def make_scene(n_frame_sets, config=CONFIG, n_markers=N_MARKERS, spread=SPREAD, seed=S.SEED0 + 4000):
    """Marker positions per frame-set and their integer pixel centres per camera: (rig, centres [FS, C, M, 2] int64, radius idx).

    Everything a frame-set needs is drawn from ITS OWN generator (seed + 1 + s), so frame-set s is the same scene whatever the
    number of frame-sets of the run: the first F0 frame-sets of an N-GPU run are the frame-sets of the 1-GPU run and the
    output checksum of rank 0 can be compared across N."""
    rig = S.config_rig(config)
    rng = np.random.default_rng(seed)
    # markers spread over the whole commonly visible volume, >= 2r+12 px apart in every view where that is achievable
    # (with 16 views and 128 markers some views inevitably show touching blobs; the detector handles them)
    X0 = S.sample_markers(rig, n_markers, rng, spread=spread, min_sep_px=56.0, margin=40.0, tries=300)
    C = len(rig["poses"])
    cen = np.empty((n_frame_sets, C, n_markers, 2), dtype=np.int64)
    radius_idx = np.empty((n_frame_sets, C, n_markers), dtype=np.int64)
    for s in range(n_frame_sets):
        rs = np.random.default_rng(seed + 1 + s)
        X = X0 + rs.uniform(-JITTER, JITTER, X0.shape)
        cen[s] = np.rint(S.marker_pixels(rig, X)).astype(np.int64)
        radius_idx[s] = rs.integers(0, 9, (C, n_markers))
    return rig, cen, radius_idx


def render_local(rig, cen, radius_idx, cam_begin, cams_local, device):
    """Frames [FS, cams_local, H, W] of this rank's cameras; the background noise of a frame is seeded by (frame-set, camera)
    alone, so a frame does not depend on how the cameras are sharded."""
    import torch
    FS = cen.shape[0]
    H, W = rig["H"], rig["W"]
    frames = torch.empty((FS, cams_local, H, W), dtype=torch.uint8, device=device)
    stamps = torch.from_numpy(S.disc_stamps()).to(device)
    for s in range(FS):
        c = torch.from_numpy(cen[s, cam_begin:cam_begin + cams_local]).to(device)
        r = torch.from_numpy(radius_idx[s, cam_begin:cam_begin + cams_local]).to(device)
        seeds = [1000 + s * 64 + cam_begin + k for k in range(cams_local)]
        S.render_batch_torch(H, W, c, r, seeds, device, stamps=stamps, out=frames[s])
    return frames


# ---------------------------------------------------------------------------------------------------------------------
# clocks (B200_PROFILING.md: sample nvidia-smi DURING the timed region)
# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            p = [x.strip() for x in line.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for nm, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm (reference's OpenCV/NumPy path on the host cores)
# ---------------------------------------------------------------------------------------------------------------------
def cpu_frame_sets(rig, host_frames, n_sets, threads):
    """Time the CPU path on n_sets frame-sets ([n, C, H, W] uint8 numpy).  Returns (seconds, frames, object points)."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import cv2_port
    if not cv2_port.available():
        return None
    pts_total = 0
    with ThreadPoolExecutor(max_workers=threads) as pool:
        t0 = time.perf_counter()
        for s in range(n_sets):
            _, obj, _ = cv2_port.frame_set(host_frames[s], rig, N_MARKERS, max_cand=MAX_CAND, max_groups=MAX_GROUPS, pool=pool)
            pts_total += len(obj)
        dt = time.perf_counter() - t0
    return dt, n_sets * host_frames.shape[1], pts_total


def host_render(rig, cen, radius_idx, n_sets):
    """CPU rendering of the same frames the device generator makes (bit-identical recipe is not required: both arms
    of a run consume their own copy of the same scene; the CPU arm uses the torch generator on the CPU device)."""
    import torch
    return render_local(rig, cen[:n_sets], radius_idx[:n_sets], 0, len(rig["poses"]), torch.device("cpu")).numpy()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    rig, cen, ridx = make_scene(1)
    frames = host_render(rig, cen, ridx, 1)
    from oracle import cv2_port
    if not cv2_port.available():
        emit({"impl": "reference", "unavailable": "opencv (cv2) is not importable on this host"})
        return 0
    cvt = None
    try:
        import cv2
        cv2.setNumThreads(threads)
        cvt = cv2.getNumThreads()
    except Exception:
        pass
    for _ in range(args.warmup):
        cpu_frame_sets(rig, frames, 1, threads)
    t = 0.0
    n_frames = 0
    pts = 0
    for _ in range(args.steps):
        dt, nf, np_ = cpu_frame_sets(rig, frames, 1, threads)
        t += dt
        n_frames += nf
        pts += np_
    value = n_frames / t
    line = {
        "impl": "reference", "metric": "frames/s (detect+match+triangulate, 16-camera 2048x2048 rig, 128 markers)",
        "value": value, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8 (detection) / f64 (geometry)", "data": "synthetic",
        "points_per_s": pts / t,
        "config": workload_config(1, 1, sample="1 frame-set (16 frames) per step"),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "os_cpu_count": os.cpu_count(),
                         "cv2_num_threads": cvt, "kind": "port",
                         "sample": "1 frame-set (16 frames 2048x2048) per step; OpenCV calls of lib/ImageOperations.py:33-65 "
                                   "(numba blur -> integer restatement) + lib/Helpers.py:178-280 control flow in NumPy with the "
                                   f"same candidate cap (max_cand {MAX_CAND}, max_groups {MAX_GROUPS}); frames over a {threads}-thread pool"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


def workload_config(n, f0, sample=None):
    cfg = {"workload": "BASELINE config 4: 16 cameras 2048x2048 u8, 128 markers, detect+match+triangulate",
           "cameras": 16, "frame": [2048, 2048], "markers": N_MARKERS, "frame_sets_per_gpu_per_step": f0,
           "frames_per_step": 16 * f0 * n, "parallelism": f"cameras sharded x{n} for detection, frame-sets sharded x{n} for geometry, 1 shard exchange (records stored straight into the matching rank's buffer over NVLink + a barrier; NCCL send/recv where peer memory is unavailable)",
           "group_cap": {"max_cand": MAX_CAND, "max_groups": MAX_GROUPS},
           "l2": "inputs per step (>=1 GB) exceed the 126 MB L2; the same resident batch is re-read every step"}
    if sample:
        cfg["sample"] = sample
    return cfg


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
def _events(n):
    import torch
    return [torch.cuda.Event(enable_timing=True) for _ in range(n)]


def _hash_tensors(*ts):
    import hashlib
    h = hashlib.sha1()
    for t in ts:
        h.update(np.ascontiguousarray(t.cpu().numpy()).tobytes())
    return h.hexdigest()[:16]


def _load_traffic():
    try:
        return json.load(open(os.path.join(REPO, "profiles", "traffic.json")))
    except Exception:
        return {}


def _parity_check(rig, frames, det, corr, cams_local):
    """GPU results of frame-set 0 against the CPU arm's (oracle/cv2_port.py) on the SAME frames, the same caps."""
    from oracle import cv2_port
    if not cv2_port.available():
        return {"checked": False, "why": "opencv not importable on this host"}
    host = frames[0].cpu().numpy()
    pts, obj, ipa = cv2_port.frame_set(host, rig, N_MARKERS, max_cand=MAX_CAND, max_groups=MAX_GROUPS)
    gpu_pts = [det.points(c) for c in range(cams_local)]
    cen_ok = gpu_pts == [[list(map(int, q)) if q[0] is not None else q for q in p] for p in pts]
    nv, no = int(corr.n_valid[0]), int(corr.n_obj[0])
    img = corr.img[0, :nv].cpu().numpy()
    got = corr.obj[0, :no].cpu().numpy()
    ipa = np.asarray(ipa)
    pairs_ok = bool(ipa.shape == img.shape and np.array_equal(ipa, img))
    obj = np.asarray(obj, dtype=np.float64).reshape(-1, 3)
    rel = None
    # the returned object points are sorted by mean error; FP32 errors of neighbouring roots may swap places, so compare as sets
    if len(obj) == len(got) and len(obj):
        d = np.linalg.norm(got[:, None, :] - obj[None, :, :], axis=2)
        rel = float((d.min(axis=1) / np.linalg.norm(got, axis=1)).max())
    return {"checked": True, "frame_set": 0, "centroid_lists_equal": bool(cen_ok), "pairs_equal": pairs_ok,
            "n_centroids": int(sum(len(p) for p in gpu_pts)), "n_roots": nv, "n_object_points": no,
            "object_points_max_rel_err": rel, "tolerance": 1e-4,
            "ok": bool(cen_ok and pairs_ok and rel is not None and rel < 1e-4)}


DUMP_BYTES = 64_000_000


def _dump_outputs(out_dir, det, corr, cams_local):
    """Write the results of one step as float64 .npy files, one per array the caller receives: the detection of rank 0's cameras
    (det_xy [FS, cams, max_blobs, 2], det_count, det_flags) and the matching of its frame-sets (corr_obj, corr_n_obj, corr_img,
    corr_n_valid, corr_err, corr_flags), frame-set s in row s.  Entries past a count are zeroed (the kernels leave them
    unspecified), so two builds compare element for element.  Above DUMP_BYTES a fixed seeded sample of the frame-sets is written;
    frame_sets.npy names the frame-sets the rows are."""
    S = corr.n_obj.shape[0]
    host = lambda t: t.cpu().numpy().astype(np.float64)
    out = {"det_xy": host(det.xy).reshape(-1, cams_local, *det.xy.shape[1:])[:S],
           "det_count": host(det.count).reshape(-1, cams_local)[:S], "det_flags": host(det.flags).reshape(-1, cams_local)[:S],
           "corr_obj": host(corr.obj), "corr_n_obj": host(corr.n_obj), "corr_img": host(corr.img),
           "corr_n_valid": host(corr.n_valid), "corr_err": host(corr.err), "corr_flags": host(corr.flags)}
    slots = np.arange(out["det_xy"].shape[2])
    out["det_xy"][slots[None, None, :] >= out["det_count"][..., None]] = 0
    rows = np.arange(corr.obj.shape[1])[None, :] >= out["corr_n_valid"][:, None]
    out["corr_img"][rows] = 0
    out["corr_err"][rows] = 0
    out["corr_obj"][np.arange(corr.obj.shape[1])[None, :] >= out["corr_n_obj"][:, None]] = 0
    keep = min(S, (DUMP_BYTES - 4096) // (sum(a.nbytes for a in out.values()) // S + 8))     # (4096: the .npy headers)
    fs = np.arange(S) if keep == S else np.sort(np.random.default_rng(0).choice(S, keep, replace=False))
    out = {k: a[fs] for k, a in out.items()}
    out["frame_sets"] = fs.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _time_loop(fn, reps, warm=3):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = _events(2)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def _extra_config(eng, name, n_markers, spread, frame_sets, device):
    """frames/s and points/s of another BASELINE config on one GPU (resident inputs): detection chain fraction included."""
    import torch
    from mocapv2_b200.pipeline import CapturePipeline
    rig, cen, ridx = make_scene(frame_sets, config=name, n_markers=n_markers, spread=spread, seed=S.SEED0 + 7000)
    mb = max(8, n_markers + n_markers // 4)
    pipe = CapturePipeline(eng, rig, max_blobs=mb, obj_count=n_markers, max_groups=MAX_GROUPS)
    frames = render_local(rig, cen, ridx, 0, pipe.cams_local, device)
    C = pipe.cams_local
    H, W = rig["H"], rig["W"]
    corr = [None]
    marks = []

    def step(rec=False):
        ev = _events(3) if rec else None
        if rec:
            ev[0].record()
        det = pipe.detect(frames)
        if rec:
            ev[1].record()
        xy, count = pipe.exchange(det, frame_sets)
        corr[0] = eng.correspond(xy, count, pipe.Fs, pipe.cams, obj_count=n_markers, max_groups=MAX_GROUPS, out=corr[0])
        if rec:
            ev[2].record()
            marks.append(ev)
        return det

    ms = _time_loop(step, 10)
    for _ in range(5):
        det = step(rec=True)
    torch.cuda.synchronize()
    det_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in marks]))
    n = frame_sets * C
    out = {"workload": f"{name}: {C} cameras {W}x{H}, {n_markers} markers, {frame_sets} frame-sets per step",
           "ms_per_step": ms, "frames_per_s": n / (ms * 1e-3), "points_per_s": float(corr[0].n_valid.sum().item()) / (ms * 1e-3),
           "detect_ms": det_ms, "detect_gbs": n * H * W / (det_ms * 1e-3) / 1e9,
           "centroids_per_frame": float(det.count.float().mean().item()), "flags_or": int(det.flags.max().item()) & 63,
           "frame_sets_with_group_cap": int((corr[0].flags & 1).sum().item()), "overlapped_detection": eng.last_pipe_info}
    del frames
    return out


def _bundle_adjustment_timing(eng):
    """bundle_adjustment on jsons/before_ba_extrinsics.json + image_points.json of the reference (tests/golden/kat_bundle_adjustment.npz):
    this repo (scipy TRF on the host, one fused GPU launch per optimiser iteration) against the same optimiser over the CPU restatement
    of the reference's residual (oracle/restate.py: numpy SVD + the cv.projectPoints restatement)."""
    from scipy import optimize
    from scipy.spatial.transform import Rotation
    from mocapv2_b200 import engine as E
    from mocapv2_b200.lib import Helpers as Hh
    from oracle import restate as R
    z = np.load(os.path.join(REPO, "tests", "golden", "kat_bundle_adjustment.npz"))
    poses = [{"R": z["R_before"][i], "t": z["t_before"][i]} for i in range(2)]
    cp = S.shipped_camera_params(2)
    E.set_default_engine(eng)
    saved = Hh.camera_params
    Hh.camera_params = np.array(cp)
    try:
        Hh.bundle_adjustment(z["image_points"], poses)                      # warm-up (table-free path, first launches)
        t0 = time.perf_counter()
        out = Hh.bundle_adjustment(z["image_points"], poses)
        ours = time.perf_counter() - t0
        stats = dict(getattr(Hh.bundle_adjustment, "last_stats", {}))
    finally:
        Hh.camera_params = saved
    err = float(max(np.abs(np.asarray(out[1]["R"]) - z["R_json"][1]).max(), np.abs(np.asarray(out[1]["t"]).ravel() - z["t_json"][1]).max()))
    groups = [list(map(list, g)) for g in z["image_points"]]

    def residual(params):
        ps = Hh.params_to_camera_poses(params, 2)
        X = R.triangulate_points(groups, ps, cp)
        return R.reprojection_errors(groups, X, ps, cp).astype(np.float32)

    x0 = np.concatenate([Rotation.from_matrix(poses[1]["R"]).as_rotvec(), np.asarray(poses[1]["t"]).ravel()])
    t0 = time.perf_counter()
    res = optimize.least_squares(residual, x0, verbose=0, loss="linear", method="trf", ftol=1E-5, xtol=1E-15)
    cpu = time.perf_counter() - t0
    ref_pose = Hh.params_to_camera_poses(res.x)
    cpu_err = float(np.abs(np.asarray(ref_pose[1]["R"]) - z["R_json"][1]).max())
    return {"fixture": "the reference's jsons/before_ba_extrinsics.json + image_points.json (54 points, 2 cameras) -> after_ba_extrinsics.json",
            "b200_s": ours, "max_abs_diff_to_after_ba_json": err, "launches": stats.get("launches"), "hypotheses_evaluated": stats.get("hypotheses"),
            "nfev": stats.get("nfev"), "njev": stats.get("njev"),
            "cpu_port_s": cpu, "cpu_port_max_abs_diff_R": cpu_err, "speedup": cpu / ours,
            "note": "same scipy optimiser and settings on both sides; the unmodified reference function took 3.8-4.6 s in the build container "
                    "(python, cv.projectPoints + scipy svd per point and evaluation)"}


def run_b200(args):
    import torch
    import torch.distributed as dist
    from mocapv2_b200.engine import CaptureEngine
    from mocapv2_b200.pipeline import CapturePipeline, StepsInFlight

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device(f"cuda:{local}")
    host_binding = None
    if world > 1:
        # a rank next to its GPU: CPU affinity + preferred memory node before any pinned buffer exists (N = 1 keeps every host
        # core for the cpu_baseline leg)
        from mocapv2_b200 import hostbind
        host_binding = hostbind.bind_to_gpu(local)
        dist.init_process_group("nccl", device_id=device)
    N = world
    F0 = args.frame_sets
    FS = F0 * N
    rig, cen, ridx = make_scene(FS)
    eng = CaptureEngine(device)
    pipe = CapturePipeline(eng, rig, max_blobs=MAX_BLOBS, obj_count=N_MARKERS, max_groups=MAX_GROUPS)
    frames = render_local(rig, cen, ridx, pipe.cam_begin, pipe.cams_local, device)
    n_local = FS * pipe.cams_local
    H, W = rig["H"], rig["W"]
    flight = StepsInFlight(pipe, args.in_flight)
    if args.no_scan_token:
        flight.scan_token = False
    corr_outs = {}

    def step_on(lane, marks=None):
        if marks is not None:
            ev = _events(4)
            ev[0].record()
        det = lane.detect(frames)
        if marks is not None:
            ev[1].record()
        xy, count = lane.exchange(det, FS)
        if marks is not None:
            ev[2].record()
        corr = corr_outs[id(lane)] = lane.eng.correspond(xy, count, lane.Fs, lane.cams, obj_count=N_MARKERS, max_groups=MAX_GROUPS,
                                                         out=corr_outs.get(id(lane)))
        if marks is not None:
            ev[3].record()
            marks.append(ev)
        return det, corr

    def step(marks=None):
        """one step on the next lane (its own stream when several steps are in flight)"""
        lane, st = flight.next_lane()
        if st is None:
            return step_on(lane, marks)
        with torch.cuda.stream(st):
            return step_on(lane, marks)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def rank_max(x):
        t = torch.tensor([float(x)], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                     # nvidia-smi needs ~100 ms to deliver its first sample: start before the warm-up
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    launches0 = eng.launches
    marks = []
    ev0, ev1 = _events(2)
    barrier()
    ev0.record()
    flight.fork()                           # the lanes start behind ev0 ...
    for k in range(args.steps):
        det, corr = step(marks)
    flight.join()                           # ... and ev1 lies behind the last step of every lane
    ev1.record()
    gpu_launches = eng.launches - launches0
    barrier()
    if args.dump_outputs and rank == 0:     # before the steps below reuse the lanes' result buffers
        _dump_outputs(args.dump_outputs, det, corr, pipe.cams_local)
    # nvidia-smi delivers a sample every ~50-100 ms: if the timed region was shorter than a second keep the same step loop
    # running (untimed) so that the clock record is taken under this very load
    # (the number of extra steps follows from the all-reduced time: every rank runs the same number of steps and lane turns)
    ms_timed = rank_max(ev0.elapsed_time(ev1))
    for _ in range(int(max(0.0, 1000.0 - ms_timed) / max(ms_timed / args.steps, 1e-3)) + 1):
        step()
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "warm-up + timed region (+ the same step loop, untimed, up to 1 s in total)"
    barrier()
    ms_total = rank_max(ev0.elapsed_time(ev1))
    phase = {"detect_ms": rank_max(np.mean([e[0].elapsed_time(e[1]) for e in marks])),
             "exchange_ms": rank_max(np.mean([e[1].elapsed_time(e[2]) for e in marks])),
             "geometry_ms": rank_max(np.mean([e[2].elapsed_time(e[3]) for e in marks])),
             "note": "CUDA events on the step's stream around detect / exchange / match+triangulate, mean over the timed steps, max over ranks"}
    pipe_info = eng.last_pipe_info

    # ---- the detection chain alone at the bench's own operating point: K detect calls, `in_flight` of them in flight (lanes) --------
    def detect_rate(reps, lanes_on):
        a_, b_ = _events(2)
        barrier()
        a_.record()
        if lanes_on:
            flight.fork()
        for _ in range(reps):
            lane, st = flight.next_lane() if lanes_on else (pipe, None)
            if st is None:
                lane.detect(frames)
            else:
                with torch.cuda.stream(st):
                    lane.detect(frames)
        if lanes_on:
            flight.join()
        b_.record()
        barrier()
        return rank_max(a_.elapsed_time(b_)) / reps
    reps_d = 2 * flight.depth * max(5, min(args.steps, 50) // (2 * flight.depth))
    detect_rate(2 * flight.depth, True)
    detect_rate(3, False)                   # (the caller's stream gets its own workspace on first use)
    phase["detect_in_flight_ms"] = detect_rate(reps_d, True)
    lane_pipe = dict(pipe.engine_pipe)
    pipe.engine_pipe = {"workers": 6, "chunks": 8}          # the single call's own best split (the lanes use fewer, larger chunks)
    detect_rate(3, False)
    phase["detect_single_call_ms"] = detect_rate(reps_d, False)
    pipe.engine_pipe = lane_pipe
    phase["steps_in_flight"] = flight.depth
    phase["note"] += ("; with several steps in flight the per-step marks are latencies under overlap -- detect_in_flight_ms is the time per detect "
                      "call of a loop of detect calls alone with the same number in flight, detect_single_call_ms one call after the other")

    # ---- the stages one after the other (the same kernels without overlap), and the overlapped call's timeline -------------------
    timers = [eng.stage_timer() for _ in range(5)]
    for t in timers:
        pipe.detect(frames, timer=t)                          # a timer selects the one-shot call: stages are separable there
    torch.cuda.synchronize()
    stage_ms = {}
    for t in timers:
        for k, v in eng.stage_timer_read(t).items():
            stage_ms.setdefault(k, []).append(v)
    stage_avg = {k: float(np.mean(v)) for k, v in stage_ms.items()}
    serial_ms = sum(stage_avg.values())
    timeline = None
    if pipe_info is not None:
        pipe.detect(frames, timeline=True)
        torch.cuda.synchronize()
        timeline = eng.pipe_timeline()
        flat = frames.view(-1, H, W)
        tma_scan_ms = _time_loop(lambda: eng.scan_cells(flat, pipe.K0, pipe.dist0, variant=1), 10)
    else:
        tma_scan_ms = None
    det, corr = step()
    torch.cuda.synchronize()

    # work accounting + output checksum of rank 0 (its geometry shard = frame-sets [0, F0): the same scene at every N)
    n_pts = torch.tensor([float(corr.n_valid.sum().item()), float((corr.flags & 1).sum().item()), float(det.count.sum().item())],
                         device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(n_pts)
    frames_per_step = 16 * F0 * N
    value = frames_per_step * args.steps / (ms_total * 1e-3)
    points_per_step = float(n_pts[0].item())
    checksum = None
    if rank == 0:
        nv = corr.n_valid.cpu().numpy()
        no = corr.n_obj.cpu().numpy()
        img = corr.img.cpu().numpy()
        obj = corr.obj.cpu().numpy()
        import hashlib
        h = hashlib.sha1()
        h.update(nv.tobytes()); h.update(no.tobytes())
        for s_ in range(len(nv)):
            h.update(np.ascontiguousarray(img[s_, :nv[s_]]).tobytes())
            h.update(np.ascontiguousarray(obj[s_, :no[s_]]).tobytes())
        checksum = {"sha1_16": h.hexdigest()[:16], "frame_sets": [0, F0],
                    "over": "rank 0's geometry shard: n_valid, n_obj, matched image points (all cameras, i.e. every rank's centroids) and object "
                            "points (raw float64 bits) of frame-sets [0, F0) -- the same scene at every N, so the value must not change with N"}

    # ---- end to end: pinned host frames -> H2D -> pipeline -> D2H of the results, every step ----------------------------
    e2e = None
    if not args.no_e2e:
        host = torch.empty(frames.shape, dtype=torch.uint8, pin_memory=True)
        host.copy_(frames)
        stage_dev = torch.empty_like(frames)
        host_obj = torch.empty(corr.obj.shape, dtype=corr.obj.dtype, pin_memory=True)
        host_nobj = torch.empty(corr.n_obj.shape, dtype=corr.n_obj.dtype, pin_memory=True)
        host_cnt = torch.empty(det.count.shape, dtype=det.count.dtype, pin_memory=True)
        copy_stream = torch.cuda.Stream(device)
        chunks = max(1, min(8, FS))
        bounds = np.linspace(0, FS, chunks + 1).astype(int)
        eng2 = CaptureEngine(device)
        eng2._tables = eng._tables
        full_buf = pipe._buffers(n_local)
        full = type(det)(full_buf.xy, full_buf.count, full_buf.flags)      # the same tensors, filled chunk by chunk below (one-shot calls)
        cl = pipe.cams_local
        dets = [type(det)(full.xy[bounds[c] * cl:bounds[c + 1] * cl], full.count[bounds[c] * cl:bounds[c + 1] * cl],
                          full.flags[bounds[c] * cl:bounds[c + 1] * cl]) for c in range(chunks)]

        e2e_corr = [None]

        def e2e_step():
            # chunked: the copy of chunk k+1 overlaps detection of chunk k (copy stream + compute stream); the detection of a chunk
            # writes its slice of the pipeline's output buffers, nothing is concatenated
            evs = []
            for c in range(chunks):
                with torch.cuda.stream(copy_stream):
                    stage_dev[bounds[c]:bounds[c + 1]].copy_(host[bounds[c]:bounds[c + 1]], non_blocking=True)
                    e = torch.cuda.Event()
                    e.record(copy_stream)
                    evs.append(e)
            for c in range(chunks):
                torch.cuda.current_stream().wait_event(evs[c])
                fr = stage_dev[bounds[c]:bounds[c + 1]].view(-1, H, W)
                eng2.detect(fr, pipe.K0, pipe.dist0, max_blobs=MAX_BLOBS, out=dets[c])
            xy, count = pipe.exchange(full, FS)
            co = e2e_corr[0] = eng.correspond(xy, count, pipe.Fs, pipe.cams, obj_count=N_MARKERS, max_groups=MAX_GROUPS, out=e2e_corr[0])
            host_obj.copy_(co.obj, non_blocking=True)
            host_nobj.copy_(co.n_obj, non_blocking=True)
            host_cnt.copy_(full.count, non_blocking=True)
            torch.cuda.current_stream().synchronize()          # the caller reads the result on the host
            return int(host_nobj.sum())

        def copy_only():
            with torch.cuda.stream(copy_stream):
                stage_dev.copy_(host, non_blocking=True)
            copy_stream.synchronize()

        e2e_step()
        barrier()
        l0 = eng.launches                                  # (the library counts its launches per process: both engines share the counter)
        t0 = time.perf_counter()
        a, b = _events(2)
        a.record()
        for _ in range(args.e2e_steps):
            e2e_step()
        b.record()
        barrier()
        wall = time.perf_counter() - t0
        ems = rank_max(max(a.elapsed_time(b), 0.0))
        # the host link alone: the same pinned bytes, one H2D copy per rank at the same time on every rank (the ceiling of e2e)
        copy_only()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            copy_only()
        t_copy = torch.tensor([time.perf_counter() - t0], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t_copy, op=dist.ReduceOp.MAX)
        copy_s = float(t_copy.item()) / args.e2e_steps
        h2d_bytes = int(frames.numel()) * N
        e2e_val = frames_per_step * args.e2e_steps / (ems * 1e-3)
        ceil_val = frames_per_step / copy_s
        e2e = {"value": e2e_val, "unit": "frames/s",
               "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": int(host_obj.numel() * 8 + host_nobj.numel() * 4 + host_cnt.numel() * 4) * N,
               "steps": args.e2e_steps, "wall_s": wall, "gpu_launches": eng.launches - l0,
               "h2d_copy_only": {"aggregate_gbs": h2d_bytes / copy_s / 1e9, "frames_per_s_ceiling": ceil_val,
                                 "e2e_over_ceiling": e2e_val / ceil_val,
                                 "how": "the step's pinned frames copied H2D on every rank at once, nothing else running (wall clock, max over ranks)"},
               "how": f"pinned host frames -> {chunks} chunked H2D copies on a copy stream overlapped with detection -> shard exchange -> "
                      "match+triangulate -> D2H of object points/counts, host sync every step"}
        del host, stage_dev

    # ---- geometry-only sweep (BASELINE config 5): P 8-view correspondences sharded over the ranks, DLT + reprojection error, FP32 ---
    geometry = None
    if not args.no_geometry:
        rig5 = S.config_rig("c5")
        cams5 = eng.cameras(rig5["poses"], rig5["camera_params"])
        Pm = torch.tensor(cams5.cpu().numpy()[:, :12].reshape(8, 3, 4), device=device)
        sweeps = []
        flops = 140 * 8 + 1609                                     # SURVEY 8d: F(N) = 140 N + 1609 per point
        for P_total in (1_000_000, 10_000_000, 100_000_000):
            P5 = P_total // N
            g5 = torch.Generator(device=device).manual_seed(5 + rank)
            pts5 = torch.empty((P5, 8, 2), device=device, dtype=torch.float32)
            blk = 2_000_000
            for o in range(0, P5, blk):                            # projected in slices: the FP64 intermediates stay small
                m = min(blk, P5 - o)
                X5 = torch.tensor(np.asarray(rig5["centre"]), device=device) + (torch.rand((m, 3), generator=g5, device=device, dtype=torch.float64) - 0.5)
                proj = torch.einsum("cij,pj->pci", Pm, torch.cat([X5, torch.ones((m, 1), device=device, dtype=torch.float64)], dim=1))
                pts5[o:o + m] = torch.floor(proj[..., :2] / proj[..., 2:3]).float()
            del X5, proj
            xyz5 = torch.empty((P5, 3), device=device)
            err5 = torch.empty((P5,), device=device)
            reps = 20 if P_total <= 10_000_000 else 5
            for _ in range(3):
                eng.triangulate(pts5, cams5, xyz=xyz5, err=err5)
            barrier()
            ga, gb = _events(2)
            ga.record()
            for _ in range(reps):
                eng.triangulate(pts5, cams5, xyz=xyz5, err=err5)
            gb.record()
            barrier()
            tms = rank_max(ga.elapsed_time(gb) / reps)
            finite = torch.tensor([float(torch.isfinite(err5).sum().item())], device=device, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(finite)
            sweeps.append({"points": P5 * N, "points_per_rank": P5, "ms": tms, "points_per_s": P5 * N / (tms * 1e-3),
                           "achieved_tflops": P5 * N * flops / (tms * 1e-3) / 1e12, "finite_results": int(finite.item())})
            del pts5, xyz5, err5
        sm_mhz = (clocks or {}).get("sm_max_mhz") or 1965.0
        peak32 = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
        best = max(sweeps, key=lambda r: r["points_per_s"])
        geometry = {"workload": "BASELINE config 5: 8-view DLT triangulation + reprojection error, FP32, points sharded over the ranks, no exchange",
                    "views": 8, "flop_per_point": flops, "sweep": sweeps, "points_per_s": best["points_per_s"],
                    "fp32_peak_tflops_per_gpu": peak32, "frac_of_fp32_pipe": best["achieved_tflops"] / (peak32 * N),
                    "peak_source": "148 SMs x 128 FP32 lanes x 2 x clocks.max.sm per GPU (no tensor cores: tiny independent solves); the fraction is "
                                   "algorithmic flops (SURVEY 8d) / time.  The pipe counters of the same kernel (ncu sm__inst_executed_pipe_fma*) are "
                                   "in profiles/ (r2_ncu_summary.md)"}

    # ---- the step in front of the path: raw Bayer GR sensor frames -> grey (RealtimeTracking_FLIR.py:103-104) ---------------
    front = None
    if rank == 0 and not args.no_extra:
        nb = 256                                                   # 1.07 GB in + 1.07 GB out: larger than L2
        raw = torch.randint(0, 256, (nb, H, W), dtype=torch.uint8, device=device)
        grey = torch.empty_like(raw)
        fms = _time_loop(lambda: eng.bayer_gr2gray(raw, out=grey), 10)
        front = {"workload": f"Bayer GR -> grey, {nb} frames {W}x{H} u8 (bilinear demosaic + BGR2GRAY, bit-identical to OpenCV)",
                 "kernel": "bayer_gr2gray_rows_kernel", "ms": fms, "frames_per_s": nb / (fms * 1e-3),
                 "algorithmic_bytes": 2 * nb * H * W, "achieved_gbs": 2 * nb * H * W / (fms * 1e-3) / 1e9}
        del raw, grey
    # raw sensor frames through front step + detection (what the realtime loop does per frame, RealtimeTracking_FLIR.py:103-105):
    # the step's resident frames read as Bayer GR mosaics -> grey -> centroid lists, one call after the other on one stream
    if front is not None and N == 1:                              # (one GPU: the pipeline's detect call is collective-free only there)
        raw4 = frames                                              # [F0, cams_local, H, W]: any byte image is a valid mosaic
        grey4 = torch.empty_like(raw4)

        cells4 = eng.empty((raw4.shape[0] * raw4.shape[1], (H + 31) // 32, (W + 31) // 32), torch.int32)

        def raw_step_two_passes():                                 # front step, then the detection with its own streaming scan
            eng.bayer_gr2gray(raw4.view(-1, H, W), out=grey4.view(-1, H, W))
            return pipe.detect(grey4)

        def raw_step():                                            # the front step also delivers the detection's hot cell boxes
            eng.bayer_gr2gray_scan(raw4.view(-1, H, W), out=grey4.view(-1, H, W), cellbox=cells4)
            return pipe.detect(grey4, cellbox=cells4)

        det2 = raw_step_two_passes()
        two = (det2.count.clone(), det2.xy.clone())
        rms2 = _time_loop(raw_step_two_passes, 10)
        bms = _time_loop(lambda: eng.bayer_gr2gray_scan(raw4.view(-1, H, W), out=grey4.view(-1, H, W), cellbox=cells4), 10)
        det_raw = raw_step()
        same_as_two = bool(torch.equal(two[0], det_raw.count) and torch.equal(two[1], det_raw.xy))
        rms = _time_loop(raw_step, 10)
        n_raw = raw4.shape[0] * raw4.shape[1]
        raw_par = None
        try:
            from oracle import cv2_port, restate as R_
            if cv2_port.available():
                want = cv2_port.find_dot(R_.bayer_gr_to_gray(raw4[0, 0].cpu().numpy()), rig["camera_params"][0]["intrinsic_matrix"],
                                         rig["camera_params"][0]["distortion_coef"])
                got = det_raw.points(0)
                raw_par = {"frame": 0, "centroid_list_equal": got == want, "n_centroids": 0 if want == [[None, None]] else len(want),
                           "against": "oracle: bayer_gr_to_gray (== cv2.cvtColor BAYER_GR2BGR -> BGR2GRAY, tests/test_oracle_cv2.py) -> cv2_port.find_dot"}
        except ImportError:
            pass
        front["raw_to_centroids"] = {"frames": n_raw, "ms": rms, "frames_per_s": n_raw / (rms * 1e-3),
                                     "how": "mocap_bayer_gr2gray_scan_batch (grey frames + the hot cell boxes of the detection) then the overlapped detection call "
                                            "without its streaming scan (mocap_detect_pipe_set_cellbox) on the same stream, CUDA events, no second call in flight",
                                     "front_step_with_scan_ms": bms,
                                     "two_passes": {"ms": rms2, "how": "mocap_bayer_gr2gray_batch then the detection call with its own scan",
                                                    "same_results": same_as_two},
                                     "parity_check": raw_par}
        del grey4, det_raw, cells4, two

    # ---- one frame through the drop-in the realtime loop calls: numpy image in, centroid list + undistorted image out ------
    latency = None
    if rank == 0 and not args.no_extra:
        from mocapv2_b200 import engine as E
        from mocapv2_b200.lib import ImageOperations as IO
        E.set_default_engine(eng)
        IO.camera_params = rig["camera_params"]
        IO.ANNOTATE = False                                        # the display-only overlays are host-side cv2 drawing
        host_frame = frames[0, 0].cpu().numpy()
        for _ in range(5):
            IO._find_dot(host_frame)
        lat = []
        for _ in range(30):
            t0 = time.perf_counter()
            _, pts_one = IO._find_dot(host_frame)
            lat.append((time.perf_counter() - t0) * 1e3)
        lat.sort()
        latency = {"call": "lib.ImageOperations._find_dot(img) on one 2048x2048 host frame (H2D + detect + undistorted image D2H)",
                   "median_ms": lat[len(lat) // 2], "min_ms": lat[0], "centroids": len(pts_one)}

    # ---- bundle adjustment (SURVEY 8f row 1, lib/Helpers.py:158-176) on the reference's own fixture, against the CPU port here --------
    ba = None
    if rank == 0 and not args.no_extra:
        try:
            ba = _bundle_adjustment_timing(eng)
        except Exception as ex:
            ba = {"error": repr(ex)}

    # ---- the other BASELINE configs on one GPU (C1: the reference's own 2-camera case, C3: 6 x 1440x1080) ---------------------
    others = None
    if world == 1 and not args.no_extra:
        others = {"c1": _extra_config(eng, "c1", 4, 0.0, 1024, device),
                  "c3": _extra_config(eng, "c3", 32, 0.42, 1024, device)}

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    # ---- roofline: the detection chain (what a step pays for its H*W bytes), and every kernel against ITS OWN traffic --------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    alg_bytes = n_local * H * W + n_local * (4 + 8 * MAX_BLOBS)          # SURVEY 8d: H*W read + (4 + 8 n_blobs) written per frame
    det_ms = phase["detect_in_flight_ms"]
    achieved = alg_bytes / (det_ms * 1e-3) / 1e9
    tr = _load_traffic()
    kernels = {"scan": "scan_hot_vec32_kernel (one-shot call) / scan_tma_kernel (overlapped call)", "group": "form_clusters_kernel",
               "filter": "piece_filter_kernel", "borders": "candidates_kernel + borders_finalize_kernel (traces, filter/centroid/order)",
               "finish": "general path for flagged frames (mark_active/compact_tiles/filter_tiles/blobs)"}
    per_kernel = {}
    for st_name, ms_ in stage_avg.items():
        ent = {"kernel": kernels.get(st_name, st_name), "ms_serial": ms_}
        t_ = tr.get(st_name)
        if t_ and ms_ > 0:
            dram = t_["dram_bytes_per_frame"] * n_local
            ent.update({"dram_bytes": dram, "dram_gbs": dram / (ms_ * 1e-3) / 1e9, "frac_of_hbm_peak": dram / (ms_ * 1e-3) / 1e9 / peak,
                        "bound": t_.get("bound", "hbm")})
        per_kernel[st_name] = ent
    if tma_scan_ms:
        per_kernel["scan_tma_alone"] = {"kernel": "scan_tma_kernel (TMA ring, timed alone)", "ms_serial": tma_scan_ms,
                                        "dram_gbs": n_local * H * W / (tma_scan_ms * 1e-3) / 1e9,
                                        "frac_of_hbm_peak": n_local * H * W / (tma_scan_ms * 1e-3) / 1e9 / peak, "bound": "hbm"}
    if front:
        front["peak_gbs"] = peak
        front["frac"] = front["achieved_gbs"] / peak
    chain_traffic = None
    if tr:
        chain_traffic = sum(v.get("dram_bytes_per_frame", 0) for k, v in tr.items() if isinstance(v, dict) and k in stage_avg) * n_local
    roofline = {"bound": "hbm", "kernel": "detection chain of a step (scan, group, filter, borders, finish; the scan overlapped with the other stages)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": chain_traffic,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "detect_ms": det_ms,
                "definition": "frames x (H*W + 4 + 8*max_blobs) bytes / time per step of ALL detection kernels of a step: CUDA events around a loop "
                              "of detect calls at the operating point of the timed loop (phase_ms.steps_in_flight calls in flight, each on its "
                              "own lane), max over ranks; single_call = one call after the other; whole_step = the timed loop itself "
                              "(detection + exchange + match + triangulate)",
                "single_call": {"ms": phase["detect_single_call_ms"], "frac": alg_bytes / (phase["detect_single_call_ms"] * 1e-3) / 1e9 / peak},
                "stages_one_after_the_other": {"ms": stage_avg, "sum_ms": serial_ms, "frac": alg_bytes / (serial_ms * 1e-3) / 1e9 / peak,
                                               "note": "the same kernels through the one-shot call (no overlap), per-stage CUDA events"},
                "overlapped_detection": pipe_info, "timeline_ms": timeline,
                "kernels": per_kernel,
                "whole_step": {"ms": ms_total / args.steps, "frac": alg_bytes / (ms_total / args.steps * 1e-3) / 1e9 / peak}}

    # ---- CPU baseline on this host (N=1 only) + parity of the timed workload against it ------------------------------------------------
    cpu = None
    parity = None
    if world == 1 and args.cpu_sample > 0:
        threads = os.cpu_count() or 1
        hf = frames[:args.cpu_sample].cpu().numpy()
        r = cpu_frame_sets(rig, hf, args.cpu_sample, threads)
        if r is not None:
            dt, nf, npts = r
            cvt = None
            try:
                import cv2
                cvt = cv2.getNumThreads()
            except Exception:
                pass
            cpu = {"value": nf / dt, "unit": "frames/s", "cores": threads, "os_cpu_count": os.cpu_count(), "cv2_num_threads": cvt, "kind": "port",
                   "sample": f"{args.cpu_sample} frame-set(s) = {nf} frames of this workload in {dt:.2f} s: OpenCV calls of "
                             "lib/ImageOperations.py:33-65 (numba blur -> its integer restatement) + lib/Helpers.py:178-280 in NumPy "
                             f"with the same candidate cap; frames over a {threads}-thread pool", "points_per_s": npts / dt}
        try:
            det, corr = step()                                   # the pipeline's result buffers were reused by the sections above
            torch.cuda.synchronize()
            parity = _parity_check(rig, frames, det, corr, pipe.cams_local)
        except Exception as ex:                                  # the check must never cost the bench line
            parity = {"checked": False, "why": repr(ex)}

    line = {
        "metric": "frames/s (detect+match+triangulate, 16-camera 2048x2048 rig, 128 markers)",
        "value": value, "unit": "frames/s", "n_gpus": N, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8 (detection, integer exact) / f32 (geometry)", "data": "synthetic",
        "config": dict(workload_config(N, F0), steps_in_flight=flight.depth,
                       in_flight_note="the timed loop keeps this many steps in flight, each on its own lane (stream, detection pipe, buffers); "
                                      "every step is complete when the timed region ends"),
        "points_per_s": points_per_step * args.steps / (ms_total * 1e-3),
        "frame_sets_with_group_cap": float(n_pts[1].item()), "centroids_per_frame": float(n_pts[2].item()) / (n_local * N),
        "phase_ms": phase, "output_checksum": checksum, "parity_check": parity,
        "e2e": e2e, "gpu_launches": gpu_launches, "collectives_per_step": 1 if N > 1 else 0,
        "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "geometry": geometry, "front_step": front, "find_dot_latency": latency, "host_binding": host_binding,
        "other_configs": others, "bundle_adjustment": ba,
    }
    emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


RESULT_OUT = sys.stdout


def emit(line: dict):
    """The ONE JSON line of the contract, on the process's real stdout."""
    RESULT_OUT.write(json.dumps(line) + "\n")
    RESULT_OUT.flush()


def main():
    # Libraries write to fd 1 behind Python's back (NCCL prints its version line there at NCCL_DEBUG=WARN/VERSION): send fd 1
    # to stderr for the whole run and keep a private handle on the real stdout for the result line.
    global RESULT_OUT
    sys.stdout.flush()
    RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
