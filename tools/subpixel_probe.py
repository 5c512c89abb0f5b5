"""Sub-pixel centroids against whole-pixel ones on the GPU: what they gain in accuracy and what they cost per step.

    python tools/subpixel_probe.py [--frame-sets 4] [--steps 20] [--rounds 3]

(a) Accuracy: C3 rig (6 cameras, 1440 x 1080), seeded frame-sets of 32 markers rendered at sub-pixel positions with
    synth.render_frameset, both centroid modes through CapturePipeline.  Image error: every kept centroid against the ideal
    undistorted projection K0 [R|t] X of the nearest marker (within 3 px); 3-D error: every matched object point within 1 cm of a
    marker.
(b) Cost: the bench's C4 step (16 cameras 2048 x 2048, 64 frame-sets = 1024 frames, detect -> match) with StepsInFlight(depth=2),
    int and sub-pixel pipelines alternating, `--rounds` rounds of `--steps` timed steps each (CUDA events), min - max per mode.
The card's name, power limit and max SM clock are printed beside the numbers.
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import bench as B  # noqa: E402
from mocapv2_b200 import synth as S  # noqa: E402
from mocapv2_b200.engine import CaptureEngine  # noqa: E402
from mocapv2_b200.pipeline import CapturePipeline, StepsInFlight  # noqa: E402

MODES = ("int", "subpixel")


def ideal_pixels(rig, X):
    K0 = np.asarray(rig["camera_params"][0]["intrinsic_matrix"], dtype=np.float64)
    out = []
    for p in rig["poses"]:
        h = (X @ np.asarray(p["R"]).T + np.asarray(p["t"]).reshape(3)) @ K0.T
        out.append(h[:, :2] / h[:, 2:3])
    return np.stack(out)


def accuracy(eng, n_sets):
    rig = S.config_rig("c3")
    C = len(rig["poses"])
    rng = np.random.default_rng(S.SEED0 + 5000)
    frames, markers = [], []
    for _ in range(n_sets):
        X = S.config_markers("c3", rig, rng)
        frames.append(S.render_frameset(rig, X, rng.integers(14, 23, (C, len(X))), rng))
        markers.append(X)
    frames = torch.from_numpy(np.stack(frames)).to(eng.device)
    print(f"(a) accuracy: C3 rig, {n_sets} frame-sets x {len(markers[0])} markers, {C} cameras {rig['W']}x{rig['H']}")
    print(f"    {'centroid':9s} {'n':>5s} {'mean dx':>8s} {'mean dy':>8s} {'rms dx':>7s} {'rms dy':>7s} {'rms px':>7s} "
          f"{'3-D n':>6s} {'3-D mean mm':>12s} {'3-D max mm':>11s}")
    for mode in MODES:
        pipe = CapturePipeline(eng, rig, max_blobs=64, obj_count=64, max_groups=64, centroids=mode)
        res = pipe.step(frames)
        torch.cuda.synchronize()
        d, e3 = [], []
        for s in range(n_sets):
            truth = ideal_pixels(rig, markers[s])
            for c in range(C):
                i = s * C + c
                for q in res.det.xy[i, :int(res.det.count[i])].cpu().numpy().astype(np.float64):
                    r = truth[c] - q
                    k = int(np.argmin((r * r).sum(axis=1)))
                    if np.abs(r[k]).max() < 3.0:
                        d.append(q - truth[c][k])
            for P in res.corr.obj[s, :int(res.corr.n_obj[s])].cpu().numpy():
                m = float(np.linalg.norm(markers[s] - P, axis=1).min())
                if m < 0.01:
                    e3.append(m * 1000.0)
        d = np.array(d)
        mean, rms = d.mean(axis=0), np.sqrt((d ** 2).mean(axis=0))
        print(f"    {mode:9s} {len(d):5d} {mean[0]:+8.3f} {mean[1]:+8.3f} {rms[0]:7.3f} {rms[1]:7.3f} {np.sqrt((d ** 2).sum(axis=1).mean()):7.3f} "
              f"{len(e3):6d} {np.mean(e3):12.3f} {np.max(e3):11.3f}", flush=True)


def timing(dev, steps, rounds, depth=2):
    FS = 64
    rig, cen, ridx = B.make_scene(FS)
    lanes = {}
    for mode in MODES:
        eng = CaptureEngine(dev)
        pipe = CapturePipeline(eng, rig, max_blobs=B.MAX_BLOBS, obj_count=B.N_MARKERS, max_groups=B.MAX_GROUPS, centroids=mode)
        lanes[mode] = StepsInFlight(pipe, depth)
    frames = B.render_local(rig, cen, ridx, 0, len(rig["poses"]), dev)
    print(f"(b) cost: C4 step, {FS} frame-sets x {len(rig['poses'])} cameras = {FS * len(rig['poses'])} frames {rig['W']}x{rig['H']}, "
          f"StepsInFlight(depth={depth}), {steps} timed steps per round", flush=True)

    def run(flight, k):
        flight.fork()
        for _ in range(k):
            r = flight.submit(frames)
        flight.join()
        return r

    outs = {m: run(lanes[m], 3) for m in MODES}                       # warm-up of every lane
    torch.cuda.synchronize()
    n = int(outs["int"].det.count.sum())
    assert torch.equal(outs["int"].det.count, outs["subpixel"].det.count) and n > 0
    ms = {m: [] for m in MODES}
    for _ in range(rounds):
        for m in MODES:
            run(lanes[m], 2)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            run(lanes[m], steps)
            b.record()
            torch.cuda.synchronize()
            ms[m].append(a.elapsed_time(b) / steps)
    for m in MODES:
        v = ms[m]
        print(f"    {m:9s} ms per step: min {min(v):.3f}  max {max(v):.3f}  rounds {' '.join(f'{x:.3f}' for x in v)}  "
              f"({n} centroids per step)", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frame-sets", type=int, default=4, help="frame-sets of the accuracy part")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    print("card:", subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                  capture_output=True, text=True).stdout.strip(), flush=True)
    accuracy(CaptureEngine(dev), a.frame_sets)
    timing(dev, a.steps, a.rounds)


if __name__ == "__main__":
    main()
