"""Correspondence alone on the bench workload (development / evidence tool): outputs of every mode for an A/B of two library builds,
and the device time of the correspondence kernels per call.

    python tools/corr_probe.py --dump DIR                 outputs of int32 / float32 lists x FP32 / FP64 mode -> DIR/*.npy, timings
    MOCAP_B200_LIB=other.so python tools/corr_probe.py --dump DIR2
    python tools/corr_probe.py --compare DIR DIR2         bit-for-bit comparison

Workload = bench.py's (BASELINE config 4: 16 cameras 2048x2048, 128 markers, 64 frame-sets, max_groups 64): the centroid lists are
detected once, then only the correspondence runs.
"""
import argparse
import os
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import bench as B  # noqa: E402
from mocapv2_b200.engine import CaptureEngine  # noqa: E402
from mocapv2_b200.pipeline import CapturePipeline  # noqa: E402

FIELDS = ("obj", "n_obj", "img", "n_valid", "err", "flags", "cand")


def outputs(res, count):
    """every output the call defines (cand rows of the roots, cameras >= 1), the rest zeroed"""
    out = {k: getattr(res, k).cpu().numpy().copy() for k in FIELDS}
    n0 = count[:, 0].cpu().numpy()
    rows = np.arange(out["cand"].shape[1])[None, :] >= n0[:, None]
    out["cand"][rows] = 0
    out["cand"][:, :, 0] = 0
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dump", default=None)
    ap.add_argument("--compare", nargs=2, default=None)
    ap.add_argument("--reps", type=int, default=200)
    a = ap.parse_args()
    if a.compare:
        bad = 0
        for f in sorted(os.listdir(a.compare[0])):
            x, y = np.load(os.path.join(a.compare[0], f)), np.load(os.path.join(a.compare[1], f))
            same = x.shape == y.shape and x.tobytes() == y.tobytes()
            bad += not same
            print(f"{f:28s} {'identical' if same else 'DIFFERENT'}")
        print("all identical" if not bad else f"{bad} arrays differ")
        raise SystemExit(1 if bad else 0)
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    eng = CaptureEngine(dev)
    FS = 64
    rig, cen, ridx = B.make_scene(FS)
    lists = {}
    for mode in ("int", "subpixel"):
        pipe = CapturePipeline(eng, rig, max_blobs=B.MAX_BLOBS, obj_count=B.N_MARKERS, max_groups=B.MAX_GROUPS, centroids=mode)
        frames = B.render_local(rig, cen, ridx, 0, pipe.cams_local, dev)
        xy, count = pipe.exchange(pipe.detect(frames), FS)
        lists[mode] = (xy.clone(), count.clone())
        del frames
    torch.cuda.synchronize()
    for mode, (xy, count) in lists.items():
        for fp64 in (False, True):
            res = eng.correspond(xy, count, pipe.Fs, pipe.cams, obj_count=B.N_MARKERS, max_groups=B.MAX_GROUPS, fp64=fp64, want_cand=True)
            torch.cuda.synchronize()
            tag = f"{mode}_{'fp64' if fp64 else 'fp32'}"
            if a.dump:
                os.makedirs(a.dump, exist_ok=True)
                for k, v in outputs(res, count).items():
                    np.save(os.path.join(a.dump, f"{tag}_{k}.npy"), v)

            def call():
                return eng.correspond(xy, count, pipe.Fs, pipe.cams, obj_count=B.N_MARKERS, max_groups=B.MAX_GROUPS, fp64=fp64, out=res)
            ms = B._time_loop(call, a.reps, warm=10)
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for _ in range(a.reps):
                    call()
                torch.cuda.synchronize()
            per = {}
            for ev in prof.key_averages():
                if ev.device_type == torch.autograd.DeviceType.CUDA:
                    per[ev.key] = per.get(ev.key, 0.0) + ev.device_time_total / a.reps
            total = sum(per.values())
            print(f"{tag}: n_valid {int(res.n_valid.sum())} over {FS} frame-sets, call {ms * 1e3:.1f} us back to back, device time "
                  f"{total:.1f} us per call: " + ", ".join(f"{k.split('(')[0][:40]} {v:.1f}" for k, v in sorted(per.items(), key=lambda t: -t[1])))


if __name__ == "__main__":
    main()
