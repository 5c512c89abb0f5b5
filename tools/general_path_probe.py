"""Time the general detection path and the drawContours outline on the bench workload's frames (development probe).

    python tools/general_path_probe.py [--frame-sets 8] [--reps 20] [--lib path/to/variant.so]

Prints the CUDA-event time per call of
  bits      detect(outputs=("bits",)): every frame through the general path, border starts straight from the runs;
  labels    detect(outputs=("bits", "labels", "blob_sums", "contours")): the general path with labels and the full contour tree;
  outline   draw_contours of the kept contours of those frames (mocap_draw_contours_batch),
and a checksum of the outputs, so that two builds can be compared in alternating runs.
"""
import argparse
import hashlib
import os
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import bench as B  # noqa: E402
from mocapv2_b200.engine import CaptureEngine  # noqa: E402
from mocapv2_b200.pipeline import CapturePipeline  # noqa: E402

ALL = ("bits", "labels", "blob_sums", "contours")


def timed(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frame-sets", type=int, default=8, help="frame-sets of the bench rig (16 frames of 2048 x 2048 each)")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--lib", default="", help="a variant library (tools/build_variant.py) instead of the product library")
    a = ap.parse_args()
    if a.lib:
        from mocapv2_b200 import _cabi
        _cabi.DEFAULT_LIB = os.path.abspath(a.lib)
        print("library:", a.lib)
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    eng = CaptureEngine(dev)
    rig, cen, ridx = B.make_scene(a.frame_sets)
    pipe = CapturePipeline(eng, rig, max_blobs=B.MAX_BLOBS, obj_count=B.N_MARKERS, max_groups=B.MAX_GROUPS)
    frames = B.render_local(rig, cen, ridx, 0, pipe.cams_local, dev).view(-1, rig["H"], rig["W"])
    K, D = pipe.K0, pipe.dist0
    mb = B.MAX_BLOBS
    out_bits = eng.detect(frames, K, D, max_blobs=mb, outputs=("bits",))
    out_all = eng.detect(frames, K, D, max_blobs=mb, outputs=ALL)
    img = frames.clone()
    eng.draw_contours(img, out_all)
    torch.cuda.synchronize()
    h = hashlib.sha1()
    for t in (out_bits.xy, out_bits.count, out_all.xy, out_all.count, out_all.extras["contours"], out_all.extras["labels"], img):
        h.update(t.cpu().numpy().tobytes())
    t_bits = timed(lambda: eng.detect(frames, K, D, max_blobs=mb, outputs=("bits",), out=out_bits), a.reps)
    t_all = timed(lambda: eng.detect(frames, K, D, max_blobs=mb, outputs=ALL, out=out_all), a.reps)
    t_draw = timed(lambda: eng.draw_contours(img, out_all), a.reps)
    print(f"frames {frames.shape[0]}  bits {t_bits:.4f} ms  labels {t_all:.4f} ms  outline {t_draw:.4f} ms  "
          f"general-path frames {int((out_bits.flags & 64).ne(0).sum())}  checksum {h.hexdigest()[:16]}")


if __name__ == "__main__":
    main()
