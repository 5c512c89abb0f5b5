"""Quick per-stage timing of the detection on the bench workload (development probe; bench.py is the contract benchmark).

    python tools/stage_probe.py [--frame-sets 64] [--reps 20]

Prints the per-stage CUDA-event times of the one-shot call (stages one after the other), the overlapped call with the
pipeline's defaults and a few (chunks, workers) variants, and checks the overlapped output against the one-shot call.
"""
import argparse
import os
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import bench as B  # noqa: E402
from mocapv2_b200.engine import CaptureEngine  # noqa: E402
from mocapv2_b200.pipeline import CapturePipeline  # noqa: E402


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
    ap.add_argument("--frame-sets", type=int, default=64)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--lib", default="", help="a variant library (tools/build_variant.py) instead of the product library")
    ap.add_argument("--grid", default="8,6;8,4;4,4;16,6", help="semicolon list of chunks,workers")
    ap.add_argument("--kernel-times", action="store_true", help="also the device time of every kernel of the one-shot call (torch.profiler)")
    a = ap.parse_args()
    if a.lib:
        from mocapv2_b200 import _cabi
        _cabi.DEFAULT_LIB = os.path.abspath(a.lib)
        print("library:", a.lib)
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    eng = CaptureEngine(dev)
    FS = a.frame_sets
    rig, cen, ridx = B.make_scene(FS)
    pipe = CapturePipeline(eng, rig, max_blobs=B.MAX_BLOBS, obj_count=B.N_MARKERS, max_groups=B.MAX_GROUPS)
    frames = B.render_local(rig, cen, ridx, 0, pipe.cams_local, dev).view(-1, rig["H"], rig["W"])
    n, H, W = frames.shape
    K, D = pipe.K0, pipe.dist0
    mb = B.MAX_BLOBS
    ref = eng.detect(frames, K, D, max_blobs=mb)
    torch.cuda.synchronize()
    acc = {}
    for _ in range(a.reps):
        t = eng.stage_timer()
        eng.detect(frames, K, D, max_blobs=mb, out=ref, timer=t)
        torch.cuda.synchronize()
        for k, v in eng.stage_timer_read(t).items():
            acc[k] = acc.get(k, 0.0) + v / a.reps
    print("one-shot stages (ms):", {k: round(v, 4) for k, v in acc.items()}, "sum", round(sum(acc.values()), 4), flush=True)
    t = timed(lambda: eng.detect(frames, K, D, max_blobs=mb, out=ref), a.reps)
    print(f"one-shot call   {t:.4f} ms", flush=True)
    if a.kernel_times:
        kernel_times(lambda: eng.detect(frames, K, D, max_blobs=mb, out=ref), a.reps)
    refxy, refc = ref.xy.clone(), ref.count.clone()
    for g in a.grid.split(";"):
        chunks, workers = (int(x) for x in g.split(","))
        e = CaptureEngine(dev)
        e._tables = eng._tables
        e.pipe_workers = workers
        cf = -(-n // chunks)
        res = e.detect_pipelined(frames, K, D, max_blobs=mb, chunk_frames=cf)
        torch.cuda.synchronize()
        same = bool(torch.equal(res.count, refc)) and all(torch.equal(res.xy[i, :int(refc[i])], refxy[i, :int(refc[i])]) for i in range(0, n, 29))
        t = timed(lambda: e.detect_pipelined(frames, K, D, max_blobs=mb, chunk_frames=cf, out=res), a.reps)
        e.detect_pipelined(frames, K, D, max_blobs=mb, chunk_frames=cf, out=res, timeline=True)
        torch.cuda.synchronize()
        tl = e.pipe_timeline()
        print(f"overlapped chunks {chunks:2d} workers {workers}: {t:.4f} ms  same={same}  scan done {tl['scan_done']:.3f} join {tl['join']:.3f}", flush=True)
        for depth in (2, 3):
            t2, outs = two_in_flight(eng, frames, K, D, mb, 2 * a.reps, chunks, workers, depth)
            same2 = all(bool(torch.equal(o.count, refc)) for o in outs)
            print(f"   {depth} calls in flight: {t2:.4f} ms per call  same={same2}", flush=True)
        for c, r in enumerate(tl["chunks"]):
            print(f"    {c:2d}: seen {r[0]:.3f}  +group {r[1] - r[0]:.3f}  +filter {r[2] - r[1]:.3f}  +borders {r[3] - r[2]:.3f}  (end {r[3]:.3f})")


def kernel_times(fn, reps):
    """mean device time per call of every kernel `fn` launches (a separate, profiled run)"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    acc = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and ev.device_time_total > 0:
            acc[ev.name] = acc.get(ev.name, 0.0) + ev.device_time_total / 1000.0 / reps
    for name, ms in sorted(acc.items(), key=lambda kv: -kv[1]):
        print(f"  kernel {ms:8.4f} ms per call  {name.split('(')[0]}", flush=True)


def two_in_flight(eng, frames, K, D, mb, reps, chunks=8, workers=6, depth=2):
    """`depth` overlapped detection calls in flight on their own streams (own pipe, workspace and outputs each)"""
    n = frames.shape[0]
    cf = -(-n // chunks)
    dev = frames.device
    streams = [torch.cuda.Stream(dev) for _ in range(depth)]
    engs, outs = [], []
    for s in streams:
        e = CaptureEngine(dev)
        e._tables = eng._tables
        e.pipe_workers = workers
        with torch.cuda.stream(s):
            outs.append(e.detect_pipelined(frames, K, D, max_blobs=mb, chunk_frames=cf))
        engs.append(e)
    torch.cuda.synchronize()

    def run(k):
        for i in range(k):
            j = i % depth
            with torch.cuda.stream(streams[j]):
                engs[j].detect_pipelined(frames, K, D, max_blobs=mb, chunk_frames=cf, out=outs[j])
    run(4)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for s in streams:
        s.wait_event(a)
    run(reps)
    for s in streams:
        torch.cuda.current_stream().wait_stream(s)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps, outs


if __name__ == "__main__":
    main()
