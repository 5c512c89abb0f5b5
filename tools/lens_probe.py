"""Cost of per-camera lenses on the bench workload (C4: 16 cameras 2048 x 2048, 64 frame-sets = 1024 frames per call), at the bench's
operating point: two overlapped detection calls in flight, 4 chunks on 4 worker streams.

    python tools/lens_probe.py [--reps 40] [--variant mocapv2_b200/_variants/map_normal.so]

Arms:
  (a) one table (camera 0's lens for every frame, today's path)
  (b) a 16-lens set of that table repeated -- outputs must equal (a); isolates the cost of the map footprint
  (c) 16 distinct lenses (synth.per_camera_lenses), frames rendered per lens
For each arm: ms per detection call in flight and frames/s, then piece_filter_kernel device time per call from torch.profiler in a
separate run.  With --variant (a library built with -DPF_MAP_EVICT=evict_normal by tools/build_variant.py) arms (a) and (c) are also
run on it, alternating with the product library: the L2 priority of the fast-map reads.
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
from mocapv2_b200 import _cabi  # noqa: E402
from mocapv2_b200 import synth as S  # noqa: E402
from mocapv2_b200.engine import CaptureEngine  # noqa: E402

CHUNKS, WORKERS = 4, 4


def scene(rig, n_frame_sets, seed=S.SEED0 + 4000):
    """bench.make_scene on a given rig (same seeds, markers projected with each camera's own lens on a per-camera rig)."""
    rng = np.random.default_rng(seed)
    X0 = S.sample_markers(rig, B.N_MARKERS, rng, spread=B.SPREAD, min_sep_px=56.0, margin=40.0, tries=300)
    C = len(rig["poses"])
    cen = np.empty((n_frame_sets, C, B.N_MARKERS, 2), dtype=np.int64)
    ridx = np.empty((n_frame_sets, C, B.N_MARKERS), dtype=np.int64)
    for s in range(n_frame_sets):
        rs = np.random.default_rng(seed + 1 + s)
        X = X0 + rs.uniform(-B.JITTER, B.JITTER, X0.shape)
        cen[s] = np.rint(S.marker_pixels(rig, X)).astype(np.int64)
        ridx[s] = rs.integers(0, 9, (C, B.N_MARKERS))
    return cen, ridx


def engines(lib_path, dev, depth=2):
    out = []
    for _ in range(depth):
        e = CaptureEngine(dev)
        if lib_path:
            e.lib = _cabi.load(lib_path)
        e.pipe_workers = WORKERS
        out.append(e)
    return out


def in_flight(engs, frames, kw, reps):
    """ms per call with len(engs) overlapped calls in flight on their own streams, and the outputs of the last calls"""
    n = frames.shape[0]
    cf = -(-n // CHUNKS)
    streams = [torch.cuda.Stream(frames.device) for _ in engs]
    outs = []
    for e, s in zip(engs, streams):
        with torch.cuda.stream(s):
            outs.append(e.detect_pipelined(frames, max_blobs=B.MAX_BLOBS, chunk_frames=cf, **kw))

    def run(k):
        for i in range(k):
            j = i % len(engs)
            with torch.cuda.stream(streams[j]):
                engs[j].detect_pipelined(frames, max_blobs=B.MAX_BLOBS, chunk_frames=cf, out=outs[j], **kw)
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


def piece_filter_ms(engs, frames, kw, reps):
    from torch.profiler import ProfilerActivity, profile
    in_flight(engs, frames, kw, 2)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        in_flight(engs, frames, kw, reps)
    tot = sum(ev.device_time_total for ev in prof.events() if ev.device_type.name == "CUDA" and "piece_filter_kernel" in ev.name)
    return tot / 1000.0 / (reps + 4 + len(engs))          # (in_flight runs reps + 4 warm-up calls + one first call per engine)


def same(r, w):
    if not (torch.equal(r.count, w.count) and torch.equal(r.flags, w.flags)):
        return False
    return all(torch.equal(r.xy[i, :int(w.count[i])], w.xy[i, :int(w.count[i])]) for i in range(len(w.count)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frame-sets", type=int, default=64)
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--rounds", type=int, default=3, help="alternating rounds over the arms")
    ap.add_argument("--variant", default="", help="library built with -DPF_MAP_EVICT=evict_normal (L2 policy A/B)")
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    FS = a.frame_sets
    rig_a = S.config_rig("c4")
    lenses = S.per_camera_lenses(16)
    rig_c = S.ring_rig(16, 2048, 2048, radius=6.0, lenses=lenses)
    H, W = rig_a["H"], rig_a["W"]
    cen, ridx = scene(rig_a, FS)
    frames_a = B.render_local(rig_a, cen, ridx, 0, 16, dev).view(-1, H, W)
    cen, ridx = scene(rig_c, FS)
    frames_c = B.render_local(rig_c, cen, ridx, 0, 16, dev).view(-1, H, W)
    n = frames_a.shape[0]
    libs = {"product": ""}
    if a.variant:
        libs["map_evict_normal"] = os.path.abspath(a.variant)
    E = {k: engines(p, dev) for k, p in libs.items()}
    K0, D0 = rig_a["camera_params"][0]["intrinsic_matrix"], rig_a["camera_params"][0]["distortion_coef"]
    e0 = E["product"][0]
    frame_lens = (torch.arange(n, dtype=torch.int32) % 16).to(dev)
    set_b = e0.lens_set([rig_a["camera_params"][0]] * 16, H, W)
    set_c = e0.lens_set(rig_c["camera_params"], H, W)
    for es in E.values():
        for e in es:
            e._tables = e0._tables
    arms = {"a": (frames_a, {"K": K0, "dist": D0}), "b": (frames_a, {"lenses": set_b, "frame_lens": frame_lens}),
            "c": (frames_c, {"lenses": set_c, "frame_lens": frame_lens})}
    print(f"C4 {n} frames of {H}x{W}; lens-set bytes: (b) {set_b.tables.numel() / 1e6:.1f} MB, (c) {set_c.tables.numel() / 1e6:.1f} MB; "
          f"one table {set_b.stride / 1e6:.1f} MB; {CHUNKS} chunks / {WORKERS} workers, 2 calls in flight", flush=True)
    plan = [(lib, arm) for lib in E for arm in arms if lib == "product" or arm != "b"]
    times = {p: [] for p in plan}
    outs = {}
    for r in range(a.rounds):
        for p in plan:
            fr, kw = arms[p[1]]
            t, o = in_flight(E[p[0]], fr, kw, a.reps)
            times[p].append(t)
            outs[p] = o[0]
    for p in plan:
        ts = times[p]
        print(f"lib {p[0]:17s} arm ({p[1]}): ms per call in flight {np.mean(ts):.4f} (min {min(ts):.4f} max {max(ts):.4f})  "
              f"frames/s {n / (np.mean(ts) / 1e3):,.0f}", flush=True)
    # correctness: (b) equals (a); (c) per frame equals the single-table call with that frame's lens (a sample)
    print("outputs (b) == (a):", same(outs[("product", "b")], outs[("product", "a")]), flush=True)
    for lib in E:
        if lib != "product":
            print(f"outputs {lib} == product: (a)", same(outs[(lib, "a")], outs[("product", "a")]),
                  "(c)", same(outs[(lib, "c")], outs[("product", "c")]), flush=True)
    rc = outs[("product", "c")]
    ok = True
    for i in range(0, n, 97):
        one = e0.detect(frames_c[i:i + 1], *lenses[i % 16], max_blobs=B.MAX_BLOBS)
        ok &= rc.points(i) == one.points(0)
    print("outputs (c) == single-table calls with each frame's lens (every 97th frame):", ok,
          " cluster-path frames", int(((rc.flags & 64) == 0).sum()), "of", n, flush=True)
    for p in plan:
        fr, kw = arms[p[1]]
        print(f"lib {p[0]:17s} arm ({p[1]}): piece_filter_kernel {piece_filter_ms(E[p[0]], fr, kw, 10):.4f} ms per call (torch.profiler)",
              flush=True)


if __name__ == "__main__":
    main()
