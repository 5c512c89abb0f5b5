"""AddressSanitizer pass over the kernel sources through the CUDA-on-CPU shim (tests/emu): compute-sanitizer is closed on the
GPU pool, so out-of-bounds accesses are hunted here.  Usage:  python tests/emu_asan.py   (rebuilds into /tmp/emu_asan, then
re-executes itself with libasan preloaded)."""
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = "/tmp/emu_asan"
LIB = os.path.join(OUT, "libmocap_emu_asan.so")


def build():
    here, csrc = os.path.join(REPO, "tests", "emu"), os.path.join(REPO, "mocapv2_b200", "csrc")
    os.makedirs(OUT, exist_ok=True)
    objs = []
    flags = ["-std=c++20", "-O1", "-g", "-fsanitize=address", "-fno-omit-frame-pointer", "-fPIC", "-I", here]
    for s in ["api.cu", "detect_filter.cu", "detect_scan_tma.cu", "detect_cluster.cu", "detect_blobs.cu", "geometry.cu"]:
        o = os.path.join(OUT, s + ".o")
        subprocess.check_call(["g++", "-x", "c++", "-ffp-contract=off", "-DMOCAP_EMU", "-Wno-attributes"] + flags + ["-c", os.path.join(csrc, s), "-o", o])
        objs.append(o)
    o = os.path.join(OUT, "cuda_emu.o")
    subprocess.check_call(["g++"] + flags + ["-c", os.path.join(here, "cuda_emu.cpp"), "-o", o])
    subprocess.check_call(["g++", "-shared", "-fsanitize=address", "-o", LIB] + objs + [o, "-lpthread"])


def run():
    import numpy as np
    import torch
    sys.path.insert(0, REPO)
    sys.path.insert(0, os.path.join(REPO, "tests"))
    sys.path.insert(0, os.path.join(REPO, "tests", "emu"))
    from mocapv2_b200 import synth as S
    from mocapv2_b200.engine import CaptureEngine
    from test_detect_parity import random_scene
    from emu_engine import EmuEngine
    eng = EmuEngine(LIB)
    K, D = S.SHIPPED_K, S.SHIPPED_DIST
    rng = np.random.default_rng(5)
    for it in range(10):
        H, W = int(rng.integers(50, 260)), int(rng.integers(50, 300))
        if it % 2:
            W = (W // 16) * 16
        img = random_scene(rng, H, W)
        a = eng.detect(torch.from_numpy(img[None].copy()), K, D, min_area=0.0, outputs=("contours",))
        b = eng.detect(torch.from_numpy(img[None].copy()), K, D, min_area=0.0, outputs=("bits", "labels", "blob_sums", "contours"))
        assert a.points(0) == b.points(0)
        c = eng.detect(torch.from_numpy(img[None].copy()), K, D, min_area=0.0)          # the cluster path proper
        assert c.points(0) == a.points(0)
    img = rng.integers(0, 40, (200, 416)).astype(np.uint8)                               # borders several trace windows wide (walk.cuh, WINDOW)
    yy, xx = np.mgrid[:200, :416]
    img[((xx - 200) / 150.0) ** 2 + ((yy - 40) / 18.0) ** 2 <= 1.0] = 255
    img[130:140, 30:416] = 255
    for x in range(30, 400, 14):
        img[140:185, x:x + 7] = 255
    img[90:120, 0:130] = 255
    assert eng.detect(torch.from_numpy(img[None].copy()), K, D, min_area=0.0).points(0) == \
        eng.detect(torch.from_numpy(img[None].copy()), K, D, min_area=0.0, outputs=("bits", "labels")).points(0)
    from test_border_walker import narrow_frame
    from util import pack_bits
    bits = torch.from_numpy(pack_bits(narrow_frame())[None].copy())                    # rows of one word, blobs on the last row
    res = eng.blobs(bits, 28, min_area=0.0, outputs=("contours",))
    res.extras["bits"] = bits
    eng.draw_contours(torch.zeros((1, 30, 28), dtype=torch.uint8), res)
    for shape in [(3, 4), (5, 8), (34, 132), (64, 128), (97, 260), (7, 10), (33, 65), (3, 8), (12, 1032), (129, 1040), (75, 16)]:  # Bayer front step, both kernels
        eng.bayer_gr2gray(torch.from_numpy(rng.integers(0, 256, (2,) + shape).astype(np.uint8)))
        eng.bayer_gr2gray_scan(torch.from_numpy(rng.integers(0, 256, (2,) + shape).astype(np.uint8)), thresh=int(rng.integers(0, 256)))
    z = np.load(os.path.join(REPO, "tests", "golden", "c1_frames.npz"))["frames"].reshape(-1, 480, 640)[:2]
    res = eng.detect(torch.from_numpy(z.copy()), K, D)
    rig = S.config_rig("c1")
    cams = eng.cameras(rig["poses"], rig["camera_params"])
    mp = max(1, int(res.count.max()))
    xy = res.xy[:, :mp].reshape(1, 2, mp, 2).contiguous()
    eng.correspond(xy, res.count.reshape(1, 2).contiguous(), torch.tensor(np.array(rig["Fs"])), cams, obj_count=4)
    eng.triangulate(torch.rand((100, 2, 2)) * 600, cams)
    print("emu + ASan: clean")


if __name__ == "__main__":
    if os.environ.get("MOCAP_ASAN_CHILD"):
        run()
    else:
        build()
        asan = subprocess.check_output(["gcc", "-print-file-name=libasan.so"], text=True).strip()
        env = dict(os.environ, LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0", MOCAP_ASAN_CHILD="1")
        sys.exit(subprocess.call([sys.executable, os.path.abspath(__file__)], env=env))
