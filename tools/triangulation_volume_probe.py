"""Error statistics behind the bounds of tests/test_triangulation_volume.py (development / evidence tool): for every case of that file,
the largest relative X error over (kappa * u), the kappa range, and the largest relative X error and |d rms px| over the well-posed
points (kappa < K0), per precision.

    python tools/triangulation_volume_probe.py            the library on the GPU
    python tools/triangulation_volume_probe.py --emu      the CPU emulation build of the same kernel sources
"""
import argparse
import os
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [REPO, os.path.join(REPO, "tests"), os.path.join(REPO, "tests", "emu")]
import test_triangulation_volume as T  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--emu", action="store_true")
    a = ap.parse_args()
    if a.emu:
        import build_emu
        from emu_engine import EmuEngine
        eng = EmuEngine(build_emu.build())
    else:
        from mocapv2_b200 import build
        from mocapv2_b200.engine import CaptureEngine
        build.build()
        eng = CaptureEngine()
        print(torch.cuda.get_device_name(0))
    worst = {}
    check = T.check_points

    def recording(X, err, Xref, kappa, eref, eown, dtype, need_well_posed=True):
        has = np.isfinite(kappa)
        rel = np.abs(X[has] - Xref[has]).max(1) / np.linalg.norm(Xref[has], axis=1)
        k = kappa[has]
        dpx = np.abs(np.sqrt(err[has]) - np.sqrt((eref if dtype == torch.float32 else eown)[has]))
        wp = k < T.K0
        row = (float((rel / (k * T.U[dtype])).max()), float(k.min()), float(k.max()), float(rel[wp].max(initial=0.0)),
               float(dpx[wp].max(initial=0.0)))
        print(f"  {case:34s} {str(dtype)[6:]}  rel/(kappa u) {row[0]:7.3f}  kappa {row[1]:8.3g} .. {row[2]:8.3g}  "
              f"well-posed: rel X {row[3]:.2e}  |d rms px| {row[4]:.2e}")
        w = worst.setdefault(dtype, [0.0, 0.0, 0.0, 0.0])
        w[0], w[1], w[2], w[3] = max(w[0], row[0]), max(w[1], row[3]), max(w[2], row[4]), max(w[3], row[2] if case.startswith("all") else 0)
        return check(X, err, Xref, kappa, eref, eown, dtype, need_well_posed)

    T.check_points = recording
    for dtype in (torch.float32, torch.float64):
        for rig, C in T.ALL_VIEW_CASES:
            for kind in ("int", "sub"):
                case = f"all-views {rig} C={C} {kind}"
                T.test_all_views_over_volume(eng, rig, C, dtype, kind)
        for rig in ("ring6_lenses", "ring16_lenses", "c5"):
            case = f"masked {rig}"
            T.test_masked_views_rank_lenses(eng, rig, dtype)
        case = "pairs of the c3 ring"
        T.test_every_pair_of_the_ring(eng, dtype)
    for dtype, w in worst.items():
        print(f"{str(dtype)[6:]}: max rel/(kappa u) {w[0]:.3g} (C_KAPPA {T.C_KAPPA[dtype]:g}); well-posed (kappa < K0 = {T.K0:g}): "
              f"max rel X {w[1]:.2e}, max |d rms px| {w[2]:.2e}; all-view kappa up to {w[3]:.3g}")


if __name__ == "__main__":
    main()
