"""The one border walker (csrc/walk.cuh, trace_border) in the places the other tests do not reach: cluster boxes taller than
1024 rows, general-path traces on tall frames and across several 64-pixel windows, and the drawContours outline.  Every
test runs on the emulation build and on the GPU (`engine` fixture)."""
import numpy as np
import pytest

from oracle import restate as R
from test_detect_parity import ALL, dev, same_contours
from util import check_blob_outputs, oracle_contour_table, pack_bits

CAPS = dict(max_blobs=512, max_contours=1024)


def test_cluster_boxes_taller_than_1024_rows(engine):
    """A bar and a ring at most 64 pixels wide and a ring wider than 64, each more than 1024 rows high, one per frame: their
    cluster boxes are traced on the 64-pixel window.  Contour table and centroids against the oracle, on the cluster path."""
    H, W = 1150, 192
    K = np.array([[1500.0, 0.0, W / 2], [0.0, 1500.0, H / 2], [0.0, 0.0, 1.0]])
    D = np.zeros(5)
    rng = np.random.default_rng(1150)
    frames = rng.integers(0, 40, (3, H, W)).astype(np.uint8)
    frames[0, 40:1110, 70:100] = 255                                    # bar, 30 wide
    frames[1, 30:1120, 60:116] = 255                                    # ring, 56 wide, with a tall hole
    frames[1, 60:1090, 78:98] = 0
    frames[2, 25:1125, 40:150] = 255                                    # ring, 110 wide
    frames[2, 70:1080, 70:120] = 0
    for ma in (0.0, 500.0):
        res = engine.detect(dev(engine, frames), K, D, min_area=ma, outputs=("contours",), **CAPS)
        for i in range(len(frames)):
            _, binimg = R.filter_frame(frames[i], K, D)
            table, pts = oracle_contour_table(binimg, ma)
            nc = int(res.extras["contour_count"][i])
            assert nc == len(table) and nc >= 1
            assert np.array_equal(res.extras["contours"][i, :nc, :7].cpu().numpy(), table)
            assert res.points(i) == (pts if pts else [[None, None]])
            assert int(res.flags[i]) & (63 | 64) & ~16 == 0                 # no capacity flag, finished by the cluster path


def tall_frame():
    """1100 x 100: a bar, a ring with a blob nested in its hole, and a comb, each taller than 1024 rows."""
    b = np.zeros((1100, 100), np.uint8)
    b[20:1080, 2:12] = 1
    b[10:1090, 20:70] = 1
    b[30:1070, 30:60] = 0
    b[300:800, 38:52] = 1
    b[5:1095, 80:84] = 1
    for y in range(5, 1095, 6):
        b[y:y + 3, 84:97] = 1
    return b


def wide_frames():
    """180 x 330: blobs wider than 64 pixels crossing several windows -- a ring with a blob nested in its hole, a bar, a comb
    whose teeth make the walker cross window edges again and again, a slanted polygon -- and blobs cut by the frame edges."""
    H, W = 180, 330
    yy, xx = np.mgrid[:H, :W]
    a = np.zeros((H, W), np.uint8)
    d2 = ((xx - 165) / 150.0) ** 2 + ((yy - 45) / 38.0) ** 2
    a[d2 <= 1.0] = 1
    a[d2 <= 0.45] = 0
    a[((xx - 165) / 60.0) ** 2 + ((yy - 45) / 10.0) ** 2 <= 1.0] = 1
    a[95:103, 0:W] = 1
    for x in range(10, 310, 11):
        a[103:140, x:x + 5] = 1
    a[np.abs((xx - 200) / 120.0) + np.abs((yy - 160 - 0.15 * (xx - 200)) / 14.0) <= 1.0] = 1
    b = np.zeros((H, W), np.uint8)
    b[0:30, 0:100] = 1                                                  # cut by the top and left edges
    b[10:20, 20:80] = 0
    b[60:170, W - 90:W] = 1                                             # cut by the right and bottom edges, with a ring inside
    b[70:160, W - 80:W - 10] = 0
    b[80:150, W - 70:W - 20] = 1
    b[90:140, W - 60:W - 30] = 0
    b[100:130, W - 50:W - 40] = 1
    b[H - 20:H, 120:200] = 1
    return [a, b]


def narrow_frame():
    """30 x 28 (one word per row): a ring with a blob inside and blobs cut by the edges."""
    b = np.zeros((30, 28), np.uint8)
    b[2:20, 3:20] = 1
    b[5:17, 6:17] = 0
    b[8:14, 9:14] = 1
    b[22:30, 0:10] = 1
    b[10:30, 23:28] = 1
    b[15:20, 25:27] = 0
    return b


def blob_cases():
    return [tall_frame()[None], np.stack(wide_frames()), narrow_frame()[None]]


def blobs(engine, b, ma, outputs):
    return engine.blobs(dev(engine, np.stack([pack_bits(x) for x in b])), b.shape[2], min_area=ma, outputs=outputs,
                        max_runs=b.shape[1] * b.shape[2] + 1, **CAPS)


def test_general_path_tall_and_wide_frames(engine):
    """The general path traces on whole frames: a frame taller than 1024 rows and frames with blobs wider than 64 pixels.
    Labels, pixel sums, contour table and centroids against the oracle; the call without label outputs (border starts
    straight from the runs) gives the same contours."""
    for b in blob_cases():
        for ma in (0.0, 30.0):
            res = blobs(engine, b, ma, ALL[1:])
            for i in range(len(b)):
                check_blob_outputs(res, i, b[i], ma)
            same_contours(res, blobs(engine, b, ma, ("contours",)))


@pytest.mark.parametrize("value", [0, 77])
def test_draw_contours_outline_against_cv2(engine, value):
    """mocap_draw_contours_batch against cv2.drawContours(img, kept, -1, colour, 2) of the contours that pass the same filter,
    pixel for pixel: rings, nested blobs, blobs wider than 64 pixels, edge-cut blobs, a frame one word wide, a tall frame."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(value)
    ma, mc = 30.0, 0.2
    drawn = 0
    for b in blob_cases():
        n, H, W = b.shape
        bits = dev(engine, np.stack([pack_bits(x) for x in b]))
        res = engine.blobs(bits, W, min_area=ma, min_circ=mc, outputs=("contours",), max_runs=H * W + 1, **CAPS)
        res.extras["bits"] = bits
        back = rng.integers(1, 256, (n, H, W)).astype(np.uint8)
        got = engine.draw_contours(dev(engine, back), res, value=value).cpu().numpy()
        for i in range(n):
            cs, _ = cv2.findContours(b[i] * 255, cv2.RETR_TREE, cv2.CHAIN_APPROX_SIMPLE)
            kept = []
            for c in cs:
                area, per = cv2.contourArea(c), cv2.arcLength(c, True)
                if per and 4 * np.pi * area / (per * per) > mc and area > ma:
                    kept.append(c)
            want = back[i].copy()
            cv2.drawContours(want, kept, -1, (value, 0, 255), 2)
            assert np.array_equal(got[i], want), f"outline differs in {(got[i] != want).sum()} pixels"
            drawn += len(kept)
    assert drawn >= 10
