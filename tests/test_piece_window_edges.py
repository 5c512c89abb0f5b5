"""The piece filter's staged source window at the frame edges.

A window that reaches past a frame edge is zero-filled there (by the TMA unit on the device, by the emulated box copy on the
CPU build).  Blobs within 4 px of every edge and corner, in a batch whose rows are multiples of 16 bytes but whose frame size is
not a multiple of 32, must give the oracle's contour table and centroids; the same frames 8 bytes apart (a frame stride no tensor
map can describe, so every piece takes its taps from global memory) must give the same results.
"""
import numpy as np
import torch

from oracle import restate as R
from util import K, D, oracle_contour_table

H, W = 200, 336                                   # W: 21 rows of 16 bytes; neither is a multiple of 32


def edge_scene(rng, gap):
    """Discs on the four corners, discs `gap` px inside the middle of every edge, bars along two edges, one blob inside."""
    yy, xx = np.mgrid[0:H, 0:W]
    img = rng.integers(0, 40, (H, W)).astype(np.uint8)

    def disc(cx, cy, r):
        img[(xx - cx) ** 2 + (yy - cy) ** 2 <= r * r] = 255

    for cx, cy in ((0, 0), (W - 1, 0), (0, H - 1), (W - 1, H - 1)):
        disc(cx + int(rng.integers(-2, 3)), cy + int(rng.integers(-2, 3)), int(rng.integers(7, 13)))
    r = 9
    for cx, cy in ((W // 2, gap + r), (W // 2, H - 1 - gap - r), (gap + r, H // 2), (W - 1 - gap - r, H // 2)):
        disc(cx, cy, r)
    img[H - 1 - gap - 5:H - gap, 60:130] = 255
    img[60:130, W - 1 - gap - 4:W - gap] = 255
    disc(W // 2 + 40, H // 2 + 20, 11)
    return img


def test_window_zero_fill_at_the_frame_edges(engine):
    rng = np.random.default_rng(31)
    frames = np.stack([edge_scene(rng, gap) for gap in (0, 1, 2, 4)])
    n = len(frames)
    dense = torch.from_numpy(frames).to(engine.device, copy=True)
    buf = torch.zeros((n, H * W + 8), dtype=torch.uint8, device=engine.device)
    buf[:, :H * W] = dense.view(n, H * W)
    strided = buf[:, :H * W].view(n, H, W)
    for ma in (0.0, 60.0):
        res = engine.detect(dense, K, D, min_area=ma, outputs=("contours",))
        ref = engine.detect(strided, K, D, min_area=ma, outputs=("contours",))
        assert torch.equal(res.count, ref.count) and torch.equal(res.extras["contour_count"], ref.extras["contour_count"])
        for i, img in enumerate(frames):
            _, binimg = R.filter_frame(img, K, D)
            table, pts = oracle_contour_table(binimg, ma)
            nc = int(res.extras["contour_count"][i])
            assert nc == len(table) and np.array_equal(res.extras["contours"][i, :nc, :7].cpu().numpy(), table)
            assert res.points(i) == pts and ref.points(i) == pts
            assert torch.equal(res.extras["contours"][i, :nc], ref.extras["contours"][i, :nc])
            assert int(res.flags[i]) & (63 | 64) & ~16 == 0 and int(res.flags[i]) == int(ref.flags[i])   # finished by the cluster path
