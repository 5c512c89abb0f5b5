"""Detection with a lens set: one undistortion table per camera in one call (MocapLensSet in mocap_detect_batch and
mocap_detect_batch_pipelined).

Every frame of a batch that mixes lenses must give exactly what the single-table call gives with that frame's K / dist, and what
the oracle gives; a set of copies of one table must give the single-table call bit for bit; a lens index outside the set flags
the frame (MOCAP_FLAG_LENS_INDEX, count 0) and leaves the other frames alone.  The `engine` tests run on the CPU emulation build
and on the GPU.
"""
import ctypes

import numpy as np
import pytest
import torch

from mocapv2_b200 import _cabi
from mocapv2_b200 import synth as S
from oracle import restate as R
from util import oracle_contour_table, unpack_bits

ALL = ("bits", "labels", "blob_sums", "contours")
H, W = 240, 320
# the lenses of test_detect_parity.py: moderate barrel (cluster path), strong (general path, reason 10), pincushion (an unmapped
# band along the border), and the identity
LENSES = [
    (np.array([[300.0, 0, W / 2], [0, 300.0, H / 2], [0, 0, 1]]), np.array([-0.20, 0.01, 0.001, -0.001, 0.0])),
    (np.array([[60.0, 0, W / 2], [0, 60.0, H / 2], [0, 0, 1]]), np.array([-0.35, 0.12, 0.0, 0.0, 0.0])),
    (np.array([[400.0, 0, W / 2], [0, 400.0, H / 2], [0, 0, 1]]), np.array([0.30, 0.0, 0.0, 0.0, 0.0])),
    (np.eye(3), np.zeros(5)),
]
ORDER = [2, 0, 3, 1, 1, 0, 2, 3, 0, 0, 3, 2, 1, 2, 0, 3]           # non-periodic lens order of the frames
MIN_AREA = 30.0


def params(lenses):
    return [{"intrinsic_matrix": K.tolist(), "distortion_coef": d.tolist()} for K, d in lenses]


def dev(engine, a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(engine.device)


def is_gpu(engine):
    return engine.device.type == "cuda"


def scene(seed, n):
    """n frames of discs (some near the border, where the pincushion lens leaves pixels unmapped) and, in every fourth, a bar."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[:H, :W]
    out = []
    for i in range(n):
        img = rng.integers(0, 40, (H, W)).astype(np.uint8)
        for _ in range(7):
            cx, cy, r = int(rng.integers(12, W - 12)), int(rng.integers(12, H - 12)), int(rng.integers(7, 15))
            img[(xx - cx) ** 2 + (yy - cy) ** 2 <= r * r] = 255
        if i % 4 == 3:
            img[40:200, 150:156] = 255
        out.append(img)
    return np.stack(out)


def n_frames(engine):
    return 16 if is_gpu(engine) else 8


def same_frame(res, i, one, j=0, with_contours=True):
    assert res.points(i) == one.points(j), f"frame {i}"
    assert int(res.flags[i]) & 63 == int(one.flags[j]) & 63
    if with_contours:
        nc = int(one.extras["contour_count"][j])
        assert int(res.extras["contour_count"][i]) == nc
        assert torch.equal(res.extras["contours"][i, :nc], one.extras["contours"][j, :nc])


@pytest.mark.parametrize("outputs", [("contours",), ALL])
def test_mixed_lenses_equal_single_table_calls_and_oracle(engine, outputs):
    n = n_frames(engine)
    frames = scene(31, n)
    order = ORDER[:n]
    ls = engine.lens_set(params(LENSES), H, W)
    res = engine.detect(dev(engine, frames), lenses=ls, frame_lens=order, min_area=MIN_AREA, outputs=outputs)
    bits = unpack_bits(res.extras["bits"], W) if "bits" in outputs else None
    paths = set()
    for i, l in enumerate(order):
        K, D = LENSES[l]
        one = engine.detect(dev(engine, frames[i:i + 1]), K, D, min_area=MIN_AREA, outputs=outputs)
        same_frame(res, i, one)
        _, binimg = R.filter_frame(frames[i], K, D)
        table, pts = oracle_contour_table(binimg, MIN_AREA)
        nc = int(res.extras["contour_count"][i])
        assert nc == len(table) and np.array_equal(res.extras["contours"][i, :nc, :7].cpu().numpy(), table)
        assert res.points(i) == (pts if pts else [[None, None]])
        assert int(res.flags[i]) & 63 == 0
        if bits is not None:
            assert np.array_equal(bits[i] != 0, binimg != 0), f"filtered binary image of frame {i}"
        paths.add((l, bool(int(res.flags[i]) & 64)))
    if outputs == ("contours",):
        assert (1, True) in paths and (0, False) in paths and (2, False) in paths      # reason 10 and the cluster path in one batch


def test_pipelined_lens_set_equals_one_shot(engine):
    n = n_frames(engine)
    frames = scene(32, n)
    order = torch.tensor(ORDER[:n], dtype=torch.int32)
    ls = engine.lens_set(params(LENSES), H, W)
    fr = dev(engine, frames)
    want = engine.detect(fr, lenses=ls, frame_lens=order, min_area=MIN_AREA, outputs=("contours",))
    for chunk in (1, 3, n):
        got = engine.detect_pipelined(fr, lenses=ls, frame_lens=order, min_area=MIN_AREA, outputs=("contours",), chunk_frames=chunk)
        for i in range(n):
            same_frame(got, i, want, i)
    # Bayer-delivered cell boxes: the grey frames' boxes come with the front step, the call runs no scan
    grey, cb = engine.bayer_gr2gray_scan(fr)
    want = engine.detect(grey, lenses=ls, frame_lens=order, min_area=MIN_AREA, outputs=("contours",))
    assert sum(want.points(i) != [[None, None]] for i in range(n)) >= n // 2
    for chunk in (2, n):
        got = engine.detect_pipelined(grey, lenses=ls, frame_lens=order, min_area=MIN_AREA, outputs=("contours",), chunk_frames=chunk,
                                      cellbox=cb)
        for i in range(n):
            same_frame(got, i, want, i)
    # a K / dist call on the same pipe after the lens-set calls undistorts with its own table
    K, D = LENSES[0]
    plain = engine.detect_pipelined(fr, K, D, min_area=MIN_AREA, chunk_frames=3)
    one = engine.detect(fr, K, D, min_area=MIN_AREA)
    for i in range(n):
        same_frame(plain, i, one, i, with_contours=False)


def identical(got, one):
    """Same counts, flags, centroids and parity outputs (entries past a count are not outputs)."""
    assert torch.equal(got.count, one.count) and torch.equal(got.flags, one.flags)
    for i in range(len(one.count)):
        c = int(one.count[i])
        assert torch.equal(got.xy[i, :c], one.xy[i, :c])
        if "contours" in one.extras:
            nc = int(one.extras["contour_count"][i])
            assert torch.equal(got.extras["contours"][i, :nc], one.extras["contours"][i, :nc])
        if "blob_sums" in one.extras:
            nb = int(one.extras["blob_count"][i])
            assert torch.equal(got.extras["blob_sums"][i, :nb], one.extras["blob_sums"][i, :nb])
    for k in ("bits", "labels", "contour_count", "blob_count"):
        if k in one.extras:
            assert torch.equal(got.extras[k], one.extras[k]), k


def test_set_of_copies_equals_single_table(engine):
    n = n_frames(engine)
    frames = scene(33, n)
    K, D = LENSES[0]
    ls = engine.lens_set(params([LENSES[0]] * 3), H, W)
    order = [i % 3 for i in range(n)][::-1]
    fr = dev(engine, frames)
    for outputs in (("contours",), ALL):
        one = engine.detect(fr, K, D, min_area=MIN_AREA, outputs=outputs)
        identical(engine.detect(fr, lenses=ls, frame_lens=order, min_area=MIN_AREA, outputs=outputs), one)
    one = engine.detect_pipelined(fr, K, D, min_area=MIN_AREA, chunk_frames=3, outputs=("contours",))
    identical(engine.detect_pipelined(fr, lenses=ls, frame_lens=order, min_area=MIN_AREA, chunk_frames=3, outputs=("contours",)), one)


@pytest.mark.parametrize("outputs", [(), ALL])
def test_lens_index_outside_the_set_flags_the_frame(engine, outputs):
    n = 6
    frames = scene(34, n)
    ls = engine.lens_set(params(LENSES), H, W)
    good = [0, 2, 1, 3, 0, 2]
    bad = [0, -1, 1, len(LENSES), 0, 2]
    fr = dev(engine, frames)
    want = engine.detect(fr, lenses=ls, frame_lens=good, min_area=MIN_AREA, outputs=outputs)
    runs = [engine.detect(fr, lenses=ls, frame_lens=bad, min_area=MIN_AREA, outputs=outputs)]
    if not outputs:
        runs.append(engine.detect_pipelined(fr, lenses=ls, frame_lens=bad, min_area=MIN_AREA, chunk_frames=4))
    for got in runs:
        for i in range(n):
            if bad[i] != good[i]:
                assert int(got.flags[i]) & _cabi.FLAG_LENS_INDEX and int(got.count[i]) == 0, i
                assert got.points(i) == [[None, None]]
            else:
                assert int(got.flags[i]) & _cabi.FLAG_LENS_INDEX == 0
                same_frame(got, i, want, i, with_contours=False)
    assert _cabi.FLAG_LENS_INDEX & _cabi.FLAG_ERRORS
    assert any(want.points(i) != [[None, None]] for i in (1, 3))    # the flagged frames do hold blobs


def test_both_calls_check_the_lens_set_argument(engine):
    """Both detection calls check the whole lens set they are given: zero lenses, a stride below the table size or not a multiple
    of 256, NULL tables and a NULL set are invalid arguments."""
    lib = engine.lib
    n = 2
    frames = dev(engine, scene(35, n))
    ls = engine.lens_set(params(LENSES[:2]), H, W)
    tb = int(lib.mocap_undistort_table_bytes(H, W))
    assert ls.stride == tb and tb % 256 == 0
    mb, mc, mr = engine.default_caps(H, W)
    out = [engine.empty((n, mb, 2), torch.int32), engine.empty((n,), torch.int32), engine.empty((n,), torch.int32)]
    nbytes = lib.mocap_detect_workspace_bytes(n, H, W, mb, mc, mr)
    pn = lib.mocap_detect_pipelined_workspace_bytes(n, H, W, mb, mc, mr, 1)
    ws = engine._workspace(max(pn, nbytes))
    P = engine._ptr
    null = ctypes.c_void_p(0)
    ref = lambda lset: ctypes.byref(lset) if lset is not None else None

    def one_shot(lset):
        return lib.mocap_detect_batch(P(frames), n, H, W, H * W, ref(lset), 216, 30.0, 0.5, mb, mc, mr, P(out[0]), P(out[1]), P(out[2]),
                                      null, null, null, null, null, null, P(ws), nbytes, engine._stream(), null)

    def piped(lset):
        return lib.mocap_detect_batch_pipelined(engine._pipe(), P(frames), n, H, W, H * W, ref(lset), 216, 30.0, 0.5, mb, mc, mr,
                                                P(out[0]), P(out[1]), P(out[2]), null, null, null, null, null, null, null,
                                                P(ws), pn, engine._stream(), 1, 0)

    base = ls.tables.data_ptr()
    for call in (one_shot, piped):
        assert call(_cabi.LensSet(base, 2, tb, None)) == _cabi.OK
        for bad in (_cabi.LensSet(base, 0, tb, None), _cabi.LensSet(base, 2, tb - 256, None), _cabi.LensSet(base, 2, tb + 16, None),
                    _cabi.LensSet(None, 2, tb, None), None):
            assert call(bad) == -1, (call.__name__, bad)
    if is_gpu(engine):
        torch.cuda.synchronize()
    with pytest.raises(ValueError):
        engine.detect(frames, *LENSES[0], lenses=ls)
    with pytest.raises(ValueError):
        engine.detect(frames, lenses=ls, frame_lens=[0])


@pytest.mark.gpu
def test_sixteen_lens_c4_batch_against_oracle_sample(gpu_engine):
    """A full-size C4 batch (2048 x 2048) from a rig of 16 distinct lenses, three frame-sets: every frame undistorted with its own
    camera's lens, an oracle sample of frames, most frames finished on the cluster path."""
    eng = gpu_engine
    lenses = S.per_camera_lenses(16)
    rig = S.ring_rig(16, 2048, 2048, radius=6.0, lenses=lenses)
    rng = np.random.default_rng(1616)
    X = S.config_markers("c4", rig, rng)
    frames = np.stack([S.render_frameset(rig, X + rng.uniform(-0.01, 0.01, X.shape), rng.integers(14, 23, (16, len(X))), rng)
                       for _ in range(3)]).reshape(48, 2048, 2048)
    ls = eng.lens_set(rig["camera_params"], 2048, 2048)
    order = torch.arange(48, dtype=torch.int32) % 16
    fr = torch.from_numpy(frames).to(eng.device)
    res = eng.detect(fr, lenses=ls, frame_lens=order)
    over = eng.detect_pipelined(fr, lenses=ls, frame_lens=order, chunk_frames=12)
    torch.cuda.synchronize()
    assert sum(int(f) & 64 == 0 for f in res.flags) >= 40
    for i in range(48):
        assert int(res.flags[i]) & _cabi.FLAG_ERRORS == 0
        assert over.points(i) == res.points(i)
    for i in (0, 5, 17, 31, 46):
        K, D = lenses[i % 16]
        assert res.points(i) == R.find_dot(frames[i], K, D), f"frame {i}"
