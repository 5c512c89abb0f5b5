"""Workspace sizes of the two detection calls, which share one layout: the general-path arrays of the batch, the TMA scan's control
block, need_general and one cluster-path block per chunk.  A workspace of exactly the reported size is enough -- the call gives the
results of detect() and writes nothing past it -- and one 256 bytes smaller is MOCAP_ERR_WORKSPACE.  The one-shot call is sized for
the parity outputs; the overlapped call by its chunk count.  The `engine` tests run on the CPU emulation build and on the GPU.
"""
import ctypes

import numpy as np
import pytest
import torch

from mocapv2_b200 import _cabi
from mocapv2_b200 import synth as S
from util import K, D

H, W, N = 240, 320, 8
GUARD = 4096                 # bytes past the reported size, filled with a pattern the call must leave alone
PATTERN = 0xA5
ERR_WORKSPACE = -2
THRESH, MIN_AREA, MIN_CIRC = 216, 30.0, 0.5


def scene(engine):
    rng = np.random.default_rng(55)
    frames = np.empty((N, H, W), np.uint8)
    for i in range(N):
        cen = np.stack([rng.integers(30, W - 30, 4), rng.integers(30, H - 30, 4)], axis=1)
        frames[i] = S.render_frame(H, W, cen, rng.integers(14, 23, 4), rng)
    return torch.from_numpy(frames).to(engine.device)


def outputs(engine, parity):
    mb, mc, _ = engine.default_caps(H, W)
    out = {"xy": engine.empty((N, mb, 2), torch.int32), "count": engine.empty((N,), torch.int32), "flags": engine.empty((N,), torch.int32)}
    if parity:
        out.update(bits=engine.empty((N, H, (W + 31) // 32), torch.int32), labels=engine.empty((N, H, W), torch.int32),
                   blob_sums=torch.zeros((N, mb, 3), dtype=torch.int64, device=engine.device), blob_count=engine.empty((N,), torch.int32),
                   contours=torch.zeros((N, mc, 8), dtype=torch.float64, device=engine.device), contour_count=engine.empty((N,), torch.int32))
    return out


@pytest.mark.parametrize("call,parity,chunk_frames,chunks", [("one_shot", False, 0, 1), ("one_shot", True, 0, 1),
                                                             ("pipelined", False, N, 1), ("pipelined", False, 3, 3),
                                                             ("pipelined", False, 1, 8)])
def test_reported_workspace_size_is_exact(engine, call, parity, chunk_frames, chunks):
    lib, P = engine.lib, engine._ptr
    mb, mc, mr = engine.default_caps(H, W)
    frames = scene(engine)
    tab = engine.table(K, D, H, W)
    lens = _cabi.LensSet(tab.data_ptr(), 1, int(lib.mocap_undistort_table_bytes(H, W)), None)
    out = outputs(engine, parity)
    ex = [P(out.get(k)) for k in ("bits", "labels", "blob_sums", "blob_count", "contours", "contour_count")]
    null = ctypes.c_void_p(0)
    if call == "one_shot":
        nbytes = int(lib.mocap_detect_workspace_bytes(N, H, W, mb, mc, mr))
    else:
        nbytes = int(lib.mocap_detect_pipelined_workspace_bytes(N, H, W, mb, mc, mr, chunk_frames))
    assert nbytes > 0 and nbytes % 256 == 0
    ws = torch.full((nbytes + GUARD,), PATTERN, dtype=torch.uint8, device=engine.device)

    def run(size):
        if call == "one_shot":
            return lib.mocap_detect_batch(P(frames), N, H, W, H * W, ctypes.byref(lens), THRESH, MIN_AREA, MIN_CIRC, mb, mc, mr,
                                          P(out["xy"]), P(out["count"]), P(out["flags"]), *ex, P(ws), size, engine._stream(), null)
        return lib.mocap_detect_batch_pipelined(engine._pipe(), P(frames), N, H, W, H * W, ctypes.byref(lens), THRESH, MIN_AREA, MIN_CIRC,
                                                mb, mc, mr, P(out["xy"]), P(out["count"]), P(out["flags"]), ex[4], ex[5],
                                                null, null, null, null, null, P(ws), size, engine._stream(), chunk_frames, 0)

    assert run(nbytes - 256) == ERR_WORKSPACE
    assert run(nbytes) == _cabi.OK
    if call == "pipelined":
        info = (ctypes.c_int * 2)()
        assert lib.mocap_detect_pipe_info(engine._pipe(), info) == _cabi.OK and info[1] == chunks
    want = engine.detect(frames, K, D, thresh=THRESH, min_area=MIN_AREA, min_circ=MIN_CIRC,
                         outputs=("bits", "labels", "blob_sums", "contours") if parity else ())
    if engine.device.type == "cuda":
        torch.cuda.synchronize()
    assert bool((ws[nbytes:] == PATTERN).all()), "the call wrote past the reported workspace size"
    assert torch.equal(out["count"], want.count) and torch.equal(out["flags"], want.flags)
    assert int(want.count.sum()) > 0
    for i in range(N):
        c = int(want.count[i])
        assert torch.equal(out["xy"][i, :c], want.xy[i, :c]), f"frame {i}"
    if parity:
        for k in ("bits", "labels", "blob_count", "contour_count"):
            assert torch.equal(out[k], want.extras[k]), k
