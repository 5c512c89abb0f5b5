"""B200 drop-in for the reference's lib/ImageOperations.py (frame -> blob centroids).

Same names and conventions as the reference module:
  _find_dot(img, print_location=False, return_filtered=False) -> (img, image_points)   lib/ImageOperations.py:33-78
    (+ keyword camera_number: undistort with that camera's calibration instead of camera 0's;
     keyword subpixel: float centroids m10/m00 rounded to float32 instead of int(m10/m00))
  image_filter_gpu(image, camera_number=0)                                             lib/ImageOperations.py:23-31
  module globals `camera_params`, `intrinsics_json`, `cuda_lock` stay assignable.
All arithmetic runs in libmocap_b200.so on the GPU (undistort + 5x5 floor-mean + threshold + 5x5 majority +
contour-polygon centroids, bit-exact with the reference's cv2/numba path); without CUDA every call raises.
"""
import json
import threading

import numpy as np

from .. import _cabi
from .. import engine as _engine

cuda_lock = threading.Lock()           # kept for API compatibility (lib/ImageOperations.py:9); the engine serialises itself

intrinsics_json = "./jsons/camera-params-in.json"      # lib/ImageOperations.py:11 (cwd-relative, like the reference)
camera_params = None                   # the reference loads this at import; here on first use, still overridable

ANNOTATE = True                        # draw the reference's display-only overlays when cv2 is importable


def _params():
    global camera_params
    if camera_params is None:
        with open(intrinsics_json) as f:
            camera_params = json.load(f)
    return camera_params


def _to_device(img, eng):
    a = np.ascontiguousarray(img)
    if a.dtype != np.uint8 or a.ndim != 2:
        raise ValueError("expected a single-channel uint8 image (H, W)")
    return eng.upload_image(a)


def _to_host(t, eng):
    """Device image (H, W) uint8 -> a NEW numpy array (callers draw on it), through the calling thread's pinned buffer."""
    return eng.download_image_async(t)()


def bayer_gr_to_gray(image):
    """The two cv2.cvtColor calls in front of _find_dot in the realtime loop (RealtimeTracking_FLIR.py:103-104), on the GPU:
    raw BayerGR sensor frame (H, W) uint8 -> grey (H, W) uint8, bit-identical to OpenCV's."""
    eng = _engine.default_engine()
    return _to_host(eng.bayer_gr2gray(_to_device(image, eng))[0], eng)


def image_filter_cpu(image, camera_number=0):
    """medianBlur(5) -> threshold(255*0.85): uint8 {0,255} image (lib/ImageOperations.py:15-21; no callers in the reference).

    Kept under its reference name; it runs on the GPU like everything else here.  `camera_number` is ignored."""
    eng = _engine.default_engine()
    return _to_host(eng.median5_threshold(_to_device(image, eng))[0], eng)


def image_filter_gpu(image, camera_number=0):
    """fast_cuda_blur(5) -> threshold(255*0.85) -> medianBlur(5): uint8 {0,255} image (lib/ImageOperations.py:23-31).

    `camera_number` is ignored exactly like in the reference.  No undistortion here (identity map)."""
    eng = _engine.default_engine()
    fr = _to_device(image, eng)
    H, W = fr.shape[1:]
    bits = eng.filter(fr, np.eye(3), np.zeros(5))[0]
    b = bits.cpu().numpy().view(np.uint8)
    return (np.unpackbits(b, axis=1, bitorder="little")[:, :W] * 255).astype(np.uint8)


def _detect_one(eng, fr, K, dist, outputs, subpixel):
    """eng.detect on one frame; capacity overflows (MOCAP_FLAG_*_OVERFLOW: more blobs / contours / runs than the default
    caps hold) are never returned as a silently short list -- the call is repeated with larger caps, like the reference,
    which has none (lib/ImageOperations.py:41-65)."""
    caps = {}
    for attempt in range(6):
        res = eng.detect(fr, K, dist, outputs=outputs, subpixel=subpixel, **caps)
        flags = int(res.flags[0])                              # device -> host read of the result
        if not flags & _cabi.FLAG_ERRORS:
            return res
        H, W = fr.shape[1:]
        mb, mc, mr = eng.default_caps(H, W, caps.get("max_blobs"), caps.get("max_contours"), caps.get("max_runs"))
        caps = {"max_blobs": 4 * mb, "max_contours": 4 * mc, "max_runs": 4 * mr}
    raise _cabi.MocapError(f"_find_dot: detection capacity exceeded even with caps {caps} (flags {flags})")


def _find_dot(img, print_location=False, return_filtered=False, *, camera_number=None, subpixel=False):
    """output: image with dot and dot coordinates -- (img, [[x, y], ...]) or (img, [[None, None]]).

    camera_number=None undistorts with camera 0's calibration, like lib/ImageOperations.py:36-38; an integer selects
    camera_params[camera_number] (the lens of the camera the frame comes from; a short list raises IndexError).
    subpixel=False returns int(m10/m00), int(m01/m00) like the reference (:59-62); subpixel=True returns Python floats, the
    float32 nearest to m10/m00 and m01/m00 -- the same blobs in the same order, without the reference's truncation bias of about
    half a pixel.  find_point_correspondance_and_object_points takes either."""
    eng = _engine.default_engine()
    cp = _params()[0 if camera_number is None else camera_number]
    K = np.array(cp["intrinsic_matrix"], dtype=np.float64)
    dist = np.array(cp["distortion_coef"], dtype=np.float64)
    with eng.thread_stream():
        fr = _to_device(img, eng)
        H, W = fr.shape[1:]
        if not ANNOTATE and not return_filtered:
            # everything of the call is queued before the first host read: H2D, the undistorted image and its way back, detection
            fetch = eng.download_image_async(eng.undistort(fr, K, dist)[0])
            res = _detect_one(eng, fr, K, dist, (), subpixel)
        else:
            # with the reference's overlays: the contour outline needs the binary image and the contour table of the same call
            res = _detect_one(eng, fr, K, dist, ("bits", "contours"), subpixel)
            if return_filtered:                               # the reference then draws on (and returns) the filtered image (:53)
                b = res.extras["bits"][0].cpu().numpy().view(np.uint8)
                canvas = eng.upload_image((np.unpackbits(b, axis=1, bitorder="little")[:, :W] * 255).astype(np.uint8))
            else:
                canvas = eng.undistort(fr, K, dist)
            if ANNOTATE:
                eng.draw_contours(canvas, res)                # cv.drawContours(..., (0, 0, 255), 2): 0 on a one-channel image
            fetch = eng.download_image_async(canvas[0])
        n = int(res.count[0])
        image_points = res.xy[0, :n].tolist() if n else []
        out = fetch()
    if ANNOTATE and image_points:
        try:                                                  # display-only overlays (lib/ImageOperations.py:67-73)
            import cv2 as cv
            for i, (x, y) in enumerate(image_points):
                x, y = int(x), int(y)                         # (sub-pixel centroids: drawn at the truncated pixel)
                label = f"({x}, {y})" if print_location else str(i)
                org = (x - 240, y - 15) if print_location else (x - 20, y - 15)
                cv.putText(out, label, org, cv.FONT_HERSHEY_SIMPLEX, 2, (0, 0, 255), 4)
                cv.circle(out, (x, y), 2, (0, 255, 0), 8)
        except ImportError:
            pass
    if len(image_points) == 0:
        image_points = [[None, None]]
    return out, image_points
