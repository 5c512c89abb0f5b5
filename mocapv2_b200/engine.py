"""Host side of the B200 capture path: device memory, streams and batching around the C-ABI.

PyTorch is plumbing here (HBM allocations, the current CUDA stream, torch.distributed); every computation of the
path happens inside libmocap_b200.so.  `CaptureEngine()` refuses to exist without a CUDA device and the built
library -- there is no CPU path.  (tests/emu/emu_engine.py subclasses the engine to drive the same host logic against the
CPU emulation build of the kernel sources; that is test infrastructure, the package never loads it.)
"""
from __future__ import annotations

import ctypes
import threading
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _cabi

THRESH_U8 = 216          # cv.threshold(x, 255*0.85) on uint8  (lib/ImageOperations.py:29)
MIN_AREA = 500.0         # area > 500                           (lib/ImageOperations.py:50)
MIN_CIRC = 0.5           # circularity > 0.5                    (lib/ImageOperations.py:50)
EPI_CUTOFF = 10.0        # distance_cutoff                      (lib/Helpers.py:219)


def pack_cameras(camera_poses, camera_params) -> np.ndarray:
    """[C, 40] float64 camera records for the C-ABI (layout in include/mocap_b200.h).

    P = K @ [R|t] is formed here in FP64 exactly like lib/Helpers.py:58-62 does per call.
    """
    C = len(camera_poses)
    if len(camera_params) < C:
        raise IndexError("camera_params shorter than camera_poses")      # the reference raises IndexError here too
    out = np.zeros((C, _cabi.CAM_STRIDE), dtype=np.float64)
    for i, pose in enumerate(camera_poses):
        R = np.asarray(pose["R"], dtype=np.float64).reshape(3, 3)
        t = np.asarray(pose["t"], dtype=np.float64).reshape(3)
        K = np.asarray(camera_params[i]["intrinsic_matrix"], dtype=np.float64).reshape(3, 3)
        d = np.zeros(5)
        dd = np.asarray(camera_params[i]["distortion_coef"], dtype=np.float64).ravel()
        d[:min(5, dd.size)] = dd[:5]
        P = K @ np.c_[R, t]
        out[i, 0:12] = P.ravel()
        out[i, 12:21] = R.ravel()
        out[i, 21:24] = t
        out[i, 24:33] = K.ravel()
        out[i, 33:38] = d
    return out


@dataclass
class DetectResult:
    xy: torch.Tensor                 # [n, max_blobs, 2] int32 (float32 sub-pixel centroids), reference output order
    count: torch.Tensor              # [n] int32 (0 == the reference's [[None, None]])
    flags: torch.Tensor              # [n] int32 MOCAP_FLAG_*
    extras: dict = field(default_factory=dict)

    def points(self, i: int):
        """Frame i as the reference returns it: [[x, y], ...] Python ints (floats for sub-pixel centroids), or [[None, None]]."""
        n = int(self.count[i])
        if n == 0:
            return [[None, None]]
        conv = float if self.xy.dtype == torch.float32 else int
        return [[conv(a), conv(b)] for a, b in self.xy[i, :n].tolist()]


@dataclass
class LensSet:
    """Undistortion tables of one or more lenses for one frame size, `stride` bytes apart in one device allocation (MocapLensSet).
    With one lens, `tables` is that lens's table."""
    tables: torch.Tensor             # [n * stride] uint8
    n: int
    stride: int
    H: int
    W: int

    def cabi(self, frame_lens: torch.Tensor | None) -> _cabi.LensSet:
        return _cabi.LensSet(self.tables.data_ptr(), self.n, self.stride, frame_lens.data_ptr() if frame_lens is not None else None)


@dataclass
class CorrespondResult:
    obj: torch.Tensor        # [S, max_pts, 3] float64, sorted by mean error, first n_obj valid
    n_obj: torch.Tensor      # [S]
    img: torch.Tensor        # [S, max_pts, C, 2] in the dtype of the centroid lists (int32 / float32), first n_valid valid (root order)
    n_valid: torch.Tensor    # [S]
    err: torch.Tensor        # [S, max_pts] float64 mean error per complete root (root order)
    flags: torch.Tensor      # [S]
    cand: torch.Tensor | None = None


class CaptureEngine:
    def __init__(self, device=None):
        if not torch.cuda.is_available():
            raise _cabi.MocapError("mocapv2_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.type != "cuda":
            raise _cabi.MocapError("mocapv2_b200 runs on CUDA devices only")
        self.lib = _cabi.load()
        self._init_state()

    def _init_state(self):
        self._tables = {}                       # (lenses, H, W) -> LensSet; table() is the one-lens entry
        # _find_dot is called from one thread per camera (RealtimeTracking_FLIR.py:309): every calling thread owns its workspace
        # (and its detection pipe), keyed by the CUDA stream it launches on, so concurrent calls never share scratch memory and
        # need no lock -- the C-ABI keeps no state.  The lock only guards the shared table cache.
        self._tls = threading.local()
        self._lock = threading.RLock()
        self._launch_base = int(self.lib.mocap_kernel_launch_count())
        self.pipe_workers = 3                   # worker streams of the overlapped detection
        self.last_pipe_info = None

    def clone(self) -> "CaptureEngine":
        """A second engine over the same library, device and undistortion tables with its own per-thread state (workspaces, detection
        pipe): a lane of pipeline.StepsInFlight."""
        other = object.__new__(type(self))
        other.device = self.device
        other.lib = self.lib
        other._init_state()
        other._tables = self._tables
        other._lock = self._lock                 # one lock for the shared table cache
        other.pipe_workers = self.pipe_workers
        return other

    # ---- plumbing ------------------------------------------------------------------------------------------------
    @property
    def launches(self) -> int:
        """Kernels the library has launched since this engine was created (counted inside the library at every launch; all
        engines of a process share the counter)."""
        return int(self.lib.mocap_kernel_launch_count()) - self._launch_base

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _device_ctx(self):
        return torch.cuda.device(self.device)

    def _retire(self, t: torch.Tensor):
        """A buffer about to be dropped stays alive until the current stream has passed the kernels that used it."""
        t.record_stream(torch.cuda.current_stream(self.device))

    # ---- one image from / to the host (the drop-in's per-frame calls; a calling thread owns its stream and staging buffers) ----
    def thread_stream(self):
        """Context manager: the calling thread's own CUDA stream.  The realtime loop calls _find_dot from one thread per camera
        (RealtimeTracking_FLIR.py:309-312); on their own streams the cameras' copies and kernels overlap."""
        st = getattr(self._tls, "stream", None)
        if st is None:
            st = self._tls.stream = torch.cuda.Stream(self.device)
        return torch.cuda.stream(st)

    def _staging(self, shape):
        """Pinned host buffers (in, out) and the device frame of one image shape, owned by the calling thread: the frame goes
        numpy -> pinned -> HBM at PCIe speed instead of through a pageable copy, and comes back the same way."""
        bufs = getattr(self._tls, "bufs", None)
        if bufs is None:
            bufs = self._tls.bufs = {}
        key = tuple(shape)
        if key not in bufs:
            if len(bufs) > 8:
                bufs.clear()
            bufs[key] = (torch.empty(key, dtype=torch.uint8, pin_memory=True), torch.empty(key, dtype=torch.uint8, pin_memory=True),
                         torch.empty((1,) + key, dtype=torch.uint8, device=self.device))
        return bufs[key]

    def upload_image(self, a: np.ndarray) -> torch.Tensor:
        """(H, W) uint8 numpy -> [1, H, W] device tensor, stream-ordered in front of the kernels that read it."""
        pin_in, _, dev = self._staging(a.shape)
        pin_in.numpy()[...] = a
        dev[0].copy_(pin_in, non_blocking=True)
        return dev

    def download_image_async(self, t: torch.Tensor):
        """Queue the copy of a device image (H, W) into the thread's pinned buffer; returns a function that waits for the stream
        and hands out a NEW numpy array (callers draw on it)."""
        _, pin_out, _ = self._staging(t.shape)
        pin_out.copy_(t, non_blocking=True)
        stream = torch.cuda.current_stream(self.device)

        def fetch():
            stream.synchronize()
            return pin_out.numpy().copy()
        return fetch

    def _check_dev(self, t: torch.Tensor, dtype, name):
        if t.device != self.device or t.dtype != dtype or not t.is_contiguous():
            raise ValueError(f"{name}: expected contiguous {dtype} tensor on {self.device}, got {t.dtype} on {t.device}")
        return t

    @staticmethod
    def _ptr(t):
        return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)

    def _workspace(self, nbytes: int) -> torch.Tensor:
        """Scratch memory of the calling thread for the stream it is launching on (grown on demand; a buffer that is replaced
        stays alive until the stream has passed the kernels that used it: record_stream)."""
        d = getattr(self._tls, "ws", None)
        if d is None:
            d = self._tls.ws = {}
        key = int(self._stream().value or 0)
        ws = d.get(key)
        if ws is None or ws.numel() < nbytes:
            if ws is not None:
                self._retire(ws)
            ws = d[key] = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
        return ws

    def empty(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.device)

    # ---- undistortion table ---------------------------------------------------------------------------------------------
    @staticmethod
    def _lens_key(K, dist):
        K = np.ascontiguousarray(np.asarray(K, dtype=np.float64).reshape(9))
        d = np.zeros(5, dtype=np.float64)
        dd = np.asarray(dist, dtype=np.float64).ravel()
        d[:min(5, dd.size)] = dd[:5]
        return K, d

    def _lens_set(self, lenses, H: int, W: int) -> LensSet:
        """The tables of lenses [(K, d), ...] (as _lens_key returns them) in one device allocation, lens i at i * stride; built once
        per list of lenses and frame size."""
        key = (tuple(K.tobytes() + d.tobytes() for K, d in lenses), H, W)
        with self._lock:                       # concurrent first calls (one thread per camera) build the tables once
            ls = self._tables.get(key)
            if ls is None:
                stride = int(self.lib.mocap_undistort_table_bytes(H, W))          # a multiple of 256
                if stride == 0:
                    raise _cabi.MocapError("unsupported frame size")
                tabs = torch.zeros(len(lenses) * stride, dtype=torch.uint8, device=self.device)
                with self._device_ctx():
                    for i, (K, d) in enumerate(lenses):
                        st = self.lib.mocap_undistort_table_build(K.ctypes.data, d.ctypes.data, H, W,
                                                                  ctypes.c_void_p(tabs.data_ptr() + i * stride), stride, self._stream())
                        _cabi.check(self.lib, st, "mocap_undistort_table_build")
                ls = self._tables[key] = LensSet(tabs, len(lenses), stride, H, W)
        return ls

    def table(self, K, dist, H: int, W: int) -> torch.Tensor:
        return self._lens_set([self._lens_key(K, dist)], H, W).tables

    def lens_set(self, camera_params, H: int, W: int) -> LensSet:
        """One undistortion table per entry of camera_params ({"intrinsic_matrix", "distortion_coef"} each, the layout of the
        reference's camera-params.json) in one device allocation: lens i = camera_params[i].  Cached like table()."""
        lenses = [self._lens_key(cp["intrinsic_matrix"], cp["distortion_coef"]) for cp in camera_params]
        if not lenses:
            raise ValueError("a lens set needs at least one lens")
        return self._lens_set(lenses, H, W)

    # ---- detection ----------------------------------------------------------------------------------------------------------
    def default_caps(self, H, W, max_blobs=None, max_contours=None, max_runs=None):
        max_blobs = 256 if max_blobs is None else int(max_blobs)
        max_contours = max(2 * max_blobs, 512) if max_contours is None else int(max_contours)
        max_runs = 4 * H + 4096 if max_runs is None else int(max_runs)
        return max_blobs, max_contours, max_runs

    def _detect_prologue(self, frames, K, dist, lenses, frame_lens, caps, outputs, out, subpixel):
        """What both detection calls check and prepare: contiguous frames and their stride, the caps, the lens set (K / dist: the
        one-lens set of its table) with the per-frame indices as an int32 device tensor [n] (or None: lens 0), and the outputs
        (centroids int32, float32 with subpixel)."""
        if lenses is not None and (K is not None or dist is not None):
            raise ValueError("pass either K / dist or lenses=, not both")
        if lenses is None and (K is None or dist is None):
            raise ValueError("K and dist are needed without lenses=")
        if frames.dim() != 3:
            raise ValueError("frames must be [n, H, W]")
        if frames.device != self.device or frames.dtype != torch.uint8:
            raise ValueError(f"frames must be uint8 on {self.device}")
        n, H, W = frames.shape
        if frames.stride(2) != 1 or frames.stride(1) != W:
            frames = frames.contiguous()
        stride = frames.stride(0) if n > 1 else H * W
        max_blobs, max_contours, max_runs = caps = self.default_caps(H, W, *caps)
        if lenses is None:
            if frame_lens is not None:
                raise ValueError("frame_lens needs lenses=")
            lenses = self._lens_set([self._lens_key(K, dist)], H, W)
        elif (lenses.H, lenses.W) != (H, W):
            raise ValueError(f"lens set built for {lenses.H}x{lenses.W}, frames are {H}x{W}")
        if frame_lens is not None:
            if not isinstance(frame_lens, torch.Tensor):
                frame_lens = torch.as_tensor(np.asarray(frame_lens, dtype=np.int32))
            frame_lens = frame_lens.to(device=self.device, dtype=torch.int32).contiguous()
            if tuple(frame_lens.shape) != (n,):
                raise ValueError(f"frame_lens must be [{n}]")
        xy_dtype = torch.float32 if subpixel else torch.int32
        if out is None:
            out = DetectResult(self.empty((n, max_blobs, 2), xy_dtype), self.empty((n,), torch.int32),
                               self.empty((n,), torch.int32))
        else:
            self._check_dev(out.xy, xy_dtype, "out.xy")                # the centroid format of the call
        ex = out.extras
        if "bits" in outputs and "bits" not in ex:
            ex["bits"] = self.empty((n, H, (W + 31) // 32), torch.int32)
        if "labels" in outputs and "labels" not in ex:
            ex["labels"] = self.empty((n, H, W), torch.int32)
        if "blob_sums" in outputs and "blob_sums" not in ex:
            ex["blob_sums"] = torch.zeros((n, max_blobs, 3), dtype=torch.int64, device=self.device)
            ex["blob_count"] = self.empty((n,), torch.int32)
        if "contours" in outputs and "contours" not in ex:
            ex["contours"] = torch.zeros((n, max_contours, 8), dtype=torch.float64, device=self.device)
            ex["contour_count"] = self.empty((n,), torch.int32)
        return frames, stride, caps, lenses, frame_lens, out

    def detect(self, frames: torch.Tensor, K=None, dist=None, *, thresh=THRESH_U8, min_area=MIN_AREA, min_circ=MIN_CIRC,
               max_blobs=None, max_contours=None, max_runs=None, outputs=(), out: DetectResult | None = None,
               timer=None, lenses: LensSet | None = None, frame_lens=None, subpixel=False) -> DetectResult:
        """_find_dot(img)[1] for a batch (lib/ImageOperations.py:33-78).  frames: [n, H, W] uint8 on the device.

        subpixel=False: int32 centroids, int(m10/m00) like the reference.  subpixel=True: float32 centroids, the float32 nearest to
        m10/m00 (include/mocap_b200.h); everything else is the same.

        outputs: any of "bits", "labels", "blob_sums", "contours" (parity outputs, see include/mocap_b200.h).
        lenses (from lens_set(), in place of K / dist): frame i is undistorted with lens frame_lens[i] ([n] int, None: lens 0);
        an index outside the set gives the frame count 0 and FLAG_LENS_INDEX.
        """
        frames, stride, caps, lenses, fl, out = self._detect_prologue(frames, K, dist, lenses, frame_lens,
                                                                      (max_blobs, max_contours, max_runs), outputs, out, subpixel)
        n, H, W = frames.shape
        ex = out.extras
        nbytes = self.lib.mocap_detect_workspace_bytes(n, H, W, *caps)
        if nbytes == 0:
            raise _cabi.MocapError("mocap_detect_workspace_bytes: unsupported shape")
        ws = self._workspace(nbytes)
        name = "mocap_detect_batch_subpixel" if subpixel else "mocap_detect_batch"
        st = getattr(self.lib, name)(
            self._ptr(frames), n, H, W, stride, ctypes.byref(lenses.cabi(fl)), int(thresh), float(min_area), float(min_circ), *caps,
            self._ptr(out.xy), self._ptr(out.count), self._ptr(out.flags),
            self._ptr(ex.get("bits")), self._ptr(ex.get("labels")), self._ptr(ex.get("blob_sums")),
            self._ptr(ex.get("blob_count")), self._ptr(ex.get("contours")), self._ptr(ex.get("contour_count")),
            self._ptr(ws), nbytes, self._stream(), ctypes.c_void_p(timer) if timer else ctypes.c_void_p(0))
        _cabi.check(self.lib, st, name)
        if fl is not None:
            self._retire(fl)
        # scan, group, filter pieces, candidates, traces+finalize + the general path's mark / compact / tiles / blobs
        return out

    # ---- overlapped detection (chunks: TMA scan of chunk k+1 beside the filter / border stages of chunk k) ----------------------
    def _pipe(self):
        """The calling thread's detection pipe (worker streams + events of the overlapped detection)."""
        key = int(self.pipe_workers)
        pipes = getattr(self._tls, "pipes", None)
        if pipes is None:
            pipes = self._tls.pipes = {}
        if key not in pipes:
            h = self.lib.mocap_detect_pipe_create(key)
            if not h:
                raise _cabi.MocapError("mocap_detect_pipe_create failed")
            pipes[key] = h
        return ctypes.c_void_p(pipes[key])

    def detect_pipelined(self, frames: torch.Tensor, K=None, dist=None, *, thresh=THRESH_U8, min_area=MIN_AREA, min_circ=MIN_CIRC,
                         max_blobs=None, max_contours=None, max_runs=None, outputs=(), out: DetectResult | None = None,
                         chunk_frames=128, timeline=False, cellbox: torch.Tensor | None = None,
                         lenses: LensSet | None = None, frame_lens=None, scatter=None, scan_token=None, subpixel=False) -> DetectResult:
        """Same results as detect() (centroid lists, optionally the contour table), computed chunk by chunk with the streaming
        scan overlapped with the other stages (mocap_detect_batch_pipelined).  cellbox: the frames' hot cell boxes from
        bayer_gr2gray_scan (same thresh) -- the call then has no streaming scan.  lenses / frame_lens as in detect().
        scatter=(xy_dst, count_dst): per-frame destination addresses (int64 device tensors [n]) of the store-to-peer epilogue.
        scan_token=(wait, done): torch.cuda.Event objects (recorded at least once, or None) the call's streaming scan waits for and
        records behind it; StepsInFlight chains the scans of its lanes this way.  subpixel as in detect(); the scatter destinations
        then receive float32 pairs."""
        if any(o != "contours" for o in outputs):
            raise ValueError("detect_pipelined offers the contour table only; use detect() for bits / labels / blob_sums")
        frames, stride, caps, lenses, fl, out = self._detect_prologue(frames, K, dist, lenses, frame_lens,
                                                                      (max_blobs, max_contours, max_runs), outputs, out, subpixel)
        n, H, W = frames.shape
        ex = out.extras
        nbytes = self.lib.mocap_detect_pipelined_workspace_bytes(n, H, W, *caps, int(chunk_frames))
        if nbytes == 0:
            raise _cabi.MocapError("mocap_detect_pipelined_workspace_bytes: unsupported shape")
        ws = self._workspace(nbytes)
        if cellbox is not None:
            if tuple(cellbox.shape) != (n, (H + 31) // 32, (W + 31) // 32):
                raise ValueError("cellbox must be [n, ceil(H/32), ceil(W/32)]")
            self._check_dev(cellbox, torch.int32, "cellbox")
        xy_dst, count_dst = scatter if scatter is not None else (None, None)
        for t in (xy_dst, count_dst):
            if t is not None:
                self._check_dev(t, torch.int64, "scatter")
        wait, done = scan_token if scan_token is not None else (None, None)
        ev = lambda e: ctypes.c_void_p(int(e.cuda_event)) if e is not None else ctypes.c_void_p(0)
        name = "mocap_detect_batch_pipelined_subpixel" if subpixel else "mocap_detect_batch_pipelined"
        st = getattr(self.lib, name)(
            self._pipe(), self._ptr(frames), n, H, W, stride, ctypes.byref(lenses.cabi(fl)), int(thresh), float(min_area), float(min_circ),
            *caps, self._ptr(out.xy), self._ptr(out.count), self._ptr(out.flags), self._ptr(ex.get("contours")),
            self._ptr(ex.get("contour_count")), self._ptr(cellbox), self._ptr(xy_dst), self._ptr(count_dst), ev(wait), ev(done),
            self._ptr(ws), nbytes, self._stream(), int(chunk_frames), 1 if timeline else 0)
        _cabi.check(self.lib, st, name)
        for t in (fl, xy_dst, count_dst):
            if t is not None:
                self._retire(t)
        info = (ctypes.c_int * 2)()
        self.lib.mocap_detect_pipe_info(self._pipe(), info)
        self.last_pipe_info = {"tma_scan": bool(info[0]), "chunks": int(info[1]), "sync_mode": int(info[0])}
        return out

    def pipe_timeline(self):
        """ms since the fork of the last detect_pipelined(timeline=True): {"scan_done", "join", "chunks": [[seen, grouped, filtered, borders], ...]}"""
        buf = (ctypes.c_float * (2 + 4 * 64))()
        k = self.lib.mocap_detect_pipe_timeline(self._pipe(), buf, len(buf))
        if k <= 0:
            return None
        v = [float(x) for x in buf[:k]]
        return {"scan_done": v[0], "join": v[1], "chunks": [v[2 + 4 * c: 6 + 4 * c] for c in range((k - 2) // 4)]}

    def scan_cells(self, frames: torch.Tensor, K, dist, *, thresh=THRESH_U8, variant=0) -> torch.Tensor:
        """The streaming scan alone: hot bounding box of every 32x32 source cell, [n, ceil(H/32), ceil(W/32)] int32 (stage parity)."""
        frames = self._check_dev(frames.contiguous(), torch.uint8, "frames")
        n, H, W = frames.shape
        tab = self.table(K, dist, H, W)
        out = self.empty((n, (H + 31) // 32, (W + 31) // 32), torch.int32)
        ws = self._workspace(4096)
        st = self.lib.mocap_scan_cells_batch(self._ptr(frames), n, H, W, H * W, self._ptr(tab), int(thresh), int(variant),
                                             self._ptr(out), self._ptr(ws), 4096, self._stream())
        _cabi.check(self.lib, st, "mocap_scan_cells_batch")
        return out

    def blobs(self, bits: torch.Tensor, W: int, *, min_area=MIN_AREA, min_circ=MIN_CIRC, max_blobs=None, max_contours=None,
              max_runs=None, outputs=()) -> DetectResult:
        """findContours -> filter -> moments (lib/ImageOperations.py:41-65) on a packed binary image [n, H, ceil(W/32)] int32."""
        bits = self._check_dev(bits, torch.int32, "bits")
        n, H, TX = bits.shape
        if TX != (W + 31) // 32:
            raise ValueError("bits row length does not match W")
        max_blobs, max_contours, max_runs = self.default_caps(H, W, max_blobs, max_contours, max_runs)
        out = DetectResult(self.empty((n, max_blobs, 2), torch.int32), self.empty((n,), torch.int32), self.empty((n,), torch.int32))
        ex = out.extras
        if "labels" in outputs:
            ex["labels"] = self.empty((n, H, W), torch.int32)
        if "blob_sums" in outputs:
            ex["blob_sums"] = torch.zeros((n, max_blobs, 3), dtype=torch.int64, device=self.device)
            ex["blob_count"] = self.empty((n,), torch.int32)
        if "contours" in outputs:
            ex["contours"] = torch.zeros((n, max_contours, 8), dtype=torch.float64, device=self.device)
            ex["contour_count"] = self.empty((n,), torch.int32)
        nbytes = self.lib.mocap_detect_workspace_bytes(n, H, W, max_blobs, max_contours, max_runs)
        if nbytes == 0:
            raise _cabi.MocapError("mocap_detect_workspace_bytes: unsupported shape")
        ws = self._workspace(nbytes)
        st = self.lib.mocap_blobs_batch(
            self._ptr(bits), n, H, W, float(min_area), float(min_circ), max_blobs, max_contours, max_runs,
            self._ptr(out.xy), self._ptr(out.count), self._ptr(out.flags), self._ptr(ex.get("labels")),
            self._ptr(ex.get("blob_sums")), self._ptr(ex.get("blob_count")), self._ptr(ex.get("contours")),
            self._ptr(ex.get("contour_count")), self._ptr(ws), nbytes, self._stream())
        _cabi.check(self.lib, st, "mocap_blobs_batch")
        return out

    def filter(self, frames: torch.Tensor, K, dist, *, thresh=THRESH_U8) -> torch.Tensor:
        """undistort -> image_filter_gpu (lib/ImageOperations.py:38-40, 23-31): packed binary image [n, H, ceil(W/32)]."""
        n, H, W = frames.shape
        frames = self._check_dev(frames.contiguous(), torch.uint8, "frames")
        tab = self.table(K, dist, H, W)
        bits = self.empty((n, H, (W + 31) // 32), torch.int32)
        nbytes = self.lib.mocap_detect_workspace_bytes(n, H, W, 1, 1, 1)
        ws = self._workspace(nbytes)
        st = self.lib.mocap_filter_batch(self._ptr(frames), n, H, W, H * W, self._ptr(tab), int(thresh), self._ptr(bits),
                                         self._ptr(ws), nbytes, self._stream())
        _cabi.check(self.lib, st, "mocap_filter_batch")
        return bits

    def draw_contours(self, img: torch.Tensor, res: DetectResult, value=0) -> torch.Tensor:
        """cv.drawContours(img, kept contours, -1, colour, 2) of _find_dot (lib/ImageOperations.py:52-55), in place on img [n, H, W]
        uint8; res must carry the "bits" and "contours" outputs of detect()."""
        img = self._check_dev(img, torch.uint8, "img")
        n, H, W = img.shape
        ex = res.extras
        if "bits" not in ex or "contours" not in ex:
            raise ValueError('draw_contours needs detect(..., outputs=("bits", "contours"))')
        st = self.lib.mocap_draw_contours_batch(self._ptr(ex["bits"]), self._ptr(ex["contours"]), self._ptr(ex["contour_count"]), n, H, W,
                                                int(ex["contours"].shape[1]), self._ptr(img), int(value), self._stream())
        _cabi.check(self.lib, st, "mocap_draw_contours_batch")
        return img

    def blur5(self, frames: torch.Tensor) -> torch.Tensor:
        """fast_cuda_blur(image, 5) (lib/CudaOperations.py:24-41) for a batch [n, H, W] uint8."""
        frames = self._check_dev(frames.contiguous(), torch.uint8, "frames")
        n, H, W = frames.shape
        out = torch.empty_like(frames)
        _cabi.check(self.lib, self.lib.mocap_blur5_batch(self._ptr(frames), n, H, W, self._ptr(out), self._stream()), "mocap_blur5_batch")
        return out

    def median5_threshold(self, frames: torch.Tensor, thresh=THRESH_U8) -> torch.Tensor:
        """image_filter_cpu (lib/ImageOperations.py:15-21): cv.medianBlur(5) -> cv.threshold for a batch [n, H, W] uint8."""
        frames = self._check_dev(frames.contiguous(), torch.uint8, "frames")
        n, H, W = frames.shape
        out = torch.empty_like(frames)
        _cabi.check(self.lib, self.lib.mocap_median5_threshold_batch(self._ptr(frames), n, H, W, int(thresh), self._ptr(out), self._stream()),
                    "mocap_median5_threshold_batch")
        return out

    def bayer_gr2gray(self, raw: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """cvtColor(BAYER_GR2BGR) -> cvtColor(BGR2GRAY) (RealtimeTracking_FLIR.py:103-104) for raw sensor frames [n, H, W] uint8."""
        raw = self._check_dev(raw.contiguous(), torch.uint8, "raw")
        n, H, W = raw.shape
        if out is None:
            out = torch.empty_like(raw)
        elif out.shape != raw.shape:
            raise ValueError("out must have the shape of raw")
        else:
            self._check_dev(out, torch.uint8, "out")
        _cabi.check(self.lib, self.lib.mocap_bayer_gr2gray_batch(self._ptr(raw), n, H, W, self._ptr(out), self._stream()),
                    "mocap_bayer_gr2gray_batch")
        return out

    def bayer_gr2gray_scan(self, raw: torch.Tensor, out: torch.Tensor | None = None, *, thresh=THRESH_U8,
                           cellbox: torch.Tensor | None = None):
        """bayer_gr2gray that also returns the hot cell boxes of the grey frames ([n, ceil(H/32), ceil(W/32)] int32, what scan_cells
        computes from them): detect_pipelined(grey, ..., cellbox=...) then skips its streaming scan (mocap_bayer_gr2gray_scan_batch)."""
        raw = self._check_dev(raw.contiguous(), torch.uint8, "raw")
        n, H, W = raw.shape
        if out is None:
            out = torch.empty_like(raw)
        elif out.shape != raw.shape:
            raise ValueError("out must have the shape of raw")
        else:
            self._check_dev(out, torch.uint8, "out")
        cells = (n, (H + 31) // 32, (W + 31) // 32)
        if cellbox is None:
            cellbox = self.empty(cells, torch.int32)
        elif tuple(cellbox.shape) != cells:
            raise ValueError("cellbox must be [n, ceil(H/32), ceil(W/32)]")
        else:
            self._check_dev(cellbox, torch.int32, "cellbox")
        nbytes = cells[0] * cells[1] * cells[2] * 8
        tls = self._tls
        mask = getattr(tls, "bayer_mask", None)                   # its own scratch: the detection workspace is in use by calls in flight
        if mask is None or mask.numel() < nbytes:
            mask = tls.bayer_mask = self.empty((nbytes,), torch.uint8)
        _cabi.check(self.lib, self.lib.mocap_bayer_gr2gray_scan_batch(self._ptr(raw), n, H, W, self._ptr(out), int(thresh), self._ptr(cellbox),
                                                                      self._ptr(mask), nbytes, self._stream()),
                    "mocap_bayer_gr2gray_scan_batch")
        return out, cellbox

    def undistort(self, frames: torch.Tensor, K, dist) -> torch.Tensor:
        """cv.undistort(img, K, dist) (lib/ImageOperations.py:38) for a batch [n, H, W] uint8."""
        frames = self._check_dev(frames.contiguous(), torch.uint8, "frames")
        n, H, W = frames.shape
        tab = self.table(K, dist, H, W)
        out = torch.empty_like(frames)
        _cabi.check(self.lib, self.lib.mocap_undistort_batch(self._ptr(frames), n, H, W, self._ptr(tab), self._ptr(out), self._stream()),
                    "mocap_undistort_batch")
        return out

    # ---- per-stage timing (bench) ---------------------------------------------------------------------------------------------
    def stage_timer(self):
        t = self.lib.mocap_stage_timer_create()
        if not t:
            raise _cabi.MocapError("mocap_stage_timer_create failed")
        return t

    def stage_timer_read(self, timer, destroy=True):
        ms = (ctypes.c_float * _cabi.N_STAGES)()
        _cabi.check(self.lib, self.lib.mocap_stage_timer_read(ctypes.c_void_p(timer), ms), "mocap_stage_timer_read")
        if destroy:
            self.lib.mocap_stage_timer_destroy(ctypes.c_void_p(timer))
        return {self.lib.mocap_stage_name(i).decode(): float(ms[i]) for i in range(_cabi.N_STAGES)}

    # ---- geometry -----------------------------------------------------------------------------------------------------------
    def cameras(self, camera_poses, camera_params) -> torch.Tensor:
        return torch.from_numpy(pack_cameras(camera_poses, camera_params)).to(self.device)

    def triangulate(self, pts: torch.Tensor, cams: torch.Tensor, valid: torch.Tensor | None = None, *, want_err=True,
                    xyz: torch.Tensor | None = None, err: torch.Tensor | None = None):
        """triangulate_points + calculate_reprojection_errors (lib/Helpers.py:43-143) for pts [P, C, 2] (f32 or f64)."""
        if pts.dtype not in (torch.float32, torch.float64):
            raise ValueError("pts must be float32 (main mode) or float64 (check mode)")
        pts = self._check_dev(pts, pts.dtype, "pts")
        cams = self._check_dev(cams, torch.float64, "cams")
        P, C, _ = pts.shape
        if valid is not None:
            valid = self._check_dev(valid, torch.uint8, "valid")
        if xyz is None:
            xyz = self.empty((P, 3), pts.dtype)
        if err is None and want_err:
            err = self.empty((P,), pts.dtype)
        if P == 0:                                  # triangulate_points([]) -> np.array([]) (Helpers.py:87-99)
            return xyz, err
        st = self.lib.mocap_triangulate_batch(self._ptr(pts), self._ptr(valid), self._ptr(cams), C, P,
                                              1 if pts.dtype == torch.float64 else 0, self._ptr(xyz), self._ptr(err), self._stream())
        _cabi.check(self.lib, st, "mocap_triangulate_batch")
        return xyz, err

    def ba_residuals(self, pts: torch.Tensor, cams_sets: torch.Tensor) -> torch.Tensor:
        """bundle_adjustment's residual (lib/Helpers.py:160-167) for several pose hypotheses in one launch, FP64:
        pts [P, C, 2] float64 (all views valid), cams_sets [S, C, 40] float64 -> mean squared reprojection errors [S, P]."""
        pts = self._check_dev(pts, torch.float64, "pts")
        cams_sets = self._check_dev(cams_sets, torch.float64, "cams_sets")
        P, C, _ = pts.shape
        S = cams_sets.shape[0]
        err = self.empty((S, P), torch.float64)
        if P == 0:
            return err
        st = self.lib.mocap_ba_residuals_batch(self._ptr(pts), self._ptr(cams_sets), S, C, P, self._ptr(err), self._stream())
        _cabi.check(self.lib, st, "mocap_ba_residuals_batch")
        return err

    def reproject(self, pts: torch.Tensor, xyz: torch.Tensor, cams: torch.Tensor, valid: torch.Tensor | None = None):
        """calculate_reprojection_errors (lib/Helpers.py:102-143) for given object points."""
        pts = self._check_dev(pts, pts.dtype, "pts")
        xyz = self._check_dev(xyz, pts.dtype, "xyz")
        cams = self._check_dev(cams, torch.float64, "cams")
        P, C, _ = pts.shape
        if valid is not None:
            valid = self._check_dev(valid, torch.uint8, "valid")
        err = self.empty((P,), pts.dtype)
        if P == 0:
            return err
        st = self.lib.mocap_reproject_batch(self._ptr(pts), self._ptr(valid), self._ptr(xyz), self._ptr(cams), C, P,
                                            1 if pts.dtype == torch.float64 else 0, self._ptr(err), self._stream())
        _cabi.check(self.lib, st, "mocap_reproject_batch")
        return err

    def correspond(self, xy: torch.Tensor, count: torch.Tensor, Fs: torch.Tensor, cams: torch.Tensor, *, obj_count=0,
                   cutoff=EPI_CUTOFF, max_groups=4096, fp64=False, want_cand=False, out: CorrespondResult | None = None) -> CorrespondResult:
        """find_point_correspondance_and_object_points (lib/Helpers.py:178-280) for S frame-sets.

        xy [S, C, max_pts, 2] centroid lists, count [S, C] int32, Fs [C-1, 3, 3] float64 (Fs[i-1]: camera 0 -> camera i).
        xy is int32 (whole-pixel centroids) or float32 (sub-pixel, detect(subpixel=True)); res.img has the dtype of xy.
        Camera-blocked input (what the shard exchange of the multi-GPU pipeline delivers) is read in place:
        xy [B, S, C/B, max_pts, 2], count [B, S, C/B] with block b holding cameras b*C/B .. (b+1)*C/B - 1.
        """
        if xy.dtype not in (torch.int32, torch.float32):
            raise ValueError(f"xy: centroid lists must be int32 or float32, not {xy.dtype}")
        xy = self._check_dev(xy, xy.dtype, "xy")
        count = self._check_dev(count, torch.int32, "count")
        cams = self._check_dev(cams, torch.float64, "cams")
        if xy.dim() == 5:
            B, S, cpb, max_pts, _ = xy.shape
            C = B * cpb
            if tuple(count.shape) != (B, S, cpb):
                raise ValueError("count must be [B, S, C/B] for camera-blocked xy")
        else:
            S, C, max_pts, _ = xy.shape
            cpb = C
        if C > 1:
            Fs = self._check_dev(Fs, torch.float64, "Fs")
            if Fs.shape[0] < C - 1:
                raise IndexError("Fs shorter than camera count - 1")        # the reference raises IndexError (Helpers.py:206)
        res = out if out is not None else CorrespondResult(
            obj=torch.zeros((S, max_pts, 3), dtype=torch.float64, device=self.device), n_obj=self.empty((S,), torch.int32),
            img=torch.zeros((S, max_pts, C, 2), dtype=xy.dtype, device=self.device), n_valid=self.empty((S,), torch.int32),
            err=torch.zeros((S, max_pts), dtype=torch.float64, device=self.device), flags=self.empty((S,), torch.int32),
            cand=self.empty((S, max_pts, C, _cabi.MAX_CAND), torch.int32) if want_cand else None)
        if out is not None:
            self._check_dev(res.img, xy.dtype, "out.img")              # written in the centroid format of xy
        if S == 0:
            return res
        nbytes = self.lib.mocap_correspond_workspace_bytes(S, C, max_pts, max_groups)
        ws = self._workspace(nbytes)
        name = "mocap_correspond_batch_subpixel" if xy.dtype == torch.float32 else "mocap_correspond_batch_blocked"
        st = getattr(self.lib, name)(
            self._ptr(xy), self._ptr(count), S, C, max_pts, cpb, self._ptr(Fs) if C > 1 else ctypes.c_void_p(0), self._ptr(cams),
            float(cutoff), int(obj_count), int(max_groups), 1 if fp64 else 0,
            self._ptr(res.obj), self._ptr(res.n_obj), self._ptr(res.img), self._ptr(res.n_valid), self._ptr(res.err),
            self._ptr(res.cand), self._ptr(res.flags), self._ptr(ws), nbytes, self._stream())
        _cabi.check(self.lib, st, name)
        return res


_default_engine = None
_default_lock = threading.Lock()


def default_engine() -> CaptureEngine:
    """Process-wide engine on the current CUDA device (created on first use; raises without CUDA)."""
    global _default_engine
    with _default_lock:
        if _default_engine is None:
            _default_engine = CaptureEngine()
        return _default_engine


def set_default_engine(engine: CaptureEngine | None):
    global _default_engine
    with _default_lock:
        _default_engine = engine
