"""Batched capture pipeline over one or several GPUs: detect -> (exchange centroid lists) -> match + triangulate.

Sharding (SURVEY.md section 8e): detection is independent per (camera, frame) and is sharded by CAMERA, so a rank keeps
its cameras' frames (and their undistortion table) resident; matching needs every camera's centroid list of a
frame-set and is sharded by FRAME-SET.  The one exchange step in between moves, per pair of ranks, exactly the records
the receiver needs -- the sender's cameras of the receiver's frame-sets, a contiguous slice of the detection output --
as ONE grouped NCCL send/recv (ncclGroupStart/End: a single launch over NVLink; gloo in the CPU tests).  Each rank
receives 1/N of what an all-gather would deliver, and the receive buffer [source rank][frame-set][camera][blob] is read
in place by the correspondence kernels (camera-blocked layout, mocap_correspond_batch_blocked): no pack, permute or copy
kernels on the step path.  No floating-point reduction crosses ranks, so N-rank outputs are bit-identical to 1-rank.

On a GPU box with peer access (NVLink / NVSwitch) the exchange needs no collective at all: the receive buffers live in
torch symmetric memory, every rank maps its peers' buffers, and the overlapped detection call stores each frame's record
straight into the slot of the rank that matches its frame-set, chunk by chunk behind the chunk's border stage
(`detect_pipelined(scatter=...)`: store-to-peer epilogue).  The exchange step is then one symmetric-memory barrier; two
receive buffers alternate so that a rank may already store step t + 1 while a peer still matches step t.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch
import torch.distributed as dist

from .engine import CaptureEngine, CorrespondResult, DetectResult


@dataclass
class StepResult:
    det: DetectResult                 # this rank's cameras, all frame-sets: [FS * cams_local, ...]
    corr: CorrespondResult            # this rank's frame-set shard, all cameras
    fs_begin: int                     # first frame-set of the shard
    fs_end: int


class CapturePipeline:
    def __init__(self, engine: CaptureEngine, rig: dict, *, max_blobs=160, obj_count=None, max_groups=64, fp64=False,
                 group=None, lens="camera0", centroids="int"):
        self.eng = engine
        self.rig = rig
        self.C = len(rig["poses"])
        self.H, self.W = rig["H"], rig["W"]
        self.max_blobs = int(max_blobs)
        self.obj_count = self.max_blobs if obj_count is None else int(obj_count)
        self.max_groups = int(max_groups)
        self.fp64 = fp64
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        if self.C % self.world:
            raise ValueError(f"{self.C} cameras do not shard over {self.world} ranks")
        self.cams_local = self.C // self.world
        self.cam_begin = self.rank * self.cams_local
        # lens="camera0": _find_dot undistorts with camera 0's calibration for every camera (lib/ImageOperations.py:36-38).
        # lens="per_camera": every camera's frames with its own calibration -- a lens set of this rank's cameras, frame i of the
        # [FS][cams_local] batch takes lens i % cams_local.
        if lens not in ("camera0", "per_camera"):
            raise ValueError(f"lens must be 'camera0' or 'per_camera', not {lens!r}")
        self.lens = lens
        # centroids="int": int(m10/m00) like _find_dot (lib/ImageOperations.py:59-62).  centroids="subpixel": the float32 nearest to
        # m10/m00 -- the same 8-byte records, so the exchange moves the same bytes; the matching then reads float32 lists.
        if centroids not in ("int", "subpixel"):
            raise ValueError(f"centroids must be 'int' or 'subpixel', not {centroids!r}")
        self.centroids = centroids
        self.subpixel = centroids == "subpixel"
        self.xy_dtype = torch.float32 if self.subpixel else torch.int32
        self.K0 = np.asarray(rig["camera_params"][0]["intrinsic_matrix"], dtype=np.float64)
        self.dist0 = np.asarray(rig["camera_params"][0]["distortion_coef"], dtype=np.float64)
        self.lenses = None
        self._frame_lens = None                 # cached [n] int32 device tensor of the lens indices
        if lens == "per_camera":
            self.lenses = engine.lens_set(rig["camera_params"][self.cam_begin:self.cam_begin + self.cams_local], self.H, self.W)
        self.cams = engine.cameras(rig["poses"], rig["camera_params"])
        self.Fs = torch.from_numpy(np.asarray(rig["Fs"], dtype=np.float64).reshape(-1, 3, 3).copy()).to(engine.device)
        self._det = None
        self._rx = None
        self.collectives = 0
        # store-to-peer exchange (symmetric memory): tried once on the first overlapped detection of a multi-rank CUDA pipeline
        self.peer_exchange = True
        self._peer = None                       # {"bufs", "hdls", "tables", "views", "turn", "n", "per"}
        # overlapped detection (engine.detect_pipelined) for batches large enough to pipeline: 8 chunks on 6 worker streams
        # (chunks x workers sweep on the C4 batch, profiles/r2_pipe_probe.log: 1.75 ms against 2.03 ms for the one-shot call;
        # 4 chunks / 4 workers 1.78 ms; tools/stage_probe.py --grid chunks,workers times other splits)
        self.scan_token = None                  # (wait, done) events of the coming overlapped detection, set by StepsInFlight
        self.pipelined_min_frames = 256
        self.engine_pipe = {"workers": 6, "chunks": 8}

    def frame_set_shard(self, n_frame_sets: int):
        if n_frame_sets % self.world:
            raise ValueError("frame-sets must divide evenly over the ranks")
        per = n_frame_sets // self.world
        return self.rank * per, (self.rank + 1) * per

    def _buffers(self, n: int):
        """Detection outputs of n frames [FS * cams_local, ...] (frame-set major: the slice of a destination rank is contiguous)."""
        if self._det is None or self._det.xy.shape[0] != n:
            mb = self.max_blobs
            self._det = DetectResult(torch.zeros((n, mb, 2), dtype=self.xy_dtype, device=self.eng.device),
                                     torch.zeros(n, dtype=torch.int32, device=self.eng.device),
                                     torch.zeros(n, dtype=torch.int32, device=self.eng.device))
            self._rx = None
        return self._det

    def _lens_args(self, n: int):
        """The lens keyword arguments of a detection call of n frames: K, dist or the lens set with the per-frame indices."""
        if self.lenses is None:
            return {"K": self.K0, "dist": self.dist0}
        if self._frame_lens is None or self._frame_lens.shape[0] != n:
            self._frame_lens = (torch.arange(n, dtype=torch.int32) % self.cams_local).to(self.eng.device)
        return {"lenses": self.lenses, "frame_lens": self._frame_lens}

    def detect(self, frames: torch.Tensor, timer=None, pipelined=None, timeline=False, cellbox=None) -> DetectResult:
        """frames [FS, cams_local, H, W] uint8 on the device -> centroid lists of this rank's cameras.  cellbox: the frames' hot cell
        boxes from CaptureEngine.bayer_gr2gray_scan (raw sensor input): the overlapped call then runs without its streaming scan."""
        FS, cl, H, W = frames.shape
        assert cl == self.cams_local and (H, W) == (self.H, self.W)
        flat = frames.view(FS * cl, H, W)
        n = FS * cl
        if pipelined is None:
            pipelined = cellbox is not None or (timer is None and n >= self.pipelined_min_frames)
        if cellbox is not None and not pipelined:
            raise ValueError("cellbox is taken by the overlapped detection call only")
        buf = self._buffers(n)
        lens_kw = self._lens_args(n)
        buf.extras.pop("peer_turn", None)                          # (set below when this call stores its records to the peers)
        if pipelined:
            self.eng.pipe_workers = self.engine_pipe["workers"]
            chunk = -(-n // self.engine_pipe["chunks"])
            peer = self._peer_setup(FS) if (self.world > 1 and self.peer_exchange) else None
            if peer is not None:
                peer["turn"] ^= 1
            self._det = self.eng.detect_pipelined(flat, max_blobs=self.max_blobs, out=buf, chunk_frames=chunk, timeline=timeline,
                                                  cellbox=cellbox, scatter=peer["tables"][peer["turn"]] if peer is not None else None,
                                                  scan_token=self.scan_token, subpixel=self.subpixel, **lens_kw)
            if peer is not None:
                self._det.extras["peer_turn"] = peer["turn"]       # the result knows which receive buffers hold its records
        else:
            self._det = self.eng.detect(flat, max_blobs=self.max_blobs, out=buf, timer=timer, subpixel=self.subpixel, **lens_kw)
        return self._det

    def _peer_setup(self, FS: int):
        """Symmetric receive buffers + the per-frame destination tables of the store-to-peer epilogue (collective, once per shape).
        Returns None -- and the pipeline keeps the NCCL exchange -- where symmetric memory is not available."""
        cl, mb = self.cams_local, self.max_blobs
        b, e = self.frame_set_shard(FS)
        per = e - b
        if self._peer is not None and self._peer["per"] == per:
            return self._peer
        if self._peer is False or self.eng.device.type != "cuda":
            return None
        try:
            import torch.distributed._symmetric_memory as symm
            group = self.group if self.group is not None else dist.group.WORLD
            xy_elems = self.world * per * cl * mb * 2
            cnt_elems = self.world * per * cl
            bufs, hdls, tables, views = [], [], [], []
            s_idx = torch.arange(FS).repeat_interleave(cl)                 # frame-set of local frame i = s * cl + c
            c_idx = torch.arange(cl).repeat(FS)
            dst = s_idx // per
            slot = (self.rank * per + s_idx % per) * cl + c_idx            # [source rank][frame-set of the shard][camera]
            for _ in range(2):
                buf = symm.empty(xy_elems + cnt_elems, dtype=torch.int32, device=self.eng.device)
                buf.zero_()
                hdl = symm.rendezvous(buf, group)
                base = torch.tensor([int(p) for p in hdl.buffer_ptrs], dtype=torch.int64)
                xy_dst = (base[dst] + slot * (mb * 2 * 4)).to(self.eng.device)
                cnt_dst = (base[dst] + (xy_elems + slot) * 4).to(self.eng.device)
                bufs.append(buf); hdls.append(hdl); tables.append((xy_dst, cnt_dst))
                views.append((buf[:xy_elems].view(self.xy_dtype).view(self.world, per, cl, mb, 2), buf[xy_elems:].view(self.world, per, cl)))
            self._peer = {"bufs": bufs, "hdls": hdls, "tables": tables, "views": views, "turn": 1, "per": per}
        except Exception as ex:                                            # no peer mapping on this box: NCCL send/recv it is
            import warnings
            warnings.warn(f"store-to-peer exchange unavailable ({ex!r}); using the NCCL exchange")
            self._peer = False
            return None
        return self._peer

    def exchange(self, det: DetectResult, FS: int):
        """The exchange step: returns (xy, count) of this rank's frame-set shard for ALL cameras, camera-blocked by source rank:
        xy [world, F0, cams_local, max_blobs, 2], count [world, F0, cams_local] (world == 1: [F0, C, ...], nothing moves)."""
        cl, mb = self.cams_local, self.max_blobs
        b, e = self.frame_set_shard(FS)
        per = e - b
        if self.world == 1:
            return det.xy.view(FS, cl, mb, 2), det.count.view(FS, cl)
        turn = det.extras.pop("peer_turn", None) if self._peer else None
        if turn is not None:
            # the records are already where their consumers read them (store-to-peer epilogue of the detection): wait for the peers
            peer = self._peer
            peer["hdls"][turn].barrier(channel=0)
            self.collectives += 1
            return peer["views"][turn]
        if self._rx is None or self._rx[0].shape[1] != per:
            self._rx = (torch.empty((self.world, per, cl, mb, 2), dtype=self.xy_dtype, device=self.eng.device),
                        torch.empty((self.world, per, cl), dtype=torch.int32, device=self.eng.device))
        rxy, rcnt = self._rx
        sxy = det.xy.view(self.world, per, cl, mb, 2)                  # [destination rank][its frame-sets][my cameras]
        scnt = det.count.view(self.world, per, cl)
        ops = []
        for k in range(1, self.world):                                 # every pair once per direction, self excluded
            dst = (self.rank + k) % self.world
            src = (self.rank - k) % self.world
            gd = dist.get_global_rank(self.group, dst) if self.group is not None else dst
            gs = dist.get_global_rank(self.group, src) if self.group is not None else src
            ops += [dist.P2POp(dist.isend, sxy[dst], gd, self.group), dist.P2POp(dist.isend, scnt[dst], gd, self.group),
                    dist.P2POp(dist.irecv, rxy[src], gs, self.group), dist.P2POp(dist.irecv, rcnt[src], gs, self.group)]
        reqs = dist.batch_isend_irecv(ops)                             # NCCL: one group = one launch
        rxy[self.rank].copy_(sxy[self.rank])                           # my own cameras of my own frame-sets: two small local copies
        rcnt[self.rank].copy_(scnt[self.rank])
        for r in reqs:
            r.wait()                                                   # (NCCL: orders the current stream after the transfer, no host sync)
        self.collectives += 1
        return rxy, rcnt

    def step(self, frames: torch.Tensor) -> StepResult:
        FS = frames.shape[0]
        det = self.detect(frames)
        xy, count = self.exchange(det, FS)
        corr = self.eng.correspond(xy, count, self.Fs, self.cams, obj_count=self.obj_count, max_groups=self.max_groups,
                                   fp64=self.fp64)
        b, e = self.frame_set_shard(FS)
        return StepResult(det, corr, b, e)


class StepsInFlight:
    """`depth` steps of a capture pipeline in flight at once (batch throughput): every lane is a CapturePipeline of its own -- own
    engine state (detection pipe with its worker streams, workspace), own output / receive buffers, own CUDA stream -- over the
    same rig and the same undistortion tables; submit() runs a step on the next lane's stream, round robin.  While the border
    stages of step t still run (latency-bound, few warps), the streaming scan and the piece filter of step t + 1 have the SMs:
    1.30 ms per 1024-frame detection with two in flight against 1.63 ms one after the other (tools/stage_probe.py).
    A step's results are valid once its lane's stream has reached the end of the step: join(), or lane_stream.synchronize()."""

    IN_FLIGHT_PIPE = {"workers": 4, "chunks": 4}

    def __init__(self, pipe: CapturePipeline, depth: int = 2):
        self.depth = max(1, int(depth))
        self.lanes = [pipe]
        for _ in range(self.depth - 1):
            eng = pipe.eng.clone()                                 # same library, device and calibration tables
            lane = CapturePipeline(eng, pipe.rig, max_blobs=pipe.max_blobs, obj_count=pipe.obj_count, max_groups=pipe.max_groups,
                                   fp64=pipe.fp64, group=pipe.group, lens=pipe.lens, centroids=pipe.centroids)
            lane.pipelined_min_frames = pipe.pipelined_min_frames
            lane.peer_exchange = pipe.peer_exchange
            self.lanes.append(lane)
        if self.depth > 1:
            # with several calls in flight fewer, larger chunks per call do better (tools/stage_probe.py: 4 chunks / 4 worker streams
            # 1.30 ms per call with two calls in flight, 8 / 6 1.36 ms; one call alone: 1.66 against 1.63 ms)
            for lane in self.lanes:
                lane.engine_pipe = dict(self.IN_FLIGHT_PIPE)
        dev = pipe.eng.device
        self.streams = [torch.cuda.Stream(dev) for _ in range(self.depth)] if dev.type == "cuda" and self.depth > 1 else [None] * self.depth
        self.turn = 0
        # scan token: the HBM-bound scans of the lanes run one after the other (each call's scan waits for the scan of the call
        # submitted before it), so that never two rings of TMA boxes sit on an SM.  Two events per lane, used in turn.
        self.scan_token = self.streams[0] is not None
        self._tok = []
        if self.scan_token:
            for _ in range(2 * self.depth):
                e = torch.cuda.Event()
                e.record()                                         # creates the CUDA event behind the object
                self._tok.append(e)

    def next_lane(self):
        """(pipeline, stream) of the next step; the stream is None with depth 1 (the caller's stream)."""
        k = self.turn % self.depth
        if self.scan_token:
            n = len(self._tok)
            prev = self._tok[(self.turn - 1) % n] if self.turn > 0 else None
            self.lanes[k].scan_token = (prev, self._tok[self.turn % n])
        self.turn += 1
        return self.lanes[k], self.streams[k]

    def fork(self):
        """Lane streams start after everything queued on the caller's stream so far (inputs, timing events)."""
        for st in self.streams:
            if st is not None:
                st.wait_stream(torch.cuda.current_stream())

    def join(self):
        """The caller's stream continues after every step submitted so far."""
        for st in self.streams:
            if st is not None:
                torch.cuda.current_stream().wait_stream(st)

    def submit(self, frames: torch.Tensor) -> StepResult:
        lane, st = self.next_lane()
        if st is None:
            return lane.step(frames)
        with torch.cuda.stream(st):
            return lane.step(frames)
