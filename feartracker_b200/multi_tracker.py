"""FEARMultiTracker: many targets tracked in one batched step, the per-track loop state resident on the device.

``FEARTracker`` follows one target at batch 1 and does its crop math and box mapping on the host.  Here the state of
every track (box, context box of the last crop, padding colour: ``FearTrack`` in include/fear_b200.h) lives on the
device, and one step for N tracks is one CUDA graph: batched context crops (``fear_track_crops_u8``) -> network and
decode with one template per track (``fear_track_u8``, Bz = N) -> box update (``fear_track_advance``).  The host only
packs a table of frame pointers and reads back the N boxes.  Every track follows exactly the trajectory
``FEARTracker(gpu_crop=True)`` would give it alone: the device reproduces image_ops' arithmetic to the last bit.

    mt = FEARMultiTracker(net, cuda_id=0, max_tracks=256, **FEAR_XS_TRACKER_KWARGS)
    mt.initialize(frames, rects)              # one frame shared by all rects, or one frame per rect
    out = mt.update(frames, frame_of_track)   # {"bbox": (N, 4) int64, "score": (N,) float32}

``frames`` is one HxWx3 uint8 array (shared by all tracks), a sequence of HxWx3 uint8 arrays / CUDA tensors whose
sizes may differ, or a CUDA uint8 tensor (F, H, W, 3) that is read in place.  ``frame_of_track[n]`` picks the frame of
track n; -1 freezes the track (its box is kept, its score is NaN).
"""
from typing import Any, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib, image_ops
from .tracker import Tracker

_ALIGN = 256  # byte alignment of each frame in the staging pool


class FEARMultiTracker:
    _device = Tracker._device

    def __init__(self, model, cuda_id=0, max_tracks: int = 256, **tracking_config: Any) -> None:
        if tracking_config.get("smooth", False) or tracking_config.get("host_normalize", False):
            raise NotImplementedError("FEARMultiTracker covers the default uint8 RGB tracking path "
                                      "(no smooth / host_normalize)")
        if not 1 <= int(max_tracks) <= 65535:
            raise ValueError(f"max_tracks must be in [1, 65535], got {max_tracks}")
        self.net = model
        self.cuda_id = cuda_id
        self.tracking_config = tracking_config
        self.max_tracks = int(max_tracks)
        self.num_tracks = 0
        self._st: Optional[Dict[str, Any]] = None
        self.net.reserve(self.max_tracks)

    # ------------------------------------------------------------------ public API
    def initialize(self, frames, rects, track_ids: Optional[Sequence[int]] = None) -> None:
        """(Re)initialise tracks.  ``rects`` (K, 4) [x, y, w, h], 0-based.  ``track_ids=None`` replaces every track
        (the tracker then holds K tracks); otherwise K existing track slots are re-initialised and the others keep
        their state.  ``frames`` is one frame shared by all rects or exactly one frame per rect."""
        rects = np.asarray(rects)
        if rects.ndim == 1:
            rects = rects[None]
        if rects.ndim != 2 or rects.shape[1] != 4 or len(rects) == 0:
            raise ValueError(f"rects must be (K, 4) [x, y, w, h], got shape {rects.shape}")
        k = len(rects)
        if track_ids is None:
            if k > self.max_tracks:
                raise ValueError(f"{k} rects exceed max_tracks={self.max_tracks}")
            ids = np.arange(k)
            n = k
        else:
            ids = np.asarray(track_ids).reshape(-1)
            if ids.dtype.kind not in "iu" or len(ids) != k or len(np.unique(ids)) != k:
                raise ValueError(f"track_ids must be {k} distinct integers, one per rect")
            if ids.min() < 0 or ids.max() >= self.num_tracks:
                raise ValueError(f"track_ids must lie in [0, {self.num_tracks})")
            n = self.num_tracks
        items = self._frame_items(frames)
        if len(items) not in (1, k):
            raise ValueError(f"initialize takes one frame shared by all rects or one frame per rect ({k}), "
                             f"got {len(items)}")
        st = self._state()
        entries, keep = self._stage_frames(items)
        rows = np.zeros(k, dtype=_lib.TRACK_DTYPE)
        for i in range(k):
            f = items[0 if len(items) == 1 else i]
            x, y, bw, bh = image_ops.clamp_bbox(rects[i], tuple(f.shape))
            pad = np.clip(np.rint(_mean_colour(f)), 0, 255).astype(np.int32)  # = image_ops.crop_params' colour
            rows[i] = (x, y, bw, bh, 0, 0, 0, 0, pad[0], pad[1], pad[2], 0)
        fot = np.full(n, -1, dtype=np.int32)
        fot[ids] = 0 if len(items) == 1 else np.arange(k)
        self._upload_table(entries, fot)
        ids_dev = torch.from_numpy(ids.astype(np.int64)).to(st["device"])
        st["tracks"][ids_dev] = torch.from_numpy(rows.view(np.int32).reshape(k, 12)).to(st["device"])
        lib, stream = _lib.load(), torch.cuda.current_stream(st["device"]).cuda_stream
        cfg = self.tracking_config
        size = int(cfg["template_size"])
        _lib.check(lib.fear_track_crops_u8(st["table"].data_ptr(), self.max_tracks, st["fot_ptr"],
                                           st["tracks"].data_ptr(), n, size, float(cfg["template_bbox_offset"]),
                                           st["template_crops"].data_ptr(), stream), "fear_track_crops_u8")
        st["zf"][ids_dev] = self.net.get_features(st["template_crops"][ids_dev])
        torch.cuda.current_stream(st["device"]).synchronize()  # the staging buffers are free again
        del keep
        self.num_tracks = n

    def update(self, frames, frame_of_track: Optional[Sequence[int]] = None) -> Dict[str, np.ndarray]:
        """One tracking step for all tracks.  ``frame_of_track`` (N,) defaults to ``arange(N)``, or to all zeros
        when a single frame is given; -1 freezes a track."""
        n = self.num_tracks
        if n == 0:
            raise RuntimeError("FEARMultiTracker.update before initialize")
        items = self._frame_items(frames)
        if frame_of_track is None:
            single = isinstance(frames, (np.ndarray, torch.Tensor)) and frames.ndim == 3
            if not single and len(items) != n:
                raise ValueError(f"{len(items)} frames for {n} tracks: pass frame_of_track")
            fot = np.zeros(n, dtype=np.int32) if single else np.arange(n, dtype=np.int32)
        else:
            fot = self._check_frame_of_track(frame_of_track, n, len(items))
        st = self._state()
        entries, keep = self._stage_frames(items)
        self._upload_table(entries, fot)
        dev = st["device"]
        use_graph = self.tracking_config.get("cuda_graph", True) and st["graph_ok"]
        if st["graph"] is not None and (st["generation"] != self.net.generation() or st["graph_n"] != n):
            # workspace re-allocated, weights re-packed, option changed or track count changed: capture again
            st["graph"], st["calls"] = None, 0
        if use_graph and st["graph"] is None and st["calls"] >= 1:
            try:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    st["boxes"] = self._step(n)
                st["graph"], st["generation"], st["graph_n"] = g, self.net.generation(), n
            except RuntimeError as exc:  # capture failed: stay eager for this tracker, loudly
                import warnings

                warnings.warn(f"FEARMultiTracker: CUDA-graph capture of the step failed ({exc}); using eager launches")
                st["graph_ok"] = False
                torch.cuda.synchronize(dev)
        if use_graph and st["graph"] is not None and st["graph_ok"]:
            st["graph"].replay()
            boxes = st["boxes"]
        else:
            boxes = self._step(n)
        st["calls"] += 1
        st["tracks_pin"][:n].copy_(st["tracks"][:n], non_blocking=True)
        st["boxes_pin"][:n].copy_(boxes, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        del keep
        bbox = st["tracks_pin"].numpy()[:n, :4].astype(np.int64)
        score = st["boxes_pin"].numpy()[:n].view(_lib.BOX_DTYPE)["score"].reshape(-1).copy()
        score[fot < 0] = np.nan
        return dict(bbox=bbox, score=score)

    # ------------------------------------------------------------------ internals
    def _step(self, n: int) -> torch.Tensor:
        """crop -> network + decode -> advance for tracks [0, n), enqueued on the current stream."""
        st, cfg, lib = self._st, self.tracking_config, _lib.load()
        stream = torch.cuda.current_stream(st["device"]).cuda_stream
        size = int(cfg["instance_size"])
        _lib.check(lib.fear_track_crops_u8(st["table"].data_ptr(), self.max_tracks, st["fot_ptr"],
                                           st["tracks"].data_ptr(), n, size, float(cfg["search_context"]),
                                           st["search"].data_ptr(), stream), "fear_track_crops_u8")
        boxes = self.net.track_boxes(st["search"][:n], st["zf"][:n])
        _lib.check(lib.fear_track_advance(boxes.data_ptr(), st["table"].data_ptr(), st["fot_ptr"],
                                          st["tracks"].data_ptr(), n, size, stream), "fear_track_advance")
        return boxes

    def _state(self) -> Dict[str, Any]:
        dev = self._device()
        if self._st is not None and self._st["device"] == dev:
            return self._st
        if self.tracking_config.get("instance_size", 256) != 256:
            raise NotImplementedError("the network takes 256x256 search crops (instance_size=256)")
        m, tsize = self.max_tracks, int(self.tracking_config["template_size"])
        table_bytes = m * _lib.FRAME_DTYPE.itemsize + m * 4
        table = torch.empty(table_bytes, dtype=torch.uint8, device=dev)
        self._st = dict(
            device=dev,
            tracks=torch.zeros((m, 12), dtype=torch.int32, device=dev),
            table_pin=torch.empty(table_bytes, dtype=torch.uint8).pin_memory(), table=table,
            fot_ptr=table.data_ptr() + m * _lib.FRAME_DTYPE.itemsize,
            search=torch.empty((m, 256, 256, 3), dtype=torch.uint8, device=dev),
            template_crops=torch.empty((m, tsize, tsize, 3), dtype=torch.uint8, device=dev),
            zf=torch.zeros((m, 256, tsize // 16, tsize // 16), dtype=torch.float32, device=dev),
            tracks_pin=torch.empty((m, 12), dtype=torch.int32).pin_memory(),
            boxes_pin=torch.empty((m, _lib.BOX_DTYPE.itemsize), dtype=torch.uint8).pin_memory(),
            pool_pin=None, pool=None,
            graph=None, graph_n=None, boxes=None, generation=None, calls=0, graph_ok=True)
        return self._st

    def _frame_items(self, frames) -> list:
        """Validate ``frames`` (no device access) and return them as a list of (H, W, 3) uint8 arrays / tensors."""
        if isinstance(frames, (np.ndarray, torch.Tensor)):
            if frames.ndim == 3:
                items = [frames]
            elif frames.ndim == 4:
                items = [frames[i] for i in range(frames.shape[0])]
            else:
                raise ValueError(f"frames must be (H, W, 3) or (F, H, W, 3), got shape {tuple(frames.shape)}")
        else:
            items = list(frames)
        if not 1 <= len(items) <= self.max_tracks:
            raise ValueError(f"between 1 and max_tracks={self.max_tracks} frames per call, got {len(items)}")
        for f in items:
            if not isinstance(f, (np.ndarray, torch.Tensor)):
                raise TypeError(f"frames must be numpy arrays or CUDA tensors, got {type(f).__name__}")
            u8 = f.dtype == (torch.uint8 if isinstance(f, torch.Tensor) else np.uint8)
            if not u8 or f.ndim != 3 or f.shape[2] != 3 or 0 in f.shape:
                raise ValueError(f"frames must be non-empty (H, W, 3) uint8 RGB, got {f.dtype} {tuple(f.shape)}")
        return items

    def _stage_frames(self, items: list) -> Tuple[List[Tuple[int, int, int]], list]:
        """Frame table entries (device pointer, h, w) and the tensors that must outlive the step.  numpy frames are
        packed into a pinned pool and uploaded in one copy; CUDA tensors are used in place."""
        st = self._st
        for f in items:
            if isinstance(f, torch.Tensor) and f.device != st["device"]:
                raise ValueError(f"CUDA frames must live on {st['device']}, got {f.device}")
        offsets, total = [], 0
        for f in items:
            if isinstance(f, np.ndarray):
                offsets.append(total)
                total += -(-f.nbytes // _ALIGN) * _ALIGN
            else:
                offsets.append(None)
        if total and (st["pool"] is None or st["pool"].numel() < total):
            cap = max(total, 2 * st["pool"].numel() if st["pool"] is not None else 0)
            st["pool_pin"] = torch.empty(cap, dtype=torch.uint8).pin_memory()
            st["pool"] = torch.empty(cap, dtype=torch.uint8, device=st["device"])
        if total:
            pin = st["pool_pin"].numpy()
            for f, off in zip(items, offsets):
                if off is not None:
                    np.copyto(pin[off:off + f.nbytes].reshape(f.shape), f)
            st["pool"][:total].copy_(st["pool_pin"][:total], non_blocking=True)
        entries, keep = [], []
        for f, off in zip(items, offsets):
            if off is not None:
                ptr = st["pool"].data_ptr() + off
            else:
                f = f.detach().contiguous()
                keep.append(f)
                ptr = f.data_ptr()
            entries.append((ptr, int(f.shape[0]), int(f.shape[1])))
        return entries, keep

    def _check_frame_of_track(self, frame_of_track, n: int, nframes: int) -> np.ndarray:
        fot = np.asarray(frame_of_track)
        if fot.shape != (n,) or fot.dtype.kind not in "iu":
            raise ValueError(f"frame_of_track must be ({n},) integers, got {fot.dtype} {fot.shape}")
        if n and (fot.min() < -1 or fot.max() >= nframes):
            raise ValueError(f"frame_of_track values must lie in [-1, {nframes}) (-1 freezes a track)")
        return fot.astype(np.int32)

    def _upload_table(self, entries, fot: np.ndarray) -> None:
        """Frame table + frame_of_track -> one pinned buffer -> one host-to-device copy."""
        st, m = self._st, self.max_tracks
        pin = st["table_pin"].numpy()
        table = pin[:m * _lib.FRAME_DTYPE.itemsize].view(_lib.FRAME_DTYPE)
        for i, (ptr, h, w) in enumerate(entries):
            table[i] = (ptr, h, w)
        pin[m * _lib.FRAME_DTYPE.itemsize:].view(np.int32)[:len(fot)] = fot
        used = m * _lib.FRAME_DTYPE.itemsize + 4 * len(fot)
        st["table"][:used].copy_(st["table_pin"][:used], non_blocking=True)


def _mean_colour(frame) -> np.ndarray:
    """np.mean(frame, axis=(0, 1)), the padding colour FEARTracker.initialize records.  For a CUDA frame the integer
    channel sums are exact and one float64 division per channel rounds exactly like numpy's."""
    if isinstance(frame, np.ndarray):
        return np.mean(frame, axis=(0, 1))
    sums = frame.sum(dim=(0, 1), dtype=torch.int64).cpu().numpy()
    return sums.astype(np.float64) / float(frame.shape[0] * frame.shape[1])
