"""Process-wide plumbing: the default library handle and host<->device staging.

One process drives one GPU (one ``Handle`` per device).  PyTorch supplies device memory, pinned
host memory and the current CUDA stream; nothing here computes.
"""

from __future__ import annotations

import os
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import _native

_handles: Dict[int, "_native.Handle"] = {}


def default_device() -> int:
    import torch

    if "LOCAL_RANK" in os.environ and torch.cuda.device_count() > 1:
        return int(os.environ["LOCAL_RANK"]) % torch.cuda.device_count()
    return torch.cuda.current_device() if torch.cuda.is_available() else 0


def get_handle(device: Optional[int] = None, **overrides) -> "_native.Handle":
    """The shared handle of a device (created on first use).  Capacities come from
    ``B200VA_MAX_*`` environment variables or keyword overrides on the first call."""
    dev = default_device() if device is None else int(device)
    h = _handles.get(dev)
    if h is None:
        cfg = dict(max_batch=int(os.environ.get("B200VA_MAX_BATCH", 64)),
                   max_anchors=int(os.environ.get("B200VA_MAX_ANCHORS", 25200)),
                   max_candidates=int(os.environ.get("B200VA_MAX_CANDIDATES", 4096)),
                   max_dets=int(os.environ.get("B200VA_MAX_DETS", 1024)),
                   max_streams=int(os.environ.get("B200VA_MAX_STREAMS", 64)),
                   max_tracks=int(os.environ.get("B200VA_MAX_TRACKS", 4096)))
        cfg.update(overrides)
        h = _native.Handle(device=dev, **cfg)
        _handles[dev] = h
    return h


def bind_process_to_gpu(device: int) -> Optional[List[int]]:
    """Pin this process to the CPU cores that are local to ``device`` (NVML's affinity mask), so that the pinned
    staging buffers it allocates afterwards are first-touched on the GPU's own NUMA node: with one process per GPU
    and eight GPUs, host -> device copies that cross the socket interconnect are what limits the upload rate.
    Returns the core list, or None when NVML or the affinity call is unavailable (nothing is changed then)."""
    try:
        import pynvml

        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[device]) if vis else device
        handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
        n_cpus = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(handle, (n_cpus + 63) // 64)
        allowed = os.sched_getaffinity(0)
        cores = [64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1]
        cores = [c for c in cores if c in allowed]
        if not cores:
            return None
        os.sched_setaffinity(0, cores)
        return cores
    except Exception:  # pragma: no cover - best effort
        return None


def reset_handles() -> None:
    for h in _handles.values():
        h.close()
    _handles.clear()


class FrameStager:
    """Host -> device staging of decoded frames into persistent per-position device buffers.

    Frame k of a call always lands in the same device tensor (per shape), so pointer-based argument
    batches can be cached by the caller.  Host frames may be numpy arrays (pageable: the driver
    stages them) or CPU torch tensors (pinned: truly asynchronous).  ``sparse_for=(h, w)`` uploads
    only the rows a letterbox to that size reads -- valid when nothing else consumes the frame."""

    def __init__(self, handle: "_native.Handle"):
        self.h = handle
        self._dev: Dict[tuple, object] = {}
        self._ids = set()
        self._keep: List = []
        self.bytes_moved = 0

    def owns(self, tensor) -> bool:
        """True for this stager's persistent device buffers (their addresses never change)."""
        return id(tensor) in self._ids

    def take_sources(self) -> List:
        """Hand the host sources of the last ``upload`` to the caller, who keeps them alive until the copies have
        run (the raw ``cudaMemcpy2DAsync`` calls are invisible to torch's caching host allocator)."""
        keep, self._keep = self._keep, []
        return keep

    def device_buffer(self, k: int, shape):
        t = self.h.torch
        key = (k, tuple(shape))
        buf = self._dev.get(key)
        if buf is None:
            buf = self._dev[key] = t.zeros(tuple(shape), dtype=t.uint8, device=self.h.device)
            self._ids.add(id(buf))
        return buf

    def upload(self, frames: Sequence, sparse_for=None, sparse_ok: Optional[Sequence[bool]] = None,
               geoms: Optional[Sequence] = None) -> List:
        """Return CUDA uint8 [H,W,3] tensors for ``frames``; CUDA tensors pass through untouched.  Host NV12 frames
        (uint8 ``[3H/2, W]`` NumPy arrays or CPU tensors, OpenCV's layout) land in CUDA ``[3H/2, W]`` tensors, half the
        bytes of BGR, sparsely under the same ``sparse_ok`` rule; ``(y, uv)`` pairs of CUDA planes pass through.
        ``geoms`` is the per-frame form of ``sparse_for``: ``geoms[k]`` (a ``Letterbox``, or None for every row) is the
        geometry ``preprocess_geom`` will letterbox frame k with, and only the rows it reads are uploaded."""
        t = self.h.torch
        out: List = [None] * len(frames)
        groups = {False: ([], [], []), True: ([], [], [])}
        nv12 = {False: ([], [], []), True: ([], [], [])}
        keep = []
        for k, f in enumerate(frames):
            if f is None:
                continue
            if (t.is_tensor(f) and f.is_cuda) or isinstance(f, (tuple, list)):
                out[k] = f
                continue
            geom = geoms[k] if geoms is not None else None
            sparse = (geom is not None if geoms is not None else bool(sparse_for)) and (sparse_ok is None or bool(sparse_ok[k]))
            if _native.is_nv12(f):
                a = f if t.is_tensor(f) else np.asarray(f)
                if t.is_tensor(a):
                    if a.dtype != t.uint8 or a.stride(1) != 1:
                        raise ValueError("NV12 frames must be uint8 [3H/2, W] with unit column stride")
                    ptr, pitch = a.data_ptr(), a.stride(0)
                else:
                    if a.dtype != np.uint8:
                        raise ValueError("NV12 frames must be uint8 [3H/2, W]")
                    if a.strides[1] != 1:
                        a = np.ascontiguousarray(a)
                    ptr, pitch = a.ctypes.data, a.strides[0]
                rows, w = int(a.shape[0]), int(a.shape[1])
                if rows % 3 or (rows // 3) % 2 or w % 2:
                    raise ValueError(f"NV12 frames are [3H/2, W] with H and W even, got {(rows, w)}")
                h = rows * 2 // 3
                keep.append(a)
                dev = self.device_buffer(k, (rows, w))
                out[k] = dev
                nv12[sparse][0].append(_native.Nv12Frame(ptr, ptr + h * pitch, pitch, pitch))
                nv12[sparse][1].append(dev)
                nv12[sparse][2].append(geom)
                continue
            if t.is_tensor(f):
                if f.dtype != t.uint8 or f.dim() != 3 or f.shape[2] != 3 or f.stride(2) != 1 or f.stride(1) != 3:
                    raise ValueError("frames must be uint8 [H, W, 3] with packed pixels")
                ptr, pitch, shape = f.data_ptr(), f.stride(0), tuple(f.shape)
            else:
                a = np.asarray(f)
                if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != 3:
                    raise ValueError("frames must be uint8 arrays of shape [H, W, 3]")
                if a.strides[2] != 1 or a.strides[1] != 3:
                    a = np.ascontiguousarray(a)
                ptr, pitch, shape = a.ctypes.data, a.strides[0], a.shape
                f = a
            keep.append(f)
            dev = self.device_buffer(k, shape)
            out[k] = dev
            groups[sparse][0].append((ptr, pitch))
            groups[sparse][1].append(dev)
            groups[sparse][2].append(geom)
        by_geom = geoms is not None
        for sparse, (ptrs, devs, gs) in groups.items():
            if devs:
                self.bytes_moved += self.h.upload_frames(ptrs, devs, sparse_for if sparse and not by_geom else None,
                                                         geoms=gs if sparse and by_geom else None)
        for sparse, (hosts, devs, gs) in nv12.items():
            if devs:
                self.bytes_moved += self.h.upload_frames_nv12(hosts, devs, sparse_for if sparse and not by_geom else None,
                                                              geoms=gs if sparse and by_geom else None)
        self._keep = keep  # sources stay alive until the caller synchronises (end of the tick)
        return out
