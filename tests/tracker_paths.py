"""Which code path one stream's tracker update takes inside the kernel, predicted from its sizes.

A restatement of the choices in ``tracker_stream`` and ``tracker_stream_impl`` (csrc/tracker_body.cuh), so that the
GPU tests can assert that each case reaches the path it was built for.  Keep the thresholds in step with the kernel:
kDetChunk = 64, kTrkPairs = 2048, kTrkThreadsMin = 256, kTrkSmemRowsMax = 3072, kCand = 6.
"""
from __future__ import annotations

from typing import NamedTuple

DET_CHUNK = 64
TRK_PAIRS = 2048
THREADS_MIN = 256
SMEM_ROWS_MAX = 3072
CAND = 6


class Path(NamedTuple):
    kind: str    # "small-staged", "small" (k_post_track only) or "general"
    table: str   # "shared" or "global" (the stream's scratch)
    phase_a: str  # "few" (pair list) or "units-G8" / "units-G4" / "units-G2" (G = detection groups per 64-row block)
    width: int   # threads the stream's update runs on


def phase_a(nd: int, tc: int, width: int) -> str:
    """Phase A of one chunk of `nd` detections against `tc` tracks (tracker_stream_impl)."""
    pairs = nd * tc + nd * nd
    if pairs <= min(TRK_PAIRS, 8 * width):
        return "few"
    nblk = (tc + 63) // 64 + 1
    return "units-G2" if nblk >= 16 else ("units-G4" if nblk >= 8 else "units-G8")


def predict(t0: int, d: int, smem_tracks: int, threads: int, fused: bool = False, tc: int | None = None,
            nd: int | None = None) -> Path:
    """Path of an update that starts with `t0` live tracks and takes `d` detections.

    `smem_tracks`: rows of the launch's shared-memory table; `threads`: the launch width after B200VA_TRK_THREADS
    (k_tracker 512, or 1024 while the handle is in its dense mode; k_post_track 256; k_dense_resolve_track 1024);
    `fused`: k_post_track (whose small instantiation the other kernels do not have).  `tc` / `nd`: tracks at the start
    of the chunk and its detection count, for a chunk after the first (default: the first chunk)."""
    need = t0 + d
    small = d <= DET_CHUNK and d * (t0 + d) <= 8 * THREADS_MIN
    # k_post_track stages a table of at most 256 rows before its NMS half, behind the NMS layout: that space holds
    # more rows than such a table plus one chunk whatever `smem_tracks` is
    if fused and small and t0 <= THREADS_MIN:
        return Path("small-staged", "shared", "few", THREADS_MIN)
    if fused and small and need <= smem_tracks:
        return Path("small", "shared", "few", THREADS_MIN)
    table = "shared" if need <= smem_tracks else "global"
    width = threads if (t0 > 96 or d > DET_CHUNK) else THREADS_MIN
    tc = t0 if tc is None else tc
    nd = min(DET_CHUNK, d) if nd is None else nd
    return Path("general", table, phase_a(nd, tc, width), width)
