"""``_native.frame_hw``: the one place that knows an NV12 frame's size (host only, no GPU)."""
import numpy as np
import torch

from realtime_video_analytics_32streams_b200 import _native, sinks


def test_frame_hw_of_every_frame_form():
    assert _native.frame_hw(np.zeros((2160, 3840, 3), np.uint8)) == (2160, 3840)
    assert _native.frame_hw(np.zeros((3240, 3840), np.uint8)) == (2160, 3840)            # host NV12 [3H/2, W]
    assert _native.frame_hw(torch.zeros((1080, 1280), dtype=torch.uint8)) == (720, 1280)  # CPU tensor NV12
    wide = torch.zeros((1620, 1952), dtype=torch.uint8)
    assert _native.frame_hw(wide[:, :1920]) == (1080, 1920)                               # pitched view
    assert _native.frame_hw((torch.zeros((720, 1280)), torch.zeros((360, 1280)))) == (720, 1280)  # (y, uv) pair


def test_preview_geometry_reads_the_luma_size():
    # a 1080p NV12 frame is 1620 rows tall; its preview is the frame's own size, a 4K frame's is 1080p
    assert sinks.preview_geometry(*_native.frame_hw(np.zeros((1620, 1920), np.uint8))) == (1.0, 1920, 1080)
    assert sinks.preview_geometry(*_native.frame_hw(np.zeros((3240, 3840), np.uint8))) == (0.5, 1920, 1080)
