"""CPU-only checks: the C-ABI library loads and exports everything include/b200va.h declares, host
geometry matches the oracle, the product never imports the oracle, and the sharding / id-aggregation
logic agrees with one shared reference-style tracker (incl. a world_size-2 gloo run)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import hotpath as O
from realtime_video_analytics_32streams_b200 import _native, sharding

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(REPO, "realtime_video_analytics_32streams_b200")


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(REPO, "include", "b200va.h")).read()
    declared = set(re.findall(r"B200VA_API\s+[\w\s\*]+?\b(b200va_\w+)\s*\(", header))
    assert len(declared) >= 19
    lib = _native.load_library()
    for name in declared:
        assert hasattr(lib, name), name
    assert declared <= set(_native.EXPORTS) | {"b200va_debug_read"}
    assert lib.b200va_version() == 200
    assert lib.b200va_error_string(-3) == b"configured capacity exceeded"


def test_library_is_sm100a_only_and_self_contained():
    out = subprocess.run(["cuobjdump", "-lelf", _native.LIB_PATH], stdout=subprocess.PIPE, text=True).stdout
    archs = set(re.findall(r"sm_\w+", out))
    assert archs == {"sm_100a"}, archs
    ldd = subprocess.run(["ldd", _native.LIB_PATH], stdout=subprocess.PIPE, text=True).stdout
    assert "libtorch" not in ldd and "libcudart" not in ldd  # static cudart, no torch types in the ABI


def test_create_without_gpu_fails_loudly_not_silently():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError):
        _native.Handle(device=0)
    # the raw C entry point reports a CUDA error instead of pretending to work
    lib = _native.load_library()
    cfg = _native.Config(0, 4, 8400, 1024, 256, 4, 256)
    h = ctypes.c_void_p()
    assert lib.b200va_create(ctypes.byref(cfg), ctypes.byref(h)) != 0
    assert not h


@pytest.mark.parametrize("hw,in_hw", [((1080, 1920), (640, 640)), ((2160, 3840), (640, 640)), ((1920, 1080), (640, 640)),
                                      ((1083, 1921), (640, 640)), ((37, 100), (64, 64)), ((600, 800), (320, 416)),
                                      ((720, 1280), (640, 640)), ((33, 77), (96, 64))])
def test_letterbox_meta_matches_oracle(hw, in_hw):
    m = _native.letterbox_meta(hw[0], hw[1], in_hw[0], in_hw[1])
    ref = O.letterbox_meta(hw[0], hw[1], in_hw[0], in_hw[1])
    assert m.as_meta() == {k: ref[k] for k in ("orig_shape", "scale", "pad")}
    assert (m.new_w, m.new_h) == ref["new_wh"]


def test_product_package_never_imports_the_oracle():
    for root, _, files in os.walk(PKG):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(root, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "/root/reference" not in src, f


def test_engine_state_machine_matches_oracle_worker_on_cpu():
    """The adaptive-FPS state of the batched driver is pure host logic: compare with the oracle's."""
    from realtime_video_analytics_32streams_b200.engine import _StreamState
    from realtime_video_analytics_32streams_b200.types import StreamConfig

    rng = np.random.default_rng(3)
    cfg = StreamConfig(name="s", adaptive_fps=True, target_fps=25, min_target_fps=5, idle_frame_tolerance=4)
    st = _StreamState(cfg)
    ow = O.StreamWorker(O.StreamSpec(name="s", adaptive_fps=True, target_fps=25, min_target_fps=5,
                                     idle_frame_tolerance=4), None, O.IouTracker(), 0.3, 0.5)
    assert st.max_process_every == ow.max_process_every == 5
    for _ in range(200):
        nd, nt = (int(rng.integers(0, 3)), int(rng.integers(0, 3))) if rng.random() < 0.2 else (0, 0)
        st.adjust(nd, nt)
        ow._adjust(nd, nt)
        assert (st.process_every, st.idle_frames) == (ow.process_every, ow.idle_frames)


def _simulate(n_streams, ticks, seed):
    rng = np.random.default_rng(seed)
    return [[int(rng.integers(0, 4)) if rng.random() < 0.4 else 0 for _ in range(n_streams)] for _ in range(ticks)]


def test_global_id_map_reproduces_one_shared_counter():
    n = 6
    counts = _simulate(n, 50, 1)
    gm = sharding.GlobalIdMap(n)
    counter = 1
    created = [0] * n
    for tick in counts:
        gm.advance(tick)
        for s, c in enumerate(tick):  # what one shared itertools.count(1) does, streams in order
            for k in range(c):
                assert gm.global_id(s, created[s] + k) == counter
                counter += 1
            created[s] += c
    assert gm.next_id == counter
    assert sharding.streams_of_rank(32, 8, 3) == [12, 13, 14, 15]
    assert sharding.streams_of_rank(5, 2, 1) == [3, 4]
    assert [sharding.rank_of_stream(s, 32, 8) for s in (0, 3, 4, 31)] == [0, 0, 1, 7]


_GLOO_WORKER = r'''
import os, sys, json
sys.path.insert(0, sys.argv[1])
import torch.distributed as dist
from realtime_video_analytics_32streams_b200 import sharding
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo")
import numpy as np
n = 6
rng = np.random.default_rng(1)
counts = [[int(rng.integers(0, 4)) if rng.random() < 0.4 else 0 for _ in range(n)] for _ in range(50)]
mine = sharding.streams_of_rank(n, world, rank)
gm = sharding.GlobalIdMap(n)
ids = []
created = {s: 0 for s in mine}
for tick in counts:
    full = sharding.all_gather_new_counts([tick[s] for s in mine], mine, n)
    assert full == tick
    gm.advance(full)
    for s in mine:
        for k in range(tick[s]):
            ids.append((s, created[s] + k, gm.global_id(s, created[s] + k)))
        created[s] += tick[s]
print("RESULT" + json.dumps({"rank": rank, "ids": ids, "next": gm.next_id}))
dist.destroy_process_group()
'''


def test_sharded_id_aggregation_two_ranks_gloo(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(_GLOO_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29571", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script), REPO], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.PIPE, text=True) for r in range(2)]
    outs = [p.communicate(timeout=180) for p in procs]
    for p, (o, e) in zip(procs, outs):
        assert p.returncode == 0, e[-2000:]
    import json

    res = [json.loads(o.split("RESULT")[1]) for o, _ in outs]
    counts = _simulate(6, 50, 1)
    counter, created, want = 1, [0] * 6, {}
    for tick in counts:
        for s, c in enumerate(tick):
            for k in range(c):
                want[(s, created[s] + k)] = counter
                counter += 1
            created[s] += c
    got = {(s, o): g for r in res for s, o, g in r["ids"]}
    assert got == want
    assert all(r["next"] == counter for r in res)


def _stand_in_reference():
    """The three reference modules the shim patches, reduced to what it touches: the backend whitelist of
    ``DetectorConfig.validate`` (config.py:155-157), ``load_config``, ``create_detector`` (detector.py:54-96) and the names
    ``pipeline.py`` imports or owns (:33, :452, the pipeline and its stream workers)."""
    import dataclasses
    import types

    import yaml

    from realtime_video_analytics_32streams_b200 import types as T

    cfg, det, pipe = (types.ModuleType(f"realtime_analytics.{m}") for m in ("config", "detector", "pipeline"))

    class ConfigError(ValueError):
        pass

    @dataclasses.dataclass
    class DetectorConfig:
        model_path: str = "yolov8n.pt"
        backend: str = "ultralytics"
        model_type: str = "yolov8"
        confidence_threshold: float = 0.5
        iou_threshold: float = 0.45
        input_size: list = None
        half: bool = False

        def validate(self):
            valid_backends = {"ultralytics", "tensorrt", "onnx", "onnxruntime", "openvino", "rknn", "rk3588"}
            if self.backend.lower() not in valid_backends:
                raise ConfigError(f"Unsupported detector backend: {self.backend}")

    @dataclasses.dataclass
    class TrackerConfig:
        type: str = "iou"
        max_age: int = 30
        max_iou_distance: float = 0.7
        min_hits: int = 3

    def load_config(path):
        with open(path) as fh:
            raw = yaml.safe_load(fh)
        full = types.SimpleNamespace(detector=DetectorConfig(**raw["detector"]), tracker=TrackerConfig(**raw["tracker"]),
                                     streams=[T.StreamConfig(**s) for s in raw["streams"]])
        full.detector.validate()
        return full

    cfg.ConfigError, cfg.DetectorConfig, cfg.TrackerConfig, cfg.load_config = ConfigError, DetectorConfig, TrackerConfig, load_config

    def create_detector(config):
        if config.backend.lower() not in ("ultralytics", "tensorrt", "onnx", "onnxruntime", "openvino", "rknn", "rk3588"):
            raise ValueError(f"Unsupported backend: {config.backend}")
        return types.SimpleNamespace(config=config)

    det.create_detector = create_detector

    class IouTracker:
        def __init__(self, config):
            self.config = config

    class AnalyticsPipeline:
        def __init__(self, config):
            self.config = config

        async def wait_closed(self):
            pass

    class StreamWorker:
        def __init__(self, context):
            self.ctx = context

        async def run(self):
            pass

        async def _process_packet(self, packet):
            pass

    def apply_roi(frame, polygons):
        return frame

    def downsample(frame, ratio):
        return frame

    class MotionFilter:
        pass

    for f in (apply_roi, downsample, MotionFilter):
        f.__module__ = "realtime_analytics.filters"
    pipe.create_detector, pipe.IouTracker, pipe.AnalyticsPipeline, pipe.StreamWorker = (create_detector, IouTracker,
                                                                                        AnalyticsPipeline, StreamWorker)
    pipe.apply_roi, pipe.downsample, pipe.MotionFilter = apply_roi, downsample, MotionFilter
    pkg = types.ModuleType("realtime_analytics")
    pkg.config, pkg.detector, pkg.pipeline = cfg, det, pipe
    return {"realtime_analytics": pkg, cfg.__name__: cfg, det.__name__: det, pipe.__name__: pipe}


def test_registration_shim_wires_the_reference_factory(monkeypatch):
    """INTEGRATION.md §3(a): after registration `backend: b200` validates, create_detector dispatches to B200Detector and
    `tracker.type: b200_iou` selects B200IouTracker; unregistering puts back everything it replaced.  Without a GPU
    construction must fail loudly (no silent CPU path).  Runs against the reference itself when B200VA_REFERENCE_SRC
    names its src/ directory, else against a stand-in of the modules the shim patches."""
    ref = os.environ.get("B200VA_REFERENCE_SRC", "")
    if os.path.isdir(ref):
        monkeypatch.syspath_prepend(ref)
    else:
        for name, module in _stand_in_reference().items():
            monkeypatch.setitem(sys.modules, name, module)
    import realtime_analytics.config as rcfg
    import realtime_analytics.detector as rdet
    import realtime_analytics.pipeline as rpipe
    import torch

    from realtime_video_analytics_32streams_b200 import register_with_reference

    with pytest.raises(rcfg.ConfigError):
        rcfg.DetectorConfig(backend="b200").validate()
    from realtime_video_analytics_32streams_b200.integration import unregister_from_reference

    register_with_reference(infer_factory=lambda cfg: (lambda x: x), batched=True)
    try:
        _check_registered_reference(rcfg, rdet, rpipe, torch)
    finally:
        unregister_from_reference()
    # everything is back: the backend id is unknown again, the stock tracker and frame filters are in place
    with pytest.raises(rcfg.ConfigError):
        rcfg.DetectorConfig(backend="b200").validate()
    assert rpipe.IouTracker.__name__ == "IouTracker" and rpipe.apply_roi.__module__.startswith("realtime_analytics")
    assert not rpipe.StreamWorker._b200va_batched


def _check_registered_reference(rcfg, rdet, rpipe, torch):
    assert rpipe.StreamWorker._b200va_batched  # the tick collector is installed (collector.py, tests/test_collector.py)
    cfg = rcfg.DetectorConfig(backend="b200", confidence_threshold=0.35, iou_threshold=0.5)
    cfg.validate()  # whitelisted now
    assert cfg.backend == "b200"
    ucfg = rcfg.DetectorConfig(backend="b200_ultralytics")
    ucfg.validate()  # the Ultralytics-semantics drop-in is whitelisted too
    assert ucfg.backend == "b200_ultralytics"
    with pytest.raises(rcfg.ConfigError):
        rcfg.DetectorConfig(backend="nope").validate()
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            rdet.create_detector(cfg)
        with pytest.raises(RuntimeError):
            rpipe.IouTracker(rcfg.TrackerConfig(type="b200_iou"))
    # other tracker types still get the reference's own class
    assert type(rpipe.IouTracker(rcfg.TrackerConfig())).__name__ == "IouTracker"
    # the YAML authored for config 4 loads with the reference's own loader
    full = rcfg.load_config(os.path.join(REPO, "config", "pipeline-4k-roi.yaml"))
    assert full.detector.backend == "b200" and full.streams[0].motion_filter and len(full.streams[0].roi_polygons) == 2
    # all 32 streams are spelled out, every one with its own hexagon + triangle, the motion gate and adaptive FPS
    from realtime_video_analytics_32streams_b200 import synth

    assert len(full.streams) == 32 and len({s.name for s in full.streams}) == 32
    for i, s in enumerate(full.streams):
        assert s.motion_filter and s.adaptive_fps and s.idle_frame_tolerance == 60 and s.min_target_fps == 5
        assert [[tuple(p) for p in poly] for poly in s.roi_polygons] == synth.synth_polygons(4000 + i, 2160, 3840)
