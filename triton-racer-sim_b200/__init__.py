"""B200-native batched observation path for Triton-Racer-Sim (drop-in behind the reference's Component API).

Import as ``triton_racer_sim_b200`` (shim at the repo root).  Public names mirror the reference:
``Component`` (components/component.py), ``ImgPreprocessing`` (components/img_preprocessing.py),
``LocationTracker`` (components/track_data_process.py:68-107) and ``MultiTrackLocationTracker`` / ``MultiTrackImgPreprocessing``
(the same for a batch of cars on several tracks, each track with its own centre line / preprocessing configuration), plus the batched pilot glue
``SpeedControl`` / ``FrameNormalise`` (components/keras_pilot.py:49-50,80-95,142-153; camera.py:36) and the per-car control
post-processing ``ControlMultiplexer`` / ``DriverAssistance`` / ``three_segment_map`` (components/controlmultiplexer.py,
components/driver_assistance.py, utils/mapping.py:9-16), and the pilots themselves: ``KerasPilot`` / ``ModelType``
(components/keras_pilot.py:16-153, utils/types.py) over ``PilotNet``, the networks of components/keras_train.py:127-245 on the
tensor cores.
"""
from .component import Component  # noqa: F401
from .config import default_config  # noqa: F401

__all__ = ["Component", "default_config", "ImgPreprocessing", "MultiTrackImgPreprocessing", "LocationTracker", "MultiTrackLocationTracker", "SpeedControl",
           "FrameNormalise", "ControlMultiplexer", "DriverAssistance", "three_segment_map", "KerasPilot", "PilotNet", "ModelType", "native"]


def __getattr__(name):
    # components import torch and load the CUDA library; keep `import triton_racer_sim_b200.synth` light
    if name in ("ImgPreprocessing", "MultiTrackImgPreprocessing", "LocationTracker", "MultiTrackLocationTracker", "SpeedControl", "FrameNormalise", "ControlMultiplexer", "DriverAssistance",
                "three_segment_map"):
        from . import components
        return getattr(components, name)
    if name in ("KerasPilot", "PilotNet", "ModelType"):
        from . import pilot
        return getattr(pilot, name)
    if name == "native":
        from . import _native
        return _native
    raise AttributeError(name)
