"""Plug-in boundary known answers produced by running WhisperJAV's own factories and ``VadGroupedFramer`` with the B200 backends
registered (``whisperjav_b200.register()``):

    python tests/golden/make_boundary_kats.py <WhisperJAV checkout>

Recorded: where each factory keeps its registry (module and dict names), the keyword arguments each factory / the framer hands the
B200 class it instantiates, the member names of the WhisperJAV protocols those objects must satisfy, and the framer's frames and
metadata for scripted device probabilities (the device stage is stubbed; no GPU).  ``librosa`` and ``soundfile`` (imported at module
level by the scene backends, absent here) are stood in for by empty modules.  Output: tests/golden/reference_boundary_kats.json,
read by tests/test_boundary.py.
"""
import json
import sys
import types
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parents[1]))
sys.path.insert(0, str(Path(sys.argv[1]).resolve()))
for name in ("librosa", "soundfile"):
    sys.modules.setdefault(name, types.ModuleType(name))

import whisperjav_b200  # noqa: E402
from whisperjav_b200.generator import B200WhisperGenerator  # noqa: E402
from whisperjav_b200.scenes import B200SceneDetector, B200SileroSceneDetector  # noqa: E402
from whisperjav_b200.segmenter import B200SpeechSegmenter  # noqa: E402
from whisperjav_b200.whisperseg import B200WhisperSegSegmenter  # noqa: E402

# the registries register() fills: module -> dict attributes
REGISTRIES = {"whisperjav.modules.speech_segmentation.factory": ["_BACKEND_REGISTRY", "_BACKEND_DEPENDENCIES"],
              "whisperjav.modules.subtitle_pipeline.generators.factory": ["_REGISTRY"],
              "whisperjav.modules.scene_detection_backends.factory": ["_BACKEND_REGISTRY", "_BACKEND_DEPENDENCIES"]}
B200_CLASSES = (B200SceneDetector, B200SileroSceneDetector, B200SpeechSegmenter, B200WhisperSegSegmenter, B200WhisperGenerator)

constructed = []   # (class name, kwargs) of every B200 object the reference code builds
segment_calls = []


def _record_init(cls):
    orig = cls.__init__

    def init(self, *args, **kwargs):
        assert not args, (cls.__name__, args)
        if type(self) is cls:   # a subclass's super().__init__ is not a construction of its own
            constructed.append((cls.__name__, dict(kwargs)))
        orig(self, **kwargs)
    cls.__init__ = init


for c in B200_CLASSES:
    _record_init(c)

done = whisperjav_b200.register()
assert all(done.values()), done

import importlib  # noqa: E402

registries = {}
for mod_name, attrs in REGISTRIES.items():
    mod = importlib.import_module(mod_name)
    registries[mod_name] = {a: {k: v for k, v in getattr(mod, a).items() if k.startswith("b200-")} for a in attrs}

from whisperjav.modules.scene_detection_backends.base import SceneDetector  # noqa: E402
from whisperjav.modules.scene_detection_backends.factory import SceneDetectorFactory  # noqa: E402
from whisperjav.modules.speech_segmentation import SpeechSegmenterFactory  # noqa: E402
from whisperjav.modules.speech_segmentation.base import SpeechSegmenter  # noqa: E402
from whisperjav.modules.subtitle_pipeline.framers.vad_grouped import VadGroupedFramer  # noqa: E402
from whisperjav.modules.subtitle_pipeline.generators.factory import TextGeneratorFactory  # noqa: E402
from whisperjav.modules.subtitle_pipeline.protocols import TextGenerator  # noqa: E402

protocols = {"SceneDetector": SceneDetector, "SpeechSegmenter": SpeechSegmenter, "TextGenerator": TextGenerator}


def creation(proto, make):
    n = len(constructed)
    obj = make()
    assert len(constructed) == n + 1 and isinstance(obj, protocols[proto])
    cls, kw = constructed[-1]
    return {"class": cls, "kwargs": kw, "protocol": proto}


factory_creations = {
    "b200-auditok": creation("SceneDetector", lambda: SceneDetectorFactory.create("b200-auditok", max_duration=20.0, pass2_max_silence_s=0.5)),
    "b200-silero": creation("SceneDetector", lambda: SceneDetectorFactory.create("b200-silero", silero_threshold=0.1)),
    "b200-vad": creation("SpeechSegmenter", lambda: SpeechSegmenterFactory.create("b200-vad", config={"threshold": 0.4, "chunk_threshold_s": 2.5})),
    "b200-whisperseg": creation("SpeechSegmenter", lambda: SpeechSegmenterFactory.create(
        "b200-whisperseg", config={"threshold": 0.35, "max_group_duration_s": 6.0})),
    "b200-whisper": creation("TextGenerator", lambda: TextGeneratorFactory.create(
        "b200-whisper", model_id="tiny", device="cuda", dtype="float16", no_repeat_ngram_size=0, max_new_tokens=444)),
}
backend_available = {k: list(SceneDetectorFactory.is_backend_available(k)) for k in ("b200-auditok", "b200-silero")}


# ---- the framer driving both B200 segmenters on scripted device probabilities
class FakeVad:
    device = "cpu"

    def probs(self, a, ns):
        import torch
        p = torch.zeros(a.shape[0], (a.shape[1] + 511) // 512)
        p[:, 100:200] = 0.9
        p[:, 400:500] = 0.9
        return p


def fake_frame_probs(self, clips):
    p = np.zeros(1500, np.float32)
    p[100:200] = 0.9
    return [p for _ in clips]


B200SpeechSegmenter._ensure_model = lambda self: FakeVad()
B200WhisperSegSegmenter.frame_probs = fake_frame_probs
for c in (B200SpeechSegmenter, B200WhisperSegSegmenter):
    orig_segment = c.segment

    def segment(self, audio, *args, _orig=orig_segment, **kwargs):
        segment_calls.append({"n_samples": len(audio), "args": list(args), "kwargs": dict(kwargs)})
        return _orig(self, audio, *args, **kwargs)
    c.segment = segment

AUDIO_SAMPLES = 480000
framer_cases = []
for backend, framer_kw in (("b200-vad", {"max_group_duration_s": 6.0, "chunk_threshold_s": 2.5}), ("b200-whisperseg", {})):
    n = len(constructed)
    framer = VadGroupedFramer(segmenter_backend=backend, **framer_kw)
    fr = framer.frame(np.zeros(AUDIO_SAMPLES, np.float32), 16000)
    assert len(constructed) == n + 1
    md = fr.metadata
    framer_cases.append({
        "backend": backend, "framer_kwargs": framer_kw, "audio_samples": AUDIO_SAMPLES, "sample_rate": 16000,
        "segmenter": {"class": constructed[-1][0], "kwargs": constructed[-1][1]}, "segment_call": segment_calls[-1],
        "frames": [[f.start, f.end] for f in fr.frames],
        "metadata": {k: md[k] for k in ("segmenter_backend", "frame_count", "total_segments", "total_groups", "groups_skipped",
                                        "speech_regions")}})

out = {"registries": registries, "factory_creations": factory_creations, "backend_available": backend_available,
       "protocol_members": {k: sorted(p.__protocol_attrs__) for k, p in protocols.items()}, "framer": framer_cases}
(HERE / "reference_boundary_kats.json").write_text(json.dumps(out, indent=1, ensure_ascii=False) + "\n")
print(json.dumps(out)[:2000])
