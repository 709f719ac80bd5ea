"""Plug-in surface contracts that need no GPU (the reference's own contract tests restated:
tests/test_anime_whisper.py:129-288, tests/test_speech_segmentation.py:170-250)."""
import importlib
import inspect
import json
import sys
import types
from pathlib import Path

import numpy as np
import pytest

import whisperjav_b200
from whisperjav_b200 import hostlogic as H
from whisperjav_b200.asr import B200WhisperASR
from whisperjav_b200.audioio import compose_srt, read_wav_mono, write_wav_pcm16
from whisperjav_b200.generator import B200WhisperGenerator
from whisperjav_b200.segmenter import B200SpeechSegmenter

BOUNDARY = json.loads((Path(__file__).parent / "golden" / "reference_boundary_kats.json").read_text())


def test_generator_protocol_surface():
    g = B200WhisperGenerator(model_id="tiny", device="cuda", dtype="float16", no_repeat_ngram_size=0, max_new_tokens=444)
    for name in ("generate", "generate_batch", "load", "unload", "cleanup"):
        assert callable(getattr(g, name))
    assert g.is_loaded is False
    with pytest.raises(RuntimeError, match="before load"):
        g.generate(Path("x.wav"))
    with pytest.raises(RuntimeError, match="before load"):
        g.generate_batch([Path("x.wav")])
    sig = inspect.signature(g.generate_batch)
    assert list(sig.parameters)[:3] == ["audio_paths", "language", "contexts"]
    g.cleanup()  # unloading an unloaded generator is a no-op
    with pytest.raises(ValueError):
        B200WhisperGenerator(no_repeat_ngram_size=5)


def test_segmenter_surface_and_postprocess():
    s = B200SpeechSegmenter(threshold=0.4, chunk_threshold_s=2.5, max_group_duration_s=6.0, version="x", variant="y")
    assert s.name == "b200-vad" and isinstance(s.display_name, str) and s.get_supported_sample_rates() == [16000]
    probs = np.zeros(938, dtype=np.float32)
    probs[100:200] = 0.9   # 3.2 s .. 6.4 s
    probs[400:500] = 0.9   # 12.8 s .. 16.0 s
    r = s._postprocess(probs, 480000, 30.0, {}, 0.0)
    assert r.method == "b200-vad" and r.num_segments == 2 and r.num_groups == 2
    seg = r.segments[0]
    # padding: start - 11200 samples, end + 20800 samples (silero.py:286-297) on top of the hysteresis regions
    assert (seg.start_sample, seg.end_sample) == (100 * 512 - 11200, 200 * 512 + 20800)
    assert (r.segments[1].start_sample, r.segments[1].end_sample) == (400 * 512 - 11200, 500 * 512 + 20800)
    assert r.segments[1].start_sample >= r.segments[0].end_sample
    assert r.to_legacy_format()[0][0]["start"] == seg.start_sample
    t = B200SpeechSegmenter(threshold=0.5, style="ten", min_silence_duration_ms=100, chunk_threshold_s=1.0)
    rt = t._postprocess(probs, 480000, 30.0, {}, 0.0)
    assert rt.num_segments == 2 and abs(rt.segments[0].start_sec - (100 * 0.032 - 0.05)) < 1e-9
    assert abs(rt.segments[0].end_sec - (200 * 0.032 + 0.15)) < 1e-9 and "raw_start" in rt.segments[0].metadata
    empty = s._postprocess(np.zeros(100, np.float32), 51200, 3.2, {}, 0.0)
    assert empty.segments == [] and empty.groups == []
    s.cleanup()


def test_asr_wrapper_signature_matches_reference():
    params = inspect.signature(B200WhisperASR.__init__).parameters
    assert list(params)[1:] == ["model_config", "params", "task", "tracer"]
    for m in ("transcribe", "transcribe_to_srt", "reset_statistics", "get_filter_statistics", "get_last_vad_segments", "cleanup"):
        assert callable(getattr(B200WhisperASR, m))


def test_wav_and_srt_io(tmp_path):
    a = (0.5 * np.sin(np.arange(16000) * 0.05)).astype(np.float32)
    write_wav_pcm16(tmp_path / "a.wav", a)
    b, sr = read_wav_mono(tmp_path / "a.wav")
    assert sr == 16000 and len(b) == len(a) and np.abs(a - b).max() < 1e-4
    srt_text = compose_srt([{"start": 1.5, "end": 3.25, "text": "こんにちは"}, {"start": 3661.001, "end": 3662.0, "text": "x"}])
    assert "1\n00:00:01,500 --> 00:00:03,250\nこんにちは\n" in srt_text and "01:01:01,001 --> 01:01:02,000" in srt_text
    assert compose_srt([]) == ""


@pytest.fixture()
def reference_registries(monkeypatch):
    """Empty stand-ins for WhisperJAV's factory modules, at the module paths and with the dict names the reference has
    (tests/golden/make_boundary_kats.py), so that ``register()`` runs as inside WhisperJAV without WhisperJAV installed."""
    mods = {}
    for mod_name, attrs in BOUNDARY["registries"].items():
        parts = mod_name.split(".")
        for i in range(1, len(parts) + 1):
            name = ".".join(parts[:i])
            if name not in mods:
                mods[name] = types.ModuleType(name)
                if i > 1:
                    setattr(mods[".".join(parts[: i - 1])], parts[i - 1], mods[name])
        for a in attrs:
            setattr(mods[mod_name], a, {})
    for name, m in mods.items():
        monkeypatch.setitem(sys.modules, name, m)
    return {n: mods[n] for n in BOUNDARY["registries"]}


def test_registration_with_reference_factories(reference_registries):
    """``register()`` fills the registries the reference's factories read, and every B200 class, built from its registered
    dotted path with the keywords the reference's factory handed it, has the members of the protocol that factory promises
    (``runtime_checkable`` protocols: isinstance checks exactly these names)."""
    done = whisperjav_b200.register()
    assert done == {"speech_segmenter": True, "text_generator": True, "scene_detector": True}
    paths = {}
    for mod_name, attrs in BOUNDARY["registries"].items():
        for a, entries in attrs.items():
            assert getattr(reference_registries[mod_name], a) == entries, (mod_name, a)
            if a.endswith("REGISTRY"):
                paths.update(entries)
    objs = {}
    for backend, c in BOUNDARY["factory_creations"].items():
        module_name, class_name = paths[backend].rsplit(".", 1)   # the factories import the module and take the class by name
        cls = getattr(importlib.import_module(module_name), class_name)
        assert cls.__name__ == c["class"]
        objs[backend] = obj = cls(**c["kwargs"])
        assert [m for m in BOUNDARY["protocol_members"][c["protocol"]] if not hasattr(obj, m)] == [], backend
    det = objs["b200-auditok"]
    assert det.name == "b200-auditok"
    assert det._config.max_duration == 20.0 and det._config.pass2_max_duration == 19.0 and det._config.pass2_max_silence == 0.5
    # what the reference's SceneDetectorFactory.is_backend_available said of the dependency entries compared above
    assert BOUNDARY["backend_available"] == {"b200-auditok": [True, ""], "b200-silero": [True, ""]}
    sil = objs["b200-silero"]
    assert sil.name == "b200-silero"
    assert sil._silero_config.max_duration == 420.0 and sil._silero_config.brute_force_chunk_s == 29.0 and sil._silero_config.silero_threshold == 0.1
    assert objs["b200-vad"].chunk_threshold_s == 2.5
    ws = objs["b200-whisperseg"]
    assert ws.name == "b200-whisperseg" and ws.max_speech_duration_s == 6.0


def test_whisperseg_surface_and_postprocess_match_reference_defaults():
    """Constructor keywords / defaults of whisperseg.py:80-141 and the probs -> segments -> groups chain on scripted frame
    probabilities (the state machine itself is pinned by the reference-generated KATs in test_host_kats.py)."""
    from whisperjav_b200.whisperseg import B200WhisperSegSegmenter
    s = B200WhisperSegSegmenter(version="x")
    assert (s.threshold, s.min_speech_duration_ms, s.min_silence_duration_ms, s.speech_pad_ms) == (0.35, 100, 100, 300)
    assert (s.chunk_threshold_s, s.max_group_duration_s, s.max_speech_duration_s) == (1.0, 29.0, 29.0)
    assert s.name == "b200-whisperseg" and s.get_supported_sample_rates() == [16000]
    p = np.zeros(1500, np.float32)
    p[100:200] = 0.9
    p[260:300] = 0.9
    r = s._postprocess(p, 30.0, 0.0)
    # whisperseg.py (SURVEY 8c): p[100:200] = 0.9 -> one segment 1.700-4.300 s (2.0 - 0.3, 4.0 + 0.3); the second region is
    # 1.2 s later, so its padding is clipped half way to the first and they fall into one group (gap < 1.0 s)
    assert abs(r.segments[0].start_sec - 1.7) < 1e-9 and r.num_segments == 2 and r.num_groups == 1
    assert B200WhisperSegSegmenter(chunk_threshold_s=None, chunk_threshold=2.0).chunk_threshold_s == 2.0


def test_reference_vad_grouped_framer_drives_the_b200_segmenters(monkeypatch):
    """The reference's own VadGroupedFramer (subtitle_pipeline/framers/vad_grouped.py:77-164) run with both B200 segmenters
    (tests/golden/make_boundary_kats.py): factory -> segment() -> groups -> TemporalFrames.  The framer builds each segmenter with
    the recorded keywords and calls segment() as recorded; every group becomes one frame, from its first segment's start to its
    last segment's end, with the group's segments as that frame's speech regions.  The device stage is replaced by the scripted
    probabilities of the reference run (no GPU here); the frames must be exactly the ones the reference's framer produced."""
    from whisperjav_b200.whisperseg import B200WhisperSegSegmenter

    class FakeVad:
        device = "cpu"

        def probs(self, a, ns):
            import torch
            p = torch.zeros(a.shape[0], (a.shape[1] + 511) // 512)
            p[:, 100:200] = 0.9
            p[:, 400:500] = 0.9
            return p

    def fake_probs(self, clips):
        p = np.zeros(1500, np.float32)
        p[100:200] = 0.9
        return [p for _ in clips]
    monkeypatch.setattr(B200SpeechSegmenter, "_ensure_model", lambda self: FakeVad())
    monkeypatch.setattr(B200WhisperSegSegmenter, "frame_probs", fake_probs)
    classes = {c.__name__: c for c in (B200SpeechSegmenter, B200WhisperSegSegmenter)}
    assert [c["backend"] for c in BOUNDARY["framer"]] == ["b200-vad", "b200-whisperseg"]
    for case in BOUNDARY["framer"]:
        seg = classes[case["segmenter"]["class"]](**case["segmenter"]["kwargs"])
        call = case["segment_call"]
        r = seg.segment(np.zeros(call["n_samples"], np.float32), *call["args"], **call["kwargs"])
        md = case["metadata"]
        assert (r.method, r.num_segments, r.num_groups) == (md["segmenter_backend"], md["total_segments"], md["total_groups"])
        groups = [g for g in r.groups if g]
        assert md["groups_skipped"] == 0 and md["frame_count"] == len(groups)   # no group below the framer's minimum length
        assert [[g[0].start_sec, g[-1].end_sec] for g in groups] == case["frames"], case["backend"]
        assert [[[x.start_sec, x.end_sec] for x in g] for g in groups] == md["speech_regions"], case["backend"]
