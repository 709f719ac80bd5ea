#!/usr/bin/env python
"""Headline benchmark: audio-seconds/sec (RTFx), whisper-large-v3, 30 s windows at batch 64.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--model large-v3] [--batch 64]
                    [--dump-outputs DIR]

One *step* = one pass of the ASR hot path over one batch of synthetic speech-shaped 30 s windows:
fused log-mel -> Whisper encoder -> cross-K/V projection -> greedy decode with the logit filters
(no-timestamps prefix as on the HF/anime path, until every row hits EOT or sample_len), synthetic seeded weights of the exact
architecture (no checkpoints offline).  ``value`` times the step with the audio already resident in
HBM; ``e2e`` times the public API (``WhisperB200.transcribe_batch``) from pinned host audio to result
dicts on the host.  Under torchrun each rank runs its own batch (weak scaling, windows are independent)
and the packed segment records are all-gathered over NCCL inside the timed region.

``--impl reference`` times the CPU restatement of the reference's openai-whisper path (oracle/, the
reference packages cannot be installed offline) on the host cores, one window per step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "audio-seconds/sec (RTFx) whisper-large-v3 30s@b64"
WINDOW_S = 30.0


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d.get("hbm_gbs", 6650.0), "tflops_burst": d.get("bf16_tflops", 1590.0),
                "tflops_sustained": d.get("bf16_tflops_sustained", 1400.0), "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def enc_gemm_flops(d, B):
    n, T, C = d.n_audio_state, d.n_audio_ctx, d.n_mels
    conv = 2 * (2 * T) * n * 3 * C + 2 * T * n * 3 * n
    per_layer = 2 * T * n * (3 * n) + 2 * T * n * n + 2 * 2 * T * n * 4 * n
    return B * (conv + d.n_audio_layer * per_layer)


def enc_attn_flops(d, B):
    return B * d.n_audio_layer * 4 * d.n_audio_head * d.n_audio_ctx * d.n_audio_ctx * 64


def decode_bytes(d, steps_run, active_steps_total, B):
    """Algorithmic HBM bytes of a decode run (SURVEY.md 8d): per step the decoder weights once, plus per
    active row the cross-K/V of every layer; self-KV and logits are second order but counted."""
    t = d.n_text_state
    w_layer = (3 * t * t + t * t + t * t + t * t + 8 * t * t) * 2  # qkv, out, cq, cout, fc1+fc2 (cross k/v proj is per window)
    weights = d.n_text_layer * w_layer + d.n_vocab * t * 2
    cross = d.n_text_layer * 2 * d.n_audio_ctx * t * 2
    logits = d.n_vocab * 2
    return steps_run * weights + active_steps_total * (cross + logits)



def time_cross_attention(dims, B, reps=3):
    """The decode step's dominant kernel (attn_dec_cross_bulk_kernel) timed alone with CUDA events on the launching stream:
    one launch per layer-sized K/V buffer, 6 distinct buffers (> L2) cycled, every row alive.  Returns (us per launch, bytes)."""
    from whisperjav_b200 import _lib
    lib = _lib.load()
    H, T, n = dims.n_text_head, dims.n_audio_ctx, dims.n_text_state
    kvs = [torch.randn(B, 2 * H, T, 64, device="cuda", dtype=torch.float16) for _ in range(6)]
    q = torch.randn(B, n, device="cuda", dtype=torch.float16)
    out = torch.empty(B, n, device="cuda", dtype=torch.float16)
    for kv in kvs:
        _lib.check(lib.wjb_attention_cross_f16(_lib.ptr(q), _lib.ptr(kv), _lib.ptr(out), B, H, T, _lib.stream_ptr()), "cross")
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        for kv in kvs:
            _lib.check(lib.wjb_attention_cross_f16(_lib.ptr(q), _lib.ptr(kv), _lib.ptr(out), B, H, T, _lib.stream_ptr()), "cross")
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / (reps * len(kvs))
    nbytes = B * 2 * T * n * 2 + 2 * B * n * 2  # K and V of every row once, q in, out back
    del kvs
    return us, nbytes


def run_ours(args):
    import torch.distributed as dist
    from whisperjav_b200 import _lib, model as M
    from whisperjav_b200.distributed import gather_segment_records, pack_records
    from whisperjav_b200.synth import DIMS, speech_shaped_audio

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL prints its version banner on stdout at init; the contract is ONE JSON line on stdout
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    dims = DIMS[args.model]
    B = args.batch
    m = M.load_model(args.model, device=f"cuda:{local}", max_batch=B)
    lib = _lib.load()
    # synthetic speech-shaped windows, all distinct (seed 1000 * config + rank * 64 + row, SURVEY.md 8d)
    clips = [speech_shaped_audio(WINDOW_S, 1000 * 2 + rank * 64 + i) for i in range(B)]
    host_audio = torch.stack([torch.from_numpy(c) for c in clips]).pin_memory()
    dev_audio = host_audio.cuda()
    ns = torch.full((B,), host_audio.shape[1], dtype=torch.int32, device="cuda")
    # HF / anime-path decode mode (forced <sot><ja><transcribe><notimestamps>): every 30 s clip is exactly one window in
    # both the resident and the end-to-end arm (in timestamp mode the seek loop re-decodes clip tails at data-dependent
    # offsets, which would make the two arms do different amounts of work); timestamp rules are covered by the parity tests
    # timestamp ids are added to the suppress list: upstream leaves them sampleable even with <|notimestamps|> (real
    # checkpoints never emit them there, random-init weights do, and transcribe() would then re-decode clip tails)
    ts0 = dims.n_vocab - 1501
    dec_kw = dict(language="ja", task="transcribe", without_timestamps=True, suppress_tokens=[-1] + list(range(ts0, dims.n_vocab)))
    preset = (args.decode or "greedy") == "preset"
    if preset:
        # the reference's shipped decode preset (balanced / fidelity, config/components/asr/openai_whisper.py:225-247): beam 2,
        # patience 1.2, timestamps on; the e2e arm adds the thresholds and, with --word-timestamps, the alignment pass
        dec_kw = dict(language="ja", task="transcribe", beam_size=2, patience=1.2, without_timestamps=False, max_initial_timestamp=0.0)
    l2_flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    def step_resident():
        mel = m.log_mel(dev_audio, ns, n_frames=3000, layout="time")
        xa = m.encode(mel)
        res = m.decode_features(xa, **dec_kw)
        if world > 1:
            rec = pack_records([(rank * B + i, 0.0, WINDOW_S, r.avg_logprob, r.no_speech_prob, r.tokens) for i, r in enumerate(res)])
            gather_segment_records(rec, device=f"cuda:{local}")
        return res

    def step_e2e():
        out = m.transcribe_batch(clips, temperature=0.0, condition_on_previous_text=False, no_speech_threshold=0.6,
                                 logprob_threshold=-1.0, compression_ratio_threshold=2.4, pinned_audio=host_audio,
                                 word_timestamps=bool(args.word_timestamps), **dec_kw)
        if world > 1:
            rec = pack_records([(rank * B + i, 0.0, WINDOW_S, s["avg_logprob"], s["no_speech_prob"], s["tokens"])
                                for i, o in enumerate(out) for s in o["segments"][:1]])
            gather_segment_records(rec, device=f"cuda:{local}")
        return out

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, profile=False):
        times, extra, res = [], [], None
        for _ in range(steps):
            l2_flush.fill_(1)  # flush L2 between timed iterations (inputs are also larger than L2)
            barrier()
            if profile:
                lib.wjb_profile_enable(1)
            s0 = dict(m.stats)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            res = fn()
            e1.record()
            barrier()
            times.append(e0.elapsed_time(e1))
            if profile:
                import ctypes as C
                ms = (C.c_float * 3)()
                cnt = (C.c_int * 3)()
                lib.wjb_profile_read(ms, cnt, 3)
                lib.wjb_profile_enable(0)
                extra.append({"ms": list(ms), "launches": list(cnt), "steps_run": m.stats["decode_steps"] - s0["decode_steps"], "res": res})
        return times, extra, res

    for _ in range(args.warmup):
        step_resident()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # stage timing (events between stages) is taken on the same timed steps
    stage = {"mel": [], "encoder": [], "decode": []}

    def step_resident_staged():
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        mel = m.log_mel(dev_audio, ns, n_frames=3000, layout="time")
        ev[1].record()
        xa = m.encode(mel)
        ev[2].record()
        res = m.decode_features(xa, **dec_kw)
        ev[3].record()
        if world > 1:
            rec = pack_records([(rank * B + i, 0.0, WINDOW_S, r.avg_logprob, r.no_speech_prob, r.tokens) for i, r in enumerate(res)])
            gather_segment_records(rec, device=f"cuda:{local}")
        torch.cuda.synchronize()
        stage["mel"].append(ev[0].elapsed_time(ev[1]))
        stage["encoder"].append(ev[1].elapsed_time(ev[2]))
        stage["decode"].append(ev[2].elapsed_time(ev[3]))
        return res

    times, extra, last_res = timed(step_resident_staged, args.steps, profile=True)
    for _ in range(min(args.warmup, 1)):
        step_e2e()
    e2e_times, _, last_e2e = timed(step_e2e, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(Path(args.dump_outputs), last_res, last_e2e)

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    total_ms = max_over_ranks(sum(times))
    e2e_ms = max_over_ranks(sum(e2e_times))
    audio_s = world * B * WINDOW_S * args.steps
    value = audio_s / (total_ms / 1e3)
    e2e_value = audio_s / (e2e_ms / 1e3)

    # ---- rooflines (rank 0's own step numbers) ------------------------------------------------
    peaks = _peaks()
    gemm_ms = np.mean([x["ms"][0] for x in extra])
    attn_ms = np.mean([x["ms"][1] for x in extra])
    gemm_launches = int(np.mean([x["launches"][0] for x in extra]))
    attn_launches = int(np.mean([x["launches"][1] for x in extra]))
    ln_launches = int(np.mean([x["launches"][2] for x in extra]))
    gemm_tf = enc_gemm_flops(dims, B) / (gemm_ms / 1e3) / 1e12
    attn_tf = enc_attn_flops(dims, B) / (attn_ms / 1e3) / 1e12
    steps_run = float(np.mean([x["steps_run"] for x in extra]))
    n_initial = 4
    active = float(np.mean([sum(min(len(r.tokens) + 1 + (n_initial - 1), x["steps_run"]) for r in x["res"]) for x in extra]))
    dec_ms = float(np.mean(stage["decode"]))
    dec_gbs = decode_bytes(dims, steps_run, active, B) / (dec_ms / 1e3) / 1e9
    mel_gbs = B * 2.688e6 / (np.mean(stage["mel"]) / 1e3) / 1e9
    shares = {"encoder_gemm": gemm_ms, "encoder_attention": attn_ms, "decode": dec_ms, "mel": float(np.mean(stage["mel"]))}
    dominant = max(shares, key=shares.get)
    rl_all = {
        "encoder_gemm": {"kernel": "gemm_tc_kernel (tcgen05)", "bound": "tensor", "achieved": gemm_tf, "peak": peaks["tflops_sustained"] / 1.0,
                         "unit": "TFLOP/s", "frac": gemm_tf / peaks["tflops_sustained"], "traffic": None, "ms_per_step": gemm_ms,
                         "launches_per_step": gemm_launches},
        "encoder_attention": {"kernel": "attn_encoder_kernel (tcgen05)", "bound": "tensor", "achieved": attn_tf, "peak": peaks["tflops_sustained"],
                              "unit": "TFLOP/s", "frac": attn_tf / peaks["tflops_sustained"], "traffic": None, "ms_per_step": attn_ms,
                              "launches_per_step": attn_launches},
        "decode": {"kernel": "decode step graph (attn_dec_cross_kernel dominant)", "bound": "hbm", "achieved": dec_gbs, "peak": peaks["hbm_gbs"],
                   "unit": "GB/s", "frac": dec_gbs / peaks["hbm_gbs"], "traffic": None, "ms_per_step": dec_ms, "decoder_steps": steps_run},
        "mel": {"kernel": "logmel_kernel", "bound": "hbm", "achieved": mel_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": mel_gbs / peaks["hbm_gbs"], "traffic": None, "ms_per_step": shares["mel"]},
    }
    if dominant == "decode":
        # the step graph is led by one kernel: the cross-attention read of every live row's encoder K/V.  Time that kernel alone,
        # live, and report it as the dominant-kernel roofline; the whole-graph figure stays in roofline_all["decode"].
        cross_us, cross_bytes = time_cross_attention(dims, B)
        cross_gbs = cross_bytes / (cross_us * 1e-6) / 1e9
        rl_all["decode_cross_attention"] = {
            "kernel": "attn_dec_cross_bulk_kernel", "bound": "hbm", "achieved": cross_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": cross_gbs / peaks["hbm_gbs"], "traffic": 495.3e6, "traffic_source": "profiles/r2_prof_decode.json (dram read 491.72 MB + write 3.1-4.0 MB per launch, ncu --set full)",
            "algorithmic_bytes_per_launch": cross_bytes, "us_per_launch": cross_us, "launches_per_decoder_step": dims.n_text_layer,
            "share_of_decode_step": cross_us * 1e-3 * dims.n_text_layer * (active / max(B * steps_run, 1.0)) / (dec_ms / max(steps_run, 1.0)),
            "note": "timed alone with every row alive; inside the step rows that reached EOT are skipped (share scaled by the live-row fraction)"}
        roofline = dict(rl_all["decode_cross_attention"])
    else:
        roofline = dict(rl_all[dominant])
    roofline["peak_source"] = peaks["source"] + (", sustained figure (kernel timed inside a long step)" if roofline["bound"] == "tensor" else "")
    tokens_out = int(np.mean([sum(len(r.tokens) for r in x["res"]) for x in extra]))
    n_layers_launch = dims.n_text_layer * 11 + 5  # per layer: 3 LN, 6 GEMM, self-, cross-attention; + embed, ln, logits, sample, advance
    gpu_launches = int(3 + gemm_launches + attn_launches + ln_launches + dims.n_text_layer + steps_run * n_layers_launch)

    out = None
    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic (seeded speech-shaped 16 kHz audio; seeded random-init weights of the exact architecture)",
            "config": {"workload": f"whisper-{args.model} full hot path: log-mel + encoder + cross-KV + greedy decode (no-timestamps prefix, logit filters on, to EOT/sample_len), "
                                   f"batch {B} x 30 s windows per GPU", "global_batch": world * B, "parallelism": f"dp{world} (windows sharded, weights replicated)",
                       "l2": "L2 flushed (256 MiB write) between timed iterations; activations/weights also exceed L2",
                       "decode_tokens_per_step": tokens_out, "decoder_steps": steps_run},
            "e2e": {"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": int(B * host_audio.shape[1] * 4),
                    "d2h_bytes_per_step": int(B * (3 + 224 + 1 + 3) * 4), "ms_per_step": e2e_ms / args.steps,
                    "api": "WhisperB200.transcribe_batch(host fp32 clips) -> result dicts"},
            "gpu_launches": gpu_launches,
            "clocks": clocks,
            "roofline": roofline, "roofline_all": rl_all,
            "stages_ms": {k: float(np.mean(v)) for k, v in stage.items()},
            "encoder_tensor_util_pct_of_measured_peak": 100.0 * (enc_gemm_flops(dims, B) + enc_attn_flops(dims, B)) / ((gemm_ms + attn_ms) / 1e3) / 1e12 / peaks["tflops_sustained"],
        }
        if preset:
            out["metric"] = METRIC + " [reference decode preset: beam 2, patience 1.2, timestamps on]"
            out["config"]["workload"] = out["config"]["workload"].replace("greedy decode (no-timestamps prefix, logit filters on, to EOT/sample_len)",
                                                                          "beam search (beam 2, patience 1.2, timestamp rules on, to EOT/sample_len)")
            out["config"]["e2e_word_timestamps"] = bool(args.word_timestamps)
        if not args.no_parity_check and not preset:
            out["parity_check"] = parity_check(m, args.model, clips[:2], dec_kw)
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(args.model)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _padded(seqs) -> np.ndarray:
    """Ragged token lists -> [n, longest] float64, -1 past each list's end (token ids are exact in float64)."""
    a = np.full((len(seqs), max((len(s) for s in seqs), default=0)), -1.0)
    for i, s in enumerate(seqs):
        a[i, : len(s)] = s
    return a


def dump_outputs(out_dir: Path, res, e2e) -> None:
    """Write what the last timed step of each arm returned to its caller as ``<name>.npy`` (float64): the resident arm's
    per-window decode results and the e2e arm's segments, one row per segment in clip order.  Audio and weights are seeded
    and the decode is deterministic, so two builds run with the same arguments can be compared file by file."""
    segs = [(i, s) for i, o in enumerate(e2e) for s in o["segments"]]
    words = [(k, w) for k, (_, s) in enumerate(segs) for w in s.get("words", [])]
    arrays = {
        "resident_tokens": _padded([r.tokens for r in res]),
        "resident_avg_logprob": np.array([r.avg_logprob for r in res]),
        "resident_sum_logprob": np.array([r.sum_logprob for r in res]),
        "resident_no_speech_prob": np.array([r.no_speech_prob for r in res]),
        "e2e_segment_clip": np.array([i for i, _ in segs], dtype=np.float64),
        "e2e_tokens": _padded([s["tokens"] for _, s in segs]),
    }
    for key in ("seek", "start", "end", "avg_logprob", "no_speech_prob", "compression_ratio", "temperature"):
        arrays["e2e_segment_" + key] = np.array([s[key] for _, s in segs], dtype=np.float64)
    if words:  # --word-timestamps: [segment row, start, end, probability] per word
        arrays["e2e_words"] = np.array([[k, w["start"], w["end"], w["probability"]] for k, w in words], dtype=np.float64)
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", a)


def parity_check(m, model_name, clips, dec_kw, sample_len=40):
    """Outside the timed region, rank 0: rows 0-1 of the benchmarked batch (same clips, same weights, same decode options)
    against the CPU oracle -- mel, encoder hidden states, then every decode step's logits and token (oracle/parity.py)."""
    from oracle import parity as P
    from oracle import whisper_oracle as wo
    from whisperjav_b200.synth import DIMS, synth_preset, synth_weights
    t0 = time.time()
    dims = DIMS[model_name]
    w = synth_weights(dims, **synth_preset(model_name))
    pw = wo.prepare_weights(w, True)
    mel = P.gpu_mel(m, clips)
    mel_err = float((mel[:, 1:-1].permute(0, 2, 1).float().cpu() - P.oracle_mel_windows(clips, dims)).abs().max())
    enc, xa = P.encoder_parity(m, w, dims, mel, prepared=pw)
    rep = P.decode_parity(m, w, dims, xa, prepared=pw, sample_len=sample_len, tie_quanta=8.0, logit_quanta=40.0, logit_rms_quanta=8.0, logprob_tol_per_step=0.06, **dec_kw)
    ok = bool(rep["ok"] and enc["ok"] and mel_err <= 1e-3)
    return {"ok": ok, "windows": rep["windows"], "steps_checked": rep["steps_checked"], "identical_windows": rep["identical_windows"],
            "tie_breaks": rep["tie_breaks"], "dlogit_quanta_max": rep["dlogit_quanta_max"], "tolerances": rep["tolerances"],
            "encoder_rel_fro": enc["rel_fro"], "mel_max_abs": mel_err, "failures": rep["failures"][:4],
            "tokens_head": [t[:16] for t in rep["tokens"]], "seconds": round(time.time() - t0, 1),
            "what": f"rows 0-1 of the timed batch vs oracle/ (CPU restatement): mel <= 1e-3, encoder <= 1e-2 rel, {sample_len}-token greedy "
                    "decode: per-step logits and ids on the device's own prefix"}


CPU_DECODE_CAP = 64  # decoder tokens per window in every CPU-baseline sample (both the cpu_baseline block and --impl reference)


def _cpu_window(model_name, sample_len, pw=None, dims=None, seed_audio=2000):
    from oracle import whisper_oracle as wo
    from whisperjav_b200.synth import speech_shaped_audio
    a = speech_shaped_audio(WINDOW_S, seed_audio)
    with wo.accumulation(torch.float32):  # the reference's arithmetic: fp32 sums (the oracle's exact float64 sums are for checking)
        t0 = time.time()
        mel = wo.pad_or_trim(wo.log_mel_spectrogram(a, dims.n_mels, padding=wo.N_SAMPLES)[:, : len(a) // 160], wo.N_FRAMES)
        xa = wo.encoder_forward(pw, dims, mel[None], True)
        t1 = time.time()
        res = wo.decode(pw, dims, None, wo.DecodingOptions(language="ja", without_timestamps=True, sample_len=sample_len,
                                                              suppress_tokens=[-1] + list(range(dims.n_vocab - 1501, dims.n_vocab))), True, audio_features=xa)
        t2 = time.time()
    return t1 - t0, t2 - t1, len(res[0].tokens)


def effective_cores() -> int:
    """Cores this process may actually use: min(cpu_count, affinity mask, cgroup cpu.max quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, n)


_CALIB = None


def pick_threads() -> int:
    """Thread count for the CPU baseline: the fastest of a few candidates on a short mix shaped like the path itself -- one
    encoder-sized GEMM (1500 x 1280 x 5120) and a run of decoder-sized GEMVs (1 x 1280 x 5120) -- because shared hosts
    oversubscribe badly at ``os.cpu_count()`` and a square-GEMM calibration picks differently from run to run."""
    global _CALIB
    cores = effective_cores()
    cands = sorted({c for c in (cores, cores // 2, 64, 32, 16) if 1 <= c <= cores})
    a = torch.randn(1500, 1280)
    w = torch.randn(5120, 1280)
    v = torch.randn(1, 1280)
    table = {}
    for c in cands:
        torch.set_num_threads(c)
        (a @ w.t(), v @ w.t())
        t0 = time.time()
        for _ in range(2):
            a @ w.t()
        t1 = time.time()
        for _ in range(200):
            v @ w.t()
        t2 = time.time()
        # one window is ~74 such GEMMs per encoder layer-equivalent and ~192 such GEMVs per token x CPU_DECODE_CAP tokens
        table[c] = {"gemm_ms": (t1 - t0) / 2 * 1e3, "gemv_us": (t2 - t1) / 200 * 1e6}
    best = min(cands, key=lambda c: table[c]["gemm_ms"] * 100 + table[c]["gemv_us"] * 1e-3 * 192 * CPU_DECODE_CAP / 4)
    _CALIB = {"candidates": table, "picked": best}
    torch.set_num_threads(best)
    return best


_THREADS = None


def _cpu_setup(model_name):
    global _THREADS
    from oracle import whisper_oracle as wo
    from whisperjav_b200.synth import DIMS, synth_preset, synth_weights
    _THREADS = pick_threads()
    dims = DIMS[model_name]
    pw = wo.prepare_weights(synth_weights(dims, **synth_preset(model_name)), True)
    return dims, pw


def cpu_baseline(model_name):
    """The oracle (CPU restatement of the reference's openai-whisper path) timed on the host cores on a bounded sample: one
    30 s window (the GPU arm's rank-0 clip 0), greedy decode capped at CPU_DECODE_CAP tokens."""
    dims, pw = _cpu_setup(model_name)
    enc_s, dec_s, ntok = _cpu_window(model_name, CPU_DECODE_CAP, pw, dims, seed_audio=2000)
    wall = enc_s + dec_s
    return {"value": WINDOW_S / wall, "unit": "audio-s/s", "cores": _THREADS, "host_cpu_count": os.cpu_count(), "kind": "port",
            "thread_calibration": _CALIB,
            "sample": f"1 window of 30 s (clip seed 2000 = row 0 of the GPU batch), whisper-{model_name}: mel+encoder {enc_s:.1f} s, greedy decode "
                      f"capped at {CPU_DECODE_CAP} tokens ({ntok} produced, {dec_s:.1f} s); batch 1 per call as the reference runs it; torch CPU fp32 "
                      "with fp16 rounding points",
            "note": "restated CPU path of openai-whisper @ c0d2f62 on synthetic weights (reference packages not installable offline); baseline only"}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    dims, pw = _cpu_setup(args.model)
    cap = CPU_DECODE_CAP
    for i in range(min(args.warmup, 1)):  # one untimed window warms the allocator / thread pool; more would only burn minutes
        _cpu_window(args.model, 8, pw, dims, 2000 + i)
    t0 = time.time()
    toks = 0
    for i in range(args.steps):
        _, _, n = _cpu_window(args.model, cap, pw, dims, 2000 + i)  # clip seeds = rows 0.. of the GPU arm's rank-0 batch
        toks += n
    wall = time.time() - t0
    value = args.steps * WINDOW_S / wall
    cb = {"value": value, "unit": "audio-s/s", "cores": _THREADS, "host_cpu_count": os.cpu_count(), "kind": "port", "thread_calibration": _CALIB,
          "sample": f"{args.steps} steps x 1 window of 30 s (batch 1 per call, as the reference does; clip seeds 2000.. = rows 0.. of the GPU "
                    f"arm's batch), greedy decode capped at {cap} tokens per window ({toks} produced)"}
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "audio-s/s", "n_gpus": int(os.environ.get("WORLD_SIZE", 1)),
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 (fp16 rounding points)", "data": "synthetic (same generators and seeds as the GPU arm)",
        "config": {"workload": f"whisper-{args.model} full hot path on host cores, 1 window per step", "note":
                   "oracle port of openai-whisper @ c0d2f62; the reference's own packages cannot be installed offline"},
        "cpu_baseline": cb, "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def run_stream(args):
    """BASELINE configs 3 / 4: long streams through the whole path the north star names -- VAD gate -> groups -> log-mel ->
    encoder -> decode -> segments -> SRT text -- timed end to end from host audio (whisperjav_b200/stream.py).  ``--workload
    stream``: one stream, balanced preset grouping (config 3).  ``--workload streams8``: eight streams, TEN-style grouping and the
    greedy no-timestamps decode of the anime path, units dealt over the ranks by speech seconds (config 4, strong scaling)."""
    import torch.distributed as dist
    from whisperjav_b200 import model as M, stream as S
    from whisperjav_b200.audioio import compose_srt
    from whisperjav_b200.distributed import gather_segment_records, pack_records
    from whisperjav_b200.segmenter import B200SpeechSegmenter
    from whisperjav_b200.scenes import B200SceneDetector
    from whisperjav_b200.synth import film_audio

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    anime = args.workload == "streams8"
    n_streams = 8 if anime else 1
    seconds = args.stream_minutes * 60.0
    m = M.load_model(args.model, device=f"cuda:{local}", max_batch=args.batch)
    seg = B200SpeechSegmenter(device=f"cuda:{local}", **(S.ANIME_VAD if anime else S.BALANCED_VAD))
    decode = dict(S.ANIME_DECODE if anime else S.BALANCED_DECODE)
    if args.decode == "greedy":
        for k in ("beam_size", "patience", "best_of"):
            decode.pop(k, None)
    if args.word_timestamps:
        decode["word_timestamps"] = True
    streams = [film_audio(seconds, (4000 if anime else 3000) + k) for k in range(n_streams)]
    scene_det = B200SceneDetector(device=f"cuda:{local}")   # reference defaults: 29 s scenes, 32 / 38 dB gates, 1.8 / 0.94 s silences
    sync = torch.cuda.synchronize

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run(strs):
        if world > 1:
            r = S.transcribe_streams_distributed(m, seg, strs, decode=decode, sync=sync, device=f"cuda:{local}", scene_detector=scene_det)
            rec = pack_records([(s_["stream"] * 10_000_000 + int(s_["start"] * 100), s_["start"], s_["end"], s_["avg_logprob"], s_["no_speech_prob"],
                                 s_["tokens"]) for s_ in r.segments])
            allr = gather_segment_records(rec, device=f"cuda:{local}")
            srt = compose_srt([{"start": x["start"], "end": x["end"], "text": M.detokenize([t for t in x["tokens"] if t < 50257])} for x in allr]) if rank == 0 else ""
        else:
            r = S.transcribe_streams(m, seg, strs, decode=decode, sync=sync, scene_detector=scene_det)
            srt = compose_srt(r.segments)
        return r, srt

    run([s_[: 16000 * 240] for s_ in streams])   # warm-up: 4 min of every stream (graph capture, allocator, VAD weights)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    p0 = dict(m.stats)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    r, srt = run(streams)
    e1.record()
    barrier()
    wall = time.perf_counter() - t0
    dev_ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([dev_ms, r.stages_s["vad"] * 1e3, r.stages_s["transcribe"] * 1e3, wall * 1e3, r.stages_s["scenes"] * 1e3], dtype=torch.float64,
                     device="cuda")
    tmax, tsum = t.clone(), t.clone()
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
    audio_s = n_streams * seconds
    if rank == 0:
        total_ms = float(tmax[0])
        print(json.dumps({
            "metric": f"audio-seconds/sec (RTFx) {'anime-shaped: TEN-style VAD + greedy decode, 8 streams' if anime else 'balanced-shaped: VAD + mel + large-v3 transcribe, 1 stream'}",
            "value": audio_s / (total_ms / 1e3), "unit": "audio-s/s", "n_gpus": world, "steps": 1, "warmup": 1, "ms_per_step": total_ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16",
            "data": "synthetic (film-shaped 16 kHz streams: chapters of seeded speech-shaped clips, room-tone gaps, in-chapter pauses; seeded random-init weights)",
            "config": {"workload": f"BASELINE config {'4' if anime else '3'}: {n_streams} x {args.stream_minutes} min stream(s) -> b200-auditok scenes (<= 29 s) -> b200-vad -> groups "
                                   f"({'chunk 0.5 s / max 5 s' if anime else 'balanced preset: chunk 2.5 s / max 6 s'}) -> transcribe_batch (batch {args.batch}, decode {args.decode or "preset"}"
                                   f"{'' if anime else ', timestamps on, thresholds on'}) -> segments -> SRT text; host audio in, host text out",
                       "decode": {k: v for k, v in decode.items()}, "parallelism": f"units dealt over {world} rank(s) by speech seconds"},
            "e2e": {"value": audio_s / (total_ms / 1e3), "unit": "audio-s/s", "h2d_bytes_per_step": int(audio_s * 16000 * 4 + r.stats["unit_audio_s"] * world * 16000 * 4),
                    "d2h_bytes_per_step": int(r.stats["units"] * world * 240 * 4), "api": "stream.transcribe_streams(host fp32 streams) -> segments -> SRT"},
            "stages_ms_max_over_ranks": {"scenes": float(tmax[4]), "vad": float(tmax[1]), "transcribe": float(tmax[2]), "wall": float(tmax[3])},
            "scenes_rank0": r.stats["scenes"],
            "straggler_ratio": float(tmax[0] / (tsum[0] / world)),
            "units_total": r.stats["units_total"], "units_rank0": r.stats["units"], "speech_s_rank0": r.stats["speech_s"],
            "windows_rank0": m.stats["windows"] - p0["windows"], "decoder_steps_rank0": m.stats["decode_steps"] - p0["decode_steps"],
            "device_passes_rank0": m.stats["device_passes"] - p0["device_passes"], "segments_out": srt.count("-->"), "srt_bytes": len(srt.encode()),
            "clocks": clocks}))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="large-v3")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--workload", default="window", choices=["window", "stream", "streams8"])
    ap.add_argument("--stream-minutes", type=float, default=120.0)
    ap.add_argument("--decode", default=None, choices=["preset", "greedy"], help="default: greedy for --workload window, preset for streams")
    ap.add_argument("--word-timestamps", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step as DIR/<name>.npy (window workload, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "window"):
        ap.error("--dump-outputs is implemented for --impl ours --workload window")
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (no CPU fallback in the product path)")
        if args.workload != "window":
            run_stream(args)
        else:
            run_ours(args)


if __name__ == "__main__":
    main()
