"""CPU restatement of openai-whisper @ c0d2f62 (the arithmetic the reference reaches
through ``whisperjav/modules/whisper_pro_asr.py:182,433``).  TEST INFRASTRUCTURE.

Each function names the upstream file it follows (upstream is *not* vendored in
/root/reference; the spec is restated in SURVEY.md section 8c):

* ``log_mel_spectrogram`` / ``pad_or_trim`` / ``mel_filters``   <- whisper/audio.py
* ``sinusoids`` / ``encoder_forward`` / ``decoder_forward``      <- whisper/model.py
* ``DecodingOptions`` / ``decode`` (greedy, logit filters),
  ``BeamSearch`` / ``decode_beam`` / ``rank_maximum_likelihood`` <- whisper/decoding.py
* ``transcribe`` (seek loop, thresholds, timestamp slicing)      <- whisper/transcribe.py

``sim_fp16=True`` reproduces the rounding points of the reference's fp16 GPU run
(``fp16=True``: ``model.half()``; every Linear/Conv/GELU/residual output is an fp16
tensor, LayerNorm and softmax compute in fp32 and cast back, logits are ``.float()``).
Sums of products are taken in float64 before each rounding point (``ACC_DTYPE``), so the
result does not depend on how many host threads share a matrix product.  Parity of the
CUDA path is asserted against this mode.
"""
from __future__ import annotations

import math
import zlib
from contextlib import contextmanager
from dataclasses import dataclass, field, replace
from typing import Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch
import torch.nn.functional as F

# ----------------------------------------------------------------------------- audio.py
SAMPLE_RATE = 16000
N_FFT = 400
HOP_LENGTH = 160
CHUNK_LENGTH = 30
N_SAMPLES = CHUNK_LENGTH * SAMPLE_RATE  # 480000
N_FRAMES = N_SAMPLES // HOP_LENGTH  # 3000
N_SAMPLES_PER_TOKEN = HOP_LENGTH * 2
FRAMES_PER_SECOND = SAMPLE_RATE // HOP_LENGTH
TOKENS_PER_SECOND = SAMPLE_RATE // N_SAMPLES_PER_TOKEN


def _hz_to_mel_slaney(f):
    f = np.asarray(f, dtype=np.float64)
    f_sp = 200.0 / 3
    mels = f / f_sp
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = np.log(6.4) / 27.0
    return np.where(f >= min_log_hz, min_log_mel + np.log(np.maximum(f, 1e-30) / min_log_hz) / logstep, mels)


def _mel_to_hz_slaney(m):
    m = np.asarray(m, dtype=np.float64)
    f_sp = 200.0 / 3
    freqs = f_sp * m
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = np.log(6.4) / 27.0
    return np.where(m >= min_log_mel, min_log_hz * np.exp(logstep * (m - min_log_mel)), freqs)


def mel_filters(n_mels: int) -> np.ndarray:
    """``librosa.filters.mel(sr=16000, n_fft=400, n_mels=n_mels)`` (Slaney scale + Slaney
    area norm) -- the matrix upstream ships as ``assets/mel_filters.npz`` (audio.py).
    Returns float32 [n_mels, 201]."""
    n_freqs = N_FFT // 2 + 1
    fftfreqs = np.linspace(0.0, SAMPLE_RATE / 2, n_freqs)
    mel_pts = np.linspace(_hz_to_mel_slaney(0.0), _hz_to_mel_slaney(SAMPLE_RATE / 2), n_mels + 2)
    hz_pts = _mel_to_hz_slaney(mel_pts)
    fdiff = np.diff(hz_pts)
    ramps = hz_pts[:, None] - fftfreqs[None, :]
    weights = np.zeros((n_mels, n_freqs), dtype=np.float64)
    for i in range(n_mels):
        lower = -ramps[i] / fdiff[i]
        upper = ramps[i + 2] / fdiff[i + 1]
        weights[i] = np.maximum(0.0, np.minimum(lower, upper))
    enorm = 2.0 / (hz_pts[2 : n_mels + 2] - hz_pts[:n_mels])
    weights *= enorm[:, None]
    return weights.astype(np.float32)


def pad_or_trim(array: torch.Tensor, length: int = N_SAMPLES, *, axis: int = -1) -> torch.Tensor:
    """audio.py::pad_or_trim."""
    if array.shape[axis] > length:
        array = array.index_select(dim=axis, index=torch.arange(length))
    if array.shape[axis] < length:
        pad_widths = [(0, 0)] * array.ndim
        pad_widths[axis] = (0, length - array.shape[axis])
        array = F.pad(array, [p for sizes in pad_widths[::-1] for p in sizes])
    return array


def log_mel_spectrogram(audio: Union[np.ndarray, torch.Tensor], n_mels: int = 80, padding: int = 0) -> torch.Tensor:
    """audio.py::log_mel_spectrogram (fp32): zero right-pad, periodic Hann(400),
    centred reflect-padded STFT(400, hop 160), drop last frame, |.|^2, mel, log10 clamp,
    global ``max - 8`` floor, ``(x + 4) / 4``.  Returns [n_mels, n_frames]."""
    if not torch.is_tensor(audio):
        audio = torch.from_numpy(np.ascontiguousarray(audio))
    audio = audio.to(torch.float32)
    if padding > 0:
        audio = F.pad(audio, (0, padding))
    window = torch.hann_window(N_FFT)
    stft = torch.stft(audio, N_FFT, HOP_LENGTH, window=window, return_complex=True)
    magnitudes = stft[..., :-1].abs() ** 2
    filters = torch.from_numpy(mel_filters(n_mels))
    mel_spec = filters @ magnitudes
    log_spec = torch.clamp(mel_spec, min=1e-10).log10()
    log_spec = torch.maximum(log_spec, log_spec.max() - 8.0)
    log_spec = (log_spec + 4.0) / 4.0
    return log_spec


# ----------------------------------------------------------------------------- model.py
@dataclass
class ModelDimensions:
    n_mels: int
    n_audio_ctx: int
    n_audio_state: int
    n_audio_head: int
    n_audio_layer: int
    n_vocab: int
    n_text_ctx: int
    n_text_state: int
    n_text_head: int
    n_text_layer: int


DIMS = {
    "tiny": ModelDimensions(80, 1500, 384, 6, 4, 51865, 448, 384, 6, 4),
    "base": ModelDimensions(80, 1500, 512, 8, 6, 51865, 448, 512, 8, 6),
    "small": ModelDimensions(80, 1500, 768, 12, 12, 51865, 448, 768, 12, 12),
    "medium": ModelDimensions(80, 1500, 1024, 16, 24, 51865, 448, 1024, 16, 24),
    "large-v2": ModelDimensions(80, 1500, 1280, 20, 32, 51865, 448, 1280, 20, 32),
    "large-v3": ModelDimensions(128, 1500, 1280, 20, 32, 51866, 448, 1280, 20, 32),
}


def sinusoids(length: int, channels: int, max_timescale: float = 10000.0) -> torch.Tensor:
    """model.py::sinusoids."""
    assert channels % 2 == 0
    log_timescale_increment = np.log(max_timescale) / (channels // 2 - 1)
    inv_timescales = torch.exp(-log_timescale_increment * torch.arange(channels // 2))
    scaled_time = torch.arange(length)[:, np.newaxis] * inv_timescales[np.newaxis, :]
    return torch.cat([torch.sin(scaled_time), torch.cos(scaled_time)], dim=1)


# Sums of products (Linear, Conv1d, attention, logits) run in ACC_DTYPE and are then rounded where the reference rounds.  A
# float32 BLAS sum on the host depends on how many threads share it; the last-bit differences flip fp16 roundings, and the
# flips grow through the layers to several fp16 quanta of the logits -- as large as the device-vs-oracle differences the
# parity checks bound.  A float64 sum is exact far below fp16 precision, so the oracle gives the same numbers whatever the
# thread count.  LayerNorm and softmax stay in float32 as upstream computes them (one row per reduction: no thread split).
ACC_DTYPE = torch.float64


@contextmanager
def accumulation(dtype: torch.dtype):
    """Run the oracle with sums of products in ``dtype``; ``torch.float32`` is the reference's own arithmetic (what
    bench.py's CPU baseline times)."""
    global ACC_DTYPE
    saved, ACC_DTYPE = ACC_DTYPE, dtype
    try:
        yield
    finally:
        ACC_DTYPE = saved


def _mm(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    return (a.to(ACC_DTYPE) @ b.to(ACC_DTYPE)).float()


def _conv1d(x, w, b, **kw):
    return F.conv1d(x.to(ACC_DTYPE), w.to(ACC_DTYPE), None if b is None else b.to(ACC_DTYPE), **kw).float()


class Rounder:
    """fp16 rounding points of the reference's ``fp16=True`` run (identity when off)."""

    def __init__(self, sim_fp16: bool):
        self.on = bool(sim_fp16)

    def __call__(self, t: torch.Tensor) -> torch.Tensor:
        return t.half().float() if self.on else t


class PreparedWeights(dict):
    """fp32 copies of the weights, already rounded the way the run will use them (see prepare_weights)."""


def prepare_weights(weights: Dict[str, torch.Tensor], sim_fp16: bool = True) -> "PreparedWeights":
    """Convert once instead of per call: fp32 tensors, fp16-rounded when ``sim_fp16`` (what
    ``weight.to(x.dtype)`` yields upstream).  LayerNorm parameters and positional buffers stay fp32."""
    out = PreparedWeights()
    for k, v in weights.items():
        f = v.float()
        keep = ("_ln." in k or ".ln." in k or ".ln_post." in k or k.endswith("positional_embedding"))
        out[k] = f if (keep or not sim_fp16) else f.half().float()
    return out


def _w(weights: Dict[str, torch.Tensor], name: str, r: Rounder) -> Optional[torch.Tensor]:
    t = weights.get(name)
    if t is None:
        return None
    if isinstance(weights, PreparedWeights):
        return t
    return r(t.float())


def _layer_norm(x, weights, prefix, r):
    # model.py::LayerNorm.forward: super().forward(x.float()).type(x.dtype)
    n = x.shape[-1]
    y = F.layer_norm(x.float(), (n,), weights[prefix + ".weight"].float(), weights[prefix + ".bias"].float(), 1e-5)
    return r(y)


def _linear(x, weights, prefix, r):
    # model.py::Linear.forward: weight/bias cast to x.dtype; fp32 accumulate, fp16 store
    w = _w(weights, prefix + ".weight", r)
    b = _w(weights, prefix + ".bias", r)
    y = _mm(x, w.t())
    if b is not None:
        y = y + b
    return r(y)


def _gelu(x, r):
    return r(F.gelu(x))  # exact erf GELU (nn.GELU default)


def _attention(q, k, v, n_head, causal: bool, r, capture: Optional[list] = None):
    """model.py::MultiHeadAttention.qkv_attention (SDPA branch: softmax(q k^T / sqrt(d)) v,
    fp32 softmax, fp16 in/out).  ``capture``: the scaled scores ``qk`` [B, H, Tq, Tk] are appended (what the
    non-SDPA branch returns next to the output and timing.py collects through forward hooks)."""
    n_batch, n_ctx, n_state = q.shape
    d = n_state // n_head
    q = q.view(n_batch, n_ctx, n_head, d).permute(0, 2, 1, 3)
    k = k.view(n_batch, k.shape[1], n_head, d).permute(0, 2, 1, 3)
    v = v.view(n_batch, v.shape[1], n_head, d).permute(0, 2, 1, 3)
    qk = _mm(q, k.transpose(-1, -2)) * (d ** -0.5)
    if causal and n_ctx > 1:
        t_k = k.shape[2]
        mask = torch.full((n_ctx, t_k), float("-inf")).triu_(1 + t_k - n_ctx)
        qk = qk + mask
    if capture is not None:
        capture.append(r(qk).float())  # fp16 matmul output under fp16=True, then timing.py's .float()
    w = r(torch.softmax(qk.float(), dim=-1))  # non-SDPA branch: softmax(qk.float()).to(q.dtype)
    out = _mm(w, v)
    return r(out.permute(0, 2, 1, 3).flatten(start_dim=2))


def encoder_forward(weights: Dict[str, torch.Tensor], dims: ModelDimensions, mel: torch.Tensor,
                    sim_fp16: bool = True, return_layers: bool = False):
    """model.py::AudioEncoder.forward.  mel [B, n_mels, 3000] -> [B, 1500, n_state]."""
    r = Rounder(sim_fp16)
    x = r(mel.float())
    x = _gelu(r(_conv1d(x, _w(weights, "encoder.conv1.weight", r), _w(weights, "encoder.conv1.bias", r), padding=1)), r)
    x = _gelu(r(_conv1d(x, _w(weights, "encoder.conv2.weight", r), _w(weights, "encoder.conv2.bias", r), stride=2, padding=1)), r)
    x = x.permute(0, 2, 1)
    pos = weights.get("encoder.positional_embedding")
    if pos is None:
        pos = sinusoids(dims.n_audio_ctx, dims.n_audio_state)
    x = r(x + pos.float())  # fp16 x + fp32 buffer -> fp32 sum, .to(x.dtype)
    layers = []
    for i in range(dims.n_audio_layer):
        p = f"encoder.blocks.{i}"
        h = _layer_norm(x, weights, p + ".attn_ln", r)
        q = _linear(h, weights, p + ".attn.query", r)
        k = _linear(h, weights, p + ".attn.key", r)
        v = _linear(h, weights, p + ".attn.value", r)
        a = _attention(q, k, v, dims.n_audio_head, False, r)
        x = r(x + _linear(a, weights, p + ".attn.out", r))
        h = _layer_norm(x, weights, p + ".mlp_ln", r)
        h = _gelu(_linear(h, weights, p + ".mlp.0", r), r)
        x = r(x + _linear(h, weights, p + ".mlp.2", r))
        if return_layers:
            layers.append(x.clone())
    x = _layer_norm(x, weights, "encoder.ln_post", r)
    return (x, layers) if return_layers else x


class DecoderState:
    """KV cache (model.py installs forward hooks on every key/value Linear; here explicit)."""

    def __init__(self):
        self.self_k: Dict[int, torch.Tensor] = {}
        self.self_v: Dict[int, torch.Tensor] = {}
        self.cross_k: Dict[int, torch.Tensor] = {}
        self.cross_v: Dict[int, torch.Tensor] = {}
        self.offset = 0


def decoder_forward(weights, dims: ModelDimensions, tokens: torch.Tensor, xa: torch.Tensor,
                    state: Optional[DecoderState] = None, sim_fp16: bool = True,
                    cross_qk: Optional[list] = None) -> torch.Tensor:
    """model.py::TextDecoder.forward with the decoding.py::PyTorchInference KV cache.
    tokens [B, T] (all tokens on the first call, then the last one) -> fp32 logits [B, T, V].
    ``cross_qk``: list that receives every layer's cross-attention scores [B, H, T, n_audio_ctx] (timing.py's hooks)."""
    r = Rounder(sim_fp16)
    if state is None:
        state = DecoderState()
    offset = state.offset
    T = tokens.shape[-1]
    emb = _w(weights, "decoder.token_embedding.weight", r)
    pos = weights["decoder.positional_embedding"].float()
    # fp32 embedding sum, then .to(xa.dtype)
    x = r(F.embedding(tokens, weights["decoder.token_embedding.weight"].float()) + pos[offset : offset + T])
    for i in range(dims.n_text_layer):
        p = f"decoder.blocks.{i}"
        h = _layer_norm(x, weights, p + ".attn_ln", r)
        q = _linear(h, weights, p + ".attn.query", r)
        k = _linear(h, weights, p + ".attn.key", r)
        v = _linear(h, weights, p + ".attn.value", r)
        if i in state.self_k:
            k = torch.cat([state.self_k[i], k], dim=1)
            v = torch.cat([state.self_v[i], v], dim=1)
        state.self_k[i], state.self_v[i] = k, v
        a = _attention(q, k, v, dims.n_text_head, True, r)
        x = r(x + _linear(a, weights, p + ".attn.out", r))
        h = _layer_norm(x, weights, p + ".cross_attn_ln", r)
        q = _linear(h, weights, p + ".cross_attn.query", r)
        if i not in state.cross_k:
            state.cross_k[i] = _linear(xa, weights, p + ".cross_attn.key", r)
            state.cross_v[i] = _linear(xa, weights, p + ".cross_attn.value", r)
        a = _attention(q, state.cross_k[i], state.cross_v[i], dims.n_text_head, False, r, cross_qk)
        x = r(x + _linear(a, weights, p + ".cross_attn.out", r))
        h = _layer_norm(x, weights, p + ".mlp_ln", r)
        h = _gelu(_linear(h, weights, p + ".mlp.0", r), r)
        x = r(x + _linear(h, weights, p + ".mlp.2", r))
    x = _layer_norm(x, weights, "decoder.ln", r)
    state.offset = offset + T
    return r(_mm(x, emb.t())).float()  # fp16 matmul output, then .float()


# ----------------------------------------------------------------------------- tokenizer.py
@dataclass
class SpecialTokens:
    """Special-token ids of the multilingual tokenizer (tokenizer.py).  The vocabulary file
    itself is not available offline; only ids matter for parity."""
    n_vocab: int
    eot: int = 50257
    sot: int = 50258
    num_languages: int = 99
    language: str = "ja"
    task: str = "transcribe"
    blank_tokens: Tuple[int, ...] = (220,)  # tokenizer.encode(" ")

    LANG_INDEX = {"en": 0, "zh": 1, "de": 2, "es": 3, "ru": 4, "ko": 5, "fr": 6, "ja": 7, "pt": 8, "tr": 9}

    def __post_init__(self):
        self.num_languages = self.n_vocab - 51765 - 1  # tokenizer.py / model.py::num_languages
        base = self.sot + 1 + self.num_languages
        self.translate = base
        self.transcribe = base + 1
        self.sot_lm = base + 2
        self.sot_prev = base + 3
        self.no_speech = base + 4
        self.no_timestamps = base + 5
        self.timestamp_begin = base + 6

    @property
    def language_token(self) -> int:
        return self.sot + 1 + self.LANG_INDEX[self.language]

    @property
    def sot_sequence(self) -> Tuple[int, ...]:
        task_tok = self.transcribe if self.task == "transcribe" else self.translate
        return (self.sot, self.language_token, task_tok)

    @property
    def non_speech_tokens(self) -> Tuple[int, ...]:
        return NON_SPEECH_SYMBOL_TOKENS


# tokenizer.py::non_speech_tokens for the multilingual vocabulary (ids of symbol tokens).  The
# same list ships in HF ``configuration_whisper.NON_SPEECH_TOKENS_MULTI`` (its first 82 entries;
# the trailing specials there are appended separately below per decoding.py::_get_suppress_tokens).
NON_SPEECH_SYMBOL_TOKENS = (
    1, 2, 7, 8, 9, 10, 14, 25, 26, 27, 28, 29, 31, 58, 59, 60, 61, 62, 63, 90, 91, 92, 93, 359, 503, 522,
    542, 873, 893, 902, 918, 922, 931, 1350, 1853, 1982, 2460, 2627, 3246, 3253, 3268, 3536, 3846, 3961,
    4183, 4667, 6585, 6647, 7273, 9061, 9383, 10428, 10929, 11938, 12033, 12331, 12562, 13793, 14157,
    14635, 15265, 15618, 16553, 16604, 18362, 18956, 20075, 21675, 22520, 26130, 26161, 26435, 28279,
    29464, 31650, 32302, 32470, 36865, 42863, 47425, 49870, 50254,
)


def placeholder_detokenize(tokens: Sequence[int]) -> str:
    """Stand-in for ``tokenizer.decode`` (no vocabulary offline): one CJK code point per id.
    Deterministic and injective enough for compression-ratio / empty-text logic."""
    return "".join(chr(0x4E00 + (int(t) % 20992)) for t in tokens)


def compression_ratio(text: str) -> float:
    """utils.py::compression_ratio."""
    text_bytes = text.encode("utf-8")
    return len(text_bytes) / len(zlib.compress(text_bytes))


# ----------------------------------------------------------------------------- decoding.py
@dataclass(frozen=True)
class DecodingOptions:
    task: str = "transcribe"
    language: Optional[str] = None
    temperature: float = 0.0
    sample_len: Optional[int] = None
    best_of: Optional[int] = None
    beam_size: Optional[int] = None
    patience: Optional[float] = None
    length_penalty: Optional[float] = None
    prompt: Optional[Union[str, List[int]]] = None
    prefix: Optional[Union[str, List[int]]] = None
    suppress_tokens: Optional[Union[str, Sequence[int]]] = "-1"
    suppress_blank: bool = True
    without_timestamps: bool = False
    max_initial_timestamp: Optional[float] = 1.0
    fp16: bool = True


@dataclass
class DecodingResult:
    tokens: List[int] = field(default_factory=list)
    text: str = ""
    avg_logprob: float = np.nan
    no_speech_prob: float = np.nan
    temperature: float = np.nan
    compression_ratio: float = np.nan
    language: str = "ja"
    sum_logprob: float = np.nan
    # diagnostics (not in upstream): per-step top-2 logit margin after filtering; under teacher forcing also the oracle's own
    # pick per step and how far below the oracle's top filtered logit the forced token sits (0 = the oracle agrees)
    margins: List[float] = field(default_factory=list)
    picks: List[int] = field(default_factory=list)
    forced_gap: List[float] = field(default_factory=list)


def get_suppress_tokens(tok: SpecialTokens, options: DecodingOptions) -> Tuple[int, ...]:
    """decoding.py::DecodingTask._get_suppress_tokens."""
    suppress_tokens = options.suppress_tokens
    if isinstance(suppress_tokens, str):
        suppress_tokens = [int(t) for t in suppress_tokens.split(",")]
    if suppress_tokens is None:
        suppress_tokens = []
    suppress_tokens = list(suppress_tokens)
    if -1 in suppress_tokens:
        suppress_tokens = [t for t in suppress_tokens if t >= 0]
        suppress_tokens.extend(tok.non_speech_tokens)
    suppress_tokens.extend([tok.transcribe, tok.translate, tok.sot, tok.sot_prev, tok.sot_lm])
    suppress_tokens.append(tok.no_speech)
    return tuple(sorted(set(suppress_tokens)))


def get_initial_tokens(tok: SpecialTokens, options: DecodingOptions, n_ctx: int) -> Tuple[int, ...]:
    """decoding.py::DecodingTask._get_initial_tokens (token-id prompts/prefixes only)."""
    sot_sequence = list(tok.sot_sequence)
    if options.without_timestamps:
        sot_sequence = sot_sequence + [tok.no_timestamps]
    tokens = list(sot_sequence)
    sample_len = options.sample_len or n_ctx // 2
    if options.prefix:
        prefix_tokens = list(options.prefix)
        if sample_len is not None:
            max_prefix_len = n_ctx // 2 - sample_len
            prefix_tokens = prefix_tokens[-max_prefix_len:]
        tokens = tokens + prefix_tokens
    if options.prompt:
        prompt_tokens = list(options.prompt)
        tokens = [tok.sot_prev] + prompt_tokens[-(n_ctx // 2 - 1):] + tokens
    return tuple(tokens)


def apply_logit_filters(logits: torch.Tensor, tokens: torch.Tensor, tok: SpecialTokens, options: DecodingOptions,
                        sample_begin: int, suppress: Tuple[int, ...], max_initial_timestamp_index: Optional[int]):
    """SuppressBlank, SuppressTokens, ApplyTimestampRules (decoding.py), in upstream order.
    In place on fp32 ``logits`` [B, V]."""
    NEG = -np.inf
    if options.suppress_blank and tokens.shape[1] == sample_begin:
        logits[:, list(tok.blank_tokens) + [tok.eot]] = NEG
    if suppress:
        logits[:, list(suppress)] = NEG
    if not options.without_timestamps:
        logits[:, tok.no_timestamps] = NEG
        for k in range(tokens.shape[0]):
            seq = tokens[k, sample_begin:].tolist()
            last_was_timestamp = len(seq) >= 1 and seq[-1] >= tok.timestamp_begin
            penultimate_was_timestamp = len(seq) < 2 or seq[-2] >= tok.timestamp_begin
            if last_was_timestamp:
                if penultimate_was_timestamp:
                    logits[k, tok.timestamp_begin:] = NEG
                else:
                    logits[k, : tok.eot] = NEG
            timestamps = [t for t in seq if t >= tok.timestamp_begin]
            if len(timestamps) > 0:
                if last_was_timestamp and not penultimate_was_timestamp:
                    timestamp_last = timestamps[-1]
                else:
                    timestamp_last = timestamps[-1] + 1
                logits[k, tok.timestamp_begin: timestamp_last] = NEG
        if tokens.shape[1] == sample_begin:
            logits[:, : tok.timestamp_begin] = NEG
            if max_initial_timestamp_index is not None:
                last_allowed = tok.timestamp_begin + max_initial_timestamp_index
                logits[:, last_allowed + 1:] = NEG
        logprobs = F.log_softmax(logits.float(), dim=-1)
        for k in range(tokens.shape[0]):
            timestamp_logprob = logprobs[k, tok.timestamp_begin:].logsumexp(dim=-1)
            max_text_token_logprob = logprobs[k, : tok.timestamp_begin].max()
            if timestamp_logprob > max_text_token_logprob:
                logits[k, : tok.timestamp_begin] = NEG


def decode(weights, dims: ModelDimensions, mel: torch.Tensor, options: DecodingOptions,
           sim_fp16: bool = True, audio_features: Optional[torch.Tensor] = None,
           return_logits: bool = False, forced_tokens: Optional[Sequence[Sequence[int]]] = None) -> List[DecodingResult]:
    """decoding.py::DecodingTask.run for greedy decoding (``beam_size is None``, T == 0).

    mel [B, n_mels, 3000] (or pre-computed ``audio_features`` [B, 1500, n_state]).
    ``forced_tokens`` (diagnostic, not upstream): per row the sampled ids to feed instead of the oracle's own picks
    (teacher forcing; a row is fed EOT once its list is exhausted).  ``picks`` / ``forced_gap`` then say, per step, what
    the oracle would have chosen on that prefix and how far below its top filtered logit the forced id sits."""
    if options.beam_size is not None:
        if return_logits:
            raise NotImplementedError("return_logits is a greedy-path diagnostic")
        return decode_beam(weights, dims, mel, options, sim_fp16, audio_features)
    if (options.best_of or 1) > 1:
        raise NotImplementedError("oracle covers greedy and beam-search decoding; sampling is checked statistically on the device path")
    if options.temperature != 0.0:
        raise NotImplementedError("oracle covers temperature 0 only")
    tok = SpecialTokens(dims.n_vocab, language=options.language or "en", task=options.task)
    n_ctx = dims.n_text_ctx
    sample_len = options.sample_len or n_ctx // 2
    initial_tokens = get_initial_tokens(tok, options, n_ctx)
    sample_begin = len(initial_tokens)
    sot_index = initial_tokens.index(tok.sot)
    suppress = get_suppress_tokens(tok, options) if options.suppress_tokens else ()
    max_initial_timestamp_index = None
    if not options.without_timestamps and options.max_initial_timestamp:
        precision = CHUNK_LENGTH / dims.n_audio_ctx
        max_initial_timestamp_index = round(options.max_initial_timestamp / precision)

    if audio_features is None:
        audio_features = encoder_forward(weights, dims, mel, sim_fp16)
    n_audio = audio_features.shape[0]
    tokens = torch.tensor([initial_tokens]).repeat(n_audio, 1)
    sum_logprobs = torch.zeros(n_audio)
    no_speech_probs = [np.nan] * n_audio
    state = DecoderState()
    margins: List[List[float]] = [[] for _ in range(n_audio)]
    picks: List[List[int]] = [[] for _ in range(n_audio)]
    forced_gap: List[List[float]] = [[] for _ in range(n_audio)]
    all_logits = []
    for i in range(sample_len):
        inp = tokens if i == 0 else tokens[:, -1:]
        logits = decoder_forward(weights, dims, inp, audio_features, state, sim_fp16)
        if i == 0:
            probs_at_sot = logits[:, sot_index].float().softmax(dim=-1)
            no_speech_probs = probs_at_sot[:, tok.no_speech].tolist()
        logits = logits[:, -1]
        if return_logits:
            all_logits.append(logits.clone())
        apply_logit_filters(logits, tokens, tok, options, sample_begin, suppress, max_initial_timestamp_index)
        # GreedyDecoder.update
        next_tokens = logits.argmax(dim=-1)
        top2 = logits.topk(2, dim=-1).values
        logprobs = F.log_softmax(logits.float(), dim=-1)
        current_logprobs = logprobs[torch.arange(n_audio), next_tokens]
        alive = tokens[:, -1] != tok.eot
        if forced_tokens is not None:
            forced = torch.tensor([(list(f)[i] if i < len(f) else tok.eot) for f in forced_tokens])
            for b in range(n_audio):
                if alive[b]:
                    picks[b].append(int(next_tokens[b]))
                    forced_gap[b].append(float(top2[b, 0] - logits[b, forced[b]]))
            next_tokens = forced
            current_logprobs = logprobs[torch.arange(n_audio), next_tokens]
        for b in range(n_audio):
            if alive[b]:
                margins[b].append(float(top2[b, 0] - top2[b, 1]))
        sum_logprobs += current_logprobs * alive
        next_tokens[~alive] = tok.eot
        tokens = torch.cat([tokens, next_tokens[:, None]], dim=-1)
        completed = bool((tokens[:, -1] == tok.eot).all())
        if completed or tokens.shape[-1] > n_ctx:
            break
    tokens = F.pad(tokens, (0, 1), value=tok.eot)  # GreedyDecoder.finalize
    results = []
    for b in range(n_audio):
        t = tokens[b]
        end = int((t == tok.eot).nonzero()[0, 0])
        out = t[sample_begin:end].tolist()
        text = placeholder_detokenize([x for x in out if x < tok.eot]).strip()
        slp = float(sum_logprobs[b])
        results.append(DecodingResult(tokens=out, text=text, avg_logprob=slp / (len(out) + 1),
                                      no_speech_prob=float(no_speech_probs[b]), temperature=options.temperature,
                                      compression_ratio=compression_ratio(text) if text else 0.0,
                                      language=options.language or "en", sum_logprob=slp, margins=margins[b],
                                      picks=picks[b], forced_gap=forced_gap[b]))
    if return_logits:
        return results, all_logits
    return results


class BeamSearch:
    """decoding.py::BeamSearchDecoder restated on plain tensors: ``update`` consumes the filtered logits of every beam row
    and returns the kept sequences plus the row each one continues (upstream calls ``inference.rearrange_kv_cache`` with
    those indices), ``finalize`` tops the finished lists up from the live beams.  Ranking of equal scores follows the
    insertion order of upstream's dicts (beam index, then top-k order) because ``sorted`` is stable.

    Parity status: restated from openai-whisper 20250625 @ c0d2f62, which is absent from this container -> unpinned against
    the reference itself; pinned only through properties (tests/test_oracle_beam.py)."""

    def __init__(self, beam_size: int, eot: int, patience: Optional[float] = None):
        self.beam_size = beam_size
        self.eot = eot
        self.patience = patience or 1.0
        self.max_candidates = round(beam_size * self.patience)
        self.finished_sequences: Optional[List[Dict[Tuple[int, ...], float]]] = None
        assert self.max_candidates > 0, f"Invalid beam size ({beam_size}) or patience ({patience})"

    def reset(self):
        self.finished_sequences = None

    def update(self, tokens: torch.Tensor, logits: torch.Tensor, sum_logprobs: torch.Tensor):
        if tokens.shape[0] % self.beam_size != 0:
            raise ValueError(f"{tokens.shape}[0] % {self.beam_size} != 0")
        n_audio = tokens.shape[0] // self.beam_size
        if self.finished_sequences is None:
            self.finished_sequences = [{} for _ in range(n_audio)]
        logprobs = F.log_softmax(logits.float(), dim=-1)
        next_tokens, source_indices, finished_sequences = [], [], []
        for i in range(n_audio):
            scores, sources, finished = {}, {}, {}
            # STEP 1: cumulative log probabilities of the candidates of every beam (identical beams collapse: dict keys)
            for j in range(self.beam_size):
                idx = i * self.beam_size + j
                prefix = tokens[idx].tolist()
                for logprob, token in zip(*logprobs[idx].topk(self.beam_size + 1)):
                    new_logprob = (sum_logprobs[idx] + logprob).item()
                    sequence = tuple(prefix + [token.item()])
                    scores[sequence] = new_logprob
                    sources[sequence] = idx
            # STEP 2: rank the candidates, keep the top beam_size live ones; EOT-terminated ones passed on the way finish
            saved = 0
            for sequence in sorted(scores, key=scores.get, reverse=True):
                if sequence[-1] == self.eot:
                    finished[sequence] = scores[sequence]
                else:
                    sum_logprobs[len(next_tokens)] = scores[sequence]
                    next_tokens.append(sequence)
                    source_indices.append(sources[sequence])
                    saved += 1
                    if saved == self.beam_size:
                        break
            finished_sequences.append(finished)
        tokens = torch.tensor(next_tokens)
        for previously_finished, newly_finished in zip(self.finished_sequences, finished_sequences):
            for seq in sorted(newly_finished, key=newly_finished.get, reverse=True):
                if len(previously_finished) >= self.max_candidates:
                    break  # the candidate list is full
                previously_finished[seq] = newly_finished[seq]
        completed = all(len(sequences) >= self.max_candidates for sequences in self.finished_sequences)
        return tokens, source_indices, completed

    def finalize(self, preceding_tokens: torch.Tensor, sum_logprobs: torch.Tensor):
        """preceding_tokens [n_audio, beam, T], sum_logprobs [n_audio, beam]."""
        sum_logprobs = sum_logprobs.cpu()
        for i, sequences in enumerate(self.finished_sequences):
            if len(sequences) < self.beam_size:  # not enough finished: take the best live beams, EOT appended
                for j in list(np.argsort(sum_logprobs[i].numpy()))[::-1]:
                    sequence = preceding_tokens[i, j].tolist() + [self.eot]
                    sequences[tuple(sequence)] = sum_logprobs[i][j].item()
                    if len(sequences) >= self.beam_size:
                        break
        tokens = [[torch.tensor(seq) for seq in sequences.keys()] for sequences in self.finished_sequences]
        sums = [list(sequences.values()) for sequences in self.finished_sequences]
        return tokens, sums


def rank_maximum_likelihood(tokens: List[List[torch.Tensor]], sum_logprobs: List[List[float]],
                            length_penalty: Optional[float] = None) -> List[int]:
    """decoding.py::MaximumLikelihoodRanker.rank: per audio the candidate with the best length-normalised log probability
    (``logprob / length``, or the Google NMT penalty ``((5 + length) / 6) ** length_penalty``)."""

    def scores(logprobs, lengths):
        result = []
        for logprob, length in zip(logprobs, lengths):
            penalty = length if length_penalty is None else ((5 + length) / 6) ** length_penalty
            result.append(logprob / penalty)
        return result

    lengths = [[len(t) for t in s] for s in tokens]
    return [int(np.argmax(scores(p, l))) for p, l in zip(sum_logprobs, lengths)]


def decode_beam(weights, dims: ModelDimensions, mel: torch.Tensor, options: DecodingOptions, sim_fp16: bool = True,
                audio_features: Optional[torch.Tensor] = None) -> List[DecodingResult]:
    """decoding.py::DecodingTask.run with ``beam_size`` set (T == 0): audio features and tokens repeated per beam, the logit
    filters applied per row, BeamSearchDecoder.update + KV-cache rearrangement every step, finalize, MaximumLikelihoodRanker."""
    if options.temperature != 0.0:
        raise NotImplementedError("beam search runs at temperature 0 (transcribe drops beam_size when t > 0)")
    n_group = options.beam_size
    tok = SpecialTokens(dims.n_vocab, language=options.language or "en", task=options.task)
    n_ctx = dims.n_text_ctx
    sample_len = options.sample_len or n_ctx // 2
    initial_tokens = get_initial_tokens(tok, options, n_ctx)
    sample_begin = len(initial_tokens)
    sot_index = initial_tokens.index(tok.sot)
    suppress = get_suppress_tokens(tok, options) if options.suppress_tokens else ()
    max_initial_timestamp_index = None
    if not options.without_timestamps and options.max_initial_timestamp:
        precision = CHUNK_LENGTH / dims.n_audio_ctx
        max_initial_timestamp_index = round(options.max_initial_timestamp / precision)
    if audio_features is None:
        audio_features = encoder_forward(weights, dims, mel, sim_fp16)
    n_audio = audio_features.shape[0]
    tokens = torch.tensor([initial_tokens]).repeat(n_audio, 1)
    # repeat text tensors by the group size
    tokens = tokens.repeat_interleave(n_group, dim=0)
    xa = audio_features.repeat_interleave(n_group, dim=0)
    n_batch = tokens.shape[0]
    sum_logprobs = torch.zeros(n_batch)
    no_speech_probs = [np.nan] * n_batch
    state = DecoderState()
    beam = BeamSearch(n_group, tok.eot, options.patience)
    for i in range(sample_len):
        inp = tokens if i == 0 else tokens[:, -1:]
        logits = decoder_forward(weights, dims, inp, xa, state, sim_fp16)
        if i == 0:
            probs_at_sot = logits[:, sot_index].float().softmax(dim=-1)
            no_speech_probs = probs_at_sot[:, tok.no_speech].tolist()
        logits = logits[:, -1]
        apply_logit_filters(logits, tokens, tok, options, sample_begin, suppress, max_initial_timestamp_index)
        tokens, source_indices, completed = beam.update(tokens, logits, sum_logprobs)
        # PyTorchInference.rearrange_kv_cache: self-attention caches follow their beams (cross K/V rows of one audio are equal)
        if source_indices != list(range(len(source_indices))):
            idx = torch.tensor(source_indices)
            for layer in list(state.self_k):
                state.self_k[layer] = state.self_k[layer][idx]
                state.self_v[layer] = state.self_v[layer][idx]
        if completed or tokens.shape[-1] > n_ctx:
            break
    no_speech_probs = no_speech_probs[::n_group]
    tokens = tokens.reshape(n_audio, n_group, -1)
    sum_logprobs = sum_logprobs.reshape(n_audio, n_group)
    cand_tokens, cand_sums = beam.finalize(tokens, sum_logprobs)
    cand_tokens = [[t[sample_begin: int((t == tok.eot).nonzero()[0, 0])] for t in s] for s in cand_tokens]
    selected = rank_maximum_likelihood(cand_tokens, cand_sums, options.length_penalty)
    results = []
    for b in range(n_audio):
        out = cand_tokens[b][selected[b]].tolist()
        slp = float(cand_sums[b][selected[b]])
        text = placeholder_detokenize([x for x in out if x < tok.eot]).strip()
        results.append(DecodingResult(tokens=out, text=text, avg_logprob=slp / (len(out) + 1), no_speech_prob=float(no_speech_probs[b]),
                                      temperature=options.temperature, compression_ratio=compression_ratio(text) if text else 0.0,
                                      language=options.language or "en", sum_logprob=slp))
    return results


# ----------------------------------------------------------------------------- transcribe.py
def slice_segments(tokens: List[int], tok: SpecialTokens, seek: int, segment_size: int,
                   result_fields: dict, detok=placeholder_detokenize, clear: bool = True, info: Optional[dict] = None):
    """The timestamp-token segmentation block of transcribe.py::transcribe.
    Returns (segments, seek_advance_frames).  ``clear=False`` leaves the "instantaneous or empty -> cleared" pass to the caller
    (upstream runs it after the word-timestamp block); ``info`` receives ``single_timestamp_ending``."""
    input_stride = 2
    time_precision = input_stride * HOP_LENGTH / SAMPLE_RATE
    time_offset = float(seek * HOP_LENGTH / SAMPLE_RATE)
    segment_duration = segment_size * HOP_LENGTH / SAMPLE_RATE

    def new_segment(start, end, toks):
        text_tokens = [t for t in toks if t < tok.eot]
        return {"seek": seek, "start": start, "end": end, "text": detok(text_tokens), "tokens": list(toks), **result_fields}

    ts = [t >= tok.timestamp_begin for t in tokens]
    single_timestamp_ending = ts[-2:] == [False, True]
    consecutive = [i + 1 for i in range(len(tokens) - 1) if ts[i] and ts[i + 1]]
    segments = []
    if len(consecutive) > 0:
        slices = list(consecutive)
        if single_timestamp_ending:
            slices.append(len(tokens))
        last_slice = 0
        for current_slice in slices:
            sliced = tokens[last_slice:current_slice]
            start_pos = sliced[0] - tok.timestamp_begin
            end_pos = sliced[-1] - tok.timestamp_begin
            segments.append(new_segment(time_offset + start_pos * time_precision, time_offset + end_pos * time_precision, sliced))
            last_slice = current_slice
        if single_timestamp_ending:
            advance = segment_size
        else:
            last_timestamp_pos = tokens[last_slice - 1] - tok.timestamp_begin
            advance = last_timestamp_pos * input_stride
    else:
        duration = segment_duration
        timestamps = [t for t in tokens if t >= tok.timestamp_begin]
        if len(timestamps) > 0 and timestamps[-1] != tok.timestamp_begin:
            last_timestamp_pos = timestamps[-1] - tok.timestamp_begin
            duration = last_timestamp_pos * time_precision
        segments.append(new_segment(time_offset, time_offset + duration, tokens))
        advance = segment_size
    if info is not None:
        info["single_timestamp_ending"] = single_timestamp_ending
    if clear:
        clear_empty_segments(segments)
    return segments, advance


def clear_empty_segments(segments: List[dict]) -> None:
    for seg in segments:
        if seg["start"] == seg["end"] or seg["text"].strip() == "":
            seg["text"] = ""
            seg["tokens"] = []
            if "words" in seg:
                seg["words"] = []


def transcribe(weights, dims: ModelDimensions, audio: np.ndarray, *, task="transcribe", language="ja",
               temperature=(0.0,), compression_ratio_threshold=2.4, logprob_threshold=-1.0,
               no_speech_threshold=0.6, condition_on_previous_text=True, sim_fp16=True, word_timestamps=False,
               prepend_punctuations="\"'“¿([{-", append_punctuations="\"'.。,，!！?？:：”)]}、",
               **decode_options) -> dict:
    """transcribe.py::transcribe (clip_timestamps="0", hallucination_silence_threshold=None, language given).
    One audio array -> {"text", "segments", "language"}.  Greedy or beam search at t == 0 (see ``decode``); with
    ``word_timestamps`` the alignment block of timing.py (oracle/timing_oracle.py)."""
    decode_options = {k: v for k, v in decode_options.items() if k not in ("verbose", "fp16")}
    mel = log_mel_spectrogram(audio, dims.n_mels, padding=N_SAMPLES)
    content_frames = mel.shape[-1] - N_FRAMES
    tok = SpecialTokens(dims.n_vocab, language=language, task=task)
    temperatures = [temperature] if isinstance(temperature, (int, float)) else list(temperature)

    def decode_with_fallback(segment):
        res = None
        for t in temperatures:
            kw = dict(decode_options)
            if t > 0:
                kw.pop("beam_size", None)
                kw.pop("patience", None)
            else:
                kw.pop("best_of", None)
            opts = DecodingOptions(task=task, language=language, temperature=t, **kw)
            res = decode(weights, dims, segment[None], opts, sim_fp16)[0]
            needs_fallback = False
            if compression_ratio_threshold is not None and res.compression_ratio > compression_ratio_threshold:
                needs_fallback = True
            if logprob_threshold is not None and res.avg_logprob < logprob_threshold:
                needs_fallback = True
            if (no_speech_threshold is not None and res.no_speech_prob > no_speech_threshold
                    and logprob_threshold is not None and res.avg_logprob < logprob_threshold):
                needs_fallback = False
            if not needs_fallback:
                break
        return res

    seek = 0
    all_tokens: List[int] = []
    all_segments: List[dict] = []
    prompt_reset_since = 0
    last_speech_timestamp = 0.0
    while seek < content_frames:
        segment_size = min(N_FRAMES, content_frames - seek)
        mel_segment = pad_or_trim(mel[:, seek: seek + segment_size], N_FRAMES)
        decode_options["prompt"] = all_tokens[prompt_reset_since:]
        result = decode_with_fallback(mel_segment)
        tokens = result.tokens
        if no_speech_threshold is not None:
            should_skip = result.no_speech_prob > no_speech_threshold
            if logprob_threshold is not None and result.avg_logprob > logprob_threshold:
                should_skip = False
            if should_skip:
                seek += segment_size
                continue
        fields = {"temperature": result.temperature, "avg_logprob": result.avg_logprob,
                  "compression_ratio": result.compression_ratio, "no_speech_prob": result.no_speech_prob}
        info: dict = {}
        current_segments, advance = slice_segments(tokens, tok, seek, segment_size, fields, clear=False, info=info)
        time_offset = float(seek * HOP_LENGTH / SAMPLE_RATE)
        seek += advance
        if word_timestamps:
            from . import timing_oracle as to
            xa = encoder_forward(weights, dims, mel_segment[None], sim_fp16)
            to.add_word_timestamps(weights, dims, current_segments, xa, segment_size, language=language, task=task,
                                   prepend_punctuations=prepend_punctuations, append_punctuations=append_punctuations,
                                   last_speech_timestamp=last_speech_timestamp, sim_fp16=sim_fp16)
            if not info["single_timestamp_ending"]:
                last_word_end = to.get_end(current_segments)
                if last_word_end is not None and last_word_end > time_offset:
                    seek = round(last_word_end * FRAMES_PER_SECOND)
            last_word_end = to.get_end(current_segments)
            if last_word_end is not None:
                last_speech_timestamp = last_word_end
        clear_empty_segments(current_segments)
        all_segments.extend([{"id": i, **s} for i, s in enumerate(current_segments, start=len(all_segments))])
        all_tokens.extend([t for s in current_segments for t in s["tokens"]])
        if not condition_on_previous_text or result.temperature > 0.5:
            prompt_reset_since = len(all_tokens)
    text = placeholder_detokenize([t for t in all_tokens if t < tok.eot])
    return {"text": text, "segments": all_segments, "language": language}
