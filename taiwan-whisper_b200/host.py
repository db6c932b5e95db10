"""Python host of the B200 path: the reference's two call sites, backed by libtwb200 (C ABI).

    fe    = B200WhisperFeatureExtractor(feature_size=128)                # WhisperFeatureExtractor
    model = B200WhisperForConditionalGeneration.from_hf(hf_model, dtype=torch.bfloat16)
    feats = fe(list_of_waveforms, sampling_rate=16000, return_tensors="pt", device="cuda")
    ids   = model.generate(feats["input_features"], max_length=256, num_beams=1,
                           return_timestamps=False, language="zh", task="transcribe")

mirrors, argument for argument and error for error,
  ref: training/run_pseudo_labelling.py:739-741 (fe call), :370-374 (fe.pad), :864-876,917-918 (generate)
  ref: prefiltering/validator_inference.py:41-47,57-69,78
torch supplies device memory, streams and (in bench.py) torch.distributed only; every FLOP of
the path runs in the library's CUDA kernels and the ops raise if the library is missing.
Three `torch.ops.twb200.*` operators expose the same entry points to graph-level callers.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import lib as _lib
from .configs import N_FRAMES, N_SAMPLES, SAMPLING_RATE

_TORCH2TW = {torch.float32: _lib.TW_F32, torch.bfloat16: _lib.TW_BF16, torch.int16: _lib.TW_I16, torch.int32: _lib.TW_I32}


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _dev_index(device) -> int:
    d = torch.device(device)
    if d.type != "cuda":
        raise ValueError("twb200 runs on CUDA (B200) devices only; there is no CPU fallback")
    return d.index if d.index is not None else torch.cuda.current_device()


# --------------------------------------------------------------------------------------------
# functional layer (device tensors in, device tensors out) — also registered as torch.ops.twb200.*
def log_mel(pcm: torch.Tensor, n_valid: Optional[torch.Tensor], n_mel: int) -> torch.Tensor:
    """pcm [B, N] int16 | float32 (cuda) -> [B, n_mel, 3000] float32.  N need not be 480000: rows are
    zero-extended / truncated to 30 s inside the kernel (HF __call__ pad/trim)."""
    if pcm.dim() != 2 or pcm.dtype not in (torch.int16, torch.float32):
        raise ValueError("log_mel expects a [B, N] int16 or float32 tensor")
    dev = _dev_index(pcm.device)
    ctx = _lib.Context.get(dev)
    pcm = pcm.contiguous()
    B = pcm.shape[0]
    out = torch.empty((B, n_mel, N_FRAMES), dtype=torch.float32, device=pcm.device)
    nv_ptr = None
    if n_valid is not None:
        n_valid = n_valid.to(device=pcm.device, dtype=torch.int32).contiguous()
        nv_ptr = n_valid.data_ptr()
    with torch.cuda.device(dev):
        ctx.check(ctx.lib.tw_logmel(ctx.handle, pcm.data_ptr(), _TORCH2TW[pcm.dtype], pcm.shape[1], nv_ptr, B, n_mel,
                                    out.data_ptr(), _stream_ptr(pcm.device)))
    return out


_DESC_FIELDS = ("d_model", "ffn", "heads", "enc_layers", "dec_layers", "n_mel", "vocab", "max_target", "dtype", "max_batch")
_TW2TORCH = {_lib.TW_F32: torch.float32, _lib.TW_BF16: torch.bfloat16}


def model_desc(handle: int) -> "_lib.ModelDesc":
    """The descriptor behind a raw `tw_model*` (int): everything the functional layer needs to size its outputs."""
    d = _lib.ModelDesc()
    rc = _lib.load_library().tw_model_get_desc(C.c_void_p(handle), C.byref(d))
    if rc != _lib.TW_OK:
        raise ValueError("twb200: not a live model handle")
    return d


def model_create(desc: Sequence[int], names: Sequence[str], weights: Sequence[torch.Tensor]) -> int:
    """tw_model_load over CUDA tensors: desc = (d_model, ffn, heads, enc_layers, dec_layers, n_mel, vocab, max_target,
    dtype, max_batch), names = HF state_dict keys.  Returns the `tw_model*` as an int — the handle every other op takes;
    the model owns repacked copies, so the weight tensors may be freed afterwards.  Release with model_free()."""
    if len(desc) != len(_DESC_FIELDS) or len(names) != len(weights) or not weights:
        raise ValueError("model_create: desc needs 10 ints and one name per weight tensor")
    dev = _dev_index(weights[0].device)
    ctx = _lib.Context.get(dev)
    keep, table = [], []
    with torch.cuda.device(dev):
        for name, t in zip(names, weights):
            t = t.detach()
            if t.dtype not in (torch.float32, torch.bfloat16):
                t = t.float()
            t = t.to(f"cuda:{dev}").contiguous()
            keep.append(t)
            table.append(_lib.Weight(name.encode(), t.data_ptr(), _TORCH2TW[t.dtype], t.numel()))
        torch.cuda.synchronize(dev)
        arr = (_lib.Weight * len(table))(*table)
        h = C.c_void_p()
        ctx.check(ctx.lib.tw_model_load(ctx.handle, C.byref(_lib.ModelDesc(*[int(v) for v in desc])), arr, len(table), C.byref(h)))
    del keep
    return int(h.value)


def model_free(handle: int) -> None:
    _lib.load_library().tw_model_free(C.c_void_p(handle))


def encoder_forward(handle: int, mel: torch.Tensor, tap_layer: int = -1):
    """mel [B, n_mel, 3000] float32 cuda -> enc_out [B, 1500, d] in the model dtype (tw_encode); with tap_layer >= 0 also
    the fp32 residual stream after that many layers."""
    d = model_desc(handle)
    if mel.dim() != 3 or mel.shape[-1] != N_FRAMES or mel.shape[-2] != d.n_mel:
        # HF raises ValueError on a wrong feature length (modeling_whisper.py:613-617)
        raise ValueError(f"Whisper expects the mel input features to be of length {N_FRAMES}, but found "
                         f"{mel.shape[-1]}. Make sure to pad the input mel features to {N_FRAMES}.")
    dev = _dev_index(mel.device)
    ctx = _lib.Context.get(dev)
    mel = mel.to(torch.float32).contiguous()
    B = mel.shape[0]
    out = torch.empty((B, 1500, d.d_model), dtype=_TW2TORCH[d.dtype], device=mel.device)
    tap = torch.empty((B, 1500, d.d_model), dtype=torch.float32, device=mel.device) if tap_layer >= 0 else None
    with torch.cuda.device(dev):
        ctx.check(ctx.lib.tw_encode(C.c_void_p(handle), mel.data_ptr(), B, out.data_ptr(), tap_layer,
                                    tap.data_ptr() if tap is not None else None, _stream_ptr(mel.device)))
    return (out, tap) if tap_layer >= 0 else out


def greedy_decode(handle: int, enc_out: torch.Tensor, prompt: Sequence[int], max_length: int, suppress: Sequence[int],
                  begin_suppress: Sequence[int], eos: int, pad: int, timestamp_begin: int, no_timestamps: int,
                  max_initial_ts: int, forced: Optional[torch.Tensor] = None, tap_steps: int = 0):
    """enc_out [B, 1500, d] (cuda, model dtype) -> (tokens int32 [B, max_length - P], lengths int32 [B]) by tw_decode_greedy.
    timestamp_begin < 0 switches the timestamp rules off; max_initial_ts < 0 = no limit.  forced / tap_steps: teacher
    forcing and post-rules logits taps for the parity tests."""
    d = model_desc(handle)
    B = enc_out.shape[0]
    n_gen = max_length - len(prompt)
    if n_gen <= 0 or max_length > d.max_target:
        raise ValueError(f"The length of the prompt ({len(prompt)}) plus the new tokens must fit max_length "
                         f"<= max_target_positions ({d.max_target}); got max_length={max_length}")
    dev = _dev_index(enc_out.device)
    ctx = _lib.Context.get(dev)
    enc_out = enc_out.to(_TW2TORCH[d.dtype]).contiguous()
    toks = torch.empty((B, n_gen), dtype=torch.int32, device=enc_out.device)
    lens = torch.empty((B,), dtype=torch.int32, device=enc_out.device)
    tap = torch.empty((tap_steps, B, d.vocab), dtype=torch.float32, device=enc_out.device) if tap_steps else None
    if forced is not None:
        forced = forced.to(enc_out.device, torch.int32).contiguous()
        assert forced.shape == (B, n_gen)
    rules, keep = _lib.make_rules(list(suppress), list(begin_suppress), int(eos), int(pad),
                                  None if timestamp_begin is None or timestamp_begin < 0 else int(timestamp_begin),
                                  int(no_timestamps), None if max_initial_ts is None or max_initial_ts < 0 else int(max_initial_ts))
    p = (C.c_int32 * len(prompt))(*[int(t) for t in prompt])
    with torch.cuda.device(dev):
        ctx.check(ctx.lib.tw_decode_greedy(
            C.c_void_p(handle), enc_out.data_ptr(), B, p, len(prompt), C.byref(rules), max_length, toks.data_ptr(),
            lens.data_ptr(), forced.data_ptr() if forced is not None else None,
            tap.data_ptr() if tap is not None else None, tap_steps, _stream_ptr(enc_out.device)))
    del keep
    return (toks, lens, tap) if tap_steps else (toks, lens)


def greedy_decode_rows(handle: int, enc_out: torch.Tensor, prompts: Sequence[Sequence[int]], lang_ids: Optional[Sequence[int]],
                       max_length: int, suppress: Sequence[int], begin_suppress: Sequence[int], eos: int, pad: int, timestamp_begin: int,
                       no_timestamps: int, max_initial_ts: int):
    """greedy_decode with one forced prompt per row (tw_decode_greedy_rows): prompts [B][P], lib.PROMPT_DETECT at index 1 = detect
    that row's language in step 0 among lang_ids.  Returns (tokens int32 [B, max_length - P], lengths int32 [B], languages int32 [B]:
    token 1 of every row's prompt as decoded)."""
    d = model_desc(handle)
    B = enc_out.shape[0]
    if len(prompts) != B:
        raise ValueError(f"{len(prompts)} prompts for {B} rows")
    n_gen = max_length - len(prompts[0])
    if n_gen <= 0 or max_length > d.max_target:
        raise ValueError(f"The length of the prompt ({len(prompts[0])}) plus the new tokens must fit max_length "
                         f"<= max_target_positions ({d.max_target}); got max_length={max_length}")
    dev = _dev_index(enc_out.device)
    ctx = _lib.Context.get(dev)
    enc_out = enc_out.to(_TW2TORCH[d.dtype]).contiguous()
    toks = torch.empty((B, n_gen), dtype=torch.int32, device=enc_out.device)
    lens = torch.empty((B,), dtype=torch.int32, device=enc_out.device)
    detect = any(p[1] == _lib.PROMPT_DETECT for p in prompts if len(p) > 1)
    langs = torch.empty((B,), dtype=torch.int32, device=enc_out.device) if detect else None
    rows, keep_rows, P = _lib.make_prompt_rows(prompts, lang_ids if detect else None, langs.data_ptr() if detect else None)
    rules, keep = _lib.make_rules(list(suppress), list(begin_suppress), int(eos), int(pad),
                                  None if timestamp_begin is None or timestamp_begin < 0 else int(timestamp_begin),
                                  int(no_timestamps), None if max_initial_ts is None or max_initial_ts < 0 else int(max_initial_ts))
    with torch.cuda.device(dev):
        ctx.check(ctx.lib.tw_decode_greedy_rows(C.c_void_p(handle), enc_out.data_ptr(), B, C.byref(rows), P, C.byref(rules), max_length,
                                                toks.data_ptr(), lens.data_ptr(), None, None, 0, _stream_ptr(enc_out.device)))
    del keep, keep_rows
    if not detect:       # every language was given: nothing to read back
        langs = torch.tensor([p[1] if len(p) > 1 else -1 for p in prompts], dtype=torch.int32, device=enc_out.device)
    return toks, lens, langs


def detect_language(handle: int, enc_out: torch.Tensor, lang_ids) -> torch.Tensor:
    """enc_out [B, 1500, d] (cuda) -> int32 [B]: the language id of every row (tw_detect_language: the logits of the step fed
    <|startoftranscript|>, masked to lang_ids, argmax — HF WhisperGenerationMixin.detect_language)."""
    d = model_desc(handle)
    if enc_out.dim() != 3 or enc_out.shape[1:] != (1500, d.d_model):
        raise ValueError(f"encoder output must be [B, 1500, {d.d_model}], got {tuple(enc_out.shape)}")
    ids = [int(t) for t in (lang_ids.tolist() if torch.is_tensor(lang_ids) else lang_ids)]
    dev = _dev_index(enc_out.device)
    ctx = _lib.Context.get(dev)
    enc_out = enc_out.to(_TW2TORCH[d.dtype]).contiguous()
    B = enc_out.shape[0]
    out = torch.empty((B,), dtype=torch.int32, device=enc_out.device)
    arr = (C.c_int32 * max(1, len(ids)))(*ids)
    with torch.cuda.device(dev):
        ctx.check(ctx.lib.tw_detect_language(C.c_void_p(handle), enc_out.data_ptr(), B, arr, len(ids), out.data_ptr(),
                                             _stream_ptr(enc_out.device)))
    return out


def decoder_logits(handle: int, enc_out: torch.Tensor, decoder_input_ids: torch.Tensor) -> torch.Tensor:
    """enc_out [B,1500,d] + decoder_input_ids [B,T] -> fp32 logits [B,T,V] of every position in ONE batched decoder pass
    (tw_decoder_logits).  The returned tensor is a view whose row pitch is V rounded up to 4 floats."""
    d = model_desc(handle)
    if decoder_input_ids.dim() != 2:
        raise ValueError("decoder_input_ids must be [batch, target_length]")
    B, T = decoder_input_ids.shape
    if B > d.max_batch:
        raise ValueError(f"batch {B} > max_batch {d.max_batch}")
    if T < 1 or T > d.max_target:
        raise ValueError(f"decoder_input_ids length {T} must be in 1..max_target_positions ({d.max_target})")
    dev = _dev_index(enc_out.device)
    ctx = _lib.Context.get(dev)
    enc_out = enc_out.to(_TW2TORCH[d.dtype]).contiguous()
    if enc_out.shape != (B, 1500, d.d_model):
        raise ValueError(f"encoder output must be [{B}, 1500, {d.d_model}], got {tuple(enc_out.shape)}")
    ids = decoder_input_ids.to(enc_out.device, torch.int32).contiguous()
    V = d.vocab
    ld = (V + 3) // 4 * 4
    buf = torch.empty((B * T, ld), dtype=torch.float32, device=enc_out.device)
    with torch.cuda.device(dev):
        ctx.check(ctx.lib.tw_decoder_logits(C.c_void_p(handle), enc_out.data_ptr(), B, ids.data_ptr(), T, buf.data_ptr(), ld,
                                            _stream_ptr(enc_out.device)))
    return buf.view(B, T, ld)[:, :, :V]


def _register_torch_ops():
    """torch.ops.twb200.{log_mel, model_create, model_free, encoder_forward, greedy_generate, decoder_logits, detect_language}: operator
    wrappers over the C ABI (CUDA tensors only, current stream).  A model is addressed by its `tw_model*` passed as an int —
    the value model_create returns — so the ops need no Python-side object (SURVEY §8b)."""
    try:
        from torch.library import custom_op
    except Exception:  # pragma: no cover
        return

    @custom_op("twb200::log_mel", mutates_args=())
    def _op_log_mel(pcm: torch.Tensor, n_valid: Optional[torch.Tensor], n_mel: int) -> torch.Tensor:
        return log_mel(pcm, n_valid, n_mel)

    @_op_log_mel.register_fake
    def _(pcm, n_valid, n_mel):
        return pcm.new_empty((pcm.shape[0], n_mel, N_FRAMES), dtype=torch.float32)

    @custom_op("twb200::model_create", mutates_args=())
    def _op_model_create(desc: Sequence[int], names: str, weights: Sequence[torch.Tensor]) -> int:
        return model_create(list(desc), names.split("\n"), list(weights))

    @custom_op("twb200::model_free", mutates_args=())
    def _op_model_free(handle: int) -> None:
        model_free(handle)

    @custom_op("twb200::encoder_forward", mutates_args=())
    def _op_encoder_forward(handle: int, mel: torch.Tensor) -> torch.Tensor:
        return encoder_forward(handle, mel)

    @_op_encoder_forward.register_fake
    def _(handle, mel):
        d = model_desc(handle)
        return mel.new_empty((mel.shape[0], 1500, d.d_model), dtype=_TW2TORCH[d.dtype])

    @custom_op("twb200::greedy_generate", mutates_args=())
    def _op_greedy_generate(handle: int, enc_out: torch.Tensor, prompt: Sequence[int], max_length: int, suppress: Sequence[int],
                            begin_suppress: Sequence[int], eos: int, pad: int, timestamp_begin: int, no_timestamps: int,
                            max_initial_ts: int) -> torch.Tensor:
        # [B, max_length - P + 1] int32: the generated ids, then the row's length in the last column
        toks, lens = greedy_decode(handle, enc_out, list(prompt), max_length, list(suppress), list(begin_suppress), eos, pad,
                                   timestamp_begin, no_timestamps, max_initial_ts)
        return torch.cat([toks, lens[:, None]], dim=1)

    @_op_greedy_generate.register_fake
    def _(handle, enc_out, prompt, max_length, suppress, begin_suppress, eos, pad, timestamp_begin, no_timestamps, max_initial_ts):
        return enc_out.new_empty((enc_out.shape[0], max_length - len(prompt) + 1), dtype=torch.int32)

    @custom_op("twb200::decoder_logits", mutates_args=())
    def _op_decoder_logits(handle: int, enc_out: torch.Tensor, decoder_input_ids: torch.Tensor) -> torch.Tensor:
        # the custom-op contract wants an owning tensor: copy the pitched view into a dense [B, T, V]
        return decoder_logits(handle, enc_out, decoder_input_ids).contiguous()

    @_op_decoder_logits.register_fake
    def _(handle, enc_out, decoder_input_ids):
        d = model_desc(handle)
        return enc_out.new_empty((decoder_input_ids.shape[0], decoder_input_ids.shape[1], d.vocab), dtype=torch.float32)

    @custom_op("twb200::detect_language", mutates_args=())
    def _op_detect_language(handle: int, enc_out: torch.Tensor, lang_ids: torch.Tensor) -> torch.Tensor:
        return detect_language(handle, enc_out, lang_ids)

    @_op_detect_language.register_fake
    def _(handle, enc_out, lang_ids):
        return enc_out.new_empty((enc_out.shape[0],), dtype=torch.int32)


# --------------------------------------------------------------------------------------------
class BatchFeature(dict):
    """Minimal stand-in for transformers.BatchFeature (dict with attribute access and .to)."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e

    def to(self, *a, **kw):
        return BatchFeature({k: (v.to(*a, **kw) if torch.is_tensor(v) else v) for k, v in self.items()})


class DeviceFeatureList(list):
    """What `fe(..., return_tensors=None)` returns as `input_features` when the extractor was built with
    `keep_on_device=True`: a list of per-clip CUDA tensors (views of one [B, n_mel, 3000] batch tensor, kept in `.batch`).
    The only thing the reference does with that list is hand it to `fe.pad(...)` (ref prefiltering/validator_inference.py:
    57-69), which returns `.batch` itself — the features never visit the host."""

    def __init__(self, batch: torch.Tensor):
        super().__init__(batch.unbind(0))
        self.batch = batch


class B200WhisperFeatureExtractor:
    """Drop-in for WhisperFeatureExtractor on the reference's call sites
    (ref: training/run_pseudo_labelling.py:739-741; prefiltering/validator_inference.py:57-69).
    The log-mel runs in the K1 CUDA kernel; `device` selects the GPU ("cuda", "cuda:1")."""

    model_input_names = ["input_features"]

    def __init__(self, feature_size: int = 80, sampling_rate: int = SAMPLING_RATE, hop_length: int = 160,
                 chunk_length: int = 30, n_fft: int = 400, padding_value: float = 0.0, device: str = "cuda",
                 keep_on_device: bool = False, **kwargs):
        if (sampling_rate, hop_length, chunk_length, n_fft) != (16000, 160, 30, 400):
            raise NotImplementedError("the B200 log-mel kernel is specialised for 16 kHz / n_fft 400 / hop 160 / 30 s")
        if feature_size not in (80, 128):
            raise ValueError("feature_size must be 80 or 128")
        self.feature_size = feature_size
        self.sampling_rate = sampling_rate
        self.hop_length = hop_length
        self.chunk_length = chunk_length
        self.n_fft = n_fft
        self.n_samples = N_SAMPLES
        self.nb_max_frames = N_FRAMES
        self.padding_value = padding_value
        self.device = device
        # return_tensors=None normally yields host numpy arrays (what `datasets.map` stores, ref run_pseudo_labelling.py:
        # 739-741); with keep_on_device the list holds CUDA views and `pad` hands the batch tensor straight to generate
        self.keep_on_device = keep_on_device

    @classmethod
    def from_hf(cls, hf_fe, device: str = "cuda"):
        return cls(feature_size=hf_fe.feature_size, sampling_rate=hf_fe.sampling_rate, hop_length=hf_fe.hop_length,
                   chunk_length=hf_fe.chunk_length, n_fft=hf_fe.n_fft, device=device)

    def __call__(self, raw_speech, sampling_rate: Optional[int] = None, return_tensors: Optional[str] = None,
                 device: Optional[str] = None, truncation: bool = True, padding: str = "max_length", **kwargs):
        if sampling_rate is not None and sampling_rate != self.sampling_rate:
            # same message shape as HF (feature_extraction_whisper.py:261-267)
            raise ValueError(
                f"The model corresponding to this feature extractor: {self.__class__.__name__} was trained using a "
                f"sampling rate of {self.sampling_rate}. Please make sure that the provided `raw_speech` input was "
                f"sampled with {self.sampling_rate} and not {sampling_rate}.")
        if kwargs.get("do_normalize") or kwargs.get("return_attention_mask") or kwargs.get("return_token_timestamps"):
            raise NotImplementedError("do_normalize / attention masks are not on the reference's call path")
        dev = device if device not in (None, "cpu") else self.device
        pcm, n_valid = self._to_device_batch(raw_speech, dev)
        feats = log_mel(pcm, n_valid, self.feature_size)
        if return_tensors == "pt":
            out = feats
        elif return_tensors is None and self.keep_on_device:
            out = DeviceFeatureList(feats)
        elif return_tensors in (None, "np"):
            arr = feats.cpu().numpy()
            out = arr if return_tensors == "np" else [a for a in arr]
        else:
            raise ValueError(f"unsupported return_tensors={return_tensors!r}")
        return BatchFeature({"input_features": out})

    def _to_device_batch(self, raw_speech, dev):
        if torch.is_tensor(raw_speech):
            t = raw_speech
            if t.dim() == 1:
                t = t[None]
            if t.dim() != 2:
                raise ValueError("Only mono-channel audio is supported for input to " + self.__class__.__name__)
            if t.dtype == torch.float64:
                t = t.float()
            if t.dtype not in (torch.int16, torch.float32):
                t = t.float()
            return t.to(dev, non_blocking=True), None
        if isinstance(raw_speech, np.ndarray) and raw_speech.ndim == 2:
            rows = list(raw_speech)
        elif isinstance(raw_speech, np.ndarray) and raw_speech.ndim > 2:
            raise ValueError("Only mono-channel audio is supported for input to " + self.__class__.__name__)
        elif isinstance(raw_speech, (list, tuple)) and len(raw_speech) and isinstance(raw_speech[0], (np.ndarray, list, tuple)):
            rows = [np.asarray(r) for r in raw_speech]
        else:
            rows = [np.asarray(raw_speech)]
        is_i16 = all(r.dtype == np.int16 for r in rows)
        n_max = min(max(len(r) for r in rows), N_SAMPLES)
        n_max = max(n_max, 8)
        buf = np.zeros((len(rows), n_max), dtype=np.int16 if is_i16 else np.float32)
        n_valid = np.zeros(len(rows), dtype=np.int32)
        for i, r in enumerate(rows):
            if r.ndim != 1:
                raise ValueError("Only mono-channel audio is supported for input to " + self.__class__.__name__)
            n = min(len(r), N_SAMPLES)          # truncation to 30 s
            buf[i, :n] = r[:n]
            n_valid[i] = n
        return torch.from_numpy(buf).to(dev), torch.from_numpy(n_valid).to(dev)

    def pad(self, processed_features, padding="longest", return_tensors: Optional[str] = None, **kwargs):
        """ref: training/run_pseudo_labelling.py:370-374, prefiltering/validator_inference.py:65-69 —
        every window is already 3000 frames long, so this only stacks."""
        feats = processed_features["input_features"] if isinstance(processed_features, dict) else \
            [f["input_features"] for f in processed_features]
        if isinstance(feats, DeviceFeatureList):
            stacked = feats.batch
        elif torch.is_tensor(feats):
            stacked = feats
        else:
            stacked = torch.stack([torch.as_tensor(f) for f in feats])
        if return_tensors in (None, "np"):
            stacked = stacked.cpu().numpy()
        elif return_tensors != "pt":
            raise ValueError(f"unsupported return_tensors={return_tensors!r}")
        return BatchFeature({"input_features": stacked})


# --------------------------------------------------------------------------------------------
def retrieve_segments(seq: np.ndarray, timestamp_begin: int, seek_num_frames: int, input_stride: int = 2):
    """Host-side restatement of WhisperGenerationMixin._retrieve_segment (generation_whisper.py:1976-2073) for one
    decoded window: split at consecutive timestamp tokens and compute by how many feature frames to advance.
    Returns (list of token arrays, segment_offset)."""
    seq = np.asarray(seq)
    ts = seq >= timestamp_begin
    single_timestamp_ending = len(seq) >= 2 and (not ts[-2]) and bool(ts[-1])
    idx = np.where(ts[:-1] & ts[1:])[0] + 1 if len(seq) >= 2 else np.zeros(0, dtype=np.int64)
    if len(idx) > 0:
        slices = idx.tolist()
        if single_timestamp_ending:
            slices.append(len(seq))
        else:
            slices[-1] += 1          # keep the last timestamp token: "it was no single ending"
        segments, last = [], 0
        for cur in slices:
            segments.append(seq[last:cur])
            last = cur
        if single_timestamp_ending:
            offset = seek_num_frames
        else:
            offset = int(seq[last - 2] - timestamp_begin) * input_stride
    else:
        segments, offset = [seq], seek_num_frames
    return segments, int(offset)


_LANG_NAMES = {"chinese": "zh", "mandarin": "zh", "english": "en", "japanese": "ja", "cantonese": "yue", "korean": "ko",
               "german": "de", "french": "fr", "spanish": "es"}


class B200WhisperForConditionalGeneration:
    """Drop-in for the `WhisperForConditionalGeneration` object the reference scripts hold, on the
    surface they touch: .eval(), .to(), .config, .generation_config, .generate(...), .module."""

    def __init__(self, hf_model, dtype=torch.bfloat16, max_batch: int = 64, device: str = "cuda",
                 output_layout: str = "4.45"):
        """output_layout: which transformers release `generate()` imitates where the releases differ (SURVEY §0.4).
        "4.45" (default; the reference pins transformers==4.45.2, ref environment.yml:175): ids start with the forced
        prompt `<|sot|><|lang|><|task|>[<|notimestamps|>]` — the layout ref run_pseudo_labelling.py:629,1009-1010
        slices with `timestamp_position` — and a <= 30 s window is decoded exactly once with return_timestamps=True.
        "5.x" (the transformers installed in this image, which pins the oracle): generated ids only, and
        return_timestamps=True runs the seek loop.  `return_prompt=` / `seek_loop=` override either per call."""
        if output_layout not in ("4.45", "5.x"):
            raise ValueError('output_layout must be "4.45" (the reference\'s pinned transformers) or "5.x"')
        self.output_layout = output_layout
        cfg = hf_model.config
        self.config = cfg
        self.generation_config = hf_model.generation_config
        self.dtype = dtype
        if dtype not in (torch.bfloat16, torch.float32):
            raise ValueError("dtype must be torch.bfloat16 (tcgen05 path) or torch.float32 (check mode)")
        self.device = torch.device(device if ":" in str(device) else f"cuda:{torch.cuda.current_device()}")
        self.ctx = _lib.Context.get(_dev_index(self.device))
        from .configs import WhisperShape
        if cfg.encoder_attention_heads != cfg.decoder_attention_heads or cfg.encoder_ffn_dim != cfg.decoder_ffn_dim:
            raise NotImplementedError("encoder/decoder widths must match (true for every Whisper checkpoint)")
        self.shape = WhisperShape("hf", cfg.num_mel_bins, cfg.d_model, cfg.encoder_ffn_dim, cfg.encoder_attention_heads,
                                  cfg.encoder_layers, cfg.decoder_layers, cfg.vocab_size, cfg.max_target_positions)
        self.max_batch = max_batch
        desc = (cfg.d_model, cfg.encoder_ffn_dim, cfg.encoder_attention_heads, cfg.encoder_layers, cfg.decoder_layers,
                cfg.num_mel_bins, cfg.vocab_size, cfg.max_target_positions, _TORCH2TW[dtype], max_batch)
        # weights snapshot (after any embedding surgery such as utils/model_utils.py:4-14) -> device; proj_out.weight is
        # tied to embed_tokens, so only the "model." tensors are passed
        sd = {k: v for k, v in hf_model.state_dict().items() if k.startswith("model.")}
        with torch.cuda.device(self.device):
            weights = [t.detach().to(self.device) for t in sd.values()]
            self.handle = model_create(desc, list(sd.keys()), weights)       # the tw_model* as an int (torch.ops take it as is)
        del weights
        self.training = False

    @classmethod
    def from_hf(cls, hf_model, dtype=torch.bfloat16, max_batch: int = 64, device: str = "cuda", output_layout: str = "4.45"):
        return cls(hf_model, dtype=dtype, max_batch=max_batch, device=device, output_layout=output_layout)

    # ---- nn.Module-ish surface the scripts touch
    def eval(self):
        return self

    def to(self, *args, **kwargs):
        return self

    @property
    def module(self):          # `model.module.generate` under DDP wrapping (ref run_pseudo_labelling.py:917)
        return self

    def parameters(self):
        return iter(())

    def close(self):
        if getattr(self, "handle", None):
            model_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def device_bytes(self) -> int:
        return int(self.ctx.lib.tw_model_bytes(C.c_void_p(self.handle)))

    # ---- generation config plumbing (generation_whisper.py:1455-1608, :1774-1812)
    def _init_tokens(self, language, task, return_timestamps):
        """The one forced prompt of a call that names a single language (or of an English-only checkpoint)."""
        if self._is_multilingual() and (language is None or isinstance(language, (list, tuple))):
            raise NotImplementedError("language=None (detection) and language lists give every row its own prompt: "
                                      "_row_prompts(language, task, return_timestamps, batch_size) builds them")
        return self._row_prompts(language, task, return_timestamps, 1)[0]

    def _is_multilingual(self):
        gc = self.generation_config
        is_multi = getattr(gc, "is_multilingual", None)
        if is_multi is None or not hasattr(gc, "lang_to_id") or not hasattr(gc, "task_to_id"):
            raise ValueError("The generation config is outdated: it needs `is_multilingual`, `lang_to_id`, `task_to_id` "
                             "and `no_timestamps_token_id` (as generation_config.json of the released checkpoints has).")
        return bool(is_multi)

    def _row_prompts(self, language, task, return_timestamps, batch_size):
        """The forced prompt of every row, as HF's _retrieve_init_tokens builds them (generation_whisper.py:1455-1608): one
        language for all rows, a list with one language per row, or language=None — detection, marked by lib.PROMPT_DETECT at
        index 1, where step 0 of the decode writes the detected id.  Detection follows HF: no task token unless `task` is given
        or `forced_decoder_ids` (generation config, else model config) force one, and a language those force is not detected."""
        gc = self.generation_config
        if not self._is_multilingual():
            if language is not None or task is not None:
                raise ValueError("Cannot specify `task` or `language` for an English-only model.")
            toks = [self.config.decoder_start_token_id]
            if not return_timestamps:
                toks.append(gc.no_timestamps_token_id)
            return [toks] * batch_size
        if isinstance(language, (list, tuple)):
            if any(l is None for l in language):
                raise TypeError(
                    "Expected `language` to be `None`, a single string (e.g. `'en'`), or a list of strings with "
                    "length equal to the batch size (e.g. `('en', 'fr')` for a batch size of 2). Got a list "
                    "containing `None`.")
            if len(language) != batch_size:
                raise ValueError(
                    "When passing a list of languages, the length of the list must match the batch size. "
                    f"Expected length of {batch_size}, but got {len(language)} languages.")
            return [self._lang_prompt(l, task, return_timestamps) for l in language]
        if language is not None:
            return [self._lang_prompt(language, task, return_timestamps)] * batch_size
        return [self._detect_prompt(task, return_timestamps)] * batch_size

    def _detect_prompt(self, task, return_timestamps):
        """_retrieve_init_tokens with language=None (generation_whisper.py:1484-1606), the language slot left to detection."""
        gc = self.generation_config
        toks = [self.config.decoder_start_token_id]
        if task is None:
            forced = getattr(gc, "forced_decoder_ids", None)
            if forced is None:
                forced = getattr(self.config, "forced_decoder_ids", None)
            if forced is not None and forced[0][0] == 1:
                i = 1
                while len(forced) > 0 and forced[0][0] == i:
                    toks.append(forced[0][1])
                    forced = forced[1:]
                    i += 1
                if len(forced) > 0:
                    raise ValueError(
                        f"You are using token ids in `forced_decoder_ids` that do not seem to correctly follow "
                        f"the prompt pattern of Whisper. Make sure that {forced} has an entry for all "
                        f"indices >= 1 and < {forced[0][0]}.")
        if len(toks) <= 1:
            toks.append(_lib.PROMPT_DETECT)
        elif toks[1] is None:
            toks[1] = _lib.PROMPT_DETECT
        if task is not None:
            if task not in gc.task_to_id:
                raise ValueError(f"The `{task}` task is not supported. The task should be one of `{list(gc.task_to_id)}`")
            toks.append(gc.task_to_id[task])
        if not return_timestamps and toks[-1] != gc.no_timestamps_token_id:
            toks.append(gc.no_timestamps_token_id)
        elif return_timestamps and toks[-1] == gc.no_timestamps_token_id:
            toks = toks[:-1]
        return [t for t in toks if t is not None]

    def _lang_prompt(self, language, task, return_timestamps):
        """One prompt with a given language (a code, "<|code|>" or a name); the task defaults to transcribe."""
        gc = self.generation_config
        toks = [self.config.decoder_start_token_id]
        lang = str(language).lower()
        if lang in gc.lang_to_id:
            lang_tok = lang
        elif f"<|{lang}|>" in gc.lang_to_id:
            lang_tok = f"<|{lang}|>"
        elif lang in _LANG_NAMES and f"<|{_LANG_NAMES[lang]}|>" in gc.lang_to_id:
            lang_tok = f"<|{_LANG_NAMES[lang]}|>"
        else:
            raise ValueError(f"Unsupported language: {language}. Language should be one of: "
                             f"{sorted(gc.lang_to_id.keys())[:8]}...")
        toks.append(gc.lang_to_id[lang_tok])
        t = "transcribe" if task is None else task
        if t not in gc.task_to_id:
            raise ValueError(f"The `{t}` task is not supported. The task should be one of `{list(gc.task_to_id)}`")
        toks.append(gc.task_to_id[t])
        if not return_timestamps:
            toks.append(gc.no_timestamps_token_id)
        return toks

    def _lang_ids(self):
        """The ids language detection chooses among: the values of generation_config.lang_to_id."""
        return sorted(int(v) for v in self.generation_config.lang_to_id.values())

    @staticmethod
    def _resolved(prompts, langs):
        """prompts with every detection slot replaced by the row's decoded language (langs: int sequence [B])."""
        return [[int(langs[b]) if (i == 1 and t == _lib.PROMPT_DETECT) else t for i, t in enumerate(p)] for b, p in enumerate(prompts)]

    def _rules(self, return_timestamps):
        gc = self.generation_config
        eos = gc.eos_token_id if not isinstance(gc.eos_token_id, (list, tuple)) else gc.eos_token_id[0]
        pad = gc.pad_token_id if gc.pad_token_id is not None else eos
        return dict(suppress=list(getattr(gc, "suppress_tokens", None) or []),
                    begin_suppress=list(getattr(gc, "begin_suppress_tokens", None) or []),
                    eos=int(eos), pad=int(pad),
                    timestamp_begin=(gc.no_timestamps_token_id + 1) if return_timestamps else None,
                    no_timestamps=int(gc.no_timestamps_token_id),
                    max_initial_ts=getattr(gc, "max_initial_timestamp_index", None))

    # ---- device-level entry points
    def encode(self, mel: torch.Tensor, tap_layer: int = -1):
        """mel [B, n_mel, 3000] float32 -> enc_out [B,1500,d] (model dtype, on the model's device); with tap_layer >= 0 also
        returns the fp32 residual stream after that many layers."""
        return encoder_forward(self.handle, torch.as_tensor(mel).to(self.device), tap_layer)

    def decode(self, enc_out: torch.Tensor, prompt, max_length: int, timestamps: bool, forced: Optional[torch.Tensor] = None,
               tap_steps: int = 0):
        r = self._rules(timestamps)
        return greedy_decode(self.handle, enc_out.to(self.device), list(prompt), max_length, r["suppress"], r["begin_suppress"],
                             r["eos"], r["pad"], -1 if r["timestamp_begin"] is None else r["timestamp_begin"], r["no_timestamps"],
                             -1 if r["max_initial_ts"] is None else r["max_initial_ts"], forced=forced, tap_steps=tap_steps)

    def decode_rows(self, enc_out: torch.Tensor, prompts, max_length: int, timestamps: bool):
        """decode with one prompt per row (_row_prompts): returns (tokens, lengths, languages int32 [B]), the languages detected
        in step 0 for rows whose prompt asks for it, the given ones elsewhere."""
        r = self._rules(timestamps)
        return greedy_decode_rows(self.handle, enc_out.to(self.device), prompts, self._lang_ids(), max_length, r["suppress"],
                                  r["begin_suppress"], r["eos"], r["pad"], -1 if r["timestamp_begin"] is None else r["timestamp_begin"],
                                  r["no_timestamps"], -1 if r["max_initial_ts"] is None else r["max_initial_ts"])

    @torch.no_grad()
    def detect_language(self, input_features=None, encoder_outputs=None, generation_config=None, num_segment_frames: int = N_FRAMES):
        """WhisperGenerationMixin.detect_language (generation_whisper.py:1610-1673): LongTensor [B] of language ids, from log-mel
        input_features [B, n_mel, >= 3000] (the first 3000 frames) or encoder_outputs ([B, 1500, d], a tuple or an object with
        last_hidden_state).  Step 0 of a decode fed <|startoftranscript|>, its logits masked to lang_to_id, argmax."""
        if input_features is None and encoder_outputs is None:
            raise ValueError("You have to specify either `input_features` or `encoder_outputs`")
        elif input_features is not None and encoder_outputs is not None:
            raise ValueError("Make sure to specify only one of `input_features` or `encoder_outputs` - not both!")
        lang_ids = self._lang_ids()
        if input_features is not None:
            feats = torch.as_tensor(input_features)[:, :, :num_segment_frames]
            encs = [self.encode(feats[s:s + self.max_batch].to(self.device).float()) for s in range(0, feats.shape[0], self.max_batch)]
        else:
            enc = encoder_outputs[0] if isinstance(encoder_outputs, (tuple, list)) else getattr(encoder_outputs, "last_hidden_state",
                                                                                                 encoder_outputs)
            enc = torch.as_tensor(enc).to(self.device)
            encs = [enc[s:s + self.max_batch] for s in range(0, enc.shape[0], self.max_batch)]
        return torch.cat([detect_language(self.handle, e, lang_ids) for e in encs]).long()

    def decoder_logits(self, enc_out: torch.Tensor, decoder_input_ids: torch.Tensor) -> torch.Tensor:
        """enc_out [B,1500,d] + decoder_input_ids [B,T] -> fp32 logits [B,T,V] of every position in ONE batched decoder pass."""
        return decoder_logits(self.handle, enc_out.to(self.device), decoder_input_ids)

    def shift_tokens_right(self, labels: torch.Tensor) -> torch.Tensor:
        """HF shift_tokens_right (modeling_whisper.py:67-81): prepend decoder_start_token_id, drop the last label, -100 -> pad."""
        start = int(self.config.decoder_start_token_id)
        pad = int(self.config.pad_token_id)
        shifted = labels.new_zeros(labels.shape)
        shifted[:, 1:] = labels[:, :-1].clone()
        shifted[:, 0] = start
        shifted.masked_fill_(shifted == -100, pad)
        return shifted

    @torch.no_grad()
    def forward(self, input_features=None, *, encoder_outputs=None, decoder_input_ids=None, labels=None, **kwargs):
        """The teacher call of the distillation step (ref knowledge-distillation/run_distillation.py:1543-1577):
        `teacher_model(**batch)` with input_features / labels / decoder_input_ids, or
        `teacher_model(encoder_outputs=BaseModelOutput(h), labels=labels)` when the frozen encoder is shared.
        Returns an object with `.logits` [B,T,V] (fp32) and `.encoder_last_hidden_state`; no loss (the reference never
        reads the teacher's)."""
        from types import SimpleNamespace
        for k, v in kwargs.items():
            if v is not None and k not in ("attention_mask", "decoder_attention_mask", "return_dict", "use_cache"):
                raise NotImplementedError(f"forward(): argument {k!r} is not supported by the B200 teacher path")
        if kwargs.get("decoder_attention_mask") is not None:
            raise NotImplementedError("forward(): decoder_attention_mask is not supported (the reference passes none)")
        if encoder_outputs is not None:
            enc = encoder_outputs[0] if isinstance(encoder_outputs, (tuple, list)) else getattr(encoder_outputs, "last_hidden_state", encoder_outputs)
        elif input_features is not None:
            feats = input_features if torch.is_tensor(input_features) else torch.as_tensor(np.asarray(input_features))
            enc = self.encode(feats.float())
        else:
            raise ValueError("You have to specify either input_features or encoder_outputs")
        if decoder_input_ids is None:
            if labels is None:
                raise ValueError("You have to specify either decoder_input_ids or labels")
            decoder_input_ids = self.shift_tokens_right(labels if torch.is_tensor(labels) else torch.as_tensor(labels))
        logits = self.decoder_logits(enc, decoder_input_ids)
        return SimpleNamespace(logits=logits, encoder_last_hidden_state=enc, loss=None)

    __call__ = forward

    def transcribe_pcm(self, pcm_host: torch.Tensor, max_length: int, return_timestamps: bool = False, language="zh",
                       task="transcribe", n_valid: Optional[torch.Tensor] = None, out_tokens: Optional[torch.Tensor] = None,
                       out_lengths: Optional[torch.Tensor] = None, return_languages: bool = False):
        """Whole path from HOST int16 PCM [B, 480000] (pinned for async copies) to HOST token ids:
        one C-ABI call = fe(...) + generate(...) of the reference.  `language`: one for every row, a list with one per row, or
        None — each row's language is detected in the decode's first step.  return_languages: also return the host int32 [B]
        language ids the rows were decoded with."""
        if pcm_host.dtype != torch.int16 or pcm_host.dim() != 2 or pcm_host.shape[1] != N_SAMPLES or pcm_host.is_cuda:
            raise ValueError("transcribe_pcm expects a host int16 tensor [B, 480000]")
        pcm_host = pcm_host.contiguous()
        B = pcm_host.shape[0]
        if B > self.max_batch:
            raise ValueError(f"batch {B} > max_batch {self.max_batch}")
        prompts = self._row_prompts(language, task, return_timestamps, B)
        n_gen = max_length - len(prompts[0])
        if n_gen <= 0 or max_length > self.shape.max_target:
            raise ValueError("max_length must exceed the prompt and fit max_target_positions")
        if out_tokens is None:
            out_tokens = torch.empty((B, n_gen), dtype=torch.int32).pin_memory()
            out_lengths = torch.empty((B,), dtype=torch.int32).pin_memory()
        r = self._rules(return_timestamps)
        rules, keep = _lib.make_rules(r["suppress"], r["begin_suppress"], r["eos"], r["pad"], r["timestamp_begin"],
                                      r["no_timestamps"], r["max_initial_ts"])
        rows, keep_rows, langs = self._prompt_rows(prompts, return_languages)
        nv = n_valid.contiguous().data_ptr() if n_valid is not None else None
        with torch.cuda.device(self.device):
            self.ctx.check(self.ctx.lib.tw_transcribe_host_rows(
                C.c_void_p(self.handle), pcm_host.data_ptr(), nv, B, C.byref(rows), len(prompts[0]), C.byref(rules), max_length,
                out_tokens.data_ptr(), out_lengths.data_ptr(), _stream_ptr(self.device)))
        del keep, keep_rows
        return (out_tokens, out_lengths, langs) if return_languages else (out_tokens, out_lengths)

    def _prompt_rows(self, prompts, want_languages: bool):
        """(PromptRows, keepalive, host int32 [B] language buffer or None) for the host-output entry points: the language ids go
        along when a row detects, the language buffer when a row detects or the caller wants the languages."""
        detect = any(len(p) > 1 and p[1] == _lib.PROMPT_DETECT for p in prompts)
        langs = torch.empty((len(prompts),), dtype=torch.int32) if (detect or want_languages) else None
        rows, keep, _ = _lib.make_prompt_rows(prompts, self._lang_ids() if detect else None,
                                              langs.data_ptr() if langs is not None else None)
        return rows, keep, langs

    # ------------------------------------------------------------------ pipelined batch loop (tw_pipeline_*)
    def enable_pipeline(self, n_enc_sms: int = 24):
        """Splits the GPU into two SM partitions (CUDA green contexts): `n_enc_sms` SMs for the front end + encoder + cross-K/V
        of the NEXT batch, the rest for the greedy decode of the current one (`transcribe_batches`).  Returns (encoder SMs,
        decode SMs) as the driver granted them (multiples of 8).  Calling it again moves the boundary (tw_pipeline_resize).
        Raises NotImplementedError when the driver has no green contexts."""
        with torch.cuda.device(self.device):
            if getattr(self, "pipeline_sms", None):
                self.ctx.check(self.ctx.lib.tw_pipeline_resize(C.c_void_p(self.handle), int(n_enc_sms)))
            else:
                self.ctx.check(self.ctx.lib.tw_pipeline_enable(C.c_void_p(self.handle), int(n_enc_sms)))
        a, b = C.c_int(0), C.c_int(0)
        self.ctx.check(self.ctx.lib.tw_pipeline_info(C.c_void_p(self.handle), C.byref(a), C.byref(b)))
        self.pipeline_sms = (a.value, b.value)
        return self.pipeline_sms

    def pipeline_stage_ms(self, slot: int):
        """(stage-1 ms, decode ms) of the slot's last group, each measured in its partition while the other stage runs; -1 for a
        stage that has not completed.  Never blocks."""
        a, b = C.c_float(-1), C.c_float(-1)
        self.ctx.check(self.ctx.lib.tw_pipeline_stage_ms(C.c_void_p(self.handle), int(slot), C.byref(a), C.byref(b)))
        return float(a.value), float(b.value)

    @staticmethod
    def _balanced_sms(n_enc: int, n_dev: int, t_enc: float, t_dec: float) -> int:
        """Encoder-partition size for the next groups from the measured stage times of the last one.  Stage 1 scales ~1 / SMs;
        the decode is HBM-bound and loses little from a smaller partition, so the rule only asks that stage 1 finishes a little
        before the decode does (target 0.92 of its time) and leaves a wide dead band (0.75 .. 1.02) against oscillation."""
        if t_enc <= 0 or t_dec <= 0:
            return n_enc
        ratio = t_enc / t_dec
        want = n_enc
        if ratio > 1.02 or ratio < 0.75:
            want = int(-(-n_enc * ratio / 0.92 // 8) * 8)          # rounded up to the partition granularity
        return max(16, min(want, (n_dev // 2) // 8 * 8))

    def transcribe_batches(self, batches, max_length: int, return_timestamps: bool = False, language="zh", task="transcribe",
                           merge: int = 1, auto_sms: bool = False, return_languages: bool = False):
        """The reference's batch loop (ref training/run_pseudo_labelling.py:915-918) as a generator: yields (tokens, lengths) — pinned
        host int32 tensors [B, max_length - P] / [B] — for every int16 PCM batch [B, 480000] of `batches` (pinned host or device
        tensors), in order.  While batch i decodes, batch i+1 is already in its log-mel / encoder / cross-K/V stage on the other SM
        partition (`enable_pipeline` first).

        `merge` > 1 decodes that many consecutive batches TOGETHER (tw_pipeline_encode_at): each is encoded on its own — the
        encoder is compute-bound, its cost follows the clip count — into consecutive rows of one slot, and one greedy decode runs
        over all rows.  A decode step streams the decoder weights and runs its chain of small dependent kernels once whatever
        the row count, so merged batches pay them once; per row nothing changes (same kernels, same arithmetic per row: ids equal
        the unmerged loop's up to the bf16 rounding of a different K|V row split).  The model needs max_batch >= the merged rows;
        results are still yielded per input batch.

        `auto_sms=True` re-balances the two partitions while the loop runs: after every group the stage times of the last one
        (tw_pipeline_stage_ms) are compared and the encoder partition is resized when stage 1 has become the bottleneck or idles
        more than a quarter of the time (`_balanced_sms`).  Full-length rows keep the decode busy ~7x longer than stage 1 needs the
        GPU; rows that end early (real audio) shift the balance towards stage 1 — the right split depends on the data.

        `language`: one language (or None: every row's is detected in the decode's first step) for all rows, or a list with one
        entry per batch of `batches` — a language, None or a list with one language per row of that batch.  Merged groups mix rows
        of different languages freely.  return_languages: yield (tokens, lengths, languages), languages the host int32 [B] ids
        the rows were decoded with."""
        if not getattr(self, "pipeline_sms", None):
            raise RuntimeError("transcribe_batches needs enable_pipeline() first")
        if merge < 1:
            raise ValueError("merge must be >= 1")
        per_batch = isinstance(language, (list, tuple))

        def batch_prompts(k, n):
            lang = (language[k] if k < len(language) else None) if per_batch else language
            return self._row_prompts(lang, task, return_timestamps, n)

        r = self._rules(return_timestamps)
        rules, keep = _lib.make_rules(r["suppress"], r["begin_suppress"], r["eos"], r["pad"], r["timestamp_begin"],
                                      r["no_timestamps"], r["max_initial_ts"])
        lib, h = self.ctx.lib, C.c_void_p(self.handle)
        it = enumerate(batches)
        pending = []                 # a batch that did not fit the current group

        def encode_group(slot):
            """Stage 1 of the next `merge` batches (fewer at the end of the loop, or when the next batch would not fit max_batch)
            into `slot`; returns the row count of each and keeps the PCM tensors alive until their decode has returned."""
            sizes, alive, prompts = [], [], []
            while len(sizes) < merge:
                kp = pending.pop() if pending else next(it, None)
                if kp is None:
                    break
                k, pcm = kp
                if pcm.dtype != torch.int16 or pcm.dim() != 2 or pcm.shape[1] != N_SAMPLES or pcm.shape[0] > self.max_batch or pcm.shape[0] == 0:
                    raise ValueError("transcribe_batches expects int16 tensors [1 <= B <= max_batch, 480000]")
                if sum(sizes) + pcm.shape[0] > self.max_batch:
                    pending.append(kp)                 # opens the next group
                    break
                pcm = pcm.contiguous()
                prompts += batch_prompts(k, pcm.shape[0])
                self.ctx.check(lib.tw_pipeline_encode_at(h, pcm.data_ptr(), None, pcm.shape[0], slot, sum(sizes)))
                sizes.append(pcm.shape[0])
                alive.append(pcm)
            return (sizes, alive, prompts) if sizes else None

        with torch.cuda.device(self.device):
            cur = encode_group(0)
            i = 0
            while cur is not None:
                nxt = encode_group((i + 1) & 1)
                B = sum(cur[0])
                P = len(cur[2][0])
                n_gen = max_length - P
                if n_gen <= 0 or max_length > self.shape.max_target:
                    raise ValueError("max_length must exceed the prompt and fit max_target_positions")
                out_tokens = torch.empty((B, n_gen), dtype=torch.int32).pin_memory()
                out_lengths = torch.empty((B,), dtype=torch.int32).pin_memory()
                rows, keep_rows, langs = self._prompt_rows(cur[2], return_languages)
                self.ctx.check(lib.tw_pipeline_decode_rows(h, i & 1, B, C.byref(rows), P, C.byref(rules), max_length,
                                                           out_tokens.data_ptr(), out_lengths.data_ptr()))
                del keep_rows
                if auto_sms and nxt is not None and sum(nxt[0]) == B:
                    # stage 1 of the NEXT group ran beside this decode: both times are of the same concurrent interval
                    t_enc, _ = self.pipeline_stage_ms((i + 1) & 1)
                    _, t_dec = self.pipeline_stage_ms(i & 1)
                    if t_enc > 0 and t_dec > 0:          # (stage 1 still running: it is the bottleneck by at least this much)
                        want = self._balanced_sms(self.pipeline_sms[0], sum(self.pipeline_sms), t_enc, t_dec)
                    elif t_dec > 0:
                        want = self._balanced_sms(self.pipeline_sms[0], sum(self.pipeline_sms), 1.25 * t_dec, t_dec)
                    else:
                        want = self.pipeline_sms[0]
                    if want != self.pipeline_sms[0]:
                        self.enable_pipeline(want)
                        self.sms_history = getattr(self, "sms_history", []) + [self.pipeline_sms]
                b0 = 0
                for n in cur[0]:
                    if return_languages:
                        yield out_tokens[b0:b0 + n], out_lengths[b0:b0 + n], langs[b0:b0 + n]
                    else:
                        yield out_tokens[b0:b0 + n], out_lengths[b0:b0 + n]
                    b0 += n
                cur = nxt
                i += 1
        del keep

    def set_row_budgets(self, budgets: Optional[Sequence[int]]):
        """Test / bench hook (tw_debug_set_row_budgets): row b of the following decode calls finishes after budgets[b]
        generated tokens exactly as if it had emitted EOS next; None switches it off.  Random-init weights never emit EOS,
        so this is how the finished-row path (pad emission, lengths, active-clip list, early exit) runs at benched shapes."""
        if budgets is None:
            self.ctx.check(self.ctx.lib.tw_debug_set_row_budgets(C.c_void_p(self.handle), None, 0))
            return
        arr = (C.c_int32 * len(budgets))(*[int(b) for b in budgets])
        self.ctx.check(self.ctx.lib.tw_debug_set_row_budgets(C.c_void_p(self.handle), arr, len(budgets)))

    def profile(self, enable: bool):
        """Reads + resets the in-situ samples of the dominant kernel, then (de)activates sampling.
        Returns (total_ms, launches); `last_profile_bytes` holds the K|V bytes of one sampled launch (one sub-batch
        of the batch when the decode step is split)."""
        ms, n, nb = C.c_float(0), C.c_int(0), C.c_double(0)
        self.ctx.check(self.ctx.lib.tw_profile(C.c_void_p(self.handle), 1 if enable else 0, C.byref(ms), C.byref(n), C.byref(nb)))
        self.last_profile_bytes = float(nb.value)
        return float(ms.value), int(n.value)

    def last_stage_ms(self):
        buf = (C.c_float * 6)()
        self.ctx.lib.tw_last_stage_ms(C.c_void_p(self.handle), buf)
        return dict(zip(("logmel", "encoder", "cross_kv", "decode", "total", "h2d"), [float(x) for x in buf]))

    # ---- the reference's call
    @torch.no_grad()
    def generate(self, input_features=None, *, max_length: Optional[int] = None, max_new_tokens: Optional[int] = None,
                 num_beams: int = 1, return_timestamps: Optional[bool] = None, language=None,
                 task: Optional[str] = None, attention_mask=None, return_prompt: Optional[bool] = None,
                 seek_loop: Optional[bool] = None, **kwargs):
        """ref: training/run_pseudo_labelling.py:864-876,917-918; prefiltering/validator_inference.py:41-47,78.
        Returns a LongTensor [B, L], EOS stripped, right-padded with pad_token_id to the batch maximum; one 30 s window
        per row.  `return_prompt` (default: True under output_layout "4.45", False under "5.x"): whether the forced prompt
        leads every row — the reference's `add_concatenated_text` (ref :1003-1012) drops `timestamp_position` = 3 leading
        ids and therefore needs it.  `seek_loop` (default: False under "4.45", True under "5.x"): with
        return_timestamps=True, run the 5.x seek loop around the window primitive — split at consecutive timestamp
        tokens, advance to the last predicted timestamp, re-encode the zero-padded remainder (generation_whisper.py:
        785-900, 1976-2073) — or decode each window exactly once (short-form behaviour of 4.45).
        `language`: one language for every row, a list with one per row, or None on a multilingual checkpoint — each row's
        language is detected (detect_language) in the first step of its decode, with HF's prompts (_row_prompts); the seek loop
        detects on a window's first pass and keeps that language for the rest of the window."""
        if return_prompt is None:
            return_prompt = self.output_layout == "4.45"
        if seek_loop is None:
            seek_loop = self.output_layout == "5.x"
        if num_beams not in (None, 1):
            raise NotImplementedError("twb200 implements greedy decoding only (num_beams=1), as the reference's "
                                      "pseudo-labelling launchers use")
        for k in ("do_sample", "prompt_ids", "assistant_model", "temperature", "logits_processor"):
            if kwargs.get(k):
                raise NotImplementedError(f"generate(..., {k}=...) is not on the reference's path")
        if input_features is None:
            raise ValueError("input_features is required")
        feats = torch.as_tensor(input_features)
        if feats.dim() != 3:
            raise ValueError("input_features must be [batch, n_mel, 3000]")
        if feats.shape[-1] != N_FRAMES:
            raise ValueError(f"Whisper expects the mel input features to be of length {N_FRAMES}, but found "
                             f"{feats.shape[-1]}. Make sure to pad the input mel features to {N_FRAMES}.")
        ts = bool(return_timestamps) if return_timestamps is not None else False
        prompts = self._row_prompts(language, task, ts, feats.shape[0])
        if max_length is None:
            if max_new_tokens is not None:
                max_length = len(prompts[0]) + max_new_tokens
            else:
                max_length = getattr(self.generation_config, "max_length", None) or self.shape.max_target
        if max_length > self.shape.max_target:
            raise ValueError(f"max_length={max_length} exceeds max_target_positions={self.shape.max_target}")
        pad = self._rules(ts)["pad"]
        if ts and seek_loop:
            return self._generate_seek_loop(feats, prompts, max_length, pad, return_prompt)
        rows, lens_all, langs = [], [], []
        for s in range(0, feats.shape[0], self.max_batch):
            chunk = feats[s:s + self.max_batch]
            enc = self.encode(chunk.to(self.device).float())
            toks, lens, lg = self.decode_rows(enc, prompts[s:s + self.max_batch], max_length, ts)
            rows.append(toks)
            lens_all.append(lens)
            langs += lg.tolist()
        toks = torch.cat(rows).long()
        lens = torch.cat(lens_all).long()
        L = int(lens.max().item()) if lens.numel() else 0
        toks = toks[:, :L]
        ar = torch.arange(L, device=toks.device)[None, :]
        toks = torch.where(ar < lens[:, None], toks, torch.full_like(toks, pad))
        if return_prompt:
            toks = torch.cat([torch.tensor(self._resolved(prompts, langs), device=toks.device, dtype=toks.dtype), toks], dim=1)
        return toks if feats.is_cuda else toks.cpu()

    def _generate_seek_loop(self, feats, prompts, max_length, pad, return_prompt):
        tsb = self.generation_config.no_timestamps_token_id + 1
        B = feats.shape[0]
        x = feats.to(self.device).float()
        seek = [0] * B
        segs = [[] for _ in range(B)]
        prompts = list(prompts)       # a row's detection slot is resolved on its first pass; the remainders reuse that prompt
        while any(s < N_FRAMES for s in seek):
            active = [i for i in range(B) if seek[i] < N_FRAMES]
            nframes = [min(N_FRAMES - seek[i], N_FRAMES) for i in active]
            chunk = torch.zeros((len(active), x.shape[1], N_FRAMES), dtype=torch.float32, device=self.device)
            for j, i in enumerate(active):
                chunk[j, :, :nframes[j]] = x[i, :, seek[i]:seek[i] + nframes[j]]
            toks_l, lens_l = [], []
            for s0 in range(0, len(active), self.max_batch):
                enc = self.encode(chunk[s0:s0 + self.max_batch])
                rows = active[s0:s0 + self.max_batch]
                t, l, lg = self.decode_rows(enc, [prompts[i] for i in rows], max_length, True)
                for i, p in zip(rows, self._resolved([prompts[i] for i in rows], lg.tolist())):
                    prompts[i] = p
                toks_l.append(t)
                lens_l.append(l)
            toks = torch.cat(toks_l).cpu().numpy()
            lens = torch.cat(lens_l).cpu().numpy()
            for j, i in enumerate(active):
                pieces, offset = retrieve_segments(toks[j, :lens[j]], tsb, nframes[j])
                if offset <= 0:                 # HF would spin here (zero-length segment); always make progress
                    offset = nframes[j]
                segs[i].extend(pieces)
                seek[i] += offset
        rows = [np.concatenate(sg) if sg else np.zeros(0, np.int64) for sg in segs]
        L = max((len(r) for r in rows), default=0)
        out = torch.full((B, L), pad, dtype=torch.long)
        for i, r in enumerate(rows):
            out[i, :len(r)] = torch.from_numpy(r.astype(np.int64))
        if return_prompt:
            out = torch.cat([torch.tensor(prompts, dtype=out.dtype), out], dim=1)
        return out.to(feats.device) if feats.is_cuda else out

    # forward() (training) is out of scope


_register_torch_ops()
