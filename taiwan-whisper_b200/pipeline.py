"""First-pass long-audio transcription on the B200 path (SURVEY §8f-3): the object
`pseudo-labelling/initial_inference.py` holds as `pipeline` (faster-whisper's `BatchedInferencePipeline`,
ref: pseudo-labelling/initial_inference.py:33-54,84-90) re-pointed at the CUDA path, and the CSV wire format its
consumer reads (`start,end,text`, ref: pseudo-labelling/prepare_dataset.py:37-53).

Differences from the reference engine, stated because parity with CTranslate2 cannot be pinned here (SURVEY §8c):
  * chunking is by fixed windows of `chunk_length` seconds (each zero-padded to 30 s on the device through the
    log-mel kernel's row pitch / n_valid interface — no window is materialised), not by the Silero VAD model;
  * decoding is the greedy timestamp mode of this package (`generate(..., return_timestamps=True)`), one window per row;
  * token ids -> text needs a tokenizer, which is third-party data (vocabulary files): pass `tokenizer` (anything with
    `.decode(ids)`) or `decode_fn`.
"""
from __future__ import annotations

import csv
from typing import Callable, Iterable, List, NamedTuple, Optional, Sequence

import numpy as np
import torch

from . import lib as _lib
from .configs import N_FRAMES, N_SAMPLES, SAMPLING_RATE

TIME_PRECISION = 0.02          # seconds per timestamp token (<|0.00|> ... <|30.00|>)


class Segment(NamedTuple):
    start: float
    end: float
    text: str
    tokens: List[int]


class TranscriptionInfo(NamedTuple):
    language: Optional[str]      # None: every window's language was detected on its own
    duration: float
    n_windows: int


def segments_from_tokens(tokens: Sequence[int], timestamp_begin: int, eos: int, window_start_s: float, window_len_s: float,
                         pad: Optional[int] = None, length: Optional[int] = None):
    """Split one decoded window at its timestamp tokens: `<|t0|> text <|t1|>` is one segment; a second timestamp right
    after a closing one opens the next segment; text without a closing timestamp runs to the end of the window.
    Ids >= eos that are not timestamps (special tokens) never reach the text.  `generate()` right-pads the rows of a batch
    with pad_token_id, which is a *text-range* id when pad != eos (50256 in large-v3's config.json): pass the row's
    `length`, or `pad` to drop the trailing padding, so that it is neither appended as text nor opens a segment.
    Returns [(start_s, end_s, [ids])]."""
    tokens = [int(t) for t in tokens]
    if length is not None:
        tokens = tokens[:int(length)]
    elif pad is not None:
        n = len(tokens)
        while n > 0 and tokens[n - 1] == pad:
            n -= 1
        tokens = tokens[:n]
    out = []
    start = None
    cur: List[int] = []
    for t in tokens:
        if t >= timestamp_begin:
            ts = min((t - timestamp_begin) * TIME_PRECISION, window_len_s)
            if cur:                                   # closes the running segment
                out.append((window_start_s + (start if start is not None else 0.0), window_start_s + ts, cur))
                cur, start = [], None
            else:
                start = ts                            # opens (or re-opens) a segment
        elif t < eos:
            cur.append(t)
    if cur:
        out.append((window_start_s + (start if start is not None else 0.0), window_start_s + window_len_s, cur))
    return out


def save_transcription_to_csv(transcriptions: Iterable, output_csv: str):
    """The reference's writer (ref: pseudo-labelling/initial_inference.py:47-54): header `start,end,text`, times as
    `%.2f` strings — what `read_pseudo_labels` (ref: pseudo-labelling/prepare_dataset.py:37-53) parses."""
    with open(output_csv, "w", newline="", encoding="utf-8") as f:
        writer = csv.DictWriter(f, fieldnames=["start", "end", "text"])
        writer.writeheader()
        for item in transcriptions:
            if isinstance(item, Segment):
                item = {"start": f"{item.start:.2f}", "end": f"{item.end:.2f}", "text": item.text}
            writer.writerow(item)


class B200BatchedInferencePipeline:
    """`pipeline.transcribe(audio=..., task="transcribe", log_progress=..., batch_size=...) -> (segments, info)` with
    `segment.start / .end / .text`, as the reference calls it (ref: pseudo-labelling/initial_inference.py:36-45).
    language=None (here and in transcribe) detects the language of every window on its own, as HF does per chunk."""

    def __init__(self, model, tokenizer=None, decode_fn: Optional[Callable[[List[int]], str]] = None, chunk_length: int = 30,
                 language: Optional[str] = "zh", use_vad_model: bool = False, max_length: int = 448):
        if use_vad_model:
            raise NotImplementedError("the Silero VAD model is third-party; this pipeline chunks by fixed windows")
        if not (1 <= chunk_length <= 30):
            raise ValueError("chunk_length must be in 1..30 seconds")
        if decode_fn is None and tokenizer is not None:
            decode_fn = lambda ids: tokenizer.decode(ids)        # noqa: E731
        self.model = model
        self.decode_fn = decode_fn
        self.chunk_samples = int(chunk_length) * SAMPLING_RATE
        self.chunk_length = float(chunk_length)
        self.language = language
        self.max_length = max_length

    # ---- audio -> device PCM
    @staticmethod
    def _load(audio) -> np.ndarray:
        if isinstance(audio, str):
            try:
                import soundfile as sf
            except ImportError as e:          # pragma: no cover - depends on the image
                raise RuntimeError("reading audio files needs the `soundfile` package; pass a 16 kHz numpy array instead") from e
            x, sr = sf.read(audio, dtype="float32", always_2d=True)
            if sr != SAMPLING_RATE:
                raise ValueError(f"expected {SAMPLING_RATE} Hz audio, got {sr} Hz (resample upstream)")
            return x.mean(axis=1)
        x = np.asarray(audio)
        if x.ndim != 1:
            raise ValueError("audio must be a path or a 1-D array of 16 kHz samples")
        return x

    def window_features(self, pcm: torch.Tensor) -> torch.Tensor:
        """1-D int16 / float32 CUDA tensor -> log-mel [n_windows, n_mel, 3000] of consecutive chunk_length windows, each
        zero-padded to 30 s: window b is row b of a strided view of the recording (pitch = chunk samples)."""
        n = pcm.shape[0]
        n_win = max(1, -(-n // self.chunk_samples))
        dev = pcm.device.index if pcm.device.index is not None else torch.cuda.current_device()
        ctx = _lib.Context.get(dev)
        n_mel = self.model.shape.n_mel
        out = torch.empty((n_win, n_mel, N_FRAMES), dtype=torch.float32, device=pcm.device)
        n_valid = torch.tensor([min(self.chunk_samples, max(0, n - b * self.chunk_samples)) for b in range(n_win)],
                               dtype=torch.int32, device=pcm.device)
        dt = _lib.TW_I16 if pcm.dtype == torch.int16 else _lib.TW_F32
        with torch.cuda.device(dev):
            ctx.check(ctx.lib.tw_logmel(ctx.handle, pcm.data_ptr(), dt, self.chunk_samples, n_valid.data_ptr(), n_win, n_mel,
                                        out.data_ptr(), torch.cuda.current_stream(pcm.device).cuda_stream))
        return out

    # ---- the reference's call
    def transcribe(self, audio, task: str = "transcribe", log_progress: bool = False, batch_size: int = 64, language: Optional[str] = None):
        x = self._load(audio)
        if x.dtype != np.int16:
            x = x.astype(np.float32)
        pcm = torch.from_numpy(np.ascontiguousarray(x)).to(self.model.device)
        feats = self.window_features(pcm)
        n_win = feats.shape[0]
        bs = max(1, min(int(batch_size), self.model.max_batch))
        gc = self.model.generation_config
        tsb = int(gc.no_timestamps_token_id) + 1
        eos = int(gc.eos_token_id if not isinstance(gc.eos_token_id, (list, tuple)) else gc.eos_token_id[0])
        pad = int(gc.pad_token_id) if getattr(gc, "pad_token_id", None) is not None else eos
        segments: List[Segment] = []
        for b0 in range(0, n_win, bs):
            ids = self.model.generate(feats[b0:b0 + bs], max_length=self.max_length, num_beams=1, return_timestamps=True,
                                      language=language or self.language, task=task, seek_loop=False, return_prompt=False)
            ids = ids.cpu().numpy()
            for j in range(ids.shape[0]):
                w = b0 + j
                w_len = min(self.chunk_length, max(0.0, len(x) / SAMPLING_RATE - w * self.chunk_length))
                for s, e, toks in segments_from_tokens(ids[j], tsb, eos, w * self.chunk_length, w_len, pad=pad):
                    text = self.decode_fn(toks) if self.decode_fn is not None else " ".join(str(t) for t in toks)
                    segments.append(Segment(s, e, text, toks))
            if log_progress:
                print(f"[twb200] windows {min(b0 + bs, n_win)}/{n_win}", flush=True)
        info = TranscriptionInfo(language or self.language, len(x) / SAMPLING_RATE, n_win)
        return iter(segments), info
