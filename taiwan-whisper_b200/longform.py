"""Chunked long-form front end (SURVEY §8f-2): cut a long recording into 30 s windows with a stride on each side
and compute their log-mel features on the GPU *without materialising the windows* — window b is row b of a
strided view of the recording (row pitch = chunk - stride_left - stride_right samples), which is exactly the
`pcm_stride` / `n_valid` interface of tw_logmel.

Window placement and the (chunk_len, stride_left, stride_right) bookkeeping restate
ref: training/flax/distil_whisper/pipeline.py:224-254 (chunk_iter_with_batch) and :325-335 (stride = chunk/6).
`stitch_windows` merges the per-window token streams of overlapping windows the way `tokenizer._decode_asr` does for
the no-timestamp case (ref :353-375 -> HF tokenization_whisper.py `_find_longest_common_sequence`);
`stitch_windows_timestamps` is the `return_timestamps=True` branch of the same function (what the reference's validator /
pseudo-labelling runs use): a state machine over the windows' tokens that opens / closes chunks at timestamp tokens, ignores
timestamps inside the strides, shifts times by the windows' offsets and resolves the overlapping text by the same longest-
common-sequence merge.  Both work on token ids; ids -> text stays with the tokenizer (third-party vocabulary data).
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import numpy as np
import torch

from . import lib as _lib
from .configs import N_FRAMES, N_SAMPLES, SAMPLING_RATE


def chunk_plan(n_samples: int, chunk_len: int = N_SAMPLES, stride_left: Optional[int] = None,
               stride_right: Optional[int] = None) -> Tuple[np.ndarray, List[Tuple[int, int, int]]]:
    """Window start indices and per-window (chunk_len_actual, stride_left, stride_right)."""
    if stride_left is None:
        stride_left = round(chunk_len / 6)
    if stride_right is None:
        stride_right = stride_left
    if chunk_len < stride_left + stride_right:
        raise ValueError("Chunk length must be superior to stride length")
    step = chunk_len - stride_left - stride_right
    starts = np.arange(0, n_samples, step)
    ends = starts + chunk_len
    sl = np.where(starts == 0, 0, stride_left)
    is_last = np.where(stride_right > 0, ends > n_samples, ends >= n_samples)
    sr = np.where(is_last, 0, stride_right)
    lens = np.minimum(ends, n_samples) - starts
    return starts, [(int(l), int(a), int(b)) for l, a, b in zip(lens, sl, sr)]


def chunked_log_mel(pcm: torch.Tensor, n_mel: int, chunk_len: int = N_SAMPLES, stride_left: Optional[int] = None,
                    stride_right: Optional[int] = None):
    """pcm: 1-D int16 / float32 CUDA tensor (one recording, 16 kHz).  Returns (features [n_windows, n_mel, 3000] f32,
    strides list) — the `{"stride": ..., "input_features": ...}` items the reference's chunker yields."""
    if pcm.dim() != 1 or not pcm.is_cuda or pcm.dtype not in (torch.int16, torch.float32):
        raise ValueError("chunked_log_mel expects a 1-D int16/float32 CUDA tensor")
    if chunk_len != N_SAMPLES:
        raise NotImplementedError("the log-mel kernel is specialised for 30 s windows")
    starts, strides = chunk_plan(pcm.shape[0], chunk_len, stride_left, stride_right)
    n = len(starts)
    step = int(starts[1] - starts[0]) if n > 1 else chunk_len
    dev = pcm.device.index if pcm.device.index is not None else torch.cuda.current_device()
    ctx = _lib.Context.get(dev)
    pcm = pcm.contiguous()
    out = torch.empty((n, n_mel, N_FRAMES), dtype=torch.float32, device=pcm.device)
    n_valid = torch.tensor([s[0] for s in strides], dtype=torch.int32, device=pcm.device)
    dt = _lib.TW_I16 if pcm.dtype == torch.int16 else _lib.TW_F32
    with torch.cuda.device(dev):
        # row b of the "batch" starts at sample b*step of the recording: zero-copy windowing
        ctx.check(ctx.lib.tw_logmel(ctx.handle, pcm.data_ptr(), dt, step, n_valid.data_ptr(), n, n_mel, out.data_ptr(),
                                    torch.cuda.current_stream(pcm.device).cuda_stream))
    return out, strides


def stitch_windows(sequences: List[List[int]]) -> List[int]:
    """Merge the token streams of consecutive overlapping windows into one stream (no-timestamp mode).

    Restates HF `_find_longest_common_sequence` (tokenization_whisper.py; called by `_decode_asr`, which
    ref: training/flax/distil_whisper/pipeline.py:353-375 calls): for each next window slide it over the tail of what
    has been kept so far; an alignment of overlap length i scores (#equal tokens) / i + i / 10000 (the epsilon prefers
    longer overlaps) and needs at least two equal tokens; at the best alignment keep the left stream up to the middle of
    the overlap and continue with the right stream from the middle of its side of the overlap."""
    if not sequences:
        return []
    left = list(sequences[0])
    total: List[int] = []
    for right in sequences[1:]:
        right = list(right)
        n_l, n_r = len(left), len(right)
        best, best_idx = 0.0, (n_l, n_l, 0, 0)
        la, ra = np.asarray(left, dtype=np.int64), np.asarray(right, dtype=np.int64)
        for i in range(1, n_l + n_r):
            l0, l1 = max(0, n_l - i), min(n_l, n_l + n_r - i)
            r0, r1 = max(0, i - n_l), min(n_r, i)
            matches = int(np.sum(la[l0:l1] == ra[r0:r1]))
            score = matches / i + i / 10000.0
            if matches > 1 and score > best:
                best, best_idx = score, (l0, l1, r0, r1)
        l0, l1, r0, r1 = best_idx
        total.extend(left[:(l0 + l1) // 2])
        left = right[(r0 + r1) // 2:]
    total.extend(left)
    return total


def stitch_windows_timestamps(outputs, timestamp_begin: int, special_ids=(), time_precision: float = 0.02,
                              segment_size: int = 1500, prompt_token_id: Optional[int] = None,
                              decoder_start_token_id: Optional[int] = None):
    """Timestamp-aware stitching of the windows of one long recording: the `return_timestamps=True` path of HF
    `_decode_asr` (tokenization_whisper.py:901-1150; called by ref training/flax/distil_whisper/pipeline.py:353-375),
    restated on token ids.

    outputs: one dict per window, in order: {"tokens": ids of the window (generated ids; a leading `<|startofprev|>` prompt
    is stripped as HF does), "stride": (chunk_len_s, stride_left_s, stride_right_s) in SECONDS (ref :357-366) or absent}.
    special_ids: ids that are neither text nor timestamps (`tokenizer.all_special_ids`: sot, language, task, notimestamps,
    eos ...) — skipped.  Returns a list of chunks {"timestamp": (start_s | None, end_s | None), "tokens": [ids]}; text is
    `tokenizer.decode(chunk["tokens"])`.  A last chunk without an end timestamp mirrors HF's "did not predict an ending
    timestamp" case."""
    special = set(int(t) for t in special_ids)
    chunks = []
    chunk = {"timestamp": [None, None], "tokens": []}
    time_offset = 0.0
    previous_tokens: List[List[int]] = []
    skip = False
    right_stride_start = None
    for output in outputs:
        token_ids = [int(t) for t in output["tokens"]]
        if token_ids and prompt_token_id is not None and token_ids[0] == prompt_token_id:      # _strip_prompt
            token_ids = token_ids[token_ids.index(decoder_start_token_id):] if decoder_start_token_id in token_ids else []
        last_timestamp = None
        first_timestamp = timestamp_begin
        cur_max_timestamp = 0.0
        prev_segments_len = 0.0
        penultimate_timestamp = 0.0
        stride = output.get("stride")
        if stride is not None:
            chunk_len, stride_left, stride_right = stride
            time_offset -= stride_left
            right_stride_start = chunk_len - stride_right
            if stride_left:
                first_timestamp = stride_left / time_precision + timestamp_begin
            if stride_right:
                for token in reversed(token_ids):
                    if token >= timestamp_begin:
                        # several timestamps may fall in the right stride; the last one is always skipped
                        if last_timestamp is not None and (token - timestamp_begin) * time_precision < right_stride_start:
                            break
                        last_timestamp = token
        current_tokens: List[int] = []
        for i, token in enumerate(token_ids):
            if token in special:
                continue
            if token >= timestamp_begin:
                timestamp = float((token - timestamp_begin) * time_precision)
                if timestamp < cur_max_timestamp:
                    # a new 30 s segment of a long-form generate() started inside this window's ids
                    last_was_single_ending = i >= 2 and not (token_ids[i - 1] >= timestamp_begin and token_ids[i - 2] >= timestamp_begin)
                    if last_was_single_ending:
                        prev_segments_len += time_precision * segment_size
                    else:
                        cur_max_timestamp = penultimate_timestamp
                        prev_segments_len += penultimate_timestamp
                penultimate_timestamp = cur_max_timestamp
                cur_max_timestamp = timestamp
                time = round((token - timestamp_begin) * time_precision + time_offset + prev_segments_len, 2)
                if last_timestamp and token >= last_timestamp:
                    skip = True                      # inside the right stride: resolved with the next window
                elif skip or (previous_tokens and token < first_timestamp):
                    skip = False
                elif chunk["timestamp"][0] is None:
                    chunk["timestamp"][0] = time
                elif time == chunk["timestamp"][0]:
                    pass                             # duplicated start token: stays a start
                else:
                    chunk["timestamp"][1] = time
                    previous_tokens.append(current_tokens)
                    chunk["tokens"] = stitch_windows(previous_tokens)
                    chunks.append(chunk)
                    previous_tokens = []
                    current_tokens = []
                    chunk = {"timestamp": [None, None], "tokens": []}
            else:
                current_tokens.append(token)
        if stride is not None:
            time_offset += chunk_len - stride_right
        if current_tokens:
            previous_tokens.append(current_tokens)
        elif not any(p for p in previous_tokens):
            chunk = {"timestamp": [None, None], "tokens": []}
            previous_tokens = []
    if previous_tokens:
        chunk["tokens"] = stitch_windows(previous_tokens)
        chunks.append(chunk)
    for c in chunks:
        c["timestamp"] = tuple(c["timestamp"])
    return chunks


def transcribe_longform(model, pcm: torch.Tensor, *, language: Optional[str] = "zh", task: str = "transcribe", max_length: int = 448,
                        return_timestamps: bool = True, batch_size: Optional[int] = None, chunk_len: int = N_SAMPLES,
                        stride_left: Optional[int] = None, stride_right: Optional[int] = None, special_ids=(), merge: int = 1):
    """Config 5 end to end for one recording (1-D int16 / float32 CUDA tensor): zero-copy windowing + log-mel
    (`chunked_log_mel`), batched one-pass greedy decode of the windows (`model.generate`), and stitching — timestamp-aware
    chunks when return_timestamps, else the merged id stream.  Mirrors ref training/flax/distil_whisper/pipeline.py:
    256-375 (preprocess_batch -> forward -> postprocess) with the windows batched `batch_size` (<= model.max_batch) at a
    time.  `merge` > 1 sends the windows through the encoder `batch_size` at a time and decodes `merge` such batches together
    (as many as fit model.max_batch): a decode step streams the decoder weights and runs its chain of small kernels once whatever
    the row count (bench.py --workload longform: 561 -> 1088 audio-s/s with 5 x 32 windows per decode); per window nothing changes.
    language=None detects the language of every window on its own (in the first step of its decode), as HF does per chunk."""
    feats, strides = chunked_log_mel(pcm, model.shape.n_mel, chunk_len, stride_left, stride_right)
    bs = min(int(batch_size or model.max_batch), model.max_batch)
    gc = model.generation_config
    eos = int(gc.eos_token_id if not isinstance(gc.eos_token_id, (list, tuple)) else gc.eos_token_id[0])
    pad = int(gc.pad_token_id) if getattr(gc, "pad_token_id", None) is not None else eos
    rows: List[List[int]] = []
    G = max(1, min(int(merge), model.max_batch // bs))
    if G > 1:
        for g0 in range(0, feats.shape[0], bs * G):
            encs = [model.encode(feats[b0:b0 + bs]) for b0 in range(g0, min(g0 + bs * G, feats.shape[0]), bs)]
            enc = encs[0] if len(encs) == 1 else torch.cat(encs)
            prompts = model._row_prompts(language, task, return_timestamps, enc.shape[0])
            toks, lens, _ = model.decode_rows(enc, prompts, max_length, return_timestamps)
            toks, lens = toks.cpu().numpy(), lens.cpu().numpy()
            for r, n in zip(toks, lens):
                r = r[:int(n)].tolist()
                while r and r[-1] == pad:
                    r.pop()
                rows.append(r)
    for b0 in range(0, feats.shape[0] if G == 1 else 0, bs):
        ids = model.generate(feats[b0:b0 + bs], max_length=max_length, num_beams=1, return_timestamps=return_timestamps,
                             language=language, task=task, seek_loop=False, return_prompt=False).cpu().numpy()
        for r in ids:
            r = r.tolist()
            while r and r[-1] == pad:
                r.pop()
            rows.append(r)
    if not return_timestamps:
        return stitch_windows(rows)
    tsb = int(gc.no_timestamps_token_id) + 1
    outs = [{"tokens": r, "stride": (s[0] / SAMPLING_RATE, s[1] / SAMPLING_RATE, s[2] / SAMPLING_RATE)} for r, s in zip(rows, strides)]
    sp = set(special_ids) | {eos, int(gc.no_timestamps_token_id)}
    return stitch_windows_timestamps(outs, tsb, sp)
