#!/usr/bin/env python
"""bench.py — RTFx (audio-seconds per second) of whisper-large-v3 pseudo-labelling on N B200.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [...]                          # the reference's own CPU path (HF)
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N    # one rank per GPU

A "step" = one batch (BASELINE.json configs[1]: whisper-large-v3, bf16, 64 synthetic 30 s clips per GPU,
greedy zh/transcribe, max_length 256 => 252 generated tokens per clip; random-init weights never emit EOS)
through the whole hot path: log-mel -> encoder -> cross-K/V -> KV-cached greedy decode.
  value   inputs (int16 PCM) already resident in HBM, tokens left in HBM, CUDA-event timed
  e2e     the same through the public host API `transcribe_pcm` (one C-ABI call, tw_transcribe_host):
          pinned HOST PCM in, HOST token ids out, copies inside the timed region
Multi-GPU: the utterance manifest is sharded (rank r owns clips [r*n, (r+1)*n)); no collective on the
data path; one final all_gather of the token rows (inside the timed region); weak scaling.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MODEL = "large-v3"
BATCH = 64
MAX_LENGTH = 256           # ref: training/run-pseudo-labelling.sh:33
CLIP_SECONDS = 30.0
POOL_CLIPS = 64            # distinct synthetic clips per rank (a manifest maps ids onto the pool)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default=MODEL)
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--max-length", type=int, default=MAX_LENGTH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity block (fp32 check model + HF bf16 comparator)")
    ap.add_argument("--no-hf-cuda", action="store_true", help="skip the same-box HF bf16/SDPA generate comparator")
    ap.add_argument("--no-ragged", action="store_true", help="skip the ragged-length variant (finished rows leave the K|V stream)")
    ap.add_argument("--no-pipeline", action="store_true",
                    help="headline = the sequential batch loop (default: stage 1 of batch i+1 overlaps the decode of batch i on SM partitions)")
    ap.add_argument("--pipeline-sms", type=int, default=0, help="SMs of the front-end / encoder partition of the pipeline (0 = 16 unmerged, 24 merged)")
    ap.add_argument("--merge", type=int, default=3,
                    help="batches of the reference loop decoded together by the pipelined loop (transcribe_batches merge=): a pipelined step "
                         "is `merge` x `batch` clips; 1 = one batch per decode")
    ap.add_argument("--workload", default="clips", choices=["clips", "longform"],
                    help="clips: BASELINE configs[1] (default); longform: configs[4] — long recordings cut into 30 s windows "
                         "(hop 20 s, stride 5 s each side), timestamp mode, windows batched, timestamp-aware stitching")
    ap.add_argument("--longform-merge", type=int, default=5,
                    help="--workload longform: encoder batches of `batch` windows decoded together (one greedy decode over batch x merge rows)")
    ap.add_argument("--recordings", type=int, default=10)
    ap.add_argument("--recording-seconds", type=int, default=600)
    ap.add_argument("--ref-clips", type=int, default=0, help="--impl reference: clips per step (0 = sized from K + W)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path returned in its last step (token ids and lengths of "
                         "rank 0) as DIR/<name>.npy, float32; inputs and weights are seeded, so two builds compare output for output")
    return ap.parse_args()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT_BYTES):
    """Writes `arrays` (name -> array, one row per clip or window) as <out_dir>/<name>.npy in float32, which holds every token
    id and length exactly.  When the files would exceed `limit` bytes in all, the same fixed seeded sample of rows is kept in
    every array and the row indices are written as rows.npy (float64)."""
    import numpy as np
    arrays = {k: np.asarray(v, dtype=np.float32) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a.nbytes for a in arrays.values()) // max(n, 1)
    budget = limit - 4096           # room for the .npy headers
    if n * row_bytes > budget:
        rows = np.sort(np.random.default_rng(0).choice(n, size=budget // (row_bytes + 8), replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1590.0, "fallback"


def sustained_tflops():
    """cuBLAS bf16 throughput held back to back for seconds (MEASURED_PEAKS.json) — the denominator that applies to a
    stage timed inside a long step; the burst figure (`peaks()`) applies to a kernel timed alone."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("bf16_tflops_sustained")
    return None


NCU_TRAFFIC_CSV = {64: "r02_decode_attention_stream_raw.csv", 128: "r02_decode_attention_stream_b128_raw.csv",
                   192: "r02_decode_attention_stream_b192_raw.csv"}


def workload_text(model, B, max_length, n_gen):
    """The workload both arms name (BASELINE.json configs[1] at the defaults); each arm appends what one of ITS steps covers."""
    return (f"whisper-{model} pseudo-labelling: batches of {B} x 30 s 16 kHz clips per GPU, log-mel + encoder + cross-K/V + greedy "
            f"decode, zh/transcribe, max_length {max_length} ({n_gen} generated tokens/clip)")


def ncu_traffic_bytes(rows=64):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of the same shape
    (profiles/r02_decode_attention_stream[_b128]_raw.csv: dram__bytes_read.sum + dram__bytes_write.sum)."""
    import csv
    p = os.path.join(ROOT, "profiles", NCU_TRAFFIC_CSV.get(rows, "missing"))
    try:
        rows = list(csv.reader(open(p)))
        hdr, units, data = rows[0], rows[1], rows[2:]
        tot = []
        for r in data:
            b = 0.0
            for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                i = hdr.index(name)
                scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[units[i]]
                b += float(r[i]) * scale
            tot.append(b)
        return sum(tot) / len(tot) if tot else None
    except Exception:
        return None


def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path (HF feature extractor + generate, fp32, all host
    threads) on a bounded sample of the workload: each step = 1 clip of the batch, full token budget."""
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to every rank; once torch has started its OpenMP pool under that setting,
    # torch.set_num_threads() no longer widens it (measured: 10x slower matmul).  This arm is the reference on ALL host
    # cores, and only rank 0 works, so lift the cap before torch is imported.
    for var in ("OMP_NUM_THREADS", "MKL_NUM_THREADS"):
        if os.environ.get(var) == "1":
            os.environ[var] = str(os.cpu_count() or 1)
    import numpy as np
    import torch
    from oracle import hf_ref
    from taiwan_whisper_b200.configs import SHAPES
    from taiwan_whisper_b200.synth import dequantise, synth_batch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sh = SHAPES[args.model]
    model = hf_ref.build_hf_model(sh, seed=1234)
    fe = hf_ref.build_hf_feature_extractor(sh.n_mel)
    # a real batch per step (at batch 1 the decoder GEMMs are weight-bandwidth-bound GEMVs, which flatters any ratio taken
    # against this arm), bounded so that the K + W steps end within minutes on the host cores
    n_steps = args.steps + args.warmup
    clips_per_step = args.ref_clips if args.ref_clips > 0 else (8 if n_steps <= 6 else (4 if n_steps <= 12 else 2))
    pcm = dequantise(synth_batch(0, clips_per_step * n_steps))

    def step(i):
        x = pcm[i * clips_per_step:(i + 1) * clips_per_step]
        feats = hf_ref.hf_features(fe, x)
        return hf_ref.hf_generate(model, feats, args.max_length, return_timestamps=False)

    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        ids = step(args.warmup + i)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"tokens": ids})
    v = clips_per_step * args.steps * CLIP_SECONDS / dt
    sample = (f"{clips_per_step} clips per step (one HF batch) of the {args.batch}-clip batch, full max_length={args.max_length}, "
              f"fp32, {cores} threads")
    print(json.dumps({
        "impl": "reference", "metric": "rtfx_audio_seconds_per_second", "value": v, "unit": "audio-s/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(args.model, args.batch, args.max_length, args.max_length - 4)
                               + f"; a step = a bounded sample of {clips_per_step} clips (one HF batch on the host CPU)",
                   "batch_per_gpu": args.batch, "clips_per_step": clips_per_step, "max_length": args.max_length,
                   "weights": "random-init (HF init, seed 1234)", "sample": sample,
                   "reference": "transformers WhisperFeatureExtractor + WhisperForConditionalGeneration.generate on host CPU"},
        "cpu_baseline": {"value": v, "unit": "audio-s/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": v, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def cpu_baseline(args, hf_cpu, n_clips=2):
    """Reference (HF) on the box's host cores: one batch of `n_clips` clips, full token budget (~15-30 s of CPU work).
    Returns (cpu_baseline dict, features [n,n_mel,3000] f32, HF fp32 ids [n, n_gen]) — the ids pin bench parity."""
    import torch
    from oracle import hf_ref
    from taiwan_whisper_b200.configs import SHAPES
    from taiwan_whisper_b200.synth import dequantise, synth_batch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sh = SHAPES[args.model]
    fe = hf_ref.build_hf_feature_extractor(sh.n_mel)
    x = dequantise(synth_batch(0, n_clips))
    t0 = time.perf_counter()
    feats = hf_ref.hf_features(fe, x)
    ids = hf_ref.hf_generate(hf_cpu, feats, args.max_length, return_timestamps=False)
    dt = time.perf_counter() - t0
    return ({"value": n_clips * CLIP_SECONDS / dt, "unit": "audio-s/s", "cores": cores, "kind": "reference",
             "sample": f"{n_clips} of the {args.batch} clips as one HF batch, full max_length={args.max_length}, HF transformers fp32 "
                       f"generate + feature extractor, {dt:.1f} s"}, feats, ids)


def parity_block(args, hf_cpu, model, feats, hf_ids, dev):
    """Parity ON the benched configuration (VERDICT r1 #1), for the clips the CPU leg decoded with HF fp32:
      fp32_identical   a full-depth fp32 check-mode instance of this library reproduces HF's ids bit for bit
      bf16_tf_agree    the benched bf16 model, teacher-forced with HF's ids, picks the same token (all positions)
      hf_bf16_tf_agree HF's own bf16 forward on this GPU, same positions — the yardstick for bf16_tf_agree"""
    import numpy as np
    import torch
    from oracle import hf_ref
    from taiwan_whisper_b200.host import B200WhisperForConditionalGeneration
    from tests.helpers import default_rules
    sh_vocab = model.shape.vocab
    prompt = model._init_tokens("zh", "transcribe", False)
    n, n_gen = hf_ids.shape
    out = {"n_clips": int(n), "n": int(n * n_gen), "against": "HF transformers fp32 generate on the host CPU, same clips and weights"}
    ft = torch.from_numpy(feats).to(dev)
    # fp32 check mode (CUDA-core kernels), full depth, free-running
    chk = B200WhisperForConditionalGeneration.from_hf(hf_cpu, dtype=torch.float32, max_batch=int(n), device=str(dev), output_layout="5.x")
    try:
        enc = chk.encode(ft)
        toks, lens = chk.decode(enc, prompt, args.max_length, False)
        toks = toks.cpu().numpy()[:, :n_gen]
        same = toks == hf_ids
        out["fp32_identical"] = bool(same.all())
        out["fp32_first_divergence"] = [int(np.argmin(r)) if not r.all() else None for r in same]
        ftoks, _ = chk.decode(enc, prompt, args.max_length, False, forced=torch.from_numpy(hf_ids.astype(np.int32)))
        out["fp32_tf_agree"] = int((ftoks.cpu().numpy()[:, :n_gen] == hf_ids).sum())
    finally:
        chk.close()
    # the benched bf16 instance, teacher-forced on the same ids
    enc = model.encode(ft)
    btoks, _ = model.decode(enc, prompt, args.max_length, False, forced=torch.from_numpy(hf_ids.astype(np.int32)))
    out["bf16_tf_agree"] = int((btoks.cpu().numpy()[:, :n_gen] == hf_ids).sum())
    hf_b = hf_ref.hf_teacher_forced_argmax(hf_cpu, feats, prompt, hf_ids, default_rules(sh_vocab, False), device=str(dev),
                                           dtype=torch.bfloat16)
    out["hf_bf16_tf_agree"] = int((hf_b == hf_ids).sum())
    out["bf16_tf_frac"] = out["bf16_tf_agree"] / out["n"]
    out["hf_bf16_tf_frac"] = out["hf_bf16_tf_agree"] / out["n"]
    return out


def hf_cuda_comparator(args, hf_cpu, host_batch, dev):
    """Same-box GPU comparator (SURVEY §2.2: "the library path PyTorch would pick"): the UNMODIFIED HF model in bf16 with
    SDPA attention, `generate` at the benched batch / max_length on this B200, features precomputed (the reference computes
    them in CPU dataloader workers).  One warm-up call, one timed call."""
    import copy
    import torch
    from oracle import hf_ref
    from taiwan_whisper_b200.host import log_mel
    m = copy.deepcopy(hf_cpu)
    try:
        m.set_attn_implementation("sdpa")
    except Exception:
        m.config._attn_implementation = "sdpa"
    m = m.to(device=dev, dtype=torch.bfloat16).eval()
    feats = log_mel(host_batch.to(dev), None, m.config.num_mel_bins).to(torch.bfloat16)     # input features only; not timed
    B = feats.shape[0]
    with torch.no_grad():
        m.generate(feats[:4], max_length=16, num_beams=1, return_timestamps=False, language="zh", task="transcribe")
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ids = m.generate(feats, max_length=args.max_length, num_beams=1, return_timestamps=False, language="zh", task="transcribe")
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    del m
    torch.cuda.empty_cache()
    return {"hf_cuda_rtfx": B * CLIP_SECONDS / dt, "hf_cuda_s_per_batch": dt, "hf_cuda_tokens": int(ids.shape[1]),
            "hf_cuda_config": f"transformers {__import__('transformers').__version__} WhisperForConditionalGeneration.generate, bf16, "
                              f"attn_implementation=sdpa, batch {B}, max_length {args.max_length}, features precomputed, 1 timed call"}


def run_longform(args, rank, world, local_rank):
    """BASELINE configs[4]: whisper-medium validator inference on long-form audio chunked into 30 s windows, batch 32
    (ref prefiltering/validator_inference.py:41-47 gen_kwargs: max_length 448, return_timestamps=True, zh/transcribe; chunking
    and stitching of ref training/flax/distil_whisper/pipeline.py:224-254,353-375).  A step = every recording once:
    zero-copy windowing + log-mel on the device, windows of all recordings batched `--batch` at a time through encoder +
    timestamp-mode greedy decode, token rows to the host, timestamp-aware stitching on the host.
      value  PCM resident in HBM, tokens left in HBM, no stitching (device work only)
      e2e    pinned HOST PCM in, stitched chunks out (H2D, D2H and the host stitching inside the timed region)"""
    import numpy as np
    import torch
    import torch.distributed as dist
    from taiwan_whisper_b200.configs import SHAPES, SAMPLING_RATE
    from taiwan_whisper_b200.hf_compat import build_hf_model
    from taiwan_whisper_b200.host import B200WhisperForConditionalGeneration
    from taiwan_whisper_b200.longform import chunked_log_mel, stitch_windows_timestamps
    from taiwan_whisper_b200.synth import synth_batch

    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    model_name = args.model if args.model != MODEL else "medium"
    sh = SHAPES[model_name]
    B = args.batch if args.batch != BATCH else 32
    max_length = args.max_length if args.max_length != MAX_LENGTH else 448
    K, W = args.steps, args.warmup
    with torch.device(dev):
        hf = build_hf_model(sh, seed=1234)
    G = max(1, args.longform_merge)          # encoder batches per decode (merged decode, as transcribe_batches(merge=) does for clips)
    model = B200WhisperForConditionalGeneration.from_hf(hf, dtype=torch.bfloat16, max_batch=B * G, device=str(dev), output_layout="5.x")
    del hf
    torch.cuda.empty_cache()
    n_rec, rec_s = args.recordings, args.recording_seconds
    clips_per_rec = -(-rec_s // 30)
    recs_host = []
    for r in range(n_rec):          # each rank owns its own recordings (manifest shard)
        x = synth_batch((rank * n_rec + r) * clips_per_rec, clips_per_rec).reshape(-1)[: rec_s * SAMPLING_RATE]
        recs_host.append(torch.from_numpy(np.ascontiguousarray(x)).pin_memory())
    recs_dev = [x.to(dev) for x in recs_host]
    prompt = model._init_tokens("zh", "transcribe", True)
    gc = model.generation_config
    tsb = int(gc.no_timestamps_token_id) + 1
    special = {int(gc.eos_token_id), int(gc.no_timestamps_token_id)}

    def windows(pcm_list):
        feats, strides = [], []
        for x in pcm_list:
            f, s = chunked_log_mel(x, sh.n_mel)
            feats.append(f)
            strides.append(s)
        return torch.cat(feats), strides

    def decode_all(feats):
        # windows go through the encoder `B` at a time (the reference pipeline's batch); G encoder batches are decoded together: a
        # decode step streams the decoder weights and runs its chain of small kernels once whatever the row count
        toks, lens = [], []
        for g0 in range(0, feats.shape[0], B * G):
            encs = [model.encode(feats[b0:b0 + B]) for b0 in range(g0, min(g0 + B * G, feats.shape[0]), B)]
            enc = encs[0] if len(encs) == 1 else torch.cat(encs)
            del encs
            t, l = model.decode(enc, prompt, max_length, True)
            toks.append(t)
            lens.append(l)
        return torch.cat(toks), torch.cat(lens)

    def stitch(toks, lens, strides):
        toks, lens = toks.cpu().numpy(), lens.cpu().numpy()
        out, w = [], 0
        for s in strides:
            outs = [{"tokens": toks[w + i, :lens[w + i]].tolist(),
                     "stride": (st[0] / SAMPLING_RATE, st[1] / SAMPLING_RATE, st[2] / SAMPLING_RATE)} for i, st in enumerate(s)]
            out.append(stitch_windows_timestamps(outs, tsb, special))
            w += len(s)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n_windows = None
    for _ in range(W):
        f, st = windows(recs_dev)
        n_windows = f.shape[0]
        decode_all(f)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = model.ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        f, st = windows(recs_dev)
        last = decode_all(f)
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"tokens": last[0].cpu(), "lengths": last[1].cpu()})
    ms = e0.elapsed_time(e1)
    launches = model.ctx.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    prof_ms, prof_n, prof_rows = 0.0, 0, 0
    if rank == 0:
        model.profile(True)
        f, st = windows(recs_dev[:max(1, -(-B * G // clips_per_rec))])
        prof_rows = min(B * G, f.shape[0])          # one merged decode at the row count of the timed loop
        decode_all(f[:prof_rows])
        torch.cuda.synchronize()
        prof_ms, prof_n = model.profile(False)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    audio_s = world * K * n_rec * rec_s
    value = audio_s / (float(t.item()) / 1000.0)
    # e2e: host PCM -> stitched chunks
    barrier()
    e0.record()
    n_chunks = 0
    for _ in range(K):
        f, st = windows([x.to(dev, non_blocking=True) for x in recs_host])
        toks, lens = decode_all(f)
        n_chunks += sum(len(c) for c in stitch(toks, lens, st))
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    if rank == 0:
        hbm, tf, which = peaks()
        n_gen = max_length - len(prompt)
        bytes_per_launch = prof_rows * 1500 * 2 * sh.d_model * 2
        roof = None
        if prof_n > 0:
            ach = bytes_per_launch / (prof_ms / prof_n / 1000.0) / 1e9
            roof = {"kernel": "decode_attention_stream (cross-attention K/V streaming, 1 launch per layer per token)", "bound": "hbm",
                    "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm, "peak_source": which, "traffic": None,
                    "launches_timed": prof_n, "avg_launch_us": 1000.0 * prof_ms / prof_n, "algorithmic_bytes_per_launch": bytes_per_launch}
        print(json.dumps({
            "metric": "rtfx_audio_seconds_per_second", "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": float(ms) / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": f"whisper-{model_name} validator inference on long-form audio: {n_rec} x {rec_s} s recordings per GPU per "
                                   f"step, 30 s windows hop 20 s (stride 5 s each side) = {n_windows} windows, encoder batches of {B}, "
                                   f"{G} of them ({B * G} rows) per greedy decode, timestamps on, "
                                   f"max_length {max_length} ({n_gen} generated tokens/window), timestamp-aware stitching",
                       "batch_per_gpu": B, "decode_rows": B * G, "max_length": max_length, "weights": "random-init (HF init, seed 1234)",
                       "parallelism": f"recordings sharded over {world} GPU(s), no data-path collective",
                       "l2": "inputs larger than L2: every decode step streams > 4 GB of K/V and weights"},
            "clocks": clocks, "gpu_launches": int(launches), "roofline": roof,
            "e2e": {"value": audio_s / (e2e_ms / 1000.0), "unit": "audio-s/s", "ms_per_step": e2e_ms / K,
                    "h2d_bytes_per_step": int(sum(x.numel() * 2 for x in recs_host)),
                    "d2h_bytes_per_step": int(n_windows * (n_gen + 1) * 4), "stitched_chunks_per_step": n_chunks // max(K, 1),
                    "api": "chunked_log_mel + generate-equivalent encode/decode + stitch_windows_timestamps (longform.transcribe_longform)"},
        }))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    import faulthandler
    import signal
    faulthandler.register(signal.SIGUSR1, all_threads=True)      # `kill -USR1` prints where a stuck run is (Python frames) and carries on
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.workload == "longform":
        run_longform(args, rank, world, local_rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from taiwan_whisper_b200.configs import SHAPES
    from taiwan_whisper_b200.hf_compat import build_hf_model
    from taiwan_whisper_b200.host import B200WhisperForConditionalGeneration, log_mel
    from taiwan_whisper_b200.synth import synth_batch

    assert torch.cuda.is_available(), "bench.py needs a B200 (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    sh = SHAPES[args.model]
    B, K, W = args.batch, args.steps, args.warmup
    G = 1 if args.no_pipeline else max(1, args.merge)      # batches per merged decode of the pipelined loop

    # random-init weights of the architecture (HF init), built directly on the GPU
    with torch.device(dev):
        hf = build_hf_model(sh, seed=1234)
    model = B200WhisperForConditionalGeneration.from_hf(hf, dtype=torch.bfloat16, max_batch=B * G, device=str(dev), output_layout="5.x")
    hf_cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:      # the CPU baseline is reported at N=1 only
        hf_cpu = hf.to("cpu")
    del hf
    torch.cuda.empty_cache()

    # manifest shard of this rank: clip ids [rank*n, (rank+1)*n) mapped onto a pool of distinct synthetic clips
    pool = torch.from_numpy(synth_batch(rank * POOL_CLIPS, POOL_CLIPS)).pin_memory()
    n_steps_total = min(W + K, 8)               # distinct host batches (the loops below cycle through them)

    def batch_host(i):
        idx = [(i * B + j) % POOL_CLIPS for j in range(B)]
        return pool[idx].pin_memory() if idx != list(range(B)) else pool[:B]

    host_batches = [batch_host(i) for i in range(n_steps_total)]
    dev_batches = [hb.to(dev) for hb in host_batches[:2]]           # resident inputs (alternate)
    prompt = model._init_tokens("zh", "transcribe", False)
    n_gen = args.max_length - len(prompt)

    def step_device(i):
        pcm = dev_batches[i % len(dev_batches)]
        mel = log_mel(pcm, None, sh.n_mel)
        enc = model.encode(mel)
        return model.decode(enc, prompt, args.max_length, False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing (`value`)
    for i in range(W):
        step_device(i)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = model.ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    outs = []
    for i in range(K):
        outs.append(step_device(W + i))
    if world > 1:       # final result gather (the only collective of the path)
        from taiwan_whisper_b200.shard import gather_token_rows
        all_toks, all_lens = gather_token_rows(torch.cat([o[0] for o in outs]), torch.cat([o[1] for o in outs]),
                                               model._rules(False)["pad"], world * K * B)
    e1.record()
    barrier()
    last_out = outs[-1]          # what the headline's timed path returned in its last step (replaced when the pipeline runs)
    ms = e0.elapsed_time(e1)
    launches = model.ctx.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    stage = model.last_stage_ms()
    # roofline pass: the same K steps again with a CUDA-event pair around one cross-attention launch per decode
    # step (per-launch events cannot ride in the replayed CUDA graph, so this pass launches the kernels directly)
    prof_ms, prof_n, prof_bytes = 0.0, 0, 0.0
    if rank == 0:
        # at the row count the headline decodes: G merged batches when the pipelined loop merges
        pcm_prof = torch.cat([dev_batches[i % len(dev_batches)] for i in range(G)]) if G > 1 else None
        model.profile(True)
        for i in range(min(K, 2)):
            if pcm_prof is None:
                step_device(W + i)
            else:
                model.decode(model.encode(log_mel(pcm_prof, None, sh.n_mel)), prompt, args.max_length, False)
        torch.cuda.synchronize()
        prof_ms, prof_n = model.profile(False)
        prof_bytes = getattr(model, "last_profile_bytes", 0.0)
        del pcm_prof
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * K * B * CLIP_SECONDS / (ms_max / 1000.0)

    # ---------------- ragged variant: real audio ends at different lengths; rows that have finished leave the active list of
    # the cross-attention stream.  Random-init weights never emit EOS, so the lengths come from per-row token budgets
    # (uniform 16 .. n_gen, seeded): same kernels, same batch, device-resident inputs, K decode batches timed.
    ragged = None
    if rank == 0 and world == 1 and not args.no_ragged:
        rng = np.random.default_rng(0)
        bud = rng.integers(16, n_gen + 1, size=B)
        model.set_row_budgets(bud.tolist())
        step_device(0)
        torch.cuda.synchronize()
        e0.record()
        for i in range(K):
            step_device(W + i)
        e1.record()
        torch.cuda.synchronize()
        r_ms = e0.elapsed_time(e1) / K
        model.set_row_budgets(None)
        ragged = {"workload": f"same batch, per-row budgets uniform 16..{n_gen} tokens (mean {bud.mean():.1f}, max {int(bud.max())}) standing in for EOS",
                  "ms_per_step": r_ms, "value": B * CLIP_SECONDS / (r_ms / 1000.0), "unit": "audio-s/s",
                  "generated_tokens": int(bud.sum()), "full_budget_tokens": int(B * n_gen)}

    # ---------------- end-to-end timing through the host API (`e2e`)
    e2e = None
    if not args.no_e2e:
        out_tok = torch.empty((B, n_gen), dtype=torch.int32).pin_memory()
        out_len = torch.empty((B,), dtype=torch.int32).pin_memory()
        for i in range(min(W, 1)):
            model.transcribe_pcm(host_batches[i], args.max_length, out_tokens=out_tok, out_lengths=out_len)
        barrier()
        e0.record()
        for i in range(K):
            model.transcribe_pcm(host_batches[(W + i) % len(host_batches)], args.max_length, out_tokens=out_tok, out_lengths=out_len)
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
        stage = model.last_stage_ms()
        e2e = {"value": world * K * B * CLIP_SECONDS / (e2e_ms / 1000.0), "unit": "audio-s/s",
               "h2d_bytes_per_step": int(host_batches[0].numel() * 2), "d2h_bytes_per_step": int(out_tok.numel() * 4 + out_len.numel() * 4),
               "ms_per_step": e2e_ms / K, "api": "B200WhisperForConditionalGeneration.transcribe_pcm -> tw_transcribe_host"}

    # ---------------- pipelined batch loop (headline when the driver has green contexts): log-mel + encoder + cross-K/V of batch i+1
    # run on a small SM partition while batch i decodes on the rest (model.transcribe_batches).  Steady state: the pipeline is
    # primed by the warm-up batches; the timed region holds exactly K stage-1 passes (batches W+1 .. W+K) and K decodes
    # (batches W .. W+K-1) and ends with a device synchronise, so the last stage-1 pass is inside it.
    seq = {"value": value, "ms_per_step": ms_max / K, "clips_per_step": B, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks}
    pipeline = None
    if not args.no_pipeline:
        try:
            sms = model.enable_pipeline(args.pipeline_sms if args.pipeline_sms > 0 else (16 if G == 1 else 24))
        except (NotImplementedError, RuntimeError) as ex:
            sms = None
            pipeline = {"unavailable": f"{type(ex).__name__}: {ex}"}
        if sms:
            def timed_pipeline(batches_fn, auto_sms=False, G=G):
                # a pipelined step = G batches of B clips: G stage-1 passes and ONE merged decode over G * B rows
                gen = model.transcribe_batches((batches_fn(i) for i in range((W + K + 1) * G)), args.max_length, merge=G, auto_sms=auto_sms)
                for _ in range(W * G):
                    next(gen)
                barrier()
                l0 = model.ctx.launch_count()
                e0.record()
                got = [next(gen) for _ in range(K * G)]
                torch.cuda.synchronize()
                e1.record()
                barrier()
                t_ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
                n_l = model.ctx.launch_count() - l0
                for _ in gen:                       # drain: decode of the extra batch, outside the timed region
                    pass
                if world > 1:
                    dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
                return float(t_ms.item()), n_l, got

            sampler = ClockSampler(local_rank)
            if rank == 0:
                sampler.start()
            p_ms, p_launches, got = timed_pipeline(lambda i: dev_batches[i % len(dev_batches)])
            last_out = (torch.cat([g[0] for g in got[-G:]]), torch.cat([g[1] for g in got[-G:]]))
            clocks = sampler.stop() if rank == 0 else None
            if world > 1:       # final result gather (the only collective of the path)
                from taiwan_whisper_b200.shard import gather_token_rows
                gather_token_rows(torch.cat([g[0] for g in got]).to(dev), torch.cat([g[1] for g in got]).to(dev),
                                  model._rules(False)["pad"], world * K * B * G)
            value = world * K * B * G * CLIP_SECONDS / (p_ms / 1000.0)
            ms_max = p_ms
            launches = p_launches
            pipeline = {"encoder_sms": sms[0], "decode_sms": sms[1], "merge": G, "clips_per_step": B * G,
                        "what": "log-mel + encoder + cross-K/V of the next batches in a CUDA green context of encoder_sms SMs, concurrent with the "
                                "greedy decode of the current ones on the other decode_sms SMs (model.transcribe_batches -> tw_pipeline_encode_at / "
                                "tw_pipeline_decode); device-resident PCM for `value`, pinned host PCM for `e2e`"
                                + (f"; merge = {G}: {G} consecutive {B}-clip batches of the reference loop are encoded one by one into one slot and "
                                   f"decoded TOGETHER as {B * G} rows (a decode step streams the weights and runs its chain of small kernels once "
                                   f"whatever the row count), so a pipelined step = {B * G} clips; `sequential` is the strict one-batch-per-call loop"
                                   if G > 1 else ""),
                        "stage_ms_in_partition": model.last_stage_ms()}
            if G > 1 and rank == 0 and world == 1:
                # the same loop with ONE batch per decode (merge = 1) on its own best split (16 encoder SMs): what merging buys
                model.enable_pipeline(16)
                u_ms, _, _ = timed_pipeline(lambda i: dev_batches[i % len(dev_batches)], G=1)
                pipeline["unmerged"] = {"merge": 1, "encoder_sms": model.pipeline_sms[0], "clips_per_step": B, "ms_per_step": u_ms / K,
                                        "value": K * B * CLIP_SECONDS / (u_ms / 1000.0), "unit": "audio-s/s"}
                model.enable_pipeline(sms[0])
            if ragged is not None:
                # the ragged variant through the same pipelined / merged loop: budgets drawn per row of the merged batch
                bud = np.random.default_rng(0).integers(16, n_gen + 1, size=B * G)
                model.set_row_budgets(bud.tolist())
                r_ms, _, _ = timed_pipeline(lambda i: dev_batches[i % len(dev_batches)])
                ragged["pipelined"] = {"ms_per_step": r_ms / K, "clips_per_step": B * G, "value": K * B * G * CLIP_SECONDS / (r_ms / 1000.0),
                                       "unit": "audio-s/s", "generated_tokens": int(bud.sum()), "full_budget_tokens": int(B * G * n_gen),
                                       "encoder_sms": model.pipeline_sms[0]}
                # rows that end early shift the balance towards stage 1: the same loop with the balance controller (auto_sms=True; it
                # settles during the warm-up groups), then back to the headline's split
                model.sms_history = []
                ra_ms, _, _ = timed_pipeline(lambda i: dev_batches[i % len(dev_batches)], auto_sms=True)
                ragged["pipelined_auto_sms"] = {"ms_per_step": ra_ms / K, "clips_per_step": B * G,
                                                "value": K * B * G * CLIP_SECONDS / (ra_ms / 1000.0), "unit": "audio-s/s",
                                                "encoder_sms": model.pipeline_sms[0], "resizes": [list(x) for x in model.sms_history]}
                model.set_row_budgets(None)
                model.enable_pipeline(sms[0])
            if not args.no_e2e:
                pe_ms, _, _ = timed_pipeline(lambda i: host_batches[i % len(host_batches)])
                e2e = {"value": world * K * B * G * CLIP_SECONDS / (pe_ms / 1000.0), "unit": "audio-s/s",
                       "h2d_bytes_per_step": int(G * host_batches[0].numel() * 2), "d2h_bytes_per_step": int(G * (B * n_gen * 4 + B * 4)),
                       "ms_per_step": pe_ms / K, "api": "B200WhisperForConditionalGeneration.transcribe_batches -> tw_pipeline_encode_at / tw_pipeline_decode"}

    if rank == 0:
        hbm, tf, which = peaks()
        tf_sus = sustained_tflops()
        if not isinstance(stage, dict):
            stage = {}
        bytes_per_launch = B * G * 1500 * 2 * sh.d_model * 2      # K|V rows of one decoder layer for the decoded rows, bf16
        if prof_bytes > 0:                                        # split decode: one launch streams one sub-batch
            bytes_per_launch = int(prof_bytes)
        roof = None
        if prof_n > 0:
            ach = bytes_per_launch / (prof_ms / prof_n / 1000.0) / 1e9
            roof = {"kernel": "decode_attention_partial (cross-attention K/V streaming, 1 launch per layer per token)",
                    "bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm, "peak_source": which,
                    "traffic": ncu_traffic_bytes(B * G) if (args.model == MODEL and B == BATCH) else None,
                    "traffic_source": f"profiles/{NCU_TRAFFIC_CSV.get(B * G, '-')} (ncu --set full, same shape: {B * G} clips per launch)",
                    "rows": f"{B * G} clips per launch (the row count of the headline's decode)",
                    "launches_timed": prof_n, "avg_launch_us": 1000.0 * prof_ms / prof_n,
                    "algorithmic_bytes_per_launch": bytes_per_launch,
                    "how": "CUDA events around one launch per decode step (middle decoder layer) on the launching stream, in a separate pass "
                           "of the same steps with plain launches (events cannot ride in the replayed CUDA graph)",
                    "peak_note": "MEASURED_PEAKS.json hbm_gbs is a COPY bandwidth (read + write); this kernel only reads, and a read-only "
                                 "stream runs up to ~2 % above it (frac may slightly exceed 1)"}
        # per-stage roofline of the last e2e step (north_star: every stage against HBM or tensor-core peak)
        d, ffn, L_e, L_d, V = sh.d_model, sh.ffn, sh.enc_layers, sh.dec_layers, sh.vocab
        enc_flops = B * (2 * 3000 * d * sh.n_mel * 3 + 2 * 1500 * d * d * 3 +
                         L_e * (8 * 1500 * d * d + 4 * 1500 * 1500 * d + 4 * 1500 * d * ffn))
        xkv_flops = B * L_d * 4 * 1500 * d * d
        w_dec = 2 * (L_d * (6 * d * d + 2 * d * ffn) + d * V)
        steps_dec = args.max_length - 1
        dec_bytes = steps_dec * (w_dec + B * L_d * 2 * 1500 * d * 2) + B * L_d * 2 * d * 2 * (steps_dec * (steps_dec + 1) // 2)
        lm_bytes = B * (480000 * 2 + sh.n_mel * 3000 * 4)
        stages = {}
        if stage.get("encoder", 0) > 0:
            stages = {
                "logmel": {"bound": "hbm", "ms": stage["logmel"], "achieved_gbs": lm_bytes / stage["logmel"] / 1e6,
                           "frac": lm_bytes / stage["logmel"] / 1e6 / hbm, "h2d_ms": stage.get("h2d")},
                "encoder": {"bound": "tensor", "ms": stage["encoder"], "achieved_tflops": enc_flops / stage["encoder"] / 1e9,
                            "frac": enc_flops / stage["encoder"] / 1e9 / tf,
                            "frac_of_sustained_peak": (enc_flops / stage["encoder"] / 1e9 / tf_sus) if tf_sus else None},
                "cross_kv": {"bound": "tensor", "ms": stage["cross_kv"], "achieved_tflops": xkv_flops / stage["cross_kv"] / 1e9,
                             "frac": xkv_flops / stage["cross_kv"] / 1e9 / tf,
                             "frac_of_sustained_peak": (xkv_flops / stage["cross_kv"] / 1e9 / tf_sus) if tf_sus else None},
                "decode": {"bound": "hbm", "ms": stage["decode"], "achieved_gbs": dec_bytes / stage["decode"] / 1e6,
                           "frac": dec_bytes / stage["decode"] / 1e6 / hbm,
                           "note": "weights + cross-K/V + self-K/V streamed once per token"},
            }
        if pipeline is not None and "encoder_sms" in pipeline and pipeline["stage_ms_in_partition"].get("decode", 0) > 0:
            rows = B * G
            mdec_bytes = steps_dec * (w_dec + rows * L_d * 2 * 1500 * d * 2) + rows * L_d * 2 * d * 2 * (steps_dec * (steps_dec + 1) // 2)
            t_alone = pipeline["stage_ms_in_partition"]["decode"]
            stages["decode_pipelined"] = {
                "bound": "hbm", "rows": rows, "sms": pipeline["decode_sms"],
                "ms_alone": t_alone, "achieved_gbs_alone": mdec_bytes / t_alone / 1e6, "frac_alone": mdec_bytes / t_alone / 1e6 / hbm,
                "ms_per_step": ms_max / K, "frac_of_step": mdec_bytes / (ms_max / K) / 1e6 / hbm,
                "note": "the decode of the pipelined loop over all merged rows on the decode partition: `alone` = the last decode of the loop "
                        "(no stage 1 running beside it); `frac_of_step` charges the whole pipelined step (stage 1 of the next batches runs "
                        "concurrently and shares HBM and the power budget) to the decode's bytes"}
        line = {
            "metric": "rtfx_audio_seconds_per_second", "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": workload_text(args.model, B, args.max_length, n_gen) + f"; a step = {G} batch(es) = {B * G} clips"
                                   + (f" (pipelined loop, {G} batches decoded together)" if G > 1 else ""),
                       "batch_per_gpu": B, "clips_per_step": B * G, "max_length": args.max_length, "weights": "random-init (HF init, seed 1234)",
                       "parallelism": f"manifest sharded over {world} GPU(s), no data-path collective",
                       "l2": "inputs larger than L2: each step streams >= 15 GB of K/V and weights (L2 is 126 MB)",
                       "pipeline": pipeline if pipeline is not None else "off (sequential batch loop)",
                       "stage_ms_last_step": stage},
            "clocks": clocks, "gpu_launches": int(launches), "e2e": e2e, "roofline": roof, "stages": stages,
        }
        if pipeline is not None and "encoder_sms" in pipeline:
            # the same K steps as a sequential loop (one batch at a time on the whole GPU): `stages` and `roofline` come from this pass
            line["sequential"] = seq
        if ragged is not None:
            line["ragged"] = ragged
        if hf_cpu is not None:
            cb, ref_feats, ref_ids = cpu_baseline(args, hf_cpu)
            line["cpu_baseline"] = cb
            if not args.no_parity:
                try:
                    line["parity"] = parity_block(args, hf_cpu, model, ref_feats, ref_ids, dev)
                except Exception as e:        # the throughput line must survive a parity-leg failure; the failure is reported
                    line["parity"] = {"error": f"{type(e).__name__}: {e}"}
            if not args.no_hf_cuda:
                try:
                    line["extra"] = hf_cuda_comparator(args, hf_cpu, host_batches[0], dev)
                except Exception as e:
                    line["extra"] = {"hf_cuda_error": f"{type(e).__name__}: {e}"}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"tokens": last_out[0].cpu(), "lengths": last_out[1].cpu()})
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
