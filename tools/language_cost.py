"""What language detection costs the pipelined batch loop: transcribe_batches(merge=3) at large-v3 shapes with language="zh"
against language=None (each row's language picked in the decode's first step), alternated within one run so that both see the
same machine state.  The pick replaces the token selection of the eagerly launched step 0; no replayed step changes.

    python tools/language_cost.py --rounds 5 --out /tmp/language_cost.json

Prints (and writes) one JSON object: the card's name and power limit, the wall time of every run of each mode, their medians
and the spread (max - min) of each mode."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30).stdout.strip().splitlines()[0]
        name, limit = [s.strip() for s in q.split(",")]
        return name, limit
    except Exception as e:          # the numbers still mean something; say where they come from
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default="large-v3")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--merge", type=int, default=3)
    ap.add_argument("--groups", type=int, default=2, help="merged decodes per run")
    ap.add_argument("--max-length", type=int, default=128)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from taiwan_whisper_b200.configs import SHAPES
    from taiwan_whisper_b200.hf_compat import build_hf_model
    from taiwan_whisper_b200.host import B200WhisperForConditionalGeneration
    from taiwan_whisper_b200.synth import synth_batch

    if not torch.cuda.is_available():
        raise SystemExit("language_cost.py measures on the GPU; there is no CPU fallback")
    dev = torch.device("cuda:0")
    B, G = args.batch, args.merge
    with torch.device(dev):
        hf = build_hf_model(SHAPES[args.shape], seed=1234)
    model = B200WhisperForConditionalGeneration.from_hf(hf, dtype=torch.bfloat16, max_batch=B * G, device=str(dev), output_layout="5.x")
    del hf
    model.enable_pipeline(24)
    pcm = torch.from_numpy(synth_batch(0, B)).pin_memory()
    batches = [pcm] * (G * args.groups)

    def run(language):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n = sum(1 for _ in model.transcribe_batches(batches, args.max_length, language=language, task="transcribe", merge=G))
        torch.cuda.synchronize()
        assert n == len(batches)
        return time.perf_counter() - t0

    modes = {"zh": "zh", "detect": None}
    for lang in modes.values():          # warm-up: graph capture, module loads
        run(lang)
    times = {k: [] for k in modes}
    for r in range(args.rounds):
        order = list(modes) if r % 2 == 0 else list(modes)[::-1]
        for k in order:
            times[k].append(run(modes[k]))
    name, limit = card()
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    res = {"gpu": name, "power_limit": limit, "shape": args.shape, "rows_per_decode": B * G, "decodes_per_run": args.groups,
           "max_length": args.max_length, "seconds": times, "median_s": med,
           "spread_s": {k: max(v) - min(v) for k, v in times.items()},
           "detect_over_zh": med["detect"] / med["zh"]}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    model.close()


if __name__ == "__main__":
    main()
