"""Language detection test helpers: the detection restated on the numpy oracle, and models with planted languages.

A random-init Whisper picks the same language for every clip: its step-0 state barely depends on the audio, so a test on such a
model cannot tell detection from a constant.  `plant_languages` rewrites the language rows of the tied embedding so that every clip
wins a chosen language by a chosen margin.  The language rows enter the step-0 logits only through the vocabulary product (the
step-0 state depends on SOT and the audio alone), so the margins can be solved for exactly: each row gets the least-norm change
that gives the clips' step-0 final-LayerNorm states the target scores (winner: `margin`, every other language: 0).  The clips'
states differ by little, so the rows grow by a large factor: they stay what a decode feeds as a token at step 1, which the
oracle and HF see the same way."""
import numpy as np
import torch

from oracle import whisper_np

SOT = 50258                     # <|startoftranscript|> of both multilingual vocabularies


def oracle_detect_language(W, enc, lang_ids, heads, n_layers):
    """HF detect_language (generation_whisper.py:1610-1673) on the oracle: logits of the decoder step fed SOT, every id outside
    lang_ids at -inf, argmax.  Returns (id, margin between the best and the second-best language logit)."""
    xkv = whisper_np.cross_kv(W, enc, n_layers)
    logits = whisper_np.decoder_forward(W, np.asarray([SOT]), whisper_np.DecoderState(n_layers), xkv, heads, n_layers)
    masked = np.full_like(logits, -np.inf)
    masked[lang_ids] = logits[lang_ids]
    top2 = np.sort(logits[lang_ids])[-2:]
    return int(np.argmax(masked)), float(top2[1] - top2[0])


@torch.no_grad()
def step0_states(hf, feats, device="cpu", chunk=32):
    """fp32 final-LayerNorm output of the decoder step fed SOT, per clip: float64 [n, d].  On CUDA with TF32 off."""
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        m = hf.to(device)
        out = []
        for s in range(0, feats.shape[0], chunk):
            f = torch.as_tensor(feats[s:s + chunk]).to(device=device, dtype=torch.float32)
            enc = m.model.encoder(f).last_hidden_state
            ids = torch.full((f.shape[0], 1), SOT, dtype=torch.long, device=device)
            h = m.model.decoder(input_ids=ids, encoder_hidden_states=enc).last_hidden_state[:, 0]
            out.append(h.double().cpu().numpy())
        hf.to("cpu")
        return np.concatenate(out)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev


@torch.no_grad()
def plant_languages(hf, states, targets, margin):
    """Rewrites the language rows of hf's tied embedding in place: clip c (state states[c]) scores `margin` on language targets[c]
    and 0 on every other language.  Returns the language ids."""
    lang_ids = sorted(int(v) for v in hf.generation_config.lang_to_id.values())
    E = hf.model.decoder.embed_tokens.weight
    R = E[lang_ids].double().numpy()                       # [L, d]
    H = np.asarray(states, np.float64)                      # [n, d]
    Y = np.zeros((H.shape[0], len(lang_ids)))
    for c, t in enumerate(targets):
        Y[c, lang_ids.index(int(t))] = margin
    R = R + (np.linalg.pinv(H) @ (Y - H @ R.T)).T          # least-norm change per row: H @ R_new.T = Y
    E[lang_ids] = torch.from_numpy(R).to(E.dtype)
    return lang_ids


def target_languages(hf, n, names=("zh", "en", "ja", "ko", "de", "fr", "es", "ru")):
    """Language ids cycling through `names`: n clips, min(n, 8) distinct languages."""
    l2i = hf.generation_config.lang_to_id
    return [l2i[f"<|{names[i % len(names)]}|>"] for i in range(n)]
