"""Shared test helpers: HF weights -> numpy dict, default rules for the oracle."""
import numpy as np

from taiwan_whisper_b200.configs import NON_SPEECH_TOKENS_MULTI, token_ids


def weights_np(hf_model):
    return {k: v.detach().float().numpy() for k, v in hf_model.state_dict().items()}


PERTURBED = "-perturbed"     # test-parameter suffix: the shape's model with perturb_hf_model applied


def split_shape(name):
    """"tiny" -> ("tiny", False); "tiny-perturbed" -> ("tiny", True)."""
    return (name[:-len(PERTURBED)], True) if name.endswith(PERTURBED) else (name, False)


def perturb_hf_model(hf_model, seed=4321):
    """Gives an HF Whisper model non-trivial biases and LayerNorms, in place: every existing bias ~ N(0, 0.05), every LayerNorm
    gamma ~ 1 + N(0, 0.1) and beta ~ N(0, 0.1), drawn tensor by tensor from one seeded generator, so every layer gets its own
    values and a parameter routed to the wrong layer or projection changes the result.  HF's init leaves every bias at 0 and every
    LayerNorm at (1, 0), where such a mistake is invisible.  Embeddings and positions are left alone (EOS keeps its zero row)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for _, mod in hf_model.named_modules():
            if isinstance(mod, torch.nn.LayerNorm):
                mod.weight.copy_(1.0 + 0.1 * torch.randn(mod.weight.shape, generator=g))
                mod.bias.copy_(0.1 * torch.randn(mod.bias.shape, generator=g))
            elif isinstance(mod, (torch.nn.Linear, torch.nn.Conv1d)) and mod.bias is not None:
                mod.bias.copy_(0.05 * torch.randn(mod.bias.shape, generator=g))
    return hf_model


def default_rules(vocab, timestamps=False, suppress=True):
    ids = token_ids(vocab)
    special = [ids.sot, ids.translate, ids.transcribe, ids.startofprev - 1, ids.startofprev, ids.nospeech]
    return dict(
        suppress=sorted(set(NON_SPEECH_TOKENS_MULTI[:-4] + special)) if suppress else [],
        begin_suppress=[220, ids.eos], eos=ids.eos,
        ts_begin=ids.timestamp_begin if timestamps else None,
        no_timestamps=ids.notimestamps, max_initial_ts=50,
    )


def prompt_ids(vocab, timestamps=False, language="zh"):
    ids = token_ids(vocab)
    p = [ids.sot, ids.lang_to_id[f"<|{language}|>"], ids.transcribe]
    if not timestamps:
        p.append(ids.notimestamps)
    return p


class StubWhisperTokenizer:
    """Duck-typed tokenizer for HF's module-level `_decode_asr` (needs no vocabulary files): text of a token list is the
    comma-joined ids, so the chunks' token lists can be read back."""

    def __init__(self, ids):
        self.ids = ids
        self.all_special_ids = list(range(ids.eos, ids.timestamp_begin))

    def convert_tokens_to_ids(self, tok):
        return {"<|notimestamps|>": self.ids.notimestamps, "<|startofprev|>": self.ids.startofprev,
                "<|startoftranscript|>": self.ids.sot}[tok]

    def _strip_prompt(self, token_ids, prompt_token_id, decoder_start_token_id):
        if token_ids and token_ids[0] == prompt_token_id:
            return token_ids[token_ids.index(decoder_start_token_id):] if decoder_start_token_id in token_ids else []
        return token_ids

    def decode(self, ids):
        return "".join(f"{int(t)}," for t in ids)
