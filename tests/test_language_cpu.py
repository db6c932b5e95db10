"""CPU: the per-row prompts of language detection and language lists against HF's _retrieve_init_tokens, and the oracle's
detection (tests/language_common.py) against live HF detect_language and generate(language=None)."""
import copy

import numpy as np
import pytest
import torch

from oracle import hf_ref, logmel_np, whisper_np
from taiwan_whisper_b200 import lib as twlib
from taiwan_whisper_b200.configs import SHAPES, token_ids
from taiwan_whisper_b200.synth import dequantise, synth_batch
from tests.helpers import default_rules, perturb_hf_model, weights_np
from tests.language_common import oracle_detect_language, plant_languages, step0_states, target_languages

STUB_LANG = 50300          # what the stubbed detection "detects"

# (generate kwargs, generation-config forced_decoder_ids): the rows of HF's language=None prompt table
CASES = [
    (dict(), None),
    (dict(task="transcribe"), None),
    (dict(return_timestamps=True), None),
    (dict(task="translate", return_timestamps=True), None),
    (dict(), "transcribe"),
    (dict(task="translate"), "transcribe"),
    (dict(language=["zh", "en"]), None),
    (dict(language=("ja", "<|ko|>"), task="translate", return_timestamps=True), None),
    (dict(language="zh"), "transcribe"),
]


def _models(vocab):
    from taiwan_whisper_b200.host import B200WhisperForConditionalGeneration as M
    hf = hf_ref.build_hf_model("micro128" if vocab == 51866 else "micro80")
    m = M.__new__(M)
    m.generation_config, m.config, m.handle = hf.generation_config, hf.config, None
    return hf, m


def _hf_init_tokens(hf, B, language=None, task=None, return_timestamps=False, forced=None):
    """HF _retrieve_init_tokens as generate() reaches it (generation config copy with language / task / return_timestamps),
    detection stubbed to STUB_LANG."""
    gc = copy.deepcopy(hf.generation_config)
    gc.language, gc.task, gc.return_timestamps = language, task, return_timestamps
    if forced is not None:
        gc.forced_decoder_ids = [[1, None], [2, gc.task_to_id[forced]]]
    hf.detect_language = lambda **kw: torch.full((B,), STUB_LANG, dtype=torch.long)
    try:
        return hf._retrieve_init_tokens(torch.zeros((B, hf.config.num_mel_bins, 3000)), B, gc, hf.config, 3000, {}).tolist()
    finally:
        del hf.detect_language


@pytest.mark.parametrize("vocab", [51865, 51866])
@pytest.mark.parametrize("case", range(len(CASES)))
def test_row_prompts_match_hf_retrieve_init_tokens(vocab, case):
    kw, forced = CASES[case]
    hf, m = _models(vocab)
    B = 2
    ref = _hf_init_tokens(hf, B, kw.get("language"), kw.get("task"), kw.get("return_timestamps", False), forced)
    if forced is not None:
        m.generation_config = copy.deepcopy(hf.generation_config)
        m.generation_config.forced_decoder_ids = [[1, None], [2, m.generation_config.task_to_id[forced]]]
    mine = m._row_prompts(kw.get("language"), kw.get("task"), kw.get("return_timestamps", False), B)
    assert m._resolved(mine, [STUB_LANG] * B) == ref
    detects = [p[1] == twlib.PROMPT_DETECT for p in mine]
    assert all(detects) == (kw.get("language") is None) and (any(detects) == all(detects))


def test_row_prompts_table_lengths():
    """The prompt lengths of HF's language=None table: 3, 4, 2, 3 and 4 with forced_decoder_ids."""
    hf, m = _models(51866)
    ids = token_ids(51866)
    D = twlib.PROMPT_DETECT
    assert m._row_prompts(None, None, False, 1) == [[ids.sot, D, ids.notimestamps]]
    assert m._row_prompts(None, "transcribe", False, 1) == [[ids.sot, D, ids.transcribe, ids.notimestamps]]
    assert m._row_prompts(None, None, True, 1) == [[ids.sot, D]]
    assert m._row_prompts(None, "translate", True, 1) == [[ids.sot, D, ids.translate]]
    assert m._row_prompts(["zh", "en"], None, False, 2) == [[ids.sot, 50260, ids.transcribe, ids.notimestamps],
                                                            [ids.sot, 50259, ids.transcribe, ids.notimestamps]]
    # a single language is the prompt _init_tokens has always built, given to every row
    assert m._row_prompts("zh", "transcribe", False, 3) == [m._init_tokens("zh", "transcribe", False)] * 3


@pytest.mark.parametrize("language, exc", [(["zh", None], TypeError), (["zh"], ValueError), (["zh", "en", "ja"], ValueError)])
def test_language_list_errors_match_hf(language, exc):
    hf, m = _models(51866)
    with pytest.raises(exc) as ref:
        _hf_init_tokens(hf, 2, language, "transcribe")
    with pytest.raises(exc) as mine:
        m._row_prompts(language, "transcribe", False, 2)
    assert str(mine.value) == str(ref.value)


def _planted_cpu(shape_name, n=6, margin=0.05):
    sh = SHAPES[shape_name]
    hf = perturb_hf_model(hf_ref.build_hf_model(sh, seed=1234))
    mel = logmel_np.log_mel(dequantise(synth_batch(0, n)), sh.n_mel)
    targets = target_languages(hf, n)
    lang_ids = plant_languages(hf, step0_states(hf, mel), targets, margin)
    return hf, mel, targets, lang_ids


@pytest.mark.parametrize("shape_name", ["tiny", "micro128"])
@pytest.mark.parametrize("planted", [False, True])
def test_oracle_detect_language_vs_hf(shape_name, planted):
    """oracle_detect_language equals HF detect_language on perturbed models (one language for every clip) and on planted ones
    (the planted language of every clip); the planted margins are what was asked for."""
    sh = SHAPES[shape_name]
    if planted:
        hf, mel, targets, lang_ids = _planted_cpu(shape_name)
    else:
        hf = perturb_hf_model(hf_ref.build_hf_model(sh, seed=1234))
        mel = logmel_np.log_mel(dequantise(synth_batch(0, 4)), sh.n_mel)
        lang_ids = sorted(hf.generation_config.lang_to_id.values())
    W = weights_np(hf)
    ref = hf.detect_language(input_features=torch.from_numpy(mel)).tolist()
    for b in range(mel.shape[0]):
        enc = whisper_np.encoder_forward(W, mel[b], sh.heads, sh.enc_layers)
        lang, margin = oracle_detect_language(W, enc, lang_ids, sh.heads, sh.dec_layers)
        assert lang == ref[b], b
        if planted:
            assert lang == targets[b] and abs(margin - 0.05) < 1e-3, (b, margin)
    if planted:
        assert len(set(ref)) == mel.shape[0]


@pytest.mark.parametrize("shape_name", ["tiny", "micro128"])
def test_hf_generate_language_none_vs_oracle(shape_name):
    """HF generate(language=None) on a planted model = the oracle's greedy decode with HF's per-row prompts, the detected
    language at index 1."""
    sh = SHAPES[shape_name]
    hf, mel, targets, lang_ids = _planted_cpu(shape_name)
    W = weights_np(hf)
    max_length = 12
    with torch.no_grad():
        ids = hf.generate(torch.from_numpy(mel), max_length=max_length, num_beams=1, task="transcribe").numpy()
    ti = token_ids(sh.vocab)
    for b in range(mel.shape[0]):
        enc = whisper_np.encoder_forward(W, mel[b], sh.heads, sh.enc_layers)
        prompt = [ti.sot, targets[b], ti.transcribe, ti.notimestamps]
        toks = whisper_np.greedy_decode(W, enc, prompt, default_rules(sh.vocab), max_length, sh.heads, sh.dec_layers)
        assert ids[b, :len(toks)].tolist() == toks, b
