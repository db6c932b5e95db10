"""GPU: language detection inside the decode's first step, per-row prompts and detect_language(), on models with planted
languages (tests/language_common.py) so that every clip of a batch has its own language."""
import functools

import numpy as np
import pytest
import torch

from oracle import hf_ref, logmel_np, whisper_np
from taiwan_whisper_b200 import lib as twlib
from taiwan_whisper_b200.configs import SHAPES, token_ids
from taiwan_whisper_b200.synth import dequantise, synth_batch
from tests.helpers import default_rules, perturb_hf_model, weights_np
from tests.language_common import oracle_detect_language, plant_languages, step0_states, target_languages

pytestmark = pytest.mark.gpu

FP32_MARGIN = 0.05        # planted margins (logits) of the fp32 models: far above the check mode's rounding
BF16_MARGIN = 1.0         # and of the bf16 ones
BF16_BAR = 0.5            # rows whose fp32 margin is at least this must detect the fp32 language in bf16 ...
BF16_MISS = 0.03          # ... all but this share of them: the bf16 step-0 logit error on the planted lv3w model reached one logit
                          # on 1 of 192 clips (B200, 1000 W)
BF16_SAME = 0.95          # share of rows two bf16 decodes of the same prompts must agree on bit for bit: the residual GEMMs add
                          # split-K partials with fp32 atomics, so a near-tie can go either way from one run to the next
MAX_LENGTH = 16


def _cuda():
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the -m gpu tests must run on a B200 (there is no CPU fallback)")


def _names(hf, ids):
    i2l = {v: k[2:-2] for k, v in hf.generation_config.lang_to_id.items()}
    return [i2l[int(t)] for t in ids]


@functools.lru_cache(maxsize=None)
def _planted_fp32(shape_name, n=6):
    sh = SHAPES[shape_name]
    hf = perturb_hf_model(hf_ref.build_hf_model(sh, seed=1234))
    mel = logmel_np.log_mel(dequantise(synth_batch(0, n)), sh.n_mel)
    targets = target_languages(hf, n)
    lang_ids = plant_languages(hf, step0_states(hf, mel), targets, FP32_MARGIN)
    return hf, mel, targets, lang_ids


def _b200(hf, dtype, max_batch, layout="5.x"):
    from taiwan_whisper_b200.host import B200WhisperForConditionalGeneration
    return B200WhisperForConditionalGeneration.from_hf(hf, dtype=dtype, max_batch=max_batch, output_layout=layout)


# ---------------------------------------------------------------------------------------------- the pick kernel
@pytest.mark.parametrize("vocab", [51865, 51866])
def test_pick_kernel_crafted_logits(vocab):
    """tw_debug_select_steps_rows on crafted step-0 logits against torch's masked argmax: ties inside the language set (the
    first id wins), the maximum outside the set, a single finite candidate, every candidate -inf, a row with a given language
    among detecting rows.  The pick writes nothing but the languages: tokens, lengths and the active list equal those of the
    same call with the picked languages given."""
    _cuda()
    from tests.gpu_common import b200_model
    m = b200_model("micro80" if vocab == 51865 else "micro128", "bf16", max_batch=256)
    ids = token_ids(vocab)
    L = sorted(ids.lang_to_id.values())
    assert len(L) == (99 if vocab == 51865 else 100)
    B, n_gen, ld = 10, 3, (vocab + 3) // 4 * 4
    g = torch.Generator().manual_seed(vocab)
    lg = torch.randn((n_gen, B, ld), generator=g) * 3
    s0 = lg[0]
    s0[0, L[3]] = s0[0, L[10]] = 40.0                        # tie inside the set
    s0[1, 100] = 99.0; s0[1, L[5]] = 30.0                    # maximum outside the set
    s0[2, L] = -float("inf"); s0[2, L[40]] = -5.0            # one finite candidate
    s0[3, L] = -float("inf")                                 # none: torch.argmax of an all -inf row is 0
    s0[4, L[-1]] = 50.0                                      # given language: the logits are not read
    s0[5, L[0]] = s0[5, L[-1]] = 45.0                        # tie across the whole set
    masked = torch.full_like(s0[:, :vocab], -float("inf"))
    masked[:, L] = s0[:, L]
    expect = masked.argmax(-1).tolist()
    expect[4] = ids.lang_to_id["<|zh|>"]
    assert expect[0] == L[3] and expect[1] == L[5] and expect[2] == L[40] and expect[3] == 0 and expect[5] == L[0]
    assert len(set(expect)) >= 6
    lg = lg.cuda()
    rules = default_rules(vocab)
    r, keep_r = twlib.make_rules(rules["suppress"], rules["begin_suppress"], rules["eos"], ids.pad, None, ids.notimestamps, 50)

    def run(prompts, lang_ids, want_langs):
        toks = torch.full((B, n_gen), -7, dtype=torch.int32, device="cuda")
        lens = torch.full((B,), -7, dtype=torch.int32, device="cuda")
        nact = torch.full((n_gen,), -7, dtype=torch.int32, device="cuda")
        act = torch.full((n_gen, B), -7, dtype=torch.int32, device="cuda")
        langs = torch.full((B,), -7, dtype=torch.int32, device="cuda")
        rows, keep, P = twlib.make_prompt_rows(prompts, lang_ids, langs.data_ptr() if want_langs else None)
        m.ctx.check(m.ctx.lib.tw_debug_select_steps_rows(
            m.handle, lg.data_ptr(), ld, B, rows, P, r, P + n_gen, None, None, None, 0, toks.data_ptr(), lens.data_ptr(),
            nact.data_ptr(), act.data_ptr(), torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        return [t.cpu().tolist() for t in (toks, lens, nact, act, langs)]

    D = twlib.PROMPT_DETECT
    tail = [ids.transcribe, ids.notimestamps]
    detect = [[ids.sot, D if b != 4 else expect[4]] + tail for b in range(B)]
    toks, lens, nact, act, langs = run(detect, L, True)
    assert langs == expect
    given = [[ids.sot, expect[b]] + tail for b in range(B)]
    assert run(given, None, False)[:4] == [toks, lens, nact, act]
    # out_lang alone (no row detects) reports the given languages
    assert run(given, None, True)[4] == expect
    # the first generated step (P = 2: position 1) follows the pick at position 0 on the same logits
    short = [[ids.sot, D if b != 4 else expect[b]] for b in range(B)]
    toks2, lens2, _, _, langs2 = run(short, L, True)
    assert langs2 == expect
    assert run([[ids.sot, e] for e in expect], None, False)[:2] == [toks2, lens2]


def test_pick_rejects_bad_rows():
    _cuda()
    from tests.gpu_common import b200_model
    m = b200_model("micro128", "bf16", max_batch=256)
    ids = token_ids(51866)
    lg = torch.zeros((2, 2, (51866 + 3) // 4 * 4), device="cuda")
    r, keep_r = twlib.make_rules([], [], ids.eos, ids.pad, None, ids.notimestamps, None)
    out = torch.zeros((2, 2), dtype=torch.int32, device="cuda")
    for prompts, langs in ([[[ids.sot, -1, ids.transcribe], [ids.sot, -1, ids.transcribe]], None],          # detect without ids
                           [[[ids.sot, 50260, ids.transcribe], [ids.eos, 50260, ids.transcribe]], None],     # SOT differs
                           [[[ids.sot, ids.transcribe, -1], [ids.sot, 50260, -1]], [50260]]):                # -1 outside slot 1
        rows, keep, P = twlib.make_prompt_rows(prompts, langs)
        rc = m.ctx.lib.tw_debug_select_steps_rows(m.handle, lg.data_ptr(), lg.shape[-1], 2, rows, P, r, P + 2, None, None, None, 0,
                                                  out.data_ptr(), out[0].data_ptr(), None, None, torch.cuda.current_stream().cuda_stream)
        assert rc == twlib.TW_E_INVALID


# ---------------------------------------------------------------------------------------------- fp32 check mode vs HF
GEN_CASES = [dict(), dict(task="transcribe"), dict(return_timestamps=True), dict(task="translate", return_timestamps=True)]


@pytest.mark.parametrize("graph", [True, False])
@pytest.mark.parametrize("shape_name", ["tiny", "micro128"])
def test_generate_language_none_fp32_vs_hf(shape_name, graph, monkeypatch):
    """Planted tiny / micro128, B = 6 clips of 6 languages, prompts of length 3, 4, 2 and 3: detect_language and the detected ids
    equal HF's and the oracle's; generate(language=None) equals HF generate(language=None) in the 5.x layout and, with the prompt
    (return_prompt), HF's per-row prompts followed by those ids; with return_timestamps the seek loop detects on a window's
    first pass only."""
    _cuda()
    monkeypatch.setenv("TWB200_GRAPH", "1" if graph else "0")
    sh = SHAPES[shape_name]
    hf, mel, targets, lang_ids = _planted_fp32(shape_name)
    m = _b200(hf, torch.float32, 8)
    feats = torch.from_numpy(mel)
    with torch.no_grad():
        ref_lang = hf.detect_language(input_features=feats).tolist()
    assert ref_lang == targets
    assert m.detect_language(input_features=feats.cuda()).tolist() == targets
    W = weights_np(hf)
    enc_np = [whisper_np.encoder_forward(W, mel[b], sh.heads, sh.enc_layers) for b in range(mel.shape[0])]
    assert [oracle_detect_language(W, e, lang_ids, sh.heads, sh.dec_layers)[0] for e in enc_np] == targets
    calls = []
    decode_rows = m.decode_rows

    def spy(enc, prompts, *a, **k):
        calls.append([list(p) for p in prompts])
        return decode_rows(enc, prompts, *a, **k)

    m.decode_rows = spy
    tsb = token_ids(sh.vocab).timestamp_begin
    pad = hf.generation_config.pad_token_id
    for kw in GEN_CASES:
        ts = kw.get("return_timestamps", False)
        with torch.no_grad():
            ref = hf.generate(feats, max_length=MAX_LENGTH, num_beams=1, **kw).numpy()
        prompts = m._resolved(m._row_prompts(None, kw.get("task"), ts, len(targets)), targets)
        calls.clear()
        ids = m.generate(feats, max_length=MAX_LENGTH, **kw).numpy()
        if ts:
            assert ids.shape == ref.shape and np.array_equal(ids, ref), (kw, ids.tolist(), ref.tolist())
        else:
            # without return_timestamps a window is decoded once; HF 5.x decodes the rest of a window again after a row that
            # emitted timestamp tokens, so those rows are not compared
            n = 0
            for b in range(len(targets)):
                r = [t for t in ref[b].tolist() if t != pad]
                if not any(t >= tsb for t in r):
                    assert [t for t in ids[b].tolist() if t != pad] == r, (kw, b)
                    n += 1
            assert n >= len(targets) // 2, kw
        first = calls[0]
        assert all(p[1] == twlib.PROMPT_DETECT for p in first)
        assert all(p[1] != twlib.PROMPT_DETECT for c in calls[1:] for p in c)          # remainders reuse the detected prompt
        with_prompt = m.generate(feats, max_length=MAX_LENGTH, return_prompt=True, **kw).numpy()
        P = len(prompts[0])
        assert with_prompt[:, :P].tolist() == prompts and np.array_equal(with_prompt[:, P:], ids), kw
        if not kw.get("return_timestamps"):
            for b in range(len(targets)):
                toks = whisper_np.greedy_decode(W, enc_np[b], prompts[b], default_rules(sh.vocab), MAX_LENGTH, sh.heads, sh.dec_layers)
                assert ids[b, :len(toks)].tolist() == toks, (kw, b)
    m.close()


def test_language_list_fp32_equals_groups():
    """A mixed language list decodes every row as decoding its language group alone does (fp32: bit for bit), through generate
    and transcribe_pcm; transcribe_pcm(language=None) detects the planted languages."""
    _cuda()
    hf, mel, targets, lang_ids = _planted_fp32("tiny")
    m = _b200(hf, torch.float32, 8)
    feats = torch.from_numpy(mel).cuda()
    mix = ["zh", "en", "zh", "ja", "en", "ja"]
    ids = m.generate(feats, max_length=MAX_LENGTH, language=mix, task="transcribe", return_prompt=True).cpu()
    assert ids[:, 1].tolist() == [hf.generation_config.lang_to_id[f"<|{c}|>"] for c in mix]
    for lang in set(mix):
        idx = [i for i, c in enumerate(mix) if c == lang]
        alone = m.generate(feats[idx], max_length=MAX_LENGTH, language=lang, task="transcribe", return_prompt=True).cpu()
        assert torch.equal(ids[idx, :alone.shape[1]], alone) and (ids[idx, alone.shape[1]:] == hf.generation_config.pad_token_id).all()
    pcm = torch.from_numpy(synth_batch(0, len(targets)))
    t0, l0, g0 = m.transcribe_pcm(pcm, MAX_LENGTH, language=None, task="transcribe", return_languages=True)
    t0, l0, g0 = t0.clone(), l0.clone(), g0.clone()
    assert g0.tolist() == targets
    t1, l1, g1 = m.transcribe_pcm(pcm, MAX_LENGTH, language=_names(hf, targets), task="transcribe", return_languages=True)
    assert torch.equal(t0, t1) and torch.equal(l0, l1) and g1.tolist() == targets
    t2, l2 = m.transcribe_pcm(pcm, MAX_LENGTH, language=None, task="transcribe")
    assert torch.equal(t0, t2) and torch.equal(l0, l2)
    m.close()


def test_detect_language_api_fp32():
    """detect_language(input_features=...) and (encoder_outputs=...) agree with HF; HF's errors; the torch op needs only the handle."""
    _cuda()
    hf, mel, targets, lang_ids = _planted_fp32("micro128")
    m = _b200(hf, torch.float32, 4)          # fewer rows than clips: detect_language runs the batch in chunks
    feats = torch.from_numpy(mel)
    with torch.no_grad():
        ref = hf.detect_language(input_features=feats)
        from transformers.modeling_outputs import BaseModelOutput
        enc_hf = hf.model.encoder(feats).last_hidden_state
        assert hf.detect_language(encoder_outputs=BaseModelOutput(last_hidden_state=enc_hf)).tolist() == ref.tolist()
    got = m.detect_language(input_features=feats)
    assert got.dtype == torch.long and got.tolist() == ref.tolist() == targets
    enc = torch.cat([m.encode(feats[:4]), m.encode(feats[4:])])
    assert m.detect_language(encoder_outputs=(enc,)).tolist() == targets
    from transformers.modeling_outputs import BaseModelOutput
    assert m.detect_language(encoder_outputs=BaseModelOutput(last_hidden_state=enc)).tolist() == targets
    for kwargs in (dict(), dict(input_features=feats, encoder_outputs=BaseModelOutput(last_hidden_state=enc_hf))):
        with pytest.raises(ValueError) as e_ref:
            hf.detect_language(**kwargs)
        with pytest.raises(ValueError) as e_mine:
            m.detect_language(**kwargs)
        assert str(e_mine.value) == str(e_ref.value)
    handle = m.handle
    out = torch.ops.twb200.detect_language(handle, enc[:4].contiguous(), torch.tensor(lang_ids, dtype=torch.int32))
    assert out.dtype == torch.int32 and out.tolist() == targets[:4]
    m.close()


# ---------------------------------------------------------------------------------------------- bf16 at the benched widths
@functools.lru_cache(maxsize=None)
def _planted_lv3w(n=192):
    from taiwan_whisper_b200.host import B200WhisperFeatureExtractor
    hf = perturb_hf_model(hf_ref.build_hf_model(SHAPES["lv3w"], seed=1234))
    # a random decoder's step-0 state moves with the audio by ~0.1 %, below bf16's resolution: sharper cross-attention (queries
    # x 100) with a larger share of the residual (output projection x 8) spreads the clips' states by several per cent
    with torch.no_grad():
        for layer in hf.model.decoder.layers:
            layer.encoder_attn.q_proj.weight.mul_(100.0)
            layer.encoder_attn.q_proj.bias.mul_(100.0)
            layer.encoder_attn.out_proj.weight.mul_(8.0)
    pcm = synth_batch(0, n)
    feats = B200WhisperFeatureExtractor(feature_size=128)(torch.from_numpy(pcm), return_tensors="pt")["input_features"]
    states = step0_states(hf, feats, device="cuda")
    targets = target_languages(hf, n)
    lang_ids = plant_languages(hf, states, targets, BF16_MARGIN)
    # the bf16 model holds the planted rows rounded to bf16: so does the fp32 reference, and its margins are those of the rounded rows
    with torch.no_grad():
        E = hf.model.decoder.embed_tokens.weight
        E[lang_ids] = E[lang_ids].bfloat16().float()
    E = E.detach().double().numpy()[lang_ids]
    s = np.sort(states @ E.T, axis=1)
    # the planted rows are long and nearly parallel: generated steps would often face near-ties between language tokens, where the
    # split-K atomics of the bf16 residual GEMMs decide.  Generation suppresses them (detection does not read the masks).
    hf.generation_config.suppress_tokens = sorted(set(hf.generation_config.suppress_tokens) | set(lang_ids))
    return hf, pcm, feats, targets, lang_ids, s[:, -1] - s[:, -2]


def _check_bf16_languages(langs, targets, margins):
    sure = margins >= BF16_BAR
    assert sure.sum() >= 0.9 * len(targets), np.sort(margins)[:10]
    bad = [(i, int(langs[i]), int(targets[i]), float(margins[i])) for i in np.flatnonzero(sure) if langs[i] != targets[i]]
    assert len(bad) <= BF16_MISS * sure.sum(), bad
    assert len(set(np.asarray(langs)[sure].tolist())) >= 4


def _same_rows(a, b):
    """Rows of a and b (token tensors [B, n], or lengths [B]) that are equal; at least BF16_SAME of them."""
    a, b = a.reshape(a.shape[0], -1), b.reshape(b.shape[0], -1)
    same = (a == b).all(1)
    assert same.float().mean().item() >= BF16_SAME, torch.nonzero(~same).flatten().tolist()


def test_detection_changes_nothing_else_bf16_b64():
    """lv3w bf16, B = 64: a language=None decode is the decode of the detected languages given as a per-row list (same B, same
    K|V row split; row for row bitwise up to the run-to-run near-ties of BF16_SAME), and the detected ids are the planted fp32
    languages where the fp32 margin is at least BF16_BAR (up to BF16_MISS).  A mixed list equals, row for row, the replay of each
    of its languages over the whole batch."""
    _cuda()
    hf, pcm, feats, targets, lang_ids, margins = _planted_lv3w()
    m = _b200(hf, torch.bfloat16, 64)
    f = feats[:64].cuda()
    enc = m.encode(f)
    det = m._row_prompts(None, "transcribe", False, 64)
    t0, l0, g0 = m.decode_rows(enc, det, MAX_LENGTH, False)
    _check_bf16_languages(g0.tolist(), targets[:64], margins[:64])
    t1, l1, g1 = m.decode_rows(enc, m._row_prompts(_names(hf, g0.tolist()), "transcribe", False, 64), MAX_LENGTH, False)
    assert torch.equal(g0, g1)
    _same_rows(t0, t1)
    _same_rows(l0, l1)
    ids_none = m.generate(f, max_length=MAX_LENGTH, task="transcribe", return_prompt=True)
    ids_list = m.generate(f, max_length=MAX_LENGTH, language=_names(hf, g0.tolist()), task="transcribe", return_prompt=True)
    assert ids_none[:, 1].tolist() == g0.tolist() == ids_list[:, 1].tolist()
    w = min(ids_none.shape[1], ids_list.shape[1])
    _same_rows(ids_none[:, :w], ids_list[:, :w])
    mix = [("zh", "en", "ja", "ko")[i % 4] for i in range(64)]
    tm, lm, gm = m.decode_rows(enc, m._row_prompts(mix, "transcribe", False, 64), MAX_LENGTH, False)
    replay_t, replay_l = torch.empty_like(tm), torch.empty_like(lm)
    for lang in set(mix):
        idx = [i for i, c in enumerate(mix) if c == lang]
        tr, lr, _ = m.decode_rows(enc, m._row_prompts(lang, "transcribe", False, 64), MAX_LENGTH, False)
        replay_t[idx], replay_l[idx] = tr[idx], lr[idx]
    _same_rows(tm, replay_t)
    _same_rows(lm, replay_l)
    m.close()


def test_detection_merged_decode_bf16_192():
    """transcribe_batches(merge=3) over 3 x 64 clips of planted mixed languages (192 merged rows): language=None is bitwise the run
    with the detected languages given per batch as per-row lists (up to BF16_SAME), and detects the planted languages."""
    _cuda()
    hf, pcm, feats, targets, lang_ids, margins = _planted_lv3w()
    m = _b200(hf, torch.bfloat16, 192)
    try:
        m.enable_pipeline(24)
    except NotImplementedError as e:
        pytest.skip(f"no green contexts: {e}")
    batches = [torch.from_numpy(pcm[i:i + 64]).pin_memory() for i in range(0, 192, 64)]

    def run(language):
        out = list(m.transcribe_batches(batches, MAX_LENGTH, language=language, task="transcribe", merge=3, return_languages=True))
        assert len(out) == 3
        return [torch.cat([o[k].clone() for o in out]) for k in range(3)]

    t0, l0, g0 = run(None)
    _check_bf16_languages(g0.tolist(), targets, margins)
    names = _names(hf, g0.tolist())
    t1, l1, g1 = run([names[i:i + 64] for i in range(0, 192, 64)])
    assert torch.equal(g0, g1)
    _same_rows(t0, t1)
    _same_rows(l0, l1)
    m.close()
