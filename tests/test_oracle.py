"""CPU: pins the numpy restatement (oracle/) against the committed golden fixtures, which
tests/golden/make_golden.py produced from the reference's own implementation (HF transformers),
and against HF live (it is in the image)."""
import os

import numpy as np
import pytest

from oracle import hf_ref, logmel_np, whisper_np
from taiwan_whisper_b200.configs import SHAPES, token_ids
from taiwan_whisper_b200.synth import dequantise, edge_case_clips, synth_batch
from tests.helpers import default_rules, perturb_hf_model, prompt_ids, weights_np

LOGMEL_TOL = 1e-4          # north_star: log-mel within 1e-4 abs


def _clips():
    clips = {f"synth{i}": c for i, c in enumerate(synth_batch(0, 2))}
    clips.update(edge_case_clips())
    return clips


@pytest.mark.parametrize("n_mel", [80, 128])
def test_logmel_oracle_vs_golden(golden_dir, n_mel):
    g = np.load(os.path.join(golden_dir, f"logmel_{n_mel}.npz"))
    for name, pcm in _clips().items():
        f = logmel_np.log_mel(dequantise(pcm), n_mel)
        assert f.shape == (n_mel, 3000) and f.dtype == np.float32
        assert np.abs(f[:, ::16] - g[name + "_sub"]).max() < LOGMEL_TOL, name
        st = g[name + "_stats"]
        assert abs(f.astype(np.float64).sum() - st[0]) < 1e-4 * f.size
        assert abs(f.min() - st[2]) < LOGMEL_TOL and abs(f.max() - st[3]) < LOGMEL_TOL


def test_logmel_silence_is_minus_1p5():
    f = logmel_np.log_mel(np.zeros(480000, np.float32), 128)
    assert np.all(f == np.float32(-1.5))


def test_mel_filter_bank_matches_hf():
    for n_mel in (80, 128):
        fe = hf_ref.build_hf_feature_extractor(n_mel)
        assert np.array_equal(fe.mel_filters, logmel_np.mel_filter_bank(n_mel))
        nz = (logmel_np.mel_filter_bank(n_mel) > 0).sum(0)
        assert nz.max() <= 16      # sparse: few taps per filter


def test_logmel_live_vs_hf():
    pcm = dequantise(synth_batch(5, 1, seed=2))
    fe = hf_ref.build_hf_feature_extractor(128)
    assert np.abs(hf_ref.hf_features(fe, pcm) - logmel_np.log_mel(pcm, 128)).max() < LOGMEL_TOL


def test_pad_or_trim():
    x = np.ones(1000, np.float32)
    y = logmel_np.pad_or_trim(x)
    assert y.shape == (480000,) and y[:1000].sum() == 1000 and y[1000:].sum() == 0
    assert logmel_np.pad_or_trim(np.ones(500000, np.float32)).shape == (480000,)


def test_sinusoids_match_hf_buffer():
    m = hf_ref.build_hf_model("micro80")
    w = m.state_dict()["model.encoder.embed_positions.weight"].numpy()
    # HF builds the table in fp32 (large arguments lose ~1e-4); the path reads the stored table
    assert np.abs(whisper_np.sinusoids(1500, 128) - w).max() < 2e-4


@pytest.mark.parametrize("shape_name", ["tiny", "micro128"])
def test_model_oracle_vs_golden(golden_dir, shape_name):
    g = np.load(os.path.join(golden_dir, f"model_{shape_name}.npz"))
    sh = SHAPES[shape_name]
    W = weights_np(hf_ref.build_hf_model(sh, seed=1234))
    mel = logmel_np.log_mel(dequantise(synth_batch(0, 2)), sh.n_mel)
    max_length = int(g["max_length"])
    for b in range(2):
        taps = []
        enc = whisper_np.encoder_forward(W, mel[b], sh.heads, sh.enc_layers, taps)
        assert np.abs(taps[0][::50, ::8] - g["stem_sub"][b]).max() < 1e-4
        assert np.abs(taps[1][::50, ::8] - g["layer1_sub"][b]).max() < 1e-4
        assert np.abs(enc[::50, ::8] - g["enc_sub"][b]).max() < 1e-4          # fp32 check-mode tolerance
        assert abs(np.linalg.norm(enc.astype(np.float64)) - g["enc_norm"][b]) < 1e-3 * g["enc_norm"][b]
        toks = whisper_np.greedy_decode(W, enc, prompt_ids(sh.vocab), default_rules(sh.vocab), max_length,
                                        sh.heads, sh.dec_layers)
        ref = g["tokens_nots"][b]
        ref = ref[:len(toks)]
        assert toks == ref.tolist()                                          # bit-identical greedy ids
        # timestamp mode: HF 5.5 runs its seek loop; the first segment of the first window must match
        toks_ts = whisper_np.greedy_decode(W, enc, prompt_ids(sh.vocab, True), default_rules(sh.vocab, True),
                                           max_length, sh.heads, sh.dec_layers)
        ref_ts = g["tokens_ts_seekloop"][b].tolist()
        n = 0
        while n < min(len(toks_ts), len(ref_ts)) and toks_ts[n] == ref_ts[n]:
            n += 1
        tsb = token_ids(sh.vocab).timestamp_begin
        assert n >= 2 and toks_ts[0] >= tsb
        if n < min(len(toks_ts), len(ref_ts)):     # divergence only at a segment boundary (<|t|><|t|>)
            assert toks_ts[n - 1] >= tsb and toks_ts[n - 2] >= tsb


def test_rules_vs_hf_processors(golden_dir):
    from tests.golden.make_golden import rules_case_logits
    g = np.load(os.path.join(golden_dir, "rules.npz"))
    for vocab in (51865, 51866):
        ids = token_ids(vocab)
        hists = [[int(t) for t in h.split(",")] if h else [] for h in g[f"v{vocab}_hists"]]
        for i in range(len(g[f"v{vocab}_mode"])):
            ci, variant = int(g[f"v{vocab}_hist"][i]), int(g[f"v{vocab}_variant"][i])
            ts = str(g[f"v{vocab}_mode"][i]) == "ts"
            logits = rules_case_logits(vocab, ci, variant, ids.timestamp_begin)
            s = whisper_np.apply_rules(logits, hists[ci], default_rules(vocab, ts))
            mask = np.unpackbits(g[f"v{vocab}_mask"][i])[:vocab].astype(bool)
            assert np.array_equal(np.isneginf(s), mask), (vocab, i)
            assert int(np.argmax(s)) == int(g[f"v{vocab}_argmax"][i])


def test_decoder_kv_cache_equals_full_recompute():
    sh = SHAPES["micro80"]
    W = weights_np(hf_ref.build_hf_model(sh, seed=7))
    mel = logmel_np.log_mel(dequantise(synth_batch(3, 1))[0], sh.n_mel)
    enc = whisper_np.encoder_forward(W, mel, sh.heads, sh.enc_layers)
    xkv = whisper_np.cross_kv(W, enc, sh.dec_layers)
    toks = prompt_ids(sh.vocab) + [100, 200, 300]
    st = whisper_np.DecoderState(sh.dec_layers)
    full = whisper_np.decoder_forward(W, np.asarray(toks), st, xkv, sh.heads, sh.dec_layers)
    st = whisper_np.DecoderState(sh.dec_layers)
    whisper_np.decoder_forward(W, np.asarray(toks[:4]), st, xkv, sh.heads, sh.dec_layers)
    for t in toks[4:]:
        inc = whisper_np.decoder_forward(W, np.asarray([t]), st, xkv, sh.heads, sh.dec_layers)
    assert np.abs(full - inc).max() < 1e-5


@pytest.mark.parametrize("shape_name", ["tiny", "micro128"])
def test_teacher_logits_oracle_vs_golden(golden_dir, shape_name):
    """Full-sequence (teacher-forced) decoder logits of the oracle vs HF model(input_features, labels).logits
    (the teacher call of ref knowledge-distillation/run_distillation.py:1543-1577)."""
    g = np.load(os.path.join(golden_dir, f"teacher_{shape_name}.npz"))
    sh = SHAPES[shape_name]
    hf = hf_ref.build_hf_model(sh, seed=1234)
    W = weights_np(hf)
    mel = logmel_np.log_mel(dequantise(synth_batch(0, 2)), sh.n_mel)
    dec = whisper_np.shift_tokens_right(g["labels"], hf.config.pad_token_id, hf.config.decoder_start_token_id)
    assert np.array_equal(dec, g["decoder_input_ids"])
    for b in range(2):
        enc = whisper_np.encoder_forward(W, mel[b], sh.heads, sh.enc_layers)
        lg = whisper_np.teacher_logits(W, enc, dec[b], sh.heads, sh.dec_layers)
        assert lg.shape == (dec.shape[1], sh.vocab)
        assert np.abs(lg[:, ::97] - g["logits_sub"][b]).max() < 1e-4
        assert np.abs(np.linalg.norm(lg.astype(np.float64), axis=-1) - g["row_norm"][b]).max() < 1e-3
        top2 = np.sort(lg, axis=-1)[:, -2:]
        solid = (top2[:, 1] - top2[:, 0]) > 1e-3
        assert np.array_equal(lg.argmax(-1)[solid], g["argmax"][b][solid])


@pytest.mark.parametrize("shape_name", ["micro80", "micro128"])
def test_oracle_vs_hf_live_perturbed(shape_name):
    """The oracle against a live HF fp32 forward of a model with non-trivial biases and LayerNorms (perturb_hf_model): encoder
    output, cross-attention K / V of every decoder layer, teacher-forced logits at every position and the first greedy steps.
    HF's init leaves biases at 0 and LayerNorms at (1, 0); the GPU tests that compare with the oracle on perturbed models rely on
    this check."""
    import torch
    sh = SHAPES[shape_name]
    hf = perturb_hf_model(hf_ref.build_hf_model(sh, seed=1234))
    W = weights_np(hf)
    assert np.abs(W["model.encoder.layers.1.fc1.bias"]).max() > 0.1
    assert np.abs(W["model.decoder.layer_norm.weight"] - 1).max() > 0.1
    mel = logmel_np.log_mel(dequantise(synth_batch(0, 2)), sh.n_mel)
    P = prompt_ids(sh.vocab)
    rules = default_rules(sh.vocab)
    n_steps = 6

    def rel(a, b):
        return float(np.abs(np.asarray(a, np.float64) - b).max() / np.abs(b).max())

    greedy = []
    with torch.no_grad():
        hf_enc = hf.model.encoder(torch.from_numpy(mel)).last_hidden_state.numpy()
        for b in range(2):
            enc = whisper_np.encoder_forward(W, mel[b], sh.heads, sh.enc_layers)
            assert rel(enc, hf_enc[b]) < 1e-4, b
            e = torch.from_numpy(hf_enc[b:b + 1])
            for l, (k, v) in enumerate(whisper_np.cross_kv(W, hf_enc[b], sh.dec_layers)):
                att = hf.model.decoder.layers[l].encoder_attn
                assert rel(k, att.k_proj(e)[0].numpy()) < 1e-4, (b, l)
                assert rel(v, att.v_proj(e)[0].numpy()) < 1e-4, (b, l)
            toks = whisper_np.greedy_decode(W, enc, P, rules, len(P) + n_steps, sh.heads, sh.dec_layers)
            assert len(toks) == n_steps
            greedy.append(toks)
            ids = P + toks
            ref = hf(encoder_outputs=(torch.from_numpy(hf_enc[b:b + 1]),),
                     decoder_input_ids=torch.tensor([ids])).logits[0].numpy()
            lg = whisper_np.teacher_logits(W, enc, ids, sh.heads, sh.dec_layers)
            assert rel(lg, ref) < 1e-4, b
            # greedy steps: HF's argmax after the rules at every generated position is the oracle's token
            for s in range(n_steps):
                assert int(np.argmax(whisper_np.apply_rules(ref[len(P) - 1 + s], toks[:s], rules))) == toks[s], (b, s)
        hf_ids = hf_ref.hf_generate(hf, mel, len(P) + n_steps)
    for b in range(2):
        assert hf_ids[b, :n_steps].tolist() == greedy[b], (b, hf_ids[b].tolist(), greedy[b])
