"""-m gpu parity at the BENCHED widths and batch sizes (VERDICT r1 item N2): large-v3 width (d 1280 / 20 heads / ffn 5120 /
V 51866 / 128 mel) at B = 64, max_length 256, and medium width (d 1024 / 16 heads / V 51865 / 80 mel) at B = 32 with the
timestamp rules and max_length 448 (ref prefiltering/validator_inference.py:41-47) — 2 + 2 layers so that the numpy oracle
finishes in seconds, every other dimension as benched: the M = 96 000 tcgen05 GEMMs with the TMA store / reduce-add
epilogues, split-K skinny GEMMs at K = 5120, the 64-row page-major cache, the 148-CTA K|V stream across clip boundaries.

fp32 check mode: ids bit-identical to the oracle on sampled rows of the batch (first, second, middle, last).
bf16: scored teacher-forced on EVERY position of the sampled rows against the fp32 ids, next to HF's own bf16 forward
(cuda, same weights, same positions): our disagreements must not exceed HF-bf16's by more than a small slack.
"""
import numpy as np
import pytest
import torch

from taiwan_whisper_b200.configs import SHAPES, token_ids
from tests.helpers import PERTURBED, default_rules, perturb_hf_model, prompt_ids, split_shape, weights_np

pytestmark = pytest.mark.gpu


def _cuda():
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the -m gpu tests must run on a B200 (there is no CPU fallback)")


_CACHE = {}


def _setup(shape_name, B, max_length, timestamps, rows):
    """batch of B distinct synthetic clips; oracle (numpy) tokens for the sampled rows"""
    key = (shape_name, B, max_length, timestamps, tuple(rows))
    if key in _CACHE:
        return _CACHE[key]
    from oracle import hf_ref, logmel_np, whisper_np
    from taiwan_whisper_b200.synth import dequantise, synth_batch
    shape_name, perturb = split_shape(shape_name)
    sh = SHAPES[shape_name]
    hf = hf_ref.build_hf_model(sh, seed=1234)
    if perturb:
        perturb_hf_model(hf)
    W = weights_np(hf)
    pcm = synth_batch(0, B)
    mel_rows = logmel_np.log_mel(dequantise(pcm[list(rows)]), sh.n_mel)
    P = prompt_ids(sh.vocab, timestamps)
    rules = default_rules(sh.vocab, timestamps)
    ora = []
    for i in range(len(rows)):
        enc = whisper_np.encoder_forward(W, mel_rows[i], sh.heads, sh.enc_layers)
        lt = []
        toks = whisper_np.greedy_decode(W, enc, P, rules, max_length, sh.heads, sh.dec_layers, logits_tap=lt)
        ora.append(dict(enc=enc, tokens=toks, logits=lt))
    _CACHE[key] = (hf, pcm, mel_rows, P, rules, ora)
    return _CACHE[key]


def _b200(hf, dtype, B):
    from taiwan_whisper_b200.host import B200WhisperForConditionalGeneration
    return B200WhisperForConditionalGeneration.from_hf(hf, dtype=dtype, max_batch=B, output_layout="5.x")


CASES = [("lv3w", 64, 256, False, (0, 1, 37, 63)), ("medw", 32, 448, True, (0, 17, 31))]


@pytest.mark.parametrize("shape_name,B,max_length,timestamps,rows", CASES + [("lv3w" + PERTURBED, 64, 256, False, (0, 1, 37, 63))])
def test_benched_width_fp32_bit_identical(shape_name, B, max_length, timestamps, rows):
    _cuda()
    from taiwan_whisper_b200.host import log_mel
    sh = SHAPES[split_shape(shape_name)[0]]
    hf, pcm, mel_rows, P, rules, ora = _setup(shape_name, B, max_length, timestamps, rows)
    m = _b200(hf, torch.float32, B)
    try:
        mel = log_mel(torch.from_numpy(pcm).cuda(), None, sh.n_mel)
        assert np.abs(mel[list(rows)].cpu().numpy() - mel_rows).max() < 1e-4
        enc = m.encode(mel)
        for i, r in enumerate(rows):
            ref = ora[i]["enc"]
            err = np.abs(enc[r].cpu().numpy() - ref).max() / np.abs(ref).max()
            assert err < 1e-4, (r, err)
        toks, lens = m.decode(enc, P, max_length, timestamps)
        toks, lens = toks.cpu().numpy(), lens.cpu().numpy()
        for i, r in enumerate(rows):
            ref = ora[i]["tokens"]
            assert lens[r] == len(ref), (r, lens[r], len(ref))
            assert toks[r, :len(ref)].tolist() == ref, (r, int(np.argmax(toks[r, :len(ref)] != np.asarray(ref))))
        # rows that are not sampled ran through the same launches: sanity only (valid ids, full length for random-init)
        assert (toks >= 0).all() and (toks < sh.vocab).all()
    finally:
        m.close()


@pytest.mark.parametrize("shape_name,B,max_length,timestamps,rows", CASES)
def test_benched_width_bf16_vs_hf_bf16(shape_name, B, max_length, timestamps, rows):
    _cuda()
    from oracle import hf_ref
    from taiwan_whisper_b200.host import log_mel
    sh = SHAPES[shape_name]
    hf, pcm, mel_rows, P, rules, ora = _setup(shape_name, B, max_length, timestamps, rows)
    n_gen = max_length - len(P)
    n_min = min(len(o["tokens"]) for o in ora)
    assert n_min == n_gen, "random-init rows run to the budget"
    m = _b200(hf, torch.bfloat16, B)
    try:
        mel = log_mel(torch.from_numpy(pcm).cuda(), None, sh.n_mel)
        enc = m.encode(mel)
        for i, r in enumerate(rows):             # bf16 encoder output at the benched width: 2e-2 relative L2
            ref = ora[i]["enc"]
            rel = np.linalg.norm(enc[r].float().cpu().numpy() - ref) / np.linalg.norm(ref)
            assert rel < 2e-2, (r, rel)
        # teacher forcing: sampled rows get the oracle's fp32 ids, the others a free-running first pass of this model
        free, _ = m.decode(enc, P, max_length, timestamps)
        forced = free.clone()
        for i, r in enumerate(rows):
            forced[r] = torch.tensor(ora[i]["tokens"], dtype=torch.int32)
        toks, _ = m.decode(enc, P, max_length, timestamps, forced=forced)
        toks = toks.cpu().numpy()
    finally:
        m.close()
    ref = np.asarray([o["tokens"] for o in ora])
    ours_dis = int((toks[list(rows)] != ref).sum())
    hf_ids = hf_ref.hf_teacher_forced_argmax(hf, mel_rows, P, ref, rules, device="cuda", dtype=torch.bfloat16)
    hf_dis = int((hf_ids != ref).sum())
    total = ref.size
    # positions with a solid fp32 margin must agree (the 99.5 % bar of north_star); all positions: no worse than HF bf16
    solid = solid_ok = 0
    for i in range(len(rows)):
        for s in range(n_gen):
            lg = ora[i]["logits"][s]
            top2 = np.partition(lg[np.isfinite(lg)], -2)[-2:]
            if top2[1] - top2[0] > 0.02:
                solid += 1
                solid_ok += int(toks[rows[i], s] == ref[i, s])
    print(f"{shape_name}: bf16 teacher-forced disagreements ours {ours_dis}/{total}, HF bf16 {hf_dis}/{total}; "
          f"fp32-margin>0.02: {solid_ok}/{solid}")
    assert solid > 0 and solid_ok / solid >= 0.995
    assert ours_dis <= hf_dis + max(4, hf_dis // 2), (ours_dis, hf_dis, total)


@pytest.mark.parametrize("B,dtype_name", [(70, "f32"), (130, "f32"), (70, "bf16"), (130, "bf16"), (260, "bf16")])
def test_decode_batches_beyond_64(B, dtype_name):
    """B > 64: the skinny GEMM runs 2-4 row blocks (fused cache append through the page table for every row block) up to 256
    rows and the general GEMM with a separate append kernel beyond: the K|V rows must reach the paged cache either way
    (ADVICE r1: the BN=256 tile ignored the column split).  tiny, distinct clips, sampled rows vs the oracle."""
    _cuda()
    from taiwan_whisper_b200.host import log_mel
    sh = SHAPES["tiny"]
    rows = (0, 64, B - 1)
    max_length = 20
    hf, pcm, mel_rows, P, rules, ora = _setup("tiny", B, max_length, False, rows)
    dtype = {"f32": torch.float32, "bf16": torch.bfloat16}[dtype_name]
    m = _b200(hf, dtype, B)
    try:
        mel = log_mel(torch.from_numpy(pcm).cuda(), None, sh.n_mel)
        enc = m.encode(mel)
        ref = np.asarray([o["tokens"] for o in ora])
        if dtype_name == "f32":
            toks, lens = m.decode(enc, P, max_length, False)
            toks = toks.cpu().numpy()
            for i, r in enumerate(rows):
                assert toks[r].tolist() == ref[i].tolist(), r
        else:
            free, _ = m.decode(enc, P, max_length, False)
            forced = free.clone()
            for i, r in enumerate(rows):
                forced[r] = torch.tensor(ref[i], dtype=torch.int32)
            toks, _ = m.decode(enc, P, max_length, False, forced=forced)
            toks = toks.cpu().numpy()
            solid = ok = 0
            for i, r in enumerate(rows):
                for s in range(ref.shape[1]):
                    lg = ora[i]["logits"][s]
                    top2 = np.partition(lg[np.isfinite(lg)], -2)[-2:]
                    if top2[1] - top2[0] > 0.02:
                        solid += 1
                        ok += int(toks[r, s] == ref[i, s])
            assert solid > 0 and ok == solid, (ok, solid)
    finally:
        m.close()


# ---------------------------------------------------------------------------------------- EOS / finished rows
def _eos_model(shape_name, scale, seed):
    """random-init never emits EOS (its embedding row is the zeroed padding_idx): give <|endoftext|> a random embedding of
    `scale` x the init std so that it wins at different steps for different clips (found with the oracle)."""
    import copy
    from oracle import hf_ref
    sh = SHAPES[shape_name]
    hf = copy.deepcopy(hf_ref.build_hf_model(sh, seed=1234))
    eos = token_ids(sh.vocab).eos
    vec = np.random.default_rng(seed).normal(0, 0.02 * scale, sh.d_model).astype(np.float32)
    with torch.no_grad():
        hf.model.decoder.embed_tokens.weight[eos] = torch.from_numpy(vec)
    return hf


@pytest.mark.parametrize("scale,seed,expect", [(6.0, 7, "ragged"), (5.5, 9, "all_early")])
@pytest.mark.parametrize("graph", [True, False])
def test_eos_finished_rows_fp32(scale, seed, expect, graph, monkeypatch):
    """EOS / finished-row path on the production step (CUDA graph replay and plain launches): rows that emit EOS at different
    steps, pad emission afterwards, out_lengths at the EOS position, the asynchronous all-finished read-back with its
    early exit and the pad fill of the unwritten tail — ids, lengths and padding equal to the oracle, twice (second call
    replays the cached graph)."""
    _cuda()
    from oracle import logmel_np, whisper_np
    from taiwan_whisper_b200.host import B200WhisperForConditionalGeneration
    from taiwan_whisper_b200.synth import dequantise, synth_batch
    shape_name, n, max_length = "micro128", 5, 48
    sh = SHAPES[shape_name]
    ids = token_ids(sh.vocab)
    hf = _eos_model(shape_name, scale, seed)
    W = weights_np(hf)
    pcm = synth_batch(0, n)
    mel = logmel_np.log_mel(dequantise(pcm), sh.n_mel)
    P, rules = prompt_ids(sh.vocab, False), default_rules(sh.vocab, False)
    ref = [whisper_np.greedy_decode(W, whisper_np.encoder_forward(W, mel[b], sh.heads, sh.enc_layers), P, rules, max_length,
                                    sh.heads, sh.dec_layers) for b in range(n)]
    n_gen = max_length - len(P)
    lens_ref = [len(r) for r in ref]
    if expect == "ragged":
        assert len(set(lens_ref)) > 1 and max(lens_ref) == n_gen and min(lens_ref) < n_gen - 8, lens_ref
    else:
        assert max(lens_ref) < n_gen - 16, lens_ref          # every row finishes early: the early exit must fire
    monkeypatch.setenv("TWB200_GRAPH", "1" if graph else "0")
    m = B200WhisperForConditionalGeneration.from_hf(hf, dtype=torch.float32, max_batch=n, output_layout="5.x")
    try:
        enc = m.encode(torch.from_numpy(mel).cuda())
        for call in range(2):
            toks, lens = m.decode(enc, P, max_length, False)
            toks, lens = toks.cpu().numpy(), lens.cpu().numpy()
            assert lens.tolist() == lens_ref, (call, lens.tolist(), lens_ref)
            for b in range(n):
                assert toks[b, :lens_ref[b]].tolist() == ref[b], (call, b)
                # HF: the EOS itself then pad for finished rows (generation/utils.py:2793-2805); pad == eos here
                assert (toks[b, lens_ref[b]:] == ids.pad).all(), (call, b, toks[b].tolist())
        out = m.generate(torch.from_numpy(mel), max_length=max_length, num_beams=1, return_timestamps=False, language="zh",
                         task="transcribe").numpy()
        assert out.shape == (n, max(lens_ref))
        for b in range(n):
            assert out[b, :lens_ref[b]].tolist() == ref[b] and (out[b, lens_ref[b]:] == ids.pad).all()
        # the fused host-buffer entry point shares the loop
        pt, pl = m.transcribe_pcm(torch.from_numpy(pcm), max_length)
        assert pl.tolist() == lens_ref
        for b in range(n):
            assert pt[b, :lens_ref[b]].tolist() == ref[b] and (pt[b, lens_ref[b]:] == ids.pad).all()
    finally:
        m.close()


def test_eos_finished_rows_bf16_structure():
    """bf16 production path with rows finishing at different steps: structural invariants (no id after a row's length except
    pad, lengths within budget, lengths mostly equal to the fp32 oracle's) on the graph-replayed step."""
    _cuda()
    from oracle import logmel_np, whisper_np
    from taiwan_whisper_b200.host import B200WhisperForConditionalGeneration
    from taiwan_whisper_b200.synth import dequantise, synth_batch
    shape_name, n, max_length = "micro128", 5, 48
    sh = SHAPES[shape_name]
    ids = token_ids(sh.vocab)
    hf = _eos_model(shape_name, 6.0, 7)
    pcm = synth_batch(0, n)
    mel = logmel_np.log_mel(dequantise(pcm), sh.n_mel)
    P = prompt_ids(sh.vocab, False)
    n_gen = max_length - len(P)
    m = B200WhisperForConditionalGeneration.from_hf(hf, dtype=torch.bfloat16, max_batch=n, output_layout="5.x")
    try:
        enc = m.encode(torch.from_numpy(mel).cuda())
        for call in range(2):
            toks, lens = m.decode(enc, P, max_length, False)
            toks, lens = toks.cpu().numpy(), lens.cpu().numpy()
            assert ((lens >= 0) & (lens <= n_gen)).all()
            for b in range(n):
                assert (toks[b, :lens[b]] != ids.eos).all()
                assert (toks[b, lens[b]:] == ids.pad).all(), (b, toks[b].tolist())
            assert len(set(lens.tolist())) > 1, lens.tolist()          # some rows finish, some run to the budget
    finally:
        m.close()


@pytest.mark.parametrize("dtype_name", ["f32", "bf16"])
def test_row_budgets_prefix_property_benched_width(dtype_name):
    """Finished-row path at the benched width and batch (large-v3 width, B = 64, max_length 256): rows are given ragged token
    budgets (tw_debug_set_row_budgets: the row ends as if EOS followed); every row must reproduce the first budget[b] ids
    of the unconstrained run — finished clips leave the K|V stream's active list without disturbing the others — then pad;
    lengths == budgets; a second batch where every row stops early takes the early exit."""
    _cuda()
    from taiwan_whisper_b200.host import log_mel
    shape_name, B, max_length = "lv3w", 64, 256
    sh = SHAPES[shape_name]
    ids = token_ids(sh.vocab)
    hf, pcm, mel_rows, P, rules, ora = _setup(shape_name, B, max_length, False, (0, 1, 37, 63))
    n_gen = max_length - len(P)
    rng = np.random.default_rng(3)
    budgets = rng.integers(1, n_gen + 1, size=B)
    budgets[0], budgets[1], budgets[63] = n_gen, 1, 17
    m = _b200(hf, {"f32": torch.float32, "bf16": torch.bfloat16}[dtype_name], B)
    try:
        mel = log_mel(torch.from_numpy(pcm).cuda(), None, sh.n_mel)
        enc = m.encode(mel)
        full, full_len = m.decode(enc, P, max_length, False)
        full = full.cpu().numpy()
        assert (full_len.cpu().numpy() == n_gen).all()
        # bf16: the K|V stream splits its rows over the CTAs by the number of active clips, so partial sums merge in another
        # order once a clip has finished and a free-running row can take the other side of a near-tie (and then diverges for
        # good).  The prefix property is therefore checked teacher-forced in bf16 (the unconstrained run's ids are fed back),
        # exactly (free-running) in fp32 check mode.
        forced = None if dtype_name == "f32" else torch.from_numpy(full.astype(np.int32))
        if forced is not None:
            base, _ = m.decode(enc, P, max_length, False, forced=forced)
            base = base.cpu().numpy()
        else:
            base = full
        for bud in (budgets, np.minimum(budgets, 40)):
            m.set_row_budgets(bud.tolist())
            for call in range(2):
                toks, lens = m.decode(enc, P, max_length, False, forced=forced)
                toks, lens = toks.cpu().numpy(), lens.cpu().numpy()
                assert lens.tolist() == bud.tolist()
                bad = 0
                for b in range(B):
                    assert (toks[b, bud[b]:] == ids.pad).all(), b
                    bad += int((toks[b, :bud[b]] != base[b, :bud[b]]).sum())
                if dtype_name == "f32":
                    assert bad == 0
                else:
                    assert bad <= 0.005 * bud.sum(), (bad, int(bud.sum()))
                if forced is not None and call == 0:        # the production (graph-replayed) bf16 step with budgets: structure only
                    ft, fl = m.decode(enc, P, max_length, False)
                    ft, fl = ft.cpu().numpy(), fl.cpu().numpy()
                    assert fl.tolist() == bud.tolist()
                    for b in range(B):
                        assert (ft[b, bud[b]:] == ids.pad).all() and (ft[b, :bud[b]] < sh.vocab).all()
            m.set_row_budgets(None)
        again, _ = m.decode(enc, P, max_length, False)
        if dtype_name == "f32":
            assert np.array_equal(again.cpu().numpy(), full)
    finally:
        m.close()


# ---------------------------------------------------------------------------------------- call-site replay
def test_call_site_replay_validator_and_pseudo_labelling():
    """The exact statement sequences of the two reference call sites, run once against the HF objects and once against the
    swapped B200 objects on the same inputs and weights:
      ref prefiltering/validator_inference.py:55-87  fe(list, sampling_rate=16000) -> fe.pad(..., return_tensors="pt") ->
                                                     model.generate(batch["input_features"], max_length=448, num_beams=1,
                                                                    return_timestamps=True, language='zh', task='transcribe')
      ref training/run_pseudo_labelling.py:864-918   gen_kwargs {max_length, num_beams, return_timestamps, language, task};
                                                     generate_fn(batch["input_features"].to(dtype=torch_dtype), **gen_kwargs)
    and the reference's own post-processing of the ids (filter_eot_tokens :837-843, add_concatenated_text :1003-1012) on the
    4.45-layout output."""
    _cuda()
    from oracle import hf_ref
    from taiwan_whisper_b200.host import B200WhisperFeatureExtractor, B200WhisperForConditionalGeneration
    from taiwan_whisper_b200.synth import dequantise, synth_batch
    sh = SHAPES["tiny"]
    tid = token_ids(sh.vocab)
    hf = hf_ref.build_hf_model(sh, seed=1234)
    hf_fe = hf_ref.build_hf_feature_extractor(sh.n_mel)
    arrays = [a[: 480000 - 1234 * i] for i, a in enumerate(dequantise(synth_batch(0, 3)))]       # ragged lengths, float32
    features = [{"idx": 10 + i, "array": a} for i, a in enumerate(arrays)]

    # ---- validator_inference.py collate_fn + generate, statement for statement
    def validator(fe, model, max_length):
        gen_kwargs = {"max_length": max_length, "num_beams": 1, "return_timestamps": True, "language": 'zh', "task": 'transcribe'}
        inputs = fe([feature['array'] for feature in features], sampling_rate=16000)
        input_features = {'input_features': inputs.input_features}
        batch = fe.pad(input_features, padding="longest", return_tensors="pt")
        batch['idx'] = torch.from_numpy(np.array([feature['idx'] for feature in features])).long().to(batch['input_features'].device)
        with torch.no_grad():
            output_ids = model.generate(batch["input_features"], **gen_kwargs)
        return batch['idx'].cpu().numpy(), output_ids

    max_length = 40
    idx_hf, ids_hf = validator(hf_fe, hf, max_length)
    m5 = B200WhisperForConditionalGeneration.from_hf(hf, dtype=torch.float32, max_batch=4, output_layout="5.x")
    m445 = B200WhisperForConditionalGeneration.from_hf(hf, dtype=torch.float32, max_batch=4)          # default: the reference's pin
    try:
        for fe in (B200WhisperFeatureExtractor.from_hf(hf_fe), B200WhisperFeatureExtractor(feature_size=sh.n_mel, keep_on_device=True)):
            idx_b, ids_b = validator(fe, m5, max_length)
            assert idx_b.tolist() == idx_hf.tolist() == [10, 11, 12]
            assert ids_b.shape == ids_hf.shape and torch.equal(ids_b.cpu(), ids_hf.cpu()), (ids_b.tolist(), ids_hf.tolist())
        # keep_on_device: the features never left the GPU between fe() and generate()
        fe_dev = B200WhisperFeatureExtractor(feature_size=sh.n_mel, keep_on_device=True)
        inputs = fe_dev([f['array'] for f in features], sampling_rate=16000)
        assert all(t.is_cuda for t in inputs.input_features)
        assert fe_dev.pad({'input_features': inputs.input_features}, padding="longest", return_tensors="pt")["input_features"].is_cuda

        # ---- run_pseudo_labelling.py: gen_kwargs as built at :864-876, call as at :917-918
        def pseudo_label(model, feats, torch_dtype, return_timestamps):
            gen_kwargs = {"max_length": max_length, "num_beams": getattr(model.generation_config, "num_beams", 1),
                          "return_timestamps": return_timestamps}
            if hasattr(model.generation_config, "is_multilingual") and model.generation_config.is_multilingual:
                gen_kwargs.update({"language": "zh", "task": "transcribe"})
            model.generation_config.forced_decoder_ids = None
            model.config.forced_decoder_ids = None
            generate_fn = model.generate
            return generate_fn(feats.to(dtype=torch_dtype), **gen_kwargs)

        feats_pt = hf_fe.pad({"input_features": hf_fe(arrays, sampling_rate=16000).input_features}, padding="longest", return_tensors="pt")["input_features"]
        for ts in (False, True):
            g_hf = pseudo_label(hf, feats_pt, torch.float32, ts)
            g_b = pseudo_label(m5, feats_pt, torch.float32, ts)
            assert torch.equal(g_b.cpu(), g_hf.cpu()), ts
            # the 4.45 layout the reference's code slices: forced prompt first, one pass per window
            g_445 = pseudo_label(m445, feats_pt, torch.float32, ts).cpu().numpy()
            prompt = [tid.sot, tid.lang_to_id["<|zh|>"], tid.transcribe] + ([] if ts else [tid.notimestamps])
            assert (g_445[:, :len(prompt)] == np.asarray(prompt)).all()
            single = m5.generate(feats_pt, max_length=max_length, num_beams=1, return_timestamps=ts, language="zh", task="transcribe",
                                 seek_loop=False).cpu().numpy()
            assert np.array_equal(g_445[:, len(prompt):], single)
            # ref :837-843 filter_eot_tokens and :1003-1012 add_concatenated_text on that output
            decoder_eot_token_id, decoder_prev_token_id, timestamp_position = tid.eos, tid.startofprev, 3
            eval_preds = [row.tolist() for row in g_445]
            for token_ids_row, gen_row in zip(eval_preds, single):
                no_eot = [t for t in token_ids_row if t != decoder_eot_token_id]
                prompt_ids_ = [decoder_prev_token_id] + no_eot[timestamp_position:]
                expect = ([] if ts else [tid.notimestamps]) + [int(t) for t in gen_row if t != decoder_eot_token_id]
                assert prompt_ids_ == [decoder_prev_token_id] + expect
    finally:
        m5.close()
        m445.close()


def test_longform_config5_end_to_end():
    """Config 5 end to end on one recording (75 s -> 4 windows of 30 s, hop 20 s): every window's timestamp-mode ids equal the
    oracle's on the zero-padded window (fp32 check mode), and the stitched chunks equal HF `_decode_asr(...,
    return_timestamps=True)` on those per-window ids (ref training/flax/distil_whisper/pipeline.py:353-375)."""
    _cuda()
    import torch as _t
    from transformers.models.whisper.tokenization_whisper import _decode_asr
    from oracle import hf_ref, logmel_np, whisper_np
    from taiwan_whisper_b200.host import B200WhisperForConditionalGeneration
    from taiwan_whisper_b200.longform import chunk_plan, transcribe_longform
    from taiwan_whisper_b200.synth import dequantise, synth_batch
    from tests.helpers import StubWhisperTokenizer
    sh = SHAPES["tiny"]
    tid = token_ids(sh.vocab)
    hf = hf_ref.build_hf_model(sh, seed=1234)
    W = weights_np(hf)
    rec = np.concatenate(list(synth_batch(0, 3)))[: 16000 * 75]
    max_length = 40
    m = B200WhisperForConditionalGeneration.from_hf(hf, dtype=torch.float32, max_batch=3, output_layout="5.x")     # 4 windows: two batches
    try:
        tok = StubWhisperTokenizer(tid)
        chunks = transcribe_longform(m, torch.from_numpy(rec).cuda(), max_length=max_length, special_ids=tok.all_special_ids)
    finally:
        m.close()
    # encoder batches of 2 windows, both decoded together (merged decode): the same chunks
    m = B200WhisperForConditionalGeneration.from_hf(hf, dtype=torch.float32, max_batch=4, output_layout="5.x")
    try:
        merged = transcribe_longform(m, torch.from_numpy(rec).cuda(), max_length=max_length, special_ids=tok.all_special_ids,
                                     batch_size=2, merge=2)
    finally:
        m.close()
    assert [(c["timestamp"], c["tokens"]) for c in merged] == [(c["timestamp"], c["tokens"]) for c in chunks]
    starts, strides = chunk_plan(len(rec))
    assert len(starts) == 4 and strides[0][1] == 0 and strides[-1][2] == 0
    P, rules = prompt_ids(sh.vocab, True), default_rules(sh.vocab, True)
    outs = []
    for s0, st in zip(starts, strides):
        win = np.zeros(480000, np.int16)
        win[: st[0]] = rec[s0:s0 + st[0]]
        mel = logmel_np.log_mel(dequantise(win[None]), sh.n_mel)[0]
        ids = whisper_np.greedy_decode(W, whisper_np.encoder_forward(W, mel, sh.heads, sh.enc_layers), P, rules, max_length, sh.heads,
                                       sh.dec_layers)
        outs.append({"tokens": _t.tensor([ids]), "stride": (st[0] / 16000, st[1] / 16000, st[2] / 16000)})
    text, opt = _decode_asr(tok, outs, return_timestamps=True, return_language=False, time_precision=0.02)
    assert [c["timestamp"] for c in chunks] == [c["timestamp"] for c in opt["chunks"]]
    assert [tok.decode(c["tokens"]) for c in chunks] == [c["text"] for c in opt["chunks"]]
    assert len(chunks) > 0
