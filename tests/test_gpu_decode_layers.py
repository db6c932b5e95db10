"""-m gpu: the bf16 decoder layer by layer, as the decode step (launch_step) and the teacher forward (decoder_logits_impl) compose
their kernels, against float64 references computed with torch on the GPU.

The models have non-trivial biases and LayerNorms (tests.helpers.perturb_hf_model), so a bias or LayerNorm routed to the wrong
layer or projection changes the numbers.  Every check recomputes one decoder layer from the kernel's own input, the fp32 residual
tap of the layer before (tw_debug_decode_taps / tw_debug_decoder_logits_taps), with a float64 MIRROR of the layer: the weights as
the model holds them (tests.test_gpu_encoder_stage._weights64: bf16 matrices, embedding and positions, q rows and q bias of both
attentions scaled by 0.125, K bias 0, fp32 biases and LayerNorms) and bf16 rounding exactly where the step stores bf16 (LayerNorm
outputs, qkv and the K|V cache row, both attention outputs, the cross-attention q, GELU(fc1)).  The self-attention of decode
position t reads the kernel's own cache rows 0 .. t-1 and the mirror's row t.

Per tapped position and layer: the K|V cache row the step wrote (fused or separate append, through the page table), the layer's
output residual, the embedding, and the post-rules logits.  The tapped run is also checked against production: its argmax against
the graph run's ids it was fed, and its logits against a run without layer taps.  Bitwise run-to-run equality is not asked for:
the split-K residual epilogue of the skinny GEMM adds its partials with fp32 atomics.
Every bar below is a measurement on a B200 with its margin.
"""
import ctypes as C
import functools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle.whisper_np import apply_rules
from taiwan_whisper_b200 import lib as twlib
from taiwan_whisper_b200.configs import SHAPES
from tests.gpu_common import EPS24, ulp_bf16
from tests.helpers import prompt_ids
from tests.test_gpu_encoder_stage import LN_TAU, _mel, _read, _weights64, bf, ln64, ln_scale

pytestmark = pytest.mark.gpu

# Measured on a B200 (1000 W power limit); each bar is 2-3x its measurement.
# Decoder layer l (kernel tap l vs the fp64 mirror run on tap l-1): max over the elements of a row of |tap - mirror| divided by
# the RMS of that row's layer update (tap l - tap l-1), maximised over every active row and tapped position of the shape's cases
# (lv3w: the absorbed cross-attention 1.46e-2, the K|V stream 1.25e-2).  As in the encoder (test_gpu_encoder_stage: up to 1.1e-2 at
# lv3w), what is left is fp32 accumulation order and the rare element whose bf16 rounding falls the other way.
MEASURED_LAYER_ERR = {"tiny": 4.78e-3, "micro128": 6.72e-4, "medw": 8.96e-3, "lv3w": 1.46e-2}
LAYER_ERR = {"tiny": 1.2e-2, "micro128": 2e-3, "medw": 1.8e-2, "lv3w": 3e-2}
# K|V cache row of position t (the step's fused or separate append): max over elements of (|kernel - fp64| - one bf16 ulp - the
# steps of the LayerNorm outputs the kernel may round the other way, see ln_bf16) / unit, unit = 2^-24 (sqrt(d) sum_k |xn_k w_k| +
# |ref|) with xn the mirror's bf16 LayerNorm output.  Measured 2.44e-2 (medw); without the LayerNorm term it reached 122 (micro128).
MEASURED_KV_ROW_C = 2.44e-2
KV_ROW_C = 7e-2
# Post-rules logits: the same measure for the fp32 logits over the final LayerNorm output and the embedding (K = d), finite
# entries only; the -inf sets must be identical (they were in every case, the timestamp rules of medw included).  Measured 0.195
# (micro128); without the LayerNorm term it reached 19.6 (lv3w B = 192).
MEASURED_LOGIT_C = 0.195
LOGIT_C = 0.5
# The tapped forced run's argmax must equal the graph run's id wherever the post-rules top-2 margin exceeds this.  Measured: the
# largest margin of a disagreeing step was 2.78e-3 (lv3w B = 64: 1 of 2304 steps; none at B = 192 / 257, whose GEMMs do not split K).
MEASURED_MARGIN = 2.78e-3
MARGIN = 8e-3
# A forced run without layer taps vs the tapped one: max |logit difference| over finite entries / RMS of the row's finite logits.
# Measured 1.46e-2 (medw; the split-K residual adds in another order), exactly 0 at B = 192 / 257.
MEASURED_RERUN_ERR = 1.46e-2
RERUN_ERR = 4e-2
# Teacher forward: layer l of decoder_logits_impl from its own tap vs the full-sequence mirror (same measure as LAYER_ERR).
MEASURED_TEACHER_LAYER_ERR = {"tiny": 9.04e-3, "lv3w": 1.30e-2, "medw": 1.15e-2}
TEACHER_LAYER_ERR = {"tiny": 1.8e-2, "lv3w": 2.6e-2, "medw": 2.3e-2}
# Teacher taps vs the step decoder's taps for the same ids, layer l: max row |teacher - step| / RMS of the step's layer-l update.
# The two forms are not re-anchored per layer, so the difference grows with depth (tiny: 9.0e-3 after layer 1, 2.45e-2 after 4).
MEASURED_TEACHER_VS_STEP = {"tiny": 2.45e-2, "lv3w": 1.96e-2, "medw": 1.77e-2}
TEACHER_VS_STEP = {"tiny": 5e-2, "lv3w": 4e-2, "medw": 3.6e-2}

MAX_BATCH = {"tiny": 4, "micro128": 4, "medw": 33, "lv3w": 257}
CHUNK = 64                   # clips per fp64 pass


def _cuda():
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the -m gpu tests must run on a B200 (there is no CPU fallback)")


def _stream():
    return torch.cuda.current_stream().cuda_stream


@functools.lru_cache(maxsize=None)
def _model(shape_name):
    from tests.gpu_common import b200_model
    return b200_model(shape_name, "bf16", max_batch=MAX_BATCH[shape_name], perturb=True)


@functools.lru_cache(maxsize=None)
def _enc(shape_name):
    """encoder output of MAX_BATCH clips, encoded once; cases decode prefixes of it"""
    return _model(shape_name).encode(_mel(shape_name, MAX_BATCH[shape_name]))


def _rules(m, timestamps):
    r = m._rules(timestamps)
    return r, dict(suppress=r["suppress"], begin_suppress=r["begin_suppress"], eos=r["eos"], ts_begin=r["timestamp_begin"],
                   no_timestamps=r["no_timestamps"], max_initial_ts=r["max_initial_ts"])


def _decode(m, enc, P, max_length, timestamps, forced, layer_taps, n_sms=0):
    """tw_debug_decode_taps, teacher-forced, every generated step's post-rules logits tapped; with layer_taps also the residual of
    every position 0 .. max_length - 2 ([n_pos, L + 1, B, d]) and every layer's self-attention K|V rows ([L, B, n_pos, 2d])."""
    sh = m.shape
    B, n_gen, n_pos, L, d = enc.shape[0], max_length - len(P), max_length - 1, sh.dec_layers, sh.d_model
    toks = torch.empty((B, n_gen), dtype=torch.int32, device="cuda")
    lens = torch.empty((B,), dtype=torch.int32, device="cuda")
    logits = torch.empty((n_gen, B, sh.vocab), dtype=torch.float32, device="cuda")
    tap = torch.empty((n_pos, L + 1, B, d), dtype=torch.float32, device="cuda") if layer_taps else None
    kv = torch.empty((L, B, n_pos, 2 * d), dtype=torch.bfloat16, device="cuda") if layer_taps else None
    r, _ = _rules(m, timestamps)
    rules, keep = twlib.make_rules(r["suppress"], r["begin_suppress"], r["eos"], r["pad"], r["timestamp_begin"], r["no_timestamps"],
                                   r["max_initial_ts"])
    p = (C.c_int32 * len(P))(*P)
    forced = forced.to("cuda", torch.int32).contiguous()
    ctx = m.ctx
    ctx.check(ctx.lib.tw_debug_decode_taps(
        C.c_void_p(m.handle), enc.data_ptr(), B, p, len(P), C.byref(rules), max_length, toks.data_ptr(), lens.data_ptr(),
        forced.data_ptr(), logits.data_ptr(), n_gen, tap.data_ptr() if layer_taps else None, 0, n_pos if layer_taps else 0,
        kv.data_ptr() if layer_taps else None, n_sms, _stream()))
    torch.cuda.synchronize()
    del keep
    return dict(toks=toks, lens=lens, logits=logits, tap=tap, kv=kv)


# ============================================================================================ the fp64 mirror
def _heads(t):
    return t.view(*t.shape[:-1], t.shape[-1] // 64, 64)


def _attend(s, v):
    """softmax over the last axis of scores s [b, n, h, k] applied to v [b, k, h, 64], rounded to bf16 -> [b, n, h*64]"""
    o = torch.einsum("bnhk,bkhe->bnhe", torch.softmax(s, -1), v)
    return bf(o.reshape(*o.shape[:2], -1))


def step_self(q, kv_own, cache, t):
    """decode self-attention of positions t [n] (rows [b, n, .]): keys / values of the kernel's cache rows 0 .. t-1 ([b, T, 2d])
    and the mirror's own row t"""
    d = q.shape[-1]
    qh, T = _heads(q), cache.shape[1]
    s = torch.einsum("bnhe,bshe->bnhs", qh, _heads(cache[..., :d]))
    s = s.masked_fill((torch.arange(T, device=q.device)[None, :] >= t[:, None])[None, :, None, :], -float("inf"))
    s_own = (qh * _heads(kv_own[..., :d])).sum(-1, keepdim=True)
    p = torch.softmax(torch.cat([s, s_own], -1), -1)
    o = torch.einsum("bnhs,bshe->bnhe", p[..., :T], _heads(cache[..., d:])) + p[..., T:] * _heads(kv_own[..., d:])
    return bf(o.reshape(*o.shape[:2], -1))


def seq_self(q, kv_own):
    """causal self-attention of the full-sequence pass over its own K|V rows [b, n, 2d]"""
    d, n = q.shape[-1], q.shape[1]
    s = torch.einsum("bnhe,bshe->bnhs", _heads(q), _heads(kv_own[..., :d]))
    s = s.masked_fill(torch.ones((n, n), dtype=torch.bool, device=q.device).triu(1)[None, :, None, :], -float("inf"))
    return _attend(s, _heads(kv_own[..., d:]))


def cross_stream(cq, store):
    """softmax(q . K^T) V over the clip's 1500 rows of the model's K|V store [b, 1500, 2d]"""
    d = cq.shape[-1]
    return _attend(torch.einsum("bnhe,bkhe->bnhk", _heads(cq), _heads(store[..., :d])), _heads(store[..., d:]))


def cross_absorbed(cq, enc, Wl):
    """absorbed form: q~_h = bf(Wk_h^T q_h), c_h = bf(softmax(q~_h . E^T) E) over the encoder output E [b, 1500, d],
    att_h = bf(Wv_h c_h + bv_h)"""
    d = cq.shape[-1]
    H = d // 64
    wk, wv, bv = Wl["wkv_c"][:d].view(H, 64, d), Wl["wkv_c"][d:].view(H, 64, d), Wl["bkv_c"][d:].view(H, 64)
    qt = bf(torch.einsum("bnhe,hec->bnhc", _heads(cq), wk))
    c = bf(torch.einsum("bnhk,bkc->bnhc", torch.softmax(torch.einsum("bnhc,bkc->bnhk", qt, enc), -1), enc))
    o = bf(torch.einsum("bnhc,hec->bnhe", c, wv) + bv)
    return o.reshape(*o.shape[:2], -1)


def ln_bf16(x, g, b):
    """bf16 LayerNorm output of the mirror, and per element the bf16 step by which the kernel's output may differ from it: one ulp
    where the fp64 value lies within the fp32 LayerNorm's error (LN_TAU of test_gpu_encoder_stage) of a bf16 rounding midpoint, so
    that the kernel may round it the other way, else 0."""
    y, xh, mu_sd = ln64(x, g, b)
    r, ulp = bf(y), ulp_bf16(y)
    near = ulp / 2 - (y - r).abs() <= LN_TAU * ln_scale(xh, mu_sd, g, b)
    return r, torch.where(near, ulp, 0.0)


def layer64(x, Wl, self_attn, cross_attn):
    """one decoder layer of launch_step / decoder_logits_impl on the residual rows x [b, n, d]; self_attn(q, own K|V rows) and
    cross_attn(q) give the bf16 attention outputs.  Returns (bf16 LayerNorm output feeding the QKV GEMM, its possible rounding
    steps (ln_bf16), unrounded K|V rows, output)."""
    d = x.shape[-1]
    xn1, step1 = ln_bf16(x, Wl["ln1_g"], Wl["ln1_b"])
    qkv = xn1 @ Wl["wqkv"].T + Wl["bqkv"]
    q, kv = bf(qkv[..., :d]), bf(qkv[..., d:])
    x = x + self_attn(q, kv) @ Wl["wo"].T + Wl["bo"]
    xn = bf(ln64(x, Wl["ln2_g"], Wl["ln2_b"])[0])
    x = x + cross_attn(bf(xn @ Wl["wq_c"].T + Wl["bq_c"])) @ Wl["wo_c"].T + Wl["bo_c"]
    xn = bf(ln64(x, Wl["ln3_g"], Wl["ln3_b"])[0])
    return xn1, step1, qkv[..., d:], x + bf(F.gelu(xn @ Wl["w1"].T + Wl["b1"])) @ Wl["w2"].T + Wl["b2"]


def _amax(t):
    """largest element, NaN if any element is NaN (and then every bar fails), inf for no elements"""
    return t.max().item() if t.numel() else float("inf")


def _worse(a, b):
    """max that keeps a NaN"""
    return a if a != a or a >= b else b


def _row_err(tap, mir, prev, mask):
    """max over rows (mask [b, n]) of max |tap - mirror| / RMS(tap - prev)"""
    return _amax(((tap - mir).abs().amax(-1) / (tap - prev).pow(2).mean(-1).sqrt())[mask])


def _gemm_excess(out, ref, xn, step, w, bf16_out):
    """per element (|out - ref| - [one bf16 ulp of ref for a bf16 output] - sum_k step_k |w_k|) / unit, unit = 2^-24 (sqrt(K)
    sum_k |xn_k w_k| + |ref|): the GEMM's fp32 accumulation after the input elements the kernel's LayerNorm may have rounded the
    other way (step, from ln_bf16)"""
    # clamped: the zero embedding row of EOS gives ref = unit = 0, where the kernel's 0 must be exact
    unit = (EPS24 * (xn.shape[-1] ** 0.5 * (xn.abs() @ w.abs().T) + ref.abs())).clamp_min(torch.finfo(torch.float64).tiny)
    return ((out - ref).abs() - (ulp_bf16(ref) if bf16_out else 0.0) - step @ w.abs().T) / unit


# ============================================================================================ a. the decode step
CASES = {
    # name: shape, B, max_length, timestamps, tapped windows (positions), TWB200_ABSORB, n_sms, ragged row budgets
    "tiny-1": ("tiny", 1, 40, False, [(0, 39)], False, 0, False),
    "micro128-3": ("micro128", 3, 40, False, [(0, 39)], False, 0, False),
    "medw-33-ts-448": ("medw", 33, 448, True, [(0, 21), (425, 447)], False, 0, False),
    "lv3w-64": ("lv3w", 64, 40, False, [(0, 39)], False, 0, False),
    "lv3w-64-absorbed": ("lv3w", 64, 40, False, [(0, 39)], True, 0, False),
    "lv3w-192": ("lv3w", 192, 40, False, [(0, 39)], False, 0, False),
    "lv3w-192-124sms": ("lv3w", 192, 40, False, [(0, 39)], False, 124, False),
    "lv3w-257": ("lv3w", 257, 40, False, [(0, 39)], False, 0, False),
    "lv3w-64-ragged": ("lv3w", 64, 40, False, [(0, 39)], False, 0, True),
}


@pytest.mark.parametrize("case", list(CASES))
def test_decode_layers_vs_fp64_mirror(case, monkeypatch):
    """tiny B = 1: M = 1, positions across the cache pages at 16 and 32; micro128: d = 128; medw B = 33 with the timestamp rules at
    max_length 448: the deepest cache; lv3w: the stream path at B = 64, the absorbed cross-attention (TWB200_ABSORB=1), the
    headline's 192 merged rows (three row blocks of the skinny GEMMs and the fused append), the same at the headline decode
    partition's 124 SMs (another split-K choice), 257 rows (the general tcgen05 GEMM and the separate kv_append kernel), and
    ragged row budgets (rows finishing at different steps leave the active list; they must emit pad and are not compared)."""
    _cuda()
    shape_name, B, max_length, ts, windows, absorb, n_sms, ragged = CASES[case]
    if absorb:
        monkeypatch.setenv("TWB200_ABSORB", "1")
    else:
        monkeypatch.delenv("TWB200_ABSORB", raising=False)
    sh = SHAPES[shape_name]
    d, L, H = sh.d_model, sh.dec_layers, sh.heads
    m = _model(shape_name)
    W = _weights64(shape_name, True)
    enc = _enc(shape_name)[:B]
    P = prompt_ids(sh.vocab, ts)
    n_gen = max_length - len(P)
    r, orules = _rules(m, ts)
    budgets = None
    if ragged:
        rng = np.random.default_rng(11)
        budgets = [int(rng.integers(1, n_gen)) if b % 2 == 0 else n_gen + 5 for b in range(B)]
    m.set_row_budgets(budgets)
    try:
        if absorb:          # poison the K|V store of these clips: the absorbed path must not read or rewrite it
            ctx = m.ctx
            nan = torch.full_like(enc, float("nan"))
            ctx.check(ctx.lib.tw_debug_cross_kv(C.c_void_p(m.handle), nan.data_ptr(), B, 0, _stream()))
        ids, lens0 = m.decode(enc, P, max_length, ts)                        # production: the CUDA graph, free-running
        run = _decode(m, enc, P, max_length, ts, ids, True, n_sms)
        again = _decode(m, enc, P, max_length, ts, ids, False, n_sms)
    finally:
        m.set_row_budgets(None)
    if absorb:
        assert torch.isnan(_read(m, -1, 0, B, 0)[1]).all(), "the K|V store was rewritten: the absorbed path did not run"
    lens = run["lens"].long()
    assert torch.equal(lens, lens0.long()), "the forced run's lengths differ from the run it was fed from"
    if ragged:
        assert len(set(lens.tolist())) > 3 and (lens < n_gen).any()
    # finished rows emit pad
    g_idx = torch.arange(n_gen, device="cuda")
    done = g_idx[None, :] >= lens[:, None]
    assert (run["toks"][done] == r["pad"]).all()

    pos = torch.cat([torch.arange(a, b) for a, b in windows]).cuda()
    n = pos.numel()
    tap = run["tap"][pos].double()                   # [n, L + 1, B, d]
    # row b is compared at position t while it is active: every prompt position, generated steps g = t - (P - 1) < lens[b]
    active = (pos[None, :] - (len(P) - 1)) < lens[:, None]                  # [B, n]
    # fed tokens per position: the prompt, then the forced ids
    fed = torch.cat([torch.tensor(P, device="cuda").expand(B, -1), ids.long()], 1)[:, :max_length - 1]
    emb = bf(W["embed"][fed[:, pos]]) + bf(W["dec_pos"][pos])[None]
    emb_err = _amax(((tap[:, 0].transpose(0, 1) - emb).abs() / emb.abs().clamp_min(1e-30))[active])

    layer_err, kv_c = [0.0] * L, -np.inf
    for c0 in range(0, B, CHUNK):
        sl = slice(c0, min(B, c0 + CHUNK))
        act = active[sl]
        for l in range(L):
            Wl = W["dec"][l]
            x_in = tap[:, l, sl].transpose(0, 1)                               # [b, n, d]
            cache = run["kv"][l, sl, :int(pos.max())].double()
            if absorb:
                e64 = enc[sl].double()
                cross = lambda cq: cross_absorbed(cq, e64, Wl)                # noqa: E731
            else:
                store = _read(m, -1, sl.start, sl.stop - sl.start, l)[1].double()
                cross = lambda cq: cross_stream(cq, store)                    # noqa: E731
            xn1, step1, kv_ref, mir = layer64(x_in, Wl, lambda q, kv: step_self(q, kv, cache, pos), cross)
            kv_k = run["kv"][l, sl][:, pos].double()
            ex = _gemm_excess(kv_k, kv_ref, xn1, step1, Wl["wqkv"][d:], True).amax(-1)
            kv_c = _worse(kv_c, _amax(ex[act]))
            layer_err[l] = _worse(layer_err[l], _row_err(tap[:, l + 1, sl].transpose(0, 1), mir, x_in, act))
            del cache, xn1, step1, kv_ref, mir, kv_k
            if not absorb:
                del store

    # post-rules logits at the tapped positions that produce a token
    lg_c, inf_mismatch = 0.0, 0
    sup = torch.zeros(sh.vocab, dtype=torch.bool, device="cuda")
    sup[torch.tensor(r["suppress"], dtype=torch.long)] = True
    beg = sup.clone()
    beg[torch.tensor(r["begin_suppress"], dtype=torch.long)] = True
    for j in range(n):
        t = int(pos[j])
        g = t - (len(P) - 1)
        if g < 0:
            continue
        rows = active[:, j].nonzero().flatten()
        if rows.numel() == 0:
            continue
        xn, step = ln_bf16(tap[j, L, rows], W["dlnf_g"], W["dlnf_b"])
        ref = xn @ W["embed"].T
        k = run["logits"][g, rows].double()
        if ts:
            hist = ids[rows, :g].cpu().numpy()
            ref_np = ref.float().cpu().numpy()
            neg = torch.from_numpy(np.stack([np.isneginf(apply_rules(ref_np[i], list(hist[i]), orules))
                                             for i in range(rows.numel())])).cuda()
        else:
            neg = (beg if g == 0 else sup)[None].expand(rows.numel(), -1)
        kneg = torch.isneginf(k)
        inf_mismatch += int((kneg != neg).any(-1).sum())
        fin = ~kneg & ~neg
        lg_c = _worse(lg_c, _amax(_gemm_excess(k, ref, xn, step, W["embed"], False)[fin]))
        del xn, step, ref, k

    # the tapped run against production: argmax vs the graph's ids, logits vs a run without layer taps
    lg, lg2 = run["logits"], again["logits"]
    act_g = ~done                                                              # [B, n_gen]
    top2 = lg.topk(2, -1).values                                               # [n_gen, B, 2]
    margin = (top2[..., 0] - top2[..., 1]).transpose(0, 1)
    differ = (run["toks"] != ids) & act_g
    worst_margin = margin[differ].max().item() if differ.any() else 0.0
    same_inf = torch.equal(torch.isneginf(lg)[act_g.T], torch.isneginf(lg2)[act_g.T])
    fin = torch.isfinite(lg) & act_g.T[..., None]
    rms = torch.where(fin, lg, 0.0).pow(2).sum(-1, keepdim=True).div(fin.sum(-1, keepdim=True).clamp_min(1)).sqrt()
    rerun = _amax(((lg2 - lg).abs() / rms)[fin])

    print(f"{case}: embed max rel err {emb_err:.3e}; layers max row |kernel - mirror| / rms(update) = "
          f"{', '.join(f'{e:.3e}' for e in layer_err)}; K|V row max (|err| - ulp) / unit = {kv_c:.3e}; logits max |err| / unit = "
          f"{lg_c:.3e}, -inf set mismatches {inf_mismatch}; argmax vs graph ids: {int(differ.sum())} differ of {int(act_g.sum())}, "
          f"largest margin among them {worst_margin:.3e}; rerun without taps: max |dlogit| / rms = {rerun:.3e}")
    assert emb_err <= 2.0 ** -23, emb_err
    for l in range(L):
        assert layer_err[l] <= LAYER_ERR[shape_name], (case, l, layer_err[l])
    assert kv_c <= KV_ROW_C, (case, kv_c)
    assert inf_mismatch == 0, (case, inf_mismatch)
    assert lg_c <= LOGIT_C, (case, lg_c)
    assert worst_margin <= MARGIN, (case, worst_margin)
    assert same_inf, case
    assert rerun <= RERUN_ERR, (case, rerun)


# ============================================================================================ b. the teacher forward
TEACHER_CASES = {"tiny-3x40": ("tiny", 3, 40), "lv3w-8x70": ("lv3w", 8, 70), "medw-2x448": ("medw", 2, 448)}


def _teacher_taps(m, enc, ids):
    sh = m.shape
    B, T = ids.shape
    ld = (sh.vocab + 3) // 4 * 4
    logits = torch.empty((B * T, ld), dtype=torch.float32, device="cuda")
    tap = torch.empty((sh.dec_layers + 1, B, T, sh.d_model), dtype=torch.float32, device="cuda")
    ids = ids.to("cuda", torch.int32).contiguous()
    ctx = m.ctx
    ctx.check(ctx.lib.tw_debug_decoder_logits_taps(C.c_void_p(m.handle), enc.data_ptr(), B, ids.data_ptr(), T, logits.data_ptr(), ld,
                                                   tap.data_ptr(), _stream()))
    torch.cuda.synchronize()
    return tap


@pytest.mark.parametrize("case", list(TEACHER_CASES))
def test_teacher_forward_layers_vs_fp64_mirror_and_step(case, monkeypatch):
    """tiny B = 3, T = 40; lv3w B = 8, T = 70 (M = 560: tile tails); medw B = 2, T = 448 (the longest causal run).  Each layer of
    decoder_logits_impl against the full-sequence mirror (causal self-attention over all T positions, cross-attention over the
    K|V store), then its taps against the step decoder's taps for the same ids, position by position."""
    _cuda()
    monkeypatch.delenv("TWB200_ABSORB", raising=False)
    shape_name, B, T = TEACHER_CASES[case]
    sh = SHAPES[shape_name]
    L = sh.dec_layers
    m = _model(shape_name)
    W = _weights64(shape_name, True)
    enc = _enc(shape_name)[:B]
    ts = shape_name == "medw"
    P = prompt_ids(sh.vocab, ts)
    max_length = min(T + 1, sh.max_target)
    gen, _ = m.decode(enc, P, max_length, ts)
    ids = torch.cat([torch.tensor(P, device="cuda").expand(B, -1), gen.long()], 1)[:, :T]
    tap = _teacher_taps(m, enc, ids).double()
    errs = []
    for l in range(L):
        store = _read(m, -1, 0, B, l)[1].double()
        _, _, _, mir = layer64(tap[l], W["dec"][l], seq_self, lambda cq: cross_stream(cq, store))
        errs.append(_row_err(tap[l + 1], mir, tap[l], torch.ones((B, T), dtype=torch.bool, device="cuda")))
        del store, mir
    step = _decode(m, enc, P, max_length, ts, gen, True)["tap"].double()       # [n_pos, L + 1, B, d]
    n_pos = step.shape[0]
    step = step.permute(1, 2, 0, 3)                                             # [L + 1, B, n_pos, d]
    emb_eq = torch.equal(step[0], tap[0, :, :n_pos])
    vs = [((tap[l, :, :n_pos] - step[l]).abs().amax(-1) / (step[l] - step[l - 1]).pow(2).mean(-1).sqrt()).max().item()
          for l in range(1, L + 1)]
    print(f"teacher {case}: layers max row |kernel - mirror| / rms(update) = {', '.join(f'{e:.3e}' for e in errs)}; "
          f"vs the step decoder over {n_pos} positions: {', '.join(f'{e:.3e}' for e in vs)}; embedding equal: {emb_eq}")
    for l in range(L):
        assert errs[l] <= TEACHER_LAYER_ERR[shape_name], (case, l, errs[l])
        assert vs[l] <= TEACHER_VS_STEP[shape_name], (case, l, vs[l])
    assert emb_eq


def test_decode_taps_argument_errors():
    _cuda()
    m = _model("tiny")
    sh = m.shape
    enc = _enc("tiny")[:1]
    P = prompt_ids(sh.vocab, False)
    r, _ = _rules(m, False)
    rules, keep = twlib.make_rules(r["suppress"], r["begin_suppress"], r["eos"], r["pad"], None, r["no_timestamps"], r["max_initial_ts"])
    p = (C.c_int32 * len(P))(*P)
    buf = torch.empty(1 << 20, dtype=torch.float32, device="cuda")
    ctx = m.ctx
    for pos0, n_pos, n_sms in [(-1, 2, 0), (0, 40, 0), (30, 10, 0), (0, 2, -1)]:
        rc = ctx.lib.tw_debug_decode_taps(C.c_void_p(m.handle), enc.data_ptr(), 1, p, len(P), C.byref(rules), 40, buf.data_ptr(),
                                          buf.data_ptr(), None, None, 0, buf.data_ptr(), pos0, n_pos, None, n_sms, _stream())
        assert rc == twlib.TW_E_INVALID, (pos0, n_pos, n_sms)
    rc = ctx.lib.tw_debug_decoder_logits_taps(C.c_void_p(m.handle), enc.data_ptr(), 1, buf.data_ptr(), 4, buf.data_ptr(), 51868, None,
                                              _stream())
    assert rc == twlib.TW_E_INVALID
    del keep
