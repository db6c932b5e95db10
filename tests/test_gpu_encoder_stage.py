"""-m gpu: the bf16 encoder stage (stage 1 of the pipeline: log-mel front end, conv stem, encoder layers, final LayerNorm,
cross-attention K|V store) kernel by kernel and layer by layer, as the model issues it, against float64 references computed with
torch on the GPU.

The models here have non-trivial biases and LayerNorms (tests.helpers.perturb_hf_model): with HF's init every bias is 0 and every
LayerNorm is (1, 0), so a bias or LayerNorm routed to the wrong layer or projection would be invisible.

- Both LayerNorm kernels (one CTA per row for M <= 512, one warp per row above) at the model widths, per element.
- Every encoder layer recomputed from the kernel's own input (the fp32 residual tap of the previous layer) by a float64 MIRROR of
  encode_impl: the weights as the model holds them (bf16, q rows and q bias scaled by 0.125, fp32 biases / LayerNorms /
  positions) and bf16 rounding exactly where the model stores bf16 (LayerNorm output, qkv, attention output, GELU(fc1)).
- The cross-attention K|V store, per decoder layer, including writes of a clip sub-range.
- The fused front end of the pipeline (the log-mel floor and scaling applied inside the conv-stem im2col) against the unfused path.
Every bar below is a measurement on a B200 with its margin.
"""
import ctypes as C
import functools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from taiwan_whisper_b200 import lib as twlib
from taiwan_whisper_b200.configs import SHAPES
from taiwan_whisper_b200.synth import synth_batch
from tests.gpu_common import EPS24, GEMM_BF16_C, ulp_bf16

pytestmark = pytest.mark.gpu

# LayerNorm in fp32 (elementwise.cu: two-pass mean / centred variance, rsqrtf): per element |out - fp64| <= LN_TAU * (|gamma| *
# (|x_hat| + |mean| / std) + |beta|).  The |mean| / std term is the fp32 rounding of the mean seen through the normalisation: it
# dominates rows whose mean is far larger than their spread (offset 1e3, std 1) and constant rows (std = sqrt(eps)).
# Measured on a B200 (1000 W power limit) over every shape of test_layernorm_kernels_vs_fp64: 1.99e-6 (fp32 output, M = 1503,
# d = 128; the other shapes 8e-9 .. 1.5e-6), and for bf16 outputs the excess over one ulp reaches 1.0e-7.  The bar is 3x the
# largest.  (A variance divided by d - 1 instead of d is ~1e-4 on this scale.)
MEASURED_LN_TAU = 1.99e-6
LN_TAU = 6e-6
# Encoder layer l (kernel tap l vs the fp64 mirror run on tap l-1): max over elements of a row of |tap - mirror| divided by the
# RMS of that row's layer update (tap l - tap l-1), maximised over every row of the batch.  What is left is fp32 accumulation
# order and the rare element whose bf16 rounding of an intermediate falls the other way; most of it is the flash kernel's bf16
# rounding of the attention probabilities before P.V, which the mirror does not do.  The conv stem (tap 0, mirrored from the
# mel) is divided by the RMS of the row's GELU(conv2) output, the positions left out, and has bars of its own.
# Per shape, the largest over its layers as measured on a B200 (1000 W power limit); each bar is twice its measurement.
MEASURED_STEM_ERR = {"tiny": 8.69e-4, "micro128": 1.23e-3, "medw": 1.06e-3, "lv3w": 2.91e-3}
STEM_ERR = {"tiny": 1.75e-3, "micro128": 2.5e-3, "medw": 2.1e-3, "lv3w": 5.8e-3}
MEASURED_LAYER_ERR = {"tiny": 8.77e-3, "micro128": 5.72e-3, "medw": 9.20e-3, "lv3w": 1.11e-2}
LAYER_ERR = {"tiny": 1.8e-2, "micro128": 1.15e-2, "medw": 1.85e-2, "lv3w": 2.2e-2}


def _cuda():
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the -m gpu tests must run on a B200 (there is no CPU fallback)")


def _ctx():
    return twlib.Context.get(torch.cuda.current_device())


def _stream():
    return torch.cuda.current_stream().cuda_stream


def ln64(x, g, b):
    """float64 LayerNorm (biased variance, eps 1e-5); also returns x_hat, |mean| / std for the error bound."""
    mu = x.mean(-1, keepdim=True)
    sd = torch.sqrt(((x - mu) ** 2).mean(-1, keepdim=True) + 1e-5)
    xh = (x - mu) / sd
    return xh * g + b, xh, mu.abs() / sd


def ln_scale(xh, mu_sd, g, b):
    return g.abs() * (xh.abs() + mu_sd) + b.abs()


def bf(t):
    return t.to(torch.bfloat16).to(torch.float64)


# ============================================================================================ a. LayerNorm kernels
def _layernorm(x, g, b, dtype):
    """tw_debug_layernorm into a buffer with two NaN sentinel rows after row M; returns (out [M, d], sentinel rows)."""
    M, d = x.shape
    out = torch.full((M + 2, d), float("nan"), dtype=dtype, device="cuda")
    ctx = _ctx()
    dt = twlib.TW_F32 if dtype == torch.float32 else twlib.TW_BF16
    ctx.check(ctx.lib.tw_debug_layernorm(ctx.handle, x.data_ptr(), g.data_ptr(), b.data_ptr(), out.data_ptr(), M, d, dt, _stream()))
    torch.cuda.synchronize()
    return out[:M], out[M:]


@pytest.mark.parametrize("M", [1, 7, 512, 513, 1503, 96000])
@pytest.mark.parametrize("d", [128, 384, 1024, 1280])
def test_layernorm_kernels_vs_fp64(M, d):
    """M <= 512: layernorm_row_kernel, above: layernorm_kernel.  Random gamma / beta; rows with mean >> std (offset 1e3, std 1), a
    constant row and a row with one large outlier.  fp32 output per element within LN_TAU of the fp64 value (scaled as above),
    bf16 output within one bf16 ulp of it (plus the same fp32 term); the two rows after the output stay NaN."""
    _cuda()
    g_ = torch.Generator(device="cuda").manual_seed(M * 13 + d)
    x = torch.randn((M, d), device="cuda", generator=g_) * 2.0 + torch.randn((M, 1), device="cuda", generator=g_)
    x[0] = 1e3 + torch.randn((d,), device="cuda", generator=g_)              # mean >> std: the two-pass variance
    if M > 1:
        x[M // 2] = 0.7321                                                       # constant row: variance 0
    if M > 2:
        x[M - 1, d // 3] = 5e3                                                   # one outlier
    gamma = 1.0 + 0.3 * torch.randn((d,), device="cuda", generator=g_)
    beta = 0.3 * torch.randn((d,), device="cuda", generator=g_)
    ref, xh, mu_sd = ln64(x.double(), gamma.double(), beta.double())
    scale = ln_scale(xh, mu_sd, gamma.double(), beta.double())
    out, sent = _layernorm(x, gamma, beta, torch.float32)
    assert torch.isnan(sent).all()
    tau = ((out.double() - ref).abs() / scale).max().item()
    print(f"layernorm M={M} d={d}: fp32 max |err| / scale = {tau:.3e}")
    assert tau <= LN_TAU, (M, d, tau)
    outb, sentb = _layernorm(x, gamma, beta, torch.bfloat16)
    assert torch.isnan(sentb.float()).all()
    excess = ((outb.double() - ref).abs() - ulp_bf16(ref)) / scale
    print(f"layernorm M={M} d={d}: bf16 max (|err| - ulp) / scale = {excess.max().item():.3e}")
    assert (excess <= LN_TAU).all(), (M, d, excess.max().item())


def test_layernorm_entry_rejects_bad_shapes():
    _cuda()
    ctx = _ctx()
    x = torch.zeros((4, 1284), device="cuda")
    g = torch.ones(1284, device="cuda")
    out = torch.zeros((4, 1284), device="cuda")
    for M, d, dt in [(4, 1284, twlib.TW_F32), (4, 6, twlib.TW_F32), (-1, 128, twlib.TW_F32), (4, 128, twlib.TW_I16)]:
        rc = ctx.lib.tw_debug_layernorm(ctx.handle, x.data_ptr(), g.data_ptr(), g.data_ptr(), out.data_ptr(), M, d, dt, _stream())
        assert rc == twlib.TW_E_INVALID, (M, d, dt)
    # M = 0 is a valid empty launch
    assert ctx.lib.tw_debug_layernorm(ctx.handle, x.data_ptr(), g.data_ptr(), g.data_ptr(), out.data_ptr(), 0, 128, twlib.TW_F32,
                                      _stream()) == twlib.TW_OK


# ============================================================================================ models and mirrors
MAX_BATCH_LV3W = 192          # the --merge 3 layout of the headline: three 64-clip batches staged into one slot
PIPELINE_SMS = 24             # the stage-1 partition of the merged headline


@functools.lru_cache(maxsize=None)
def _model(shape_name):
    """The perturbed bf16 model of the shape; lv3w: the single large model of the file (max_batch 192), with the pipeline enabled
    here, once, for the fused stage-1 test, so that every test of the file sees the same model state.  With the pipeline on, the
    model's own K|V store (tw_decode_greedy's, tw_debug_cross_kv's) is slot 0's; the fused test stages into slot 1."""
    from tests.gpu_common import b200_model
    if shape_name != "lv3w":
        return b200_model(shape_name, "bf16", max_batch=4, perturb=True)
    m = b200_model(shape_name, "bf16", max_batch=MAX_BATCH_LV3W, perturb=True)
    try:
        m.enable_pipeline(PIPELINE_SMS)
    except NotImplementedError as e:          # TW_E_UNSUPPORTED: no green contexts on this driver
        m.pipeline_unsupported = str(e)
    return m


@functools.lru_cache(maxsize=None)
def _weights64(shape_name, rounded):
    """float64 device copies of the encoder / decoder weights: as the model holds them (rounded: bf16 matrices, token embedding and
    decoder positions, q rows and q bias scaled by 0.125) or exactly as HF holds them (the unrounded fp64 run)."""
    from tests.gpu_common import hf_model
    sd = {k: v.detach().to("cuda", torch.float64) for k, v in hf_model(shape_name, 1234, True).state_dict().items()}
    sh = SHAPES[shape_name]
    r = bf if rounded else (lambda t: t)
    E = "model.encoder."
    W = dict(conv1_w=r(sd[E + "conv1.weight"]), conv1_b=sd[E + "conv1.bias"], conv2_w=r(sd[E + "conv2.weight"]),
             conv2_b=sd[E + "conv2.bias"], pos=sd[E + "embed_positions.weight"], lnf_g=sd[E + "layer_norm.weight"],
             lnf_b=sd[E + "layer_norm.bias"], layers=[], kv=[])
    for l in range(sh.enc_layers):
        p = f"{E}layers.{l}."
        a = p + "self_attn."
        W["layers"].append(dict(
            ln1_g=sd[p + "self_attn_layer_norm.weight"], ln1_b=sd[p + "self_attn_layer_norm.bias"],
            wqkv=torch.cat([r(0.125 * sd[a + "q_proj.weight"]), r(sd[a + "k_proj.weight"]), r(sd[a + "v_proj.weight"])]),
            bqkv=torch.cat([0.125 * sd[a + "q_proj.bias"], torch.zeros_like(sd[a + "v_proj.bias"]), sd[a + "v_proj.bias"]]),
            wo=r(sd[a + "out_proj.weight"]), bo=sd[a + "out_proj.bias"],
            ln3_g=sd[p + "final_layer_norm.weight"], ln3_b=sd[p + "final_layer_norm.bias"],
            w1=r(sd[p + "fc1.weight"]), b1=sd[p + "fc1.bias"], w2=r(sd[p + "fc2.weight"]), b2=sd[p + "fc2.bias"]))
    for l in range(sh.dec_layers):
        a = f"model.decoder.layers.{l}.encoder_attn."
        W["kv"].append(dict(w=torch.cat([r(sd[a + "k_proj.weight"]), r(sd[a + "v_proj.weight"])]),
                            b=torch.cat([torch.zeros_like(sd[a + "v_proj.bias"]), sd[a + "v_proj.bias"]])))
    # decoder: the self-attention and MLP as in the encoder, the cross-attention q projection and out projection (its K|V
    # projection is W["kv"]), layer norms 1 / 2 / 3 in front of self-attention / cross-attention / MLP
    Dc = "model.decoder."
    W.update(embed=r(sd[Dc + "embed_tokens.weight"]), dec_pos=r(sd[Dc + "embed_positions.weight"]),
             dlnf_g=sd[Dc + "layer_norm.weight"], dlnf_b=sd[Dc + "layer_norm.bias"], dec=[])
    for l in range(sh.dec_layers):
        p = f"{Dc}layers.{l}."
        a, c = p + "self_attn.", p + "encoder_attn."
        W["dec"].append(dict(
            ln1_g=sd[p + "self_attn_layer_norm.weight"], ln1_b=sd[p + "self_attn_layer_norm.bias"],
            wqkv=torch.cat([r(0.125 * sd[a + "q_proj.weight"]), r(sd[a + "k_proj.weight"]), r(sd[a + "v_proj.weight"])]),
            bqkv=torch.cat([0.125 * sd[a + "q_proj.bias"], torch.zeros_like(sd[a + "v_proj.bias"]), sd[a + "v_proj.bias"]]),
            wo=r(sd[a + "out_proj.weight"]), bo=sd[a + "out_proj.bias"],
            ln2_g=sd[p + "encoder_attn_layer_norm.weight"], ln2_b=sd[p + "encoder_attn_layer_norm.bias"],
            wq_c=r(0.125 * sd[c + "q_proj.weight"]), bq_c=0.125 * sd[c + "q_proj.bias"],
            wkv_c=W["kv"][l]["w"], bkv_c=W["kv"][l]["b"], wo_c=r(sd[c + "out_proj.weight"]), bo_c=sd[c + "out_proj.bias"],
            ln3_g=sd[p + "final_layer_norm.weight"], ln3_b=sd[p + "final_layer_norm.bias"],
            w1=r(sd[p + "fc1.weight"]), b1=sd[p + "fc1.bias"], w2=r(sd[p + "fc2.weight"]), b2=sd[p + "fc2.bias"]))
    return W


def stem64(mel, W, r):
    """conv stem of encode_impl: im2col of r(mel), conv1 + bias, GELU, stored (r) as h0; conv2 (stride 2) + bias, GELU, +
    positions into the fp32 residual.  mel [b, n_mel, 3000] -> [b, 1500, d]."""
    h0 = r(F.gelu(F.conv1d(r(mel.double()), W["conv1_w"], W["conv1_b"], padding=1)))
    return F.gelu(F.conv1d(h0, W["conv2_w"], W["conv2_b"], stride=2, padding=1)).transpose(1, 2) + W["pos"]


def layer64(x, P, H, r):
    """one encoder layer of encode_impl on the residual x [b, 1500, d]; r is applied where the model stores bf16."""
    b, S, d = x.shape
    xn = r(ln64(x, P["ln1_g"], P["ln1_b"])[0])
    q, k, v = r(xn @ P["wqkv"].T + P["bqkv"]).view(b, S, 3, H, d // H).permute(2, 0, 3, 1, 4)
    att = r(torch.softmax(q @ k.transpose(-1, -2), -1) @ v).transpose(1, 2).reshape(b, S, d)
    x = x + att @ P["wo"].T + P["bo"]
    xn = r(ln64(x, P["ln3_g"], P["ln3_b"])[0])
    return x + r(F.gelu(xn @ P["w1"].T + P["b1"])) @ P["w2"].T + P["b2"]


def _mel(shape_name, B, seed=7):
    from taiwan_whisper_b200.host import log_mel
    return log_mel(torch.from_numpy(synth_batch(seed, B)).cuda(), None, SHAPES[shape_name].n_mel)


# ============================================================================================ b. encoder layers
@pytest.mark.parametrize("shape_name,B", [("tiny", 1), ("micro128", 2), ("medw", 3), ("lv3w", 64)])
def test_encoder_layers_vs_fp64_mirror(shape_name, B):
    """tiny: N = 384 (a 256-column tile and a 128-column tail), M = 1500 / 3000 tails; micro128: d = 128; medw: conv1 K = 240 (a
    partial K block), tiles across clip boundaries; lv3w at B = 64: M = 96 000 as in the headline encoder, many tiles per
    persistent CTA.  Each layer against the mirror of its own input; enc_out within one bf16 ulp (plus the fp32 LayerNorm term) of
    fp64 LayerNorm(last tap); two encoder runs bitwise equal."""
    _cuda()
    sh = SHAPES[shape_name]
    m = _model(shape_name)
    Wm, Wp = _weights64(shape_name, True), _weights64(shape_name, False)
    mel = _mel(shape_name, B)
    taps, encs = [], []
    for l in range(sh.enc_layers + 1):
        e, t = m.encode(mel, tap_layer=l)
        encs.append(e)
        taps.append(t)
    enc = encs[-1]
    torch.cuda.synchronize()
    chunk = 4                  # clips per fp64 pass
    errs = []
    for l in range(sh.enc_layers + 1):
        err = num = den = 0.0
        for c0 in range(0, B, chunk):
            sl = slice(c0, min(B, c0 + chunk))
            tap = taps[l][sl].double()
            if l == 0:
                mir, pure = stem64(mel[sl], Wm, bf), stem64(mel[sl], Wp, lambda t: t)
                prev = torch.zeros_like(tap)
                upd = mir - Wm["pos"]          # GELU(conv2) of the mirror
            else:
                prev = taps[l - 1][sl].double()
                mir = layer64(prev, Wm["layers"][l - 1], sh.heads, bf)
                pure = layer64(prev, Wp["layers"][l - 1], sh.heads, lambda t: t)
                upd = tap - prev
            rms = upd.pow(2).mean(-1).sqrt()
            err = max(err, ((tap - mir).abs().amax(-1) / rms).max().item())
            num += (mir - pure).pow(2).sum().item()
            den += (pure - prev).pow(2).sum().item()
            del tap, mir, pure, prev, upd
        mir_rel = (num / den) ** 0.5
        print(f"{shape_name} B={B} {'stem' if l == 0 else f'layer {l}'}: max row |kernel - mirror| / rms(update) = {err:.3e}; "
              f"mirror vs unrounded fp64, relative L2 of the update = {mir_rel:.3e}")
        errs.append(err)
    # final LayerNorm: enc_out vs fp64 LN of the last tap
    ex = 0.0
    for c0 in range(0, B, chunk):
        sl = slice(c0, min(B, c0 + chunk))
        ref, xh, mu_sd = ln64(taps[-1][sl].double(), Wm["lnf_g"], Wm["lnf_b"])
        ex = max(ex, (((enc[sl].double() - ref).abs() - ulp_bf16(ref)) / ln_scale(xh, mu_sd, Wm["lnf_g"], Wm["lnf_b"])).max().item())
    print(f"{shape_name} B={B} final LayerNorm: max (|err| - ulp) / scale = {ex:.3e}")
    assert errs[0] <= STEM_ERR[shape_name], (shape_name, "stem", errs[0])
    for l in range(1, sh.enc_layers + 1):
        assert errs[l] <= LAYER_ERR[shape_name], (shape_name, l, errs[l])
    assert ex <= LN_TAU, ex
    for e in encs[:-1]:
        assert torch.equal(e.view(torch.int16), enc.view(torch.int16)), "two encoder runs differ"


# ============================================================================================ c. cross-attention K|V store
def _cross_kv(m, enc, clip0):
    ctx = m.ctx
    ctx.check(ctx.lib.tw_debug_cross_kv(C.c_void_p(m.handle), enc.data_ptr(), enc.shape[0], clip0, _stream()))


def _read(m, slot, clip0, B, layer, with_enc=False):
    """tw_debug_read_stage1 -> (enc [B, 1500, d] or None, K|V rows [B, 1500, 2d]) of the model's dtype."""
    ctx = m.ctx
    d = m.shape.d_model
    enc = torch.empty((B, 1500, d), dtype=torch.bfloat16, device="cuda") if with_enc else None
    kv = torch.empty((B, 1500, 2 * d), dtype=torch.bfloat16, device="cuda")
    ctx.check(ctx.lib.tw_debug_read_stage1(C.c_void_p(m.handle), slot, clip0, B, enc.data_ptr() if with_enc else None, layer,
                                           kv.data_ptr(), _stream()))
    torch.cuda.synchronize()
    return enc, kv


def _kv_excess(kv, enc, P):
    """max over elements of (|kv - fp64 ref| - 1 bf16 ulp) / (2^-24 sqrt(K) sum_k |e_k w_k|), clip by clip."""
    K = enc.shape[-1]
    worst = -np.inf
    for i in range(enc.shape[0]):
        e = enc[i].double()
        ref = e @ P["w"].T + P["b"]
        unit = EPS24 * (K ** 0.5 * (e.abs() @ P["w"].abs().T) + ref.abs())
        worst = max(worst, (((kv[i].double() - ref).abs() - ulp_bf16(ref)) / unit).max().item())
    return worst


def test_cross_kv_store_vs_fp64():
    """Every decoder layer's K|V rows = bf16(enc . [Wk; Wv]^T + [0; bv]) within one bf16 ulp (plus the GEMM's fp32 term) for the
    whole store (192 clips), then for a sub-range written at clip0 > 0, whose neighbours must stay bitwise unchanged."""
    _cuda()
    m = _model("lv3w")
    sh = SHAPES["lv3w"]
    W = _weights64("lv3w", True)
    g = torch.Generator(device="cuda").manual_seed(5)
    full = torch.randn((MAX_BATCH_LV3W, 1500, sh.d_model), device="cuda", generator=g).bfloat16()
    _cross_kv(m, full, 0)
    sub = m.encode(_mel("lv3w", 3, seed=9))
    clip0 = 101
    before, excess = [], []
    for l in range(sh.dec_layers):
        _, kv = _read(m, -1, 0, MAX_BATCH_LV3W, l)
        excess.append(_kv_excess(kv, full, W["kv"][l]))
        print(f"cross K|V layer {l}, whole store: max (|err| - ulp) / unit = {excess[-1]:.3e}")
        before.append(kv)
    assert max(excess) <= GEMM_BF16_C, excess
    _cross_kv(m, sub, clip0)
    for l in range(sh.dec_layers):
        _, kv = _read(m, -1, 0, MAX_BATCH_LV3W, l)
        ex = _kv_excess(kv[clip0:clip0 + 3], sub, W["kv"][l])
        print(f"cross K|V layer {l}, clips {clip0}..{clip0 + 2}: max (|err| - ulp) / unit = {ex:.3e}")
        assert ex <= GEMM_BF16_C, (l, ex)
        keep = torch.ones(MAX_BATCH_LV3W, dtype=torch.bool, device="cuda")
        keep[clip0:clip0 + 3] = False
        assert torch.equal(kv[keep].view(torch.int16), before[l][keep].view(torch.int16)), l
        assert not torch.equal(kv[clip0:clip0 + 3], before[l][clip0:clip0 + 3])


# ============================================================================================ d. fused stage 1
def _parts(n_parts, B, seed):
    """int16 clips of different loudness with ragged n_valid (empty, short, partial and full rows)."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n_parts):
        pcm = synth_batch(seed * 10 + i, B).astype(np.float32)
        gain = 10.0 ** rng.uniform(-3.5, 0.3, size=(B, 1))
        nv = rng.integers(0, 480001, size=B).astype(np.int32)
        # every part: a quiet partial clip (its silent tail sits on the -10 floor, below clip_max - 8) and a loud short one (its
        # silent tail is lifted to clip_max - 8)
        gain[0], nv[0] = 10.0 ** -3.5, 200_000
        gain[-1], nv[-1] = 1.0, 12_345
        if B > 2:
            nv[1], nv[2] = 0, 480_000
        pcm = np.clip(np.rint(pcm * gain), -32768, 32767).astype(np.int16)
        out.append((torch.from_numpy(pcm).cuda(), nv))
    return out


@pytest.mark.parametrize("shape_name,B", [("micro128", 2), ("lv3w", 64)])
def test_fused_stage1_bitwise_vs_unfused(shape_name, B):
    """tw_pipeline_encode_at (log-mel without its second pass, the per-clip floor and (x + 4) / 4 applied in the conv-stem im2col,
    encoder and cross-K|V in the stage-1 SM partition) at clip0 = 0, B, 2B of slot 1: the encoder rows and every layer's K|V rows
    are bitwise those of tw_logmel -> tw_encode -> tw_debug_cross_kv on the whole device.  Restaging the middle part with other
    data leaves the other two bitwise unchanged."""
    _cuda()
    from tests.gpu_common import b200_model
    from taiwan_whisper_b200.host import log_mel
    sh = SHAPES[shape_name]
    m = _model(shape_name) if shape_name == "lv3w" else b200_model.__wrapped__(shape_name, "bf16", 3 * B, 1234, True)
    try:
        if shape_name == "lv3w":
            if getattr(m, "pipeline_unsupported", None):
                pytest.skip(f"no green contexts on this driver: {m.pipeline_unsupported}")
        else:
            try:
                m.enable_pipeline(16)
            except NotImplementedError as e:
                pytest.skip(f"no green contexts on this driver: {e}")
        h, ctx = C.c_void_p(m.handle), m.ctx
        slot = 1

        def stage(pcm, nv, clip0):
            torch.cuda.synchronize()
            ctx.check(ctx.lib.tw_pipeline_encode_at(h, pcm.data_ptr(), nv.ctypes.data_as(C.POINTER(C.c_int32)), B, slot, clip0))

        def fused(clip0):
            parts = [_read(m, slot, clip0, B, l, with_enc=(l == 0)) for l in range(sh.dec_layers)]
            return parts[0][0], [kv for _, kv in parts]

        def unfused(pcm, nv, clip0):
            mel = log_mel(pcm, torch.from_numpy(nv), sh.n_mel)
            enc = m.encode(mel)
            _cross_kv(m, enc, clip0)
            torch.cuda.synchronize()
            return mel, enc, [_read(m, -1, clip0, B, l)[1] for l in range(sh.dec_layers)]

        data = _parts(3, B, 3)
        for i, (pcm, nv) in enumerate(data):
            stage(pcm, nv, i * B)
        got = [fused(i * B) for i in range(3)]
        floors = set()
        for i, (pcm, nv) in enumerate(data):
            mel, enc, kvs = unfused(pcm, nv, i * B)
            lo, hi = mel.amin((1, 2)), mel.amax((1, 2))
            # the floor clip_max - 8 lands 2 below the clip's maximum after the (x + 4) / 4 scaling (up to fp32 rounding)
            floors |= {"clip_max - 8" for b in range(B) if abs(lo[b] - (hi[b] - 2.0)) < 1e-5 and hi[b] > 0.5}
            floors |= {"-10" for b in range(B) if lo[b] == -1.5 and hi[b] - 2.0 < -1.5}
            assert torch.equal(got[i][0].view(torch.int16), enc.view(torch.int16)), f"part {i}: encoder rows differ"
            for l in range(sh.dec_layers):
                assert torch.equal(got[i][1][l].view(torch.int16), kvs[l].view(torch.int16)), f"part {i}: K|V rows of layer {l} differ"
        assert floors == {"clip_max - 8", "-10"}, floors
        pcm, nv = _parts(1, B, 4)[0]
        stage(pcm, nv, B)
        again = [fused(i * B) for i in range(3)]
        for i in (0, 2):
            assert torch.equal(again[i][0].view(torch.int16), got[i][0].view(torch.int16)), i
            for l in range(sh.dec_layers):
                assert torch.equal(again[i][1][l].view(torch.int16), got[i][1][l].view(torch.int16)), (i, l)
        assert not torch.equal(again[1][0], got[1][0])
    finally:
        torch.cuda.synchronize()
        if shape_name != "lv3w":
            m.close()
