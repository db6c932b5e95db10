"""-m gpu: parity of the CUDA path (through the C ABI) with the oracle on the same seeded inputs.

Tolerances (north_star): log-mel 1e-4 abs; encoder hidden states 1e-4 in fp32 check mode and 2e-2
relative in bf16; greedy ids bit-identical in fp32 check mode; bf16 token agreement measured
teacher-forced (see DESIGN.md §parity for why free-running agreement is not defined for
random-init weights: the reference's own bf16 run agrees with its fp32 run on ~74 % of tokens).
"""
import os

import numpy as np
import pytest
import torch

from oracle import logmel_np
from taiwan_whisper_b200.configs import SHAPES, token_ids
from taiwan_whisper_b200.synth import dequantise, edge_case_clips, synth_batch
from tests.helpers import PERTURBED, default_rules, prompt_ids, split_shape

pytestmark = pytest.mark.gpu

LOGMEL_TOL = 1e-4


def _cuda():
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the -m gpu tests must run on a B200 (there is no CPU fallback)")


# ------------------------------------------------------------------------------------------ log-mel
@pytest.mark.parametrize("n_mel", [80, 128])
@pytest.mark.parametrize("in_dtype", ["i16", "f32"])
def test_logmel_vs_oracle(n_mel, in_dtype):
    _cuda()
    from taiwan_whisper_b200.host import log_mel
    clips = list(synth_batch(0, 3)) + list(edge_case_clips().values())
    pcm = np.stack(clips)
    ref = logmel_np.log_mel(dequantise(pcm), n_mel)
    x = torch.from_numpy(pcm if in_dtype == "i16" else dequantise(pcm)).cuda()
    out = log_mel(x, None, n_mel).cpu().numpy()
    assert out.shape == ref.shape and out.dtype == np.float32
    err = np.abs(out - ref).reshape(len(clips), -1).max(1)
    assert err.max() < LOGMEL_TOL, err
    assert np.all(out[3] == np.float32(-1.5))          # silence


def test_logmel_vs_golden(golden_dir):
    _cuda()
    from taiwan_whisper_b200.host import log_mel
    clips = {f"synth{i}": c for i, c in enumerate(synth_batch(0, 2))}
    clips.update(edge_case_clips())
    for n_mel in (80, 128):
        g = np.load(os.path.join(golden_dir, f"logmel_{n_mel}.npz"))
        x = torch.from_numpy(np.stack(list(clips.values()))).cuda()
        out = log_mel(x, None, n_mel).cpu().numpy()
        for i, name in enumerate(clips):
            assert np.abs(out[i][:, ::16] - g[name + "_sub"]).max() < LOGMEL_TOL, (n_mel, name)


def test_logmel_ragged_and_long():
    """short rows are zero-extended, long rows truncated to 30 s, n_valid masks the tail."""
    _cuda()
    from taiwan_whisper_b200.host import B200WhisperFeatureExtractor
    fe = B200WhisperFeatureExtractor(feature_size=80)
    a = dequantise(synth_batch(11, 1)[0])
    rows = [a[:80_000], a, np.concatenate([a, a[:1000]]), a[:12_345], np.zeros(0, np.float32)]
    out = fe(rows, sampling_rate=16000, return_tensors="np")["input_features"]
    ref = np.stack([logmel_np.log_mel(logmel_np.pad_or_trim(r), 80) for r in rows])
    assert out.shape == (5, 80, 3000)
    assert np.abs(out - ref).max() < LOGMEL_TOL
    with pytest.raises(ValueError):
        fe(rows[0], sampling_rate=8000)


def test_chunked_longform_logmel():
    """zero-copy windowing of a long recording (strided rows + n_valid) == log-mel of each padded window."""
    _cuda()
    from taiwan_whisper_b200.longform import chunk_plan, chunked_log_mel
    rec = np.concatenate([synth_batch(20, 2).reshape(-1), synth_batch(22, 1)[0][:123_456]])     # 67.7 s
    feats, strides = chunked_log_mel(torch.from_numpy(rec).cuda(), 80)
    starts, ref_strides = chunk_plan(len(rec))
    assert strides == ref_strides and feats.shape == (len(starts), 80, 3000)
    x = dequantise(rec)
    for i, st in enumerate(starts):
        ref = logmel_np.log_mel(logmel_np.pad_or_trim(x[st:st + 480000]), 80)
        assert np.abs(feats[i].cpu().numpy() - ref).max() < LOGMEL_TOL, i


def test_logmel_empty_batch():
    _cuda()
    from taiwan_whisper_b200.host import log_mel
    out = log_mel(torch.zeros((0, 480000), dtype=torch.int16, device="cuda"), None, 128)
    assert out.shape == (0, 128, 3000)


# ------------------------------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("M,N,K", [(128, 256, 128), (1500, 1280, 1280), (300, 384, 240), (64, 1280, 1280), (257, 520, 1536),
                                   (3000, 5120, 1280), (4, 51866, 384),
                                   # encoder dispatch shapes: tiny's qkv, micro128's fc1, medw's conv1, lv3w's conv2
                                   (3000, 128, 384), (1500, 128, 512), (3000, 1024, 240), (3000, 1280, 3840)])
@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
def test_gemm_tcgen05_vs_torch(M, N, K, mode):
    """tcgen05 GEMM and epilogues per element against fp64 (bars: tests.gpu_common); the CUDA-core kernel against fp32 torch."""
    _cuda()
    from tests import gpu_common as gc
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K + mode)
    A = (torch.randn((M, K), device="cuda", generator=g) * 0.5).bfloat16()
    W = (torch.randn((N, K), device="cuda", generator=g) * 0.05).bfloat16()
    bias = torch.randn((N,), device="cuda", generator=g) * 0.1
    C0 = torch.randn((M, N), device="cuda", generator=g)
    period = 1500 if (M, N, K) == (3000, 1280, 3840) else 100      # lv3w's conv2 epilogue adds positions[row % 1500]
    pos = torch.randn((period, N), device="cuda", generator=g)
    rows = torch.arange(M, device="cuda") % period
    out = gc.gemm_debug(A, W, bias, mode, True, C_init=C0, pos=pos, period=period)
    worst = -np.inf
    for r0 in range(0, M, 1024):                   # fp64 in row blocks: [M, N] float64 temporaries stay small
        sl = slice(r0, min(M, r0 + 1024))
        a, w = A[sl].double(), W.double()
        acc = a @ w.T + bias.double()
        unit = gc.EPS24 * K ** 0.5 * (a.abs() @ w.abs().T)
        ref = {0: acc, 1: torch.nn.functional.gelu(acc), 2: C0[sl].double() + acc,
               3: torch.nn.functional.gelu(acc) + pos[rows[sl]].double(), 4: acc}[mode]
        unit = unit + gc.EPS24 * ref.abs()
        if mode in (1, 3):
            unit = unit + gc.EPS24 * acc.abs()
        err = (out[sl].double() - ref).abs()
        if mode in (0, 1):
            err = err - gc.ulp_bf16(ref)
        worst = max(worst, (err / unit).max().item())
    c = {0: gc.GEMM_BF16_C, 1: gc.GEMM_BF16_GELU_C, 2: gc.GEMM_F32_C, 3: gc.GEMM_F32_GELU_C, 4: gc.GEMM_F32_C}[mode]
    print(f"gemm {M}x{N}x{K} mode {mode}: max (|err| - ulp) / unit = {worst:.3e}")
    assert worst <= c, (worst, c)
    acc = A.float() @ W.float().T + bias
    ref = {0: acc, 1: torch.nn.functional.gelu(acc), 2: C0 + acc, 3: torch.nn.functional.gelu(acc) + pos[rows], 4: acc}[mode]
    tol = 2e-2 if mode in (0, 1) else 2e-3          # bf16 output rounding vs fp32 output
    simt = gc.gemm_debug(A, W, bias, mode, False, C_init=C0, pos=pos, period=period).float()
    assert (simt - ref).abs().max().item() < tol * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("M,N,K", [(64, 1280, 1280), (64, 3840, 1280), (3, 5120, 1280), (64, 1280, 5120), (1, 51866, 1280),
                                   (5, 384, 384), (64, 128, 128), (2, 384, 1536), (64, 51865, 384), (7, 1152, 384),
                                   (128, 3840, 1280), (128, 1280, 5120), (128, 5120, 1280), (70, 1280, 1280), (65, 1152, 384),
                                   (130, 384, 1536), (192, 3840, 1280), (256, 1280, 5120), (200, 51866, 384)])
@pytest.mark.parametrize("mode", [0, 1, 2, 4])
def test_gemm_skinny_vs_torch(M, N, K, mode):
    """tcgen05 skinny GEMM of the decode steps (M <= 64 per row block; merged decode batches run 2-4 row blocks)."""
    _cuda()
    from tests.gpu_common import gemm_debug
    impl = 3
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K + mode)
    A = (torch.randn((M, K), device="cuda", generator=g) * 0.5).bfloat16()
    W = (torch.randn((N, K), device="cuda", generator=g) * 0.05).bfloat16()
    bias = torch.randn((N,), device="cuda", generator=g) * 0.1
    C0 = torch.randn((M, N), device="cuda", generator=g)
    acc = A.float() @ W.float().T + bias
    ref = {0: acc, 1: torch.nn.functional.gelu(acc), 2: C0 + acc, 4: acc}[mode]
    out = gemm_debug(A, W, bias, mode, impl, C_init=C0).float()
    tol = 2e-2 if mode in (0, 1) else 2e-3
    err = (out - ref).abs().max().item()
    assert err < tol * max(1.0, ref.abs().max().item()), (err, ref.abs().max().item())


def test_gemm_fp32_check_mode_vs_torch():
    _cuda()
    from tests.gpu_common import gemm_debug
    torch.backends.cuda.matmul.allow_tf32 = False
    g = torch.Generator(device="cuda").manual_seed(5)
    for (M, N, K) in [(130, 70, 33), (1500, 384, 384), (3, 51865, 128)]:
        A = torch.randn((M, K), device="cuda", generator=g)
        W = torch.randn((N, K), device="cuda", generator=g) * 0.05
        bias = torch.randn((N,), device="cuda", generator=g)
        ref = (A.double() @ W.double().T + bias.double()).float()
        out = gemm_debug(A, W, bias, 4, False)
        assert (out - ref).abs().max().item() < 1e-4


# ------------------------------------------------------------------------------------------ attention kernels
def _attn_ref(qkv, B, S, H):
    d = H * 64
    x = qkv.float().view(B, S, 3, H, 64)
    q, k, v = x[:, :, 0].transpose(1, 2), x[:, :, 1].transpose(1, 2), x[:, :, 2].transpose(1, 2)
    p = torch.softmax(q @ k.transpose(-1, -2), -1)
    return (p @ v).transpose(1, 2).reshape(B * S, d)


@pytest.mark.parametrize("B,S,H", [(2, 1500, 6), (1, 128, 2), (3, 200, 2), (1, 1500, 20)])
@pytest.mark.parametrize("impl", [0, 1])
def test_encoder_attention_kernels_vs_torch(B, S, H, impl):
    _cuda()
    from taiwan_whisper_b200 import lib as twlib
    ctx = twlib.Context.get(torch.cuda.current_device())
    d = H * 64
    g = torch.Generator(device="cuda").manual_seed(B * 100 + S + H)
    qkv = torch.randn((B * S, 3 * d), device="cuda", generator=g)
    qkv[:, :d] *= 0.3          # q is pre-scaled on the real path
    qkv = qkv.bfloat16()
    out = torch.zeros((B * S, d), device="cuda", dtype=torch.bfloat16)
    ctx.check(ctx.lib.tw_debug_encoder_attention(ctx.handle, qkv.data_ptr(), out.data_ptr(), B, S, H, twlib.TW_BF16, impl,
                                                 torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    ref = _attn_ref(qkv, B, S, H)
    err = (out.float() - ref).abs().max().item()
    assert err < 2e-2, err                       # bf16 P and bf16 output rounding


def test_encoder_attention_tc_repeated_runs():
    """The tcgen05 flash kernel at the shape that puts two CTAs on most SMs (20 heads x 1500 keys), 150 runs on fresh inputs:
    every run within tolerance.  Regression test for hazards between tcgen05 instructions on aliased tensor-memory columns
    (P V (j) reading P(j) while Q K^T (j+2) overwrites the score buffer it lives in), which corrupted a few rows in a few
    per cent of the launches."""
    _cuda()
    from taiwan_whisper_b200 import lib as twlib
    ctx = twlib.Context.get(torch.cuda.current_device())
    B, S, H = 1, 1500, 20
    d = H * 64
    bad = []
    for it in range(150):
        g = torch.Generator(device="cuda").manual_seed(1000 + it)
        qkv = torch.randn((B * S, 3 * d), device="cuda", generator=g)
        qkv[:, :d] *= 0.3
        qkv = qkv.bfloat16()
        out = torch.zeros((B * S, d), device="cuda", dtype=torch.bfloat16)
        ctx.check(ctx.lib.tw_debug_encoder_attention(ctx.handle, qkv.data_ptr(), out.data_ptr(), B, S, H, twlib.TW_BF16, 1,
                                                     torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        err = (out.float() - _attn_ref(qkv, B, S, H)).abs().max().item()
        if err >= 2e-2:
            bad.append((it, err))
    assert not bad, bad


@pytest.mark.parametrize("B,Sq,Sk,H,causal", [(3, 70, 70, 2, True), (2, 300, 300, 2, True), (1, 128, 128, 6, True),
                                              (3, 70, 1500, 6, False), (2, 129, 200, 2, False), (1, 448, 1500, 20, False)])
@pytest.mark.parametrize("impl,dtype", [(0, "f32"), (0, "bf16"), (1, "bf16")])
def test_general_attention_kernels_vs_torch(B, Sq, Sk, H, causal, impl, dtype):
    """Attention of the full-sequence decoder pass: separate query and key/value matrices with their own row pitches and
    column offsets (packed QKV for the causal self-attention, q vs the K|V store for the cross-attention)."""
    _cuda()
    from taiwan_whisper_b200 import lib as twlib
    ctx = twlib.Context.get(torch.cuda.current_device())
    tdt = torch.float32 if dtype == "f32" else torch.bfloat16
    d = 64 * H
    g = torch.Generator(device="cuda").manual_seed(B * 1000 + Sq + Sk + H)
    if causal:       # packed [B*S, 3d]: q | k | v
        qkv = (torch.randn((B * Sq, 3 * d), device="cuda", generator=g) * 0.5).to(tdt)
        q_t, q_ld, q_col0, kv_t, kv_ld, k_col0, v_col0 = qkv, 3 * d, 0, qkv, 3 * d, d, 2 * d
        qf = qkv[:, :d].float().view(B, Sq, H, 64)
        kf = qkv[:, d:2 * d].float().view(B, Sk, H, 64)
        vf = qkv[:, 2 * d:].float().view(B, Sk, H, 64)
    else:            # q [B*Sq, d] and a K|V store [B*Sk, 2d]
        q_t = (torch.randn((B * Sq, d), device="cuda", generator=g) * 0.5).to(tdt)
        kv_t = (torch.randn((B * Sk, 2 * d), device="cuda", generator=g) * 0.5).to(tdt)
        q_ld, q_col0, kv_ld, k_col0, v_col0 = d, 0, 2 * d, 0, d
        qf = q_t.float().view(B, Sq, H, 64)
        kf = kv_t[:, :d].float().view(B, Sk, H, 64)
        vf = kv_t[:, d:].float().view(B, Sk, H, 64)
    sc = torch.einsum("bqhd,bkhd->bhqk", qf, kf)
    if causal:
        sc = sc.masked_fill(torch.ones((Sq, Sk), device="cuda", dtype=torch.bool).triu(1), float("-inf"))
    ref = torch.einsum("bhqk,bkhd->bqhd", torch.softmax(sc, -1), vf).reshape(B * Sq, d)
    out = torch.full((B * Sq, d), 7.0, device="cuda", dtype=tdt)
    ctx.check(ctx.lib.tw_debug_attention(ctx.handle, q_t.data_ptr(), q_ld, q_col0, kv_t.data_ptr(), kv_ld, k_col0, v_col0, out.data_ptr(),
                                         B, Sq, Sk, H, twlib.TW_F32 if dtype == "f32" else twlib.TW_BF16, impl, int(causal),
                                         torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    err = (out.float() - ref).abs().max().item()
    assert err < (2e-5 if dtype == "f32" else 2e-2), err


@pytest.mark.parametrize("M,H,K,group_n", [(64, 20, 64, 1280), (64, 20, 1280, 64), (3, 6, 64, 384), (5, 6, 384, 64), (64, 2, 128, 64),
                                            (64, 16, 64, 1024)])
def test_gemm_grouped_vs_torch(M, H, K, group_n):
    """Grouped form of the skinny GEMM (absorbed cross-attention: q~_h = Wk_h^T q_h with K = 64, o_h = Wv_h c_h + bv_h with K = d)."""
    _cuda()
    from taiwan_whisper_b200 import lib as twlib
    ctx = twlib.Context.get(torch.cuda.current_device())
    N = H * group_n
    g = torch.Generator(device="cuda").manual_seed(M + H + K + group_n)
    A = (torch.randn((M, H * K), device="cuda", generator=g) * 0.5).bfloat16()
    W = (torch.randn((N, K), device="cuda", generator=g) * 0.05).bfloat16()
    bias = torch.randn((N,), device="cuda", generator=g) * 0.1
    out = torch.empty((M, N), device="cuda", dtype=torch.bfloat16)
    ctx.check(ctx.lib.tw_debug_gemm_grouped(ctx.handle, A.data_ptr(), W.data_ptr(), bias.data_ptr(), out.data_ptr(), M, N, K, group_n,
                                            torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    ref = torch.einsum("mhk,hnk->mhn", A.float().view(M, H, K), W.float().view(H, group_n, K)).reshape(M, N) + bias
    err = (out.float() - ref).abs().max().item()
    assert err < 2e-2 * max(1.0, ref.abs().max().item()), (err, ref.abs().max().item())


def _absorbed_ref(qt, enc, B, Tk, H):
    d = 64 * H
    E = enc.float().view(-1, Tk, d)[:B]
    q = qt.float()[:B * H].view(B, H, d)
    sc = torch.einsum("bhd,btd->bht", q, E)
    return torch.einsum("bht,btd->bhd", torch.softmax(sc, -1), E).reshape(B, H * d)


@pytest.mark.parametrize("Tk,B,H", [(1500, 64, 20), (1500, 3, 6), (1500, 32, 16), (200, 5, 2), (64, 1, 12), (1, 2, 8), (129, 7, 20)])
@pytest.mark.parametrize("rev", [0, 1])
def test_absorbed_attention_kernel_vs_torch(Tk, B, H, rev):
    """Absorbed cross-attention (absorb.cu): c[b, h] = softmax_k(q~[b, h] . E[b, k]) E[b] against torch fp32 on the same bf16 inputs;
    score magnitudes chosen so that the lazy reference maximum moves several times per clip."""
    _cuda()
    from taiwan_whisper_b200 import lib as twlib
    ctx = twlib.Context.get(torch.cuda.current_device())
    d = 64 * H
    g = torch.Generator(device="cuda").manual_seed(Tk * 3 + B * 5 + H)
    enc = torch.randn((B * Tk, d), device="cuda", generator=g).bfloat16()
    qt = torch.zeros((B * H + 24, d), device="cuda", dtype=torch.bfloat16)
    # per-(clip, head) scale: some heads nearly uniform, some peaked (scores up to ~ +-40)
    scale = torch.rand((B * H, 1), device="cuda", generator=g) * 8.0 / d ** 0.5
    qt[:B * H] = (torch.randn((B * H, d), device="cuda", generator=g) * scale).bfloat16()
    out = torch.zeros((B, H * d), device="cuda", dtype=torch.bfloat16)
    ctx.check(ctx.lib.tw_debug_absorbed_attention(ctx.handle, qt.data_ptr(), enc.data_ptr(), Tk, B, H, out.data_ptr(), None, None, rev,
                                                  torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    ref = _absorbed_ref(qt, enc, B, Tk, H)
    err = (out.float() - ref).abs().max().item()
    assert err < 2e-2 * max(1.0, ref.abs().max().item()), (err, ref.abs().max().item())


def test_absorbed_attention_active_list():
    """Only the clips of the compacted active list are streamed; their results equal the full run, the others are untouched."""
    _cuda()
    from taiwan_whisper_b200 import lib as twlib
    ctx = twlib.Context.get(torch.cuda.current_device())
    Tk, B, H = 1500, 9, 6
    d = 64 * H
    g = torch.Generator(device="cuda").manual_seed(77)
    enc = torch.randn((B * Tk, d), device="cuda", generator=g).bfloat16()
    qt = torch.zeros((B * H + 24, d), device="cuda", dtype=torch.bfloat16)
    qt[:B * H] = (torch.randn((B * H, d), device="cuda", generator=g) * 3.0 / d ** 0.5).bfloat16()
    act = [0, 3, 4, 8]
    active = torch.tensor(act + [0] * (B - len(act)), device="cuda", dtype=torch.int32)
    n_active = torch.tensor([len(act)], device="cuda", dtype=torch.int32)
    out = torch.full((B, H * d), 7.0, device="cuda", dtype=torch.bfloat16)
    ctx.check(ctx.lib.tw_debug_absorbed_attention(ctx.handle, qt.data_ptr(), enc.data_ptr(), Tk, B, H, out.data_ptr(), active.data_ptr(),
                                                  n_active.data_ptr(), 0, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    ref = _absorbed_ref(qt, enc, B, Tk, H)
    for b in range(B):
        if b in act:
            assert (out[b].float() - ref[b]).abs().max().item() < 2e-2 * max(1.0, ref.abs().max().item()), b
        else:
            assert (out[b].float() == 7.0).all(), b


@pytest.mark.parametrize("Tk,B,H", [(1500, 3, 6), (1, 2, 2), (37, 5, 20), (448, 64, 2)])
@pytest.mark.parametrize("entry", ["tw_debug_decode_attention", "tw_debug_self_attention"])
def test_decode_attention_kernel_vs_torch(Tk, B, H, entry):
    _cuda()
    from taiwan_whisper_b200 import lib as twlib
    ctx = twlib.Context.get(torch.cuda.current_device())
    d = H * 64
    g = torch.Generator(device="cuda").manual_seed(Tk + B + H)
    for dt, tw_dt, tol in ((torch.float32, twlib.TW_F32, 1e-4), (torch.bfloat16, twlib.TW_BF16, 1e-2)):
        stride = (Tk + 3) * 2 * d                    # clip stride larger than Tk rows (as the self-attention cache has)
        kv = torch.randn((B, Tk + 3, 2 * d), device="cuda", generator=g).to(dt)
        q = (torch.randn((B, d), device="cuda", generator=g) * 0.3).to(dt)
        out = torch.zeros((B, d), device="cuda", dtype=dt)
        ctx.check(getattr(ctx.lib, entry)(ctx.handle, q.data_ptr(), d, kv.data_ptr(), stride, Tk, B, H, tw_dt,
                                           out.data_ptr(), torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        x = kv[:, :Tk].float().view(B, Tk, 2, H, 64)
        sc = torch.einsum("bhd,bthd->bht", q.float().view(B, H, 64), x[:, :, 0])
        ref = torch.einsum("bht,bthd->bhd", torch.softmax(sc, -1), x[:, :, 1]).reshape(B, d)
        err = (out.float() - ref).abs().max().item()
        assert err < tol, (dt, err)


@pytest.mark.parametrize("Tk,B,H", [(1, 2, 2), (16, 3, 6), (37, 5, 20), (448, 7, 2)])
def test_paged_self_attention_vs_torch(Tk, B, H):
    """Decoder self-attention over the paged K|V cache with an arbitrary (shuffled) page table: 16 positions per page."""
    _cuda()
    from taiwan_whisper_b200 import lib as twlib
    ctx = twlib.Context.get(torch.cuda.current_device())
    d = H * 64
    pages_per_clip = (Tk + 15) // 16
    pt_stride = pages_per_clip + 2                      # table rows are longer than what a clip uses
    n_pages = B * pages_per_clip + 3
    g = torch.Generator(device="cuda").manual_seed(Tk * 31 + B + H)
    perm = torch.randperm(n_pages, device="cuda", generator=g)[:B * pages_per_clip].view(B, pages_per_clip)
    table = torch.full((B, pt_stride), -1, dtype=torch.int32, device="cuda")
    table[:, :pages_per_clip] = perm.to(torch.int32)
    for dt, tw_dt, tol in ((torch.float32, twlib.TW_F32, 1e-4), (torch.bfloat16, twlib.TW_BF16, 1e-2)):
        pool = torch.randn((n_pages, 16, 2 * d), device="cuda", generator=g).to(dt)
        q = (torch.randn((B, d), device="cuda", generator=g) * 0.3).to(dt)
        out = torch.zeros((B, d), device="cuda", dtype=dt)
        ctx.check(ctx.lib.tw_debug_self_attention_paged(ctx.handle, q.data_ptr(), d, pool.data_ptr(), table.data_ptr(), pt_stride, Tk, B,
                                                        H, tw_dt, out.data_ptr(), torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        kv = pool[perm.reshape(-1)].view(B, pages_per_clip * 16, 2 * d)[:, :Tk]          # gather each clip's logical rows
        x = kv.float().view(B, Tk, 2, H, 64)
        sc = torch.einsum("bhd,bthd->bht", q.float().view(B, H, 64), x[:, :, 0])
        ref = torch.einsum("bht,bthd->bhd", torch.softmax(sc, -1), x[:, :, 1]).reshape(B, d)
        err = (out.float() - ref).abs().max().item()
        assert err < tol, (dt, err)


# ------------------------------------------------------------------------------------------ encoder
@pytest.mark.parametrize("shape_name", ["tiny", "micro128", "tiny" + PERTURBED])
def test_encoder_fp32_check_mode(shape_name):
    _cuda()
    from tests.gpu_common import b200_model, oracle_run
    shape_name, perturb = split_shape(shape_name)
    sh = SHAPES[shape_name]
    pcm, mel, ora = oracle_run(shape_name, 2, 24, perturb=perturb)
    m = b200_model(shape_name, "f32", perturb=perturb)
    melt = torch.from_numpy(mel).cuda()
    for layer in range(sh.enc_layers + 1):
        enc, tap = m.encode(melt, tap_layer=layer)
        for b in range(2):
            ref = ora[b]["taps"][layer]
            err = np.abs(tap[b].cpu().numpy() - ref).max() / np.abs(ref).max()
            assert err < 1e-4, (layer, b, err)
    enc = m.encode(melt).cpu().numpy()
    for b in range(2):
        assert np.abs(enc[b] - ora[b]["enc"]).max() < 1e-4 * max(1.0, np.abs(ora[b]["enc"]).max())


@pytest.mark.parametrize("shape_name", ["tiny", "micro128"])
def test_encoder_bf16(shape_name):
    _cuda()
    from tests.gpu_common import b200_model, oracle_run
    pcm, mel, ora = oracle_run(shape_name, 2, 24)
    m = b200_model(shape_name, "bf16")
    enc = m.encode(torch.from_numpy(mel).cuda()).float().cpu().numpy()
    for b in range(2):
        ref = ora[b]["enc"]
        rel = np.linalg.norm(enc[b] - ref) / np.linalg.norm(ref)
        assert rel < 2e-2, rel


def test_encoder_rejects_wrong_length():
    _cuda()
    from tests.gpu_common import b200_model
    m = b200_model("micro128", "f32")
    with pytest.raises(ValueError):
        m.generate(torch.zeros((1, 128, 2999)), max_length=16, language="zh", task="transcribe")


# ------------------------------------------------------------------------------------------ decode
@pytest.mark.parametrize("shape_name", ["tiny", "micro128", "tiny" + PERTURBED])
@pytest.mark.parametrize("timestamps", [False, True])
def test_greedy_tokens_fp32_bit_identical(shape_name, timestamps):
    _cuda()
    from tests.gpu_common import b200_model, oracle_run
    shape_name, perturb = split_shape(shape_name)
    sh = SHAPES[shape_name]
    max_length = 40
    pcm, mel, ora = oracle_run(shape_name, 3, max_length, timestamps, perturb=perturb)
    m = b200_model(shape_name, "f32", perturb=perturb)
    ids = m.generate(torch.from_numpy(mel), max_length=max_length, num_beams=1, return_timestamps=timestamps,
                     language="zh", task="transcribe", seek_loop=False).numpy()
    for b in range(3):
        ref = ora[b]["tokens"]
        assert ids[b, :len(ref)].tolist() == ref, (b, ids[b].tolist(), ref)
        assert np.all(ids[b, len(ref):] == token_ids(sh.vocab).pad)
    # post-rules logits of the first steps (mask pattern identical, values within fp32 noise)
    enc = m.encode(torch.from_numpy(mel).cuda())
    toks, lens, tap = m.decode(enc, prompt_ids(sh.vocab, timestamps), max_length, timestamps, tap_steps=4)
    tap = tap.cpu().numpy()
    for s in range(4):
        for b in range(3):
            ref = ora[b]["logits"][s]
            assert np.array_equal(np.isneginf(tap[s, b]), np.isneginf(ref)), (s, b)
            fin = np.isfinite(ref)
            assert np.abs(tap[s, b][fin] - ref[fin]).max() < 1e-4


def test_greedy_tokens_fp32_full_length():
    """Maximum size: max_length = max_target_positions (448) — every page of the paged self-attention cache and every
    learned position are used; ids stay bit-identical to the oracle."""
    _cuda()
    from tests.gpu_common import b200_model, oracle_run
    sh = SHAPES["tiny"]
    pcm, mel, ora = oracle_run("tiny", 1, sh.max_target, False)
    m = b200_model("tiny", "f32")
    ids = m.generate(torch.from_numpy(mel), max_length=sh.max_target, num_beams=1, return_timestamps=False, language="zh",
                     task="transcribe").numpy()
    ref = ora[0]["tokens"]
    assert len(ref) > 300, len(ref)                       # random-init weights do not emit EOS early
    assert ids[0, :len(ref)].tolist() == ref
    with pytest.raises(ValueError):                        # HF: prompt + new tokens must fit max_target_positions
        m.generate(torch.from_numpy(mel), max_length=sh.max_target + 1, language="zh", task="transcribe")


def test_tokens_vs_hf_golden(golden_dir):
    _cuda()
    from tests.gpu_common import b200_model
    from taiwan_whisper_b200.host import B200WhisperFeatureExtractor
    for shape_name in ("tiny", "micro128"):
        g = np.load(os.path.join(golden_dir, f"model_{shape_name}.npz"))
        sh = SHAPES[shape_name]
        fe = B200WhisperFeatureExtractor(feature_size=sh.n_mel)
        feats = fe(list(dequantise(synth_batch(0, 2))), sampling_rate=16000, return_tensors="pt")["input_features"]
        m = b200_model(shape_name, "f32")
        ids = m.generate(feats, max_length=int(g["max_length"]), num_beams=1, return_timestamps=False, language="zh",
                         task="transcribe").cpu().numpy()
        ref = g["tokens_nots"]
        assert ids.shape == ref.shape and np.array_equal(ids, ref)


def test_timestamp_seek_loop_vs_hf_golden(golden_dir):
    """return_timestamps=True: the host seek loop around the CUDA window primitive reproduces transformers 5.5's output
    (several encoder/decoder passes per clip) token for token; seek_loop=False gives the single-window decode."""
    _cuda()
    from tests.gpu_common import b200_model, oracle_run
    from taiwan_whisper_b200.host import B200WhisperFeatureExtractor
    for shape_name in ("tiny", "micro128"):
        g = np.load(os.path.join(golden_dir, f"model_{shape_name}.npz"))
        sh = SHAPES[shape_name]
        fe = B200WhisperFeatureExtractor(feature_size=sh.n_mel)
        feats = fe(list(dequantise(synth_batch(0, 2))), sampling_rate=16000, return_tensors="pt")["input_features"]
        m = b200_model(shape_name, "f32")
        max_length = int(g["max_length"])
        ids = m.generate(feats, max_length=max_length, num_beams=1, return_timestamps=True, language="zh",
                         task="transcribe").cpu().numpy()
        ref = g["tokens_ts_seekloop"]
        assert ids.shape == ref.shape and np.array_equal(ids, ref), (shape_name, ids.tolist(), ref.tolist())
        single = m.generate(feats, max_length=max_length, num_beams=1, return_timestamps=True, language="zh",
                            task="transcribe", seek_loop=False).cpu().numpy()
        pcm, mel, ora = oracle_run(shape_name, 2, max_length, True)
        for b in range(2):
            t = ora[b]["tokens"]
            assert single[b, :len(t)].tolist() == t


@pytest.mark.parametrize("shape_name", ["tiny", "micro128", "tiny" + PERTURBED])
def test_tokens_bf16_teacher_forced(shape_name):
    """bf16: feed the oracle's fp32 tokens back (teacher forcing) and compare the per-step argmax.
    Positions whose fp32 top-1/top-2 margin is below the bf16 noise floor are excluded from the 99.5 % bar
    (and counted separately)."""
    _cuda()
    from tests.gpu_common import b200_model, oracle_run
    shape_name, perturb = split_shape(shape_name)
    sh = SHAPES[shape_name]
    max_length = 64
    pcm, mel, ora = oracle_run(shape_name, 3, max_length, False, perturb=perturb)
    m = b200_model(shape_name, "bf16", perturb=perturb)
    P = prompt_ids(sh.vocab, False)
    n_gen = max_length - len(P)
    forced = torch.tensor([o["tokens"][:n_gen] for o in ora], dtype=torch.int32)
    enc = m.encode(torch.from_numpy(mel).cuda())
    toks, lens = m.decode(enc, P, max_length, False, forced=forced)
    toks = toks.cpu().numpy()
    agree = solid = solid_agree = 0
    for b in range(3):
        for s in range(n_gen):
            lg = ora[b]["logits"][s]
            top2 = np.partition(lg[np.isfinite(lg)], -2)[-2:]
            margin = top2[1] - top2[0]
            ok = toks[b, s] == ora[b]["tokens"][s]
            agree += ok
            if margin > 0.02:
                solid += 1
                solid_agree += ok
    total = 3 * n_gen
    print(f"bf16 teacher-forced agreement {agree}/{total}; margin>0.02: {solid_agree}/{solid}")
    assert solid > 0 and solid_agree / solid >= 0.995
    assert agree / total >= 0.80


@pytest.mark.parametrize("shape_name", ["tiny", "micro128", "tiny" + PERTURBED])
def test_teacher_logits_fp32_vs_oracle_and_golden(golden_dir, shape_name):
    """tw_decoder_logits (teacher forward of the distillation step) in fp32 check mode: every position's logits vs the
    oracle and vs the HF golden fixture (the fixture's model only: a perturbed model is compared with the oracle)."""
    _cuda()
    from tests.gpu_common import b200_model, hf_model
    from oracle import whisper_np
    from tests.helpers import weights_np
    shape_name, perturb = split_shape(shape_name)
    g = np.load(os.path.join(golden_dir, f"teacher_{shape_name}.npz"))
    sh = SHAPES[shape_name]
    m = b200_model(shape_name, "f32", perturb=perturb)
    mel = logmel_np.log_mel(dequantise(synth_batch(0, 2)), sh.n_mel)
    out = m(input_features=torch.from_numpy(mel), labels=torch.from_numpy(g["labels"]))
    lg = out.logits.cpu().numpy()
    assert lg.shape == (2, g["labels"].shape[1], sh.vocab) and lg.dtype == np.float32
    if not perturb:
        assert np.abs(lg[:, :, ::97] - g["logits_sub"]).max() < 1e-4
    W = weights_np(hf_model(shape_name, perturb=perturb))
    enc = out.encoder_last_hidden_state.float().cpu().numpy()
    ref = whisper_np.teacher_logits(W, enc[0], g["decoder_input_ids"][0], sh.heads, sh.dec_layers)
    assert np.abs(lg[0] - ref).max() < 1e-4
    # the shared-encoder form of the call: teacher_model(encoder_outputs=..., labels=...)
    out2 = m(encoder_outputs=(out.encoder_last_hidden_state,), labels=torch.from_numpy(g["labels"]))
    assert torch.equal(out2.logits, out.logits)


@pytest.mark.parametrize("shape_name,T", [("tiny", 24), ("micro128", 70)])
def test_teacher_logits_bf16(shape_name, T):
    """bf16 product path (tcgen05 GEMMs at M = B*T rows, TMA-stored fp32 logits with a padded row pitch): relative L2 of
    the logits vs the fp32 oracle, and the full-sequence pass must agree with the KV-cached step decoder fed the same
    tokens (same kernels' arithmetic, different schedule)."""
    _cuda()
    from tests.gpu_common import b200_model, oracle_run, hf_model
    from oracle import whisper_np
    from tests.helpers import weights_np
    sh = SHAPES[shape_name]
    P = prompt_ids(sh.vocab, False)
    pcm, mel, ora = oracle_run(shape_name, 3, 64, False)
    rows = [(P + o["tokens"] + [0] * T)[:T] for o in ora]
    dec = torch.tensor(rows, dtype=torch.int64)
    m = b200_model(shape_name, "bf16")
    enc = m.encode(torch.from_numpy(mel).cuda())
    lg = m.decoder_logits(enc, dec).cpu().numpy()
    assert lg.shape == (3, T, sh.vocab)
    W = weights_np(hf_model(shape_name))
    for b in range(3):
        ref = whisper_np.teacher_logits(W, ora[b]["enc"], rows[b], sh.heads, sh.dec_layers)
        rel = np.linalg.norm(lg[b] - ref) / np.linalg.norm(ref)
        assert rel < 2e-2, (b, rel)
    # teacher-forced step decode: position len(P)-1+s of the full pass predicts generated token s
    n_gen = T - len(P)
    forced = torch.tensor([(o["tokens"] + [0] * T)[:n_gen] for o in ora], dtype=torch.int32)
    toks, lens = m.decode(enc, P, T, False, forced=forced)
    toks = toks.cpu().numpy()
    r = default_rules(sh.vocab, False)
    agree = total = 0
    for b in range(3):
        for s in range(min(n_gen, len(ora[b]["tokens"]))):
            row = lg[b, len(P) - 1 + s].copy()
            row[np.asarray(r["suppress"])] = -np.inf
            if s == 0:
                row[np.asarray(r["begin_suppress"])] = -np.inf
            top2 = np.sort(row)[-2:]
            if top2[1] - top2[0] > 0.02:
                total += 1
                agree += int(np.argmax(row) == toks[b, s])
    assert total > 20 and agree / total >= 0.995, (agree, total)


def test_teacher_logits_argument_errors():
    _cuda()
    from tests.gpu_common import b200_model
    m = b200_model("tiny", "f32")
    enc = torch.zeros((1, 1500, 384), device="cuda")
    with pytest.raises(ValueError):
        m.decoder_logits(enc, torch.zeros((1, 449), dtype=torch.int64))          # > max_target_positions
    with pytest.raises(ValueError):
        m()                                                                        # neither features nor encoder outputs
    with pytest.raises(ValueError):
        m(encoder_outputs=(enc,))                                                  # neither ids nor labels


def test_transcribe_host_path_matches_generate():
    _cuda()
    from tests.gpu_common import b200_model, oracle_run
    shape_name = "micro128"
    sh = SHAPES[shape_name]
    max_length = 32
    pcm, mel, ora = oracle_run(shape_name, 3, 40, False)
    m = b200_model(shape_name, "f32")
    toks, lens = m.transcribe_pcm(torch.from_numpy(pcm).pin_memory(), max_length)
    for b in range(3):
        n = max_length - 4
        assert toks[b, :n].tolist() == ora[b]["tokens"][:n]
    ms = m.last_stage_ms()
    assert ms["total"] > 0 and ms["encoder"] > 0


@pytest.mark.parametrize("dtype_name", ["f32", "bf16"])
def test_pipelined_batch_loop_matches_sequential(dtype_name):
    """transcribe_batches (stage 1 of batch i+1 on a small SM partition while batch i decodes on the rest, tw_pipeline_*) returns,
    batch by batch, what the one-call path returns: ids equal to the oracle's in fp32 check mode; in bf16 the same lengths and the
    same ids as transcribe_pcm wherever the two free-running decodes have not parted at a near-tie (the K|V stream is split over a
    different number of CTAs, so partial sums round differently)."""
    _cuda()
    from tests.gpu_common import b200_model, oracle_run
    shape_name = "micro128"
    max_length = 32
    n = max_length - 4
    pcm, mel, ora = oracle_run(shape_name, 3, 40, False)
    m = b200_model.__wrapped__(shape_name, dtype_name)       # a private model: enabling the pipeline allocates the second buffer set
    try:
        sms = m.enable_pipeline(16)
    except NotImplementedError as e:
        pytest.skip(f"no green contexts on this driver: {e}")
    assert sms[0] >= 8 and sms[0] + sms[1] <= torch.cuda.get_device_properties(0).multi_processor_count
    host = torch.from_numpy(pcm).pin_memory()
    # five batches: host and device inputs, a short last batch, clips in a different order per batch
    orders = [[0, 1, 2], [2, 0, 1], [1, 2, 0], [0, 2, 1], [1, 0]]
    batches = [host[o].pin_memory() if i % 2 == 0 else host[o].cuda() for i, o in enumerate(orders)]
    seq = [m.transcribe_pcm(host[o].pin_memory(), max_length) for o in orders]
    seq = [(t.clone(), l.clone()) for t, l in seq]
    got = list(m.transcribe_batches(batches, max_length))
    assert len(got) == len(orders)
    for o, (toks, lens), (st, sl) in zip(orders, got, seq):
        assert toks.shape == (len(o), n) and lens.tolist() == sl.tolist()
        for j, b in enumerate(o):
            if dtype_name == "f32":
                assert toks[j].tolist() == ora[b]["tokens"][:n], (o, j)
            else:
                agree = (toks[j] == st[j]).float().mean().item()
                assert toks[j, :4].tolist() == st[j, :4].tolist() and agree >= 0.5, (o, j, agree)
    ms = m.last_stage_ms()
    assert ms["encoder"] > 0 and ms["decode"] > 0
    # merged decode: groups of 2 / 3 batches decoded as one batch (max_batch 4: [3] | [3] ... cannot merge, so use 2-clip batches)
    small = [[0, 1], [2, 0], [1, 2], [0, 2], [1]]
    sb = [host[o].pin_memory() if i % 2 else host[o].cuda() for i, o in enumerate(small)]
    sseq = [tuple(x.clone() for x in m.transcribe_pcm(host[o].pin_memory(), max_length)) for o in small]
    for merge in (2, 3):
        got = list(m.transcribe_batches(sb, max_length, merge=merge))
        assert len(got) == len(small)
        for o, (toks, lens), (st, sl) in zip(small, got, sseq):
            assert toks.shape == (len(o), n) and lens.tolist() == sl.tolist()
            for j, b in enumerate(o):
                if dtype_name == "f32":
                    assert toks[j].tolist() == ora[b]["tokens"][:n], (merge, o, j)
                else:
                    agree = (toks[j] == st[j]).float().mean().item()
                    assert toks[j, :4].tolist() == st[j, :4].tolist() and agree >= 0.5, (merge, o, j, agree)
    # moving the partition boundary (tw_pipeline_resize) and the balance controller: same ids whatever the split
    sms2 = m.enable_pipeline(32)
    assert sms2[0] == 32 and sms2[0] + sms2[1] == sms[0] + sms[1]
    assert m.pipeline_stage_ms(0)[0] != 0.0
    for auto in (False, True):
        got = list(m.transcribe_batches(sb, max_length, merge=2, auto_sms=auto))
        for o, (toks, lens), (st, sl) in zip(small, got, sseq):
            assert lens.tolist() == sl.tolist()
            for j, b in enumerate(o):
                if dtype_name == "f32":
                    assert toks[j].tolist() == ora[b]["tokens"][:n], (auto, o, j)
                else:
                    assert toks[j, :4].tolist() == st[j, :4].tolist(), (auto, o, j)
    t_enc, t_dec = m.pipeline_stage_ms(0)
    assert t_enc > 0 and t_dec > 0
    # the one-call path still works on the whole GPU afterwards
    t2, _ = m.transcribe_pcm(host[orders[0]].pin_memory(), max_length)
    assert t2.tolist() == seq[0][0].tolist()


def test_generate_argument_errors():
    _cuda()
    from tests.gpu_common import b200_model
    m = b200_model("micro128", "f32")
    f = torch.zeros((1, 128, 3000))
    with pytest.raises(NotImplementedError):
        m.generate(f, max_length=16, num_beams=4, language="zh", task="transcribe")
    with pytest.raises(ValueError):
        m.generate(f, max_length=16, language="xx-unknown", task="transcribe")
    with pytest.raises(ValueError):
        m.generate(f, max_length=1000, language="zh", task="transcribe")


def test_torch_ops_registered():
    _cuda()
    import taiwan_whisper_b200.host  # noqa: F401
    x = torch.from_numpy(synth_batch(0, 1)).cuda()
    out = torch.ops.twb200.log_mel(x, None, 80)
    assert out.shape == (1, 80, 3000)
    nv = torch.tensor([16000], dtype=torch.int32, device="cuda")          # n_valid: only the first second is audio
    short = torch.ops.twb200.log_mel(x, nv, 80)
    x0 = x.clone(); x0[:, 16000:] = 0
    assert torch.equal(short, torch.ops.twb200.log_mel(x0, None, 80))
    # model-level ops take the raw tw_model* (what model_create returns); no Python object is involved
    from tests.gpu_common import b200_model, hf_model
    from taiwan_whisper_b200 import lib as twlib
    sh = SHAPES["tiny"]
    sd = {k: v.detach().cuda() for k, v in hf_model("tiny").state_dict().items() if k.startswith("model.")}
    desc = [sh.d_model, sh.ffn, sh.heads, sh.enc_layers, sh.dec_layers, sh.n_mel, sh.vocab, sh.max_target, twlib.TW_F32, 2]
    h = torch.ops.twb200.model_create(desc, "\n".join(sd.keys()), list(sd.values()))
    assert isinstance(h, int) and h != 0
    try:
        m = b200_model("tiny", "f32")
        enc = torch.ops.twb200.encoder_forward(h, out)
        assert torch.equal(enc, m.encode(out))
        P = prompt_ids(sh.vocab, False)
        r = m._rules(False)
        packed = torch.ops.twb200.greedy_generate(h, enc, P, 16, r["suppress"], r["begin_suppress"], r["eos"], r["pad"], -1,
                                                  r["no_timestamps"], -1 if r["max_initial_ts"] is None else r["max_initial_ts"])
        toks, lens = m.decode(enc, P, 16, False)
        assert torch.equal(packed[:, :-1], toks) and torch.equal(packed[:, -1], lens)
        ids = torch.tensor([P + [11, 12, 13]], device="cuda")
        lg = torch.ops.twb200.decoder_logits(h, enc, ids)
        assert lg.shape == (1, 7, sh.vocab) and lg.is_contiguous() and torch.equal(lg, m.decoder_logits(enc, ids))
        # the class's own handle is the same kind of object
        assert torch.equal(torch.ops.twb200.encoder_forward(m.handle, out), enc)
    finally:
        torch.ops.twb200.model_free(h)


@pytest.mark.parametrize("chunk_length", [30, 7])
def test_first_pass_pipeline(chunk_length):
    """B200BatchedInferencePipeline (initial_inference.py's `pipeline.transcribe`): zero-copy fixed-window features equal
    the oracle's log-mel of the zero-padded windows, and the segments carry the window's greedy timestamp-mode tokens."""
    _cuda()
    from tests.gpu_common import b200_model
    from taiwan_whisper_b200.pipeline import B200BatchedInferencePipeline, segments_from_tokens
    sh = SHAPES["tiny"]
    m = b200_model("tiny", "f32")
    rec = np.concatenate([c for c in synth_batch(0, 3)])[: 16000 * 70 + 123]            # 70 s and a bit, int16
    pipe = B200BatchedInferencePipeline(m, decode_fn=lambda ids: ",".join(map(str, ids)), chunk_length=chunk_length, max_length=40)
    L = chunk_length * 16000
    n_win = -(-len(rec) // L)
    feats = pipe.window_features(torch.from_numpy(rec).cuda())
    assert feats.shape == (n_win, sh.n_mel, 3000)
    for w in (0, n_win - 1):
        win = np.zeros(480000, np.float32)
        piece = dequantise(rec[w * L:(w + 1) * L])
        win[:len(piece)] = piece
        assert np.abs(feats[w].cpu().numpy() - logmel_np.log_mel(win[None], sh.n_mel)[0]).max() < LOGMEL_TOL
    segs, info = pipe.transcribe(rec, batch_size=3)
    segs = list(segs)
    assert info.n_windows == n_win and abs(info.duration - len(rec) / 16000) < 1e-6
    ids = m.generate(feats[:3], max_length=40, return_timestamps=True, language="zh", task="transcribe", seek_loop=False).cpu().numpy()
    ref = []
    ti = token_ids(sh.vocab)
    for w in range(min(3, n_win)):                    # the first batch of windows (the model instance holds 4 rows)
        w_len = min(float(chunk_length), len(rec) / 16000 - w * chunk_length)
        ref += segments_from_tokens(ids[w], ti.timestamp_begin, ti.eos, w * float(chunk_length), w_len)
    assert [(s.start, s.end, s.tokens) for s in segs][:len(ref)] == ref
    for s in segs:
        assert 0.0 <= s.start <= s.end <= len(rec) / 16000 + 1e-6 and s.text == ",".join(map(str, s.tokens))


@pytest.mark.parametrize("shape_name,dtype_name", [("tiny", "f32"), ("micro128", "bf16")])
def test_workspace_bytes_matches_allocation(shape_name, dtype_name):
    """tw_workspace_bytes (host arithmetic) == what tw_model_load actually allocated."""
    _cuda()
    from taiwan_whisper_b200 import lib as twlib
    from tests.gpu_common import b200_model
    sh = SHAPES[shape_name]
    m = b200_model(shape_name, dtype_name)
    desc = twlib.ModelDesc(sh.d_model, sh.ffn, sh.heads, sh.enc_layers, sh.dec_layers, sh.n_mel, sh.vocab, sh.max_target,
                           twlib.TW_F32 if dtype_name == "f32" else twlib.TW_BF16, m.max_batch)
    assert int(m.ctx.lib.tw_workspace_bytes(desc)) == m.device_bytes()
