"""Helpers for the -m gpu parity tests (CUDA path through the C ABI vs the oracle)."""
import ctypes as C
import functools

import numpy as np
import torch

from oracle import hf_ref, logmel_np, whisper_np
from taiwan_whisper_b200 import lib as twlib
from taiwan_whisper_b200.configs import SHAPES
from taiwan_whisper_b200.synth import dequantise, synth_batch
from tests.helpers import default_rules, perturb_hf_model, prompt_ids, weights_np

EPS24 = 2.0 ** -24
# bf16 GEMMs (gemm_tc.cu) per element against fp64: |out - ref| <= [one bf16 ulp of ref, for bf16 outputs] + c * unit with
# unit = 2^-24 * (sqrt(K) * sum_k |a_k w_k| + |ref|): the fp32 accumulation and the fp32 epilogue.  The GELU epilogues (modes 1
# and 3) add 2^-24 * |a.w + b| to the unit for the erf approximation of gelu_erf_fast (A&S 7.1.26 with MUFU ex2 / rcp).
# c per output kind, measured on a B200 (1000 W power limit) over every shape of test_gemm_tcgen05_vs_torch (and, for bf16 stores,
# every clip of the cross-attention K|V store in test_gpu_encoder_stage); each bar is twice its largest measurement.  (For bf16
# outputs the one-ulp term dominates, so c stays small there.)
MEASURED_GEMM_BF16_C = 0.0706         # bf16 store: the K|V store, layer 0 (mode 0 of the GEMM test: 0.045)
GEMM_BF16_C = 0.14
MEASURED_GEMM_BF16_GELU_C = 0.0227    # bf16 GELU (mode 1)
GEMM_BF16_GELU_C = 0.046
MEASURED_GEMM_F32_C = 0.218           # fp32 accumulate / store (modes 2, 4)
GEMM_F32_C = 0.44
MEASURED_GEMM_F32_GELU_C = 0.248      # fp32 GELU + positions (mode 3)
GEMM_F32_GELU_C = 0.5


def ulp_bf16(x):
    """spacing of bf16 numbers at |x| (8 significant bits): 2^(e - 8) for |x| = f * 2^e, f in [0.5, 1)."""
    _, e = torch.frexp(x.abs().clamp_min(2.0 ** -126))
    return torch.exp2((e - 8).to(x.dtype))


def hf_model(shape_name, seed=1234, perturb=False):
    """HF model of the shape; perturb: with non-trivial biases and LayerNorms (tests.helpers.perturb_hf_model).  One cached model
    per (shape, seed, perturb), however the arguments are passed."""
    return _hf_model(shape_name, seed, perturb)


@functools.lru_cache(maxsize=None)
def _hf_model(shape_name, seed, perturb):
    m = hf_ref.build_hf_model(SHAPES[shape_name], seed=seed)
    return perturb_hf_model(m) if perturb else m


def b200_model(shape_name, dtype_name, max_batch=4, seed=1234, perturb=False):
    """The B200 model of hf_model(shape_name, seed, perturb); one cached model per argument set, however the arguments are passed.
    b200_model.__wrapped__(...) builds a private, uncached one."""
    return _b200_model(shape_name, dtype_name, max_batch, seed, perturb)


@functools.lru_cache(maxsize=None)
def _b200_model(shape_name, dtype_name, max_batch=4, seed=1234, perturb=False):
    from taiwan_whisper_b200.host import B200WhisperForConditionalGeneration
    dtype = {"f32": torch.float32, "bf16": torch.bfloat16}[dtype_name]
    # the oracle is transformers 5.x (generated ids only, seek loop on): the tests ask for that layout explicitly
    return B200WhisperForConditionalGeneration.from_hf(hf_model(shape_name, seed, perturb), dtype=dtype, max_batch=max_batch,
                                                       output_layout="5.x")


b200_model.__wrapped__ = _b200_model.__wrapped__


@functools.lru_cache(maxsize=None)
def oracle_run(shape_name, n_clips, max_length, timestamps=False, seed=1234, perturb=False):
    """Oracle (numpy restatement) outputs: mel, taps, enc, tokens, per-step post-rules logits."""
    sh = SHAPES[shape_name]
    W = weights_np(hf_model(shape_name, seed, perturb))
    pcm = synth_batch(0, n_clips)
    mel = logmel_np.log_mel(dequantise(pcm), sh.n_mel)
    out = []
    for b in range(n_clips):
        taps = []
        enc = whisper_np.encoder_forward(W, mel[b], sh.heads, sh.enc_layers, taps)
        lt = []
        toks = whisper_np.greedy_decode(W, enc, prompt_ids(sh.vocab, timestamps), default_rules(sh.vocab, timestamps),
                                        max_length, sh.heads, sh.dec_layers, logits_tap=lt)
        out.append(dict(taps=taps, enc=enc, tokens=toks, logits=lt))
    return pcm, mel, out


def gemm_debug(A, W, bias, mode, use_tc, out_dtype=None, C_init=None, pos=None, period=1):
    """Calls tw_debug_gemm on cuda tensors; returns C."""
    ctx = twlib.Context.get(torch.cuda.current_device())
    M, K = A.shape
    N = W.shape[0]
    dt = twlib.TW_BF16 if A.dtype == torch.bfloat16 else twlib.TW_F32
    if mode in (0, 1):
        Cc = torch.empty((M, N), dtype=A.dtype, device=A.device)
    else:
        Cc = C_init.clone() if C_init is not None else torch.zeros((M, N), dtype=torch.float32, device=A.device)
    ctx.check(ctx.lib.tw_debug_gemm(ctx.handle, A.data_ptr(), W.data_ptr(), bias.data_ptr() if bias is not None else None,
                                    Cc.data_ptr(), M, N, K, dt, mode, pos.data_ptr() if pos is not None else None, period,
                                    int(use_tc), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return Cc
