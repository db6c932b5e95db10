// Token selection on the device: logits rules + argmax + finished/pad bookkeeping, one CTA per row,
// one pass over the 51,865/51,866-wide fp32 logits with warp-shuffle reductions.  No host sync per token
// (the reference syncs every token at generation/utils.py:2805 and B times per token inside
// WhisperTimeStampLogitsProcessor, logits_process.py:2002-2004).
//
// Rules restated from transformers/generation/logits_process.py:
//   SuppressTokensAtBeginLogitsProcessor :1855-1863, SuppressTokensLogitsProcessor :1896-1903,
//   WhisperTimeStampLogitsProcessor :1996-2044; order per generation_whisper.py:1774-1812.
// Selection / finish logic: generation/utils.py:2793-2805 (argmax, first max wins; finished rows emit pad).
#include "kernels.cuh"

namespace tw {

constexpr int SEL_THREADS = 1024;

struct Best {
    float v;
    int i;
};
__device__ __forceinline__ Best better(Best a, Best b) {          // first index wins ties
    if (b.v > a.v || (b.v == a.v && b.i < a.i)) return b;
    return a;
}
__device__ __forceinline__ Best warp_best(Best x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        Best y;
        y.v = __shfl_xor_sync(0xffffffffu, x.v, o);
        y.i = __shfl_xor_sync(0xffffffffu, x.i, o);
        x = better(x, y);
    }
    return x;
}
// (max, sum exp(x - max)) pairs for a streaming logsumexp
__device__ __forceinline__ void lse_merge(float& m, float& s, float m2, float s2) {
    const float mn = fmaxf(m, m2);
    if (mn == -INFINITY) { m = mn; s = 0.0f; return; }
    s = s * __expf(m - mn) + s2 * __expf(m2 - mn);
    m = mn;
}

// masked score of token i for this row (everything except the "timestamps dominate" rule)
__device__ __forceinline__ float masked_score(float raw, bool suppressed, int i, const RulesDev& R, bool first, bool ts_mode,
                                              bool last_ts, bool pen_ts, int ts_forbid_end) {
    if (suppressed) return -INFINITY;
    if (ts_mode) {
        if (i == R.no_timestamps) return -INFINITY;
        if (last_ts) {
            if (pen_ts) { if (i >= R.ts_begin) return -INFINITY; }
            else { if (i < R.eos) return -INFINITY; }
        }
        if (i >= R.ts_begin && i < ts_forbid_end) return -INFINITY;
        if (first) {
            if (i < R.ts_begin) return -INFINITY;
            if (R.max_initial_ts >= 0 && i > R.ts_begin + R.max_initial_ts) return -INFINITY;
        }
    }
    return raw;
}

__global__ void __launch_bounds__(SEL_THREADS)
select_tokens_kernel(const float* __restrict__ logits, int64_t ld_logits, int V, const int32_t* __restrict__ d_step, RulesDev R, DecodeState S,
                     int32_t* __restrict__ out_tokens, int32_t* __restrict__ out_lengths, const int32_t* __restrict__ forced,
                     float* __restrict__ logits_tap) {
    __shared__ Best s_text[32], s_ts[32];
    __shared__ float s_m[32], s_s[32];
    __shared__ int s_dom;
    pdl_trigger();
    pdl_wait();
    const int b = blockIdx.x;
    const int pos = d_step[STEP_POS], P = d_step[STEP_P], out_stride = d_step[STEP_STRIDE];
    const int gen_index = pos - (P - 1);
    if (gen_index < 0) {                       // still consuming the forced prompt: feed the next prompt token
        if (threadIdx.x == 0) S.cur_tok[b] = S.prompt[b * PROMPT_MAX + pos + 1];
        return;
    }
    if (gen_index >= out_stride) return;
    if (S.finished[b] != 0 && !logits_tap) {     // a finished row emits pad and feeds pad; its logits are not read
        if (threadIdx.x == 0) {
            out_tokens[(int64_t)b * out_stride + gen_index] = R.pad;
            S.cur_tok[b] = R.pad;
        }
        return;
    }
    if (logits_tap) logits_tap = (gen_index < d_step[STEP_TAP]) ? logits_tap + (int64_t)gen_index * gridDim.x * V : nullptr;
    const float* row = logits + (int64_t)b * ld_logits;
    const bool ts_mode = R.ts_begin >= 0;
    const int n_hist = S.n_gen[b];
    const bool first = (n_hist == 0);
    bool last_ts = false, pen_ts = false;
    int ts_forbid_end = 0;
    if (ts_mode) {
        const int lt = S.last_tok[b], pt = S.prev_tok[b], lts = S.last_ts[b];
        last_ts = n_hist >= 1 && lt >= R.ts_begin;
        pen_ts = n_hist < 2 || pt >= R.ts_begin;
        if (lts >= 0) ts_forbid_end = (last_ts && !pen_ts) ? lts : lts + 1;
    }
    const int split = ts_mode ? R.ts_begin : V;     // [0,split) text, [split,V) timestamps

    Best bt = {-INFINITY, 0x7fffffff}, bs = {-INFINITY, 0x7fffffff};
    float lm = -INFINITY, ls = 0.0f;
    // Four consecutive tokens per load (float4 logits, 4 mask bytes as one word each), U such groups in flight per thread, every
    // load issued unconditionally before the first use.  The first version loaded scalars and short-circuited the two mask bytes
    // (`suppress || (first && begin)`): the second byte load hung on the first one's result, 16 dependent L2 round trips per
    // iteration — 36 us per token for 13 MB (ncu source page: every stall sample on the mask tests), now bandwidth-shaped.
    // Rows are 16-byte aligned (ld_logits % 4 == 0) and padded to a multiple of 4 floats; the masks are padded likewise.
    constexpr int U = 4;
    const int V4 = (V + 3) >> 2;                       // groups of 4 tokens
    const float4* row4 = reinterpret_cast<const float4*>(row);
    const uint32_t* sup4 = reinterpret_cast<const uint32_t*>(R.suppress_mask);
    const uint32_t* beg4 = reinterpret_cast<const uint32_t*>(R.begin_suppress_mask);
    for (int base = threadIdx.x; base < V4; base += SEL_THREADS * U) {
        float4 raw[U];
        uint32_t sm[U], bm[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int g = min(base + u * SEL_THREADS, V4 - 1);      // clamped: the duplicate group is skipped below
            raw[u] = __ldg(row4 + g);
            sm[u] = __ldg(sup4 + g);
            bm[u] = __ldg(beg4 + g);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int g = base + u * SEL_THREADS;
            if (g >= V4) continue;
            const uint32_t mask = first ? (sm[u] | bm[u]) : sm[u];
            const float r4[4] = {raw[u].x, raw[u].y, raw[u].z, raw[u].w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int i = 4 * g + j;
                if (i >= V) continue;
                const float v = masked_score(r4[j], ((mask >> (8 * j)) & 0xffu) != 0, i, R, first, ts_mode, last_ts, pen_ts, ts_forbid_end);
                if (i < split) {
                    bt = better(bt, Best{v, i});
                } else {
                    bs = better(bs, Best{v, i});
                    if (v > -INFINITY) lse_merge(lm, ls, v, 1.0f);
                }
            }
        }
    }
    bt = warp_best(bt);
    bs = warp_best(bs);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float m2 = __shfl_xor_sync(0xffffffffu, lm, o), s2 = __shfl_xor_sync(0xffffffffu, ls, o);
        lse_merge(lm, ls, m2, s2);
    }
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { s_text[w] = bt; s_ts[w] = bs; s_m[w] = lm; s_s[w] = ls; }
    __syncthreads();
    if (w == 0) {
        bt = s_text[lane]; bs = s_ts[lane]; lm = s_m[lane]; ls = s_s[lane];
        bt = warp_best(bt);
        bs = warp_best(bs);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float m2 = __shfl_xor_sync(0xffffffffu, lm, o), s2 = __shfl_xor_sync(0xffffffffu, ls, o);
            lse_merge(lm, ls, m2, s2);
        }
        if (lane == 0) {
            // log_softmax's normaliser cancels on both sides of logsumexp(ts) > max(text)
            const float lse_ts = (ls > 0.0f) ? lm + logf(ls) : -INFINITY;
            const bool dominate = ts_mode && (lse_ts > bt.v);
            Best pick = dominate ? bs : better(bt, bs);
            int tok = pick.i;
            if (pick.v == -INFINITY) tok = dominate ? split : 0;   // everything masked: torch.argmax returns 0 / first ts
            const bool was_finished = S.finished[b] != 0;
            if (was_finished) tok = R.pad;
            out_tokens[(int64_t)b * out_stride + gen_index] = tok;
            int nxt = forced ? forced[(int64_t)b * out_stride + gen_index] : tok;
            // per-row token budget (test / bench hook): the row ends here as if this token had been followed by EOS
            const bool budget_end = S.row_budget && gen_index + 1 >= S.row_budget[b];
            if (!was_finished) {
                if (nxt == R.eos) {
                    S.finished[b] = 1;
                    out_lengths[b] = (tok == R.eos) ? gen_index : gen_index + 1;
                    atomicSub(S.n_unfinished, 1);
                } else {
                    out_lengths[b] = gen_index + 1;
                    S.prev_tok[b] = S.last_tok[b];
                    S.last_tok[b] = nxt;
                    if (ts_mode && nxt >= R.ts_begin) S.last_ts[b] = nxt;
                    S.n_gen[b] = n_hist + 1;
                    if (budget_end) {
                        S.finished[b] = 1;
                        atomicSub(S.n_unfinished, 1);
                    }
                }
            } else {
                nxt = R.pad;
            }
            S.cur_tok[b] = nxt;
            s_dom = dominate ? 1 : 0;
        }
    }
    if (logits_tap) {           // parity tap: the post-rules scores of this step
        __syncthreads();
        const bool dom = s_dom != 0;
        float* tap = logits_tap + (int64_t)b * V;
        for (int i = threadIdx.x; i < V; i += SEL_THREADS) {
            const bool sup = (R.suppress_mask[i] != 0) || (first && R.begin_suppress_mask[i] != 0);
            float v = masked_score(row[i], sup, i, R, first, ts_mode, last_ts, pen_ts, ts_forbid_end);
            if (dom && i < split) v = -INFINITY;
            tap[i] = v;
        }
    }
}

void select_tokens(const float* logits, int64_t ld_logits, int V, int B, const int32_t* d_step, const RulesDev& rules, const DecodeState& st,
                   int32_t* out_tokens, int32_t* out_lengths, const int32_t* forced, float* logits_tap, cudaStream_t stream) {
    launch_k(select_tokens_kernel, dim3(B), dim3(SEL_THREADS), 0, stream, logits, ld_logits, V, d_step, rules, st, out_tokens, out_lengths, forced,
             logits_tap);
}

// Language detection (HF WhisperGenerationMixin.detect_language, generation_whisper.py:1610-1673): the logits of the step fed SOT,
// every id outside lang_ids set to -inf, argmax.  One warp per row over the <= MAX_LANG_IDS candidates.
constexpr int PICK_WARPS = 4;
__global__ void __launch_bounds__(PICK_WARPS * 32)
pick_language_kernel(const float* __restrict__ logits, int64_t ld_logits, int B, const int32_t* __restrict__ lang_ids, int n_lang,
                     DecodeState S, int32_t* __restrict__ out_lang) {
    pdl_trigger();
    pdl_wait();
    const int b = blockIdx.x * PICK_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= B) return;
    int32_t* slot = S.prompt + (int64_t)b * PROMPT_MAX + 1;
    int tok = *slot;
    if (tok == PROMPT_DETECT) {
        const float* row = logits + (int64_t)b * ld_logits;
        Best best = {-INFINITY, 0x7fffffff};
        for (int j = lane; j < n_lang; j += 32) {
            const int id = lang_ids[j];
            best = better(best, Best{row[id], id});
        }
        best = warp_best(best);
        // all candidates -inf: the masked row is -inf everywhere and torch.argmax returns index 0
        tok = best.v == -INFINITY ? 0 : best.i;
    }
    if (lane == 0) {
        *slot = tok;
        S.cur_tok[b] = tok;
        if (out_lang) out_lang[b] = tok;
    }
}

void pick_language(const float* logits, int64_t ld_logits, int B, const int32_t* lang_ids, int n_lang, const DecodeState& st,
                   int32_t* out_lang, cudaStream_t stream) {
    launch_k(pick_language_kernel, dim3(ceil_div(B, PICK_WARPS)), dim3(PICK_WARPS * 32), 0, stream, logits, ld_logits, B, lang_ids, n_lang,
             st, out_lang);
}

__global__ void decode_state_init_kernel(DecodeState S, int B, int first_tok) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) {
        S.cur_tok[b] = first_tok;
        S.finished[b] = 0;
        S.n_gen[b] = 0;
        S.last_tok[b] = -1;
        S.prev_tok[b] = -1;
        S.last_ts[b] = -1;
        S.active[b] = b;
    }
    if (b == 0) { *S.n_unfinished = B; *S.n_active = B; }
}
void decode_state_init(const DecodeState& st, int B, int first_tok, cudaStream_t stream) {
    decode_state_init_kernel<<<ceil_div(B, 128), 128, 0, stream>>>(st, B, first_tok);
}

__global__ void set_cur_tok_kernel(int32_t* cur, int B, int tok) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) cur[b] = tok;
}
void set_cur_tok(const DecodeState& st, int B, int tok, cudaStream_t stream) {
    set_cur_tok_kernel<<<ceil_div(B, 128), 128, 0, stream>>>(st.cur_tok, B, tok);
}

}  // namespace tw
