// Launcher declarations shared by the model orchestration (model.cu).
#pragma once
#include "common.cuh"

namespace tw {

// ---- log-mel (logmel.cu)
int logmel_init(tw_ctx* ctx);
void logmel_destroy(tw_ctx* ctx);
// finalize = false: stop after the first pass — `out` holds log10(max(mel, 1e-10)) and *clip_max_out the device array of
// per-clip maxima; the caller applies max(x, clipmax - 8) and (x + 4) / 4 itself (the conv-stem im2col of the fused path)
int logmel_run(tw_ctx* ctx, const void* pcm, int pcm_dtype, int64_t pcm_stride, const int32_t* n_valid, int B, int n_mel,
               float* out, cudaStream_t st, bool finalize = true, const float** clip_max_out = nullptr);

// ---- GEMM  C[M,N] = epilogue(A[M,K] . W[N,K]^T + bias)   (torch Linear layout)
enum Epi {
    EPI_STORE = 0,     // C (T)   = acc + bias
    EPI_GELU = 1,      // C (T)   = gelu(acc + bias)
    EPI_RESID = 2,     // C (f32) += acc + bias                      (residual stream)
    EPI_GELU_POS = 3,  // C (f32) = gelu(acc + bias) + pos[row % pos_period]   (conv2 + sinusoids)
    EPI_F32 = 4,       // C (f32) = acc + bias                      (logits)
};

struct GemmEpi {
    int mode = EPI_STORE;
    const float* bias = nullptr;  // [N] or null
    void* C = nullptr;
    int64_t ldc = 0;
    const float* pos = nullptr;   // [pos_period, N] f32 (EPI_GELU_POS)
    int pos_period = 1;
    // column split of the store epilogues (skinny kernel only): columns >= n_split go to C2[m*ldc2 + n - n_split]
    // (the fused QKV projection writes K|V straight into the self-attention cache row of this position)
    int n_split = 0x7fffffff;
    void* C2 = nullptr;
    int64_t ldc2 = 0;
    const int32_t* d_row2 = nullptr;   // device int: extra row offset (*d_row2 * row2_stride elements) into C2 — the cache position
    int64_t row2_stride = 0;
    // paged self-attention cache: when page_table is given, output row m at position pos = *d_row2 lands in pool row
    // kv_page_row(page_table, pt_stride, m, pos) of C2 (row pitch row2_stride) instead of m*ldc2 + pos*row2_stride
    const int32_t* page_table = nullptr;
    int pt_stride = 0;
    // grouped GEMM (skinny kernel only): the output columns form groups of group_n, and group g multiplies its own K-wide slice of
    // A — columns [g*K, (g+1)*K) of an A matrix that is n_groups*K wide — against rows [g*group_n, (g+1)*group_n) of W [N, K].
    // Used by the absorbed cross-attention: q~_h = Wk_h^T q_h (group = head, K = 64) and o_h = Wv_h c_h (group = head, K = d).
    int group_n = 0;
};

// CUDA-core FMA GEMM, fp32 accumulate in a fixed order; the fp32 check-mode path (T = float)
// and the bring-up / cross-check path for T = bf16.
template <typename T>
void gemm_simt(const T* A, int64_t lda, const T* W, int64_t ldw, int M, int N, int K, const GemmEpi& epi, cudaStream_t st);

// tcgen05 / TMEM / TMA GEMM (gemm_tc.cu), bf16 x bf16 -> fp32.  Returns TW_E_UNSUPPORTED when the
// shape cannot be tiled (caller must not fall back silently: model.cu reports the error).
int gemm_tc_init(tw_ctx* ctx);
int gemm_tc(tw_ctx* ctx, const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* W, int64_t ldw, int M, int N, int K,
            const GemmEpi& epi, cudaStream_t st);

// tcgen05 GEMM specialised for M <= 64 (gemm_tc_skinny.cu): 4 K blocks per TMA box through 3-D tensor maps
int gemm_tc_skinny_init(tw_ctx* ctx);
bool gemm_tc_skinny_supported(int M, int N, int K, const GemmEpi& epi);
int gemm_tc_skinny(tw_ctx* ctx, const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* W, int64_t ldw, int M, int N, int K,
                   const GemmEpi& epi, cudaStream_t st);

// ---- paged self-attention K|V cache: TW_KV_PAGE positions per page; page_table[clip * pt_stride + pos / TW_KV_PAGE] is the
// physical page of a clip's logical page inside the layer's pool [n_pages][TW_KV_PAGE][2d]
constexpr int TW_KV_PAGE = 16;
__host__ __device__ __forceinline__ int64_t kv_page_row(const int32_t* page_table, int pt_stride, int clip, int pos) {
    return (int64_t)page_table[(int64_t)clip * pt_stride + pos / TW_KV_PAGE] * TW_KV_PAGE + pos % TW_KV_PAGE;
}

// ---- elementwise / normalisation (elementwise.cu)
template <typename T>
void layernorm(const float* x, const float* gamma, const float* beta, T* out, int M, int d, cudaStream_t st);
// mel f32 [B,n_mel,3000] -> A1 T [B*3000, 3*n_mel], column = tap*n_mel + channel (pad 1); clip_max (optional, [B]): mel is
// the first-pass output of the log-mel kernel and the per-clip floor + scaling are applied here
template <typename T>
void im2col_conv1(const float* mel, T* out, int B, int n_mel, cudaStream_t st, const float* clip_max = nullptr);
// h0 T [B*3000, d] -> A2 T [B*1500, 3*d], column = tap*d + channel (stride 2, pad 1)
template <typename T>
void im2col_conv2(const T* h0, T* out, int B, int d, cudaStream_t st);
struct DecodeState;
// Decode-step state lives on the device so that one captured CUDA graph can be replayed for every token:
//   d_step[0] = pos (position of the token being fed), [1] = P (prompt length), [2] = stride of out_tokens,
//   [3] = number of steps whose post-rules logits are tapped.  The forced prompt tokens are per row (DecodeState::prompt).
constexpr int STEP_POS = 0, STEP_P = 1, STEP_STRIDE = 2, STEP_TAP = 3, STEP_INTS = 8;
// row b's forced prompt occupies prompt[b * PROMPT_MAX .. b * PROMPT_MAX + P); PROMPT_DETECT at index 1 = detect the language
constexpr int PROMPT_MAX = 24, PROMPT_DETECT = -1, MAX_LANG_IDS = 128;
// x[b] = E[tok[b]] + P[pos]   (f32 residual stream)
template <typename T>
void embed_tokens(const int32_t* tok, const T* E, const T* P, const int32_t* d_step, float* x, int B, int d, cudaStream_t st);
// full token sequences: x[b*T + t] = E[tok[b*T + t]] + P[t]
template <typename T>
void embed_tokens_seq(const int32_t* tok, const T* E, const T* P, float* x, int B, int Tn, int d, int vocab, cudaStream_t st);
// cache[b][pos][0:2d] = qkv[b][d:3d]   (with a page table: pool row kv_page_row(table, pt_stride, b, pos))
template <typename T>
void kv_append(const T* qkv, T* cache, const int32_t* d_step, int B, int d, int max_len, cudaStream_t st,
               const int32_t* page_table = nullptr, int pt_stride = 0);
// position += 1 and rebuild the active-clip list from the finished flags
void advance_step(int32_t* d_step, const DecodeState& S, int B, cudaStream_t st);
void copy_f32(const float* src, float* dst, int64_t n, cudaStream_t st);

// ---- attention (attention.cu)
// encoder self-attention on qkv T [B*S, 3d] (q pre-scaled), S keys per clip, out T [B*S, d]
template <typename T>
void encoder_attention_simt(const T* qkv, T* out, int B, int S, int H, cudaStream_t st);
// general CUDA-core attention: Sq queries per clip (q rows, pitch q_ld) x Sk keys/values per clip (k / v rows, pitch kv_ld),
// optional causal mask; out T [B*Sq, d].  Used by the full-sequence decoder pass (teacher logits) for the causal
// self-attention and the cross-attention over the K|V store.
template <typename T>
void attention_simt(const T* q, int64_t q_ld, const T* k, const T* v, int64_t kv_ld, T* out, int B, int Sq, int Sk, int H, bool causal,
                    cudaStream_t st);
// tcgen05 flash attention (attention_tc.cu), bf16 only
int encoder_attention_tc(tw_ctx* ctx, const __nv_bfloat16* qkv, __nv_bfloat16* out, int B, int S, int H, cudaStream_t st);
// the same kernel on separate query and key/value matrices, optionally causal (full-sequence decoder pass)
int attention_tc(tw_ctx* ctx, const __nv_bfloat16* q, int64_t q_ld, int q_col0, const __nv_bfloat16* kv, int64_t kv_ld, int k_col0,
                 int v_col0, __nv_bfloat16* out, int B, int Sq, int Sk, int H, bool causal, cudaStream_t st);
// decode attention (1 query per clip) over kv rows [Tk][2d] (K|V), clip stride kv_clip_stride elements.
// q T [B, q_stride]; partial workspace f32 [decode_attention_partial_floats]; out T [B, d].
template <typename T>
// d_tk (nullable): device int, the number of rows is *d_tk + 1 (self-attention cache at position pos) instead of Tk
void decode_attention(const T* q, int64_t q_stride, const T* kv, int64_t kv_clip_stride, int Tk, const int32_t* d_tk, int B, int H,
                      float* partial, T* out, cudaStream_t st, cudaEvent_t ev0 = nullptr, cudaEvent_t ev1 = nullptr,
                      const int32_t* active = nullptr, const int32_t* n_active = nullptr);
size_t decode_attention_partial_floats(int B, int H);
// the K|V stream kernel launches one CTA per SM: n = SMs of the partition its stream runs in (0 = the whole device); returns the
// previous count
int decode_attention_set_sms(int n);
// single-launch self-attention over the short decoder cache (Tk = *d_tk + 1 when d_tk is given).  Two kernels with the same row
// order and arithmetic: registers (4 rows in flight per warp) and a cp.async shared-memory ring (8 rows); SA_VARIANT_DEFAULT takes
// the ring for bf16 and the register kernel for fp32 (TWB200_SA_RING=0 / 1 overrides that default for the process).
enum { SA_VARIANT_DEFAULT = 0, SA_VARIANT_REGISTER = 1, SA_VARIANT_RING = 2 };
template <typename T>
void self_attention_decode(const T* q, int64_t q_stride, const T* kv, int64_t kv_clip_stride, int Tk, const int32_t* d_tk, int B, int H,
                           T* out, cudaStream_t st, const int32_t* page_table = nullptr, int pt_stride = 0,
                           const int32_t* finished = nullptr, int variant = SA_VARIANT_DEFAULT);

// ---- absorbed cross-attention (absorb.cu), bf16 only: scores and values straight from the encoder output through per-head
// q~ = Wk_h^T q_h; returns c_h = softmax(q~_h . E^T) E per clip and head.  qt [B*H + ABSORB_QT_PAD rows, d] (row clip*H + h),
// enc [B*Tk, d], partial f32 [absorbed_attention_partial_floats], ctx_out [B, H*d]; rev walks the key tiles backwards.
constexpr int ABSORB_QT_PAD = 24;
int absorbed_attention_init(tw_ctx* ctx);
bool absorbed_attention_supported(int H, int d);
size_t absorbed_attention_partial_floats(int B, int H, int d);
int absorbed_attention(tw_ctx* ctx, const __nv_bfloat16* qt, const __nv_bfloat16* enc, int Tk, int B, int H, int d, float* partial,
                       __nv_bfloat16* ctx_out, cudaStream_t st, const int32_t* active = nullptr, const int32_t* n_active = nullptr,
                       int rev = 0, cudaEvent_t ev0 = nullptr, cudaEvent_t ev1 = nullptr, long long* trace = nullptr);

// ---- token selection (select.cu)
struct RulesDev {
    const uint8_t* suppress_mask;        // [V] 1 = always suppressed
    const uint8_t* begin_suppress_mask;  // [V] 1 = suppressed at the first generated position
    int eos, pad, ts_begin, no_timestamps, max_initial_ts;
};
struct DecodeState {
    int32_t* cur_tok;     // [B] token fed to the next step
    int32_t* finished;    // [B]
    int32_t* n_gen;       // [B] tokens fed back so far (history length)
    int32_t* last_tok;    // [B] history[-1]
    int32_t* prev_tok;    // [B] history[-2]
    int32_t* last_ts;     // [B] most recent timestamp token in the history (or -1)
    int32_t* n_unfinished;  // [1]
    // clips that have not emitted EOS, compacted in clip order, and their count: rebuilt by advance_step at the end of every
    // step, consumed by the cross-attention K|V stream (finished clips are not streamed) — see attention.cu
    int32_t* active;      // [B]
    int32_t* n_active;    // [1]
    // optional per-row budget of generated tokens (test / bench hook, tw_debug_set_row_budgets): row b finishes after
    // row_budget[b] tokens exactly as if it had emitted EOS there; null = off
    const int32_t* row_budget;
    int32_t* prompt;      // [max_batch][PROMPT_MAX] forced prompt of every row (slot 1 is rewritten by the language pick)
};
// one CTA per row: rules -> argmax -> finished/pad bookkeeping -> next input token
// (inside the forced prompt it only feeds the next prompt token)
void select_tokens(const float* logits, int64_t ld_logits, int V, int B, const int32_t* d_step, const RulesDev& rules, const DecodeState& st,
                   int32_t* out_tokens, int32_t* out_lengths, const int32_t* forced, float* logits_tap, cudaStream_t stream);
// the language pick of step 0 (in place of select_tokens there): row b whose prompt slot 1 is PROMPT_DETECT takes the argmax of its
// logits over lang_ids (first id wins ties); every row then feeds its slot 1, and out_lang[b] (nullable) records it
void pick_language(const float* logits, int64_t ld_logits, int B, const int32_t* lang_ids, int n_lang, const DecodeState& st,
                   int32_t* out_lang, cudaStream_t stream);
void decode_state_init(const DecodeState& st, int B, int first_tok, cudaStream_t stream);
void set_cur_tok(const DecodeState& st, int B, int tok, cudaStream_t stream);

}  // namespace tw
