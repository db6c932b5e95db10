/* twb200.h — C ABI of libtwb200.so, the B200-native (sm_100a) Whisper teacher-inference path.
 *
 * Drop-in boundary for the hot path of forbes110/taiwan-whisper.  The reference reaches this
 * arithmetic through two Python calls into HuggingFace transformers:
 *   feature_extractor(raw_speech, sampling_rate=16000)
 *       ref: training/run_pseudo_labelling.py:739, prefiltering/validator_inference.py:57-60
 *   model.generate(input_features, max_length=, num_beams=1, return_timestamps=, language=, task=)
 *       ref: training/run_pseudo_labelling.py:864-876,917-918, prefiltering/validator_inference.py:41-47,78
 * Each entry point below names the reference interface it replaces.  The Python host
 * (taiwan-whisper_b200/host.py, ctypes) mirrors those two call signatures on top of this ABI;
 * INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions: plain C types; every call returns 0 (TW_OK) or a negative TW_E_* code and the
 * message is read with tw_last_error(ctx); no C++ exception crosses the ABI.  Calls are
 * stream-ordered and asynchronous unless they take host output buffers.  A ctx is bound to one
 * device and is NOT thread-safe (one ctx per device per process, as `accelerate launch` gives
 * one process per GPU: ref training/run-pseudo-labelling.sh:19).  Buffers passed in are owned by
 * the caller; workspace, KV cache and CUDA graphs are owned by the ctx / model.
 * There is no CPU fallback: without a CUDA device every call fails with TW_E_CUDA.
 */
#ifndef TWB200_H
#define TWB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define TW_API __attribute__((visibility("default")))
#else
#define TW_API
#endif

#define TWB200_ABI_VERSION 1

enum {
    TW_OK = 0,
    TW_E_INVALID = -1,     /* bad argument (maps to ValueError in the host) */
    TW_E_CUDA = -2,        /* CUDA runtime / driver failure */
    TW_E_NOMEM = -3,
    TW_E_UNSUPPORTED = -4, /* e.g. num_beams != 1 (maps to NotImplementedError) */
    TW_E_SHAPE = -5,       /* feature length != 3000 etc. (HF raises ValueError) */
    TW_E_STATE = -6
};

enum { TW_F32 = 0, TW_BF16 = 1, TW_I16 = 2, TW_I32 = 3 };

#define TW_N_SAMPLES 480000 /* 30 s @ 16 kHz */
#define TW_N_FRAMES 3000
#define TW_N_CTX 1500

typedef struct tw_ctx tw_ctx;
typedef struct tw_model tw_model;

TW_API int tw_abi_version(void);
TW_API int tw_ctx_create(int device, tw_ctx** out);
TW_API void tw_ctx_destroy(tw_ctx* ctx);
TW_API const char* tw_last_error(const tw_ctx* ctx);
/* number of kernels this ctx has launched so far (evidence for bench.py's gpu_launches) */
TW_API uint64_t tw_launch_count(const tw_ctx* ctx);

/* ---- log-mel front end ------------------------------------------------------------------
 * Replaces WhisperFeatureExtractor.__call__ (transformers/models/whisper/
 * feature_extraction_whisper.py:135-164; in-reference twin training/flax/distil_whisper/
 * pipeline.py:40-58), called at ref training/run_pseudo_labelling.py:739 and
 * prefiltering/validator_inference.py:57-60, including the pad/trim to 480000 samples of
 * ref prefiltering/validator_inference.py:131-137.
 *   pcm        device, row b starts at pcm + b * pcm_stride samples; int16 (dequantised x/32768) or float32
 *   n_valid    device int32 [B] or NULL: row b has n_valid[b] readable samples (NULL: pcm_stride); samples beyond
 *              that read as 0 and anything beyond 480000 is truncated.  Rows may overlap (pcm_stride < n_valid):
 *              windows of a long recording are taken without copying (taiwan-whisper_b200/longform.py)
 *   out        device float32 [B, n_mel, 3000]
 * n_mel must be 80 or 128. */
TW_API int tw_logmel(tw_ctx* ctx, const void* pcm, int pcm_dtype, int64_t pcm_stride, const int32_t* n_valid, int B,
              int n_mel, float* out, void* stream);

/* ---- model -------------------------------------------------------------------------------
 * Replaces WhisperForConditionalGeneration (encoder: modeling_whisper.py:593-647, decoder
 * :691-798, tied LM head :1081) as loaded at ref training/run_pseudo_labelling.py:566-577 and
 * prefiltering/validator_inference.py:30. */
typedef struct {
    int32_t d_model, ffn, heads, enc_layers, dec_layers, n_mel, vocab, max_target; /* max_target: 448 */
    int32_t dtype;    /* TW_BF16: bf16 storage, fp32 accumulate (tcgen05); TW_F32: fp32 check mode (CUDA-core FMA) */
    int32_t max_batch;
} tw_model_desc;

/* One named tensor.  Names are the HF state_dict keys ("model.encoder.conv1.weight", ...).
 * Pointers are DEVICE pointers borrowed only during tw_model_load: the model keeps its own
 * repacked copies, so the caller may free them afterwards.  dtype: TW_F32 or TW_BF16. */
typedef struct {
    const char* name;
    const void* ptr;
    int32_t dtype;
    int64_t numel;
} tw_weight;

TW_API int tw_model_load(tw_ctx* ctx, const tw_model_desc* desc, const tw_weight* table, size_t n, tw_model** out);
TW_API void tw_model_free(tw_model* m);
/* bytes of device memory the model holds for weights + workspace at max_batch */
TW_API size_t tw_model_bytes(const tw_model* m);
/* the descriptor the model was loaded with (what a caller that only holds the handle needs to size its buffers:
 * torch.ops.twb200.* take the tw_model* as an int64, see taiwan-whisper_b200/host.py) */
TW_API int tw_model_get_desc(const tw_model* m, tw_model_desc* out);
/* Device bytes tw_model_load would allocate for this descriptor (repacked weights, workspace, cross-attention K|V store,
 * paged self-attention pools) — host arithmetic only, usable for sizing max_batch against the 180 GB of a B200 before loading. */
TW_API size_t tw_workspace_bytes(const tw_model_desc* desc);

/* WhisperEncoder.forward on B windows: mel float32 [B, n_mel, 3000] (device) ->
 * enc_out [B, 1500, d_model] in the model dtype (device).  tap_layer >= 0 additionally copies the
 * fp32 residual stream after `tap_layer` layers (0 = after the conv stem + positions) to tap_out
 * [B,1500,d] float32 (parity tests); pass -1 / NULL otherwise. */
TW_API int tw_encode(tw_model* m, const float* mel, int B, void* enc_out, int tap_layer, float* tap_out, void* stream);

/* Logits rules of WhisperGenerationMixin._retrieve_logit_processors (generation_whisper.py:1774-1812;
 * processors logits_process.py:1812-2044).  Host arrays, copied during the call. */
typedef struct {
    const int32_t* suppress;       /* SuppressTokensLogitsProcessor ids */
    int32_t n_suppress;
    const int32_t* begin_suppress; /* SuppressTokensAtBeginLogitsProcessor ids (first generated position only) */
    int32_t n_begin_suppress;
    int32_t eos, pad;
    int32_t timestamp_begin;       /* >= 0 enables WhisperTimeStampLogitsProcessor; -1 = return_timestamps=False */
    int32_t no_timestamps;         /* <|notimestamps|> id */
    int32_t max_initial_timestamp_index; /* < 0: unset */
} tw_rules;

/* KV-cached greedy decoding of GenerationMixin._sample (generation/utils.py:2658-2805) for one
 * 30 s window per row.
 *   enc_out     device [B,1500,d] model dtype (from tw_encode)
 *   prompt      host int32 [P]: forced tokens <|sot|><|zh|><|transcribe|>[<|notimestamps|>]
 *               (_retrieve_init_tokens, generation_whisper.py:1455-1608), same for every row
 *   max_length  total length incl. prompt (HF max_length); P < max_length <= max_target
 *   out_tokens  device int32 [B, max_length - P]: generated ids; after a row's EOS: pad
 *   out_lengths device int32 [B]: number of generated tokens before EOS
 *   forced      device int32 [B, max_length - P] or NULL: teacher forcing (diagnostic) — token fed
 *               back at each step instead of the argmax; out_tokens still records the argmax
 *   logits_tap  device float32 [tap_steps, B, vocab] or NULL: post-rules logits of the first steps */
TW_API int tw_decode_greedy(tw_model* m, const void* enc_out, int B, const int32_t* prompt, int P, const tw_rules* rules,
                     int max_length, int32_t* out_tokens, int32_t* out_lengths, const int32_t* forced,
                     float* logits_tap, int tap_steps, void* stream);

/* The whole path with HOST buffers: pinned (or pageable) int16 PCM in, token ids out —
 * H2D copy, log-mel, encoder, cross-K/V, greedy decode, D2H copy, stream-synchronised on return.
 * One call = the reference's feature_extractor(...) + model.generate(...) for a batch.
 *   pcm_host        int16 [B, 480000]
 *   out_tokens_host int32 [B, max_length - P], out_lengths_host int32 [B] */
TW_API int tw_transcribe_host(tw_model* m, const int16_t* pcm_host, const int32_t* n_valid_host, int B,
                       const int32_t* prompt, int P, const tw_rules* rules, int max_length,
                       int32_t* out_tokens_host, int32_t* out_lengths_host, void* stream);

/* Two-stage pipeline over SM partitions: the batch loop of the reference (ref training/run_pseudo_labelling.py:915-918,
 * `for step, (batch, file_ids) in enumerate(...): generated_ids = generate_fn(batch["input_features"], **gen_kwargs)`) handles one
 * batch at a time; here the front end + encoder + cross-K/V of batch i+1 run concurrently with the greedy decode of batch i.  The decode
 * is HBM-bound and runs as fast on ~5/6 of the SMs; the encoder is tensor-bound and needs little HBM bandwidth.  The GPU is split into
 * two CUDA green contexts (driver-level SM partitions); stage 1 runs in the small one, stage 2 in the rest.
 *   tw_pipeline_enable   n_enc_sms SMs (8 .. half the device; the driver rounds to its granularity) for stage 1; allocates the second
 *                        encoder-output / K|V-store pair.  TW_E_UNSUPPORTED when the driver has no green contexts.
 *   tw_pipeline_resize   moves the boundary between the two partitions (both stages are drained first; batches already staged in a slot
 *                        stay valid).  The balance depends on the workload: full-length rows (252 tokens) keep the decode partition busy
 *                        ~7x longer than stage 1 needs the GPU, rows that end early (real audio) shift work towards stage 1.
 *   tw_pipeline_stage_ms device time of the slot's last stage 1 (all parts of the group) and of its last decode, each measured inside its
 *                        partition while the other stage runs; -1 for a stage that has not completed.  Never blocks: the input of a
 *                        balance controller (host.py transcribe_batches(auto_sms=True)).
 *   tw_pipeline_encode   ASYNCHRONOUS stage 1 of a batch into slot 0 / 1: copy of int16 PCM [B, 480000] (host — it must stay valid until
 *                        the matching tw_pipeline_decode returns — or device), log-mel, encoder, cross-K/V.  Waits (on the device)
 *                        for the decode that last used the slot.
 *   tw_pipeline_encode_at  the same for a batch that becomes clips clip0 .. clip0 + B - 1 of the slot: several batches of the
 *                        reference's loop are staged one after the other into one slot and decoded TOGETHER by one tw_pipeline_decode
 *                        call over clip0 + B rows (merged decode).  A decode step streams the decoder weights once whatever the row
 *                        count, so two 64-clip batches decoded as 128 rows pay the weight / small-kernel chain of every token once
 *                        instead of twice; the model must have been loaded with max_batch >= the merged row count.
 *   tw_pipeline_decode   stage 2 of the batch(es) in `slot`: greedy decode of rows 0 .. B - 1, ids to HOST buffers, synchronised on
 *                        return (arguments as tw_transcribe_host).
 * Use: encode(b0, 0); for i: { encode(b[i+1], (i+1)&1); decode(i&1) -> ids of b[i] }.  Ids equal tw_transcribe_host's up to the
 * bf16 rounding of a different row split of the K|V stream. */
TW_API int tw_pipeline_enable(tw_model* m, int n_enc_sms);
TW_API int tw_pipeline_resize(tw_model* m, int n_enc_sms);
TW_API int tw_pipeline_info(const tw_model* m, int* n_enc_sms, int* n_dec_sms);
TW_API int tw_pipeline_stage_ms(tw_model* m, int slot, float* stage1_ms, float* decode_ms);
TW_API int tw_pipeline_encode(tw_model* m, const int16_t* pcm, const int32_t* n_valid_host, int B, int slot);
TW_API int tw_pipeline_encode_at(tw_model* m, const int16_t* pcm, const int32_t* n_valid_host, int B, int slot, int clip0);
TW_API int tw_pipeline_decode(tw_model* m, int slot, int B, const int32_t* prompt, int P, const tw_rules* rules, int max_length,
                              int32_t* out_tokens_host, int32_t* out_lengths_host);

/* Per-stage device time of the last tw_transcribe_host / tw_decode_greedy call in ms (CUDA events on the call's
 * stream): [0] log-mel, [1] encoder, [2] cross-K/V, [3] decode (incl. the D2H of the ids), [4] total, [5] H2D copy. */
TW_API int tw_last_stage_ms(tw_model* m, float out_ms[6]);

/* In-situ CUDA-event timing of the path's dominant kernel (the decode cross-attention K/V streaming
 * kernel, one sampled launch per decode step at the middle decoder layer).  Reads and resets the
 * accumulated samples (either pointer may be NULL), then enables/disables sampling for later calls. */
TW_API int tw_profile(tw_model* m, int enable, float* total_ms, int* launches, double* bytes_per_launch);

/* Teacher forward of the distillation step: logits of EVERY position of decoder_input_ids in one batched decoder pass.
 * Replaces teacher_model(encoder_outputs=..., labels=...) / teacher_model(**batch) followed by `.logits`
 * (ref knowledge-distillation/run_distillation.py:1543-1577; HF WhisperForConditionalGeneration.forward,
 * modeling_whisper.py:1000-1100 with the decoder of :691-798 under the causal mask).
 *   enc_out            device, model dtype, [B, 1500, d_model] (output of tw_encode)
 *   decoder_input_ids  device int32 [B, T], 1 <= T <= max_target_positions (HF shift_tokens_right is done by the caller)
 *   logits             device float32 [B*T, ld_logits], ld_logits >= vocab and a multiple of 4 (16-byte row pitch); columns
 *                      >= vocab are not written.  fp32 like HF's `.logits.float()`.
 * Uses the encoder workspace: must not overlap a tw_encode / tw_transcribe_host call on another stream. */
TW_API int tw_decoder_logits(tw_model* m, const void* enc_out, int B, const int32_t* decoder_input_ids, int T, float* logits,
                             int64_t ld_logits, void* stream);

/* Test / profiling entry point: decoder self-attention over the PAGED K|V cache.  pool: [n_pages][16][2*64*H] (a page holds
 * 16 positions, row = K(d) then V(d)); page_table: device int32 [B][pt_stride], physical page of each clip's logical page;
 * Tk rows per clip.  The model keeps one such pool per decoder layer and rewrites the table for every decode call. */
TW_API int tw_debug_self_attention_paged(tw_ctx* ctx, const void* q, int64_t q_stride, const void* pool, const int32_t* page_table,
                                         int pt_stride, int Tk, int B, int H, int dtype, void* out, void* stream);

/* Test / profiling entry point: attention of the full-sequence decoder pass.  Sq query rows per clip in q (row pitch q_ld
 * elements, head h at column q_col0 + 64 h) against Sk key / value rows per clip in kv (pitch kv_ld, K at k_col0 + 64 h, V at
 * v_col0 + 64 h); causal != 0 masks keys later than the query (needs Sq == Sk).  out [B*Sq, 64 H].  impl 1 = tcgen05 kernel
 * (bf16), 0 = CUDA-core kernel. */
TW_API int tw_debug_attention(tw_ctx* ctx, const void* q, int64_t q_ld, int q_col0, const void* kv, int64_t kv_ld, int k_col0,
                              int v_col0, void* out, int B, int Sq, int Sk, int H, int dtype, int impl, int causal, void* stream);

/* Test / profiling switch (calling thread): tw_debug_* launches carry the programmatic-dependent-launch attribute. */
TW_API void tw_debug_set_pdl(int on);
/* Test / bench hook: per-row budgets of generated tokens for the following decode calls (host array of n <= max_batch ints;
 * n = 0 switches it off).  Row b finishes after budgets[b] tokens exactly as if it had emitted EOS next: out_lengths[b] =
 * budgets[b], pad afterwards, the row leaves the active list of the cross-attention stream.  Random-init weights never
 * emit EOS, so this is how the finished-row path is exercised at the benched shapes (bench.py --ragged). */
TW_API int tw_debug_set_row_budgets(tw_model* m, const int32_t* budgets_host, int n);

/* Test / profiling entry point: one GEMM of the path, C[M,N] = epilogue(A[M,K] . W[N,K]^T + bias)
 * (torch nn.Linear layout), row-major dense operands.  dtype TW_BF16 (use_tc = 1: tcgen05 kernel,
 * 3: tcgen05 skinny kernel for M <= 64 with K % 64 == 0, 0: CUDA-core kernel) or TW_F32 (CUDA-core check-mode kernel).  epi_mode: 0 store (dtype), 1 GELU
 * (dtype), 2 C(f32) += , 3 C(f32) = GELU(.) + pos[row % pos_period], 4 C(f32) = . */
TW_API int tw_debug_gemm(tw_ctx* ctx, const void* A, const void* W, const float* bias, void* C, int M, int N, int K, int dtype,
                  int epi_mode, const float* pos, int pos_period, int use_tc, void* stream);

/* Test / profiling entry point: grouped form of the decode-step GEMM (bf16, M <= 64): the N output columns form groups of
 * group_n; group g multiplies columns [g*K, (g+1)*K) of A [M, K*N/group_n] with rows [g*group_n, (g+1)*group_n) of W [N, K].
 * The absorbed cross-attention uses it with group = head: q~_h = Wk_h^T q_h (K = 64) and o_h = Wv_h c_h + bv_h (K = d). */
TW_API int tw_debug_gemm_grouped(tw_ctx* ctx, const void* A, const void* W, const float* bias, void* C, int M, int N, int K, int group_n,
                                 void* stream);
/* Test / profiling entry point: absorbed decoder cross-attention (bf16).  qt: [B*H + 24 rows, 64*H], row clip*H + h = q~ of that
 * clip and head (the 24 trailing rows only need to be readable); enc: [B*Tk, 64*H] encoder output; out: [B, H*64*H], row clip,
 * columns [h*d, (h+1)*d) = softmax_k(q~_h . enc[clip, k]) . enc[clip]  (HF modeling_whisper.py:284-358 with K and V projected after
 * the contraction).  active / n_active (device, nullable): compacted list of the clips to process; rev != 0 walks the keys backwards. */
TW_API int tw_debug_absorbed_attention(tw_ctx* ctx, const void* qt, const void* enc, int Tk, int B, int H, void* out, const int32_t* active,
                                       const int32_t* n_active, int rev, void* stream);

/* Test / profiling entry points for the two attention kernels of the path (device buffers):
 *   decode attention: q [B, q_stride] (first H*64 elements used), K|V rows kv [B][Tk][2*H*64] with clip
 *   stride kv_clip_stride elements -> out [B, H*64]   (softmax(q.K^T).V per head, q pre-scaled)
 *   encoder attention: qkv [B*S, 3*H*64] -> out [B*S, H*64]; impl 0 = CUDA-core kernel, 1 = tcgen05 flash kernel (bf16) */
TW_API int tw_debug_decode_attention(tw_ctx* ctx, const void* q, int64_t q_stride, const void* kv, int64_t kv_clip_stride,
                                     int Tk, int B, int H, int dtype, void* out, void* stream);
/* same contract as tw_debug_decode_attention, through the single-launch short-cache self-attention kernel */
TW_API int tw_debug_self_attention(tw_ctx* ctx, const void* q, int64_t q_stride, const void* kv, int64_t kv_clip_stride, int Tk,
                                   int B, int H, int dtype, void* out, void* stream);
TW_API int tw_debug_encoder_attention(tw_ctx* ctx, const void* qkv, void* out, int B, int S, int H, int dtype, int impl,
                                      void* stream);

/* Test entry points for the kernels of one decode step in the form the step issues them: state on the device (position, finished
 * flags, active-clip list, page table) and the SM count of the partition the step runs in.  Device buffers unless noted.
 *
 * tw_debug_select_steps: the greedy loop of tw_decode_greedy (same decode state, step header, rules upload and per-row budgets) with
 *   caller-supplied logits in place of the model forward.  logits float32 [max_length - P, B, ld_logits] (16-byte aligned, ld_logits
 *   >= vocab and a multiple of 4): scores of generated step g at logits + g*B*ld_logits; columns >= vocab are never selected.
 *   prompt / rules (host), forced, logits_tap, tap_steps, out_tokens [B, max_length - P], out_lengths [B]: as tw_decode_greedy.
 *   row_budgets (host int32 [B], nullable): the budgets of tw_debug_set_row_budgets for this call only (they are off afterwards);
 *   NULL leaves the budgets set with tw_debug_set_row_budgets in effect.  n_active [max_length - P] and active
 *   [max_length - P, B] (nullable): the active-clip count and list after every generated step.
 * tw_debug_kv_append: the self-attention QKV projection C [M, 3d] = A [M, d] . W [3d, d]^T + bias of a decode step at position *d_pos,
 *   whose K|V columns land in pool row page_table[m * pt_stride + pos / 16] * 16 + pos % 16 (pool [n_pages][16][2d]).
 *   fused = 1 (bf16, M <= 256): one skinny GEMM that stores columns >= d in the pool instead of C (C[:, d:] is not written);
 *   fused = 0: the GEMM into C, then the append kernel (bf16 or fp32).  n_sms > 0 sizes the GEMM for a partition of that many SMs.
 * tw_debug_self_attention_step: decoder self-attention with Tk = *d_pos + 1 rows per clip read on the device (old rows are fetched
 *   before the programmatic-dependency wait); kv / page_table as tw_debug_self_attention(_paged) (page_table NULL: contiguous rows,
 *   clip stride kv_clip_stride).  finished (int32 [B], nullable): rows whose flag is set are not computed and their out rows are left
 *   as they were.  variant: 0 the build's default kernel, 1 registers, 2 shared-memory ring.
 * tw_debug_decode_attention_step: the cross-attention K|V stream of tw_debug_decode_attention over the compacted active-clip list
 *   (active int32 [B], n_active int32 [1], both NULL = every clip): only clips active[0 .. *n_active) are computed, other out rows
 *   are left as they were.  n_sms > 0: the stream runs as in a pipeline partition of that many SMs. */
TW_API int tw_debug_select_steps(tw_model* m, const float* logits, int64_t ld_logits, int B, const int32_t* prompt, int P,
                                 const tw_rules* rules, int max_length, const int32_t* row_budgets, const int32_t* forced, float* logits_tap,
                                 int tap_steps, int32_t* out_tokens, int32_t* out_lengths, int32_t* n_active, int32_t* active, void* stream);
TW_API int tw_debug_kv_append(tw_ctx* ctx, const void* A, const void* W, const float* bias, void* C, void* pool, const int32_t* page_table,
                              int pt_stride, const int32_t* d_pos, int M, int d, int dtype, int fused, int n_sms, void* stream);
TW_API int tw_debug_self_attention_step(tw_ctx* ctx, const void* q, int64_t q_stride, const void* kv, int64_t kv_clip_stride,
                                        const int32_t* page_table, int pt_stride, const int32_t* d_pos, const int32_t* finished, int B, int H,
                                        int dtype, int variant, void* out, void* stream);
TW_API int tw_debug_decode_attention_step(tw_ctx* ctx, const void* q, int64_t q_stride, const void* kv, int64_t kv_clip_stride, int Tk,
                                          int B, int H, int dtype, const int32_t* active, const int32_t* n_active, int n_sms, void* out,
                                          void* stream);

/* Test entry points for the encoder stage (stage 1: encoder + cross-attention K|V store) in the form the model issues it.
 * tw_debug_layernorm: out [M, d] (dtype TW_F32 / TW_BF16) = LayerNorm of the float32 rows x [M, d] with float32 gamma / beta [d],
 *   through the launcher the model uses, so M picks the kernel as in the model (one CTA per row for M <= 512, one warp per row
 *   above).  TW_E_INVALID for M < 0, d > 1280, d % 4 != 0, another dtype or a null buffer; M = 0 launches nothing.
 * tw_debug_cross_kv: the cross-attention K|V projection of every decoder layer for clips clip0 .. clip0 + B - 1 into the model's
 *   own K|V store (the one tw_decode_greedy reads; with the pipeline on, slot 0's), from enc_out [B, 1500, d_model] in the model
 *   dtype.  Rows of other clips are not written.
 * tw_debug_read_stage1: copies (cudaMemcpyAsync on `stream`) the rows of clips clip0 .. clip0 + B - 1: the encoder output of pipeline
 *   slot 0 / 1 into enc_out [B, 1500, d_model] (nullable; must be NULL for slot -1) and decoder layer `layer`'s K|V rows into kv_out
 *   [B, 1500, 2 d_model] (nullable), from the slot's store or, for slot -1, from the model's own store.  For slots 0 / 1 the copies
 *   first wait for the slot's last tw_pipeline_encode(_at). */
TW_API int tw_debug_layernorm(tw_ctx* ctx, const float* x, const float* gamma, const float* beta, void* out, int M, int d, int dtype,
                              void* stream);
TW_API int tw_debug_cross_kv(tw_model* m, const void* enc_out, int B, int clip0, void* stream);
TW_API int tw_debug_read_stage1(tw_model* m, int slot, int clip0, int B, void* enc_out, int layer, void* kv_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TWB200_H */
