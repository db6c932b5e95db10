// Host orchestration of the Whisper teacher-inference path and the C ABI (include/twb200.h).
// One tw_model = repacked weights + workspace + KV stores for up to max_batch 30 s windows.
//
// Call order per batch (what the reference does with feature_extractor(...) + model.generate(...),
// ref: training/run_pseudo_labelling.py:739,917-918; prefiltering/validator_inference.py:57-60,78):
//   log-mel (K1) -> conv stem as im2col + GEMM with fused GELU(+positions) -> L_enc x {LN, QKV GEMM,
//   attention, out-proj GEMM (+residual), LN, fc1 GEMM (+GELU), fc2 GEMM (+residual)} -> LN
//   -> cross-attention K/V for every decoder layer (once per window) -> greedy loop on the device.
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <tuple>
#include <vector>

#include "kernels.cuh"

using namespace tw;

namespace tw {
thread_local bool g_pdl = false;
}

namespace {

// ---- weight repack kernels -----------------------------------------------------------------
template <typename Dst>
__global__ void repack_copy_kernel(const void* __restrict__ src, int src_dtype, Dst* __restrict__ dst, int64_t n, float scale) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float v = (src_dtype == TW_F32) ? reinterpret_cast<const float*>(src)[i]
                                              : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(src)[i]);
        dst[i] = from_f32<Dst>(v * scale);
    }
}
// conv weight [d_out, C, 3] -> [d_out, 3*C] with column = tap*C + c
template <typename Dst>
__global__ void repack_conv_kernel(const void* __restrict__ src, int src_dtype, Dst* __restrict__ dst, int d_out, int C) {
    const int64_t n = (int64_t)d_out * C * 3;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int tap = (int)(i % 3);
        const int c = (int)((i / 3) % C);
        const int64_t o = i / (3 * (int64_t)C);
        const float v = (src_dtype == TW_F32) ? reinterpret_cast<const float*>(src)[i]
                                              : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(src)[i]);
        dst[o * 3 * C + (int64_t)tap * C + c] = from_f32<Dst>(v);
    }
}
__global__ void fill_f32_kernel(float* p, int64_t n, float v) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}
__global__ void mask_from_ids_kernel(const int32_t* ids, int n, uint8_t* mask, int V) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && ids[i] >= 0 && ids[i] < V) mask[ids[i]] = 1;
}

inline int nblocks(int64_t n) {
    int64_t b = (n + 255) / 256;
    return (int)(b > 148 * 16 ? 148 * 16 : (b < 1 ? 1 : b));
}

struct AttnW {
    void* qkv_w = nullptr;   // [3d, d] (q rows pre-scaled by head_dim^-0.5; exact, 0.125)
    float* qkv_b = nullptr;  // [3d] (k part zero: k_proj has no bias)
    void* q_w = nullptr;     // cross-attn: [d, d] scaled
    float* q_b = nullptr;
    void* kv_w = nullptr;    // cross-attn: [2d, d] = [Wk; Wv]
    float* kv_b = nullptr;   // [2d] = [0; bv]
    void* kt_w = nullptr;    // cross-attn, absorbed path (bf16): [H*d, 64], row h*d + c = Wk[h*64 .. h*64+63, c] (per-head Wk^T)
    void* o_w = nullptr;     // [d, d]
    float* o_b = nullptr;
};
struct LayerW {
    float *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr, *ln3_g = nullptr, *ln3_b = nullptr;
    AttnW self, cross;
    void* fc1_w = nullptr;
    float* fc1_b = nullptr;
    void* fc2_w = nullptr;
    float* fc2_b = nullptr;
};

}  // namespace

struct GraphKey {
    int B, eos, pad, ts_begin, no_ts, max_init, budget;
    const void* enc;       // the absorbed cross-attention reads the encoder output directly: the graph bakes the pointer in
    const void* xkv;       // K|V store of the call (the pipeline alternates between two)
    int sms;               // SMs the step was sized for (and, under the pipeline, the partition the graph was captured in)
    bool operator<(const GraphKey& o) const {
        return std::tie(B, eos, pad, ts_begin, no_ts, max_init, budget, enc, xkv, sms) <
               std::tie(o.B, o.eos, o.pad, o.ts_begin, o.no_ts, o.max_init, o.budget, o.enc, o.xkv, o.sms);
    }
};
struct GraphEntry {
    cudaGraphExec_t exec;
    uint64_t kernels;
};

struct tw_model {
    tw_ctx* ctx = nullptr;
    tw_model_desc desc{};
    int esz = 2;                 // bytes per element of the model dtype
    bool use_tc = false;         // tcgen05 GEMMs (bf16 only)
    bool use_tc_attn = false;    // tcgen05 encoder attention (bf16 only)
    bool use_tc_skinny = true;   // tcgen05 skinny GEMM with multi-K-block TMA boxes for M <= 64
    std::vector<void*> allocs;
    size_t bytes = 0;
    // weights
    void *conv1_w = nullptr, *conv2_w = nullptr;
    float *conv1_b = nullptr, *conv2_b = nullptr, *enc_pos = nullptr, *enc_lnf_g = nullptr, *enc_lnf_b = nullptr;
    std::vector<LayerW> enc, dec;
    void *embed = nullptr, *dec_pos = nullptr;
    float *dec_lnf_g = nullptr, *dec_lnf_b = nullptr;
    // workspace
    int16_t* ws_pcm = nullptr;
    int32_t* ws_nvalid = nullptr;
    float* ws_mel = nullptr;
    void *ws_a1 = nullptr, *ws_h0 = nullptr, *ws_a2qkv = nullptr, *ws_xn = nullptr, *ws_att = nullptr, *ws_hmid = nullptr,
         *ws_enc = nullptr;
    float* ws_x = nullptr;
    void* xkv = nullptr;       // [L_dec][maxB*1500][2d]
    // paged self-attention K|V cache: per decoder layer a pool [max_batch * kv_pages][TW_KV_PAGE][2d]; one page table
    // [max_batch][kv_pages] (physical page of each clip's logical page) shared by all layers, rewritten per decode call
    void* self_kv = nullptr;
    int kv_pages = 0;                  // logical pages per clip = ceil(max_target / TW_KV_PAGE)
    int32_t* d_page_table = nullptr;
    int32_t* h_page_table = nullptr;   // pinned staging
    float *dx = nullptr, *dlogits = nullptr, *dpartial = nullptr;
    int64_t ld_logits = 0;     // row pitch of dlogits: vocab rounded up to 4 floats (16-byte rows for the TMA-store epilogue)
    void *dxn = nullptr, *dqkv = nullptr, *datt = nullptr, *dq = nullptr, *dhmid = nullptr;
    // absorbed cross-attention (bf16 product path, decode batches <= 64): q~ [maxB*H + pad, d], c [maxB, H*d], partial records
    bool absorb_ok = false;      // the model has the weights / buffers of the absorbed path
    bool absorb_now = false;     // the decode call in progress uses it
    const void* cur_enc = nullptr;   // encoder output of the decode call in progress
    void *dqt = nullptr, *dctx = nullptr;
    float* dab_partial = nullptr;
    int32_t* dstate = nullptr;  // decode state: 8 arrays of maxB ints + counters (DecodeState)
    int32_t* d_row_budget = nullptr;   // [maxB] per-row token budgets (tw_debug_set_row_budgets)
    bool row_budget_on = false;
    uint8_t *d_suppress = nullptr, *d_begin_suppress = nullptr;
    int32_t* d_ids_tmp = nullptr;
    int32_t *d_out_tok = nullptr, *d_out_len = nullptr;
    int32_t* h_flag = nullptr;   // pinned
    int32_t* h_step = nullptr;   // pinned staging of the step header
    int32_t* d_step = nullptr;   // device step state (kernels.cuh STEP_*)
    // per-row forced prompts [max_batch][PROMPT_MAX] and the language ids detection chooses among, rewritten per decode call
    // from pinned staging (h_rows: the prompt table, then MAX_LANG_IDS ids); d_out_lang: languages of the host-output calls
    int32_t* d_row_prompt = nullptr;
    int32_t* d_lang_ids = nullptr;
    int32_t* h_rows = nullptr;
    int32_t* d_out_lang = nullptr;
    int n_lang_now = 0;          // language ids of the decode call in progress
    bool pick_now = false;       // its step 0 runs the language pick in place of the selection
    bool use_graph = true;       // replay one captured CUDA graph per decode step
    bool use_pdl = true;         // programmatic dependent launch inside the decode step
    cudaStream_t cap_stream = nullptr;
    // Two-stage pipeline over SM partitions (tw_pipeline_*): the front end + encoder + cross-K/V of batch i+1 run in a small green
    // context while the decode of batch i runs in the rest of the GPU.  Decode is HBM-bound and does not need every SM (its time
    // is the same on 124 as on 148); the encoder is tensor-bound and needs almost no HBM bandwidth.
    struct Pipeline {
        bool on = false;
        int n_enc = 0, n_dec = 0, n_dev = 0;
        CUgreenCtx g_enc = nullptr, g_dec = nullptr;
        cudaStream_t s_enc = nullptr, s_dec = nullptr, s_cap = nullptr;    // s_cap: graph capture inside the decode partition
        void* enc_out[2] = {nullptr, nullptr};
        void* xkv[2] = {nullptr, nullptr};
        cudaEvent_t enc_done[2] = {nullptr, nullptr}, dec_done[2] = {nullptr, nullptr};
        // per-slot stage timing (tw_pipeline_stage_ms): stage 1 of the slot's group (first part's start .. last part's end), its decode
        cudaEvent_t enc_t0[2] = {nullptr, nullptr}, enc_t1[2] = {nullptr, nullptr}, dec_t0[2] = {nullptr, nullptr}, dec_t1[2] = {nullptr, nullptr};
        bool enc_timed[2] = {false, false}, dec_timed[2] = {false, false};
        bool dec_pending[2] = {false, false};
        bool in_decode = false;
    } pipe;
    std::map<GraphKey, GraphEntry> graphs;
    double prof_bytes = 0.0;     // K|V bytes of one profiled cross-attention launch
    // debug timeline (TWB200_TRACE=<position>): CUDA events after every kernel of two middle decoder layers at that
    // position (non-graph path only), printed to stderr at the end of the decode call
    int trace_pos = -1;
    int skip_mask = 0;           // TWB200_SKIP (timing experiments only, results are garbage): kernels left out of the decode step —
                                 // 1 LayerNorms, 2 self-attention, 4 cross-attention stream, 8 QKV, 16 self out-proj, 32 cross q, 64 cross out-proj, 128 fc1, 256 fc2
    std::vector<std::pair<cudaEvent_t, std::string>> trace;
    // in-situ timing of the dominant kernel (cross-attention K/V streaming) for bench.py's roofline
    bool prof_on = false;
    std::vector<cudaEvent_t> prof_ev;   // pairs
    int prof_used = 0;
    cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // [6]: before the H2D copy, [7]: decode start (pipeline)
    bool ev_valid[8] = {false, false, false, false, false, false, false, false};
};

namespace {

int dev_alloc(tw_model* m, void** p, size_t bytes) {
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) {
        m->ctx->set_error(TW_E_NOMEM, std::string("cudaMalloc failed: ") + cudaGetErrorString(e));
        return TW_E_NOMEM;
    }
    m->allocs.push_back(*p);
    m->bytes += bytes;
    return TW_OK;
}

struct WeightTable {
    std::map<std::string, const tw_weight*> by_name;
    const tw_weight* get(tw_ctx* ctx, const std::string& name, int64_t numel) const {
        auto it = by_name.find(name);
        if (it == by_name.end()) {
            ctx->set_error(TW_E_INVALID, "tw_model_load: missing weight " + name);
            return nullptr;
        }
        if (it->second->numel != numel) {
            ctx->set_error(TW_E_SHAPE, "tw_model_load: weight " + name + " has " + std::to_string(it->second->numel) +
                                           " elements, expected " + std::to_string(numel));
            return nullptr;
        }
        if (it->second->dtype != TW_F32 && it->second->dtype != TW_BF16) {
            ctx->set_error(TW_E_INVALID, "tw_model_load: weight " + name + " must be float32 or bfloat16");
            return nullptr;
        }
        return it->second;
    }
};

// kt[h*d + c][j] = w[h*64 + j][c]: per-head transpose of a [d, d] projection (absorbed cross-attention, q~_h = Wk_h^T q_h)
template <typename T>
__global__ void head_transpose_kernel(const T* __restrict__ w, T* __restrict__ kt, int H, int d) {
    const int64_t n = (int64_t)d * d;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int j = (int)(i % 64);
        const int64_t hc = i / 64;
        const int c = (int)(hc % d), h = (int)(hc / d);
        kt[i] = w[(int64_t)(h * 64 + j) * d + c];
    }
}

template <typename T>
int put(tw_model* m, const WeightTable& wt, const std::string& name, int64_t numel, T* dst, float scale = 1.0f) {
    const tw_weight* w = wt.get(m->ctx, name, numel);
    if (!w) return m->ctx->err_code;
    repack_copy_kernel<T><<<nblocks(numel), 256>>>(w->ptr, w->dtype, dst, numel, scale);
    return TW_OK;
}

template <typename T>
int load_attn(tw_model* m, const WeightTable& wt, const std::string& pre, AttnW& a, bool cross) {
    const int d = m->desc.d_model;
    const int64_t dd = (int64_t)d * d;
    const float qs = 0.125f;    // head_dim 64 -> 64^-0.5, a power of two: folding it into Wq/bq is exact
    if (!cross) {
        TW_CHECK(dev_alloc(m, &a.qkv_w, 3 * dd * sizeof(T)));
        TW_CHECK(dev_alloc(m, (void**)&a.qkv_b, 3 * d * sizeof(float)));
        fill_f32_kernel<<<nblocks(3 * d), 256>>>(a.qkv_b, 3 * d, 0.0f);
        T* w = (T*)a.qkv_w;
        TW_CHECK(put<T>(m, wt, pre + "q_proj.weight", dd, w, qs));
        TW_CHECK(put<T>(m, wt, pre + "k_proj.weight", dd, w + dd));
        TW_CHECK(put<T>(m, wt, pre + "v_proj.weight", dd, w + 2 * dd));
        TW_CHECK(put<float>(m, wt, pre + "q_proj.bias", d, a.qkv_b, qs));
        TW_CHECK(put<float>(m, wt, pre + "v_proj.bias", d, a.qkv_b + 2 * d));
    } else {
        TW_CHECK(dev_alloc(m, &a.q_w, dd * sizeof(T)));
        TW_CHECK(dev_alloc(m, (void**)&a.q_b, d * sizeof(float)));
        TW_CHECK(dev_alloc(m, &a.kv_w, 2 * dd * sizeof(T)));
        TW_CHECK(dev_alloc(m, (void**)&a.kv_b, 2 * d * sizeof(float)));
        fill_f32_kernel<<<nblocks(2 * d), 256>>>(a.kv_b, 2 * d, 0.0f);
        TW_CHECK(put<T>(m, wt, pre + "q_proj.weight", dd, (T*)a.q_w, qs));
        TW_CHECK(put<float>(m, wt, pre + "q_proj.bias", d, a.q_b, qs));
        TW_CHECK(put<T>(m, wt, pre + "k_proj.weight", dd, (T*)a.kv_w));
        TW_CHECK(put<T>(m, wt, pre + "v_proj.weight", dd, (T*)a.kv_w + dd));
        TW_CHECK(put<float>(m, wt, pre + "v_proj.bias", d, a.kv_b + d));
        if (m->absorb_ok) {
            TW_CHECK(dev_alloc(m, &a.kt_w, dd * sizeof(T)));
            head_transpose_kernel<T><<<nblocks(dd), 256>>>((const T*)a.kv_w, (T*)a.kt_w, m->desc.heads, d);
        }
    }
    TW_CHECK(dev_alloc(m, &a.o_w, dd * sizeof(T)));
    TW_CHECK(dev_alloc(m, (void**)&a.o_b, d * sizeof(float)));
    TW_CHECK(put<T>(m, wt, pre + "out_proj.weight", dd, (T*)a.o_w));
    TW_CHECK(put<float>(m, wt, pre + "out_proj.bias", d, a.o_b));
    return TW_OK;
}

int load_ln(tw_model* m, const WeightTable& wt, const std::string& pre, float** g, float** b) {
    const int d = m->desc.d_model;
    TW_CHECK(dev_alloc(m, (void**)g, d * sizeof(float)));
    TW_CHECK(dev_alloc(m, (void**)b, d * sizeof(float)));
    TW_CHECK(put<float>(m, wt, pre + ".weight", d, *g));
    TW_CHECK(put<float>(m, wt, pre + ".bias", d, *b));
    return TW_OK;
}

template <typename T>
int load_mlp(tw_model* m, const WeightTable& wt, const std::string& pre, LayerW& L) {
    const int d = m->desc.d_model, f = m->desc.ffn;
    TW_CHECK(dev_alloc(m, &L.fc1_w, (size_t)f * d * sizeof(T)));
    TW_CHECK(dev_alloc(m, (void**)&L.fc1_b, f * sizeof(float)));
    TW_CHECK(dev_alloc(m, &L.fc2_w, (size_t)f * d * sizeof(T)));
    TW_CHECK(dev_alloc(m, (void**)&L.fc2_b, d * sizeof(float)));
    TW_CHECK(put<T>(m, wt, pre + "fc1.weight", (int64_t)f * d, (T*)L.fc1_w));
    TW_CHECK(put<float>(m, wt, pre + "fc1.bias", f, L.fc1_b));
    TW_CHECK(put<T>(m, wt, pre + "fc2.weight", (int64_t)f * d, (T*)L.fc2_w));
    TW_CHECK(put<float>(m, wt, pre + "fc2.bias", d, L.fc2_b));
    return TW_OK;
}

template <typename T>
int load_weights(tw_model* m, const WeightTable& wt) {
    const tw_model_desc& D = m->desc;
    const int d = D.d_model;
    const std::string E = "model.encoder.", Dc = "model.decoder.";
    // conv stem
    TW_CHECK(dev_alloc(m, &m->conv1_w, (size_t)d * 3 * D.n_mel * sizeof(T)));
    TW_CHECK(dev_alloc(m, &m->conv2_w, (size_t)d * 3 * d * sizeof(T)));
    TW_CHECK(dev_alloc(m, (void**)&m->conv1_b, d * sizeof(float)));
    TW_CHECK(dev_alloc(m, (void**)&m->conv2_b, d * sizeof(float)));
    TW_CHECK(dev_alloc(m, (void**)&m->enc_pos, (size_t)TW_N_CTX * d * sizeof(float)));
    {
        const tw_weight* w1 = wt.get(m->ctx, E + "conv1.weight", (int64_t)d * D.n_mel * 3);
        const tw_weight* w2 = wt.get(m->ctx, E + "conv2.weight", (int64_t)d * d * 3);
        if (!w1 || !w2) return m->ctx->err_code;
        repack_conv_kernel<T><<<nblocks((int64_t)d * D.n_mel * 3), 256>>>(w1->ptr, w1->dtype, (T*)m->conv1_w, d, D.n_mel);
        repack_conv_kernel<T><<<nblocks((int64_t)d * d * 3), 256>>>(w2->ptr, w2->dtype, (T*)m->conv2_w, d, d);
    }
    TW_CHECK(put<float>(m, wt, E + "conv1.bias", d, m->conv1_b));
    TW_CHECK(put<float>(m, wt, E + "conv2.bias", d, m->conv2_b));
    TW_CHECK(put<float>(m, wt, E + "embed_positions.weight", (int64_t)TW_N_CTX * d, m->enc_pos));
    m->enc.resize(D.enc_layers);
    for (int l = 0; l < D.enc_layers; ++l) {
        const std::string p = E + "layers." + std::to_string(l) + ".";
        LayerW& L = m->enc[l];
        TW_CHECK(load_ln(m, wt, p + "self_attn_layer_norm", &L.ln1_g, &L.ln1_b));
        TW_CHECK(load_attn<T>(m, wt, p + "self_attn.", L.self, false));
        TW_CHECK(load_ln(m, wt, p + "final_layer_norm", &L.ln3_g, &L.ln3_b));
        TW_CHECK(load_mlp<T>(m, wt, p, L));
    }
    TW_CHECK(load_ln(m, wt, E + "layer_norm", &m->enc_lnf_g, &m->enc_lnf_b));
    // decoder
    TW_CHECK(dev_alloc(m, &m->embed, (size_t)D.vocab * d * sizeof(T)));
    TW_CHECK(dev_alloc(m, &m->dec_pos, (size_t)D.max_target * d * sizeof(T)));
    TW_CHECK(put<T>(m, wt, Dc + "embed_tokens.weight", (int64_t)D.vocab * d, (T*)m->embed));
    TW_CHECK(put<T>(m, wt, Dc + "embed_positions.weight", (int64_t)D.max_target * d, (T*)m->dec_pos));
    m->dec.resize(D.dec_layers);
    for (int l = 0; l < D.dec_layers; ++l) {
        const std::string p = Dc + "layers." + std::to_string(l) + ".";
        LayerW& L = m->dec[l];
        TW_CHECK(load_ln(m, wt, p + "self_attn_layer_norm", &L.ln1_g, &L.ln1_b));
        TW_CHECK(load_attn<T>(m, wt, p + "self_attn.", L.self, false));
        TW_CHECK(load_ln(m, wt, p + "encoder_attn_layer_norm", &L.ln2_g, &L.ln2_b));
        TW_CHECK(load_attn<T>(m, wt, p + "encoder_attn.", L.cross, true));
        TW_CHECK(load_ln(m, wt, p + "final_layer_norm", &L.ln3_g, &L.ln3_b));
        TW_CHECK(load_mlp<T>(m, wt, p, L));
    }
    TW_CHECK(load_ln(m, wt, Dc + "layer_norm", &m->dec_lnf_g, &m->dec_lnf_b));
    TW_CUDA_OK(m->ctx, cudaDeviceSynchronize());
    TW_CUDA_OK(m->ctx, cudaGetLastError());
    return TW_OK;
}

int alloc_workspace(tw_model* m) {
    const tw_model_desc& D = m->desc;
    const size_t B = D.max_batch, d = D.d_model, e = m->esz;
    const size_t M = B * TW_N_CTX;
    TW_CHECK(dev_alloc(m, (void**)&m->ws_pcm, B * TW_N_SAMPLES * sizeof(int16_t)));
    TW_CHECK(dev_alloc(m, (void**)&m->ws_nvalid, B * sizeof(int32_t)));
    TW_CHECK(dev_alloc(m, (void**)&m->ws_mel, B * D.n_mel * TW_N_FRAMES * sizeof(float)));
    TW_CHECK(dev_alloc(m, &m->ws_a1, B * TW_N_FRAMES * 3 * D.n_mel * e));
    TW_CHECK(dev_alloc(m, &m->ws_h0, B * TW_N_FRAMES * d * e));
    TW_CHECK(dev_alloc(m, &m->ws_a2qkv, M * 3 * d * e));
    TW_CHECK(dev_alloc(m, (void**)&m->ws_x, M * d * sizeof(float)));
    TW_CHECK(dev_alloc(m, &m->ws_xn, M * d * e));
    TW_CHECK(dev_alloc(m, &m->ws_att, M * d * e));
    TW_CHECK(dev_alloc(m, &m->ws_hmid, M * D.ffn * e));
    TW_CHECK(dev_alloc(m, &m->ws_enc, M * d * e));
    TW_CHECK(dev_alloc(m, &m->xkv, (size_t)D.dec_layers * M * 2 * d * e));
    m->kv_pages = (D.max_target + TW_KV_PAGE - 1) / TW_KV_PAGE;
    TW_CHECK(dev_alloc(m, &m->self_kv, (size_t)D.dec_layers * B * m->kv_pages * TW_KV_PAGE * 2 * d * e));
    TW_CHECK(dev_alloc(m, (void**)&m->d_page_table, B * m->kv_pages * sizeof(int32_t)));
    TW_CUDA_OK(m->ctx, cudaMallocHost(&m->h_page_table, B * m->kv_pages * sizeof(int32_t)));
    TW_CHECK(dev_alloc(m, (void**)&m->dx, B * d * sizeof(float)));
    TW_CHECK(dev_alloc(m, &m->dxn, B * d * e));
    TW_CHECK(dev_alloc(m, &m->dqkv, B * 3 * d * e));
    TW_CHECK(dev_alloc(m, &m->datt, B * d * e));
    TW_CHECK(dev_alloc(m, &m->dq, B * d * e));
    TW_CHECK(dev_alloc(m, &m->dhmid, B * D.ffn * e));
    if (m->absorb_ok) {
        const size_t Bd = B < 64 ? B : 64;          // the absorbed path serves decode batches of up to 64 clips (skinny GEMMs)
        TW_CHECK(dev_alloc(m, &m->dqt, (Bd * D.heads + ABSORB_QT_PAD) * d * e));
        TW_CUDA_OK(m->ctx, cudaMemset(m->dqt, 0, (Bd * D.heads + ABSORB_QT_PAD) * d * e));
        TW_CHECK(dev_alloc(m, &m->dctx, Bd * D.heads * d * e));
        TW_CUDA_OK(m->ctx, cudaMemset(m->dctx, 0, Bd * D.heads * d * e));
        TW_CHECK(dev_alloc(m, (void**)&m->dab_partial, absorbed_attention_partial_floats((int)Bd, D.heads, (int)d) * sizeof(float)));
    }
    m->ld_logits = ((int64_t)D.vocab + 3) / 4 * 4;
    TW_CHECK(dev_alloc(m, (void**)&m->dlogits, B * (size_t)m->ld_logits * sizeof(float)));
    const size_t partial_floats = decode_attention_partial_floats((int)B, D.heads);
    TW_CHECK(dev_alloc(m, (void**)&m->dpartial, partial_floats * sizeof(float)));
    TW_CUDA_OK(m->ctx, cudaMemset(m->dpartial, 0, partial_floats * sizeof(float)));
    TW_CHECK(dev_alloc(m, (void**)&m->dstate, (8 * B + 8) * sizeof(int32_t)));
    m->d_row_budget = m->dstate + 7 * B;
    // the selection kernel reads the masks four bytes at a time: padded to whole words (pad bytes stay zero)
    TW_CHECK(dev_alloc(m, (void**)&m->d_suppress, D.vocab + 16));
    TW_CHECK(dev_alloc(m, (void**)&m->d_begin_suppress, D.vocab + 16));
    TW_CUDA_OK(m->ctx, cudaMemset(m->d_suppress, 0, D.vocab + 16));
    TW_CUDA_OK(m->ctx, cudaMemset(m->d_begin_suppress, 0, D.vocab + 16));
    TW_CHECK(dev_alloc(m, (void**)&m->d_ids_tmp, 4096 * sizeof(int32_t)));
    TW_CHECK(dev_alloc(m, (void**)&m->d_out_tok, B * D.max_target * sizeof(int32_t)));
    TW_CHECK(dev_alloc(m, (void**)&m->d_out_len, B * sizeof(int32_t)));
    for (auto& ev : m->ev) TW_CUDA_OK(m->ctx, cudaEventCreate(&ev));
    TW_CUDA_OK(m->ctx, cudaMallocHost(&m->h_flag, 64));
    TW_CUDA_OK(m->ctx, cudaMallocHost(&m->h_step, STEP_INTS * sizeof(int32_t)));
    TW_CHECK(dev_alloc(m, (void**)&m->d_step, STEP_INTS * sizeof(int32_t)));
    TW_CHECK(dev_alloc(m, (void**)&m->d_row_prompt, (B * PROMPT_MAX + MAX_LANG_IDS) * sizeof(int32_t)));
    m->d_lang_ids = m->d_row_prompt + B * PROMPT_MAX;
    TW_CUDA_OK(m->ctx, cudaMallocHost(&m->h_rows, (B * PROMPT_MAX + MAX_LANG_IDS) * sizeof(int32_t)));
    TW_CHECK(dev_alloc(m, (void**)&m->d_out_lang, B * sizeof(int32_t)));
    TW_CUDA_OK(m->ctx, cudaStreamCreateWithFlags(&m->cap_stream, cudaStreamNonBlocking));
    return TW_OK;
}

// ---- GEMM dispatch: tcgen05 for bf16 (unless TWB200_GEMM=simt), CUDA-core FMA for the fp32 check mode
template <typename T>
int gemm(tw_model* m, const T* A, int64_t lda, const T* W, int64_t ldw, int M, int N, int K, const GemmEpi& epi, cudaStream_t st);

template <>
int gemm<float>(tw_model* m, const float* A, int64_t lda, const float* W, int64_t ldw, int M, int N, int K, const GemmEpi& epi,
                cudaStream_t st) {
    gemm_simt<float>(A, lda, W, ldw, M, N, K, epi, st);
    m->ctx->launches += 1;
    return TW_OK;
}
template <>
int gemm<__nv_bfloat16>(tw_model* m, const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* W, int64_t ldw, int M, int N, int K,
                        const GemmEpi& epi, cudaStream_t st) {
    m->ctx->launches += 1;
    if (m->use_tc && m->use_tc_skinny && gemm_tc_skinny_supported(M, N, K, epi)) return gemm_tc_skinny(m->ctx, A, lda, W, ldw, M, N, K, epi, st);
    if (m->use_tc) return gemm_tc(m->ctx, A, lda, W, ldw, M, N, K, epi, st);
    gemm_simt<__nv_bfloat16>(A, lda, W, ldw, M, N, K, epi, st);
    return TW_OK;
}

template <typename T>
int enc_attention(tw_model* m, const T* qkv, T* att, int B, cudaStream_t st);
template <>
int enc_attention<float>(tw_model* m, const float* qkv, float* att, int B, cudaStream_t st) {
    encoder_attention_simt<float>(qkv, att, B, TW_N_CTX, m->desc.heads, st);
    return TW_OK;
}
template <>
int enc_attention<__nv_bfloat16>(tw_model* m, const __nv_bfloat16* qkv, __nv_bfloat16* att, int B, cudaStream_t st) {
    if (m->use_tc_attn) return encoder_attention_tc(m->ctx, qkv, att, B, TW_N_CTX, m->desc.heads, st);
    encoder_attention_simt<__nv_bfloat16>(qkv, att, B, TW_N_CTX, m->desc.heads, st);
    return TW_OK;
}

// attention on separate query / key-value matrices (full-sequence decoder pass): tcgen05 kernel for bf16, CUDA-core kernel
// for the fp32 check mode (and for bf16 with TWB200_ATTN=simt)
template <typename T>
int seq_attention(tw_model* m, const T* q, int64_t q_ld, int q_col0, const T* kv, int64_t kv_ld, int k_col0, int v_col0, T* out, int B,
                  int Sq, int Sk, bool causal, cudaStream_t st);
template <>
int seq_attention<float>(tw_model* m, const float* q, int64_t q_ld, int q_col0, const float* kv, int64_t kv_ld, int k_col0, int v_col0,
                         float* out, int B, int Sq, int Sk, bool causal, cudaStream_t st) {
    attention_simt<float>(q + q_col0, q_ld, kv + k_col0, kv + v_col0, kv_ld, out, B, Sq, Sk, m->desc.heads, causal, st);
    return TW_OK;
}
template <>
int seq_attention<__nv_bfloat16>(tw_model* m, const __nv_bfloat16* q, int64_t q_ld, int q_col0, const __nv_bfloat16* kv, int64_t kv_ld,
                                 int k_col0, int v_col0, __nv_bfloat16* out, int B, int Sq, int Sk, bool causal, cudaStream_t st) {
    if (m->use_tc_attn) return attention_tc(m->ctx, q, q_ld, q_col0, kv, kv_ld, k_col0, v_col0, out, B, Sq, Sk, m->desc.heads, causal, st);
    attention_simt<__nv_bfloat16>(q + q_col0, q_ld, kv + k_col0, kv + v_col0, kv_ld, out, B, Sq, Sk, m->desc.heads, causal, st);
    return TW_OK;
}

inline GemmEpi mk_epi(int mode, const float* bias, void* C, int64_t ldc, const float* pos = nullptr, int period = 1) {
    GemmEpi e;
    e.mode = mode; e.bias = bias; e.C = C; e.ldc = ldc; e.pos = pos; e.pos_period = period;
    return e;
}

template <typename T>
int encode_impl(tw_model* m, const float* mel, int B, void* enc_out, int tap_layer, float* tap_out, cudaStream_t st,
                const float* mel_clip_max = nullptr) {
    const tw_model_desc& D = m->desc;
    const int d = D.d_model, M = B * TW_N_CTX, M0 = B * TW_N_FRAMES, K1 = 3 * D.n_mel;
    tw_ctx* ctx = m->ctx;
    T* a1 = (T*)m->ws_a1; T* h0 = (T*)m->ws_h0; T* a2 = (T*)m->ws_a2qkv; T* qkv = (T*)m->ws_a2qkv;
    T* xn = (T*)m->ws_xn; T* att = (T*)m->ws_att; T* hmid = (T*)m->ws_hmid;
    float* x = m->ws_x;
    im2col_conv1<T>(mel, a1, B, D.n_mel, st, mel_clip_max);
    TW_CHECK(gemm<T>(m, a1, K1, (const T*)m->conv1_w, K1, M0, d, K1, mk_epi(EPI_GELU, m->conv1_b, h0, d), st));
    im2col_conv2<T>(h0, a2, B, d, st);
    TW_CHECK(gemm<T>(m, a2, 3 * d, (const T*)m->conv2_w, 3 * d, M, d, 3 * d,
                     mk_epi(EPI_GELU_POS, m->conv2_b, x, d, m->enc_pos, TW_N_CTX), st));
    ctx->launches += 2;
    if (tap_layer == 0 && tap_out) { copy_f32(x, tap_out, (int64_t)M * d, st); ctx->launches += 1; }
    // programmatic dependent launch along this chain was measured and lost (encoder 157.4 vs 152.7 ms per 64 clips: the early-
    // resident dependents hold shared memory / TMEM while they wait), so the encoder's kernels are plain stream-ordered launches
    for (int l = 0; l < D.enc_layers; ++l) {
        const LayerW& L = m->enc[l];
        layernorm<T>(x, L.ln1_g, L.ln1_b, xn, M, d, st);
        TW_CHECK(gemm<T>(m, xn, d, (const T*)L.self.qkv_w, d, M, 3 * d, d, mk_epi(EPI_STORE, L.self.qkv_b, qkv, 3 * d), st));
        TW_CHECK(enc_attention<T>(m, qkv, att, B, st));
        TW_CHECK(gemm<T>(m, att, d, (const T*)L.self.o_w, d, M, d, d, mk_epi(EPI_RESID, L.self.o_b, x, d), st));
        layernorm<T>(x, L.ln3_g, L.ln3_b, xn, M, d, st);
        TW_CHECK(gemm<T>(m, xn, d, (const T*)L.fc1_w, d, M, D.ffn, d, mk_epi(EPI_GELU, L.fc1_b, hmid, D.ffn), st));
        TW_CHECK(gemm<T>(m, hmid, D.ffn, (const T*)L.fc2_w, D.ffn, M, d, D.ffn, mk_epi(EPI_RESID, L.fc2_b, x, d), st));
        ctx->launches += 3;
        if (tap_layer == l + 1 && tap_out) { copy_f32(x, tap_out, (int64_t)M * d, st); ctx->launches += 1; }
    }
    layernorm<T>(x, m->enc_lnf_g, m->enc_lnf_b, (T*)enc_out, M, d, st);
    ctx->launches += 1;
    TW_CUDA_OK(ctx, cudaGetLastError());
    return TW_OK;
}

template <typename T>
int cross_kv_impl(tw_model* m, const void* enc_out, int B, cudaStream_t st, int clip0 = 0) {
    const tw_model_desc& D = m->desc;
    const int d = D.d_model, M = B * TW_N_CTX;
    for (int l = 0; l < D.dec_layers; ++l) {
        // rows of clips clip0 .. clip0 + B - 1 of the layer's store (clip0 > 0: a later part of a merged decode batch)
        T* dst = (T*)m->xkv + ((size_t)l * D.max_batch + clip0) * TW_N_CTX * 2 * d;
        TW_CHECK(gemm<T>(m, (const T*)enc_out, d, (const T*)m->dec[l].cross.kv_w, d, M, 2 * d, d,
                         mk_epi(EPI_STORE, m->dec[l].cross.kv_b, dst, 2 * d), st));
    }
    TW_CUDA_OK(m->ctx, cudaGetLastError());
    return TW_OK;
}

// Full-sequence (teacher-forced) decoder pass: logits for every position of decoder_input_ids [B, Tn] in one batched
// pass at M = B * Tn rows — the teacher forward of the distillation step (ref knowledge-distillation/run_distillation.py:
// 1543-1577: teacher_model(encoder_outputs=..., labels=...) / teacher_model(**batch); HF WhisperDecoder.forward
// modeling_whisper.py:691-798 with the causal mask, WhisperForConditionalGeneration.forward :1081).  Reuses the GEMM /
// LayerNorm kernels of the encoder at these row counts and the encoder's workspace (both passes are never in flight
// together); attention is the encoder's tcgen05 flash kernel on separate query / key-value matrices (causal over the Tn
// tokens, then over the K|V store), the general CUDA-core kernel in fp32 check mode.
// tap (nullable): fp32 [L_dec + 1, B*Tn, d], the residual after the embedding and after every decoder layer.
template <typename T>
int decoder_logits_impl(tw_model* m, int B, const int32_t* ids, int Tn, float* logits, int64_t ld_logits, cudaStream_t st,
                        float* tap = nullptr) {
    const tw_model_desc& D = m->desc;
    tw_ctx* ctx = m->ctx;
    const int d = D.d_model, V = D.vocab, M = B * Tn;
    float* x = m->ws_x;
    T* xn = (T*)m->ws_xn; T* qkv = (T*)m->ws_a2qkv; T* att = (T*)m->ws_att; T* hmid = (T*)m->ws_hmid; T* q = (T*)m->ws_h0;
    const size_t cross_layer = (size_t)D.max_batch * TW_N_CTX * 2 * d;
    embed_tokens_seq<T>(ids, (const T*)m->embed, (const T*)m->dec_pos, x, B, Tn, d, V, st);
    if (tap) { copy_f32(x, tap, (int64_t)M * d, st); ctx->launches += 1; }
    for (int l = 0; l < D.dec_layers; ++l) {
        const LayerW& L = m->dec[l];
        const T* xkv = (const T*)m->xkv + l * cross_layer;
        layernorm<T>(x, L.ln1_g, L.ln1_b, xn, M, d, st);
        TW_CHECK(gemm<T>(m, xn, d, (const T*)L.self.qkv_w, d, M, 3 * d, d, mk_epi(EPI_STORE, L.self.qkv_b, qkv, 3 * d), st));
        TW_CHECK(seq_attention<T>(m, qkv, 3 * d, 0, qkv, 3 * d, d, 2 * d, att, B, Tn, Tn, true, st));
        TW_CHECK(gemm<T>(m, att, d, (const T*)L.self.o_w, d, M, d, d, mk_epi(EPI_RESID, L.self.o_b, x, d), st));
        layernorm<T>(x, L.ln2_g, L.ln2_b, xn, M, d, st);
        TW_CHECK(gemm<T>(m, xn, d, (const T*)L.cross.q_w, d, M, d, d, mk_epi(EPI_STORE, L.cross.q_b, q, d), st));
        TW_CHECK(seq_attention<T>(m, q, d, 0, xkv, 2 * d, 0, d, att, B, Tn, TW_N_CTX, false, st));
        TW_CHECK(gemm<T>(m, att, d, (const T*)L.cross.o_w, d, M, d, d, mk_epi(EPI_RESID, L.cross.o_b, x, d), st));
        layernorm<T>(x, L.ln3_g, L.ln3_b, xn, M, d, st);
        TW_CHECK(gemm<T>(m, xn, d, (const T*)L.fc1_w, d, M, D.ffn, d, mk_epi(EPI_GELU, L.fc1_b, hmid, D.ffn), st));
        TW_CHECK(gemm<T>(m, hmid, D.ffn, (const T*)L.fc2_w, D.ffn, M, d, D.ffn, mk_epi(EPI_RESID, L.fc2_b, x, d), st));
        ctx->launches += 5;       // 3 LN, 2 attention; the GEMMs count themselves
        if (tap) { copy_f32(x, tap + (size_t)(l + 1) * M * d, (int64_t)M * d, st); ctx->launches += 1; }
    }
    layernorm<T>(x, m->dec_lnf_g, m->dec_lnf_b, xn, M, d, st);
    TW_CHECK(gemm<T>(m, xn, d, (const T*)m->embed, d, M, V, d, mk_epi(EPI_F32, nullptr, logits, ld_logits), st));
    ctx->launches += 2;           // embed, LN
    TW_CUDA_OK(ctx, cudaGetLastError());
    return TW_OK;
}

int upload_rules(tw_model* m, const tw_rules* R, RulesDev* out, cudaStream_t st) {
    tw_ctx* ctx = m->ctx;
    const int V = m->desc.vocab;
    if (R->n_suppress < 0 || R->n_begin_suppress < 0 || R->n_suppress + R->n_begin_suppress > 4096) {
        ctx->set_error(TW_E_INVALID, "tw_rules: too many suppress ids");
        return TW_E_INVALID;
    }
    TW_CUDA_OK(ctx, cudaMemsetAsync(m->d_suppress, 0, V, st));
    TW_CUDA_OK(ctx, cudaMemsetAsync(m->d_begin_suppress, 0, V, st));
    if (R->n_suppress > 0) {
        TW_CUDA_OK(ctx, cudaMemcpyAsync(m->d_ids_tmp, R->suppress, R->n_suppress * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        mask_from_ids_kernel<<<ceil_div(R->n_suppress, 256), 256, 0, st>>>(m->d_ids_tmp, R->n_suppress, m->d_suppress, V);
    }
    if (R->n_begin_suppress > 0) {
        int32_t* tmp = m->d_ids_tmp + R->n_suppress;
        TW_CUDA_OK(ctx, cudaMemcpyAsync(tmp, R->begin_suppress, R->n_begin_suppress * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        mask_from_ids_kernel<<<ceil_div(R->n_begin_suppress, 256), 256, 0, st>>>(tmp, R->n_begin_suppress, m->d_begin_suppress, V);
    }
    // the host arrays may be pageable: make sure the copies are done before the caller reuses them
    TW_CUDA_OK(ctx, cudaStreamSynchronize(st));
    out->suppress_mask = m->d_suppress;
    out->begin_suppress_mask = m->d_begin_suppress;
    out->eos = R->eos;
    out->pad = R->pad;
    out->ts_begin = R->timestamp_begin;
    out->no_timestamps = R->no_timestamps;
    out->max_initial_ts = R->max_initial_timestamp_index;
    return TW_OK;
}

__global__ void fill_pad_kernel(int32_t* out_tokens, int B, int stride, int from_g, int pad) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int span = stride - from_g;
    if (span > 0 && i < B * span) out_tokens[(int64_t)(i / span) * stride + from_g + (i % span)] = pad;
}

struct StepIo {
    int32_t* out_tokens;
    int32_t* out_lengths;
    const int32_t* forced;
    float* logits_tap;
    float* layer_tap;    // nullable: fp32 [L_dec + 1, B, d], the residual after the embedding and after every layer of this step
    int32_t* out_lang;   // nullable: [B] the language each row is decoded with (written by the language pick of step 0)
};

// Absorbed cross-attention of one decoder layer (absorb.cu): q [B, d] -> att [B, d] (the input of the output projection).
//   q~ = per-head Wk^T q (grouped GEMM, K = 64), c = softmax(q~ . E^T) E streamed from the encoder output, o = per-head Wv c + bv
template <typename T>
int cross_absorbed(tw_model* m, const LayerW& L, const T* q, T* att, int B, int layer, cudaStream_t st, cudaEvent_t e0, cudaEvent_t e1,
                   const DecodeState& S);
template <>
int cross_absorbed<float>(tw_model* m, const LayerW&, const float*, float*, int, int, cudaStream_t, cudaEvent_t, cudaEvent_t, const DecodeState&) {
    m->ctx->set_error(TW_E_UNSUPPORTED, "absorbed cross-attention is a bf16 path");
    return TW_E_UNSUPPORTED;
}
template <>
int cross_absorbed<__nv_bfloat16>(tw_model* m, const LayerW& L, const __nv_bfloat16* q, __nv_bfloat16* att, int B, int layer, cudaStream_t st,
                                  cudaEvent_t e0, cudaEvent_t e1, const DecodeState& S) {
    typedef __nv_bfloat16 T;
    const int d = m->desc.d_model, H = m->desc.heads;
    const char* er = getenv("TWB200_AB_REV");
    const bool serpentine = !(er && strcmp(er, "0") == 0);
    GemmEpi qe = mk_epi(EPI_STORE, nullptr, m->dqt, (int64_t)H * d);
    qe.group_n = d;
    TW_CHECK(gemm<T>(m, q, d, (const T*)L.cross.kt_w, 64, B, H * d, 64, qe, st));
    TW_CHECK(absorbed_attention(m->ctx, (const T*)m->dqt, (const T*)m->cur_enc, TW_N_CTX, B, H, d, m->dab_partial, (T*)m->dctx, st, S.active,
                                S.n_active, serpentine ? (layer & 1) : 0, e0, e1));
    GemmEpi ve = mk_epi(EPI_STORE, L.cross.kv_b + d, att, d);
    ve.group_n = 64;
    TW_CHECK(gemm<T>(m, (const T*)m->dctx, (int64_t)H * d, (const T*)L.cross.kv_w + (size_t)d * d, d, B, d, d, ve, st));
    return TW_OK;
}

// One decode step (all kernels of one token position).  Position, prompt and output stride are read from
// m->d_step on the device, so the same launch sequence — or one captured CUDA graph — serves every position.
template <typename T>
// pick: step 0 of a call that detects languages (or reports them) — the language pick replaces the token selection.  Step 0 is
// always launched eagerly (the graph is captured at pos >= 1), so the replayed step never contains the pick.
int launch_step(tw_model* m, int B, const RulesDev& R, const DecodeState& S, const StepIo& io, cudaStream_t st, bool pick = false,
                bool trace = false) {
    const tw_model_desc& D = m->desc;
    tw_ctx* ctx = m->ctx;
    const int d = D.d_model, V = D.vocab, H = D.heads;
    float* x = m->dx;
    T* xn = (T*)m->dxn; T* qkv = (T*)m->dqkv; T* att = (T*)m->datt; T* q = (T*)m->dq; T* hmid = (T*)m->dhmid;
    const size_t self_layer = (size_t)D.max_batch * m->kv_pages * TW_KV_PAGE * 2 * d;      // one layer's page pool
    const size_t cross_layer = (size_t)D.max_batch * TW_N_CTX * 2 * d;
    const int32_t* d_pos = m->d_step + STEP_POS;
    // PDL only on the bf16 product path: every kernel launched below goes through launch_k and executes pdl_wait()
    const bool pdl_on = m->use_pdl && sizeof(T) == 2 && m->use_tc;
    struct FlagScope {
        explicit FlagScope(bool pdl) { g_pdl = pdl; }
        ~FlagScope() { g_pdl = false; }
    } flag_scope(pdl_on);
    auto mark = [&](int l, const char* name) {
        if (!trace || (l >= 0 && l != D.dec_layers / 2 && l != D.dec_layers / 2 + 1)) return;
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return;
        cudaEventRecord(e, st);
        m->trace.emplace_back(e, "L" + std::to_string(l) + " " + name);
    };
    // the step's first kernel is launched with a FULL dependency on the previous step (no programmatic early start): every
    // later kernel of the step starts after this one did, so state written by the previous step's select / advance kernels
    // (finished flags, active-clip list) may be read by them even ahead of their own griddepcontrol.wait
    g_pdl = false;
    embed_tokens<T>(S.cur_tok, (const T*)m->embed, (const T*)m->dec_pos, m->d_step, x, B, d, st);
    g_pdl = pdl_on;
    mark(-1, "embed");
    // taps: plain stream-ordered copies (no programmatic early start), so each reads x after the kernel before it is done
    if (io.layer_tap) { copy_f32(x, io.layer_tap, (int64_t)B * d, st); ctx->launches += 1; }
    const int32_t* pt = m->d_page_table;
    const int skip = m->skip_mask;
    for (int l = 0; l < D.dec_layers; ++l) {
        const LayerW& L = m->dec[l];
        T* cache = (T*)m->self_kv + l * self_layer;                       // the layer's page pool
        if (!(skip & 1)) layernorm<T>(x, L.ln1_g, L.ln1_b, xn, B, d, st);
        mark(l, "ln1");
        GemmEpi qe = mk_epi(EPI_STORE, L.self.qkv_b, qkv, 3 * d);
        // the K|V columns of the fused QKV projection land in the cache row of this position — only the skinny tcgen05
        // kernel (M <= 256) implements the column split; larger batches append with a separate kernel
        const bool fused_append = (sizeof(T) == 2) && m->use_tc && m->use_tc_skinny && gemm_tc_skinny_supported(B, 3 * d, d, qe);
        if (fused_append) {
            qe.n_split = d;
            qe.C2 = cache;
            qe.ldc2 = 0;
            qe.d_row2 = d_pos;
            qe.row2_stride = 2 * d;
            qe.page_table = pt;
            qe.pt_stride = m->kv_pages;
        }
        if (!(skip & 8)) TW_CHECK(gemm<T>(m, xn, d, (const T*)L.self.qkv_w, d, B, 3 * d, d, qe, st));
        mark(l, "qkv");
        if (!fused_append) { kv_append<T>(qkv, cache, m->d_step, B, d, D.max_target, st, pt, m->kv_pages); ctx->launches += 1; }
        if (!(skip & 2)) self_attention_decode<T>(qkv, 3 * d, cache, 0, 0, d_pos, B, H, att, st, pt, m->kv_pages, S.finished);
        mark(l, "self_attn");
        if (!(skip & 16)) TW_CHECK(gemm<T>(m, att, d, (const T*)L.self.o_w, d, B, d, d, mk_epi(EPI_RESID, L.self.o_b, x, d), st));
        mark(l, "self_o");
        if (!(skip & 1)) layernorm<T>(x, L.ln2_g, L.ln2_b, xn, B, d, st);
        mark(l, "ln2");
        if (!(skip & 32)) TW_CHECK(gemm<T>(m, xn, d, (const T*)L.cross.q_w, d, B, d, d, mk_epi(EPI_STORE, L.cross.q_b, q, d), st));
        mark(l, "cross_q");
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (m->prof_on && l == D.dec_layers / 2 && m->prof_used + 2 <= (int)m->prof_ev.size()) {
            e0 = m->prof_ev[m->prof_used];
            e1 = m->prof_ev[m->prof_used + 1];
            m->prof_used += 2;
            m->prof_bytes = (double)B * TW_N_CTX * (m->absorb_now ? 1 : 2) * d * sizeof(T);
        }
        if (skip & 4) {
        } else if (m->absorb_now) {
            TW_CHECK(cross_absorbed<T>(m, L, q, att, B, l, st, e0, e1, S));
        } else {
            decode_attention<T>(q, d, (const T*)m->xkv + l * cross_layer, (int64_t)TW_N_CTX * 2 * d, TW_N_CTX, nullptr, B, H, m->dpartial, att,
                                st, e0, e1, S.active, S.n_active);
        }
        mark(l, "cross_attn+combine");
        if (!(skip & 64)) TW_CHECK(gemm<T>(m, att, d, (const T*)L.cross.o_w, d, B, d, d, mk_epi(EPI_RESID, L.cross.o_b, x, d), st));
        mark(l, "cross_o");
        if (!(skip & 1)) layernorm<T>(x, L.ln3_g, L.ln3_b, xn, B, d, st);
        mark(l, "ln3");
        if (!(skip & 128)) TW_CHECK(gemm<T>(m, xn, d, (const T*)L.fc1_w, d, B, D.ffn, d, mk_epi(EPI_GELU, L.fc1_b, hmid, D.ffn), st));
        mark(l, "fc1");
        if (!(skip & 256)) TW_CHECK(gemm<T>(m, hmid, D.ffn, (const T*)L.fc2_w, D.ffn, B, d, D.ffn, mk_epi(EPI_RESID, L.fc2_b, x, d), st));
        mark(l, "fc2");
        ctx->launches += 6;       // 3 LN, self-attention, cross-attention stream + combine; the GEMMs count themselves
        if (io.layer_tap) { copy_f32(x, io.layer_tap + (size_t)(l + 1) * B * d, (int64_t)B * d, st); ctx->launches += 1; }
    }
    layernorm<T>(x, m->dec_lnf_g, m->dec_lnf_b, xn, B, d, st);
    TW_CHECK(gemm<T>(m, xn, d, (const T*)m->embed, d, B, V, d, mk_epi(EPI_F32, nullptr, m->dlogits, m->ld_logits), st));
    if (pick) pick_language(m->dlogits, m->ld_logits, B, m->d_lang_ids, m->n_lang_now, S, io.out_lang, st);
    else select_tokens(m->dlogits, m->ld_logits, V, B, m->d_step, R, S, io.out_tokens, io.out_lengths, io.forced, io.logits_tap, st);
    advance_step(m->d_step, S, B, st);
    ctx->launches += 4;           // embed, LN, select (or the language pick), advance
    return TW_OK;
}

// Decode state of one call (the model's dstate arrays, initialised for B rows), the cleared out_lengths, the step header (position 0,
// prompt length, output stride, tapped steps), the per-row prompt table and the language ids on the device: shared by decode_impl and
// tw_debug_select_steps.  rows.prompts is host [B][P] (checked by check_prompt_rows).
int begin_decode(tw_model* m, int B, const tw_prompt_rows& rows, int P, int max_length, int32_t* out_lengths, float* logits_tap,
                 int tap_steps, cudaStream_t st, DecodeState* out) {
    const tw_model_desc& D = m->desc;
    tw_ctx* ctx = m->ctx;
    DecodeState& S = *out;
    S.cur_tok = m->dstate;
    S.finished = m->dstate + D.max_batch;
    S.n_gen = m->dstate + 2 * D.max_batch;
    S.last_tok = m->dstate + 3 * D.max_batch;
    S.prev_tok = m->dstate + 4 * D.max_batch;
    S.last_ts = m->dstate + 5 * D.max_batch;
    S.active = m->dstate + 6 * D.max_batch;
    S.row_budget = m->row_budget_on ? m->d_row_budget : nullptr;
    S.n_unfinished = m->dstate + 8 * D.max_batch;
    S.n_active = m->dstate + 8 * D.max_batch + 1;
    S.prompt = m->d_row_prompt;
    decode_state_init(S, B, rows.prompts[0], st);          // SOT: the same in every row
    TW_CUDA_OK(ctx, cudaMemsetAsync(out_lengths, 0, B * sizeof(int32_t), st));
    // step header -> device (pinned staging so the copy is stream-ordered)
    int32_t* hs = m->h_step;
    TW_CUDA_OK(ctx, cudaStreamSynchronize(st));          // previous call may still be reading h_step
    for (int i = 0; i < STEP_INTS; ++i) hs[i] = 0;
    hs[STEP_POS] = 0; hs[STEP_P] = P; hs[STEP_STRIDE] = max_length - P; hs[STEP_TAP] = logits_tap ? tap_steps : 0;
    TW_CUDA_OK(ctx, cudaMemcpyAsync(m->d_step, hs, STEP_INTS * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    // prompt table (rows B .. max_batch - 1 are not read) and language ids, from pinned staging like the step header
    int32_t* hp = m->h_rows;
    bool detect = false;
    for (int b = 0; b < B; ++b)
        for (int i = 0; i < PROMPT_MAX; ++i) {
            hp[b * PROMPT_MAX + i] = i < P ? rows.prompts[(size_t)b * P + i] : 0;
            detect |= (i == 1 && i < P && hp[b * PROMPT_MAX + i] == PROMPT_DETECT);
        }
    TW_CUDA_OK(ctx, cudaMemcpyAsync(m->d_row_prompt, hp, (size_t)B * PROMPT_MAX * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    m->n_lang_now = rows.lang_ids ? rows.n_lang : 0;
    if (m->n_lang_now > 0) {
        int32_t* hl = hp + D.max_batch * PROMPT_MAX;
        for (int j = 0; j < m->n_lang_now; ++j) hl[j] = rows.lang_ids[j];
        TW_CUDA_OK(ctx, cudaMemcpyAsync(m->d_lang_ids, hl, m->n_lang_now * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    }
    m->pick_now = detect || rows.out_lang;
    ctx->launches += 1;
    return TW_OK;
}

// Residual taps of a decode call (tw_debug_decode_taps): positions pos0 .. pos0 + n_pos - 1 into layer [n_pos, L_dec + 1, B, d].
struct DecodeTaps {
    float* layer = nullptr;
    int pos0 = 0, n_pos = 0;
};

template <typename T>
int decode_impl(tw_model* m, int B, const tw_prompt_rows& rows, int P, const RulesDev& R, int max_length, int32_t* out_tokens,
                int32_t* out_lengths, const int32_t* forced, float* logits_tap, int tap_steps, cudaStream_t st,
                const DecodeTaps& taps = DecodeTaps{}) {
    tw_ctx* ctx = m->ctx;
    const int n_gen_max = max_length - P;
    DecodeState S;
    TW_CHECK(begin_decode(m, B, rows, P, max_length, out_lengths, logits_tap, tap_steps, st, &S));
    // page table of this call: only the ceil(max_length / TW_KV_PAGE) pages a clip can reach are mapped, page-major
    // (logical page p of clip b -> physical page p*B + b), so a call touches a dense prefix of every layer's pool whose
    // size follows B and max_length, and the B cache rows written by one step are adjacent
    {
        const int pages_call = (max_length + TW_KV_PAGE - 1) / TW_KV_PAGE;
        for (int b = 0; b < B; ++b)
            for (int p = 0; p < m->kv_pages; ++p) m->h_page_table[b * m->kv_pages + p] = p < pages_call ? p * B + b : -1;
        TW_CUDA_OK(ctx, cudaMemcpyAsync(m->d_page_table, m->h_page_table, (size_t)B * m->kv_pages * sizeof(int32_t),
                                        cudaMemcpyHostToDevice, st));
    }

    // CUDA graph of one step: production path only (no teacher forcing / taps / per-launch profiling events)
    const bool want_graph = m->use_graph && !forced && !logits_tap && !taps.layer && !m->prof_on && m->trace_pos < 0;
    // the graph bakes in its output pointers: decode into the model-owned buffers, copy out at the end
    StepIo io{out_tokens, out_lengths, forced, logits_tap, nullptr, rows.out_lang};
    if (want_graph) io = StepIo{m->d_out_tok, m->d_out_len, nullptr, nullptr, nullptr, rows.out_lang};
    if (want_graph) TW_CUDA_OK(ctx, cudaMemsetAsync(m->d_out_len, 0, B * sizeof(int32_t), st));
    m->skip_mask = getenv("TWB200_SKIP") ? atoi(getenv("TWB200_SKIP")) : 0;      // re-read per call: one process can sweep masks
    GraphKey key{B, R.eos, R.pad, R.ts_begin, R.no_timestamps, R.max_initial_ts, (m->row_budget_on ? 1 : 0) | (m->skip_mask << 1),
                 m->absorb_now ? m->cur_enc : nullptr, m->xkv, ctx->sm_count};
    cudaGraphExec_t exec = nullptr;
    uint64_t exec_kernels = 0;

    int32_t* h_unfinished = m->h_flag;
    *h_unfinished = B;
    bool check_pending = false;
    int steps_done = 0;
    for (int pos = 0; pos < max_length - 1; ++pos) {
        if (want_graph && pos >= 1 && !exec) {
            auto it = m->graphs.find(key);
            if (it != m->graphs.end()) {
                exec = it->second.exec;
                exec_kernels = it->second.kernels;
            } else {
                // capture one step on the model's private stream (nothing executes during capture)
                cudaGraph_t graph = nullptr;
                const uint64_t l0 = ctx->launches;
                // kernel nodes run in the context of the CAPTURE stream: under the pipeline that must be the decode partition
                cudaStream_t cap = m->pipe.in_decode ? m->pipe.s_cap : m->cap_stream;
                TW_CUDA_OK(ctx, cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal));
                int rc = launch_step<T>(m, B, R, S, io, cap);
                cudaError_t ce = cudaStreamEndCapture(cap, &graph);
                if (rc != TW_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
                if (ce != cudaSuccess || !graph) {
                    ctx->set_error(TW_E_CUDA, std::string("decode graph capture failed: ") + cudaGetErrorString(ce));
                    return TW_E_CUDA;
                }
                exec_kernels = ctx->launches - l0;
                ctx->launches = l0;                       // nothing ran during capture
                ce = cudaGraphInstantiate(&exec, graph, 0);
                cudaGraphDestroy(graph);
                if (ce != cudaSuccess) {
                    ctx->set_error(TW_E_CUDA, std::string("cudaGraphInstantiate failed: ") + cudaGetErrorString(ce));
                    return TW_E_CUDA;
                }
                m->graphs[key] = GraphEntry{exec, exec_kernels};
            }
        }
        if (exec) {
            TW_CUDA_OK(ctx, cudaGraphLaunch(exec, st));
            ctx->launches += exec_kernels;
        } else {
            const bool tapped = taps.layer && pos >= taps.pos0 && pos < taps.pos0 + taps.n_pos;
            io.layer_tap = tapped ? taps.layer + (size_t)(pos - taps.pos0) * (m->desc.dec_layers + 1) * B * m->desc.d_model : nullptr;
            TW_CHECK(launch_step<T>(m, B, R, S, io, st, pos == 0 && m->pick_now, pos == m->trace_pos));
        }
        ++steps_done;
        const int g = pos - (P - 1);
        // early exit when every row has emitted EOS: the count is copied back every 8 tokens and read 8
        // tokens later, so the launch queue never drains (random-init models never emit EOS)
        if (g >= 0 && (g & 7) == 7) {
            bool all_done = false;
            if (check_pending) {
                TW_CUDA_OK(ctx, cudaEventSynchronize(m->ev[5]));
                all_done = (*h_unfinished <= 0);
            }
            if (!all_done) {
                TW_CUDA_OK(ctx, cudaMemcpyAsync(h_unfinished, S.n_unfinished, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
                TW_CUDA_OK(ctx, cudaEventRecord(m->ev[5], st));
                check_pending = true;
            }
            if (all_done) {
                if (g + 1 < n_gen_max) {
                    fill_pad_kernel<<<ceil_div(B * (n_gen_max - g - 1), 256), 256, 0, st>>>(io.out_tokens, B, n_gen_max, g + 1, R.pad);
                    ctx->launches += 1;
                }
                break;
            }
        }
    }
    if (want_graph && out_tokens != m->d_out_tok) {
        TW_CUDA_OK(ctx, cudaMemcpyAsync(out_tokens, m->d_out_tok, (size_t)B * n_gen_max * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        TW_CUDA_OK(ctx, cudaMemcpyAsync(out_lengths, m->d_out_len, B * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    }
    if (!m->trace.empty()) {
        cudaStreamSynchronize(st);
        fprintf(stderr, "[twb200 trace] position %d, B=%d (us since the embed kernel finished)\n", m->trace_pos, B);
        for (size_t i = 1; i < m->trace.size(); ++i) {
            float ms = 0.0f;
            cudaEventElapsedTime(&ms, m->trace[0].first, m->trace[i].first);
            fprintf(stderr, "[twb200 trace] %9.1f us  %s\n", ms * 1000.0f, m->trace[i].second.c_str());
        }
        for (auto& t : m->trace) cudaEventDestroy(t.first);
        m->trace.clear();
    }
    TW_CUDA_OK(ctx, cudaGetLastError());
    return TW_OK;
}

// <|startoftranscript|> of the multilingual Whisper vocabularies (51865 and 51866 ids), the token detection feeds
constexpr int WHISPER_SOT = 50258;

bool check_model(tw_model* m, const char* fn) {
    return m && m->ctx && fn;
}

// The absorbed cross-attention (absorb.cu) serves the bf16 tensor-core path at decode batches the skinny GEMMs take (<= 64 clips);
// TWB200_ABSORB=0 keeps the per-layer K|V store (A/B knob).  Larger batches and the fp32 check mode stream the K|V store.
bool use_absorb(const tw_model* m, int B) {
    const char* e = getenv("TWB200_ABSORB");       // read per call: tests switch it between decode calls
    const bool env_on = e && strcmp(e, "1") == 0;  // opt-in: measured slower than the K|V stream (profiles/r02_absorbed_attention.md)
    return env_on && m->absorb_ok && m->use_tc && m->use_tc_skinny && B <= 64;
}

// cross-attention K|V of every decoder layer (once per window) — not needed when the decode reads the encoder output directly
int cross_kv_for_decode(tw_model* m, const void* enc_out, int B, cudaStream_t st) {
    m->cur_enc = enc_out;
    m->absorb_now = use_absorb(m, B);
    if (m->absorb_now) return TW_OK;
    return m->desc.dtype == TW_BF16 ? cross_kv_impl<__nv_bfloat16>(m, enc_out, B, st) : cross_kv_impl<float>(m, enc_out, B, st);
}

}  // namespace

// =============================================================================================
// C ABI
extern "C" {

int tw_abi_version(void) { return TWB200_ABI_VERSION; }

int tw_ctx_create(int device, tw_ctx** out) {
    if (!out) return TW_E_INVALID;
    *out = nullptr;
    tw_ctx* ctx = new (std::nothrow) tw_ctx();
    if (!ctx) return TW_E_NOMEM;
    ctx->device = device;
    *out = ctx;        // returned even on failure so that tw_last_error can be read
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        ctx->set_error(TW_E_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e) +
                                      " (libtwb200 has no CPU fallback)");
        return TW_E_CUDA;
    }
    TW_CUDA_OK(ctx, cudaSetDevice(device));
    cudaDeviceProp prop;
    TW_CUDA_OK(ctx, cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        ctx->set_error(TW_E_UNSUPPORTED, "libtwb200 is built for sm_100a (B200) only; found sm_" + std::to_string(prop.major) +
                                             std::to_string(prop.minor));
        return TW_E_UNSUPPORTED;
    }
    ctx->sm_count = prop.multiProcessorCount;
    if (getenv("TWB200_SM_LIMIT")) ctx->sm_count = atoi(getenv("TWB200_SM_LIMIT"));       // experiment: persistent grids on fewer SMs
    TW_CHECK(logmel_init(ctx));
    TW_CHECK(gemm_tc_init(ctx));
    TW_CHECK(gemm_tc_skinny_init(ctx));
    TW_CHECK(absorbed_attention_init(ctx));
    return TW_OK;
}

void tw_ctx_destroy(tw_ctx* ctx) {
    if (!ctx) return;
    logmel_destroy(ctx);
    delete ctx;
}

const char* tw_last_error(const tw_ctx* ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }
uint64_t tw_launch_count(const tw_ctx* ctx) { return ctx ? ctx->launches : 0; }

int tw_logmel(tw_ctx* ctx, const void* pcm, int pcm_dtype, int64_t pcm_stride, const int32_t* n_valid, int B, int n_mel, float* out,
              void* stream) {
    if (!ctx) return TW_E_INVALID;
    if (B < 0) { ctx->set_error(TW_E_INVALID, "tw_logmel: B < 0"); return TW_E_INVALID; }
    return logmel_run(ctx, pcm, pcm_dtype, pcm_stride, n_valid, B, n_mel, out, (cudaStream_t)stream);
}

int tw_model_load(tw_ctx* ctx, const tw_model_desc* desc, const tw_weight* table, size_t n, tw_model** out) {
    if (!ctx || !desc || !table || !out) return TW_E_INVALID;
    *out = nullptr;
    const tw_model_desc& D = *desc;
    if (D.d_model <= 0 || D.heads <= 0 || D.d_model != D.heads * 64 || D.d_model > 1280 || D.d_model % 8 != 0) {
        ctx->set_error(TW_E_INVALID, "tw_model_load: d_model must be heads*64 and <= 1280");
        return TW_E_INVALID;
    }
    if ((D.n_mel != 80 && D.n_mel != 128) || D.ffn <= 0 || D.ffn % 8 != 0 || D.enc_layers <= 0 || D.dec_layers <= 0 || D.vocab <= 0 ||
        D.max_target <= 1 || D.max_batch <= 0 || D.max_batch > 4096 || (D.dtype != TW_BF16 && D.dtype != TW_F32)) {
        ctx->set_error(TW_E_INVALID, "tw_model_load: bad model descriptor");
        return TW_E_INVALID;
    }
    tw_model* m = new (std::nothrow) tw_model();
    if (!m) return TW_E_NOMEM;
    m->ctx = ctx;
    m->desc = D;
    m->esz = D.dtype == TW_BF16 ? 2 : 4;
    const char* g = getenv("TWB200_GEMM");
    m->use_tc = (D.dtype == TW_BF16) && !(g && strcmp(g, "simt") == 0);
    const char* ga = getenv("TWB200_ATTN");
    m->use_tc_attn = (D.dtype == TW_BF16) && !(ga && strcmp(ga, "simt") == 0);
    const char* gg = getenv("TWB200_GRAPH");
    m->use_graph = !(gg && strcmp(gg, "0") == 0);
    const char* g3 = getenv("TWB200_TC_SKINNY");
    m->use_tc_skinny = !(g3 && strcmp(g3, "0") == 0);
    const char* gp = getenv("TWB200_PDL");
    m->use_pdl = !(gp && strcmp(gp, "0") == 0);
    const char* gtr = getenv("TWB200_TRACE");
    m->trace_pos = gtr ? atoi(gtr) : -1;
    m->skip_mask = getenv("TWB200_SKIP") ? atoi(getenv("TWB200_SKIP")) : 0;
    m->absorb_ok = (D.dtype == TW_BF16) && absorbed_attention_supported(D.heads, D.d_model);
    WeightTable wt;
    for (size_t i = 0; i < n; ++i)
        if (table[i].name) wt.by_name[table[i].name] = &table[i];
    int r = (D.dtype == TW_BF16) ? load_weights<__nv_bfloat16>(m, wt) : load_weights<float>(m, wt);
    if (r == TW_OK) r = alloc_workspace(m);
    if (r != TW_OK) {
        tw_model_free(m);
        return r;
    }
    *out = m;
    return TW_OK;
}

namespace { void pipeline_drop_partitions(tw_model* m); }

void tw_model_free(tw_model* m) {
    if (!m) return;
    for (void* p : m->allocs) cudaFree(p);
    if (m->h_flag) cudaFreeHost(m->h_flag);
    if (m->h_step) cudaFreeHost(m->h_step);
    if (m->h_page_table) cudaFreeHost(m->h_page_table);
    for (auto& kv : m->graphs) cudaGraphExecDestroy(kv.second.exec);
    if (m->cap_stream) cudaStreamDestroy(m->cap_stream);
    if (m->pipe.on) {
        cudaDeviceSynchronize();
        for (int i = 0; i < 2; ++i) {
            if (m->pipe.enc_done[i]) cudaEventDestroy(m->pipe.enc_done[i]);
            if (m->pipe.dec_done[i]) cudaEventDestroy(m->pipe.dec_done[i]);
            for (cudaEvent_t e : {m->pipe.enc_t0[i], m->pipe.enc_t1[i], m->pipe.dec_t0[i], m->pipe.dec_t1[i]})
                if (e) cudaEventDestroy(e);
        }
        pipeline_drop_partitions(m);
    }
    for (auto& ev : m->ev)
        if (ev) cudaEventDestroy(ev);
    for (auto& ev : m->prof_ev) cudaEventDestroy(ev);
    delete m;
}

size_t tw_model_bytes(const tw_model* m) { return m ? m->bytes : 0; }

int tw_model_get_desc(const tw_model* m, tw_model_desc* out) {
    if (!m || !out) return TW_E_INVALID;
    *out = m->desc;
    return TW_OK;
}

size_t tw_workspace_bytes(const tw_model_desc* desc) {
    // Device bytes tw_model_load will allocate for this descriptor (repacked weights + workspace + K|V stores), without
    // touching a device: the same expressions as load_weights / alloc_workspace (a -m gpu test pins the two together).
    if (!desc) return 0;
    const tw_model_desc& D = *desc;
    if (D.d_model <= 0 || D.ffn <= 0 || D.enc_layers <= 0 || D.dec_layers <= 0 || D.vocab <= 0 || D.max_batch <= 0 || D.max_target <= 0 ||
        (D.dtype != TW_BF16 && D.dtype != TW_F32))
        return 0;
    const size_t e = D.dtype == TW_BF16 ? 2 : 4, f4 = sizeof(float);
    const size_t d = D.d_model, ffn = D.ffn, V = D.vocab, B = D.max_batch, M = B * TW_N_CTX, dd = d * d;
    auto al = [](size_t b) { return b == 0 ? (size_t)16 : b; };      // dev_alloc never asks for 0 bytes
    const size_t ln = 2 * al(d * f4);
    const size_t attn_self = al(3 * dd * e) + al(3 * d * f4) + al(dd * e) + al(d * f4);
    const bool absorb = D.dtype == TW_BF16 && absorbed_attention_supported(D.heads, D.d_model);
    const size_t attn_cross = al(dd * e) + al(d * f4) + al(2 * dd * e) + al(2 * d * f4) + al(dd * e) + al(d * f4) + (absorb ? al(dd * e) : 0);
    const size_t mlp = al(ffn * d * e) + al(ffn * f4) + al(ffn * d * e) + al(d * f4);
    size_t w = al(d * 3 * D.n_mel * e) + al(d * 3 * d * e) + 2 * al(d * f4) + al((size_t)TW_N_CTX * d * f4);
    w += (size_t)D.enc_layers * (ln + attn_self + ln + mlp) + ln;
    w += al(V * d * e) + al((size_t)D.max_target * d * e);
    w += (size_t)D.dec_layers * (ln + attn_self + ln + attn_cross + ln + mlp) + ln;
    const size_t kv_pages = (D.max_target + TW_KV_PAGE - 1) / TW_KV_PAGE;
    size_t ws = al(B * TW_N_SAMPLES * sizeof(int16_t)) + al(B * sizeof(int32_t)) + al(B * D.n_mel * TW_N_FRAMES * f4) +
                al(B * TW_N_FRAMES * 3 * D.n_mel * e) + al(B * TW_N_FRAMES * d * e) + al(M * 3 * d * e) + al(M * d * f4) +
                al(M * d * e) + al(M * d * e) + al(M * ffn * e) + al(M * d * e) + al((size_t)D.dec_layers * M * 2 * d * e) +
                al((size_t)D.dec_layers * B * kv_pages * TW_KV_PAGE * 2 * d * e) + al(B * kv_pages * sizeof(int32_t)) +
                al(B * d * f4) + al(B * d * e) + al(B * 3 * d * e) + al(B * d * e) + al(B * d * e) + al(B * ffn * e) + al(B * ((V + 3) / 4 * 4) * f4) +
                al(decode_attention_partial_floats((int)B, D.heads) * f4) + al((8 * B + 8) * sizeof(int32_t)) + al(V + 16) + al(V + 16) +
                al(4096 * sizeof(int32_t)) + al(B * D.max_target * sizeof(int32_t)) + al(B * sizeof(int32_t)) + al(STEP_INTS * sizeof(int32_t)) +
                al((B * PROMPT_MAX + MAX_LANG_IDS) * sizeof(int32_t)) + al(B * sizeof(int32_t));
    if (absorb) {
        const size_t Bd = B < 64 ? B : 64;
        ws += al((Bd * D.heads + ABSORB_QT_PAD) * d * e) + al(Bd * D.heads * d * e) +
              al(absorbed_attention_partial_floats((int)Bd, D.heads, (int)d) * f4);
    }
    return w + ws;
}

int tw_encode(tw_model* m, const float* mel, int B, void* enc_out, int tap_layer, float* tap_out, void* stream) {
    if (!check_model(m, "tw_encode")) return TW_E_INVALID;
    if (B <= 0 || B > m->desc.max_batch || !mel || !enc_out) {
        m->ctx->set_error(TW_E_INVALID, "tw_encode: bad batch (1..max_batch) or null buffer");
        return TW_E_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    return m->desc.dtype == TW_BF16 ? encode_impl<__nv_bfloat16>(m, mel, B, enc_out, tap_layer, tap_out, st)
                                    : encode_impl<float>(m, mel, B, enc_out, tap_layer, tap_out, st);
}

// per-row prompts: host [B][P] ids, PROMPT_DETECT allowed at index 1 (then lang_ids are needed), the same SOT in every row
static int check_prompt_rows(tw_model* m, int B, const tw_prompt_rows& rows, int P) {
    tw_ctx* ctx = m->ctx;
    const int V = m->desc.vocab;
    if (!rows.prompts || P < 1 || P > PROMPT_MAX) {
        ctx->set_error(TW_E_INVALID, "decode: null prompt, or a prompt that is empty or longer than 24 tokens");
        return TW_E_INVALID;
    }
    bool detect = false;
    for (int b = 0; b < B; ++b)
        for (int i = 0; i < P; ++i) {
            const int t = rows.prompts[(size_t)b * P + i];
            if (i == 1 && t == PROMPT_DETECT) { detect = true; continue; }
            if (t < 0 || t >= V) {
                ctx->set_error(TW_E_INVALID, "decode: prompt token out of range");
                return TW_E_INVALID;
            }
            if (i == 0 && t != rows.prompts[0]) {
                ctx->set_error(TW_E_INVALID, "decode: every row's prompt must start with the same token (SOT)");
                return TW_E_INVALID;
            }
        }
    if (rows.lang_ids || detect) {
        if (!rows.lang_ids || rows.n_lang < 1 || rows.n_lang > MAX_LANG_IDS) {
            ctx->set_error(TW_E_INVALID, "decode: language detection needs 1 .. 128 language ids");
            return TW_E_INVALID;
        }
        for (int j = 0; j < rows.n_lang; ++j)
            if (rows.lang_ids[j] < 0 || rows.lang_ids[j] >= V) {
                ctx->set_error(TW_E_INVALID, "decode: language id out of range");
                return TW_E_INVALID;
            }
    }
    if (rows.out_lang && P < 2) {
        ctx->set_error(TW_E_INVALID, "decode: out_lang needs a prompt with a language slot (P >= 2)");
        return TW_E_INVALID;
    }
    return TW_OK;
}

static int check_decode_args(tw_model* m, int B, const tw_prompt_rows& rows, int P, const tw_rules* rules, int max_length) {
    tw_ctx* ctx = m->ctx;
    if (B <= 0 || B > m->desc.max_batch || !rules) {
        ctx->set_error(TW_E_INVALID, "decode: bad batch or null argument");
        return TW_E_INVALID;
    }
    if (P < 1 || max_length <= P || max_length > m->desc.max_target) {
        // HF raises ValueError when prompt + new tokens exceed max_target_positions (generation_whisper.py:1922-1931)
        ctx->set_error(TW_E_INVALID, "decode: need 1 <= P < max_length <= max_target_positions (" +
                                         std::to_string(m->desc.max_target) + ")");
        return TW_E_INVALID;
    }
    return check_prompt_rows(m, B, rows, P);
}

// the single prompt of the original entry points, given to every row
struct BroadcastPrompt {
    std::vector<int32_t> ids;
    tw_prompt_rows rows{};
    BroadcastPrompt(const tw_model* m, const int32_t* prompt, int P, int B) {
        if (m && prompt && P > 0 && P <= PROMPT_MAX && B > 0 && B <= m->desc.max_batch) {     // else the argument checks reject the call
            ids.resize((size_t)B * P);
            for (int b = 0; b < B; ++b) std::copy(prompt, prompt + P, ids.begin() + (size_t)b * P);
            rows.prompts = ids.data();
        }
    }
};

// tw_decode_greedy after its argument checks; tw_debug_decode_taps adds residual taps
static int decode_greedy_call(tw_model* m, const void* enc_out, int B, const tw_prompt_rows& rows, int P, const tw_rules* rules, int max_length,
                              int32_t* out_tokens, int32_t* out_lengths, const int32_t* forced, float* logits_tap, int tap_steps,
                              cudaStream_t st, const DecodeTaps& taps) {
    RulesDev R;
    TW_CHECK(upload_rules(m, rules, &R, st));
    cudaEventRecord(m->ev[2], st);
    int r = cross_kv_for_decode(m, enc_out, B, st);
    if (r != TW_OK) return r;
    cudaEventRecord(m->ev[3], st);
    r = m->desc.dtype == TW_BF16
            ? decode_impl<__nv_bfloat16>(m, B, rows, P, R, max_length, out_tokens, out_lengths, forced, logits_tap, tap_steps, st, taps)
            : decode_impl<float>(m, B, rows, P, R, max_length, out_tokens, out_lengths, forced, logits_tap, tap_steps, st, taps);
    cudaEventRecord(m->ev[4], st);
    m->ev_valid[2] = m->ev_valid[3] = m->ev_valid[4] = true;
    m->ev_valid[0] = m->ev_valid[1] = m->ev_valid[6] = m->ev_valid[7] = false;
    return r;
}

int tw_decode_greedy_rows(tw_model* m, const void* enc_out, int B, const tw_prompt_rows* rows, int P, const tw_rules* rules,
                          int max_length, int32_t* out_tokens, int32_t* out_lengths, const int32_t* forced, float* logits_tap,
                          int tap_steps, void* stream) {
    if (!check_model(m, "tw_decode_greedy")) return TW_E_INVALID;
    if (!rows) {
        m->ctx->set_error(TW_E_INVALID, "tw_decode_greedy_rows: null rows");
        return TW_E_INVALID;
    }
    TW_CHECK(check_decode_args(m, B, *rows, P, rules, max_length));
    if (!enc_out || !out_tokens || !out_lengths) {
        m->ctx->set_error(TW_E_INVALID, "tw_decode_greedy: null buffer");
        return TW_E_INVALID;
    }
    return decode_greedy_call(m, enc_out, B, *rows, P, rules, max_length, out_tokens, out_lengths, forced, logits_tap, tap_steps,
                              (cudaStream_t)stream, DecodeTaps{});
}

int tw_decode_greedy(tw_model* m, const void* enc_out, int B, const int32_t* prompt, int P, const tw_rules* rules, int max_length,
                     int32_t* out_tokens, int32_t* out_lengths, const int32_t* forced, float* logits_tap, int tap_steps,
                     void* stream) {
    BroadcastPrompt bp(m, prompt, P, B);
    return tw_decode_greedy_rows(m, enc_out, B, &bp.rows, P, rules, max_length, out_tokens, out_lengths, forced, logits_tap, tap_steps,
                                 stream);
}

int tw_detect_language(tw_model* m, const void* enc_out, int B, const int32_t* lang_ids, int n_lang, int32_t* out_lang, void* stream) {
    if (!check_model(m, "tw_detect_language")) return TW_E_INVALID;
    tw_ctx* ctx = m->ctx;
    if (B <= 0 || B > m->desc.max_batch || !enc_out || !out_lang) {
        ctx->set_error(TW_E_INVALID, "tw_detect_language: bad batch (1..max_batch) or null buffer");
        return TW_E_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    // step 0 of a decode whose every row detects: prompt [SOT, detect], max_length 2 (one step, nothing generated, no graph)
    std::vector<int32_t> prompts((size_t)B * 2);
    for (int b = 0; b < B; ++b) { prompts[2 * b] = WHISPER_SOT; prompts[2 * b + 1] = PROMPT_DETECT; }
    tw_prompt_rows rows{prompts.data(), lang_ids, n_lang, out_lang};
    TW_CHECK(check_prompt_rows(m, B, rows, 2));
    TW_CHECK(cross_kv_for_decode(m, enc_out, B, st));
    RulesDev R{m->d_suppress, m->d_begin_suppress, -1, -1, -1, -1, -1};     // no token is selected
    int r = m->desc.dtype == TW_BF16 ? decode_impl<__nv_bfloat16>(m, B, rows, 2, R, 2, m->d_out_tok, m->d_out_len, nullptr, nullptr, 0, st)
                                     : decode_impl<float>(m, B, rows, 2, R, 2, m->d_out_tok, m->d_out_len, nullptr, nullptr, 0, st);
    if (r == TW_OK) TW_CUDA_OK(ctx, cudaGetLastError());
    return r;
}

int tw_debug_decode_taps(tw_model* m, const void* enc_out, int B, const int32_t* prompt, int P, const tw_rules* rules, int max_length,
                         int32_t* out_tokens, int32_t* out_lengths, const int32_t* forced, float* logits_tap, int tap_steps,
                         float* layer_tap, int pos0, int n_pos, void* self_kv_out, int n_sms, void* stream) {
    if (!check_model(m, "tw_debug_decode_taps")) return TW_E_INVALID;
    BroadcastPrompt bp(m, prompt, P, B);
    TW_CHECK(check_decode_args(m, B, bp.rows, P, rules, max_length));
    tw_ctx* ctx = m->ctx;
    if (!enc_out || !out_tokens || !out_lengths || (layer_tap && (pos0 < 0 || n_pos < 0 || pos0 + n_pos > max_length - 1)) || n_sms < 0) {
        ctx->set_error(TW_E_INVALID, "tw_debug_decode_taps: null buffer, tapped positions outside 0 .. max_length - 2 or n_sms < 0");
        return TW_E_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    DecodeTaps taps;
    taps.layer = layer_tap;
    taps.pos0 = pos0;
    taps.n_pos = layer_tap ? n_pos : 0;
    // every launch sized for a partition of n_sms SMs, as the pipeline's decode stage sizes them
    const int sms_before = ctx->sm_count;
    const int da_before = decode_attention_set_sms(n_sms);
    if (n_sms > 0) ctx->sm_count = n_sms;
    int r = decode_greedy_call(m, enc_out, B, bp.rows, P, rules, max_length, out_tokens, out_lengths, forced, logits_tap, tap_steps, st, taps);
    decode_attention_set_sms(da_before);
    ctx->sm_count = sms_before;
    if (r != TW_OK || !self_kv_out) return r;
    // the self-attention K|V rows of positions 0 .. max_length - 2, read through the page table this call wrote
    const tw_model_desc& D = m->desc;
    const size_t e = m->esz, row = 2 * (size_t)D.d_model * e, n_rows = max_length - 1;
    const size_t self_layer = (size_t)D.max_batch * m->kv_pages * TW_KV_PAGE * row;
    for (int l = 0; l < D.dec_layers; ++l)
        for (int b = 0; b < B; ++b)
            for (size_t p0 = 0; p0 < n_rows; p0 += TW_KV_PAGE) {
                const int page = m->h_page_table[b * m->kv_pages + p0 / TW_KV_PAGE];
                const size_t rows = n_rows - p0 < (size_t)TW_KV_PAGE ? n_rows - p0 : (size_t)TW_KV_PAGE;
                const char* src = (const char*)m->self_kv + l * self_layer + (size_t)page * TW_KV_PAGE * row;
                char* dst = (char*)self_kv_out + (((size_t)l * B + b) * n_rows + p0) * row;
                TW_CUDA_OK(ctx, cudaMemcpyAsync(dst, src, rows * row, cudaMemcpyDeviceToDevice, st));
            }
    return TW_OK;
}

// tw_decoder_logits with an optional residual tap (tw_debug_decoder_logits_taps)
static int decoder_logits_call(tw_model* m, const void* enc_out, int B, const int32_t* decoder_input_ids, int T, float* logits,
                               int64_t ld_logits, cudaStream_t st, float* tap) {
    if (!check_model(m, "tw_decoder_logits")) return TW_E_INVALID;
    tw_ctx* ctx = m->ctx;
    if (B <= 0 || B > m->desc.max_batch || !enc_out || !decoder_input_ids || !logits) {
        ctx->set_error(TW_E_INVALID, "tw_decoder_logits: bad batch (1..max_batch) or null buffer");
        return TW_E_INVALID;
    }
    if (T < 1 || T > m->desc.max_target) {
        // HF: the decoder has max_target_positions learned positions (modeling_whisper.py:719-745)
        ctx->set_error(TW_E_INVALID, "tw_decoder_logits: need 1 <= T <= max_target_positions (" + std::to_string(m->desc.max_target) + ")");
        return TW_E_INVALID;
    }
    if (ld_logits < m->desc.vocab || ((ld_logits * 4) % 16) || (reinterpret_cast<uintptr_t>(logits) & 15)) {
        ctx->set_error(TW_E_INVALID, "tw_decoder_logits: logits need a 16-byte aligned base and a row pitch >= vocab that is a multiple of 4 floats");
        return TW_E_INVALID;
    }
    int r = m->desc.dtype == TW_BF16 ? cross_kv_impl<__nv_bfloat16>(m, enc_out, B, st) : cross_kv_impl<float>(m, enc_out, B, st);
    if (r != TW_OK) return r;
    return m->desc.dtype == TW_BF16 ? decoder_logits_impl<__nv_bfloat16>(m, B, decoder_input_ids, T, logits, ld_logits, st, tap)
                                    : decoder_logits_impl<float>(m, B, decoder_input_ids, T, logits, ld_logits, st, tap);
}

int tw_decoder_logits(tw_model* m, const void* enc_out, int B, const int32_t* decoder_input_ids, int T, float* logits,
                      int64_t ld_logits, void* stream) {
    return decoder_logits_call(m, enc_out, B, decoder_input_ids, T, logits, ld_logits, (cudaStream_t)stream, nullptr);
}

int tw_debug_decoder_logits_taps(tw_model* m, const void* enc_out, int B, const int32_t* decoder_input_ids, int T, float* logits,
                                 int64_t ld_logits, float* tap, void* stream) {
    if (m && !tap) {
        m->ctx->set_error(TW_E_INVALID, "tw_debug_decoder_logits_taps: null tap");
        return TW_E_INVALID;
    }
    return decoder_logits_call(m, enc_out, B, decoder_input_ids, T, logits, ld_logits, (cudaStream_t)stream, tap);
}

int tw_transcribe_host(tw_model* m, const int16_t* pcm_host, const int32_t* n_valid_host, int B, const int32_t* prompt, int P,
                       const tw_rules* rules, int max_length, int32_t* out_tokens_host, int32_t* out_lengths_host, void* stream) {
    BroadcastPrompt bp(m, prompt, P, B);
    return tw_transcribe_host_rows(m, pcm_host, n_valid_host, B, &bp.rows, P, rules, max_length, out_tokens_host, out_lengths_host, stream);
}

int tw_transcribe_host_rows(tw_model* m, const int16_t* pcm_host, const int32_t* n_valid_host, int B, const tw_prompt_rows* rows_host,
                            int P, const tw_rules* rules, int max_length, int32_t* out_tokens_host, int32_t* out_lengths_host, void* stream) {
    if (!check_model(m, "tw_transcribe_host")) return TW_E_INVALID;
    if (!rows_host) {
        m->ctx->set_error(TW_E_INVALID, "tw_transcribe_host_rows: null rows");
        return TW_E_INVALID;
    }
    TW_CHECK(check_decode_args(m, B, *rows_host, P, rules, max_length));
    tw_prompt_rows rows = *rows_host;
    rows.out_lang = rows_host->out_lang ? m->d_out_lang : nullptr;      // decoded on the device, copied to the host buffer below
    if (!pcm_host || !out_tokens_host || !out_lengths_host) {
        m->ctx->set_error(TW_E_INVALID, "tw_transcribe_host: null buffer");
        return TW_E_INVALID;
    }
    tw_ctx* ctx = m->ctx;
    cudaStream_t st = (cudaStream_t)stream;
    const tw_model_desc& D = m->desc;
    const int n_gen = max_length - P;
    RulesDev R;
    TW_CHECK(upload_rules(m, rules, &R, st));
    cudaEventRecord(m->ev[6], st);
    TW_CUDA_OK(ctx, cudaMemcpyAsync(m->ws_pcm, pcm_host, (size_t)B * TW_N_SAMPLES * sizeof(int16_t), cudaMemcpyHostToDevice, st));
    const int32_t* nv = nullptr;
    if (n_valid_host) {
        TW_CUDA_OK(ctx, cudaMemcpyAsync(m->ws_nvalid, n_valid_host, B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        nv = m->ws_nvalid;
    }
    cudaEventRecord(m->ev[0], st);
    // the per-clip floor and scaling of the log-mel (its second pass) ride in the conv-stem im2col
    const float* clip_max = nullptr;
    TW_CHECK(logmel_run(ctx, m->ws_pcm, TW_I16, TW_N_SAMPLES, nv, B, D.n_mel, m->ws_mel, st, false, &clip_max));
    cudaEventRecord(m->ev[1], st);
    int r = D.dtype == TW_BF16 ? encode_impl<__nv_bfloat16>(m, m->ws_mel, B, m->ws_enc, -1, nullptr, st, clip_max)
                               : encode_impl<float>(m, m->ws_mel, B, m->ws_enc, -1, nullptr, st, clip_max);
    if (r != TW_OK) return r;
    cudaEventRecord(m->ev[2], st);
    r = cross_kv_for_decode(m, m->ws_enc, B, st);
    if (r != TW_OK) return r;
    cudaEventRecord(m->ev[3], st);
    r = D.dtype == TW_BF16
            ? decode_impl<__nv_bfloat16>(m, B, rows, P, R, max_length, m->d_out_tok, m->d_out_len, nullptr, nullptr, 0, st)
            : decode_impl<float>(m, B, rows, P, R, max_length, m->d_out_tok, m->d_out_len, nullptr, nullptr, 0, st);
    if (r != TW_OK) return r;
    TW_CUDA_OK(ctx, cudaMemcpyAsync(out_tokens_host, m->d_out_tok, (size_t)B * n_gen * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    TW_CUDA_OK(ctx, cudaMemcpyAsync(out_lengths_host, m->d_out_len, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (rows.out_lang)
        TW_CUDA_OK(ctx, cudaMemcpyAsync(rows_host->out_lang, m->d_out_lang, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    cudaEventRecord(m->ev[4], st);
    TW_CUDA_OK(ctx, cudaStreamSynchronize(st));
    for (int i = 0; i < 5; ++i) m->ev_valid[i] = true;
    m->ev_valid[6] = true;
    m->ev_valid[7] = false;
    return TW_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Pipeline over SM partitions
namespace {
typedef CUresult (*PfnGetDevResource)(CUdevice, CUdevResource*, CUdevResourceType);
typedef CUresult (*PfnSmSplit)(CUdevResource*, unsigned int*, const CUdevResource*, CUdevResource*, unsigned int, unsigned int);
typedef CUresult (*PfnGenDesc)(CUdevResourceDesc*, CUdevResource*, unsigned int);
typedef CUresult (*PfnGreenCreate)(CUgreenCtx*, CUdevResourceDesc, CUdevice, unsigned int);
typedef CUresult (*PfnGreenStream)(CUstream*, CUgreenCtx, unsigned int, int);
void* driver_entry(const char* name) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint(name, &fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) return nullptr;
    return fn;
}
// every persistent grid of the library is sized from these two numbers
void set_active_sms(tw_model* m, int n) {
    m->ctx->sm_count = n;
    decode_attention_set_sms(n);
}
}  // namespace

namespace {
// SM partitions of the pipeline: two green contexts (n_enc_sms SMs / the rest) and their streams
int pipeline_make_partitions(tw_model* m, int n_enc_sms) {
    tw_ctx* ctx = m->ctx;
    auto pGetRes = reinterpret_cast<PfnGetDevResource>(driver_entry("cuDeviceGetDevResource"));
    auto pSplit = reinterpret_cast<PfnSmSplit>(driver_entry("cuDevSmResourceSplitByCount"));
    auto pDesc = reinterpret_cast<PfnGenDesc>(driver_entry("cuDevResourceGenerateDesc"));
    auto pCreate = reinterpret_cast<PfnGreenCreate>(driver_entry("cuGreenCtxCreate"));
    auto pStream = reinterpret_cast<PfnGreenStream>(driver_entry("cuGreenCtxStreamCreate"));
    if (!pGetRes || !pSplit || !pDesc || !pCreate || !pStream) {
        ctx->set_error(TW_E_UNSUPPORTED, "tw_pipeline_enable: this driver has no green contexts (SM partitions)");
        return TW_E_UNSUPPORTED;
    }
    auto& P = m->pipe;
    CUdevResource all, small, rest;
    auto fail = [&](const char* what, CUresult r) {
        ctx->set_error(TW_E_CUDA, std::string("tw_pipeline_enable: ") + what + " failed (" + std::to_string((int)r) + ")");
        return TW_E_CUDA;
    };
    CUresult r = pGetRes((CUdevice)ctx->device, &all, CU_DEV_RESOURCE_TYPE_SM);
    if (r != CUDA_SUCCESS) return fail("cuDeviceGetDevResource", r);
    P.n_dev = (int)all.sm.smCount;
    if (n_enc_sms < 8 || n_enc_sms > P.n_dev / 2) {
        ctx->set_error(TW_E_INVALID, "tw_pipeline_enable: the encoder partition needs between 8 SMs and half of the device");
        return TW_E_INVALID;
    }
    unsigned nb = 1;
    r = pSplit(&small, &nb, &all, &rest, 0, (unsigned)n_enc_sms);
    if (r != CUDA_SUCCESS || nb != 1) return fail("cuDevSmResourceSplitByCount", r);
    CUdevResourceDesc d_small, d_rest;
    if ((r = pDesc(&d_small, &small, 1)) != CUDA_SUCCESS || (r = pDesc(&d_rest, &rest, 1)) != CUDA_SUCCESS) return fail("cuDevResourceGenerateDesc", r);
    if ((r = pCreate(&P.g_enc, d_small, (CUdevice)ctx->device, CU_GREEN_CTX_DEFAULT_STREAM)) != CUDA_SUCCESS) return fail("cuGreenCtxCreate", r);
    if ((r = pCreate(&P.g_dec, d_rest, (CUdevice)ctx->device, CU_GREEN_CTX_DEFAULT_STREAM)) != CUDA_SUCCESS) return fail("cuGreenCtxCreate", r);
    CUstream se, sd, sc;
    if ((r = pStream(&se, P.g_enc, CU_STREAM_NON_BLOCKING, 0)) != CUDA_SUCCESS || (r = pStream(&sd, P.g_dec, CU_STREAM_NON_BLOCKING, 0)) != CUDA_SUCCESS ||
        (r = pStream(&sc, P.g_dec, CU_STREAM_NON_BLOCKING, 0)) != CUDA_SUCCESS)
        return fail("cuGreenCtxStreamCreate", r);
    P.n_enc = (int)small.sm.smCount;
    P.n_dec = (int)rest.sm.smCount;
    P.s_enc = (cudaStream_t)se;
    P.s_dec = (cudaStream_t)sd;
    P.s_cap = (cudaStream_t)sc;
    return TW_OK;
}
void pipeline_drop_partitions(tw_model* m) {
    auto& P = m->pipe;
    for (cudaStream_t* s : {&P.s_enc, &P.s_dec, &P.s_cap}) {
        if (*s) cudaStreamDestroy(*s);
        *s = nullptr;
    }
    if (auto destroy = reinterpret_cast<CUresult (*)(CUgreenCtx)>(driver_entry("cuGreenCtxDestroy"))) {
        if (P.g_enc) destroy(P.g_enc);
        if (P.g_dec) destroy(P.g_dec);
    }
    P.g_enc = P.g_dec = nullptr;
}
}  // namespace

int tw_pipeline_enable(tw_model* m, int n_enc_sms) {
    if (!check_model(m, "tw_pipeline_enable")) return TW_E_INVALID;
    tw_ctx* ctx = m->ctx;
    if (m->pipe.on) return TW_OK;
    auto& P = m->pipe;
    TW_CHECK(pipeline_make_partitions(m, n_enc_sms));
    // second set of the buffers the two stages hand over: encoder output and cross-attention K|V store
    const tw_model_desc& D = m->desc;
    const size_t M = (size_t)D.max_batch * TW_N_CTX, d = D.d_model, e = m->esz;
    P.enc_out[0] = m->ws_enc;
    P.xkv[0] = m->xkv;
    TW_CHECK(dev_alloc(m, &P.enc_out[1], M * d * e));
    TW_CHECK(dev_alloc(m, &P.xkv[1], (size_t)D.dec_layers * M * 2 * d * e));
    for (int i = 0; i < 2; ++i) {
        TW_CUDA_OK(ctx, cudaEventCreateWithFlags(&P.enc_done[i], cudaEventDisableTiming));
        TW_CUDA_OK(ctx, cudaEventCreateWithFlags(&P.dec_done[i], cudaEventDisableTiming));
        for (cudaEvent_t* e : {&P.enc_t0[i], &P.enc_t1[i], &P.dec_t0[i], &P.dec_t1[i]}) TW_CUDA_OK(ctx, cudaEventCreate(e));
    }
    P.on = true;
    return TW_OK;
}

int tw_pipeline_resize(tw_model* m, int n_enc_sms) {
    if (!check_model(m, "tw_pipeline_resize")) return TW_E_INVALID;
    tw_ctx* ctx = m->ctx;
    auto& P = m->pipe;
    if (!P.on) {
        ctx->set_error(TW_E_INVALID, "tw_pipeline_resize: pipeline not enabled");
        return TW_E_INVALID;
    }
    // both stages drained (a batch staged in a slot stays valid: the buffers do not move), the decode graphs captured in the
    // old decode partition dropped (a graph's kernel nodes run in the context of its capture stream)
    TW_CUDA_OK(ctx, cudaStreamSynchronize(P.s_enc));
    TW_CUDA_OK(ctx, cudaStreamSynchronize(P.s_dec));
    for (auto& kv : m->graphs) cudaGraphExecDestroy(kv.second.exec);
    m->graphs.clear();
    const int old_enc = P.n_enc;
    pipeline_drop_partitions(m);
    int r = pipeline_make_partitions(m, n_enc_sms);
    if (r != TW_OK) {
        // keep the pipeline usable: back to the previous split
        const std::string msg = ctx->err;
        pipeline_drop_partitions(m);
        if (pipeline_make_partitions(m, old_enc) != TW_OK) P.on = false;
        ctx->set_error(r, msg);
        return r;
    }
    return TW_OK;
}

int tw_pipeline_stage_ms(tw_model* m, int slot, float* stage1_ms, float* decode_ms) {
    if (!check_model(m, "tw_pipeline_stage_ms")) return TW_E_INVALID;
    auto& P = m->pipe;
    if (!P.on || slot < 0 || slot > 1) {
        m->ctx->set_error(TW_E_INVALID, "tw_pipeline_stage_ms: pipeline not enabled or bad slot");
        return TW_E_INVALID;
    }
    // never blocks: a stage that has not completed (or was never run) reads as -1
    if (stage1_ms) {
        *stage1_ms = -1.0f;
        if (P.enc_timed[slot] && cudaEventQuery(P.enc_t1[slot]) == cudaSuccess) cudaEventElapsedTime(stage1_ms, P.enc_t0[slot], P.enc_t1[slot]);
    }
    if (decode_ms) {
        *decode_ms = -1.0f;
        if (P.dec_timed[slot] && cudaEventQuery(P.dec_t1[slot]) == cudaSuccess) cudaEventElapsedTime(decode_ms, P.dec_t0[slot], P.dec_t1[slot]);
    }
    cudaGetLastError();      // cudaErrorNotReady of a query is not an error of the library
    return TW_OK;
}

int tw_pipeline_info(const tw_model* m, int* n_enc_sms, int* n_dec_sms) {
    if (!m) return TW_E_INVALID;
    if (n_enc_sms) *n_enc_sms = m->pipe.on ? m->pipe.n_enc : 0;
    if (n_dec_sms) *n_dec_sms = m->pipe.on ? m->pipe.n_dec : 0;
    return TW_OK;
}

int tw_pipeline_encode(tw_model* m, const int16_t* pcm, const int32_t* n_valid_host, int B, int slot) {
    return tw_pipeline_encode_at(m, pcm, n_valid_host, B, slot, 0);
}

int tw_pipeline_encode_at(tw_model* m, const int16_t* pcm, const int32_t* n_valid_host, int B, int slot, int clip0) {
    if (!check_model(m, "tw_pipeline_encode")) return TW_E_INVALID;
    tw_ctx* ctx = m->ctx;
    auto& P = m->pipe;
    if (!P.on || slot < 0 || slot > 1 || B <= 0 || clip0 < 0 || clip0 + B > m->desc.max_batch || !pcm) {
        ctx->set_error(TW_E_INVALID, "tw_pipeline_encode: pipeline not enabled, bad slot (0 / 1), bad batch / clip offset or null buffer");
        return TW_E_INVALID;
    }
    if (clip0 > 0 && use_absorb(m, 1)) {      // (the first part would have skipped its K|V projection)
        ctx->set_error(TW_E_UNSUPPORTED, "tw_pipeline_encode_at: merged decode batches are not available on the absorbed cross-attention path");
        return TW_E_UNSUPPORTED;
    }
    const tw_model_desc& D = m->desc;
    cudaStream_t st = P.s_enc;
    // the decode that last read this slot's encoder output / K|V store must have finished
    if (P.dec_pending[slot]) TW_CUDA_OK(ctx, cudaStreamWaitEvent(st, P.dec_done[slot], 0));
    const int sms_before = ctx->sm_count;
    set_active_sms(m, P.n_enc);
    void* const xkv_before = m->xkv;
    m->xkv = P.xkv[slot];
    int r = TW_OK;
    do {
        cudaEventRecord(m->ev[6], st);
        if (clip0 == 0) { cudaEventRecord(P.enc_t0[slot], st); P.enc_timed[slot] = false; }
        if (cudaMemcpyAsync(m->ws_pcm, pcm, (size_t)B * TW_N_SAMPLES * sizeof(int16_t), cudaMemcpyDefault, st) != cudaSuccess) { r = TW_E_CUDA; break; }
        const int32_t* nv = nullptr;
        if (n_valid_host) {
            if (cudaMemcpyAsync(m->ws_nvalid, n_valid_host, B * sizeof(int32_t), cudaMemcpyDefault, st) != cudaSuccess) { r = TW_E_CUDA; break; }
            nv = m->ws_nvalid;
        }
        cudaEventRecord(m->ev[0], st);
        const float* clip_max = nullptr;
        if ((r = logmel_run(ctx, m->ws_pcm, TW_I16, TW_N_SAMPLES, nv, B, D.n_mel, m->ws_mel, st, false, &clip_max)) != TW_OK) break;
        cudaEventRecord(m->ev[1], st);
        void* const enc_part = (char*)P.enc_out[slot] + (size_t)clip0 * TW_N_CTX * D.d_model * m->esz;
        r = D.dtype == TW_BF16 ? encode_impl<__nv_bfloat16>(m, m->ws_mel, B, enc_part, -1, nullptr, st, clip_max)
                               : encode_impl<float>(m, m->ws_mel, B, enc_part, -1, nullptr, st, clip_max);
        if (r != TW_OK) break;
        cudaEventRecord(m->ev[2], st);
        if (!use_absorb(m, B))
            r = D.dtype == TW_BF16 ? cross_kv_impl<__nv_bfloat16>(m, enc_part, B, st, clip0) : cross_kv_impl<float>(m, enc_part, B, st, clip0);
        if (r != TW_OK) break;
        cudaEventRecord(m->ev[3], st);
        if (cudaEventRecord(P.enc_done[slot], st) != cudaSuccess) { r = TW_E_CUDA; break; }
        cudaEventRecord(P.enc_t1[slot], st);
        P.enc_timed[slot] = true;
    } while (0);
    m->xkv = xkv_before;
    set_active_sms(m, sms_before);
    if (r == TW_E_CUDA && ctx->err_code != TW_E_CUDA) ctx->set_error(TW_E_CUDA, std::string("tw_pipeline_encode: ") + cudaGetErrorString(cudaGetLastError()));
    return r;
}

int tw_pipeline_decode(tw_model* m, int slot, int B, const int32_t* prompt, int P_len, const tw_rules* rules, int max_length,
                       int32_t* out_tokens_host, int32_t* out_lengths_host) {
    BroadcastPrompt bp(m, prompt, P_len, B);
    return tw_pipeline_decode_rows(m, slot, B, &bp.rows, P_len, rules, max_length, out_tokens_host, out_lengths_host);
}

int tw_pipeline_decode_rows(tw_model* m, int slot, int B, const tw_prompt_rows* rows_host, int P_len, const tw_rules* rules, int max_length,
                            int32_t* out_tokens_host, int32_t* out_lengths_host) {
    if (!check_model(m, "tw_pipeline_decode")) return TW_E_INVALID;
    if (!rows_host) {
        m->ctx->set_error(TW_E_INVALID, "tw_pipeline_decode_rows: null rows");
        return TW_E_INVALID;
    }
    TW_CHECK(check_decode_args(m, B, *rows_host, P_len, rules, max_length));
    tw_prompt_rows rows = *rows_host;
    rows.out_lang = rows_host->out_lang ? m->d_out_lang : nullptr;      // decoded on the device, copied to the host buffer below
    tw_ctx* ctx = m->ctx;
    auto& P = m->pipe;
    if (!P.on || slot < 0 || slot > 1 || !out_tokens_host || !out_lengths_host) {
        ctx->set_error(TW_E_INVALID, "tw_pipeline_decode: pipeline not enabled, bad slot (0 / 1) or null buffer");
        return TW_E_INVALID;
    }
    const tw_model_desc& D = m->desc;
    cudaStream_t st = P.s_dec;
    const int n_gen = max_length - P_len;
    RulesDev R;
    TW_CHECK(upload_rules(m, rules, &R, st));
    TW_CUDA_OK(ctx, cudaStreamWaitEvent(st, P.enc_done[slot], 0));
    const int sms_before = ctx->sm_count;
    set_active_sms(m, P.n_dec);
    void* const xkv_before = m->xkv;
    m->xkv = P.xkv[slot];
    m->cur_enc = P.enc_out[slot];
    m->absorb_now = use_absorb(m, B);
    P.in_decode = true;
    cudaEventRecord(m->ev[7], st);
    cudaEventRecord(P.dec_t0[slot], st);
    P.dec_timed[slot] = false;
    int r = D.dtype == TW_BF16
                ? decode_impl<__nv_bfloat16>(m, B, rows, P_len, R, max_length, m->d_out_tok, m->d_out_len, nullptr, nullptr, 0, st)
                : decode_impl<float>(m, B, rows, P_len, R, max_length, m->d_out_tok, m->d_out_len, nullptr, nullptr, 0, st);
    P.in_decode = false;
    m->xkv = xkv_before;
    set_active_sms(m, sms_before);
    if (r != TW_OK) return r;
    TW_CUDA_OK(ctx, cudaMemcpyAsync(out_tokens_host, m->d_out_tok, (size_t)B * n_gen * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    TW_CUDA_OK(ctx, cudaMemcpyAsync(out_lengths_host, m->d_out_len, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (rows.out_lang)
        TW_CUDA_OK(ctx, cudaMemcpyAsync(rows_host->out_lang, m->d_out_lang, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    cudaEventRecord(m->ev[4], st);
    cudaEventRecord(P.dec_t1[slot], st);
    P.dec_timed[slot] = true;
    TW_CUDA_OK(ctx, cudaEventRecord(P.dec_done[slot], st));
    P.dec_pending[slot] = true;
    TW_CUDA_OK(ctx, cudaStreamSynchronize(st));
    for (int i = 0; i < 5; ++i) m->ev_valid[i] = true;
    m->ev_valid[6] = m->ev_valid[7] = true;
    return TW_OK;
}

int tw_debug_gemm_grouped(tw_ctx* ctx, const void* A, const void* W, const float* bias, void* C, int M, int N, int K, int group_n,
                          void* stream) {
    if (!ctx || !A || !W || !C || group_n <= 0 || N % group_n) return TW_E_INVALID;
    GemmEpi e = mk_epi(EPI_STORE, bias, C, N);
    e.group_n = group_n;
    ctx->launches += 1;
    return gemm_tc_skinny(ctx, (const __nv_bfloat16*)A, (int64_t)K * (N / group_n), (const __nv_bfloat16*)W, K, M, N, K, e, (cudaStream_t)stream);
}

int tw_debug_absorbed_attention(tw_ctx* ctx, const void* qt, const void* enc, int Tk, int B, int H, void* out, const int32_t* active,
                                const int32_t* n_active, int rev, void* stream) {
    if (!ctx || !qt || !enc || !out || B <= 0 || H <= 0 || Tk <= 0) return TW_E_INVALID;
    const int d = 64 * H;
    cudaStream_t st = (cudaStream_t)stream;
    float* partial = nullptr;
    TW_CUDA_OK(ctx, cudaMalloc(&partial, absorbed_attention_partial_floats(B, H, d) * sizeof(float)));
    ctx->launches += 2;
    long long* trace = nullptr;                  // TWB200_AB_TRACE=1: pipeline timeline of CTA 0 (clock64), printed to stderr
    if (getenv("TWB200_AB_TRACE")) {
        TW_CUDA_OK(ctx, cudaMalloc(&trace, 16 * 64 * sizeof(long long)));
        TW_CUDA_OK(ctx, cudaMemset(trace, 0, 16 * 64 * sizeof(long long)));
    }
    const int r = absorbed_attention(ctx, (const __nv_bfloat16*)qt, (const __nv_bfloat16*)enc, Tk, B, H, d, partial, (__nv_bfloat16*)out, st,
                                     active, n_active, rev, nullptr, nullptr, trace);
    cudaStreamSynchronize(st);
    if (trace) {
        std::vector<long long> h(16 * 64);
        cudaMemcpy(h.data(), trace, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
        long long t0 = 0;
        for (long long v : h) if (v && (!t0 || v < t0)) t0 = v;
        for (int t = 0; t < 16; ++t) {
            fprintf(stderr, "[ab trace] tile %2d:", t);
            for (int i = 0; i < 40; ++i) if (h[t * 64 + i]) fprintf(stderr, " %d:%lld", i, h[t * 64 + i] - t0);
            fprintf(stderr, "\n");
        }
        cudaFree(trace);
    }
    cudaFree(partial);
    if (r == TW_OK) TW_CUDA_OK(ctx, cudaGetLastError());
    return r;
}

int tw_debug_gemm(tw_ctx* ctx, const void* A, const void* W, const float* bias, void* C, int M, int N, int K, int dtype, int epi_mode,
                  const float* pos, int pos_period, int use_tc, void* stream) {
    if (!ctx || !A || !W || !C) return TW_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    GemmEpi e = mk_epi(epi_mode, bias, C, N, pos, pos_period > 0 ? pos_period : 1);
    ctx->launches += 1;
    if (dtype == TW_F32) {
        gemm_simt<float>((const float*)A, K, (const float*)W, K, M, N, K, e, st);
    } else if (dtype == TW_BF16) {
        if (use_tc == 3) return gemm_tc_skinny(ctx, (const __nv_bfloat16*)A, K, (const __nv_bfloat16*)W, K, M, N, K, e, st);
        if (use_tc) return gemm_tc(ctx, (const __nv_bfloat16*)A, K, (const __nv_bfloat16*)W, K, M, N, K, e, st);
        gemm_simt<__nv_bfloat16>((const __nv_bfloat16*)A, K, (const __nv_bfloat16*)W, K, M, N, K, e, st);
    } else {
        ctx->set_error(TW_E_INVALID, "tw_debug_gemm: dtype");
        return TW_E_INVALID;
    }
    TW_CUDA_OK(ctx, cudaGetLastError());
    return TW_OK;
}

int tw_debug_layernorm(tw_ctx* ctx, const float* x, const float* gamma, const float* beta, void* out, int M, int d, int dtype,
                       void* stream) {
    if (!ctx) return TW_E_INVALID;
    if (!x || !gamma || !beta || !out || M < 0 || d <= 0 || d > 1280 || d % 4 || (dtype != TW_F32 && dtype != TW_BF16)) {
        ctx->set_error(TW_E_INVALID, "tw_debug_layernorm: need M >= 0, 0 < d <= 1280 with d % 4 == 0, dtype float32 / bfloat16 and non-null buffers");
        return TW_E_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == TW_F32) layernorm<float>(x, gamma, beta, (float*)out, M, d, st);
    else layernorm<__nv_bfloat16>(x, gamma, beta, (__nv_bfloat16*)out, M, d, st);
    ctx->launches += 1;
    TW_CUDA_OK(ctx, cudaGetLastError());
    return TW_OK;
}

int tw_debug_cross_kv(tw_model* m, const void* enc_out, int B, int clip0, void* stream) {
    if (!check_model(m, "tw_debug_cross_kv")) return TW_E_INVALID;
    if (!enc_out || B <= 0 || clip0 < 0 || clip0 + B > m->desc.max_batch) {
        m->ctx->set_error(TW_E_INVALID, "tw_debug_cross_kv: need 1 <= B, 0 <= clip0, clip0 + B <= max_batch and an encoder output");
        return TW_E_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    return m->desc.dtype == TW_BF16 ? cross_kv_impl<__nv_bfloat16>(m, enc_out, B, st, clip0) : cross_kv_impl<float>(m, enc_out, B, st, clip0);
}

int tw_debug_read_stage1(tw_model* m, int slot, int clip0, int B, void* enc_out, int layer, void* kv_out, void* stream) {
    if (!check_model(m, "tw_debug_read_stage1")) return TW_E_INVALID;
    tw_ctx* ctx = m->ctx;
    const tw_model_desc& D = m->desc;
    auto& P = m->pipe;
    if (slot < -1 || slot > 1 || (slot >= 0 && !P.on) || (slot < 0 && enc_out) || B <= 0 || clip0 < 0 || clip0 + B > D.max_batch ||
        (kv_out && (layer < 0 || layer >= D.dec_layers))) {
        ctx->set_error(TW_E_INVALID, "tw_debug_read_stage1: bad slot (-1, or 0 / 1 with the pipeline on; no encoder output for -1), clip range or layer");
        return TW_E_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t d = D.d_model, e = m->esz, rows = (size_t)B * TW_N_CTX;
    if (slot >= 0) TW_CUDA_OK(ctx, cudaStreamWaitEvent(st, P.enc_done[slot], 0));
    if (enc_out) {
        const char* src = (const char*)P.enc_out[slot] + (size_t)clip0 * TW_N_CTX * d * e;
        TW_CUDA_OK(ctx, cudaMemcpyAsync(enc_out, src, rows * d * e, cudaMemcpyDeviceToDevice, st));
    }
    if (kv_out) {
        const char* store = (const char*)(slot >= 0 ? P.xkv[slot] : m->xkv);
        const char* src = store + ((size_t)layer * D.max_batch + clip0) * TW_N_CTX * 2 * d * e;
        TW_CUDA_OK(ctx, cudaMemcpyAsync(kv_out, src, rows * 2 * d * e, cudaMemcpyDeviceToDevice, st));
    }
    return TW_OK;
}

}  // extern "C"

namespace {
// partial-record workspace of the tw_debug_* K|V stream launches: one allocation for every shape they accept (B <= 4096, H <= 20),
// zeroed when the call shape changes (it holds the arrival counters)
int debug_da_scratch(tw_ctx* ctx, int B, int H, float** out) {
    static float* scratch = nullptr;
    static int scratch_B = -1, scratch_H = -1;
    const size_t floats = decode_attention_partial_floats(4096, 20);
    if (!scratch) TW_CUDA_OK(ctx, cudaMalloc(&scratch, floats * sizeof(float)));
    if (B != scratch_B || H != scratch_H) {
        TW_CUDA_OK(ctx, cudaMemset(scratch, 0, floats * sizeof(float)));
        scratch_B = B; scratch_H = H;
    }
    *out = scratch;
    return TW_OK;
}
}  // namespace

extern "C" {

int tw_debug_decode_attention(tw_ctx* ctx, const void* q, int64_t q_stride, const void* kv, int64_t kv_clip_stride, int Tk, int B,
                              int H, int dtype, void* out, void* stream) {
    if (!ctx || !q || !kv || !out || B <= 0 || B > 4096 || Tk <= 0 || H <= 0 || H > 20) return TW_E_INVALID;
    float* scratch = nullptr;
    TW_CHECK(debug_da_scratch(ctx, B, H, &scratch));
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == TW_BF16)
        decode_attention<__nv_bfloat16>((const __nv_bfloat16*)q, q_stride, (const __nv_bfloat16*)kv, kv_clip_stride, Tk, nullptr, B, H,
                                        scratch, (__nv_bfloat16*)out, st);
    else
        decode_attention<float>((const float*)q, q_stride, (const float*)kv, kv_clip_stride, Tk, nullptr, B, H, scratch, (float*)out,
                                st);
    ctx->launches += 2;
    TW_CUDA_OK(ctx, cudaGetLastError());
    return TW_OK;
}

int tw_debug_self_attention(tw_ctx* ctx, const void* q, int64_t q_stride, const void* kv, int64_t kv_clip_stride, int Tk, int B, int H,
                            int dtype, void* out, void* stream) {
    if (!ctx || !q || !kv || !out || B <= 0 || Tk <= 0 || H <= 0) return TW_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == TW_BF16)
        self_attention_decode<__nv_bfloat16>((const __nv_bfloat16*)q, q_stride, (const __nv_bfloat16*)kv, kv_clip_stride, Tk, nullptr, B,
                                             H, (__nv_bfloat16*)out, st);
    else
        self_attention_decode<float>((const float*)q, q_stride, (const float*)kv, kv_clip_stride, Tk, nullptr, B, H, (float*)out, st);
    ctx->launches += 1;
    TW_CUDA_OK(ctx, cudaGetLastError());
    return TW_OK;
}

int tw_debug_self_attention_paged(tw_ctx* ctx, const void* q, int64_t q_stride, const void* pool, const int32_t* page_table,
                                  int pt_stride, int Tk, int B, int H, int dtype, void* out, void* stream) {
    if (!ctx || !q || !pool || !page_table || !out || B <= 0 || Tk <= 0 || H <= 0 || pt_stride <= 0) return TW_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == TW_BF16)
        self_attention_decode<__nv_bfloat16>((const __nv_bfloat16*)q, q_stride, (const __nv_bfloat16*)pool, 0, Tk, nullptr, B, H,
                                             (__nv_bfloat16*)out, st, page_table, pt_stride);
    else
        self_attention_decode<float>((const float*)q, q_stride, (const float*)pool, 0, Tk, nullptr, B, H, (float*)out, st, page_table,
                                     pt_stride);
    ctx->launches += 1;
    TW_CUDA_OK(ctx, cudaGetLastError());
    return TW_OK;
}

int tw_debug_decode_attention_step(tw_ctx* ctx, const void* q, int64_t q_stride, const void* kv, int64_t kv_clip_stride, int Tk, int B,
                                   int H, int dtype, const int32_t* active, const int32_t* n_active, int n_sms, void* out, void* stream) {
    if (!ctx || !q || !kv || !out || B <= 0 || B > 4096 || Tk <= 0 || H <= 0 || H > 20 || (!active) != (!n_active) ||
        (dtype != TW_BF16 && dtype != TW_F32))
        return TW_E_INVALID;
    float* scratch = nullptr;
    TW_CHECK(debug_da_scratch(ctx, B, H, &scratch));
    cudaStream_t st = (cudaStream_t)stream;
    // the grid of the stream kernel and the partition's SM count, as set_active_sms sets them for a pipeline stage
    const int sms_before = ctx->sm_count;
    const int da_before = decode_attention_set_sms(n_sms > 0 ? n_sms : 0);
    if (n_sms > 0) ctx->sm_count = n_sms;
    if (dtype == TW_BF16)
        decode_attention<__nv_bfloat16>((const __nv_bfloat16*)q, q_stride, (const __nv_bfloat16*)kv, kv_clip_stride, Tk, nullptr, B, H,
                                        scratch, (__nv_bfloat16*)out, st, nullptr, nullptr, active, n_active);
    else
        decode_attention<float>((const float*)q, q_stride, (const float*)kv, kv_clip_stride, Tk, nullptr, B, H, scratch, (float*)out, st,
                                nullptr, nullptr, active, n_active);
    decode_attention_set_sms(da_before);
    ctx->sm_count = sms_before;
    ctx->launches += 2;
    TW_CUDA_OK(ctx, cudaGetLastError());
    return TW_OK;
}

int tw_debug_self_attention_step(tw_ctx* ctx, const void* q, int64_t q_stride, const void* kv, int64_t kv_clip_stride, const int32_t* page_table,
                                 int pt_stride, const int32_t* d_pos, const int32_t* finished, int B, int H, int dtype, int variant, void* out,
                                 void* stream) {
    if (!ctx || !q || !kv || !d_pos || !out || B <= 0 || H <= 0 || (page_table && pt_stride <= 0) || variant < SA_VARIANT_DEFAULT ||
        variant > SA_VARIANT_RING || (dtype != TW_BF16 && dtype != TW_F32))
        return TW_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == TW_BF16)
        self_attention_decode<__nv_bfloat16>((const __nv_bfloat16*)q, q_stride, (const __nv_bfloat16*)kv, kv_clip_stride, 0, d_pos, B, H,
                                             (__nv_bfloat16*)out, st, page_table, pt_stride, finished, variant);
    else
        self_attention_decode<float>((const float*)q, q_stride, (const float*)kv, kv_clip_stride, 0, d_pos, B, H, (float*)out, st, page_table,
                                     pt_stride, finished, variant);
    ctx->launches += 1;
    TW_CUDA_OK(ctx, cudaGetLastError());
    return TW_OK;
}

int tw_debug_kv_append(tw_ctx* ctx, const void* A, const void* W, const float* bias, void* C, void* pool, const int32_t* page_table,
                       int pt_stride, const int32_t* d_pos, int M, int d, int dtype, int fused, int n_sms, void* stream) {
    if (!ctx || !A || !W || !C || !pool || !page_table || !d_pos || M <= 0 || d <= 0 || pt_stride <= 0 ||
        (dtype != TW_BF16 && dtype != TW_F32) || (fused && dtype != TW_BF16))
        return TW_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    const int sms_before = ctx->sm_count;
    if (n_sms > 0) ctx->sm_count = n_sms;          // the skinny GEMM sizes its tiles and grid from it
    GemmEpi e = mk_epi(EPI_STORE, bias, C, 3 * d);
    int r = TW_OK;
    if (dtype == TW_BF16) {
        typedef __nv_bfloat16 T;
        const bool skinny = gemm_tc_skinny_supported(M, 3 * d, d, e);
        if (fused) {
            // as launch_step issues it: the K|V columns go to the pool row of (row, *d_pos) through the page table
            e.n_split = d;
            e.C2 = pool;
            e.ldc2 = 0;
            e.d_row2 = d_pos;
            e.row2_stride = 2 * d;
            e.page_table = page_table;
            e.pt_stride = pt_stride;
            if (!skinny) {
                ctx->set_error(TW_E_UNSUPPORTED, "tw_debug_kv_append: the fused append needs the skinny GEMM (M <= 256, d % 64 == 0)");
                r = TW_E_UNSUPPORTED;
            } else {
                r = gemm_tc_skinny(ctx, (const T*)A, d, (const T*)W, d, M, 3 * d, d, e, st);
            }
        } else {
            r = skinny ? gemm_tc_skinny(ctx, (const T*)A, d, (const T*)W, d, M, 3 * d, d, e, st)
                       : gemm_tc(ctx, (const T*)A, d, (const T*)W, d, M, 3 * d, d, e, st);
            if (r == TW_OK) kv_append<T>((const T*)C, (T*)pool, d_pos, M, d, 0, st, page_table, pt_stride);
        }
    } else {
        gemm_simt<float>((const float*)A, d, (const float*)W, d, M, 3 * d, d, e, st);
        kv_append<float>((const float*)C, (float*)pool, d_pos, M, d, 0, st, page_table, pt_stride);
    }
    ctx->sm_count = sms_before;
    ctx->launches += fused ? 1 : 2;
    if (r == TW_OK) TW_CUDA_OK(ctx, cudaGetLastError());
    return r;
}

int tw_debug_encoder_attention(tw_ctx* ctx, const void* qkv, void* out, int B, int S, int H, int dtype, int impl, void* stream) {
    if (!ctx || !qkv || !out || B <= 0 || S <= 0 || H <= 0) return TW_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == TW_BF16 && impl == 1) {
        ctx->launches += 1;
        return encoder_attention_tc(ctx, (const __nv_bfloat16*)qkv, (__nv_bfloat16*)out, B, S, H, st);
    }
    if (dtype == TW_BF16)
        encoder_attention_simt<__nv_bfloat16>((const __nv_bfloat16*)qkv, (__nv_bfloat16*)out, B, S, H, st);
    else
        encoder_attention_simt<float>((const float*)qkv, (float*)out, B, S, H, st);
    ctx->launches += 1;
    TW_CUDA_OK(ctx, cudaGetLastError());
    return TW_OK;
}

int tw_debug_attention(tw_ctx* ctx, const void* q, int64_t q_ld, int q_col0, const void* kv, int64_t kv_ld, int k_col0, int v_col0,
                       void* out, int B, int Sq, int Sk, int H, int dtype, int impl, int causal, void* stream) {
    if (!ctx || !q || !kv || !out || B <= 0 || Sq <= 0 || Sk <= 0 || H <= 0) return TW_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    ctx->launches += 1;
    if (dtype == TW_BF16 && impl == 1)
        return attention_tc(ctx, (const __nv_bfloat16*)q, q_ld, q_col0, (const __nv_bfloat16*)kv, kv_ld, k_col0, v_col0,
                            (__nv_bfloat16*)out, B, Sq, Sk, H, causal != 0, st);
    if (dtype == TW_BF16)
        attention_simt<__nv_bfloat16>((const __nv_bfloat16*)q + q_col0, q_ld, (const __nv_bfloat16*)kv + k_col0,
                                      (const __nv_bfloat16*)kv + v_col0, kv_ld, (__nv_bfloat16*)out, B, Sq, Sk, H, causal != 0, st);
    else
        attention_simt<float>((const float*)q + q_col0, q_ld, (const float*)kv + k_col0, (const float*)kv + v_col0, kv_ld, (float*)out,
                              B, Sq, Sk, H, causal != 0, st);
    TW_CUDA_OK(ctx, cudaGetLastError());
    return TW_OK;
}

void tw_debug_set_pdl(int on) { g_pdl = on != 0; }

int tw_debug_set_row_budgets(tw_model* m, const int32_t* budgets_host, int n) {
    if (!m || n < 0 || n > m->desc.max_batch || (n > 0 && !budgets_host)) return TW_E_INVALID;
    m->row_budget_on = n > 0;
    if (n > 0) {
        std::vector<int32_t> tmp(m->desc.max_batch, 0x7fffffff);
        for (int i = 0; i < n; ++i) tmp[i] = budgets_host[i] < 1 ? 1 : budgets_host[i];
        TW_CUDA_OK(m->ctx, cudaMemcpy(m->d_row_budget, tmp.data(), tmp.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    }
    return TW_OK;
}

int tw_debug_select_steps(tw_model* m, const float* logits, int64_t ld_logits, int B, const int32_t* prompt, int P, const tw_rules* rules,
                          int max_length, const int32_t* row_budgets, const int32_t* forced, float* logits_tap, int tap_steps,
                          int32_t* out_tokens, int32_t* out_lengths, int32_t* n_active, int32_t* active, void* stream) {
    BroadcastPrompt bp(m, prompt, P, B);
    return tw_debug_select_steps_rows(m, logits, ld_logits, B, &bp.rows, P, rules, max_length, row_budgets, forced, logits_tap, tap_steps,
                                      out_tokens, out_lengths, n_active, active, stream);
}

int tw_debug_select_steps_rows(tw_model* m, const float* logits, int64_t ld_logits, int B, const tw_prompt_rows* rows, int P,
                               const tw_rules* rules, int max_length, const int32_t* row_budgets, const int32_t* forced, float* logits_tap,
                               int tap_steps, int32_t* out_tokens, int32_t* out_lengths, int32_t* n_active, int32_t* active, void* stream) {
    if (!check_model(m, "tw_debug_select_steps")) return TW_E_INVALID;
    if (!rows) {
        m->ctx->set_error(TW_E_INVALID, "tw_debug_select_steps_rows: null rows");
        return TW_E_INVALID;
    }
    TW_CHECK(check_decode_args(m, B, *rows, P, rules, max_length));
    tw_ctx* ctx = m->ctx;
    const int V = m->desc.vocab, n_gen = max_length - P;
    if (!logits || !out_tokens || !out_lengths || ld_logits < V || (ld_logits % 4) || (reinterpret_cast<uintptr_t>(logits) & 15) ||
        (logits_tap && (tap_steps < 0 || tap_steps > n_gen))) {
        ctx->set_error(TW_E_INVALID, "tw_debug_select_steps: null buffer, or logits without a 16-byte aligned base and a row pitch >= vocab "
                                     "that is a multiple of 4 floats, or tap_steps outside 0 .. max_length - P");
        return TW_E_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    RulesDev R;
    TW_CHECK(upload_rules(m, rules, &R, st));
    const bool budgets_before = m->row_budget_on;
    TW_CHECK(tw_debug_set_row_budgets(m, row_budgets, row_budgets ? B : 0));
    DecodeState S;
    int r = begin_decode(m, B, *rows, P, max_length, out_lengths, logits_tap, tap_steps, st, &S);
    // the decode loop of decode_impl with the logits of generated step g read from logits + g * B * ld_logits instead of the model
    // (prompt steps read those of step 0; so does the language pick of position 0)
    for (int pos = 0; r == TW_OK && pos < max_length - 1; ++pos) {
        const int g = pos - (P - 1);
        const float* lg = logits + (int64_t)(g > 0 ? g : 0) * B * ld_logits;
        if (pos == 0 && m->pick_now) pick_language(lg, ld_logits, B, m->d_lang_ids, m->n_lang_now, S, rows->out_lang, st);
        else select_tokens(lg, ld_logits, V, B, m->d_step, R, S, out_tokens, out_lengths, forced, logits_tap, st);
        advance_step(m->d_step, S, B, st);
        ctx->launches += 2;
        if (g >= 0 && n_active && cudaMemcpyAsync(n_active + g, S.n_active, sizeof(int32_t), cudaMemcpyDeviceToDevice, st) != cudaSuccess) r = TW_E_CUDA;
        if (g >= 0 && active && cudaMemcpyAsync(active + (int64_t)g * B, S.active, B * sizeof(int32_t), cudaMemcpyDeviceToDevice, st) != cudaSuccess)
            r = TW_E_CUDA;
    }
    // budgets given here apply to this call only; without them the budgets of tw_debug_set_row_budgets stay as they were
    if (row_budgets) m->row_budget_on = false;
    else m->row_budget_on = budgets_before;
    if (r == TW_E_CUDA) ctx->set_error(TW_E_CUDA, std::string("tw_debug_select_steps: ") + cudaGetErrorString(cudaGetLastError()));
    if (r == TW_OK) TW_CUDA_OK(ctx, cudaGetLastError());
    return r;
}

int tw_profile(tw_model* m, int enable, float* total_ms, int* launches, double* bytes_per_launch) {
    if (!m) return TW_E_INVALID;
    if (total_ms || launches) {
        float tot = 0.0f;
        int n = 0;
        for (int i = 0; i + 1 < m->prof_used; i += 2) {
            float ms = 0.0f;
            if (cudaEventSynchronize(m->prof_ev[i + 1]) == cudaSuccess &&
                cudaEventElapsedTime(&ms, m->prof_ev[i], m->prof_ev[i + 1]) == cudaSuccess) {
                tot += ms;
                ++n;
            }
        }
        if (total_ms) *total_ms = tot;
        if (launches) *launches = n;
    }
    if (bytes_per_launch) *bytes_per_launch = m->prof_bytes;   // K|V bytes of one profiled launch
    m->prof_used = 0;
    m->prof_on = enable != 0;
    if (m->prof_on && m->prof_ev.empty()) {
        m->prof_ev.resize(2 * 2048);
        for (auto& ev : m->prof_ev) {
            if (cudaEventCreate(&ev) != cudaSuccess) {
                m->ctx->set_error(TW_E_CUDA, "tw_profile: cudaEventCreate failed");
                return TW_E_CUDA;
            }
        }
    }
    return TW_OK;
}

int tw_last_stage_ms(tw_model* m, float out_ms[6]) {
    if (!m || !out_ms) return TW_E_INVALID;
    for (int i = 0; i < 6; ++i) out_ms[i] = 0.0f;
    for (int i = 0; i < 4; ++i)
        if (m->ev_valid[i] && m->ev_valid[i + 1]) {
            // under the pipeline the decode stage starts at its own event (the stages run on different streams)
            cudaEvent_t a = (i == 3 && m->ev_valid[7]) ? m->ev[7] : m->ev[i];
            if (cudaEventSynchronize(m->ev[i + 1]) == cudaSuccess && cudaEventSynchronize(a) == cudaSuccess)
                cudaEventElapsedTime(&out_ms[i], a, m->ev[i + 1]);
        }
    if (m->ev_valid[6] && m->ev_valid[0]) cudaEventElapsedTime(&out_ms[5], m->ev[6], m->ev[0]);
    int first = m->ev_valid[6] ? 6 : -1;
    for (int i = 0; i < 5 && first < 0; ++i)
        if (m->ev_valid[i]) first = i;
    if (first >= 0 && first != 4 && m->ev_valid[4] && !m->ev_valid[7]) cudaEventElapsedTime(&out_ms[4], m->ev[first], m->ev[4]);
    return TW_OK;
}

}  // extern "C"
