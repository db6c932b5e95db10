// Attention kernels.
//  * encoder_attention_simt: tiled online-softmax attention in fp32 on CUDA cores — the fp32
//    check-mode path and the bring-up path for bf16 (the tcgen05 flash kernel is attention_tc.cu).
//  * decode_attention: one query per clip against a K|V row store (cross-attention K/V computed once
//    per window, or the self-attention cache).  HBM-bound streaming kernel: each CTA owns a
//    contiguous chunk of rows for ALL heads (rows are [K(d) | V(d)] contiguous), online softmax per
//    head in registers, partials merged by a second tiny kernel (flash-decoding split over time).
// Arithmetic: HF WhisperAttention.forward (modeling_whisper.py:284-358): q already scaled by
// head_dim^-0.5 (folded into the weights), softmax in fp32, no mask in the encoder.
#include <stdlib.h>

#include "kernels.cuh"

namespace tw {

constexpr int HD = 64;   // Whisper head_dim is 64 for every checkpoint size

// ------------------------------------------------------------------------------------------------
constexpr int EA_BQ = 64, EA_BK = 64, EA_THREADS = 256;

struct EaSmem {
    float q[EA_BQ][HD + 1];
    float k[EA_BK][HD + 1];
    float v[EA_BK][HD + 4];
    float s[EA_BQ][EA_BK + 1];
    float m[EA_BQ], l[EA_BQ], scale[EA_BQ];
};

// General form: Sq queries per clip (rows of q, pitch q_ld) against Sk keys / values per clip (rows of k and v, pitch
// kv_ld); causal = key index <= query index (decoder self-attention over a full token sequence).  The encoder case is
// q = qkv, k = qkv + d, v = qkv + 2d, pitches 3d, Sq = Sk = S.
template <typename T>
__global__ void __launch_bounds__(EA_THREADS)
encoder_attention_simt_kernel(const T* __restrict__ q, int64_t q_ld, const T* __restrict__ k, const T* __restrict__ v, int64_t kv_ld,
                              T* __restrict__ out, int S, int Sk, int H, int causal) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    EaSmem& sm = *reinterpret_cast<EaSmem*>(smem_raw);
    const int d = H * HD;
    const int q0 = blockIdx.x * EA_BQ, h = blockIdx.y, b = blockIdx.z;
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;        // 16 x 16 threads, 4 x 4 outputs each
    const T* qbase = q + (int64_t)b * S * q_ld;
    const T* kbase = k + (int64_t)b * Sk * kv_ld;
    const T* vbase = v + (int64_t)b * Sk * kv_ld;

    for (int i = tid; i < EA_BQ * HD; i += EA_THREADS) {
        const int r = i / HD, c = i % HD;
        sm.q[r][c] = (q0 + r < S) ? to_f32(qbase[(int64_t)(q0 + r) * q_ld + h * HD + c]) : 0.0f;
    }
    if (tid < EA_BQ) {
        sm.m[tid] = -INFINITY;
        sm.l[tid] = 0.0f;
    }
    float o[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) o[i][j] = 0.0f;

    const int k_end = causal ? min(Sk, q0 + EA_BQ) : Sk;      // causal: key tiles past the last query of the block are all masked
    for (int k0 = 0; k0 < k_end; k0 += EA_BK) {
        __syncthreads();
        for (int i = tid; i < EA_BK * HD; i += EA_THREADS) {
            const int r = i / HD, c = i % HD;
            const bool ok = k0 + r < Sk;
            const int64_t row = (int64_t)(k0 + r) * kv_ld;
            sm.k[r][c] = ok ? to_f32(kbase[row + h * HD + c]) : 0.0f;
            sm.v[r][c] = ok ? to_f32(vbase[row + h * HD + c]) : 0.0f;
        }
        __syncthreads();
        // S tile = Q K^T, 4x4 per thread (rows ty*4.., cols tx*4..)
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
#pragma unroll 8
        for (int c = 0; c < HD; ++c) {
            float a[4], bb[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = sm.q[ty * 4 + i][c];
#pragma unroll
            for (int j = 0; j < 4; ++j) bb[j] = sm.k[tx * 4 + j][c];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int kc = k0 + tx * 4 + j;
                sm.s[ty * 4 + i][tx * 4 + j] = (kc < Sk && !(causal && kc > q0 + ty * 4 + i)) ? acc[i][j] : -INFINITY;
            }
        __syncthreads();
        // online softmax: warp w handles rows w*8 .. w*8+7, lanes cover 64 columns (2 each)
        {
            const int w = tid >> 5, lane = tid & 31;
            for (int r = w * 8; r < w * 8 + 8; ++r) {
                const float s0 = sm.s[r][lane], s1 = sm.s[r][lane + 32];
                const float mx = warp_max(fmaxf(s0, s1));
                const float m_old = sm.m[r];
                const float m_new = fmaxf(m_old, mx);
                const float p0 = __expf(s0 - m_new), p1 = __expf(s1 - m_new);
                const float ps = warp_sum(p0 + p1);
                sm.s[r][lane] = p0;
                sm.s[r][lane + 32] = p1;
                if (lane == 0) {
                    const float sc = (m_old == -INFINITY) ? 0.0f : __expf(m_old - m_new);
                    sm.scale[r] = sc;
                    sm.l[r] = sm.l[r] * sc + ps;
                    sm.m[r] = m_new;
                }
            }
        }
        __syncthreads();
        // O = O*scale + P V ; 4x4 per thread (rows ty*4.., dims tx*4..)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float sc = sm.scale[ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) o[i][j] *= sc;
        }
#pragma unroll 8
        for (int kk = 0; kk < EA_BK; ++kk) {
            const float4 vv = *reinterpret_cast<const float4*>(&sm.v[kk][tx * 4]);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float p = sm.s[ty * 4 + i][kk];
                o[i][0] = fmaf(p, vv.x, o[i][0]);
                o[i][1] = fmaf(p, vv.y, o[i][1]);
                o[i][2] = fmaf(p, vv.z, o[i][2]);
                o[i][3] = fmaf(p, vv.w, o[i][3]);
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = q0 + ty * 4 + i;
        if (r >= S) continue;
        const float inv = 1.0f / sm.l[ty * 4 + i];
        T* orow = out + ((int64_t)b * S + r) * d + h * HD + tx * 4;
#pragma unroll
        for (int j = 0; j < 4; ++j) orow[j] = from_f32<T>(o[i][j] * inv);
    }
}

template <typename T>
void attention_simt(const T* q, int64_t q_ld, const T* k, const T* v, int64_t kv_ld, T* out, int B, int Sq, int Sk, int H, bool causal,
                    cudaStream_t st) {
    static bool attr_set[2] = {false, false};
    const int which = sizeof(T) == 4 ? 0 : 1;
    if (!attr_set[which]) {
        cudaFuncSetAttribute(encoder_attention_simt_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(EaSmem));
        attr_set[which] = true;
    }
    dim3 grid(ceil_div(Sq, EA_BQ), H, B);
    encoder_attention_simt_kernel<T><<<grid, EA_THREADS, sizeof(EaSmem), st>>>(q, q_ld, k, v, kv_ld, out, Sq, Sk, H, causal ? 1 : 0);
}
template void attention_simt<float>(const float*, int64_t, const float*, const float*, int64_t, float*, int, int, int, int, bool, cudaStream_t);
template void attention_simt<__nv_bfloat16>(const __nv_bfloat16*, int64_t, const __nv_bfloat16*, const __nv_bfloat16*, int64_t,
                                            __nv_bfloat16*, int, int, int, int, bool, cudaStream_t);

template <typename T>
void encoder_attention_simt(const T* qkv, T* out, int B, int S, int H, cudaStream_t st) {
    const int d = H * HD;
    attention_simt<T>(qkv, 3 * d, qkv + d, qkv + 2 * d, 3 * d, out, B, S, S, H, false, st);
}
template void encoder_attention_simt<float>(const float*, float*, int, int, int, cudaStream_t);
template void encoder_attention_simt<__nv_bfloat16>(const __nv_bfloat16*, __nv_bfloat16*, int, int, int, cudaStream_t);

// ------------------------------------------------------------------------------------------------
// decode attention — persistent TMA-bulk streaming kernel.
//
// The B*Tk rows of the K|V store are one flat stream split evenly over G = #SM CTAs (each CTA owns
// R consecutive rows, possibly spanning a clip boundary).  A producer warp issues cp.async.bulk copies
// of 8-row stages (8 x 2d elements, contiguous in HBM) into a shared-memory ring (mbarrier
// complete_tx), 8 consumer warps take one row each per stage: per-head dot products with the query
// held in registers, online softmax, P.V accumulation, all in fp32.  At the end of a clip segment the
// warps merge through shared memory (tree merge, 4-record buffer) and emit one partial record (m, l, o[64])
// per head; a small second kernel merges the records of a clip.  Record index = cta + clip (unique, <= G + B - 2).
// Variants measured on B200 and rejected (profiles/r01_split_decode.md): the refill issued by the last warp to release a
// stage (shared-memory counter), and warp-private rings of single-row copies — both 10-15 % slower.
constexpr int DA_WARPS = 8;        // consumer warps
// rows per warp per stage: with two, their dot products / exponentials are independent chains.  The one-row kernel was bound by the
// consumer warps' latency per row, not by HBM (its rate followed the number of SMs: 5.32 TB/s on 148, 4.64 on 124); with two rows it
// is HBM-bound (5.83 TB/s on 148 SMs, 5.80 on 124).  The fp32 check mode keeps one row (its stage would not fit twice).
template <typename T> struct DaRows { static constexpr int RPW = sizeof(T) == 2 ? 2 : 1; static constexpr int SROWS = DA_WARPS * RPW; };
constexpr int DA_MAXSLOT = 5;      // ceil(H*8/32) with H <= 20
constexpr int DA_PSTRIDE = HD + 2; // partial record: m, l, o[64]
constexpr int DA_MAX_STAGES = 8;

__device__ __forceinline__ uint32_t da_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void da_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void da_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void da_mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void da_mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "DA_WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DA_WAIT_DONE;\n"
        "bra DA_WAIT_LOOP;\n"
        "DA_WAIT_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void da_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(policy) : "memory");
}

template <typename T> struct Vec8;
template <> struct Vec8<float> {
    static __device__ __forceinline__ void load_shared(const float* p, float* f) {
        const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
        f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
    }
};
template <> struct Vec8<__nv_bfloat16> {
    static __device__ __forceinline__ void load_shared(const __nv_bfloat16* p, float* f) {
        const uint4 raw = *reinterpret_cast<const uint4*>(p);
        // bf16 -> f32 is a 16-bit shift: low half and high half of each word
        f[0] = __uint_as_float(raw.x << 16); f[1] = __uint_as_float(raw.x & 0xffff0000u);
        f[2] = __uint_as_float(raw.y << 16); f[3] = __uint_as_float(raw.y & 0xffff0000u);
        f[4] = __uint_as_float(raw.z << 16); f[5] = __uint_as_float(raw.z & 0xffff0000u);
        f[6] = __uint_as_float(raw.w << 16); f[7] = __uint_as_float(raw.w & 0xffff0000u);
    }
};

// rows per CTA for a stream of total_rows split over at most `grid` CTAs (same formula on host and device)
__host__ __device__ inline int da_rows_per_cta(int64_t total_rows, int grid) {
    int64_t g = (total_rows + DA_WARPS - 1) / DA_WARPS;
    if (g > grid) g = grid;
    if (g < 1) g = 1;
    return (int)((total_rows + g - 1) / g);
}

struct DaPlan {
    int G;        // CTAs
    int R;        // rows per CTA
    int stages;
    size_t smem;
};
static DaPlan da_plan(int total_rows, int H, int esz, int sm_count, int max_stages, int nw) {
    DaPlan p;
    int g = ceil_div(total_rows, DA_WARPS);
    if (g > sm_count) g = sm_count;
    if (g < 1) g = 1;
    p.G = g;
    p.R = ceil_div(total_rows, g);
    const size_t stage_bytes = (size_t)nw * (esz == 2 ? 2 : 1) * 2 * H * HD * esz;
    const size_t merge_bytes = (size_t)nw * H * DA_PSTRIDE * sizeof(float);
    int st = (int)((220 * 1024 - merge_bytes) / stage_bytes);
    if (st > DA_MAX_STAGES) st = DA_MAX_STAGES;
    if (st > max_stages) st = max_stages;
    if (st < 2) st = 2;
    p.stages = st;
    p.smem = st * stage_bytes + merge_bytes + 256;
    return p;
}

// NW = consumer warps = rows per stage (+ the producer warp = 9 warps)
template <typename T>
__global__ void __launch_bounds__((DA_WARPS + 1) * 32, 1)
decode_attention_stream(const T* __restrict__ q, int64_t q_stride, const T* __restrict__ kv, int64_t kv_clip_stride, int Tk,
                        const int32_t* __restrict__ d_tk, int B, int H, int stages, int kv_static, float* __restrict__ partial,
                        const int32_t* __restrict__ active, const int32_t* __restrict__ n_active) {
    constexpr int NW = DA_WARPS;
    constexpr int DA_RPW = DaRows<T>::RPW, DA_SROWS = DaRows<T>::SROWS;
    extern __shared__ __align__(128) unsigned char da_raw[];
    const int d = H * HD;
    const int row_elems = 2 * d;
    const uint32_t stage_bytes = (uint32_t)DA_SROWS * row_elems * sizeof(T);
    T* ring = reinterpret_cast<T*>(da_raw);
    float* merge = reinterpret_cast<float*>(da_raw + (size_t)stages * stage_bytes);
    uint64_t* bars = reinterpret_cast<uint64_t*>(da_raw + (size_t)stages * stage_bytes + (size_t)NW * H * DA_PSTRIDE * sizeof(float));
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + DA_MAX_STAGES;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    pdl_trigger();
    // kv_static: the K|V store was written long before the previous kernel (cross-attention K/V of the window), so the
    // producer may start streaming it while the previous kernel (the q projection) is still running
    if (!(kv_static && warp == NW)) pdl_wait();
    if (d_tk) Tk = *d_tk + 1;
    // active list (decode loop): only the clips that have not emitted EOS are streamed; slot s of the flat row stream is
    // clip active[s].  The list was written by the previous step's advance kernel, which every kernel of this step is
    // ordered after (the step's first kernel is launched with a full dependency), so it may be read before the wait.
    if (active) B = *n_active;
    const int64_t total = (int64_t)B * Tk;
    const int R = da_rows_per_cta(total, gridDim.x);
    const int64_t row_begin = (int64_t)blockIdx.x * R;
    const int64_t row_end = min(total, row_begin + R);
    if (row_begin >= total) return;             // short caches do not need every CTA

    if (threadIdx.x == 0) {
        for (int s = 0; s < stages; ++s) {
            da_mbar_init(da_smem_u32(&full_bar[s]), 1);
            da_mbar_init(da_smem_u32(&empty_bar[s]), NW);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp == NW) {
        // ===================== producer =====================
        if (lane == 0) {
            // the K|V store is streamed once per launch and is far larger than L2: mark the lines evict-first
            uint64_t policy;
            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
            int stage = 0;
            uint32_t phase = 0;
            int64_t r = row_begin;
            while (r < row_end) {
                const int b = (int)(r / Tk);                         // slot in the row stream
                const int64_t seg_end = min(row_end, (int64_t)(b + 1) * Tk);
                const T* src_clip = kv + (int64_t)(active ? active[b] : b) * kv_clip_stride;
                for (int64_t r0 = r; r0 < seg_end; r0 += DA_SROWS) {
                    const int nrows = (int)min((int64_t)DA_SROWS, seg_end - r0);
                    da_mbar_wait(da_smem_u32(&empty_bar[stage]), phase ^ 1);
                    const uint32_t bytes = (uint32_t)nrows * row_elems * sizeof(T);
                    const uint32_t fb = da_smem_u32(&full_bar[stage]);
                    da_mbar_expect_tx(fb, bytes);
                    da_bulk_g2s(da_smem_u32(reinterpret_cast<unsigned char*>(ring) + (size_t)stage * stage_bytes),
                                src_clip + (r0 - (int64_t)b * Tk) * row_elems, bytes, fb, policy);
                    if (++stage == stages) { stage = 0; phase ^= 1; }
                }
                r = seg_end;
            }
            if (kv_static) pdl_wait();               // every thread of the grid observes the dependency before exiting
        }
        return;
    }

    // ===================== consumers =====================
    const int nslots = H * 8;
    int stage = 0;
    uint32_t phase = 0;
    int64_t r = row_begin;
    while (r < row_end) {
        const int b = (int)(r / Tk);                                 // slot in the row stream
        const int64_t seg_end = min(row_end, (int64_t)(b + 1) * Tk);
        const T* qb = q + (int64_t)(active ? active[b] : b) * q_stride;
        float qf[DA_MAXSLOT][8], of[DA_MAXSLOT][8], mrun[DA_MAXSLOT], lrun[DA_MAXSLOT];
#pragma unroll
        for (int s = 0; s < DA_MAXSLOT; ++s) {
            const int slot = lane + 32 * s;
            mrun[s] = -INFINITY;
            lrun[s] = 0.0f;
#pragma unroll
            for (int e = 0; e < 8; ++e) { of[s][e] = 0.0f; qf[s][e] = 0.0f; }
            if (slot < nslots) {
#pragma unroll
                for (int e = 0; e < 8; ++e) qf[s][e] = to_f32(qb[slot * 8 + e]);
            }
        }
        for (int64_t r0 = r; r0 < seg_end; r0 += DA_SROWS) {
            const int nrows = (int)min((int64_t)DA_SROWS, seg_end - r0);
            da_mbar_wait(da_smem_u32(&full_bar[stage]), phase);
            if (warp < nrows) {
                // this warp's rows of the stage: warp and warp + DA_WARPS (the second one may be past the segment)
                const T* row0 = reinterpret_cast<const T*>(reinterpret_cast<const unsigned char*>(ring) + (size_t)stage * stage_bytes) +
                                (size_t)warp * row_elems;
                const T* row1 = row0 + (size_t)DA_WARPS * row_elems;
                const bool two = DA_RPW == 2 && warp + DA_WARPS < nrows;   // warp-uniform
                // math is unconditional (idle slots carry zeros) so the shuffles stay warp-converged
#pragma unroll
                for (int s = 0; s < DA_MAXSLOT; ++s) {
                    const int slot = lane + 32 * s;
                    float k0[8], v0[8], k1[8], v1[8];
                    if (slot < nslots) {
                        Vec8<T>::load_shared(row0 + slot * 8, k0);
                        Vec8<T>::load_shared(row0 + d + slot * 8, v0);
                    } else {
#pragma unroll
                        for (int e = 0; e < 8; ++e) { k0[e] = 0.0f; v0[e] = 0.0f; }
                    }
                    if (two && slot < nslots) {
                        Vec8<T>::load_shared(row1 + slot * 8, k1);
                        Vec8<T>::load_shared(row1 + d + slot * 8, v1);
                    } else {
#pragma unroll
                        for (int e = 0; e < 8; ++e) { k1[e] = 0.0f; v1[e] = 0.0f; }
                    }
                    float dot0 = 0.0f, dot1 = 0.0f;
#pragma unroll
                    for (int e = 0; e < 8; ++e) { dot0 = fmaf(qf[s][e], k0[e], dot0); dot1 = fmaf(qf[s][e], k1[e], dot1); }
                    dot0 += __shfl_xor_sync(0xffffffffu, dot0, 1);
                    dot1 += __shfl_xor_sync(0xffffffffu, dot1, 1);
                    dot0 += __shfl_xor_sync(0xffffffffu, dot0, 2);
                    dot1 += __shfl_xor_sync(0xffffffffu, dot1, 2);
                    dot0 += __shfl_xor_sync(0xffffffffu, dot0, 4);
                    dot1 += __shfl_xor_sync(0xffffffffu, dot1, 4);
                    if (!two) dot1 = -INFINITY;                             // exp(-inf - m) = 0: the absent row adds nothing
                    const float m_new = fmaxf(mrun[s], fmaxf(dot0, dot1));
                    const float sc = __expf(mrun[s] - m_new);     // exp(-inf) = 0 on the first row
                    const float p0 = __expf(dot0 - m_new), p1 = __expf(dot1 - m_new);
                    lrun[s] = lrun[s] * sc + (p0 + p1);
                    mrun[s] = m_new;
#pragma unroll
                    for (int e = 0; e < 8; ++e) of[s][e] = fmaf(p1, v1[e], fmaf(p0, v0[e], of[s][e] * sc));
                }
            }
            __syncwarp();
            if (lane == 0) da_mbar_arrive(da_smem_u32(&empty_bar[stage]));
            if (++stage == stages) { stage = 0; phase ^= 1; }
        }
        // unsplit decode: all 8 warps post their records, then 256 threads reduce them in parallel (shortest tail;
        // the tree merge below costs ~2 us more per launch in situ)
        // ---- merge the 8 warps of this clip segment -> one partial record per head
#pragma unroll
        for (int s = 0; s < DA_MAXSLOT; ++s) {
            const int slot = lane + 32 * s;
            if (slot < nslots) {
                const int h = slot >> 3, e0 = (slot & 7) * 8;
                float* rec = merge + ((size_t)warp * H + h) * DA_PSTRIDE;
                if ((slot & 7) == 0) { rec[0] = mrun[s]; rec[1] = lrun[s]; }
#pragma unroll
                for (int e = 0; e < 8; ++e) rec[2 + e0 + e] = of[s][e];
            }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(NW * 32) : "memory");
        float* prec_base = partial + ((size_t)blockIdx.x + b) * H * DA_PSTRIDE;
        for (int i = threadIdx.x; i < H * HD; i += NW * 32) {
            const int h = i / HD, e = i % HD;
            float m = -INFINITY;
#pragma unroll
            for (int w = 0; w < NW; ++w) m = fmaxf(m, merge[((size_t)w * H + h) * DA_PSTRIDE]);
            float l = 0.0f, o = 0.0f;
#pragma unroll
            for (int w = 0; w < NW; ++w) {
                const float* rec = merge + ((size_t)w * H + h) * DA_PSTRIDE;
                const float sc = (rec[0] == -INFINITY) ? 0.0f : __expf(rec[0] - m);
                l += rec[1] * sc;
                o += rec[2 + e] * sc;
            }
            float* prec = prec_base + (size_t)h * DA_PSTRIDE;
            if (e == 0) { prec[0] = m; prec[1] = l; }
            prec[2 + e] = o;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(NW * 32) : "memory");
        r = seg_end;
    }
}

// HPC heads per CTA (64 threads each): 1 -> H x B CTAs of 64 threads, 4 -> ceil(H/4) x B CTAs of 256 threads
template <typename T, int HPC>
__global__ void __launch_bounds__(HD * HPC)
decode_attention_combine(const float* __restrict__ partial, int Tk, const int32_t* __restrict__ d_tk, int B, int grid, int H,
                         T* __restrict__ out, const int32_t* __restrict__ active, const int32_t* __restrict__ n_active) {
    pdl_trigger();
    pdl_wait();
    const int h = blockIdx.x * HPC + (threadIdx.x >> 6), b = blockIdx.y, e = threadIdx.x & 63;      // b: slot in the row stream
    if (h >= H) return;
    if (d_tk) Tk = *d_tk + 1;
    int clip = b;
    if (active) {
        B = *n_active;
        if (b >= B) return;                  // finished clips keep their stale row (its logits are never read)
        clip = active[b];
    }
    const int R = da_rows_per_cta((int64_t)B * Tk, grid);
    const int c_first = (int)(((int64_t)b * Tk) / R), c_last = (int)((((int64_t)b + 1) * Tk - 1) / R);
    float m = -INFINITY;
    for (int c = c_first; c <= c_last; ++c) m = fmaxf(m, partial[((size_t)(c + b) * H + h) * DA_PSTRIDE]);
    float l = 0.0f, o = 0.0f;
    for (int c = c_first; c <= c_last; ++c) {
        const float* rec = partial + ((size_t)(c + b) * H + h) * DA_PSTRIDE;
        const float sc = (rec[0] == -INFINITY) ? 0.0f : __expf(rec[0] - m);
        l += rec[1] * sc;
        o += rec[2 + e] * sc;
    }
    out[(int64_t)clip * H * HD + h * HD + e] = from_f32<T>(o / l);
}

// ------------------------------------------------------------------------------------------------
// Self-attention over the short decoder cache (Tk = pos + 1 <= 448 rows): one CTA per (clip, group of 4 heads),
// 8 warps striding over the rows with 4 rows of K|V in flight per warp, online softmax per head in registers,
// warps merged through shared memory, normalised output written directly (single launch, no partial records).
constexpr int SA_HG = 4;            // heads per CTA: 4 x 64 dims = 32 lanes x 8 elements
constexpr int SA_WARPS = 8;
constexpr int SA_MAX_PAGES = 64;     // page-table entries of one clip staged in shared memory (Whisper: 448 / 16 = 28)

template <typename T> struct Ld8;
template <> struct Ld8<float> {
    struct Raw { float4 a, b; };
    static __device__ __forceinline__ Raw load(const float* p) {
        Raw r; r.a = *reinterpret_cast<const float4*>(p); r.b = *reinterpret_cast<const float4*>(p + 4); return r;
    }
    static __device__ __forceinline__ void unpack(const Raw& r, float* f) {
        f[0] = r.a.x; f[1] = r.a.y; f[2] = r.a.z; f[3] = r.a.w; f[4] = r.b.x; f[5] = r.b.y; f[6] = r.b.z; f[7] = r.b.w;
    }
};
template <> struct Ld8<__nv_bfloat16> {
    typedef uint4 Raw;
    static __device__ __forceinline__ Raw load(const __nv_bfloat16* p) { return *reinterpret_cast<const uint4*>(p); }
    static __device__ __forceinline__ void unpack(const Raw& raw, float* f) {
        f[0] = __uint_as_float(raw.x << 16); f[1] = __uint_as_float(raw.x & 0xffff0000u);
        f[2] = __uint_as_float(raw.y << 16); f[3] = __uint_as_float(raw.y & 0xffff0000u);
        f[4] = __uint_as_float(raw.z << 16); f[5] = __uint_as_float(raw.z & 0xffff0000u);
        f[6] = __uint_as_float(raw.w << 16); f[7] = __uint_as_float(raw.w & 0xffff0000u);
    }
};

// SA_UNR = rows in flight per warp
template <typename T, int SA_UNR>
__global__ void __launch_bounds__(SA_WARPS * 32, sizeof(T) == 2 ? 3 : 1)   // 3 CTAs / SM (<= 85 registers): the 5 x B grid of a 64-clip batch is one wave, and two CTAs fit next to a decode-step GEMM CTA
self_attention_decode_kernel(const T* __restrict__ q, int64_t q_stride, const T* __restrict__ kv, int64_t kv_clip_stride, int Tk,
                             const int32_t* __restrict__ d_tk, int H, T* __restrict__ out, const int32_t* __restrict__ page_table,
                             int pt_stride, const int32_t* __restrict__ finished, int early) {
    __shared__ float s_rec[SA_WARPS][SA_HG][HD + 2];
    __shared__ int32_t s_pt[SA_MAX_PAGES];
    pdl_trigger();
    const int hg = blockIdx.x, b = blockIdx.y;
    // a clip that has emitted EOS no longer reads its cache (flags written by the previous step's select kernel; ordering
    // as for the active list of the K|V stream kernel); the wait keeps the programmatic-dependency chain intact
    if (finished && finished[b]) { pdl_wait(); return; }
    // the page table is fixed for the whole decode call: stage this clip's row in shared memory before the dependency wait,
    // so that the per-row page lookup is not a dependent global load in front of every K|V row fetch
    const bool pt_smem = page_table && pt_stride <= SA_MAX_PAGES;
    if (pt_smem && (int)threadIdx.x < pt_stride) s_pt[threadIdx.x] = page_table[(int64_t)b * pt_stride + threadIdx.x];
    if (!early) pdl_wait();                          // q and the newest cache row come from the QKV GEMM just before
    if (pt_smem) __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (d_tk) Tk = *d_tk + 1;
    const int d = H * HD;
    const int col = hg * SA_HG * HD + lane * 8;       // this lane's 8 dims inside the row
    const bool active = col < d;
    // contiguous cache: row r of clip b at kv + b*kv_clip_stride + r*2d; paged cache: pool row kv_page_row(table, ., b, r)
    const T* kvb = kv + (page_table ? 0 : (int64_t)b * kv_clip_stride) + (active ? col : 0);
    const int32_t* ptb = page_table ? (pt_smem ? s_pt : page_table + (int64_t)b * pt_stride) : nullptr;
    auto row_ptr = [&](int r) -> const T* {
        const int64_t pr = ptb ? (int64_t)ptb[r / TW_KV_PAGE] * TW_KV_PAGE + r % TW_KV_PAGE : (int64_t)r;
        return kvb + pr * 2 * d;
    };
    float qf[8], of[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { qf[e] = 0.0f; of[e] = 0.0f; }
    float mrun = -INFINITY, lrun = 0.0f;
    auto consume = [&](const typename Ld8<T>::Raw& kraw, const typename Ld8<T>::Raw& vraw) {
        float kf[8], vf[8];
        if (active) { Ld8<T>::unpack(kraw, kf); Ld8<T>::unpack(vraw, vf); }
        else {
#pragma unroll
            for (int e = 0; e < 8; ++e) { kf[e] = 0.0f; vf[e] = 0.0f; }
        }
        float dot = 0.0f;
#pragma unroll
        for (int e = 0; e < 8; ++e) dot = fmaf(qf[e], kf[e], dot);
        dot += __shfl_xor_sync(0xffffffffu, dot, 1);
        dot += __shfl_xor_sync(0xffffffffu, dot, 2);
        dot += __shfl_xor_sync(0xffffffffu, dot, 4);
        const float m_new = fmaxf(mrun, dot);
        const float sc = __expf(mrun - m_new);
        const float p = __expf(dot - m_new);
        lrun = lrun * sc + p;
        mrun = m_new;
#pragma unroll
        for (int e = 0; e < 8; ++e) of[e] = fmaf(p, vf[e], of[e] * sc);
    };
    // Rows of earlier positions were written by earlier steps: with `early` (decode step: Tk = position + 1 read before the wait,
    // like the active list) the first batch of them is loaded into registers, and the later ones are pulled into L2, BEFORE the
    // dependency wait, i.e. under the QKV GEMM that is still running (its CTAs leave room for one CTA of this kernel per SM).  Only
    // q and the newest row depend on that GEMM.
    const int n_old = early ? Tk - 1 : Tk;            // rows [0, n_old) may be read before the wait
    typename Ld8<T>::Raw kr[SA_UNR], vr[SA_UNR];
    auto load_batch = [&](int base, int lim) {
#pragma unroll
        for (int u = 0; u < SA_UNR; ++u) {
            const int r = base + u * SA_WARPS;
            if (r < lim && active) {
                const T* rp = row_ptr(r);
                kr[u] = Ld8<T>::load(rp);
                vr[u] = Ld8<T>::load(rp + d);
            }
        }
    };
    int r0 = warp, lim = n_old;
    load_batch(r0, lim);
    if (early) {
        // one 128-byte line per lane: lanes 0-3 the K part of this CTA's 4 heads, lanes 4-7 the V part
        if (lane < 8 && hg * SA_HG * HD + (lane & 3) * 64 < d) {
            for (int r = warp + SA_UNR * SA_WARPS; r < n_old; r += SA_WARPS) {
                const int64_t pr = ptb ? (int64_t)ptb[r / TW_KV_PAGE] * TW_KV_PAGE + r % TW_KV_PAGE : (int64_t)r;
                const T* lp = kv + (page_table ? 0 : (int64_t)b * kv_clip_stride) + pr * 2 * d + (lane >> 2) * d + hg * SA_HG * HD + (lane & 3) * 64;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(lp));
            }
        }
        pdl_wait();
    }
    if (active) {
#pragma unroll
        for (int e = 0; e < 8; ++e) qf[e] = to_f32(q[(int64_t)b * q_stride + col + e]);
    }
    while (true) {
#pragma unroll
        for (int u = 0; u < SA_UNR; ++u)
            if (r0 + u * SA_WARPS < lim) consume(kr[u], vr[u]);                  // warp-uniform
        r0 += SA_WARPS * SA_UNR;
        if (r0 >= Tk) break;
        lim = Tk;
        load_batch(r0, lim);
    }
    // early path: the newest row when it falls inside the first batch (Tk - 1 < SA_UNR * SA_WARPS), which the loop above skipped
    if (early && Tk - 1 < SA_UNR * SA_WARPS && (Tk - 1) % SA_WARPS == warp) {
        typename Ld8<T>::Raw k1, v1;
        if (active) {
            const T* rp = row_ptr(Tk - 1);
            k1 = Ld8<T>::load(rp);
            v1 = Ld8<T>::load(rp + d);
        }
        consume(k1, v1);
    }
    {
        float* rec = s_rec[warp][lane >> 3];
        if ((lane & 7) == 0) { rec[0] = mrun; rec[1] = lrun; }
#pragma unroll
        for (int e = 0; e < 8; ++e) rec[2 + (lane & 7) * 8 + e] = of[e];
    }
    __syncthreads();
    {
        const int hh = threadIdx.x >> 6, e = threadIdx.x & 63;       // 256 threads = 4 heads x 64 dims
        const int h = hg * SA_HG + hh;
        if (h < H) {
            float m = -INFINITY;
#pragma unroll
            for (int w = 0; w < SA_WARPS; ++w) m = fmaxf(m, s_rec[w][hh][0]);
            float l = 0.0f, o = 0.0f;
#pragma unroll
            for (int w = 0; w < SA_WARPS; ++w) {
                const float sc = (s_rec[w][hh][0] == -INFINITY) ? 0.0f : __expf(s_rec[w][hh][0] - m);
                l += s_rec[w][hh][1] * sc;
                o += s_rec[w][hh][2 + e] * sc;
            }
            out[(int64_t)b * d + h * HD + e] = from_f32<T>(o / l);
        }
    }
}

// ---- ring variant: the same row order and arithmetic (bit-identical output), but K|V rows land in a per-warp shared-memory ring
// of SA_RING rows through 16-byte cp.async copies issued SA_RING rows ahead, so every warp keeps SA_RING rows (1 KB each for the
// CTA's 4 heads in bf16) in flight ALL the time.  The register version above has 4 rows in flight per warp only while it waits
// and none while it consumes (measured ~3.5 TB/s marginal on the cache at 192 merged rows, where this kernel is ~12 % of a decode
// step); the ring holds 8.  Each lane reads back exactly the bytes it copied itself: no cross-lane hand-over, no barrier — only
// cp.async.wait_group.  Every iteration commits one group (an empty one when the warp has run out of rows), so "all but the
// newest SA_RING - 1 groups complete" always means "the oldest row in the ring has arrived".
constexpr int SA_RING = 8;

__device__ __forceinline__ void sa_cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void sa_cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void sa_cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <typename T>
__global__ void __launch_bounds__(SA_WARPS * 32, sizeof(T) == 2 ? 3 : 1)
self_attention_decode_ring_kernel(const T* __restrict__ q, int64_t q_stride, const T* __restrict__ kv, int64_t kv_clip_stride, int Tk,
                                  const int32_t* __restrict__ d_tk, int H, T* __restrict__ out, const int32_t* __restrict__ page_table,
                                  int pt_stride, const int32_t* __restrict__ finished, int early) {
    constexpr int SEG = 8 * (int)sizeof(T);            // bytes of K (and of V) one lane owns per row
    extern __shared__ __align__(16) unsigned char sa_ring[];      // [warp][slot][K|V][lane][SEG]
    __shared__ float s_rec[SA_WARPS][SA_HG][HD + 2];
    __shared__ int32_t s_pt[SA_MAX_PAGES];
    pdl_trigger();
    const int hg = blockIdx.x, b = blockIdx.y;
    if (finished && finished[b]) { pdl_wait(); return; }
    const bool pt_smem = page_table && pt_stride <= SA_MAX_PAGES;
    if (pt_smem && (int)threadIdx.x < pt_stride) s_pt[threadIdx.x] = page_table[(int64_t)b * pt_stride + threadIdx.x];
    if (!early) pdl_wait();
    if (pt_smem) __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (d_tk) Tk = *d_tk + 1;
    const int d = H * HD;
    const int col = hg * SA_HG * HD + lane * 8;
    const bool active = col < d;
    const T* kvb = kv + (page_table ? 0 : (int64_t)b * kv_clip_stride) + (active ? col : 0);
    const int32_t* ptb = page_table ? (pt_smem ? s_pt : page_table + (int64_t)b * pt_stride) : nullptr;
    auto row_ptr = [&](int r) -> const T* {
        const int64_t pr = ptb ? (int64_t)ptb[r / TW_KV_PAGE] * TW_KV_PAGE + r % TW_KV_PAGE : (int64_t)r;
        return kvb + pr * 2 * d;
    };
    unsigned char* my = sa_ring + ((size_t)warp * SA_RING * 2 * 32 + lane) * SEG;       // + (slot * 2 + kv) * 32 * SEG
    auto issue = [&](int i) {              // i-th row of this warp (row warp + i * SA_WARPS) into slot i % SA_RING; one group
        if (active) {
            const T* rp = row_ptr(warp + i * SA_WARPS);
            unsigned char* dst = my + (size_t)((i % SA_RING) * 2) * 32 * SEG;
#pragma unroll
            for (int o = 0; o < SEG; o += 16) {
                sa_cp_async16(dst + o, reinterpret_cast<const unsigned char*>(rp) + o);
                sa_cp_async16(dst + 32 * SEG + o, reinterpret_cast<const unsigned char*>(rp + d) + o);
            }
        }
        sa_cp_commit();
    };
    float qf[8], of[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { qf[e] = 0.0f; of[e] = 0.0f; }
    float mrun = -INFINITY, lrun = 0.0f;
    const int n_old = early ? Tk - 1 : Tk;                                     // rows [0, n_old) may be read before the wait
    const int n_mine = Tk > warp ? (Tk - warp + SA_WARPS - 1) / SA_WARPS : 0;     // rows of this warp
    const int n_old_mine = n_old > warp ? (n_old - warp + SA_WARPS - 1) / SA_WARPS : 0;
    int issued = 0;
    for (; issued < SA_RING && issued < n_old_mine; ++issued) issue(issued);
    if (early) {
        // rows beyond the ring: one 128-byte line per lane into L2 (lanes 0-3 the K part of this CTA's 4 heads, lanes 4-7 the V part)
        if (lane < 8 && hg * SA_HG * HD + (lane & 3) * 64 < d) {
            for (int r = warp + SA_RING * SA_WARPS; r < n_old; r += SA_WARPS) {
                const int64_t pr = ptb ? (int64_t)ptb[r / TW_KV_PAGE] * TW_KV_PAGE + r % TW_KV_PAGE : (int64_t)r;
                const T* lp = kv + (page_table ? 0 : (int64_t)b * kv_clip_stride) + pr * 2 * d + (lane >> 2) * d + hg * SA_HG * HD + (lane & 3) * 64;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(lp));
            }
        }
        pdl_wait();
    }
    if (active) {
#pragma unroll
        for (int e = 0; e < 8; ++e) qf[e] = to_f32(q[(int64_t)b * q_stride + col + e]);
    }
    // top the ring up to SA_RING groups (the newest row may be issued now; empty groups once the warp has no more rows)
    for (int g = issued; g < SA_RING; ++g) {
        if (issued < n_mine) issue(issued++);
        else sa_cp_commit();
    }
    for (int c = 0; c < n_mine; ++c) {
        sa_cp_wait<SA_RING - 1>();
        const unsigned char* src = my + (size_t)((c % SA_RING) * 2) * 32 * SEG;
        float kf[8], vf[8];
        if (active) {
            typename Ld8<T>::Raw kraw = Ld8<T>::load(reinterpret_cast<const T*>(src));
            typename Ld8<T>::Raw vraw = Ld8<T>::load(reinterpret_cast<const T*>(src + 32 * SEG));
            Ld8<T>::unpack(kraw, kf);
            Ld8<T>::unpack(vraw, vf);
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) { kf[e] = 0.0f; vf[e] = 0.0f; }
        }
        float dot = 0.0f;
#pragma unroll
        for (int e = 0; e < 8; ++e) dot = fmaf(qf[e], kf[e], dot);
        dot += __shfl_xor_sync(0xffffffffu, dot, 1);
        dot += __shfl_xor_sync(0xffffffffu, dot, 2);
        dot += __shfl_xor_sync(0xffffffffu, dot, 4);
        const float m_new = fmaxf(mrun, dot);
        const float sc = __expf(mrun - m_new);
        const float p = __expf(dot - m_new);
        lrun = lrun * sc + p;
        mrun = m_new;
#pragma unroll
        for (int e = 0; e < 8; ++e) of[e] = fmaf(p, vf[e], of[e] * sc);
        if (issued < n_mine) issue(issued++);          // into the slot just consumed
        else sa_cp_commit();
    }
    sa_cp_wait<0>();
    {
        float* rec = s_rec[warp][lane >> 3];
        if ((lane & 7) == 0) { rec[0] = mrun; rec[1] = lrun; }
#pragma unroll
        for (int e = 0; e < 8; ++e) rec[2 + (lane & 7) * 8 + e] = of[e];
    }
    __syncthreads();
    {
        const int hh = threadIdx.x >> 6, e = threadIdx.x & 63;
        const int h = hg * SA_HG + hh;
        if (h < H) {
            float m = -INFINITY;
#pragma unroll
            for (int w = 0; w < SA_WARPS; ++w) m = fmaxf(m, s_rec[w][hh][0]);
            float l = 0.0f, o = 0.0f;
#pragma unroll
            for (int w = 0; w < SA_WARPS; ++w) {
                const float sc = (s_rec[w][hh][0] == -INFINITY) ? 0.0f : __expf(s_rec[w][hh][0] - m);
                l += s_rec[w][hh][1] * sc;
                o += s_rec[w][hh][2 + e] * sc;
            }
            out[(int64_t)b * d + h * HD + e] = from_f32<T>(o / l);
        }
    }
}

template <typename T>
void self_attention_decode(const T* q, int64_t q_stride, const T* kv, int64_t kv_clip_stride, int Tk, const int32_t* d_tk, int B, int H,
                           T* out, cudaStream_t st, const int32_t* page_table, int pt_stride, const int32_t* finished, int variant) {
    dim3 grid(ceil_div(H, SA_HG), B);
    // early: old cache rows are fetched before the programmatic-dependency wait (only inside the decode step, where the row count
    // comes from the device-side position and rows below it are older than the previous kernel); TWB200_SA_EARLY=0 switches it off
    static const bool early_on = !(getenv("TWB200_SA_EARLY") && atoi(getenv("TWB200_SA_EARLY")) == 0);
    // ring variant (cp.async into shared memory, 8 rows in flight per warp all the time): bf16 default; TWB200_SA_RING=0 / 1 forces
    static const int ring_env = getenv("TWB200_SA_RING") ? atoi(getenv("TWB200_SA_RING")) : -1;
    const bool ring = variant == SA_VARIANT_RING || (variant == SA_VARIANT_DEFAULT && (ring_env >= 0 ? ring_env != 0 : sizeof(T) == 2));
    if (ring) {
        constexpr int smem = SA_WARPS * SA_RING * 2 * 32 * 8 * (int)sizeof(T);
        static bool attr_set = false;
        if (!attr_set) {
            cudaFuncSetAttribute(self_attention_decode_ring_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
            attr_set = true;
        }
        launch_k(self_attention_decode_ring_kernel<T>, grid, dim3(SA_WARPS * 32), smem, st, q, q_stride, kv, kv_clip_stride, Tk, d_tk, H, out,
                 page_table, pt_stride, finished, (early_on && d_tk) ? 1 : 0);
        return;
    }
    launch_k(self_attention_decode_kernel<T, 4>, grid, dim3(SA_WARPS * 32), 0, st, q, q_stride, kv, kv_clip_stride, Tk, d_tk, H, out,
             page_table, pt_stride, finished, (early_on && d_tk) ? 1 : 0);
}
template void self_attention_decode<float>(const float*, int64_t, const float*, int64_t, int, const int32_t*, int, int, float*,
                                           cudaStream_t, const int32_t*, int, const int32_t*, int);
template void self_attention_decode<__nv_bfloat16>(const __nv_bfloat16*, int64_t, const __nv_bfloat16*, int64_t, int, const int32_t*,
                                                   int, int, __nv_bfloat16*, cudaStream_t, const int32_t*, int, const int32_t*, int);

static int g_da_sm_dev = 0;       // SMs of the device: sizes the partial-record workspace
static int g_da_sm_count = 0;     // CTAs of the stream kernel = SMs the launching stream may use (decode_attention_set_sms)
size_t decode_attention_partial_floats(int B, int H) {
    if (g_da_sm_dev == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&g_da_sm_dev, cudaDevAttrMultiProcessorCount, dev);
        if (g_da_sm_dev <= 0) g_da_sm_dev = 148;
        if (g_da_sm_count == 0) g_da_sm_count = g_da_sm_dev;
    }
    return (size_t)(g_da_sm_dev + B) * H * DA_PSTRIDE;
}
int decode_attention_set_sms(int n) {
    (void)decode_attention_partial_floats(1, 1);
    const int prev = g_da_sm_count;
    g_da_sm_count = (n > 0 && n < g_da_sm_dev) ? n : g_da_sm_dev;
    return prev;
}

template <typename T>
void decode_attention(const T* q, int64_t q_stride, const T* kv, int64_t kv_clip_stride, int Tk, const int32_t* d_tk, int B, int H,
                      float* partial, T* out, cudaStream_t st, cudaEvent_t ev0, cudaEvent_t ev1, const int32_t* active,
                      const int32_t* n_active) {
    (void)decode_attention_partial_floats(B, H);
    static const int env_stages = getenv("TWB200_DA_STAGES") ? atoi(getenv("TWB200_DA_STAGES")) : 0;      // tuning knob
    DaPlan p = da_plan(B * Tk, H, (int)sizeof(T), g_da_sm_count, env_stages >= 2 ? env_stages : DA_MAX_STAGES, DA_WARPS);
    if (d_tk || active) p.G = g_da_sm_count;     // row count only known on the device: launch every CTA
    static bool attr_set[2] = {false, false};
    const int which = sizeof(T) == 4 ? 0 : 1;
    if (!attr_set[which]) {
        cudaFuncSetAttribute(decode_attention_stream<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
        attr_set[which] = true;
    }
    if (ev0) cudaEventRecord(ev0, st);
    const int kv_static = d_tk ? 0 : 1;
    launch_k(decode_attention_stream<T>, dim3(p.G), dim3((DA_WARPS + 1) * 32), p.smem, st, q, q_stride, kv, kv_clip_stride, Tk, d_tk, B, H,
             p.stages, kv_static, partial, active, n_active);
    if (ev1) cudaEventRecord(ev1, st);
    // measured (A/B, large-v3, 64 clips): 256-thread CTAs (4 heads) 1222.7 ms per decode vs 1229.8 ms with 64-thread CTAs
    launch_k(decode_attention_combine<T, 4>, dim3(ceil_div(H, 4), B), dim3(HD * 4), 0, st, partial, Tk, d_tk, B, p.G, H, out, active, n_active);
}
template void decode_attention<float>(const float*, int64_t, const float*, int64_t, int, const int32_t*, int, int, float*, float*,
                                      cudaStream_t, cudaEvent_t, cudaEvent_t, const int32_t*, const int32_t*);
template void decode_attention<__nv_bfloat16>(const __nv_bfloat16*, int64_t, const __nv_bfloat16*, int64_t, int, const int32_t*, int, int,
                                              float*, __nv_bfloat16*, cudaStream_t, cudaEvent_t, cudaEvent_t, const int32_t*, const int32_t*);

}  // namespace tw
