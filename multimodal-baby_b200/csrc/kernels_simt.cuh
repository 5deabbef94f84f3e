// HBM-/L2-bound SIMT kernels of the CVCL contrastive path (sm_100a):
//   K1  length-masked embedding-bag mean + L2-norm (flat), per-token gather + norm (spatial)
//   K4b merge of the per-tile online-softmax partials -> loss / accuracy / entropy / LSE
//   K5e embedding-table gradient scatter
//   K7  n-way cosine evaluation (fp32 end to end, first-index argmax)
//   casts / transposes feeding the tensor-core GEMMs
// Coalescing rule used throughout: one warp owns one row of E contiguous floats and moves it as
// 16-byte vectors (lane-contiguous float4), so every request is a full 512-byte line group.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>
#include "gemm_sm100.cuh"   // RowStat
#include "host_util.h"

namespace cvcl {

constexpr int kMaxVec = 8;            // E <= 32 lanes * 4 floats * kMaxVec = 1024

// launch with programmatic stream serialization: the kernel's blocks may be scheduled while the
// previous kernel drains; every kernel here starts with griddepcontrol.wait, so this is safe.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ void store_bf16x4(__nv_bfloat16* dst, float4 v) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 q; q.x = *reinterpret_cast<uint32_t*>(&a); q.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(dst) = q;
}

// --------------------------------------------------------------------------------------
// K1: text encoder, embedding branch.  reference: multimodal.py:496-503 (+ :743 normalise)
//   flat      : feat[b] = normalise( sum_l table[ids[b,l]] / len[b] )
//   per_token : tok[b,l] = normalise(table[ids[b,l]])           (spatial text features, :498)
//               pooled[b] = sum_l tok[b,l] * pool_scale / len[b] (spatial "mean" similarity, :765-770)
// All L positions are visited in order; id 0 (<pad>) is skipped because nn.Embedding(padding_idx=0)
// keeps that row at exactly zero, so the sum is unchanged.  ids outside [0,V) set *status.
// --------------------------------------------------------------------------------------
struct TextFwdParams {
    const long long* ids;      // [B, L] int64
    const long long* lens;     // [B]    int64
    const float* table;        // [V, E] fp32
    int B, L, E, V;
    int normalize;
    int per_token;             // 0: flat, 1: spatial
    float pool_scale;          // per_token: 1/(H*W)
    float* feat_f32;           // [B, E]          (nullable)
    __nv_bfloat16* feat_bf16;  int ld_bf16;     // [B, ld]  (nullable)
    float* inv_norm;           // flat: [B]; per_token: [B*L]   (nullable)
    float* tok_f32;            // per_token: [B*L, E]  (nullable)
    __nv_bfloat16* tok_bf16;   // per_token: [B*L, E]  (nullable)
    int* status;               // set to 1 on an out-of-range id (nullable)
};

__global__ void __launch_bounds__(128) text_encoder_fwd_kernel(const TextFwdParams p) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= p.B) return;
    const int b = warp;
    const int nch = (p.E + 127) >> 7;          // float4 chunks per lane; tail chunk is lane-masked
    constexpr int kInFlight = 4;               // token rows gathered before they are consumed
    float4 acc[kMaxVec];
#pragma unroll
    for (int c = 0; c < kMaxVec; ++c) acc[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    const long long* idrow = p.ids + static_cast<size_t>(b) * p.L;
    for (int l0 = 0; l0 < p.L; l0 += 32) {
        // one coalesced load of up to 32 ids, then broadcast by shuffle
        long long my_id = (l0 + lane < p.L) ? __ldg(idrow + l0 + lane) : 0;
        if (my_id < 0 || my_id >= p.V) { if (p.status) atomicExch(p.status, 1); my_id = 0; }
        const int nl = min(32, p.L - l0);
        if (!p.per_token) {
            // flat: only non-pad tokens matter; compact them so the gathers stay dense
            unsigned live = __ballot_sync(0xffffffffu, my_id != 0 && lane < nl);
            while (live) {
                int src_lane[kInFlight]; int n = 0;
#pragma unroll
                for (int k = 0; k < kInFlight; ++k) {
                    src_lane[k] = -1;
                    if (live) { src_lane[k] = __ffs(live) - 1; live &= live - 1; ++n; }
                }
                float4 r[kInFlight][4];
#pragma unroll
                for (int k = 0; k < kInFlight; ++k) {
                    const long long id = __shfl_sync(0xffffffffu, my_id, src_lane[k] < 0 ? 0 : src_lane[k]);
                    const float4* src = reinterpret_cast<const float4*>(p.table + static_cast<size_t>(id) * p.E);
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        r[k][c] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (src_lane[k] >= 0 && c < nch && (c * 32 + lane) * 4 < p.E) r[k][c] = __ldg(src + c * 32 + lane);
                    }
                }
#pragma unroll
                for (int k = 0; k < kInFlight; ++k)        // position order, as sum(dim=1) does
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        acc[c].x += r[k][c].x; acc[c].y += r[k][c].y; acc[c].z += r[k][c].z; acc[c].w += r[k][c].w;
                    }
                if (nch > 4) {                               // E > 512: remaining chunks, same tokens
#pragma unroll
                    for (int k = 0; k < kInFlight; ++k) {
                        if (src_lane[k] < 0) continue;
                        const long long id = __shfl_sync(0xffffffffu, my_id, src_lane[k]);
                        const float4* src = reinterpret_cast<const float4*>(p.table + static_cast<size_t>(id) * p.E);
#pragma unroll
                        for (int c = 4; c < kMaxVec; ++c)
                            if (c < nch && (c * 32 + lane) * 4 < p.E) {
                                const float4 v = __ldg(src + c * 32 + lane);
                                acc[c].x += v.x; acc[c].y += v.y; acc[c].z += v.z; acc[c].w += v.w;
                            }
                    }
                }
                (void)n;
            }
        } else {
            // per token: tok = normalise(row).  Pads (id 0) are exact zero rows: written when the token output is
            // wanted, never fetched.  Live tokens go in groups of four whose rows are in flight together (one
            // dependent round trip per token made this the slowest kernel of the spatial step: 81 us at B = 1024).
            const unsigned in_range = nl == 32 ? 0xffffffffu : ((1u << nl) - 1u);
            unsigned live = __ballot_sync(0xffffffffu, my_id != 0 && lane < nl);
            if (p.tok_f32 || p.tok_bf16 || p.inv_norm) {
                unsigned pad = ~live & in_range;
                const float pad_inv = 1.f / (p.normalize ? fmaxf(0.f, 1e-12f) : 1.f);
                while (pad) {
                    const int k = __ffs(pad) - 1; pad &= pad - 1;
                    const size_t tok = static_cast<size_t>(b) * p.L + l0 + k;
                    if (lane == 0 && p.inv_norm) p.inv_norm[tok] = pad_inv;
#pragma unroll
                    for (int c = 0; c < kMaxVec; ++c) {
                        if (c < nch && (c * 32 + lane) * 4 < p.E) {
                            const size_t off = tok * p.E + (c * 32 + lane) * 4;
                            if (p.tok_f32) *reinterpret_cast<float4*>(p.tok_f32 + off) = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (p.tok_bf16) *reinterpret_cast<uint2*>(p.tok_bf16 + off) = make_uint2(0u, 0u);
                        }
                    }
                }
            }
            constexpr int kG = 4;
            while (live) {
                int pos[kG];
#pragma unroll
                for (int k = 0; k < kG; ++k) {
                    pos[k] = -1;
                    if (live) { pos[k] = __ffs(live) - 1; live &= live - 1; }
                }
                float4 r[kG][kMaxVec];
#pragma unroll
                for (int k = 0; k < kG; ++k) {
                    const long long id = __shfl_sync(0xffffffffu, my_id, pos[k] < 0 ? 0 : pos[k]);
                    const float4* src = reinterpret_cast<const float4*>(p.table + static_cast<size_t>(id) * p.E);
#pragma unroll
                    for (int c = 0; c < kMaxVec; ++c) {
                        r[k][c] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (pos[k] >= 0 && c < nch && (c * 32 + lane) * 4 < p.E) r[k][c] = __ldg(src + c * 32 + lane);
                    }
                }
                float ssq[kG];
#pragma unroll
                for (int k = 0; k < kG; ++k) {
                    ssq[k] = 0.f;
#pragma unroll
                    for (int c = 0; c < kMaxVec; ++c)
                        ssq[k] += r[k][c].x * r[k][c].x + r[k][c].y * r[k][c].y + r[k][c].z * r[k][c].z + r[k][c].w * r[k][c].w;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1)                     // four independent butterfly chains
#pragma unroll
                    for (int k = 0; k < kG; ++k) ssq[k] += __shfl_xor_sync(0xffffffffu, ssq[k], o);
#pragma unroll
                for (int k = 0; k < kG; ++k) {                       // position order, as sum(dim=1) does
                    if (pos[k] < 0) continue;
                    const size_t tok = static_cast<size_t>(b) * p.L + l0 + pos[k];
                    const float denom = p.normalize ? fmaxf(sqrtf(ssq[k]), 1e-12f) : 1.f;
                    // one reciprocal per token, then multiplies (the reference divides element-wise: at most 1 ulp
                    // apart; 16 IEEE divisions per lane and token were two thirds of this kernel's instructions)
                    const float rinv = 1.f / denom;
                    if (lane == 0 && p.inv_norm) p.inv_norm[tok] = rinv;
#pragma unroll
                    for (int c = 0; c < kMaxVec; ++c) {
                        if (c < nch && (c * 32 + lane) * 4 < p.E) {
                            float4 t = make_float4(r[k][c].x * rinv, r[k][c].y * rinv, r[k][c].z * rinv, r[k][c].w * rinv);
                            const size_t off = tok * p.E + (c * 32 + lane) * 4;
                            if (p.tok_f32) *reinterpret_cast<float4*>(p.tok_f32 + off) = t;
                            if (p.tok_bf16) store_bf16x4(p.tok_bf16 + off, t);
                            acc[c].x += t.x; acc[c].y += t.y; acc[c].z += t.z; acc[c].w += t.w;
                        }
                    }
                }
            }
        }
    }
    const float flen = static_cast<float>(__ldg(p.lens + b));
    float ssq = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxVec; ++c) {
        if (!p.per_token) {
            acc[c].x /= flen; acc[c].y /= flen; acc[c].z /= flen; acc[c].w /= flen;
        } else {
            const float sc = p.pool_scale;
            acc[c].x = acc[c].x * sc / flen; acc[c].y = acc[c].y * sc / flen;
            acc[c].z = acc[c].z * sc / flen; acc[c].w = acc[c].w * sc / flen;
        }
        ssq += acc[c].x * acc[c].x + acc[c].y * acc[c].y + acc[c].z * acc[c].z + acc[c].w * acc[c].w;
    }
    float denom = 1.f;
    if (!p.per_token) {
        ssq = warp_sum(ssq);
        denom = p.normalize ? fmaxf(sqrtf(ssq), 1e-12f) : 1.f;
        if (lane == 0 && p.inv_norm) p.inv_norm[b] = 1.f / denom;
    }
#pragma unroll
    for (int c = 0; c < kMaxVec; ++c) {
        const int e = (c * 32 + lane) * 4;
        if (c < nch && e < p.E) {
            float4 t = make_float4(acc[c].x / denom, acc[c].y / denom, acc[c].z / denom, acc[c].w / denom);
            if (p.feat_f32) *reinterpret_cast<float4*>(p.feat_f32 + static_cast<size_t>(b) * p.E + e) = t;
            if (p.feat_bf16) store_bf16x4(p.feat_bf16 + static_cast<size_t>(b) * p.ld_bf16 + e, t);
        }
    }
}

// K1, flat, small batches (E <= 512): one 128-thread block per utterance instead of one warp.  Warp w
// owns the 128-column slice w (one float4 per lane), so 8 token rows are in flight per lane and an
// utterance's rows arrive in one or two round trips instead of len/4: at B = 512 the warp-per-utterance
// form is bound by those serial round trips (512 warps on 148 SMs), not by bandwidth.  Per element the
// additions happen in the same (position) order as in the kernel above.
__global__ void __launch_bounds__(128) text_encoder_flat_wide_kernel(const TextFwdParams p) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int b = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e = (warp * 32 + lane) * 4;
    const bool col_ok = e < p.E;
    constexpr int kInFlight = 8;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    const long long* idrow = p.ids + static_cast<size_t>(b) * p.L;
    for (int l0 = 0; l0 < p.L; l0 += 32) {
        long long my_id = (l0 + lane < p.L) ? __ldg(idrow + l0 + lane) : 0;
        if (my_id < 0 || my_id >= p.V) { if (p.status) atomicExch(p.status, 1); my_id = 0; }
        const int nl = min(32, p.L - l0);
        unsigned live = __ballot_sync(0xffffffffu, my_id != 0 && lane < nl);
        while (live) {
            float4 r[kInFlight];
#pragma unroll
            for (int k = 0; k < kInFlight; ++k) {
                r[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (live) {
                    const int src_lane = __ffs(live) - 1;
                    live &= live - 1;
                    const long long id = __shfl_sync(0xffffffffu, my_id, src_lane);
                    if (col_ok) r[k] = __ldg(reinterpret_cast<const float4*>(p.table + static_cast<size_t>(id) * p.E + e));
                }
            }
#pragma unroll
            for (int k = 0; k < kInFlight; ++k) {           // position order, as sum(dim=1) does
                acc.x += r[k].x; acc.y += r[k].y; acc.z += r[k].z; acc.w += r[k].w;
            }
        }
    }
    const float flen = static_cast<float>(__ldg(p.lens + b));
    acc.x /= flen; acc.y /= flen; acc.z /= flen; acc.w /= flen;
    // the row sum of squares is reduced in the order of the warp-per-utterance kernel: per lane over its
    // 4 chunks (= the 4 warps here), then the butterfly over lanes
    float part = acc.x * acc.x + acc.y * acc.y + acc.z * acc.z + acc.w * acc.w;
    __shared__ float s_part[4][32];
    s_part[warp][lane] = part;
    __syncthreads();
    float ssq = ((0.f + s_part[0][lane]) + s_part[1][lane]) + s_part[2][lane] + s_part[3][lane];
    ssq = warp_sum(ssq);
    const float denom = p.normalize ? fmaxf(sqrtf(ssq), 1e-12f) : 1.f;
    if (threadIdx.x == 0 && p.inv_norm) p.inv_norm[b] = 1.f / denom;
    if (col_ok) {
        const float4 t = make_float4(acc.x / denom, acc.y / denom, acc.z / denom, acc.w / denom);
        if (p.feat_f32) *reinterpret_cast<float4*>(p.feat_f32 + static_cast<size_t>(b) * p.E + e) = t;
        if (p.feat_bf16) store_bf16x4(p.feat_bf16 + static_cast<size_t>(b) * p.ld_bf16 + e, t);
    }
}

// plain row gather table[ids] -> [B*L, E] fp32: the `text_outputs` tensor the reference API
// returns (multimodal.py:496,575,584).  One warp per token row.
__global__ void __launch_bounds__(256) embedding_gather_kernel(const long long* ids, const float* table,
                                                               float* out, int n_tok, int E, int V) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= n_tok) return;
    long long id = __ldg(ids + warp);
    if (id < 0 || id >= V) id = 0;
    const float4* src = reinterpret_cast<const float4*>(table + static_cast<size_t>(id) * E);
    float4* dst = reinterpret_cast<float4*>(out + static_cast<size_t>(warp) * E);
    for (int c = lane; c < (E >> 2); c += 32) dst[c] = __ldg(src + c);
}

// --------------------------------------------------------------------------------------
// K5e: d table[v] += g[b] for every position l with ids[b,l] = v != 0   (flat)
//      per_token: g is [B*L, E] (one gradient row per token)
// g already contains the normalise-backward and the 1/len factor.  Row 0 never receives a
// gradient (nn.Embedding padding_idx=0, multimodal.py:311-312).  fp32 vector atomics.
// --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) embedding_scatter_add_kernel(const long long* ids, const float* g,
                                                                    float* dtable, int B, int L, int E,
                                                                    int V, int per_token) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;      // one warp per token position
    const int lane = threadIdx.x & 31;
    if (warp >= B * L) return;
    const long long id = __ldg(ids + warp);
    if (id <= 0 || id >= V) return;
    const int row = per_token ? warp : warp / L;
    const float4* src = reinterpret_cast<const float4*>(g + static_cast<size_t>(row) * E);
    float4* dst = reinterpret_cast<float4*>(dtable + static_cast<size_t>(id) * E);
    for (int c = lane; c < (E >> 2); c += 32) atomicAdd(dst + c, __ldg(src + c));
}

// spatial text backward: per token recompute tok = normalise(table[id]) and apply
//   g_tok = dtok[b,l] (+ dpool[b] * pool_scale / len[b])      (either input nullable)
//   d e   = (g_tok - tok <tok, g_tok>) * inv_norm             (F.normalize backward)
// then scatter-add into d table.  One warp per token.
__global__ void __launch_bounds__(256) text_token_bwd_kernel(const long long* ids, const long long* lens,
                                                             const float* table, const float* dtok,
                                                             const float* dpool, float pool_scale,
                                                             float* dtable, int B, int L, int E, int V,
                                                             int normalize) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= B * L) return;
    const long long id = __ldg(ids + warp);
    if (id <= 0 || id >= V) return;
    const int b = warp / L;
    const int nch = (E + 127) >> 7;
    const float4* src = reinterpret_cast<const float4*>(table + static_cast<size_t>(id) * E);
    const float ps = dpool ? pool_scale / static_cast<float>(__ldg(lens + b)) : 0.f;
    float4 e[kMaxVec], g[kMaxVec];
    float ssq = 0.f, dot = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxVec; ++c) {
        e[c] = make_float4(0.f, 0.f, 0.f, 0.f); g[c] = e[c];
        if (c < nch && (c * 32 + lane) * 4 < E) {
            e[c] = __ldg(src + c * 32 + lane);
            if (dtok) g[c] = __ldg(reinterpret_cast<const float4*>(dtok + static_cast<size_t>(warp) * E) + c * 32 + lane);
            if (dpool) {
                float4 q = __ldg(reinterpret_cast<const float4*>(dpool + static_cast<size_t>(b) * E) + c * 32 + lane);
                g[c].x = fmaf(q.x, ps, g[c].x); g[c].y = fmaf(q.y, ps, g[c].y);
                g[c].z = fmaf(q.z, ps, g[c].z); g[c].w = fmaf(q.w, ps, g[c].w);
            }
        }
        ssq += e[c].x * e[c].x + e[c].y * e[c].y + e[c].z * e[c].z + e[c].w * e[c].w;
        dot += e[c].x * g[c].x + e[c].y * g[c].y + e[c].z * g[c].z + e[c].w * g[c].w;
    }
    ssq = warp_sum(ssq); dot = warp_sum(dot);
    float inv = 1.f, k = 0.f;
    if (normalize) {
        const float denom = fmaxf(sqrtf(ssq), 1e-12f);
        inv = 1.f / denom;
        k = dot * inv * inv * inv;         // <tok,g> * tok * inv = e * dot / denom^3
        if (sqrtf(ssq) < 1e-12f) k = 0.f;  // clamp active: y = x / eps, dy/dx = 1/eps
    }
    float4* dst = reinterpret_cast<float4*>(dtable + static_cast<size_t>(id) * E);
#pragma unroll
    for (int c = 0; c < kMaxVec; ++c) {
        if (c < nch && (c * 32 + lane) * 4 < E) {
            float4 o = make_float4(g[c].x * inv - e[c].x * k, g[c].y * inv - e[c].y * k,
                                   g[c].z * inv - e[c].z * k, g[c].w * inv - e[c].w * k);
            atomicAdd(dst + c * 32 + lane, o);
        }
    }
}

// --------------------------------------------------------------------------------------
// K4b: merge per-tile online-softmax partials; emits per-row LSE and the five scalars of
// multimodal.py:808-818.  Deterministic: each block writes its partial sums, the last block to
// finish (atomic ticket) adds them in block order.
// out[0..4] = loss, image_accuracy, text_accuracy, image_entropy, text_entropy
// (scaled by inv_rows = 1/B_global so that shards can be summed across ranks).
// --------------------------------------------------------------------------------------
struct FinalizeParams {
    const RowStat* part[2]; int m_pad[2]; int n_tiles[2]; int M[2];
    const float* diag[2];
    int diag_off[2];
    float* lse[2];               // [M]
    int* argmax[2];              // [M] (nullable)
    float inv_rows;              // 1 / B_global
    float* block_part;           // [gridDim.x * 6]
    unsigned int* ticket;        // zero-initialised, reset by the kernel
    float* out;                  // [8]
};

__global__ void __launch_bounds__(256) infonce_finalize_kernel(const FinalizeParams p) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    __shared__ float red[6][8];
    __shared__ bool is_last;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    float ce[2] = {0.f, 0.f}, ent[2] = {0.f, 0.f}, acc[2] = {0.f, 0.f};
    const int total = p.M[0] + p.M[1];
    if (tid < total) {
        const int z = tid < p.M[0] ? 0 : 1;
        const int m = z ? tid - p.M[0] : tid;
        const RowStat* base = p.part[z] + m;
        const size_t stride = p.m_pad[z];
        const int nt = p.n_tiles[z];
        float mx = -INFINITY, l = 0.f, a = 0.f; int arg = 0x7fffffff;
        // one pass, 4 independent loads in flight; online merge (strict >: the first tile wins ties)
        for (int t0 = 0; t0 < nt; t0 += 4) {
            RowStat rs[4];
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (t0 + k < nt) rs[k] = base[static_cast<size_t>(t0 + k) * stride];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (t0 + k < nt) {
                    if (rs[k].m > mx) {
                        const float w = __expf(mx - rs[k].m);          // mx = -inf -> 0
                        l *= w; a *= w; mx = rs[k].m; arg = rs[k].arg;
                        l += rs[k].l; a += rs[k].a;
                    } else {
                        const float w = __expf(rs[k].m - mx);
                        l = fmaf(rs[k].l, w, l); a = fmaf(rs[k].a, w, a);
                    }
                }
            }
        }
        const float lse = mx + logf(l);
        p.lse[z][m] = lse;
        if (p.argmax[z]) p.argmax[z][m] = arg;
        ce[z] = lse - p.diag[z][m];
        ent[z] = lse - a / l;
        acc[z] = (arg == m + p.diag_off[z]) ? 1.f : 0.f;
    }
    float v[6] = {ce[0], ce[1], ent[0], ent[1], acc[0], acc[1]};
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 6; ++i) { v[i] = warp_sum(v[i]); if (lane == 0) red[i][w] = v[i]; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 0; i < 6; ++i) {
            float s = 0.f;
            for (int k = 0; k < (blockDim.x >> 5); ++k) s += red[i][k];
            p.block_part[blockIdx.x * 6 + i] = s;
        }
        __threadfence();
        const unsigned int t = atomicAdd(p.ticket, 1u);
        is_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last && threadIdx.x < 32) {          // deterministic: fixed lane-strided order + tree
        __threadfence();
        float s[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (unsigned int b = threadIdx.x; b < gridDim.x; b += 32)
#pragma unroll
            for (int i = 0; i < 6; ++i) s[i] += p.block_part[b * 6 + i];
#pragma unroll
        for (int i = 0; i < 6; ++i) s[i] = warp_sum(s[i]);
        if (threadIdx.x == 0) {
            p.out[0] = (s[0] + s[1]) * 0.5f * p.inv_rows;
            p.out[1] = s[4] * p.inv_rows;
            p.out[2] = s[5] * p.inv_rows;
            p.out[3] = s[2] * p.inv_rows;
            p.out[4] = s[3] * p.inv_rows;
            *p.ticket = 0u;
        }
    }
}

// --------------------------------------------------------------------------------------
// K7: Labeled-S style n-way evaluation, fp32 end to end.
// reference: multimodal_lit.py:466-511 / eval.py:196-214: per trial the 4 frame embeddings and the
// label embedding are L2-normalised, dotted, scaled; pred = argmax (first maximal index).
// One warp per trial; E <= 1024.
// --------------------------------------------------------------------------------------
// per-trial arithmetic of K7 on register-resident rows (x: kWays candidate rows, t: label row; 4 float4 per
// lane each): screen on raw dots, exact reference arithmetic for near-ties / NaNs / requested logits.
template <int kWays>
__device__ __forceinline__ void eval_trial_from_regs(float4 (&x)[kWays][4], float4 (&t)[4], int trial, int lane,
                                                     int normalize, float scale, int* pred, float* logits) {
    float best = -INFINITY; int arg = 0;
        float tss = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) tss += t[c].x * t[c].x + t[c].y * t[c].y + t[c].z * t[c].z + t[c].w * t[c].w;
        tss = warp_sum(tss);
        if (normalize && logits == nullptr) {
            // Screen: raw sums of squares and raw dots, one division per candidate (cos = <x,t>/(|x||t|)).
            // It differs from the reference arithmetic below (element-wise x/|x| and t/|t| before the
            // products) by a few 1e-6 in the cosine at most, so it can only change the winner when the
            // two best cosines agree to 1e-4; only those trials (and NaNs) take the exact path.
            const float dt = fmaxf(sqrtf(tss), 1e-12f);
            float ss[kWays], dot[kWays];
#pragma unroll
            for (int w = 0; w < kWays; ++w) {
                ss[w] = 0.f; dot[w] = 0.f;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    ss[w] = fmaf(x[w][c].x, x[w][c].x, ss[w]); ss[w] = fmaf(x[w][c].y, x[w][c].y, ss[w]);
                    ss[w] = fmaf(x[w][c].z, x[w][c].z, ss[w]); ss[w] = fmaf(x[w][c].w, x[w][c].w, ss[w]);
                    dot[w] = fmaf(x[w][c].x, t[c].x, dot[w]); dot[w] = fmaf(x[w][c].y, t[c].y, dot[w]);
                    dot[w] = fmaf(x[w][c].z, t[c].z, dot[w]); dot[w] = fmaf(x[w][c].w, t[c].w, dot[w]);
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                for (int w = 0; w < kWays; ++w) {
                    ss[w] += __shfl_xor_sync(0xffffffffu, ss[w], o);
                    dot[w] += __shfl_xor_sync(0xffffffffu, dot[w], o);
                }
            }
            float b1 = -INFINITY, b2 = -INFINITY; int a1 = 0;
#pragma unroll
            for (int w = 0; w < kWays; ++w) {
                const float v = dot[w] / (fmaxf(sqrtf(ss[w]), 1e-12f) * dt);
                if (v > b1) { b2 = b1; b1 = v; a1 = w; } else if (v > b2) { b2 = v; }
            }
            if (b1 - b2 > 1e-4f) {            // false for NaN / inf: those go through the exact path
                if (lane == 0) pred[trial] = a1;
                return;
            }
        }
        if (normalize) {
            const float d = fmaxf(sqrtf(tss), 1e-12f);
#pragma unroll
            for (int c = 0; c < 4; ++c) { t[c].x /= d; t[c].y /= d; t[c].z /= d; t[c].w /= d; }
        }
#pragma unroll
        for (int w = 0; w < kWays; ++w) {
            float ss = 0.f;
#pragma unroll
            for (int c = 0; c < 4; ++c)
                ss += x[w][c].x * x[w][c].x + x[w][c].y * x[w][c].y + x[w][c].z * x[w][c].z + x[w][c].w * x[w][c].w;
            float d = 1.f;
            if (normalize) d = fmaxf(sqrtf(warp_sum(ss)), 1e-12f);
            float dot = 0.f;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                dot = fmaf(x[w][c].x / d, t[c].x, dot); dot = fmaf(x[w][c].y / d, t[c].y, dot);
                dot = fmaf(x[w][c].z / d, t[c].z, dot); dot = fmaf(x[w][c].w / d, t[c].w, dot);
            }
            dot = warp_sum(dot) * scale;
            if (logits && lane == 0) logits[static_cast<size_t>(trial) * kWays + w] = dot;
            if (dot > best) { best = dot; arg = w; }
        }
    if (lane == 0) pred[trial] = arg;
}

template <int kWays>      // kWays > 0: all candidate rows are fetched before any reduction (MLP)
__global__ void __launch_bounds__(256) eval_nway_kernel(const float* img, const float* txt,
                                                        const int* txt_index, int n_trials, int n_way,
                                                        int E, int normalize, float scale, int* pred,
                                                        float* logits) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= n_trials) return;
    const int ti = txt_index ? __ldg(txt_index + warp) : warp;
    const float4* tsrc = reinterpret_cast<const float4*>(txt + static_cast<size_t>(ti) * E);
    float best = -INFINITY; int arg = 0;
    if constexpr (kWays > 0) {
        // E <= 512: 4 float4 per lane per row; kWays image rows + the text row in flight together
        float4 t[4], x[kWays][4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            t[c] = make_float4(0.f, 0.f, 0.f, 0.f);
            if ((c * 32 + lane) * 4 < E) t[c] = __ldg(tsrc + c * 32 + lane);
        }
#pragma unroll
        for (int w = 0; w < kWays; ++w) {
            const float4* isrc = reinterpret_cast<const float4*>(img + (static_cast<size_t>(warp) * kWays + w) * E);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                x[w][c] = make_float4(0.f, 0.f, 0.f, 0.f);
                if ((c * 32 + lane) * 4 < E) x[w][c] = __ldg(isrc + c * 32 + lane);
            }
        }
        eval_trial_from_regs<kWays>(x, t, warp, lane, normalize, scale, pred, logits);
        return;
    } else {
        const int nch = (E + 127) >> 7;
        float4 t[kMaxVec];
        float tss = 0.f;
#pragma unroll
        for (int c = 0; c < kMaxVec; ++c) {
            t[c] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (c < nch && (c * 32 + lane) * 4 < E) t[c] = __ldg(tsrc + c * 32 + lane);
            tss += t[c].x * t[c].x + t[c].y * t[c].y + t[c].z * t[c].z + t[c].w * t[c].w;
        }
        if (normalize) {
            const float d = fmaxf(sqrtf(warp_sum(tss)), 1e-12f);
#pragma unroll
            for (int c = 0; c < kMaxVec; ++c) { t[c].x /= d; t[c].y /= d; t[c].z /= d; t[c].w /= d; }
        }
        for (int w = 0; w < n_way; ++w) {
            const float4* isrc = reinterpret_cast<const float4*>(img + (static_cast<size_t>(warp) * n_way + w) * E);
            float4 x[kMaxVec];
            float ss = 0.f;
#pragma unroll
            for (int c = 0; c < kMaxVec; ++c) {
                x[c] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (c < nch && (c * 32 + lane) * 4 < E) x[c] = __ldg(isrc + c * 32 + lane);
                ss += x[c].x * x[c].x + x[c].y * x[c].y + x[c].z * x[c].z + x[c].w * x[c].w;
            }
            float d = 1.f;
            if (normalize) d = fmaxf(sqrtf(warp_sum(ss)), 1e-12f);
            float dot = 0.f;
#pragma unroll
            for (int c = 0; c < kMaxVec; ++c) {
                dot = fmaf(x[c].x / d, t[c].x, dot); dot = fmaf(x[c].y / d, t[c].y, dot);
                dot = fmaf(x[c].z / d, t[c].z, dot); dot = fmaf(x[c].w / d, t[c].w, dot);
            }
            dot = warp_sum(dot) * scale;
            if (logits && lane == 0) logits[static_cast<size_t>(warp) * n_way + w] = dot;
            if (dot > best) { best = dot; arg = w; }
        }
    }
    if (lane == 0) pred[warp] = arg;
}

// K7, streaming form for large trial counts: persistent blocks, the candidate rows of kEvalGroup
// consecutive trials (contiguous in memory: kEvalGroup * n_way * E floats) arrive by ONE bulk async copy
// (cp.async.bulk, mbarrier complete_tx) into a ring of shared-memory stages filled by a producer warp,
// so HBM reads never pause while the consumer warps reduce: warp w owns trial w of a stage.  The
// warp-per-trial kernel above loads, then reduces, then loads again in lockstep waves (47 % of the HBM
// peak on 100 000 frames); this one keeps kStages * 32 KB per block in flight all the time.
// Arithmetic per trial is the same as eval_nway_kernel<kWays> (screen + exact path).
constexpr int kEvalGroup = 4;          // trials per stage = consumer warps
constexpr int kEvalStages = 2;

template <int kWays>
__global__ void __launch_bounds__(32 * (kEvalGroup + 1)) eval_nway_stream_kernel(
        const float* img, const float* txt, const int* txt_index, int n_trials, int E, int normalize, float scale,
        int* pred, float* logits) {
    extern __shared__ __align__(128) unsigned char eval_smem[];
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t trial_bytes = static_cast<uint32_t>(kWays) * E * 4u;
    const uint32_t stage_bytes = kEvalGroup * trial_bytes;
    uint64_t* full = reinterpret_cast<uint64_t*>(eval_smem);
    uint64_t* empty = full + kEvalStages;
    unsigned char* ring = eval_smem + 128;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kEvalStages; ++s) { ptx::mbar_init(full + s, 1); ptx::mbar_init(empty + s, kEvalGroup); }
        ptx::fence_mbar_init();
    }
    __syncthreads();
    const int n_groups = (n_trials + kEvalGroup - 1) / kEvalGroup;
    if (warp == kEvalGroup) {                      // producer warp: one elected lane issues the copies
        if (lane == 0) {
            int it = 0;
            for (int g = blockIdx.x; g < n_groups; g += gridDim.x, ++it) {
                const int s = it % kEvalStages;
                if (it >= kEvalStages) ptx::mbar_wait(empty + s, ((it / kEvalStages) - 1) & 1);
                const int t0 = g * kEvalGroup;
                const int nt = min(kEvalGroup, n_trials - t0);
                const uint32_t bytes = static_cast<uint32_t>(nt) * trial_bytes;
                ptx::mbar_arrive_expect_tx(full + s, bytes);
                ptx::bulk_load_1d(ring + static_cast<size_t>(s) * stage_bytes,
                                  img + static_cast<size_t>(t0) * kWays * E, bytes, full + s);
            }
        }
        return;
    }
    // The label row of a trial is two dependent loads away (txt_index, then the row: about 2 us of
    // latency per trial when taken in line -- ncu showed the consumer warps parked on exactly that), so it
    // is software-pipelined: the index is fetched two groups ahead, the row one group ahead.
    auto trial_of = [&](int k) -> int {
        const long long g = blockIdx.x + static_cast<long long>(k) * gridDim.x;
        return g < n_groups ? static_cast<int>(g) * kEvalGroup + warp : n_trials;
    };
    auto load_idx = [&](int trial) -> int {
        if (trial >= n_trials) return -1;
        return txt_index ? __ldg(txt_index + trial) : trial;
    };
    auto load_row = [&](int ti, float4 (&t)[4]) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            t[c] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (ti >= 0 && (c * 32 + lane) * 4 < E)
                t[c] = __ldg(reinterpret_cast<const float4*>(txt + static_cast<size_t>(ti) * E) + c * 32 + lane);
        }
    };
    float4 t_cur[4], t_nxt[4];
    load_row(load_idx(trial_of(0)), t_cur);
    int idx_nxt = load_idx(trial_of(1));
    int it = 0;
    for (int g = blockIdx.x; g < n_groups; g += gridDim.x, ++it) {
        const int s = it % kEvalStages;
        const int trial = g * kEvalGroup + warp;
        const int idx_nn = load_idx(trial_of(it + 2));
        load_row(idx_nxt, t_nxt);
        ptx::mbar_wait(full + s, (it / kEvalStages) & 1);
        if (trial < n_trials) {
            const float4* rows = reinterpret_cast<const float4*>(ring + static_cast<size_t>(s) * stage_bytes +
                                                                 static_cast<size_t>(warp) * trial_bytes);
            float4 x[kWays][4];
#pragma unroll
            for (int w = 0; w < kWays; ++w)
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    x[w][c] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if ((c * 32 + lane) * 4 < E) x[w][c] = rows[w * (E >> 2) + c * 32 + lane];
                }
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(empty + s);          // rows are in registers: release the stage
            eval_trial_from_regs<kWays>(x, t_cur, trial, lane, normalize, scale, pred, logits);
        } else {
            if (lane == 0) ptx::mbar_arrive(empty + s);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) t_cur[c] = t_nxt[c];
        idx_nxt = idx_nn;
    }
}

// --------------------------------------------------------------------------------------
// Grad-CAM attention maps for the flat head (SURVEY 8f item 4; multimodal/attention_maps.py:111-165).
// The saliency layer is layer4, followed by the global average pool and fc, so the head is linear in the
// pooled activation and d output / d act[n,c,h,w] does not depend on (h,w): no trunk backward is needed.
//   pooled[n,c] = mean_hw act[n,c,:]            u[n] = W pooled[n] + b            (:143, ResNet forward)
//   g[n] = target[n]                            or (t - y <y,t>) / ||u||, y = u/||u||   (:144-146)
//   alpha[n,c] = (W^T g[n])[c] / HW             (= grad.mean((2,3)), :114)
//   cam[n,p] = max(0, sum_c act[n,c,p] alpha[n,c])                                  (:116-119)
// fp32 throughout.  act is NCHW contiguous ([N, K, HW]).
// --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gradcam_pool_kernel(const float* act, float* pooled, long long n_rows, int HW) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const long long row = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= n_rows) return;
    const float* src = act + row * HW;
    float s = 0.f;
    for (int i = lane; i < HW; i += 32) s += __ldg(src + i);
    s = warp_sum(s);
    if (lane == 0) pooled[row] = s / static_cast<float>(HW);
}

// u[n,e] = b[e] + <pooled[n,:], W[e,:]>: one warp per output, float4 loads (K % 4 == 0)
__global__ void __launch_bounds__(256) gradcam_head_kernel(const float* pooled, const float* w, const float* bias,
                                                           float* u, int N, int E, int K) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int o = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (o >= N * E) return;
    const int n = o / E, e = o - n * E;
    const float4* a = reinterpret_cast<const float4*>(pooled + static_cast<size_t>(n) * K);
    const float4* b = reinterpret_cast<const float4*>(w + static_cast<size_t>(e) * K);
    float s = 0.f;
    for (int i = lane; i < (K >> 2); i += 32) {
        const float4 x = __ldg(a + i), y = __ldg(b + i);
        s = fmaf(x.x, y.x, s); s = fmaf(x.y, y.y, s); s = fmaf(x.z, y.z, s); s = fmaf(x.w, y.w, s);
    }
    s = warp_sum(s);
    if (lane == 0) u[o] = s + (bias ? __ldg(bias + e) : 0.f);
}

// C[m,n] = bias[n] + <A[m,:], W[n,:]>, all fp32 with fp32 FMA accumulation (the exact-mode projection head of the
// evaluation path: reference `fc` in fp32, multimodal.py:186-192).  64 x 64 output tile per 256-thread block, 4 x 4
// outputs per thread, 16-deep k slabs staged in shared memory (k-major, +1 padding); K % 4 == 0.
__global__ void __launch_bounds__(256) linear_f32_kernel(const float* A, int lda, const float* W, int ldw,
                                                         const float* bias, int M, int N, int K, float* C, int ldc) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    __shared__ float sa[16][65];
    __shared__ float sw[16][65];
    const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;             // outputs rows ty*4.., cols tx*4..
    const int lr = threadIdx.x >> 2, lk = (threadIdx.x & 3) * 4;        // loader: row lr (0..63), k offset lk
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int k0 = 0; k0 < K; k0 += 16) {
        float4 va = make_float4(0.f, 0.f, 0.f, 0.f), vw = make_float4(0.f, 0.f, 0.f, 0.f);
        if (m0 + lr < M && k0 + lk < K) va = __ldg(reinterpret_cast<const float4*>(A + static_cast<size_t>(m0 + lr) * lda + k0 + lk));
        if (n0 + lr < N && k0 + lk < K) vw = __ldg(reinterpret_cast<const float4*>(W + static_cast<size_t>(n0 + lr) * ldw + k0 + lk));
        __syncthreads();
        sa[lk][lr] = va.x; sa[lk + 1][lr] = va.y; sa[lk + 2][lr] = va.z; sa[lk + 3][lr] = va.w;
        sw[lk][lr] = vw.x; sw[lk + 1][lr] = vw.y; sw[lk + 2][lr] = vw.z; sw[lk + 3][lr] = vw.w;
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            float a[4], w[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { a[i] = sa[kk][ty * 4 + i]; w[i] = sw[kk][tx * 4 + i]; }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n < N) C[static_cast<size_t>(m) * ldc + n] = acc[i][j] + (bias ? __ldg(bias + n) : 0.f);
        }
    }
}

// dst[m,:] = src[m,:] / max(||src[m,:]||, 1e-12)  (F.normalize, fp32; one warp per row, E % 4 == 0)
__global__ void __launch_bounds__(256) normalize_rows_f32_kernel(const float* src, float* dst, long long M, int E) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const long long m = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (m >= M) return;
    const float4* p = reinterpret_cast<const float4*>(src + m * E);
    float ssq = 0.f;
    for (int i = lane; i < (E >> 2); i += 32) {
        const float4 v = __ldg(p + i);
        ssq += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    }
    ssq = warp_sum(ssq);
    const float d = fmaxf(sqrtf(ssq), 1e-12f);
    float4* q = reinterpret_cast<float4*>(dst + m * E);
    for (int i = lane; i < (E >> 2); i += 32) {
        const float4 v = __ldg(p + i);
        q[i] = make_float4(v.x / d, v.y / d, v.z / d, v.w / d);
    }
}

// per row of scores [M, N] (ld): the first maximum and its index (torch.argmax / np.argmax semantics: the lowest index
// wins ties; a NaN row entry wins like in torch).  One warp per row; merged into (best, arg) that already hold the
// result of earlier column chunks when `merge` (chunked nearest-neighbour search), col0 = index of column 0.
__global__ void __launch_bounds__(256) row_argmax_f32_kernel(const float* scores, long long ld, long long M, int N,
                                                             int col0, int merge, float* best, int* arg) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const long long m = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (m >= M) return;
    const float* row = scores + m * ld;
    float b = -INFINITY; int a = 0x7fffffff; bool nan_seen = false;
    for (int n = lane; n < N; n += 32) {
        const float v = __ldg(row + n);
        if (v != v) { if (!nan_seen) { nan_seen = true; b = v; a = n; } }
        else if (!nan_seen && (v > b || a == 0x7fffffff)) { b = v; a = n; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, b, o);
        const int oa = __shfl_xor_sync(0xffffffffu, a, o);
        const bool o_nan = ob != ob, m_nan = b != b;
        bool take;
        if (o_nan || m_nan) take = o_nan && (!m_nan || oa < a);
        else take = (ob > b) || (ob == b && oa < a);
        if (take) { b = ob; a = oa; }
    }
    if (lane == 0 && a != 0x7fffffff) {
        a += col0;
        if (merge) {
            const float pb = best[m]; const int pa = arg[m];
            const bool p_nan = pb != pb, m_nan = b != b;
            const bool keep_prev = p_nan || (!m_nan && pb >= b);         // earlier chunk = lower indices: wins ties
            if (keep_prev) { b = pb; a = pa; }
        }
        best[m] = b; arg[m] = a;
    }
}

// out[b*HW + p, e] = bias[e] + sum_k W[e,k] x[b,k,p]: the spatial 1x1-conv head in fp32 (reference Conv2d(2048, E, 1),
// multimodal.py:181-185), reading the layer4 map x [B,K,HW] in the NCHW layout the trunk emits and writing NHWC rows.
// Same tiling and fp32 FMA order as linear_f32_kernel (64 x 64 tile, 4 x 4 per thread, 16-deep k slabs); only the
// A loader differs: for a fixed k the 64 rows of a tile are consecutive locations, so each thread fetches 4 scalars
// of one row at k, k+4, k+8, k+12 (coalesced along p) instead of a float4 along k.  Row tiles run along blockIdx.x
// (B*HW reaches millions of rows).
__global__ void __launch_bounds__(256) conv1x1_f32_kernel(const float* x, const float* W, const float* bias, int M,
                                                          int N, int K, int HW, float* C) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    __shared__ float sa[16][65];
    __shared__ float sw[16][65];
    const int m0 = blockIdx.x * 64, n0 = blockIdx.y * 64;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int lr = threadIdx.x >> 2, lk = (threadIdx.x & 3) * 4;        // W loader, as linear_f32_kernel
    const int am = threadIdx.x & 63, ak = threadIdx.x >> 6;             // A loader: row am, k = ak + 4j
    const int m_a = m0 + am;
    const float* arow = nullptr;
    if (m_a < M) {
        const int b = m_a / HW, p = m_a - b * HW;
        arow = x + static_cast<size_t>(b) * K * HW + p;
    }
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int k0 = 0; k0 < K; k0 += 16) {
        float va[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + ak + 4 * j;
            va[j] = (arow && k < K) ? __ldg(arow + static_cast<size_t>(k) * HW) : 0.f;
        }
        float4 vw = make_float4(0.f, 0.f, 0.f, 0.f);
        if (n0 + lr < N && k0 + lk < K) vw = __ldg(reinterpret_cast<const float4*>(W + static_cast<size_t>(n0 + lr) * K + k0 + lk));
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; ++j) sa[ak + 4 * j][am] = va[j];
        sw[lk][lr] = vw.x; sw[lk + 1][lr] = vw.y; sw[lk + 2][lr] = vw.z; sw[lk + 3][lr] = vw.w;
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            float a[4], w[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { a[i] = sa[kk][ty * 4 + i]; w[i] = sw[kk][tx * 4 + i]; }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n < N) C[static_cast<size_t>(m) * N + n] = acc[i][j] + (bias ? __ldg(bias + n) : 0.f);
        }
    }
}

// Spatial "max" score in fp32 for evaluation (multimodal.py:771-780):
//   logit[m, c] = scale * (sum_{l < len[c]} max_p <img[m,p,:], tok[c,l,:]>) / len[c]
// Rows of a label past its length are <pad> rows, zero after the per-token normalisation, and add exactly 0 in the
// reference, so they are skipped.  Trial mode (n_way >= 1): image m is scored against label txt_index[m / n_way]
// (identity when null) and out is [M]; category mode (n_way == 0): against all C labels, out [M, C].
// One block per image.  The image's HW x E block is read from HBM once into shared memory (row stride ld4 float4,
// padded so the quarter-warps of a k-split read distinct banks); the label token rows follow in chunks of <= tt rows,
// staged in shared memory as well.  Thread (w, ks) owns work item w = (group of 4 token rows, location p) and the
// k-slice ks (float4 indices ks, ks + KS, ...): four fp32 FMA chains, then a fixed butterfly over the KS lanes of the
// item.  Maximum over the locations (NaN propagates, as torch.amax), then one thread adds the token maxima of each
// label in position order.  No atomics: a replay is bit-identical.  A label index outside [0, C) scores NaN.
struct SpatialMaxScoreParams {
    const float* img;          // [M, HW, E] fp32, normalised location features (NHWC rows)
    const float* tok;          // [C, L, E]  fp32 per-token text features
    const long long* lens;     // [C]
    const int* txt_index;      // [M / n_way] (trial mode, nullable)
    int M, HW, E, C, L, n_way;
    int tt;                    // token rows per chunk (multiple of 4)
    int ks;                    // k-split lanes per work item (power of 2 <= 32, divides E/4)
    int ld4;                   // shared-memory row stride of the image block, float4 units
    float scale;               // exp(s)
    float* out;
};

__global__ void __launch_bounds__(256) spatial_max_scores_f32_kernel(const SpatialMaxScoreParams p) {
    extern __shared__ __align__(16) unsigned char sms_smem[];
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int m = blockIdx.x;
    const int tid = threadIdx.x;
    const int E4 = p.E >> 2;
    float4* img_s = reinterpret_cast<float4*>(sms_smem);                         // [HW][ld4]
    float4* tok_s = img_s + static_cast<size_t>(p.HW) * p.ld4;                   // [tt][E4]
    float* dots = reinterpret_cast<float*>(tok_s + static_cast<size_t>(p.tt) * E4);   // [tt][HW]
    float* tmax = dots + static_cast<size_t>(p.tt) * p.HW;                       // [tt]
    int* slot_c = reinterpret_cast<int*>(tmax + p.tt);                           // [tt] label of the row
    int* slot_l = slot_c + p.tt;                                                 // [tt] position (-1: last of label)
    int* ctrl = slot_l + p.tt;                                                   // [0] rows in the chunk, [1] done

    const float4* src = reinterpret_cast<const float4*>(p.img) + static_cast<size_t>(m) * p.HW * E4;
    const int n4 = p.HW * E4;
    for (int i0 = tid; i0 < n4; i0 += 4 * 256) {                                 // 4 loads in flight per thread
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * 256;
            if (i < n4) v[u] = __ldcs(src + i);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * 256;
            if (i < n4) { const int q = i / E4; img_s[q * p.ld4 + (i - q * E4)] = v[u]; }
        }
    }

    int c_cur = 0, c_end = p.C, l_cur = 0;           // thread 0's cursor over (label, position)
    float run = 0.f;                                 // thread 0's running sum of the current label
    if (p.n_way > 0) {
        const int trial = m / p.n_way;
        c_cur = p.txt_index ? __ldg(p.txt_index + trial) : trial;
        c_end = c_cur + 1;
        if (c_cur < 0 || c_cur >= p.C) {
            if (tid == 0) p.out[m] = __int_as_float(0x7fffffff);
            return;
        }
    }
    const int ks = tid & (p.ks - 1);
    const int w = tid / p.ks;
    while (true) {
        __syncthreads();                             // previous chunk consumed (and the image block stored)
        if (tid == 0) {
            int nt = 0;
            while (nt < p.tt && c_cur < c_end) {
                const long long len = __ldg(p.lens + c_cur);
                const int n = static_cast<int>(len < 0 ? 0 : (len > p.L ? p.L : len));
                if (n == 0) {                        // no token: 0 / len as the reference computes it
                    const float v = (0.f / static_cast<float>(len)) * p.scale;
                    p.out[p.n_way > 0 ? static_cast<size_t>(m) : static_cast<size_t>(m) * p.C + c_cur] = v;
                    ++c_cur; continue;
                }
                slot_c[nt] = c_cur;
                slot_l[nt] = (l_cur == n - 1) ? -1 : l_cur;
                ++nt;
                if (++l_cur == n) { l_cur = 0; ++c_cur; }
            }
            ctrl[0] = nt; ctrl[1] = nt == 0;
        }
        __syncthreads();
        const int nt = ctrl[0];
        if (ctrl[1]) break;
        for (int i = tid; i < p.tt * E4; i += 256) {
            const int r = i / E4, e = i - r * E4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < nt) {
                const int c = slot_c[r];
                int l = slot_l[r];
                if (l < 0) {                                         // last row of its label: position len - 1
                    const long long len = __ldg(p.lens + c);
                    l = static_cast<int>(len > p.L ? p.L : len) - 1;
                }
                v = __ldg(reinterpret_cast<const float4*>(p.tok) + (static_cast<size_t>(c) * p.L + l) * E4 + e);
            }
            tok_s[i] = v;
        }
        __syncthreads();
        const int n_items = ((nt + 3) >> 2) * p.HW;
        {
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            const int g = w / p.HW, q = w - g * p.HW;
            if (w < n_items) {
                const float4* xr = img_s + q * p.ld4;
                const float4* t0 = tok_s + static_cast<size_t>(g) * 4 * E4;
                for (int i = ks; i < E4; i += p.ks) {
                    const float4 xv = xr[i];
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const float4 tv = t0[r * E4 + i];
                        acc[r] = fmaf(xv.x, tv.x, acc[r]); acc[r] = fmaf(xv.y, tv.y, acc[r]);
                        acc[r] = fmaf(xv.z, tv.z, acc[r]); acc[r] = fmaf(xv.w, tv.w, acc[r]);
                    }
                }
            }
            for (int o = p.ks >> 1; o > 0; o >>= 1)
#pragma unroll
                for (int r = 0; r < 4; ++r) acc[r] += __shfl_xor_sync(0xffffffffu, acc[r], o);
            if (w < n_items && ks == 0)
#pragma unroll
                for (int r = 0; r < 4; ++r) dots[(g * 4 + r) * p.HW + q] = acc[r];
        }
        __syncthreads();
        if (tid < nt) {
            float mx = -INFINITY;
            for (int q = 0; q < p.HW; ++q) {
                const float v = dots[tid * p.HW + q];
                if (mx == mx && !(v <= mx)) mx = v;                  // a NaN location wins and stays
            }
            tmax[tid] = mx;
        }
        __syncthreads();
        if (tid == 0) {
            for (int r = 0; r < nt; ++r) {
                run += tmax[r];
                if (slot_l[r] < 0) {
                    const int c = slot_c[r];
                    const float v = (run / static_cast<float>(__ldg(p.lens + c))) * p.scale;
                    p.out[p.n_way > 0 ? static_cast<size_t>(m) : static_cast<size_t>(m) * p.C + c] = v;
                    run = 0.f;
                }
            }
        }
    }
}

// g[n,:] from u[n,:] and target[n,:]: one warp per image (F.normalize backward, eps 1e-12)
__global__ void __launch_bounds__(128) gradcam_g_kernel(const float* u, const float* target, float* g, int N, int E,
                                                        int normalize) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (n >= N) return;
    const float* ur = u + static_cast<size_t>(n) * E;
    const float* tr = target + static_cast<size_t>(n) * E;
    float* gr = g + static_cast<size_t>(n) * E;
    if (!normalize) {
        for (int e = lane; e < E; e += 32) gr[e] = __ldg(tr + e);
        return;
    }
    float ssq = 0.f;
    for (int e = lane; e < E; e += 32) { const float v = ur[e]; ssq = fmaf(v, v, ssq); }
    ssq = warp_sum(ssq);
    const float nrm = sqrtf(ssq);
    const float denom = fmaxf(nrm, 1e-12f);
    float dot = 0.f;
    for (int e = lane; e < E; e += 32) dot = fmaf(ur[e] / denom, __ldg(tr + e), dot);
    dot = warp_sum(dot);
    if (nrm < 1e-12f) dot = 0.f;                 // clamp active: y = u / eps, dy/du = I / eps
    for (int e = lane; e < E; e += 32) gr[e] = (__ldg(tr + e) - (ur[e] / denom) * dot) / denom;
}

// alpha[n,c] = sum_e g[n,e] W[e,c] / HW: one thread per (n,c), coalesced over c
__global__ void __launch_bounds__(256) gradcam_alpha_kernel(const float* g, const float* w, float* alpha, int N, int E,
                                                            int K, float inv_hw) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = blockIdx.y;
    if (c >= K) return;
    const float* gr = g + static_cast<size_t>(n) * E;
    float s = 0.f;
#pragma unroll 4
    for (int e = 0; e < E; ++e) s = fmaf(__ldg(gr + e), __ldg(w + static_cast<size_t>(e) * K + c), s);
    alpha[static_cast<size_t>(n) * K + c] = s * inv_hw;
}

// cam[n,p] = max(0, sum_c act[n,c,p] alpha[n,c]): one block per image, 4 channel groups x 64 lanes (HW <= 64)
__global__ void __launch_bounds__(256) gradcam_cam_kernel(const float* act, const float* alpha, float* cam, int K, int HW) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    __shared__ float part[4][64];
    const int n = blockIdx.x;
    const int q = threadIdx.x >> 6, p = threadIdx.x & 63;
    const float* a = act + static_cast<size_t>(n) * K * HW;
    const float* al = alpha + static_cast<size_t>(n) * K;
    const int c0 = q * ((K + 3) / 4), c1 = min(K, c0 + (K + 3) / 4);
    float s = 0.f;
    if (p < HW) {
#pragma unroll 4
        for (int c = c0; c < c1; ++c) s = fmaf(__ldg(a + static_cast<size_t>(c) * HW + p), __ldg(al + c), s);
    }
    part[q][p] = s;
    __syncthreads();
    if (q == 0 && p < HW) cam[static_cast<size_t>(n) * HW + p] = fmaxf(((part[0][p] + part[1][p]) + part[2][p]) + part[3][p], 0.f);
}

// bicubic resize of [N, h, w] maps to [N, H, W] as F.interpolate(mode="bicubic", align_corners=False)
// does it (attention_maps.py:158-163): Keys kernel with A = -0.75, source index (dst + 0.5) * in/out - 0.5,
// border taps clamped; rows first, then columns.
__device__ __forceinline__ void cubic_coeffs(float t, float* c) {
    const float A = -0.75f;
    const float x1 = t, x2 = 1.f - t;
    c[0] = ((A * (x1 + 1.f) - 5.f * A) * (x1 + 1.f) + 8.f * A) * (x1 + 1.f) - 4.f * A;
    c[1] = ((A + 2.f) * x1 - (A + 3.f)) * x1 * x1 + 1.f;
    c[2] = ((A + 2.f) * x2 - (A + 3.f)) * x2 * x2 + 1.f;
    c[3] = ((A * (x2 + 1.f) - 5.f * A) * (x2 + 1.f) + 8.f * A) * (x2 + 1.f) - 4.f * A;
}

__global__ void __launch_bounds__(256) bicubic_upsample_kernel(const float* in, float* out, int N, int h, int w, int H,
                                                               int W) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long total = static_cast<long long>(N) * H * W;
    if (idx >= total) return;
    const int ox = static_cast<int>(idx % W);
    const int oy = static_cast<int>((idx / W) % H);
    const int n = static_cast<int>(idx / (static_cast<long long>(W) * H));
    const float sy = static_cast<float>(h) / static_cast<float>(H), sx = static_cast<float>(w) / static_cast<float>(W);
    const float ry = sy * (static_cast<float>(oy) + 0.5f) - 0.5f, rx = sx * (static_cast<float>(ox) + 0.5f) - 0.5f;
    const float fy = floorf(ry), fx = floorf(rx);
    const int iy = static_cast<int>(fy), ix = static_cast<int>(fx);
    float cy[4], cx[4];
    cubic_coeffs(ry - fy, cy);
    cubic_coeffs(rx - fx, cx);
    const float* src = in + static_cast<size_t>(n) * h * w;
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int yy = min(max(iy - 1 + i, 0), h - 1);
        float row = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int xx = min(max(ix - 1 + j, 0), w - 1);
            row = fmaf(__ldg(src + yy * w + xx), cx[j], row);
        }
        acc = fmaf(row, cy[i], acc);
    }
    out[idx] = acc;
}

// contiguous fp32 -> bf16 cast, 8 elements per thread (two 16-byte loads, one 16-byte store)
__global__ void __launch_bounds__(256) cast_f32_bf16_kernel(const float* src, __nv_bfloat16* dst, long long n8) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n8;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(src) + 2 * i);
        const float4 b = __ldg(reinterpret_cast<const float4*>(src) + 2 * i + 1);
        __nv_bfloat162 p0 = __floats2bfloat162_rn(a.x, a.y), p1 = __floats2bfloat162_rn(a.z, a.w);
        __nv_bfloat162 p2 = __floats2bfloat162_rn(b.x, b.y), p3 = __floats2bfloat162_rn(b.z, b.w);
        uint4 q;
        q.x = *reinterpret_cast<uint32_t*>(&p0); q.y = *reinterpret_cast<uint32_t*>(&p1);
        q.z = *reinterpret_cast<uint32_t*>(&p2); q.w = *reinterpret_cast<uint32_t*>(&p3);
        reinterpret_cast<uint4*>(dst)[i] = q;
    }
}

// --------------------------------------------------------------------------------------
// casts / transposes:  src [batch][R][C] (fp32 or bf16)  ->  dst [batch][R][C] bf16 (nullable)
//                                                         and dst_t [batch][C][R] bf16 (nullable)
// 32x32 tiles through shared memory so both outputs are written coalesced.  With batch = B,
// R = 2048, C = 49 this is the NCHW -> NHWC conversion of the layer4 map for the spatial head.
// --------------------------------------------------------------------------------------
template <typename TIn>
__global__ void __launch_bounds__(256) cast_transpose_kernel(const TIn* src, __nv_bfloat16* dst,
                                                             __nv_bfloat16* dst_t, int R, int C,
                                                             long long ld_src, long long ld_dst,
                                                             long long ld_t, long long bs_src,
                                                             long long bs_dst, long long bs_t) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    __shared__ float tile[32][33];
    const int bz = blockIdx.z;
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;     // 32 x 8
    for (int i = ty; i < 32; i += 8) {
        const int r = r0 + i, c = c0 + tx;
        float v = 0.f;
        if (r < R && c < C) {
            if constexpr (sizeof(TIn) == 4) v = src[bz * bs_src + r * ld_src + c];
            else v = __bfloat162float(src[bz * bs_src + r * ld_src + c]);
            if (dst) dst[bz * bs_dst + r * ld_dst + c] = __float2bfloat16_rn(v);
        }
        tile[i][tx] = v;
    }
    if (!dst_t) return;
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int c = c0 + i, r = r0 + tx;
        if (r < R && c < C) dst_t[bz * bs_t + c * ld_t + r] = __float2bfloat16_rn(tile[tx][i]);
    }
}


// --------------------------------------------------------------------------------------
// stand-alone backward of the flat text encoder (used when encode_text is differentiated on
// its own): dm = F.normalize-backward(g) / len, then the embedding scatter.  One warp per row.
// --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) embedding_bag_bwd_kernel(const long long* ids, const long long* lens,
                                                                const float* g, const float* feat,
                                                                const float* inv_norm, int normalize,
                                                                float* dtable, int B, int L, int E, int V) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= B) return;
    const int nch = (E + 127) >> 7;
    float4 r[kMaxVec], f[kMaxVec];
    float dot = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxVec; ++c) {
        r[c] = make_float4(0.f, 0.f, 0.f, 0.f); f[c] = r[c];
        if (c < nch && (c * 32 + lane) * 4 < E) {
            r[c] = __ldg(reinterpret_cast<const float4*>(g + static_cast<size_t>(warp) * E) + c * 32 + lane);
            if (normalize) f[c] = __ldg(reinterpret_cast<const float4*>(feat + static_cast<size_t>(warp) * E) + c * 32 + lane);
        }
        dot += r[c].x * f[c].x + r[c].y * f[c].y + r[c].z * f[c].z + r[c].w * f[c].w;
    }
    dot = warp_sum(dot);
    const float inv = normalize ? __ldg(inv_norm + warp) : 1.f;
    const float sc = inv / static_cast<float>(__ldg(lens + warp));
#pragma unroll
    for (int c = 0; c < kMaxVec; ++c) {
        r[c].x = (r[c].x - f[c].x * dot) * sc; r[c].y = (r[c].y - f[c].y * dot) * sc;
        r[c].z = (r[c].z - f[c].z * dot) * sc; r[c].w = (r[c].w - f[c].w * dot) * sc;
    }
    for (int l = 0; l < L; ++l) {
        const long long id = __ldg(ids + static_cast<size_t>(warp) * L + l);
        if (id <= 0 || id >= V) continue;
        float4* dst = reinterpret_cast<float4*>(dtable + static_cast<size_t>(id) * E);
#pragma unroll
        for (int c = 0; c < kMaxVec; ++c)
            if (c < nch && (c * 32 + lane) * 4 < E) atomicAdd(dst + c * 32 + lane, r[c]);
    }
}

// stand-alone F.normalize backward on rows: du = (g - feat <feat,g>) * inv_norm.
// Outputs (nullable): fp32 [M,E], bf16 [M,ld], bf16 transposed [E,ld_t], dbias[E] += sum_m du.
__global__ void __launch_bounds__(256) rownorm_bwd_kernel(const float* g, const float* feat,
                                                          const float* inv_norm, int M, int E, int normalize,
                                                          float* du_f32, __nv_bfloat16* du_bf16, int ld,
                                                          __nv_bfloat16* du_bf16_t, int ld_t, float* dbias) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= M) return;
    const int nch = (E + 127) >> 7;
    float4 r[kMaxVec], f[kMaxVec];
    float dot = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxVec; ++c) {
        r[c] = make_float4(0.f, 0.f, 0.f, 0.f); f[c] = r[c];
        if (c < nch && (c * 32 + lane) * 4 < E) {
            r[c] = __ldg(reinterpret_cast<const float4*>(g + static_cast<size_t>(warp) * E) + c * 32 + lane);
            if (normalize) f[c] = __ldg(reinterpret_cast<const float4*>(feat + static_cast<size_t>(warp) * E) + c * 32 + lane);
        }
        dot += r[c].x * f[c].x + r[c].y * f[c].y + r[c].z * f[c].z + r[c].w * f[c].w;
    }
    dot = warp_sum(dot);
    const float inv = normalize ? __ldg(inv_norm + warp) : 1.f;
#pragma unroll
    for (int c = 0; c < kMaxVec; ++c) {
        const int e = (c * 32 + lane) * 4;
        if (c < nch && e < E) {
            float4 o = make_float4((r[c].x - f[c].x * dot) * inv, (r[c].y - f[c].y * dot) * inv,
                                   (r[c].z - f[c].z * dot) * inv, (r[c].w - f[c].w * dot) * inv);
            if (du_f32) *reinterpret_cast<float4*>(du_f32 + static_cast<size_t>(warp) * E + e) = o;
            if (du_bf16) store_bf16x4(du_bf16 + static_cast<size_t>(warp) * ld + e, o);
            if (du_bf16_t) {
                du_bf16_t[static_cast<size_t>(e) * ld_t + warp] = __float2bfloat16_rn(o.x);
                du_bf16_t[static_cast<size_t>(e + 1) * ld_t + warp] = __float2bfloat16_rn(o.y);
                du_bf16_t[static_cast<size_t>(e + 2) * ld_t + warp] = __float2bfloat16_rn(o.z);
                du_bf16_t[static_cast<size_t>(e + 3) * ld_t + warp] = __float2bfloat16_rn(o.w);
            }
            if (dbias) {
                atomicAdd(dbias + e, o.x); atomicAdd(dbias + e + 1, o.y);
                atomicAdd(dbias + e + 2, o.z); atomicAdd(dbias + e + 3, o.w);
            }
        }
    }
}

// second half of the split-K feature-gradient path (long contractions: sharded global batches).
// acc [M, E] fp32 holds Gs . other summed over the K-splits; this warp-per-row pass applies what the
// EpiNormBwdT epilogue does in the single-kernel path, in the same order:
//   g = acc + diag_coef[m] * diag[m + diag_off];  du = (g - feat <feat, g>) * inv_norm;  out = du / len
// Outputs: fp32 [M, ld_f32] (may alias acc) or bf16 [M, ld_bf16]; dbias[E] += column sums (shared-memory
// pre-reduction over the 8 rows of a block, then one global atomic per column and block).
__device__ __forceinline__ float4 load_bf16x4(const __nv_bfloat16* p) {
    const uint2 q = *reinterpret_cast<const uint2*>(p);
    const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&q.x);
    const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162*>(&q.y);
    return make_float4(__low2float(a), __high2float(a), __low2float(b), __high2float(b));
}

__global__ void __launch_bounds__(256) featgrad_finish_kernel(const float* acc, int ld_acc, const __nv_bfloat16* feat,
                                                              int ld_feat, const __nv_bfloat16* diag, int ld_diag,
                                                              int diag_rows, int diag_off, const float* diag_coef,
                                                              const float* inv_norm, int normalize,
                                                              const long long* row_len, int M, int E, float* out_f32,
                                                              int ld_f32, __nv_bfloat16* out_bf16, int ld_bf16,
                                                              float* dbias) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    __shared__ float s_col[128 * kMaxVec];
    const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const int nch = (E + 127) >> 7;
    if (dbias) {
        for (int i = threadIdx.x; i < E; i += blockDim.x) s_col[i] = 0.f;
        __syncthreads();
    }
    if (m < M) {
        float4 g[kMaxVec], f[kMaxVec];
        float dot = 0.f;
        const bool use_diag = diag != nullptr && m + diag_off < diag_rows;
        const float dc = use_diag ? __ldg(diag_coef + m) : 0.f;
#pragma unroll
        for (int c = 0; c < kMaxVec; ++c) {
            g[c] = make_float4(0.f, 0.f, 0.f, 0.f); f[c] = g[c];
            const int e = (c * 32 + lane) * 4;
            if (c < nch && e < E) {
                g[c] = *reinterpret_cast<const float4*>(acc + static_cast<size_t>(m) * ld_acc + e);
                if (use_diag) {
                    const float4 d = load_bf16x4(diag + static_cast<size_t>(m + diag_off) * ld_diag + e);
                    g[c].x = fmaf(dc, d.x, g[c].x); g[c].y = fmaf(dc, d.y, g[c].y);
                    g[c].z = fmaf(dc, d.z, g[c].z); g[c].w = fmaf(dc, d.w, g[c].w);
                }
                if (normalize) f[c] = load_bf16x4(feat + static_cast<size_t>(m) * ld_feat + e);
            }
            dot = fmaf(f[c].x, g[c].x, dot); dot = fmaf(f[c].y, g[c].y, dot);
            dot = fmaf(f[c].z, g[c].z, dot); dot = fmaf(f[c].w, g[c].w, dot);
        }
        dot = warp_sum(dot);
        const float inv = normalize ? __ldg(inv_norm + m) : 1.f;
        const float rs = row_len ? 1.f / static_cast<float>(row_len[m]) : 1.f;
#pragma unroll
        for (int c = 0; c < kMaxVec; ++c) {
            const int e = (c * 32 + lane) * 4;
            if (c < nch && e < E) {
                float4 o = g[c];
                if (normalize)
                    o = make_float4((g[c].x - f[c].x * dot) * inv, (g[c].y - f[c].y * dot) * inv,
                                    (g[c].z - f[c].z * dot) * inv, (g[c].w - f[c].w * dot) * inv);
                o.x *= rs; o.y *= rs; o.z *= rs; o.w *= rs;
                if (out_f32) *reinterpret_cast<float4*>(out_f32 + static_cast<size_t>(m) * ld_f32 + e) = o;
                if (out_bf16) store_bf16x4(out_bf16 + static_cast<size_t>(m) * ld_bf16 + e, o);
                if (dbias) {
                    atomicAdd(s_col + e, o.x); atomicAdd(s_col + e + 1, o.y);
                    atomicAdd(s_col + e + 2, o.z); atomicAdd(s_col + e + 3, o.w);
                }
            }
        }
    }
    if (dbias) {
        __syncthreads();
        for (int i = threadIdx.x; i < E; i += blockDim.x) atomicAdd(dbias + i, s_col[i]);
    }
}

// sum over the HW locations of a [B, HW, E] fp32 map (image factor of the spatial "mean"
// similarity, multimodal.py:765-770).  Thread = 4 consecutive channels, coalesced over E.
__global__ void __launch_bounds__(128) spatial_pool_kernel(const float* src, int B, int HW, int E,
                                                           float* out_f32, __nv_bfloat16* out_bf16, int ld,
                                                           __nv_bfloat16* out_bf16_t, int ld_t) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int b = blockIdx.y;
    const int e = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (e >= E) return;
    const float4* p = reinterpret_cast<const float4*>(src + (static_cast<size_t>(b) * HW) * E + e);
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int h = 0; h < HW; ++h) {
        const float4 v = __ldg(p + static_cast<size_t>(h) * (E >> 2));
        a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
    if (out_f32) *reinterpret_cast<float4*>(out_f32 + static_cast<size_t>(b) * E + e) = a;
    if (out_bf16) store_bf16x4(out_bf16 + static_cast<size_t>(b) * ld + e, a);
    if (out_bf16_t) {
        out_bf16_t[static_cast<size_t>(e) * ld_t + b] = __float2bfloat16_rn(a.x);
        out_bf16_t[static_cast<size_t>(e + 1) * ld_t + b] = __float2bfloat16_rn(a.y);
        out_bf16_t[static_cast<size_t>(e + 2) * ld_t + b] = __float2bfloat16_rn(a.z);
        out_bf16_t[static_cast<size_t>(e + 3) * ld_t + b] = __float2bfloat16_rn(a.w);
    }
}


// backward of spatial_pool: d src[b, h, :] = g[b, :] for every location h (the sum's gradient is a broadcast).
// Thread = 4 consecutive channels of one image; the row is read once and stored HW times with streaming stores.
__global__ void __launch_bounds__(128) spatial_pool_bwd_kernel(const float* g, int B, int HW, int E, float* dst) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int b = blockIdx.y;
    const int e = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (e >= E) return;
    const float4 v = __ldg(reinterpret_cast<const float4*>(g + static_cast<size_t>(b) * E + e));
    float4* p = reinterpret_cast<float4*>(dst + (static_cast<size_t>(b) * HW) * E + e);
    for (int h = 0; h < HW; ++h) __stcs(p + static_cast<size_t>(h) * (E >> 2), v);
}

// --------------------------------------------------------------------------------------
// spatial "max" similarity backward (SIMT gather form, v1).  g = dL/dmatch [Bi,Bt];
// coef[i,t] = g[i,t] / len[t].  With hw* = argmax location saved by the forward:
//   dtok[t,l,:]  = sum_i    coef[i,t] * img[i, hw*(i,t,l), :]
//   dimg[i,hw,:] = sum_{t,l : hw*(i,t,l) = hw} coef[i,t] * tok[t,l,:]
// (autograd of einsum + amax + sum + div, multimodal.py:775-780; ties only occur for all-zero pad
// tokens, whose contributions vanish).  One warp per output row, bf16 row gathers from L2.
// --------------------------------------------------------------------------------------
__device__ __forceinline__ void fma_bf16x8(float* acc, uint4 q, float c) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float2 f = __bfloat1622float2(h[k]);
        acc[2 * k] = fmaf(c, f.x, acc[2 * k]);
        acc[2 * k + 1] = fmaf(c, f.y, acc[2 * k + 1]);
    }
}

__global__ void __launch_bounds__(256) spatial_max_dtok_kernel(const float* g, const long long* lens,
                                                               const long long* ids,
                                                               const unsigned char* amax_ti,
                                                               const __nv_bfloat16* img, float* dtok,
                                                               int Bi, int Bt, int L, int HW, int E) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= Bt * L) return;
    const int t = warp / L;
    const int nv = E >> 3;                        // uint4 (8 bf16) chunks per row; lane handles nv/32 (E%256==0 fast)
    float acc[4][8];
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[c][k] = 0.f;
    if (ids == nullptr || __ldg(ids + warp) != 0) {
        const float invlen = 1.f / static_cast<float>(__ldg(lens + t));
        for (int i0 = 0; i0 < Bi; i0 += 32) {
            const int ii = i0 + lane;
            const int a_l = ii < Bi ? amax_ti[static_cast<size_t>(warp) * Bi + ii] : 0;
            const float c_l = ii < Bi ? __ldg(g + static_cast<size_t>(ii) * Bt + t) * invlen : 0.f;
            const int n = min(32, Bi - i0);
            for (int k = 0; k < n; ++k) {
                const int a = __shfl_sync(0xffffffffu, a_l, k);
                const float c = __shfl_sync(0xffffffffu, c_l, k);
                const uint4* src = reinterpret_cast<const uint4*>(img + (static_cast<size_t>(i0 + k) * HW + a) * E);
#pragma unroll
                for (int cc = 0; cc < 4; ++cc)
                    if (cc * 32 + lane < nv) fma_bf16x8(acc[cc], __ldg(src + cc * 32 + lane), c);
            }
        }
    }
    float* dst = dtok + static_cast<size_t>(warp) * E;
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
        if (cc * 32 + lane < nv) {
            float4* d4 = reinterpret_cast<float4*>(dst + (cc * 32 + lane) * 8);
            d4[0] = make_float4(acc[cc][0], acc[cc][1], acc[cc][2], acc[cc][3]);
            d4[1] = make_float4(acc[cc][4], acc[cc][5], acc[cc][6], acc[cc][7]);
        }
    }
}

__global__ void __launch_bounds__(256) spatial_max_dimg_kernel(const float* g, const long long* lens,
                                                               const unsigned char* amax_it,
                                                               const __nv_bfloat16* tok, float* dimg,
                                                               int Bi, int Bt, int L, int HW, int E) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= Bi * HW) return;
    const int i = warp / HW, hw = warp % HW;
    const int nv = E >> 3;
    float acc[4][8];
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[c][k] = 0.f;
    const int ntl = Bt * L;
    const unsigned char* arow = amax_it + static_cast<size_t>(i) * ntl;
    for (int tl0 = 0; tl0 < ntl; tl0 += 32) {
        const int tl = tl0 + lane;
        const bool hit = tl < ntl && arow[tl] == hw;
        unsigned mask = __ballot_sync(0xffffffffu, hit);
        while (mask) {
            const int k = __ffs(mask) - 1;
            mask &= mask - 1;
            const int x = tl0 + k, t = x / L;
            const float c = __ldg(g + static_cast<size_t>(i) * Bt + t) / static_cast<float>(__ldg(lens + t));
            const uint4* src = reinterpret_cast<const uint4*>(tok + static_cast<size_t>(x) * E);
#pragma unroll
            for (int cc = 0; cc < 4; ++cc)
                if (cc * 32 + lane < nv) fma_bf16x8(acc[cc], __ldg(src + cc * 32 + lane), c);
        }
    }
    float* dst = dimg + static_cast<size_t>(warp) * E;
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
        if (cc * 32 + lane < nv) {
            float4* d4 = reinterpret_cast<float4*>(dst + (cc * 32 + lane) * 8);
            d4[0] = make_float4(acc[cc][0], acc[cc][1], acc[cc][2], acc[cc][3]);
            d4[1] = make_float4(acc[cc][4], acc[cc][5], acc[cc][6], acc[cc][7]);
        }
    }
}

// --------------------------------------------------------------------------------------
// InfoNCE statistics from MATERIALISED similarity blocks (spatial "max" path: the match matrix is
// small next to the B*B*L*HW contraction that produced it).  Row block match_r [b,N] (b image
// rows against all N texts) and column block match_c [N,b] (all N images against b texts); the
// positive of local row / column m sits at (m, m + diag_off) / (m + diag_off, m).  One device:
// match_r == match_c == match [B,B], b = N = B, diag_off = 0.
// One warp per row (z=0: image rows of match_r) or per column (z=1: text columns of match_c);
// writes the same RowStat partials (n_tiles = 1) that infonce_finalize_kernel merges.
// --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) match_stats_kernel(const float* match_r, const float* match_c, int b, int N,
                                                          int diag_off, float scale, RowStat* part0, RowStat* part1,
                                                          float* diag0, float* diag1, unsigned int* ticket) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    if (blockIdx.x == 0 && threadIdx.x == 0) *ticket = 0u;        // finalize's ticket (runs after us)
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= 2 * b) return;
    const int z = warp < b ? 0 : 1;
    const int m = z ? warp - b : warp;
    const int n = N;
    const size_t stride = z ? b : 1;
    const float* base = z ? match_c + m : match_r + static_cast<size_t>(m) * N;
    float mx = -INFINITY; int arg = 0x7fffffff;
    for (int j = lane; j < n; j += 32) {
        const float x = base[j * stride] * scale;
        if (x > mx) { mx = x; arg = j; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float om = __shfl_xor_sync(0xffffffffu, mx, o);
        const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
        if (om > mx || (om == mx && oa < arg)) { mx = om; arg = oa; }
    }
    float l = 0.f, a = 0.f;
    for (int j = lane; j < n; j += 32) {
        const float x = base[j * stride] * scale;
        const float e = __expf(x - mx);
        l += e; a = fmaf(e, x, a);
    }
    l = warp_sum(l); a = warp_sum(a);
    if (lane == 0) {
        RowStat rs; rs.m = mx; rs.l = l; rs.a = a; rs.arg = arg;
        (z ? part1 : part0)[m] = rs;
        (z ? diag1 : diag0)[m] = base[static_cast<size_t>(m + diag_off) * stride] * scale;
    }
}

// d loss / d match = scale * G,  x = scale * match, over the row block (blockIdx.y = 0) and the column block
// (blockIdx.y = 1, skipped when dmatch_c is null):
//   G_r[i,t] = coef * (exp(x - lse0[i])     + exp(x - lse1_all[t]) - 2 [t = i + diag_off])   match_r [b,N]
//   G_c[i,t] = coef * (exp(x - lse0_all[i]) + exp(x - lse1[t])     - 2 [i = t + diag_off])   match_c [N,b]
// d scale = sum G_r * x over the row block only (each pair's logit counted once over the ranks).  With ds_part
// ([gridDim.x] floats) and ticket (zeroed before the launch) the row-block blocks write their partial sums and the
// last one to finish adds them in block order, so a replay is bit-identical; without them each warp adds its sum
// into *dscale atomically.
__global__ void __launch_bounds__(256) match_grad_kernel(const float* match_r, const float* match_c, int b, int N,
                                                         int diag_off, float scale, float coef, const float* lse0,
                                                         const float* lse1_all, const float* lse0_all,
                                                         const float* lse1, float* dmatch_r, float* dmatch_c,
                                                         float* dscale, float* ds_part, unsigned int* ticket) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int z = blockIdx.y;
    if (z == 1 && !dmatch_c) return;
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const int cols = z ? b : N;
    float ds = 0.f;
    if (idx < static_cast<long long>(b) * N) {
        const int i = static_cast<int>(idx / cols), t = static_cast<int>(idx % cols);
        const float x = (z ? match_c : match_r)[idx] * scale;
        const float lr = z ? lse0_all[i] : lse0[i], lc = z ? lse1[t] : lse1_all[t];
        // the positive as (P_row - 1) + (P_col - 1) with expm1: P_row + P_col - 2 cancels when the pair is confident,
        // and the rounding of the exponentials would be left as the whole value (at one pair it is exactly 0)
        float gg = (z ? i == t + diag_off : t == i + diag_off) ? expm1f(x - lr) + expm1f(x - lc)
                                                                : __expf(x - lr) + __expf(x - lc);
        gg *= coef;
        (z ? dmatch_c : dmatch_r)[idx] = gg * scale;
        ds = gg * x;
    }
    if (z == 1) return;
    ds = warp_sum(ds);
    if (!ds_part) {
        if ((threadIdx.x & 31) == 0 && dscale) atomicAdd(dscale, ds);
        return;
    }
    __shared__ float red[8];
    __shared__ bool is_last;
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ds;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f;
        for (int k = 0; k < (blockDim.x >> 5); ++k) s += red[k];
        ds_part[blockIdx.x] = s;
        __threadfence();
        is_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (is_last && threadIdx.x < 32) {          // fixed lane-strided order + tree
        __threadfence();
        float s = 0.f;
        for (unsigned int k = threadIdx.x; k < gridDim.x; k += 32) s += ds_part[k];
        s = warp_sum(s);
        if (threadIdx.x == 0) { *dscale = s; *ticket = 0u; }
    }
}


// --------------------------------------------------------------------------------------
// spatial "max" backward, tensor-core form: expand the saved arg-max into the (mostly zero) bf16
// matrix  P[(t,l), (i,hw)] = [hw = hw*(i,t,l)] * g[i,t] / len[t]  so that both gradients become
// plain GEMMs on the tcgen05 engine:  dtok = P . img   and   dimg = P^T . tok  (P read MN-major).
// One block per token row; threads sweep the Bi*HW columns coalesced.
// --------------------------------------------------------------------------------------
// Row compaction of the token axis: pad positions (l >= len[t]) carry no gradient, and they are 44 % of the [Bt, L]
// slots at the corpus' mean length of 14.  offs[t] = number of real tokens before utterance t (exclusive scan,
// one block), offs[Bt] = their total Mv -- a DEVICE-side size: the GEMMs that follow read it as their row /
// contraction limit, so no host sync is needed and the step stays graph-capturable.
__global__ void __launch_bounds__(1024) token_row_offsets_kernel(const long long* lens, int Bt, int L, int* offs) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    __shared__ int part[1024];
    const int per = (Bt + 1023) / 1024;
    const int t0 = threadIdx.x * per;
    int s = 0;
    for (int t = t0; t < t0 + per && t < Bt; ++t) {
        const long long n = __ldg(lens + t);
        s += static_cast<int>(n < 0 ? 0 : (n > L ? L : n));
    }
    part[threadIdx.x] = s;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {                   // Hillis-Steele inclusive scan of the per-thread sums
        const int v = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
        __syncthreads();
        part[threadIdx.x] += v;
        __syncthreads();
    }
    int run = threadIdx.x ? part[threadIdx.x - 1] : 0;
    for (int t = t0; t < t0 + per && t < Bt; ++t) {
        offs[t] = run;
        const long long n = __ldg(lens + t);
        run += static_cast<int>(n < 0 ? 0 : (n > L ? L : n));
    }
    if (threadIdx.x == 1023) offs[Bt] = part[1023];
}

// One block per (t, l) slot.  Real token: row r = offs[t] + l of the compacted P (bf16, [Mv, Bi*HW]) =
// [hw = argmax(i,t,l)] * g[i,t] / len[t], and row r of the compacted token features.  Pad slot number j (in slot
// order): ZERO row Mv + j of both while that is below the next multiple of 128 -- the contraction of dimg = P^T . tok
// runs in 64-row chunks and must read finite values up to the end of its last chunk.
__global__ void __launch_bounds__(256) spatial_max_expand_kernel(const float* g, const long long* lens,
                                                                 const unsigned char* amax_ti,
                                                                 __nv_bfloat16* P, long long ldp,
                                                                 int Bi, int Bt, int L, int HW,
                                                                 const int* offs, const __nv_bfloat16* tok,
                                                                 __nv_bfloat16* tokc, int E) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int tl = blockIdx.x;
    const int t = tl / L, l = tl - t * L;
    const long long len_raw = __ldg(lens + t);
    const int len = static_cast<int>(len_raw < 0 ? 0 : (len_raw > L ? L : len_raw));
    const int ncol = Bi * HW;
    const int off_t = __ldg(offs + t), mv = __ldg(offs + Bt);
    if (l >= len) {                                                   // pad slot
        const int zr = mv + (tl - (off_t + len));
        if (zr >= ((mv + 127) / 128) * 128 || zr >= Bt * L) return;
        uint4* prow = reinterpret_cast<uint4*>(P + static_cast<size_t>(zr) * ldp);
        for (int c = threadIdx.x; c < static_cast<int>(ldp / 8); c += blockDim.x) prow[c] = make_uint4(0u, 0u, 0u, 0u);
        uint4* trow = reinterpret_cast<uint4*>(tokc + static_cast<size_t>(zr) * E);
        for (int c = threadIdx.x; c < E / 8; c += blockDim.x) trow[c] = make_uint4(0u, 0u, 0u, 0u);
        return;
    }
    const int r = off_t + l;
    {
        const uint4* src = reinterpret_cast<const uint4*>(tok + static_cast<size_t>(tl) * E);
        uint4* dst = reinterpret_cast<uint4*>(tokc + static_cast<size_t>(r) * E);
        for (int c = threadIdx.x; c < E / 8; c += blockDim.x) dst[c] = __ldg(src + c);
    }
    const float invlen = 1.f / static_cast<float>(len_raw);
    const unsigned char* arow = amax_ti + static_cast<size_t>(tl) * Bi;
    __nv_bfloat16* prow = P + static_cast<size_t>(r) * ldp;
    // eight columns (one 16-byte store) per thread: the window touches at most two images (HW >= 8) and is all zero
    // unless an arg-max lies inside it, so g is fetched for about one window in six.  ldp is a multiple of 8 and P is
    // 16-byte aligned (the caller's workspace), so every full window is one aligned store.
    for (int c = threadIdx.x * 8; c < ncol; c += blockDim.x * 8) {
        const int i0 = c / HW;
        const int h0 = c - i0 * HW;                        // window = locations h0.. of image i0, then image i0 + 1
        int k0 = static_cast<int>(arow[i0]) - h0, k1 = -1;  // positions of the (at most two) non-zeros in the window
        float v0 = 0.f, v1 = 0.f;
        if (k0 >= 0 && k0 < 8) v0 = __ldg(g + static_cast<size_t>(i0) * Bt + t) * invlen; else k0 = -1;
        if (HW - h0 < 8 && i0 + 1 < Bi) {
            k1 = HW - h0 + static_cast<int>(arow[i0 + 1]);
            if (k1 < 8) v1 = __ldg(g + static_cast<size_t>(i0 + 1) * Bt + t) * invlen; else k1 = -1;
        }
        unsigned int w[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float lo = (2 * q == k0) ? v0 : ((2 * q == k1) ? v1 : 0.f);
            const float hi = (2 * q + 1 == k0) ? v0 : ((2 * q + 1 == k1) ? v1 : 0.f);
            const __nv_bfloat162 o = __floats2bfloat162_rn(lo, hi);
            w[q] = *reinterpret_cast<const unsigned int*>(&o);
        }
        if (c + 8 <= ncol) *reinterpret_cast<uint4*>(prow + c) = make_uint4(w[0], w[1], w[2], w[3]);
        else {
            for (int k = 0; c + k < ncol; ++k) {
                const unsigned int word = w[k >> 1];
                const unsigned short h = (k & 1) ? static_cast<unsigned short>(word >> 16) : static_cast<unsigned short>(word & 0xffffu);
                reinterpret_cast<unsigned short*>(prow)[c + k] = h;
            }
            for (int k = ncol - c; k < 8 && c + k < static_cast<int>(ldp); ++k)      // the padding columns up to ldp
                reinterpret_cast<unsigned short*>(prow)[c + k] = 0;
        }
    }
}

// d tok [Bt*L, E] fp32 from its compacted form: real tokens copy row offs[t] + l, pad slots are zero.  One warp per slot.
__global__ void __launch_bounds__(256) token_rows_scatter_kernel(const float* src, const long long* lens, const int* offs,
                                                                 float* dst, int Bt, int L, int E) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const long long w = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= static_cast<long long>(Bt) * L) return;
    const int t = static_cast<int>(w / L), l = static_cast<int>(w - static_cast<long long>(t) * L);
    const long long len_raw = __ldg(lens + t);
    const int len = static_cast<int>(len_raw < 0 ? 0 : (len_raw > L ? L : len_raw));
    float4* d = reinterpret_cast<float4*>(dst + w * E);
    if (l < len) {
        const float4* s = reinterpret_cast<const float4*>(src + static_cast<size_t>(__ldg(offs + t) + l) * E);
        for (int c = lane; c < E / 4; c += 32) d[c] = __ldg(s + c);
    } else {
        for (int c = lane; c < E / 4; c += 32) d[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}


// --------------------------------------------------------------------------------------
// Fused AdamW for the head parameters (the optimiser the reference configures,
// multimodal_lit.py:112-128: torch.optim.AdamW, decoupled weight decay).  One pass over p, g, m, v
// (28 B / parameter); optionally refreshes the bf16 shadow copy that the head GEMM consumes, so the
// per-step fp32->bf16 cast of W disappears from a training loop.  Same update order as
// torch.optim.AdamW (single-tensor path): decay, moments, bias-corrected step.
// --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) adamw_step_kernel(float* p, const float* g, float* m, float* v,
                                                         long long n, float lr, float beta1, float beta2,
                                                         float eps, float wd, float bc1, float bc2_sqrt,
                                                         float grad_scale, __nv_bfloat16* shadow) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const float step_size = lr / bc1;
    for (long long i = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) * 4; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x * 4) {
        if (i + 4 <= n) {
            float4 P = *reinterpret_cast<float4*>(p + i);
            const float4 G = __ldg(reinterpret_cast<const float4*>(g + i));
            float4 M = *reinterpret_cast<float4*>(m + i), V = *reinterpret_cast<float4*>(v + i);
            float pp[4] = {P.x, P.y, P.z, P.w}, gg[4] = {G.x, G.y, G.z, G.w};
            float mm[4] = {M.x, M.y, M.z, M.w}, vv[4] = {V.x, V.y, V.z, V.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float gk = gg[k] * grad_scale;
                pp[k] *= 1.f - lr * wd;
                mm[k] = mm[k] + (gk - mm[k]) * (1.f - beta1);            // lerp, as torch does
                vv[k] = vv[k] * beta2 + gk * gk * (1.f - beta2);
                const float denom = sqrtf(vv[k]) / bc2_sqrt + eps;
                pp[k] -= step_size * (mm[k] / denom);
            }
            *reinterpret_cast<float4*>(p + i) = make_float4(pp[0], pp[1], pp[2], pp[3]);
            *reinterpret_cast<float4*>(m + i) = make_float4(mm[0], mm[1], mm[2], mm[3]);
            *reinterpret_cast<float4*>(v + i) = make_float4(vv[0], vv[1], vv[2], vv[3]);
            if (shadow) store_bf16x4(shadow + i, make_float4(pp[0], pp[1], pp[2], pp[3]));
        } else {
            for (long long j = i; j < n; ++j) {
                const float gk = g[j] * grad_scale;
                float pj = p[j] * (1.f - lr * wd);
                const float mj = m[j] + (gk - m[j]) * (1.f - beta1);
                const float vj = v[j] * beta2 + gk * gk * (1.f - beta2);
                pj -= step_size * (mj / (sqrtf(vj) / bc2_sqrt + eps));
                p[j] = pj; m[j] = mj; v[j] = vj;
                if (shadow) shadow[j] = __float2bfloat16_rn(pj);
            }
        }
    }
}


// The same update for up to kAdamMaxTensors tensors in ONE launch, with the step counter kept on the
// device: bias corrections are computed in the kernel from *step_dev + 1 and the last block to finish
// (atomic ticket) increments it, so the launch can be captured in a CUDA graph and replayed (a host-side
// step number would be baked into the graph).  Used by GraphedContrastiveStep to make a whole train step
// -- forward, backward, optimizer, refreshed bf16 weight shadow -- one graph.
constexpr int kAdamMaxTensors = 8;
struct AdamMultiParams {
    float* p[kAdamMaxTensors]; const float* g[kAdamMaxTensors]; float* m[kAdamMaxTensors]; float* v[kAdamMaxTensors];
    __nv_bfloat16* shadow[kAdamMaxTensors];
    long long n4_begin[kAdamMaxTensors + 1];       // prefix sums of ceil(n / 4) per tensor
    long long n[kAdamMaxTensors];
    float lr[kAdamMaxTensors], wd[kAdamMaxTensors];
    int count;
    float beta1, beta2, eps, grad_scale;
    int* step_dev;               // [1] completed steps; this launch performs step *step_dev + 1
    unsigned int* ticket;        // [1] zero on entry, left zero on exit
};

__global__ void __launch_bounds__(256) adamw_multi_kernel(const AdamMultiParams a) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int step = *reinterpret_cast<volatile int*>(a.step_dev) + 1;
    const float bc1 = 1.f - powf(a.beta1, static_cast<float>(step));
    const float bc2_sqrt = sqrtf(1.f - powf(a.beta2, static_cast<float>(step)));
    const long long total4 = a.n4_begin[a.count];
    for (long long q = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; q < total4;
         q += static_cast<long long>(gridDim.x) * blockDim.x) {
        int t = 0;
#pragma unroll
        for (int k = 1; k < kAdamMaxTensors; ++k) if (k < a.count && q >= a.n4_begin[k]) t = k;
        const long long i = (q - a.n4_begin[t]) * 4;
        const long long n = a.n[t];
        const float lr = a.lr[t], wd = a.wd[t];
        const float step_size = lr / bc1;
        float* p = a.p[t]; const float* g = a.g[t]; float* m = a.m[t]; float* v = a.v[t];
        const int cnt = (i + 4 <= n) ? 4 : static_cast<int>(n - i);
        float pp[4], gg[4], mm[4], vv[4];
        if (cnt == 4) {
            const float4 P = *reinterpret_cast<const float4*>(p + i), G = *reinterpret_cast<const float4*>(g + i);
            const float4 M = *reinterpret_cast<const float4*>(m + i), V = *reinterpret_cast<const float4*>(v + i);
            pp[0] = P.x; pp[1] = P.y; pp[2] = P.z; pp[3] = P.w; gg[0] = G.x; gg[1] = G.y; gg[2] = G.z; gg[3] = G.w;
            mm[0] = M.x; mm[1] = M.y; mm[2] = M.z; mm[3] = M.w; vv[0] = V.x; vv[1] = V.y; vv[2] = V.z; vv[3] = V.w;
        } else {
            for (int k = 0; k < cnt; ++k) { pp[k] = p[i + k]; gg[k] = g[i + k]; mm[k] = m[i + k]; vv[k] = v[i + k]; }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (k < cnt) {
                const float gk = gg[k] * a.grad_scale;
                pp[k] *= 1.f - lr * wd;
                mm[k] = mm[k] + (gk - mm[k]) * (1.f - a.beta1);
                vv[k] = vv[k] * a.beta2 + gk * gk * (1.f - a.beta2);
                const float denom = sqrtf(vv[k]) / bc2_sqrt + a.eps;
                pp[k] -= step_size * (mm[k] / denom);
            }
        }
        if (cnt == 4) {
            *reinterpret_cast<float4*>(p + i) = make_float4(pp[0], pp[1], pp[2], pp[3]);
            *reinterpret_cast<float4*>(m + i) = make_float4(mm[0], mm[1], mm[2], mm[3]);
            *reinterpret_cast<float4*>(v + i) = make_float4(vv[0], vv[1], vv[2], vv[3]);
            if (a.shadow[t]) store_bf16x4(a.shadow[t] + i, make_float4(pp[0], pp[1], pp[2], pp[3]));
        } else {
            for (int k = 0; k < cnt; ++k) {
                p[i + k] = pp[k]; m[i + k] = mm[k]; v[i + k] = vv[k];
                if (a.shadow[t]) a.shadow[t][i + k] = __float2bfloat16_rn(pp[k]);
            }
        }
    }
    // every block has read the step number before any block can pass the ticket as the last one
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(a.ticket, 1u) == gridDim.x - 1) {
            *a.step_dev = step;
            *a.ticket = 0u;
            __threadfence();
        }
    }
}


// --------------------------------------------------------------------------------------
// All-gather over NVLink peer memory: every rank exposes its block in symmetric memory; after a
// cross-rank barrier each rank pulls the other ranks' blocks with 16-byte loads from the PEER
// pointers (NVSwitch gives every peer full bandwidth) into its local gathered buffer.  Replaces an
// NCCL all-gather (17 us measured for 1 MB per rank at 2 GPUs) by a 6 us barrier + this copy.
// blockIdx.y = source rank; grid-stride over the block's 16-byte words.
// --------------------------------------------------------------------------------------
struct PeerPtrs { const void* p[8]; };

__global__ void __launch_bounds__(256) p2p_gather_kernel(const PeerPtrs peers, unsigned char* dst,
                                                         long long bytes_per_rank, long long dst_stride,
                                                         int skip_rank) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int r = blockIdx.y;
    if (r == skip_rank) return;
    const uint4* src = reinterpret_cast<const uint4*>(peers.p[r]);
    uint4* out = reinterpret_cast<uint4*>(dst + static_cast<long long>(r) * dst_stride);
    const long long n16 = bytes_per_rank >> 4;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n16;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        uint4 v;
        asm volatile("ld.global.relaxed.sys.v4.u32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(src + i) : "memory");
        out[i] = v;
    }
}


// --------------------------------------------------------------------------------------
// bias + L2 normalise rows of a fp32 matrix in place (second half of the split-K projection head
// used when M is small: u = x.W^T is accumulated by 8 K-splits with fp32 atomics, then this warp-per-
// row pass adds the bias, normalises (F.normalize, eps 1e-12) and emits fp32 / bf16 / inv_norm).
// --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) bias_norm_rows_kernel(float* u, int ld_u, const float* bias, int M, int E,
                                                             int normalize, __nv_bfloat16* out_bf16, int ld_bf16,
                                                             float* inv_norm) {
    ptx::pdl_launch_dependents(); ptx::pdl_wait();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= M) return;
    const int nch = (E + 127) >> 7;
    float4 r[kMaxVec];
    float ssq = 0.f;
    float* row = u + static_cast<size_t>(warp) * ld_u;
#pragma unroll
    for (int c = 0; c < kMaxVec; ++c) {
        r[c] = make_float4(0.f, 0.f, 0.f, 0.f);
        const int e = (c * 32 + lane) * 4;
        if (c < nch && e < E) {
            r[c] = *reinterpret_cast<const float4*>(row + e);
            if (bias) {
                const float4 b = __ldg(reinterpret_cast<const float4*>(bias + e));
                r[c].x += b.x; r[c].y += b.y; r[c].z += b.z; r[c].w += b.w;
            }
        }
        ssq += r[c].x * r[c].x + r[c].y * r[c].y + r[c].z * r[c].z + r[c].w * r[c].w;
    }
    ssq = warp_sum(ssq);
    const float denom = normalize ? fmaxf(sqrtf(ssq), 1e-12f) : 1.f;
    if (lane == 0 && inv_norm) inv_norm[warp] = 1.f / denom;
#pragma unroll
    for (int c = 0; c < kMaxVec; ++c) {
        const int e = (c * 32 + lane) * 4;
        if (c < nch && e < E) {
            const float4 t = make_float4(r[c].x / denom, r[c].y / denom, r[c].z / denom, r[c].w / denom);
            *reinterpret_cast<float4*>(row + e) = t;
            if (out_bf16) store_bf16x4(out_bf16 + static_cast<size_t>(warp) * ld_bf16 + e, t);
        }
    }
}

}  // namespace cvcl
