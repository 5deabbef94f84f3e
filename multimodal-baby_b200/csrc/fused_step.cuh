// The flat contrastive train step as ONE persistent kernel (sm_100a).
//
// reference: MultiModalModel.calculate_contrastive_loss (multimodal/multimodal.py:796-822) + loss.backward()
// for embedding_type = "flat": text encoder (:496-503), projection head (:186-192), F.normalize (:736,:743),
// similarity + symmetric InfoNCE (:755,:783-787,:801-818) and their autograd (SURVEY 8 rows a1-a14).
//
// Why one kernel: at 512 pairs the step is ~3.2 GFLOP / ~31 MB (about 5 us of roofline work) and the
// ten-kernel version spent its 78 us on launch gaps, per-launch TMEM/barrier set-up and 16-32-CTA grids
// (profiles/r01_step_phases_n1.txt).  Here one co-resident grid (one CTA per SM, cooperative launch) walks
// through the phases with grid-wide barriers (one atomic counter in L2); TMEM, the mbarrier ring and the
// tensor maps are set up once.  No atomics on data anywhere: every reduction is a fixed-order sum, so the
// whole step is bit-reproducible.
//
//   P0  head GEMM, split over the contraction so that ~128 CTAs each stream 1/KS of K (tcgen05, fp32
//       partial tile -> its own slab by TMA store: no atomics, no memset)   ||   text encoder on the two
//       auxiliary warps of every CTA and, before the accumulator arrives, on the epilogue warps (one warp per
//       utterance, 12 table rows in flight per lane)   ||   zeroing of the token-count matrix
//   P1  slab sum (fixed order) + bias + L2 normalise -> bf16 image features, 1/norm (warp per row); the same
//       warp writes row r of the token-count matrix C[r, v] = #{l : ids[r,l] = v != 0} (bf16, exact)
//   P2  similarity tiles: both directions as row problems (direction 0: images x texts, direction 1:
//       texts x images), the 128x128 fp32 tile stays in TMEM; online-softmax row statistics per tile
//   P3  merge the statistics (row LSEs of both directions), dL/dlogits from the SAME TMEM tile (no
//       recompute GEMM), written as the bf16 A operand straight into swizzled shared memory, then
//       dQ_partial = Gs_tile . K_block (tcgen05) -> slab by TMA store.  P2/P3 run on QS CTAs per tile, each
//       owning E/QS output columns of dQ (the tile GEMM is repeated: latency, not flops, is the limit here)
//   P4  slab sum + the diagonal of G in fp32 + F.normalize backward; image rows -> bf16 du (operand of dW) and
//       per-CTA bias partials; text rows -> /len -> bf16 dm (operand of the embedding gradient)
//   P5  dW = du^T x  and  d table = C^T dm  (the embedding-bag backward as a GEMM against the token counts:
//       nn.Embedding(padding_idx=0) semantics fall out of C[:,0] = 0), both operands MN-major, read in place,
//       fp32 tiles by TMA store; the last CTA adds the per-block partial sums of loss / accuracy / entropy /
//       ds / db in a fixed order.
//
// Sharded use (SURVEY 8e) enters through the same code: Q = the local pairs, K = the gathered features,
// diag_off = rank * B (see StepParams::kf16 / part_all).  Nothing is exchanged by a separate kernel: P0 / P1 store each
// feature row into every rank's gathered buffers, P2 stores its softmax partials into every rank's copy (the column
// LSEs of P3 are merged from those), P5 stores each partial gradient tile into the scratch of the rank that owns it and
//   P6  (sharded only) the owner adds the `world` partial tiles in rank order and stores the sum into every rank's
//       gradient block; the scalars and d bias go one-shot.
// Four of the grid barriers then also span the ranks (flag words over NVLink, grid_sync with xstage >= 0).
#pragma once
#include "gemm_sm100.cuh"
#include "kernels_simt.cuh"

namespace cvcl {
namespace fused {

// Helpers are force-inlined: every phase runs once per launch, so the kernel is one long instruction stream
// and the sequential instruction prefetch only works on fall-through code (measured at 512 pairs: 40.4 us
// with the helpers inlined vs 43.1 us as shared functions, although the latter is smaller).
#ifdef CVCL_FUSED_NOINLINE
#define CVCL_HELPER __device__ __noinline__
#else
#define CVCL_HELPER __device__ __forceinline__
#endif
constexpr int kThreads = 256;                    // warp 0 TMA, warp 1 MMA + TMEM, warps 2..5 epilogue, 6..7 auxiliary
constexpr int kWarps = kThreads / 32;
constexpr int kStages = 4;
constexpr int kStages2 = 6;                       // P2 only: the Gs region is idle then and extends the ring
constexpr int kStageBytes = 32768;               // A 128x64 bf16 + B 128x64 bf16 (or one 64 x 256 MN-major slab)
constexpr int kRingBytes = kStages * kStageBytes;
constexpr int kGsOff = kRingBytes;               // dL/dlogits as the A operand: up to 2 tiles x 2 k-chunks x 16 KB
constexpr int kGsBytes = 65536;
constexpr int kMiscOff = kGsOff + kGsBytes;
constexpr int kMiscBytes = 20480;
constexpr int kSmemBytes = kMiscOff + kMiscBytes + 1024;     // + alignment slack
constexpr int kMaxT = 2;                         // similarity tiles per CTA (same row block)
constexpr int kNumSync = 8;
constexpr int kSmall = 8 + 4 + 512 + 4;          // out5 | ds | d bias (E <= 512), padded: one-shot exchange block per rank

struct alignas(64) StepMaps {
    CUtensorMap x_k;         // x16   [B, K]        box 64 x 128   (P0 A)
    CUtensorMap w_k;         // w16   [E, K]        box 64 x 128   (P0 B)
    CUtensorMap hp_out;      // hpart [KS*Bp, E] f32 box 32 x 128  (P0 out)
    CUtensorMap q_k[2];      // local features of direction z (0: images, 1: texts) [B, E] box 64 x 128 (P2 A)
    CUtensorMap kf_k[2];     // key features of direction z (0: texts, 1: images) [Bg, E] box 64 x 128 (P2 B)
    CUtensorMap kf_mn[2];    // the same tensors, box 64 x 64 (P3 B, MN-major)
    CUtensorMap dq_out;      // dqpart [2*nPart*Bp, E] f32 box 32 x 128 (P3 out)
    CUtensorMap du_mn;       // du16 [B, E]  box 64 x 64  (P5 A, MN-major)
    CUtensorMap x_mn;        // x16  [B, K]  box 64 x 64  (P5 B, MN-major)
    CUtensorMap dw_out;      // dW [E, K] f32 box 32 x 128 (P5 out)
    CUtensorMap c_mn;        // token counts C [B, V] bf16 (ld Vp) box 64 x 64 (P5 A, MN-major)
    CUtensorMap dm_mn;       // dm16 [B, E] box 64 x 64 (P5 B, MN-major)
    CUtensorMap dt_out;      // d table [V, E] f32 box 32 x 128 (P5 out)
};

struct StepParams {
    // ---- inputs
    const long long* ids; const long long* lens; const float* table; const float* bias;
    const float* log_scale_dev;          // device scalar s (nullable: use log_scale)
    float log_scale;
    int B, L, E, K, V, normalize, need_grads;
    int Bg, diag_off;                    // global batch and the column offset of the local positives
    // ---- derived tiling
    int Bp;                              // B rounded up to 128
    int nMB, nEB, nCB;                   // row blocks (local), E / 128, column blocks (global)
    int KS, kc_per_split, num_kc;        // head split-K
    int T, nPart;                        // similarity tiles per CTA, partial slabs per row block
    int QS;                              // CTAs per similarity tile; each owns E / QS columns of dQ
    int Vp;                              // leading dimension of the token-count matrix (V rounded up to 8)
    int dw_bn;                           // 64 or 128: width of a dW tile
    int phase_limit;                     // measurement / debugging: leave after phase k (0 = run all)
    // ---- workspace
    float* hpart;                        // [KS][Bp][E]
    __nv_bfloat16* q16[2]; int ldq;      // local features, bf16 (0: img16, 1: txt16)
    const __nv_bfloat16* kf16[2]; int ldk;   // key features (0: texts, 1: images) [Bg, ldk]
    float* invn[2];                      // [Bp] 1 / max(||u||, 1e-12) per direction
    RowStat* part[2];                    // [nCB][Bp]
    float* diag[2];                      // [Bp] logit at the positive
    float* lse[2];                       // [Bp] (local rows)
    float* gdiag[2];                     // [Bp] bf16(Gs_ii) as P3 put it into the dQ operand (local rows)
    // sharded only (null on one GPU): the (max, sum) softmax partials of EVERY row of direction z, gathered:
    // part_all[z][partial 0..2*nCB)[global row 0..Bg) -- P2 stores its partials into every rank's copy, so the column
    // LSEs of P3 (rows that other ranks own, SURVEY 8e) need no exchange phase of their own
    const float2* part_all[2];
    // ---- sharding (SURVEY 8e): rank `rank` of `world` owns pairs [diag_off, diag_off + B) of the global batch.
    // Every rank maps every rank's gathered buffers (symmetric memory over NVLink): the phases that PRODUCE
    // features / LSEs store them straight into all ranks' buffers, and the grid barrier that follows carries a
    // cross-rank stage.  world == 1: the tables hold the local buffers and nothing crosses a link.
    int world, rank;
    __nv_bfloat16* peer_kf[2][8];        // [z][p]: rank p's gathered key features of direction z ([Bg, ldk])
    float2* peer_part[2][8];             // [z][p]: rank p's part_all[z]
    unsigned int* peer_flags[8];         // rank p's flag words [4 stages][8 source ranks], epochs only grow
    unsigned int* epoch;                 // local: launches completed so far (this launch signals epoch + 1)
    // gradient sum over the ranks inside the kernel (sharded, reduce != 0).  Tile t of P5 (a 128 x 128 fp32 block of
    // dW or d table) is OWNED by rank t % world: every rank stores its partial tile straight from P5's epilogue into
    // the owner's scratch [source rank][slot t / world][128][128] (row stores over NVLink), a cross-rank barrier
    // follows, the owner adds the `world` partials in RANK order (bit-identical everywhere) and stores the sum into
    // the final dW / d table of EVERY rank (peer_stats[q] = rank q's block [out5(8) | ds(4) | db(E) | d table | dW]);
    // the closing cross-rank barrier makes the sums visible and fences the reuse of all exchange buffers.  The
    // scalars and d bias (8 + 4 + E floats) go one-shot: each rank stores its partials into slot `rank` of every
    // rank's peer_small [world][kSmall] and adds them up locally.
    float* peer_stats[8];
    float* peer_scratch[8];
    float* peer_small[8];
    unsigned long long xtimeout_ns;      // a cross-rank barrier that waits longer sets *fault and traps (a rank may
                                         // legitimately stall between steps: the default is NCCL-watchdog sized)
    int reduce;                          // 0: outputs are this rank's partial sums; 1: summed over the ranks in P6
    int nslot;                           // scratch slots per source rank = ceil(P5 tiles / world)
    float* rb_part;                      // [2*nMB][6]
    float* dspart;                       // [nMB*nPart]
    float* dqpart;                       // [2][nPart][Bp][E]
    __nv_bfloat16* du16;                 // [Bp][E]
    __nv_bfloat16* dm16;                 // [Bp][E]  d mean-embedding / len (text side)
    __nv_bfloat16* cmat;                 // [Bp][Vp] token counts
    float* dbpart;                       // [grid][E]
    unsigned int* sync;                  // [kNumSync] zero on entry, left zero on exit
    unsigned long long* timing;          // [48] globaltimer stamps of CTA 0 (nullable): [0..15] barriers, [16..] in-phase
    int* status;                         // out-of-range token id -> 1 (nullable)
    int* fault;                          // barrier time-out code (nullable)
    // ---- outputs
    float* out5;                         // loss, image_accuracy, text_accuracy, image_entropy, text_entropy
    float* img_f32; float* txt_f32;      // [B,E] fp32 features (nullable)
    float* dW; float* dbias; float* dtable; float* dscale;
    float inv_rows;                      // 1 / Bg
};

// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ unsigned int ld_acquire_gpu(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }

// bounded mbarrier wait: a protocol bug traps (loud failure) instead of hanging the device
__device__ __forceinline__ void mbar_wait_b(uint64_t* bar, uint32_t parity) {
    unsigned int it = 0;
    while (!ptx::mbar_try_wait(bar, parity)) {
        if (++it > 40000000u) __trap();
    }
}

// Grid-wide barrier k (k = 0, 1, ... in program order): every CTA is resident (cooperative launch, one
// CTA per SM), so spinning on one L2 counter cannot starve anybody.  Fence + add and an acquire-spin by
// thread 0 (measured 1.5 us; atom.add.release was slower); bar.sync makes the CTA's writes part of the release.  kWriterFence: this phase wrote global
// memory with ordinary stores that a later phase reads through TMA (async proxy), so every thread orders its
// stores against the async proxy first; the TMA-issuing thread fences again after the barrier.
__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// The spin of a grid barrier after its first 4096 failed probes (in practice a barrier completes long before):
// the globaltimer is sampled every 4096 probes from here on, and a wait longer than timeout_ns stores `code` into
// *fault and traps.  kSys: wait at system scope until the word has reached `target` as a wrapping epoch (cross-rank
// flags, sharded instance only); else at GPU scope until the counter is >= target.  Out of line because a step never
// gets here: inlined, this fault path sat in every barrier of the instruction stream that each launch fetches again
// after the L2 flush between steps.
template <bool kSys>
__device__ __noinline__ void grid_wait_cold(const unsigned int* w, unsigned int target, unsigned long long timeout_ns,
                                            int* fault, int code) {
    const unsigned long long t0 = globaltimer_ns();
    unsigned int it = 0;
    while (kSys ? static_cast<int>(ld_acquire_sys(w) - target) < 0 : ld_acquire_gpu(w) < target) {
        if ((++it & 4095u) == 0 && globaltimer_ns() - t0 > timeout_ns) {
            if (fault) atomicExch(fault, code);
            __threadfence_system();
            __trap();
        }
    }
}

// xstage >= 0 (sharded runs; only the kSharded instance has this code): the barrier also spans the ranks.  Every
// CTA fences its stores at system scope before it arrives; the LAST local arrival (it has seen all the others
// through the counter) stores this launch's epoch into flag word [xstage][rank] of every peer, and every CTA then also waits until its own
// words [xstage][peer] carry the epoch: all stores a peer issued before ITS barrier have landed here.
template <bool kWriterFence, bool kSharded>
CVCL_HELPER void grid_sync(const StepParams& p, int k, int xstage = -1, unsigned int epoch = 0) {
    if (kWriterFence) fence_proxy_async_all();
    __syncthreads();
    if (threadIdx.x < 32) {
        // warp 0: lane 0 arrives on the local counter; in a cross-rank barrier lane q talks to rank q, so the `world`
        // signals and the `world` polls run side by side instead of one release (fence + store) after the other
        // (measured at 8 ranks: ~14 us per barrier for seven serial releases)
        const int lane = threadIdx.x;
        const bool cross = kSharded && xstage >= 0 && p.world > 1;
        const unsigned int target = static_cast<unsigned int>(k + 1) * gridDim.x;
        unsigned int prev = 0;
        if (lane == 0) {
            if (cross) __threadfence_system(); else __threadfence();
            prev = atomicAdd(p.sync, 1u);
        }
        prev = __shfl_sync(0xffffffffu, prev, 0);
        __syncwarp();                       // memory ordering lane 0 -> the signalling lanes (shfl alone gives none)
        if (cross) {
            const bool peer = lane < p.world && lane != p.rank;
            // the LAST local arrival has seen every other CTA's arrival (each behind that CTA's system-scope fence):
            // its release stores publish the whole rank's writes
            if (prev == target - 1 && peer) st_release_sys(p.peer_flags[lane] + xstage * 8 + p.rank, epoch);
            if (peer) {
                const unsigned int* w = p.peer_flags[p.rank] + xstage * 8 + lane;
                unsigned int it = 0;
#pragma unroll 1
                while (static_cast<int>(ld_acquire_sys(w) - epoch) < 0) {
                    if (++it == 4096u) {              // fault code 200 + 10 xstage + lane: a peer never reached this step
                        grid_wait_cold<true>(w, epoch, p.xtimeout_ns, p.fault, 200 + 10 * xstage + lane);
                        break;
                    }
                }
            }
            __syncwarp();
        }
        if (lane == 0) {
            unsigned int it = 0;
#pragma unroll 1
            while (ld_acquire_gpu(p.sync) < target) {
                if (++it == 4096u) {                  // fault code 100 + k after 2 s: a CTA never arrived
                    grid_wait_cold<false>(p.sync, target, 2000000000ull, p.fault, 100 + k);
                    break;
                }
            }
            fence_proxy_async_all();                                  // thread 0 = warp 0 lane 0 issues the TMA loads
            if (blockIdx.x == 0 && p.timing) p.timing[k + 1] = globaltimer_ns();
        }
        __syncwarp();
    }
    __syncthreads();
}

struct Ring {
    int stage; uint32_t phase;
    __device__ __forceinline__ void next() { if (++stage == kStages) { stage = 0; phase ^= 1u; } }
};

// one utterance per warp: feat = normalise(sum_l table[ids[b,l]] / len[b]) in position order
// (same arithmetic, same order as text_encoder_fwd_kernel; E <= 512)
template <bool kSharded>
CVCL_HELPER void text_row(const StepParams& p, int b, int lane) {
    const int nch = p.E >> 7;
    constexpr int kInFlight = 12;          // covers half of the utterances (mean length 14) in one round trip
    float4 acc[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    const long long* idrow = p.ids + static_cast<size_t>(b) * p.L;
    const float flen = static_cast<float>(__ldg(p.lens + b));          // fetched with the ids, used at the end
    for (int l0 = 0; l0 < p.L; l0 += 32) {
        long long my_id = (l0 + lane < p.L) ? __ldg(idrow + l0 + lane) : 0;
        if (my_id < 0 || my_id >= p.V) { if (p.status) atomicExch(p.status, 1); my_id = 0; }
        unsigned live = __ballot_sync(0xffffffffu, my_id != 0 && l0 + lane < p.L);
        while (live) {
            float4 r[kInFlight][4];
#pragma unroll
            for (int k = 0; k < kInFlight; ++k) {
                int src_lane = -1;
                if (live) { src_lane = __ffs(live) - 1; live &= live - 1; }
                const long long id = __shfl_sync(0xffffffffu, my_id, src_lane < 0 ? 0 : src_lane);
                const float4* src = reinterpret_cast<const float4*>(p.table + static_cast<size_t>(id) * p.E);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    r[k][c] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (src_lane >= 0 && c < nch) r[k][c] = __ldg(src + c * 32 + lane);
                }
            }
#pragma unroll
            for (int k = 0; k < kInFlight; ++k)
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    acc[c].x += r[k][c].x; acc[c].y += r[k][c].y; acc[c].z += r[k][c].z; acc[c].w += r[k][c].w;
                }
        }
    }
    // one reciprocal per row, then multiplies (the reference divides element-wise: at most 1 ulp apart)
    const float rlen = 1.f / flen;
    float ssq = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        acc[c].x *= rlen; acc[c].y *= rlen; acc[c].z *= rlen; acc[c].w *= rlen;
        ssq += acc[c].x * acc[c].x + acc[c].y * acc[c].y + acc[c].z * acc[c].z + acc[c].w * acc[c].w;
    }
    ssq = warp_sum(ssq);
    const float inv = p.normalize ? 1.f / fmaxf(sqrtf(ssq), 1e-12f) : 1.f;
    if (lane == 0) p.invn[1][b] = inv;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        if (c < nch) {
            const int e = (c * 32 + lane) * 4;
            const float4 t = make_float4(acc[c].x * inv, acc[c].y * inv, acc[c].z * inv, acc[c].w * inv);
            if (p.txt_f32) *reinterpret_cast<float4*>(p.txt_f32 + static_cast<size_t>(b) * p.E + e) = t;
            for (int pp = 0; pp < (kSharded ? p.world : 1); ++pp)      // texts are the keys of direction 0
                store_bf16x4(p.peer_kf[0][pp] + static_cast<size_t>(p.diag_off + b) * p.ldk + e, t);
        }
    }
}

// fp32 accumulator columns [tc0, tc0 + ncols) of this thread's row -> swizzled staging columns [sc0, sc0 + ncols)
// (boxes of 32 fp32 columns, 128 rows each)
CVCL_HELPER void stage_f32_cols(uint32_t tmem_row, int tc0, int sc0, int ncols, unsigned char* stage, int row) {
#pragma unroll 1
    for (int c = 0; c < ncols; c += 32) {
        float v[32];
        ptx::tmem_ld_32x32(tmem_row + tc0 + c, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            uint4 q;
            q.x = __float_as_uint(v[4 * j]); q.y = __float_as_uint(v[4 * j + 1]);
            q.z = __float_as_uint(v[4 * j + 2]); q.w = __float_as_uint(v[4 * j + 3]);
            swz_st16(stage, row, (sc0 + c + 4 * j) * 4, q);
        }
    }
}

// v[i] for a per-thread i in [0, 32): a select tree over the five bits of i, 31 selects (a 32-way compare / select
// scan takes twice the instructions, and indexing v with i would put it in local memory)
CVCL_HELPER float select32(const float (&v)[32], int i) {
    float s[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) s[q] = (i & 1) ? v[2 * q + 1] : v[2 * q];
#pragma unroll
    for (int b = 1; b < 5; ++b)
#pragma unroll
        for (int q = 0; q < (16 >> b); ++q) s[q] = ((i >> b) & 1) ? s[2 * q + 1] : s[2 * q];
    return s[0];
}

// online merge of per-tile softmax partials (strict >: the first tile wins ties, as torch.argmax does);
// the partials are fetched first (independent loads), then merged in tile order
CVCL_HELPER void merge_stats(const RowStat* base, size_t stride, int n, float& gm, float& gl, float& ga,
                                            int& garg) {
    gm = -INFINITY; gl = 0.f; ga = 0.f; garg = 0x7fffffff;
    for (int t0 = 0; t0 < n; t0 += 8) {
        float4 q[8];
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (t0 + k < n) q[k] = __ldcg(reinterpret_cast<const float4*>(base + static_cast<size_t>(t0 + k) * stride));
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (t0 + k < n) {
                const float rm = q[k].x, rl = q[k].y, ra = q[k].z; const int rarg = __float_as_int(q[k].w);
                if (rm > gm) { const float w = __expf(gm - rm); gl = gl * w + rl; ga = ga * w + ra; gm = rm; garg = rarg; }
                else { const float w = __expf(rm - gm); gl = fmaf(rl, w, gl); ga = fmaf(ra, w, ga); }
            }
        }
    }
}

__device__ __forceinline__ uint4 ld_relaxed_sys_v4(const uint4* q) {
    uint4 v;
    asm volatile("ld.global.relaxed.sys.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(q) : "memory");
    return v;
}

// log-sum-exp of one row from its gathered (max, sum) partials
CVCL_HELPER float merge_ml(const float2* base, size_t stride, int n) {
    float gm = -INFINITY, gl = 0.f;
    for (int t0 = 0; t0 < n; t0 += 8) {
        float2 q[8];
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (t0 + k < n) q[k] = __ldcg(base + static_cast<size_t>(t0 + k) * stride);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (t0 + k < n) {
                const float rm = q[k].x, rl = q[k].y;
                if (rm > gm) { gl = gl * __expf(gm - rm) + rl; gm = rm; }
                else gl = fmaf(rl, __expf(rm - gm), gl);
            }
        }
    }
    return gm + logf(gl);
}

#define CVCL_STAMP(i) do { if (cta == 0 && p.timing) p.timing[i] = globaltimer_ns(); } while (0)

// Two instances: kSharded = true serves the sharded entry (any world size, world 1 included) and keeps every
// cross-rank path; kSharded = false is the single-GPU step, compiled without them.  The phases run once per launch
// and the L2 flush between training steps evicts the code too, so every SASS byte of a path that the single-GPU
// step never takes is still fetched on the way through (the sharded-only code is a quarter of the kernel).
template <bool kSharded>
__global__ void __launch_bounds__(kThreads, 1)
flat_step_kernel(const __grid_constant__ StepMaps maps, const __grid_constant__ StepParams p) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    unsigned char* misc = smem + kMiscOff;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(misc);             // [kStages]
    uint64_t* empty_bar = full_bar + kStages;                            // [kStages]
    uint64_t* tfull_bar = empty_bar + kStages;                           // accumulator complete
    uint64_t* gs_bar = tfull_bar + 1;                                    // Gs tiles written, S tile consumed
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(gs_bar + 1);
    int* s_next = reinterpret_cast<int*>(misc + 128);                    // [kWarps] work-queue tickets
    uint64_t* full2_bar = reinterpret_cast<uint64_t*>(misc + 160);       // [kStages2] P2 ring (ring + idle Gs region)
    uint64_t* empty2_bar = full2_bar + kStages2;                         // [kStages2]
    float* lk = reinterpret_cast<float*>(misc + 256);                    // [256] column LSE terms (P3)
    float* red = reinterpret_cast<float*>(misc + 256 + 1024);            // [64] block reductions
    float* sdb = reinterpret_cast<float*>(misc + 2048);                  // [kWarps][512] bias partials (P4)

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int G = gridDim.x;
    const int cta = blockIdx.x;

    if (threadIdx.x == 0) {
        if (cta == 0 && p.timing) p.timing[0] = globaltimer_ns();
        for (int s = 0; s < kStages; ++s) { ptx::mbar_init(&full_bar[s], 1); ptx::mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < kStages2; ++s) { ptx::mbar_init(&full2_bar[s], 1); ptx::mbar_init(&empty2_bar[s], 1); }
        ptx::mbar_init(tfull_bar, 1);
        ptx::mbar_init(gs_bar, kThreads);
        ptx::fence_mbar_init();
        ptx::prefetch_tmap(&maps.x_k); ptx::prefetch_tmap(&maps.w_k); ptx::prefetch_tmap(&maps.hp_out);
    }
    if (warp == 1) ptx::tmem_alloc<512>(tmem_ptr_smem);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    Ring ring{0, 0};                       // producer and MMA issuer walk the same sequence of stages
    uint32_t tfull_uses = 0;               // MMA issuer and epilogue warps count accumulator hand-overs alike
    // Epilogue work is shared by ALL eight warps: a warp may only touch TMEM lanes 32*(warp%4)..+31, so two
    // warps serve each lane quadrant and split the columns of a tile in halves (warps 2..5: half 0, warps
    // 0, 1, 6, 7: half 1; the TMA / MMA warps join once their lane 0 has issued everything).  One warp per
    // scheduler cannot hide the TMEM / MUFU latencies of these passes (measured: 0.62 us per 32 columns).
    const int quad = warp & 3;
    const int half = (warp >= 2 && warp < 6) ? 0 : 1;
    const int row = quad * 32 + lane;      // accumulator row of this thread
    const uint32_t tmem_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    float* lrow = reinterpret_cast<float*>(misc + 256 + 1024 + 256);     // [128] row LSE terms shared by the halves (P3)
    const float s_log = p.log_scale_dev ? __ldg(p.log_scale_dev) : p.log_scale;
    const float scale = expf(s_log);
    constexpr float kLog2e = 1.4426950408889634f;
    int sync_k = 0;
    // cross-rank flag value of this launch (sharded runs; every CTA reads it before any CTA can bump it at exit)
    const bool reduce = kSharded && p.reduce;        // sum the gradients over the ranks in P5 / P6
    const unsigned int xepoch = (kSharded && p.epoch) ? *reinterpret_cast<volatile unsigned int*>(p.epoch) + 1u : 0u;

    if (p.phase_limit == 100) {            // measurement: the cost of the grid barrier alone
#pragma unroll 1                           // one barrier body in the instruction stream, not six
        for (int i = 0; i < 6; ++i) grid_sync<false, kSharded>(p, sync_k++);
        goto done;
    }

    // ============================================================================ P0
    {
        const int n_items = p.nMB * p.nEB * p.KS;
        const bool has = cta < n_items;
        const int ks = cta / (p.nMB * p.nEB);
        const int tile = cta % (p.nMB * p.nEB);
        const int mb = tile / p.nEB, nb = tile % p.nEB;
        const int kc0 = ks * p.kc_per_split;
        const int kc1 = min(kc0 + p.kc_per_split, p.num_kc);
        if (warp == 0) {
            if (lane == 0 && has) {
                for (int kc = kc0; kc < kc1; ++kc) {
                    mbar_wait_b(&empty_bar[ring.stage], ring.phase ^ 1u);
                    unsigned char* sa = smem + ring.stage * kStageBytes;
                    ptx::mbar_arrive_expect_tx(&full_bar[ring.stage], kStageBytes);
                    ptx::tma_load_2d(sa, &maps.x_k, &full_bar[ring.stage], kc * kBK, mb * kBM);
                    ptx::tma_load_2d(sa + 16384, &maps.w_k, &full_bar[ring.stage], kc * kBK, nb * 128);
                    ring.next();
                }
            }
            __syncwarp();
        } else if (warp == 1) {
            if (lane == 0 && has) {
                constexpr uint32_t idesc = ptx::make_idesc_bf16(kBM, 128, false, false);
                for (int kc = kc0; kc < kc1; ++kc) {
                    mbar_wait_b(&full_bar[ring.stage], ring.phase);
                    ptx::tc_fence_after();
                    const uint32_t sa = ptx::smem_u32(smem + ring.stage * kStageBytes);
                    const uint64_t adesc = ptx::make_kmajor_sw128_desc(sa);
                    const uint64_t bdesc = ptx::make_kmajor_sw128_desc(sa + 16384);
#pragma unroll
                    for (int k = 0; k < kBK / kUmmaK; ++k)
                        ptx::umma_bf16(tmem_base, adesc + 2 * k, bdesc + 2 * k, idesc, (kc > kc0 || k > 0) ? 1u : 0u);
                    ptx::umma_commit(&empty_bar[ring.stage]);
                    if (kc == kc1 - 1) ptx::umma_commit(tfull_bar);
                    ring.next();
                }
            }
            __syncwarp();
        }
        // zero this CTA's slice of the token-count matrix (filled in P1, consumed in P5)
        if (p.need_grads) {
            const size_t n16 = static_cast<size_t>(p.B) * p.Vp * 2 / 16;
            uint4* dst = reinterpret_cast<uint4*>(p.cmat);
            for (size_t i = static_cast<size_t>(cta) * kThreads + threadIdx.x; i < n16; i += static_cast<size_t>(G) * kThreads)
                dst[i] = make_uint4(0u, 0u, 0u, 0u);
        }
        // text encoder: one warp per utterance, static assignment -- slot j of CTA c owns utterance j*G + c and
        // the slots go to the auxiliary warps first (6, 7), then to the epilogue warps (2..5), which encode
        // theirs before the accumulator of the head tile is ready (~2 us after the loads were issued anyway).
        // (Measured alternative: only the auxiliary warps here and the rest on P1's idle warps -- P0 -0.6 us,
        // P1 +1.6 us, dropped.)
        if (warp >= 2) {
            const int slot = warp >= 6 ? warp - 6 : warp;
            for (int u = slot * G + cta; u < p.B; u += 6 * G) text_row<kSharded>(p, u, lane);
            if (warp == 2 && lane == 0) CVCL_STAMP(18);
        }
        if (has) {                                          // all eight warps drain the head tile
            mbar_wait_b(tfull_bar, tfull_uses & 1u);
            ptx::tc_fence_after();
            if (threadIdx.x == 64) CVCL_STAMP(16);
            stage_f32_cols(tmem_row, 64 * half, 64 * half, 64, smem, row);   // the ring is idle: all MMAs have retired
            ptx::fence_proxy_async_smem();
            ptx::tc_fence_before();
            __syncthreads();
            if (threadIdx.x == 64) {
#pragma unroll
                for (int b4 = 0; b4 < 4; ++b4)
                    ptx::tma_store_2d(&maps.hp_out, smem + b4 * 16384, nb * 128 + b4 * 32, ks * p.Bp + mb * kBM);
                tma_store_commit();
                tma_store_wait_all();
                CVCL_STAMP(17);
            }
        }
        if (has) ++tfull_uses;
    }
    // (the ring state is only ever used by lane 0 of warps 0 and 1, which walk identical sequences)
    grid_sync<true, kSharded>(p, sync_k++);
    if (p.phase_limit == 1) goto done;

    // ============================================================================ P1
    {
        const int nch = p.E >> 7;
        const size_t slab = static_cast<size_t>(p.Bp) * p.E;
        for (int r = cta * kWarps + warp; r < p.B; r += G * kWarps) {
            float4 acc[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[c] = make_float4(0.f, 0.f, 0.f, 0.f);
            const float* base = p.hpart + static_cast<size_t>(r) * p.E;
            // the token ids of the row (for the count matrix below) are fetched with the slabs
            const long long id0 = (p.need_grads && lane < p.L) ? __ldg(p.ids + static_cast<size_t>(r) * p.L + lane) : 0;
            for (int k0 = 0; k0 < p.KS; k0 += 8) {
                float4 v[8][4];
#pragma unroll
                for (int k = 0; k < 8; ++k)
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        v[k][c] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (k0 + k < p.KS && c < nch)
                            v[k][c] = __ldcg(reinterpret_cast<const float4*>(base + (k0 + k) * slab) + c * 32 + lane);
                    }
#pragma unroll
                for (int k = 0; k < 8; ++k)
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        acc[c].x += v[k][c].x; acc[c].y += v[k][c].y; acc[c].z += v[k][c].z; acc[c].w += v[k][c].w;
                    }
            }
            float ssq = 0.f;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                if (c < nch && p.bias) {
                    const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias) + c * 32 + lane);
                    acc[c].x += b4.x; acc[c].y += b4.y; acc[c].z += b4.z; acc[c].w += b4.w;
                }
                ssq += acc[c].x * acc[c].x + acc[c].y * acc[c].y + acc[c].z * acc[c].z + acc[c].w * acc[c].w;
            }
            ssq = warp_sum(ssq);
            const float inv = p.normalize ? 1.f / fmaxf(sqrtf(ssq), 1e-12f) : 1.f;
            if (lane == 0) p.invn[0][r] = inv;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                if (c < nch) {
                    const int e = (c * 32 + lane) * 4;
                    const float4 t = make_float4(acc[c].x * inv, acc[c].y * inv, acc[c].z * inv, acc[c].w * inv);
                    if (p.img_f32) *reinterpret_cast<float4*>(p.img_f32 + static_cast<size_t>(r) * p.E + e) = t;
                    for (int pp = 0; pp < (kSharded ? p.world : 1); ++pp)  // images are the keys of direction 1
                        store_bf16x4(p.peer_kf[1][pp] + static_cast<size_t>(p.diag_off + r) * p.ldk + e, t);
                }
            }
            if (p.need_grads) {
                // row r of the token-count matrix: C[r, v] = #{l : ids[r, l] = v}, v != 0 (this warp owns the row)
                __nv_bfloat16* crow = p.cmat + static_cast<size_t>(r) * p.Vp;
                const long long* idrow = p.ids + static_cast<size_t>(r) * p.L;
                for (int l0 = 0; l0 < p.L; l0 += 32) {
                    const long long id = l0 == 0 ? id0 : ((l0 + lane < p.L) ? __ldg(idrow + l0 + lane) : 0);
                    const bool valid = id > 0 && id < p.V;
                    const unsigned grp = __match_any_sync(0xffffffffu, valid ? static_cast<int>(id) : -1 - lane);
                    if (valid && lane == __ffs(grp) - 1) {
                        float cnt = static_cast<float>(__popc(grp));
                        if (l0 > 0) cnt += __bfloat162float(crow[id]);     // earlier chunk of a long utterance
                        crow[id] = __float2bfloat16_rn(cnt);
                    }
                    __syncwarp();
                }
            }
        }
        if (threadIdx.x == 0) CVCL_STAMP(19);
    }
    grid_sync<true, kSharded>(p, sync_k++, 0, xepoch);               // sharded: every rank's features are in place behind this
    if (p.phase_limit == 2) goto done;

    {
        // ======================================================================== P2
        // similarity CTA: direction z, local row block rb, partial index pi (column blocks pi*T + j), and
        // q = which E/QS columns of dQ this CTA produces in P3 (the S tile itself is computed by all QS CTAs)
        const int n_sim = 2 * p.nMB * p.nPart * p.QS;
        const bool has = cta < n_sim;
        const int qs = cta % p.QS;
        const int tix = cta / p.QS;
        const int z = tix / (p.nMB * p.nPart);
        const int rem = tix % (p.nMB * p.nPart);
        const int rb = rem / p.nPart, pi = rem % p.nPart;
        const int num_ke = p.E / kBK;
        const int M = p.B, N = p.Bg;
        const int m = rb * kBM + row;                       // local row of this epilogue thread
        const int dcol = m + p.diag_off;
        // this phase runs once per launch on its own 6-deep ring: 6 of the 8 k-chunks are in flight at once
        int st2 = 0; uint32_t ph2 = 0;
        if (warp == 0) {
            if (lane == 0 && has) {
                for (int j = 0; j < p.T; ++j)
                    for (int kc = 0; kc < num_ke; ++kc) {
                        mbar_wait_b(&empty2_bar[st2], ph2 ^ 1u);
                        unsigned char* sa = smem + st2 * kStageBytes;
                        ptx::mbar_arrive_expect_tx(&full2_bar[st2], kStageBytes);
                        ptx::tma_load_2d(sa, &maps.q_k[z], &full2_bar[st2], kc * kBK, rb * kBM);
                        ptx::tma_load_2d(sa + 16384, &maps.kf_k[z], &full2_bar[st2], kc * kBK, (pi * p.T + j) * 128);
                        if (++st2 == kStages2) { st2 = 0; ph2 ^= 1u; }
                    }
            }
            __syncwarp();
        } else if (warp == 1) {
            if (lane == 0 && has) {
                constexpr uint32_t idesc = ptx::make_idesc_bf16(kBM, 128, false, false);
                for (int j = 0; j < p.T; ++j)
                    for (int kc = 0; kc < num_ke; ++kc) {
                        mbar_wait_b(&full2_bar[st2], ph2);
                        ptx::tc_fence_after();
                        const uint32_t sa = ptx::smem_u32(smem + st2 * kStageBytes);
                        const uint64_t adesc = ptx::make_kmajor_sw128_desc(sa);
                        const uint64_t bdesc = ptx::make_kmajor_sw128_desc(sa + 16384);
#pragma unroll
                        for (int k = 0; k < kBK / kUmmaK; ++k)
                            ptx::umma_bf16(tmem_base + 128 * j, adesc + 2 * k, bdesc + 2 * k, idesc, (kc > 0 || k > 0) ? 1u : 0u);
                        ptx::umma_commit(&empty2_bar[st2]);
                        if (j == p.T - 1 && kc == num_ke - 1) ptx::umma_commit(tfull_bar);
                        if (++st2 == kStages2) { st2 = 0; ph2 ^= 1u; }
                    }
            }
            __syncwarp();
        }
        if (has) {
            mbar_wait_b(tfull_bar, tfull_uses & 1u);
            ptx::tc_fence_after();
            if (threadIdx.x == 64) CVCL_STAMP(20);
            if (qs == 0) {                                  // the statistics are written once per tile
                // raw-domain online softmax (see EpiSimStats); each thread owns 64 columns of its row, so a
                // 128-column tile contributes two partials per row: index (column block)*2 + half
                const float sc2 = scale * kLog2e;
                for (int j = 0; j < p.T; ++j) {
                    const int n0 = (pi * p.T + j) * 128 + 64 * half;
                    float mx = -INFINITY, l = 0.f, a = 0.f; int arg = n0;
#pragma unroll 1
                    for (int c = 0; c < 64; c += 32) {
                        float v[32];
                        ptx::tmem_ld_32x32(tmem_row + 128 * j + 64 * half + c, v);
                        const int n = n0 + c;
                        if (n >= N) continue;                               // warp-uniform
                        const bool full = n + 32 <= N;
                        if (!full) {
#pragma unroll
                            for (int q = 0; q < 32; ++q) if (n + q >= N) v[q] = -INFINITY;
                        }
                        float cm = v[0];
#pragma unroll
                        for (int q = 1; q < 32; ++q) cm = fmaxf(cm, v[q]);
                        if (cm > mx) {
                            int k = 31;
#pragma unroll
                            for (int q = 31; q >= 0; --q) if (v[q] == cm) k = q;
                            arg = n + k;
                        }
                        if (dcol >= n && dcol < n + 32 && m < M) p.diag[z][m] = select32(v, dcol - n) * scale;
                        const float nm = fmaxf(mx, cm);
                        const float corr = exp2f((mx - nm) * sc2);
                        l *= corr; a *= corr;
                        const float nm2 = nm * sc2;
#pragma unroll
                        for (int q = 0; q < 32; ++q) {
                            const float e = exp2f(fmaf(v[q], sc2, -nm2));
                            l += e;
                            a = fmaf(e, full ? v[q] : (n + q < N ? v[q] : 0.f), a);
                        }
                        mx = nm;
                    }
                    if (m < M) {
                        RowStat rs; rs.m = mx * scale; rs.l = l; rs.a = a * scale; rs.arg = arg;
                        const int pidx = (pi * p.T + j) * 2 + half;
                        p.part[z][static_cast<size_t>(pidx) * p.Bp + m] = rs;
                        if (kSharded && p.world > 1) {  // (max, sum) of this row's partial -> every rank's gathered copy
                            const size_t o = static_cast<size_t>(pidx) * p.Bg + p.diag_off + m;
                            for (int pp = 0; pp < p.world; ++pp) p.peer_part[z][pp][o] = make_float2(rs.m, rs.l);
                        }
                    }
                }
            }
            ptx::tc_fence_before();
            if (threadIdx.x == 64) CVCL_STAMP(21);
        }
        if (has) ++tfull_uses;
        grid_sync<false, kSharded>(p, sync_k++, 1, xepoch);          // sharded: every rank's softmax partials are in place behind this
        if (p.phase_limit == 3) goto done;

        // ======================================================================== P3
        const int wq = p.E / p.QS;                          // dQ columns of this CTA: [qs*wq, qs*wq + wq)
        const int nH = (wq + 255) / 256;
        const int num_kc3 = 2 * p.T;
        // the key-feature slabs of the dQ GEMM do not depend on anything computed in this phase: the producer fetches
        // as many as the ring holds NOW and the rest after its share of the Gs pass (it is an epilogue thread too:
        // waiting here for a slot that only the MMA can free -- which waits for the Gs pass -- would deadlock)
        const int n_fill3 = num_kc3 * nH;
        auto fill3 = [&](int idx) {
            const int kc = idx / nH, h = idx % nH;
            const int nh = min(256, wq - 256 * h);
            mbar_wait_b(&empty_bar[ring.stage], ring.phase ^ 1u);
            unsigned char* sb = smem + ring.stage * kStageBytes;
            ptx::mbar_arrive_expect_tx(&full_bar[ring.stage], static_cast<uint32_t>(nh) * 128);
            const int crow = (pi * p.T + (kc >> 1)) * 128 + (kc & 1) * 64;
            for (int jb = 0; jb < nh / 64; ++jb)
                ptx::tma_load_2d(sb + jb * 8192, &maps.kf_mn[z], &full_bar[ring.stage], qs * wq + 256 * h + 64 * jb, crow);
            ring.next();
        };
        if (has && p.need_grads && warp == 0 && lane == 0)
            for (int idx = 0; idx < min(n_fill3, kStages); ++idx) fill3(idx);
        __syncwarp();
        if (has) {
            // (a) half 0: the LSE of this thread's ROW (+ cross-entropy / entropy / accuracy terms on the lead
            //     CTA); half 1: the LSE of COLUMN `row` of the tile = a row of the other direction, merged here from
            //     its partials (one GPU: the local ones; sharded: the gathered (max, sum) pairs).  Both halves run
            //     at the same time on different warps: one round trip to L2 instead of three.
            const bool lead = pi == 0 && qs == 0;
            const float w = scale * (0.5f * p.inv_rows);             // exp(s) * coef
            const float l2w = log2f(w);
            float v6[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (half == 0) {
                float lse_row = 0.f;
                if (m < M) {
                    float gm, gl, ga; int garg;
                    const float dg = lead ? __ldcg(p.diag[z] + m) : 0.f;
                    merge_stats(p.part[z] + m, p.Bp, 2 * p.nCB, gm, gl, ga, garg);
                    lse_row = gm + logf(gl);
                    if (lead) {
                        p.lse[z][m] = lse_row;
                        v6[z] = lse_row - dg;
                        v6[2 + z] = lse_row - ga / gl;
                        v6[4 + z] = (garg == dcol) ? 1.f : 0.f;
                    }
                }
                lrow[row] = (m < M) ? lse_row * kLog2e - l2w : INFINITY;     // dead rows -> 0
            } else if (p.need_grads) {
                for (int j = 0; j < p.T; ++j) {
                    const int n = (pi * p.T + j) * 128 + row;
                    float lkv = INFINITY;
                    if (n < N) {
                        float lse_c;
                        if (kSharded && p.part_all[1 - z]) lse_c = merge_ml(p.part_all[1 - z] + n, p.Bg, 2 * p.nCB);
                        else {
                            float cm_, cl_, ca_; int carg_;
                            merge_stats(p.part[1 - z] + n, p.Bp, 2 * p.nCB, cm_, cl_, ca_, carg_);
                            lse_c = cm_ + logf(cl_);
                        }
                        lkv = lse_c * kLog2e - l2w;
                    }
                    lk[128 * j + row] = lkv;
                }
            }
            if (lead) {                                      // fixed-order block sum -> rb_part (half 0 warps: 2..5)
                if (half == 0) {
#pragma unroll
                    for (int i = 0; i < 6; ++i) {
                        const float sv = warp_sum(v6[i]);
                        if (lane == 0) red[(warp - 2) * 6 + i] = sv;
                    }
                }
            }
            __syncthreads();
            if (lead && threadIdx.x < 6)
                p.rb_part[(z * p.nMB + rb) * 6 + threadIdx.x] =
                    red[threadIdx.x] + red[6 + threadIdx.x] + red[12 + threadIdx.x] + red[18 + threadIdx.x];
            if (threadIdx.x == 64) CVCL_STAMP(22);
            if (p.need_grads) {
                // (c) Gs = w * (softmax_row + softmax_col) from the tile still in TMEM -> bf16 A operand; this
                //     thread's 64 columns are exactly k-chunk `half` of the operand
                const float lq = lrow[row];
                const float sc2 = scale * kLog2e;
                float ds = 0.f;
                for (int j = 0; j < p.T; ++j) {
                    unsigned char* gs_tile = smem + kGsOff + j * 32768;
                    const int n0 = (pi * p.T + j) * 128;
#pragma unroll 1
                    for (int c = 64 * half; c < 64 * half + 64; c += 32) {
                        float v[32];
                        ptx::tmem_ld_32x32(tmem_row + 128 * j + c, v);
                        const int n = n0 + c;
                        const bool has_diag = dcol >= n && dcol < n + 32;     // warp-uniform: one chunk per warp
                        const float dv = has_diag ? select32(v, dcol - n) : 0.f;
                        float g[32];
#pragma unroll
                        for (int q4 = 0; q4 < 8; ++q4) {
                            const float4 k4 = *reinterpret_cast<const float4*>(lk + 128 * j + c + 4 * q4);
                            const float kk[4] = {k4.x, k4.y, k4.z, k4.w};
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                const float r = v[4 * q4 + q];
                                const float gg = exp2f(fmaf(r, sc2, -lq)) + exp2f(fmaf(r, sc2, -kk[q]));
                                ds = fmaf(gg, r, ds);
                                g[4 * q4 + q] = gg;
                            }
                        }
                        // the diagonal stays in the bf16 operand; its rounded value goes to P4, which replaces it by the
                        // whole G_ii in fp32: w (P_row + P_col) and -2w nearly cancel when a pair is confident, and the
                        // bf16 rounding of the first would be left as the whole gradient.  G_ii is recomputed from dv by
                        // the expression that gave g[dcol - n] above (the same float, without a second 32-way scan)
                        if (has_diag && qs == 0 && m < M) {
                            const float gd = exp2f(fmaf(dv, sc2, -lq)) + exp2f(fmaf(dv, sc2, -lk[128 * j + dcol - n0]));
                            p.gdiag[z][m] = __bfloat162float(__float2bfloat16_rn(gd));
                        }
                        ds = fmaf(-2.f * w, dv, ds);
#pragma unroll
                        for (int q = 0; q < 4; ++q) swz_st16(gs_tile, row, (c + 8 * q) * 2, pack_bf16x8(g + 8 * q));
                    }
                }
                // dL/ds partial of this tile (direction 0 only).  Written BEFORE the arrival below: the reader (thread 64,
                // behind tfull_bar, which fires after gs_bar) is then ordered after every warp's write (racecheck found
                // the write after the arrival unordered)
                if (z == 0 && qs == 0) {
                    ds = warp_sum(ds);
                    if (lane == 0) red[32 + warp] = ds;
                }
                ptx::fence_proxy_async_smem();              // generic smem writes -> tcgen05 (async proxy) reads
                ptx::tc_fence_before();                     // the S tile has been read: its columns may be overwritten
                ptx::mbar_arrive(gs_bar);
                if (threadIdx.x == 64) CVCL_STAMP(23);
                if (warp == 0 && lane == 0)
                    for (int idx = kStages; idx < n_fill3; ++idx) fill3(idx);      // slots free up as the MMAs retire
                if (warp == 1 && lane == 0) {
                    mbar_wait_b(gs_bar, 0);                 // single use per launch
                    ptx::tc_fence_after();
                    for (int kc = 0; kc < num_kc3; ++kc)
                        for (int h = 0; h < nH; ++h) {
                            const int nh = min(256, wq - 256 * h);
                            const uint32_t idesc = ptx::make_idesc_bf16(kBM, nh, false, true);
                            mbar_wait_b(&full_bar[ring.stage], ring.phase);
                            ptx::tc_fence_after();
                            const uint32_t sa = ptx::smem_u32(smem + kGsOff + kc * 16384);
                            const uint32_t sb = ptx::smem_u32(smem + ring.stage * kStageBytes);
                            const uint64_t adesc = ptx::make_kmajor_sw128_desc(sa);
                            const uint64_t bdesc = ptx::make_mnmajor_sw128_desc(sb, 8192);
#pragma unroll
                            for (int k = 0; k < kBK / kUmmaK; ++k)
                                ptx::umma_bf16(tmem_base + 256 * h, adesc + 2 * k, bdesc + 128 * k, idesc,
                                               (kc > 0 || k > 0) ? 1u : 0u);
                            ptx::umma_commit(&empty_bar[ring.stage]);
                            if (kc == num_kc3 - 1 && h == nH - 1) ptx::umma_commit(tfull_bar);
                            ring.next();
                        }
                }
                __syncwarp();
                // dQ partial [128, wq] -> slab (z, pi), columns qs*wq..: 128 columns per pass (64 per thread),
                // two staging halves
                mbar_wait_b(tfull_bar, tfull_uses & 1u);
                ptx::tc_fence_after();
                if (threadIdx.x == 64) {
                    CVCL_STAMP(24);
                    if (z == 0 && qs == 0) {                // warps in fixed order
                        float dsum = 0.f;
                        for (int wv = 0; wv < kWarps; ++wv) dsum += red[32 + wv];
                        p.dspart[rb * p.nPart + pi] = dsum;
                    }
                }
                const int out_row = ((z * p.nPart + pi) * p.Bp) + rb * kBM;
                for (int q = 0; q < wq / 128; ++q) {
                    unsigned char* stg = smem + (q & 1) * 65536;
                    if (q >= 2) { if (threadIdx.x == 64) tma_store_wait_read<1>(); __syncthreads(); }
                    stage_f32_cols(tmem_row, 128 * q + 64 * half, 64 * half, 64, stg, row);
                    ptx::fence_proxy_async_smem();
                    __syncthreads();
                    if (threadIdx.x == 64) {
#pragma unroll
                        for (int b4 = 0; b4 < 4; ++b4)
                            ptx::tma_store_2d(&maps.dq_out, stg + b4 * 16384, qs * wq + 128 * q + b4 * 32, out_row);
                        tma_store_commit();
                    }
                }
                if (threadIdx.x == 64) { tma_store_wait_all(); CVCL_STAMP(25); }
                ptx::tc_fence_before();
                ++tfull_uses;
            }
        }
    }
    grid_sync<false, kSharded>(p, sync_k++);
    if (p.phase_limit == 4) goto done;

    if (p.need_grads) {
        // ======================================================================== P4
        // task t < B: text row t (direction 1) -> bf16 d mean-embedding / len (operand of the embedding gradient);
        // task B + r: image row r (direction 0) -> bf16 du (operand of dW) + bias partials
        const int nch = p.E >> 7;
        const size_t slab = static_cast<size_t>(p.Bp) * p.E;
        const float wg = scale * (0.5f * p.inv_rows);
        float4 dbacc[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) dbacc[c] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int t = cta * kWarps + warp; t < 2 * p.B; t += G * kWarps) {
            const int z = t < p.B ? 1 : 0;
            const int r = z ? t : t - p.B;
            float4 acc[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[c] = make_float4(0.f, 0.f, 0.f, 0.f);
            const float* base = p.dqpart + (static_cast<size_t>(z) * p.nPart * p.Bp + r) * p.E;
            // the positives of the other modality (the diagonal of G, in fp32) and this row's own features
            const __nv_bfloat16* posrow = p.kf16[z] + static_cast<size_t>(p.diag_off + r) * p.ldk;
            const __nv_bfloat16* qrow = p.q16[z] + static_cast<size_t>(r) * p.ldq;
            uint2 pr[4], qr[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                pr[c] = make_uint2(0u, 0u); qr[c] = make_uint2(0u, 0u);
                if (c < nch) {
                    pr[c] = __ldcg(reinterpret_cast<const uint2*>(posrow + (c * 32 + lane) * 4));
                    qr[c] = __ldcg(reinterpret_cast<const uint2*>(qrow + (c * 32 + lane) * 4));
                }
            }
            const float inv = p.normalize ? __ldcg(p.invn[z] + r) : 1.f;
            const float rs = z ? 1.f / static_cast<float>(__ldg(p.lens + r)) : 1.f;
            // the diagonal of G in fp32: the slabs hold bf16(Gs_ii) K_i, replaced here by G_ii K_i with
            // G_ii = w (P_row,ii - 1 + P_col,ii - 1) (at one pair, exactly 0)
            const float dg = __ldcg(p.diag[z] + r);
            const float dcoef = wg * (expm1f(dg - __ldcg(p.lse[z] + r)) + expm1f(dg - __ldcg(p.lse[1 - z] + r)))
                                - __ldcg(p.gdiag[z] + r);
            for (int k0 = 0; k0 < p.nPart; k0 += 4) {
                float4 v[4][4];
#pragma unroll
                for (int k = 0; k < 4; ++k)
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        v[k][c] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (k0 + k < p.nPart && c < nch)
                            v[k][c] = __ldcg(reinterpret_cast<const float4*>(base + (k0 + k) * slab) + c * 32 + lane);
                    }
#pragma unroll
                for (int k = 0; k < 4; ++k)
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        acc[c].x += v[k][c].x; acc[c].y += v[k][c].y; acc[c].z += v[k][c].z; acc[c].w += v[k][c].w;
                    }
            }
            float4 qf[4];
            float dot = 0.f;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const float2 p0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&pr[c].x));
                const float2 p1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&pr[c].y));
                const float2 q0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&qr[c].x));
                const float2 q1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&qr[c].y));
                acc[c].x = fmaf(dcoef, p0.x, acc[c].x); acc[c].y = fmaf(dcoef, p0.y, acc[c].y);
                acc[c].z = fmaf(dcoef, p1.x, acc[c].z); acc[c].w = fmaf(dcoef, p1.y, acc[c].w);
                qf[c] = make_float4(q0.x, q0.y, q1.x, q1.y);
                dot = fmaf(qf[c].x, acc[c].x, dot); dot = fmaf(qf[c].y, acc[c].y, dot);
                dot = fmaf(qf[c].z, acc[c].z, dot); dot = fmaf(qf[c].w, acc[c].w, dot);
            }
            if (p.normalize) dot = warp_sum(dot); else dot = 0.f;
            __nv_bfloat16* orow = (z ? p.dm16 : p.du16) + static_cast<size_t>(r) * p.E;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                acc[c].x = (acc[c].x - qf[c].x * dot) * inv * rs; acc[c].y = (acc[c].y - qf[c].y * dot) * inv * rs;
                acc[c].z = (acc[c].z - qf[c].z * dot) * inv * rs; acc[c].w = (acc[c].w - qf[c].w * dot) * inv * rs;
                if (c < nch) {
                    store_bf16x4(orow + (c * 32 + lane) * 4, acc[c]);
                    if (z == 0) {
                        dbacc[c].x += acc[c].x; dbacc[c].y += acc[c].y; dbacc[c].z += acc[c].z; dbacc[c].w += acc[c].w;
                    }
                }
            }
        }
        // per-CTA bias partial: warps in fixed order
#pragma unroll
        for (int c = 0; c < 4; ++c)
            if (c < nch) *reinterpret_cast<float4*>(sdb + warp * 512 + (c * 32 + lane) * 4) = dbacc[c];
        __syncthreads();
        for (int e = threadIdx.x; e < p.E; e += kThreads) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) s += sdb[w * 512 + e];
            p.dbpart[static_cast<size_t>(cta) * p.E + e] = s;
        }
        if (threadIdx.x == 0) CVCL_STAMP(26);
    }
    if (p.need_grads) grid_sync<true, kSharded>(p, sync_k++);
    if (p.phase_limit == 5) goto done;

    if (p.need_grads) {
        // ======================================================================== P5
        // tiles [0, n_dw): dW[e, k] = sum_b du[b, e] x[b, k];  tiles [n_dw, ...): dtable[v, e] = sum_b C[b, v] dm[b, e]
        const int bn = p.dw_bn;
        const int n_dw = p.nEB * (p.K / bn);
        const int n_dt = ((p.V + 127) / 128) * p.nEB;
        const int num_kc5 = (p.B + kBK - 1) / kBK;
        for (int t = cta; t < n_dw + n_dt; t += G - 1) {   // the last CTA is kept for the final sums
            if (cta == G - 1) break;
            const bool is_dw = t < n_dw;
            const int u = is_dw ? t : t - n_dw;
            const int eb = u % p.nEB, ot = u / p.nEB;       // ot: k tile (dW) or vocabulary tile (d table)
            const int tn = is_dw ? bn : 128;                // tile width
            const CUtensorMap* mA = is_dw ? &maps.du_mn : &maps.c_mn;
            const CUtensorMap* mB = is_dw ? &maps.x_mn : &maps.dm_mn;
            const int a_col = is_dw ? eb * 128 : ot * 128;
            const int b_col = is_dw ? ot * bn : eb * 128;
            if (warp == 0) {
                if (lane == 0) {
                    for (int kc = 0; kc < num_kc5; ++kc) {
                        mbar_wait_b(&empty_bar[ring.stage], ring.phase ^ 1u);
                        unsigned char* sa = smem + ring.stage * kStageBytes;
                        ptx::mbar_arrive_expect_tx(&full_bar[ring.stage], 16384u + static_cast<uint32_t>(tn) * 128u);
                        ptx::tma_load_2d(sa, mA, &full_bar[ring.stage], a_col, kc * kBK);
                        ptx::tma_load_2d(sa + 8192, mA, &full_bar[ring.stage], a_col + 64, kc * kBK);
                        for (int jb = 0; jb < tn / 64; ++jb)
                            ptx::tma_load_2d(sa + 16384 + jb * 8192, mB, &full_bar[ring.stage], b_col + 64 * jb, kc * kBK);
                        ring.next();
                    }
                }
                __syncwarp();
            } else if (warp == 1) {
                if (lane == 0) {
                    const uint32_t idesc = ptx::make_idesc_bf16(kBM, tn, true, true);
                    for (int kc = 0; kc < num_kc5; ++kc) {
                        mbar_wait_b(&full_bar[ring.stage], ring.phase);
                        ptx::tc_fence_after();
                        const uint32_t sa = ptx::smem_u32(smem + ring.stage * kStageBytes);
                        const uint64_t adesc = ptx::make_mnmajor_sw128_desc(sa, 8192);
                        const uint64_t bdesc = ptx::make_mnmajor_sw128_desc(sa + 16384, 8192);
#pragma unroll
                        for (int k = 0; k < kBK / kUmmaK; ++k)
                            ptx::umma_bf16(tmem_base, adesc + 128 * k, bdesc + 128 * k, idesc, (kc > 0 || k > 0) ? 1u : 0u);
                        ptx::umma_commit(&empty_bar[ring.stage]);
                        if (kc == num_kc5 - 1) ptx::umma_commit(tfull_bar);
                        ring.next();
                    }
                }
                __syncwarp();
            }
            {
                // all eight warps drain the tile (each thread: its row, half of the columns)
                mbar_wait_b(tfull_bar, tfull_uses & 1u);
                ptx::tc_fence_after();
                if (threadIdx.x == 64) CVCL_STAMP(27);
                stage_f32_cols(tmem_row, (tn / 2) * half, (tn / 2) * half, tn / 2, smem, row);
                ptx::fence_proxy_async_smem();
                ptx::tc_fence_before();
                __syncthreads();
                if (reduce) {
                    // partial tile -> scratch of the rank that owns tile t: every warp copies 16 rows out of the staging
                    // boxes with 512-byte row stores (posted stores over NVLink; measured faster than a TMA store to peer
                    // memory, which drained at ~270 GB/s)
                    float* dstt = p.peer_scratch[t % p.world] +
                                  static_cast<size_t>(p.rank * p.nslot + t / p.world) * 128 * 128;
#pragma unroll
                    for (int i = 0; i < 16; i += 8) {
                        uint4 v[8];
#pragma unroll
                        for (int k = 0; k < 8; ++k) v[k] = swz_ld16(smem, warp * 16 + i + k, lane * 16);
#pragma unroll
                        for (int k = 0; k < 8; ++k)
                            *reinterpret_cast<uint4*>(dstt + (warp * 16 + i + k) * 128 + lane * 4) = v[k];
                    }
                } else if (threadIdx.x == 64) {
                    if (is_dw) {
                        for (int b4 = 0; b4 < tn / 32; ++b4)
                            ptx::tma_store_2d(&maps.dw_out, smem + b4 * 16384, ot * bn + b4 * 32, eb * 128);
                    } else {
                        for (int b4 = 0; b4 < 4; ++b4)            // rows >= V are clipped by the tensor map
                            ptx::tma_store_2d(&maps.dt_out, smem + b4 * 16384, eb * 128 + b4 * 32, ot * 128);
                    }
                    tma_store_commit();
                    tma_store_wait_read<0>();
                    CVCL_STAMP(28);
                }
            }
            ++tfull_uses;
            __syncthreads();                                // staging / accumulator reuse across tiles
            ptx::tc_fence_after();
        }
    }

    // ---- final sums by the last CTA, every one in a fixed order (deterministic).  This CTA is the tail of the
    // kernel, so every partial is fetched with independent loads (one or two round trips to L2), never one
    // dependent load per addend.
    if (cta == G - 1) {
        float* fs = reinterpret_cast<float*>(smem);                      // the ring is idle: this CTA ran no P5 tile
        const int n_rb = 2 * p.nMB * 6, n_ds = p.need_grads ? p.nMB * p.nPart : 0;
        for (int i = threadIdx.x; i < n_rb + n_ds; i += kThreads)
            fs[i] = i < n_rb ? __ldcg(p.rb_part + i) : __ldcg(p.dspart + (i - n_rb));
        float* dbs = fs + 1024;                                          // [2][512]
        if (p.need_grads) {
            // d bias: per-CTA partials of P4 in CTA order; only the CTAs that held image rows there contribute
            // (tasks [B, 2B) of P4's warp-per-row schedule) unless the schedule wrapped around the grid
            const bool wrapped = 2 * p.B > G * kWarps;
            const int c_lo = wrapped ? 0 : p.B / kWarps;
            const int c_hi = wrapped ? G : (2 * p.B + kWarps - 1) / kWarps;
            const int col4 = threadIdx.x & 127, grp = threadIdx.x >> 7;  // two interleaved row groups
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            if (col4 * 4 < p.E) {
                for (int c0 = c_lo + grp; c0 < c_hi; c0 += 16) {
                    float4 v[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const int c = c0 + 2 * k;
                        v[k] = c < c_hi ? __ldcg(reinterpret_cast<const float4*>(p.dbpart + static_cast<size_t>(c) * p.E) + col4)
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
#pragma unroll
                    for (int k = 0; k < 8; ++k) { acc.x += v[k].x; acc.y += v[k].y; acc.z += v[k].z; acc.w += v[k].w; }
                }
                *reinterpret_cast<float4*>(dbs + grp * 512 + col4 * 4) = acc;
            }
        }
        __syncthreads();
        float* fin = fs + 2048;                                          // [kSmall]: out5(8) | ds(4) | d bias
        if (p.need_grads)
            for (int e = threadIdx.x; e < p.E; e += kThreads) fin[12 + e] = dbs[e] + dbs[512 + e];
        if (threadIdx.x == 0) {
            float s6[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            for (int b = 0; b < 2 * p.nMB; ++b) {
                const int z = b / p.nMB;
                s6[z] += fs[b * 6 + z];
                s6[2 + z] += fs[b * 6 + 2 + z];
                s6[4 + z] += fs[b * 6 + 4 + z];
            }
            fin[0] = (s6[0] + s6[1]) * 0.5f * p.inv_rows;
            fin[1] = s6[4] * p.inv_rows;
            fin[2] = s6[5] * p.inv_rows;
            fin[3] = s6[2] * p.inv_rows;
            fin[4] = s6[3] * p.inv_rows;
            fin[5] = fin[6] = fin[7] = 0.f;
            float ds = 0.f;
            for (int i = 0; i < n_ds; ++i) ds += fs[n_rb + i];
            fin[8] = ds; fin[9] = fin[10] = fin[11] = 0.f;
        }
        __syncthreads();
        const int n_fin = p.need_grads ? 12 + p.E : 8;
        if (reduce) {                                    // this rank's partials -> slot `rank` of every rank's block
            for (int i = threadIdx.x; i < n_fin; i += kThreads) {
                const float v = fin[i];
                for (int pp = 0; pp < p.world; ++pp) p.peer_small[pp][p.rank * kSmall + i] = v;
            }
        } else {
            for (int i = threadIdx.x; i < n_fin; i += kThreads) {
                const float v = fin[i];
                if (i < 5) p.out5[i] = v;
                else if (i == 8) p.dscale[0] = v;
                else if (i >= 12) p.dbias[i - 12] = v;
            }
        }
    }

    if (reduce) {
        // ======================================================================== P6 (sharded)
        grid_sync<false, kSharded>(p, sync_k++, 2, xepoch);          // every rank's partial tiles and scalars have landed here
        // (a) scalars + d bias: one-shot, summed locally in rank order (CTA 0)
        if (cta == 0) {
            const int n_fin = p.need_grads ? 12 + p.E : 8;
            const float* sm = p.peer_small[p.rank];
            for (int i = threadIdx.x; i < n_fin; i += kThreads) {
                float v = 0.f;
                for (int q = 0; q < p.world; ++q) v += __ldcg(sm + q * kSmall + i);
                if (i < 5) p.out5[i] = v;
                else if (i == 8) p.dscale[0] = v;
                else if (i >= 12) p.dbias[i - 12] = v;
            }
        }
        // (b) the tiles this rank owns: one warp per tile row (512 bytes), `world` partials summed in rank order,
        //     the sum stored into the final dW / d table of every rank
        if (p.need_grads) {
            const int n_dw = p.nEB * (p.K / 128);
            const int n_t = n_dw + ((p.V + 127) / 128) * p.nEB;
            const int n_own = (n_t - p.rank + p.world - 1) / p.world;            // tiles rank, rank + world, ...
            const size_t off_dt = 12 + static_cast<size_t>(p.E);
            const size_t off_dw = off_dt + static_cast<size_t>(p.V) * p.E;
            const float* scr = p.peer_scratch[p.rank];
            const size_t src_stride = static_cast<size_t>(p.nslot) * 128 * 128;
            constexpr int U = 4;
            const int n_rows = n_own * 128;
            for (int r0 = cta * kWarps + warp; r0 < n_rows; r0 += U * G * kWarps) {
                float4 v[U][8];
                size_t dst[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int r = r0 + u * G * kWarps;
                    dst[u] = ~static_cast<size_t>(0);
                    if (r < n_rows) {
                        const int slot = r >> 7, rr = r & 127;
                        const int t = slot * p.world + p.rank;
                        const bool is_dw = t < n_dw;
                        const int uu = is_dw ? t : t - n_dw;
                        const int eb = uu % p.nEB, ot = uu / p.nEB;
                        if (is_dw) dst[u] = off_dw + static_cast<size_t>(eb * 128 + rr) * p.K + ot * 128 + lane * 4;
                        else if (ot * 128 + rr < p.V) dst[u] = off_dt + static_cast<size_t>(ot * 128 + rr) * p.E + eb * 128 + lane * 4;
                        if (dst[u] != ~static_cast<size_t>(0)) {
                            const float* src = scr + (static_cast<size_t>(slot) * 128 + rr) * 128 + lane * 4;
#pragma unroll
                            for (int q = 0; q < 8; ++q)
                                if (q < p.world) v[u][q] = __ldcg(reinterpret_cast<const float4*>(src + q * src_stride));
                        }
                    }
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if (dst[u] != ~static_cast<size_t>(0)) {
                        float4 acc = v[u][0];
#pragma unroll
                        for (int q = 1; q < 8; ++q)
                            if (q < p.world) { acc.x += v[u][q].x; acc.y += v[u][q].y; acc.z += v[u][q].z; acc.w += v[u][q].w; }
                        for (int q = 0; q < p.world; ++q)
                            *reinterpret_cast<float4*>(p.peer_stats[q] + dst[u]) = acc;
                    }
                }
            }
        }
        grid_sync<false, kSharded>(p, sync_k++, 3, xepoch);          // every rank's block holds the global sums behind this
    }

done:
    // leave the barrier counter and the work queue zeroed for the next launch: the last CTA through the exit
    // ticket resets them (every CTA has passed its last grid barrier before it takes a ticket)
    __syncthreads();
    if (threadIdx.x == 0) {
        if (cta == 0 && p.timing) p.timing[15] = globaltimer_ns();
        __threadfence();
        if (atomicAdd(p.sync + 1, 1u) == static_cast<unsigned int>(G - 1)) {
            p.sync[0] = 0u; p.sync[1] = 0u; p.sync[2] = 0u;
            if (kSharded && p.epoch) *p.epoch = xepoch;
            __threadfence();
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) ptx::tmem_dealloc<512>(tmem_base);
}

#undef CVCL_STAMP

}  // namespace fused
}  // namespace cvcl
