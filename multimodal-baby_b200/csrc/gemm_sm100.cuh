// tcgen05 / TMEM / TMA GEMM engine for the CVCL contrastive path (sm_100a only).
//
//   D[m, n] = sum_k A[m, k] * B[n, k]        A: [M, K] bf16 row-major (K-major operand)
//                                            B: [N, K] bf16 row-major (K-major operand)
//
// One CTA = one 128 x BN output tile, fp32 accumulator in TMEM (BN columns), operands staged by
// TMA into 128B-swizzled shared memory through a STAGES-deep mbarrier ring.
// Warp roles (192 threads):  warp 0 = TMA producer (one elected lane)
//                            warp 1 = TMEM allocator + tcgen05.mma issuer (one elected lane)
//                            warps 2..5 = epilogue; warp w owns TMEM lanes 32*(w%4) .. +31,
//                                         i.e. thread <-> one accumulator row.
// The epilogue is a policy class (Epi) with two phases; between them an optional cluster barrier
// lets the CTAs that share a row block (cluster along N) exchange per-row partial reductions
// through distributed shared memory (used by the L2-normalise epilogues).
// blockIdx.z selects one of two independent problems ("directions": image->text and text->image)
// so that the symmetric InfoNCE needs a single launch.
#pragma once
#include "ptx.cuh"
#include <cuda_bf16.h>

namespace cvcl {

constexpr int kBM = 128;          // UMMA M
constexpr int kBK = 64;           // one 128-byte swizzle atom of bf16 along K
constexpr int kUmmaK = 16;
constexpr int kGemmThreads = 192;
constexpr int kEpiThreads = 128;

struct GemmShape {
    int M[2];            // rows of the output per direction
    int N[2];            // columns of the output per direction
    int K;               // contraction length (same for both directions)
    int m_stride;        // tile origin step along M (kBM unless tiles overlap/segment)
    int n_stride;        // tile origin step along N
    int aux_row_off[2];  // row offset of each epilogue input tile relative to m0
    int k_splits;        // > 1: blockIdx.z splits the contraction (single direction, additive epilogue)
    int n_fast;          // 1: consecutive CTAs walk the N tiles of one M tile first (the few CTAs that share an A
                         //    row block run together and the second reads it from L2; no clusters in this mode)
    // device-side problem size (nullable; plain one-tile-per-CTA kernel without clusters / split-K only): a size the
    // host does not know without a sync, e.g. the number of non-pad token rows.  CTAs whose tile starts at or beyond
    // *m_limit leave at once; the contraction stops after ceil(*k_limit / 64) chunks (operands must be finite --
    // zero -- between *k_limit and the end of that chunk).
    const int* m_limit;
    const int* k_limit;
};

// All tensor maps of one launch (passed as a single __grid_constant__ parameter).
struct alignas(64) GemmMaps {
    CUtensorMap a[2], b[2];   // operands per direction
    CUtensorMap aux[2];       // epilogue INPUT tiles, bf16 [M,N] row-major (e.g. features, positives)
    CUtensorMap out[2];       // epilogue OUTPUT tile per direction (bf16 or fp32, [M,N] row-major)
};

struct EpiCtx {
    uint32_t tmem_row;   // TMEM address of this thread's row, column 0 of the accumulator
    int row;             // 0..127 within the tile
    int m0, n0, z;       // tile origin and direction
    int tile_m, tile_n;  // tile indices
    int epi_tid;         // 0..127
    unsigned char* scratch;
    unsigned char* aux[2];          // smem: epilogue input tiles (128B-swizzled TMA boxes)
    unsigned char* out_stage;       // smem: output staging (reuses the operand ring after the mainloop)
    const CUtensorMap* out_map;
    int bar_base;                   // named-barrier id offset of this epilogue group (0 unless persistent)
};

// ---- swizzled shared-memory tile access (layout written / read by TMA with SWIZZLE_128B) --------
// A tile is a sequence of boxes of 128 rows x 128 bytes; box b covers byte columns [128b, 128b+128).
// Row r of a box sits at r*128; its 16-byte chunk c is stored at chunk position c ^ (r & 7).
__device__ __forceinline__ unsigned char* swz_ptr(unsigned char* tile, int row, int byte_col) {
    const int box = byte_col >> 7, chunk = (byte_col & 127) >> 4;
    return tile + box * (kBM * 128) + row * 128 + ((chunk ^ (row & 7)) << 4);
}
__device__ __forceinline__ uint4 swz_ld16(unsigned char* tile, int row, int byte_col) {
    return *reinterpret_cast<const uint4*>(swz_ptr(tile, row, byte_col));
}
__device__ __forceinline__ void swz_st16(unsigned char* tile, int row, int byte_col, uint4 v) {
    *reinterpret_cast<uint4*>(swz_ptr(tile, row, byte_col)) = v;
}
__device__ __forceinline__ uint4 pack_bf16x8(const float* v) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
    __nv_bfloat162 c = __floats2bfloat162_rn(v[4], v[5]), d = __floats2bfloat162_rn(v[6], v[7]);
    uint4 q;
    q.x = *reinterpret_cast<uint32_t*>(&a); q.y = *reinterpret_cast<uint32_t*>(&b);
    q.z = *reinterpret_cast<uint32_t*>(&c); q.w = *reinterpret_cast<uint32_t*>(&d);
    return q;
}
__device__ __forceinline__ void unpack_bf16x8(uint4 q, float* v) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
    for (int k = 0; k < 4; ++k) { const float2 f = __bfloat1622float2(h[k]); v[2 * k] = f.x; v[2 * k + 1] = f.y; }
}
// After every epilogue thread has written its row into out_stage: publish to the async proxy,
// then one thread stores the boxes with TMA (rows / columns beyond the tensor are clipped).
template <int BN, int ELEM>
__device__ __forceinline__ void out_tile_commit(const EpiCtx& cx) {
    ptx::fence_proxy_async_smem();
    ptx::named_bar_sync(2 + cx.bar_base, kEpiThreads);
    if (cx.epi_tid == 0) {
        constexpr int kBoxCols = 128 / ELEM;
#pragma unroll
        for (int b = 0; b < BN / kBoxCols; ++b)
            ptx::tma_store_2d(cx.out_map, cx.out_stage + b * (kBM * 128), cx.n0 + b * kBoxCols, cx.m0);
        ptx::tma_store_commit_and_wait();
    }
}

template <int BN, int STAGES, int NAUX>
struct GemmSmem {
    static constexpr int kABytes = kBM * kBK * 2;
    static constexpr int kBBytes = BN * kBK * 2;
    static constexpr int kStageBytes = kABytes + kBBytes;
    static constexpr int kAuxBytes = kBM * BN * 2;
    static constexpr int kAuxOff = STAGES * kStageBytes;
    static constexpr int kBarOff = kAuxOff + NAUX * kAuxBytes;
    static constexpr int kScratchOff = kBarOff + 256;
    template <class Epi>
    static constexpr int total() { return kScratchOff + Epi::kScratchBytes + 1024 /*align slack*/; }
};

// D[m, n] = sum_k A[m, k] * B[n, k].  Operand storage per template flag:
//   K-major  (flag false): memory [rows = M or N, cols = K] row-major  (contraction contiguous)
//   MN-major (flag true) : memory [rows = K, cols = M or N] row-major  (contraction strided) --
//                          lets a backward GEMM consume a forward tensor without a transposed copy.
template <int BN, int STAGES, class Epi, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_bf16_kernel(const __grid_constant__ GemmMaps maps, const GemmShape gs, const typename Epi::Params ep) {
    static_assert(BN == 64 || BN == 128 || BN == 256, "BN");
    using L = GemmSmem<BN, STAGES, Epi::kNumAux>;
    static_assert(Epi::kOutElemBytes == 0 || STAGES * L::kStageBytes >= kBM * BN * Epi::kOutElemBytes,
                  "output staging must fit in the operand ring");
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tmem_full_bar = empty_bar + STAGES;
    uint64_t* aux_bar = tmem_full_bar + 1;
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(aux_bar + 1);
    unsigned char* scratch = smem + L::kScratchOff;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const bool split = gs.k_splits > 1;
    const int z = split ? 0 : blockIdx.z;
    const CUtensorMap* tmA = &maps.a[z];
    const CUtensorMap* tmB = &maps.b[z];
    int bx = blockIdx.x, by = blockIdx.y;
    if (gs.n_fast) {
        const int lin = blockIdx.y * gridDim.x + blockIdx.x;
        by = lin % static_cast<int>(gridDim.y); bx = lin / static_cast<int>(gridDim.y);
    }
    const int m0 = bx * gs.m_stride;
    const int n0 = by * gs.n_stride;
    int num_k_all = (gs.K + kBK - 1) / kBK;
    if (gs.m_limit || gs.k_limit) {
        ptx::pdl_wait();                   // the limits were written by an earlier kernel of the stream
        if (gs.m_limit && m0 >= __ldg(gs.m_limit)) return;       // whole CTA, before any barrier / TMEM set-up
        if (gs.k_limit) {
            int lim = (__ldg(gs.k_limit) + kBK - 1) / kBK;
            lim = lim < 1 ? 1 : lim;
            num_k_all = lim < num_k_all ? lim : num_k_all;
        }
    }
    const int per_split = split ? (num_k_all + gs.k_splits - 1) / gs.k_splits : num_k_all;
    const int kc_begin = split ? blockIdx.z * per_split : 0;
    const int kc_end = (kc_begin + per_split < num_k_all) ? kc_begin + per_split : num_k_all;

    ptx::pdl_launch_dependents();          // the next kernel may begin its prologue on idle SMs
    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(tmA);
        ptx::prefetch_tmap(tmB);
        for (int s = 0; s < STAGES; ++s) {
            ptx::mbar_init(&full_bar[s], 1);
            ptx::mbar_init(&empty_bar[s], 1);
        }
        ptx::mbar_init(tmem_full_bar, 1);
        ptx::mbar_init(aux_bar, 1);
        ptx::fence_mbar_init();
    }
    if (warp == 1) {
        ptx::tmem_alloc<(BN < 32 ? 32 : BN)>(tmem_ptr_smem);
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;
    ptx::pdl_wait();                       // everything above overlapped the previous kernel's tail

    if (warp == 0) {
        // ------------------------------------------------------------ TMA producer
        if (lane == 0) {
            if constexpr (Epi::kNumAux > 0) {
                ptx::mbar_arrive_expect_tx(aux_bar, Epi::kNumAux * L::kAuxBytes);
#pragma unroll
                for (int i = 0; i < Epi::kNumAux; ++i)
#pragma unroll
                    for (int j = 0; j < BN / 64; ++j)
                        ptx::tma_load_2d(smem + L::kAuxOff + i * L::kAuxBytes + j * (kBM * 128), &maps.aux[i],
                                         aux_bar, n0 + 64 * j, m0 + gs.aux_row_off[i]);
            }
            int stage = 0; uint32_t phase = 0;
            for (int kc = kc_begin; kc < kc_end; ++kc) {
                ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
                unsigned char* sa = smem + stage * L::kStageBytes;
                unsigned char* sb = sa + L::kABytes;
                ptx::mbar_arrive_expect_tx(&full_bar[stage], L::kStageBytes);
                if constexpr (A_MN) {
#pragma unroll
                    for (int j = 0; j < kBM / 64; ++j)
                        ptx::tma_load_2d(sa + j * (kBK * 128), tmA, &full_bar[stage], m0 + 64 * j, kc * kBK);
                } else {
                    ptx::tma_load_2d(sa, tmA, &full_bar[stage], kc * kBK, m0);
                }
                if constexpr (B_MN) {
#pragma unroll
                    for (int j = 0; j < BN / 64; ++j)
                        ptx::tma_load_2d(sb + j * (kBK * 128), tmB, &full_bar[stage], n0 + 64 * j, kc * kBK);
                } else {
                    ptx::tma_load_2d(sb, tmB, &full_bar[stage], kc * kBK, n0);
                }
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            constexpr uint32_t idesc = ptx::make_idesc_bf16(kBM, BN, A_MN, B_MN);
            // per UMMA_K=16 step the start address advances by 32 B (K-major: inside the swizzle atom)
            // or by 16 rows * 128 B (MN-major), in 16-byte descriptor units
            constexpr uint32_t a_step = A_MN ? (kUmmaK * 128) >> 4 : (kUmmaK * 2) >> 4;
            constexpr uint32_t b_step = B_MN ? (kUmmaK * 128) >> 4 : (kUmmaK * 2) >> 4;
            int stage = 0; uint32_t phase = 0;
            for (int kc = kc_begin; kc < kc_end; ++kc) {
                ptx::mbar_wait(&full_bar[stage], phase);
                ptx::tc_fence_after();
                const uint32_t sa = ptx::smem_u32(smem + stage * L::kStageBytes);
                const uint32_t sb = sa + L::kABytes;
                const uint64_t adesc = A_MN ? ptx::make_mnmajor_sw128_desc(sa, kBK * 128) : ptx::make_kmajor_sw128_desc(sa);
                const uint64_t bdesc = B_MN ? ptx::make_mnmajor_sw128_desc(sb, kBK * 128) : ptx::make_kmajor_sw128_desc(sb);
#pragma unroll
                for (int k = 0; k < kBK / kUmmaK; ++k) {
                    ptx::umma_bf16(tmem_base, adesc + a_step * k, bdesc + b_step * k, idesc,
                                   (kc > kc_begin || k > 0) ? 1u : 0u);
                }
                ptx::umma_commit(&empty_bar[stage]);      // frees the smem slot when MMAs retire
                if (kc == kc_end - 1) ptx::umma_commit(tmem_full_bar);
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        }
        __syncwarp();
    }

    EpiCtx cx;
    cx.epi_tid = threadIdx.x - 64;
    const int quad = warp & 3;                    // TMEM lane quadrant this warp may access
    cx.row = quad * 32 + lane;
    cx.tmem_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    cx.m0 = m0; cx.n0 = n0; cx.z = z; cx.tile_m = bx; cx.tile_n = by;
    cx.scratch = scratch;
    cx.aux[0] = smem + L::kAuxOff;
    cx.aux[1] = smem + L::kAuxOff + (Epi::kNumAux > 1 ? L::kAuxBytes : 0);
    cx.out_stage = smem;                          // operand ring is idle once tmem_full has fired
    cx.out_map = &maps.out[z];
    cx.bar_base = 0;

    if (warp >= 2) {
        if constexpr (Epi::kNumAux > 0) ptx::mbar_wait(aux_bar, 0);
        ptx::mbar_wait(tmem_full_bar, 0);
        ptx::tc_fence_after();
        Epi::template phase1<BN>(cx, gs, ep);
    }
    if constexpr (Epi::kClusterReduce) {
        ptx::tc_fence_before();
        ptx::cluster_sync_all();
        ptx::tc_fence_after();
        if (warp >= 2) Epi::template phase2<BN>(cx, gs, ep);
        ptx::tc_fence_before();
        ptx::cluster_sync_all();
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) ptx::tmem_dealloc<(BN < 32 ? 32 : BN)>(tmem_base);
}

// -------------------------------------------------------------------------------------------------
// Persistent variant for large problems (K-major operands, non-cluster epilogues): one CTA per SM
// loops over output tiles.  The accumulator is double-buffered in TMEM (2 x BN columns), so the MMAs
// of tile i+1 run while the epilogue warps drain tile i, and the per-CTA costs (launch, TMEM
// allocation, barrier init, descriptor fetch, store drain at exit) are paid once per SM instead of
// once per tile.  Tiles are enumerated direction-major with the M index fastest, so the CTAs that
// run concurrently share the same B (key) tile in L2.
// -------------------------------------------------------------------------------------------------
template <int BN, int STAGES, int OUT_BYTES, int SCRATCH>
struct PersistSmem {
    static constexpr int kGroups = BN / 128;                 // epilogue groups: 128 columns each
    static constexpr int kABytes = kBM * kBK * 2;
    static constexpr int kBBytes = BN * kBK * 2;
    static constexpr int kStageBytes = kABytes + kBBytes;
    static constexpr int kOutOff = STAGES * kStageBytes;
    static constexpr int kOutBytes = kBM * 128 * OUT_BYTES;  // per group
    static constexpr int kBarOff = kOutOff + kGroups * kOutBytes;
    static constexpr int kScratchOff = kBarOff + 256;
    static constexpr int kScratchBytes = (SCRATCH + 15) / 16 * 16;   // per group
    static constexpr int total() { return kScratchOff + kGroups * kScratchBytes + 1024; }
};

struct TileGrid { int tiles_m[2], tiles_n[2], total; };

// The MMA tile is 128 x BN; the epilogue sees it as BN/128 independent 128 x 128 tiles, each drained
// by its own group of four warps (one thread per row), so a BN = 256 CTA runs 8 epilogue warps.
template <int BN, int STAGES, class Epi>
__global__ void __launch_bounds__(64 + 128 * (BN / 128), 1)
gemm_bf16_persistent_kernel(const __grid_constant__ GemmMaps maps, const GemmShape gs, const TileGrid tg,
                            const typename Epi::Params ep) {
    static_assert(!Epi::kClusterReduce && Epi::kNumAux == 0, "persistent kernel: streaming epilogues only");
    static_assert(BN == 128 || BN == 256, "BN");
    using L = PersistSmem<BN, STAGES, Epi::kOutElemBytes, Epi::kScratchBytes>;
    constexpr int kGroups = L::kGroups;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tfull_bar = empty_bar + STAGES;          // [2] accumulator ready for the epilogue
    uint64_t* tempty_bar = tfull_bar + 2;              // [2] accumulator drained (one arrival per epilogue warp)
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int num_k = (gs.K + kBK - 1) / kBK;
    const int count0 = tg.tiles_m[0] * tg.tiles_n[0];

    ptx::pdl_launch_dependents();
    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&maps.a[0]); ptx::prefetch_tmap(&maps.b[0]);
        ptx::prefetch_tmap(&maps.a[1]); ptx::prefetch_tmap(&maps.b[1]);
        for (int s = 0; s < STAGES; ++s) { ptx::mbar_init(&full_bar[s], 1); ptx::mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { ptx::mbar_init(&tfull_bar[a], 1); ptx::mbar_init(&tempty_bar[a], 4 * kGroups); }
        ptx::fence_mbar_init();
    }
    if (warp == 1) ptx::tmem_alloc<2 * BN>(tmem_ptr_smem);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;
    ptx::pdl_wait();

    auto decode = [&](int t, int& z, int& tm, int& tn) {
        z = t >= count0 ? 1 : 0;
        const int local = z ? t - count0 : t;
        tm = local % tg.tiles_m[z];
        tn = local / tg.tiles_m[z];
    };

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int t = blockIdx.x; t < tg.total; t += gridDim.x) {
                int z, tm, tn; decode(t, z, tm, tn);
                const int m0 = tm * gs.m_stride, n0 = tn * gs.n_stride;
                for (int kc = 0; kc < num_k; ++kc) {
                    ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
                    unsigned char* sa = smem + stage * L::kStageBytes;
                    ptx::mbar_arrive_expect_tx(&full_bar[stage], L::kStageBytes);
                    ptx::tma_load_2d(sa, &maps.a[z], &full_bar[stage], kc * kBK, m0);
                    ptx::tma_load_2d(sa + L::kABytes, &maps.b[z], &full_bar[stage], kc * kBK, n0);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = ptx::make_idesc_bf16(kBM, BN, false, false);
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int t = blockIdx.x; t < tg.total; t += gridDim.x) {
                ptx::mbar_wait(&tempty_bar[acc], acc_phase ^ 1);     // epilogue has drained this buffer
                ptx::tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                for (int kc = 0; kc < num_k; ++kc) {
                    ptx::mbar_wait(&full_bar[stage], phase);
                    ptx::tc_fence_after();
                    const uint32_t sa = ptx::smem_u32(smem + stage * L::kStageBytes);
                    const uint64_t adesc = ptx::make_kmajor_sw128_desc(sa);
                    const uint64_t bdesc = ptx::make_kmajor_sw128_desc(sa + L::kABytes);
#pragma unroll
                    for (int k = 0; k < kBK / kUmmaK; ++k)
                        ptx::umma_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kc > 0 || k > 0) ? 1u : 0u);
                    ptx::umma_commit(&empty_bar[stage]);
                    if (kc == num_k - 1) ptx::umma_commit(&tfull_bar[acc]);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                acc ^= 1; if (acc == 0) acc_phase ^= 1;
            }
        }
        __syncwarp();
    } else {
        EpiCtx cx;
        const int grp = (warp - 2) >> 2;               // which 128-column slice of the MMA tile
        cx.epi_tid = (threadIdx.x - 64) & 127;
        const int quad = warp & 3;
        cx.row = quad * 32 + lane;
        cx.scratch = smem + L::kScratchOff + grp * L::kScratchBytes;
        cx.aux[0] = cx.aux[1] = nullptr;
        cx.out_stage = smem + L::kOutOff + grp * L::kOutBytes;
        cx.bar_base = 4 * grp;                         // named barriers 1..3 (+4 per group)
        int acc = 0; uint32_t acc_phase = 0;
        for (int t = blockIdx.x; t < tg.total; t += gridDim.x) {
            int z, tm, tn; decode(t, z, tm, tn);
            cx.z = z; cx.tile_m = tm; cx.tile_n = tn * kGroups + grp;
            cx.m0 = tm * gs.m_stride; cx.n0 = tn * gs.n_stride + grp * 128;
            cx.out_map = &maps.out[z];
            cx.tmem_row = tmem_base + acc * BN + grp * 128 + (static_cast<uint32_t>(quad * 32) << 16);
            ptx::mbar_wait(&tfull_bar[acc], acc_phase);
            ptx::tc_fence_after();
            Epi::template phase1<128>(cx, gs, ep);
            ptx::tc_fence_before();
            ptx::named_bar_sync(3 + cx.bar_base, kEpiThreads);   // scratch / staging reuse across tiles
            if (lane == 0) ptx::mbar_arrive(&tempty_bar[acc]);
            acc ^= 1; if (acc == 0) acc_phase ^= 1;
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) ptx::tmem_dealloc<2 * BN>(tmem_base);
}

// =====================================================================================
// Epilogue policies.  Interface: kClusterReduce, kScratchBytes, kNumAux (epilogue input tiles
// fetched by TMA), kOutElemBytes (0: no staged output, 2: bf16 tile, 4: fp32 tile stored by TMA),
// Params, phase1<BN>() and, for cluster epilogues, phase2<BN>().
// =====================================================================================

// ---- plain store C = alpha * acc, fp32, staged in smem and written with TMA (dW, big logits) ----
struct EpiStoreF32 {
    static constexpr bool kClusterReduce = false;
    static constexpr int kScratchBytes = 16;
    static constexpr int kNumAux = 0;
    static constexpr int kOutElemBytes = 4;
    struct Params { float alpha; };
    template <int BN>
    static __device__ __forceinline__ void phase1(const EpiCtx& cx, const GemmShape&, const Params& p) {
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
            float v[32];
            ptx::tmem_ld_32x32(cx.tmem_row + c, v);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                uint4 q;
                q.x = __float_as_uint(v[4 * j] * p.alpha); q.y = __float_as_uint(v[4 * j + 1] * p.alpha);
                q.z = __float_as_uint(v[4 * j + 2] * p.alpha); q.w = __float_as_uint(v[4 * j + 3] * p.alpha);
                swz_st16(cx.out_stage, cx.row, (c + 4 * j) * 4, q);
            }
        }
        out_tile_commit<BN, 4>(cx);
    }
    template <int BN>
    static __device__ __forceinline__ void phase2(const EpiCtx&, const GemmShape&, const Params&) {}
};

// ---- split-K partial: C += alpha * acc with fp32 vector atomics (C zero-initialised by the caller) ----
struct EpiAtomicAddF32 {
    static constexpr bool kClusterReduce = false;
    static constexpr int kScratchBytes = 16;
    static constexpr int kNumAux = 0;
    static constexpr int kOutElemBytes = 0;
    struct Params { float* C; int ldc; float alpha; };
    template <int BN>
    static __device__ __forceinline__ void phase1(const EpiCtx& cx, const GemmShape& gs, const Params& p) {
        const int m = cx.m0 + cx.row;
        const int M = gs.M[0], N = gs.N[0];
        float* crow = p.C + static_cast<size_t>(m) * p.ldc;
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
            float v[32];
            ptx::tmem_ld_32x32(cx.tmem_row + c, v);
            if (m >= M) continue;
            const int n = cx.n0 + c;
            if (n + 32 <= N) {
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    atomicAdd(reinterpret_cast<float4*>(crow + n) + j,
                              make_float4(v[4 * j] * p.alpha, v[4 * j + 1] * p.alpha, v[4 * j + 2] * p.alpha, v[4 * j + 3] * p.alpha));
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) if (n + j < N) atomicAdd(crow + n + j, v[j] * p.alpha);
            }
        }
    }
    template <int BN>
    static __device__ __forceinline__ void phase2(const EpiCtx&, const GemmShape&, const Params&) {}
};

// ---- same, direct global stores: for outputs whose row pitch is not 16-byte aligned (the 4 x 3 /
// 4 x 1 logits of the inference API) ----
struct EpiStoreF32Direct {
    static constexpr bool kClusterReduce = false;
    static constexpr int kScratchBytes = 16;
    static constexpr int kNumAux = 0;
    static constexpr int kOutElemBytes = 0;
    struct Params { float* C[2]; int ldc[2]; float alpha; };
    template <int BN>
    static __device__ __forceinline__ void phase1(const EpiCtx& cx, const GemmShape& gs, const Params& p) {
        const int m = cx.m0 + cx.row;
        const int M = gs.M[cx.z], N = gs.N[cx.z];
        float* crow = p.C[cx.z] + static_cast<size_t>(m) * p.ldc[cx.z];
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
            float v[32];
            ptx::tmem_ld_32x32(cx.tmem_row + c, v);     // warp-collective: no early exit above
            if (m >= M) continue;
            const int n = cx.n0 + c;
#pragma unroll
            for (int j = 0; j < 32; ++j)
                if (n + j < N) crow[n + j] = v[j] * p.alpha;
        }
    }
    template <int BN>
    static __device__ __forceinline__ void phase2(const EpiCtx&, const GemmShape&, const Params&) {}
};

// ---- projection head: + bias, L2-normalise the full row (cluster along N), store ------
// reference: multimodal.py:186-192 (fc) / 181-185 (1x1 conv) + F.normalize at :736
struct EpiHeadNorm {
    static constexpr bool kClusterReduce = true;
    static constexpr int kScratchBytes = kBM * 4;
    static constexpr int kNumAux = 0;
    static constexpr int kOutElemBytes = 2;          // bf16 features by TMA store
    struct Params {
        const float* bias;          // [N] or null
        int normalize;
        float* out_f32;  int ld_f32;        // [M, ld] fp32 copy of the features (nullable)
        int store_bf16;                     // stage + TMA-store the bf16 tile (maps.out[0])
        float* inv_norm;            // [M]  1 / max(||u||, 1e-12)
    };
    static __device__ __forceinline__ void add_bias(float* v, const float* bias, int n, int N) {
        if (!bias) return;
        if (n + 32 <= N) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 b = __ldg(reinterpret_cast<const float4*>(bias + n) + j);
                v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
            }
        } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) if (n + j < N) v[j] += __ldg(bias + n + j);
        }
    }
    template <int BN>
    static __device__ __forceinline__ void phase1(const EpiCtx& cx, const GemmShape& gs, const Params& p) {
        const int N = gs.N[cx.z];
        float ssq = 0.f;
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
            float v[32];
            ptx::tmem_ld_32x32(cx.tmem_row + c, v);
            const int n = cx.n0 + c;
            if (n >= N) continue;
            add_bias(v, p.bias, n, N);
#pragma unroll
            for (int j = 0; j < 32; ++j) if (n + j < N) ssq = fmaf(v[j], v[j], ssq);
        }
        reinterpret_cast<float*>(cx.scratch)[cx.row] = ssq;
    }
    template <int BN>
    static __device__ __forceinline__ void phase2(const EpiCtx& cx, const GemmShape& gs, const Params& p) {
        const int M = gs.M[cx.z], N = gs.N[cx.z];
        const int m = cx.m0 + cx.row;
        const float* my = reinterpret_cast<const float*>(cx.scratch) + cx.row;
        float tot = 0.f;
        const uint32_t nc = ptx::cluster_nctarank();
        for (uint32_t r = 0; r < nc; ++r) tot += ptx::ld_dsmem_f32(my, r);
        const float denom = p.normalize ? fmaxf(sqrtf(tot), 1e-12f) : 1.f;
        if (m < M && cx.tile_n == 0 && p.inv_norm) p.inv_norm[m] = 1.f / denom;
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
            float v[32];
            ptx::tmem_ld_32x32(cx.tmem_row + c, v);
            const int n = cx.n0 + c;
            if (n < N) add_bias(v, p.bias, n, N);
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = (n + j < N) ? v[j] / denom : 0.f;
            if (p.out_f32 && m < M && n < N) {
                float* dst = p.out_f32 + static_cast<size_t>(m) * p.ld_f32 + n;
                if (n + 32 <= N && (p.ld_f32 & 3) == 0) {
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        reinterpret_cast<float4*>(dst)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) if (n + j < N) dst[j] = v[j];
                }
            }
            if (p.store_bf16) {
#pragma unroll
                for (int j = 0; j < 4; ++j) swz_st16(cx.out_stage, cx.row, (c + 8 * j) * 2, pack_bf16x8(v + 8 * j));
            }
        }
        if (p.store_bf16) out_tile_commit<BN, 2>(cx);
    }
};

// ---- similarity tile -> online-softmax row statistics (never stores the logits) -------
// reference: multimodal.py:755,783-787 (match, logit_scale) and 808-818 (CE, argmax, entropy)
struct RowStat { float m, l, a; int arg; };          // max, sum exp(x-m), sum exp(x-m)*x, argmax
struct EpiSimStats {
    static constexpr bool kClusterReduce = false;
    static constexpr int kScratchBytes = 256;
    static constexpr int kNumAux = 0;
    static constexpr int kOutElemBytes = 0;
    struct Params {
        float scale;                // exp(s)
        int diag_off[2];            // positive of row r is column r + diag_off[z]
        RowStat* part[2];           // [n_tiles][m_pad]
        int m_pad[2];
        float* diag[2];             // [M]  logit at the positive
        unsigned int* ticket;       // zeroed here for the merge kernel that follows (unfused path)
        // fused merge (small problems): the last CTA of a row block merges that block's partials,
        // the last row block to finish adds the block sums in a fixed order -> no merge kernel
        int fuse_merge;
        int n_tiles[2], tiles_m[2];
        unsigned int* rb_ticket;    // [1 + tiles_m[0] + tiles_m[1]], zero on entry, left zero on exit
        float* rb_part;             // [(tiles_m[0] + tiles_m[1]) * 6]
        float* lse[2]; int* argmax[2];
        float inv_rows; float* out5;
    };
    template <int BN>
    static __device__ __forceinline__ void phase1(const EpiCtx& cx, const GemmShape& gs, const Params& p) {
        const int M = gs.M[cx.z], N = gs.N[cx.z];
        const int m = cx.m0 + cx.row;
        const int dcol = m + p.diag_off[cx.z];
        constexpr float kLog2e = 1.4426950408889634f;
        if (!p.fuse_merge && cx.tile_m == 0 && cx.tile_n == 0 && cx.z == 0 && cx.epi_tid == 0) *p.ticket = 0u;
        // Work on the raw dot products r (logit = scale * r, scale > 0): the scale is folded into the
        // exp2 argument, so the hot loop is FMNMX + FFMA + MUFU.EX2 + FADD + FFMA per element.
        float mx = -INFINITY, l = 0.f, a = 0.f;        // mx, a in the raw domain
        int arg = cx.n0;
        const float sc2 = p.scale * kLog2e;
        auto chunk = [&](float* v, int c) {
            const int n = cx.n0 + c;
            if (n >= N) return;                         // warp-uniform
            const bool full = n + 32 <= N;              // warp-uniform
            if (!full) {
#pragma unroll
                for (int j = 0; j < 32; ++j) if (n + j >= N) v[j] = -INFINITY;
            }
            float cm = v[0];
#pragma unroll
            for (int j = 1; j < 32; ++j) cm = fmaxf(cm, v[j]);
            if (cm > mx) {                              // rare after the first chunks: locate the first max
                int k = 31;
#pragma unroll
                for (int j = 31; j >= 0; --j) if (v[j] == cm) k = j;
                arg = n + k;
            }
            if (dcol >= n && dcol < n + 32 && m < M) { // the positive lives in exactly one chunk per row
                float dv = 0.f;
#pragma unroll
                for (int j = 0; j < 32; ++j) if (n + j == dcol) dv = v[j];
                p.diag[cx.z][m] = dv * p.scale;
            }
            const float nm = fmaxf(mx, cm);
            const float corr = exp2f((mx - nm) * sc2);             // mx = -inf -> 0
            l *= corr; a *= corr;
            const float nm2 = nm * sc2;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const float e = exp2f(fmaf(v[j], sc2, -nm2));      // masked columns: exp2(-inf) = 0
                l += e;
                a = fmaf(e, full ? v[j] : (n + j < N ? v[j] : 0.f), a);
            }
            mx = nm;
        };
        // two register buffers: the TMEM load of the next 32 columns is in flight during the math
        float va[32], vb[32];
        ptx::tmem_ld_32x32_issue(cx.tmem_row, va);
#pragma unroll 1
        for (int c = 0; c < BN; c += 64) {
            ptx::tmem_ld_wait();
            ptx::tmem_ld_32x32_issue(cx.tmem_row + c + 32, vb);
            chunk(va, c);
            ptx::tmem_ld_wait();
            if (c + 64 < BN) ptx::tmem_ld_32x32_issue(cx.tmem_row + c + 64, va);
            chunk(vb, c + 32);
        }
        if (m < M) {
            RowStat rs; rs.m = mx * p.scale; rs.l = l; rs.a = a * p.scale; rs.arg = arg;
            p.part[cx.z][static_cast<size_t>(cx.tile_n) * p.m_pad[cx.z] + m] = rs;
        }
        if (!p.fuse_merge) return;
        // ---- fused merge: threadFenceReduction pattern per row block, then across row blocks ----
        float* red = reinterpret_cast<float*>(cx.scratch);               // [4][6] + flag
        int* flag = reinterpret_cast<int*>(cx.scratch + 128);
        const int z = cx.z;
        const int rb = (z ? p.tiles_m[0] : 0) + cx.tile_m;
        __threadfence();
        ptx::named_bar_sync(1 + cx.bar_base, kEpiThreads);
        if (cx.epi_tid == 0) *flag = (atomicAdd(p.rb_ticket + 1 + rb, 1u) == static_cast<unsigned>(p.n_tiles[z] - 1));
        ptx::named_bar_sync(1 + cx.bar_base, kEpiThreads);
        if (!*flag) return;
        __threadfence();
        float v6[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (m < M) {
            const RowStat* base = p.part[z] + m;
            const size_t stride = p.m_pad[z];
            float gm = -INFINITY, gl = 0.f, ga = 0.f; int garg = 0x7fffffff;
            for (int t = 0; t < p.n_tiles[z]; ++t) {                  // strict >: the first tile wins ties
                const float4 q = __ldcg(reinterpret_cast<const float4*>(base + static_cast<size_t>(t) * stride));
                const float rm = q.x, rl = q.y, ra = q.z; const int rarg = __float_as_int(q.w);
                if (rm > gm) { const float w = __expf(gm - rm); gl = gl * w + rl; ga = ga * w + ra; gm = rm; garg = rarg; }
                else { const float w = __expf(rm - gm); gl = fmaf(rl, w, gl); ga = fmaf(ra, w, ga); }
            }
            const float lse = gm + logf(gl);
            p.lse[z][m] = lse;
            if (p.argmax[z]) p.argmax[z][m] = garg;
            v6[z] = lse - __ldcg(p.diag[z] + m);                       // cross-entropy term
            v6[2 + z] = lse - ga / gl;                                 // entropy
            v6[4 + z] = (garg == m + p.diag_off[z]) ? 1.f : 0.f;       // retrieval hit
        }
#pragma unroll
        for (int i = 0; i < 6; ++i) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v6[i] += __shfl_xor_sync(0xffffffffu, v6[i], o);
            if ((cx.row & 31) == 0) red[(cx.row >> 5) * 6 + i] = v6[i];
        }
        ptx::named_bar_sync(1 + cx.bar_base, kEpiThreads);
        if (cx.epi_tid == 0) {
            for (int i = 0; i < 6; ++i) p.rb_part[rb * 6 + i] = red[i] + red[6 + i] + red[12 + i] + red[18 + i];
            __threadfence();
            const int nrb = p.tiles_m[0] + p.tiles_m[1];
            if (atomicAdd(p.rb_ticket, 1u) == static_cast<unsigned>(nrb - 1)) {
                __threadfence();
                float s6[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                for (int b = 0; b < nrb; ++b)                          // fixed order: deterministic
                    for (int i = 0; i < 6; ++i) s6[i] += __ldcg(p.rb_part + b * 6 + i);
                p.out5[0] = (s6[0] + s6[1]) * 0.5f * p.inv_rows;
                p.out5[1] = s6[4] * p.inv_rows;
                p.out5[2] = s6[5] * p.inv_rows;
                p.out5[3] = s6[2] * p.inv_rows;
                p.out5[4] = s6[3] * p.inv_rows;
                for (int b = 0; b <= nrb; ++b) p.rb_ticket[b] = 0u;    // leave the tickets zeroed
            }
        }
    }
    template <int BN>
    static __device__ __forceinline__ void phase2(const EpiCtx&, const GemmShape&, const Params&) {}
};

// ---- similarity tile -> row AND column softmax statistics in ONE pass (multimodal.py:755 computes `match` once and
// :808-810 reads it along both axes).  EpiSimStats above evaluates S once per direction (two GEMMs and two exp
// passes); here each 128 x 128 slice of an image x text tile yields the partial of its 128 image rows (direction 0)
// and, through a transposed butterfly over the lanes, the partial of its 128 text columns (direction 1: rows of S^T,
// partial index = the image row block).  One exp per element serves both: the exponent uses the FIXED reference
// `scale` (unit-norm features: every raw product is <= 1, so exp(scale*(r-1)) never overflows and, for
// scale <= 32, never leaves the normal fp32 range); each partial is rescaled once to its true maximum so the
// merge (infonce_finalize_kernel) and the arg-max logic are unchanged.  Single device, square problem, full tiles.
struct EpiSimStats1P {
    static constexpr bool kClusterReduce = false;
    static constexpr int kPitch = 36;                                  // floats per row of a warp's transpose buffer
    static constexpr int kWarpBuf = 32 * kPitch * 4;                   // 4608 bytes
    static constexpr int kScratchBytes = 4 * 128 * 16 + 4 * kWarpBuf;  // column partials of the four warps + buffers
    static constexpr int kNumAux = 0;
    static constexpr int kOutElemBytes = 0;
    struct Params {
        float scale;                // exp(s)
        RowStat* part[2];           // [0]: [N/128][m_pad0] image rows; [1]: [M/128][m_pad1] text rows
        int m_pad[2];
        float* diag[2];             // logit at the positive (identical for both directions)
        unsigned int* ticket;       // zeroed here for the merge kernel that follows
    };
    // Column reduction over the 32 rows a warp holds (one row per lane, 32 columns each) through a shared-memory
    // transpose: every lane stores its row (8 x 16 bytes, conflict-free at a pitch of 36 floats), then lane
    // (rg, cg) = (lane / 8, lane % 8) reads columns 4cg..4cg+3 of rows 8rg..8rg+7 with 16-byte loads and the four
    // row groups are folded with two shuffles.  A first version reduced with 31-step lane butterflies: 3x the
    // instructions in long dependent chains, 9.7 us per 128 x 256 tile -- slower than evaluating S twice.
    static __device__ __forceinline__ void store_row(float* buf, int lane, const float (&x)[32]) {
#pragma unroll
        for (int j = 0; j < 8; ++j)
            *reinterpret_cast<float4*>(buf + lane * kPitch + 4 * j) = make_float4(x[4 * j], x[4 * j + 1], x[4 * j + 2], x[4 * j + 3]);
    }
    static __device__ __forceinline__ float4 cols_sum(float* buf, int lane, const float (&x)[32]) {
        store_row(buf, lane, x);
        __syncwarp();
        const int rg = lane >> 3, cg = lane & 7;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float4 q = *reinterpret_cast<const float4*>(buf + (8 * rg + k) * kPitch + 4 * cg);
            acc.x += q.x; acc.y += q.y; acc.z += q.z; acc.w += q.w;
        }
        __syncwarp();                                                  // the buffer is reused right away
#pragma unroll
        for (int o = 8; o <= 16; o <<= 1) {
            acc.x += __shfl_xor_sync(0xffffffffu, acc.x, o); acc.y += __shfl_xor_sync(0xffffffffu, acc.y, o);
            acc.z += __shfl_xor_sync(0xffffffffu, acc.z, o); acc.w += __shfl_xor_sync(0xffffffffu, acc.w, o);
        }
        return acc;
    }
    template <int BN>
    static __device__ __forceinline__ void phase1(const EpiCtx& cx, const GemmShape&, const Params& p) {
        static_assert(BN == 128, "one 128-column slice per epilogue group");
        constexpr float kLog2e = 1.4426950408889634f;
        const int m = cx.m0 + cx.row;                          // image row of this thread
        const int lane = cx.row & 31, wq = cx.row >> 5;
        if (cx.tile_m == 0 && cx.tile_n == 0 && cx.epi_tid == 0) *p.ticket = 0u;
        const float sc2 = p.scale * kLog2e;
        float4* colp = reinterpret_cast<float4*>(cx.scratch);  // [4 warps][128 columns]: sum e, sum e*r, max r, row
        float* buf = reinterpret_cast<float*>(cx.scratch + 4 * 128 * 16 + wq * kWarpBuf);
        const int rg = lane >> 3, cg = lane & 7;
        const int row0 = cx.m0 + wq * 32 + 8 * rg;             // first of the eight rows this lane folds per column
        float rmx = -INFINITY, rl = 0.f, ra = 0.f; int rarg = cx.n0;
        // (one register buffer: prefetching the next 32 columns into a second one spilled and measured slower, 1.80 vs 1.71 ms)
#pragma unroll 1
        for (int c = 0; c < 128; c += 32) {
            float v[32];
            ptx::tmem_ld_32x32(cx.tmem_row + c, v);
            const int n = cx.n0 + c;
            float cm = v[0];
#pragma unroll
            for (int j = 1; j < 32; ++j) cm = fmaxf(cm, v[j]);
            if (cm > rmx) {                                    // strict >: the first maximum of the row
                int k = 31;
#pragma unroll
                for (int j = 31; j >= 0; --j) if (v[j] == cm) k = j;
                rarg = n + k; rmx = cm;
            }
            if (m >= n && m < n + 32) {                        // the positive (square problem: column m)
                float dv = 0.f;
#pragma unroll
                for (int j = 0; j < 32; ++j) if (n + j == m) dv = v[j];
                p.diag[0][m] = dv * p.scale; p.diag[1][m] = dv * p.scale;
            }
            float e[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) { e[j] = exp2f(fmaf(v[j], sc2, -sc2)); rl += e[j]; }
            const float4 ce = cols_sum(buf, lane, e);
#pragma unroll
            for (int j = 0; j < 32; ++j) { e[j] *= v[j]; ra += e[j]; }
            const float4 ca = cols_sum(buf, lane, e);
            // column maxima with the lowest row on ties: rows ascend inside a lane, then the row groups fold
            store_row(buf, lane, v);
            __syncwarp();
            float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY}; int id[4] = {row0, row0, row0, row0};
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const float4 q = *reinterpret_cast<const float4*>(buf + (8 * rg + k) * kPitch + 4 * cg);
                const float qq[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int t = 0; t < 4; ++t) if (qq[t] > mx[t]) { mx[t] = qq[t]; id[t] = row0 + k; }
            }
            __syncwarp();
#pragma unroll
            for (int o = 8; o <= 16; o <<= 1) {
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const float ov = __shfl_xor_sync(0xffffffffu, mx[t], o);
                    const int oid = __shfl_xor_sync(0xffffffffu, id[t], o);
                    if (ov > mx[t] || (ov == mx[t] && oid < id[t])) { mx[t] = ov; id[t] = oid; }
                }
            }
            if (rg == 0) {                                     // lanes 0..7: columns c + 4cg .. c + 4cg + 3
                float4* dst = colp + wq * 128 + c + 4 * cg;
                dst[0] = make_float4(ce.x, ca.x, mx[0], __int_as_float(id[0]));
                dst[1] = make_float4(ce.y, ca.y, mx[1], __int_as_float(id[1]));
                dst[2] = make_float4(ce.z, ca.z, mx[2], __int_as_float(id[2]));
                dst[3] = make_float4(ce.w, ca.w, mx[3], __int_as_float(id[3]));
            }
        }
        {   // row partial, rescaled from the fixed reference to its own maximum
            const float f = exp2f((1.f - rmx) * sc2);
            RowStat rs; rs.m = rmx * p.scale; rs.l = rl * f; rs.a = ra * f * p.scale; rs.arg = rarg;
            p.part[0][static_cast<size_t>(cx.tile_n) * p.m_pad[0] + m] = rs;
        }
        ptx::named_bar_sync(1 + cx.bar_base, kEpiThreads);
        {   // column partial of text row n0 + epi_tid: the four warps in row order (strict >: the lowest row wins ties)
            float l = 0.f, a = 0.f, mx = -INFINITY; int arg = 0;
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                const float4 q = colp[w * 128 + cx.epi_tid];
                l += q.x; a += q.y;
                if (q.z > mx) { mx = q.z; arg = __float_as_int(q.w); }
            }
            const float f = exp2f((1.f - mx) * sc2);
            RowStat rs; rs.m = mx * p.scale; rs.l = l * f; rs.a = a * f * p.scale; rs.arg = arg;
            p.part[1][static_cast<size_t>(cx.tile_m) * p.m_pad[1] + cx.n0 + cx.epi_tid] = rs;
        }
    }
    template <int BN>
    static __device__ __forceinline__ void phase2(const EpiCtx&, const GemmShape&, const Params&) {}
};


// ---- backward, step 1: recompute the logits tile and emit dL/dlogits (bf16) --------------
// G = (softmax_row + softmax_col - 2*I) / (2B)  (SURVEY section 8 row a14; the autograd of
// multimodal.py:808-810).  The bf16 matrix written here is Gs = exp(s)*coef*(softmax_row +
// softmax_col) only, diagonal included: the -2*I term is ~B times larger than any other entry, and
// rounding it to bf16 would dominate the error of every column sum of G (they cancel to ~0).  Per row
// the epilogue also stores gdiag[m] = G_ii - bf16(Gs_ii) in fp32, G_ii = w (expm1(S_ii - lse_q) +
// expm1(S_ii - lse_k)): w (P_row + P_col) and -2w nearly cancel when a pair is confident, and the
// bf16 rounding of the first would otherwise be left as the whole gradient of that row.  The
// consumers (EpiNormBwdT, featgrad_finish_kernel) add gdiag[m] * pos[m]: dI = Gs*T + gdiag o T_pos.
// Direction z=1 (sharded runs only) has the operands swapped and emits the column block Gs^T.
struct EpiGradG {
    static constexpr bool kClusterReduce = false;
    static constexpr int kScratchBytes = 256 * 4;
    static constexpr int kNumAux = 0;
    static constexpr int kOutElemBytes = 2;
    struct Params {
        float scale;                 // exp(s)
        float coef;                  // upstream / (2 * B_global)
        int diag_off[2];
        const float* lse_q[2];       // [M]  log-sum-exp of this direction's rows
        const float* lse_k[2];       // [N]  log-sum-exp of the other direction (columns here)
        float* gdiag[2];             // [M]  G_ii - bf16(Gs_ii) of each row (fp32)
        float* dscale_accum;         // d loss / d s  (atomicAdd, direction 0 only; nullable)
    };
    template <int BN>
    static __device__ __forceinline__ void phase1(const EpiCtx& cx, const GemmShape& gs, const Params& p) {
        const int M = gs.M[cx.z], N = gs.N[cx.z];
        const int m = cx.m0 + cx.row;
        constexpr float kLog2e = 1.4426950408889634f;
        // Gs = w * (2^(r*sc2 - lse_q*log2e) + 2^(r*sc2 - lse_k*log2e)), w = exp(s)*coef: fold log2(w)
        // into both offsets so each softmax term is one FFMA + one MUFU.EX2.
        const float w = p.scale * p.coef;
        const float l2w = log2f(w);
        float* lk = reinterpret_cast<float*>(cx.scratch);
        for (int j = cx.epi_tid; j < BN; j += kEpiThreads)
            lk[j] = (cx.n0 + j < N) ? __ldg(p.lse_k[cx.z] + cx.n0 + j) * kLog2e - l2w : INFINITY;
        ptx::named_bar_sync(1 + cx.bar_base, kEpiThreads);
        const float lq = (m < M) ? __ldg(p.lse_q[cx.z] + m) * kLog2e - l2w : INFINITY;   // dead rows -> 0
        const int dcol = m + p.diag_off[cx.z];
        const float sc2 = p.scale * kLog2e;
        float ds = 0.f;
        auto chunk = [&](float* v, int c) {
            const int n = cx.n0 + c;
            float dv = 0.f;
            if (dcol >= n && dcol < n + 32) {           // the -2*I term (fp32) touches one chunk per row
#pragma unroll
                for (int j = 0; j < 32; ++j) if (n + j == dcol) dv = v[j];
            }
            float g[32];
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
                const float4 k4 = *reinterpret_cast<const float4*>(lk + c + 4 * j4);   // masked columns: +inf -> 0
                const float kk[4] = {k4.x, k4.y, k4.z, k4.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int j = 4 * j4 + q;
                    const float r = v[j];
                    const float gg = exp2f(fmaf(r, sc2, -lq)) + exp2f(fmaf(r, sc2, -kk[q]));
                    ds = fmaf(gg, r, ds);                              // G * logit = Gs * raw dot
                    g[j] = gg;
                }
            }
            if (dcol >= n && dcol < n + 32 && m < M) {  // warp-uniform: one chunk of the diagonal tile per warp
                float gd = 0.f;
#pragma unroll
                for (int j = 0; j < 32; ++j) if (n + j == dcol) gd = g[j];
                const float sii = dv * p.scale;
                const float gii = w * (expm1f(sii - __ldg(p.lse_q[cx.z] + m)) + expm1f(sii - __ldg(p.lse_k[cx.z] + dcol)));
                p.gdiag[cx.z][m] = gii - __bfloat162float(__float2bfloat16_rn(gd));
            }
            ds = fmaf(-2.f * w, dv, ds);
#pragma unroll
            for (int j = 0; j < 4; ++j) swz_st16(cx.out_stage, cx.row, (c + 8 * j) * 2, pack_bf16x8(g + 8 * j));
        };
        float va[32], vb[32];
        ptx::tmem_ld_32x32_issue(cx.tmem_row, va);
#pragma unroll 1
        for (int c = 0; c < BN; c += 64) {
            ptx::tmem_ld_wait();
            ptx::tmem_ld_32x32_issue(cx.tmem_row + c + 32, vb);
            chunk(va, c);
            ptx::tmem_ld_wait();
            if (c + 64 < BN) ptx::tmem_ld_32x32_issue(cx.tmem_row + c + 64, va);
            chunk(vb, c + 32);
        }
        out_tile_commit<BN, 2>(cx);
        if (cx.z == 0 && p.dscale_accum) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) ds += __shfl_xor_sync(0xffffffffu, ds, o);
            if ((cx.row & 31) == 0) atomicAdd(p.dscale_accum, ds);
        }
    }
    template <int BN>
    static __device__ __forceinline__ void phase2(const EpiCtx&, const GemmShape&, const Params&) {}
};

// ---- backward, step 2: dFeat = Gs * Other (+ the diagonal correction), then the F.normalize backward ----
//   acc[m,:] += diag_coef[m] * pos[m,:]                   (pos = positives of the other modality)
//   du = (acc - feat * <feat, acc>) * inv_norm            (cluster along N supplies the dot)
// feat and pos tiles arrive by TMA (aux 0 / aux 1).  Output tile by TMA store: bf16 du (image side,
// operand of the dW GEMM; + dbias column sums) or fp32 scaled by 1/len (text side: d mean-embedding).
template <bool kOutF32>
struct EpiNormBwdT {
    static constexpr bool kClusterReduce = true;
    static constexpr int kScratchBytes = kBM * 4;
    static constexpr int kNumAux = 2;
    static constexpr int kOutElemBytes = kOutF32 ? 4 : 2;
    struct Params {
        const float* inv_norm;                      // [M]
        int normalize;
        const long long* row_len;                   // [M] int64 lengths (nullable): out *= 1/len
        int use_diag;
        const float* diag_coef;                     // [M] gdiag of EpiGradG (read when use_diag)
        float* dbias;                               // [N] atomicAdd (nullable)
    };
    static __device__ __forceinline__ float row_diag_coef(const EpiCtx& cx, const GemmShape& gs, const Params& p) {
        const int m = cx.m0 + cx.row;
        return (p.use_diag && m < gs.M[cx.z]) ? __ldg(p.diag_coef + m) : 0.f;
    }
    template <int BN>
    static __device__ __forceinline__ void load_acc(const EpiCtx& cx, const Params& p, float dc, int c, float* v) {
        ptx::tmem_ld_32x32(cx.tmem_row + c, v);
        if (p.use_diag) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float d[8];
                unpack_bf16x8(swz_ld16(cx.aux[1], cx.row, (c + 8 * j) * 2), d);
#pragma unroll
                for (int k = 0; k < 8; ++k) v[8 * j + k] = fmaf(dc, d[k], v[8 * j + k]);
            }
        }
    }
    template <int BN>
    static __device__ __forceinline__ void phase1(const EpiCtx& cx, const GemmShape& gs, const Params& p) {
        const int N = gs.N[cx.z];
        const float dc = row_diag_coef(cx, gs, p);
        float dot = 0.f;
        if (p.normalize) {
#pragma unroll 1
            for (int c = 0; c < BN; c += 32) {
                float v[32];
                load_acc<BN>(cx, p, dc, c, v);
                const int n = cx.n0 + c;
                if (n >= N) continue;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float f[8];
                    unpack_bf16x8(swz_ld16(cx.aux[0], cx.row, (c + 8 * j) * 2), f);   // OOB columns are 0
#pragma unroll
                    for (int k = 0; k < 8; ++k) dot = fmaf(f[k], v[8 * j + k], dot);
                }
            }
        }
        reinterpret_cast<float*>(cx.scratch)[cx.row] = dot;
    }
    template <int BN>
    static __device__ __forceinline__ void phase2(const EpiCtx& cx, const GemmShape& gs, const Params& p) {
        const int M = gs.M[cx.z], N = gs.N[cx.z];
        const int m = cx.m0 + cx.row;
        const bool rv = m < M;
        const float* my = reinterpret_cast<const float*>(cx.scratch) + cx.row;
        float dot = 0.f;
        const uint32_t nc = ptx::cluster_nctarank();
        for (uint32_t r = 0; r < nc; ++r) dot += ptx::ld_dsmem_f32(my, r);
        const float inv = (p.normalize && rv) ? __ldg(p.inv_norm + m) : 1.f;
        const float rs = (p.row_len && rv) ? 1.f / static_cast<float>(p.row_len[m]) : 1.f;
        const float dc = row_diag_coef(cx, gs, p);
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
            float v[32];
            load_acc<BN>(cx, p, dc, c, v);
            const int n = cx.n0 + c;
            if (p.normalize) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float f[8];
                    unpack_bf16x8(swz_ld16(cx.aux[0], cx.row, (c + 8 * j) * 2), f);
#pragma unroll
                    for (int k = 0; k < 8; ++k) v[8 * j + k] = (v[8 * j + k] - f[k] * dot) * inv;
                }
            }
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = (rv && n + j < N) ? v[j] * rs : 0.f;
            if constexpr (kOutF32) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    uint4 q;
                    q.x = __float_as_uint(v[4 * j]); q.y = __float_as_uint(v[4 * j + 1]);
                    q.z = __float_as_uint(v[4 * j + 2]); q.w = __float_as_uint(v[4 * j + 3]);
                    swz_st16(cx.out_stage, cx.row, (c + 4 * j) * 4, q);
                }
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) swz_st16(cx.out_stage, cx.row, (c + 8 * j) * 2, pack_bf16x8(v + 8 * j));
            }
            if (p.dbias && n < N) {
                // column sums over the 32 rows of this warp: butterfly transpose-reduce (31 shuffles
                // for 32 columns); lane j ends up owning column j.
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const bool upper = (cx.row & o) != 0;
#pragma unroll
                    for (int j = 0; j < o; ++j) {
                        const float send = upper ? v[j] : v[j + o];
                        const float keep = upper ? v[j + o] : v[j];
                        v[j] = keep + __shfl_xor_sync(0xffffffffu, send, o);
                    }
                }
                const int col = n + (cx.row & 31);
                if (col < N) atomicAdd(p.dbias + col, v[0]);
            }
        }
        out_tile_commit<BN, kOutElemBytes>(cx);
    }
};

// ---- spatial "max" similarity (multimodal.py:771-780) -----------------------------------------
// GEMM rows = text tokens (t,l), columns = image locations (i,hw).  A 128 x 256 tile holds
// TPM = 128/L whole texts and IPN = 256/HW whole images (tile origins step by TPM*L / IPN*HW).
// Thread = one token row: running max + argmax over each image's HW columns (in-thread), then the
// L token maxima of a text are summed through shared memory and divided by len[t]:
//   match[i,t] = sum_l max_hw <img[i,hw,:], tok[t,l,:]> / len[t]       (never stores [B,B,L,HW])
// The argmax location is kept (uint8, both [i][t,l] and [t,l][i] layouts) for the backward.
struct EpiSpatialMax {
    static constexpr bool kClusterReduce = false;
    static constexpr int kMaxIPN = 16;
    static constexpr int kScratchBytes = kBM * kMaxIPN * 4;
    static constexpr int kNumAux = 0;
    static constexpr int kOutElemBytes = 0;
    struct Params {
        int L, HW, TPM, IPN;          // tokens per text, locations per image, texts / images per tile
        int Bt, Bi;
        const long long* lens;        // [Bt]
        float* match;                 // [Bi, Bt]
        unsigned char* amax_it;       // [Bi, Bt*L]
        unsigned char* amax_ti;       // [Bt*L, Bi]
    };
    // Static-segment fast path (HW known at compile time, e.g. the 7x7 = 49 locations of the ResNeXt
    // layer4 map): the chunk loop is fully unrolled, so every column's image slot is a compile-time
    // constant, the running maxima live in registers, and the hot loop is one FMNMX per element; the
    // arg-max scan only runs when a chunk improves its segment's maximum.
    template <int BN, int HW>
    static __device__ __forceinline__ void phase1_static(const EpiCtx& cx, const Params& p) {
        constexpr int IPN = BN / HW;
        float* vals = reinterpret_cast<float*>(cx.scratch);          // [128][IPN]
        const int r = cx.row;
        const int grow = cx.m0 + r;
        const bool row_ok = r < p.TPM * p.L && grow < p.Bt * p.L;
        const int img0 = cx.tile_n * IPN;
        float best[IPN]; int barg[IPN];
#pragma unroll
        for (int q = 0; q < IPN; ++q) { best[q] = -INFINITY; barg[q] = 0; }
        float va[32], vb[32];
        ptx::tmem_ld_32x32_issue(cx.tmem_row, va);
#pragma unroll
        for (int c = 0; c < BN; c += 32) {
            float* v = ((c >> 5) & 1) ? vb : va;
            ptx::tmem_ld_wait();
            if (c + 32 < BN) ptx::tmem_ld_32x32_issue(cx.tmem_row + c + 32, ((c >> 5) & 1) ? va : vb);
            // a 32-column chunk touches at most two image segments
#pragma unroll
            for (int part = 0; part < 2; ++part) {
                const int q = c / HW + part;                          // compile-time after unrolling
                const int lo = part == 0 ? 0 : (c / HW + 1) * HW - c;
                const int hi = part == 0 ? ((c / HW + 1) * HW - c < 32 ? (c / HW + 1) * HW - c : 32) : 32;
                if (q < IPN && lo < hi && lo < 32) {
                    float cm = v[lo];
#pragma unroll
                    for (int j = lo + 1; j < hi; ++j) cm = fmaxf(cm, v[j]);
                    if (cm > best[q]) {                               // strict >: earlier columns win ties
                        int k = hi - 1;
#pragma unroll
                        for (int j = hi - 1; j >= lo; --j) if (v[j] == cm) k = j;
                        best[q] = cm; barg[q] = c + k - q * HW;
                    }
                }
            }
        }
#pragma unroll
        for (int q = 0; q < IPN; ++q) {
            vals[r * IPN + q] = best[q];
            const int i = img0 + q;
            if (row_ok && i < p.Bi) {
                p.amax_it[static_cast<size_t>(i) * (p.Bt * p.L) + grow] = static_cast<unsigned char>(barg[q]);
                p.amax_ti[static_cast<size_t>(grow) * p.Bi + i] = static_cast<unsigned char>(barg[q]);
            }
        }
        ptx::named_bar_sync(1 + cx.bar_base, kEpiThreads);
        if (cx.epi_tid < p.TPM * IPN) {
            const int tt = cx.epi_tid / IPN, qq = cx.epi_tid % IPN;
            const int t = cx.tile_m * p.TPM + tt, i = img0 + qq;
            if (t < p.Bt && i < p.Bi) {
                float s = 0.f;
                for (int l = 0; l < p.L; ++l) s += vals[(tt * p.L + l) * IPN + qq];
                p.match[static_cast<size_t>(i) * p.Bt + t] = s / static_cast<float>(p.lens[t]);
            }
        }
    }
    template <int BN>
    static __device__ __forceinline__ void phase1(const EpiCtx& cx, const GemmShape& gs, const Params& p) {
        if constexpr (BN == 256) {
            if (p.HW == 49 && p.IPN == 5) { phase1_static<256, 49>(cx, p); return; }
        }
        float* vals = reinterpret_cast<float*>(cx.scratch);          // [128][IPN]
        const int r = cx.row;
        const int grow = cx.m0 + r;                                  // global token row
        const bool row_ok = r < p.TPM * p.L && grow < p.Bt * p.L;
        const int img0 = cx.tile_n * p.IPN;                          // first image of this tile
        int q = 0, nextb = p.HW, hw = 0;
        float best = -INFINITY; int barg = 0;
        const int ncols = p.IPN * p.HW;
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
            float v[32];
            ptx::tmem_ld_32x32(cx.tmem_row + c, v);
            if (c >= ncols) continue;                                // warp-uniform
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const int col = c + j;
                if (col < ncols) {
                    if (v[j] > best) { best = v[j]; barg = hw; }     // strict >: first maximum
                    ++hw;
                    if (col + 1 == nextb) {                          // end of image q's segment
                        vals[r * p.IPN + q] = best;
                        const int i = img0 + q;
                        if (row_ok && i < p.Bi) {
                            p.amax_it[static_cast<size_t>(i) * (p.Bt * p.L) + grow] = static_cast<unsigned char>(barg);
                            p.amax_ti[static_cast<size_t>(grow) * p.Bi + i] = static_cast<unsigned char>(barg);
                        }
                        ++q; nextb += p.HW; hw = 0; best = -INFINITY; barg = 0;
                    }
                }
            }
        }
        ptx::named_bar_sync(1 + cx.bar_base, kEpiThreads);
        if (cx.epi_tid < p.TPM * p.IPN) {
            const int tt = cx.epi_tid / p.IPN, qq = cx.epi_tid % p.IPN;
            const int t = cx.tile_m * p.TPM + tt, i = img0 + qq;
            if (t < p.Bt && i < p.Bi) {
                float s = 0.f;
                for (int l = 0; l < p.L; ++l) s += vals[(tt * p.L + l) * p.IPN + qq];
                p.match[static_cast<size_t>(i) * p.Bt + t] = s / static_cast<float>(p.lens[t]);
            }
        }
    }
    template <int BN>
    static __device__ __forceinline__ void phase2(const EpiCtx&, const GemmShape&, const Params&) {}
};

}  // namespace cvcl
