// libcvcl_b200.so -- C-ABI entry points (see include/cvcl_b200.h for the contract and the
// reference file:line each one replaces).  Links only cudart; no libtorch, no CPU path.
#include "../../include/cvcl_b200.h"
#include "gemm_launch.cuh"
#include "kernels_simt.cuh"
#include "peer_collectives.cuh"
#include "fused_step.cuh"
#include <cmath>
#include <cstdlib>
#include <cstring>

using namespace cvcl;

namespace {

constexpr int kBN = 128;
constexpr int kStages = 4;

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
// the fused step zeroes the split-K scratch on its side stream; it tells the head entry point so
inline bool& head_scratch_zeroed() { static thread_local bool v = false; return v; }
inline bool head_splitk_disabled() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("CVCL_B200_HEAD_SPLITK"); v = (e && e[0] == '0') ? 1 : 0; }
    return v == 1;
}
inline int warps_grid(long long n_warps, int block = 256) {
    return static_cast<int>((n_warps * 32 + block - 1) / block);
}
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
inline int pad8(int x) { return (x + 7) / 8 * 8; }

struct SimWs {               // carve-up of the sim workspace
    RowStat* part[2]; int m_pad[2]; int n_tiles[2]; int tiles_m[2];
    float* diag[2]; float* block_part; unsigned int* ticket; unsigned int* rb_ticket; float* rb_part;
    size_t bytes;
};
inline int sim_bn(int N0, int N1) { return (N0 > N1 ? N0 : N1) >= 4096 ? 256 : 128; }   // tile width of the sim kernels
SimWs carve_sim_ws(void* ws, int M0, int N0, int M1, int N1) {
    SimWs w{};
    const int bn = 128;                 // epilogue tile width (the MMA tile may be 256 wide)
    const int M[2] = {M0, M1}, N[2] = {N0, N1};
    size_t off = 0;
    unsigned char* base = static_cast<unsigned char*>(ws);
    w.ticket = reinterpret_cast<unsigned int*>(base + off); off += 256;
    w.tiles_m[0] = ceil_div(M0, kBM); w.tiles_m[1] = ceil_div(M1, kBM);
    w.rb_ticket = reinterpret_cast<unsigned int*>(base + off);
    off += align_up(sizeof(unsigned int) * (1 + w.tiles_m[0] + w.tiles_m[1]), 256);
    w.rb_part = reinterpret_cast<float*>(base + off);
    off += align_up(sizeof(float) * 6 * (w.tiles_m[0] + w.tiles_m[1]), 256);
    for (int z = 0; z < 2; ++z) {
        w.m_pad[z] = ceil_div(M[z], kBM) * kBM;
        w.n_tiles[z] = ceil_div(N[z], bn);
        w.part[z] = reinterpret_cast<RowStat*>(base + off);
        off += align_up(sizeof(RowStat) * static_cast<size_t>(w.m_pad[z]) * w.n_tiles[z], 256);
        w.diag[z] = reinterpret_cast<float*>(base + off);
        off += align_up(sizeof(float) * static_cast<size_t>(w.m_pad[z]), 256);
    }
    const int fin_blocks = ceil_div(M0 + M1, 256);
    w.block_part = reinterpret_cast<float*>(base + off);
    off += align_up(sizeof(float) * 6 * static_cast<size_t>(fin_blocks), 256);
    w.bytes = off;
    return w;
}

}  // namespace

extern "C" {

int cvcl_abi_version(void) { return CVCL_ABI_VERSION; }
const char* cvcl_last_error(void) { return last_error_buf(); }
unsigned long long cvcl_launch_count(void) { return __atomic_load_n(&launch_counter(), __ATOMIC_RELAXED); }

// Host staging memory for the H2D copy of a batch: page-locked and (optionally) WRITE-COMBINED.  The CPU never
// caches write-combined lines, so the DMA engine reads them from DRAM without snooping the CPU caches (measured on
// this pool's hosts: 2.2 MB from an ordinary pinned buffer whose lines sit in a CPU cache takes ~200 us instead of
// 46 us).  The CPU should only WRITE such a buffer (reads are uncached and slow).
void* cvcl_host_alloc(size_t bytes, int write_combined) {
    void* p = nullptr;
    const unsigned int flags = cudaHostAllocPortable | (write_combined ? cudaHostAllocWriteCombined : 0u);
    if (bytes == 0 || cudaHostAlloc(&p, bytes, flags) != cudaSuccess) {
        cudaGetLastError();
        fail(CVCL_ERR_CUDA, "host_alloc: cudaHostAlloc(%zu bytes) failed", bytes);
        return nullptr;
    }
    return p;
}

int cvcl_host_free(void* p) {
    if (p) CVCL_CHECK_CUDA(cudaFreeHost(p));
    return CVCL_OK;
}

// ------------------------------------------------------------------------------------ K1
int cvcl_text_encoder_fwd(const int64_t* ids, const int64_t* lens, const float* table,
                          int B, int L, int E, int V, int normalize, int per_token, float pool_scale,
                          float* feat_f32, void* feat_bf16, int ld_bf16,
                          float* inv_norm, float* tok_f32, void* tok_bf16, int* status, void* stream) {
    if (B == 0) return CVCL_OK;
    CVCL_REQUIRE(ids && lens && table, "text_encoder_fwd: null input");
    CVCL_REQUIRE(B >= 0 && L > 0 && V > 0, "text_encoder_fwd: bad shape B=%d L=%d V=%d", B, L, V);
    CVCL_REQUIRE(E > 0 && E % 4 == 0 && E <= 128 * kMaxVec, "text_encoder_fwd: E=%d must be a multiple of 4, <= %d", E, 128 * kMaxVec);
    CVCL_REQUIRE((reinterpret_cast<uintptr_t>(table) & 15) == 0, "text_encoder_fwd: table not 16-byte aligned");
    if (B == 0) return CVCL_OK;
    TextFwdParams p{};
    p.ids = reinterpret_cast<const long long*>(ids); p.lens = reinterpret_cast<const long long*>(lens);
    p.table = table; p.B = B; p.L = L; p.E = E; p.V = V; p.normalize = normalize; p.per_token = per_token;
    p.pool_scale = pool_scale; p.feat_f32 = feat_f32;
    p.feat_bf16 = static_cast<__nv_bfloat16*>(feat_bf16); p.ld_bf16 = ld_bf16;
    p.inv_norm = inv_norm; p.tok_f32 = tok_f32; p.tok_bf16 = static_cast<__nv_bfloat16*>(tok_bf16);
    p.status = status;
    if (!per_token && E <= 512 && B <= 4096)      // small batch: block per utterance, 8 rows in flight per lane
        CVCL_CHECK_CUDA(launch_pdl(text_encoder_flat_wide_kernel, dim3(B), dim3(128), 0, as_stream(stream), p));
    else
        CVCL_CHECK_CUDA(launch_pdl(text_encoder_fwd_kernel, dim3(warps_grid(B, 128)), dim3(128), 0, as_stream(stream), p));
    count_launch();
    return CVCL_OK;
}

int cvcl_embedding_gather(const int64_t* ids, const float* table, float* out, int n_tok, int E, int V,
                          void* stream) {
    CVCL_REQUIRE(ids && table && out, "embedding_gather: null pointer");
    CVCL_REQUIRE(E > 0 && E % 4 == 0, "embedding_gather: E=%d must be a multiple of 4", E);
    if (n_tok == 0) return CVCL_OK;
    CVCL_CHECK_CUDA(launch_pdl(embedding_gather_kernel, dim3(warps_grid(n_tok)), dim3(256), 0, as_stream(stream), reinterpret_cast<const long long*>(ids), table, out, n_tok, E, V));
    count_launch();
    return CVCL_OK;
}

int cvcl_embedding_scatter_add(const int64_t* ids, const float* g, float* dtable, int B, int L, int E,
                               int V, int per_token, void* stream) {
    CVCL_REQUIRE(ids && g && dtable, "embedding_scatter_add: null pointer");
    CVCL_REQUIRE(E > 0 && E % 4 == 0 && E <= 128 * kMaxVec, "embedding_scatter_add: bad E=%d", E);
    if (B == 0) return CVCL_OK;
    if (per_token) { B = B * L; L = 1; }
    CVCL_CHECK_CUDA(launch_pdl(embedding_scatter_add_kernel, dim3(warps_grid(static_cast<long long>(B) * L)), dim3(256), 0, as_stream(stream), reinterpret_cast<const long long*>(ids), g, dtable, B, L, E, V, per_token));
    count_launch();
    return CVCL_OK;
}

int cvcl_text_token_bwd(const int64_t* ids, const int64_t* lens, const float* table, const float* dtok,
                        const float* dpool, float pool_scale, float* dtable, int B, int L, int E, int V,
                        int normalize, void* stream) {
    CVCL_REQUIRE(ids && lens && table && dtable && (dtok || dpool), "text_token_bwd: null pointer");
    CVCL_REQUIRE(E > 0 && E % 4 == 0 && E <= 128 * kMaxVec, "text_token_bwd: bad E=%d", E);
    if (B == 0) return CVCL_OK;
    CVCL_CHECK_CUDA(launch_pdl(text_token_bwd_kernel, dim3(warps_grid(static_cast<long long>(B) * L)), dim3(256), 0, as_stream(stream), reinterpret_cast<const long long*>(ids), reinterpret_cast<const long long*>(lens), table, dtok, dpool, pool_scale, dtable, B, L, E, V, normalize));
    count_launch();
    return CVCL_OK;
}

int cvcl_cast_transpose(const void* src, int src_is_bf16, void* dst, void* dst_t, int batch, int R, int C,
                        int64_t ld_src, int64_t ld_dst, int64_t ld_t, int64_t bs_src, int64_t bs_dst,
                        int64_t bs_t, void* stream) {
    CVCL_REQUIRE(src && (dst || dst_t), "cast_transpose: null pointer");
    if (batch == 0 || R == 0 || C == 0) return CVCL_OK;
    CVCL_REQUIRE(batch <= 65535 && ceil_div(R, 32) <= 65535, "cast_transpose: grid too large");
    if (!src_is_bf16 && dst && !dst_t && batch == 1 && ld_src == C && ld_dst == C &&
        (static_cast<long long>(R) * C) % 8 == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0 &&
        (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {                 // contiguous: vectorised cast
        const long long n8 = static_cast<long long>(R) * C / 8;
        const int blocks = static_cast<int>(n8 / 256 + 1 < 148 * 16 ? n8 / 256 + 1 : 148 * 16);
        CVCL_CHECK_CUDA(launch_pdl(cast_f32_bf16_kernel, dim3(blocks), dim3(256), 0, as_stream(stream), static_cast<const float*>(src), static_cast<__nv_bfloat16*>(dst), n8));
        count_launch();
        return CVCL_OK;
    }
    dim3 grid(ceil_div(C, 32), ceil_div(R, 32), batch);
    if (src_is_bf16)
        CVCL_CHECK_CUDA(launch_pdl(cast_transpose_kernel<__nv_bfloat16>, dim3(grid), dim3(256), 0, as_stream(stream), static_cast<const __nv_bfloat16*>(src), static_cast<__nv_bfloat16*>(dst), static_cast<__nv_bfloat16*>(dst_t), R, C, ld_src, ld_dst, ld_t, bs_src, bs_dst, bs_t));
    else
        CVCL_CHECK_CUDA(launch_pdl(cast_transpose_kernel<float>, dim3(grid), dim3(256), 0, as_stream(stream), static_cast<const float*>(src), static_cast<__nv_bfloat16*>(dst), static_cast<__nv_bfloat16*>(dst_t), R, C, ld_src, ld_dst, ld_t, bs_src, bs_dst, bs_t));
    count_launch();
    return CVCL_OK;
}

int cvcl_embedding_bag_bwd(const int64_t* ids, const int64_t* lens, const float* g, const float* feat,
                           const float* inv_norm, int normalize, float* dtable, int B, int L, int E, int V,
                           void* stream) {
    CVCL_REQUIRE(ids && lens && g && dtable, "embedding_bag_bwd: null pointer");
    CVCL_REQUIRE(!normalize || (feat && inv_norm), "embedding_bag_bwd: normalize needs feat and inv_norm");
    CVCL_REQUIRE(E > 0 && E % 4 == 0 && E <= 128 * kMaxVec, "embedding_bag_bwd: bad E=%d", E);
    if (B == 0) return CVCL_OK;
    CVCL_CHECK_CUDA(launch_pdl(embedding_bag_bwd_kernel, dim3(warps_grid(B)), dim3(256), 0, as_stream(stream), reinterpret_cast<const long long*>(ids), reinterpret_cast<const long long*>(lens), g, feat, inv_norm, normalize, dtable, B, L, E, V));
    count_launch();
    return CVCL_OK;
}

int cvcl_rownorm_bwd(const float* g, const float* feat, const float* inv_norm, int M, int E, int normalize,
                     float* du_f32, void* du_bf16, int ld, void* du_bf16_t, int ld_t, float* dbias,
                     void* stream) {
    CVCL_REQUIRE(g, "rownorm_bwd: null pointer");
    CVCL_REQUIRE(!normalize || (feat && inv_norm), "rownorm_bwd: normalize needs feat and inv_norm");
    CVCL_REQUIRE(E > 0 && E % 4 == 0 && E <= 128 * kMaxVec, "rownorm_bwd: bad E=%d", E);
    if (M == 0) return CVCL_OK;
    CVCL_CHECK_CUDA(launch_pdl(rownorm_bwd_kernel, dim3(warps_grid(M)), dim3(256), 0, as_stream(stream), g, feat, inv_norm, M, E, normalize, du_f32, static_cast<__nv_bfloat16*>(du_bf16), ld, static_cast<__nv_bfloat16*>(du_bf16_t), ld_t, dbias));
    count_launch();
    return CVCL_OK;
}

int cvcl_spatial_pool(const float* src, int B, int HW, int E, float* out_f32, void* out_bf16, int ld,
                      void* out_bf16_t, int ld_t, void* stream) {
    CVCL_REQUIRE(src && (out_f32 || out_bf16 || out_bf16_t), "spatial_pool: null pointer");
    CVCL_REQUIRE(E > 0 && E % 4 == 0 && HW > 0, "spatial_pool: bad shape");
    if (B == 0) return CVCL_OK;
    for (int b0 = 0; b0 < B; b0 += 65535) {              // grid.y holds at most 65535 maps per launch
        const int nb = B - b0 < 65535 ? B - b0 : 65535;
        dim3 grid(ceil_div(E / 4, 128), nb);
        CVCL_CHECK_CUDA(launch_pdl(spatial_pool_kernel, dim3(grid), dim3(128), 0, as_stream(stream),
                                   src + static_cast<size_t>(b0) * HW * E, nb, HW, E,
                                   out_f32 ? out_f32 + static_cast<size_t>(b0) * E : nullptr,
                                   out_bf16 ? static_cast<__nv_bfloat16*>(out_bf16) + static_cast<size_t>(b0) * ld : nullptr, ld,
                                   out_bf16_t ? static_cast<__nv_bfloat16*>(out_bf16_t) + b0 : nullptr, ld_t));
        count_launch();
    }
    return CVCL_OK;
}

int cvcl_linear_f32(const float* A, int lda, const float* W, int ldw, const float* bias, int M, int N, int K,
                    float* C, int ldc, void* stream) {
    CVCL_REQUIRE(A && W && C, "linear_f32: null pointer");
    CVCL_REQUIRE(M >= 0 && N > 0 && K > 0 && K % 4 == 0 && lda % 4 == 0 && ldw % 4 == 0, "linear_f32: bad shape");
    CVCL_REQUIRE(((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(W)) & 15) == 0,
                 "linear_f32: 16-byte alignment required");
    if (M == 0) return CVCL_OK;
    dim3 grid(ceil_div(N, 64), ceil_div(M, 64));
    CVCL_CHECK_CUDA(launch_pdl(linear_f32_kernel, grid, dim3(256), 0, as_stream(stream), A, lda, W, ldw, bias, M, N, K, C, ldc));
    count_launch();
    return CVCL_OK;
}

int cvcl_conv1x1_f32(const float* x, const float* w, const float* bias, int B, int K, int HW, int E, float* out,
                     void* stream) {
    CVCL_REQUIRE(x && w && out, "conv1x1_f32: null pointer");
    CVCL_REQUIRE(B >= 0 && K > 0 && K % 4 == 0 && HW > 0 && E > 0, "conv1x1_f32: bad shape B=%d K=%d HW=%d E=%d", B, K, HW, E);
    CVCL_REQUIRE((reinterpret_cast<uintptr_t>(w) & 15) == 0, "conv1x1_f32: weight not 16-byte aligned");
    const long long M = static_cast<long long>(B) * HW;
    CVCL_REQUIRE(M <= 0x7fffffffLL - 64 && ceil_div(E, 64) <= 65535, "conv1x1_f32: too many rows / channels");
    if (M == 0) return CVCL_OK;
    dim3 grid(static_cast<unsigned>((M + 63) / 64), ceil_div(E, 64));
    CVCL_CHECK_CUDA(launch_pdl(conv1x1_f32_kernel, grid, dim3(256), 0, as_stream(stream), x, w, bias,
                               static_cast<int>(M), E, K, HW, out));
    count_launch();
    return CVCL_OK;
}

int cvcl_spatial_max_scores_f32(const float* img, const float* tok, const int64_t* lens, const int* txt_index, int M,
                                int HW, int E, int C, int L, int n_way, float log_scale, float* out, void* stream) {
    CVCL_REQUIRE(img && tok && lens && out, "spatial_max_scores_f32: null pointer");
    CVCL_REQUIRE(M >= 0 && C > 0 && L > 0 && n_way >= 0, "spatial_max_scores_f32: bad shape M=%d C=%d L=%d n_way=%d",
                 M, C, L, n_way);
    CVCL_REQUIRE(HW > 0 && HW <= 256, "spatial_max_scores_f32: HW=%d must be in [1, 256]", HW);
    CVCL_REQUIRE(E > 0 && E % 4 == 0, "spatial_max_scores_f32: E=%d must be a multiple of 4", E);
    CVCL_REQUIRE(((reinterpret_cast<uintptr_t>(img) | reinterpret_cast<uintptr_t>(tok)) & 15) == 0,
                 "spatial_max_scores_f32: 16-byte alignment required");
    CVCL_REQUIRE(n_way == 0 || M % n_way == 0, "spatial_max_scores_f32: M=%d is not a multiple of n_way=%d", M, n_way);
    CVCL_REQUIRE(n_way == 0 || txt_index || M / n_way <= C,
                 "spatial_max_scores_f32: %d trials without txt_index need as many labels (C=%d)", M / n_way, C);
    if (M == 0) return CVCL_OK;
    const int E4 = E / 4;
    // token rows per chunk: every row a label needs in one chunk where possible, at most 4 rows per work item and
    // 256 work items per block
    const int rows_wanted = n_way > 0 ? L : (C * L < 64 ? C * L : 64);
    int tt = (rows_wanted + 3) / 4 * 4;
    const int tt_cap = 4 * (256 / HW) < 64 ? 4 * (256 / HW) : 64;
    if (tt > tt_cap) tt = tt_cap;
    int max_smem = 0, dev = 0;
    CVCL_CHECK_CUDA(cudaGetDevice(&dev));
    CVCL_CHECK_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    int ks = 0, ld4 = 0;
    size_t smem = 0;
    for (;; tt -= 4) {
        CVCL_REQUIRE(tt >= 4, "spatial_max_scores_f32: the %d x %d image block does not fit in shared memory", HW, E);
        const int items = (tt / 4) * HW;
        ks = 1;
        while (ks < 32 && 2 * ks * items <= 256 && E4 % (2 * ks) == 0) ks *= 2;
        // quarter-warps of 8 lanes read 8 distinct 16-byte bank groups when the row stride is = ks (mod 8)
        ld4 = ks >= 8 ? E4 : E4 + ((ks - E4 % 8) + 8) % 8;
        smem = static_cast<size_t>(HW) * ld4 * 16 + static_cast<size_t>(tt) * E4 * 16 +
               static_cast<size_t>(tt) * HW * 4 + static_cast<size_t>(tt) * 12 + 8;
        if (smem <= static_cast<size_t>(max_smem)) break;
    }
    static thread_local unsigned attr_mask = 0;         // per device: function attributes live in the device's context
    const int attr_dev = dev >= 0 && dev < 32 ? dev : 0;
    if (!((attr_mask >> attr_dev) & 1u)) {
        CVCL_CHECK_CUDA(cudaFuncSetAttribute(spatial_max_scores_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             max_smem));
        attr_mask |= 1u << attr_dev;
    }
    SpatialMaxScoreParams p{};
    p.img = img; p.tok = tok; p.lens = reinterpret_cast<const long long*>(lens); p.txt_index = txt_index;
    p.M = M; p.HW = HW; p.E = E; p.C = C; p.L = L; p.n_way = n_way; p.tt = tt; p.ks = ks; p.ld4 = ld4;
    p.scale = expf(log_scale); p.out = out;
    CVCL_CHECK_CUDA(launch_pdl(spatial_max_scores_f32_kernel, dim3(M), dim3(256), smem, as_stream(stream), p));
    count_launch();
    return CVCL_OK;
}

int cvcl_normalize_rows_f32(const float* src, float* dst, long long M, int E, void* stream) {
    CVCL_REQUIRE(src && dst, "normalize_rows_f32: null pointer");
    CVCL_REQUIRE(M >= 0 && E > 0 && E % 4 == 0, "normalize_rows_f32: bad shape");
    if (M == 0) return CVCL_OK;
    CVCL_CHECK_CUDA(launch_pdl(normalize_rows_f32_kernel, dim3(warps_grid(M)), dim3(256), 0, as_stream(stream), src, dst, M, E));
    count_launch();
    return CVCL_OK;
}

int cvcl_row_argmax_f32(const float* scores, long long ld, long long M, int N, int col0, int merge, float* best,
                        int* arg, void* stream) {
    CVCL_REQUIRE(scores && best && arg, "row_argmax_f32: null pointer");
    CVCL_REQUIRE(M >= 0 && N > 0 && ld >= N, "row_argmax_f32: bad shape");
    if (M == 0) return CVCL_OK;
    CVCL_CHECK_CUDA(launch_pdl(row_argmax_f32_kernel, dim3(warps_grid(M)), dim3(256), 0, as_stream(stream), scores, ld, M, N,
                               col0, merge, best, arg));
    count_launch();
    return CVCL_OK;
}

int cvcl_spatial_pool_bwd(const float* g, int B, int HW, int E, float* dst, void* stream) {
    CVCL_REQUIRE(g && dst, "spatial_pool_bwd: null pointer");
    CVCL_REQUIRE(E > 0 && E % 4 == 0 && HW > 0, "spatial_pool_bwd: bad shape");
    if (B == 0) return CVCL_OK;
    dim3 grid(ceil_div(E / 4, 128), B);
    CVCL_CHECK_CUDA(launch_pdl(spatial_pool_bwd_kernel, dim3(grid), dim3(128), 0, as_stream(stream), g, B, HW, E, dst));
    count_launch();
    return CVCL_OK;
}

// m_limit / k_limit: device-side sizes (see GemmShape); null = the host shapes
static int gemm_f32out_limited(const void* A, int lda, int a_mn, const void* Bm, int ldb, int b_mn, int M, int N, int K,
                               float alpha, float* C, int ldc, const int* m_limit, const int* k_limit, void* stream);

int cvcl_gemm_f32out(const void* A, int lda, int a_mn, const void* Bm, int ldb, int b_mn, int M, int N, int K,
                     float alpha, float* C, int ldc, void* stream) {
    return gemm_f32out_limited(A, lda, a_mn, Bm, ldb, b_mn, M, N, K, alpha, C, ldc, nullptr, nullptr, stream);
}

static int gemm_f32out_limited(const void* A, int lda, int a_mn, const void* Bm, int ldb, int b_mn, int M, int N, int K,
                               float alpha, float* C, int ldc, const int* m_limit, const int* k_limit, void* stream) {
    CVCL_REQUIRE(A && Bm && C, "gemm_f32out: null pointer");
    CVCL_REQUIRE(M > 0 && N > 0 && K > 0, "gemm_f32out: bad shape");
    GemmOperands op{}; op.ndir = 1;
    op.A[0] = a_mn ? mat(A, K, M, lda) : mat(A, M, K, lda);
    op.B[0] = b_mn ? mat(Bm, K, N, ldb) : mat(Bm, N, K, ldb);
    op.out[0] = mat(C, M, N, ldc);
    GemmShape gs{}; gs.M[0] = gs.M[1] = M; gs.N[0] = gs.N[1] = N; gs.K = K; gs.m_stride = kBM; gs.n_stride = kBN;
    gs.m_limit = m_limit; gs.k_limit = k_limit;
    cudaStream_t st = as_stream(stream);
    if ((ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(C) & 15) == 0) {
        EpiStoreF32::Params ep{}; ep.alpha = alpha;
        if (K >= 2048 && N >= 256 && ceil_div(M, kBM) * ceil_div(N, 256) >= sm_count()) {
            // long contraction, enough tiles: 128 x 256 tiles read A once per 256 columns
            // (measured 975 -> 1127 TF/s at 32768 x 512 x 32768)
            gs.n_stride = 256;
            // few column tiles, long rows of A (the spatial-max backward: A = the 2.5 GB arg-max matrix, N = E): let
            // the column tiles of one row block run side by side so A crosses HBM once (ncu: 5.2 GB read for a
            // 2.5 GB operand with the row-block-major order)
            gs.n_fast = ceil_div(N, 256) <= 4 ? 1 : 0;
            if (!a_mn && !b_mn) return launch_gemm<256, 3, EpiStoreF32, false, false>(op, gs, ep, 1, st);
            if (!a_mn && b_mn) return launch_gemm<256, 3, EpiStoreF32, false, true>(op, gs, ep, 1, st);
            if (a_mn && !b_mn) return launch_gemm<256, 3, EpiStoreF32, true, false>(op, gs, ep, 1, st);
            return launch_gemm<256, 3, EpiStoreF32, true, true>(op, gs, ep, 1, st);
        }
        // 2-deep ring = 64 KB (also the fp32 staging tile): three CTAs per SM hide each other's
        // prologue / epilogue (measured 430 -> 707 TF/s at 16384^2 x 512)
        if (!a_mn && !b_mn) return launch_gemm<kBN, 2, EpiStoreF32, false, false>(op, gs, ep, 1, st);
        if (!a_mn && b_mn) return launch_gemm<kBN, 2, EpiStoreF32, false, true>(op, gs, ep, 1, st);
        if (a_mn && !b_mn) return launch_gemm<kBN, 2, EpiStoreF32, true, false>(op, gs, ep, 1, st);
        return launch_gemm<kBN, 2, EpiStoreF32, true, true>(op, gs, ep, 1, st);
    }
    EpiStoreF32Direct::Params ep{}; ep.C[0] = ep.C[1] = C; ep.ldc[0] = ep.ldc[1] = ldc; ep.alpha = alpha;
    if (!a_mn && !b_mn) return launch_gemm<kBN, kStages, EpiStoreF32Direct, false, false>(op, gs, ep, 1, st);
    if (!a_mn && b_mn) return launch_gemm<kBN, kStages, EpiStoreF32Direct, false, true>(op, gs, ep, 1, st);
    if (a_mn && !b_mn) return launch_gemm<kBN, kStages, EpiStoreF32Direct, true, false>(op, gs, ep, 1, st);
    return launch_gemm<kBN, kStages, EpiStoreF32Direct, true, true>(op, gs, ep, 1, st);
}

// ------------------------------------------------------------------------------------ K2
int cvcl_head_proj_norm_fwd(const void* x, int ldx, const void* w, int ldw, const float* bias,
                            int M, int E, int K, int normalize,
                            float* out_f32, int ld_f32, void* out_bf16, int ld_bf16,
                            float* inv_norm, void* stream) {
    CVCL_REQUIRE(x && w, "head_proj_norm_fwd: null operand");
    CVCL_REQUIRE(M > 0 && E > 0 && K > 0, "head_proj_norm_fwd: bad shape M=%d E=%d K=%d", M, E, K);
    const int cluster = ceil_div(E, kBN);
    if (cluster > 8)
        return fail(CVCL_ERR_UNSUPPORTED, "head_proj_norm_fwd: E=%d needs a cluster of %d > 8 CTAs", E, cluster);
    GemmOperands op{}; op.ndir = 1;
    op.A[0] = mat(x, M, K, ldx); op.B[0] = mat(w, E, K, ldw);
    op.out[0] = out_bf16 ? mat(out_bf16, M, E, ld_bf16) : mat(x, M, K, ldx);
    GemmShape gs{}; gs.M[0] = gs.M[1] = M; gs.N[0] = gs.N[1] = E; gs.K = K; gs.m_stride = kBM; gs.n_stride = kBN;
    {
        // small M (e.g. 512 pairs): 16 tiles cannot fill 148 SMs and each would stream all of K
        // serially.  Split the contraction 8-ways over blockIdx.z (fp32 vector atomics into the fp32
        // output buffer), then one warp-per-row pass adds the bias and normalises.
        const int tiles = ceil_div(M, kBM) * ceil_div(E, kBN);
        const int chunks = ceil_div(K, kBK);
        if (out_f32 && tiles * 4 <= sm_count() && chunks >= 16 && ld_f32 % 4 == 0 && E % 4 == 0 &&
            (reinterpret_cast<uintptr_t>(out_f32) & 15) == 0 && !head_splitk_disabled()) {
            int splits = sm_count() / tiles;
            if (splits > chunks / 4) splits = chunks / 4;
            while (splits > 1 && ceil_div(chunks, splits) * (splits - 1) >= chunks) --splits;
            if (splits > 1) {
                if (!head_scratch_zeroed())
                    CVCL_CHECK_CUDA(cudaMemsetAsync(out_f32, 0, sizeof(float) * static_cast<size_t>(M) * ld_f32, as_stream(stream)));
                gs.k_splits = splits;
                EpiAtomicAddF32::Params ea{}; ea.C = out_f32; ea.ldc = ld_f32; ea.alpha = 1.f;
                int rc = launch_gemm<kBN, 4, EpiAtomicAddF32, false, false>(op, gs, ea, 1, as_stream(stream));
                if (rc) return rc;
                CVCL_CHECK_CUDA(launch_pdl(bias_norm_rows_kernel, dim3(warps_grid(M, 128)), dim3(128), 0, as_stream(stream),
                                           out_f32, ld_f32, bias, M, E, normalize, static_cast<__nv_bfloat16*>(out_bf16),
                                           ld_bf16, inv_norm));
                count_launch();
                return CVCL_OK;
            }
        }
    }
    EpiHeadNorm::Params ep{};
    ep.bias = bias; ep.normalize = normalize; ep.out_f32 = out_f32; ep.ld_f32 = ld_f32;
    ep.store_bf16 = out_bf16 != nullptr; ep.inv_norm = inv_norm;
    // small M: few CTAs, a 6-deep ring keeps 192 KB in flight per SM (latency-bound mainloop);
    // large M (spatial head, M = B*49): 3-deep ring so two CTAs share an SM and one's cluster
    // epilogue overlaps the other's MMAs
    if (ceil_div(M, kBM) * cluster > 2 * sm_count())
        return launch_gemm<kBN, 3, EpiHeadNorm, false, false>(op, gs, ep, cluster, as_stream(stream));
    return launch_gemm<kBN, 6, EpiHeadNorm, false, false>(op, gs, ep, cluster, as_stream(stream));
}

// ------------------------------------------------------------------------------------ K3+K4
size_t cvcl_sim_workspace_bytes(int M0, int N0, int M1, int N1) {
    return carve_sim_ws(nullptr, M0, N0, M1, N1).bytes;
}

static int sim_infonce_fwd_impl(const void* img_q, const void* txt_k, const void* txt_q, const void* img_k,
                               int ld, int M0, int N0, int M1, int N1, int E, float log_scale,
                               int diag_off, float inv_rows, void* workspace,
                               float* lse0, float* lse1, int* argmax0, int* argmax1, float* out5,
                               void* stream, bool tickets_zeroed, bool unit_norm = false) {
    CVCL_REQUIRE(img_q && txt_k && txt_q && img_k && workspace && lse0 && lse1 && out5,
                 "sim_infonce_fwd: null pointer");
    CVCL_REQUIRE(M0 > 0 && N0 > 0 && M1 > 0 && N1 > 0 && E > 0, "sim_infonce_fwd: bad shape");
    CVCL_REQUIRE(diag_off >= 0 && M0 + diag_off <= N0 && M1 + diag_off <= N1,
                 "sim_infonce_fwd: positives out of range (M0=%d N0=%d M1=%d N1=%d diag_off=%d)", M0, N0, M1, N1, diag_off);
    SimWs w = carve_sim_ws(workspace, M0, N0, M1, N1);
    GemmOperands op{}; op.ndir = 2;
    op.A[0] = mat(img_q, M0, E, ld); op.B[0] = mat(txt_k, N0, E, ld);
    op.A[1] = mat(txt_q, M1, E, ld); op.B[1] = mat(img_k, N1, E, ld);
    GemmShape gs{}; gs.M[0] = M0; gs.N[0] = N0; gs.M[1] = M1; gs.N[1] = N1; gs.K = E;
    gs.m_stride = kBM; gs.n_stride = kBN;
    EpiSimStats::Params ep{};
    ep.scale = expf(log_scale);
    for (int z = 0; z < 2; ++z) {
        ep.diag_off[z] = diag_off; ep.part[z] = w.part[z]; ep.m_pad[z] = w.m_pad[z]; ep.diag[z] = w.diag[z];
    }
    ep.ticket = w.ticket;
    // small problems: merge inside the similarity kernel (saves a launch on the critical path)
    const bool fuse = sim_bn(N0, N1) == 128 && w.tiles_m[0] + w.tiles_m[1] <= 256;
    ep.fuse_merge = fuse;
    for (int z = 0; z < 2; ++z) { ep.n_tiles[z] = w.n_tiles[z]; ep.tiles_m[z] = w.tiles_m[z]; }
    ep.rb_ticket = w.rb_ticket; ep.rb_part = w.rb_part;
    ep.lse[0] = lse0; ep.lse[1] = lse1; ep.argmax[0] = argmax0; ep.argmax[1] = argmax1;
    ep.inv_rows = inv_rows; ep.out5 = out5;
    if (fuse && !tickets_zeroed)
        CVCL_CHECK_CUDA(cudaMemsetAsync(w.rb_ticket, 0, sizeof(unsigned int) * (1 + w.tiles_m[0] + w.tiles_m[1]), as_stream(stream)));
    // two CTAs fit per SM (96 KB ring, <= 256 TMEM columns each) so one tile's softmax epilogue
    // overlaps another tile's MMAs; wide tiles (fewer per-CTA fixed costs, less smem traffic per
    // flop) once the problem is large enough to fill the machine anyway
    int rc;
    // one similarity pass for both directions (EpiSimStats1P): single device (queries = keys), square, full tiles,
    // unit-norm features (the caller's promise) and a scale that keeps exp(scale*(r-1)) in the normal fp32 range
    const bool one_pass = unit_norm && sim_bn(N0, N1) == 256 && img_q == img_k && txt_q == txt_k && M0 == N1 &&
                          M1 == N0 && M0 == N0 && diag_off == 0 && M0 % 256 == 0 && ep.scale <= 32.f &&
                          getenv("CVCL_B200_SIM_TWO_PASS") == nullptr;
    if (one_pass) {
        EpiSimStats1P::Params e1{};
        e1.scale = ep.scale;
        for (int z = 0; z < 2; ++z) { e1.part[z] = w.part[z]; e1.m_pad[z] = w.m_pad[z]; e1.diag[z] = w.diag[z]; }
        e1.ticket = w.ticket;
        op.ndir = 1;
        gs.n_stride = 256;
        rc = launch_gemm_persistent<256, 3, EpiSimStats1P>(op, gs, e1, as_stream(stream));   // 3-deep ring: room for the transpose buffers
    } else if (sim_bn(N0, N1) == 256) {       // large: persistent CTAs, double-buffered TMEM accumulator
        gs.n_stride = 256;
        rc = launch_gemm_persistent<256, 4, EpiSimStats>(op, gs, ep, as_stream(stream));
    } else {
        rc = launch_gemm<kBN, 3, EpiSimStats, false, false>(op, gs, ep, 1, as_stream(stream));
    }
    if (rc || fuse) return rc;
    FinalizeParams fp{};
    for (int z = 0; z < 2; ++z) {
        fp.part[z] = w.part[z]; fp.m_pad[z] = w.m_pad[z]; fp.n_tiles[z] = w.n_tiles[z];
        fp.diag[z] = w.diag[z]; fp.diag_off[z] = diag_off;
    }
    fp.M[0] = M0; fp.M[1] = M1; fp.lse[0] = lse0; fp.lse[1] = lse1;
    fp.argmax[0] = argmax0; fp.argmax[1] = argmax1; fp.inv_rows = inv_rows;
    fp.block_part = w.block_part; fp.ticket = w.ticket; fp.out = out5;
    CVCL_CHECK_CUDA(launch_pdl(infonce_finalize_kernel, dim3(ceil_div(M0 + M1, 256)), dim3(256), 0, as_stream(stream), fp));
    count_launch();
    return CVCL_OK;
}

int cvcl_sim_infonce_fwd(const void* img_q, const void* txt_k, const void* txt_q, const void* img_k,
                         int ld, int M0, int N0, int M1, int N1, int E, float log_scale,
                         int diag_off, float inv_rows, void* workspace,
                         float* lse0, float* lse1, int* argmax0, int* argmax1, float* out5,
                         int unit_norm, void* stream) {
    return sim_infonce_fwd_impl(img_q, txt_k, txt_q, img_k, ld, M0, N0, M1, N1, E, log_scale, diag_off, inv_rows,
                                workspace, lse0, lse1, argmax0, argmax1, out5, stream, false, unit_norm != 0);
}

int cvcl_sim_logits_fwd(const void* img, const void* txt, int ld, int Ni, int Nt, int E, float log_scale,
                        float* lpi, float* lpt, void* stream) {
    CVCL_REQUIRE(img && txt && (lpi || lpt), "sim_logits_fwd: null pointer");
    CVCL_REQUIRE(Ni > 0 && Nt > 0 && E > 0, "sim_logits_fwd: bad shape Ni=%d Nt=%d E=%d", Ni, Nt, E);
    const float alpha = expf(log_scale);
    int rc = 0;
    if (lpi) rc = cvcl_gemm_f32out(img, ld, 0, txt, ld, 0, Ni, Nt, E, alpha, lpi, Nt, stream);
    if (!rc && lpt) rc = cvcl_gemm_f32out(txt, ld, 0, img, ld, 0, Nt, Ni, E, alpha, lpt, Ni, stream);
    return rc;
}

// ------------------------------------------------------------------------------------ K5
int cvcl_sim_infonce_bwd_g(const void* img_q, const void* txt_k, const void* txt_q, const void* img_k,
                           int ld, int M0, int N0, int M1, int N1, int E, float log_scale, int diag_off,
                           float coef, const float* lse_q0, const float* lse_k0, const float* lse_q1,
                           const float* lse_k1, void* Gs0, int ldg0, void* Gs1, int ldg1, float* gdiag0,
                           float* gdiag1, float* dscale, void* stream) {
    CVCL_REQUIRE(img_q && txt_k && lse_q0 && lse_k0 && Gs0 && gdiag0, "sim_infonce_bwd_g: null pointer");
    CVCL_REQUIRE(!Gs1 || (txt_q && img_k && lse_q1 && lse_k1 && gdiag1), "sim_infonce_bwd_g: direction 1 needs its operands");
    CVCL_REQUIRE(diag_off >= 0 && M0 + diag_off <= N0 && (!Gs1 || M1 + diag_off <= N1),
                 "sim_infonce_bwd_g: positives out of range (M0=%d N0=%d M1=%d N1=%d diag_off=%d)", M0, N0, M1, N1, diag_off);
    CVCL_REQUIRE(M0 > 0 && N0 > 0 && E > 0, "sim_infonce_bwd_g: bad shape");
    GemmOperands op{}; op.ndir = Gs1 ? 2 : 1;
    op.A[0] = mat(img_q, M0, E, ld); op.B[0] = mat(txt_k, N0, E, ld); op.out[0] = mat(Gs0, M0, N0, ldg0);
    GemmShape gs{}; gs.M[0] = gs.M[1] = M0; gs.N[0] = gs.N[1] = N0; gs.K = E; gs.m_stride = kBM; gs.n_stride = kBN;
    EpiGradG::Params ep{};
    ep.scale = expf(log_scale); ep.coef = coef; ep.diag_off[0] = ep.diag_off[1] = diag_off;
    ep.lse_q[0] = ep.lse_q[1] = lse_q0; ep.lse_k[0] = ep.lse_k[1] = lse_k0; ep.gdiag[0] = ep.gdiag[1] = gdiag0;
    if (Gs1) {
        op.A[1] = mat(txt_q, M1, E, ld); op.B[1] = mat(img_k, N1, E, ld); op.out[1] = mat(Gs1, M1, N1, ldg1);
        gs.M[1] = M1; gs.N[1] = N1; ep.lse_q[1] = lse_q1; ep.lse_k[1] = lse_k1; ep.gdiag[1] = gdiag1;
    }
    ep.dscale_accum = dscale;
    if (sim_bn(N0, Gs1 ? N1 : N0) == 256) {
        gs.n_stride = 256;
        return launch_gemm_persistent<256, 3, EpiGradG>(op, gs, ep, as_stream(stream));
    }
    return launch_gemm<kBN, 2, EpiGradG, false, false>(op, gs, ep, 1, as_stream(stream));
}

int cvcl_feat_grad_norm_bwd(const void* Gs, int ldg, int gs_transposed, const void* other, int ld_other,
                            int M, int E, int Kc, const void* feat_bf16, int ld_feat, const float* inv_norm,
                            int normalize, const int64_t* row_len, const void* diag_feat, int ld_diag,
                            int diag_rows, int diag_off, const float* diag_coef, float* out_f32, int ld_f32,
                            void* out_bf16, int ld_bf16, float* dbias, void* stream) {
    return cvcl_feat_grad_norm_bwd_ws(Gs, ldg, gs_transposed, other, ld_other, M, E, Kc, feat_bf16, ld_feat, inv_norm,
                                      normalize, row_len, diag_feat, ld_diag, diag_rows, diag_off, diag_coef, out_f32,
                                      ld_f32, out_bf16, ld_bf16, dbias, nullptr, stream);
}

int cvcl_feat_grad_norm_bwd_ws(const void* Gs, int ldg, int gs_transposed, const void* other, int ld_other,
                               int M, int E, int Kc, const void* feat_bf16, int ld_feat, const float* inv_norm,
                               int normalize, const int64_t* row_len, const void* diag_feat, int ld_diag,
                               int diag_rows, int diag_off, const float* diag_coef, float* out_f32, int ld_f32,
                               void* out_bf16, int ld_bf16, float* dbias, float* acc_scratch, void* stream) {
    CVCL_REQUIRE(Gs && other, "feat_grad_norm_bwd: null operand");
    CVCL_REQUIRE(!diag_feat || diag_coef, "feat_grad_norm_bwd: diag_feat needs its per-row diag_coef");
    {
        // Long contraction (sharded global batch: Kc = world * b) on few output tiles: every CTA of the
        // single-kernel path would stream all of Kc serially (0.3 us per 64-wide chunk).  Split the
        // contraction over blockIdx.z into an fp32 accumulator (vector atomics), then one warp-per-row
        // pass applies the diagonal term, the normalise backward, 1/len and the bias column sums.
        float* acc = acc_scratch ? acc_scratch : out_f32;
        const int ld_acc = acc_scratch ? E : ld_f32;
        const int tiles = ceil_div(M, kBM) * ceil_div(E, kBN);
        const int chunks = ceil_div(Kc, kBK);
        if (acc && chunks >= 24 && tiles * 2 <= sm_count() && E % 4 == 0 && ld_acc % 4 == 0 && E <= 128 * kMaxVec &&
            (reinterpret_cast<uintptr_t>(acc) & 15) == 0 && (ld_feat % 4 == 0) && (ld_diag % 4 == 0 || !diag_feat) &&
            (out_f32 != nullptr) != (out_bf16 != nullptr) && (!normalize || (feat_bf16 && inv_norm))) {
            int splits = sm_count() / tiles;
            if (splits > chunks / 6) splits = chunks / 6;
            while (splits > 1 && ceil_div(chunks, splits) * (splits - 1) >= chunks) --splits;
            if (splits > 1) {
                cudaStream_t st = as_stream(stream);
                CVCL_CHECK_CUDA(cudaMemsetAsync(acc, 0, sizeof(float) * static_cast<size_t>(M) * ld_acc, st));
                GemmOperands op{}; op.ndir = 1;
                op.A[0] = gs_transposed ? mat(Gs, Kc, M, ldg) : mat(Gs, M, Kc, ldg);
                op.B[0] = mat(other, Kc, E, ld_other);
                GemmShape gs{}; gs.M[0] = gs.M[1] = M; gs.N[0] = gs.N[1] = E; gs.K = Kc; gs.m_stride = kBM; gs.n_stride = kBN;
                gs.k_splits = splits;
                EpiAtomicAddF32::Params ea{}; ea.C = acc; ea.ldc = ld_acc; ea.alpha = 1.f;
                int rc = gs_transposed ? launch_gemm<kBN, 3, EpiAtomicAddF32, true, true>(op, gs, ea, 1, st)
                                       : launch_gemm<kBN, 3, EpiAtomicAddF32, false, true>(op, gs, ea, 1, st);
                if (rc) return rc;
                CVCL_CHECK_CUDA(launch_pdl(featgrad_finish_kernel, dim3(warps_grid(M)), dim3(256), 0, st, acc, ld_acc,
                                           static_cast<const __nv_bfloat16*>(feat_bf16), ld_feat,
                                           static_cast<const __nv_bfloat16*>(diag_feat), ld_diag, diag_rows, diag_off,
                                           diag_coef, inv_norm, normalize, reinterpret_cast<const long long*>(row_len), M, E,
                                           out_f32, ld_f32, static_cast<__nv_bfloat16*>(out_bf16), ld_bf16, dbias));
                count_launch();
                return CVCL_OK;
            }
        }
    }
    CVCL_REQUIRE((out_f32 != nullptr) != (out_bf16 != nullptr), "feat_grad_norm_bwd: exactly one of out_f32 / out_bf16");
    CVCL_REQUIRE(!normalize || (feat_bf16 && inv_norm), "feat_grad_norm_bwd: normalize needs feat and inv_norm");
    CVCL_REQUIRE(feat_bf16 || diag_feat, "feat_grad_norm_bwd: needs feat or diag_feat (use cvcl_gemm_f32out otherwise)");
    CVCL_REQUIRE(M > 0 && E > 0 && Kc > 0, "feat_grad_norm_bwd: bad shape");
    const int cluster = ceil_div(E, kBN);
    if (cluster > 8)
        return fail(CVCL_ERR_UNSUPPORTED, "feat_grad_norm_bwd: E=%d needs a cluster of %d > 8 CTAs", E, cluster);
    GemmOperands op{}; op.ndir = 1;
    op.A[0] = gs_transposed ? mat(Gs, Kc, M, ldg) : mat(Gs, M, Kc, ldg);
    op.B[0] = mat(other, Kc, E, ld_other);                         // MN-major: features as stored
    const Mat fm = feat_bf16 ? mat(feat_bf16, M, E, ld_feat) : mat(diag_feat, diag_rows, E, ld_diag);
    const Mat dm = diag_feat ? mat(diag_feat, diag_rows, E, ld_diag) : fm;
    op.aux[0] = fm; op.aux[1] = dm;
    op.out[0] = out_f32 ? mat(out_f32, M, E, ld_f32) : mat(out_bf16, M, E, ld_bf16);
    GemmShape gs{}; gs.M[0] = gs.M[1] = M; gs.N[0] = gs.N[1] = E; gs.K = Kc; gs.m_stride = kBM; gs.n_stride = kBN;
    gs.aux_row_off[0] = 0; gs.aux_row_off[1] = diag_feat ? diag_off : 0;
    cudaStream_t st = as_stream(stream);
    constexpr int kSt = 3;                                         // 2 aux tiles share the smem budget
    if (out_f32) {
        EpiNormBwdT<true>::Params ep{};
        ep.inv_norm = inv_norm; ep.normalize = normalize; ep.row_len = reinterpret_cast<const long long*>(row_len);
        ep.use_diag = diag_feat != nullptr; ep.diag_coef = diag_coef; ep.dbias = dbias;
        return gs_transposed ? launch_gemm<kBN, kSt, EpiNormBwdT<true>, true, true>(op, gs, ep, cluster, st)
                             : launch_gemm<kBN, kSt, EpiNormBwdT<true>, false, true>(op, gs, ep, cluster, st);
    }
    EpiNormBwdT<false>::Params ep{};
    ep.inv_norm = inv_norm; ep.normalize = normalize; ep.row_len = reinterpret_cast<const long long*>(row_len);
    ep.use_diag = diag_feat != nullptr; ep.diag_coef = diag_coef; ep.dbias = dbias;
    return gs_transposed ? launch_gemm<kBN, kSt, EpiNormBwdT<false>, true, true>(op, gs, ep, cluster, st)
                         : launch_gemm<kBN, kSt, EpiNormBwdT<false>, false, true>(op, gs, ep, cluster, st);
}

int cvcl_head_weight_grad(const void* du, int ld_du, const void* x, int ld_x, int E, int K, int M,
                          float* dW, int ld_dw, void* stream) {
    CVCL_REQUIRE(du && x && dW, "head_weight_grad: null pointer");
    CVCL_REQUIRE(E > 0 && K > 0 && M > 0, "head_weight_grad: bad shape");
    // dW[e,k] = sum_m du[m,e] * x[m,k]: both operands MN-major (the contraction index m strides)
    const int tiles = ceil_div(E, kBM) * ceil_div(K, kBN);
    const int chunks = ceil_div(M, kBK);
    if (tiles < sm_count() && chunks >= 64 && (ld_dw & 3) == 0 && (reinterpret_cast<uintptr_t>(dW) & 15) == 0) {
        // long contraction, few output tiles (spatial head: M = B*49): split the contraction over
        // blockIdx.z so every SM has work; partial tiles are added with fp32 vector atomics
        int splits = ceil_div(2 * sm_count(), tiles);
        if (splits > chunks / 8) splits = chunks / 8;
        // every split must own at least one chunk: ceil(chunks / splits) * (splits - 1) < chunks
        while (splits > 1 && ceil_div(chunks, splits) * (splits - 1) >= chunks) --splits;
        if (splits > 1) {
            CVCL_CHECK_CUDA(cudaMemsetAsync(dW, 0, sizeof(float) * static_cast<size_t>(E) * ld_dw, as_stream(stream)));
            GemmOperands op{}; op.ndir = 1;
            op.A[0] = mat(du, M, E, ld_du); op.B[0] = mat(x, M, K, ld_x);
            GemmShape gs{}; gs.M[0] = gs.M[1] = E; gs.N[0] = gs.N[1] = K; gs.K = M; gs.m_stride = kBM; gs.n_stride = kBN;
            gs.k_splits = splits;
            EpiAtomicAddF32::Params ep{}; ep.C = dW; ep.ldc = ld_dw; ep.alpha = 1.f;
            return launch_gemm<kBN, 3, EpiAtomicAddF32, true, true>(op, gs, ep, 1, as_stream(stream));
        }
    }
    return cvcl_gemm_f32out(du, ld_du, 1, x, ld_x, 1, E, K, M, 1.f, dW, ld_dw, stream);
}

// ------------------------------------------------------------------------------------ fused flat step
namespace {
// Independent kernels of the step run on a second stream (fork/join with events) so that under
// stream capture they become parallel branches of the CUDA graph: K1 || (cast W -> K2),
// dI || dT, dW || embedding scatter.  One side stream + 4 events per host thread, created lazily.
struct SideStream {
    cudaStream_t s = nullptr;
    cudaStream_t s2 = nullptr;        // gradient-buffer memset branch (4.8 MB, needed only by the backward)
    cudaEvent_t fork[3] = {nullptr, nullptr, nullptr}, join[3] = {nullptr, nullptr, nullptr};
    bool ok = false;
    int init() {
        if (ok) return CVCL_OK;
        CVCL_CHECK_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        CVCL_CHECK_CUDA(cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking));
        for (int i = 0; i < 3; ++i) {
            CVCL_CHECK_CUDA(cudaEventCreateWithFlags(&fork[i], cudaEventDisableTiming));
            CVCL_CHECK_CUDA(cudaEventCreateWithFlags(&join[i], cudaEventDisableTiming));
        }
        ok = true;
        return CVCL_OK;
    }
};
// one set per (host thread, device): streams and events belong to the device that was current when they were created
SideStream& side_stream() {
    static thread_local SideStream per_dev[16];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) dev = 0;
    return per_dev[dev];
}

struct FlatWs {
    __nv_bfloat16 *w16, *x16, *img16, *txt16, *G0, *du16;
    float *invn_i, *invn_t, *lse0, *lse1, *gdiag, *dm, *u32;
    void* sim; int ldB; size_t bytes;
};
FlatWs carve_flat_ws(void* ws, int B, int L, int E, int K, int V) {
    (void)L; (void)V;
    FlatWs f{};
    unsigned char* base = static_cast<unsigned char*>(ws);
    size_t off = 0;
    f.ldB = pad8(B);
    auto take = [&](size_t bytes) { void* p = base + off; off += align_up(bytes, 256); return p; };
    f.w16 = static_cast<__nv_bfloat16*>(take(2ull * E * K));
    f.x16 = static_cast<__nv_bfloat16*>(take(2ull * B * K));
    f.img16 = static_cast<__nv_bfloat16*>(take(2ull * B * E));
    f.txt16 = static_cast<__nv_bfloat16*>(take(2ull * B * E));
    f.G0 = static_cast<__nv_bfloat16*>(take(2ull * B * f.ldB));
    f.du16 = static_cast<__nv_bfloat16*>(take(2ull * B * E));
    f.invn_i = static_cast<float*>(take(4ull * B));
    f.invn_t = static_cast<float*>(take(4ull * B));
    f.lse0 = static_cast<float*>(take(4ull * B));
    f.lse1 = static_cast<float*>(take(4ull * B));
    f.gdiag = static_cast<float*>(take(4ull * B));
    f.dm = static_cast<float*>(take(4ull * B * E));
    f.u32 = static_cast<float*>(take(4ull * B * E));
    f.sim = base + off;
    off += align_up(cvcl_sim_workspace_bytes(B, B, B, B), 256);
    f.bytes = off;
    return f;
}
}  // namespace

size_t cvcl_flat_step_workspace_bytes(int B, int L, int E, int K, int V) {
    return carve_flat_ws(nullptr, B, L, E, K, V).bytes;
}

int cvcl_flat_step_layout(int B, int L, int E, int K, int V, long long* out, int n) {
    CVCL_REQUIRE(out && B > 0, "flat_step_layout: need out and B > 0");
    const FlatWs f = carve_flat_ws(nullptr, B, L, E, K, V);
    auto off = [](const void* p) { return static_cast<long long>(reinterpret_cast<uintptr_t>(p)); };
    const long long v[] = {off(f.img16), off(f.txt16), off(f.invn_i), off(f.invn_t), off(f.lse0), off(f.lse1),
                           off(f.G0), off(f.du16), off(f.dm), off(f.gdiag), f.ldB, static_cast<long long>(f.bytes)};
    for (int i = 0; i < n && i < (int)(sizeof(v) / sizeof(v[0])); ++i) out[i] = v[i];
    return CVCL_OK;
}

int cvcl_flat_contrastive_step(const void* x, int x_is_bf16, const int64_t* ids, const int64_t* lens,
                               const float* w, const float* bias, const float* table,
                               int B, int L, int E, int K, int V, int normalize, float log_scale,
                               int need_grads, void* workspace,
                               float* out5, float* img_feat_f32, float* txt_feat_f32,
                               float* dW, float* dbias, float* dtable, float* dscale,
                               int* status, void* stream) {
    CVCL_REQUIRE(x && ids && lens && w && table && workspace && out5, "flat_contrastive_step: null pointer");
    CVCL_REQUIRE(!need_grads || (dW && dbias && dtable && dscale), "flat_contrastive_step: null gradient output");
    CVCL_REQUIRE(B > 0 && E % 8 == 0 && K % 8 == 0, "flat_contrastive_step: need B>0, E%%8==0, K%%8==0 (B=%d E=%d K=%d)", B, E, K);
    cudaStream_t st = as_stream(stream);
    FlatWs f = carve_flat_ws(workspace, B, L, E, K, V);
    SideStream& ss = side_stream();
    int rc;
    if ((rc = ss.init())) return rc;
    void* side = ss.s;
    // measurement hook (tools/step_phases.py): stop after phase k of {1 encoders, 2 similarity + InfoNCE,
    // 3 Gs, 4 dI and dT}; 11 / 12 run only the head chain / only the text encoder of phase 1
    int limit = 0;
    if (const char* e = getenv("CVCL_B200_STEP_PHASES")) limit = atoi(e);
    // ---- forward: [memsets -> text encoder] (side) || [cast W -> head GEMM] (main)
    CVCL_CHECK_CUDA(cudaEventRecord(ss.fork[0], st));
    CVCL_CHECK_CUDA(cudaStreamWaitEvent(ss.s, ss.fork[0], 0));
    // all accumulators are zeroed off the critical path, first thing on the side stream
    float* img_f32 = img_feat_f32 ? img_feat_f32 : f.u32;      // also the split-K accumulator of the head
    CVCL_CHECK_CUDA(cudaMemsetAsync(img_f32, 0, sizeof(float) * static_cast<size_t>(B) * E, ss.s));
    {   // row-block tickets of the fused merge
        SimWs sw = carve_sim_ws(f.sim, B, B, B, B);
        CVCL_CHECK_CUDA(cudaMemsetAsync(sw.rb_ticket, 0, sizeof(unsigned int) * (1 + sw.tiles_m[0] + sw.tiles_m[1]), ss.s));
    }
    CVCL_CHECK_CUDA(cudaEventRecord(ss.fork[2], ss.s));          // head GEMM (split-K atomics) waits for this only
    if (need_grads) {          // third branch: nothing before the backward reads these
        CVCL_CHECK_CUDA(cudaStreamWaitEvent(ss.s2, ss.fork[0], 0));
        if (dbias == dscale + 4 && dtable == dbias + E) {
            CVCL_CHECK_CUDA(cudaMemsetAsync(dscale, 0, sizeof(float) * (4 + E + static_cast<size_t>(V) * E), ss.s2));
        } else {
            CVCL_CHECK_CUDA(cudaMemsetAsync(dscale, 0, sizeof(float), ss.s2));
            CVCL_CHECK_CUDA(cudaMemsetAsync(dbias, 0, sizeof(float) * E, ss.s2));
            CVCL_CHECK_CUDA(cudaMemsetAsync(dtable, 0, sizeof(float) * static_cast<size_t>(V) * E, ss.s2));
        }
        CVCL_CHECK_CUDA(cudaEventRecord(ss.join[2], ss.s2));
    }
    if (limit != 11 && (rc = cvcl_text_encoder_fwd(ids, lens, table, B, L, E, V, normalize, 0, 1.f, txt_feat_f32, f.txt16, E,
                                                   f.invn_t, nullptr, nullptr, status, side))) return rc;
    CVCL_CHECK_CUDA(cudaEventRecord(ss.join[0], ss.s));
    if (limit == 12) {
        CVCL_CHECK_CUDA(cudaStreamWaitEvent(st, ss.join[0], 0));
        if (need_grads) CVCL_CHECK_CUDA(cudaStreamWaitEvent(st, ss.join[2], 0));
        return CVCL_OK;
    }
    if ((rc = cvcl_cast_transpose(w, 0, f.w16, nullptr, 1, E, K, K, K, 0, 0, 0, 0, stream))) return rc;
    const void* x16 = x;
    if (!x_is_bf16 || (reinterpret_cast<uintptr_t>(x) & 15)) {
        if ((rc = cvcl_cast_transpose(x, x_is_bf16, f.x16, nullptr, 1, B, K, K, K, 0, 0, 0, 0, stream))) return rc;
        x16 = f.x16;
    }
    CVCL_CHECK_CUDA(cudaStreamWaitEvent(st, ss.fork[2], 0));
    head_scratch_zeroed() = true;
    rc = cvcl_head_proj_norm_fwd(x16, K, f.w16, K, bias, B, E, K, normalize, img_f32, E, f.img16, E, f.invn_i, stream);
    head_scratch_zeroed() = false;
    if (rc) return rc;
    CVCL_CHECK_CUDA(cudaStreamWaitEvent(st, ss.join[0], 0));
    if (limit == 1 || limit == 11) {
        if (need_grads) CVCL_CHECK_CUDA(cudaStreamWaitEvent(st, ss.join[2], 0));
        return CVCL_OK;
    }
    // ---- K3 + K4
    if ((rc = sim_infonce_fwd_impl(f.img16, f.txt16, f.txt16, f.img16, E, B, B, B, B, E, log_scale, 0,
                                   1.f / static_cast<float>(B), f.sim, f.lse0, f.lse1, nullptr, nullptr, out5, stream,
                                   true))) return rc;
    if (!need_grads) return CVCL_OK;
    // ---- K5: Gs (one orientation) -> dI (K-major Gs, main) || dT (the same Gs read MN-major, side)
    CVCL_CHECK_CUDA(cudaStreamWaitEvent(st, ss.join[2], 0));     // gradient accumulators are zero (ds is the first user)
    if (limit == 2) return CVCL_OK;
    const float coef = 0.5f / static_cast<float>(B);
    if ((rc = cvcl_sim_infonce_bwd_g(f.img16, f.txt16, nullptr, nullptr, E, B, B, 0, 0, E, log_scale, 0, coef,
                                     f.lse0, f.lse1, nullptr, nullptr, f.G0, f.ldB, nullptr, 0, f.gdiag, nullptr, dscale,
                                     stream))) return rc;
    if (limit == 3) return CVCL_OK;
    CVCL_CHECK_CUDA(cudaEventRecord(ss.fork[1], st));
    CVCL_CHECK_CUDA(cudaStreamWaitEvent(ss.s, ss.fork[1], 0));
    if ((rc = cvcl_feat_grad_norm_bwd(f.G0, f.ldB, 1, f.img16, E, B, E, B, f.txt16, E, f.invn_t, normalize,
                                      lens, f.img16, E, B, 0, f.gdiag, f.dm, E, nullptr, 0, nullptr, side))) return rc;
    // ... then the embedding scatter follows dT on the side stream while dI -> dW run on the main one
    if (limit != 4 && (rc = cvcl_embedding_scatter_add(ids, f.dm, dtable, B, L, E, V, 0, side))) return rc;
    CVCL_CHECK_CUDA(cudaEventRecord(ss.join[1], ss.s));
    if ((rc = cvcl_feat_grad_norm_bwd(f.G0, f.ldB, 0, f.txt16, E, B, E, B, f.img16, E, f.invn_i, normalize,
                                      nullptr, f.txt16, E, B, 0, f.gdiag, nullptr, 0, f.du16, E, dbias, stream))) return rc;
    if (limit != 4 && (rc = cvcl_head_weight_grad(f.du16, E, x16, K, E, K, B, dW, K, stream))) return rc;
    CVCL_CHECK_CUDA(cudaStreamWaitEvent(st, ss.join[1], 0));
    return CVCL_OK;
}

// ------------------------------------------------------------------------------------ fused flat step, one kernel
namespace {
struct FusedPlan {
    int Bp, nMB, nEB, nCB, KS, kc_per_split, num_kc, T, nPart, QS, Vp, dw_bn, grid;
    size_t off_ctrl, off_hpart, off_img16, off_txt16, off_invn, off_part, off_diag, off_lse, off_rbpart, off_dspart,
           off_dqpart, off_du16, off_dbpart, off_dm16, off_cmat, off_gdiag, bytes;
};
// -> 0 when the persistent kernel covers the shape, else the reason (unsupported, not an error)
const char* plan_fused(FusedPlan* f, int B, int L, int E, int K, int V, int world = 1) {
    const int G = sm_count();
    if (B < 1) return "B < 1";
    if (L < 1) return "L < 1";
    // the token-count matrix of P1/P5 is bf16, which holds integers exactly only up to 256
    if (L > 256) return "L > 256: a token count above 256 is not exact in the bf16 count matrix";
    if (E % 128 != 0 || E < 128 || E > 512) return "E must be 128, 256, 384 or 512";
    if (K % 64 != 0 || K < 64) return "K must be a multiple of 64";
    if (V < 1) return "V < 1";
    if (world != 1 && world != 2 && world != 4 && world != 8) return "world size must be 1, 2, 4 or 8";
    if (world > 1 && B % 128 != 0) return "sharded: pairs per rank must be a multiple of 128";
    if (world > 1 && K % 128 != 0) return "sharded: K must be a multiple of 128";
    f->grid = G;
    f->Bp = ceil_div(B, 128) * 128;
    f->nMB = f->Bp / 128; f->nEB = E / 128;
    f->nCB = world == 1 ? f->nMB : world * f->nMB;            // column blocks span the GLOBAL batch
    int n_tiles = 2 * f->nMB * f->nCB;
    f->T = 1;
    if (const char* e = getenv("CVCL_B200_FUSED_FORCE_T")) { if (atoi(e) == 2 && f->nCB % 2 == 0) f->T = 2; }   // test hook
    if (n_tiles > G) f->T = 2;                                // two tiles of one row block per CTA (TMEM: 2 x 128 columns)
    if (f->nCB % f->T != 0 || n_tiles / f->T > G) return "batch too large for the similarity phase";
    f->nPart = f->nCB / f->T;
    n_tiles /= f->T;
    f->QS = 1;                                   // CTAs per similarity tile: the largest divisor of E/128 that fits
    for (int d = f->nEB; d >= 1; --d)
        if (f->nEB % d == 0 && n_tiles * d <= G) { f->QS = d; break; }
    if (const char* e = getenv("CVCL_B200_FUSED_FORCE_QS")) {                  // test hook (the 8-rank layout: QS = 1)
        const int d = atoi(e);
        if (d >= 1 && f->nEB % d == 0 && n_tiles * d <= G) f->QS = d;
    }
    const int tiles = f->nMB * f->nEB;
    if (tiles > G) return "batch too large for the head phase";
    f->num_kc = K / 64;
    int ks = G / tiles; if (ks > f->num_kc) ks = f->num_kc;
    f->kc_per_split = ceil_div(f->num_kc, ks);
    f->KS = ceil_div(f->num_kc, f->kc_per_split);
    f->dw_bn = (K % 128 == 0) ? 128 : 64;
    f->Vp = pad8(V);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes, 256); return o; };
    const size_t Bp = f->Bp;
    f->off_ctrl = take(1024);
    f->off_hpart = take(4ull * f->KS * Bp * E);
    f->off_img16 = take(2ull * Bp * E);
    f->off_txt16 = take(2ull * Bp * E);
    f->off_invn = take(4ull * 2 * Bp);
    f->off_part = take(sizeof(RowStat) * 2ull * 2 * f->nCB * Bp);      // two half-tile partials per column block
    f->off_diag = take(4ull * 2 * Bp);
    f->off_lse = take(4ull * 2 * Bp);
    f->off_rbpart = take(4ull * 2 * f->nMB * 6);
    f->off_dspart = take(4ull * f->nMB * f->nPart);
    f->off_dqpart = take(4ull * 2 * f->nPart * Bp * E);
    f->off_du16 = take(2ull * Bp * E);
    f->off_dbpart = take(4ull * G * E);
    f->off_dm16 = take(2ull * Bp * E);
    f->off_cmat = take(2ull * Bp * f->Vp);
    f->off_gdiag = take(4ull * 2 * Bp);
    f->bytes = off;
    return nullptr;
}

// sharding descriptor of the one-kernel step (null = one GPU)
struct FusedShard {
    int world, rank;
    void* const* peer_txt_all;      // [world] rank p's gathered text features  [world*B, E] bf16
    void* const* peer_img_all;      // [world] rank p's gathered image features [world*B, E] bf16
    void* const* peer_part_all;     // [world] rank p's gathered softmax partials [2][2*nCB][world*B] float2
    void* const* peer_flags;        // [world] rank p's flag words (32 x u32, zero before first use)
    unsigned int* epoch;            // local u32, zero before first use
    void* const* peer_stats;        // [world] rank p's block [out5 | ds | db | d table | dW] (nullable: no in-kernel sum)
    void* const* peer_scratch;      // [world] rank p's scatter scratch
    long long reduce_floats;        // floats of the block to sum over the ranks in the kernel (0: none)
};
}  // namespace

int cvcl_flat_fused_supported(int B, int L, int E, int K, int V) {
    FusedPlan f{};
    return plan_fused(&f, B, L, E, K, V) == nullptr ? 1 : 0;
}

size_t cvcl_flat_fused_workspace_bytes(int B, int L, int E, int K, int V) {
    FusedPlan f{};
    return plan_fused(&f, B, L, E, K, V) == nullptr ? f.bytes : 0;
}

int cvcl_flat_fused_layout(int B, int L, int E, int K, int V, long long* out, int n) {
    FusedPlan f{};
    const char* why = plan_fused(&f, B, L, E, K, V);
    if (why) return fail(CVCL_ERR_UNSUPPORTED, "flat_fused_layout: %s", why);
    const long long v[] = {(long long)f.off_ctrl, (long long)f.off_hpart, (long long)f.off_img16, (long long)f.off_txt16,
                           (long long)f.off_invn, (long long)f.off_part, (long long)f.off_diag, (long long)f.off_lse,
                           (long long)f.off_rbpart, (long long)f.off_dspart, (long long)f.off_dqpart, (long long)f.off_du16,
                           (long long)f.off_dbpart, (long long)f.bytes, f.Bp, f.KS, f.nPart, f.dw_bn, f.grid, f.nCB,
                           (long long)f.off_dm16, (long long)f.off_cmat, f.QS, f.Vp, (long long)f.off_gdiag};
    for (int i = 0; i < n && i < (int)(sizeof(v) / sizeof(v[0])); ++i) out[i] = v[i];
    return CVCL_OK;
}

static int flat_step_fused_impl(const void* x16, const void* w16, const int64_t* ids, const int64_t* lens,
                                const float* bias, const float* table, int B, int L, int E, int K, int V,
                                int normalize, float log_scale, const float* log_scale_dev, int need_grads,
                                void* workspace, float* out5, float* img_feat_f32, float* txt_feat_f32,
                                float* dW, float* dbias, float* dtable, float* dscale, int* status, int phase_limit,
                                const FusedShard* sh, void* stream) {
    CVCL_REQUIRE(x16 && w16 && ids && lens && table && workspace && out5, "flat_step_fused: null pointer");
    CVCL_REQUIRE(!need_grads || (dW && dbias && dtable && dscale), "flat_step_fused: null gradient output");
    CVCL_REQUIRE(L >= 1 && V >= 1, "flat_step_fused: bad shape");
    const int world = sh ? sh->world : 1, rank = sh ? sh->rank : 0;
    CVCL_REQUIRE(rank >= 0 && rank < world, "flat_step_fused: rank %d outside [0,%d)", rank, world);
    FusedPlan f{};
    if (const char* why = plan_fused(&f, B, L, E, K, V, world))
        return fail(CVCL_ERR_UNSUPPORTED, "flat_step_fused: %s (B=%d L=%d E=%d K=%d world=%d)", why, B, L, E, K, world);
    CVCL_REQUIRE(((reinterpret_cast<uintptr_t>(workspace) | reinterpret_cast<uintptr_t>(table) |
                   reinterpret_cast<uintptr_t>(bias)) & 15) == 0, "flat_step_fused: 16-byte alignment required");
    CVCL_REQUIRE(!need_grads || ((reinterpret_cast<uintptr_t>(dtable) | reinterpret_cast<uintptr_t>(dW)) & 15) == 0,
                 "flat_step_fused: gradient outputs must be 16-byte aligned");
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    fused::StepParams p{};
    p.ids = reinterpret_cast<const long long*>(ids); p.lens = reinterpret_cast<const long long*>(lens);
    p.table = table; p.bias = bias; p.log_scale_dev = log_scale_dev; p.log_scale = log_scale;
    p.B = B; p.L = L; p.E = E; p.K = K; p.V = V; p.normalize = normalize; p.need_grads = need_grads;
    p.Bg = B * world; p.diag_off = rank * B;
    p.world = world; p.rank = rank;
    p.Bp = f.Bp; p.nMB = f.nMB; p.nEB = f.nEB; p.nCB = f.nCB; p.KS = f.KS; p.kc_per_split = f.kc_per_split;
    p.num_kc = f.num_kc; p.T = f.T; p.nPart = f.nPart; p.QS = f.QS; p.Vp = f.Vp; p.dw_bn = f.dw_bn;
    p.phase_limit = phase_limit;
    p.hpart = reinterpret_cast<float*>(ws + f.off_hpart);
    p.ldq = E; p.ldk = E;
    if (sh) {
        // gathered buffers in peer-mapped symmetric memory: kf16[0] = all texts, kf16[1] = all images; the local
        // features are the slice [rank*B, rank*B + B) of this rank's own copies
        for (int r = 0; r < world; ++r) {
            CVCL_REQUIRE(sh->peer_txt_all[r] && sh->peer_img_all[r] && sh->peer_part_all[r] && sh->peer_flags[r],
                         "flat_step_fused: null peer pointer %d", r);
            p.peer_kf[0][r] = static_cast<__nv_bfloat16*>(sh->peer_txt_all[r]);
            p.peer_kf[1][r] = static_cast<__nv_bfloat16*>(sh->peer_img_all[r]);
            p.peer_part[0][r] = static_cast<float2*>(sh->peer_part_all[r]);
            p.peer_part[1][r] = static_cast<float2*>(sh->peer_part_all[r]) + static_cast<size_t>(2) * f.nCB * p.Bg;
            p.peer_flags[r] = static_cast<unsigned int*>(sh->peer_flags[r]);
        }
        p.epoch = sh->epoch;
        {   // CVCL_B200_PEER_TIMEOUT_MS (default 10 minutes, as for the peer collectives)
            const char* e = getenv("CVCL_B200_PEER_TIMEOUT_MS");
            const long long ms = e ? atoll(e) : 600000ll;
            p.xtimeout_ns = static_cast<unsigned long long>(ms > 0 ? ms : 600000ll) * 1000000ull;
        }
        if (sh->reduce_floats > 0 && world > 1) {
            const int n_tiles5 = f.nEB * (K / 128) + ceil_div(V, 128) * f.nEB;
            p.nslot = ceil_div(n_tiles5, world);
            p.reduce = 1;
            CVCL_REQUIRE(sh->peer_stats && sh->peer_scratch, "flat_step_fused: null gradient-sum table");
            CVCL_REQUIRE(sh->reduce_floats % 4 == 0, "flat_step_fused: reduce_floats must be a multiple of 4");
            const long long n_g = 4ll + E + static_cast<long long>(V) * E + static_cast<long long>(E) * K;
            CVCL_REQUIRE(sh->reduce_floats == 8 || (need_grads && sh->reduce_floats == 8 + n_g),
                         "flat_step_fused: reduce_floats must be 8 or 8 + the gradient block (%lld)", 8 + n_g);
            for (int r = 0; r < world; ++r) {
                CVCL_REQUIRE(sh->peer_stats[r] && sh->peer_scratch[r], "flat_step_fused: null gradient-sum pointer %d", r);
                p.peer_stats[r] = static_cast<float*>(sh->peer_stats[r]);
                p.peer_scratch[r] = static_cast<float*>(sh->peer_scratch[r]);
                p.peer_small[r] = p.peer_scratch[r] + static_cast<size_t>(world) * p.nslot * 128 * 128;
            }
            float* blk = p.peer_stats[rank];
            CVCL_REQUIRE(out5 == blk, "flat_step_fused: out5 must be the start of this rank's block");
            CVCL_REQUIRE(!need_grads || (dscale == blk + 8 && dbias == blk + 12 && dtable == blk + 12 + E &&
                                         dW == blk + 12 + E + static_cast<size_t>(V) * E),
                         "flat_step_fused: gradient outputs must lie in this rank's block (layout [out5|ds|db|dtable|dW])");
        }
        p.kf16[0] = p.peer_kf[0][rank]; p.kf16[1] = p.peer_kf[1][rank];
        p.q16[0] = p.peer_kf[1][rank] + static_cast<size_t>(p.diag_off) * E;
        p.q16[1] = p.peer_kf[0][rank] + static_cast<size_t>(p.diag_off) * E;
    } else {
        p.q16[0] = reinterpret_cast<__nv_bfloat16*>(ws + f.off_img16);
        p.q16[1] = reinterpret_cast<__nv_bfloat16*>(ws + f.off_txt16);
        p.kf16[0] = p.q16[1]; p.kf16[1] = p.q16[0];
        p.peer_kf[0][0] = p.q16[1]; p.peer_kf[1][0] = p.q16[0];
        p.epoch = nullptr;
    }
    for (int z = 0; z < 2; ++z) {
        p.invn[z] = reinterpret_cast<float*>(ws + f.off_invn) + z * f.Bp;
        p.part[z] = reinterpret_cast<RowStat*>(ws + f.off_part) + static_cast<size_t>(z) * 2 * f.nCB * f.Bp;
        p.diag[z] = reinterpret_cast<float*>(ws + f.off_diag) + z * f.Bp;
        p.lse[z] = reinterpret_cast<float*>(ws + f.off_lse) + z * f.Bp;
        p.gdiag[z] = reinterpret_cast<float*>(ws + f.off_gdiag) + z * f.Bp;
        p.part_all[z] = (sh && world > 1) ? p.peer_part[z][rank] : nullptr;
    }
    p.rb_part = reinterpret_cast<float*>(ws + f.off_rbpart);
    p.dspart = reinterpret_cast<float*>(ws + f.off_dspart);
    p.dqpart = reinterpret_cast<float*>(ws + f.off_dqpart);
    p.du16 = reinterpret_cast<__nv_bfloat16*>(ws + f.off_du16);
    p.dbpart = reinterpret_cast<float*>(ws + f.off_dbpart);
    p.dm16 = reinterpret_cast<__nv_bfloat16*>(ws + f.off_dm16);
    p.cmat = reinterpret_cast<__nv_bfloat16*>(ws + f.off_cmat);
    p.sync = reinterpret_cast<unsigned int*>(ws + f.off_ctrl);
    p.fault = reinterpret_cast<int*>(ws + f.off_ctrl + 64);
    p.timing = reinterpret_cast<unsigned long long*>(ws + f.off_ctrl + 128);
    p.status = status;
    p.out5 = out5; p.img_f32 = img_feat_f32; p.txt_f32 = txt_feat_f32;
    p.dW = dW; p.dbias = dbias; p.dtable = dtable; p.dscale = dscale;
    p.inv_rows = 1.f / static_cast<float>(p.Bg);

    // the 16 tensor maps depend only on the pointers and the shape: a training loop passes the same ones every
    // step (torch's caching allocator hands back the same blocks), so the last set is kept per host thread
    struct MapKey { const void* x16; const void* w16; void* ws; float* dW; float* dtable; const void* kf0; const void* kf1;
                    const void* scr[8]; int B, E, K, V, need, world, rank, T, reduce; };
    static thread_local MapKey last_key{};
    static thread_local fused::StepMaps maps;
    static thread_local bool maps_valid = false;
    MapKey key{};                                    // zero the padding: the key is compared with memcmp
    key.x16 = x16; key.w16 = w16; key.ws = workspace; key.dW = dW; key.dtable = dtable; key.kf0 = p.kf16[0];
    key.kf1 = p.kf16[1]; key.B = B; key.E = E; key.K = K; key.V = V; key.need = need_grads; key.world = world;
    key.rank = rank; key.T = f.T; key.reduce = p.reduce;
    if (p.reduce) for (int r = 0; r < world; ++r) key.scr[r] = p.peer_scratch[r];
    int rc;
    if (!maps_valid || memcmp(&key, &last_key, sizeof(MapKey)) != 0) {
        maps_valid = false;
        if ((rc = make_tmap(&maps.x_k, x16, 2, B, K, K, 64, 128))) return rc;
        if ((rc = make_tmap(&maps.w_k, w16, 2, E, K, K, 64, 128))) return rc;
        if ((rc = make_tmap(&maps.hp_out, p.hpart, 4, static_cast<uint64_t>(f.KS) * f.Bp, E, E, 32, 128))) return rc;
        for (int z = 0; z < 2; ++z) {
            if ((rc = make_tmap(&maps.q_k[z], p.q16[z], 2, B, E, p.ldq, 64, 128))) return rc;
            if ((rc = make_tmap(&maps.kf_k[z], p.kf16[z], 2, p.Bg, E, p.ldk, 64, 128))) return rc;
            if ((rc = make_tmap(&maps.kf_mn[z], p.kf16[z], 2, p.Bg, E, p.ldk, 64, 64))) return rc;
        }
        if ((rc = make_tmap(&maps.dq_out, p.dqpart, 4, 2ull * f.nPart * f.Bp, E, E, 32, 128))) return rc;
        if ((rc = make_tmap(&maps.du_mn, p.du16, 2, B, E, E, 64, 64))) return rc;
        if ((rc = make_tmap(&maps.x_mn, x16, 2, B, K, K, 64, 64))) return rc;
        if ((rc = make_tmap(&maps.c_mn, p.cmat, 2, B, V, f.Vp, 64, 64))) return rc;
        if ((rc = make_tmap(&maps.dm_mn, p.dm16, 2, B, E, E, 64, 64))) return rc;
        if (need_grads) {
            if ((rc = make_tmap(&maps.dw_out, dW, 4, E, K, K, 32, 128))) return rc;
            if ((rc = make_tmap(&maps.dt_out, dtable, 4, V, E, E, 32, 128))) return rc;
        } else {
            maps.dw_out = maps.hp_out; maps.dt_out = maps.hp_out;
        }
        last_key = key;
        maps_valid = true;
    }

    // the instance follows the entry, not the world size: the sharded entry at world 1 still runs the sharded
    // instance (epoch counter, flag words), so that the two can be compared against each other.  (nvcc lists the
    // instance named last first in `cuobjdump -sass`, where test_host_logic.py looks for the peer-memory barrier.)
    void (*kernel)(const fused::StepMaps, const fused::StepParams) =
        sh == nullptr ? fused::flat_step_kernel<false> : fused::flat_step_kernel<true>;
    static thread_local unsigned attr_mask[2] = {0, 0};   // per device and instance: function attributes live in the
    int attr_dev = 0;                                      // device's context
    if (cudaGetDevice(&attr_dev) != cudaSuccess || attr_dev < 0 || attr_dev > 31) attr_dev = 0;
    if (!((attr_mask[sh != nullptr] >> attr_dev) & 1u)) {
        CVCL_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, fused::kSmemBytes));
        attr_mask[sh != nullptr] |= 1u << attr_dev;
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(f.grid);
    cfg.blockDim = dim3(fused::kThreads);
    cfg.dynamicSmemBytes = fused::kSmemBytes;
    cfg.stream = as_stream(stream);
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;          // all CTAs co-resident: the grid barriers cannot starve
    at[0].val.cooperative = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    CVCL_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kernel, maps, p));
    count_launch();
    return CVCL_OK;
}

int cvcl_flat_step_fused(const void* x16, const void* w16, const int64_t* ids, const int64_t* lens,
                         const float* bias, const float* table, int B, int L, int E, int K, int V,
                         int normalize, float log_scale, const float* log_scale_dev, int need_grads,
                         void* workspace, float* out5, float* img_feat_f32, float* txt_feat_f32,
                         float* dW, float* dbias, float* dtable, float* dscale, int* status, int phase_limit,
                         void* stream) {
    return flat_step_fused_impl(x16, w16, ids, lens, bias, table, B, L, E, K, V, normalize, log_scale, log_scale_dev,
                                need_grads, workspace, out5, img_feat_f32, txt_feat_f32, dW, dbias, dtable, dscale, status,
                                phase_limit, nullptr, stream);
}

int cvcl_flat_fused_sharded_supported(int B, int L, int E, int K, int V, int world) {
    FusedPlan f{};
    return plan_fused(&f, B, L, E, K, V, world) == nullptr ? 1 : 0;
}

size_t cvcl_flat_fused_sharded_workspace_bytes(int B, int L, int E, int K, int V, int world) {
    FusedPlan f{};
    return plan_fused(&f, B, L, E, K, V, world) == nullptr ? f.bytes : 0;
}

size_t cvcl_flat_fused_sharded_scratch_bytes(int B, int L, int E, int K, int V, int world) {
    FusedPlan f{};
    if (plan_fused(&f, B, L, E, K, V, world) != nullptr || world < 2) return 0;
    const int n_tiles5 = f.nEB * (K / 128) + ceil_div(V, 128) * f.nEB;
    const size_t nslot = ceil_div(n_tiles5, world);
    return align_up(static_cast<size_t>(world) * nslot * 128 * 128 * 4 + static_cast<size_t>(world) * fused::kSmall * 4, 256);
}

size_t cvcl_flat_fused_sharded_part_bytes(int B, int world) {
    if (B < 1 || world < 1) return 0;
    const size_t nCB = static_cast<size_t>(world) * ceil_div(B, 128);
    return 2 * (2 * nCB) * (static_cast<size_t>(world) * B) * sizeof(float2);
}

int cvcl_flat_step_fused_sharded(const void* x16, const void* w16, const int64_t* ids, const int64_t* lens,
                                 const float* bias, const float* table, int B, int L, int E, int K, int V,
                                 int normalize, float log_scale, const float* log_scale_dev, int need_grads,
                                 void* workspace, float* out5, float* img_feat_f32, float* txt_feat_f32,
                                 float* dW, float* dbias, float* dtable, float* dscale, int* status, int phase_limit,
                                 int world, int rank, void* const* peer_txt_all, void* const* peer_img_all,
                                 void* const* peer_part_all, void* const* peer_flags, unsigned int* epoch,
                                 void* const* peer_stats, void* const* peer_scratch, long long reduce_floats,
                                 void* stream) {
    CVCL_REQUIRE(peer_txt_all && peer_img_all && peer_part_all && peer_flags && epoch,
                 "flat_step_fused_sharded: null peer table");
    CVCL_REQUIRE(world >= 1 && world <= 8, "flat_step_fused_sharded: world size %d", world);
    CVCL_REQUIRE(reduce_floats >= 0, "flat_step_fused_sharded: reduce_floats < 0");
    FusedShard sh{world, rank, peer_txt_all, peer_img_all, peer_part_all, peer_flags, epoch, peer_stats, peer_scratch,
                  reduce_floats};
    return flat_step_fused_impl(x16, w16, ids, lens, bias, table, B, L, E, K, V, normalize, log_scale, log_scale_dev,
                                need_grads, workspace, out5, img_feat_f32, txt_feat_f32, dW, dbias, dtable, dscale, status,
                                phase_limit, &sh, stream);
}

// ------------------------------------------------------------------------------------ K6 spatial max
int cvcl_spatial_max_fwd(const void* tok, const void* img, const int64_t* lens, int Bt, int L, int Bi, int HW,
                         int E, float* match, unsigned char* amax_it, unsigned char* amax_ti, void* stream) {
    CVCL_REQUIRE(tok && img && lens && match && amax_it && amax_ti, "spatial_max_fwd: null pointer");
    CVCL_REQUIRE(Bt > 0 && Bi > 0 && E > 0, "spatial_max_fwd: bad shape");
    CVCL_REQUIRE(L >= 1 && L <= kBM && HW >= 1 && HW <= 256, "spatial_max_fwd: need L<=128, HW<=256 (L=%d HW=%d)", L, HW);
    constexpr int BN = 256;
    EpiSpatialMax::Params ep{};
    ep.L = L; ep.HW = HW; ep.TPM = kBM / L; ep.IPN = BN / HW; ep.Bt = Bt; ep.Bi = Bi;
    if (ep.IPN > EpiSpatialMax::kMaxIPN) ep.IPN = EpiSpatialMax::kMaxIPN;
    ep.lens = reinterpret_cast<const long long*>(lens); ep.match = match;
    ep.amax_it = amax_it; ep.amax_ti = amax_ti;
    GemmOperands op{}; op.ndir = 1;
    op.A[0] = mat(tok, Bt * L, E, E); op.B[0] = mat(img, Bi * HW, E, E);
    GemmShape gs{}; gs.M[0] = gs.M[1] = Bt * L; gs.N[0] = gs.N[1] = Bi * HW; gs.K = E;
    gs.m_stride = ep.TPM * L; gs.n_stride = ep.IPN * HW;
    return launch_gemm<BN, 2, EpiSpatialMax, false, false>(op, gs, ep, 1, as_stream(stream));   // 96 KB ring: 2 CTAs/SM
}

namespace {
struct SpatialBwdWs { size_t off_p, off_offs, off_tokc, off_dtokc, bytes; int ntlp; };
SpatialBwdWs spatial_bwd_ws(int Bt, int L, int Bi, int HW, int E) {
    SpatialBwdWs w{};
    w.ntlp = ceil_div(Bt * L, 128) * 128;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes, 256); return o; };
    w.off_p = take(2ull * w.ntlp * pad8(Bi * HW));            // compacted arg-max matrix P (bf16)
    w.off_offs = take(4ull * (Bt + 2));                       // token-row offsets, [Bt] = number of real tokens
    w.off_tokc = take(2ull * w.ntlp * E);                     // compacted token features (bf16)
    w.off_dtokc = take(4ull * w.ntlp * E);                    // compacted d tok (fp32)
    w.bytes = off;
    return w;
}
}  // namespace

size_t cvcl_spatial_max_bwd_workspace_bytes(int Bt, int L, int Bi, int HW, int E) {
    return spatial_bwd_ws(Bt, L, Bi, HW, E).bytes;
}

int cvcl_spatial_max_bwd(const float* gmatch, const int64_t* lens, const int64_t* ids,
                         const unsigned char* amax_it, const unsigned char* amax_ti, const void* tok,
                         const void* img, int Bt, int L, int Bi, int HW, int E, float* dtok, float* dimg,
                         void* workspace, void* stream) {
    CVCL_REQUIRE(gmatch && lens && amax_it && amax_ti && tok && img, "spatial_max_bwd: null pointer");
    CVCL_REQUIRE(E % 8 == 0 && E <= 1024, "spatial_max_bwd: E=%d must be a multiple of 8, <= 1024", E);
    if (workspace && HW >= 8) {         // (the expansion kernel's 8-column windows assume a map of >= 8 locations)
        // tensor-core form on COMPACTED token rows (pad positions dropped; their count is only known on the device):
        // offsets -> P_c (bf16, [Mv, Bi*HW]) + tok_c -> two GEMMs with a device-side row / contraction limit -> d tok
        // scattered back.  P_c is read K-major for dtok and MN-major (transposed in place) for dimg, the features are
        // read MN-major as stored.
        CVCL_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "spatial_max_bwd: workspace must be 256-byte aligned");
        const int ntl = Bt * L, ncol = Bi * HW, ldp = pad8(ncol);
        const SpatialBwdWs w = spatial_bwd_ws(Bt, L, Bi, HW, E);
        unsigned char* base = static_cast<unsigned char*>(workspace);
        __nv_bfloat16* P = reinterpret_cast<__nv_bfloat16*>(base + w.off_p);
        int* offs = reinterpret_cast<int*>(base + w.off_offs);
        __nv_bfloat16* tokc = reinterpret_cast<__nv_bfloat16*>(base + w.off_tokc);
        float* dtokc = reinterpret_cast<float*>(base + w.off_dtokc);
        cudaStream_t st = as_stream(stream);
        CVCL_CHECK_CUDA(launch_pdl(token_row_offsets_kernel, dim3(1), dim3(1024), 0, st,
                                   reinterpret_cast<const long long*>(lens), Bt, L, offs));
        count_launch();
        CVCL_CHECK_CUDA(launch_pdl(spatial_max_expand_kernel, dim3(ntl), dim3(256), 0, st, gmatch,
                                   reinterpret_cast<const long long*>(lens), amax_ti, P, static_cast<long long>(ldp),
                                   Bi, Bt, L, HW, static_cast<const int*>(offs), static_cast<const __nv_bfloat16*>(tok), tokc, E));
        count_launch();
        int rc;
        if (dtok) {
            if ((rc = gemm_f32out_limited(P, ldp, 0, img, E, 1, ntl, E, ncol, 1.f, dtokc, E, offs + Bt, nullptr, stream))) return rc;
            CVCL_CHECK_CUDA(launch_pdl(token_rows_scatter_kernel, dim3(warps_grid(ntl)), dim3(256), 0, st,
                                       static_cast<const float*>(dtokc), reinterpret_cast<const long long*>(lens),
                                       static_cast<const int*>(offs), dtok, Bt, L, E));
            count_launch();
        }
        if (dimg && (rc = gemm_f32out_limited(P, ldp, 1, tokc, E, 1, ncol, E, ntl, 1.f, dimg, E, nullptr, offs + Bt, stream))) return rc;
        return CVCL_OK;
    }
    if (dtok) {
        CVCL_CHECK_CUDA(launch_pdl(spatial_max_dtok_kernel, dim3(warps_grid(static_cast<long long>(Bt) * L)), dim3(256), 0, as_stream(stream), gmatch, reinterpret_cast<const long long*>(lens), reinterpret_cast<const long long*>(ids), amax_ti, static_cast<const __nv_bfloat16*>(img), dtok, Bi, Bt, L, HW, E));
        count_launch();
    }
    if (dimg) {
        CVCL_CHECK_CUDA(launch_pdl(spatial_max_dimg_kernel, dim3(warps_grid(static_cast<long long>(Bi) * HW)), dim3(256), 0, as_stream(stream), gmatch, reinterpret_cast<const long long*>(lens), amax_it, static_cast<const __nv_bfloat16*>(tok), dimg, Bi, Bt, L, HW, E));
        count_launch();
    }
    return CVCL_OK;
}

int cvcl_match_infonce_block_fwd(const float* match_r, const float* match_c, int b, int N, int diag_off,
                                 float log_scale, float inv_rows, void* workspace, float* lse0, float* lse1,
                                 int* argmax0, int* argmax1, float* out5, void* stream) {
    CVCL_REQUIRE(match_r && match_c && workspace && lse0 && lse1 && out5, "match_infonce_fwd: null pointer");
    CVCL_REQUIRE(b > 0 && N > 0, "match_infonce_fwd: bad shape");
    CVCL_REQUIRE(diag_off >= 0 && b + diag_off <= N, "match_infonce_fwd: positives out of range (b=%d N=%d diag_off=%d)",
                 b, N, diag_off);
    SimWs w = carve_sim_ws(workspace, b, N, b, N);
    CVCL_CHECK_CUDA(launch_pdl(match_stats_kernel, dim3(warps_grid(2ll * b)), dim3(256), 0, as_stream(stream), match_r, match_c, b, N, diag_off, expf(log_scale), w.part[0], w.part[1], w.diag[0], w.diag[1], w.ticket));
    count_launch();
    FinalizeParams fp{};
    for (int z = 0; z < 2; ++z) {
        fp.part[z] = w.part[z]; fp.m_pad[z] = w.m_pad[z]; fp.n_tiles[z] = 1; fp.diag[z] = w.diag[z];
        fp.diag_off[z] = diag_off; fp.M[z] = b;
    }
    fp.lse[0] = lse0; fp.lse[1] = lse1; fp.argmax[0] = argmax0; fp.argmax[1] = argmax1;
    fp.inv_rows = inv_rows; fp.block_part = w.block_part; fp.ticket = w.ticket; fp.out = out5;
    CVCL_CHECK_CUDA(launch_pdl(infonce_finalize_kernel, dim3(ceil_div(2 * b, 256)), dim3(256), 0, as_stream(stream), fp));
    count_launch();
    return CVCL_OK;
}

int cvcl_match_infonce_fwd(const float* match, int B, float log_scale, float inv_rows, void* workspace,
                           float* lse0, float* lse1, int* argmax0, int* argmax1, float* out5, void* stream) {
    return cvcl_match_infonce_block_fwd(match, match, B, B, 0, log_scale, inv_rows, workspace, lse0, lse1, argmax0,
                                        argmax1, out5, stream);
}

namespace {
int match_grad_blocks(int b, int N) { return static_cast<int>((static_cast<long long>(b) * N + 255) / 256); }

int match_grad_launch(const float* match_r, const float* match_c, int b, int N, int diag_off, float log_scale,
                      float coef, const float* lse0, const float* lse1_all, const float* lse0_all, const float* lse1,
                      float* dmatch_r, float* dmatch_c, float* dscale, void* workspace, void* stream) {
    const int nb = match_grad_blocks(b, N);
    unsigned int* ticket = nullptr;
    float* ds_part = nullptr;
    if (workspace) {
        ticket = static_cast<unsigned int*>(workspace);
        ds_part = reinterpret_cast<float*>(static_cast<unsigned char*>(workspace) + 256);
        CVCL_CHECK_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned int), as_stream(stream)));
    }
    CVCL_CHECK_CUDA(launch_pdl(match_grad_kernel, dim3(nb, dmatch_c ? 2 : 1), dim3(256), 0, as_stream(stream),
                               match_r, match_c, b, N, diag_off, expf(log_scale), coef, lse0, lse1_all, lse0_all, lse1,
                               dmatch_r, dmatch_c, dscale, ds_part, ticket));
    count_launch();
    return CVCL_OK;
}
}  // namespace

size_t cvcl_match_infonce_block_bwd_workspace_bytes(int b, int N) {
    return 256 + align_up(sizeof(float) * static_cast<size_t>(match_grad_blocks(b, N)), 256);
}

int cvcl_match_infonce_block_bwd(const float* match_r, const float* match_c, int b, int N, int diag_off,
                                 float log_scale, float coef, const float* lse0, const float* lse1_all,
                                 const float* lse0_all, const float* lse1, float* dmatch_r, float* dmatch_c,
                                 float* dscale, void* workspace, void* stream) {
    CVCL_REQUIRE(match_r && match_c && lse0 && lse1_all && lse0_all && lse1 && dmatch_r && dmatch_c && dscale && workspace,
                 "match_infonce_block_bwd: null pointer");
    CVCL_REQUIRE(b > 0 && N > 0 && diag_off >= 0 && b + diag_off <= N,
                 "match_infonce_block_bwd: bad shape (b=%d N=%d diag_off=%d)", b, N, diag_off);
    CVCL_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "match_infonce_block_bwd: workspace must be 256-byte aligned");
    return match_grad_launch(match_r, match_c, b, N, diag_off, log_scale, coef, lse0, lse1_all, lse0_all, lse1,
                             dmatch_r, dmatch_c, dscale, workspace, stream);
}

int cvcl_match_infonce_bwd(const float* match, int B, float log_scale, float coef, const float* lse0,
                           const float* lse1, float* dmatch, float* dscale, void* stream) {
    CVCL_REQUIRE(match && lse0 && lse1 && dmatch, "match_infonce_bwd: null pointer");
    return match_grad_launch(match, match, B, B, 0, log_scale, coef, lse0, lse1, lse0, lse1, dmatch, nullptr, dscale,
                             nullptr, stream);
}

// ------------------------------------------------------------------------------------ peer-memory gather
int cvcl_p2p_gather(const void* const* peer_ptrs, int world, int skip_rank, long long bytes_per_rank, void* dst,
                    long long dst_stride_bytes, void* stream) {
    CVCL_REQUIRE(peer_ptrs && dst, "p2p_gather: null pointer");
    CVCL_REQUIRE(world >= 1 && world <= 8, "p2p_gather: world size %d not in [1,8]", world);
    CVCL_REQUIRE(bytes_per_rank % 16 == 0 && dst_stride_bytes % 16 == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0,
                 "p2p_gather: 16-byte granularity required");
    if (bytes_per_rank == 0) return CVCL_OK;
    PeerPtrs pp{};
    for (int r = 0; r < world; ++r) {
        CVCL_REQUIRE(peer_ptrs[r] && (reinterpret_cast<uintptr_t>(peer_ptrs[r]) & 15) == 0, "p2p_gather: bad peer pointer %d", r);
        pp.p[r] = peer_ptrs[r];
    }
    long long blocks = (bytes_per_rank / 16 + 255) / 256;
    if (blocks > 64) blocks = 64;
    CVCL_CHECK_CUDA(launch_pdl(p2p_gather_kernel, dim3(static_cast<unsigned>(blocks), world), dim3(256), 0, as_stream(stream),
                               pp, static_cast<unsigned char*>(dst), bytes_per_rank, dst_stride_bytes, skip_rank));
    count_launch();
    return CVCL_OK;
}

// ------------------------------------------------------------------------------------ peer collectives
namespace {
int fill_peer_table(PeerTable* t, void* const* peer_data, void* const* peer_flags, unsigned int* epoch, int* status,
                    int world, int rank, unsigned int timeout_ms, const char* who) {
    CVCL_REQUIRE(world >= 1 && world <= kPeerMaxWorld, "%s: world size %d not in [1,%d]", who, world, kPeerMaxWorld);
    CVCL_REQUIRE(rank >= 0 && rank < world, "%s: rank %d outside [0,%d)", who, rank, world);
    CVCL_REQUIRE(peer_flags && epoch, "%s: null flag / epoch pointer", who);
    for (int r = 0; r < world; ++r) {
        CVCL_REQUIRE(peer_flags[r] && (reinterpret_cast<uintptr_t>(peer_flags[r]) & 3) == 0, "%s: bad flag pointer %d", who, r);
        t->flags[r] = static_cast<uint32_t*>(peer_flags[r]);
        if (peer_data) {
            CVCL_REQUIRE(peer_data[r] && (reinterpret_cast<uintptr_t>(peer_data[r]) & 15) == 0, "%s: bad peer pointer %d", who, r);
            t->data[r] = peer_data[r];
        }
    }
    t->epoch = epoch; t->status = status;
    t->timeout_ms = (timeout_ms & 0x7fffffffu) ? timeout_ms : ((timeout_ms & 0x80000000u) | 600000u);
    return CVCL_OK;
}
}  // namespace

size_t cvcl_peer_flag_words(void) { return kPeerFlagWords; }
int cvcl_peer_max_blocks(void) { return kPeerMaxBlocks; }

int cvcl_peer_allgather(void* const* peer_data, void* const* peer_flags, unsigned int* epoch, int* status, int world,
                        int rank, long long seg_bytes, int nseg, long long src_seg_stride_bytes, void* dst,
                        long long dst_seg_stride_bytes, unsigned int timeout_ms, void* stream) {
    CVCL_REQUIRE(peer_data && dst, "peer_allgather: null pointer");
    CVCL_REQUIRE(seg_bytes > 0 && nseg >= 1, "peer_allgather: empty exchange");
    CVCL_REQUIRE(seg_bytes % 16 == 0 && src_seg_stride_bytes % 16 == 0 && dst_seg_stride_bytes % 16 == 0 &&
                 (reinterpret_cast<uintptr_t>(dst) & 15) == 0, "peer_allgather: 16-byte granularity required");
    PeerTable t{};
    int rc = fill_peer_table(&t, peer_data, peer_flags, epoch, status, world, rank, timeout_ms, "peer_allgather");
    if (rc != CVCL_OK) return rc;
    const long long total16 = seg_bytes / 16 * nseg * world;
    long long blocks = (total16 + 4LL * kPeerThreads - 1) / (4LL * kPeerThreads);     // same on every rank
    blocks = blocks < 1 ? 1 : (blocks > kPeerMaxBlocks ? kPeerMaxBlocks : blocks);
    peer_allgather_kernel<<<static_cast<unsigned>(blocks), kPeerThreads, 0, as_stream(stream)>>>(
        t, world, rank, seg_bytes / 16, nseg, src_seg_stride_bytes / 16, static_cast<uint4*>(dst), dst_seg_stride_bytes / 16);
    CVCL_CHECK_CUDA(cudaGetLastError());
    count_launch();
    return CVCL_OK;
}

int cvcl_peer_allreduce_f32(void* const* peer_data, void* const* peer_flags, unsigned int* epoch, int* status, int world,
                            int rank, long long n, unsigned int timeout_ms, void* stream) {
    CVCL_REQUIRE(peer_data, "peer_allreduce_f32: null pointer");
    CVCL_REQUIRE(n > 0 && n % 4 == 0, "peer_allreduce_f32: n=%lld must be a positive multiple of 4", n);
    if (world != 1 && world != 2 && world != 4 && world != 8)
        return fail(CVCL_ERR_UNSUPPORTED, "peer_allreduce_f32: world size %d (supported: 1, 2, 4, 8)", world);
    if (world == 1) return CVCL_OK;
    PeerTable t{};
    int rc = fill_peer_table(&t, peer_data, peer_flags, epoch, status, world, rank, timeout_ms, "peer_allreduce_f32");
    if (rc != CVCL_OK) return rc;
    const long long n4 = n / 4, per = (n4 + world - 1) / world;
    long long blocks = (per + 2LL * kPeerThreads - 1) / (2LL * kPeerThreads);           // same on every rank
    blocks = blocks < 1 ? 1 : (blocks > kPeerMaxBlocks ? kPeerMaxBlocks : blocks);
    const dim3 grid(static_cast<unsigned>(blocks));
    cudaStream_t st = as_stream(stream);
    if (world == 2) peer_allreduce_f32_kernel<2><<<grid, kPeerThreads, 0, st>>>(t, rank, n4);
    else if (world == 4) peer_allreduce_f32_kernel<4><<<grid, kPeerThreads, 0, st>>>(t, rank, n4);
    else peer_allreduce_f32_kernel<8><<<grid, kPeerThreads, 0, st>>>(t, rank, n4);
    CVCL_CHECK_CUDA(cudaGetLastError());
    count_launch();
    return CVCL_OK;
}

int cvcl_peer_allgather_push(void* const* peer_dst, void* const* peer_flags, unsigned int* epoch, int* status, int world,
                             int rank, const void* src, long long seg_bytes, int nseg, long long src_seg_stride_bytes,
                             long long dst_seg_stride_bytes, unsigned int timeout_ms, void* stream) {
    CVCL_REQUIRE(peer_dst && src, "peer_allgather_push: null pointer");
    CVCL_REQUIRE(seg_bytes > 0 && nseg >= 1, "peer_allgather_push: empty exchange");
    CVCL_REQUIRE(seg_bytes % 16 == 0 && src_seg_stride_bytes % 16 == 0 && dst_seg_stride_bytes % 16 == 0 &&
                 (reinterpret_cast<uintptr_t>(src) & 15) == 0, "peer_allgather_push: 16-byte granularity required");
    PeerTable t{};
    int rc = fill_peer_table(&t, peer_dst, peer_flags, epoch, status, world, rank, timeout_ms, "peer_allgather_push");
    if (rc != CVCL_OK) return rc;
    const long long per16 = seg_bytes / 16 * nseg;
    long long blocks = (per16 + 4LL * kPeerThreads - 1) / (4LL * kPeerThreads);        // same on every rank
    blocks = blocks < 1 ? 1 : (blocks > kPeerMaxBlocks ? kPeerMaxBlocks : blocks);
    CVCL_CHECK_CUDA(launch_pdl(peer_allgather_push_kernel, dim3(static_cast<unsigned>(blocks)), dim3(kPeerThreads), 0,
                               as_stream(stream), t, world, rank, static_cast<const uint4*>(src), seg_bytes / 16, nseg,
                               src_seg_stride_bytes / 16, dst_seg_stride_bytes / 16));
    count_launch();
    return CVCL_OK;
}

size_t cvcl_peer_allreduce_scratch_bytes(long long n, int world) {
    if (n <= 0 || world < 1) return 0;
    const long long n4 = (n + 3) / 4, per = (n4 + world - 1) / world;
    return static_cast<size_t>(per) * world * 16;
}

int cvcl_peer_allreduce_push_f32(void* const* peer_data, void* const* peer_scratch, void* const* peer_flags,
                                 unsigned int* epoch, int* status, int world, int rank, long long n,
                                 unsigned int timeout_ms, void* stream) {
    CVCL_REQUIRE(peer_data && peer_scratch, "peer_allreduce_push_f32: null pointer");
    CVCL_REQUIRE(n > 0 && n % 4 == 0, "peer_allreduce_push_f32: n=%lld must be a positive multiple of 4", n);
    if (world != 1 && world != 2 && world != 4 && world != 8)
        return fail(CVCL_ERR_UNSUPPORTED, "peer_allreduce_push_f32: world size %d (supported: 1, 2, 4, 8)", world);
    if (world == 1) return CVCL_OK;
    PeerTable t{};
    int rc = fill_peer_table(&t, peer_data, peer_flags, epoch, status, world, rank, timeout_ms, "peer_allreduce_push_f32");
    if (rc != CVCL_OK) return rc;
    for (int r = 0; r < world; ++r) {
        CVCL_REQUIRE(peer_scratch[r] && (reinterpret_cast<uintptr_t>(peer_scratch[r]) & 15) == 0,
                     "peer_allreduce_push_f32: bad scratch pointer %d", r);
        t.aux[r] = peer_scratch[r];
    }
    const long long n4 = n / 4, per = (n4 + world - 1) / world;
    long long blocks = (per + 2LL * kPeerThreads - 1) / (2LL * kPeerThreads);           // same on every rank
    blocks = blocks < 1 ? 1 : (blocks > kPeerMaxBlocks ? kPeerMaxBlocks : blocks);
    const dim3 grid(static_cast<unsigned>(blocks)), block(kPeerThreads);
    cudaStream_t st = as_stream(stream);
    if (world == 2) CVCL_CHECK_CUDA(launch_pdl(peer_allreduce_push_f32_kernel<2>, grid, block, 0, st, t, rank, n4));
    else if (world == 4) CVCL_CHECK_CUDA(launch_pdl(peer_allreduce_push_f32_kernel<4>, grid, block, 0, st, t, rank, n4));
    else CVCL_CHECK_CUDA(launch_pdl(peer_allreduce_push_f32_kernel<8>, grid, block, 0, st, t, rank, n4));
    count_launch();
    return CVCL_OK;
}

int cvcl_peer_barrier(void* const* peer_flags, unsigned int* epoch, int* status, int world, int rank,
                      unsigned int timeout_ms, void* stream) {
    PeerTable t{};
    int rc = fill_peer_table(&t, nullptr, peer_flags, epoch, status, world, rank, timeout_ms, "peer_barrier");
    if (rc != CVCL_OK) return rc;
    if (world == 1) return CVCL_OK;
    peer_barrier_kernel<<<1, 32, 0, as_stream(stream)>>>(t, world, rank);
    CVCL_CHECK_CUDA(cudaGetLastError());
    count_launch();
    return CVCL_OK;
}

// ------------------------------------------------------------------------------------ fused AdamW
int cvcl_adamw_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                    float beta2, float eps, float weight_decay, int step, float grad_scale, void* bf16_shadow,
                    void* stream) {
    CVCL_REQUIRE(p && g && m && v, "adamw_step: null pointer");
    CVCL_REQUIRE(n >= 0 && step >= 1, "adamw_step: bad n / step");
    CVCL_REQUIRE(((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
                   reinterpret_cast<uintptr_t>(v)) & 15) == 0, "adamw_step: tensors must be 16-byte aligned");
    if (n == 0) return CVCL_OK;
    const float bc1 = 1.f - powf(beta1, static_cast<float>(step));
    const float bc2_sqrt = sqrtf(1.f - powf(beta2, static_cast<float>(step)));
    long long blocks = (n / 4 + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    if (blocks < 1) blocks = 1;
    CVCL_CHECK_CUDA(launch_pdl(adamw_step_kernel, dim3(static_cast<unsigned>(blocks)), dim3(256), 0, as_stream(stream),
                               p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, bc1, bc2_sqrt, grad_scale,
                               static_cast<__nv_bfloat16*>(bf16_shadow)));
    count_launch();
    return CVCL_OK;
}

int cvcl_adamw_multi_step(int count, float* const* p, const float* const* g, float* const* m, float* const* v,
                          const long long* n, void* const* bf16_shadow, const float* lr, const float* weight_decay,
                          float beta1, float beta2, float eps, float grad_scale, int* step_dev,
                          unsigned int* ticket, void* stream) {
    CVCL_REQUIRE(count >= 1 && count <= kAdamMaxTensors, "adamw_multi_step: 1..%d tensors (got %d)", kAdamMaxTensors, count);
    CVCL_REQUIRE(p && g && m && v && n && lr && weight_decay && step_dev && ticket, "adamw_multi_step: null pointer");
    AdamMultiParams a{};
    a.count = count; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.grad_scale = grad_scale;
    a.step_dev = step_dev; a.ticket = ticket;
    long long off = 0;
    for (int t = 0; t < count; ++t) {
        CVCL_REQUIRE(p[t] && g[t] && m[t] && v[t] && n[t] > 0, "adamw_multi_step: bad tensor %d", t);
        CVCL_REQUIRE(((reinterpret_cast<uintptr_t>(p[t]) | reinterpret_cast<uintptr_t>(g[t]) |
                       reinterpret_cast<uintptr_t>(m[t]) | reinterpret_cast<uintptr_t>(v[t])) & 15) == 0 || n[t] < 4,
                     "adamw_multi_step: tensor %d must be 16-byte aligned", t);
        a.p[t] = p[t]; a.g[t] = g[t]; a.m[t] = m[t]; a.v[t] = v[t]; a.n[t] = n[t];
        a.shadow[t] = bf16_shadow ? static_cast<__nv_bfloat16*>(bf16_shadow[t]) : nullptr;
        a.lr[t] = lr[t]; a.wd[t] = weight_decay[t];
        a.n4_begin[t] = off;
        off += (n[t] + 3) / 4;
    }
    a.n4_begin[count] = off;
    for (int t = count + 1; t <= kAdamMaxTensors; ++t) a.n4_begin[t] = off;
    long long blocks = (off + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    CVCL_CHECK_CUDA(launch_pdl(adamw_multi_kernel, dim3(static_cast<unsigned>(blocks)), dim3(256), 0, as_stream(stream), a));
    count_launch();
    return CVCL_OK;
}

// ------------------------------------------------------------------------------------ Grad-CAM
size_t cvcl_gradcam_workspace_bytes(int N, int K, int E) {
    if (N <= 0 || K <= 0 || E <= 0) return 0;
    return sizeof(float) * (2ull * N * K + 2ull * N * E);
}

int cvcl_gradcam_flat(const float* act, const float* w, const float* bias, const float* target, int N, int K, int HW,
                      int E, int normalize, void* workspace, float* cam, void* stream) {
    CVCL_REQUIRE(act && w && target && workspace && cam, "gradcam_flat: null pointer");
    CVCL_REQUIRE(N >= 0 && K > 0 && E > 0 && HW > 0, "gradcam_flat: bad shape");
    CVCL_REQUIRE(HW <= 64, "gradcam_flat: HW=%d > 64 locations", HW);
    CVCL_REQUIRE(K % 4 == 0 && (reinterpret_cast<uintptr_t>(w) & 15) == 0 && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0,
                 "gradcam_flat: K %% 4 == 0 and 16-byte aligned weight / workspace required");
    if (N == 0) return CVCL_OK;
    cudaStream_t st = as_stream(stream);
    float* pooled = static_cast<float*>(workspace);
    float* alpha = pooled + static_cast<size_t>(N) * K;
    float* u = alpha + static_cast<size_t>(N) * K;
    float* g = u + static_cast<size_t>(N) * E;
    const long long rows = static_cast<long long>(N) * K;
    CVCL_CHECK_CUDA(launch_pdl(gradcam_pool_kernel, dim3(warps_grid(rows)), dim3(256), 0, st, act, pooled, rows, HW));
    count_launch();
    CVCL_CHECK_CUDA(launch_pdl(gradcam_head_kernel, dim3(warps_grid(static_cast<long long>(N) * E)), dim3(256), 0, st,
                               static_cast<const float*>(pooled), w, bias, u, N, E, K));
    count_launch();
    CVCL_CHECK_CUDA(launch_pdl(gradcam_g_kernel, dim3(warps_grid(N, 128)), dim3(128), 0, st, static_cast<const float*>(u),
                               target, g, N, E, normalize));
    count_launch();
    CVCL_CHECK_CUDA(launch_pdl(gradcam_alpha_kernel, dim3(ceil_div(K, 256), N), dim3(256), 0, st,
                               static_cast<const float*>(g), w, alpha, N, E, K, 1.f / static_cast<float>(HW)));
    count_launch();
    CVCL_CHECK_CUDA(launch_pdl(gradcam_cam_kernel, dim3(N), dim3(256), 0, st, act, static_cast<const float*>(alpha), cam, K, HW));
    count_launch();
    return CVCL_OK;
}

int cvcl_bicubic_upsample(const float* in, int N, int h, int w, int H, int W, float* out, void* stream) {
    CVCL_REQUIRE(in && out, "bicubic_upsample: null pointer");
    CVCL_REQUIRE(N >= 0 && h > 0 && w > 0 && H > 0 && W > 0, "bicubic_upsample: bad shape");
    const long long total = static_cast<long long>(N) * H * W;
    if (total == 0) return CVCL_OK;
    CVCL_CHECK_CUDA(launch_pdl(bicubic_upsample_kernel, dim3(static_cast<unsigned>((total + 255) / 256)), dim3(256), 0,
                               as_stream(stream), in, out, N, h, w, H, W));
    count_launch();
    return CVCL_OK;
}

// ------------------------------------------------------------------------------------ K7
int cvcl_eval_nway_fwd(const float* img, const float* txt, const int* txt_index, int n_trials, int n_way,
                       int E, int normalize, float log_scale, int* pred, float* logits, void* stream) {
    CVCL_REQUIRE(img && txt && pred, "eval_nway_fwd: null pointer");
    CVCL_REQUIRE(n_trials >= 0 && n_way > 0, "eval_nway_fwd: bad shape");
    CVCL_REQUIRE(E > 0 && E % 4 == 0 && E <= 128 * kMaxVec, "eval_nway_fwd: bad E=%d", E);
    if (n_trials == 0) return CVCL_OK;
    if (n_way == 4 && E <= 512 && n_trials >= 4096 && !(logits && normalize) && (reinterpret_cast<uintptr_t>(img) & 15) == 0) {
        // streaming form: persistent blocks, 32 KB stages filled by bulk async copies
        const int smem = 128 + kEvalStages * kEvalGroup * 4 * E * 4;
        static thread_local unsigned attr_mask = 0;     // per device: function attributes live in the device's context
        int attr_dev = 0;
        if (cudaGetDevice(&attr_dev) != cudaSuccess || attr_dev < 0 || attr_dev > 31) attr_dev = 0;
        if (!((attr_mask >> attr_dev) & 1u)) {
            CVCL_CHECK_CUDA(cudaFuncSetAttribute(eval_nway_stream_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 128 + kEvalStages * kEvalGroup * 4 * 512 * 4));
            attr_mask |= 1u << attr_dev;
        }
        const int n_groups = ceil_div(n_trials, kEvalGroup);
        const int grid = n_groups < 3 * sm_count() ? n_groups : 3 * sm_count();
        CVCL_CHECK_CUDA(launch_pdl(eval_nway_stream_kernel<4>, dim3(grid), dim3(32 * (kEvalGroup + 1)), smem,
                                   as_stream(stream), img, txt, txt_index, n_trials, E, normalize, expf(log_scale), pred,
                                   logits));
    } else if (n_way == 4 && E <= 512)
        CVCL_CHECK_CUDA(launch_pdl(eval_nway_kernel<4>, dim3(warps_grid(n_trials)), dim3(256), 0, as_stream(stream), img, txt, txt_index, n_trials, n_way, E, normalize, expf(log_scale), pred, logits));
    else
        CVCL_CHECK_CUDA(launch_pdl(eval_nway_kernel<0>, dim3(warps_grid(n_trials)), dim3(256), 0, as_stream(stream), img, txt, txt_index, n_trials, n_way, E, normalize, expf(log_scale), pred, logits));
    count_launch();
    return CVCL_OK;
}

}  // extern "C"
