// exl_common.cuh -- shared declarations for libexl_b200.so (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cublas_v2.h>
#include <cstdint>
#include <cstdio>
#include <cstdarg>
#include <cstring>
#include <atomic>
#include "../../include/exl_b200.h"

// Q4 matrix handle (reference: class Q4Matrix, exllama_ext/cuda_func/q4_matrix.cuh:8-46).
// qweight/qzeros/scales are borrowed device pointers; x_map is owned.
struct exl_q4_matrix
{
    int device;
    int K;            // height (input features)
    int N;            // width  (output features)
    int groups;
    int groupsize;
    uint32_t* qweight;   // [K/8, N]
    uint32_t* qzeros;    // [groups, N/8]
    half* scales;        // [groups, N]
    uint32_t* x_map;     // [K] or nullptr (act-order: x column feeding sequential row k)
    // TMA descriptor of qweight as a 2-D int32 tensor [K/8, N], box 16 rows x 32 columns, 128-byte swizzle (q4_gemv.cu)
    alignas(64) CUtensorMap tmap_w;
    // same tensor, box 8 rows x 128 columns, no swizzle: the packed-word tile of one k-block of the tcgen05 GEMM (q4_gemm_tc.cu)
    alignas(64) CUtensorMap tmap_wp;
    // decode_step.cu: ONE op per 8 KB unit -- qweight viewed as [N/32][K/8][32] (dims fastest first: 32 columns, k8-row, column group),
    // box 32 x 16 x 4 with the 128-byte swizzle: the same shared-memory image as four tmap_w boxes side by side.  valid3 == 0 when
    // N % 32 != 0.
    alignas(64) CUtensorMap tmap_w3;
    // scales [groups, N] fp16, box 128 columns x R group rows; qzeros [groups, N/8] u32, box 16 words x R rows;
    // R = group rows per 128-row K stage (groupsize 32: 4, 64: 2, >= 128: 1)
    alignas(64) CUtensorMap tmap_sc;
    alignas(64) CUtensorMap tmap_qz;
    int valid3;
};

struct ExlTuning
{
    int matmul_recons_thd = 8;
    int fused_mlp_thd = 2;
    int sdp_thd = 8;
    bool matmul_fused_remap = false;
    bool rmsnorm_no_half2 = false, rope_no_half2 = false, matmul_no_half2 = false, silu_no_half2 = false;
    bool concurrent_streams = false;
};

// Per-device state: borrowed scratch from prepare_buffers (reference: CudaBuffers, cuda_buffers.cuh:15-49)
// plus library-owned split-K workspace and a cuBLAS handle.
struct ExlDevice
{
    bool init = false;
    int device = -1;
    int num_sms = 0;
    // borrowed
    half* temp_state = nullptr;  int64_t temp_state_numel = 0;
    half* temp_mlp = nullptr;    int64_t temp_mlp_numel = 0;
    float* temp_zeros_float = nullptr; int max_zeros_float = 0;
    half* temp_dq = nullptr;     int64_t temp_dq_numel = 0;
    // owned
    // library-owned scratch for callers that never called prepare_buffers (or passed buffers that are too small).
    // One buffer PER ROLE: nested users (fused block -> q4_matmul -> act-order gather / reconstruct) never alias and a
    // role is only ever grown by its own user, so no pointer handed out earlier in the same op can be freed under it.
    half* own[4] = {nullptr, nullptr, nullptr, nullptr};  int64_t own_numel[4] = {0, 0, 0, 0};
    cublasHandle_t blas = nullptr;
    int gemv_ctas_per_sm = 0;
    // tensor-parallel one-shot all-reduce over NVLink peer memory (q4_gemv.cu, GV_EPI_ALLREDUCE)
    int tp_rank = 0, tp_world = 1;
    unsigned char* tp_local = nullptr;                 // this rank's workspace (cudaMalloc, exported through cudaIpc)
    unsigned char* tp_peers[8] = {nullptr};            // every rank's workspace mapped into this process (own = tp_local)
};

// workspace layout (identical on every rank): receive slots [parity 2][src rank 8][tile TP_MAX_TILES][row 8][128] fp32,
// flags [parity 2][src rank 8][tile] u32, then {epoch, done} u32
constexpr int TP_MAX_RANKS = 8;
constexpr int TP_MAX_TILES = 256;
constexpr size_t TP_DATA_BYTES = (size_t)2 * TP_MAX_RANKS * TP_MAX_TILES * 8 * 128 * sizeof(float);
constexpr size_t TP_FLAG_BYTES = (size_t)2 * TP_MAX_RANKS * TP_MAX_TILES * sizeof(unsigned);
constexpr size_t TP_WS_BYTES = TP_DATA_BYTES + TP_FLAG_BYTES + 256;       // + control words {epoch, done, timeouts}
constexpr unsigned TP_SPIN_LIMIT = 1u << 23;                                // polls of the own flag word (~ seconds) before giving up

extern ExlTuning g_tuning;
extern std::atomic<int64_t> g_launches;
extern const char* g_last_q4_path;
extern const char* g_last_tc_config;
extern char g_last_gemv_config[512];

enum ExlScratchRole { SCR_NORM = 0, SCR_MLP = 1, SCR_DQ = 2, SCR_REMAP = 3 };
int exl_own_scratch(ExlDevice* ds, int role, int64_t numel, half** out);   // grow-only, lazy; not CUDA-graph safe on first use

int exl_set_err(int code, const char* fmt, ...);
ExlDevice* exl_device_state(int device);          // lazily initialised; nullptr + error on failure
int exl_current_device_of(const void* ptr);       // device index owning a device pointer, or -1

#define EXL_CUDA_TRY(expr)                                                                   \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess)                                                               \
            return exl_set_err(EXL_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,                 \
                               cudaGetErrorString(_e), __FILE__, __LINE__);                  \
    } while (0)

#define EXL_CHECK_LAUNCH(name)                                                               \
    do {                                                                                     \
        g_launches.fetch_add(1, std::memory_order_relaxed);                                  \
        cudaError_t _e = cudaGetLastError();                                                 \
        if (_e != cudaSuccess)                                                               \
            return exl_set_err(EXL_ERR_CUDA, "launch of %s failed: %s", name,                \
                               cudaGetErrorString(_e));                                      \
    } while (0)

struct DeviceGuard
{
    int prev = -1; bool changed = false;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (dev >= 0 && dev != prev) { cudaSetDevice(dev); changed = true; } }
    ~DeviceGuard() { if (changed) cudaSetDevice(prev); }
};

// ---- internal entry points shared between translation units -------------------------------------

// q4_gemv.cu : skinny-M fused unpack + scale/zero + GEMV (M <= 8), up to 3 matrices sharing x.
enum GemvPrologue { GV_PRO_PLAIN = 0, GV_PRO_RMSNORM = 1 };
enum GemvEpilogue { GV_EPI_STORE = 0, GV_EPI_SILU_MUL = 1, GV_EPI_ROPE_CACHE = 2, GV_EPI_ALLREDUCE = 3 };

struct GemvFused
{
    // prologue (GV_PRO_RMSNORM): x_staged = (x * half(rsqrt(mean(x^2) + eps))) * norm_w, also written to norm_out if set
    const half* norm_w = nullptr;
    float eps = 0.f;
    // epilogue GV_EPI_ROPE_CACHE (q4_attn): mats = {q, k, v}
    const half* sin = nullptr; const half* cos = nullptr;
    int head_dim = 0, num_heads = 0, num_kv_heads = 0, past_len = 0, max_seq_len = 0, q_len = 1;
    half* key_cache = nullptr; half* value_cache = nullptr;
};

int exl_gemv_launch(ExlDevice* ds, const half* x, int M, const exl_q4_matrix* const* mats, half* const* outs,
                    int num_mats, bool no_zero, int prologue, int epilogue, const GemvFused* fused, cudaStream_t stream);

// q4_matrix.cu
int exl_encode_weight_tmap(exl_q4_matrix* w);
int exl_reconstruct_launch(const exl_q4_matrix* w, half* out, cudaStream_t stream);

// q4_gemm_tc.cu : tcgen05 fused-dequant GEMM (prefill)
int exl_tc_gemm_launch(ExlDevice* ds, const half* x, int M, const exl_q4_matrix* w, half* out, bool no_zero, cudaStream_t stream);
bool exl_tc_gemm_supported(const exl_q4_matrix* w, int M);

// elementwise.cu
int exl_rms_norm_launch(const half* x, const half* w, half* out, float eps, int rows, int dim, cudaStream_t stream);
int exl_rope_launch(half* x, const half* sin, const half* cos, int bsz, int rows_per_batch, int head_dim, int num_heads, int past_len, cudaStream_t stream);
int exl_silu_mul_launch(half* x, const half* y, int height, int width, cudaStream_t stream);
int exl_update_cache_launch(const half* k, const half* v, half* kc, half* vc, int head_dim, int kvh, int q_len, int max_seq, int past_len, cudaStream_t stream);
int exl_column_remap_launch(const half* x, half* x_new, int M, int K, const uint32_t* x_map, cudaStream_t stream);

// decode_attn.cu
int exl_decode_attn_launch(const half* q, const half* kc, const half* vc, half* out, int heads, int kv_heads, int head_dim,
                           int seq, int max_seq, float scale, cudaStream_t stream);

// half_matmul.cu
int exl_half_matmul_cublas_launch(ExlDevice* ds, const half* x, const half* w, half* out, int M, int K, int N, bool no_zero, cudaStream_t stream);
int exl_half_matmul_custom_launch(const half* x, const half* w, half* out, int M, int K, int N, cudaStream_t stream);

constexpr int GV_TILE_N = 128;
constexpr int GV_MAXM = 8;
