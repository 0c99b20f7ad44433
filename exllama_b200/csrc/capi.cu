// capi.cu -- extern "C" entry points of libexl_b200.so (see include/exl_b200.h) and the host-side state behind
// them: tuning parameters, per-device scratch (reference: exllama_ext/cuda_buffers.cu), the Q4 handle registry
// (reference: q4_matrix.cu:13-24) and the decode-block orchestration (reference: q4_attn.cu:74-228,
// q4_mlp.cu:100-199).  No torch types; no CPU compute fallback.
#include "exl_common.cuh"
#include <vector>
#include <mutex>
#include <cstring>
#include <cstdlib>
#include <cmath>

ExlTuning g_tuning;
std::atomic<int64_t> g_launches{0};
const char* g_last_q4_path = "none";
const char* g_last_tc_config = "none";
char g_last_gemv_config[512] = "";      // q4_gemv launches of the last exl_q4_* call (cleared on entry, appended by launch_cfg)

static thread_local char t_err[1024] = "";
static ExlDevice g_devices[EXL_MAX_DEVICES];
static std::vector<exl_q4_matrix*> g_matrices;
static std::mutex g_mutex;

int exl_make_sequential_launch(uint32_t* qweight, uint32_t* tmp, const uint32_t* x_map, int K, int N, cudaStream_t stream);

int exl_set_err(int code, const char* fmt, ...)
{
    va_list ap; va_start(ap, fmt);
    vsnprintf(t_err, sizeof(t_err), fmt, ap);
    va_end(ap);
    return code;
}

ExlDevice* exl_device_state(int device)
{
    if (device < 0 || device >= EXL_MAX_DEVICES) { exl_set_err(EXL_ERR_ARG, "invalid device index %d", device); return nullptr; }
    ExlDevice* ds = &g_devices[device];
    if (ds->init) return ds;
    std::lock_guard<std::mutex> lock(g_mutex);
    if (ds->init) return ds;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || device >= count) {
        exl_set_err(EXL_ERR_CUDA, "no CUDA device %d available (%s); libexl_b200 has no CPU fallback", device,
                    e != cudaSuccess ? cudaGetErrorString(e) : "index out of range");
        cudaGetLastError();
        return nullptr;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { exl_set_err(EXL_ERR_CUDA, "cudaGetDeviceProperties failed"); return nullptr; }
    if (prop.major != 10) {
        exl_set_err(EXL_ERR_CUDA, "device %d is sm_%d%d; libexl_b200 is built for sm_100a (B200) only", device, prop.major, prop.minor);
        return nullptr;
    }
    DeviceGuard guard(device);
    ds->device = device;
    ds->num_sms = prop.multiProcessorCount;
    if (cublasCreate(&ds->blas) != CUBLAS_STATUS_SUCCESS) { exl_set_err(EXL_ERR_CUDA, "cublasCreate failed"); return nullptr; }
    cudaDeviceSynchronize();
    ds->init = true;
    return ds;
}

// library-owned scratch for callers that never called prepare_buffers (lazy; not CUDA-graph safe on first use)
int exl_own_scratch(ExlDevice* ds, int role, int64_t numel, half** out)
{
    if (ds->own_numel[role] < numel) {
        // growing = synchronize + cudaFree + cudaMalloc; during stream capture the synchronize fails and the error is returned
        // (call the op once eagerly, or prepare_buffers, before capturing a graph)
        if (ds->own[role]) { EXL_CUDA_TRY(cudaDeviceSynchronize()); cudaFree(ds->own[role]); }
        ds->own[role] = nullptr; ds->own_numel[role] = 0;
        EXL_CUDA_TRY(cudaMalloc(&ds->own[role], (size_t)numel * sizeof(half)));
        ds->own_numel[role] = numel;
    }
    *out = ds->own[role];
    return EXL_OK;
}

extern "C" {

const char* exl_last_error(void) { return t_err; }
int exl_version(void) { return 100; }
int64_t exl_launch_count(void) { return g_launches.load(); }
const char* exl_last_q4_path(void) { return g_last_q4_path; }
const char* exl_last_tc_config(void) { return g_last_tc_config; }
const char* exl_last_gemv_config(void) { return g_last_gemv_config[0] ? g_last_gemv_config : "none"; }

int exl_set_tuning_params(int matmul_recons_thd, int fused_mlp_thd, int sdp_thd, int matmul_fused_remap,
                          int rmsnorm_no_half2, int rope_no_half2, int matmul_no_half2, int silu_no_half2,
                          int concurrent_streams)
{
    g_tuning.matmul_recons_thd = matmul_recons_thd;
    g_tuning.fused_mlp_thd = fused_mlp_thd;
    g_tuning.sdp_thd = sdp_thd;
    g_tuning.matmul_fused_remap = matmul_fused_remap != 0;
    g_tuning.rmsnorm_no_half2 = rmsnorm_no_half2 != 0;
    g_tuning.rope_no_half2 = rope_no_half2 != 0;
    g_tuning.matmul_no_half2 = matmul_no_half2 != 0;
    g_tuning.silu_no_half2 = silu_no_half2 != 0;
    g_tuning.concurrent_streams = concurrent_streams != 0;
    return EXL_OK;
}

int exl_prepare_buffers(int device, void* temp_state, int64_t temp_state_numel, void* temp_mlp, int64_t temp_mlp_numel,
                        void* temp_zeros_float, int max_zeros_float, void* temp_dq, int64_t temp_dq_numel)
{
    ExlDevice* ds = exl_device_state(device);
    if (!ds) return EXL_ERR_CUDA;
    ds->temp_state = (half*)temp_state; ds->temp_state_numel = temp_state_numel;
    ds->temp_mlp = (half*)temp_mlp; ds->temp_mlp_numel = temp_mlp_numel;
    ds->temp_zeros_float = (float*)temp_zeros_float; ds->max_zeros_float = max_zeros_float;
    ds->temp_dq = (half*)temp_dq; ds->temp_dq_numel = temp_dq_numel;
    return EXL_OK;
}

int exl_cleanup(void)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    for (exl_q4_matrix* m : g_matrices) {
        if (m->x_map) { DeviceGuard guard(m->device); cudaFree(m->x_map); }   // (the reference leaks x_map, q4_matrix.cu:55-57)
        delete m;
    }
    g_matrices.clear();
    for (int i = 0; i < EXL_MAX_DEVICES; i++) {
        ExlDevice* ds = &g_devices[i];
        ds->temp_state = nullptr; ds->temp_mlp = nullptr; ds->temp_zeros_float = nullptr; ds->temp_dq = nullptr;
        ds->temp_state_numel = ds->temp_mlp_numel = ds->temp_dq_numel = 0; ds->max_zeros_float = 0;
        if (ds->tp_local) {
            // tensor-parallel workspace: unmap the peers' buffers, free our own (peers must have stopped launching)
            DeviceGuard guard(i);
            for (int p = 0; p < TP_MAX_RANKS; p++) {
                if (ds->tp_peers[p] && ds->tp_peers[p] != ds->tp_local) cudaIpcCloseMemHandle(ds->tp_peers[p]);
                ds->tp_peers[p] = nullptr;
            }
            cudaFree(ds->tp_local);
            ds->tp_local = nullptr; ds->tp_rank = 0; ds->tp_world = 1;
        }
    }
    return EXL_OK;
}

int exl_make_q4(void* qweight, void* qzeros, void* scales, const int32_t* g_idx_host, int K, int N, int groups,
                int device, void* stream_, exl_q4_matrix** out_handle)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!out_handle) return exl_set_err(EXL_ERR_ARG, "make_q4: out_handle is NULL");
    if (K <= 0 || N <= 0 || groups <= 0 || K % 8 != 0 || N % 8 != 0 || K % groups != 0)
        return exl_set_err(EXL_ERR_ARG, "make_q4: bad shape K=%d N=%d groups=%d", K, N, groups);
    ExlDevice* ds = exl_device_state(device);
    if (!ds) return EXL_ERR_CUDA;
    DeviceGuard guard(device);

    exl_q4_matrix* m = new exl_q4_matrix();
    m->device = device; m->K = K; m->N = N; m->groups = groups; m->groupsize = K / groups;
    m->qweight = (uint32_t*)qweight; m->qzeros = (uint32_t*)qzeros; m->scales = (half*)scales; m->x_map = nullptr;

    if (g_idx_host) {
        // Stable counting sort of rows by group: x_map[new_row] = old_row (semantics of q4_matrix.cu:110-139).
        std::vector<uint32_t> start((size_t)groups + 1, 0), x_map((size_t)K);
        for (int k = 0; k < K; k++) {
            const int32_t g = g_idx_host[k];
            if (g < 0 || g >= groups) { delete m; return exl_set_err(EXL_ERR_ARG, "make_q4: g_idx[%d]=%d out of range", k, g); }
            start[(size_t)g + 1]++;
        }
        for (int g = 0; g < groups; g++) start[(size_t)g + 1] += start[g];
        for (int k = 0; k < K; k++) x_map[start[g_idx_host[k]]++] = (uint32_t)k;

        uint32_t* tmp = nullptr;
        if (cudaMalloc(&m->x_map, (size_t)K * sizeof(uint32_t)) != cudaSuccess ||
            cudaMalloc(&tmp, (size_t)(K / 8) * N * sizeof(uint32_t)) != cudaSuccess) {
            delete m; return exl_set_err(EXL_ERR_CUDA, "make_q4: cudaMalloc failed");
        }
        cudaError_t ec = cudaMemcpyAsync(m->x_map, x_map.data(), (size_t)K * sizeof(uint32_t), cudaMemcpyHostToDevice, stream);
        int rc = ec == cudaSuccess ? exl_make_sequential_launch(m->qweight, tmp, m->x_map, K, N, stream)
                                   : exl_set_err(EXL_ERR_CUDA, "make_q4: x_map upload failed: %s", cudaGetErrorString(ec));
        cudaError_t e = cudaStreamSynchronize(stream);     // x_map (host vector) and tmp die here
        cudaFree(tmp);
        if (rc != EXL_OK || e != cudaSuccess) {
            cudaFree(m->x_map); delete m;
            return rc != EXL_OK ? rc : exl_set_err(EXL_ERR_CUDA, "make_q4: %s", cudaGetErrorString(e));
        }
    }
    if (int rc = exl_encode_weight_tmap(m)) { if (m->x_map) cudaFree(m->x_map); delete m; return rc; }
    {
        std::lock_guard<std::mutex> lock(g_mutex);
        g_matrices.push_back(m);
    }
    *out_handle = m;
    return EXL_OK;
}

int exl_q4_info(const exl_q4_matrix* w, int* K, int* N, int* groups, int* groupsize, int* has_x_map, int* device)
{
    if (!w) return exl_set_err(EXL_ERR_STATE, "q4_info: NULL handle");
    if (K) *K = w->K; if (N) *N = w->N; if (groups) *groups = w->groups; if (groupsize) *groupsize = w->groupsize;
    if (has_x_map) *has_x_map = w->x_map != nullptr; if (device) *device = w->device;
    return EXL_OK;
}

int exl_q4_get_x_map_host(const exl_q4_matrix* w, uint32_t* out_host)
{
    if (!w || !w->x_map) return exl_set_err(EXL_ERR_STATE, "q4_get_x_map: no x_map");
    DeviceGuard guard(w->device);
    EXL_CUDA_TRY(cudaMemcpy(out_host, w->x_map, (size_t)w->K * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return EXL_OK;
}

static int q4_matmul_recons_cublas(ExlDevice* ds, const half* x, int M, const exl_q4_matrix* w, half* out, bool no_zero, cudaStream_t stream)
{
    // reference prefill path: column_remap -> reconstruct -> Hgemm (q4_matmul.cu:301-344); kept as an explicit,
    // selectable GPU path (force_path = 3) and as the large-M route until the tcgen05 kernel covers a shape.
    const int64_t dq_numel = (int64_t)w->K * w->N;
    half* dq = ds->temp_dq_numel >= dq_numel ? ds->temp_dq : nullptr;
    half* xm = nullptr;
    const int64_t xm_numel = w->x_map ? (int64_t)M * w->K : 0;
    if (w->x_map && ds->temp_state_numel >= xm_numel) xm = ds->temp_state;
    if (!dq) { int rc = exl_own_scratch(ds, SCR_DQ, dq_numel, &dq); if (rc != EXL_OK) return rc; }
    if (w->x_map && !xm) { int rc = exl_own_scratch(ds, SCR_REMAP, xm_numel, &xm); if (rc != EXL_OK) return rc; }
    const half* xin = x;
    if (w->x_map) {
        int rc = exl_column_remap_launch(x, xm, M, w->K, w->x_map, stream);
        if (rc != EXL_OK) return rc;
        xin = xm;
    }
    int rc = exl_reconstruct_launch(w, dq, stream);
    if (rc != EXL_OK) return rc;
    return exl_half_matmul_cublas_launch(ds, xin, dq, out, M, w->K, w->N, no_zero, stream);
}

static int q4_matmul_dispatch(ExlDevice* ds, const half* x, int M, const exl_q4_matrix* w, half* out, bool no_zero,
                              int force_path, cudaStream_t stream)
{
    if (M <= 0) return EXL_OK;
    int path = force_path;
    // the skinny kernel streams 32-row x 32-column boxes and quantises x per 32 * 2^n-row group (q4_gemv.cu: exl_gemv_launch); any other
    // shape takes the general route (reconstruct + cuBLAS, the reference's own large-M path, q4_matmul.cu:301-344) instead of failing
    const int gs32 = w->groupsize / 32;
    const bool gemv_ok = w->K % 32 == 0 && w->N % 32 == 0 && (w->groups == 1 || (w->groupsize % 32 == 0 && (gs32 & (gs32 - 1)) == 0));
    if (path == 0 && !gemv_ok) path = 3;
    if (path == 0) {
        // M <= 8: one skinny pass.  8 < M <= 48: still HBM-bound, a few skinny passes (each re-streams the packed weights,
        // 0.5 B / weight) beat a tensor-core tile that is mostly padding.  Above: tcgen05 fused-dequant GEMM.
        if (M <= EXL_SKINNY_MAX_M) path = 1;
        else if (M <= 48 || !exl_tc_gemm_supported(w, M)) path = (M <= 64) ? 1 : 3;
        else path = 2;
    }
    if (path == 1) {
        g_last_q4_path = "skinny_mma";
        for (int m0 = 0; m0 < M; m0 += GV_MAXM) {
            const int mc = (M - m0 < GV_MAXM) ? (M - m0) : GV_MAXM;
            half* o = out + (size_t)m0 * w->N;
            int rc = exl_gemv_launch(ds, x + (size_t)m0 * w->K, mc, &w, &o, 1, no_zero, GV_PRO_PLAIN, GV_EPI_STORE, nullptr, stream);
            if (rc != EXL_OK) return rc;
        }
        return EXL_OK;
    }
    if (path == 2) {
        g_last_q4_path = "tc_gemm";
        return exl_tc_gemm_launch(ds, x, M, w, out, no_zero, stream);
    }
    if (path == 3) {
        g_last_q4_path = "recons_cublas";
        return q4_matmul_recons_cublas(ds, x, M, w, out, no_zero, stream);
    }
    return exl_set_err(EXL_ERR_ARG, "q4_matmul: bad force_path %d", force_path);
}

int exl_q4_matmul(const void* x, int M, const exl_q4_matrix* w, void* out, int no_zero, int force_path, void* stream)
{
    g_last_gemv_config[0] = 0;
    if (!w) return exl_set_err(EXL_ERR_STATE, "q4_matmul: NULL handle");
    ExlDevice* ds = exl_device_state(w->device);
    if (!ds) return EXL_ERR_CUDA;
    DeviceGuard guard(w->device);
    return q4_matmul_dispatch(ds, (const half*)x, M, w, (half*)out, no_zero != 0, force_path, (cudaStream_t)stream);
}

int exl_q4_reconstruct(const exl_q4_matrix* w, void* out, void* stream)
{
    if (!w) return exl_set_err(EXL_ERR_STATE, "q4_reconstruct: NULL handle");
    if (!exl_device_state(w->device)) return EXL_ERR_CUDA;
    DeviceGuard guard(w->device);
    return exl_reconstruct_launch(w, (half*)out, (cudaStream_t)stream);
}

int exl_q4_matmul_lora(const void* x, int M, const exl_q4_matrix* w, void* out, const void* lora_A, const void* lora_B,
                       int rank, void* lora_temp, void* stream_)
{
    g_last_gemv_config[0] = 0;
    if (!w) return exl_set_err(EXL_ERR_STATE, "q4_matmul_lora: NULL handle");
    ExlDevice* ds = exl_device_state(w->device);
    if (!ds) return EXL_ERR_CUDA;
    DeviceGuard guard(w->device);
    cudaStream_t stream = (cudaStream_t)stream_;
    // lora_temp = x @ A; out = lora_temp @ B; out += x @ W   (exllama_ext.cpp:269-323)
    int rc = exl_half_matmul_cublas_launch(ds, (const half*)x, (const half*)lora_A, (half*)lora_temp, M, w->K, rank, false, stream);
    if (rc != EXL_OK) return rc;
    rc = exl_half_matmul_cublas_launch(ds, (const half*)lora_temp, (const half*)lora_B, (half*)out, M, rank, w->N, false, stream);
    if (rc != EXL_OK) return rc;
    return q4_matmul_dispatch(ds, (const half*)x, M, w, (half*)out, true, 0, stream);
}

int exl_column_remap(const void* x, void* x_new, int M, int K, const uint32_t* x_map, void* stream)
{
    return exl_column_remap_launch((const half*)x, (half*)x_new, M, K, x_map, (cudaStream_t)stream);
}

int exl_half_matmul(const void* x, const void* w, void* out, int M, int K, int N, void* stream)
{
    return exl_half_matmul_custom_launch((const half*)x, (const half*)w, (half*)out, M, K, N, (cudaStream_t)stream);
}

int exl_half_matmul_cublas(const void* x, const void* w, void* out, int M, int K, int N, int no_zero, void* stream)
{
    int dev = 0; cudaGetDevice(&dev);
    ExlDevice* ds = exl_device_state(dev);
    if (!ds) return EXL_ERR_CUDA;
    return exl_half_matmul_cublas_launch(ds, (const half*)x, (const half*)w, (half*)out, M, K, N, no_zero != 0, (cudaStream_t)stream);
}

int exl_rms_norm(const void* x, const void* w, void* out, float epsilon, int rows, int dim, int device, void* stream)
{
    if (!exl_device_state(device)) return EXL_ERR_CUDA;
    DeviceGuard guard(device);
    return exl_rms_norm_launch((const half*)x, (const half*)w, (half*)out, epsilon, rows, dim, (cudaStream_t)stream);
}

int exl_rope(void* x, const void* sin, const void* cos, int bsz, int rows_per_batch, int head_dim, int num_heads,
             int past_len, void* stream)
{
    return exl_rope_launch((half*)x, (const half*)sin, (const half*)cos, bsz, rows_per_batch, head_dim, num_heads, past_len, (cudaStream_t)stream);
}

int exl_silu_mul(void* x, const void* y, int height, int width, void* stream)
{
    return exl_silu_mul_launch((half*)x, (const half*)y, height, width, (cudaStream_t)stream);
}

int exl_update_cache(const void* key_states, const void* value_states, void* key_cache, void* value_cache,
                     int head_dim, int num_kv_heads, int q_len, int max_seq_len, int past_len, void* stream)
{
    return exl_update_cache_launch((const half*)key_states, (const half*)value_states, (half*)key_cache, (half*)value_cache,
                                   head_dim, num_kv_heads, q_len, max_seq_len, past_len, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------------------
// fused decoder blocks
// ---------------------------------------------------------------------------------------------------------

int exl_q4_attn(void* x_, const void* rms_norm_weight, float epsilon, void* query_states, void* key_states, void* value_states,
                const exl_q4_matrix* q_proj, const exl_q4_matrix* k_proj, const exl_q4_matrix* v_proj,
                const void* sin, const void* cos, int bsz, int q_len, int dim, int head_dim, int num_heads,
                int num_kv_heads, int past_len, void* key_cache, void* value_cache, int max_seq_len,
                const void* q_a, const void* q_b, int q_rank, const void* k_a, const void* k_b, int k_rank,
                const void* v_a, const void* v_b, int v_rank, void* lora_temp, int device, void* stream_)
{
    g_last_gemv_config[0] = 0;
    if (!q_proj || !k_proj || !v_proj) return exl_set_err(EXL_ERR_STATE, "q4_attn: NULL handle");
    ExlDevice* ds = exl_device_state(device);
    if (!ds) return EXL_ERR_CUDA;
    DeviceGuard guard(device);
    cudaStream_t stream = (cudaStream_t)stream_;
    half* x = (half*)x_;
    const int rows = bsz * q_len;
    const bool lora = q_rank || k_rank || v_rank;

    // Single-launch path: RMS norm folded into the x staging, q/k/v as one stream-K work list, RoPE and the
    // KV-cache write folded into the epilogue (replaces 8 launches of q4_attn_cuda, q4_attn.cu:130-165).
    if (!lora && bsz == 1 && rows <= GV_MAXM && head_dim == GV_TILE_N &&
        q_proj->x_map == k_proj->x_map && q_proj->x_map == v_proj->x_map &&
        q_proj->groups == k_proj->groups && q_proj->groups == v_proj->groups) {
        const exl_q4_matrix* mats[3] = {q_proj, k_proj, v_proj};
        half* outs[3] = {(half*)query_states, (half*)key_states, (half*)value_states};
        GemvFused f;
        f.norm_w = (const half*)rms_norm_weight; f.eps = epsilon;
        f.sin = (const half*)sin; f.cos = (const half*)cos; f.head_dim = head_dim; f.num_heads = num_heads;
        f.num_kv_heads = num_kv_heads; f.past_len = past_len; f.max_seq_len = max_seq_len; f.q_len = q_len;
        f.key_cache = (half*)key_cache; f.value_cache = (half*)value_cache;
        return exl_gemv_launch(ds, x, rows, mats, outs, 3, false, GV_PRO_RMSNORM, GV_EPI_ROPE_CACHE, &f, stream);
    }

    // General path (LoRA, act-order with distinct x_maps, other head sizes): same sequence as q4_attn_cuda.
    // The hidden width is the projections' K, not the caller's `dim` (= query_states.size(2), exllama_ext.cpp:470): under
    // tensor parallelism the query width is hidden / tp while x, the norm and the q/k/v inputs are hidden wide.
    const int hid = q_proj->K;
    if (k_proj->K != hid || v_proj->K != hid) return exl_set_err(EXL_ERR_ARG, "q4_attn: q/k/v projections disagree on the input width");
    (void)dim;
    half* temp_x;
    if (ds->temp_state && ds->temp_state_numel >= 2 * (int64_t)rows * hid) temp_x = ds->temp_state + (size_t)rows * hid;
    else { int rc = exl_own_scratch(ds, SCR_NORM, (int64_t)rows * hid, &temp_x); if (rc != EXL_OK) return rc; }
    int rc = exl_rms_norm_launch(x, (const half*)rms_norm_weight, temp_x, epsilon, rows, hid, stream);
    if (rc != EXL_OK) return rc;
    struct P { const exl_q4_matrix* w; half* out; const void* a; const void* b; int rank; };
    P proj[3] = {{q_proj, (half*)query_states, q_a, q_b, q_rank}, {k_proj, (half*)key_states, k_a, k_b, k_rank},
                 {v_proj, (half*)value_states, v_a, v_b, v_rank}};
    for (int i = 0; i < 3; i++) {
        if (proj[i].rank) {
            rc = exl_half_matmul_cublas_launch(ds, temp_x, (const half*)proj[i].a, (half*)lora_temp, rows, hid, proj[i].rank, false, stream);
            if (rc != EXL_OK) return rc;
            rc = exl_half_matmul_cublas_launch(ds, (const half*)lora_temp, (const half*)proj[i].b, proj[i].out, rows, proj[i].rank, proj[i].w->N, false, stream);
            if (rc != EXL_OK) return rc;
        }
        rc = q4_matmul_dispatch(ds, temp_x, rows, proj[i].w, proj[i].out, proj[i].rank != 0, 0, stream);
        if (rc != EXL_OK) return rc;
    }
    rc = exl_rope_launch((half*)query_states, (const half*)sin, (const half*)cos, bsz, q_len * num_heads, head_dim, num_heads, past_len, stream);
    if (rc != EXL_OK) return rc;
    rc = exl_rope_launch((half*)key_states, (const half*)sin, (const half*)cos, bsz, q_len * num_kv_heads, head_dim, num_kv_heads, past_len, stream);
    if (rc != EXL_OK) return rc;
    return exl_update_cache_launch((const half*)key_states, (const half*)value_states, (half*)key_cache, (half*)value_cache,
                                   head_dim, num_kv_heads, q_len, max_seq_len, past_len, stream);
}

int exl_q4_attn_2(void* x, const void* attn_output, const exl_q4_matrix* o_proj, int height,
                  const void* o_a, const void* o_b, int o_rank, void* lora_temp, void* stream_)
{
    g_last_gemv_config[0] = 0;
    if (!o_proj) return exl_set_err(EXL_ERR_STATE, "q4_attn_2: NULL handle");
    ExlDevice* ds = exl_device_state(o_proj->device);
    if (!ds) return EXL_ERR_CUDA;
    DeviceGuard guard(o_proj->device);
    cudaStream_t stream = (cudaStream_t)stream_;
    if (o_rank) {
        int rc = exl_half_matmul_cublas_launch(ds, (const half*)attn_output, (const half*)o_a, (half*)lora_temp, height, o_proj->K, o_rank, false, stream);
        if (rc != EXL_OK) return rc;
        rc = exl_half_matmul_cublas_launch(ds, (const half*)lora_temp, (const half*)o_b, (half*)x, height, o_rank, o_proj->N, true, stream);
        if (rc != EXL_OK) return rc;
    }
    return q4_matmul_dispatch(ds, (const half*)attn_output, height, o_proj, (half*)x, true, 0, stream);
}

static int q4_mlp_impl(void* x_, const void* rms_norm_weight, float epsilon, const exl_q4_matrix* gate, const exl_q4_matrix* up,
               const exl_q4_matrix* down, int height, int dim, const void* gate_a, const void* gate_b, int gate_rank,
               const void* up_a, const void* up_b, int up_rank, const void* down_a, const void* down_b, int down_rank,
               void* lora_temp, int device, void* stream_, bool add_residual, bool all_reduce = false)
{
    g_last_gemv_config[0] = 0;
    if (!gate || !up || !down) return exl_set_err(EXL_ERR_STATE, "q4_mlp: NULL handle");
    ExlDevice* ds = exl_device_state(device);
    if (!ds) return EXL_ERR_CUDA;
    DeviceGuard guard(device);
    cudaStream_t stream = (cudaStream_t)stream_;
    half* x = (half*)x_;
    const int inter = up->N;
    const bool lora = gate_rank || up_rank || down_rank;

    // activation scratch [2, height, inter]: borrowed temp_mlp when it is known to be big enough, else owned
    half* temp_mlp = nullptr;
    const int64_t mlp_numel = 2 * (int64_t)height * inter;
    const bool have_norm = ds->temp_state && ds->temp_state_numel >= 2 * (int64_t)height * dim;
    if (ds->temp_mlp && ds->temp_mlp_numel >= mlp_numel) temp_mlp = ds->temp_mlp;
    if (!temp_mlp) { int rc = exl_own_scratch(ds, SCR_MLP, mlp_numel, &temp_mlp); if (rc != EXL_OK) return rc; }

    if (!lora && height <= GV_MAXM && gate->x_map == up->x_map && gate->N == up->N && gate->groups == up->groups) {
        // two launches instead of six (q4_mlp.cu:118-197): [norm -> gate,up -> silu*mul], [down += residual]
        const exl_q4_matrix* mats[2] = {gate, up};
        half* outs[2] = {temp_mlp, temp_mlp};
        GemvFused f; f.norm_w = (const half*)rms_norm_weight; f.eps = epsilon;
        int rc = exl_gemv_launch(ds, x, height, mats, outs, 2, false, GV_PRO_RMSNORM, GV_EPI_SILU_MUL, &f, stream);
        if (rc != EXL_OK) return rc;
        if (all_reduce) {
            half* o = x;
            return exl_gemv_launch(ds, temp_mlp, height, &down, &o, 1, true, GV_PRO_PLAIN, GV_EPI_ALLREDUCE, nullptr, stream);
        }
        return q4_matmul_dispatch(ds, temp_mlp, height, down, x, add_residual, 0, stream);
    }
    if (all_reduce) return exl_set_err(EXL_ERR_ARG, "q4_mlp_ar: only the fused decode configuration (rows <= 8, no act-order mismatch) is supported");

    half* temp_x = have_norm ? ds->temp_state + (size_t)height * dim : nullptr;
    if (!temp_x) { int rc = exl_own_scratch(ds, SCR_NORM, (int64_t)height * dim, &temp_x); if (rc != EXL_OK) return rc; }
    half* t0 = temp_mlp; half* t1 = temp_mlp + (size_t)height * inter;
    int rc = exl_rms_norm_launch(x, (const half*)rms_norm_weight, temp_x, epsilon, height, dim, stream);
    if (rc != EXL_OK) return rc;
    if (gate_rank) {
        rc = exl_half_matmul_cublas_launch(ds, temp_x, (const half*)gate_a, (half*)lora_temp, height, dim, gate_rank, false, stream); if (rc) return rc;
        rc = exl_half_matmul_cublas_launch(ds, (const half*)lora_temp, (const half*)gate_b, t0, height, gate_rank, inter, false, stream); if (rc) return rc;
    }
    if (up_rank) {
        rc = exl_half_matmul_cublas_launch(ds, temp_x, (const half*)up_a, (half*)lora_temp, height, dim, up_rank, false, stream); if (rc) return rc;
        rc = exl_half_matmul_cublas_launch(ds, (const half*)lora_temp, (const half*)up_b, t1, height, up_rank, inter, false, stream); if (rc) return rc;
    }
    rc = q4_matmul_dispatch(ds, temp_x, height, gate, t0, gate_rank != 0, 0, stream); if (rc) return rc;
    rc = q4_matmul_dispatch(ds, temp_x, height, up, t1, up_rank != 0, 0, stream); if (rc) return rc;
    rc = exl_silu_mul_launch(t0, t1, height, inter, stream); if (rc) return rc;
    if (down_rank) {
        rc = exl_half_matmul_cublas_launch(ds, t0, (const half*)down_a, (half*)lora_temp, height, inter, down_rank, false, stream); if (rc) return rc;
        rc = exl_half_matmul_cublas_launch(ds, (const half*)lora_temp, (const half*)down_b, x, height, down_rank, dim, true, stream); if (rc) return rc;
    }
    return q4_matmul_dispatch(ds, t0, height, down, x, add_residual || down_rank != 0, 0, stream);
}

int exl_q4_mlp(void* x_, const void* rms_norm_weight, float epsilon, const exl_q4_matrix* gate, const exl_q4_matrix* up,
               const exl_q4_matrix* down, int height, int dim, const void* gate_a, const void* gate_b, int gate_rank,
               const void* up_a, const void* up_b, int up_rank, const void* down_a, const void* down_b, int down_rank,
               void* lora_temp, int device, void* stream_)
{
    return q4_mlp_impl(x_, rms_norm_weight, epsilon, gate, up, down, height, dim, gate_a, gate_b, gate_rank, up_a, up_b, up_rank,
                       down_a, down_b, down_rank, lora_temp, device, stream_, true);
}

int exl_q4_mlp_tp(void* x, const void* rms_norm_weight, float epsilon, const exl_q4_matrix* gate, const exl_q4_matrix* up,
                  const exl_q4_matrix* down, int height, int dim, int add_residual, int device, void* stream)
{
    return q4_mlp_impl(x, rms_norm_weight, epsilon, gate, up, down, height, dim, nullptr, nullptr, 0, nullptr, nullptr, 0,
                       nullptr, nullptr, 0, nullptr, device, stream, add_residual != 0);
}

int exl_q4_mlp_ar(void* x, const void* rms_norm_weight, float epsilon, const exl_q4_matrix* gate, const exl_q4_matrix* up,
                  const exl_q4_matrix* down, int height, int dim, int device, void* stream)
{
    return q4_mlp_impl(x, rms_norm_weight, epsilon, gate, up, down, height, dim, nullptr, nullptr, 0, nullptr, nullptr, 0,
                       nullptr, nullptr, 0, nullptr, device, stream, true, true);
}

int exl_q4_attn_2_ar(void* x, const void* attn_output, const exl_q4_matrix* o_proj, int height, void* stream)
{
    g_last_gemv_config[0] = 0;
    if (!o_proj) return exl_set_err(EXL_ERR_STATE, "q4_attn_2_ar: NULL handle");
    ExlDevice* ds = exl_device_state(o_proj->device);
    if (!ds) return EXL_ERR_CUDA;
    if (height > GV_MAXM) return exl_set_err(EXL_ERR_ARG, "q4_attn_2_ar: rows %d > %d", height, GV_MAXM);
    DeviceGuard guard(o_proj->device);
    half* o = (half*)x;
    return exl_gemv_launch(ds, (const half*)attn_output, height, &o_proj, &o, 1, true, GV_PRO_PLAIN, GV_EPI_ALLREDUCE, nullptr, (cudaStream_t)stream);
}

int exl_tp_workspace_alloc(int device, void** local_ptr, void* ipc_handle)
{
    ExlDevice* ds = exl_device_state(device);
    if (!ds) return EXL_ERR_CUDA;
    DeviceGuard guard(device);
    if (!ds->tp_local) {
        EXL_CUDA_TRY(cudaMalloc(&ds->tp_local, TP_WS_BYTES));
        EXL_CUDA_TRY(cudaMemset(ds->tp_local, 0, TP_WS_BYTES));
        EXL_CUDA_TRY(cudaDeviceSynchronize());
    }
    cudaIpcMemHandle_t h;
    EXL_CUDA_TRY(cudaIpcGetMemHandle(&h, ds->tp_local));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ipc handle size");
    memcpy(ipc_handle, &h, 64);
    *local_ptr = ds->tp_local;
    return EXL_OK;
}

int exl_tp_workspace_open(int device, const void* ipc_handle, void** peer_ptr)
{
    if (!exl_device_state(device)) return EXL_ERR_CUDA;
    DeviceGuard guard(device);
    cudaIpcMemHandle_t h;
    memcpy(&h, ipc_handle, 64);
    EXL_CUDA_TRY(cudaIpcOpenMemHandle(peer_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return EXL_OK;
}

int exl_tp_init(int device, int rank, int world, void* const* workspace_ptrs)
{
    ExlDevice* ds = exl_device_state(device);
    if (!ds) return EXL_ERR_CUDA;
    if (world < 1 || world > TP_MAX_RANKS || rank < 0 || rank >= world) return exl_set_err(EXL_ERR_ARG, "tp_init: bad rank %d / world %d", rank, world);
    if (!ds->tp_local || workspace_ptrs[rank] != ds->tp_local) return exl_set_err(EXL_ERR_STATE, "tp_init: own workspace entry must be the pointer from exl_tp_workspace_alloc");
    ds->tp_rank = rank; ds->tp_world = world;
    for (int i = 0; i < TP_MAX_RANKS; i++) ds->tp_peers[i] = i < world ? (unsigned char*)workspace_ptrs[i] : nullptr;
    return EXL_OK;
}

int exl_tp_status(int device, unsigned* timeouts)
{
    ExlDevice* ds = exl_device_state(device);
    if (!ds) return EXL_ERR_CUDA;
    if (!ds->tp_local) return exl_set_err(EXL_ERR_STATE, "tp_status: no workspace on device %d", device);
    DeviceGuard guard(device);
    EXL_CUDA_TRY(cudaMemcpy(timeouts, ds->tp_local + TP_DATA_BYTES + TP_FLAG_BYTES + 2 * sizeof(unsigned), sizeof(unsigned), cudaMemcpyDeviceToHost));
    return EXL_OK;
}

int exl_q4_attn_2_tp(void* x, const void* attn_output, const exl_q4_matrix* o_proj, int height, int add_residual, void* stream)
{
    g_last_gemv_config[0] = 0;
    if (!o_proj) return exl_set_err(EXL_ERR_STATE, "q4_attn_2_tp: NULL handle");
    ExlDevice* ds = exl_device_state(o_proj->device);
    if (!ds) return EXL_ERR_CUDA;
    DeviceGuard guard(o_proj->device);
    return q4_matmul_dispatch(ds, (const half*)attn_output, height, o_proj, (half*)x, add_residual != 0, 0, (cudaStream_t)stream);
}

int exl_decode_attn(const void* q, const void* key_cache, const void* value_cache, void* out, int num_heads, int num_kv_heads,
                    int head_dim, int seq_len, int max_seq_len, void* stream)
{
    return exl_decode_attn_launch((const half*)q, (const half*)key_cache, (const half*)value_cache, (half*)out, num_heads, num_kv_heads,
                                  head_dim, seq_len, max_seq_len, 1.0f / sqrtf((float)head_dim), (cudaStream_t)stream);
}

int exl_q4_matmul_host(const void* x_host, int M, const exl_q4_matrix* w, void* out_host, void* d_x, void* d_out, void* stream_)
{
    g_last_gemv_config[0] = 0;
    if (!w) return exl_set_err(EXL_ERR_STATE, "q4_matmul_host: NULL handle");
    ExlDevice* ds = exl_device_state(w->device);
    if (!ds) return EXL_ERR_CUDA;
    DeviceGuard guard(w->device);
    cudaStream_t stream = (cudaStream_t)stream_;
    EXL_CUDA_TRY(cudaMemcpyAsync(d_x, x_host, (size_t)M * w->K * sizeof(half), cudaMemcpyHostToDevice, stream));
    int rc = q4_matmul_dispatch(ds, (const half*)d_x, M, w, (half*)d_out, false, 0, stream);
    if (rc != EXL_OK) return rc;
    EXL_CUDA_TRY(cudaMemcpyAsync(out_host, d_out, (size_t)M * w->N * sizeof(half), cudaMemcpyDeviceToHost, stream));
    EXL_CUDA_TRY(cudaStreamSynchronize(stream));
    return EXL_OK;
}

// ---------------------------------------------------------------------------------------------------------
// repetition penalty (host; cpu_func/rep_penalty.cpp).  Sampling helper, not a performance path.
// ---------------------------------------------------------------------------------------------------------

int exl_rep_penalty(int vocab_size, const uint64_t* seq, float* rep_mask, float penalty_max, int sustain, int decay, int seq_len)
{
    // newest token gets penalty_max for `sustain` tokens, then the penalty decays linearly to 1 over `decay` tokens
    for (int i = 0; i < vocab_size; i++) rep_mask[i] = 1.0f;
    const float step = decay ? (1.0f - penalty_max) / (float)decay : 0.0f;
    int hold = sustain == -1 ? seq_len : sustain;
    int first = seq_len - hold - decay;
    if (first < 0) first = 0;
    float p = penalty_max;
    for (int i = seq_len - 1; i >= first; i--) {
        const uint64_t tok = seq[i];
        if (tok >= (uint64_t)vocab_size) return exl_set_err(EXL_ERR_ARG, "rep_penalty: token %llu outside vocabulary", (unsigned long long)tok);
        if (p > rep_mask[tok]) rep_mask[tok] = p;
        if (--hold < 0) p += step;
    }
    return EXL_OK;
}

int exl_apply_rep_penalty(int vocab_size, const uint64_t* seq, float penalty_max, int sustain, int decay, int seq_len, float* logits)
{
    std::vector<unsigned char> seen((size_t)vocab_size, 0);
    const float step = decay ? (1.0f - penalty_max) / (float)decay : 0.0f;
    int hold = sustain == -1 ? seq_len : sustain;
    int first = seq_len - hold - decay;
    if (first < 0) first = 0;
    float p = penalty_max;
    for (int i = seq_len - 1; i >= first; i--) {
        const uint64_t tok = seq[i];
        if (tok >= (uint64_t)vocab_size) return exl_set_err(EXL_ERR_ARG, "apply_rep_penalty: token %llu outside vocabulary", (unsigned long long)tok);
        if (!seen[tok]) {
            if (logits[tok] > 0.0f) logits[tok] /= p; else logits[tok] *= p;
            seen[tok] = 1;
        }
        if (--hold < 0) p += step;
    }
    return EXL_OK;
}

} // extern "C"
