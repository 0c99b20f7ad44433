/*
 * exl_b200.h -- C ABI of libexl_b200.so: the B200 (sm_100a) implementation of the
 * exllama_ext operator surface (GPTQ 4-bit matmul + the fused Llama ops around it).
 *
 * Drop-in boundary.  The reference binds this path as a torch C++ extension
 * (pybind11 module `exllama_ext`, /root/reference/exllama_ext/exllama_ext.cpp:743-762,
 * loaded by cuda_ext.py:43-64).  Every entry point below is what one of those 16
 * pybind functions needs underneath once the torch::Tensor arguments are
 * reduced to raw pointers and sizes; the citation on each declaration is the
 * reference function it replaces.  exllama_b200/csrc/pybind_shim.cpp is the
 * reference-side binding (same 16 names, same signatures); INTEGRATION.md shows it.
 *
 * Conventions
 *  - plain C: pointers, ints, floats.  No torch / C++ types.
 *  - all `half` data is IEEE binary16, passed as void*.
 *  - device pointers unless the name says `_host`.
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *    The reference launches on the legacy default stream; the shim passes
 *    at::cuda::getCurrentCUDAStream().
 *  - return value: 0 on success, non-zero error code otherwise;
 *    exl_last_error() returns a human-readable message for the calling thread.
 *  - like the reference, the library keeps global per-process state (tuning,
 *    per-device scratch, handle list) and is not re-entrant across host threads.
 *  - there is NO CPU fallback anywhere: if no sm_100 device is present the
 *    compute entry points fail with EXL_ERR_CUDA.
 */
#ifndef EXL_B200_H
#define EXL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EXL_OK            0
#define EXL_ERR_ARG       1   /* bad shape / unsupported configuration */
#define EXL_ERR_CUDA      2   /* CUDA runtime / launch error */
#define EXL_ERR_STATE     3   /* missing prepare_buffers / bad handle */

#define EXL_MAX_DEVICES   16  /* cuda_buffers.cuh:9 */

typedef struct exl_q4_matrix exl_q4_matrix;   /* opaque; reference: class Q4Matrix, q4_matrix.cuh:8-46 */

const char* exl_last_error(void);
int exl_version(void);

/* --- tuning / buffers ------------------------------------------------------ */

/* exllama_ext.cpp:89-112 set_tuning_params.  The *_no_half2 and concurrent_streams
   flags are accepted and stored for API compatibility; the sm_100a kernels have a
   single code path (fp32 accumulation) and fuse what concurrent_streams overlapped. */
int exl_set_tuning_params(int matmul_recons_thd, int fused_mlp_thd, int sdp_thd, int matmul_fused_remap,
                          int rmsnorm_no_half2, int rope_no_half2, int matmul_no_half2, int silu_no_half2,
                          int concurrent_streams);

/* exllama_ext.cpp:126-152 prepare_buffers / cuda_buffers.cu:66-89.  Borrowed scratch:
   temp_state half[temp_state_numel], temp_mlp half[temp_mlp_numel], temp_zeros_float float[max_zeros_float],
   temp_dq half[temp_dq_numel].  (The reference passes no size for temp_mlp/temp_dq; pass 0 for "unknown".) */
int exl_prepare_buffers(int device, void* temp_state, int64_t temp_state_numel,
                        void* temp_mlp, int64_t temp_mlp_numel,
                        void* temp_zeros_float, int max_zeros_float,
                        void* temp_dq, int64_t temp_dq_numel);

/* exllama_ext.cpp:117-121 cleanup: frees every Q4 handle and per-device scratch. */
int exl_cleanup(void);

/* --- Q4 matrix --------------------------------------------------------------- */

/* exllama_ext.cpp:157-194 make_q4 + q4_matrix.cu:26-53,104-168.
   qweight int32 [K/8, N], qzeros int32 [groups, N/8], scales half [groups, N] are BORROWED device memory.
   g_idx_host: int32 [K] on the host, or NULL.  When given, the rows of qweight are re-ordered by group
   IN PLACE in the caller's buffer (as the reference does) and the library keeps x_map[K] on the device. */
int exl_make_q4(void* qweight, void* qzeros, void* scales, const int32_t* g_idx_host,
                int K, int N, int groups, int device, void* stream, exl_q4_matrix** out_handle);

int exl_q4_info(const exl_q4_matrix* w, int* K, int* N, int* groups, int* groupsize, int* has_x_map, int* device);
/* copies the device x_map (uint32 [K]) to the host; for tests */
int exl_q4_get_x_map_host(const exl_q4_matrix* w, uint32_t* out_host);

/* exllama_ext.cpp:199-240 q4_matmul: out[M,N] (=|+=) x[M,K] . W.  no_zero != 0 accumulates into out
   (q4_matmul.cu:78-82).  Dispatch: skinny-M fused unpack+GEMV kernel for M <= EXL_SKINNY_MAX_M, tensor-core
   (tcgen05) fused-dequant GEMM above. force_path: 0 auto, 1 skinny, 2 tensor-core GEMM, 3 reconstruct+cuBLAS. */
int exl_q4_matmul(const void* x, int M, const exl_q4_matrix* w, void* out, int no_zero, int force_path, void* stream);

/* q4_matrix.cu:212-223 Q4Matrix::reconstruct: out half [K, N] = dequantised W (bit-exact with the reference). */
int exl_q4_reconstruct(const exl_q4_matrix* w, void* out, void* stream);

/* exllama_ext.cpp:245-324 q4_matmul_lora: out = (x.A).B + x.W;  lora_temp half [M, rank]. */
int exl_q4_matmul_lora(const void* x, int M, const exl_q4_matrix* w, void* out,
                       const void* lora_A, const void* lora_B, int rank, void* lora_temp, void* stream);

/* exllama_ext.cpp:328-355 column_remap: x_new[m,i] = x[m, x_map[i]] */
int exl_column_remap(const void* x, void* x_new, int M, int K, const uint32_t* x_map, void* stream);

/* --- fp16 matmul ------------------------------------------------------------- */

/* exllama_ext.cpp:359-386 half_matmul (custom kernel; the reference requires a pre-zeroed out and
   accumulates, half_matmul.cu:15-54): out[M,N] += x[M,K] . w[K,N] */
int exl_half_matmul(const void* x, const void* w, void* out, int M, int K, int N, void* stream);
/* exllama_ext.cpp:390-420 half_matmul_cublas: out = x.w (no_zero: out += x.w), half_matmul.cu:83-125 */
int exl_half_matmul_cublas(const void* x, const void* w, void* out, int M, int K, int N, int no_zero, void* stream);

/* --- small fused ops --------------------------------------------------------- */

/* exllama_ext.cpp:606-641 rms_norm / rms_norm.cu:178-213. out may alias x. */
int exl_rms_norm(const void* x, const void* w, void* out, float epsilon, int rows, int dim, int device, void* stream);

/* exllama_ext.cpp:645-678 rope_ / rope.cu:100-125, in place.
   x half [bsz, rows_per_batch, head_dim], sin/cos half [max_seq, head_dim]. */
int exl_rope(void* x, const void* sin, const void* cos, int bsz, int rows_per_batch, int head_dim,
             int num_heads, int past_len, void* stream);

/* q4_mlp.cu:46-88 silu_mul: x = silu(x) * y, elementwise over [height, width] */
int exl_silu_mul(void* x, const void* y, int height, int width, void* stream);

/* q4_attn.cu:19-72 update_cache: cache[h, past_len + t, :] = states[t, h, :] */
int exl_update_cache(const void* key_states, const void* value_states, void* key_cache, void* value_cache,
                     int head_dim, int num_kv_heads, int q_len, int max_seq_len, int past_len, void* stream);

/* --- fused decoder blocks (decode path) --------------------------------------- */

/* exllama_ext.cpp:424-509 q4_attn / q4_attn.cu:74-204:
   rms_norm(x) -> q,k,v projections -> RoPE(q,k) -> write k,v into the cache at past_len.
   LoRA pointers may be NULL (rank 0). */
int exl_q4_attn(void* x, const void* rms_norm_weight, float epsilon,
                void* query_states, void* key_states, void* value_states,
                const exl_q4_matrix* q_proj, const exl_q4_matrix* k_proj, const exl_q4_matrix* v_proj,
                const void* sin, const void* cos,
                int bsz, int q_len, int dim, int head_dim, int num_heads, int num_kv_heads, int past_len,
                void* key_cache, void* value_cache, int max_seq_len,
                const void* q_a, const void* q_b, int q_rank,
                const void* k_a, const void* k_b, int k_rank,
                const void* v_a, const void* v_b, int v_rank,
                void* lora_temp, int device, void* stream);

/* exllama_ext.cpp:511-542 q4_attn_2 / q4_attn.cu:206-228: x += attn_output . o_proj (+ LoRA) */
int exl_q4_attn_2(void* x, const void* attn_output, const exl_q4_matrix* o_proj, int height,
                  const void* o_a, const void* o_b, int o_rank, void* lora_temp, void* stream);

/* exllama_ext.cpp:546-602 q4_mlp / q4_mlp.cu:100-199:
   x += down( silu(gate(norm(x))) * up(norm(x)) ) */
int exl_q4_mlp(void* x, const void* rms_norm_weight, float epsilon,
               const exl_q4_matrix* gate, const exl_q4_matrix* up, const exl_q4_matrix* down,
               int height, int dim,
               const void* gate_a, const void* gate_b, int gate_rank,
               const void* up_a, const void* up_b, int up_rank,
               const void* down_a, const void* down_b, int down_rank,
               void* lora_temp, int device, void* stream);

/* --- decode attention (SURVEY.md 8f-1: the ranked-first "next" row; not part of the reference's extension) ------------ */

/* Single-query attention over the KV cache, replacing the torch ops of ExLlamaAttention.fused (model.py:372-409):
   out[h, :] = softmax(q[h] . K[kvh(h), 0:seq]^T / sqrt(head_dim)) . V[kvh(h), 0:seq]      (fp32 arithmetic, fp16 in/out)
   q, out: half [num_heads * head_dim] (one token); caches: half [num_kv_heads, max_seq_len, head_dim]; head_dim == 128.
   Ordering precondition (programmatic dependent launch): the kernel loads cache rows 0 .. seq_len-2 BEFORE it waits for
   the kernel launched immediately before it on `stream` (griddepcontrol.wait); only q and row seq_len-1 are read after
   the wait.  A preceding kernel that releases its dependents early (griddepcontrol.launch_dependents -- this library's
   GEMV kernels, i.e. exl_q4_attn / exl_q4_matmul with <= 8 rows, do) may therefore produce q and cache row seq_len-1, as
   exl_q4_attn with q_len 1 does, but must not write older cache rows: after a multi-token exl_q4_attn (q_len 2..8) put
   any other kernel or a stream synchronisation before this call.  Kernels that never release early (torch ops, copies)
   are ordered as usual. */
int exl_decode_attn(const void* q, const void* key_cache, const void* value_cache, void* out,
                    int num_heads, int num_kv_heads, int head_dim, int seq_len, int max_seq_len, void* stream);

/* --- whole decode step as ONE persistent kernel (SURVEY.md 8f-4 "host loop"; 8f-2 lm_head + final norm) ------------- */

/* Everything ExLlama.forward does for one new token of one sequence (model.py:1053-1077: per layer ExLlamaAttention.fused
   :322-417 and ExLlamaMLP.fused :238-263, then the final norm and lm_head), in one cooperative launch -- see
   exllama_b200/csrc/decode_step.cu.  The plan borrows every pointer in the descriptor (weights, norms, caches, tables);
   they must stay valid and fixed for the plan's lifetime.  Restrictions: head_dim 128, kv_heads == heads, groupsize 32 * 2^n
   (or one group), widths multiples of 128, act-order (g_idx) matrices only with tp_world == 1; anything else ->
   EXL_ERR_ARG (use the per-op entry points). */
typedef struct exl_decode_plan exl_decode_plan;
typedef struct exl_decode_desc {
    int n_layers, num_heads, head_dim, max_seq_len, vocab;
    float rms_eps;
    const exl_q4_matrix* const* mats;   /* [n_layers * 7]: q, k, v, o, gate, up, down of each layer (handles from exl_make_q4) */
    const void* const* ln1;              /* [n_layers] input_layernorm weight, half [hidden] */
    const void* const* ln2;              /* [n_layers] post_attention_layernorm weight */
    void* const* key_cache;              /* [n_layers] half [num_heads, max_seq_len, head_dim] (model.py:557-585) */
    void* const* value_cache;
    const void* sin; const void* cos;    /* half [max_seq_len, head_dim] (model.py:864-877) */
    const void* final_norm;              /* half [hidden] or NULL */
    const void* lm_head;                 /* half [vocab, hidden] (nn.Linear weight, model.py:845-846) or NULL: no head */
    /* tensor parallel (SURVEY.md 8e; 0 / 1 = single GPU): this rank's column shards of q, k, v, gate, up (num_heads = LOCAL heads) and
       row shards of o, down; norms, tables, x and the head replicated.  The row-parallel partials are exchanged over NVLink inside the same
       kernel ({value, launch-epoch} 8-byte stores into every peer's slot buffer, polled by the consumer and summed in rank order):
       no separate collective, no cross-GPU barrier. */
    int tp_rank, tp_world;
} exl_decode_desc;

int exl_decode_plan_create(const exl_decode_desc* desc, exl_decode_plan** out_plan);
int exl_decode_plan_destroy(exl_decode_plan* plan);
/* Tensor parallel set-up: export this rank's 64-byte cudaIpc handle, exchange (e.g. through torch.distributed), import all of
   them (world x 64 bytes in rank order) on every rank before the first exl_decode_step; every rank must then call
   exl_decode_step for the same token at about the same time (a rank that waits longer than 4 s for its peers traps). */
int exl_decode_plan_ipc_export(exl_decode_plan* plan, void* handle64);
int exl_decode_plan_ipc_import(exl_decode_plan* plan, const void* handles, int world);
int exl_decode_plan_info(const exl_decode_plan* plan, int* grid, int* ring_stages, int64_t* smem_bytes, int64_t* barriers_per_step);

/* Bring-up aid: with EXL_DS_TRACE=1 in the environment when the plan is created, every CTA stamps %globaltimer at its phase
   boundaries of the first 4 layers; this copies the [grid][4][24] stamps of the last launch to the host. */
int exl_decode_plan_trace(exl_decode_plan* plan, unsigned long long* out_host, int64_t capacity);

/* One token: x_in half [hidden] (the embedding row), attends over cache rows [0, past_len) plus the new row, which it
   writes at past_len.  x_out (optional) receives the final hidden state before the final norm, logits float [vocab]
   (required iff the plan has an lm_head).  CUDA-graph capturable; successive calls need no host synchronisation. */
int exl_decode_step(exl_decode_plan* plan, const void* x_in, int past_len, void* x_out, void* logits, void* stream);

/* --- tensor-parallel variants (new functionality; the reference has no tensor parallelism, SURVEY.md 8e) ----- */

/* As exl_q4_attn_2 / exl_q4_mlp, but with add_residual == 0 the row-parallel projection OVERWRITES x with this rank's
   partial product instead of accumulating into it, so that one in-place all-reduce over the ranks (rank 0 keeps the
   residual) yields x_old + sum(partials) everywhere. */
int exl_q4_attn_2_tp(void* x, const void* attn_output, const exl_q4_matrix* o_proj, int height, int add_residual, void* stream);
int exl_q4_mlp_tp(void* x, const void* rms_norm_weight, float epsilon,
                  const exl_q4_matrix* gate, const exl_q4_matrix* up, const exl_q4_matrix* down,
                  int height, int dim, int add_residual, int device, void* stream);

/* Fused projection + all-reduce over NVLink peer memory (one kernel: the GEMV epilogue pushes its tile into every peer's
   receive slot, flags it, and sums the partials of all ranks in rank order -- no NCCL call, CUDA-graph capturable).
   Setup, once per process and device: every rank allocates a workspace and exports it through cudaIpc, the 64-byte
   handles are exchanged by the host (any transport), peers are opened, then exl_tp_init installs the pointer table. */
int exl_tp_workspace_alloc(int device, void** local_ptr, void* ipc_handle_64bytes);
int exl_tp_workspace_open(int device, const void* ipc_handle_64bytes, void** peer_ptr);
int exl_tp_init(int device, int rank, int world, void* const* workspace_ptrs /* [world], own entry = local_ptr */);

/* Number of flag waits of the fused all-reduce that gave up (bounded spin) since the workspace was allocated; 0 = healthy. */
int exl_tp_status(int device, unsigned* timeouts);
/* x += all_reduce_sum(attn_output_local . o_proj_rowshard)            (every rank ends with the same x) */
int exl_q4_attn_2_ar(void* x, const void* attn_output, const exl_q4_matrix* o_proj, int height, void* stream);
/* x += all_reduce_sum(down_rowshard(silu(gate(n)) * up(n))),  n = rms_norm(x)   */
int exl_q4_mlp_ar(void* x, const void* rms_norm_weight, float epsilon,
                  const exl_q4_matrix* gate, const exl_q4_matrix* up, const exl_q4_matrix* down,
                  int height, int dim, int device, void* stream);

/* --- sampling helper (CPU, like the reference) --------------------------------- */

/* cpu_func/rep_penalty.cpp:5-31 */
int exl_rep_penalty(int vocab_size, const uint64_t* sequence_host, float* rep_mask_host,
                    float penalty_max, int sustain, int decay, int seq_len);
/* cpu_func/rep_penalty.cpp:36-74 (one batch row) */
int exl_apply_rep_penalty(int vocab_size, const uint64_t* sequence_host, float penalty_max,
                          int sustain, int decay, int seq_len, float* logits_host);

/* --- host-buffer entry point (end-to-end measurement and non-torch callers) ----- */

/* q4_matmul with HOST x / out: copies x H2D, runs exl_q4_matmul, copies out D2H, synchronises `stream`.
   x_host / out_host should be pinned for full speed.  d_x / d_out are caller-provided device staging
   buffers of M*K and M*N halves. */
int exl_q4_matmul_host(const void* x_host, int M, const exl_q4_matrix* w, void* out_host,
                       void* d_x, void* d_out, void* stream);

/* --- introspection for benchmarks ------------------------------------------------ */

/* number of kernel launches issued by this library since process start (all entry points) */
int64_t exl_launch_count(void);
/* name of the code path the last exl_q4_matmul call took ("skinny_mma", "tc_gemm", "recons_cublas") */
const char* exl_last_q4_path(void);
/* tile configuration of the last tcgen05 GEMM launch: "128x128", "256x128" or "256x256" (M x N per CTA), with the suffix
   "+mc" when the x tile was multicast across a 2-CTA cluster; "none" before the first one */
const char* exl_last_tc_config(void);
/* decode GEMV (q4_gemv_kernel) launches of the last exl_q4_* call, in launch order and separated by "; ", each
   "<prologue>+<epilogue> cs=<cluster size = K split> chunk=<x staging chunk, 128-k stages> items=<clusters>", e.g.
   "rmsnorm+silu_mul cs=2 chunk=8 items=86; plain+store cs=4 chunk=8 items=32" for a fused q4_mlp; "none" when it made none */
const char* exl_last_gemv_config(void);

#define EXL_SKINNY_MAX_M 8

#ifdef __cplusplus
}
#endif
#endif /* EXL_B200_H */
