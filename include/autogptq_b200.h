/*
 * autogptq_b200.h - C ABI of the B200-native GPTQ W4A16 QuantLinear hot path.
 *
 * Drop-in boundary (SURVEY.md 8b).  Every entry point replaces a pybind11 torch-extension
 * function the reference's QuantLinear modules call today; the reference interface each
 * one stands in for is cited as file:line relative to /root/reference.
 *
 * Conventions
 *   - plain C, no torch / CUDA types in signatures: device and host pointers are `void*`
 *     or typed plain pointers, the CUDA stream is passed as `void*` (a cudaStream_t;
 *     NULL = legacy default stream).  The caller owns every buffer.
 *   - all functions return 0 on success or a negative AGB200_E* code; the message for the
 *     calling thread is available from agb200_last_error().  No exceptions cross the ABI.
 *   - no hidden global state besides a per-device attribute cache; thread-safe.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails
 *     with AGB200_ECUDA.
 *
 * Packed layout (unchanged from the reference checkpoint contract,
 * auto_gptq/nn_modules/qlinear/qlinear_cuda_old.py:50-79, pack :110-200):
 *   qweight int32 [K/8, N]   nibble j of word (r,n) = row 8r+j of column n
 *   qzeros  int32 [G,  N/8]  nibble j of word (g,c) = column 8c+j, stores zero-1
 *   scales  f16/bf16 [G, N]  (same dtype as x)
 *   zero rule: z = (nibble + 1) & 0xF  (every reference .cu kernel;
 *              exllamav2/cuda/q_gemm_kernel_gptq.cuh:128)
 *   W[k,n] = scales[g(k),n] * (q[k,n] - z[g(k),n]);  y = x W (+ bias)
 *   g(k) = k / group_size.  Act-order (desc_act) layers are first re-sorted with
 *   agb200_w4_make_sequential (the exllama transform) and then run with `perm`.
 */
#ifndef AUTOGPTQ_B200_H_
#define AUTOGPTQ_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AGB200_ABI_VERSION 4

/* element types of x / y / scales / bias */
#define AGB200_F16 0
#define AGB200_BF16 1

/* error codes */
#define AGB200_OK 0
#define AGB200_EINVAL (-1)   /* bad shape / alignment / dtype / null pointer */
#define AGB200_ECUDA (-2)    /* CUDA runtime error (message has cudaGetErrorString) */
#define AGB200_ENOSUP (-3)   /* valid GPTQ layer this build does not handle */
#define AGB200_EWORKSPACE (-4) /* workspace too small */

/* kernel selection for agb200_w4a16_forward_ex */
#define AGB200_KERNEL_AUTO 0
#define AGB200_KERNEL_GEMV 1   /* CUDA-core FHFMA GEMV, M <= AGB200_GEMV_MAX_M per pass (AUTO: M = 1) */
#define AGB200_KERNEL_GEMM 2   /* tcgen05 / TMEM tensor-core GEMM */
#define AGB200_KERNEL_SKINNY 3 /* decode batches M <= 8: warp-level MMA on subnormal-encoded nibbles, cluster split-K (AUTO: M = 5..8) */
/* 4 and 5 are unused (they named kernels that were removed); a caller that passes them gets AGB200_EINVAL */
#define AGB200_KERNEL_IMMA 6 /* decode batches M <= 8: integer tensor cores on raw nibbles, x as 24-bit block fixed point (AUTO: M = 2..4) */
#define AGB200_GEMV_MAX_M 4
#define AGB200_SKINNY_MAX_M 8
#define AGB200_IMMA_MAX_M 8

int agb200_abi_version(void);
const char* agb200_last_error(void);

/* Number of CUDA devices visible, or a negative error.  Used by the host side to fail loudly. */
int agb200_device_count(void);

/*
 * y[M,N] = x[M,K] * dequant(qweight,qzeros,scales) (+ bias), all pointers DEVICE memory.
 *
 * Replaces, for 4-bit layers:
 *   exllamav2  gemm_half_q_half(a, b_handle, c, force_cuda)   autogptq_extension/exllamav2/ext.cpp:95-126
 *   exllama    q4_matmul(x, w4_handle, out)                   autogptq_extension/exllama/exllama_ext.cpp:176-217
 *   cuda_old   vecquant4matmul_faster_old / _old              autogptq_extension/cuda_256/autogptq_cuda_256.cpp:174-187
 *   cuda       vecquant4matmul (g_idx)                        same file
 *   marlin     mul(A, B, C, s, workspace, ...)                autogptq_extension/marlin/marlin_cuda.cpp:30-75
 * plus the Python-side `output.add_(bias)` (qlinear_exllamav2.py:193-194), which is fused here.
 *
 *   x, y      [M,K] / [M,N], row-major, dtype `dtype`; y is caller-allocated
 *             (qlinear_exllamav2.py:39 torch.empty).
 *   qweight_tc  NULL, or the tensor-core copy of qweight made by agb200_w4_prepare_tc (same shape; nibbles of
 *             every word reordered so that adjacent k unpack into one 16-bit pair).  Needed by the tcgen05 path
 *             (M > 8); the decode kernels (M <= 8) read the checkpoint layout `qweight` directly.  This is the
 *             analogue of the load-time shuffle the reference does IN PLACE (exllamav2/cuda/q_matrix.cu:19-42).
 *   perm      NULL, or int32[K]: x column gathered for sorted row j is perm[j]; qweight must then be
 *             the matrix produced by agb200_w4_make_sequential (exllama q4_matrix.cu:105-169,
 *             column_remap.cu:29-36 semantics).
 *   bias      NULL or [N] of `dtype`.
 *   group_size  >0; pass K for the reference's group_size=-1.  G = ceil(K/group_size).
 *   workspace DEVICE scratch of at least agb200_w4a16_workspace_bytes(M,K,N) bytes; it is
 *             used by the tensor-core path (permuted x of act-order layers).  May be NULL when that
 *             function returns 0.
 *   stream    cudaStream_t the work is enqueued on (the reference launches on the legacy default
 *             stream, q_gemm.cu:47,85; we take the stream explicitly so CUDA graphs capture it).
 * Constraints: K % 8 == 0, N % 8 == 0, pointers 16-byte aligned.
 */
int agb200_w4a16_forward(const void* x, const int32_t* qweight, const int32_t* qweight_tc, const int32_t* qzeros,
                         const void* scales, const int32_t* perm, const void* bias, void* y,
                         int M, int K, int N, int group_size, int dtype,
                         void* workspace, size_t workspace_bytes, void* stream);

/* Same, with an explicit kernel choice and tuning knobs (tests / benchmarks).
 *   kernel   AGB200_KERNEL_*
 *   tune0/1  GEMV: tune0 = lanes along N per warp (8|16|32, 0=auto), tune1 = split-K (1|2|4|8, 0=auto),
 *            flags bit0 = biased-exponent unpack instead of the subnormal unpack.
 *            SKINNY: tune1 = split-K (1|2|4|8, 0=auto), flags bit0 as for GEMV.
 *            IMMA: tune0 = 0 auto | 2 register-ring persistent form | 1, 4 tile-per-CTA form
 *                  with that many warps along N;
 *                  tune1 = split-K of the tile-per-CTA form (1|2|4|8, 0=auto).
 *            GEMM: tune0 = x-row tile (16..256, 0=auto), tune1 = split-K (0=auto). */
int agb200_w4a16_forward_ex(const void* x, const int32_t* qweight, const int32_t* qweight_tc, const int32_t* qzeros,
                            const void* scales, const int32_t* perm, const void* bias, void* y,
                            int M, int K, int N, int group_size, int dtype,
                            void* workspace, size_t workspace_bytes, void* stream,
                            int kernel, int tune0, int tune1, int flags);

size_t agb200_w4a16_workspace_bytes(int M, int K, int N);

/*
 * Grouped forward: `n_layers` (<= 4) sibling layers that consume the SAME x (q|k|v, gate|up) in ONE launch, for
 * decode batches M <= AGB200_IMMA_MAX_M.  Arrays of `n_layers` entries; perm[i] / bias[i] may be NULL, and the
 * arrays `perm` / `bias` themselves may be NULL.  All layers share K, group_size and dtype; N[i] % 8 == 0.
 * The reference's counterpart is its fused-QKV injection, which concatenates the packed tensors instead
 * (auto_gptq/nn_modules/fused_llama_attn.py:171-207); here the checkpoint tensors stay separate.
 * For larger M (or shapes the decode kernels cannot take) the call simply runs the layers one after another.
 */
int agb200_w4a16_forward_group(const void* x, int n_layers, const int32_t* const* qweight, const int32_t* const* qweight_tc,
                               const int32_t* const* qzeros, const void* const* scales, const int32_t* const* perm,
                               const void* const* bias, void* const* y, const int* N, int M, int K, int group_size,
                               int dtype, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Decode chain: ONE persistent launch for a whole list of dependent QuantLinear stages (M <= AGB200_CHAIN_MAX_M rows).
 *
 * A stage is up to four sibling layers that consume the same x (q|k|v, gate|up; a single layer is a stage of one).
 * A stage's x is either a caller-owned buffer that is ready when the launch starts, or the `y` buffer of a layer of an
 * EARLIER stage of the same chain (matched by pointer).  The launch streams the weights of ALL stages back to back
 * through a shared-memory ring (TMA) without pausing at layer boundaries; only the arithmetic of a stage waits for its x,
 * and it does so by polling the data itself (outputs travel between stages as {value pair, launch tag} words in plan
 * memory - no flags, fences or grid barriers).  This is what the reference approximates by injecting fused modules
 * (auto_gptq/nn_modules/fused_llama_attn.py:171-207, fused_llama_mlp.py:131-245) - here the checkpoint tensors stay
 * separate and the fusion is across DEPENDENT layers as well.  The reference has no counterpart of the cross-layer part:
 * its kernels are one launch per layer on the legacy stream (exllamav2/cuda/q_gemm.cu:47,85).
 *
 * x transforms at a stage input (x_mode):
 *   AGB200_CHAIN_X_PLAIN      x
 *   AGB200_CHAIN_X_SILU_MUL   silu(x) * x2, both rounded to `dtype` like the reference's LlamaMLP act_fn(gate) * up
 *                             (fused_llama_mlp.py:154-166): the down_proj stage of an MLP reads gate / up directly
 *   AGB200_CHAIN_X_SUM_PARTS  x = sum of x_parts partial vectors: the all-reduce of row-parallel tensor parallelism
 *                             (SURVEY 8e).  `x` then points to a caller-owned, zero-initialised buffer of
 *                             x_parts * x_part_stride 8-byte words ([part][M][K/2]; agb200_chain_parts_bytes) that the
 *                             PEERS fill: a row-parallel layer of rank r lists in y_peers, for every rank, the address of
 *                             part r inside that rank's buffer (peer memory, e.g. cudaIpcOpenMemHandle), and its epilogue
 *                             stores the tagged words there - a one-shot all-reduce with one NVLink one-way latency.  All
 *                             ranks must run the same number of launches of their chains (the tag is the launch count).
 * Act-order layers: pass the matrix produced by agb200_w4_make_sequential as qweight and `perm` (shared by the stage).
 * Constraints: K % 128 == 0, K <= 32768, group_size % 128 == 0 (pass K for -1), N % 32 == 0,
 * 16-byte aligned pointers.
 *
 * Ownership: `plan` is caller-owned DEVICE memory of agb200_chain_plan_bytes(...) bytes (descriptor tables, TMA tensor
 * maps, inter-stage words, counters) that must stay alive and untouched until agb200_chain_destroy; the handle is a
 * small host object.  agb200_chain_forward only enqueues one cooperative launch on `stream` (CUDA-graph capturable).
 * The device must be otherwise idle enough for one CTA per SM to be co-resident (cooperative launch fails otherwise).
 */
#define AGB200_CHAIN_MAX_M 2
#define AGB200_CHAIN_MAX_PEERS 8
#define AGB200_CHAIN_X_PLAIN 0
#define AGB200_CHAIN_X_SILU_MUL 1
#define AGB200_CHAIN_X_SUM_PARTS 2
#define AGB200_CHAIN_DEBUG_NO_DEPS 1   /* measurement aid: do not wait for x (results are garbage) */
#define AGB200_CHAIN_DEBUG_NO_MATH 2   /* measurement aid: consumers only free ring slots (results are garbage) */
#define AGB200_CHAIN_DEBUG_NO_CONVERT 4 /* measurement aid: x is not re-read per stage (results are garbage) */
#define AGB200_CHAIN_DEBUG_PROFILE 8   /* record per-CTA cycle counters, read back with agb200_chain_profile */

typedef struct agb200_chain_layer {
  const int32_t* qweight;   /* [K/8, N] (row-sorted copy for act-order layers) */
  const int32_t* qzeros;    /* [G, N/8] */
  const void* scales;       /* [G, N] of the chain's dtype */
  const void* bias;         /* [N] or NULL */
  void* y;                  /* [M, N] output of the chain's dtype; may be NULL when y_peers is given */
  void* const* y_peers;     /* NULL, or DEVICE array of n_peers addresses (see X_SUM_PARTS) */
  int32_t N;
  int32_t n_peers;          /* 0, or 1..AGB200_CHAIN_MAX_PEERS */
} agb200_chain_layer;

typedef struct agb200_chain_stage {
  const void* x;            /* [M, K] of the chain's dtype, or the parts buffer for X_SUM_PARTS */
  const void* x2;           /* X_SILU_MUL: second operand [M, K]; else NULL */
  const int32_t* perm;      /* int32[K] or NULL (see agb200_w4a16_forward) */
  int32_t K;
  int32_t group_size;       /* > 0; pass K for -1 */
  int32_t n_layers;         /* 1..4 */
  int32_t x_mode;           /* AGB200_CHAIN_X_* */
  int32_t x_parts;          /* X_SUM_PARTS: number of partial vectors; else 0 */
  int32_t reserved;
  int64_t x_part_stride;    /* X_SUM_PARTS: 8-byte words between consecutive parts (>= M * K / 2) */
  agb200_chain_layer layer[4];
} agb200_chain_stage;

size_t agb200_chain_plan_bytes(const agb200_chain_stage* stages, int n_stages, int M);
/* Bytes of one X_SUM_PARTS buffer: parts * M * K / 2 words of 8 bytes. */
size_t agb200_chain_parts_bytes(int parts, int M, int K);
int agb200_chain_create(const agb200_chain_stage* stages, int n_stages, int M, int dtype, void* plan, size_t plan_bytes,
                        void** handle_out);
/* flags: 0, or AGB200_CHAIN_DEBUG_* bits (benchmarks only). */
int agb200_chain_forward(void* handle, int flags, void* stream);
int agb200_chain_destroy(void* handle);
/* Facts about a created chain for logs / benchmarks: ring slots, dynamic shared memory bytes, grid size. */
int agb200_chain_info(void* handle, int* slots, int* smem_bytes, int* grid);
/* After a forward with AGB200_CHAIN_DEBUG_PROFILE (and a stream synchronisation): copies grid x 3 x 8 cycle counters
 * {total, wait for x, convert x, wait for weights, unpack + MMA, flush, tile end, -} of one warp per consumer
 * group to out_host; returns the number of entries or a negative error.  Measurement aid. */
int agb200_chain_profile(void* handle, long long* out_host, int max_entries);
/* Every wait inside the chain kernel is bounded; a timeout (a protocol bug, or a peer rank that died) traps the launch
 * after writing {site (0 = none), stage, CTA, warp, detail} to host-mapped words.  They stay readable after the CUDA
 * context is lost; agb200_chain_forward refuses to launch again once they are set. */
int agb200_chain_diag(int* out5);

/*
 * Peer-visible device memory for the X_SUM_PARTS buffers of tensor-parallel chains: plain cudaMalloc'd, zero-filled
 * memory plus CUDA IPC handles (one process per GPU; the host side exchanges the 64-byte handles, e.g. with
 * torch.distributed.all_gather_object).  agb200_peer_open maps a peer's allocation into this process with peer access
 * enabled (NVLink / NVSwitch); the returned pointer is what goes into agb200_chain_layer.y_peers tables.
 * The reference has no counterpart (no tensor parallelism: modeling/_utils.py:341-377 only places whole layers).
 */
#define AGB200_PEER_HANDLE_BYTES 64
int agb200_peer_alloc(size_t bytes, void** ptr_out);
int agb200_peer_free(void* ptr);
int agb200_peer_export(const void* ptr, void* handle_out /* AGB200_PEER_HANDLE_BYTES */);
int agb200_peer_open(const void* handle /* AGB200_PEER_HANDLE_BYTES */, void** ptr_out);
int agb200_peer_close(void* ptr);

/*
 * Next-layer prefetch hint (optional, decode): names up to 8 device ranges - typically the packed weights and scales of
 * the layer(s) that will run NEXT - which the decode kernel launched by the next agb200_w4a16_forward* call of this
 * thread pulls into L2 while it computes, so that the DRAM stream does not pause at the kernel boundary.  The hint is
 * consumed by that call (kernels that do not support it ignore it); wrong ranges cost bandwidth, never correctness.
 * The reference has no counterpart (its kernels are launched one at a time on the legacy stream, q_gemm.cu:47,85).
 */
int agb200_w4_prefetch_hint(int n, const void* const* ptrs, const size_t* bytes);

/*
 * End-to-end variant with HOST activations: copies x_host -> device staging, runs the forward
 * and copies y back to y_host, all on `stream` (asynchronous when the host buffers are pinned).
 * `staging` is device scratch of agb200_w4a16_host_staging_bytes(M,K,N) bytes: x, y and the forward's workspace are
 * carved from it, so act-order layers on the tensor-core path need no other buffer.  A smaller buffer returns
 * AGB200_EWORKSPACE before anything is copied or launched.  Pageable host buffers make the copies synchronous.
 */
int agb200_w4a16_forward_host(const void* x_host, const int32_t* qweight, const int32_t* qweight_tc, const int32_t* qzeros,
                              const void* scales, const int32_t* perm, const void* bias, void* y_host,
                              int M, int K, int N, int group_size, int dtype,
                              void* staging, size_t staging_bytes, void* stream);
size_t agb200_w4a16_host_staging_bytes(int M, int K, int N);

/*
 * Load-time act-order transform (desc_act): gather packed rows so that groups become contiguous.
 *   qweight_out nibble-row j = qweight_in nibble-row perm[j]; perm is int32[K] on the DEVICE.
 * Non-destructive (the reference's make_sequential rewrites qweight in place:
 * exllama/cuda_func/q4_matrix.cu:105-169, exllamav2/cuda/q_matrix.cu:502-627).
 * `perm` itself (stable argsort of g_idx) is computed by the host side.
 */
int agb200_w4_make_sequential(const int32_t* qweight_in, const int32_t* perm, int32_t* qweight_out,
                              int K, int N, void* stream);

/*
 * Load-time: tensor-core copy of a packed matrix (non-destructive; same size as qweight).  Word-wise nibble
 * permutation: output nibble positions [0,4,1,5,2,6,3,7] hold rows 8r+[0..7].  Apply it to the matrix that
 * is actually run (i.e. after agb200_w4_make_sequential for act-order layers).
 */
int agb200_w4_prepare_tc(const int32_t* qweight_in, int32_t* qweight_tc_out, int K, int N, void* stream);

/*
 * Full dequantisation W[K,N] (dtype) - the `reconstruct` kernels of the reference
 * (exllamav2/cuda/q_matrix.cu:158-279, exllama/cuda_func/q4_matrix.cu:171-211).  Test/debug aid;
 * not on the forward path.  g_idx may be NULL (sequential groups) or int32[K] (arbitrary row->group).
 */
int agb200_w4_dequantize(const int32_t* qweight, const int32_t* qzeros, const void* scales,
                         const int32_t* g_idx, void* w_out, int K, int N, int group_size, int dtype,
                         void* stream);

/* x_out[m, j] = x[m, perm[j]]  (exllama/cuda_func/column_remap.cu:9-63). */
int agb200_permute_columns(const void* x, const int32_t* perm, void* x_out, int M, int K, int dtype,
                           void* stream);

/* Static facts about the build, for logs: returns e.g. "sm_100a tcgen05+tma gemv=fhfma". */
const char* agb200_build_info(void);

#ifdef __cplusplus
}
#endif
#endif /* AUTOGPTQ_B200_H_ */
