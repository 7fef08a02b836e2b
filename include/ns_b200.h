/*
 * ns_b200.h -- C ABI of libns_b200.so: the B200-native (sm_100a) replacement for neural-speed's low-bit
 * weight-only matmul path.  Plain pointers and sizes only; no torch / C++ types cross this boundary.
 *
 * Every entry point names the reference interface it replaces (paths relative to /root/reference).
 * Three groups:
 *   1. bestla_*          host-buffer drop-ins with the exact signatures of neural_speed/core/ne_bestla.h:21-83.
 *                        `weiptr` is a serialized BesTLA blob in HOST memory (bestla/bestla/bestla_storage.h:697-834);
 *                        activations / outputs are HOST fp32.  The library uploads + repacks each blob once
 *                        (cached by address), runs the CUDA kernels, copies the result back.
 *   2. bestla_device_*   device-resident set modelled on the reference's NS_SYCL block, ne_bestla.h:85-112
 *                        (void* queue == cudaStream_t).  Activations / outputs are DEVICE fp32.
 *   3. ns_* / BTLAGemm*  ggml Q4_0 path (ne_compute_forward_mul_mat_q_f32, core/ne_layers.c:7085), the weight
 *                        packing API (core/layers/bestla_gemm.h:30-58, models/model_utils/quant_utils.cpp:226-400)
 *                        and handles for fused / graph-captured decode.
 *
 * Error convention (mirrors the reference, SURVEY.md 8b): *_support() are pure probes returning bool;
 * *_forward() print "Err: ..." and abort() on invalid input or when no CUDA device / kernel image is usable
 * (there is NO CPU fallback in this library); pack functions return false / 0 on failure;
 * ns_* functions return 0 on success and a negative NS_E_* code otherwise (message via ns_last_error()).
 */
#ifndef NS_B200_H
#define NS_B200_H
#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#include "ns_ne_abi.h"

#ifdef __cplusplus
extern "C" {
#endif

#define NS_API __attribute__((visibility("default")))

/* ------------------------------------------------------------------------------------------------ enums */
/* weight element formats in the device ("NSB") layout */
enum ns_wfmt { NS_W_S4 = 0, NS_W_S8 = 1, NS_W_NF4 = 2, NS_W_Q6K = 3 /* ggml block_q6_K, only via ns_weight_from_q6_K */ };
/* scale storage */
enum ns_stype { NS_S_F32 = 0, NS_S_BF16 = 1, NS_S_F16 = 2 };
/* activation numerics ("compute type"): which reference arithmetic the kernel reproduces
 *   NS_COMP_F32     fp32 activations, w = (q-zp)*scale in fp32, fp32 FMA      (BesTLA CompFp32, kernel_ref.h:2490)
 *   NS_COMP_BF16    activations and dequantised weights rounded to bf16, fp32 accumulate (BesTLA CompBf16)
 *   NS_COMP_INT8    u8-asym per-K-block activations x int weights, exact integer block dots
 *                   (BesTLA CompInt8, kernel_ref.h:1825 + :2372)
 *   NS_COMP_Q8_0    ggml: s8 activations per 32, fp16 scales, round-half-even (quantize.h:447, vec_dot.h:131)
 *   NS_COMP_INT8_S8 s8-sym per-K-block activations (kernel_ref.h:1886 + :2432)
 */
enum ns_comp { NS_COMP_F32 = 0, NS_COMP_BF16 = 1, NS_COMP_INT8 = 2, NS_COMP_Q8_0 = 3, NS_COMP_INT8_S8 = 4 };
/* ne_comp_type, neural_speed/core/data_types.h:55-62 */
enum ns_ne_comp_type { NS_NE_COMP_UNDEF = 0, NS_NE_COMP_F32 = 1, NS_NE_COMP_BF16 = 2, NS_NE_COMP_F16 = 3, NS_NE_COMP_INT8 = 4 };
/* BTLA_DTYPE raw values, bestla/bestla/bestla.h:38-87 */
#define NS_BTLA_F32 32u
#define NS_BTLA_BF16 (16u | (1u << 16))
#define NS_BTLA_F16 16u
#define NS_BTLA_S8 (8u | (1u << 8))
#define NS_BTLA_S4_CLIP (4u | (1u << 8))
#define NS_BTLA_F4_NF4 (4u | (2u << 16))
#define NS_BTLA_F4_BNB (4u | (1u << 16)) /* 4-bit float codebooks of bestla.h:82-84, kernel_ref.h:1209-1321 */
#define NS_BTLA_F4_E2M1 4u
/* bit-plane integer types (bestla.h:75-81, storage bestla_storage.h:724-745): held on the device in the 4-bit (2, 3 bits) or
 * 8-bit (5, 6, 7 bits) container, same integers, same scales and zero points */
#define NS_BTLA_S2_CLIP (2u | (1u << 8))
#define NS_BTLA_S3_CLIP (3u | (1u << 8))
#define NS_BTLA_S5_CLIP (5u | (1u << 8))
#define NS_BTLA_S6_CLIP (6u | (1u << 8))
#define NS_BTLA_S7_CLIP (7u | (1u << 8))

#define NS_OK 0
#define NS_E_INVALID (-1)
#define NS_E_NODEVICE (-2)
#define NS_E_CUDA (-3)
#define NS_E_UNSUPPORTED (-4)

NS_API const char* ns_last_error(void);
NS_API const char* ns_version(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
NS_API unsigned long long ns_launch_count(void);

/* ------------------------------------------------------------------ 1. ne_bestla.h host-buffer drop-ins */
/* ne_bestla.h:33 / core/layers/ne_bestla.cpp:19.  Selects cuda:0 lazily; aborts later if none. */
NS_API void bestla_init(void);
/* ne_bestla.h:25-27.  Host threads are irrelevant on the GPU path; kept for ABI compatibility. */
NS_API int bestla_set_threads(int nth);
NS_API void* bestla_get_thread_handle(void);
NS_API void bestla_timer(bool init);

/* ne_bestla.h:35 / core/layers/inner_product.cpp:20 -- M * pad128(K) * 4 bytes, as the reference */
NS_API unsigned long long bestla_f32f32_get_workspace_size(int m, int n, int k, void* wptr);
/* ne_bestla.h:37 / inner_product.cpp:28 -- C[m][n] = A[m][k] . dequant(W)  (lda is ignored, K is used: bestla_gemm.cpp:44) */
NS_API void bestla_f32f32_forward(float* activation, void* weiptr, float* output, int m, int n, int k, int lda, int ldo,
                                  void* workspace);
/* ne_bestla.h:40-42 / inner_product.cpp:113,132 -- bias epilogue */
NS_API bool bestla_fusion_add_f32f32_support(void* weiptr, int m, int n, int k);
NS_API void bestla_fusion_add_f32f32_forward(float* activation, void* weiptr, float* bias, float* output, int m, int n,
                                             int k, int lda, int ldo, bool boardcast_bias, void* workspace);
/* ne_bestla.h:44-51 / core/layers/ip_fusion_qkv.cpp:155,163,194 -- out = [3][M][N] */
NS_API unsigned long long bestla_fusion_QKV_f32f32_get_workspace_size(int m, int n, int k, void* w1ptr);
NS_API bool bestla_fusion_QKV_f32f32_support(void* wqptr, void* wkptr, void* wvptr, int m, int n, int k);
NS_API void bestla_fusion_QKV_f32f32_forward(float* activation, void* wqptr, void* wkptr, void* wvptr, float* output,
                                             int m, int n, int k, int lda, int ldo, void* workspace);
/* ne_bestla.h:53-66 / core/layers/ip_fusion_ffn.cpp:20,724-740 -- out = (silu(x W1) * (x W3)) W2 */
NS_API unsigned long long bestla_fusion_FFN_f32f32_get_workspace_size(int seq, int fin, int fmid, int fout, void* w1ptr,
                                                                      void* w2ptr);
NS_API bool bestla_fusion_FFN_SiLu_f32f32_support(void* w1ptr, void* w2ptr, void* w3ptr, int seq, int fin, int fmid,
                                                  int fout);
NS_API void bestla_fusion_FFN_SiLu_f32f32_forward(float* activation, void* w1ptr, void* w2ptr, void* w3ptr, float* tmp1,
                                                  float* tmp2, float* output, int seq, int fin, int fmid, int fout,
                                                  void* workspace);
/* ne_bestla.h:75 / ne_bestla.cpp:74 -- dequantise a blob to fp32 [n][ld] (ld >= k) */
/* GELU feed-forward nodes of the non-Llama architectures (ne_bestla.h:53-73, ip_fusion_ffn.cpp:729-779);
 * tanh-GELU of kernel_ref.h:1570.  Gelu_Mul: tmp2 = gelu(x W1) * (x W3); GeLu: tmp1 = gelu(x W1); Add_GeLu adds b1/b2. */
NS_API bool bestla_fusion_FFN_Gelu_Mul_f32f32_support(void* w1ptr, void* w2ptr, void* w3ptr, int seq, int fin, int fmid,
                                                      int fout);
NS_API void bestla_fusion_FFN_Gelu_Mul_f32f32_forward(float* activation, void* w1ptr, void* w2ptr, void* w3ptr, float* tmp1,
                                                      float* tmp2, float* output, int seq, int fin, int fmid, int fout,
                                                      void* workspace);
NS_API bool bestla_fusion_FFN_GeLu_f32f32_support(void* w1ptr, void* w2ptr, int seq, int fin, int fmid, int fout);
NS_API void bestla_fusion_FFN_GeLu_f32f32_forward(float* activation, void* w1ptr, void* w2ptr, float* tmp1, float* output,
                                                  int seq, int fin, int fmid, int fout, void* workspace);
NS_API bool bestla_fusion_FFN_Add_GeLu_f32f32_support(void* w1ptr, void* w2ptr, int seq, int fin, int fmid, int fout);
NS_API void bestla_fusion_FFN_Add_GeLu_f32f32_forward(float* activation, void* w1ptr, void* w2ptr, float* b1ptr, float* b2ptr,
                                                      float* tmp1, float* output, int seq, int fin, int fmid, int fout,
                                                      bool boardcast_bias, void* workspace);
NS_API void bestla_unpackweight_fp32(void* wptr, int n, int k, float* fp32data, int ld);
/* ne_bestla.h:77: quantise f32 [n][ld] into dstptr with the attributes of the blob srcptr (host only) */
NS_API void bestla_packweight_copyattr(const float* f32ptr, void* dstptr, int n, int k, int ld, void* srcptr);

/* The entry points that take the graph engine's own structs (ne_bestla.h:24-32,85; core/layers/ne_bestla.cpp:42,114-166,176,205).
 * The struct layouts are restated in ns_ne_abi.h (struct ns_ne_tensor == struct ne_tensor, ne.h:161-206); with these exported,
 * the reference's ne_graph_compute (ne_layers.c:11915) links against this library unchanged.
 *   bestla_support           which nodes the library takes (BesTLA matmuls, fused QKV / FFN, contiguous add / mul / norms), host
 *                            work-buffer size, n_tasks = 1
 *   bestla_backend_support   every result lives on the host (NE_BACKEND_CPU) outside the device-resident route
 *   bestla_parallel_for      INIT / COMPUTE / FINALIZE over the node's tasks (host threads for the engine's own ggml nodes)
 *   bestla_mul / _add / _layernormalization  host-buffer element-wise ops ne_layers.c:4622,5677,6541,6625 call directly (CUDA
 *                            kernels behind host staging, like the matmul drop-ins) */
NS_API bool bestla_support(struct ns_ne_tensor* node, int n_threads, size_t* workspace, size_t* dev_workspace);
NS_API int bestla_backend_support(struct ns_ne_tensor* src0, struct ns_ne_tensor* src1, int op);
NS_API void bestla_parallel_for(ns_forward_compute_fptr fcomp, struct ns_ne_compute_params* mainparams, struct ns_ne_tensor* node);
NS_API void bestla_mul(int batch, int vsize, const float* tensor, const float* vector, int vstep, float* out);
NS_API void bestla_add(int batch, int vsize, const float* tensor, const float* vector, int vstep, float* out);
NS_API void bestla_layernormalization(int norm_count, int norm_size, bool isrms, float epsilon, const float* FpIn, float* FpOut);

/* ------------------------------------------------------------------ 2. device-resident set (NS_SYCL analogue) */
/* ne_bestla.h:86-95.  device = opaque context owning one CUDA stream on cuda:<current>; queue = cudaStream_t */
NS_API void* bestla_create_device(bool profile);
NS_API void* bestla_get_device_queue(void* device);
NS_API void bestla_release_device(void* device);
NS_API size_t bestla_device_gmem_size(void* device);
NS_API void* bestla_device_malloc(size_t size, void* queue);
NS_API void bestla_device_free(void* ptr, void* queue);
NS_API void bestla_device_memcpy(void* dstptr, const void* srcptr, size_t size, void* queue);
NS_API void bestla_device_memcpy_sync(void* dstptr, const void* srcptr, size_t size, void* queue);
NS_API void bestla_device_sync(void* queue);
/* ne_bestla.h:96-97 / ne_bestla_sycl.cpp:94.  hoststor = serialized blob (host); devstor = host descriptor of
 * bestla_device_storage_size() bytes filled by the call; deviceptr = device buffer of at least
 * ns_device_storage_bytes(hoststor) bytes that receives the repacked weight. */
NS_API size_t bestla_device_storage_size(void);
NS_API size_t ns_device_storage_bytes(const void* hoststor);
NS_API void bestla_device_load_storage(void* hoststor, void* devstor, void* deviceptr, void* queue);
/* ne_bestla.h:98-99 / ne_bestla_sycl.cpp:152.  activation/output are DEVICE fp32; weiptr = devstor descriptor.
 * workspace: device scratch of >= ns_device_workspace_bytes(m, k) bytes (or NULL: library-owned scratch). */
NS_API size_t ns_device_workspace_bytes(int m, int k);
NS_API void bestla_device_f32f32_forward(float* activation, void* weiptr, float* output, int m, int n, int k, int lda,
                                         int ldo, void* workspace, void* queue);

/* ------------------------------------------------------------------ 3a. weight handles (device resident) */
typedef struct ns_weight ns_weight; /* opaque: repacked weight in HBM + metadata */

/* ggml rows: src0 of ne_compute_forward_mul_mat_q_f32 (ne_layers.c:7085): n rows of k/32 block_q4_0
 * (data_types.h:79-83), row stride nb01 bytes.  `rows` may be a host or a device pointer (rows_on_device). */
NS_API ns_weight* ns_weight_from_q4_0(const void* rows, int n, int k, size_t nb01, int rows_on_device, void* queue);
/* serialized BesTLA blob (host memory), StorageWeightKBlockNInteger / NFloat */
/* N rows of K/256 block_q6_K (core/data_types.h:133-138, 210 bytes each), row stride nb01: the type of output.weight in
 * llama.cpp "Q4_0" GGUF files.  ns_mul_mat on it reproduces quantize_row_q8_K + ggml_vec_dot_q6_K_q8_K
 * (vectors/cpu/quantize.h:1020, core/layers/vec_dot.h:907) bit for bit; plain matmul only (no fused QKV/FFN). */
NS_API ns_weight* ns_weight_from_q6_K(const void* rows, int n, int k, size_t nb01, int rows_on_device, void* queue);
NS_API ns_weight* ns_weight_from_btla_blob(const void* blob, void* queue);
/* same, with the number of bytes readable at `blob` (file-backed blobs: the parser never reads past it) */
NS_API ns_weight* ns_weight_from_btla_blob_n(const void* blob, size_t nbytes, void* queue);
/* canonical unpacked container as BTLAGemmPackB takes it (bestla_gemm.h:46-50): q int8 [k][n] (values, e.g.
 * nibble-8), scales f32 [k/g][n], zp int8 [k/g][n] or NULL, shuffle int[k] or NULL.  Host pointers. */
NS_API ns_weight* ns_weight_from_unpacked(const int8_t* q, const float* scales, const int8_t* zp, const int* shuffle, int n,
                                          int k, int group, int wfmt, int stype, int comp, void* queue);
NS_API void ns_weight_free(ns_weight* w);
NS_API int ns_weight_info(const ns_weight* w, int* n, int* k, int* group, int* wfmt, int* stype, int* comp, int* asym);
NS_API int ns_weight_set_comp(ns_weight* w, int comp);
/* packed bytes one GEMV must read from HBM for this weight (roofline numerator, SURVEY.md 8d) */
NS_API size_t ns_weight_algorithmic_bytes(const ns_weight* w);
/* benchmark aid: device weight of the given geometry with random codes, scales in [0.005, 0.02] and zero points (no host data) */
NS_API ns_weight* ns_weight_random(int n, int k, int group, int wfmt, int stype, int comp, int asym, unsigned seed, void* queue);
/* dequantise to device fp32 [n][ld] (debug / parity; replaces bestla_unpackweight_fp32 on device) */
NS_API int ns_weight_dequant_f32(const ns_weight* w, float* dst_dev, int ld, void* queue);

/* ------------------------------------------------------------------ 3b. device matmuls on handles */
/* dst[m][n] (ldo) = act[m][k] (lda) . W^T ; act/dst device fp32.  flags: NS_MM_* ; bias/residual may be NULL. */
#define NS_MM_BIAS_BCAST 1   /* bias is [n] broadcast over m (else [m][ldo]) */
#define NS_MM_FORCE_GEMV 2   /* always use the dp4a/FMA GEMV path (exact-integer numerics) regardless of m */
#define NS_MM_FORCE_TC 4     /* always use the tcgen05 tensor-core path (bf16 numerics) */
NS_API int ns_mul_mat(const ns_weight* w, const float* act, int lda, float* dst, int ldo, int m, const float* bias,
                      const float* residual, int flags, void* workspace, void* queue);
/* three weights sharing one activation (ne_mul_qkv): dst = [3][m][ldo], weights may differ in n */
NS_API int ns_mul_qkv(const ns_weight* wq, const ns_weight* wk, const ns_weight* wv, const float* act, int lda, float* dst,
                      int ldo, int m, void* workspace, void* queue);
/* ne_ffn_silu: tmp = silu(act.W1^T) * (act.W3^T) [m][fmid];  dst = tmp.W2^T [m][fout] */
/* GELU variants on device buffers: w3 != NULL -> Gelu_Mul (b1/b2 must be NULL); w3 == NULL -> (Add_)GeLu with optional biases */
NS_API int ns_ffn_gelu(const ns_weight* w1, const ns_weight* w2, const ns_weight* w3, const float* b1, const float* b2,
                       int bias_bcast, const float* act, int lda, float* tmp, float* dst, int ldo, int m, void* workspace,
                       void* queue);
NS_API int ns_ffn_silu(const ns_weight* w1, const ns_weight* w2, const ns_weight* w3, const float* act, int lda, float* tmp,
                       float* dst, int ldo, int m, void* workspace, void* queue);

/* The RMSNorm in front of a matmul node folded into the node's launch: ne_rms_norm + ne_mul(norm weight) + ne_mul_mat /
 * ne_mul_qkv / ne_ffn_silu (models/llama/llama.cpp:205-215, :601-612, :703-712) as ONE kernel -- every CTA of the decode GEMV
 * reads the whole activation row for the fused NE_TASK_INIT quantiser anyway, so the sum of squares costs a block reduction
 * instead of a one-CTA kernel and a launch boundary.  Decode rows only (m <= 2, int4 weights with an integer compute type):
 * ns_rmsnorm_fusable says whether a set of 1..3 weights qualifies; the calls return NS_E_UNSUPPORTED otherwise.
 *   ns_rmsnorm_mul_mat   dst = W (rms_norm(act) * norm_w) [+ residual]
 *   ns_rmsnorm_mul_qkv   dst[3][m][ldo] as ns_mul_qkv
 *   ns_rmsnorm_ffn_silu  dst = W2 (silu(W1 xn) * (W3 xn)) [+ residual],  xn = rms_norm(act) * norm_w */
NS_API int ns_rmsnorm_fusable(const ns_weight* const* weights, int nw, int m);
NS_API int ns_rmsnorm_mul_mat(const ns_weight* w, const float* act, int lda, const float* norm_w, float norm_eps, float* dst, int ldo,
                              int m, const float* residual, void* workspace, void* queue);
NS_API int ns_rmsnorm_mul_qkv(const ns_weight* wq, const ns_weight* wk, const ns_weight* wv, const float* act, int lda,
                              const float* norm_w, float norm_eps, float* dst, int ldo, int m, void* workspace, void* queue);
NS_API int ns_rmsnorm_ffn_silu(const ns_weight* w1, const ns_weight* w2, const ns_weight* w3, const float* act, int lda,
                               const float* norm_w, float norm_eps, float* tmp, float* dst, int ldo, int m, const float* residual,
                               void* workspace, void* queue);

/* Expert-indexed nodes of mixture-of-experts models: ne_mul_mat_id and ne_mul_id_ffn_silu / _gelu
 * (core/ne_layers.c:2384-2460; ne_compute_forward_mul_mat_id_q_f32 :7345-7498, _q_f32_bestla :7783-7916, dispatch :7918-7943,
 * ne_compute_forward_ffn_id_silu / _gelu :8053-8111).  dst[t] = W[e_t] . act[t] with e_t = ids[t * ids_stride + id]
 * (ids = the int32 top-k selection [n_tokens][n_used], id = which of the n_used slots this node serves, ids_stride >= n_used).
 * The reference walks the tokens of every expert one by one; here tokens are grouped by expert and every expert's weights are
 * read once per node.  ids may live on the host (ids_on_device = 0, what ne_graph_compute has) or on the device (one small
 * D2H + stream sync per node: the host sizes the per-expert launches).  Expert ids outside [0, n_as) -> NS_E_INVALID.
 * flags: NS_MM_* of ns_mul_mat (e.g. NS_MM_FORCE_GEMV keeps the exact-integer path whatever the group size).
 * ns_ffn_id: gelu = 0 SiLU(gate) * up (Mixtral), 1 GELU(gate) * up; tmp [2][m][fmid] floats.
 * ns_mul_mat_id_q4_0_f32_host: the ggml-type host-buffer drop-in (expert_rows[e] = dst->opt[e]->data, ids = ids->data). */
NS_API int ns_mul_mat_id(const ns_weight* const* experts, int n_as, const int32_t* ids, int ids_stride, int id, int ids_on_device,
                         const float* act, int lda, float* dst, int ldo, int m, int flags, void* queue);
NS_API int ns_ffn_id(const ns_weight* const* gate, const ns_weight* const* down, const ns_weight* const* up, int n_as, int gelu,
                     const int32_t* ids, int ids_stride, int id, int ids_on_device, const float* act, int lda, float* tmp, float* dst,
                     int ldo, int m, void* queue);
/* the host-side grouping ns_mul_mat_id / ns_ffn_id perform, on its own (no device): order[m] = token indices sorted stably by expert
 * (the matrix_rows lists of ne_layers.c:7440-7449, flattened), span[2 * n_as] = per expert [begin, end) inside order.  Returns 1 when
 * the tokens already lie grouped (no gather / scatter needed), 0 otherwise, NS_E_INVALID on an expert id outside [0, n_as). */
NS_API int ns_moe_plan(const int32_t* ids, int ids_stride, int id, int m, int n_as, int* order, int* span);
NS_API int ns_mul_mat_id_q4_0_f32_host(const void* const* expert_rows, int n_as, size_t nb01, const int32_t* ids, int ids_stride,
                                       int id, const float* src1, float* dst, int ne00, int ne01, int ne11);

/* The two phases of a reference matmul node, separately (ne_compute_forward_mul_mat_q_f32: NE_TASK_INIT quantises src1
 * into wdata, NE_TASK_COMPUTE runs the dots; core/ne_layers.c:7143-7203):
 *   ns_prepare_activation  act[m][k] (device fp32) -> activation image in `workspace` (m <= 4 rows per image)
 *   ns_matmul_prepared     runs 1..3 weights against a prepared image.  mode: 0 plain, 1 concat ([nw][m][ldo] output,
 *                          ne_mul_qkv), 2 gate/up + SiLU*mul (ne_ffn_silu first half; aux may receive silu(gate)). */
NS_API int ns_prepare_activation(const ns_weight* w, const float* act, int lda, int m, void* workspace, void* queue);
NS_API int ns_matmul_prepared(const ns_weight* const* weights, int nw, int mode, const void* workspace, float* dst, int ldo,
                              int m, const float* bias, int bias_bcast, const float* residual, float* aux, void* queue);

/* CUDA-graph capture of a sequence of calls on one queue (replaces the reference's per-token graph rebuild +
 * ne_graph_compute, models/llama/llama.cpp:136-143 / core/ne_layers.c:11915): begin, issue ns_* device calls with
 * caller-provided workspaces (no allocation may happen while capturing), end -> executable graph handle. */
typedef struct ns_graph ns_graph;
NS_API int ns_graph_begin(void* queue);
NS_API ns_graph* ns_graph_end(void* queue);
NS_API int ns_graph_launch(ns_graph* g, void* queue);
NS_API void ns_graph_free(ns_graph* g);

/* The host drop-ins (bestla_*_forward, ns_mul_mat_*_host) upload and repack a host weight once and cache the device copy by
 * host address + a checksum sampled over the whole payload.  ns_host_cache_clear() releases every cached copy (call it when the
 * model context that owned the host weights is freed: the reference frees its weights with the context, model_files.h:1490-1499). */
NS_API void ns_host_cache_clear(void);
NS_API size_t ns_host_cache_entries(void);

/* ggml drop-in with HOST buffers: ne_compute_forward_mul_mat_q_f32 (ne_layers.c:7085) for NE_TYPE_Q4_0:
 * dst[ne11][ne01] = src1[ne11][ne00] x src0 rows.  src0 is uploaded/repacked once and cached by address. */
NS_API int ns_mul_mat_q4_0_f32_host(const void* src0_rows, size_t nb01, const float* src1, float* dst, int ne00, int ne01,
                                    int ne11);

/* ------------------------------------------------------------------ 3c. quantisers / packing API */
/* device RTN->Q4_0 (quantize_row_q4_0_reference, quantize.h:243): src f32 [n][k] device -> dst block_q4_0 rows device */
/* same for NE_TYPE_Q6_K weights (ne_layers.c:320-327) */
NS_API int ns_mul_mat_q6_K_f32_host(const void* src0_rows, size_t nb01, const float* src1, float* dst, int ne00, int ne01,
                                    int ne11);
NS_API int ns_device_quantize_q4_0(const float* src_dev, void* dst_dev, int n, int k, void* queue);
/* device activation quantiser exposed for parity tests: one of ns_comp; outputs are device buffers
 * q: [m][k] (int8/uint8), scale: [m][k/g] f32, zp: [m][k/g] int32 (u8 mode, else untouched) */
NS_API int ns_device_quantize_act(const float* act_dev, int lda, int m, int k, int group, int comp, void* q_dev,
                                  float* scale_dev, int* zp_dev, void* queue);

/* ---- device-resident Llama-family eval step (SURVEY 8 f.1) ----------------------------------------------------------
 * Mirrors model_eval for the llama architecture (models/llama/llama.cpp:190-720): embedding lookup, RMSNorm, fused
 * QKV / three matmuls (GQA), RoPE mode 0, fp16 KV cache, softmax attention, o-proj + residual, RMSNorm, SiLU FFN + residual,
 * final RMSNorm, lm_head, greedy argmax (lowest index on ties, model_utils.cpp:2963-2985).  Weights are ns_weight handles
 * (borrowed: they must outlive the context); norms and the embedding table are fp32 host arrays copied to the device.
 * One-token evals replay one CUDA graph; ns_llama_generate feeds each argmax to the next step on the device. */
typedef struct ns_llama ns_llama;
typedef struct ns_llama_hparams {
  int n_vocab, n_embd, n_head, n_head_kv, n_layer, n_ff, n_ctx;
  float norm_eps;   /* hparams.norm_eps   (<= 0: 1e-6)  */
  float rope_theta; /* hparams.freq_base  (<= 0: 10000) */
  float rope_scale; /* hparams.freq_scale (<= 0: 1)     */
} ns_llama_hparams;
enum ns_llama_tensor {
  NS_LT_TOK_EMBD = 0, /* others[0]  [n_vocab][n_embd] f32 */
  NS_LT_OUT_NORM = 1, /* others[1]  [n_embd] f32          */
  NS_LT_OUTPUT = 2,   /* others[2]  n_vocab x n_embd weight (any ns_weight format, incl. Q6_K) */
  NS_LT_ATTN_NORM = 3, NS_LT_WQ = 4, NS_LT_WK = 5, NS_LT_WV = 6, NS_LT_WO = 7, /* layers[il].norm[0], attn[0..3] */
  NS_LT_FFN_NORM = 8, NS_LT_W1 = 9, NS_LT_W2 = 10, NS_LT_W3 = 11               /* layers[il].norm[1], ffn[0..2]  */
};
NS_API ns_llama* ns_llama_create(const ns_llama_hparams* hp, void* queue);
NS_API void ns_llama_free(ns_llama* ctx);
NS_API int ns_llama_set_f32(ns_llama* ctx, int tensor, int layer, const float* host, size_t count);
NS_API int ns_llama_set_weight(ns_llama* ctx, int tensor, int layer, const ns_weight* w);
/* evaluate n_tokens new tokens after n_past cached ones; logits_host (nullable) gets the n_vocab logits of the LAST token,
 * next_token (nullable) its greedy pick.  Synchronous (host buffers). */
NS_API int ns_llama_eval(ns_llama* ctx, const int32_t* tokens, int n_tokens, int n_past, float* logits_host, int32_t* next_token);
/* greedy generation of n_new tokens starting with first_token at position n_past; out_tokens[i] = pick after step i */
NS_API int ns_llama_generate(ns_llama* ctx, int32_t first_token, int n_past, int n_new, int32_t* out_tokens);
/* Numerics of prompt evaluation.  Matmuls of up to 32 new tokens reproduce the reference's exact integer block sums (GEMV /
 * integer tensor cores); longer prompts run the bf16 tcgen05 GEMM (measured logit deviation <= 4e-2 of max|logit| on the toy
 * models of tests/test_gpu_llama.py, KV cache entries differ at bf16 precision).  on = 1 evaluates long prompts in pieces of 32
 * tokens instead: reference numerics for the whole prompt at about 1/6 of the prefill throughput. */
NS_API int ns_llama_set_exact_prefill(ns_llama* ctx, int on);
NS_API unsigned long long ns_llama_kv_bytes(const ns_llama* ctx);
/* Test / debug surfaces: what one layer's attention saw and wrote, so that it can be checked against a reference outside
 * the engine.  With a tap on `layer`, every eval (and every step of a one-token graph) copies, on the context's stream,
 *   qkv_dst  <- the layer's q | k | v before RoPE: [m][n_embd] | [m][kvd] | [m][kvd] floats (kvd = n_head_kv * head size),
 *   attn_dst <- the attention output [m][n_embd] floats,
 * both device pointers.  An eval of more than max_rows tokens fails.  layer < 0 removes the tap.  Setting or removing a tap
 * rebuilds the one-token graph; without a tap the enqueued work is unchanged. */
NS_API int ns_llama_set_tap(ns_llama* ctx, int layer, float* qkv_dst, float* attn_dst, int max_rows);
/* device pointers to the fp16 KV cache of `layer`: k and v are each [n_head_kv][n_ctx][head size] */
NS_API int ns_llama_kv_cache(const ns_llama* ctx, int layer, const void** k, const void** v);

/* ---- tensor-parallel exchange step over NVLink peer memory (SURVEY 8e) --------------------------------------------
 * One-shot sum all-reduce replacing reduce_add / ne_all_reduce (core/parallel_context.cpp:47, ne_layers.c:5466) for the
 * [M, n_embd] fp32 partials after o-proj / down-proj (llama.cpp:592,693).  One process per GPU: each creates a context,
 * the hosts exchange the ns_comm_get_handle blobs (e.g. torch.distributed all_gather) and call ns_comm_open_peers.
 * Every rank gets bit-identical sums (fixed rank order).  max_elems bounds n of later calls. */
typedef struct ns_comm ns_comm;
/* several ranks' communicators inside ONE process (loopback on one device, or one host process driving peer-enabled GPUs): wire
 * them by plain device pointers instead of cudaIpc handles; comms[r] is rank r */
NS_API int ns_comm_link_local(ns_comm* const* comms, int world);
NS_API size_t ns_comm_handle_bytes(void);
NS_API ns_comm* ns_comm_create(int rank, int world, size_t max_elems, void* queue);
NS_API int ns_comm_get_handle(ns_comm* c, void* handle_out);
NS_API int ns_comm_open_peers(ns_comm* c, const void* all_handles);
NS_API int ns_comm_all_reduce_f32(ns_comm* c, float* data, size_t n, const float* residual, void* queue);
NS_API int ns_comm_status(ns_comm* c);
NS_API void ns_comm_free(ns_comm* c);

/* core/layers/bestla_gemm.h:37-56 (C++ in the reference; same names/argument meaning, extern "C" here).
 * QuantType/ScaleDtype are raw BTLA_DTYPE values, CompType an ne_comp_type.  ThreadPool is ignored. */
NS_API size_t BTLAGemmPackBSize(size_t N, size_t K, size_t BlkSize, uint32_t QuantType, uint32_t ScaleDtype, bool isAsym,
                                int CompType, int* shuffle_indice);
NS_API bool BTLAGemmQuantPackB(void* PackedBuf, const float* FpData, size_t N, size_t K, size_t ldb, size_t BlkSize,
                               uint32_t QuantType, uint32_t ScaleDtype, bool isAsym, int CompType, bool isTrans,
                               void* ThreadPool);
NS_API bool BTLAGemmPackB(void* PackedBuf, const int8_t* QData, const float* Scales, const int8_t* Zp, size_t N, size_t K,
                          size_t ldb, size_t BlkSize, uint32_t QuantType, uint32_t ScaleDtype, bool isAsym, int CompType,
                          int* shuffle_indice, void* ThreadPool);
NS_API bool BTLAGemmUnPackB(float* FpData, const void* PackedBuf, size_t N, size_t K, size_t ldb, void* ThreadPool);
/* Tensor-parallel shard of a blob: bestla_split_weight (models/model_utils/model_files.h:1538-1562) -- unpack, slice the
 * [dst_k][dst_n] block at (k_rank, n_rank) (or the rank's third of each fused Q/K/V projection), re-quantise with the source
 * blob's attributes.  ns_split_weight_size gives the bytes `dst` must hold (0 = unsupported). Host only. */
NS_API size_t ns_split_weight_size(const void* src, size_t dst_n, size_t dst_k);
NS_API bool ns_split_weight(const void* src, void* dst, size_t src_n, size_t src_k, size_t dst_n, size_t dst_k, size_t n_rank,
                            size_t k_rank, bool qkv_fusion);
/* host Q4_0 row quantiser (ne_quantize_q4_0 path; quantize.h:243) for the weight-packing API */
NS_API void ns_quantize_row_q4_0(const float* x, void* y, int k);

#ifdef __cplusplus
}
#endif
#endif /* NS_B200_H */
