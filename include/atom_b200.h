/*
 * atom_b200.h -- C ABI of libatom_b200.so: the B200 (sm_100a) implementation of the efeslab/Atom W4A4 hot path.
 *
 * One entry point per function that the reference binds into Python through
 * pybind11 (/root/reference/e2e/punica-atom/punica/ops/csrc/punica_ops.cc:270-279).  Plain pointers and sizes only;
 * every pointer is a DEVICE pointer owned by the caller, outputs are pre-allocated by the caller (exactly as
 * punica/ops/__init__.py:21-219 does with torch.empty) and the library keeps no reference to them.
 *
 * Conventions
 *   - return value: 0 on success, negative ATOM_E_* otherwise; atom_last_error() returns a thread-local message.
 *     (The reference returns void and never checks cudaGetLastError; its KV ops raise via TORCH_CHECK.)
 *   - `stream` is a cudaStream_t passed as void*.  The reference launches on the legacy default stream; pass the
 *     caller's current stream (NULL = legacy default).  All entry points are asynchronous and graph-capturable
 *     (no allocation, no synchronisation; TMA descriptors are built on the host per call).
 *   - layouts are the reference's, unchanged (see DESIGN.md section 3).
 */
#ifndef ATOM_B200_H_
#define ATOM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define ATOM_API __attribute__((visibility("default")))
#else
#define ATOM_API
#endif

#define ATOM_OK 0
#define ATOM_E_INVALID (-1) /* bad shape / alignment / null pointer */
#define ATOM_E_CUDA (-2)    /* a CUDA runtime or driver call failed  */
#define ATOM_E_UNSUPPORTED (-3)

/* gemm flags */
#define ATOM_GEMM_AUTO 0u
#define ATOM_GEMM_NO_SPLITK 1u   /* bit-exact accumulation order (groups 0..G-1 then keeper) even for small M */
#define ATOM_GEMM_FORCE_TALL 2u  /* tokens on the MMA-M axis regardless of M */
#define ATOM_GEMM_FORCE_SKINNY 4u /* channels on the MMA-M axis (requires M <= 128 per tile; any M works) */
#define ATOM_GEMM_SPLITK2 16u     /* decode shapes: force a 2-way K split (default: chosen from the tile count) */
#define ATOM_GEMM_SPLITK4 32u     /* decode shapes: force a 4-way K split */
#define ATOM_GEMM_SPLITK8 64u     /* decode shapes, M <= 32: force an 8-way K split (cluster of 8) */
/* atom_gemm_i4_o16, atom_gemm_i4_o16_push and atom_gemm_i4_o4 reject any other bit with ATOM_E_INVALID */

ATOM_API int atom_version(void);
ATOM_API const char* atom_last_error(void);

/* Reorder.cuh:39-50 / punica/ops/__init__.py:137 -- the scale layout contract shared by quantise kernels and GEMM */
ATOM_API int atom_scale_index(int row);
ATOM_API int atom_scale_size(int rows);

/* replaces reorder_fp16_i4 (punica_ops.cc:251-260 -> run_reorder_fp16_i4<128,4096>, Reorder.cuh:205-228)
 *   hidden        f16 [seq_len, hidden_dim]      reorder_index i16 [hidden_dim]
 *   o_outliers    i8  [seq_len, 128]             o_norms       u8  [seq_len, (hidden_dim-128)/2]
 *   outlier_scales f16 [scale_size(seq_len)]     norm_scales   f16 [hidden_dim/128-1, scale_size(seq_len)]
 * hidden_dim: any multiple of 128 (the reference is compiled for 4096 only). */
ATOM_API int atom_reorder_fp16_i4(const void* hidden, const void* reorder_index, int seq_len, int hidden_dim, void* o_outliers,
                         void* o_norms, void* outlier_scales, void* norm_scales, void* stream);

/* replaces rmsnorm_fp16_i4 (punica_ops.cc:239-249 -> run_rmsnorm_fp16_i4<128,4096>, RMSNorm.cuh:255-285) */
ATOM_API int atom_rmsnorm_fp16_i4(const void* hidden, const void* weight, float eps, const void* reorder_index, int seq_len,
                         int hidden_dim, void* o_outliers, void* o_norms, void* outlier_scales, void* norm_scales,
                         void* stream);

/* EXTENSION (launch-count reduction, SURVEY.md 8 f4): the residual add of the decoder layer
 * (punica/models/llama.py:266-292, `hidden = residual + hidden`) folded into the following rmsnorm_fp16_i4:
 * sum_out = hidden + residual (FP16 RN, bit-identical to the separate add), then exactly rmsnorm_fp16_i4(sum_out, ...). */
ATOM_API int atom_add_rmsnorm_fp16_i4(const void* hidden, const void* residual, void* sum_out, const void* weight, float eps,
                             const void* reorder_index, int seq_len, int hidden_dim, void* o_outliers, void* o_norms,
                             void* outlier_scales, void* norm_scales, void* stream);

/* replaces activate_fp16_i4 (punica_ops.cc:73-80 -> run_activate_fp16_i4<128,11008>, Activate.cuh:194-218) */
ATOM_API int atom_activate_fp16_i4(const void* a, const void* b, int seq_len, int hidden_dim, void* o_outliers, void* o_norms,
                          void* outlier_scales, void* norm_scales, void* stream);

/* replaces dense_layer_gemm_i4_fp16 (punica_ops.cc:226-237 -> DenseLayerGEMM_i4<nv_half>, DenseLayerGEMM_i4.cu:723-793)
 *   a u8 [M,(K-128)/2]  b u8 [N,(K-128)/2]  a_scale f16 [K/128-1, scale_size(M)]  b_scale f16 [K/128-1, N]
 *   a_keeper i8 [M,128] b_keeper i8 [N,128] a_keeper_scale f16 [scale_size(M)]    b_keeper_scale f16 [N]
 *   d f16 [M,N].   K includes the 128 keeper channels (as in the e2e launcher).  N % 8 == 0, K % 128 == 0, K >= 256.
 * Bit-identity: every path accumulates the groups in the reference's order (0..G-1, keeper last) and is bit-identical to the
 * reference kernel, EXCEPT flags = ATOM_GEMM_AUTO with M <= 128 when the dispatcher splits K over a cluster (channel tiles
 * alone would not fill the GPU): the FP32 partials are then summed per K slice, <= 1 fp16 ulp on < 2 % of the outputs (inside
 * the operator's 1e-3 contract).  ATOM_GEMM_NO_SPLITK restores the reference's order at decode sizes.
 * The weights (b, b_scale, b_keeper, b_keeper_scale) are read before the preceding kernel on `stream` has completed
 * (programmatic dependent launch): they must not be written by the kernel launched immediately before this call. */
ATOM_API int atom_gemm_i4_o16(const void* a, const void* b, const void* a_scale, const void* b_scale, const void* a_keeper,
                     const void* b_keeper, const void* a_keeper_scale, const void* b_keeper_scale, void* d, int64_t M,
                     int64_t N, int64_t K, uint32_t flags, void* stream);

/* replaces dense_layer_gemm_i4_o4 (punica_ops.cc:211-224 -> DenseLayerGEMM_i4_o4, DenseLayerGEMM_i4_o4.cu:808-856)
 *   d u8 [M, N/2] (asymmetric INT4 per 128-column head), d_scale f16 [M, N/128, 2] = (scale, zero).  N % 128 == 0. */
ATOM_API int atom_gemm_i4_o4(const void* a, const void* b, const void* a_scale, const void* b_scale, const void* a_keeper,
                    const void* b_keeper, const void* a_keeper_scale, const void* b_keeper_scale, void* d,
                    void* d_scale, int64_t M, int64_t N, int64_t K, uint32_t flags, void* stream);

/* EXTENSION (launch-count reduction, SURVEY.md 8 f4): the q, k and v projections of LlamaAttention
 * (punica/models/llama.py:146-156: dense_layer_gemm_i4_fp16 for q, dense_layer_gemm_i4_o4 for k and v, same input) as ONE
 * launch over row-concatenated weights  b_qkv u8 [3H,(K-128)/2], b_scale_qkv f16 [K/128-1, 3H], b_keeper_qkv i8 [3H,128],
 * b_keeper_scale_qkv f16 [3H]  (rows [0,H) = q, [H,2H) = k, [2H,3H) = v).  Outputs are bit-identical to the three separate
 * calls: q f16 [M,H]; k, v u8 [M,H/2] with k_scale, v_scale f16 [M,H/128,2].  M <= 64: one decode-kernel launch whose
 * channel tile selects the epilogue; larger M: three launches on the row slices. */
ATOM_API int atom_gemm_i4_qkv(const void* a, const void* b_qkv, const void* a_scale, const void* b_scale_qkv, const void* a_keeper,
                     const void* b_keeper_qkv, const void* a_keeper_scale, const void* b_keeper_scale_qkv, void* q, void* k,
                     void* k_scale, void* v, void* v_scale, int64_t M, int64_t H, int64_t K, uint32_t flags, void* stream);

/* EXTENSION (launch-count reduction, SURVEY.md 8 f4): LlamaMLP's gate_proj, up_proj and activate_fp16_i4
 * (punica/models/llama.py:85-87) as ONE launch for decode batches (M <= 64; ATOM_E_UNSUPPORTED above): weights
 * row-concatenated  b_gu u8 [2I,(K-128)/2] (rows [0,I) = gate, [I,2I) = up), b_scale_gu f16 [K/128-1, 2I], b_keeper_gu
 * i8 [2I,128], b_keeper_scale_gu f16 [2I].  Outputs: the activation 4-tuple of activate_fp16_i4(gate, up) -- o_outliers i8
 * [M,128], o_norms u8 [M,(I-128)/2], outlier_scales f16 [scale_size(M)], norm_scales f16 [I/128-1, scale_size(M)] --
 * bit-identical to the three separate calls (both projections are rounded to FP16 before the activation, as there). */
ATOM_API int atom_gemm_i4_gateup_act(const void* a, const void* b_gu, const void* a_scale, const void* b_scale_gu, const void* a_keeper,
                            const void* b_keeper_gu, const void* a_keeper_scale, const void* b_keeper_scale_gu, void* o_outliers,
                            void* o_norms, void* outlier_scales, void* norm_scales, int64_t M, int64_t I, int64_t K, uint32_t flags,
                            void* stream);

/* Debug aid (no reference counterpart): when non-NULL, every GEMM CTA writes 128 clock64() stamps of its pipeline
 * stages to device_buffer[cta*128 ...] (layout in gemm_i4_sm100.cuh).  NULL switches tracing off. */
ATOM_API int atom_gemm_set_trace(void* device_buffer);

/* EXPERIMENTAL (no reference counterpart; not yet run on hardware): programmatic dependent launch.  When enabled (also via
 * ATOM_B200_PDL=1 in the environment) every kernel is launched with programmatic stream serialization: its prologue -- for
 * the GEMM including the first weight tiles -- overlaps the tail of the preceding kernel; everything that reads that
 * kernel's output waits on griddepcontrol.wait.  Results are unchanged.  Off by default. */
ATOM_API int atom_set_pdl(int enable);

/* replaces batch_decode_i4 (punica_ops.cc:82-120 -> FlashInferBatchDecodeKernel_i4<128>, flashinfer_impl.cuh:9-46)
 *   o,q f16 [B,H,128]  kv_data u8 [pages,L,2,H,P,64]  kv_param f16 [pages,L,2,H,P,2]
 *   kv_indptr i32 [B+1]  kv_indices i32 [nnz]  last_page_offset i32 [B] */
ATOM_API int atom_batch_decode_i4(void* o, const void* q, const void* kv_data, const void* kv_param, const void* kv_indptr,
                         const void* kv_indices, const void* last_page_offset, int num_layers, int layer_idx,
                         int num_heads, int page_size, int batch_size, void* stream);

/* EXTENSION (SURVEY.md 8 f3): the prefill attention the reference leaves as a placeholder
 * (punica/models/llama.py:171-190, SDPA over torch.randn K/V): causal attention of every prompt over its own just-quantised
 * K/V -- the o4 outputs of the k/v projections, x = nibble * scale - zero (quantization.cuh:76) -- with RoPE(theta 1e4) on q
 * and k at positions 0..len-1, head_dim 128.
 *   q f16 [T, H*128]; k, v u8 [T, H*64]; k_param, v_param f16 [T, H, 2]; seqlen_indptr i32 [B+1]; pos_of_token i32 [T];
 *   rope_table f32 [max_len, 64, 2] = (cos, sin)(pos * 1e4^(-i/64)); k_f16, v_f16 f16 [T, H*128] scratch (caller-owned,
 *   holds RoPE(dequant k) and dequant v afterwards); out f16 [T, H*128].  max_len >= the longest prompt. */
ATOM_API int atom_prefill_attention_i4(const void* q, const void* k, const void* k_param, const void* v, const void* v_param,
                              const void* seqlen_indptr, const void* pos_of_token, const void* rope_table, void* k_f16, void* v_f16,
                              void* out, int total_tokens, int batch_size, int max_len, int num_heads, void* stream);

/* EXTENSION (SURVEY.md 8e; the reference has no multi-GPU code): one-shot all-reduce (sum) of an FP16 vector over NVLink peer
 * memory for the tensor-parallel row-parallel projections.  peer_buffers: DEVICE array of `world` pointers to every rank's
 * receive buffer, f16 [3][world][slot_elems], every half initialised to 0x8000 (FP16 -0.0: the "not yet arrived" pattern;
 * a -0.0 input element is transmitted as +0.0), e.g. allocated and exchanged with torch.distributed._symmetric_memory;
 * state: local u32 [atom_allreduce_state_words()], zeroed once.  Every rank must make the same sequence of calls.
 * No flags, fences or barriers: the payload is its own arrival signal (three rotating buffers on a device-side call counter).
 * Graph-capturable; the sum is formed in rank order in FP32 and is bit-identical on all ranks. */
ATOM_API int atom_allreduce_push_f16(const void* in, void* out, const void* peer_buffers, void* state, int64_t numel,
                            int64_t slot_elems, int rank, int world, void* stream);
ATOM_API int atom_allreduce_state_words(void);

/* The same all-reduce with its two halves fused into the kernels around it (decode batches, M <= 64):
 *   atom_gemm_i4_o16_push            the row-parallel projection (o_proj / down_proj shard): atom_gemm_i4_o16 whose epilogue stores D
 *                                    into slot [call % 3][rank] of EVERY rank's receive buffer instead of a local tensor;
 *   atom_reduce_add_rmsnorm_fp16_i4  atom_add_rmsnorm_fp16_i4 whose `hidden` input is the sum over the ranks of those slots: each
 *                                    16-byte chunk is polled until its payload has arrived, summed in rank order in FP32 and rounded
 *                                    to FP16 (bit-identical to what atom_allreduce_push_f16 would have delivered), then added to the
 *                                    residual, normalised and quantised as usual.  hidden_dim % 1024 == 0.
 * The pair must be called in this order with the same (peer_buffers, state) and M x N = seq_len x hidden_dim; pairs and stand-alone
 * atom_allreduce_push_f16 calls on the same buffers may be mixed freely (one call counter). */
ATOM_API int atom_gemm_i4_o16_push(const void* a, const void* b, const void* a_scale, const void* b_scale, const void* a_keeper,
                          const void* b_keeper, const void* a_keeper_scale, const void* b_keeper_scale, const void* peer_buffers,
                          void* state, int64_t slot_elems, int rank, int world, int64_t M, int64_t N, int64_t K, uint32_t flags,
                          void* stream);
ATOM_API int atom_reduce_add_rmsnorm_fp16_i4(const void* peer_buffers, void* state, int64_t slot_elems, int rank, int world,
                                    const void* residual, void* sum_out, const void* weight, float eps, const void* reorder_index,
                                    int seq_len, int hidden_dim, void* o_outliers, void* o_norms, void* outlier_scales,
                                    void* norm_scales, void* stream);

/* replaces append_kv_i4 (punica_ops.cc:166-209 -> FlashInferAppendKvKernel_i4<128>, flashinfer_impl.cuh:73-96)
 *   k,v u8 [B,H,64]  k_param,v_param f16 [B,H,2] */
ATOM_API int atom_append_kv_i4(void* kv_data, void* kv_param, const void* kv_indptr, const void* kv_indices,
                      const void* last_page_offset, const void* k, const void* v, const void* k_param,
                      const void* v_param, int num_layers, int layer_idx, int num_heads, int page_size, int batch_size,
                      void* stream);

/* replaces init_kv_i4 (punica_ops.cc:122-164 -> FlashInferInitKvKernel_i4<128>, flashinfer_impl.cuh:48-71)
 *   k,v u8 [sum(len),H,64]  params f16 [sum(len),H,2]  seqlen_indptr i32 [B+1]; total_tokens = seqlen_indptr[B] */
ATOM_API int atom_init_kv_i4(void* kv_data, void* kv_param, const void* kv_indptr, const void* kv_indices,
                    const void* last_page_offset, const void* k, const void* v, const void* k_param,
                    const void* v_param, const void* seqlen_indptr, int total_tokens, int num_layers, int layer_idx,
                    int num_heads, int page_size, int batch_size, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ATOM_B200_H_ */
