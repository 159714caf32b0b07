/*
 * b200_ops.h — C-ABI of libb200ops.so: the hand-written sm_100a kernels for the GGUF-quantized
 * decode / prefill hot path.  Plain pointers and sizes only (device pointers unless stated);
 * no ggml, no torch, no C++ types.  Every entry point names the reference function it replaces
 * (paths relative to /root/reference/llama.cpp/).
 *
 * The ggml backend plug-in (include/ggml_b200.h, libggml-b200.so) is a thin adapter that maps
 * ggml_cgraph nodes onto these calls; tests/ and bench.py bind this header with ctypes.
 *
 * Conventions
 *   - tensor data use ggml's in-memory formats (ggml/src/ggml-common.h:170-344) unless a
 *     function says "repacked" (see b200_repack_rows).
 *   - all launches are asynchronous on `stream` (a cudaStream_t passed as void*).
 *   - return value: B200_OK or a negative b200_status; nothing aborts the process
 *     (the reference's CUDA_CHECK aborts: ggml-cuda/common.cuh:142-150).
 *   - there is NO CPU fallback: without a CUDA device every compute call returns B200_ERR_CUDA.
 */
#ifndef B200_OPS_H
#define B200_OPS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#  define B200_API __declspec(dllexport)
#else
#  define B200_API __attribute__((visibility("default")))
#endif

enum b200_status {
    B200_OK              =  0,
    B200_ERR_UNSUPPORTED = -1,   /* type / shape not handled by the hot path               */
    B200_ERR_INVALID     = -2,   /* bad argument (alignment, size not a block multiple ...) */
    B200_ERR_CUDA        = -3,   /* CUDA runtime error (see b200_last_error)                */
};

/* numerically equal to enum ggml_type (ggml/include/ggml.h:377-418) */
enum b200_type {
    B200_TYPE_F32  = 0,
    B200_TYPE_F16  = 1,
    B200_TYPE_Q4_0 = 2,
    B200_TYPE_Q5_0 = 6,
    B200_TYPE_Q8_0 = 8,
    B200_TYPE_Q4_K = 12,
    B200_TYPE_Q5_K = 13,
    B200_TYPE_Q6_K = 14,
    /* formats only the wide kernels (b200_mul_mat_vec_wide / b200_mul_mat_id / b200_get_rows_q) read, in ggml's own block layout */
    B200_TYPE_Q4_1   = 3,
    B200_TYPE_Q5_1   = 7,
    B200_TYPE_Q2_K   = 10,
    B200_TYPE_Q3_K   = 11,
    B200_TYPE_IQ4_NL = 20,
    B200_TYPE_IQ4_XS = 23,
    B200_TYPE_MXFP4  = 39,
};

/* ---- library / device ------------------------------------------------------------------ */
B200_API int         b200_abi_version(void);               /* bumps on any signature change   */
B200_API int         b200_device_count(void);              /* 0 when no CUDA device            */
B200_API int         b200_device_sm_count(int device);
B200_API const char *b200_last_error(void);                /* thread-local, never NULL         */
B200_API int64_t     b200_kernel_launches(void);           /* kernels launched by this library */
/* B200_TRACE=1 (read once per process): CTA 0 and the last CTA of every decode matvec / fused attention launch record a timeline —
 * 12 x u64 per record: [0] %globaltimer at entry, [1..6] clock64 stamps, [8] launch info, [10] clock64 at exit, [11] %globaltimer at
 * exit (layout: csrc/common.cuh, reader: tools/trace_decode.py).  The dump copies up to max_records records out, resets the counter
 * and returns the number copied.  Debugging aid; not part of the compute interface. */
B200_API int         b200_mmv_trace_dump(unsigned long long * out, int max_records);
B200_API int         b200_fa_trace_dump(unsigned long long * out, int max_records);

/* block geometry of a weight / cache type: elements and bytes per block, bytes per row of k */
B200_API int64_t b200_block_elems(int type);
B200_API int64_t b200_block_bytes(int type);
B200_API int64_t b200_row_bytes(int type, int64_t k);

/* ---- weight repack (load time) --------------------------------------------------------- *
 * Q4_0 / Q8_0 / Q6_K blocks are 18 / 34 / 210 bytes, which defeats 16-byte loads
 * (ggml-cuda reads them with 2-/4-byte loads: vecdotq.cuh:18-29).  We permute the bytes
 * INSIDE each row, in place, into a structure-of-arrays row:
 *     Q4_0: [qs 16B x nb][d f16 x nb]          Q8_0: [qs 32B x nb][d f16 x nb]
 *     Q6_K: [ql 128B x nb][qh 64B x nb][scales 16B x nb][d f16 x nb]
 * Row size and row offsets are unchanged, so ggml views / strides stay valid.  Q4_K / Q5_K
 * (144 / 176-byte blocks) are left as they are.  b200_unpack_rows is the exact inverse.
 * Replaces nothing in ggml-cuda; plays the role ggml-cpu/repack.cpp plays for the CPU backend. */
B200_API int b200_repack_rows(int type, void *rows, int64_t nrows, int64_t k, void *stream);
B200_API int b200_unpack_rows(int type, void *rows, int64_t nrows, int64_t k, void *stream);
B200_API int b200_type_is_repacked(int type);              /* 1 for Q4_0/Q5_0/Q8_0/Q6_K       */
/* Rows of the 32-element block types whose k is not a multiple of 256 (Qwen2-72B's ffn_down: k = 29568, where the reference
 * quantiser falls back from Q4_K / Q6_K to Q5_0 / Q8_0, src/llama-quant.cpp:442-470) live in a private layout padded with zero
 * blocks (d = 0) to b200_padded_k(type, k); row stride = b200_row_bytes(type, b200_padded_k).  Out of place (dst != src):
 * forward = ggml rows -> repacked + padded, inverse = back.  Q5_0 repacked row: [qs 16B x nb][qh 4B x nb][d f16 x nb]. */
B200_API int64_t b200_padded_k(int type, int64_t k);
B200_API int b200_repack_rows_padded(int type, const void *src, void *dst, int64_t nrows, int64_t k, int inverse, void *stream);

/* ---- activation quantisation (replaces quantize_row_q8_1_cuda, ggml-cuda/quantize.cu:148-160)
 * We quantise the way the CPU ORACLE does, so integer partial sums are bit-identical:
 *   K-quant weights  -> q8_K: 256-wide, iscale=-127/max, f32 d, bsums/16 (ggml-quants.c:2555-2592)
 *   Q4_0/Q8_0 weights-> q8_0: 32-wide, d=max/127 as f16, RNE (ggml-cpu/arch/x86/quants.c:290-360)
 * Output is an SoA "act buffer" per column (all sections 16-byte aligned):
 *   kind 0 (q8_K): int8 qs[k] | float d[k/256] | int16 bsums[k/16]
 *   kind 1 (q8_0): int8 qs[k] | float d[k/32] (value of the f16-rounded scale) | int16 bsum[k/32]
 * b200_act_col_bytes gives the per-column stride. */
B200_API int     b200_act_kind_for(int weight_type);       /* 0 = q8_K, 1 = q8_0, <0 unsupported */
B200_API int64_t b200_act_col_bytes(int kind, int64_t k);
B200_API int64_t b200_act_d_offset(int kind, int64_t k);
B200_API int64_t b200_act_bsum_offset(int kind, int64_t k);
B200_API int b200_quantize_act(int kind, const float *x, int64_t x_col_stride /* floats */,
                               void *act, int64_t k, int64_t ncols, void *stream);
/* ... for a padded weight layout: the act buffer covers k elements, of which only the first k_valid exist in x (the rest are 0) */
B200_API int b200_quantize_act2(int kind, const float *x, int64_t x_col_stride, void *act, int64_t k, int64_t k_valid, int64_t ncols, void *stream);

/* fused RMS_NORM * weight -> act buffer (and optionally the f32 normalised row too);
 * replaces rms_norm_f32<…,do_multiply> + quantize_q8_1 (norm.cu:107-164, quantize.cu:4-48) */
B200_API int b200_rms_norm_quantize(const float *x, const float *w, float *y_or_null, void *act0, int kind0,
                                    void *act1_or_null, int kind1, int64_t k, int64_t ncols, float eps, void *stream);

/* ---- MUL_MAT, decode matvec (replaces ggml_cuda_mul_mat_vec_q, mmvq.cu:500-570,139-226) -
 * dst[c][r] = sum_k W[r][k] * x[c][k] (+ bias[r]) (+ residual[c][r]),  ncols <= 8
 *   W        : m rows of `type` (repacked for Q4_0/Q5_0/Q8_0/Q6_K), row stride b200_row_bytes(type,k), k % 256 == 0 (padded layout otherwise),
 *              16-byte aligned, readable up to the next 16-byte boundary past the end
 *   act      : act buffer of kind b200_act_kind_for(type), ncols columns
 *   dst      : f32, column stride dst_col_stride floats
 *   bias     : f32 [m] or NULL (Qwen2 QKV bias, binbcast.cu)   residual: f32 like dst or NULL */
B200_API int b200_mul_mat_vec_q(int type, const void *W, const void *act, float *dst, int64_t dst_col_stride,
                                const float *bias, const float *residual,
                                int64_t m, int64_t k, int64_t ncols, void *stream);

/* several weight matrices against the same act buffer in ONE launch (fused QKV / gate+up):
 * descriptors live in device or pinned host memory; n_mats <= 4 */
typedef struct b200_mmv_desc {
    const void  *W;        /* weights of `type`                         */
    float       *dst;      /* f32 output [ncols][m] (col stride = m)    */
    const float *bias;     /* optional                                  */
    int64_t      m;
    int32_t      type;
    int32_t      _pad;
} b200_mmv_desc;
B200_API int b200_mul_mat_vec_q_multi(const b200_mmv_desc *descs, int n_mats, const void *act_q8K, const void *act_q80,
                                      int64_t k, int64_t ncols, void *stream);

/* general form: up to 4 matrices (or gate+up with SwiGLU) against one activation, with the activation
 * optionally produced INSIDE the kernel prologue from f32 (act_source 1) or from f32 through RMS_NORM * weight
 * (act_source 2) — fuses rms_norm + mul + quantize_q8 + mul_mat_vec_q (+ bias / residual / SwiGLU) into one launch
 * (the reference runs 3-5 kernels: norm.cu:444-495, quantize.cu:148-160, mmvq.cu:500-570, binbcast.cu, unary.cu:291) */
typedef struct b200_mmv_launch {
    b200_mmv_desc mats[4];
    const float  *residual[4];      /* optional, same layout as the mat's dst                        */
    int64_t       dst_col_stride[4];/* floats; 0 = m                                                  */
    int32_t       n_mats;
    int32_t       swiglu;           /* 1: mats[0] = gate, mats[1] = up, result in mats[0].dst         */
    int64_t       k, ncols;
    int32_t       act_source;       /* 0: act_q8K/act_q80 buffers, 1: quantise x, 2: rms_norm(x)*norm_w then quantise */
    float         eps;
    const void   *act_q8K, *act_q80;
    const float  *x;  int64_t x_col_stride;
    const float  *norm_w;
    float        *y_out;            /* optional f32 copy of the (normalised) activation [ncols][k]    */
    int64_t       k_valid;          /* 0 = k; else: x holds only k_valid elements per column, the weights are padded to k (zero blocks) */
} b200_mmv_launch;
B200_API int b200_mul_mat_vec_q_launch(const b200_mmv_launch *launch, void *stream);

/* gate & up matvec + SwiGLU in one launch: dst[c][r] = silu(Wg[r].x[c]) * (Wu[r].x[c])
 * (replaces 2x mul_mat_vec_q + unary_gated_op_kernel, unary.cu:209-230) */
B200_API int b200_mul_mat_vec_q_swiglu(int type_gate, const void *Wg, int type_up, const void *Wu,
                                       const void *act_q8K, const void *act_q80, float *dst,
                                       int64_t m, int64_t k, int64_t ncols, void *stream);

/* ---- the wide kernels: more weight formats, MUL_MAT_ID, GET_ROWS on quantised tables (SURVEY.md §8 f2 / f3 / f4) ------------------
 * One format-generic matvec (csrc/mmvq_ext.cu, per-format arithmetic in csrc/extfmt.cuh) for what the tuned kernels above do not carry.
 * Weight layouts: Q4_1 / Q5_1 / Q2_K / Q3_K / IQ4_NL / IQ4_XS / MXFP4 in ggml's block layout (ggml-common.h:176-300,414-428), any
 * k that is a multiple of the block size; Q4_0 / Q5_0 / Q8_0 / Q4_K / Q5_K / Q6_K as everywhere in this library ("repacked" for the
 * first three and Q6_K), k % 256 == 0 (Q6_K: k % 512 == 0).  Activations are f32: every CTA quantises the column it needs in its
 * prologue the way the CPU oracle does (q8_0 / q8_1 / q8_K by the weight's vec_dot_type, ggml-cpu/ggml-cpu.c:209-303), so integer
 * sums match the oracle's and no activation buffer exists in HBM.  Replaces the remaining vec_dot_*_q8_1 of ggml-cuda/vecdotq.cuh
 * behind mul_mat_vec_q (mmvq.cu:139-226). */
B200_API int     b200_wide_type_supported(int type);                 /* 1 for the 13 formats above                      */
B200_API int     b200_wide_shape_supported(int type, int64_t k);     /* 1 if rows of k elements of `type` can be read   */
B200_API int64_t b200_wide_row_bytes(int type, int64_t k);
/* dst[c][r] = sum_k W[r][k] x[c][k] (+ bias[r]) (+ residual[c][r]); x f32 [ncols][k] with column stride x_col_stride floats (16-byte
 * aligned columns); any ncols (one pass over the weights per group of up to 8 columns) */
B200_API int b200_mul_mat_vec_wide(int type, const void *W, const float *x, int64_t x_col_stride, float *dst, int64_t dst_col_stride,
                                   const float *bias, const float *residual, int64_t m, int64_t k, int64_t ncols, void *stream);
/* MUL_MAT_ID — mixture-of-experts routing (replaces ggml_cuda_mul_mat_id, ggml-cuda.cu:2064-2205; contract ggml.c:3064-3106):
 *   dst[t][s][:] = as[ids[t][s]] * b[t][s % n_b1]     t < n_tok, s < n_used
 *   as  : n_expert matrices of m rows (layout as above), expert e at as + e * expert_stride_bytes
 *   b   : f32, column (t, j) at b + t * b_tok_stride + j * b_slot_stride (floats), n_b1 = 1 (up / gate: shared) or n_used (down)
 *   ids : i32 on the DEVICE, (t, s) at ids[t * ids_tok_stride + s]; read by the kernel — no device->host synchronisation
 *         (the reference copies ids to the host and synchronises per op: ggml-cuda.cu:2115-2125).  Out-of-range ids write nothing.
 *   dst : f32, row block (t, s) at dst + t * dst_tok_stride + s * dst_slot_stride (floats) */
B200_API int b200_mul_mat_id(int type, const void *as, int64_t expert_stride_bytes, const float *b, int64_t b_tok_stride, int64_t b_slot_stride, int64_t n_b1,
                             const int32_t *ids, int64_t ids_tok_stride, float *dst, int64_t dst_tok_stride, int64_t dst_slot_stride,
                             int64_t m, int64_t k, int64_t n_expert, int64_t n_used, int64_t n_tok, void *stream);
/* MUL_MAT_ID for prefill: the same contract and arguments as b200_mul_mat_id, plus a workspace.  For ubatches of at least 9 tokens
 * with at least 4 (token, slot) pairs per expert (n_tok * n_used >= 4 * n_expert: where it measured faster) on Q4_K / Q5_K / Q6_K experts whose shape the tensor-core MUL_MAT takes (b200_mul_mat_q: k % 256 == 0, Q6_K k % 2048 == 0, not
 * switched off by B200_MMQ_DISABLE_TC), with n_expert <= 256, n_tok * n_used <= 16384 and b200_mul_mat_id's alignment rules, it runs
 * three kernels: a routing kernel groups the (token, slot) pairs by expert ON THE DEVICE (stable: increasing (t, s) inside an expert;
 * ids outside [0, n_expert) dropped), the activations are quantised to q8_K gathered in that order, and the tensor-core GEMM reads
 * each expert's weights once per 128 pairs.  Every other call is exactly b200_mul_mat_id.  No device->host synchronisation (the
 * reference sorts on the host: ggml-cuda/mmq.cu:145-228), so a captured CUDA graph stays valid when the ids change between replays.
 * b200_mul_mat_id_q_workspace returns 0 exactly when the call takes b200_mul_mat_id (workspace may then be NULL); otherwise the
 * workspace (256-byte aligned) must hold that many bytes. */
B200_API int64_t b200_mul_mat_id_q_workspace(int type, int64_t m, int64_t k, int64_t n_expert, int64_t n_used, int64_t n_tok);
B200_API int b200_mul_mat_id_q(int type, const void *as, int64_t expert_stride_bytes, const float *b, int64_t b_tok_stride, int64_t b_slot_stride, int64_t n_b1,
                               const int32_t *ids, int64_t ids_tok_stride, float *dst, int64_t dst_tok_stride, int64_t dst_slot_stride,
                               int64_t m, int64_t k, int64_t n_expert, int64_t n_used, int64_t n_tok, void *workspace, void *stream);
/* GET_ROWS on a quantised table: dst row i = de-quantised row ids[i] of src (replaces k_get_rows, ggml-cuda/getrows.cu:5-67; values
 * bit-identical to ggml's dequantize_row_*: products rounded separately).  The token-embedding lookup on the device. */
B200_API int b200_get_rows_q(int type, const void *src, int64_t src_row_stride_bytes, int64_t nrows, const int32_t *ids, float *dst,
                             int64_t dst_row_stride /* floats */, int64_t ncols, int64_t n_ids, void *stream);

/* Mixture-of-experts router glue (llama.cpp/src/llama-graph.cpp build_moe_ffn; csrc/glue_ext.cu): with these a Mixtral-style FFN stays on the
 * device from its RMS_NORM to the residual ADD.  Numerics are the CPU oracle's (ggml-cpu/ops.cpp): double-precision sums, the reference's
 * exchange sort (tie order is part of TOP_K's contract).  Strides in elements unless stated.
 *   b200_binary_strided : dst = a op b with ggml's broadcasting (op 0 add, 1 mul, 2 div); ne / nb as in ggml (nb in BYTES); replaces the strided and
 *                         broadcast cases of k_bin_bcast (binbcast.cu:26-93): the expert-weight MUL ([E,n_used,n_tok] * [1,n_used,n_tok]), the DIV of the
 *                         weight normalisation and the ADDs over expert slices (views with a row stride of n_used * E)
 *   b200_soft_max_rows  : SOFT_MAX without mask (softmax.cu:47-165)       b200_argsort_rows : ARGSORT (argsort.cu)     b200_sum_rows : sumrows.cu
 *   b200_get_rows_f32_batched : dst[:, i, b] = src[:, ids[i, b], b] (getrows.cu, batched)      b200_mul_mat_f32 : the f32 router matmul (ffn_gate_inp) */
B200_API int b200_binary_strided(int op, const float *a, const int64_t *a_nb, const float *b, const int64_t *b_ne, const int64_t *b_nb,
                                 float *dst, const int64_t *ne, const int64_t *d_nb, void *stream);
B200_API int b200_soft_max_rows(const float *x, int64_t x_row_stride, float *y, int64_t y_row_stride, int64_t ncols, int64_t nrows, float scale, void *stream);
B200_API int b200_argsort_rows(const float *x, int64_t x_row_stride, int32_t *idx, int64_t idx_row_stride, int64_t ncols, int64_t nrows, int descending, void *stream);
B200_API int b200_sum_rows(const float *x, int64_t x_row_stride, float *y, int64_t ncols, int64_t nrows, void *stream);
B200_API int b200_get_rows_f32_batched(const float *src, int64_t src_row_stride, int64_t src_batch_stride, int64_t n_src_rows, const int32_t *ids, int64_t ids_batch_stride,
                                       float *dst, int64_t dst_row_stride, int64_t dst_batch_stride, int64_t ncols, int64_t n_ids, int64_t n_batch, void *stream);
/* SCALE / SILU / SIGMOID (op 0 / 1 / 2) on contiguous f32: the unary ops of MoE gating variants (shared-expert gates, weight scaling); unary.cu / scale.cu */
B200_API int b200_unary(int op, const float *x, float *y, int64_t n, float s, float b, void *stream);
B200_API int b200_mul_mat_f32(const float *W, int64_t w_row_stride, const float *x, int64_t x_col_stride, float *dst, int64_t dst_col_stride,
                              int64_t m, int64_t k, int64_t ncols, void *stream);

/* Attention WITHOUT -fa (llama-graph.cpp build_attn_mha, non-flash branch; llama-box's default): KQ = K^T Q and KQV = V^T softmax(KQ) are batched
 * MUL_MATs over f16 views of the KV cache (K permuted, V stored TRANSPOSED by an element-wise SET_ROWS, llama-kv-cache-unified.cpp:1157-1167), with a masked
 * SOFT_MAX in between and a CONT of the permuted result.  Replaces the cuBLAS batched route of ggml-cuda (ggml-cuda.cu:1800-1977), soft_max_f32 with mask
 * (softmax.cu:47-165), k_set_rows for one-element rows and cpy/cont.  Numerics: the CPU oracle's (f32 operand rounded to f16, f32 accumulation).
 *   b200_mul_mat_f16   : dst[i0, i1, i2] = sum_k A[k, i0, i2 / r2] * f16(B[k, i1, i2]); A f16 with byte strides a_nb1 / a_nb2 and a_ne2 batches (GQA broadcast),
 *                        B f32 (b_nb1 / b_nb2 bytes), dst f32 (row i1 at d_nb1, batch at d_nb2 bytes)
 *   b200_soft_max_mask : x, y f32 [ncols, n_tok, n_head] contiguous; mask f32 / f16, row t at t * mask_row_stride elements; ALiBi slopes from max_bias
 *   b200_scatter_rows1 : dst[ids[i]] = src[i] (dst F16 or F32)                    b200_binary_strided(op 3) : CONT */
B200_API int b200_mul_mat_f16(const void *A, int64_t a_nb1, int64_t a_nb2, int64_t a_ne2, const float *B, int64_t b_nb1, int64_t b_nb2, float *dst, int64_t d_nb1, int64_t d_nb2,
                              int64_t m, int64_t n, int64_t n_batch, int64_t k, void *stream);
B200_API int b200_soft_max_mask(const float *x, float *y, const void *mask, int mask_is_f16, int64_t mask_row_stride, int64_t ncols, int64_t n_tok, int64_t n_head,
                                float scale, float max_bias, void *stream);
B200_API int b200_scatter_rows1(const float *src, const int64_t *ids, void *dst, int dst_type, int64_t n, int64_t n_dst, void *stream);

/* KV cache type q4_0 (`-ctk q4_0 -ctv q4_0`): the cache keeps ggml's native 18-byte blocks.  SET_ROWS writes what ggml's from_float writes
 * (ggml-quants.c quantize_row_q4_0_ref; replaces k_set_rows_quant<block_q4_0>, ggml-cuda/set-rows.cu:13-52); FLASH_ATTN_EXT follows the CPU
 * oracle (q8_0 query x Q4_0 K in integers, f32 online softmax, V expanded to f32; replaces the q4_0-q4_0 flash_attn_vec_ext instances,
 * ggml-cuda/fattn.cu:184).  Arguments as b200_set_rows / b200_flash_attn_ext; head size 64 or 128; no workspace. */
B200_API int b200_set_rows_q4_0(const float *src, int64_t src_row_stride /* floats */, const int64_t *ids, void *dst, int64_t dst_row_stride /* bytes */,
                                int64_t ncols, int64_t nrows, void *stream);
B200_API int b200_flash_attn_q4_0(const float *q, int64_t q_tok_stride, int64_t q_head_stride, const void *k, int64_t k_row_stride, int64_t k_head_stride,
                                  const void *v, int64_t v_row_stride, int64_t v_head_stride, const void *mask, int64_t mask_row_stride, float *dst,
                                  int64_t d, int64_t n_head, int64_t n_head_kv, int64_t n_tok, int64_t n_kv, float scale, float max_bias, float logit_softcap, void *stream);

/* FLASH_ATTN_EXT for any head size that is a multiple of 32 up to 256 (Gemma 256, Phi 96, ... — b200_flash_attn_ext carries 64 and 128) over an F16, Q8_0 or
 * Q4_0 cache in ggml's layout; wide path, arguments as b200_flash_attn_ext, no workspace (replaces the other head sizes of fattn.cu:271-338) */
B200_API int b200_flash_attn_any(int kv_type, const float *q, int64_t q_tok_stride, int64_t q_head_stride, const void *k, int64_t k_row_stride, int64_t k_head_stride,
                                 const void *v, int64_t v_row_stride, int64_t v_head_stride, const void *mask, int64_t mask_row_stride, float *dst,
                                 int64_t d, int64_t n_head, int64_t n_head_kv, int64_t n_tok, int64_t n_kv, float scale, float max_bias, float logit_softcap, void *stream);

/* ---- MUL_MAT, batched / prefill (replaces ggml_cuda_mul_mat_q, mmq.cu:71-143) -----------
 * dst[c][r] for any ncols; X is f32 [ncols][k].  Internally: activation quantisation as above,
 * then tiles on the tensor cores (tcgen05, TMEM accumulators) when ncols >= B200_MMQ_MIN_COLS,
 * else column groups of 8 through the matvec kernel.  `workspace` must hold
 * b200_mul_mat_q_workspace(type,m,k,ncols) bytes. */
B200_API int64_t b200_mul_mat_q_workspace(int type, int64_t m, int64_t k, int64_t ncols);
B200_API int b200_mul_mat_q(int type, const void *W, const float *X, int64_t x_col_stride,
                            float *dst, int64_t dst_col_stride, int64_t m, int64_t k, int64_t ncols,
                            void *workspace, void *stream);
/* ... for a padded weight layout: k = b200_padded_k(type, k_valid); X holds k_valid elements per column */
B200_API int b200_mul_mat_q2(int type, const void *W, const float *X, int64_t x_col_stride,
                             float *dst, int64_t dst_col_stride, int64_t m, int64_t k, int64_t k_valid, int64_t ncols,
                             void *workspace, void *stream);

/* ---- RMS_NORM (+MUL) (replaces ggml_cuda_op_rms_norm[_fused], norm.cu:420-495) ---------- */
B200_API int b200_rms_norm(const float *x, const float *w_or_null, float *y, int64_t ncols, int64_t nrows,
                           int64_t x_row_stride, int64_t y_row_stride, float eps, void *stream);

/* ---- ROPE (replaces ggml_cuda_op_rope, rope.cu:324-446) ---------------------------------
 * x,y: [n_tok][n_head][head_dim] f32 with strides in floats; pos i32 [n_tok];
 * mode 0 = NORM, 2 = NEOX.  theta is built iteratively like the CPU oracle (ops.cpp:6077-6086). */
typedef struct b200_rope_params {
    int32_t n_dims, mode, n_ctx_orig, _pad;
    float freq_base, freq_scale, ext_factor, attn_factor, beta_fast, beta_slow;
} b200_rope_params;
B200_API int b200_rope(const float *x, float *y, const int32_t *pos, const float *freq_factors_or_null,
                       int64_t head_dim, int64_t n_head, int64_t n_tok,
                       int64_t x_head_stride, int64_t x_tok_stride, int64_t y_head_stride, int64_t y_tok_stride,
                       const b200_rope_params *p, void *stream);

/* ---- SET_ROWS (KV store; replaces ggml_cuda_op_set_rows, set-rows.cu:166-275) ------------
 * dst row ids[i] <- convert(src row i);  dst_type F32 / F16 / Q8_0 (ggml-native layout) */
B200_API int b200_set_rows(const float *src, int64_t src_row_stride /* floats */, const int64_t *ids,
                           void *dst, int dst_type, int64_t dst_row_stride /* bytes */,
                           int64_t ncols, int64_t nrows, void *stream);

/* fused decode-step tail of the QKV projection: rope(q) in place, rope(k) -> K cache row,
 * v -> V cache row (replaces 2x rope + 2x set_rows launches) */
B200_API int b200_rope_kv_store(float *q, const float *k, const float *v, const int32_t *pos, const float *freq_factors_or_null,
                                const int64_t *kv_ids, void *k_cache, void *v_cache, int kv_type, int64_t kv_row_stride,
                                int64_t head_dim, int64_t n_head, int64_t n_head_kv, int64_t n_tok,
                                const b200_rope_params *p, void *stream);

/* same, with q roped out of place and separate K / V row-id tensors and row strides (what the ggml graph provides) */
B200_API int b200_rope_kv_store2(const float *q_src, float *q_dst, const float *k, const float *v, const int32_t *pos, const float *freq_factors_or_null,
                                 const int64_t *k_ids, const int64_t *v_ids, void *k_cache, void *v_cache, int kv_type,
                                 int64_t k_row_stride, int64_t v_row_stride, int64_t head_dim, int64_t n_head, int64_t n_head_kv, int64_t n_tok,
                                 const b200_rope_params *p, void *stream);

/* ---- FLASH_ATTN_EXT (replaces ggml_cuda_flash_attn_ext, fattn.cu:271-338) ----------------
 *   q    f32, element (d, tok, head) at q + tok*q_tok_stride + head*q_head_stride (floats)
 *   k,v  cache rows of kv_type (F16 or Q8_0): (pos, kv_head) at base + pos*row_stride + kv_head*head_stride (bytes)
 *   mask f16 [n_tok_padded][n_kv] (row stride mask_row_stride halves) or NULL; -inf = masked
 *   dst  f32 [n_tok][n_head][dv] contiguous
 *   workspace: b200_flash_attn_workspace(...) bytes for split-KV partials + completion counters; zero it ONCE
 *   (the counters reset themselves at the end of every launch) */
B200_API int64_t b200_flash_attn_workspace(int64_t dv, int64_t n_head, int64_t n_tok, int64_t n_kv);
B200_API int b200_flash_attn_ext(const float *q, int64_t q_tok_stride, int64_t q_head_stride,
                                 const void *k, int64_t k_row_stride, int64_t k_head_stride,
                                 const void *v, int64_t v_row_stride, int64_t v_head_stride,
                                 const void *mask, int64_t mask_row_stride, float *dst,
                                 int kv_type, int64_t dk, int64_t dv, int64_t n_head, int64_t n_head_kv,
                                 int64_t n_tok, int64_t n_kv, float scale, float max_bias, float logit_softcap,
                                 void *workspace, void *stream);

/* decode token (n_tok = 1): ROPE(q), ROPE(k) -> K cache cell k_ids[0], v -> V cache cell v_ids[0] and FLASH_ATTN_EXT over
 * n_kv cells in ONE launch (replaces rope x2 + set_rows x2 + flash_attn_vec + combine of the reference: ggml-cuda/rope.cu,
 * set-rows.cu, fattn.cu).  q_src/k_new/v_new: this token's projections, f32 [n_head|n_head_kv][hd]; q_dst receives the roped
 * query (a declared graph output); caches as in b200_flash_attn_ext with heads contiguous inside a cell. */
B200_API int b200_rope_kv_flash_attn(const float *q_src, float *q_dst, const float *k_new, const float *v_new, const int32_t *pos,
                                     const float *freq_factors_or_null, const int64_t *k_ids, const int64_t *v_ids,
                                     void *k_cache, void *v_cache, int kv_type, int64_t k_cell_stride, int64_t k_head_stride,
                                     int64_t v_cell_stride, int64_t v_head_stride, const void *mask_f16_or_null, float *dst,
                                     int64_t head_dim, int64_t n_head, int64_t n_head_kv, int64_t n_kv, const b200_rope_params *p,
                                     float scale, float max_bias, float softcap, void *workspace, void *stream);

/* the same with a per-token cos/sin table shared by all layers (the table depends on the position only): rope_tab = 2*head_dim
 * floats of caller scratch; tab_mode 0 = this launch computes the table and stores it there, 1 = an earlier launch for the same
 * token and rope parameters did.  rope_tab NULL = every launch computes its own. */
B200_API int b200_rope_kv_flash_attn2(const float *q_src, float *q_dst, const float *k_new, const float *v_new, const int32_t *pos,
                                      const float *freq_factors_or_null, const int64_t *k_ids, const int64_t *v_ids,
                                      void *k_cache, void *v_cache, int kv_type, int64_t k_cell_stride, int64_t k_head_stride,
                                      int64_t v_cell_stride, int64_t v_head_stride, const void *mask_f16_or_null, float *dst,
                                      int64_t head_dim, int64_t n_head, int64_t n_head_kv, int64_t n_kv, const b200_rope_params *p,
                                      float scale, float max_bias, float softcap, void *workspace, float *rope_tab, int tab_mode, void *stream);

/* ---- glue (replaces binbcast.cu, unary.cu:291, getrows.cu, cpy.cu) ----------------------- */
B200_API int b200_add(const float *a, const float *b, float *y, int64_t ncols, int64_t nrows, int64_t b_rows, void *stream);
B200_API int b200_mul(const float *a, const float *b, float *y, int64_t ncols, int64_t nrows, int64_t b_rows, void *stream);
B200_API int b200_swiglu(const float *gate, const float *up, float *y, int64_t n, void *stream);
B200_API int b200_get_rows_f32(const float *src, int64_t src_row_stride, const int32_t *ids, float *dst, int64_t ncols, int64_t n_ids, void *stream);
B200_API int b200_cpy_f32_f16(const float *src, void *dst_f16, int64_t n, void *stream);
B200_API int b200_argmax_f32(const float *x, int32_t *idx_out, int64_t n, int64_t nrows, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* B200_OPS_H */
