// mmq.cu — batched MUL_MAT on quantised weights (prefill / ubatches of more than 8 tokens), host dispatch.
// Replaces ggml_cuda_mul_mat_q (ggml-cuda/mmq.cu:71-143).
//   * K-quants (Q4_K / Q5_K / Q6_K): the tcgen05 tile kernel of mmq_tc.cu (tensor cores, TMEM accumulators, TMA staging),
//     integer-exact against the CPU oracle;
//   * Q4_0 / Q8_0 (per-32 f16 block scales): activations quantised like the CPU oracle (quantize.cu) and columns streamed
//     through the matvec kernel in groups of 8 (weights re-read from L2 / HBM per group).
#include "common.cuh"

bool    b200_mmq_tc_supported(int type, int64_t m, int64_t k, int64_t ncols);
int64_t b200_mmq_tc_workspace(int64_t k, int64_t ncols);
int     b200_mmq_tc(int type, const void * W, const float * X, int64_t x_col_stride, float * dst, int64_t ldd, int64_t m, int64_t k, int64_t ncols, void * workspace, void * stream);
bool    b200_mmq_tc_id_routable(int64_t n_expert, int64_t n_used, int64_t n_tok);
int64_t b200_mmq_tc_id_workspace(int64_t k, int64_t n_expert, int64_t n_used, int64_t n_tok);
int     b200_mmq_tc_id(int type, const void * as, int64_t expert_stride_bytes, const float * b, int64_t b_tok_stride, int64_t b_slot_stride, int64_t n_b1,
                       const int32_t * ids, int64_t ids_tok_stride, float * dst, int64_t dst_tok_stride, int64_t dst_slot_stride,
                       int64_t m, int64_t k, int64_t n_expert, int64_t n_used, int64_t n_tok, void * workspace, void * stream);

extern "C" int64_t b200_mul_mat_q_workspace(int type, int64_t m, int64_t k, int64_t ncols) {
    const int kind = b200_act_kind_for(type);
    if (kind < 0 || k <= 0 || k % 256 != 0 || ncols <= 0) return 0;
    const int64_t vec = ncols * act_col_bytes(kind, k);
    const int64_t tc = b200_mmq_tc_supported(type, m, k, ncols) ? b200_mmq_tc_workspace(k, ncols) : 0;
    return vec > tc ? vec : tc;
}

extern "C" int b200_mul_mat_q(int type, const void * W, const float * X, int64_t x_col_stride, float * dst, int64_t dst_col_stride,
                              int64_t m, int64_t k, int64_t ncols, void * workspace, void * stream) {
    return b200_mul_mat_q2(type, W, X, x_col_stride, dst, dst_col_stride, m, k, k, ncols, workspace, stream);
}
// k: length of the (padded) weight rows, a multiple of 256; k_valid <= k: elements that exist in X (padded weight layout, see b200_padded_k)
extern "C" int b200_mul_mat_q2(int type, const void * W, const float * X, int64_t x_col_stride, float * dst, int64_t dst_col_stride,
                               int64_t m, int64_t k, int64_t k_valid, int64_t ncols, void * workspace, void * stream) {
    const int kind = b200_act_kind_for(type);
    if (kind < 0) { b200_set_error("mul_mat_q: unsupported weight type %d", type); return B200_ERR_UNSUPPORTED; }
    if (!workspace || ((uintptr_t)workspace & 15)) { b200_set_error("mul_mat_q: workspace missing or unaligned"); return B200_ERR_INVALID; }
    if (k_valid == k && b200_mmq_tc_supported(type, m, k, ncols)) return b200_mmq_tc(type, W, X, x_col_stride, dst, dst_col_stride, m, k, ncols, workspace, stream);
    int s = b200_quantize_act2(kind, X, x_col_stride, workspace, k, k_valid, ncols, stream);
    if (s != B200_OK) return s;
    const int64_t colb = act_col_bytes(kind, k);
    for (int64_t c0 = 0; c0 < ncols; c0 += 8) {
        const int64_t nc = ncols - c0 < 8 ? ncols - c0 : 8;
        s = b200_mul_mat_vec_q(type, W, (const uint8_t *)workspace + c0 * colb, dst + c0 * dst_col_stride, dst_col_stride, nullptr, nullptr, m, k, nc, stream);
        if (s != B200_OK) return s;
    }
    return B200_OK;
}

// ---- MUL_MAT_ID prefill: the grouped tensor-core path (routing on the device, then mmq_tc.cu's GEMM with a per-expert row map) ----
// When it pays (profiles/r3_moe_prefill.jsonl: B200, 1000 W power limit, L2 overwritten before every call; per-column / grouped in us):
//   pairs per expert n_tok * n_used / n_expert >= 4.  Mixtral-8x7B (E 8, U 2): ffn_up 14336 x 4096 Q4_K 452 / 245 at 16 tokens, ffn_down
//   4096 x 14336 Q6_K 440 / 616 at 9 and 826 / 618 at 16; Qwen3-30B-A3B-like (E 128, U 8, 768 x 2048 Q4_K) 119 / 140 at 32 (2 pairs per
//   expert) and 223 / 171 at 64 (4).  (Mixtral ffn_up alone would already gain at 9 tokens, 267 / 183; its ffn_down would lose.)
// Never below 9 tokens: decode and the <= 8-token verify batches keep b200_mul_mat_id's one launch per op.
#define B200_MMID_MIN_TOK 9
#define B200_MMID_MIN_PAIRS_PER_EXPERT 4

extern "C" int64_t b200_mul_mat_id_q_workspace(int type, int64_t m, int64_t k, int64_t n_expert, int64_t n_used, int64_t n_tok) {
    if (type != B200_TYPE_Q4_K && type != B200_TYPE_Q5_K && type != B200_TYPE_Q6_K) return 0;
    if (n_tok < B200_MMID_MIN_TOK || n_tok * n_used < B200_MMID_MIN_PAIRS_PER_EXPERT * n_expert || !b200_mmq_tc_id_routable(n_expert, n_used, n_tok) || !b200_mmq_tc_supported(type, m, k, n_tok)) return 0;
    return b200_mmq_tc_id_workspace(k, n_expert, n_used, n_tok);
}

extern "C" int b200_mul_mat_id_q(int type, const void * as, int64_t expert_stride_bytes, const float * b, int64_t b_tok_stride, int64_t b_slot_stride, int64_t n_b1,
                                 const int32_t * ids, int64_t ids_tok_stride, float * dst, int64_t dst_tok_stride, int64_t dst_slot_stride,
                                 int64_t m, int64_t k, int64_t n_expert, int64_t n_used, int64_t n_tok, void * workspace, void * stream) {
    // b200_mul_mat_id's argument checks: when they fail, that call reports the error
    const bool args_ok = as && b && ids && dst && m > 0 && n_b1 > 0 && !((uintptr_t)as & 15) && !((uintptr_t)b & 15) && !(b_tok_stride & 3) && !(b_slot_stride & 3) &&
                         !(expert_stride_bytes & 15) && !((uintptr_t)dst & 3);
    if (!args_ok || b200_mul_mat_id_q_workspace(type, m, k, n_expert, n_used, n_tok) == 0)
        return b200_mul_mat_id(type, as, expert_stride_bytes, b, b_tok_stride, b_slot_stride, n_b1, ids, ids_tok_stride, dst, dst_tok_stride, dst_slot_stride,
                               m, k, n_expert, n_used, n_tok, stream);
    if (b200_device_count() <= 0) { b200_set_error("no CUDA device"); return B200_ERR_CUDA; }
    if (!workspace || ((uintptr_t)workspace & 255)) { b200_set_error("mul_mat_id_q: workspace missing or not 256-byte aligned"); return B200_ERR_INVALID; }
    return b200_mmq_tc_id(type, as, expert_stride_bytes, b, b_tok_stride, b_slot_stride, n_b1, ids, ids_tok_stride, dst, dst_tok_stride, dst_slot_stride,
                          m, k, n_expert, n_used, n_tok, workspace, stream);
}
