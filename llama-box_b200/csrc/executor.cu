// executor.cu — graph executor: node list -> fused kernel launches -> CUDA-graph capture / replay.
// C-ABI in include/b200_graph.h.  Replaces ggml-cuda's evaluate_and_capture_cuda_graph / compute_forward
// (ggml/src/ggml-cuda/ggml-cuda.cu:2845-3010, 2207-2493), its RMS_NORM+MUL fusion (:2784-2843) and the
// graph-property check that decides on re-capture (:2726-2782).  Host code only; kernels live in the
// other translation units and are reached through the same C-ABI the tests use (b200_ops.h).
#include "common.cuh"
#include "../../include/b200_graph.h"
#include "mk.h"
#include "ropeutil.cuh"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <unordered_map>
#include <vector>

namespace {

inline bool is_weight_type(int t) { return t == B200_TYPE_Q4_0 || t == B200_TYPE_Q5_0 || t == B200_TYPE_Q8_0 || t == B200_TYPE_Q4_K || t == B200_TYPE_Q5_K || t == B200_TYPE_Q6_K; }
// the wide path (mmvq_ext.cu): formats beyond the tuned five, MUL_MAT_ID, GET_ROWS on quantised tables — GGML_B200_WIDE=1 (b200_graph.h)
inline bool wide_on() { static const bool on = [] { const char * e = getenv("GGML_B200_WIDE"); return e && *e && *e != '0'; }(); return on; }
inline bool is_wide_only_type(int t) { return t == B200_TYPE_Q4_1 || t == B200_TYPE_Q5_1 || t == B200_TYPE_Q2_K || t == B200_TYPE_Q3_K || t == B200_TYPE_IQ4_NL || t == B200_TYPE_IQ4_XS || t == B200_TYPE_MXFP4; }
inline int64_t nrows_of(const b200_tensor & t) { return t.ne[1] * t.ne[2] * t.ne[3]; }
inline int64_t nelem(const b200_tensor & t) { return t.ne[0] * t.ne[1] * t.ne[2] * t.ne[3]; }
inline int64_t elem_size(int type) {
    switch (type) { case B200_TYPE_F32: case B200_TYPE_I32: return 4; case B200_TYPE_F16: return 2; case B200_TYPE_I64: return 8; default: return 0; }
}
// fully contiguous f32/f16/int tensor in ggml's sense
inline bool contiguous(const b200_tensor & t) {
    const int64_t es = elem_size(t.type);
    if (es == 0) return false;
    int64_t s = es;
    for (int i = 0; i < 4; i++) { if (t.ne[i] != 1 && t.nb[i] != s) return false; s *= t.ne[i]; }
    return true;
}
inline bool same_shape(const b200_tensor & a, const b200_tensor & b) { return a.ne[0] == b.ne[0] && a.ne[1] == b.ne[1] && a.ne[2] == b.ne[2] && a.ne[3] == b.ne[3]; }
inline bool aligned16(const void * p) { return ((uintptr_t)p & 15) == 0; }
inline bool is_output(const b200_tensor & t) { return (t.flags & B200_TENSOR_FLAG_OUTPUT) != 0; }   // the caller reads it: never elide or fuse away
inline float f32_param(const b200_node & n, int i) { float f; memcpy(&f, &n.op_params[i], 4); return f; }

inline size_t tensor_bytes(const b200_tensor & t) {
    if (!t.data) return 0;
    if (is_weight_type(t.type)) return (size_t)(nrows_of(t) > 0 ? (t.ne[1] - 1) * t.nb[1] + (t.ne[2] - 1) * t.nb[2] + (t.ne[3] - 1) * t.nb[3] + type_block_bytes(t.type) * (t.ne[0] / type_block_elems(t.type)) : 0);
    if (is_wide_only_type(t.type)) return (size_t)(nrows_of(t) > 0 ? (t.ne[1] - 1) * t.nb[1] + (t.ne[2] - 1) * t.nb[2] + (t.ne[3] - 1) * t.nb[3] + b200_wide_row_bytes(t.type, t.ne[0]) : 0);
    size_t b = (size_t)elem_size(t.type);
    for (int i = 0; i < 4; i++) b += (size_t)(t.ne[i] - 1) * (size_t)t.nb[i];
    return b;
}
inline bool overlaps(const b200_tensor & a, const b200_tensor & b) {
    if (!a.data || !b.data) return false;
    const uintptr_t a0 = (uintptr_t)a.data, a1 = a0 + tensor_bytes(a), b0 = (uintptr_t)b.data, b1 = b0 + tensor_bytes(b);
    return a0 < b1 && b0 < a1;
}

// the tuned formats reach the wide kernels in the library's weight layout, which exists only where the load-time repack applies
// (the same rule as mul_mat_ok / the plug-in's repack_k_ok: whole 256-element units, Q6_K rows 16-byte aligned)
inline bool lib_layout_ok(int type, int64_t k) { return !is_weight_type(type) || (k % 256 == 0 && (type != B200_TYPE_Q6_K || k % 2048 == 0)); }
// MUL_MAT on a format only the wide matvec reads (ggml block layout, any k that is a block multiple)
bool mul_mat_wide_ok(const b200_node & n) {
    const b200_tensor & w = n.src[0], & x = n.src[1], & d = n.dst;
    if (!wide_on() || !is_wide_only_type(w.type) || x.type != B200_TYPE_F32 || d.type != B200_TYPE_F32) return false;
    const int64_t k = w.ne[0], m = w.ne[1];
    if (!b200_wide_shape_supported(w.type, k) || m <= 0 || w.ne[2] != 1 || w.ne[3] != 1 || x.ne[2] != 1 || x.ne[3] != 1) return false;
    if (w.nb[1] != b200_wide_row_bytes(w.type, k)) return false;
    if (x.ne[0] != k || x.nb[0] != 4 || (x.nb[1] & 15) || d.ne[0] != m || d.ne[1] != x.ne[1] || d.nb[0] != 4 || (d.nb[1] & 3)) return false;
    return aligned16(w.data) && aligned16(x.data);
}
// MUL_MAT_ID (ggml.c:3064-3106): as [k, m, n_expert], b f32 [k, n_b1, n_tok] (n_b1 = 1 or n_used), ids i32 [n_used, n_tok], dst f32 [m, n_used, n_tok]
bool mul_mat_id_ok(const b200_node & n) {
    if (!wide_on() || n.n_src < 3) return false;
    const b200_tensor & w = n.src[0], & x = n.src[1], & ids = n.src[2], & d = n.dst;
    if (!(is_weight_type(w.type) || is_wide_only_type(w.type)) || x.type != B200_TYPE_F32 || d.type != B200_TYPE_F32 || ids.type != B200_TYPE_I32) return false;
    const int64_t k = w.ne[0], m = w.ne[1], ne = w.ne[2], n_used = ids.ne[0], n_tok = ids.ne[1];
    if (!b200_wide_shape_supported(w.type, k) || m <= 0 || ne <= 0 || w.ne[3] != 1 || n_used <= 0 || n_tok <= 0 || ids.ne[2] != 1 || ids.ne[3] != 1) return false;
    if (!lib_layout_ok(w.type, k)) return false;
    if (w.nb[1] != b200_wide_row_bytes(w.type, k) || w.nb[2] < w.nb[1] * m || (w.nb[2] & 15)) return false;
    if (x.ne[0] != k || x.nb[0] != 4 || x.ne[1] <= 0 || n_used % x.ne[1] != 0 || x.ne[2] != n_tok || x.ne[3] != 1 || (x.nb[1] & 15) || (x.nb[2] & 15)) return false;
    if (d.ne[0] != m || d.ne[1] != n_used || d.ne[2] != n_tok || d.ne[3] != 1 || d.nb[0] != 4 || (d.nb[1] & 3) || (d.nb[2] & 3)) return false;
    if (ids.nb[0] != 4 || (ids.nb[1] & 3)) return false;
    return aligned16(w.data) && aligned16(x.data);
}
// GET_ROWS on a quantised table (token embeddings): src rows of a weight format, ids i32 [n], dst f32 [ncols, n] contiguous
bool get_rows_q_ok(const b200_node & n) {
    if (!wide_on() || n.n_src < 2) return false;
    const b200_tensor & s = n.src[0], & ids = n.src[1], & d = n.dst;
    if (!(is_weight_type(s.type) || is_wide_only_type(s.type)) || ids.type != B200_TYPE_I32 || d.type != B200_TYPE_F32) return false;
    if (!lib_layout_ok(s.type, s.ne[0])) return false;
    if (is_weight_type(s.type) && s.nb[1] != b200_wide_row_bytes(s.type, s.ne[0])) return false;     // the load-time repack works on whole, dense tensors
    if (!b200_wide_shape_supported(s.type, s.ne[0]) || s.ne[1] <= 0 || s.ne[2] != 1 || s.ne[3] != 1 || s.nb[1] < b200_wide_row_bytes(s.type, s.ne[0]) || (s.nb[1] & 1)) return false;
    if (ids.ne[1] != 1 || ids.ne[2] != 1 || ids.ne[3] != 1 || ids.nb[0] != 4 || d.ne[0] != s.ne[0] || d.ne[1] != ids.ne[0] || !contiguous(d)) return false;
    return aligned16(s.data) && aligned16(d.data);
}

// ---- mixture-of-experts router glue (wide path): small f32 ops of build_moe_ffn (llama-graph.cpp:820-1010)
inline bool f32_strided(const b200_tensor & t) { return t.type == B200_TYPE_F32 && t.data && !((uintptr_t)t.data & 3) && !((t.nb[0] | t.nb[1] | t.nb[2] | t.nb[3]) & 3) && t.ne[0] > 0 && t.ne[1] > 0 && t.ne[2] > 0 && t.ne[3] > 0; }
// ADD / MUL / DIV with ggml's broadcasting over any strides (the expert-weight MUL, the weight-normalising DIV, the ADDs over expert slices)
bool bin_strided_ok(const b200_node & n) {
    if (!wide_on() || n.n_src < 2) return false;
    const b200_tensor & a = n.src[0], & b = n.src[1], & d = n.dst;
    if (!f32_strided(a) || !f32_strided(b) || !f32_strided(d) || !same_shape(a, d)) return false;
    for (int i = 0; i < 4; i++) if (d.ne[i] % b.ne[i] != 0) return false;
    return true;
}
// the f32 router matrix (ffn_gate_inp [n_embd, n_expert]) times the activations
bool mul_mat_f32_ok(const b200_node & n) {
    const b200_tensor & w = n.src[0], & x = n.src[1], & d = n.dst;
    if (!wide_on() || w.type != B200_TYPE_F32 || x.type != B200_TYPE_F32 || d.type != B200_TYPE_F32) return false;
    if (w.ne[2] != 1 || w.ne[3] != 1 || x.ne[2] != 1 || x.ne[3] != 1 || w.ne[1] <= 0 || w.ne[1] > 1024 || w.ne[0] <= 0) return false;     // router-sized only
    if (w.nb[0] != 4 || (w.nb[1] & 3) || x.ne[0] != w.ne[0] || x.nb[0] != 4 || (x.nb[1] & 3) || d.ne[0] != w.ne[1] || d.ne[1] != x.ne[1] || d.nb[0] != 4 || (d.nb[1] & 3)) return false;
    return w.data && x.data && !(((uintptr_t)w.data | (uintptr_t)x.data | (uintptr_t)d.data) & 3);
}
bool rows2d_f32(const b200_tensor & t) { return t.type == B200_TYPE_F32 && t.nb[0] == 4 && contiguous(t) && !((uintptr_t)t.data & 3); }
bool soft_max_ok(const b200_node & n) {
    if (!wide_on() || n.n_src < 1 || (n.n_src > 2 && n.src[2].id)) return false;                                        // sinks: not on this path
    if (!rows2d_f32(n.src[0]) || !rows2d_f32(n.dst) || !same_shape(n.src[0], n.dst) || n.src[0].ne[0] > 65536) return false;
    if (n.n_src > 1 && n.src[1].id) {                        // with a mask: attention without -fa — x [n_kv, n_tok, n_head], one mask row per token
        const b200_tensor & m = n.src[1], & x = n.src[0];
        if ((m.type != B200_TYPE_F32 && m.type != B200_TYPE_F16) || m.nb[0] != (m.type == B200_TYPE_F16 ? 2 : 4) || m.ne[0] != x.ne[0] || m.ne[1] < x.ne[1] || m.ne[2] != 1 || m.ne[3] != 1) return false;
        if (x.ne[3] != 1 || (m.nb[1] % m.nb[0]) || !m.data || ((uintptr_t)m.data & (m.nb[0] - 1))) return false;
        return true;
    }
    return f32_param(n, 1) == 0.0f;
}
// batched MUL_MAT with an f16 src0 view (attention without -fa: KQ over the permuted K cache, KQV over the transposed V cache; GQA broadcast over dim 2)
bool mul_mat_f16_ok(const b200_node & n) {
    const b200_tensor & w = n.src[0], & x = n.src[1], & d = n.dst;
    if (!wide_on() || w.type != B200_TYPE_F16 || x.type != B200_TYPE_F32 || d.type != B200_TYPE_F32) return false;
    if (w.ne[3] != 1 || x.ne[3] != 1 || d.ne[3] != 1 || w.ne[0] <= 0 || w.ne[1] <= 0 || w.ne[2] <= 0 || x.ne[1] <= 0 || x.ne[2] <= 0 || x.ne[2] % w.ne[2] != 0) return false;
    if (w.nb[0] != 2 || ((w.nb[1] | w.nb[2]) & 1) || x.ne[0] != w.ne[0] || x.nb[0] != 4 || ((x.nb[1] | x.nb[2]) & 3)) return false;
    if (d.ne[0] != w.ne[1] || d.ne[1] != x.ne[1] || d.ne[2] != x.ne[2] || d.nb[0] != 4 || ((d.nb[1] | d.nb[2]) & 3)) return false;
    if (d.ne[0] * d.ne[1] * d.ne[2] > ((int64_t)1 << 31)) return false;
    return w.data && x.data && d.data && !((uintptr_t)w.data & 1) && !(((uintptr_t)x.data | (uintptr_t)d.data) & 3);
}
// SET_ROWS whose rows are single elements (the transposed V cache): src [1, n] f32, ids i64 [n], dst [1, N] f16 / f32
bool set_rows1_ok(const b200_node & n) {
    if (!wide_on() || n.n_src < 2) return false;
    const b200_tensor & s = n.src[0], & ids = n.src[1], & d = n.dst;
    if (s.type != B200_TYPE_F32 || ids.type != B200_TYPE_I64 || (d.type != B200_TYPE_F16 && d.type != B200_TYPE_F32)) return false;
    if (s.ne[0] != 1 || d.ne[0] != 1 || s.ne[2] != 1 || s.ne[3] != 1 || d.ne[2] != 1 || d.ne[3] != 1 || ids.ne[0] != s.ne[1] || ids.ne[1] != 1 || ids.ne[2] != 1) return false;
    if (s.nb[1] != 4 || ids.nb[0] != 8 || d.nb[1] != (d.type == B200_TYPE_F16 ? 2 : 4)) return false;
    return s.data && ids.data && d.data && !((uintptr_t)s.data & 3) && !((uintptr_t)ids.data & 7) && !((uintptr_t)d.data & (d.nb[1] - 1));
}
bool cont_ok(const b200_node & n) {
    if (!wide_on() || n.n_src < 1) return false;
    return f32_strided(n.src[0]) && n.dst.type == B200_TYPE_F32 && contiguous(n.dst) && n.dst.data && !((uintptr_t)n.dst.data & 3) && nelem(n.src[0]) == nelem(n.dst);
}
bool argsort_ok(const b200_node & n) {
    if (!wide_on() || n.n_src < 1) return false;
    const b200_tensor & s = n.src[0], & d = n.dst;
    return rows2d_f32(s) && d.type == B200_TYPE_I32 && contiguous(d) && same_shape(s, d) && s.ne[0] <= 4096 && (n.op_params[0] == 0 || n.op_params[0] == 1) && !((uintptr_t)d.data & 3);
}
bool sum_rows_ok(const b200_node & n) {
    if (!wide_on() || n.n_src < 1) return false;
    const b200_tensor & s = n.src[0], & d = n.dst;
    return rows2d_f32(s) && rows2d_f32(d) && d.ne[0] == 1 && d.ne[1] == s.ne[1] && d.ne[2] == s.ne[2] && d.ne[3] == s.ne[3];
}
// GET_ROWS f32, one id list, 16-byte rows (the output-row gather of the last layer)
bool get_rows_f32_ok(const b200_node & n) {
    const b200_tensor & s = n.src[0], & ids = n.src[1], & d = n.dst;
    return n.n_src >= 2 && s.type == B200_TYPE_F32 && ids.type == B200_TYPE_I32 && s.nb[0] == 4 && (s.nb[1] & 15) == 0 && s.ne[2] == 1 && s.ne[3] == 1 &&
           s.ne[0] % 4 == 0 && aligned16(s.data) && d.type == B200_TYPE_F32 && contiguous(d) && aligned16(d.data) && ids.ne[1] == 1 && ids.ne[2] == 1 && d.ne[1] == ids.ne[0];
}
// GET_ROWS f32 with one id list per batch (ggml.c:3620-3650): src [c, r, b], ids [n, b], dst [c, n, b]
bool get_rows_f32_batched_ok(const b200_node & n) {
    if (!wide_on() || n.n_src < 2) return false;
    const b200_tensor & s = n.src[0], & ids = n.src[1], & d = n.dst;
    if (s.type != B200_TYPE_F32 || ids.type != B200_TYPE_I32 || d.type != B200_TYPE_F32 || !f32_strided(s) || s.nb[0] != 4 || s.ne[3] != 1 || ids.ne[2] != 1 || ids.ne[3] != 1) return false;
    if (ids.nb[0] != 4 || (ids.nb[1] & 3) || ids.ne[1] != s.ne[2] || !contiguous(d) || d.ne[0] != s.ne[0] || d.ne[1] != ids.ne[0] || d.ne[2] != s.ne[2] || d.ne[3] != 1) return false;
    return ids.data && !(((uintptr_t)ids.data | (uintptr_t)d.data) & 3);
}

bool mul_mat_ok(const b200_node & n) {
    const b200_tensor & w = n.src[0], & x = n.src[1], & d = n.dst;
    if (is_wide_only_type(w.type)) return mul_mat_wide_ok(n);
    if (w.type == B200_TYPE_F32) return mul_mat_f32_ok(n);
    if (w.type == B200_TYPE_F16) return mul_mat_f16_ok(n);
    if (!is_weight_type(w.type) || x.type != B200_TYPE_F32 || d.type != B200_TYPE_F32) return false;
    const int64_t k = w.ne[0], m = w.ne[1];
    // 32-element block types: any multiple of 32 (rows padded to 256 in the private weight layout, see common.cuh padded_k)
    if (k <= 0 || (type_is_block32(w.type) ? k % 32 != 0 : k % 256 != 0) || (w.type == B200_TYPE_Q6_K && k % 2048 != 0)) return false;
    if (w.ne[2] != 1 || w.ne[3] != 1 || x.ne[2] != 1 || x.ne[3] != 1) return false;            // no broadcast batches on this path
    if (w.nb[1] != type_block_bytes(w.type) * (k / type_block_elems(w.type))) return false;
    if (x.ne[0] != k || x.nb[0] != 4 || (x.nb[1] & 15) || d.ne[0] != m || d.ne[1] != x.ne[1] || d.nb[0] != 4 || (d.nb[1] & 3)) return false;
    return aligned16(w.data) && aligned16(x.data);
}
bool rows_f32_ok(const b200_tensor & t) { return t.type == B200_TYPE_F32 && contiguous(t) && t.ne[0] % 4 == 0 && aligned16(t.data); }
bool bin_ok(const b200_node & n) {
    const b200_tensor & a = n.src[0], & b = n.src[1], & d = n.dst;
    if (!rows_f32_ok(a) || !rows_f32_ok(d) || !same_shape(a, d) || b.type != B200_TYPE_F32 || !contiguous(b) || !aligned16(b.data)) return false;
    if (same_shape(a, b)) return true;
    return b.ne[0] == a.ne[0] && b.ne[2] == 1 && b.ne[3] == 1 && b.ne[1] > 0 && a.ne[1] % b.ne[1] == 0;
}
bool rope_ok(const b200_node & n) {
    const b200_tensor & x = n.src[0], & p = n.src[1], & d = n.dst;
    if (x.type != B200_TYPE_F32 || d.type != B200_TYPE_F32 || p.type != B200_TYPE_I32 || x.nb[0] != 4 || d.nb[0] != 4) return false;
    if (x.ne[3] != 1 || !same_shape(x, d) || (x.ne[0] & 1) || p.ne[0] < x.ne[2]) return false;
    const int mode = n.op_params[2], n_dims = n.op_params[1];
    if ((mode & ~2) || n_dims <= 0 || n_dims > x.ne[0] || (n_dims & 1)) return false;
    if ((x.nb[1] | x.nb[2] | d.nb[1] | d.nb[2]) & 3) return false;
    if (n.n_src > 2 && n.src[2].data && (n.src[2].type != B200_TYPE_F32 || n.src[2].ne[0] < n_dims / 2)) return false;
    return true;
}
bool set_rows_ok(const b200_node & n) {
    const b200_tensor & s = n.src[0], & ids = n.src[1], & d = n.dst;
    if (s.type != B200_TYPE_F32 || ids.type != B200_TYPE_I64 || s.nb[0] != 4 || (s.nb[1] & 15) || !aligned16(s.data)) return false;
    const bool q4 = d.type == B200_TYPE_Q4_0 && wide_on();          // KV cache type q4_0: wide path (fattn_ext.cu)
    if (d.type != B200_TYPE_F32 && d.type != B200_TYPE_F16 && d.type != B200_TYPE_Q8_0 && !q4) return false;
    if (q4 && (s.ne[1] > 65535 || (((uintptr_t)d.data | (uintptr_t)d.nb[1] | (uintptr_t)d.nb[2] | (uintptr_t)d.nb[3]) & 1))) return false;
    // batches (ggml.c:3661-3686): dst [ne0, rows, ne2, ne3], src [ne0, n, ne2, ne3], ids [n, ne11, ne12] broadcast over dims 2/3
    if (s.ne[2] != d.ne[2] || s.ne[3] != d.ne[3] || s.ne[0] != d.ne[0] || s.ne[0] % 32 != 0 || ids.ne[0] != s.ne[1] || ids.ne[3] != 1) return false;
    if (ids.ne[1] <= 0 || ids.ne[2] <= 0 || s.ne[2] % ids.ne[1] != 0 || s.ne[3] % ids.ne[2] != 0) return false;
    if ((s.nb[2] | s.nb[3]) & 15) return false;
    if (d.type != B200_TYPE_Q8_0 && !q4 && (((uintptr_t)d.data | (uintptr_t)d.nb[1] | (uintptr_t)d.nb[2] | (uintptr_t)d.nb[3]) & 15)) return false;
    return true;
}
bool fattn_ok(const b200_node & n) {
    const b200_tensor & q = n.src[0], & k = n.src[1], & v = n.src[2], & d = n.dst;
    if (n.n_src > 4 && n.src[4].data) return false;                                  // attention sinks: not on this path
    if (q.type != B200_TYPE_F32 || d.type != B200_TYPE_F32 || k.type != v.type) return false;
    if (k.type != B200_TYPE_F16 && k.type != B200_TYPE_Q8_0 && !(k.type == B200_TYPE_Q4_0 && wide_on())) return false;
    if (k.type == B200_TYPE_Q4_0 && ((((uintptr_t)k.data | (uintptr_t)v.data) & 1) || ((k.nb[1] | k.nb[2] | v.nb[1] | v.nb[2]) & 1))) return false;
    const int64_t dk = q.ne[0], dv = v.ne[0];
    const bool any_d = wide_on() && dk % 32 == 0 && dk > 0 && dk <= 256;                 // head sizes beyond 64 / 128: the wide attention kernel (fattn_ext.cu)
    if (dk != dv || ((dk != 64 && dk != 128) && !any_d) || k.ne[0] != dk) return false;
    if (q.ne[3] != 1 || k.ne[3] != 1 || v.ne[3] != 1 || k.ne[1] != v.ne[1] || k.ne[2] != v.ne[2] || k.ne[2] <= 0 || q.ne[2] % k.ne[2] != 0) return false;
    if (q.nb[0] != 4 || (q.nb[1] & 15) || (q.nb[2] & 15) || !aligned16(q.data)) return false;
    if (k.type == B200_TYPE_F16 && (dk == 64 || dk == 128) && ((((uintptr_t)k.data | (uintptr_t)v.data) & 15) || ((k.nb[1] | k.nb[2] | v.nb[1] | v.nb[2]) & 15))) return false;
    if (dk != 64 && dk != 128 && ((((uintptr_t)k.data | (uintptr_t)v.data) & 1) || ((k.nb[1] | k.nb[2] | v.nb[1] | v.nb[2]) & 1))) return false;
    if (!contiguous(d) || d.ne[0] != dv || d.ne[1] != q.ne[2] || d.ne[2] != q.ne[1] || q.ne[1] > 65535) return false;
    if (n.n_src > 3 && n.src[3].data) {
        const b200_tensor & m = n.src[3];
        if (m.type != B200_TYPE_F16 || m.nb[0] != 2 || m.ne[0] != k.ne[1] || m.ne[1] < q.ne[1] || m.ne[2] != 1 || m.ne[3] != 1) return false;
    }
    return true;
}

bool node_ok(const b200_node & n) {
    if (n.op > B200_OP_NONE && n.op < B200_OP_COUNT && nelem(n.dst) == 0) return true;   // empty result (a ubatch without outputs): nothing to run, like ggml_is_empty nodes in ggml-cuda.cu:2858
    switch (n.op) {
        case B200_OP_NONE:     return true;
        case B200_OP_MUL_MAT:  return n.n_src >= 2 && mul_mat_ok(n);
        case B200_OP_RMS_NORM: return n.n_src >= 1 && rows_f32_ok(n.src[0]) && rows_f32_ok(n.dst) && same_shape(n.src[0], n.dst) && n.src[0].ne[0] * 4 <= 200 * 1024;
        case B200_OP_MUL: case B200_OP_ADD: return n.n_src >= 2 && (bin_ok(n) || bin_strided_ok(n));
        case B200_OP_DIV:      return bin_strided_ok(n);
        case B200_OP_SOFT_MAX: return soft_max_ok(n);
        case B200_OP_ARGSORT:  return argsort_ok(n);
        case B200_OP_SUM_ROWS: return sum_rows_ok(n);
        case B200_OP_ROPE:     return n.n_src >= 2 && rope_ok(n);
        case B200_OP_SET_ROWS: return n.n_src >= 2 && (set_rows_ok(n) || set_rows1_ok(n));
        case B200_OP_CONT:     return cont_ok(n);
        case B200_OP_SCALE:    return wide_on() && n.n_src >= 1 && rows2d_f32(n.src[0]) && rows2d_f32(n.dst) && same_shape(n.src[0], n.dst);
        case B200_OP_UNARY:    return wide_on() && n.n_src >= 1 && rows2d_f32(n.src[0]) && rows2d_f32(n.dst) && same_shape(n.src[0], n.dst) && (n.op_params[0] == 10 || n.op_params[0] == 7);
        case B200_OP_FLASH_ATTN_EXT: return n.n_src >= 3 && fattn_ok(n);
        case B200_OP_GLU_SWIGLU: return n.n_src >= 2 && rows_f32_ok(n.src[0]) && rows_f32_ok(n.src[1]) && rows_f32_ok(n.dst) && same_shape(n.src[0], n.src[1]) && same_shape(n.src[0], n.dst);
        case B200_OP_MUL_MAT_ID: return mul_mat_id_ok(n);
        case B200_OP_GET_ROWS: {
            const b200_tensor & s = n.src[0], & ids = n.src[1], & d = n.dst;
            if (n.n_src >= 2 && s.type != B200_TYPE_F32) return get_rows_q_ok(n);
            return n.n_src >= 2 && (get_rows_f32_ok(n) || get_rows_f32_batched_ok(n));
        }
        case B200_OP_CPY: {
            const b200_tensor & s = n.src[0], & d = n.dst;
            return n.n_src >= 1 && s.type == B200_TYPE_F32 && contiguous(s) && contiguous(d) && nelem(s) == nelem(d) && (d.type == B200_TYPE_F16 || d.type == B200_TYPE_F32) && aligned16(s.data) && ((uintptr_t)d.data & 7) == 0;
        }
        default: return false;
    }
}

struct GraphEntry { cudaGraphExec_t exec = nullptr; int64_t kernels = 0; uint64_t last_use = 0; };

} // namespace

struct b200_executor {
    int device = 0;
    // workspace: [act q8_K][act q8_0][fattn partials]
    uint8_t * ws = nullptr; size_t ws_bytes = 0;
    size_t off_act[2] = {0, 0}, act_bytes[2] = {0, 0}, off_fa = 0, fa_bytes = 0;
    uint64_t act_id[2] = {0, 0}; const void * act_ptr[2] = {nullptr, nullptr}; int64_t act_cols[2] = {0, 0};
    // a RMS_NORM(+MUL) whose only consumers are decode matvecs is not launched: the matvec prologue computes it
    struct { uint64_t out_id = 0; const void * out_data = nullptr; b200_tensor x, out; const float * w = nullptr; float eps = 0; } norm;
    std::unordered_map<uint64_t, GraphEntry> graphs;
    std::unordered_map<uint64_t, int> seen;      // topology -> times seen before capture (first sighting runs eagerly)
    uint64_t tick = 0;
    int64_t last_kernels = 0, captures = 0, replays = 0;
    bool env_no_graphs = false, env_no_fusion = false, env_no_mega = false, env_mega = false, env_mega_mmv = false;
    // persistent decode kernel (decode_mk.cu): compiled phase programs, resident on the device, keyed by content
    struct DevProg { MkPhase * dev = nullptr; MkPhase * host = nullptr; int n = 0; };
    std::unordered_map<uint64_t, DevProg> progs;
    unsigned long long * mk_sync = nullptr;       // grid-barrier counters (zeroed once; the kernel cleans up after itself)
    int64_t mk_launches = 0, mk_phases = 0;
};

namespace {

// a kernel launch — or, in a dry run, just its count
#define KL(call) (dry ? (plan_note(#call), (int)B200_OK) : (int)(call))

struct Runner {
    b200_executor * ex; const b200_node * nodes; int n; cudaStream_t st; bool fuse;
    std::vector<uint8_t> done;
    std::unordered_map<uint64_t, int> uses;
    // ---- persistent decode kernel: phases recorded instead of launched, flushed as ONE launch ----------------
    bool mega = false, mega_mmv = false;
    bool dry = false; int64_t planned = 0;      // dry run (b200_executor_plan): walk the list, count launches, touch no device
    void plan_note(const char * what) { planned++; static const bool dbg = getenv("B200_PLAN_DEBUG") != nullptr; if (dbg) fprintf(stderr, "plan %3lld: %.40s\n", (long long)planned, what); }
    std::vector<MkPhase> pend;
    struct RopePend { bool valid = false; const float * q_src; float * q_dst; const float * k, * v; const int32_t * pos; const float * ff;
                      const int64_t * k_ids, * v_ids; void * k_cache, * v_cache; int kv_type; int64_t k_rs, v_rs, hd, nh, nhk; b200_rope_params p; } rope_pend;

    int mk_flush() {
        int s = B200_OK;
        if (dry && !pend.empty()) { plan_note("mk_launch(persistent kernel program)"); pend.clear(); }
        if (!pend.empty()) {
            // content hash -> device-resident program (uploaded once; replayed graphs keep pointing at it)
            uint64_t h = 0xcbf29ce484222325ull;
            const uint64_t * w = (const uint64_t *)pend.data();
            for (size_t i = 0; i < pend.size() * sizeof(MkPhase) / 8; i++) { h ^= w[i]; h *= 0x100000001b3ull; h ^= h >> 29; }
            auto it = ex->progs.find(h);
            if (it == ex->progs.end()) {
                b200_executor::DevProg dp; dp.n = (int)pend.size();
                const size_t bytes = pend.size() * sizeof(MkPhase);
                B200_CUDA(cudaMallocHost((void **)&dp.host, bytes));
                B200_CUDA(cudaMalloc((void **)&dp.dev, bytes));
                memcpy(dp.host, pend.data(), bytes);
                B200_CUDA(cudaMemcpyAsync(dp.dev, dp.host, bytes, cudaMemcpyHostToDevice, st));
                it = ex->progs.emplace(h, dp).first;
            }
            if (!ex->mk_sync) { B200_CUDA(cudaMalloc((void **)&ex->mk_sync, 16)); B200_CUDA(cudaMemsetAsync(ex->mk_sync, 0, 16, st)); }
            s = mk_launch(it->second.dev, it->second.n, ex->mk_sync, st);
            ex->mk_launches++; ex->mk_phases += (int64_t)pend.size();
            pend.clear();
            if (s != B200_OK) return s;
        }
        if (rope_pend.valid) {
            const RopePend & r = rope_pend;
            rope_pend.valid = false;
            s = KL(b200_rope_kv_store2(r.q_src, r.q_dst, r.k, r.v, r.pos, r.ff, r.k_ids, r.v_ids, r.k_cache, r.v_cache, r.kv_type, r.k_rs, r.v_rs, r.hd, r.nh, r.nhk, 1, &r.p, st));
        }
        return s;
    }
    int mk_flush_rope_only() { return rope_pend.valid ? mk_flush() : B200_OK; }
    // a decode matvec launch as a phase of the persistent kernel (Q4_K / Q6_K, one column, in-kernel activation)
    bool mk_try_mmv(const b200_mmv_launch & L) {
        // (round 1 sent the lone 525 MB output matrix here: 5.2 vs 4.1 TB/s.  With the lean matvec instances the per-op kernel is the
        //  faster one — 534 vs 521 tok/s — so this is opt-in now: GGML_B200_LMHEAD_MEGAKERNEL=1)
        static const bool big_on = getenv("GGML_B200_LMHEAD_MEGAKERNEL") != nullptr;
        const bool big = big_on && L.n_mats == 1 && !L.swiglu && (int64_t)L.mats[0].m * L.k >= ((int64_t)192 << 20) && !ex->env_no_mega && fuse;
        if (!((mega && mega_mmv) || big) || L.ncols != 1 || (L.act_source != 1 && L.act_source != 2) || L.y_out || !mk_phase_ok_k(L.k, L.act_source) || L.n_mats < 1 || L.n_mats > MK_MAX_MATS) return false;
        for (int q = 0; q < L.n_mats; q++) {
            const b200_mmv_desc & d = L.mats[q];
            if ((d.type != B200_TYPE_Q4_K && d.type != B200_TYPE_Q6_K) || d.m <= 0 || (d.m & 1) || d.m > 0x7fffffff || !d.W || !d.dst) return false;
            if (((uintptr_t)d.dst & 7) || (L.residual[q] && ((uintptr_t)L.residual[q] & 3))) return false;
        }
        if (L.swiglu && (L.n_mats != 2 || L.mats[0].type != L.mats[1].type || L.mats[0].m != L.mats[1].m)) return false;
        if (rope_pend.valid && mk_flush() != B200_OK) return false;
        MkPhase ph; memset(&ph, 0, sizeof(ph));
        ph.kind = MK_MMV;
        ph.mmv.n_mats = L.n_mats; ph.mmv.swiglu = L.swiglu; ph.mmv.act_source = L.act_source; ph.mmv.k = (int32_t)L.k; ph.mmv.eps = L.eps;
        ph.mmv.x = L.x; ph.mmv.norm_w = L.act_source == 2 ? L.norm_w : nullptr;
        for (int q = 0; q < L.n_mats; q++) {
            const b200_mmv_desc & d = L.mats[q];
            MkMat & m = ph.mmv.mat[q];
            m.W = (const uint8_t *)d.W; m.dst = d.dst; m.bias = d.bias; m.residual = L.residual[q];
            m.rb = type_block_bytes(d.type) * (L.k / 256); m.m = (int32_t)d.m; m.type = d.type;
        }
        pend.push_back(ph);
        return true;
    }
    int launch_mmv(const b200_mmv_launch & L) {
        if (mk_try_mmv(L)) return B200_OK;
        const int s = mk_flush();
        if (s != B200_OK) return s;
        return KL(b200_mul_mat_vec_q_launch(&L, st));
    }
    // does this FLASH_ATTN_EXT consume exactly what the recorded rope + KV store of the same token produces?
    bool attn_matches(const b200_node & n) const {
        if (!rope_pend.valid) return false;
        const RopePend & r = rope_pend;
        const b200_tensor & q = n.src[0], & k = n.src[1], & v = n.src[2];
        if (q.data != r.q_dst || q.ne[1] != 1 || q.ne[0] != r.hd || q.ne[2] != r.nh || q.nb[2] != r.hd * 4) return false;
        if (k.data != r.k_cache || v.data != r.v_cache || k.type != r.kv_type || k.nb[1] != r.k_rs || v.nb[1] != r.v_rs || k.ne[2] != r.nhk) return false;
        if (r.hd != 64 && r.hd != 128) return false;
        const int64_t hs = r.kv_type == B200_TYPE_F16 ? r.hd * 2 : r.hd / 32 * 34;      // heads contiguous inside a cell, as SET_ROWS wrote them
        if (k.nb[2] != hs || v.nb[2] != hs || n.dst.type != B200_TYPE_F32 || !contiguous(n.dst)) return false;
        return true;
    }
    // ... as one launch of the split-KV attention kernel (fattn.cu, FaFuse)
    // the cos/sin table of a decode token depends on its position only: the first attention launch of a list computes it into
    // executor scratch, the other layers (same positions tensor, same rope parameters) load it
    struct { bool valid = false; const int32_t * pos = nullptr; const float * ff = nullptr; b200_rope_params p; int64_t hd = 0; } tab;
    int launch_fused_attn(const b200_node & n) {
        const RopePend r = rope_pend;
        rope_pend.valid = false;
        const int fs = mk_flush(); if (fs != B200_OK) return fs;
        const b200_tensor & k = n.src[1], & v = n.src[2];
        const void * mask = n.n_src > 3 ? n.src[3].data : nullptr;
        float * rope_tab = nullptr; int tab_mode = 0;
        if (dry || (ex->ws && ex->fa_bytes >= 1024)) {
            rope_tab = dry ? (float *)(uintptr_t)0x20000 : (float *)(ex->ws + ex->off_fa + ex->fa_bytes - 1024);
            tab_mode = tab.valid && tab.pos == r.pos && tab.ff == r.ff && tab.hd == r.hd && memcmp(&tab.p, &r.p, sizeof(r.p)) == 0;
            tab.valid = true; tab.pos = r.pos; tab.ff = r.ff; tab.p = r.p; tab.hd = r.hd;
        }
        return KL(b200_rope_kv_flash_attn2(r.q_src, r.q_dst, r.k, r.v, r.pos, r.ff, r.k_ids, r.v_ids, r.k_cache, r.v_cache, r.kv_type, k.nb[1], k.nb[2], v.nb[1], v.nb[2],
                                        mask, (float *)n.dst.data, r.hd, r.nh, r.nhk, k.ne[1], &r.p, f32_param(n, 0), f32_param(n, 1), f32_param(n, 2), ex->ws + ex->off_fa,
                                        rope_tab, tab_mode, st));
    }
    // ... or as a phase of the persistent kernel
    bool mk_try_attn(const b200_node & n) {
        if (!mega || !attn_matches(n)) return false;
        const RopePend & r = rope_pend;
        const b200_tensor & k = n.src[1], & v = n.src[2];
        const void * mask = n.n_src > 3 ? n.src[3].data : nullptr;
        const int64_t n_kv = k.ne[1];
        const int64_t gq = r.nh / r.nhk;
        const int G = gq % 4 == 0 ? 4 : (gq % 2 == 0 ? 2 : 1);
        const int64_t n_tiles = r.nh / G;
        int64_t want = b200_sm_count() / n_tiles; if (want < 1) want = 1;
        int64_t maxs = (n_kv + 31) / 32; if (maxs > 64) maxs = 64;
        if (want > maxs) want = maxs;
        int64_t len = (n_kv + want - 1) / want; len = (len + 3) / 4 * 4;
        const int64_t n_splits = (n_kv + len - 1) / len;
        if (n_tiles * (int64_t)sizeof(unsigned int) > 256 * 1024) return false;
        MkPhase ph; memset(&ph, 0, sizeof(ph));
        ph.kind = MK_ATTN;
        MkAttn & A = ph.attn;
        A.q_src = r.q_src; A.q_dst = r.q_dst; A.k = r.k; A.v = r.v; A.pos = r.pos; A.ff = r.ff; A.k_ids = r.k_ids; A.v_ids = r.v_ids;
        A.k_cache = (uint8_t *)r.k_cache; A.v_cache = (uint8_t *)r.v_cache; A.mask = (const uint16_t *)mask; A.dst = (float *)n.dst.data;
        A.counters = (unsigned int *)(ex->ws + ex->off_fa); A.ws = (float *)(ex->ws + ex->off_fa + 256 * 1024);
        A.k_rs = k.nb[1]; A.k_hs = k.nb[2]; A.v_rs = v.nb[1]; A.v_hs = v.nb[2];
        A.kv_type = r.kv_type; A.hd = (int32_t)r.hd; A.n_head = (int32_t)r.nh; A.n_head_kv = (int32_t)r.nhk; A.n_kv = (int32_t)n_kv;
        A.split_len = (int32_t)len; A.n_splits = (int32_t)n_splits;
        float scale = f32_param(n, 0); const float max_bias = f32_param(n, 1), softcap = f32_param(n, 2);
        A.nh_log2 = 1 << (int)floor(log2((double)r.nh));
        A.m0 = powf(2.0f, -(max_bias) / (float)A.nh_log2); A.m1 = powf(2.0f, -(max_bias / 2.0f) / (float)A.nh_log2);
        if (softcap != 0.0f) scale /= softcap;
        A.scale = scale; A.max_bias = max_bias; A.softcap = softcap;
        A.rp = rope_host_params(&r.p);
        rope_pend.valid = false;
        pend.push_back(ph);
        return true;
    }

    int use_count(const b200_tensor & t) const { auto it = uses.find(t.id); return it == uses.end() ? 0 : it->second; }
    int next_compute(int i) const { for (int j = i + 1; j < n; j++) if (!done[j] && nodes[j].op != B200_OP_NONE) return j; return -1; }

    void invalidate_act(const b200_tensor & written) {
        for (int kd = 0; kd < 2; kd++) if (ex->act_id[kd] && ex->act_ptr[kd] == written.data) ex->act_id[kd] = 0;
        if (ex->norm.out_id && (overlaps(written, ex->norm.x) || overlaps(written, ex->norm.out))) ex->norm.out_id = 0;
    }
    // how a decode matvec obtains its activation: from a pending norm (2), or by quantising the f32 tensor itself (1)
    void fill_act_source(b200_mmv_launch & L, const b200_tensor & x) const {
        if (ex->norm.out_id && ex->norm.out_id == x.id && ex->norm.out_data == x.data) {
            L.act_source = 2; L.x = (const float *)ex->norm.x.data; L.x_col_stride = ex->norm.x.nb[1] / 4; L.norm_w = ex->norm.w; L.eps = ex->norm.eps;
        } else {
            L.act_source = 1; L.x = (const float *)x.data; L.x_col_stride = x.nb[1] / 4; L.norm_w = nullptr; L.eps = 0.0f;
        }
        L.act_q8K = nullptr; L.act_q80 = nullptr; L.y_out = nullptr;
    }
    uint8_t * act_buf(int kind) const { return ex->ws + ex->off_act[kind]; }

    // make sure the act buffer of `kind` holds the quantised form of x (n cols of k)
    int ensure_act(const b200_tensor & x, int kind, int64_t k_pad) {
        if (ex->act_id[kind] == x.id && x.id != 0 && ex->act_ptr[kind] == x.data && ex->act_cols[kind] == x.ne[1] && k_pad == x.ne[0]) return B200_OK;
        int s = KL(b200_quantize_act2(kind, (const float *)x.data, x.nb[1] / 4, act_buf(kind), k_pad, x.ne[0], x.ne[1], st));
        if (s != B200_OK) return s;
        ex->act_id[kind] = x.id; ex->act_ptr[kind] = x.data; ex->act_cols[kind] = x.ne[1];
        return B200_OK;
    }

    int run_rms_norm(int i) {
        const b200_node & n = nodes[i];
        const float eps = f32_param(n, 0);
        const b200_tensor & x = n.src[0];
        const int64_t ncols = x.ne[0], nrows = nrows_of(x);
        // RMS_NORM -> MUL(weight row): llama-graph.cpp:605-619 (build_norm)
        const int j = fuse ? next_compute(i) : -1;
        if (j >= 0 && nodes[j].op == B200_OP_MUL && use_count(n.dst) == 1) {
            const b200_node & mu = nodes[j];
            const b200_tensor * w = nullptr;
            if (mu.src[0].id == n.dst.id && mu.src[0].data == n.dst.data) w = &mu.src[1];
            else if (mu.src[1].id == n.dst.id && mu.src[1].data == n.dst.data) w = &mu.src[0];
            if (w && w->ne[0] == ncols && nrows_of(*w) == 1 && same_shape(mu.dst, x)) {
                done[j] = 1;
                // all consumers are decode-shaped quantised MUL_MATs of this tensor: no kernel at all, the matvec
                // prologue normalises and quantises (b200_mul_mat_vec_q_launch act_source = 2)
                if (nrows <= 8 && ncols % 256 == 0 && mu.dst.nb[1] == ncols * 4 && x.nb[1] == ncols * 4 && !is_output(n.dst) && !is_output(mu.dst)) {
                    int consumers = 0, mm = 0;
                    for (int q = j + 1; q < this->n; q++) for (int sidx = 0; sidx < nodes[q].n_src && sidx < B200_MAX_SRC; sidx++)
                        if (nodes[q].src[sidx].id == mu.dst.id) { consumers++; if (nodes[q].op == B200_OP_MUL_MAT && sidx == 1 && !done[q] && nodes[q].src[1].ne[1] <= 8 && is_weight_type(nodes[q].src[0].type)) mm++; }
                    if (consumers > 0 && consumers == mm) {
                        ex->norm.out_id = mu.dst.id; ex->norm.out_data = mu.dst.data; ex->norm.x = x; ex->norm.out = mu.dst;
                        ex->norm.w = (const float *)w->data; ex->norm.eps = eps;
                        // a normalised tensor that no later node overwrites is still there when the graph ends, and the caller may
                        // read it (libllama fetches result_norm as the embeddings output without flagging it: llama-context.cpp:1115-1151):
                        // materialise it as well — the matvec prologue still recomputes it, so the weight stream is not delayed
                        // (only the LAST norm of a list can be that tensor: it feeds the output matrix)
                        bool survives = true;
                        for (int q = j + 1; q < this->n && survives; q++)
                            if (nodes[q].op == B200_OP_RMS_NORM || (nodes[q].op != B200_OP_NONE && overlaps(nodes[q].dst, mu.dst))) survives = false;
                        if (survives) {
                            { const int fs = mk_flush(); if (fs != B200_OK) return fs; }
                            // ggml-alloc may have placed the normalised tensor IN PLACE over x: then it cannot be both written now and
                            // recomputed from x later — the consumers quantise the materialised tensor instead (act_source 1)
                            if (overlaps(mu.dst, x)) ex->norm.out_id = 0;
                            return KL(b200_rms_norm((const float *)x.data, (const float *)w->data, (float *)mu.dst.data, ncols, nrows, ncols, ncols, eps, st));
                        }
                        return B200_OK;
                    }
                }
                // if the next consumer is a decode-shaped quantised MUL_MAT, emit its activation format too
                const int c = next_compute(j);
                if (c >= 0 && nodes[c].op == B200_OP_MUL_MAT && is_weight_type(nodes[c].src[0].type) && nodes[c].src[1].id == mu.dst.id && nodes[c].src[1].data == mu.dst.data &&
                    nrows <= 8 && ncols % 256 == 0 && mu.dst.nb[1] == ncols * 4) {
                    const int kind = b200_act_kind_for(nodes[c].src[0].type);
                    { const int fs = mk_flush(); if (fs != B200_OK) return fs; }
                    int s = KL(b200_rms_norm_quantize((const float *)x.data, (const float *)w->data, (float *)mu.dst.data, act_buf(kind), kind, nullptr, 0, ncols, nrows, eps, st));
                    if (s != B200_OK) return s;
                    invalidate_act(mu.dst);
                    ex->act_id[kind] = mu.dst.id; ex->act_ptr[kind] = mu.dst.data; ex->act_cols[kind] = nrows;
                    return B200_OK;
                }
                invalidate_act(mu.dst);
                { const int fs = mk_flush(); if (fs != B200_OK) return fs; }
                return KL(b200_rms_norm((const float *)x.data, (const float *)w->data, (float *)mu.dst.data, ncols, nrows, ncols, ncols, eps, st));
            }
        }
        invalidate_act(n.dst);
        { const int fs = mk_flush(); if (fs != B200_OK) return fs; }
        return KL(b200_rms_norm((const float *)x.data, nullptr, (float *)n.dst.data, ncols, nrows, ncols, ncols, eps, st));
    }

    // may node j (a later MUL_MAT of the same activation) be executed now, at position i?
    bool can_hoist(int i, int j) const {
        const b200_tensor & d = nodes[j].dst;
        for (int q = i; q < j; q++) {
            if (done[q]) continue;
            const b200_node & m = nodes[q];
            if (m.op == B200_OP_NONE) continue;
            if (overlaps(d, m.dst)) return false;
            for (int s = 0; s < m.n_src && s < B200_MAX_SRC; s++) if (overlaps(d, m.src[s])) return false;
        }
        return true;
    }

    // ---- the whole attention block of a decode token as TWO launches, even when the graph allocator recycles buffers -------
    // libllama's graph reuses the buffer of the un-roped Q for K and V (llama-graph allocations), which forbids hoisting the
    // K / V projections next to Q's — and with that every later fusion.  All intermediates of the block (Q/K/V before rope,
    // roped K) have exactly one consumer inside the block, so they are never materialised in the graph's buffers at all: the
    // three projections go to executor scratch in one launch, the fused rope + KV-store + attention launch reads them there.
    //   MUL_MAT(q)[+bias] ROPE  MUL_MAT(k)[+bias] ROPE  MUL_MAT(v)[+bias]  SET_ROWS(k) SET_ROWS(v) [CPY mask] FLASH_ATTN_EXT
    // (llama-model.cpp:6004-6043, llama-kv-cache-unified.cpp:1103-1160, llama-graph.cpp:1236-1265)
    int sole_consumer(int from, const b200_tensor & t, const b200_tensor ** as_seen) const {
        uint64_t id = t.id;
        for (int hop = 0; hop < 5; hop++) {
            auto it = uses.find(id);
            if (it == uses.end() || it->second != 1) return -1;
            int c = -1, sidx = -1;
            for (int q = from + 1; q < n && c < 0; q++) for (int sx = 0; sx < nodes[q].n_src && sx < B200_MAX_SRC; sx++) if (nodes[q].src[sx].id == id) { c = q; sidx = sx; break; }
            if (c < 0) return -1;
            if (nodes[c].op != B200_OP_NONE) { *as_seen = &nodes[c].src[sidx]; return c; }
            id = nodes[c].dst.id; from = c;
        }
        return -1;
    }
    bool try_attn_block(int i, int & status) {
        const b200_node & mq = nodes[i];
        const b200_tensor & x = mq.src[1];
        if (x.ne[1] != 1 || (!dry && !ex->ws)) return false;
        if (padded_k(mq.src[0].type, mq.src[0].ne[0]) != mq.src[0].ne[0]) return false;      // padded weight rows: the generic path handles k_valid
        struct Proj { int mm = -1, add = -1; const b200_tensor * out = nullptr; const float * bias = nullptr; } P[3];
        int rope[2] = { -1, -1 };
        int cur = i;
        for (int j = 0; j < 3; j++) {
            if (j > 0) { cur = next_compute(cur); if (cur < 0 || nodes[cur].op != B200_OP_MUL_MAT || !is_weight_type(nodes[cur].src[0].type)) return false; }
            const b200_node & mm = nodes[cur];
            if (mm.src[1].id != x.id || mm.src[1].data != x.data || mm.src[0].ne[0] != mq.src[0].ne[0] || mm.dst.nb[1] != mm.src[0].ne[1] * 4) return false;
            if (is_output(mm.dst)) return false;
            P[j].mm = cur; P[j].out = &mm.dst;
            const int a = next_compute(cur);
            if (a >= 0 && nodes[a].op == B200_OP_ADD && use_count(mm.dst) == 1 && nodes[a].src[0].data == mm.dst.data && nrows_of(nodes[a].src[1]) == 1 &&
                nodes[a].src[1].ne[0] == mm.src[0].ne[1] && nodes[a].dst.nb[1] == mm.src[0].ne[1] * 4) {
                P[j].add = a; P[j].out = &nodes[a].dst; P[j].bias = (const float *)nodes[a].src[1].data; cur = a;
            }
            if (j < 2) {
                const b200_tensor * seen = nullptr;
                const int r = sole_consumer(cur, *P[j].out, &seen);
                if (r < 0 || nodes[r].op != B200_OP_ROPE || r != next_compute(cur)) return false;
                rope[j] = r; cur = r;
            }
        }
        const b200_node & rq = nodes[rope[0]], & rk = nodes[rope[1]];
        if (memcmp(rq.op_params, rk.op_params, sizeof(rq.op_params)) != 0 || rq.src[1].data != rk.src[1].data) return false;
        if ((rq.n_src > 2 ? rq.src[2].data : nullptr) != (rk.n_src > 2 ? rk.src[2].data : nullptr)) return false;
        if (is_output(*P[0].out) || is_output(*P[1].out) || is_output(*P[2].out) || is_output(rk.dst)) return false;   // never materialised by the fused launches
        const b200_tensor & q3 = rq.src[0], & k3 = rk.src[0];
        const int64_t hd = q3.ne[0], nh = q3.ne[1], nhk = k3.ne[1];
        auto dense3 = [&](const b200_tensor & t) { return t.nb[0] == 4 && t.nb[1] == t.ne[0] * 4 && t.nb[2] == t.ne[0] * t.ne[1] * 4; };
        if (q3.ne[2] != 1 || k3.ne[2] != 1 || k3.ne[0] != hd || !dense3(q3) || !dense3(k3) || !dense3(rq.dst) || (hd != 64 && hd != 128)) return false;
        if (nh * hd != nodes[P[0].mm].src[0].ne[1] || nhk * hd != nodes[P[1].mm].src[0].ne[1] || nhk * hd != nodes[P[2].mm].src[0].ne[1] || (nhk * hd) % 256 != 0) return false;
        // KV stores: K consumes exactly the roped K, V exactly the V projection (through views), each once
        const b200_tensor * seen = nullptr;
        const int sk = sole_consumer(rope[1], rk.dst, &seen);
        if (sk < 0 || nodes[sk].op != B200_OP_SET_ROWS || seen != &nodes[sk].src[0] || seen->ne[0] != nhk * hd || seen->ne[1] != 1) return false;
        const int sv = sole_consumer(P[2].add >= 0 ? P[2].add : P[2].mm, *P[2].out, &seen);
        if (sv < 0 || nodes[sv].op != B200_OP_SET_ROWS || seen != &nodes[sv].src[0] || seen->ne[0] != nhk * hd || seen->ne[1] != 1) return false;
        if (sk != next_compute(P[2].add >= 0 ? P[2].add : P[2].mm) || sv != next_compute(sk)) return false;
        const b200_node & SK = nodes[sk], & SV = nodes[sv];
        if (SK.dst.type != SV.dst.type || (SK.dst.type != B200_TYPE_F16 && SK.dst.type != B200_TYPE_Q8_0) || SK.dst.ne[2] != 1 || SV.dst.ne[2] != 1) return false;
        // the roped Q goes to FLASH_ATTN_EXT only; mask casts in between are independent of the block and run first
        const int fa = sole_consumer(rope[0], rq.dst, &seen);
        if (fa < 0 || nodes[fa].op != B200_OP_FLASH_ATTN_EXT || seen != &nodes[fa].src[0]) return false;
        for (int q = next_compute(sv); q >= 0 && q < fa; q = next_compute(q)) if (nodes[q].op != B200_OP_CPY) return false;
        b200_rope_params p; memset(&p, 0, sizeof(p));
        p.n_dims = rq.op_params[1]; p.mode = rq.op_params[2]; p.n_ctx_orig = rq.op_params[4];
        p.freq_base = f32_param(rq, 5); p.freq_scale = f32_param(rq, 6); p.ext_factor = f32_param(rq, 7);
        p.attn_factor = f32_param(rq, 8); p.beta_fast = f32_param(rq, 9); p.beta_slow = f32_param(rq, 10);
        if ((p.mode & ~2) || p.n_dims > hd || p.n_dims % 8 != 0 || (p.mode == 2 && p.n_dims % 16 != 0)) return false;
        const b200_node & F = nodes[fa];
        // executor scratch behind the attention workspace: q | k | v projections of this token
        const size_t fa_ws = (size_t)b200_flash_attn_workspace(hd, nh, 1, F.src[1].ne[1]);
        if (!dry && (((fa_ws + 255) & ~(size_t)255) + (size_t)(nh + 2 * nhk) * hd * 4 + 1024 > ex->fa_bytes)) return false;
        float * sq = dry ? (float *)(uintptr_t)0x10000 : (float *)(ex->ws + ex->off_fa + ((fa_ws + 255) & ~(size_t)255));
        float * skn = sq + nh * hd, * svn = skn + nhk * hd;
        RopePend r;
        r.valid = true; r.q_src = sq; r.q_dst = (float *)rq.dst.data; r.k = skn; r.v = svn; r.pos = (const int32_t *)rq.src[1].data;
        r.ff = rq.n_src > 2 ? (const float *)rq.src[2].data : nullptr; r.k_ids = (const int64_t *)SK.src[1].data; r.v_ids = (const int64_t *)SV.src[1].data;
        r.k_cache = SK.dst.data; r.v_cache = SV.dst.data; r.kv_type = SK.dst.type; r.k_rs = SK.dst.nb[1]; r.v_rs = SV.dst.nb[1]; r.hd = hd; r.nh = nh; r.nhk = nhk; r.p = p;
        rope_pend = r;
        if (!attn_matches(F)) { rope_pend.valid = false; return false; }
        rope_pend.valid = false;
        // ---- commit: the projections (they read the pending norm / x NOW), then independent mask casts that sat between the
        //      KV stores and the attention (their output may recycle x's buffer), then the attention launch
        b200_mmv_launch L; memset(&L, 0, sizeof(L));
        L.k = mq.src[0].ne[0]; L.ncols = 1; L.n_mats = 3;
        fill_act_source(L, x);
        float * outs[3] = { sq, skn, svn };
        for (int j = 0; j < 3; j++) {
            const b200_node & mm = nodes[P[j].mm];
            L.mats[j] = { mm.src[0].data, outs[j], P[j].bias, mm.src[0].ne[1], mm.src[0].type, 0 };
            if (j) done[P[j].mm] = 1;
            if (P[j].add >= 0) done[P[j].add] = 1;
        }
        status = launch_mmv(L);
        done[rope[0]] = done[rope[1]] = done[sk] = done[sv] = done[fa] = 1;
        if (status != B200_OK) return true;
        for (int q = next_compute(sv); q >= 0 && q < fa; q = next_compute(q)) { status = run_node(q); done[q] = 1; if (status != B200_OK) return true; }
        rope_pend = r;
        status = (mega && mk_try_attn(F)) ? (int)B200_OK : launch_fused_attn(F);      // a phase of the persistent kernel, or its own launch
        invalidate_act(rq.dst); invalidate_act(F.dst);
        return true;
    }

    int run_mul_mat(int i) {
        const b200_node & n = nodes[i];
        const b200_tensor & w = n.src[0], & x = n.src[1];
        const int64_t kv = w.ne[0], k = padded_k(w.type, kv), m = w.ne[1], ncols = x.ne[1];   // kv: elements that exist in x; k: padded weight rows
        if (w.type == B200_TYPE_F16) {
            // attention without -fa: KQ / KQV over f16 views of the KV cache (GQA broadcast over dim 2)
            { const int fs = mk_flush(); if (fs != B200_OK) return fs; }
            invalidate_act(n.dst);
            return KL(b200_mul_mat_f16(w.data, w.nb[1], w.nb[2], w.ne[2], (const float *)x.data, x.nb[1], x.nb[2], (float *)n.dst.data, n.dst.nb[1], n.dst.nb[2],
                                       w.ne[1], x.ne[1], x.ne[2], w.ne[0], st));
        }
        if (w.type == B200_TYPE_F32) {
            // the f32 router matrix of a mixture-of-experts layer (ffn_gate_inp): router-sized, one warp per output
            { const int fs = mk_flush(); if (fs != B200_OK) return fs; }
            invalidate_act(n.dst);
            return KL(b200_mul_mat_f32((const float *)w.data, w.nb[1] / 4, (const float *)x.data, x.nb[1] / 4, (float *)n.dst.data, n.dst.nb[1] / 4, m, kv, ncols, st));
        }
        if (is_wide_only_type(w.type)) {
            // a format only the wide matvec reads (mmvq_ext.cu): f32 activations in, quantised inside the kernel; one pass over the weights per column
            { const int fs = mk_flush(); if (fs != B200_OK) return fs; }
            invalidate_act(n.dst);
            return KL(b200_mul_mat_vec_wide(w.type, w.data, (const float *)x.data, x.nb[1] / 4, (float *)n.dst.data, n.dst.nb[1] / 4, nullptr, nullptr, m, kv, ncols, st));
        }
        if (ncols > 8) {
            { const int fs = mk_flush(); if (fs != B200_OK) return fs; }
            invalidate_act(n.dst);
            ex->act_id[0] = ex->act_id[1] = 0;           // the batched path owns the act buffers
            const int kind = b200_act_kind_for(w.type);
            return KL(b200_mul_mat_q2(w.type, w.data, (const float *)x.data, x.nb[1] / 4, (float *)n.dst.data, n.dst.nb[1] / 4, m, k, kv, ncols, act_buf(kind), st));
        }
        int s = B200_OK;
        if (fuse && ncols == 1 && try_attn_block(i, s)) return s;
        b200_mmv_launch L; memset(&L, 0, sizeof(L));
        L.k = k; L.ncols = ncols; L.k_valid = kv;
        if (fuse) {
            // (1) up, gate, GLU (llama-graph.cpp:647-693): MUL_MAT(up,x) MUL_MAT(gate,x) GLU(gate,up)
            const int j = next_compute(i);
            if (j >= 0 && nodes[j].op == B200_OP_MUL_MAT && is_weight_type(nodes[j].src[0].type) && nodes[j].src[1].id == x.id && nodes[j].src[1].data == x.data && nodes[j].src[0].ne[1] == m && nodes[j].src[1].ne[1] == ncols) {
                const int g = next_compute(j);
                const bool x_live = g >= 0 && (overlaps(nodes[g].dst, x) || (ex->norm.out_id && ex->norm.out_id == x.id && overlaps(nodes[g].dst, ex->norm.x)));   // late CTAs still quantise x in their prologue
                if (g >= 0 && nodes[g].op == B200_OP_GLU_SWIGLU && use_count(n.dst) == 1 && use_count(nodes[j].dst) == 1 &&
                    n.dst.nb[1] == m * 4 && nodes[j].dst.nb[1] == m * 4 && !x_live && !is_output(n.dst) && !is_output(nodes[j].dst)) {
                    const b200_node & G = nodes[g];
                    const b200_node * gate = nullptr, * up = nullptr;
                    if (G.src[0].data == nodes[j].dst.data && G.src[1].data == n.dst.data) { gate = &nodes[j]; up = &n; }
                    else if (G.src[0].data == n.dst.data && G.src[1].data == nodes[j].dst.data) { gate = &n; up = &nodes[j]; }
                    if (gate && G.dst.nb[1] == m * 4) {
                        fill_act_source(L, x);
                        L.n_mats = 2; L.swiglu = 1;
                        L.mats[0] = { gate->src[0].data, (float *)G.dst.data, nullptr, m, gate->src[0].type, 0 };
                        L.mats[1] = { up->src[0].data, (float *)G.dst.data, nullptr, m, up->src[0].type, 0 };
                        done[j] = done[g] = 1;
                        s = launch_mmv(L);
                        invalidate_act(G.dst);
                        return s;
                    }
                }
            }
            // (2) several projections of one activation (QKV, llama-model.cpp:6004-6022) in one launch;
            //     later MUL_MATs are hoisted only if their outputs alias nothing that is still live
            int group[MAX_GROUP] = { i }; int ng = 1;
            for (int j2 = i + 1; j2 < n_limit(i) && ng < MAX_GROUP; j2++) {
                if (done[j2] || nodes[j2].op != B200_OP_MUL_MAT || !is_weight_type(nodes[j2].src[0].type)) continue;
                const b200_node & o = nodes[j2];
                if (o.src[1].id != x.id || o.src[1].data != x.data || o.src[1].ne[1] != ncols || o.src[0].ne[0] != kv || padded_k(o.src[0].type, kv) != k) continue;
                if (o.dst.nb[1] != o.src[0].ne[1] * 4 || !can_hoist(i, j2)) continue;
                if (overlaps(o.dst, x) || (ex->norm.out_id && ex->norm.out_id == x.id && overlaps(o.dst, ex->norm.x))) continue;
                group[ng++] = j2;
            }
            if (ng > 1 && n.dst.nb[1] == m * 4) {
                fill_act_source(L, x);
                L.n_mats = ng;
                const b200_tensor * written[2 * MAX_GROUP]; int nw = 0;
                for (int q = 0; q < ng; q++) {
                    const b200_node & o = nodes[group[q]];
                    L.mats[q] = { o.src[0].data, (float *)o.dst.data, nullptr, o.src[0].ne[1], o.src[0].type, 0 };
                    if (q) done[group[q]] = 1;
                    written[nw++] = &o.dst;
                    // bias ADD right after the projection (Qwen2 QKV bias, llama-model.cpp:6006-6020)
                    const int a = next_compute(group[q]);
                    if (a >= 0 && nodes[a].op == B200_OP_ADD && use_count(o.dst) == 1 && !is_output(o.dst) && nodes[a].src[0].data == o.dst.data && nrows_of(nodes[a].src[1]) == 1 &&
                        nodes[a].src[1].ne[0] == o.src[0].ne[1] && nodes[a].dst.nb[1] == o.src[0].ne[1] * 4 && (q == 0 || can_hoist(i, a)) &&
                        !overlaps(nodes[a].dst, x) && !(ex->norm.out_id && ex->norm.out_id == x.id && overlaps(nodes[a].dst, ex->norm.x))) {
                        L.mats[q].bias = (const float *)nodes[a].src[1].data; L.mats[q].dst = (float *)nodes[a].dst.data; done[a] = 1;
                        written[nw++] = &nodes[a].dst;
                    }
                }
                s = launch_mmv(L);
                for (int q = 0; q < nw; q++) invalidate_act(*written[q]);
                return s;
            }
            // (3) epilogue: + bias row, + residual (wo / ffn_down followed by ADD, llama-model.cpp:6052,6095)
            const float * bias = nullptr, * resid = nullptr; const b200_tensor * out = &n.dst;
            int cur = i;
            for (int step = 0; step < 2; step++) {
                const int a = next_compute(cur);
                if (a < 0 || nodes[a].op != B200_OP_ADD || use_count(*out) != 1 || is_output(*out)) break;
                const b200_node & A = nodes[a];
                const b200_tensor * other = A.src[0].data == out->data ? &A.src[1] : (A.src[1].data == out->data ? &A.src[0] : nullptr);
                if (!other || A.dst.nb[1] != out->nb[1] || !same_shape(A.dst, *out)) break;
                if (overlaps(A.dst, x) || (ex->norm.out_id && ex->norm.out_id == x.id && overlaps(A.dst, ex->norm.x))) break;   // other CTAs still read the activation
                if (!bias && !resid && nrows_of(*other) == 1 && other->ne[0] == m) bias = (const float *)other->data;
                else if (!resid && same_shape(*other, *out) && other->nb[1] == out->nb[1]) resid = (const float *)other->data;
                else break;
                done[a] = 1; out = &A.dst; cur = a;
            }
            fill_act_source(L, x);
            L.n_mats = 1;
            L.mats[0] = { w.data, (float *)out->data, bias, m, w.type, 0 };
            L.residual[0] = resid; L.dst_col_stride[0] = out->nb[1] / 4;
            s = launch_mmv(L);
            invalidate_act(*out);
            return s;
        }
        const int kind = b200_act_kind_for(w.type);
        s = mk_flush();
        if (s != B200_OK) return s;
        s = ensure_act(x, kind, k);
        if (s != B200_OK) return s;
        invalidate_act(n.dst);
        return KL(b200_mul_mat_vec_q(w.type, w.data, act_buf(kind), (float *)n.dst.data, n.dst.nb[1] / 4, nullptr, nullptr, m, k, ncols, st));
    }
    static constexpr int MAX_GROUP = 4;
    int last_status = B200_OK;

    // ROPE(q) ROPE(k) SET_ROWS(k -> K cache) SET_ROWS(v -> V cache) -> one launch (llama-model.cpp:6029-6043 +
    // llama-kv-cache-unified.cpp:1103-1160).  The roped K is consumed only by the KV store, so it is never written as f32.
    bool try_rope_kv_store(int i) {
        const b200_node & rq = nodes[i];
        const int j = next_compute(i); if (j < 0 || nodes[j].op != B200_OP_ROPE) return false;
        const b200_node & rk = nodes[j];
        const int sk = next_compute(j); if (sk < 0 || nodes[sk].op != B200_OP_SET_ROWS) return false;
        const int sv = next_compute(sk); if (sv < 0 || nodes[sv].op != B200_OP_SET_ROWS) return false;
        const b200_node & SK = nodes[sk], & SV = nodes[sv];
        if (memcmp(rq.op_params, rk.op_params, sizeof(rq.op_params)) != 0 || rq.src[1].data != rk.src[1].data) return false;
        if ((rq.n_src > 2 ? rq.src[2].data : nullptr) != (rk.n_src > 2 ? rk.src[2].data : nullptr)) return false;
        const b200_tensor & q = rq.src[0], & k = rk.src[0], & v = SV.src[0];
        const int64_t hd = q.ne[0], nh = q.ne[1], nhk = k.ne[1], nt = q.ne[2];
        auto dense3 = [&](const b200_tensor & t) { return t.nb[0] == 4 && t.nb[1] == t.ne[0] * 4 && t.nb[2] == t.ne[0] * t.ne[1] * 4; };
        if (!dense3(q) || !dense3(k) || !dense3(rq.dst) || !dense3(rk.dst) || k.ne[0] != hd || k.ne[2] != nt || (nhk * hd) % 256 != 0) return false;
        // K store consumes exactly the roped K (through a reshape view), V store a dense [n_embd_v, n_tok] f32 tensor
        if (SK.src[0].data != rk.dst.data || SK.src[0].ne[0] != nhk * hd || SK.src[0].ne[1] != nt || SK.src[0].nb[1] != nhk * hd * 4) return false;
        if (v.ne[0] != nhk * hd || v.ne[1] != nt || v.nb[1] != nhk * hd * 4 || v.ne[2] != 1 || SK.src[0].ne[2] != 1 || SK.dst.ne[2] != 1 || SV.dst.ne[2] != 1) return false;
        if (SK.dst.type != SV.dst.type || (SK.dst.type != B200_TYPE_F16 && SK.dst.type != B200_TYPE_Q8_0) || is_output(rk.dst)) return false;
        // the roped K must have no other reader: it feeds SET_ROWS directly or through exactly one view node
        // (identity by tensor id — buffers are recycled by the graph allocator, pointers are not identities)
        if (SK.src[0].id != rk.dst.id) {
            if (use_count(rk.dst) != 1 || use_count(SK.src[0]) != 1) return false;
            bool via_view = false;
            for (int q2 = j + 1; q2 < sk; q2++) if (nodes[q2].op == B200_OP_NONE && nodes[q2].dst.id == SK.src[0].id && nodes[q2].src[0].id == rk.dst.id) via_view = true;
            if (!via_view) return false;
        } else if (use_count(rk.dst) != 1) return false;
        b200_rope_params p; memset(&p, 0, sizeof(p));
        p.n_dims = rq.op_params[1]; p.mode = rq.op_params[2]; p.n_ctx_orig = rq.op_params[4];
        p.freq_base = f32_param(rq, 5); p.freq_scale = f32_param(rq, 6); p.ext_factor = f32_param(rq, 7);
        p.attn_factor = f32_param(rq, 8); p.beta_fast = f32_param(rq, 9); p.beta_slow = f32_param(rq, 10);
        const float * ff = rq.n_src > 2 ? (const float *)rq.src[2].data : nullptr;
        if (nt == 1 && (hd == 64 || hd == 128) && rq.dst.data && (p.mode & ~2) == 0 && p.n_dims <= hd && p.n_dims % 8 == 0 && (p.mode != 2 || p.n_dims % 16 == 0)) {
            // decode token: recorded, and merged with the FLASH_ATTN_EXT that follows (one fused launch, or a phase of the persistent kernel)
            last_status = mk_flush_rope_only();
            RopePend & r = rope_pend;
            r.valid = true; r.q_src = (const float *)q.data; r.q_dst = (float *)rq.dst.data; r.k = (const float *)k.data; r.v = (const float *)v.data;
            r.pos = (const int32_t *)rq.src[1].data; r.ff = ff; r.k_ids = (const int64_t *)SK.src[1].data; r.v_ids = (const int64_t *)SV.src[1].data;
            r.k_cache = SK.dst.data; r.v_cache = SV.dst.data; r.kv_type = SK.dst.type; r.k_rs = SK.dst.nb[1]; r.v_rs = SV.dst.nb[1]; r.hd = hd; r.nh = nh; r.nhk = nhk; r.p = p;
        } else {
            last_status = mk_flush();
            if (last_status == B200_OK)
            last_status = KL(b200_rope_kv_store2((const float *)q.data, (float *)rq.dst.data, (const float *)k.data, (const float *)v.data, (const int32_t *)rq.src[1].data, ff,
                                              (const int64_t *)SK.src[1].data, (const int64_t *)SV.src[1].data, SK.dst.data, SV.dst.data, SK.dst.type,
                                              SK.dst.nb[1], SV.dst.nb[1], hd, nh, nhk, nt, &p, st));
        }
        done[j] = done[sk] = done[sv] = 1;
        invalidate_act(rq.dst);
        return true;
    }
    int n_limit(int i) const { return i + 24 < n ? i + 24 : n; }

    // does this node read or write anything the recorded (not yet launched) rope + KV store produces or consumes?
    bool touches_rope_pend(const b200_node & n) const {
        const RopePend & r = rope_pend;
        auto range = [](const void * p, int64_t bytes) { b200_tensor t; memset(&t, 0, sizeof(t)); t.data = (void *)p; t.type = B200_TYPE_F32; t.ne[0] = bytes / 4; t.ne[1] = t.ne[2] = t.ne[3] = 1; t.nb[0] = 4; t.nb[1] = t.nb[2] = t.nb[3] = bytes; return t; };
        const b200_tensor qd = range(r.q_dst, r.nh * r.hd * 4), qs = range(r.q_src, r.nh * r.hd * 4), kn = range(r.k, r.nhk * r.hd * 4), vn = range(r.v, r.nhk * r.hd * 4);
        for (int s = 0; s < n.n_src && s < B200_MAX_SRC; s++) {
            const b200_tensor & t = n.src[s];
            if (!t.data) continue;
            if (overlaps(t, qd) || t.data == r.k_cache || t.data == r.v_cache) return true;      // reads the roped Q or the KV cells
        }
        return overlaps(n.dst, qd) || overlaps(n.dst, qs) || overlaps(n.dst, kn) || overlaps(n.dst, vn) || n.dst.data == r.k_cache || n.dst.data == r.v_cache;
    }

    int run_node(int i) {
        const b200_node & n = nodes[i];
        if (rope_pend.valid && n.op != B200_OP_NONE && n.op != B200_OP_FLASH_ATTN_EXT && touches_rope_pend(n)) {
            const int fs = mk_flush(); if (fs != B200_OK) return fs;
        }
        if (mega && n.op != B200_OP_NONE && n.op != B200_OP_MUL_MAT && n.op != B200_OP_ROPE && n.op != B200_OP_FLASH_ATTN_EXT && n.op != B200_OP_RMS_NORM) {
            const int fs = mk_flush(); if (fs != B200_OK) return fs;            // everything else is an ordinary launch: keep program order
        }
        switch (n.op) {
            case B200_OP_NONE: return B200_OK;
            case B200_OP_RMS_NORM: return run_rms_norm(i);
            case B200_OP_MUL_MAT:  return run_mul_mat(i);
            case B200_OP_MUL: case B200_OP_ADD: case B200_OP_DIV: {
                invalidate_act(n.dst);
                const b200_tensor & a = n.src[0], & b = n.src[1];
                if (n.op == B200_OP_DIV || !bin_ok(n))        // broadcast over other dims / strided views (MoE router glue): the general kernel
                    return KL(b200_binary_strided(n.op == B200_OP_ADD ? 0 : (n.op == B200_OP_MUL ? 1 : 2), (const float *)a.data, a.nb, (const float *)b.data, b.ne, b.nb,
                                                  (float *)n.dst.data, n.dst.ne, n.dst.nb, st));
                const int64_t rows = nrows_of(a), brows = same_shape(a, b) ? rows : b.ne[1];
                return KL(n.op == B200_OP_ADD ? b200_add((const float *)a.data, (const float *)b.data, (float *)n.dst.data, a.ne[0], rows, brows, st)
                                              : b200_mul((const float *)a.data, (const float *)b.data, (float *)n.dst.data, a.ne[0], rows, brows, st));
            }
            case B200_OP_ROPE: {
                if (fuse && try_rope_kv_store(i)) return last_status;
                { const int fs = mk_flush(); if (fs != B200_OK) return fs; }
                invalidate_act(n.dst);
                const b200_tensor & x = n.src[0];
                b200_rope_params p; memset(&p, 0, sizeof(p));
                p.n_dims = n.op_params[1]; p.mode = n.op_params[2]; p.n_ctx_orig = n.op_params[4];
                p.freq_base = f32_param(n, 5); p.freq_scale = f32_param(n, 6); p.ext_factor = f32_param(n, 7);
                p.attn_factor = f32_param(n, 8); p.beta_fast = f32_param(n, 9); p.beta_slow = f32_param(n, 10);
                const float * ff = n.n_src > 2 ? (const float *)n.src[2].data : nullptr;
                return KL(b200_rope((const float *)x.data, (float *)n.dst.data, (const int32_t *)n.src[1].data, ff, x.ne[0], x.ne[1], x.ne[2],
                                    x.nb[1] / 4, x.nb[2] / 4, n.dst.nb[1] / 4, n.dst.nb[2] / 4, &p, st));
            }
            case B200_OP_SCALE:
                invalidate_act(n.dst);
                return KL(b200_unary(0, (const float *)n.src[0].data, (float *)n.dst.data, nelem(n.dst), f32_param(n, 0), f32_param(n, 1), st));
            case B200_OP_UNARY:
                invalidate_act(n.dst);
                return KL(b200_unary(n.op_params[0] == 10 ? 1 : 2, (const float *)n.src[0].data, (float *)n.dst.data, nelem(n.dst), 0.0f, 0.0f, st));
            case B200_OP_CONT: {
                invalidate_act(n.dst);
                const b200_tensor & s0 = n.src[0];
                const int64_t one[4] = { 1, 1, 1, 1 }, four[4] = { 4, 4, 4, 4 };
                const int64_t dnb[4] = { 4, 4 * s0.ne[0], 4 * s0.ne[0] * s0.ne[1], 4 * s0.ne[0] * s0.ne[1] * s0.ne[2] };    // dst is contiguous: src0's logical order
                return KL(b200_binary_strided(3, (const float *)s0.data, s0.nb, (const float *)s0.data, one, four, (float *)n.dst.data, s0.ne, dnb, st));
            }
            case B200_OP_SET_ROWS: {
                const b200_tensor & s = n.src[0], & ids = n.src[1];
                if (s.ne[0] == 1 && !set_rows_ok(n))         // one-element rows: the transposed V cache of attention without -fa
                    return KL(b200_scatter_rows1((const float *)s.data, (const int64_t *)ids.data, n.dst.data, n.dst.type, s.ne[1], n.dst.ne[1], st));
                for (int64_t i3 = 0; i3 < s.ne[3]; i3++) for (int64_t i2 = 0; i2 < s.ne[2]; i2++) {
                    const int64_t i11 = i2 % ids.ne[1], i12 = i3 % ids.ne[2];
                    if (n.dst.type == B200_TYPE_Q4_0) {
                        const int r4 = KL(b200_set_rows_q4_0((const float *)((const char *)s.data + i2 * s.nb[2] + i3 * s.nb[3]), s.nb[1] / 4,
                                                            (const int64_t *)((const char *)ids.data + i11 * ids.nb[1] + i12 * ids.nb[2]),
                                                            (char *)n.dst.data + i2 * n.dst.nb[2] + i3 * n.dst.nb[3], n.dst.nb[1], s.ne[0], s.ne[1], st));
                        if (r4 != B200_OK) return r4;
                        continue;
                    }
                    const int r = KL(b200_set_rows((const float *)((const char *)s.data + i2 * s.nb[2] + i3 * s.nb[3]), s.nb[1] / 4,
                                                (const int64_t *)((const char *)ids.data + i11 * ids.nb[1] + i12 * ids.nb[2]),
                                                (char *)n.dst.data + i2 * n.dst.nb[2] + i3 * n.dst.nb[3], n.dst.type, n.dst.nb[1], s.ne[0], s.ne[1], st));
                    if (r != B200_OK) return r;
                }
                return B200_OK;
            }
            case B200_OP_FLASH_ATTN_EXT: {
                invalidate_act(n.dst);
                const b200_tensor & q = n.src[0], & k = n.src[1], & v = n.src[2];
                const void * mask = n.n_src > 3 ? n.src[3].data : nullptr;
                const int64_t mrs = mask ? n.src[3].nb[1] / 2 : 0;
                if (mk_try_attn(n)) return B200_OK;
                if (attn_matches(n)) return launch_fused_attn(n);
                { const int fs = mk_flush(); if (fs != B200_OK) return fs; }
                if (q.ne[0] != 64 && q.ne[0] != 128)
                    return KL(b200_flash_attn_any(k.type, (const float *)q.data, q.nb[1] / 4, q.nb[2] / 4, k.data, k.nb[1], k.nb[2], v.data, v.nb[1], v.nb[2], mask, mrs,
                                                  (float *)n.dst.data, q.ne[0], q.ne[2], k.ne[2], q.ne[1], k.ne[1], f32_param(n, 0), f32_param(n, 1), f32_param(n, 2), st));
                if (k.type == B200_TYPE_Q4_0)
                    return KL(b200_flash_attn_q4_0((const float *)q.data, q.nb[1] / 4, q.nb[2] / 4, k.data, k.nb[1], k.nb[2], v.data, v.nb[1], v.nb[2], mask, mrs,
                                                   (float *)n.dst.data, q.ne[0], q.ne[2], k.ne[2], q.ne[1], k.ne[1], f32_param(n, 0), f32_param(n, 1), f32_param(n, 2), st));
                return KL(b200_flash_attn_ext((const float *)q.data, q.nb[1] / 4, q.nb[2] / 4, k.data, k.nb[1], k.nb[2], v.data, v.nb[1], v.nb[2], mask, mrs,
                                           (float *)n.dst.data, k.type, q.ne[0], v.ne[0], q.ne[2], k.ne[2], q.ne[1], k.ne[1],
                                           f32_param(n, 0), f32_param(n, 1), f32_param(n, 2), ex->ws + ex->off_fa, st));
            }
            case B200_OP_GLU_SWIGLU:
                invalidate_act(n.dst);
                return KL(b200_swiglu((const float *)n.src[0].data, (const float *)n.src[1].data, (float *)n.dst.data, nelem(n.dst), st));
            case B200_OP_SOFT_MAX:
                invalidate_act(n.dst);
                if (n.n_src > 1 && n.src[1].id)
                    return KL(b200_soft_max_mask((const float *)n.src[0].data, (float *)n.dst.data, n.src[1].data, n.src[1].type == B200_TYPE_F16, n.src[1].nb[1] / n.src[1].nb[0],
                                                 n.src[0].ne[0], n.src[0].ne[1], n.src[0].ne[2], f32_param(n, 0), f32_param(n, 1), st));
                return KL(b200_soft_max_rows((const float *)n.src[0].data, n.src[0].ne[0], (float *)n.dst.data, n.dst.ne[0], n.src[0].ne[0], nrows_of(n.src[0]), f32_param(n, 0), st));
            case B200_OP_ARGSORT:
                return KL(b200_argsort_rows((const float *)n.src[0].data, n.src[0].ne[0], (int32_t *)n.dst.data, n.dst.ne[0], n.src[0].ne[0], nrows_of(n.src[0]), n.op_params[0] == 1, st));
            case B200_OP_SUM_ROWS:
                invalidate_act(n.dst);
                return KL(b200_sum_rows((const float *)n.src[0].data, n.src[0].ne[0], (float *)n.dst.data, n.src[0].ne[0], nrows_of(n.src[0]), st));
            case B200_OP_MUL_MAT_ID: {
                // expert routing on the device: the kernels read ids themselves (no stream synchronisation, unlike ggml-cuda.cu:2115-2125).
                // Prefill ubatches take the grouped tensor-core path (3 launches, its workspace is the q8_K act buffer); decode / verify
                // batches the one-launch matvec of b200_mul_mat_id
                invalidate_act(n.dst);
                const b200_tensor & w = n.src[0], & x = n.src[1], & ids = n.src[2];
                if (b200_mul_mat_id_q_workspace(w.type, w.ne[1], w.ne[0], w.ne[2], ids.ne[0], ids.ne[1]) > 0) {
                    ex->act_id[0] = ex->act_id[1] = 0;       // the grouped path owns the act buffers
                    if (dry) planned += 2;                   // routing + gathered quantisation ahead of the GEMM
                }
                return KL(b200_mul_mat_id_q(w.type, w.data, w.nb[2], (const float *)x.data, x.nb[2] / 4, x.nb[1] / 4, x.ne[1], (const int32_t *)ids.data, ids.nb[1] / 4,
                                            (float *)n.dst.data, n.dst.nb[2] / 4, n.dst.nb[1] / 4, w.ne[1], w.ne[0], w.ne[2], ids.ne[0], ids.ne[1], act_buf(0), st));
            }
            case B200_OP_GET_ROWS:
                invalidate_act(n.dst);
                if (n.src[0].type == B200_TYPE_F32 && !get_rows_f32_ok(n))
                    return KL(b200_get_rows_f32_batched((const float *)n.src[0].data, n.src[0].nb[1] / 4, n.src[0].nb[2] / 4, n.src[0].ne[1], (const int32_t *)n.src[1].data, n.src[1].nb[1] / 4,
                                                        (float *)n.dst.data, n.dst.nb[1] / 4, n.dst.nb[2] / 4, n.src[0].ne[0], n.src[1].ne[0], n.src[0].ne[2], st));
                if (n.src[0].type != B200_TYPE_F32)
                    return KL(b200_get_rows_q(n.src[0].type, n.src[0].data, n.src[0].nb[1], n.src[0].ne[1], (const int32_t *)n.src[1].data, (float *)n.dst.data, n.dst.nb[1] / 4,
                                              n.src[0].ne[0], n.src[1].ne[0], st));
                return KL(b200_get_rows_f32((const float *)n.src[0].data, n.src[0].nb[1] / 4, (const int32_t *)n.src[1].data, (float *)n.dst.data, n.src[0].ne[0], n.src[1].ne[0], st));
            case B200_OP_CPY:
                invalidate_act(n.dst);
                if (n.dst.type == B200_TYPE_F16) return KL(b200_cpy_f32_f16((const float *)n.src[0].data, n.dst.data, nelem(n.dst), st));
                return KL(b200_check(cudaMemcpyAsync(n.dst.data, n.src[0].data, (size_t)nelem(n.dst) * 4, cudaMemcpyDeviceToDevice, st), "cpy f32"));
            default:
                b200_set_error("executor: op %d not supported", n.op);
                return B200_ERR_UNSUPPORTED;
        }
    }

    int run_all() {
        done.assign(n, 0);
        uses.clear();
        for (int i = 0; i < n; i++) for (int s = 0; s < nodes[i].n_src && s < B200_MAX_SRC; s++) if (nodes[i].src[s].id) uses[nodes[i].src[s].id]++;
        ex->act_id[0] = ex->act_id[1] = 0;
        ex->norm.out_id = 0;
        pend.clear(); rope_pend.valid = false; tab.valid = false;
        for (int i = 0; i < n; i++) {
            if (done[i] || nelem(nodes[i].dst) == 0) continue;       // empty tensors (prompt ubatches that request no logits) are skipped
            const int s = run_node(i);
            if (s != B200_OK) return s;
        }
        return mk_flush();
    }
};

uint64_t mix(uint64_t h, uint64_t v) { h ^= v + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2); return h * 0xff51afd7ed558ccdull; }

uint64_t topology_key(const b200_node * nodes, int n, int flags) {
    uint64_t h = 0x12345678abcdefull ^ (uint64_t)n ^ ((uint64_t)flags << 48);
    for (int i = 0; i < n; i++) {
        const b200_node & nd = nodes[i];
        h = mix(h, (uint64_t)nd.op | ((uint64_t)nd.n_src << 32));
        h = mix(h, (uint64_t)(uintptr_t)nd.dst.data); h = mix(h, (uint64_t)nd.dst.ne[0] ^ ((uint64_t)nd.dst.ne[1] << 24) ^ ((uint64_t)nd.dst.ne[2] << 48)); h = mix(h, (uint64_t)nd.dst.nb[1]);
        for (int s = 0; s < nd.n_src && s < B200_MAX_SRC; s++) {
            const b200_tensor & t = nd.src[s];
            h = mix(h, (uint64_t)(uintptr_t)t.data); h = mix(h, (uint64_t)t.ne[0] ^ ((uint64_t)t.ne[1] << 24) ^ ((uint64_t)t.ne[2] << 48)); h = mix(h, (uint64_t)t.nb[1] ^ ((uint64_t)t.nb[2] << 20) ^ ((uint64_t)t.type << 56));
        }
        if (nd.op != B200_OP_NONE) for (int p = 0; p < 12; p += 2) h = mix(h, (uint64_t)(uint32_t)nd.op_params[p] | ((uint64_t)(uint32_t)nd.op_params[p + 1] << 32));
    }
    return h;
}

// workspace needs of a node list (no allocation may happen during stream capture)
int plan_workspace(b200_executor * ex, const b200_node * nodes, int n) {
    size_t act[2] = { 0, 0 }, fa = 0;
    for (int i = 0; i < n; i++) {
        const b200_node & nd = nodes[i];
        if (nd.op == B200_OP_MUL_MAT) {
            const int64_t k = (nd.src[0].ne[0] + 255) / 256 * 256, cols = nd.src[1].ne[1];
            for (int kd = 0; kd < 2; kd++) { const size_t b = (size_t)(cols * act_col_bytes(kd, k)); if (b > act[kd]) act[kd] = b; }
            if (cols > 8 && is_weight_type(nd.src[0].type)) {   // batched path: the tensor-core kernel's pre-tiled activation image
                const int kd = b200_act_kind_for(nd.src[0].type);
                const size_t b = (size_t)b200_mul_mat_q_workspace(nd.src[0].type, nd.src[0].ne[1], k, cols);
                if (kd >= 0 && b > act[kd]) act[kd] = b;
            }
        } else if (nd.op == B200_OP_MUL_MAT_ID && nd.n_src >= 3) {   // grouped prefill path: routing + the gathered B image
            const size_t b = (size_t)b200_mul_mat_id_q_workspace(nd.src[0].type, nd.src[0].ne[1], nd.src[0].ne[0], nd.src[0].ne[2], nd.src[2].ne[0], nd.src[2].ne[1]);
            if (b > act[0]) act[0] = b;
        } else if (nd.op == B200_OP_RMS_NORM) {
            for (int kd = 0; kd < 2; kd++) { const size_t b = (size_t)(8 * act_col_bytes(kd, (nd.src[0].ne[0] + 255) / 256 * 256)); if (b > act[kd]) act[kd] = b; }
        } else if (nd.op == B200_OP_FLASH_ATTN_EXT) {
            size_t b = (size_t)b200_flash_attn_workspace(nd.src[2].ne[0], nd.src[0].ne[2], nd.src[0].ne[1], nd.src[1].ne[1]);
            if (nd.src[0].ne[1] == 1) b = ((b + 255) & ~(size_t)255) + (size_t)(nd.src[0].ne[2] + 2 * nd.src[1].ne[2]) * nd.src[0].ne[0] * 4 + 512;   // + q|k|v scratch of try_attn_block
            b = ((b + 255) & ~(size_t)255) + 1024;                // + the per-token rope table (last KiB of the region)
            if (b > fa) fa = b;
        }
    }
    if (act[0] <= ex->act_bytes[0] && act[1] <= ex->act_bytes[1] && fa <= ex->fa_bytes && ex->ws) return B200_OK;
    for (int kd = 0; kd < 2; kd++) if (act[kd] < ex->act_bytes[kd]) act[kd] = ex->act_bytes[kd];
    if (fa < ex->fa_bytes) fa = ex->fa_bytes;
    auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t total = up(act[0]) + up(act[1]) + up(fa) + 256;
    // growing invalidates every captured graph (they hold the old pointers)
    for (auto & g : ex->graphs) if (g.second.exec) cudaGraphExecDestroy(g.second.exec);
    ex->graphs.clear();
    if (ex->ws) { cudaDeviceSynchronize(); cudaFree(ex->ws); ex->ws = nullptr; }
    if (cudaMalloc((void **)&ex->ws, total) != cudaSuccess || cudaMemset(ex->ws, 0, total) != cudaSuccess) {   /* zeroed once: flash-attn split counters */ cudaGetLastError(); b200_set_error("executor: cannot allocate %zu bytes of workspace", total); return B200_ERR_CUDA; }
    ex->ws_bytes = total;
    ex->off_act[0] = 0; ex->off_act[1] = up(act[0]); ex->off_fa = up(act[0]) + up(act[1]);
    ex->act_bytes[0] = act[0]; ex->act_bytes[1] = act[1]; ex->fa_bytes = fa;
    return B200_OK;
}

} // namespace

extern "C" b200_executor * b200_executor_create(int device) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) { cudaGetLastError(); b200_set_error("executor: no CUDA device %d", device); return nullptr; }
    b200_executor * ex = new b200_executor();
    ex->device = device;
    ex->env_no_graphs = getenv("GGML_B200_DISABLE_GRAPHS") != nullptr;
    ex->env_no_fusion = getenv("GGML_B200_DISABLE_FUSION") != nullptr;
    ex->env_no_mega   = getenv("GGML_B200_DISABLE_MEGAKERNEL") != nullptr;
    ex->env_mega      = getenv("GGML_B200_MEGAKERNEL") != nullptr;       // opt-in for callers that cannot pass flags (the ggml plug-in)
    ex->env_mega_mmv  = getenv("GGML_B200_MEGA_MMV") != nullptr;
    return ex;
}

extern "C" void b200_executor_free(b200_executor * ex) {
    if (!ex) return;
    cudaSetDevice(ex->device);
    for (auto & g : ex->graphs) if (g.second.exec) cudaGraphExecDestroy(g.second.exec);
    if (ex->ws) cudaFree(ex->ws);
    for (auto & pr : ex->progs) { if (pr.second.dev) cudaFree(pr.second.dev); if (pr.second.host) cudaFreeHost(pr.second.host); }
    if (ex->mk_sync) cudaFree(ex->mk_sync);
    delete ex;
}

extern "C" int b200_executor_wide_enabled(void) { return wide_on() ? 1 : 0; }
extern "C" int b200_executor_supports(const b200_node * node) { return node && node_ok(*node) ? 1 : 0; }

extern "C" int b200_executor_compute(b200_executor * ex, const b200_node * nodes, int n_nodes, void * stream, int flags) {
    if (!ex || (!nodes && n_nodes > 0) || n_nodes < 0) { b200_set_error("executor: bad arguments"); return B200_ERR_INVALID; }
    B200_CUDA(cudaSetDevice(ex->device));
    for (int i = 0; i < n_nodes; i++) if (!node_ok(nodes[i])) { b200_set_error("executor: node %d (op %d) is not supported", i, nodes[i].op); return B200_ERR_UNSUPPORTED; }
    int s = plan_workspace(ex, nodes, n_nodes);
    if (s != B200_OK) return s;
    cudaStream_t st = (cudaStream_t)stream;
    Runner r{ ex, nodes, n_nodes, st, (flags & B200_EXEC_FUSION) && !ex->env_no_fusion, {}, {} };
    r.mega = r.fuse && ((flags & B200_EXEC_MEGAKERNEL) || ex->env_mega) && !ex->env_no_mega;
    r.mega_mmv = r.mega && ((flags & B200_EXEC_MEGA_MMV) || ex->env_mega_mmv);

    // CUDA graphs only pay for small-batch (decode / verify) lists; prefill lists are few big kernels
    bool small = true;
    for (int i = 0; i < n_nodes && small; i++) if (nodes[i].op == B200_OP_MUL_MAT && nodes[i].src[1].ne[1] > 8) small = false;
    // the legacy default stream cannot be captured
    const bool use_graph = (flags & B200_EXEC_CUDA_GRAPHS) && !ex->env_no_graphs && small && n_nodes >= 8 && st != nullptr && st != cudaStreamLegacy;
    if (!use_graph) {
        const int64_t l0 = b200_kernel_launches();
        s = r.run_all();
        ex->last_kernels = b200_kernel_launches() - l0;
        return s;
    }
    const uint64_t key = topology_key(nodes, n_nodes, flags);
    ex->tick++;
    auto it = ex->graphs.find(key);
    if (it == ex->graphs.end() && ex->seen[key]++ == 0) {
        // first sighting: run eagerly (also warms per-function attributes outside of capture), like the
        // reference's warm-up evaluation (ggml-cuda.cu:2964-2976)
        if (ex->seen.size() > 4096) ex->seen.clear();
        const int64_t l0 = b200_kernel_launches();
        s = r.run_all();
        ex->last_kernels = b200_kernel_launches() - l0;
        return s;
    }
    if (it == ex->graphs.end()) {
        if (ex->graphs.size() >= 64) {                      // evict the least recently used entry
            auto lru = ex->graphs.begin();
            for (auto g = ex->graphs.begin(); g != ex->graphs.end(); ++g) if (g->second.last_use < lru->second.last_use) lru = g;
            if (lru->second.exec) cudaGraphExecDestroy(lru->second.exec);
            ex->graphs.erase(lru);
        }
        cudaGraph_t graph = nullptr;
        B200_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed));
        const int64_t l0 = b200_kernel_launches();
        s = r.run_all();
        const int64_t kernels = b200_kernel_launches() - l0;
        b200_count_launch(-(int)kernels);                    // recorded, not run: counted at launch below
        cudaError_t e = cudaStreamEndCapture(st, &graph);
        if (s != B200_OK) { if (graph) cudaGraphDestroy(graph); return s; }
        B200_CUDA(e);
        GraphEntry ge; ge.kernels = kernels;
        e = cudaGraphInstantiate(&ge.exec, graph, 0);
        cudaGraphDestroy(graph);
        B200_CUDA(e);
        ex->captures++;
        it = ex->graphs.emplace(key, ge).first;
    } else {
        ex->replays++;
    }
    it->second.last_use = ex->tick;
    ex->last_kernels = it->second.kernels;
    b200_count_launch((int)it->second.kernels);
    B200_CUDA(cudaGraphLaunch(it->second.exec, st));
    return B200_OK;
}

extern "C" int64_t b200_executor_plan(const b200_node * nodes, int n_nodes, int flags) {
    if ((!nodes && n_nodes > 0) || n_nodes < 0) { b200_set_error("executor_plan: bad arguments"); return B200_ERR_INVALID; }
    for (int i = 0; i < n_nodes; i++) if (!node_ok(nodes[i])) { b200_set_error("executor_plan: node %d (op %d) is not supported", i, nodes[i].op); return B200_ERR_UNSUPPORTED; }
    b200_executor tmp;                                   // never touches a device
    Runner r{ &tmp, nodes, n_nodes, nullptr, (flags & B200_EXEC_FUSION) != 0, {}, {} };
    r.mega = r.fuse && (flags & B200_EXEC_MEGAKERNEL); r.mega_mmv = r.mega && (flags & B200_EXEC_MEGA_MMV);
    r.dry = true;
    const int s = r.run_all();
    return s == B200_OK ? r.planned : (int64_t)s;
}

extern "C" int64_t b200_executor_last_kernels(const b200_executor * ex)  { return ex ? ex->last_kernels : 0; }
extern "C" int64_t b200_executor_graph_captures(const b200_executor * ex) { return ex ? ex->captures : 0; }
extern "C" int64_t b200_executor_graph_replays(const b200_executor * ex)  { return ex ? ex->replays : 0; }
extern "C" int64_t b200_executor_mk_launches(const b200_executor * ex)     { return ex ? ex->mk_launches : 0; }
extern "C" int64_t b200_executor_mk_phases(const b200_executor * ex)       { return ex ? ex->mk_phases : 0; }
