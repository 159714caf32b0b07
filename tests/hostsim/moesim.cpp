// moesim.cpp — TEST INFRASTRUCTURE.  Runs the SOURCE of the grouped MUL_MAT_ID's device code — the routing kernel (moe_route.cuh) and the
// dense / gathered activation quantiser of the tensor-core MUL_MAT (mmq_quant.cuh) — on the CPU under tests/hostsim/simt.h, host pointers
// instead of device pointers.  Launch geometry as in mmq_tc.cu (b200_mmq_tc / b200_mmq_tc_id).  Loaded by tests/test_moe_prefill_simt.py.
#include "simt.h"

#include "../../llama-box_b200/csrc/mmq_quant.cuh"

extern "C" {
int sim_moe_max_tiles(int64_t n_expert, int64_t n_pairs) { return (int)moe_max_tiles(n_expert, n_pairs); }
void sim_moe_route(const int32_t * ids, int64_t ids_tok_stride, int n_expert, int n_used, int n_tok, int32_t * perm, void * tiles, int32_t * n_gtiles) {
    simt::launch(dim3(1), dim3(MR_THREADS), 0, [=] { moe_route_kernel(ids, ids_tok_stride, n_expert, n_used, n_tok, perm, (MoeTile *)tiles, n_gtiles); });
}
// B image of ncols dense columns (x + c * x_col_stride)
void sim_quantize_mmq(const float * x, int64_t x_col_stride, int64_t ncols, int64_t k, void * ws) {
    const TcGeom g = tc_geom(k, ncols);
    simt::launch(dim3((unsigned)(k / 256), (unsigned)(g.nt * 16)), dim3(256), 0, [=] { quantize_mmq_kernel<false>(x, x_col_stride, ncols, k, (uint8_t *)ws, g, TcGather{}); });
}
// B image of g_max group tiles gathered through perm / tiles (b laid out as b200_mul_mat_id's b)
void sim_quantize_mmq_gather(const float * b, int64_t b_tok_stride, int64_t b_slot_stride, int64_t n_b1, int64_t k, const int32_t * perm, const void * tiles,
                             const int32_t * n_gtiles, int64_t g_max, void * ws) {
    const TcGeom g = tc_geom(k, g_max * 128);
    TcGather ga = {}; ga.perm = perm; ga.tiles = (const MoeTile *)tiles; ga.n_gtiles = n_gtiles; ga.slot_stride = b_slot_stride; ga.n_b1 = (int32_t)n_b1;
    simt::launch(dim3((unsigned)(k / 256), (unsigned)(g_max * 16)), dim3(256), 0, [=] { quantize_mmq_kernel<true>(b, b_tok_stride, 0, k, (uint8_t *)ws, g, ga); });
}
}
