// mmq_quant.cuh — activation quantisation into the B image of the tensor-core MUL_MAT (mmq_tc.cu), dense or gathered by expert
// (grouped MUL_MAT_ID).  Kept in a header so that tests/hostsim/kernsim.cpp runs the same source under the SIMT emulation
// (tests/test_moe_route_simt.py compares the gathered image with the dense one).
#pragma once
#include "common.cuh"
#include "moe_route.cuh"

#define TC_TN 128
#define TC_PANEL 2048             // one K-chunk (8 f16 = 16 bytes) of 128 rows

// ---- workspace geometry (the B image) ------------------------------------------------------------------------------
// per 128-token tile nt: Bq[nt][kq = k/64][chunk 0..7][n 0..127][8 f16]   (16 KB per 64-k quarter)
//                        Bm[nt][sb][chunk 0..1][n][8 f16]                  (q8_K bsums, 4 KB per super-block)
//                        D8[nt][sb][n] f32                                 (512 B per super-block)
struct TcGeom { int64_t nt, kq, nsb, off_bq, off_bm, off_d8, total; };
static inline TcGeom tc_geom(int64_t k, int64_t ncols) {
    TcGeom g;
    g.nt = (ncols + TC_TN - 1) / TC_TN; g.kq = k / 64; g.nsb = k / 256;
    g.off_bq = 0;
    g.off_bm = g.nt * g.kq * 16384;
    g.off_d8 = g.off_bm + g.nt * g.nsb * 4096;
    g.total  = g.off_d8 + g.nt * g.nsb * 512;
    return g;
}

// column gather of the grouped MUL_MAT_ID: column c of group tile g is pair perm[tiles[g].first + c] = (t, s), read from
// x + t * x_col_stride + (s % n_b1) * slot_stride; tiles >= *n_gtiles are not written, columns past tiles[g].count are zeros
struct TcGather { const int32_t * perm; const MoeTile * tiles; const int32_t * n_gtiles; int64_t slot_stride; int32_t n_b1, _pad; };

// one warp per (token, super-block); exactly quantize_row_q8_K_ref: first index of the largest |x|, iscale = -127/max,
// nearest-int (RNE), MIN(127, .), d = 1/iscale, bsums per 16
template <bool GATHER>
__global__ void __launch_bounds__(256) quantize_mmq_kernel(const float * __restrict__ x, int64_t x_col_stride, int64_t ncols, int64_t k,
                                                          uint8_t * __restrict__ ws, TcGeom g, TcGather ga) {
    pdl_wait();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t sb = blockIdx.x;
    const int64_t n = (int64_t)blockIdx.y * 8 + warp;                // token (padded range: < nt * 128)
    const int64_t nt = n >> 7; const int nl = (int)(n & 127);
    float v[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
    if (GATHER) {
        if (nt >= *ga.n_gtiles) return;                               // uniform over the CTA (its 8 columns lie in one tile)
        const MoeTile tl = ga.tiles[nt];
        if (nl < tl.count) {
            const int32_t pr = ga.perm[tl.first + nl];
            const float4 * p = (const float4 *)(x + (int64_t)(pr >> 16) * x_col_stride + (int64_t)((pr & 0xffff) % ga.n_b1) * ga.slot_stride + sb * 256 + lane * 8);
            const float4 a = p[0], b = p[1];
            v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
        }
    } else if (n < ncols) {
        const float4 * p = (const float4 *)(x + n * x_col_stride + sb * 256 + lane * 8);
        const float4 a = p[0], b = p[1];
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
    float am = 0.0f; int ai = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) { const float a = fabsf(v[j]); if (a > am) { am = a; ai = lane * 8 + j; } }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float am2 = __shfl_xor_sync(0xffffffffu, am, o);
        const int   ai2 = __shfl_xor_sync(0xffffffffu, ai, o);
        if (am2 > am || (am2 == am && ai2 < ai)) { am = am2; ai = ai2; }
    }
    float mine = 0.0f;
#pragma unroll
    for (int j = 0; j < 8; j++) if ((ai & 7) == j) mine = v[j];
    const float maxv = __shfl_sync(0xffffffffu, mine, ai >> 3);
    int q[8]; int s = 0; float d = 0.0f;
    if (am != 0.0f) {
        const float iscale = __fdiv_rn(-127.0f, maxv);
#pragma unroll
        for (int j = 0; j < 8; j++) { const int t = __float2int_rn(__fmul_rn(iscale, v[j])); q[j] = t > 127 ? 127 : t; s += q[j]; }
        d = __fdiv_rn(1.0f, iscale);
    } else {
#pragma unroll
        for (int j = 0; j < 8; j++) q[j] = 0;
    }
    // 8 consecutive elements = one K-chunk of the panel; element order inside a chunk is (0,2,1,3,4,6,5,7): the order in
    // which the weight transform extracts nibbles from a 32-bit word (see unpack in the GEMM kernel)
    auto h2 = [](int a, int b) { return (uint32_t)__half_as_ushort(__int2half_rn(a)) | ((uint32_t)__half_as_ushort(__int2half_rn(b)) << 16); };
    uint4 pk; pk.x = h2(q[0], q[2]); pk.y = h2(q[1], q[3]); pk.z = h2(q[4], q[6]); pk.w = h2(q[5], q[7]);
    const int64_t kq = sb * 4 + (lane >> 3); const int c = lane & 7;
    *(uint4 *)(ws + g.off_bq + ((nt * g.kq + kq) * 8 + c) * TC_PANEL + nl * 16) = pk;
    s += __shfl_xor_sync(0xffffffffu, s, 1);                          // bsum of 16 elements (|.| <= 2032: exact in f16)
    if ((lane & 1) == 0) {
        const int grp = lane >> 1;
        *(__half *)(ws + g.off_bm + ((nt * g.nsb + sb) * 2 + (grp >> 3)) * TC_PANEL + nl * 16 + (grp & 7) * 2) = __int2half_rn(s);
    }
    if (lane == 0) *(float *)(ws + g.off_d8 + ((nt * g.nsb + sb) * 128 + nl) * 4) = d;
    pdl_trigger();
}
