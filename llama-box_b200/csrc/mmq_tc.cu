// mmq_tc.cu — batched MUL_MAT on K-quant weights (prefill / large ubatches) on the 5th-generation tensor cores (sm_100a):
// tcgen05.mma with TMEM accumulators, TMA (cp.async.bulk) staging, warp-specialised, persistent.
//
// Replaces ggml_cuda_mul_mat_q / mul_mat_q<type,mmq_x> (ggml-cuda/mmq.cu:71-143, mmq.cuh:3047-3370: int8 mma.sync tiles
// with per-32 f32 scale FMAs in the inner loop, stream-K fixup :3373-3522) and quantize_mmq_q8_1 (quantize.cu:50-146).
// The arithmetic is the CPU ORACLE's, not ggml-cuda's: activations are quantised to q8_K exactly like
// quantize_row_q8_K_ref (ggml-quants.c:2555-2592) and the per-super-block integer sums of ggml_vec_dot_q{4,5,6}_K_q8_K
// (ggml-cpu/quants.c:550-758) are reproduced EXACTLY by the tensor cores:
//
//     dst[n][r] = sum_sb  d_w[r,sb] * d_x[n,sb] * isum[r,n,sb]  -  dmin_w[r,sb] * d_x[n,sb] * imin[r,n,sb]
//     isum = sum_j sc_j * (sum_{k in sub-block j} q_k * q8_k)          imin = sum_j m_j * bsum_j
//
//   * A operand (weights): a transform warpgroup unpacks the packed quants from shared memory into f16 INTEGERS with the
//     6-bit sub-block scale folded in, a[r][k] = sc_j * q  (<= 63*15 = 945 for Q4_K, <= 63*31 = 1953 for Q5_K: exact in f16),
//     written as UMMA K-major core matrices.  Q6_K's sc * (q - 32) reaches +-4096, which f16 holds only when even: the
//     product is split as (sc & ~1) * (q - 32)  [even, exact]  +  (sc & 1) * (q - 32)  [|.| <= 32], two K-passes into ONE
//     accumulator.
//   * B operand (activations): q8 values as f16 integers (|q8| <= 127), pre-tiled in HBM in the exact shared-memory image so
//     that one bulk copy brings a [128 tokens x 64 k] panel.
//   * tcgen05.mma kind::f16, M = 128, N <= 128, K = 16 per instruction, f32 accumulate in TMEM: every product and every
//     partial sum is an integer below 2^24, so the accumulation is EXACT and isum equals the oracle's int32 bit for bit.
//     imin is one more K = 16 MMA per super-block (A = m_j as f16, B = the q8_K bsums as f16) into its own TMEM columns.
//   * epilogue warps drain TMEM once per super-block (tcgen05.ld), apply d_w * d_x and dmin_w * d_x in f32 — the only
//     floating-point rounding on the path, the same two roundings per super-block the oracle performs — and keep the f32
//     running sums in registers.  TMEM is double-buffered (2 x (isum 128 cols + imin 128 cols) = all 512 columns), so the
//     drain of super-block s overlaps the MMAs of s + 1.
//
// Warp roles (448 threads, one persistent CTA per SM):
//     warps 0-3 / 4-7  epilogue, columns 0-63 / 64-127 (warp % 4 = TMEM lane quadrant)
//     warps 8-11       transform: thread t owns weight row t of the tile; packed blocks come straight from global memory into
//                      registers, one super-block ahead
//     warp 12          TMA producer: the activation panels of each stage (cp.async.bulk, mbarrier complete_tx)
//     warp 13          TMEM allocation + the single MMA-issuing thread
// Shared memory (per CTA): 2 A stages x 32 KB (128 rows x 128 k f16) + 2 B stages x 32 KB + raw weight blocks x 2 + the
// imin operands + scale rings, ~200 KB.  Data movement: weights are read from HBM once per 128-token tile (L2 serves the
// other token tiles of the same rows, which run on neighbouring CTAs), activations stream from L2.
#include "common.cuh"
#include "mmq_quant.cuh"          // TcGeom / tc_geom, quantize_mmq_kernel (the B image), MoeTile

#include <cuda_fp16.h>
#include <cstdio>
#include <cstdlib>

#define TC_TM 128
#define TC_THREADS 448
#define TC_STAGE_A 32768
#define TC_STAGE_B 32768

// ---- tcgen05 / TMEM primitives (inline PTX; SASS: UTCHMMA, LDTM, UTCBAR, ...) -------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after()  { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t * bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t * bar) {          // arrives on `bar` when every MMA issued so far by this thread has completed
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(bar)) : "memory");
}
// shared-memory matrix descriptor, K-major, no swizzle ("interleaved" core matrices of 8 rows x 16 bytes):
//   element (row r, 16-byte K-chunk c) lives at  start + c * LBO + (r / 8) * SBO + (r % 8) * 16
// (cute::UMMA::SmemDescriptor, canonical layout ((8,n),2):((1,SBO),LBO) in 16-byte units; bits 46-47 = 1 on sm_100)
__device__ __forceinline__ uint64_t tc_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
}
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

struct TcArgs {
    const uint8_t * W;          // weights, `type` rows (Q6_K: repacked rows, see repack.cu)
    const uint8_t * ws;         // B image (quantize_mmq_kernel)
    float *         dst;        // [ncols][ldd] f32
    int64_t m, k, ncols, ldd, rb;
    TcGeom g;
    int32_t nsb, n_mtiles, n_tiles, type;
    uint32_t lbo, sbo;          // descriptor strides (bytes): K-chunk stride / 8-row-group stride
    unsigned long long * prof;  // bring-up: per-role cycle counters of CTA 0 (B200_MMQ_PROF), normally null
    // grouped instances (MUL_MAT_ID) only: the routing of moe_route_kernel; column c of group tile g is pair
    // gperm[gtiles[g].first + c] = (t, s), weights of expert gtiles[g].expert at W + expert * expert_stride
    const MoeTile * gtiles; const int32_t * gperm; const int32_t * n_gtiles;
    int64_t expert_stride, dst_tok_stride, dst_slot_stride;
};
// wait on an mbarrier, optionally accounting the cycles to a profile counter
__device__ __forceinline__ void mbar_wait_p(uint64_t * bar, uint32_t parity, unsigned long long * acc) {
    if (acc) { const long long t0 = clock64(); mbar_wait(bar, parity); *acc += (unsigned long long)(clock64() - t0); }
    else mbar_wait(bar, parity);
}

// ---- per-type geometry of the raw (packed) weight blocks staged in shared memory ------------------------------------
template <int T> struct TcType;
// RAW_SLOTS: depth of the packed-weight ring.  The raw producer warp runs ahead of everything else (its only dependency is
// the transform having consumed a slot), so that HBM latency of the weight stream is hidden behind RAW_SLOTS - 1 super-blocks
template <> struct TcType<B200_TYPE_Q4_K> { static constexpr int STAGES = 2, RAW = 128 * 144, HAS_MIN = 1, B_BYTES = 32768, RAW_SLOTS = 4; };
template <> struct TcType<B200_TYPE_Q5_K> { static constexpr int STAGES = 2, RAW = 128 * 176, HAS_MIN = 1, B_BYTES = 32768, RAW_SLOTS = 3; };
// Q6_K rows are repacked [ql 128B x nb][qh 64B x nb][scales 16B x nb][d f16 x nb]; staged with padded row strides
// (144 / 80 / 16 bytes) so that thread-per-row 16-byte reads are bank-conflict free; d is fetched 8 super-blocks at a time
template <> struct TcType<B200_TYPE_Q6_K> { static constexpr int STAGES = 4, RAW = 128 * (144 + 80 + 16), HAS_MIN = 0, B_BYTES = 16384, RAW_SLOTS = 2; };

// shared memory map
struct TcSmem {
    static constexpr int A = 0, B = A + 2 * TC_STAGE_A, AM = B + 2 * TC_STAGE_B, BM = AM + 2 * 4096, RAWO = BM + 2 * 4096;
    static constexpr int RAW_BYTES = 73728;                  // ring of packed weight blocks: 4 x 18 KB (Q4_K), 3 x 22 KB (Q5_K), 2 x 30 KB (Q6_K)
    static constexpr int DC = RAWO + RAW_BYTES;              // Q6_K d cache: 2 x 128 rows x 16 B
    static constexpr int RS = DC + 2 * 2048;                 // row scales ring: 4 x 128 x float2
    static constexpr int D8 = RS + 4 * 1024;                 // d_x ring: 4 x 128 f32
    static constexpr int BAR = D8 + 4 * 512;                 // mbarriers
    static constexpr int TOTAL = BAR + 256;
};

__device__ __forceinline__ uint32_t hfma2_u(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d; asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d;
}
__device__ __forceinline__ uint32_t hmul2_u(uint32_t a, uint32_t b) { uint32_t d; asm("mul.rn.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b)); return d; }
__device__ __forceinline__ uint32_t hsub2_u(uint32_t a, uint32_t b) { uint32_t d; asm("sub.rn.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b)); return d; }
__device__ __forceinline__ uint32_t h2_of_int(int v) { const uint32_t h = __half_as_ushort(__int2half_rn(v)); return h | (h << 16); }

// 6-bit scales / mins of a q4_K / q5_K block header (ggml-quants.c:703-711), all 8 at once
__device__ __forceinline__ void k4_unpack(uint32_t y, uint32_t z, uint32_t w, uint32_t & sc03, uint32_t & sc47, uint32_t & mn03, uint32_t & mn47) {
    sc03 = y & 0x3f3f3f3fu; mn03 = z & 0x3f3f3f3fu;
    sc47 = (w & 0x0f0f0f0fu) | (((y >> 6) & 0x03030303u) << 4);
    mn47 = ((w >> 4) & 0x0f0f0f0fu) | (((z >> 6) & 0x03030303u) << 4);
}

// GROUPED: work items are (m-tile, group tile) with the group-tile count read from device memory (*args.n_gtiles); items of one
// (expert, m-tile) are adjacent, so concurrently running CTAs share weight rows through L2
template <int T, bool GROUPED>
__global__ void __launch_bounds__(TC_THREADS, 1) mmq_tc_kernel(const __grid_constant__ TcArgs args) {
    using TT = TcType<T>;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t * bars = (uint64_t *)(smem + TcSmem::BAR);
    uint64_t * raw_full = bars, * raw_empty = bars + 4, * b_full = bars + 8, * a_full = bars + 10, * ab_empty = bars + 12, * acc_full = bars + 14, * acc_empty = bars + 16;
    uint32_t * tmem_slot = (uint32_t *)(bars + 18);
    constexpr int RSL = TT::RAW_SLOTS;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    if (tid == 0) {
        for (int i = 0; i < 4; i++) { mbar_init(&raw_full[i], 1); mbar_init(&raw_empty[i], 4); }
        for (int i = 0; i < 2; i++) {
            mbar_init(&b_full[i], 1); mbar_init(&a_full[i], 4);
            mbar_init(&ab_empty[i], 1); mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 8);
        }
        mbar_fence_init();
    }
    if (warp == 13) {                                              // TMEM: all 512 columns (one CTA per SM)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    pdl_wait();

    const int nsb = args.nsb;
    const int64_t NT = GROUPED ? (int64_t)*args.n_gtiles : args.g.nt;   // N tiles: group tiles are written by the routing kernel before this grid
    const int n_tiles = GROUPED ? args.n_mtiles * (int)NT : args.n_tiles;
    unsigned long long w0 = 0, w1 = 0, w2 = 0;                       // profile: cycles in this role's three kinds of waits
    const bool prof = args.prof != nullptr && blockIdx.x == 0;
    unsigned long long * pw0 = prof ? &w0 : nullptr, * pw1 = prof ? &w1 : nullptr, * pw2 = prof ? &w2 : nullptr;
    const long long t_start = clock64();

    if (warp == 12) {
        // ===================== TMA producer: activation panels, one per stage (+ the bsum panel and d_x with the first) =====================
        uint32_t it = 0, sbc = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int64_t nt = tile % NT;
            for (int sb = 0; sb < nsb; sb++, sbc++) {
                const int rs = sbc & 1;
                for (int s = 0; s < TT::STAGES; s++, it++) {
                    const int st = it & 1;
                    mbar_wait_p(&ab_empty[st], ((it >> 1) & 1) ^ 1, pw0);
                    if (lane == 0) {
                        const uint32_t extra = s == 0 ? (512u + (TT::HAS_MIN ? 4096u : 0u)) : 0u;
                        mbar_expect_tx(&b_full[st], (uint32_t)TT::B_BYTES + extra);
                        const int64_t kq0 = (int64_t)sb * 4 + (TT::STAGES == 2 ? s * 2 : s);
                        const uint8_t * src = args.ws + args.g.off_bq + (nt * args.g.kq + kq0) * 16384;
                        uint8_t * dstb = smem + TcSmem::B + st * TC_STAGE_B;
                        for (int o = 0; o < TT::B_BYTES; o += 8192) bulk_g2s(dstb + o, src + o, 8192, &b_full[st]);
                        if (s == 0) {
                            if (TT::HAS_MIN) bulk_g2s(smem + TcSmem::BM + rs * 4096, args.ws + args.g.off_bm + (nt * nsb + sb) * 4096, 4096, &b_full[st]);
                            bulk_g2s(smem + TcSmem::D8 + (sbc & 3) * 512, args.ws + args.g.off_d8 + (nt * nsb + sb) * 512, 512, &b_full[st]);
                        }
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp == 13) {
        // ===================== MMA issuer (one thread) =====================
        if (lane == 0) {
            uint32_t it = 0, sbc = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const int64_t nt = tile % NT;
                const int64_t nval = GROUPED ? (int64_t)args.gtiles[nt].count : (args.ncols - nt * TC_TN < TC_TN ? args.ncols - nt * TC_TN : TC_TN);
                const uint32_t n_eff = (uint32_t)((nval + 15) & ~15);
                // instruction descriptor (cute::UMMA::InstrDescriptor): D = f32, A = B = f16, both K-major, N >> 3 at bit 17, M >> 4 at bit 24
                const uint32_t idesc = (1u << 4) | ((n_eff >> 3) << 17) | ((uint32_t)(TC_TM >> 4) << 24);
                for (int sb = 0; sb < nsb; sb++, sbc++) {
                    const int rs = sbc & 1;
                    mbar_wait_p(&acc_empty[rs], ((sbc >> 1) & 1) ^ 1, pw0);       // epilogue has drained this TMEM buffer
                    tc_fence_after();
                    const uint32_t d_main = tmem + rs * 128, d_min = tmem + 256 + rs * 128;
                    for (int s = 0; s < TT::STAGES; s++, it++) {
                        const int st = it & 1; const uint32_t ph = (it >> 1) & 1;
                        mbar_wait_p(&b_full[st], ph, pw1);
                        mbar_wait_p(&a_full[st], ph, pw2);
                        tc_fence_after();
                        const uint32_t a0 = smem_u32(smem + TcSmem::A + st * TC_STAGE_A), b0 = smem_u32(smem + TcSmem::B + st * TC_STAGE_B);
#pragma unroll
                        for (int j = 0; j < 8; j++) {
                            const uint32_t bj = TT::STAGES == 2 ? j : (j & 3);    // Q6_K: the even and the odd-scale pass read the same 64-k panel
                            tc_mma_f16(d_main, tc_desc(a0 + j * 2 * TC_PANEL, args.lbo, args.sbo), tc_desc(b0 + bj * 2 * TC_PANEL, args.lbo, args.sbo), idesc, (s | j) ? 1u : 0u);
                        }
                        if (TT::HAS_MIN && s == TT::STAGES - 1)
                            tc_mma_f16(d_min, tc_desc(smem_u32(smem + TcSmem::AM + rs * 4096), args.lbo, args.sbo), tc_desc(smem_u32(smem + TcSmem::BM + rs * 4096), args.lbo, args.sbo), idesc, 0u);
                        tc_commit(&ab_empty[st]);                          // stage buffers reusable once these MMAs have completed
                    }
                    tc_commit(&acc_full[rs]);                              // accumulators of this super-block complete
                }
            }
        }
        __syncwarp();
    } else if (warp >= 8 && warp < 12) {
        // ===================== transform: packed quants -> f16 sc*q core matrices =====================
        // Thread t owns weight row t of the tile and reads its packed block of the NEXT super-block straight from global memory
        // into registers (9-14 16-byte loads, issued one super-block ahead, so HBM / L2 latency hides behind the conversion of
        // the current one).  (A first version staged the blocks through shared memory with one cp.async.bulk per row: a
        // warp-wide bulk copy is issued lane by lane through uniform registers, ~65 cycles each — 128 rows cost 8 K cycles per
        // super-block and starved everything else; profiles/README.md.)
        constexpr int NW = T == B200_TYPE_Q4_K ? 9 : (T == B200_TYPE_Q5_K ? 11 : 13);
        const int t = tid - 8 * 32;                                      // weight row of the tile
        const int64_t nb = args.k / 256;
        uint32_t it = 0, sbc = 0;
        uint4 nxt[NW]; uint16_t nxt_d = 0;
        auto fetch = [&](int tile, int sb) {
            const int64_t m0 = (int64_t)(tile / NT) * TC_TM;
            int64_t r = m0 + t; if (r >= args.m) r = args.m - 1;             // rows past the end: any valid row (their results are never stored)
            const uint8_t * W = GROUPED ? args.W + (int64_t)args.gtiles[tile % NT].expert * args.expert_stride : args.W;
            const uint8_t * row = W + r * args.rb;
            if (T == B200_TYPE_Q6_K) {
                const uint4 * ql = (const uint4 *)(row + (int64_t)sb * 128), * qh = (const uint4 *)(row + nb * 128 + (int64_t)sb * 64);
#pragma unroll
                for (int i = 0; i < 8; i++) nxt[i] = __ldg(ql + i);
#pragma unroll
                for (int i = 0; i < 4; i++) nxt[8 + i] = __ldg(qh + i);
                nxt[12] = __ldg((const uint4 *)(row + nb * 192 + (int64_t)sb * 16));
                nxt_d = __ldg((const uint16_t *)(row + nb * 208 + (int64_t)sb * 2));
            } else {
                const uint4 * p = (const uint4 *)(row + (int64_t)sb * (T == B200_TYPE_Q4_K ? 144 : 176));
#pragma unroll
                for (int i = 0; i < NW; i++) nxt[i] = __ldg(p + i);
            }
        };
        if (blockIdx.x < n_tiles) fetch(blockIdx.x, 0);
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            for (int sb = 0; sb < nsb; sb++, sbc++) {
                const int rs = sbc & 1;                                  // accumulator / imin-operand slot
                uint4 cur[NW]; const uint16_t cur_d = nxt_d;
#pragma unroll
                for (int i = 0; i < NW; i++) cur[i] = nxt[i];
                {   // prefetch the next super-block (of this tile, or the first one of this CTA's next tile)
                    int ntile = tile, nsbi = sb + 1;
                    if (nsbi == nsb) { nsbi = 0; ntile = tile + gridDim.x; }
                    if (ntile < n_tiles) fetch(ntile, nsbi);
                }
                float2 * rscale = (float2 *)(smem + TcSmem::RS + (sbc & 3) * 1024);
                if (T == B200_TYPE_Q4_K || T == B200_TYPE_Q5_K) {
                    constexpr int QW = T == B200_TYPE_Q4_K ? 1 : 3;       // first 16-byte word of qs
                    const uint4 hdr = cur[0];
                    uint32_t sc03, sc47, mn03, mn47;
                    k4_unpack(hdr.y, hdr.z, hdr.w, sc03, sc47, mn03, mn47);
                    uint32_t qhw[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
                    if (T == B200_TYPE_Q5_K) { qhw[0] = cur[1].x; qhw[1] = cur[1].y; qhw[2] = cur[1].z; qhw[3] = cur[1].w; qhw[4] = cur[2].x; qhw[5] = cur[2].y; qhw[6] = cur[2].z; qhw[7] = cur[2].w; }
#pragma unroll
                    for (int s = 0; s < 2; s++, it++) {                   // half super-block = 128 k = one stage
                        const int st = it & 1;
                        mbar_wait_p(&ab_empty[st], ((it >> 1) & 1) ^ 1, pw1);
                        uint8_t * As = smem + TcSmem::A + st * TC_STAGE_A + t * 16;
#pragma unroll
                        for (int gg = 0; gg < 2; gg++) {
                            const int grp = 2 * s + gg;                   // 64-element group: low nibbles = sub-block 2grp, high = 2grp + 1
                            const uint32_t scw = grp < 2 ? sc03 : sc47;
                            const int sc_lo = (scw >> (16 * (grp & 1))) & 63, sc_hi = (scw >> (16 * (grp & 1) + 8)) & 63;
                            const uint32_t m_lo = h2_of_int(sc_lo), m_hi = h2_of_int(sc_hi);
                            const uint32_t c_lo = h2_of_int(-1024 * sc_lo), c_hi = h2_of_int(-64 * sc_hi);
                            const uint4 qa = cur[QW + grp * 2], qb = cur[QW + grp * 2 + 1];
                            const uint32_t w[8] = { qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w };
#pragma unroll
                            for (int i = 0; i < 4; i++) {
                                uint4 lo, hi;
                                uint32_t * plo = (uint32_t *)&lo, * phi = (uint32_t *)&hi;
#pragma unroll
                                for (int u = 0; u < 2; u++) {
                                    const uint32_t ww = w[2 * i + u];
                                    uint32_t l0 = (ww & 0x000F000Fu) | 0x64006400u, l1 = ((ww >> 8) & 0x000F000Fu) | 0x64006400u;      // 1024 + q  (elements e, e+2 | e+1, e+3)
                                    uint32_t h0 = (ww & 0x00F000F0u) | 0x54005400u, h1 = ((ww >> 8) & 0x00F000F0u) | 0x54005400u;      // 64 + q    (high nibbles, elements + 32)
                                    if (T == B200_TYPE_Q5_K) {                                                                         // fifth bit: bit (sub-block) of qh[l]
                                        const uint32_t hw = qhw[2 * i + u];
                                        l0 |= ((hw >> (2 * grp)) & 0x00010001u) << 4;      l1 |= ((hw >> (2 * grp + 8)) & 0x00010001u) << 4;
                                        h0 |= ((hw >> (2 * grp + 1)) & 0x00010001u) << 8;  h1 |= ((hw >> (2 * grp + 9)) & 0x00010001u) << 8;
                                    }
                                    plo[2 * u] = hfma2_u(l0, m_lo, c_lo); plo[2 * u + 1] = hfma2_u(l1, m_lo, c_lo);     // exact: sc * q
                                    phi[2 * u] = hfma2_u(h0, m_hi, c_hi); phi[2 * u + 1] = hfma2_u(h1, m_hi, c_hi);
                                }
                                *(uint4 *)(As + (gg * 8 + i) * TC_PANEL) = lo;
                                *(uint4 *)(As + (gg * 8 + 4 + i) * TC_PANEL) = hi;
                            }
                        }
                        if (s == 0) {
                            // imin operand: m_j duplicated for its two 16-element halves; d, dmin for the epilogue
                            uint8_t * Am = smem + TcSmem::AM + rs * 4096 + t * 16;
                            uint4 m0, m1;
                            m0.x = h2_of_int(mn03 & 63); m0.y = h2_of_int((mn03 >> 8) & 63); m0.z = h2_of_int((mn03 >> 16) & 63); m0.w = h2_of_int((mn03 >> 24) & 63);
                            m1.x = h2_of_int(mn47 & 63); m1.y = h2_of_int((mn47 >> 8) & 63); m1.z = h2_of_int((mn47 >> 16) & 63); m1.w = h2_of_int((mn47 >> 24) & 63);
                            *(uint4 *)Am = m0; *(uint4 *)(Am + TC_PANEL) = m1;
                            rscale[t] = make_float2(h2f((uint16_t)(hdr.x & 0xffff)), h2f((uint16_t)(hdr.x >> 16)));
                        }
                        fence_async_smem();                               // generic-proxy writes -> visible to the tensor core (async proxy)
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&a_full[st]);
                    }
                } else {
                    // ---- Q6_K: q = ql | qh << 4 (0..63), value sc * (q - 32), scales int8 per 16 elements (ggml-quants.c dequantize_row_q6_K)
                    const uint32_t scw[4] = { cur[12].x, cur[12].y, cur[12].z, cur[12].w };
#pragma unroll
                    for (int s = 0; s < 4; s++, it++) {                   // quarter super-block = 64 k: chunks 0-7 = even-scale part, 8-15 = odd-scale part
                        const int st = it & 1;
                        mbar_wait_p(&ab_empty[st], ((it >> 1) & 1) ^ 1, pw1);
                        uint8_t * As = smem + TcSmem::A + st * TC_STAGE_A + t * 16;
                        const int hh = s >> 1, u2 = s & 1;
                        const uint4 qha = cur[8 + hh * 2], qhb = cur[8 + hh * 2 + 1];
                        const uint32_t qhw[8] = { qha.x, qha.y, qha.z, qha.w, qhb.x, qhb.y, qhb.z, qhb.w };
#pragma unroll
                        for (int tt = 0; tt < 2; tt++) {
                            const int tg = 2 * u2 + tt;                   // 32-element group of the half: elements 128 hh + 32 tg + l
                            const uint4 qa = cur[hh * 4 + (tg & 1) * 2], qb = cur[hh * 4 + (tg & 1) * 2 + 1];
                            const uint32_t w[8] = { qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w };
                            const int nsh = 4 * (tg >> 1), hsh = 2 * tg;
#pragma unroll
                            for (int i = 0; i < 4; i++) {
                                const int sidx = 8 * hh + 2 * tg + (i >> 1);                          // scale of elements 8i .. 8i+7 of the group
                                const int sc = (int)(int8_t)((scw[sidx >> 2] >> (8 * (sidx & 3))) & 0xff);
                                const int sce = sc & ~1;
                                const uint32_t m_e = h2_of_int(sce), m_o = h2_of_int(sc - sce);
                                uint4 ev, od;
                                uint32_t * pe = (uint32_t *)&ev, * po = (uint32_t *)&od;
#pragma unroll
                                for (int u = 0; u < 2; u++) {
                                    const uint32_t q4 = ((w[2 * i + u] >> nsh) & 0x0F0F0F0Fu) | (((qhw[2 * i + u] >> hsh) & 0x03030303u) << 4);
                                    const uint32_t x0 = hsub2_u((q4 & 0x00FF00FFu) | 0x64006400u, 0x64206420u);       // (1024 + q) - 1056 = q - 32, elements (e, e+2)
                                    const uint32_t x1 = hsub2_u(((q4 >> 8) & 0x00FF00FFu) | 0x64006400u, 0x64206420u); // elements (e+1, e+3)
                                    pe[2 * u] = hmul2_u(x0, m_e); pe[2 * u + 1] = hmul2_u(x1, m_e);                  // even scale part: exact (even integers <= 4096)
                                    po[2 * u] = hmul2_u(x0, m_o); po[2 * u + 1] = hmul2_u(x1, m_o);
                                }
                                *(uint4 *)(As + (tt * 4 + i) * TC_PANEL) = ev;
                                *(uint4 *)(As + (8 + tt * 4 + i) * TC_PANEL) = od;
                            }
                        }
                        if (s == 0) rscale[t] = make_float2(h2f(cur_d), 0.0f);
                        fence_async_smem();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&a_full[st]);
                    }
                }
            }
        }
    } else {
        // ===================== epilogue: TMEM -> f32 running sums in registers -> dst =====================
        const int quad = warp & 3, ch = warp >> 2;
        const int r = quad * 32 + lane;                                   // tile row = TMEM lane
        uint32_t sbc = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int64_t mt = tile / NT, nt = tile % NT;
            MoeTile gt = {};
            if (GROUPED) gt = args.gtiles[nt];
            const int64_t nval = GROUPED ? (int64_t)gt.count : (args.ncols - nt * TC_TN < TC_TN ? args.ncols - nt * TC_TN : TC_TN);
            const int n_eff = (int)((nval + 15) & ~15);
            float acc[64];
#pragma unroll
            for (int c = 0; c < 64; c++) acc[c] = 0.0f;
            for (int sb = 0; sb < nsb; sb++, sbc++) {
                const int rs = sbc & 1;
                mbar_wait_p(&acc_full[rs], (sbc >> 1) & 1, pw0);
                tc_fence_after();
                const float2 dd = ((const float2 *)(smem + TcSmem::RS + (sbc & 3) * 1024))[r];
                const float * d8 = (const float *)(smem + TcSmem::D8 + (sbc & 3) * 512) + ch * 64;
                const uint32_t tbase = tmem + ((uint32_t)(quad * 32) << 16) + rs * 128 + ch * 64;
#pragma unroll
                for (int c0 = 0; c0 < 64; c0 += 16) {
                    if (ch * 64 + c0 < n_eff) {                            // warp-uniform
                        uint32_t vm[16], vn[16];
                        tc_ld16(tbase + c0, vm);
                        if (TT::HAS_MIN) tc_ld16(tbase + 256 + c0, vn);
                        tc_ld_wait();
#pragma unroll
                        for (int c = 0; c < 16; c++) {
                            const float dx = d8[c0 + c];
                            float u = __fmul_rn(__fmul_rn(dd.x, dx), __uint_as_float(vm[c]));               // d * isum       (ggml-cpu/quants.c:615-620)
                            if (TT::HAS_MIN) u = __fsub_rn(u, __fmul_rn(__fmul_rn(dd.y, dx), __uint_as_float(vn[c])));   // - dmin * imin
                            acc[c0 + c] = __fadd_rn(acc[c0 + c], u);
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[rs]);
            }
            const int64_t row = mt * TC_TM + r;
            if (GROUPED) {
                if (row < args.m) {
#pragma unroll
                    for (int c = 0; c < 64; c++) {
                        const int n = ch * 64 + c;
                        if (n < gt.count) {                                // pair (t, s) of column n -> dst row block (t, s)
                            const int32_t pr = args.gperm[gt.first + n];
                            args.dst[(int64_t)(pr >> 16) * args.dst_tok_stride + (int64_t)(pr & 0xffff) * args.dst_slot_stride + row] = acc[c];
                        }
                    }
                }
            } else if (row < args.m) {
#pragma unroll
                for (int c = 0; c < 64; c++) {
                    const int64_t n = nt * TC_TN + ch * 64 + c;
                    if (n < args.ncols) args.dst[n * args.ldd + row] = acc[c];
                }
            }
        }
    }

    if (prof && lane == 0) {                                           // [warp][total, wait0, wait1, wait2]
        unsigned long long * o = args.prof + warp * 4;
        o[0] = (unsigned long long)(clock64() - t_start); o[1] = w0; o[2] = w1; o[3] = w2;
    }
    // ---- teardown
    pdl_trigger();
    tc_fence_before();
    __syncthreads();
    if (warp == 13) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(512u) : "memory");
}

// ---- host ----------------------------------------------------------------------------------------------------------
bool b200_mmq_tc_supported(int type, int64_t m, int64_t k, int64_t ncols) {
    static const bool off = getenv("B200_MMQ_DISABLE_TC") != nullptr;     // debugging: stream column groups through the matvec kernel instead (still the GPU)
    if (off || m <= 0 || ncols < 9) return false;
    if (type == B200_TYPE_Q4_K || type == B200_TYPE_Q5_K) return k > 0 && k % 256 == 0;
    if (type == B200_TYPE_Q6_K) return k > 0 && k % 2048 == 0;
    return false;
}
int64_t b200_mmq_tc_workspace(int64_t k, int64_t ncols) { return tc_geom(k, ncols).total; }

template <int T, bool GROUPED> static int tc_launch(const TcArgs & a, cudaStream_t st) {
    static bool attr[64] = { false };
    int dev = 0; cudaGetDevice(&dev);
    if (!attr[dev & 63]) { B200_CUDA(cudaFuncSetAttribute(mmq_tc_kernel<T, GROUPED>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem::TOTAL)); attr[dev & 63] = true; }
    int grid = a.n_tiles < b200_sm_count() ? a.n_tiles : b200_sm_count();
    B200_CUDA(b200_launch_pdl(mmq_tc_kernel<T, GROUPED>, dim3((unsigned)grid), dim3(TC_THREADS), (size_t)TcSmem::TOTAL, st, a));
    b200_count_launch();
    return B200_OK;
}

int b200_mmq_tc(int type, const void * W, const float * X, int64_t x_col_stride, float * dst, int64_t ldd, int64_t m, int64_t k, int64_t ncols, void * workspace, void * stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (((uintptr_t)W | (uintptr_t)X | (uintptr_t)workspace) & 15 || (x_col_stride & 3)) { b200_set_error("mul_mat_q: pointers must be 16-byte aligned"); return B200_ERR_INVALID; }
    TcArgs a;
    a.W = (const uint8_t *)W; a.ws = (const uint8_t *)workspace; a.dst = dst; a.m = m; a.k = k; a.ncols = ncols; a.ldd = ldd;
    a.rb = (k / 256) * type_block_bytes(type);
    a.g = tc_geom(k, ncols);
    a.lbo = (uint32_t)TC_PANEL; a.sbo = 128u;
    static unsigned long long * prof_buf = nullptr;                        // B200_MMQ_PROF=1: per-role wait cycles of CTA 0, printed after each launch (bring-up only)
    static const bool want_prof = getenv("B200_MMQ_PROF") != nullptr;
    if (want_prof && !prof_buf) { cudaMalloc((void **)&prof_buf, 16 * 4 * 8); }
    a.prof = want_prof ? prof_buf : nullptr;
    a.nsb = (int32_t)(k / 256); a.n_mtiles = (int32_t)((m + TC_TM - 1) / TC_TM); a.n_tiles = (int32_t)(a.n_mtiles * a.g.nt); a.type = type;
    dim3 qgrid((unsigned)a.nsb, (unsigned)(a.g.nt * 16));
    B200_CUDA(b200_launch_pdl(quantize_mmq_kernel<false>, qgrid, dim3(256), 0, st, X, x_col_stride, ncols, k, (uint8_t *)workspace, a.g, TcGather{}));
    b200_count_launch();
    int rc = B200_ERR_UNSUPPORTED;
    switch (type) {
        case B200_TYPE_Q4_K: rc = tc_launch<B200_TYPE_Q4_K, false>(a, st); break;
        case B200_TYPE_Q5_K: rc = tc_launch<B200_TYPE_Q5_K, false>(a, st); break;
        case B200_TYPE_Q6_K: rc = tc_launch<B200_TYPE_Q6_K, false>(a, st); break;
    }
    if (want_prof && rc == B200_OK) {
        unsigned long long h[16 * 4];
        cudaStreamSynchronize(st); cudaMemcpy(h, prof_buf, sizeof(h), cudaMemcpyDeviceToHost);
        const char * role[14] = { "epi", "epi", "epi", "epi", "epi", "epi", "epi", "epi", "xform", "xform", "xform", "xform", "b-tma", "mma" };
        fprintf(stderr, "mmq_tc prof (CTA 0, cycles): type %d m %lld k %lld n %lld tiles %d\n", type, (long long)m, (long long)k, (long long)ncols, a.n_tiles);
        for (int w = 0; w < 14; w += (w < 8 ? 4 : (w < 12 ? 2 : 1)))
            fprintf(stderr, "  warp %2d %-8s total %9llu  wait0 %9llu  wait1 %9llu  wait2 %9llu\n", w, role[w], h[w * 4], h[w * 4 + 1], h[w * 4 + 2], h[w * 4 + 3]);
        fprintf(stderr, "  (epi: wait0 = acc_full | xform: wait1 = ab_empty | mma: wait0 = acc_empty, wait1 = b_full, wait2 = a_full | b-tma: wait0 = ab_empty)\n");
    }
    return rc;
}

// ---- grouped MUL_MAT_ID (b200_mul_mat_id_q): routing, gathered quantisation, grouped GEMM -----------------------------
// workspace: [B image of moe_max_tiles group tiles][tile table][n_gtiles][perm], sections 256-byte aligned
struct TcIdGeom { int64_t g_max, off_tiles, off_cnt, off_perm, total; TcGeom g; };
static TcIdGeom tc_id_geom(int64_t k, int64_t n_expert, int64_t n_pairs) {
    auto up = [](int64_t x) { return (x + 255) & ~(int64_t)255; };
    TcIdGeom r;
    r.g_max = moe_max_tiles(n_expert, n_pairs);
    r.g = tc_geom(k, r.g_max * TC_TN);
    r.off_tiles = up(r.g.total);
    r.off_cnt = r.off_tiles + up(r.g_max * (int64_t)sizeof(MoeTile));
    r.off_perm = r.off_cnt + 256;
    r.total = r.off_perm + up(n_pairs * 4);
    return r;
}
bool b200_mmq_tc_id_routable(int64_t n_expert, int64_t n_used, int64_t n_tok) {
    return n_expert > 0 && n_expert <= MR_MAX_EXPERT && n_used > 0 && n_tok > 0 && n_used * n_tok <= MR_MAX_PAIRS;
}
int64_t b200_mmq_tc_id_workspace(int64_t k, int64_t n_expert, int64_t n_used, int64_t n_tok) { return tc_id_geom(k, n_expert, n_used * n_tok).total; }

// arguments as b200_mul_mat_id (validated by the caller, b200_mul_mat_id_q); workspace: b200_mmq_tc_id_workspace bytes, 256-byte aligned
int b200_mmq_tc_id(int type, const void * as, int64_t expert_stride_bytes, const float * b, int64_t b_tok_stride, int64_t b_slot_stride, int64_t n_b1,
                   const int32_t * ids, int64_t ids_tok_stride, float * dst, int64_t dst_tok_stride, int64_t dst_slot_stride,
                   int64_t m, int64_t k, int64_t n_expert, int64_t n_used, int64_t n_tok, void * workspace, void * stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (!b200_mmq_tc_id_routable(n_expert, n_used, n_tok)) {
        b200_set_error("mul_mat_id: grouped routing takes at most %d experts and %d (token, slot) pairs", MR_MAX_EXPERT, MR_MAX_PAIRS); return B200_ERR_UNSUPPORTED;
    }
    if (((uintptr_t)as | (uintptr_t)b | (uintptr_t)workspace) & 15 || (b_tok_stride & 3) || (b_slot_stride & 3) || (expert_stride_bytes & 15)) {
        b200_set_error("mul_mat_id: pointers must be 16-byte aligned"); return B200_ERR_INVALID;
    }
    const TcIdGeom G = tc_id_geom(k, n_expert, n_used * n_tok);
    uint8_t * ws = (uint8_t *)workspace;
    MoeTile * tiles = (MoeTile *)(ws + G.off_tiles); int32_t * cnt = (int32_t *)(ws + G.off_cnt); int32_t * perm = (int32_t *)(ws + G.off_perm);
    B200_CUDA(b200_launch_pdl(moe_route_kernel, dim3(1), dim3(MR_THREADS), 0, st, ids, ids_tok_stride, (int)n_expert, (int)n_used, (int)n_tok, perm, tiles, cnt));
    b200_count_launch();
    TcGather ga = {};
    ga.perm = perm; ga.tiles = tiles; ga.n_gtiles = cnt; ga.slot_stride = b_slot_stride; ga.n_b1 = (int32_t)n_b1;
    const dim3 qgrid((unsigned)(k / 256), (unsigned)(G.g_max * 16));
    B200_CUDA(b200_launch_pdl(quantize_mmq_kernel<true>, qgrid, dim3(256), 0, st, b, b_tok_stride, (int64_t)0, k, ws, G.g, ga));
    b200_count_launch();
    TcArgs a = {};
    a.W = (const uint8_t *)as; a.ws = ws; a.dst = dst; a.m = m; a.k = k; a.ncols = 0; a.ldd = 0;
    a.rb = (k / 256) * type_block_bytes(type);
    a.g = G.g;
    a.lbo = (uint32_t)TC_PANEL; a.sbo = 128u;
    a.nsb = (int32_t)(k / 256); a.n_mtiles = (int32_t)((m + TC_TM - 1) / TC_TM);
    a.n_tiles = (int32_t)(a.n_mtiles * G.g_max);                              // upper bound: sizes the persistent grid; the kernel reads the real count
    a.type = type;
    a.gtiles = tiles; a.gperm = perm; a.n_gtiles = cnt;
    a.expert_stride = expert_stride_bytes; a.dst_tok_stride = dst_tok_stride; a.dst_slot_stride = dst_slot_stride;
    switch (type) {
        case B200_TYPE_Q4_K: return tc_launch<B200_TYPE_Q4_K, true>(a, st);
        case B200_TYPE_Q5_K: return tc_launch<B200_TYPE_Q5_K, true>(a, st);
        case B200_TYPE_Q6_K: return tc_launch<B200_TYPE_Q6_K, true>(a, st);
    }
    b200_set_error("mul_mat_id: grouped path has no kernel for type %d", type);
    return B200_ERR_UNSUPPORTED;
}
