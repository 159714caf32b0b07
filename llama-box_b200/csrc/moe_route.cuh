// moe_route.cuh — expert routing of the grouped MUL_MAT_ID (launch code: mmq_tc.cu, b200_mmq_tc_id).
// Reads the (token, slot) -> expert ids ON THE DEVICE and groups the pairs by expert, so that the tensor-core GEMM can read each
// expert's weight tile once per 128 pairs instead of once per pair; the reference copies the ids to the host and sorts there,
// synchronising the stream twice per op (ggml-cuda/mmq.cu:145-228).  Kept in a header so that tests/hostsim/kernsim.cpp runs the
// same source under the SIMT emulation (tests/test_moe_route_simt.py): no atomics, only __syncthreads.
#pragma once
#include "common.cuh"

constexpr int MR_THREADS = 512;
constexpr int MR_MAX_EXPERT = 256;
constexpr int MR_MAX_PAIRS = 16384;       // n_tok * n_used; the expert of every pair is staged in shared memory (int16: 32 KB)
constexpr int MR_TILE = 128;              // pairs per group tile = the GEMM's N tile

// one group tile: `count` (<= 128) consecutive entries of perm, starting at `first`, all routed to `expert`
struct MoeTile { int32_t expert, first, count, _pad; };

// perm entry of pair (t, s): t << 16 | s  (t < MR_MAX_PAIRS, s < 65536)
__host__ __device__ inline int32_t moe_pair_pack(int64_t t, int64_t s) { return (int32_t)((t << 16) | s); }

// upper bound of the number of group tiles: sum over the non-empty experts (at most min(E, P) of them) of ceil(count / 128)
__host__ __device__ inline int64_t moe_max_tiles(int64_t n_expert, int64_t n_pairs) {
    return (n_pairs + (MR_TILE - 1) * (n_expert < n_pairs ? n_expert : n_pairs)) / MR_TILE;
}

// One CTA.  Outputs:
//   perm[0 .. n_valid)   pairs grouped by expert, expert-major, and inside an expert in increasing (t, s) order (deterministic)
//   tiles[0 .. n_gtiles) one entry per 128-pair chunk of each expert's list, in expert order
//   *n_gtiles            the number of tiles (read on the device by the kernels that follow; nothing goes to the host)
// Ids outside [0, n_expert) are dropped (b200_mul_mat_id's contract: such pairs write nothing).
// Work split: S = the largest power of two with n_expert * S <= MR_THREADS threads per expert; sub-thread j of expert e counts,
// then writes, the pairs of e inside the j-th contiguous chunk of the pair range, at the offset a block-wide exclusive scan of the
// counts (in (e, j) order) gives it.
__global__ void __launch_bounds__(MR_THREADS) moe_route_kernel(const int32_t * __restrict__ ids, int64_t ids_tok_stride, int n_expert, int n_used, int n_tok,
                                                              int32_t * __restrict__ perm, MoeTile * __restrict__ tiles, int32_t * __restrict__ n_gtiles) {
    __shared__ int16_t sid[MR_MAX_PAIRS];
    __shared__ int32_t scan[MR_THREADS];
    __shared__ int32_t efirst[MR_MAX_EXPERT], eend[MR_MAX_EXPERT], etile[MR_MAX_EXPERT];
    pdl_wait();                                                        // ids come from an earlier kernel (ARGSORT / top-k)
    const int tid = threadIdx.x;
    const int P = n_tok * n_used;
    for (int p = tid; p < P; p += MR_THREADS) {
        const int t = p / n_used, s = p - t * n_used;
        const int e = ids[(int64_t)t * ids_tok_stride + s];
        sid[p] = (int16_t)(e >= 0 && e < n_expert ? e : -1);
    }
    int S = 1;
    while (n_expert * S * 2 <= MR_THREADS) S *= 2;
    const int e = tid / S, j = tid - e * S;
    const bool active = e < n_expert;
    const int chunk = (P + S - 1) / S;
    const int lo = j * chunk < P ? j * chunk : P, hi = lo + chunk < P ? lo + chunk : P;
    __syncthreads();

    int cnt = 0;
    if (active)
        for (int p = lo; p < hi; p++) cnt += sid[p] == e;
    scan[tid] = cnt;
    __syncthreads();
    for (int o = 1; o < MR_THREADS; o <<= 1) {                         // inclusive scan (Hillis-Steele)
        const int v = tid >= o ? scan[tid - o] : 0;
        __syncthreads();
        scan[tid] += v;
        __syncthreads();
    }
    const int excl = scan[tid] - cnt;
    if (active && j == 0) efirst[e] = excl;
    if (active && j == S - 1) eend[e] = scan[tid];
    __syncthreads();
    if (tid == 0) {
        int g = 0;
        for (int x = 0; x < n_expert; x++) { etile[x] = g; g += (eend[x] - efirst[x] + MR_TILE - 1) / MR_TILE; }
        *n_gtiles = g;
    }
    __syncthreads();

    if (active) {
        int o = excl;
        for (int p = lo; p < hi; p++)
            if (sid[p] == e) { const int t = p / n_used; perm[o++] = moe_pair_pack(t, p - t * n_used); }
    }
    for (int x = tid; x < n_expert; x += MR_THREADS) {
        const int f = efirst[x], c = eend[x] - f;
        int g = etile[x];
        for (int i = 0; i < c; i += MR_TILE, g++) {
            MoeTile mt; mt.expert = x; mt.first = f + i; mt.count = c - i < MR_TILE ? c - i : MR_TILE; mt._pad = 0;
            tiles[g] = mt;
        }
    }
    pdl_trigger();
}
