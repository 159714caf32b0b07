"""CPU: the grouped MUL_MAT_ID path of the prefill (b200_mul_mat_id_q) without a GPU.
  * the routing kernel (llama-box_b200/csrc/moe_route.cuh) and the gathered activation quantiser (mmq_quant.cuh) run from their CUDA SOURCE under
    the SIMT emulation (tests/hostsim/simt.h) and are compared with a numpy model / with the dense quantiser on the same columns;
  * the routing decision of b200_mul_mat_id_q is read from b200_mul_mat_id_q_workspace (0 = the per-column matvec of b200_mul_mat_id)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from refutil import ROOT, ptr

SIM_DIR = os.path.join(ROOT, "tests", "hostsim")
CSRC = os.path.join(ROOT, "llama-box_b200", "csrc")
CUDA_INC = "/usr/local/cuda/include"
Q4_0, Q8_0, Q4_K, Q5_K, Q6_K = 2, 8, 12, 13, 14
WIDE_ONLY = (3, 7, 10, 11, 20, 23, 39)


@pytest.fixture(scope="module")
def K():
    if not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")):
        pytest.skip("CUDA headers not installed")
    so = os.path.join(SIM_DIR, "libmoesim.so")
    deps = [os.path.join(SIM_DIR, f) for f in ("moesim.cpp", "simt.h")] + [os.path.join(CSRC, f) for f in ("moe_route.cuh", "mmq_quant.cuh", "common.cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++20", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-w", "-I" + CUDA_INC, "-x", "c++",
                               os.path.join(SIM_DIR, "moesim.cpp"), "-o", so])
    L = C.CDLL(so)
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int
    L.sim_moe_max_tiles.argtypes = [i64, i64]
    L.sim_moe_route.argtypes = [vp, i64, i32, i32, i32, vp, vp, vp]
    L.sim_quantize_mmq.argtypes = [vp, i64, i64, i64, vp]
    L.sim_quantize_mmq_gather.argtypes = [vp, i64, i64, i64, i64, vp, vp, vp, i64, vp]
    return L


def route_model(ids, n_expert):
    """numpy model: pairs (t, s) grouped by expert in increasing (t, s) order, ids outside [0, n_expert) dropped; 128-pair tiles in expert order"""
    n_tok, n_used = ids.shape
    perm, tiles = [], []
    for e in range(n_expert):
        pairs = [(t, s) for t in range(n_tok) for s in range(n_used) if ids[t, s] == e]
        for i in range(0, len(pairs), 128):
            tiles.append((e, len(perm) + i, min(128, len(pairs) - i)))
        perm += pairs
    return perm, tiles


def run_route(K, ids_full, n_used, n_expert):
    """ids_full: [n_tok, row] i32 with the (t, s) id at column s (row stride = ids_full.shape[1])"""
    n_tok = ids_full.shape[0]
    P = n_tok * n_used
    g_max = K.sim_moe_max_tiles(n_expert, P)
    perm = np.full(P, -7, np.int32)
    tiles = np.full((g_max + 1, 4), -7, np.int32)                 # one guard entry past the bound
    cnt = np.full(4, -7, np.int32)
    K.sim_moe_route(ptr(ids_full), ids_full.shape[1], n_expert, n_used, n_tok, ptr(perm), ptr(tiles), ptr(cnt))
    return perm, tiles, int(cnt[0]), g_max


def check_route(K, ids_full, n_used, n_expert):
    ids = ids_full[:, :n_used]
    want_perm, want_tiles = route_model(ids, n_expert)
    perm, tiles, n_gt, g_max = run_route(K, ids_full, n_used, n_expert)
    assert n_gt == len(want_tiles) and n_gt <= g_max
    got_pairs = [(int(v) >> 16, int(v) & 0xffff) for v in perm[:len(want_perm)]]
    assert got_pairs == want_perm
    assert np.all(perm[len(want_perm):] == -7)                      # nothing written for dropped pairs
    assert [tuple(int(x) for x in r[:3]) for r in tiles[:n_gt]] == want_tiles
    assert np.all(tiles[g_max] == -7)
    return want_tiles


@pytest.mark.parametrize("E,U,T", [(8, 2, 9), (8, 2, 512), (128, 8, 512), (256, 8, 2048)])
def test_route_kernel_vs_model(K, E, U, T):
    rng = np.random.default_rng(E * 1000 + U * 100 + T)
    ids = np.stack([rng.permutation(E)[:U] for _ in range(T)]).astype(np.int32)
    check_route(K, ids, U, E)


def test_route_all_pairs_on_one_expert_and_empty_experts(K):
    E, U, T = 8, 2, 300                                             # expert 5 gets every slot 0 (300 pairs = 3 tiles), slot 1 goes to 2 or 6
    rng = np.random.default_rng(1)
    ids = np.stack([np.full(T, 5), rng.choice([2, 6], T)], axis=1).astype(np.int32)
    tiles = check_route(K, ids, U, E)
    assert [t[0] for t in tiles].count(5) == 3 and {t[0] for t in tiles} == {2, 5, 6}


def test_route_drops_out_of_range_ids(K):
    E, U, T = 8, 4, 64
    rng = np.random.default_rng(2)
    ids = rng.integers(-1, E + 3, (T, U)).astype(np.int32)          # -1 and >= n_expert are dropped
    ids[0, :] = -1
    check_route(K, ids, U, E)


def test_route_strided_ids(K):
    """ids as llama's top-k view of the ARGSORT output: [n_used, n_tok] with row stride n_expert"""
    E, U, T = 16, 2, 100
    rng = np.random.default_rng(3)
    full = np.stack([rng.permutation(E) for _ in range(T)]).astype(np.int32)
    check_route(K, full, U, E)


def tc_geom(k, ncols):
    nt, kq, nsb = (ncols + 127) // 128, k // 64, k // 256
    off_bm = nt * kq * 16384
    off_d8 = off_bm + nt * nsb * 4096
    return dict(nt=nt, kq=kq, nsb=nsb, off_bm=off_bm, off_d8=off_d8, total=off_d8 + nt * nsb * 512)


def tile_sections(img, g, i):
    """(Bq, Bm, D8) bytes of 128-column tile i of a B image"""
    return (img[i * g["kq"] * 16384:(i + 1) * g["kq"] * 16384],
            img[g["off_bm"] + i * g["nsb"] * 4096:g["off_bm"] + (i + 1) * g["nsb"] * 4096],
            img[g["off_d8"] + i * g["nsb"] * 512:g["off_d8"] + (i + 1) * g["nsb"] * 512])


@pytest.mark.parametrize("n_b1", [1, 3])
def test_gathered_quantiser_equals_dense_image(K, n_b1):
    """the gathered B image (column c of group tile g = b[t, s % n_b1] of pair perm[first + c]) equals the image quantize_mmq_kernel makes of the same
    columns laid out densely, tile by tile; columns past a tile's count are zeros"""
    E, U, T, k = 4, 3, 70, 512
    rng = np.random.default_rng(n_b1)
    ids = np.stack([rng.permutation(E)[:U] for _ in range(T)]).astype(np.int32)
    ids[:, 0] = 1                                                   # expert 1: 70 + ~35 pairs (a second, partial tile)
    ids[5, 2] = -1
    b = (rng.standard_normal((T, n_b1, k)) * 2).astype(np.float32)
    b[3, 0, 256:512] = 0                                            # an all-zero super-block
    perm, tiles, n_gt, g_max = run_route(K, ids, U, E)
    g = tc_geom(k, g_max * 128)
    img = np.full(g["total"], 0xAB, np.uint8)
    K.sim_quantize_mmq_gather(ptr(b), n_b1 * k, k, n_b1, k, ptr(perm), ptr(tiles), ptr(np.array([n_gt, 0, 0, 0], np.int32)), g_max, ptr(img))
    # the same columns, dense: tile i's columns at i * 128 .. i * 128 + count, zeros elsewhere
    X = np.zeros((n_gt * 128, k), np.float32)
    for i in range(n_gt):
        e, first, count = (int(v) for v in tiles[i, :3])
        for c in range(count):
            pr = int(perm[first + c]); t, s = pr >> 16, pr & 0xffff
            assert ids[t, s] == e
            X[i * 128 + c] = b[t, s % n_b1]
    gd = tc_geom(k, n_gt * 128)
    dense = np.full(gd["total"], 0xCD, np.uint8)
    K.sim_quantize_mmq(ptr(X), k, n_gt * 128, k, ptr(dense))
    for i in range(n_gt):
        for a, d in zip(tile_sections(img, g, i), tile_sections(dense, gd, i)):
            assert np.array_equal(a, d), i
    for i in range(n_gt, g_max):                                    # tiles past the count are not touched
        assert all(np.all(s == 0xAB) for s in tile_sections(img, g, i))


# ---- the routing decision of b200_mul_mat_id_q --------------------------------------------------------------------------------------
MIXTRAL_UP = (Q4_K, 14336, 4096, 8, 2)
MIXTRAL_DOWN = (Q6_K, 4096, 14336, 8, 2)                            # k = 14336 = 7 x 2048
QWEN3_MOE = (Q4_K, 768, 2048, 128, 8)


def b_image_bytes(k, n_expert, n_pairs):
    g_max = (n_pairs + 127 * min(n_expert, n_pairs)) // 128
    return tc_geom(k, g_max * 128)["total"]


def min_grouped_tokens(E, U):
    """the dispatch rule: at least 9 tokens and at least 4 (token, slot) pairs per expert"""
    return max(9, -(-4 * E // U))


@pytest.mark.parametrize("shape", [MIXTRAL_UP, MIXTRAL_DOWN, QWEN3_MOE, (Q5_K, 1024, 512, 8, 2)])
def test_workspace_covers_the_grouped_path(b200, shape):
    t, m, k, E, U = shape
    n0 = min_grouped_tokens(E, U)
    for n_tok in (n0, 64, 512):
        ws = b200.lib.b200_mul_mat_id_q_workspace(t, m, k, E, U, n_tok)
        assert ws > 0 and ws >= b_image_bytes(k, E, n_tok * U) + n_tok * U * 4
    assert b200.lib.b200_mul_mat_id_q_workspace(t, m, k, E, U, n0 - 1) == 0


def test_workspace_is_zero_on_the_per_column_path(b200):
    W = b200.lib.b200_mul_mat_id_q_workspace
    for n_tok in range(1, 9):                                       # decode and verify batches keep the one-launch matvec, whatever the routing density
        assert W(Q4_K, 14336, 4096, 8, 2, n_tok) == 0 and W(Q4_K, 4096, 4096, 2, 2, n_tok) == 0
    assert W(Q4_K, 4096, 4096, 2, 2, 9) > 0
    assert W(Q4_K, 768, 2048, 128, 8, 63) == 0 and W(Q4_K, 768, 2048, 128, 8, 64) > 0   # fewer than 4 pairs per expert
    for t in WIDE_ONLY + (Q4_0, Q8_0):
        assert W(t, 4096, 4096, 8, 2, 64) == 0
    assert W(Q6_K, 4096, 1536, 8, 2, 64) == 0                       # Q6_K: k % 2048 != 0
    assert W(Q6_K, 4096, 2048, 8, 2, 64) > 0
    assert W(Q4_K, 4096, 4096, 257, 8, 2048) == 0                   # beyond the routing kernel: > 256 experts, > 16384 pairs
    assert W(Q4_K, 4096, 4096, 8, 8, 2049) == 0 and W(Q4_K, 4096, 4096, 8, 8, 2048) > 0


def test_workspace_honours_the_tensor_core_switch():
    code = ("import sys; sys.path.insert(0, 'tests'); from conftest import load_pkg; L = load_pkg().ops.lib; "
            "print(L.b200_mul_mat_id_q_workspace(12, 14336, 4096, 8, 2, 512))")
    env = dict(os.environ, B200_MMQ_DISABLE_TC="1")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.split()[-1] == "0"
