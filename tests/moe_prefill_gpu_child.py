"""Child process of tests/test_gpu_moe_prefill.py: runs ONE group of grouped MUL_MAT_ID checks (b200_mul_mat_id_q) on cuda:0 and prints a JSON line.
A separate process so that a faulting kernel cannot poison the CUDA context of the pytest process that runs the rest of the GPU suite."""
import importlib
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from conftest import load_pkg  # noqa: E402
from refutil import Q4_K, Q6_K, oracle, ptr, rand_blocks, row_bytes  # noqa: E402

import torch  # noqa: E402

pkg = load_pkg()
ops = pkg.ops
L = ops.lib


def rel(got, want):
    return float(np.abs(got - want).max() / max(np.abs(want).max(), 1e-30))


def make_ids(rng, mode, E, U, T):
    """[T, row] i32 ids (row = U, or E for the strided top-k view)"""
    if mode == "strided":
        return np.stack([rng.permutation(E) for _ in range(T)]).astype(np.int32)
    ids = np.stack([rng.permutation(E)[:U] for _ in range(T)]).astype(np.int32)
    if mode == "skewed":                                      # expert E-1 takes slot 0 of every token (> 128 pairs), experts 0 and 1 get nothing
        ids[:, 0] = E - 1
        ids[:, 1:] = rng.integers(2, E - 1, (T, U - 1))
    elif mode == "dropped":                                   # -1 and >= n_expert: those (t, s) blocks of dst are not written
        ids[::3, 0] = -1
        ids[1::5, U - 1] = E + 2
    return ids


class Case:
    """one MUL_MAT_ID problem on the device: weights repacked in place (the library layout), ids, activations, a sentinel-filled dst"""

    def __init__(self, t, m, k, E, U, T, n_b1, mode, seed):
        rng = np.random.default_rng(seed)
        self.t, self.m, self.k, self.E, self.U, self.T, self.n_b1 = t, m, k, E, U, T, n_b1
        self.W = rand_blocks(rng, t, E * m, k)
        self.rb = row_bytes(t, k)
        self.Wd = torch.from_numpy(np.concatenate([self.W.reshape(-1), np.zeros(64, np.uint8)])).cuda()
        ops.check(L.b200_repack_rows(t, ops.p(self.Wd), E * m, k, ops.stream()))
        self.b = rng.standard_normal((T, n_b1, k)).astype(np.float32)
        self.bd = torch.from_numpy(self.b).cuda()
        self.ids = make_ids(rng, mode, E, U, T)
        self.idd = torch.from_numpy(self.ids).cuda()
        self.ws_bytes = int(L.b200_mul_mat_id_q_workspace(t, m, k, E, U, T))
        self.ws = torch.zeros(max(self.ws_bytes, 256), dtype=torch.uint8, device="cuda")
        self.dst = torch.full((T, U, m), 7.0, dtype=torch.float32, device="cuda")

    def args(self, dst):
        return (self.t, ops.p(self.Wd), self.m * self.rb, ops.p(self.bd), self.n_b1 * self.k, self.k, self.n_b1, ops.p(self.idd), self.ids.shape[1],
                ops.p(dst), self.U * self.m, self.m, self.m, self.k, self.E, self.U, self.T)

    def grouped(self):
        self.dst.fill_(7.0)
        ops.check(L.b200_mul_mat_id_q(*self.args(self.dst), ops.p(self.ws), ops.stream()))
        torch.cuda.synchronize()
        return self.dst.cpu().numpy()

    def per_column(self):
        d = torch.full_like(self.dst, 7.0)
        ops.check(L.b200_mul_mat_id(*self.args(d), ops.stream()))
        torch.cuda.synchronize()
        return d.cpu().numpy()

    def want(self, rows=None):
        """the oracle (CPU): all rows, or a row sample (weights of those rows only); dropped pairs keep the sentinel"""
        rows = np.arange(self.m) if rows is None else rows
        Ws = np.ascontiguousarray(self.W.reshape(self.E, self.m, -1)[:, rows, :])
        out = np.full((self.T, self.U, rows.size), 7.0, np.float32)
        oracle().orc_mul_mat_id(self.t, ptr(Ws), ptr(self.b), ptr(np.ascontiguousarray(self.ids)), ptr(out), rows.size, self.k, self.E, self.U, self.T,
                                self.n_b1, self.ids.shape[1])
        return out


def check(c, rows=None):
    g1 = c.grouped()
    g2 = c.grouped()
    pc = c.per_column()
    w = c.want(rows)
    sel = (slice(None), slice(None), rows if rows is not None else slice(None))
    return {"ws": c.ws_bytes, "err": rel(g1[sel], w), "err_per_column": rel(pc[sel], w), "vs_per_column": rel(g1, pc),
            "bit_identical": bool(np.array_equal(g1, g2)), "sentinel_kept": bool(np.all(g1[c.ids[:, :c.U] < 0] == 7.0) and np.all(g1[c.ids[:, :c.U] >= c.E] == 7.0))}


def do_suite(t):
    """one weight type: n_tok 9 / 64 / 512 x shared / per-slot activations, skewed routing, dropped ids, strided ids; m = 200 (not a multiple of 128)"""
    k = 2048 if t == Q6_K else 1024
    out = {}
    for T in (9, 64, 512):
        for n_b1 in (1, 4):
            out[f"T{T}_b1{n_b1}"] = check(Case(t, 200, k, 8, 4, T, n_b1, "random", 100 * t + T + n_b1))
    for mode in ("skewed", "dropped", "strided"):
        out[mode] = check(Case(t, 200, k, 8, 4, 300, 1, mode, 7 * t + len(mode)))
    return out


SHAPES = {"qwen3_moe": (Q4_K, 768, 2048, 128, 8, 1), "mixtral_up": (Q4_K, 14336, 4096, 8, 2, 1), "mixtral_down": (Q6_K, 4096, 14336, 8, 2, 2)}


def do_shape(name, T):
    """a model-sized expert stack, checked on a row sample (every tile position: first and last rows, the m-tile edges, random rows)"""
    t, m, k, E, U, n_b1 = SHAPES[name]
    c = Case(t, m, k, E, U, T, n_b1, "random", T + m)
    rng = np.random.default_rng(m)
    rows = np.unique(np.concatenate([[0, 127, 128, m - 1], rng.choice(m, 60, replace=False)]))
    return check(c, rows)


def do_graph():
    """capture ONE call on a stream, then replay it with different ids written into the same buffer: each replay against the oracle"""
    c = Case(Q4_K, 256, 1024, 8, 2, 64, 1, "random", 5)
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    c.grouped()                                               # warm-up outside the capture (kernel attributes are set on first use)
    with torch.cuda.graph(g, stream=s):
        ops.check(L.b200_mul_mat_id_q(*c.args(c.dst), ops.p(c.ws), ops.stream()))
    errs, counts = [], []
    rng = np.random.default_rng(9)
    for rep in range(4):
        if rep == 1:
            c.ids = make_ids(rng, "skewed", 8, 2, 64)
        elif rep == 2:
            c.ids = make_ids(rng, "dropped", 8, 2, 64)
        elif rep == 3:
            c.ids = make_ids(rng, "random", 8, 2, 64)
        c.idd.copy_(torch.from_numpy(c.ids))
        c.dst.fill_(7.0)
        g.replay()
        torch.cuda.synchronize()
        errs.append(rel(c.dst.cpu().numpy(), c.want()))
        counts.append(int(np.sum((c.ids >= 0) & (c.ids < 8))))
    return {"ws": c.ws_bytes, "errs": errs, "valid_pairs": counts}


def do_executor(n_tok):
    """MUL_MAT_ID(up), MUL_MAT_ID(gate), GLU, MUL_MAT_ID(down) through the graph executor with the ids as an input tensor; every node's output against
    the oracle applied to that node's inputs as the executor computed them; eager run, capture, replays with the ids changed in place"""
    assert os.environ.get("GGML_B200_WIDE") == "1"
    G = importlib.import_module("llama_box_b200.graph")
    E, FF, NE, NU = 1024, 2048, 8, 2
    O = oracle()
    rng = np.random.default_rng(n_tok)
    Wup, Wgate, Wdown = rand_blocks(rng, Q4_K, NE * FF, E), rand_blocks(rng, Q4_K, NE * FF, E), rand_blocks(rng, Q6_K, NE * E, FF)
    x = rng.standard_normal((n_tok, E)).astype(np.float32)
    keep = {}

    def wdev(name, t, W, k):
        d = torch.from_numpy(np.concatenate([W.reshape(-1), np.zeros(64, np.uint8)])).cuda()
        ops.check(L.b200_repack_rows(t, ops.p(d), W.shape[0], k, ops.stream()))
        keep[name] = d
        return d.data_ptr()

    def f32(name, shape):
        keep[name] = torch.zeros(shape, dtype=torch.float32, device="cuda")
        return keep[name].data_ptr()
    keep["x"] = torch.from_numpy(x).cuda()
    keep["ids"] = torch.zeros((n_tok, NU), dtype=torch.int32, device="cuda")
    nl = G.NodeList()
    xt = G.T(keep["x"].data_ptr(), G.F32, [E, 1, n_tok], [4, 4 * E, 4 * E, 4 * E * n_tok])
    sel = G.T(keep["ids"].data_ptr(), G.I32, [NU, n_tok])
    up = nl.add(G.OP_MUL_MAT_ID, G.T(f32("up", (n_tok, NU, FF)), G.F32, [FF, NU, n_tok]), [G.T(wdev("wu", Q4_K, Wup, E), G.Q4_K, [E, FF, NE]), xt, sel])
    gate = nl.add(G.OP_MUL_MAT_ID, G.T(f32("gate", (n_tok, NU, FF)), G.F32, [FF, NU, n_tok]), [G.T(wdev("wg", Q4_K, Wgate, E), G.Q4_K, [E, FF, NE]), xt, sel])
    act = nl.add(G.OP_GLU_SWIGLU, G.T(f32("act", (n_tok, NU, FF)), G.F32, [FF, NU, n_tok]), [gate, up], [2, 0])
    down = nl.add(G.OP_MUL_MAT_ID, G.T(f32("down", (n_tok, NU, E)), G.F32, [E, NU, n_tok]), [G.T(wdev("wd", Q6_K, Wdown, FF), G.Q6_K, [FF, E, NE]), act, sel])
    for h in (up, gate, act, down):                           # reshapes of the outputs as ggml records them (op NONE); 8 nodes: a list the executor captures
        nl.view_op(G.T(h.ptr, G.F32, [h.ne[0], h.ne[1] * h.ne[2]]), h)
    nodes = nl.build()
    ex = G.Executor(0)
    sup = [bool(ex.supports(nodes[i])) for i in range(len(nodes))]
    runs = []
    side = torch.cuda.Stream()
    for rep in range(4):                                      # eager, capture, replay, replay — new ids before every run
        ids = np.stack([rng.permutation(NE)[:NU] for _ in range(n_tok)]).astype(np.int32)
        if rep == 2:
            ids[:, 0] = NE - 1                                # skewed: one expert takes every token
        keep["ids"].copy_(torch.from_numpy(ids))
        for name in ("up", "gate", "act", "down"):
            keep[name].fill_(7.0)
        with torch.cuda.stream(side):                         # the legacy default stream cannot be captured: the executor runs it eagerly
            ex.compute(nodes)
        torch.cuda.synchronize()
        got = {n: keep[n].cpu().numpy() for n in ("up", "gate", "act", "down")}
        w_up = np.zeros_like(got["up"]); w_gate = np.zeros_like(got["gate"]); w_down = np.zeros_like(got["down"])
        O.orc_mul_mat_id(Q4_K, ptr(Wup), ptr(x), ptr(ids), ptr(w_up), FF, E, NE, NU, n_tok, 1, NU)
        O.orc_mul_mat_id(Q4_K, ptr(Wgate), ptr(x), ptr(ids), ptr(w_gate), FF, E, NE, NU, n_tok, 1, NU)
        w_act = np.zeros_like(got["act"]); O.orc_swiglu(ptr(np.ascontiguousarray(got["gate"])), ptr(np.ascontiguousarray(got["up"])), ptr(w_act), w_act.size)
        O.orc_mul_mat_id(Q6_K, ptr(Wdown), ptr(np.ascontiguousarray(got["act"])), ptr(ids), ptr(w_down), E, FF, NE, NU, n_tok, NU, NU)
        runs.append({"up": rel(got["up"], w_up), "gate": rel(got["gate"], w_gate), "act": rel(got["act"], w_act), "down": rel(got["down"], w_down),
                     "kernels": int(ex.last_kernels)})
    ws = [int(L.b200_mul_mat_id_q_workspace(Q4_K, FF, E, NE, NU, n_tok)), int(L.b200_mul_mat_id_q_workspace(Q6_K, E, FF, NE, NU, n_tok))]
    return {"supports": sup, "runs": runs, "captures": int(ex.captures), "replays": int(ex.replays), "ws": ws, "plan": G.plan(nodes)}


if __name__ == "__main__":
    torch.cuda.set_device(0)
    what, args = sys.argv[1], sys.argv[2:]
    if what == "suite":
        r = do_suite(int(args[0]))
    elif what == "shape":
        r = do_shape(args[0], int(args[1]))
    elif what == "graph":
        r = do_graph()
    elif what == "executor":
        r = do_executor(int(args[0]))
    else:
        raise SystemExit(f"unknown check {what}")
    print("RESULT " + json.dumps(r))
