"""MUL_MAT_ID prefill: the per-column matvec (b200_mul_mat_id) against the grouped tensor-core path (b200_mul_mat_id_q) on the same inputs.

Shapes: Mixtral-8x7B (8 experts, 2 used; ffn_up / ffn_gate 14336 x 4096 Q4_K, ffn_down 4096 x 14336 Q6_K with per-slot activations) and a
Qwen3-30B-A3B-like stack (128 experts, 8 used, 768 x 2048 Q4_K); n_tok in {8, 9, 16, 32, 64, 128, 512}; random ids (distinct experts per token).
Timing: CUDA events around each call, the two paths alternating pass by pass after a warm-up, and the L2 overwritten (a 256 MB write) before
every timed call, so that expert stacks smaller than the 126 MB L2 (the Qwen3-like one) are read from HBM as in a real forward pass.
At 8 tokens b200_mul_mat_id_q IS b200_mul_mat_id (below the grouping threshold): that row measures the dispatch's own overhead.
Output: one JSON line per case (and the card's name and power limit first) to stdout and --out.
    python tools/moe_prefill_bench.py --out profiles/r3_moe_prefill.jsonl"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

SHAPES = {  # name: (type, m, k, n_expert, n_used, n_b1)
    "mixtral_up": (12, 14336, 4096, 8, 2, 1),
    "mixtral_down": (14, 4096, 14336, 8, 2, 2),
    "qwen3_moe_up": (12, 768, 2048, 128, 8, 1),
}
TOKENS = (8, 9, 16, 32, 64, 128, 512)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from conftest import load_pkg
    assert torch.cuda.is_available(), "needs a CUDA device"
    ops = load_pkg().ops
    L = ops.lib
    torch.cuda.set_device(0)
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    lines = [json.dumps({"card": torch.cuda.get_device_name(0), "nvidia_smi": q, "l2_flush": "256 MB write before every timed call"})]
    print(lines[-1], flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    rng = np.random.default_rng(0)
    for name, (t, m, k, E, U, n_b1) in SHAPES.items():
        rb = ops.row_bytes(t, k)
        W = torch.randint(0, 256, (E * m * rb + 64,), dtype=torch.uint8, device="cuda")
        # valid f16 scales: random bytes give NaN/Inf scales that are still fine for timing, but keep d small and finite anyway
        Wv = W[:E * m * rb].view(E * m, rb)
        if t == 14:
            Wv[:, rb - 2 * (k // 256):].view(torch.float16).fill_(1e-4)
        else:
            Wv.view(E * m, k // 256, 144 if t == 12 else 176)[:, :, :4].view(torch.float16).fill_(1e-3)
        for T in TOKENS:
            b = torch.randn((T, n_b1, k), dtype=torch.float32, device="cuda")
            ids_np = np.stack([rng.permutation(E)[:U] for _ in range(T)]).astype(np.int32)
            ids = torch.from_numpy(ids_np).cuda()
            dst = torch.empty((T, U, m), dtype=torch.float32, device="cuda")
            wsb = int(L.b200_mul_mat_id_q_workspace(t, m, k, E, U, T))
            ws = torch.empty(max(wsb, 256), dtype=torch.uint8, device="cuda")
            args = (t, ops.p(W), m * rb, ops.p(b), n_b1 * k, k, n_b1, ops.p(ids), U, ops.p(dst), U * m, m, m, k, E, U, T)
            st = ops.stream()
            run = {"per_column": lambda: ops.check(L.b200_mul_mat_id(*args, st)),
                   "grouped": lambda: ops.check(L.b200_mul_mat_id_q(*args, ops.p(ws), st))}
            for _ in range(a.warmup):
                for f in run.values():
                    f()
            tot = {key: 0.0 for key in run}
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for _ in range(a.passes):
                for key, f in run.items():
                    flush.fill_(1)
                    e0.record(); f(); e1.record()
                    e1.synchronize()
                    tot[key] += e0.elapsed_time(e1) * 1e3 / a.passes
            pairs = T * U
            counts = np.bincount(ids_np.reshape(-1), minlength=E)
            tiles = int(np.sum((counts + 127) // 128))
            r = {"shape": name, "type": t, "m": m, "k": k, "n_expert": E, "n_used": U, "n_tok": T, "grouped_path": wsb > 0,
                 "us_per_column": round(tot["per_column"], 2), "us_grouped": round(tot["grouped"], 2),
                 "speedup": round(tot["per_column"] / tot["grouped"], 3),
                 "tflops_per_column": round(2 * m * k * pairs / tot["per_column"] * 1e-6, 2), "tflops_grouped": round(2 * m * k * pairs / tot["grouped"] * 1e-6, 2),
                 "weight_bytes_per_column": pairs * m * rb, "weight_bytes_grouped": (tiles * m * rb) if wsb > 0 else pairs * m * rb}
            lines.append(json.dumps(r))
            print(lines[-1], flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
