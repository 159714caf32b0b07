"""GPU: the grouped tensor-core MUL_MAT_ID of the prefill (b200_mul_mat_id_q: routing on the device, gathered q8_K activations, mmq_tc.cu's GEMM with a
per-expert row map) against the C oracle, against the per-column path (b200_mul_mat_id), inside a CUDA graph whose ids change between replays, through
the graph executor and through the unmodified libllama.  Every check runs in a child process (tests/moe_prefill_gpu_child.py) so that a faulting
kernel cannot poison the CUDA context of the rest of the GPU suite."""
import json
import os
import re
import subprocess
import sys

import pytest

from refutil import ROOT, have_ref

pytestmark = pytest.mark.gpu
CHILD = os.path.join(ROOT, "tests", "moe_prefill_gpu_child.py")
BOUND = 2e-5                                                  # the dense tensor-core MUL_MAT's bound (test_gpu_ops.py)


def child(*args, wide=False, timeout=1200):
    env = dict(os.environ)
    env.pop("GGML_B200_WIDE", None)
    if wide:
        env["GGML_B200_WIDE"] = "1"
    r = subprocess.run([sys.executable, CHILD] + [str(a) for a in args], capture_output=True, text=True, env=env, timeout=timeout)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1]
    return json.loads(line[7:])


def assert_case(name, r):
    assert r["ws"] > 0, (name, r)                             # the grouped path really ran
    assert r["err"] <= BOUND and r["err_per_column"] <= BOUND and r["vs_per_column"] <= BOUND, (name, r)
    assert r["bit_identical"] and r["sentinel_kept"], (name, r)


@pytest.mark.parametrize("wtype", [12, 13, 14])
def test_grouped_mul_mat_id_vs_oracle_and_per_column(wtype):
    """n_tok 9 / 64 / 512 with shared (n_b1 = 1) and per-slot (n_b1 = n_used) activations, skewed routing (one expert > 128 pairs, two with none),
    ids -1 and >= n_expert (sentinel-filled dst untouched), strided ids (llama's top-k view); m = 200; two runs bit-identical"""
    o = child("suite", wtype)
    assert len(o) == 9, o
    for name, r in o.items():
        assert_case(name, r)


@pytest.mark.parametrize("shape,n_tok", [("qwen3_moe", 512), ("qwen3_moe", 64), ("mixtral_up", 512), ("mixtral_down", 512), ("mixtral_down", 16)])
def test_grouped_mul_mat_id_model_shapes(shape, n_tok):
    """Qwen3-MoE-like (E 128, U 8, 768 x 2048 Q4_K) and Mixtral-8x7B ffn_up (14336 x 4096 Q4_K) / ffn_down (4096 x 14336 Q6_K), checked on a row sample;
    64 / 16 tokens: the smallest ubatches that take the grouped path for these shapes (4 pairs per expert)"""
    assert_case(shape, child("shape", shape, n_tok))


def test_grouped_mul_mat_id_in_a_cuda_graph_with_changing_ids():
    """one captured call replayed with different ids in the same buffer (random, skewed, dropped, random): nothing about the routing is baked in"""
    o = child("graph")
    assert o["ws"] > 0 and len(o["errs"]) == 4, o
    assert max(o["errs"]) <= BOUND, o
    assert len(set(o["valid_pairs"])) > 1, o                  # the replays really saw different routings


@pytest.mark.parametrize("n_tok,kernels", [(4, 4), (64, 10)])
def test_executor_moe_ffn_grouped_vs_oracle(n_tok, kernels):
    """GGML_B200_WIDE=1: MUL_MAT_ID(up), MUL_MAT_ID(gate), GLU, MUL_MAT_ID(down) with ids as an input tensor.  64 tokens: routing + quantisation + GEMM per
    MUL_MAT_ID (10 launches); 4 tokens: one matvec launch per MUL_MAT_ID as before (4).  Eager run, capture and replays with the ids changed in place."""
    o = child("executor", n_tok, wide=True)
    assert all(o["supports"]), o
    assert (min(o["ws"]) > 0) == (n_tok >= 9), o
    for r in o["runs"]:
        assert r["up"] <= BOUND and r["gate"] <= BOUND and r["down"] <= BOUND and r["act"] <= 1e-6, o
        assert r["kernels"] == kernels, o
    assert o["plan"] == kernels, o
    assert o["captures"] >= 1 and o["replays"] >= 2, o


@pytest.fixture(scope="module")
def product():
    import test_gpu_product as P
    for key in [k for k, path in P._models.items() if not os.path.exists(path)]:
        del P._models[key]
    yield P
    for path in list(P._models.values()):
        try:
            os.remove(path)
        except OSError:
            pass


@pytest.mark.skipif(not have_ref(), reason="oracle/_ref (reference build) not present")
def test_libllama_moe_prefill_over_the_grouped_path(tmp_path, tmp_path_factory, product):
    """the unmodified libllama on the test-moe file (Q4_K_M) with a 300-token prompt: one prefill ubatch, so every MUL_MAT_ID of it takes the grouped
    path.  The scheduler must place MUL_MAT_ID on the B200 backend, and the run must be as close to ggml-cpu as ggml-cpu's own other builds are."""
    P = product
    gguf = P.model_file(tmp_path_factory, "test-moe", "Q4_K_M", 2)
    cpu = P.drv(gguf, str(tmp_path / "cpu"), False, prompt_len=300, gen=9)
    others = P.cpu_builds(tmp_path, tmp_path_factory, gguf, prompt_len=300, gen=9)
    gpu = P.drv(gguf, str(tmp_path / "gpu"), True, prompt_len=300, gen=9, extra_env=dict(GGML_B200_WIDE="1", GGML_SCHED_DEBUG="2", LLAMA_DRV_LOG_DEBUG="1"))
    placed = re.findall(r"node #\s*\d+ \(\s*MUL_MAT_ID\w*\):.*?\[\s*(\w+)", gpu["stderr"])
    assert placed and all(b.startswith("B200") for b in placed), (len(placed), sorted(set(placed)))
    P.assert_within_reference_self_consistency(gpu, cpu, others, "grouped MUL_MAT_ID: test-moe Q4_K_M, 300-token prompt")
