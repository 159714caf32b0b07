#!/usr/bin/env python3
"""bench.py — decode tokens/s of the GGUF-quantised hot path on B200 (BASELINE.json metric).

A "step" is one batch-1 decode token of Llama-3-8B Q4_K_M (synthetic random-valid GGUF blocks of that
architecture — no weights ship with the reference and there is no network): the full node list libllama
emits for one token (32 layers + lm_head, 7 quantised matvecs / layer, rms_norm, rope, KV store,
flash-attention over an F16 KV cache), run on hand-written sm_100a kernels.

N = 1
  value        : tokens/s with every input resident in HBM (graph executor C-ABI, token feedback through an on-device argmax)
  e2e          : the PRODUCT PATH — the unmodified reference libllama (llama_decode loop, oracle/drivers/llama_drv.cpp bound
                 in-process with ctypes) driving libggml-b200.so through ggml's backend C-ABI on a synthetic GGUF of the same
                 shape: host token in, embedding row / positions / KV indices / mask uploaded by the scheduler, logits
                 read back to the host, host argmax — what llama-box does per token (httpserver.hpp:3591, :4285-4299)
  roofline     : the dominant kernel family (quantised matvec) timed IN SITU: the step's own node list with the attention
                 nodes left out (same fused launches, same in-kernel rms_norm + quantise prologues, residual epilogues, lm_head),
                 replayed as a CUDA graph; algorithmic weight bytes / CUDA-event time, against MEASURED_PEAKS.json
  cpu_baseline : the reference's own ggml-cpu path (oracle/_ref: unmodified libllama + libggml-cpu built from
                 /root/reference) on the box's host cores, same architecture / quant mix
  gpu_reference: (informational) the reference's own ggml-cuda backend (oracle/_ref_cuda, built unmodified for sm_100) on the
                 same GGUF through the same driver — the GPU bar to beat
  depth, prefill: (informational) the same metric at n_past ~3800, and prefill tok/s (config 3) through the product path
  --impl reference : the CPU path as its own arm (3 repeats, threads = CPUs this process may run on)

N > 1 (torchrun): the reference's LLAMA_SPLIT_MODE_LAYER through the product boundary: ONE process (rank 0) drives all N devices
with --tensor-split 1,..,1 at true batch 1 (libllama's scheduler hands the hidden state from device to device through the
plug-in's cpy_tensor_async = one cudaMemcpyPeerAsync over NVLink per boundary); the other ranks hold their GPU, join the
barriers and the max-over-ranks reduction.  At batch 1 the devices run one after the other, so tok/s cannot exceed the 1-GPU
figure (SURVEY.md §7); reported with the exposed handoff time per token.  The N-sequences-in-flight pipeline of round 1 is
kept as a separately named extra (`aggregate_pipeline`), never as the bs=1 metric.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "decode tok/s Llama-3-8B Q4_K_M bs=1"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="llama3-8b")
    ap.add_argument("--ftype", default="Q4_K_M")
    ap.add_argument("--kv", default="f16", choices=["f16", "q8_0"], help="KV cache type (-ctk / -ctv)")
    ap.add_argument("--ctx", type=int, default=4096)
    ap.add_argument("--n-past", type=int, default=512, help="KV positions already in the cache when decoding starts")
    ap.add_argument("--layers", type=int, default=0, help="override layer count (debug only; makes the number INVALID)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the informational legs (depth, prefill, gpu_reference, aggregate_pipeline)")
    ap.add_argument("--no-graphs", action="store_true")
    ap.add_argument("--no-fusion", action="store_true")
    ap.add_argument("--mega", action="store_true", help="experimental: attention as a phase of the persistent decode kernel")
    ap.add_argument("--mega-mmv", action="store_true", help="experimental: attention and the matvecs inside the persistent decode kernel")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (logits f32, next token) as DIR/<name>.npy; "
                    "the inputs are seeded, so two builds can be compared output for output (N = 1 only)")
    args = ap.parse_args()
    if args.dump_outputs and args.gpus > 1:
        ap.error("--dump-outputs is supported for --gpus 1 only")
    return args


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)"""

    def __init__(self, gpu_index=0):
        self.proc, self.lines, self.gpu, self.t_begin = None, [], gpu_index, None

    def start(self):
        q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", str(int(os.environ.get("B200_BENCH_CLOCK_MS", "100"))), "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def mark_begin(self):
        """the sampler is started before the warm-up (nvidia-smi needs ~0.1 s to produce its first line); samples taken
        from here on are the ones inside the timed region"""
        self.t_begin = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t_end = time.time()
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        inside = [ln for (t, ln) in self.lines if self.t_begin is None or self.t_begin <= t <= t_end + 0.02]
        window = "timed region"
        if not inside:                                   # region shorter than the sampling period: fall back to the loaded warm-up samples
            inside = [ln for (t, ln) in self.lines][-3:]; window = "warm-up (timed region shorter than one sample)"
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm), "window": window}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def kernel_traffic():
    """per-launch DRAM bytes of the dominant kernels from the round's committed `ncu --set full` capture
    (profiles/r2_kernel_traffic.json, written by tools/ncu_summarise.py from the .ncu-rep); None when absent"""
    p = os.path.join(ROOT, "profiles", "r2_kernel_traffic.json")
    try:
        return json.load(open(p))
    except (OSError, ValueError):
        return None


# ------------------------------------------------------------------------------------------------ synthetic GGUF + reference drivers
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
REF_CUDA = os.path.join(ROOT, "oracle", "_ref_cuda", "libggml-cuda.so")
PLUGIN = os.path.join(ROOT, "llama-box_b200", "libggml-b200.so")


def gguf_path(args):
    shm = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else "/tmp"
    return os.path.join(shm, f"b200_bench_{args.model}_{args.ftype}{'_L%d' % args.layers if args.layers else ''}.gguf")


def ensure_gguf(args):
    path = gguf_path(args)
    if os.path.exists(path):
        return path
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "make_gguf.py"), "--config", args.model, "--ftype", args.ftype, "--out", path + ".tmp%d" % os.getpid()]
    if args.layers:
        cmd += ["--layers", str(args.layers)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stderr[-2000:]); return None
    os.replace(path + ".tmp%d" % os.getpid(), path)
    return path


def host_threads():
    """threads for the ggml-cpu arm: the CPUs this process may actually run on (a cgroup / affinity-limited lease reports far
    fewer than os.cpu_count(), and oversubscribing ggml-cpu's spinning thread pool is what made round 1's CPU arm swing 5x
    between boxes); capped at 64 — decode is memory-bound and ggml-cpu's per-op barrier cost grows with the thread count"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(n, 64)), n


def drv_subprocess(args, plugin, ngl, prompt_len, gen, threads=8, repeat=1, extra=(), timeout=900):
    """oracle/_ref/llama_drv in its own process (CPU arm, and the reference's ggml-cuda leg: two GPU backends never share a process)"""
    drv = os.path.join(REF_DIR, "llama_drv")
    path = ensure_gguf(args)
    if not os.path.exists(drv) or path is None:
        return None
    env = dict(os.environ, LD_LIBRARY_PATH=REF_DIR + ":" + os.environ.get("LD_LIBRARY_PATH", ""))
    env.pop("GGML_BACKEND_PATH", None)
    cmd = [drv, "--model", path, "--ngl", str(ngl), "--threads", str(threads), "--ctx", str(args.ctx), "--prompt-len", str(prompt_len), "--gen", str(gen),
           "--repeat", str(repeat), "--fa", "--ctk", args.kv, "--ctv", args.kv] + list(extra)
    if plugin:
        cmd += ["--plugin", plugin]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=timeout)
    except subprocess.TimeoutExpired:
        return {"error": "timeout"}
    if r.returncode != 0:
        return {"error": (r.stderr or r.stdout)[-400:]}
    return json.loads(r.stdout.strip().splitlines()[-1])


def cpu_reference(args, gen, prompt_len, repeat=1):
    """the UNMODIFIED reference on the host cores (ggml-cpu).  Returns dict(value, cores, sample, runs) or None."""
    threads, avail = host_threads()
    out = drv_subprocess(args, None, 0, prompt_len, gen, threads=threads, repeat=repeat, timeout=1500)
    if not out or "error" in out:
        if out:
            sys.stderr.write("cpu reference failed: %s\n" % out["error"])
        return None
    runs = sorted(out.get("decode_tps_runs") or [out["decode_tps"]])
    med = runs[len(runs) // 2]
    return dict(value=med, cores=threads, runs=runs,
                sample=f"{repeat} x {gen - 1} greedy decode tokens after a {prompt_len}-token prompt, {args.model} {args.ftype} synthetic GGUF, -fa, {args.kv} KV, "
                       f"ggml-cpu {threads} threads ({avail} CPUs in this process's affinity mask, os.cpu_count() = {os.cpu_count()}); median of the repeats")


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.time()
    res = cpu_reference(args, gen=max(2, args.steps + 1), prompt_len=args.n_past, repeat=3)
    if res is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/llama_drv (reference build) or gguf generation missing on this box"}))
        return
    tps = res["value"]
    line = {"metric": METRIC, "value": tps, "unit": "tok/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 / tps if tps else None, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "q4_K x q8_K int8 dot, f32 accumulate",
            "data": "synthetic", "impl": "reference",
            "config": workload_config(args, "ggml-cpu (unmodified reference build)"),
            "cpu_baseline": {"value": tps, "unit": "tok/s", "cores": res["cores"], "kind": "reference", "sample": res["sample"], "runs": res["runs"]},
            "e2e": {"value": tps, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0, "wall_s": time.time() - t0}
    print(json.dumps(line))


def workload_config(args, backend, **more):
    """the SAME dict for both arms (the driver compares them textually)"""
    cfg = {"workload": f"{args.model} {args.ftype} batch-1 decode, -c {args.ctx}, n_past {args.n_past}, {args.kv.upper()} KV, flash-attn", "backend": backend}
    cfg.update(more)
    return cfg


# ------------------------------------------------------------------------------------------------ product path (libllama + plug-in, in-process)
def product_decode(args, ts, n_past, steps, warmup, prefill_probe=0):
    """libllama's llama_decode loop over libggml-b200.so inside THIS process.  Returns a dict with tok/s measured (a) with CUDA
    events on device 0 around the loop and (b) by the wall clock, the per-step host<->device bytes, handoff statistics."""
    import numpy as np
    import torch
    from drvutil import Drv
    path = ensure_gguf(args)
    if path is None or not os.path.exists(PLUGIN):
        return None
    os.environ.setdefault("GGML_B200_HANDOFF_TIMING", "1")
    home = torch.cuda.current_device()
    d = Drv(path, plugin=PLUGIN, ngl=99, ts=ts, ctx=max(args.ctx, 4096), ubatch=512, threads=8, fa=True, ctk=args.kv, ctv=args.kv)
    try:
        rng = np.random.default_rng(42)
        V = d.n_vocab
        prompt = rng.integers(0, V, size=max(1, n_past)).tolist()
        t0 = time.perf_counter()
        for i in range(0, len(prompt), 2048):
            d.decode(prompt[i:i + 2048])
        lg = d.logits()
        tok = int(np.argmax(lg))
        prefill_s = time.perf_counter() - t0
        for _ in range(warmup):
            d.decode([tok]); tok = int(np.argmax(d.logits()))
        d.handoff_stats(reset=True)
        torch.cuda.set_device(home)                       # the plug-in switches the calling thread's current device as it walks the splits
        ndev = torch.cuda.device_count()
        for i in range(ndev):
            torch.cuda.synchronize(i)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        w0 = time.perf_counter()
        for _ in range(steps):
            d.decode([tok])                              # host token in; the scheduler uploads embedding row, pos, KV idx, mask
            tok = int(np.argmax(d.logits()))             # logits D2H (llama_get_logits_ith synchronises), greedy sampling on the host
        for i in range(ndev):
            torch.cuda.synchronize(i)
        wall = time.perf_counter() - w0
        torch.cuda.set_device(home)
        e1.record(); torch.cuda.synchronize()
        dev_ms = e0.elapsed_time(e1)
        hs = d.handoff_stats()
        n_kv = (d.n_past + 255) // 256 * 256
        out = {"tps_device": 1000.0 * steps / dev_ms, "tps_wall": steps / wall, "ms_per_step": 1000.0 * wall / steps, "n_past_end": d.n_past,
               "prefill_tps": len(prompt) / prefill_s, "n_devices": d.n_devices,
               # per step: embedding row f32[n_embd] + pos i32 + KV idx i64 x2 (K and V) + out id i32 + mask f32[n_kv x 64] up; logits down
               "h2d": d.n_embd * 4 + 4 + 16 + 4 + n_kv * 64 * 4, "d2h": V * 4, "handoff": hs}
        if prefill_probe:
            d.reset()
            pp = rng.integers(0, V, size=prefill_probe).tolist()
            d.decode(pp[:512]); d.sync(); d.reset()       # warm-up ubatch (graph shapes, workspace growth)
            t0 = time.perf_counter()
            for i in range(0, len(pp), 2048):
                d.decode(pp[i:i + 2048])
            d.logits()
            out["prefill_probe"] = {"n_tokens": prefill_probe, "tok_s": prefill_probe / (time.perf_counter() - t0), "ubatch": 512}
        return out
    finally:
        d.close()
        torch.cuda.set_device(home)


# ------------------------------------------------------------------------------------------------ GPU arm, N = 1
def run_b200(args):
    import torch
    import torch.distributed as dist
    from conftest import load_pkg
    pkg = load_pkg()
    import importlib
    G = importlib.import_module("llama_box_b200.graph"); M = importlib.import_module("llama_box_b200.model")
    ops = pkg.ops

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: there is no CPU fallback"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        return run_b200_multi(args, G, M, ops, rank, world, local)

    kvt = G.F16 if args.kv == "f16" else G.Q8_0
    model = M.SyntheticLlama(args.model, args.ftype, n_ctx=args.ctx, kv_type=kvt, n_layer=args.layers or None)
    ex = G.Executor(local)
    flags = (0 if args.no_graphs else G.EXEC_CUDA_GRAPHS) | (0 if args.no_fusion else G.EXEC_FUSION) | ((G.EXEC_MEGAKERNEL if (args.mega or args.mega_mmv) else 0) | (G.EXEC_MEGA_MMV if args.mega_mmv else 0) if not args.no_fusion else 0)
    stream = torch.cuda.Stream()
    hbm_peak, peak_src = peaks()

    res = device_resident_leg(args, model, ex, ops, G, stream, flags, args.n_past, args.steps, args.warmup, local, clocks=True, dump_dir=args.dump_outputs)
    tps, ms_per_step = res["tps"], res["ms_per_step"]

    # ---- roofline leg: the matvec launches of the step, in situ
    roof = mmvq_roofline_insitu(args, model, ex, ops, G, stream, flags, hbm_peak)
    roof["peak_source"] = peak_src
    roof["whole_step"] = whole_step(model, res, hbm_peak)
    roof["attention_and_rest_ms"] = ms_per_step - roof["ms_per_token_matvec_only"]

    depth = None
    if not args.no_extras and args.ctx >= 4096:
        n_deep = args.ctx - 2 * (32 + 8) - 40
        r2 = device_resident_leg(args, model, ex, ops, G, stream, flags, n_deep, 32, 4, local, clocks=False)
        depth = {"n_past": n_deep, "value": r2["tps"], "unit": "tok/s", "ms_per_step": r2["ms_per_step"], "whole_step": whole_step(model, r2, hbm_peak)}

    e2e_exec = None
    if not args.no_e2e:
        e2e_exec = run_e2e_executor(args, model, ex, ops, G, stream, flags, V=model.c["n_vocab"])

    # free the executor-level model before the product-path process state grows (both hold a full copy of the weights)
    launches, kernels_per_step, captures, replays = res["launches"], res["kernels_per_step"], int(ex.captures), int(ex.replays)
    del model, ex
    torch.cuda.empty_cache()

    # ---- e2e: the product path (libllama + libggml-b200.so through the ggml backend C-ABI), in this process
    e2e = None
    prefill = None
    if not args.no_e2e:
        pr = product_decode(args, "", args.n_past, args.steps, min(args.warmup, 8), prefill_probe=(0 if args.no_extras else 4096))
        if pr:
            e2e = {"value": pr["tps_wall"], "unit": "tok/s", "h2d_bytes_per_step": pr["h2d"], "d2h_bytes_per_step": pr["d2h"], "ms_per_step": pr["ms_per_step"],
                   "device_timed": pr["tps_device"],
                   "api": "llama_decode of the unmodified reference libllama (in-process, oracle/_ref/libllama_drv.so) over libggml-b200.so (ggml backend C-ABI): host token in, logits D2H, host argmax"}
            if "prefill_probe" in pr:
                prefill = {"metric": "prefill tok/s Llama-3-8B Q4_K_M, 4096-token prompt in 512-token ubatches (config 3)", "value": pr["prefill_probe"]["tok_s"], "unit": "tok/s",
                           "api": "llama_decode over libggml-b200.so", "first_prompt_tok_s": pr["prefill_tps"]}
        elif e2e_exec:
            e2e = dict(e2e_exec, note="product-path leg unavailable on this box (oracle/_ref or the plug-in missing): executor C-ABI with host buffers instead")

    # ---- CPU baseline (reference build on the host cores), bounded sample
    cpu = None
    if not args.no_cpu_baseline:
        r = cpu_reference(args, gen=17, prompt_len=min(args.n_past, 128), repeat=1)
        cpu = ({"value": r["value"], "unit": "tok/s", "cores": r["cores"], "kind": "reference", "sample": r["sample"]} if r else
               {"value": None, "unit": "tok/s", "cores": 0, "kind": "reference", "sample": "unavailable: oracle/_ref not present on this box"})

    # ---- the reference's own GPU backend (informational)
    gpu_ref = None
    if not args.no_extras and os.path.exists(REF_CUDA):
        o = drv_subprocess(args, REF_CUDA, 99, min(args.n_past, 512), 65, timeout=600)
        if o and "error" not in o:
            gpu_ref = {"decode_tok_s": o["decode_tps"], "prefill_tok_s": o["prefill_tps"], "backend": "ggml-cuda, unmodified, sm_100 build (oracle/_ref_cuda), CUDA graphs on, -fa",
                       "sample": "64 greedy tokens after a %d-token prompt, wall clock of llama_drv" % o["prompt_len"]}
            o2 = drv_subprocess(args, REF_CUDA, 99, 4096, 2, timeout=600)
            if o2 and "error" not in o2:
                gpu_ref["prefill_4096_tok_s"] = o2["prefill_tps"]
        else:
            gpu_ref = {"error": (o or {}).get("error", "unavailable")}

    line = {"metric": METRIC, "value": tps, "unit": "tok/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "q4_K/q6_K x q8_K int8 dot (dp4a), f32 accumulate", "data": "synthetic",
            "config": workload_config(args, "libggml-b200.so / libb200ops.so", n_layer=res["n_layer"], streamed_weight_bytes=res["weight_bytes"], kv_bytes_per_pos=res["kv_bytes_per_pos"],
                                      l2_policy="inputs (4.6 GB of weights per step) larger than L2; no flush needed", cuda_graphs=not args.no_graphs, fusion=not args.no_fusion,
                                      persistent_decode_kernel=("attention+matvec" if args.mega_mmv else ("attention" if args.mega else "off")), parallelism="single GPU"),
            "clocks": res["clocks"], "e2e": e2e, "e2e_executor": e2e_exec, "gpu_launches": int(launches), "kernels_per_step": int(kernels_per_step),
            "graph_captures": captures, "graph_replays": replays, "roofline": roof, "cpu_baseline": cpu,
            "depth": depth, "prefill": prefill, "gpu_reference": gpu_ref}
    if args.layers:
        line["config"]["INVALID"] = "layer count overridden (debug run)"
    print(json.dumps(line))


def whole_step(model, res, hbm_peak):
    b = res["weight_bytes"] + res["n_kv_mid"] * res["kv_bytes_per_pos"] + res["kv_bytes_per_pos"]
    ach = b / (res["ms_per_step"] * 1e-3) / 1e9
    return {"bytes": b, "achieved": ach, "unit": "GB/s", "frac": ach / hbm_peak, "frac_of_8TBs": ach / 8000.0}


def n_kv_of(pos):
    return max(256, (pos + 1 + 255) // 256 * 256)


def device_resident_leg(args, model, ex, ops, G, stream, flags, n_past, steps, warmup, local, clocks, dump_dir=None):
    """`value`: every input already in HBM — 3 tiny D2D copies + the token graph + on-device argmax feeding the next step.
    dump_dir: where to write the last timed step's logits and next token (see dump_outputs)"""
    import torch
    c = model.c
    V = c["n_vocab"]
    kvt = model.kv_type
    gen = torch.Generator(device="cuda"); gen.manual_seed(7)
    rowb = G.row_size(kvt, c["n_head_kv"] * c["head_dim"])
    for ly in model.layers:                           # KV cache content for the positions already "decoded"
        for key in ("k_cache", "v_cache"):
            if kvt == G.F16:
                n = n_past * rowb // 2
                ly[key].view(torch.float16)[:n] = (torch.randn(n, device="cuda", generator=gen) * 0.5).half()
            else:                                     # q8_0 rows: random int8 + a sane f16 scale per 34-byte block
                nb = n_past * rowb // 34
                blk = torch.randint(0, 256, (nb, 34), dtype=torch.uint8, device="cuda", generator=gen)
                blk[:, 0:2] = (torch.rand(nb, device="cuda", generator=gen) * 0.01 + 0.002).half().view(torch.uint8).reshape(nb, 2)
                ly[key][:nb * 34] = blk.reshape(-1)
    total = warmup + steps
    assert n_kv_of(n_past + total + 2) <= args.ctx, "ctx too small for n_past + steps"
    pos_dev = torch.arange(n_past, n_past + total + 2, dtype=torch.int32, device="cuda")
    idx_dev = pos_dev.to(torch.int64)
    graphs, mask_dev = {}, {}

    def nodes_for(n_kv):
        if n_kv not in graphs:
            graphs[n_kv] = model.build(1, n_kv)
        return graphs[n_kv]

    def device_step(i):
        pos = n_past + i
        nodes, io = nodes_for(n_kv_of(pos))
        io["pos"].copy_(pos_dev[i:i + 1], non_blocking=True)
        io["kv_idx"].copy_(idx_dev[i:i + 1], non_blocking=True)
        io["mask"][0].copy_(mask_dev[i], non_blocking=True)
        ex.compute(nodes, flags, stream=C.c_void_p(stream.cuda_stream))
        ops.check(ops.lib.b200_argmax_f32(ops.p(io["logits"]), ops.p(io["tokens"]), V, 1, C.c_void_p(stream.cuda_stream)))
        return io

    with torch.cuda.stream(stream):
        for i in range(total + 1):
            pos = n_past + i
            m = torch.full((n_kv_of(pos),), float("-inf")); m[:pos + 1] = 0
            mask_dev[i] = m.cuda()
        nodes, io = nodes_for(n_kv_of(n_past))
        io["tokens"].fill_(1); io["out_ids"].fill_(0)
        sampler = ClockSampler(local) if clocks else None
        if sampler:
            sampler.start()
        for i in range(warmup):
            device_step(i)
        stream.synchronize()
        if sampler:
            sampler.mark_begin()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ops.lib.b200_kernel_launches()
        torch.cuda.synchronize()
        e0.record(stream)
        for i in range(warmup, total):
            last_io = device_step(i)
        e1.record(stream)
        torch.cuda.synchronize()
        launches = ops.lib.b200_kernel_launches() - l0
        ms = e0.elapsed_time(e1)
        clk = sampler.stop() if sampler else None
    if dump_dir and steps > 0:
        dump_outputs(dump_dir, last_io)
    ms_per_step = ms / steps
    return {"tps": 1000.0 / ms_per_step, "ms_per_step": ms_per_step, "launches": launches, "kernels_per_step": ex.last_kernels + 1, "clocks": clk,
            "weight_bytes": model.streamed_weight_bytes(), "kv_bytes_per_pos": model.kv_bytes_per_pos(), "n_kv_mid": n_kv_of(n_past + warmup + steps // 2), "n_layer": len(model.layers)}


def dump_outputs(out_dir, io):
    """What a caller of the timed decode step receives: the logits of the step (f32 [1, n_vocab], 0.5 MB for Llama-3's
    vocabulary) and the greedy next token the on-device argmax fed back (as f64, exact).  Written after the timing."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "logits.npy"), io["logits"].float().cpu().numpy())
    np.save(os.path.join(out_dir, "next_token.npy"), io["tokens"].cpu().numpy().astype(np.float64))


def mmvq_roofline_insitu(args, model, ex, ops, G, stream, flags, hbm_peak):
    """the quantised matvec launches of one decode token exactly as the step issues them: the step's node list without the
    attention nodes (same QKV / wo+residual / gate+up+SwiGLU / down+residual / lm_head launches with their in-kernel
    rms_norm + quantise prologues), replayed by the executor as a CUDA graph; CUDA events on the launching stream.
    The 4.6 GB working set defeats L2 between launches."""
    import torch
    st = C.c_void_p(stream.cuda_stream)
    nodes, io = model.build(1, 256, skip_attention=True)
    with torch.cuda.stream(stream):
        io["tokens"].fill_(1); io["out_ids"].fill_(0)
        for _ in range(4):
            ex.compute(nodes, flags, stream=st)          # eager once, capture, replay
        stream.synchronize()
        nl = ex.last_kernels
        reps = 10
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            ex.compute(nodes, flags, stream=st)
        e1.record(stream)
        stream.synchronize()
    ms = e0.elapsed_time(e1) / reps
    wbytes = sum(sum(ly[k].nbytes for k in ("wq", "wk", "wv", "wo", "gate", "up", "down")) for ly in model.layers) + model.output.nbytes
    ach = wbytes / (ms * 1e-3) / 1e9
    traffic, src = None, "no committed ncu capture for this round yet (profiles/r2_kernel_traffic.json)"
    kt = kernel_traffic()
    if kt and "mmvq_per_token_dram_bytes" in kt:
        traffic, src = int(kt["mmvq_per_token_dram_bytes"]), kt.get("source", "profiles/r2_kernel_traffic.json")
    return {"bound": "hbm", "kernel": "quantised matvec launches of one token, in situ (mmvq_kernel + the lm_head launch; %d kernels incl. the embedding gather)" % nl,
            "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "frac_of_8TBs": ach / 8000.0, "traffic": traffic, "traffic_source": src,
            "bytes_per_token": wbytes, "launches_per_token": int(nl), "avg_launch_us": ms * 1e3 / max(1, nl), "ms_per_token_matvec_only": ms}


def run_e2e_executor(args, model, ex, ops, G, stream, flags, V):
    """secondary end-to-end figure at the kernel library's own C-ABI (b200_executor_compute): pinned host inputs, logits D2H, host argmax"""
    import torch
    st = C.c_void_p(stream.cuda_stream)
    total = args.warmup + args.steps
    base = args.n_past + total + 2
    n_kv_max = n_kv_of(base + total + 8)
    if n_kv_max > args.ctx:
        return None
    h_tok = torch.zeros(1, dtype=torch.int32).pin_memory(); h_pos = torch.zeros(1, dtype=torch.int32).pin_memory(); h_idx = torch.zeros(1, dtype=torch.int64).pin_memory()
    h_mask = torch.full((n_kv_max,), float("-inf")).pin_memory(); h_logits = torch.zeros(V).pin_memory()
    h_tok[0] = 1
    graphs = {}

    def step(i):
        pos = base + i
        n_kv = n_kv_of(pos)
        if n_kv not in graphs:
            graphs[n_kv] = model.build(1, n_kv)
        nodes, io = graphs[n_kv]
        h_pos[0] = pos; h_idx[0] = pos; h_mask[:n_kv].fill_(float("-inf")); h_mask[:pos + 1] = 0
        with torch.cuda.stream(stream):
            io["tokens"].copy_(h_tok, non_blocking=True); io["pos"].copy_(h_pos, non_blocking=True); io["kv_idx"].copy_(h_idx, non_blocking=True)
            io["mask"][0].copy_(h_mask[:n_kv], non_blocking=True)
            ex.compute(nodes, flags, stream=st)
            h_logits.copy_(io["logits"][0], non_blocking=True)
        stream.synchronize()
        h_tok[0] = int(torch.argmax(h_logits))
        return 4 + 4 + 8 + n_kv * 4, V * 4
    for i in range(min(args.warmup, 4)):
        step(i)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0.record(stream)
    h2d = d2h = 0
    n = args.steps
    for i in range(min(args.warmup, 4), min(args.warmup, 4) + n):
        a, b = step(i); h2d += a; d2h += b
    e1.record(stream)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ms = max(e0.elapsed_time(e1), wall * 1e3) / n
    return {"value": 1000.0 / ms, "unit": "tok/s", "h2d_bytes_per_step": h2d // n, "d2h_bytes_per_step": d2h // n, "ms_per_step": ms,
            "api": "b200_executor_compute (C-ABI, include/b200_graph.h) with pinned host inputs, logits D2H, host argmax"}


# ------------------------------------------------------------------------------------------------ GPU arm, N > 1
def run_b200_multi(args, G, M, ops, rank, world, local):
    """N > 1: the product boundary with --tensor-split over the N devices of this box, true batch 1, driven from rank 0."""
    import torch
    import torch.distributed as dist
    hbm_peak, peak_src = peaks()
    line = None
    # The other ranks must WAIT ON THE CPU while rank 0 drives every device through libllama: an NCCL barrier is a kernel spinning on
    # their GPU, and the product path's layers on that GPU would time-slice against it (measured: 80 tok/s instead of ~500).
    cpu_group = dist.new_group(backend="gloo")
    dist.barrier()
    torch.cuda.synchronize()
    if rank == 0:
        sampler = ClockSampler(0); sampler.start()
        one = product_decode(args, ",".join(["1"] + ["0"] * (world - 1)), args.n_past, args.steps, min(args.warmup, 8))    # all layers on device 0, same process
        sampler.mark_begin()
        multi = product_decode(args, ",".join(["1"] * world), args.n_past, args.steps, min(args.warmup, 8))
        clocks = sampler.stop()
        if multi is None:
            line = {"metric": METRIC, "value": None, "unit": "tok/s", "n_gpus": world, "error": "product path unavailable (oracle/_ref or plug-in missing)"}
        else:
            hs = multi["handoff"] or {}
            cps = hs.get("copies", 0) / max(1, args.steps)
            exposed = (multi["ms_per_step"] - one["ms_per_step"]) * 1e3 if one else None
            # bytes one token streams: weights once (spread over the devices) + KV of its position
            cfg = M.CONFIGS[args.model]; L = args.layers or cfg["n_layer"]
            kvrow = 2 * L * G.row_size(G.F16 if args.kv == "f16" else G.Q8_0, cfg["n_head_kv"] * cfg["head_dim"])
            wb = weight_bytes_of(M, G, ops, args)
            step_bytes = wb + n_kv_of(args.n_past + args.steps // 2) * kvrow
            ach = step_bytes / (1e-3 * 1000.0 / multi["tps_device"]) / 1e9
            line = {"metric": METRIC, "value": multi["tps_device"], "unit": "tok/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                    "ms_per_step": 1000.0 / multi["tps_device"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                    "dtype": "q4_K/q6_K x q8_K int8 dot (dp4a), f32 accumulate", "data": "synthetic",
                    "config": workload_config(args, "libggml-b200.so through the unmodified libllama (one process, %d devices)" % world,
                                              parallelism=f"layer split, --tensor-split {','.join(['1'] * world)} (LLAMA_SPLIT_MODE_LAYER), true batch 1: devices run one after the other",
                                              l2_policy="inputs larger than L2"),
                    "clocks": clocks,
                    "e2e": {"value": multi["tps_wall"], "unit": "tok/s", "h2d_bytes_per_step": multi["h2d"], "d2h_bytes_per_step": multi["d2h"], "ms_per_step": multi["ms_per_step"],
                            "api": "llama_decode of the unmodified reference libllama (in-process) over libggml-b200.so, --tensor-split over %d devices; wall clock incl. host sampling" % world},
                    "handoff": {"copies_per_token": cps, "bytes_per_copy": (hs.get("bytes", 0) / hs["copies"]) if hs.get("copies") else None,
                                "device_us_per_copy": (hs.get("device_us", 0.0) / hs["copies"]) if hs.get("copies") else None,
                                "host_us_per_copy": (hs.get("host_us", 0.0) / hs["copies"]) if hs.get("copies") else None,
                                "exposed_us_per_token": exposed,
                                "how": "device_us: CUDA events around cudaMemcpyPeerAsync on the source stream; exposed: ms/token with --ts over N devices minus ms/token with every layer on device 0, same process, same run"},
                    "single_device_same_process": {"value": one["tps_device"], "ms_per_step": 1000.0 / one["tps_device"]} if one else None,
                    "gpu_launches": int(ops.lib.b200_kernel_launches()),
                    "roofline": {"bound": "hbm", "kernel": "whole decode step (devices run serially at batch 1)", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                                 "traffic": None, "peak_source": peak_src + " (one device streams at a time)"},
                    "cpu_baseline": None}
    # every rank: barrier + max over ranks of the timed region (ranks other than 0 contribute 0: they only hold their device)
    torch.cuda.set_device(local)
    dist.barrier(group=cpu_group)
    t = torch.tensor([line["ms_per_step"] if (line and line.get("value")) else 0.0], device=torch.device("cuda", local))
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    agg = None
    if not args.no_extras:
        agg = run_b200_pipeline(args, G, M, ops, rank, world, local)
    if rank == 0:
        line["aggregate_pipeline"] = agg
        print(json.dumps(line))
    dist.barrier()
    dist.destroy_process_group()


def weight_bytes_of(M, G, ops, args):
    cfg = M.CONFIGS[args.model]; L = args.layers or cfg["n_layer"]
    mix, out_t = M.type_mix(args.ftype, L, cfg["n_ff"], args.model == "qwen2-72b")
    E, H, HK, D, FF, V = cfg["n_embd"], cfg["n_head"], cfg["n_head_kv"], cfg["head_dim"], cfg["n_ff"], cfg["n_vocab"]
    b = V * ops.row_bytes(out_t, E)
    for t in mix:
        b += H * D * ops.row_bytes(t["wq"], E) + HK * D * (ops.row_bytes(t["wk"], E) + ops.row_bytes(t["wv"], E)) + E * ops.row_bytes(t["wo"], H * D)
        b += FF * (ops.row_bytes(t["gate"], E) + ops.row_bytes(t["up"], E)) + E * ops.row_bytes(t["down"], FF)
    return b


def run_b200_pipeline(args, G, M, ops, rank, world, local):
    """(extra, separately named) `world` independent sequences in flight over the same layer split, one process per GPU:
    rank r owns a contiguous range of layers and their KV; the hidden state [n_embd] f32 goes to rank r+1 with one NCCL
    send/recv per boundary, the sampled token back to rank 0.  Schedule = llama-box_b200/pipeline.py (covered on CPU by
    tests/test_pipeline_gloo.py).  Value = tokens leaving the last stage per second, ALL sequences — an aggregate-throughput
    figure, not the bs=1 metric."""
    import importlib
    import torch
    import torch.distributed as dist
    P = importlib.import_module("llama_box_b200.pipeline")
    full = M.CONFIGS[args.model]
    L = args.layers or full["n_layer"]
    lo, hi = P.layer_range(rank, world, L)
    first, last = rank == 0, rank == world - 1
    kvt = G.F16 if args.kv == "f16" else G.Q8_0
    model = M.SyntheticLlama(args.model, args.ftype, n_ctx=args.ctx, kv_type=kvt, n_layer=L, layer_range=(lo, hi), first=first, last=last, n_seq=world)
    c = model.c
    V = c["n_vocab"]
    if kvt == G.F16:
        gen = torch.Generator(device="cuda"); gen.manual_seed(7 + rank)
        for ly in model.layers:
            for caches in (ly["k_caches"], ly["v_caches"]):
                for cache in caches:
                    n = args.n_past * G.row_size(G.F16, c["n_head_kv"] * c["head_dim"]) // 2
                    cache.view(torch.float16)[:n] = (torch.randn(n, device="cuda", generator=gen) * 0.5).half()
    ex = G.Executor(local)
    flags = (0 if args.no_graphs else G.EXEC_CUDA_GRAPHS) | (0 if args.no_fusion else G.EXEC_FUSION)
    steps, warm = args.steps, args.warmup
    total_ticks = warm + world - 1 + steps
    steps_per_seq = (total_ticks + world - 1) // world + 1
    assert n_kv_of(args.n_past + steps_per_seq) <= args.ctx
    stream = torch.cuda.current_stream()
    st = C.c_void_p(stream.cuda_stream)
    graphs = {}
    neg = torch.full((n_kv_of(args.n_past + steps_per_seq),), float("-inf"), device="cuda")
    tok = torch.ones(1, dtype=torch.int32, device="cuda")
    seq_pos = [args.n_past] * world

    def stage(seq, inp, t):
        pos = seq_pos[seq]; seq_pos[seq] += 1
        n_kv = n_kv_of(pos)
        key = (n_kv, seq)
        if key not in graphs:
            graphs[key] = model.build(1, n_kv, seq=seq)
        nodes, io = graphs[key]
        if first:
            io["tokens"].copy_(inp if inp is not None else tok)
        io["pos"].fill_(pos); io["kv_idx"].fill_(pos)
        m = neg[:n_kv].clone(); m[:pos + 1] = 0
        io["mask"][0].copy_(m)
        ex.compute(nodes, flags, stream=st)
        if last:
            ops.check(ops.lib.b200_argmax_f32(ops.p(io["logits"]), ops.p(tok), V, 1, st))
            return tok
        return io["hidden_out"]

    hidden_in = model._buf("hidden_in", [1, c["n_embd"]])      # the same buffer in every node list of this stage

    def recv(src):
        buf = tok if first else hidden_in
        dist.recv(buf, src=src)
        return buf

    def send(x, dst):
        return dist.isend(x.clone(), dst=dst)                    # the stage overwrites its output buffer on the next tick

    class Timer:
        def __init__(self):
            self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tm = Timer()
    marks = {"t0": warm + world - 1}

    def stage_timed(seq, inp, t):
        if t == marks["t0"]:
            torch.cuda.synchronize(); tm.e0.record(stream)
        return stage(seq, inp, t)
    dist.barrier()
    P.run(rank, world, total_ticks, stage_timed, recv, send)
    tm.e1.record(stream)
    torch.cuda.synchronize()
    # ranks that never reached tick t0 inside stage_timed (cannot happen: every rank runs every tick >= rank) would have no e0
    ms = torch.tensor([tm.e0.elapsed_time(tm.e1)], device="cuda")
    dist.barrier()
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    del model, ex
    torch.cuda.empty_cache()
    ms_per_tick = float(ms.item()) / steps
    return {"metric": "aggregate decode tok/s, %d sequences in flight (one per pipeline stage), Llama-3-8B Q4_K_M" % world, "value": 1000.0 / ms_per_tick, "unit": "tok/s",
            "ms_per_tick": ms_per_tick, "note": "NOT the bs=1 metric: every GPU streams its 1/N slice of the weights for a different sequence each tick; "
            "one process per GPU, NCCL send/recv of the hidden state, schedule in llama-box_b200/pipeline.py"}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference_arm(args)
    run_b200(args)


if __name__ == "__main__":
    main()
