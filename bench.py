#!/usr/bin/env python
"""bench.py — the hot-path benchmark (driver contract: python bench.py --gpus N --steps K --warmup W).

Workload (BASELINE.json `metric`): Llama-3-8B geometry (32 layers, 32 q heads, 8 kv heads, D=128), 32K-token
prompt, PyramidKV budget 128 (window 8, kernel 7, maxpool — the reference runners' knobs, run_longbench.py:219-237),
bf16, synthetic N(0,1) Q/K/V of that shape (no checkpoints offline). One STEP = the eviction of one prompt:
all 32 layers' `update_kv` (window scoring -> pool -> per-layer pyramidal top-k -> K/V gather-compact).

  value      = ms per step with Q/K/V already resident in HBM (CUDA events, max over ranks)
  e2e        = the same through the reference-facing plugin call `PyramidKVCluster.update_kv` with pinned HOST
               buffers: H2D of K/V/Q-window and D2H of the compacted K/V inside the timed region
  roofline   = the dominant kernel (the K scan / window-score kernel): algorithmic bytes Hkv*S*D*2 per launch
               / its CUDA-event duration, against MEASURED_PEAKS.json's hbm_gbs
  cpu_baseline = the reference op chain (oracle/torch_chain.py, bit-identical restatement of update_kv incl.
               repeat_kv) on this box's host cores, bounded sample, rank 0 only
  --impl reference = only that CPU arm, same JSON contract.
N>1: weak scaling, one independent prompt per rank, no data-path collective (the path shards by prompt/layer/head).
--workload 70b runs the layer-sharded Llama-3-70B configuration (configs[4]) with the NVLink hand-off.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (layers, Hq, Hkv, D, S, budget, window, kernel, pooling)
    "llama3-8b-32k-b128": (32, 32, 8, 128, 32768, 128, 8, 7, "maxpool"),
    "llama3-8b-8k-b128": (32, 32, 8, 128, 8192, 128, 8, 7, "maxpool"),
    "llama3-8b-32k-b2048": (32, 32, 8, 128, 32768, 2048, 8, 7, "maxpool"),
    "llama3-70b-32k-b2048": (80, 64, 8, 128, 32768, 2048, 8, 7, "maxpool"),
    "llama3-8b-128k-b128": (8, 32, 8, 128, 131072, 128, 8, 7, "maxpool"),     # 8 layers only (memory); timing experiments
}
DEFAULT_WORKLOAD = "llama3-8b-32k-b128"
METRIC = "prefill+evict ms"


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    return rank, world, local


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clock / throttle sampling DURING the timed regions (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,utilization.gpu,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.gpu, self.proc = gpu_index, None
        self.path = tempfile.mktemp(prefix="pkv_clocks_", suffix=".csv")

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9 or not f[1].isdigit():
                    continue
                util = int(f[4]) if f[4].isdigit() else 0
                if util > 0:
                    sm.append(int(f[1]))
                smax = int(f[2]) if f[2].isdigit() else smax
                for nm, v in zip(names, f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            os.unlink(self.path)
        except OSError:
            pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples_under_load": len(sm)}


def make_config(workload, method, n_gpus):
    """The workload description BOTH arms print (the driver compares the two `config` dicts)."""
    L, Hq, Hkv, D, S, B, W, ks, pool = WORKLOADS[workload]
    return {"workload": f"{workload}: Llama-3-8B geometry, {method}, {L} layers x update_kv per step" if "8b" in workload else workload,
            "seq_len": S, "budget": B, "window": W, "kernel_size": ks, "pooling": pool, "method": method,
            "layers": L, "q_heads": Hq, "kv_heads": Hkv, "head_dim": D,
            "l2": f"inputs larger than L2: {2 * L * Hkv * S * D * 2 / 2**30:.1f} GiB of distinct K/V per step (L2 = 126 MB), no flush needed",
            "parallelism": f"{n_gpus} independent prompts, one per GPU" if n_gpus > 1 else "1 GPU"}


def budgets(workload):
    from pyramidkv_b200 import ops
    L, Hq, Hkv, D, S, B, W, ks, pool = WORKLOADS[workload]
    return [ops.layer_budget("pyramidkv", B, W, L, l, S)[1] for l in range(L)]


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_arm(workload, steps, warmup, sample_layers=4, method="pyramidkv", budget_s=150.0):
    """The reference op chain on host cores (torch CPU kernels). One step = `sample_layers` REAL layers of the workload
    (spread over the pyramid); the reported value is that time scaled to the whole prompt (x L / sample_layers, flagged
    `extrapolated`). The thread count is swept first (torch's bf16 CPU GEMMs degrade badly when over-subscribed) and the
    best setting is used; the sample shrinks if `steps` of it would not fit `budget_s` seconds."""
    from oracle import torch_chain as tc
    L, Hq, Hkv, D, S, B, W, ks, pool = WORKLOADS[workload]
    cores = os.cpu_count() or 1
    g = torch.Generator().manual_seed(0)
    q = torch.randn(1, Hq, S, D, generator=g).bfloat16()
    k = torch.randn(1, Hkv, S, D, generator=g).bfloat16()
    v = torch.randn(1, Hkv, S, D, generator=g).bfloat16()

    def layer(l):   # repeat_kv is part of the reference's path (llama_model.py:158-159)
        tc.update_kv(method, tc.repeat_kv(k, Hq // Hkv), q, tc.repeat_kv(v, Hq // Hkv), W, B, ks, pool, L, l)

    sweep = {}
    for nt in sorted({n for n in (16, 32, 64, 128, cores) if n <= cores} or {cores}):
        torch.set_num_threads(nt)
        layer(0)
        t0 = time.perf_counter()
        layer(L // 2)
        sweep[nt] = time.perf_counter() - t0
    best = min(sweep, key=sweep.get)
    torch.set_num_threads(best)
    t_layer = sweep[best]
    while sample_layers > 1 and (steps + warmup) * sample_layers * t_layer > budget_s:
        sample_layers -= 1
    layers = [(i * L) // sample_layers for i in range(sample_layers)]

    def step():
        for l in layers:
            layer(l)

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    ms_prompt = dt * 1e3 * L / sample_layers
    return {"value": ms_prompt, "unit": "ms", "cores": best, "host_cores": cores, "kind": "port", "extrapolated": True,
            "measured_s_per_step": dt, "sample_layers": sample_layers, "scale_factor": L / sample_layers,
            "thread_sweep_s_per_layer": {str(n): round(t, 4) for n, t in sweep.items()},
            "sample": f"layers {layers} of {L} per step x {steps} steps, scaled x{L / sample_layers:g}; torch {torch.__version__} CPU op chain "
                      f"(oracle/torch_chain.py == the reference's update_kv + repeat_kv, bit-identical), bf16, {best} threads (best of the sweep)"}


def gpu_chain_baseline(wl, layers=(0, 15, 31), reps=3):
    """The reference's op chain (repeat_kv x2 + update_kv as stock torch CUDA ops, oracle/torch_chain.py) on THIS GPU with
    the same inputs: the B-gpu-chain baseline of BASELINE.md. Extrapolated from a few layers to the whole prompt."""
    from oracle import torch_chain as tc
    G = wl.Hq // wl.Hkv
    S, W = wl.S, wl.W
    times = []
    for l in layers:
        if l >= wl.L:
            continue
        K = wl.K[l].permute(1, 0, 2)[None]        # [1, Hkv, S, D] view of the HF layout
        V = wl.V[l].permute(1, 0, 2)[None]
        if wl.method == "h2o":
            Q = wl.Qfull[l].permute(1, 0, 2)[None]
        else:
            Q = torch.zeros(1, wl.Hq, S, wl.D, dtype=torch.bfloat16, device=wl.dev)
            Q[0, :, S - W:, :] = wl.Qw[l].permute(1, 0, 2)
        def run():
            tc.update_kv(wl.method, tc.repeat_kv(K, G), Q, tc.repeat_kv(V, G), W, wl.B, wl.ks, wl.pool, wl.L_model, l)
        run(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            run()
        e1.record(); torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) / reps)
        del Q
    per_layer = sum(times) / len(times)
    return {"ms_per_prompt": per_layer * wl.L, "ms_per_layer": per_layer, "sample": f"layers {list(layers)} x {reps} reps, extrapolated x{wl.L}",
            "what": "torch CUDA op chain == reference update_kv + repeat_kv (oracle/torch_chain.py), same inputs, same GPU"}


# ------------------------------------------------------------------------------------------------ GPU arm
class Workload:
    def __init__(self, name, device, score_kernel="auto", kv_layout="hf", method="pyramidkv", layers=0, layer_range=None, inputs_ready=True):
        from pyramidkv_b200 import ops
        self.name, self.method = name, method
        self.L, self.Hq, self.Hkv, self.D, self.S, self.B, self.W, self.ks, self.pool = WORKLOADS[name]
        self.dev = device
        self.L_model = self.L
        self.k_l = [ops.layer_budget(method, self.B, self.W, self.L, l, self.S)[1] for l in range(self.L)]
        if layers:
            self.L = min(self.L, layers)
            self.k_l = self.k_l[: self.L]
        if layer_range is not None:          # layer-sharded run: this rank owns layers [a, b) of the model
            a, b = layer_range
            self.k_l = self.k_l[a:b]
            self.L = b - a
        g = torch.Generator(device=device).manual_seed(1234 + (device.index or 0))
        L, S, Hkv, Hq, D, W = self.L, self.S, self.Hkv, self.Hq, self.D, self.W
        # HF physical layout [S, H, D] per layer (what q/k/v_proj(...).view().transpose(1, 2) produces)
        self.K = torch.empty(L, S, Hkv, D, dtype=torch.bfloat16, device=device)
        self.V = torch.empty(L, S, Hkv, D, dtype=torch.bfloat16, device=device)
        for l in range(L):
            self.K[l] = torch.randn(S, Hkv, D, generator=g, device=device, dtype=torch.float32).bfloat16()
            self.V[l] = torch.randn(S, Hkv, D, generator=g, device=device, dtype=torch.float32).bfloat16()
        if method == "h2o":   # H2O scores every query row: the whole Q is an input
            self.Qfull = torch.empty(L, S, Hq, D, dtype=torch.bfloat16, device=device)
            for l in range(L):
                self.Qfull[l] = torch.randn(S, Hq, D, generator=g, device=device, dtype=torch.float32).bfloat16()
            self.Qw = self.Qfull[:, S - W:]
        else:
            self.Qw = torch.randn(L, W, Hq, D, generator=g, device=device, dtype=torch.float32).bfloat16()   # window rows only
        self.kc = [torch.empty(Hq, k + W, D, dtype=torch.bfloat16, device=device) for k in self.k_l]
        self.vc = [torch.empty(Hq, k + W, D, dtype=torch.bfloat16, device=device) for k in self.k_l]
        if kv_layout == "head_major":     # experiment: physically [H, S, D] (contiguous per head) instead of HF's [S, H, D]
            self.K = self.K.permute(0, 2, 1, 3).contiguous().permute(0, 2, 1, 3)
            self.V = self.V.permute(0, 2, 1, 3).contiguous().permute(0, 2, 1, 3)
        qsrc = self.Qfull if method == "h2o" else self.Qw
        self.plans = [ops.plan_evict(method, qsrc[l].permute(1, 0, 2), self.K[l].permute(1, 0, 2), self.V[l].permute(1, 0, 2),
                                     W, self.k_l[l], self.kc[l], self.vc[l], self.ks, self.pool, score_kernel=score_kernel,
                                     inputs_ready=inputs_ready and os.environ.get("PKV_BENCH_INPUTS_READY", "1") != "0") for l in range(L)]
        # inputs_ready (PKV_FLAG_INPUTS_READY): Q/K/V of every layer are resident and no kernel in flight writes them, so the
        # K scan of a layer may start under the tail of the previous launch (programmatic dependent launch)
        # Layer batch (pkv_evict_prefill_batch): the same evictions, all layers in one pass — what the patched forward does
        # with pkv_defer_eviction (the default): every layer gets its own workspace, four launches per 32 layers.
        self.batch = None
        if method in ("pyramidkv", "snapkv") and L >= 2 and os.environ.get("PKV_BENCH_BATCH", "1") != "0":
            wss = ops.batch_workspaces(self.plans[0], L, max(self.k_l))
            bp = [ops.plan_evict(method, qsrc[l].permute(1, 0, 2), self.K[l].permute(1, 0, 2), self.V[l].permute(1, 0, 2),
                                 W, self.k_l[l], self.kc[l], self.vc[l], self.ks, self.pool, score_kernel=score_kernel,
                                 inputs_ready=inputs_ready and os.environ.get("PKV_BENCH_INPUTS_READY", "1") != "0", workspace=wss[l]) for l in range(L)]
            if ops.batch_supported(bp):
                self.batch = ops.EvictBatch(bp)

    def step(self, stage="all"):
        from pyramidkv_b200 import ops
        if stage == "batch":
            return self.batch.run()
        for p in self.plans:
            ops.run_stage(p, stage)

    def algorithmic_bytes(self):
        e = 2
        scan = self.Hkv * self.S * self.D * e + self.Hq * self.W * self.D * e
        rows = [4 * self.Hq * (k + self.W) * self.D * e for k in self.k_l]
        return scan, rows


def decode_bench(wl, gen=64):
    """Second half of BASELINE.json's metric (decode tok/s): `gen` decode steps over the compacted cache of every layer —
    pkv_decode_attn (append fused into the attention kernel) against the reference's op chain on the same GPU
    (repeat_kv + torch.cat + eager attention, llama_model.py:165-183). Attention path only: the model's GEMMs are not ours."""
    from oracle import torch_chain as tc
    from pyramidkv_b200 import ops
    dev, L, Hq, Hkv, D, W = wl.dev, wl.L, wl.Hq, wl.Hkv, wl.D, wl.W
    G = Hq // Hkv
    kc = [torch.zeros(Hq, k + W + gen, D, dtype=torch.bfloat16, device=dev) for k in wl.k_l]
    vc = [torch.zeros(Hq, k + W + gen, D, dtype=torch.bfloat16, device=dev) for k in wl.k_l]
    for l in range(L):
        kc[l][:, : wl.k_l[l] + W].copy_(wl.kc[l]); vc[l][:, : wl.k_l[l] + W].copy_(wl.vc[l])
    g = torch.Generator(device=dev).manual_seed(7)
    q = torch.randn(L, Hq, D, generator=g, device=dev, dtype=torch.float32).bfloat16()
    kn = torch.randn(L, Hkv, D, generator=g, device=dev, dtype=torch.float32).bfloat16()
    vn = torch.randn(L, Hkv, D, generator=g, device=dev, dtype=torch.float32).bfloat16()
    out = torch.empty(Hq, D, dtype=torch.bfloat16, device=dev)

    def ours():
        for t in range(gen):
            for l in range(L):
                ops.decode_attn(q[l], kc[l], vc[l], wl.k_l[l] + W + t + 1, kn[l], vn[l], out=out)

    def chain():
        K = [wl.kc[l][None] for l in range(L)]; V = [wl.vc[l][None] for l in range(L)]
        for t in range(gen):
            for l in range(L):
                K[l] = torch.cat([K[l], tc.repeat_kv(kn[l][None, :, None, :], G)], dim=2)
                V[l] = torch.cat([V[l], tc.repeat_kv(vn[l][None, :, None, :], G)], dim=2)
                tc.eager_decode_attn(q[l][None, :, None, :], K[l], V[l])

    res = {}
    for name, fn in (("host_launched_tok_s", ours), ("gpu_chain_tok_s", chain)):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        res[name] = gen / (e0.elapsed_time(e1) * 1e-3)
    # the same 32-layer step captured ONCE in a CUDA graph — the row count comes from a device counter
    # (pkv_decode_attn_graph) — and replayed per token: what pyramidkv_b200/generate.py's static loop does
    step = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = torch.empty(ops.decode_workspace_bytes(Hq, D), dtype=torch.uint8, device=dev)

    def one_step():
        for l in range(L):
            ops.decode_attn(q[l], kc[l], vc[l], wl.k_l[l] + W + 1, kn[l], vn[l], out=out, step=step, max_length=wl.k_l[l] + W + gen, workspace=ws)
        step.add_(1)

    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        one_step()
    torch.cuda.current_stream(dev).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        one_step()
    for _ in range(2):
        step.zero_()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _t in range(gen):
            graph.replay()
        e1.record()
        torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / gen
    res["value"] = 1e3 / ms_step
    bytes_step = sum(2 * Hq * (k + W + gen / 2) * D * 2 + 2 * Hq * D * 2 for k in wl.k_l)          # SURVEY.md 8d: bytes_decode(l, t), mean over t
    peak = peaks()[0]
    res["roofline"] = {"bound": "hbm (launch/latency-bound at this size)", "algorithmic_bytes_per_step": bytes_step, "us_per_step": ms_step * 1e3,
                       "achieved": bytes_step / (ms_step * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": bytes_step / (ms_step * 1e-3) / 1e9 / peak,
                       "note": f"{L} launches of decode_kernel (+ combine) per step, ~{bytes_step / L / 1e6:.1f} MB each, cache rows L2-resident across steps"}
    res.update({"unit": "tok/s", "what": f"{gen} decode steps x {L} layers of attention over the compacted cache (k_l + {W} + t rows per head), "
                "append fused; value = one CUDA-graph replay per step (the static generate loop), host_launched = one ctypes call per layer",
                "speedup_vs_gpu_chain": res["value"] / res["gpu_chain_tok_s"]})
    return res


DUMP_ROWS = 1 << 15     # --dump-outputs: K and V rows of D=128 float32 -> 2 x 16 MiB


def dump_outputs(wl, out_dir):
    """Writes what the last timed step returned: every layer's compacted K and V cache ([Hq, k_l + W, D] bf16), their rows
    concatenated over layers and heads ([sum_l Hq * (k_l + W), D]), as float32 (exact for bf16). Larger outputs are cut to
    DUMP_ROWS rows at the same seeded positions for K and V, so two builds can be compared row for row."""
    k = torch.cat([c.reshape(-1, wl.D) for c in wl.kc])
    v = torch.cat([c.reshape(-1, wl.D) for c in wl.vc])
    if k.shape[0] > DUMP_ROWS:
        rows = torch.randperm(k.shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values.to(k.device)
        k, v = k[rows], v[rows]
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "k_cache.npy"), k.float().cpu().numpy())
    np.save(os.path.join(out_dir, "v_cache.npy"), v.float().cpu().numpy())


def timed(fn, steps, barrier):
    barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    barrier()
    return e0.elapsed_time(e1) / steps


def sharded_70b_measure(workload, rank, world, device, barrier, steps, warmup, score_kernel="auto", kv_layout="hf", method="pyramidkv"):
    """BASELINE.json configs[4]: Llama-3-70B geometry, the reference's device_map-style contiguous layer sharding over the
    GPUs of one box (run_longbench.py:390). Each rank evicts its own layers (local work, no collective); the stage boundary
    hands the hidden state [S, 8192] bf16 to the next rank with one NCCL send/recv over NVLink. Strong scaling: total work
    is fixed; the pipeline is sequential for one prompt (like device_map=auto), so the hand-offs sit on the critical path.
    Returns a dict on rank 0 (times are MAX over ranks), None elsewhere."""
    import torch.distributed as dist
    from pyramidkv_b200 import _lib, ops
    from pyramidkv_b200.sharding import layer_ranges, max_over_ranks, run_pipeline
    L, Hq, Hkv, D, S, B, W, ks, pool = WORKLOADS[workload]
    a, b = layer_ranges(L, world)[rank]
    wl = Workload(workload, device, score_kernel, kv_layout, method, layer_range=(a, b))
    hidden = torch.randn(S, 8192, device=device, dtype=torch.float32).bfloat16()      # 512 MiB at 32K

    use_batch = wl.batch is not None     # the rank's layers in one pass, launched after its last layer (deferred eviction)

    def stage(l, h):
        if not use_batch:
            ops.run_stage(wl.plans[l - a], "all")
        elif l == b - 1:
            wl.batch.run()
        return h

    def step():
        run_pipeline(hidden if rank == 0 else None, hidden, L, stage)

    def step_one_prompt():       # nothing of the next prompt starts before this one has left the last rank
        step()
        torch.cuda.synchronize()
        barrier()

    for _ in range(max(warmup, 3)):
        step()
    l0 = _lib.launch_count()
    ms_pipelined = timed(step, steps, barrier)                  # back-to-back prompts: rank 0 starts prompt i+1 while rank 1 works on prompt i
    launches = (_lib.launch_count() - l0) // steps             # this rank's kernels per step
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step_one_prompt()
    ms = (time.perf_counter() - t0) * 1e3 / steps               # one prompt at a time, like device_map=auto (includes one barrier per prompt)
    ms_local = timed(wl.batch.run if use_batch else wl.step, steps, barrier)   # this rank's layers alone, no hand-off
    # one stage-boundary hand-off alone (rank 0 -> rank 1), device-timed on both ends
    def handoff():
        if rank == 0:
            dist.send(hidden, dst=1)
        elif rank == 1:
            dist.recv(hidden, src=0)
    for _ in range(2):
        handoff()
    ms_hand = timed(handoff, max(3, steps // 2), barrier)
    ms, ms_local_max, ms_hand, ms_pipelined = max_over_ranks([ms, ms_local, ms_hand, ms_pipelined], device)
    t = torch.tensor([ms_local, float(launches)], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    out = None
    if rank == 0:
        hb = int(hidden.numel() * 2)
        out = {"workload": f"{workload}: {L} layers sharded contiguously over {world} GPUs (device_map=auto style), one prompt",
               "evict_path": "layer batch per rank (four launches per 32 layers)" if use_batch else "three launches per layer",
               "ms": ms, "ms_pipelined_prompts": ms_pipelined, "layers_per_rank": [y - x for x, y in layer_ranges(L, world)],
               "evict_ms_sum_over_ranks": float(t[0]), "evict_ms_slowest_rank": ms_local_max,
               "handoff_ms": ms_hand, "handoff_bytes": hb, "handoff_gbps": hb / (ms_hand * 1e-3) / 1e9, "handoffs_per_step": world - 1,
               "handoff_share": (world - 1) * ms_hand / ms, "launches_per_step_all_ranks": int(t[1]),
               "note": "ms = ONE prompt at a time (like accelerate's device_map: one GPU busy at a time): sum of the ranks' eviction times + "
                       "(N-1) hand-offs of the [S, 8192] bf16 hidden state over NVLink (NCCL send/recv) + one barrier; ms_pipelined_prompts = "
                       "back-to-back prompts, stage r works on prompt i while stage r-1 works on prompt i+1; no data-path collective"}
    del wl, hidden
    torch.cuda.empty_cache()
    return out


def sharded_70b_arm(args, rank, world, device, barrier):
    """`--workload llama3-70b-32k-b2048` under torchrun: the layer-sharded configuration as the headline line."""
    import torch.distributed as dist
    r = sharded_70b_measure(args.workload, rank, world, device, barrier, args.steps, args.warmup, args.score_kernel, args.kv_layout, args.method)
    out = None
    if rank == 0:
        L, Hq, Hkv, D, S, B, W, ks, pool = WORKLOADS[args.workload]
        cfg = make_config(args.workload, args.method, world)
        cfg["parallelism"] = f"pp{world} (layer-sharded, sequential like device_map=auto)"
        out = {"metric": METRIC, "value": r["ms"], "unit": "ms", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
               "ms_per_step": r["ms"], "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
               "config": cfg, "sharded_70b": r, "gpu_launches": int(r["launches_per_step_all_ranks"] * args.steps)}
    dist.barrier()
    dist.destroy_process_group()
    return out


def whole_model_numbers(device, ctx=32768, budget=128, new_tokens=128, fused_rope=True):
    """The other two numbers of BASELINE.json's metric, through the plugin on the real architecture: prefill_total_ms (dense
    prefill + eviction of all 32 layers, HF forward with pyramidkv.monkeypatch.replace_llama) and whole-model decode tok/s
    (static loop: pre-reserved compacted cache, one CUDA-graph replay per token — pyramidkv_b200/generate.py — and the stock
    HF loop). Random-init Llama-3-8B (no checkpoints offline), synthetic prompt."""
    import contextlib
    import io
    import transformers
    from transformers.cache_utils import DynamicCache
    from pyramidkv.monkeypatch import replace_llama, restore
    from pyramidkv_b200.generate import StaticDecoder
    cfg = transformers.LlamaConfig(hidden_size=4096, intermediate_size=14336, num_hidden_layers=32, num_attention_heads=32,
                                   num_key_value_heads=8, head_dim=128, vocab_size=128256, rope_theta=5e5, max_position_embeddings=65536)
    cfg._attn_implementation = "sdpa"
    torch.manual_seed(42)
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.bfloat16)
    try:
        with torch.device(device):
            model = transformers.LlamaForCausalLM(cfg).eval()
    finally:
        torch.set_default_dtype(old)
    with contextlib.redirect_stdout(io.StringIO()):
        replace_llama("pyramidkv")
    try:
        for layer in model.model.layers:                         # run_longbench.py:253-261
            c = layer.self_attn.config
            c.window_size, c.max_capacity_prompt, c.kernel_size, c.pooling = 8, budget, 7, "maxpool"
        model.config.pkv_fused_rope = fused_rope          # f2: pkv_rope_inplace (bit-identical to HF's ten-launch op chain)
        ids = torch.randint(1, cfg.vocab_size, (1, ctx), generator=torch.Generator().manual_seed(0)).to(device)

        def prefill():
            cache = DynamicCache(config=model.config)
            out = model(input_ids=ids, past_key_values=cache, use_cache=True, logits_to_keep=1)
            return out.logits[:, -1].argmax(-1, keepdim=True), cache

        res = {"model": "llama3-8b (random init)", "ctx": ctx, "budget": budget, "new_tokens": new_tokens, "attn_implementation": "sdpa",
               "fused_rope": bool(fused_rope)}
        with torch.no_grad():
            prefill()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            tok, cache = prefill()
            e1.record()
            torch.cuda.synchronize()
            res["prefill_total_ms"] = e0.elapsed_time(e1)
            dec = StaticDecoder(model, cache, tok, max_steps=new_tokens + 3, use_graph=True)
            dec.run(3)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dec.run(new_tokens)
            e1.record()
            torch.cuda.synchronize()
            res["decode_tok_s"] = new_tokens / (e0.elapsed_time(e1) * 1e-3)
            res["decode_ms_per_tok"] = e0.elapsed_time(e1) / new_tokens
            res["decode_loop"] = "static (CUDA graph replay per token)"
            # stock HF loop for comparison (Python + launch overhead included: it is what generate() pays)
            tok2, cache2 = prefill()
            pos = ctx
            n_hf = 32
            for i in range(3 + n_hf):
                if i == 3:
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                out = model(input_ids=tok2, past_key_values=cache2, use_cache=True, position_ids=torch.tensor([[pos]], device=device))
                tok2 = out.logits[:, -1].argmax(-1, keepdim=True)
                pos += 1
            torch.cuda.synchronize()
            res["decode_tok_s_hf_loop"] = n_hf / (time.perf_counter() - t0)
        weight_bytes = sum(p.numel() * p.element_size() for p in model.parameters())
        res["decode_weight_floor_ms"] = weight_bytes / (peaks()[0] * 1e9) * 1e3
        return res
    finally:
        restore()
        del model
        torch.cuda.empty_cache()


def gpu_arm(args, rank, world, local):
    from pyramidkv_b200 import _lib, ops
    from pyramidkv_b200.kv_cluster import PyramidKVCluster
    _lib.lib()      # built by `python -m pyramidkv_b200.build`; the benchmark compiles nothing and writes nothing into the tree
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    use_dist = world > 1
    if use_dist:
        import torch.distributed as dist
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):   # keeps NCCL's version banner (env or /etc/nccl.conf) out of the one-JSON-line stdout
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=device)
        barrier = lambda: dist.barrier()
    else:
        barrier = lambda: None

    sharded = world > 1 and args.workload.startswith("llama3-70b")
    if sharded:
        if args.dump_outputs:
            raise SystemExit("bench.py: --dump-outputs is not available for the layer-sharded 70B run")
        return sharded_70b_arm(args, rank, world, device, barrier)
    wl = Workload(args.workload, device, args.score_kernel, args.kv_layout, args.method, args.layers)
    if args.profile_only:
        if args.stage not in ("all", "batch"):
            wl.step()                      # the later stages read what the earlier ones left in the workspace
        for _ in range(args.warmup + args.steps):
            wl.step(args.stage)
        torch.cuda.synchronize()
        return None
    fused_path = min(ops.single_launch(p) for p in wl.plans)   # 0 staged, 1 fused stages 1-2 + select kernel, 2 one launch per layer
    single = fused_path == 2
    sampler = ClockSampler(local)
    for _ in range(max(args.warmup, 3)):
        wl.step()
    torch.cuda.synchronize()
    sampler.start()

    # ---- value: whole-job, inputs resident in HBM ----
    n0 = _lib.launch_count()
    ms_step = timed(wl.step, args.steps, barrier)
    launches = (_lib.launch_count() - n0) // args.steps
    if args.dump_outputs and rank == 0 and wl.batch is None:
        dump_outputs(wl, args.dump_outputs)

    # ---- the layer batch: all layers in one pass (what the patched forward runs with pkv_defer_eviction) ----
    ms_batch, batch_ms, launches_batch = None, {}, 0
    if wl.batch is not None:
        for _ in range(3):
            wl.batch.run()
        n0 = _lib.launch_count()
        ms_batch = timed(wl.batch.run, args.steps, barrier)
        launches_batch = (_lib.launch_count() - n0) // args.steps
        if args.dump_outputs and rank == 0:        # before the stage timings below overwrite the caches
            dump_outputs(wl, args.dump_outputs)
        for st in ("scores", "pool", "select"):
            wl.batch.run(st)
            batch_ms[st] = timed(lambda s=st: wl.batch.run(s), max(3, args.steps // 2), barrier)

    # ---- the dominant kernel alone: the fused K scan + softmax + pool launch (or the staged K scan) ----
    ms_scanpool = None
    if fused_path >= 1:
        wl.step("scan_pool")
        ms_scanpool = timed(lambda: wl.step("scan_pool"), args.steps, barrier) / wl.L
    # ---- the staged kernels one by one ----
    wl.step("scores")
    ms_scores = timed(lambda: wl.step("scores"), args.steps, barrier) / wl.L   # per launch
    stage_ms = {"scores": ms_scores}
    for st in ("pool", "topk", "gather"):
        wl.step(st)
        stage_ms[st] = timed(lambda s=st: wl.step(s), max(3, args.steps // 2), barrier) / wl.L

    # ---- e2e: reference-facing plugin call with pinned host buffers ----
    L, Hq, Hkv, D, S, W = wl.L, wl.Hq, wl.Hkv, wl.D, wl.S, wl.W
    n_host = 4   # distinct pinned layer buffers, cycled (content does not affect copy time)
    hk = [wl.K[i % L].cpu().pin_memory().permute(1, 0, 2)[None] for i in range(n_host)]     # [1, Hkv, S, D], physically [S, Hkv, D]
    hv = [wl.V[i % L].cpu().pin_memory().permute(1, 0, 2)[None] for i in range(n_host)]
    hq = [torch.zeros(S, Hq, D, dtype=torch.bfloat16).pin_memory().permute(1, 0, 2)[None] for _ in range(n_host)]
    for i in range(n_host):
        if wl.method == "h2o":
            hq[i][0].copy_(wl.Qfull[i % L].permute(1, 0, 2).cpu())
        else:
            hq[i][0, :, S - W:, :] = wl.Qw[i % L].permute(1, 0, 2).cpu()
    from pyramidkv_b200 import kv_cluster as kvc
    if wl.method == "pyramidkv":
        clusters = [PyramidKVCluster(num_hidden_layers=wl.L_model, layer_idx=l, window_size=W, max_capacity_prompt=wl.B,
                                     kernel_size=wl.ks, pooling=wl.pool) for l in range(L)]
    else:
        cls = {"snapkv": kvc.SnapKVCluster, "h2o": kvc.H2OKVCluster, "streamingllm": kvc.StreamingLLMKVCluster}[wl.method]
        clusters = [cls(window_size=W, max_capacity_prompt=wl.B, kernel_size=wl.ks, pooling=wl.pool) for l in range(L)]
    d2h, h2d_c = [0], [0]

    def e2e_step():
        up = down = 0
        for l in range(L):
            clusters[l].update_kv(hk[l % n_host], hq[l % n_host], hv[l % n_host], None, Hq // Hkv)
        for l in range(L):
            up += clusters[l].last_h2d_bytes          # counted by the plugin from the tensors it actually copies
            down += clusters[l].last_d2h_bytes
        d2h[0], h2d_c[0] = down, up

    e2e_steps = max(2, min(args.steps, 5))
    if args.quick:      # A/B runs of the resident-HBM numbers only (not a valid bench line: no e2e, no baselines)
        ms_e2e, e2e_steps = 0.0, 0
    else:
        e2e_step()
        ms_e2e = timed(e2e_step, e2e_steps, barrier)
    h2d = h2d_c[0]
    clocks = sampler.stop()

    if use_dist:
        import torch.distributed as dist
        t = torch.tensor([ms_step, ms_e2e, ms_scores, ms_batch or 0.0, batch_ms.get("scores", 0.0)], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step, ms_e2e, ms_scores = t.tolist()[:3]
        if ms_batch is not None:
            ms_batch, batch_ms["scores"] = t.tolist()[3:]

    out = None
    if rank == 0:
        peak, peak_src = peaks()
        scan_bytes, row_bytes = wl.algorithmic_bytes()
        whole_bytes = L * scan_bytes + sum(row_bytes)
        whole_frac = whole_bytes / (ms_step * 1e-3) / 1e9 / peak
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("fused_kernel_dram_bytes_per_launch" if fused_path else "score_kernel_dram_bytes_per_launch")
        if single:
            # one launch per layer does everything: its average duration over the timed region IS the step time / L
            per_launch_bytes = whole_bytes / L
            us_launch = ms_step * 1e3 / L
            roof = {"bound": "hbm", "kernel": "evict_fused_kernel (K scan + softmax + pool + select + gather: the whole eviction of a layer in one launch)",
                    "achieved": per_launch_bytes / (us_launch * 1e-6) / 1e9, "peak": peak, "unit": "GB/s",
                    "frac": per_launch_bytes / (us_launch * 1e-6) / 1e9 / peak, "whole_step_frac": whole_frac, "traffic": traffic,
                    "algorithmic_bytes_per_launch": per_launch_bytes, "us_per_launch": us_launch, "peak_source": peak_src,
                    "staged_k_scan_kernel": {"us_per_launch": ms_scores * 1e3, "frac": scan_bytes / (ms_scores * 1e-3) / 1e9 / peak,
                                             "note": "score_tc5_kernel of the staged path (PKV_FLAG_STAGED), for comparison"}}
        elif fused_path == 1:
            achieved = scan_bytes / (ms_scanpool * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": "evict_fused_kernel (stages 1-2 in one launch: K scan on tcgen05/TMA, softmax, window sums, pool; logits stay in TMEM)",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "whole_step_frac": whole_frac, "traffic": traffic,
                    "algorithmic_bytes_per_launch": scan_bytes, "us_per_launch": ms_scanpool * 1e3, "peak_source": peak_src,
                    "staged_k_scan_kernel": {"us_per_launch": ms_scores * 1e3, "frac": scan_bytes / (ms_scores * 1e-3) / 1e9 / peak,
                                             "note": "score_tc5_kernel of the staged path (PKV_FLAG_STAGED) alone, for comparison; the staged path adds the pool kernel"}}
        else:
            achieved = scan_bytes / (ms_scores * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": "stage-1 window-score (K scan)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "whole_step_frac": whole_frac, "traffic": traffic, "algorithmic_bytes_per_launch": scan_bytes,
                    "us_per_launch": ms_scores * 1e3, "peak_source": peak_src}
        per_layer = {"ms": ms_step, "us_per_layer": ms_step * 1e3 / L, "launches_per_step": int(launches), "whole_step_frac": whole_frac,
                     "k_scan_kernel": {"us_per_launch": ms_scores * 1e3, "frac": scan_bytes / (ms_scores * 1e-3) / 1e9 / peak},
                     "note": "pkv_evict_prefill layer by layer (pkv_defer_eviction off): three launches per layer"}
        if ms_batch is not None:
            # the pass the plugin runs by default: one persistent score launch over the K of ALL layers
            achieved = L * scan_bytes / (batch_ms["scores"] * 1e-3) / 1e9
            n_launch = -(-L // 32)
            if os.path.exists(tp) and L == 32 and wl.S == 32768 and wl.Hkv == 8:      # the ncu capture is of this shape
                traffic = json.load(open(tp)).get("batch_score_kernel_dram_bytes_per_launch", traffic)
            roof = {"bound": "hbm", "kernel": "score_tc5_kernel over all layers of the prompt (layer batch: one persistent launch per 32 layers)",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "whole_step_frac": whole_bytes / (ms_batch * 1e-3) / 1e9 / peak, "traffic": traffic,
                    "traffic_note": "DRAM bytes of the launch (ncu): K + Q once, plus the logits it writes (0.52 GB: they do not fit the L2 across 32 layers)",
                    "algorithmic_bytes_per_launch": L * scan_bytes / n_launch, "us_per_launch": batch_ms["scores"] * 1e3 / n_launch, "peak_source": peak_src,
                    "per_layer_k_scan_kernel": per_layer["k_scan_kernel"]}
            launches_pl, ms_pl = launches, ms_step
            ms_step, launches = ms_batch, launches_batch
        cfg = make_config(args.workload, wl.method, world)
        out = {
            "metric": METRIC, "value": ms_step, "unit": "ms", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": False, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": cfg,
            "run": {"score_kernel": args.score_kernel, "kv_layout": args.kv_layout, "evict_path": "layer batch: all layers in one pass, four launches per 32 layers (pkv_evict_prefill_batch)" if ms_batch is not None else {0: "staged launches", 1: "fused stages 1-2 + select kernel (2 launches per layer)", 2: "one launch per layer"}[fused_path],
                    "value_is": "evict_ms: all layers' update_kv with Q/K/V resident in HBM (the dense prefill GEMMs/attention are in whole_model.prefill_total_ms)"},
            "e2e": {"value": ms_e2e, "unit": "ms", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h[0],
                    "api": "PyramidKVCluster.update_kv(pinned host K/Q/V) per layer: K + window Q go up, compacted K + indices come down, "
                           "V rows are picked on the host with those indices (V never crosses the bus)", "steps": e2e_steps},
            "gpu_launches": int(launches * args.steps),
            "gpu_launches_per_step": int(launches),
            "clocks": clocks,
            "roofline": roof,
            "stages_us_per_layer": {**{k: v * 1e3 for k, v in stage_ms.items()}, **({"scan_pool_fused": ms_scanpool * 1e3} if ms_scanpool else {})},
            **({"per_layer_calls": per_layer, "batch_stages_ms": batch_ms} if ms_batch is not None else {}),
            "us_per_layer": ms_step * 1e3 / L,
            "evict_algorithmic_gbps": whole_bytes / (ms_step * 1e-3) / 1e9,
            "prompts_per_s_all_gpus": world * 1e3 / ms_step,
        }
        if world == 1 and not args.quick:
            try:
                out["decode"] = decode_bench(wl)
            except Exception as e:
                out["decode"] = {"error": repr(e)[:200]}
            try:
                out["gpu_chain_baseline"] = gpu_chain_baseline(wl)
                out["speedup_vs_gpu_chain"] = out["gpu_chain_baseline"]["ms_per_prompt"] / ms_step
            except Exception as e:   # e.g. out of memory on a shared box: the baseline is informative only
                out["gpu_chain_baseline"] = {"error": repr(e)[:200]}
            if wl.method != "h2o":     # the reference's H2O materialises [1,H,S,S]: not runnable at these sizes
                out["cpu_baseline"] = cpu_reference_arm(args.workload, steps=2, warmup=1, method=wl.method, budget_s=25.0)
            if wl.method == "h2o":     # dense S x S scoring: tensor-pipe roofline (2 passes x 2*Hq*S^2*D FLOP per layer)
                flops = 2 * 2 * Hq * S * S * D
                tf = flops / ((stage_ms["scores"] + stage_ms["pool"]) * 1e-3) / 1e12
                pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"] if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 1400.0
                out["roofline"] = {"bound": "tensor", "kernel": "h2o_tc5_kernel (row statistics + column sums, tcgen05 + TMA)" if os.environ.get("PKV_H2O", "t")[:1] != "m" else "h2o_kernel (row statistics + column sums, mma.sync)", "achieved": tf, "peak": pk,
                                   "unit": "TFLOP/s", "frac": tf / pk, "traffic": None, "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"}
    # ---- N = 1: the whole-model numbers of the metric; N > 1: the layer-sharded 70B split north_star names ----
    del hk, hv, hq, clusters
    if world == 1 and args.whole_model and not args.quick and wl.method == "pyramidkv" and "8b-32k" in args.workload and not args.layers:
        del wl
        torch.cuda.empty_cache()
        try:
            out["whole_model"] = whole_model_numbers(device)
        except Exception as e:
            out["whole_model"] = {"error": repr(e)[:300]}
    elif use_dist and args.sharded_70b:
        del wl
        torch.cuda.empty_cache()
        try:
            r70 = sharded_70b_measure("llama3-70b-32k-b2048", rank, world, device, barrier, max(3, min(args.steps, 10)), 3, args.score_kernel, args.kv_layout)
        except Exception as e:
            r70 = {"error": repr(e)[:300]}
        if rank == 0:
            out["sharded_70b"] = r70
    if use_dist:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--score-kernel", default="auto", choices=["auto", "mma", "tcgen05"], help="stage-1 kernel (auto = tcgen05+TMA when the shape allows)")
    ap.add_argument("--method", default="pyramidkv", choices=["pyramidkv", "snapkv", "h2o", "streamingllm"])
    ap.add_argument("--budget", type=int, default=0, help="override max_capacity_prompt of the workload")
    ap.add_argument("--seq-len", type=int, default=0, help="override the prompt length of the workload")
    ap.add_argument("--layers", type=int, default=0, help="evict only the first N layers of the workload (timing experiments)")
    ap.add_argument("--kv-layout", default="hf", choices=["hf", "head_major"], help="physical K/V layout: hf = [S,H,D] (what HF hands over), head_major = [H,S,D]")
    ap.add_argument("--stage", default="all", choices=["all", "scores", "pool", "topk", "gather", "batch"], help="with --profile-only: run only this stage of the staged API")
    ap.add_argument("--whole-model", type=int, default=1, help="N=1, default workload: also build the random-init Llama-3-8B and report prefill_total_ms / decode tok/s through the plugin")
    ap.add_argument("--sharded-70b", type=int, default=1, help="N>1: after the weak-scaling numbers also run the layer-sharded Llama-3-70B arm (configs[4]) and report it under sharded_70b")
    ap.add_argument("--quick", type=int, default=0, help="1: only the resident-HBM eviction numbers (A/B runs; skips e2e, decode and the baselines - not a bench line)")
    ap.add_argument("--profile-only", action="store_true", help="run warmup+steps of the resident-HBM loop and exit (for ncu; prints no bench line)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the compacted K/V caches of the last timed step to DIR/k_cache.npy and DIR/v_cache.npy (float32; "
                         "a fixed seeded sample of rows when larger; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.profile_only):
        ap.error("--dump-outputs writes the outputs of the timed GPU path: not with --impl reference or --profile-only")
    if args.budget or args.seq_len or args.layers or args.method != "pyramidkv":
        L, Hq, Hkv, D, S, B, W, ks, pool = WORKLOADS[args.workload]
        B = args.budget or B
        if args.method == "streamingllm":
            W = B - 4                                      # run_longbench.py:222-223
        name = f"{args.workload}+{args.method}" + (f"+b{B}" if args.budget else "") + (f"+s{args.seq_len}" if args.seq_len else "") + (f"+l{args.layers}" if args.layers else "")
        WORKLOADS[name] = (L, Hq, Hkv, D, args.seq_len or S, B, W, ks, pool)
        args.workload = name
    rank, world, local = dist_env()
    # stdout carries exactly ONE JSON line: everything else that writes to file descriptor 1 during the run (NCCL prints its
    # version banner there at NCCL_DEBUG=VERSION and =WARN, from the environment or /etc/nccl.conf) is sent to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    if world != args.gpus and world == 1 and args.gpus > 1:
        print(f"bench.py: --gpus {args.gpus} needs torchrun (one rank per GPU); launch with python -m torch.distributed.run", file=sys.stderr)
        sys.exit(2)

    if args.impl == "reference":
        if rank != 0:
            return
        L = WORKLOADS[args.workload][0]
        r = cpu_reference_arm(args.workload, steps=max(1, args.steps), warmup=max(1, min(args.warmup, 2)), method=args.method)
        S, B, W = WORKLOADS[args.workload][4], WORKLOADS[args.workload][5], WORKLOADS[args.workload][6]
        emit({
            "impl": "reference", "metric": METRIC, "value": r["value"], "unit": "ms", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": r["value"], "higher_is_better": False, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": make_config(args.workload, args.method, args.gpus),
            "cpu_baseline": r, "e2e": {"value": r["value"], "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        })
        return

    out = gpu_arm(args, rank, world, local)
    if rank == 0 and out is not None:
        emit(out)


if __name__ == "__main__":
    main()
