#!/usr/bin/env python
"""bench.py — headline benchmark of the xKV hot path on B200 (contract: see the task statement).

Workload (BASELINE.json configs[1], `--config 2`, the default): Llama-3.1-8B-shaped KV (32 layers, 8 KV heads x 128),
64K context, batch 1, xKV-4 (8 groups of 4 layers, rank_k 512 / rank_v 768).  One *step* = prefill compression of the
whole cache: every group's K and V gathered and factorised (16 matrices of 65536 x 4096).  `value` is GB/s of bf16 KV
consumed with inputs resident in HBM; `e2e` is the same through host buffers (pinned H2D of the KV and D2H of the
factors inside the timed region); `decode` is the fused reconstruct + attention over the factors (tok/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config 2|3|4|5] [--dump-outputs DIR]

N > 1 is launched with torchrun.  The headline `value` is the contract's weak-scaling number (every rank compresses a
whole 8-group cache of its own: layer groups are independent, no data-path collective).  Two more multi-GPU records
measure the partitions BASELINE.json names:
  strong         ONE cache's 8 groups split over the ranks by parallel.assign_groups (1 group per GPU at N = 8);
  token_sharded  configs[3] (Llama-3.1-70B shape, xKV-8, 128K): one K and one V matrix 131072 x 8192 (rank 1024 / 1536)
                 with token rows split over the ranks; the only collective is the NCCL all-reduce of the packed upper
                 triangle of each n x n fp32 Gram (factorize_batch(process_group=...)).
The default run also reports `append` (north-star step 4), `other_configs` (configs[2] and [4] on this GPU) and, at
N = 1, `gpu_reference` (the reference's own library path, torch.linalg.svd, on the same device) and `cpu_baseline`.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark leaves the source tree as it found it (it may be read-only)

# BASELINE.json configs (index = position in `configs`, 1-based as SURVEY.md section 8 numbers them)
CONFIGS = {
    2: dict(title="xKV-4, Llama-3.1-8B 64K", model="Llama-3.1-8B-shaped KV", layers=32, group=4, heads=8, head_dim=128,
            tokens=65536, rank_k=512, rank_v=768, merge_value=True, alpha_k=1.0, alpha_v=0.5),
    3: dict(title="single SVD (layer_group_size 1), Llama-3.1-8B 64K", model="Llama-3.1-8B-shaped KV", layers=32, group=1,
            heads=8, head_dim=128, tokens=65536, rank_k=128, rank_v=192, merge_value=True, alpha_k=1.0, alpha_v=0.5),
    4: dict(title="xKV-8, Llama-3.1-70B 128K", model="Llama-3.1-70B-shaped KV", layers=80, group=8, heads=8, head_dim=128,
            tokens=131072, rank_k=1024, rank_v=1536, merge_value=True, alpha_k=1.0, alpha_v=0.5),
    5: dict(title="xKV-4 on MLA latents, DeepSeek-V2-Lite 32K", model="DeepSeek-V2-Lite MLA latents (kv_lora_rank 512)",
            layers=27, group=4, heads=1, head_dim=512, tokens=32768, rank_k=512, rank_v=None, merge_value=False,
            alpha_k=1.0, alpha_v=0.5),
}
METRIC = "KV GB/s compressed (prefill, {title})"
SAMPLE_TOKENS = 4096   # tokens of the library-SVD sample on the GPU and of the configs[0]-shaped CPU check


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="xkv_b200", choices=["xkv_b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--tokens", type=int, default=0, help="override the configuration's context length")
    ap.add_argument("--cpu-sample-tokens", type=int, default=0,
                    help="context length of the CPU arm's per-step sample (ONE K matrix); 0 = the configuration's own")
    ap.add_argument("--cpu-config1-tokens", type=int, default=SAMPLE_TOKENS,
                    help="reference arm: one whole group (K + V) at this many tokens, BASELINE.json configs[0]'s shape, is "
                         "timed once per run (0 = skip)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-decode", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip strong / token_sharded / append / other_configs / gpu_reference")
    ap.add_argument("--streams", type=int, default=8, help="CUDA streams the K / V batches are spread over")
    ap.add_argument("--e2e-chunk", type=int, default=1, help="layer groups per pipelined chunk of the host-buffer path")
    ap.add_argument("--packed", action="store_true", help="gather every group into a packed matrix first (round 1's path) "
                    "instead of reading the layer tensors in place")
    ap.add_argument("--factorize-opts", default="", help="JSON of FactorizeOptions overrides for the timed step (tuning experiments)")
    ap.add_argument("--no-graph", action="store_true", help="enqueue every kernel from the host instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the factors of the last step to DIR/<name>.npy (float32, sampled rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the factors of the xkv_b200 arm; the reference arm keeps no outputs")
    return args


def config_of(args):
    c = dict(CONFIGS[args.config])
    if args.tokens:
        c["tokens"] = args.tokens
    if not getattr(args, "cpu_sample_tokens", 0):
        args.cpu_sample_tokens = c["tokens"]
    return c


def group_sizes(c):
    """Layer groups of the configuration: consecutive chunks, the last one may be short (configurations.py:267-273)."""
    full, rest = divmod(c["layers"], c["group"])
    return [c["group"]] * full + ([rest] if rest else [])


def kv_bytes_of(c):
    sides = 2 if c["merge_value"] else 1
    return sides * c["layers"] * c["tokens"] * c["heads"] * c["head_dim"] * 2


def reference_sample_text(c, tokens):
    g = min(c["group"], 4)
    return (f"ONE K matrix of a {g}-layer group per step, {tokens} x {g * c['heads'] * c['head_dim']} "
            f"({tokens} tokens, {c['heads']} KV heads x {c['head_dim']}), through the reference's fake_svd arithmetic: "
            f"torch.linalg.svd fp32 (full, whatever the rank) -> truncate to rank {c['rank_k']} -> multiply back; GB/s of the "
            f"matrix's own bf16 bytes.  The cache is {2 * len(group_sizes(c)) if c['merge_value'] else len(group_sizes(c))} "
            f"such matrices (a V matrix costs the same SVD)")


def workload_config(args, c):
    ng = len(group_sizes(c))
    return {
        "workload": f"{c['model']}, {c['layers']} layers x {c['heads']} KV heads x {c['head_dim']}, {c['tokens']} tokens, "
                    f"batch 1, xKV-{c['group']} ({ng} groups), rank_k {c['rank_k']} / rank_v {c['rank_v']}",
        "baseline_config": args.config, "tokens": c["tokens"], "groups_per_gpu": ng,
        "parallelism": f"layer-groups x{args.gpus}", "l2": f"inputs ({kv_bytes_of(c) / 1e9:.1f} GB per step) exceed L2",
        "cuda_streams": args.streams,
        # what `--impl reference` times per step (the CPU arm cannot run the 64K workload in minutes); both arms carry
        # the same text so that the two `config` objects are equal by content
        "reference_arm_sample": reference_sample_text(c, args.cpu_sample_tokens),
    }


# ----------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the reference's own arithmetic (oracle port of fake_svd etc.)
# ----------------------------------------------------------------------------------------------
def cpu_reference_step(c, sample_tokens: int, seed: int = 0):
    """One bounded sample of the workload on the host cores: ONE K matrix of a layer group at `sample_tokens` tokens (the
    configuration's own context length by default: the cost of the reference's full SVD is far from linear in the token
    count, a short sample would misstate its throughput) through the oracle's fake_svd. Returns (seconds, bytes_of_kv)."""
    import torch
    from oracle import xkv_oracle as O
    from xkv_b200 import synthetic

    g = min(c["group"], 4)
    keys = synthetic.make_group_kv(g, c["heads"], sample_tokens, c["head_dim"], c["alpha_k"], seed)
    x = torch.cat(keys, dim=1).float()
    t0 = time.perf_counter()
    O.fake_svd(x, c["rank_k"])
    dt = time.perf_counter() - t0
    nbytes = g * c["heads"] * sample_tokens * c["head_dim"] * 2
    return dt, nbytes


def cpu_config1_group(c, tokens: int):
    """BASELINE.json configs[0]: one whole layer group (K and V) at 4K tokens through the oracle's grouped merge, once."""
    from oracle import xkv_oracle as O
    from xkv_b200 import synthetic

    g = min(c["group"], 4)
    keys = synthetic.make_group_kv(g, c["heads"], tokens, c["head_dim"], c["alpha_k"], 11)
    vals = synthetic.make_group_kv(g, c["heads"], tokens, c["head_dim"], c["alpha_v"], 12)
    t0 = time.perf_counter()
    O.merge_group(keys, vals, c["rank_k"], c["rank_v"] if c["merge_value"] else None, True, c["merge_value"])
    dt = time.perf_counter() - t0
    nbytes = (2 if c["merge_value"] else 1) * g * c["heads"] * tokens * c["head_dim"] * 2
    return {"tokens": tokens, "what": f"one {g}-layer group, K rank {c['rank_k']}" + (f" + V rank {c['rank_v']}" if c["merge_value"] else ""),
            "seconds": dt, "GBps_of_bf16_KV": nbytes / dt / 1e9,
            "note": "BASELINE.json configs[0]'s shape; square-ish matrices: the SVD's n^3 terms dominate, GB/s is ~5x lower "
                    "than at the 64K context of the headline"}


def run_reference_arm(args):
    import torch

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    c = config_of(args)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    for _ in range(args.warmup):
        cpu_reference_step(c, args.cpu_sample_tokens)
    times = []
    nbytes = 0
    for i in range(args.steps):
        dt, nbytes = cpu_reference_step(c, args.cpu_sample_tokens, seed=i)
        times.append(dt)
    total = sum(times)
    value = nbytes * len(times) / total / 1e9
    sample = reference_sample_text(c, args.cpu_sample_tokens)
    line = {
        "impl": "reference", "metric": METRIC.format(title=c["title"]), "value": value, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, c),
        "cpu_baseline": {"value": value, "unit": "GB/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if args.cpu_config1_tokens:
        try:
            line["cpu_baseline"]["config1_check"] = cpu_config1_group(c, args.cpu_config1_tokens)
        except Exception as ex:   # the per-step sample stands on its own
            line["cpu_baseline"]["config1_check"] = {"error": f"{type(ex).__name__}: {ex}"}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            parts = [p.strip() for p in s.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# the B200 arm
# ----------------------------------------------------------------------------------------------
class Ctx:
    """Process-level state of one bench run (rank, device, collectives, timing helpers)."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        try:
            self.peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            self.peaks = {}
        self.peak_tf = float(self.peaks.get("bf16_tflops_sustained", 1400.0))
        self.peak_hbm = float(self.peaks.get("hbm_gbs", 6550.0))

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_ms(self, ms: float) -> float:
        t = self.torch.tensor([ms], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()

    def time_steps(self, fn, steps: int, warmup: int = 1) -> float:
        """ms per call of fn(): barrier + synchronize on both sides, CUDA events, max over ranks."""
        torch = self.torch
        for _ in range(warmup):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        return self.max_ms(e0.elapsed_time(e1)) / steps


def make_cache(c, dev, seed_base=0):
    """Synthetic KV of one model: keys[g][i] / vals[g][i] (1, H, S, D) bf16 views of token-major memory."""
    from xkv_b200 import synthetic

    keys, vals = [], []
    for g, size in enumerate(group_sizes(c)):
        keys.append(synthetic.make_group_kv(size, c["heads"], c["tokens"], c["head_dim"], c["alpha_k"],
                                            1234 + seed_base + g, device=dev))
        vals.append(synthetic.make_group_kv(size, c["heads"], c["tokens"], c["head_dim"], c["alpha_v"],
                                            5678 + seed_base + g, device=dev) if c["merge_value"] else None)
    return keys, vals


def ctx_args_packed(step) -> bool:
    return bool(getattr(step, "packed", False))


class CompressStep:
    """The timed step: compress every layer group of a cache (equal-sized groups in one call, a short last group in
    another), replayed as a CUDA graph unless --no-graph."""

    def __init__(self, ctx, c, keys, vals, streams, graph=True):
        from xkv_b200 import compress, factorize

        self.torch = ctx.torch
        self.opts = factorize.FactorizeOptions(**json.loads(getattr(ctx.args, "factorize_opts", "") or "{}"))
        sizes = [len(k) for k in keys]
        self.calls = []
        for size in sorted(set(sizes), reverse=True):
            idx = [i for i, s in enumerate(sizes) if s == size]
            self.calls.append(([keys[i] for i in idx], [vals[i] if vals[i] is not None else keys[i] for i in idx], idx))
        self.c, self.streams, self.compress = c, streams, compress
        self.packed = bool(getattr(ctx.args, "packed", False))
        self.graph = None
        self.n_groups = len(keys)
        self.out = None
        if graph and self.n_groups:
            self.enqueue()
            ctx.torch.cuda.synchronize()
            self.graph = ctx.torch.cuda.CUDAGraph()
            with ctx.torch.cuda.graph(self.graph):
                self.out = self.enqueue()

    def enqueue(self):
        out = [None] * self.n_groups
        for ks, vs, idx in self.calls:
            res = self.compress.compress_groups(ks, vs, self.c["rank_k"], self.c["rank_v"], merge_value=self.c["merge_value"],
                                                opts=self.opts, num_streams=self.streams, in_place=not ctx_args_packed(self))
            for i, r in zip(idx, res):
                out[i] = r
        return out

    def __call__(self):
        if self.graph is not None:
            self.graph.replay()
            return self.out
        self.out = self.enqueue()
        return self.out


DUMP_BYTES = 64 * 10**6     # --dump-outputs: all files together stay below this
DUMP_SEED = 0


def dump_outputs(factors, out_dir, budget=DUMP_BYTES):
    """Write what one compress step returns (a GroupFactors per layer group) as float32 .npy files: for group g and side
    s in (k, v), `group{g}_{s}_A` (token factor, tokens x rank), `group{g}_{s}_V` (right factor, n x rank) and
    `group{g}_{s}_sigma` (leading singular values).  A 2-D factor with more rows than the budget allows is written as a
    fixed sample of its rows: the ascending indices numpy.random.default_rng(DUMP_SEED).choice(rows, k, replace=False),
    one k for every 2-D array, so equal shapes give equal rows in every run.  Returns {name: shape written}."""
    import numpy as np
    import torch

    arrays = {}
    for g, gf in enumerate(factors):
        for side, f in (("k", gf.key), ("v", gf.value)):
            if f is None:
                continue
            arrays[f"group{g}_{side}_A"] = f.A
            arrays[f"group{g}_{side}_V"] = f.V
            if f.sigma_lead is not None:
                arrays[f"group{g}_{side}_sigma"] = f.sigma_lead
    header = 256                # bound on a .npy header (128 bytes for these shapes)
    fixed = header * len(arrays) + sum(4 * t.numel() for t in arrays.values() if t.dim() == 1)
    cols = sum(t.shape[1] for t in arrays.values() if t.dim() == 2)
    max_rows = (budget - fixed) // (4 * cols) if cols else 0
    if cols and max_rows < 1:
        raise ValueError(f"--dump-outputs: {len(arrays)} arrays do not fit in {budget} bytes")
    os.makedirs(out_dir, exist_ok=True)
    shapes = {}
    for name, t in arrays.items():
        if t.dim() == 2 and t.shape[0] > max_rows:
            rows = np.sort(np.random.default_rng(DUMP_SEED).choice(t.shape[0], max_rows, replace=False))
            t = t.index_select(0, torch.from_numpy(rows).to(t.device))
        a = t.float().cpu().numpy()
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
        shapes[name] = list(a.shape)
    return shapes


def gram_roofline(ctx, c, keys, ms_step):
    """Roofline of the dominant kernel: the symmetric Gram GEMM (tcgen05), one launch over the K matrices of the
    equal-sized groups, timed with the CUDA events the library records around that launch on its stream."""
    from xkv_b200 import compress, factorize

    size = c["group"]
    groups = [k for k in keys if len(k) == size][:16]
    nb = len(groups)
    S, n = c["tokens"], size * c["heads"] * c["head_dim"]
    xk = compress.pack_groups(groups)
    fk = factorize.factorize_batch(xk, c["rank_k"], factorize.FactorizeOptions(profile=True))
    stages = fk[0].timings
    del fk, xk
    gram_ms = stages["gram_gemm"]
    alg_flops = nb * float(S) * n * n      # symmetric half of 2 m n^2 per matrix
    achieved = alg_flops / (gram_ms * 1e-3) / 1e12
    traffic = None
    try:
        per_matrix = json.load(open(os.path.join(ROOT, "profiles", "gram_traffic.json"))).get("dram_bytes_per_matrix")
        if per_matrix is not None and S == 65536 and n == 4096:
            traffic = per_matrix * nb
    except Exception:
        pass
    ranks = c["rank_k"] + (c["rank_v"] or 0)
    alg_pipeline = 4.0 * S * sum(g * c["heads"] * c["head_dim"] for g in group_sizes(c)) * ranks
    return {
        "kernel": "gemm_pair_kernel<1,1> (Gram X^T X, symmetric 256 x 256 tiles per CTA pair, tcgen05 cta_group::2 M256 N256 K16)",
        "bound": "tensor", "achieved": achieved, "peak": ctx.peak_tf, "unit": "TFLOP/s", "frac": achieved / ctx.peak_tf,
        "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if ctx.peaks else "fallback 1.4 PFLOP/s",
        "traffic": traffic, "launch_ms": gram_ms, "matrices_per_launch": nb,
        "algorithmic_flops_per_launch": alg_flops, "stages_ms_k_batch": stages,
        "pipeline_algorithmic_frac": (alg_pipeline / (ms_step * 1e-3) / 1e12) / ctx.peak_tf,
    }


def hbm_roofline(ctx, c, ms_step):
    """Whole-step roofline of a skinny-rank configuration (SURVEY section 8d: rank below the ridge => HBM-bound):
    algorithmic bytes = two bf16 reads of every matrix + the factor writes."""
    S = c["tokens"]
    total = 0.0
    for g in group_sizes(c):
        n = g * c["heads"] * c["head_dim"]
        for r in (c["rank_k"], c["rank_v"] if c["merge_value"] else None):
            if r:
                total += 2.0 * S * n * 2 + (S * r + r * n) * 2.0
    achieved = total / (ms_step * 1e-3) / 1e9
    return {"kernel": "whole compress step (Gram pass + projection pass over X)", "bound": "hbm", "achieved": achieved,
            "peak": ctx.peak_hbm, "unit": "GB/s", "frac": achieved / ctx.peak_hbm, "traffic": None,
            "algorithmic_bytes_per_step": total,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs" if ctx.peaks else "fallback 6550 GB/s"}


def bench_decode(ctx, c, factors, no_graph):
    """Fused reconstruct + RoPE + attention over the factors, all layers = one token (Llama-shaped configurations)."""
    from xkv_b200 import ops, synthetic

    torch = ctx.torch
    dev = ctx.dev
    S, H, D, L, G = c["tokens"], c["heads"], c["head_dim"], c["layers"], c["group"]
    cos, sin = synthetic.llama3_rope(S, D, device=dev)
    cos, sin = cos[0].contiguous(), sin[0].contiguous()
    hq = 4 * H
    gen = torch.Generator(device=dev).manual_seed(7)
    q = torch.randn(L, hq, D, device=dev, generator=gen).bfloat16()
    kt = torch.randn(L, H, 1, D, device=dev, generator=gen).bfloat16()
    vt = torch.randn(L, H, 1, D, device=dev, generator=gen).bfloat16()
    ws = torch.empty(ops.decode_workspace_bytes(hq, S, 1, c["rank_v"]) + 4096, dtype=torch.uint8, device=dev)
    o = torch.empty(hq, D, dtype=torch.bfloat16, device=dev)
    hd = H * D

    def one_token():
        for l in range(L):
            gf = factors[l // G]
            i = l % G
            ops.decode_attention(q[l], gf.key.A, gf.key.V[i * hd:(i + 1) * hd], gf.value.A, gf.value.V[i * hd:(i + 1) * hd],
                                 H, cos, sin, kt[l], vt[l], 1.0 / math.sqrt(D), out=o, workspace=ws)

    for _ in range(3):
        one_token()
    ctx.barrier()
    l0 = ops.launch_count()
    one_token()
    launches_per_token = ops.launch_count() - l0
    token_graph = None
    if not no_graph:
        torch.cuda.synchronize()
        token_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(token_graph):
            one_token()
    ms_tok = ctx.time_steps(token_graph.replay if token_graph is not None else one_token, 8, warmup=1)
    flops_k = 2.0 * S * c["rank_k"] * H * D * L
    bytes_a = float(S) * (c["rank_k"] + c["rank_v"]) * 2 * L
    rec = {
        "metric": f"decode tok/s reconstructed (attention over the factored cache, {L} layers, batch 1, {S} context)",
        "tok_s": ctx.world * 1e3 / ms_tok, "ms_per_token": ms_tok, "us_per_layer": 1e3 * ms_tok / L,
        "equiv_dense_kv_GBps": ctx.world * L * 2.0 * S * H * D * 2 / (ms_tok * 1e-3) / 1e9,
        "gpu_launches_per_token": launches_per_token,
        "launch_mode": "cuda-graph replay" if token_graph is not None else "host enqueue",
        "roofline": {"bound": "tensor", "achieved": flops_k / (ms_tok * 1e-3) / 1e12, "peak": ctx.peak_tf,
                     "unit": "TFLOP/s", "frac": flops_k / (ms_tok * 1e-3) / 1e12 / ctx.peak_tf,
                     "hbm_frac": bytes_a / (ms_tok * 1e-3) / 1e9 / ctx.peak_hbm,
                     "note": "whole decode step (scores + softmax + P*A_v + combine) against the K^ reconstruction flops"},
    }
    del ws
    if ctx.rank == 0:
        # context, not a target: the library attention (torch SDPA, GQA) over an UNCOMPRESSED bf16 cache of one layer of the
        # same shape -- what the reference's decode costs once its dense K^ / V^ exist (llama.py:58-69)
        try:
            import torch.nn.functional as F

            kd = torch.randn(1, H, S, D, device=dev, dtype=torch.bfloat16)
            vd = torch.randn(1, H, S, D, device=dev, dtype=torch.bfloat16)
            qd = torch.randn(1, hq, 1, D, device=dev, dtype=torch.bfloat16)
            for _ in range(3):
                F.scaled_dot_product_attention(qd, kd, vd, enable_gqa=True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(32):
                F.scaled_dot_product_attention(qd, kd, vd, enable_gqa=True)
            e1.record()
            torch.cuda.synchronize()
            rec["dense_sdpa_us_per_layer"] = 1e3 * e0.elapsed_time(e1) / 32
            rec["dense_sdpa_note"] = ("torch SDPA over an uncompressed bf16 cache of the same shape (library kernel, "
                                      "reported for context)")
        except Exception as ex:
            rec["dense_sdpa_note"] = f"not measured: {type(ex).__name__}"
    return rec


def bench_strong(ctx, c, streams, no_graph, ms_weak):
    """ONE cache's layer groups split over the ranks (parallel.assign_groups: contiguous, balanced; 1 group per GPU at
    N = 8 for config 2).  No data-path collective: a rank's groups are independent of everybody else's.  Every rank
    regenerates only the groups it owns (seeded by GROUP, not by rank: the ranks hold disjoint parts of one cache)."""
    from xkv_b200 import parallel, synthetic

    sizes = group_sizes(c)
    mine = parallel.assign_groups(len(sizes), ctx.world, ctx.rank)
    per_rank = [len(parallel.assign_groups(len(sizes), ctx.world, r)) for r in range(ctx.world)]
    if ctx.world == 1:
        return {"scaling": "strong", "groups_per_rank": per_rank, "ms_per_step": ms_weak,
                "value": kv_bytes_of(c) / (ms_weak * 1e-3) / 1e9, "unit": "GB/s", "note": "N = 1: the headline step itself"}
    keys, vals = [], []
    for g in mine:
        keys.append(synthetic.make_group_kv(sizes[g], c["heads"], c["tokens"], c["head_dim"], c["alpha_k"], 1234 + g, device=ctx.dev))
        vals.append(synthetic.make_group_kv(sizes[g], c["heads"], c["tokens"], c["head_dim"], c["alpha_v"], 5678 + g, device=ctx.dev)
                    if c["merge_value"] else None)
    step = CompressStep(ctx, c, keys, vals, streams, graph=not no_graph) if mine else (lambda: None)
    ms = ctx.time_steps(step, max(3, min(ctx.args.steps, 10)), warmup=2)
    return {"scaling": "strong", "groups_per_rank": per_rank, "ms_per_step": ms, "unit": "GB/s",
            "value": kv_bytes_of(c) / (ms * 1e-3) / 1e9,
            "ideal_ms": ms_weak / ctx.world, "efficiency_vs_one_gpu_step": (ms_weak / ctx.world) / ms,
            "note": "one cache split by layer group, time = slowest rank, no data-path collective"}


def bench_token_sharded(ctx):
    """configs[3]: Llama-3.1-70B-shaped KV (80 layers, 8 KV heads x 128), xKV-8 at 128K: the WHOLE cache, 10 groups = 20
    matrices 131072 x 8192 (K rank 1024, V rank 1536), with the token rows of every matrix split over the ranks
    (parallel.token_shard).  factorize_token_sharded: every rank runs the Gram of ITS rows, the packed upper triangle of
    matrix i is summed onto rank i mod N (NCCL reduce), that rank alone derives the right factor and broadcasts it, every
    rank projects its own rows.  At N = 1 the same 20 matrices go through the single-GPU driver."""
    from xkv_b200 import factorize, parallel

    torch, dist = ctx.torch, ctx.dist
    c = CONFIGS[4]
    S, n = c["tokens"], c["group"] * c["heads"] * c["head_dim"]
    ngroups = len(group_sizes(c))
    b, e = parallel.token_shard(S, ctx.world, ctx.rank)
    rows = e - b

    def shard(alpha, seed):
        # X = T diag(s) W^T + noise with W shared by all ranks (same seed) and the rows of T i.i.d. (rank-local seed):
        # the shards are rows of ONE matrix with a power-law spectrum
        gw = torch.Generator(device=ctx.dev).manual_seed(seed)
        w = torch.linalg.qr(torch.randn(n, 2048, generator=gw, device=ctx.dev))[0]
        s = torch.arange(1, 2049, device=ctx.dev, dtype=torch.float32) ** (-alpha)
        gt = torch.Generator(device=ctx.dev).manual_seed(seed * 1000 + ctx.rank)
        out = torch.empty(rows, n, dtype=torch.bfloat16, device=ctx.dev)
        for lo in range(0, rows, 16384):
            hi = min(lo + 16384, rows)
            t = torch.randn(hi - lo, 2048, generator=gt, device=ctx.dev) / S ** 0.5
            x = (t * s) @ w.t()
            x += 1e-3 * s[0] / S ** 0.5 * torch.randn(hi - lo, n, generator=gt, device=ctx.dev)
            out[lo:hi] = x.to(torch.bfloat16)
        return out

    jobs = []
    for g in range(ngroups):
        jobs.append((shard(c["alpha_k"], 41 + 2 * g), c["rank_k"]))
        jobs.append((shard(c["alpha_v"], 42 + 2 * g), c["rank_v"]))
    group = dist.group.WORLD if ctx.world > 1 else None
    opts = factorize.FactorizeOptions()
    comm = {"ms": 0.0, "bytes": 0}
    ws = None
    if group is None:
        ws = torch.empty(max(factorize.workspace_bytes(ngroups, rows, n, r, opts) for _, r in jobs[:2]), dtype=torch.uint8,
                         device=ctx.dev)

    def step(timed=False):
        if group is None:     # one GPU: the K matrices in one batch, the V matrices in another
            for r in (c["rank_k"], c["rank_v"]):
                factorize.factorize_batch([x for x, rr in jobs if rr == r], r, opts, workspace=ws)
            return
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)] if timed else None
        factorize.factorize_token_sharded(jobs, group, opts, comm_events=ev)
        if ev is not None:
            torch.cuda.synchronize()
            comm["ms"] += ev[0].elapsed_time(ev[1])
            comm["bytes"] += ev[2]

    ms = ctx.time_steps(step, 2, warmup=1)
    step(timed=True)    # one more step with events around the collectives (synchronises, so outside the timed loop)
    ar_ms = ctx.max_ms(comm["ms"])
    kv = kv_bytes_of(c)
    rec = {
        "workload": f"{c['model']}, {c['layers']} layers, xKV-8 at {S} tokens: {len(jobs)} matrices {S} x {n} (rank {c['rank_k']} / "
                    f"{c['rank_v']}), token rows split over {ctx.world} rank(s)",
        "scaling": "strong", "tokens_per_rank": rows, "matrices": len(jobs), "ms_per_step": ms,
        "value": kv / (ms * 1e-3) / 1e9, "unit": "GB/s",
        "collective": ("NCCL all-reduce(sum, fp32) of the packed upper triangle of each n x n Gram (overlapping the next Gram) + "
                       "broadcast of the right factor (bf16) from the rank that derived it") if group is not None else None,
        "collective_bytes_per_step": comm["bytes"], "full_gram_allreduce_bytes": len(jobs) * n * n * 4,
        "gram_to_factors_ms_per_step": ar_ms,
        "note": "gram_to_factors_ms: from the first Gram to the last right factor received (Grams, collectives and the owners' "
                "small-matrix stages overlap inside it); the projections follow",
    }
    del jobs, ws
    torch.cuda.empty_cache()
    return rec


def bench_append(ctx, c, factors):
    """North-star step 4: project T new token rows of a group onto its right factors (xkv_append_project_batch: the K and
    the V factor of a group in ONE launch), HBM-bound on reading V (n x r bf16).  One timed pass = every group of the
    cache once (8 launches, 84 MB of right factors at config 2), replayed as a CUDA graph; the L2 flush (a 256 MiB memset)
    is enqueued first and the start event after it, so the interval holds the launches only, no host latency."""
    from xkv_b200 import ops

    torch = ctx.torch
    n = factors[0].key.V.shape[0]
    out = {}
    lib_ws = torch.empty(1 << 24, dtype=torch.uint8, device=ctx.dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=ctx.dev)   # > L2: the factors are read from HBM
    for T in (1, 8):
        xk = torch.randn(T, n, device=ctx.dev).bfloat16()
        xv = torch.randn(T, n, device=ctx.dev).bfloat16()
        oks = [torch.empty(T, gf.key.rank, dtype=torch.bfloat16, device=ctx.dev) for gf in factors]
        ovs = [torch.empty(T, gf.value.rank, dtype=torch.bfloat16, device=ctx.dev) for gf in factors]

        def run():
            for gf, ok, ov in zip(factors, oks, ovs):
                ops.append_project_many([xk, xv], [gf.key.V, gf.value.V], [ok, ov], workspace=lib_ws)

        run()
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            run()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        total = 0.0
        reps = 5
        for _ in range(reps):
            torch.cuda.synchronize()
            flush.zero_()
            e0.record()
            graph.replay()
            e1.record()
            torch.cuda.synchronize()
            total += e0.elapsed_time(e1)
        ms = total / reps
        nbytes = sum(n * (gf.key.rank + gf.value.rank) * 2 for gf in factors)
        out[f"T{T}"] = {"us_per_group": 1e3 * ms / len(factors), "V_bytes_read": nbytes, "groups": len(factors),
                        "GBps": nbytes / (ms * 1e-3) / 1e9, "hbm_frac": nbytes / (ms * 1e-3) / 1e9 / ctx.peak_hbm}
        del graph
    del flush, lib_ws
    out["note"] = ("a_new (T x r) = x_new (T x n) V (n x r) for the K and the V factor of every group (one launch per group), "
                   "L2 flushed before every pass; bound: HBM read of V")
    return out


def bench_other_config(ctx, idx, streams):
    """Compress step of another BASELINE.json configuration on this GPU (rank 0's device; N-independent)."""
    c = CONFIGS[idx]
    torch = ctx.torch
    keys, vals = make_cache(c, ctx.dev, seed_base=1000 * idx)
    step = CompressStep(ctx, c, keys, vals, streams, graph=True)
    for _ in range(2):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(3):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 3
    rec = {"workload": workload_config(ctx.args, c)["workload"], "ms_per_step": ms,
           "value": kv_bytes_of(c) / (ms * 1e-3) / 1e9, "unit": "GB/s"}
    ridge = ctx.peak_tf * 1e12 / (ctx.peak_hbm * 1e9)
    if max(c["rank_k"], c["rank_v"] or 0) < ridge:      # two-pass flops per byte = rank: below the ridge the step is HBM-bound
        rec["roofline"] = hbm_roofline(ctx, c, ms)
    else:
        ranks = c["rank_k"] + (c["rank_v"] or 0)
        alg = 4.0 * c["tokens"] * sum(g * c["heads"] * c["head_dim"] for g in group_sizes(c)) * ranks
        rec["roofline"] = {"bound": "tensor", "achieved": alg / (ms * 1e-3) / 1e12, "peak": ctx.peak_tf, "unit": "TFLOP/s",
                           "frac": alg / (ms * 1e-3) / 1e12 / ctx.peak_tf,
                           "note": "whole step against SURVEY 8d's two-pass algorithmic flops 4 m n r"}
    del step, keys, vals
    torch.cuda.empty_cache()
    return rec


def bench_mla_decode(ctx):
    """configs[4] decode: one token over the factored latent cache of a DeepSeek-V2-Lite-shaped model (27 layers, 16 heads,
    kv_lora_rank 512, rope dim 64, 32K context, xKV-4 rank 512) in the factors' rank space (xkv_decode_absorbed: scores and
    values are two streaming passes over the group's token factor A; the latents are never rebuilt, kv_b_proj never runs
    over the cache).  The per-head folding of the query / unfolding of the result (a few 16 x 512 x 512 products) belongs
    to the attention module and is not part of the cache kernel timed here."""
    from xkv_b200 import ops

    torch = ctx.torch
    c = CONFIGS[5]
    S, r, L, hq, dr = c["tokens"], c["rank_k"], c["layers"], 16, 64
    gen = torch.Generator(device=ctx.dev).manual_seed(3)
    ngroups = len(group_sizes(c))
    a = [(torch.randn(S, r, device=ctx.dev, generator=gen) * 0.3).bfloat16() for _ in range(ngroups)]
    kpe = [torch.randn(S, dr, device=ctx.dev, generator=gen).bfloat16() for _ in range(L)]
    inv_rms = [(0.5 + torch.rand(S, device=ctx.dev, generator=gen)).float() for _ in range(L)]
    q_hat = torch.randn(L, hq, r, device=ctx.dev, generator=gen).bfloat16()
    q_pe = torch.randn(L, hq, dr, device=ctx.dev, generator=gen).bfloat16()
    ws = torch.empty(int(ops._lib.load().xkv_decode_absorbed_workspace_bytes(hq, S, r)) + 4096, dtype=torch.uint8, device=ctx.dev)

    def one_token():
        for l in range(L):
            ops.decode_absorbed(q_hat[l], a[l // c["group"]], 0.07, row_scale=inv_rms[l], bias_q=q_pe[l], bias_k=kpe[l], workspace=ws)

    for _ in range(2):
        one_token()
    torch.cuda.synchronize()
    l0 = ops.launch_count()
    one_token()
    launches = ops.launch_count() - l0
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        one_token()
    graph.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(8):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 8
    nbytes = L * (2.0 * S * r * 2 + S * dr * 2)        # A is read for the scores and again for the values
    return {"metric": f"decode tok/s over the factored MLA latent cache ({L} layers, {hq} heads, rank {r}, {S} context)",
            "tok_s": 1e3 / ms, "us_per_layer": 1e3 * ms / L, "gpu_launches_per_token": launches,
            "roofline": {"bound": "hbm", "achieved": nbytes / (ms * 1e-3) / 1e9, "peak": ctx.peak_hbm, "unit": "GB/s",
                         "frac": nbytes / (ms * 1e-3) / 1e9 / ctx.peak_hbm,
                         "note": "token factor read twice (scores, values) + k_pe once, per layer"},
            "reference_path_note": "the reference re-expands the whole cache every step: S x 512 reconstruction + RMSNorm + "
                                   "kv_b_proj (S x 512 x 4096) per layer, 1.4e11 flop per layer at 32K"}


def bench_gpu_reference(ctx, c):
    """The reference's own library path ON THIS GPU (SURVEY section 0: the bar is torch.linalg.svd / cuSOLVER + cuBLAS):
    fake_svd's arithmetic (fp32 svd -> truncate -> multiply back) for one K and one V matrix of ONE group at the bounded
    sample's context length, next to this library on the same matrices.  Context, not the contract's reference arm."""
    from xkv_b200 import compress, synthetic

    torch = ctx.torch
    S = SAMPLE_TOKENS
    g = min(c["group"], 4)
    keys = synthetic.make_group_kv(g, c["heads"], S, c["head_dim"], c["alpha_k"], 77, device=ctx.dev)
    vals = synthetic.make_group_kv(g, c["heads"], S, c["head_dim"], c["alpha_v"], 78, device=ctx.dev)
    nbytes = 2 * g * c["heads"] * S * c["head_dim"] * 2

    def ref():
        for layers, r in ((keys, c["rank_k"]), (vals, c["rank_v"])):
            x = torch.cat(layers, dim=1).transpose(1, 2).reshape(1, S, -1).float()
            u, s, vh = torch.linalg.svd(x, full_matrices=False)
            (u[:, :, :r] @ (torch.diag_embed(s[:, :r]) @ vh[:, :r, :])).to(torch.bfloat16)

    def ours():
        compress.compress_groups([keys], [vals], c["rank_k"], c["rank_v"])

    out = {}
    for name, fn, reps in (("torch_linalg_svd", ref, 2), ("xkv_b200", ours, 5)):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        out[name] = {"ms": ms, "GBps": nbytes / (ms * 1e-3) / 1e9}
    out["speedup"] = out["torch_linalg_svd"]["ms"] / out["xkv_b200"]["ms"]
    out["sample"] = f"one {g}-layer group at {S} tokens (K rank {c['rank_k']} + V rank {c['rank_v']}), fp32 SVD on the same B200"
    return out


def run_xkv_arm(args):
    ctx = Ctx(args)
    torch = ctx.torch
    from xkv_b200 import compress, ops

    c = config_of(args)
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    warmup = max(args.warmup, 3)
    kv_bytes = kv_bytes_of(c)

    # ---- synthetic KV, resident in HBM (seeded per rank: the headline gives every rank a cache of its own) ----
    keys, vals = make_cache(c, dev, seed_base=100 * rank)
    step = CompressStep(ctx, c, keys, vals, args.streams, graph=not args.no_graph)
    for _ in range(warmup):
        out = step()
    ctx.barrier()
    sampler = ClockSampler(ctx.local)
    if rank == 0:
        sampler.start()
    # kernels per step: a replayed graph launches the captured kernels without passing through the library's counter
    c0 = ops.launch_count()
    step.enqueue()
    launches_per_step = ops.launch_count() - c0
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier()
    torch.cuda.profiler.start()      # no-op unless run under `ncu --profile-from-start off` (launch list of the timed steps)
    e0.record()
    for _ in range(args.steps):
        out = step()
    e1.record()
    ctx.barrier()
    torch.cuda.profiler.stop()
    ms_step = ctx.max_ms(e0.elapsed_time(e1)) / args.steps
    clocks = sampler.stop() if rank == 0 else None
    value = world * kv_bytes / (ms_step * 1e-3) / 1e9
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)

    ridge = ctx.peak_tf * 1e12 / (ctx.peak_hbm * 1e9)
    # SURVEY 8d: the two-pass minimum does 4 m n r flops over 4 m n bytes, i.e. r flop/B: HBM-bound below the ridge
    skinny = max(c["rank_k"], c["rank_v"] or 0) < ridge
    roofline = hbm_roofline(ctx, c, ms_step) if skinny else gram_roofline(ctx, c, keys, ms_step)
    line = {
        "metric": METRIC.format(title=c["title"]), "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
        "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": workload_config(args, c),
        "gpu_launches": launches_per_step * args.steps, "roofline": roofline,
        "launch_mode": "cuda-graph replay" if step.graph is not None else "host enqueue",
    }

    if not args.no_decode and c["merge_value"] and c["head_dim"] in (64, 128):
        line["decode"] = bench_decode(ctx, c, out, args.no_graph)
    if not args.no_extras and args.config == 2:
        line["append"] = bench_append(ctx, c, out)

    # ---- end to end through the public API with HOST buffers ----
    uniform = len(set(group_sizes(c))) == 1 and c["merge_value"]
    if not args.no_e2e and uniform:
        # the synthetic cache is moved to pinned host memory and the device copies are dropped: every e2e step starts from
        # HOST buffers and ends with the factors back in HOST buffers; device staging is allocated once, outside the loop
        h_keys = [[t.transpose(1, 2).contiguous().cpu().pin_memory() for t in grp] for grp in keys]
        h_vals = [[t.transpose(1, 2).contiguous().cpu().pin_memory() for t in grp] for grp in vals]
        h_out = []
        for g in group_sizes(c):
            n_cols = g * c["heads"] * c["head_dim"]
            for r in (c["rank_k"], c["rank_v"]):
                h_out.append(torch.empty(c["tokens"], r, dtype=torch.bfloat16).pin_memory())
                h_out.append(torch.empty(r, n_cols, dtype=torch.bfloat16).pin_memory())
        d2h_bytes = sum(t.numel() * t.element_size() for t in h_out)
        del step, out, keys, vals
        torch.cuda.empty_cache()
        staging = compress.host_staging(h_keys, h_vals, dev)

        def e2e_step():
            compress.compress_groups_from_host(h_keys, h_vals, c["rank_k"], c["rank_v"], dev, chunk_groups=args.e2e_chunk,
                                               host_out=h_out, staging=staging)

        n_e2e = min(args.steps, 3)
        ms_e2e = ctx.time_steps(e2e_step, n_e2e, warmup=1)
        def h2d_only():   # context for the e2e number: the same host -> device copies with no work behind them
            for dst, src in ((staging[0], h_keys), (staging[1], h_vals)):
                for dg, hg in zip(dst, src):
                    for d, h in zip(dg, hg):
                        d.copy_(h, non_blocking=True)

        ms_h2d = ctx.time_steps(h2d_only, 2, warmup=1)
        line["e2e"] = {"value": world * kv_bytes / (ms_e2e * 1e-3) / 1e9, "unit": "GB/s",
                       "h2d_bytes_per_step": kv_bytes, "d2h_bytes_per_step": d2h_bytes, "ms_per_step": ms_e2e,
                       "steps": n_e2e, "h2d_copy_alone_ms": ms_h2d,
                       "note": "K and V sides pipelined separately behind their own copies; the step is one pass of the KV over "
                               "PCIe (h2d_copy_alone_ms: the same pinned-host -> device copies with nothing behind them) plus "
                               "the last K chain and its copy-back"}
        del staging, h_keys, h_vals, h_out
        torch.cuda.empty_cache()
    else:
        del step, out, keys, vals
        torch.cuda.empty_cache()

    if not args.no_extras and args.config == 2:
        line["strong"] = bench_strong(ctx, c, args.streams, args.no_graph, ms_step)
        torch.cuda.empty_cache()
        line["token_sharded"] = bench_token_sharded(ctx)
        if rank == 0:
            line["other_configs"] = {"3": bench_other_config(ctx, 3, args.streams), "5": bench_other_config(ctx, 5, args.streams)}
            line["other_configs"]["5"]["decode"] = bench_mla_decode(ctx)
            if world == 1:
                line["gpu_reference"] = bench_gpu_reference(ctx, c)
        ctx.barrier()

    if rank == 0:
        line["clocks"] = clocks
        if not args.no_cpu_baseline and world == 1:
            cores = os.cpu_count() or 1
            torch.set_num_threads(cores)
            dt, nbytes = cpu_reference_step(c, args.cpu_sample_tokens)
            line["cpu_baseline"] = {
                "value": nbytes / dt / 1e9, "unit": "GB/s", "cores": cores, "kind": "port",
                "sample": reference_sample_text(c, args.cpu_sample_tokens) + f", {dt:.1f} s"}
        print(json.dumps(line), flush=True)
    if world > 1:
        ctx.dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_xkv_arm(args)


if __name__ == "__main__":
    main()
