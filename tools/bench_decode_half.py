"""Cost of a decode step over a one-sided layer group (one slot factored, the other dense) at config 2's layer shape:
S = 65536 prefix tokens, 32 q / 8 kv heads x 128, rank 512 / 768, 16 tail tokens, random factors and dense slots.

    python tools/bench_decode_half.py [--S 65536] [--tq 1 4 8 16] [--reps 40] [--out DIR]

For each Tq, one JSON line with microseconds per layer (CUDA-graph replay) of
  key_only_fused      xkv_decode_attention_half: K factored (rank 512), V a dense (S, H, D) slot
  value_only_fused    xkv_decode_attention_half: V factored (rank 768), K a dense rotated slot
  both_fused          xkv_decode_attention_multi with both sides factored (the reference point)
  key_only_dense      what a key-only layer ran before: materialise K^ (tcgen05 GEMM + bf16 RoPE), cat both sides with
                      the tail, SDPA with the causal mask
  value_only_dense    the same with V^ materialised and the dense keys concatenated
then one line per Tq in {1, max} with each new kernel's time (torch.profiler, a run of its own after the timed replays)
against its HBM floor over 7.7 TB/s (the data-sheet figure): the dense slot, S * H * D * 2 bytes = 134 MB (17.4 us), plus
the fp32 scores the key kernel writes or the bf16 probabilities the value kernel reads.  Every line carries the card's
name and power limit, read in the same run.  Working sets: A_k + dense V slot = 201 MB, A_v + dense K slot = 235 MB,
both above the 126 MB L2, so every replay streams them from HBM.  Lines also go to DIR/decode_half_b200.jsonl with --out."""
import argparse
import json
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F
from xkv_b200 import ops, synthetic

ap = argparse.ArgumentParser()
ap.add_argument("--S", type=int, default=65536)
ap.add_argument("--tq", type=int, nargs="+", default=[1, 4, 8, 16])
ap.add_argument("--reps", type=int, default=40)
ap.add_argument("--tail", type=int, default=16, help="decode tokens already in the tail before the step")
ap.add_argument("--out", default=None)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_decode_half: needs a CUDA device")

S, H, D, HQ, RK, RV = args.S, 8, 128, 32, 512, 768
HBM_BYTES_PER_S = 7.7e12
dev = "cuda"
torch.manual_seed(0)
a_k = (torch.randn(S, RK, device=dev) * 0.05).bfloat16()
a_v = (torch.randn(S, RV, device=dev) * 0.05).bfloat16()
v_k = torch.randn(H * D, RK, device=dev).bfloat16()
v_v = torch.randn(H * D, RV, device=dev).bfloat16()
k_dense = torch.randn(S, H, D, device=dev).bfloat16()      # rotated keys, token-major as the cache keeps them
v_dense = torch.randn(S, H, D, device=dev).bfloat16()
cos, sin = synthetic.llama3_rope(S, D, device=dev)
cos, sin = cos[0].contiguous(), sin[0].contiguous()
scale = 1.0 / math.sqrt(D)
T0, TQMAX = args.tail, max(args.tq)
k_tail = torch.randn(H, T0 + TQMAX, D, device=dev).bfloat16()
v_tail = torch.randn(H, T0 + TQMAX, D, device=dev).bfloat16()
q_all = torch.randn(HQ, TQMAX, D, device=dev).bfloat16()
ws = torch.empty(ops.decode_workspace_bytes(HQ * TQMAX, S, T0 + TQMAX, RV) + 4096, dtype=torch.uint8, device=dev)
x_hat = torch.empty(S, H * D, dtype=torch.bfloat16, device=dev)


def card():
    name = torch.cuda.get_device_name()
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def graph_time(fn, reps):
    """Microseconds per call of fn, replayed as a CUDA graph of `reps` calls (one warm-up replay)."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / reps


def calls(tq):
    T = T0 + tq
    q3 = q_all[:, :tq].contiguous()
    out = torch.empty(HQ, tq, D, dtype=torch.bfloat16, device=dev)
    kt, vt = k_tail[:, :T], v_tail[:, :T]

    def key_only():
        ops.decode_attention_half(q3, H, a_k=a_k, vk_layer=v_k, v_dense=v_dense, cos=cos, sin=sin, k_tail=kt, v_tail=vt,
                                  scale=scale, out=out, workspace=ws)

    def value_only():
        ops.decode_attention_half(q3, H, a_v=a_v, vv_layer=v_v, k_dense=k_dense, k_tail=kt, v_tail=vt, scale=scale,
                                  out=out, workspace=ws)

    def both():
        ops.decode_attention(q3, a_k, v_k, a_v, v_v, H, cos, sin, kt, vt, scale, out=out, workspace=ws)

    mask = torch.ones(tq, S + T, dtype=torch.bool, device=dev).tril(S + T - tq)

    def sdpa(k_prefix, v_prefix):
        k = torch.cat([k_prefix.transpose(0, 1), kt], 1)[None]
        v = torch.cat([v_prefix.transpose(0, 1), vt], 1)[None]
        F.scaled_dot_product_attention(q3[None], k, v, attn_mask=mask, scale=scale, enable_gqa=True)

    def key_only_dense():
        ops.gemm_grouped([ops.make_problem([a_k], [v_k], x_hat, M=S, N=H * D, K=RK)])
        ops.rope_bf16_(x_hat.view(S, H, D), cos, sin)
        sdpa(x_hat.view(S, H, D), v_dense)

    def value_only_dense():
        ops.gemm_grouped([ops.make_problem([a_v], [v_v], x_hat, M=S, N=H * D, K=RV)])
        sdpa(k_dense, x_hat.view(S, H, D))

    return key_only, value_only, both, key_only_dense, value_only_dense


def kernel_times(tq, runs=10):
    """Mean device time (us) of the new kernels over `runs` eager calls of each one-sided path."""
    from torch.profiler import ProfilerActivity, profile

    key_only, value_only = calls(tq)[:2]
    for fn in (key_only, value_only):
        fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(runs):
            key_only()
            value_only()
        torch.cuda.synchronize()
    tot = {}
    for ev in prof.events():
        for tag in ("decode_dense_scores_kernel", "decode_dense_values_kernel"):
            if tag in ev.name:
                n, us = tot.get(tag, (0, 0.0))
                tot[tag] = (n + 1, us + ev.device_time)
    return {tag: us / n for tag, (n, us) in tot.items()}


def main():
    name, power = card()
    lines = []
    for tq in args.tq:
        key_only, value_only, both, key_only_dense, value_only_dense = calls(tq)
        reps = max(4, args.reps // 4)
        rec = {"S": S, "Hq": HQ, "H": H, "D": D, "rk": RK, "rv": RV, "tail_before": T0, "Tq": tq,
               "key_only_fused_us_per_layer": round(graph_time(key_only, args.reps), 2),
               "value_only_fused_us_per_layer": round(graph_time(value_only, args.reps), 2),
               "both_fused_us_per_layer": round(graph_time(both, args.reps), 2),
               "key_only_dense_us_per_layer": round(graph_time(key_only_dense, reps), 2),
               "value_only_dense_us_per_layer": round(graph_time(value_only_dense, reps), 2),
               "gpu": name, "power_limit": power}
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    slot = S * H * D * 2
    for tq in (1, TQMAX):
        kt = kernel_times(tq)
        rows = HQ * tq
        # bytes each kernel must move: the dense slot, plus the fp32 scores it writes (keys) or the bf16 probabilities it
        # reads (values) -- at Tq = 16 the scores are as large as the key slot
        need = {"decode_dense_scores_kernel": slot + rows * S * 4, "decode_dense_values_kernel": slot + rows * S * 2}
        rec = {"S": S, "Hq": HQ, "H": H, "D": D, "Tq": tq, "dense_slot_bytes": slot,
               "hbm_floor_basis": "bytes the kernel must move / 7.7 TB/s (data sheet)"}
        for tag, us in sorted(kt.items()):
            floor_us = need[tag] / HBM_BYTES_PER_S * 1e6
            rec[tag + "_bytes"] = need[tag]
            rec[tag + "_us"] = round(us, 2)
            rec[tag + "_hbm_floor_us"] = round(floor_us, 2)
            rec[tag + "_fraction_of_floor"] = round(floor_us / us, 3)
        rec.update(gpu=name, power_limit=power)
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "decode_half_b200.jsonl"), "w") as f:
            f.writelines(json.dumps(r) + "\n" for r in lines)


main()
