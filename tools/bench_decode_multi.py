"""Cost of a multi-token decode step (speculative verification) at config 2's layer shape: S = 65536 compressed tokens,
32 q / 8 kv heads x 128, rank 512 / 768, random factors as in tools/run_decode_once.py.

    python tools/bench_decode_multi.py [--S 65536] [--tq 1 2 4 8 16] [--reps 50] [--out DIR]

For each Tq, one JSON line with microseconds per layer of
  fused       one xkv_decode_attention_multi call over Tq query tokens (CUDA-graph replay)
  sequential  Tq single-token calls, the tail growing by one token each (CUDA-graph replay)
  dense       what the patched attention does past the fused bounds: materialise K^ / V^ (tcgen05 GEMM + bf16 RoPE),
              append the tail and run SDPA with the causal mask (CUDA-graph replay)
and the card's name and power limit, read in the same run.  The factors (160 MB) exceed the 126 MB L2: every replay
streams them from HBM.  Lines also go to DIR/bench_decode_multi.jsonl when --out is given."""
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
ap.add_argument("--tq", type=int, nargs="+", default=[1, 2, 4, 8, 16])
ap.add_argument("--reps", type=int, default=50)
ap.add_argument("--tail", type=int, default=16, help="decode tokens already in the tail before the step")
ap.add_argument("--out", default=None)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_decode_multi: needs a CUDA device")

S, H, D, HQ, RK, RV = args.S, 8, 128, 32, 512, 768
dev = "cuda"
torch.manual_seed(0)
a_k = (torch.randn(S, RK, device=dev) * 0.05).bfloat16()
a_v = (torch.randn(S, RV, device=dev) * 0.05).bfloat16()
v_k = torch.randn(H * D, RK, device=dev).bfloat16()
v_v = torch.randn(H * D, RV, device=dev).bfloat16()
cos, sin = synthetic.llama3_rope(S, D, device=dev)
cos, sin = cos[0].contiguous(), sin[0].contiguous()
scale = 1.0 / math.sqrt(D)
T0, TQMAX = args.tail, max(args.tq)
k_tail = torch.randn(H, T0 + TQMAX, D, device=dev).bfloat16()
v_tail = torch.randn(H, T0 + TQMAX, D, device=dev).bfloat16()
q_all = torch.randn(HQ, TQMAX, D, device=dev).bfloat16()
ws = torch.empty(ops.decode_workspace_bytes(HQ * TQMAX, S, T0 + TQMAX, RV) + 4096, dtype=torch.uint8, device=dev)
k_hat = torch.empty(S, H * D, dtype=torch.bfloat16, device=dev)
v_hat = torch.empty(S, H * D, dtype=torch.bfloat16, device=dev)


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


def main():
    name, power = card()
    lines = []
    for tq in args.tq:
        T = T0 + tq
        q3 = q_all[:, :tq].contiguous()
        out3 = torch.empty(HQ, tq, D, dtype=torch.bfloat16, device=dev)
        qs = [q_all[:, t].contiguous() for t in range(tq)]
        out1 = torch.empty(HQ, D, dtype=torch.bfloat16, device=dev)

        def fused():
            ops.decode_attention(q3, a_k, v_k, a_v, v_v, H, cos, sin, k_tail[:, :T], v_tail[:, :T], scale, out=out3,
                                 workspace=ws)

        def sequential():
            for t in range(tq):
                ops.decode_attention(qs[t], a_k, v_k, a_v, v_v, H, cos, sin, k_tail[:, :T0 + t + 1],
                                     v_tail[:, :T0 + t + 1], scale, out=out1, workspace=ws)

        mask = torch.ones(tq, S + T, dtype=torch.bool, device=dev).tril(S + T - tq)

        def dense():
            ops.gemm_grouped([ops.make_problem([a_k], [v_k], k_hat, M=S, N=H * D, K=RK),
                              ops.make_problem([a_v], [v_v], v_hat, M=S, N=H * D, K=RV)])
            ops.rope_bf16_(k_hat.view(S, H, D), cos, sin)
            k = torch.cat([k_hat.view(S, H, D).transpose(0, 1), k_tail[:, :T]], 1)[None]
            v = torch.cat([v_hat.view(S, H, D).transpose(0, 1), v_tail[:, :T]], 1)[None]
            F.scaled_dot_product_attention(q3[None], k, v, attn_mask=mask, scale=scale, enable_gqa=True)

        reps = max(4, args.reps // tq)
        rec = {"S": S, "Hq": HQ, "H": H, "D": D, "rk": RK, "rv": RV, "tail_before": T0, "Tq": tq,
               "fused_us_per_layer": round(graph_time(fused, args.reps), 2),
               "sequential_us_per_layer": round(graph_time(sequential, reps), 2),
               "dense_us_per_layer": round(graph_time(dense, max(4, args.reps // 5)), 2),
               "gpu": name, "power_limit": power}
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_decode_multi.jsonl"), "w") as f:
            f.writelines(json.dumps(r) + "\n" for r in lines)


main()
