"""Decode layers over random factors at config 2's shape, bracketed by cudaProfilerStart/Stop (for ncu).

    python tools/run_decode_once.py [S] [layers] [--variant N] [--graph]

Prints one JSON line: microseconds per layer enqueued from the host, and (with --graph) replayed as a CUDA graph."""
import argparse
import json
import math
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from xkv_b200 import _lib, ops, synthetic

ap = argparse.ArgumentParser()
ap.add_argument("S", type=int, nargs="?", default=65536)
ap.add_argument("layers", type=int, nargs="?", default=4)
ap.add_argument("--variant", type=int, default=0)
ap.add_argument("--graph", action="store_true")
ap.add_argument("--rk", type=int, default=512)
ap.add_argument("--rv", type=int, default=768)
args = ap.parse_args()
S, layers = args.S, args.layers
H, D, HQ, RK, RV, G = 8, 128, 32, args.rk, args.rv, 4
n = G * H * D
dev = "cuda"
a_k = torch.randn(S, RK, device=dev).bfloat16()
a_v = torch.randn(S, RV, device=dev).bfloat16()
v_k = torch.randn(n, RK, device=dev).bfloat16()
v_v = torch.randn(n, RV, device=dev).bfloat16()
cos, sin = synthetic.llama3_rope(S, D, device=dev)
cos, sin = cos[0].contiguous(), sin[0].contiguous()
q = torch.randn(HQ, D, device=dev).bfloat16()
kt = torch.randn(H, 1, D, device=dev).bfloat16()
vt = torch.randn(H, 1, D, device=dev).bfloat16()
_lib.load().xkv_decode_set_variant(args.variant)
ws = torch.empty(ops.decode_workspace_bytes(HQ, S, 1, RV) + 4096, dtype=torch.uint8, device=dev)
o = torch.empty(HQ, D, dtype=torch.bfloat16, device=dev)


def run():
    for l in range(layers):
        i = l % G
        ops.decode_attention(q, a_k, v_k[i * H * D:(i + 1) * H * D], a_v, v_v[i * H * D:(i + 1) * H * D], H, cos, sin,
                             kt, vt, 1.0 / math.sqrt(D), out=o, workspace=ws)


run()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
torch.cuda.profiler.start()
e0.record()
run()
e1.record()
torch.cuda.synchronize()
torch.cuda.profiler.stop()
res = {"S": S, "layers": layers, "variant": args.variant,
       "us_per_layer_host_enqueue": 1e3 * e0.elapsed_time(e1) / layers}
if args.graph:
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        run()
    g.replay()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(8):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    res["us_per_layer_graph"] = 1e3 * e0.elapsed_time(e1) / (8 * layers)
print(json.dumps(res))
