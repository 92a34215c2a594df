"""Stage breakdown of factorize_batch on a B200 (CUDA events). Not a bench line."""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from xkv_b200 import factorize, ops, synthetic


def main():
    S = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
    B = int(sys.argv[2]) if len(sys.argv) > 2 else 8
    rank = int(sys.argv[3]) if len(sys.argv) > 3 else 512
    n = 4096
    xs = [synthetic.group_matrix(S, n, 1.0, seed=b, device="cuda") for b in range(B)]
    opts = factorize.FactorizeOptions(profile=True)
    for rep in range(2):
        torch.cuda.synchronize()
        l0 = ops.launch_count()
        t0 = time.perf_counter()
        fs = factorize.factorize_batch(xs, rank, opts)
        t_host = time.perf_counter() - t0
        torch.cuda.synchronize()
        t_all = time.perf_counter() - t0
        print(json.dumps({"S": S, "B": B, "rank": rank, "rep": rep, "host_enqueue_s": t_host, "wall_s": t_all,
                          "launches": ops.launch_count() - l0, "stages_ms": fs[0].timings,
                          "sum_ms": sum(fs[0].timings.values())}))
    # un-profiled wall time with events around the whole call
    for rep in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fs = factorize.factorize_batch(xs, rank)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        print(json.dumps({"S": S, "B": B, "rank": rank, "total_ms": ms,
                          "GBps_of_KV": B * S * n * 2 / ms / 1e6}))
    x = xs[0].double()
    xh = fs[0].reconstruct().double()
    print(json.dumps({"rel_err": (torch.linalg.norm(x - xh) / torch.linalg.norm(x)).item()}))


if __name__ == "__main__":
    main()
