"""Accuracy / time of the factorisation on the parity cases and the 64K x 4096 batch (B200). Design aid, not a bench line."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from xkv_b200 import factorize, synthetic

CASES = [(1024, 1024, 128, 1.0), (1024, 1024, 192, 0.5), (2048, 2048, 256, 1.0), (4096, 4096, 512, 1.0),
         (4096, 4096, 768, 0.5), (4096, 4096, 512, None), (1536, 2048, 512, 1.0), (2048, 8192, 1024, 0.5)]


def rel(x, xh):
    return (torch.linalg.norm(x.double() - xh.double()) / torch.linalg.norm(x.double())).item()


def main():
    refs = []
    for (t, c, r, a) in CASES:
        x = synthetic.group_matrix(t, c, a, seed=1234, device="cuda")
        u, s, vh = torch.linalg.svd(x.float(), full_matrices=False)
        ref = ((u[:, :r] * s[:r]) @ vh[:r]).to(torch.bfloat16)
        refs.append((x, rel(x, ref), s))
    big_k = [synthetic.group_matrix(65536, 4096, 1.0, seed=b, device="cuda") for b in range(8)]
    ratios, sig = [], []
    for (t, c, r, a), (x, e_ref, s) in zip(CASES, refs):
        (f,) = factorize.factorize_batch([x], r)
        ratios.append(round(rel(x, f.reconstruct()) / e_ref, 5))
        if a is not None:
            sig.append(((f.sigma_lead[:16] - s[:16]).abs() / s[:16]).max().item())
    times = {}
    for rk in (512, 768):
        factorize.factorize_batch(big_k, rk)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fs = factorize.factorize_batch(big_k, rk)
        e1.record()
        torch.cuda.synchronize()
        times[rk] = round(e0.elapsed_time(e1), 2)
    e64 = rel(big_k[0], fs[0].reconstruct())
    print(json.dumps({"ratios": ratios, "max_ratio": max(ratios), "sigma_dev": max(sig), "ms_64k_b8": times,
                      "err64k_r768": round(e64, 6)}), flush=True)


if __name__ == "__main__":
    main()
