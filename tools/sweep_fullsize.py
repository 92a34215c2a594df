"""Accuracy of the factorisation at FULL size (64K x 4096 etc.) against the Eckart-Young optimum from the fp64 Gram
(tests/test_fullsize_gpu.py).  Design aid, not a bench line."""
import json
import math
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from xkv_b200 import factorize, synthetic

CASES = [(65536, 4096, 512, 1.0), (65536, 4096, 768, 0.5), (32768, 2048, 512, 1.0), (65536, 1024, 128, 1.0)]
STORAGE = 1.96e-3   # three bf16 roundings (A, V, product) of 2^-9/sqrt(3) relative each


def optimum(x, rank):
    n = x.shape[1]
    g = torch.zeros(n, n, dtype=torch.float64, device=x.device)
    for lo in range(0, x.shape[0], 16384):
        xd = x[lo:lo + 16384].double()
        g.addmm_(xd.t(), xd)
    lam = torch.linalg.eigvalsh(g).flip(0).clamp_min(0)
    return math.sqrt((lam[rank:].sum() / lam.sum()).item())


def rel_err(x, f):
    num = den = 0.0
    vt = f.Vt.float()
    for lo in range(0, x.shape[0], 16384):
        xs = x[lo:lo + 16384].float()
        xh = (f.A[lo:lo + 16384].float() @ vt).to(torch.bfloat16).float()
        num += (xs - xh).double().pow(2).sum().item()
        den += xs.double().pow(2).sum().item()
    return math.sqrt(num / den)


def main():
    data = []
    for (t, c, r, a) in CASES:
        x = synthetic.group_matrix(t, c, a, seed=4321, device="cuda")
        data.append((x, r, optimum(x, r)))
    row = []
    for x, r, e_opt in data:
        (f,) = factorize.factorize_batch([x], r)
        e = rel_err(x, f)
        alg = math.sqrt(max(e * e - STORAGE ** 2, 0.0))
        row.append((round(e / e_opt, 5), round(alg / e_opt, 5)))
    print(json.dumps({"ratio_raw_and_algorithmic": row}), flush=True)


if __name__ == "__main__":
    main()
