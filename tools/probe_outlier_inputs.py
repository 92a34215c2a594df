"""Robustness probe: inputs whose energy sits in a few channels (unmixed columns with decaying scales; outlier channels)
against the reference SVD.  usage: [ONLY=substr] python tools/probe_outlier_inputs.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from xkv_b200 import factorize, synthetic
def colscale(m, n, p=0.7, seed=1):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(m, n, device="cuda", generator=g)
    x *= (torch.arange(1, n + 1, device="cuda") ** -p)
    return x.to(torch.bfloat16)
def outliers(m, n, alpha, k=4, gain=30.0):
    x = synthetic.group_matrix(m, n, alpha, seed=3, device="cuda").float()
    x[:, torch.arange(k) * 97 % n] *= gain
    return (x * (4.0 / x.abs().max())).to(torch.bfloat16)
def rel(x, xh): return (torch.linalg.norm(x.double() - xh.double()) / torch.linalg.norm(x.double())).item()
cases = [("colscale 4096x2048 r448", colscale(4096, 2048), 448), ("colscale 4096x4096 r512", colscale(4096, 4096), 512),
         ("colscale p=1.0 4096x2048 r512", colscale(4096, 2048, 1.0), 512),
         ("outliers a=1 4096x4096 r512", outliers(4096, 4096, 1.0), 512), ("outliers a=0.5 4096x4096 r768", outliers(4096, 4096, 0.5), 768),
         ("outliers x300 a=1 4096x4096 r512", outliers(4096, 4096, 1.0, 8, 300.0), 512)]
ONLY = os.environ.get("ONLY")
for name, x, r in cases:
    if ONLY and ONLY not in name:
        continue
    u, s, vh = torch.linalg.svd(x.float(), full_matrices=False)
    e_ref = rel(x, ((u[:, :r] * s[:r]) @ vh[:r]).to(torch.bfloat16))
    (f,) = factorize.factorize_batch([x], r)
    torch.cuda.synchronize()
    fin = bool(torch.isfinite(f.A).all() and torch.isfinite(f.Vt).all())
    e = rel(x, f.reconstruct()) if fin else float("nan")
    print(name, "finite", fin, "ref", round(e_ref, 6), "ours", round(e, 6), "ratio", round(e / e_ref, 4),
          "sigma dev", ((f.sigma_lead[:16] - s[:16]).abs() / s[:16]).max().item(), flush=True)
