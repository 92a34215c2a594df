"""torchrun --nproc-per-node N (N = 1 runs the same path on one GPU): token-sharded factorisation
(factorize_token_sharded: Gram all-reduce over NCCL, the small-matrix stages on each matrix's owner, broadcast of the
right factor) against the single-GPU factorisation of the whole matrix, then token-sharded DECODE over the sharded
factors (each rank attends over its own rows of A_k / A_v, one all-gather of (Hq x (D+1)) floats, flash-decoding merge)
against the fused kernel over the whole context."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist
from xkv_b200 import factorize, parallel, synthetic

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
dist.init_process_group("nccl", device_id=dev)
S, n, r = 8192, 2048, 256
x = synthetic.group_matrix(S, n, 1.0, seed=42, device=dev)      # same seed: identical on every rank
b, e = parallel.token_shard(S, world, rank)
(f_shard,) = factorize.factorize_token_sharded([(x[b:e].contiguous(), r)], dist.group.WORLD)
(f_full,) = factorize.factorize_batch([x], r)
torch.cuda.synchronize()
xd = x.double()
err_full = (torch.linalg.norm(xd - f_full.reconstruct().double()) / torch.linalg.norm(xd)).item()
rec_local = f_shard.reconstruct().double()
num = torch.linalg.norm(xd[b:e] - rec_local) ** 2
dist.all_reduce(num)
err_shard = (num.sqrt() / torch.linalg.norm(xd)).item()
same_v = (f_shard.Vt.float() - f_full.Vt.float()).abs().max().item()
ok = err_shard <= 1.002 * err_full
if rank == 0:
    print(f"token-sharded x{world}: rel err {err_shard:.6f} vs single-GPU {err_full:.6f}; max|Vt diff| {same_v:.3e}; "
          f"{'OK' if ok else 'FAIL'}")
# ---- several matrices and ranks: the small-matrix stages distributed over the owners ----
x2 = synthetic.group_matrix(S, n, 0.5, seed=44, device=dev)
jobs = [(x[b:e].contiguous(), r), (x2[b:e].contiguous(), 384), (x[b:e].contiguous(), 192)]
fs = factorize.factorize_token_sharded(jobs, dist.group.WORLD)
torch.cuda.synchronize()
for (xl, rr), f, full_x in zip(jobs, fs, (x, x2, x)):
    (f1,) = factorize.factorize_batch([full_x], rr)
    e1 = (torch.linalg.norm(full_x.double() - f1.reconstruct().double()) / torch.linalg.norm(full_x.double())).item()
    num = torch.linalg.norm(xl.double() - f.reconstruct().double()) ** 2
    dist.all_reduce(num)
    e2 = (num.sqrt() / torch.linalg.norm(full_x.double())).item()
    vt_all = [torch.empty_like(f.Vt) for _ in range(world)]
    dist.all_gather(vt_all, f.Vt)
    same = all(torch.equal(vt_all[0], v) for v in vt_all)
    okd = e2 <= 1.002 * e1 and same
    ok = ok and okd
    if rank == 0:
        print(f"distributed small stages x{world}, rank {rr}: rel err {e2:.6f} vs single-GPU {e1:.6f}; same Vt on every rank: {same}; "
              f"{'OK' if okd else 'FAIL'}")

# ---- decode over the token shards: K and V factors of one 4-layer group (8 kv heads x 64), layer 1 of the group ----
import math
from xkv_b200 import ops

H, D, qpk, layer = 8, 64, 4, 1
xv = synthetic.group_matrix(S, n, 0.5, seed=43, device=dev)
(fk_s,) = [f_shard]
(fv_s,) = factorize.factorize_token_sharded([(xv[b:e].contiguous(), r)], dist.group.WORLD)
g = torch.Generator(device=dev).manual_seed(5)
q = torch.randn(H * qpk, D, generator=g, device=dev).bfloat16()
k_tail = torch.randn(H, 2, D, generator=g, device=dev).bfloat16()
v_tail = torch.randn(H, 2, D, generator=g, device=dev).bfloat16()
cos, sin = synthetic.llama3_rope(S, D, device=dev)
cos, sin = cos[0].contiguous(), sin[0].contiguous()
rows = slice(layer * H * D, (layer + 1) * H * D)
last = rank == world - 1
lse = torch.empty(H * qpk, device=dev)
o_local = ops.decode_attention(q, fk_s.A, fk_s.V[rows], fv_s.A, fv_s.V[rows], H, cos[b:e], sin[b:e],
                               k_tail if last else None, v_tail if last else None, 1.0 / math.sqrt(D), lse_out=lse)
merged = parallel.merge_token_shards(o_local, lse, dist.group.WORLD)
# reference: all rows gathered on every rank, one fused call over the whole context
def gather_rows(t):
    parts = [torch.empty(parallel.token_shard(S, world, p)[1] - parallel.token_shard(S, world, p)[0], t.shape[1],
                         dtype=t.dtype, device=dev) for p in range(world)]
    dist.all_gather(parts, t.contiguous())
    return torch.cat(parts)
a_k_all, a_v_all = gather_rows(fk_s.A), gather_rows(fv_s.A)
full = ops.decode_attention(q, a_k_all, fk_s.V[rows], a_v_all, fv_s.V[rows], H, cos, sin, k_tail, v_tail, 1.0 / math.sqrt(D))
torch.cuda.synchronize()
derr = (merged.float() - full.float()).abs().max().item()
dscale = full.float().abs().max().item()
ok_dec = derr <= 2e-2 * dscale
if rank == 0:
    print(f"token-sharded decode x{world}: max|diff| {derr:.5f} (output scale {dscale:.3f}); {'OK' if ok_dec else 'FAIL'}")
dist.destroy_process_group()
sys.exit(0 if (ok and ok_dec) else 1)
