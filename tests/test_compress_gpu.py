"""GPU: the pipelined host-buffer path (compress_groups_from_host) produces factors as good as the HBM-resident
path (compress_groups) and returns them in the caller's pinned host buffers.  (The factors are not bit-equal:
the Gaussian test matrix of a factorisation is seeded by the matrix's position in its batch, and the pipeline cuts
the groups into different batches.)"""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("chunk_groups", [1, 2, 3])
def test_host_pipeline_equals_resident_path(chunk_groups):
    from xkv_b200 import compress, synthetic

    dev = torch.device("cuda", 0)
    g, h, s, d, ng, rk, rv = 2, 2, 1024, 64, 3, 64, 96
    keys = [synthetic.make_group_kv(g, h, s, d, 1.0, 10 + i, device=dev) for i in range(ng)]
    vals = [synthetic.make_group_kv(g, h, s, d, 0.5, 20 + i, device=dev) for i in range(ng)]
    ref = compress.compress_groups(keys, vals, rk, rv)
    h_keys = [[t.transpose(1, 2).contiguous().cpu().pin_memory() for t in grp] for grp in keys]
    h_vals = [[t.transpose(1, 2).contiguous().cpu().pin_memory() for t in grp] for grp in vals]
    n = g * h * d
    host_out = []
    for _ in range(ng):
        for r in (rk, rv):
            host_out.append(torch.empty(s, r, dtype=torch.bfloat16).pin_memory())
            host_out.append(torch.empty(r, n, dtype=torch.bfloat16).pin_memory())
    out, host = compress.compress_groups_from_host(h_keys, h_vals, rk, rv, dev, chunk_groups=chunk_groups,
                                                   host_out=host_out)
    torch.cuda.synchronize()
    assert len(out) == ng and len(host) == 4 * ng
    k = 0
    for gi, (a, b) in enumerate(zip(out, ref)):
        for fa, fb, layers in ((a.key, b.key, keys[gi]), (a.value, b.value, vals[gi])):
            x = torch.cat(layers, dim=1).transpose(1, 2).reshape(s, n).double()
            ea = (torch.linalg.norm(x - fa.reconstruct().double()) / torch.linalg.norm(x)).item()
            eb = (torch.linalg.norm(x - fb.reconstruct().double()) / torch.linalg.norm(x)).item()
            assert abs(ea - eb) <= 2e-3 * eb, (ea, eb)
            assert torch.equal(host[k], fa.A.cpu()) and torch.equal(host[k + 1], fa.Vt.cpu())
            k += 2


@pytest.mark.parametrize("g,h,s,d,rk,rv", [(4, 8, 4096, 128, 512, 768), (2, 2, 1000, 64, 64, 64), (3, 1, 2048, 512, 256, 256),
                                           (8, 8, 2048, 128, 1024, 1536),
                                           (7, 8, 2048, 128, 896, 1344)])   # the non-uniform config's 7-layer group
def test_in_place_and_packed_paths_give_bit_identical_factors(g, h, s, d, rk, rv):
    """Per-layer tensor maps (no gather, no packed copy) against the gather kernel + packed matrix: the same tiles in
    the same order, so the factors must be bit-identical.  Token-major layer tensors with a padded row stride (the MLA
    latent is a slice of a wider projection output) are covered by the (3, 1, 2048, 512) case."""
    from xkv_b200 import compress, ops, synthetic

    keys = [t.cuda() for t in synthetic.make_group_kv(g, h, s, d, 1.0, seed=5)]
    vals = [t.cuda() for t in synthetic.make_group_kv(g, h, s, d, 0.5, seed=6)]
    if h == 1:   # rows of a wider buffer: (S, D + 64) memory, the layer is its first D columns
        wide = [torch.zeros(s, d + 64, dtype=torch.bfloat16, device="cuda") for _ in range(2 * g)]
        for w, t in zip(wide, keys + vals):
            w[:, :d] = t[0, 0]
        keys = [w[:, :d].view(1, s, 1, d).transpose(1, 2) for w in wide[:g]]
        vals = [w[:, :d].view(1, s, 1, d).transpose(1, 2) for w in wide[g:]]
    before = ops.launch_count()
    (a,) = compress.compress_groups([keys], [vals], rk, rv, in_place=True)
    mid = ops.launch_count()
    (b,) = compress.compress_groups([keys], [vals], rk, rv, in_place=False)
    after = ops.launch_count()
    torch.cuda.synchronize()
    for fa, fb in ((a.key, b.key), (a.value, b.value)):
        assert torch.equal(fa.Vt, fb.Vt) and torch.equal(fa.V, fb.V) and torch.equal(fa.A, fb.A)
    assert (after - mid) - (mid - before) == 2      # the packed path launches the gather kernel once per side


def test_head_major_layers_fall_back_to_the_gather():
    from xkv_b200 import compress, factorize, synthetic

    keys = [t.cuda().contiguous() for t in synthetic.make_group_kv(2, 2, 512, 64, 1.0, seed=7)]   # (1, H, S, D) head-major
    assert factorize.layer_rows(keys[0]) is None
    (gf,) = compress.compress_groups([keys], [keys], 32, 32)
    torch.cuda.synchronize()
    assert torch.isfinite(gf.key.A).all()
