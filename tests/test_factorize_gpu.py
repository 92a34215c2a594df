"""GPU parity of the stored factorisation against the reference's own torch SVD path.

Reference: fake_svd (fake_layer_merge_dynamic_cache.py:11-29) = torch.linalg.svd in fp32, truncate,
multiply back, cast to the cache dtype (:176).  Factors are compared through the reconstruction
(singular vectors are sign/rotation ambiguous).  Tolerances are BASELINE.json's:
  * relative Frobenius reconstruction error <= 1.01 x the reference's at equal rank,
  * leading singular values within 1e-3 relative.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ref_fake_svd(x_bf16: torch.Tensor, rank: int):
    """The reference's arithmetic on the same device: fp32 SVD, truncate, multiply back, cast to bf16."""
    x = x_bf16.float()[None]  # (bs=1, S, n), as fake_svd sees it after its reshape
    u, s, vh = torch.linalg.svd(x, full_matrices=False)
    approx = torch.matmul(u[:, :, :rank], torch.matmul(torch.diag_embed(s[:, :rank]), vh[:, :rank, :]))
    return approx[0].to(torch.bfloat16), s[0]


def _rel_err(x, xh):
    x = x.double()
    return (torch.linalg.norm(x - xh.double()) / torch.linalg.norm(x)).item()


@pytest.mark.parametrize(
    "tokens,cols,rank,alpha",
    [
        (1024, 1024, 128, 1.0),    # single-layer shape (config 3 columns), skinny rank
        (1024, 1024, 192, 0.5),
        (2048, 2048, 256, 1.0),
        (4096, 4096, 512, 1.0),    # config 1, K rank
        (4096, 4096, 768, 0.5),    # config 1, V rank
        (4096, 4096, 512, None),   # i.i.d. Gaussian: worst case for any low-rank method
        (1536, 2048, 512, 1.0),    # fewer tokens than columns
        (2048, 8192, 1024, 0.5),   # config 4 columns (xKV-8 on 8 kv heads x 128): sketch width 1088, 17 Cholesky blocks
    ],
)
def test_reconstruction_matches_reference_svd(tokens, cols, rank, alpha):
    from xkv_b200 import factorize, synthetic

    x = synthetic.group_matrix(tokens, cols, alpha, seed=1234, device="cuda")
    ref_hat, s_ref = _ref_fake_svd(x, rank)
    (f,) = factorize.factorize_batch([x], rank)
    torch.cuda.synchronize()
    assert f.A.shape == (tokens, rank) and f.Vt.shape == (rank, cols) and f.V.shape == (cols, rank)
    assert torch.equal(f.V, f.Vt.t())
    e_ref = _rel_err(x, ref_hat)
    e_ours = _rel_err(x, f.reconstruct())
    print(f"tokens={tokens} cols={cols} r={rank} alpha={alpha}: err ref={e_ref:.6f} ours={e_ours:.6f} "
          f"ratio={e_ours / e_ref:.5f}")
    assert e_ours <= 1.01 * e_ref
    # right factor is orthonormal (to bf16 rounding)
    vt = f.Vt.float()
    assert (vt @ vt.t() - torch.eye(rank, device="cuda")).abs().max().item() < 2e-2
    if alpha is not None:
        k = 16
        rel = ((f.sigma_lead[:k] - s_ref[:k]).abs() / s_ref[:k]).max().item()
        print(f"   leading singular values: max rel dev {rel:.2e}")
        assert rel < 1e-3


def test_steep_spectrum_at_high_rank_meets_the_bf16_storage_floor():
    """Where the reference's own error drops below ~2 % (steep spectrum, high rank: config 4 columns at alpha = 1,
    rank 1024) the 1 % criterion is tighter than what factors STORED in bf16 can deliver: rounding A and V adds
    ~0.3 % of ||X|| in quadrature (DESIGN.md section 2, "known floor"; the reference rounds the dense product once).
    The algorithmic part must still be within 1 %: the excess over the reference is bounded by that floor."""
    from xkv_b200 import factorize, synthetic

    x = synthetic.group_matrix(2048, 8192, 1.0, seed=1234, device="cuda")
    ref_hat, _ = _ref_fake_svd(x, 1024)
    (f,) = factorize.factorize_batch([x], 1024)
    torch.cuda.synchronize()
    e_ref, e_ours = _rel_err(x, ref_hat), _rel_err(x, f.reconstruct())
    print(f"steep/high-rank: err ref={e_ref:.6f} ours={e_ours:.6f} ratio={e_ours / e_ref:.5f}")
    assert e_ref < 0.02
    assert e_ours ** 2 <= (1.01 * e_ref) ** 2 + 3e-3 ** 2


@pytest.mark.parametrize(
    "tokens,cols,rank,alpha",
    [
        (520, 4096, 512, 1.0),    # short prompt: fewer tokens than the sketch is wide (576): rank-deficient Gram
        (577, 2048, 512, 0.5),    # odd token count
        (1000, 1024, 128, 1.0),   # tokens < columns, not a multiple of the tile
        (130, 1024, 128, 1.0),    # rank just below the token count
        (4096, 4096, 500, 1.0),   # rank not a multiple of 64 (ragged Rayleigh-Ritz window)
        (4096, 4096, 1, 1.0),     # rank 1
        (3000, 4096, 37, 0.5),
    ],
)
def test_ragged_short_and_odd_inputs(tokens, cols, rank, alpha):
    """Edge cases of the reference's slicing semantics (cache:21-23): any 0 < rank < min(tokens, columns) must give the
    truncated SVD.  Where the reference's error is tiny (rank close to the token count) the bf16 storage of the factors
    enters in quadrature, as in the steep-spectrum test below."""
    from xkv_b200 import factorize, synthetic

    x = synthetic.group_matrix(tokens, cols, alpha, seed=5, device="cuda")
    ref_hat, _ = _ref_fake_svd(x, rank)
    (f,) = factorize.factorize_batch([x], rank)
    torch.cuda.synchronize()
    e_ref, e_ours = _rel_err(x, ref_hat), _rel_err(x, f.reconstruct())
    print(f"tokens={tokens} cols={cols} r={rank}: err ref={e_ref:.6f} ours={e_ours:.6f}")
    assert torch.isfinite(f.A).all() and torch.isfinite(f.Vt).all()
    assert e_ours ** 2 <= (1.01 * e_ref) ** 2 + 3e-3 ** 2


def _colscale(m, n, p):
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(m, n, device="cuda", generator=g)
    x *= torch.arange(1, n + 1, device="cuda") ** -p
    return x.to(torch.bfloat16)


def _outliers(m, n, alpha, k, gain):
    from xkv_b200 import synthetic

    x = synthetic.group_matrix(m, n, alpha, seed=3, device="cuda").float()
    x[:, torch.arange(k, device="cuda") * 97 % n] *= gain
    return (x * (4.0 / x.abs().max())).to(torch.bfloat16)


@pytest.mark.parametrize(
    "name,make,rank",
    [
        ("unmixed columns, scales i^-0.7", lambda: _colscale(4096, 2048, 0.7), 448),
        ("unmixed columns, scales i^-1", lambda: _colscale(4096, 2048, 1.0), 512),
        ("4 outlier channels x30, alpha 1", lambda: _outliers(4096, 4096, 1.0, 4, 30.0), 512),
        ("4 outlier channels x30, alpha 0.5", lambda: _outliers(4096, 4096, 0.5, 4, 30.0), 768),
        ("8 outlier channels x300", lambda: _outliers(4096, 4096, 1.0, 8, 300.0), 512),
    ],
)
def test_energy_concentrated_in_a_few_channels(name, make, rank):
    """KV caches of real models carry a few massive channels.  With the energy in a few columns the rounding errors of
    the bf16 limbs add up coherently (a 3-term first pass broke down -> NaN on every one of these inputs; it is 6-term
    now), and with a gain of 300 the Gram of the once-orthogonalised sketch is numerically indefinite: the lightly
    shifted Cholesky is then redone heavily shifted on a device decision.  The bf16 storage of A and V is relative to the
    outlier channels' magnitude and enters in quadrature (4e-3: two factor roundings + the product's, vs the
    reference's single rounding of the dense product)."""
    from xkv_b200 import factorize

    x = make()
    ref_hat, s_ref = _ref_fake_svd(x, rank)
    (f,) = factorize.factorize_batch([x], rank)
    torch.cuda.synchronize()
    assert torch.isfinite(f.A).all() and torch.isfinite(f.Vt).all(), name
    e_ref, e_ours = _rel_err(x, ref_hat), _rel_err(x, f.reconstruct())
    print(f"{name}: err ref={e_ref:.6f} ours={e_ours:.6f}")
    assert e_ours ** 2 <= (1.01 * e_ref) ** 2 + 4e-3 ** 2
    rel = ((f.sigma_lead[:16] - s_ref[:16]).abs() / s_ref[:16]).max().item()
    assert rel < 2e-3


def test_device_decided_second_pass():
    """Single-pass power steps add a second CholeskyQR pass per matrix on a DEVICE decision (a Cholesky pivot below
    0.05).  A batch mixing a benign and a steep matrix must meet the bar for both."""
    from xkv_b200 import factorize, synthetic

    xs = [synthetic.group_matrix(2048, 4096, a, seed=77 + i, device="cuda") for i, a in enumerate((0.5, 1.0))]
    fs = factorize.factorize_batch(xs, 512)
    torch.cuda.synchronize()
    for x, f, a in zip(xs, fs, (0.5, 1.0)):
        ref_hat, _ = _ref_fake_svd(x, 512)
        e_ref, e_ours = _rel_err(x, ref_hat), _rel_err(x, f.reconstruct())
        print(f"alpha={a}: err ref={e_ref:.6f} ours={e_ours:.6f} ratio={e_ours / e_ref:.5f}")
        assert e_ours <= 1.01 * e_ref


def test_batch_of_two_ranks_shapes_and_determinism():
    from xkv_b200 import factorize, synthetic

    xs = [synthetic.group_matrix(1024, 1024, 1.0, seed=s, device="cuda") for s in (1, 2, 3)]
    f1 = factorize.factorize_batch(xs, 128)
    f2 = factorize.factorize_batch(xs, 128)
    torch.cuda.synchronize()
    for a, b in zip(f1, f2):
        assert torch.equal(a.A, b.A) and torch.equal(a.Vt, b.Vt)   # same seed -> bit-identical factors
    assert not torch.equal(f1[0].Vt, f1[1].Vt)


def test_rejects_rank_that_does_not_fit():
    from xkv_b200 import _lib, factorize

    x = torch.zeros(64, 256, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(_lib.XkvError):
        factorize.factorize_batch([x], 128)      # rank > tokens
    with pytest.raises(_lib.XkvError):
        factorize.factorize_batch([torch.zeros(512, 256, device="cuda", dtype=torch.bfloat16)], 256)  # sketch > cols
