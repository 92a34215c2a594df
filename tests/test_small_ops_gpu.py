"""GPU checks of the small fp32 kernels against torch (each is a restatement of one torch call)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def test_reduce_slabs_and_symmetrize():
    from xkv_b200 import ops

    torch.manual_seed(0)
    slabs = torch.randn(3, 200, 200, device="cuda")
    out = torch.empty(200, 200, device="cuda")
    ops.reduce_slabs(slabs, out, symmetrize=False)
    torch.cuda.synchronize()
    assert torch.allclose(out, slabs.sum(0), atol=1e-5)
    ops.reduce_slabs(slabs, out, symmetrize=True)
    torch.cuda.synchronize()
    up = torch.triu(slabs.sum(0))
    ref = up + torch.triu(up, 1).t()
    assert torch.allclose(out, ref, atol=1e-5)


@pytest.mark.parametrize("n,slabs_n", [(200, 3), (256, 1), (40, 2)])
def test_symmetrize_split_equals_reduce_then_split(n, slabs_n):
    """One-pass Gram post-processing = reduce_slabs(symmetrize) followed by split_bf16, bit for bit; garbage below the
    diagonal of the slabs (tiles the symmetric GEMM never writes) must not leak."""
    from xkv_b200 import ops

    torch.manual_seed(1)
    batch = 3
    slabs = [torch.randn(slabs_n, n, n, device="cuda") * 11.0 for _ in range(batch)]
    ref = []
    for sl in slabs:
        g = torch.empty(n, n, device="cuda")
        ops.reduce_slabs(sl, g, symmetrize=True)
        limbs = [torch.empty(n, n, device="cuda", dtype=torch.bfloat16) for _ in range(3)]
        ops.split_bf16(g, *limbs)
        ref.append(limbs)
    poisoned = []
    for sl in slabs:
        p = sl.clone()
        low = torch.tril(torch.ones(n, n, device="cuda", dtype=torch.bool), -32)   # strictly below the diagonal tiles
        p[:, low] = float("nan")
        poisoned.append(p)
    hi, mid, lo = ([torch.full((n, n), 7.0, device="cuda", dtype=torch.bfloat16) for _ in range(batch)] for _ in range(3))
    ops.symmetrize_split_bf16(poisoned, hi, mid, lo)
    torch.cuda.synchronize()
    for b in range(batch):
        assert torch.equal(hi[b], ref[b][0]) and torch.equal(mid[b], ref[b][1]) and torch.equal(lo[b], ref[b][2])


def test_pass_flags_and_launch_predicate():
    """Device-side conditional passes: flags from the Cholesky pivots; predicated launches leave the skipped matrices'
    buffers untouched and process the others."""
    from xkv_b200 import ops

    l, dev = 128, "cuda"
    torch.manual_seed(3)
    good = torch.eye(l, device=dev) + 0.01 * torch.randn(l, l, device=dev)
    good = (good + good.t()) / 2
    v = torch.randn(l, 3, device=dev)
    bad = (v @ v.t()) / 3 + 1e-4 * torch.eye(l, device=dev)      # numerically rank 3: tiny pivots after the third
    bad = bad / bad.diagonal().max()
    ss = [good.clone(), bad.clone(), good.clone()]
    linvs = [torch.full((l, l), 7.0, device=dev) for _ in ss]
    ops.cholesky_inverse(ss, linvs, shift=1e-6)
    flags = torch.full((3,), -1, device=dev, dtype=torch.int32)
    ops.pass_flags(linvs, 0.05, flags)
    torch.cuda.synchronize()
    assert flags.tolist() == [0, 1, 0]
    # predicated Cholesky: only matrix 1 is redone (heavier shift); the others keep their inverse bit for bit
    before = [t.clone() for t in linvs]
    ss2 = [good.clone(), bad.clone(), good.clone()]
    with ops.launch_predicate(flags):
        ops.cholesky_inverse(ss2, linvs, shift=3e-4)
    torch.cuda.synchronize()
    assert torch.equal(linvs[0], before[0]) and torch.equal(linvs[2], before[2])
    assert not torch.equal(linvs[1], before[1])
    assert torch.equal(ss2[0], good) and torch.equal(ss2[2], good)          # S of a skipped matrix is not even touched
    # predicated row normalisation
    ys = [torch.randn(8, 64, device=dev) * 5 for _ in range(3)]
    keep = [y.clone() for y in ys]
    with ops.launch_predicate(flags):
        ops.shift_normalize_rows(ys)
    torch.cuda.synchronize()
    assert torch.equal(ys[0], keep[0]) and torch.equal(ys[2], keep[2])
    assert torch.allclose(ys[1].norm(dim=1), torch.ones(8, device=dev), atol=1e-5)
    # outside the context everything runs again
    ops.shift_normalize_rows(ys)
    torch.cuda.synchronize()
    assert torch.allclose(ys[0].norm(dim=1), torch.ones(8, device=dev), atol=1e-5)
    # a full 16-matrix predicated Cholesky at sketch width 1600 (25 blocks, the widest clusters), every other matrix
    # skipped: the skipped ones at b >= 8 keep S and Linv bit for bit, the others get what an unpredicated launch gives
    l, batch = 1600, 16
    torch.manual_seed(4)
    grams = [_unit_row_gram(l).float() for _ in range(batch)]
    flags = torch.tensor([b % 2 for b in range(batch)], device=dev, dtype=torch.int32)
    ss = [g.clone() for g in grams]
    linvs = [torch.full((l, l), 7.0, device=dev) for _ in range(batch)]
    with ops.launch_predicate(flags):
        ops.cholesky_inverse(ss, linvs, shift=1e-6)
    singles = []
    for b in range(1, batch, 2):
        li = torch.full((l, l), float("nan"), device=dev)
        ops.cholesky_inverse([grams[b].clone()], [li], shift=1e-6)
        singles.append(li)
    torch.cuda.synchronize()
    for b in range(0, batch, 2):
        assert torch.equal(ss[b], grams[b]), f"S of skipped matrix {b} was written"
        assert (linvs[b] == 7.0).all(), f"Linv of skipped matrix {b} was written"
    for b, li in zip(range(1, batch, 2), singles):
        assert torch.equal(linvs[b], li), f"predicated matrix {b} differs from its own launch"


def test_split_bf16_limbs_reconstruct_fp32():
    from xkv_b200 import ops

    x = torch.randn(64, 256, device="cuda") * 37.0
    h, m, l = (torch.empty(64, 256, device="cuda", dtype=torch.bfloat16) for _ in range(3))
    ops.split_bf16(x, h, m, l)
    torch.cuda.synchronize()
    assert torch.equal(h, x.bfloat16())
    rec = h.float() + m.float() + l.float()
    assert (rec - x).abs().max().item() <= 2e-7 * x.abs().max().item()


def test_fill_gaussian_is_deterministic_and_normal():
    from xkv_b200 import ops

    a = torch.empty(512, 1024, device="cuda", dtype=torch.bfloat16)
    b = torch.empty_like(a)
    ops.fill_gaussian_bf16(a, 7)
    ops.fill_gaussian_bf16(b, 7)
    torch.cuda.synchronize()
    assert torch.equal(a, b)
    af = a.float()
    assert abs(af.mean().item()) < 0.01 and abs(af.std().item() - 1.0) < 0.01
    ops.fill_gaussian_bf16(b, 8)
    torch.cuda.synchronize()
    assert not torch.equal(a, b)


def test_normalize_rows_with_limbs():
    from xkv_b200 import ops

    ys = [torch.randn(64, 512, device="cuda") * (i + 1) for i in range(3)]
    ref = [y / y.norm(dim=1, keepdim=True) for y in ys]
    hi = [torch.empty(64, 512, device="cuda", dtype=torch.bfloat16) for _ in ys]
    mid = [torch.empty_like(h) for h in hi]
    lo = [torch.empty_like(h) for h in hi]
    ops.normalize_rows(ys, hi, mid, lo)
    torch.cuda.synchronize()
    for y, r, h, m, l in zip(ys, ref, hi, mid, lo):
        assert torch.allclose(y, r, atol=1e-6)
        assert (h.float() + m.float() + l.float() - y).abs().max().item() < 1e-7


def test_shift_normalize_rows_and_rdiag():
    """Y <- Y - c Q, unit rows + limbs, diag(R) bookkeeping and the shift update."""
    from xkv_b200 import ops

    torch.manual_seed(3)
    qs = [torch.linalg.qr(torch.randn(512, 64, device="cuda"))[0].t().contiguous() for _ in range(3)]
    ys = [q * torch.linspace(5.0, 1.0, 64, device="cuda")[:, None] + 0.01 * torch.randn(64, 512, device="cuda") for q in qs]
    shifts = torch.tensor([0.25, 0.5, 0.0], device="cuda")
    zs = [y - c * q for y, q, c in zip(ys, qs, shifts)]
    norms = [z.norm(dim=1) for z in zs]
    refs = [z / nz[:, None] for z, nz in zip(zs, norms)]
    hi = [torch.empty(64, 512, device="cuda", dtype=torch.bfloat16) for _ in ys]
    mid = [torch.empty_like(h) for h in hi]
    rdiag = [torch.full((64,), 7.0, device="cuda") for _ in ys]
    ops.shift_normalize_rows(ys, qs, shifts, rdiag, True, hi, mid, None)
    torch.cuda.synchronize()
    for y, r, h, m, rd, nz in zip(ys, refs, hi, mid, rdiag, norms):
        assert torch.allclose(y, r, atol=1e-6)
        assert (h.float() + m.float() - y).abs().max().item() < 1e-4
        assert torch.allclose(rd, nz, rtol=1e-5)
    # second pass multiplies the norms in; the Cholesky diagonal divides by Linv_jj
    ys2 = [torch.randn(64, 512, device="cuda") for _ in ys]
    n2 = [y.norm(dim=1) for y in ys2]
    ops.shift_normalize_rows(ys2, None, None, rdiag, False)
    linvs = [torch.rand(64, 64, device="cuda") + 0.5 for _ in ys]
    ops.rdiag_update(rdiag, linvs)
    torch.cuda.synchronize()
    for rd, a, b, li in zip(rdiag, norms, n2, linvs):
        assert torch.allclose(rd, a * b / li.diagonal(), rtol=1e-5)
    c_ref = torch.stack([0.5 * (rd[-8:].mean() + c) for rd, c in zip(rdiag, shifts)])
    ops.ritz_shift_update(rdiag, shifts, 8, 0.5)
    torch.cuda.synchronize()
    assert torch.allclose(shifts, c_ref, rtol=1e-5)


def _unit_row_gram(l):
    """fp64 S = Y Y^T of an l x 3l Gaussian Y with unit rows: the Gram CholeskyQR factors (condition ~14 at any l)."""
    y = torch.randn(l, 3 * l, device="cuda", dtype=torch.float64)
    y = y / y.norm(dim=1, keepdim=True)
    return y @ y.t()


@pytest.mark.parametrize("l,cond", [(64, 10.0), (192, 1e3), (576, 1e4), (832, 1e2), (1600, 1e3)])
def test_cholesky_inverse(l, cond):
    from xkv_b200 import ops

    torch.manual_seed(l)
    batch = 3
    ss, refs, linvs = [], [], []
    for b in range(batch):
        q = torch.linalg.qr(torch.randn(l, l, device="cuda", dtype=torch.float64))[0]
        ev = torch.logspace(0, -torch.log10(torch.tensor(cond)).item(), l, device="cuda", dtype=torch.float64)
        s = (q * ev) @ q.t()
        d = s.diagonal().rsqrt()
        s = s * d[:, None] * d[None, :]      # unit diagonal, as after row normalisation
        refs.append(s)
        ss.append(s.float().contiguous())
        linvs.append(torch.full((l, l), float("nan"), device="cuda"))
    ops.cholesky_inverse(ss, linvs, shift=0.0, pivot_floor=1e-9)
    torch.cuda.synchronize()
    for s64, li in zip(refs, linvs):
        assert not torch.isnan(li).any()
        assert torch.equal(torch.triu(li, 1), torch.zeros_like(li))
        eye = li.double() @ s64 @ li.double().t()
        err = (eye - torch.eye(l, device="cuda", dtype=torch.float64)).abs().max().item()
        assert err < 5e-3 * max(1.0, cond / 1e3), f"Linv S Linv^T deviates from I by {err}"


@pytest.mark.parametrize("l,batch", [
    (128, 1), (320, 2), (576, 8), (1088, 2),
    (256, 1), (512, 2), (1024, 3),   # 4, 8 and 16 blocks: the inverse phase's super-block pairs come out even
    (1216, 1),                       # 19 blocks: the widest 8-CTA cluster
    (1280, 1),                       # 20 blocks: the narrowest 16-CTA cluster
    (1408, 2), (1600, 1),            # the sketch widths of ranks 1344 and 1536 (non-uniform config, config 4 V)
    (1600, 16),                      # a full batch of the widest: 16 clusters of 16 CTAs if the device keeps them resident
])
def test_cholesky_inverse_limbs_match_fp32_inverse(l, batch):
    """The fused kernel's bf16 limbs of Linv (the GEMM operand) add up to the fp32 Linv it writes; the inverse
    agrees with torch's Cholesky + triangular solve in fp64.  The cluster size follows the number of 64-column blocks
    (1, 2, 4, 8 CTAs; 16 from 20 blocks), so the widths cover every size.  S is well conditioned (~14 at any l), and
    the fp32 error of its Cholesky inverse grows only slowly with l (LAPACK's fp32 factor and triangular solve: 2.4e-7
    relative at l = 1088, 2.5e-7 at l = 1600), so the 1e-4 bound of the narrow cases holds for the widest ones too."""
    from xkv_b200 import ops

    torch.manual_seed(l + batch)
    ss, refs = [], []
    for b in range(batch):
        s = _unit_row_gram(l)
        refs.append(torch.linalg.inv(torch.linalg.cholesky(s + 1e-6 * torch.eye(l, device="cuda", dtype=torch.float64))))
        ss.append(s.float().contiguous())
    linvs = [torch.full((l, l), float("nan"), device="cuda") for _ in range(batch)]
    limbs = [[torch.full((l, l), float("nan"), device="cuda", dtype=torch.bfloat16) for _ in range(batch)] for _ in range(3)]
    ops.cholesky_inverse(ss, linvs, shift=1e-6, pivot_floor=1e-12, limbs=limbs)
    torch.cuda.synchronize()
    for b in range(batch):
        li = linvs[b]
        assert not torch.isnan(li).any()
        assert torch.equal(torch.triu(li, 1), torch.zeros_like(li))
        rel = (li.double() - refs[b]).abs().max().item() / refs[b].abs().max().item()
        print(f"l={l} matrix {b}/{batch}: Linv rel. deviation {rel:.2e}")
        assert rel < 1e-4, f"Linv deviates from the fp64 inverse by {rel}"
        total = limbs[0][b].float() + limbs[1][b].float() + limbs[2][b].float()
        assert (total - li).abs().max().item() <= 1e-6 * li.abs().max().item()


@pytest.mark.parametrize("l", [576, 1280, 1600])
def test_cholesky_inverse_is_independent_of_batch_position_and_strides(l):
    """The same S matrices in one 16-matrix launch and in 16 single-matrix launches give bit-identical Linv and limbs.
    Each output tile's products are applied in a fixed (k, t) order whichever CTA of the cluster runs them, and the
    matrices of a launch are independent along blockIdx.y; so neither the batch position nor the cluster size (from 20
    blocks on, a single matrix gets 16 CTAs and a full batch 16 or 8 depending on how many 16-CTA clusters the device
    keeps resident) may change a bit.  The batched launch also reads S and writes Linv with rows l + 64 apart and the
    limbs with rows l + 24 apart; the NaN in the padding columns must stay untouched."""
    from xkv_b200 import ops

    torch.manual_seed(17 + l)
    batch, nan = 16, float("nan")
    grams = [_unit_row_gram(l).float() for _ in range(batch)]

    def padded(pad, dtype):
        return torch.full((l, l + pad), nan, device="cuda", dtype=dtype)

    s_buf = [padded(64, torch.float32) for _ in range(batch)]
    for buf, g in zip(s_buf, grams):
        buf[:, :l] = g
    li_buf = [padded(64, torch.float32) for _ in range(batch)]
    limb_buf = [[padded(24, torch.bfloat16) for _ in range(batch)] for _ in range(3)]
    ops.cholesky_inverse([t[:, :l] for t in s_buf], [t[:, :l] for t in li_buf], shift=1e-6, pivot_floor=1e-12,
                         limbs=[[t[:, :l] for t in side] for side in limb_buf])
    singles = []
    for g in grams:
        li = torch.full((l, l), nan, device="cuda")
        limbs = [[torch.full((l, l), nan, device="cuda", dtype=torch.bfloat16)] for _ in range(3)]
        ops.cholesky_inverse([g.clone()], [li], shift=1e-6, pivot_floor=1e-12, limbs=limbs)
        singles.append((li, [side[0] for side in limbs]))
    torch.cuda.synchronize()
    for b, (li, limbs) in enumerate(singles):
        assert not torch.isnan(li).any()
        assert torch.equal(li_buf[b][:, :l], li), f"Linv of matrix {b} depends on the launch"
        for i, (side, one) in enumerate(zip(limb_buf, limbs)):
            assert torch.equal(side[b][:, :l], one), f"limb {i} of matrix {b} depends on the launch"
        for t in [s_buf[b], li_buf[b]] + [side[b] for side in limb_buf]:
            assert torch.isnan(t[:, l:]).all(), f"padding of matrix {b} was written"


def test_cholesky_inverse_rejects_batches_with_mixed_layouts():
    """The library takes one row stride for every S and Linv (S's) and one for every limb (hi[0]'s): a batch whose
    matrices differ in shape or stride is refused before anything is launched.  (Every odd matrix here is larger than
    what the library would address, so a launch that is not refused stays in bounds.)"""
    from xkv_b200 import _lib, ops

    l, nan = 128, float("nan")
    s = _unit_row_gram(l).float()
    big = _unit_row_gram(l + 64).float()

    def linvs():
        return [torch.full((l, l), nan, device="cuda") for _ in range(2)]

    def limbs():
        return [[torch.full((l, l), nan, device="cuda", dtype=torch.bfloat16) for _ in range(2)] for _ in range(3)]

    wide = torch.full((l, l + 64), nan, device="cuda")
    wide_limb = torch.full((l, l + 64), nan, device="cuda", dtype=torch.bfloat16)
    cases = {
        "Linv strided unlike S": ([s.clone(), s.clone()], [linvs()[0], wide[:, :l]], None),
        "S strided unlike ss[0]": ([s.clone(), big[:l, :l]], linvs(), None),
        "S of another size": ([s.clone(), big.clone()], linvs(), None),
        "Linv of another size": ([s.clone(), s.clone()], [linvs()[0], torch.full((l + 64, l + 64), nan, device="cuda")],
                                 None),
        "fp64 S": ([s.clone(), s.double()], linvs(), None),
        "mid limb strided unlike hi[0]": ([s.clone(), s.clone()], linvs(), limbs()),
        "hi limb strided unlike hi[0]": ([s.clone(), s.clone()], linvs(), limbs()),
    }
    cases["mid limb strided unlike hi[0]"][2][1][1] = wide_limb[:, :l]
    cases["hi limb strided unlike hi[0]"][2][0][1] = wide_limb[:, :l]
    for name, (ss, lis, lb) in cases.items():
        with pytest.raises(_lib.XkvError):
            ops.cholesky_inverse(ss, lis, shift=1e-6, limbs=lb)
            torch.cuda.synchronize()
            pytest.fail(f"{name}: accepted")
    torch.cuda.synchronize()
    assert torch.isnan(wide).all() and torch.isnan(wide_limb).all()


def test_cholesky_shift_keeps_indefinite_gram_finite():
    """The fp32 Gram of a nearly rank-deficient sketch is indefinite; the shifted factorisation must stay
    finite and equal the factor of S + shift*I."""
    from xkv_b200 import ops

    torch.manual_seed(3)
    l = 192
    u = torch.randn(l, 6, device="cuda", dtype=torch.float64)
    s = u @ u.t()
    d = s.diagonal().rsqrt()
    s = s * d[:, None] * d[None, :] + 1e-6 * torch.randn(l, l, device="cuda", dtype=torch.float64)
    s = 0.5 * (s + s.t())
    s32 = s.float().contiguous()
    linv = torch.full((l, l), float("nan"), device="cuda")
    shift = 1e-3
    ops.cholesky_inverse([s32.clone()], [linv], shift=shift, pivot_floor=1e-12)
    torch.cuda.synchronize()
    assert torch.isfinite(linv).all()
    ref = torch.linalg.inv(torch.linalg.cholesky(s32.double() + shift * torch.eye(l, device="cuda", dtype=torch.float64)))
    assert ((linv.double() - ref).norm() / ref.norm()).item() < 1e-2


@pytest.mark.parametrize("w", [32, 128, 160])
def test_jacobi_window_eigh(w):
    from xkv_b200 import ops

    torch.manual_seed(w)
    count = 5
    ts, refs = [], []
    for b in range(count):
        a = torch.randn(w, w, device="cuda", dtype=torch.float64)
        s = a @ a.t() / w + torch.diag(torch.linspace(3, 0, w, device="cuda", dtype=torch.float64))
        refs.append(s)
        ts.append(s.float().contiguous())
    evals = [torch.empty(w, device="cuda") for _ in range(count)]
    wts = [torch.empty(w, w, device="cuda") if b != 1 else None for b in range(count)]
    ops.jacobi_eigh(ts, evals, wts, sweeps=10)
    torch.cuda.synchronize()
    for s64, ev, wt in zip(refs, evals, wts):
        ref = torch.linalg.eigvalsh(s64).flip(0)
        assert torch.allclose(ev.double(), ref, rtol=1e-4, atol=1e-5)
        if wt is not None:
            wd = wt.double()
            assert (wd @ wd.t() - torch.eye(w, device="cuda", dtype=torch.float64)).abs().max().item() < 1e-4
            assert (wd @ s64 @ wd.t() - torch.diag(ev.double())).abs().max().item() < 1e-3


def test_convert_bf16_and_transpose():
    from xkv_b200 import ops

    x = torch.randn(100, 264, device="cuda")
    d = torch.empty(100, 264, device="cuda", dtype=torch.bfloat16)
    dt = torch.empty(264, 104, device="cuda", dtype=torch.bfloat16)[:, :100]
    ops.convert_bf16(x, d, dt)
    torch.cuda.synchronize()
    assert torch.equal(d, x.bfloat16())
    assert torch.equal(dt, x.bfloat16().t())


def test_slerp_merge_matches_reference_function():
    """SLERP / MiniCache branch against the oracle's restatement of fake_minicache_merge (pinned to the
    reference by tests/golden) on bf16 rows; the kernel computes in fp32, the reference in the tensor dtype."""
    from oracle import xkv_oracle as O
    from xkv_b200 import ops

    torch.manual_seed(4)
    rows, d = 4096, 128
    x1 = torch.randn(rows, d, device="cuda").bfloat16()
    x2 = (x1.float() + 0.4 * torch.randn(rows, d, device="cuda")).bfloat16()
    x2[7] = (x1[7].float() * 2.0).bfloat16()          # a parallel row -> linear-interpolation branch
    e1, e2 = ops.slerp_merge(x1, x2, 0.6, 0.05)
    torch.cuda.synchronize()
    r1, r2 = O.fake_minicache_merge(x1.float(), x2.float(), t=0.6, gamma=0.05)
    for got, ref in ((e1, r1), (e2, r2)):
        err = (got.float() - ref).abs().max().item() / ref.abs().max().item()
        assert err < 2e-2
    # rows below the divergence threshold are copied through untouched (reference cache:96-99)
    _, mask, _, _ = O.slerp_merge_rows_batch(x1.float(), x2.float(), t=0.6, gamma=0.05)
    keep = ~mask.squeeze(-1)
    assert keep.any() and torch.equal(e1[keep], x1[keep]) and torch.equal(e2[keep], x2[keep])


@pytest.mark.parametrize("n", [64, 200, 1024, 4096])
def test_gram_pack_unpack_upper(n):
    """Payload of the token-sharded Gram all-reduce: pack keeps row r's columns from 32 * (r // 32); unpack mirrors the
    upper triangle. Bit-exact against indexing."""
    from xkv_b200 import ops

    g = torch.randn(n, n, device="cuda")
    g = g + g.t()
    packed = ops.gram_pack_upper(g)
    assert packed.numel() == ops.gram_packed_elems(n)
    ref = torch.cat([g[r, (r // 32) * 32:] for r in range(0, n, max(1, n // 64))])   # spot rows
    offs = [0]
    for r in range(n):
        offs.append(offs[-1] + n - (r // 32) * 32)
    got = torch.cat([packed[offs[r]: offs[r + 1]] for r in range(0, n, max(1, n // 64))])
    assert torch.equal(got, ref)
    noisy = g + torch.tril(torch.randn(n, n, device="cuda"), -1)     # garbage below the diagonal must not survive
    full = torch.empty(n, n, device="cuda")
    ops.gram_unpack_upper(ops.gram_pack_upper(noisy), full)
    torch.cuda.synchronize()
    assert torch.equal(full, g)
