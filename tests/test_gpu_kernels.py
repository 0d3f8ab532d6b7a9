"""Parity of the CUDA path (through the C ABI) against the CPU oracle -- kernels in isolation.

Tolerances: embeddings / projections 1e-4 relative (north star); indices bit-exact on identical scores.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import mmrec_oracle as O  # noqa: E402


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from mmrec_b200 import _lib
    _lib.require_device()
    return torch.device("cuda:0")


def rel(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def rand_coo(n_rows, n_cols, nnz, seed, dup_frac=0.1):
    g = torch.Generator().manual_seed(seed)
    r = torch.randint(0, n_rows, (nnz,), generator=g)
    c = torch.randint(0, n_cols, (nnz,), generator=g)
    nd = int(nnz * dup_frac)
    if nd:
        src = torch.randint(0, nnz, (nd,), generator=g)
        r = torch.cat([r, r[src]]); c = torch.cat([c, c[src]])
    v = torch.rand(r.numel(), generator=g) - 0.5
    p = torch.randperm(r.numel(), generator=g)
    return r[p], c[p], v[p]


# ------------------------------------------------------------------------------------------------ K1c
@pytest.mark.parametrize("n_rows,n_cols,nnz", [(1, 1, 1), (7, 5, 0), (300, 200, 5000), (2000, 3000, 40000), (5, 100000, 3000)])
def test_csr_from_coo_coalesce_semantics(dev, n_rows, n_cols, nnz):
    from mmrec_b200.ops import CSR
    r, c, v = rand_coo(n_rows, n_cols, nnz, seed=nnz + n_rows)
    A = CSR.from_coo(r.to(dev), c.to(dev), v.to(dev), n_rows, n_cols)
    ref = torch.sparse_coo_tensor(torch.stack([r, c]), v, (n_rows, n_cols)).coalesce()
    assert A.nnz == ref._nnz()
    rp = A.rowptr.cpu().numpy()
    assert rp[0] == 0 and rp[-1] == A.nnz and np.all(np.diff(rp) >= 0)
    if A.nnz:
        rows, cols, vals = [t.cpu() for t in A.coo()]
        assert np.array_equal(torch.stack([rows, cols]).numpy(), ref.indices().numpy())       # row-major, sorted cols
        np.testing.assert_allclose(vals.numpy(), ref.values().numpy(), rtol=1e-6, atol=1e-7)
    # duplicates kept when asked
    B = CSR.from_coo(r.to(dev), c.to(dev), None, n_rows, n_cols, sum_duplicates=False)
    assert B.nnz == r.numel()


def test_csr_transpose_and_plan(dev):
    from mmrec_b200.ops import CSR
    r, c, v = rand_coo(500, 300, 8000, seed=3, dup_frac=0)
    # one very long row so that the plan must split it
    r = torch.cat([r, torch.full((3000,), 7)]); c = torch.cat([c, torch.randint(0, 300, (3000,))]); v = torch.cat([v, torch.rand(3000)])
    A = CSR.from_coo(r.to(dev), c.to(dev), v.to(dev), 500, 300, seg=128)
    assert A.longest_row >= 290 and A.n_split >= 1 and A.n_tasks > 500 and A.n_slots >= 2
    t = A.tasks.cpu().numpy().reshape(-1, 4)
    lens = t[:, 2] - t[:, 1]
    assert lens.max() <= A.seg and lens.sum() == A.nnz
    assert np.all(np.diff(lens) <= 0)                       # sorted longest first ...
    assert A.n_cta_tasks == int((lens > A.light_max).sum())   # ... so the CTA-run tasks are a prefix
    At = A.t()
    np.testing.assert_allclose(At.to_dense().cpu().numpy(), A.to_dense().cpu().numpy().T, rtol=0, atol=0)


# ------------------------------------------------------------------------------------------------ K1
@pytest.mark.parametrize("d", [32, 64, 128, 256, 48, 5])
@pytest.mark.parametrize("use_plan", [True, False])
def test_spmm_matches_oracle(dev, d, use_plan):
    from mmrec_b200 import ops
    from mmrec_b200.ops import CSR
    n_rows, n_cols = 1500, 900
    r, c, v = rand_coo(n_rows, n_cols, 20000, seed=d)
    r = torch.cat([r, torch.full((2500,), 11), torch.full((700,), 1499)])
    c = torch.cat([c, torch.randint(0, n_cols, (3200,))]); v = torch.cat([v, torch.rand(3200) - 0.5])
    r[r == 5] = 6                                           # an empty row
    X = torch.randn(n_cols, d, generator=torch.Generator().manual_seed(1))
    A = CSR.from_coo(r.to(dev), c.to(dev), v.to(dev), n_rows, n_cols)
    ref = torch.sparse.mm(torch.sparse_coo_tensor(torch.stack([r, c]), v, (n_rows, n_cols)), X)
    Y = torch.full((n_rows, d), float("nan"), device=dev)
    ops.spmm_raw(A, X.to(dev), Y=Y, use_plan=use_plan)
    assert rel(Y, ref) < 1e-5
    assert torch.all(Y[5] == 0)
    # bit-reproducible run to run (fixed summation order, also for split rows)
    Y2 = torch.empty_like(Y)
    for _ in range(3):
        ops.spmm_raw(A, X.to(dev), Y=Y2, use_plan=use_plan)
        assert torch.equal(Y, Y2)
    assert int(A.counters.abs().sum().item()) == 0          # split-row counters are self-cleaning


@pytest.mark.parametrize("d", [64, 128, 40])
def test_spmm_fused_epilogues(dev, d):
    from mmrec_b200 import ops
    from mmrec_b200.ops import CSR
    n = 800
    r, c, v = rand_coo(n, n, 9000, seed=9)
    A = CSR.from_coo(r.to(dev), c.to(dev), v.to(dev), n, n)
    Ad = A.to_dense().cpu()
    X = torch.randn(n, d); base = torch.randn(n, d); ref0 = torch.randn(n, d)
    # acc_out = (acc_in + y) / div, in place
    acc = base.clone().to(dev)
    Y = torch.empty(n, d, device=dev)
    ops.spmm_raw(A, X.to(dev), Y=Y, acc_in=acc, acc_out=acc, acc_div=4.0)
    y = Ad @ X
    assert rel(Y, y) < 1e-5 and rel(acc, (base + y) / 4.0) < 1e-5
    # acc_out only, no acc_in
    acc2 = torch.empty(n, d, device=dev)
    ops.spmm_raw(A, X.to(dev), acc_out=acc2)
    assert rel(acc2, y) < 1e-5
    # LayerGCN gate (layergcn.py:132-133)
    Yg = torch.empty(n, d, device=dev)
    ops.spmm_raw(A, X.to(dev), Y=Yg, gate_ref=ref0.to(dev))
    w = torch.nn.functional.cosine_similarity(y, ref0, dim=-1)
    assert rel(Yg, w.unsqueeze(1) * y) < 1e-5


def test_propagate_mean_forward_backward_vs_oracle(dev, golden):
    from mmrec_b200 import graph, ops
    g = golden("freedom_tiny.npz")
    U, I = int(g["n_users"]), int(g["n_items"])
    adj = graph.build_norm_adj((g["inter_row"], g["inter_col"]), U, I, dev)
    oadj = O.norm_adj_coo(g["inter_row"], g["inter_col"], U, I)
    ego = torch.cat([torch.from_numpy(g["param0.user_embedding.weight"]), torch.from_numpy(g["param0.item_id_embedding.weight"])])
    for L in (0, 1, 2, 3, 4):
        e1 = ego.clone().to(dev).requires_grad_(True)
        e2 = ego.clone().requires_grad_(True)
        out = ops.propagate_mean(adj, e1, L)
        ref = O.propagate_mean(oadj, e2, L)
        assert rel(out, ref) < 1e-5
        w = torch.randn_like(ref)
        (out * w.to(dev)).sum().backward()
        (ref * w).sum().backward()
        assert rel(e1.grad, e2.grad) < 1e-5
    # spmm with base, directed matrix (needs the explicit transpose in backward)
    mm = torch.sparse_coo_tensor(torch.from_numpy(g["mm_adj_idx"]), torch.from_numpy(g["mm_adj_val"]), (I, I))
    M = ops.CSR.from_torch_sparse(mm.to(dev))
    assert M.nnz < g["mm_adj_val"].shape[0]                 # duplicates were summed
    h1 = ego[U:].clone().to(dev).requires_grad_(True); b1 = torch.randn(I, 64, device=dev, requires_grad=True)
    h2 = ego[U:].clone().requires_grad_(True); b2 = b1.detach().cpu().requires_grad_(True)
    o1 = ops.spmm(M, h1, base=b1); o2 = b2 + torch.sparse.mm(mm, h2)
    assert rel(o1, o2) < 1e-5
    w = torch.randn(I, 64)
    (o1 * w.to(dev)).sum().backward(); (o2 * w).sum().backward()
    assert rel(h1.grad, h2.grad) < 1e-5 and rel(b1.grad, b2.grad) < 1e-6


def test_bipartite_norm_and_pruning_vs_reference(dev, golden):
    from mmrec_b200 import graph
    g = golden("freedom_tiny.npz")
    U, I = int(g["n_users"]), int(g["n_items"])
    pr = graph.EdgePruner((g["inter_row"], g["inter_col"]), U, I, dev)
    assert np.array_equal(pr.edge_indices.cpu().numpy(), g["edge_indices"])
    ev = pr.edge_values.cpu().numpy()
    # 1/sqrt with IEEE sqrt+div: identical bits to torch.pow(x, -0.5) on CPU, or within 1 ulp
    assert np.max(np.abs(ev.view(np.int32).astype(np.int64) - g["edge_values"].view(np.int32).astype(np.int64))) <= 1
    A = pr.adj_from_keep(torch.from_numpy(g["prune_keep_idx"]).to(dev))
    n = U + I
    ref = torch.sparse_coo_tensor(torch.from_numpy(g["masked_adj_idx"]), torch.from_numpy(g["masked_adj_val"]), (n, n)).to_dense()
    np.testing.assert_allclose(A.to_dense().cpu().numpy(), ref.numpy(), rtol=2e-7, atol=0)
    assert A.nnz == g["masked_adj_val"].shape[0]
    A2, keep = pr.sample(float(g["cfg_dropout"]))
    assert keep.numel() == g["prune_keep_idx"].shape[0] and len(torch.unique(keep)) == keep.numel()
    assert A2.nnz == 2 * keep.numel()


# ------------------------------------------------------------------------------------------------ K2
@pytest.mark.parametrize("n,F,d", [(700, 256, 64), (1000, 4096, 64), (333, 130, 64), (257, 384, 32), (300, 512, 128),
                                   (129, 200, 256), (64, 77, 96), (50, 64, 300)])
@pytest.mark.parametrize("path", ["tc", "simt"])
def test_project_matches_oracle(dev, n, F, d, path):
    from mmrec_b200 import ops
    ops.set_project_path(path == "tc")
    g = torch.Generator().manual_seed(n + F)
    X = torch.randn(n, F, generator=g); W = torch.randn(d, F, generator=g) / F ** 0.5; b = torch.randn(d, generator=g)
    idx = torch.randint(0, n, (n // 2 + 3,), generator=g)
    Xd, Wd, bd = X.to(dev), W.to(dev), b.to(dev)
    assert rel(ops.project(Xd, Wd, bd), O.project(X, W, b)) < 1e-5
    assert rel(ops.project(Xd, Wd, None), O.project(X, W, None)) < 1e-5
    assert rel(ops.project(Xd, Wd, bd, idx=idx.to(dev)), O.project(X, W, b, idx=idx)) < 1e-5
    assert rel(ops.project(Xd, Wd, bd, l2_normalize=True), O.project(X, W, b, l2_normalize=True)) < 1e-5
    # autograd (backward of nn.Linear + gather)
    X1, W1, b1 = Xd.clone().requires_grad_(True), Wd.clone().requires_grad_(True), bd.clone().requires_grad_(True)
    X2, W2, b2 = X.clone().requires_grad_(True), W.clone().requires_grad_(True), b.clone().requires_grad_(True)
    w = torch.randn(idx.numel(), d, generator=g)
    (ops.project(X1, W1, b1, idx=idx.to(dev)) * w.to(dev)).sum().backward()
    (O.project(X2, W2, b2, idx=idx) * w).sum().backward()
    assert rel(X1.grad, X2.grad) < 1e-5 and rel(W1.grad, W2.grad) < 1e-5 and rel(b1.grad, b2.grad) < 1e-5
    ops.set_project_path(True)


# ------------------------------------------------------------------------------------------------ K3
@pytest.mark.parametrize("B,I,k", [(1, 50, 50), (3, 51, 1), (127, 1000, 50), (300, 7000, 50), (64, 5000, 1024), (4097, 333, 20)])
def test_topk_exact_on_identical_scores(dev, B, I, k):
    from mmrec_b200 import ops
    g = torch.Generator().manual_seed(B * 7 + I)
    S = torch.randn(B, I, generator=g)
    S = (S * 8).round() / 8                                                           # many exact ties
    S[0, :] = 0.25                                                                    # a fully tied row
    nm = min(B * 5, B * I // 2)
    mask = torch.stack([torch.randint(0, B, (nm,), generator=g), torch.randint(0, I, (nm,), generator=g)])
    ref = S.clone()
    ref[mask[0], mask[1]] = -1e10
    rv, ri = O.topk_tie_low_index(ref.numpy(), k)
    Sd = S.clone().to(dev)
    val, idx = ops.mask_topk(Sd, mask.to(dev), k)
    assert torch.equal(Sd.cpu(), ref)                       # in-place mask, like the trainer
    assert np.array_equal(idx.cpu().numpy(), ri)
    assert np.array_equal(val.cpu().numpy(), rv)
    tv, _ = torch.topk(ref, k, dim=-1)                      # values agree with torch.topk exactly
    assert torch.equal(val.cpu(), tv)
    v2, i2 = ops.mask_topk(S.clone().to(dev), None, k, item_offset=1000)
    assert torch.equal(i2.cpu() - 1000, torch.from_numpy(O.topk_tie_low_index(S.numpy(), k)[1]))


@pytest.mark.parametrize("B,U,I,d,k", [(128, 500, 700, 64, 50), (4096, 5000, 7000, 64, 50), (1000, 1000, 333, 64, 20),
                                       (77, 300, 20000, 128, 50), (513, 600, 900, 32, 10), (200, 200, 500, 48, 5),
                                       (700, 900, 40000, 64, 50), (300, 300, 70001, 96, 20)])
@pytest.mark.parametrize("path", ["simt", "tc", "fused"])
def test_score_and_fused_topk(dev, B, U, I, d, k, path):
    from mmrec_b200 import ops
    ops.set_score_path(path)
    try:
        g = torch.Generator().manual_seed(B + I)
        ue = torch.randn(U, d, generator=g) * 0.1; ie = torch.randn(I, d, generator=g) * 0.1
        users = torch.randint(0, U, (B,), generator=g)
        nm = B * 8
        mask = torch.stack([torch.randint(0, B, (nm,), generator=g), torch.randint(0, I, (nm,), generator=g)])
        S = ops.score(ue.to(dev), ie.to(dev), users.to(dev))
        ref = O.full_sort_scores(ue.double(), ie.double(), users)
        scale = ref.abs().max().item()
        assert (S.cpu().double() - ref).abs().max().item() < 2e-6 * scale + 1e-9      # fp32-level accuracy
        assert S.shape == (B, I) and S.is_contiguous()
        # fused path == the unfused path on the kernel's own scores (identical arithmetic -> identical indices)
        val, idx = ops.score_topk(ue.to(dev), ie.to(dev), users.to(dev), mask.to(dev), k)
        Sm = S.clone()
        v2, i2 = ops.mask_topk(Sm, mask.to(dev), k)
        if path != "fused":
            assert torch.equal(idx, i2) and torch.equal(val, v2)
        else:   # finalists are scored by an fp32 fmaf chain, S by 3xTF32: the same values to rounding, near ties may swap
            dif = (idx != i2).any(dim=1)
            assert dif.float().mean().item() <= 0.05
            assert (val - v2).abs().max().item() < 4e-6 * scale
            if I >= 16 * 2 * k:                             # the certified-filter kernels ran (not the tc fallback) and served every row
                assert ops.fused_fallback_rows() == 0
        # against the fp64 re-score: every disagreement must be a near tie, and the SETS must agree up to near ties
        refm = ref.clone(); refm[mask[0], mask[1]] = -1e10
        rv, ri = O.topk_tie_low_index(refm.numpy(), k)
        got = idx.cpu().numpy()
        bad = np.nonzero((got != ri).any(axis=1))[0]
        for b in bad:
            cols = np.nonzero(got[b] != ri[b])[0]
            gap = np.abs(refm[b, got[b, cols]].numpy() - refm[b, ri[b, cols]].numpy()).max()
            assert gap < 4e-6 * scale, f"row {b}: non-tie mismatch, gap {gap}"
        assert len(bad) <= max(2, B // 20)
    finally:
        ops.set_score_path("auto")


def _ref_topk(ue, ie, users, mask, k):
    ref = O.full_sort_scores(ue.double(), ie.double(), users)
    if mask is not None:
        ref[mask[0], mask[1]] = -1e10
    return ref, O.topk_tie_low_index(ref.numpy(), k)


def _check_near_tie(idx, ref, ri, scale):
    got = idx.cpu().numpy()
    for b in np.nonzero((got != ri).any(axis=1))[0]:
        cols = np.nonzero(got[b] != ri[b])[0]
        gap = np.abs(ref[b, got[b, cols]].numpy() - ref[b, ri[b, cols]].numpy()).max()
        assert gap < 4e-6 * scale, f"row {b}: non-tie mismatch, gap {gap}"


def test_fused_topk_operand_scaling(dev):
    """The filter's fp16 operands are scaled by powers of two (per user row, per catalogue): tiny, huge and mixed
    magnitudes must neither overflow nor lose the certificate (every row served by the filter, result = fp32 top-k).
    Random tables cannot exercise the filter's margin: the masked-item rows and the group granularity leave more slack
    than fp16 rounding takes, so a wrong margin or a wrong row norm still passes here.  tests/test_gpu_score_cf.py holds
    the adversarial catalogue, the exact power-of-two scale invariance and the fp64 acceptance rule that would catch it."""
    from mmrec_b200 import ops
    ops.set_score_path("fused")
    try:
        g = torch.Generator().manual_seed(5)
        B, U, I, d, k = 300, 300, 5000, 64, 50
        for su, si, mix in [(1e-6, 1e-7, False), (3e4, 2e3, False), (1.0, 1.0, True), (1e-20, 1e-15, False)]:
            ue = torch.randn(U, d, generator=g) * su; ie = torch.randn(I, d, generator=g) * si
            if mix:     # rows and columns spanning 12 orders of magnitude
                ue *= 10.0 ** torch.randint(-6, 6, (U, 1), generator=g).float()
                ie *= 10.0 ** torch.randint(-3, 3, (1, d), generator=g).float()
            users = torch.arange(B)
            mask = torch.stack([torch.randint(0, B, (B * 8,), generator=g), torch.randint(0, I, (B * 8,), generator=g)])
            val, idx = ops.score_topk(ue.to(dev), ie.to(dev), users.to(dev), mask.to(dev), k)
            assert ops.fused_fallback_rows() == 0
            ref = ue.double() @ ie.double().T
            ref[mask[0], mask[1]] = -float("inf")
            ri = torch.from_numpy(O.topk_tie_low_index(ref.numpy(), k)[1])
            got = idx.cpu()
            for b in torch.nonzero((got != ri).any(dim=1)).flatten().tolist():
                cols = torch.nonzero(got[b] != ri[b]).flatten()
                gap = (ref[b, got[b, cols]] - ref[b, ri[b, cols]]).abs().max().item()
                assert gap < 4e-6 * ref[b][torch.isfinite(ref[b])].abs().max().item(), f"row {b}: non-tie mismatch"
            chk = (ue[users][:, None, :].double() * ie[got].double()).sum(-1)
            assert ((chk - val.cpu().double()).abs() <= 2e-6 * chk.abs().max(dim=1, keepdim=True).values + 1e-300).all()
    finally:
        ops.set_score_path("auto")


def test_fused_topk_edge_cases(dev):
    """The fused tcgen05 path (forced): heavy users (more masked items than there are item groups -> exact kernel),
    unsorted mask, degenerate (all-equal) scores, ragged sizes, d = 32 / 128."""
    from mmrec_b200 import ops
    ops.set_score_path("fused")
    g = torch.Generator().manual_seed(11)
    for (B, U, I, d, k) in [(300, 400, 3000, 64, 50), (129, 200, 2049, 128, 20), (1, 10, 1700, 32, 50), (4097, 4100, 2600, 64, 50),
                            (257, 300, 16500, 40, 50)]:
        ue = torch.randn(U, d, generator=g) * 0.1; ie = torch.randn(I, d, generator=g) * 0.1
        users = torch.randint(0, U, (B,), generator=g)
        rows = [torch.randint(0, B, (B * 6,), generator=g)]; cols = [torch.randint(0, I, (B * 6,), generator=g)]
        heavy = min(B - 1, 7)
        rows.append(torch.full((900,), heavy)); cols.append(torch.randperm(I, generator=g)[:900])   # a heavy user
        mask = torch.stack([torch.cat(rows), torch.cat(cols)])
        mask = mask[:, torch.randperm(mask.shape[1], generator=g)]                                  # unsorted on purpose
        val, idx = ops.score_topk(ue.to(dev), ie.to(dev), users.to(dev), mask.to(dev), k)
        # the same mask row-major (what the evaluation loader emits: the one-pass sorted CSR build) gives the same answer
        srt = mask[:, torch.argsort(mask[0], stable=True)]
        val_s, idx_s = ops.score_topk(ue.to(dev), ie.to(dev), users.to(dev), srt.to(dev), k)
        assert torch.equal(idx, idx_s) and torch.equal(val, val_s)
        ref, (rv, ri) = _ref_topk(ue, ie, users, mask, k)
        _check_near_tie(idx, ref, ri, ref[ref > -1e9].abs().max().item())
        hit = torch.zeros(B, I, dtype=torch.bool); hit[mask[0], mask[1]] = True
        assert not hit.gather(1, idx.cpu()).any()
        assert torch.all(val[:, :-1] >= val[:, 1:])
        # the values are the fp32 scores of the returned items
        chk = (ue[users][:, None, :].double() * ie[idx.cpu()].double()).sum(-1)
        assert (chk - val.cpu().double()).abs().max().item() < 2e-6 * ref[ref > -1e9].abs().max().item()
        # a catalogue packed once gives the same answer as packing inside the call
        cat = ops.Catalog(ie.to(dev))
        val_c, idx_c = ops.score_topk(ue.to(dev), cat.item_e, users.to(dev), mask.to(dev), k, catalog=cat)
        assert torch.equal(idx, idx_c) and torch.equal(val, val_c)
    # all scores equal: nothing to threshold on -> exact kernel, ties resolve to the lowest indices
    ue = torch.zeros(64, 64); ie = torch.randn(2000, 64, generator=g)
    val, idx = ops.score_topk(ue.to(dev), ie.to(dev), None, None, 50)
    assert torch.equal(idx.cpu(), torch.arange(50).expand(64, 50)) and torch.all(val == 0)
    # a mask that covers almost the whole catalogue of one user
    ue = torch.randn(130, 64, generator=g); ie = torch.randn(1200, 64, generator=g)
    mask = torch.stack([torch.zeros(1150, dtype=torch.int64), torch.randperm(1200, generator=g)[:1150]])
    val, idx = ops.score_topk(ue.to(dev), ie.to(dev), None, mask.to(dev), 50)
    ref, (rv, ri) = _ref_topk(ue, ie, torch.arange(130), mask, 50)
    _check_near_tie(idx, ref, ri, ref[ref > -1e9].abs().max().item())
    ops.set_score_path("auto")


def test_score_without_user_index_and_strided_inputs(dev):
    from mmrec_b200 import ops
    ue = torch.randn(300, 64, device=dev); ie = torch.randn(411, 64, device=dev)
    S = ops.score(ue, ie)
    assert rel(S, ue.cpu() @ ie.cpu().t()) < 1e-5
    big = torch.randn(300, 128, device=dev)
    S2 = ops.score(big[:, :64], ie)                         # non-contiguous view is made contiguous
    assert rel(S2, big[:, :64].cpu() @ ie.cpu().t()) < 1e-5


def test_topk_merge_equals_global_topk(dev):
    from mmrec_b200 import ops
    g = torch.Generator().manual_seed(5)
    B, I, k, parts = 700, 4000, 50, 8
    S = torch.randn(B, I, generator=g)
    S[:, 100] = S[:, 3100]                                  # ties across shards
    shard = I // parts
    vals, idxs = [], []
    for p in range(parts):
        v, i = ops.mask_topk(S[:, p * shard:(p + 1) * shard].contiguous().to(dev), None, k, item_offset=p * shard)
        vals.append(v); idxs.append(i)
    mv, mi = ops.topk_merge(torch.stack(vals), torch.stack(idxs))
    rv, ri = O.topk_tie_low_index(S.numpy(), k)
    assert np.array_equal(mi.cpu().numpy(), ri) and np.array_equal(mv.cpu().numpy(), rv)


# ------------------------------------------------------------------------------------------------ full size
def test_full_size_properties_baby(dev):
    """BASELINE.json configs[1] sizes (20k users, 7k items, 160k edges, d=64): size-independent properties."""
    from mmrec_b200 import graph, ops
    from mmrec_b200.utils import synth
    g = synth.named("baby")
    U, I = g.n_users, g.n_items
    tu, ti = g.train
    A = graph.build_norm_adj((tu, ti), U, I, dev)
    n = U + I
    assert A.nnz == 2 * len(tu)
    gen = torch.Generator().manual_seed(0)
    x = torch.randn(n, 64, generator=gen).to(dev); y = torch.randn(n, 64, generator=gen).to(dev)
    Ax, Ay, Axy = (torch.empty(n, 64, device=dev) for _ in range(3))
    ops.spmm_raw(A, x, Y=Ax); ops.spmm_raw(A, y, Y=Ay); ops.spmm_raw(A, x + y, Y=Axy)
    assert rel(Axy, Ax + Ay) < 1e-6                                           # linearity
    assert abs(((Ax * y).sum() - (x * Ay).sum()).item()) < 1e-3 * (Ax * y).abs().sum().item()   # symmetry <Ax,y>=<x,Ay>
    ones = torch.ones(n, 64, device=dev); A1 = torch.empty(n, 64, device=dev)
    ops.spmm_raw(A, ones, Y=A1)
    rows, _, vals = A.coo()
    rs = torch.zeros(n, device=dev, dtype=torch.float64).index_add_(0, rows, vals.double())
    assert ((A1[:, 0].double() - rs).abs() / rs.abs().clamp_min(1.0)).max().item() < 2e-6   # A 1 = row sums
    emb = ops.propagate_mean(A, x * 0.05, 3)
    ue, ie = emb[:U].contiguous(), emb[U:].contiguous()
    users = torch.arange(0, 4096, device=dev)
    mask = torch.stack([torch.from_numpy(tu[tu < 4096]), torch.from_numpy(ti[tu < 4096])]).to(dev)
    val, idx = ops.score_topk(ue, ie, users, mask, 50)
    assert torch.all(val[:, :-1] >= val[:, 1:])                               # sorted
    assert idx.min() >= 0 and idx.max() < I
    assert all(len(set(r)) == 50 for r in idx[:64].cpu().tolist())          # no repeats
    re = (ue[users][:, None, :] * ie[idx]).sum(-1)                            # values are the scores of the indices
    assert (re - val).abs().max().item() < 1e-5 * val.abs().max().item() + 1e-9
    hit = torch.zeros(4096, I, dtype=torch.bool, device=dev); hit[mask[0], mask[1]] = True
    assert not hit.gather(1, idx).any()                                       # masked train positives never returned
    val2, idx2 = ops.score_topk(ue, ie, users, mask, 50)
    assert torch.equal(idx, idx2) and torch.equal(val, val2)                  # idempotent / deterministic
    ops.set_score_path("fused")                                               # fused == unfused on the same arithmetic
    val3, idx3 = ops.score_topk(ue, ie, users, mask, 50)
    ops.set_score_path("auto")
    same = (idx3 == idx).all(dim=1).float().mean().item()
    assert same > 0.99 and (val3 - val).abs().max().item() < 1e-5 * val.abs().max().item() + 1e-9


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_peer_sum_rank_order_and_epilogue(dev, world):
    """K4 (mmrec_peer_sum_f32) on one device: the partials are ordinary buffers here, the arithmetic is what is under
    test -- rank-order summation (bit-exact against the same torch loop) and the layer-mean epilogue."""
    from mmrec_b200 import ops
    g = torch.Generator(device=dev); g.manual_seed(world)
    n = 4 * 1237
    parts = [torch.randn(n, device=dev, generator=g) for _ in range(world)]
    acc = torch.randn(n, device=dev, generator=g)
    ref_sum = parts[0].clone()
    for p in parts[1:]:
        ref_sum = ref_sum + p
    for div in (1.0, 4.0):
        s_out = torch.empty(n, device=dev); a_out = acc.clone()
        ops.peer_sum([p.data_ptr() for p in parts], n, acc_in=a_out, acc_out=a_out, acc_div=div, sum_out=s_out)
        assert torch.equal(s_out, ref_sum)
        ref_acc = (acc + ref_sum) / div if div != 1.0 else acc + ref_sum
        assert torch.equal(a_out, ref_acc)
    with pytest.raises(Exception):
        ops.peer_sum([p.data_ptr() for p in parts], n - 1, sum_out=torch.empty(n, device=dev))


@pytest.mark.parametrize("world,B,k", [(2, 300, 50), (3, 17, 20), (8, 64, 50)])
def test_topk_merge_peers_matches_contiguous_merge(dev, world, B, k):
    """mmrec_topk_merge_peers (lists by pointer, local -> global relabel inside) == mmrec_topk_merge on the gathered,
    relabelled lists; ties resolve to the lower global index in both."""
    from mmrec_b200 import ops
    g = torch.Generator().manual_seed(world * 1000 + B)
    vals = torch.sort((torch.randint(0, 40, (world, B, k), generator=g).float() / 8.0), dim=-1, descending=True).values   # many ties
    idx = torch.stack([torch.stack([torch.randperm(5000, generator=g)[:k] for _ in range(B)]) for _ in range(world)])
    for p in range(world):                                  # input contract: equal values inside a list come in ascending index order
        for b in range(B):
            for x in vals[p, b].unique():
                sel = (vals[p, b] == x).nonzero().flatten()
                idx[p, b, sel] = torch.sort(idx[p, b, sel]).values
    vd = [vals[p].contiguous().to(dev) for p in range(world)]
    idd = [idx[p].contiguous().to(dev) for p in range(world)]
    v1, i1 = ops.topk_merge_peers([t.data_ptr() for t in vd], [t.data_ptr() for t in idd], B, k, dev, idx_mul=world, idx_add=1)
    glob = torch.stack([idd[p] * world + p for p in range(world)])
    v2, i2 = ops.topk_merge(torch.stack(vd), glob)
    assert torch.equal(v1, v2) and torch.equal(i1, i2)


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_peer_reduce_push_equals_peer_sum(dev, world):
    """mmrec_peer_reduce_push_f32 on one device, the `world` ranks played in turn: every rank sums its slice in rank order and
    stores it into every destination, so after all ranks ran every destination holds the rank-order sum (bit-identical to
    mmrec_peer_sum_f32), and the sliced accumulator reproduces the layer-mean epilogue."""
    from mmrec_b200 import ops
    g = torch.Generator(device=dev); g.manual_seed(10 + world)
    n = 4 * 1531                                            # not a multiple of world * 4: ragged last slice
    parts = [torch.randn(n, device=dev, generator=g) for _ in range(world)]
    acc0 = torch.randn(n, device=dev, generator=g)
    ref = parts[0].clone()
    for p in parts[1:]:
        ref = ref + p
    per = ((n // 4 + world - 1) // world) * 4
    for final in (False, True):
        dst = [torch.full((n,), float("nan"), device=dev) for _ in range(world)]
        accs = []
        for r in range(world):
            lo, hi = min(per * r, n), min(per * r + per, n)
            acc = torch.zeros(per, device=dev)
            ops.peer_reduce_push([p.data_ptr() for p in parts], [t.data_ptr() for t in dst], n, r, acc_in=acc0[lo:hi].contiguous(),
                                 acc_out=acc, acc_div=4.0, final_layer=final)
            accs.append((lo, hi, acc))
        want = (acc0 + ref) / 4.0 if final else ref
        for t in dst:
            assert torch.equal(t, want)
        if not final:
            for lo, hi, acc in accs:
                assert torch.equal(acc[:hi - lo], (acc0 + ref)[lo:hi])


def test_peer_gather_and_row_range_merge(dev):
    from mmrec_b200 import ops
    g = torch.Generator().manual_seed(3)
    world, n_each = 3, 4 * 77
    src = [torch.randn(n_each, generator=g).to(dev) for _ in range(world)]
    dst = torch.empty(world * n_each, device=dev)
    ops.peer_gather([t.data_ptr() for t in src], n_each, dst)
    assert torch.equal(dst, torch.cat(src))
    # merge of a row range == the same rows of the full merge
    B, k = 37, 20
    vals = torch.sort(torch.randint(0, 30, (world, B, k), generator=g).float() / 4.0, dim=-1, descending=True).values
    idx = torch.stack([torch.stack([torch.sort(torch.randperm(900, generator=g)[:k]).values for _ in range(B)]) for _ in range(world)])
    # (within a list equal values must come in ascending index order: sort the indices inside runs of equal values)
    for p in range(world):
        for b in range(B):
            v = vals[p, b]
            for x in v.unique():
                sel = (v == x).nonzero().flatten()
                idx[p, b, sel] = torch.sort(idx[p, b, sel]).values
    vd = [vals[p].contiguous().to(dev) for p in range(world)]
    idd = [idx[p].contiguous().to(dev) for p in range(world)]
    fv, fi = ops.topk_merge_peers([t.data_ptr() for t in vd], [t.data_ptr() for t in idd], B, k, dev, idx_mul=world, idx_add=1)
    rv, ri = ops.topk_merge_peers([t.data_ptr() for t in vd], [t.data_ptr() for t in idd], B, k, dev, idx_mul=world, idx_add=1, row0=11, n_rows=9)
    assert torch.equal(rv, fv[11:20]) and torch.equal(ri, fi[11:20])
    glob = torch.stack([idd[p] * world + p for p in range(world)])
    v2, i2 = ops.topk_merge(torch.stack(vd), glob)
    assert torch.equal(fv, v2) and torch.equal(fi, i2)


def test_device_evaluator_matches_host_metrics(dev):
    """f2: mmrec_topk_metrics_f64 (hit matrix + Recall / NDCG / Precision / MAP sums on the device) against the numpy
    implementation of the reference's metric definitions (mmrec_b200/utils/topk_evaluator.py, pinned to the reference's
    numbers by tests/test_oracle_golden.py)."""
    from mmrec_b200.utils import topk_evaluator as TE

    class Loader:
        def __init__(self, pos):
            self.pos = pos

        def get_eval_items(self):
            return self.pos

        def get_eval_len_list(self):
            return np.array([len(p) for p in self.pos], dtype=np.int64)

    rng = np.random.default_rng(0)
    n, I, K = 3001, 900, 50
    pos = [rng.choice(I, size=rng.integers(1, 70), replace=False).astype(np.int64) for _ in range(n)]
    topk = np.stack([rng.permutation(I)[:K] for _ in range(n)]).astype(np.int64)
    for u in range(0, n, 7):                                # some users with many hits, some with a full list of hits
        h = min(len(pos[u]), K)
        topk[u, :h] = pos[u][:h]
    cfg = {"metrics": ["Recall", "NDCG", "Precision", "MAP"], "topk": [5, 10, 20, 50], "device_evaluator": None}
    ev = TE.TopKEvaluator(cfg)
    batches = [torch.from_numpy(topk[lo:lo + 1024]).to(dev) for lo in range(0, n, 1024)]
    got = ev.evaluate(batches, Loader(pos))
    want = ev.evaluate([b.cpu() for b in batches], Loader(pos))
    assert got.keys() == want.keys()
    for key in want:
        assert abs(got[key] - want[key]) <= 1.0001e-4, (key, got[key], want[key])      # both rounded to 4 decimals
    # un-rounded: float64 sums in a different order
    from mmrec_b200 import ops
    hit = TE.hit_matrix(topk, pos)
    pos_len = np.array([len(p) for p in pos])
    disc = 1.0 / np.log2(np.arange(1, K + 1) + 1.0)
    ptr = torch.from_numpy(np.concatenate([[0], np.cumsum(pos_len)])).to(dev)
    items = torch.from_numpy(np.concatenate([np.sort(p) for p in pos])).to(dev)
    sums = torch.zeros(4, K, dtype=torch.float64, device=dev)
    ops.topk_metric_sums(torch.from_numpy(topk).to(dev), ptr, items, torch.from_numpy(disc).to(dev), torch.from_numpy(np.cumsum(disc)).to(dev), sums)
    mean = (sums / n).cpu().numpy()
    for row, fn in enumerate((TE.recall_, TE.ndcg_, TE.precision_, TE.map_)):
        np.testing.assert_allclose(mean[row], fn(hit, pos_len), rtol=1e-12, atol=1e-14)


@pytest.mark.parametrize("d,L,mm_layers", [(64, 3, 1), (64, 1, 1), (128, 2, 2), (32, 4, 0), (64, 2, 0)])
def test_spmm_chain_equals_separate_launches(dev, d, L, mm_layers):
    """mmrec_spmm_chain_f32 (all SpMMs of a propagation in one cooperative launch, grid barriers in between) runs the same
    kernel body as mmrec_spmm_f32: bit-identical to the one-launch-per-SpMM path, also when replayed from a CUDA graph."""
    from mmrec_b200 import ops
    from mmrec_b200.ops import CSR
    U, I = 900, 500
    n = U + I
    r, c, v = rand_coo(U, I, 7000, seed=d + L, dup_frac=0)
    r = torch.cat([r, torch.full((1500,), 3)]); c = torch.cat([c, torch.randint(0, I, (1500,))]); v = torch.cat([v, torch.rand(1500) - 0.5])   # a row the plan splits
    A = CSR.from_coo(torch.cat([r, c + U]).to(dev), torch.cat([c + U, r]).to(dev), torch.cat([v, v]).to(dev), n, n, symmetric=True)
    mr, mc, mv = rand_coo(I, I, 4000, seed=77)
    M = CSR.from_coo(mr.to(dev), mc.to(dev), mv.to(dev), I, I)
    ego = torch.randn(n, d, generator=torch.Generator().manual_seed(2)).to(dev)
    want = ops._propagate_mean_post_unfused(A, ego, L, M if mm_layers else None, ego[U:] if mm_layers else None, max(mm_layers, 1), U)
    got = ops.propagate_mean_fused(A, ego, L, post_csr=M if mm_layers else None, post_x=ego[U:] if mm_layers else None,
                                   post_layers=max(mm_layers, 1), post_row0=U)
    assert torch.equal(got, want)
    # oracle
    adj = torch.sparse_coo_tensor(torch.stack([torch.cat([r, c + U]), torch.cat([c + U, r])]), torch.cat([v, v]), (n, n))
    ref = O.propagate_mean(adj, ego.cpu(), L)
    if mm_layers:
        h = ego.cpu()[U:]
        mm = torch.sparse_coo_tensor(torch.stack([mr, mc]), mv, (I, I))
        for _ in range(mm_layers):
            h = torch.sparse.mm(mm, h)
        ref = torch.cat([ref[:U], ref[U:] + h])
    assert rel(got, ref) < 1e-5
    # replay from a CUDA graph (cooperative launches are capturable)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        ops.propagate_mean_fused(A, ego, L)
        torch.cuda.synchronize()
        gph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gph, stream=side):
            out = ops.propagate_mean_fused(A, ego, L)
    torch.cuda.synchronize()
    out.zero_(); gph.replay(); torch.cuda.synchronize()
    assert torch.equal(out, ops._propagate_mean_post_unfused(A, ego, L, None, None, 1, 0))
    assert int(A.counters.abs().sum().item()) == 0


@pytest.mark.parametrize("d", [64, 128])
def test_panel_csr_equals_plain_csr(dev, d):
    """ops.PanelCSR (column panels multiplied one after the other, Y accumulating: the form for graphs whose dense operand
    does not fit the L2) against the unpanelled CSR and the oracle, forward and backward of propagate_mean."""
    from mmrec_b200 import ops
    from mmrec_b200.ops import CSR, PanelCSR
    n = 3000
    r, c, v = rand_coo(n, n, 40000, seed=d)
    rr, cc, vv = torch.cat([r, c]).to(dev), torch.cat([c, r]).to(dev), torch.cat([v, v]).to(dev)       # symmetric
    A = CSR.from_coo(rr, cc, vv, n, n, symmetric=True)
    P = PanelCSR.from_coo(rr, cc, vv, n, n, d, panel_bytes=700 * 4 * d, symmetric=True)               # ~5 panels
    assert len(P.panels) >= 3 and P.nnz == A.nnz
    X = torch.randn(n, d, generator=torch.Generator().manual_seed(1)).to(dev)
    base = torch.randn(n, d, generator=torch.Generator().manual_seed(2)).to(dev)
    Y1, Y2 = torch.empty(n, d, device=dev), torch.empty(n, d, device=dev)
    a1, a2 = base.clone(), base.clone()
    ops.spmm_raw(A, X, Y=Y1, acc_in=a1, acc_out=a1, acc_div=3.0)
    ops.spmm_raw(P, X, Y=Y2, acc_in=a2, acc_out=a2, acc_div=3.0)
    assert rel(Y2, Y1) < 1e-6 and rel(a2, a1) < 1e-6
    e1 = X.clone().requires_grad_(True); e2 = X.clone().requires_grad_(True)
    o1 = ops.propagate_mean(A, e1, 3); o2 = ops.propagate_mean(P, e2, 3)
    assert rel(o2, o1) < 1e-6
    w = torch.randn_like(o1)
    (o1 * w).sum().backward(); (o2 * w).sum().backward()
    assert rel(e2.grad, e1.grad) < 1e-6
    ref = O.propagate_mean(torch.sparse_coo_tensor(torch.stack([rr.cpu(), cc.cpu()]), vv.cpu(), (n, n)), X.cpu(), 3)
    assert rel(o2, ref) < 1e-5
