"""The certified-filter top-k (`csrc/score_cf.cu`, `ops.score_topk` on the fused path) against fp64.

Acceptance rule, shared by every GPU case.  fp64 scores `s = U[users] I^T` and `a = |U[users]| |I|^T` are computed on the
device (cuBLAS DGEMM, in row chunks).  The kernel's values are fp32 `fmaf` chains of four products followed by a
butterfly over L = 8 / 16 / 32 partials (`cf_dot_thread`), so every product goes through at most h = 4 + log2 L roundings
and `|v - s| <= beta = h 2^-24 (1 + 1e-6) a` per pair.  A row passes when
  * its values are non-increasing and equal values come in ascending item order;
  * its indices are distinct, lie in [item_offset, item_offset + n_items) and are not masked -- unless the row has fewer
    than k unmasked items: masked items then count as exactly -1e10 (`src/common/trainer.py:307`);
  * every returned item has `|v_i - s_i| <= beta_i`;
  * every unmasked item j that was not returned has `s_j <= v_k + beta_j` (v_k = the last returned value).
That is exactly "an fp32 top-k under this rounding", at any overall scale.  Rows the fused path does not serve (fewer
than 2k item groups, k > 256) go through the 3xTF32 GEMM + top-k kernels, whose bound is looser (`_beta_factor`).

Random tables cannot exercise the filter's margin (`cf_thr_kernel`: thr = t - 2 eps'): the extra rows for masked items
and the 16-item group granularity leave far more slack than fp16 rounding takes.  The adversarial catalogue below does:
fp16 rounding of the scaled operands scores the true top-k (A items) about 0.63 eps' too low and their nearest rivals
(B items) about 0.62 eps' too high, so a margin of half the certified one loses A items.  A host emulation of the filter
(CPU tests, no GPU needed) checks that the construction stays adversarial.
"""
import os
import re

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu

CF_EPS, CF_EPS_SUB = 1.125 / 1024, 2.0 ** -24           # csrc/score_cf.cu
MASKED = -1e10                                          # value of a masked item (src/common/trainer.py:307)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from mmrec_b200 import _lib
    _lib.require_device()
    return torch.device("cuda:0")


# ------------------------------------------------------------------------------------------------ host emulation
def cf_gw(n_items):
    return 1 if n_items <= 16384 else (2 if n_items <= 32768 else (4 if n_items <= 65536 else 8))


def cf_lpr(d):
    return 8 if d <= 32 else (16 if d <= 64 else 32)


def scale_for(m):
    """`cf_scale_for`: the power of two that brings a largest magnitude m into [2^14, 2^15) (1 for 0, inf, NaN and
    m < 2^-113)."""
    m = float(m)
    if m == 0.0 or not np.isfinite(m):
        return 1.0
    e = np.frexp(m)[1] - 1                               # floor(log2 m)
    return 1.0 if e + 127 < 14 else 2.0 ** (14 - e)


def f16(x):
    """fp32 -> fp16 round-to-nearest-even (what `__floats2half2_rn` does), back to float64."""
    return np.asarray(x, np.float32).astype(np.float16).astype(np.float64)


def cf_emulate(U, I, masks, k, margin_mul=1.0):
    """The filter of score_cf.cu on the host, for rows U (float32 [B, d]) against I (float32 [n, d]): operands scaled
    by `cf_scale_for` and rounded to fp16, the need-th largest maximum of groups of 16 gw items (need = k + mask entries
    of the row), threshold = that minus margin_mul x the kernel's margin (exact norms of the scaled rows), candidates
    re-scored exactly.  The threshold is the exact need-th largest group maximum, as the radix search of cf_thr_kernel
    finds it for more than 1024 groups; the 16-bit search used for fewer groups only lowers it further.
    Returns (top-k index list per row, per-row eps' = CF_EPS |u| max|i| in the scaled domain, per-row scaled fp16 scores)."""
    n, d = I.shape
    si = scale_for(np.abs(I).max())
    Is = I.astype(np.float64) * si
    Ih = f16(I * np.float32(si))
    mn = np.sqrt((Is ** 2).sum(1)).max()
    w = 16 * cf_gw(n)
    G = -(-n // w)
    S = I.astype(np.float64) @ U.astype(np.float64).T
    got, eps1, approx = [], [], []
    for r, u in enumerate(U):
        su = scale_for(np.abs(u).max())
        uh = f16(u * np.float32(su))
        un = np.sqrt(((u.astype(np.float64) * su) ** 2).sum())
        st = Ih @ uh
        need = k + len(masks[r])
        assert need <= G, "the emulation covers rows the filter serves"
        pad = np.full(G * w, -np.inf)
        pad[:n] = st
        t = np.sort(pad.reshape(G, w).max(1))[::-1][need - 1]
        margin = 2 * (CF_EPS * un * mn + CF_EPS_SUB * np.sqrt(d) * (un + mn + 1)) * margin_mul
        cand = np.nonzero(st >= t - margin)[0]
        cand = cand[~np.isin(cand, masks[r])]
        s = S[:, r]
        got.append(cand[np.lexsort((cand, -s[cand]))][:k])
        eps1.append(CF_EPS * un * mn)
        approx.append(st / (su * si))                   # back in the unscaled domain
    return got, np.array(eps1), approx


def adversarial(d, n_items, n_users, k=50, n_b=80, n_mask_b=0, seed=0):
    """Catalogue on which fp16 rounding pushes the true top-k below its rivals.  P = first d/2 coordinates, Q = the rest.
    User elements sit on fp16 rounding midpoints after scaling (8196 -/+ 2^-10 -> scaled by 2 -> 16392 -/+ 2^-9; fp16 step
    16 there): below the midpoint on P (rounds down), above it on Q (rounds up).  k A items (8196 - 2^-10 on P, 0 on Q:
    round down, step 8) and n_b B items (8196 + 2^-10 on Q with one element exactly 8192, 0 on P: round up) sit one per
    group; s(B) < s(A) by ~4 / (32 * 8196) relative.  One element -2^14 pins the catalogue scale to 1; the filler is
    positive, in [1, 32), scores ~1e2 below s(A).  n_mask_b B items of every row are masked (need = k + n_mask_b).
    Returns float32 U [n_users, d], I [n_items, d], masks (list of item arrays), A (item ids, ascending)."""
    rng = np.random.default_rng(seed)
    P, Q = np.arange(d // 2), np.arange(d // 2, d)
    lo, hi = np.float32(8196 - 2.0 ** -10), np.float32(8196 + 2.0 ** -10)
    w = 16 * cf_gw(n_items)
    assert (k + n_b + 3) * w <= n_items
    I = (2.0 ** rng.uniform(0, 5, (n_items, d))).astype(np.float32)
    I[n_items - 1, 0] = -2.0 ** 14
    A = np.arange(k) * w + (7 * np.arange(k)) % w
    Bi = (k + 2 + np.arange(n_b)) * w + (5 * np.arange(n_b)) % w
    I[A] = 0
    I[np.ix_(A, P)] = lo
    I[Bi] = 0
    I[np.ix_(Bi, Q)] = hi
    I[Bi, Q[0]] = 8192
    u = np.zeros(d, np.float32)
    u[P], u[Q] = lo, hi
    U = np.repeat(u[None], n_users, 0)
    masks = [np.sort(rng.choice(Bi, n_mask_b, replace=False)) for _ in range(n_users)]
    return U, I, masks, A


ADV_CASES = [(64, 140001, 0), (32, 140001, 0), (128, 140001, 0), (64, 140001, 20), (64, 5000, 0)]


@pytest.mark.parametrize("d,n_items,n_mask_b", ADV_CASES)
def test_adversarial_catalogue_defeats_half_the_margin_in_emulation(d, n_items, n_mask_b):
    """Host emulation of the filter: the fp16 rounding swing between A and B items exceeds 1.1 eps' (half the margin
    is 1 eps'), the certified margin keeps the exact top-k, half of it loses A items on every row."""
    k = 50
    U, I, masks, A = adversarial(d, n_items, 4, k=k, n_mask_b=n_mask_b, seed=d + n_mask_b)
    got, eps1, approx = cf_emulate(U, I, masks, k, 1.0)
    s = I.astype(np.float64) @ U[0].astype(np.float64)
    assert np.all(s[A] == s[A[0]]) and s[A[0]] > np.sort(np.delete(s, A))[-1]          # A is the exact top-k
    Bi = np.argsort(-np.delete(s, A))                                                    # (the B items come next)
    b_items = np.delete(np.arange(n_items), A)[Bi[:80]]
    for r in range(len(U)):
        err = (approx[r] - s) / (eps1[r] / (scale_for(np.abs(U[r]).max()) * scale_for(np.abs(I).max())))
        swing = err[b_items].min() - err[A].max()
        assert swing > 1.1, f"row {r}: fp16 swing {swing:.3f} eps' no longer beats half the margin"
        assert np.array_equal(np.sort(got[r]), A), f"row {r}: the certified margin lost a top-k item"
    half, _, _ = cf_emulate(U, I, masks, k, 0.5)
    for r in range(len(U)):
        assert len(np.intersect1d(half[r], A)) < k, f"row {r}: half the margin still keeps every A item"


def test_emulation_scale_matches_kernel_rule():
    """`scale_for` is cf_scale_for: the largest magnitude lands in [2^14, 2^15); tiny / zero / non-finite -> 1."""
    for m in (1.0, 3.0, 2.0 ** 14, 2.0 ** 15 - 1, 1e-30, 1e30, 8196.0, 2.0 ** -113):
        sc = scale_for(m)
        assert 2.0 ** 14 <= m * sc < 2.0 ** 15
    for m in (0.0, float("inf"), float("nan"), 2.0 ** -114, 1e-45):
        assert scale_for(m) == 1.0


# ------------------------------------------------------------------------------------------------ GPU reference + rule
def _beta_factor(d, fused):
    if fused:
        return (4 + int(np.log2(cf_lpr(d)))) * 2.0 ** -24 * (1 + 1e-6)
    # 3xTF32: the dropped lo.lo term and the re-rounded lo parts (~2^-20 of |u||i| per product) plus fp32 accumulation
    # over the K steps of three MMA chains
    return (d + 16) * 2.0 ** -22


def _mask_coo(masks, device=None):
    rows = np.concatenate([np.full(len(m), r, np.int64) for r, m in enumerate(masks)] + [np.zeros(0, np.int64)])
    cols = np.concatenate([np.asarray(m, np.int64) for m in masks] + [np.zeros(0, np.int64)])
    t = torch.from_numpy(np.stack([rows, cols]))
    return t if device is None else t.to(device)


def check_topk(ue, ie, users, mask, k, val, idx, item_offset=0, fused=True, rows=None, chunk=256):
    """The acceptance rule above, on the device.  ue / ie fp32 tables, users int64 [B] (or None), mask [2, nnz] in global
    item ids (or None), val / idx the kernel's result.  `rows` limits the check to some rows."""
    n, d = ie.shape
    B = idx.shape[0]
    assert idx.shape == (B, k) and val.shape == (B, k)
    uid = users if users is not None else torch.arange(B, device=ie.device)
    I64, Ia = ie.double(), ie.double().abs()
    bf = _beta_factor(d, fused)
    li = idx - item_offset
    assert bool(((li >= 0) & (li < n)).all()), "index outside the catalogue shard"
    assert bool((val[:, :-1] >= val[:, 1:]).all()), "values not non-increasing"
    eq = val[:, :-1] == val[:, 1:]
    assert not bool((eq & (idx[:, :-1] >= idx[:, 1:])).any()), "equal values not in ascending item order"
    srt = li.sort(dim=1).values
    assert not bool((srt[:, 1:] == srt[:, :-1]).any()), "repeated index"
    if mask is not None and mask.numel():
        mr, mc = mask[0].to(ie.device), mask[1].to(ie.device) - item_offset
        keep = (mc >= 0) & (mc < n)
        mr, mc = mr[keep], mc[keep]
    else:
        mr = mc = torch.zeros(0, dtype=torch.int64, device=ie.device)
    sel = torch.arange(B, device=ie.device) if rows is None else torch.as_tensor(rows, device=ie.device)
    for c0 in range(0, sel.numel(), chunk):
        r = sel[c0:c0 + chunk]
        uu = ue[uid[r]].double()
        s = uu @ I64.T
        beta = bf * (uu.abs() @ Ia.T)
        pos = torch.full((B,), -1, dtype=torch.int64, device=ie.device)
        pos[r] = torch.arange(r.numel(), device=ie.device)
        hit = pos[mr] >= 0
        m = torch.zeros(r.numel(), n, dtype=torch.bool, device=ie.device)
        m[pos[mr[hit]], mc[hit]] = True
        few = (n - m.sum(1)) < k                                      # fewer than k unmasked items: masked ones fill in
        s = torch.where(m, torch.full_like(s, MASKED), s)
        beta = torch.where(m, torch.zeros_like(beta), beta)
        elig = ~m | few[:, None]
        ri, rv = li[r], val[r].double()
        assert bool(elig.gather(1, ri).all()), f"rows {r[~elig.gather(1, ri).all(1)].tolist()[:8]}: masked item returned"
        err = (rv - s.gather(1, ri)).abs() - beta.gather(1, ri)
        bad = (err > 0).any(1)
        assert not bool(bad.any()), f"rows {r[bad].tolist()[:8]}: a value is not the score of its index (excess {err.max().item():.3g})"
        ret = torch.zeros_like(m)
        ret.scatter_(1, ri, True)
        miss = elig & ~ret & (s > rv[:, -1:] + beta)
        bad = miss.any(1)
        assert not bool(bad.any()), f"rows {r[bad].tolist()[:8]}: an item above the k-th value was left out"


def _score_topk(ue, ie, users, mask, k, **kw):
    from mmrec_b200 import ops
    val, idx = ops.score_topk(ue, ie, users, mask, k, **kw)
    return val, idx, ops.fused_fallback_rows()


def _randn(shape, g, scale=0.1):
    return torch.randn(*shape, generator=g) * scale


def _rand_masks(B, n, per_row, g, heavy=None):
    masks = [torch.randint(0, n, (per_row,), generator=g).numpy() for _ in range(B)]
    if heavy is not None:
        row, cnt = heavy
        masks[row] = torch.randperm(n, generator=g)[:cnt].numpy()
    return masks


# ------------------------------------------------------------------------------------------------ adversarial catalogue
@gpu
@pytest.mark.parametrize("d,n_items,n_mask_b", ADV_CASES)
def test_adversarial_catalogue_exact_top_k(dev, d, n_items, n_mask_b):
    """On the adversarial catalogue the filter must still return exactly the fp64 top-k (the gap s(A) - s(B) is far
    above beta), with every row served by the filter."""
    k, B = 50, 256
    U, I, masks, A = adversarial(d, n_items, B, k=k, n_mask_b=n_mask_b, seed=d + n_mask_b)
    ue, ie = torch.from_numpy(U).to(dev), torch.from_numpy(I).to(dev)
    mask = _mask_coo(masks, dev) if n_mask_b else None
    users = torch.arange(B, device=dev)
    val, idx, fb = _score_topk(ue, ie, users, mask, k)
    assert fb == 0
    assert torch.equal(idx.cpu(), torch.from_numpy(A).expand(B, k))
    check_topk(ue, ie, users, mask, k, val, idx)


# ------------------------------------------------------------------------------------------------ scale invariance
SCALE_EXPS = [-120, -100, -92, -64, 0, 32, 48, 60]


def _normal_at(ue, ie, side, e):
    """Every element, product and score of the tables stays a finite normal fp32 when `side` is scaled by 2^e, and the
    largest magnitude stays at or above 2^-113 (below that cf_scale_for leaves a table unscaled, by design)."""
    tiny, huge = 2.0 ** -126, 2.0 ** 127
    def span(x):
        a = x.abs().double()
        return a[a > 0].min().item(), a.max().item()
    (ul, uh), (il, ih) = span(ue), span(ie)
    a_max = (ue.double().abs() @ ie.double().abs().T).max().item()
    xl, xh = (ul, uh) if side == "user" else (il, ih)
    return (xl * 2.0 ** e >= tiny and xh * 2.0 ** e < huge and ul * il * 2.0 ** e >= tiny and a_max * 2.0 ** e < huge
            and xh * 2.0 ** e >= 2.0 ** -113)


@pytest.fixture(scope="module")
def scale_tables(dev):
    g = torch.Generator().manual_seed(3)
    U, I, _, A = adversarial(64, 140001, 64, seed=1)
    # positive (no cancellation into subnormal partial sums), in [128, 256): every exponent of SCALE_EXPS applies
    rand_u = torch.rand(256, 64, generator=g) * 128 + 128
    rand_i = torch.rand(20000, 64, generator=g) * 128 + 128
    tables = {"adversarial": (torch.from_numpy(U).to(dev), torch.from_numpy(I).to(dev), A),
              "random": (rand_u.to(dev), rand_i.to(dev), None)}
    base = {}
    for name, (ue, ie, A_) in tables.items():
        val, idx, fb = _score_topk(ue, ie, None, None, 50)
        assert fb == 0
        check_topk(ue, ie, None, None, 50, val, idx)
        if A_ is not None:
            assert torch.equal(idx.cpu(), torch.from_numpy(A_).expand(idx.shape[0], 50))
        base[name] = (val, idx)
    return tables, base


@gpu
@pytest.mark.parametrize("e", [e for e in SCALE_EXPS if e != 0])
@pytest.mark.parametrize("side", ["user", "item"])
@pytest.mark.parametrize("table", ["adversarial", "random"])
def test_power_of_two_scale_invariance(dev, scale_tables, table, side, e):
    """Scaling one side by 2^e scales every fp32 operation of the result exactly and leaves the filter's scaled domain
    unchanged: indices bit-identical, values exactly v(0) 2^e, no row sent to the exact kernel.  The row norms of the
    margin must therefore be right at any magnitude (tiny rows whose squares underflow, huge ones whose squares overflow)."""
    tables, base = scale_tables
    ue, ie, _ = tables[table]
    if not _normal_at(ue, ie, side, e):
        pytest.skip(f"2^{e} takes the {table} table out of the normal fp32 range")
    ue2, ie2 = (ue * 2.0 ** e, ie) if side == "user" else (ue, ie * 2.0 ** e)
    val, idx, fb = _score_topk(ue2, ie2, None, None, 50)
    v0, i0 = base[table]
    wrong = (idx != i0).any(1).sum().item()
    assert wrong == 0, f"{wrong} of {idx.shape[0]} rows changed their top-k at 2^{e}"
    assert torch.equal(val, v0 * 2.0 ** e)
    assert fb == 0, f"{fb} rows went to the exact kernel at 2^{e}"


# ------------------------------------------------------------------------------------------------ branch matrix
BRANCHES = (
    # (id, n_items, d, k, extra)          group width cf_gw: 1 / 2 / 4 / 8, both sides of each boundary
    [(f"gw_items{n}", n, 64, 50, {}) for n in (16384, 16385, 32768, 32769, 65536, 65537)]
    # threshold search: 16-bit search over 16 x 32 keys (512 groups), over 32 x 32 (1024 groups), radix histogram (1094)
    + [("thr_coarse16", 8192, 64, 50, {}), ("thr_coarse32", 16384, 64, 50, {}), ("thr_histogram", 140001, 64, 50, {})]
    # G >= 2k decides fused / unfused under "auto": 96 groups at 1536 items, 104 at 1537
    + [("unfused_1536", 1536, 64, 50, {}), ("fused_1537", 1537, 64, 50, {})]
    # KP 32 / 64 / 128, L 8 / 16 / 32, scalar loads (d % 4 != 0, or rows off 16-byte alignment)
    + [(f"d{d}", 5000, d, 50, {}) for d in (1, 3, 31, 32, 33, 63, 64, 65, 100, 127, 128)]
    + [("d64_offset_views", 5000, 64, 50, {"offset_views": True})]
    # k up to the fused limit; 257 takes the unfused path
    + [(f"k{k}", 10000, 64, k, {}) for k in (1, 2, 50, 100, 256, 257)]
    # a shard of a larger catalogue: global item ids, mask entries of other shards never match
    + [("item_offset", 5000, 64, 50, {"item_offset": 3 * 5000})]
)


@gpu
@pytest.mark.parametrize("n_items,d,k,extra", [b[1:] for b in BRANCHES], ids=[b[0] for b in BRANCHES])
def test_branch_matrix(dev, n_items, d, k, extra):
    """Every branch of the fused path (and its boundary to the unfused one) under the acceptance rule.  Each case has
    one heavy row (more masked items than item groups), so the exact kernel runs next to the finalists kernel."""
    g = torch.Generator().manual_seed(n_items * 131 + d * 7 + k)
    B, n_u = 300, 400
    off = extra.get("item_offset", 0)
    if extra.get("offset_views"):
        ue = _randn((n_u * d + 1,), g).to(dev)[1:].view(n_u, d)
        ie = _randn((n_items * d + 1,), g).to(dev)[1:].view(n_items, d)
        assert ue.data_ptr() % 16 == 4 and ie.data_ptr() % 16 == 4
    else:
        ue, ie = _randn((n_u, d), g).to(dev), _randn((n_items, d), g).to(dev)
    users = torch.randint(0, n_u, (B,), generator=g).to(dev)
    G = -(-n_items // (16 * cf_gw(n_items)))
    masks = _rand_masks(B, n_items, 8, g, heavy=(B // 3, min(n_items - 1, G + 10)))
    masks = [m + off for m in masks]
    if off:                                                   # ids of the shards before and after this one
        masks = [np.concatenate([m, torch.randint(0, off, (3,), generator=g).numpy(),
                                 off + n_items + torch.randint(0, 5000, (3,), generator=g).numpy()]) for m in masks]
    mask = _mask_coo(masks, dev)
    fused = k <= 256 and -(-n_items // 128) * (8 // cf_gw(n_items)) >= 2 * k     # score_cf_supported
    val, idx, fb = _score_topk(ue, ie, users, mask, k, item_offset=off)
    if fused:
        assert fb >= 1                                        # the heavy row went through cf_exact_kernel
    else:
        assert fb == -1                                       # the unfused kernels served the call
    check_topk(ue, ie, users, mask, k, val, idx, item_offset=off, fused=fused)


# ------------------------------------------------------------------------------------------------ mask CSR builds
def _logical_mask(B, n, g):
    """Duplicate pairs, empty first and last rows, one heavy row (more masked items than item groups)."""
    masks = _rand_masks(B, n, 6, g, heavy=(B // 2, 400))
    masks[0] = masks[B - 1] = np.zeros(0, np.int64)
    for r in torch.randint(1, B - 1, (500,), generator=g).tolist():
        if len(masks[r]):
            masks[r] = np.concatenate([masks[r], masks[r][:1]])
    return masks


@gpu
def test_mask_builds_agree_bit_for_bit(dev):
    """One logical mask through the one-pass sorted build, the one-CTA build (unsorted), and the library-scan build
    (B > 8192, or more than 2^18 entries): the shared rows must come out bit-identical (the final values are the same fp32
    arithmetic whatever the candidate set)."""
    g = torch.Generator().manual_seed(21)
    n, d, k, B = 5000, 64, 50, 8192
    ue, ie = _randn((B + 1, d), g).to(dev), _randn((n, d), g).to(dev)
    masks = _logical_mask(B, n, g)
    srt = _mask_coo(masks, dev)
    shuf = srt[:, torch.randperm(srt.shape[1], generator=g).to(dev)]
    users = torch.arange(B, device=dev)
    v1, i1, _ = _score_topk(ue, ie, users, srt, k)                                    # sorted: one pass in cf_prep_kernel
    v2, i2, _ = _score_topk(ue, ie, users, shuf, k)                                   # mask_csr_small_kernel
    big = _mask_coo(masks + [np.array([1, 2, 3, 2])], dev)
    v3, i3, _ = _score_topk(ue, ie, torch.arange(B + 1, device=dev), big, k)         # B > 8192: count + scan + fill
    check_topk(ue, ie, users, srt, k, v1, i1)
    for v, i in ((v2, i2), (v3[:B], i3[:B])):
        assert torch.equal(i, i1) and torch.equal(v, v1)
    # 512 rows: 2^18 + 1 entries (large path) against the same mask minus one duplicate pair (2^18 entries, small path)
    n, B = 65536, 512
    ie = _randn((n, d), g).to(dev)
    masks = _rand_masks(B, n, 8, g)
    rest = (1 << 18) - 8 * 500
    for j, r in enumerate(range(500, 512)):                                           # 12 heavy rows (need > groups)
        masks[r] = torch.randperm(n, generator=g)[:rest // 12 + (j < rest % 12)].numpy()
    assert sum(len(m) for m in masks) == 1 << 18
    dup = [m.copy() for m in masks]
    dup[7] = np.concatenate([dup[7], dup[7][:1]])
    users = torch.arange(B, device=dev)
    mask_big, mask_small = _mask_coo(dup, dev), _mask_coo(masks, dev)
    assert mask_big.shape[1] == (1 << 18) + 1
    v1, i1, _ = _score_topk(ue, ie, users, mask_big, k)
    v2, i2, _ = _score_topk(ue, ie, users, mask_small, k)
    assert torch.equal(i1, i2) and torch.equal(v1, v2)
    check_topk(ue, ie, users, mask_small, k, v2, i2)


# ------------------------------------------------------------------------------------------------ exact-kernel routes
def _route_tables(n, d, g, n_copies=600):
    """Random tables with two reserved coordinates: 0 holds 3.0 on `n_copies` identical item rows (0 elsewhere on them)
    and is 0 for random users; 1 is >= 1 on every item and 0 for random users."""
    ie = _randn((n, d), g)
    ie[:, 0] = (torch.rand(n, generator=g) - 0.5) * 0.1
    ie[:, 1] = 1 + torch.rand(n, generator=g)
    copies = torch.randperm(n, generator=g)[:n_copies].sort().values
    ie[copies] = 0
    ie[copies, 0], ie[copies, 1] = 3.0, 1.0
    return ie, copies


def _route_users(n_u, d, g):
    ue = _randn((n_u, d), g)
    ue[:, :2] = 0
    return ue


def _exact_route_counts(capfd):
    from mmrec_b200 import ops
    capfd.readouterr()
    os.environ["MMREC_DEBUG"] = "1"
    try:
        n = ops.fused_fallback_rows()
    finally:
        del os.environ["MMREC_DEBUG"]
    err = capfd.readouterr().err
    m = re.search(r"exact-path rows (\d+) of (\d+) \(need > groups (\d+), non-finite (\d+), > \d+ candidates (\d+), < k kept (\d+)\)", err)
    assert m, err
    vals = [int(x) for x in m.groups()]
    assert vals[0] == n
    return dict(zip(["rows", "of", "need", "nonfinite", "cap", "kept"], vals))


@gpu
def test_exact_kernel_routes(dev, capfd):
    """Rows the filter hands to cf_exact_kernel: need > groups (a heavy user; a user with fewer than k unmasked items),
    more than 512 candidates (600 copies of the best item: the 50 lowest copy indices), non-finite scores (+inf in a
    coordinate every item has >= 1: items 0..k-1, values +inf).  The other rows are bit-identical to the same call
    without the special rows."""
    g = torch.Generator().manual_seed(8)
    n, d, k, B = 5000, 64, 50, 300
    ie, copies = _route_tables(n, d, g)
    ue = _route_users(B, d, g)
    masks = _rand_masks(B, n, 8, g)
    heavy, few, cap, inf = 0, 57, 128, B - 1
    masks[heavy] = torch.randperm(n, generator=g)[:400].numpy()               # need 450 > 313 groups
    masks[few] = torch.randperm(n, generator=g)[:n - 30].numpy()               # 30 unmasked items
    ue[cap] = 0; ue[cap, 0] = 1.0
    ue[inf] = 0; ue[inf, 1] = float("inf")
    ue, ie = ue.to(dev), ie.to(dev)
    users = torch.arange(B, device=dev)
    mask = _mask_coo(masks, dev)
    val, idx, fb = _score_topk(ue, ie, users, mask, k)
    cnt = _exact_route_counts(capfd)
    assert cnt == {"rows": 4, "of": B, "need": 2, "nonfinite": 1, "cap": 1, "kept": 0}, cnt
    assert torch.equal(idx[cap].cpu(), copies[:k]) and bool((val[cap] == 3.0).all())
    assert torch.equal(idx[inf].cpu(), torch.arange(k)) and bool((val[inf] == float("inf")).all())
    assert bool((val[few, 30:] == MASKED).all())
    finite = [r for r in range(B) if r != inf]
    check_topk(ue, ie, users, mask, k, val, idx, rows=finite)
    keep = [r for r in range(B) if r not in (heavy, few, cap, inf)]
    kt = torch.tensor(keep, device=dev)
    v2, i2, fb2 = _score_topk(ue, ie, kt, _mask_coo([masks[r] for r in keep], dev), k)
    assert fb2 == 0
    assert torch.equal(i2, idx[kt]) and torch.equal(v2, val[kt])


# ------------------------------------------------------------------------------------------------ several row blocks
@gpu
def test_several_row_blocks_1m_items(dev):
    """1 000 000 items, d = 64, B = 4096: row blocks of 3328 and 768 rows.  The heavy row and the 600-copies row sit in
    the first block; every row passes the acceptance rule, the rows on both sides of the block edge equal a call of their
    own, and the flags the diagnostic reads are those of the last block (none flagged there)."""
    g = torch.Generator().manual_seed(9)
    n, d, k, B = 1_000_000, 64, 50, 4096
    ie, copies = _route_tables(n, d, g)
    ue = _route_users(B, d, g)
    masks = _rand_masks(B, n, 8, g, heavy=(5, 8000))                            # need 8050 > 7813 groups
    cap = 100
    ue[cap] = 0; ue[cap, 0] = 1.0
    ue, ie = ue.to(dev), ie.to(dev)
    users = torch.arange(B, device=dev)
    mask = _mask_coo(masks, dev)
    val, idx, fb = _score_topk(ue, ie, users, mask, k)
    assert fb == 0
    assert torch.equal(idx[cap].cpu(), copies[:k]) and bool((val[cap] == 3.0).all())
    check_topk(ue, ie, users, mask, k, val, idx)
    edge = torch.tensor([3327, 3328], device=dev)
    v2, i2, _ = _score_topk(ue, ie, edge, _mask_coo([masks[3327], masks[3328]], dev), k)
    assert torch.equal(i2, idx[edge]) and torch.equal(v2, val[edge])


# ------------------------------------------------------------------------------------------------ CUDA graph replay
@gpu
def test_captured_score_topk_replays_on_new_user_table(dev):
    """score_topk with a packed catalogue, captured on a side stream (as bench.py does) and replayed after the user
    table was rewritten in place, equals an eager call on the new table."""
    from mmrec_b200 import ops
    g = torch.Generator().manual_seed(13)
    n, d, k, B = 7000, 64, 50, 2048
    ue, ie = _randn((B, d), g).to(dev), _randn((n, d), g).to(dev)
    users = torch.arange(B, device=dev)
    mask = _mask_coo(_rand_masks(B, n, 8, g, heavy=(3, 500)), dev)
    cat = ops.Catalog(ie)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for _ in range(2):
            ops.score_topk(ue, ie, users, mask, k, catalog=cat)
        torch.cuda.synchronize()
        gph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gph, stream=side):
            val, idx = ops.score_topk(ue, ie, users, mask, k, catalog=cat)
    torch.cuda.synchronize()
    for rep in range(2):
        ue.copy_(_randn((B, d), g).to(dev))
        gph.replay()
        torch.cuda.synchronize()
        ve, ie_ = ops.score_topk(ue, ie, users, mask, k, catalog=cat)
        assert torch.equal(idx, ie_) and torch.equal(val, ve), f"replay {rep}"
        check_topk(ue, ie, users, mask, k, val, idx)
