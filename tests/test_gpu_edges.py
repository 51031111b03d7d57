"""GPU tests of the tcgen05 sweeps and the fused seg-CE kernels at their tile and chunk edges, against float64.

The explicit sweeps (k_tc_fwd / k_tc_bwd) work on 128-row anchor tiles and 256-column contrast tiles (128-column
halves in the epilogue); the bank mode's transposed POS sweep (k_tc_pos_t) on blocks of at most 64 anchors of one class
and switches to the row-tile POS sweep above 4096 anchors; the seg-CE kernels loop over class chunks of at most 32
(forward) and 24 (backward) classes.  The shapes here sit on, just before and just after each of those edges.

Tolerances are those of DESIGN §2: tensor path loss <= 2e-5 relative to the float64 closed form on the bf16-rounded
operands and <= 1e-4 relative to the fp32 operands, gradient max-abs <= 4e-3 * max|g| and relative Frobenius <= 2e-3;
bank class blocks as in test_gpu_parity.test_tensor_path_bank_positives_by_class_blocks; seg-CE loss <= 2e-6 relative,
gradient <= 1e-5 * max|g|.  Positive counts (rowstats[4]) are exact.  The float64 references run on DEV."""
import pytest
import torch
import torch.nn.functional as F

import contrastiveseg_b200 as cs
from contrastiveseg_b200 import functional as Fn
from oracle import ref_port as P
from helpers import bank_infonce_chunked, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PAD_VALUE = 48.0           # contrast pad rows: a kernel that reads one as data gets exp(48 / T) into its sums


def _bf(x):
    return x.to(torch.bfloat16).to(x.dtype)


def _closed_form(a, ya, c, yc, T, bT, diag=None, self_contrast=False):
    """float64 InfoNCE of oracle.ref_port.infonce_closed_form; diag=None removes no column from the positives (the
    kernels' diag_col=NULL).  Rows without a positive give NaN like the reference."""
    if diag is not None or self_contrast:
        return P.infonce_closed_form(a, ya, c, yc, T, bT, self_contrast, diag_cols=diag)
    l = (a @ c.t()) / T
    m = l.max(1, keepdim=True).values
    e = torch.exp(l - m)
    same = ya.view(-1, 1) == yc.view(1, -1)
    neg = (e * (~same)).sum(1, keepdim=True)
    npos = same.sum(1, keepdim=True).to(a.dtype)
    logp = (l - m) - torch.log(e + neg)
    row_loss = -(T / bT) * (logp * same).sum(1, keepdim=True) / npos
    cc = (T / bT) / (a.shape[0] * npos)
    inv = 1.0 / (e + neg)
    s = (same * inv).sum(1, keepdim=True)
    G = torch.where(same, -cc * (1 - e * inv), torch.zeros_like(e)) + torch.where(~same, cc * e * s, torch.zeros_like(e))
    return dict(loss=row_loss.mean(), dA=(G @ c) / T, row_loss=row_loss[:, 0], npos=npos[:, 0])


def _check_tc(a, ya, c, yc, T, loss, st, dA, diag=None, self_contrast=False):
    """loss vs both float64 closed forms, positive counts exact, gradient vs the bf16-operand closed form."""
    a64, c64 = a.double().to(DEV), c.double().to(DEV)
    ya, yc = ya.to(DEV), yc.to(DEV)
    cf16 = _closed_form(_bf(a64), ya, _bf(c64), yc, T, 0.07, diag, self_contrast)
    cf32 = _closed_form(a64, ya, c64, yc, T, 0.07, diag, self_contrast)
    assert torch.equal(st[4].double(), cf16["npos"].to(st.device))
    ref = cf16["dA"]
    err = dA.double().to(DEV) - ref
    if ref.abs().max().item() == 0.0:            # one contrast column (N = 1): no negatives, zero loss and gradient
        # up to the approximate exp/log of the path: 2e-5 of the loss unit T / bT, 1e-5 per gradient element
        assert abs(loss.item()) <= 2e-5 * T / 0.07 and err.abs().max().item() <= 1e-5
        return
    assert rel_err(loss.item(), cf16["loss"].item()) < 2e-5, (loss.item(), cf16["loss"].item())
    if a.shape[0] >= 128:   # below, the bf16 rounding of the operands alone can move the loss by more than 1e-4
        assert rel_err(loss.item(), cf32["loss"].item()) < 1e-4, (loss.item(), cf32["loss"].item())
    assert err.abs().max().item() <= 4e-3 * ref.abs().max().item()
    assert (err.norm() / ref.norm()).item() < 2e-3


def _labels_with_partners(n, K, g):
    """n labels over K classes, each class used at least twice (every self-contrast row has a positive), shuffled."""
    K = max(1, min(K, n // 2))
    y = torch.arange(n) % K
    return y[torch.randperm(n, generator=g)]


def _unit(n, g, D=256):
    return F.normalize(torch.randn(n, D, generator=g), dim=1)


def _contrast16(c, alloc, pad=True):
    """bf16 copy of the contrast rows, rows [N, alloc) filled with PAD_VALUE instead of zeros when pad=True."""
    c16 = Fn.to_bf16_rows(c.to(DEV), alloc)
    if pad and alloc > c.shape[0]:
        c16[c.shape[0]:] = PAD_VALUE
    return c16


def _alloc(N):
    return -(-N // 256) * 256 + 256           # one spare 256-row tile beyond the rounding the sweeps need


# ---------------------------------------------------------------------------------------------------------------------
# 1. explicit tcgen05 sweeps (Fn.infonce_tc_forward / infonce_tc_backward)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("A", [2, 127, 128, 129, 255, 256, 257, 1023, 1024, 1025, 4097])
def test_tc_self_mode_at_row_tile_edges(A):
    """Self-contrast (mode 0): the anchors are the columns; A on, before and after the 128-row and 256-column tiles."""
    g = torch.Generator().manual_seed(1000 + A)
    a, ya = _unit(A, g), _labels_with_partners(A, 19, g)
    loss, st, state = Fn.infonce_tc_forward(a.to(DEV), ya.to(DEV), temperature=0.1, base_temperature=0.07)
    dA = Fn.infonce_tc_backward(state, st)
    _check_tc(a, ya, a, ya, 0.1, loss, st, dA, self_contrast=True)


EXPLICIT = [(1, 1), (1, 257), (127, 256), (128, 255), (128, 256), (129, 257), (127, 511), (128, 512), (129, 513),
            (1000, 1), (1000, 255), (1000, 65537), (129, 65537)]


@pytest.mark.parametrize("A,N", EXPLICIT)
def test_tc_explicit_mode_at_tile_edges(A, N):
    """Explicit contrast set (mode 2, sorted labels), A x N on the tile edges, rows [N, alloc) of contrast_bf16 filled
    with large values: columns >= n_cols must never be read as data.  diag_col (anchor i's own column i) where N >= A
    and N > 1."""
    g = torch.Generator().manual_seed(7 * A + N)
    K = min(19, N)
    a, c = _unit(A, g), _unit(N, g)
    yc = torch.sort(torch.randint(0, K, (N,), generator=g)).values
    cnt = torch.bincount(yc, minlength=K)
    diag = torch.arange(A) if N >= max(A, 2) else None
    ok = torch.nonzero(cnt >= (2 if diag is not None else 1))[:, 0]      # every row keeps a positive
    ya = ok[torch.randint(0, ok.numel(), (A,), generator=g)]
    loss, st, state = Fn.infonce_tc_forward(a.to(DEV), ya.to(DEV), contrast_bf16=_contrast16(c, _alloc(N)),
                                            contrast_cls=yc.to(DEV), n_cols=N,
                                            diag_col=None if diag is None else diag.to(DEV), temperature=0.07,
                                            base_temperature=0.07)
    dA = Fn.infonce_tc_backward(state, st)
    _check_tc(a, ya, c, yc, 0.07, loss, st, dA, diag=diag)


BLOCKS = [[1, 127, 128, 129, 256], [129, 1, 256, 127, 128], [128, 128, 1, 129, 127, 256]]


@pytest.mark.parametrize("sorted_cols", [True, False])
@pytest.mark.parametrize("blocks", range(len(BLOCKS)))
def test_tc_class_blocks_on_half_tile_boundaries(blocks, sorted_cols):
    """Class blocks of 1, 127, 128, 129 and 256 columns: 128-column half tiles that hold one class (the fast path of the
    sorted sweep) next to ones that straddle a class boundary (the per-column compare).  sorted_cols=False: the same
    columns shuffled, labels compared column by column.  Pad rows non-zero, no diagonal removed (every class, also the
    1-column one, is a positive for its anchors)."""
    lens = BLOCKS[blocks]
    g = torch.Generator().manual_seed(31 + blocks)
    yc = torch.repeat_interleave(torch.arange(len(lens)), torch.tensor(lens))
    N, A = yc.numel(), 257
    a, c = _unit(A, g), _unit(N, g)
    ya = torch.randint(0, len(lens), (A,), generator=g)
    if not sorted_cols:
        p = torch.randperm(N, generator=g)
        c, yc = c[p], yc[p]
    loss, st, state = Fn.infonce_tc_forward(a.to(DEV), ya.to(DEV), contrast_bf16=_contrast16(c, _alloc(N)),
                                            contrast_cls=yc.to(DEV), n_cols=N, temperature=0.1, base_temperature=0.07,
                                            sorted_cols=sorted_cols)
    dA = Fn.infonce_tc_backward(state, st)
    _check_tc(a, ya, c, yc, 0.1, loss, st, dA)


def test_tc_nan_safe_row_without_positive():
    """One anchor whose class has no column: NaN like the reference without nan_safe, a zero row loss and a zero gradient
    row with it; every other row as the closed form (mean over all A rows)."""
    g = torch.Generator().manual_seed(5)
    A, N = 129, 257
    a, c = _unit(A, g), _unit(N, g)
    yc = torch.sort(torch.randint(0, 6, (N,), generator=g)).values
    ya = yc[torch.randint(0, N, (A,), generator=g)]
    ya[77] = 11                                                   # no column of class 11
    c16 = _contrast16(c, _alloc(N))
    kw = dict(contrast_bf16=c16, contrast_cls=yc.to(DEV), n_cols=N, temperature=0.1, base_temperature=0.07)
    loss, _, _ = Fn.infonce_tc_forward(a.to(DEV), ya.to(DEV), **kw)
    assert torch.isnan(loss).item()
    loss, st, state = Fn.infonce_tc_forward(a.to(DEV), ya.to(DEV), nan_safe=True, **kw)
    dA = Fn.infonce_tc_backward(state, st).double().to(DEV)
    cf = _closed_form(_bf(a.double()).to(DEV), ya.to(DEV), _bf(c.double()).to(DEV), yc.to(DEV), 0.1, 0.07)
    assert torch.equal(st[4].double(), cf["npos"].to(st.device))
    want = torch.nan_to_num(cf["row_loss"], nan=0.0).mean().item()
    assert rel_err(loss.item(), want) < 2e-5, (loss.item(), want)
    assert dA[77].abs().max().item() == 0.0
    keep = torch.arange(A, device=DEV) != 77
    ref = torch.nan_to_num(cf["dA"], nan=0.0)[keep]
    assert (dA[keep] - ref).abs().max().item() <= 4e-3 * ref.abs().max().item()


# ---------------------------------------------------------------------------------------------------------------------
# 2. bank mode at class-block and anchor-block edges
# ---------------------------------------------------------------------------------------------------------------------
COUNTS = [1, 63, 64, 65, 128, 129]


def _bank_case(K, M, counts, seed):
    """Anchors with counts[c] rows of class c, in the engine's class-rank order 1..K-1, 0; bank shadow rebuilt from the
    fp32 queues with its pad rows beyond (K-1)*2M (and one spare tile) set to PAD_VALUE."""
    from contrastiveseg_b200 import _abi
    from contrastiveseg_b200.bank import shadow_rows
    g = torch.Generator().manual_seed(seed)
    order = list(range(1, K)) + [0]
    ya = torch.cat([torch.full((counts[c],), c, dtype=torch.long) for c in order])
    A = ya.numel()
    a = _unit(A, g)
    segq = F.normalize(torch.randn(K, M, 256, generator=g), dim=2)
    pixq = F.normalize(torch.randn(K, M, 256, generator=g), dim=2)
    shadow = torch.empty((shadow_rows(K, M) + 256, 256), dtype=torch.bfloat16, device=DEV)
    segq_d, pixq_d = segq.to(DEV), pixq.to(DEV)
    lib = _abi.load()
    _abi.check(lib.pcl_bank_shadow_rebuild(segq_d.data_ptr(), pixq_d.data_ptr(), K, M, 256, shadow.data_ptr(), None))
    torch.cuda.synchronize()
    shadow[(K - 1) * 2 * M:] = PAD_VALUE
    loss, st, state = Fn.infonce_tc_forward(a.to(DEV), ya.to(DEV), bank=(shadow, K, 2 * M),
                                            diag_col=torch.arange(A).to(DEV), temperature=0.1, base_temperature=0.07)
    dA = Fn.infonce_tc_backward(state, st).double().to(DEV)
    cf = bank_infonce_chunked(_bf(a.double()).to(DEV), ya, torch.arange(A), _bf(segq.double()).to(DEV),
                              _bf(pixq.double()).to(DEV), 0.1, 0.07)
    assert torch.equal(st[4].double(), cf["npos"].to(st.device))
    assert abs(loss.item() - cf["loss"].item()) <= 5e-5 * abs(cf["loss"].item()), (loss.item(), cf["loss"].item())
    assert (dA - cf["dA"]).abs().max().item() <= 6e-3 * cf["dA"].abs().max().item()


@pytest.mark.parametrize("M", [63, 64, 65, 127, 128, 129])
def test_tc_bank_class_blocks_at_tile_edges(M):
    """R = 2M on, before and after the 128/256-column tiles; per-class anchor counts around the 64-anchor blocks of
    k_tc_pos_t, class 0 (positives: the analytic zero tail) included."""
    K = 8
    rot = M % len(COUNTS)
    counts = [COUNTS[(c + rot) % len(COUNTS)] for c in range(K)]
    _bank_case(K, M, counts, seed=M)


@pytest.mark.parametrize("A", [4096, 4097, 6000])
def test_tc_bank_pos_sweep_crossover(A):
    """A <= 4096: transposed POS sweep; A > 4096: the row-tile POS sweep.  Both against the same float64 reference."""
    K, M = 19, 65
    g = torch.Generator().manual_seed(A)
    counts = [COUNTS[i % len(COUNTS)] for i in range(K)]
    rest = A - sum(counts)
    extra = torch.bincount(torch.randint(0, K, (rest,), generator=g), minlength=K).tolist()
    _bank_case(K, M, [n + e for n, e in zip(counts, extra)], seed=A)


# ---------------------------------------------------------------------------------------------------------------------
# 5. seg-CE over several class chunks
# ---------------------------------------------------------------------------------------------------------------------
def _segce_case(B, K, h, w, H, W, weighted, ign, seed):
    g = torch.Generator().manual_seed(seed)
    seg = torch.randn(B, K, h, w, generator=g) * 2.0
    target = torch.randint(0, K, (B, H, W), generator=g)
    target[torch.rand(B, H, W, generator=g) < 0.2] = ign
    weight = (torch.rand(K, generator=g) + 0.5) if weighted else None
    s1 = seg.clone().to(DEV).requires_grad_(True)
    loss = cs.upsample_cross_entropy(s1, target.to(DEV), weight.to(DEV) if weighted else None, ign)
    loss.backward(torch.tensor(0.7, device=DEV))
    s2 = seg.clone().double().to(DEV).requires_grad_(True)
    ref = P.seg_cross_entropy(s2, target.to(DEV), ign, weight.double().to(DEV) if weighted else None)
    ref.backward(torch.tensor(0.7, dtype=torch.float64, device=DEV))
    assert rel_err(loss.item(), ref.item()) < 2e-6, (loss.item(), ref.item())
    gmax = s2.grad.abs().max().item()
    assert (s1.grad.double().to(DEV) - s2.grad).abs().max().item() <= 1e-5 * gmax


@pytest.mark.parametrize("ign", [-1, 255])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("K", [24, 25, 32, 33, 59, 150, 171])
def test_segce_class_chunks(K, weighted, ign):
    """Forward chunks of <= 32 classes, backward chunks of <= 24: K on and across both chunk sizes, and the reference
    configs' K = 59 / 150 / 171, on a small up-sampling geometry."""
    _segce_case(2, K, 9, 11, 37, 45, weighted, ign, seed=K * 4 + 2 * weighted + (ign > 0))


@pytest.mark.parametrize("weighted", [False, True])
def test_segce_coco_stuff_geometry(weighted):
    """BASELINE configs[3] geometry: 171 classes, 66x66 logits up-sampled to 520x520, B = 2."""
    _segce_case(2, 171, 66, 66, 520, 520, weighted, 255 if weighted else -1, seed=171)


def test_contrast_ce_wrapper_171_classes_fused_toggle():
    """ContrastCELoss at K = 171 (configs[3] geometry): the same loss and gradients with fused_seg_ce on and off."""
    from contrastiveseg_b200.synth import make_contrast_batch
    data = make_contrast_batch(B=2, D=32, h=66, w=66, num_classes=171, img_stride=8, block=40, seed=171, himg=520, wimg=520)
    seg, tgt, emb = data["seg"].to(DEV), data["target"].to(DEV), data["embed"].to(DEV)
    out = []
    for fused in (True, False):
        cfg = cs.Configer({"data": {"num_classes": 171}, "network": {"stride": 8},
                           "loss": {"params": {"ce_ignore_index": -1, "ce_reduction": "elementwise_mean"}},
                           "contrast": {"temperature": 0.1, "base_temperature": 0.07, "max_samples": 1024, "max_views": 10,
                                        "loss_weight": 0.1, "use_rmi": False, "use_lovasz": False, "fused_seg_ce": fused}})
        crit = cs.ContrastCELoss(cfg).to(DEV)
        crit.contrast_criterion.perm_fn = P.PermRecorder(torch.Generator().manual_seed(1))
        s, e = seg.clone().requires_grad_(True), emb.clone().requires_grad_(True)
        loss = crit({"seg": s, "embed": e}, tgt, with_embed=True)
        loss.backward()
        out.append((loss.item(), s.grad.clone(), e.grad.clone()))
    assert rel_err(out[0][0], out[1][0]) < 5e-6
    assert (out[0][1] - out[1][1]).abs().max().item() <= 2e-5 * out[1][1].abs().max().item()
    assert torch.equal(out[0][2], out[1][2])                      # same anchors, same contrast gradient
