"""GPU tests of the captured steps against float64, with the anchors the host model of the device sampler predicts (the
file sorts after the non-capturing GPU tests on purpose: it captures CUDA graphs).

* the fused small-anchor step (k_self_fused) at anchor counts A = TC * V chosen on the 128/256 tile edges, and with A
  changing between replays of one captured graph (rows of an earlier, larger replay must not leak into a smaller one);
* the steps bench.py times, built the way bench.Workload builds them: S1 (fused, B = 8 and B = 1, full fill and
  sparse_reset) and S2 (bank step with enqueue, M = 5000), including the bank after every replay.

The expected anchors of replay r come from contrastiveseg_b200.rng (counter r + 1), not from the step's workspace, so the
scan, the plan and the selection are checked along with the loss kernel.  Tolerances as in test_gpu_edges.py."""
import pytest
import torch

import contrastiveseg_b200 as cs
from contrastiveseg_b200 import rng
from oracle import ref_port as P
from helpers import bank_infonce_chunked, rel_err

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]
DEV = "cuda:0"


def _bf(x):
    return x.to(torch.bfloat16).to(x.dtype)


def model_anchors(lab, prd, K, ms, mv, seed, counter):
    """Host model of the device sampler: [(image, class, pixel, reference row)] of the eager call / replay with this
    counter, in the reference's row order (view-major: row = view * TC + pair)."""
    step_seed = rng.device_step_seed(seed, counter)
    B = lab.shape[0]
    kept = [(b, c) for b in range(B) for c in range(K) if int((lab[b] == c).sum()) > mv]
    TC = len(kept)
    if TC == 0:
        return []
    V = min(ms // TC, mv)
    out = []
    for t, (b, c) in enumerate(kept):
        is_c = lab[b] == c
        hard = (is_c & (prd[b] != c)).nonzero()[:, 0].tolist()
        easy = (is_c & (prd[b] == c)).nonzero()[:, 0].tolist()
        kh, ke = P.split_hard_easy(len(hard), len(easy), V)
        views = [hard[rng.device_rank(step_seed, b, c, K, False, j, len(hard))] for j in range(kh)]
        views += [easy[rng.device_rank(step_seed, b, c, K, True, j, len(easy))] for j in range(ke)]
        out += [(b, c, px, v * TC + t) for v, px in enumerate(views)]
    return out


def check_step_against_model(embed, lab, prd, K, opts, counter, loss, grad, bank=None):
    """Loss and gradient rows of one replay against float64 on the model's anchors; exact zeros at every other pixel.
    bank=(segment_queue, pixel_queue) before the replay: bank mode (bank_infonce_chunked on the bf16-rounded queues)."""
    B, D, h, w = embed.shape
    anc = model_anchors(lab, prd, K, opts.max_samples, opts.max_views, opts.seed, counter)
    A = len(anc)
    assert A > 0
    img, cls, pix, ref = (torch.tensor(x, dtype=torch.long) for x in zip(*anc))
    X = embed.permute(0, 2, 3, 1).reshape(B, h * w, D)
    rows = X[img.to(X.device), pix.to(X.device)].double().to(DEV)
    G = grad.permute(0, 2, 3, 1).reshape(B, h * w, D)
    got = G[img.to(G.device), pix.to(G.device)].double().to(DEV)
    mask = torch.zeros(B, h * w, dtype=torch.bool, device=G.device)
    mask[img.to(G.device), pix.to(G.device)] = True
    assert int((G[~mask] != 0).sum().item()) == 0                 # nothing outside the sampled pixels
    T, bT = opts.temperature, opts.base_temperature
    if bank is None:
        cf16 = P.infonce_closed_form(_bf(rows), cls.to(DEV), _bf(rows), cls.to(DEV), T, bT, True)
        cf32 = P.infonce_closed_form(rows, cls.to(DEV), rows, cls.to(DEV), T, bT, True)
        assert rel_err(loss.item(), cf16["loss"].item()) < 2e-5, (loss.item(), cf16["loss"].item())
        if A >= 128:     # below, the bf16 rounding of the operands alone moves the loss by more than 1e-4 (A = 4: 4e-4)
            assert rel_err(loss.item(), cf32["loss"].item()) < 1e-4, (loss.item(), cf32["loss"].item())
        ref_g = cf16["dA"]
        err = got - ref_g
        assert err.abs().max().item() <= 4e-3 * ref_g.abs().max().item()
        # Frobenius: the kernel rounds the gradient tile G (A x A) to bf16 before dA = (G X + G^T X) / T, so
        # |dA err| <= u (|G| |X| + |G|^T |X|) / T elementwise, u = 2^-9.  G's rows nearly cancel, which puts this above
        # 2e-3 * |dA| at A ~ 1024 (measured 2.1e-3 .. 2.4e-3 relative on a B200 at 1000 W); max-abs stays within 4e-3.
        Xa, Ga = _bf(rows).abs(), cf16["G"].abs()
        bound = 2.0 ** -9 * ((Ga @ Xa + Ga.t() @ Xa) / T).norm().item()
        assert err.norm().item() <= bound, (err.norm().item(), bound, (err.norm() / ref_g.norm()).item())
    else:
        segq, pixq = bank
        cf = bank_infonce_chunked(_bf(rows), cls, ref, _bf(segq.double().to(DEV)), _bf(pixq.double().to(DEV)), T, bT)
        assert abs(loss.item() - cf["loss"].item()) <= 5e-5 * abs(cf["loss"].item()), (loss.item(), cf["loss"].item())
        assert (got - cf["dA"]).abs().max().item() <= 6e-3 * cf["dA"].abs().max().item()
    return A


def exact_label_map(B, h, w, K, pairs, g):
    """(B, h, w) labels: pair (b, c, n) puts n pixels of class c at random places of image b; every other pixel is the
    ignore label.  Plus (B, K, h, w) logits whose argmax is a prediction with roughly half of every class's pixels
    easy, and that prediction (B, h * w)."""
    lab = torch.full((B, h * w), -1, dtype=torch.long)
    for b, c, n in pairs:
        free = (lab[b] == -1).nonzero()[:, 0]
        lab[b, free[torch.randperm(free.numel(), generator=g)[:n]]] = c
    easy = torch.rand(B, h * w, generator=g) < 0.5
    prd = torch.where(easy & (lab >= 0), lab, (lab + 1 + torch.randint(0, K - 1, (B, h * w), generator=g)) % K)
    seg = torch.randn(B, K, h * w, generator=g)
    seg.scatter_add_(1, prd.unsqueeze(1), torch.full((B, 1, h * w), 8.0))
    return lab.view(B, h, w), seg.view(B, K, h, w), prd


def _opts(K, ms, mv, seed=5):
    return cs.ContrastOptions(temperature=0.1, base_temperature=0.07, max_samples=ms, max_views=mv, seed=seed,
                              precision="bf16", num_classes=K)


# (A, TC, V, max_samples, max_views): A = TC * V = TC * min(max_samples // TC, max_views)
EXACT = [(4, 2, 2, 1024, 2), (128, 2, 64, 1024, 64), (129, 3, 43, 130, 43), (256, 4, 64, 1024, 64),
         (258, 2, 129, 300, 129), (1023, 3, 341, 1023, 341), (1024, 8, 128, 1024, 128)]


@pytest.mark.parametrize("A,TC,V,ms,mv", EXACT)
def test_fused_step_at_exact_anchor_counts(A, TC, V, ms, mv):
    """Fused step on label maps built so that exactly TC (image, class) pairs qualify, A = TC * V on the 128-row /
    256-column tile edges (max_samples, which sizes the tile grid, also off the multiples of 128).  Three replays."""
    B, h, w, D, K = 4, 48, 48, 256, 19
    assert A == TC * V == TC * min(ms // TC, mv)
    g = torch.Generator().manual_seed(A)
    pairs = [(t % B, 1 + t, mv + 1 + int(torch.randint(0, 40, (1,), generator=g))) for t in range(TC)]
    lab, seg, prd = exact_label_map(B, h, w, K, pairs, g)
    embed = torch.nn.functional.normalize(torch.randn(B, D, h, w, generator=g), dim=1)
    opts = _opts(K, ms, mv)
    step = cs.GraphedContrastStep(embed.to(DEV), lab.to(DEV), seg=seg.to(DEV), options=opts)
    assert step.fused
    for r in range(3):
        loss, grad = step.replay()
        torch.cuda.synchronize()
        assert check_step_against_model(embed, lab.view(B, -1), prd, K, opts, r + 1, loss, grad) == A


def _one_view_pairs(A, B, seed):
    """max_views = 1: A qualifying pairs give A anchors; every class sits in >= 2 images (a positive for every row)."""
    g = torch.Generator().manual_seed(seed)
    pairs = []
    c = 0
    while len(pairs) < A:
        k = min(A - len(pairs), B, max(2, A // 2))                # at least two classes (negatives for every row)
        k = k if A - len(pairs) - k != 1 else k - 1                 # never leave a class with a single image
        imgs = torch.randperm(B, generator=g)[:k].tolist()
        pairs += [(b, c, 2 + int(torch.randint(0, 2, (1,), generator=g))) for b in imgs]
        c += 1
    return pairs, g


@pytest.mark.parametrize("sparse_reset", [False, True])
def test_fused_step_anchor_count_changes_between_replays(sparse_reset):
    """One captured fused step, new inputs copied into its static tensors between replays so that A goes
    1024 -> 129 -> 4 -> 1024 (max_views = 1, A = number of qualifying pairs).  The bf16 pad rows of a smaller replay must
    be zero (selection) and masked (row < A, cj < A in the fused kernel): every replay equals float64 on its own anchors,
    and the gradient is exactly zero outside them — with sparse_reset also at the pixels of the previous replay."""
    B, h, w, D, K = 8, 16, 32, 256, 130
    inputs = []
    for i, A in enumerate((1024, 129, 4, 1024)):
        pairs, g = _one_view_pairs(A, B, seed=10 + i)
        lab, seg, prd = exact_label_map(B, h, w, K, pairs, g)
        embed = torch.nn.functional.normalize(torch.randn(B, D, h, w, generator=g), dim=1)
        inputs.append((A, embed, lab, seg, prd))
    opts = _opts(K, 1024, 1)
    _, e0, l0, s0, _ = inputs[0]
    embed_d, lab_d, seg_d = e0.to(DEV), l0.to(DEV), s0.to(DEV)
    step = cs.GraphedContrastStep(embed_d, lab_d, seg=seg_d, options=opts, sparse_reset=sparse_reset)
    assert step.fused and step.sparse_reset == sparse_reset
    for r, (A, embed, lab, seg, prd) in enumerate(inputs):
        embed_d.copy_(embed.to(DEV)); lab_d.copy_(lab.to(DEV)); seg_d.copy_(seg.to(DEV))
        loss, grad = step.replay()
        torch.cuda.synchronize()
        assert check_step_against_model(embed, lab.view(B, -1), prd, K, opts, r + 1, loss, grad) == A, r


# ---------------------------------------------------------------------------------------------------------------------
# the benched shapes (bench.py S1 / S2, built like bench.Workload)
# ---------------------------------------------------------------------------------------------------------------------
def _bench_step(cfg, bank, sparse_reset=False, seed=304):
    import bench
    host = bench.make_inputs(cfg, seed, None, bank)
    inp = {k: host[k].to(DEV) for k in ("embed", "seg", "target")}
    crit = cs.PixelContrastLoss(bench.engine_configer(cfg, bank, "bf16"))
    opts = crit.options()
    opts.num_classes = cfg["K"]
    kw, mbank = {}, None
    if bank:
        mbank = cs.MemoryBank(cfg["K"], cfg["M"], cfg["D"], with_shadow=True).to(DEV)
        mbank.segment_queue.copy_(host["segment_queue"]); mbank.pixel_queue.copy_(host["pixel_queue"])
        mbank.sync_shadow()
        kw = dict(segment_queue=mbank.segment_queue, pixel_queue=mbank.pixel_queue, bank_shadow=mbank.shadow,
                  enqueue=dict(bank=mbank, network_stride=cfg["net_stride"], pixel_update_freq=cfg["F"]))
    step = cs.GraphedContrastStep(inp["embed"], inp["target"], seg=inp["seg"], options=opts, sparse_reset=sparse_reset, **kw)
    lab = P.downsample_labels(host["target"], cfg["h"], cfg["w"]).reshape(cfg["B"], -1)
    prd = host["seg"].argmax(1).reshape(cfg["B"], -1)
    return step, host, lab, prd, opts, mbank


@pytest.mark.parametrize("sparse_reset", [False, True])
@pytest.mark.parametrize("B", [8, 1])
def test_bench_s1_fused_step_matches_float64(B, sparse_reset):
    """bench.py's headline step (S1: fused bf16 graphed step, 128x256, K = 19, max_samples 1024, max_views 100) at B = 8
    and at the B = 1 of strong scaling on 8 GPUs: three replays against the host-model anchors and float64."""
    import bench
    cfg = dict(bench.S1, B=B)
    step, host, lab, prd, opts, _ = _bench_step(cfg, False, sparse_reset)
    assert step.fused
    for r in range(3):
        loss, grad = step.replay()
        torch.cuda.synchronize()
        check_step_against_model(host["embed"], lab, prd, cfg["K"], opts, r + 1, loss, grad)


def _model_perms(labels, K, stride, F, seed):
    """The permutations the reference's enqueue would have to draw to pick the device's rows: per (image, class > 0) slot
    in the reference's order, device_bank_rank for the first min(n, F) entries, then the remaining values."""
    sub = labels[:, ::stride, ::stride].reshape(labels.shape[0], -1)
    perms = []
    for b in range(sub.shape[0]):
        for c in [int(x) for x in torch.unique(sub[b]).tolist() if 0 < x < K]:
            n = int((sub[b] == c).sum())
            head = [rng.device_bank_rank(seed, b * K + c, j, n) for j in range(min(n, F))]
            rest = sorted(set(range(n)) - set(head))
            perms.append(torch.tensor(head + rest, dtype=torch.long))
    return perms


def test_device_bank_rank_is_the_packet_kernels_draw():
    """rng.device_bank_rank pinned to k_bank_rows: the packet built from ranks given explicitly by the model equals the
    packet the kernel draws itself from the seed, bit for bit."""
    import ctypes as C
    from contrastiveseg_b200 import _abi
    from contrastiveseg_b200.synth import make_contrast_batch
    K, F, stride, seed = 7, 5, 2, 0xDEADBEEF12345
    data = make_contrast_batch(B=2, D=32, h=24, w=20, num_classes=K, img_stride=2, block=6, seed=8)
    keys, labels = data["embed"].to(DEV), data["target"].to(DEV)
    lib = _abi.load()
    g = _abi.BankGeom(2, 32, 24, 20, labels.shape[1], labels.shape[2], K, 16, stride, F)
    sub = data["target"][:, ::stride, ::stride].reshape(2, -1)
    ranks = torch.zeros(2 * K, F, dtype=torch.int32)
    for b in range(2):
        for c in range(1, K):
            n = int((sub[b] == c).sum())
            for j in range(min(n, F)):
                ranks[b * K + c, j] = rng.device_bank_rank(seed, b * K + c, j, n)
    assert int((ranks != 0).sum()) > 10
    ranks = ranks.to(DEV)
    out = []
    for rk in (None, ranks):
        scratch = torch.zeros(int(lib.pcl_bank_scratch_floats(C.byref(g))), device=DEV)
        packet = torch.zeros(int(lib.pcl_bank_packet_floats(C.byref(g))), device=DEV)
        _abi.check(lib.pcl_bank_packet(C.byref(g), keys.data_ptr(), labels.data_ptr(), _abi.ptr(rk), seed,
                                       scratch.data_ptr(), packet.data_ptr(), None))
        torch.cuda.synchronize()
        out.append(packet)
    assert torch.equal(out[0], out[1])


def test_bench_s2_graphed_bank_step_matches_float64_and_the_reference_enqueue():
    """bench.py's bank block (S2: graphed bank step with enqueue, K = 19, M = 5000, F = 10): every replay's loss and
    gradient against float64 on the bank as it was before the replay, and the bank after the replay against
    oracle.ref_port.dequeue_and_enqueue with the device's draws: pointers exact, rows within the apply bounds, the bf16
    shadow equal to bf16 of the rows."""
    from contrastiveseg_b200 import bank as bank_mod
    import bench
    cfg = bench.S2
    K, M, D, F, stride = cfg["K"], cfg["M"], cfg["D"], cfg["F"], cfg["net_stride"]
    step, host, lab, prd, opts, mbank = _bench_step(cfg, True)
    names = ("segment_queue", "segment_queue_ptr", "pixel_queue", "pixel_queue_ptr")
    ref = [getattr(mbank, n).detach().cpu().clone() for n in names]
    for r in range(3):
        before = (mbank.segment_queue.clone(), mbank.pixel_queue.clone())
        loss, grad = step.replay()
        torch.cuda.synchronize()
        check_step_against_model(host["embed"], lab, prd, K, opts, r + 1, loss, grad, bank=before)
        seed = (bank_mod.enqueue_seed(304) + 1 + r) & 0xFFFFFFFFFFFFFFFF
        replay = P.PermReplay(_model_perms(host["target"], K, stride, F, seed))
        P.dequeue_and_enqueue(host["embed"], host["target"], *ref, network_stride=stride, memory_size=M,
                              pixel_update_freq=F, perm_fn=replay)
        assert replay.pos == len(replay.draws)
        mine = [getattr(mbank, n).detach().cpu() for n in names]
        assert torch.equal(mine[1], ref[1]) and torch.equal(mine[3], ref[3]), r
        assert (mine[0] - ref[0]).abs().max().item() <= 2e-6, r
        assert (mine[2] - ref[2]).abs().max().item() <= 2e-7, r
        rows = torch.cat((mbank.segment_queue[1:], mbank.pixel_queue[1:]), dim=1).reshape(-1, D)
        assert torch.equal(mbank.shadow[: rows.shape[0]], rows.to(torch.bfloat16)), r
