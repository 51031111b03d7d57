"""TEST INFRASTRUCTURE: differential fuzzing of the engine (real SIMT kernel sources on the host-fiber emulator,
tests/emu) against the oracle over random geometries.  Used by tests/test_emu_fuzz.py (bounded) and
tools/emu_fuzz.py (long runs).  Every fuzzer returns a list of failure descriptions (empty = clean).

It found the out-of-bounds wrap write for pixel_update_freq > memory_size (now refused, csrc/pcl_bank.cu: make_dims)."""
import math
import random

import torch
import torch.nn.functional as F

import contrastiveseg_b200 as cs
from contrastiveseg_b200 import _abi, functional as Fn
from contrastiveseg_b200.synth import make_bank, make_contrast_batch
from oracle import ref_port as P


def _cfg(T, bT, ms, mv, K):
    return cs.Configer({"data": {"num_classes": K},
                        "contrast": {"temperature": T, "base_temperature": bT, "max_samples": ms, "max_views": mv,
                                     "loss_weight": 0.1},
                        "loss": {"params": {"ce_ignore_index": -1}}, "network": {"stride": 8}})


def _rel(a, b):
    return abs(a - b) / max(abs(b), 1e-9)


def fuzz_loss(seed: int, n: int):
    """PixelContrastLoss (exact path, injected permutations) vs the float64 oracle: random batch / embedding / image
    sizes (divisible and not), class counts, sampling limits, with and without bank, seg logits or predictions.
    Degenerate inputs: the reference raises (no class qualifies, zero views) -> the engine returns an exact zero;
    rows without positives -> NaN on both sides."""
    rng = random.Random(seed)
    bad = []
    for it in range(n):
        B, D, h, w = rng.randint(1, 3), rng.choice([32, 64]), rng.randint(3, 36), rng.randint(3, 36)
        K, ms, mv = rng.randint(2, 12), rng.randint(4, 160), rng.randint(1, 16)
        block, boost = rng.choice([2, 3, 5, 8, 16]), rng.choice([0.0, 1.0, 2.0, 4.0])
        if rng.random() < 0.5:
            st = rng.choice([1, 2, 4])
            himg, wimg = h * st, w * st
        else:
            himg, wimg = rng.randint(h, 4 * h + 3), rng.randint(w, 4 * w + 3)
        mem, M = rng.random() < 0.4, rng.randint(2, 24)
        T, bT, s = rng.choice([0.07, 0.1, 0.5]), rng.choice([0.07, 0.1]), rng.randint(0, 10 ** 6)
        use_seg = rng.random() < 0.5
        desc = (f"loss seed={seed} it={it} B={B} D={D} hw={h}x{w} img={himg}x{wimg} K={K} ms={ms} mv={mv} block={block} "
                f"boost={boost} mem={mem} M={M} T={T} seg={use_seg}")
        data = make_contrast_batch(B=B, D=D, h=h, w=w, num_classes=K, img_stride=1, block=block, boost=boost, seed=s,
                                   himg=himg, wimg=wimg)
        bank = make_bank(K, M, D, s + 1) if mem else None
        rec = P.PermRecorder(torch.Generator().manual_seed(s))
        e64 = data["embed"].double().requires_grad_(True)
        q = torch.cat((bank["segment_queue"], bank["pixel_queue"]), 1).double() if mem else None
        predict = data["seg"].argmax(1)
        why = None
        try:
            ref = P.pixel_contrast_loss(e64, data["target"], predict, temperature=T, base_temperature=bT, max_samples=ms,
                                        max_views=mv, queue=q, perm_fn=rec)
            ref.backward()
        except (RuntimeError, IndexError, ValueError) as ex:
            why = type(ex).__name__
        crit = cs.PixelContrastLoss(_cfg(T, bT, ms, mv, K))
        crit.perm_fn = P.PermReplay(rec.draws) if why is None else (lambda k: torch.randperm(k))
        embed = data["embed"].clone().requires_grad_(True)
        queue = (bank["segment_queue"].clone(), bank["pixel_queue"].clone()) if mem else None
        loss = crit(embed, data["target"], predict=None if use_seg else predict, seg=data["seg"] if use_seg else None,
                    queue=queue)
        loss.backward()
        if why == "IndexError":
            continue          # more anchors than bank columns (Q1): the reference crashes, the engine masks nothing
        if why is not None:
            if not (loss.item() == 0.0 and embed.grad.abs().max().item() == 0.0):
                bad.append(f"degenerate input not answered with an exact zero: {desc} ({why}) loss={loss.item()}")
            continue
        lv, rv = loss.item(), ref.item()
        if math.isnan(rv):
            if not math.isnan(lv):
                bad.append(f"reference NaN, engine {lv}: {desc}")
            continue
        gerr = (embed.grad.double() - e64.grad).abs().max().item() / max(e64.grad.abs().max().item(), 1e-9)
        if _rel(lv, rv) > 5e-6 or gerr > 2e-5:
            bad.append(f"mismatch rel={_rel(lv, rv):.2e} gerr={gerr:.2e}: {desc}")
    return bad


def fuzz_bank(seed: int, n: int):
    """dequeue_and_enqueue over several steps (wrap-around, stride mismatch Q6, overlapping writes Q4) vs the oracle:
    pointers exact, rows to rounding; configurations the reference rejects must be rejected too."""
    rng = random.Random(seed)
    bad = []
    names = ("segment_queue", "segment_queue_ptr", "pixel_queue", "pixel_queue_ptr")
    for it in range(n):
        B, D, h, w, K = rng.randint(1, 3), rng.choice([32, 64]), rng.randint(3, 30), rng.randint(3, 30), rng.randint(2, 10)
        M, Fq, s, img_s = rng.randint(2, 20), rng.randint(1, 12), rng.choice([1, 2, 3, 4, 8]), rng.choice([1, 2, 4])
        block, steps, sd = rng.choice([2, 4, 8, 16]), rng.randint(1, 5), rng.randint(0, 10 ** 6)
        desc = f"bank seed={seed} it={it} B={B} D={D} hw={h}x{w} K={K} M={M} F={Fq} stride={s} img_stride={img_s} steps={steps}"
        b0 = make_bank(K, M, D, sd)
        ref = [b0[k].clone() for k in names]
        mine = [b0[k].clone() for k in names]
        done = True
        for st in range(steps):
            data = make_contrast_batch(B=B, D=D, h=h, w=w, num_classes=K, img_stride=img_s, block=block, seed=sd + st)
            rec = P.PermRecorder(torch.Generator().manual_seed(sd + st))
            r_ok = True
            try:
                P.dequeue_and_enqueue(data["embed"], data["target"], *ref, network_stride=s, memory_size=M,
                                      pixel_update_freq=Fq, perm_fn=rec)
            except (RuntimeError, IndexError):
                r_ok = False
            m_ok = True
            try:
                cs.dequeue_and_enqueue(data["embed"].clone(), data["target"], *mine, network_stride=s, memory_size=M,
                                       pixel_update_freq=Fq, distributed=False,
                                       perm_fn=P.PermReplay(rec.draws) if r_ok else (lambda k: torch.randperm(k)))
            except _abi.PclError:
                m_ok = False
            grid = -(-h * img_s // s) * -(-w * img_s // s)          # positions of labels[:, ::s, ::s]
            if r_ok and not m_ok and (Fq > M or grid > h * w):
                # refused up front from the geometry alone (documented): pixel_update_freq > memory_size, or a label
                # grid with more positions than feature columns (Q6) — the reference only fails there when the data
                # happens to put a labelled position / a large class beyond the limit
                done = False
                break
            if r_ok != m_ok:
                bad.append(f"refusal differs (reference ok={r_ok}, engine ok={m_ok}): {desc}")
                done = False
                break
            if not r_ok:
                done = False
                break
        if not done:
            continue
        if not (torch.equal(ref[1], mine[1]) and torch.equal(ref[3], mine[3])):
            bad.append(f"pointers differ: {desc}")
            continue
        e_seg, e_pix = (ref[0] - mine[0]).abs().max().item(), (ref[2] - mine[2]).abs().max().item()
        if e_seg > 2e-6 or e_pix > 2e-7:
            bad.append(f"rows differ seg={e_seg:.1e} pix={e_pix:.1e}: {desc}")
    return bad


def fuzz_segce(seed: int, n: int):
    """Fused bilinear(align_corners) up/down-sampling + weighted CE with ignore vs the float64 torch ops."""
    rng = random.Random(seed)
    bad = []
    for it in range(n):
        B, K, h, w = rng.randint(1, 3), rng.randint(2, 60), rng.randint(1, 20), rng.randint(1, 24)
        H, W, weighted, ign = rng.randint(1, 60), rng.randint(1, 60), rng.random() < 0.5, rng.choice([-1, 255, 0])
        g = torch.Generator().manual_seed(rng.randint(0, 10 ** 6))
        seg = torch.randn(B, K, h, w, generator=g) * 2
        target = torch.randint(0, K, (B, H, W), generator=g)
        target[torch.rand(B, H, W, generator=g) < 0.2] = ign
        weight = (torch.rand(K, generator=g) + 0.5) if weighted else None
        desc = f"segce seed={seed} it={it} B={B} K={K} {h}x{w}->{H}x{W} weighted={weighted} ignore={ign}"
        s1 = seg.clone().requires_grad_(True)
        loss = cs.upsample_cross_entropy(s1, target, weight, ign)
        loss.backward(torch.tensor(0.7))
        s2 = seg.clone().double().requires_grad_(True)
        ref = P.seg_cross_entropy(s2, target, ign, weight.double() if weighted else None)
        ref.backward(torch.tensor(0.7, dtype=torch.float64))
        if math.isnan(ref.item()):
            if not math.isnan(loss.item()):
                bad.append(f"reference NaN, engine {loss.item()}: {desc}")
            continue
        gerr = (s1.grad.double() - s2.grad).abs().max().item() / max(s2.grad.abs().max().item(), 1e-9)
        if _rel(loss.item(), ref.item()) > 3e-6 or gerr > 2e-5:
            bad.append(f"mismatch rel={_rel(loss.item(), ref.item()):.2e} gerr={gerr:.2e}: {desc}")
    return bad


def fuzz_device_sampling(seed: int, n: int, check_sampling):
    """Device RNG (keyed bijection, no injected permutations), optional fused normalise: every anchor a valid distinct
    pixel of its (image, class, hard|easy) group; loss / gradient vs the oracle evaluated on exactly those anchors."""
    rng = random.Random(seed)
    bad = []
    for it in range(n):
        B, D, h, w = rng.randint(1, 3), rng.choice([32, 64]), rng.randint(4, 40), rng.randint(4, 40)
        K, ms, mv = rng.randint(2, 10), rng.randint(4, 200), rng.randint(1, 16)
        block, st, boost = rng.choice([2, 4, 8, 16]), rng.choice([1, 2, 4]), rng.choice([0.0, 2.0, 4.0])
        mem, norm, sd = rng.random() < 0.4, rng.random() < 0.4, rng.randint(0, 10 ** 6)
        desc = f"devrng seed={seed} it={it} B={B} D={D} {h}x{w} K={K} ms={ms} mv={mv} block={block} st={st} mem={mem} norm={norm}"
        data = make_contrast_batch(B=B, D=D, h=h, w=w, num_classes=K, img_stride=st, block=block, boost=boost, seed=sd)
        bank = make_bank(K, rng.randint(8, 30), D, sd + 1)
        crit = cs.PixelContrastLoss(_cfg(0.1, 0.07, ms, mv, K))
        embed = (data["embed_raw"] if norm else data["embed"]).clone().requires_grad_(True)
        queue = (bank["segment_queue"].clone(), bank["pixel_queue"].clone()) if mem else None
        loss = crit(embed, data["target"], seg=data["seg"], queue=queue, normalize=norm)
        loss.backward()
        ws = Fn.last_workspace(embed.device)
        TC, V, A = ws.plan_header()[:3]
        lab = P.downsample_labels(data["target"], h, w).reshape(B, -1)
        prd = data["seg"].argmax(1).reshape(B, -1)
        if TC == 0 or V == 0:
            if loss.item() != 0.0:
                bad.append(f"degenerate input, loss {loss.item()}: {desc}")
            continue
        try:
            _, _, A2, meta = check_sampling(ws, lab, prd, ms, mv)
        except AssertionError as ex:
            bad.append(f"invalid sample set ({str(ex)[:120]}): {desc}")
            continue
        pix, img, cls, refrow = meta
        if mem and A > bank["segment_queue"].shape[0] * 2 * bank["segment_queue"].shape[1]:
            continue
        e64 = (data["embed_raw"] if norm else data["embed"]).double().requires_grad_(True)
        Xf = (F.normalize(e64, dim=1) if norm else e64).permute(0, 2, 3, 1).reshape(B, -1, D)
        inv = torch.empty(A, dtype=torch.long)
        inv[refrow] = torch.arange(A)
        anchors, ya = Xf[img, pix][inv], cls[inv].double()
        if mem:
            contrast, yc = P.flatten_queue(torch.cat((bank["segment_queue"], bank["pixel_queue"]), 1).double())
            lo = P.infonce_dense(anchors, ya, contrast, yc, 0.1, 0.07)
        else:
            lo = P.infonce_dense(anchors, ya, anchors, ya, 0.1, 0.07)
        lo.backward()
        if math.isnan(lo.item()):
            if not math.isnan(loss.item()):
                bad.append(f"reference NaN, engine {loss.item()}: {desc}")
            continue
        gerr = (embed.grad.double() - e64.grad).abs().max().item() / max(e64.grad.abs().max().item(), 1e-9)
        if _rel(loss.item(), lo.item()) > 5e-6 or gerr > 3e-5:
            bad.append(f"mismatch rel={_rel(loss.item(), lo.item()):.2e} gerr={gerr:.2e}: {desc}")
    return bad


def fuzz_topk(seed: int, n: int):
    """a10 top-k kernels vs the sort-based oracle: explicit / self / bank (zero tail) operands; exact dyadic data (ties,
    strict gradient check) and unit-norm data (near-ties: loss strict, gradient in norm)."""
    rng = random.Random(seed)
    bad = []
    for it in range(n):
        A, N, D, ncls = rng.randint(2, 150), rng.randint(2, 400), rng.choice([32, 64]), rng.randint(2, 8)
        k, exact, mode = rng.randint(1, 60), rng.random() < 0.5, rng.choice(["explicit", "self", "bank"])
        g = torch.Generator().manual_seed(rng.randint(0, 10 ** 6))
        desc = f"topk seed={seed} it={it} A={A} N={N} D={D} classes={ncls} k={k} exact={exact} mode={mode}"
        if exact:
            den = 4 if D == 32 else 8                       # keeps exp(l - m) inside the fp32 range
            mk = lambda *s: torch.randint(-3, 4, s, generator=g).double() / den      # noqa: E731
            T, bT = 0.125, 0.25
        else:
            mk = lambda *s: F.normalize(torch.randn(*s, generator=g), dim=-1).double()   # noqa: E731
            T, bT = 0.1, 0.07
        a, ya = mk(A, D), torch.randint(0, ncls, (A,), generator=g)
        if mode == "explicit":
            c, yc, diag = mk(N, D), torch.randint(0, ncls, (N,), generator=g), torch.arange(A) % N
            o = P.infonce_topk(a, ya, c, yc, T, bT, k, False, diag_cols=diag)
            loss, rs, st = Fn.infonce_forward(a.float(), ya, contrast=c.float(), contrast_cls=yc, diag_col=diag,
                                              temperature=T, base_temperature=bT, topk=k)
        elif mode == "self":
            o = P.infonce_topk(a, ya, a, ya, T, bT, k, True)
            loss, rs, st = Fn.infonce_forward(a.float(), ya, temperature=T, base_temperature=bT, topk=k)
        else:
            K, M = ncls, rng.randint(1, 12)
            if A > K * 2 * M:
                continue
            segq, pixq = mk(K, M, D), mk(K, M, D)
            if exact:
                pixq[:, ::3] = 0
            ya = ya[torch.argsort(torch.where(ya == 0, K, ya), stable=True)]
            contrast, yc = P.flatten_queue(torch.cat((segq, pixq), 1))
            o = P.infonce_topk(a, ya, contrast, yc.long(), T, bT, k, False)
            loss, rs, st = Fn.infonce_forward(a.float(), ya, queues=(segq.float(), pixq.float()),
                                              diag_col=torch.arange(A), temperature=T, base_temperature=bT, topk=k)
        dA = Fn.infonce_backward(st, rs).double()
        lo = o["loss"].item()
        if math.isnan(lo):
            if not math.isnan(loss.item()):
                bad.append(f"reference NaN, engine {loss.item()}: {desc}")
            continue
        if exact:
            gerr, tol = (dA - o["dA"]).abs().max().item() / max(o["dA"].abs().max().item(), 1e-9), 2e-5
        else:
            gerr, tol = (torch.linalg.norm(dA - o["dA"]) / max(torch.linalg.norm(o["dA"]).item(), 1e-9)).item(), 5e-2
        if _rel(loss.item(), lo) > 1e-5 or gerr > tol:
            bad.append(f"mismatch rel={_rel(loss.item(), lo):.2e} gerr={gerr:.2e}: {desc}")
    return bad


def _bf(x):
    return x.to(torch.bfloat16).to(torch.float32)


def fuzz_tensor_path(seed: int, n: int):
    """tcgen05 sweeps (functional model) on explicit operands: self-contrast, explicit contrast set (sorted / unsorted
    labels), bank through the bf16 shadow; ragged A and N (not multiples of the 128 x 256 tile), few / many classes.
    Loss and positive counts against the float64 closed form on the bf16-rounded operands; gradient within the bf16
    tolerance of the path (max-abs 6e-3 * max|g|, relative Frobenius 5e-3)."""
    from contrastiveseg_b200.bank import shadow_rows
    rng = random.Random(seed)
    bad = []
    lib = _abi.load()
    for it in range(n):
        A, N, ncls = rng.randint(1, 420), rng.randint(1, 1500), rng.randint(1, 20)
        T, mode, clustered = rng.choice([0.07, 0.1, 0.5]), rng.choice(["self", "sorted", "unsorted", "bank"]), rng.choice([0.0, 0.5])
        g = torch.Generator().manual_seed(rng.randint(0, 10 ** 6))
        desc = f"tensor seed={seed} it={it} A={A} N={N} classes={ncls} T={T} mode={mode} clustered={clustered}"
        centers = F.normalize(torch.randn(ncls + 1, 256, generator=g), dim=1)
        ya = torch.randint(0, ncls, (A,), generator=g)
        a = F.normalize(torch.randn(A, 256, generator=g) + clustered * 16 * centers[ya], dim=1)
        if mode == "self":
            loss, st, state = Fn.infonce_tc_forward(a, ya, temperature=T, base_temperature=0.07)
            cf = P.infonce_closed_form(_bf(a).double(), ya, _bf(a).double(), ya, T, 0.07, self_contrast=True)
        elif mode in ("sorted", "unsorted"):
            yc = torch.randint(0, ncls, (N,), generator=g)
            if mode == "sorted":
                yc = torch.sort(yc).values
            c = F.normalize(torch.randn(N, 256, generator=g) + clustered * 16 * centers[yc], dim=1)
            c16 = Fn.to_bf16_rows(c, -(-N // 256) * 256)
            diag = torch.arange(A) % N
            loss, st, state = Fn.infonce_tc_forward(a, ya, contrast_bf16=c16, contrast_cls=yc, n_cols=N, diag_col=diag,
                                                    temperature=T, base_temperature=0.07, sorted_cols=(mode == "sorted"))
            cf = P.infonce_closed_form(_bf(a).double(), ya, _bf(c).double(), yc, T, 0.07, self_contrast=False, diag_cols=diag)
        else:
            K, M = max(ncls, 2), rng.randint(1, 40)
            if A > K * 2 * M:
                continue
            ya = torch.randint(0, K, (A,), generator=g)
            ya = ya[torch.argsort(torch.where(ya == 0, K, ya), stable=True)]
            a = F.normalize(torch.randn(A, 256, generator=g) + clustered * 16 * centers[ya], dim=1)
            segq = F.normalize(torch.randn(K, M, 256, generator=g), dim=2)
            pixq = F.normalize(torch.randn(K, M, 256, generator=g), dim=2)
            shadow = torch.empty((shadow_rows(K, M), 256), dtype=torch.bfloat16)
            _abi.check(lib.pcl_bank_shadow_rebuild(segq.data_ptr(), pixq.data_ptr(), K, M, 256, shadow.data_ptr(), None))
            loss, st, state = Fn.infonce_tc_forward(a, ya, bank=(shadow, K, 2 * M), diag_col=torch.arange(A),
                                                    temperature=T, base_temperature=0.07)
            contrast, yc = P.flatten_queue(torch.cat((_bf(segq), _bf(pixq)), 1).double())
            cf = P.infonce_closed_form(_bf(a).double(), ya, contrast, yc.long(), T, 0.07, self_contrast=False)
        dA = Fn.infonce_tc_backward(state, st).double()
        lo = cf["loss"].item()
        if math.isnan(lo):
            if not math.isnan(loss.item()):
                bad.append(f"reference NaN, engine {loss.item()}: {desc}")
            continue
        if not torch.equal(st[4].double(), cf["npos"]):
            bad.append(f"positive counts differ: {desc}")
            continue
        # the gradient reference uses the same bf16-rounded operands (the rounding of the operands is not under test)
        gmax = cf["dA"].abs().max().item()
        gabs = (dA - cf["dA"]).abs().max().item() / max(gmax, 1e-9)
        gfro = ((dA - cf["dA"]).norm() / max(cf["dA"].norm().item(), 1e-9)).item()
        # (a loss that is exactly 0 in real arithmetic — a single class, no negatives — comes out as ~1e-8 of ex2/lg2
        # approximation noise on the tensor path: absolute floor next to the relative bound)
        if abs(loss.item() - lo) > 5e-5 * abs(lo) + 1e-6 or gabs > 6e-3 or gfro > 5e-3:   # (tiny contrast sets average less)
            bad.append(f"mismatch rel={_rel(loss.item(), lo):.2e} gabs={gabs:.2e} gfro={gfro:.2e}: {desc}")
    return bad


def fuzz_graphed_step(seed: int, n: int):
    """GraphedContrastStep's launch sequence (device-side rank draw, optional pre-zeroed scatter-only backward) against the
    eager autograd step over random geometries: replay r must sample, and compute, exactly what eager step r+1 does."""
    from contrastiveseg_b200 import graph_step
    rng = random.Random(seed)
    bad = []
    saved = (graph_step.GraphedContrastStep._capture, graph_step.GraphedContrastStep._fork_zero_fill,
             graph_step.GraphedContrastStep._join_zero_fill)
    graph_step.GraphedContrastStep._capture = lambda self, warmup: None            # no CUDA graphs on a CPU: run eagerly
    graph_step.GraphedContrastStep._fork_zero_fill = lambda self: self._side_branch(0)
    graph_step.GraphedContrastStep._join_zero_fill = lambda self: None
    try:
        for it in range(n):
            B, D, h, w = rng.randint(1, 3), rng.choice([32, 64]), rng.randint(4, 30), rng.randint(4, 30)
            K, ms, mv = rng.randint(2, 9), rng.randint(4, 150), rng.randint(1, 12)
            st, block, mem = rng.choice([1, 2, 4]), rng.choice([2, 4, 8]), rng.random() < 0.4
            norm, overlap, sd = rng.random() < 0.3, rng.random() < 0.5, rng.randint(0, 10 ** 6)
            desc = f"graph seed={seed} it={it} B={B} D={D} {h}x{w} K={K} ms={ms} mv={mv} mem={mem} norm={norm} overlap={overlap}"
            data = make_contrast_batch(B=B, D=D, h=h, w=w, num_classes=K, img_stride=st, block=block, seed=sd)
            bank = make_bank(K, rng.randint(4, 20), D, sd + 1)
            kw = dict(segment_queue=bank["segment_queue"], pixel_queue=bank["pixel_queue"]) if mem else {}
            opts = cs.ContrastOptions(temperature=0.1, base_temperature=0.07, max_samples=ms, max_views=mv, seed=sd % 1000,
                                      num_classes=K, normalize=norm)
            src = data["embed_raw"] if norm else data["embed"]
            step = cs.GraphedContrastStep(src.clone(), data["target"], seg=data["seg"], options=opts,
                                          overlap_zero_fill=overlap, **kw)
            for r in range(2):
                loss, grad = step.replay()
                meta, lv, gv = step.ws.anchor_meta.clone(), loss.clone(), grad.clone()
                Fn._step_counter[0] = r
                e = src.clone().requires_grad_(True)
                l2 = cs.pixel_contrast_loss(e, data["target"], seg=data["seg"], options=opts, **kw)
                ws = Fn.last_workspace(e.device)
                l2.backward()
                same_l = torch.equal(l2.detach(), lv) or (torch.isnan(l2) and torch.isnan(lv))
                ok_g = torch.allclose(e.grad, gv, rtol=3e-6, atol=0, equal_nan=True)
                if not (torch.equal(ws.anchor_meta, meta) and same_l and ok_g):
                    bad.append(f"replay {r} differs from the eager step: {desc}")
                    break
    finally:
        (graph_step.GraphedContrastStep._capture, graph_step.GraphedContrastStep._fork_zero_fill,
         graph_step.GraphedContrastStep._join_zero_fill) = saved
    return bad


def fuzz_trainer_hook(seed: int, n: int):
    """The whole hook of trainer_contrastive.py:209-255 over several iterations with an evolving bank, reference RNG
    stream (rng='torch_cpu', same torch seed on both sides): loss -> enqueue -> backward.  Loss, d/d seg, d/d embed and
    the bank after every iteration against the oracle — in particular the gradient must not see the rows the enqueue
    of the same iteration writes (the reference's autograd holds a copy of the bank; the engine holds the write back)."""
    rng = random.Random(seed)
    bad = []
    names = ("segment_queue", "segment_queue_ptr", "pixel_queue", "pixel_queue_ptr")
    for it in range(n):
        B, D, h, w, K = rng.randint(1, 2), rng.choice([32, 64]), rng.randint(6, 20), rng.randint(6, 20), rng.randint(3, 7)
        st, block, M, Fq = rng.choice([1, 2]), rng.choice([2, 4, 8]), rng.randint(6, 16), rng.randint(1, 5)
        ms, mv, warm, iters, sd = rng.randint(8, 80), rng.randint(1, 6), rng.randint(0, 2), rng.randint(2, 4), rng.randint(0, 10 ** 6)
        T, lw = rng.choice([0.07, 0.1]), 0.1
        desc = f"hook seed={seed} it={it} B={B} D={D} {h}x{w} K={K} stride={st} M={M} F={Fq} ms={ms} mv={mv} warmup={warm} iters={iters}"
        cfg = cs.Configer({"data": {"num_classes": K}, "network": {"stride": st},
                           "loss": {"loss_type": "mem_contrast_ce_loss", "params": {"ce_ignore_index": -1}},
                           "contrast": {"temperature": T, "base_temperature": 0.07, "max_samples": ms, "max_views": mv,
                                        "loss_weight": lw, "use_rmi": False, "use_lovasz": False, "warmup_iters": warm,
                                        "with_memory": True, "memory_size": M, "pixel_update_freq": Fq, "rng": "torch_cpu"}})
        bank = cs.MemoryBank(K, M, D)
        b0 = make_bank(K, M, D, sd)
        for k in names:
            getattr(bank, k).copy_(b0[k])
        ref = [b0[k].clone().double() if "ptr" not in k else b0[k].clone() for k in names]
        hook = cs.ContrastTrainerHook(cfg, bank)
        ok = True
        for step in range(iters):
            data = make_contrast_batch(B=B, D=D, h=h, w=w, num_classes=K, img_stride=st, block=block, seed=sd + step)
            with_embed = step >= warm
            # reference side (float64), torch RNG stream seeded
            torch.manual_seed(sd + step)
            s64, e64 = data["seg"].double().requires_grad_(True), data["embed"].double().requires_grad_(True)
            try:
                lo = P.contrast_ce_loss({"seg": s64, "embed": e64, "segment_queue": ref[0], "pixel_queue": ref[2]},
                                        data["target"], with_embed=with_embed, loss_weight=lw, temperature=T,
                                        base_temperature=0.07, max_samples=ms, max_views=mv, with_memory=True)
                P.dequeue_and_enqueue(data["embed"].double(), data["target"], *ref, network_stride=st, memory_size=M,
                                      pixel_update_freq=Fq)
                lo.backward()
            except (RuntimeError, IndexError, ValueError):
                ok = None                       # degenerate draw (no class qualifies, A > bank columns, ...): skip the case
                break
            # engine side, same stream
            torch.manual_seed(sd + step)
            seg, emb = data["seg"].clone().requires_grad_(True), data["embed"].clone().requires_grad_(True)
            out = {"seg": seg, "embed": emb, "key": emb.detach(), "lb_key": data["target"]}
            loss = hook.loss_step(out, data["target"], iters=step)
            loss.backward()
            if math.isnan(lo.item()):
                if not math.isnan(loss.item()):
                    bad.append(f"reference NaN, engine {loss.item()} at iteration {step}: {desc}")
                ok = None
                break
            ge = (emb.grad.double() - e64.grad).abs().max().item() / max(e64.grad.abs().max().item(), 1e-9)
            gs = (seg.grad.double() - s64.grad).abs().max().item() / max(s64.grad.abs().max().item(), 1e-9)
            eb = max((bank.segment_queue.double() - ref[0]).abs().max().item(), (bank.pixel_queue.double() - ref[2]).abs().max().item())
            ptr_ok = torch.equal(bank.segment_queue_ptr, ref[1]) and torch.equal(bank.pixel_queue_ptr, ref[3])
            if _rel(loss.item(), lo.item()) > 5e-6 or ge > 3e-5 or gs > 3e-5 or eb > 3e-6 or not ptr_ok:
                bad.append(f"iteration {step}: rel={_rel(loss.item(), lo.item()):.1e} d_embed={ge:.1e} d_seg={gs:.1e} bank={eb:.1e} "
                           f"ptr_ok={ptr_ok}: {desc}")
                ok = False
                break
            # fp32 bank rows drift from the float64 reference by rounding only; re-align so the drift cannot accumulate
            ref[0], ref[2] = bank.segment_queue.double().clone(), bank.pixel_queue.double().clone()
    return bad


def fuzz_wrappers(seed: int, n: int):
    """ContrastCELoss / MemContrastCELoss end to end (fused up-sample + CE kernels for the seg half, pixel contrast on the
    reference RNG stream), warm-up and post-warm-up, optional class weights: loss, d/d seg, d/d embed vs the oracle."""
    from contrastiveseg_b200 import loss as loss_mod
    rng = random.Random(seed)
    bad = []
    saved = loss_mod.ContrastCELoss._can_fuse
    loss_mod.ContrastCELoss._can_fuse = lambda self, ce, s: self.fused_seg_ce and ce.ce_loss.reduction == "mean"
    try:
        for it in range(n):
            B, D, h, w, K = rng.randint(1, 2), rng.choice([32, 64]), rng.randint(5, 18), rng.randint(5, 18), rng.randint(2, 8)
            mem, with_embed, weighted = rng.random() < 0.5, rng.random() < 0.7, rng.random() < 0.4
            ms, mv, M, sd = rng.randint(8, 90), rng.randint(1, 8), rng.randint(4, 14), rng.randint(0, 10 ** 6)
            if rng.random() < 0.5:
                st = rng.choice([2, 4])
                himg, wimg = h * st, w * st
            else:
                himg, wimg = rng.randint(h, 3 * h + 2), rng.randint(w, 3 * w + 2)
            T, lw = rng.choice([0.07, 0.1]), rng.choice([0.1, 1.0])
            desc = (f"wrapper seed={seed} it={it} B={B} D={D} {h}x{w}->{himg}x{wimg} K={K} mem={mem} with_embed={with_embed} "
                    f"weighted={weighted} ms={ms} mv={mv}")
            data = make_contrast_batch(B=B, D=D, h=h, w=w, num_classes=K, img_stride=1, block=rng.choice([2, 4, 8]), seed=sd,
                                       himg=himg, wimg=wimg)
            bank = make_bank(K, M, D, sd + 1)
            g = torch.Generator().manual_seed(sd)
            cew = (torch.rand(K, generator=g) + 0.5) if weighted else None
            params = {"ce_ignore_index": -1, "ce_reduction": "elementwise_mean"}
            if weighted:
                params["ce_weight"] = cew.tolist()
            cfg = cs.Configer({"data": {"num_classes": K}, "network": {"stride": 8}, "loss": {"params": params},
                               "contrast": {"temperature": T, "base_temperature": 0.07, "max_samples": ms, "max_views": mv,
                                            "loss_weight": lw, "use_rmi": False, "use_lovasz": False, "rng": "torch_cpu"}})
            crit = (cs.MemContrastCELoss if mem else cs.ContrastCELoss)(cfg)
            extra = {"segment_queue": bank["segment_queue"], "pixel_queue": bank["pixel_queue"]} if mem else {}
            torch.manual_seed(sd)
            s64, e64 = data["seg"].double().requires_grad_(True), data["embed"].double().requires_grad_(True)
            try:
                lo = P.contrast_ce_loss(dict({"seg": s64, "embed": e64}, **{k: v.double() for k, v in extra.items()}),
                                        data["target"], with_embed=with_embed, loss_weight=lw, temperature=T, base_temperature=0.07,
                                        max_samples=ms, max_views=mv, with_memory=mem, ce_weight=cew.double() if weighted else None)
                lo.backward()
            except (RuntimeError, IndexError, ValueError):
                continue
            torch.manual_seed(sd)
            seg, emb = data["seg"].clone().requires_grad_(True), data["embed"].clone().requires_grad_(True)
            loss = crit(dict({"seg": seg, "embed": emb}, **extra), data["target"], with_embed=with_embed)
            loss.backward()
            if math.isnan(lo.item()):
                if not math.isnan(loss.item()):
                    bad.append(f"reference NaN, engine {loss.item()}: {desc}")
                continue
            ge = (emb.grad.double() - e64.grad).abs().max().item() / max(e64.grad.abs().max().item(), 1e-9)
            gs = (seg.grad.double() - s64.grad).abs().max().item() / max(s64.grad.abs().max().item(), 1e-9)
            if _rel(loss.item(), lo.item()) > 5e-6 or ge > 3e-5 or gs > 3e-5:
                bad.append(f"mismatch rel={_rel(loss.item(), lo.item()):.1e} d_embed={ge:.1e} d_seg={gs:.1e}: {desc}")
    finally:
        loss_mod.ContrastCELoss._can_fuse = saved
    return bad
