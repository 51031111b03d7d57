"""Generate golden vectors by running the UNMODIFIED reference (located by oracle.ref_loader.reference_root()).

Run where a reference tree is reachable:  python tests/golden/make_golden.py [aux | random_seeds]
Writes tests/golden/*.npz.  The reference is fp32 PyTorch; every torch.randperm it draws is
recorded so that the engine / the port can replay identical sample indices.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))

from oracle.ref_loader import DictConfiger, load_reference, patched_randperm  # noqa: E402
from oracle.ref_port import PermRecorder  # noqa: E402
from contrastiveseg_b200.synth import make_bank, make_contrast_batch  # noqa: E402

import types  # noqa: E402


def cfg_dict(T, bT, max_samples, max_views, loss_weight=0.1, ignore=-1, with_memory=False, memory_size=0,
             pixel_update_freq=0):
    d = {
        "contrast": {"temperature": T, "base_temperature": bT, "max_samples": max_samples,
                     "max_views": max_views, "loss_weight": loss_weight, "use_rmi": False,
                     "use_lovasz": False, "proj_dim": 256, "stride": 8, "warmup_iters": 0},
        "loss": {"params": {"ce_ignore_index": ignore, "ce_reduction": "elementwise_mean"}},
        "network": {"stride": 8},
    }
    if with_memory:
        d["contrast"].update(with_memory=True, memory_size=memory_size, pixel_update_freq=pixel_update_freq)
    return d


def pack_perms(draws):
    lens = np.array([len(d) for d in draws], dtype=np.int64)
    flat = np.concatenate([d.numpy() for d in draws]) if draws and lens.sum() else np.zeros(0, np.int64)
    return flat.astype(np.int64), lens


def loss_case(name, *, B, D, h, w, K, stride, block, T, bT, max_samples, max_views, seed, mem=None,
              himg=None, wimg=None, boost=2.0):
    ref = load_reference()
    data = make_contrast_batch(B=B, D=D, h=h, w=w, num_classes=K, img_stride=stride, block=block, seed=seed,
                               himg=himg, wimg=wimg, boost=boost)
    cfg = DictConfiger(cfg_dict(T, bT, max_samples, max_views))
    embed = data["embed"].clone().requires_grad_(True)
    predict = data["seg"].argmax(1)
    rec = PermRecorder(torch.Generator().manual_seed(seed + 1))
    captured = {}
    if mem is None:
        crit = ref.nomem.PixelContrastLoss(cfg)
    else:
        crit = ref.mem.PixelContrastLoss(cfg)
    orig = crit._hard_anchor_sampling

    def spy(X, y_hat, y):
        X_, y_ = orig(X, y_hat, y)
        captured["X_"], captured["y_"] = X_.detach().clone(), y_.detach().clone()
        return X_, y_
    crit._hard_anchor_sampling = spy
    queue = None
    extra = {}
    if mem is not None:
        bank = make_bank(K, mem["M"], D, seed + 2)
        queue = torch.cat((bank["segment_queue"], bank["pixel_queue"]), dim=1)
        extra = dict(segment_queue=bank["segment_queue"].numpy(), pixel_queue=bank["pixel_queue"].numpy())
    with patched_randperm(rec):
        if mem is None:
            loss = crit(embed, data["target"], predict)
        else:
            loss = crit(embed, data["target"], predict, queue)
    loss.backward()
    flat, lens = pack_perms(rec.draws)
    out = dict(embed=data["embed"].numpy(), target=data["target"].numpy(), predict=predict.numpy(),
               seg=data["seg"].numpy(), perm_flat=flat, perm_lens=lens, loss=np.float32(loss.item()),
               grad_embed=embed.grad.numpy(), X_=captured["X_"].numpy(), y_=captured["y_"].numpy(),
               params=np.array([T, bT, max_samples, max_views, K, -1], dtype=np.float64), **extra)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(f"{name}: loss={loss.item():.7f} TC={captured['X_'].shape[0]} V={captured['X_'].shape[1]}")


def wrapper_case(name, *, with_embed, mem, seed=11):
    ref = load_reference()
    B, D, h, w, K, stride = 2, 32, 16, 20, 5, 2
    data = make_contrast_batch(B=B, D=D, h=h, w=w, num_classes=K, img_stride=stride, block=4, seed=seed)
    d = cfg_dict(0.1, 0.07, 48, 5, loss_weight=0.1, with_memory=mem, memory_size=10, pixel_update_freq=3)
    cfg = DictConfiger(d)
    seg = data["seg"].clone().requires_grad_(True)
    embed = data["embed"].clone().requires_grad_(True)
    preds = {"seg": seg, "embed": embed}
    extra = {}
    if mem:
        bank = make_bank(K, 10, D, seed + 2)
        preds["segment_queue"], preds["pixel_queue"] = bank["segment_queue"], bank["pixel_queue"]
        extra = dict(segment_queue=bank["segment_queue"].numpy(), pixel_queue=bank["pixel_queue"].numpy())
        crit = ref.mem.ContrastCELoss(cfg)
    else:
        crit = ref.nomem.ContrastCELoss(cfg)
    rec = PermRecorder(torch.Generator().manual_seed(seed + 1))
    with patched_randperm(rec):
        loss = crit(preds, data["target"], with_embed=with_embed)
    loss.backward()
    flat, lens = pack_perms(rec.draws)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), embed=data["embed"].numpy(), seg=data["seg"].numpy(),
                        target=data["target"].numpy(), perm_flat=flat, perm_lens=lens,
                        loss=np.float32(loss.item()), grad_embed=embed.grad.numpy(), grad_seg=seg.grad.numpy(),
                        params=np.array([0.1, 0.07, 48, 5, K, -1, 0.1, float(with_embed), float(mem)]), **extra)
    print(f"{name}: loss={loss.item():.7f}")


def aux_wrapper_case(name, *, with_embed, seed=13, weighted=False):
    """lib/loss/loss_contrast.py:192-234 ContrastAuxCELoss (the class the DeepLab / HRNet-OCR contrast scripts select):
    FSAuxCELoss (lib/loss/loss_helper.py:301-313) on the bilinearly up-sampled [seg_aux, seg] + the pixel-contrast term."""
    ref = load_reference()
    B, D, h, w, K, stride = 2, 32, 13, 17, 6, 4
    data = make_contrast_batch(B=B, D=D, h=h, w=w, num_classes=K, img_stride=stride, block=8, seed=seed)
    d = cfg_dict(0.1, 0.07, 48, 5, loss_weight=0.1)
    d["network"]["loss_weights"] = {"seg_loss": 1.0, "aux_loss": 0.4}
    ce_w = None
    if weighted:
        ce_w = [0.8, 1.1, 0.9, 1.3, 1.0, 0.7]
        d["loss"]["params"]["ce_weight"] = ce_w
    cfg = DictConfiger(d)
    g = torch.Generator().manual_seed(seed + 5)
    seg = data["seg"].clone().requires_grad_(True)
    seg_aux = (data["seg"] * 0.5 + torch.randn(data["seg"].shape, generator=g)).requires_grad_(True)
    embed = data["embed"].clone().requires_grad_(True)
    crit = ref.nomem.ContrastAuxCELoss(cfg)
    rec = PermRecorder(torch.Generator().manual_seed(seed + 1))
    with patched_randperm(rec):
        loss = crit({"seg": seg, "seg_aux": seg_aux, "embed": embed}, data["target"], with_embed=with_embed)
    loss.backward()
    flat, lens = pack_perms(rec.draws)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), embed=data["embed"].numpy(), seg=data["seg"].numpy(),
                        seg_aux=seg_aux.detach().numpy(), target=data["target"].numpy(), perm_flat=flat, perm_lens=lens,
                        loss=np.float32(loss.item()), grad_embed=embed.grad.numpy(), grad_seg=seg.grad.numpy(),
                        grad_seg_aux=seg_aux.grad.numpy(),
                        ce_weight=np.array(ce_w if ce_w else [], dtype=np.float32),
                        params=np.array([0.1, 0.07, 48, 5, K, -1, 0.1, float(with_embed), 1.0, 0.4]))
    print(f"{name}: loss={loss.item():.7f}")


def enqueue_case(name, *, B, D, h, w, K, img_stride, net_stride, M, Fq, steps, seed):
    ref = load_reference()
    bank = make_bank(K, M, D, seed + 2)
    sq, sp, pq, pp = (bank["segment_queue"].clone(), bank["segment_queue_ptr"].clone(),
                      bank["pixel_queue"].clone(), bank["pixel_queue_ptr"].clone())
    me = types.SimpleNamespace(network_stride=net_stride, memory_size=M, pixel_update_freq=Fq)
    out = dict(sq0=sq.numpy().copy(), pq0=pq.numpy().copy(),
               params=np.array([net_stride, M, Fq, steps, K], dtype=np.int64))
    for s in range(steps):
        data = make_contrast_batch(B=B, D=D, h=h, w=w, num_classes=K, img_stride=img_stride, block=4 * img_stride,
                                   seed=seed + 10 * s)
        rec = PermRecorder(torch.Generator().manual_seed(seed + 100 + s))
        with patched_randperm(rec):
            ref.enqueue(me, data["embed"], data["target"], sq, sp, pq, pp)
        flat, lens = pack_perms(rec.draws)
        out[f"keys{s}"] = data["embed"].numpy()
        out[f"labels{s}"] = data["target"].numpy()
        out[f"perm_flat{s}"], out[f"perm_lens{s}"] = flat, lens
        out[f"sq{s + 1}"], out[f"pq{s + 1}"] = sq.numpy().copy(), pq.numpy().copy()
        out[f"sp{s + 1}"], out[f"pp{s + 1}"] = sp.numpy().copy(), pp.numpy().copy()
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(f"{name}: steps={steps} final seg ptr={sp.tolist()} pix ptr={pp.tolist()}")


def input_sums(*tensors):
    """float64 sums of the inputs a case regenerates from contrastiveseg_b200.synth: a golden made from other data fails
    loudly instead of comparing unrelated numbers."""
    return np.array([t.double().sum().item() for t in tensors], dtype=np.float64)


def random_seeds_case(name="random_seeds"):
    """Reference outputs for tests/test_oracle_vs_reference.py: the loss on synth seeds 31-33 with and without the bank,
    and five enqueue steps.  Only outputs and recorded permutations are stored; the tests regenerate the inputs."""
    ref = load_reference()
    out = {}
    for seed in (31, 32, 33):
        K, D = 6, 32
        data = make_contrast_batch(B=3, D=D, h=20, w=24, num_classes=K, img_stride=2, block=6, seed=seed, boost=1.5)
        predict = data["seg"].argmax(1)
        for mem in (False, True):
            cfg = DictConfiger(cfg_dict(0.1, 0.07, 50, 7))
            key = f"s{seed}_mem{int(mem)}_"
            sums = [data["embed"], data["target"], predict]
            queue = None
            if mem:
                bank = make_bank(K, 15, D, seed)
                queue = torch.cat((bank["segment_queue"], bank["pixel_queue"]), 1)
                sums.append(queue)
            rec = PermRecorder(torch.Generator().manual_seed(seed))
            embed = data["embed"].clone().requires_grad_(True)
            crit = (ref.mem if mem else ref.nomem).PixelContrastLoss(cfg)
            with patched_randperm(rec):
                loss = crit(embed, data["target"], predict, queue) if mem else crit(embed, data["target"], predict)
            loss.backward()
            out[key + "perm_flat"], out[key + "perm_lens"] = pack_perms(rec.draws)
            out[key + "loss"] = np.float64(loss.item())
            out[key + "grad_embed"] = embed.grad.numpy()
            out[key + "input_sums"] = input_sums(*sums)
    K, D, M, Fq = 5, 16, 6, 4
    bank = make_bank(K, M, D, 3)
    state = [bank[k].clone() for k in ("segment_queue", "segment_queue_ptr", "pixel_queue", "pixel_queue_ptr")]
    me = types.SimpleNamespace(network_stride=2, memory_size=M, pixel_update_freq=Fq)
    out["enq_input_sums"] = input_sums(*state)
    for s in range(5):
        data = make_contrast_batch(B=2, D=D, h=12, w=12, num_classes=K, img_stride=2, block=6, seed=50 + s)
        rec = PermRecorder(torch.Generator().manual_seed(s))
        with patched_randperm(rec):
            ref.enqueue(me, data["embed"], data["target"], *state)
        out[f"enq{s}_perm_flat"], out[f"enq{s}_perm_lens"] = pack_perms(rec.draws)
        out[f"enq{s}_input_sums"] = input_sums(data["embed"], data["target"])
        for k, t in zip(("sq", "sp", "pq", "pp"), state):
            out[f"enq{s}_{k}"] = t.numpy().copy()
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(f"{name}: " + " ".join(f"{k[:-4]}={v:.7f}" for k, v in out.items() if k.endswith("loss")))


if __name__ == "__main__":
    only = sys.argv[1:]
    if only == ["aux"]:              # add the round-2 cases without touching the committed round-1 files
        torch.manual_seed(0)
        aux_wrapper_case("wrapper_aux_embed", with_embed=True)
        aux_wrapper_case("wrapper_aux_warmup_weighted", with_embed=False, weighted=True)
        sys.exit(0)
    if only == ["random_seeds"]:
        random_seeds_case()
        sys.exit(0)
    torch.manual_seed(0)
    loss_case("nomem_small", B=2, D=32, h=24, w=24, K=5, stride=2, block=8, T=0.1, bT=0.07,
              max_samples=40, max_views=6, seed=1)
    loss_case("nomem_oddv", B=3, D=32, h=20, w=28, K=6, stride=2, block=8, T=0.07, bT=0.07,
              max_samples=64, max_views=5, seed=2)
    loss_case("nomem_mv1", B=2, D=32, h=16, w=16, K=4, stride=4, block=16, T=0.1, bT=0.07,
              max_samples=32, max_views=1, seed=3)
    loss_case("nomem_nondiv", B=2, D=32, h=13, w=10, K=4, stride=4, block=10, T=0.1, bT=0.07,
              max_samples=24, max_views=4, seed=4, himg=50, wimg=37)
    loss_case("nomem_d256", B=2, D=256, h=16, w=32, K=7, stride=4, block=16, T=0.1, bT=0.07,
              max_samples=128, max_views=10, seed=5)
    loss_case("mem_small", B=2, D=32, h=24, w=24, K=5, stride=2, block=8, T=0.07, bT=0.07,
              max_samples=40, max_views=6, seed=6, mem=dict(M=12))
    loss_case("mem_d256", B=2, D=256, h=16, w=32, K=7, stride=4, block=16, T=0.07, bT=0.07,
              max_samples=128, max_views=10, seed=7, mem=dict(M=40))
    wrapper_case("wrapper_nomem_embed", with_embed=True, mem=False)
    wrapper_case("wrapper_nomem_warmup", with_embed=False, mem=False)
    wrapper_case("wrapper_mem_embed", with_embed=True, mem=True)
    aux_wrapper_case("wrapper_aux_embed", with_embed=True)
    aux_wrapper_case("wrapper_aux_warmup_weighted", with_embed=False, weighted=True)
    enqueue_case("enqueue_aligned", B=2, D=32, h=16, w=16, K=5, img_stride=2, net_stride=2, M=7, Fq=3,
                 steps=6, seed=21)
    enqueue_case("enqueue_q6", B=2, D=32, h=16, w=16, K=5, img_stride=2, net_stride=4, M=9, Fq=4,
                 steps=4, seed=22)
    random_seeds_case()
