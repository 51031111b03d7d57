#!/usr/bin/env python
"""bench.py — contrast-loss fwd+bwd throughput on synthetic Cityscapes-shaped batches (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl engine|reference] [--workload s1|s2]
                    [--dump-outputs DIR]

Workload s1 = BASELINE configs[1]: HRNet-W48 pixel-contrast (no bank), 1024x512 input -> 256x128 embedding,
19 classes, batch 8 PER GPU (weak scaling; the no-bank loss has no cross-rank exchange, SURVEY §8e).
Workload s2 = configs[2] shape per rank (bank 19x(5000+5000)x256, one image per rank, bank merge allgather).
A "step" = one pass of the hot path over one batch: label/argmax/key scan, anchor selection + gather, InfoNCE
forward, InfoNCE backward and the dense embedding-gradient write (+ bank enqueue for s2).
Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

S1 = dict(B=8, D=256, h=128, w=256, K=19, stride=4, block=32, T=0.1, bT=0.07, max_samples=1024, max_views=100)
S2 = dict(B=1, D=256, h=128, w=256, K=19, stride=4, block=32, T=0.07, bT=0.07, max_samples=1024, max_views=100,
          M=5000, F=10, net_stride=4)
# BASELINE configs[3] (SURVEY §8 C4/S3), opt-in: ResNet-101 DeepLab-V3 + region memory on COCO-Stuff 520x520, 171 classes,
# 2 images per rank; the dilated-8 backbone yields a 66x66 embedding (nearest label index floor(dst*520/66), not ::8) and
# the bank's labels[:, ::8, ::8] grid (65x65) is flat-index-misaligned with the 4356 feature columns (Q6)
S3 = dict(B=2, D=256, h=66, w=66, K=171, stride=8, block=40, himg=520, wimg=520, T=0.07, bT=0.07, max_samples=1024,
          max_views=100, M=5000, F=10, net_stride=8)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"],
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture
    (profiles/ncu_traffic.json, written by tools/ncu_traffic.py from a .ncu-rep); None if not captured."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None
    return json.load(open(p)).get(kernel, {}).get("dram_bytes")


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return
        time.sleep(0.12)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        self.lines = [l for l in out.splitlines() if l.strip()]

    def summary(self):
        sm, smax, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax = max(smax, float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": smax or None, "reasons": sorted(reasons), "samples": len(sm)}


def pin_to_gpu_local_cpus(dev_index: int):
    """Multi-rank runs: bind this process to the CPUs NVML reports as local to its GPU (NUMA-aware launch path; the
    step is host-launch-bound, and ranks scheduled on the far socket launched ~45 % slower at N=8).  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(dev_index).uuid)
        h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        ncpu = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [i for i in range(ncpu) if (mask[i // 64] >> (i % 64)) & 1]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def make_inputs(cfg, seed, device=None, bank=False):
    from contrastiveseg_b200.synth import make_bank, make_contrast_batch
    d = make_contrast_batch(B=cfg["B"], D=cfg["D"], h=cfg["h"], w=cfg["w"], num_classes=cfg["K"],
                            img_stride=cfg["stride"], block=cfg["block"], seed=seed, himg=cfg.get("himg"),
                            wimg=cfg.get("wimg"))
    out = dict(embed=d["embed"], seg=d["seg"], target=d["target"])
    if bank:
        out.update(make_bank(cfg["K"], cfg["M"], cfg["D"], seed + 1000))
    if device is not None:
        out = {k: v.to(device) for k, v in out.items()}
    return out


def engine_configer(cfg, bank=False, precision="bf16"):
    import contrastiveseg_b200 as cs
    d = {"data": {"num_classes": cfg["K"]}, "network": {"stride": cfg.get("net_stride", 4)},
         "loss": {"params": {"ce_ignore_index": -1, "ce_reduction": "elementwise_mean"}},
         "contrast": {"temperature": cfg["T"], "base_temperature": cfg["bT"], "max_samples": cfg["max_samples"],
                      "max_views": cfg["max_views"], "loss_weight": 0.1, "use_rmi": False, "rng": "device",
                      "precision": precision}}
    if bank:
        # bank sweeps run on the tcgen05 path (bf16 operands through the bank shadow)
        d["contrast"].update(with_memory=True, memory_size=cfg["M"], pixel_update_freq=cfg["F"])
    return cs.Configer(d)


# ---------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on the host cores (the reference is Python and cannot
# travel to the GPU box; oracle/ref_port.py restates it op for op and is pinned to it by golden vectors)
# ---------------------------------------------------------------------------------------------------
def cpu_port_step(inp, cfg, bank=False):
    from oracle import ref_port as P
    embed = inp["embed"].clone().requires_grad_(True)
    predict = inp["seg"].argmax(1)
    queue = torch.cat((inp["segment_queue"], inp["pixel_queue"]), 1) if bank else None
    loss = P.pixel_contrast_loss(embed, inp["target"], predict, temperature=cfg["T"], base_temperature=cfg["bT"],
                                 max_samples=cfg["max_samples"], max_views=cfg["max_views"], queue=queue,
                                 per_pair_gather=True)
    loss.backward()
    if bank:
        P.dequeue_and_enqueue(inp["embed"], inp["target"], inp["segment_queue"], inp["segment_queue_ptr"],
                              inp["pixel_queue"], inp["pixel_queue_ptr"], network_stride=cfg["net_stride"],
                              memory_size=cfg["M"], pixel_update_freq=cfg["F"])
    return float(loss.item())


def calibrate_cpu(cfg, bank):
    """Pick the host thread count that runs the port fastest (torch CPU ops stop scaling well before 128 threads)
    and time one single-image step with it."""
    cores = os.cpu_count() or 1
    c1 = dict(cfg); c1["B"] = 1
    inp = make_inputs(c1, 304, None, bank)
    best = (None, float("inf"))
    for th in sorted({min(cores, t) for t in (8, 16, 32, 64, cores)}):
        torch.set_num_threads(th)
        cpu_port_step(inp, c1, bank)
        t0 = time.perf_counter()
        cpu_port_step(inp, c1, bank)
        dt = time.perf_counter() - t0
        if dt < best[1]:
            best = (th, dt)
    torch.set_num_threads(best[0])
    return best


_REF_CACHE = {}


def real_reference_step(inp, cfg, bank):
    """The UNMODIFIED reference modules (lib/loss/loss_contrast*.py, Trainer._dequeue_and_enqueue) when a reference tree
    is reachable ($CSEG_REF, /root/reference, baseline/_ref): never the case on a stock GPU box, where the port runs."""
    from oracle import ref_loader as RL
    import types
    key = (bank, cfg["T"], cfg["bT"], cfg["max_samples"], cfg["max_views"])
    if key not in _REF_CACHE:
        ref = RL.load_reference()
        d = {"contrast": {"temperature": cfg["T"], "base_temperature": cfg["bT"], "max_samples": cfg["max_samples"],
                          "max_views": cfg["max_views"], "loss_weight": 0.1, "use_rmi": False, "use_lovasz": False},
             "loss": {"params": {"ce_ignore_index": -1, "ce_reduction": "elementwise_mean"}}, "network": {"stride": cfg.get("net_stride", 4)}}
        mod = (ref.mem if bank else ref.nomem).PixelContrastLoss(RL.DictConfiger(d))
        _REF_CACHE[key] = (ref, mod)
    ref, mod = _REF_CACHE[key]
    embed = inp["embed"].clone().requires_grad_(True)
    predict = inp["seg"].argmax(1)
    if bank:
        queue = torch.cat((inp["segment_queue"], inp["pixel_queue"]), 1)
        loss = mod(embed, inp["target"], predict, queue)
    else:
        loss = mod(embed, inp["target"], predict)
    loss.backward()
    if bank:
        me = types.SimpleNamespace(network_stride=cfg["net_stride"], memory_size=cfg["M"], pixel_update_freq=cfg["F"])
        ref.enqueue(me, inp["embed"], inp["target"], inp["segment_queue"], inp["segment_queue_ptr"], inp["pixel_queue"],
                    inp["pixel_queue_ptr"])
    return float(loss.item())


def reference_kind():
    try:
        from oracle import ref_loader as RL
        if RL.reference_root() is not None:
            RL.load_reference()
            return "reference"
    except Exception:                                    # noqa: BLE001
        pass
    return "port"


def run_reference(args, cfg, bank, rank):
    """Reference arm: the reference's own CPU path on the box's host cores, SAME config as the engine arm (full batch).
    The reference is Python and does not travel to the GPU box, so there it is the op-for-op port (oracle/ref_port.py,
    pinned to the reference by golden vectors); where a reference tree is reachable the unmodified modules run."""
    if rank != 0:
        return None
    kind = reference_kind()
    step = real_reference_step if kind == "reference" else cpu_port_step
    threads, t1 = calibrate_cpu(cfg, bank)
    inp = make_inputs(cfg, 304, None, bank)
    # Bounded run: one probe step at the full batch (it doubles as the first warm-up step); if --steps/--warmup of those
    # would take longer than REF_BUDGET_S, every step becomes a smaller sample of the same workload (fewer images of the
    # batch: the reference's backward is super-linear in the batch, one dense (B,HW,D) SelectBackward per (image, class)).
    full_b, cfg_full = cfg["B"], cfg
    tp = time.perf_counter()
    step(inp, cfg, bank)
    probe = time.perf_counter() - tp
    n_total = args.steps + max(args.warmup - 1, 0)
    budget = float(os.environ.get("PCL_BENCH_REF_BUDGET_S", "400"))
    if probe * n_total > budget and full_b > 1:
        b_s = full_b
        while b_s > 1 and probe * (b_s / full_b) ** 1.5 * n_total > budget:
            b_s //= 2
        cfg = dict(cfg, B=b_s)
        inp = make_inputs(cfg, 304, None, bank)
    for _ in range(max(args.warmup - 1, 0)):
        step(inp, cfg, bank)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step(inp, cfg, bank)
    dt = time.perf_counter() - t0
    ms = dt / args.steps * 1e3
    val = cfg["B"] * args.steps / dt
    what = (f"the full workload (batch {full_b})" if cfg["B"] == full_b else
            f"a {cfg['B']}-image sample of the batch of {full_b} (a full-batch step takes {probe:.1f} s here)")
    sample = (f"{args.steps} steps of {what} after {args.warmup} warm-up on {threads} of "
              f"{os.cpu_count()} host threads (fastest of 8/16/32/64/all, calibrated on one image), fp32 torch CPU, "
              + ("the unmodified reference modules" if kind == "reference" else
                 "per-(image,class) gather + autograd backward like the reference (oracle/ref_port.py)"))
    return {"impl": "reference", "metric": "contrast-loss fwd+bwd throughput", "value": val, "unit": "images/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(cfg_full, bank),
            "cpu_baseline": {"value": val, "unit": "images/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def workload_config(cfg, bank, B=None):
    name = ("HRNet-W48 pixel-contrast + pixel/region memory bank" if bank else "HRNet-W48 pixel-contrast (no memory bank)")
    data = "synthetic Cityscapes 1024x512 19-class"
    if cfg["K"] == 171:
        name, data = "ResNet-101 DeepLab-V3 pixel-contrast + region memory", "synthetic COCO-Stuff 520x520 171-class"
    return {"workload": f"{name}, {data} -> embed {cfg['D']}x{cfg['h']}x{cfg['w']}, "
                        f"batch {B or cfg['B']} per GPU, max_samples {cfg['max_samples']}, max_views {cfg['max_views']}",
            "per_gpu_batch": B or cfg["B"], "parallelism": "dp (images sharded, no data-path collective)" if not bank
            else "dp + one NCCL all_gather of the bank enqueue packet per step"}


# ---------------------------------------------------------------------------------------------------
# engine arm
# ---------------------------------------------------------------------------------------------------
def stage_timings(cfg, inp, dev, precision, iters=20):
    """CUDA-event time of every C-ABI stage on the launching stream (dominant-kernel roofline)."""
    import ctypes as C
    from contrastiveseg_b200 import _abi, functional as Fn
    lib = _abi.load()
    geom = _abi.Geom(cfg["B"], cfg["D"], cfg["h"], cfg["w"], inp["target"].shape[1], inp["target"].shape[2], cfg["K"],
                     cfg["max_samples"], cfg["max_views"], -1)
    ws = Fn.ContrastWorkspace(dev, geom, 0, 0, 0, 0)
    d = ws.desc
    d.embed, d.labels, d.seg = inp["embed"].data_ptr(), inp["target"].data_ptr(), inp["seg"].data_ptr()
    d.temperature, d.base_temperature, d.seed = cfg["T"], cfg["bT"], 12345
    grad = torch.empty_like(inp["embed"])
    d.grad_embed = grad.data_ptr()
    stream = torch.cuda.current_stream(dev).cuda_stream
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    sw = _abi.SweepDesc()
    ms_ = cfg["max_samples"]
    sw.anchors, sw.anchor_cls = ws.anchors_f32.data_ptr(), ws.anchor_meta.data_ptr() + 8 * ms_
    sw.diag_col, sw.plan = ws.anchor_meta.data_ptr() + 12 * ms_, ws.plan.data_ptr()
    sw.a_rows, sw.D, sw.mode = ms_, cfg["D"], 0
    sw.temperature, sw.base_temperature = cfg["T"], cfg["bT"]
    td = _abi.TcDesc()
    td.anchors_bf16, td.anchor_cls = ws.anchors_bf16.data_ptr(), sw.anchor_cls
    td.diag_col, td.plan, td.a_rows, td.D, td.mode = sw.diag_col, sw.plan, ms_, cfg["D"], 0
    td.contrast_norm_bound, td.temperature, td.base_temperature = 1.0, cfg["T"], cfg["bT"]
    g = C.byref(geom)
    if precision == "bf16":
        fwd = lambda: lib.pcl_infonce_tc_fwd(C.byref(td), d.row_m2, d.partials, d.rowstats, d.loss, stream)
        bwd = lambda: lib.pcl_infonce_tc_bwd(C.byref(td), d.row_m2, d.rowstats, None, d.dpartials, d.dA, stream)
    else:
        fwd = lambda: lib.pcl_infonce_fwd(C.byref(sw), d.partials, d.rowstats, d.loss, stream)
        bwd = lambda: lib.pcl_infonce_bwd(C.byref(sw), d.rowstats, None, d.dpartials, d.dA, stream)
    stages = {
        "class_stats": lambda: lib.pcl_class_stats(g, d.labels, d.seg, None, d.keys, d.chunk_pref, d.counts, stream),
        "plan_anchors": lambda: lib.pcl_plan_anchors(g, d.counts, d.plan, stream),
        "select_gather": lambda: lib.pcl_select_gather(g, d.embed, d.keys, d.chunk_pref, d.plan, None, 12345, 0,
                                                       d.anchor_meta, d.anchors_f32, d.anchors_bf16, d.inv_norm,
                                                       d.norm_max, stream),
        "infonce_fwd": fwd,
        "infonce_bwd": bwd,
        "scatter_grad": lambda: lib.pcl_scatter_grad(g, d.plan, d.anchor_meta, d.dA, d.anchors_f32, d.inv_norm, 0,
                                                     d.grad_embed, stream),
    }
    out = {}
    acc = {k: 0.0 for k in stages}
    for it in range(iters + 2):
        flush.zero_()
        for name, fn in stages.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            st = fn()
            e1.record()
            _abi.check(st, name)
            torch.cuda.synchronize(dev)
            if it >= 2:
                acc[name] += e0.elapsed_time(e1)
    for k in acc:
        out[k] = acc[k] / iters
    A = int(ws.plan[2].item())
    return out, A


def train_iter_bench(cfg, inp, dev, precision, iters=10):
    """BASELINE.json's second figure, "train iters/sec": one synthetic training iteration = producer fwd -> ContrastCELoss
    (fused seg CE + pixel contrast) -> backward -> SGD step.  The reference's HRNet-W48 cannot travel to the GPU box and
    is outside the hot-path scope, so the producer is a stand-in with the same output contract and tensor sizes
    (lib/models/nets/hrnet.py:76-95: 720-channel stride-4 features -> 19-class head + 720->720->256 projection head
    with the engine's L2-normalise): the number shows the loss step's share of an iteration, not HRNet's speed."""
    import torch.nn as nn
    import contrastiveseg_b200 as cs

    class StandIn(nn.Module):
        def __init__(self, K, D, C=720):
            super().__init__()
            self.body = nn.Sequential(nn.Conv2d(3, 64, 3, 2, 1), nn.BatchNorm2d(64), nn.ReLU(inplace=True),
                                      nn.Conv2d(64, C, 3, 2, 1), nn.BatchNorm2d(C), nn.ReLU(inplace=True))
            self.cls = nn.Conv2d(C, K, 1)
            self.proj = cs.ProjectionHead(C, D, proj="convmlp", bn_type="torchbn")

        def forward(self, x):
            f = self.body(x)
            return {"seg": self.cls(f), "embed": self.proj(f)}

    torch.manual_seed(304)
    net = StandIn(cfg["K"], cfg["D"]).to(dev)
    opt = torch.optim.SGD(net.parameters(), lr=0.01, momentum=0.9, weight_decay=5e-4)
    crit = cs.ContrastCELoss(engine_configer(cfg, False, precision)).to(dev)
    H, W = inp["target"].shape[1], inp["target"].shape[2]
    x = torch.randn(cfg["B"], 3, H, W, device=dev)

    def it():
        out = net(x)
        loss = crit(out, inp["target"], with_embed=True)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        return loss
    for _ in range(3):
        it()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(iters):
        loss = it()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / iters
    ok = bool(torch.isfinite(loss).item())
    # The same iteration with the REFERENCE's loss step in place of the engine's (SURVEY 8(d): "the reference ATen path
    # on the B200 itself"): the CPU port's torch ops follow their input's device, so on CUDA tensors they are the
    # reference's own op sequence (per-(image, class) nonzero/randperm/index loop, dense A x N temporaries, one
    # SelectBackward per pair).  A baseline leg like cpu_baseline: measured beside the engine, never part of it.
    ref_ms, ref_err = None, None
    try:
        from oracle import ref_port as P
        kw = dict(with_embed=True, loss_weight=0.1, temperature=cfg["T"], base_temperature=cfg["bT"],
                  max_samples=cfg["max_samples"], max_views=cfg["max_views"], ignore_label=-1)

        def it_ref():
            out = net(x)
            l = P.contrast_ce_loss(out, inp["target"], **kw)
            opt.zero_grad(set_to_none=True)
            l.backward()
            opt.step()
            return l
        for _ in range(2):
            it_ref()
        n_ref = max(3, iters // 2)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(n_ref):
            it_ref()
        e1.record()
        torch.cuda.synchronize(dev)
        ref_ms = e0.elapsed_time(e1) / n_ref
    except Exception as exc:                              # noqa: BLE001
        ref_err = f"{type(exc).__name__}: {exc}"[:200]
    del net, opt, x
    torch.cuda.empty_cache()
    ref_block = ({"ms_per_iter": ref_ms, "iters_per_s": 1e3 / ref_ms, "speedup_of_the_iteration": ref_ms / ms,
                  "what": "same producer, optimiser and batch; loss step = the reference's op sequence (oracle port's "
                          "torch ops on CUDA tensors: ATen kernels, host loop with device syncs), fp32"}
                 if ref_ms else {"error": ref_err})
    return {"iters_per_s": 1e3 / ms, "ms_per_iter": ms, "global_batch": cfg["B"], "finite_loss": ok,
            "with_reference_loss_step": ref_block,
            "producer": "stand-in conv stem -> 720ch stride-4 features -> 19-class head + 720-720-256 projection head "
                        "(engine L2-normalise); fp32, SGD momentum 0.9; not HRNet-W48",
            "loss": "ContrastCELoss (fused seg CE + pixel contrast, with_embed=True)"}


# ---------------------------------------------------------------------------------------------------
# engine arm: every workload is measured through the public graphed-step API (GraphedContrastStep): ONE CUDA-graph replay
# per step (bank steps on several ranks: two replays around the NCCL all_gather of the enqueue packet).
# ---------------------------------------------------------------------------------------------------
L2_BYTES = 126 << 20


def working_set_bytes(cfg, bank):
    hw = cfg["h"] * cfg["w"]
    himg, wimg = cfg.get("himg") or cfg["h"] * cfg["stride"], cfg.get("wimg") or cfg["w"] * cfg["stride"]
    ws = cfg["B"] * (2 * cfg["D"] * hw * 4 + cfg["K"] * hw * 4 + himg * wimg * 8)
    if bank:
        ws += (cfg["K"] - 1) * 2 * cfg["M"] * cfg["D"] * 2          # the bf16 shadow the sweeps stream
    return ws


def rotation_sets(cfg, bank):
    """Timing rule: inputs larger than L2, or flush.  A step's working set (embed + dense gradient + seg + labels
    [+ bank shadow]) above ~1.2x L2 needs nothing; below that the bench rotates over R independent input/gradient
    buffer sets (R x working set > 2.2 x L2), so no timed step finds its inputs in L2 and no flush sits in the timed
    region."""
    ws = working_set_bytes(cfg, bank)
    if ws >= 1.2 * L2_BYTES:
        return 1
    return max(2, min(8, -(-int(2.2 * L2_BYTES) // ws)))


DUMP_GRAD_BYTES = 48 << 20          # keeps a --dump-outputs directory under 64 MB


def output_sample(loss, grad):
    """Host copy of one step's outputs for --dump-outputs.  The dense gradient (268 MB at the s1 shape) is cut down to a
    fixed, seeded subset of its D channels at every pixel, so every sampled anchor column still shows up; a gradient that
    fits the budget is kept whole.  grad_embed_channels lists the channels kept."""
    B, D, h, w = grad.shape
    keep = max(1, min(D, DUMP_GRAD_BYTES // (B * h * w * 4)))
    ch = torch.arange(D) if keep == D else torch.randperm(D, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    g = grad.detach().index_select(1, ch.to(grad.device)).float().cpu()
    return {"loss": np.float32(loss.item()), "grad_embed": g.numpy(),
            "grad_embed_channels": ch.double().numpy()}


def write_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


class Workload:
    """One measured workload: R rotating input sets, one GraphedContrastStep per set (bank steps share the bank)."""

    def __init__(self, args, name, cfg, bank, rank, world, dev, sparse_reset=False):
        import contrastiveseg_b200 as cs
        self.sparse_reset = sparse_reset
        self.args, self.name, self.cfg, self.bank, self.rank, self.world, self.dev = args, name, cfg, bank, rank, world, dev
        self.R = 1 if os.environ.get("PCL_BENCH_TINY") else rotation_sets(cfg, bank)
        self.host = [make_inputs(cfg, 304 + rank + 1000 * r, None, bank) for r in range(self.R)]
        self.inp = [{k: v.to(dev) for k, v in h.items() if k in ("embed", "seg", "target")} for h in self.host]
        self.crit = cs.PixelContrastLoss(engine_configer(cfg, bank, args.precision))
        self.mbank = None
        if bank:
            self.mbank = cs.MemoryBank(cfg["K"], cfg["M"], cfg["D"], with_shadow=(args.precision == "bf16")).to(dev)
            self.mbank.segment_queue.copy_(self.host[0]["segment_queue"]); self.mbank.pixel_queue.copy_(self.host[0]["pixel_queue"])
            if args.precision == "bf16":
                self.mbank.sync_shadow()
        self.steps = []
        self.graph_error = None
        opts = self.crit.options()
        opts.num_classes = cfg["K"]
        try:
            for r in range(self.R):
                kw = {}
                if bank:
                    kw = dict(segment_queue=self.mbank.segment_queue, pixel_queue=self.mbank.pixel_queue,
                              bank_shadow=self.mbank.shadow,
                              enqueue=dict(bank=self.mbank, network_stride=cfg["net_stride"], pixel_update_freq=cfg["F"]))
                self.steps.append(cs.GraphedContrastStep(self.inp[r]["embed"], self.inp[r]["target"], seg=self.inp[r]["seg"],
                                                         options=opts, capture=not args.no_graph,
                                                         sparse_reset=self.sparse_reset, **kw))
        except Exception as exc:                                   # noqa: BLE001  (never lose the whole line)
            self.graph_error = f"{type(exc).__name__}: {exc}"[:300]
            self.steps = []

    # ---- the step, two ways ----
    def replay(self, i):
        return self.steps[i % self.R].replay()[0]

    def eager(self, i):
        inp = self.inp[i % self.R]
        e = inp["embed"].detach().requires_grad_(True)
        queue = (self.mbank.segment_queue, self.mbank.pixel_queue) if self.bank else None
        loss = self.crit(e, inp["target"], seg=inp["seg"], queue=queue, bank_shadow=self.mbank.shadow if self.bank else None)
        if self.bank:
            self.mbank.enqueue(e.detach(), inp["target"], network_stride=self.cfg["net_stride"], pixel_update_freq=self.cfg["F"])
        loss.backward()
        self.eager_out = (loss.detach(), e.grad)
        return loss

    def step_outputs(self, i):
        """What step i handed its caller: (loss, d loss/d embed).  Graph steps keep them in static buffers until the
        same step object replays again."""
        if self.steps:
            st = self.steps[i % self.R]
            return st.loss, st.grad
        return self.eager_out

    def barrier(self):
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(self.dev)

    def reduce_max(self, values):
        t = torch.tensor(values, dtype=torch.float64, device=self.dev)
        if self.world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def time_loop(self, fn, steps, warmup, sampler=None, after_timed=None):
        """K steps bracketed by barrier + synchronize, CUDA events on the launching stream, max over ranks.
        after_timed(K - 1) runs once the timed steps have finished, before any further step.
        Returns (device ms per step, host enqueue ms per step, clock window description)."""
        for i in range(max(warmup, 3)):
            fn(i)
        self.barrier()
        if sampler is not None and self.rank == 0:
            sampler.start()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        self.barrier()
        t0 = time.perf_counter()
        ev[0].record()
        for i in range(steps):
            fn(i)
        ev[1].record()
        t_host = time.perf_counter() - t0               # host time to enqueue the K steps (no sync inside)
        self.barrier()
        if after_timed is not None:
            after_timed(steps - 1)
        window = "timed region"
        if sampler is not None:
            # nvidia-smi samples every 200 ms; a short timed region would see no sample, so the SAME loop keeps running
            # (untimed) until the sampler has covered >= 0.9 s under load
            while time.perf_counter() - t0 < 0.9:
                window = "timed region + untimed continuation of the same step loop to 0.9 s"
                for i in range(50):
                    fn(i)
                torch.cuda.synchronize(self.dev)
            if self.rank == 0:
                sampler.stop()
        ms, host = self.reduce_max([ev[0].elapsed_time(ev[1]) / steps, t_host / steps * 1e3])
        return ms, host, window

    def e2e(self, fn, steps):
        """Same step with HOST inputs: pinned embed/seg/target copied H2D every step, loss read back (D2H)."""
        pin = [{k: h[k].pin_memory() for k in ("embed", "seg", "target")} for h in self.host]
        h2d = sum(pin[0][k].numel() * pin[0][k].element_size() for k in pin[0])

        def one(i):
            r = i % self.R
            for k in pin[r]:
                self.inp[r][k].copy_(pin[r][k], non_blocking=True)
            return fn(i).item()
        for i in range(3):
            one(i)
        self.barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            one(i)
        self.barrier()
        (dt,) = self.reduce_max([time.perf_counter() - t0])
        return self.world * self.cfg["B"] * steps / dt, h2d

    def graph_timeline(self, reps=20):
        """Per-kernel times INSIDE the captured step (fused path): %globaltimer stamps the kernels write into the step's
        sync buffer when its word 7 is set (csrc/pcl_common.cuh) — min block start / max block end per kernel, averaged
        over `reps` replays after the timed region.  The only way to see the kernels of one graph replay as they overlap
        (CUDA events cannot be recorded inside a replay; ncu serialises the nodes)."""
        st = self.steps[0] if self.steps else None
        if st is None or not getattr(st, "fused", False):
            return None
        sync = st.ws.sync
        names = ["k_keys (scan + totals + plan)", "k_select", "k_self_fused", "k_scatter_reduce", "k_fill_zero_excl"]
        acc = {n: [0.0, 0.0, 0.0] for n in names}
        span = 0.0
        imax = (1 << 63) - 1
        n_ok = 0
        for _ in range(reps):
            tl = sync[16:16 + 32].view(torch.int64)
            tl[0::2] = imax
            tl[1::2] = 0
            sync[7] = 1
            st.replay()
            torch.cuda.synchronize(self.dev)
            sync[7] = 0
            t = tl.cpu().tolist()
            live = [k for k in range(5) if t[2 * k] != imax and t[2 * k + 1] > 0]
            if not live:
                continue
            t0 = min(t[2 * k] for k in live)
            n_ok += 1
            span += (max(t[2 * k + 1] for k in live) - t0) / 1e3
            for k in live:
                a = acc[names[k]]
                a[0] += (t[2 * k] - t0) / 1e3; a[1] += (t[2 * k + 1] - t0) / 1e3; a[2] += (t[2 * k + 1] - t[2 * k]) / 1e3
        if n_ok == 0:
            return None
        return {"replays": n_ok, "span_us": span / n_ok,
                "kernels": {n: {"start_us": round(a[0] / n_ok, 2), "end_us": round(a[1] / n_ok, 2), "dur_us": round(a[2] / n_ok, 2)}
                            for n, a in acc.items() if a[1] > 0}}

    def kernels_per_step(self):
        """Kernels of this library per step, counted by the library itself around one eager pass of the step's own launch
        sequence (what the graph replays)."""
        from contrastiveseg_b200 import _abi
        lib = _abi.load()
        if not self.steps:
            return None
        st = self.steps[0]
        snap = None
        if self.bank:
            b = self.mbank
            snap = [t.clone() for t in (b.segment_queue, b.segment_queue_ptr, b.pixel_queue, b.pixel_queue_ptr)]
        n0 = lib.pcl_launch_count()
        with torch.cuda.device(self.dev):
            st._enqueue(torch.cuda.current_stream(self.dev).cuda_stream)
        n = int(lib.pcl_launch_count() - n0)
        torch.cuda.synchronize(self.dev)
        if snap is not None:                               # this extra step is not part of any measurement
            for t, v in zip((b.segment_queue, b.segment_queue_ptr, b.pixel_queue, b.pixel_queue_ptr), snap):
                t.copy_(v)
            if b.shadow is not None:
                b.sync_shadow()
        return n

    def measure(self, sampler=None, with_eager=False, with_e2e=True, keep_outputs=False):
        """keep_outputs: self.outputs = a host copy (output_sample) of what the last timed step returned."""
        a = self.args
        out = {"workload": workload_config(self.cfg, self.bank)["workload"], "per_gpu_batch": self.cfg["B"],
               "rotation_sets": self.R, "working_set_mb": round(working_set_bytes(self.cfg, self.bank) / 1e6, 1)}
        fn, mode = (self.replay, "graph") if self.steps else (self.eager, "eager")
        if not self.steps:
            out["graph_error"] = self.graph_error or "disabled (--no-graph)"

        def keep(i):
            self.outputs = output_sample(*self.step_outputs(i))
        ms, host, window = self.time_loop(fn, a.steps, a.warmup, sampler, after_timed=keep if keep_outputs else None)
        out.update(mode=mode, ms_per_step=ms, value=self.world * self.cfg["B"] / (ms / 1e3), host_ms_per_step=host,
                   clock_window=window, kernels_per_step=self.kernels_per_step())
        if with_e2e:
            e_steps = max(3, min(a.steps, 50))
            ev, h2d = self.e2e(fn, e_steps)
            out["e2e"] = {"value": ev, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "steps": e_steps,
                          "h2d_gbs_per_gpu": h2d * ev / (self.world * self.cfg["B"]) / 1e9,
                          "note": "PCIe-bound: pinned H2D copies reach 55 GB/s on this box (tools/h2d_probe.py), the step itself is 2 % of e2e"}
        if with_eager and self.steps:
            ems, ehost, _ = self.time_loop(self.eager, a.steps, a.warmup)
            out["eager"] = {"ms_per_step": ems, "value": self.world * self.cfg["B"] / (ems / 1e3), "host_ms_per_step": ehost}
        if self.bank and self.world > 1 and self.steps:
            # the one data-path collective: NCCL all_gather of the enqueue packet, timed alone on the device
            st = self.steps[0]
            for _ in range(5):
                st._gather()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            self.barrier()
            e0.record()
            for _ in range(50):
                st._gather()
            e1.record()
            self.barrier()
            (g_ms,) = self.reduce_max([e0.elapsed_time(e1) / 50])
            out["allgather_ms"] = g_ms
            out["packet_bytes_per_rank"] = int(st.enq["packet"].numel() * 4)
        losses = [float(fn(i).item()) for i in range(2)]
        out["finite_loss"] = all(x == x and abs(x) < 1e30 for x in losses)
        return out

    def close(self):
        self.steps = []
        self.inp = self.host = None
        from contrastiveseg_b200 import functional as Fn
        Fn.clear_workspaces()
        torch.cuda.empty_cache()


def step_algorithmic_bytes(cfg, A, bank):
    """SURVEY §8d: labels at the embedding stride + seg (argmax) + gather + dense-gradient write (+ the bank shadow once per
    sweep, forward and backward, + the enqueue's pass over the keys)."""
    hw = cfg["h"] * cfg["w"]
    b = cfg["B"] * hw * 8 + cfg["B"] * cfg["K"] * hw * 4 + A * cfg["D"] * 4 + cfg["B"] * cfg["D"] * hw * 4
    if bank:
        b += 2 * (cfg["K"] - 1) * 2 * cfg["M"] * cfg["D"] * 2 + cfg["B"] * cfg["D"] * hw * 4
    return b


def run_engine(args, cfg, bank, rank, world, dev):
    import contrastiveseg_b200 as cs
    from contrastiveseg_b200 import _abi
    _abi.load()
    peaks = load_peaks()
    sampler = ClockSampler(dev.index)
    # ---- headline: the workload named on the command line (default s1 = BASELINE configs[1]), weak scaling ----
    head = Workload(args, args.workload, cfg, bank, rank, world, dev)
    hm = head.measure(sampler=sampler, with_eager=True, keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, head.outputs)
    A_live = int(head.steps[0].ws.plan[2].item()) if head.steps else 0
    timeline = head.graph_timeline() if not os.environ.get("PCL_BENCH_TINY") else None
    inp0 = head.inp[0]
    stages = {}
    if rank == 0 and not bank and world == 1:
        stages, A_live = stage_timings(cfg, inp0, dev, args.precision)
    wrapper = train = tens = None
    if rank == 0 and world == 1 and not bank and not os.environ.get("PCL_BENCH_HEADLINE_ONLY"):
        embed = inp0["embed"].detach().requires_grad_(True)
        wrapper = {}
        for name, fused in (("fused_seg_ce_ms", True), ("torch_seg_ce_ms", False)):
            cw = engine_configer(cfg, bank, args.precision)
            cw.add(["contrast", "fused_seg_ce"], fused)
            mod = cs.ContrastCELoss(cw).to(dev)
            seg_l = inp0["seg"].clone().requires_grad_(True)

            def wstep():
                embed.grad = None; seg_l.grad = None
                mod({"seg": seg_l, "embed": embed}, inp0["target"], with_embed=True).backward()
            for _ in range(5):
                wstep()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            e0.record()
            for _ in range(30):
                wstep()
            e1.record()
            torch.cuda.synchronize(dev)
            wrapper[name] = e0.elapsed_time(e1) / 30
        if not os.environ.get("PCL_BENCH_NO_TRAIN_ITER"):
            try:
                train = train_iter_bench(cfg, inp0, dev, args.precision)
                train["loss_step_ms"] = wrapper.get("fused_seg_ce_ms")
                train["loss_step_share"] = wrapper.get("fused_seg_ce_ms") / train["ms_per_iter"]
            except Exception as exc:                      # noqa: BLE001
                train = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        if cfg["D"] == 256:
            tens = tensor_sweep_roofline(dev, peaks)
    # ---- cpu baseline (rank 0, N=1 only): bounded sample of the same workload at the SAME batch ----
    cpu = None
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        threads, t1 = calibrate_cpu(cfg, bank)
        ih = head.host[0]
        t0 = time.perf_counter()
        cpu_port_step(ih, cfg, bank)
        cdt = time.perf_counter() - t0
        n_cpu = 1
        if cdt < 8.0:                                   # small geometries: a few more steps
            n_cpu = 3
            t0 = time.perf_counter()
            for _ in range(n_cpu):
                cpu_port_step(ih, cfg, bank)
            cdt = (time.perf_counter() - t0) / n_cpu
        cpu = {"value": cfg["B"] / cdt, "unit": "images/s", "cores": threads, "kind": "port",
               "sample": f"{n_cpu} step(s) of the full workload (batch {cfg['B']}) after the calibration pass, fp32 torch CPU on "
                         f"{threads} of {os.cpu_count()} host threads (fastest setting), {cdt * 1e3:.0f} ms/step"}
    head.close()
    # ---- the memory-bank step (BASELINE configs[2]: one image per rank + ONE NCCL all_gather of the enqueue packet per
    #      step) and strong scaling of the headline (global batch fixed), measured in the same run at every N ----
    blocks = {}
    if not bank and not os.environ.get("PCL_BENCH_HEADLINE_ONLY"):
        # the same step with the dense gradient kept across replays (GraphedContrastStep(sparse_reset=True)): only the A*D
        # entries of the previous replay are cleared instead of re-filling B*D*h*w zeros.  Reported next to the headline,
        # not as the headline: it puts a contract on the caller (nobody else writes the buffer).
        try:
            ws_ = Workload(args, args.workload + "-sparse-reset", cfg, False, rank, world, dev, sparse_reset=True)
            blocks["sparse_reset"] = dict(ws_.measure(with_e2e=False), config="headline workload, dense gradient buffer persistent "
                                          "across replays: the previous replay's A*D entries are cleared, no 268 MB refill")
            ws_.close()
        except Exception as exc:                          # noqa: BLE001
            blocks["sparse_reset"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    if not os.environ.get("PCL_BENCH_HEADLINE_ONLY") and args.workload == "s1":
        s2 = dict(S2)
        if os.environ.get("PCL_BENCH_TINY"):
            s2.update(B=1, D=32, h=16, w=16, K=5, stride=2, block=8, max_samples=32, max_views=4, M=8, F=2, net_stride=2)
        try:
            w2 = Workload(args, "s2", s2, True, rank, world, dev)
            blocks["bank"] = dict(w2.measure(with_e2e=False), config="BASELINE configs[2]: HRNet-W48 + pixel/region memory bank "
                                  "(19 x (5000+5000) x 256), one image per rank, max_views 100, bank merged by one NCCL "
                                  "all_gather of the enqueue packet per step; weak scaling (value = world images per step)")
            w2.close()
        except Exception as exc:                          # noqa: BLE001
            blocks["bank"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        if world > 1 and cfg["B"] % world == 0:
            cs_ = dict(cfg); cs_["B"] = cfg["B"] // world
            try:
                w3 = Workload(args, "s1-strong", cs_, False, rank, world, dev)
                blocks["strong"] = dict(w3.measure(with_e2e=False), config=f"headline workload with the global batch {cfg['B']} "
                                        f"split over {world} ranks (lib/datasets/data_loader.py:137)")
                w3.close()
            except Exception as exc:                      # noqa: BLE001
                blocks["strong"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    if rank != 0:
        return None
    # ---- roofline of what was timed: the whole step against the HBM peak (the step is one graph; its kernels are
    #      latency-bound except the dense-gradient fill, so the per-step fraction is the honest figure) ----
    alg = step_algorithmic_bytes(cfg, A_live, bank)
    ach = alg / (hm["ms_per_step"] * 1e-3) / 1e9
    step_roof = {"achieved": ach, "frac": ach / peaks["hbm_gbs"], "algorithmic_bytes": alg,
                 "what": "all algorithmic bytes of the step (SURVEY 8d) over the timed ms_per_step"}
    fill = (timeline or {}).get("kernels", {}).get("k_fill_zero_excl")
    if fill and fill["dur_us"] > 0:
        # dominant kernel of the timed path: the engine's zero-fill of the dense gradient, timed INSIDE the graph replay
        fb = cfg["B"] * cfg["D"] * cfg["h"] * cfg["w"] * 4
        fa = fb / (fill["dur_us"] * 1e-6) / 1e9
        roof = {"kernel": "k_fill_zero_excl (dense-gradient zero-fill on 116 SMs it owns, next to the InfoNCE kernel on the other 32; "
                          "the HBM floor of the step; runs in the timed graph)",
                "bound": "hbm", "achieved": fa, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": fa / peaks["hbm_gbs"],
                "traffic": ncu_traffic("k_fill_zero_excl"), "peak_source": peaks["source"], "algorithmic_bytes": fb,
                "launch_us": fill["dur_us"], "timed_by": "in-graph %globaltimer stamps, mean of 20 replays (bench.py: graph_timeline)",
                "step": step_roof, "anchors": A_live, "kernels_per_step": hm["kernels_per_step"]}
    else:
        roof = {"kernel": "whole step (one CUDA-graph replay: all kernels of the loss step)" if hm["mode"] == "graph" else "whole step (eager)",
                "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"],
                "traffic": ncu_traffic("step"), "peak_source": peaks["source"], "algorithmic_bytes": alg,
                "anchors": A_live, "kernels_per_step": hm["kernels_per_step"]}
    clocks = dict(sampler.summary(), window=hm["clock_window"])
    kps = hm["kernels_per_step"] or 0
    conf = dict(workload_config(cfg, bank),
                step="one CUDA-graph replay per step (GraphedContrastStep)" if hm["mode"] == "graph" else "eager autograd call per step",
                l2=("inputs larger than L2 (working set %.0f MB vs 126 MB)" % hm["working_set_mb"]) if hm["rotation_sets"] == 1
                else f"rotating over {hm['rotation_sets']} input/gradient buffer sets ({hm['working_set_mb']:.0f} MB each) so that no step finds its inputs in L2")
    return {"metric": "contrast-loss fwd+bwd throughput", "value": hm["value"], "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": hm["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic", "config": conf, "clocks": clocks,
            "e2e": hm.get("e2e"), "gpu_launches": kps * args.steps, "roofline": roof, "cpu_baseline": cpu,
            "stage_ms": stages, "host_enqueue_ms_per_step": hm["host_ms_per_step"], "tensor_roofline": tens,
            "contrast_ce_wrapper": wrapper, "train_iter": train, "precision": args.precision,
            "cuda_graph": hm["mode"] == "graph", "graph_error": hm.get("graph_error"), "eager": hm.get("eager"),
            "graph_timeline": timeline, "sparse_reset": blocks.get("sparse_reset"),
            "bank": blocks.get("bank"), "strong": blocks.get("strong"), "impl": "engine"}


def tensor_sweep_roofline(dev, peaks, A=16384, N=65536, iters=5):
    """The dense contraction alone (similarity + negative-sum sweep on tcgen05) at one S4 point (BASELINE configs[4]):
    algorithmic FLOPs 2*A*N*D over the CUDA-event time, vs the measured bf16 peak."""
    from contrastiveseg_b200 import functional as Fn
    g = torch.Generator().manual_seed(7)
    a = torch.nn.functional.normalize(torch.randn(A, 256, generator=g), dim=1).to(dev)
    c = torch.nn.functional.normalize(torch.randn(N, 256, generator=g), dim=1).to(dev)
    ya = torch.sort(torch.randint(0, 19, (A,), generator=g)).values.to(dev)
    yc = torch.sort(torch.randint(0, 19, (N,), generator=g)).values.to(dev)
    c16 = Fn.to_bf16_rows(c, -(-N // 256) * 256)
    diag = torch.arange(A, device=dev) % N
    out = {}
    for name, neg_only in (("neg_sweep", True), ("forward", False)):
        run = lambda: Fn.infonce_tc_forward(a, ya, contrast_bf16=c16, contrast_cls=yc, n_cols=N, diag_col=diag,
                                            temperature=0.07, base_temperature=0.07, neg_only=neg_only)
        for _ in range(3):
            res = run()
        ts = []
        for _ in range(iters):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); res = run(); e1.record()
            torch.cuda.synchronize(dev)
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        out[name] = ts[len(ts) // 2]
    state = res
    loss, st, stt = state
    tb = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); Fn.infonce_tc_backward(stt, st); e1.record()
        torch.cuda.synchronize(dev)
        tb.append(e0.elapsed_time(e1))
    tb.sort()
    out["backward"] = tb[len(tb) // 2]
    fl = 2.0 * A * N * 256
    ach = fl / (out["neg_sweep"] * 1e-3) / 1e12
    return {"kernel": "k_tc_fwd<NEG> (anchor x bank similarity + negative-sum sweep, tcgen05)", "bound": "tensor",
            "workload": f"S4 sweep point A={A} x N={N}, D=256, bf16 operands", "achieved": ach,
            "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops"],
            "peak_source": peaks["source"], "traffic": None, "ms": out,
            "forward_tflops": fl / (out["forward"] * 1e-3) / 1e12, "backward_tflops": fl / (out["backward"] * 1e-3) / 1e12}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps [engine 200, reference 3]")
    ap.add_argument("--warmup", type=int, default=None, help="warm-up steps [engine 10, reference 1]")
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--workload", default="s1", choices=["s1", "s2", "s3"],
                    help="s1 = BASELINE configs[1] (headline), s2 = configs[2] (memory bank), s3 = configs[3] (171 classes)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (default): the workload's batch per GPU; strong: the workload's batch split over the ranks "
                         "(global batch fixed, as lib/datasets/data_loader.py:137 does), SURVEY §8d asks for both")
    ap.add_argument("--no-graph", action="store_true",
                    help="run GraphedContrastStep's launch sequence eagerly instead of as a captured CUDA graph")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"],
                    help="InfoNCE sweeps: bf16 operands on tcgen05 tensor cores (default) or the exact fp32 SIMT sweep")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="engine arm: write the loss and d loss/d embed of the last timed step (rank 0) as DIR/<name>.npy; "
                         "the gradient as a fixed channel sample when it exceeds 48 MB")
    args = ap.parse_args()
    ref_arm = args.impl == "reference"
    if args.steps is None:                           # the defaults are sized for the GPU arm
        args.steps = 3 if ref_arm else 200
    if args.warmup is None:
        args.warmup = 1 if ref_arm else 10
    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    if ref_arm and args.dump_outputs:
        raise SystemExit("--dump-outputs writes what the engine computed: use it with --impl engine")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = dict({"s1": S1, "s2": S2, "s3": S3}[args.workload])
    bank = args.workload in ("s2", "s3")
    if args.scaling == "strong":
        if cfg["B"] % world != 0:
            raise SystemExit(f"--scaling strong: global batch {cfg['B']} is not divisible by {world} ranks")
        cfg["B"] //= world
    if os.environ.get("PCL_BENCH_TINY"):            # contract tests on small hosts: same code path, toy geometry
        cfg.update(B=2, D=32, h=16, w=16, K=5, stride=2, block=8, max_samples=32, max_views=4)
        if bank:
            cfg.update(M=8, F=2, net_stride=2)
    if ref_arm:
        res = run_reference(args, cfg, bank, rank)
        if res is not None:
            print(json.dumps(res), flush=True)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl engine needs a CUDA device (the engine has no CPU path)")
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    pin_to_gpu_local_cpus(dev.index)          # NUMA-local host threads for the launch path, at every N (incl. 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=dev)
    res = run_engine(args, cfg, bank, rank, world, dev)
    if res is not None:
        print(json.dumps(res), flush=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
