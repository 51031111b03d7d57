"""CPU execution of the engine's REAL kernel sources (tests/emu: the .cu files compiled for host fibers; the tensor path
against a functional model of mbarrier / TMA / tcgen05): the GPU tests of test_gpu_parity.py / test_gpu_topk.py /
test_gpu_zpending.py are re-run here with DEV = "cpu", through the same Python layer and the same C ABI (all but the
full-size ones), and the small cases of test_gpu_edges.py / test_gpu_zpending_edges.py.  This covers the kernel logic (indices,
barriers, reductions, selection, sampling, bank update, top-k select, graph rank draw) on machines without a GPU; it
proves nothing about the hardware build (that is what `-m gpu` is for) and floating point differs from the GPU in the
last bits (no FMA contraction), which the parity tolerances absorb.  TEST INFRASTRUCTURE: the product never loads the
emulation library (`_abi.load` refuses it)."""
import pytest
import torch

import contrastiveseg_b200 as cs
import emu_harness
import test_gpu_parity as G
import test_gpu_zpending as PD
import test_gpu_topk as TK
import test_gpu_edges as GE
import test_gpu_zpending_edges as ZE


@pytest.fixture
def emu(monkeypatch):
    lib = emu_harness.use_emulation(monkeypatch)
    for m in (G, TK, PD, GE, ZE):
        monkeypatch.setattr(m, "DEV", "cpu")
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    # the GPU tests rely on `.to(DEV)` producing a NEW tensor (host -> device copy); `.to("cpu")` would alias the source
    orig_to = torch.Tensor.to

    def to(self, *a, **k):
        r = orig_to(self, *a, **k)
        if r is self and len(a) == 1 and not k and isinstance(a[0], str) and a[0] == "cpu":
            return self.clone()
        return r

    monkeypatch.setattr(torch.Tensor, "to", to)
    return lib


def _case(fn, **kw):
    ident = fn.__name__.replace("test_", "") + ("[" + "-".join(str(v) for v in kw.values()) + "]" if kw else "")
    return pytest.param(fn, kw, id=ident)


PARITY = (
    [_case(G.test_loss_and_grad_match_reference, name=n)
     for n in ("nomem_small", "nomem_oddv", "nomem_mv1", "nomem_nondiv", "mem_small")] +
    [_case(G.test_concatenated_queue_tensor_is_accepted, name="mem_small")] +
    [_case(G.test_contrast_ce_wrapper, name=n, mem=m) for n, m in (("wrapper_nomem_embed", False),
                                                                   ("wrapper_nomem_warmup", False),
                                                                   ("wrapper_mem_embed", True))] +
    [_case(G.test_contrast_auxce_wrapper, name=n, fused=f) for n, f in (("wrapper_aux_embed", True),
                                                                        ("wrapper_aux_warmup_weighted", True),
                                                                        ("wrapper_aux_embed", False))] +
    [_case(G.test_bank_enqueue_matches_reference, name=n) for n in ("enqueue_aligned", "enqueue_q6")] +
    [_case(G.test_bank_enqueue_shape_error_like_reference)] +
    [_case(G.test_l2_normalize_matches_torch, shape=s) for s in ((2, 256, 16, 32), (1, 32, 7, 9), (3, 320, 5, 8))] +
    [_case(G.test_fused_normalize_path_equals_normalise_then_loss)] +
    [_case(G.test_device_rng_sampling_is_valid_and_loss_matches_oracle_on_same_indices, mem=m) for m in (False, True)] +
    [_case(G.test_device_rng_changes_between_steps_and_is_seed_reproducible),
     _case(G.test_explicit_infonce_modes_and_nan_semantics),
     _case(G.test_empty_inputs_give_zero_loss_not_a_crash),
     _case(G.test_torch_cpu_rng_mode_draws_the_reference_stream),
     _case(G.test_trainer_hook_end_to_end_with_bank),
     _case(G.test_workspace_is_released_when_the_graph_is_dropped_without_backward)] +
    [_case(G.test_fused_upsample_cross_entropy, B=b, K=k, h=h, w=w, H=H, W=W, weighted=wt)
     for b, k, h, w, H, W, wt in ((2, 5, 16, 20, 32, 40, False), (1, 19, 13, 10, 50, 37, True), (2, 7, 8, 8, 8, 8, False),
                                  (1, 3, 5, 7, 1, 9, True))]
)


@pytest.mark.parametrize("fn,kw", PARITY)
def test_gpu_parity_cases_on_emulated_kernels(emu, fn, kw):
    fn(**kw)


TOPK = (
    [_case(TK.test_topk_explicit_exact_data, A=a, N=n, k=k) for a, n, k in ((70, 333, 9), (130, 1000, 1), (64, 200, 64),
                                                                            (200, 129, 40))] +
    [_case(TK.test_topk_self_contrast_exact_data, k=k) for k in (3, 50)] +
    [_case(TK.test_topk_bank_mode_with_zero_tail, k=k) for k in (5, 37, 10 ** 6)] +
    [_case(TK.test_topk_through_the_loss_module, name=n) for n in ("nomem_small", "mem_small")]
)


TOPK += (
    [_case(TK.test_tc_topk_explicit_exact_data, A=a, N=n, k=k) for a, n, k in ((70, 333, 9), (200, 600, 40))] +
    [_case(TK.test_tc_topk_self_contrast_exact_data, k=3)] +
    [_case(TK.test_tc_topk_bank_mode_with_zero_tail, k=k) for k in (5, 10 ** 6)] +
    [_case(TK.test_tc_topk_through_the_loss_module, name=n) for n in ("nomem_d256", "mem_d256")]
)


@pytest.mark.parametrize("fn,kw", TOPK)
def test_topk_kernels_on_emulation(emu, fn, kw):
    """a10: the radix-select / weighted-sweep kernels of csrc/pcl_topk.cu against the sort-based oracle."""
    fn(**kw)


TENSOR = (
    [_case(G.test_tc_pipeline_raw_logits, A=a, N=n) for a, n in ((128, 256), (200, 1000))] +
    [_case(G.test_tc_forward_matches_oracle, A=a, N=n, T=t, self_mode=sm) for a, n, t, sm in ((200, 1000, 0.1, False),
                                                                                          (912, 912, 0.1, True))] +
    [_case(G.test_tc_backward_matches_oracle, A=200, N=1000, T=0.1, self_mode=False)] +      # self mode: fuzz_tensor_path
    [_case(G.test_loss_module_on_tensor_path, name=n) for n in ("nomem_d256", "mem_d256")] +
    [_case(G.test_bank_shadow_tracks_enqueue_and_tensor_path_uses_it),
     _case(PD.test_enqueue_between_loss_and_backward_does_not_change_the_gradient, precision="bf16")]
)


@pytest.mark.parametrize("fn,kw", TENSOR)
def test_tensor_path_on_the_functional_tcgen05_model(emu, fn, kw):
    """csrc/pcl_infonce_tc.cu (TMA-fed tcgen05 sweeps) compiled against tests/emu/shim/ptx_sm100.cuh, a functional model
    of mbarrier / TMA (SWIZZLE_128B) / tcgen05.mma (shared-memory descriptors, K- and MN-major) / tensor memory: the
    warp-specialised pipelines, descriptor arithmetic, class tests and epilogues run on the CPU.  The kernels are the
    ones verified on the B200, so a pass also confirms that the model reads descriptors the way the hardware does."""
    fn(**kw)


@pytest.mark.parametrize("mem,overlap", [(False, False), (False, True), (True, True)])
def test_graphed_step_tensor_path_on_emulation(emu, monkeypatch, mem, overlap):
    from contrastiveseg_b200 import graph_step
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_capture", lambda self, warmup: None)
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_fork_zero_fill", lambda self: self._side_branch(0))
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_join_zero_fill", lambda self: None)
    PD.test_graphed_step_equals_eager_step("bf16", mem, overlap)


@pytest.mark.parametrize("precision,D", [("fp32", 64), ("bf16", 256)])
def test_topk_inside_the_captured_step_on_emulation(emu, monkeypatch, precision, D):
    from contrastiveseg_b200 import graph_step
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_capture", lambda self, warmup: None)
    TK.test_topk_inside_the_captured_step_equals_the_eager_step(precision, D)


@pytest.mark.parametrize("geom", [dict(B=2, h=32, w=32, K=7, ms=128, mv=8), dict(B=3, h=32, w=48, K=9, ms=700, mv=40)])
def test_fused_small_anchor_step_on_emulation(emu, monkeypatch, geom):
    """csrc/pcl_infonce_fused.cu on the functional tcgen05 model (one phase per launch: the emulator runs the blocks of a
    grid one after another, so the two inter-CTA barriers become launch boundaries), the scan with the plan folded into
    its last block, the selection with the device-side seed counter and the reducing scatter."""
    from contrastiveseg_b200 import graph_step, _abi
    lib = _abi.load()

    monkeypatch.setattr(graph_step.GraphedContrastStep, "_capture", lambda self, warmup: None)
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_fork_zero_fill", lambda self: self._side_branch(0))
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_join_zero_fill", lambda self: None)
    PD.test_fused_small_anchor_step_matches_the_streaming_path_and_the_oracle(geom)
    PD.test_fused_step_with_no_qualifying_class_gives_zero_loss()
    if geom["ms"] == 700:
        PD.test_fused_step_sparse_reset_equals_full_fill()


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_graphed_bank_step_on_emulation(emu, monkeypatch, precision):
    """The bank step's launch sequence incl. the device-seeded enqueue packet (pcl_bank_packet_dev) == the trainer order."""
    from contrastiveseg_b200 import graph_step
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_capture", lambda self, warmup: None)
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_fork_zero_fill", lambda self: self._side_branch(0))
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_join_zero_fill", lambda self: None)
    PD.test_graphed_bank_step_with_enqueue_equals_the_trainer_order(precision)


@pytest.mark.parametrize("K,M,A,seed", [(5, 300, 200, 1), (12, 70, 150, 3), (40, 130, 260, 5), (171, 8, 400, 6)])
def test_tensor_path_bank_positives_by_class_blocks_on_emulation(emu, K, M, A, seed):
    """k_tc_pos_t on the functional tcgen05 / TMA model: blocks cut into several partial slots, several blocks per class."""
    G.test_tensor_path_bank_positives_by_class_blocks(K, M, A, seed)


@pytest.mark.parametrize("world,M,B", [(5, 4, 2), (8, 7, 3), (3, 40, 2)])
def test_bank_apply_of_many_ranks_on_emulation(emu, monkeypatch, world, M, B):
    """Last-writer-wins apply of world * B slots per class == the reference applied image by image."""
    PD.test_bank_apply_of_many_ranks_equals_the_sequential_reference(monkeypatch, world, M, B)


def test_fuzz_bank_apply_of_many_ranks_on_emulation(emu, monkeypatch):
    """Random (ranks, ring size, images per rank): the last-writer-wins apply == the reference applied image by image."""
    import random
    rng = random.Random(20)
    for _ in range(10):
        world, M, B = rng.randint(1, 9), rng.randint(3, 30), rng.randint(1, 3)
        PD.test_bank_apply_of_many_ranks_equals_the_sequential_reference(monkeypatch, world, M, B)


def test_bank_write_waits_for_backward_on_emulation(emu):
    """Gradient bit-identical with / without an enqueue between loss and backward; final bank equals an immediate enqueue."""
    PD.test_enqueue_between_loss_and_backward_does_not_change_the_gradient("fp32")


@pytest.mark.parametrize("overlap", [False, True])
def test_graphed_step_sequence_on_emulation(emu, monkeypatch, overlap):
    """GraphedContrastStep's launch sequence run eagerly (no CUDA graph on a CPU): the device-side rank draw
    (csrc/pcl_graph.cu) reproduces the eager sampling stream, the scatter-only backward equals the fused writer."""
    from contrastiveseg_b200 import graph_step
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_capture", lambda self, warmup: None)
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_fork_zero_fill", lambda self: self._side_branch(0))
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_join_zero_fill", lambda self: None)
    PD.test_graphed_step_equals_eager_step("fp32", False, overlap)


def test_product_refuses_the_emulation_library(monkeypatch):
    """No CPU path in the product: pointing the loader at the emulation build is an error, not a fallback."""
    import emu_harness as H
    from contrastiveseg_b200 import _abi
    H.emu_library()
    monkeypatch.setenv("PCL_B200_LIB", H.build_emu.LIB)
    monkeypatch.setattr(_abi, "_lib", None)
    with pytest.raises(_abi.PclError, match="emulation"):
        _abi.load()


def test_update_freq_larger_than_memory_is_refused(emu):
    """Found by differential fuzzing on the emulator: with pixel_update_freq > memory_size the wrap branch of the bank
    write would start before row 0 (the reference raises once a class has more than memory_size pixels).  The engine
    refuses the configuration up front — also in the real library, where the check runs before any CUDA call."""
    import ctypes as C
    from contrastiveseg_b200 import _abi
    from contrastiveseg_b200.synth import make_bank, make_contrast_batch
    data = make_contrast_batch(B=1, D=32, h=8, w=8, num_classes=4, img_stride=1, block=8, seed=1)
    b = make_bank(4, 3, 32, 2)
    with pytest.raises(_abi.PclError, match="shape"):
        cs.dequeue_and_enqueue(data["embed"], data["target"], b["segment_queue"], b["segment_queue_ptr"], b["pixel_queue"],
                               b["pixel_queue_ptr"], network_stride=1, memory_size=3, pixel_update_freq=5, distributed=False)
    import contrastiveseg_b200.build as build
    real = C.CDLL(build.library_path())
    real.pcl_bank_packet.restype = C.c_int32
    g = _abi.BankGeom(1, 32, 8, 8, 8, 8, 4, 3, 1, 5)
    assert real.pcl_bank_packet(C.byref(g), None, None, None, C.c_uint64(0), None, None, None) == -4


def test_full_size_cityscapes_batch_on_emulation(emu):
    """BASELINE configs[1] at full size (B=8, 256 x 128 x 256 embedding, 19 classes, up to 1024 anchors) through the
    emulated kernels: the size-independent properties of the GPU test (valid distinct anchors, loss == oracle on the same
    anchors, dense gradient zero outside the sampled columns)."""
    G.test_full_size_cityscapes_batch_properties()


def test_results_do_not_depend_on_the_thread_schedule():
    """Between synchronisation points the GPU may run the threads of a block in any order; the emulator's default is
    ascending.  Re-run a cross-section of the emulated cases (SIMT sweeps, selection, bank, top-k, the tcgen05 pipelines,
    the bit-exact graph/eager comparison) with a randomly permuted order: a failure here means a missing barrier."""
    import os
    import subprocess
    import sys
    env = dict(os.environ, PCL_EMU_SCHED="random:20260923")
    sel = ("loss_and_grad_match_reference and mem_small or bank_enqueue_matches_reference and q6 or topk_explicit_exact_data and 333 "
           "or tc_backward_matches_oracle or graphed_step_sequence_on_emulation and True or fused_upsample and 19")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-p", "no:cacheprovider",
                        "-k", sel], env=env, capture_output=True, text=True, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and "failed" not in r.stdout


def test_baseline_config0_geometry_on_emulation(emu, monkeypatch):
    """BASELINE configs[0] (the CPU plumbing case): bs 2, 256 x 256 input, stride 8 -> 32 x 32 x 256 embedding, 19 classes,
    the reference's default sampling limits — the whole ContrastCELoss (fused seg CE + pixel contrast) on the emulated
    kernels against the oracle on the reference's RNG stream."""
    from contrastiveseg_b200 import loss as loss_mod
    from contrastiveseg_b200.synth import make_contrast_batch
    monkeypatch.setattr(loss_mod.ContrastCELoss, "_can_fuse", lambda self, ce, s: self.fused_seg_ce)
    data = make_contrast_batch(B=2, D=256, h=32, w=32, num_classes=19, img_stride=8, block=96, seed=304)
    cfgd = cs.cityscapes_contrast_config()
    cfgd["contrast"]["rng"] = "torch_cpu"
    crit = cs.ContrastCELoss(cs.Configer(cfgd))
    torch.manual_seed(304)
    s64, e64 = data["seg"].double().requires_grad_(True), data["embed"].double().requires_grad_(True)
    ref = G.P.contrast_ce_loss({"seg": s64, "embed": e64}, data["target"], with_embed=True, loss_weight=0.1, temperature=0.1,
                               base_temperature=0.07, max_samples=1024, max_views=100)
    ref.backward()
    torch.manual_seed(304)
    seg, emb = data["seg"].clone().requires_grad_(True), data["embed"].clone().requires_grad_(True)
    loss = crit({"seg": seg, "embed": emb}, data["target"], with_embed=True)
    loss.backward()
    assert G.rel_err(loss.item(), ref.item()) < 2e-6
    assert (emb.grad.double() - e64.grad).abs().max().item() <= 1e-5 * e64.grad.abs().max().item()
    assert (seg.grad.double() - s64.grad).abs().max().item() <= 1e-5 * s64.grad.abs().max().item()
    assert emb.grad.abs().max().item() > 0


def test_device_sampler_equals_its_host_model(emu):
    """The pixels the selection kernels pick in device-RNG mode are exactly those of the host model of the sampler
    (contrastiveseg_b200.rng.device_rank): same seed derivation, same keyed bijection, same rank -> pixel order."""
    from contrastiveseg_b200 import functional as Fn, rng
    from contrastiveseg_b200.synth import make_contrast_batch
    K, ms, mv = 6, 60, 5
    data = make_contrast_batch(B=2, D=32, h=20, w=24, num_classes=K, img_stride=2, block=8, seed=9)
    opts = cs.ContrastOptions(max_samples=ms, max_views=mv, num_classes=K, seed=77)
    lab = G.P.downsample_labels(data["target"], 20, 24).reshape(2, -1)
    prd = data["seg"].argmax(1).reshape(2, -1)
    for call in (1, 2, 3):
        Fn._step_counter[0] = call - 1
        cs.pixel_contrast_loss(data["embed"], data["target"], seg=data["seg"], options=opts)
        ws = Fn.last_workspace(data["embed"].device)
        TC, V, A = ws.plan_header()[:3]
        pix, img, cls, _ = (t[:A].tolist() for t in ws.anchor_meta.view(4, -1))
        got = sorted(zip(img, cls, pix))
        seed = rng.device_step_seed(77, call)
        want = []
        for b in range(2):
            for c in range(K):
                is_c = lab[b] == c
                if int(is_c.sum()) <= mv:
                    continue
                hard = (is_c & (prd[b] != c)).nonzero()[:, 0].tolist()
                easy = (is_c & (prd[b] == c)).nonzero()[:, 0].tolist()
                kh, ke = G.P.split_hard_easy(len(hard), len(easy), V)
                want += [(b, c, hard[rng.device_rank(seed, b, c, K, False, j, len(hard))]) for j in range(kh)]
                want += [(b, c, easy[rng.device_rank(seed, b, c, K, True, j, len(easy))]) for j in range(ke)]
        assert got == sorted(want)


EDGES = (
    [_case(GE.test_tc_self_mode_at_row_tile_edges, A=a) for a in (2, 129, 257)] +
    [_case(GE.test_tc_explicit_mode_at_tile_edges, A=a, N=n) for a, n in ((1, 1), (128, 255), (129, 257), (129, 513))] +
    [_case(GE.test_tc_class_blocks_on_half_tile_boundaries, blocks=0, sorted_cols=s) for s in (True, False)] +
    [_case(GE.test_tc_nan_safe_row_without_positive)] +
    [_case(GE.test_tc_bank_class_blocks_at_tile_edges, M=m) for m in (63, 128)] +
    [_case(GE.test_segce_class_chunks, K=k, weighted=wt, ign=ig) for k, wt, ig in ((25, False, -1), (33, True, 255),
                                                                                 (59, True, -1), (171, False, 255))]
)


@pytest.mark.parametrize("fn,kw", EDGES)
def test_tile_and_chunk_edges_on_emulation(emu, fn, kw):
    """The small cases of test_gpu_edges.py: tcgen05 sweeps at 128/256 tile edges, class blocks on half-tile boundaries
    (sorted and shuffled columns), non-zero contrast pad rows, nan_safe, and seg-CE over several class chunks."""
    fn(**kw)


def _uncaptured(monkeypatch):
    from contrastiveseg_b200 import graph_step
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_capture", lambda self, warmup: None)
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_fork_zero_fill", lambda self: self._side_branch(0))
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_join_zero_fill", lambda self: None)


@pytest.mark.parametrize("A,TC,V,ms,mv", [(4, 2, 2, 1024, 2), (129, 3, 43, 130, 43)])
def test_fused_step_at_exact_anchor_counts_on_emulation(emu, monkeypatch, A, TC, V, ms, mv):
    """The fused step's launch sequence (uncaptured) at exact anchor counts against the host model and float64."""
    _uncaptured(monkeypatch)
    ZE.test_fused_step_at_exact_anchor_counts(A, TC, V, ms, mv)


def test_fused_step_anchor_count_changes_on_emulation(emu, monkeypatch):
    """A = 1024 -> 129 -> 4 -> 1024 through one step object with sparse_reset: no row of a larger replay leaks."""
    _uncaptured(monkeypatch)
    ZE.test_fused_step_anchor_count_changes_between_replays(True)


def test_device_bank_rank_on_emulation(emu):
    """The host model of the enqueue draw equals k_bank_rows' own draw (packets bit for bit)."""
    ZE.test_device_bank_rank_is_the_packet_kernels_draw()
