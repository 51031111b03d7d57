"""bench.py JSON contract of the reference arm (runs on CPU with a toy geometry: PCL_BENCH_TINY=1)."""
import json
import os
import subprocess
import sys

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _run(extra):
    env = dict(os.environ, PCL_BENCH_TINY="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1"] + extra, capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_reference_arm_json_line():
    d = _run([])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None and d["value"] > 0 and "workload" in d["config"]


def test_reference_arm_bank_workload():
    d = _run(["--workload", "s2"])
    assert d["impl"] == "reference" and "memory bank" in d["config"]["workload"]


def _run_engine_on_emulator(monkeypatch, workload="s1", dump=None):
    """bench.run_engine end to end on the CPU: the engine's kernels on the host-fiber emulator (tests/emu), CUDA events /
    pinned memory / graph capture stubbed, toy geometry.  Exercises everything between argument parsing and the JSON line."""
    import types
    import torch
    sys.path.insert(0, ROOT)
    import bench
    import emu_harness
    from contrastiveseg_b200 import graph_step
    emu_harness.use_emulation(monkeypatch)

    class Ev:
        def __init__(self, **k):
            pass

        def record(self):
            pass

        def elapsed_time(self, other):
            return 2.0

    monkeypatch.setattr(torch.cuda, "Event", Ev)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(torch.cuda, "empty_cache", lambda: None)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self: self)
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_capture", lambda self, warmup: None)
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_fork_zero_fill", lambda self: self._side_branch(0))
    monkeypatch.setattr(graph_step.GraphedContrastStep, "_join_zero_fill", lambda self: None)
    monkeypatch.setenv("PCL_BENCH_TINY", "1")
    orig_stage = bench.stage_timings
    monkeypatch.setattr(bench, "stage_timings", lambda *a, **k: orig_stage(*a, iters=2))        # the default 20 only averages
    args = types.SimpleNamespace(steps=4, warmup=3, precision="fp32", workload=workload, scaling="weak", no_graph=False,
                                 no_cpu_baseline=False, gpus=1, dump_outputs=dump)
    cfg = dict(bench.S1 if workload == "s1" else bench.S2)
    cfg.update(B=2, D=32, h=16, w=16, K=5, stride=2, block=8, max_samples=32, max_views=4)
    if workload != "s1":
        cfg.update(M=8, F=2, net_stride=2)
    res = bench.run_engine(args, cfg, workload != "s1", 0, 1, torch.device("cpu"))
    return json.loads(json.dumps(res))                     # must be JSON-serialisable as is


REQUIRED = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline")


def test_engine_arm_line_on_the_emulator(monkeypatch):
    res = _run_engine_on_emulator(monkeypatch)
    for k in REQUIRED:
        assert k in res, k
    assert res["impl"] == "engine" and res["cuda_graph"] is True and res["config"]["step"].startswith("one CUDA-graph replay")
    assert res["ms_per_step"] == 0.5 and res["value"] == 2 * 4 / 2e-3          # 4 steps in the stubbed 2 ms
    assert res["eager"]["ms_per_step"] == 0.5
    r = res["roofline"]
    assert r["bound"] == "hbm" and r["kernel"].startswith("whole step") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert r["algorithmic_bytes"] > 2 * 32 * 16 * 16 * 4 and r["kernels_per_step"] >= 4
    assert res["gpu_launches"] == r["kernels_per_step"] * 4
    assert res["cpu_baseline"]["kind"] in ("port", "reference") and "batch 2" in res["cpu_baseline"]["sample"]
    assert res["train_iter"] and "error" not in res["train_iter"] and res["train_iter"]["finite_loss"] is True
    assert set(res["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} and res["e2e"]["h2d_bytes_per_step"] > 0
    # the memory-bank step (BASELINE configs[2]) is measured in the same run
    bank = res["bank"]
    assert "error" not in bank and bank["mode"] == "graph" and bank["finite_loss"] and bank["kernels_per_step"] > r["kernels_per_step"]
    assert bank["value"] == 1 * 4 / 2e-3 and res["strong"] is None


def test_engine_arm_dumps_the_last_timed_step(monkeypatch, tmp_path):
    import numpy as np
    import bench
    monkeypatch.setenv("PCL_BENCH_HEADLINE_ONLY", "1")
    monkeypatch.setattr(bench, "DUMP_GRAD_BYTES", 8 * 2 * 16 * 16 * 4)     # 8 of the toy gradient's 32 channels
    seen, replays = [], []
    orig_sample, orig_replay = bench.output_sample, bench.Workload.replay

    def spy(loss, grad):
        seen.append((loss.item(), grad.clone()))
        return orig_sample(loss, grad)

    def replay(self, i):
        loss = orig_replay(self, i)
        replays.append(loss.item())
        return loss
    monkeypatch.setattr(bench, "output_sample", spy)
    monkeypatch.setattr(bench.Workload, "replay", replay)
    _run_engine_on_emulator(monkeypatch, dump=str(tmp_path))
    assert sorted(os.listdir(tmp_path)) == ["grad_embed.npy", "grad_embed_channels.npy", "loss.npy"]
    loss, grad, ch = (np.load(os.path.join(tmp_path, n + ".npy")) for n in ("loss", "grad_embed", "grad_embed_channels"))
    assert len(seen) == 1 and loss.dtype == grad.dtype == np.float32 and ch.dtype == np.float64
    # 3 warm-up + 4 timed replays: the dump is the 7th, although the run replays the step again afterwards
    assert len(replays) > 7 and replays[6] != replays[-1]
    assert loss.shape == () and float(loss) == seen[0][0] == replays[6]
    idx = ch.astype(np.int64)
    assert grad.shape == (2, 8, 16, 16) and list(idx) == sorted(set(idx)) and 0 <= idx[0] and idx[-1] < 32
    assert np.array_equal(grad, seen[0][1][:, idx].numpy()) and np.count_nonzero(grad) > 0


def test_engine_arm_bank_workload_as_headline(monkeypatch):
    monkeypatch.setenv("PCL_BENCH_NO_TRAIN_ITER", "1")
    res = _run_engine_on_emulator(monkeypatch, workload="s2")
    assert "memory bank" in res["config"]["workload"] and res["cuda_graph"] is True and res["bank"] is None
    assert res["roofline"]["algorithmic_bytes"] > 0 and res["e2e"]["value"] > 0
