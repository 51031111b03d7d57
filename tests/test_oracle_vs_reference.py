"""The CPU port against the unmodified reference on random synthetic inputs.

The reference's outputs and the permutations it drew are stored in tests/golden/random_seeds.npz
(tests/golden/make_golden.py random_seeds); the inputs are regenerated here from contrastiveseg_b200.synth."""
import numpy as np
import pytest
import torch

from oracle import ref_port as P
from contrastiveseg_b200.synth import make_bank, make_contrast_batch
from helpers import load_golden, rel_err, unpack_perms


@pytest.fixture(scope="module")
def golden():
    return load_golden("random_seeds")


def _check_inputs(stored, *tensors):
    sums = np.array([t.double().sum().item() for t in tensors])
    assert np.allclose(sums, stored, rtol=1e-12, atol=1e-9), "synth inputs differ from those the golden was made from"


@pytest.mark.parametrize("seed", [31, 32, 33])
@pytest.mark.parametrize("mem", [False, True])
def test_loss_random_seeds(seed, mem, golden):
    key = f"s{seed}_mem{int(mem)}_"
    K, D = 6, 32
    data = make_contrast_batch(B=3, D=D, h=20, w=24, num_classes=K, img_stride=2, block=6, seed=seed, boost=1.5)
    predict = data["seg"].argmax(1)
    inputs = [data["embed"], data["target"], predict]
    queue = None
    if mem:
        bank = make_bank(K, 15, D, seed)
        queue = torch.cat((bank["segment_queue"], bank["pixel_queue"]), 1)
        inputs.append(queue)
    _check_inputs(golden[key + "input_sums"], *inputs)
    replay = P.PermReplay(unpack_perms(golden[key + "perm_flat"], golden[key + "perm_lens"]))
    e2 = data["embed"].clone().requires_grad_(True)
    l2 = P.pixel_contrast_loss(e2, data["target"], predict, temperature=0.1, base_temperature=0.07, max_samples=50,
                               max_views=7, queue=queue, perm_fn=replay)
    l2.backward()
    assert replay.pos == len(replay.draws)
    assert rel_err(l2.item(), golden[key + "loss"]) < 2e-6
    assert torch.allclose(e2.grad, torch.from_numpy(golden[key + "grad_embed"]), rtol=1e-4, atol=1e-9)


def test_enqueue_random(golden):
    K, D, M, Fq = 5, 16, 6, 4
    bank = make_bank(K, M, D, 3)
    b = [bank[k].clone() for k in ("segment_queue", "segment_queue_ptr", "pixel_queue", "pixel_queue_ptr")]
    _check_inputs(golden["enq_input_sums"], *b)
    for s in range(5):
        data = make_contrast_batch(B=2, D=D, h=12, w=12, num_classes=K, img_stride=2, block=6, seed=50 + s)
        _check_inputs(golden[f"enq{s}_input_sums"], data["embed"], data["target"])
        replay = P.PermReplay(unpack_perms(golden[f"enq{s}_perm_flat"], golden[f"enq{s}_perm_lens"]))
        P.dequeue_and_enqueue(data["embed"], data["target"], *b, network_stride=2, memory_size=M,
                              pixel_update_freq=Fq, perm_fn=replay)
        assert replay.pos == len(replay.draws)
        for k, y in zip(("sq", "sp", "pq", "pp"), b):
            assert torch.allclose(torch.from_numpy(golden[f"enq{s}_{k}"]).float(), y.float(), atol=1e-6)
