"""Training step parity (SURVEY.md §8f rank 2, BASELINE config 5): the façade's batch step vs the
UNMODIFIED reference train.py (golden: one 64-sample batch, seed-0 net, CPU fp32).  CPU: fp32, tight
tolerance.  GPU: bf16 autocast, loss within 2e-2."""
import json
import os

import numpy as np
import pytest
import torch

from scripts.golden_train import train_batch


@pytest.fixture(scope="module")
def gold(golden_dir):
    with open(os.path.join(golden_dir, "train_reference.json")) as f:
        return json.load(f)


def _step(device_is_gpu):
    from chinesechesszero_b200.train import TrainPipeline

    states, probs, winners = train_batch()
    torch.manual_seed(0)
    pipe = TrainPipeline(batch_size=len(states), net_kwargs=dict(use_gpu=device_is_gpu))
    assert pipe.policy_value_net.device.type == ("cuda" if device_is_gpu else "cpu")
    r = pipe.train_step(torch.tensor(states, dtype=torch.float32), torch.tensor(probs, dtype=torch.float32),
                        torch.tensor(winners, dtype=torch.float32))
    # end-of-pass multiplier update (train.py:269-279)
    if pipe.last_kl > pipe.kl_targ * 2 and pipe.lr_multiplier > 0.05:
        pipe.lr_multiplier = max(0.05, pipe.lr_multiplier / 1.2)
    elif pipe.last_kl < pipe.kl_targ / 2 and pipe.lr_multiplier < 2.0:
        pipe.lr_multiplier = min(2.0, pipe.lr_multiplier * 1.2)
    return pipe, r


def test_cpu_fp32_step_matches_reference(gold):
    pipe, r = _step(False)
    g = gold["log"]
    assert not r["rolled_back"]
    assert abs(r["loss"] - g["loss"]) < 2e-4 and abs(r["policy_loss"] - g["policy_loss"]) < 2e-4
    assert abs(r["value_loss"] - g["value_loss"]) < 2e-4 and abs(r["entropy"] - g["entropy"]) < 2e-4
    assert abs(r["kl"] - g["kl"]) < 2e-4
    assert pipe.lr_multiplier == gold["lr_multiplier_after"]


@pytest.mark.gpu
def test_gpu_bf16_step_within_tolerance(gold):
    pipe, r = _step(True)
    g = gold["log"]
    assert not r["rolled_back"]
    assert abs(r["loss"] - g["loss"]) < 2e-2 and abs(r["policy_loss"] - g["policy_loss"]) < 2e-2
    assert abs(r["value_loss"] - g["value_loss"]) < 2e-2 and abs(r["entropy"] - g["entropy"]) < 2e-2
    assert abs(r["kl"] - g["kl"]) < 5e-3


def test_policy_update_runs_over_npy_replay(tmp_path):
    from chinesechesszero_b200.train import TrainPipeline

    states, probs, winners = train_batch(8)
    np.save(tmp_path / "states.npy", states)
    np.save(tmp_path / "mcts.npy", probs)
    np.save(tmp_path / "winners.npy", winners)
    torch.manual_seed(1)
    pipe = TrainPipeline(data_dir=str(tmp_path), batch_size=8, net_kwargs=dict(num_channels=16, resblocks_num=1))
    loss0, ent0 = pipe.policy_update(generator=torch.Generator().manual_seed(0))
    for _ in range(5):
        loss, ent = pipe.policy_update(generator=torch.Generator().manual_seed(0))
    assert np.isfinite(loss) and loss < loss0 and 0.05 <= pipe.lr_multiplier <= 2.0
    # mcts rows that do not sum to one are rejected like the reference does (train.py:134-138)
    bad = probs.copy()
    bad[0] *= 0.5
    with pytest.raises(ValueError):
        pipe.train_step(torch.tensor(states, dtype=torch.float32), torch.tensor(bad, dtype=torch.float32),
                        torch.tensor(winners, dtype=torch.float32))


def test_step_backup_restores_weights_and_optimizer_state():
    """The rollback copy (train.py:155-163, 200-206): after restore() the weights, BN statistics, Adam moments and step
    counters are the ones saved before the step -- also when the step being undone was the optimizer's first."""
    from chinesechesszero_b200.train import TrainPipeline

    states, probs, winners = train_batch(8)
    torch.manual_seed(2)
    pipe = TrainPipeline(batch_size=8, net_kwargs=dict(num_channels=16, resblocks_num=1))
    pv = pipe.policy_value_net
    net, opt = pv.policy_value_net, pv.optimizer
    batch = tuple(torch.tensor(a, dtype=torch.float32) for a in (states, probs, winners))

    def snapshot():
        return ({k: v.clone() for k, v in net.state_dict().items()},
                {i: {k: (v.clone() if torch.is_tensor(v) else v) for k, v in st.items()} for i, st in
                 enumerate(opt.state[p] for g in opt.param_groups for p in g["params"] if p in opt.state)})

    # first step: the optimizer has no state yet
    w0, s0 = snapshot()
    assert not s0
    pipe.train_step(*batch)
    assert len(opt.state) > 0
    pipe._backup.restore(net, opt)
    w1, s1 = snapshot()
    assert not s1 and all(torch.equal(w0[k], w1[k]) for k in w0)
    # later step: moments and step counters come back
    pipe.train_step(*batch)
    pipe.train_step(*batch)
    w2, s2 = snapshot()
    r = pipe.train_step(*batch)   # backs up (w2, s2), then steps
    assert not r["rolled_back"]
    w_after, _ = snapshot()
    assert any(not torch.equal(w2[k], w_after[k]) for k in w2)
    pipe._backup.restore(net, opt)
    w3, s3 = snapshot()
    assert all(torch.equal(w2[k], w3[k]) for k in w2)
    assert s2.keys() == s3.keys()
    for i in s2:
        for k, v in s2[i].items():
            assert torch.equal(v, s3[i][k]) if torch.is_tensor(v) else v == s3[i][k]
