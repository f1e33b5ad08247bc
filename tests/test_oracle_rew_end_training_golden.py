"""CPU: the reward / termination model's training row (RewEndModel.forward + backward, rew_end_model.py:57-90) against the
unmodified reference (tests/golden/rew_end_training.npz, written by training_oracle/make_rew_end_golden.py):
  * the oracle's loss, logits and fp32 gradients, and the write-through of the final observation into batch.obs;
  * the product's RewEndModel.forward host logic (substitution, mask, losses, confusion matrices) with the oracle standing in
    for the native autograd node;
  * the error budget of the native precision plan (fp16 emulation vs fp32) on the fixture and at the trainer's batch shape."""
import os
import types

import numpy as np
import pytest
import torch

from oracle import fp16_oracle as E
from oracle import torch_oracle as O
from training_oracle import rew_end as R

WSEED = 778
# bounds of the GPU tests (tests/test_gpu_rew_end_training.py); the emulated budget must sit inside them with room to spare
WHOLE_BOUND, TENSOR_BOUND, NEGLIGIBLE = 1e-3, 4e-3, 1e-4


def _fixture(golden_dir):
    g = np.load(os.path.join(golden_dir, "rew_end_training.npz"))
    sd = O.seeded_state_dict(O.rew_end_shapes(O.RewEndCfg()), WSEED)
    assert abs(O.state_checksum(sd) - float(g["weights_checksum"])) < 1e-6 * float(g["weights_checksum"])
    batch = {k: torch.from_numpy(g[k]) for k in ("obs", "act", "rew", "end", "mask_padding", "final_obs")}
    return g, sd, batch


def _check_grads(named_grads, g, rtol_norm=2e-4):   # the rule of tests/test_oracle_training_golden.py
    keys, norms, samples = O.grad_summary(named_grads)
    assert keys == [str(k) for k in g["grad_keys"]]
    ref_n, ref_s = g["grad_norms"], g["grad_samples"]
    total = float(np.sqrt((ref_n ** 2).sum()))
    assert np.all(np.abs(norms - ref_n) <= rtol_norm * ref_n + 1e-6 * total), float(np.max(np.abs(norms - ref_n) / (ref_n + 1e-12)))
    numel = np.array([gr.numel() for _, gr in named_grads], np.float64)
    scale = (ref_n / np.sqrt(numel))[:, None]
    assert np.all(np.abs(samples - ref_s) <= 2e-4 * np.abs(ref_s) + 2e-3 * scale + 1e-9)


def _count_confusion(logits, target, n):
    m = np.zeros((n, n), np.int64)
    for t, p in zip(target, logits.argmax(1)):
        m[int(t), int(p)] += 1
    return m


def test_oracle_rew_end_loss_and_gradients_match_reference(golden_dir):
    g, sd, b = _fixture(golden_dir)
    for v in sd.values():
        v.requires_grad_(True)
    obs = b["obs"].clone()
    loss, loss_rew, loss_end, lr, le, _, _ = R.rew_end_loss(obs, b["act"], b["rew"], b["end"], b["mask_padding"], b["final_obs"], sd,
                                                            O.RewEndCfg())
    for got, key in ((loss, "loss"), (loss_rew, "loss_rew"), (loss_end, "loss_end")):
        assert abs(got.item() - float(g[key])) <= 2e-5 * abs(float(g[key])), (key, got.item(), float(g[key]))
    assert torch.allclose(lr, torch.from_numpy(g["logits_rew"]), rtol=1e-4, atol=1e-5)
    assert torch.allclose(le, torch.from_numpy(g["logits_end"]), rtol=1e-4, atol=1e-5)
    # the final frames went into the caller's obs (the reference's view assignment), at frame argmax(end) + 1
    assert torch.equal(obs, torch.from_numpy(g["obs_after"]))
    assert torch.equal(obs[0, 3], b["final_obs"][0]) and torch.equal(obs[1, 5], b["final_obs"][1])
    assert not torch.equal(obs, b["obs"])
    loss.backward()
    _check_grads([(k, v.grad) for k, v in sd.items()], g)


def test_product_rew_end_forward_host_logic_matches_reference(golden_dir, monkeypatch):
    """RewEndModel.forward with the oracle's differentiable predict_rew_end in place of the native node (no GPU needed)."""
    from diamond_b200.models import rew_end_model as M

    g, sd, b = _fixture(golden_dir)
    cfg = O.RewEndCfg()
    model = M.RewEndModel(M.RewEndModelConfig(cfg.lstm_dim, cfg.img_channels, cfg.img_size, cfg.cond_channels, list(cfg.depths),
                                              list(cfg.channels), list(cfg.attn_depths), cfg.num_actions))
    model.load_state_dict(sd)
    params = dict(model.named_parameters())

    class _OracleFn:
        @staticmethod
        def apply(module, names, obs, act, next_obs, *ps):
            lr, le, _ = O.predict_rew_end(obs, act, next_obs, dict(zip(names, ps)), cfg)
            return lr, le
    monkeypatch.setattr(M, "_RewEndFn", _OracleFn)
    info = [{"final_observation": b["final_obs"][0]}, {"final_observation": b["final_obs"][1]}, {}, {}]
    batch = types.SimpleNamespace(obs=b["obs"].clone(), act=b["act"], rew=b["rew"], end=b["end"], mask_padding=b["mask_padding"], info=info)
    loss, metrics = model(batch)
    assert abs(loss.item() - float(g["loss"])) <= 2e-5 * float(g["loss"])
    for k in ("loss_rew", "loss_end"):
        assert abs(metrics[k].item() - float(g[k])) <= 2e-5 * float(g[k]), k
    assert metrics["loss_total"].item() == loss.item() and not metrics["loss_total"].requires_grad
    assert torch.equal(batch.obs, torch.from_numpy(g["obs_after"]))
    mask = b["mask_padding"][:, :-1]
    t_rew = b["rew"][:, :-1][mask].sign().long().add(1).numpy()
    t_end = b["end"][:, :-1][mask].numpy()
    for key, logits, target, n in (("rew", g["logits_rew"], t_rew, 3), ("end", g["logits_end"], t_end, 2)):
        cm = metrics["confusion_matrix"][key]
        assert cm.dtype == torch.int64 and cm.shape == (n, n)
        assert np.array_equal(cm.numpy(), _count_confusion(logits, target, n)), key
    loss.backward()
    _check_grads([(k, p.grad) for k, p in params.items()], g)


def _budget(got, want):
    whole, per = E.rel_errors(got, want)
    total = float(sum(w.double().pow(2).sum() for w in want.values())) ** 0.5
    shares = {k: per[k] * float(want[k].double().norm()) / total for k in per}
    worst = max(per, key=per.get)
    over = [k for k in per if per[k] >= TENSOR_BOUND and shares[k] >= NEGLIGIBLE]
    return whole, worst, per[worst], over


def test_error_budget_fixture_batch(golden_dir):
    """fp16 emulation of the native path vs the fp32 oracle on the fixture batch (DESIGN.md section 2)."""
    _, sd, b = _fixture(golden_dir)
    cfg = O.RewEndCfg()
    want = R.parameter_grads(b, sd, cfg)
    got = R.parameter_grads(b, sd, cfg, emulated=True)
    whole, worst, e_worst, over = _budget(got, want)
    print(f"rew_end budget, fixture: whole {whole:.2e}, worst tensor {worst} {e_worst:.2e}")
    assert whole < 0.5 * WHOLE_BOUND and not over, (whole, over)
    # why the training plan's forward convs are split-fp16: with single-fp16 operands the forward's rounding alone moves the
    # LSTM input weights' gradient (fp32 arithmetic) enough to exceed the whole-gradient bound
    single, _, _, _ = _budget(R.parameter_grads(b, sd, cfg, emulated=True, split_forward=False), want)
    print(f"rew_end budget, fixture, single-fp16 forward: whole {single:.2e}")
    assert single > WHOLE_BOUND


def test_error_budget_trainer_shape():
    """The same at b = 32, T = 19 (4 distinct sequences x 8): one loss scale for the whole batch, as the native call uses."""
    cfg = O.RewEndCfg()
    sd = O.seeded_state_dict(O.rew_end_shapes(cfg), WSEED)
    seqs = R.trainer_sequences()
    want = R.trainer_batch_grads(seqs, sd, cfg)
    got = R.trainer_batch_grads(seqs, sd, cfg, emulated=True)
    whole, worst, e_worst, over = _budget(got, want)
    print(f"rew_end budget, trainer shape: whole {whole:.2e}, worst tensor {worst} {e_worst:.2e}")
    assert whole < 0.5 * WHOLE_BOUND and not over, (whole, over)
