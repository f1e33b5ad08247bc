"""GPU: native RewEndModel.forward + loss.backward() (rew_end_model.py:57-90; dmd_rew_end_forward_train / dmd_rew_end_backward)
against the reference's fixture (tests/golden/rew_end_training.npz) and the fp32 oracle (training_oracle/rew_end.py), at the
fixture's shape and at the trainer's (b = 32, T = 19).  Bounds: loss within 2e-3; whole gradient (relative L2 over all
parameters) < 1e-3; every tensor < 4e-3 or a negligible share of the whole (e * n < 1e-4 * total, the rule of
test_gpu_training.py); per-tensor norms vs the fixture within 4e-3 * ref + 1e-4 * total.  The CPU error budget of this
precision plan is 3.3e-4 whole (tests/test_oracle_rew_end_training_golden.py)."""
import ctypes as C
import os
import types

import numpy as np
import pytest
import torch

from oracle import torch_oracle as O
from training_oracle import rew_end as R

pytestmark = pytest.mark.gpu
WSEED = 778


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    return torch.device("cuda:0")


def _model(dev, sd=None):
    from diamond_b200.models.rew_end_model import RewEndModel, RewEndModelConfig

    cfg = O.RewEndCfg()
    m = RewEndModel(RewEndModelConfig(cfg.lstm_dim, cfg.img_channels, cfg.img_size, cfg.cond_channels, list(cfg.depths), list(cfg.channels),
                                      list(cfg.attn_depths), cfg.num_actions))
    m.load_state_dict(sd if sd is not None else O.seeded_state_dict(O.rew_end_shapes(cfg), WSEED))
    return m.to(dev)


def _batch(t, dev):
    """A data.Batch-like object on the device; info carries the final observations of the dead sequences, in batch order."""
    dead = t["end"][:, :-1].bool().any(dim=1)
    fo = iter(t["final_obs"]) if t.get("final_obs") is not None else iter(())
    info = [{"final_observation": next(fo).to(dev)} if d else {} for d in dead]
    return types.SimpleNamespace(obs=t["obs"].clone().to(dev), act=t["act"].to(dev), rew=t["rew"].to(dev), end=t["end"].to(dev),
                                 mask_padding=t["mask_padding"].to(dev), info=info)


def _fixture():
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rew_end_training.npz"))
    return g, {k: torch.from_numpy(g[k]) for k in ("obs", "act", "rew", "end", "mask_padding", "final_obs")}


def _errors(model, want):
    got = {k: p.grad.detach().double().cpu() for k, p in model.named_parameters()}
    want = {k: v.double() for k, v in want.items()}
    total = sum(float(w.pow(2).sum()) for w in want.values()) ** 0.5
    whole = sum(float((got[k] - want[k]).pow(2).sum()) for k in want) ** 0.5 / total
    per = {k: float((got[k] - want[k]).norm() / want[k].norm().clamp_min(1e-300)) for k in want}
    bad = {k: e for k, e in per.items() if e >= 4e-3 and e * float(want[k].norm()) >= 1e-4 * total}
    worst = max(per, key=per.get)
    return whole, worst, per[worst], bad, got, total


def test_fixture_loss_gradients_and_metrics():
    dev = _dev()
    g, t = _fixture()
    m = _model(dev)
    batch = _batch(t, dev)
    loss, metrics = m(batch)
    loss.backward()
    for got, key in ((loss, "loss"), (metrics["loss_rew"], "loss_rew"), (metrics["loss_end"], "loss_end")):
        assert abs(got.item() - float(g[key])) <= 2e-3 * abs(float(g[key])), (key, got.item(), float(g[key]))
    assert torch.equal(batch.obs.cpu(), torch.from_numpy(g["obs_after"]))
    mask = t["mask_padding"][:, :-1]
    targets = {"rew": t["rew"][:, :-1][mask].sign().long().add(1), "end": t["end"][:, :-1][mask]}
    for key, n in (("rew", 3), ("end", 2)):
        ref = torch.bincount(targets[key] * n + torch.from_numpy(g["logits_" + key]).argmax(1), minlength=n * n).reshape(n, n)
        cm = metrics["confusion_matrix"][key]
        assert cm.dtype == torch.int64 and torch.equal(cm.cpu(), ref), key
    sd = O.seeded_state_dict(O.rew_end_shapes(O.RewEndCfg()), WSEED)
    want = R.parameter_grads(t, sd, O.RewEndCfg())
    whole, worst, e_worst, bad, got, total = _errors(m, want)
    print(f"rew_end fixture: loss {loss.item():.6f} (ref {float(g['loss']):.6f}); whole {whole:.2e}; worst {worst} {e_worst:.2e}")
    assert whole < 1e-3 and not bad, (whole, bad)
    keys, norms, _ = O.grad_summary(list(got.items()))
    ref_n = g["grad_norms"]
    assert keys == [str(k) for k in g["grad_keys"]]
    tot = float(np.sqrt((ref_n ** 2).sum()))
    assert np.all(np.abs(norms - ref_n) <= 4e-3 * ref_n + 1e-4 * tot)


def test_trainer_shape_gradients():
    dev = _dev()
    cfg = O.RewEndCfg()
    sd = O.seeded_state_dict(O.rew_end_shapes(cfg), WSEED)
    seqs = R.trainer_sequences()
    full = R.trainer_batch(seqs)
    m = _model(dev, sd)
    loss, _ = m(_batch(full, dev))
    loss.backward()
    with torch.no_grad():
        ref_loss = R.rew_end_loss(full["obs"].clone(), full["act"], full["rew"], full["end"], full["mask_padding"], full["final_obs"], sd, cfg)[0]
    want = R.trainer_batch_grads(seqs, sd, cfg)
    whole, worst, e_worst, bad, _, _ = _errors(m, want)
    print(f"rew_end trainer shape (b=32, T=19): loss {loss.item():.6f} (oracle {ref_loss.item():.6f}); whole {whole:.2e}; "
          f"worst {worst} {e_worst:.2e}")
    assert abs(loss.item() - ref_loss.item()) <= 2e-3 * abs(ref_loss.item())
    assert whole < 1e-3 and not bad, (whole, bad)


def _rel(a, b):
    return float((a - b).norm() / b.norm())


def test_inference_unaffected_and_two_adamw_steps():
    dev = _dev()
    g, t = _fixture()
    cfg = O.RewEndCfg()
    m = _model(dev)
    obs, act = t["obs"].to(dev), t["act"].to(dev)

    def predict():
        lr, le, (hx, cx) = m.predict_rew_end(obs[:, :-1], act[:, :-1], obs[:, 1:])
        return [x.clone() for x in (lr, le, hx, cx)]
    before = predict()
    loss0, _ = m(_batch(t, dev))
    loss0.backward()
    after = predict()
    assert max(_rel(a, b) for a, b in zip(after, before)) < 1e-4
    opt = torch.optim.AdamW(m.parameters(), lr=3e-4, weight_decay=1e-2)
    losses = [loss0.item()]
    opt.step()
    opt.zero_grad()
    loss1, _ = m(_batch(t, dev))
    loss1.backward()
    losses.append(loss1.item())
    opt.step()
    assert losses[1] < losses[0], losses
    with torch.no_grad():
        loss2, _ = m(_batch(t, dev))
    losses.append(loss2.item())
    assert losses[2] < losses[1], losses
    sd2 = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    lr, le, _ = O.predict_rew_end(t["obs"][:, :-1], t["act"][:, :-1], t["obs"][:, 1:], sd2, cfg)
    got = predict()
    print("rew_end losses over two AdamW steps:", losses, "predict vs oracle after:", _rel(got[0].cpu(), lr), _rel(got[1].cpu(), le))
    assert _rel(got[0].cpu(), lr) < 2e-3 and _rel(got[1].cpu(), le) < 2e-3


def test_autograd_semantics():
    dev = _dev()
    _, t = _fixture()
    m = _model(dev)
    loss, _ = m(_batch(t, dev))
    loss.backward()
    flat = m.last_flat_grad
    lo, hi = flat.data_ptr(), flat.data_ptr() + flat.numel() * 4
    assert all(lo <= p.grad.data_ptr() < hi for p in m.parameters())
    once = {k: p.grad.clone() for k, p in m.named_parameters()}
    offs, nums, _ = m.grad_layout()
    index = {k: i for i, k in enumerate(m.state_dict().keys())}
    loss, _ = m(_batch(t, dev))
    loss.backward()
    second = {k: m.last_flat_grad[offs[index[k]]:offs[index[k]] + nums[index[k]]].view_as(p) for k, p in m.named_parameters()}
    # the second pass ADDS to .grad (AccumulateGrad): to fp32 order.  The two passes themselves agree to fp16 noise only: the
    # GroupNorm sums are fp64 atomics, and a last-ulp difference can flip an fp16 rounding downstream (DESIGN.md section 2)
    for k, p in m.named_parameters():
        assert torch.allclose(p.grad, once[k] + second[k], rtol=1e-5, atol=1e-7 * float(once[k].abs().max())), k
    rerun = max(_rel(second[k], once[k]) for k in once if once[k].norm() > 0)
    print(f"rew_end: two identical training passes differ by at most {rerun:.2e} per tensor")
    assert rerun < 4e-3
    m.zero_grad(set_to_none=True)
    pool = m.__dict__.get("_tws_pool", [])
    n_pool = len(pool)
    with torch.no_grad():
        l_ng, metrics = m(_batch(t, dev))
    assert len(m.__dict__.get("_tws_pool", [])) == n_pool and not l_ng.requires_grad
    # without autograd the call runs predict_rew_end on the inference plan, whose ResBlock / Downsample convs read single-fp16
    # operands (the training plan's are split-fp16): the same loss to that precision (measured 1.3e-5 relative)
    assert abs(l_ng.item() - loss.item()) <= 2e-4 * abs(loss.item())
    assert all(p.grad is None for p in m.parameters())


def test_rejections_fail_loudly():
    dev = _dev()
    from diamond_b200 import _lib

    lib = _lib.lib()
    m = _model(dev)
    h = m._native()
    b, t = 2, 3
    g_rew, g_end = torch.zeros(b, t, 3, device=dev), torch.zeros(b, t, 2, device=dev)
    offs, nums, total = m.grad_layout()
    flat = torch.empty(total, device=dev)
    need = lib.dmd_rew_end_train_workspace_bytes(h, b, t)
    assert need > 0
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    with pytest.raises(RuntimeError, match="no matching dmd_rew_end_forward_train"):
        _lib.check(lib.dmd_rew_end_backward(h, b, t, g_rew.data_ptr(), g_end.data_ptr(), flat.data_ptr(), total, ws.data_ptr(),
                                            _lib.current_stream()))
    obs = torch.zeros(b, t, 3, 64, 64, device=dev)
    act = torch.zeros(b, t, dtype=torch.long, device=dev)
    small = torch.empty(need // 2, dtype=torch.uint8, device=dev)
    with pytest.raises(RuntimeError, match="workspace too small"):
        _lib.check(lib.dmd_rew_end_forward_train(h, b, t, obs.data_ptr(), obs.data_ptr(), act.data_ptr(), g_rew.data_ptr(), g_end.data_ptr(),
                                                 small.data_ptr(), small.numel(), _lib.current_stream()))
    with pytest.raises(RuntimeError, match="b and t must be positive"):
        _lib.check(lib.dmd_rew_end_forward_train(h, b, 0, obs.data_ptr(), obs.data_ptr(), act.data_ptr(), g_rew.data_ptr(), g_end.data_ptr(),
                                                 ws.data_ptr(), ws.numel(), _lib.current_stream()))
    assert lib.dmd_rew_end_train_workspace_bytes(h, b, 0) == 0 and b"positive" in lib.dmd_last_error()
    wrong = types.SimpleNamespace(obs=torch.zeros(b, t + 1, 3, 32, 32, device=dev), act=torch.zeros(b, t + 1, dtype=torch.long, device=dev),
                                  rew=torch.zeros(b, t + 1, device=dev), end=torch.zeros(b, t + 1, dtype=torch.long, device=dev),
                                  mask_padding=torch.ones(b, t + 1, dtype=torch.bool, device=dev), info=[{}] * b)
    with pytest.raises(RuntimeError, match="img_size"):
        m(wrong)
    assert lib.dmd_rew_end_grad_layout(h, None, None, 3) == -1 and b"expected" in lib.dmd_last_error()
