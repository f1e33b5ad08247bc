"""Writes tests/golden/rew_end_training.npz by running the UNMODIFIED reference RewEndModel.forward + backward (imported by
oracle/ref_import.py, torcheval stubbed) on seeded weights and a small batch that covers the final-frame substitution:

    python training_oracle/make_rew_end_golden.py

Batch: b = 4 sequences of T = 6 frames (5 steps): one dies mid-sequence and is followed by padding, one dies on its last step,
one has a masked tail without death, one is plain; rewards are drawn from {-1, 0, 2}.  The stub confusion matrix returns
nothing, so the fixture records the masked logits (the tests count the matrices from them); the data seed is the first one
whose masked logits all have a top-2 margin that a GPU's error cannot flip."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_import  # noqa: E402
from oracle import torch_oracle as O  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "rew_end_training.npz")
WSEED = 778
B, T = 4, 6
MIN_MARGIN = 0.05   # top-2 logit gap, in units of the masked logits' rms


def batch_tensors(seed: int):
    """(obs, act, rew, end, mask_padding, final_obs) of the fixture's batch for one data seed."""
    rng = np.random.default_rng(seed)
    obs = torch.from_numpy(rng.integers(0, 256, size=(B, T, 3, 64, 64)).astype(np.float32)).div(255).mul(2).sub(1)
    act = torch.from_numpy(rng.integers(0, O.RewEndCfg().num_actions, size=(B, T)).astype(np.int64))
    rew = torch.from_numpy(rng.choice([-1.0, 0.0, 0.0, 2.0], size=(B, T)).astype(np.float32))
    end = torch.zeros(B, T, dtype=torch.long)
    mask = torch.ones(B, T, dtype=torch.bool)
    end[0, 2] = 1; mask[0, 3:] = False; obs[0, 4:] = 0.0; rew[0, 3:] = 0.0   # dies at step 2, then padding
    end[1, T - 2] = 1                                                        # dies on its last step
    mask[2, 3:] = False                                                      # masked tail, no death
    final_obs = torch.from_numpy(rng.integers(0, 256, size=(2, 3, 64, 64)).astype(np.float32)).div(255).mul(2).sub(1)
    return obs, act, rew, end, mask, final_obs


def main():
    ns = ref_import.load()
    R = ns.rew_end_model
    cfg = O.RewEndCfg()
    sd = O.seeded_state_dict(O.rew_end_shapes(cfg), WSEED)
    torch.set_num_threads(8)
    for dseed in range(200, 300):
        m = R.RewEndModel(R.RewEndModelConfig(cfg.lstm_dim, cfg.img_channels, cfg.img_size, cfg.cond_channels, list(cfg.depths),
                                              list(cfg.channels), list(cfg.attn_depths), cfg.num_actions))
        assert [(k, tuple(v.shape)) for k, v in m.state_dict().items()] == O.rew_end_shapes(cfg)
        m.load_state_dict(sd)
        obs, act, rew, end, mask, final_obs = batch_tensors(dseed)
        obs_in = obs.clone()
        info = [{"final_observation": final_obs[0]}, {"final_observation": final_obs[1]}, {}, {}]
        batch = ns.data.Batch(obs=obs, act=act, rew=rew, end=end, trunc=torch.zeros_like(end), mask_padding=mask, info=info,
                              segment_ids=[None] * B)
        captured = {}
        real = m.predict_rew_end

        def tap(*a, **k):
            out = real(*a, **k)
            captured["logits"] = out[:2]
            return out
        m.predict_rew_end = tap
        loss, metrics = m(batch)
        mk = mask[:, :-1]
        lr, le = (x.detach()[mk] for x in captured["logits"])
        rms = float(torch.cat((lr.flatten(), le.flatten())).pow(2).mean().sqrt())
        margin = min(float((x.topk(2, dim=1).values[:, 0] - x.topk(2, dim=1).values[:, 1]).min()) for x in (lr, le)) / rms
        if margin < MIN_MARGIN:
            continue
        loss.backward()
        grads = [(k, p.grad) for k, p in m.named_parameters()]
        assert all(g is not None for _, g in grads)
        keys, norms, samples = O.grad_summary(grads)
        np.savez_compressed(OUT, weights_checksum=np.float64(O.state_checksum(sd)), data_seed=np.int64(dseed), obs=obs_in.numpy(),
                            act=act.numpy(), rew=rew.numpy(), end=end.numpy(), mask_padding=mask.numpy(), final_obs=final_obs.numpy(),
                            obs_after=batch.obs.numpy(), loss=np.float64(loss.item()), loss_rew=np.float64(metrics["loss_rew"].item()),
                            loss_end=np.float64(metrics["loss_end"].item()), logits_rew=lr.numpy(), logits_end=le.numpy(),
                            grad_keys=np.array(keys), grad_norms=norms, grad_samples=samples)
        print("rew_end_training data seed", dseed, "loss", loss.item(), "margin/rms", margin, "grad norm",
              float(np.sqrt((norms ** 2).sum())), "size", os.path.getsize(OUT))
        return
    raise RuntimeError("no data seed gives a large enough logit margin")


if __name__ == "__main__":
    main()
