"""One RewEndModel training step at the trainer's shape (b = 32, T = 19: 576 encoder rows), timed with CUDA events after a
warm-up: forward + loss, backward, clip_grad_norm_(100) and AdamW (trainer.py:361-376).  Native (diamond_b200) against an
eager torch port of the reference (oracle/torch_oracle.py encoder, nn.LSTM, TF32 on, as bench.py's reference arm), on the same
GPU; prints the card name and power limit with the times.

    python scripts/time_rew_end_train.py [--steps 20 --warmup 5]
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import torch_oracle as O  # noqa: E402
from training_oracle import rew_end as R  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


class TorchRewEnd(torch.nn.Module):
    """The reference's forward as eager torch ops on the GPU (rew_end_model.py:42-90)."""

    def __init__(self, sd, cfg):
        super().__init__()
        self.cfg = cfg
        self.p = torch.nn.ParameterDict({k.replace(".", "__"): torch.nn.Parameter(v.clone()) for k, v in sd.items()})
        self.lstm = torch.nn.LSTM(sd["lstm.weight_ih_l0"].shape[1], cfg.lstm_dim, batch_first=True)
        with torch.no_grad():
            for k in ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0"):
                getattr(self.lstm, k).copy_(sd["lstm." + k])

    def sd(self):
        return {k.replace("__", "."): v for k, v in self.p.items()}

    def forward(self, batch):
        sd, cfg = self.sd(), self.cfg
        obs, act, nxt = batch["obs"][:, :-1], batch["act"][:, :-1], batch["obs"][:, 1:]
        e, mask = batch["end"][:, :-1], batch["mask_padding"][:, :-1]
        dead = e.bool().any(dim=1)
        if dead.any():
            nxt[dead, e[dead].argmax(dim=1)] = batch["final_obs"]
        b, t, c, h, w = obs.shape
        x = O.rew_end_encoder(torch.cat((obs.reshape(b * t, c, h, w), nxt.reshape(b * t, c, h, w)), dim=1),
                              sd["act_emb.weight"][act.reshape(b * t)], sd, cfg).reshape(b, t, -1)
        y, _ = self.lstm(x)
        logits = F.linear(F.silu(F.linear(y, sd["head.0.weight"], sd["head.0.bias"])), sd["head.2.weight"])[mask]
        tr = batch["rew"][:, :-1][mask].sign().long().add(1)
        return F.cross_entropy(logits[:, :3], tr) + F.cross_entropy(logits[:, 3:], e[mask])


def time_steps(step, steps, warmup):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        step()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    from diamond_b200.models.rew_end_model import RewEndModel, RewEndModelConfig

    cfg = O.RewEndCfg()
    sd = O.seeded_state_dict(O.rew_end_shapes(cfg), 778)
    full = {k: (v.to(dev) if v is not None else None) for k, v in R.trainer_batch(R.trainer_sequences()).items()}
    dead = full["end"][:, :-1].bool().any(dim=1).tolist()
    fo = iter(full["final_obs"])
    info = [{"final_observation": next(fo)} if d else {} for d in dead]

    m = RewEndModel(RewEndModelConfig(cfg.lstm_dim, cfg.img_channels, cfg.img_size, cfg.cond_channels, list(cfg.depths), list(cfg.channels),
                                      list(cfg.attn_depths), cfg.num_actions))
    m.load_state_dict(sd)
    m = m.to(dev)
    opt = torch.optim.AdamW(m.parameters(), lr=1e-4, weight_decay=1e-2, eps=1e-8)

    class B:
        pass

    def native_step():
        bt = B()
        bt.obs, bt.act, bt.rew, bt.end, bt.mask_padding, bt.info = full["obs"].clone(), full["act"], full["rew"], full["end"], full["mask_padding"], info
        opt.zero_grad(set_to_none=True)
        loss, _ = m(bt)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(m.parameters(), 100.0)
        opt.step()

    ref = TorchRewEnd(sd, cfg).to(dev)
    ropt = torch.optim.AdamW(ref.parameters(), lr=1e-4, weight_decay=1e-2, eps=1e-8)

    def ref_step():
        batch = dict(full, obs=full["obs"].clone())
        ropt.zero_grad(set_to_none=True)
        loss = ref(batch)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(ref.parameters(), 100.0)
        ropt.step()

    t_native = time_steps(native_step, args.steps, args.warmup)
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    t_ref = time_steps(ref_step, args.steps, args.warmup)
    print(json.dumps({"card": card(), "shape": "b=32 T=19 (576 encoder rows)", "steps": args.steps, "warmup": args.warmup,
                      "native_ms_per_step": round(t_native, 3), "torch_tf32_ms_per_step": round(t_ref, 3),
                      "speedup": round(t_ref / t_native, 2)}))


if __name__ == "__main__":
    main()
