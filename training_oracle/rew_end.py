"""RewEndModel.forward (src/models/rew_end_model.py:57-90) as a loss on plain tensors, in two precisions:

* `rew_end_loss`: what the reference computes (fp32), built on torch_oracle.predict_rew_end;
* `emulated_rew_end_loss`: what the native training path computes (csrc/api.cu dmd_rew_end_forward_train / _backward), with
  the rounding rules of oracle/fp16_oracle.py: every encoder conv split-fp16 (exact) in the forward -- the training plan's
  precision plan; the inference plan keeps single-fp16 ResBlock / Downsample convs -- and in the backward fp16 dgrad / wgrad
  operands under ONE power-of-two loss scale chosen from max|dL/d(encoder output)| of the call (loss_scale_kernel).
  Attention, GroupNorm statistics (fp64), FiLM, the action embedding, the LSTM and the head are fp32.
  `split_forward=False` emulates single-fp16 forward convs (the plan this one replaced).

The difference between the two on a batch is the error budget the GPU tests are held to (DESIGN.md section 2)."""
from typing import Dict, Optional

import torch
import torch.nn.functional as F
from torch import Tensor

from oracle import fp16_oracle as E
from oracle import torch_oracle as O


def _substitute_final_obs(obs: Tensor, end: Tensor, final_obs: Optional[Tensor]):
    """rew_end_model.py:58-70: returns (obs[:, :-1], next_obs) views; the final frames are written through next_obs into
    `obs` itself, as the reference's view assignment does."""
    o, nxt, e = obs[:, :-1], obs[:, 1:], end[:, :-1]
    dead = e.bool().any(dim=1)                                             # :66
    if dead.any():
        nxt[dead, e[dead].argmax(dim=1)] = final_obs                       # :68-70
    return o, nxt


def _losses(logits_rew: Tensor, logits_end: Tensor, rew: Tensor, end: Tensor, mask_padding: Tensor):
    r, e, mask = rew[:, :-1], end[:, :-1], mask_padding[:, :-1]            # :61-63
    logits_rew, logits_end = logits_rew[mask], logits_end[mask]            # :73-74
    target_rew = r[mask].sign().long().add(1)                              # :75
    target_end = e[mask]                                                   # :76
    loss_rew = F.cross_entropy(logits_rew, target_rew)                     # :78
    loss_end = F.cross_entropy(logits_end, target_end)                     # :79
    return loss_rew + loss_end, loss_rew, loss_end, logits_rew, logits_end, target_rew, target_end   # :80


def rew_end_loss(obs: Tensor, act: Tensor, rew: Tensor, end: Tensor, mask_padding: Tensor, final_obs: Optional[Tensor], sd: O.SD,
                 cfg: O.RewEndCfg):
    """The reference's loss on the tensors of a data.Batch (obs [b, T, c, h, w]; act / rew / end / mask_padding [b, T]).
    final_obs [n_dead, c, h, w] stacks info[i]["final_observation"] of the sequences that end, in batch order (:69); it is
    written into `obs`.  Returns (loss, loss_rew, loss_end, masked logits_rew, masked logits_end, target_rew, target_end)."""
    o, nxt = _substitute_final_obs(obs, end, final_obs)
    logits_rew, logits_end, _ = O.predict_rew_end(o, act[:, :-1], nxt, sd, cfg)   # :72
    return _losses(logits_rew, logits_end, rew, end, mask_padding)


class _ScaleTap(torch.autograd.Function):
    """Identity on the encoder output; its backward records max|dL/dx| and, unless the scale was given, picks the loss scale
    of the call from it before any encoder conv's backward runs (dmd_rew_end_backward: absmax -> loss_scale_kernel)."""

    @staticmethod
    def forward(ctx, x, emu, scale):
        ctx.emu, ctx.scale = emu, scale
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        ctx.emu.gmax = float(g.abs().max())
        ctx.emu.scale = E.loss_scale(g) if ctx.scale is None else ctx.scale
        return g, None, None


def _resblock(x, cond, sd, p, emu, split):  # blocks.py:141-147; oracle/fp16_oracle.py _resblock with the conv precision as a choice
    r = E._conv(x, sd, p + "proj", emu, padding=0, split=True) if (p + "proj.weight") in sd else x
    x = E._conv(F.silu(E._ada_group_norm(x, cond, sd, p + "norm1.", emu)), sd, p + "conv1", emu, split=split)
    x = E._conv(F.silu(E._ada_group_norm(x, cond, sd, p + "norm2.", emu)), sd, p + "conv2", emu, split=split)
    x = x + r
    if (p + "attn.qkv_proj.weight") in sd:
        x = O.self_attention(x, sd, p + "attn.")
    return x


def emulated_encoder(x: Tensor, cond: Tensor, sd: O.SD, cfg: O.RewEndCfg, emu: E.Emulation, scale: Optional[float] = None,
                     split_forward: bool = True) -> Tensor:
    """rew_end_model.py:127-132 as PlanBuilder::build_rew_end lays it out for a training plan."""
    p = "encoder."
    x = E._conv(x, sd, p + "conv_in", emu, split=True)
    for i, n in enumerate(list(cfg.depths) + [2]):
        if 0 < i < len(cfg.depths):
            x = E._conv(x, sd, f"{p}downsamples.{i}.conv", emu, stride=2, split=split_forward)
        for j in range(n):
            x = _resblock(x, cond, sd, f"{p}blocks.{i}.resblocks.{j}.", emu, split_forward)
    return _ScaleTap.apply(x, emu, scale)


def emulated_rew_end_loss(obs: Tensor, act: Tensor, rew: Tensor, end: Tensor, mask_padding: Tensor, final_obs: Optional[Tensor],
                          sd: O.SD, cfg: O.RewEndCfg, emu: Optional[E.Emulation] = None, scale: Optional[float] = None,
                          split_forward: bool = True):
    """rew_end_loss as the native path computes it (see the module docstring).  During backward emu.scale becomes `scale`, or
    the call's own loss scale when it is None, and emu.gmax records max|dL/d(encoder output)|."""
    emu = emu or E.Emulation(scale=1.0)
    o, nxt = _substitute_final_obs(obs, end, final_obs)
    a = act[:, :-1]
    b, t, c, h, w = o.shape
    x = emulated_encoder(torch.cat((o.reshape(b * t, c, h, w), nxt.reshape(b * t, c, h, w)), dim=1),
                         sd["act_emb.weight"][a.reshape(b * t)], sd, cfg, emu, scale, split_forward).reshape(b, t, -1)
    hx = x.new_zeros(b, cfg.lstm_dim)
    cx = x.new_zeros(b, cfg.lstm_dim)
    outs = []
    for k in range(t):
        gates = F.linear(x[:, k], sd["lstm.weight_ih_l0"], sd["lstm.bias_ih_l0"]) + F.linear(hx, sd["lstm.weight_hh_l0"], sd["lstm.bias_hh_l0"])
        i, f, g, og = gates.chunk(4, dim=1)
        cx = torch.sigmoid(f) * cx + torch.sigmoid(i) * torch.tanh(g)
        hx = torch.sigmoid(og) * torch.tanh(cx)
        outs.append(hx)
    y = torch.stack(outs, dim=1)
    logits = F.linear(F.silu(F.linear(y, sd["head.0.weight"], sd["head.0.bias"])), sd["head.2.weight"])
    return _losses(logits[:, :, :3], logits[:, :, 3:], rew, end, mask_padding)


def parameter_grads(batch: Dict[str, Tensor], sd: O.SD, cfg: O.RewEndCfg, emulated: bool = False, scale: Optional[float] = None,
                    emu: Optional[E.Emulation] = None, split_forward: bool = True) -> Dict[str, Tensor]:
    """Gradients of the loss with respect to every parameter, fp32 oracle or emulation (`scale`: see emulated_rew_end_loss).
    batch: obs / act / rew / end / mask_padding / final_obs (final_obs may be None); obs is copied, so the caller's tensor
    keeps its frames."""
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items()}
    args = (batch["obs"].clone(), batch["act"], batch["rew"], batch["end"], batch["mask_padding"], batch.get("final_obs"), sd, cfg)
    loss = (emulated_rew_end_loss(*args, emu=emu or E.Emulation(scale=1.0), scale=scale, split_forward=split_forward) if emulated
            else rew_end_loss(*args))[0]
    loss.backward()
    return {k: v.grad for k, v in sd.items()}


# ----------------------------------------------------------------------------------------------- the trainer's batch shape
# trainer.yaml:106-116: b = 32 sequences of seq_length = 19 frames (18 steps: 576 encoder rows per training step).  The batch repeats 4
# distinct sequences 8 times each, so its gradient is a count-weighted sum of 4 single-sequence oracle passes.
TRAINER_B, TRAINER_T, TRAINER_REPEAT = 32, 19, 8


def trainer_sequences(seed: int = 4242):
    """4 single-sequence batches (b = 1, T = 19): dies mid-sequence then padding, dies on its last step, masked tail without
    death, plain.  Rewards in {-1, 0, 2}."""
    rng = torch.Generator().manual_seed(seed)
    T, seqs = TRAINER_T, []
    for kind in range(4):
        obs = torch.randint(0, 256, (1, T, 3, 64, 64), generator=rng).float().div(255).mul(2).sub(1)
        act = torch.randint(0, O.RewEndCfg().num_actions, (1, T), generator=rng)
        rew = torch.tensor([-1.0, 0.0, 0.0, 2.0])[torch.randint(0, 4, (1, T), generator=rng)]
        end = torch.zeros(1, T, dtype=torch.long)
        mask = torch.ones(1, T, dtype=torch.bool)
        final_obs = None
        if kind == 0:
            end[0, 9] = 1; mask[0, 10:] = False; obs[0, 11:] = 0.0; rew[0, 10:] = 0.0
        elif kind == 1:
            end[0, T - 2] = 1
        elif kind == 2:
            mask[0, 12:] = False
        if kind < 2:
            final_obs = torch.randint(0, 256, (1, 3, 64, 64), generator=rng).float().div(255).mul(2).sub(1)
        seqs.append(dict(obs=obs, act=act, rew=rew, end=end, mask_padding=mask, final_obs=final_obs))
    return seqs


def trainer_batch(seqs):
    """The b = 32 batch: sequence n is seqs[n % 4]; final_obs stacked in batch order, as the reference stacks info[i]."""
    idx = [n % len(seqs) for n in range(TRAINER_B)]
    out = {k: torch.cat([seqs[i][k] for i in idx]) for k in ("obs", "act", "rew", "end", "mask_padding")}
    out["final_obs"] = torch.cat([seqs[i]["final_obs"] for i in idx if seqs[i]["final_obs"] is not None])
    return out


def selected_rows(seq) -> int:
    return int(seq["mask_padding"][:, :-1].sum())


def trainer_batch_grads(seqs, sd: O.SD, cfg: O.RewEndCfg, emulated: bool = False) -> Dict[str, Tensor]:
    """Gradient of the trainer_batch loss: sum over the distinct sequences of (copies * selected rows / all selected rows) x
    that sequence's own gradient (both cross-entropies are means over the batch's selected rows).  Emulated: the call's one
    loss scale comes from the largest feature gradient of the whole batch, found by a first pass per sequence."""
    n = [selected_rows(s) for s in seqs]
    total = TRAINER_REPEAT * sum(n)
    w = [TRAINER_REPEAT * ni / total for ni in n]
    scales = [None] * len(seqs)
    if emulated:
        gmax = []
        for s in seqs:
            emu = E.Emulation(scale=1.0)
            parameter_grads(s, sd, cfg, emulated=True, emu=emu)
            gmax.append(emu.gmax)
        S = E.loss_scale(torch.tensor([ni / total * g for ni, g in zip(n, gmax)]))
        scales = [S * ni / total for ni in n]   # (S * batch gradient) in the units of the sequence's own gradient
    out = None
    for s, wi, sc in zip(seqs, w, scales):
        g = parameter_grads(s, sd, cfg, emulated=emulated, scale=sc)
        out = {k: wi * v for k, v in g.items()} if out is None else {k: out[k] + wi * v for k, v in g.items()}
    return out
