"""Imagined-rollout driver for the actor-critic update: drop-in for the generator the reference builds with
`make_env_loop` (src/coroutines/env_loop.py:12-74) — same `.send(num_steps)` protocol, same 9-tuple, same results bit for
bit (tests/test_env_host_logic.py checks it against the reference's recorded outputs), different mechanics:

* results are written into tensors preallocated for the whole rollout instead of per-step lists that are stacked;
* the bootstrap values are assembled once at the end with a single `where` over (dead, V(final obs), V(next obs)) instead of
  being patched step by step;
* one device->host synchronisation per step (`dead.any()`), where the reference pays three.

The arithmetic lives in `model.predict_act_value` (native actor-critic, autograd node per call) and `env.step` (native
sampler)."""
import random
from typing import Any, Dict, List, Tuple

import torch
from torch.distributions.categorical import Categorical


class ImaginationLoop:
    def __init__(self, env, model, epsilon: float = 0.0) -> None:
        self.env, self.model, self.epsilon = env, model, epsilon
        self._obs = None
        self._hx = self._cx = None

    def _start(self) -> None:
        n, dev = self.env.num_envs, self.model.device
        self._hx = torch.zeros(n, self.model.lstm_dim, device=dev)
        self._cx = torch.zeros(n, self.model.lstm_dim, device=dev)
        seed = random.randint(0, 2**31 - 1)                      # env_loop.py:21: python RNG stream kept
        self._obs, _ = self.env.reset(seed=[seed + i for i in range(n)])

    def send(self, num_steps: int) -> Tuple[Any, ...]:
        if self._obs is None:
            self._start()
        model, env = self.model, self.env
        obs, hx, cx = self._obs, self._hx.detach(), self._cx.detach()   # truncated BPTT across updates (env_loop.py:25)
        b, dev = obs.size(0), obs.device
        all_obs = obs.new_empty(b, num_steps, *obs.shape[1:])
        acts = torch.empty(b, num_steps, dtype=torch.long, device=dev)
        rews = ends = truncs = None
        logits_steps: List[torch.Tensor] = []
        val_steps: List[torch.Tensor] = []
        v_next = torch.empty(b, num_steps, device=dev)            # V(obs_{t+1}) without gradient
        v_final = torch.zeros(b, num_steps, device=dev)           # V(final observation) where an episode ended at t
        died = torch.zeros(b, num_steps, dtype=torch.bool, device=dev)
        infos: List[Dict[str, Any]] = []
        for t in range(num_steps):
            logits, val, (hx, cx) = model.predict_act_value(obs, (hx, cx))
            act = Categorical(logits=logits, validate_args=False).sample()   # validate_args costs a device->host sync per call
            if random.random() < self.epsilon:                    # drawn every step, like the reference (env_loop.py:34)
                act = torch.randint(low=0, high=env.num_actions, size=(b,), device=dev)
            nxt, rew, end, trunc, info = env.step(act)
            if rews is None:
                rews = torch.empty(b, num_steps, dtype=rew.dtype, device=dev)
                ends = torch.empty(b, num_steps, dtype=end.dtype, device=dev)
                truncs = torch.empty(b, num_steps, dtype=trunc.dtype, device=dev)
            if t > 0:
                v_next[:, t - 1] = val.detach()
            dead = torch.logical_or(end, trunc)
            if bool(dead.any()):                                  # the step's only host sync
                with torch.no_grad():
                    _, v_fin, _ = model.predict_act_value(info["final_observation"], (hx[dead], cx[dead]))
                v_final[dead, t] = v_fin
                died[:, t] = dead
                keep = 1 - dead.float().unsqueeze(1)              # recurrent state of finished episodes restarts at zero
                hx, cx = hx * keep, cx * keep
                if "burnin_obs" in info:                          # ... and is burnt in on the new episode's context frames
                    ctx = info["burnin_obs"]
                    for i in range(ctx.size(1)):
                        _, _, (hx[dead], cx[dead]) = model.predict_act_value(ctx[:, i], (hx[dead], cx[dead]))
            all_obs[:, t], acts[:, t], rews[:, t], ends[:, t], truncs[:, t] = obs, act, rew, end, trunc
            logits_steps.append(logits)
            val_steps.append(val)
            infos.append(info)
            obs = nxt
        with torch.no_grad():                                     # bootstrap value of the last next_obs; hx/cx not advanced
            _, v_last, _ = model.predict_act_value(obs, (hx, cx))
        v_next[:, num_steps - 1] = v_last
        val_bootstrap = torch.where(died, v_final, v_next)
        self._obs, self._hx, self._cx = obs, hx, cx
        return (all_obs, acts, rews, ends, truncs, torch.stack(logits_steps, dim=1), torch.stack(val_steps, dim=1), val_bootstrap, infos)


def make_env_loop(env, model, epsilon: float = 0.0) -> ImaginationLoop:
    """Same call as the reference's coroutine factory (env_loop.py:12-15); the returned object answers `.send(num_steps)`."""
    return ImaginationLoop(env, model, epsilon)
