"""WorldModelEnv: the batched imagined environment of the actor-critic phase (reference surface:
src/envs/world_model_env.py:25-139 — same constructor, `reset` / `step` / `predict_next_obs` / `predict_rew_end`, same
results given the same RNG streams; tests/test_env_host_logic.py checks the index work bit for bit against the reference's
recorded outputs).  The mechanics are B200-first:

* the frame stack and the action stack are DEVICE-RESIDENT RINGS (`_frames` (T, B, C, H, W), `_acts` (T, B)); the
  reference's two `roll` copies per step (world_model_env.py:74-75) are an index increment, and the native sampler reads the
  ring in place and writes the new frame straight into the slot that just became free (one CUDA graph per ring head);
* initial conditions are preloaded into one pool per refill and handed out by slicing, instead of python lists of
  per-sample tensors that are re-stacked on every reset;
* `obs_buffer` / `act_buffer` remain available as properties that materialise the logical (oldest -> newest) order.
"""
from dataclasses import dataclass
from typing import Any, Dict, List, Optional, Tuple

import torch
from torch import Tensor
from torch.distributions.categorical import Categorical

from ..models.diffusion import Denoiser, DiffusionSampler, DiffusionSamplerConfig

ResetOutput = Tuple[torch.FloatTensor, Dict[str, Any]]
StepOutput = Tuple[Tensor, Tensor, Tensor, Tensor, Dict[str, Any]]


@dataclass
class WorldModelEnvConfig:  # world_model_env.py:18-22
    horizon: int
    num_batches_to_preload: int
    diffusion_sampler: DiffusionSamplerConfig


class _InitialConditionPool:
    """Fresh episodes for dead environments (world_model_env.py:107-139): real segments are preloaded
    `num_batches_to_preload` batches at a time, the reward/termination LSTM is burnt in on each batch, and requests for `k`
    initial conditions are served in order; what is left when a request does not fit is dropped and the pool is refilled
    (the reference's generator does exactly this)."""

    def __init__(self, env: "WorldModelEnv", data_loader, num_batches: int) -> None:
        self.env, self.num_batches = env, num_batches
        self.batches = iter(data_loader)
        self.obs = self.act = self.hx = self.cx = None
        self.cursor = 0

    def _refill(self) -> None:
        env = self.env
        obs_, act_, hx_, cx_ = [], [], [], []
        for _ in range(self.num_batches):
            batch = next(self.batches)
            obs, act = batch.obs.to(env.device), batch.act.to(env.device)
            with torch.no_grad():
                *_, (hx, cx) = env.rew_end_model.predict_rew_end(obs[:, :-1], act[:, :-1], obs[:, 1:])
            assert hx.size(0) == cx.size(0) == 1
            obs_.append(obs); act_.append(act); hx_.append(hx[0]); cx_.append(cx[0])
        self.obs, self.act, self.hx, self.cx = (torch.cat(v) for v in (obs_, act_, hx_, cx_))
        self.cursor = 0

    def take(self, k: int):
        if self.obs is None or self.cursor + k > self.obs.size(0):
            self._refill()
            while k > self.obs.size(0):   # a request larger than one refill can never be served by the reference either
                self._refill()
        sl = slice(self.cursor, self.cursor + k)
        self.cursor += k
        return self.obs[sl], self.act[sl], (self.hx[sl].unsqueeze(0), self.cx[sl].unsqueeze(0))


class WorldModelEnv:
    def __init__(self, denoiser: Denoiser, rew_end_model, data_loader, cfg: WorldModelEnvConfig,
                 return_denoising_trajectory: bool = False) -> None:
        self.sampler = DiffusionSampler(denoiser, cfg.diffusion_sampler)
        self.rew_end_model = rew_end_model
        self.horizon = cfg.horizon
        self.return_denoising_trajectory = return_denoising_trajectory
        self.num_envs = data_loader.batch_sampler.batch_size
        self._pool = _InitialConditionPool(self, data_loader, cfg.num_batches_to_preload)
        self._frames: Optional[Tensor] = None   # (T, B, C, H, W) ring, logical slot k at physical (head + k) % T
        self._acts: Optional[Tensor] = None     # (T, B) ring
        self._head = 0
        self._use_ring_sampler = hasattr(self.sampler, "sample_ring")

    @property
    def device(self) -> torch.device:
        return self.sampler.denoiser.device

    # ------------------------------------------------------------------ ring helpers
    def _slot(self, k: int) -> int:
        return (self._head + k) % self._frames.size(0)

    def _order(self) -> List[int]:
        t = self._frames.size(0)
        return [(self._head + k) % t for k in range(t)]

    @property
    def obs_buffer(self) -> Tensor:   # (B, T, C, H, W), oldest -> newest, like the reference attribute
        return self._frames[self._order()].transpose(0, 1)

    @property
    def act_buffer(self) -> Tensor:   # (B, T)
        return self._acts[self._order()].transpose(0, 1)

    def _write_stacks(self, rows, obs: Tensor, act: Tensor) -> None:
        """frames / actions of the environments `rows` (bool mask or slice) <- logical stacks obs (k, T, C, H, W), act (k, T)."""
        for k in range(self._frames.size(0)):
            p = self._slot(k)
            self._frames[p, rows] = obs[:, k]
            self._acts[p, rows] = act[:, k]

    # ------------------------------------------------------------------ reference surface
    @torch.no_grad()
    def reset(self, **kwargs) -> ResetOutput:  # world_model_env.py:45-53
        obs, act, (hx, cx) = self._pool.take(self.num_envs)
        b, t = obs.shape[:2]
        self._frames = obs.new_empty(t, b, *obs.shape[2:])
        self._acts = act.new_empty(t, b)
        self._head = 0
        self._write_stacks(slice(None), obs, act)
        self.hx_rew_end, self.cx_rew_end = hx.clone(), cx.clone()
        self.ep_len = torch.zeros(self.num_envs, dtype=torch.long, device=obs.device)
        return self._frames[self._slot(t - 1)].clone(), {}

    @torch.no_grad()
    def reset_dead(self, dead: torch.BoolTensor) -> None:  # world_model_env.py:55-62
        obs, act, (hx, cx) = self._pool.take(int(dead.sum().item()))
        self._write_stacks(dead, obs, act)
        self.hx_rew_end[:, dead] = hx
        self.cx_rew_end[:, dead] = cx
        self.ep_len[dead] = 0

    @torch.no_grad()
    def step(self, act: torch.LongTensor) -> StepOutput:  # world_model_env.py:64-89
        t = self._frames.size(0)
        self._acts[self._slot(t - 1)] = act
        next_obs, denoising_trajectory = self.predict_next_obs()
        rew, end = self.predict_rew_end(next_obs.unsqueeze(1))

        self.ep_len += 1
        trunc = (self.ep_len >= self.horizon).long()

        # the reference rolls both buffers by one and writes next_obs last: here the oldest slot becomes the newest
        free = self._head
        self._head = (self._head + 1) % t
        if next_obs.data_ptr() != self._frames[free].data_ptr():
            self._frames[free] = next_obs
        # the action slot that became "newest" keeps the oldest action until the next step overwrites it -- as after the
        # reference's roll, where act_buffer[:, -1] holds the rolled-around oldest action

        dead = torch.logical_or(end, trunc)
        info: Dict[str, Any] = {}
        if self.return_denoising_trajectory:
            info["denoising_trajectory"] = torch.stack(list(denoising_trajectory), dim=1)
        if dead.any():
            final = self._frames[free][dead]            # copy (boolean indexing) before the dead envs are re-initialised
            self.reset_dead(dead)
            info["final_observation"] = final
            info["burnin_obs"] = self.obs_buffer[dead, :-1]
        # the returned observation must stay valid while later steps re-initialise dead environments in the ring: hand out a copy
        # (the reference's per-step roll made two full copies of both buffers; this is one frame)
        return self._frames[free].clone(), rew, end, trunc, info

    # kept as plain re-bindable methods: trainer.py:183-184 may wrap them
    @torch.no_grad()
    def predict_next_obs(self) -> Tuple[Tensor, List[Tensor]]:  # world_model_env.py:91-93
        if self._use_ring_sampler and "sample" not in self.sampler.__dict__:
            # native path: the sampler reads the ring in place; the new frame lands in the slot that is about to be freed.
            # It is still logical slot 0 (read by every denoising step) -- the final Euler update writes it last, in stream order.
            traj = self.sampler.sample_ring(self._frames, self._acts, self._head, self._frames[self._head])
            return self._frames[self._head], traj.unbind(0)
        return self.sampler.sample(self.obs_buffer, self.act_buffer)

    @torch.no_grad()
    def predict_rew_end(self, next_obs: Tensor) -> Tuple[Tensor, Tensor]:  # world_model_env.py:95-105
        t = self._frames.size(0)
        last = self._slot(t - 1)
        logits_rew, logits_end, (self.hx_rew_end, self.cx_rew_end) = self.rew_end_model.predict_rew_end(
            self._frames[last].unsqueeze(1), self._acts[last].unsqueeze(1), next_obs, (self.hx_rew_end, self.cx_rew_end))
        rew = Categorical(logits=logits_rew, validate_args=False).sample().squeeze(1) - 1.0  # {-1, 0, 1}
        end = Categorical(logits=logits_end, validate_args=False).sample().squeeze(1)
        return rew, end
