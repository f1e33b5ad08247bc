"""CPU: index / buffer logic of the WorldModelEnv and env-loop mirrors must be BIT-EXACT against the reference
(SURVEY.md 8 a20/a24), driven by identical fake networks and identical RNG streams.  What the unmodified reference returned
under these fakes is stored in tests/golden/env_host_logic.npz (oracle/make_golden.py runs the helpers below on it): the
env-loop outputs and lambda returns in full, and the 401 tensors of the 40-step WorldModelEnv run as digests (dtype, shape,
SHA-256 of the bytes), which keeps the fixture small.  The oracle-free invariants at the end need no fixture."""
import hashlib
import os
import random
from types import SimpleNamespace

import numpy as np
import torch

from diamond_b200.coroutines.env_loop import make_env_loop
from diamond_b200.envs import world_model_env as mine
from diamond_b200.models.actor_critic import compute_lambda_returns

LAMBDAS = (0.0, 0.95)


class FakeDenoiser:
    device = torch.device("cpu")
    cfg = SimpleNamespace(sigma_data=0.5, sigma_offset_noise=0.3)


class FakeRewEnd:
    """Deterministic stand-in for RewEndModel.predict_rew_end: logits depend on the inputs, hidden state evolves."""

    def predict_rew_end(self, obs, act, next_obs, hx_cx=None):
        b, t = obs.shape[:2]
        feat = obs.flatten(2).mean(-1) + 0.5 * next_obs.flatten(2).mean(-1) + 0.1 * act.float()
        if hx_cx is None:
            hx = torch.zeros(1, b, 4); cx = torch.zeros(1, b, 4)
        else:
            hx, cx = hx_cx
        hx = hx + feat.sum(1)[None, :, None]
        cx = cx * 0.5 + 1
        logits_rew = torch.stack([feat, -feat, feat * 0.3], -1) * 3 + hx[0, :, :1, None].transpose(1, 2) * 0.01
        logits_end = torch.stack([feat * 0 + 1.2, feat * 4], -1)
        return logits_rew, logits_end, (hx, cx)


class Loader:
    def __init__(self, b, t, seed):
        self.batch_sampler = SimpleNamespace(batch_size=b)
        self.b, self.t, self.seed = b, t, seed

    def __iter__(self):
        g = torch.Generator().manual_seed(self.seed)
        while True:
            yield SimpleNamespace(obs=torch.rand(self.b, self.t, 3, 8, 8, generator=g) * 2 - 1,
                                  act=torch.randint(0, 4, (self.b, self.t), generator=g))


def _fake_sample(self, prev_obs, prev_act):
    x = prev_obs[:, -1] * 0.9 + 0.05 * prev_act[:, -1].float()[:, None, None, None] + 0.01 * torch.randn(prev_obs[:, -1].shape)
    return x, [x, x]


def _run_env(envmod, cfg_cls, sampler_cfg, steps=40, seed=3):
    torch.manual_seed(seed)
    env = envmod.WorldModelEnv(FakeDenoiser(), FakeRewEnd(), Loader(6, 5, 11), cfg_cls(7, 3, sampler_cfg), return_denoising_trajectory=True)
    env.sampler.sample = _fake_sample.__get__(env.sampler)
    out = [env.reset()[0].clone()]
    g = torch.Generator().manual_seed(seed + 1)
    for _ in range(steps):
        act = torch.randint(0, 4, (6,), generator=g)
        obs, rew, end, trunc, info = env.step(act)
        out += [obs.clone(), rew.clone(), end.clone(), trunc.clone(), env.ep_len.clone(), env.act_buffer.clone(), env.obs_buffer.clone()]
        for k in ("final_observation", "burnin_obs", "denoising_trajectory"):
            out.append(info[k].clone() if k in info else torch.zeros(0))
    return out


def _golden(golden_dir, prefix):
    """The tensors stored under `prefix`_000, `prefix`_001, ... in the reference fixture, in order."""
    g = np.load(os.path.join(golden_dir, "env_host_logic.npz"))
    return [torch.from_numpy(g[k]) for k in sorted(k for k in g.files if k.startswith(prefix + "_"))]


def digest(t: torch.Tensor) -> str:
    """dtype, shape and SHA-256 of the bytes of a CPU tensor: two tensors without NaNs have equal digests exactly when they
    have the same dtype and shape and are bit-equal."""
    a = t.contiguous().numpy()
    return f"{a.dtype} {tuple(a.shape)} {hashlib.sha256(a.tobytes()).hexdigest()}"


def test_world_model_env_matches_reference_bit_for_bit(golden_dir):
    a = np.load(os.path.join(golden_dir, "env_host_logic.npz"))["env_digests"].tolist()
    b = [digest(t) for t in _run_env(mine, mine.WorldModelEnvConfig, mine.DiffusionSamplerConfig(3))]
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert x == y, f"tensor {i} of the rollout: reference {x}, mirror {y}"


class FakePolicy(torch.nn.Module):
    lstm_dim = 4
    device = torch.device("cpu")

    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.tensor(0.3))

    def predict_act_value(self, obs, hx_cx):
        hx, cx = hx_cx
        f = obs.flatten(1).mean(1, keepdim=True)
        hx = torch.tanh(hx * 0.5 + f * self.w)
        cx = cx * 0.9 + f
        logits = torch.cat([hx[:, :2] + f, cx[:, :2] - f], 1)
        return logits, (hx.sum(1) + cx.sum(1)) * self.w, (hx, cx)


def _run_loop(loop_factory, envmod, cfg_cls, sampler_cfg):
    torch.manual_seed(5); random.seed(5)
    env = envmod.WorldModelEnv(FakeDenoiser(), FakeRewEnd(), Loader(6, 5, 12), cfg_cls(5, 3, sampler_cfg))
    env.sampler.sample = _fake_sample.__get__(env.sampler)
    loop = loop_factory(env, FakePolicy())
    res = []
    for _ in range(3):
        *tensors, infos = loop.send(6)
        res += [t.detach().clone() for t in tensors]
    return res


def lambda_return_inputs():
    """rew, end, trunc, val_bootstrap of the lambda-return check (4 envs x 9 steps, a few terminations and truncations)."""
    g = torch.Generator().manual_seed(0)
    rew = torch.randn(4, 9, generator=g) * 2; end = (torch.rand(4, 9, generator=g) < 0.1).long()
    trunc = (torch.rand(4, 9, generator=g) < 0.1).long(); vb = torch.randn(4, 9, generator=g)
    return rew, end, trunc, vb


def test_env_loop_and_lambda_returns_match_reference_bit_for_bit(golden_dir):
    a = _golden(golden_dir, "loop")
    b = _run_loop(make_env_loop, mine, mine.WorldModelEnvConfig, mine.DiffusionSamplerConfig(3))
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x.shape == y.shape and torch.equal(x, y)
    want = _golden(golden_dir, "lambda_returns")
    assert len(want) == len(LAMBDAS)
    for lam, w in zip(LAMBDAS, want):
        assert torch.equal(compute_lambda_returns(*lambda_return_inputs(), 0.985, lam), w)


def test_world_model_env_invariants_without_reference():
    """Always runs: truncation at the horizon, ep_len reset, frame stack shifted by exactly one frame per step."""
    torch.manual_seed(0)
    env = mine.WorldModelEnv(FakeDenoiser(), FakeRewEnd(), Loader(6, 5, 11), mine.WorldModelEnvConfig(4, 3, mine.DiffusionSamplerConfig(3)))
    env.sampler.sample = _fake_sample.__get__(env.sampler)
    env.reset()
    for _ in range(12):
        prev = env.obs_buffer.clone()
        prev_len = env.ep_len.clone()
        obs, rew, end, trunc, info = env.step(torch.zeros(6, dtype=torch.long))
        dead = torch.logical_or(end, trunc)
        assert torch.equal(trunc.bool(), prev_len + 1 >= 4)
        assert torch.all(env.ep_len[dead] == 0) and torch.equal(env.ep_len[~dead], prev_len[~dead] + 1)
        assert torch.equal(env.obs_buffer[~dead, :-1], prev[~dead, 1:])
        assert set(rew.unique().tolist()) <= {-1.0, 0.0, 1.0}
