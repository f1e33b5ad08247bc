"""Generates tests/golden/*.npz by running the UNMODIFIED reference (imported from /root/reference/src with test-side
stub modules, oracle/ref_import.py) on seeded inputs and seeded 'de-zeroed' weights.  Run in the build container:

    python oracle/make_golden.py

The fixtures pin oracle/torch_oracle.py (CPU tests) and the CUDA path (GPU tests) to the reference itself.
Weights are NOT stored (17 MB); they are regenerated from the seed by torch_oracle.seeded_state_dict and guarded by a
checksum stored in the fixture.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_import  # noqa: E402
from oracle import torch_oracle as O  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

CASES = {
    # SURVEY.md 8d cfg 1 shape (default agent config), batch 2 so per-sample sigma / cond paths are exercised
    "denoiser_default": dict(
        inner=O.InnerCfg(), h=64, w=64, b=2, wseed=1234, iseed=77, sigmas=[0.7, 3.0],
        sampler=O.SamplerCfg(num_steps_denoising=3), rng_seed=0,
    ),
    # small net: 3 levels, attention inside a level, Heun + churn, odd batch, 6 actions, 2 conditioning frames
    "denoiser_small_heun": dict(
        inner=O.InnerCfg(img_channels=3, num_steps_conditioning=2, cond_channels=64, depths=[1, 2, 1],
                         channels=[32, 64, 32], attn_depths=[0, 0, 1], num_actions=6),
        h=32, w=32, b=3, wseed=4321, iseed=78, sigmas=[0.05, 1.0, 12.0],
        sampler=O.SamplerCfg(num_steps_denoising=4, order=2, s_churn=1.0), rng_seed=5,
    ),
    # UNet pad / crop path (blocks.py:225-229,245): 60 x 62 is not a multiple of 2^3, the U-Net runs at 64 x 64 on the
    # zero-padded conv_in output and its result is cropped back before norm_out / conv_out
    "denoiser_padded": dict(
        inner=O.InnerCfg(), h=60, w=62, b=2, wseed=1357, iseed=79, sigmas=[0.4, 5.0],
        sampler=O.SamplerCfg(num_steps_denoising=3), rng_seed=3,
    ),
}


def build_reference(ns, inner: O.InnerCfg, sd):
    D = ns.diffusion
    cfg = D.DenoiserConfig(
        D.InnerModelConfig(inner.img_channels, inner.num_steps_conditioning, inner.cond_channels, list(inner.depths),
                           list(inner.channels), list(inner.attn_depths), num_actions=inner.num_actions),
        sigma_data=0.5, sigma_offset_noise=0.3)
    den = D.Denoiser(cfg)
    ref_keys = list(den.inner_model.state_dict().keys())
    assert ref_keys == list(sd.keys()), "oracle key order differs from the reference's state_dict"
    for k, v in den.inner_model.state_dict().items():
        assert tuple(v.shape) == tuple(sd[k].shape), (k, v.shape, sd[k].shape)
    den.inner_model.load_state_dict(sd)
    return den.eval()


def main(only=None):
    ns = ref_import.load()
    torch.set_num_threads(8)
    os.makedirs(OUT, exist_ok=True)
    for name, c in CASES.items():
        if only and name not in only:
            continue
        inner = c["inner"]
        sd = O.seeded_state_dict(O.inner_model_shapes(inner), c["wseed"])
        den = build_reference(ns, inner, sd)
        obs, act, x_noisy = O.synthetic_inputs(c["b"], inner, c["h"], c["w"], c["iseed"])
        sig = torch.tensor(c["sigmas"], dtype=torch.float32)
        b, t, ch, h, w = obs.shape
        obs_flat = obs.reshape(b, t * ch, h, w)
        with torch.no_grad():
            cs = den.compute_conditioners(sig)
            mo = den.compute_model_output(x_noisy, obs_flat, act, cs)
            dn = den.wrap_model_output(x_noisy, mo, cs)
            dn2 = den.denoise(x_noisy, sig, obs_flat, act)
            assert torch.equal(dn, dn2)
            # full sampler, reference draws its own noise from the global torch RNG
            s = c["sampler"]
            sampler = ns.diffusion.DiffusionSampler(den, ns.diffusion.DiffusionSamplerConfig(
                s.num_steps_denoising, s.sigma_min, s.sigma_max, s.rho, s.order, s.s_churn, s.s_tmin, s.s_tmax, s.s_noise))
            torch.manual_seed(c["rng_seed"])
            x, traj = sampler.sample(obs, act)
            # replay the RNG stream to capture the noise tensors the reference consumed (diffusion_sampler.py:36,42)
            torch.manual_seed(c["rng_seed"])
            x0 = torch.randn(b, ch, h, w)
            assert torch.equal(x0, traj[0])
            n_sig = len(sampler.sigmas)
            gamma_ = min(s.s_churn / (n_sig - 1), 2**0.5 - 1)
            eps = np.zeros((n_sig - 1, b, ch, h, w), np.float32)
            for i, sg in enumerate(sampler.sigmas[:-1]):
                if gamma_ > 0 and s.s_tmin <= sg <= s.s_tmax:
                    eps[i] = (torch.randn(b, ch, h, w) * s.s_noise).numpy()
                    if s.order == 2 and sampler.sigmas[i + 1] != 0:
                        pass  # Heun draws no extra noise
        np.savez_compressed(
            os.path.join(OUT, name + ".npz"),
            weights_checksum=np.float64(O.state_checksum(sd)),
            sigmas_in=sig.numpy(), model_output=mo.numpy(), denoised=dn.numpy(),
            sampler_sigmas=sampler.sigmas.numpy(), x0=x0.numpy(), eps=eps, sample_x=x.numpy(),
            trajectory=torch.stack(traj).numpy(),
        )
        print(name, "model_output rms", float(mo.pow(2).mean().sqrt()), "sample rms", float(x.pow(2).mean().sqrt()),
              "size", os.path.getsize(os.path.join(OUT, name + ".npz")))


def make_actor_critic():
    """Reference ActorCritic.predict_act_value over 3 recurrent steps (hidden state carried), seeded de-zeroed weights."""
    ns = ref_import.load()
    AC = ns.actor_critic
    cfg = O.ActorCriticCfg()
    sd = O.seeded_actor_critic_state_dict(cfg, 555)
    ac = AC.ActorCritic(AC.ActorCriticConfig(cfg.lstm_dim, cfg.img_channels, cfg.img_size, list(cfg.channels), list(cfg.down), cfg.num_actions)).eval()
    assert [(k, tuple(v.shape)) for k, v in ac.state_dict().items()] == O.actor_critic_shapes(cfg)
    ac.load_state_dict(sd)
    rng = np.random.default_rng(91)
    b = 5
    obs = torch.from_numpy(rng.integers(0, 256, size=(3, b, 3, 64, 64)).astype(np.float32)).div(255).mul(2).sub(1)
    hx = torch.from_numpy(rng.standard_normal((b, 512)).astype(np.float32)) * 0.3
    cx = torch.from_numpy(rng.standard_normal((b, 512)).astype(np.float32)) * 0.3
    logits, vals = [], []
    h, c = hx, cx
    with torch.no_grad():
        for t in range(3):
            out = ac.predict_act_value(obs[t], (h, c))
            logits.append(out.logits_act); vals.append(out.val); h, c = out.hx_cx
    np.savez_compressed(os.path.join(OUT, "actor_critic_default.npz"), weights_checksum=np.float64(O.state_checksum(sd)),
                        hx0=hx.numpy(), cx0=cx.numpy(), logits=torch.stack(logits).numpy(), val=torch.stack(vals).numpy(),
                        hx=h.numpy(), cx=c.numpy())
    print("actor_critic_default logits rms", float(torch.stack(logits).pow(2).mean().sqrt()))


TRAIN_CASES = {
    # default agent config, one autoregressive step, every sample valid
    "denoiser_default_training": dict(case="denoiser_default", b=2, seq=1, mask_off=[], rng_seed=21, dseed=301),
    # small net, two autoregressive steps (the second conditions on the first step's denoised frame), one padded sample
    "denoiser_small_training": dict(case="denoiser_small_heun", b=3, seq=2, mask_off=[(1, -1)], rng_seed=22, dseed=302),
}


def make_denoiser_training():
    """Reference Denoiser.forward (training loss, denoiser.py:93-122) + backward on seeded weights / batches.  The fixture
    records the standard-normal draws the reference consumed from the global RNG, the loss and a gradient summary."""
    ns = ref_import.load()
    D = ns.diffusion
    for name, tc in TRAIN_CASES.items():
        c = CASES[tc["case"]]
        inner = c["inner"]
        sd = O.seeded_state_dict(O.inner_model_shapes(inner), c["wseed"])
        den = build_reference(ns, inner, sd).train()
        sig_cfg = O.SigmaDistCfg()
        den.setup_training(D.SigmaDistributionConfig(sig_cfg.loc, sig_cfg.scale, sig_cfg.sigma_min, sig_cfg.sigma_max))
        rng = np.random.default_rng(tc["dseed"])
        b, n, T = tc["b"], inner.num_steps_conditioning, inner.num_steps_conditioning + tc["seq"]
        ch, h, w = inner.img_channels, c["h"], c["w"]
        obs = torch.from_numpy(rng.integers(0, 256, size=(b, T, ch, h, w)).astype(np.float32)).div(255).mul(2).sub(1)
        act = torch.from_numpy(rng.integers(0, inner.num_actions, size=(b, T)).astype(np.int64))
        mask = torch.ones(b, T, dtype=torch.bool)
        for (bi, ti) in tc["mask_off"]:
            mask[bi, ti] = False
        batch = ns.data.Batch(obs=obs, act=act, rew=torch.zeros(b, T), end=torch.zeros(b, T, dtype=torch.long),
                              trunc=torch.zeros(b, T, dtype=torch.long), mask_padding=mask, info=[{}] * b, segment_ids=[None] * b)
        torch.manual_seed(tc["rng_seed"])
        loss, logs = den(batch)
        loss.backward()
        # replay the RNG stream: per step randn(b) [sigma], randn(b, c, 1, 1) [offset], randn(b, c, h, w) [noise]
        torch.manual_seed(tc["rng_seed"])
        raw_sigma, raw_off, raw_noise = [], [], []
        for _ in range(tc["seq"]):
            raw_sigma.append(torch.randn(b)); raw_off.append(torch.randn(b, ch, 1, 1)); raw_noise.append(torch.randn(b, ch, h, w))
        grads = [(k, p.grad) for k, p in den.inner_model.named_parameters()]
        assert all(g is not None for _, g in grads)
        keys, norms, samples = O.grad_summary(grads)
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, weights_checksum=np.float64(O.state_checksum(sd)), obs=obs.numpy(), act=act.numpy(),
                            mask_padding=mask.numpy(), raw_sigma=torch.stack(raw_sigma).numpy(), raw_offset=torch.stack(raw_off).numpy(),
                            raw_noise=torch.stack(raw_noise).numpy(), loss=np.float64(loss.item()), grad_keys=np.array(keys),
                            grad_norms=norms, grad_samples=samples)
        print(name, "loss", loss.item(), "grad norm", float(np.sqrt((norms**2).sum())), "size", os.path.getsize(path))


class _ScriptedEnv:
    """Deterministic stand-in for TorchEnv / WorldModelEnv (envs/env.py, world_model_env.py:58-106 surface used by
    env_loop.py): returns pre-generated observations, rewards and termination flags, ignores the action."""

    def __init__(self, obs_seq, rew, end, trunc, final_obs, num_actions):
        self.obs_seq, self.rew, self.end, self.trunc, self.final_obs = obs_seq, rew, end, trunc, final_obs
        self.num_envs, self.num_actions, self.t = obs_seq.size(1), num_actions, 0

    def reset(self, seed=None):
        self.t = 0
        return self.obs_seq[0], {}

    def step(self, act):
        t = self.t
        dead = torch.logical_or(self.end[t].bool(), self.trunc[t].bool())
        info = {"final_observation": self.final_obs[t]} if dead.any() else {}
        self.t += 1
        return self.obs_seq[t + 1], self.rew[t], self.end[t], self.trunc[t], info


def make_actor_critic_training():
    """Reference ActorCritic.forward (loss, actor_critic.py:75-98) through the reference's own make_env_loop
    (env_loop.py:12-74) over a scripted environment with two terminations, + backward (BPTT through the LSTM)."""
    ns = ref_import.load()
    AC = ns.actor_critic
    cfg = O.ActorCriticCfg()
    sd = O.seeded_actor_critic_state_dict(cfg, 556)
    ac = AC.ActorCritic(AC.ActorCriticConfig(cfg.lstm_dim, cfg.img_channels, cfg.img_size, list(cfg.channels), list(cfg.down), cfg.num_actions))
    ac.load_state_dict(sd)
    lc = O.ActorCriticLossCfg(backup_every=5)
    rng = np.random.default_rng(92)
    T, b = lc.backup_every, 4
    obs_seq = torch.from_numpy(rng.integers(0, 256, size=(T + 1, b, 3, 64, 64)).astype(np.float32)).div(255).mul(2).sub(1)
    rew = torch.from_numpy(rng.choice([-1.0, 0.0, 0.0, 2.0], size=(T, b)).astype(np.float32))
    end = torch.zeros(T, b, dtype=torch.long); trunc = torch.zeros(T, b, dtype=torch.long)
    end[1, 2] = 1; trunc[3, 0] = 1; end[T - 1, 1] = 1   # mid-rollout termination, truncation, termination on the last step
    final_obs = {}
    for t in range(T):
        dead = torch.logical_or(end[t].bool(), trunc[t].bool())
        if dead.any():
            final_obs[t] = torch.from_numpy(rng.integers(0, 256, size=(int(dead.sum()), 3, 64, 64)).astype(np.float32)).div(255).mul(2).sub(1)
    env = _ScriptedEnv(obs_seq, rew, end, trunc, final_obs, cfg.num_actions)
    ac.setup_training(env, AC.ActorCriticLossConfig(lc.backup_every, lc.gamma, lc.lambda_, lc.weight_value_loss, lc.weight_entropy_loss))
    torch.manual_seed(31)
    # capture what the env loop hands to the loss (the sampled actions are data for the oracle)
    captured = {}
    real_loop = ac.env_loop

    class _Tap:
        def send(self, n):
            out = real_loop.send(n)
            captured["out"] = out
            return out
    ac.env_loop = _Tap()
    loss, metrics = ac()
    loss.backward()
    _, act, rew_o, end_o, trunc_o, logits, val, val_bootstrap, _ = captured["out"]
    grads = [(k, p.grad) for k, p in ac.named_parameters()]
    assert all(g is not None for _, g in grads)
    keys, norms, samples = O.grad_summary(grads)
    path = os.path.join(OUT, "actor_critic_training.npz")
    fo_t = np.array(sorted(final_obs.keys()), np.int64)
    np.savez_compressed(path, weights_checksum=np.float64(O.state_checksum(sd)), obs_seq=obs_seq.numpy(), rew=rew.numpy(), end=end.numpy(),
                        trunc=trunc.numpy(), final_obs_t=fo_t, **{f"final_obs_{t}": final_obs[t].numpy() for t in final_obs},
                        act=act.numpy(), logits=logits.detach().numpy(), val=val.detach().numpy(), val_bootstrap=val_bootstrap.numpy(),
                        loss=np.float64(loss.item()), metric_keys=np.array(list(metrics.keys())),
                        metric_vals=np.array([float(v) for v in metrics.values()], np.float64),
                        grad_keys=np.array(keys), grad_norms=norms, grad_samples=samples)
    print("actor_critic_training loss", loss.item(), "grad norm", float(np.sqrt((norms**2).sum())), "size", os.path.getsize(path))


def make_rew_end():
    """Reference RewEndModel.predict_rew_end (SURVEY.md 8 f1): a 3-step burn-in call that returns the LSTM state, then two
    single-step calls carrying it -- the way WorldModelEnv uses it (world_model_env.py:96-105, :120-129)."""
    ns = ref_import.load()
    R = ns.rew_end_model
    cfg = O.RewEndCfg()
    sd = O.seeded_state_dict(O.rew_end_shapes(cfg), 777)
    m = R.RewEndModel(R.RewEndModelConfig(cfg.lstm_dim, cfg.img_channels, cfg.img_size, cfg.cond_channels, list(cfg.depths),
                                          list(cfg.channels), list(cfg.attn_depths), cfg.num_actions)).eval()
    assert [(k, tuple(v.shape)) for k, v in m.state_dict().items()] == O.rew_end_shapes(cfg)
    m.load_state_dict(sd)
    rng = np.random.default_rng(93)
    b = 3
    frames = torch.from_numpy(rng.integers(0, 256, size=(b, 6, 3, 64, 64)).astype(np.float32)).div(255).mul(2).sub(1)
    act = torch.from_numpy(rng.integers(0, cfg.num_actions, size=(b, 5)).astype(np.int64))
    out = {}
    with torch.no_grad():
        lr, le, hc = m.predict_rew_end(frames[:, 0:3], act[:, 0:3], frames[:, 1:4])
        out.update(burn_rew=lr.numpy(), burn_end=le.numpy())
        for k in (3, 4):
            lr, le, hc = m.predict_rew_end(frames[:, k:k + 1], act[:, k:k + 1], frames[:, k + 1:k + 2], hc)
            out.update({f"step{k}_rew": lr.numpy(), f"step{k}_end": le.numpy()})
    path = os.path.join(OUT, "rew_end_default.npz")
    np.savez_compressed(path, weights_checksum=np.float64(O.state_checksum(sd)), frames=frames.numpy(), act=act.numpy(),
                        hx=hc[0].numpy(), cx=hc[1].numpy(), **out)
    print("rew_end_default logits rms", float(np.sqrt((out["burn_rew"] ** 2).mean())), "size", os.path.getsize(path))


def _test_module(name):
    """tests/<name>.py, loaded by path (tests/ is not a package): the fixtures below run the same helpers as the test."""
    import importlib.util

    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "tests", name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def make_oracle_vs_reference():
    """tests/test_oracle_vs_reference.py: the reference's denoise / model output on the small net of that test, and the EDM
    pieces of its training forward (noise-level draw, apply_noise, conditioners, wrap) on one RNG stream."""
    T = _test_module("test_oracle_vs_reference")

    ns = ref_import.load()
    D = ns.diffusion
    torch.set_num_threads(8)
    sd = O.seeded_state_dict(O.inner_model_shapes(T.INNER), T.WSEED)
    den = build_reference(ns, T.INNER, sd)
    obs, act, x = O.synthetic_inputs(3, T.INNER, 32, 32, T.ISEED)
    sig = torch.tensor(T.SIGMAS)
    obs_flat = obs.reshape(3, 12, 32, 32)
    with torch.no_grad():
        dn = den.denoise(x, sig, obs_flat, act)
        mo = den.compute_model_output(x, obs_flat, act, den.compute_conditioners(sig))
    edm = D.Denoiser(D.DenoiserConfig(D.InnerModelConfig(*T.EDM_INNER), 0.5, 0.3))
    edm.setup_training(D.SigmaDistributionConfig(*T.EDM_SIGMA_DIST))
    edm_x = torch.from_numpy(np.random.default_rng(94).random((5, 3, 16, 16), dtype=np.float32)) * 2 - 1
    pieces = T.edm_pieces(edm, edm_x)
    path = os.path.join(OUT, "oracle_vs_reference.npz")
    np.savez_compressed(path, weights_checksum=np.float64(O.state_checksum(sd)), denoised=dn.numpy(), model_output=mo.numpy(),
                        edm_x=edm_x.numpy(), **{"edm_" + k: v.numpy() for k, v in pieces.items()})
    print("oracle_vs_reference size", os.path.getsize(path))


def make_reference_surface():
    """tests/test_host_logic.py: the reference Denoiser's state_dict layout for each config of that test, and the weight-decay
    split utils.configure_opt makes of the default Denoiser (names of the parameters in its two AdamW groups)."""
    import dataclasses
    import json

    T = _test_module("test_host_logic")

    ns = ref_import.load()
    D = ns.diffusion

    def reference_denoiser(inner):
        return D.Denoiser(D.DenoiserConfig(D.InnerModelConfig(inner.img_channels, inner.num_steps_conditioning, inner.cond_channels,
                                                              list(inner.depths), list(inner.channels), list(inner.attn_depths),
                                                              inner.num_actions), 0.5, 0.3))

    layouts = [{"inner": dataclasses.asdict(inner),
                "layout": [[k, list(v.shape)] for k, v in reference_denoiser(inner).state_dict().items()]} for inner in T.LAYOUT_CASES]
    den = reference_denoiser(O.InnerCfg())
    names = {id(p): n for n, p in den.named_parameters()}
    opt = ns.utils.configure_opt(den, 1e-4, 1e-2, 1e-8)
    decay, no_decay = ([names[id(p)] for p in g["params"]] for g in opt.param_groups)
    path = os.path.join(OUT, "reference_surface.json")
    with open(path, "w") as f:
        json.dump({"denoiser_state_dict": layouts, "configure_opt": {"decay": decay, "no_decay": no_decay}}, f, separators=(",", ":"))
        f.write("\n")
    print("reference_surface decay / no_decay", len(decay), len(no_decay), "size", os.path.getsize(path))


def make_env_host_logic():
    """tests/test_env_host_logic.py: what the reference's WorldModelEnv and make_env_loop return when driven by that test's fake
    networks and RNG streams, and its compute_lambda_returns on that test's inputs.  The 401 tensors of the WorldModelEnv run
    (1.8 MB of incompressible frames) are stored as digests."""
    T = _test_module("test_env_host_logic")

    ns = ref_import.load()
    ref_env = ns.envs.world_model_env
    env = T._run_env(ref_env, ref_env.WorldModelEnvConfig, ns.diffusion.DiffusionSamplerConfig(3))
    loop = T._run_loop(ns.env_loop.make_env_loop, ref_env, ref_env.WorldModelEnvConfig, ns.diffusion.DiffusionSamplerConfig(3))
    lam = [ns.actor_critic.compute_lambda_returns(*T.lambda_return_inputs(), 0.985, x) for x in T.LAMBDAS]
    assert not any(t.is_floating_point() and bool(t.isnan().any()) for t in env)   # digests compare NaNs as equal
    arrays = {"env_digests": np.array([T.digest(t) for t in env])}
    for prefix, ts in (("loop", loop), ("lambda_returns", lam)):
        arrays.update({f"{prefix}_{i:03d}": t.numpy() for i, t in enumerate(ts)})
    path = os.path.join(OUT, "env_host_logic.npz")
    np.savez_compressed(path, **arrays)
    print("env_host_logic tensors", len(arrays), "size", os.path.getsize(path))


if __name__ == "__main__":
    which = sys.argv[1:] or ["inference", "training", "host"]
    named = [w for w in which if w in CASES]   # e.g. `python oracle/make_golden.py denoiser_padded`: only that fixture
    if named:
        main(named)
    if "inference" in which:
        main()
        make_actor_critic()
        make_rew_end()
    if "training" in which:
        make_denoiser_training()
        make_actor_critic_training()
    if "host" in which:
        make_oracle_vs_reference()
        make_reference_surface()
        make_env_host_logic()
