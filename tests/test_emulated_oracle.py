"""CPU: the per-tensor bound that tests/test_gpu_backward_emulated.py holds the native backward to
(fp16_oracle.PER_TENSOR_BOUND, set by how far fp16 rounding amplifies fp32 summation order) still catches wrong backward
kernels.  Each mutation below is one plausible kernel bug,
applied to the emulation itself; its emulation-vs-emulation error must exceed the bound by at least 5x on some tensor.
A legitimate implementation choice -- a power-of-two gradient scale per tensor instead of once per call -- must stay
inside it.  Finally the emulation's distance from the fp32 oracle must agree with oracle/grad_error_budget.py, the CPU
budget the backward kernels were designed against."""
import os

import numpy as np
import pytest
import torch

from oracle import fp16_oracle as E
from oracle import torch_oracle as O

# two levels: a Downsample / Upsample pair, a 1x1 projection of a 64 + 32 concat, attention at C = 64; three images
INNER = O.InnerCfg(num_steps_conditioning=2, cond_channels=64, depths=[1, 1], channels=[32, 64], attn_depths=[0, 1])
B, H, W = 3, 16, 16


@pytest.fixture(scope="module")
def problem():
    sd = O.seeded_state_dict(O.inner_model_shapes(INNER), 2024)
    obs, act, x0 = O.synthetic_inputs(B, INNER, H, W, 2025)
    rng = np.random.default_rng(2026)
    c_noise = torch.from_numpy(rng.normal(0.0, 0.5, size=B)).float()
    go = torch.from_numpy(rng.standard_normal((B, INNER.img_channels, H, W))).float() * 1e-2
    args = (sd, INNER, x0 * 0.7, c_noise, obs.reshape(B, -1, H, W) / 0.5, act, go)
    scale = E.loss_scale(go)
    return args, scale, E.parameter_grads(*args, E.Emulation(scale))


MUTATIONS = {
    "a_wgrad_drops_one_image": dict(drop_wgrad_image=("unet.d_blocks.1.resblocks.0.conv1", 1)),
    "b_zero_insertion_shifted_one_pixel": dict(zero_insert_shift=1),
    "c_groupnorm_bwd_without_mean_term": dict(gn_drop_mean_term=True),
    "d_film_shift_gradient_dropped": dict(drop_film_shift="unet.u_blocks.0.resblocks.1.norm2."),
}


@pytest.mark.parametrize("name", sorted(MUTATIONS))
def test_subtle_backward_bug_exceeds_the_gpu_bound(problem, name):
    args, scale, want = problem
    got = E.parameter_grads(*args, E.Emulation(scale, **MUTATIONS[name]))
    _, per = E.rel_errors(got, want)
    worst = max(per, key=per.get)
    print(f"{name}: worst tensor error {per[worst]:.3e} ({worst}), GPU bound {E.PER_TENSOR_BOUND:.1e}, "
          f"ratio {per[worst] / E.PER_TENSOR_BOUND:.0f}x")
    assert per[worst] >= 5 * E.PER_TENSOR_BOUND


def test_per_tensor_gradient_scale_stays_inside_the_bound(problem):
    args, scale, want = problem
    got = E.parameter_grads(*args, E.Emulation(scale, per_tensor_scale=True))
    _, per = E.rel_errors(got, want)
    worst = max(per, key=per.get)
    print(f"e_per_tensor_scale: worst tensor error {per[worst]:.3e} ({worst}), GPU bound {E.PER_TENSOR_BOUND:.1e}")
    assert per[worst] <= E.PER_TENSOR_BOUND


def test_emulation_matches_the_gradient_error_budget(golden_dir):
    """Same fixture (denoiser_default_training: default net, B = 2, one step): the emulation's whole-gradient distance from
    the fp32 oracle agrees with grad_error_budget's "+ wgrad fp16" row.  The two differ in where they round (the budget keeps
    the backward of conv_in / the projections exact and scales each gradient operand separately), not in what they round."""
    from oracle import grad_error_budget as GB
    from oracle.make_golden import CASES, TRAIN_CASES

    name = "denoiser_default_training"
    tc = TRAIN_CASES[name]
    c = CASES[tc["case"]]
    inner, cfg = c["inner"], O.DenoiserCfg(inner=c["inner"])
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    assert tc["seq"] == 1 and not tc["mask_off"]
    obs, act = torch.from_numpy(g["obs"]), torch.from_numpy(g["act"])
    raw_sigma, raw_offset, raw_noise = (torch.from_numpy(g[k][0]) for k in ("raw_sigma", "raw_offset", "raw_noise"))
    n = inner.num_steps_conditioning
    b = obs.size(0)
    sigma = O.training_sigma(raw_sigma, O.SigmaDistCfg())
    noisy = O.apply_noise(obs[:, n], sigma, raw_offset, raw_noise, cfg.sigma_offset_noise)
    c_in, c_out, c_skip, c_noise = O.conditioners(sigma, cfg)
    sd = O.seeded_state_dict(O.inner_model_shapes(inner), c["wseed"])
    args = (noisy * c_in, c_noise, obs[:, :n].reshape(b, -1, *obs.shape[-2:]) / cfg.sigma_data, act[:, :n])
    target = (obs[:, n] - c_skip * noisy) / c_out

    def loss_grads(emu):   # mse_loss(model output, target) back-propagated, as grad_error_budget does it
        p = {k: v.clone().requires_grad_(k != "noise_emb.weight") for k, v in sd.items()}
        mo = O.inner_model(*args, p, inner) if emu is None else E.inner_model(*args, p, inner, emu)
        go = 2 * (mo.detach() - target) / mo.numel()
        if emu is not None:
            emu.scale = E.loss_scale(go)   # read by the backward: the native call's S comes from this grad_out
        mo.backward(go)
        return {k: v.grad for k, v in p.items() if v.grad is not None}

    ref, emu = loss_grads(None), loss_grads(E.Emulation(1.0))
    whole, _ = E.rel_errors(emu, ref)
    _, budget, _ = GB.run(name, (1, 1, 1), (0, 0, 0))
    print(f"emulation vs fp32 oracle {whole:.3e}; grad_error_budget {budget:.3e}")
    assert 0.8 * budget <= whole <= 1.25 * budget, (whole, budget)
