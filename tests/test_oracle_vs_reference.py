"""CPU: the oracle restatement and the Denoiser's host-side EDM pieces against what the unmodified reference computed on the
same seeds (tests/golden/oracle_vs_reference.npz, written by oracle/make_golden.py from the reference itself)."""
import os

import numpy as np
import torch

from oracle import torch_oracle as O

# the small net of the first test: 3 levels, attention inside the middle level, 5 actions
INNER = O.InnerCfg(depths=[1, 1, 1], channels=[32, 32, 64], attn_depths=[0, 1, 0], cond_channels=64, num_actions=5)
WSEED, ISEED = 31337, 9
SIGMAS = [0.01, 0.5, 7.0]
# the EDM-pieces test: InnerModelConfig arguments, SigmaDistributionConfig arguments, RNG seed of the draws
EDM_INNER = (3, 2, 64, [1, 1], [32, 32], [0, 0], 4)
EDM_SIGMA_DIST = (-0.4, 1.2, 2e-3, 20)
EDM_SEED = 123
EDM_S0 = 1.7   # 0-dim sigma, as DiffusionSampler passes it in the reference (diffusion_sampler.py:44)
EDM_FIELDS = ("sigma", "noisy", "c_in", "c_out", "c_skip", "c_noise", "wrapped")


def edm_pieces(den, x):
    """Noise-level draw, apply_noise, conditioners and the wrap + truncating quantiser of a Denoiser (the reference's or
    diamond_b200's) on one RNG stream; then the conditioners of the 0-dim sigma EDM_S0."""
    torch.manual_seed(EDM_SEED)
    sigma = den.sample_sigma_training(x.size(0), torch.device("cpu"))
    noisy = den.apply_noise(x, sigma, 0.3)
    cs = den.compute_conditioners(sigma)
    model_out = torch.randn(x.shape)
    wrapped = den.wrap_model_output(noisy, model_out, cs)
    out = dict(zip(EDM_FIELDS, (sigma, noisy, cs.c_in, cs.c_out, cs.c_skip, cs.c_noise, wrapped)))
    out.update({"s0_" + k: v for k, v in vars(den.compute_conditioners(torch.tensor(EDM_S0))).items()})
    return out


def _golden(golden_dir):
    return np.load(os.path.join(golden_dir, "oracle_vs_reference.npz"))


def test_blocks_and_denoise_match_live_reference(golden_dir):
    torch.set_num_threads(8)
    g = _golden(golden_dir)
    sd = O.seeded_state_dict(O.inner_model_shapes(INNER), WSEED)
    assert abs(O.state_checksum(sd) - float(g["weights_checksum"])) < 1e-6 * float(g["weights_checksum"])
    obs, act, x = O.synthetic_inputs(3, INNER, 32, 32, ISEED)
    sig = torch.tensor(SIGMAS)
    cfg = O.DenoiserCfg(inner=INNER)
    with torch.no_grad():
        got = O.denoise(x, sig, obs.reshape(3, 12, 32, 32), act, sd, cfg)
        got_mo = O.model_output(x, sig, obs.reshape(3, 12, 32, 32), act, sd, cfg)
    want, want_mo = torch.from_numpy(g["denoised"]), torch.from_numpy(g["model_output"])
    assert torch.allclose(got_mo, want_mo, rtol=1e-5, atol=1e-5)
    assert float((got != want).float().mean()) < 1e-3


def test_denoiser_host_side_edm_pieces_match_the_live_reference(golden_dir):
    """The torch-level pieces of diamond_b200's Denoiser that the TRAINING forward uses on the host side (noise-level draw,
    apply_noise, conditioners, wrap + truncating quantiser) against the unmodified reference on the same RNG stream: bit-equal."""
    from diamond_b200.models.diffusion import Denoiser, DenoiserConfig, InnerModelConfig, SigmaDistributionConfig

    g = _golden(golden_dir)
    mine = Denoiser(DenoiserConfig(InnerModelConfig(*EDM_INNER), 0.5, 0.3))
    mine.setup_training(SigmaDistributionConfig(*EDM_SIGMA_DIST))
    got = edm_pieces(mine, torch.from_numpy(g["edm_x"]))
    assert sorted(got) == sorted(k[len("edm_"):] for k in g.files if k.startswith("edm_") and k != "edm_x")
    for k, v in got.items():
        want = torch.from_numpy(g["edm_" + k])
        assert v.shape == want.shape and torch.equal(v, want), k
