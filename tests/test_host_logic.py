"""CPU: host-side mirror of the reference's module surface (no kernel launches)."""
import dataclasses
import json
import os

import pytest
import torch

from diamond_b200.models.diffusion import (Denoiser, DenoiserConfig, DiffusionSamplerConfig, InnerModelConfig)
from diamond_b200.models.diffusion.diffusion_sampler import build_sigmas
from oracle import torch_oracle as O

# Denoiser configs whose state_dict layout is pinned to the reference's (tests/golden/reference_surface.json)
LAYOUT_CASES = [O.InnerCfg(), O.InnerCfg(depths=[1, 2, 1], channels=[32, 64, 32], attn_depths=[0, 0, 1], cond_channels=64,
                                         num_steps_conditioning=2, num_actions=6)]


def _denoiser(inner: O.InnerCfg) -> Denoiser:
    return Denoiser(DenoiserConfig(InnerModelConfig(inner.img_channels, inner.num_steps_conditioning, inner.cond_channels,
                                                    list(inner.depths), list(inner.channels), list(inner.attn_depths),
                                                    inner.num_actions), 0.5, 0.3))


def _reference_surface(golden_dir):
    with open(os.path.join(golden_dir, "reference_surface.json")) as f:
        return json.load(f)


@pytest.mark.parametrize("inner", LAYOUT_CASES)
def test_state_dict_keys_and_shapes_match_the_reference_layout(inner, golden_dir):
    den = _denoiser(inner)
    want = O.inner_model_shapes(inner)
    got = [(k, tuple(v.shape)) for k, v in den.inner_model.state_dict().items()]
    assert got == want
    ref = _reference_surface(golden_dir)["denoiser_state_dict"][LAYOUT_CASES.index(inner)]
    assert ref["inner"] == dataclasses.asdict(inner)
    assert [(k, tuple(s)) for k, s in ref["layout"]] == [(k, tuple(v.shape)) for k, v in den.state_dict().items()]


def test_default_denoiser_has_the_reference_parameter_count_and_init():
    den = _denoiser(O.InnerCfg())
    assert sum(p.numel() for p in den.parameters()) == 4_405_955  # SURVEY.md F6
    sd = den.inner_model.state_dict()
    # zero-initialised layers (blocks.py:59-60,139; inner_model.py:42)
    assert float(sd["conv_out.weight"].abs().sum()) == 0
    assert float(sd["unet.d_blocks.0.resblocks.0.conv2.weight"].abs().sum()) == 0
    assert float(sd["unet.mid_blocks.resblocks.0.attn.out_proj.weight"].abs().sum()) == 0
    w = sd["unet.downsamples.1.conv.weight"].flatten(1)  # orthogonal (blocks.py:97)
    assert torch.allclose(w @ w.t(), torch.eye(64), atol=1e-4)


def test_reference_configure_opt_accepts_the_mirror(golden_dir):
    """utils.configure_opt classifies parameters by isinstance(owner, nn.Conv2d/Linear/GroupNorm/...) and asserts full
    coverage (utils.py:129-166): its rule (restated by the oracle) splits the mirror exactly as the reference split its own
    default Denoiser, 114 decay / 121 no-decay (SURVEY.md 8b)."""
    den = _denoiser(O.InnerCfg())
    decay, no_decay = O.weight_decay_split(den)
    ref = _reference_surface(golden_dir)["configure_opt"]
    assert (decay, no_decay) == (ref["decay"], ref["no_decay"])
    assert [len(decay), len(no_decay)] == [114, 121]


def test_sigma_schedule_matches_reference_values():
    s = build_sigmas(3, 2e-3, 5, 7, torch.device("cpu"))
    assert torch.allclose(s, torch.tensor([5.0, 0.28308, 0.002, 0.0]), atol=1e-5)  # SURVEY.md 3.3
    assert torch.equal(s, O.build_sigmas(3, 2e-3, 5, 7))
    assert DiffusionSamplerConfig(3).order == 1


def test_training_needs_setup_and_cpu_is_rejected():
    den = _denoiser(O.InnerCfg())
    with pytest.raises(RuntimeError):  # denoiser.py:52: setup_training first
        den(None)
    with pytest.raises(RuntimeError):  # no CPU fallback: the native executor refuses non-CUDA parameters
        den.denoise(torch.zeros(1, 3, 64, 64), torch.ones(1), torch.zeros(1, 12, 64, 64), torch.zeros(1, 4, dtype=torch.long))
    from diamond_b200.models.diffusion import SigmaDistributionConfig

    den.setup_training(SigmaDistributionConfig(-0.4, 1.2, 2e-3, 20))
    from types import SimpleNamespace

    batch = SimpleNamespace(obs=torch.zeros(2, 5, 3, 64, 64), act=torch.zeros(2, 5, dtype=torch.long), mask_padding=torch.ones(2, 5, dtype=torch.bool))
    with pytest.raises(RuntimeError):  # the training forward is native too: CPU tensors are refused, not silently computed
        den(batch)


def test_synthetic_generators_match_the_oracle_rule():
    """diamond_b200.synthetic (used by bench.py / smoke for the PRODUCT path) and the oracle's seeded weights agree, so the
    GPU tests can compare a model initialised by one with the oracle evaluated on the other."""
    from diamond_b200.synthetic import frame_stacks, randomize_module_

    inner = O.InnerCfg(depths=[1, 1, 1, 1])
    den = _denoiser(inner)
    randomize_module_(den.inner_model, 42)
    sd = O.seeded_state_dict(O.inner_model_shapes(inner), 42)
    for k, v in den.inner_model.state_dict().items():
        assert torch.equal(v, sd[k]), k
    obs, act, x0 = frame_stacks(3, 4, 3, 64, 64, 4, 7)
    o2, a2, x2 = O.synthetic_inputs(3, inner, 64, 64, 7)
    assert torch.equal(obs, o2) and torch.equal(act, a2) and torch.equal(x0, x2)


def test_copies_of_a_native_module_do_not_share_the_native_handle():
    """copy.deepcopy / pickle of a module with a native executor (EMA copies, multiprocessing): the copy must start without
    the raw handle, the packed weights and the cached layouts of the original (a shared handle would be freed twice)."""
    import copy
    import pickle

    from diamond_b200.models.actor_critic import ActorCritic, ActorCriticConfig
    from diamond_b200.models.diffusion import InnerModelConfig
    from diamond_b200.models.diffusion.inner_model import InnerModel

    im = InnerModel(InnerModelConfig(3, 2, 64, [1, 1], [32, 32], [0, 0], 4))
    ac = ActorCritic(ActorCriticConfig(64, 3, 16, [32, 32], [1, 1], 4))
    for m in (im, ac):
        m._state_tensors()
        m.__dict__["_h"] = 0xDEAD           # stands in for a live native handle (never dereferenced on this CPU box)
        m.__dict__["_wkey"] = ("stale",)
        m.__dict__["_packed"] = torch.zeros(4)
        m.__dict__["_ws_pool"] = [torch.zeros(1)]
        m.__dict__["_gv_layout"] = ([0], [1], 1)
        try:
            for clone in (copy.deepcopy(m), pickle.loads(pickle.dumps(m))):
                assert clone._h is None and clone._wkey is None and clone._packed is None
                assert "_ws_pool" not in clone.__dict__ and "_gv_layout" not in clone.__dict__ and "_state_tensor_cache" not in clone.__dict__
                assert list(clone.state_dict().keys()) == list(m.state_dict().keys())
                assert all(torch.equal(a, b) for a, b in zip(clone.state_dict().values(), m.state_dict().values()))
            assert m._h == 0xDEAD and m._wkey == ("stale",)   # the original keeps its own state
        finally:
            m.__dict__["_h"] = None         # __del__ must not hand the fake handle to the library
