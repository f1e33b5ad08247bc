"""GPU: the native denoiser backward (dmd_inner_model_forward_train + dmd_denoiser_backward, driven through InnerModel under
autograd) against oracle/fp16_oracle.py, which restates the roundings of the native training plan, tensor by tensor, with no
tensor exempt, at the batch sizes training runs at.  The fp32 oracle stays the second side (whole gradient).

Batches are REPLICATED: D = 5 distinct samples (own obs, action, noisy frame, c_noise and grad_out) at slot i mod 5, so
neighbouring images differ and every tile boundary falls between different samples.  Every op is per sample, so the
parameter gradient is sum_d n_d g_d; each g_d is one single-sample oracle pass evaluated with the native call's loss scale S
(one power of two per backward call, from max|grad_out| over the whole batch).

Measured on a B200 (1000 W, 1965 MHz), worst single tensor vs the emulation / whole gradient vs fp32: default net
B = 1, 5, 33, 64, 256: 2.36e-3, 2.36e-3, 2.26e-3, 2.12e-3, 2.03e-3 / <= 8.96e-4; small 1.66e-3 / 9.05e-4; attn64
9.5e-4 / 8.15e-4; nonsquare 1.12e-3 / 9.06e-4.  The per-tensor bound (fp16_oracle.PER_TENSOR_BOUND = 5e-3) sits at the
floor that fp16 re-rounding puts under ANY whole-network emulation (the emulation in fp32 vs in fp64: 2.4e-3), not at
fp32 accumulation order; the wrong kernels of tests/test_emulated_oracle.py land 74x to 244x above it."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

D = 5   # distinct samples of a replicated batch


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    return torch.device("cuda:0")


def _configs():
    from oracle import torch_oracle as O

    small = O.InnerCfg(img_channels=3, num_steps_conditioning=2, cond_channels=64, depths=[1, 2, 1], channels=[32, 64, 32],
                       attn_depths=[0, 0, 1], num_actions=6)
    return {
        # name: (inner config, H, W, weight seed, scalar c_noise, fp32 whole-gradient bound); the input seed follows the weight seed
        "default": (O.InnerCfg(), 64, 64, 1234, False, 1e-3),
        # 3 levels, attention inside level 2 at C = 32 (attn_bwd_kernel<32>) and in the mid blocks
        "small": (small, 32, 32, 4321, True, 1.25e-3),
        # attention level with 64 channels inside the levels (attn_bwd_kernel<64>), 1x1 projection of a 64 + 32 concat
        "attn64": (O.InnerCfg(cond_channels=128, depths=[1, 1], channels=[32, 64], attn_depths=[0, 1]), 16, 16, 99, False, 1.25e-3),
        # non-square, no padding: PH != PW in every PLC16 geometry; the last level is 4 x 16 = the 64 attention tokens
        "nonsquare": (small, 16, 64, 4321, False, 1.25e-3),
    }


_SAMPLES, _GRADS = {}, {}


def _samples(name):
    """D distinct single-sample inputs, already rescaled as InnerModel receives them."""
    if name not in _SAMPLES:
        from oracle import torch_oracle as O

        inner, h, w, wseed, scalar, _ = _configs()[name]
        obs, act, x0 = O.synthetic_inputs(D, inner, h, w, wseed + 1 + h)
        rng = np.random.default_rng(wseed + 2 + w)
        sigma = np.exp(rng.normal(-0.4, 1.2, size=D)).clip(2e-3, 20)
        c_noise = torch.from_numpy(np.log(np.sqrt(sigma ** 2 + 0.09)) / 4).float()
        if scalar:
            c_noise = c_noise[:1]
        # one sample dominates max|grad_out|: the others run with less headroom under the batch-wide scale
        amp = torch.tensor([0.6, 0.25, 1.0, 0.05, 0.4]) * 1e-2
        go = torch.from_numpy(rng.standard_normal((D, inner.img_channels, h, w))).float() * amp[:, None, None, None]
        noisy = x0 * torch.from_numpy(1 / np.sqrt(sigma ** 2 + 0.09 + 0.25)).float()[:, None, None, None]
        _SAMPLES[name] = (noisy, c_noise, obs.reshape(D, -1, h, w) / 0.5, act, go)
    return _SAMPLES[name]


def _oracle_grads(name, d, scale):
    """g_d of sample d: emulated with loss scale `scale`, or the fp32 oracle when scale is None (cached across batch sizes)."""
    key = (name, d, scale)
    if key not in _GRADS:
        from oracle import fp16_oracle as E
        from oracle import torch_oracle as O

        inner, _, _, wseed, scalar, _ = _configs()[name]
        sd = O.seeded_state_dict(O.inner_model_shapes(inner), wseed)
        noisy, c_noise, obs, act, go = _samples(name)
        cn = c_noise if scalar else c_noise[d:d + 1]
        emu = None if scale is None else E.Emulation(scale)
        _GRADS[key] = E.parameter_grads(sd, inner, noisy[d:d + 1], cn, obs[d:d + 1], act[d:d + 1], go[d:d + 1], emu)
    return _GRADS[key]


def _replicated_sum(name, B, scale):
    n = [len(range(d, B, D)) for d in range(D)]
    out = {}
    for d in range(D):
        if n[d]:
            for k, g in _oracle_grads(name, d, scale).items():
                out[k] = out[k] + n[d] * g if k in out else n[d] * g
    return out


def _native_grads(name, B, dev):
    from diamond_b200 import _lib
    from diamond_b200.models.diffusion.inner_model import InnerModel, InnerModelConfig
    from oracle import torch_oracle as O

    inner, h, w, wseed, scalar, _ = _configs()[name]
    model = InnerModel(InnerModelConfig(inner.img_channels, inner.num_steps_conditioning, inner.cond_channels, list(inner.depths),
                                        list(inner.channels), list(inner.attn_depths), inner.num_actions))
    model.load_state_dict(O.seeded_state_dict(O.inner_model_shapes(inner), wseed))
    model = model.to(dev).train()
    need = _lib.lib().dmd_denoiser_train_workspace_bytes(model.native(), B, h, w)
    assert need > 0, _lib.lib().dmd_last_error().decode()
    free, _ = torch.cuda.mem_get_info(dev)
    if need + (1 << 30) > free:   # workspace + ~1 GB of inputs, gradients and allocator slack
        pytest.skip(f"B={B} at {h}x{w} needs a {need / 2**30:.1f} GB training workspace; {free / 2**30:.1f} GB free on this device")
    idx = torch.arange(B) % D
    noisy, c_noise, obs, act, go = _samples(name)
    cn = c_noise if scalar else c_noise[idx]
    out = model(noisy[idx].to(dev), cn.to(dev), obs[idx].to(dev), act[idx].to(dev))
    out.backward(go[idx].to(dev))
    torch.cuda.synchronize()
    return {k: p.grad.detach().cpu() for k, p in model.named_parameters()}


def _check(name, B):
    from oracle import fp16_oracle as E

    dev = _dev()
    go = _samples(name)[4]
    scale = E.loss_scale(go[:min(B, D)])   # the native call's S: max|grad_out| over the whole (replicated) batch
    got = _native_grads(name, B, dev)
    emu = _replicated_sum(name, B, scale)
    ref = _replicated_sum(name, B, None)
    assert set(got) == set(emu) == set(ref)
    whole_e, per_e = E.rel_errors(got, emu)
    whole_f, per_f = E.rel_errors(got, ref)
    print(f"\n{name} B={B} S=2^{int(np.log2(scale))}: whole-gradient error vs emulation {whole_e:.3e}, vs fp32 {whole_f:.3e}")
    print("    vs emulation   vs fp32      |g|        tensor")
    for k in sorted(per_e, key=per_e.get, reverse=True):
        print(f"    {per_e[k]:9.3e}   {per_f[k]:9.3e}   {float(emu[k].norm()):9.3e}  {k}")
    worst = max(per_e, key=per_e.get)
    bound_f = _configs()[name][5]
    assert per_e[worst] <= E.PER_TENSOR_BOUND, (name, B, worst, per_e[worst])
    assert whole_f < bound_f, (name, B, whole_f)


@pytest.mark.parametrize("B", [1, 5, 33, 64, 256])
def test_default_net_backward_matches_fp16_emulation(B):
    """Default net at 64x64, per-sample c_noise.  B = 33 / 64 put tiles across many images and split wgrad's K over many
    CTAs; B = 256 (the benchmarked training batch) hits the colsum / absmax grid caps and hundreds of rows of fp32 atomics in
    embedding_bwd / film_wgrad and the FiLM split-K GEMM at its largest M."""
    _check("default", B)


@pytest.mark.parametrize("name", ["small", "attn64", "nonsquare"])
def test_other_nets_backward_matches_fp16_emulation(name):
    """small: scalar c_noise; attn64: attn_bwd_kernel<64> inside the levels; nonsquare: 16x64."""
    _check(name, 7)
