"""CPU ORACLE — test infrastructure only (see oracle/README.md): the denoiser's InnerModel as the native TRAINING path
computes it, i.e. with the roundings its kernels apply, layer by layer as make_train_plan / BwdBuilder (csrc/api.cu) build
the plan.  torch_oracle.py states what the reference computes; this module states what the sm_100a kernels compute, so
that a test can hold them to a bound set by fp32 accumulation order instead of by fp16 operand rounding.

Forward
  * ResBlock conv1 / conv2, Downsample and Upsample 3x3 convs, conv_out: single-fp16 operands (activation and weight rounded
    to nearest), fp32 accumulation.  conv_out is single-fp16 in every plan (api.cu build_structure: split-fp16 there costs 3x
    on an N = 16 conv for 3.2e-4).
  * conv_in and the 1x1 skip projections read the raw residual stream in split-fp16 ([hi | lo | hi] x [W_hi | W_hi | W_lo],
    exact to ~2^-22): treated as exact.
  * attention, including its 1x1 qkv / out projections: fp32 (attn_cluster_kernel).
  * GroupNorm statistics: fp64 (fp64 atomics in the producing conv's epilogue).
Backward (one call = one power-of-two scale S, loss_scale_kernel)
  * every conv's gradient operand is (S * dL/dy) rounded to fp16; its weight operand (dgrad) and activation operand (wgrad)
    are the fp16 roundings of the forward's.  This holds for the split-fp16 layers too: their wgrad / dgrad read only the hi
    part of the raw operand.  Results are fp32 and carry S until written (x 1/S).
  * the stride-2 adjoint is a stride-1 conv of the zero-inserted gradient; the Upsample adjoint sums 2x2 blocks.
  * GroupNorm backward is the closed form over (image, group); everything else (bias sums, FiLM, cond MLP, action
    embedding, attention) is fp32.
Since S is a power of two, carrying unscaled fp32 gradients and rounding (S * g) at each conv operand is the same
arithmetic as carrying S through fp32 buffers.  Inputs may be fp64: everything between the fp16 roundings then runs in fp64.  `Emulation` also carries the mutations tests/test_emulated_oracle.py uses to
show that the GPU bound would catch a subtly wrong kernel.
"""
import math
from dataclasses import dataclass
from typing import Dict, Optional, Tuple

import torch
import torch.nn.functional as F
from torch import Tensor

from oracle import torch_oracle as O


# Per-tensor relative L2 error allowed between the native backward and this emulation (tests/test_gpu_backward_emulated.py);
# tests/test_emulated_oracle.py shows that subtly wrong kernels land far outside it.  It cannot be much tighter at
# whole-network scale: a difference d << u (u = one fp16 ulp) in front of a rounding flips ~d/u of the elements by one ulp,
# so the next layer sees sqrt(d * u) > d, and after a few re-rounded layers two computations that differ only in fp32
# summation order are a full fp16 rounding apart.  Measured on the CPU: this emulation run in fp32 vs in fp64 differs by up
# to 2.4e-3 on single tensors of the default net (1.0e-3 when only the GroupNorm backward changes precision), and by 1e-6
# when the gradient operands are not rounded.  Native vs emulation on a B200 (DESIGN.md section 2): worst 2.4e-3.
PER_TENSOR_BOUND = 5e-3


def loss_scale(grad_out: Tensor) -> float:
    """loss_scale_kernel (csrc/bwd_kernels.cuh): S = 2^(12 - e), e the frexpf exponent of max|grad_out| over the whole
    batch of the backward call; 1 when that maximum is zero or not finite."""
    m = float(grad_out.detach().abs().max())
    if m == 0.0 or not math.isfinite(m):
        return 1.0
    return 2.0 ** (12 - math.frexp(m)[1])


def _h(t: Tensor) -> Tensor:
    return t.half().to(t.dtype)


@dataclass
class Emulation:
    scale: float                                    # S of the backward call being emulated
    # mutations (all off: the faithful emulation)
    per_tensor_scale: bool = False                  # a power-of-two scale chosen per gradient operand instead of once per call
    drop_wgrad_image: Optional[Tuple[str, int]] = None  # (conv weight key, image): that image's term left out of that wgrad
    zero_insert_shift: int = 0                      # column offset of the stride-2 adjoint's zero insertion (0 = correct)
    gn_drop_mean_term: bool = False                 # GroupNorm backward without the mean-gradient term of the closed form
    drop_film_shift: Optional[str] = None           # AdaGroupNorm prefix whose shift receives no gradient

    def q(self, g: Tensor) -> Tensor:
        """The fp16 gradient operand of a conv, expressed in unscaled units."""
        s = loss_scale(g) if self.per_tensor_scale else self.scale
        return _h(g * s) / s


class _Conv(torch.autograd.Function):
    """One nn.Conv2d of the plan.  split: split-fp16 forward (exact); otherwise single-fp16 operands."""

    @staticmethod
    def forward(ctx, x, w, b, key, stride, padding, split, emu):
        ctx.save_for_backward(x, w)
        ctx.cfg = (key, stride, padding, emu)
        return F.conv2d(x, w, b, stride=stride, padding=padding) if split else F.conv2d(_h(x), _h(w), b, stride=stride, padding=padding)

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        key, stride, padding, emu = ctx.cfg
        gq = emu.q(gy)
        if stride == 2:  # zero insertion: gq at the even pixels of the input grid, then the stride-1 adjoint
            z = gq.new_zeros(gq.shape[:2] + x.shape[2:])
            o = emu.zero_insert_shift
            z[:, :, 0::2, o::2] = gq[..., : z[:, :, 0::2, o::2].shape[-1]]
            gq = z
        gw_op = gq
        if emu.drop_wgrad_image is not None and emu.drop_wgrad_image[0] == key:
            gw_op = gq.clone()
            gw_op[emu.drop_wgrad_image[1]] = 0
        gx = torch.nn.grad.conv2d_input(x.shape, _h(w), gq, padding=padding) if ctx.needs_input_grad[0] else None
        gw = torch.nn.grad.conv2d_weight(_h(x), w.shape, gw_op, padding=padding)
        return gx, gw, gy.sum(dim=(0, 2, 3)), None, None, None, None, None


class _GroupNorm(torch.autograd.Function):
    """Normalisation over (image, group) without affine; fp64 statistics; the closed-form backward of norm_bwd_pass1/2:
    dx = rstd * (g - mean(g) - xhat * mean(g * xhat))."""

    @staticmethod
    def _stats(x, groups):
        xg = x.double().reshape(x.size(0), groups, -1)
        mean = xg.mean(-1, keepdim=True)
        rstd = (xg.var(-1, unbiased=False, keepdim=True) + O.GN_EPS).rsqrt()
        return xg, mean, rstd

    @staticmethod
    def forward(ctx, x, groups, emu):
        ctx.save_for_backward(x)
        ctx.cfg = (groups, emu)
        xg, mean, rstd = _GroupNorm._stats(x, groups)
        return ((xg - mean) * rstd).reshape(x.shape).to(x.dtype)

    @staticmethod
    def backward(ctx, gy):
        (x,) = ctx.saved_tensors
        groups, emu = ctx.cfg
        xg, mean, rstd = _GroupNorm._stats(x, groups)
        xhat = (xg - mean) * rstd
        g = gy.double().reshape(xg.shape)
        m1 = 0.0 if emu.gn_drop_mean_term else g.mean(-1, keepdim=True)
        gx = rstd * (g - m1 - xhat * (g * xhat).mean(-1, keepdim=True))
        return gx.reshape(x.shape).to(x.dtype), None, None


def _conv(x, sd, key, emu, stride=1, padding=1, split=False):
    return _Conv.apply(x, sd[key + ".weight"], sd[key + ".bias"], key, stride, padding, split, emu)


def _ada_group_norm(x, cond, sd, p, emu):  # blocks.py:41-45
    scale, shift = F.linear(cond, sd[p + "linear.weight"], sd[p + "linear.bias"])[:, :, None, None].chunk(2, dim=1)
    if p == emu.drop_film_shift:
        shift = shift.detach()
    return _GroupNorm.apply(x, O._groups(x.size(1)), emu) * (1 + scale) + shift


def _resblock(x, cond, sd, p, emu):  # blocks.py:141-147; api.cu PlanBuilder::resblock
    r = _conv(x, sd, p + "proj", emu, padding=0, split=True) if (p + "proj.weight") in sd else x
    x = _conv(F.silu(_ada_group_norm(x, cond, sd, p + "norm1.", emu)), sd, p + "conv1", emu)
    x = _conv(F.silu(_ada_group_norm(x, cond, sd, p + "norm2.", emu)), sd, p + "conv2", emu)
    x = x + r
    if (p + "attn.qkv_proj.weight") in sd:
        x = O.self_attention(x, sd, p + "attn.")
    return x


def _resblocks(x, cond, sd, p, n, emu, to_cat=None):  # blocks.py:170-177
    outs = []
    for i in range(n):
        if to_cat is not None:
            x = torch.cat((x, to_cat[i]), dim=1)
        x = _resblock(x, cond, sd, f"{p}resblocks.{i}.", emu)
        outs.append(x)
    return x, outs


def _unet(x, cond, sd, cfg: O.InnerCfg, emu):  # blocks.py:222-246 without pad / crop (training rejects padded sizes)
    div = 2 ** (len(cfg.channels) - 1)
    assert x.size(-2) % div == 0 and x.size(-1) % div == 0, "the native training path rejects sizes that need the UNet pad"
    p = "unet."
    d_outputs = []
    for i, depth in enumerate(cfg.depths):
        if i > 0:
            x = _conv(x, sd, f"{p}downsamples.{i}.conv", emu, stride=2)
        x_down = x
        x, outs = _resblocks(x, cond, sd, f"{p}d_blocks.{i}.", depth, emu)
        d_outputs.append((x_down, *outs))
    x, _ = _resblocks(x, cond, sd, f"{p}mid_blocks.", 2, emu)
    for i, skip in enumerate(reversed(d_outputs)):
        if i > 0:
            x = _conv(F.interpolate(x, scale_factor=2.0, mode="nearest"), sd, f"{p}upsamples.{i}.conv", emu)
        x, _ = _resblocks(x, cond, sd, f"{p}u_blocks.{i}.", len(skip), emu, list(skip[::-1]))
    return x


def inner_model(noisy: Tensor, c_noise: Tensor, obs: Tensor, act: Tensor, sd: O.SD, cfg: O.InnerCfg, emu: Emulation) -> Tensor:
    """inner_model.py:44-49 as the native training plan computes it (fp32 inputs; c_noise [b] or [1])."""
    emb = F.embedding(act, sd["act_emb.0.weight"]).flatten(1)
    cond = O.fourier_features(c_noise, sd["noise_emb.weight"]) + emb
    cond = F.linear(F.silu(F.linear(cond, sd["cond_proj.0.weight"], sd["cond_proj.0.bias"])), sd["cond_proj.2.weight"], sd["cond_proj.2.bias"])
    x = _conv(torch.cat((obs, noisy), dim=1), sd, "conv_in", emu, split=True)
    x = _unet(x, cond, sd, cfg, emu)
    x = _GroupNorm.apply(x, O._groups(x.size(1)), emu) * sd["norm_out.norm.weight"][:, None, None] + sd["norm_out.norm.bias"][:, None, None]
    return _conv(F.silu(x), sd, "conv_out", emu)


def parameter_grads(sd: O.SD, cfg: O.InnerCfg, noisy: Tensor, c_noise: Tensor, obs: Tensor, act: Tensor, grad_out: Tensor,
                    emu: Optional[Emulation] = None) -> Dict[str, Tensor]:
    """Gradients of <inner_model(...), grad_out> with respect to every parameter: emulated when `emu` is given (its `scale`
    is the S of the native call, which for a sub-batch is NOT loss_scale(grad_out of the sub-batch)), else the plain fp32
    oracle (torch_oracle.inner_model).  noise_emb.weight is a buffer and gets none."""
    sd = {k: v.detach().clone().requires_grad_(k != "noise_emb.weight") for k, v in sd.items()}
    out = O.inner_model(noisy, c_noise, obs, act, sd, cfg) if emu is None else inner_model(noisy, c_noise, obs, act, sd, cfg, emu)
    out.backward(grad_out)
    return {k: v.grad for k, v in sd.items() if v.grad is not None}


def rel_errors(got: Dict[str, Tensor], want: Dict[str, Tensor]):
    """(whole-gradient relative L2 error, {key: relative L2 error of that tensor}), in fp64."""
    num = den = 0.0
    per = {}
    for k, w in want.items():
        d = got[k].double() - w.double()
        num += float(d.pow(2).sum())
        den += float(w.double().pow(2).sum())
        per[k] = float(d.norm() / w.double().norm().clamp_min(1e-300))
    return math.sqrt(num / den), per
