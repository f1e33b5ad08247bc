"""RewEndModel (reference: src/models/rew_end_model.py) with a native sm_100a `predict_rew_end` (SURVEY.md 8 f1).

The reward / termination model runs once per imagined step between the sampler and the policy (world_model_env.py:97) and
over the burn-in frames of every fresh episode (:120-129).  Parameters live under the reference's names (state_dict keys,
`Agent.load`, `configure_opt`'s isinstance split keep working); the arithmetic — encoder ResBlocks at C = 32 with FiLM on
the action embedding, two attention blocks, LSTM over time, SiLU head — runs in `dmd_rew_end_predict`.

Training (`forward`, rew_end_model.py:57-90; SURVEY.md 8 f2) is native too: the host logic of the reference (final-frame
substitution, mask, cross-entropy losses, confusion matrices) is torch on the device, and everything with FLOPs is one
autograd node, `_RewEndFn`: `dmd_rew_end_forward_train` keeps the activations, `dmd_rew_end_backward` writes every parameter
gradient into one flat buffer whose views become `.grad`."""
import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch import Tensor

from .. import _lib
from ..utils import LossAndLogs, NativeStateMixin, init_lstm
from .blocks import Downsample, ResBlocks, _NativeOnly, conv3x3


@dataclass
class RewEndModelConfig:  # rew_end_model.py:15-24
    lstm_dim: int
    img_channels: int
    img_size: int
    cond_channels: int
    depths: List[int]
    channels: List[int]
    attn_depths: List[int]
    num_actions: Optional[int] = None


class RewEndEncoder(_NativeOnly):  # rew_end_model.py:93-125 (parameter container; executed natively)
    def __init__(self, in_channels: int, cond_channels: int, depths: List[int], channels: List[int], attn_depths: List[int]) -> None:
        super().__init__()
        assert len(depths) == len(channels) == len(attn_depths)
        self.conv_in = conv3x3(in_channels, channels[0])
        blocks = []
        for i, n in enumerate(depths):
            c1, c2 = channels[max(0, i - 1)], channels[i]
            blocks.append(ResBlocks([c1] + [c2] * (n - 1), [c2] * n, cond_channels, attn_depths[i]))
        blocks.append(ResBlocks([channels[-1]] * 2, [channels[-1]] * 2, cond_channels, True))
        self.blocks = nn.ModuleList(blocks)
        self.downsamples = nn.ModuleList([nn.Identity()] + [Downsample(c) for c in channels[:-1]] + [nn.Identity()])


class RewEndModel(NativeStateMixin, nn.Module):
    def __init__(self, cfg: RewEndModelConfig) -> None:  # rew_end_model.py:27-41 (same registration order)
        super().__init__()
        self.cfg = cfg
        self.encoder = RewEndEncoder(2 * cfg.img_channels, cfg.cond_channels, cfg.depths, cfg.channels, cfg.attn_depths)
        self.act_emb = nn.Embedding(cfg.num_actions, cfg.cond_channels)
        input_dim_lstm = cfg.channels[-1] * (cfg.img_size // 2 ** (len(cfg.depths) - 1)) ** 2
        self.lstm = nn.LSTM(input_dim_lstm, cfg.lstm_dim, batch_first=True)
        self.head = nn.Sequential(nn.Linear(cfg.lstm_dim, cfg.lstm_dim), nn.SiLU(), nn.Linear(cfg.lstm_dim, 3 + 2, bias=False))
        init_lstm(self.lstm)
        self._h = None
        self._h_dev = None
        self._wkey = None
        self._packed = None
        self._ws = None

    def __del__(self):
        try:
            if self._h is not None:
                _lib.lib().dmd_rew_end_destroy(self._h)
        except Exception:
            pass

    @property
    def device(self) -> torch.device:
        return self.act_emb.weight.device

    def _native(self):
        lib = _lib.lib()
        dev = self.device
        if dev.type != "cuda":
            raise RuntimeError("diamond_b200 runs on CUDA (sm_100a) only; move the model to a cuda device")
        self.require_current_device(dev)
        if self._h is None or self._h_dev != dev.index:
            if self._h is not None:
                lib.dmd_rew_end_destroy(self._h)
            c = self.cfg
            cc = _lib.RewEndConfigC()
            cc.lstm_dim, cc.img_channels, cc.img_size, cc.cond_channels, cc.num_levels = c.lstm_dim, c.img_channels, c.img_size, c.cond_channels, len(c.channels)
            for i in range(len(c.channels)):
                cc.depths[i], cc.channels[i], cc.attn_depths[i] = int(c.depths[i]), int(c.channels[i]), int(bool(c.attn_depths[i]))
            cc.num_actions = int(c.num_actions)
            h = lib.dmd_rew_end_create(C.byref(cc))
            if not h:
                raise RuntimeError("diamond_b200: " + lib.dmd_last_error().decode())
            self._h, self._h_dev, self._wkey, self._packed, self._ws = h, dev.index, None, None, None
        tensors = self._state_tensors()
        wkey = tuple((t.data_ptr(), t._version) for t in tensors)
        if wkey != self._wkey:
            n = lib.dmd_rew_end_num_tensors(self._h)
            if n != len(tensors):
                raise RuntimeError(f"native rew_end model expects {n} tensors, module has {len(tensors)}")
            for t in tensors:
                if t.dtype != torch.float32 or not t.is_contiguous():
                    raise RuntimeError("parameters must be contiguous fp32")
            if self._packed is None:
                self._packed = torch.empty(lib.dmd_rew_end_packed_bytes(self._h), dtype=torch.uint8, device=dev)
            arr = (C.c_void_p * n)(*[t.data_ptr() for t in tensors])
            _lib.check(lib.dmd_rew_end_set_weights(self._h, arr, n, self._packed.data_ptr(), _lib.current_stream()))
            self._wkey = wkey
        return self._h

    @torch.no_grad()
    def predict_rew_end(self, obs: Tensor, act: Tensor, next_obs: Tensor,
                        hx_cx: Optional[Tuple[Tensor, Tensor]] = None) -> Tuple[Tensor, Tensor, Tuple[Tensor, Tensor]]:
        # rew_end_model.py:42-55.  hx_cx: each (1, b, lstm_dim) like torch.nn.LSTM
        lib = _lib.lib()
        h = self._native()
        b, t, c, hh, ww = obs.shape
        dev = obs.device
        obs_, nxt_, act_ = obs.float().contiguous(), next_obs.float().contiguous(), act.long().contiguous()
        hx = cx = None
        if hx_cx is not None:
            hx, cx = hx_cx[0].reshape(b, -1).float().contiguous(), hx_cx[1].reshape(b, -1).float().contiguous()
        rew = torch.empty(b, t, 3, device=dev)
        end = torch.empty(b, t, 2, device=dev)
        hx_o = torch.empty(b, self.cfg.lstm_dim, device=dev)
        cx_o = torch.empty(b, self.cfg.lstm_dim, device=dev)
        need = lib.dmd_rew_end_workspace_bytes(h, b * t)
        if need == 0:
            raise RuntimeError("diamond_b200: " + lib.dmd_last_error().decode())
        if self._ws is None or self._ws.numel() < need or self._ws.device != dev:
            self._ws = torch.empty(need, dtype=torch.uint8, device=dev)
        _lib.check(lib.dmd_rew_end_predict(h, b, t, obs_.data_ptr(), nxt_.data_ptr(), act_.data_ptr(), _lib.ptr(hx), _lib.ptr(cx),
                                           rew.data_ptr(), end.data_ptr(), hx_o.data_ptr(), cx_o.data_ptr(), self._ws.data_ptr(),
                                           self._ws.numel(), _lib.current_stream()))
        return rew, end, (hx_o.unsqueeze(0), cx_o.unsqueeze(0))

    # ------------------------------------------------------------------ training plumbing
    def grad_layout(self):
        """(offsets, numels, total) of the flat fp32 gradient buffer the native backward fills (state_dict order)."""
        lib = _lib.lib()
        h = self._native()
        n = lib.dmd_rew_end_num_tensors(h)
        offs, nums = (C.c_longlong * n)(), (C.c_longlong * n)()
        total = lib.dmd_rew_end_grad_layout(h, offs, nums, n)
        if total < 0:
            raise RuntimeError("diamond_b200: " + lib.dmd_last_error().decode())
        return list(offs), list(nums), int(total)

    def acquire_train_workspace(self, nbytes: int) -> Tensor:
        """A training workspace holds one forward's activations until its backward has run; pooled across steps."""
        pool = self.__dict__.setdefault("_tws_pool", [])
        for i, ws in enumerate(pool):
            if ws.numel() >= nbytes and ws.device == self.device:
                return pool.pop(i)
        return torch.empty(nbytes, dtype=torch.uint8, device=self.device)

    def release_train_workspace(self, ws: Tensor) -> None:
        pool = self.__dict__.setdefault("_tws_pool", [])
        if len(pool) < 2:
            pool.append(ws)

    def _check_frames(self, obs: Tensor) -> None:
        s = self.cfg.img_size
        if obs.dim() != 5 or obs.shape[-2:] != (s, s) or obs.shape[2] != self.cfg.img_channels:
            raise RuntimeError(f"diamond_b200: rew_end frames must be (b, t, {self.cfg.img_channels}, {s}, {s}) (img_size of the "
                               f"config), got {tuple(obs.shape)}")

    # ------------------------------------------------------------------ reference surface
    def forward(self, batch) -> LossAndLogs:  # rew_end_model.py:57-90
        obs = batch.obs[:, :-1]
        act = batch.act[:, :-1]
        next_obs = batch.obs[:, 1:]
        rew = batch.rew[:, :-1]
        end = batch.end[:, :-1]
        mask = batch.mask_padding[:, :-1]

        # :67-71 when dead, the frame after the last step (padding) becomes the true final observation.  next_obs is a view:
        # the assignment writes through into batch.obs, so the frame is also obs of the following step, as in the reference
        dead = end.bool().any(dim=1)
        if dead.any():
            final_obs = torch.stack([i["final_observation"] for i, d in zip(batch.info, dead) if d]).to(obs.device)
            next_obs[dead, end[dead].argmax(dim=1)] = final_obs

        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            names = [k for k, _ in self.named_parameters()]
            params = [p for _, p in self.named_parameters()]
            logits_rew, logits_end = _RewEndFn.apply(self, names, obs, act, next_obs, *params)
        else:
            self._check_frames(obs)
            logits_rew, logits_end, _ = self.predict_rew_end(obs, act, next_obs)
        logits_rew = logits_rew[mask]
        logits_end = logits_end[mask]
        target_rew = rew[mask].sign().long().add(1)  # clipped to {-1, 0, 1}
        target_end = end[mask]

        loss_rew = F.cross_entropy(logits_rew, target_rew)
        loss_end = F.cross_entropy(logits_end, target_end)
        loss = loss_rew + loss_end

        metrics = {
            "loss_rew": loss_rew.detach(),
            "loss_end": loss_end.detach(),
            "loss_total": loss.detach(),
            "confusion_matrix": {
                "rew": confusion_matrix(logits_rew, target_rew, 3),
                "end": confusion_matrix(logits_end, target_end, 2),
            },
        }
        return loss, metrics


def confusion_matrix(logits: Tensor, target: Tensor, num_classes: int) -> Tensor:
    """torcheval's multiclass_confusion_matrix as the reference calls it (rew_end_model.py:84-85): int64 [n, n], rows the true
    class, columns the arg-max prediction."""
    n = num_classes
    idx = target.long() * n + logits.detach().argmax(dim=1)
    return torch.bincount(idx, minlength=n * n).reshape(n, n)


class _RewEndFn(torch.autograd.Function):
    """predict_rew_end from a zero LSTM state under autograd: forward = dmd_rew_end_forward_train (activations stay in the
    training workspace), backward = dmd_rew_end_backward (all parameter gradients in one flat buffer, returned as views).
    The frames and actions get no gradient."""

    @staticmethod
    def forward(ctx, module, names, obs, act, next_obs, *params):
        lib = _lib.lib()
        h = module._native()
        module._check_frames(obs)
        b, t = obs.shape[:2]
        dev = obs.device
        obs_, nxt_, act_ = obs.detach().float().contiguous(), next_obs.detach().float().contiguous(), act.long().contiguous()
        rew = torch.empty(b, t, 3, device=dev)
        end = torch.empty(b, t, 2, device=dev)
        need = lib.dmd_rew_end_train_workspace_bytes(h, b, t)
        if need == 0:
            raise RuntimeError("diamond_b200: " + lib.dmd_last_error().decode())
        ws = module.acquire_train_workspace(need)
        _lib.check(lib.dmd_rew_end_forward_train(h, b, t, obs_.data_ptr(), nxt_.data_ptr(), act_.data_ptr(), rew.data_ptr(),
                                                 end.data_ptr(), ws.data_ptr(), ws.numel(), _lib.current_stream()))
        ctx.module, ctx.names, ctx.bt, ctx.ws, ctx.keep = module, names, (b, t), ws, (obs_, nxt_, act_)
        return rew, end

    @staticmethod
    def backward(ctx, g_rew, g_end):
        lib = _lib.lib()
        module = ctx.module
        h = module._native()
        b, t = ctx.bt
        dev = ctx.ws.device
        g_rew = torch.zeros(b, t, 3, device=dev) if g_rew is None else g_rew.float().contiguous()
        g_end = torch.zeros(b, t, 2, device=dev) if g_end is None else g_end.float().contiguous()
        offs, nums, total = module.grad_layout()
        flat = torch.empty(total, dtype=torch.float32, device=dev)
        _lib.check(lib.dmd_rew_end_backward(h, b, t, g_rew.data_ptr(), g_end.data_ptr(), flat.data_ptr(), total, ctx.ws.data_ptr(),
                                            _lib.current_stream()))
        index = {k: i for i, k in enumerate(module.state_dict().keys())}
        grads = []
        for name, p in zip(ctx.names, module.parameters()):
            i = index[name]
            grads.append(flat[offs[i]:offs[i] + nums[i]].view_as(p))
        module.release_train_workspace(ctx.ws)
        module.last_flat_grad = flat   # one contiguous buffer: what a data-parallel step all-reduces in a single collective
        return (None, None, None, None, None, *grads)
