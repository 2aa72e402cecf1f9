"""Output head of the image models: truncated logistic over S bins (reference lib/models/models.py:20-74, :248-282).

Only the head lives here — the score networks (U-Net, DiT, ...) stay the reference's stock PyTorch modules.  The
reference turns the two numbers per dimension the U-Net emits (`model_output == 'logistic_pars'`,
lib/networks/unet.py:450-452) into an (B, D, S) logits tensor with ~20 elementwise passes; here

* inside this package's samplers (`ops.fused_head()` context, no gradients) `TruncatedLogisticHead.head_forward` returns
  an `ops.LogisticHead`, which the samplers pass straight into the fused reverse-step kernel: the logits never exist in
  memory.  Any other caller of `model(x, t)` gets the (B, D, S) logits tensor, as from the reference;
* `sample_logistic(...)` is the reference's function with the same signature, backed by one CUDA pass
  (`ctdd_logistic_logits`) when no gradient is required;
* with gradients enabled (training) the head is one `autograd.Function`: the same forward kernel, and a backward kernel
  (`ctdd_logistic_logits_backward`) that recomputes the head from (mu, log_scale) and reads the incoming (B, D, S) gradient
  once — instead of autograd through ~20 saved (B, D, S) tensors.  Host inputs are refused (no fallback), and so are
  dtypes other than fp32 or bf16 for both.  bf16 (mu, log_scale) — a network under torch.autocast(dtype=torch.bfloat16),
  or one converted to bf16 — give bf16 logits: the fp32 values rounded once, which the losses read as they are
  (DESIGN.md §3).
"""
from __future__ import annotations

import torch

from ... import ops


def log_minus_exp(a, b, eps=1e-6):
    """log(exp(a) - exp(b)) for b < a with the reference's guard (lib/models/models.py:20-25)."""
    return a + torch.log1p(-torch.exp(b - a) + eps)


def _logistic_logits_autograd(mu, log_scale, S, fix_logistic):
    """Differentiable head on the training path: CUDA forward + backward kernels (CUDA tensors; like the rest of the
    package there is no CPU / PyTorch fallback).  fp32 (mu, log_scale) give fp32 logits, bf16 ones bf16 logits."""
    if not (mu.is_cuda and log_scale.is_cuda):
        raise RuntimeError("ctdd_b200: the truncated-logistic head runs on CUDA tensors only (no CPU fallback)")
    if mu.dtype == torch.bfloat16 and log_scale.dtype == torch.bfloat16:
        out_dtype = torch.bfloat16
    elif mu.dtype == torch.float32 and log_scale.dtype == torch.float32:
        out_dtype = torch.float32
    else:
        raise RuntimeError(f"ctdd_b200: the truncated-logistic head takes float32 or bfloat16 (mu, log_scale), both of one "
                           f"dtype; got {mu.dtype}, {log_scale.dtype} - cast the network output")
    return ops.logistic_logits_autograd(mu, log_scale, S, fix_logistic, out_dtype=out_dtype).view(*mu.shape, S)


def sample_logistic(net_out, B, C, D, S, fix_logistic, device):
    """Same signature and result layout as the reference's sample_logistic (lib/models/models.py:28-74):
    net_out = (mu, log_scale), each (B, C, H, W) -> logits (B, C, H, W, S)."""
    mu, log_scale = net_out[0], net_out[1]
    if torch.is_grad_enabled() and (mu.requires_grad or log_scale.requires_grad):
        return _logistic_logits_autograd(mu, log_scale, S, fix_logistic)
    return ops.logistic_logits(mu, log_scale, S, fix_logistic).view(*mu.shape, S)


class TruncatedLogisticHead:
    """Mixin for image x0-prediction models whose network returns (mu, log_scale) — the tail of
    ImageX0PredBasePaul.forward (reference lib/models/models.py:248-290).  Needs `self.S` and `self.fix_logistic`."""

    def head_forward(self, net_out, B, D):
        mu, log_scale = net_out[0], net_out[1]
        if torch.is_grad_enabled() and (mu.requires_grad or log_scale.requires_grad):
            return _logistic_logits_autograd(mu, log_scale, self.S, self.fix_logistic).view(B, D, self.S)
        if ops.fused_head_enabled():      # this package's samplers: the head is evaluated inside the reverse-step kernel
            return ops.LogisticHead(mu, log_scale, self.fix_logistic)
        return ops.logistic_logits(mu, log_scale, self.S, self.fix_logistic).view(B, D, self.S)


class EMA:
    """Exponential moving average of the trainable parameters — the reference's mixin (lib/models/models.py:729-826),
    same attributes, methods, state-dict keys and error behaviour.  Inherit it FIRST so its state_dict functions win.

    `update_ema` is the only hot method (once per optimiser step): the reference runs three torch kernels per parameter
    tensor from a Python loop; here one `ctdd_ema_update` launch walks a device table of every (shadow, parameter) pair.
    The result is bitwise the reference's (same fp32 roundings)."""

    def __init__(self, cfg):
        self.decay = cfg.model.ema_decay
        self.device = cfg.device
        if self.decay < 0.0 or self.decay > 1.0:
            raise ValueError("Decay must be between 0 and 1")
        self.shadow_params = []
        self.collected_params = []
        self.num_updates = 0
        self._ema_table = None

    def _trainable(self):
        return [p for p in self.parameters() if p.requires_grad]

    def init_ema(self):
        self.shadow_params = [p.clone().detach() for p in self._trainable()]
        self._ema_table = None

    def update_ema(self):
        if len(self.shadow_params) == 0:
            raise ValueError("Shadow params not initialized before first ema update!")
        self.num_updates += 1
        decay = min(self.decay, (1 + self.num_updates) / (10 + self.num_updates))
        params = self._trainable()
        shadows = self.shadow_params
        if any(s.device != p.device for s, p in zip(shadows, params)):
            # the reference moves both to cfg.device on the fly (and so updates a copy); keep the shadows with the model
            self.shadow_params = shadows = [s.to(p.device) for s, p in zip(shadows, params)]
        table = getattr(self, "_ema_table", None)
        if table is None or not table.matches(shadows, params):
            table = self._ema_table = ops.EmaTable(shadows, [p.data for p in params])
        with torch.no_grad():
            table.update(1.0 - decay)

    def state_dict(self, *args, **kwargs):
        sd = torch.nn.Module.state_dict(self, *args, **kwargs)
        sd["ema_decay"] = self.decay
        sd["ema_num_updates"] = self.num_updates
        sd["ema_shadow_params"] = self.shadow_params
        return sd

    def move_shadow_params_to_model_params(self):
        for s_param, param in zip(self.shadow_params, self._trainable()):
            param.data.copy_(s_param.data)

    def move_model_params_to_collected_params(self):
        self.collected_params = [param.clone() for param in self.parameters()]

    def move_collected_params_to_model_params(self):
        for c_param, param in zip(self.collected_params, self.parameters()):
            param.data.copy_(c_param.data)

    def load_state_dict(self, state_dict, *args, **kwargs):
        missing, unexpected = torch.nn.Module.load_state_dict(self, state_dict, strict=False)
        if len(missing) > 0:
            print("Missing keys: ", missing)
            raise ValueError
        if sorted(unexpected) != ["ema_decay", "ema_num_updates", "ema_shadow_params"]:
            print("Unexpected keys: ", unexpected)
            raise ValueError
        self.decay = state_dict["ema_decay"]
        self.num_updates = state_dict["ema_num_updates"]
        self.shadow_params = state_dict["ema_shadow_params"]
        self._ema_table = None

    def train(self, mode=True):
        if self.training == mode:
            print("Dont call model.train() with the same mode twice! Otherwise EMA parameters may overwrite original parameters")
            print("Current model training mode: ", self.training)
            print("Requested training mode: ", mode)
            raise ValueError
        torch.nn.Module.train(self, mode)
        if mode:
            if len(self.collected_params) > 0:
                self.move_collected_params_to_model_params()
            else:
                print("model.train(True) called but no ema collected parameters!")
        else:
            self.move_model_params_to_collected_params()
            self.move_shadow_params_to_model_params()
        return self
