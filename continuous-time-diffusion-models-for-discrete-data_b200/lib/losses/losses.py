"""Training losses — drop-in for the in-scope classes of the reference's lib/losses/losses.py.

Same registered names, config keys and `calc_loss` signatures (BOTH argument orders the reference uses are accepted:
`(state, minibatch[, label])` and `(minibatch, state[, writer])`, SURVEY.md §8b).  What runs where:
  * time draw `ts` and the network forward stay in PyTorch (as in the reference);
  * q_{t|0} for the B distinct times: `ctdd_build_qt0` (one matrix per sample, lib/losses/losses.py:39);
  * forward noising x_t ~ q_{t|0}(.|x_0) and the one-jump proposal x~ (losses.py:46-101): `ctdd_noise_xt`;
  * every (B,D,S)-sized term of CT-ELBO / SDDM-ELBO / ratio matching, forward and backward w.r.t. the logits:
    `ctdd_loss_forward` / `ctdd_loss_backward` behind one autograd.Function (ops.loss_terms), on the logits as the
    network emits them (fp32, or bf16 under torch.autocast(dtype=torch.bfloat16), with a bf16 gradient back);
  * the final O(B) combination (means, nll weights, lambda mixing) is torch arithmetic on (B,) vectors.
`reverse_logscale` materialises (B,D,S,S) in the reference (infeasible at S=256); here it is the same fused kernel as
`reverse_prob`: the log-sum-exp over k of log p_k + log q[k,s] IS log(sum_k p_k q[k,s]) without the 1e-35 guard, and
-1e9 where no term survives (csrc/ctdd_loss.cu), so no (B,D,S,S) tensor and no PyTorch loss body exists.
EBMAux / BinEBMAux / d3pm_loss are out of scope (SURVEY.md §2 row 5b).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from ... import _native as nat
from ... import ops
from . import losses_utils

_CRM_TYPES = {"rm": 0, "mle": 1, "elbo": 2}


def _seed_from_torch() -> int:
    return int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())


def _dense(out, S):
    """A model evaluated without gradients may hand back its truncated-logistic head un-expanded (ops.LogisticHead);
    the loss terms need the logits tensor."""
    return out.logits(S) if isinstance(out, ops.LogisticHead) else out


def _split_args(a, b):
    """Accept (state, minibatch) or (minibatch, state)."""
    return (a, b) if isinstance(a, dict) else (b, a)


class _LossBase:
    #: test hooks (not reference config keys): fixed time draw, Philox seed / offset for the noising kernels
    ts_override = None
    seed = None
    noise_offset = 0
    #: global index of this rank's first sample (data-parallel training: the noising draws are keyed on the GLOBAL sample,
    #: so N ranks with batch slices reproduce the single-process run of the concatenated batch)
    batch_offset = 0

    def __init_subclass__(cls, **kw):
        # calc_loss runs with the model's device current (the kernels launch on the current device's stream)
        super().__init_subclass__(**kw)
        fn = cls.__dict__.get("calc_loss")
        if fn is not None:
            import functools

            @functools.wraps(fn)
            def calc_loss(self, a, b, *args, **kwargs):
                state = a if isinstance(a, dict) else b
                model = state.get("model") if isinstance(state, dict) else None
                with nat.on_device(getattr(model, "device", None)):
                    return fn(self, a, b, *args, **kwargs)
            cls.calc_loss = calc_loss

    def _prepare(self, model, minibatch, t_hi, clamp_max=None, want_tilde=True):
        if len(minibatch.shape) == 4:
            B, C, H, W = minibatch.shape
            minibatch = minibatch.view(B, C * H * W)
        B, D = minibatch.shape
        device = model.device
        if torch.device(device).type != "cuda":
            raise RuntimeError("ctdd_b200 losses run on CUDA devices only; there is no CPU fallback")
        if self.ts_override is not None:
            ts = self.ts_override.to(device=device, dtype=torch.float32)
        else:
            ts = torch.rand((B,), device=device) * (t_hi - self.min_time) + self.min_time
            if clamp_max is not None:
                ts = torch.clamp(ts, max=clamp_max)
        Q, QT = model._build_qt0(model._transition_delta(ts), inverse=True, want_transpose=True)
        beta = model._rate_scalar(ts).to(torch.float32).contiguous()
        Rb, _ = model.base_rate_tables(Q.device)
        x0 = minibatch.to(device=Q.device, dtype=torch.int32).contiguous()
        seed = self.seed if self.seed is not None else _seed_from_torch()
        xt, xtil = ops.noise_xt(Q, Rb, beta, x0, seed, self.noise_offset, batch_offset=self.batch_offset, want_tilde=want_tilde)
        return dict(B=B, D=D, ts=ts, Q=Q, QT=QT, beta=beta, Rb=Rb, x0=x0, xt=xt, x_tilde=xtil, minibatch=minibatch)


# ------------------------------------------------------------------------------------------------------ tauLDR
class _CTElboFamily(_LossBase):
    def __init__(self, cfg):
        self.cfg = cfg
        self.ratio_eps = cfg.loss.eps_ratio
        self.nll_weight = cfg.loss.nll_weight
        self.min_time = cfg.loss.min_time
        self.one_forward_pass = cfg.loss.one_forward_pass
        self.max_t = cfg.training.max_t

    def _terms(self, state, minibatch, model_args=()):
        """-> (neg_elbo, nll) as 0-dim tensors (reference losses.py:108-284)."""
        model = state["model"]
        c = self._prepare(model, minibatch, self.max_t)
        logits = _dense(model(c["xt"].long(), c["ts"], *model_args), model.S)
        kw = dict(Q=c["Q"], QT=c["QT"], Rb=c["Rb"], beta=c["beta"], x0=c["x0"], eps=self.ratio_eps)
        if self.one_forward_pass:
            reg, outer, norm, _, ce = ops.loss_terms(logits, nat.LOSS_CTELBO, xt=c["x_tilde"], x_tilde=c["x_tilde"], **kw)
        else:
            # reg term at x_t with p(x_t); signal term at x~ with a second forward pass (losses.py:114-118, :157-160)
            reg, _, _, _, ce = ops.loss_terms(logits, nat.LOSS_CTELBO, xt=c["xt"], x_tilde=c["x_tilde"], **kw)
            logits_sig = _dense(model(c["x_tilde"].long(), c["ts"], *model_args), model.S)
            _, outer, norm, _, _ = ops.loss_terms(logits_sig, nat.LOSS_CTELBO, xt=c["x_tilde"], x_tilde=c["x_tilde"], **kw)
        neg_elbo = torch.mean(-outer / norm) + torch.mean(reg)
        nll = torch.sum(ce) / (c["B"] * c["D"])
        return neg_elbo, nll


@losses_utils.register_loss
class CTElbo(_CTElboFamily):
    """tauLDR CT-ELBO + nll_weight * CE (reference losses.py:11-287)."""

    def calc_loss(self, a, b, label=None):
        state, minibatch = _split_args(a, b)
        neg_elbo, nll = self._terms(state, minibatch)
        return neg_elbo + self.nll_weight * nll


@losses_utils.register_loss
class NLL(_CTElboFamily):
    """Returns only the cross-entropy term; the noising path is the CT-ELBO's (reference losses.py:1503-1778)."""

    def calc_loss(self, a, b, label=None):
        state, minibatch = _split_args(a, b)
        _, nll = self._terms(state, minibatch)
        return nll


@losses_utils.register_loss
class CTElboLambda(_CTElboFamily):
    """w * neg_elbo + (1 - w) * nll with w = n_iter / n_iters (reference losses.py:1782-2058)."""

    def calc_loss(self, a, b, label=None):
        state, minibatch = _split_args(a, b)
        neg_elbo, nll = self._terms(state, minibatch)
        w = state["n_iter"] / self.cfg.training.n_iters
        return w * neg_elbo + (1 - w) * nll


@losses_utils.register_loss
class CondCTElbo(_LossBase):
    """Prefix-conditioned CT-ELBO (reference losses.py:547-781): the first `loss.condition_dim` dimensions are clean
    conditioning, the rest is noised; with one_forward_pass the logits come from model(cat(cond, x~))."""

    def __init__(self, cfg):
        self.cfg = cfg
        self.ratio_eps = cfg.loss.eps_ratio
        self.nll_weight = cfg.loss.nll_weight
        self.min_time = cfg.loss.min_time
        self.one_forward_pass = cfg.loss.one_forward_pass
        self.condition_dim = cfg.loss.condition_dim

    def calc_loss(self, a, b, writer=None):
        state, minibatch = _split_args(a, b)
        model = state["model"]
        if len(minibatch.shape) == 4:
            minibatch = minibatch.view(minibatch.shape[0], -1)
        cd = self.condition_dim
        conditioner, data = minibatch[:, :cd], minibatch[:, cd:]
        c = self._prepare(model, data, 1.0)
        cond = conditioner.to(c["xt"].device).long()
        kw = dict(Q=c["Q"], QT=c["QT"], Rb=c["Rb"], beta=c["beta"], x0=c["x0"], eps=self.ratio_eps)

        def sliced(x):
            return _dense(model(torch.concat((cond, x.long()), dim=1), c["ts"]), model.S)[:, cd:, :].contiguous()

        if self.one_forward_pass:
            logits = sliced(c["x_tilde"])
            reg, outer, norm, _, ce = ops.loss_terms(logits, nat.LOSS_CTELBO, xt=c["x_tilde"], x_tilde=c["x_tilde"], **kw)
        else:
            # the reference's second pass overwrites x_logits (losses.py:660-666), so its cross-entropy term (:777-779)
            # is taken at the logits of x~, not of x_t
            logits = sliced(c["xt"])
            reg, _, _, _, _ = ops.loss_terms(logits, nat.LOSS_CTELBO, xt=c["xt"], x_tilde=c["x_tilde"], **kw)
            _, outer, norm, _, ce = ops.loss_terms(sliced(c["x_tilde"]), nat.LOSS_CTELBO, xt=c["x_tilde"],
                                                   x_tilde=c["x_tilde"], **kw)
        neg_elbo = torch.mean(-outer / norm) + torch.mean(reg)
        return neg_elbo + self.nll_weight * torch.sum(ce) / (c["B"] * c["D"])


# ------------------------------------------------------------------------------------------------------ SDDM
class _SDDMFamily(_LossBase):
    def __init__(self, cfg):
        self.cfg = cfg
        self.ratio_eps = cfg.loss.eps_ratio
        self.nll_weight = cfg.loss.nll_weight
        self.min_time = cfg.loss.min_time
        self.one_forward_pass = cfg.loss.one_forward_pass

    def _terms(self, state, minibatch):
        model = state["model"]
        if not self.one_forward_pass:
            raise NotImplementedError("one_forward_pass=False is broken in the reference for ScoreElbo/SDDMElbo "
                                      "(undefined logits_sig, losses.py:1386-1390); only True is supported")
        c = self._prepare(model, minibatch, 1.0, clamp_max=0.99999)
        logits = _dense(model(c["x_tilde"].long(), c["ts"]), model.S)
        branch = nat.branch_for(self.cfg.loss.name, self.cfg.loss.logit_type)
        reg, outer, norm, rm, ce = ops.loss_terms(logits, nat.LOSS_SDDM, Q=c["Q"], QT=c["QT"], Rb=c["Rb"], beta=c["beta"],
                                                  x0=c["x0"], xt=c["x_tilde"], eps=self.ratio_eps, logit_branch=branch)
        neg_elbo = torch.mean(-outer / norm) + torch.mean(reg)
        return neg_elbo, torch.sum(rm) / c["B"], torch.sum(ce) / (c["B"] * c["D"])


@losses_utils.register_loss
class ScoreElbo(_SDDMFamily):
    """SDDM ELBO + nll_weight * sum(-ll_x~)/B (reference losses.py:1245-1500)."""

    def calc_loss(self, a, b, writer=None):
        state, minibatch = _split_args(a, b)
        neg_elbo, rm, _ = self._terms(state, minibatch)
        return neg_elbo + self.nll_weight * rm


@losses_utils.register_loss
class SDDMElbo(_SDDMFamily):
    """SDDM ELBO + nll_weight * CE(logits, x0) (reference losses.py:290-544)."""

    def calc_loss(self, a, b, writer=None):
        state, minibatch = _split_args(a, b)
        neg_elbo, _, ce = self._terms(state, minibatch)
        return neg_elbo + self.nll_weight * ce


# ------------------------------------------------------------------------------------------------------ CRM
class _CatRMFamily(_LossBase):
    def __init__(self, cfg):
        self.cfg = cfg
        self.ratio_eps = cfg.loss.eps_ratio
        self.min_time = cfg.loss.min_time
        self.S = self.cfg.data.S
        self.D = self.cfg.model.concat_dim

    def _terms(self, state, minibatch, t_hi, clamp_max):
        model = state["model"]
        if self.cfg.loss.loss_type not in _CRM_TYPES:
            raise ValueError("Unknown loss_type: %s" % self.cfg.loss.loss_type)
        c = self._prepare(model, minibatch, t_hi, clamp_max=clamp_max, want_tilde=False)
        logits = _dense(model(c["xt"].long(), c["ts"]), model.S)
        branch = nat.branch_for(self.cfg.loss.name, self.cfg.loss.logit_type)
        crm, _, _, _, ce = ops.loss_terms(logits, nat.LOSS_CRM, Q=c["Q"], QT=c["QT"], Rb=c["Rb"], beta=c["beta"], x0=c["x0"],
                                          xt=c["xt"], eps=self.ratio_eps, logit_branch=branch,
                                          crm_type=_CRM_TYPES[self.cfg.loss.loss_type])
        return torch.sum(crm) * (1 - self.cfg.loss.ce_coeff) / c["B"], torch.sum(ce) / (c["B"] * c["D"])


@losses_utils.register_loss
class CatRM(_CatRMFamily):
    """Categorical ratio matching (reference losses.py:785-890)."""

    def calc_loss(self, a, b, label=None):
        state, minibatch = _split_args(a, b)
        crm, _ = self._terms(state, minibatch, 1.0, 0.99999)
        return crm


@losses_utils.register_loss
class CatRMNLL(_CatRMFamily):
    """Ratio matching + nll_weight * CE (reference losses.py:1134-1242); times ~ U(min_time, max_t), unclamped."""

    def __init__(self, cfg):
        super().__init__(cfg)
        self.max_t = cfg.training.max_t
        self.nll_weight = cfg.loss.nll_weight

    def calc_loss(self, a, b, writer=None):
        state, minibatch = _split_args(a, b)
        crm, ce = self._terms(state, minibatch, self.max_t, None)
        return crm + self.nll_weight * ce


@losses_utils.register_loss
class NLLOriginal(_LossBase):
    """CE of model(x_t, ts, label) against x_0 with x_t ~ q_{t|0} (reference losses.py:1048-1103)."""

    def __init__(self, cfg):
        self.cfg = cfg
        self.min_time = cfg.loss.min_time

    def calc_loss(self, a, b, label=None):
        state, minibatch = _split_args(a, b)
        model = state["model"]
        c = self._prepare(model, minibatch, 1.0, want_tilde=False)
        logits = _dense(model(c["xt"].long(), c["ts"], label), model.S)
        return F.cross_entropy(logits.permute(0, 2, 1), c["x0"].long())
