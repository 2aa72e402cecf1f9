"""Reverse-CTMC samplers — drop-in for the reference's lib/sampling/sampling.py.

Same registered class names, `__init__(cfg)` / `sample(model, N[, conditioner])` signatures, config keys and
return arities as TAUnSDDM/lib/sampling/sampling.py (TauL :81-234, LBJF :237-356, MidPointTauL :359-526,
PCTauL :529-646, ConditionalTauLeaping :649-758, ConditionalPCTauLeaping :761-905).  The score network is
still called as `model(x, t_ones)`; everything between its logits and the next state — softmax, the
(N*D x S)(S x S) contraction against q_{t|0}, the forward-rate multiply, Poisson / Euler / midpoint updates —
is ONE fused kernel launch per reverse-rate evaluation (`ctdd_reverse_step`, include/ctdd.h).

Differences a caller can observe (all documented in DESIGN.md):
  * the state stays an int32 CUDA tensor; the network always receives `x.long()` (the reference drifts to
    float32 after the first jump, sampling.py:155-160);
  * q_{t|0} is built once per distinct time, not N identical copies (quirk B.10);
  * no per-step host sync: the jump statistics are accumulated on the device and read back once;
  * randomness is counter-based Philox keyed on (seed, call, global row, state); the seed is drawn from
    torch's default generator, so `torch.manual_seed` makes sampling reproducible.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

from ... import _native as nat
from ... import ops
from . import sampling_utils


def _seed_from_torch() -> int:
    return int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())


def _initial_probs(S, initial_dist, initial_dist_std):
    """target distribution of get_initial_samples (reference sampling.py:14-28) as fp32 weights."""
    if initial_dist == "uniform":
        return np.full(S, 1.0 / S, dtype=np.float32)
    if initial_dist == "gaussian":
        target = np.exp(-((np.arange(1, S + 1) - S // 2) ** 2) / (2 * initial_dist_std ** 2))
        return (target / np.sum(target)).astype(np.float32)
    raise NotImplementedError("Unrecognized initial dist " + initial_dist)


def get_initial_samples(N, D, device, S, initial_dist, initial_dist_std=None, seed=None, row_offset=0):
    """x ~ initial distribution, (N, D) int32 CUDA (reference sampling.py:14-28 returns int64)."""
    probs = torch.from_numpy(_initial_probs(S, initial_dist, initial_dist_std)).to(device)
    x = torch.empty((N, D), dtype=torch.int32, device=device)
    seed = _seed_from_torch() if seed is None else seed
    nat.check(nat.lib().ctdd_sample_categorical_shared(nat.ptr(probs), S, N * D, row_offset, seed, 0, nat.ptr(x),
                                                       nat.stream()), "ctdd_sample_categorical_shared")
    return x


class StepEngine:
    """Per-`sample()` state: q_{t|0} tables for every time of the schedule, Philox seed/offsets, statistics."""

    def __init__(self, cfg, model, N, D, S, times, branch, eps, impl=nat.IMPL_AUTO, seed=None, row_offset=0,
                 max_calls=None):
        self.model, self.N, self.D, self.S = model, N, D, S
        self.device = torch.device(model.device)
        if self.device.type != "cuda":
            raise RuntimeError("ctdd_b200 samplers run on CUDA devices only (model.device=%s); there is no CPU fallback"
                               % (model.device,))
        self.branch, self.eps, self.impl = branch, float(eps), impl
        self.seed = _seed_from_torch() if seed is None else int(seed)
        self.row_offset = int(row_offset)
        self.call = 0
        self.times = [float(t) for t in times]
        self.Q, self.QT, self.beta = model.qt0_tables(self.times, self.device)
        self.Rb, self.RbT = model.base_rate_tables(self.device)
        self.tc_bytes = int(nat.lib().ctdd_tc_tables_bytes(S)) if S == 256 else 0
        self.tc_tables = self.tc_static = None
        if self.tc_bytes > 0 and impl != nat.IMPL_SIMT and branch in (nat.BRANCH_TAULDR, nat.BRANCH_SDDM_REVERSE_PROB):
            self.tc_tables = ops.prep_tc_tables(self.Q, self.QT, self.Rb, self.eps, branch)
            self.tc_static = ops.prep_tc_static(self.Rb)
        ws = int(nat.lib().ctdd_step_workspace_bytes(N * D, S, impl))
        self.workspace = torch.empty((max(ws, 1),), dtype=torch.uint8, device=self.device) if ws > 0 else None
        ncalls = max_calls if max_calls is not None else 4 * len(self.times) + 8
        self.stats = torch.zeros((ncalls, nat.STAT_COUNT), dtype=torch.int64, device=self.device)
        # Per-step host work is kept to pointer arithmetic: the time vectors of the whole schedule are built once, the
        # state ping-pongs between three resident buffers, and ONE ctdd_step_params struct is reused - only the fields
        # that change from step to step are rewritten (the reference allocates ~25 tensors and syncs once per step).
        self._t_all = torch.tensor(self.times, dtype=torch.float32, device=self.device).view(-1, 1).expand(-1, N).contiguous()
        self._xbuf = [torch.empty((N, D), dtype=torch.int32, device=self.device) for _ in range(3)]
        self._xptr = [b.data_ptr() for b in self._xbuf]
        self._q0, self._qt0 = self.Q.data_ptr(), self.QT.data_ptr()
        self._tc0 = self.tc_tables.data_ptr() if self.tc_tables is not None else 0
        self._stats0 = self.stats.data_ptr()
        self._fn = nat.lib().ctdd_reverse_step
        self._p = nat.StepParams(
            mode=0, branch=branch, impl=impl, N=N, D=D, S=S, row_offset=self.row_offset, ld_logits=S,
            batch_stride_logits=D * S, Rb=self.Rb.data_ptr(), RbT=self.RbT.data_ptr(),
            tc_static=(self.tc_static.data_ptr() if self.tc_static is not None else None), eps=self.eps, seed=self.seed,
            workspace=(self.workspace.data_ptr() if self.workspace is not None else None))

    def t_ones(self, tidx):
        return self._t_all[tidx]

    def _fast_step(self, mode, logits, x_eval, tidx, h, reject_multi, x_base, row):
        """The common case of step(): dense contiguous fp32 / bf16 / fp16 logits or an un-materialised head (fp32 or
        bf16 (mu, log_scale)), state update only."""
        N, D, S = self.N, self.D, self.S
        p = self._p
        if isinstance(logits, ops.LogisticHead):
            mu, ls, fix = logits.as_tuple()
            mu, ls, head_bs, head_dt = ops._head_views(mu, ls, N, D)
            p.head = nat.HEAD_LOGISTIC_FIX if fix else nat.HEAD_LOGISTIC
            p.head_mu, p.head_log_scale, p.head_batch_stride, p.logits = mu.data_ptr(), ls.data_ptr(), int(head_bs), None
            p.head_dtype = head_dt      # rewritten every call, like logits_dtype: the struct is reused
        else:
            p.head, p.head_mu, p.head_log_scale, p.head_batch_stride = nat.HEAD_LOGITS, None, None, 0
            p.logits = logits.data_ptr()
            # the struct is reused across calls, whose logits may alternate between fp32, bf16 and fp16
            p.logits_dtype = nat.logits_dtype_of(logits)
        xe = x_eval.data_ptr()
        xb = x_base.data_ptr() if x_base is not None else 0
        k = 0
        while self._xptr[k] == xe or self._xptr[k] == xb:      # an output buffer that is neither input
            k += 1
        ss = S * S * 4
        p.mode, p.x_eval, p.x_base, p.x_out = mode, xe, (xb or None), self._xptr[k]
        p.Q, p.QT = self._q0 + tidx * ss, self._qt0 + tidx * ss
        p.tc_tables = (self._tc0 + tidx * self.tc_bytes) if self._tc0 else None
        p.beta, p.h, p.reject_multi, p.offset = float(self.beta[tidx]), float(h), (1 if reject_multi else 0), self.call
        p.stats_out = self._stats0 + row * nat.STAT_COUNT * 8
        p.rr_out = p.ratio_out = None
        rc = self._fn(p, torch.cuda.current_stream().cuda_stream)
        if rc != 0:
            nat.check(rc, "ctdd_reverse_step")
        return self._xbuf[k]

    def step(self, mode, logits, x_eval, tidx, h, reject_multi=False, x_base=None, draws=True,
             want_rr=False, want_ratio=False, logits_view=None, stats=None):
        """One fused reverse-rate evaluation + state update. Returns (x_new, stats_row_index).

        `draws=False` marks an evaluation that consumes no randomness (midpoint drift, rates only): the Philox
        call counter is not advanced. `stats` overrides the row of self.stats the counters are added to."""
        N, D, S = self.N, self.D, self.S
        off_elems, bstride, head = 0, None, None
        if logits_view is not None:  # (full model output, c): rows live at full[:, c:, :]
            logits, c = logits_view
            if isinstance(logits, ops.LogisticHead):
                logits = logits.slice_dims(c)
            else:
                off_elems, bstride = c * S, logits.shape[1] * S
        if isinstance(logits, ops.LogisticHead):   # truncated-logistic output head: fused into the step kernel
            head, logits = logits.as_tuple(), None
        row = self.call if self.call < self.stats.shape[0] else self.stats.shape[0] - 1
        fast = (logits_view is None and stats is None and not want_rr and not want_ratio and mode != nat.MODE_EXACT
                and x_eval.dtype == torch.int32 and x_eval.is_contiguous() and x_eval.device == self.device
                and (x_base is None or (x_base.dtype == torch.int32 and x_base.is_contiguous()))
                and torch.cuda.current_device() == (self.device.index or 0)
                and ((head is not None and self.tc_tables is not None)
                     or (head is None and logits.dtype in ops._LOGITS_DTYPES and logits.is_contiguous()
                         and logits.is_cuda)))
        if fast:
            x_out = self._fast_step(mode, ops.LogisticHead(*head) if head is not None else logits, x_eval, tidx, h,
                                    reject_multi, x_base, row)
            if draws:
                self.call += 1
            return x_out, row
        out = ops.reverse_step(
            mode, self.branch, logits, x_eval, self.Q[tidx], self.QT[tidx], self.Rb, self.RbT, self.beta[tidx], h,
            self.eps, N=N, D=D, S=S, x_base=x_base, reject_multi=reject_multi, seed=self.seed, offset=self.call,
            row_offset=self.row_offset, impl=self.impl,
            tc_tables=(self.tc_tables[tidx] if self.tc_tables is not None else None), tc_static=self.tc_static,
            workspace=self.workspace,
            stats=(stats if stats is not None else self.stats[row]), want_rr=want_rr, want_ratio=want_ratio,
            logits_offset_elems=off_elems, batch_stride=bstride, head=head)
        x_out = out["x"]
        if want_rr or want_ratio:
            self.last_rates = (out["rr"], out["ratio"])
        if draws:
            self.call += 1
        return x_out, row

    def stats_host(self):
        return self.stats.cpu().numpy()


def _as_state(x, device):
    return x.to(device=device, dtype=torch.int32).contiguous()


def get_reverse_rates(model, logits, x, t_ones, cfg, N, D, S):
    """Functional form of the reference's get_reverse_rates (sampling.py:31-78): returns (reverse_rates, ratio),
    both (N, D, S), entry s == x not zeroed.  All entries of t_ones must be equal (as in every sampler)."""
    t = float(t_ones.reshape(-1)[0].item())
    branch = nat.branch_for(cfg.loss.name, getattr(cfg.loss, "logit_type", None)
                            if cfg.loss.name not in nat.TAULDR_LOSSES else None)
    eng = StepEngine(cfg, model, N, D, S, [t], branch, cfg.sampler.eps_ratio, seed=0, max_calls=1)
    eng.step(nat.MODE_RATES_ONLY, logits, _as_state(x, eng.device), 0, 0.0, draws=False, want_rr=True, want_ratio=True)
    return eng.last_rates


def _branch_of(cfg):
    name = cfg.loss.name
    return nat.branch_for(name, None if name in nat.TAULDR_LOSSES else cfg.loss.logit_type)


def _dense(logits, S):
    """Logits tensor of a model output (materialises a LogisticHead)."""
    return logits.logits(S) if isinstance(logits, ops.LogisticHead) else logits


def _final_argmax(model, x, min_t, N, device):
    out = model(x.long(), min_t * torch.ones((N,), device=device))
    p_0gt = F.softmax(_dense(out, getattr(model, "S", None)), dim=2, dtype=torch.float32)   # 2-byte logits: fp32 ties as for fp32
    return torch.max(p_0gt, dim=2)[1]


class _SamplerBase:
    #: optional knobs (not reference config keys): Philox seed, global row offset for batch sharding, kernel family
    seed = None
    row_offset = 0
    impl = nat.IMPL_AUTO

    def __init_subclass__(cls, **kw):
        # every sampler runs with model.device current (the kernels launch on the current device's stream); a model on
        # cuda:1 while cuda:0 is current is legal in the reference and must be legal here
        super().__init_subclass__(**kw)
        fn = cls.__dict__.get("sample")
        if fn is not None:
            import functools

            @functools.wraps(fn)
            def sample(self, model, *args, **kwargs):
                # ... and with the un-materialised output head switched on: StepEngine fuses it into the step kernel
                with nat.on_device(getattr(model, "device", None)), ops.fused_head():
                    return fn(self, model, *args, **kwargs)
            cls.sample = sample


@sampling_utils.register_sampler
class TauL(_SamplerBase):
    """Tau-leaping (reference sampling.py:81-234)."""

    def __init__(self, cfg):
        self.cfg = cfg
        self.max_t = cfg.training.max_t
        self.D = cfg.model.concat_dim
        self.S = self.cfg.data.S
        self.num_steps = cfg.sampler.num_steps
        self.min_t = cfg.sampler.min_t
        self.initial_dist = cfg.sampler.initial_dist
        self.corrector_entry_time = cfg.sampler.corrector_entry_time
        self.num_corrector_steps = cfg.sampler.num_corrector_steps
        self.eps_ratio = cfg.sampler.eps_ratio
        self.is_ordinal = cfg.sampler.is_ordinal
        self.loss_name = cfg.loss.name

    def sample(self, model, N):
        initial_dist_std = self.cfg.model.Q_sigma
        device = model.device
        with torch.no_grad():
            ts = np.concatenate((np.linspace(self.max_t, self.min_t, self.num_steps), np.array([0])))
            eng = StepEngine(self.cfg, model, N, self.D, self.S, ts[:-1], _branch_of(self.cfg), self.eps_ratio,
                             impl=self.impl, seed=self.seed, row_offset=self.row_offset,
                             max_calls=self.num_steps * (1 + self.num_corrector_steps) + 1)
            x = get_initial_samples(N, self.D, device, self.S, self.initial_dist, initial_dist_std, eng.seed,
                                    self.row_offset)
            reject = not self.is_ordinal
            pred_rows = []
            for idx, t in enumerate(ts[0:-1]):
                h = ts[idx] - ts[idx + 1]
                t_ones = eng.t_ones(idx)
                logits = model(x.long(), t_ones)
                x, row = eng.step(nat.MODE_TAU_LEAP, logits, x, idx, h, reject)
                pred_rows.append(row)
                if t <= self.corrector_entry_time:
                    for _ in range(self.num_corrector_steps):
                        logits = model(x.long(), t_ones)
                        x, _ = eng.step(nat.MODE_TAU_LEAP_CORR, logits, x, idx, h, reject)
            if self.loss_name == "CTElbo" or self.loss_name == "NLL":
                x_0max = _final_argmax(model, x, self.min_t, N, device)
            else:
                x_0max = x
            st = eng.stats_host()
            change_dim = [st[r, nat.STAT_CHANGED_BASE] / N for r in pred_rows]
            return x_0max.detach().cpu().numpy().astype(int), change_dim


@sampling_utils.register_sampler
class LBJF(_SamplerBase):
    """Euler / LBJF with optional corrector (reference sampling.py:237-356)."""

    def __init__(self, cfg):
        self.cfg = cfg
        self.max_t = cfg.training.max_t
        self.D = cfg.model.concat_dim
        self.S = self.cfg.data.S
        self.num_steps = cfg.sampler.num_steps
        self.min_t = cfg.sampler.min_t
        self.initial_dist = cfg.sampler.initial_dist
        self.corrector_entry_time = cfg.sampler.corrector_entry_time
        self.num_corrector_steps = cfg.sampler.num_corrector_steps
        self.eps_ratio = cfg.sampler.eps_ratio
        self.loss_name = cfg.loss.name

    def sample(self, model, N):
        initial_dist_std = self.cfg.model.Q_sigma
        device = model.device
        with torch.no_grad():
            ts = np.concatenate((np.linspace(self.max_t, self.min_t, self.num_steps), np.array([0])))
            eng = StepEngine(self.cfg, model, N, self.D, self.S, ts[:-1], _branch_of(self.cfg), self.eps_ratio,
                             impl=self.impl, seed=self.seed, row_offset=self.row_offset,
                             max_calls=self.num_steps * (1 + self.num_corrector_steps) + 1)
            x = get_initial_samples(N, self.D, device, self.S, self.initial_dist, initial_dist_std, eng.seed,
                                    self.row_offset)
            pred_rows = []
            for idx, t in enumerate(ts[0:-1]):
                h = ts[idx] - ts[idx + 1]
                t_ones = eng.t_ones(idx)
                logits = model(x.long(), t_ones)
                x_new, row = eng.step(nat.MODE_EULER, logits, x, idx, h)
                pred_rows.append(row)
                if t <= self.corrector_entry_time:
                    for _ in range(self.num_corrector_steps):
                        logits = model(x_new.long(), t_ones)
                        x_new, _ = eng.step(nat.MODE_EULER_CORR, logits, x_new, idx, h)
                x = x_new
            if self.loss_name == "CTElbo":
                x_0max = _final_argmax(model, x, self.min_t, N, device)
            else:
                x_0max = x
            st = eng.stats_host()
            change_dim = [st[r, nat.STAT_CHANGED_BASE] / N for r in pred_rows]
            return x_0max.detach().cpu().numpy().astype(int), change_dim


@sampling_utils.register_sampler
class MidPointTauL(_SamplerBase):
    """Midpoint tau-leaping (reference sampling.py:359-526). The reference's per-dataset `state_change`
    tables (:376-388) all equal s - x; the kernel uses s - x directly, so every data.name works
    (incl. DiscreteCIFAR10 / DiscreteMNIST, which fail in the reference — quirk B.5)."""

    def __init__(self, cfg):
        self.cfg = cfg
        self.max_t = cfg.training.max_t
        self.D = cfg.model.concat_dim
        self.S = self.cfg.data.S
        self.num_steps = cfg.sampler.num_steps
        self.min_t = cfg.sampler.min_t
        self.initial_dist = cfg.sampler.initial_dist
        self.corrector_entry_time = cfg.sampler.corrector_entry_time
        self.num_corrector_steps = cfg.sampler.num_corrector_steps
        self.is_ordinal = cfg.sampler.is_ordinal
        self.device = cfg.device
        self.eps_ratio = cfg.sampler.eps_ratio
        self.loss_name = cfg.loss.name

    def sample(self, model, N):
        initial_dist_std = self.cfg.model.Q_sigma
        device = model.device
        with torch.no_grad():
            h = (self.max_t - self.min_t) / self.num_steps
            # time grid exactly as the reference's while-loop walks it (t -= h in fp64; t - h/2 as fp32 tensor op)
            times, t = [], self.max_t
            while t - 0.5 * h > self.min_t:
                t05 = float((torch.tensor(t, dtype=torch.float64).to(torch.float32) * torch.ones(1) - 0.5 * h)[0])
                times += [t, t05]
                t = t - h
            nst = len(times) // 2
            eng = StepEngine(self.cfg, model, N, self.D, self.S, times, _branch_of(self.cfg), self.eps_ratio,
                             impl=self.impl, seed=self.seed, row_offset=self.row_offset, max_calls=2 * nst + 1)
            x = get_initial_samples(N, self.D, device, self.S, self.initial_dist, initial_dist_std, eng.seed,
                                    self.row_offset)
            drift_stats = torch.zeros((max(nst, 1), nat.STAT_COUNT), dtype=torch.int64, device=eng.device)
            jump_rows = []
            for i in range(nst):
                logits = model(x.long(), eng.t_ones(2 * i))
                x_prime, _ = eng.step(nat.MODE_MIDPOINT_DRIFT, logits, x, 2 * i, h, draws=False, stats=drift_stats[i])
                logits_prime = model(x_prime.long(), eng.t_ones(2 * i + 1))
                x, row = eng.step(nat.MODE_MIDPOINT_JUMP, logits_prime, x_prime, 2 * i + 1, h,
                                  not self.is_ordinal, x_base=x)
                jump_rows.append(row)
            if self.loss_name == "CTElbo":
                x_0max = _final_argmax(model, x, self.min_t, N, device)
            else:
                x_0max = x
            st, ds = eng.stats_host(), drift_stats.cpu().numpy()
            ND = N * self.D
            change_jump = []
            if self.is_ordinal:
                for r in jump_rows:
                    j, m = st[r, nat.STAT_ROWS_JUMPED], st[r, nat.STAT_ROWS_MULTI]
                    change_jump.append(float(m) / float(j) if j else float("nan"))
            change_dim = [st[r, nat.STAT_NONZERO_JUMP] / ND for r in jump_rows]
            change_dim_first = [ds[i, nat.STAT_CHANGED_BASE] / ND for i in range(nst)]
            change_1to2 = [st[r, nat.STAT_CHANGED_EVAL] / ND for r in jump_rows]
            return (x_0max.detach().cpu().numpy().astype(int), change_jump, change_dim, change_dim_first, change_1to2)


def _pc_loop(sampler_cfg, model, N, D, S, cfg, conditioner=None, condition_dim=0, reject=False, init_std=None,
             seed=None, row_offset=0, impl=nat.IMPL_AUTO):
    """Shared body of PCTauL / ConditionalPCTauLeaping (reference sampling.py:553-646, :796-905): tauLDR rates
    whatever loss.name says, grid linspace(1, min_t + 1/num_steps, num_steps), corrector at t - h with step
    corrector_step_size_multiplier * h, final argmax always."""
    scfg = sampler_cfg
    num_steps, min_t = scfg.num_steps, scfg.min_t
    device = model.device
    h0 = 1.0 / num_steps
    ts = np.linspace(1.0, min_t + h0, num_steps)
    steps = list(enumerate(ts[0:-1]))
    times = []
    for idx, t in steps:
        times += [t, t - (ts[idx] - ts[idx + 1])]
    eng = StepEngine(cfg, model, N, D, S, times, nat.BRANCH_TAULDR, scfg.eps_ratio, impl=impl, seed=seed,
                     row_offset=row_offset, max_calls=len(steps) * (1 + scfg.num_corrector_steps) + 1)
    x = get_initial_samples(N, D, device, S, scfg.initial_dist, init_std, eng.seed, row_offset)

    def logits_of(xx, tidx):
        if conditioner is None:
            return model(xx.long(), eng.t_ones(tidx)), None
        full = model(torch.concat((conditioner, xx.long()), dim=1), eng.t_ones(tidx))
        return full, (full, condition_dim)

    for idx, t in steps:
        h = ts[idx] - ts[idx + 1]
        lg, view = logits_of(x, 2 * idx)
        x, _ = eng.step(nat.MODE_TAU_LEAP, lg, x, 2 * idx, h, reject, logits_view=view)
        if t <= scfg.corrector_entry_time:
            for _ in range(scfg.num_corrector_steps):
                lg, view = logits_of(x, 2 * idx + 1)
                x, _ = eng.step(nat.MODE_TAU_LEAP_CORR, lg, x, 2 * idx + 1, scfg.corrector_step_size_multiplier * h,
                                reject, logits_view=view)
    return x, eng


@sampling_utils.register_sampler
class PCTauL(_SamplerBase):
    """Predictor-corrector tau-leaping (reference sampling.py:529-646); returns a bare ndarray."""

    def __init__(self, cfg):
        self.cfg = cfg

    def sample(self, model, N):
        D, S = self.cfg.model.concat_dim, self.cfg.data.S
        with torch.no_grad():
            x, _ = _pc_loop(self.cfg.sampler, model, N, D, S, self.cfg, init_std=200, seed=self.seed,
                            row_offset=self.row_offset, impl=self.impl)
            x_0max = _final_argmax(model, x, self.cfg.sampler.min_t, N, model.device)
            return x_0max.detach().cpu().numpy().astype(int)


@sampling_utils.register_sampler
class ConditionalTauLeaping(_SamplerBase):
    """Prefix-conditioned tau-leaping (reference sampling.py:649-758). The reference computes the multi-jump
    rejection mask and then overwrites it (:734-744), so no rejection is applied here either (quirk B.6)."""

    def __init__(self, cfg):
        self.cfg = cfg

    def sample(self, model, N, conditioner):
        assert conditioner.shape[0] == N
        condition_dim = self.cfg.sampler.condition_dim
        total_D = self.cfg.data.shape[0]
        sample_D = total_D - condition_dim
        S = self.cfg.data.S
        scfg = self.cfg.sampler
        init_std = model.Q_sigma if scfg.initial_dist == "gaussian" else None
        device = model.device
        with torch.no_grad():
            conditioner = conditioner.to(device).long()
            ts = np.concatenate((np.linspace(1.0, scfg.min_t, scfg.num_steps), np.array([0])))
            eng = StepEngine(self.cfg, model, N, sample_D, S, ts[:-1], nat.BRANCH_TAULDR, scfg.eps_ratio,
                             impl=self.impl, seed=self.seed, row_offset=self.row_offset, max_calls=scfg.num_steps + 1)
            x = get_initial_samples(N, sample_D, device, S, scfg.initial_dist, init_std, eng.seed, self.row_offset)
            for idx, t in enumerate(ts[0:-1]):
                h = ts[idx] - ts[idx + 1]
                full = model(torch.concat((conditioner, x.long()), dim=1), eng.t_ones(idx))
                x, _ = eng.step(nat.MODE_TAU_LEAP, full, x, idx, h, False, logits_view=(full, condition_dim))
            full = model(torch.concat((conditioner, x.long()), dim=1), scfg.min_t * torch.ones((N,), device=device))
            x_0max = torch.max(F.softmax(_dense(full, S), dim=2, dtype=torch.float32)[:, condition_dim:, :], dim=2)[1]
            output = torch.concat((conditioner, x_0max), dim=1)
            return output.detach().cpu().numpy().astype(int)


@sampling_utils.register_sampler
class ConditionalPCTauLeaping(_SamplerBase):
    """Prefix-conditioned predictor-corrector tau-leaping (reference sampling.py:761-905)."""

    def __init__(self, cfg):
        self.cfg = cfg

    def sample(self, model, N, conditioner):
        assert conditioner.shape[0] == N
        condition_dim = self.cfg.sampler.condition_dim
        total_D = self.cfg.data.shape[0]
        sample_D = total_D - condition_dim
        S = self.cfg.data.S
        scfg = self.cfg.sampler
        init_std = model.Q_sigma if scfg.initial_dist == "gaussian" else None
        device = model.device
        with torch.no_grad():
            conditioner = conditioner.to(device).long()
            x, _ = _pc_loop(scfg, model, N, sample_D, S, self.cfg, conditioner=conditioner, condition_dim=condition_dim,
                            reject=bool(scfg.reject_multiple_jumps), init_std=init_std, seed=self.seed,
                            row_offset=self.row_offset, impl=self.impl)
            full = model(torch.concat((conditioner, x.long()), dim=1), scfg.min_t * torch.ones((N,), device=device))
            x_0max = torch.max(F.softmax(_dense(full, S), dim=2, dtype=torch.float32)[:, condition_dim:, :], dim=2)[1]
            output = torch.concat((conditioner, x_0max), dim=1)
            return output.detach().cpu().numpy().astype(int)


# Sampler names that the reference's configs use but its registry never had (SURVEY.md §5): map them onto the
# class that implements that algorithm so those configs run unchanged.
for _alias, _cls in (("TauLeaping", TauL), ("ElboTauL", TauL), ("LBJFSampling", LBJF), ("CRMLBJF", LBJF),
                     ("CRMTauL", TauL), ("CRMMidPointTauL", MidPointTauL), ("ElboLBJF", LBJF)):
    sampling_utils.register_alias(_alias, _cls)


@sampling_utils.register_sampler
class ExactSampling(_SamplerBase):
    """Exact one-step posterior sampling for small state spaces (reference sampling.py:975-1061):
    x_{t-h} ~ Cat_s'( sum_k p_{0|t}(k | x_t) q_{t-h|0}[k, s'] * q_{t|t-h}[s', x_t] ).

    The reference materialises an (N, D, S, S) tensor and a logsumexp per step; here the contraction, the multiply by the
    gathered q_{t|t-h} column and the categorical draw are one kernel (CTDD_MODE_EXACT).  Only `model.log_prob == 'cat'`
    networks are supported (the EBM score functions are out of scope, SURVEY.md section 2)."""

    def __init__(self, cfg):
        self.cfg = cfg
        self.D = cfg.model.concat_dim
        self.S = self.cfg.data.S
        self.num_steps = cfg.sampler.num_steps
        self.min_t = cfg.sampler.min_t
        self.initial_dist = cfg.sampler.initial_dist
        self.max_t = cfg.training.max_t
        if getattr(cfg.model, "log_prob", "cat") != "cat":
            raise NotImplementedError("ExactSampling: only model.log_prob == 'cat' is supported")

    def sample(self, model, N):
        initial_dist_std = self.cfg.model.Q_sigma
        device = torch.device(model.device)
        if device.type != "cuda":
            raise RuntimeError("ctdd_b200 samplers run on CUDA devices only; there is no CPU fallback")
        S, D = self.S, self.D
        with torch.no_grad():
            ts = np.concatenate((np.linspace(self.max_t, self.min_t, self.num_steps), np.array([0])))
            seed = _seed_from_torch() if self.seed is None else int(self.seed)
            # q_{t-h|0} and q_{t|t-h} for every step, built once (the reference builds N identical copies per step)
            t_hi = torch.tensor([float(t) for t in ts[:-1]], dtype=torch.float64).to(torch.float32).to(device)
            t_lo = torch.tensor([float(t) for t in ts[:-1]], dtype=torch.float64).to(torch.float32)
            t_lo = (t_lo - torch.tensor([float(ts[i] - ts[i + 1]) for i in range(len(ts) - 1)], dtype=torch.float64)
                    .to(torch.float32)).to(device)        # t - h in the reference's fp32 arithmetic (sampling.py:1027)
            Q = model.transition(t_lo).contiguous()
            QT = Q.transpose(1, 2).contiguous()
            W = model.transit_between(t_lo, t_hi).contiguous()       # W[i][s', x] = q_{t|t-h}[s', x]
            WT = W.transpose(1, 2).contiguous()                      # [x][s']
            Rb, _ = model.base_rate_tables(device)
            stats = torch.zeros((len(ts) - 1, nat.STAT_COUNT), dtype=torch.int64, device=device)
            x = get_initial_samples(N, D, device, S, self.initial_dist, initial_dist_std, seed, self.row_offset)
            for idx, t in enumerate(ts[0:-1]):
                logits = _dense(model(x.long(), float(t) * torch.ones((N,), device=device)), S)
                x = ops.reverse_step(nat.MODE_EXACT, nat.BRANCH_SDDM_REVERSE_PROB, logits, x, Q[idx], QT[idx], Rb, WT[idx],
                                     0.0, 0.0, 0.0, N=N, D=D, S=S, seed=seed, offset=idx, row_offset=self.row_offset,
                                     impl=nat.IMPL_SIMT, stats=stats[idx])["x"]
            st = stats.cpu().numpy()
            change_jump = [st[i, nat.STAT_CHANGED_EVAL] / (N * D) for i in range(len(ts) - 1)]
            return x.detach().cpu().numpy().astype(int), change_jump

