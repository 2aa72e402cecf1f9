"""Thin tensor-level wrappers over the C ABI (include/ctdd.h): explicit tables in, tensors out.

The sampler / loss classes in lib/ build on these; tests call them directly to inject the oracle's q_{t|0}.
"""
from __future__ import annotations

import torch

from . import _native as nat

# dtypes of (N, D, S) logits and of their gradients that the kernels read and write as they are (2-byte ones are widened
# on load, exactly); any other dtype is widened to an fp32 copy first
_LOGITS_DTYPES = (torch.float32, torch.bfloat16, torch.float16)


@nat.on_tensor_device
def build_qt0(U, Uinv, lam, d_int, normalize=True, clamp_below=1e-8, want_transpose=False):
    """Q_b = U diag(exp(lam*d_int[b])) Uinv -> (B,S,S) [and Q^T]."""
    B, S = d_int.shape[0], U.shape[0]
    Q = torch.empty((B, S, S), dtype=torch.float32, device=d_int.device)
    QT = torch.empty_like(Q) if want_transpose else None
    nat.check(nat.lib().ctdd_build_qt0(nat.ptr(U), nat.ptr(Uinv), nat.ptr(lam), nat.ptr(d_int.contiguous()), B, S,
                                       1 if normalize else 0, clamp_below, nat.ptr(Q), nat.ptr(QT), nat.stream()),
              "ctdd_build_qt0")
    return (Q, QT) if want_transpose else Q


@nat.on_tensor_device
def prep_tc_tables(Q, QT, Rb, eps, branch):
    """Per-time-point tables of the tcgen05 path; Q/QT are (T,S,S). Returns a (T, bytes) uint8 tensor or None."""
    T, S = Q.shape[0], Q.shape[-1]
    nbytes = int(nat.lib().ctdd_tc_tables_bytes(S))
    if nbytes <= 0:
        return None
    out = torch.empty((T, nbytes), dtype=torch.uint8, device=Q.device)
    nat.check(nat.lib().ctdd_prep_tc_tables(nat.ptr(Q), nat.ptr(QT), nat.ptr(Rb), T, S, float(eps), branch, nat.ptr(out),
                                            nat.stream()), "ctdd_prep_tc_tables")
    return out


@nat.on_tensor_device
def prep_tc_static(Rb):
    """Time-independent tables of the tcgen05 path (uint8 blob) or None when the path is unavailable for this S."""
    S = Rb.shape[-1]
    nbytes = int(nat.lib().ctdd_tc_static_bytes(S))
    if nbytes <= 0:
        return None
    # the blob must sit on a ctdd_tc_static_align() boundary: over-allocate and take the aligned window (a view, so the
    # storage stays alive with it)
    align = int(nat.lib().ctdd_tc_static_align())
    buf = torch.empty((nbytes + align,), dtype=torch.uint8, device=Rb.device)
    skip = (-buf.data_ptr()) % align
    out = buf[skip:skip + nbytes]
    nat.check(nat.lib().ctdd_prep_tc_static(nat.ptr(Rb), S, nat.ptr(out), nat.stream()), "ctdd_prep_tc_static")
    return out


@nat.on_tensor_device
def reverse_step(mode, branch, logits, x_eval, Q, QT, Rb, RbT, beta, h, eps, *, N, D, S, x_base=None,
                 reject_multi=False, seed=0, offset=0, row_offset=0, impl=nat.IMPL_AUTO, tc_tables=None, tc_static=None,
                 workspace=None, stats=None, want_rr=False, want_ratio=False, logits_offset_elems=0,
                 batch_stride=None, head=None, x_out=None):
    """One fused reverse-rate evaluation (+ state update). Returns dict(x=..., rr=..., ratio=...).

    `head=(mu, log_scale, fix_logistic)` replaces `logits` (pass None) by the parameters of the truncated-logistic
    output head (reference lib/models/models.py:248-282): mu / log_scale are (N, D)-shaped views whose batch
    stride may exceed D (the two torch.chunk halves of a (B, 2C, H, W) network output), fp32, or bf16 both (read as
    they are; any other dtype is widened to fp32).  On the tcgen05 path the logits are never materialised; elsewhere
    they are built once with `logistic_logits`, as fp32.  Dense `logits` are read as they are in fp32, bf16 or fp16."""
    dev = x_eval.device
    head_kind, head_mu, head_ls, head_bs, head_dt = nat.HEAD_LOGITS, None, None, 0, nat.DTYPE_F32
    if head is not None:
        mu, ls, fix = head
        mu, ls, head_bs, head_dt = _head_views(mu, ls, N, D)
        use_tc = S == 256 and tc_tables is not None and impl != nat.IMPL_SIMT and mode != nat.MODE_EXACT and \
            branch in (nat.BRANCH_TAULDR, nat.BRANCH_SDDM_REVERSE_PROB)
        if use_tc:
            head_kind, head_mu, head_ls = (nat.HEAD_LOGISTIC_FIX if fix else nat.HEAD_LOGISTIC), mu, ls
            logits = None
        else:
            logits = logistic_logits(mu, ls, S, fix)
    if logits is not None:
        if logits.dtype not in _LOGITS_DTYPES:     # bf16 / fp16 are read as they are (widened on load, exactly)
            logits = logits.float()
        logits = logits.contiguous()
    if mode == nat.MODE_RATES_ONLY:
        x_out = None
    elif x_out is None:
        x_out = torch.empty((N, D), dtype=torch.int32, device=dev)
    elif x_out.dtype != torch.int32 or tuple(x_out.shape) != (N, D) or not x_out.is_contiguous():
        raise ValueError("x_out must be a contiguous (N, D) int32 tensor")
    rr = torch.empty((N, D, S), dtype=torch.float32, device=dev) if want_rr else None
    ratio = torch.empty((N, D, S), dtype=torch.float32, device=dev) if want_ratio else None
    if workspace is None:
        ws = int(nat.lib().ctdd_step_workspace_bytes(N * D, S, impl))
        workspace = torch.empty((ws,), dtype=torch.uint8, device=dev) if ws > 0 else None
    p = nat.StepParams(
        mode=mode, branch=branch, impl=impl, N=N, D=D, S=S, row_offset=int(row_offset),
        logits=(nat.ptr(logits) + logits.element_size() * int(logits_offset_elems)) if logits is not None else None, ld_logits=S,
        batch_stride_logits=(int(batch_stride) if batch_stride is not None else D * S),
        x_eval=nat.ptr(x_eval), x_base=nat.ptr(x_base),
        Q=nat.ptr(Q), QT=nat.ptr(QT), Rb=nat.ptr(Rb), RbT=nat.ptr(RbT), tc_tables=nat.ptr(tc_tables), tc_static=nat.ptr(tc_static),
        beta=float(beta), h=float(h), eps=float(eps), reject_multi=1 if reject_multi else 0,
        seed=int(seed), offset=int(offset),
        x_out=nat.ptr(x_out), rr_out=nat.ptr(rr), ratio_out=nat.ptr(ratio),
        stats_out=(stats.data_ptr() if stats is not None else None), workspace=nat.ptr(workspace),
        head=head_kind, head_mu=(head_mu.data_ptr() if head_mu is not None else None),
        head_log_scale=(head_ls.data_ptr() if head_ls is not None else None), head_batch_stride=int(head_bs),
        logits_dtype=(nat.logits_dtype_of(logits) if logits is not None else nat.DTYPE_F32), head_dtype=head_dt)
    nat.check(nat.lib().ctdd_reverse_step(p, nat.stream()), "ctdd_reverse_step")
    return {"x": x_out, "rr": rr, "ratio": ratio}


class _LogisticLogitsFn(torch.autograd.Function):
    """Differentiable truncated-logistic head: forward `ctdd_logistic_logits_ex`, backward `ctdd_logistic_logits_backward_ex`
    (recomputes the head from its two inputs; nothing of size (N, D, S) is saved).

    bf16 (mu, log_scale) are saved and read as they are, and an fp32, bf16 or fp16 incoming gradient is read as it is;
    other dtypes are widened to fp32 copies.  The kernels widen on load, so the gradients equal those of the fp32 call on the
    widened tensors bit for bit; they are returned in the inputs' dtypes."""

    @staticmethod
    def forward(ctx, mu, log_scale, S, fix_logistic, out_dtype):
        N = mu.shape[0]
        D = mu.numel() // N
        mu_c = mu.detach().reshape(N, D).contiguous()
        ls_c = log_scale.detach().reshape(N, D).contiguous()
        if not (mu_c.dtype == torch.bfloat16 and ls_c.dtype == torch.bfloat16):
            mu_c, ls_c = mu_c.float(), ls_c.float()
        ctx.save_for_backward(mu_c, ls_c)
        ctx.meta = (S, bool(fix_logistic), tuple(mu.shape), mu.dtype, log_scale.dtype)
        return logistic_logits(mu_c, ls_c, S, fix_logistic, out_dtype=out_dtype)

    @staticmethod
    @nat.on_tensor_device
    def backward(ctx, grad_logits):
        mu_c, ls_c = ctx.saved_tensors
        S, fix, shape, dt_mu, dt_ls = ctx.meta
        N, D = mu_c.shape
        g = grad_logits.contiguous()
        if g.dtype not in _LOGITS_DTYPES:
            g = g.float()
        elif g.dtype != torch.float32 and g.data_ptr() % 8:
            # the kernel's accumulation order depends on 4-element alignment: keep the order of an aligned fp32 gradient
            g = g.clone()
        dmu = torch.empty((N, D), dtype=torch.float32, device=mu_c.device)
        dls = torch.empty_like(dmu)
        nat.check(nat.lib().ctdd_logistic_logits_backward_ex(mu_c.data_ptr(), ls_c.data_ptr(), nat.logits_dtype_of(mu_c),
                                                             nat.ptr(g), nat.logits_dtype_of(g), N, D, D, S,
                                                             1 if fix else 0, dmu.data_ptr(), dls.data_ptr(), nat.stream()),
                  "ctdd_logistic_logits_backward_ex")
        return dmu.view(shape).to(dt_mu), dls.view(shape).to(dt_ls), None, None, None


@nat.on_tensor_device
def logistic_logits_autograd(mu, log_scale, S, fix_logistic=False, out_dtype=None):
    """(N, D, S) logits of the head, differentiable w.r.t. mu and log_scale (training path).  `out_dtype` is
    torch.float32 (the default, None), torch.bfloat16 or torch.float16: the fp32 logits rounded once to that type,
    which is what the 2-byte loss path (`loss_terms`) reads; its gradient then arrives in that type and is read as it
    is."""
    return _LogisticLogitsFn.apply(mu, log_scale, S, fix_logistic, torch.float32 if out_dtype is None else out_dtype)


# Opt-in for the un-materialised head: only code that knows how to consume an ops.LogisticHead (this package's samplers,
# which fuse it into the reverse-step kernel) switches it on; every other caller of model(x, t) gets the (B, D, S) logits
# tensor the reference returns.
import contextlib
import threading

_head_mode = threading.local()


def fused_head_enabled() -> bool:
    return bool(getattr(_head_mode, "on", False))


@contextlib.contextmanager
def fused_head(on: bool = True):
    """Inside this context a TruncatedLogisticHead model evaluated without gradients returns an ops.LogisticHead (the two
    numbers per dimension) instead of the (B, D, S) logits."""
    prev = fused_head_enabled()
    _head_mode.on = bool(on)
    try:
        yield
    finally:
        _head_mode.on = prev


class LogisticHead:
    """What a model's forward may return instead of (N, D, S) logits when its output layer is the truncated-logistic
    head (reference lib/models/models.py:248-282, cfg.model.model_output == 'logistic_pars'): the two numbers per
    dimension the network emits.  The samplers hand them to the fused reverse step, so the logits are never
    materialised; `.logits(S)` builds them (one kernel) for the callers that need the tensor (final argmax)."""

    def __init__(self, mu, log_scale, fix_logistic=False):
        if mu.shape != log_scale.shape:
            raise ValueError(f"mu {tuple(mu.shape)} and log_scale {tuple(log_scale.shape)} differ in shape")
        self.mu, self.log_scale, self.fix_logistic = mu, log_scale, bool(fix_logistic)

    def flat(self):
        """(N, D) views (no copy for contiguous tensors or torch.chunk halves)."""
        N = self.mu.shape[0]
        return self.mu.reshape(N, -1) if self.mu[0].is_contiguous() else self.mu.contiguous().view(N, -1), \
            self.log_scale.reshape(N, -1) if self.log_scale[0].is_contiguous() else self.log_scale.contiguous().view(N, -1)

    def slice_dims(self, c):
        """The head of dimensions c.. (conditional samplers keep the first c dimensions fixed)."""
        mu, ls = self.flat()
        return LogisticHead(mu[:, c:], ls[:, c:], self.fix_logistic)

    def logits(self, S):
        mu, ls = self.flat()
        return logistic_logits(mu, ls, S, self.fix_logistic)

    def as_tuple(self):
        mu, ls = self.flat()
        return mu, ls, self.fix_logistic


def _head_views(mu, ls, N, D):
    """(mu, log_scale) as CUDA tensors addressable as base[n * batch_stride + d]; returns (mu, ls, batch_stride, dtype)
    with dtype nat.DTYPE_BF16 when both are bf16 (read as they are; the kernels widen on load) and nat.DTYPE_F32
    otherwise (any other dtype, or a bf16 / fp32 mix, is widened to fp32).  Accepts (N, D) or (N, C, H, W) tensors,
    contiguous or the two halves of torch.chunk(out, 2, dim=1)."""
    keep = mu.dtype == torch.bfloat16 and ls.dtype == torch.bfloat16

    def flat(t):
        if not t.is_cuda:
            raise RuntimeError("ctdd_b200 kernels need CUDA tensors; got a host tensor (there is no CPU fallback)")
        if not keep and t.dtype != torch.float32:
            t = t.float()
        if t.shape[0] != N or t.numel() != N * D:
            raise ValueError(f"head tensor of shape {tuple(t.shape)} does not hold N={N} x D={D} values")
        inner = t[0]
        if N > 1 and not inner.is_contiguous():
            t = t.contiguous()
        elif N == 1 and not t.is_contiguous():
            t = t.contiguous()
        return t, (t.stride(0) if N > 1 else D)
    mu, bs_mu = flat(mu)
    ls, bs_ls = flat(ls)
    if bs_mu != bs_ls:
        mu, ls, bs_mu = mu.contiguous(), ls.contiguous(), D
    return mu, ls, bs_mu, (nat.DTYPE_BF16 if keep else nat.DTYPE_F32)


_OUT_DTYPES = {torch.float32: nat.DTYPE_F32, torch.bfloat16: nat.DTYPE_BF16, torch.float16: nat.DTYPE_F16}


@nat.on_tensor_device
def logistic_logits(mu, log_scale, S, fix_logistic=False, out=None, out_dtype=torch.float32):
    """Truncated-logistic head -> (N, D, S) logits in one pass (replaces sample_logistic, models.py:28-74).

    bf16 (mu, log_scale) are read as they are; the logits are computed in fp32 either way and stored as `out_dtype`
    (torch.float32, or torch.bfloat16 / torch.float16: rounded once to nearest even)."""
    if out_dtype not in _OUT_DTYPES:
        raise ValueError(f"logistic_logits: out_dtype must be torch.float32, torch.bfloat16 or torch.float16, got {out_dtype}")
    N = mu.shape[0]
    D = mu.numel() // N
    mu, ls, bs, in_dt = _head_views(mu, log_scale, N, D)
    if out is None:
        out = torch.empty((N, D, S), dtype=out_dtype, device=mu.device)
    elif out.shape != (N, D, S) or out.dtype != out_dtype:
        raise ValueError(f"out must be a {out_dtype} ({N}, {D}, {S}) tensor")
    nat.check(nat.lib().ctdd_logistic_logits_ex(mu.data_ptr(), ls.data_ptr(), in_dt, N, D, int(bs), S,
                                                1 if fix_logistic else 0, nat.ptr(out), _OUT_DTYPES[out_dtype],
                                                nat.stream()), "ctdd_logistic_logits_ex")
    return out


def _as_f32_rows(x):
    if x.dim() != 2:
        x = x.reshape(x.shape[0], -1)
    return x.to(torch.float32).contiguous()


@nat.on_tensor_device
def pair_similarity(x, y, bd=0.1, hamming=False):
    """(N, M) matrix exp(-bd * sum_d |x_d - y_d|) (or D - sum_d |.| with hamming=True), metrics.py:6-22."""
    x, y = _as_f32_rows(x), _as_f32_rows(y)
    if x.shape[1] != y.shape[1]:
        raise ValueError("pair_similarity: x and y differ in the number of dimensions")
    K = torch.empty((x.shape[0], y.shape[0]), dtype=torch.float32, device=x.device)
    if K.numel():
        nat.check(nat.lib().ctdd_pair_similarity(nat.ptr(x), x.shape[0], nat.ptr(y), y.shape[0], x.shape[1], float(bd),
                                                 1 if hamming else 0, nat.ptr(K), nat.stream()), "ctdd_pair_similarity")
    return K


@nat.on_tensor_device
def pair_similarity_sums(x, y, bd=0.1, hamming=False):
    """float64 tensor (3,): sum_{i != j} k(x_i, x_j), sum_{i != j} k(y_i, y_j), sum_{i, j} k(x_i, y_j) — the three sums
    of binary_mmd (metrics.py:25-48), no (N, M) or (N, M, D) tensor."""
    x, y = _as_f32_rows(x), _as_f32_rows(y)
    if x.shape[1] != y.shape[1]:
        raise ValueError("pair_similarity_sums: x and y differ in the number of dimensions")
    nat.ptr(x), nat.ptr(y)
    L = nat.lib()
    N, M, D = x.shape[0], y.shape[0], x.shape[1]
    out = torch.empty(3, dtype=torch.float64, device=x.device)
    scratch = torch.empty(max(1, int(L.ctdd_pair_partials(max(N, M), max(N, M)))), dtype=torch.float64, device=x.device)
    for slot, (a, na, b, nb, self_) in enumerate(((x, N, x, N, 1), (y, M, y, M, 1), (x, N, y, M, 0))):
        nat.check(L.ctdd_pair_similarity_sum(a.data_ptr(), na, b.data_ptr(), nb, D, float(bd), self_, 1 if hamming else 0,
                                             scratch.data_ptr(), out.data_ptr() + 8 * slot, nat.stream()),
                  "ctdd_pair_similarity_sum")
    return out


@nat.on_tensor_device
def state_histogram(x, S, counts=None):
    """Per-dimension state counts of samples x (N, D) -> int32 (D, S); pass `counts` (from an earlier call) to accumulate.
    Raises if any state lies outside [0, S)."""
    if x.dim() != 2:
        x = x.reshape(x.shape[0], -1)
    x = x.to(torch.int32).contiguous()
    N, D = x.shape
    buf = torch.zeros(D * S + 1, dtype=torch.int32, device=x.device)
    nat.check(nat.lib().ctdd_state_histogram(nat.ptr(x), N, D, S, nat.ptr(buf), nat.stream()), "ctdd_state_histogram")
    if int(buf[-1]) != 0:
        raise ValueError(f"state_histogram: {int(buf[-1])} states outside [0, {S})")
    h = buf[:-1].view(D, S)
    if counts is not None:
        counts += h
        return counts
    return h


class EmaTable:
    """Device table of (shadow, param, n) chunk records for `ctdd_ema_update` — every trainable tensor of a model is
    updated in ONE launch (replaces the per-parameter loop of EMA.update_ema, reference lib/models/models.py:745-758).

    The table is built once and rebuilt only when a tensor moved (load_state_dict replaces the shadow list, `.to()`
    re-allocates parameters): `matches()` compares the recorded data pointers."""

    def __init__(self, shadows, params):
        if len(shadows) != len(params):
            raise ValueError("EMA: shadow and parameter lists differ in length")
        chunk = int(nat.lib().ctdd_ema_chunk_elems())
        recs, dev = [], None
        for s, p in zip(shadows, params):
            if s.shape != p.shape:
                raise ValueError(f"EMA: shadow {tuple(s.shape)} vs parameter {tuple(p.shape)}")
            if s.dtype != torch.float32 or p.dtype != torch.float32:
                raise RuntimeError("ctdd_ema_update handles float32 parameters only")
            nat.ptr(s), nat.ptr(p)          # CUDA + contiguous, or raise: there is no CPU path
            if dev is None:
                dev = s.device
            if s.device != dev or p.device != dev:
                raise RuntimeError("EMA: all shadow tensors and parameters must live on one device")
            n, sp, pp = s.numel(), s.data_ptr(), p.data_ptr()
            for o in range(0, n, chunk):
                recs.append((sp + 4 * o, pp + 4 * o, min(chunk, n - o)))
        self.key = self._key(shadows, params)
        self.n_chunks = len(recs)
        self.elements = sum(r[2] for r in recs)
        self.table = (torch.tensor(recs, dtype=torch.int64).to(dev) if recs else None)

    @staticmethod
    def _key(shadows, params):
        return tuple(t.data_ptr() for t in shadows) + tuple(t.data_ptr() for t in params)

    def matches(self, shadows, params):
        return self.key == self._key(shadows, params)

    def update(self, one_minus_decay):
        """shadow <- shadow - one_minus_decay * (shadow - param), in place, on the current stream."""
        if self.n_chunks:
            with nat.on_device(self.table.device):
                nat.check(nat.lib().ctdd_ema_update(self.table.data_ptr(), self.n_chunks, float(one_minus_decay), nat.stream()),
                          "ctdd_ema_update")


@nat.on_tensor_device
def sample_categorical_shared(probs, rows, seed, offset=0, row_offset=0):
    x = torch.empty((rows,), dtype=torch.int32, device=probs.device)
    nat.check(nat.lib().ctdd_sample_categorical_shared(nat.ptr(probs.contiguous()), probs.shape[0], rows, row_offset,
                                                       int(seed), int(offset), nat.ptr(x), nat.stream()),
              "ctdd_sample_categorical_shared")
    return x


@nat.on_tensor_device
def noise_xt(Q, Rb, beta, x0, seed, offset=0, batch_offset=0, want_tilde=True):
    """x_t ~ Cat(Q[b, x0, :]) and the one-jump proposal x~ (lib/losses/losses.py:46-101). x0: (B,D) int32."""
    B, D = x0.shape
    S = Q.shape[-1]
    xt = torch.empty((B, D), dtype=torch.int32, device=x0.device)
    xtilde = torch.empty_like(xt) if want_tilde else None
    nat.check(nat.lib().ctdd_noise_xt(nat.ptr(Q.contiguous()), nat.ptr(Rb), nat.ptr(beta.contiguous()) if beta is not None else None,
                                      nat.ptr(x0.contiguous()), B, D, S, int(batch_offset), int(seed), int(offset),
                                      nat.ptr(xt), nat.ptr(xtilde), nat.stream()), "ctdd_noise_xt")
    return xt, xtilde


@nat.on_tensor_device
def bgemm256(X, M, out=None):
    """out[b,d,n] = sum_k X[b,d,k] * M[b,n,k] on tcgen05 (S = 256; 3 x BF16 split precision).  X: (B,D,256), M: (B,256,256)."""
    B, D, S = X.shape
    if S != 256 or tuple(M.shape) != (B, 256, 256):
        raise ValueError(f"bgemm256 needs X (B,D,256) and M (B,256,256); got {tuple(X.shape)}, {tuple(M.shape)}")
    X = X.contiguous().float()
    M = M.contiguous().float()
    if out is None:
        out = torch.empty((B, D, S), dtype=torch.float32, device=X.device)
    nat.check(nat.lib().ctdd_bgemm256_tc(nat.ptr(X), nat.ptr(M), B, D, nat.ptr(out), nat.stream()), "ctdd_bgemm256_tc")
    return out


class _LossTerms(torch.autograd.Function):
    """Per-sample loss terms (out_a, out_b, out_c, out_d, out_nll), each (B,), differentiable w.r.t. `logits`
    through the fused backward kernel (include/ctdd.h: ctdd_loss_forward / ctdd_loss_backward).

    fp32, bf16 and fp16 logits are read as they are; bf16 and fp16 ones (a network under torch.autocast, with
    dtype=torch.bfloat16 or its default fp16) get a gradient of their own dtype, equal to the fp32 gradient of their
    widening rounded once to that dtype (fp16: +-inf where it overflows, which a GradScaler detects).  Other dtypes are
    widened to an fp32 copy and autograd casts the gradient back."""
    #: S == 256: run the two contractions on tcgen05 (set False to force the CUDA-core kernel, e.g. as a cross-check)
    use_tc = True

    @staticmethod
    def forward(ctx, logits, kind, logit_branch, crm_type, Q, QT, Rb, beta, x0, xt, x_tilde, eps):
        B, D, S = logits.shape
        dev = logits.device
        if logits.dtype in (torch.bfloat16, torch.float16):
            logits = logits.contiguous()
            if logits.data_ptr() % 16:          # e.g. a contiguous view at an odd storage offset: 16-byte rows needed
                logits = logits.clone()
        else:
            logits = logits.contiguous().float()
        outs = torch.zeros((5, B), dtype=torch.float32, device=dev)
        nbytes = int(nat.lib().ctdd_loss_workspace_bytes(kind, B, S))
        ws = torch.empty((max(nbytes, 4),), dtype=torch.uint8, device=dev)
        # S == 256: scratch of the tensor-core contractions (u = A Q is kept in it for the backward call)
        wants_tc = _LossTerms.use_tc and kind != nat.LOSS_CTELBO and logit_branch != nat.BRANCH_SDDM_DIRECT
        nscr = int(nat.lib().ctdd_loss_tc_scratch_bytes(B, D, S)) if wants_tc else 0
        scr = torch.empty((nscr,), dtype=torch.uint8, device=dev) if nscr > 0 else None
        p = nat.LossParams(kind=kind, logit_type=logit_branch, crm_type=crm_type, B=B, D=D, S=S,
                           logits=nat.ptr(logits), Q=nat.ptr(Q), QT=nat.ptr(QT), Rb=nat.ptr(Rb), beta=nat.ptr(beta),
                           x0=nat.ptr(x0), xt=nat.ptr(xt), x_tilde=nat.ptr(x_tilde), eps=float(eps),
                           out_a=outs[0].data_ptr(), out_b=outs[1].data_ptr(), out_c=outs[2].data_ptr(),
                           out_d=outs[3].data_ptr(), out_nll=outs[4].data_ptr(), workspace=nat.ptr(ws),
                           tc_scratch=nat.ptr(scr), logits_dtype=nat.logits_dtype_of(logits))
        nat.check(nat.lib().ctdd_loss_forward(p, nat.stream()), "ctdd_loss_forward")
        ctx.scr = scr
        ctx.save_for_backward(logits, Q, QT, Rb, beta, x0, xt, x_tilde if x_tilde is not None else xt, ws)
        ctx.meta = (kind, logit_branch, crm_type, float(eps), x_tilde is not None)
        return outs[0], outs[1], outs[2], outs[3], outs[4]

    @staticmethod
    def backward(ctx, ga, gb, gc, gd, gn):
        with nat.on_device(ctx.saved_tensors[0].device):
            return _LossTerms._backward(ctx, ga, gb, gc, gd, gn)

    @staticmethod
    def _backward(ctx, ga, gb, gc, gd, gn):
        logits, Q, QT, Rb, beta, x0, xt, x_tilde, ws = ctx.saved_tensors
        kind, logit_branch, crm_type, eps, has_tilde = ctx.meta
        B, D, S = logits.shape
        z = lambda g: (g if g is not None else torch.zeros((B,), device=logits.device)).contiguous().float()
        ga, gb, gd, gn = z(ga), z(gb), z(gd), z(gn)
        grad = torch.empty_like(logits)             # the logits' dtype: bf16 / fp16 logits get a bf16 / fp16 gradient
        p = nat.LossParams(kind=kind, logit_type=logit_branch, crm_type=crm_type, B=B, D=D, S=S,
                           logits=nat.ptr(logits), Q=nat.ptr(Q), QT=nat.ptr(QT), Rb=nat.ptr(Rb), beta=nat.ptr(beta),
                           x0=nat.ptr(x0), xt=nat.ptr(xt), x_tilde=(nat.ptr(x_tilde) if has_tilde else None), eps=eps,
                           ga=nat.ptr(ga), gb=nat.ptr(gb), gd=nat.ptr(gd), gn=nat.ptr(gn), grad_logits=nat.ptr(grad),
                           workspace=nat.ptr(ws), tc_scratch=nat.ptr(ctx.scr), logits_dtype=nat.logits_dtype_of(logits))
        nat.check(nat.lib().ctdd_loss_backward(p, nat.stream()), "ctdd_loss_backward")
        return (grad,) + (None,) * 11


@nat.on_tensor_device
def loss_terms(logits, kind, Q, QT, Rb, beta, x0, xt, x_tilde=None, eps=1e-9, logit_branch=nat.BRANCH_SDDM_REVERSE_PROB,
               crm_type=0):
    """(out_a, out_b, out_c, out_d, out_nll) per sample — see ctdd_loss_params in include/ctdd.h."""
    return _LossTerms.apply(logits, kind, logit_branch, crm_type, Q.contiguous(), QT.contiguous(), Rb, beta.contiguous().float(),
                            x0.contiguous(), xt.contiguous(), x_tilde.contiguous() if x_tilde is not None else None, eps)
