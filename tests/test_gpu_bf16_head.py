"""bf16 (mu, log_scale) in the truncated-logistic head: the standalone head (forward and backward), the head fused into the
reverse step and its non-fused fallbacks, the samplers and the training path under torch.autocast.  The bar is bit
equality with the same call on the widened fp32 tensors; a bf16 logits output is that call's fp32 output rounded to bf16."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import cases, head_oracle as ho, ref_harness as rh
from oracle.make_golden_head import FWD, HEAD_SAMPLERS
from helpers import oracle_forward, product_model, fwd_cfg

gpu = pytest.mark.gpu
bf16 = torch.bfloat16


def _nat():
    from ctdd_b200 import _native as nat
    return nat


def _inputs(N, D, seed, lo=-3.0, hi=3.0):
    """(N, D) bf16 (mu, log_scale) on the device."""
    mu, ls = ho.head_inputs(N * D, seed, lo, hi)
    return mu.view(N, D).to(bf16).cuda(), ls.view(N, D).to(bf16).cuda()


# rows outside what tanh emits (|mu| >= 1) and extreme scales (test_gpu_head.test_fused_head_edge_rows)
EDGE_MU = [1.0, -1.0, 0.0, 2.5, -3.0, 0.999, -0.2, 0.3, 1.5, -1.5, 0.7, -0.7, 0.1, 40.0, -40.0, 0.0]
EDGE_LS = [0.0, 0.0, -6.0, -2.0, -2.0, 6.0, 8.0, -8.0, 3.0, 3.0, -4.0, 1.0, 2.0, -1.0, -1.0, 12.0]


def _edge_inputs():
    return (torch.tensor(EDGE_MU).view(1, -1).to(bf16).cuda(), torch.tensor(EDGE_LS).view(1, -1).to(bf16).cuda())


# ------------------------------------------------------------------------------------------------------- head forward
@gpu
@pytest.mark.parametrize("S", [256, 32, 5])
def test_head_forward_bf16_inputs_and_output(S):
    """bf16 inputs: fp32 logits equal the fp32 call on the widened inputs bit for bit, bf16 logits equal those rounded
    to bf16; random rows, the edge rows, and the two torch.chunk halves of a (B, 2C, H, W) tensor."""
    from ctdd_b200 import ops
    mu, ls = _inputs(6, 50, 11 + S)
    em, el = _edge_inputs()
    both = torch.cat([mu.view(6, 2, 5, 5), ls.view(6, 2, 5, 5)], dim=1)          # (B, 2C, H, W)
    cm, cl = torch.chunk(both, 2, dim=1)
    assert not cm.is_contiguous()
    for fix in (False, True):
        for m, l in ((mu, ls), (em, el), (cm, cl)):
            ref = ops.logistic_logits(m.float(), l.float(), S, fix)
            got = ops.logistic_logits(m, l, S, fix)
            assert got.dtype == torch.float32 and torch.equal(got, ref), (S, fix)
            got16 = ops.logistic_logits(m, l, S, fix, out_dtype=bf16)
            assert got16.dtype == bf16 and torch.equal(got16, ref.to(bf16)), (S, fix)
            # fp32 inputs with a bf16 output: the same rounding
            assert torch.equal(ops.logistic_logits(m.float(), l.float(), S, fix, out_dtype=bf16), ref.to(bf16))
        assert torch.isfinite(ops.logistic_logits(em, el, S, fix)).all()
        # LogisticHead.logits (final argmax, evaluation) reads the bf16 head as it is
        assert torch.equal(ops.LogisticHead(cm, cl, fix).logits(S), ops.LogisticHead(cm.float(), cl.float(), fix).logits(S))


@gpu
@pytest.mark.parametrize("out_dtype", [torch.float32, bf16])
def test_head_forward_misaligned_output(out_dtype):
    """An output one element off its 4-element alignment takes the one-logit-per-thread kernel: same values."""
    from ctdd_b200 import ops
    N, D, S = 3, 40, 256
    mu, ls = _inputs(N, D, 5)
    ref = ops.logistic_logits(mu.float(), ls.float(), S, True).to(out_dtype)
    buf = torch.zeros(N * D * S + 1, dtype=out_dtype, device="cuda")
    out = buf[1:].view(N, D, S)
    assert out.data_ptr() % 8 != 0
    got = ops.logistic_logits(mu, ls, S, True, out=out, out_dtype=out_dtype)
    assert got.data_ptr() == out.data_ptr() and torch.equal(got, ref)


# ------------------------------------------------------------------------------------------------------- head backward
def _raw_backward(mu, ls, g, S, fix):
    """ctdd_logistic_logits_backward_ex on (N, D) inputs and (N, D, S) gradient of fp32 / bf16: fp32 (dmu, dls)."""
    nat = _nat()
    N, D = mu.shape
    dmu = torch.empty((N, D), dtype=torch.float32, device="cuda")
    dls = torch.empty_like(dmu)
    nat.check(nat.lib().ctdd_logistic_logits_backward_ex(mu.data_ptr(), ls.data_ptr(), nat.logits_dtype_of(mu), g.data_ptr(),
                                                         nat.logits_dtype_of(g), N, D, D, S, 1 if fix else 0,
                                                         dmu.data_ptr(), dls.data_ptr(), nat.stream()), "backward_ex")
    return dmu, dls


def _fp32_backward(mu, ls, g, S, fix):
    """The fp32 entry point on widened copies."""
    nat = _nat()
    mu, ls, g = mu.float().contiguous(), ls.float().contiguous(), g.float().contiguous()
    N, D = mu.shape
    dmu, dls = torch.empty_like(mu), torch.empty_like(ls)
    nat.check(nat.lib().ctdd_logistic_logits_backward(mu.data_ptr(), ls.data_ptr(), g.data_ptr(), N, D, D, S, 1 if fix else 0,
                                                      dmu.data_ptr(), dls.data_ptr(), nat.stream()), "backward")
    return dmu, dls


@gpu
@pytest.mark.parametrize("S", [256, 32, 5])
def test_head_backward_every_dtype_combination(S):
    """bf16 / fp32 inputs x bf16 / fp32 incoming gradient: grad_mu / grad_log_scale (fp32, before any cast) equal the fp32
    kernel's on the widened tensors bit for bit; the autograd function returns them cast to the inputs' dtype."""
    from ctdd_b200 import ops
    N, D = 6, 50
    mu, ls = _inputs(N, D, 31 + S, -2.5, 2.5)
    em, el = _edge_inputs()
    gen = torch.Generator(device="cuda").manual_seed(S)
    for m16, l16 in ((mu, ls), (em, el)):
        n, d = m16.shape
        g32 = torch.randn((n, d, S), generator=gen, device="cuda")
        g16 = g32.to(bf16)
        for fix in (False, True):
            want = _fp32_backward(m16, l16, g16, S, fix)
            for m, l in ((m16, l16), (m16.float(), l16.float())):
                for g in (g16, g16.float()):
                    got = _raw_backward(m, l, g, S, fix)
                    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), (S, fix, m.dtype, g.dtype)
                    assert torch.isfinite(got[0]).all() and torch.isfinite(got[1]).all()
            # autograd: bf16 leaves, bf16 logits, bf16 upstream gradient
            mc, lc = m16.clone().requires_grad_(True), l16.clone().requires_grad_(True)
            out = ops.logistic_logits_autograd(mc, lc, S, fix, out_dtype=bf16)
            assert out.dtype == bf16 and torch.equal(out, ops.logistic_logits(m16.float(), l16.float(), S, fix).to(bf16))
            out.backward(g16)
            assert mc.grad.dtype == bf16 and torch.equal(mc.grad, want[0].to(bf16))
            assert lc.grad.dtype == bf16 and torch.equal(lc.grad, want[1].to(bf16))


@gpu
def test_head_backward_misaligned_bf16_gradient():
    """A bf16 incoming gradient one element off 8-byte alignment: the autograd function realigns it, so the result is
    that of the aligned fp32 gradient."""
    from ctdd_b200 import ops
    N, D, S = 4, 30, 256
    mu, ls = _inputs(N, D, 3)
    g = torch.randn((N, D, S), device="cuda").to(bf16)
    buf = torch.zeros(N * D * S + 1, dtype=bf16, device="cuda")
    buf[1:] = g.reshape(-1)
    gv = buf[1:].view(N, D, S)
    assert gv.data_ptr() % 8 != 0
    mc, lc = mu.clone().requires_grad_(True), ls.clone().requires_grad_(True)
    ops.logistic_logits_autograd(mc, lc, S, False, out_dtype=bf16).backward(gv)
    want = _fp32_backward(mu, ls, g, S, False)
    assert torch.equal(mc.grad, want[0].to(bf16)) and torch.equal(lc.grad, want[1].to(bf16))


# ------------------------------------------------------------------------------------------------------- fused step
def _tables(fp, t):
    tt = torch.tensor([t], dtype=torch.float64).to(torch.float32)
    Q = fp.transition(tt)[0]
    return dict(Q=Q.cuda().contiguous(), QT=Q.t().contiguous().cuda(), Rb=fp.base_rate.cuda().contiguous(),
                RbT=fp.base_rate.t().contiguous().cuda(), beta=float(fp.beta(tt)[0]))


def _step(mode, branch, head, x, tb, h, S, N, D, **kw):
    from ctdd_b200 import ops
    stats = torch.zeros(8, dtype=torch.int64, device="cuda")
    out = ops.reverse_step(mode, branch, None, x, tb["Q"], tb["QT"], tb["Rb"], tb["RbT"], tb["beta"], h, 1e-9, N=N, D=D,
                           S=S, stats=stats, head=head, **kw)
    out["stats"] = stats
    return out


def _same(a, b, what):
    for k in ("x", "stats", "rr", "ratio"):
        if a.get(k) is None and b.get(k) is None:
            continue
        assert a[k].dtype == b[k].dtype and torch.equal(a[k], b[k]), (what, k)


def _both(mu, ls, fix, call, what):
    """call(head) with the bf16 (mu, log_scale) and with their widened copies: bit-identical outputs."""
    a, b = call((mu, ls, fix)), call((mu.float(), ls.float(), fix))
    _same(a, b, what)
    return a


def _chunked(N, D, seed, lo=-3.0, hi=3.0):
    """The two torch.chunk halves of a bf16 (N, 2D) network output (batch stride 2D) and of its widening."""
    mu, ls = _inputs(N, D, seed, lo, hi)
    both = torch.cat([mu, ls], dim=1)
    return torch.chunk(both, 2, dim=1), torch.chunk(both.float(), 2, dim=1)


STEP_CASES = [
    # N, D, fix, loss, logit_type, t, h
    (6, 40, False, "CTElbo", None, 0.9, 0.004),
    (6, 40, True, "CatRM", "reverse_prob", 0.3, 0.01),
    (3, 75, True, "NLL", None, 0.05, 0.02),            # 225 rows: ragged last tile
    (5, 61, False, "SDDMElbo", "reverse_prob", 0.6, 0.03),
]


@gpu
@pytest.mark.parametrize("sc", STEP_CASES, ids=[f"{c[3]}-fix{int(c[2])}-D{c[1]}" for c in STEP_CASES])
def test_fused_head_every_mode_bit_equal(sc):
    """Every mode of step_q_kernel and both Euler modes of step_tc_kernel with the head fused: bf16 (mu, log_scale) give
    the states, counters and (rates only) rr / ratio of the widened call; contiguous and chunked views, a non-zero
    row offset."""
    nat = _nat()
    N, D, fix, loss_name, logit_type, t, h = sc
    S = 256
    fp = oracle_forward(FWD)
    tb = _tables(fp, t)
    branch = nat.branch_for(loss_name, logit_type)
    from ctdd_b200 import ops
    tct = ops.prep_tc_tables(tb["Q"][None], tb["QT"][None], tb["Rb"], 1e-9, branch)[0]
    tcs = ops.prep_tc_static(tb["Rb"])
    mu, ls = _inputs(N, D, 17 + N + D)
    g = np.random.Generator(np.random.PCG64(3))
    centre = np.clip(np.round((mu.float().cpu().numpy() + 1.0) * S / 2.0 - 0.5), 0, S - 1).astype(np.int64)
    x = torch.from_numpy(np.clip(centre + g.integers(-4, 5, (N, D)), 0, S - 1)).to(torch.int32).cuda()
    xb = torch.from_numpy(np.clip(x.cpu().numpy() + g.integers(-1, 2, (N, D)), 0, S - 1)).to(torch.int32).cuda()
    (cm, cl), _ = _chunked(N, D, 17 + N + D)
    runs = [(nat.MODE_TAU_LEAP, dict(reject_multi=False, offset=3)), (nat.MODE_TAU_LEAP, dict(reject_multi=True, offset=3)),
            (nat.MODE_TAU_LEAP_CORR, dict(offset=5)), (nat.MODE_MIDPOINT_DRIFT, dict(offset=0)),
            (nat.MODE_MIDPOINT_JUMP, dict(reject_multi=True, offset=7, x_base=xb)),
            (nat.MODE_EULER, dict(offset=9)), (nat.MODE_EULER_CORR, dict(offset=10)),
            (nat.MODE_RATES_ONLY, dict(want_rr=True, want_ratio=True))]
    moved = 0
    for mode, extra in runs:
        for m, l in ((mu, ls), (cm, cl)):
            for row0 in (0, 8 * 37):
                kw = dict(impl=nat.IMPL_TC, tc_tables=tct, tc_static=tcs, seed=4242, row_offset=row0, **extra)
                out = _both(m, l, fix, lambda hd: _step(mode, branch, hd, x, tb, h, S, N, D, **kw), (mode, extra, row0))
                if out["x"] is not None:
                    moved += int((out["x"] != x).sum())
    assert moved > 0


@gpu
def test_fused_head_ragged_rows_and_shards():
    """Row counts that are no multiple of 8 or of the 128-row tile, and two shards against one launch."""
    from ctdd_b200 import ops
    nat = _nat()
    S = 256
    fp = oracle_forward(FWD)
    tb = _tables(fp, 0.5)
    for branch in (nat.BRANCH_TAULDR, nat.BRANCH_SDDM_REVERSE_PROB):
        tct = ops.prep_tc_tables(tb["Q"][None], tb["QT"][None], tb["Rb"], 1e-9, branch)[0]
        tcs = ops.prep_tc_static(tb["Rb"])
        for mode in (nat.MODE_TAU_LEAP, nat.MODE_EULER):
            for (N, D) in ((1, 1), (7, 1), (129, 1), (13, 21), (40, 37)):
                (cm, cl), _ = _chunked(N, D, 23 + N)
                x = torch.randint(0, S, (N, D), generator=torch.Generator(device="cuda").manual_seed(N), device="cuda",
                                  dtype=torch.int32)
                kw = dict(impl=nat.IMPL_TC, tc_tables=tct, tc_static=tcs, seed=31, offset=6)
                row0 = 8 * 37
                full = _both(cm, cl, True, lambda hd: _step(mode, branch, hd, x, tb, 0.08, S, N, D, row_offset=row0, **kw),
                             (N, D))
                if N * D >= 16:
                    lo = _both(cm[:8], cl[:8], True, lambda hd: _step(mode, branch, hd, x[:8], tb, 0.08, S, 8, D,
                                                                      row_offset=row0, **kw), "lo")
                    hi = _both(cm[8:], cl[8:], True, lambda hd: _step(mode, branch, hd, x[8:], tb, 0.08, S, N - 8, D,
                                                                      row_offset=row0 + 8 * D, **kw), "hi")
                    assert torch.equal(full["x"], torch.cat([lo["x"], hi["x"]]))
                    assert torch.equal(full["stats"], lo["stats"] + hi["stats"])


@gpu
def test_non_fused_fallbacks_materialise_fp32_logits_from_bf16():
    """S = 32, IMPL_SIMT at S = 256 and the exact mode: the logits are built from the bf16 head without a widening copy
    and stay fp32 - the results equal the widened call's.  head_dtype is ignored for dense logits."""
    from ctdd_b200 import ops
    nat = _nat()
    for fwd, impl, modes in (("gauss32", nat.IMPL_AUTO, (nat.MODE_TAU_LEAP, nat.MODE_EULER, nat.MODE_EXACT)),
                             ("gauss256", nat.IMPL_SIMT, (nat.MODE_TAU_LEAP, nat.MODE_EULER))):
        fp = oracle_forward(fwd)
        S = fp.S
        N, D = 4, 20
        tb = _tables(fp, 0.4)
        (cm, cl), _ = _chunked(N, D, 9, -1.0, 2.0)
        x = torch.randint(0, S, (N, D), dtype=torch.int32, device="cuda")
        for branch in (nat.BRANCH_TAULDR, nat.BRANCH_SDDM_REVERSE_PROB):
            for mode in modes:
                _both(cm, cl, False, lambda hd: _step(mode, branch, hd, x, tb, 0.02, S, N, D, impl=impl, seed=5, offset=2,
                                                      want_rr=(mode != nat.MODE_EXACT)), (fwd, branch, mode))
    # dense logits with a nonsense head_dtype: ignored, as logits_dtype is ignored for a head
    fp = oracle_forward("gauss32")
    tb = _tables(fp, 0.4)
    N, D, S = 4, 20, 32
    logits = ops.logistic_logits(*_inputs(N, D, 4), S, False)
    x = torch.randint(0, S, (N, D), dtype=torch.int32, device="cuda")
    out = torch.empty_like(x)
    p = nat.StepParams(mode=nat.MODE_TAU_LEAP, branch=nat.BRANCH_TAULDR, impl=nat.IMPL_SIMT, N=N, D=D, S=S, logits=logits.data_ptr(),
                       ld_logits=S, batch_stride_logits=D * S, x_eval=x.data_ptr(), Q=tb["Q"].data_ptr(), QT=tb["QT"].data_ptr(),
                       Rb=tb["Rb"].data_ptr(), RbT=tb["RbT"].data_ptr(), beta=tb["beta"], h=0.02, eps=1e-9, seed=5,
                       x_out=out.data_ptr(), head_dtype=7)
    nat.check(nat.lib().ctdd_reverse_step(p, nat.stream()), "dense logits, head_dtype ignored")
    want = ops.reverse_step(nat.MODE_TAU_LEAP, nat.BRANCH_TAULDR, logits, x, tb["Q"], tb["QT"], tb["Rb"], tb["RbT"], tb["beta"],
                            0.02, 1e-9, N=N, D=D, S=S, impl=nat.IMPL_SIMT, seed=5)["x"]
    assert torch.equal(out, want)


@gpu
def test_step_engine_reads_bf16_head_without_widening_copy():
    """StepEngine.step with a bf16 LogisticHead takes the fast path and allocates nothing: no cast kernel, no fp32 copy
    (an fp16 head, which is widened, does allocate); its samples equal those of the widened head."""
    from ctdd_b200 import make_config, ops
    from ctdd_b200.lib.sampling.sampling import StepEngine
    nat = _nat()
    N, D, S = 256, 1024, 256
    cfg = fwd_cfg("gauss256", make_config)
    m = product_model("gauss256", cfg, D, 3, 0.3, 12.0)
    m.device = torch.device("cuda", torch.cuda.current_device())     # the fast path compares devices with their index
    eng = StepEngine(cfg, m, N, D, S, [0.5], nat.BRANCH_TAULDR, 1e-9, seed=1)
    (cm, cl), (fm_, fl) = _chunked(N, D, 8)
    x = torch.randint(0, S, (N, D), generator=torch.Generator(device="cuda").manual_seed(1), device="cuda", dtype=torch.int32)

    def allocations(head):
        torch.cuda.synchronize()
        n0 = torch.cuda.memory_stats()["allocation.all.allocated"]
        x_new, _ = eng.step(nat.MODE_TAU_LEAP, head, x, 0, 0.01, draws=False)
        torch.cuda.synchronize()
        return torch.cuda.memory_stats()["allocation.all.allocated"] - n0, x_new.clone()

    allocations(ops.LogisticHead(cm, cl))                                       # warm-up
    n_bf16, a = allocations(ops.LogisticHead(cm, cl))
    n_f32, b = allocations(ops.LogisticHead(fm_, fl))
    n_f16, _ = allocations(ops.LogisticHead(cm.half(), cl.half()))
    assert n_bf16 == 0 and n_f32 == 0 and n_f16 > 0, (n_bf16, n_f32, n_f16)
    assert torch.equal(a, b)
    assert eng._p.head_dtype == nat.DTYPE_F32                                   # rewritten on every call


# ------------------------------------------------------------------------------------------------------- samplers
def _head_model(cfg, S, D, seed, fix, dtype):
    """HeadStubNet x rate mixin x TruncatedLogisticHead whose (mu, log_scale) are rounded to bf16 and handed over as
    `dtype`."""
    from ctdd_b200.lib.models import forward_model as fm, models
    mixin = getattr(fm, cases.FORWARD[FWD]["mixin"])

    class M(rh.HeadStubNet, mixin, models.TruncatedLogisticHead):
        def __init__(self):
            rh.HeadStubNet.__init__(self, S, D, seed)
            mixin.__init__(self, cfg, "cuda")
            self.fix_logistic = fix

        def forward(self, x, t):
            B, Dx = x.shape
            mu, ls = self.head_params(x, t)
            return self.head_forward((mu.to(bf16).to(dtype), ls.to(bf16).to(dtype)), B, Dx)

    m = M().to("cuda")
    m.device = "cuda"
    return m


MIDPOINT_CASE = ("head_midpoint", "MidPointTauL", FWD, 8, 12, "CatRM", "reverse_prob", True, dict(num_steps=6, min_t=0.01),
                 1.0, 305)


def _sample(case, dtype):
    from ctdd_b200 import make_config
    from ctdd_b200.lib.sampling import sampling_utils
    import ctdd_b200.lib.sampling.sampling  # noqa: F401
    name, cls, fwd, N, D, loss_name, logit_type, fix, over, max_t, seed = case
    cfg = cases.sampler_cfg(make_config, case)
    cfg.device = "cuda"
    m = _head_model(cfg, cfg.data.S, D, seed, fix, dtype)
    cfg.sampler.name = cls
    sampler = sampling_utils.get_sampler(cfg)
    sampler.seed = seed
    args = ()
    if "condition_dim" in over:
        g = np.random.Generator(np.random.PCG64(seed))
        args = (torch.from_numpy(g.integers(0, cfg.data.S, (N, over["condition_dim"]))),)
    res = sampler.sample(m, N, *args)
    return res if isinstance(res, tuple) else (res,)


@gpu
@pytest.mark.parametrize("case", HEAD_SAMPLERS + [MIDPOINT_CASE], ids=[c[0] for c in HEAD_SAMPLERS + [MIDPOINT_CASE]])
def test_samplers_take_bf16_head(case):
    """TauL, LBJF, MidPointTauL and ConditionalTauLeaping on a head model whose (mu, log_scale) are bf16: the same samples
    and diagnostics as with their fp32 widening."""
    a, b = _sample(case, bf16), _sample(case, torch.float32)
    assert len(a) == len(b)
    for u, v in zip(a, b):
        np.testing.assert_array_equal(np.asarray(u), np.asarray(v), err_msg=case[0])


# ------------------------------------------------------------------------------------------------------- training
TRAIN_CASES = [
    # loss class, overrides, CUDA-core (CTElbo) or tensor-core loss path
    ("CTElbo", dict()),
    ("SDDMElbo", dict(logit_type="reverse_prob", nll_weight=0.01)),
    ("CatRMNLL", dict(logit_type="reverse_prob", loss_type="rm", nll_weight=0.01)),
]


def _train_step(cls, over, reference, monkeypatch):
    """One Standard.step under torch.autocast(bf16) on a small image network ending in a 1x1 nn.Conv2d that emits
    (mu, log_scale) as the two torch.chunk halves of (B, 2C, H, W).  `reference`: the head on mu.float(),
    log_scale.float(), its logits cast to bf16.  Returns (loss, parameter gradients, logits dtypes seen by the loss)."""
    from ctdd_b200 import make_config, ops
    from ctdd_b200.lib.models import forward_model as fm, models
    from ctdd_b200.lib.losses import losses_utils
    import ctdd_b200.lib.losses.losses  # noqa: F401
    import ctdd_b200.lib.training.training as tr
    B, C, H, W, S = 4, 3, 8, 8, 256
    D = C * H * W
    case = ("train", cls, "gauss256", B, D, over, 1.0, 7, 0)
    cfg = cases.loss_cfg(make_config, case, device="cuda")
    step_cfg = make_config(model=dict(name="head"), training=dict(clip_grad=False, grad_norm=1.0, warmup=0),
                           optimizer=dict(lr=0.0), device="cuda")

    class M(torch.nn.Module, fm.GaussianTargetRate, models.TruncatedLogisticHead):
        def __init__(self):
            torch.nn.Module.__init__(self)
            fm.GaussianTargetRate.__init__(self, cfg, "cuda")
            self.S, self.fix_logistic = S, True
            self.emb = torch.nn.Embedding(S, 8)
            self.out = torch.nn.Conv2d(8 * C, 2 * C, 1)

        def forward(self, x, t, *args):
            Bx = x.shape[0]
            e = self.emb(x.view(Bx, C, H, W)).permute(0, 1, 4, 2, 3).reshape(Bx, 8 * C, H, W) + t.view(-1, 1, 1, 1)
            mu, ls = torch.chunk(self.out(e), 2, dim=1)         # bf16 under autocast
            mu = torch.tanh(mu)
            if reference:
                return ops.logistic_logits_autograd(mu.float(), ls.float(), S, True).view(Bx, D, S).to(bf16)
            return self.head_forward((mu, ls), Bx, D)

    torch.manual_seed(0)
    m = M().to("cuda")
    m.device = "cuda"
    seen = []
    real = ops.loss_terms

    def spy(logits, *a, **k):
        seen.append(logits.dtype)
        return real(logits, *a, **k)
    monkeypatch.setattr(ops, "loss_terms", spy)
    loss_obj = losses_utils.get_loss(cfg)
    loss_obj.seed = 3
    loss_obj.ts_override = torch.linspace(0.1, 0.9, B)
    x0 = torch.randint(0, S, (B, D), generator=torch.Generator().manual_seed(1)).cuda()
    state = {"model": m, "optimizer": torch.optim.SGD(m.parameters(), lr=0.0), "n_iter": 1}
    with torch.autocast("cuda", dtype=bf16):
        loss = tr.Standard(step_cfg).step(state, loss_obj, x0)
    monkeypatch.undo()
    return loss, [p.grad.detach().clone() for p in m.parameters()], seen


@gpu
@pytest.mark.parametrize("cls,over", TRAIN_CASES, ids=[c[0] for c in TRAIN_CASES])
def test_training_step_under_autocast(cls, over, monkeypatch):
    """The head under real autocast gets bf16 (mu, log_scale), raises nothing and hands bf16 logits to the loss; the
    loss and the parameter gradients agree with the cast-to-fp32 reference."""
    loss, grads, seen = _train_step(cls, over, False, monkeypatch)
    rloss, rgrads, rseen = _train_step(cls, over, True, monkeypatch)
    assert seen and all(d == bf16 for d in seen) and seen == rseen
    assert torch.isfinite(loss) and abs(float(loss) - float(rloss)) <= 1e-5 * abs(float(rloss)), (float(loss), float(rloss))
    for g, r in zip(grads, rgrads):
        assert torch.isfinite(g).all()
        assert float((g.float() - r.float()).abs().max()) <= 1e-3 * float(r.float().abs().max()), cls
    assert max(float(g.abs().max()) for g in grads) > 0


def _loss_problem(B, D, seed):
    """Per-sample q_{t|0} and noised states of an SDDM loss call at S = 256."""
    from ctdd_b200 import ops
    fp = oracle_forward("gauss256")
    g = np.random.Generator(np.random.PCG64(seed))
    ts = torch.from_numpy(g.uniform(0.05, 0.95, B).astype(np.float32))
    Q = fp.transition(ts).float()
    c = dict(Q=Q.cuda().contiguous(), QT=Q.transpose(1, 2).contiguous().cuda(), Rb=fp.base_rate.cuda().contiguous(),
             beta=fp.beta(ts).float().cuda().contiguous(), x0=torch.from_numpy(g.integers(0, 256, (B, D))).to(torch.int32).cuda())
    c["xt"], c["xtil"] = ops.noise_xt(c["Q"], c["Rb"], c["beta"], c["x0"], seed, 0)
    return c


def _sddm(logits, c):
    from ctdd_b200 import ops
    nat = _nat()
    outs = ops.loss_terms(logits, nat.LOSS_SDDM, c["Q"], c["QT"], c["Rb"], c["beta"], c["x0"], c["xtil"], eps=1e-9,
                          logit_branch=nat.BRANCH_SDDM_REVERSE_PROB)
    return outs[0].sum() + 0.5 * outs[1].sum() + 0.01 * outs[4].sum()


@gpu
def test_head_loss_chain_is_bit_equal():
    """Ops level, deterministic: the bf16 gradient ctdd_loss_backward gives the head's bf16 logits, fed to the head
    backward, yields grad_mu / grad_log_scale equal to the fp32 kernel's on that gradient widened."""
    from ctdd_b200 import ops
    B, D, S = 4, 96, 256
    c = _loss_problem(B, D, 5)
    mu, ls = _inputs(B, D, 6, -1.0, 2.0)
    for leaf_dtype in (bf16, torch.float32):
        mc = mu.to(leaf_dtype, copy=True).requires_grad_(True)
        lc = ls.to(leaf_dtype, copy=True).requires_grad_(True)
        logits = ops.logistic_logits_autograd(mc, lc, S, False, out_dtype=bf16)
        logits.retain_grad()
        _sddm(logits, c).backward()
        assert logits.grad.dtype == bf16
        want = _fp32_backward(mu, ls, logits.grad, S, False)
        assert mc.grad.dtype == leaf_dtype
        assert torch.equal(mc.grad, want[0].to(leaf_dtype)) and torch.equal(lc.grad, want[1].to(leaf_dtype)), leaf_dtype


@gpu
def test_peak_memory_of_head_and_loss():
    """B = 64, D = 3072, S = 256: head + SDDMElbo forward + backward from bf16 (mu, log_scale) peaks at least
    1.5 B D S bytes below the cast-to-fp32 route (fp32 head, fp32 logits and gradient); the logits and the gradient each
    halve, 2 B D S bytes in all."""
    from ctdd_b200 import ops
    B, D, S = 64, 3072, 256
    c = _loss_problem(B, D, 9)
    mu, ls = _inputs(B, D, 10, -1.0, 2.0)
    mu.requires_grad_(True)
    ls.requires_grad_(True)

    def peak(widen):
        mu.grad = ls.grad = None
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        if widen:
            logits = ops.logistic_logits_autograd(mu.float(), ls.float(), S, False)
        else:
            logits = ops.logistic_logits_autograd(mu, ls, S, False, out_dtype=bf16)
        _sddm(logits, c).backward()
        del logits
        torch.cuda.synchronize()
        assert mu.grad.dtype == bf16
        return torch.cuda.max_memory_allocated() - base

    peak(False)                                                 # warm-up: the allocator's first blocks
    new, old = peak(False), peak(True)
    assert old - new >= 1.5 * B * D * S, (old, new)


# ------------------------------------------------------------------------------------------------------- CPU
def test_unknown_head_dtype_is_refused_before_any_cuda_call():
    """The ABI checks need no device: an unknown head_dtype with a logistic head, or an unknown dtype given to either
    _ex entry point, returns status 2 with a message."""
    nat = _nat()
    L = nat.lib()
    dummy = 0x1000
    p = nat.StepParams(mode=nat.MODE_TAU_LEAP, branch=nat.BRANCH_TAULDR, impl=nat.IMPL_TC, N=2, D=3, S=256, x_eval=dummy,
                       Q=dummy, QT=dummy, Rb=dummy, RbT=dummy, x_out=dummy, head=nat.HEAD_LOGISTIC, head_mu=dummy,
                       head_log_scale=dummy, head_batch_stride=3, head_dtype=7)
    assert L.ctdd_reverse_step(ctypes.byref(p), None) == 2
    assert b"head_dtype" in L.ctdd_last_error()
    assert nat.StepParams.head_dtype.offset > nat.StepParams.logits_dtype.offset
    for bad in ((7, 0), (0, 7), (-1, 1)):
        assert L.ctdd_logistic_logits_ex(dummy, dummy, bad[0], 2, 3, 3, 256, 0, dummy, bad[1], None) == 2
        assert b"dtype" in L.ctdd_last_error()
        assert L.ctdd_logistic_logits_backward_ex(dummy, dummy, bad[0], dummy, bad[1], 2, 3, 3, 256, 0, dummy, dummy, None) == 2
        assert b"dtype" in L.ctdd_last_error()
