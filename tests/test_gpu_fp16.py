"""fp16 logits (what torch.autocast("cuda") emits with no dtype) on every reverse-step, loss and head path.  The bar is bit
equality with the same call on the widened fp32 tensors; a 2-byte output (the loss gradient, the head's logits) is that
call's fp32 output rounded once to fp16, ±inf where it overflows.  The shapes and cases are those of the bf16 files;
the dtype-independent helpers come from there, and every input is generated in fp16 here."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import cases, head_oracle as ho, ref_harness as rh
from helpers import oracle_forward, product_model, fwd_cfg
import test_gpu_bf16_logits as bl
import test_gpu_bf16_losses as bo
import test_gpu_bf16_head as bh

gpu = pytest.mark.gpu
f16 = torch.float16


def _nat():
    from ctdd_b200 import _native as nat
    return nat


def _with_subnormals(a, g):
    """fp32 array with 2 % of its entries replaced by values that are subnormal in fp16 (|v| < 2^-14)."""
    pick = g.random(a.shape) < 0.02
    return np.where(pick, g.uniform(-6e-5, 6e-5, a.shape), a).astype(np.float32)


# ------------------------------------------------------------------------------------------------------- step
def _problem(fwd, N, D, t, seed, width, scale=0.5):
    """The inputs of the bf16 file's step cases, with the logits rounded to fp16."""
    fp = oracle_forward(fwd)
    S = fp.S
    g = np.random.Generator(np.random.PCG64(seed))
    x0 = g.integers(0, S, (N, D))
    logits = scale * 4.0 * g.standard_normal((N, D, S))
    if width is not None:
        logits = logits - (np.arange(S)[None, None, :] - x0[:, :, None]) ** 2 / (2.0 * width ** 2)
    x = np.clip(x0 + g.integers(-2, 3, (N, D)), 0, S - 1)
    lh = torch.from_numpy(_with_subnormals(logits, g)).to(f16).cuda()
    return fp, lh, torch.from_numpy(x).to(torch.int32).cuda(), S


@gpu
@pytest.mark.parametrize("impl_name", ["simt", "auto"])
@pytest.mark.parametrize("sc", bl.STEP_CASES, ids=[f"{c[0]}-{c[5]}-{c[6]}-D{c[2]}" for c in bl.STEP_CASES])
def test_step_every_mode_and_path_bit_equal(sc, impl_name):
    """Every mode on the CUDA-core kernels and on what IMPL_AUTO picks; at S = 256 with tcgen05 tables IMPL_TC is forced,
    so every fp16 step_q_kernel and step_tc_kernel runs."""
    nat = _nat()
    fwd, N, D, t, h, loss_name, logit_type, width = sc
    fp, lh, x, S = _problem(fwd, N, D, t, 11, width)
    tb = bl._tables(fp, t)
    branch = nat.branch_for(loss_name, logit_type)
    impl, tct, tcs = nat.IMPL_SIMT, None, None
    if impl_name == "auto":
        tct, tcs = bl._tc(tb, branch, S)
        impl = nat.IMPL_TC if tct is not None else nat.IMPL_AUTO
    g = np.random.Generator(np.random.PCG64(5))
    xb = torch.from_numpy(np.clip(x.cpu().numpy() + g.integers(-1, 2, x.shape), 0, S - 1)).to(torch.int32).cuda()
    kw = dict(impl=impl, tc_tables=tct, tc_static=tcs, seed=4242)
    runs = [(nat.MODE_TAU_LEAP, dict(reject_multi=False, offset=3)), (nat.MODE_TAU_LEAP, dict(reject_multi=True, offset=3)),
            (nat.MODE_TAU_LEAP_CORR, dict(offset=5)), (nat.MODE_MIDPOINT_DRIFT, dict(offset=0)),
            (nat.MODE_MIDPOINT_JUMP, dict(reject_multi=True, offset=7, x_base=xb)),
            (nat.MODE_EULER, dict(offset=9)), (nat.MODE_EULER_CORR, dict(offset=10)),
            (nat.MODE_RATES_ONLY, dict(want_rr=True, want_ratio=True))]
    if impl != nat.IMPL_TC:
        runs += [(nat.MODE_TAU_LEAP, dict(offset=4, want_rr=True, want_ratio=True)), (nat.MODE_EXACT, dict(offset=11))]
    moved = 0
    for mode, extra in runs:
        out = bl._both(lh, lambda L: bl._step(mode, branch, L, x, tb, h, S, N, D, **kw, **extra), (mode, extra.get("reject_multi")))
        if out["x"] is not None:
            moved += int((out["x"] != x).sum())
    assert moved > 0


@gpu
@pytest.mark.parametrize("fwd,loss_name,mode_name", [("univar2_sqrtcos", "CTElbo", "tau_leap"), ("univar3_logsqr", "CTElbo", "euler"),
                                                     ("univar5_log", "CTElbo", "tau_leap"), ("gauss256", "CTElbo", "tau_leap"),
                                                     ("gauss256", "CatRM", "euler")])
def test_step_ragged_rows_row_offset_and_shards(fwd, loss_name, mode_name):
    """Row counts that are no multiple of 8 or of the 128-row pair tile, a non-zero row offset, and two shards against
    one launch."""
    nat = _nat()
    mode = nat.MODE_EULER if mode_name == "euler" else nat.MODE_TAU_LEAP
    for (N, D) in ((1, 1), (7, 1), (129, 1), (13, 21), (40, 37)):
        fp, lh, x, S = _problem(fwd, N, D, 0.5, 23 + N, 12.0 if fwd == "gauss256" else None)
        tb = bl._tables(fp, 0.5)
        branch = nat.branch_for(loss_name, "reverse_prob")
        tct, tcs = bl._tc(tb, branch, S)
        kw = dict(impl=(nat.IMPL_TC if tct is not None else nat.IMPL_AUTO), tc_tables=tct, tc_static=tcs, seed=31, offset=6)
        row0 = 8 * 37
        full = bl._both(lh, lambda L: bl._step(mode, branch, L, x, tb, 0.08, S, N, D, row_offset=row0, **kw), (N, D))
        if N * D >= 16:
            n_lo = 8
            lo = bl._both(lh[:n_lo], lambda L: bl._step(mode, branch, L, x[:n_lo], tb, 0.08, S, n_lo, D, row_offset=row0, **kw),
                          "lo")
            hi = bl._both(lh[n_lo:], lambda L: bl._step(mode, branch, L, x[n_lo:], tb, 0.08, S, N - n_lo, D,
                                                         row_offset=row0 + n_lo * D, **kw), "hi")
            assert torch.equal(full["x"], torch.cat([lo["x"], hi["x"]]))
            assert torch.equal(full["stats"], lo["stats"] + hi["stats"])


@gpu
def test_step_small_s_grid_stride_kernel_at_scale():
    """The S = 2 tau-leap kernel strides over its capped grid (C1 at 8x its batch: 16.8 M rows)."""
    nat = _nat()
    fp = oracle_forward("univar2_sqrtcos")
    tb = bl._tables(fp, 0.6)
    N, D, S = 1 << 19, 32, 2
    gen = torch.Generator(device="cuda").manual_seed(3)
    lh = (torch.randn((N, D, S), generator=gen, device="cuda") * 2.0).to(f16)
    x = torch.randint(0, S, (N, D), generator=gen, device="cuda", dtype=torch.int32)
    out = bl._both(lh, lambda L: bl._step(nat.MODE_TAU_LEAP, nat.BRANCH_TAULDR, L, x, tb, 0.05, S, N, D, reject_multi=True,
                                          seed=2, offset=1), "C1x8")
    assert int(out["stats"][nat.STAT_CHANGED_BASE]) > 0


@gpu
@pytest.mark.parametrize("fwd,loss_name,logit_type", [("gauss256", "CTElbo", None), ("gauss256", "CatRM", "reverse_prob"),
                                                      ("gauss32", "CTElbo", None)])
def test_step_strided_views(fwd, loss_name, logit_type):
    """logits[:, c:, :] of an fp16 (N, D_total, S) tensor on the tcgen05 path (S = 256) and the CUDA-core path: equal to
    the widened view and to a contiguous fp16 copy."""
    nat = _nat()
    for (N, Dfull, c) in ((3, 29, 8), (6, 200, 72), (40, 340, 40)):
        D = Dfull - c
        fp, lh_full, x_full, S = _problem(fwd, N, Dfull, 0.35, 41 + N, 12.0 if fwd == "gauss256" else 3.0)
        tb = bl._tables(fp, 0.35)
        branch = nat.branch_for(loss_name, logit_type)
        tct, tcs = bl._tc(tb, branch, S)
        x = x_full[:, c:].contiguous()
        impl = nat.IMPL_TC if tct is not None else nat.IMPL_SIMT
        for mode in (nat.MODE_TAU_LEAP, nat.MODE_TAU_LEAP_CORR, nat.MODE_MIDPOINT_DRIFT, nat.MODE_EULER):
            kw = dict(impl=impl, tc_tables=tct, tc_static=tcs, seed=11, offset=3)
            view = bl._both(lh_full, lambda L: bl._step(mode, branch, L, x, tb, 0.01, S, N, D, logits_offset_elems=c * S,
                                                        batch_stride=Dfull * S, **kw), (N, Dfull, c, mode))
            copy = bl._step(mode, branch, lh_full[:, c:, :].contiguous(), x, tb, 0.01, S, N, D, **kw)
            bl._assert_same(view, copy, ("copy", N, Dfull, c, mode))


@gpu
def test_step_misaligned_fp16_rows_leave_the_tensor_path():
    """An fp16 view whose batch stride is a multiple of 4 but not of 8 elements (16-byte aligned for fp32, not for fp16):
    IMPL_TC refuses it, IMPL_AUTO runs it on the CUDA-core path and matches the widened view there."""
    from ctdd_b200 import ops
    nat = _nat()
    N, D = 5, 24
    fp, lh, x, S = _problem("gauss256", N, D, 0.35, 7, 12.0)
    tb = bl._tables(fp, 0.35)
    tct, tcs = bl._tc(tb, nat.BRANCH_TAULDR, S)
    stride = D * S + 4
    buf = torch.zeros((N, stride), dtype=f16, device="cuda")
    buf[:, :D * S] = lh.reshape(N, D * S)
    kw = dict(tc_tables=tct, tc_static=tcs, seed=3, offset=2, batch_stride=stride)
    with pytest.raises(RuntimeError, match="rc=3"):
        bl._step(nat.MODE_TAU_LEAP, nat.BRANCH_TAULDR, buf, x, tb, 0.01, S, N, D, impl=nat.IMPL_TC, **kw)
    for mode in (nat.MODE_TAU_LEAP, nat.MODE_EULER):
        a = bl._step(mode, nat.BRANCH_TAULDR, buf, x, tb, 0.01, S, N, D, impl=nat.IMPL_AUTO, **kw)
        b = bl._step(mode, nat.BRANCH_TAULDR, buf.float(), x, tb, 0.01, S, N, D, impl=nat.IMPL_SIMT, **kw)
        bl._assert_same(a, b, mode)
    assert ops.reverse_step(nat.MODE_TAU_LEAP, nat.BRANCH_TAULDR, buf.float(), x, tb["Q"], tb["QT"], tb["Rb"], tb["RbT"],
                            tb["beta"], 0.01, 1e-9, N=N, D=D, S=S, impl=nat.IMPL_TC, **kw)["x"] is not None


@gpu
def test_step_full_c4_size_tau_leap():
    """One tau-leap step at the C4 shape (B = 1024, D = 3072, S = 256): the 1.6 GB fp16 tensor against its 3.2 GB
    widened copy."""
    nat = _nat()
    B, D, S = 1024, 3072, 256
    fp = oracle_forward("gauss256")
    tb = bl._tables(fp, 0.5)
    tct, tcs = bl._tc(tb, nat.BRANCH_TAULDR, S)
    gen = torch.Generator(device="cuda").manual_seed(9)
    x = torch.randint(0, S, (B, D), generator=gen, device="cuda", dtype=torch.int32)
    lh = torch.randn((B, D, S), generator=gen, device="cuda", dtype=f16)
    lh -= ((torch.arange(S, device="cuda", dtype=torch.float32).view(1, 1, S) - x.unsqueeze(-1)) ** 2 / 128.0).to(f16)
    kw = dict(impl=nat.IMPL_TC, tc_tables=tct, tc_static=tcs, seed=5, offset=1)
    a = bl._step(nat.MODE_TAU_LEAP, nat.BRANCH_TAULDR, lh, x, tb, 0.01, S, B, D, **kw)
    lf = lh.float()
    del lh
    b = bl._step(nat.MODE_TAU_LEAP, nat.BRANCH_TAULDR, lf, x, tb, 0.01, S, B, D, **kw)
    bl._assert_same(a, b, "C4")
    assert int(a["stats"][nat.STAT_CHANGED_BASE]) > 0


def _sample(case, to_fp32):
    """A sampler run on the stub network whose logits end in .half() (to_fp32: then .float())."""
    from ctdd_b200 import make_config
    from ctdd_b200.lib.sampling import sampling_utils
    import ctdd_b200.lib.sampling.sampling  # noqa: F401
    name, cls, fwd, N, D, loss_name, logit_type, stub, over, max_t, seed = case
    cfg = cases.sampler_cfg(make_config, case)
    cfg.device = "cuda"
    S = cfg.data.S
    m = product_model(fwd, cfg, D, seed, stub[0], stub[1])
    net = m.forward
    m.forward = (lambda x, t: net(x, t).half().float()) if to_fp32 else (lambda x, t: net(x, t).half())
    cfg.sampler.name = cls
    sampler = sampling_utils.get_sampler(cfg)
    sampler.seed = seed
    args = ()
    if "condition_dim" in over:
        g = np.random.Generator(np.random.PCG64(seed))
        args = (torch.from_numpy(g.integers(0, S, (N, over["condition_dim"]))),)
    res = sampler.sample(m, N, *args)
    return res if isinstance(res, tuple) else (res,)


@gpu
@pytest.mark.parametrize("name", bl.SAMPLER_CASES)
def test_samplers_take_fp16_network_output(name):
    """The same seeded sampler with the network's fp16 logits and with their fp32 widening: identical samples and
    diagnostics."""
    case = bl._by_name(name)
    a, b = _sample(case, False), _sample(case, True)
    assert len(a) == len(b)
    for u, v in zip(a, b):
        np.testing.assert_array_equal(np.asarray(u), np.asarray(v), err_msg=name)


@gpu
def test_step_engine_reads_fp16_without_widening_copy():
    """StepEngine.step with fp16 logits allocates less than 1/16 of an fp32 (N, D, S) tensor (no hidden .float())."""
    from ctdd_b200 import make_config
    from ctdd_b200.lib.sampling.sampling import StepEngine
    nat = _nat()
    N, D, S = 256, 1024, 256
    cfg = fwd_cfg("gauss256", make_config)
    m = product_model("gauss256", cfg, D, 3, 0.3, 12.0)
    for impl in (nat.IMPL_AUTO, nat.IMPL_SIMT):
        eng = StepEngine(cfg, m, N, D, S, [0.5], nat.BRANCH_TAULDR, 1e-9, impl=impl, seed=1)
        gen = torch.Generator(device="cuda").manual_seed(1)
        lh = torch.randn((N, D, S), generator=gen, device="cuda", dtype=f16)
        x = torch.randint(0, S, (N, D), generator=gen, device="cuda", dtype=torch.int32)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        x_new, _ = eng.step(nat.MODE_TAU_LEAP, lh, x, 0, 0.01)
        torch.cuda.synchronize()
        assert torch.cuda.max_memory_allocated() - base < N * D * S * 4 // 16, impl
        # and the fast path gives what the widened logits give
        x_ref, _ = StepEngine(cfg, m, N, D, S, [0.5], nat.BRANCH_TAULDR, 1e-9, impl=impl, seed=1).step(
            nat.MODE_TAU_LEAP, lh.float(), x, 0, 0.01)
        assert torch.equal(x_new, x_ref), impl


# ------------------------------------------------------------------------------------------------------- losses
def _loss_problem(fwd, B, D, seed, width):
    """The bf16 loss file's problems with the logits rounded to fp16."""
    from ctdd_b200 import ops
    fp = oracle_forward(fwd)
    S = fp.S
    g = np.random.Generator(np.random.PCG64(seed))
    ts = torch.from_numpy(g.uniform(0.05, 0.95, B).astype(np.float32))
    Q = fp.transition(ts).float()
    x0 = g.integers(0, S, (B, D))
    logits = 2.0 * g.standard_normal((B, D, S))
    if width is not None:
        logits = logits - (np.arange(S)[None, None, :] - x0[:, :, None]) ** 2 / (2.0 * width ** 2)
    c = dict(Q=Q.cuda().contiguous(), QT=Q.transpose(1, 2).contiguous().cuda(), Rb=fp.base_rate.cuda().contiguous(),
             beta=fp.beta(ts).float().cuda().contiguous(), x0=torch.from_numpy(x0).to(torch.int32).cuda())
    c["xt"], c["xtil"] = ops.noise_xt(c["Q"], c["Rb"], c["beta"], c["x0"], seed, 0)
    return c, torch.from_numpy(_with_subnormals(logits, g)).to(f16).cuda(), S


def _loss_compare(lh, kind, branch, crm, c, R, what):
    oh, gh = bo._fwd_bwd(lh, kind, branch, crm, c)
    of, gf = bo._fwd_bwd(lh.float(), kind, branch, crm, c)
    assert torch.isfinite(gf).all() and all(torch.isfinite(o).all() for o in of), what
    assert gh.dtype == f16 and gf.dtype == torch.float32, what
    assert torch.equal(gh, gf.half()), what
    bound = bo._atomic_bound(lh, kind, branch, crm, c, R)
    for k, (a, b) in enumerate(zip(oh, of)):
        if bound is None:
            assert torch.equal(a, b), (what, k)
        else:
            assert ((a.double() - b.double()).abs() <= bound[k]).all(), (what, k, (a - b).abs().max().item())
    assert gf.abs().max() > 0, what


@gpu
@pytest.mark.parametrize("shape", bo.SHAPES, ids=[f"{s[0]}-B{s[1]}-D{s[2]}" for s in bo.SHAPES])
@pytest.mark.parametrize("kind_case", bo.KINDS, ids=[k[0] for k in bo.KINDS])
def test_loss_every_path_and_kind(shape, kind_case):
    """CUDA-core kernel at S = 3, 32 and 256, and the tensor-core path at S = 256 (SDDM and CRM with reverse_prob /
    reverse_logscale)."""
    from ctdd_b200 import ops
    fwd, B, D, width = shape
    _, kind, branch, crm = kind_case
    c, lh, S = _loss_problem(fwd, B, D, 17 + D, width)
    R = 32 if S == 256 else 8
    for tc in ((True, False) if S == 256 and kind != 0 and branch != "direct" else (True,)):
        ops._LossTerms.use_tc = tc
        try:
            _loss_compare(lh, kind, branch, crm, c, R, (kind_case[0], shape, tc))
        finally:
            ops._LossTerms.use_tc = True


@gpu
@pytest.mark.parametrize("kind_case", [bo.KINDS[0], bo.KINDS[1]], ids=["ctelbo", "sddm_tc"])
def test_loss_c5_size_gradient_bit_equal(kind_case):
    """B = 16, D = 3072, S = 256: SDDM on the tensor-core path and CT-ELBO."""
    _, kind, branch, crm = kind_case
    c, lh, _ = _loss_problem("gauss256", 16, 3072, 5, 12.0)
    _, gh = bo._fwd_bwd(lh, kind, branch, crm, c)
    _, gf = bo._fwd_bwd(lh.float(), kind, branch, crm, c)
    assert gh.dtype == f16 and torch.equal(gh, gf.half())


def _class_loss(case, to_fp32):
    """calc_loss + backward() with the stub network ending in .half() (to_fp32: then .float())."""
    from ctdd_b200 import make_config
    from ctdd_b200.lib.models import forward_model as fm
    from ctdd_b200.lib.losses import losses_utils
    from oracle.make_golden_losses import minibatch_for
    import ctdd_b200.lib.losses.losses  # noqa: F401
    name, cls, fwd, B, D, over, t_hi, seed, n_iter = case
    cfg = cases.loss_cfg(make_config, case, device="cuda")
    S, cd = cfg.data.S, over.get("condition_dim", 0)
    mixin = getattr(fm, cases.FORWARD[fwd]["mixin"])
    seen = []

    class M(rh.StubNet, mixin):
        def __init__(self):
            rh.StubNet.__init__(self, S, D + cd, seed, 1.0, 3.0 if S > 8 else None)
            mixin.__init__(self, cfg, "cuda")

        def forward(self, x, t, label=None):
            out = self.net(x, t).half()
            out.retain_grad()
            seen.append(out)
            return out.float() if to_fp32 else out

    m = M().to("cuda")
    m.device = "cuda"
    loss_obj = losses_utils.get_loss(cfg)
    x0, u, _ = minibatch_for(case)
    loss_obj.ts_override = (u * (t_hi - 0.01) + 0.01).cuda()
    loss_obj.seed = seed
    state = {"model": m, "optimizer": None, "n_iter": n_iter}
    loss = loss_obj.calc_loss(x0.cuda(), state) if cls in cases.LOSS_MINIBATCH_FIRST else loss_obj.calc_loss(state, x0.cuda())
    loss.backward()
    return loss.detach(), m.w.grad.detach().clone(), seen


@gpu
@pytest.mark.parametrize("name", bo.LOSS_CLASS_CASES)
def test_loss_classes_take_fp16_network_output(name):
    """Every loss class on a network whose output is fp16, against the same network widening it: the loss, d loss / d w
    and the fp16 logits gradient the network sees are bit-equal (at most two CTAs per sample: no atomic reordering)."""
    case = next(c for c in cases.LOSSES if c[0] == name)
    lh, wh, seen_h = _class_loss(case, False)
    lf, wf, seen_f = _class_loss(case, True)
    assert torch.isfinite(lh) and torch.equal(lh, lf), (lh.item(), lf.item())
    assert torch.equal(wh, wf) and wh.abs().max() > 0
    assert len(seen_h) == len(seen_f)
    for a, b in zip(seen_h, seen_f):
        assert a.grad is not None and a.grad.dtype == f16 and torch.equal(a.grad, b.grad)


@gpu
def test_loss_under_default_autocast_with_linear_output_layer(monkeypatch):
    """SDDMElbo on a network with an nn.Linear output layer under torch.autocast("cuda") with no dtype: the logits
    reaching ops.loss_terms are fp16 and the step ends with finite gradients."""
    from ctdd_b200 import make_config, ops
    from ctdd_b200.lib.models import forward_model as fm
    from ctdd_b200.lib.losses import losses_utils
    import ctdd_b200.lib.losses.losses  # noqa: F401
    case = ("autocast", "SDDMElbo", "gauss256", 4, 40, dict(logit_type="reverse_prob", nll_weight=0.01), 1.0, 7, 0)
    cfg = cases.loss_cfg(make_config, case, device="cuda")
    S, D = 256, 40

    class M(torch.nn.Module, fm.GaussianTargetRate):
        def __init__(self):
            torch.nn.Module.__init__(self)
            fm.GaussianTargetRate.__init__(self, cfg, "cuda")
            self.emb = torch.nn.Embedding(S, 64)
            self.out = torch.nn.Linear(64, S)

        def forward(self, x, t):
            return self.out(self.emb(x) + t.view(-1, 1, 1))

    torch.manual_seed(0)
    m = M().to("cuda")
    m.device = "cuda"
    dtypes = []
    real = ops.loss_terms

    def spy(logits, *a, **k):
        dtypes.append(logits.dtype)
        return real(logits, *a, **k)
    monkeypatch.setattr(ops, "loss_terms", spy)
    loss_obj = losses_utils.get_loss(cfg)
    loss_obj.seed = 3
    x0 = torch.randint(0, S, (4, D), device="cuda")
    with torch.autocast("cuda"):
        loss = loss_obj.calc_loss(x0, {"model": m, "optimizer": None, "n_iter": 0})
    loss.backward()
    assert dtypes == [f16]
    assert torch.isfinite(loss)
    for p in m.parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all()
    assert m.out.weight.grad.abs().max() > 0


@gpu
@pytest.mark.parametrize("kind_case", [bo.KINDS[0], bo.KINDS[1]], ids=["ctelbo", "sddm_tc"])
def test_loss_peak_memory_of_forward_backward(kind_case):
    """B = 64, D = 3072, S = 256: forward + backward with fp16 logits allocates no more than the tensor-core scratch, the
    table workspace, the fp16 gradient (2 B D S bytes) and a few MB."""
    nat = _nat()
    B, D, S = 64, 3072, 256
    _, kind, branch, crm = kind_case
    c, lh, _ = _loss_problem("gauss256", B, D, 9, 12.0)
    lh.requires_grad_(True)
    tc = kind != nat.LOSS_CTELBO
    bound = (int(nat.lib().ctdd_loss_tc_scratch_bytes(B, D, S)) if tc else 0) + int(nat.lib().ctdd_loss_workspace_bytes(kind, B, S))
    bound += 2 * B * D * S + (8 << 20)

    def rise():
        lh.grad = None
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        outs = bo._call(lh, kind, branch, crm, c)
        sum(w * o.sum() for w, o in zip(bo.SEED_W, outs)).backward()
        torch.cuda.synchronize()
        assert lh.grad.dtype == f16
        return torch.cuda.max_memory_allocated() - base

    rise()                                                    # warm-up: the allocator's first blocks
    assert rise() <= bound


@gpu
def test_loss_misaligned_fp16_view():
    """A contiguous fp16 view one element off 16-byte alignment: ops.loss_terms gives the outputs and gradient of an
    aligned copy (it clones the view)."""
    nat = _nat()
    B, D, S = 3, 29, 256
    c, lh, _ = _loss_problem("gauss256", B, D, 13, 12.0)
    buf = torch.zeros(B * D * S + 1, dtype=f16, device="cuda")
    buf[1:] = lh.reshape(-1)
    assert buf[1:].data_ptr() % 16 != 0
    for kind, branch, crm in ((nat.LOSS_SDDM, "reverse_prob", 0), (nat.LOSS_CRM, "reverse_prob", 2), (nat.LOSS_CTELBO, None, 0)):
        leaf = buf.detach().clone().requires_grad_(True)
        a = bo._call(leaf[1:].view(B, D, S), kind, branch, crm, c)
        sum(w * o.sum() for w, o in zip(bo.SEED_W, a)).backward()
        b, gb = bo._fwd_bwd(lh, kind, branch, crm, c)
        assert all(torch.equal(x.detach(), y) for x, y in zip(a, b)), kind
        assert leaf.grad.dtype == f16 and torch.equal(leaf.grad[1:].view(B, D, S), gb), kind


@gpu
def test_loss_gradient_overflow_gives_inf_where_fp32_rounding_does():
    """A loss scale that takes the fp16 logits gradient past 65504: the fp16 gradient holds ±inf exactly where the fp32
    gradient rounded to fp16 does (what torch.amp.GradScaler looks for), on the tensor-core and CUDA-core paths."""
    nat = _nat()
    c, lh, _ = _loss_problem("gauss256", 3, 40, 19, 12.0)
    for kind, branch in ((nat.LOSS_SDDM, "reverse_prob"), (nat.LOSS_CTELBO, None)):
        grads = []
        for L in (lh, lh.float()):
            leaf = L.detach().clone().requires_grad_(True)
            outs = bo._call(leaf, kind, branch, 0, c)
            ((outs[0].sum() + 0.01 * outs[4].sum()) * 2.0 ** 24).backward()
            grads.append(leaf.grad)
        gh, gf = grads
        want = gf.half()
        assert torch.isinf(want).any() and torch.isfinite(want).any(), kind
        assert gh.dtype == f16 and torch.equal(gh, want), kind


# ------------------------------------------------------------------------------------------------------- head
def _inputs(N, D, seed, lo=-3.0, hi=3.0):
    """(N, D) fp32 (mu, log_scale) on the device (the head takes fp32 or bf16 ones; fp16 ones are widened)."""
    mu, ls = ho.head_inputs(N * D, seed, lo, hi)
    return mu.view(N, D).cuda(), ls.view(N, D).cuda()


@gpu
@pytest.mark.parametrize("S", [256, 32, 5])
def test_head_forward_fp16_output(S):
    """logistic_logits(out_dtype=float16) equals the fp32 logits .half(), for fp32, bf16 and fp16 inputs: random rows,
    the edge rows, and the two torch.chunk halves of a (B, 2C, H, W) tensor; also into an output one element off its
    4-element alignment (the one-logit-per-thread kernel)."""
    from ctdd_b200 import ops
    mu, ls = _inputs(6, 50, 11 + S)
    em = torch.tensor(bh.EDGE_MU).view(1, -1).cuda()
    el = torch.tensor(bh.EDGE_LS).view(1, -1).cuda()
    both = torch.cat([mu.view(6, 2, 5, 5), ls.view(6, 2, 5, 5)], dim=1)
    cm, cl = torch.chunk(both, 2, dim=1)
    for fix in (False, True):
        for m, l in ((mu, ls), (em, el), (cm, cl)):
            for dt in (torch.float32, torch.bfloat16, f16):
                mi, li = m.to(dt), l.to(dt)
                ref = ops.logistic_logits(mi.float(), li.float(), S, fix)
                got = ops.logistic_logits(mi, li, S, fix, out_dtype=f16)
                assert got.dtype == f16 and torch.equal(got, ref.half()), (S, fix, dt)
        N, D = mu.shape
        buf = torch.zeros(N * D * S + 1, dtype=f16, device="cuda")
        out = buf[1:].view(N, D, S)
        got = ops.logistic_logits(mu, ls, S, fix, out=out, out_dtype=f16)
        assert got.data_ptr() == out.data_ptr() and torch.equal(got, ops.logistic_logits(mu, ls, S, fix).half())


@gpu
@pytest.mark.parametrize("S", [256, 32, 5])
def test_head_backward_fp16_gradient(S):
    """An fp16 incoming gradient, aligned and one element off 8-byte alignment, read by the raw entry point and by the
    autograd function: grad_mu / grad_log_scale equal the fp32 kernel's on the widened gradient bit for bit."""
    from ctdd_b200 import ops
    N, D = 6, 50
    mu, ls = _inputs(N, D, 31 + S, -2.5, 2.5)
    gen = torch.Generator(device="cuda").manual_seed(S)
    gh = torch.randn((N, D, S), generator=gen, device="cuda").half()
    buf = torch.zeros(N * D * S + 1, dtype=f16, device="cuda")
    buf[1:] = gh.reshape(-1)
    gv = buf[1:].view(N, D, S)
    assert gv.data_ptr() % 8 != 0
    for fix in (False, True):
        want = bh._fp32_backward(mu, ls, gh, S, fix)
        for m, l in ((mu, ls), (mu.to(torch.bfloat16), ls.to(torch.bfloat16))):
            want_m = bh._fp32_backward(m, l, gh, S, fix)
            got = bh._raw_backward(m, l, gh, S, fix)
            assert torch.equal(got[0], want_m[0]) and torch.equal(got[1], want_m[1]), (S, fix, m.dtype)
        for g in (gh, gv):
            mc, lc = mu.clone().requires_grad_(True), ls.clone().requires_grad_(True)
            out = ops.logistic_logits_autograd(mc, lc, S, fix, out_dtype=f16)
            assert out.dtype == f16
            out.backward(g)
            assert torch.equal(mc.grad, want[0]) and torch.equal(lc.grad, want[1]), (S, fix, g.data_ptr() % 8)
        # fp16 leaves: saved widened, gradients returned in fp16
        mh, lh = mu.half().requires_grad_(True), ls.half().requires_grad_(True)
        ops.logistic_logits_autograd(mh, lh, S, fix, out_dtype=f16).backward(gh)
        want_h = bh._fp32_backward(mu.half(), ls.half(), gh, S, fix)
        assert mh.grad.dtype == f16 and torch.equal(mh.grad, want_h[0].half()) and torch.equal(lh.grad, want_h[1].half())


@gpu
def test_head_loss_chain_from_fp16_head_is_bit_equal():
    """fp16 (mu, log_scale) through the model head (fp16 logits) into SDDMElbo's loss and back: grad_mu / grad_log_scale
    equal those of the chain built by hand from widened tensors (head on the fp32 inputs, its logits .half())."""
    from ctdd_b200 import ops
    from ctdd_b200.lib.models import models
    B, D, S = 4, 96, 256
    c = bh._loss_problem(B, D, 5)
    mu, ls = _inputs(B, D, 6, -1.0, 2.0)
    mu, ls = mu.half(), ls.half()
    mh, lh = mu.clone().requires_grad_(True), ls.clone().requires_grad_(True)
    logits = models._logistic_logits_autograd(mh, lh, S, False).view(B, D, S)
    assert logits.dtype == f16
    bh._sddm(logits, c).backward()
    mr, lr = mu.float().requires_grad_(True), ls.float().requires_grad_(True)
    ref = ops.logistic_logits_autograd(mr, lr, S, False).half()
    bh._sddm(ref, c).backward()
    assert torch.equal(logits.detach(), ref.detach())
    assert mh.grad.dtype == f16 and torch.equal(mh.grad, mr.grad.half()) and torch.equal(lh.grad, lr.grad.half())
    with pytest.raises(RuntimeError, match="one dtype"):
        models._logistic_logits_autograd(mh, lh.float(), S, False)


# ------------------------------------------------------------------------------------------------------- training
def _amp_step(cls, over, reference, scale, monkeypatch):
    """calc_loss under torch.autocast("cuda") (fp16) on a small image network ending in a 1x1 nn.Conv2d that emits
    (mu, log_scale) as the two torch.chunk halves of (B, 2C, H, W), then scaler.scale(loss).backward() and
    scaler.step().  `reference`: the head on mu.float(), log_scale.float(), its logits cast to fp16.  Returns (loss,
    parameter gradients before the step, whether the parameters moved, the scaler, logits dtypes seen by the loss)."""
    from ctdd_b200 import make_config, ops
    from ctdd_b200.lib.models import forward_model as fm, models
    from ctdd_b200.lib.losses import losses_utils
    import ctdd_b200.lib.losses.losses  # noqa: F401
    B, C, H, W, S = 4, 3, 8, 8, 256
    D = C * H * W
    case = ("amp", cls, "gauss256", B, D, over, 1.0, 7, 0)
    cfg = cases.loss_cfg(make_config, case, device="cuda")

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
            mu, ls = torch.chunk(self.out(e), 2, dim=1)         # fp16 under autocast
            mu = torch.tanh(mu)
            if reference:
                return ops.logistic_logits_autograd(mu.float(), ls.float(), S, True).view(Bx, D, S).half()
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
    opt = torch.optim.SGD(m.parameters(), lr=0.1)
    scaler = torch.amp.GradScaler("cuda", init_scale=scale, growth_interval=1000)
    before = [p.detach().clone() for p in m.parameters()]
    state = {"model": m, "optimizer": opt, "n_iter": 1}
    with torch.backends.cudnn.flags(enabled=True, benchmark=False, deterministic=True):
        with torch.autocast("cuda"):
            loss = loss_obj.calc_loss(x0, state) if cls in cases.LOSS_MINIBATCH_FIRST else loss_obj.calc_loss(state, x0)
        scaler.scale(loss).backward()
        grads = [p.grad.detach().clone() for p in m.parameters()]
        scaler.step(opt)
        scaler.update()
    monkeypatch.undo()
    moved = any(not torch.equal(a, p.detach()) for a, p in zip(before, m.parameters()))
    return loss.detach(), grads, moved, scaler, seen


AMP_CASES = [("CTElbo", dict()), ("SDDMElbo", dict(logit_type="reverse_prob", nll_weight=0.01))]


@gpu
@pytest.mark.parametrize("cls,over", AMP_CASES, ids=[c[0] for c in AMP_CASES])
def test_training_step_under_default_autocast_with_grad_scaler(cls, over, monkeypatch):
    """The image head under real fp16 autocast raises nothing and hands fp16 logits to the loss; the loss and the scaled
    parameter gradients agree with the widened chain up to the order of the loss kernels' atomicAdds (SDDMElbo's
    weights of the per-sample terms depend on their sums), and the scaler takes the step.  (This small network's fp16
    gradients already overflow at a scale of 2^10, so it runs at 1.)"""
    loss, grads, moved, scaler, seen = _amp_step(cls, over, False, 1.0, monkeypatch)
    rloss, rgrads, _, _, rseen = _amp_step(cls, over, True, 1.0, monkeypatch)
    assert seen and all(d == f16 for d in seen) and seen == rseen
    assert torch.isfinite(loss) and abs(float(loss) - float(rloss)) <= 1e-5 * abs(float(rloss)), (float(loss), float(rloss))
    for g, r in zip(grads, rgrads):
        assert torch.isfinite(g).all()
        assert float((g.float() - r.float()).abs().max()) <= 1e-3 * float(r.float().abs().max()), cls
    assert max(float(g.abs().max()) for g in grads) > 0
    assert moved and scaler.get_scale() == 1.0


@gpu
def test_training_step_overflow_is_skipped_by_grad_scaler(monkeypatch):
    """A loss scale that overflows the fp16 logits gradient: the gradients hold non-finite values, the scaler skips the
    step (the parameters stay) and lowers its scale."""
    cls, over = AMP_CASES[1]
    _, grads, moved, scaler, seen = _amp_step(cls, over, False, 2.0 ** 40, monkeypatch)
    assert seen == [f16]
    assert any(not torch.isfinite(g).all() for g in grads)
    assert not moved and scaler.get_scale() < 2.0 ** 40


# ------------------------------------------------------------------------------------------------------- CPU
def test_fp16_dtype_value_and_refusals_before_any_cuda_call():
    """No device needed: DTYPE_F16 is 2; unknown dtypes are still refused with status 2 by the step, loss and head entry
    points, and so is F16 as head_dtype and as the head's in_dtype."""
    nat = _nat()
    L = nat.lib()
    assert (nat.DTYPE_F32, nat.DTYPE_BF16, nat.DTYPE_F16) == (0, 1, 2)
    assert nat.logits_dtype_of(torch.empty(1, dtype=f16)) == nat.DTYPE_F16
    dummy = 0x1000
    for bad in (3, 7, -1):
        p = nat.StepParams(mode=nat.MODE_TAU_LEAP, branch=nat.BRANCH_TAULDR, impl=nat.IMPL_SIMT, N=2, D=3, S=4,
                           logits=dummy, ld_logits=4, batch_stride_logits=12, x_eval=dummy, Q=dummy, QT=dummy, Rb=dummy,
                           RbT=dummy, x_out=dummy, logits_dtype=bad)
        assert L.ctdd_reverse_step(ctypes.byref(p), None) == 2 and b"logits_dtype" in L.ctdd_last_error()
        ptrs = {k: dummy for k in ("logits", "Q", "QT", "Rb", "beta", "x0", "xt", "x_tilde", "out_a", "out_b", "out_c",
                                   "out_d", "out_nll", "ga", "gb", "gd", "gn", "grad_logits", "workspace")}
        lp = nat.LossParams(kind=nat.LOSS_CTELBO, B=2, D=3, S=4, eps=1e-9, logits_dtype=bad, **ptrs)
        for fn in (L.ctdd_loss_forward, L.ctdd_loss_backward):
            assert fn(ctypes.byref(lp), None) == 2 and b"logits_dtype" in L.ctdd_last_error()
        assert L.ctdd_logistic_logits_ex(dummy, dummy, 0, 2, 3, 3, 256, 0, dummy, bad, None) == 2
        assert L.ctdd_logistic_logits_backward_ex(dummy, dummy, 0, dummy, bad, 2, 3, 3, 256, 0, dummy, dummy, None) == 2
    # fp16 (mu, log_scale) are widened by the caller: the fused head and the head entry points refuse them
    p = nat.StepParams(mode=nat.MODE_TAU_LEAP, branch=nat.BRANCH_TAULDR, impl=nat.IMPL_TC, N=2, D=3, S=256, x_eval=dummy,
                       Q=dummy, QT=dummy, Rb=dummy, RbT=dummy, x_out=dummy, head=nat.HEAD_LOGISTIC, head_mu=dummy,
                       head_log_scale=dummy, head_batch_stride=3, head_dtype=nat.DTYPE_F16)
    assert L.ctdd_reverse_step(ctypes.byref(p), None) == 2 and b"head_dtype" in L.ctdd_last_error()
    assert L.ctdd_logistic_logits_ex(dummy, dummy, nat.DTYPE_F16, 2, 3, 3, 256, 0, dummy, nat.DTYPE_F16, None) == 2
    assert b"dtype" in L.ctdd_last_error()
    assert L.ctdd_logistic_logits_backward_ex(dummy, dummy, nat.DTYPE_F16, dummy, nat.DTYPE_F16, 2, 3, 3, 256, 0, dummy,
                                              dummy, None) == 2
    assert b"dtype" in L.ctdd_last_error()
