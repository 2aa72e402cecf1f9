"""bf16 logits in the reverse step: a call with bf16 logits L returns the states, counters, rr and ratio of the same call
on L.float() bit for bit, on every kernel path, in every mode and branch, and through every sampler class."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import cases
from helpers import oracle_forward, product_model

gpu = pytest.mark.gpu


def _nat():
    from ctdd_b200 import _native as nat
    return nat


def _tables(fp, t, dev="cuda"):
    tt = torch.tensor([t], dtype=torch.float64).to(torch.float32)
    Q = fp.transition(tt)[0]
    return dict(Q=Q.to(dev).contiguous(), QT=Q.t().contiguous().to(dev), Rb=fp.base_rate.to(dev).contiguous(),
                RbT=fp.base_rate.t().contiguous().to(dev), beta=float(fp.beta(tt)[0]))


def _problem(fwd, N, D, t, seed, width, scale=0.5):
    """The inputs of test_gpu_parity's STEP_CASES, with the logits rounded to bf16."""
    fp = oracle_forward(fwd)
    S = fp.S
    g = np.random.Generator(np.random.PCG64(seed))
    x0 = g.integers(0, S, (N, D))
    s = np.arange(S)
    logits = scale * 4.0 * g.standard_normal((N, D, S))
    if width is not None:
        logits = logits - (s[None, None, :] - x0[:, :, None]) ** 2 / (2.0 * width ** 2)
    x = np.clip(x0 + g.integers(-2, 3, (N, D)), 0, S - 1)
    lb = torch.from_numpy(logits.astype(np.float32)).to(torch.bfloat16).cuda()
    return fp, lb, torch.from_numpy(x).to(torch.int32).cuda(), S


def _tc(tb, branch, S):
    from ctdd_b200 import ops
    nat = _nat()
    if S != 256 or branch not in (nat.BRANCH_TAULDR, nat.BRANCH_SDDM_REVERSE_PROB):
        return None, None
    return ops.prep_tc_tables(tb["Q"][None], tb["QT"][None], tb["Rb"], 1e-9, branch)[0], ops.prep_tc_static(tb["Rb"])


def _step(mode, branch, logits, x, tb, h, S, N, D, **kw):
    from ctdd_b200 import ops
    stats = torch.zeros(8, dtype=torch.int64, device="cuda")
    out = ops.reverse_step(mode, branch, logits, x, tb["Q"], tb["QT"], tb["Rb"], tb["RbT"], tb["beta"], h, 1e-9, N=N, D=D,
                           S=S, stats=stats, **kw)
    out["stats"] = stats
    return out


def _assert_same(a, b, what):
    for k in ("x", "stats", "rr", "ratio"):
        if a.get(k) is None and b.get(k) is None:
            continue
        assert a[k].dtype == b[k].dtype and torch.equal(a[k], b[k]), (what, k)


def _both(lb, call, what):
    """call(logits) with the bf16 logits and with their widened copy: bit-identical outputs."""
    a, b = call(lb), call(lb.float())
    _assert_same(a, b, what)
    return a


STEP_CASES = [
    # fwd, N, D, t, h, loss, logit_type, width  (test_gpu_parity.STEP_CASES, plus the S = 2 tauLDR branch that selects the
    # lean small-S instantiations and the S = 256 branches of the CUDA-core block kernel)
    ("gauss256", 6, 40, 0.9, 0.004, "CTElbo", None, 12.0),
    ("gauss256", 6, 40, 0.2, 0.01, "CatRM", "reverse_prob", 12.0),
    ("gauss32", 16, 33, 0.5, 0.02, "NLL", None, 3.0),
    ("gauss32", 16, 33, 0.5, 0.02, "CatRM", "direct", 3.0),
    ("gauss32", 16, 33, 0.5, 0.02, "ScoreElbo", "reverse_logscale", 3.0),
    ("univar3_logsqr", 32, 225, 0.4, 0.05, "CTElbo", None, None),
    ("univar2_sqrtcos", 64, 32, 0.6, 0.05, "CatRMNLL", "reverse_prob", None),
    ("univar5_log", 24, 19, 0.6, 0.05, "CTElbo", None, None),
    ("univar2_sqrtcos", 64, 33, 0.6, 0.05, "CTElbo", None, None),
    ("gauss256", 6, 40, 0.5, 0.01, "CatRM", "direct", 12.0),
    ("gauss256", 6, 40, 0.5, 0.01, "ScoreElbo", "reverse_logscale", 12.0),
]


@gpu
@pytest.mark.parametrize("impl_name", ["simt", "auto"])
@pytest.mark.parametrize("sc", STEP_CASES, ids=[f"{c[0]}-{c[5]}-{c[6]}-D{c[2]}" for c in STEP_CASES])
def test_every_mode_and_path_bit_equal(sc, impl_name):
    """Every mode (reject_multi on and off where it applies), on the CUDA-core kernels and on what IMPL_AUTO picks; at
    S = 256 with tcgen05 tables IMPL_TC is forced, so every step_q_kernel mode and both Euler modes run there."""
    nat = _nat()
    fwd, N, D, t, h, loss_name, logit_type, width = sc
    fp, lb, x, S = _problem(fwd, N, D, t, 11, width)
    tb = _tables(fp, t)
    branch = nat.branch_for(loss_name, logit_type)
    impl, tct, tcs = nat.IMPL_SIMT, None, None
    if impl_name == "auto":
        tct, tcs = _tc(tb, branch, S)
        impl = nat.IMPL_TC if tct is not None else nat.IMPL_AUTO
    g = np.random.Generator(np.random.PCG64(5))
    xb = torch.from_numpy(np.clip(x.cpu().numpy() + g.integers(-1, 2, x.shape), 0, S - 1)).to(torch.int32).cuda()
    kw = dict(impl=impl, tc_tables=tct, tc_static=tcs, seed=4242)
    runs = [(nat.MODE_TAU_LEAP, dict(reject_multi=False, offset=3)), (nat.MODE_TAU_LEAP, dict(reject_multi=True, offset=3)),
            (nat.MODE_TAU_LEAP_CORR, dict(offset=5)), (nat.MODE_MIDPOINT_DRIFT, dict(offset=0)),
            (nat.MODE_MIDPOINT_JUMP, dict(reject_multi=True, offset=7, x_base=xb)),
            (nat.MODE_EULER, dict(offset=9)), (nat.MODE_EULER_CORR, dict(offset=10)),
            (nat.MODE_RATES_ONLY, dict(want_rr=True, want_ratio=True))]
    if impl != nat.IMPL_TC:       # the CUDA-core kernels also write the rates in sampling modes; only they have the exact mode
        runs += [(nat.MODE_TAU_LEAP, dict(offset=4, want_rr=True, want_ratio=True)), (nat.MODE_EXACT, dict(offset=11))]
    moved = 0
    for mode, extra in runs:
        out = _both(lb, lambda L: _step(mode, branch, L, x, tb, h, S, N, D, **kw, **extra), (mode, extra.get("reject_multi")))
        if out["x"] is not None:
            moved += int((out["x"] != x).sum())
    assert moved > 0                                                              # the steps do move states


@gpu
def test_fp16_logits_keep_the_widening_copy():
    """fp16 (not served natively) is still widened to fp32 before the step: same results as the fp32 call."""
    nat = _nat()
    fp, lb, x, S = _problem("gauss32", 16, 33, 0.5, 3, 3.0)
    tb = _tables(fp, 0.5)
    lf = lb.float()
    a = _step(nat.MODE_TAU_LEAP, nat.BRANCH_TAULDR, lf.half(), x, tb, 0.02, S, 16, 33, seed=1, offset=1, want_rr=True)
    b = _step(nat.MODE_TAU_LEAP, nat.BRANCH_TAULDR, lf.half().float(), x, tb, 0.02, S, 16, 33, seed=1, offset=1, want_rr=True)
    _assert_same(a, b, "fp16")


@gpu
@pytest.mark.parametrize("fwd,loss_name,mode_name", [("univar2_sqrtcos", "CTElbo", "tau_leap"), ("univar3_logsqr", "CTElbo", "euler"),
                                                     ("univar5_log", "CTElbo", "tau_leap"), ("gauss256", "CTElbo", "tau_leap"),
                                                     ("gauss256", "CatRM", "euler")])
def test_ragged_rows_row_offset_and_shards(fwd, loss_name, mode_name):
    """Row counts that are no multiple of 8 or of the 128-row pair tile (1, 7, 129, several tiles), a non-zero row offset,
    and two shards against one launch - bf16 against the widened logits each time."""
    nat = _nat()
    mode = nat.MODE_EULER if mode_name == "euler" else nat.MODE_TAU_LEAP
    for (N, D) in ((1, 1), (7, 1), (129, 1), (13, 21), (40, 37)):
        fp, lb, x, S = _problem(fwd, N, D, 0.5, 23 + N, 12.0 if fwd == "gauss256" else None)
        tb = _tables(fp, 0.5)
        branch = nat.branch_for(loss_name, "reverse_prob")
        tct, tcs = _tc(tb, branch, S)
        kw = dict(impl=(nat.IMPL_TC if tct is not None else nat.IMPL_AUTO), tc_tables=tct, tc_static=tcs, seed=31, offset=6)
        row0 = 8 * 37
        full = _both(lb, lambda L: _step(mode, branch, L, x, tb, 0.08, S, N, D, row_offset=row0, **kw), (N, D))
        if N * D >= 16:
            n_lo = 8                                               # 8 * D rows: the second shard's offset stays a multiple of 8
            lo = _both(lb[:n_lo], lambda L: _step(mode, branch, L, x[:n_lo], tb, 0.08, S, n_lo, D, row_offset=row0, **kw), "lo")
            hi = _both(lb[n_lo:], lambda L: _step(mode, branch, L, x[n_lo:], tb, 0.08, S, N - n_lo, D,
                                                  row_offset=row0 + n_lo * D, **kw), "hi")
            assert torch.equal(full["x"], torch.cat([lo["x"], hi["x"]]))
            assert torch.equal(full["stats"], lo["stats"] + hi["stats"])


@gpu
def test_small_s_grid_stride_kernel_at_scale():
    """The S = 2 tau-leap kernel strides over its capped grid when the batch has more rows than the grid has threads
    times 8 (C1 at 8x its batch: 16.8 M rows)."""
    nat = _nat()
    fp = oracle_forward("univar2_sqrtcos")
    tb = _tables(fp, 0.6)
    N, D, S = 1 << 19, 32, 2
    gen = torch.Generator(device="cuda").manual_seed(3)
    lb = (torch.randn((N, D, S), generator=gen, device="cuda") * 2.0).to(torch.bfloat16)
    x = torch.randint(0, S, (N, D), generator=gen, device="cuda", dtype=torch.int32)
    out = _both(lb, lambda L: _step(nat.MODE_TAU_LEAP, nat.BRANCH_TAULDR, L, x, tb, 0.05, S, N, D, reject_multi=True, seed=2,
                                    offset=1), "C1x8")
    assert int(out["stats"][nat.STAT_CHANGED_BASE]) > 0


@gpu
@pytest.mark.parametrize("fwd,loss_name,logit_type", [("gauss256", "CTElbo", None), ("gauss256", "CatRM", "reverse_prob"),
                                                      ("gauss32", "CTElbo", None)])
def test_strided_views(fwd, loss_name, logit_type):
    """logits[:, c:, :] of a bf16 (N, D_total, S) tensor (the conditional samplers' view) on the tcgen05 path (S = 256)
    and the CUDA-core path: equal to the widened view and to a contiguous bf16 copy."""
    nat = _nat()
    for (N, Dfull, c) in ((3, 29, 8), (6, 200, 72), (40, 340, 40)):
        D = Dfull - c
        fp, lb_full, x_full, S = _problem(fwd, N, Dfull, 0.35, 41 + N, 12.0 if fwd == "gauss256" else 3.0)
        tb = _tables(fp, 0.35)
        branch = nat.branch_for(loss_name, logit_type)
        tct, tcs = _tc(tb, branch, S)
        x = x_full[:, c:].contiguous()
        impl = nat.IMPL_TC if tct is not None else nat.IMPL_SIMT
        for mode in (nat.MODE_TAU_LEAP, nat.MODE_TAU_LEAP_CORR, nat.MODE_MIDPOINT_DRIFT, nat.MODE_EULER):
            kw = dict(impl=impl, tc_tables=tct, tc_static=tcs, seed=11, offset=3)
            view = _both(lb_full, lambda L: _step(mode, branch, L, x, tb, 0.01, S, N, D, logits_offset_elems=c * S,
                                                  batch_stride=Dfull * S, **kw), (N, Dfull, c, mode))
            copy = _step(mode, branch, lb_full[:, c:, :].contiguous(), x, tb, 0.01, S, N, D, **kw)
            _assert_same(view, copy, ("copy", N, Dfull, c, mode))


@gpu
def test_misaligned_bf16_rows_leave_the_tensor_path():
    """A bf16 view whose batch stride is a multiple of 4 but not of 8 elements (16-byte aligned for fp32, not for bf16):
    IMPL_TC refuses it, IMPL_AUTO runs it on the CUDA-core path and matches the widened view there."""
    from ctdd_b200 import ops
    nat = _nat()
    N, D = 5, 24
    fp, lb, x, S = _problem("gauss256", N, D, 0.35, 7, 12.0)
    tb = _tables(fp, 0.35)
    tct, tcs = _tc(tb, nat.BRANCH_TAULDR, S)
    stride = D * S + 4
    buf = torch.zeros((N, stride), dtype=torch.bfloat16, device="cuda")
    buf[:, :D * S] = lb.reshape(N, D * S)
    kw = dict(tc_tables=tct, tc_static=tcs, seed=3, offset=2, batch_stride=stride)
    with pytest.raises(RuntimeError, match="rc=3"):
        _step(nat.MODE_TAU_LEAP, nat.BRANCH_TAULDR, buf, x, tb, 0.01, S, N, D, impl=nat.IMPL_TC, **kw)
    for mode in (nat.MODE_TAU_LEAP, nat.MODE_EULER):
        a = _step(mode, nat.BRANCH_TAULDR, buf, x, tb, 0.01, S, N, D, impl=nat.IMPL_AUTO, **kw)
        b = _step(mode, nat.BRANCH_TAULDR, buf.float(), x, tb, 0.01, S, N, D, impl=nat.IMPL_SIMT, **kw)
        _assert_same(a, b, mode)
    # the same stride in fp32 is 16-byte aligned: the tensor path takes it (and the bf16 call above did not)
    assert ops.reverse_step(nat.MODE_TAU_LEAP, nat.BRANCH_TAULDR, buf.float(), x, tb["Q"], tb["QT"], tb["Rb"], tb["RbT"],
                            tb["beta"], 0.01, 1e-9, N=N, D=D, S=S, impl=nat.IMPL_TC, **kw)["x"] is not None


@gpu
def test_full_c4_size_tau_leap():
    """One tau-leap step at the C4 shape (B = 1024, D = 3072, S = 256): the 1.6 GB bf16 tensor against its 3.2 GB
    widened copy."""
    nat = _nat()
    B, D, S = 1024, 3072, 256
    fp = oracle_forward("gauss256")
    tb = _tables(fp, 0.5)
    tct, tcs = _tc(tb, nat.BRANCH_TAULDR, S)
    gen = torch.Generator(device="cuda").manual_seed(9)
    x = torch.randint(0, S, (B, D), generator=gen, device="cuda", dtype=torch.int32)
    lb = torch.randn((B, D, S), generator=gen, device="cuda", dtype=torch.bfloat16)
    lb -= ((torch.arange(S, device="cuda", dtype=torch.float32).view(1, 1, S) - x.unsqueeze(-1)) ** 2 / 128.0).to(torch.bfloat16)
    kw = dict(impl=nat.IMPL_TC, tc_tables=tct, tc_static=tcs, seed=5, offset=1)
    a = _step(nat.MODE_TAU_LEAP, nat.BRANCH_TAULDR, lb, x, tb, 0.01, S, B, D, **kw)
    lf = lb.float()
    del lb
    b = _step(nat.MODE_TAU_LEAP, nat.BRANCH_TAULDR, lf, x, tb, 0.01, S, B, D, **kw)
    _assert_same(a, b, "C4")
    assert int(a["stats"][nat.STAT_CHANGED_BASE]) > 0


# ------------------------------------------------------------------------------------------------------- samplers
def _by_name(name):
    return next(c for c in cases.SAMPLERS + cases.SAMPLERS_S256 if c[0] == name)


def _sample(case, dtype):
    """Run a sampler on the stub network whose logits are rounded to bf16; `dtype` is what the network hands over."""
    from ctdd_b200 import make_config
    from ctdd_b200.lib.sampling import sampling_utils
    import ctdd_b200.lib.sampling.sampling  # noqa: F401
    name, cls, fwd, N, D, loss_name, logit_type, stub, over, max_t, seed = case
    cfg = cases.sampler_cfg(make_config, case)
    cfg.device = "cuda"
    S = cfg.data.S
    m = product_model(fwd, cfg, D, seed, stub[0], stub[1])
    net = m.forward
    m.forward = lambda x, t: net(x, t).to(torch.bfloat16).to(dtype)
    cfg.sampler.name = cls
    sampler = sampling_utils.get_sampler(cfg)
    sampler.seed = seed
    args = ()
    if "condition_dim" in over:
        g = np.random.Generator(np.random.PCG64(seed))
        args = (torch.from_numpy(g.integers(0, S, (N, over["condition_dim"]))),)
    res = sampler.sample(m, N, *args)
    return res if isinstance(res, tuple) else (res,)


SAMPLER_CASES = ["taul_gauss256_corr_crm", "taul_uni2_nonord", "lbjf_univar3_pc", "lbjf_gauss256", "midpoint_univar3",
                 "midpoint_gauss256_tauldr", "pctaul_gauss32", "condtaul_gauss32", "condpctaul_gauss32", "exact_univar3"]


@gpu
@pytest.mark.parametrize("name", SAMPLER_CASES)
def test_samplers_take_bf16_network_output(name):
    """The same seeded sampler run with the network's bf16 logits and with their fp32 widening: identical samples and
    diagnostics."""
    case = _by_name(name)
    a, b = _sample(case, torch.bfloat16), _sample(case, torch.float32)
    assert len(a) == len(b)
    for u, v in zip(a, b):
        np.testing.assert_array_equal(np.asarray(u), np.asarray(v), err_msg=name)


@gpu
def test_step_engine_reads_bf16_without_widening_copy():
    """StepEngine.step with bf16 logits allocates nothing of the size of the logits (no hidden .float())."""
    from ctdd_b200 import make_config
    from ctdd_b200.lib.sampling.sampling import StepEngine
    from helpers import fwd_cfg
    nat = _nat()
    N, D, S = 256, 1024, 256                                       # fp32 (N, D, S) would be 256 MiB
    cfg = fwd_cfg("gauss256", make_config)
    m = product_model("gauss256", cfg, D, 3, 0.3, 12.0)
    for impl in (nat.IMPL_AUTO, nat.IMPL_SIMT):
        eng = StepEngine(cfg, m, N, D, S, [0.5], nat.BRANCH_TAULDR, 1e-9, impl=impl, seed=1)
        gen = torch.Generator(device="cuda").manual_seed(1)
        lb = torch.randn((N, D, S), generator=gen, device="cuda", dtype=torch.bfloat16)
        x = torch.randint(0, S, (N, D), generator=gen, device="cuda", dtype=torch.int32)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        x_new, _ = eng.step(nat.MODE_TAU_LEAP, lb, x, 0, 0.01)
        torch.cuda.synchronize()
        assert torch.cuda.max_memory_allocated() - base < N * D * S * 4 // 16, impl
        assert x_new.shape == (N, D)


# ------------------------------------------------------------------------------------------------------- CPU
def test_unknown_logits_dtype_is_refused_before_any_cuda_call():
    """The ABI check needs no device: dummy non-null pointers, an unknown logits_dtype -> status 2 and a message."""
    nat = _nat()
    L = nat.lib()
    dummy = 0x1000
    p = nat.StepParams(mode=nat.MODE_TAU_LEAP, branch=nat.BRANCH_TAULDR, impl=nat.IMPL_SIMT, N=2, D=3, S=4,
                       logits=dummy, ld_logits=4, batch_stride_logits=12, x_eval=dummy, Q=dummy, QT=dummy, Rb=dummy, RbT=dummy,
                       x_out=dummy, logits_dtype=7)
    assert L.ctdd_reverse_step(ctypes.byref(p), None) == 2
    assert b"logits_dtype" in L.ctdd_last_error()
    assert (nat.DTYPE_F32, nat.DTYPE_BF16) == (0, 1)
    assert nat.StepParams.logits_dtype.offset > nat.StepParams.head_batch_stride.offset
