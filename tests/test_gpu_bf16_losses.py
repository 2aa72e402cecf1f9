"""bf16 logits in the training losses: ops.loss_terms with bf16 logits L returns the per-sample terms of the same call on
L.float() (bit for bit up to the order of the per-CTA atomicAdds) and a bf16 gradient equal to that call's fp32 gradient
rounded to bf16, bit for bit, on every kernel path, for every loss kind and through every loss class."""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import cases, ref_harness as rh
from oracle.make_golden_losses import minibatch_for
from helpers import oracle_forward

gpu = pytest.mark.gpu

# fixed weights of (out_a, out_b, out_c, out_d, out_nll) in the backward seed: the gradient does not depend on the outputs
SEED_W = (1.0, 0.3, 0.0, 0.1, 0.01)


def _nat():
    from ctdd_b200 import _native as nat
    return nat


def _problem(fwd, B, D, seed, width):
    """Per-sample q_{t|0}, noised states and logits (rounded to bf16) for B samples of D dimensions."""
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
    return c, torch.from_numpy(logits.astype(np.float32)).to(torch.bfloat16).cuda(), S


# (name, kind, logit branch, crm_type)
KINDS = [("ctelbo", 0, None, 0), ("sddm_rp", 2, "reverse_prob", 0), ("sddm_logscale", 2, "reverse_logscale", 0),
         ("sddm_direct", 2, "direct", 0), ("crm_rm", 1, "reverse_prob", 0), ("crm_mle", 1, "reverse_prob", 1),
         ("crm_elbo", 1, "reverse_prob", 2), ("crm_mle_direct", 1, "direct", 1)]


def _call(logits, kind, branch, crm, c, rows=None):
    """ops.loss_terms on every sample's rows `rows` (None: all of them); the CT-ELBO family with x~, SDDM at x~, ratio
    matching at x_t."""
    from ctdd_b200 import ops
    nat = _nat()
    sl = lambda t: t if rows is None else t[:, rows].contiguous()
    xt = c["xt"] if kind == nat.LOSS_CRM else c["xtil"]
    kw = dict(Q=c["Q"], QT=c["QT"], Rb=c["Rb"], beta=c["beta"], x0=sl(c["x0"]), xt=sl(xt),
              x_tilde=sl(c["xtil"]) if kind == nat.LOSS_CTELBO else None, eps=1e-9, crm_type=crm)
    if branch is not None:
        kw["logit_branch"] = nat.branch_for("CatRM", branch)
    return ops.loss_terms(logits if rows is None else logits[:, rows], kind, **kw)


def _fwd_bwd(logits, kind, branch, crm, c):
    lg = logits.detach().clone().requires_grad_(True)
    outs = _call(lg, kind, branch, crm, c)
    sum(w * o.sum() for w, o in zip(SEED_W, outs)).backward()
    return [o.detach() for o in outs], lg.grad


def _atomic_bound(logits, kind, branch, crm, c, R):
    """Largest difference two runs may show in each per-sample output: each CTA adds its partial P_c (computed the same
    way in both runs) to the output with atomicAdd, in an order that may differ.  Accumulating n partials from 0 in fp32
    is off the exact sum by at most (n - 1) u sum_c |P_c| (u = 2^-24), so two orders differ by at most twice that.
    sum_c |P_c| comes from one call per CTA's row block: out_a, out_b, out_d and out_nll are sums of per-row terms, so the
    call on a row block returns that CTA's partial exactly.  out_c (sig_norm) also depends on the whole sample through
    baseZ, but its terms w / Z are all >= 0, so sum_c |P_c| = |out_c|."""
    D = logits.shape[1]
    n = math.ceil(D / R)
    if n == 1:
        return None                                            # one CTA per sample: no reordering, bit-equal outputs
    with torch.no_grad():
        full = [o.double().abs() for o in _call(logits.float(), kind, branch, crm, c)]
        mass = [torch.zeros_like(full[0]) for _ in range(5)]
        for d0 in range(0, D, R):
            for k, o in enumerate(_call(logits.float(), kind, branch, crm, c, slice(d0, d0 + R))):
                mass[k] += o.double().abs()
    mass[2] = full[2]
    return [2.0 * (n - 1) * 2.0 ** -24 * m * 1.001 + 1e-30 for m in mass]


def _compare(lb, kind, branch, crm, c, R, what):
    ob, gb = _fwd_bwd(lb, kind, branch, crm, c)
    of, gf = _fwd_bwd(lb.float(), kind, branch, crm, c)
    assert torch.isfinite(gf).all() and all(torch.isfinite(o).all() for o in of), what
    assert gb.dtype == torch.bfloat16 and gf.dtype == torch.float32, what
    assert torch.equal(gb, gf.to(torch.bfloat16)), what
    bound = _atomic_bound(lb, kind, branch, crm, c, R)
    for k, (a, b) in enumerate(zip(ob, of)):
        if bound is None:
            assert torch.equal(a, b), (what, k)
        else:
            assert ((a.double() - b.double()).abs() <= bound[k]).all(), (what, k, (a - b).abs().max().item())
    assert gf.abs().max() > 0, what
    return ob, gb


# (forward process, B, D, width): one CTA per sample, and ragged D over several CTAs (B > 1, row tails of both tilings).
# At S = 256 the width keeps the logits within 21 of each other: the `direct` branch takes exp(ll_s - ll_x) of them.
SHAPES = [("univar3_logsqr", 3, 5, None), ("univar3_logsqr", 4, 45, None), ("gauss32", 3, 8, 3.0), ("gauss32", 4, 45, 3.0),
          ("gauss256", 3, 32, 40.0), ("gauss256", 3, 100, 40.0)]


@gpu
@pytest.mark.parametrize("shape", SHAPES, ids=[f"{s[0]}-B{s[1]}-D{s[2]}" for s in SHAPES])
@pytest.mark.parametrize("kind_case", KINDS, ids=[k[0] for k in KINDS])
def test_every_path_and_kind_through_loss_terms(shape, kind_case):
    """CUDA-core kernel at S = 3 and S = 32 (8-row CTAs) and at S = 256 (32-row CTAs: CT-ELBO, the `direct` branch, and
    SDDM / CRM with use_tc = False), and the tensor-core path at S = 256 (SDDM and CRM with reverse_prob /
    reverse_logscale)."""
    from ctdd_b200 import ops
    fwd, B, D, width = shape
    _, kind, branch, crm = kind_case
    c, lb, S = _problem(fwd, B, D, 17 + D, width)
    R = 32 if S == 256 else 8
    tc_modes = (True, False) if S == 256 and kind != 0 and branch != "direct" else (True,)
    for tc in tc_modes:
        ops._LossTerms.use_tc = tc
        try:
            _compare(lb, kind, branch, crm, c, R, (kind_case[0], shape, tc))
        finally:
            ops._LossTerms.use_tc = True


@gpu
@pytest.mark.parametrize("kind_case", [KINDS[0], KINDS[1]], ids=["ctelbo", "sddm_tc"])
def test_c5_size_gradient_bit_equal(kind_case):
    """B = 16, D = 3072, S = 256 (the C5 shape at a small batch): SDDM on the tensor-core path and CT-ELBO."""
    B, D, S = 16, 3072, 256
    _, kind, branch, crm = kind_case
    c, lb, _ = _problem("gauss256", B, D, 5, 12.0)
    _, gb = _fwd_bwd(lb, kind, branch, crm, c)
    lf = lb.float()
    _, gf = _fwd_bwd(lf, kind, branch, crm, c)
    assert gb.dtype == torch.bfloat16 and torch.equal(gb, gf.to(torch.bfloat16))


# ------------------------------------------------------------------------------------------------------- loss classes
LOSS_CLASS_CASES = ["ctelbo_gauss32", "ctelbo_gauss256", "ctelbo_gauss32_2pass", "nll_univar3", "ctelbolambda_uni2",
                    "condctelbo_gauss32", "condctelbo_gauss32_2pass", "catrm_gauss32_rm", "catrm_gauss32_mle_direct",
                    "catrmnll_gauss256", "scoreelbo_gauss32", "sddmelbo_gauss256", "sddmelbo_uni2_direct"]


def _class_loss(case, to_fp32):
    """calc_loss + backward() with the stub network ending in .to(torch.bfloat16) (to_fp32: then .float())."""
    from ctdd_b200 import make_config
    from ctdd_b200.lib.models import forward_model as fm
    from ctdd_b200.lib.losses import losses_utils
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
            out = self.net(x, t).to(torch.bfloat16)
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
@pytest.mark.parametrize("name", LOSS_CLASS_CASES)
def test_loss_classes_take_bf16_network_output(name):
    """Every loss class on a network whose output is bf16, against the same network widening it to fp32.  Every case has
    at most two CTAs per sample, and two partials added to zero give the same float in either order, so the atomic
    bound is zero here: the loss, d loss / d w and the logits gradient the network sees are bit-equal, and that gradient
    is bf16 on both routes (on the fp32 route autograd rounds it when it passes the .float())."""
    case = next(c for c in cases.LOSSES if c[0] == name)
    lb, wb, seen_b = _class_loss(case, False)
    lf, wf, seen_f = _class_loss(case, True)
    assert torch.isfinite(lb) and torch.equal(lb, lf), (lb.item(), lf.item())
    assert torch.equal(wb, wf) and wb.abs().max() > 0
    assert len(seen_b) == len(seen_f)
    for a, b in zip(seen_b, seen_f):
        assert a.grad is not None and a.grad.dtype == torch.bfloat16 and torch.equal(a.grad, b.grad)


@gpu
def test_real_autocast_with_linear_output_layer(monkeypatch):
    """SDDMElbo on a network with an nn.Linear output layer run under torch.autocast("cuda", dtype=torch.bfloat16): the
    logits reaching ops.loss_terms are bf16 and the step ends with finite gradients."""
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
    with torch.autocast("cuda", dtype=torch.bfloat16):
        loss = loss_obj.calc_loss(x0, {"model": m, "optimizer": None, "n_iter": 0})
    loss.backward()
    assert dtypes == [torch.bfloat16]
    assert torch.isfinite(loss)
    for p in m.parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all()
    assert m.out.weight.grad.abs().max() > 0


# ------------------------------------------------------------------------------------------------------- memory
@gpu
@pytest.mark.parametrize("kind_case", [KINDS[0], KINDS[1]], ids=["ctelbo", "sddm_tc"])
def test_peak_memory_of_forward_backward(kind_case):
    """B = 64, D = 3072, S = 256: forward + backward with bf16 logits allocates no more than the tensor-core scratch, the
    table workspace, the bf16 gradient (2 B D S bytes) and a few MB.  The former route (.float() before the loss, the
    gradient cast back by autograd) also holds the 4 B D S-byte copy and the fp32 gradient, at least 4 B D S bytes more."""
    from ctdd_b200 import ops
    nat = _nat()
    B, D, S = 64, 3072, 256
    _, kind, branch, crm = kind_case
    c, lb, _ = _problem("gauss256", B, D, 9, 12.0)
    lb.requires_grad_(True)
    tc = kind != nat.LOSS_CTELBO
    bound = (int(nat.lib().ctdd_loss_tc_scratch_bytes(B, D, S)) if tc else 0) + int(nat.lib().ctdd_loss_workspace_bytes(kind, B, S))
    bound += 2 * B * D * S + (8 << 20)

    def rise(widen):
        lb.grad = None
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        outs = _call(lb.float() if widen else lb, kind, branch, crm, c)
        sum(w * o.sum() for w, o in zip(SEED_W, outs)).backward()
        torch.cuda.synchronize()
        assert lb.grad.dtype == torch.bfloat16
        return torch.cuda.max_memory_allocated() - base

    rise(False)                                               # warm-up: the allocator's first blocks
    new, old = rise(False), rise(True)
    assert new <= bound, (new, bound)
    assert old >= bound + 4 * B * D * S, (old, bound)


# ------------------------------------------------------------------------------------------------------- alignment
@gpu
def test_misaligned_bf16_view():
    """A contiguous bf16 view one element off 16-byte alignment: ops.loss_terms gives the outputs and gradient of an
    aligned copy (it clones the view).  The raw ABI call with that pointer on the tensor-core path returns status 2 and
    launches nothing."""
    nat = _nat()
    B, D, S = 3, 29, 256
    c, lb, _ = _problem("gauss256", B, D, 13, 12.0)
    buf = torch.zeros(B * D * S + 1, dtype=torch.bfloat16, device="cuda")
    buf[1:] = lb.reshape(-1)
    view = buf[1:].view(B, D, S)
    assert view.is_contiguous() and view.data_ptr() % 16 != 0
    for kind, branch, crm in ((nat.LOSS_SDDM, "reverse_prob", 0), (nat.LOSS_CRM, "reverse_prob", 2), (nat.LOSS_CTELBO, None, 0)):
        leaf = buf.detach().clone().requires_grad_(True)
        a = _call(leaf[1:].view(B, D, S), kind, branch, crm, c)       # the view itself, misaligned, reaches ops.loss_terms
        sum(w * o.sum() for w, o in zip(SEED_W, a)).backward()
        b, gb = _fwd_bwd(lb, kind, branch, crm, c)                     # an aligned copy
        assert all(torch.equal(x.detach(), y) for x, y in zip(a, b)), kind
        assert leaf.grad.dtype == torch.bfloat16 and torch.equal(leaf.grad[1:].view(B, D, S), gb), kind
    # the raw call: SDDM reverse_prob at S = 256 with a scratch buffer is the tensor-core path
    L = nat.lib()
    outs = torch.zeros((5, B), device="cuda")
    ws = torch.empty(int(L.ctdd_loss_workspace_bytes(nat.LOSS_SDDM, B, S)), dtype=torch.uint8, device="cuda")
    scr = torch.empty(int(L.ctdd_loss_tc_scratch_bytes(B, D, S)), dtype=torch.uint8, device="cuda")
    grad = torch.empty(B * D * S + 8, dtype=torch.bfloat16, device="cuda")
    common = dict(kind=nat.LOSS_SDDM, logit_type=nat.BRANCH_SDDM_REVERSE_PROB, B=B, D=D, S=S, Q=c["Q"].data_ptr(),
                  QT=c["QT"].data_ptr(), Rb=c["Rb"].data_ptr(), beta=c["beta"].data_ptr(), x0=c["x0"].data_ptr(),
                  xt=c["xtil"].data_ptr(), eps=1e-9, out_a=outs[0].data_ptr(), out_b=outs[1].data_ptr(),
                  out_c=outs[2].data_ptr(), out_d=outs[3].data_ptr(), out_nll=outs[4].data_ptr(), ga=outs[0].data_ptr(),
                  gb=outs[0].data_ptr(), gd=outs[0].data_ptr(), gn=outs[0].data_ptr(), workspace=ws.data_ptr(),
                  tc_scratch=scr.data_ptr(), logits_dtype=nat.DTYPE_BF16)
    stream = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    n0 = nat.launch_count()
    p = nat.LossParams(logits=view.data_ptr(), grad_logits=grad.data_ptr(), **common)
    assert L.ctdd_loss_forward(ctypes.byref(p), stream) == 2 and b"aligned" in L.ctdd_last_error()
    assert L.ctdd_loss_backward(ctypes.byref(p), stream) == 2
    p = nat.LossParams(logits=lb.data_ptr(), grad_logits=grad[1:].data_ptr(), **common)
    assert L.ctdd_loss_backward(ctypes.byref(p), stream) == 2 and b"aligned" in L.ctdd_last_error()
    assert nat.launch_count() == n0
    torch.cuda.synchronize()


@gpu
def test_fp16_logits_keep_the_widening_copy():
    """fp16 (not served natively) is still widened to an fp32 copy: the outputs of the fp32 call, and a gradient that
    autograd casts back to fp16."""
    nat = _nat()
    c, lb, _ = _problem("gauss32", 3, 8, 21, 3.0)
    lh = lb.half()
    a, ga = _fwd_bwd(lh, nat.LOSS_SDDM, "reverse_prob", 0, c)
    b, gb = _fwd_bwd(lh.float(), nat.LOSS_SDDM, "reverse_prob", 0, c)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert ga.dtype == torch.float16 and torch.equal(ga, gb.half())


# ------------------------------------------------------------------------------------------------------- CPU
def test_unknown_logits_dtype_is_refused_before_any_cuda_call():
    """The ABI check needs no device: dummy non-null pointers, an unknown logits_dtype -> status 2 and a message naming
    the field, from the forward and the backward call."""
    nat = _nat()
    L = nat.lib()
    dummy = 0x1000
    ptrs = {k: dummy for k in ("logits", "Q", "QT", "Rb", "beta", "x0", "xt", "x_tilde", "out_a", "out_b", "out_c", "out_d",
                               "out_nll", "ga", "gb", "gd", "gn", "grad_logits", "workspace")}
    p = nat.LossParams(kind=nat.LOSS_CTELBO, B=2, D=3, S=4, eps=1e-9, logits_dtype=7, **ptrs)
    for fn in (L.ctdd_loss_forward, L.ctdd_loss_backward):
        assert fn(ctypes.byref(p), None) == 2
        assert b"logits_dtype" in L.ctdd_last_error()
    assert nat.LossParams.logits_dtype.offset > nat.LossParams.tc_scratch.offset
