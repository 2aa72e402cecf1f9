"""Every kernel family of libctdd_b200.so once at its configuration size (SURVEY §8d): CUDA-event time, algorithmic
bytes / FLOP and the resulting GB/s / TFLOP/s, one JSON line per kernel.  Not part of the product.

    python tools/kernel_zoo.py                      # timings (3 warm-ups, mean of 10)
    ZOO_NCU=1 ncu --set full --clock-control none -k regex:'<names>' python tools/kernel_zoo.py    # one launch each
"""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from ctdd_b200 import _native as nat, make_config, ops  # noqa: E402
from ctdd_b200.lib.models import forward_model as fm  # noqa: E402

NCU = bool(os.environ.get("ZOO_NCU"))
dev = torch.device("cuda")
PEAK_HBM, PEAK_FMA = 6529.0, 148 * 128 * 2 * 1.965e-3      # GB/s measured (MEASURED_PEAKS.json), TFLOP/s fp32 FMA nominal
try:
    PEAK_HBM = float(json.load(open(os.path.join(os.path.dirname(bench.__file__), "MEASURED_PEAKS.json")))["hbm_gbs"])
except Exception:
    pass


def timed(fn, reps=10, warm=3):
    if NCU:
        fn()
        torch.cuda.synchronize()
        return float("nan")
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def report(name, what, ms, bytes_=None, flop=None, note="", peak=None):
    rec = {"kernel": name, "workload": what, "ms": round(ms, 5)}
    if peak is not None:
        rec["peak_fwd_bwd_MB"] = round(peak / 2 ** 20, 1)
    if bytes_ is not None:
        rec["alg_bytes"] = int(bytes_)
        rec["GB/s"] = round(bytes_ / ms / 1e6, 1)
        rec["frac_hbm_peak"] = round(bytes_ / ms / 1e6 / PEAK_HBM, 3)
    if flop is not None:
        rec["alg_flop"] = int(flop)
        rec["TFLOP/s"] = round(flop / ms / 1e9, 2)
    if note:
        rec["note"] = note
    print(json.dumps(rec), flush=True)


def model_for(wname):
    w = bench.WORKLOADS[wname]
    cfg = make_config(data=dict(S=w["S"]), model=dict(w["model"], Q_sigma=w["model"].get("Q_sigma", 20.0)), device="cuda")
    return w, getattr(fm, bench.MIXIN[w["fwd"]])(cfg, "cuda")


def steps():
    # C1 / C2 also at 16 x the configuration's batch (VERDICT r1 #10: the HBM-rate claim of the small-S kernels is made there;
    # at the configurations' own batch the inputs fit in L2 and back-to-back Python calls time the host).  The C4 Euler line
    # times the Euler kernel at the C4 shape: no configuration samples with Euler at S = 256.  Every line has a bf16 twin
    # (the logits a network run under torch.autocast(dtype=torch.bfloat16) emits), and the C4 tau-leap step is also timed
    # through the route bf16 logits took before the kernels read them: a .float() copy, then the fp32 step.
    for wname, t, mult, mname in (("C1", 0.5, 1, None), ("C1", 0.5, 16, None), ("C2", 0.1, 1, None), ("C2", 0.1, 16, None),
                                  ("C3", 0.5, 1, None), ("C4", 0.5, 1, None), ("C4", 0.5, 1, "euler")):
        w, model = model_for(wname)
        mname = mname or w["mode"]
        S, D, B = w["S"], w["D"], w["B"] * mult
        Q, QT, beta = model.qt0_tables([t], dev)
        Rb, RbT = model.base_rate_tables(dev)
        branch = nat.branch_for(w["loss"], None)
        mode = nat.MODE_EULER if mname == "euler" else nat.MODE_TAU_LEAP
        tc = ops.prep_tc_tables(Q, QT, Rb, 1e-9, branch) if S == 256 else None
        tcs = ops.prep_tc_static(Rb) if tc is not None else None
        lg, x0 = bench.synth_logits(B, D, S, 7, dev, None)
        x = x0.to(torch.int32)
        ws = torch.empty((max(1, int(nat.lib().ctdd_step_workspace_bytes(B * D, S, 0))),), dtype=torch.uint8, device=dev)
        h = (w["max_t"] - w["min_t"]) / w["num_steps"]

        def run(logits):
            ops.reverse_step(mode, branch, logits, x, Q[0], QT[0], Rb, RbT, beta[0], h, 1e-9, N=B, D=D, S=S,
                             reject_multi=not w["ordinal"], seed=1, offset=0, tc_tables=(tc[0] if tc is not None else None),
                             tc_static=tcs, workspace=ws)
        name = f"step_small_kernel<{S}>" if S != 256 else ("step_tc_kernel" if mname == "euler" else "step_q_kernel")
        what = f"{wname}: S={S} D={D} N={B} {mname} t={t}"
        report(name, what, timed(lambda: run(lg)), bytes_=4.0 * B * D * S + 8.0 * B * D,
               flop=2.0 * B * D * S * S if S == 256 else None)
        lgb = lg.to(torch.bfloat16)
        del lg
        report(name, what + " bf16 logits", timed(lambda: run(lgb)), bytes_=2.0 * B * D * S + 8.0 * B * D,
               flop=2.0 * B * D * S * S if S == 256 else None)
        if wname == "C4" and mname == "tau_leap":
            report("widening copy + " + name, what + " bf16 logits through .float() and the fp32 step", timed(lambda: run(lgb.float())),
                   bytes_=2.0 * B * D * S + 8.0 * B * D, note="the copy reads 2 and writes 4 bytes per logit on top of the step")
        del lgb
    # C4 with the truncated-logistic head fused into the step (the CIFAR10 configuration's head): the (mu, log_scale) pair
    # as the two torch.chunk halves of a (B, 2D) network output, fp32, bf16 (a U-Net under torch.autocast), and bf16
    # through the former per-step widening (.float() of the (B, 2D) output, then the fp32 head step)
    w, model = model_for("C4")
    S, D, B = w["S"], w["D"], w["B"]
    Q, QT, beta = model.qt0_tables([0.5], dev)
    Rb, RbT = model.base_rate_tables(dev)
    branch = nat.branch_for(w["loss"], None)
    tc = ops.prep_tc_tables(Q, QT, Rb, 1e-9, branch)
    tcs = ops.prep_tc_static(Rb)
    gen = torch.Generator(device=dev).manual_seed(5)
    out32 = torch.cat([torch.tanh(torch.randn((B, D), generator=gen, device=dev)),
                       0.5 * torch.randn((B, D), generator=gen, device=dev) - 1.0], 1)
    out16 = out32.to(torch.bfloat16)
    x = torch.randint(0, S, (B, D), generator=gen, device=dev, dtype=torch.int32)
    h = (w["max_t"] - w["min_t"]) / w["num_steps"]
    for mname, mode, kname in (("tau_leap", nat.MODE_TAU_LEAP, "step_q_kernel<HEAD>"), ("euler", nat.MODE_EULER, "step_tc_kernel<HEAD>")):
        def run_head(out, widen=False):
            mu_v, ls_v = torch.chunk(out.float() if widen else out, 2, dim=1)
            ops.reverse_step(mode, branch, None, x, Q[0], QT[0], Rb, RbT, beta[0], h, 1e-9, N=B, D=D, S=S, seed=1, offset=0,
                             tc_tables=tc[0], tc_static=tcs, head=(mu_v, ls_v, False))
        what = f"C4: S={S} D={D} N={B} {mname} t=0.5, fused head"
        report(kname, what, timed(lambda: run_head(out32)), bytes_=8.0 * B * D + 8.0 * B * D, flop=2.0 * B * D * S * S)
        report(kname, what + " bf16 (mu, log_scale)", timed(lambda: run_head(out16)), bytes_=4.0 * B * D + 8.0 * B * D,
               flop=2.0 * B * D * S * S)
        report("widening copy + " + kname, what + " bf16 (mu, log_scale) through .float() and the fp32 step",
               timed(lambda: run_head(out16, True)), bytes_=4.0 * B * D + 8.0 * B * D,
               note="the copy reads 2 and writes 4 bytes per head parameter on top of the step")
    del out32, out16
    # CUDA-core block kernel at S = 256 (SDDM direct branch / cross-check path), and the exact-posterior branch sizes
    w, model = model_for("C3")
    S, D, B = 256, 784, 64
    Q, QT, beta = model.qt0_tables([0.5], dev)
    Rb, RbT = model.base_rate_tables(dev)
    lg, x0 = bench.synth_logits(B, D, S, 8, dev, None)
    x = x0.to(torch.int32)

    def run_block(logits):
        ops.reverse_step(nat.MODE_TAU_LEAP, nat.BRANCH_TAULDR, logits, x, Q[0], QT[0], Rb, RbT, beta[0], 1e-3, 1e-9, N=B, D=D, S=S,
                         seed=1, offset=0, impl=nat.IMPL_SIMT)
    for logits, esz, tag in ((lg, 4, ""), (lg.to(torch.bfloat16), 2, " bf16 logits")):
        report("step_block_kernel", f"S=256 D=784 N={B} tau_leap (CUDA-core path){tag}", timed(lambda: run_block(logits)),
               bytes_=esz * B * D * S + 8.0 * B * D, flop=2.0 * B * D * S * S)


def forward_process():
    w, model = model_for("C4")
    S, D = 256, 3072
    for B in (128, 1024):
        ts = torch.rand(B, device=dev) * 0.98 + 0.01

        def run_q():
            model._build_qt0(model._transition_delta(ts), inverse=True, want_transpose=True)
        report("qt0_fused_kernel", f"q_t|0 for B={B} distinct times, S=256 (Q and Q^T)", timed(run_q),
               bytes_=8.0 * B * S * S, flop=2.0 * B * S * S * S)
    B = 128
    ts = torch.rand(B, device=dev) * 0.98 + 0.01
    Q, QT = model._build_qt0(model._transition_delta(ts), inverse=True, want_transpose=True)
    beta = model._rate_scalar(ts).float().contiguous()
    Rb, _ = model.base_rate_tables(dev)
    x0 = torch.randint(0, S, (B, D), device=dev, dtype=torch.int32)
    report("noise_xt_kernel + xtilde_kernel", f"x_t ~ q_t|0(.|x0) and x~, B={B} D={D} S=256", timed(lambda: ops.noise_xt(Q, Rb, beta, x0, 1, 0)),
           bytes_=12.0 * B * D, note="row gathers of Q[b, x0, :] come from L2 (B * 256 KB of Q)")
    probs = torch.softmax(-((torch.arange(S, device=dev) - 128.0) / 40.0) ** 2, 0).contiguous()
    rows = 1024 * D
    report("categorical_shared_kernel", f"initial states, {rows} rows, S=256", timed(lambda: ops.sample_categorical_shared(probs, rows, 1)),
           bytes_=4.0 * rows)


def losses():
    # Each line has a bf16 twin (the logits a network run under torch.autocast(dtype=torch.bfloat16) emits, read as they
    # are, with a bf16 gradient) and a line for the route bf16 logits took before the kernels read them: a .float() copy
    # before ops.loss_terms, the fp32 gradient cast back to bf16 by autograd.  The three run alternately, and each reports
    # the peak device memory of one forward + backward over what was allocated before it.
    w, model = model_for("C4")
    S = 256
    Rb, _ = model.base_rate_tables(dev)
    for name, kind, B, D in (("C3 CatRMNLL", nat.LOSS_CRM, 64, 784), ("C5 SDDMElbo", nat.LOSS_SDDM, 64, 3072),
                             ("C5 CTElbo", nat.LOSS_CTELBO, 64, 3072)):
        ts = torch.rand(B, device=dev) * 0.98 + 0.01
        Q, QT = model._build_qt0(model._transition_delta(ts), inverse=True, want_transpose=True)
        beta = model._rate_scalar(ts).float().contiguous()
        x0 = torch.randint(0, S, (B, D), device=dev, dtype=torch.int32)
        xt, xtil = ops.noise_xt(Q, Rb, beta, x0, 1, 0)
        lf32 = (torch.randn(B, D, S, device=dev) - (torch.arange(S, device=dev).view(1, 1, S) - x0.unsqueeze(-1)) ** 2 / 128.0)
        lb16 = lf32.to(torch.bfloat16)

        def fwd(logits):
            return ops.loss_terms(logits, kind, Q=Q, QT=QT, Rb=Rb, beta=beta, x0=x0, xt=xtil if kind != nat.LOSS_CRM else xt,
                                  x_tilde=xtil if kind == nat.LOSS_CTELBO else None, eps=1e-9)

        def fwd_bwd(leaf, widen):
            sum(o.sum() for o in fwd(leaf.float() if widen else leaf)).backward()
            leaf.grad = None

        def peak(leaf, widen):
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            fwd_bwd(leaf, widen)
            torch.cuda.synchronize()
            return torch.cuda.max_memory_allocated() - base
        for tag, leaf, esz, widen in (("", lf32, 4, False), (" bf16 logits", lb16, 2, False),
                                      (" bf16 logits through .float()", lb16, 2, True)):
            leaf.requires_grad_(True)
            with torch.no_grad():
                ms_f = timed(lambda: fwd(leaf.float() if widen else leaf))
            ms_fb = timed(lambda: fwd_bwd(leaf, widen))
            note = "the copy reads 2 and writes 4 bytes per logit, the gradient cast reads 4 and writes 2" if widen else ""
            report(("widening copy + " if widen else "") + "loss_kernel<0>", f"{name} forward, B={B} D={D} S=256{tag}", ms_f,
                   bytes_=esz * B * D * S, flop=2.0 * B * D * S * S, note=note)
            report(("widening copy + " if widen else "") + "loss_kernel<0> + loss_kernel<1>",
                   f"{name} forward + backward (torch autograd glue included){tag}", ms_fb, bytes_=3.0 * esz * B * D * S,
                   flop=6.0 * B * D * S * S, note=note, peak=peak(leaf, widen))


def head():
    # fp32 head; bf16 (mu, log_scale) with bf16 logits and a bf16 incoming gradient (a U-Net under torch.autocast feeding
    # the bf16 loss path); and the former route for bf16 network output: .float() of mu / log_scale, then the fp32 head
    B, D, S = 128, 3072, 256
    mu32 = torch.tanh(torch.randn(B, D, device=dev))
    ls32 = torch.randn(B, D, device=dev)
    g32 = torch.randn(B, D, S, device=dev)
    for tag, dt, widen in (("", torch.float32, False), (" bf16 in / bf16 out / bf16 gradient", torch.bfloat16, False),
                           (" bf16 in through .float(), fp32 head", torch.bfloat16, True)):
        mu = mu32.to(dt).requires_grad_(True)
        ls = ls32.to(dt).requires_grad_(True)
        out_dt = torch.bfloat16 if (dt == torch.bfloat16 and not widen) else torch.float32
        esz = 2 if out_dt == torch.bfloat16 else 4
        g = g32.to(out_dt)

        def fwd():
            if widen:
                return ops.logistic_logits_autograd(mu.float(), ls.float(), S, False)
            return ops.logistic_logits_autograd(mu, ls, S, False, out_dtype=out_dt)
        with torch.no_grad():
            report("logistic_logits_kernel", f"head forward B={B} D={D} S=256{tag}", timed(fwd), bytes_=esz * B * D * S)

        def fb():
            out = fwd()
            out.backward(g.view_as(out))
            mu.grad = ls.grad = None
        report("logistic_logits_kernel + logistic_backward_kernel", f"head forward + backward B={B} D={D} S=256{tag}",
               timed(fb), bytes_=2.0 * esz * B * D * S)
    del g32, g
    # The image training leg: head + SDDMElbo loss terms (tensor-core path), forward + backward, from bf16 network output
    # (torch.autocast) against the cast-to-fp32 route (fp32 head, fp32 logits into the loss, fp32 gradient back)
    w, model = model_for("C5")
    Rb, _ = model.base_rate_tables(dev)
    for B in (64, 512):
        gen = torch.Generator(device=dev).manual_seed(B)
        Q, QT, beta = model.qt0_tables([0.05 + 0.9 * (i + 0.5) / B for i in range(B)], dev)
        beta = torch.tensor([float(b) for b in beta], dtype=torch.float32, device=dev)
        x0 = torch.randint(0, S, (B, D), generator=gen, device=dev, dtype=torch.int32)
        _, xtil = ops.noise_xt(Q, Rb, beta, x0, 3, 0)
        mu = torch.tanh(torch.randn(B, D, generator=gen, device=dev)).to(torch.bfloat16).requires_grad_(True)
        ls = (torch.randn(B, D, generator=gen, device=dev) - 1.0).to(torch.bfloat16).requires_grad_(True)

        def leg(widen):
            if widen:
                logits = ops.logistic_logits_autograd(mu.float(), ls.float(), S, False)
            else:
                logits = ops.logistic_logits_autograd(mu, ls, S, False, out_dtype=torch.bfloat16)
            outs = ops.loss_terms(logits, nat.LOSS_SDDM, Q, QT, Rb, beta, x0, xtil, eps=1e-9,
                                  logit_branch=nat.BRANCH_SDDM_REVERSE_PROB)
            (outs[0].sum() + outs[1].sum() + 0.01 * outs[4].sum()).backward()
            mu.grad = ls.grad = None

        def peak(widen):
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            leg(widen)
            torch.cuda.synchronize()
            return torch.cuda.max_memory_allocated() - base
        for tag, widen in ((" bf16 (mu, log_scale), bf16 logits", False), (" bf16 (mu, log_scale) through .float(), fp32 logits", True)):
            report("head + SDDM loss_terms", f"image training leg B={B} D={D} S=256 forward + backward{tag}",
                   timed(lambda: leg(widen)), note="torch autograd glue included", peak=peak(widen))
        del Q, QT, mu, ls


if __name__ == "__main__":
    which = sys.argv[1:] or ["steps", "forward_process", "losses", "head"]
    for k in which:
        globals()[k]()
