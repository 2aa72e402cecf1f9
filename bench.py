#!/usr/bin/env python
"""bench.py — reverse-CTMC hot-path benchmark (driver contract: see the task statement / DESIGN.md §Measurement).

A "step" is ONE reverse-rate evaluation fused with the tau-leaping state update (TauL predictor step,
reference lib/sampling/sampling.py:119-160) over the per-GPU batch of the named workload, on synthetic logits.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C4|C3|C2|C1] [--impl ours|reference] [--dump-outputs DIR]

Workloads (BASELINE.json configs / SURVEY.md §8d):
  C4  CIFAR10-shape  S=256 D=3072 B=1024/GPU GaussianTargetRate, TauL   <- default (the metric's config)
  C3  MNIST-shape    S=256 D=784  B=1024/GPU
  C2  maze           S=3   D=225  B=16384/GPU UniformVariantRate(log_sqr), Euler (LBJF) step
  C1  synthetic      S=2   D=32   B=65536/GPU UniformVariantRate(sqrt_cos), TauL non-ordinal
  C5  CIFAR10-shape  S=256 D=3072 MidPointTauL step (2 reverse-rate evaluations) + SDDMElbo calc_loss forward+backward on
      synthetic logits (1-parameter stub network); --total-batch B (64..4096) is sharded over the GPUs, --sweep runs them all

Metric: reverse-step TFLOP/s with algorithmic work 2*B*D*S^2 per step (for S<=8 workloads the line also carries
GB/s, which is what bounds them).  Weak scaling: every rank owns B rows; no data-path collective.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "C4": dict(S=256, D=3072, B=1024, fwd="gaussian", mode="tau_leap", ordinal=True, loss="CTElbo", num_steps=1000, cpu_N=8,
               model=dict(rate_sigma=6.0, Q_sigma=512.0, time_exp=100.0, time_base=3.0), max_t=1.0, min_t=0.01),
    "C3": dict(S=256, D=784, B=1024, fwd="gaussian", mode="tau_leap", ordinal=True, loss="CTElbo", num_steps=1000, cpu_N=32,
               model=dict(rate_sigma=6.0, Q_sigma=512.0, time_exp=100.0, time_base=3.0), max_t=1.0, min_t=0.01),
    "C2": dict(S=3, D=225, B=16384, fwd="uniform_variant", mode="euler", ordinal=True, loss="CTElbo", num_steps=500, cpu_N=1024,
               model=dict(rate_const=2.0, t_func="log_sqr"), max_t=1.0, min_t=0.001),
    "C5": dict(S=256, D=3072, B=512, fwd="gaussian", mode="midpoint", ordinal=True, loss="SDDMElbo", num_steps=1000, cpu_N=4,
               model=dict(rate_sigma=6.0, Q_sigma=512.0, time_exp=100.0, time_base=3.0), max_t=1.0, min_t=0.01),
    "C1": dict(S=2, D=32, B=65536, fwd="uniform_variant", mode="tau_leap", ordinal=False, loss="CTElbo", num_steps=500, cpu_N=4096,
               model=dict(rate_const=2.0, t_func="sqrt_cos"), max_t=0.99999, min_t=0.007),
}
MIXIN = {"gaussian": "GaussianTargetRate", "uniform_variant": "UniformVariantRate"}


def synth_logits(B, D, S, seed, device, x0=None):
    """Denoiser-like synthetic logits (SURVEY §8d family L2): -(s - x0)^2 / (2*8^2) + randn."""
    g = torch.Generator(device=device).manual_seed(seed)
    if x0 is None:
        x0 = torch.randint(0, S, (B, D), generator=g, device=device)
    s = torch.arange(S, device=device, dtype=torch.float32)
    out = torch.randn((B, D, S), generator=g, device=device)
    if S > 8:
        out -= (s.view(1, 1, S) - x0.unsqueeze(-1).float()) ** 2 / (2.0 * 8.0 ** 2)
    return out, x0


class ClockSampler:
    """Samples SM clock and throttle reasons of this rank's GPU DURING the timed region: NVML (the library behind
    nvidia-smi) polled every 2 ms from a thread; falls back to an `nvidia-smi -lms` subprocess when pynvml is missing."""

    NAMES = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.rows, self._stop = index, [], threading.Event()
        self.proc = self.nvml = self.t = None

    def _sample_nvml(self):
        nv, h = self.nvml
        try:
            sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            try:
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
            except Exception:
                rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            self.rows.append((float(sm), float(self.mx), int(rs)))
        except Exception:
            pass

    def _poll_nvml(self):
        while not self._stop.is_set():
            self._sample_nvml()
            time.sleep(0.002)

    def __enter__(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            # CUDA_VISIBLE_DEVICES may renumber devices: resolve through the PCI bus id torch reports
            try:
                bus = torch.cuda.get_device_properties(self.index).pci_bus_id
                dom = torch.cuda.get_device_properties(self.index).pci_domain_id
                dev = torch.cuda.get_device_properties(self.index).pci_device_id
                h = nv.nvmlDeviceGetHandleByPciBusId(f"{dom:08x}:{bus:02x}:{dev:02x}.0")
            except Exception:
                h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.nvml = (nv, h)
            self.mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)   # also pays NVML's first-call latency up front
            nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            self.t = threading.Thread(target=self._poll_nvml, daemon=True)
            self.t.start()
            return self
        except Exception:
            self.nvml = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        bits = {v: k for k, v in self.NAMES.items()}
        for line in self.proc.stdout:
            c = [x.strip() for x in line.split(",")]
            try:
                rs = sum(bits[n] for n, v in zip(names, c[3:7]) if v.lower().startswith("active"))
                self.rows.append((float(c[0]), float(c[1]), rs))
            except Exception:
                continue

    def __exit__(self, *a):
        self._stop.set()
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        elif self.t is not None:
            self.t.join(timeout=1)
            if not self.rows:      # a timed region shorter than the thread's start-up: one sample at its end
                self._sample_nvml()

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = [r[0] for r in self.rows]
        reasons = sorted({n for r in self.rows for bit, n in self.NAMES.items() if r[2] & bit})
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(r[1] for r in self.rows)), "reasons": reasons,
                "samples": len(sm), "source": "nvml" if self.nvml else "nvidia-smi"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tc_burst=d["bf16_tflops"], tc_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tc_burst=1590.0, tc_sustained=1400.0, src="fallback")


# ---------------------------------------------------------------------------------------------------------------
# CPU baseline.  Preferred: the UNMODIFIED reference (its get_reverse_rates with the six N*D*S index tensors, its rate
# mixins) staged under baseline/_ref/ by tools/stage_reference.py - kind "reference".  Fallback when that copy is absent:
# the oracle port (a torch-CPU restatement that gathers with a broadcast index and never builds those index tensors,
# i.e. it is FASTER than the reference: the ratio against it is conservative) - kind "port".

def _reference_modules():
    try:
        from oracle import ref_harness as rh
        if not rh.reference_available():
            return None, None
        return rh, rh.import_reference()
    except Exception as e:      # missing dependency of the reference on this box
        sys.stderr.write(f"reference arm: cannot import the staged reference ({e}); using the oracle port\n")
        return None, None


def cpu_reference_step_time(w, n_cpu, steps, warmup):
    """Seconds per reverse step (get_reverse_rates + Poisson / Euler update as TauL.sample / LBJF.sample compose them,
    lib/sampling/sampling.py:119-160, :278-293) on all host cores, N = n_cpu samples.  Returns (seconds, kind)."""
    import torch.nn as nn
    torch.set_num_threads(os.cpu_count() or 1)
    S, D = w["S"], w["D"]
    logits, x0 = synth_logits(n_cpu, D, S, 1234, "cpu")
    x = x0.clone()
    ts = np.linspace(w["max_t"], w["min_t"], steps + warmup)
    h = (w["max_t"] - w["min_t"]) / w["num_steps"]
    rh, ref = _reference_modules()
    if ref is not None:
        mcfg = dict(w["model"], concat_dim=D)
        mcfg.setdefault("Q_sigma", 20.0)
        cfg = rh.make_cfg(data=dict(S=S, shape=[D], name="DiscreteCIFAR10"), model=mcfg, training=dict(max_t=w["max_t"]),
                          sampler=dict(eps_ratio=1e-9), loss=dict(name=w["loss"], logit_type="reverse_prob", eps_ratio=1e-9),
                          device="cpu")
        mixin = getattr(ref.fm, MIXIN[w["fwd"]])

        class RefModel(nn.Module, mixin):
            def __init__(self):
                nn.Module.__init__(self)
                mixin.__init__(self, cfg, "cpu")

        model = RefModel()
        model.device = "cpu"
        rates = lambda t_ones, xx: ref.ss.get_reverse_rates(model, logits, xx, t_ones, cfg, n_cpu, D, S)[0]
        kind = "reference"
    else:
        from oracle import ctmc_oracle as oc
        fp = oc.ForwardProcess(w["fwd"], S, **w["model"])
        rates = lambda t_ones, xx: oc.reverse_rates(logits, xx, fp.transition(t_ones), fp.rate(t_ones), w["loss"],
                                                    "reverse_prob", 1e-9)[0]
        kind = "port"
    times = []
    with torch.no_grad():
        for i, t in enumerate(ts):
            t0 = time.perf_counter()
            t_ones = float(t) * torch.ones((n_cpu,))
            rr = rates(t_ones, x)
            oh = torch.nn.functional.one_hot(x.long(), S)
            rz = rr * (1 - oh)                                     # sampling.py:127-128
            if w["mode"] == "euler":                               # sampling.py:278-293
                tot = rz.sum(-1, keepdim=True)
                P = rz * h + torch.clip(1.0 - h * tot, min=0) * oh
                P = P / P.sum(-1, keepdim=True)
                x = torch.distributions.categorical.Categorical(logits=torch.log(P + 1e-35).view(-1, S)).sample().view(n_cpu, D)
            else:                                                  # sampling.py:129-160
                k = torch.poisson(rz * h)
                if not w["ordinal"]:
                    k = k * (k.sum(-1, keepdim=True) <= 1)
                diff = torch.arange(S).view(1, 1, S) - x.unsqueeze(-1)
                x = torch.clamp(x + (k * diff).sum(-1), 0, S - 1).long()
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    return float(np.mean(times)), kind


def flops_per_step(B, D, S):
    return 2.0 * B * D * S * S


DUMP_BYTES = 64 << 20


def dump_outputs(d, arrays):
    """Write the arrays of the last timed step as d/<name>.npy: integer states as float32 (exact below 2^24), int64
    counters as float64, 64 MB at most in all.  Arrays are taken smallest first, each whole when it fits an equal share of
    what is left, else as a fixed, seeded sample of its flat elements of that size."""
    os.makedirs(d, exist_ok=True)
    out = {k: v.detach().cpu().numpy().astype(np.float64 if v.dtype in (torch.int64, torch.float64) else np.float32)
           for k, v in arrays.items()}
    left = DUMP_BYTES
    for i, (k, a) in enumerate(sorted(out.items(), key=lambda kv: kv[1].nbytes)):
        share = left // (len(out) - i)
        if a.nbytes > share:
            keep = max(1, share // a.itemsize)
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        left -= a.nbytes
        np.save(os.path.join(d, k + ".npy"), a)


def run_reference(args, w, rank, world):
    if rank != 0:
        return
    if args.workload == "C5":
        return run_reference_c5(args, w)
    n_cpu = w["cpu_N"]
    t, kind = cpu_reference_step_time(w, n_cpu, args.steps, args.warmup)
    val = flops_per_step(n_cpu, w["D"], w["S"]) / t / 1e12
    what = ("the reference's own get_reverse_rates + rate mixins (unmodified files staged under baseline/_ref/), update lines of "
            "TauL.sample / LBJF.sample" if kind == "reference" else
            "oracle port of the reference's get_reverse_rates + update (no staged reference on this box; the port skips the "
            "reference's six N*D*S index tensors, so it is the faster of the two)")
    line = {
        "impl": "reference", "metric": "reverse_step_tflops", "value": val, "unit": "TFLOP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: S={w['S']} D={w['D']} {w['mode']} step, CPU sample N={n_cpu} rows of the B={w['B']} batch"},
        "cpu_baseline": {"value": val, "unit": "TFLOP/s", "cores": os.cpu_count(), "kind": kind,
                         "sample": f"N={n_cpu} samples x D={w['D']} per step, {args.steps} steps: {what}",
                         "sample_steps_per_s": n_cpu / t},
        "e2e": {"value": val, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------
def run_ours(args, w, rank, world, local_rank):
    import torch.distributed as dist
    from ctdd_b200 import _native as nat, make_config, ops
    from ctdd_b200.lib.models import forward_model as fm

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    S, D, B = w["S"], w["D"], w["B"]
    if args.batch:
        B = args.batch          # diagnostic: other batch sizes of the same workload (the bench line names the B it ran)
    K, W = args.steps, args.warmup
    cfg = make_config(data=dict(S=S), model=dict(w["model"], Q_sigma=w["model"].get("Q_sigma", 20.0)), device=str(dev))
    model = getattr(fm, MIXIN[w["fwd"]])(cfg, str(dev))
    nsteps = K + W
    ts = np.linspace(w["max_t"], w["min_t"], nsteps)       # timed steps are spread over the whole schedule
    h = (w["max_t"] - w["min_t"]) / w["num_steps"]
    Q, QT, beta = model.qt0_tables(list(ts), dev)
    Rb, RbT = model.base_rate_tables(dev)
    branch = nat.branch_for(w["loss"], None)
    mode = nat.MODE_EULER if w["mode"] == "euler" else nat.MODE_TAU_LEAP
    impl = {"auto": nat.IMPL_AUTO, "simt": nat.IMPL_SIMT, "tc": nat.IMPL_TC}[args.kernels]
    tc = ops.prep_tc_tables(Q, QT, Rb, 1e-9, branch) if (S == 256 and impl != nat.IMPL_SIMT) else None
    tcs = ops.prep_tc_static(Rb) if tc is not None else None
    ws_bytes = int(nat.lib().ctdd_step_workspace_bytes(B * D, S, impl))
    workspace = torch.empty((max(ws_bytes, 1),), dtype=torch.uint8, device=dev)
    # two logits buffers (each >> L2 at the S=256 workloads) alternate between steps
    nbuf = 2
    bufs = []
    x0 = None
    for i in range(nbuf):
        lg, x0 = synth_logits(B, D, S, 1234 + 17 * rank + i, dev, None)
        bufs.append(lg)
    x = torch.clamp(x0 + torch.randint(-3, 4, x0.shape, device=dev), 0, S - 1).to(torch.int32)
    row_offset = rank * B * D          # B is a multiple of 8, so every rank's first global row is 8-aligned
    stats = torch.zeros((nsteps, 8), dtype=torch.int64, device=dev)
    # L2 flush for inputs smaller than L2; 1 GB so that the fill also outlasts the host's launch path (else the event
    # pair around a 10-microsecond kernel times the Python call, not the kernel)
    flush = torch.empty((1 << 30,), dtype=torch.uint8, device=dev) if B * D * S * 4 < (512 << 20) else None

    def step(i, xin, logits):
        return ops.reverse_step(mode, branch, logits, xin, Q[i], QT[i], Rb, RbT, beta[i], h, 1e-9, N=B, D=D, S=S,
                                reject_multi=not w["ordinal"], seed=0xC7DD, offset=i, row_offset=row_offset, impl=impl,
                                tc_tables=(tc[i] if tc is not None else None), tc_static=tcs, workspace=workspace,
                                stats=stats[i])["x"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for i in range(W):
        x = step(i, x, bufs[i % nbuf])
    barrier()
    launches0 = nat.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        t_start.record()
        for j in range(K):
            if flush is not None:
                flush.fill_(j & 0xFF)          # L2 flush between timed iterations for inputs smaller than L2
            ev[j][0].record()
            x = step(W + j, x, bufs[(W + j) % nbuf])
            ev[j][1].record()
        t_end.record()
        barrier()
    launches = nat.launch_count() - launches0
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))   # step kernels only (flush excluded)
    total_ms = t_start.elapsed_time(t_end)
    ms_per_step = kern_ms if flush is not None else total_ms / K
    t_ms = torch.tensor([ms_per_step], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms = float(t_ms.item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"x": x, "stats": stats[W + K - 1]})

    # ---- end to end through the C ABI with HOST buffers: H2D logits + state, step, D2H new state, every step ----
    e2e_steps = max(1, min(K, args.e2e_steps))
    chunk = max(8, min(B, (192 << 20) // (D * S * 4)) // 8 * 8)   # ~192 MB logits per chunk (multiple of 8 rows), double-buffered
    nchunks = (B + chunk - 1) // chunk
    host_logits = torch.empty((B, D, S), dtype=torch.float32, pin_memory=True)
    host_logits.copy_(bufs[0])
    host_x = torch.empty((B, D), dtype=torch.int32, pin_memory=True)
    host_x.copy_(x)
    host_out = torch.empty((B, D), dtype=torch.int32, pin_memory=True)
    dl = [torch.empty((chunk, D, S), dtype=torch.float32, device=dev) for _ in range(2)]
    dx = [torch.empty((chunk, D), dtype=torch.int32, device=dev) for _ in range(2)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(2)]
    cws = [torch.empty((max(int(nat.lib().ctdd_step_workspace_bytes(chunk * D, S, impl)), 1),), dtype=torch.uint8, device=dev)
           for _ in range(2)]

    def e2e_step(i):
        for c in range(nchunks):
            lo, hi = c * chunk, min(B, (c + 1) * chunk)
            n = hi - lo
            s = streams[c & 1]
            with torch.cuda.stream(s):
                dl[c & 1][:n].copy_(host_logits[lo:hi], non_blocking=True)
                dx[c & 1][:n].copy_(host_x[lo:hi], non_blocking=True)
                ro = row_offset + lo * D
                out = ops.reverse_step(mode, branch, dl[c & 1][:n], dx[c & 1][:n], Q[i], QT[i], Rb, RbT, beta[i], h, 1e-9,
                                       N=n, D=D, S=S, reject_multi=not w["ordinal"], seed=0xC7DD, offset=i,
                                       row_offset=ro, impl=impl, tc_tables=(tc[i] if tc is not None else None),
                                       tc_static=tcs, workspace=cws[c & 1])["x"]
                host_out[lo:hi].copy_(out, non_blocking=True)
        for s in streams:
            s.synchronize()

    e2e_step(0)
    barrier()
    t0 = time.perf_counter()
    for j in range(e2e_steps):
        e2e_step(W + j)
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    t_e = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_ms = float(t_e.item())

    # ---- the same step with the network's truncated-logistic head fused in (SURVEY §8f rank 1; the CIFAR10 config's own
    # head, config_tauUnet_cifar10.py:59): inputs are the (mu, log_scale) pair per dimension, the logits never exist
    fused = None
    if tc is not None and w["mode"] == "tau_leap":
        g = torch.Generator(device=dev).manual_seed(99 + rank)
        noise = torch.randn((B, 2 * D), device=dev, generator=g)
        heads = []
        for i in range(nsteps):    # denoiser-like: mean near the clean value, scale growing with the noise level
            mu = torch.tanh((x0.float() + 0.5) / (S / 2.0) - 1.0 + 0.05 * noise[:, :D])
            ls = (-1.5 + 2.5 * float(ts[i])) + 0.3 * noise[:, D:]
            heads.append(torch.cat([mu, ls], 1))
        xh = torch.clamp(x0 + torch.randint(-3, 4, x0.shape, device=dev, generator=g), 0, S - 1).to(torch.int32)

        def head_step(i, xin):
            mu_v, ls_v = torch.chunk(heads[i], 2, dim=1)
            return ops.reverse_step(mode, branch, None, xin, Q[i], QT[i], Rb, RbT, beta[i], h, 1e-9, N=B, D=D, S=S,
                                    reject_multi=not w["ordinal"], seed=0xC7DD, offset=i, row_offset=row_offset, impl=impl,
                                    tc_tables=tc[i], tc_static=tcs, workspace=workspace, head=(mu_v, ls_v, False))["x"]

        for i in range(W):
            xh = head_step(i, xh)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for j in range(K):
            xh = head_step(W + j, xh)
        f1.record()
        barrier()
        fused_ms = f0.elapsed_time(f1) / K
        mu_v, ls_v = torch.chunk(heads[W], 2, dim=1)
        ops.logistic_logits(mu_v, ls_v, S, False, out=bufs[0])
        f0.record()
        for _ in range(3):
            ops.logistic_logits(mu_v, ls_v, S, False, out=bufs[0])
        f1.record()
        torch.cuda.synchronize(dev)
        head_ms = f0.elapsed_time(f1) / 3
        # end to end from HOST buffers: 2 floats + 1 state per dimension in, 1 state out, EVERY step.  Three streams and two
        # buffer sets: the H2D copy of step j + 1, the kernel of step j and the D2H read-back of step j - 1 overlap, so a
        # step costs the slowest of the three instead of their sum (and the host link is shared more evenly when 8 ranks
        # feed their GPUs at once).
        host_head = torch.empty((B, 2 * D), dtype=torch.float32, pin_memory=True)
        host_head.copy_(heads[W])
        NBUF = 2
        dev_head = [torch.empty((B, 2 * D), dtype=torch.float32, device=dev) for _ in range(NBUF)]
        dev_x = [torch.empty((B, D), dtype=torch.int32, device=dev) for _ in range(NBUF)]
        host_outs = [torch.empty((B, D), dtype=torch.int32, pin_memory=True) for _ in range(NBUF)]
        s_in, s_run, s_out = (torch.cuda.Stream(device=dev) for _ in range(3))
        ev_in = [torch.cuda.Event() for _ in range(NBUF)]
        ev_run = [torch.cuda.Event() for _ in range(NBUF)]
        hws = [torch.empty((max(ws_bytes, 1),), dtype=torch.uint8, device=dev) for _ in range(NBUF)]
        dev_out = [torch.empty((B, D), dtype=torch.int32, device=dev) for _ in range(NBUF)]
        ev_out = [torch.cuda.Event() for _ in range(NBUF)]

        def head_e2e(i, k):
            with torch.cuda.stream(s_in):
                s_in.wait_event(ev_run[k])                 # the kernel that last read this buffer set has finished
                dev_head[k].copy_(host_head, non_blocking=True)
                dev_x[k].copy_(host_x, non_blocking=True)
                ev_in[k].record(s_in)
            with torch.cuda.stream(s_run):
                s_run.wait_event(ev_in[k])
                s_run.wait_event(ev_out[k])                # the read-back that last used this output buffer has finished
                mu_h, ls_h = torch.chunk(dev_head[k], 2, dim=1)
                out = ops.reverse_step(mode, branch, None, dev_x[k], Q[i], QT[i], Rb, RbT, beta[i], h, 1e-9, N=B, D=D, S=S,
                                       reject_multi=not w["ordinal"], seed=0xC7DD, offset=i, row_offset=row_offset, impl=impl,
                                       tc_tables=tc[i], tc_static=tcs, workspace=hws[k], head=(mu_h, ls_h, False),
                                       x_out=dev_out[k])["x"]
                ev_run[k].record(s_run)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_run[k])
                host_outs[k].copy_(out, non_blocking=True)
                ev_out[k].record(s_out)

        def drain():
            for st_ in (s_in, s_run, s_out):
                st_.synchronize()

        for j in range(2):
            head_e2e(j, j % NBUF)
        drain()
        barrier()
        t0 = time.perf_counter()
        for j in range(K):
            head_e2e(W + j, j % NBUF)
        drain()
        barrier()
        fe_ms = (time.perf_counter() - t0) * 1e3 / K
        t_f = torch.tensor([fused_ms, fe_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_f, op=dist.ReduceOp.MAX)
        fused_ms, fe_ms = float(t_f[0].item()), float(t_f[1].item())
        fl_ = flops_per_step(B, D, S)
        fused = {"what": "same step, truncated-logistic head (mu, log_scale per dimension) evaluated inside the kernel; "
                         "no (B,D,S) logits tensor", "ms_per_step": fused_ms, "tflops": world * fl_ / (fused_ms * 1e-3) / 1e12,
                 "standalone_head_kernel_ms": head_ms,
                 "e2e": {"ms_per_step": fe_ms, "tflops": world * fl_ / (fe_ms * 1e-3) / 1e12,
                         "h2d_bytes_per_step": int(B * 2 * D * 4 + B * D * 4), "d2h_bytes_per_step": int(B * D * 4),
                         "note": "C-ABI step fed from pinned HOST head parameters + state every step, new state read back every "
                                 "step; H2D / kernel / D2H of consecutive steps overlap on three streams"}}
        del heads, noise

    # ---- the sampler CLASS end to end (the reference-facing API): TauL.sample(model, B) with a stub network that returns
    # resident logits (network cost excluded on both sides, SURVEY §8d); includes q_{t|0} / table builds for the schedule,
    # the initial samples, one kernel launch per step, the statistics read-back and the final .cpu() of the samples
    loop = None
    if w["mode"] == "tau_leap":
        import torch.nn as nn
        from ctdd_b200.lib.sampling import sampling_utils
        import ctdd_b200.lib.sampling.sampling  # noqa: F401
        loop_steps = w["num_steps"]     # the whole schedule: the step length h decides the jump rates, a short schedule is not representative
        mcfg = dict(w["model"], concat_dim=D)
        mcfg.setdefault("Q_sigma", 20.0)
        scfg = make_config(data=dict(S=S, shape=[D], name="DiscreteCIFAR10"), model=mcfg, training=dict(max_t=w["max_t"]),
                           sampler=dict(name="TauL", num_steps=loop_steps, min_t=w["min_t"], eps_ratio=1e-9,
                                        initial_dist="gaussian" if S > 8 else "uniform", num_corrector_steps=0,
                                        corrector_step_size_multiplier=1.5, corrector_entry_time=0.0, is_ordinal=w["ordinal"]),
                           loss=dict(name="CTElboLambda", eps_ratio=1e-9, logit_type="reverse_prob"), device=str(dev))
        mixin = getattr(fm, MIXIN[w["fwd"]])

        class Stub(nn.Module, mixin):
            """Denoiser-like stand-in for the score network: logits[n,d,s] = -(s - x[n,d])^2 / (2 * 8^2), written in place
            into one resident buffer (three elementwise torch kernels; timed separately as `stub_network_ms`).  The logits
            must follow the state: with logits that ignore x the reverse rates explode and the run measures nothing real."""

            def __init__(self):
                nn.Module.__init__(self)
                mixin.__init__(self, scfg, str(dev))
                self.out = bufs[0]
                self.s_row = torch.arange(S, device=dev, dtype=torch.float32).view(1, 1, S)

            def forward(self, x, t):
                torch.sub(self.s_row, x.unsqueeze(-1).to(torch.float32), out=self.out)
                self.out.square_().mul_(-1.0 / 128.0)
                return self.out

        stub = Stub()
        stub.device = str(dev)
        sampler = sampling_utils.get_sampler(scfg)
        sampler.seed, sampler.row_offset, sampler.impl = 0xC7DD, row_offset, impl
        barrier()
        t0 = time.perf_counter()
        if world > 1:      # the sampler's only collective - the final all-gather of the samples - is inside the timing
            from ctdd_b200.dist import sample_sharded
            res = sample_sharded(sampler, stub, world * B)
            xs = np.asarray(res[0])[rank * B:(rank + 1) * B]
        else:
            xs, _ = sampler.sample(stub, B)
        barrier()
        loop_ms = (time.perf_counter() - t0) * 1e3 / loop_steps
        # what the schedule's tables cost (q_{t|0} for 1000 time points + the tensor-path tables), amortised per step
        torch.cuda.synchronize(dev)
        t1 = time.perf_counter()
        tq, tqt, tbeta = stub.qt0_tables(list(np.linspace(w["max_t"], w["min_t"], loop_steps)), dev)
        ttc = ops.prep_tc_tables(tq, tqt, Rb, 1e-9, branch) if S == 256 else None
        torch.cuda.synchronize(dev)
        tables_ms = (time.perf_counter() - t1) * 1e3 / loop_steps
        # the step kernel alone over THIS schedule (40 time points spread over all of it, stub logits of the final states):
        # the bench's own K steps skip the first W / (K + W) of the schedule, where a step costs up to 3x the average
        xs_d = torch.from_numpy(np.asarray(xs)).to(dev).to(torch.int32)
        lg_s = stub(xs_d, None)
        sched_ms = []
        hs = (w["max_t"] - w["min_t"]) / loop_steps
        for i in np.linspace(0, loop_steps - 1, 40).astype(int):
            ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ea.record()
            ops.reverse_step(mode, branch, lg_s, xs_d, tq[i], tqt[i], Rb, RbT, tbeta[i], hs, 1e-9, N=B, D=D, S=S,
                             reject_multi=not w["ordinal"], seed=0xC7DD, offset=int(i), row_offset=row_offset, impl=impl,
                             tc_tables=(ttc[i] if ttc is not None else None), tc_static=tcs, workspace=workspace)
            eb.record()
            torch.cuda.synchronize(dev)
            sched_ms.append(ea.elapsed_time(eb))
        sched_kernel_ms = float(np.mean(sched_ms))
        del tq, tqt, ttc
        t_l = torch.tensor([loop_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_l, op=dist.ReduceOp.MAX)
        loop_ms = float(t_l.item())
        # the stub network alone, same call pattern
        xs_dev = torch.from_numpy(np.asarray(xs)).to(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stub(xs_dev, None)
        e0.record()
        for _ in range(4):
            stub(xs_dev, None)
        e1.record()
        torch.cuda.synchronize(dev)
        stub_ms = e0.elapsed_time(e1) / 4
        loop = {"api": "TauL.sample(model, B), whole schedule, stub network whose logits follow the state; includes the "
                       "q_{t|0} / table build for every time point and the final read-back", "steps": loop_steps,
                "ms_per_step": loop_ms, "stub_network_ms": stub_ms, "table_build_ms_per_step": tables_ms,
                "sampler_ms_per_step": loop_ms - stub_ms,
                "step_kernel_ms_over_this_schedule": sched_kernel_ms,
                "host_overhead_ms_per_step": loop_ms - stub_ms - tables_ms - sched_kernel_ms,
                "overhead_note": "loop - stub network - tables - step kernel over the same schedule; +-0.1 ms (the stub's "
                                 "stand-alone time is not exactly its in-loop time)",
                "includes_final_gather": world > 1,
                "samples_per_s": world * B / (loop_steps * loop_ms * 1e-3)}

    if rank != 0:
        return
    pk = peaks()
    fl = flops_per_step(B, D, S)
    tfl = world * fl / (ms * 1e-3) / 1e12
    bytes_step = 4.0 * B * D * S + 8.0 * B * D          # fp32 logits once + int32 state in/out
    tensor_bound = S >= 64
    if tensor_bound:
        roof = {"bound": "tensor", "achieved": fl / (kern_ms * 1e-3) / 1e12, "peak": pk["tc_burst"], "unit": "TFLOP/s",
                "traffic": None, "peak_source": pk["src"] + " bf16 dense (burst)",
                "note": "algorithmic 2*B*D*S^2 per launch; the kernel spends 3 bf16 tensor passes per algorithmic FLOP "
                        "(split precision), so 1/3 is the ceiling of this fraction",
                "hbm_gbs": bytes_step / (kern_ms * 1e-3) / 1e9}
        # DRAM bytes of one launch from the committed summary of the latest ncu --set full capture of this kernel at this
        # shape (profiles/ncu_traffic.json); null when none is committed
        if impl != nat.IMPL_SIMT and not args.batch:
            roof["traffic"] = ncu_traffic(args.workload)
        t_floor = max(bytes_step / (pk["hbm"] * 1e9), 3.0 * fl / (pk["tc_burst"] * 1e12))
        roof["t_floor_ms"] = t_floor * 1e3
        roof["frac_of_3pass_floor"] = t_floor / (kern_ms * 1e-3)
    else:
        roof = {"bound": "hbm", "achieved": bytes_step / (kern_ms * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                "traffic": None, "peak_source": pk["src"] + " copy bandwidth"}
    roof["frac"] = roof["achieved"] / roof["peak"]
    roof["kernel_ms"] = kern_ms
    line = {
        "metric": "reverse_step_tflops", "value": tfl, "unit": "TFLOP/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"{args.workload}: S={S} D={D} B={B}/GPU {w['fwd']} rate, {w['mode']} reverse step "
                               f"(TauL predictor, lib/sampling/sampling.py:119-160)",
                   "l2": "inputs larger than L2 (2 alternating logits buffers)" if flush is None else "L2 flushed between timed steps",
                   "kernels": args.kernels, "times": "steps spread over the schedule max_t..min_t",
                   "samples_per_s_at_num_steps": world * B / (w["num_steps"] * ms * 1e-3), "num_steps": w["num_steps"],
                   "sampler_loop": loop, "fused_head": fused},
        "roofline": roof,
        "e2e": None,
        "gpu_launches": int(launches),
        "clocks": clk.summary(),
        "gbytes_per_s": world * bytes_step / (ms * 1e-3) / 1e9,
    }
    dense = {"value": world * fl / (e2e_ms * 1e-3) / 1e12, "unit": "TFLOP/s", "ms_per_step": e2e_ms,
             "h2d_bytes_per_step": int(B * D * S * 4 + B * D * 4), "d2h_bytes_per_step": int(B * D * 4),
             "h2d_gbytes_per_s_per_gpu": (B * D * S * 4 + B * D * 4) / (e2e_ms * 1e-3) / 1e9,
             "note": "C-ABI reverse step fed from pinned HOST (N,D,S) fp32 logits + state, chunked on 2 streams, new state read "
                     "back: bound by the host link (3.2 GB per step and GPU), not by the kernel"}
    if fused is not None:
        # The reference-facing call of the CIFAR10 config ends in the truncated-logistic head
        # (config/cifar10_config/config_tauUnet_cifar10.py:59: model_output = 'logistic_pars'): the host hands over the two
        # numbers per dimension the U-Net emits plus the state, the step kernel evaluates the head itself.  That is the
        # declared end-to-end figure; the dense-logits leg is kept next to it.
        fe = fused["e2e"]
        line["e2e"] = {"value": fe["tflops"], "unit": "TFLOP/s", "ms_per_step": fe["ms_per_step"],
                       "h2d_bytes_per_step": fe["h2d_bytes_per_step"], "d2h_bytes_per_step": fe["d2h_bytes_per_step"],
                       "path": "ctdd_reverse_step with the fused truncated-logistic head (mu, log_scale, state from pinned HOST "
                               "memory every step; new state copied back)", "dense_logits_leg": dense}
    else:
        line["e2e"] = dense
    if world == 1 and not args.no_cpu:
        n_cpu = w["cpu_N"]
        tc_, kind_ = cpu_reference_step_time(w, n_cpu, args.cpu_steps, 1)
        line["cpu_baseline"] = {"value": flops_per_step(n_cpu, D, S) / tc_ / 1e12, "unit": "TFLOP/s", "cores": os.cpu_count(),
                                "kind": kind_, "sample": f"N={n_cpu} samples x D={D}, {args.cpu_steps} steps of "
                                + ("the staged unmodified reference (get_reverse_rates + TauL update)" if kind_ == "reference"
                                   else "the oracle port"),
                                "ms_per_step": tc_ * 1e3, "sample_steps_per_s": n_cpu / tc_}
    emit(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------
# C5: MidPointTauL step + SDDM CT-ELBO loss, batch sweep (BASELINE.json configs[4])

def _c5_cfg(make_cfg, w, D, S, device):
    mcfg = dict(w["model"], concat_dim=D)
    return make_cfg(data=dict(S=S, shape=[D], name="DiscreteCIFAR10"), model=mcfg, training=dict(max_t=w["max_t"], n_iters=1000),
                    sampler=dict(name="MidPointTauL", num_steps=w["num_steps"], min_t=w["min_t"], eps_ratio=1e-9,
                                 initial_dist="gaussian", num_corrector_steps=0, corrector_step_size_multiplier=1.5,
                                 corrector_entry_time=0.0, is_ordinal=True),
                    loss=dict(name="SDDMElbo", eps_ratio=1e-9, nll_weight=0.01, min_time=0.01, one_forward_pass=True,
                              logit_type="reverse_prob", loss_type="rm", ce_coeff=0.0), device=device)


def c5_flops(B, D, S):
    return dict(midpoint=4.0 * B * D * S * S, loss=6.0 * B * D * S * S)     # 2 evaluations; 2 forward + 1 backward contraction


def run_reference_c5(args, w):
    """CPU arm of C5 on N = cpu_N samples: SDDMElbo.calc_loss forward + backward of the staged UNMODIFIED reference (else
    the oracle's restatement) with the 1-parameter stub network, and the two reverse-rate evaluations of a MidPointTauL
    step (the reference's own MidPointTauL cannot run for DiscreteCIFAR10 - SURVEY quirk B.5 - so that half always uses
    get_reverse_rates of the reference / the port plus the drift and jump lines of sampling.py:423-503)."""
    import torch.nn as nn
    torch.set_num_threads(os.cpu_count() or 1)
    S, D, n = w["S"], w["D"], w["cpu_N"]
    logits, x0 = synth_logits(n, D, S, 1234, "cpu")
    rh, ref = _reference_modules()
    kind = "reference" if ref is not None else "port"
    from oracle import ref_harness as rh2, ctmc_oracle as oc, loss_oracle as lo
    cfg = _c5_cfg(rh2.make_cfg, w, D, S, "cpu")
    h = (w["max_t"] - w["min_t"]) / w["num_steps"]
    fp = oc.ForwardProcess(w["fwd"], S, **w["model"])
    if ref is not None:
        mixin = ref.fm.GaussianTargetRate

        class RefModel(nn.Module, mixin):
            def __init__(self):
                nn.Module.__init__(self)
                mixin.__init__(self, cfg, "cpu")
                self.w = nn.Parameter(torch.zeros(1))

            def forward(self, x, t):
                return logits + self.w

        model = RefModel()
        model.device = "cpu"
        loss_obj = ref.lu.get_loss(cfg)
        state = {"model": model, "optimizer": None, "n_iter": 0}
        loss_fn = lambda: loss_obj.calc_loss(x0, state)
        rates = lambda t_ones, xx: ref.ss.get_reverse_rates(model, logits, xx, t_ones, cfg, n, D, S)[0]
    else:
        wparam = torch.zeros(1, requires_grad=True)
        ts = torch.rand(n) * 0.98 + 0.01
        loss_fn = lambda: lo.loss_value("SDDMElbo", fp, lambda x, t, label=None: logits + wparam, x0, ts, seed=1, eps=1e-9,
                                        nll_weight=0.01, logit_type="reverse_prob", loss_type="rm", ce_coeff=0.0)
        rates = lambda t_ones, xx: oc.reverse_rates(logits, xx, fp.transition(t_ones), fp.rate(t_ones), "SDDMElbo",
                                                    "reverse_prob", 1e-9)[0]
    tl, tm = [], []
    for i in range(args.steps + args.warmup):
        t0 = time.perf_counter()
        loss_fn().backward()
        t1 = time.perf_counter()
        with torch.no_grad():
            t_ones = 0.5 * torch.ones((n,))
            x = x0.clone()
            oh = torch.nn.functional.one_hot(x, S)
            rz = rates(t_ones, x) * (1 - oh)
            diff = (torch.arange(S).view(1, 1, S) - x.unsqueeze(-1)).float()
            xp = torch.clamp(x + torch.round(0.5 * h * (rz * diff).sum(-1)).long(), 0, S - 1)
            rz2 = rates(t_ones - 0.5 * h, xp) * (1 - torch.nn.functional.one_hot(xp, S))
            k = torch.poisson(rz2 * h)
            x = torch.clamp(x + (k * (torch.arange(S).view(1, 1, S) - xp.unsqueeze(-1))).sum(-1), 0, S - 1).long()
        t2 = time.perf_counter()
        if i >= args.warmup:
            tl.append(t1 - t0)
            tm.append(t2 - t1)
    t_loss, t_mid = float(np.mean(tl)), float(np.mean(tm))
    fl = c5_flops(n, D, S)
    val = (fl["midpoint"] + fl["loss"]) / (t_loss + t_mid) / 1e12
    line = {"impl": "reference", "metric": "c5_step_tflops", "value": val, "unit": "TFLOP/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": (t_loss + t_mid) * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"C5: S={S} D={D} MidPointTauL step + SDDMElbo fwd+bwd, CPU sample N={n}",
                       "loss_ms": t_loss * 1e3, "midpoint_ms": t_mid * 1e3},
            "cpu_baseline": {"value": val, "unit": "TFLOP/s", "cores": os.cpu_count(), "kind": kind,
                             "sample": f"N={n} samples x D={D}: calc_loss + backward and two reverse-rate evaluations per step, "
                                       f"{args.steps} steps"},
            "e2e": {"value": val, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(json.dumps(line))


def run_ours_c5(args, w, rank, world, local_rank):
    import torch.distributed as dist
    import torch.nn as nn
    from ctdd_b200 import _native as nat, make_config, ops
    from ctdd_b200.lib.models import forward_model as fm
    from ctdd_b200.lib.losses import losses_utils
    import ctdd_b200.lib.losses.losses  # noqa: F401

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    S, D = w["S"], w["D"]
    K, W = args.steps, args.warmup
    totals = [64, 128, 256, 512, 1024, 2048, 4096] if args.sweep else [args.total_batch or (args.batch or w["B"]) * world]
    cfg = _c5_cfg(make_config, w, D, S, str(dev))
    h = (w["max_t"] - w["min_t"]) / w["num_steps"]
    Bmax = max(-(-t // world) for t in totals)

    class Stub(nn.Module, fm.GaussianTargetRate):
        """1-parameter stand-in for the score network: logits = resident synthetic logits + w (so backward is exercised)."""

        def __init__(self):
            nn.Module.__init__(self)
            fm.GaussianTargetRate.__init__(self, cfg, str(dev))
            self.w = nn.Parameter(torch.zeros(1, device=dev))
            self.buf, self.x0 = synth_logits(Bmax, D, S, 1234 + 17 * rank, dev)

        def forward(self, x, t):
            return self.buf[: x.shape[0]] + self.w

    model = Stub()
    model.device = str(dev)
    loss_obj = losses_utils.get_loss(cfg)
    loss_obj.seed = 0xC7DD
    state = {"model": model, "optimizer": None, "n_iter": 0}
    t_mid_sched = [0.9, 0.5, 0.1]      # the midpoint step is timed at three points of the schedule
    Q, QT, beta = model.qt0_tables([t for tt in t_mid_sched for t in (tt, tt - 0.5 * h)], dev)
    Rb, RbT = model.base_rate_tables(dev)
    branch = nat.BRANCH_SDDM_REVERSE_PROB
    tc = ops.prep_tc_tables(Q, QT, Rb, 1e-9, branch)
    tcs = ops.prep_tc_static(Rb)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def one(B, clk=False):
        lg = model.buf[:B]
        x = torch.clamp(model.x0[:B] + 2, 0, S - 1).to(torch.int32)
        row_offset = rank * B * D
        kw = dict(N=B, D=D, S=S, seed=0xC7DD, row_offset=row_offset, tc_static=tcs)

        def mid(i, j):
            xp = ops.reverse_step(nat.MODE_MIDPOINT_DRIFT, branch, lg, x, Q[2 * j], QT[2 * j], Rb, RbT, beta[2 * j], h, 1e-9,
                                  offset=i, tc_tables=tc[2 * j], **kw)["x"]
            return ops.reverse_step(nat.MODE_MIDPOINT_JUMP, branch, lg, xp, Q[2 * j + 1], QT[2 * j + 1], Rb, RbT, beta[2 * j + 1],
                                    h, 1e-9, offset=i, x_base=x, tc_tables=tc[2 * j + 1], **kw)["x"]

        def loss_step():
            model.w.grad = None
            loss = loss_obj.calc_loss(model.x0[:B], state)
            loss.backward()
            return loss

        for i in range(W):
            mid(i, i % 3)
            loss_step()
        barrier()
        n0 = nat.launch_count()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        tm = tl = 0.0
        ctx = ClockSampler(local_rank) if clk else None
        if ctx:
            ctx.__enter__()
        for i in range(K):
            ev[0].record()
            xm = mid(W + i, i % 3)
            ev[1].record()
            loss = loss_step()
            ev[2].record()
            torch.cuda.synchronize(dev)
            tm += ev[0].elapsed_time(ev[1])
            tl += ev[1].elapsed_time(ev[2])
        if ctx:
            ctx.__exit__(None, None, None)
        barrier()
        launches = nat.launch_count() - n0
        last = {"x": xm, "loss": loss.detach(), "grad_w": model.w.grad.detach().clone()}
        # end to end through the public API with HOST inputs: the minibatch comes from pinned host memory, the loss value
        # is read back (.item()), one MidPointTauL-style step on the resident logits in between
        host_mb = torch.empty((B, D), dtype=torch.int64, pin_memory=True)
        host_mb.copy_(model.x0[:B])
        t0 = time.perf_counter()
        for i in range(max(1, min(K, args.e2e_steps))):
            mb = host_mb.to(dev, non_blocking=True)
            model.w.grad = None
            loss = loss_obj.calc_loss(mb, state)
            loss.backward()
            mid(W + i, i % 3)
            float(loss.item())
        torch.cuda.synchronize(dev)
        e2e = (time.perf_counter() - t0) * 1e3 / max(1, min(K, args.e2e_steps))
        t = torch.tensor([tm / K, tl / K, e2e], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), float(t[2]), launches, (ctx.summary() if ctx else None), last

    rows = []
    for tot in totals:
        B = -(-tot // world)
        tmid, tloss, e2e, launches, clocks, last = one(B, clk=(tot == totals[-1]))
        rows.append(dict(total_batch=B * world, per_gpu=B, midpoint_ms=tmid, loss_ms=tloss, e2e_ms=e2e, launches=launches, clocks=clocks))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)       # the largest batch of a sweep
    if rank != 0:
        return
    r = rows[-1]
    B = r["per_gpu"]
    fl = c5_flops(B, D, S)
    ms = r["midpoint_ms"] + r["loss_ms"]
    pk = peaks()
    dom = "loss" if r["loss_ms"] >= r["midpoint_ms"] else "midpoint"
    dom_ms = r[dom + "_ms"]
    roof = {"bound": "tensor", "kernel": "loss_kernel<fwd/bwd> (ctdd_loss.cu)" if dom == "loss" else "step_q_kernel (ctdd_step_tcq.cu)",
            "achieved": fl[dom] / (dom_ms * 1e-3) / 1e12, "peak": pk["tc_burst"], "unit": "TFLOP/s", "traffic": ncu_traffic("C5"),
            "peak_source": pk["src"] + " bf16 dense (burst)",
            "note": "algorithmic FLOP of the dominant part (loss: 6*B*D*S^2, midpoint step: 4*B*D*S^2) / its CUDA-event time"}
    roof["frac"] = roof["achieved"] / roof["peak"]
    line = {"metric": "c5_step_tflops", "value": world * (fl["midpoint"] + fl["loss"]) / (ms * 1e-3) / 1e12, "unit": "TFLOP/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"C5: S={S} D={D} total batch {r['total_batch']} ({B}/GPU): MidPointTauL step (drift + jump "
                                   f"evaluation, sampling.py:390-526) + SDDMElbo.calc_loss forward+backward (losses.py:290-544), "
                                   f"1-parameter stub network", "l2": "inputs larger than L2 at B >= 64 (0.2 GB of logits per 64 samples)",
                       "midpoint_ms": r["midpoint_ms"], "loss_ms": r["loss_ms"],
                       "midpoint_tflops": world * fl["midpoint"] / (r["midpoint_ms"] * 1e-3) / 1e12,
                       "loss_tflops": world * fl["loss"] / (r["loss_ms"] * 1e-3) / 1e12,
                       "sweep": rows if args.sweep else None},
            "roofline": roof,
            "e2e": {"value": world * (fl["midpoint"] + fl["loss"]) / (r["e2e_ms"] * 1e-3) / 1e12, "unit": "TFLOP/s",
                    "ms_per_step": r["e2e_ms"], "h2d_bytes_per_step": int(B * D * 8), "d2h_bytes_per_step": 4,
                    "note": "calc_loss(minibatch from pinned HOST memory) + backward + loss.item(), then one midpoint step"},
            "gpu_launches": int(r["launches"]), "clocks": r["clocks"]}
    emit(json.dumps(line))


def ncu_traffic(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel of `workload` per launch, from the committed
    summary of the latest `ncu --set full` capture (profiles/ncu_traffic.json, written by tools/ncu_summary.py); None when
    no capture of this workload is committed."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return json.load(open(p)).get(workload, {}).get("dram_bytes")
    except Exception:
        return None


_RESULT_OUT = None


def emit(line):
    """Print the result line on the process's original stdout."""
    out = _RESULT_OUT if _RESULT_OUT is not None else sys.stdout
    out.write(line + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C4", choices=list(WORKLOADS))
    ap.add_argument("--kernels", default="auto", choices=["auto", "simt", "tc"])
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-steps", type=int, default=5)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--batch", type=int, default=0, help="override the per-GPU batch of the workload (diagnostic)")
    ap.add_argument("--total-batch", type=int, default=0, help="C5: total batch over all GPUs (64..4096)")
    ap.add_argument("--sweep", action="store_true", help="C5: run the whole batch sweep 64..4096 (the line reports the largest)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (new states; C1-C4: its counters, C5: "
                         "loss and gradient) as DIR/<name>.npy, rank 0's rows; inputs are seeded, so runs compare (C5's "
                         "loss and gradient are float sums in no fixed order: compare those with a tolerance)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed (--impl ours)")
    # stdout carries exactly ONE JSON line: libraries that write to file descriptor 1 (NCCL prints its version banner
    # there when NCCL_DEBUG is set) are sent to stderr for the whole run; the result line goes to the saved descriptor
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    # the default generators draw the starting states (C1-C4) and the loss's time draws (C5): seeded, so that the same
    # arguments give the same inputs in every run
    torch.manual_seed(0xC7DD)
    w = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, w, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        (run_ours_c5 if args.workload == "C5" else run_ours)(args, w, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
