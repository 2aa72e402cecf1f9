"""Reverse-step kernels against the oracle on inputs whose fp32 reverse rates are EXACT, so every kernel family, whatever
its summation order, must reproduce the oracle's rates, prefix sums, jump counts and picks bit for bit - at any noise
level, up to chunk totals far above the Cornish-Fisher switch (lambda > 64) and the 4096-pick cap.

The inputs (exact_problem):
  * q_{t|0} entries are powers of two 2^-a, a in [1, A_MAX], and eps = 0: 1 / (Q[k, x] + eps) is exact, and so is the
    3 x BF16 split of the tensor path (the high part holds the value, the others are zero);
  * every logits row has 1, 2 or 4 tied maxima at 0 and -1e4 elsewhere: the softmax is exactly 2^-m on every path
    (ex2.approx / rcp.approx included);
  * the base rates are dyadic ({1..7} x 2^-4) inside a band |i - j| <= BAND (diagonal = minus the row sum), so some
    32-state chunks lie outside the band of a state; for S > 8 some states have no incoming rate, so rows there have
    no reverse rate at all and sit next to rows at the pick cap;
  * beta and h are powers of two (the tensor path's unscaled tau-leap variant scales only the chunk total).
Every value the maps consume is then a multiple of some 2^E below 2^(E + 24): sums in any order are exact
(_assert_exact checks that on the CPU before a kernel runs).  The only place where device and oracle may still differ is
the count's threshold arithmetic (expf against numpy's exp, normcdfinvf against ndtri): a row may then differ only when
its count margin (oracle/rng.py poisson_count_margin) is at most 1e-6, and at most 2 rows per call may.

The CPU test at the top checks that margin against what a perturbation of the rates actually does."""
import time

import numpy as np
import pytest
import torch

from oracle import ctmc_oracle as oc, rng

BETA = 8.0
EPS = 0.0
A_MAX = 4
BAND = 40
SEED = 0x5EED
ROW0 = 8 * 1021                   # row offset of every call: a multiple of 8 (a batch behind other ranks' rows)
COUNT_TIE = 1e-6                  # count margin below which device and oracle may decide differently
MAX_TIES = 2                      # ... and at most this many such rows per call

_ties_seen = []                   # (what, rows) of every tolerated mismatch, reported at the end of the module


# ---------------------------------------------------------------------------------------------------------------
# CPU: the count margin of the tie rule, above and below the Cornish-Fisher switch

@pytest.mark.parametrize("lo,hi", [(0.5, 64.0), (64.5, 500.0)], ids=["exact_pmf", "cornish_fisher"])
@pytest.mark.parametrize("d", [1e-4, 1e-5])
def test_count_margin_predicts_which_counts_flip(lo, hi, d):
    """Single-state rows, every rate perturbed by +-d (relative): a row whose count flips has margin <= 1.05 d, and a
    row with margin <= d / 2 flips."""
    n = 20000
    g = np.random.Generator(np.random.PCG64(3))
    lam = g.uniform(lo, hi, n).astype(np.float32)
    grow = np.arange(n, dtype=np.uint64) + np.uint64(ROW0)
    v0 = rng.count_units(grow, 5, SEED, 0, True)        # one state: the count call shared by 4 rows
    K = rng.poisson_from_unit(lam, v0)
    margin = rng.poisson_rows_margin(lam[:, None], ROW0, 5, SEED, picks=False)
    assert np.array_equal(margin, rng.poisson_count_margin(lam, v0))
    flip = np.zeros(n, dtype=bool)
    for sgn in (1.0, -1.0):
        flip |= rng.poisson_from_unit((lam.astype(np.float64) * (1.0 + sgn * d)).astype(np.float32), v0) != K
    assert flip.sum() >= 5, flip.sum()                                      # the test does see flips
    assert np.all(margin[flip] <= 1.05 * d), (margin[flip] / d).max()
    assert np.all(flip[margin <= d / 2]), np.flatnonzero(~flip & (margin <= d / 2))[:8]


def test_cornish_fisher_rounds_like_the_fused_device_code():
    """lam > 64: f = fma(fma(z, z, -1), 0.16666667, fma(sqrtf(lam), z, lam)), each fused operation rounded once, then
    rint - against an exact rational evaluation of the same three fused operations."""
    from fractions import Fraction
    g = np.random.Generator(np.random.PCG64(8))
    lam = g.uniform(64.5, 5000.0, 3000).astype(np.float32)
    v = g.uniform(1e-6, 1.0, 3000).astype(np.float32)
    z, f = rng._cornish_fisher(lam, v)

    def rn32(q):      # exact rational -> nearest fp32, ties to even
        lo = np.float32(float(q))
        if Fraction(float(lo)) == q:
            return lo
        a = lo if Fraction(float(lo)) < q else np.nextafter(lo, np.float32(-np.inf))
        b = np.nextafter(a, np.float32(np.inf))
        da, db = q - Fraction(float(a)), Fraction(float(b)) - q
        if da != db:
            return a if da < db else b
        return a if (a.view(np.uint32) & 1) == 0 else b

    for i in range(0, 3000, 7):
        Z, L = Fraction(float(z[i])), Fraction(float(lam[i]))
        t = rn32(Fraction(float(np.sqrt(lam[i]))) * Z + L)
        u = rn32(Z * Z - 1)
        want = rn32(Fraction(float(u)) * Fraction(float(np.float32(0.16666667))) + Fraction(float(t)))
        assert f[i] == want, (i, f[i], want)
    # 4097 * (16773121 * 2^-30) = 2^6 + 2^-30 exactly; + 2^30 rounds in fp64 to 2^30 + 2^6, halfway between two fp32
    # values: the exact residual (+2^-30) rounds it up, where a second round-to-even would go down to 2^30
    assert rng._fma32(np.float32(4097.0), np.float32(16773121 * 2.0 ** -30), np.float32(2.0 ** 30)) == np.float32(2.0 ** 30 + 128)


# ---------------------------------------------------------------------------------------------------------------
# exact inputs


def exact_problem(S, N, D, seed, band=BAND, x_mode="uniform"):
    """(Q (S, S), Rb (S, S), logits (N, D, S), x (N, D) int64) with exact fp32 reverse rates (module docstring)."""
    g = np.random.Generator(np.random.PCG64(seed))
    Q = np.exp2(-g.integers(1, A_MAX + 1, (S, S))).astype(np.float32)
    i, j = np.arange(S)[:, None], np.arange(S)[None, :]
    Rb = (g.integers(1, 8, (S, S)) * 2.0 ** -4) * ((np.abs(i - j) <= band) & (i != j))
    if S > 8:     # quiet states: no forward jump leads into them, so a row at one has no reverse rate at all
        quiet = (g.random(S) < 0.15) | np.isin(np.arange(S), (1, S - 2))
        Rb[:, quiet] = 0.0
    Rb[np.arange(S), np.arange(S)] = -Rb.sum(1)
    Rb = Rb.astype(np.float32)
    rows = N * D
    logits = np.full((rows, S), -1.0e4, dtype=np.float32)
    nhot = g.choice([m for m in (1, 2, 4) if m <= S], rows)
    for r in range(rows):
        logits[r, g.choice(S, nhot[r], replace=False)] = 0.0
    if x_mode == "uniform":
        x = g.integers(0, S, rows)
    else:       # x_mode = "edges": states near both ends (clamping) and in the middle
        x = np.where(g.random(rows) < 0.5, g.integers(0, min(S, 4), rows), S - 1 - g.integers(0, min(S, 4), rows))
        x = np.where(g.random(rows) < 0.3, g.integers(0, S, rows), x)
    return Q, Rb, logits.reshape(N, D, S), x.reshape(N, D).astype(np.int64)


def reference_rates(Q, Rb, logits, x):
    """fp64 (ratio, rr) of the tauLDR branch with eps = 0 (rr keeps its s == x entry), asserted to be fp32 values."""
    N, D, S = logits.shape
    lg = logits.reshape(-1, S).astype(np.float64)
    e = np.exp(lg - lg.max(1, keepdims=True))
    p = e / e.sum(1, keepdims=True)
    xf = x.reshape(-1)
    Q64 = Q.astype(np.float64)
    ratio = (p / Q64.T[xf]) @ Q64
    rr = BETA * Rb.astype(np.float64).T[xf] * ratio
    for a in (ratio, rr):
        assert np.array_equal(a.astype(np.float32).astype(np.float64), a), "rates are not fp32 values"
    return ratio, rr


def _lsb_exponent(v):
    """exponent of the lowest set bit of every non-zero fp32 value (v is fp64 holding fp32 values)."""
    m, e = np.frexp(np.abs(v))
    mi = (m * 2.0 ** 24).astype(np.int64)
    tz = np.zeros(mi.shape, np.int64)
    nz = mi != 0
    t = np.where(nz, mi, 1)
    while True:
        odd = (t & 1) == 1
        if odd.all():
            break
        tz += ~odd
        t = np.where(odd, t, t >> 1)
    return np.where(nz, e - 24 + tz, 10 ** 6)


def _assert_exact(vals, what):
    """Every row of vals (rows, n; fp64 holding fp32 values) sums exactly in fp32 in ANY order: its values are multiples
    of 2^E and the sum of their magnitudes is below 2^(E + 24)."""
    vals = np.asarray(vals, np.float64)
    assert np.array_equal(vals.astype(np.float32).astype(np.float64), vals), (what, "values are not fp32")
    E = _lsb_exponent(vals).min(axis=1)
    mag = np.abs(vals).sum(axis=1)
    ok = (mag == 0) | (mag < np.exp2(np.minimum(E, 200) + 24.0))
    assert ok.all(), (what, "inexact row sums", np.flatnonzero(~ok)[:8])


def _chunks(a, S):
    return [a[:, c0:min(c0 + rng.JUMP_CHUNK, S)] for c0 in range(0, S, rng.JUMP_CHUNK)]


class Problem:
    """One exact problem on the GPU and its fp64 / oracle references."""

    def __init__(self, S, N, D, seed, impl, x_mode="uniform"):
        self.S, self.N, self.D, self.impl = S, N, D, impl
        Q, Rb, logits, x = exact_problem(S, N, D, seed, x_mode=x_mode)
        self.Q, self.Rb, self.logits, self.x = Q, Rb, logits, x
        self.ratio64, self.rr64 = reference_rates(Q, Rb, logits, x)
        onehot = np.eye(S, dtype=bool)[x.reshape(-1)]
        self.rz64 = np.where(onehot, 0.0, self.rr64)
        self.rzc64 = np.where(onehot, 0.0, self.rr64 + BETA * Rb.astype(np.float64)[x.reshape(-1)])
        self.nat = None

    def _upload(self):
        from ctdd_b200 import _native as nat, ops
        self.nat, self.ops = nat, ops
        Q, Rb, impl = self.Q, self.Rb, self.impl
        dev = "cuda"
        self.tQ, self.tQT = torch.from_numpy(Q).to(dev), torch.from_numpy(np.ascontiguousarray(Q.T)).to(dev)
        self.tRb, self.tRbT = torch.from_numpy(Rb).to(dev), torch.from_numpy(np.ascontiguousarray(Rb.T)).to(dev)
        self.tlog = torch.from_numpy(self.logits).to(dev)
        self.tx = torch.from_numpy(self.x).to(torch.int32).to(dev)
        self.tct = self.tcs = None
        if impl == nat.IMPL_TC:
            self.tct = ops.prep_tc_tables(self.tQ[None], self.tQT[None], self.tRb, EPS, nat.BRANCH_TAULDR)[0]
            self.tcs = ops.prep_tc_static(self.tRb)

    def step(self, mode, h, offset, reject=False, x_base=None, want_rr=False, row_offset=ROW0):
        if self.nat is None:
            self._upload()
        stats = torch.zeros(8, dtype=torch.int64, device="cuda")
        out = self.ops.reverse_step(mode, self.nat.BRANCH_TAULDR, self.tlog, self.tx, self.tQ, self.tQT, self.tRb, self.tRbT,
                                    BETA, h, EPS, N=self.N, D=self.D, S=self.S, impl=self.impl, tc_tables=self.tct,
                                    tc_static=self.tcs, reject_multi=reject, seed=SEED, offset=offset,
                                    row_offset=row_offset, stats=stats,
                                    x_base=None if x_base is None else torch.from_numpy(x_base).to(torch.int32).cuda(),
                                    want_rr=want_rr, want_ratio=want_rr)
        x = None if mode == self.nat.MODE_RATES_ONLY else out["x"].cpu().numpy().astype(np.int64).reshape(-1)
        return x, stats.cpu().numpy()[:5], out

    # ----- oracle side
    def tau_leap(self, corr, h, offset, reject, x_base=None, row_offset=ROW0):
        rz = self.rzc64 if corr else self.rz64
        lam64 = rz * h
        for c in _chunks(lam64, self.S):
            _assert_exact(c, "tau-leap chunk")
        t = torch.from_numpy(rz.astype(np.float32).reshape(self.N, self.D, self.S))
        xe = torch.from_numpy(self.x)
        xb = xe if x_base is None else torch.from_numpy(x_base)
        want, st = oc.tau_leap_update(t, xe, xb, h, self.S, reject, offset, SEED, row_offset=row_offset)
        lam = lam64.astype(np.float32)
        margin = rng.poisson_rows_margin(lam, row_offset, offset, SEED, picks=False)
        ost = np.array([st["changed_base"], st["nonzero_jump"], st["changed_eval"], st["rows_jumped"], st["rows_multi"]])
        return want.numpy().reshape(-1), ost, margin, lam

    def euler(self, corr, h, offset, row_offset=ROW0):
        rz = self.rzc64 if corr else self.rz64
        _assert_exact(rz * h, "Euler total")
        tot = (rz * h).sum(1)
        P = rz * h
        xf = self.x.reshape(-1)
        P[np.arange(P.shape[0]), xf] = np.maximum(0.0, 1.0 - tot)
        _assert_exact(P, "Euler probabilities")
        t = torch.from_numpy(rz.astype(np.float32).reshape(self.N, self.D, self.S))
        want, _ = oc.euler_update(t, torch.from_numpy(self.x), h, self.S, offset, SEED, row_offset=row_offset)
        want = want.numpy().reshape(-1)
        ch = int((want != xf).sum())
        return want, np.array([ch, 0, ch, 0, 0]), (tot > 1.0)

    def drift(self, h):
        diff = np.arange(self.S)[None, :] - self.x.reshape(-1, 1)
        _assert_exact(self.rz64 * diff, "drift sum")
        val = 0.5 * h * (self.rz64 * diff).sum(1)
        ch = np.round(val).astype(np.int64)                         # half to even, like rintf
        want = np.clip(self.x.reshape(-1) + ch, 0, self.S - 1)
        t = torch.from_numpy(self.rz64.astype(np.float32).reshape(self.N, self.D, self.S))
        assert np.array_equal(oc.midpoint_drift(t, torch.from_numpy(self.x), h, self.S).numpy().reshape(-1), want)
        xf = self.x.reshape(-1)
        nch = int((want != xf).sum())
        return want, np.array([nch, int((ch != 0).sum()), nch, 0, 0]), val


def _check(what, got, gst, want, wst, margin=None):
    """States and the five counters equal; a row may differ only at a count tie (margin <= COUNT_TIE), at most MAX_TIES."""
    bad = np.flatnonzero(got != want)
    if bad.size:
        assert margin is not None, (what, "mismatching rows", bad[:8], got[bad[:8]], want[bad[:8]])
        assert bad.size <= MAX_TIES and np.all(margin[bad] <= COUNT_TIE), \
            (what, "mismatch that is not a count tie", bad[:8], margin[bad[:8]], got[bad[:8]], want[bad[:8]])
        _ties_seen.append((what, bad.size))
        assert np.all(np.abs(gst - wst) <= 2 * bad.size), (what, gst, wst)
    else:
        assert np.array_equal(gst, wst), (what, "counters", gst, wst)


def _chunk_stats(lam, row_offset, offset, shared):
    """Per (row, chunk): chunk totals (fp32) and counts K of the map."""
    rows, S = lam.shape
    grow = np.arange(rows, dtype=np.uint64) + np.uint64(row_offset)
    tots, Ks = [], []
    for ci, c in enumerate(_chunks(lam, S)):
        tot = np.cumsum(c, axis=1, dtype=np.float32)[:, -1]
        Ks.append(rng.poisson_from_unit(tot, rng.count_units(grow, offset, SEED, ci << 16, shared)))
        tots.append(tot)
    return np.stack(tots, 1), np.stack(Ks, 1)


class Coverage:
    def __init__(self):
        self.max_tot = 0.0
        self.cap = 0
        self.reg_batches = 0
        self.dealt_batches = 0
        self.dealt_multi_round = 0
        self.clamp_lo = self.clamp_hi = 0
        self.mixed = 0            # tcq batches holding a row without jumps and a chunk at the pick cap

    def add_jump(self, lam, x_base, x_eval, row_offset, offset, S, tcq):
        tots, Ks = _chunk_stats(lam, row_offset, offset, S <= rng.JUMP_SHARED_MAX_S)
        self.max_tot = max(self.max_tot, float(tots.max()))
        self.cap += int((Ks >= rng.JUMP_PICK_CAP).sum())
        if tcq:       # batches of 32 consecutive rows of the launch, per chunk: register picks (max K <= 3) or dealt
            rows = lam.shape[0]
            for b0 in range(0, rows, 32):
                Kc = np.minimum(Ks[b0:b0 + 32], rng.JUMP_PICK_CAP)
                mx = Kc.max(axis=0)
                self.reg_batches += int(((mx > 0) & (mx <= 3)).sum())
                self.dealt_batches += int((mx > 3).sum())
                self.dealt_multi_round += int((Kc.sum(axis=0)[mx > 3] > 32).sum())

    def add_clamp(self, unclamped, S):
        self.clamp_lo += int((unclamped < 0).sum())
        self.clamp_hi += int((unclamped > S - 1).sum())


def _unclamped(P, lam, x_eval, x_base, row_offset, offset):
    k, _ = rng.poisson_rows(lam, row_offset, offset, SEED)
    return x_base + (k * (np.arange(P.S)[None, :] - x_eval[:, None])).sum(1)


# ---------------------------------------------------------------------------------------------------------------
# GPU


def _nat():
    from ctdd_b200 import _native as nat
    return nat


H_SWEEP = [2.0 ** -12, 2.0 ** -8, 2.0 ** -5, 2.0 ** -2, 2.0 ** 2, 2.0 ** 5]


@pytest.mark.gpu
@pytest.mark.parametrize("path,S", [("tc", 256), ("block", 9), ("block", 33), ("block", 100), ("block", 256)]
                         + [("small", s) for s in range(2, 9)])
def test_rates_are_exact_on_every_path(path, S):
    """The premise: MODE_RATES_ONLY's rr_out and ratio_out equal the fp64 rates bit for bit (the tensor path at S = 256,
    the block kernel, the general small-S kernel)."""
    nat = _nat()
    impl = nat.IMPL_TC if path == "tc" else nat.IMPL_SIMT
    P = Problem(S, 13, 29, 100 + S, impl)
    _, _, out = P.step(nat.MODE_RATES_ONLY, 0.0, 0, want_rr=True)
    rr = out["rr"].cpu().numpy().reshape(-1, S).astype(np.float64)
    ratio = out["ratio"].cpu().numpy().reshape(-1, S).astype(np.float64)
    assert np.array_equal(ratio, P.ratio64), np.argwhere(ratio != P.ratio64)[:8]
    assert np.array_equal(rr, P.rr64), np.argwhere(rr != P.rr64)[:8]


def _sweep_jump_modes(P, cov, what, tcq, hs, modes=("tau", "tau_reject", "corr", "mid_jump")):
    nat = _nat()
    g = np.random.Generator(np.random.PCG64(P.S))
    xf = P.x.reshape(-1)
    xb = np.clip(xf + g.integers(-3, 4, xf.shape), 0, P.S - 1)
    for hi, h in enumerate(hs):
        for mi, m in enumerate(modes):
            off = 16 * hi + mi + 1
            if m == "mid_jump":
                got, gst, _ = P.step(nat.MODE_MIDPOINT_JUMP, h, off, reject=True, x_base=xb.reshape(P.N, P.D))
                want, wst, margin, lam = P.tau_leap(False, h, off, True, x_base=xb.reshape(P.N, P.D))
                base = xb
            else:
                mode = nat.MODE_TAU_LEAP_CORR if m == "corr" else nat.MODE_TAU_LEAP
                got, gst, _ = P.step(mode, h, off, reject=(m == "tau_reject"))
                want, wst, margin, lam = P.tau_leap(m == "corr", h, off, m == "tau_reject")
                base = xf
            _check(f"{what} {m} h={h}", got, gst, want, wst, margin)
            cov.add_jump(lam, base, xf, ROW0, off, P.S, tcq)
            if m == "tau":
                cov.add_clamp(_unclamped(P, lam, xf, base, ROW0, off), P.S)


def _sweep_drift(P, what, hs):
    nat = _nat()
    for h in hs:
        got, gst, _ = P.step(nat.MODE_MIDPOINT_DRIFT, h, 0)
        want, wst, _ = P.drift(h)
        _check(f"{what} drift h={h}", got, gst, want, wst)


def _sweep_euler(P, what, hs, modes=("euler", "euler_corr")):
    nat = _nat()
    clamped = 0
    for hi, h in enumerate(hs):
        for m in modes:
            off = 200 + hi
            mode = nat.MODE_EULER_CORR if m == "euler_corr" else nat.MODE_EULER
            got, gst, _ = P.step(mode, h, off)
            want, wst, clamp = P.euler(m == "euler_corr", h, off)
            _check(f"{what} {m} h={h}", got, gst, want, wst)
            clamped += int(clamp.sum())
    return clamped


@pytest.mark.gpu
def test_tensor_path_sweep_matches_oracle_bit_for_bit():
    """S = 256 on the tcgen05 path over h = 2^-12 .. 2^2: the tau-leap kernel (with and without reject_multi: the
    unscaled variant; the corrector: scaled + R_t[x, :]; midpoint jump with x_base != x_eval; midpoint drift, whose exact
    values land on .5) and the Euler kernel at h * sum(rates) > 1 (diagonal clamped to 0).  Proves from the oracle that
    it reached chunk totals above 64, chunks at the 4096-pick cap, batches on both pick paths with dealt rounds beyond
    the first, and rows clamped at both ends."""
    nat = _nat()
    t0 = time.time()
    cov = Coverage()
    P = Problem(256, 13, 29, 7, nat.IMPL_TC)                          # 377 rows: ragged tile
    _sweep_jump_modes(P, cov, "tcq", True, H_SWEEP)
    _sweep_drift(P, "tcq", [2.0 ** -6, 2.0 ** -3, 1.0])
    clamped = _sweep_euler(P, "tc", [2.0 ** -2, 1.0])
    Pw = Problem(256, 24, 250, 8, nat.IMPL_TC)                        # 6000 rows: several tiles per CTA pair
    _sweep_jump_modes(Pw, cov, "tcq wide", True, [2.0 ** -8, 2.0 ** -5], modes=("tau", "corr"))
    clamped += _sweep_euler(Pw, "tc wide", [1.0])
    assert cov.max_tot > 64.0 * 8 and cov.cap > 0, (cov.max_tot, cov.cap)
    assert cov.reg_batches > 0 and cov.dealt_batches > 0 and cov.dealt_multi_round > 0, vars(cov)
    assert cov.clamp_lo > 0 and cov.clamp_hi > 0, vars(cov)
    assert clamped > 0
    print(f"\ntensor path sweep: {time.time() - t0:.1f} s, coverage {vars(cov)}")


@pytest.mark.gpu
def test_tensor_path_mixed_noise_batch():
    """One 32-row batch holds rows with no jump next to rows at the pick cap: logits rows whose hot entries give tiny
    or huge ratios, x at both ends.  Exercises the switch between register and dealt picks, dealt loops of several
    rounds and idle lanes beyond the last pick."""
    nat = _nat()
    S, N, D = 256, 3, 64
    P = Problem(S, N, D, 21, nat.IMPL_TC, x_mode="edges")
    cov = Coverage()
    for off, h in ((3, 2.0 ** -3), (4, 2.0 ** 5), (5, 2.0 ** -9)):
        got, gst, _ = P.step(nat.MODE_TAU_LEAP, h, off)
        want, wst, margin, lam = P.tau_leap(False, h, off, False)
        _check(f"mixed h={h}", got, gst, want, wst, margin)
        cov.add_jump(lam, P.x.reshape(-1), P.x.reshape(-1), ROW0, off, S, True)
        tots, Ks = _chunk_stats(lam, ROW0, off, False)
        Kr = np.minimum(Ks, rng.JUMP_PICK_CAP).sum(1)
        for b0 in range(0, N * D, 32):
            kb = Kr[b0:b0 + 32]
            if (kb == 0).any() and (Ks[b0:b0 + 32] >= rng.JUMP_PICK_CAP).any():
                cov.mixed += 1
    assert cov.mixed > 0 and cov.dealt_multi_round > 0 and cov.reg_batches > 0, vars(cov)


@pytest.mark.gpu
@pytest.mark.parametrize("S", [9, 33, 100, 256])
def test_block_kernel_sweep_matches_oracle_bit_for_bit(S):
    """The CUDA-core block kernel (the tensor path's on-GPU cross-check) in every mode, from S = 9 (the smallest S it
    serves) through partial last chunks (33, 100) to 256."""
    nat = _nat()
    cov = Coverage()
    P = Problem(S, 13, 29, 30 + S, nat.IMPL_SIMT)
    _sweep_jump_modes(P, cov, f"block S={S}", False, [2.0 ** -8, 2.0 ** -2, 2.0 ** 5] if S > 9 else [2.0 ** -4, 2.0 ** 2, 2.0 ** 7])
    _sweep_drift(P, f"block S={S}", [2.0 ** -4, 1.0])
    _sweep_euler(P, f"block S={S}", [2.0 ** -6, 2.0])
    assert cov.max_tot > 64.0 and cov.cap > 0, (cov.max_tot, cov.cap)


@pytest.mark.gpu
@pytest.mark.parametrize("S", list(range(2, 9)))
def test_small_kernels_match_oracle_bit_for_bit(S):
    """S <= 8: the general instantiation at every S (want_rr forces it at S = 2 and 3, where the samplers' calls take
    the lean ones), and at S = 2 / 3 the lean instantiations (grid-stride S = 2 tau-leap, corrector, Euler)."""
    nat = _nat()
    P = Problem(S, 13, 29, 60 + S, nat.IMPL_SIMT)
    cov = Coverage()
    hs = [2.0 ** -3, 2.0, 2.0 ** 5, 2.0 ** 10]
    for lean in ((False, True) if S <= 3 else (False,)):
        what = f"small S={S} {'lean' if lean else 'general'}"
        for hi, h in enumerate(hs):
            for m in ("tau", "corr"):
                off = 8 * hi + (m == "corr") + 1
                got, gst, _ = P.step(nat.MODE_TAU_LEAP_CORR if m == "corr" else nat.MODE_TAU_LEAP, h, off, want_rr=not lean)
                want, wst, margin, lam = P.tau_leap(m == "corr", h, off, False)
                _check(f"{what} {m} h={h}", got, gst, want, wst, margin)
                cov.add_jump(lam, P.x.reshape(-1), P.x.reshape(-1), ROW0, off, S, False)
            for m in ("euler", "euler_corr"):
                off = 100 + hi
                got, gst, _ = P.step(nat.MODE_EULER_CORR if m == "euler_corr" else nat.MODE_EULER, h, off, want_rr=not lean)
                want, wst, _ = P.euler(m == "euler_corr", h, off)
                _check(f"{what} {m} h={h}", got, gst, want, wst)
        if not lean:
            g = np.random.Generator(np.random.PCG64(S))
            xb = np.clip(P.x.reshape(-1) + g.integers(-1, 2, P.N * P.D), 0, S - 1)
            got, gst, _ = P.step(nat.MODE_MIDPOINT_JUMP, 2.0, 77, reject=True, x_base=xb.reshape(P.N, P.D), want_rr=True)
            want, wst, margin, _ = P.tau_leap(False, 2.0, 77, True, x_base=xb.reshape(P.N, P.D))
            _check(f"{what} mid_jump", got, gst, want, wst, margin)
            for h in (2.0 ** -2, 2.0):
                got, gst, _ = P.step(nat.MODE_MIDPOINT_DRIFT, h, 0, want_rr=True)
                want, wst, _ = P.drift(h)
                _check(f"{what} drift h={h}", got, gst, want, wst)
    assert cov.max_tot > 64.0 and cov.cap > 0, (cov.max_tot, cov.cap)


@pytest.mark.gpu
@pytest.mark.parametrize("path,S", [("tc", 256), ("block", 100), ("small", 2), ("small", 5)])
def test_rows_straddling_global_row_2_pow_32(path, S):
    """row_offset = 2^32 - 64: the launch's rows cross global row 2^32, so the Philox counters use their high row byte."""
    nat = _nat()
    impl = nat.IMPL_TC if path == "tc" else nat.IMPL_SIMT
    P = Problem(S, 4, 40, 90 + S, impl)
    row0 = 2 ** 32 - 64
    for off, h in ((1, 2.0 ** -2), (2, 2.0 ** 2)):
        got, gst, _ = P.step(nat.MODE_TAU_LEAP, h, off, row_offset=row0)
        want, wst, margin, _ = P.tau_leap(False, h, off, False, row_offset=row0)
        _check(f"{path} S={S} 2^32 h={h}", got, gst, want, wst, margin)
        if off == 1:      # (at the larger h every row of S = 2 jumps, whatever the draws)
            other, _, _ = P.step(nat.MODE_TAU_LEAP, h, off, row_offset=row0 + 2 ** 32)
            assert not np.array_equal(got, other)                   # the high row byte does change the draws
    got, gst, _ = P.step(nat.MODE_EULER, 2.0, 9, row_offset=row0)
    want, wst, _ = P.euler(False, 2.0, 9, row_offset=row0)
    _check(f"{path} S={S} 2^32 euler", got, gst, want, wst)


def teardown_module(module):
    print(f"\ncount ties tolerated in {__name__}: {sum(n for _, n in _ties_seen)} {_ties_seen}")
