"""TEST INFRASTRUCTURE ONLY — CPU restatement of the device RNG maps (csrc/ctdd_common.cuh).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this
package; the product path (ctdd_b200) never does.

The reference (TAUnSDDM) draws with torch.poisson / Categorical.sample / torch.rand and sets no seeds, so
"identical inputs and injected uniforms" (BASELINE.json north_star) needs a shared uniform -> sample map.
This module defines that map with the fp32 roundings the CUDA kernels make (fused multiply-adds rounded once, like FFMA),
except where a device math function has no bit-exact host twin: expf in the Poisson pmf recurrence and in P(K >= 1)
(numpy's exp may differ by an ulp) and normcdfinvf in the Cornish-Fisher quantile (fp64 ndtri rounded to fp32 here: a
few ulps apart).  Those can move a jump count only when its uniform sits within ~1e-6 (relative rate) of a threshold;
poisson_count_margin finds such rows:

  * Philox4x32-10 (Salmon et al., SC'11; Random123 constants) keyed on (seed), counter =
    (state s | sub-index, global-row group, call offset, stream id);
  * tau-leap jump counts of one row (poisson_rows): the S independent Poisson(lam_s) counts are drawn through the
    superposition identity, chunk by chunk: the states are cut into chunks of 32 consecutive states (one warp of the
    tensor-path epilogue owns one chunk of a row); per chunk, total K ~ Poisson(sum of the chunk's lam_s) by upper-tail
    inverse CDF on the chunk's first uniform, then K categorical picks over lam_s / sum by inverse CDF on further
    uniforms of the same chunk — the same joint law as S independent draws (tests/test_rng_maps.py checks marginals
    and independence); chunks are independent of one another, so no warp waits for another warp's total;
    Philox call c of chunk q of row g: counter ((q << 16) + c, g, offset, STREAM_JUMP); word 0 of call 0 is the
    total's uniform, words 1..3 picks 0..2, call 1 + (j-3)//4 word (j-3)%4 pick j >= 3;
    state spaces of at most 8 states (one chunk; a row is only 4*S + 8 bytes, so a Philox call per row would be the
    whole cost of the step): the total's uniform of row g is instead word g & 3 of the call
    (0, g >> 2, offset, STREAM_JUMP_COUNT) shared by 4 consecutive rows, like the per-row uniforms below; the picks
    (rare) still come from the row's own STREAM_JUMP calls, words 1..3 of call 0 first;
  * per-row uniforms (Euler, initial state, noising): one call serves 4 consecutive rows (word row & 3);
  * v = (word + 0.5) * 2^-32 in fp32; Poisson by upper-tail inverse CDF; categorical by sequential fp32 cumsum.
"""
from __future__ import annotations

import numpy as np

STREAM_JUMP = 0       # per-row tau-leap draws (total count + picks)
STREAM_JUMP_COUNT = 1  # S <= JUMP_SHARED_MAX_S: the total count's uniform, one call per 4 consecutive rows
JUMP_SHARED_MAX_S = 8
JUMP_PICK_CAP = 4096  # picks evaluated per chunk of a row (rows whose total exceeds it are clamp-saturated anyway)
JUMP_CHUNK = 32       # consecutive states that share one superposition draw (one warp of the tensor-path epilogue)
STREAM_ROW = 2
STREAM_INIT = 3
STREAM_NOISE_XT = 4
STREAM_TILDE_DIM = 5
STREAM_TILDE_VAL = 6

_M0 = np.uint64(0xD2511F53)
_M1 = np.uint64(0xCD9E8D57)
_W0 = 0x9E3779B9
_W1 = 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0: int, k1: int):
    """Vectorised Philox4x32-10. c* are broadcastable uint32 arrays; returns 4 uint32 arrays."""
    c0, c1, c2, c3 = np.broadcast_arrays(
        np.asarray(c0, dtype=np.uint64), np.asarray(c1, dtype=np.uint64),
        np.asarray(c2, dtype=np.uint64), np.asarray(c3, dtype=np.uint64))
    c0, c1, c2, c3 = c0 & _MASK, c1 & _MASK, c2 & _MASK, c3 & _MASK
    k0 &= 0xFFFFFFFF
    k1 &= 0xFFFFFFFF
    for _ in range(10):
        p0 = _M0 * c0
        p1 = _M1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK
        n0 = hi1 ^ c1 ^ np.uint64(k0)
        n2 = hi0 ^ c3 ^ np.uint64(k1)
        c0, c1, c2, c3 = n0, lo1, n2, lo0
        k0 = (k0 + _W0) & 0xFFFFFFFF
        k1 = (k1 + _W1) & 0xFFFFFFFF
    return (c0.astype(np.uint32), c1.astype(np.uint32), c2.astype(np.uint32), c3.astype(np.uint32))


def _c3(stream: int, offset: int, hi_bits):
    return (np.uint64(stream) | (np.uint64((offset >> 32) & 0xFFFF) << np.uint64(8))
            | ((np.asarray(hi_bits, dtype=np.uint64) & np.uint64(0xFF)) << np.uint64(24)))


def u32_to_unit(word: np.ndarray) -> np.ndarray:
    """(word + 0.5) * 2^-32 in fp32 with a single rounding (device: I2F.RN then FFMA)."""
    f = word.astype(np.uint32).astype(np.float32)  # round-to-nearest-even, like cvt.rn.f32.u32
    return (f.astype(np.float64) * 2.0 ** -32 + 2.0 ** -33).astype(np.float32)


def rowjump_words(grow: np.ndarray, offset: int, seed: int, call) -> np.ndarray:
    """uint32 (len(grow), 4): Philox call `call` (scalar or per-row array) of the tau-leap stream of global rows grow."""
    grow = np.asarray(grow, dtype=np.uint64)
    w = philox4x32_10(np.asarray(call, dtype=np.uint64), grow & _MASK, np.uint64(offset & 0xFFFFFFFF),
                      _c3(STREAM_JUMP, offset, grow >> np.uint64(32)), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return np.stack(w, axis=-1)


def rowjump_total_unit(rows: int, row_offset: int, offset: int, seed: int) -> np.ndarray:
    """fp32 (rows,): the uniform that decides the total jump count of chunk 0 of a row with more than 8 states."""
    grow = np.arange(rows, dtype=np.uint64) + np.uint64(row_offset)
    return u32_to_unit(rowjump_words(grow, offset, seed, 0)[:, 0])


def rowjump_pick_units(grow: np.ndarray, offset: int, seed: int, npicks: int, call_base: int = 0) -> np.ndarray:
    """fp32 (len(grow), npicks): pick uniforms j = 0..npicks-1 of the given global rows (chunk with Philox call base call_base)."""
    grow = np.asarray(grow, dtype=np.uint64)
    out = np.empty((grow.shape[0], npicks), dtype=np.float32)
    first = rowjump_words(grow, offset, seed, call_base)
    for j in range(min(3, npicks)):
        out[:, j] = u32_to_unit(first[:, 1 + j])
    for c in range(1, 1 + (max(npicks - 3, 0) + 3) // 4):
        w = rowjump_words(grow, offset, seed, call_base + c)
        for i in range(4):
            j = 3 + 4 * (c - 1) + i
            if j < npicks:
                out[:, j] = u32_to_unit(w[:, i])
    return out


def row_units(rows: int, row_offset: int, offset: int, stream: int, seed: int, sub: int = 0) -> np.ndarray:
    """fp32 (rows,) per-row uniforms v in (0, 1]."""
    return row_units_at(np.arange(rows, dtype=np.uint64) + np.uint64(row_offset), offset, stream, seed, sub)


def row_units_at(grow: np.ndarray, offset: int, stream: int, seed: int, sub: int = 0) -> np.ndarray:
    """fp32 (len(grow),) per-row uniforms of the given global rows: word grow & 3 of the call of row group grow >> 2."""
    grow = np.asarray(grow, dtype=np.uint64)
    rows = grow.shape[0]
    w = philox4x32_10(np.uint64(sub), (grow >> np.uint64(2)) & _MASK, np.uint64(offset & 0xFFFFFFFF),
                      _c3(stream, offset, grow >> np.uint64(34)), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    words = np.stack(w, axis=-1)
    return u32_to_unit(words[np.arange(rows), (grow & np.uint64(3)).astype(np.int64)])


def _fma32(a, b, c):
    """fp32 fused multiply-add (device FFMA): a * b + c rounded once to nearest even.

    The product of two fp32 values is exact in fp64; the fp64 sum may round, and rounding that sum again to fp32 is
    wrong only when the fp64 sum lands exactly halfway between two fp32 values: then the sign of the exact residual of
    the sum (two-sum) decides."""
    a, b, c = np.broadcast_arrays(np.asarray(a, np.float32).astype(np.float64), np.asarray(b, np.float32).astype(np.float64),
                                  np.asarray(c, np.float32).astype(np.float64))
    p = a * b
    s = p + c
    bv = s - p
    err = (p - (s - bv)) + (c - bv)           # p + c == s + err exactly
    with np.errstate(over="ignore", invalid="ignore"):
        r = s.astype(np.float32)
        up = s > r.astype(np.float64)
        nxt = np.nextafter(r, np.where(up, np.float32(np.inf), np.float32(-np.inf)).astype(np.float32))
        mid = (r.astype(np.float64) + nxt.astype(np.float64)) * 0.5
        tie = (s != r.astype(np.float64)) & (s == mid) & (err != 0)
        beyond = np.where(up, err > 0, err < 0)        # the exact value lies past the midpoint, towards nxt
    return np.where(tie & beyond, nxt, r).astype(np.float32)


def poisson_sf0(lam: np.ndarray) -> np.ndarray:
    """P(K >= 1), fp32: 3-term series below 2^-6, else 1 - exp(-lam)."""
    lam = lam.astype(np.float32)
    t = _fma32(lam, np.float32(-0.16666667), np.float32(0.5))
    u = _fma32(-lam, t, np.float32(1.0))
    small = (lam * u).astype(np.float32)
    with np.errstate(over="ignore", under="ignore"):
        big = (np.float32(1.0) - np.exp(-lam).astype(np.float32)).astype(np.float32)
    return np.where(lam < np.float32(0.015625), small, big)


def _cornish_fisher(lam: np.ndarray, v: np.ndarray):
    """lam > 64: (z, f) of the device's Cornish-Fisher quantile f = lam + sqrt(lam) z + (z^2 - 1) / 6, z the upper-tail
    normal quantile of v, all fp32.  The device evaluates f as three fused multiply-adds (each rounded once):
    t = fma(sqrtf(lam), z, lam), u = fma(z, z, -1), f = fma(u, 0.16666667, t).  Its z comes from normcdfinvf, this one
    from fp64 ndtri rounded to fp32: the two may differ by a few ulps of z (poisson_rows_margin allows for it)."""
    from scipy.special import ndtri
    lb = np.minimum(np.asarray(lam, np.float32), np.float32(1.0e9))
    z = (-ndtri(np.asarray(v, np.float32).astype(np.float64))).astype(np.float32)
    t = _fma32(np.sqrt(lb).astype(np.float32), z, lb)
    u = _fma32(z, z, np.float32(-1.0))
    return z, _fma32(u, np.float32(0.16666667), t)


def poisson_from_unit(lam: np.ndarray, v: np.ndarray) -> np.ndarray:
    """Upper-tail inverse CDF  k = #{j >= 0 : v < P(K > j)}  (int64), with the device's fp32 roundings: lam <= 64 the
    pmf recurrence in the device's op order (exp may differ from the device's expf by an ulp); lam > 64 the
    Cornish-Fisher quantile of _cornish_fisher (z may differ by a few ulps)."""
    lam = np.asarray(lam, dtype=np.float32)
    v = np.asarray(v, dtype=np.float32)
    k = np.zeros(lam.shape, dtype=np.int64)
    pos = lam > 0
    sf = poisson_sf0(np.where(pos, lam, np.float32(1.0)))
    act = pos & (v < sf)
    idx = np.flatnonzero(act)
    if idx.size == 0:
        return k
    l = lam.ravel()[idx]
    vv = v.ravel()[idx]
    s = sf.ravel()[idx].copy()
    out = np.ones(idx.size, dtype=np.int64)
    small = l <= np.float32(64.0)
    # exact recurrence
    si = np.flatnonzero(small)
    if si.size:
        ls, vs, ss = l[si], vv[si], s[si]
        with np.errstate(under="ignore"):
            p = np.exp(-ls).astype(np.float32)
        kmax = (ls + np.float32(10.0) * np.sqrt(ls).astype(np.float32) + np.float32(12.0)).astype(np.float32).astype(np.int64)
        kk = np.ones(si.size, dtype=np.int64)
        live = kk < kmax
        while live.any():
            p = np.where(live, ((p * ls).astype(np.float32) / kk.astype(np.float32)).astype(np.float32), p)
            ss = np.where(live, (ss - p).astype(np.float32), ss)
            stop = live & (vs >= ss)
            live = live & ~stop
            kk = np.where(live, kk + 1, kk)
            live = live & (kk < kmax)
        out[si] = kk
    bi = np.flatnonzero(~small)
    if bi.size:
        _, kf = _cornish_fisher(l[bi], vv[bi])
        kf = np.rint(kf)
        kf = np.where(kf > 1.0, kf, 1.0)
        kf = np.minimum(kf, 2.0e9)
        out[bi] = kf.astype(np.int64)
    k.ravel()[idx] = out
    return k


def inv_cdf(weights: np.ndarray, v: np.ndarray) -> np.ndarray:
    """Row-wise categorical draw: first index with sequential-fp32 cumsum > v * total.

    weights (rows, n) fp32 unnormalised; v (rows,) in (0,1]. Falls back to the last positive weight.
    """
    w = np.asarray(weights, dtype=np.float32)
    cum = np.cumsum(w, axis=1, dtype=np.float32)  # sequential accumulation in fp32
    tot = cum[:, -1]
    target = (np.minimum(np.asarray(v, np.float32), np.float32(0.99999994)) * tot).astype(np.float32)
    gt = cum > target[:, None]
    first = gt.argmax(axis=1)
    none = ~gt.any(axis=1)
    if none.any():
        posw = w > 0
        last = np.where(posw.any(axis=1), w.shape[1] - 1 - posw[:, ::-1].argmax(axis=1), 0)
        first = np.where(none, last, first)
    return first.astype(np.int64)


def count_units(grow: np.ndarray, offset: int, seed: int, call_base: int, shared: bool) -> np.ndarray:
    """fp32 (len(grow),): the uniform that decides a chunk's total jump count (module docstring)."""
    if shared:
        return row_units_at(grow, offset, STREAM_JUMP_COUNT, seed)
    return u32_to_unit(rowjump_words(grow, offset, seed, call_base)[:, 0])


def _poisson_chunk(lam: np.ndarray, grow: np.ndarray, call_base: int, offset: int, seed: int, shared: bool = False):
    """One chunk of states of poisson_rows: (counts (rows, n) int64, K (rows,) int64); Philox calls call_base + c."""
    rows, n = lam.shape
    cum = np.cumsum(lam, axis=1, dtype=np.float32)
    tot = cum[:, -1]
    v0 = count_units(grow, offset, seed, call_base, shared)
    K = poisson_from_unit(tot, v0)
    counts = np.zeros((rows, n), dtype=np.int64)
    idx = np.flatnonzero(K > 0)
    if idx.size == 0:
        return counts, K
    Kc = np.minimum(K[idx], JUMP_PICK_CAP)
    kmax = int(Kc.max())
    picks = rowjump_pick_units(grow[idx], offset, seed, kmax, call_base)
    w = lam[idx]
    c = cum[idx]
    t = tot[idx]
    posw = w > 0
    last = np.where(posw.any(axis=1), n - 1 - posw[:, ::-1].argmax(axis=1), 0)
    for j in range(kmax):
        live = Kc > j
        if not live.any():
            break
        target = (np.minimum(picks[:, j], np.float32(0.99999994)) * t).astype(np.float32)
        gt = c > target[:, None]
        s_j = np.where(gt.any(axis=1), gt.argmax(axis=1), last)
        li = np.flatnonzero(live)
        np.add.at(counts, (idx[li], s_j[li]), 1)
    return counts, K


def poisson_rows(lam: np.ndarray, row_offset: int, offset: int, seed: int):
    """Jump counts k[r, s] ~ independent Poisson(lam[r, s]) through the chunked superposition map (module docstring).

    lam (rows, S) fp32 >= 0. Returns (counts (rows, S) int64, total (rows,) int64); counts.sum(1) == sum over the
    chunks of min(K_chunk, cap).  The S states are cut into chunks of JUMP_CHUNK = 32 consecutive states; every chunk
    is an independent superposition draw.  Op order of the CUDA-core kernels: sequential fp32 cumsum over the chunk's
    states, total = last cumsum entry, K = poisson_from_unit(total, v0) (module docstring: expf / normcdfinvf are the
    only host-device differences), pick j = first s with cum[s] > min(v_j, 1 - 2^-24) * total; Philox call index of
    chunk c = (c << 16) + call.
    """
    lam = np.ascontiguousarray(lam, dtype=np.float32)
    rows, S = lam.shape
    grow = np.arange(rows, dtype=np.uint64) + np.uint64(row_offset)
    counts = np.zeros((rows, S), dtype=np.int64)
    K = np.zeros(rows, dtype=np.int64)
    for ci, c0 in enumerate(range(0, S, JUMP_CHUNK)):
        c1 = min(c0 + JUMP_CHUNK, S)
        kc, Kc = _poisson_chunk(lam[:, c0:c1], grow, ci << 16, offset, seed, shared=S <= JUMP_SHARED_MAX_S)
        counts[:, c0:c1] = kc
        K += Kc
    return counts, K


# ------------------------------------------------------------------------------------------------------
# tie margins: how close the deciding uniforms of a row sit to a threshold of the maps above.  The tensor path
# computes the rates with ~3e-5 relative error and sums them in a different order than this module, so it may
# legitimately decide differently ONLY when a uniform sits within the rate tolerance of a threshold
# (BASELINE.json north_star: "bit-exact except where the reference rate sits within ... of a Poisson threshold").
# The parity tests assert that every mismatching row has a margin below the rate tolerance.


CF_Z_ULPS = 8   # normcdfinvf (device) against ndtri rounded to fp32 (oracle): a few ulps of z apart


def poisson_count_margin(tot: np.ndarray, v0: np.ndarray) -> np.ndarray:
    """fp64: smallest RELATIVE change of the rate total `tot` (fp32) that would move K = poisson_from_unit(tot, v0).

    tot <= 64 (exact pmf recurrence): v0 against the two neighbouring thresholds P(K > j), j in {K-1, K}; a relative
    change d of tot moves P(K > j) by pmf(j) * tot * d, so the margin is |v0 - P(K > j)| / (pmf(j) * tot).
    tot > 64 (Cornish-Fisher): K = rint(f), f = tot + sqrt(tot) z + (z^2 - 1)/6 (_cornish_fisher), so K moves when f
    crosses K -+ 1/2 (only K + 1/2 when K = 1 is the clamp); a relative change d moves f by
    tot (1 + z / (2 sqrt(tot))) d.  The distance is first reduced by what CF_Z_ULPS ulps of z move f, so a row the two
    quantile functions may decide differently has margin 0.  inf where tot <= 0."""
    from scipy.stats import poisson as sp
    tot = np.asarray(tot, np.float32)
    v0 = np.asarray(v0, np.float32)
    K = poisson_from_unit(tot, v0)
    t = np.where(tot > 0, tot, np.float32(1.0)).astype(np.float64)
    v = v0.astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore", under="ignore"):
        m = np.abs(v - sp.sf(K, t)) / np.maximum(sp.pmf(K, t) * t, 1e-300)
        m1 = np.abs(v - sp.sf(K - 1, t)) / np.maximum(sp.pmf(np.maximum(K - 1, 0), t) * t, 1e-300)
    m = np.where(K >= 1, np.minimum(m, m1), m)
    big = (tot > np.float32(64.0)) & (v0 < poisson_sf0(np.where(tot > 0, tot, np.float32(1.0))))
    if big.any():
        z, f = _cornish_fisher(tot[big], v0[big])
        z64, f64, t64, Kb = z.astype(np.float64), f.astype(np.float64), t[big], K[big]
        dist = np.abs(f64 - (Kb + 0.5))
        dist = np.where(Kb > 1, np.minimum(dist, np.abs(f64 - (Kb - 0.5))), dist)
        dz = CF_Z_ULPS * np.spacing(np.abs(z)).astype(np.float64)
        slack = (np.sqrt(t64) + np.abs(z64) / 3.0) * dz + np.spacing(np.abs(f)).astype(np.float64)
        slope = np.maximum(t64 * (1.0 + z64 / (2.0 * np.sqrt(t64))), 1e-300)
        m[big] = np.maximum(dist - slack, 0.0) / slope
    return np.where(tot > 0, m, np.inf)


def poisson_rows_margin(lam: np.ndarray, row_offset: int, offset: int, seed: int, picks: bool = True) -> np.ndarray:
    """fp64 (rows,): smallest RELATIVE rate change that would move a decision of poisson_rows on that row.

    Per chunk: (a) the count (poisson_count_margin of the chunk total); (b) with `picks`, every pick:
    |v_j * total - cum[s]| / total for the two prefix sums around the chosen state.  inf when the row has no positive
    rate."""
    lam = np.ascontiguousarray(lam, dtype=np.float32)
    rows, S = lam.shape
    grow = np.arange(rows, dtype=np.uint64) + np.uint64(row_offset)
    margin = np.full(rows, np.inf)
    for ci, c0 in enumerate(range(0, S, JUMP_CHUNK)):
        w = lam[:, c0:min(c0 + JUMP_CHUNK, S)]
        cum = np.cumsum(w, axis=1, dtype=np.float32).astype(np.float64)
        tot = cum[:, -1]
        v0 = count_units(grow, offset, seed, ci << 16, S <= JUMP_SHARED_MAX_S)
        K = poisson_from_unit(tot.astype(np.float32), v0)
        margin = np.minimum(margin, poisson_count_margin(tot.astype(np.float32), v0))
        idx = np.flatnonzero(K > 0)
        if idx.size == 0 or not picks:
            continue
        Kc = np.minimum(K[idx], JUMP_PICK_CAP)
        kmax = int(Kc.max())
        pu = rowjump_pick_units(grow[idx], offset, seed, kmax, ci << 16).astype(np.float64)
        c = cum[idx]
        for j in range(kmax):
            live = np.flatnonzero(Kc > j)
            if live.size == 0:
                break
            target = np.minimum(pu[live, j], 0.99999994) * tot[idx[live]]
            d = np.abs(c[live] - target[:, None]).min(axis=1) / tot[idx[live]]
            margin[idx[live]] = np.minimum(margin[idx[live]], d)
    return margin


def inv_cdf_margin(weights: np.ndarray, v: np.ndarray) -> np.ndarray:
    """fp64 (rows,): distance of v * total to the nearest cumulative sum, relative to the total (inv_cdf's tie margin)."""
    w = np.asarray(weights, dtype=np.float32)
    cum = np.cumsum(w, axis=1, dtype=np.float32).astype(np.float64)
    tot = cum[:, -1]
    target = np.minimum(np.asarray(v, np.float64), 0.99999994) * tot
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(tot > 0, np.abs(cum - target[:, None]).min(axis=1) / np.where(tot > 0, tot, 1.0), np.inf)
