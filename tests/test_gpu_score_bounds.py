"""The DP's two scoring shortcuts, tested item by item at their edges (kp_debug_self_score runs the same device functions
as kp_dp_rows_kernel / kp_dp_fiber_kernel):

- the score filter's float32 lower bound lb must satisfy lb <= s for the reference's float64 score s, or a pattern
  could be wrongly ruled out of being kept whole;
- kp_self_score_fast must decide RN_f32(s) and the "rounded up" bit exactly whenever it claims to, with
  |s~ - s| <= 2^-46 a + 2^-49 (M + U), and decline outside its window.

Whole DPs compared with the oracle rarely reach these edges: most patterns fail the filter by a wide margin.  Here the
inputs are built to sit on them: rates solved for exactly (beta = (M + alpha) / p - (M + U + alpha)) at every switch of
the two paths, counts around 2^24 and 2^32, extreme alpha / beta, penalties that cancel the log terms, and scores on
float32 rounding boundaries.
"""
import decimal

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EPS_A, EPS_C = 2.0 ** -46, 2.0 ** -49        # the bound kp_self_score_fast uses: eps = 2^-46 a + 2^-49 (M + U)
CLAIM_A, CLAIM_C = 2.0 ** -48, 2.0 ** -51    # the error its comment derives
ALPHAS = np.array([0.0, 1e-300, 1e-3, 0.8, 10.0, 1e4])
PENS = np.array([0.0, 1e-30, 0.5, 6.0, 1e6, 1e12, -0.5, -6.0])
COUNT_EDGES = np.array([0, 1, 2, 3, 7, 100, 12345] + [2 ** 24 + k for k in range(-8, 9)] +
                       [2 ** 31 - 1, 2 ** 31, 2 ** 31 + 1, 2 ** 32 - 2, 2 ** 32 - 1], dtype=np.int64)
WIDE_EDGES = np.array([2 ** 32, 2 ** 32 + 1, 2 ** 33 + 3, 2 ** 40, 2 ** 45 + 1, 2 ** 50], dtype=np.int64)
# switches of the two paths, as rates p: fast window top (also q = 1 - p at the near-1 edge of log), series switch,
# fast window bottom, the filter's series / __logf switch, p at the near-1 edge of log, p at the smallest normal,
# and where 1 - p rounds to 1
SWITCHES = np.array([2.0 ** -4, 2.0 ** -8, 2.0 ** -1000, 0.03125, 0.9375, 2.0 ** -1022, 2.0 ** -54, 2.0 ** -53])
N_PER_WIDTH = 1_500_000


def _totals(rng, n, wide):
    edges = np.concatenate([COUNT_EDGES, WIDE_EDGES]) if wide else COUNT_EDGES
    top = 50 if wide else 32
    T = np.where(rng.random(n) < 0.5, rng.choice(edges, n), np.exp2(rng.uniform(0, top, n)).astype(np.int64))
    return np.minimum(T, 2 ** 50 if wide else 2 ** 32 - 1)


def _target_rates(rng, n):
    p = np.exp2(rng.uniform(-1010, np.log2(0.999), n))
    near = rng.random(n) < 0.4
    s = rng.choice(SWITCHES, n)
    k = rng.integers(-64, 65, n).astype(np.float64)
    fl = (s == 0.03125) & (rng.random(n) < 0.5)    # the filter decides in float32: its ulps too
    ps = np.where(fl, s * (1.0 + k * 2.0 ** -23), s + k * np.spacing(s))
    return np.where(near, ps, p)


def _solve(rng, T, alpha, p):
    """(M, beta) with M + U = T and (M + alpha) / (T + alpha + beta) = p, beta in [0, 1e300]."""
    n = T.size
    g = np.where(rng.random(n) < 0.3, 1.0, 1.0 + 4.0 * rng.random(n))
    Tf = T.astype(np.float64)
    with np.errstate(over="ignore", invalid="ignore"):
        Mf = np.minimum(Tf, np.ceil(np.maximum(0.0, p * (Tf + alpha) - alpha) * g))
    M = np.nan_to_num(Mf).astype(np.int64)
    r = rng.random(n)
    M = np.where(r < 0.05, 0, np.where(r < 0.1, T, M))           # M = 0, U = 0
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        beta = (M + alpha) / p - (T.astype(np.float64) + alpha)
    beta = np.clip(np.nan_to_num(beta, nan=0.0, posinf=1e300), 0.0, 1e300)
    return M, beta


def _generate(rng, wide):
    """Items (M, U, alpha, beta, penalty, kind); kind: 0 random / switch rates, 1 den near 2^+-500, 2 cancelling
    penalty, 3 score on a float32 rounding boundary."""
    n = N_PER_WIDTH
    T = _totals(rng, n, wide)
    alpha = rng.choice(ALPHAS, n)
    M, beta = _solve(rng, T, alpha, _target_rates(rng, n))
    pen = rng.choice(PENS, n)
    kind = np.zeros(n, np.int8)
    # den = M + U + alpha + beta within a few ulps of 2^-500 (no counts) or 2^500 (huge beta)
    m = n // 20
    big = rng.random(m) < 0.5
    d0 = np.where(big, 2.0 ** 500, 2.0 ** -500)
    d0 = d0 + rng.integers(-64, 65, m) * np.spacing(d0)
    pr = np.exp2(rng.uniform(-30, -5, m))
    T[:m] = np.where(big, rng.choice(COUNT_EDGES[:8], m), 0)
    M[:m] = np.where(big, np.minimum(T[:m], rng.integers(0, 4, m)), 0)
    alpha[:m] = np.where(big, rng.choice(ALPHAS, m), d0 * pr)
    beta[:m] = np.where(big, d0, d0 - d0 * pr)
    kind[:m] = 1
    return M, T - M, alpha, beta, pen, kind


def _oracle_scores(oracle, M, U, alpha, beta, pen):
    out = np.empty(M.size)
    a = [np.ascontiguousarray(x, dtype=np.float64) for x in (alpha, beta, pen)]
    Mu, Uu = np.ascontiguousarray(M, dtype=np.uint64), np.ascontiguousarray(U, dtype=np.uint64)
    oracle.lib().kpo_self_score_array(a[0].ctypes.data, a[1].ctypes.data, a[2].ctypes.data, Mu.ctypes.data, Uu.ctypes.data,
                                      out.ctypes.data, M.size)
    return out


def _special_penalties(rng, oracle, M, U, alpha, beta, pen, kind):
    """Overwrite a slice of the items' penalties: -RN(s at pen 0) (1 + delta), and shifts that put s on a float32 value or
    within a few double ulps of a float32 midpoint (kp_self_score_fast's rounded-up bit and undecidable exit)."""
    n = M.size
    s0 = _oracle_scores(oracle, M, U, alpha, beta, np.zeros(n))
    ok = np.isfinite(s0) & (s0 > 0) & (s0 < 2.0 ** 100) & (kind == 0)
    idx = rng.permutation(np.flatnonzero(ok))
    c, r = idx[: n // 10], idx[n // 10: n // 4]
    # and every item with U = 0: there a = pen + t1 can be large against M + U, where the fast score's error is largest
    # relative to its bound
    r = np.union1d(r, np.setdiff1d(np.flatnonzero(ok & (U == 0)), c))
    delta = rng.choice([0.0, 1e-9, -1e-9, 1e-7, -1e-7, 1e-5, -1e-5, 1e-3, -1e-3, 2.0 ** -52, -2.0 ** -52, 2.0 ** -50], c.size)
    pen[c] = -s0[c] * (1.0 + delta)
    kind[c] = 2
    # the target: a float32 value just above s0, or up to 2^30 times s0 (the penalty then dominates a = pen + t1 + t2 and
    # the rounding of the final additions decides), or the midpoint above it; then exactly there or a few double ulps off
    up = np.where(rng.random(r.size) < 0.5, 1.0, np.exp2(rng.uniform(0, 30, r.size)))
    f = np.minimum(s0[r] * up, 2.0 ** 100).astype(np.float32)
    f = np.where(f.astype(np.float64) > s0[r], f, np.nextafter(f, np.float32(np.inf)))
    fd, fn = f.astype(np.float64), np.nextafter(f, np.float32(np.inf)).astype(np.float64)
    X = np.where(rng.random(r.size) < 0.5, fd, 0.5 * (fd + fn))
    X = X + np.where(rng.random(r.size) < 0.4, 0, rng.integers(-3, 4, r.size)) * np.spacing(X)
    pen[r] = X - s0[r]
    for _ in range(3):   # s = (pen + t1) + t2 rounds: walk pen until s lands on X
        s = _oracle_scores(oracle, M[r], U[r], alpha[r], beta[r], pen[r])
        pen[r] = np.maximum(0.0, pen[r] + (X - s))
    kind[r] = 3


def _split4(rng, x):
    """Per-base counts (n, 4) that sum to x: skewed shares, often some or all but one zero."""
    n = x.size
    w = rng.random((n, 4)) ** 3 * (rng.random((n, 4)) < 0.8)
    w[:, 0] += 1e-9
    w /= w.sum(axis=1, keepdims=True)
    parts = np.floor(x[:, None].astype(np.float64) * w[:, :3]).astype(np.int64)
    last = x - parts.sum(axis=1)
    bad = last < 0
    parts[bad] = 0
    last[bad] = x[bad]
    out = np.concatenate([parts, last[:, None]], axis=1)
    return np.take_along_axis(out, rng.permuted(np.tile(np.arange(4), (n, 1)), axis=1), axis=1)


def _device(M4, U4, alpha, beta, pen, wide):
    from kmerpapa_b200 import _native

    n = alpha.size
    r = dict(lb=np.empty(n, np.float32), ok=np.empty(n, np.uint8), sf=np.empty(n, np.float32), rup=np.empty(n, np.uint8),
             st=np.empty(n), exact=np.empty(n))
    args = [np.ascontiguousarray(x) for x in (M4, U4, alpha, beta, pen, wide.astype(np.uint8))]
    _native.check(_native.lib().kp_debug_self_score(0, *[a.ctypes.data for a in args], n, r["lb"].ctypes.data,
                                                    r["ok"].ctypes.data, r["sf"].ctypes.data, r["rup"].ctypes.data,
                                                    r["st"].ctypes.data, r["exact"].ctypes.data), "kp_debug_self_score")
    return r


def _first(what, mask, M, U, alpha, beta, pen, **cols):
    i = np.flatnonzero(mask)
    if i.size == 0:
        return None
    j = i[0]
    extra = ", ".join(f"{k}={v[j]!r}" for k, v in cols.items())
    return (f"{what}: {i.size} of {mask.size} items, first (M={M[j]}, U={U[j]}, alpha={alpha[j]!r}, beta={beta[j]!r}, "
            f"pen={pen[j]!r}, {extra})")


def _true_scores(M, U, alpha, beta, pen):
    """pen - 2M ln p - 2U ln(1 - p) at 50 digits from the exact values of the float64 inputs, and the error the
    reference's float64 evaluation may make (a few ulps of each term, plus the rounding of p and 1 - p)."""
    decimal.getcontext().prec = 50
    D = decimal.Decimal
    true, tol = np.empty(M.size), np.empty(M.size)
    u = 2.0 ** -53
    for i in range(M.size):
        m, uu = int(M[i]), int(U[i])
        p = (D(m) + D(alpha[i])) / (D(m + uu) + D(alpha[i]) + D(beta[i]))
        q = 1 - p
        t1 = -2 * m * p.ln() if m > 0 else D(0)
        t2 = -2 * uu * q.ln() if uu > 0 else D(0)
        true[i] = float(D(pen[i]) + t1 + t2)
        pf, qf = float(p), float(q)
        tol[i] = 8 * u * (abs(pen[i]) + float(t1) + float(t2)) + 2 * m * 5 * u + 2 * uu * u * (4 * pf / qf + 2)
    return true, tol


@pytest.mark.parametrize("wide", [False, True], ids=["narrow", "wide"])
def test_score_paths_at_their_edges(oracle, wide):
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    rng = np.random.default_rng(2024 + wide)
    M, U, alpha, beta, pen, kind = _generate(rng, wide)
    _special_penalties(rng, oracle, M, U, alpha, beta, pen, kind)
    M4, U4 = _split4(rng, M), _split4(rng, U)
    assert np.array_equal(M4.sum(axis=1), M) and np.array_equal(U4.sum(axis=1), U) and (M4 >= 0).all() and (U4 >= 0).all()
    d = _device(M4, U4, alpha, beta, pen, np.full(M.size, wide))
    s = _oracle_scores(oracle, M, U, alpha, beta, pen)
    T = (M + U).astype(np.float64)
    ok = d["ok"] == 1
    fails = []
    cols = dict(M=M, U=U, alpha=alpha, beta=beta, pen=pen)

    # (a) the exact path is the reference's score, bit for bit
    nan = np.isnan(s)
    fails.append(_first("(a) exact NaN-ness differs", np.isnan(d["exact"]) != nan, **cols, exact=d["exact"], s=s))
    fails.append(_first("(a) exact score differs", ~nan & (d["exact"].view(np.uint64) != s.view(np.uint64)), **cols,
                        exact=d["exact"], s=s))
    # (b) where the fast path decides, it decides right, within the error bound it uses
    with np.errstate(over="ignore", invalid="ignore"):
        sf_ref = s.astype(np.float32)
        err = np.abs(d["st"] - s)
    fails.append(_first("(b) fast sf != RN_f32(s)", ok & (d["sf"].view(np.uint32) != sf_ref.view(np.uint32)), **cols,
                        sf=d["sf"], s=s))
    fails.append(_first("(b) fast rounded-up bit wrong", ok & ((d["rup"] == 1) != (d["sf"].astype(np.float64) > s)), **cols,
                        sf=d["sf"], s=s))
    fails.append(_first("(b) |s~ - s| above 2^-46 a + 2^-49 (M + U)", ok & ~(err <= EPS_A * np.abs(s) + EPS_C * T), **cols,
                        st=d["st"], s=s))
    claim = err[ok] / (CLAIM_A * np.abs(s[ok]) + CLAIM_C * T[ok])
    print(f"wide={wide}: fast path decided {ok.sum()} of {ok.size}; largest |s~ - s| / (2^-48 a + 2^-51 (M + U)) = "
          f"{claim.max() if claim.size else 0.0:.3g}")
    # (c) it declines outside its window
    den = (T + alpha) + beta
    with np.errstate(invalid="ignore", divide="ignore"):
        p = (M + alpha) / den
    outside = ((pen < 0) | (p >= 2.0 ** -4 * (1 + 2.0 ** -40)) | (p < 2.0 ** -1000 * (1 - 2.0 ** -40)) | ~(den >= 2.0 ** -500)
               | ~(den < 2.0 ** 500) | ~(d["st"] < 2.0 ** 120))
    fails.append(_first("(c) fast path decided outside its window", ok & outside, **cols, p=p, den=den, st=d["st"]))
    # (d) the filter's bound is a lower bound (NaN: never skips)
    lbd = d["lb"].astype(np.float64)
    fails.append(_first("(d) filter lb > s", lbd > s, **cols, lb=d["lb"], s=s))
    # (e) inside the window the fast path almost never declines: only where s +- eps holds a float32 value or a midpoint
    # between two (s exactly on a float32 value, e.g. s = pen when M = 0 and 1 - p rounds to 1, is such a case)
    with np.errstate(over="ignore", invalid="ignore"):
        dist = np.abs(s - sf_ref.astype(np.float64))
        half = np.spacing(np.abs(sf_ref)).astype(np.float64) / 4    # half the smaller float32 spacing around sf
        eps2 = 2 * (EPS_A * np.abs(s) + EPS_C * T)
        decidable = (dist > eps2) & (dist < half - eps2)
    inside = ((kind == 0) & (pen >= 0) & (p < 2.0 ** -4 * (1 - 2.0 ** -40)) & (p >= 2.0 ** -1000 * (1 + 2.0 ** -40))
              & (den >= 2.0 ** -500) & (den < 2.0 ** 500) & (s > 0) & (s < 2.0 ** 119) & decidable)
    declined = (~ok & inside).sum() / max(inside.sum(), 1)
    print(f"wide={wide}: {inside.sum()} items inside the fast window, {declined:.2e} declined")
    if inside.sum() < N_PER_WIDTH // 20:
        fails.append(f"(e) only {inside.sum()} items inside the fast window")
    elif declined >= 1e-3:
        fails.append(f"(e) the fast path declined {declined:.2e} of {inside.sum()} items inside its window")

    # 50-digit cross-check of the oracle export, the exact path and the bound on a subsample
    sub = rng.choice(np.flatnonzero(np.isfinite(s) & (p > 0) & (p < 1)), 20_000, replace=False)
    true, tol = _true_scores(M[sub], U[sub], alpha[sub], beta[sub], pen[sub])
    sc = {k: v[sub] for k, v in cols.items()}
    fails.append(_first("oracle score far from the 50-digit score", ~(np.abs(s[sub] - true) <= tol), **sc, s=s[sub],
                        true=true, tol=tol))
    fails.append(_first("device exact score far from the 50-digit score", ~(np.abs(d["exact"][sub] - true) <= tol), **sc,
                        exact=d["exact"][sub], true=true))
    fails.append(_first("filter lb above the 50-digit score", lbd[sub] > true, **sc, lb=d["lb"][sub], true=true))

    fails = [f for f in fails if f]
    assert not fails, "\n".join(fails)


def test_level0_score_at_the_edges(oracle):
    """kp_debug_leaf_score (scipy's xlogy / xlog1py restated) against the oracle's level-0 score over the same edge
    generators: one launch per (alpha, beta, penalty) drawn from the edge items, over the edge counts plus that item."""
    import torch

    from kmerpapa_b200 import _native

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    rng = np.random.default_rng(77)
    M, U, alpha, beta, pen, kind = _generate(rng, True)
    _special_penalties(rng, oracle, M, U, alpha, beta, pen, kind)
    edges = np.concatenate([COUNT_EDGES, WIDE_EDGES])
    eM = np.concatenate([rng.choice(edges, 300), np.zeros(20, np.int64), rng.choice(edges, 20)])
    eU = np.concatenate([rng.choice(edges, 300), rng.choice(edges, 20), np.zeros(20, np.int64)])
    L, O = _native.lib(), oracle.lib()
    bad = []
    for i in rng.choice(M.size, 300, replace=False):
        Mi = np.ascontiguousarray(np.append(eM, M[i]), dtype=np.int64)
        Ui = np.ascontiguousarray(np.append(eU, U[i]), dtype=np.int64)
        out = np.empty(Mi.size)
        a, b, c = float(alpha[i]), float(beta[i]), float(pen[i])
        _native.check(L.kp_debug_leaf_score(0, Mi.ctypes.data, Ui.ctypes.data, Mi.size, a, b, c, out.ctypes.data),
                      "kp_debug_leaf_score")
        ref = np.array([O.kpo_leaf_score(a, b, c, int(x), int(y)) for x, y in zip(Mi, Ui)])
        same = (out.view(np.uint64) == ref.view(np.uint64)) | (np.isnan(out) & np.isnan(ref))
        bad += [(int(Mi[j]), int(Ui[j]), a, b, c, out[j], ref[j]) for j in np.flatnonzero(~same)]
    assert not bad, f"{len(bad)} level-0 scores differ, first (M, U, alpha, beta, pen, device, oracle) = {bad[:3]}"
