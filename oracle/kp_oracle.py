"""ctypes front end of the CPU oracle (oracle/kp_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  Nothing under kmerpapa_b200/ imports this module.

The grid/selection logic restated here follows
/root/reference/src/kmerpapa/algorithms/bottum_up_array_penalty_plus_pseudo_CV.py:127-177 and
/root/reference/src/kmerpapa/CV_tools.py:5-62 (fold sampler, numpy RandomState stream).
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libkp_oracle.so")
_lib = None

CODE = {"A": "A", "C": "C", "G": "G", "T": "T", "R": "AG", "Y": "CT", "S": "GC", "W": "AT", "K": "GT",
        "M": "AC", "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG", "N": "ACGT"}


def build(force=False):
    """Compile oracle/kp_oracle.c -> oracle/_build/libkp_oracle.so (gcc, OpenMP)."""
    src = os.path.join(_HERE, "kp_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.run(["make", "-C", _HERE], check=True, stdout=subprocess.DEVNULL)
    return _SO


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        L = ctypes.CDLL(_SO)
        vp, i64, u64, dbl, cint = ctypes.c_void_p, ctypes.c_int64, ctypes.c_uint64, ctypes.c_double, ctypes.c_int
        L.kpo_log.restype = dbl
        L.kpo_log.argtypes = [dbl]
        L.kpo_log1p.restype = dbl
        L.kpo_log1p.argtypes = [dbl]
        L.kpo_log_mismatches.restype = i64
        L.kpo_log_mismatches.argtypes = [vp, i64]
        L.kpo_log_array.argtypes = [vp, vp, i64]
        L.kpo_log1p_array.argtypes = [vp, vp, i64]
        L.kpo_plan_info.argtypes = [ctypes.c_char_p, ctypes.POINTER(u64), ctypes.POINTER(u64), ctypes.POINTER(cint)]
        L.kpo_kmer_patnums.argtypes = [ctypes.c_char_p, vp]
        L.kpo_num2pattern.argtypes = [ctypes.c_char_p, u64, ctypes.c_char_p]
        L.kpo_leaf_score.restype = dbl
        L.kpo_leaf_score.argtypes = [dbl, dbl, dbl, u64, u64]
        L.kpo_self_score_array.argtypes = [vp, vp, vp, vp, vp, vp, i64]
        L.kpo_single_dp.argtypes = [ctypes.c_char_p, vp, vp, vp, dbl, dbl, dbl, vp, vp, vp, vp, cint]
        L.kpo_backtrack.restype = i64
        L.kpo_backtrack.argtypes = [ctypes.c_char_p, vp, vp, i64]
        L.kpo_cv_job.argtypes = [ctypes.c_char_p, vp, vp, vp, vp, vp, vp, dbl, dbl, dbl, vp, vp, cint]
        L.kpo_max_threads.restype = cint
        _lib = L
    return _lib


def plan_info(gen_pat):
    npat, nkmer, lvl = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_int()
    rc = lib().kpo_plan_info(gen_pat.encode(), ctypes.byref(npat), ctypes.byref(nkmer), ctypes.byref(lvl))
    if rc:
        raise ValueError(f"bad general pattern {gen_pat!r} (rc={rc})")
    return npat.value, nkmer.value, lvl.value


def kmers_of(gen_pat):
    """k-mers matched by gen_pat in k-mer index order (first position fastest)."""
    out = [""]
    for ch in reversed(gen_pat):
        out = [b + s for s in out for b in CODE[ch]]
    return out


def num2pattern(gen_pat, num):
    buf = ctypes.create_string_buffer(len(gen_pat) + 1)
    lib().kpo_num2pattern(gen_pat.encode(), int(num), buf)
    return buf.value.decode()


def kmer_patnums(gen_pat):
    _, nkmer, _ = plan_info(gen_pat)
    out = np.empty(nkmer, dtype=np.uint64)
    lib().kpo_kmer_patnums(gen_pat.encode(), out.ctypes.data)
    return out


def _u64(a):
    return np.ascontiguousarray(a, dtype=np.uint64)


def single_dp(gen_pat, kmerM, kmerU, alpha, beta, penalty, leaf_score=None, nthreads=0):
    """Full tables of one DP.  Returns dict(score f32[npat], M, U u64[npat], split u8[npat])."""
    npat, nkmer, _ = plan_info(gen_pat)
    kmerM, kmerU = _u64(kmerM), _u64(kmerU)
    assert kmerM.shape == (nkmer,) and kmerU.shape == (nkmer,)
    score = np.empty(npat, dtype=np.float32)
    M = np.empty(npat, dtype=np.uint64)
    U = np.empty(npat, dtype=np.uint64)
    split = np.empty(npat, dtype=np.uint8)
    ls = None
    if leaf_score is not None:
        ls = np.ascontiguousarray(leaf_score, dtype=np.float32)
    rc = lib().kpo_single_dp(gen_pat.encode(), kmerM.ctypes.data, kmerU.ctypes.data,
                             ls.ctypes.data if ls is not None else None,
                             float(alpha), float(beta), float(penalty),
                             score.ctypes.data, M.ctypes.data, U.ctypes.data, split.ctypes.data, int(nthreads))
    if rc:
        raise RuntimeError(f"kpo_single_dp rc={rc}")
    return {"score": score, "M": M, "U": U, "split": split}


def backtrack(gen_pat, split):
    cap = 1 << 16
    while True:
        out = np.empty(cap, dtype=np.uint64)
        n = lib().kpo_backtrack(gen_pat.encode(), split.ctypes.data, out.ctypes.data, cap)
        if n <= cap:
            return out[:n]
        cap = int(n)


def partition_names(gen_pat, split):
    return [num2pattern(gen_pat, p) for p in backtrack(gen_pat, split)]


def cv_job(gen_pat, kmerMtot, kmerUtot, kmerMte, kmerUte, alpha, beta, penalty, leaf=None, nthreads=0):
    """One (fold, alpha, penalty) job.  Returns (train f32[npat], test f32[npat])."""
    npat, nkmer, _ = plan_info(gen_pat)
    arrs = [_u64(a) for a in (kmerMtot, kmerUtot, kmerMte, kmerUte)]
    train = np.empty(npat, dtype=np.float32)
    test = np.empty(npat, dtype=np.float32)
    lt = lte = None
    if leaf is not None:
        lt = np.ascontiguousarray(leaf[0], dtype=np.float32)
        lte = np.ascontiguousarray(leaf[1], dtype=np.float32)
    rc = lib().kpo_cv_job(gen_pat.encode(), *[a.ctypes.data for a in arrs],
                          lt.ctypes.data if lt is not None else None, lte.ctypes.data if lte is not None else None,
                          float(alpha), float(beta), float(penalty), train.ctypes.data, test.ctypes.data, int(nthreads))
    if rc:
        raise RuntimeError(f"kpo_cv_job rc={rc}")
    return train, test


# ---------------------------------------------------------------------------------------------
# CV driver restated (host logic of _CV.py:127-177 and CV_tools.py:5-62)
# ---------------------------------------------------------------------------------------------
def sample_folds(gen_pat, kmerM, kmerU, nfolds, prng):
    """Held-out counts per fold, shape (nkmer, nfolds) each, drawn exactly like CV_tools.py:30-62:
    k-mers sorted as strings, colours = [all M..., all U...], nfolds-1 sequential multivariate
    hypergeometric draws of n//nfolds balls from numpy's legacy RandomState, last fold = remainder."""
    kmers = kmers_of(gen_pat)
    order = sorted(range(len(kmers)), key=lambda i: kmers[i])
    n = len(kmers)
    colors = np.empty(2 * n, dtype=np.uint64)
    for r, i in enumerate(order):
        colors[r] = kmerM[i]
        colors[n + r] = kmerU[i]
    total = int(colors.sum())
    n_samples = total // nfolds
    samples = np.empty((2 * n, nfolds), dtype=np.uint64)
    for f in range(nfolds - 1):
        remaining = np.cumsum(colors[::-1])[::-1]
        res = np.zeros(2 * n, dtype=np.uint64)
        m = n_samples
        for i in range(2 * n - 1):
            if m < 1:
                break
            res[i] = prng.hypergeometric(colors[i], remaining[i + 1], m)
            m -= res[i]
        res[-1] = m
        samples[:, f] = res
        colors -= res
    samples[:, nfolds - 1] = colors
    Mf = np.empty((n, nfolds), dtype=np.uint64)
    Uf = np.empty((n, nfolds), dtype=np.uint64)
    for r, i in enumerate(order):
        Mf[i] = samples[r]
        Uf[i] = samples[n + r]
    return Mf, Uf


def cv_grid(gen_pat, kmerM, kmerU, alphas, penalties, nfolds, seed, nthreads=0, folds=None):
    """Returns dict(rows=[(alpha, penalty, np.float32 test)], best=(alpha, penalty, test),
    per_job={(a_i,p_i): (train f32[nf], test f32[nf])}).  iterations == 1 only."""
    prng = np.random.RandomState(seed)
    if folds is None:
        Mf, Uf = sample_folds(gen_pat, kmerM, kmerU, nfolds, prng)
    else:
        Mf, Uf = folds
    npat, _, _ = plan_info(gen_pat)
    Mtot = Mf.sum(axis=1)
    Utot = Uf.sum(axis=1)
    M_sum_test = Mf.sum(axis=0)
    U_sum_test = Uf.sum(axis=0)
    M_sum_train = M_sum_test.sum() - M_sum_test
    U_sum_train = U_sum_test.sum() - U_sum_test
    per_job = {}
    for a_i, alpha in enumerate(alphas):
        my = M_sum_train / (M_sum_train + U_sum_train)
        betas = (alpha * (1.0 - my)) / my
        for p_i, penalty in enumerate(penalties):
            tr = np.empty(nfolds, dtype=np.float32)
            te = np.empty(nfolds, dtype=np.float32)
            for f in range(nfolds):
                train, test = cv_job(gen_pat, Mtot, Utot, Mf[:, f], Uf[:, f], alpha, betas[f], penalty, nthreads=nthreads)
                tr[f], te[f] = train[npat - 1], test[npat - 1]
            per_job[(a_i, p_i)] = (tr, te)
    rows, best, best_vals = [], 1e100, (None, None)
    for a_i, alpha in enumerate(alphas):
        for p_i, penalty in enumerate(penalties):
            test = sum(list(per_job[(a_i, p_i)][1])) / 1
            rows.append((alpha, penalty, test))
            if test < best:
                best_vals, best = (alpha, penalty), test
    return {"rows": rows, "best": (best_vals[0], best_vals[1], best), "per_job": per_job, "folds": (Mf, Uf)}


# ---------------------------------------------------------------------------------------------
# Greedy (top-down) partition: restatement of the reference's
# src/kmerpapa/algorithms/greedy_penalty_plus_pseudo.py:17-35 (train_loss, test_logLik) and :155-196
# (greedy_res_kmer_table_ord) in plain Python floats (math.log is the libm log numba calls).
# ---------------------------------------------------------------------------------------------
COMPLEMENTS = {"R": [("A", "G")], "Y": [("C", "T")], "S": [("G", "C")], "W": [("A", "T")], "K": [("G", "T")], "M": [("A", "C")],
               "V": [("A", "S"), ("C", "R"), ("G", "M")], "H": [("A", "Y"), ("C", "W"), ("T", "M")],
               "D": [("A", "K"), ("G", "W"), ("T", "R")], "B": [("C", "K"), ("G", "Y"), ("T", "S")],
               "N": [("S", "W"), ("K", "M"), ("R", "Y"), ("A", "B"), ("C", "D"), ("G", "H"), ("T", "V")]}


def _greedy_loss(M, U, alpha, beta, penalty):
    import math

    M, U = float(M), float(U)
    p = (M + alpha) / (M + U + alpha + beta)
    s = penalty
    if M > 0:
        s += -2.0 * M * math.log(p)
    if U > 0:
        s += -2.0 * U * math.log(1 - p)
    return s


def _greedy_test_ll(M, U, Mt, Ut, alpha, beta):
    import math

    M, U, Mt, Ut = float(M), float(U), float(Mt), float(Ut)
    p = (M + alpha) / (M + U + alpha + beta)
    s = 0.0
    if Mt > 0:
        s += -2.0 * Mt * math.log(p)
    if Ut > 0:
        s += -2.0 * Ut * math.log(1 - p)
    return s


def greedy(gen_pat, kmerM, kmerU, alpha, beta, penalty, testM=None, testU=None):
    """Returns (score, [patterns in the reference's order], [loss per pattern], [held-out LL per pattern] or None).
    kmerM/kmerU (and the held-out tables): counts in k-mer index order (kmers_of)."""
    index = {k: i for i, k in enumerate(kmers_of(gen_pat))}

    def counts(pattern, tabs):
        ks = [index[k] for k in kmers_of(pattern)]
        return [sum(int(t[i]) for i in ks) for t in tabs]

    tabs = [kmerM, kmerU] + ([testM, testU] if testM is not None else [])

    def rec(pattern):
        c = counts(pattern, tabs)
        best = _greedy_loss(c[0], c[1], alpha, beta, penalty)
        mine = (best, [pattern], [best], [_greedy_test_ll(c[0], c[1], c[2], c[3], alpha, beta)] if testM is not None else None)
        if all(ch in "ACGT" for ch in pattern):
            return mine
        choice = None
        for i, ch in enumerate(pattern):
            for c1, c2 in COMPLEMENTS.get(ch, []):
                p1, p2 = pattern[:i] + c1 + pattern[i + 1:], pattern[:i] + c2 + pattern[i + 1:]
                a, b = counts(p1, tabs[:2]), counts(p2, tabs[:2])
                s = _greedy_loss(a[0], a[1], alpha, beta, penalty) + _greedy_loss(b[0], b[1], alpha, beta, penalty)
                if s < best:
                    best, choice = s, (p1, p2)
        if choice is None:
            return mine
        s1, n1, l1, t1 = rec(choice[0])
        s2, n2, l2, t2 = rec(choice[1])
        return s1 + s2, n1 + n2, l1 + l2, (t1 + t2 if testM is not None else None)

    return rec(gen_pat)

