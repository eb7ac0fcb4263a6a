"""The greedy (top-down) pattern partition and its grid-search cross validation, on the GPU.

Drop-in for the parts of the reference's src/kmerpapa/algorithms/greedy_penalty_plus_pseudo.py that cli.py uses
(`greedy_partition` :285-300, called from cli.py:276; `GridSearchCV` :340-355 with `CrossValidation` :303-337,
called from cli.py:224-225 for --greedy / --greedyCV): same names, arguments and return values.  The recursion
(greedy_res_kmer_table_ord, :155-196) runs as a breadth-first sweep of kp_greedy: one launch per depth, one CTA per
pattern, float64 losses with the reference's rounding, leaves returned in the reference's depth-first order.
`BaysianOptimizationCV` needs scikit-optimize, which this build does not depend on.
"""
import ctypes

import numpy as np

from .. import CV_tools, iupac
from .._native import KpError
from ..engine import _torch, get_plan, grow_capacity
from ..score_utils import get_betas


def _kmer_table(genpat, contextD):
    kmers = iupac.matches(genpat)
    table = np.zeros((len(kmers), 2), dtype=np.uint64)
    for i, context in enumerate(kmers):
        table[i, 0], table[i, 1] = contextD[context][0], contextD[context][1]
    return kmers, table


def _greedy(plan, kM, kU, alpha, beta, penalty, test=None, cap=65536):
    """(pattern numbers in the reference's order, float64 losses, float64 held-out LLs or None, float64 score)."""
    torch = _torch()

    def run(cap):
        ws = plan._buffer("greedy_ws", int(plan.lib.kp_greedy_ws_bytes(cap)), torch.uint8)
        pats = np.empty(cap, dtype=np.uint64)
        loss = np.empty(cap, dtype=np.float64)
        tst = np.empty(cap, dtype=np.float64)
        n, total = ctypes.c_uint64(0), ctypes.c_double(0.0)
        rc = plan.lib.kp_greedy(plan.handle, kM.data_ptr(), kU.data_ptr(), test[0].data_ptr() if test else None,
                                test[1].data_ptr() if test else None, float(alpha), float(beta), float(penalty), ws.data_ptr(),
                                cap, pats.ctypes.data, loss.ctypes.data, tst.ctypes.data, ctypes.byref(n), ctypes.byref(total),
                                plan._stream())
        return rc, (pats, loss, tst, n.value, total.value)

    pats, loss, tst, k, total = grow_capacity(plan.lib, "kp_greedy", cap, 1 << 24, run)
    return pats[:k].copy(), loss[:k].copy(), (tst[:k].copy() if test else None), total


def greedy_partition(genpat, contextD, alpha, beta, penalty, args):
    """Returns (score, n_pos, n_neg, patterns).  Like the reference, beta is recomputed from the table's totals."""
    kmers, table = _kmer_table(genpat, contextD)
    MU = table.sum(axis=0)
    beta = get_betas(alpha, MU[0], MU[1])
    plan = get_plan(genpat, lite=True)
    kM, kU = plan.upload_kmer_tables(table[:, 0], table[:, 1], name="greedy_k")
    pats, _, _, score = _greedy(plan, kM, kU, alpha, beta, penalty)
    PE = iupac.PatternEnumeration(genpat)
    return score, MU[0], MU[1], [PE.num2pattern(p) for p in pats]


class CrossValidation:
    def __init__(self, genpat, contextD, nfolds=2, nit=1, seed=None, verbosity=1):
        self.nfolds, self.nit, self.seed, self.genpat = nfolds, nit, seed, genpat
        _, self.kmer_table = _kmer_table(genpat, contextD)
        prng = np.random.RandomState(seed)
        self.fold_kmer_table = CV_tools.make_all_folds(self.kmer_table, nfolds, nit, prng)
        self.plan = get_plan(genpat, lite=True)

    def loglik(self, alpha, penalty):
        """Mean over the repeats of the summed held-out -2 log-likelihood of the greedy partitions of the train folds."""
        ll_list = []
        for repeat in range(self.nit):
            test_ll = 0.0
            for fold in range(self.nfolds):
                held = self.fold_kmer_table[repeat][fold]
                train = self.kmer_table - held
                train_MU = train.sum(axis=0)
                beta = get_betas(alpha, train_MU[0], train_MU[1])
                kM, kU = self.plan.upload_kmer_tables(train[:, 0], train[:, 1], name="greedy_tr")
                tM, tU = self.plan.upload_kmer_tables(held[:, 0], held[:, 1], name="greedy_te")
                _, _, tst, _ = _greedy(self.plan, kM, kU, alpha, beta, penalty, test=(tM, tU))
                for this_ll in tst:        # sequential float64 sum over the leaves in the reference's order
                    test_ll += float(this_ll)
            ll_list.append(test_ll)
        return sum(ll_list) / len(ll_list)


class GridSearchCV(CrossValidation):
    def __init__(self, genpat, contextD, penalties, pseudo_counts, nfolds=2, nit=1, seed=None, verbosity=1):
        super().__init__(genpat, contextD, nfolds=nfolds, nit=nit, seed=seed)
        self.penalties, self.pseudo_counts = penalties, pseudo_counts

    def get_best_a_c(self):
        best_combo, best_ll = (None, None), 1e100
        for a in self.pseudo_counts:
            for c in self.penalties:
                ll = self.loglik(a, c)
                if ll < best_ll:
                    best_ll, best_combo = ll, (a, c)
        return best_combo + (best_ll,)


class BaysianOptimizationCV(CrossValidation):
    def __init__(self, *a, **k):
        raise KpError("--BayesOpt needs scikit-optimize (skopt), which is not part of this build")
