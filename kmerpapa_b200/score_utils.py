"""Scalar score helpers of the host side (reference: src/kmerpapa/score_utils.py)."""
from scipy.special import xlog1py, xlogy


def get_betas(alpha, M, U):
    """beta per fold from the fold's train totals (score_utils.py:22-35): mu = M/(M+U), beta = alpha(1-mu)/mu."""
    mu = M / (M + U)
    return (alpha * (1.0 - mu)) / mu


def beta_from_totals(alpha, n_mut, n_unmut):
    """beta of the final fit (cli.py:261-262), plain Python floats."""
    mu = n_mut / (n_mut + n_unmut)
    return (alpha * (1.0 - mu)) / mu


def loss_from_terms(terms, penalty=0):
    """-2 * (sum of the per-pattern terms xlogy(M, p) + xlog1py(U, -p)) + penalty per pattern; float64, summed in
    order."""
    total, n = 0.0, 0
    for t in terms:
        total += t
        n += 1
    return -2 * total + n * penalty


def get_loss(counts, alpha, beta, penalty=0):
    """-2 log-likelihood (+ penalty per pattern) of a partition given (n_pos, n_neg) per pattern
    (score_utils.py:3-20); float64, summed in list order."""
    def terms():
        for n_pos, n_neg in counts:
            p = (n_pos + alpha) / (n_pos + n_neg + alpha + beta)
            yield xlogy(n_pos, p) + xlog1py(n_neg, -p)

    return loss_from_terms(terms(), penalty)
