"""Convergence diagnostics of several chains' draws (Engine.run_chains)."""
import numpy as np


def split_rhat(draws):
    """Split-R-hat of Gelman et al., Bayesian Data Analysis (3rd ed.), section 11.4, per parameter.

    draws: array (chains, sweeps, m), or (chains, sweeps) for one parameter.  Each chain is cut into two halves (a middle
    draw of an odd count is dropped), and with W the mean within-half variance and B / S the variance of the half means,
    R-hat = sqrt(((S - 1) / S W + B / S) / W).  Values near 1 say the halves agree; well above 1 they have not mixed."""
    x = np.asarray(draws, dtype=np.float64)
    one = x.ndim == 2
    if one:
        x = x[:, :, None]
    if x.ndim != 3 or x.shape[1] < 4:
        raise ValueError("split_rhat: draws must have shape (chains, sweeps >= 4, m), got %s" % (np.shape(draws),))
    h = x.shape[1] // 2
    halves = np.concatenate([x[:, :h], x[:, x.shape[1] - h:]], axis=0)       # (2 chains, h, m)
    W = halves.var(axis=1, ddof=1).mean(axis=0)
    B_over_S = halves.mean(axis=1).var(axis=0, ddof=1)
    rhat = np.sqrt(((h - 1) / h * W + B_over_S) / W)
    return rhat[0] if one else rhat
