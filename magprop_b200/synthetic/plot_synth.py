"""Posterior summaries of a finished chain -- the numerical part of the reference's
``code/synthetic_datasets/plot_synth.py`` (``:150-223``); the plots themselves are out of scope.

``posterior_summary`` reproduces: pairwise correlation coefficients (``:150-157``), the 2.5/50/97.5
percentiles after un-logging columns 2.. (``:160-166``), the best-fit model at the data and on the
grid through the CUDA path (``:180,206``), reduced chi-square / AICc (``:181-191``) and the LaTeX
table row (``:193-203``).  Two reference defects are kept visible rather than silently changed:
the burn-in ``skip`` is computed but never applied (``:142-143``), and ``aicc`` is called with
(ymod, y) swapped (``:183``) -- symmetric in the statistic, so the value is the same."""
import math

import numpy as np

from ..magnetar.fit_stats import aicc, from_lnlike, redchisq
from .funcs import model_lum

NAMES = ["B", "P_i", "MdiscI", "RdiscI", "epsilon", "delta"]
PERCENTILES = (2.5, 50.0, 97.5)


def _latex_row(grb, trip, chisq_r):
    cells = " & ".join("$%s^{+%s}_{-%s}$" % t for t in trip)
    return "\n\n%s & %s & $%s$ \\\\ [2pt]" % (grb, cells, chisq_r)


def percentiles_from_order_statistics(n, select, unlog=False):
    """``np.percentile(col, PERCENTILES)`` (method "linear") of a column of n values, from its order statistics:
    ``select(ranks)`` returns the values at those 0-based ranks of the column sorted ascending, NaNs last.  With
    ``unlog`` the percentiles are those of ``10 ** col``, the two neighbouring values being un-logged before they are
    interpolated.  NumPy 2's rule is restated operation for operation -- q = p / 100, the virtual index (n-1)*q, its
    floor k and weight gamma, and the two-sided interpolation of ``_lerp`` -- so the result equals np.percentile's
    exactly (up to the sign of a zero: np.percentile takes it from wherever its partition leaves -0.0 and +0.0).  A
    column holding a NaN has NaN percentiles, as np.percentile gives."""
    rules = []
    for p in PERCENTILES:
        v = (n - 1) * (p / 100.0)
        if v >= n - 1:                          # NumPy takes the last value twice, gamma measured from index -1
            rules.append((n - 1, n - 1, v + 1.0))
        else:
            k = math.floor(v)
            rules.append((k, k + 1, v - k))
    ranks = sorted({r for k0, k1, _ in rules for r in (k0, k1)} | {n - 1})
    vals = dict(zip(ranks, select(ranks)))
    if np.isnan(vals[n - 1]):                   # NaNs sort last: rank n-1 is NaN iff the column holds one
        return [math.nan] * len(rules)
    out = []
    for k0, k1, gamma in rules:
        a, b = np.array([vals[k0], vals[k1]])
        if unlog:
            a, b = 10.0 ** np.array([a, b])     # the array power np.percentile's caller applies to the column
        d = b - a
        out.append(float(b - d * (1.0 - gamma) if gamma >= 0.5 else a + d * gamma))
    return out


def posterior_summary_device(chain, x, y, yerr, grb="", truths=None, n_burn=0):
    """``posterior_summary`` for a chain that is still on the GPU (``DeviceEnsemble.run(store=True)[0]``, any
    shape ``[..., Npars]``, a float64 CUDA tensor): the correlations and percentiles are reductions over the chain
    where it lies (``mp_chain_moments``, ``mp_chain_order_statistics``) and the fit statistics come from the
    likelihood kernel's chi-square -- a few dozen numbers cross PCIe instead of the chain.  The reductions run on
    torch's current stream.  The percentiles equal the host version's bit for bit (exact order statistics, un-logged
    and interpolated by NumPy's rule, ``percentiles_from_order_statistics``).  The correlations agree to the rounding
    of the covariance sums and are clipped to [-1, 1] as np.corrcoef clips them."""
    import torch

    from .. import _cache
    from .. import _capi as A
    from ..engine import chain_moments, chain_order_statistics
    from .mcmc_eqns import DEVICE
    flat = chain.reshape(-1, chain.shape[-1]).contiguous()
    n, Npars = flat.shape
    dev = flat.device.index or 0
    stream = torch.cuda.current_stream(flat.device).cuda_stream
    stats = {"Nburn": n_burn}
    _, cov = chain_moments(flat.data_ptr(), n, Npars, device=dev, stream=stream)
    sd = np.sqrt(np.diag(cov))
    stats["correlations"] = [float(np.clip(cov[i, j] / sd[i] / sd[j], -1.0, 1.0))     # np.corrcoef's operations
                             for i in range(Npars) for j in range(i + 1, Npars)]
    trip = []
    for col in range(Npars):
        out = percentiles_from_order_statistics(
            n, lambda ranks: chain_order_statistics(flat.data_ptr(), n, Npars, col, ranks, device=dev, stream=stream),
            unlog=col >= 2)                                                # out of log-space (plot_synth.py:160)
        trip.append((out[1], out[2] - out[1], out[1] - out[0]))
    pars = [t[0] for t in trip]
    stats["pars"] = {nm: tuple(float(v) for v in t) for nm, t in zip(NAMES, trip)}
    if truths is not None:
        stats["pars"]["truths"] = [float(v) for v in truths]
    # fit statistics of the median parameters from the kernel's chi-square (lnlike = -chi2/2)
    x, y, yerr = (np.asarray(a, float) for a in (x, y, yerr))
    lk = _cache.get(A.script_model_spec(unlog=False), None, x, y, yerr, device=DEVICE)
    lnl, status, _ = lk.lnprob(np.asarray(pars, float).reshape(1, -1), return_info=True)
    if status[0] & A.WALKER_INTEGRATOR_FAIL:
        raise RuntimeError("the median parameters flag in model_lum")
    chisq_r, aic = from_lnlike(lnl[0], y.size, Npars)
    stats["stats"] = {"aicc": float(aic), "chi_square_red": float(chisq_r)}
    stats["latex"] = _latex_row(grb, trip, stats["stats"]["chi_square_red"])
    return stats, pars


def posterior_summary(samples, x, y, yerr, grb="", truths=None, n_burn=0):
    samples = np.array(samples, dtype=np.float64)
    Npars = samples.shape[1]
    stats = {"Nburn": n_burn}
    corrs = []
    for i in range(Npars):
        for j in range(i + 1, Npars):
            corrs.append(float(np.corrcoef(samples[:, i], samples[:, j])[0, 1]))
    stats["correlations"] = corrs
    samples[:, 2:] = 10.0 ** samples[:, 2:]                          # out of log-space
    trip = [(v[1], v[2] - v[1], v[1] - v[0]) for v in zip(*np.percentile(samples, [2.5, 50.0, 97.5], axis=0))]
    pars = [t[0] for t in trip]
    stats["pars"] = {n: tuple(float(v) for v in t) for n, t in zip(NAMES, trip)}
    if truths is not None:
        stats["pars"]["truths"] = [float(v) for v in truths]
    ymod = model_lum(pars, xdata=x)
    if isinstance(ymod, str):
        raise RuntimeError("the median parameters flag in model_lum")
    y, yerr = np.asarray(y, float), np.asarray(yerr, float)
    stats["stats"] = {"aicc": float(aicc(ymod, y, yerr, Npars)),
                      "chi_square_red": float(redchisq(y, ymod, deg=Npars, sd=yerr))}
    stats["latex"] = _latex_row(grb, trip, stats["stats"]["chi_square_red"])
    fit = model_lum(pars)                                            # [t, Ltot, Lprop, Ldip] on the grid
    return stats, pars, ymod, fit
