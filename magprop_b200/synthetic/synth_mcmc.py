"""The MCMC driver around the likelihood -- what the reference's
``code/synthetic_datasets/synth_mcmc.py`` does with emcee, on the device-resident ensemble.

    res = run("Humped", x, y, yerr, n_walk=50, n_step=500, seed=1)      # fused stretch move on the GPU
    write_outputs(dirname, "Humped", res)                                # the reference's file set

Covered (SURVEY.md section 8, row f1): initial ball (``synth_mcmc.py:175-176``), the sampler run
(``:178-185``), ``{GRB}_chain.csv`` with its ``Npars, Nwalk, Nstep`` header (``:188-194``), the
per-parameter and ``_lnp`` files (``:197-213``), mean acceptance fraction and integrated
autocorrelation time (``:216-221``), ``{GRB}_info.json`` (``:223-226``; written with plain Python
numbers -- the reference's ``json.dump`` of a NumPy array raises).  Not covered: argparse CLI, trace plot.
"""
import json
import os

import numpy as np

truths = {                                                       # synth_mcmc.py:16-21 (log-space for 2..5)
    "Humped": np.array([1.0, 5.0, -3.0, 2.0, -1.0, 0.0]),
    "Classic": np.array([1.0, 5.0, -3.0, 3.0, -1.0, 0.0]),
    "Sloped": np.array([1.0, 1.0, -3.0, 2.0, 1.0, 1.0]),
    "Stuttering": np.array([1.0, 5.0, -5.0, 2.0, -1.0, 2.0]),
}


def initial_ball(grb, n_walk, n_pars=6, rng=None):
    """synth_mcmc.py:175-176: ``truths[grb] + 1e-4*randn(Npars)`` per walker, drawn walker by walker."""
    rng = rng or np.random
    p0 = np.array(truths[grb])
    return np.array([p0 + 1.0e-4 * rng.randn(n_pars) for _ in range(n_walk)])


class RunResult:
    """chain[walker, step, dim] and lnprobability[walker, step] as emcee's ``sampler.chain`` /
    ``sampler.lnprobability`` index them (synth_mcmc.py:193-194), plus the acceptance fractions."""

    def __init__(self, chain_swd, lnp_sw, acceptance_fraction, seed):
        self._chain = np.asarray(chain_swd)          # [step, walker, dim]
        self._lnp = np.asarray(lnp_sw)               # [step, walker]
        self.acceptance_fraction = np.asarray(acceptance_fraction)
        self.seed = seed

    @property
    def chain(self):
        return self._chain.transpose(1, 0, 2)

    @property
    def lnprobability(self):
        return self._lnp.T

    def get_chain(self):
        return self._chain

    def get_log_prob(self):
        return self._lnp

    def get_autocorr_time(self, **kw):
        return integrated_time(self._chain, **kw)


def run(grb, x, y, yerr, n_walk, n_step, seed=0, p0=None, device=0, dist=None, fbad=None, moves=None):
    """One chain of ``n_step`` stretch-move steps for ``n_walk`` walkers, positions resident on the GPU
    (one fused launch per half-step; with ``dist`` the ensemble is sharded over the ranks).  ``moves``: emcee 3's
    argument (``DeviceEnsemble``), e.g. ``[(DEMove(), 0.8), (DESnookerMove(), 0.2)]``; None is the stretch move.  ``fbad``: the
    reference's bad-parameter file (``synth_mcmc.py:159,181``, ``mcmc_eqns.py:72-79``) -- proposals whose likelihood
    was not finite are logged on the device and appended to it after the run (by rank 0)."""
    from .. import _capi as A
    from ..engine import Likelihood, time_grid
    from ..sampler import DeviceEnsemble
    from .mcmc_eqns import lower, upper

    rng = np.random.RandomState(seed)
    if p0 is None:
        p0 = initial_ball(grb, n_walk, rng=rng)
    p0 = np.asarray(p0, dtype=np.float64)
    lk = Likelihood(A.script_model_spec(), time_grid(None), x, y, yerr, lower, upper, device=device)
    try:
        ens = DeviceEnsemble.from_likelihood(lk, n_walk, p0.shape[1], a=2.0, seed=seed, dist=dist, moves=moves)
        ens.initialise(p0)
        chain, lnp = ens.run(n_step, store=True)
        ens.check_peers()
        res = RunResult(chain.cpu().numpy(), lnp.cpu().numpy(), ens.acceptance_fraction().cpu().numpy(), seed)
        bad, dropped = ens.drain_bad()
        res.bad_rows, res.bad_dropped = bad, dropped
        if fbad is not None and ens.rank == 0 and len(bad):
            from .mcmc_eqns import _write_bad
            _write_bad(fbad, bad)
        ens.close()
    finally:
        lk.close()
    return res


def run_tempered(grb, x, y, yerr, n_walk, ntemps, n_step, beta_min, seed=0, discard=None, device=0, moves=None):
    """A parallel-tempered run (``TemperedEnsemble``): ``ntemps`` temperatures on a geometric ladder from 1 down to
    ``beta_min``, ``n_walk`` walkers each, every temperature started from ``initial_ball``.  Returns the ``RunResult``
    of the cold chain (``write_outputs`` and ``posterior_summary_device`` take it as they take ``run``'s) with
    ``log_evidence`` / ``log_evidence_err`` (``thermodynamic_log_evidence`` over the steps after ``discard``; None:
    the first half), ``betas``, ``swap_acceptance`` [ntemps - 1] and the device-resident cold chain and lnp of every
    temperature (``chain_device``, ``lnp_device``) attached.  The ladder should reach the prior:
    ``beta_min * <lnL>_{beta_min}`` is the part of ln Z the hottest temperature stands for.  ``moves`` as for ``run``."""
    from .. import _capi as A
    from ..engine import Likelihood, time_grid
    from ..sampler import TemperedEnsemble, geometric_betas, thermodynamic_log_evidence
    from .mcmc_eqns import lower, upper

    betas = geometric_betas(ntemps, beta_min)
    discard = n_step // 2 if discard is None else int(discard)
    rng = np.random.RandomState(seed)
    p0 = np.stack([initial_ball(grb, n_walk, rng=rng) for _ in range(ntemps)])
    lk = Likelihood(A.script_model_spec(), time_grid(None), x, y, yerr, lower, upper, device=device)
    try:
        ens = TemperedEnsemble.from_likelihood(lk, n_walk, p0.shape[2], betas, a=2.0, seed=seed, moves=moves)
        ens.initialise(p0)
        chain, lnp = ens.run(n_step, store=True)
        log_z, dlog_z = thermodynamic_log_evidence(betas, lnp, discard=discard)
        res = RunResult(chain.cpu().numpy(), lnp[:, 0].cpu().numpy(), ens.acceptance_fraction()[0].cpu().numpy(), seed)
        res.log_evidence, res.log_evidence_err = log_z, dlog_z
        res.betas = betas
        res.swap_acceptance = ens.swap_acceptance_fraction().cpu().numpy()
        res.chain_device, res.lnp_device = chain, lnp        # CUDA tensors [n_step, n_walk, ndim], [n_step, ntemps, n_walk]
    finally:
        lk.close()
    return res


def run_smc(grb, x, y, yerr, n_particles, seed=0, moves=None, device=0, max_stages=1000, **smc_kw):
    """Sequential Monte Carlo (``SMCSampler``): ``n_particles`` drawn uniformly in the script prior box
    (``mcmc_eqns.lower`` / ``upper``) with ``np.random.RandomState(seed)``, annealed to the posterior.  Returns the
    ``RunResult`` of the final, equally weighted population as a one-step chain [1, n_particles, 6] (``write_outputs``
    and ``posterior_summary_device`` take it as they take ``run``'s; its acceptance fraction is that of the steps at
    beta = 1 after the last stage), with ``log_evidence``, the stage history ``betas``, ``ess``, ``steps``,
    ``stage_acceptance``, ``n_evaluations`` and the device-resident population (``chain_device`` [1, N, 6],
    ``lnp_device`` [1, N]) attached.  ``moves`` and ``smc_kw`` (target_ess, p_move, min_steps, max_steps) as for
    ``SMCSampler``."""
    from .. import _capi as A
    from ..engine import Likelihood, time_grid
    from ..sampler import SMCSampler
    from .mcmc_eqns import lower, upper

    rng = np.random.RandomState(seed)
    p0 = lower + (upper - lower) * rng.rand(int(n_particles), lower.size)
    lk = Likelihood(A.script_model_spec(), time_grid(None), x, y, yerr, lower, upper, device=device)
    try:
        smc = SMCSampler.from_likelihood(lk, int(n_particles), lower.size, seed=seed, moves=moves, **smc_kw)
        out = smc.run(p0, max_stages=max_stages)
        chain, lnp = out.coords.clone()[None], out.lnp.clone()[None]
        acc = (smc.accepted.double() / out.final_steps).cpu().numpy()
        res = RunResult(chain.cpu().numpy(), lnp.cpu().numpy(), acc, seed)
        res.log_evidence = out.log_evidence
        res.betas, res.ess, res.steps, res.stage_acceptance = out.betas, out.ess, out.steps, out.acceptance
        res.final_steps, res.n_evaluations = out.final_steps, out.n_evaluations
        res.chain_device, res.lnp_device = chain, lnp
    finally:
        lk.close()
    return res


# ---- integrated autocorrelation time (emcee.autocorr, restated; emcee is not installed) -----------
def _next_pow_two(n):
    i = 1
    while i < n:
        i = i << 1
    return i


def function_1d(x):
    """Normalised autocorrelation function of a 1-D series via FFT."""
    x = np.atleast_1d(x)
    if len(x.shape) != 1:
        raise ValueError("invalid dimensions for 1D autocorrelation function")
    n = _next_pow_two(len(x))
    f = np.fft.fft(x - np.mean(x), n=2 * n)
    acf = np.fft.ifft(f * np.conjugate(f))[: len(x)].real
    acf /= acf[0]
    return acf


def _auto_window(taus, c):
    m = np.arange(len(taus)) < c * taus
    if np.any(m):
        return int(np.argmin(m))
    return len(taus) - 1


class AutocorrError(Exception):
    def __init__(self, tau, *args):
        self.tau = tau
        super().__init__(*args)


def integrated_time(x, c=5, tol=50, quiet=False):
    """Integrated autocorrelation time per dimension of a chain [step, walker, dim] (Sokal's automatic
    windowing, as emcee's ``integrated_time``: ACF averaged over walkers, window = first M with
    M >= c*tau(M); raises ``AutocorrError`` when the chain is shorter than ``tol*tau`` unless ``quiet``)."""
    x = np.atleast_1d(x)
    if len(x.shape) == 1:
        x = x[:, np.newaxis, np.newaxis]
    if len(x.shape) == 2:
        x = x[:, :, np.newaxis]
    if len(x.shape) != 3:
        raise ValueError("invalid dimensions")
    n_t, n_w, n_d = x.shape
    f = np.zeros((n_d, n_t))
    for d in range(n_d):
        for k in range(n_w):
            f[d] += function_1d(x[:, k, d])
        f[d] /= n_w
    return _tau_from_acf(lambda lo, hi: f[:, lo:hi], n_t, n_d, c, tol, quiet)


def _tau_from_acf(acf, n_t, n_d, c, tol, quiet):
    """Sokal's window and emcee's length check on a walker-averaged ACF of ``n_t`` rows that ``acf(lo, hi)`` delivers
    as lags [lo, hi) ([n_d, hi - lo]).  Lags are requested in blocks [0, L) with L = min(n_t, 128), 256, ... until every
    dimension's window lies inside them, so about twice the window is computed instead of all n_t lags.  The result is
    the full-length one bit for bit: ``np.cumsum`` adds in order, so the taus of a prefix are the prefix of the taus,
    and the first M with M >= c*tau(M) is decided as soon as the prefix holds one M that passes and one that fails."""
    f = np.empty((n_d, 0))
    tau_est = np.empty(n_d)
    done = np.zeros(n_d, dtype=bool)
    L = 0
    while not done.all():
        hi = min(n_t, max(128, 2 * L))
        f = np.concatenate([f, acf(L, hi)], axis=1)
        L = hi
        for d in np.flatnonzero(~done):
            taus = 2.0 * np.cumsum(f[d]) - 1.0
            m = np.arange(L) < c * taus
            if L == n_t:
                window = _auto_window(taus, c)
            elif np.isnan(taus[0]):          # every tau is NaN (a constant series): so is the estimate, whatever the window
                window = 0
            elif m.any() and not m.all():
                window = int(np.argmin(m))
            else:
                continue
            tau_est[d] = taus[window]
            done[d] = True
    flag = tol * tau_est > n_t
    if np.any(flag):
        msg = ("The chain is shorter than {0} times the integrated autocorrelation time for {1} parameter(s). "
               "Use this estimate with caution and run a longer chain!\n").format(tol, np.sum(flag))
        msg += "N/{0} = {1:.0f};\ntau: {2}".format(tol, n_t / tol, tau_est)
        if not quiet:
            raise AutocorrError(tau_est, msg)
    return tau_est


def integrated_time_device(chain, c=5, tol=50, quiet=False, discard=0, thin=1):
    """``integrated_time`` of a float64 CUDA tensor chain [n_steps, nwalkers, ndim], computed where the chain lies:
    the walker-averaged autocorrelation function comes from ``mp_chain_autocorr`` for the lags Sokal's window needs,
    and only [ndim, L] numbers reach the host.  Same window, same ``AutocorrError``, as ``integrated_time``.

    ``discard`` / ``thin`` follow emcee 3's ``EnsembleSampler.get_autocorr_time(discard, thin)``: the rows are those of
    ``Backend.get_value``, ``chain[discard + thin - 1::thin]``, and the returned tau is multiplied by ``thin`` (the
    length check and the tau an ``AutocorrError`` carries are those of the thinned chain, as there)."""
    import torch
    from ..engine import chain_autocorr
    if not (isinstance(chain, torch.Tensor) and chain.is_cuda and chain.dtype == torch.float64 and chain.dim() == 3):
        raise ValueError("integrated_time_device: chain must be a float64 CUDA tensor [n_steps, nwalkers, ndim]")
    discard, thin = int(discard), int(thin)
    n_steps, n_w, n_d = chain.shape
    first = discard + thin - 1
    if discard < 0 or thin < 1 or first >= n_steps:
        raise ValueError("integrated_time_device: no rows left after discard / thin")
    chain = chain.contiguous()
    n_t = len(range(first, n_steps, thin))
    device = chain.device.index
    stream = torch.cuda.current_stream(chain.device).cuda_stream

    def acf(lo, hi):
        return chain_autocorr(chain.data_ptr(), n_steps, n_w, n_d, first, thin, lo, hi, device=device, stream=stream)

    return thin * _tau_from_acf(acf, n_t, n_d, c, tol, quiet)


# ---- the reference's output files ------------------------------------------------------------
def create_filenames(GRB, root="."):
    """synth_mcmc.py:71-105 (the dataset directory must exist; the bad-parameter file is truncated)."""
    data_dirname = os.path.join(root, "data", "synthetic_datasets", GRB)
    if not os.path.exists(data_dirname):
        raise FileNotFoundError("Please make sure your chosen dataset exists.")
    plot_dirname = os.path.join(root, "plots", "synthetic_datasets", GRB)
    os.makedirs(plot_dirname, exist_ok=True)
    fdata = os.path.join(data_dirname, f"{GRB}.csv")
    fchain = os.path.join(data_dirname, f"{GRB}_chain.csv")
    fbad = os.path.join(data_dirname, f"{GRB}_bad.csv")
    finfo = os.path.join(data_dirname, f"{GRB}_info.json")
    fplot = os.path.join(plot_dirname, f"{GRB}_trace.png")
    open(fbad, "w").close()
    return fdata, fchain, fbad, finfo, fplot, data_dirname


def write_outputs(fn, GRB, res, quiet_autocorr=True):
    """Write ``{GRB}_chain.csv``, ``{fn}_{k}.csv``, ``{fn}_lnp.csv`` and ``{GRB}_info.json`` in the
    reference's formats (synth_mcmc.py:188-226).  ``fn`` is the dataset directory; the per-parameter
    files are named ``f"{fn}_{k}.csv"`` exactly as the reference builds them (next to the directory).
    Returns the info dictionary."""
    chain, lnp = res.chain, res.lnprobability                 # [walker, step, dim], [walker, step]
    Nwalk, Nstep, Npars = chain.shape
    fchain = os.path.join(fn, f"{GRB}_chain.csv")
    with open(fchain, "w") as f:
        f.write(f"{Npars}, {Nwalk}, {Nstep}\n")
        rows = np.concatenate([chain.transpose(1, 0, 2).reshape(Nstep * Nwalk, Npars),
                               lnp.T.reshape(Nstep * Nwalk, 1)], axis=1)
        for r in rows:                                        # step-major, walker-minor (:190-194)
            f.write(", ".join(f"{v:.6f}" for v in r) + "\n")
    for k in range(Npars):                                    # one line per step (:197-204)
        with open(f"{fn}_{k}.csv", "w") as f:
            for j in range(Nstep):
                f.write(", ".join(f"{v:.6f}" for v in chain[:, j, k]) + "\n")
    with open(f"{fn}_lnp.csv", "w") as f:                     # (:207-213)
        for j in range(Nstep):
            f.write(", ".join(f"{v:.6f}" for v in lnp[:, j]) + "\n")
    tau = res.get_autocorr_time(quiet=quiet_autocorr)
    info = {"Npars": int(Npars), "Nwalk": int(Nwalk), "Nstep": int(Nstep), "seed": int(res.seed),
            "acceptance_fraction": float(np.mean(res.acceptance_fraction)), "tau": [float(t) for t in tau]}
    with open(os.path.join(fn, f"{GRB}_info.json"), "w") as f:
        json.dump(info, f)
    return info


def read_chain(fchain):
    """Inverse of the ``_chain.csv`` writer: (samples [Nstep*Nwalk, Npars], lnp, (Npars, Nwalk, Nstep)) --
    how plot_synth.py:139-143 reads it back."""
    with open(fchain) as f:
        Npars, Nwalk, Nstep = (int(v) for v in f.readline().split(","))
    arr = np.loadtxt(fchain, delimiter=",", skiprows=1)
    return arr[:, :Npars], arr[:, Npars], (Npars, Nwalk, Nstep)
