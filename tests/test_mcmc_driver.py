"""Row f1: the MCMC driver around the likelihood -- autocorrelation time, the reference's chain file
formats (CPU), and an end-to-end device-resident run + posterior summary (GPU)."""
import json
import os

import numpy as np
import pytest

from magprop_b200.synthetic import synth_mcmc as S


def test_integrated_time_ar1():
    rng = np.random.RandomState(0)
    phi, n = 0.8, 60000
    x = np.zeros((n, 6, 2))
    e = rng.randn(n, 6, 2)
    for i in range(1, n):
        x[i] = phi * x[i - 1] + e[i]
    tau = S.integrated_time(x)
    assert np.abs(tau / ((1 + phi) / (1 - phi)) - 1.0).max() < 0.06
    with pytest.raises(S.AutocorrError):
        S.integrated_time(x[:200])
    assert S.integrated_time(x[:200], quiet=True).shape == (2,)
    # direct O(N^2) autocorrelation agrees with the FFT form
    s = x[:512, 0, 0] - x[:512, 0, 0].mean()
    direct = np.array([np.sum(s[: len(s) - k] * s[k:]) for k in range(64)])
    assert np.allclose(S.function_1d(x[:512, 0, 0])[:64], direct / direct[0], atol=1e-12)


def test_initial_ball_draw_order():
    a = S.initial_ball("Sloped", 10, rng=np.random.RandomState(5))
    rng = np.random.RandomState(5)
    b = np.array([S.truths["Sloped"] + 1.0e-4 * rng.randn(6) for _ in range(10)])     # synth_mcmc.py:175-176
    assert (a == b).all()


def test_chain_files_have_the_reference_format(tmp_path):
    rng = np.random.RandomState(2)
    Nstep, Nwalk, Npars = 7, 12, 6
    chain = rng.randn(Nstep, Nwalk, Npars)
    lnp = -np.abs(rng.randn(Nstep, Nwalk)) * 100
    res = S.RunResult(chain, lnp, np.full(Nwalk, 0.25), seed=11)
    d = tmp_path / "data" / "synthetic_datasets" / "Humped"
    d.mkdir(parents=True)
    fdata, fchain, fbad, finfo, fplot, fn = S.create_filenames("Humped", root=str(tmp_path))
    assert fn == str(d) and os.path.exists(fbad) and os.path.getsize(fbad) == 0
    info = S.write_outputs(fn, "Humped", res)
    # the writer of synth_mcmc.py:188-213, literally
    lines = [f"{Npars}, {Nwalk}, {Nstep}\n"]
    for j in range(Nstep):
        for i in range(Nwalk):
            lines.append("".join(f"{res.chain[i, j, k]:.6f}, " for k in range(Npars)) + f"{res.lnprobability[i, j]:.6f}\n")
    assert open(fchain).read() == "".join(lines)
    for k in range(Npars):
        want = "".join(", ".join(f"{res.chain[i, j, k]:.6f}" for i in range(Nwalk)) + "\n" for j in range(Nstep))
        assert open(f"{fn}_{k}.csv").read() == want
    want = "".join(", ".join(f"{res.lnprobability[i, j]:.6f}" for i in range(Nwalk)) + "\n" for j in range(Nstep))
    assert open(f"{fn}_lnp.csv").read() == want
    assert json.load(open(finfo)) == info and info["Nwalk"] == Nwalk and info["acceptance_fraction"] == 0.25
    samples, lp, shape = S.read_chain(fchain)
    assert shape == (Npars, Nwalk, Nstep) and samples.shape == (Nstep * Nwalk, Npars)
    assert np.allclose(samples[:Nwalk], chain[0], atol=5e-7) and np.allclose(lp[:Nwalk], lnp[0], atol=5e-7)


@pytest.mark.gpu
def test_device_run_and_posterior_summary(built, golden, tmp_path):
    from magprop_b200.synthetic import generate_data as G
    from magprop_b200.synthetic import plot_synth as P
    from oracle import magprop_oracle as O

    # generate_data.py recipe on the GPU curve == the committed golden dataset (made from the reference curve)
    x, y, yerr = G.generate("Humped", seed=O.SYNTH_SEED + sum(map(ord, "Humped")))   # oracle/make_goldens.py's seeding
    g = golden["lnprob_script"]
    assert (x == g["Humped_x"]).all()
    # (the golden dataset was drawn from the reference's default-tolerance curve, itself up to 1e-5 from the
    # converged light curve at isolated nodes -- SURVEY.md fact 6)
    assert np.abs(yerr / g["Humped_yerr"] - 1).max() < 2e-5 and np.abs(y - g["Humped_y"]).max() < 1e-4 * np.abs(g["Humped_y"]).max()

    res = S.run("Humped", g["Humped_x"], g["Humped_y"], g["Humped_yerr"], n_walk=50, n_step=60, seed=3)
    assert res.chain.shape == (50, 60, 6) and res.lnprobability.shape == (50, 60)
    assert np.isfinite(res.lnprobability).all()
    assert 0.2 < res.acceptance_fraction.mean() < 0.9
    # the stored lnprob is the oracle's lnprob of the stored position
    pos = res.get_chain()[-1, :8]
    want = O.lnprob_batch(pos, g["Humped_x"], g["Humped_y"], g["Humped_yerr"], O.script_spec(), O.SCRIPT_LOWER,
                          O.SCRIPT_UPPER, tight=True)
    assert np.abs(res.get_log_prob()[-1, :8] / want - 1).max() < 1e-6
    # the ensemble climbs from the 1e-4 ball towards the posterior bulk
    assert res.get_log_prob()[-1].mean() > res.get_log_prob()[0].mean() - 5.0
    d = tmp_path / "data" / "synthetic_datasets" / "Humped"
    d.mkdir(parents=True)
    info = S.write_outputs(str(d), "Humped", res)
    assert len(info["tau"]) == 6
    samples, lp, _ = S.read_chain(str(d / "Humped_chain.csv"))
    stats, pars, ymod, fit = P.posterior_summary(samples, g["Humped_x"], g["Humped_y"], g["Humped_yerr"], grb="Humped",
                                                 truths=G.GRBs["Humped"])
    assert len(stats["correlations"]) == 15 and fit.shape == (4, 10001) and ymod.shape == (50,)
    assert abs(np.log10(pars[2]) + 3.0) < 0.5 and 0.3 < stats["stats"]["chi_square_red"] < 5.0
    assert stats["latex"].count("&") == 7


@pytest.mark.gpu
def test_posterior_summary_on_the_device_matches_the_host_one(built, golden):
    """Row f4 as a device reduction: correlations, percentiles (exact order statistics by radix select) and the fit
    statistics from the kernel's chi-square == the host NumPy summary of the same chain."""
    import torch
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, chain_moments, chain_order_statistics, time_grid
    from magprop_b200.sampler import DeviceEnsemble
    from magprop_b200.synthetic import plot_synth as P
    from oracle import magprop_oracle as O
    g = golden["lnprob_script"]
    x, y, yerr = g["Humped_x"], g["Humped_y"], g["Humped_yerr"]
    lk = Likelihood(A.script_model_spec(), time_grid(None), x, y, yerr, O.SCRIPT_LOWER, O.SCRIPT_UPPER)
    ens = DeviceEnsemble.from_likelihood(lk, 64, 6, seed=5)
    ens.initialise(O.SYNTH_TRUTHS_LOG["Humped"] + 1e-3 * np.random.RandomState(2).randn(64, 6))
    chain, _ = ens.run(120, store=True)                       # [120, 64, 6] on the device
    torch.cuda.synchronize()
    host = chain.cpu().numpy().reshape(-1, 6)
    n = host.shape[0]
    # the two primitives
    mean, cov = chain_moments(chain.data_ptr(), n, 6)
    assert np.allclose(mean, host.mean(axis=0), rtol=1e-13) and np.allclose(cov, np.cov(host.T), rtol=1e-10, atol=0)
    ranks = [0, 1, n // 3, n - 2, n - 1]
    for col in (0, 3, 5):
        assert np.array_equal(chain_order_statistics(chain.data_ptr(), n, 6, col, ranks), np.sort(host[:, col])[ranks])
    neg = torch.tensor([[-1.5, 0.0], [2.0, -0.0], [-3.0, 7.0], [0.5, -2.0]], dtype=torch.float64, device="cuda")
    assert np.array_equal(chain_order_statistics(neg.data_ptr(), 4, 2, 0, [0, 1, 2, 3]), [-3.0, -1.5, 0.5, 2.0])
    # the summary
    s_dev, p_dev = P.posterior_summary_device(chain, x, y, yerr, grb="Humped")
    s_host, p_host, _, _ = P.posterior_summary(host, x, y, yerr, grb="Humped")
    assert np.array_equal(p_dev, p_host)
    assert np.allclose(s_dev["correlations"], s_host["correlations"], rtol=1e-9, atol=1e-12)
    for k in s_host["pars"]:
        assert np.allclose(s_dev["pars"][k], s_host["pars"][k], rtol=1e-12, atol=1e-300)
    assert abs(s_dev["stats"]["chi_square_red"] / s_host["stats"]["chi_square_red"] - 1) < 1e-9
    assert abs(s_dev["stats"]["aicc"] - s_host["stats"]["aicc"]) < 1e-9 * abs(s_host["stats"]["aicc"])
    lk.close()


def test_fit_statistics_from_lnlike():
    from magprop_b200.magnetar import fit_stats as F
    rng = np.random.RandomState(0)
    y, m, e = rng.rand(30) + 1, rng.rand(30) + 1, 0.1 + rng.rand(30)
    chi2 = np.sum(((y - m) / e) ** 2)
    r, a = F.from_lnlike(-0.5 * chi2, 30, 6)
    assert np.isclose(r, F.redchisq(y, m, deg=6, sd=e), rtol=1e-14) and np.isclose(a, F.aicc(y, m, e, 6), rtol=1e-14)
    assert F.redchisq(y, m) == np.sum((y - m) ** 2) and F.redchisq(y, m, sd=e) == chi2
    with pytest.raises(ValueError):
        F.aicc(y, m[:-1], e, 6)
