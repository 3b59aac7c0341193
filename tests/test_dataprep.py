"""Row f2 (data preparation) and row f4 (fit statistics): host functions against goldens generated from
the unmodified reference (oracle/make_goldens_dataprep.py) and against the reference's own test values."""
import os

import numpy as np
import pytest

from magprop_b200.dataprep import WMAP9, clean_raw, k_correct_grb, k_correction, luminosity_distance_cm, sgrbs
from magprop_b200.magnetar import fit_stats

GOLD = os.path.join(os.path.dirname(__file__), "golden", "dataprep.npz")


def test_wmap9_comoving_distance_known_answers():
    # astropy documentation, "from astropy.cosmology import WMAP9 as cosmo; cosmo.comoving_distance([0.5, 1.0, 1.5])"
    want = np.array([1916.06941724, 3363.07062107, 4451.7475201])
    got = WMAP9.comoving_distance_mpc([0.5, 1.0, 1.5])
    assert np.abs(got / want - 1.0).max() < 2e-9
    assert luminosity_distance_cm(0.0) == 0.0
    z = 0.9364
    assert np.isclose(luminosity_distance_cm(z), (1 + z) * WMAP9.comoving_distance_mpc(z)[0] * 3.08568e24, rtol=1e-15)


def test_k_correction_matches_reference():
    g = np.load(GOLD)
    assert list(g["grbs"]) == sgrbs                              # clean_data.py:6-8 order == kcorr_sgrbs.csv order
    for grb in ("061210", "080123", "051227"):
        raw = g[f"{grb}_in"]
        cols = dict(zip(("t", "tpos", "tneg", "flux", "fluxpos", "fluxneg"), raw.T))
        gamma, sigma, z, dl = g[f"{grb}_props"]
        k = k_correction(cols, gamma, sigma, z, dl)
        for c in ("t", "tpos", "tneg", "Lum50", "Lum50pos", "Lum50neg"):
            assert (k[c] == g[f"{grb}_{c}"]).all(), (grb, c)     # same operation order: bit-exact
        full = k_correct_grb(cols, gamma, sigma, z)
        assert np.abs(full["Lum50err"] / g[f"{grb}_Lum50err"] - 1.0).max() < 1e-14


def test_clean_raw_strips_plot_package_rows(tmp_path):
    p = tmp_path / "x_raw.txt"
    p.write_text("READ TERR 1 2\n! batSNR5flux\n0.02\t0.02\t-0.02\t9.4e-08\t9.6e-09\t-9.6e-09\nNO NO NO NO NO NO\n"
                 "! xrtwtslew\n1.5\t0.5\t-0.5\t2e-09\t1e-10\t-2e-10\n")
    cols = clean_raw(str(p))
    assert cols["t"].tolist() == [0.02, 1.5] and cols["fluxneg"].tolist() == [-9.6e-09, -2e-10]


def test_fit_stats_reference_values():
    # the reference's own tests (tests/test_funcs.py:153-182) use noisy_gaussian.csv; here the closed forms
    rng = np.random.RandomState(0)
    y, m, e = rng.rand(40), rng.rand(40), 0.1 + rng.rand(40)
    chi = np.sum(((y - m) / e) ** 2)
    assert fit_stats.redchisq(y, m, sd=e) == chi
    assert fit_stats.redchisq(y, m, deg=6, sd=e) == chi / (40 - 1.0 - 6)
    assert fit_stats.redchisq(y, m) == np.sum((y - m) ** 2.0)
    assert fit_stats.aicc(y, m, e, 6) == -chi + 12.0 + (12.0 * 7.0) / (40 - 6 - 1.0)
    with pytest.raises(ValueError):
        fit_stats.aicc(y, m[:-1], e, 6)
