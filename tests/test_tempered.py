"""Parallel-tempered ensembles and thermodynamic-integration evidence: the NumPy restatement against the
host-compiled kernel helpers, the sampler on a Gaussian with a known evidence, argument checks of the C
ABI (CPU); the fused tempered half-step and swap against the restatement, determinism, and the evidence of a
synthetic dataset against importance sampling (GPU)."""
import ctypes as C
from math import erf

import numpy as np
import pytest

import ensemble_ref as E
from magprop_b200.sampler import (DeviceEnsemble, StretchMove, TemperedEnsemble, geometric_betas,
                                  thermodynamic_log_evidence)

SIG = np.array([1.0, 2.0, 0.5])
BOX = 10.0
# ln of the Gaussian's mass inside the box, minus ln of the box volume: -8.987
LN_Z_GAUSS = sum(np.log(erf(BOX / (s * np.sqrt(2.0)))) for s in SIG) - 3 * np.log(2 * BOX)


def gauss_box_lnprob(q):
    """Normalised 3-D Gaussian likelihood, sigma = (1, 2, 0.5), inside the box [-10, 10]^3 (-inf outside)."""
    q = np.asarray(q)
    lnl = -0.5 * np.sum((q / SIG) ** 2, axis=1) - np.sum(np.log(SIG * np.sqrt(2 * np.pi)))
    return np.where(np.all(np.abs(q) <= BOX, axis=1), lnl, -np.inf)


@pytest.fixture(scope="module")
def tempered_rng(tmp_path_factory):
    """tests/hostsim/tempered_rng.cpp -- the kernels' tempering helpers of magprop_rng.cuh -- built for the host."""
    import os
    import subprocess
    from conftest import ROOT
    so = str(tmp_path_factory.mktemp("tempered_rng") / "tempered_rng.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "tempered_rng.cpp")], check=True)
    lib = C.CDLL(so)
    vp = C.c_void_p
    lib.tr_tempered_rows.argtypes = [C.c_int, C.c_int, C.c_ulonglong, C.c_ulonglong, C.c_int, C.c_int, vp, vp, vp, vp]
    lib.tr_tempered_rows.restype = None
    lib.tr_pt_swap_accept.argtypes = [C.c_ulonglong, C.c_ulonglong, C.c_uint, C.c_double, C.c_double, C.c_double,
                                      C.c_double]
    return lib


def test_host_compiled_mapping_and_swap_decision_match_the_restatement(tempered_rng):
    rng = np.random.RandomState(1)
    for n, T in ((12, 1), (12, 5), (256, 8), (2048, 8)):
        for step, split, randomize in ((0, 0, 1), (3, 1, 1), (12345, 0, 0)):
            m = T * (n // 2)
            pj = rng.randint(0, n // 2, size=m).astype(np.int32)
            t, row, part = (np.empty(m, np.int32) for _ in range(3))
            tempered_rng.tr_tempered_rows(n, T, 99, step, split, randomize, pj.ctypes.data, t.ctypes.data, row.ctypes.data,
                                         part.ctypes.data)
            wt, wrow, wcomp = E.tempered_rows(n, T, 99, step, split, bool(randomize))
            assert np.array_equal(t, wt) and np.array_equal(row, wrow)
            assert np.array_equal(part, wcomp[wt, pj])
            assert np.array_equal(np.sort(row // n), wt)                      # movers stay in their temperature
    vals = np.concatenate([-rng.exponential(50.0, 400), [-np.inf] * 4])
    for k in range(400):
        row = int(rng.randint(0, 1 << 20))
        bh, bc = sorted(rng.rand(2))
        lh, lc = rng.choice(vals), rng.choice(vals)
        got = tempered_rng.tr_pt_swap_accept(5, 77 + (k << 33), row, bc, bh, lh, lc)
        want = E.swap_accept(5, 77 + (k << 33), np.array([row]), bc, bh, np.array([lh]), np.array([lc]))[0]
        assert got == int(want), (row, bc, bh, lh, lc)


# ---- the sampler on a Gaussian with a known evidence ----------------------------------------------------
def _tempered(betas, n, seed, p0, nsteps):
    ens = TemperedEnsemble(E.NumpyBackend(gauss_box_lnprob), n, 3, betas, seed=seed, device="cpu")
    ens.initialise(p0)
    chain, lps = ens.run(nsteps)
    return ens, chain.numpy(), lps.numpy()


def test_tempered_gaussian_recovers_evidence_and_posterior():
    assert abs(LN_Z_GAUSS - (-8.987)) < 1e-3
    betas = geometric_betas(32, 1e-6)
    ens, chain, lps = _tempered(betas, 32, 3, 0.1 * np.random.RandomState(2).randn(32, 3), 3000)
    log_z, dlog_z = thermodynamic_log_evidence(betas, lps, discard=1000)
    assert abs(log_z - LN_Z_GAUSS) < 0.25, (log_z, dlog_z)
    assert np.isfinite(dlog_z) and dlog_z < 0.25
    sd = chain[1000:].reshape(-1, 3).std(axis=0)
    assert np.allclose(sd, SIG, rtol=0.12), sd
    swap = ens.swap_acceptance_fraction().numpy()
    assert swap.shape == (31,) and (swap > 0).all() and (swap < 1).all(), swap
    acc = ens.acceptance_fraction().numpy()
    assert acc.shape == (32, 32) and 0.2 < acc[0].mean() < 0.9
    assert lps.shape == (3000, 32, 32) and np.array_equal(lps[:, 0], gauss_box_lnprob(chain.reshape(-1, 3)).reshape(3000, 32))


def test_one_temperature_is_the_device_ensemble():
    p0 = np.random.RandomState(4).randn(16, 3)
    ens, chain, lps = _tempered([1.0], 16, 9, p0, 40)
    ref = DeviceEnsemble(E.NumpyBackend(gauss_box_lnprob), 16, 3, seed=9, device="cpu")
    ref.set_state(p0, gauss_box_lnprob(p0))
    rc, rl = ref.run(40, store=True)
    assert np.array_equal(chain, rc.numpy()) and np.array_equal(lps[:, 0], rl.numpy())
    assert np.array_equal(ens.acceptance_fraction().numpy()[0], ref.acceptance_fraction().numpy())
    assert ens.swap_acceptance_fraction().shape == (0,)


def test_initialise_broadcasts_and_checks_shapes():
    ens = TemperedEnsemble(E.NumpyBackend(gauss_box_lnprob), 8, 3, [1.0, 0.5, 0.1], device="cpu")
    p0 = np.random.RandomState(0).randn(8, 3)
    ens.initialise(p0)
    assert np.array_equal(ens.coords.numpy().reshape(3, 8, 3), np.broadcast_to(p0, (3, 8, 3)))
    assert np.array_equal(ens.lnp.numpy(), gauss_box_lnprob(ens.coords.numpy()))
    with pytest.raises(ValueError):
        ens.initialise(np.zeros((2, 8, 3)))
    with pytest.raises(ValueError):
        TemperedEnsemble(E.NumpyBackend(gauss_box_lnprob), 8, 3, [1.0, 0.5], device="cpu", dist=object())
    with pytest.raises(NotImplementedError):
        ens.run_until_converged(10)


# ---- the evidence estimate ----------------------------------------------------------------------------
def test_thermodynamic_log_evidence_closed_form_and_checks():
    d = 6
    for T, beta_min in ((2, 0.5), (16, 1e-3), (33, 1e-9)):
        betas = geometric_betas(T, beta_min)
        assert betas[0] == 1.0 and betas[-1] == beta_min and (np.diff(betas) < 0).all()
        lnp = np.broadcast_to((-d / (2 * betas))[None, :, None], (5, T, 4))
        log_z, dlog_z = thermodynamic_log_evidence(betas, lnp)
        assert abs(log_z - ((d / 2) * np.log(beta_min) - d / 2)) < 1e-12 * (1 + abs(log_z))
        assert dlog_z >= 0
    betas = geometric_betas(4, 1e-2)
    lnp = np.full((3, 4, 2), -1.0)
    assert thermodynamic_log_evidence(betas, lnp, discard=2)[0] == thermodynamic_log_evidence(betas, lnp)[0]
    for bad in ([1.0, 0.1, 0.5, 0.01], [0.9, 0.5, 0.1, 0.01], [1.0, 0.5, 0.5, 0.1], [1.0, 0.5, -0.1, -0.2], [1.0]):
        with pytest.raises(ValueError):
            thermodynamic_log_evidence(bad, np.full((3, len(bad), 2), -1.0))
    for v in (-np.inf, np.nan):
        x = lnp.copy()
        x[2, 1, 0] = v
        with pytest.raises(ValueError):
            thermodynamic_log_evidence(betas, x)
    thermodynamic_log_evidence(betas, np.where(np.arange(3)[:, None, None] < 1, -np.inf, lnp), discard=1)
    with pytest.raises(ValueError):
        thermodynamic_log_evidence(betas, lnp[:, :3])
    with pytest.raises(ValueError):
        geometric_betas(4, 1.5)


def test_capi_tempered_argument_checks_without_device(built):
    """Every argument of the tempered entry points is checked on the host: MP_ERR_BAD_ARG, no device touched."""
    from magprop_b200 import _capi as A
    lib = A.load()

    def desc(**kw):
        e = A.Ensemble()
        e.coords, e.lnp, e.nwalkers, e.ndim, e.a, e.seed, e.world = 0x1000, 0x2000, 8, 6, 2.0, 1, 1
        for k, v in kw.items():
            setattr(e, k, v)
        return e

    def both(e, betas, ntemps=None):
        b = np.ascontiguousarray(betas, dtype=np.float64)
        nt = b.size if ntemps is None else ntemps
        r1 = lib.mp_tempered_swap(C.byref(e), nt, A.ptr(b), 0, None, None)
        r2 = lib.mp_tempered_half_step(None, C.byref(e), nt, A.ptr(b), 0, 0, None)
        return r1, r2

    ok = [1.0, 0.5, 0.1]
    for betas in ([1.0, 0.5, 0.5], [0.9, 0.5], [1.0, 0.1, 0.5], [1.0, 0.5, 0.0], [1.0, -0.5], [1.0, np.nan],
                  [1.0, 0.5, np.inf], [2.0, 1.0]):
        assert both(desc(), betas) == (A.MP_ERR_BAD_ARG,) * 2, betas
    assert both(desc(), ok, ntemps=0) == (A.MP_ERR_BAD_ARG,) * 2
    assert both(desc(), np.geomspace(1, 1e-3, A.MP_MAX_TEMPS + 1)) == (A.MP_ERR_BAD_ARG,) * 2
    assert both(desc(world=2), ok) == (A.MP_ERR_BAD_ARG,) * 2
    assert both(desc(n_peers=1), ok) == (A.MP_ERR_BAD_ARG,) * 2
    assert both(desc(pack_out=0x3000), ok) == (A.MP_ERR_BAD_ARG,) * 2
    assert both(desc(nwalkers=7), ok) == (A.MP_ERR_BAD_ARG,) * 2
    assert both(desc(coords=None), ok) == (A.MP_ERR_BAD_ARG,) * 2
    assert both(desc(nwalkers=1 << 29), np.geomspace(1, 1e-3, 4)) == (A.MP_ERR_BAD_ARG,) * 2
    assert lib.mp_tempered_swap(C.byref(desc()), 3, None, 0, None, None) == A.MP_ERR_BAD_ARG
    b = np.array(ok)
    assert lib.mp_tempered_half_step(None, C.byref(desc()), 3, A.ptr(b), 0, 0, None) == A.MP_ERR_BAD_ARG   # null handle


# ---- on the GPU -----------------------------------------------------------------------------------------
def _humped(golden):
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, time_grid
    from oracle import magprop_oracle as O
    g = golden["lnprob_script"]
    return Likelihood(A.script_model_spec(), time_grid(None), g["Humped_x"], g["Humped_y"], g["Humped_yerr"],
                      O.SCRIPT_LOWER, O.SCRIPT_UPPER)


def _spread_start(T, n, seed):
    """Cold temperatures in a ball around the truth, hot ones spread over the prior box."""
    from oracle import magprop_oracle as O
    rng = np.random.RandomState(seed)
    p0 = np.empty((T, n, 6))
    for t in range(T):
        if t < T // 2:
            p0[t] = O.SYNTH_TRUTHS_LOG["Humped"] + 1e-2 * (t + 1) * rng.randn(n, 6)
        else:
            p0[t] = O.SCRIPT_LOWER + (O.SCRIPT_UPPER - O.SCRIPT_LOWER) * rng.rand(n, 6)
    return p0


@pytest.mark.gpu
def test_tempered_kernels_match_the_restatement(built, golden):
    """T = 8 x n = 2048 on Humped: 8192 movers per half-step, so the launch is work-list ordered, and the hot
    temperatures spread over the prior feed the stiff queue.  Half-steps, swaps, acceptance and swap counters equal
    the NumPy restatement driven by the device likelihood, bit for bit."""
    import torch
    lk = _humped(golden)
    T, n = 8, 2048
    betas = geometric_betas(T, 1e-4)
    p0 = _spread_start(T, n, 0)
    ens = TemperedEnsemble.from_likelihood(lk, n, 6, betas, seed=21)
    ens.initialise(p0)
    torch.cuda.synchronize()
    coords = p0.reshape(T * n, 6).copy()
    lnp = ens.lnp.cpu().numpy().copy()
    assert np.array_equal(lnp, lk.lnprob(coords))
    acc, swaps = np.zeros(T * n, np.int32), np.zeros(T - 1, np.int32)
    stiff = []
    for step in range(3):
        for split in (0, 1):
            ens.backend.tempered_half_step(ens, step, split)
            stiff.append(lk.last_stiff_count())
            t, rows, comp = E.tempered_rows(n, T, 21, step, split)
            E.half_step(coords, lnp, rows, t, comp, StretchMove(2.0), 21, 2 * step + split, lk.lnprob, betas=betas,
                        accepted=acc)
            assert np.array_equal(ens.coords.cpu().numpy(), coords) and np.array_equal(ens.lnp.cpu().numpy(), lnp)
        ens.backend.tempered_swap(ens, step)
        E.swap(coords, lnp, betas, n, 21, step, swaps)
        ens.step += 1
        torch.cuda.synchronize()
        assert np.array_equal(ens.coords.cpu().numpy(), coords) and np.array_equal(ens.lnp.cpu().numpy(), lnp)
    assert np.array_equal(ens.accepted.cpu().numpy(), acc) and np.array_equal(ens.swap_accepted.cpu().numpy(), swaps)
    assert min(stiff) > 0, stiff
    assert 0 < acc.sum() < T * n * 3 and swaps.sum() > 0
    lk.close()


@pytest.mark.gpu
def test_one_temperature_equals_device_ensemble_on_gpu(built, golden):
    import torch
    from oracle import magprop_oracle as O
    lk = _humped(golden)
    p0 = O.SYNTH_TRUTHS_LOG["Humped"] + 1e-2 * np.random.RandomState(3).randn(64, 6)
    te = TemperedEnsemble.from_likelihood(lk, 64, 6, [1.0], seed=5)
    te.initialise(p0)
    c1, l1 = te.run(6)
    de = DeviceEnsemble.from_likelihood(lk, 64, 6, seed=5)
    de.initialise(p0)
    c2, l2 = de.run(6, store=True)
    torch.cuda.synchronize()
    assert torch.equal(c1, c2) and torch.equal(l1[:, 0], l2)
    assert torch.equal(te.accepted, de.accepted) and torch.equal(te.status, de.status)
    lk.close()


@pytest.mark.gpu
def test_tempered_runs_are_deterministic_across_streams(built, golden):
    import torch
    lk = _humped(golden)
    T, n = 4, 128
    betas = geometric_betas(T, 1e-3)
    p0 = _spread_start(T, n, 1)
    out = []
    for use_side in (False, True):
        st = torch.cuda.Stream() if use_side else torch.cuda.current_stream()
        with torch.cuda.stream(st):
            e = TemperedEnsemble.from_likelihood(lk, n, 6, betas, seed=8)
            e.initialise(p0)
            c, l = e.run(5)
            out.append((c, l, e.accepted.clone(), e.swap_accepted.clone()))
        torch.cuda.synchronize()
    for a, b in zip(*out):
        assert torch.equal(a, b)
    lk.close()


@pytest.mark.gpu
def test_run_concurrently_equals_run(built, golden):
    """run_concurrently advances a tempered ensemble beside a plain one as run advances each: every temperature moves,
    the swaps run, and the stored lnp holds every temperature."""
    import torch
    from magprop_b200.sampler import run_concurrently
    lk = _humped(golden)
    T, n = 4, 128
    betas = geometric_betas(T, 1e-3)
    p0 = _spread_start(T, n, 2)
    out = []
    for together in (False, True):
        te = TemperedEnsemble.from_likelihood(lk, n, 6, betas, seed=12)
        te.initialise(p0)
        de = DeviceEnsemble.from_likelihood(lk, 64, 6, seed=13)
        de.initialise(p0[0, :64])
        res = run_concurrently([te, de], 5, store=True) if together else [te.run(5), de.run(5, store=True)]
        torch.cuda.synchronize()
        assert te.step == de.step == 5
        out.append([*res[0], *res[1], te.accepted.clone(), te.swap_accepted.clone(), de.accepted.clone()])
    for a, b in zip(*out):
        assert a.shape == b.shape and torch.equal(a, b)
    assert out[0][1].shape == (5, T, n) and out[0][5].sum() > 0
    lk.close()


@pytest.mark.gpu
def test_run_tempered_evidence_matches_importance_sampling(built, golden):
    """ln Z of Sloped by thermodynamic integration (run_tempered) against an independent importance-sampling
    estimate: 2^22 draws from a multivariate Student-t fitted to the cold chain, evaluated by the device likelihood."""
    import torch
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, chain_moments, time_grid
    from magprop_b200.synthetic.mcmc_eqns import lower, upper
    from magprop_b200.synthetic.synth_mcmc import run_tempered
    g = golden["lnprob_script"]
    x, y, yerr = g["Sloped_x"], g["Sloped_y"], g["Sloped_yerr"]
    res = run_tempered("Sloped", x, y, yerr, n_walk=64, ntemps=24, n_step=3000, beta_min=1e-6, seed=2)
    assert res.get_chain().shape == (3000, 64, 6) and res.swap_acceptance.shape == (23,)
    assert (res.swap_acceptance > 0).all()
    flat = res.chain_device[1500:].reshape(-1, 6).contiguous()
    mu, cov = chain_moments(flat.data_ptr(), flat.shape[0], 6)
    nu, N = 5.0, 1 << 22
    scale = cov * (nu - 2.0) / nu
    L = np.linalg.cholesky(scale)
    gen = torch.Generator(device="cuda").manual_seed(11)
    z = torch.randn((N, 6), dtype=torch.float64, device="cuda", generator=gen)
    w = (torch.randn((N, int(nu)), dtype=torch.float64, device="cuda", generator=gen) ** 2).sum(dim=1) / nu   # chi2(nu)/nu
    draws = (torch.as_tensor(mu, device="cuda") + (z @ torch.as_tensor(L.T, device="cuda")) / w.sqrt()[:, None]).contiguous()
    lk = Likelihood(A.script_model_spec(), time_grid(None), x, y, yerr, lower, upper)
    lnp = torch.empty(N, dtype=torch.float64, device="cuda")
    lk.lnprob_device(draws.data_ptr(), N, 6, lnp.data_ptr())
    torch.cuda.synchronize()
    lk.close()
    # log density of the Student-t proposal, and the box prior's normalisation
    from math import lgamma, log, pi
    sol = torch.linalg.solve_triangular(torch.as_tensor(L, device="cuda"), (draws - torch.as_tensor(mu, device="cuda")).T,
                                        upper=False)
    maha = (sol * sol).sum(dim=0)
    lq = (lgamma((nu + 6) / 2) - lgamma(nu / 2) - 3 * log(nu * pi) - float(np.log(np.diag(L)).sum())
          - (nu + 6) / 2 * torch.log1p(maha / nu))
    lw = (lnp - float(np.log(upper - lower).sum()) - lq).cpu().numpy()
    m = lw[np.isfinite(lw)].max()
    wts = np.where(np.isfinite(lw), np.exp(lw - m), 0.0)
    ess = wts.sum() ** 2 / (wts ** 2).sum()
    log_z_is = m + np.log(wts.mean())
    sigma_is = wts.std() / np.sqrt(N) / wts.mean()
    tol = max(0.5, 3.0 * np.hypot(res.log_evidence_err, sigma_is))
    print(f"Sloped: TI {res.log_evidence:.4f} +- {res.log_evidence_err:.4f}, IS {log_z_is:.4f} +- {sigma_is:.4f}, "
          f"ESS {ess:.0f}, swap acceptance {np.round(res.swap_acceptance, 3).tolist()}")
    assert ess >= 1000
    assert abs(res.log_evidence - log_z_is) <= tol, (res.log_evidence, res.log_evidence_err, log_z_is, sigma_is)
