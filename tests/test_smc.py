"""Sequential Monte Carlo with adaptive tempering: the host-compiled stage uniform against the restatement, the sampler
on the NumPy restatement (a Gaussian in a box with a known evidence, two separated modes, determinism), the new header
and every argument check of the C ABI without a GPU (CPU); the weights, resampling and annealed half-step kernels
against NumPy and the restatement, and the evidence and posterior of Sloped against importance sampling (GPU)."""
import ctypes as C
import math
import os
from math import erf

import numpy as np
import pytest

import ensemble_ref as E
import smc_ref as R
from conftest import ROOT
from magprop_b200.sampler import DEMove, DESnookerMove, DeviceEnsemble, SMCSampler, StretchMove

SIG = np.array([1.0, 2.0, 0.5])
BOX = 10.0
# ln of the Gaussian's mass inside the box, minus ln of the box volume: -8.987
LN_Z_GAUSS = sum(np.log(erf(BOX / (s * np.sqrt(2.0)))) for s in SIG) - 3 * np.log(2 * BOX)


def gauss_box_lnprob(q):
    """Normalised 3-D Gaussian likelihood, sigma = (1, 2, 0.5), inside the box [-10, 10]^3 (-inf outside)."""
    q = np.asarray(q)
    lnl = -0.5 * np.sum((q / SIG) ** 2, axis=1) - np.sum(np.log(SIG * np.sqrt(2 * np.pi)))
    return np.where(np.all(np.abs(q) <= BOX, axis=1), lnl, -np.inf)


def _smc(fn, n, ndim, seed, p0, **kw):
    smc = SMCSampler(R.NumpyBackend(fn), n, ndim, seed=seed, device="cpu", **kw)
    return smc, smc.run(p0)


def lnz_sd(res, n):
    """Monte Carlo standard deviation of ln Z from the stages' ESS: the relative variance of each stage's mean weight
    is about (N / ESS - 1) / N for a well-mixed population, and the stages add."""
    return math.sqrt(float(np.sum(n / res.ess - 1.0)) / n)


# ---- the stage uniform --------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def smc_rng(tmp_path_factory):
    """tests/hostsim/smc_rng.cpp -- smc_stage_uniform of magprop_rng.cuh -- built for the host."""
    import subprocess
    so = str(tmp_path_factory.mktemp("smc_rng") / "smc_rng.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, os.path.join(ROOT, "tests", "hostsim", "smc_rng.cpp")],
                   check=True)
    lib = C.CDLL(so)
    lib.sr_stage_uniform.argtypes = [C.c_ulonglong, C.c_ulonglong]
    lib.sr_stage_uniform.restype = C.c_double
    return lib


def test_host_compiled_stage_uniform_matches_the_restatement(smc_rng):
    rng = np.random.RandomState(3)
    pairs = [(0, 0), (1, 0), (0, 1), ((1 << 64) - 1, (1 << 64) - 1), (5, 1 << 33)]
    pairs += [(int(s), int(t)) for s, t in zip(rng.randint(0, 1 << 62, 200, dtype=np.int64), rng.randint(0, 1 << 40, 200))]
    us = []
    for seed, stage in pairs:
        got = smc_rng.sr_stage_uniform(seed, stage)
        assert got == R.stage_uniform(seed, stage), (seed, stage)
        us.append(got)
    assert 0.0 < min(us) and max(us) < 1.0 and len(set(us)) == len(us)
    # word 7 is nobody else's: the choice uniform of the same counter (word 6) differs
    assert R.stage_uniform(9, 4) != float(E.u01(*E._block(9, 4, np.zeros(1, np.uint64), 6)[:2])[0])


# ---- the restatement's primitives ---------------------------------------------------------------------------------
def test_restated_ancestors_follow_the_weights():
    rng = np.random.RandomState(0)
    for n in (1, 2, 63, 64, 65, 1000, 4097):
        w = rng.exponential(size=n) * (rng.rand(n) < 0.7)
        if not w.any():
            w[-1] = 1.0
        cum, total = R.prefix_sum(w)
        assert total == cum[-1] and (np.diff(cum) >= 0).all() and abs(total - math.fsum(w)) <= 1e-12 * total
        a = R.ancestors(w, 7, 3)
        assert (w[a] > 0).all()
        counts = np.bincount(a, minlength=n)
        assert (np.abs(counts - n * w / total) <= 1.0 + 1e-9).all()
    assert np.array_equal(R.ancestors(np.zeros(5), 1, 1), np.arange(5))
    m, w, s1, s2 = R.smc_weights([-np.inf, np.nan, 3.0, 1.0, np.inf], 0.5)
    assert m == 3.0 and np.array_equal(w, [0.0, 0.0, 1.0, np.exp(-1.0), 0.0]) and s1 == 1.0 + np.exp(-1.0)
    assert R.smc_weights([-np.inf] * 3, 1.0)[::2] == (-math.inf, 0.0)


# ---- the sampler on the restatement ---------------------------------------------------------------------------------
def test_smc_gaussian_recovers_evidence_and_sigmas():
    """2048 particles from the box prior: ln Z within 4 Monte Carlo standard deviations of the closed form, and every
    axis's mean and sigma within 4 standard errors (effective population N / 2)."""
    assert abs(LN_Z_GAUSS - (-8.987)) < 1e-3
    n = 2048
    for seed in (0, 1, 2):
        p0 = np.random.RandomState(seed).uniform(-BOX, BOX, (n, 3))
        smc, res = _smc(gauss_box_lnprob, n, 3, seed, p0)
        sd = lnz_sd(res, n)
        assert abs(res.log_evidence - LN_Z_GAUSS) < 4 * sd, (seed, res.log_evidence, sd)
        c = res.coords.numpy()
        n_eff = n / 2
        assert (np.abs(c.mean(axis=0)) < 4 * SIG / np.sqrt(n_eff)).all(), c.mean(axis=0)
        assert (np.abs(c.std(axis=0) / SIG - 1.0) < 4 / np.sqrt(2 * n_eff)).all(), c.std(axis=0)
        assert res.betas[-1] == 1.0 and (np.diff(res.betas) > 0).all() and res.n_stages >= 2
        assert (res.ess >= 0.5 * n * (1 - 1e-12)).all() and (res.ess <= n).all()
        assert (res.steps >= 2).all() and (res.steps <= 50).all() and res.final_steps >= 2
        assert res.n_evaluations == n * (1 + res.steps.sum() + res.final_steps)
        assert smc.step == res.steps.sum() + res.final_steps
        assert np.array_equal(res.lnp.numpy(), gauss_box_lnprob(c))


def two_modes_lnprob(q):
    """0.3 N((-4, 0), 0.5^2 I) + 0.7 N((4, 0), 0.5^2 I) in the box [-10, 10]^2: 16 sigma apart."""
    q = np.asarray(q)
    r1 = ((q - [-4.0, 0.0]) ** 2).sum(axis=1) / 0.25
    r2 = ((q - [4.0, 0.0]) ** 2).sum(axis=1) / 0.25
    lnl = np.logaddexp(np.log(0.3) - 0.5 * r1, np.log(0.7) - 0.5 * r2) - np.log(2 * np.pi * 0.25)
    return np.where(np.all(np.abs(q) <= BOX, axis=1), lnl, -np.inf)


def test_smc_weighs_two_separated_modes():
    """The final population splits 0.3 / 0.7 between two modes 16 sigma apart, within 4 binomial standard deviations
    (a single ensemble chain started in one mode stays there)."""
    n = 4096
    for seed in (0, 1):
        p0 = np.random.RandomState(10 + seed).uniform(-BOX, BOX, (n, 2))
        _, res = _smc(two_modes_lnprob, n, 2, seed, p0)
        frac = float((res.coords.numpy()[:, 0] < 0).mean())
        assert abs(frac - 0.3) < 4 * math.sqrt(0.3 * 0.7 / n), (seed, frac)
        assert abs(res.log_evidence - (-2 * math.log(2 * BOX))) < 4 * lnz_sd(res, n)


def test_smc_is_deterministic_per_seed():
    n = 256
    p0 = np.random.RandomState(4).uniform(-BOX, BOX, (n, 3))
    out = [_smc(gauss_box_lnprob, n, 3, seed, p0, moves=mv)[1] for seed, mv in ((5, None), (5, None), (6, None),
                                                                                  (5, StretchMove()))]
    a, b = out[0], out[1]
    assert np.array_equal(a.coords.numpy(), b.coords.numpy()) and np.array_equal(a.lnp.numpy(), b.lnp.numpy())
    assert a.log_evidence == b.log_evidence and np.array_equal(a.betas, b.betas) and np.array_equal(a.steps, b.steps)
    for other in out[2:]:
        assert not np.array_equal(a.coords.numpy(), other.coords.numpy()) and a.log_evidence != other.log_evidence


def test_smc_sampler_arguments():
    f = gauss_box_lnprob
    for kw in (dict(target_ess=0.0), dict(target_ess=1.0), dict(target_ess=np.nan), dict(target_ess=-0.5),
               dict(p_move=1.0), dict(p_move=0.0), dict(min_steps=0), dict(min_steps=5, max_steps=4), dict(max_steps=2.5),
               dict(dist=object()), dict(moves=[]), dict(moves=StretchMove(1.0))):
        with pytest.raises(ValueError):
            SMCSampler(R.NumpyBackend(f), 64, 3, device="cpu", **kw)
    smc = SMCSampler(R.NumpyBackend(f), 64, 3, device="cpu")
    assert [(type(m).__name__, w) for m, w in smc.moves] == [("DEMove", 0.8), ("DESnookerMove", 0.2)]
    with pytest.raises(NotImplementedError):
        smc.run_until_converged(10)
    with pytest.raises(RuntimeError):
        smc.run(np.full((64, 3), 2 * BOX))                    # no particle inside the box: no finite lnp
    with pytest.raises(RuntimeError):
        smc.run(np.random.RandomState(0).uniform(-BOX, BOX, (64, 3)), max_stages=1)
    assert [smc._steps_for(a) for a in (0.0, 1.0, 0.5, 0.01, 0.99)] == [50, 2, 7, 50, 2]


# ---- the C ABI without a GPU ---------------------------------------------------------------------------------------
def test_smc_header_declares_the_smc_exports(built):
    import re
    from magprop_b200 import _capi as A
    src = open(os.path.join(ROOT, "include", "magprop_smc.h")).read()
    names = sorted(set(re.findall(r"\b(mp_[a-z0-9_]+)\s*\(", re.sub(r"/\*.*?\*/", "", src, flags=re.S))))
    assert names == sorted(A.SMC_EXPORTS) and not set(names) & set(A.EXPORTS)
    lib = A.load()
    for nm in names:
        assert hasattr(lib, nm), nm
    assert f"#define MP_SMC_TILE {A.MP_SMC_TILE}" in src and R.TILE == A.MP_SMC_TILE


def test_capi_smc_argument_checks_without_device(built):
    """Every argument check of the three entry points: MP_ERR_BAD_ARG with its own message, before any device work.
    The pointers are fake, so no call may reach a device: the handle is null and the device index is -1, on which a call
    that passed every check fails before it touches a GPU."""
    from magprop_b200 import _capi as A
    lib = A.load()
    out = np.empty(3)

    def weights(lnp=0x1000, n=8, dbeta=0.5, o=True):
        rc = lib.mp_smc_weights(lnp, n, dbeta, None, A.ptr(out) if o else None, -1, None)
        return rc, lib.mp_last_error().decode()

    for kw, word in ((dict(lnp=None), "null"), (dict(o=False), "null"), (dict(n=0), "n must"), (dict(n=-5), "n must"),
                     (dict(dbeta=-1e-300), "dbeta"), (dict(dbeta=np.nan), "dbeta"), (dict(dbeta=np.inf), "dbeta")):
        rc, msg = weights(**kw)
        assert rc == A.MP_ERR_BAD_ARG and word in msg, (kw, msg)

    n, d = 100, 3
    base = dict(w=0x10000, n=n, ndim=d, ci=0x20000, li=0x30000, co=0x40000, lo=0x50000, anc=0x60000)

    def resample(**kw):
        a = dict(base, **kw)
        rc = lib.mp_smc_resample(a["w"], a["n"], a["ndim"], 1, 2, a["ci"], a["li"], a["co"], a["lo"], a["anc"], -1, None)
        return rc, lib.mp_last_error().decode()

    cases = [(dict(w=None), "null"), (dict(ci=None), "null"), (dict(li=None), "null"), (dict(co=None), "null"),
             (dict(lo=None), "null"), (dict(n=0), "n must"), (dict(n=-1), "n must"), (dict(ndim=0), "ndim"),
             (dict(ndim=10), "ndim"),
             (dict(co=0x20000 + n * d * 8 - 8), "overlaps an input"),          # coords_out's first row = coords_in's last
             (dict(lo=0x10000 + 8 * (n - 1)), "overlaps an input"),           # lnp_out starts at w's last entry
             (dict(anc=0x30000), "overlaps an input"), (dict(co=0x30000 - 8), "overlaps an input"),
             (dict(lo=0x40000 + 8), "two outputs"), (dict(anc=0x50000 + 8 * n - 8), "two outputs")]
    for kw, word in cases:
        rc, msg = resample(**kw)
        assert rc == A.MP_ERR_BAD_ARG and word in msg, (kw, msg)
    # adjacent ranges do not overlap, and a null ancestors array is allowed: these pass every check and stop at device -1
    for kw in (dict(), dict(co=0x20000 + n * d * 8), dict(anc=None), dict(lo=0x10000 + 8 * n)):
        rc, msg = resample(**kw)
        assert rc == A.MP_ERR_CUDA and "no such CUDA device" in msg, (kw, msg)
    rc, msg = weights()
    assert rc == A.MP_ERR_CUDA and "no such CUDA device" in msg, msg

    def desc(**kw):
        e = A.Ensemble()
        e.coords, e.lnp, e.nwalkers, e.ndim, e.a, e.seed, e.world = 0x1000, 0x2000, 8, 6, 2.0, 1, 1
        for k, v in kw.items():
            setattr(e, k, v)
        return e

    moves = (A.Move * 1)((A.MP_MOVE_DE, 0, 1.0, 0.0, 0.0, 1e-5, 0.0))

    def annealed(e=None, beta=0.5, split=0, mv=moves, nm=1):
        e = desc() if e is None else e
        rc = lib.mp_annealed_moves_half_step(None, C.byref(e), beta, C.addressof(mv) if mv is not None else None, nm, 0,
                                             split, None)
        return rc, lib.mp_last_error().decode()

    for kw, word in ((dict(beta=0.0), "beta"), (dict(beta=-0.5), "beta"), (dict(beta=1.0 + 1e-15), "beta"),
                     (dict(beta=np.nan), "beta"), (dict(beta=np.inf), "beta"), (dict(split=2), "split"),
                     (dict(mv=None), "n_moves"), (dict(nm=0), "n_moves"),
                     (dict(e=desc(world=2)), "one rank"), (dict(e=desc(n_peers=1)), "one rank"),
                     (dict(e=desc(pack_out=0x3000)), "one rank"), (dict(e=desc(ndim=0)), "ndim"),
                     (dict(e=desc(ndim=10)), "ndim"), (dict(e=desc(nwalkers=7)), "even"),
                     (dict(e=desc(coords=None)), "null ensemble"), (dict(e=desc(nwalkers=2)), "partners")):
        rc, msg = annealed(**kw)
        assert rc == A.MP_ERR_BAD_ARG and word in msg, (kw, msg)
    for beta in (1e-300, 0.37, 1.0):
        rc, msg = annealed(beta=beta)
        assert rc == A.MP_ERR_BAD_ARG and "null handle" in msg, (beta, msg)


# ---- on the GPU ---------------------------------------------------------------------------------------------------
def _ulps(a, b):
    """|a - b| in units of the spacing at b (0 where both are 0)."""
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where((a == 0) & (b == 0), 0.0, np.abs(a - b) / np.spacing(np.abs(b)))


@pytest.mark.gpu
def test_smc_weights_match_numpy(built):
    import torch
    from magprop_b200.engine import smc_weights
    rng = np.random.RandomState(1)
    side = torch.cuda.Stream()
    for n in (1, 2, 255, 256, 257, 1184 * 256 - 1, 1184 * 256, 1184 * 256 + 1, (1 << 20) + 17):
        lnp = -(10.0 ** rng.uniform(-1.0, 9.0, n))          # lnp over 10 decades, as prior draws give
        if n > 2:
            lnp[rng.rand(n) < 0.05] = -np.inf
            lnp[rng.randint(n)] = np.nan
        d_lnp = torch.as_tensor(lnp, device="cuda")
        for dbeta in (0.0, 1e-12, 1e-9, 1e-6, 1e-3, 0.37, 1.0):
            m, w_np, _, _ = R.smc_weights(lnp, dbeta)
            d_w = torch.empty(n, dtype=torch.float64, device="cuda")
            got = smc_weights(d_lnp.data_ptr(), n, dbeta, d_w.data_ptr())
            w = d_w.cpu().numpy()
            assert got[0] == m, (n, dbeta)
            assert _ulps(w, w_np).max() <= 2, (n, dbeta, _ulps(w, w_np).max())
            s1, s2 = math.fsum(w), math.fsum(w * w)
            assert abs(got[1] - s1) <= 1e-13 * s1 and abs(got[2] - s2) <= 1e-13 * s2, (n, dbeta, got, s1, s2)
            assert smc_weights(d_lnp.data_ptr(), n, dbeta) == got
            with torch.cuda.stream(side):
                d_w2 = torch.empty(n, dtype=torch.float64, device="cuda")
                got2 = smc_weights(d_lnp.data_ptr(), n, dbeta, d_w2.data_ptr(), stream=side.cuda_stream)
            torch.cuda.synchronize()
            assert got2 == got and torch.equal(d_w2, d_w)
    for n in (1, 300):
        d = torch.full((n,), -np.inf, dtype=torch.float64, device="cuda")
        assert smc_weights(d.data_ptr(), n, 0.5) == (-math.inf, 0.0, 0.0)


@pytest.mark.gpu
def test_smc_resample_matches_the_restatement(built):
    """Fed the device's own weights, the ancestors and gathered rows equal the restatement's bit for bit; every count lies
    within 1 of n w_j / total, and no particle of weight 0 is drawn."""
    import torch
    from magprop_b200.engine import smc_resample, smc_weights
    rng = np.random.RandomState(2)
    side = torch.cuda.Stream()
    for n, ndim in ((1, 6), (2, 1), (63, 9), (65, 6), (1000, 6), (4097, 3), (1 << 24, 2)):
        lnp = -(10.0 ** rng.uniform(-1.0, 3.0, n))
        if n > 1:
            lnp[rng.rand(n) < 0.1] = -np.inf
        d_lnp = torch.as_tensor(lnp, device="cuda")
        d_w = torch.empty(n, dtype=torch.float64, device="cuda")
        smc_weights(d_lnp.data_ptr(), n, 0.05, d_w.data_ptr())
        coords = torch.arange(n * ndim, dtype=torch.float64, device="cuda").view(n, ndim)
        outs = []
        for st in (torch.cuda.current_stream(), side):
            with torch.cuda.stream(st):
                c_out = torch.empty_like(coords)
                l_out = torch.empty_like(d_lnp)
                anc = torch.empty(n, dtype=torch.int64, device="cuda")
                smc_resample(d_w.data_ptr(), n, ndim, 77, n + 3, coords.data_ptr(), d_lnp.data_ptr(), c_out.data_ptr(),
                             l_out.data_ptr(), anc.data_ptr(), stream=st.cuda_stream)
            torch.cuda.synchronize()
            outs.append((anc.cpu().numpy(), c_out.cpu().numpy(), l_out.cpu().numpy()))
        a, c, lo = outs[0]
        assert all(np.array_equal(x, y) for x, y in zip(outs[0], outs[1]))
        w = d_w.cpu().numpy()
        want = R.ancestors(w, 77, n + 3)
        assert np.array_equal(a, want), (n, np.flatnonzero(a != want)[:5])
        assert np.array_equal(c, np.arange(n * ndim, dtype=np.float64).reshape(n, ndim)[want]) and np.array_equal(lo, lnp[want])
        total = R.prefix_sum(w)[1]
        assert (w[a] > 0).all()
        assert (np.abs(np.bincount(a, minlength=n) - n * w / total) <= 1.0 + 1e-6).all()
        del coords, c_out, outs
    # a zero total (which the driver never passes): a_i = i
    z = torch.zeros(5, dtype=torch.float64, device="cuda")
    c_in = torch.arange(5.0, dtype=torch.float64, device="cuda")[:, None]
    c_out, l_out, anc = torch.empty_like(c_in), torch.empty_like(z), torch.empty(5, dtype=torch.int64, device="cuda")
    smc_resample(z.data_ptr(), 5, 1, 1, 1, c_in.data_ptr(), z.data_ptr(), c_out.data_ptr(), l_out.data_ptr(), anc.data_ptr())
    torch.cuda.synchronize()
    assert anc.cpu().tolist() == list(range(5)) and torch.equal(c_out, c_in)


def _humped(golden):
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, time_grid
    from oracle import magprop_oracle as O
    g = golden["lnprob_script"]
    return Likelihood(A.script_model_spec(), time_grid(None), g["Humped_x"], g["Humped_y"], g["Humped_yerr"],
                      O.SCRIPT_LOWER, O.SCRIPT_UPPER)


def _ball(n, seed, sigma=1e-2):
    from oracle import magprop_oracle as O
    return O.SYNTH_TRUTHS_LOG["Humped"] + sigma * np.random.RandomState(seed).randn(n, 6)


def _prior_wide(n, seed):
    """Half a ball, half spread over the prior box: the spread half feeds the stiff queue."""
    from oracle import magprop_oracle as O
    rng = np.random.RandomState(seed)
    p = np.concatenate([_ball(n // 2, seed, 0.05), O.SCRIPT_LOWER + (O.SCRIPT_UPPER - O.SCRIPT_LOWER) * rng.rand(n - n // 2, 6)])
    return p[rng.permutation(n)]


KINDS = {"stretch": StretchMove(), "de": DEMove(), "snooker": DESnookerMove(), "mix": [(DEMove(), 0.8), (DESnookerMove(), 0.2)]}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(KINDS))
def test_annealed_half_step_matches_the_restatement(built, golden, kind):
    """At beta = 1e-9, 0.37 and 1, 64 walkers from the ball and 16 384 prior-wide walkers (8192 movers: the ordered
    work list, the stiff queue) equal the restatement with the ladder [beta] bit for bit, half-step by half-step; at
    beta = 1 the run equals mp_ensemble_moves_half_step's."""
    import torch
    lk = _humped(golden)
    for n, p0, nsteps in ((64, _ball(64, 7), 3), (16384, _prior_wide(16384, 8), 2 if kind == "mix" else 1)):
        for beta in (1e-9, 0.37, 1.0):
            smc = SMCSampler.from_likelihood(lk, n, 6, seed=5, moves=KINDS[kind])
            smc.beta = beta
            smc.initialise(p0)
            torch.cuda.synchronize()
            coords, lnp = p0.copy(), smc.lnp.cpu().numpy().copy()
            acc = np.zeros(n, np.int32)
            stiff = []
            for step in range(nsteps):
                mv = E.step_move(smc.moves, 5, step)
                for split in (0, 1):
                    smc.backend.annealed_half_step(smc, step, split)
                    stiff.append(lk.last_stiff_count())
                    t, rows, comp = E.tempered_rows(n, 1, 5, step, split)
                    E.half_step(coords, lnp, rows, t, comp, mv, 5, 2 * step + split, lk.lnprob, betas=[beta], accepted=acc)
                    assert np.array_equal(smc.coords.cpu().numpy(), coords), (n, beta, step, split)
                    assert np.array_equal(smc.lnp.cpu().numpy(), lnp), (n, beta, step, split)
            assert np.array_equal(smc.accepted.cpu().numpy(), acc) and acc.sum() > 0
            if n > 64:
                assert min(stiff) > 0, stiff
            if beta == 1.0:
                ens = DeviceEnsemble.from_likelihood(lk, n, 6, seed=5, moves=KINDS[kind])
                ens.initialise(p0)
                for step in range(nsteps):
                    for split in (0, 1):
                        ens.backend.half_step(ens, step, split)
                torch.cuda.synchronize()
                for a, b in ((ens.coords, smc.coords), (ens.lnp, smc.lnp), (ens.accepted, smc.accepted), (ens.status, smc.status)):
                    assert torch.equal(a, b)
    lk.close()


# Seed-to-seed standard deviation (ddof = 1) of ln Z on Sloped with 2^14 particles and run_smc's defaults: 8 seeds of
# tools/smc_bench.py, profiles/r06_smc_bench.txt (one NVIDIA B200, 1000 W power limit).
SLOPED_LNZ_SD_2P14 = 0.1844


def _student_t_is(res, x, y, yerr, n_draws=1 << 22, nu=5.0, seed=11):
    """Importance sampling of Sloped's evidence: draws from a multivariate Student-t fitted to the SMC final population,
    evaluated by the device likelihood.  Returns (ln Z, its standard error, ESS, draws, normalised weights)."""
    import torch
    from math import lgamma, log, pi
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, chain_moments, time_grid
    from magprop_b200.synthetic.mcmc_eqns import lower, upper
    flat = res.chain_device.reshape(-1, 6).contiguous()
    mu, cov = chain_moments(flat.data_ptr(), flat.shape[0], 6)
    L = np.linalg.cholesky(cov * (nu - 2.0) / nu)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    z = torch.randn((n_draws, 6), dtype=torch.float64, device="cuda", generator=gen)
    chi = (torch.randn((n_draws, int(nu)), dtype=torch.float64, device="cuda", generator=gen) ** 2).sum(dim=1) / nu
    draws = (torch.as_tensor(mu, device="cuda") + (z @ torch.as_tensor(L.T, device="cuda")) / chi.sqrt()[:, None]).contiguous()
    lk = Likelihood(A.script_model_spec(), time_grid(None), x, y, yerr, lower, upper)
    lnp = torch.empty(n_draws, dtype=torch.float64, device="cuda")
    lk.lnprob_device(draws.data_ptr(), n_draws, 6, lnp.data_ptr())
    torch.cuda.synchronize()
    lk.close()
    sol = torch.linalg.solve_triangular(torch.as_tensor(L, device="cuda"), (draws - torch.as_tensor(mu, device="cuda")).T,
                                        upper=False)
    maha = (sol * sol).sum(dim=0)
    lq = (lgamma((nu + 6) / 2) - lgamma(nu / 2) - 3 * log(nu * pi) - float(np.log(np.diag(L)).sum())
          - (nu + 6) / 2 * torch.log1p(maha / nu))
    lw = (lnp - float(np.log(upper - lower).sum()) - lq).cpu().numpy()
    m = lw[np.isfinite(lw)].max()
    wts = np.where(np.isfinite(lw), np.exp(lw - m), 0.0)
    ess = wts.sum() ** 2 / (wts ** 2).sum()
    return m + np.log(wts.mean()), wts.std() / np.sqrt(n_draws) / wts.mean(), ess, draws.cpu().numpy(), wts / wts.sum()


@pytest.mark.gpu
def test_run_smc_on_sloped_matches_importance_sampling(built, golden):
    """run_smc on Sloped with 2^14 particles: the same seed gives the same bits, on a side stream too; ln Z agrees with
    an importance-sampling estimate within 4 seed standard deviations (SLOPED_LNZ_SD_2P14), and the final population's
    mean and sigma of every parameter with the IS-weighted ones within 4 Monte Carlo standard errors."""
    import time

    import torch
    from magprop_b200.synthetic.synth_mcmc import run_smc
    g = golden["lnprob_script"]
    x, y, yerr = g["Sloped_x"], g["Sloped_y"], g["Sloped_yerr"]
    n = 1 << 14
    runs = []
    for use_side in (False, False, True):
        st = torch.cuda.Stream() if use_side else torch.cuda.current_stream()
        t0 = time.perf_counter()
        with torch.cuda.stream(st):
            res = run_smc("Sloped", x, y, yerr, n, seed=3)
        torch.cuda.synchronize()
        runs.append((res, time.perf_counter() - t0))
    res = runs[0][0]
    for other, _ in runs[1:]:
        assert torch.equal(other.chain_device, res.chain_device) and torch.equal(other.lnp_device, res.lnp_device)
        assert other.log_evidence == res.log_evidence and np.array_equal(other.betas, res.betas)
    assert res.get_chain().shape == (1, n, 6) and res.betas[-1] == 1.0
    log_z_is, sigma_is, ess, draws, wn = _student_t_is(res, x, y, yerr)
    pop = res.get_chain()[0]
    mean_is = wn @ draws
    sd_is = np.sqrt(wn @ (draws - mean_is) ** 2)
    n_eff = n / 4                                     # resampled, then mutated: at least a quarter of the particles
    mean_err = np.abs(pop.mean(axis=0) - mean_is) / (sd_is * np.sqrt(1 / n_eff + 1 / ess))
    sd_err = np.abs(pop.std(axis=0) / sd_is - 1.0) / np.sqrt(1 / (2 * n_eff) + 1 / (2 * ess))
    print(f"Sloped SMC 2^14: ln Z {res.log_evidence:.4f}, IS {log_z_is:.4f} +- {sigma_is:.4f} (ESS {ess:.0f}); "
          f"{res.betas.size} stages, {res.n_evaluations} evaluations, {runs[0][1]:.2f} s per run; "
          f"mean errors {np.round(mean_err, 2).tolist()}, sigma errors {np.round(sd_err, 2).tolist()}")
    assert ess >= 1000
    assert abs(res.log_evidence - log_z_is) <= 4 * math.hypot(SLOPED_LNZ_SD_2P14, sigma_is)
    assert mean_err.max() < 4 and sd_err.max() < 4
