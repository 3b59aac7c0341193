"""emcee 3's KDEMove on the device ensembles: the host-compiled Gaussian draws equal the NumPy restatement bit for bit and
a high-precision Box-Muller closely, the constants and every argument check hold without a GPU, and the restatement
samples known Gaussians, relaxes two separated modes to their weights and gives SMC the right evidence (CPU); the
kernels equal the restatement bit for bit across the launch paths, streams do not matter, a degenerate complement
leaves its movers in place, and SMC with the KDE move agrees with importance sampling on Sloped (GPU)."""
import ctypes as C
import math
import os

import numpy as np
import pytest

import ensemble_ref as E
import kde_ref as K
import test_moves as TM
import test_smc as TS
from conftest import ROOT
from magprop_b200.sampler import (DEMove, DESnookerMove, DeviceEnsemble, KDEMove, SMCSampler, TemperedEnsemble,
                                  move_table)

KDE_MIX = [(KDEMove(), 0.5), (DEMove(), 0.4), (DESnookerMove(), 0.1)]
KINDS = {"kde": KDEMove(), "kde_mix": KDE_MIX}


# ---- the restatement with the KDE move (kde_ref) driving the samplers on the CPU -------------------------------------
def sample_gaussian(d, moves, nsteps, nwalkers, seed=1):
    """test_moves.sample_gaussian with kde_ref's backend."""
    mu, cov, lnprob = TM.gaussian(d)
    rng = np.random.RandomState(seed)
    p0 = mu + 0.1 * rng.multivariate_normal(np.zeros(d), cov, size=nwalkers)
    ens = DeviceEnsemble(K.NumpyBackend(lnprob), nwalkers, d, seed=seed, device="cpu", moves=moves)
    ens.set_state(p0, lnprob(p0))
    chain, _ = ens.run(nsteps, store=True)
    return mu, cov, chain.numpy()[nsteps // 4:], ens


def _smc(fn, n, ndim, seed, p0, **kw):
    smc = SMCSampler(K.SMCBackend(fn), n, ndim, seed=seed, device="cpu", **kw)
    return smc, smc.run(p0)


def _check_against_restatement(lk, fn, n, p0, moves, seed, nsteps, ntemps=1, betas=None):
    """test_moves._check_against_restatement with kde_ref's half-step: the device ensemble half-step by half-step and
    the restatement beside it, every state equal.  Returns the stiff count of every device half-step and the move kind
    of every step."""
    import torch
    if betas is None:
        ens = DeviceEnsemble.from_likelihood(lk, n, 6, seed=seed, moves=moves)
    else:
        ens = TemperedEnsemble.from_likelihood(lk, n, 6, betas, seed=seed, moves=moves)
    ens.initialise(p0)
    torch.cuda.synchronize()
    coords = p0.reshape(-1, 6).copy()
    lnp = ens.lnp.cpu().numpy().copy()
    acc = np.zeros(coords.shape[0], np.int32)
    stiff, kinds = [], []
    half = n // 2
    for step in range(nsteps):
        mv = E.step_move(ens.moves, seed, step)
        kinds.append(mv.kind)
        for split in (0, 1):
            x0 = coords.copy()
            if betas is None:
                ens.backend.half_step(ens, step, split)
                stiff.append(lk.last_stiff_count())          # (synchronises: the launch is complete)
                order = E.ensemble_order(n, seed, step)
                rows = order[split * half:(split + 1) * half]
                comp = order[(1 - split) * half:(2 - split) * half][None, :]
                q, a = K.half_step(coords, lnp, rows, np.zeros(half, np.int64), comp, mv, seed, 2 * step + split, fn,
                                   accepted=acc)
            else:
                ens.backend.tempered_half_step(ens, step, split)
                stiff.append(lk.last_stiff_count())
                t, rows, comp = E.tempered_rows(n, ntemps, seed, step, split)
                q, a = K.half_step(coords, lnp, rows, t, comp, mv, seed, 2 * step + split, fn, betas=betas, accepted=acc)
            got = ens.coords.cpu().numpy()
            assert np.array_equal(got, coords), (step, split, TM._mismatch(got, coords, x0, rows, q, a, n))
            assert np.array_equal(ens.lnp.cpu().numpy(), lnp), (step, split)
        if betas is not None:
            ens.backend.tempered_swap(ens, step)
            E.swap(coords, lnp, betas, n, seed, step)
        ens.step += 1
    torch.cuda.synchronize()
    assert np.array_equal(ens.coords.cpu().numpy(), coords) and np.array_equal(ens.accepted.cpu().numpy(), acc)
    assert 0 < acc.sum() < acc.size * nsteps
    return stiff, kinds


# ---- host-compiled draws == the restatement ------------------------------------------------------------------
@pytest.fixture(scope="module")
def kde_rng(tmp_path_factory):
    """tests/hostsim/kde_rng.cpp -- the KDE move's draws of magprop_rng.cuh -- built for the host."""
    import subprocess
    so = str(tmp_path_factory.mktemp("kde_rng") / "kde_rng.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "kde_rng.cpp")], check=True)
    lib = C.CDLL(so)
    vp = C.c_void_p
    lib.kr_gauss_pair.argtypes = [vp, vp, C.c_long, vp, vp]
    lib.kr_draws.argtypes = [C.c_ulonglong, C.c_ulonglong, C.c_uint, C.c_long, C.c_int, vp, vp, vp]
    return lib


def _host_gauss(lib, u1, u2):
    z0, z1 = np.empty(u1.size), np.empty(u1.size)
    lib.kr_gauss_pair(u1.ctypes.data, u2.ctypes.data, u1.size, z0.ctypes.data, z1.ctypes.data)
    return z0, z1


def test_host_compiled_kde_draws_match_the_restatement(kde_rng):
    """2^20 counters at ndim 9 (five Box-Muller pairs each) and a few seeds and half-steps at every ndim."""
    cases = [(7, 3, 0, 1 << 20, 9), ((1 << 64) - 1, (1 << 40) + 5, (1 << 31) - 100, 100, 9)]
    cases += [(12345 + d, 17 * d, 1000 * d, 2000, d) for d in range(1, 10)]
    for seed, hs, me0, n, d in cases:
        uc, z, ua = np.empty(n), np.empty((n, d)), np.empty(n)
        kde_rng.kr_draws(seed, hs, me0, n, d, uc.ctypes.data, z.ctypes.data, ua.ctypes.data)
        rows = np.arange(me0, me0 + n, dtype=np.uint64)
        ruc, rz = K.kde_draws(seed, hs, rows, d)
        assert np.array_equal(uc, ruc) and np.array_equal(z, rz), (seed, hs, d)
        assert np.array_equal(ua, K.accept_uniform(K.KDE, seed, hs, rows)), (seed, hs, d)
        assert np.isfinite(z).all()
    # words 8 .. 13 are the KDE move's own: its accept uniform is none of the other kinds'
    rows = np.arange(1000, dtype=np.uint64)
    ua = K.accept_uniform(K.KDE, 5, 9, rows)
    for kind in (E.STRETCH, E.DE, E.SNOOKER):
        assert not np.isin(ua, E.accept_uniform(kind, 5, 9, rows)).any()
    # edge uniforms: the extremes of u01, the quadrant boundaries and the reflection point
    u = np.array([0.5 / 2 ** 53, 1.0 - 0.5 / 2 ** 53, 0.25, 0.5, 0.75, 0.125, 0.375, 1e-300 + 0.5 / 2 ** 53,
                  math.sqrt(0.5), 0.7071067811865476, 0.7071067811865475, 0.999999, 1e-6])
    u1, u2 = np.repeat(u, u.size), np.tile(u, u.size)
    for a, b in zip(_host_gauss(kde_rng, u1, u2), K.gauss_pair(u1, u2)):
        assert np.array_equal(a, b)


def test_gauss_pair_is_accurate_and_normal(kde_rng):
    """Within 1e-14 max(1, |z|) of Box-Muller in 50-digit arithmetic; the first and second members pass a KS test
    against N(0, 1) and are uncorrelated."""
    import mpmath
    from scipy import stats
    rng = np.random.RandomState(11)
    u1 = np.concatenate([rng.rand(3000), 10.0 ** -rng.uniform(0, 16, 500), 1.0 - 10.0 ** -rng.uniform(1, 15, 500)])
    u2 = np.concatenate([rng.rand(3500), np.arange(500) / 500.0 + 0.5 / 2 ** 53])
    z0, z1 = _host_gauss(kde_rng, u1, u2)
    mpmath.mp.dps = 50
    worst = 0.0
    for a, b, g0, g1 in zip(u1, u2, z0, z1):
        r = mpmath.sqrt(-2 * mpmath.log(mpmath.mpf(float(a))))
        th = 2 * mpmath.pi * mpmath.mpf(float(b))
        for got, want in ((g0, r * mpmath.cos(th)), (g1, r * mpmath.sin(th))):
            worst = max(worst, float(abs(mpmath.mpf(float(got)) - want)) / max(1.0, abs(float(want))))
    assert worst < 1e-14, worst
    n = 1 << 18
    b = E._block(3, 1, np.arange(n, dtype=np.uint64), 9)
    g0, g1 = K.gauss_pair(E.u01(b[0], b[1]), E.u01(b[2], b[3]))
    for g in (g0, g1):
        assert stats.kstest(g, "norm").pvalue > 1e-3
    assert abs(np.corrcoef(g0, g1)[0, 1]) < 5 / math.sqrt(n)


# ---- the C ABI and the Python layer without a GPU -----------------------------------------------------------------
def test_header_constants_match_capi(built, tmp_path):
    import subprocess
    from magprop_b200 import _capi as A
    src = tmp_path / "kde.c"
    src.write_text('#include <stdio.h>\n#include "magprop_b200.h"\n'
                   'int main(void) { printf("%d %d %d\\n", MP_MOVE_KDE, MP_KDE_MAX_CENTRES, MP_ABI_VERSION); return 0; }\n')
    exe = tmp_path / "kde"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert [int(v) for v in out] == [A.MP_MOVE_KDE, A.MP_KDE_MAX_CENTRES, 2] == [4, 4096, 2]
    assert KDEMove.kind == A.MP_MOVE_KDE


def test_capi_kde_argument_checks_without_device(built):
    """MP_ERR_BAD_ARG with each check's own message from the plain, tempered and annealed entry points, before any
    device work (the handle is null: a call that passed every check would fail on that instead)."""
    from magprop_b200 import _capi as A
    lib = A.load()
    K, D = A.MP_MOVE_KDE, A.MP_MOVE_DE

    def desc(nwalkers=16, ndim=6, world=1, rank=0, pack=None):
        e = A.Ensemble()
        e.coords, e.lnp, e.nwalkers, e.ndim, e.a, e.seed, e.world, e.rank = 0x1000, 0x2000, nwalkers, ndim, 2.0, 1, world, rank
        e.pack_out = pack
        return e

    def mv(kind, weight=1.0, gamma0=0.0):
        return (kind, 0, weight, 2.0, gamma0, 1e-5, 1.7)

    def three(table, **kw):
        arr = (A.Move * len(table))(*table)
        betas = np.array([1.0, 0.5])
        out = [lib.mp_ensemble_moves_half_step(None, C.byref(desc(**kw)), C.addressof(arr), len(table), 0, 0, None)]
        msgs = [lib.mp_last_error().decode()]
        out.append(lib.mp_tempered_moves_half_step(None, C.byref(desc(**kw)), 2, A.ptr(betas), C.addressof(arr), len(table),
                                                   0, 0, None))
        msgs.append(lib.mp_last_error().decode())
        out.append(lib.mp_annealed_moves_half_step(None, C.byref(desc(**kw)), 0.5, C.addressof(arr), len(table), 0, 0, None))
        msgs.append(lib.mp_last_error().decode())
        return out, msgs

    for g in (-1.0, np.nan, np.inf, -np.inf):
        out, msgs = three([mv(K, gamma0=g)])
        assert out == [A.MP_ERR_BAD_ARG] * 3 and all("KDE move needs a bandwidth factor" in m for m in msgs), msgs
    # a half needs ndim + 1 walkers for a weighted KDE move: 6 walkers per half at ndim 6 are too few, 7 enough
    for nwalkers, ndim, table, bad in ((12, 6, [mv(K)], True), (14, 6, [mv(K)], False), (4, 1, [mv(K)], False),
                                       (4, 2, [mv(K)], True), (12, 6, [mv(D), mv(K, weight=0.0)], False)):
        out, msgs = three(table, nwalkers=nwalkers, ndim=ndim)
        assert out == [A.MP_ERR_BAD_ARG] * 3
        assert all(("partners" in m) == bad for m in msgs), (nwalkers, ndim, msgs)
        if not bad:
            assert all("null handle" in m for m in msgs), msgs
    # one rank only: the plain entry point is the one that takes a sharded ensemble
    for kw in (dict(world=2), dict(pack=0x3000)):
        arr = (A.Move * 1)(mv(K))
        assert lib.mp_ensemble_moves_half_step(None, C.byref(desc(**kw)), C.addressof(arr), 1, 0, 0, None) == A.MP_ERR_BAD_ARG
        assert "KDE move runs on one rank" in lib.mp_last_error().decode()
        arr = (A.Move * 2)(mv(D), mv(K, weight=0.0))      # a zero-weight KDE move does not count
        assert lib.mp_ensemble_moves_half_step(None, C.byref(desc(**kw)), C.addressof(arr), 2, 0, 0, None) == A.MP_ERR_BAD_ARG
        assert "null handle" in lib.mp_last_error().decode()
    e = desc()
    e.n_peers = 1
    e.world = 2
    arr = (A.Move * 1)(mv(K))
    assert lib.mp_ensemble_moves_half_step(None, C.byref(e), C.addressof(arr), 1, 0, 0, None) == A.MP_ERR_BAD_ARG
    assert "KDE move runs on one rank" in lib.mp_last_error().decode()


class _FakeDist:
    """Just enough of torch.distributed for DeviceEnsemble to see two ranks."""

    def is_initialized(self):
        return True

    def get_world_size(self):
        return 2

    def get_rank(self):
        return 0

    def get_backend(self):
        return "gloo"


def test_bad_kde_moves_raise_value_error():
    _, _, lnprob = TM.gaussian(3)
    for bw in ("silverman", "Scott", lambda kde: 0.5, 0.0, -1.0, np.nan, np.inf, True, [0.5], "0.5"):
        with pytest.raises(ValueError):
            move_table(KDEMove(bw))
        with pytest.raises(ValueError):
            DeviceEnsemble(K.NumpyBackend(lnprob), 16, 3, device="cpu", moves=KDEMove(bw))
    with pytest.raises(ValueError):                 # a half of 3 < ndim + 1 = 4
        DeviceEnsemble(K.NumpyBackend(lnprob), 6, 3, device="cpu", moves=KDEMove())
    with pytest.raises(ValueError):
        TemperedEnsemble(K.NumpyBackend(lnprob), 6, 3, [1.0, 0.5], device="cpu", moves=[DEMove(), KDEMove()])
    with pytest.raises(ValueError):
        SMCSampler(K.SMCBackend(lnprob), 6, 3, device="cpu", moves=KDEMove())
    with pytest.raises(ValueError):
        DeviceEnsemble(K.NumpyBackend(lnprob), 16, 3, device="cpu", dist=_FakeDist(), moves=KDE_MIX)
    with pytest.raises(ValueError):
        move_table(KDEMove(), half=3, ndim=3)
    DeviceEnsemble(K.NumpyBackend(lnprob), 8, 3, device="cpu", moves=KDEMove())
    DeviceEnsemble(K.NumpyBackend(lnprob), 6, 3, device="cpu", moves=[DEMove(), (KDEMove(), 0.0)])
    move_table(KDEMove(), half=3)                   # without ndim: two centres
    _, arr = move_table([KDEMove(), KDEMove("scott"), KDEMove(0.3), (KDEMove(np.float32(2.0)), 2.0)])
    assert [(m.kind, m.weight, m.gamma0) for m in arr] == [(4, 1.0, 0.0), (4, 1.0, 0.0), (4, 1.0, 0.3), (4, 2.0, 2.0)]


# ---- the restatement samples known targets ------------------------------------------------------------------------
@pytest.mark.parametrize("d", [2, 6])
def test_restatement_samples_correlated_gaussians(d):
    """The Gaussians of test_moves: correlation 0.99, scales over three decades."""
    mu, cov, chain, ens = sample_gaussian(d, KDEMove(), nsteps=3000, nwalkers=32 * (d // 2))
    tau = TM.assert_recovers(mu, cov, chain)
    assert tau.max() < 20, tau
    acc = float(ens.acceptance_fraction().mean())
    assert 0.2 < acc < 1.0, acc


def test_restatement_keeps_a_gaussian_with_more_walkers_than_centres():
    """8448 walkers put 4224 in each complement, more than the 4096 centres.  Started from the target itself, 8 steps
    leave it there: mean and covariance of the final population within 5 standard errors of the truth, and the
    proposals were accepted (a wrong Hastings factor over the capped centre set would shift or shrink the population)."""
    d, n = 2, 8448
    mu, cov, lnprob = TM.gaussian(d)
    p0 = np.random.RandomState(6).multivariate_normal(mu, cov, size=n)
    ens = DeviceEnsemble(K.NumpyBackend(lnprob), n, d, seed=6, device="cpu", moves=KDEMove())
    ens.set_state(p0, lnprob(p0))
    ens.run(8)
    flat = ens.coords.numpy()
    sd = np.sqrt(np.diag(cov))
    assert (np.abs(flat.mean(axis=0) - mu) / (sd / np.sqrt(n)) < 5).all()
    c = np.cov(flat.T)
    assert (np.abs(c - cov) / np.sqrt((np.outer(np.diag(cov), np.diag(cov)) + cov ** 2) / n) < 5).all()
    acc = float(ens.acceptance_fraction().mean())
    assert 0.5 < acc < 1.0, acc


def test_restatement_relaxes_two_separated_modes():
    """Walkers started 50/50 in test_smc's two modes, 16 sigma apart, end 0.3 / 0.7 within 4 binomial deviations."""
    n = 2048
    rng = np.random.RandomState(2)
    p0 = np.concatenate([[-4.0, 0.0] + 0.5 * rng.randn(n // 2, 2), [4.0, 0.0] + 0.5 * rng.randn(n // 2, 2)])
    ens = DeviceEnsemble(K.NumpyBackend(TS.two_modes_lnprob), n, 2, seed=4, device="cpu", moves=KDEMove())
    ens.set_state(p0, TS.two_modes_lnprob(p0))
    ens.run(60)
    frac = float((ens.coords.numpy()[:, 0] < 0).mean())
    assert abs(frac - 0.3) < 4 * math.sqrt(0.3 * 0.7 / n), frac


def test_smc_with_kde_recovers_the_evidence():
    """SMC with KDEMove() on the Gaussian in a box: ln Z = -8.987 within 4 Monte Carlo standard deviations."""
    n = 2048
    for seed in (0, 1):
        p0 = np.random.RandomState(seed).uniform(-TS.BOX, TS.BOX, (n, 3))
        smc, res = _smc(TS.gauss_box_lnprob, n, 3, seed, p0, moves=KDEMove())
        assert abs(res.log_evidence - TS.LN_Z_GAUSS) < 4 * TS.lnz_sd(res, n), (seed, res.log_evidence)
        c = res.coords.numpy()
        assert (np.abs(c.std(axis=0) / TS.SIG - 1.0) < 4 / np.sqrt(n)).all(), c.std(axis=0)


# ---- on the GPU ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(KINDS))
def test_kde_matches_the_restatement_small(built, golden, kind):
    """64 walkers from the ball: q, lnp and the accepted counts equal the restatement half-step by half-step."""
    lk = TM._humped(golden)
    _, kinds = _check_against_restatement(lk, lk.lnprob, 64, TM._ball(64, 7), KINDS[kind], 31, 8)
    assert K.KDE in kinds and (kind == "kde" or set(kinds) >= {K.KDE, E.DE})
    lk.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(KINDS))
def test_kde_matches_the_restatement_ordered(built, golden, kind):
    """16 384 prior-wide walkers: 8192 movers (the ordered work list, proposals copied in order_key_kernel, the stiff
    queue) against complements of 8192, of which the first 4096 are the centres."""
    lk = TM._humped(golden)
    stiff, kinds = _check_against_restatement(lk, lk.lnprob, 16384, TM._prior_wide(16384, 8), KINDS[kind], 2,
                                                 1 if kind == "kde" else 2)
    assert K.KDE in kinds and min(stiff) > 0, (kinds, stiff)
    lk.close()


@pytest.mark.gpu
def test_kde_matches_the_restatement_across_slabs(built):
    """On the dataset with data on all 10 001 nodes, 65 536 walkers move 32 768 per half-step: the KDE proposals are
    formed slab by slab."""
    import test_launch_paths as LP
    x = LP.x_wide()
    y, yerr = LP.data_for(x, 5, noise=0.05, err=0.1)
    lk = LP.script_handle(x, y, yerr)
    n = 65536
    assert n // 2 > LP.slab_bound(10001)
    rng = np.random.RandomState(405)
    p0 = np.concatenate([LP.ball(rng, n // 2, 3e-2), LP.ball(rng, n // 2, 0.3)])[rng.permutation(n)]
    fn = lambda q: LP.host_batched(lk, q)[0]
    _, kinds = _check_against_restatement(lk, fn, n, p0, KDEMove(), 4, 1)
    assert kinds == [K.KDE]
    lk.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(KINDS))
def test_tempered_kde_matches_the_restatement(built, golden, kind):
    """T = 4 x n = 2048: each temperature's own centres, factor and bandwidth."""
    from magprop_b200.sampler import geometric_betas
    lk = TM._humped(golden)
    betas = geometric_betas(4, 1e-3)
    p0 = np.stack([TM._ball(2048, 1), TM._ball(2048, 2, 0.05), TM._prior_wide(2048, 3), TM._prior_wide(2048, 4)])
    _, kinds = _check_against_restatement(lk, lk.lnprob, 2048, p0, KINDS[kind], 4, 3, ntemps=4, betas=betas)
    assert K.KDE in kinds
    lk.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(KINDS))
def test_annealed_kde_matches_the_restatement(built, golden, kind):
    """At beta = 1e-9, 0.37 and 1, 64 walkers from the ball and 16 384 prior-wide walkers equal the restatement with the
    ladder [beta]; at beta = 1 the run equals mp_ensemble_moves_half_step's."""
    import torch
    lk = TM._humped(golden)
    for n, p0, nsteps in ((64, TM._ball(64, 7), 3), (16384, TM._prior_wide(16384, 8), 1)):
        for beta in (1e-9, 0.37, 1.0):
            smc = SMCSampler.from_likelihood(lk, n, 6, seed=12, moves=KINDS[kind])
            smc.beta = beta
            smc.initialise(p0)
            torch.cuda.synchronize()
            coords, lnp = p0.copy(), smc.lnp.cpu().numpy().copy()
            acc = np.zeros(n, np.int32)
            for step in range(nsteps):
                mv = E.step_move(smc.moves, 12, step)
                for split in (0, 1):
                    smc.backend.annealed_half_step(smc, step, split)
                    t, rows, comp = E.tempered_rows(n, 1, 12, step, split)
                    K.half_step(coords, lnp, rows, t, comp, mv, 12, 2 * step + split, lk.lnprob, betas=[beta], accepted=acc)
                    assert np.array_equal(smc.coords.cpu().numpy(), coords), (n, beta, step, split)
                    assert np.array_equal(smc.lnp.cpu().numpy(), lnp), (n, beta, step, split)
            assert np.array_equal(smc.accepted.cpu().numpy(), acc) and acc.sum() > 0
            if beta == 1.0:
                ens = DeviceEnsemble.from_likelihood(lk, n, 6, seed=12, moves=KINDS[kind])
                ens.initialise(p0)
                for step in range(nsteps):
                    for split in (0, 1):
                        ens.backend.half_step(ens, step, split)
                torch.cuda.synchronize()
                for a, b in ((ens.coords, smc.coords), (ens.lnp, smc.lnp), (ens.accepted, smc.accepted)):
                    assert torch.equal(a, b)
    lk.close()


@pytest.mark.gpu
def test_kde_is_identical_when_repeated_and_on_a_side_stream(built, golden):
    import torch
    from magprop_b200.sampler import geometric_betas
    lk = TM._humped(golden)
    out = []
    for use_side in (False, False, True):
        st = torch.cuda.Stream() if use_side else torch.cuda.current_stream()
        with torch.cuda.stream(st):
            e = DeviceEnsemble.from_likelihood(lk, 128, 6, seed=8, moves=KDE_MIX)
            e.initialise(TM._ball(128, 9))
            c, l = e.run(6, store=True)
            t = TemperedEnsemble.from_likelihood(lk, 64, 6, geometric_betas(3, 1e-2), seed=8, moves=KDEMove())
            t.initialise(TM._ball(64, 10))
            tc, tl = t.run(6)
            out.append((c, l, e.accepted.clone(), e.status.clone(), tc, tl, t.accepted.clone()))
        torch.cuda.synchronize()
    for other in out[1:]:
        for a, b in zip(out[0], other):
            assert torch.equal(a, b)
    assert int(out[0][2].sum()) > 0 and int(out[0][6].sum()) > 0
    lk.close()


@pytest.mark.gpu
def test_kde_with_a_degenerate_complement_stays_put(built, golden):
    """Every walker shares one coordinate: the complement's covariance is singular, so every mover proposes its own
    position with ln f = -inf and is rejected; coords and lnp stay as they were, with no NaN.  (The shared value has
    few mantissa bits, so the sums of 32 copies are exact and the variance is exactly 0, not a rounding residue.)"""
    import torch
    lk = TM._humped(golden)
    p0 = TM._ball(64, 12)
    p0[:, 2] = np.round(TM._ball(1, 13)[0, 2] * 8.0) / 8.0
    ens = DeviceEnsemble.from_likelihood(lk, 64, 6, seed=9, moves=KDEMove())
    ens.initialise(p0)
    lnp0 = ens.lnp.clone()
    ens.run(3)
    torch.cuda.synchronize()
    assert torch.equal(ens.coords.cpu(), torch.as_tensor(p0)) and torch.equal(ens.lnp, lnp0)
    assert int(ens.accepted.sum()) == 0 and torch.isfinite(ens.lnp).all() and not torch.isnan(ens.coords).any()
    lk.close()


# Seed-to-seed standard deviation (ddof = 1) of ln Z on Sloped with 2^14 particles, run_smc(moves=KDEMove()): 8 seeds of
# tools/smc_bench.py --moves kde, profiles/r07_kde_bench.txt (one NVIDIA B200, 1000 W power limit).
SLOPED_KDE_LNZ_SD_2P14 = 0.0836


@pytest.mark.gpu
def test_run_smc_with_kde_on_sloped_matches_importance_sampling(built, golden):
    """run_smc(moves=KDEMove()) on Sloped with 2^14 particles: the same seed gives the same bits, on a side stream too;
    ln Z agrees with test_smc's importance-sampling estimate within 4 seed standard deviations (SLOPED_KDE_LNZ_SD_2P14),
    and the population's mean and sigma of every parameter with the IS-weighted ones within 4 standard errors."""
    import torch
    from magprop_b200.synthetic.synth_mcmc import run_smc
    g = golden["lnprob_script"]
    x, y, yerr = g["Sloped_x"], g["Sloped_y"], g["Sloped_yerr"]
    n = 1 << 14
    runs = []
    for use_side in (False, False, True):
        st = torch.cuda.Stream() if use_side else torch.cuda.current_stream()
        with torch.cuda.stream(st):
            runs.append(run_smc("Sloped", x, y, yerr, n, seed=3, moves=KDEMove()))
        torch.cuda.synchronize()
    res = runs[0]
    for other in runs[1:]:
        assert torch.equal(other.chain_device, res.chain_device) and torch.equal(other.lnp_device, res.lnp_device)
        assert other.log_evidence == res.log_evidence and np.array_equal(other.betas, res.betas)
    log_z_is, sigma_is, ess, draws, wn = TS._student_t_is(res, x, y, yerr)
    pop = res.get_chain()[0]
    mean_is = wn @ draws
    sd_is = np.sqrt(wn @ (draws - mean_is) ** 2)
    n_eff = n / 4
    mean_err = np.abs(pop.mean(axis=0) - mean_is) / (sd_is * np.sqrt(1 / n_eff + 1 / ess))
    sd_err = np.abs(pop.std(axis=0) / sd_is - 1.0) / np.sqrt(1 / (2 * n_eff) + 1 / (2 * ess))
    print(f"Sloped SMC 2^14 with KDEMove: ln Z {res.log_evidence:.4f}, IS {log_z_is:.4f} +- {sigma_is:.4f} (ESS {ess:.0f}); "
          f"{res.betas.size} stages, {res.n_evaluations} evaluations; mean errors {np.round(mean_err, 2).tolist()}, "
          f"sigma errors {np.round(sd_err, 2).tolist()}")
    assert ess >= 1000
    assert abs(res.log_evidence - log_z_is) <= 4 * math.hypot(SLOPED_KDE_LNZ_SD_2P14, sigma_is)
    assert mean_err.max() < 4 and sd_err.max() < 4
