"""emcee 3's moves on the device ensembles: the NumPy restatement of the DE and snooker moves samples known Gaussians,
the host-compiled draws, partner picks and move choice equal it, the mp_move layout and every argument check of the
two entry points hold without a GPU, and a sharded run equals a single one under gloo (CPU); the kernels equal the
restatement bit for bit across the launch paths, the plain stretch-move entry points equal the sampler's default
ensembles, streams do not matter, and stretch and the mix agree on the Humped posterior (GPU)."""
import ctypes as C
import os

import numpy as np
import pytest

import ensemble_ref as E
from conftest import ROOT
from magprop_b200.sampler import DEMove, DESnookerMove, DeviceEnsemble, StretchMove, TemperedEnsemble, move_table
from magprop_b200.synthetic.synth_mcmc import integrated_time

MIX = [(DEMove(), 0.8), (DESnookerMove(), 0.2)]
KINDS = {"stretch": None, "de": DEMove(), "snooker": DESnookerMove(), "mix": MIX}


# ---- the restatement samples known Gaussians ---------------------------------------------------------------
def gaussian(d):
    """Mean, covariance and log-density of a d-dimensional Gaussian, correlated at 0.99 between every pair, with
    scales spread over three decades."""
    sig = np.logspace(0.0, 3.0, d)
    corr = np.full((d, d), 0.99) + 0.01 * np.eye(d)
    cov = corr * np.outer(sig, sig)
    mu = 3.0 * sig
    prec = np.linalg.inv(cov)

    def lnprob(q):
        r = np.asarray(q) - mu
        return -0.5 * np.einsum("ij,jk,ik->i", r, prec, r)
    return mu, cov, lnprob


def sample_gaussian(d, moves, nsteps=6000, nwalkers=32, seed=1):
    mu, cov, lnprob = gaussian(d)
    rng = np.random.RandomState(seed)
    p0 = mu + 0.1 * rng.multivariate_normal(np.zeros(d), cov, size=nwalkers)
    ens = DeviceEnsemble(E.NumpyBackend(lnprob), nwalkers, d, seed=seed, device="cpu", moves=moves)
    ens.set_state(p0, lnprob(p0))
    chain, _ = ens.run(nsteps, store=True)
    return mu, cov, chain.numpy()[nsteps // 4:], ens


def assert_recovers(mu, cov, chain, nsig=5.0):
    """Mean and covariance within nsig Monte Carlo standard errors, with N/tau effective samples."""
    tau = integrated_time(chain, quiet=True)
    n_eff = chain.shape[0] * chain.shape[1] / tau.max()
    flat = chain.reshape(-1, chain.shape[2])
    sd = np.sqrt(np.diag(cov))
    mean_err = np.abs(flat.mean(axis=0) - mu) / (sd / np.sqrt(n_eff))
    c = np.cov(flat.T)
    cov_err = np.abs(c - cov) / np.sqrt((np.outer(np.diag(cov), np.diag(cov)) + cov ** 2) / n_eff)
    assert mean_err.max() < nsig and cov_err.max() < nsig, (tau, mean_err, cov_err)
    return tau


@pytest.mark.parametrize("d", [2, 6])
@pytest.mark.parametrize("kind", ["de", "snooker", "mix"])
def test_restatement_samples_correlated_gaussians(kind, d):
    mu, cov, chain, ens = sample_gaussian(d, KINDS[kind])
    assert_recovers(mu, cov, chain)
    acc = float(ens.acceptance_fraction().mean())
    assert 0.05 < acc < 0.95, acc


# ---- host-compiled helpers == the restatement --------------------------------------------------------------
@pytest.fixture(scope="module")
def moves_rng(tmp_path_factory):
    """tests/hostsim/moves_rng.cpp -- the moves' helpers of magprop_rng.cuh -- built for the host."""
    import subprocess
    so = str(tmp_path_factory.mktemp("moves_rng") / "moves_rng.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "moves_rng.cpp")], check=True)
    lib = C.CDLL(so)
    vp = C.c_void_p
    lib.mr_move_draws.argtypes = [C.c_ulonglong, C.c_ulonglong, C.c_uint, vp]
    lib.mr_accept_uniform.argtypes = [C.c_int, C.c_ulonglong, C.c_ulonglong, C.c_uint]
    lib.mr_accept_uniform.restype = C.c_double
    lib.mr_de_pair.argtypes = [C.c_double, C.c_double, C.c_uint, vp]
    lib.mr_snooker_triple.argtypes = [C.c_double, C.c_double, C.c_double, C.c_uint, vp]
    lib.mr_choose_move.argtypes = [C.c_ulonglong, C.c_ulonglong, vp, C.c_int]
    return lib


def test_host_compiled_draws_and_partner_picks_match_the_restatement(moves_rng):
    rng = np.random.RandomState(3)
    u4 = np.empty(4)
    jk, zr = np.empty(2, np.uint32), np.empty(3, np.uint32)
    for it in range(3000):
        seed, hs, row = int(rng.randint(0, 1 << 62)), int(rng.randint(0, 1 << 40)), int(rng.randint(0, 1 << 31))
        if it % 3 == 0:
            seed, hs = it, it // 3
        moves_rng.mr_move_draws(seed, hs, row, u4.ctypes.data)
        want = [float(w[0]) for w in E.move_draws(seed, hs, np.array([row]))]
        assert u4.tolist() == want, (seed, hs, row)
        for kind in (E.STRETCH, E.DE, E.SNOOKER):
            ua = moves_rng.mr_accept_uniform(kind, seed, hs, row)
            assert ua == float(E.accept_uniform(kind, seed, hs, np.array([row]))[0]), (kind, seed, hs, row)
            assert (ua == u4[3]) == (kind != E.STRETCH), (kind, seed, hs, row)
        for nc in (2, 3, 4, 7, 1000, 1 << 20):
            moves_rng.mr_de_pair(u4[0], u4[1], nc, jk.ctypes.data)
            j, k = E.de_pair(np.array([u4[0]]), np.array([u4[1]]), nc)
            assert (int(jk[0]), int(jk[1])) == (int(j[0]), int(k[0])) and jk[0] != jk[1] and jk.max() < nc
            if nc >= 3:
                moves_rng.mr_snooker_triple(u4[0], u4[1], u4[2], nc, zr.ctypes.data)
                want = [int(v[0]) for v in E.snooker_triple(np.array([u4[0]]), np.array([u4[1]]), np.array([u4[2]]), nc)]
                assert zr.tolist() == want and len(set(want)) == 3 and max(want) < nc
    # the picks cover their ranges uniformly: every ordered pair of 3, every ordered triple of 4
    u = [rng.rand(60000) for _ in range(3)]
    j, k = E.de_pair(u[0], u[1], 3)
    assert np.abs(np.bincount(j * 3 + k, minlength=9)[[1, 2, 3, 5, 6, 7]] / 10000.0 - 1.0).max() < 0.06
    z, r1, r2 = E.snooker_triple(u[0], u[1], u[2], 4)
    counts = np.bincount(z * 16 + r1 * 4 + r2, minlength=64)
    assert (counts > 0).sum() == 24 and np.abs(counts[counts > 0] / 2500.0 - 1.0).max() < 0.12


def test_host_compiled_move_choice_matches_the_restatement(moves_rng):
    rng = np.random.RandomState(4)
    tables = [[1.0], [0.8, 0.2], [0.0, 1.0], [1.0, 0.0], [0.3, 0.0, 0.5, 0.2], [1e-300, 1.0], [5.0] * 8]
    for w in tables:
        wa = np.array(w)
        picks = []
        for step in list(range(500)) + [int(s) for s in rng.randint(0, 1 << 62, size=100)]:
            got = moves_rng.mr_choose_move(77, step, wa.ctypes.data, len(w))
            assert got == E.choose_move(77, step, w), (w, step)
            assert w[got] > 0.0
            picks.append(got)
        freq = np.bincount(picks[:500], minlength=len(w)) / 500.0
        assert np.abs(freq - wa / wa.sum()).max() < 0.08, (w, freq)


# ---- the C ABI without a GPU --------------------------------------------------------------------------------
def test_move_struct_matches_the_header(built, tmp_path):
    """mp_move as ctypes lays it out == as a C compiler lays out the header's definition."""
    import subprocess
    from magprop_b200 import _capi as A
    fields = [f[0] for f in A.Move._fields_]
    prog = ['#include <stdio.h>', '#include <stddef.h>', '#include "magprop_b200.h"', 'int main(void) {',
            '  printf("%zu %d %d %d %d\\n", sizeof(mp_move), MP_MOVE_STRETCH, MP_MOVE_DE, MP_MOVE_DE_SNOOKER, MP_MAX_MOVES);']
    prog += [f'  printf("%zu\\n", offsetof(mp_move, {f}));' for f in fields]
    prog += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(prog))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert [int(v) for v in out[:5]] == [C.sizeof(A.Move), A.MP_MOVE_STRETCH, A.MP_MOVE_DE, A.MP_MOVE_DE_SNOOKER,
                                         A.MP_MAX_MOVES]
    assert [int(v) for v in out[5:]] == [getattr(A.Move, f).offset for f in fields]
    assert len(A.EXPORTS) == 36 and len(set(A.EXPORTS)) == 36


def test_capi_move_argument_checks_without_device(built):
    """Every argument check of both entry points: MP_ERR_BAD_ARG with the check's own message, before any device work
    (the handle is null: a call that passed every check would fail on that instead)."""
    from magprop_b200 import _capi as A
    lib = A.load()

    def desc(nwalkers=8):
        e = A.Ensemble()
        e.coords, e.lnp, e.nwalkers, e.ndim, e.a, e.seed, e.world = 0x1000, 0x2000, nwalkers, 6, 2.0, 1, 1
        return e

    def mv(kind, weight=1.0, a=2.0, gamma0=0.0, sigma=1e-5, gammas=1.7):
        return (kind, 0, weight, a, gamma0, sigma, gammas)

    def both(table, n=None, nwalkers=8):
        arr = (A.Move * max(1, len(table)))(*table)
        nm = len(table) if n is None else n
        betas = np.array([1.0, 0.5])
        r1 = lib.mp_ensemble_moves_half_step(None, C.byref(desc(nwalkers)), C.addressof(arr), nm, 0, 0, None)
        m1 = lib.mp_last_error().decode()
        r2 = lib.mp_tempered_moves_half_step(None, C.byref(desc(nwalkers)), 2, A.ptr(betas), C.addressof(arr), nm, 0, 0, None)
        m2 = lib.mp_last_error().decode()
        return r1, r2, m1, m2

    S, D, K = A.MP_MOVE_STRETCH, A.MP_MOVE_DE, A.MP_MOVE_DE_SNOOKER
    cases = [
        ([mv(S)], 0, "n_moves"), ([mv(S)] * 9, None, "n_moves"), ([mv(3)], None, "unknown"), ([mv(-1)], None, "unknown"),
        ([mv(S, weight=-1.0)], None, "weights"), ([mv(S, weight=np.nan)], None, "weights"),
        ([mv(S, weight=np.inf)], None, "weights"), ([mv(S, weight=0.0), mv(D, weight=0.0)], None, "sum"),
        ([mv(S, weight=1e308), mv(D, weight=1e308)], None, "sum"),
        ([mv(S, a=1.0)], None, "a > 1"), ([mv(S, a=0.5)], None, "a > 1"), ([mv(S, a=np.nan)], None, "a > 1"),
        ([mv(D, sigma=1.0)], None, "sigma"), ([mv(D, sigma=-0.1)], None, "sigma"), ([mv(D, sigma=np.nan)], None, "sigma"),
        ([mv(D, gamma0=-1.0)], None, "gamma0"), ([mv(D, gamma0=np.nan)], None, "gamma0"),
        ([mv(K, gammas=0.0)], None, "gammas"), ([mv(K, gammas=-1.7)], None, "gammas"),
        ([mv(S), mv(K, gammas=np.inf)], None, "gammas"),
    ]
    for table, n, word in cases:
        r1, r2, m1, m2 = both(table, n)
        assert (r1, r2) == (A.MP_ERR_BAD_ARG,) * 2 and word in m1 and word in m2, (table, m1, m2)
    # too few walkers in a half for the partners of a move that has weight; a zero-weight move does not count
    for table, nwalkers, bad in (([mv(D)], 2, True), ([mv(D)], 4, False), ([mv(K)], 4, True), ([mv(K)], 6, False),
                                 ([mv(S), mv(K, weight=0.0)], 2, False)):
        r1, r2, m1, m2 = both(table, nwalkers=nwalkers)
        assert (r1, r2) == (A.MP_ERR_BAD_ARG,) * 2
        assert ("partners" in m1 and "partners" in m2) == bad, (table, nwalkers, m1)
        if not bad:
            assert "null handle" in m1 and "null handle" in m2
    assert lib.mp_ensemble_moves_half_step(None, C.byref(desc()), None, 1, 0, 0, None) == A.MP_ERR_BAD_ARG
    assert "n_moves" in lib.mp_last_error().decode()
    arr = (A.Move * 1)(mv(D))
    assert lib.mp_ensemble_moves_half_step(None, C.byref(desc()), C.addressof(arr), 1, 0, 2, None) == A.MP_ERR_BAD_ARG
    assert "split" in lib.mp_last_error().decode()
    assert lib.mp_tempered_moves_half_step(None, C.byref(desc()), 2, A.ptr(np.array([1.0, 2.0])), C.addressof(arr), 1, 0, 0,
                                           None) == A.MP_ERR_BAD_ARG
    assert "betas" in lib.mp_last_error().decode()


def test_bad_moves_raise_value_error():
    _, _, lnprob = gaussian(3)
    bad = [[], [StretchMove()] * 9, "de", [DEMove(), "x"], [(DEMove(), -1.0)], [(DEMove(), np.nan)], [(DEMove(), 0.0)],
           [(DEMove(), "heavy")], [(DEMove(), 1.0, 2.0)], StretchMove(1.0), StretchMove(np.inf), DEMove(sigma=1.0),
           DEMove(sigma=-1e-3), DEMove(gamma0=0.0), DEMove(gamma0=-1.0), DESnookerMove(0.0), DESnookerMove(-1.0),
           [(StretchMove(), 1e308), (DEMove(), 1e308)]]
    for moves in bad:
        with pytest.raises(ValueError):
            move_table(moves)
        with pytest.raises(ValueError):
            DeviceEnsemble(E.NumpyBackend(lnprob), 8, 3, device="cpu", moves=moves)
    with pytest.raises(ValueError):
        DeviceEnsemble(E.NumpyBackend(lnprob), 4, 2, device="cpu", moves=DESnookerMove())     # half of 2 < 3
    with pytest.raises(ValueError):
        TemperedEnsemble(E.NumpyBackend(lnprob), 4, 2, [1.0, 0.5], device="cpu", moves=[DEMove(), DESnookerMove()])
    DeviceEnsemble(E.NumpyBackend(lnprob), 4, 2, device="cpu", moves=[DEMove(), (DESnookerMove(), 0.0)])
    table, arr = move_table([DEMove(0.1, 1.5), (DESnookerMove(2.0), 3.0), StretchMove(3.0)])
    assert [w for _, w in table] == [1.0, 3.0, 1.0]
    assert [(m.kind, m.weight, m.a, m.gamma0, m.sigma, m.gammas) for m in arr] == [
        (1, 1.0, 0.0, 1.5, 0.1, 0.0), (2, 3.0, 0.0, 0.0, 0.0, 2.0), (0, 1.0, 3.0, 0.0, 0.0, 0.0)]
    assert move_table(DEMove())[1][0].gamma0 == 0.0                     # None: 2.38 / sqrt(2 ndim) in the library


# ---- sharded == single under gloo -----------------------------------------------------------------------------
def _run_mix(dist, nsteps=25):
    _, _, lnprob = gaussian(3)
    p0 = gaussian(3)[0] + np.random.RandomState(5).randn(32, 3) * [1.0, 30.0, 1000.0]
    ens = DeviceEnsemble(E.NumpyBackend(lnprob), 32, 3, seed=11, device="cpu", dist=dist, moves=MIX)
    ens.set_state(p0, lnprob(p0))
    chain, lps = ens.run(nsteps, store=True)
    return chain.numpy(), lps.numpy(), ens.acceptance_fraction().numpy(), ens.exchange


def _gloo_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    chain, lps, acc, exchange = _run_mix(dist)
    if rank == 0:
        np.savez(out, chain=chain, lps=lps, acc=acc, exchange=exchange)
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_mix_matches_single_rank(tmp_path):
    import torch.multiprocessing as mp
    single = _run_mix(None)
    out = str(tmp_path / "r0.npz")
    port = 31500 + (os.getpid() % 2000)
    mp.spawn(_gloo_worker, args=(2, port, out), nprocs=2, join=True)
    two = np.load(out)
    assert str(two["exchange"]) == "allgather" and single[3] == "none"
    assert np.array_equal(two["chain"], single[0]) and np.array_equal(two["lps"], single[1])
    assert np.array_equal(two["acc"], single[2])
    kinds = {E.choose_move(11, s, [0.8, 0.2]) for s in range(25)}
    assert kinds == {0, 1}                                              # both moves ran
    assert 0.05 < single[2].mean() < 0.95


# ---- on the GPU ---------------------------------------------------------------------------------------------------
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


def _with_n_rhs(ens):
    import torch
    ens.n_rhs = torch.zeros(ens.ntemps * ens.nwalkers, dtype=torch.int32, device=ens.device)
    ens.desc.n_rhs = ens.n_rhs.data_ptr()
    return ens


def _state(ens):
    return [ens.coords.cpu(), ens.lnp.cpu(), ens.accepted.cpu(), ens.status.cpu(), ens.n_rhs.cpu()]


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["ball64", "prior16k", "tempered"])
def test_one_stretch_move_equals_the_default_call(built, golden, case):
    """The plain entry points mp_ensemble_half_step / mp_tempered_half_step (the stretch move of e->a), driven on an
    ensemble's descriptor, == that ensemble run by the sampler (moves=None: [StretchMove(a)] through the moves entry
    points), bit for bit in coords, lnp, accepted, status and n_rhs."""
    import torch
    from magprop_b200 import _capi as A
    from magprop_b200.sampler import geometric_betas
    lib = A.load()
    lk = _humped(golden)
    out = []
    for plain in (False, True):
        if case == "tempered":
            ens = _with_n_rhs(TemperedEnsemble.from_likelihood(lk, 256, 6, geometric_betas(4, 1e-2), seed=3))
            ens.initialise(np.stack([_ball(256, 1), _ball(256, 2, 0.05), _prior_wide(256, 3), _prior_wide(256, 4)]))
            nsteps = 4
        else:
            n, p0 = (64, _ball(64, 1)) if case == "ball64" else (16384, _prior_wide(16384, 2))
            ens = _with_n_rhs(DeviceEnsemble.from_likelihood(lk, n, 6, seed=3))
            ens.initialise(p0)
            nsteps = 4 if n == 64 else 2
        if not plain:
            ens.run(nsteps, store=False)
        else:
            stream = torch.cuda.current_stream().cuda_stream or None
            for step in range(nsteps):
                for split in (0, 1):
                    if case == "tempered":
                        A.check(lib.mp_tempered_half_step(lk._h, C.byref(ens.desc), ens.ntemps, A.ptr(ens.betas), step,
                                                          split, stream))
                    else:
                        A.check(lib.mp_ensemble_half_step(lk._h, C.byref(ens.desc), step, split, stream))
                if case == "tempered":
                    ens.backend.tempered_swap(ens, step)
        torch.cuda.synchronize()
        out.append(_state(ens))
    for a, b in zip(*out):
        assert torch.equal(a, b)
    assert out[0][2].sum() > 0
    lk.close()


def _mismatch(got, want, x0, rows, q, acc, n):
    """Where the device rows differ from the restatement's: enough to tell a proposal from an accept decision."""
    bad = np.flatnonzero((got != want).any(axis=1))
    pos = {int(r): i for i, r in enumerate(rows)}
    lines = [f"{bad.size} rows differ; temperatures {np.bincount(bad // n).tolist()}"]
    for r in bad[:6]:
        i = pos.get(int(r), -1)
        lines.append(f"row {r}: mover {i}, restatement accepted {bool(acc[i]) if i >= 0 else None}, device row is the old row "
                     f"{np.array_equal(got[r], x0[r])}, is the restatement's proposal {np.array_equal(got[r], q[i]) if i >= 0 else None}")
    return "\n".join(lines)


def _check_against_restatement(lk, fn, n, p0, moves, seed, nsteps, ntemps=1, betas=None):
    """Run the device ensemble half-step by half-step and the restatement beside it; every state must be equal.
    Returns the stiff count of every device half-step (read straight after it) and the move kind of every step."""
    import torch
    from magprop_b200.sampler import TemperedEnsemble as TE
    if betas is None:
        ens = DeviceEnsemble.from_likelihood(lk, n, 6, seed=seed, moves=moves)
    else:
        ens = TE.from_likelihood(lk, n, 6, betas, seed=seed, moves=moves)
    ens.initialise(p0)
    torch.cuda.synchronize()
    coords = p0.reshape(-1, 6).copy()
    lnp = ens.lnp.cpu().numpy().copy()
    acc = np.zeros(coords.shape[0], np.int32)
    table = ens.moves
    stiff, kinds = [], []
    half = n // 2
    for step in range(nsteps):
        mv = E.step_move(table, seed, step)
        kinds.append(mv.kind)
        for split in (0, 1):
            x0 = coords.copy()
            if betas is None:
                ens.backend.half_step(ens, step, split)
                stiff.append(lk.last_stiff_count())          # (synchronises: the launch is complete)
                order = E.ensemble_order(n, seed, step)
                rows = order[split * half:(split + 1) * half]
                comp = order[(1 - split) * half:(2 - split) * half][None, :]
                q, a = E.half_step(coords, lnp, rows, np.zeros(half, np.int64), comp, mv, seed, 2 * step + split, fn,
                                    accepted=acc)
            else:
                ens.backend.tempered_half_step(ens, step, split)
                stiff.append(lk.last_stiff_count())
                t, rows, comp = E.tempered_rows(n, ntemps, seed, step, split)
                q, a = E.half_step(coords, lnp, rows, t, comp, mv, seed, 2 * step + split, fn, betas=betas, accepted=acc)
            got = ens.coords.cpu().numpy()
            assert np.array_equal(got, coords), (step, split, _mismatch(got, coords, x0, rows, q, a, n))
            assert np.array_equal(ens.lnp.cpu().numpy(), lnp), (step, split)
        if betas is not None:
            ens.backend.tempered_swap(ens, step)
            E.swap(coords, lnp, betas, n, seed, step)
        ens.step += 1
    torch.cuda.synchronize()
    assert np.array_equal(ens.coords.cpu().numpy(), coords) and np.array_equal(ens.accepted.cpu().numpy(), acc)
    assert 0 < acc.sum() < acc.size * nsteps
    return stiff, kinds


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["stretch", "de", "snooker", "mix"])
def test_moves_match_the_restatement_small(built, golden, kind):
    """64 walkers from the ball (small launches: the ordered warp-per-walker reduce)."""
    lk = _humped(golden)
    _, kinds = _check_against_restatement(lk, lk.lnprob, 64, _ball(64, 7), KINDS[kind], 31, 8)
    if kind == "mix":
        assert set(kinds) == {1, 2}
    lk.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["stretch", "de", "snooker", "mix"])
def test_moves_match_the_restatement_ordered(built, golden, kind):
    """16 384 walkers from a prior-wide start: 8192 movers per half-step, so the work list is ordered and the proposals
    are formed in order_key_kernel; the spread walkers feed the stiff queue."""
    lk = _humped(golden)
    stiff, kinds = _check_against_restatement(lk, lk.lnprob, 16384, _prior_wide(16384, 8), KINDS[kind], 5,
                                              3 if kind == "mix" else 1)
    assert min(stiff) > 0, stiff
    lk.close()


@pytest.mark.gpu
def test_moves_match_the_restatement_across_slabs(built):
    """On the dataset with data on all 10 001 nodes, 45 056 walkers move 22 528 per half-step: two slabs.  Every move
    kind equals the restatement driven by single-slab host batches."""
    import test_launch_paths as LP
    x = LP.x_wide()
    y, yerr = LP.data_for(x, 5, noise=0.05, err=0.1)
    lk = LP.script_handle(x, y, yerr)
    n = 45056
    assert n // 2 > LP.slab_bound(10001)
    rng = np.random.RandomState(404)
    p0 = np.concatenate([LP.ball(rng, n // 2, 3e-2), LP.ball(rng, n // 2, 0.3)])[rng.permutation(n)]
    fn = lambda q: LP.host_batched(lk, q)[0]
    # steps 0 and 1 of seed 4 run DE then snooker under the mix
    assert [E.choose_move(4, s, [0.8, 0.2]) for s in (0, 1)] == [0, 1]
    _, kinds = _check_against_restatement(lk, fn, n, p0, MIX, 4, 2)
    assert kinds == [1, 2]
    lk.close()


@pytest.mark.gpu
def test_tempered_moves_match_the_restatement(built, golden):
    """T = 4 x n = 2048: 4096 movers per half-step over four temperatures, hot ones spread over the prior."""
    from magprop_b200.sampler import geometric_betas
    lk = _humped(golden)
    betas = geometric_betas(4, 1e-3)
    p0 = np.stack([_ball(2048, 1), _ball(2048, 2, 0.05), _prior_wide(2048, 3), _prior_wide(2048, 4)])
    stiff, kinds = _check_against_restatement(lk, lk.lnprob, 2048, p0, MIX, 4, 3, ntemps=4, betas=betas)
    assert set(kinds) == {1, 2} and max(stiff) > 0
    lk.close()


@pytest.mark.gpu
def test_moves_are_identical_on_a_side_stream(built, golden):
    import torch
    from magprop_b200.sampler import geometric_betas
    lk = _humped(golden)
    out = []
    for use_side in (False, True):
        st = torch.cuda.Stream() if use_side else torch.cuda.current_stream()
        with torch.cuda.stream(st):
            e = DeviceEnsemble.from_likelihood(lk, 128, 6, seed=8, moves=MIX)
            e.initialise(_ball(128, 9))
            c, l = e.run(6, store=True)
            t = TemperedEnsemble.from_likelihood(lk, 64, 6, geometric_betas(3, 1e-2), seed=8, moves=MIX)
            t.initialise(_ball(64, 10))
            tc, tl = t.run(6)
            out.append((c, l, e.accepted.clone(), e.status.clone(), tc, tl, t.accepted.clone()))
        torch.cuda.synchronize()
    for a, b in zip(*out):
        assert torch.equal(a, b)
    lk.close()


@pytest.mark.gpu
def test_stretch_and_mix_agree_on_the_humped_posterior(built, golden):
    """Each run until run_until_converged stops; the medians agree within 4 combined Monte Carlo standard errors,
    sigma * sqrt(tau / N), over the second half of each chain."""
    lk = _humped(golden)
    res = {}
    for name, moves in (("stretch", None), ("mix", MIX)):
        ens = DeviceEnsemble.from_likelihood(lk, 128, 6, seed=21, moves=moves)
        ens.initialise(_ball(128, 22, 1e-4))
        chain, _, hist, converged = ens.run_until_converged(100000, check_every=1000, tau_rtol=0.05)
        assert converged, (name, hist[-1])
        c = chain[chain.shape[0] // 2:].cpu().numpy()
        tau = integrated_time(c, quiet=True)
        flat = c.reshape(-1, 6)
        res[name] = (np.median(flat, axis=0), flat.std(axis=0) * np.sqrt(tau / flat.shape[0]), tau, chain.shape[0])
        print(name, "steps", chain.shape[0], "tau", np.round(tau, 1), "acceptance", float(ens.acceptance_fraction().mean()))
    (m1, e1, _, _), (m2, e2, _, _) = res["stretch"], res["mix"]
    z = np.abs(m1 - m2) / np.hypot(e1, e2)
    assert z.max() < 4.0, z
    lk.close()


@pytest.mark.gpu
def test_nccl_sharded_mix_matches_single_gpu(built):
    """Two ranks over NCCL run the 0.8 DE / 0.2 snooker mix with peer reads and with the all-gather, and reproduce the
    single-GPU chain bit for bit.  Needs two visible GPUs."""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29543", os.path.join(ROOT, "tools", "check_dist_mcmc.py")],
                       capture_output=True, text=True, timeout=300, env=dict(os.environ, MOVES="mix"))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stdout.count("sharded == single: True") == 2
