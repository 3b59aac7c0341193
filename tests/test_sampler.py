"""Ensemble drivers: RNG known answers, host sampler sanity, the multi-rank
driver under gloo (world_size 2, CPU), and the fused device half-step (GPU)."""
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, relerr
import ensemble_ref as E
from magprop_b200.sampler import DeviceEnsemble, EnsembleSampler, StretchMove, rank_slice


def test_philox_known_answers():
    # Random123 kat_vectors, philox4x32 10 rounds
    f = lambda c, k: tuple(int(v) for v in E.philox4x32_10(*[np.uint64(x) for x in c], *k))
    assert f((0, 0, 0, 0), (0, 0)) == (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)
    assert f((0xffffffff,) * 4, (0xffffffff,) * 2) == (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)
    assert f((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0)) == \
        (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)
    rows = np.arange(20000)
    u = np.concatenate(E.stretch_draws(7, 3, rows) + (E.accept_uniform(E.STRETCH, 7, 3, rows),))
    assert 0.0 < u.min() and u.max() < 1.0 and abs(u.mean() - 0.5) < 0.01


def gauss_lnprob(q):
    return -0.5 * np.sum((np.asarray(q) / np.array([1.0, 2.0, 0.5])) ** 2, axis=1)


def test_host_sampler_recovers_gaussian():
    s = EnsembleSampler(40, 3, gauss_lnprob, vectorize=True, seed=1)
    p0 = 0.1 * np.random.RandomState(0).randn(40, 3)
    s.run_mcmc(p0, 1500)
    flat = s.get_chain()[500:].reshape(-1, 3)
    assert np.allclose(flat.std(axis=0), [1.0, 2.0, 0.5], rtol=0.15)
    assert 0.3 < s.acceptance_fraction.mean() < 0.9
    assert s.get_log_prob().shape == (1500, 40)
    with pytest.raises(ValueError):
        EnsembleSampler(5, 3, gauss_lnprob)
    bad = EnsembleSampler(8, 3, lambda q: np.full(len(q), np.nan), seed=0)
    with pytest.raises(ValueError):
        bad.run_mcmc(np.zeros((8, 3)), 1)


def test_rank_slice():
    assert rank_slice(8, 0, 2) == (0, 4) and rank_slice(8, 1, 2) == (4, 8)
    with pytest.raises(ValueError):
        rank_slice(7, 0, 2)


def test_ensemble_order_is_a_keyed_permutation(hostsim):
    """The per-step random halves: the kernels' permutation (compiled for the host) == the NumPy restatement,
    a bijection for every size, different from step to step, and an unbiased split."""
    import ctypes as C
    for n in (12, 50, 256, 4096, 100000):
        got = np.empty(n, dtype=np.int32)
        for step in (0, 1, 12345):
            hostsim.hs_ensemble_order(n, C.c_ulonglong(17), C.c_ulonglong(step), 1, got.ctypes.data_as(C.c_void_p))
            want = E.ensemble_order(n, 17, step)
            assert (got == want).all()
            assert np.array_equal(np.sort(got), np.arange(n))
        hostsim.hs_ensemble_order(n, C.c_ulonglong(17), C.c_ulonglong(5), 0, got.ctypes.data_as(C.c_void_p))
        assert np.array_equal(got, np.arange(n))                       # randomize_split = 0: fixed halves
    # the inverse (which rank moved a walker last, for the peer-read exchange): P^-1(P(g)) == g for every position
    for n in (12, 50, 4096, 100000, 2097152):
        assert hostsim.hs_ensemble_order_roundtrip(n, C.c_ulonglong(17), C.c_ulonglong(3)) == 0
    # over many steps every walker lands in half 0 about half of the time, and pairs decorrelate
    n = 64
    in0 = np.array([E.ensemble_order(n, 3, s)[: n // 2] for s in range(400)])
    freq = np.array([(in0 == w).any(axis=1).mean() for w in range(n)])
    assert np.abs(freq - 0.5).max() < 0.1
    both = np.mean([(0 in r) and (1 in r) for r in in0])
    assert abs(both - 0.25) < 0.08


def _run_ensemble(dist, nsteps=25, randomize=True):
    rng = np.random.RandomState(5)
    p0 = rng.randn(32, 3)
    ens = DeviceEnsemble(E.NumpyBackend(gauss_lnprob), 32, 3, a=2.0, seed=11, device="cpu", dist=dist,
                         randomize_split=randomize)
    ens.set_state(p0, gauss_lnprob(p0))
    chain, lps = ens.run(nsteps, store=True)
    return chain.numpy(), lps.numpy(), ens.acceptance_fraction().numpy(), ens.exchange


def _gloo_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    chain, lps, acc, exchange = _run_ensemble(dist)
    fixed = _run_ensemble(dist, randomize=False)
    if rank == 0:
        np.savez(out, chain=chain, lps=lps, acc=acc, exchange=exchange, fixed_chain=fixed[0])
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_ensemble_matches_single_rank(tmp_path):
    """world_size-2 gloo run == single-process run, bit for bit (counter-based RNG and keyed split, each half
    shared out over the ranks, ONE packed all-gather of the moved rows per half-step)."""
    import torch.multiprocessing as mp
    single = _run_ensemble(None)
    single_fixed = _run_ensemble(None, randomize=False)
    out = str(tmp_path / "r0.npz")
    port = 29500 + (os.getpid() % 2000)
    mp.spawn(_gloo_worker, args=(2, port, out), nprocs=2, join=True)
    two = np.load(out)
    assert str(two["exchange"]) == "allgather" and single[3] == "none"
    assert (two["chain"] == single[0]).all() and (two["lps"] == single[1]).all()
    assert (two["acc"] == single[2]).all()
    assert (two["fixed_chain"] == single_fixed[0]).all()
    assert not (single_fixed[0] == single[0]).all()          # the random split does change the chain
    assert 0.2 < single[2].mean() < 0.95


def test_device_ensemble_and_host_sampler_agree_statistically():
    """emcee's move semantics on both drivers: the device-ensemble logic (random keyed halves, NumPy double of
    the kernel) and the host EnsembleSampler (emcee's shuffle) sample the same 3-D Gaussian -- moments and
    acceptance agree; fixed halves do too (a valid move, just not emcee's default)."""
    sig = np.array([1.0, 2.0, 0.5])
    p0 = 0.1 * np.random.RandomState(0).randn(40, 3)
    host = EnsembleSampler(40, 3, gauss_lnprob, vectorize=True, seed=1)
    host.run_mcmc(p0, 2000)
    hflat = host.get_chain()[500:].reshape(-1, 3)
    res = {}
    for randomize in (True, False):
        ens = DeviceEnsemble(E.NumpyBackend(gauss_lnprob), 40, 3, a=2.0, seed=2, device="cpu", randomize_split=randomize)
        ens.set_state(p0, gauss_lnprob(p0))
        chain, _ = ens.run(2000, store=True)
        flat = chain.numpy()[500:].reshape(-1, 3)
        res[randomize] = (flat, float(ens.acceptance_fraction().mean()))
        assert np.allclose(flat.std(axis=0), sig, rtol=0.12), flat.std(axis=0)
        assert np.abs(flat.mean(axis=0)).max() < 0.25
        assert np.allclose(flat.std(axis=0), hflat.std(axis=0), rtol=0.15)
        assert abs(res[randomize][1] - host.acceptance_fraction.mean()) < 0.05
    # kurtosis of a Gaussian: the chains are not just matching a variance
    k = ((res[True][0] / res[True][0].std(axis=0)) ** 4).mean(axis=0)
    assert np.allclose(k, 3.0, atol=0.5)


@pytest.mark.gpu
def test_device_half_step_matches_numpy_double(built, golden):
    import torch
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, time_grid
    from oracle import magprop_oracle as O
    g = golden["lnprob_script"]
    lk = Likelihood(A.script_model_spec(), time_grid(None), g["Humped_x"], g["Humped_y"], g["Humped_yerr"],
                    O.SCRIPT_LOWER, O.SCRIPT_UPPER)
    rng = np.random.RandomState(3)
    n = 64
    p0 = O.SYNTH_TRUTHS_LOG["Humped"] + 1e-2 * rng.randn(n, 6)
    ens = DeviceEnsemble.from_likelihood(lk, n, 6, a=2.0, seed=99)
    ens.initialise(p0)
    torch.cuda.synchronize()
    lnp0 = ens.lnp.cpu().numpy()
    assert relerr(lnp0, lk.lnprob(p0)).max() == 0.0
    # numpy double driven by the SAME device likelihood, same keyed random halves
    coords, lnp, acc = p0.copy(), lnp0.copy(), np.zeros(n, np.int32)
    half = n // 2
    nsteps = 6
    chain, lps = ens.run(nsteps, store=True)
    torch.cuda.synchronize()
    order_d = torch.empty(n, dtype=torch.int32, device="cuda")
    for it in range(nsteps):
        order = E.ensemble_order(n, 99, it)
        A.check(A.load().mp_ensemble_order(n, 99, it, 1, order_d.data_ptr(), None))
        assert (order_d.cpu().numpy() == order).all()
        for split in (0, 1):
            active = order[split * half:(split + 1) * half]
            comp = order[(1 - split) * half:(2 - split) * half]
            E.half_step(coords, lnp, active, np.zeros(half, np.int64), comp[None, :], StretchMove(2.0), 99, 2 * it + split,
                        lk.lnprob, accepted=acc)
        assert (chain[it].cpu().numpy() == coords).all()
        assert (lps[it].cpu().numpy() == lnp).all()
    assert (ens.accepted.cpu().numpy() == acc).all()
    assert 0 < acc.sum() < n * nsteps
    assert np.isfinite(lnp).all()
    # fixed halves (randomize_split=False) == the explicit-list entry point mp_stretch_half_step
    fixed = DeviceEnsemble.from_likelihood(lk, n, 6, a=2.0, seed=99, randomize_split=False)
    fixed.initialise(p0)
    fixed.run(3)
    c2 = torch.from_numpy(p0).cuda(); l2 = torch.from_numpy(lnp0).cuda()
    idx = torch.arange(n, dtype=torch.int32, device="cuda")
    for it in range(3):
        for split in (0, 1):
            act = idx[:half] if split == 0 else idx[half:]
            cmp_ = idx[half:] if split == 0 else idx[:half]
            lk.stretch_half_step(c2.data_ptr(), l2.data_ptr(), n, 6, act.data_ptr(), half, cmp_.data_ptr(), half, 2.0, 99,
                                 2 * it + split)
    torch.cuda.synchronize()
    assert torch.equal(fixed.coords, c2) and torch.equal(fixed.lnp, l2)
    lk.close()


@pytest.mark.gpu
def test_device_ensemble_logs_bad_proposals_and_status(built, golden):
    """The {GRB}_bad.csv side channel on the device path (mcmc_eqns.py:72-79): proposals whose likelihood is not
    finite are logged with their parameters, and the per-walker status word says why."""
    import torch
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, time_grid
    from oracle import magprop_oracle as O
    g = golden["lnprob_script"]
    # a step budget of 20 makes every integration fail: each in-prior proposal is a bad row
    lk = Likelihood(A.script_model_spec(max_steps=20), time_grid(None), g["Humped_x"], g["Humped_y"], g["Humped_yerr"],
                    O.SCRIPT_LOWER, O.SCRIPT_UPPER)
    n = 32
    p0 = O.SYNTH_TRUTHS_LOG["Humped"] + 1e-3 * np.random.RandomState(1).randn(n, 6)
    ens = DeviceEnsemble.from_likelihood(lk, n, 6, seed=4)
    ens.set_state(p0, np.zeros(n))
    ens.run(2)
    torch.cuda.synchronize()
    rows, dropped = ens.drain_bad()
    st = ens.status.cpu().numpy()
    assert dropped == 0 and rows.shape == (2 * n, 6)
    assert ((st & A.WALKER_INTEGRATOR_FAIL) != 0).all()
    assert (ens.accepted.cpu().numpy() == 0).all() and np.array_equal(ens.coords.cpu().numpy(), p0)
    assert np.abs(rows - O.SYNTH_TRUTHS_LOG["Humped"]).max() < 0.1          # they are proposals around the ball
    assert ens.drain_bad()[0].shape == (0, 6)
    lk.close()


@pytest.mark.gpu
def test_run_concurrently_matches_sequential_runs(built, golden):
    """Three datasets' ensembles advanced side by side (one stream each) give the chains of three separate runs."""
    import torch
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, time_grid
    from magprop_b200.sampler import run_concurrently
    from oracle import magprop_oracle as O
    g = golden["lnprob_script"]
    names = ("Classic", "Sloped", "Stuttering")

    def make():
        liks, ens = [], []
        for k, n in enumerate(names):
            lk = Likelihood(A.script_model_spec(), time_grid(None), g[f"{n}_x"], g[f"{n}_y"], g[f"{n}_yerr"],
                            O.SCRIPT_LOWER, O.SCRIPT_UPPER)
            e = DeviceEnsemble.from_likelihood(lk, 64, 6, a=2.0, seed=5 + k)
            e.initialise(O.SYNTH_TRUTHS_LOG[n] + 1e-3 * np.random.RandomState(k).randn(64, 6))
            liks.append(lk); ens.append(e)
        return liks, ens

    liks, ens = make()
    seq = [e.run(8, store=True) for e in ens]
    torch.cuda.synchronize()
    for lk in liks:
        lk.close()
    liks, ens = make()
    par = run_concurrently(ens, 8, store=True)
    torch.cuda.synchronize()
    for (c0, l0), (c1, l1), e in zip(seq, par, ens):
        assert torch.equal(c0, c1) and torch.equal(l0, l1) and e.step == 8
    for lk in liks:
        lk.close()


@pytest.mark.gpu
def test_nccl_sharded_ensemble_matches_single_gpu(built):
    """Two ranks over NCCL, each moving half of every half-ensemble and all-gathering the updates, reproduce the
    single-GPU chain bit for bit (counter-based RNG, no cross-rank state).  Needs two visible GPUs."""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29541", os.path.join(root, "tools", "check_dist_mcmc.py")],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stdout.count("sharded == single: True") == 2
