"""Integrated autocorrelation time on the device (mp_chain_autocorr, integrated_time_device) and the
convergence-stopped ensemble run (DeviceEnsemble.run_until_converged).

CPU: argument checks of the C entry point, the lag-doubling window logic against ``integrated_time`` (bit for bit),
and ``run_until_converged`` on the NumPy double of the kernel, single-rank and under gloo.
GPU: ACF and tau parity against the NumPy path, determinism, a chain of more than 2^31 doubles, and the real sampler."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import has_gpu, relerr
import stretch_ref as R
from magprop_b200.sampler import DeviceEnsemble
from magprop_b200.synthetic import synth_mcmc as S


def ar1(rng, n, nw, nd, phi=0.8):
    e = rng.randn(n, nw, nd)
    x = np.empty_like(e)
    x[0] = e[0] / np.sqrt(1 - phi * phi)
    for i in range(1, n):
        x[i] = phi * x[i - 1] + e[i]
    return x + rng.randn(1, nw, nd) * 3.0          # walker offsets: the mean subtraction matters


def random_walk(rng, n, nw, nd):
    return np.cumsum(rng.randn(n, nw, nd), axis=0) + 100.0


def host_acf(x):
    """Mean over walkers of emcee's function_1d, [ndim, n] (integrated_time's own accumulation)."""
    n_t, n_w, n_d = x.shape
    f = np.zeros((n_d, n_t))
    with np.errstate(invalid="ignore"):
        for d in range(n_d):
            for k in range(n_w):
                f[d] += S.function_1d(x[:, k, d])
            f[d] /= n_w
    return f


def gauss_lnprob(q):
    return -0.5 * np.sum((np.asarray(q) / np.array([1.0, 2.0, 0.5])) ** 2, axis=1)


# ---- CPU ----------------------------------------------------------------------------------------------------
def test_chain_autocorr_argument_checks(built):
    from magprop_b200 import _capi as A
    lib = A.load()
    out = np.empty(64)
    fake = C.c_void_p(4096)          # never dereferenced: the checks come before the device is touched
    good = dict(d_chain=fake, n_steps=20, nwalkers=4, ndim=2, first=0, thin=1, lag_begin=0, lag_end=5, acf=A.ptr(out),
                device=0, stream=None)

    def call(**kw):
        a = dict(good, **kw)
        return lib.mp_chain_autocorr(a["d_chain"], a["n_steps"], a["nwalkers"], a["ndim"], a["first"], a["thin"],
                                     a["lag_begin"], a["lag_end"], a["acf"], a["device"], a["stream"])

    bad = [dict(d_chain=None), dict(acf=None), dict(nwalkers=0), dict(ndim=0), dict(ndim=A.MP_MAX_NDIM + 1),
           dict(thin=0), dict(first=-1), dict(first=20), dict(lag_begin=-1), dict(lag_end=0), dict(lag_begin=3, lag_end=3),
           dict(lag_end=21),                               # more lags than rows
           dict(first=10, thin=3, lag_end=5)]              # rows 10, 13, 16, 19: n = 4 < 5
    for kw in bad:
        assert call(**kw) == A.MP_ERR_BAD_ARG, kw
    with pytest.raises(ValueError):
        A.check(call(thin=0))
    if not has_gpu():                                      # valid arguments, no device
        assert call() == A.MP_ERR_CUDA and call(first=10, thin=3, lag_end=4) == A.MP_ERR_CUDA


class _Provider:
    """ACF blocks from NumPy, recording which lag ranges were asked for."""

    def __init__(self, x):
        self.f, self.calls = host_acf(x), []

    def __call__(self, lo, hi):
        self.calls.append((lo, hi))
        return self.f[:, lo:hi]


def _same_outcome(x, **kw):
    """integrated_time and the lag-doubling driver on the same ACF: the same tau bit for bit, or the same error."""
    p = _Provider(x)
    n_t, _, n_d = x.shape
    c, tol, quiet = kw.get("c", 5), kw.get("tol", 50), kw.get("quiet", False)
    try:
        want = S.integrated_time(x, **kw)
    except S.AutocorrError as e:
        with pytest.raises(S.AutocorrError) as got:
            S._tau_from_acf(p, n_t, n_d, c, tol, quiet)
        assert np.array_equal(got.value.tau, e.tau, equal_nan=True) and str(got.value) == str(e)
        return None, p.calls
    got = S._tau_from_acf(p, n_t, n_d, c, tol, quiet)
    assert np.array_equal(got, want, equal_nan=True), (got, want)
    return got, p.calls


def test_window_driver_matches_integrated_time_bit_for_bit():
    rng = np.random.RandomState(0)
    # AR(1): the window (~5 tau ~ 45) lies in the first block
    tau, calls = _same_outcome(ar1(rng, 5000, 8, 3))
    assert calls == [(0, 128)] and np.all(np.abs(tau / 9.0 - 1) < 0.25)
    # strongly correlated AR(1): the window needs more blocks, each block asked for once
    tau, calls = _same_outcome(ar1(rng, 6000, 4, 2, phi=0.98), quiet=True)
    assert calls[0] == (0, 128) and len(calls) >= 2
    assert all(a[1] == b[0] for a, b in zip(calls, calls[1:])) and calls[-1][1] < 6000
    # a random walk too short for its correlation: the window only lies in the last block, every lag is computed.
    # (The sample ACF of a centred series sums to tau(n-1) = 0 up to rounding, so some M < n always passes.)
    tau, calls = _same_outcome(random_walk(rng, 300, 6, 2), quiet=True, c=50)
    assert calls == [(0, 128), (128, 256), (256, 300)]
    # length check: raises on the short chain (same message and tau), passes on the long one
    _same_outcome(ar1(rng, 200, 6, 2))
    with pytest.raises(S.AutocorrError):
        S.integrated_time(ar1(rng, 200, 6, 2))
    assert _same_outcome(ar1(rng, 3000, 6, 2))[0] is not None
    # a constant walker and n = 1: NaN on both sides
    x = ar1(rng, 400, 4, 2)
    x[:, 1, 0] = 1.0
    tau, _ = _same_outcome(x, quiet=True)
    assert np.isnan(tau[0]) and np.isfinite(tau[1])
    tau, calls = _same_outcome(ar1(rng, 1, 4, 2))
    assert np.isnan(tau).all() and calls == [(0, 1)]
    for n in (2, 3, 37, 129, 257):
        _same_outcome(random_walk(rng, n, 4, 3), quiet=True)
        _same_outcome(ar1(rng, n, 4, 3), quiet=True, c=3)


def _converging(dist=None, max_steps=3000):
    rng = np.random.RandomState(5)
    p0 = rng.randn(32, 3)
    ens = DeviceEnsemble(R.NumpyBackend(gauss_lnprob), 32, 3, a=2.0, seed=11, device="cpu", dist=dist)
    ens.set_state(p0, gauss_lnprob(p0))
    chain, lps, hist, conv = ens.run_until_converged(max_steps, check_every=50, n_tau=10, tau_rtol=0.1)
    return chain.numpy(), lps.numpy(), hist, conv, ens.step


def _fresh_run(nsteps):
    rng = np.random.RandomState(5)
    p0 = rng.randn(32, 3)
    ens = DeviceEnsemble(R.NumpyBackend(gauss_lnprob), 32, 3, a=2.0, seed=11, device="cpu")
    ens.set_state(p0, gauss_lnprob(p0))
    chain, lps = ens.run(nsteps, store=True)
    return chain.numpy(), lps.numpy()


def test_run_until_converged_numpy_backend():
    chain, lps, hist, conv, step = _converging()
    n = chain.shape[0]
    assert conv and n == step and n % 50 == 0 and n < 3000
    assert hist.shape == (n // 50, 3) and lps.shape == (n, 32)

    def passes(k):                        # the criterion at check k (step 50*(k+1)), from the returned history
        prev = hist[k - 1] if k else np.full(3, np.inf)
        return bool(np.all(50 * (k + 1) > 10 * hist[k]) and np.all(np.abs(prev - hist[k]) / hist[k] < 0.1))

    assert passes(len(hist) - 1) and not any(passes(k) for k in range(len(hist) - 1))
    for k in range(len(hist)):            # the history is tau of the chain so far
        assert np.array_equal(hist[k], S.integrated_time(chain[:50 * (k + 1)], quiet=True))
    fresh_chain, fresh_lps = _fresh_run(n)
    assert np.array_equal(chain, fresh_chain) and np.array_equal(lps, fresh_lps)
    # max_steps reached first: not converged, stopped there; a trailing partial block gets no check
    short = _converging(max_steps=n - 50)
    assert not short[3] and short[0].shape[0] == n - 50 and len(short[2]) == (n - 50) // 50
    odd = _converging(max_steps=120)
    assert not odd[3] and odd[0].shape[0] == 120 and len(odd[2]) == 2
    assert np.array_equal(odd[0], fresh_chain[:120])


def _gloo_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    chain, lps, hist, conv, step = _converging(dist)
    np.savez(f"{out}.{rank}.npz", chain=chain, lps=lps, hist=hist, conv=conv, step=step)
    dist.barrier()
    dist.destroy_process_group()


def test_run_until_converged_two_ranks_match_single_rank(tmp_path):
    import torch.multiprocessing as mp
    single = _converging()
    out = str(tmp_path / "conv")
    port = 29500 + ((os.getpid() + 1000) % 2000)
    mp.spawn(_gloo_worker, args=(2, port, out), nprocs=2, join=True)
    for r in range(2):
        got = np.load(f"{out}.{r}.npz")
        assert int(got["step"]) == single[4] and bool(got["conv"]) == single[3]
        assert np.array_equal(got["chain"], single[0]) and np.array_equal(got["lps"], single[1])
        assert np.array_equal(got["hist"], single[2])


# ---- GPU ----------------------------------------------------------------------------------------------------
def _dev(x):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _acf(t, **kw):
    from magprop_b200.engine import chain_autocorr
    n_steps, nw, nd = t.shape
    return chain_autocorr(t.data_ptr(), n_steps, nw, nd, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("n_steps", [1, 2, 3, 37, 512, 4099])
def test_chain_autocorr_matches_numpy(built, n_steps):
    rng = np.random.RandomState(n_steps)
    worst = 0.0
    for nw in (2, 64, 1000):
        for nd in (1, 6, 9):
            for make in (ar1, random_walk):
                x = make(rng, n_steps, nw, nd)
                d = _dev(x)
                for first, thin in ((0, 1), (3, 2), (10, 7)):
                    if first >= n_steps:
                        continue
                    xs = x[first::thin]
                    n = xs.shape[0]
                    f = host_acf(xs)
                    ranges = [(0, n)] if n <= 600 else [(0, 300), (128, 256), (n - 150, n)]
                    if n > 3:
                        ranges.append((1, min(n, 3)))
                    for lo, hi in ranges:
                        got = _acf(d, first=first, thin=thin, lag_begin=lo, lag_end=hi)
                        want = f[:, lo:hi]
                        assert got.shape == want.shape
                        assert np.array_equal(np.isnan(got), np.isnan(want)), (nw, nd, first, thin, lo, hi)
                        ok = ~np.isnan(want)
                        if ok.any():
                            worst = max(worst, float(np.abs(got[ok] - want[ok]).max()))
                        assert worst <= 1e-12, (nw, nd, first, thin, lo, hi, worst)
    if n_steps == 1:
        assert np.isnan(_acf(_dev(np.zeros((1, 4, 2))))).all()


@pytest.mark.gpu
def test_integrated_time_device_matches_host(built):
    rng = np.random.RandomState(7)
    raised = 0
    for n_steps in (1, 2, 37, 300, 2000, 4099):
        for nw, nd in ((2, 1), (64, 6), (200, 9)):
            for make in (ar1, random_walk):
                x = make(rng, n_steps, nw, nd)
                d = _dev(x)
                for discard, thin in ((0, 1), (5, 1), (10, 3)):
                    first = discard + thin - 1
                    if first >= n_steps:
                        continue
                    xs = x[first::thin]
                    try:
                        want = thin * S.integrated_time(xs)
                    except S.AutocorrError as e:
                        raised += 1
                        with pytest.raises(S.AutocorrError) as got:
                            S.integrated_time_device(d, discard=discard, thin=thin)
                        assert relerr(got.value.tau, e.tau).max() <= 1e-10 or np.isnan(e.tau).any()
                        want = thin * S.integrated_time(xs, quiet=True)
                    got = S.integrated_time_device(d, discard=discard, thin=thin, quiet=True)
                    assert np.array_equal(np.isnan(got), np.isnan(want))
                    ok = ~np.isnan(want)
                    assert (relerr(got[ok], want[ok]) <= 1e-10).all(), (n_steps, nw, nd, discard, thin, got, want)
    assert raised > 0
    # n = 1, and a walker held at exactly 1.0: NaN on both sides
    x = ar1(rng, 1, 8, 3)
    assert np.isnan(S.integrated_time_device(_dev(x))).all() and np.isnan(S.integrated_time(x)).all()
    x = ar1(rng, 500, 8, 3)
    x[:, 2, 1] = 1.0
    got, want = S.integrated_time_device(_dev(x), quiet=True), S.integrated_time(x, quiet=True)
    assert np.isnan(got[1]) and np.isnan(want[1])
    assert relerr(got[[0, 2]], want[[0, 2]]).max() <= 1e-10
    with pytest.raises(ValueError):
        S.integrated_time_device(_dev(x), discard=500)
    with pytest.raises(ValueError):
        S.integrated_time_device(x)


@pytest.mark.gpu
def test_chain_autocorr_is_deterministic(built):
    import torch
    rng = np.random.RandomState(3)
    for shape in ((500, 64, 6), (1000, 4096, 5)):
        d = _dev(ar1(rng, *shape))
        a = _acf(d, lag_end=256)
        b = _acf(d, lag_end=256)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            c = _acf(d, lag_end=256, stream=side.cuda_stream)
        assert a.tobytes() == b.tobytes() == c.tobytes()


@pytest.mark.gpu
def test_chain_autocorr_beyond_32bit_indexing(built):
    """2^18 walkers x 2048 steps x 5 = 2.7e9 doubles (21.5 GB): 8 seeded base series tiled across the walkers."""
    import torch
    rng = np.random.RandomState(11)
    base = ar1(rng, 2048, 8, 5, phi=0.9)                    # [step, base, dim]
    chain = _dev(base).repeat(1, 1 << 15, 1)                 # walker w holds base series w % 8
    assert chain.numel() > 2 ** 31 and chain.shape == (2048, 1 << 18, 5)
    want = host_acf(base)
    for lo, hi in ((0, 200), (1900, 2048)):
        got = _acf(chain, lag_begin=lo, lag_end=hi)
        assert np.abs(got - want[:, lo:hi]).max() <= 1e-12
    got = _acf(chain, first=1000, thin=3, lag_end=100)
    assert np.abs(got - host_acf(base[1000::3])[:, :100]).max() <= 1e-12
    del chain
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_autocorr_and_converged_run_on_the_real_sampler(built, golden):
    import torch
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, time_grid
    from oracle import magprop_oracle as O
    g = golden["lnprob_script"]
    lk = Likelihood(A.script_model_spec(), time_grid(None), g["Humped_x"], g["Humped_y"], g["Humped_yerr"],
                    O.SCRIPT_LOWER, O.SCRIPT_UPPER)
    p0 = O.SYNTH_TRUTHS_LOG["Humped"] + 1e-3 * np.random.RandomState(2).randn(64, 6)

    def fresh():
        e = DeviceEnsemble.from_likelihood(lk, 64, 6, seed=5)
        e.initialise(p0)
        return e

    chain, _ = fresh().run(300, store=True)
    torch.cuda.synchronize()
    host = chain.cpu().numpy()
    got, want = S.integrated_time_device(chain, quiet=True), S.integrated_time(host, quiet=True)
    assert relerr(got, want).max() <= 1e-10
    got = S.integrated_time_device(chain, quiet=True, discard=100, thin=2)
    assert relerr(got, 2 * S.integrated_time(host[101::2], quiet=True)).max() <= 1e-10

    c2, l2, hist, conv = fresh().run_until_converged(max_steps=400, check_every=50)
    n = c2.shape[0]
    assert n % 50 == 0 and hist.shape == (n // 50, 6) and (conv or n == 400)
    c3, l3 = fresh().run(n, store=True)
    assert torch.equal(c2, c3) and torch.equal(l2, l3)
    h2 = c2.cpu().numpy()
    for k in range(hist.shape[0]):
        assert relerr(hist[k], S.integrated_time(h2[:50 * (k + 1)], quiet=True)).max() <= 1e-10
    lk.close()
