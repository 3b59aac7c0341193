"""Posterior summaries of a device-resident chain (mp_chain_moments, mp_chain_order_statistics and
plot_synth.posterior_summary_device, DESIGN.md row f4) against exact host references.

References: the mean is math.fsum(col) / n; the covariance is two-pass, centred on the reference mean, with the
products summed by math.fsum -- or in Fractions, exactly, for small n and planted values; order statistics are np.sort
with NaNs last and -0.0 before +0.0 (the total order the kernel's keys define), compared bit for bit, any NaN equal to
any NaN.  The moment bars follow from the depth of the kernels' summation tree (``depth``), not from observed errors.

CPU: the entry points' argument checks, and the percentile rule of posterior_summary_device against np.percentile.
GPU: moments and order statistics across the grid-stride boundaries, special values and ties; identical bits from
repeated calls and on a side stream; ordering on the caller's stream; the device summary against the host one; and,
where the memory is free, a chain past 2^31 elements and a column of more than 2^32 rows."""
import ctypes as C
import math
import warnings
from fractions import Fraction

import numpy as np
import pytest

from conftest import has_gpu
from magprop_b200.synthetic import plot_synth as P

U = 2.0 ** -53                         # unit roundoff of float64
BLOCKS, THREADS = 1184, 256            # the moment kernels' grid (mp_chain_moments)
NS = [1, 2, 255, 256, 257, BLOCKS * THREADS - 1, BLOCKS * THREADS, BLOCKS * THREADS + 1, 3 * BLOCKS * THREADS + 17]


def gamma(L):
    return L * U / (1.0 - L * U)


def depth(n):
    """The most roundings any element of a column meets on its way into a moment kernel's sum: the serial terms of its
    thread, 5 warp-shuffle levels, the 8 warps of its block, and the finishing sum over the blocks in block order."""
    blocks = min(-(-n // THREADS), BLOCKS)
    return -(-n // (blocks * THREADS)) + 5 + 8 + blocks


def ref_moments(x):
    """Mean, covariance (n - 1 normalisation, 1 for n = 1) and the bars' ingredients: the reference mean's own error
    bound r[d] and sabs[a, b] = sum |c_a| |c_b| of the centred values.  Exact (Fractions) up to 3000 rows."""
    n, nd = x.shape
    exact = n <= 3000
    if exact:
        fx = [[Fraction(float(v)) for v in x[:, d]] for d in range(nd)]
        mu = [sum(col) / n for col in fx]
        mean = np.array([float(m) for m in mu])
        r = U * np.abs(mean)                               # the one rounding of the exact mean
        cen = [[v - m for v in col] for col, m in zip(fx, mu)]
        cov = np.array([[float(sum(p * q for p, q in zip(cen[a], cen[b])) / max(n - 1, 1)) for b in range(nd)]
                        for a in range(nd)])
    else:
        mean = np.array([math.fsum(x[:, d]) / n for d in range(nd)])
        r = 2 * U * np.abs(mean)                           # fsum rounds once, the division once
        c = x - mean
        cov = np.array([[math.fsum(c[:, a] * c[:, b]) / max(n - 1, 1) for b in range(nd)] for a in range(nd)])
    c = np.abs(x - mean)
    sabs = c.T @ c                                         # a bound's size, not a result: its own rounding is immaterial
    return mean, cov, r, sabs


def check_moments(x, mean, cov):
    """mean and cov from the device within the summation-tree bars of the reference."""
    n, nd = x.shape
    L = depth(n)
    rmean, rcov, r, sabs = ref_moments(x)
    mbar = gamma(L + 1) * np.abs(x).sum(axis=0) / n + r    # + 1: the division by n
    err = np.abs(mean - rmean)
    assert (err <= mbar).all(), (n, nd, err, mbar)
    # The device centres on its mean m = mu + delta: sum (x_a - m_a)(x_b - m_b) = R_ab + n delta_a delta_b exactly,
    # as sum (x - mu) = 0.  Two roundings of the centred values, L of the sum, one of the division (and the
    # reference's own three products-and-division roundings and centring): gamma(L + 8).
    d = err + 2 * r
    cbar = (gamma(L + 8) * sabs + n * np.outer(d, d)) / max(n - 1, 1)
    cerr = np.abs(cov - rcov)
    assert (cerr <= cbar).all(), (n, nd, cerr.max(), cbar)
    assert np.array_equal(cov, cov.T)


def ref_sorted(col):
    """np.sort, with the zeros ordered -0.0 before +0.0 (np.sort leaves them in any order; NaNs are last either way)."""
    s = np.sort(col)
    z = np.flatnonzero(s == 0)
    s[z] = np.where(np.arange(z.size) < np.signbit(col[col == 0]).sum(), -0.0, 0.0)
    return s


def same_bits(got, want):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    nan = np.isnan(want)
    return (got.shape == want.shape and np.array_equal(np.isnan(got), nan)
            and np.array_equal(got[~nan].view(np.uint64), want[~nan].view(np.uint64)))


def from_bits(*patterns):
    return np.array(patterns, dtype=np.uint64).view(np.float64)


# ---- CPU ----------------------------------------------------------------------------------------------------
def test_chain_summary_argument_checks(built):
    from magprop_b200 import _capi as A
    lib = A.load()
    if has_gpu():                         # a real chain, so an implementation that reads before it checks cannot fault
        import torch
        real = torch.zeros((10, 3), dtype=torch.float64, device="cuda")
        fake = C.c_void_p(real.data_ptr())
    else:                                 # never dereferenced: the checks come before the device is touched
        fake = C.c_void_p(4096)
    mean, cov, vals = np.empty(16), np.empty(256), np.empty(8)
    ranks = np.array([0, 1, 2], dtype=np.int64)

    def mom(d_chain=fake, n=10, ndim=3, mean=A.ptr(mean), cov=A.ptr(cov)):
        return lib.mp_chain_moments(d_chain, n, ndim, mean, cov, 0, None)

    def osel(d_chain=fake, n=10, ndim=3, col=1, ranks=A.ptr(ranks), n_ranks=3, values=A.ptr(vals)):
        return lib.mp_chain_order_statistics(d_chain, n, ndim, col, ranks, n_ranks, values, 0, None)

    bad_mom = [dict(d_chain=None), dict(mean=None), dict(cov=None), dict(n=0), dict(n=-1), dict(ndim=0),
               dict(ndim=A.MP_MAX_NDIM + 1)]
    for kw in bad_mom:
        assert mom(**kw) == A.MP_ERR_BAD_ARG, kw
    bad_sel = [dict(d_chain=None), dict(ranks=None), dict(values=None), dict(n=0), dict(ndim=0), dict(col=-1),
               dict(col=3), dict(n_ranks=-1)]
    for kw in bad_sel:
        assert osel(**kw) == A.MP_ERR_BAD_ARG, kw
    for bad_rank in (-1, 10):             # ranks outside [0, n) are refused before any device work
        r = np.array([0, bad_rank, 2], dtype=np.int64)
        assert osel(ranks=A.ptr(r)) == A.MP_ERR_BAD_ARG
    with pytest.raises(ValueError):
        A.check(mom(ndim=0))
    if not has_gpu():                     # valid arguments, no device
        assert mom() == A.MP_ERR_CUDA and mom(ndim=A.MP_MAX_NDIM) == A.MP_ERR_CUDA
        assert osel() == A.MP_ERR_CUDA and osel(n_ranks=0) == A.MP_ERR_CUDA


def test_percentile_rule_matches_numpy():
    """posterior_summary_device's percentiles from two order statistics == np.percentile of the whole column, the
    un-logged columns included.  Compared by value: np.percentile's sign of a zero result depends on where its
    partition leaves -0.0 and +0.0, which nothing orders."""
    rng = np.random.RandomState(12)
    for t in range(3000):
        n = int(rng.randint(1, 60)) if t % 3 == 0 else int(rng.randint(1, 5001))
        col = rng.randn(n) * 0.5 - 1.0
        if t % 5 == 0:
            col = np.round(col, 1)                           # ties
        unlog = bool(t % 2)
        s = np.sort(col)
        got = P.percentiles_from_order_statistics(n, lambda r: s[r], unlog=unlog)
        want = np.percentile(10.0 ** col if unlog else col, P.PERCENTILES)
        assert np.array_equal(got, want), (t, n, unlog, got, want)
    for n in (1, 2, 3, 41, 401, 4001):                       # (n - 1) q integral, or nearly, for every q
        col = rng.randn(n)
        s = np.sort(col)
        assert np.array_equal(P.percentiles_from_order_statistics(n, lambda r: s[r]), np.percentile(col, P.PERCENTILES))
    # a NaN anywhere makes every percentile NaN, as np.percentile's does
    col = np.array([1.0, -2.0, np.nan, 0.5, 3.0])
    s = np.sort(col)
    got = P.percentiles_from_order_statistics(5, lambda r: s[r], unlog=True)
    assert np.isnan(got).all() and np.isnan(np.percentile(10.0 ** col, P.PERCENTILES)).all()


# ---- GPU ----------------------------------------------------------------------------------------------------
def _dev(x):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _padded(x, before=3, after=2):
    """x on the device as a row-offset view into a larger allocation whose other rows are NaN: a read outside the
    view's rows poisons the result."""
    import torch
    n, nd = x.shape
    buf = torch.full((before + n + after, nd), float("nan"), dtype=torch.float64, device="cuda")
    buf[before:before + n] = _dev(x)
    return buf, buf[before:before + n]


def _moments(t, **kw):
    from magprop_b200.engine import chain_moments
    return chain_moments(t.data_ptr(), t.shape[0], t.shape[1], **kw)


def _select(t, col, ranks, **kw):
    from magprop_b200.engine import chain_order_statistics
    return chain_order_statistics(t.data_ptr(), t.shape[0], t.shape[1], col, ranks, **kw)


def dataset(kind, n, nd, rng):
    if kind == "gauss":
        return rng.randn(n, nd) * rng.uniform(0.5, 2.0, nd) + rng.uniform(-3, 3, nd)
    if kind == "offset":                                     # the two-pass centring: the spread is 1e-10 of the level
        return 1e6 + 1e-4 * rng.randn(n, nd)
    if kind == "scales":                                     # columns from 1e-8 to 1e8
        return rng.randn(n, nd) * np.logspace(-8, 8, nd) + np.logspace(-7, 9, nd)
    if kind == "collinear":                                  # a constant, a duplicated and a negated column
        x = rng.randn(n, nd) + 5.0
        x[:, 0] = 2.5
        if nd >= 3:
            x[:, 2] = x[:, 1]
        if nd >= 4:
            x[:, 3] = -x[:, 1]
        return x
    raise ValueError(kind)


@pytest.mark.gpu
@pytest.mark.parametrize("n", NS)
def test_chain_moments_match_the_reference(built, n):
    rng = np.random.RandomState(n)
    for nd in (1, 2, 5, 6, 9):
        for kind in ("gauss", "offset", "scales", "collinear"):
            x = dataset(kind, n, nd, rng)
            _, view = _padded(x)
            mean, cov = _moments(view)
            check_moments(x, mean, cov)
            if n == 1:                                       # the library's convention: / max(n - 1, 1)
                assert np.array_equal(mean, x[0]) and not cov.any()
            if kind == "collinear":
                assert mean[0] == 2.5 and not cov[0].any() and not cov[:, 0].any()   # constant: exactly 0
                if nd >= 3:                                  # identical sums in identical order
                    assert mean[2] == mean[1] and cov[1, 2] == cov[1, 1] == cov[2, 2]
                if nd >= 4:
                    assert mean[3] == -mean[1] and cov[1, 3] == -cov[1, 1] and cov[3, 3] == cov[1, 1]


def _special_column():
    specials = np.concatenate([
        [0.0, -0.0, np.inf, -np.inf, np.finfo(np.float64).max, -np.finfo(np.float64).max, 5e-324, -5e-324,
         np.finfo(np.float64).tiny, -np.finfo(np.float64).tiny, 1.0, -1.0],
        from_bits(0x7FF8000000000000, 0x7FF0000000000001, 0x7FFFFFFFFFFFFFFF,    # positive NaNs, payloads
                  0xFFF8000000000000, 0xFFF0000000000123, 0xFFFFFFFFFFFFFFFF)])  # negative NaNs (0/0 on x86)
    return np.concatenate([specials, specials[[0, 1, 1, 2, 5, 6, 7, 12, 15]], [3.5, -2.25]])


def _low_digit_column(rng, n):
    """Values whose top 48 bits agree (two groups, one negative), so only the last pass tells them apart."""
    lo = rng.randint(0, 1 << 16, n).astype(np.uint64)
    hi = np.where(rng.rand(n) < 0.5, np.uint64(0x3FF3C0CA42830000), np.uint64(0xC00921FB54440000))
    return (hi | lo).view(np.float64)


def _top_digit_column(rng, n):
    """Values that differ only in the top 16 bits: magnitudes, signs, infinities' and NaNs' exponents."""
    top = rng.randint(0, 1 << 16, n).astype(np.uint64)
    return ((top << np.uint64(48)) | np.uint64(0x0000_1234_5678_9ABC)).view(np.float64)


def _tie_column(rng, n):
    """Long runs of few values (a stuck walker, a prior edge)."""
    return rng.choice(np.array([-1.5, 0.0, 2.0, 7.0, 7.000000000000001]), size=n, p=[0.1, 0.2, 0.3, 0.2, 0.2])


@pytest.mark.gpu
def test_order_statistics_special_values_and_all_ranks(built):
    col = _special_column()
    rng = np.random.RandomState(4)
    col = col[rng.permutation(col.size)]
    n = col.size
    for nd, c in ((1, 0), (3, 2)):
        x = rng.randn(n, nd)
        x[:, c] = col
        _, view = _padded(x)
        want = ref_sorted(col)
        got = _select(view, c, np.arange(n))
        assert same_bits(got, want), (got, want)
        k = int(np.isnan(col).sum())                         # every NaN last, negative ones included
        assert k == 8 and np.isnan(got[-k:]).all() and got[-k - 1] == np.inf and got[0] == -np.inf
        assert same_bits(_select(view, c, [n - 1, 0, 3, 3, n - 1, 7]), want[[n - 1, 0, 3, 3, n - 1, 7]])
        assert _select(view, c, []).shape == (0,)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 257, 3 * BLOCKS * THREADS + 17])
def test_order_statistics_every_column_of_a_nine_wide_chain(built, n):
    """Each column stresses one part of the select: low-digit ties, top-digit differences, tie runs, specials."""
    rng = np.random.RandomState(100 + n)
    x = np.empty((n, 9))
    x[:, 0] = rng.randn(n)
    x[:, 1] = _low_digit_column(rng, n)
    x[:, 2] = _top_digit_column(rng, n)
    x[:, 3] = _tie_column(rng, n)
    x[:, 4] = -np.abs(rng.randn(n)) * 1e-300                 # negative, subnormal and tiny
    x[:, 5] = np.resize(_special_column(), n)
    x[:, 6] = 1e6 + 1e-4 * rng.randn(n)
    x[:, 7] = np.where(rng.rand(n) < 0.5, 0.0, -0.0)         # only signed zeros
    x[:, 8] = rng.randint(-3, 4, n).astype(np.float64)
    _, view = _padded(x)
    for c in range(9):
        want = ref_sorted(x[:, c])
        if n <= 300:
            ranks = np.arange(n)
        else:                                                # the ends, a few inside, and both ends of every run
            starts = np.flatnonzero(np.r_[True, want[1:].view(np.uint64) != want[:-1].view(np.uint64)])
            runs = np.unique(np.r_[starts, starts - 1, starts + 1][:200])
            ranks = np.r_[0, 1, n // 2, n - 2, n - 1, rng.randint(0, n, 8), runs[(runs >= 0) & (runs < n)][:40]]
            ranks = rng.permutation(ranks)                   # unsorted, possibly repeated
        assert same_bits(_select(view, c, ranks), want[ranks]), (n, c)


@pytest.mark.gpu
def test_order_statistics_tie_runs_and_bad_ranks(built):
    from magprop_b200.engine import chain_order_statistics
    rng = np.random.RandomState(9)
    n = 2 * BLOCKS * THREADS + 5
    col = np.sort(_tie_column(rng, n))                       # runs laid out in order, then shuffled
    bounds = np.flatnonzero(np.r_[True, col[1:] != col[:-1], True])
    col = col[rng.permutation(n)]
    t = _dev(col.reshape(-1, 1))
    want = ref_sorted(col)
    ranks = np.unique(np.r_[bounds[:-1], bounds[1:] - 1, (bounds[:-1] + bounds[1:]) // 2])   # first, last, inside
    assert same_bits(_select(t, 0, ranks[::-1]), want[ranks[::-1]])
    for bad in (-1, n):
        with pytest.raises(ValueError):
            chain_order_statistics(t.data_ptr(), n, 1, 0, [0, bad])
        assert same_bits(_select(t, 0, [0, n - 1]), want[[0, n - 1]])   # the next call on the chain succeeds
    assert same_bits(_select(t, 0, [n // 2]), want[[n // 2]])


@pytest.fixture(scope="module")
def ensemble_chain(built, golden):
    """A DeviceEnsemble chain of the Humped fit [120, 64, 6] on the device, its host copy and the dataset."""
    import torch
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, time_grid
    from magprop_b200.sampler import DeviceEnsemble
    from oracle import magprop_oracle as O
    g = golden["lnprob_script"]
    x, y, yerr = g["Humped_x"], g["Humped_y"], g["Humped_yerr"]
    lk = Likelihood(A.script_model_spec(), time_grid(None), x, y, yerr, O.SCRIPT_LOWER, O.SCRIPT_UPPER)
    ens = DeviceEnsemble.from_likelihood(lk, 64, 6, seed=5)
    ens.initialise(O.SYNTH_TRUTHS_LOG["Humped"] + 1e-3 * np.random.RandomState(2).randn(64, 6))
    chain, _ = ens.run(120, store=True)
    torch.cuda.synchronize()
    yield chain, chain.cpu().numpy().reshape(-1, 6), (x, y, yerr)
    lk.close()


def _near_truth(n, seed):
    from oracle import magprop_oracle as O
    return O.SYNTH_TRUTHS_LOG["Humped"] + 1e-3 * np.random.RandomState(seed).randn(n, 6)


def _summary_bytes(s, p):
    return (repr(s), np.asarray(p).tobytes())


@pytest.mark.gpu
def test_summaries_are_deterministic(built, ensemble_chain):
    """Two calls and a call on a side stream: identical bytes, for a chain of many blocks and for a sampler's chain."""
    import torch
    chain, _, (x, y, yerr) = ensemble_chain
    big = _dev(_near_truth(3 * BLOCKS * THREADS + 17, 1))
    for t in (big, chain.reshape(-1, 6)):
        n = t.shape[0]
        ranks = [0, 7, n // 3, n // 2, n - 1]

        def run(**kw):
            m, c = _moments(t, **kw)
            o = [_select(t, col, ranks, **kw) for col in range(6)]
            return m.tobytes() + c.tobytes() + b"".join(v.tobytes() for v in o)

        a, b = run(), run()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            c = run(stream=side.cuda_stream)
        assert a == b == c
    for t in (big, chain):
        first = _summary_bytes(*P.posterior_summary_device(t, x, y, yerr))
        assert _summary_bytes(*P.posterior_summary_device(t, x, y, yerr)) == first
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            assert _summary_bytes(*P.posterior_summary_device(t, x, y, yerr)) == first


@pytest.mark.gpu
def test_summaries_run_on_the_callers_stream(built, ensemble_chain):
    """The chain is written by work queued on a side stream behind a ~0.1 s sleep; the summaries are asked for on
    that stream without a synchronisation and must see the written chain."""
    import torch
    _, host, (x, y, yerr) = ensemble_chain
    src = _dev(host)
    want_s, want_p, _, _ = P.posterior_summary(host, x, y, yerr)
    n = host.shape[0]
    ranks = [0, n // 2, n - 1]
    for primitives in (False, True):
        chain = src * 1.001                                  # what the chain held before
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            torch.cuda._sleep(200_000_000)
            chain.copy_(src)
            if primitives:
                mean, cov = _moments(chain, stream=side.cuda_stream)
                sel = _select(chain, 4, ranks, stream=side.cuda_stream)
            else:
                s, p = P.posterior_summary_device(chain, x, y, yerr)
        torch.cuda.synchronize()
        if primitives:
            check_moments(host, mean, cov)
            assert same_bits(sel, ref_sorted(host[:, 4])[ranks])
        else:
            assert np.array_equal(p, want_p) and s["pars"] == want_s["pars"]


def _corr_bar(x):
    """Reference correlations and bars on cov[a, b] / sd_a / sd_b from the covariance bars of check_moments, with the
    device mean's error at its bar (first order, with a 1e-3 margin for the second)."""
    n = x.shape[0]
    L = depth(n)
    _, rcov, r, sabs = ref_moments(x)
    d = gamma(L + 1) * np.abs(x).sum(axis=0) / n + 2 * r
    cbar = (gamma(L + 8) * sabs + n * np.outer(d, d)) / max(n - 1, 1)
    sd = np.sqrt(np.diag(rcov))
    rel = np.diag(cbar) / np.diag(rcov)
    rcorr = rcov / sd[:, None] / sd[None, :]
    bar = (cbar / np.outer(sd, sd) + np.abs(rcorr) * (rel[:, None] / 2 + rel[None, :] / 2 + 4 * U)) * 1.001
    iu = np.triu_indices(x.shape[1], 1)
    return rcorr[iu], bar[iu]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3, 41, 401, 7680])
def test_device_summary_equals_the_host_summary(built, ensemble_chain, n):
    """Percentiles bit for bit against posterior_summary on the same chain (so the median, the errors and the LaTeX
    cells), correlations within the covariance bars; n = 41 and 401 make (n - 1) q integral, n = 7680 is the whole
    sampler's chain."""
    chain, host, (x, y, yerr) = ensemble_chain
    if n == 7680:
        t, h = chain, host
    elif n == 3:
        # exactly collinear columns: 3, 4 and 5 have the centred values (h, h, -2h), (-h, -h, 2h) and (-h, -h, 2h),
        # so cov = +-3h^2 exactly, where cov / sd / sd rounds to 1 + 2^-52
        h = np.array(_near_truth(3, 3))
        h[:, 4] = [-1.0625, -1.0625, -0.875]
        h[:, 5] = h[:, 4] + 1.0
        h[:, 3] = 1.0 - h[:, 4]
        t = _dev(h)
    else:
        h = host[:n].copy()
        t = _dev(h)
    with warnings.catch_warnings(), np.errstate(all="ignore"):
        warnings.simplefilter("ignore", RuntimeWarning)          # n = 1: no spread, NaN correlations on both sides
        s_dev, p_dev = P.posterior_summary_device(t, x, y, yerr, grb="Humped")
        s_host, p_host, _, _ = P.posterior_summary(h, x, y, yerr, grb="Humped")
    assert np.array_equal(p_dev, p_host)
    assert s_dev["pars"] == s_host["pars"]
    corr = np.array(s_dev["correlations"])
    if n == 1:
        assert np.isnan(corr).all() and np.isnan(s_host["correlations"]).all()
        return
    assert (np.abs(corr) <= 1.0).all()
    want, bar = _corr_bar(h)
    assert (np.abs(corr - want) <= bar).all(), (n, np.abs(corr - want), bar)
    if n == 3:
        iu = list(zip(*np.triu_indices(6, 1)))
        assert corr[iu.index((3, 4))] == corr[iu.index((3, 5))] == -1.0 and corr[iu.index((4, 5))] == 1.0


# ---- large chains: skipped, with the reason, where the memory is not free ---------------------------------------
def _need(nbytes):
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes + (2 << 30):
        pytest.skip(f"needs {nbytes / 1e9:.1f} GB of free device memory, {free / 1e9:.1f} GB free")


@pytest.mark.gpu
def test_summaries_beyond_32bit_element_indexing(built):
    """ndim 9 x 2^28 rows (19.3 GB), 2^12 copies of a seeded 2^16-row block: i * ndim + col passes 2^31."""
    import torch
    rows, nd, base_rows = 1 << 28, 9, 1 << 16
    _need(rows * nd * 8)
    rng = np.random.RandomState(21)
    base = rng.randn(base_rows, nd) * np.arange(1, nd + 1) + np.arange(nd)
    base[:, 8] = np.round(base[:, 8], 2)                     # ties in the column checked
    chain = _dev(base).repeat(rows // base_rows, 1)
    assert chain.numel() > 2 ** 31
    reps = rows // base_rows
    mean, cov = _moments(chain)
    # the tiled chain's exact moments from the block's: the same mean, reps times the centred sums
    fx = [[Fraction(float(v)) for v in base[:, d]] for d in (0, 8)]
    mu = [sum(c) / base_rows for c in fx]
    L = depth(rows)
    for j, d in enumerate((0, 8)):
        assert abs(mean[d] - float(mu[j])) <= gamma(L + 1) * np.abs(base[:, d]).sum() / base_rows + U * abs(mean[d])
        s2 = reps * sum((v - mu[j]) ** 2 for v in fx[j])
        var = s2 / (rows - 1)
        sabs = reps * float(sum(abs(v - mu[j]) ** 2 for v in fx[j]))
        delta = abs(Fraction(float(mean[d])) - mu[j])
        bar = (gamma(L + 8) * sabs + rows * float(delta) ** 2 * 4) / (rows - 1)
        assert abs(Fraction(float(cov[d, d])) - var) <= Fraction(bar), (d, float(cov[d, d]), float(var), bar)
    ref = np.sort(base[:, 8])
    ranks = np.array([0, reps - 1, reps, rows // 2, rows - reps - 1, rows - reps, rows - 1, 123456789])
    assert same_bits(_select(chain, 8, ranks), ref[ranks // reps])
    del chain
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_summaries_of_more_than_2_32_rows(built):
    """n = 2^32 + 2^20 rows (34.4 GB) of 1.0 with 1000 planted 0.5 and 1000 planted 2.0: the 1.0 bin holds more than
    2^32 counts in every pass; every partial sum is a multiple of 0.5 below 2^53, so the mean is exact."""
    import torch
    n = (1 << 32) + (1 << 20)
    _need(n * 8)
    rng = np.random.RandomState(32)
    pos = np.unique(rng.randint(0, n, 2200, dtype=np.int64))
    pos = pos[rng.permutation(pos.size)][:2000]
    chain = torch.ones((n, 1), dtype=torch.float64, device="cuda")
    chain[torch.from_numpy(pos[:1000]).cuda(), 0] = 0.5
    chain[torch.from_numpy(pos[1000:]).cuda(), 0] = 2.0
    got = _select(chain, 0, [999, 1000, n - 1001, n - 1000, n - 1])
    assert same_bits(got, [0.5, 1.0, 1.0, 2.0, 2.0]), got
    mean, cov = _moments(chain)
    mu = Fraction(n + 500, n)
    assert mean[0] == float(mu)
    var = (1000 * (Fraction(1, 2) - mu) ** 2 + 1000 * (2 - mu) ** 2 + (n - 2000) * (1 - mu) ** 2) / (n - 1)
    sabs = float(var) * (n - 1)
    bar = gamma(depth(n) + 8) * sabs / (n - 1) + n * (2 * U) ** 2 / (n - 1)
    assert abs(Fraction(float(cov[0, 0])) - var) <= Fraction(bar), (float(cov[0, 0]), float(var), bar)
    del chain
    torch.cuda.empty_cache()
