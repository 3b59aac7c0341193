"""Credible bands of the model light curve over posterior draws: mp_columns_order_statistics, Likelihood.curve_band and
plot_synth.posterior_band_device, against np.sort and np.percentile.

References: order statistics are np.sort of every column with -0.0 ordered before +0.0 and NaNs given their sign bit
cleared (the total order of mp_chain_order_statistics), compared bit for bit.  Bands are np.percentile(curves, q,
axis=0) of the same physical draws' curves from the host-pointer Likelihood.curves, compared by value with NaN equal to
NaN: np.percentile takes the sign of a zero from wherever its partition leaves -0.0 and +0.0.

CPU: the percentile helpers against np.percentile, the C ABI's argument checks, the header constant, and the Python
argument checks.  GPU: the selection across column counts, strides, ranks and special values; the band against NumPy
with and without the ODE state; draws whose integration fails."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT, has_gpu
from magprop_b200.synthetic import plot_synth as P

QS = (0.0, 2.5, 16.0, 50.0, 84.0, 97.5, 100.0)


def same_value(got, want):
    """Equal values, NaN equal to NaN, -0.0 equal to +0.0."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    return got.shape == want.shape and np.array_equal(got, want, equal_nan=True)


def same_bits(got, want):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    return got.shape == want.shape and np.array_equal(got.view(np.uint64), want.view(np.uint64))


def band_columns(n, rng):
    """[n, 12] columns: ties, repeated values, magnitudes from 1e-300 to 1e300, signed zeros, infinities, a NaN."""
    cols = [rng.randn(n),
            np.round(rng.randn(n), 1),                                            # ties
            rng.choice([-1.5, 2.0, 7.0, 7.000000000000001], n),                   # long runs of few values
            np.full(n, 3.25),                                                      # one value repeated
            rng.randn(n) * 10.0 ** rng.uniform(-300, 300, n),                      # wide magnitudes, both signs
            np.abs(rng.randn(n)) * 10.0 ** rng.uniform(-5, 5, n),
            np.where(rng.rand(n) < 0.5, 0.0, -0.0),                                # only signed zeros
            rng.choice([0.0, -0.0, 1e-300, -1e-300], n),
            np.where(rng.rand(n) < 0.1, np.inf, rng.randn(n)),
            np.where(rng.rand(n) < 0.1, -np.inf, rng.randn(n)),
            rng.choice([-np.inf, np.inf], n),
            np.where(np.arange(n) == n // 2, np.nan, rng.randn(n))]               # a NaN: NaN percentiles
    return np.stack(cols, axis=1)


# ---- CPU ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2, 3, 10, 4097])
def test_percentile_helpers_match_numpy(n):
    """The array helpers fed exact order statistics from np.sort == np.percentile(x, q, axis=0), column by column."""
    rng = np.random.RandomState(n)
    x = band_columns(n, rng)
    for q in (QS, (50.0,), (97.5, 2.5, 2.5, 100.0, 0.0), rng.uniform(0, 100, 9)):
        s = np.sort(x, axis=0)
        k0, k1, gamma, ranks = P.percentile_ranks(n, q)
        assert ranks[-1] == n - 1 and np.array_equal(ranks, np.unique(np.r_[k0, k1, n - 1]))
        with np.errstate(invalid="ignore"):
            want = np.percentile(x, q, axis=0)
        got = P.interpolate_percentiles(s[k0], s[k1], gamma, s[n - 1])
        assert same_value(got, want), (n, q)
        nz = want != 0                                        # every non-zero result to the bit
        assert same_bits(got[nz], want[nz])
    # (n - 1) q integral or nearly so for every q
    for m in (41, 401, 4001):
        col = rng.randn(m, 3)
        s = np.sort(col, axis=0)
        k0, k1, gamma, _ = P.percentile_ranks(m, QS)
        assert same_bits(P.interpolate_percentiles(s[k0], s[k1], gamma, s[m - 1]), np.percentile(col, QS, axis=0))


def test_columns_order_statistics_argument_checks(built):
    from magprop_b200 import _capi as A
    lib = A.load()
    n, n_cols, ld = 10, 4, 5
    span = ((n - 1) * ld + n_cols) * 8
    if has_gpu():                         # real buffers, so an implementation that reads before it checks cannot fault
        import torch
        real = torch.zeros(1 << 16, dtype=torch.float64, device="cuda")
        x = real.data_ptr()
    else:                                 # never dereferenced: the checks come before the device is touched
        x = 1 << 20
    far = x + (1 << 18)
    ranks = np.array([0, 9, 3, 3], dtype=np.int64)

    def call(d_x=x, n=n, n_cols=n_cols, ld=ld, ranks=A.ptr(ranks), n_ranks=4, d_out=far):
        return lib.mp_columns_order_statistics(C.c_void_p(d_x) if d_x else None, n, n_cols, ld, ranks, n_ranks,
                                               C.c_void_p(d_out) if d_out else None, 0, None)

    bad = [dict(d_x=0), dict(d_out=0), dict(ranks=None), dict(n=0), dict(n=-1), dict(n=A.MP_COLUMN_SELECT_MAX + 1),
           dict(n_cols=0), dict(n_cols=-1), dict(ld=n_cols - 1), dict(n_ranks=0), dict(n_ranks=-1),
           dict(d_out=x), dict(d_out=x + span - 8), dict(d_out=x - 4 * n_cols * 8 + 8), dict(d_out=x + 16)]
    for kw in bad:
        assert call(**kw) == A.MP_ERR_BAD_ARG, kw
    for bad_rank in (-1, n, 1 << 40):
        r = np.array([0, bad_rank, 2], dtype=np.int64)
        assert call(ranks=A.ptr(r), n_ranks=3) == A.MP_ERR_BAD_ARG, bad_rank
    from magprop_b200.engine import columns_order_statistics
    with pytest.raises(ValueError):
        columns_order_statistics(x, n, n_cols, ld, [0, n], far)
    if not has_gpu():                     # valid arguments, no device; out just before or just after x's span
        for d_out in (far, x + span, x - 4 * n_cols * 8):
            assert call(d_out=d_out) == A.MP_ERR_CUDA
        assert call(n=A.MP_COLUMN_SELECT_MAX, ld=n_cols, d_out=x + A.MP_COLUMN_SELECT_MAX * n_cols * 8) == A.MP_ERR_CUDA


def test_band_header_matches_the_binding(built):
    """include/magprop_band.h defines MP_COLUMN_SELECT_MAX as _capi does, and declares exactly BAND_EXPORTS, which the
    library exports."""
    from magprop_b200 import _capi as A
    src = open(os.path.join(ROOT, "include", "magprop_band.h")).read()
    m = re.search(r"^#define MP_COLUMN_SELECT_MAX (\d+)$", src, flags=re.M)
    assert m and int(m.group(1)) == A.MP_COLUMN_SELECT_MAX == 16384
    code = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    assert sorted(set(re.findall(r"\b(mp_[a-z0-9_]+)\s*\(", code))) == A.BAND_EXPORTS
    lib = A.load()
    for name in A.BAND_EXPORTS:
        assert hasattr(lib, name) and name not in A.EXPORTS + A.SMC_EXPORTS


def test_band_arguments_are_checked_before_any_device_work(monkeypatch):
    """Bad arguments raise ValueError before a handle, a launch or a CUDA tensor is touched: the handle here has no
    device behind it, and making one would raise."""
    import torch
    from magprop_b200 import _cache
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood

    def no_handle(*a, **k):
        raise AssertionError("a handle was asked for")

    monkeypatch.setattr(_cache, "get", no_handle)
    lk = Likelihood.__new__(Likelihood)   # no handle: any call into the library would fail
    lk.device = 0
    ok = torch.zeros((8, 6), dtype=torch.float64)
    for q in ([-1.0], [100.5], [50.0, np.nan], [np.inf], []):
        with pytest.raises(ValueError, match="percentiles"):
            lk.curve_band(ok, q)
        with pytest.raises(ValueError, match="percentiles"):
            P.posterior_band_device(ok, percentiles=q)
    for pars in (np.zeros((8, 6)), ok.float(), ok[0], ok.reshape(2, 4, 6)):
        with pytest.raises(ValueError, match="2-D float64"):
            lk.curve_band(pars, (50.0,))
    for S in (0, A.MP_COLUMN_SELECT_MAX + 1):
        with pytest.raises(ValueError, match="number of draws"):
            lk.curve_band(torch.zeros((S, 6), dtype=torch.float64), (50.0,))
    with pytest.raises(ValueError, match="cuda:0"):      # a host tensor
        lk.curve_band(ok, (50.0,))
    for n_draws in (0, -3, A.MP_COLUMN_SELECT_MAX + 1, 2.5, True):
        with pytest.raises(ValueError, match="n_draws"):
            P.posterior_band_device(ok, n_draws=n_draws)
    with pytest.raises(ValueError, match="unknown model knobs"):
        P.posterior_band_device(ok, rtol=1e-6)
    for chain in (ok, ok.numpy(), ok.float(), torch.zeros((8, 5), dtype=torch.float64),
                  torch.zeros((0, 6), dtype=torch.float64)):
        with pytest.raises(ValueError, match="chain"):
            P.posterior_band_device(chain)


# ---- GPU ----------------------------------------------------------------------------------------------------
NAN_POS, NAN_NEG = np.array([0x7FF8000000000000, 0xFFF8000000000000], dtype=np.uint64).view(np.float64)


def select_columns(n, n_cols, rng):
    """[n, n_cols]: per column a Gaussian, wide magnitudes, or ties, with planted +-0.0, +-inf and NaNs of either sign
    (one payload, so the sorted NaNs are the same bits whatever their order)."""
    kind = rng.randint(0, 3, n_cols)
    x = np.where(kind == 0, rng.randn(n, n_cols),
                 np.where(kind == 1, rng.randn(n, n_cols) * 10.0 ** rng.uniform(-300, 300, (n, n_cols)),
                          rng.choice([-2.0, 0.5, 0.5000000000000001, 3.0], (n, n_cols))))
    special = np.array([0.0, -0.0, np.inf, -np.inf, NAN_POS, NAN_NEG])
    plant = rng.rand(n, n_cols) < 0.06
    x[plant] = special[rng.randint(0, special.size, int(plant.sum()))]
    return x


def sorted_reference(x):
    """np.sort of every column in the library's total order: -0.0 before +0.0, NaNs with the sign bit cleared."""
    s = np.sort(x.T, axis=1).T                               # rows sorted along the contiguous axis
    zero = s == 0
    rank_in_zeros = np.cumsum(zero, axis=0) - 1
    n_neg = ((x == 0) & np.signbit(x)).sum(axis=0)
    s[zero] = np.where(rank_in_zeros < n_neg[None, :], -0.0, 0.0)[zero]
    s[np.isnan(s)] = NAN_POS
    return s


@pytest.mark.gpu
@pytest.mark.parametrize("n_cols", [1, 129, 30003])
@pytest.mark.parametrize("n", [1, 2, 31, 1000, 4096, 16384])
def test_columns_order_statistics_match_np_sort(built, n, n_cols):
    import torch
    from magprop_b200.engine import columns_order_statistics
    rng = np.random.RandomState(n * 7 + n_cols)
    x = select_columns(n, n_cols, rng)
    want = sorted_reference(x)
    ld = n_cols + 3 if n_cols != 30003 else n_cols           # rows with a gap between them, except at the largest size
    buf = torch.full((n * ld + 5,), float("nan"), dtype=torch.float64, device="cuda")   # NaN outside the columns
    view = buf[2:2 + n * ld].view(n, ld)
    view[:, :n_cols] = torch.from_numpy(x).cuda()
    if n <= 31 or (n == 1000 and n_cols == 129):             # every rank (1000: four launches of 256 ranks)
        ranks = rng.permutation(n)
    else:                                                    # the ends, a few inside, unsorted and repeated
        ranks = rng.permutation(np.r_[0, 1, n // 2, n - 2, n - 1, rng.randint(0, n, 12), n - 1, 0])
    ranks = np.r_[ranks, ranks[:3]]

    def run(stream=0):
        out = torch.full((ranks.size, n_cols), 7.0, dtype=torch.float64, device="cuda")
        columns_order_statistics(view.data_ptr(), n, n_cols, ld, ranks, out.data_ptr(), stream=stream)
        return out.cpu().numpy()

    got = run()
    assert same_bits(got, want[ranks]), (n, n_cols)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        again = run(side.cuda_stream)
    assert got.tobytes() == again.tobytes()


@pytest.fixture(scope="module")
def humped_chain(built, golden):
    """A DeviceEnsemble chain of the Humped fit [120, 64, 6] on the device."""
    import torch
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, time_grid
    from magprop_b200.sampler import DeviceEnsemble
    from oracle import magprop_oracle as O
    g = golden["lnprob_script"]
    lk = Likelihood(A.script_model_spec(), time_grid(None), g["Humped_x"], g["Humped_y"], g["Humped_yerr"],
                    O.SCRIPT_LOWER, O.SCRIPT_UPPER)
    ens = DeviceEnsemble.from_likelihood(lk, 64, 6, seed=5)
    ens.initialise(O.SYNTH_TRUTHS_LOG["Humped"] + 1e-2 * np.random.RandomState(2).randn(64, 6))
    chain, _ = ens.run(120, store=True)
    torch.cuda.synchronize()
    yield chain
    lk.close()


def physical_draws(chain, n_draws):
    """The draws posterior_band_device takes, un-logged the same way (on the device)."""
    import torch
    flat = chain.reshape(-1, 6)
    n = flat.shape[0]
    rows = np.arange(n_draws) * n // n_draws if n > n_draws else np.arange(n)
    logp = flat[torch.from_numpy(rows).cuda()]
    pars = logp.clone()
    pars[:, 2:] = torch.pow(10.0, pars[:, 2:])
    host = pars.cpu().numpy()
    ref = logp.cpu().numpy()
    ref[:, 2:] = 10.0 ** ref[:, 2:]
    assert np.allclose(host, ref, rtol=4e-16, atol=0)         # the host's un-logging, to the last bit or so
    return pars, host


def curves_both_ways(lk, pars, host, node_stride):
    """Host-pointer curves (the reference's arrays) and a check that the device path returns the same bits."""
    import torch
    out, state, status = lk.curves(host, node_stride=node_stride, with_state=True)
    S, Gs = host.shape[0], lk.curve_nodes(node_stride)
    d_out = torch.empty((S, 3, Gs), dtype=torch.float64, device="cuda")
    d_state = torch.empty((S, 2, Gs), dtype=torch.float64, device="cuda")
    d_status = torch.empty(S, dtype=torch.int32, device="cuda")
    lk.curves_device(pars.data_ptr(), S, 6, node_stride, d_out.data_ptr(), d_state.data_ptr(), d_status.data_ptr(),
                     torch.cuda.current_stream().cuda_stream)
    assert same_bits(d_out.cpu().numpy(), out) and same_bits(d_state.cpu().numpy(), state)
    assert np.array_equal(d_status.cpu().numpy(), status)
    return out, state, status


def check_band(band, out, state, status, q, with_state):
    keep = (status & 2) == 0
    assert band.n_used == int(keep.sum()) and band.n_flagged == int((~keep).sum())
    assert np.array_equal(band.percentiles, np.asarray(q, dtype=np.float64))
    want = np.percentile(out[keep], q, axis=0)
    for i, name in enumerate(("ltot", "lprop", "ldip")):
        assert same_value(getattr(band, name), want[:, i]), name
    if with_state:
        want = np.percentile(state[keep], q, axis=0)
        assert same_value(band.mdisc, want[:, 0]) and same_value(band.omega, want[:, 1])
    else:
        assert band.mdisc is None and band.omega is None


@pytest.mark.gpu
@pytest.mark.parametrize("with_state", [False, True])
@pytest.mark.parametrize("node_stride", [1, 7])
def test_posterior_band_equals_numpy(built, humped_chain, node_stride, with_state):
    import torch
    from magprop_b200 import _cache
    from magprop_b200 import _capi as A
    n_draws = 1000
    band = P.posterior_band_device(humped_chain, n_draws=n_draws, node_stride=node_stride, with_state=with_state)
    pars, host = physical_draws(humped_chain, n_draws)
    lk = _cache.get(A.script_model_spec(unlog=False), None, device=0)
    out, state, status = curves_both_ways(lk, pars, host, node_stride)
    q = (2.5, 16.0, 50.0, 84.0, 97.5)
    check_band(band, out, state, status, q, with_state)
    assert np.array_equal(band.t, lk.node_times(node_stride)) and band.ltot.shape == (5, band.t.size)
    # any percentiles, on a side stream, from the Likelihood directly: the same bits
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        other = lk.curve_band(pars, QS, node_stride=node_stride, with_state=with_state)
    check_band(other, out, state, status, QS, with_state)
    assert same_bits(other.ltot[1:6], band.ltot) and same_bits(other.ldip[1:6], band.ldip)
    if node_stride == 7 and not with_state:                  # fewer rows than n_draws: every row, 7680 draws
        whole = P.posterior_band_device(humped_chain, n_draws=16384, node_stride=node_stride)
        pars, host = physical_draws(humped_chain, 16384)
        out, state, status = lk.curves(host, node_stride=node_stride, with_state=True)
        assert whole.n_used + whole.n_flagged == 7680
        check_band(whole, out, state, status, q, False)


@pytest.mark.gpu
def test_flagged_draws_are_left_out(built, humped_chain):
    """A step budget small enough to fail part of the draws: n_flagged counts them, the band is np.percentile over the
    rest, draws whose state turns non-finite (the reference clamps their luminosity to 0 there) stay in, and a set of
    only failing draws raises."""
    import torch
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, time_grid
    from oracle import magprop_oracle as O
    rng = np.random.RandomState(11)
    lo, hi = np.asarray(O.SCRIPT_LOWER), np.asarray(O.SCRIPT_UPPER)
    wide = lo + (hi - lo) * rng.rand(300, 6)                 # prior-wide draws: step counts spread widely
    wide[:, 2:] = 10.0 ** wide[:, 2:]
    _, posterior = physical_draws(humped_chain, 300)
    nan_state = np.array([[1.0, 5.0, -3.0, 2.0, -1.0, 0.0], [2.0, 3.0, -2.0, 1.0, -0.5, 0.5]])  # log values, unconverted
    host = np.concatenate([wide, posterior, nan_state])
    pars = torch.from_numpy(host).cuda()
    for max_steps in (40, 80, 160, 320, 640, 1280, 2560):
        lk = Likelihood(A.script_model_spec(unlog=False, max_steps=max_steps), time_grid(None))
        out, state, status = lk.curves(host, node_stride=11, with_state=True)
        failed = (status & A.WALKER_INTEGRATOR_FAIL) != 0
        if 0 < failed.sum() < 0.8 * host.shape[0]:
            break
        lk.close()
    assert 0 < failed.sum() < host.shape[0], failed.sum()
    kept_nan = ((status & A.WALKER_NONFINITE_STATE) != 0) & ~failed
    assert kept_nan[-2:].any() and np.isfinite(out[kept_nan]).all()   # kept: counted in n_used below
    band = lk.curve_band(pars, QS, node_stride=11, with_state=True)
    assert band.n_flagged == int(failed.sum()) and band.n_used == int((~failed).sum())
    check_band(band, out, state, status, QS, True)
    with pytest.raises(RuntimeError):
        lk.curve_band(pars[torch.from_numpy(np.flatnonzero(failed)).cuda()], QS, node_stride=11)
    lk.close()
