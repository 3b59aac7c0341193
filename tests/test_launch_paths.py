"""Every way one evaluation launch can run (``launch_eval`` in magprop_kernels.cu) gives every walker the same result.

How a launch runs depends on its size and on the dataset: the number of slabs, whether the work list is ordered, the
explicit integrator's block size, the implicit integrator's build, the reduce form (warp per walker, ordered warp per
walker, thread per walker) and whether the dataset or the node times are staged in shared memory.  DESIGN.md section 3
promises that a walker's arithmetic is the same in every slot and that the form depends on the dataset only.  These
tests hold each decision at and across its boundary:
  * bit for bit, against the same walkers evaluated in launches that take the other side of the boundary;
  * against the converged oracle (TOL_TIGHT), on datasets built to sit on either side of the dataset-driven
    boundaries.  A CPU test checks that the builders put them there.
Slab and ordering counts come from the handle's kernel counter: a slab costs 4 kernels (2 without data), plus 2 when
its work list is ordered."""
import ctypes as C

import numpy as np
import pytest

from conftest import relerr
import stretch_ref as R
import tempered_ref as TR
from magprop_b200 import _capi as A
from magprop_b200.engine import Likelihood, time_grid
from oracle import magprop_oracle as O

TOL_TIGHT = 5e-7
GRID = time_grid(None)
BATCH = 4000                 # a single slab, not ordered, on every dataset here


def slab_bound(Nn):
    """An upper bound on the walkers of one slab over Nn nodes (slab_walkers without the record sizes)."""
    return 3 * 2 ** 29 // (8 * Nn + 16)


def same(a, b):
    """Bitwise equality, -inf == -inf and NaN == NaN."""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and bool(((a == b) | (np.isnan(a) & np.isnan(b))).all())


def unlog(theta):
    p = np.array(theta, dtype=np.float64)
    p[..., 2:] = 10.0 ** p[..., 2:]
    return p


def prior_uniform(rng, W, pad=0.0):
    return rng.uniform(O.SCRIPT_LOWER - pad, O.SCRIPT_UPPER + pad, size=(W, 6))


def ball(rng, W, sigma, name="Sloped"):
    return np.clip(O.SYNTH_TRUTHS_LOG[name] + sigma * rng.randn(W, 6), O.SCRIPT_LOWER, O.SCRIPT_UPPER)


def host_batched(lk, theta, size=BATCH):
    """lnp, status, n_rhs of theta evaluated through the host call in batches of `size`."""
    parts = [lk.lnprob(theta[i:i + size], return_info=True) for i in range(0, len(theta), size)]
    return tuple(np.concatenate([p[k] for p in parts]) for k in range(3))


def assert_same_results(got, want):
    for g, w in zip(got, want):
        assert same(g, w)


# ---- datasets ----------------------------------------------------------------------------------------------
# Each builder returns data times on the 10 001-node grid of the synthetic datasets; the CPU test below checks that
# the node program puts each on the side of its boundary that its name claims.
def _inside(i, frac=0.5):
    """A time strictly inside grid interval [i, i + 1]."""
    return GRID[i] + frac * (GRID[i + 1] - GRID[i])


def x_off_node_64():
    """32 off-node data in non-adjacent intervals: 64 nodes, the largest dataset of the thread-per-walker reduce."""
    return np.array([_inside(100 + 300 * k) for k in range(32)])


def x_off_node_65():
    """The 64-node dataset plus one datum on a node of its own: 65 nodes, the smallest of the warp-per-walker reduce."""
    return np.append(x_off_node_64(), GRID[50])


def _x_rows(D):
    # D data over 24 non-adjacent intervals: 48 nodes
    per = (D + 23) // 24
    return np.array([_inside(200 + 400 * (k % 24), (k // 24 + 1) / (per + 1)) for k in range(D)])


def x_rows_staged():
    """48 nodes, D = 160: the reduce's shared-memory need Nn + 4D + ceil(D/2) is 768, exactly its budget."""
    return _x_rows(160)


def x_rows_unstaged():
    """48 nodes, D = 161: need 773, one datum over the budget, so the thread-per-walker reduce reads global memory."""
    return _x_rows(161)


def x_nodes_512():
    """512 on-node data: the advance kernel stages all 512 node times in shared memory."""
    return GRID[5 + 19 * np.arange(512)]


def x_nodes_513():
    """513 on-node data: one node too many to stage."""
    return GRID[5 + 19 * np.arange(513)]


def x_interp_edges():
    """Interpolation edges in one unsorted dataset: the first grid time, a duplicated node, a node and the next
    double above it, a duplicated off-node time and a time strictly inside the last interval (8 nodes)."""
    x = np.array([GRID[0], GRID[300], GRID[300], GRID[2000], np.nextafter(GRID[2000], np.inf), _inside(5000, 0.3),
                  _inside(5000, 0.3), _inside(9999, 0.5)])
    return x[np.random.RandomState(8).permutation(x.size)]


def x_wide():
    """Data on all 10 001 grid nodes."""
    return GRID.copy()


def need_of(Nn, D):
    return Nn + 4 * D + (D + 1) // 2


# name -> (builder, node count, reduce's shared-memory need or None)
BOUNDARY_DATASETS = {
    "off_node_64": (x_off_node_64, 64, None),
    "off_node_65": (x_off_node_65, 65, None),
    "rows_staged": (x_rows_staged, 48, 768),
    "rows_unstaged": (x_rows_unstaged, 48, 773),
    "nodes_512": (x_nodes_512, 512, None),
    "nodes_513": (x_nodes_513, 513, None),
    "interp_edges": (x_interp_edges, 8, None),
    "wide": (x_wide, 10001, None),
}


def node_count(hostsim, x):
    D = x.size
    ones = np.ones(D)
    nn = C.c_int(0)
    ngi = np.zeros(2 * D + 2, np.int32); lo = np.zeros(D, np.int32); dx = np.zeros(D); Dx = np.zeros(D)
    order = np.zeros(D, np.int32)
    assert hostsim.hs_node_program(A.ptr(GRID), GRID.size, A.ptr(x), A.ptr(ones), A.ptr(ones), D, C.byref(nn), A.ptr(ngi),
                                   A.ptr(lo), A.ptr(dx), A.ptr(Dx), A.ptr(order)) == 0
    return nn.value


@pytest.mark.parametrize("name", sorted(BOUNDARY_DATASETS))
def test_boundary_datasets_sit_on_their_boundaries(hostsim, name):
    build, want_nodes, want_need = BOUNDARY_DATASETS[name]
    x = build()
    Nn = node_count(hostsim, x)
    assert Nn == want_nodes
    if want_need is not None:
        assert need_of(Nn, x.size) == want_need
    if name == "wide":
        assert slab_bound(Nn) == 20126


def sloped_curve():
    return O.model(O.SYNTH_TRUTHS["Sloped"], O.script_spec())


def data_for(x, seed, noise=0.1, err=0.2):
    """y from the script model at the Sloped truth with seeded noise, yerr = err * y."""
    y = np.interp(x, GRID, sloped_curve()[1])
    y = y * (1.0 + noise * np.random.RandomState(seed).randn(x.size))
    return y, err * y


def script_handle(x, y, yerr):
    return Likelihood(A.script_model_spec(), GRID, x, y, yerr, O.SCRIPT_LOWER, O.SCRIPT_UPPER)


@pytest.fixture(scope="module")
def wide(built):
    """The wide dataset: y = the Sloped truth's model with 5 % noise on every grid node, yerr = 0.1 y."""
    x = x_wide()
    y, yerr = data_for(x, 5, noise=0.05, err=0.1)
    return x, y, yerr


def sloped50(golden):
    g = golden["lnprob_script"]
    return script_handle(g["Sloped_x"], g["Sloped_y"], g["Sloped_yerr"])


# ---- 1. the rows-form node buffer after a larger launch --------------------------------------------------
@pytest.mark.gpu
def test_rows_launch_after_a_larger_coarse_curves_launch(built, golden):
    """A curves call of 20 000 walkers at a coarse node stride (2 nodes) grows a lane's records past its node buffer;
    a thread-per-walker launch of fewer walkers on the 50-point dataset must still lay its node values out within the
    buffer it grew.  Host form (curves, lnprob, model_at_data share lane 0) and device form (one torch stream)."""
    import torch
    rng = np.random.RandomState(101)
    pars_c = unlog(prior_uniform(rng, 20000))
    th4, th9 = prior_uniform(rng, 4000, 0.02), prior_uniform(rng, 9000, 0.02)
    pars4 = unlog(prior_uniform(rng, 4000))
    fresh = sloped50(golden)
    want4, want9 = fresh.lnprob(th4, return_info=True), fresh.lnprob(th9, return_info=True)
    want_m = fresh.model_at_data(pars4, return_status=True)
    fresh.close()

    lk = sloped50(golden)
    assert lk.curve_nodes(10000) == 2
    k0 = lk.kernels_launched()
    lk.curves(pars_c, node_stride=10000)
    assert lk.kernels_launched() - k0 == 6                             # one slab, ordered
    k0 = lk.kernels_launched()
    assert_same_results(lk.lnprob(th4, return_info=True), want4)
    assert lk.kernels_launched() - k0 == 4                             # rows, not ordered
    k0 = lk.kernels_launched()
    assert_same_results(lk.lnprob(th9, return_info=True), want9)
    assert lk.kernels_launched() - k0 == 6                             # rows, ordered
    assert_same_results(lk.model_at_data(pars4, return_status=True), want_m)

    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d_pars = torch.from_numpy(pars_c).cuda()
        d_out = torch.empty((20000, 3, 2), dtype=torch.float64, device="cuda")
        lk.curves_device(d_pars.data_ptr(), 20000, 6, 10000, d_out.data_ptr(), stream=s.cuda_stream)
        for th, want, kernels in ((th4, want4, 4), (th9, want9, 6)):
            W = th.shape[0]
            d_th = torch.from_numpy(th).cuda()
            d_lnp = torch.empty(W, dtype=torch.float64, device="cuda")
            d_st, d_nr = (torch.empty(W, dtype=torch.int32, device="cuda") for _ in range(2))
            k0 = lk.kernels_launched()
            lk.lnprob_device(d_th.data_ptr(), W, 6, d_lnp.data_ptr(), d_st.data_ptr(), d_nr.data_ptr(), stream=s.cuda_stream)
            assert lk.kernels_launched() - k0 == kernels
            s.synchronize()
            assert_same_results((d_lnp.cpu().numpy(), d_st.cpu().numpy(), d_nr.cpu().numpy()), want)
    torch.cuda.synchronize()
    lk.close()


# ---- 2./3. several slabs -------------------------------------------------------------------------------------
def _device_lnprob(lk, d_theta, W, stream=0):
    import torch
    d_lnp = torch.empty(W, dtype=torch.float64, device="cuda")
    d_st, d_nr = (torch.empty(W, dtype=torch.int32, device="cuda") for _ in range(2))
    lk.lnprob_device(d_theta.data_ptr(), W, 6, d_lnp.data_ptr(), d_st.data_ptr(), d_nr.data_ptr(), stream=stream)
    return d_lnp, d_st, d_nr


@pytest.mark.gpu
def test_multi_slab_lnprob_on_the_wide_dataset(built, wide):
    """45 000 walkers on 10 001 data nodes run as 3 slabs: a ball, a prior-uniform spread and prior rejects, shuffled,
    equal the same walkers in single-slab batches -- through the device call and the host call."""
    import torch
    rng = np.random.RandomState(202)
    theta = np.concatenate([ball(rng, 15000, 1e-2), prior_uniform(rng, 27000), prior_uniform(rng, 3000)])
    rows, cols = np.arange(42000, 45000), rng.randint(0, 6, 3000)
    theta[rows, cols] = np.where(rng.rand(3000) < 0.5, O.SCRIPT_LOWER[cols] - 1e-9, O.SCRIPT_UPPER[cols] + 1e-9)
    theta = theta[rng.permutation(theta.shape[0])]
    W = theta.shape[0]
    assert W > 2 * slab_bound(10001)
    lk = script_handle(*wide)
    d_theta = torch.from_numpy(theta).cuda()
    k0 = lk.kernels_launched()
    big = _device_lnprob(lk, d_theta, W)
    assert lk.kernels_launched() - k0 >= 3 * 4
    parts = []
    for i in range(0, W, BATCH):
        n = min(BATCH, W - i)
        k0 = lk.kernels_launched()
        parts.append(_device_lnprob(lk, d_theta[i:i + n], n))
        assert lk.kernels_launched() - k0 == 4
    torch.cuda.synchronize()
    got = tuple(t.cpu().numpy() for t in big)
    want = tuple(torch.cat([p[k] for p in parts]).cpu().numpy() for k in range(3))
    assert_same_results(got, want)
    assert_same_results(lk.lnprob(theta, return_info=True), want)
    st = want[1]
    assert (st & A.WALKER_PRIOR_REJECT).astype(bool).sum() >= 3000 and np.isfinite(want[0]).sum() > 10000
    lk.close()


@pytest.mark.gpu
def test_multi_slab_curves_on_every_node(built):
    """curves_device of 2 slab bounds + 17 walkers at node stride 1 (at least 3 slabs) equals the same walkers in
    launches of 4000.  Needs about 12 GB of device memory: the full output alone is 9.7 GB."""
    import torch
    rng = np.random.RandomState(303)
    W = 2 * slab_bound(10001) + 17
    pars = np.column_stack([rng.uniform(0.5, 5, W), rng.uniform(1, 8, W), 10 ** rng.uniform(-5, -2.5, W),
                            10 ** rng.uniform(1.8, 3.2, W), 10 ** rng.uniform(-1.5, 1.5, W), 10 ** rng.uniform(-0.5, 2, W)])
    lk = Likelihood(A.script_model_spec(unlog=False), GRID)
    G = lk.curve_nodes(1)
    assert G == 10001
    d_pars = torch.from_numpy(pars).cuda()
    out = torch.empty((W, 3, G), dtype=torch.float64, device="cuda")
    st = torch.empty(W, dtype=torch.int32, device="cuda")
    k0 = lk.kernels_launched()
    lk.curves_device(d_pars.data_ptr(), W, 6, 1, out.data_ptr(), 0, st.data_ptr())
    assert lk.kernels_launched() - k0 >= 3 * 4
    part = torch.empty((BATCH, 3, G), dtype=torch.float64, device="cuda")
    pst = torch.empty(BATCH, dtype=torch.int32, device="cuda")
    for i in range(0, W, BATCH):
        n = min(BATCH, W - i)
        lk.curves_device(d_pars[i:].data_ptr(), n, 6, 1, part.data_ptr(), 0, pst.data_ptr())
        a, b = out[i:i + n], part[:n]
        assert bool(((a == b) | (a.isnan() & b.isnan())).all()), i
        assert torch.equal(st[i:i + n], pst[:n])
    torch.cuda.synchronize()
    ok = (st == 0).sum().item()
    assert ok > W // 2
    del out, part
    torch.cuda.empty_cache()
    lk.close()


# ---- 4./5. moves across slabs -----------------------------------------------------------------------------------
@pytest.mark.gpu
def test_ensemble_half_steps_across_slabs(built, wide):
    """A 65 536-walker ensemble on the wide dataset moves 32 768 walkers per half-step: 2 slabs.  Two steps equal
    the restatement driven by single-slab host batches, bit for bit; fixed halves equal the explicit-list call."""
    import torch
    from magprop_b200.sampler import DeviceEnsemble
    lk = script_handle(*wide)
    rng = np.random.RandomState(404)
    n = 65536
    p0 = np.concatenate([ball(rng, n // 2, 3e-2), ball(rng, n // 2, 0.3)])[rng.permutation(n)]
    fn = lambda q: host_batched(lk, q)[0]
    ens = DeviceEnsemble.from_likelihood(lk, n, 6, a=2.0, seed=99)
    ens.initialise(p0)
    torch.cuda.synchronize()
    lnp0 = ens.lnp.cpu().numpy()
    assert same(lnp0, fn(p0))
    coords, lnp, acc = p0.copy(), lnp0.copy(), np.zeros(n, np.int32)
    half = n // 2
    assert half > slab_bound(10001)
    k0 = lk.kernels_launched()
    chain, lps = ens.run(2, store=True)
    torch.cuda.synchronize()
    assert lk.kernels_launched() - k0 >= 4 * 8
    for it in range(2):
        order = R.ensemble_order(n, 99, it)
        for split in (0, 1):
            R.half_step(coords, lnp, order[split * half:(split + 1) * half], order[(1 - split) * half:(2 - split) * half],
                        2.0, 99, 2 * it + split, fn, acc)
        assert np.array_equal(chain[it].cpu().numpy(), coords)
        assert same(lps[it].cpu().numpy(), lnp)
    assert np.array_equal(ens.accepted.cpu().numpy(), acc)
    assert 0 < acc.sum() < 2 * n
    fixed = DeviceEnsemble.from_likelihood(lk, n, 6, a=2.0, seed=99, randomize_split=False)
    fixed.initialise(p0)
    fixed.run(1)
    c2 = torch.from_numpy(p0).cuda(); l2 = torch.from_numpy(lnp0).cuda()
    idx = torch.arange(n, dtype=torch.int32, device="cuda")
    for split in (0, 1):
        act, cmp_ = (idx[:half], idx[half:]) if split == 0 else (idx[half:], idx[:half])
        lk.stretch_half_step(c2.data_ptr(), l2.data_ptr(), n, 6, act.data_ptr(), half, cmp_.data_ptr(), half, 2.0, 99, split)
    torch.cuda.synchronize()
    assert torch.equal(fixed.coords, c2) and torch.equal(fixed.lnp, l2)
    lk.close()


@pytest.mark.gpu
def test_tempered_half_steps_across_slabs(built, wide):
    """T = 3 x n = 16 384 on the wide dataset: 24 576 movers per half-step, so the slab boundary falls inside the
    hottest temperature.  Two steps with swaps equal the restatement driven by single-slab host batches."""
    import torch
    from magprop_b200.sampler import TemperedEnsemble, geometric_betas
    lk = script_handle(*wide)
    T, n = 3, 16384
    assert slab_bound(10001) < T * n // 2
    betas = geometric_betas(T, 1e-2)
    rng = np.random.RandomState(505)
    p0 = np.stack([ball(rng, n, 2e-2), ball(rng, n, 0.2), prior_uniform(rng, n)])
    fn = lambda q: host_batched(lk, q)[0]
    ens = TemperedEnsemble.from_likelihood(lk, n, 6, betas, seed=21)
    ens.initialise(p0)
    torch.cuda.synchronize()
    coords = p0.reshape(T * n, 6).copy()
    lnp = ens.lnp.cpu().numpy().copy()
    assert same(lnp, fn(coords))
    acc, swaps = np.zeros(T * n, np.int32), np.zeros(T - 1, np.int32)
    for step in range(2):
        for split in (0, 1):
            k0 = lk.kernels_launched()
            ens.backend.tempered_half_step(ens, step, split)
            assert lk.kernels_launched() - k0 >= 8
            TR.half_step(coords, lnp, betas, n, split, 2.0, 21, step, fn, acc)
            assert np.array_equal(ens.coords.cpu().numpy(), coords) and same(ens.lnp.cpu().numpy(), lnp)
        ens.backend.tempered_swap(ens, step)
        TR.swap(coords, lnp, betas, n, 21, step, swaps)
        ens.step += 1
        torch.cuda.synchronize()
        assert np.array_equal(ens.coords.cpu().numpy(), coords) and same(ens.lnp.cpu().numpy(), lnp)
    assert np.array_equal(ens.accepted.cpu().numpy(), acc) and np.array_equal(ens.swap_accepted.cpu().numpy(), swaps)
    assert 0 < acc.sum() < T * n * 2
    lk.close()


# ---- 6./7. integrator builds and work-list ordering ----------------------------------------------------------------
@pytest.mark.gpu
def test_integrator_block_sizes_and_stiff_builds_agree(built, golden):
    """262 144 prior-uniform walkers in one launch (64-thread blocks, the 16-warp implicit build) equal the same
    walkers in launches of sm_count * 256 - 1 (32-thread blocks) and of 100 000 (64-thread blocks, the 12-warp
    implicit build)."""
    import torch
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    rng = np.random.RandomState(606)
    theta = prior_uniform(rng, 262144, 0.02)
    lk = sloped50(golden)
    big = lk.lnprob(theta, return_info=True)
    assert lk.last_stiff_count() > 10000
    for size in (sm * 256 - 1, 100000):
        assert_same_results(host_batched(lk, theta, size), big)
    assert 0 < (big[1] & A.WALKER_PRIOR_REJECT).astype(bool).sum() < theta.shape[0]
    lk.close()


@pytest.mark.gpu
def test_ordered_and_unordered_launches_agree(built, golden):
    """The same 10 000 walkers after a tight ball (the next launch takes its walkers as they come) and after a
    prior-uniform spread (the next launch orders its work list) equal each other and launches below the ordering
    threshold."""
    rng = np.random.RandomState(707)
    X = ball(rng, 10000, 0.2)
    tight, spread = ball(rng, 10000, 1e-4), prior_uniform(rng, 10000)
    lk = sloped50(golden)
    want = host_batched(lk, X, 5000)
    lk.lnprob(tight)
    k0 = lk.kernels_launched()
    assert_same_results(lk.lnprob(X, return_info=True), want)
    assert lk.kernels_launched() - k0 == 4
    lk.lnprob(spread)
    k0 = lk.kernels_launched()
    assert_same_results(lk.lnprob(X, return_info=True), want)
    assert lk.kernels_launched() - k0 == 6
    assert np.isfinite(want[0]).sum() > 9000
    lk.close()


# ---- 8. a handle without data ----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_handle_without_data_is_the_prior(built):
    lk = Likelihood(A.script_model_spec(), GRID, lower=O.SCRIPT_LOWER, upper=O.SCRIPT_UPPER)
    rng = np.random.RandomState(808)
    for W in (1, 2049, 9000):
        theta = prior_uniform(rng, W, 0.5)
        theta[0] = O.SCRIPT_UPPER                                          # inclusive bounds
        k0 = lk.kernels_launched()
        lnp, st, nr = lk.lnprob(theta, return_info=True)
        assert lk.kernels_launched() - k0 == 2
        inside = np.all((theta >= O.SCRIPT_LOWER) & (theta <= O.SCRIPT_UPPER), axis=1)
        assert (lnp[inside] == 0.0).all() and np.isneginf(lnp[~inside]).all()
        assert ((st & A.WALKER_PRIOR_REJECT) != 0).tolist() == (~inside).tolist()
        assert (nr[~inside] == 0).all()
        if W > 1:
            assert 0 < inside.sum() < W
    lk.close()


@pytest.mark.gpu
def test_data_only_at_the_first_grid_time(built):
    """A dataset that ends where the integration starts needs no step: the initial state is the whole solution, and
    lnprob is finite and equal to the converged oracle's, in the warp-per-walker and the thread-per-walker reduce."""
    lk = Likelihood(A.script_model_spec(), GRID, [GRID[0], GRID[0]], [2.0, 1.5], [0.5, 0.3], O.SCRIPT_LOWER, O.SCRIPT_UPPER)
    theta = np.concatenate([ball(np.random.RandomState(818), 8, 0.1), prior_uniform(np.random.RandomState(819), 2992)])
    lnp, st, _ = lk.lnprob(theta, return_info=True)
    assert (st == 0).all() and np.isfinite(lnp).all()
    assert_same_results(lk.lnprob(theta[:16], return_info=True)[:2], (lnp[:16], st[:16]))
    for p, got in zip(unlog(theta[:8]), lnp[:8]):
        L0 = O.model(p, O.script_spec(), tight=True)[1][0]
        assert relerr(got, -0.5 * (((2.0 - L0) / 0.5) ** 2 + ((1.5 - L0) / 0.3) ** 2)) < TOL_TIGHT
    lk.close()


# ---- against the converged oracle at the dataset boundaries --------------------------------------------------------------
@pytest.fixture(scope="module")
def oracle_walkers():
    """16 walkers -- 12 around the Sloped truth, 4 prior-uniform -- and one converged oracle curve per walker (Ltot/1e50
    on every grid node, or None where the oracle's integration fails)."""
    rng = np.random.RandomState(909)
    theta = np.concatenate([ball(rng, 12, 0.1), prior_uniform(rng, 4)])
    curves = []
    for p in unlog(theta):
        c = O.model(p, O.script_spec(), tight=True)
        curves.append(None if isinstance(c, str) else c[1])
    return theta, curves


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(set(BOUNDARY_DATASETS) - {"wide"}))
def test_boundary_datasets_match_the_converged_oracle(built, oracle_walkers, name):
    theta, curves = oracle_walkers
    build, Nn, _ = BOUNDARY_DATASETS[name]
    x = build()
    y, yerr = data_for(x, 11)
    lk = script_handle(x, y, yerr)
    lnp, st, nr = lk.lnprob(theta, return_info=True)
    mod, mst = lk.model_at_data(unlog(theta), return_status=True)
    ok = np.array([c is not None for c in curves]) & ((st & A.WALKER_INTEGRATOR_FAIL) == 0)
    assert ok.sum() >= 12
    want_mod = np.array([np.interp(x, GRID, c) if c is not None else np.full(x.size, np.nan) for c in curves])
    want_lnp = -0.5 * np.sum(((y - want_mod) / yerr) ** 2, axis=1)
    assert relerr(lnp[ok], want_lnp[ok]).max() < TOL_TIGHT
    assert relerr(mod[ok], want_mod[ok]).max() < TOL_TIGHT
    assert not np.isnan(lnp).any()
    # the same walkers in a 2000-walker launch (warp per walker, summed in datum order when Nn <= 64) and a
    # 3000-walker launch (thread per walker when Nn <= 64): the same bits
    for W in (2000, 3000):
        idx = np.arange(W) % theta.shape[0]
        assert_same_results(lk.lnprob(theta[idx], return_info=True), (lnp[idx], st[idx], nr[idx]))
        assert_same_results(lk.model_at_data(unlog(theta[idx]), return_status=True), (mod[idx], mst[idx]))
    lk.close()
