"""Host-side owner of a CUDA likelihood handle (thin layer over the C ABI).

``Likelihood`` is what the drop-in modules (``magprop_b200.magnetar`` and
``magprop_b200.synthetic``) and the samplers call.  NumPy in, NumPy out for the
host-pointer entry points; raw device pointers (``torch.Tensor.data_ptr()``)
for the ``*_device`` ones.  No CPU fallback exists: every method ends in a CUDA
launch or raises ``MagpropCudaError``.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi as A

N_GRID = 10001


def time_grid(GRBtype=None) -> np.ndarray:
    """The reference's model grids (funcs.py:19, magnetar/funcs.py:132-141)."""
    if GRBtype is None or GRBtype == "L":
        return np.logspace(0.0, 6.0, num=N_GRID, base=10.0)
    if GRBtype == "S":
        return np.logspace(-3.0, 6.0, num=N_GRID, base=10.0)
    raise ValueError("Please provide a valid value for GRBtype.\nOptions are: L, S, or None.")


def _f64(a, ndim=None):
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
    if ndim is not None and a.ndim != ndim:
        raise ValueError(f"expected a {ndim}-D array, got shape {a.shape}")
    return a


class Likelihood:
    """One (model spec, prior, grid, dataset) bound to one GPU."""

    def __init__(self, spec: A.ModelSpec, grid, x=None, y=None, yerr=None, lower=None, upper=None,
                 device: int = 0):
        self._lib = A.load()
        self.spec = spec
        self.grid = _f64(grid, 1)
        self.device = int(device)
        self._h = C.c_void_p()
        self._prior = A.prior_spec(lower, upper)
        if x is None:
            self.D = 0
            xs = ys = es = None
            px = py = pe = None
        else:
            xs, ys, es = _f64(x, 1), _f64(y, 1), _f64(yerr, 1)
            if not (xs.shape == ys.shape == es.shape):
                raise ValueError("x, y, yerr must have the same length")
            self.D = xs.size
            px, py, pe = A.ptr(xs), A.ptr(ys), A.ptr(es)
        A.check(self._lib.mp_create(C.byref(spec), C.byref(self._prior), A.ptr(self.grid), self.grid.size,
                                    px, py, pe, self.D, self.device, C.byref(self._h)))

    # -- lifetime -------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.mp_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_prior(self, lower, upper):
        self._prior = A.prior_spec(lower, upper)
        A.check(self._lib.mp_set_prior(self._h, C.byref(self._prior)))

    # -- hot path ---------------------------------------------------------------
    def lnprob(self, theta, return_info: bool = False):
        """lnprob for every row of theta[W, ndim] in one launch (host arrays)."""
        theta = _f64(theta)
        single = theta.ndim == 1
        theta = np.atleast_2d(theta)
        W, ndim = theta.shape
        lnp = np.empty(W, dtype=np.float64)
        status = np.empty(W, dtype=np.int32)
        nrhs = np.empty(W, dtype=np.int32)
        A.check(self._lib.mp_lnprob_batch(self._h, A.ptr(theta), W, ndim, A.ptr(lnp), A.ptr(status), A.ptr(nrhs)))
        if return_info:
            return lnp, status, nrhs
        return float(lnp[0]) if single else lnp

    def lnprob_async(self, theta: np.ndarray, lnp: np.ndarray, status=None, nrhs=None):
        """Queue lnprob of theta[W, ndim] into the caller's (ideally pinned) float64 buffer ``lnp`` and return
        at once; the result is valid after ``synchronize()``.  Several handles can be in flight together."""
        for name, arr, dt in (("theta", theta, np.float64), ("lnp", lnp, np.float64), ("status", status, np.int32),
                              ("nrhs", nrhs, np.int32)):
            # the pointers go to C as they are: anything but a C-contiguous array of the right type would be read as garbage
            if arr is not None and not (isinstance(arr, np.ndarray) and arr.dtype == dt and arr.flags.c_contiguous):
                raise ValueError(f"lnprob_async: {name} must be a C-contiguous {np.dtype(dt).name} ndarray")
        if theta.ndim != 2 or lnp.shape != (theta.shape[0],):
            raise ValueError("lnprob_async: theta must be [W, ndim] and lnp [W]")
        W, ndim = theta.shape
        A.check(self._lib.mp_lnprob_batch_async(self._h, A.ptr(theta), W, ndim, A.ptr(lnp),
                                                A.ptr(status) if status is not None else None,
                                                A.ptr(nrhs) if nrhs is not None else None))

    def synchronize(self):
        A.check(self._lib.mp_synchronize(self._h))

    def lnprob_device(self, d_theta: int, W: int, ndim: int, d_lnp: int, d_status: int = 0, d_nrhs: int = 0,
                      stream: int = 0):
        """Enqueue lnprob on device buffers (raw pointers); does not synchronise."""
        A.check(self._lib.mp_lnprob_batch_device(self._h, d_theta, W, ndim, d_lnp, d_status or None,
                                                 d_nrhs or None, stream or None))

    def model_at_data(self, pars, return_status=False):
        pars = np.atleast_2d(_f64(pars))
        W, ndim = pars.shape
        out = np.empty((W, self.D), dtype=np.float64)
        status = np.empty(W, dtype=np.int32)
        A.check(self._lib.mp_model_at_data(self._h, A.ptr(pars), W, ndim, A.ptr(out), A.ptr(status)))
        return (out, status) if return_status else out

    def curve_nodes(self, node_stride=1) -> int:
        return int(self._lib.mp_curve_nodes(self._h, node_stride))

    def curves(self, pars, node_stride=1, with_state=False):
        """(Ltot, Lprop, Ldip)/1e50 on every node_stride-th grid node: [W,3,Gs]."""
        pars = np.atleast_2d(_f64(pars))
        W, ndim = pars.shape
        Gs = self.curve_nodes(node_stride)
        out = np.empty((W, 3, Gs), dtype=np.float64)
        state = np.empty((W, 2, Gs), dtype=np.float64) if with_state else None
        status = np.empty(W, dtype=np.int32)
        A.check(self._lib.mp_model_curves(self._h, A.ptr(pars), W, ndim, node_stride, A.ptr(out),
                                          A.ptr(state) if with_state else None, A.ptr(status)))
        return (out, state, status) if with_state else (out, status)

    def curves_device(self, d_pars, W, ndim, node_stride, d_out, d_state=0, d_status=0, stream=0):
        A.check(self._lib.mp_model_curves_device(self._h, d_pars, W, ndim, node_stride, d_out, d_state or None,
                                                 d_status or None, stream or None))

    def node_times(self, node_stride=1) -> np.ndarray:
        idx = list(range(0, self.grid.size, max(1, node_stride)))
        if idx[-1] != self.grid.size - 1:
            idx.append(self.grid.size - 1)
        return self.grid[idx]

    def last_stiff_count(self) -> int:
        """Walkers of the last launch that were handed to the implicit integrator (synchronises)."""
        n = C.c_int32(0)
        A.check(self._lib.mp_last_stiff_count(self._h, C.byref(n)))
        return n.value

    def kernels_launched(self) -> int:
        """Kernels of the evaluation pipeline launched through this handle so far."""
        return int(self._lib.mp_kernels_launched(self._h))

    def stretch_half_step(self, d_coords, d_lnp, nwalkers, ndim, d_active, n_active, d_complement,
                          n_complement, a, seed, step, d_accepted=0, d_nrhs=0, stream=0):
        A.check(self._lib.mp_stretch_half_step(self._h, d_coords, d_lnp, nwalkers, ndim, d_active, n_active,
                                               d_complement, n_complement, float(a), int(seed), int(step),
                                               d_accepted or None, d_nrhs or None, stream or None))


def rhs_batch(spec: A.ModelSpec, y, t, pars, knobs, device=0) -> np.ndarray:
    """Coupled RHS (dMdisc/dt, domega/dt) on the device for states y[W,2]."""
    lib = A.load()
    y = np.atleast_2d(_f64(y)); t = np.atleast_1d(_f64(t)); pars = np.atleast_2d(_f64(pars))
    knobs = _f64(knobs, 1)
    W = y.shape[0]
    out = np.empty((W, 2), dtype=np.float64)
    A.check(lib.mp_rhs_batch(C.byref(spec), A.ptr(y), A.ptr(t), A.ptr(pars), A.ptr(knobs), W, A.ptr(out), device))
    return out


def fp64_peak_tflops(device=0) -> float:
    lib = A.load()
    v = C.c_double(0.0)
    A.check(lib.mp_fp64_peak_tflops(device, C.byref(v)))
    return v.value


def chain_moments(d_chain: int, n: int, ndim: int, device=0, stream=0):
    """Column means and covariance matrix of a device-resident chain [n, ndim] (raw pointer)."""
    lib = A.load()
    mean = np.empty(ndim); cov = np.empty((ndim, ndim))
    A.check(lib.mp_chain_moments(d_chain, n, ndim, A.ptr(mean), A.ptr(cov), device, stream or None))
    return mean, cov


def smc_weights(d_lnp: int, n: int, dbeta: float, d_w: int = 0, device=0, stream=0):
    """(m, S1, S2) of the incremental weights w_i = exp(dbeta (lnp_i - m)) of a device array lnp [n] (raw pointer),
    m its largest finite entry; ``d_w`` (raw pointer, or 0) receives the weights.  Synchronises ``stream``."""
    lib = A.load()
    out = np.empty(3)
    A.check(lib.mp_smc_weights(d_lnp, n, float(dbeta), d_w or None, A.ptr(out), device, stream or None))
    return float(out[0]), float(out[1]), float(out[2])


def smc_resample(d_w: int, n: int, ndim: int, seed: int, stage: int, d_coords_in: int, d_lnp_in: int, d_coords_out: int,
                 d_lnp_out: int, d_ancestors: int = 0, device=0, stream=0):
    """Systematic resampling of n particles (raw device pointers) by the weights d_w into the out buffers, with the
    stage's uniform from (seed, stage); ``d_ancestors`` (int64 [n], or 0) receives the ancestor indices.  Enqueued on
    ``stream``, not synchronised."""
    lib = A.load()
    A.check(lib.mp_smc_resample(d_w, n, ndim, int(seed), int(stage), d_coords_in, d_lnp_in, d_coords_out, d_lnp_out,
                                d_ancestors or None, device, stream or None))


def chain_order_statistics(d_chain: int, n: int, ndim: int, col: int, ranks, device=0, stream=0) -> np.ndarray:
    """Exact order statistics (0-based ranks) of one column of a device-resident chain [n, ndim]."""
    lib = A.load()
    ranks = np.ascontiguousarray(ranks, dtype=np.int64)
    out = np.empty(ranks.size)
    A.check(lib.mp_chain_order_statistics(d_chain, n, ndim, col, A.ptr(ranks), ranks.size, A.ptr(out), device, stream or None))
    return out


def chain_autocorr(d_chain: int, n_steps: int, nwalkers: int, ndim: int, first=0, thin=1, lag_begin=0, lag_end=None,
                   device=0, stream=0) -> np.ndarray:
    """Walker-averaged normalised autocorrelation function [ndim, lag_end - lag_begin] of a device-resident chain
    [n_steps, nwalkers, ndim] (raw pointer), over rows first, first + thin, ...; ``lag_end=None``: every lag of the
    retained rows.  The mean over walkers of emcee's ``function_1d`` (``synth_mcmc.function_1d``)."""
    lib = A.load()
    n = (int(n_steps) - int(first) + int(thin) - 1) // int(thin) if thin >= 1 else 0
    lag_end = n if lag_end is None else int(lag_end)
    out = np.empty((max(0, int(ndim)), max(0, lag_end - int(lag_begin))))
    A.check(lib.mp_chain_autocorr(d_chain, n_steps, nwalkers, ndim, first, thin, lag_begin, lag_end, A.ptr(out), device,
                                  stream or None))
    return out


def gompertz_curves(pars, n_steps=10 ** 6, stride=1, alpha=0.1, cs7=1.0, k=0.9, omass=1.4, dipeff=1.0, propeff=1.0, device=0):
    """The comparison model of the reference's figure 5 (``code/figure_5.py:222-363``) on the device:
    returns ``(t, curves)`` with ``curves[W, 3, n_out]`` = Ltot, Lprop, Ldip (/1e50) at ``t = 1 + i*stride`` s."""
    lib = A.load()
    pars = np.atleast_2d(_f64(pars))
    if pars.shape[1] != 6:
        raise ValueError("pars must be [W, 6]")
    knobs = np.array([alpha, cs7, k, omass, dipeff, propeff], dtype=np.float64)
    n_out = (int(n_steps) + int(stride) - 1) // int(stride)
    out = np.empty((pars.shape[0], 3, n_out), dtype=np.float64)
    A.check(lib.mp_gompertz_curves(A.ptr(pars), pars.shape[0], A.ptr(knobs), int(n_steps), int(stride), A.ptr(out), device))
    return 1.0 + np.arange(n_out, dtype=np.float64) * stride, out
