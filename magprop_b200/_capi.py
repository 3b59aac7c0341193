"""ctypes binding of include/magprop_b200.h (the C ABI of the CUDA library).

There is deliberately no fallback: if ``libmagprop_b200.so`` is missing or the
box has no CUDA device, importing is fine but the first compute call raises
``MagpropCudaError`` -- the product has no CPU path.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

MP_MAX_NDIM = 9
MP_ABI_VERSION = 2
MP_MAX_PEERS = 15
MP_MAX_TEMPS = 256
MP_MOVE_STRETCH, MP_MOVE_DE, MP_MOVE_DE_SNOOKER = range(3)
MP_MOVE_KDE = 4                 # (kind 3 is not assigned)
MP_MAX_MOVES = 8
MP_KDE_MAX_CENTRES = 4096

MP_OK, MP_ERR_BAD_ARG, MP_ERR_DATA_RANGE, MP_ERR_CUDA, MP_ERR_BAD_GRID, MP_ERR_NO_DATA = range(6)

WALKER_OK = 0
WALKER_PRIOR_REJECT = 1
WALKER_INTEGRATOR_FAIL = 2
WALKER_NONFINITE_STATE = 4
WALKER_NONFINITE_LNLIKE = 8


class ModelSpec(C.Structure):
    """mp_model_spec (include/magprop_b200.h)."""
    _fields_ = [
        ("inertia_factor", C.c_double), ("mdot_factor", C.c_double),
        ("rhs_n", C.c_double), ("rhs_alpha", C.c_double), ("rhs_cs7", C.c_double), ("rhs_k", C.c_double),
        ("lum_n", C.c_double), ("lum_alpha", C.c_double), ("lum_cs7", C.c_double), ("lum_k", C.c_double),
        ("dipeff", C.c_double), ("propeff", C.c_double), ("f_beam", C.c_double),
        ("breakup_rhs", C.c_double), ("breakup_lum", C.c_double),
        ("lprop_binding_term", C.c_int32), ("unlog_mask", C.c_int32),
        ("rtol", C.c_double), ("max_steps", C.c_int32), ("dipole_torque", C.c_int32),
    ]


class PriorSpec(C.Structure):
    """mp_prior_spec."""
    _fields_ = [("ndim", C.c_int32), ("enabled", C.c_int32),
                ("lower", C.c_double * MP_MAX_NDIM), ("upper", C.c_double * MP_MAX_NDIM)]


class Ensemble(C.Structure):
    """mp_ensemble (include/magprop_b200.h): a device-resident ensemble and how this rank moves it."""
    _fields_ = [("coords", C.c_void_p), ("lnp", C.c_void_p), ("nwalkers", C.c_int32), ("ndim", C.c_int32),
                ("a", C.c_double), ("seed", C.c_uint64), ("randomize_split", C.c_int32),
                ("rank", C.c_int32), ("world", C.c_int32),
                ("accepted", C.c_void_p), ("status", C.c_void_p), ("n_rhs", C.c_void_p),
                ("n_peers", C.c_int32),
                ("peer_coords", C.c_void_p * MP_MAX_PEERS), ("peer_lnp", C.c_void_p * MP_MAX_PEERS),
                ("synced_step", C.c_uint64),
                ("pack_out", C.c_void_p), ("bad_rows", C.c_void_p), ("bad_count", C.c_void_p),
                ("bad_capacity", C.c_int32)]


class Move(C.Structure):
    """mp_move (include/magprop_b200.h): one entry of a weighted list of ensemble moves."""
    _fields_ = [("kind", C.c_int32), ("pad", C.c_int32), ("weight", C.c_double), ("a", C.c_double),
                ("gamma0", C.c_double), ("sigma", C.c_double), ("gammas", C.c_double)]


def script_model_spec(n=10.0, alpha=0.1, cs7=1.0, k=0.9, dipeff=1.0, propeff=1.0, f_beam=1.0,
                      unlog=True, rtol=0.0, max_steps=0) -> ModelSpec:
    """The model of code/synthetic_datasets/funcs.py:146-236 (kwargs forwarded to the RHS)."""
    return ModelSpec(0.35, 3.0, n, alpha, cs7, k, n, alpha, cs7, k, dipeff, propeff, f_beam,
                     0.27, 0.27, 1, 0b111100 if unlog else 0, rtol, max_steps, 0)


def packaged_model_spec(dipeff=0.05, propeff=0.4, f_beam=1.0, n=1.0, alpha=0.1, cs7=1.0, k=0.9,
                        rtol=0.0, max_steps=0) -> ModelSpec:
    """The model of magnetar/funcs.py:105-220: kwargs reach only the luminosity
    stage (:150-151 does not forward them), and rot_param > 0.0 there (:193)."""
    return ModelSpec(4.0 / 5.0, 1.0, 1.0, 0.1, 1.0, 0.9, n, alpha, cs7, k, dipeff, propeff, f_beam,
                     0.27, 0.0, 0, 0, rtol, max_steps, 0)


def figure_model_spec(n=10.0, alpha=0.1, cs7=1.0, k=0.9, rtol=0.0, max_steps=0, bucciantini=False) -> ModelSpec:
    """The model the paper-figure scripts inline (code/figure_1.py:13,65, figure_4.py:14,114-177):
    I = 4/5 M R^2, (3 Mdisc/tvisc)^(-2/7), break-up test 0.27 in both stages, Lprop with the binding
    term, unit efficiencies, physical (not log) parameters, n swept per figure (1/10/50).
    ``bucciantini=True``: the RHS uses the dipole torque of Bucciantini et al. (2006) as figure_3.py:105-164 does."""
    return ModelSpec(4.0 / 5.0, 3.0, n, alpha, cs7, k, n, alpha, cs7, k, 1.0, 1.0, 1.0,
                     0.27, 0.27, 1, 0, rtol, max_steps, 1 if bucciantini else 0)


def prior_spec(lower=None, upper=None) -> PriorSpec:
    p = PriorSpec()
    if lower is None:
        p.ndim, p.enabled = 0, 0
        return p
    lower = np.asarray(lower, dtype=np.float64)
    upper = np.asarray(upper, dtype=np.float64)
    if lower.shape != upper.shape or lower.ndim != 1 or not (1 <= lower.size <= MP_MAX_NDIM):
        raise ValueError("prior bounds must be two 1-D arrays of equal length <= 9")
    p.ndim, p.enabled = lower.size, 1
    for i in range(lower.size):
        p.lower[i] = lower[i]
        p.upper[i] = upper[i]
    return p


class MagpropCudaError(RuntimeError):
    pass


_LIB = None
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


def lib_path() -> str:
    if os.environ.get("MAGPROP_B200_LIB"):      # developer override (A/B builds of the same CUDA library)
        return os.environ["MAGPROP_B200_LIB"]
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "libmagprop_b200.so")


def declare(lib):
    """Attach argtypes/restypes for every symbol the header declares."""
    vp = C.c_void_p
    lib.mp_abi_version.restype = C.c_int
    lib.mp_device_count.restype = C.c_int
    lib.mp_last_error.restype = C.c_char_p
    lib.mp_create.argtypes = [C.POINTER(ModelSpec), C.POINTER(PriorSpec), vp, C.c_int32,
                              vp, vp, vp, C.c_int32, C.c_int32, C.POINTER(vp)]
    lib.mp_destroy.argtypes = [vp]
    lib.mp_destroy.restype = None
    lib.mp_set_prior.argtypes = [vp, C.POINTER(PriorSpec)]
    lib.mp_lnprob_batch.argtypes = [vp, vp, C.c_int32, C.c_int32, vp, vp, vp]
    lib.mp_lnprob_batch_async.argtypes = [vp, vp, C.c_int32, C.c_int32, vp, vp, vp]
    lib.mp_synchronize.argtypes = [vp]
    lib.mp_lnprob_batch_device.argtypes = [vp, vp, C.c_int32, C.c_int32, vp, vp, vp, vp]
    lib.mp_model_at_data.argtypes = [vp, vp, C.c_int32, C.c_int32, vp, vp]
    lib.mp_curve_nodes.argtypes = [vp, C.c_int32]
    lib.mp_curve_nodes.restype = C.c_int32
    lib.mp_model_curves.argtypes = [vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp]
    lib.mp_model_curves_device.argtypes = [vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, vp]
    lib.mp_rhs_batch.argtypes = [C.POINTER(ModelSpec), vp, vp, vp, vp, C.c_int32, vp, C.c_int32]
    lib.mp_stretch_half_step.argtypes = [vp, vp, vp, C.c_int32, C.c_int32, vp, C.c_int32, vp, C.c_int32,
                                         C.c_double, C.c_uint64, C.c_uint64, vp, vp, vp]
    lib.mp_ensemble_half_step.argtypes = [vp, C.POINTER(Ensemble), C.c_uint64, C.c_int32, vp]
    lib.mp_ensemble_sync.argtypes = [C.POINTER(Ensemble), C.c_uint64, vp]
    lib.mp_ensemble_unpack.argtypes = [C.POINTER(Ensemble), C.c_uint64, C.c_int32, vp, vp]
    lib.mp_ensemble_order.argtypes = [C.c_int32, C.c_uint64, C.c_uint64, C.c_int32, vp, vp]
    lib.mp_tempered_half_step.argtypes = [vp, C.POINTER(Ensemble), C.c_int32, vp, C.c_uint64, C.c_int32, vp]
    lib.mp_ensemble_moves_half_step.argtypes = [vp, C.POINTER(Ensemble), vp, C.c_int32, C.c_uint64, C.c_int32, vp]
    lib.mp_tempered_moves_half_step.argtypes = [vp, C.POINTER(Ensemble), C.c_int32, vp, vp, C.c_int32, C.c_uint64,
                                                C.c_int32, vp]
    lib.mp_tempered_swap.argtypes = [C.POINTER(Ensemble), C.c_int32, vp, C.c_uint64, vp, vp]
    lib.mp_peer_alloc.argtypes = [C.c_int32, C.c_uint64, C.POINTER(vp), C.c_char_p]
    lib.mp_peer_open.argtypes = [C.c_int32, C.c_char_p, C.POINTER(vp)]
    lib.mp_peer_close.argtypes = [C.c_int32, vp]
    lib.mp_peer_free.argtypes = [C.c_int32, vp]
    lib.mp_peer_barrier.argtypes = [C.c_int32, vp, C.POINTER(vp), C.c_int32, C.c_int32, C.c_uint64, vp, vp]
    lib.mp_chain_moments.argtypes = [vp, C.c_int64, C.c_int32, vp, vp, C.c_int32, vp]
    lib.mp_chain_order_statistics.argtypes = [vp, C.c_int64, C.c_int32, C.c_int32, vp, C.c_int32, vp, C.c_int32, vp]
    lib.mp_chain_autocorr.argtypes = [vp, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                      vp, C.c_int32, vp]
    lib.mp_gompertz_curves.argtypes = [vp, C.c_int32, vp, C.c_int64, C.c_int32, vp, C.c_int32]
    lib.mp_kernels_launched.argtypes = [vp]
    lib.mp_kernels_launched.restype = C.c_int64
    lib.mp_fp64_peak_tflops.argtypes = [C.c_int32, _dp]
    lib.mp_last_stiff_count.argtypes = [vp, _ip]
    lib.mp_smc_weights.argtypes = [vp, C.c_int64, C.c_double, vp, vp, C.c_int32, vp]
    lib.mp_smc_resample.argtypes = [vp, C.c_int64, C.c_int32, C.c_uint64, C.c_uint64, vp, vp, vp, vp, vp, C.c_int32, vp]
    lib.mp_annealed_moves_half_step.argtypes = [vp, C.POINTER(Ensemble), C.c_double, vp, C.c_int32, C.c_uint64, C.c_int32,
                                                vp]
    return lib


EXPORTS = ["mp_abi_version", "mp_device_count", "mp_last_error", "mp_create", "mp_destroy",
           "mp_set_prior", "mp_lnprob_batch", "mp_lnprob_batch_async", "mp_synchronize", "mp_lnprob_batch_device", "mp_model_at_data",
           "mp_curve_nodes", "mp_model_curves", "mp_model_curves_device", "mp_rhs_batch",
           "mp_stretch_half_step", "mp_fp64_peak_tflops", "mp_last_stiff_count",
           "mp_ensemble_half_step", "mp_ensemble_sync", "mp_ensemble_unpack", "mp_ensemble_order",
           "mp_tempered_half_step", "mp_tempered_swap", "mp_ensemble_moves_half_step", "mp_tempered_moves_half_step",
           "mp_chain_moments", "mp_chain_order_statistics", "mp_chain_autocorr", "mp_gompertz_curves", "mp_kernels_launched",
           "mp_peer_alloc", "mp_peer_open", "mp_peer_close", "mp_peer_free", "mp_peer_barrier"]
# The entry points include/magprop_smc.h declares (sequential Monte Carlo), exported by the same library.
SMC_EXPORTS = ["mp_smc_weights", "mp_smc_resample", "mp_annealed_moves_half_step"]
MP_SMC_TILE = 64


def load():
    """Load the CUDA library (built in-tree by __graft_entry__.build())."""
    global _LIB
    if _LIB is None:
        path = lib_path()
        if not os.path.exists(path):
            raise MagpropCudaError(
                f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(magprop_b200 has no CPU fallback)")
        _LIB = declare(C.CDLL(path))
        if _LIB.mp_abi_version() != MP_ABI_VERSION:
            raise MagpropCudaError("libmagprop_b200.so ABI version mismatch; rebuild")
    return _LIB


def check(rc: int):
    if rc == MP_OK:
        return
    msg = load().mp_last_error().decode(errors="replace")
    if rc == MP_ERR_DATA_RANGE:
        # interp1d(bounds_error=True) raises ValueError (funcs.py:233-234)
        raise ValueError(msg or "A value in x_new is outside the interpolation range.")
    if rc in (MP_ERR_BAD_ARG, MP_ERR_BAD_GRID, MP_ERR_NO_DATA):
        raise ValueError(msg or f"magprop_b200: bad argument (code {rc})")
    raise MagpropCudaError(msg or f"magprop_b200: CUDA error (code {rc})")


def ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)
