"""Closing a likelihood handle returns its device memory.

A handle owns device buffers of several kinds: the dataset, staging for the host-pointer calls, the work space of its
two own lanes, the work space of a lane for every caller stream it has seen, and a tempered ladder per lane.  Six
open / use / close cycles that touch every kind must leave the device's free memory where one warm cycle left it."""
import numpy as np
import pytest

from magprop_b200 import _capi as A
from magprop_b200.engine import Likelihood, time_grid
from oracle import magprop_oracle as O

N_HOST = 1 << 18       # one chunk on one of the handle's own lanes; ~0.3 GB of work space by slab_walkers' per-walker size
N_SIDE = 4096
CYCLES = 6
SLACK = 256 << 20      # a leaked lane would cost about 2 GB over the six cycles


def _cycle(golden, theta):
    import torch
    from magprop_b200.sampler import TemperedEnsemble, geometric_betas
    g = golden["lnprob_script"]
    lk = Likelihood(A.script_model_spec(), time_grid(None), g["Humped_x"], g["Humped_y"], g["Humped_yerr"],
                    O.SCRIPT_LOWER, O.SCRIPT_UPPER, device=0)
    assert np.isfinite(lk.lnprob(theta)).all()
    pars = theta[:N_SIDE].copy()
    pars[:, 2:] = 10.0 ** pars[:, 2:]
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):                       # a lane of the caller's stream
        d_th = torch.from_numpy(theta[:N_SIDE]).cuda()
        d_lnp = torch.empty(N_SIDE, dtype=torch.float64, device="cuda")
        lk.lnprob_device(d_th.data_ptr(), N_SIDE, 6, d_lnp.data_ptr(), stream=side.cuda_stream)
        d_pars = torch.from_numpy(pars[:256]).cuda()
        d_out = torch.empty((256, 3, lk.curve_nodes(10)), dtype=torch.float64, device="cuda")
        lk.curves_device(d_pars.data_ptr(), 256, 6, 10, d_out.data_ptr(), stream=side.cuda_stream)
    side.synchronize()
    assert torch.isfinite(d_lnp).all()
    assert np.isfinite(lk.model_at_data(pars[:64])).all()
    ens = TemperedEnsemble.from_likelihood(lk, 64, 6, geometric_betas(3, 0.1), seed=5)
    ens.initialise(theta[:64])
    ens.run(2, store=False)
    torch.cuda.synchronize()
    lk.close()
    del d_th, d_lnp, d_pars, d_out, ens
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_closing_a_handle_returns_its_device_memory(built, golden):
    import torch
    rng = np.random.RandomState(11)
    theta = np.clip(O.SYNTH_TRUTHS_LOG["Humped"] + 1e-3 * rng.randn(N_HOST, 6), O.SCRIPT_LOWER, O.SCRIPT_UPPER)
    _cycle(golden, theta)                               # context, module load, torch's allocator
    free_warm = torch.cuda.mem_get_info()[0]
    for _ in range(CYCLES):
        _cycle(golden, theta)
    free_after = torch.cuda.mem_get_info()[0]
    assert free_warm - free_after < SLACK, (free_warm - free_after) / 2 ** 20
