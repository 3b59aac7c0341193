"""NumPy restatement of the SMC primitives (include/magprop_smc.h, magprop_smc.cu, smc_stage_uniform in magprop_rng.cuh)
and a CPU backend for ``SMCSampler`` (test double).

The weights and their sums are stated in exact terms: the kernels add in their own block order, so the tests compare
the sums against ``math.fsum`` within a relative bar.  The prefix sum, the stage uniform and the ancestor rule are the
kernels' to the bit: the same tiles, the same left-to-right additions, the same Philox counter."""
import math

import numpy as np

import ensemble_ref as E

TILE = 64          # MP_SMC_TILE


def smc_weights(lnp, dbeta):
    """(m, w, S1, S2): m the largest finite lnp (-inf if none), w_i = exp(dbeta (lnp_i - m)) for finite lnp_i, else 0;
    S1 and S2 exactly rounded (math.fsum)."""
    lnp = np.asarray(lnp, dtype=np.float64)
    fin = np.isfinite(lnp)
    if not fin.any():
        return -math.inf, np.zeros(lnp.size), 0.0, 0.0
    m = float(lnp[fin].max())
    w = np.zeros(lnp.size)
    w[fin] = np.exp(dbeta * (lnp[fin] - m))
    return m, w, math.fsum(w), math.fsum(w * w)


def prefix_sum(w):
    """(cum, total) in the documented order: within each tile of TILE a running sum from 0, left to right; the tiles'
    bases a running sum of the tile totals, left to right; cum_j = base of j's tile + running sum at j."""
    w = np.asarray(w, dtype=np.float64)
    n = w.size
    K = (n + TILE - 1) // TILE
    pad = np.zeros(K * TILE)
    pad[:n] = w
    p = np.cumsum(pad.reshape(K, TILE), axis=1)         # np.cumsum adds in order; the zero padding adds nothing
    base = np.concatenate([[0.0], np.cumsum(p[:, -1])])
    cum = (base[:-1, None] + p).ravel()[:n]
    return cum, float(base[K])


def stage_uniform(seed, stage):
    r = E._block(seed, stage, np.zeros(1, dtype=np.uint64), 7)
    return float(E.u01(r[0], r[1])[0])


def ancestors(w, seed, stage):
    """a_i = the smallest j with cum_j > (i + u)(total / n), clamped to the last j with w_j > 0; a_i = i if total == 0."""
    w = np.asarray(w, dtype=np.float64)
    n = w.size
    cum, total = prefix_sum(w)
    if not total > 0.0:
        return np.arange(n, dtype=np.int64)
    u = stage_uniform(seed, stage)
    target = (np.arange(n, dtype=np.float64) + u) * (total / n)
    a = np.searchsorted(cum, target, side="right")
    return np.minimum(a, np.flatnonzero(w > 0.0)[-1]).astype(np.int64)


class NumpyBackend(E.NumpyBackend):
    """``ensemble_ref.NumpyBackend`` with the SMC primitives: the annealed half-step is the restatement's half-step with
    the ladder [beta]; the weights and resampling as above, on the sampler's CPU tensors."""

    def annealed_half_step(self, ens, step, split):
        t, rows, comp = E.tempered_rows(ens.nwalkers, 1, ens.seed, step, split, ens.randomize_split)
        E.half_step(ens.coords.numpy(), ens.lnp.numpy(), rows, t, comp, E.step_move(ens.moves, ens.seed, step), ens.seed,
                    2 * step + split, self.lnprob_fn, betas=[ens.beta], accepted=ens.accepted.numpy())

    def smc_weights(self, ens, dbeta, write):
        m, w, s1, s2 = smc_weights(ens.lnp.numpy(), dbeta)
        if write:
            ens.weights.numpy()[:] = w
        return m, s1, s2

    def smc_resample(self, ens, stage):
        a = ancestors(ens.weights.numpy(), ens.seed, stage)
        ens.resampled_coords.numpy()[:] = ens.coords.numpy()[a]
        ens.resampled_lnp.numpy()[:] = ens.lnp.numpy()[a]
