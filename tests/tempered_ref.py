"""NumPy restatement of the parallel-tempered half-step and swap (test double).

Same draws, same mover -> row mapping and the same arithmetic order as ``draw_for`` / ``deliver`` with a ladder and
``pt_swap_kernel`` in magprop_kernels.cu (``tempered_mover`` / ``pt_swap_accept`` in magprop_rng.cuh), built on
``stretch_ref``'s Philox and ensemble order.  Arrays are the flat [T*n, ndim] / [T*n] of the device ensemble, row
r = t*n + w."""
import numpy as np

import stretch_ref as R


def tempered_rows(n, ntemps, seed, step, split, randomize=True):
    """(temperature, row) of every mover of half-step `split` of MCMC step `step`, in mover order, and the rows of
    each temperature's complementary half [T, n/2]."""
    half = n // 2
    order = R.ensemble_order(n, seed, step, randomize)
    t = np.repeat(np.arange(ntemps), half)
    rows = (np.arange(ntemps)[:, None] * n + order[split * half:(split + 1) * half][None, :]).ravel()
    comp = np.arange(ntemps)[:, None] * n + order[(1 - split) * half:(2 - split) * half][None, :]
    return t, rows, comp


def half_step(coords, lnp, betas, n, split, a, seed, step, lnprob_fn, accepted=None, randomize=True):
    """In place: half-step `split` of MCMC step `step` of every temperature.  Returns the proposals and the accept mask
    in mover order.  With one temperature this is ``stretch_ref.half_step`` on ``ensemble_order``'s halves."""
    betas = np.asarray(betas, dtype=np.float64)
    ndim = coords.shape[1]
    half = n // 2
    t, rows, comp = tempered_rows(n, betas.size, seed, step, split, randomize)
    uz, up, ua = R.draws(seed, 2 * step + split, rows)
    zr = (a - 1.0) * uz + 1.0
    z = zr * zr / a
    pj = np.minimum((up * half).astype(np.int64), half - 1)
    c = coords[comp[t, pj]]
    x = coords[rows]
    q = c + -((c + -x) * z[:, None])
    lp_new = np.asarray(lnprob_fn(q), dtype=np.float64)
    b = betas[t]
    with np.errstate(invalid="ignore"):
        lnpdiff = ((ndim - 1.0) * np.log(z) + b * lp_new) + -(b * lnp[rows])
    acc = lnpdiff > np.log(ua)
    coords[rows[acc]] = q[acc]
    lnp[rows[acc]] = lp_new[acc]
    if accepted is not None:
        accepted[rows[acc]] += 1
    return q, acc


def swap_uniform(seed, step, rows):
    """u of the swap decision of the pairs whose hot row is `rows`: Philox counter (step, row, word 3)."""
    rows = np.asarray(rows, dtype=np.uint64)
    z = np.zeros_like(rows)
    r = R.philox4x32_10(z + np.uint64(step & 0xFFFFFFFF), z + np.uint64((step >> 32) & 0xFFFFFFFF), rows, z + np.uint64(3),
                        seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return R.u01(r[0], r[1])


def swap_accept(seed, step, rows_hot, beta_cold, beta_hot, lnp_hot, lnp_cold):
    with np.errstate(invalid="ignore"):
        return np.log(swap_uniform(seed, step, rows_hot)) < (beta_cold - beta_hot) * (lnp_hot - lnp_cold)


def swap(coords, lnp, betas, n, seed, step, counts=None):
    """In place: the swap pass of MCMC step `step`, pairs (t-1, t) from the hottest down, column by column."""
    betas = np.asarray(betas, dtype=np.float64)
    j = np.arange(n)
    for t in range(betas.size - 1, 0, -1):
        hot, cold = t * n + j, (t - 1) * n + j
        acc = swap_accept(seed, step, hot, betas[t - 1], betas[t], lnp[hot], lnp[cold])
        h, c = hot[acc], cold[acc]
        coords[h], coords[c] = coords[c].copy(), coords[h].copy()
        lnp[h], lnp[c] = lnp[c].copy(), lnp[h].copy()
        if counts is not None:
            counts[t - 1] += int(acc.sum())


class NumpyTemperedBackend(R.NumpyBackend):
    """CPU stand-in for ``CudaBackend`` under a ``TemperedEnsemble`` (CPU tensors, caller's log-probability)."""

    def tempered_half_step(self, ens, step, split):
        half_step(ens.coords.numpy(), ens.lnp.numpy(), ens.betas, ens.nwalkers, split, ens.a, ens.seed, step,
                  self.lnprob_fn, ens.accepted.numpy(), ens.randomize_split)

    def tempered_swap(self, ens, step):
        swap(ens.coords.numpy(), ens.lnp.numpy(), ens.betas, ens.nwalkers, ens.seed, step, ens.swap_accepted.numpy())
