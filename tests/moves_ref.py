"""NumPy restatement of the device ensemble's moves (test double): the stretch, differential-evolution and snooker
proposals, the move choice and the partner rules of ``propose_de`` / ``deliver`` in magprop_kernels.cu and
``move_draws`` / ``de_pair`` / ``snooker_triple`` / ``choose_move`` in magprop_rng.cuh, in the kernels' operation
order (the snooker sums are loops over the coordinates, as the kernel adds them).  Built on ``stretch_ref``'s Philox
and ensemble order and ``tempered_ref``'s mover -> row mapping; the log-probability is the caller's."""
import math

import numpy as np

import stretch_ref as R
import tempered_ref as TR

STRETCH, DE, SNOOKER = 0, 1, 2


def pick_index(u, m):
    """The partner rule: position min(floor(u m), m - 1) of m."""
    return np.minimum((np.asarray(u) * m).astype(np.int64), m - 1)


def move_draws(seed, hs, rows):
    """The four uniforms of a DE / snooker mover: Philox blocks (hs, row, 4) and (hs, row, 5)."""
    rows = np.asarray(rows, dtype=np.uint64)
    z = np.zeros_like(rows)
    lo, hi = np.uint64(hs & 0xFFFFFFFF), np.uint64((hs >> 32) & 0xFFFFFFFF)
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    a = R.philox4x32_10(z + lo, z + hi, rows, z + np.uint64(4), k0, k1)
    b = R.philox4x32_10(z + lo, z + hi, rows, z + np.uint64(5), k0, k1)
    return R.u01(a[0], a[1]), R.u01(a[2], a[3]), R.u01(b[0], b[1]), R.u01(b[2], b[3])


def de_pair(uj, uk, nc):
    j = pick_index(uj, nc)
    k = pick_index(uk, nc - 1)
    return j, k + (k >= j)


def snooker_triple(uz, u1, u2, nc):
    z = pick_index(uz, nc)
    r1 = pick_index(u1, nc - 1)
    r1 = r1 + (r1 >= z)
    lo, hi = np.minimum(z, r1), np.maximum(z, r1)
    r2 = pick_index(u2, nc - 2)
    r2 = r2 + (r2 >= lo)
    r2 = r2 + (r2 >= hi)
    return z, r1, r2


def choose_move(seed, step, weights):
    """Index of the move MCMC step `step` runs: u from Philox (step, 0, 6), the first k with u W < cum_k."""
    one = np.zeros(1, dtype=np.uint64)
    r = R.philox4x32_10(one + np.uint64(step & 0xFFFFFFFF), one + np.uint64((step >> 32) & 0xFFFFFFFF), one,
                        one + np.uint64(6), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    u = float(R.u01(r[0], r[1])[0])
    W = 0.0
    for w in weights:
        W += w
    uw, cum, last = u * W, 0.0, 0
    for k, w in enumerate(weights):
        cum += w
        if w > 0.0:
            last = k
        if uw < cum:
            return k
    return last


def half_step(coords, lnp, rows, t, comp, move, seed, hs, lnprob_fn, betas=None, accepted=None):
    """In place: move the walkers of `rows` (mover order; temperature t of each) against their temperature's complement
    comp[t] with `move` (a StretchMove, DEMove or DESnookerMove) at half-step counter `hs`.  Returns (q, accept)."""
    rows, t = np.asarray(rows), np.asarray(t)
    ndim, nc = coords.shape[1], comp.shape[1]
    x = coords[rows]
    n = rows.size
    if move.kind == STRETCH:
        a = move.a
        uz, up, ua = R.draws(seed, hs, rows)
        zr = (a - 1.0) * uz + 1.0
        z = zr * zr / a
        c = coords[comp[t, pick_index(up, nc)]]
        q = c + -((c + -x) * z[:, None])
        lnf = (ndim - 1.0) * np.log(z)
    elif move.kind == DE:
        uj, uk, ug, ua = move_draws(seed, hs, rows)
        j, k = de_pair(uj, uk, nc)
        g0 = move.gamma0 if move.gamma0 else 2.38 / math.sqrt(2.0 * ndim)
        s3 = move.sigma * math.sqrt(3.0)
        g = g0 * (1.0 + s3 * (2.0 * ug - 1.0))
        q = x + g[:, None] * (coords[comp[t, j]] - coords[comp[t, k]])
        lnf = np.zeros(n)
    else:
        uz, u1, u2, ua = move_draws(seed, hs, rows)
        jz, j1, j2 = snooker_triple(uz, u1, u2, nc)
        zc, c1, c2 = coords[comp[t, jz]], coords[comp[t, j1]], coords[comp[t, j2]]
        e = x - zc
        ee, dd = np.zeros(n), np.zeros(n)
        for c in range(ndim):
            ee = ee + e[:, c] * e[:, c]
            dd = dd + (c1[:, c] - c2[:, c]) * e[:, c]
        live = ee != 0.0
        with np.errstate(invalid="ignore", divide="ignore"):
            f = np.where(live, (move.gammas * dd) / ee, 0.0)
            q = np.where(live[:, None], x + f[:, None] * e, x)
            nq = np.zeros(n)
            for c in range(ndim):
                w = q[:, c] - zc[:, c]
                nq = nq + w * w
            lnf = np.where(~live, 0.0, np.where(nq == 0.0, -np.inf, (0.5 * (ndim - 1.0)) * np.log(nq / ee)))
    lp_new = np.asarray(lnprob_fn(q), dtype=np.float64)
    lq, lx = lp_new, lnp[rows]
    if betas is not None:
        b = np.asarray(betas, dtype=np.float64)[t]
        lq, lx = b * lq, b * lx
    with np.errstate(invalid="ignore"):
        acc = ((lnf + lq) + -lx) > np.log(ua)
    coords[rows[acc]] = q[acc]
    lnp[rows[acc]] = lp_new[acc]
    if accepted is not None:
        accepted[rows[acc]] += 1
    return q, acc


def step_move(moves, seed, step):
    """The move of MCMC step `step` from a list of (move, weight)."""
    return moves[choose_move(seed, step, [w for _, w in moves])][0]


class NumpyMovesBackend(TR.NumpyTemperedBackend):
    """CPU stand-in for ``CudaBackend`` under a ``DeviceEnsemble`` or ``TemperedEnsemble`` with ``moves``: the same
    half-steps on NumPy views of the ensemble's CPU tensors (``moves=None``: the stretch restatements)."""

    def half_step(self, ens, step, split):
        if ens.moves is None:
            return super().half_step(ens, step, split)
        coords, lnp, acc = ens.coords.numpy(), ens.lnp.numpy(), ens.accepted.numpy()
        _, active, comp = self._sets(ens, step, split)
        half_step(coords, lnp, active, np.zeros(active.size, np.int64), comp[None, :], step_move(ens.moves, ens.seed, step),
                  ens.seed, 2 * step + split, self.lnprob_fn, accepted=acc)
        if ens.pack is not None:
            p = ens.pack.numpy()
            p[:, :ens.ndim] = coords[active]
            p[:, ens.ndim] = lnp[active]

    def tempered_half_step(self, ens, step, split):
        if ens.moves is None:
            return super().tempered_half_step(ens, step, split)
        t, rows, comp = TR.tempered_rows(ens.nwalkers, ens.ntemps, ens.seed, step, split, ens.randomize_split)
        half_step(ens.coords.numpy(), ens.lnp.numpy(), rows, t, comp, step_move(ens.moves, ens.seed, step), ens.seed,
                  2 * step + split, self.lnprob_fn, betas=ens.betas, accepted=ens.accepted.numpy())
