"""NumPy restatement of the device ensemble's half-step and replica swap (test double).

The same counter-based RNG (Philox4x32-10, Salmon et al. 2011), the same draw layout, mover -> row mapping and
partner rules, and the same arithmetic order as ``propose()`` / ``propose_de`` / ``deliver()`` and ``pt_swap_kernel``
in magprop_kernels.cu and the helpers of magprop_rng.cuh (the snooker sums are loops over the coordinates, as the
kernel adds them), with the log-probability supplied by the caller.  One half-step covers every move kind, with or
without a temperature ladder.  Arrays are the flat [T*n, ndim] / [T*n] of the device ensemble, row r = t*n + w.
Used (a) to check the kernels bit for bit on the GPU and (b) as the CPU stand-in for them in the gloo tests of the
multi-rank driver."""
import math

import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK = np.uint64(0xFFFFFFFF)
STRETCH, DE, SNOOKER = 0, 1, 2


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Vectorised over the counter words (uint64 arrays holding 32-bit values)."""
    c0, c1, c2, c3 = [np.asarray(c, dtype=np.uint64) & MASK for c in (c0, c1, c2, c3)]
    k0, k1 = int(k0) & 0xFFFFFFFF, int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0 = M0 * c0
        p1 = M1 * c2
        n0 = (p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0)
        n1 = p1 & MASK
        n2 = (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1)
        n3 = p0 & MASK
        c0, c1, c2, c3 = n0 & MASK, n1, n2 & MASK, n3
        k0 = (k0 + W0) & 0xFFFFFFFF
        k1 = (k1 + W1) & 0xFFFFFFFF
    return c0, c1, c2, c3


def u01(hi, lo):
    v = ((hi << np.uint64(32)) | lo) >> np.uint64(11)
    return (v.astype(np.float64) + 0.5) * (1.0 / 9007199254740992.0)


def _block(seed, hs, rows, word):
    """Philox counter (hs, row, word) keyed by the seed, for every row."""
    rows = np.asarray(rows, dtype=np.uint64)
    z = np.zeros_like(rows)
    return philox4x32_10(z + np.uint64(hs & 0xFFFFFFFF), z + np.uint64((hs >> 32) & 0xFFFFFFFF), rows,
                         z + np.uint64(word), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)


# ---- the ensemble order: keyed permutation of [0, n) (perm_at / make_split_perm in magprop_rng.cuh) ----
def _mix32(x):
    x = x & MASK
    x ^= x >> np.uint64(16); x = (x * np.uint64(0x7feb352d)) & MASK
    x ^= x >> np.uint64(15); x = (x * np.uint64(0x846ca68b)) & MASK
    x ^= x >> np.uint64(16)
    return x


def ensemble_order(n, seed, step, randomize=True):
    """order[g] = walker at position g of the ensemble order of MCMC step `step`; halves are g < n/2, g >= n/2."""
    g = np.arange(n, dtype=np.uint64)
    if not randomize:
        return g.astype(np.int64)
    hb = 1
    while (1 << (2 * hb)) < n:
        hb += 1
    mask = np.uint64((1 << hb) - 1)
    k = _block(seed, step, np.zeros(1, dtype=np.uint64), 2)
    k0, k1 = np.uint64(int(k[0][0])), np.uint64(int(k[1][0]))
    x = g.copy()
    todo = np.ones(n, dtype=bool)
    while todo.any():
        xx = x[todo]
        L, R = xx >> np.uint64(hb), xx & mask
        for r in range(6):
            F = _mix32(((R + np.uint64((r * 0x9E3779B9) & 0xFFFFFFFF)) & MASK) ^ (k1 if r & 1 else k0)) & mask
            L, R = R, L ^ F
        xx = (L << np.uint64(hb)) | R
        x[todo] = xx
        todo[todo] = xx >= np.uint64(n)
    return x.astype(np.int64)


def tempered_rows(n, ntemps, seed, step, split, randomize=True):
    """(temperature, row) of every mover of half-step `split` of MCMC step `step`, in mover order, and the rows of
    each temperature's complementary half [T, n/2] (``tempered_mover`` / ``tempered_partner``; T = 1 is the plain
    ensemble)."""
    half = n // 2
    order = ensemble_order(n, seed, step, randomize)
    t = np.repeat(np.arange(ntemps), half)
    rows = (np.arange(ntemps)[:, None] * n + order[split * half:(split + 1) * half][None, :]).ravel()
    comp = np.arange(ntemps)[:, None] * n + order[(1 - split) * half:(2 - split) * half][None, :]
    return t, rows, comp


# ---- the moves' draws, partner picks and choice (magprop_rng.cuh) ---------------------------------------------
def pick_index(u, m):
    """The partner rule: position min(floor(u m), m - 1) of m."""
    return np.minimum((np.asarray(u) * m).astype(np.int64), m - 1)


def stretch_draws(seed, hs, rows):
    """(u_z, u_partner) of the stretch move: Philox block (hs, row, 0)."""
    r = _block(seed, hs, rows, 0)
    return u01(r[0], r[1]), u01(r[2], r[3])


def move_draws(seed, hs, rows):
    """The four uniforms of a DE / snooker mover: Philox blocks (hs, row, 4) and (hs, row, 5)."""
    a, b = _block(seed, hs, rows, 4), _block(seed, hs, rows, 5)
    return u01(a[0], a[1]), u01(a[2], a[3]), u01(b[0], b[1]), u01(b[2], b[3])


def accept_uniform(kind, seed, hs, rows):
    """The accept draw: the stretch move's from words 0-1 of block (hs, row, 1); DE's and snooker's from words 2-3 of
    block (hs, row, 5), = move_draws(...)[3]."""
    if kind == STRETCH:
        r = _block(seed, hs, rows, 1)
        return u01(r[0], r[1])
    r = _block(seed, hs, rows, 5)
    return u01(r[2], r[3])


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
    r = _block(seed, step, np.zeros(1, dtype=np.uint64), 6)
    u = float(u01(r[0], r[1])[0])
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


def step_move(moves, seed, step):
    """The move of MCMC step `step` from a list of (move, weight)."""
    return moves[choose_move(seed, step, [w for _, w in moves])][0]


# ---- the half-step ------------------------------------------------------------------------------------------
def half_step(coords, lnp, rows, t, comp, move, seed, hs, lnprob_fn, betas=None, accepted=None):
    """In place: move the walkers of `rows` (mover order; temperature t of each) against their temperature's complement
    comp[t] with `move` (a StretchMove, DEMove or DESnookerMove) at half-step counter `hs`.  ``betas``: the ladder the
    accept test weighs the log-probabilities by (None: untempered).  Returns (q, accept)."""
    rows, t = np.asarray(rows), np.asarray(t)
    ndim, nc = coords.shape[1], comp.shape[1]
    x = coords[rows]
    n = rows.size
    if move.kind == STRETCH:
        a = move.a
        uz, up = stretch_draws(seed, hs, rows)
        zr = (a - 1.0) * uz + 1.0
        z = zr * zr / a
        c = coords[comp[t, pick_index(up, nc)]]
        q = c + -((c + -x) * z[:, None])
        lnf = (ndim - 1.0) * np.log(z)
    elif move.kind == DE:
        uj, uk, ug, _ = move_draws(seed, hs, rows)
        j, k = de_pair(uj, uk, nc)
        g0 = move.gamma0 if move.gamma0 else 2.38 / math.sqrt(2.0 * ndim)
        s3 = move.sigma * math.sqrt(3.0)
        g = g0 * (1.0 + s3 * (2.0 * ug - 1.0))
        q = x + g[:, None] * (coords[comp[t, j]] - coords[comp[t, k]])
        lnf = np.zeros(n)
    else:
        uz, u1, u2, _ = move_draws(seed, hs, rows)
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
    ua = accept_uniform(move.kind, seed, hs, rows)
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


# ---- the replica exchange (pt_swap_accept in magprop_rng.cuh, pt_swap_kernel) ----------------------------------
def swap_uniform(seed, step, rows):
    """u of the swap decision of the pairs whose hot row is `rows`: Philox counter (step, row, word 3)."""
    r = _block(seed, step, rows, 3)
    return u01(r[0], r[1])


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


class NumpyBackend:
    """CPU stand-in for ``magprop_b200.sampler.CudaBackend`` under a ``DeviceEnsemble`` or ``TemperedEnsemble``: the
    same half-steps and swaps on NumPy views of the ensemble's (CPU) tensors, with the log-probability supplied by the
    caller."""

    peer_capable = False

    def __init__(self, lnprob_fn):
        self.lnprob_fn = lnprob_fn

    def _sets(self, ens, step, split):
        n, half = ens.nwalkers, ens.nwalkers // 2
        order = ensemble_order(n, ens.seed, step, ens.randomize_split)
        m = half // ens.world
        pos0 = split * half + ens.rank * m
        return order, order[pos0:pos0 + m], order[(1 - split) * half:(1 - split) * half + half]

    def half_step(self, ens, step, split):
        coords, lnp = ens.coords.numpy(), ens.lnp.numpy()
        _, active, comp = self._sets(ens, step, split)
        half_step(coords, lnp, active, np.zeros(active.size, np.int64), comp[None, :], step_move(ens.moves, ens.seed, step),
                  ens.seed, 2 * step + split, self.lnprob_fn, accepted=ens.accepted.numpy())
        if ens.pack is not None:
            p = ens.pack.numpy()
            p[:, :ens.ndim] = coords[active]
            p[:, ens.ndim] = lnp[active]

    def unpack(self, ens, step, split, gathered):
        order, _, _ = self._sets(ens, step, split)
        half = ens.nwalkers // 2
        rows = order[split * half:split * half + half]
        g = gathered.numpy()
        ens.coords.numpy()[rows] = g[:, :ens.ndim]
        ens.lnp.numpy()[rows] = g[:, ens.ndim]

    def lnprob_all(self, ens):
        ens.lnp.numpy()[:] = self.lnprob_fn(ens.coords.numpy())

    def tempered_half_step(self, ens, step, split):
        t, rows, comp = tempered_rows(ens.nwalkers, ens.ntemps, ens.seed, step, split, ens.randomize_split)
        half_step(ens.coords.numpy(), ens.lnp.numpy(), rows, t, comp, step_move(ens.moves, ens.seed, step), ens.seed,
                  2 * step + split, self.lnprob_fn, betas=ens.betas, accepted=ens.accepted.numpy())

    def tempered_swap(self, ens, step):
        swap(ens.coords.numpy(), ens.lnp.numpy(), ens.betas, ens.nwalkers, ens.seed, step, ens.swap_accepted.numpy())
