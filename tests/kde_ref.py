"""NumPy restatement of the KDE move (MP_MOVE_KDE in include/magprop_b200.h; kde_log, gauss_pair and kde_gaussians in
magprop_rng.cuh; magprop_kde.cu) beside ``ensemble_ref``, and CPU backends that run it (test double).

The Gaussians, the centre pick, the tiled mean and covariance sums, the Cholesky factor, the proposal q and the
whitening are stated operation for operation, so q equals the device's bit for bit; ln f carries NumPy's ``exp`` and
``log`` where the device has libdevice's, and enters nothing but the accept comparison.  ``half_step`` is
``ensemble_ref.half_step`` with the KDE move added: every other kind is delegated to it unchanged."""
import math

import numpy as np

import ensemble_ref as E
import smc_ref as R

KDE = 4
KDE_MAX_CENTRES, KDE_TILE = 4096, 64


def accept_uniform(kind, seed, hs, rows):
    """The accept draw: the KDE move's from words 2-3 of block (hs, row, 8); the other kinds' as ensemble_ref's."""
    if kind == KDE:
        r = E._block(seed, hs, rows, 8)
        return E.u01(r[2], r[3])
    return E.accept_uniform(kind, seed, hs, rows)


_LOG_P = [1.0 / k for k in range(23, 2, -2)]
_SIN_P = [(-1) ** k / math.factorial(2 * k + 1) for k in range(9, 0, -1)]
_COS_P = [(-1) ** k / math.factorial(2 * k) for k in range(10, 0, -1)]


def kde_log(x):
    """ln x for positive normal x, operation for operation as kde_log."""
    x = np.asarray(x, dtype=np.float64)
    b = x.view(np.uint64)
    e = ((b >> np.uint64(52)) & np.uint64(0x7FF)).astype(np.int64) - 1023
    m = ((b & np.uint64(0x000FFFFFFFFFFFFF)) | np.uint64(0x3FF0000000000000)).view(np.float64)
    big = m > 1.4142135623730951
    m = np.where(big, m * 0.5, m)
    e = e + big
    s = (m - 1.0) / (m + 1.0)
    s2 = s * s
    p = np.full_like(s, _LOG_P[0])
    for c in _LOG_P[1:] + [1.0]:
        p = p * s2 + c
    ed = e.astype(np.float64)
    return ed * 6.93147180369123816490e-01 + (ed * 1.90821492927058770002e-10 + (2.0 * s) * p)


def gauss_pair(u1, u2):
    """One Box-Muller pair per (u1, u2), as gauss_pair."""
    u1, u2 = np.asarray(u1, dtype=np.float64), np.asarray(u2, dtype=np.float64)
    r = np.sqrt(-2.0 * kde_log(u1))
    t = 4.0 * u2
    quad = t.astype(np.int64)
    f = t - quad.astype(np.float64)
    refl = f > 0.5
    x = np.where(refl, 1.0 - f, f) * 1.5707963267948966
    x2 = x * x
    p = np.full_like(x, _SIN_P[0])
    for c in _SIN_P[1:]:
        p = p * x2 + c
    s = x + x * (x2 * p)
    q = np.full_like(x, _COS_P[0])
    for c in _COS_P[1:]:
        q = q * x2 + c
    c = 1.0 + x2 * q
    s, c = np.where(refl, c, s), np.where(refl, s, c)
    C = np.select([quad == 1, quad == 2, quad == 3], [-s, -c, s], c)
    S = np.select([quad == 1, quad == 2, quad == 3], [c, -s, -c], s)
    return r * C, r * S


def kde_draws(seed, hs, rows, ndim):
    """(u_c, z [n, ndim]): the centre uniform from block (hs, row, 8), the normals from blocks (hs, row, 9 + k)."""
    r = E._block(seed, hs, rows, 8)
    z = np.empty((np.asarray(rows).size, ndim))
    for k in range((ndim + 1) // 2):
        b = E._block(seed, hs, rows, 9 + k)
        a, c = gauss_pair(E.u01(b[0], b[1]), E.u01(b[2], b[3]))
        z[:, 2 * k] = a
        if 2 * k + 1 < ndim:
            z[:, 2 * k + 1] = c
    return E.u01(r[0], r[1]), z


def _tiled_sum(v):
    """Sum over axis 0 in tiles of KDE_TILE, each tile left to right, then the tile sums left to right."""
    K = (v.shape[0] + KDE_TILE - 1) // KDE_TILE
    pad = np.zeros((K * KDE_TILE,) + v.shape[1:])
    pad[:v.shape[0]] = v
    tiles = np.cumsum(pad.reshape((K, KDE_TILE) + v.shape[1:]), axis=1)[:, -1]
    return np.cumsum(tiles, axis=0)[-1]


def kde_fit(cent):
    """(mu, L, ok) of centres [M, d]: tiled sums, Sigma = S2 / (M - 1), Cholesky in row order."""
    M, d = cent.shape
    mu = _tiled_sum(cent) / float(M)
    e = cent - mu
    S2 = _tiled_sum(e[:, :, None] * e[:, None, :])
    L = np.zeros((d, d))
    for i in range(d):
        for j in range(i + 1):
            v = float(S2[i, j]) / float(M - 1)
            for c in range(j):
                v = v - float(L[i, c]) * float(L[j, c])
            if i == j:
                if not (v > 0.0 and math.isfinite(v)):
                    return mu, L, False
                L[i, i] = math.sqrt(v)
            else:
                L[i, j] = v / float(L[j, j])
    return mu, L, True


def kde_whiten(p, mu, L, h):
    """y = L^-1 (p - mu) / h by forward substitution, rows ascending; p [n, d]."""
    d = p.shape[1]
    w = np.empty_like(p)
    for r in range(d):
        s = p[:, r] - mu[r]
        for c in range(r):
            s = s - L[r, c] * w[:, c]
        w[:, r] = s / L[r, r]
    return w / h


def kde_lk(y, white, chunk=1024):
    """-0.5 min_j r2_j + log(sum_j exp(-0.5 (r2_j - min))), j ascending, for every row of y."""
    out = np.empty(y.shape[0])
    for i0 in range(0, y.shape[0], chunk):
        yy = y[i0:i0 + chunk]
        r = np.zeros((yy.shape[0], white.shape[0]))
        for c in range(y.shape[1]):
            e = yy[:, None, c] - white[None, :, c]
            r = r + e * e
        m = r.min(axis=1)
        s = np.cumsum(np.exp(-0.5 * (r - m[:, None])), axis=1)[:, -1]
        out[i0:i0 + chunk] = -0.5 * m + np.log(s)
    return out


def kde_bandwidth(move, M, ndim):
    b = move.bw_method
    return math.pow(M, -1.0 / (ndim + 4)) if (b is None or isinstance(b, str)) else float(b)


def kde_propose(coords, x, rows, t, comp, move, seed, hs):
    """(q, ln f) of the KDE move for movers at x (rows, temperatures t) against comp[t]."""
    n, ndim = x.shape
    M = min(comp.shape[1], KDE_MAX_CENTRES)
    h = kde_bandwidth(move, M, ndim)
    uc, z = kde_draws(seed, hs, rows, ndim)
    q, lnf = x.copy(), np.full(n, -np.inf)
    for tt in np.unique(t):
        sel = np.flatnonzero(t == tt)
        cent = coords[comp[tt, :M]]
        mu, L, ok = kde_fit(cent)
        if not ok:
            continue
        cj = cent[E.pick_index(uc[sel], M)]
        for r in range(ndim):
            s = np.zeros(sel.size)
            for c in range(r + 1):
                s = s + L[r, c] * z[sel, c]
            q[sel, r] = cj[:, r] + h * s
        white = kde_whiten(cent, mu, L, h)
        lnf[sel] = kde_lk(kde_whiten(x[sel], mu, L, h), white) - kde_lk(kde_whiten(q[sel], mu, L, h), white)
    return q, lnf


def half_step(coords, lnp, rows, t, comp, move, seed, hs, lnprob_fn, betas=None, accepted=None):
    """``ensemble_ref.half_step`` for every move kind, the KDE move included (same arguments, same result)."""
    if move.kind != KDE:
        return E.half_step(coords, lnp, rows, t, comp, move, seed, hs, lnprob_fn, betas=betas, accepted=accepted)
    rows, t = np.asarray(rows), np.asarray(t)
    q, lnf = kde_propose(coords, coords[rows], rows, t, comp, move, seed, hs)
    ua = accept_uniform(KDE, seed, hs, rows)
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


class NumpyBackend(E.NumpyBackend):
    """``ensemble_ref.NumpyBackend`` whose half-steps run every move kind through ``half_step`` above."""

    def half_step(self, ens, step, split):
        coords, lnp = ens.coords.numpy(), ens.lnp.numpy()
        _, active, comp = self._sets(ens, step, split)
        half_step(coords, lnp, active, np.zeros(active.size, np.int64), comp[None, :], E.step_move(ens.moves, ens.seed, step),
                  ens.seed, 2 * step + split, self.lnprob_fn, accepted=ens.accepted.numpy())
        if ens.pack is not None:
            p = ens.pack.numpy()
            p[:, :ens.ndim] = coords[active]
            p[:, ens.ndim] = lnp[active]

    def tempered_half_step(self, ens, step, split):
        t, rows, comp = E.tempered_rows(ens.nwalkers, ens.ntemps, ens.seed, step, split, ens.randomize_split)
        half_step(ens.coords.numpy(), ens.lnp.numpy(), rows, t, comp, E.step_move(ens.moves, ens.seed, step), ens.seed,
                  2 * step + split, self.lnprob_fn, betas=ens.betas, accepted=ens.accepted.numpy())


class SMCBackend(R.NumpyBackend):
    """``smc_ref.NumpyBackend`` whose annealed half-steps run every move kind through ``half_step`` above."""

    def annealed_half_step(self, ens, step, split):
        t, rows, comp = E.tempered_rows(ens.nwalkers, 1, ens.seed, step, split, ens.randomize_split)
        half_step(ens.coords.numpy(), ens.lnp.numpy(), rows, t, comp, E.step_move(ens.moves, ens.seed, step), ens.seed,
                  2 * step + split, self.lnprob_fn, betas=[ens.beta], accepted=ens.accepted.numpy())
