"""Ensemble (stretch-move) drivers for the batched likelihood.

The reference hands its ``lnprob`` to emcee (``synth_mcmc.py:178-185``: default
``StretchMove(a=2)``, ``Pool``-parallel).  emcee is not installed in this image,
so this module carries the minimum needed to run and measure the path:

``EnsembleSampler``     host-side stretch move with emcee's call pattern; the
                        log-probability is any callable, normally
                        ``mcmc_eqns.lnprob_batch`` with ``vectorize=True``
                        (one kernel launch per half-step).
``DeviceEnsemble``      positions stay on the GPU; proposal + likelihood +
                        accept are ONE fused launch per half-step
                        (``mp_ensemble_half_step``).  With ``torch.distributed``
                        initialised every rank holds a replica of the ensemble and
                        moves its share of the active half.  ``exchange="peer"``: the
                        replicas are mapped into one another over NVLink; a rank writes
                        what it moves into its own replica and the kernels read the rows
                        they need from the replica of the rank that moved them last -- no
                        collective, one flag barrier per half-step (``sync()`` completes
                        a replica for reading the chain out).  ``exchange="allgather"``:
                        the moved rows packed into ONE all-gather per half-step (gloo in
                        the CPU tests).
``TemperedEnsemble``    parallel tempering as emcee 2's ``PTSampler`` / ptemcee do
                        it: T temperatures x n walkers moved in ONE fused launch
                        per half-step (``mp_tempered_half_step``), then one swap
                        pass per step (``mp_tempered_swap``).
``thermodynamic_log_evidence``  ln Z by thermodynamic integration over the ladder.
``StretchMove``, ``DEMove``, ``DESnookerMove``  emcee 3's ``moves=``: both ensembles take a move, a list of
                        moves or a list of ``(move, weight)`` and run one of them per step
                        (``mp_ensemble_moves_half_step`` / ``mp_tempered_moves_half_step``).

Move semantics (Goodman & Weare 2010, as emcee's RedBlueMove implements them;
SURVEY.md appendix C): every step the walkers are split into two halves at random
(``randomize_split=True``, emcee's default); for each half S with complement C:
z = ((a-1)u+1)^2/a,  q = c_j - (c_j - s) z  with j uniform in C (with
replacement),  accept iff  (ndim-1) ln z + lp(q) - lp(s) > ln u'.   C includes
the updates made by the first half-step of the same step.  On the device the
random split is a permutation keyed by (seed, step) that every thread of every
rank evaluates on the fly (include/magprop_b200.h, ``mp_ensemble``).
"""
from __future__ import annotations

import ctypes as C

import numpy as np


class EnsembleSampler:
    """Minimal host-side stand-in for ``emcee.EnsembleSampler`` (stretch move only)."""

    def __init__(self, nwalkers, ndim, log_prob_fn, args=(), kwargs=None, vectorize=True, a=2.0, seed=None):
        if nwalkers % 2 or nwalkers < 2 * ndim:
            raise ValueError("nwalkers must be even and at least 2*ndim")
        self.nwalkers, self.ndim, self.a = nwalkers, ndim, float(a)
        self.log_prob_fn, self.args, self.kwargs = log_prob_fn, tuple(args), dict(kwargs or {})
        self.vectorize = vectorize
        self.random = np.random.RandomState(seed)
        self.chain = None          # [nsteps, nwalkers, ndim]
        self.log_prob = None       # [nsteps, nwalkers]
        self.naccepted = np.zeros(nwalkers, dtype=np.int64)
        self.iteration = 0

    def compute_log_prob(self, coords):
        coords = np.ascontiguousarray(coords, dtype=np.float64)
        if not np.isfinite(coords).all():
            raise ValueError("At least one parameter value was infinite or NaN")
        if self.vectorize:
            lp = np.asarray(self.log_prob_fn(coords, *self.args, **self.kwargs), dtype=np.float64)
        else:
            lp = np.array([self.log_prob_fn(c, *self.args, **self.kwargs) for c in coords], dtype=np.float64)
        if np.isnan(lp).any():
            raise ValueError("Probability function returned NaN")
        return lp

    def run_mcmc(self, p0, nsteps):
        coords = np.array(p0, dtype=np.float64).reshape(self.nwalkers, self.ndim)
        lp = self.compute_log_prob(coords)
        chain = np.empty((nsteps, self.nwalkers, self.ndim))
        lps = np.empty((nsteps, self.nwalkers))
        for it in range(nsteps):
            inds = np.arange(self.nwalkers) % 2
            self.random.shuffle(inds)
            for split in (0, 1):
                S = np.where(inds == split)[0]
                Cset = np.where(inds != split)[0]
                ns = S.size
                zz = ((self.a - 1.0) * self.random.rand(ns) + 1.0) ** 2.0 / self.a
                rint = self.random.randint(Cset.size, size=ns)
                c = coords[Cset[rint]]
                q = c - (c - coords[S]) * zz[:, None]
                new_lp = self.compute_log_prob(q)
                lnpdiff = (self.ndim - 1.0) * np.log(zz) + new_lp - lp[S]
                accept = lnpdiff > np.log(self.random.rand(ns))
                coords[S[accept]] = q[accept]
                lp[S[accept]] = new_lp[accept]
                self.naccepted[S[accept]] += 1
            chain[it] = coords
            lps[it] = lp
            self.iteration += 1
        self.chain = chain if self.chain is None else np.concatenate([self.chain, chain])
        self.log_prob = lps if self.log_prob is None else np.concatenate([self.log_prob, lps])
        return coords, lp

    def get_chain(self):
        return self.chain

    def get_log_prob(self):
        return self.log_prob

    @property
    def acceptance_fraction(self):
        return self.naccepted / max(1, self.iteration)


# ---- emcee 3's moves= ------------------------------------------------------------------------------------
class StretchMove:
    """emcee's ``StretchMove(a=2.0)``: the affine-invariant stretch move (Goodman & Weare 2010), scale ``a`` > 1."""
    kind = 0

    def __init__(self, a=2.0):
        self.a = float(a)

    def _check(self):
        if not (np.isfinite(self.a) and self.a > 1.0):
            raise ValueError("StretchMove needs a > 1")

    def _fill(self, m):
        m.a = self.a

    def __repr__(self):
        return f"StretchMove(a={self.a})"


class DEMove:
    """emcee's ``DEMove(sigma=1e-5, gamma0=None)``: differential evolution (Nelson et al. 2014),
    q = x + g (c_j - c_k) for an ordered pair of distinct walkers j, k of the complement.  g is ``gamma0`` (None:
    2.38 / sqrt(2 ndim)) times 1 + a jitter of standard deviation ``sigma`` -- uniform here, Gaussian in emcee
    (include/magprop_b200.h, mp_move, says why)."""
    kind = 1

    def __init__(self, sigma=1.0e-5, gamma0=None):
        self.sigma = float(sigma)
        self.gamma0 = None if gamma0 is None else float(gamma0)

    def _check(self):
        if not 0.0 <= self.sigma < 1.0:
            raise ValueError("DEMove needs 0 <= sigma < 1")
        if self.gamma0 is not None and not (np.isfinite(self.gamma0) and self.gamma0 > 0.0):
            raise ValueError("DEMove needs gamma0 > 0 (or None for 2.38 / sqrt(2 ndim))")

    def _fill(self, m):
        m.sigma, m.gamma0 = self.sigma, 0.0 if self.gamma0 is None else self.gamma0

    def __repr__(self):
        return f"DEMove(sigma={self.sigma}, gamma0={self.gamma0})"


class DESnookerMove:
    """emcee's ``DESnookerMove(gammas=1.7)``: the snooker update of ter Braak & Vrugt (2008) -- x moves along the line
    through a third walker z by ``gammas`` times the projection of the difference of two more onto it, with the
    Hastings factor (|q - z| / |x - z|)^(ndim - 1)."""
    kind = 2

    def __init__(self, gammas=1.7):
        self.gammas = float(gammas)

    def _check(self):
        if not (np.isfinite(self.gammas) and self.gammas > 0.0):
            raise ValueError("DESnookerMove needs gammas > 0")

    def _fill(self, m):
        m.gammas = self.gammas

    def __repr__(self):
        return f"DESnookerMove(gammas={self.gammas})"


_PARTNERS = {0: 1, 1: 2, 2: 3}        # distinct complement walkers a move needs


def move_table(moves, half=None):
    """``moves`` as emcee accepts it -- a move, a list of moves (equal weights) or a list of ``(move, weight)`` --
    checked (``ValueError``) and returned as ``(list of (move, weight), ctypes array of mp_move)``.  ``half``: the
    walkers in a half of the ensemble (per temperature), which must hold every partner a weighted move draws."""
    from . import _capi as A
    single = (StretchMove, DEMove, DESnookerMove)
    if isinstance(moves, single):
        moves = [moves]
    try:
        items = list(moves)
    except TypeError:
        raise ValueError("moves must be a move, a list of moves or a list of (move, weight)") from None
    if not 1 <= len(items) <= A.MP_MAX_MOVES:
        raise ValueError(f"between 1 and {A.MP_MAX_MOVES} moves")
    table = []
    for it in items:
        if isinstance(it, single):
            mv, w = it, 1.0
        elif isinstance(it, (tuple, list)) and len(it) == 2 and isinstance(it[0], single):
            mv, w = it
        else:
            raise ValueError(f"not a move or (move, weight): {it!r}")
        try:
            w = float(w)
        except (TypeError, ValueError):
            raise ValueError(f"bad move weight: {it!r}") from None
        if not (np.isfinite(w) and w >= 0.0):
            raise ValueError("move weights must be finite and >= 0")
        mv._check()
        if half is not None and w > 0.0 and half < _PARTNERS[mv.kind]:
            raise ValueError(f"{mv!r} needs at least {_PARTNERS[mv.kind]} walkers in each half of the ensemble")
        table.append((mv, w))
    total = sum(w for _, w in table)
    if not (np.isfinite(total) and total > 0.0):
        raise ValueError("move weights must have a positive, finite sum")
    arr = (A.Move * len(table))()
    for m, (mv, w) in zip(arr, table):
        m.kind, m.weight = mv.kind, w
        mv._fill(m)
    return table, arr


def rank_slice(n_items: int, rank: int, world: int):
    """Contiguous equal share of n_items for `rank`; n_items must divide evenly."""
    if n_items % world:
        raise ValueError(f"half-ensemble of {n_items} walkers does not split evenly over {world} ranks")
    m = n_items // world
    return rank * m, (rank + 1) * m


class _RawCuda:
    """A raw device allocation presented through ``__cuda_array_interface__`` (so torch can view it)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False),
                                         "version": 3, "strides": None}


class CudaBackend:
    """The CUDA library as the mover of a ``DeviceEnsemble`` (``mp_ensemble_half_step`` and friends)."""

    peer_capable = True

    def __init__(self, lik):
        import torch
        from . import _capi as A
        self.A, self.lik, self.lib, self.torch = A, lik, A.load(), torch
        self.device = torch.device("cuda", lik.device)
        self._own = []          # (ptr, tensor) blocks from mp_peer_alloc
        self._opened = []       # peer mappings from mp_peer_open

    def stream(self):
        return self.torch.cuda.current_stream(self.device).cuda_stream

    def alloc_shared(self, nbytes):
        """Zeroed device memory other processes can map (CUDA IPC): (uint8 tensor view, 64-byte handle)."""
        ptr = C.c_void_p()
        handle = C.create_string_buffer(64)
        self.A.check(self.lib.mp_peer_alloc(self.lik.device, nbytes, C.byref(ptr), handle))
        t = self.torch.as_tensor(_RawCuda(ptr.value, nbytes), device=self.device)
        self._own.append((ptr.value, t))
        return t, handle.raw

    def open_peer(self, handle: bytes) -> int:
        ptr = C.c_void_p()
        self.A.check(self.lib.mp_peer_open(self.lik.device, handle, C.byref(ptr)))
        self._opened.append(ptr.value)
        return ptr.value

    def release(self):
        for p in self._opened:
            self.lib.mp_peer_close(self.lik.device, p)
        self._opened = []
        for p, _ in self._own:
            self.lib.mp_peer_free(self.lik.device, p)
        self._own = []

    def half_step(self, ens, step, split):
        self.A.check(self.lib.mp_ensemble_moves_half_step(self.lik._h, C.byref(ens.desc), C.addressof(ens._moves_c),
                                                          len(ens._moves_c), step, split, self.stream() or None))

    def unpack(self, ens, step, split, gathered):
        self.A.check(self.lib.mp_ensemble_unpack(C.byref(ens.desc), step, split, gathered.data_ptr(), self.stream() or None))

    def sync(self, ens, step):
        self.A.check(self.lib.mp_ensemble_sync(C.byref(ens.desc), step, self.stream() or None))

    def barrier(self, ens, epoch):
        self.A.check(self.lib.mp_peer_barrier(self.lik.device, ens._flags.data_ptr(), ens._peer_flag_ptrs, ens.rank,
                                              ens.world, epoch, ens._error.data_ptr(), self.stream() or None))

    def lnprob_all(self, ens):
        self.lik.lnprob_device(ens.coords.data_ptr(), ens.coords.shape[0], ens.ndim, ens.lnp.data_ptr(), 0, 0, self.stream())

    def tempered_half_step(self, ens, step, split):
        self.A.check(self.lib.mp_tempered_moves_half_step(self.lik._h, C.byref(ens.desc), ens.ntemps, self.A.ptr(ens.betas),
                                                          C.addressof(ens._moves_c), len(ens._moves_c), step, split,
                                                          self.stream() or None))

    def tempered_swap(self, ens, step):
        self.A.check(self.lib.mp_tempered_swap(C.byref(ens.desc), ens.ntemps, self.A.ptr(ens.betas), step,
                                               ens.swap_accepted.data_ptr(), self.stream() or None))


class DeviceEnsemble:
    """Ensemble whose positions live on the device (replicated on every rank of a distributed run).

    ``backend`` performs the half-steps: ``CudaBackend`` on a GPU (see ``from_likelihood``); the tests inject a
    NumPy double so the sharding / exchange logic runs under gloo on the CPU.

    ``moves`` (emcee 3's argument, see ``move_table``): one of the given moves per step, chosen by weight from the
    seed; None is ``StretchMove(a)``, and otherwise ``a`` is unused.
    """

    BAD_CAPACITY = 4096
    PEER_READ_MAX_BYTES = 256 << 20
    ntemps = 1                  # rows = ntemps * nwalkers (TemperedEnsemble)

    def __init__(self, backend, nwalkers, ndim, a=2.0, seed=0, device="cuda", dist=None, randomize_split=True,
                 exchange="auto", moves=None):
        import torch
        from . import _capi as A
        if nwalkers % 2 or nwalkers < 2 * ndim:
            raise ValueError("nwalkers must be even and at least 2*ndim")
        self.moves, self._moves_c = move_table(StretchMove(a) if moves is None else moves, nwalkers // 2)
        self.torch, self.backend = torch, backend
        self.nwalkers, self.ndim, self.a, self.seed = nwalkers, ndim, float(a), int(seed)
        self.randomize_split = bool(randomize_split)
        self.device = torch.device(device)
        self.dist = dist if (dist is not None and dist.is_initialized() and dist.get_world_size() > 1) else None
        self.rank = self.dist.get_rank() if self.dist else 0
        self.world = self.dist.get_world_size() if self.dist else 1
        half = nwalkers // 2
        lo, hi = rank_slice(half, self.rank, self.world)
        self.n_mine = hi - lo
        if self.world - 1 > A.MP_MAX_PEERS:
            raise ValueError(f"at most {A.MP_MAX_PEERS + 1} ranks")
        # ---- how the moved rows travel
        if not self.dist:
            exchange = "none"
        elif exchange == "auto":
            # Peer reads touch the other ranks' replicas at random rows: fine while a replica stays within reach of the
            # GPU's address-translation caches, 4x slower than the all-gather beyond (measured on 8 B200: 2^21 walkers
            # 2.0 vs 2.4 ms per step in favour of the reads, 10^7 walkers 36.8 vs 9.4 ms against them).
            small = nwalkers * (ndim + 1) * 8 <= self.PEER_READ_MAX_BYTES
            exchange = "peer" if (small and getattr(backend, "peer_capable", False)
                                  and self.dist.get_backend() == "nccl") else "allgather"
        if exchange not in ("none", "peer", "allgather"):
            raise ValueError("exchange must be 'auto', 'peer' or 'allgather'")
        self._peer_ptrs = []
        self._epoch = 0
        if exchange == "peer":
            exchange = self._setup_peer_block()          # falls back to "allgather" if a mapping fails on any rank
        rows = self.ntemps * nwalkers
        if exchange != "peer":
            self.coords = torch.empty((rows, ndim), dtype=torch.float64, device=self.device)
            self.lnp = torch.empty(rows, dtype=torch.float64, device=self.device)
        self.exchange = exchange
        self.accepted = torch.zeros(rows, dtype=torch.int32, device=self.device)
        self.status = torch.zeros(rows, dtype=torch.int32, device=self.device)
        self.bad_rows = torch.zeros((self.BAD_CAPACITY, ndim), dtype=torch.float64, device=self.device)
        self.bad_count = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.pack = self.gathered = None
        if exchange == "allgather":
            self.pack = torch.empty((self.n_mine, ndim + 1), dtype=torch.float64, device=self.device)
            self.gathered = torch.empty((half, ndim + 1), dtype=torch.float64, device=self.device)
        self.step = 0
        self._synced_step = 0       # the replicas held every row when this step began (peer exchange)
        # ---- the C descriptor
        d = A.Ensemble()
        d.coords, d.lnp = self.coords.data_ptr(), self.lnp.data_ptr()
        d.nwalkers, d.ndim, d.a, d.seed = nwalkers, ndim, self.a, self.seed
        d.randomize_split, d.rank, d.world = int(self.randomize_split), self.rank, self.world
        d.accepted, d.status, d.n_rhs = self.accepted.data_ptr(), self.status.data_ptr(), None
        d.n_peers = len(self._peer_ptrs)
        for k, (pc, pl) in enumerate(self._peer_ptrs):
            d.peer_coords[k], d.peer_lnp[k] = pc, pl
        d.synced_step = 0
        d.pack_out = self.pack.data_ptr() if self.pack is not None else None
        d.bad_rows, d.bad_count, d.bad_capacity = self.bad_rows.data_ptr(), self.bad_count.data_ptr(), self.BAD_CAPACITY
        self.desc = d

    # -- peer-mapped replicas --------------------------------------------------------------------
    def _setup_peer_block(self):
        """One IPC-exportable block per rank: coords | lnp | flags[16] | error.  Every rank maps every other
        rank's block.  Returns the exchange mode that holds on ALL ranks."""
        t, n, ndim = self.torch, self.nwalkers, self.ndim
        nb_c, nb_l, nb_f = n * ndim * 8, n * 8, 16 * 8
        ok = 1
        try:
            block, handle = self.backend.alloc_shared(nb_c + nb_l + nb_f + 8)
        except Exception:
            ok, block, handle = 0, None, b""
        handles = [None] * self.world
        self.dist.all_gather_object(handles, handle)
        ptrs = {}
        if ok:
            try:
                for r, hd in enumerate(handles):
                    if r != self.rank:
                        if len(hd) != 64:
                            raise RuntimeError("peer has no block")
                        ptrs[r] = self.backend.open_peer(hd)
            except Exception:
                ok = 0
        flag = t.tensor([ok], dtype=t.int32, device=self.device)
        self.dist.all_reduce(flag, op=self.dist.ReduceOp.MIN)
        if int(flag.item()) != 1:
            self.backend.release()
            return "allgather"
        self.coords = block[:nb_c].view(t.float64).view(n, ndim)
        self.lnp = block[nb_c:nb_c + nb_l].view(t.float64)
        self._flags = block[nb_c + nb_l:nb_c + nb_l + nb_f].view(t.int64)
        self._error = block[nb_c + nb_l + nb_f:].view(t.int32)
        self._peer_ptrs = [(ptrs[r], ptrs[r] + nb_c) for r in range(self.world) if r != self.rank]
        arr = (C.c_void_p * self.world)()
        for r in range(self.world):
            arr[r] = (ptrs[r] + nb_c + nb_l) if r != self.rank else None
        self._peer_flag_ptrs = arr
        return "peer"

    @classmethod
    def from_likelihood(cls, lik, nwalkers, ndim, a=2.0, seed=0, dist=None, randomize_split=True, exchange="auto",
                        moves=None):
        import torch
        ens = cls(CudaBackend(lik), nwalkers, ndim, a=a, seed=seed, device=torch.device("cuda", lik.device), dist=dist,
                  randomize_split=randomize_split, exchange=exchange, moves=moves)
        ens._lik = lik
        return ens

    def close(self):
        """Unmap the peers' replicas and free this rank's (after every rank is done with them)."""
        if self.exchange == "peer":
            self.torch.cuda.synchronize(self.device)
            self.dist.barrier()
            self.backend.release()
            self.exchange = "closed"

    # -- state ----------------------------------------------------------------------------------------
    def set_state(self, coords, lnp):
        t = self.torch
        self.coords.copy_(t.as_tensor(np.asarray(coords), dtype=t.float64).to(self.device)
                          if not isinstance(coords, t.Tensor) else coords)
        self.lnp.copy_(t.as_tensor(np.asarray(lnp), dtype=t.float64).to(self.device)
                       if not isinstance(lnp, t.Tensor) else lnp)
        self._sync_ranks()

    def initialise(self, p0):
        """Positions from p0 and their lnprob from the likelihood (GPU ensembles only)."""
        self.set_state(p0, np.zeros(self.ntemps * self.nwalkers))
        self.backend.lnprob_all(self)
        self._sync_ranks()

    def _sync_ranks(self):
        # peers read this replica during a half-step: nobody may start one before everybody's state is in place
        if self.exchange == "peer":
            self.torch.cuda.synchronize(self.device)
            self.dist.barrier()
            self._synced_step = self.step
            self.desc.synced_step = self.step

    def sync(self):
        """Complete this rank's replica (``exchange="peer"``: between the half-steps a replica is current only for
        the rows its rank moved last).  Call before reading ``coords`` / ``lnp``; a no-op for the other exchanges."""
        if self.exchange != "peer" or self._synced_step == self.step:
            return
        self._epoch += 1
        self.backend.barrier(self, self._epoch)          # every rank has finished writing ...
        self.backend.sync(self, self.step)
        self._epoch += 1
        self.backend.barrier(self, self._epoch)          # ... and reading, before anyone moves on
        self._synced_step = self.step
        self.desc.synced_step = self.step

    # -- stepping ---------------------------------------------------------------------------------------
    def _half(self, split):
        """This rank's share of half `split` of the current step, then the exchange."""
        self.backend.half_step(self, self.step, split)
        if self.exchange == "peer":
            self._epoch += 1
            self.backend.barrier(self, self._epoch)
        elif self.exchange == "allgather":
            self.dist.all_gather_into_tensor(self.gathered, self.pack)
            self.backend.unpack(self, self.step, split, self.gathered)

    def run(self, nsteps, store=False):
        """nsteps steps (2 half-steps each).  Returns the chain
        [nsteps, nwalkers, ndim] and lnprob [nsteps, nwalkers] when store=True."""
        chain, lps = self._buffers(nsteps) if store else (None, None)
        self._advance(nsteps, chain, lps, 0)
        self.sync()
        return (chain, lps) if store else None

    def _buffers(self, nsteps):
        """Empty chain and lnprob buffers of ``nsteps`` steps, in the shapes ``run`` returns."""
        t = self.torch
        return (t.empty((nsteps, self.nwalkers, self.ndim), dtype=t.float64, device=self.device),
                t.empty((nsteps, self.nwalkers), dtype=t.float64, device=self.device))

    def _advance(self, nsteps, chain=None, lps=None, row=0):
        """nsteps steps; with ``chain``, rows row, row + 1, ... of chain / lps receive the state after each step."""
        for it in range(nsteps):
            self._half(0)
            self._half(1)
            self.step += 1
            if chain is not None:
                self.sync()
                chain[row + it].copy_(self.coords)
                lps[row + it].copy_(self.lnp)

    def run_until_converged(self, max_steps, check_every=100, n_tau=50, tau_rtol=0.01, c=5):
        """Run until the chain has converged, as emcee's "monitoring convergence" recipe does: every ``check_every``
        steps the integrated autocorrelation time tau of the chain so far is computed (without the length check), and
        the run stops once every parameter has ``step > n_tau * tau`` and ``|tau - tau_prev| / tau < tau_rtol`` (tau_prev:
        the previous check's; a NaN tau never passes).  Stops at ``max_steps`` otherwise.  The chain is stored in one
        ``[max_steps, nwalkers, ndim]`` buffer on the ensemble's device; tau comes from ``integrated_time_device``
        there, from ``integrated_time`` for a CPU ensemble.  With ``dist`` every rank decides from its full replica
        and the decision is all-reduced, so all ranks stop at the same step.

        Returns ``(chain[:n], lnp[:n], tau_history [n_checks, ndim], converged)``; the chain is that of ``run(n)``."""
        from .synthetic.synth_mcmc import integrated_time, integrated_time_device
        max_steps, check_every = int(max_steps), int(check_every)
        if max_steps < 1 or check_every < 1:
            raise ValueError("max_steps and check_every must be positive")
        t = self.torch
        chain, lps = self._buffers(max_steps)
        history, tau_prev, converged, n = [], np.full(self.ndim, np.inf), False, 0
        while n < max_steps and not converged:
            k = min(check_every, max_steps - n)
            self._advance(k, chain, lps, n)
            n += k
            if n % check_every:
                break
            if self.device.type == "cuda":
                tau = integrated_time_device(chain[:n], c=c, quiet=True)
            else:
                tau = integrated_time(chain[:n].numpy(), c=c, quiet=True)
            history.append(tau)
            with np.errstate(invalid="ignore", divide="ignore"):
                ok = bool(np.all(n > n_tau * tau) and np.all(np.abs(tau_prev - tau) / tau < tau_rtol))
            if self.dist:
                flag = t.tensor([int(ok)], dtype=t.int32, device=self.device)
                self.dist.all_reduce(flag, op=self.dist.ReduceOp.MIN)
                ok = bool(flag.item())
            converged, tau_prev = ok, tau
        self.sync()
        return chain[:n], lps[:n], np.array(history).reshape(len(history), self.ndim), converged

    def check_peers(self):
        """Raise if a cross-GPU barrier timed out (a peer died)."""
        if self.exchange == "peer" and int(self._error.cpu()[0]) != 0:
            raise RuntimeError("DeviceEnsemble: a peer did not reach the half-step barrier within 10 s")

    def acceptance_fraction(self):
        acc = self.accepted.clone()
        if self.dist:
            self.dist.all_reduce(acc)
        return acc.double() / max(1, self.step)

    def drain_bad(self):
        """Proposals whose likelihood was not finite since the last call -- the rows the reference appends to
        ``{GRB}_bad.csv`` (mcmc_eqns.py:72-79) -- as a NumPy array [k, ndim] (all ranks' rows on every rank).
        Returns (rows, dropped): `dropped` counts rows beyond the device log's capacity."""
        n = int(self.bad_count.cpu()[0])
        rows = self.bad_rows[:min(n, self.BAD_CAPACITY)].cpu().numpy().copy()
        dropped = max(0, n - self.BAD_CAPACITY)
        self.bad_count.zero_()
        if self.dist:
            parts = [None] * self.world
            self.dist.all_gather_object(parts, (rows, dropped))
            rows = np.concatenate([p[0] for p in parts], axis=0)
            dropped = sum(p[1] for p in parts)
        return rows, dropped


def _ladder(betas):
    """betas as a float64 array, checked: 1-D, 1 <= T <= MP_MAX_TEMPS, betas[0] == 1, strictly decreasing, all > 0."""
    from ._capi import MP_MAX_TEMPS
    b = np.ascontiguousarray(betas, dtype=np.float64)
    if b.ndim != 1 or not 1 <= b.size <= MP_MAX_TEMPS:
        raise ValueError(f"betas must be a 1-D array of 1 to {MP_MAX_TEMPS} inverse temperatures")
    if b[0] != 1.0 or not (b > 0.0).all() or not (np.diff(b) < 0.0).all():
        raise ValueError("betas must start at 1, decrease strictly and stay positive")
    return b


def geometric_betas(ntemps, beta_min):
    """A geometric ladder of ``ntemps`` inverse temperatures from 1 down to ``beta_min`` (both included)."""
    ntemps = int(ntemps)
    if ntemps < 1:
        raise ValueError("ntemps must be positive")
    if ntemps == 1:
        return np.ones(1)
    if not 0.0 < beta_min < 1.0:
        raise ValueError("beta_min must lie in (0, 1)")
    b = np.geomspace(1.0, float(beta_min), ntemps)
    b[0], b[-1] = 1.0, float(beta_min)
    return _ladder(b)


def _ti_log_beta(b, mean_lnl):
    """int_0^1 <lnL>_beta dbeta: the trapezoid rule in ln(beta) on beta <lnL>_beta over the (descending) ladder, plus
    beta_min <lnL>_{beta_min} for [0, beta_min]."""
    f, x = b * mean_lnl, np.log(b)
    return float(np.sum(0.5 * (f[:-1] + f[1:]) * (x[:-1] - x[1:])) + b[-1] * mean_lnl[-1])


def thermodynamic_log_evidence(betas, lnp, discard=0):
    """ln Z = int_0^1 <lnL>_beta dbeta from the stored log-probabilities of a tempered run, ``lnp`` [nsteps, T, n] (as
    ``TemperedEnsemble.run`` returns it; NumPy or torch).  <lnL>_beta is the mean of temperature beta's lnp over the
    steps after ``discard`` and all walkers -- lnp is lnlike + lnprior, which is lnlike inside a top-hat prior.  The
    integral is the trapezoid rule in ln(beta) on beta <lnL>_beta, plus beta_min <lnL>_{beta_min} for [0, beta_min]
    (ptemcee's appended zero).  In ln(beta) a ladder that spans decades is integrated far better than in beta: on a
    3-D Gaussian in a box with 32 geometric temperatures down to 1e-6 the plain-beta trapezoid is 0.13 nats off, this
    rule 0.045.  The error estimate is |ln Z - the same rule on every other temperature|, as ptemcee's.  (ptemcee is
    not installed here: these conventions follow its source, not a test against it.)  Returns (ln Z, d ln Z)."""
    b = _ladder(betas)
    if b.size < 2:
        raise ValueError("thermodynamic integration needs at least two temperatures")
    if hasattr(lnp, "cpu"):
        lnp = lnp.cpu().numpy()
    lnp = np.asarray(lnp, dtype=np.float64)
    if lnp.ndim != 3 or lnp.shape[1] != b.size:
        raise ValueError("lnp must be [nsteps, ntemps, nwalkers] with ntemps == len(betas)")
    kept = lnp[int(discard):]
    if kept.shape[0] == 0:
        raise ValueError("no steps left after discard")
    if not np.isfinite(kept).all():
        raise ValueError("lnp holds non-finite values: <lnL> is undefined")
    mean = kept.mean(axis=(0, 2))
    log_z = _ti_log_beta(b, mean)
    return log_z, abs(log_z - _ti_log_beta(b[::2], mean[::2]))


class TemperedEnsemble(DeviceEnsemble):
    """Parallel-tempered ensemble on one device (emcee 2's ``PTSampler``, continued by ptemcee): ``ntemps =
    len(betas)`` temperatures of ``nwalkers`` walkers each, rows ``t*nwalkers + w`` of ``coords`` / ``lnp``.  Every
    temperature is an ensemble moved as ``DeviceEnsemble`` moves one, accepting on ``beta_t * lnp``; all temperatures
    move in one launch per half-step, and once per step walker j of each temperature may swap places with walker j
    of the next colder one, from the hottest pair down (semantics: ``mp_tempered_half_step`` / ``mp_tempered_swap``
    in include/magprop_b200.h).  ``lnp`` is untempered.  One device only: ``dist`` raises ``ValueError``.  ``moves`` as
    for ``DeviceEnsemble``: the step's move is the same for every temperature.
    ``backend`` as for ``DeviceEnsemble``, with ``tempered_half_step`` and ``tempered_swap``."""

    def __init__(self, backend, nwalkers, ndim, betas, a=2.0, seed=0, device="cuda", randomize_split=True, dist=None,
                 moves=None):
        import torch
        if dist is not None:
            raise ValueError("a tempered ensemble runs on one device: dist is not supported")
        self.betas = _ladder(betas)
        self.ntemps = self.betas.size
        if self.ntemps * nwalkers >= 1 << 31:
            raise ValueError("ntemps * nwalkers must be below 2^31")
        super().__init__(backend, nwalkers, ndim, a=a, seed=seed, device=device, randomize_split=randomize_split,
                         moves=moves)
        self.swap_accepted = torch.zeros(self.ntemps - 1, dtype=torch.int32, device=self.device)

    @classmethod
    def from_likelihood(cls, lik, nwalkers, ndim, betas, a=2.0, seed=0, randomize_split=True, dist=None, moves=None):
        import torch
        ens = cls(CudaBackend(lik), nwalkers, ndim, betas, a=a, seed=seed, device=torch.device("cuda", lik.device),
                  randomize_split=randomize_split, dist=dist, moves=moves)
        ens._lik = lik
        return ens

    def initialise(self, p0):
        """Positions from p0 -- [ntemps, nwalkers, ndim], or [nwalkers, ndim] for every temperature -- and their lnprob."""
        p0 = np.asarray(p0, dtype=np.float64)
        T, n, d = self.ntemps, self.nwalkers, self.ndim
        if p0.shape == (n, d):
            p0 = np.repeat(p0[None], T, axis=0)
        elif p0.shape != (T, n, d):
            raise ValueError(f"p0 must be [{T}, {n}, {d}] or [{n}, {d}]")
        super().initialise(p0.reshape(T * n, d))

    def run(self, nsteps, store=True):
        """nsteps tempered steps: half-steps 0 and 1 of every temperature, then the swaps.  With ``store`` returns the
        cold chain [nsteps, nwalkers, ndim] and the lnp of every temperature [nsteps, ntemps, nwalkers], both as they
        stand after the step's swaps."""
        chain, lps = self._buffers(nsteps) if store else (None, None)
        self._advance(nsteps, chain, lps, 0)
        return (chain, lps) if store else None

    def _buffers(self, nsteps):
        chain, _ = super()._buffers(nsteps)
        return chain, self.torch.empty((nsteps, self.ntemps, self.nwalkers), dtype=self.torch.float64, device=self.device)

    def _advance(self, nsteps, chain=None, lps=None, row=0):
        for it in range(nsteps):
            self.backend.tempered_half_step(self, self.step, 0)
            self.backend.tempered_half_step(self, self.step, 1)
            self.backend.tempered_swap(self, self.step)
            self.step += 1
            if chain is not None:
                chain[row + it].copy_(self.coords[:self.nwalkers])
                lps[row + it].copy_(self.lnp.view(self.ntemps, self.nwalkers))

    def run_until_converged(self, *args, **kwargs):
        raise NotImplementedError("tempered runs do not stop on convergence; integrated_time_device gives tau of the "
                                  "cold chain run() returns")

    def acceptance_fraction(self):
        """Accepted stretch moves per step, [ntemps, nwalkers]."""
        return super().acceptance_fraction().view(self.ntemps, self.nwalkers)

    def swap_acceptance_fraction(self):
        """Accepted swaps per step and column of each adjacent pair (t-1, t), [ntemps - 1]."""
        return self.swap_accepted.double() / (max(1, self.step) * self.nwalkers)


def run_concurrently(ensembles, nsteps, store=False):
    """Advance several independent device ensembles (e.g. one per dataset / burst) ``nsteps`` steps each, every
    ensemble on its own CUDA stream with the launches interleaved step by step, so that small ensembles --
    which are latency-bound, a few warps each -- share the GPU instead of queueing behind one another.
    (Ensembles on ONE likelihood handle are fine: the library keeps a stiff queue per stream.)
    Returns a list of (chain, lnprob) per ensemble when ``store`` (else None)."""
    import torch
    streams = [torch.cuda.Stream(device=e.device) for e in ensembles]
    for e, st in zip(ensembles, streams):
        st.wait_stream(torch.cuda.current_stream(e.device))
    out = [e._buffers(nsteps) if store else (None, None) for e in ensembles]
    for it in range(nsteps):
        for e, st, (chain, lps) in zip(ensembles, streams, out):
            with torch.cuda.stream(st):
                e._advance(1, chain, lps, it)
    for e, st in zip(ensembles, streams):
        torch.cuda.current_stream(e.device).wait_stream(st)
    return out if store else None
