"""Device-resident affine-invariant ensemble sampler (stretch move).

Replaces ``emcee.EnsembleSampler`` + its default ``StretchMove(a=2)`` for the drivers' call
sites (emcee/emcee_radex.py:483-499, emcee/emcee_radex_2comp.py:557-574; SURVEY.md 3.5): walkers,
log-probabilities, proposals and the accept test live on the GPU; ``lnprob`` is the fused
kernel (or the solve pipeline) of libradex_b200; nothing crosses PCIe per step.

Red/blue split
  emcee's default ``randomize_split=True`` draws a new balanced random labelling of the walkers every
  step.  Here the labelling is a keyed bijection evaluated per BLOCK of ``split_block`` consecutive
  walkers from (seed, step, block) -- see ``csrc/stretch.cuh`` -- so every rank can evaluate it for any
  walker without communication.  ``randomize_split=False`` is the parity split (even ids / odd ids).

Sub-ensembles (BASELINE.json configs[3], all sources of flux.dat fitted concurrently)
  ``nsources`` independent ensembles of ``nwalkers // nsources`` walkers share one state array; a
  walker's partner is drawn from the complementary half of its own sub-ensemble and its log-probability
  is evaluated against its own source (``CudaEngine`` over several ``SLEDModel``s: one fused launch
  with a per-walker source row).

Sharding
  With G ranks, rank r owns the contiguous global ids [r N/G, (r+1) N/G).  Per half-step each rank
  needs the *positions* of the whole complementary half: one ``all_gather_into_tensor`` (NCCL over
  NVLink on GPUs, gloo on CPU) of (N/2G) x ndim doubles per rank.  The Philox streams are keyed by
  (seed, step, half, global id) and the gathered half is in global slot order, so the chain is
  independent of G.  On one GPU the whole loop runs inside the library (``rb_stretch_run_dev``; small
  ensembles replay a CUDA graph of one step) -- same kernels, same chain.

Posterior statistics where the chain lives
  ``get_quantiles`` (exact ``np.percentile`` of every source's flattened chain) and ``get_autocorr_time``
  (emcee's integrated autocorrelation time) read the stored chain in place on every rank (csrc/chain_stats.cuh):
  only 256-bin digit histograms and per-lag sums cross ranks (``all_reduce``) and PCIe, never the chain.

The arithmetic is behind an ``engine`` object so that the host logic (sharding, gather order,
bookkeeping) can be exercised on CPU by the test-suite's engine (tests/ref_engine.py); the
package itself only ships the CUDA engine -- there is no CPU fallback in the product path.
"""
from __future__ import annotations

import ctypes as C
import logging

import numpy as np
import torch

from . import _lib

logger = logging.getLogger("radex_emcee_b200.sampler")

ACF_LAG_BLOCK = 128            # lags per rb_chain_acf_dev call; get_autocorr_time stops once every window is found
NO_PREFIX = np.uint64(0xFFFFFFFFFFFFFFFF)


class AutocorrError(Exception):
    """emcee's ``AutocorrError``: the chain is shorter than ``tol`` integrated autocorrelation times.  ``tau`` holds
    the estimate (in thinned steps, as emcee's ``integrated_time`` returns it)."""

    def __init__(self, tau, *args, **kwargs):
        self.tau = tau
        super().__init__(*args, **kwargs)


class ChainView:
    """One rank's stored chain as the chain-statistics kernels read it (rb_chain_view): chunks [steps_i, nlocal, ndim]
    in place, and emcee's ``discard`` / ``thin`` over the concatenated step index (steps discard + thin - 1,
    discard + 2 thin - 1, ...)."""

    def __init__(self, chunks, nlocal, ndim, gid_base, walkers_per_source, discard, thin):
        self.chunks = list(chunks)
        self.nlocal, self.ndim, self.gid_base = int(nlocal), int(ndim), int(gid_base)
        self.walkers_per_source, self.discard, self.thin = int(walkers_per_source), int(discard), int(thin)
        if self.discard < 0 or self.thin < 1:
            raise ValueError("discard must be >= 0 and thin >= 1")
        self.nsteps = sum(int(c.shape[0]) for c in self.chunks)
        self.nsel = len(range(self.discard + self.thin - 1, self.nsteps, self.thin))

    def c_struct(self):
        if len(self.chunks) > _lib.RB_MAX_CHUNKS:
            raise ValueError("at most %d chunks" % _lib.RB_MAX_CHUNKS)
        v = _lib.rb_chain_view()
        for k, c in enumerate(self.chunks):
            if not c.is_contiguous() or tuple(c.shape[1:]) != (self.nlocal, self.ndim) or c.dtype != torch.float64:
                raise ValueError("chain chunks must be contiguous float64 [steps, nlocal, ndim]")
            v.chunk[k] = c.data_ptr()
            v.steps[k] = int(c.shape[0])
        v.nchunks, v.ndim, v.nlocal, v.gid_base = len(self.chunks), self.ndim, self.nlocal, self.gid_base
        v.walkers_per_source, v.discard, v.thin = self.walkers_per_source, self.discard, self.thin
        return v


def _distinct_prefixes(pre):
    """pre [..., m] uint64 -> (table [..., P] of the distinct prefixes, padded with NO_PREFIX; slot [..., m] of each)."""
    order = np.argsort(pre, axis=-1, kind="stable")
    srt = np.take_along_axis(pre, order, axis=-1)
    new = np.ones(srt.shape, dtype=bool)
    new[..., 1:] = srt[..., 1:] != srt[..., :-1]
    rank = np.cumsum(new, axis=-1) - 1
    table = np.full(pre.shape[:-1] + (int(rank.max()) + 1,), NO_PREFIX, dtype=np.uint64)
    np.put_along_axis(table, rank, srt, axis=-1)
    slot = np.empty_like(rank)
    np.put_along_axis(slot, order, rank, axis=-1)
    return table, slot


def _key_to_double(key):
    """Inverse of the kernels' order-preserving key (csrc/chain_stats.cuh order_key)."""
    key = np.asarray(key, dtype=np.uint64)
    neg = (key >> np.uint64(63)) == 0
    return np.where(neg, ~key, key ^ np.uint64(1 << 63)).view(np.float64)


class SLEDModel:
    """Everything the lnprob kernels need for one source."""

    def __init__(self, ncomp, Jup, flux, eflux, bounds, tbg, T_d=None, opts=None):
        if ncomp not in (1, 2):
            raise ValueError("ncomp must be 1 or 2")
        self.ncomp = ncomp
        self.ndim = 4 * ncomp
        self.Jup = np.asarray(Jup, dtype=np.int64)
        self.flux = np.asarray(flux, dtype=np.float64)
        self.eflux = np.asarray(eflux, dtype=np.float64)
        self.bounds = np.ascontiguousarray(bounds, dtype=np.float64)
        if self.bounds.shape != (self.ndim, 2):
            raise ValueError("bounds must have shape (%d, 2)" % self.ndim)
        self.tbg = float(tbg)
        self.T_d = None if T_d is None else float(T_d)
        self.opts = opts


class SplitSpec:
    """The red/blue split of an ensemble (rb_split of the C ABI)."""

    def __init__(self, nwalkers, walkers_per_source, block, randomize, seed):
        self.nwalkers, self.walkers_per_source, self.block = int(nwalkers), int(walkers_per_source), int(block)
        self.randomize, self.seed = bool(randomize), int(seed)
        if self.nwalkers % self.walkers_per_source or self.walkers_per_source % self.block or self.block % 2:
            raise ValueError("need split_block | walkers per source | nwalkers and an even split_block")

    def c_struct(self):
        return _lib.rb_split(self.nwalkers, self.walkers_per_source, self.block, int(self.randomize), 0, self.seed)


def default_split_block(walkers_per_source, randomize):
    """Blocks the split is balanced over.  The chain depends on it, so the rule only looks at the
    ensemble: an eighth of a large sub-ensemble (any rank count up to 8 owns whole blocks), the whole
    sub-ensemble otherwise (exactly emcee's balanced random labelling)."""
    if not randomize:
        return 2
    W = int(walkers_per_source)
    return W // 8 if (W >= 1024 and W % 16 == 0) else W


class CudaEngine:
    """Stretch-move + lnprob arithmetic on one GPU through the C ABI (device pointers).
    ``model``: one SLEDModel, or a list of them (one per source, same ncomp)."""

    def __init__(self, ctx: _lib.Context, model):
        if not torch.cuda.is_available():
            raise _lib.RadexB200Error("CudaEngine needs a CUDA device; there is no CPU fallback")
        self.ctx = ctx
        self.models = list(model) if isinstance(model, (list, tuple)) else [model]
        self.model = self.models[0]
        if any(m.ncomp != self.model.ncomp for m in self.models):
            raise ValueError("all sources of one ensemble must have the same number of components")
        self.device = torch.device("cuda", ctx.device)
        self.L = _lib.load()
        self.obs = _lib.make_obs(self.model.Jup, self.model.flux, self.model.eflux)
        self.opts = self.model.opts if self.model.opts is not None else _lib.default_opts()
        self.srcset = _lib.SourceSet(ctx, self.model.ncomp,
                                     [_lib.make_source(m.ncomp, m.Jup, m.flux, m.eflux, m.bounds, m.tbg, m.T_d)
                                      for m in self.models])
        self.nsolves = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.total_solves = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.launches = 0

    def _bind_stream(self):
        self.ctx.set_stream(torch.cuda.current_stream(self.device).cuda_stream)

    def lnprob(self, P: torch.Tensor, src_id=None) -> torch.Tensor:
        self._bind_stream()
        n = P.shape[0]
        out = torch.empty(n, dtype=torch.float64, device=self.device)
        if len(self.models) > 1 and src_id is None:
            raise ValueError("src_id is required with more than one source")
        _lib.check(self.L.rb_lnprob_src_dev(self.ctx.handle, self.srcset.handle, n, P.data_ptr(),
                                            src_id.data_ptr() if src_id is not None else None, C.byref(self.opts),
                                            out.data_ptr(), self.nsolves.data_ptr()))
        self.total_solves += self.nsolves
        self.launches += 1
        return out

    # ---- first form of the C ABI (separate half arrays, parity split) -------------------------------
    def propose(self, S, Cpos, a, seed, step, half, gid0, gid_stride):
        self._bind_stream()
        ns, ndim = S.shape
        Q = torch.empty_like(S)
        logfac = torch.empty(ns, dtype=torch.float64, device=self.device)
        _lib.check(self.L.rb_stretch_propose_dev(self.ctx.handle, ns, ndim, S.data_ptr(), Cpos.shape[0], Cpos.data_ptr(),
                                                 a, seed, step, half, gid0, gid_stride, Q.data_ptr(), logfac.data_ptr()))
        self.launches += 1
        return Q, logfac

    def accept(self, S, lnp, Q, lnp_new, logfac, seed, step, half, gid0, gid_stride, naccept):
        self._bind_stream()
        ns, ndim = S.shape
        _lib.check(self.L.rb_stretch_accept_dev(self.ctx.handle, ns, ndim, S.data_ptr(), lnp.data_ptr(), Q.data_ptr(),
                                                lnp_new.data_ptr(), logfac.data_ptr(), seed, step, half, gid0,
                                                gid_stride, naccept.data_ptr()))
        self.launches += 1

    # ---- second form: the ensemble stays in place -----------------------------------------------------
    def pack(self, split, step, half, gid_base, X):
        self._bind_stream()
        nlocal, ndim = X.shape
        out = torch.empty((nlocal // 2, ndim), dtype=torch.float64, device=self.device)
        sp = split.c_struct()
        _lib.check(self.L.rb_stretch_pack_dev(self.ctx.handle, C.byref(sp), step, half, gid_base, nlocal, ndim,
                                              X.data_ptr(), out.data_ptr()))
        self.launches += 1
        return out

    def propose2(self, split, step, half, gid_base, X, Call, a):
        self._bind_stream()
        nlocal, ndim = X.shape
        Q = torch.empty((nlocal // 2, ndim), dtype=torch.float64, device=self.device)
        logfac = torch.empty(nlocal // 2, dtype=torch.float64, device=self.device)
        src_id = torch.empty(nlocal // 2, dtype=torch.int32, device=self.device)
        sp = split.c_struct()
        _lib.check(self.L.rb_stretch_propose2_dev(self.ctx.handle, C.byref(sp), step, half, gid_base, nlocal, ndim,
                                                  X.data_ptr(), Call.data_ptr(), a, Q.data_ptr(), logfac.data_ptr(),
                                                  src_id.data_ptr()))
        self.launches += 1
        return Q, logfac, src_id

    def accept2(self, split, step, half, gid_base, X, lnp, Q, lnp_new, logfac, naccept, counters):
        self._bind_stream()
        nlocal, ndim = X.shape
        sp = split.c_struct()
        _lib.check(self.L.rb_stretch_accept2_dev(self.ctx.handle, C.byref(sp), step, half, gid_base, nlocal, ndim,
                                                 X.data_ptr(), lnp.data_ptr(), Q.data_ptr(), lnp_new.data_ptr(),
                                                 logfac.data_ptr(), naccept.data_ptr(), counters.data_ptr()))
        self.launches += 1

    # ---- chain statistics (csrc/chain_stats.cuh) -------------------------------------------------------
    def chain_hist(self, view, nsrc, cols, pass_, prefix):
        """One digit pass: counts [nsrc, ncol, nprefix, 256] (int64) for the prefixes [nsrc, ncol, nprefix] (uint64)
        and, on pass 0, NaN counts [nsrc, ncol]."""
        self._bind_stream()
        ncol, P = len(cols), prefix.shape[2]
        ci = (C.c_int32 * ncol)(*[i for i, _ in cols])
        cj = (C.c_int32 * ncol)(*[j for _, j in cols])
        pre = torch.from_numpy(np.ascontiguousarray(prefix, dtype=np.uint64).view(np.int64)).to(self.device)
        counts = torch.zeros((nsrc, ncol, P, 256), dtype=torch.int64, device=self.device)
        nans = torch.zeros((nsrc, ncol), dtype=torch.int64, device=self.device) if pass_ == 0 else None
        vs = view.c_struct()
        _lib.check(self.L.rb_chain_hist_dev(self.ctx.handle, C.byref(vs), nsrc, ncol, ci, cj, pass_, P, pre.data_ptr(),
                                            counts.data_ptr(), nans.data_ptr() if nans is not None else None))
        self.launches += 1
        return counts, nans

    def chain_moments(self, view):
        self._bind_stream()
        mean = torch.empty((view.nlocal, view.ndim), dtype=torch.float64, device=self.device)
        c0 = torch.empty_like(mean)
        vs = view.c_struct()
        _lib.check(self.L.rb_chain_moments_dev(self.ctx.handle, C.byref(vs), mean.data_ptr(), c0.data_ptr()))
        self.launches += 1
        return mean, c0

    def chain_acf(self, view, nsrc, mean, c0, k0, k1):
        """[nsrc, k1 - k0, ndim]: sum over each source's local walkers of c_k / c_0."""
        self._bind_stream()
        out = torch.empty((nsrc, k1 - k0, view.ndim), dtype=torch.float64, device=self.device)
        vs = view.c_struct()
        _lib.check(self.L.rb_chain_acf_dev(self.ctx.handle, C.byref(vs), nsrc, mean.data_ptr(), c0.data_ptr(), k0, k1,
                                           out.data_ptr()))
        self.launches += 1
        return out

    def run_native(self, split, a, step0, nsteps, X, lnp, naccept, counters, thin, chain, lnp_chain):
        """nsteps steps of the whole (single-rank) ensemble inside the library."""
        self._bind_stream()
        sp = split.c_struct()
        _, l0 = self.ctx.counters()
        _lib.check(self.L.rb_stretch_run_dev(self.ctx.handle, self.srcset.handle, C.byref(sp), a, step0, nsteps,
                                             C.byref(self.opts), X.data_ptr(), lnp.data_ptr(), naccept.data_ptr(),
                                             counters.data_ptr(), thin,
                                             chain.data_ptr() if chain is not None else None,
                                             lnp_chain.data_ptr() if lnp_chain is not None else None))
        self.launches += self.ctx.counters()[1] - l0


def walkers_independent(coords):
    """emcee's check of an initial ensemble (ensemble.py, ``walkers_independent``): finite, no degenerate
    dimension, condition number of the normalised, centred coordinates <= 1e8."""
    coords = np.asarray(coords, dtype=np.float64)
    if not np.all(np.isfinite(coords)):
        return False
    Cm = coords - np.mean(coords, axis=0)[None, :]
    colmax = np.amax(np.abs(Cm), axis=0)
    if np.any(colmax == 0):
        return False
    Cm = Cm / colmax
    Cm = Cm / np.sqrt(np.sum(Cm ** 2, axis=0))
    return bool(np.linalg.cond(Cm) <= 1e8)


class StretchSampler:
    """``EnsembleSampler``-like driver: ``run_mcmc``, ``get_chain``, ``get_log_prob``, ``reset``,
    ``acceptance_fraction`` (per walker, like emcee), ``get_autocorr_time``, and ``get_quantiles`` (exact
    percentiles of the stored chain without moving it)."""

    def __init__(self, nwalkers, ndim, engine, a=2.0, seed=0, group=None, randomize_split=True, nsources=1,
                 split_block=None, native=True, time_gather=False):
        self.dist = torch.distributed if (torch.distributed.is_available() and torch.distributed.is_initialized()) else None
        self.group = group
        self.world = self.dist.get_world_size(group) if self.dist else 1
        self.rank = self.dist.get_rank(group) if self.dist else 0
        nwalkers, nsources = int(nwalkers), int(nsources)
        if nwalkers % (2 * self.world) != 0:
            raise ValueError("nwalkers must be a multiple of 2*world_size")
        if nsources < 1 or nwalkers % nsources or (nwalkers // nsources) % 2:
            raise ValueError("nwalkers must be an even multiple of nsources")
        if nwalkers // nsources < 2 * ndim:
            raise ValueError("emcee requires nwalkers >= 2*ndim")
        self.nwalkers, self.ndim, self.nsources = nwalkers, int(ndim), nsources
        self.engine = engine
        self.device = engine.device
        self.a = float(a)
        self.seed = int(seed)
        self.nlocal = self.nwalkers // self.world          # walkers owned by this rank: global ids gid_base ...
        self.gid_base = self.rank * self.nlocal
        W = self.nwalkers // nsources
        block = int(split_block) if split_block else default_split_block(W, randomize_split)
        self.split = SplitSpec(self.nwalkers, W, block, randomize_split, self.seed)
        if self.nlocal % block:
            raise ValueError("every rank must own whole split blocks: nwalkers/world_size = %d is not a multiple of "
                             "split_block = %d (pass split_block, or randomize_split=False)" % (self.nlocal, block))
        self.native = bool(native) and self.world == 1 and hasattr(engine, "run_native")
        self.time_gather = bool(time_gather)
        self._gather_events = []
        self.step = 0
        self.X = None                                       # [nlocal, ndim]
        self.lnp = None                                     # [nlocal]
        self.naccept = torch.zeros(self.nlocal, dtype=torch.int64, device=self.device)
        self.counters = torch.zeros(2, dtype=torch.int64, device=self.device)     # NaN log-probabilities, solves
        self.reset()

    # ---- storage --------------------------------------------------------------------------------
    def reset(self):
        self._chain, self._lnp_chain = [], []
        self.naccept.zero_()
        self.nsteps_done = 0

    def _gather(self, t: torch.Tensor) -> torch.Tensor:
        if self.world == 1:
            return t
        out = torch.empty((self.world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        if self.time_gather and t.is_cuda:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            self.dist.all_gather_into_tensor(out, t.contiguous(), group=self.group)
            e1.record()
            self._gather_events.append((e0, e1))
        else:
            self.dist.all_gather_into_tensor(out, t.contiguous(), group=self.group)
        return out

    def gather_ms(self):
        """Device time spent in the all-gathers since the last call (needs time_gather=True)."""
        ms = sum(a.elapsed_time(b) for a, b in self._gather_events)
        self._gather_events = []
        return ms

    def _src_of_local(self):
        gid = self.gid_base + torch.arange(self.nlocal, device=self.device)
        return (gid // self.split.walkers_per_source).to(torch.int32)

    def set_state(self, p0, check=True):
        """p0: global (nwalkers, ndim) array, identical on every rank."""
        p0 = np.asarray(p0, dtype=np.float64)
        if p0.shape != (self.nwalkers, self.ndim):
            raise ValueError("p0 must have shape (nwalkers, ndim)")
        W = self.split.walkers_per_source
        if check:
            for s in range(self.nsources):
                if not walkers_independent(p0[s * W:(s + 1) * W]):
                    raise ValueError("Initial state has a large condition number. Make sure that your walkers are "
                                     "linearly independent for the best performance")
        loc = np.array(p0[self.gid_base:self.gid_base + self.nlocal], dtype=np.float64, order="C", copy=True)   # never alias the caller's array
        self.X = torch.from_numpy(loc).to(self.device)
        self.lnp = self.engine.lnprob(self.X, self._src_of_local() if self.nsources > 1 else None)
        if bool(torch.isnan(self.lnp).any()):      # emcee: "Probability function returned NaN"; -inf is allowed
            raise ValueError("Probability function returned NaN")

    # ---- the move -------------------------------------------------------------------------------
    def _half_step(self, half):
        eng, sp = self.engine, self.split
        Call = self._gather(eng.pack(sp, self.step, 1 - half, self.gid_base, self.X))
        Q, logfac, src_id = eng.propose2(sp, self.step, half, self.gid_base, self.X, Call, self.a)
        lnp_new = eng.lnprob(Q, src_id if self.nsources > 1 else None)
        eng.accept2(sp, self.step, half, self.gid_base, self.X, self.lnp, Q, lnp_new, logfac, self.naccept,
                    self.counters)

    def run_mcmc(self, p0, nsteps, store=True, thin=1):
        if p0 is not None:
            self.set_state(p0)
        if self.X is None:
            raise ValueError("no initial state")
        nsteps, thin = int(nsteps), int(thin)
        if self.native and nsteps > 0:
            # `thin` counts from this call's first step in the library; keep it aligned with nsteps_done
            nstore = (self.nsteps_done + nsteps) // thin - self.nsteps_done // thin if store else 0
            aligned = self.nsteps_done % thin == 0
            if store and nstore and aligned:
                chain = torch.empty((nstore, self.nlocal, self.ndim), dtype=torch.float64, device=self.device)
                lchain = torch.empty((nstore, self.nlocal), dtype=torch.float64, device=self.device)
            else:
                chain = lchain = None
            if not store or aligned:
                self.engine.run_native(self.split, self.a, self.step, nsteps, self.X, self.lnp, self.naccept,
                                       self.counters, thin, chain, lchain)
                self.step += nsteps
                self.nsteps_done += nsteps
                if chain is not None:
                    self._chain.append(chain)
                    self._lnp_chain.append(lchain)
                self._check_nan()
                return None
        # one chunk per call, as in the native loop: the chain-statistics kernels take at most RB_MAX_CHUNKS chunks
        nstore = (self.nsteps_done + nsteps) // thin - self.nsteps_done // thin if store else 0
        chain = torch.empty((nstore, self.nlocal, self.ndim), dtype=torch.float64, device=self.device)
        lchain = torch.empty((nstore, self.nlocal), dtype=torch.float64, device=self.device)
        k = 0
        try:
            for _ in range(nsteps):
                self._half_step(0)
                self._half_step(1)
                self.step += 1
                self.nsteps_done += 1
                if store and (self.nsteps_done % thin == 0):
                    chain[k].copy_(self.X)
                    lchain[k].copy_(self.lnp)
                    k += 1
        finally:
            if k:
                self._chain.append(chain[:k])
                self._lnp_chain.append(lchain[:k])
        self._check_nan()
        return None

    def _check_nan(self):
        if int(self.counters[0].item()) > 0:
            raise ValueError("Probability function returned NaN")

    # ---- results --------------------------------------------------------------------------------
    def get_last_sample(self):
        """(positions (nwalkers, ndim), lnprob (nwalkers,)) gathered over ranks, as numpy."""
        return self._gather(self.X).cpu().numpy(), self._gather(self.lnp).cpu().numpy()

    def _stacked(self, parts, tail, discard, thin):
        discard, thin = int(discard), int(thin)
        if discard < 0 or thin < 1:
            raise ValueError("discard must be >= 0 and thin >= 1")
        if not parts:
            return np.empty((0, self.nwalkers) + tail)
        loc = torch.cat(parts)[discard + thin - 1::thin]     # steps, nlocal, ...  (emcee's selection)
        if self.world > 1:
            loc = self._gather(loc.transpose(0, 1).contiguous()).transpose(0, 1)
        return loc.cpu().numpy()

    def get_chain(self, flat=False, discard=0, thin=1):
        """(steps, nwalkers, ndim) like emcee v3's ``get_chain``: steps discard + thin - 1, discard + 2 thin - 1, ...
        Gathers the whole selection onto every rank and copies it to the host; for summaries of a large chain use
        ``get_quantiles`` / ``get_autocorr_time``, which leave it on the device."""
        c = self._stacked(self._chain, (self.ndim,), discard, thin)
        return c.reshape(-1, self.ndim) if flat else c

    def get_log_prob(self, flat=False, discard=0, thin=1):
        c = self._stacked(self._lnp_chain, (), discard, thin)
        return c.reshape(-1) if flat else c

    # ---- posterior statistics on the device -----------------------------------------------------------
    def _chain_view(self, discard, thin):
        if len(self._chain) > _lib.RB_MAX_CHUNKS:         # more run_mcmc calls than the kernels take chunks
            self._chain = [torch.cat(self._chain)]
        return ChainView(self._chain, self.nlocal, self.ndim, self.gid_base, self.split.walkers_per_source, discard, thin)

    def _allreduce(self, t):
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group)
        return t

    def _columns(self, columns):
        cols = []
        for c in (range(self.ndim) if columns is None else columns):
            i, j = (c, -1) if isinstance(c, (int, np.integer)) else tuple(c)
            i, j = int(i), int(j)
            if not (0 <= i < self.ndim and -1 <= j < self.ndim) or (j == -1 and not isinstance(c, (int, np.integer))):
                raise ValueError("a column is a parameter index or a pair of them, in [0, %d)" % self.ndim)
            cols.append((i, j))
        if not 1 <= len(cols) <= _lib.RB_CHAIN_MAX_COLS:
            raise ValueError("between 1 and %d columns" % _lib.RB_CHAIN_MAX_COLS)
        return cols

    def _order_statistics(self, view, cols, ranks):
        """Values of the given 0-based ranks (ascending) of every (source, column): [nsources, len(ranks), ncol], and
        which (source, column) holds a NaN.  Radix select, 8 digit passes over the chain per group of ranks."""
        S, ncol = self.nsources, len(cols)
        out = np.empty((S, len(ranks), ncol))
        has_nan = None
        per = max(1, _lib.RB_CHAIN_MAX_HIST // ncol)
        for g0 in range(0, len(ranks), per):
            m = len(ranks[g0:g0 + per])
            rem = np.broadcast_to(np.asarray(ranks[g0:g0 + per], dtype=np.int64), (S, ncol, m)).copy()
            pre = np.zeros((S, ncol, m), dtype=np.uint64)
            for p in range(8):
                if p == 0:
                    table, slot = np.zeros((S, ncol, 1), dtype=np.uint64), np.zeros((S, ncol, m), dtype=np.int64)
                else:
                    table, slot = _distinct_prefixes(pre)
                counts, nans = self.engine.chain_hist(view, S, cols, p, table)
                counts = self._allreduce(counts).cpu().numpy()
                if p == 0 and has_nan is None:
                    has_nan = self._allreduce(nans).cpu().numpy() > 0
                h = np.take_along_axis(counts, slot[..., None], axis=2)             # [S, ncol, m, 256]
                cum = np.cumsum(h, axis=-1)
                digit = np.minimum((cum <= rem[..., None]).sum(axis=-1), 255)      # (a NaN column holds fewer values)
                rem -= np.take_along_axis(cum - h, digit[..., None], axis=-1)[..., 0]
                pre = (pre << np.uint64(8)) | digit.astype(np.uint64)
            out[:, g0:g0 + m] = _key_to_double(pre).transpose(0, 2, 1)
        return out, has_nan

    def get_quantiles(self, q, discard=0, thin=1, columns=None):
        """Percentiles of the stored chain per source: [nsources, len(q), ncol], every value equal to
        ``np.percentile(get_chain(flat=True, discard=discard, thin=thin)[rows of the source], q, axis=0)`` (numpy's
        default 'linear' method; NaN where a column holds a NaN).  A column is a parameter index ``i`` or a pair
        ``(i, j)`` for x[i] + x[j]; the default is the ``ndim`` parameters.  The chain is read in place; only digit
        histograms cross ranks and PCIe.  The two order statistics around each percentile are exact (radix select on
        the device), and the interpolation between them is numpy's own arithmetic (numpy/lib/_function_base_impl.py:
        _quantile, _get_indexes, _get_gamma, _lerp)."""
        view = self._chain_view(discard, thin)
        cols = self._columns(columns)
        qq = np.true_divide(np.asarray(q, dtype=np.float64).reshape(-1), np.float64(100))
        if not (np.all(qq >= 0) and np.all(qq <= 1)):
            raise ValueError("Percentiles must be in the range [0, 100]")
        n = view.nsel * self.split.walkers_per_source
        if n == 0:
            raise ValueError("no stored samples are selected")
        v = (n - 1) * qq
        prev = np.floor(v)
        nxt = prev + 1
        above = v >= n - 1
        prev[above] = -1
        nxt[above] = -1
        gamma = np.asanyarray(v - prev, dtype=v.dtype)
        ip, inx = prev.astype(np.intp) % n, nxt.astype(np.intp) % n
        ranks = np.unique(np.concatenate([ip, inx]))
        xs, has_nan = self._order_statistics(view, cols, ranks)
        a, b = xs[:, np.searchsorted(ranks, ip)], xs[:, np.searchsorted(ranks, inx)]
        t = gamma[None, :, None]
        with np.errstate(invalid="ignore"):
            diff = np.subtract(b, a)
            out = np.asanyarray(np.add(a, diff * t))
            np.subtract(b, diff * (1 - t), out=out, where=t >= 0.5)
        out[np.broadcast_to(has_nan[:, None, :], out.shape)] = np.nan
        return out

    def _integrated_time(self, discard, thin, c):
        """emcee's integrated_time per (source, parameter) with the device acf: (tau in thinned steps, window, n_t)."""
        view = self._chain_view(discard, thin)
        n_t = view.nsel
        if n_t == 0:
            raise ValueError("no stored samples are selected")
        mean, c0 = self.engine.chain_moments(view)
        blocks, k1 = [], 0
        while True:
            k0, k1 = k1, min(n_t, k1 + ACF_LAG_BLOCK)
            rho = self._allreduce(self.engine.chain_acf(view, self.nsources, mean, c0, k0, k1))
            blocks.append(rho.cpu().numpy() / self.split.walkers_per_source)         # f: mean of rho over the walkers
            taus = 2.0 * np.cumsum(np.concatenate(blocks, axis=1), axis=1) - 1.0
            m = np.arange(k1)[None, :, None] < c * taus
            # emcee's auto_window is settled once m turns False after a True; a NaN series is False throughout
            settled = (m[:, 0] & (~m).any(axis=1)) | np.isnan(taus[:, 0])
            if k1 == n_t or settled.all():
                break
        window = np.where(m.any(axis=1), m.argmin(axis=1), n_t - 1)
        tau = np.take_along_axis(taus, np.minimum(window, k1 - 1)[:, None], axis=1)[:, 0]
        return np.where(window < k1, tau, np.nan), window, n_t

    def get_autocorr_time(self, discard=0, thin=1, c=5, tol=50, quiet=False):
        """Integrated autocorrelation time per (source, parameter), [nsources, ndim], in steps: emcee's
        ``get_autocorr_time`` / ``integrated_time`` (f = mean over the source's walkers of the normalised
        autocovariance, taus = 2 cumsum(f) - 1, emcee's auto_window with constant ``c``) with the autocovariance summed
        directly on the device.  Raises ``AutocorrError`` when tol * tau exceeds the number of selected steps (a
        warning only, with ``quiet``).  A walker whose chain is constant makes its source's tau NaN."""
        tau, _, n_t = self._integrated_time(discard, thin, c)
        flag = tol * tau > n_t
        if np.any(flag):
            msg = ("The chain is shorter than {0} times the integrated autocorrelation time for {1} parameter(s). Use this "
                   "estimate with caution and run a longer chain!\nN/{0} = {2:.0f};\ntau: {3}").format(
                       tol, int(np.sum(flag)), n_t / tol, tau)
            if not quiet:
                raise AutocorrError(tau, msg)
            logger.warning(msg)
        return thin * tau

    @property
    def acceptance_fraction(self):
        """Per walker, like ``EnsembleSampler.acceptance_fraction`` (shape (nwalkers,))."""
        n = self._gather(self.naccept)
        return n.cpu().numpy().astype(np.float64) / max(1, self.nsteps_done)

    @property
    def total_solves(self):
        return int(self.counters[1].item())
