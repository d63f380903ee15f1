"""Host protocol of the device chain statistics on CPU (sampler.get_quantiles / get_autocorr_time): a numpy engine
restates the three kernels of csrc/chain_stats.cuh, so that the radix-select narrowing, numpy's interpolation, the
all_reduce over ranks (gloo, world_size 2) and emcee's window logic are checked without a GPU; the new C entry points
refuse bad views and report the missing device."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import ref_engine
from radex_emcee_b200 import _lib
from radex_emcee_b200.sampler import NO_PREFIX, AutocorrError, ChainView, StretchSampler

QS = [0, 16, 50, 84, 100, 37.5]


class StatsEngine(ref_engine.NumpyEngine):
    """NumpyEngine plus numpy restatements of rb_chain_hist_dev / rb_chain_moments_dev / rb_chain_acf_dev."""

    @staticmethod
    def _selected(view):
        full = np.concatenate([c.numpy() for c in view.chunks]) if view.chunks else np.empty((0, view.nlocal, view.ndim))
        return full[view.discard + view.thin - 1::view.thin]

    @staticmethod
    def _sources(view):
        return (view.gid_base + np.arange(view.nlocal)) // view.walkers_per_source

    def chain_hist(self, view, nsrc, cols, pass_, prefix):
        X, src = self._selected(view), self._sources(view)
        P = prefix.shape[2]
        counts = np.zeros((nsrc, len(cols), P, 256), np.int64)
        nans = np.zeros((nsrc, len(cols)), np.int64)
        for c, (i, j) in enumerate(cols):
            x = X[:, :, i] if j < 0 else X[:, :, i] + X[:, :, j]
            for s in np.unique(src):
                v = x[:, src == s].ravel()
                nans[s, c] = np.isnan(v).sum()
                u = v[~np.isnan(v)].view(np.uint64)
                key = np.where(u >> np.uint64(63) == 1, ~u, u | np.uint64(1 << 63))
                digit = ((key >> np.uint64(56 - 8 * pass_)) & np.uint64(255)).astype(np.int64)
                for p in range(P):
                    if prefix[s, c, p] == NO_PREFIX:
                        continue
                    hit = np.ones(key.shape, bool) if pass_ == 0 else (key >> np.uint64(64 - 8 * pass_)) == prefix[s, c, p]
                    counts[s, c, p] += np.bincount(digit[hit], minlength=256)
        return torch.from_numpy(counts), (torch.from_numpy(nans) if pass_ == 0 else None)

    def chain_moments(self, view):
        X = self._selected(view)
        mean = X.sum(axis=0) / X.shape[0]
        return torch.from_numpy(mean), torch.from_numpy(((X - mean) ** 2).sum(axis=0))

    def chain_acf(self, view, nsrc, mean, c0, k0, k1):
        y = self._selected(view) - mean.numpy()
        n = y.shape[0]
        src = self._sources(view)
        out = np.zeros((nsrc, k1 - k0, view.ndim))
        with np.errstate(invalid="ignore", divide="ignore"):
            rho = np.stack([(y[:n - k] * y[k:]).sum(axis=0) for k in range(k0, k1)]) / c0.numpy()   # [lags, nlocal, ndim]
        for s in np.unique(src):
            out[s] = rho[:, src == s].sum(axis=1)
        return torch.from_numpy(out)


def gauss_lnprob(P):
    return -0.5 * np.sum((np.atleast_2d(P) / np.array([1.0, 2.0, 0.5])) ** 2, axis=1)


def sampler_with_chain(chunks, nsources=1):
    """A sampler whose stored chain is `chunks` (arrays [steps, nwalkers, ndim]) -- the statistics read only that."""
    nw, ndim = chunks[0].shape[1:]
    s = StretchSampler(nw, ndim, StatsEngine(gauss_lnprob), nsources=nsources, randomize_split=False)
    s._chain = [torch.from_numpy(np.ascontiguousarray(c, dtype=np.float64)) for c in chunks]
    return s


def percentile_ref(chain, nsources, q, cols, discard=0, thin=1):
    sel = np.concatenate(chain)[discard + thin - 1::thin]
    W = sel.shape[1] // nsources
    out = []
    for s in range(nsources):
        flat = sel[:, s * W:(s + 1) * W].reshape(-1, sel.shape[2])
        cc = np.column_stack([flat[:, c] if np.isscalar(c) else flat[:, c[0]] + flat[:, c[1]] for c in cols])
        with np.errstate(invalid="ignore"):
            out.append(np.percentile(cc, q, axis=0))
    return np.array(out)


def test_quantiles_equal_numpy_percentile_single_process():
    rng = np.random.default_rng(3)
    T, nw, ndim = 23, 48, 4
    X = rng.standard_normal((T, nw, ndim)) * [1.0, 1e-3, 30.0, 1.0] + [0.0, 5.0, -1.0, 0.0]
    X[:, :, 3] = np.round(X[:, :, 3] * 2) / 2              # heavy ties, both signs, +-0
    X[::3, ::5, 3] = -0.0
    X[:, 16:32, 1] = 7.25                                   # a constant column in source 1
    X[4, 40, 2] = np.inf
    X[5, 41, 2] = -np.inf
    X[6, 44, 0] = np.nan                                    # source 2, column 0 holds a NaN
    chunks = [X[:7], X[7:8], X[8:]]
    s = sampler_with_chain(chunks, nsources=3)
    cols = [0, 1, 2, 3, (0, 1), (3, 3)]
    for discard, thin in ((0, 1), (5, 2), (6, 3), (0, 7)):
        got = s.get_quantiles(QS, discard=discard, thin=thin, columns=cols)
        ref = percentile_ref(chunks, 3, QS, cols, discard, thin)
        assert got.shape == (3, len(QS), len(cols))
        assert np.array_equal(got, ref, equal_nan=True), (discard, thin, got - ref)
        if discard == 0 and thin == 1:
            assert np.isnan(got[2, :, 0]).all() and not np.isnan(got[:2, :, 0]).any()
    # default columns are the parameters; a scalar q is one percentile
    np.testing.assert_array_equal(s.get_quantiles(50)[:, 0], percentile_ref(chunks, 3, [50], [0, 1, 2, 3])[:, 0])
    with pytest.raises(ValueError):
        s.get_quantiles([101])
    with pytest.raises(ValueError):
        s.get_quantiles([50], columns=[4])
    with pytest.raises(ValueError):
        s.get_quantiles([50], thin=0)
    with pytest.raises(ValueError):
        s.get_quantiles([50], discard=T)


def test_many_ranks_are_split_into_groups():
    """More requested order statistics than one histogram pass holds (RB_CHAIN_MAX_HIST): several groups."""
    rng = np.random.default_rng(4)
    X = rng.standard_normal((9, 32, 3))
    s = sampler_with_chain([X])
    q = np.linspace(0, 100, 41)
    cols = [0, 1, 2, (0, 2), (1, 2), (0, 1)] * 3
    assert 2 * len(q) * len(cols) > _lib.RB_CHAIN_MAX_HIST
    np.testing.assert_array_equal(s.get_quantiles(q, columns=cols), percentile_ref([X], 1, q, cols))


def test_chain_selection_follows_emcee():
    """get_chain / get_log_prob (discard, thin): emcee's backend slice [discard + thin - 1 :: thin]; defaults unchanged."""
    rng = np.random.default_rng(5)
    s = StretchSampler(32, 3, StatsEngine(gauss_lnprob), seed=2)
    s.run_mcmc(rng.standard_normal((32, 3)), 7)
    s.run_mcmc(None, 6, thin=2)
    full, lfull = s.get_chain(), s.get_log_prob()
    assert full.shape == (10, 32, 3) and len(s._chain) == 2
    for discard, thin in ((0, 1), (2, 3), (9, 1), (4, 20)):
        np.testing.assert_array_equal(s.get_chain(discard=discard, thin=thin), full[discard + thin - 1::thin])
        np.testing.assert_array_equal(s.get_log_prob(flat=True, discard=discard, thin=thin),
                                      lfull[discard + thin - 1::thin].reshape(-1))
    np.testing.assert_array_equal(s.get_chain(flat=True), full.reshape(-1, 3))


# ---- emcee's integrated_time, restated with numpy (emcee/autocorr.py) --------------------------------------------
def _next_pow_two(n):
    i = 1
    while i < n:
        i = i << 1
    return i


def _function_1d(x):
    n = _next_pow_two(len(x))
    f = np.fft.fft(x - np.mean(x), n=2 * n)
    acf = np.fft.ifft(f * np.conjugate(f))[: len(x)].real
    with np.errstate(invalid="ignore"):
        acf /= acf[0]
    return acf


def _auto_window(taus, c):
    m = np.arange(len(taus)) < c * taus
    if np.any(m):
        return np.argmin(m)
    return len(taus) - 1


def emcee_integrated_time(x, c=5):
    """x [n_t, n_w, n_d] -> (tau_est [n_d], windows [n_d])."""
    n_t, n_w, n_d = x.shape
    tau, win = np.empty(n_d), np.empty(n_d, dtype=int)
    for d in range(n_d):
        f = np.zeros(n_t)
        for k in range(n_w):
            f += _function_1d(x[:, k, d])
        f /= n_w
        taus = 2.0 * np.cumsum(f) - 1.0
        win[d] = _auto_window(taus, c)
        tau[d] = taus[win[d]]
    return tau, win


def ar1_chain(rng, T, nw, phis):
    phis = np.asarray(phis)
    x = np.empty((T, nw, len(phis)))
    x[0] = rng.standard_normal((nw, len(phis)))
    for t in range(1, T):
        x[t] = phis * x[t - 1] + np.sqrt(1 - phis ** 2) * rng.standard_normal((nw, len(phis)))
    return x


def test_autocorr_time_matches_emcee():
    rng = np.random.default_rng(6)
    X = ar1_chain(rng, 700, 40, [0.3, 0.8, 0.95, 0.0])
    chunks = [X[:250], X[250:260], X[260:]]
    s = sampler_with_chain(chunks, nsources=2)
    for discard, thin in ((0, 1), (120, 1), (33, 2)):
        tau, win, n_t = s._integrated_time(discard, thin, 5)
        sel = X[discard + thin - 1::thin]
        assert n_t == sel.shape[0]
        for src in range(2):
            ref_tau, ref_win = emcee_integrated_time(sel[:, src * 20:(src + 1) * 20])
            np.testing.assert_array_equal(win[src], ref_win)
            np.testing.assert_allclose(tau[src], ref_tau, rtol=1e-10)
    got = s.get_autocorr_time(quiet=True)
    assert got.shape == (2, 4) and (got[:, 2] > got[:, 1]).all() and (got[:, 1] > got[:, 0]).all()
    np.testing.assert_allclose(s.get_autocorr_time(thin=2, quiet=True), 2 * s._integrated_time(0, 2, 5)[0], rtol=0)


def test_constant_walker_and_short_chain():
    rng = np.random.default_rng(7)
    X = ar1_chain(rng, 300, 16, [0.5, 0.5])
    X[:, 3, 1] = 0.25                                       # a stuck walker: c_0 = 0 -> NaN, as emcee's acf /= acf[0]
    s = sampler_with_chain([X], nsources=2)
    tau = s.get_autocorr_time(quiet=True)
    assert np.isnan(tau[0, 1]) and np.isfinite(tau[0, 0]) and np.isfinite(tau[1]).all()
    ref_tau, _ = emcee_integrated_time(X[:, :8])
    assert np.isnan(ref_tau[1])
    short = sampler_with_chain([ar1_chain(rng, 60, 16, [0.9, 0.9])])
    with pytest.raises(AutocorrError) as e:
        short.get_autocorr_time()
    assert e.value.tau.shape == (1, 2)
    np.testing.assert_array_equal(short.get_autocorr_time(quiet=True), e.value.tau)


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        s = _two_call_run()
        assert s.world == world and s.gid_base == rank * 24
        q = s.get_quantiles(QS, discard=3, thin=2, columns=[0, 1, 2, (0, 1)])
        tau = s.get_autocorr_time(discard=2, quiet=True)
        if rank == 0:
            np.savez(out, q=q, tau=tau)
    finally:
        dist.destroy_process_group()


def _two_call_run():
    """48 walkers, 3 sources of 16 (with two ranks, source 1 spans both), two run_mcmc calls (two chunks)."""
    rng = np.random.default_rng(9)
    s = StretchSampler(48, 3, StatsEngine(gauss_lnprob), seed=12, nsources=3, split_block=8)
    s.run_mcmc(rng.standard_normal((48, 3)), 9)
    s.run_mcmc(None, 12)
    return s


def test_world_size_2_matches_single_process(tmp_path):
    ref = _two_call_run()
    q_ref = ref.get_quantiles(QS, discard=3, thin=2, columns=[0, 1, 2, (0, 1)])
    np.testing.assert_array_equal(q_ref, percentile_ref([ref.get_chain()], 3, QS, [0, 1, 2, (0, 1)], 3, 2))
    tau_ref = ref.get_autocorr_time(discard=2, quiet=True)
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    out = str(tmp_path / "stats2.npz")
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    got = np.load(out)
    np.testing.assert_array_equal(got["q"], q_ref)
    np.testing.assert_allclose(got["tau"], tau_ref, rtol=1e-12)


# ---- the C entry points -------------------------------------------------------------------------------------------
def _view(**kw):
    t = torch.zeros((5, 8, 3), dtype=torch.float64)
    v = ChainView([t, t], 8, 3, 0, 8, 0, 1).c_struct()
    for k, val in kw.items():
        setattr(v, k, val)
    return v, t


def _call(name, v, ncol=1, col_i=0, col_j=-1):
    L = _lib.load()
    buf = (C.c_double * 4096)()
    p = C.cast(buf, C.c_void_p)
    if name == "hist":
        ci, cj = (C.c_int32 * ncol)(*([col_i] * ncol)), (C.c_int32 * ncol)(*([col_j] * ncol))
        return L.rb_chain_hist_dev(None, C.byref(v), 1, ncol, ci, cj, 0, 1, p, p, p)
    if name == "moments":
        return L.rb_chain_moments_dev(None, C.byref(v), p, p)
    return L.rb_chain_acf_dev(None, C.byref(v), 1, p, p, 0, 4, p)


@pytest.mark.parametrize("name", ["hist", "moments", "acf"])
def test_entry_points_check_the_view(name):
    for bad in (dict(nchunks=_lib.RB_MAX_CHUNKS + 1), dict(thin=0), dict(thin=-2), dict(ndim=0), dict(discard=-1)):
        v, _ = _view(**bad)
        assert _call(name, v) == -1, bad                    # RB_ERR_ARG
    if name == "hist":
        v, _ = _view()
        assert _call(name, v, col_i=3) == -1
        assert _call(name, v, col_j=3) == -1
        assert _call(name, v, ncol=_lib.RB_CHAIN_MAX_COLS + 1) == -1


@pytest.mark.parametrize("name", ["hist", "moments", "acf"])
def test_entry_points_need_a_device(name):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    v, _ = _view()
    assert _call(name, v) == -3                             # RB_ERR_CUDA
    assert "no CUDA device" in _lib.load().rb_last_error().decode()


def test_chain_view_layout_matches_the_header(tmp_path):
    import subprocess
    from conftest import ROOT
    src = tmp_path / "layout.c"
    src.write_text(r'''
#include <stdio.h>
#include <stddef.h>
#include "radex_b200.h"
#define P(f) printf(#f " %zu\n", offsetof(rb_chain_view, f))
int main(void) {
  printf("size %zu\n", sizeof(rb_chain_view));
  P(chunk); P(steps); P(nchunks); P(ndim); P(nlocal); P(gid_base); P(walkers_per_source); P(discard); P(thin);
  printf("RB_MAX_CHUNKS %d\nRB_CHAIN_MAX_DIM %d\nRB_CHAIN_MAX_COLS %d\nRB_CHAIN_MAX_HIST %d\n", RB_MAX_CHUNKS,
         RB_CHAIN_MAX_DIM, RB_CHAIN_MAX_COLS, RB_CHAIN_MAX_HIST);
  return 0;
}
''')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = dict(line.rsplit(" ", 1) for line in subprocess.check_output([str(exe)], text=True).strip().splitlines())
    assert int(got.pop("size")) == C.sizeof(_lib.rb_chain_view)
    for k in ("RB_MAX_CHUNKS", "RB_CHAIN_MAX_DIM", "RB_CHAIN_MAX_COLS", "RB_CHAIN_MAX_HIST"):
        assert int(got.pop(k)) == getattr(_lib, k), k
    for field, off in got.items():
        assert int(off) == getattr(_lib.rb_chain_view, field).offset, field
