"""Host protocol of the posterior-predictive SLEDs on CPU (sampler.get_predicted_fluxes / get_predictive_quantiles): a
numpy engine evaluates a toy SLED model in place of rb_predict_sled_dev, so that the gather order, the per-plane
percentiles and the all_reduce over ranks (gloo, world_size 2) are checked without a GPU; the new C entry point refuses
bad arguments and reports the missing device."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from radex_emcee_b200 import _lib
from radex_emcee_b200.sampler import ChainView, StretchSampler
from test_chain_stats_cpu import QS, StatsEngine

NLINE = 40
T_MAX = 4.0      # log10 T above which the toy model is out of range, as pyradex is above 1e4 K


def toy_surf(theta4, jup):
    """A made-up brightness per line: [..., nlines] from [..., 4] (log n, log T, log N, log size); NaN out of range."""
    J = np.asarray(jup, dtype=np.float64)
    n, T, N = (10.0 ** theta4[..., i, None] for i in range(3))
    s = 1e-36 * N * J ** 2 * np.exp(-J * J / (T + 1.0)) / (1.0 + 1e3 / n)
    return np.where(theta4[..., 1, None] > T_MAX, np.nan, s)


class SledEngine(StatsEngine):
    """StatsEngine plus a numpy rb_predict_sled_dev over toy_surf, with the same planes and the same flux expression."""

    def __init__(self, lnprob_fn, ncomp):
        super().__init__(lnprob_fn)
        self.ncomp = ncomp

    def predict_sled(self, view, jup):
        jup = np.asarray(jup)
        if jup.size < 1 or jup.size > _lib.RB_MAX_OBS or jup.min() < 1 or jup.max() > NLINE:
            raise _lib.RadexB200Error("bad jup")
        X = self._selected(view)
        comp = [toy_surf(X[..., 4 * c:4 * c + 4], jup) * (10.0 ** X[..., 4 * c + 3, None]) * 1.0e23
                for c in range(self.ncomp)]
        planes = comp if self.ncomp == 1 else [comp[0] + comp[1]] + comp
        return torch.from_numpy(np.ascontiguousarray(np.stack(planes)))


CENTRE = np.array([3.0, 1.5, 16.5, -10.0, 4.0, 2.5, 17.0, -10.5])


def toy_lnprob(P):
    P = np.atleast_2d(P)
    return -0.5 * np.sum(((P - CENTRE[:P.shape[1]]) / 0.3) ** 2, axis=1)


def run(ncomp, nwalkers=48, nsources=3, hot=False):
    """Two run_mcmc calls (two chunks); `hot`: a walker of source 0 pushed out of the toy model's range."""
    ndim = 4 * ncomp
    rng = np.random.default_rng(21 + ncomp)
    s = StretchSampler(nwalkers, ndim, SledEngine(toy_lnprob, ncomp), seed=5, nsources=nsources, split_block=8)
    s.run_mcmc(CENTRE[:ndim] + 0.3 * rng.standard_normal((nwalkers, ndim)), 7)
    s.run_mcmc(None, 9)
    if hot:
        s._chain[1][3, 2, 1] = T_MAX + 0.1                 # step 10, walker 2, component 1's log T
    return s


def reference_fluxes(s, jup, discard, thin):
    X = s.get_chain(discard=discard, thin=thin)
    comp = [toy_surf(X[..., 4 * c:4 * c + 4], jup) * (10.0 ** X[..., 4 * c + 3, None]) * 1.0e23
            for c in range(s.ndim // 4)]
    return np.stack(comp if len(comp) == 1 else [comp[0] + comp[1]] + comp)


def percentile_of_planes(F, nsources, q):
    """[nsources, nplanes, len(q), nlines] from the gathered planes [nplanes, steps, nwalkers, nlines]."""
    W = F.shape[2] // nsources
    out = np.empty((nsources, F.shape[0], len(q), F.shape[3]))
    for s in range(nsources):
        for p in range(F.shape[0]):
            with np.errstate(invalid="ignore"):
                out[s, p] = np.percentile(F[p][:, s * W:(s + 1) * W].reshape(-1, F.shape[3]), q, axis=0)
    return out


@pytest.mark.parametrize("ncomp", [1, 2])
def test_predicted_fluxes_and_quantiles_single_process(ncomp):
    s = run(ncomp, hot=True)
    jup = [5, 1, 11, 5, 40]                                 # unsorted, repeated, the last line of the table
    for discard, thin in ((0, 1), (5, 2), (6, 3)):
        F = s.get_predicted_fluxes(jup, discard=discard, thin=thin)
        np.testing.assert_array_equal(F, reference_fluxes(s, jup, discard, thin))
        assert F.shape == ((1 if ncomp == 1 else 3), len(range(discard + thin - 1, 16, thin)), 48, len(jup))
        np.testing.assert_array_equal(s.get_predicted_fluxes(jup, discard=discard, thin=thin, flat=True),
                                      F.reshape(F.shape[0], -1, len(jup)))
        got = s.get_predictive_quantiles(jup, QS, discard=discard, thin=thin)
        assert got.shape == (3, F.shape[0], len(QS), len(jup))
        assert np.array_equal(got, percentile_of_planes(F, 3, QS), equal_nan=True), (discard, thin)
    F = s.get_predicted_fluxes(jup)
    got = s.get_predictive_quantiles(jup, [16, 50, 84])
    # the hot sample: NaN in its component's plane and in the total, a NaN column in source 0's quantiles only
    assert np.isnan(F[0, 3 + 7, 2]).all() and np.isnan(got[0, 0]).all() and not np.isnan(got[1:]).any()
    if ncomp == 2:
        assert np.isnan(F[1, 10, 2]).all() and np.isfinite(F[2, 10, 2]).all()
        assert np.isnan(got[0, 1]).all() and not np.isnan(got[0, 2]).any()
    with pytest.raises(ValueError):
        s.get_predictive_quantiles(jup, [101])
    with pytest.raises(ValueError):
        s.get_predicted_fluxes([])
    with pytest.raises(ValueError):
        s.get_predicted_fluxes(list(range(1, 18)))
    with pytest.raises(ValueError):
        s.get_predictive_quantiles(jup, [50], discard=16)


def test_chain_quantiles_unchanged_by_the_shared_interpolation():
    """get_quantiles goes through the same interpolation helper: still np.percentile of the flat chain under ==."""
    s = run(2)
    flat = s.get_chain(flat=True, discard=2, thin=3)
    ref = np.stack([np.percentile(flat.reshape(-1, 48, 8)[:, k * 16:(k + 1) * 16].reshape(-1, 8), QS, axis=0)
                    for k in range(3)])
    np.testing.assert_array_equal(s.get_quantiles(QS, discard=2, thin=3), ref)


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        s = run(2)
        assert s.world == world and s.gid_base == rank * 24
        F = s.get_predicted_fluxes([3, 1, 3], discard=3, thin=2)
        q = s.get_predictive_quantiles([3, 1, 3], QS, discard=3, thin=2)
        if rank == 0:
            np.savez(out, F=F, q=q)
    finally:
        dist.destroy_process_group()


def test_world_size_2_matches_single_process(tmp_path):
    """48 walkers in 3 sources of 16 over two ranks of 24: source 1 is split across the ranks."""
    ref = run(2)
    F_ref = ref.get_predicted_fluxes([3, 1, 3], discard=3, thin=2)
    q_ref = ref.get_predictive_quantiles([3, 1, 3], QS, discard=3, thin=2)
    np.testing.assert_array_equal(q_ref, percentile_of_planes(F_ref, 3, QS))
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    out = str(tmp_path / "sled2.npz")
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    got = np.load(out)
    np.testing.assert_array_equal(got["F"], F_ref)
    np.testing.assert_array_equal(got["q"], q_ref)


# ---- the C entry point --------------------------------------------------------------------------------------------
def _call(nlines=3, jup=(1, 2, 3), view=True, set_=True, flux=True, **vkw):
    t = torch.zeros((5, 8, 4), dtype=torch.float64)
    v = ChainView([t, t], 8, 4, 0, 8, 0, 1).c_struct()
    for k, val in vkw.items():
        setattr(v, k, val)
    buf = (C.c_double * 4096)()
    j = (C.c_int32 * max(1, len(jup)))(*jup)
    return _lib.load().rb_predict_sled_dev(None, C.cast(buf, C.c_void_p) if set_ else None, C.byref(v) if view else None,
                                           nlines, j, None, C.cast(buf, C.c_void_p) if flux else None, None)


def test_entry_point_checks_its_arguments():
    assert _call(nlines=0) == -1                            # RB_ERR_ARG
    assert _call(nlines=17, jup=tuple(range(1, 18))) == -1
    assert _call(jup=(1, 0, 2)) == -1
    assert "J must be in 1..nline" in _lib.load().rb_last_error().decode()
    assert _call(jup=(-3, 1, 2)) == -1
    assert _call(view=False) == -1
    assert _call(set_=False) == -1
    assert _call(flux=False) == -1
    for bad in (dict(thin=0), dict(discard=-1), dict(nchunks=_lib.RB_MAX_CHUNKS + 1), dict(nchunks=-1)):
        assert _call(**bad) == -1, bad
    L = _lib.load()
    assert L.rb_predict_sled_dev(None, None, None, 1, None, None, None, None) == -1


def test_entry_point_needs_a_device():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    assert _call() == -3                                    # RB_ERR_CUDA
    assert "no CUDA device" in _lib.load().rb_last_error().decode()


def test_entry_point_matches_the_header(tmp_path):
    """The declaration in include/radex_b200.h, compiled as C, against the ctypes signature of _lib.py."""
    import subprocess
    from conftest import ROOT
    src = tmp_path / "decl.c"
    src.write_text(r'''
#include "radex_b200.h"
int (*const f)(rb_ctx *, const rb_srcset *, const rb_chain_view *, int32_t, const int32_t *, const rb_opts *, double *,
               int64_t *) = rb_predict_sled_dev;
''')
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic-errors", "-fsyntax-only", "-I",
                           os.path.join(ROOT, "include"), str(src)])
    res, args = _lib.SIGNATURES["rb_predict_sled_dev"]
    assert res is C.c_int
    assert args == [C.c_void_p, C.c_void_p, C.POINTER(_lib.rb_chain_view), C.c_int32, C.POINTER(C.c_int32),
                    C.POINTER(_lib.rb_opts), C.c_void_p, C.c_void_p]
