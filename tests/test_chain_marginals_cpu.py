"""Host protocol of the corner-plot marginals, covariance and nearest sample on CPU (StretchSampler.get_histograms /
get_covariance / get_nearest_sample): a numpy engine restates the three kernels of csrc/chain_marginals.cuh, so that the
edges, numpy's errors, the pair order, the rank combination (gloo, world_size 2) and the driver's metrics are checked
without a GPU; the new C entry points refuse bad arguments and report the missing device."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from radex_emcee_b200 import _lib, driver
from radex_emcee_b200.sampler import ChainView, StretchSampler
from test_chain_stats_cpu import StatsEngine, gauss_lnprob


class MarginalsEngine(StatsEngine):
    """StatsEngine plus numpy restatements of rb_chain_marginals_dev / rb_chain_sums_dev / rb_chain_nearest_dev."""

    @staticmethod
    def bins(e, x):
        """The kernel's bin rule: (edges <= x) - 1, x == e[B] in bin B - 1, -1 when not counted."""
        B = len(e) - 1
        k = np.searchsorted(e, x, side="right") - 1
        k[x == e[B]] = B - 1
        return np.where((k >= 0) & (k < B), k, -1)

    def _columns_of(self, view, cols):
        X, src = self._selected(view), self._sources(view)
        vals = [X[:, :, i] if j < 0 else X[:, :, i] + X[:, :, j] for i, j in cols]
        return vals, src

    def chain_marginals(self, view, nsrc, cols, edges, pairs=True):
        vals, src = self._columns_of(view, cols)
        ncol, B = len(cols), edges.shape[2] - 1
        h1 = np.zeros((nsrc, ncol, B), np.int64)
        h2 = np.zeros((nsrc, ncol * (ncol - 1) // 2, B, B), np.int64)
        for s in np.unique(src):
            k = [self.bins(edges[s, c], vals[c][:, src == s].ravel()) for c in range(ncol)]
            for c in range(ncol):
                h1[s, c] = np.bincount(k[c][k[c] >= 0], minlength=B)
            p = 0
            for a in range(ncol):
                for b in range(a + 1, ncol):
                    ok = (k[a] >= 0) & (k[b] >= 0)
                    h2[s, p] = np.bincount(k[a][ok] * B + k[b][ok], minlength=B * B).reshape(B, B)
                    p += 1
        return torch.from_numpy(h1), (torch.from_numpy(h2) if pairs else None)

    def chain_sums(self, view, nsrc, center):
        X, src = self._selected(view), self._sources(view)
        s1 = np.zeros((nsrc, view.ndim))
        s2 = np.zeros((nsrc, view.ndim, view.ndim))
        for s in np.unique(src):
            y = X[:, src == s].reshape(-1, view.ndim) - center[s]
            s1[s] = y.sum(axis=0)
            s2[s] = y.T @ y
        return torch.from_numpy(s1), torch.from_numpy(s2)

    def chain_nearest(self, view, nsrc, target, chol):
        X, src = self._selected(view), self._sources(view)
        W = view.walkers_per_source
        d2 = np.full(nsrc, np.inf)
        idx = np.full(nsrc, -1, np.int64)
        x = np.zeros((nsrc, view.ndim))
        for s in np.unique(src):
            loc = np.flatnonzero(src == s)
            Y = X[:, loc]                                            # [nsel, nw, ndim]
            w = np.linalg.solve(chol[s], (Y - target[s]).reshape(-1, view.ndim).T)
            dd = np.einsum("ij,ij->j", w, w)
            i = int(np.argmin(dd))
            j, k = divmod(i, len(loc))
            d2[s], x[s] = dd[i], Y[j, k]
            idx[s] = j * W + view.gid_base + loc[k] - s * W
        return torch.from_numpy(d2), torch.from_numpy(idx), torch.from_numpy(x)


def sampler_with_chain(chunks, nsources=1):
    nw, ndim = chunks[0].shape[1:]
    s = StretchSampler(nw, ndim, MarginalsEngine(gauss_lnprob), nsources=nsources, randomize_split=False)
    s._chain = [torch.from_numpy(np.ascontiguousarray(c, dtype=np.float64)) for c in chunks]
    return s


def column(flat, c):
    return flat[:, c] if np.isscalar(c) else flat[:, c[0]] + flat[:, c[1]]


def source_slices(chunks, nsources, discard=0, thin=1):
    sel = np.concatenate(chunks)[discard + thin - 1::thin]
    W = sel.shape[1] // nsources
    return [sel[:, s * W:(s + 1) * W].reshape(-1, sel.shape[2]) for s in range(nsources)]


def check_histograms(s, chunks, nsources, bins, cols, discard=0, thin=1, rng=None):
    edges, h1, h2, pairs = s.get_histograms(bins, discard=discard, thin=thin, columns=cols, range=rng)
    ncol = len(cols)
    assert pairs == [(a, b) for a in range(ncol) for b in range(a + 1, ncol)]
    assert h1.dtype == np.int64 and h2.shape == (nsources, len(pairs), bins, bins)
    for src, flat in enumerate(source_slices(chunks, nsources, discard, thin)):
        r = None if rng is None else np.broadcast_to(np.asarray(rng, dtype=np.float64), (nsources, ncol, 2))[src]
        for c in range(ncol):
            h, e = np.histogram(column(flat, cols[c]), bins, range=None if r is None else tuple(r[c]))
            np.testing.assert_array_equal(edges[src, c], e)
            np.testing.assert_array_equal(h1[src, c], h)
        for p, (a, b) in enumerate(pairs):
            h, ea, eb = np.histogram2d(column(flat, cols[a]), column(flat, cols[b]), bins,
                                       range=None if r is None else [tuple(r[a]), tuple(r[b])])
            np.testing.assert_array_equal(h2[src, p], h)
            np.testing.assert_array_equal(edges[src, a], ea)
            np.testing.assert_array_equal(edges[src, b], eb)
    return edges, h1, h2


def test_histograms_equal_numpy_across_chunks():
    rng = np.random.default_rng(11)
    T, nw, ndim = 23, 3 * 16, 4
    X = rng.standard_normal((T, nw, ndim)) * [1.0, 1e-3, 30.0, 1.0] + [0.0, 5.0, -1.0, 0.0]
    X[:, :, 3] = np.round(X[:, :, 3] * 2) / 2             # ties on the edges
    X[::3, ::5, 3] = -0.0
    X[:, 16:32, 1] = 7.25                                   # a constant column in source 1
    chunks = [X[:7], X[7:8], X[8:]]
    s = sampler_with_chain(chunks, nsources=3)
    cols = [0, 1, 2, 3, (0, 1)]
    for discard, thin in ((0, 1), (5, 2), (6, 3)):
        for bins in (1, 7, 20):
            check_histograms(s, chunks, 3, bins, cols, discard, thin)
    check_histograms(s, chunks, 3, 100, [3], 0, 1)          # one column: no pairs


def test_histogram_edge_values():
    """Values exactly on interior edges, the maximum on the last edge, +-0, an explicit range that excludes values, +-inf."""
    rng = np.random.default_rng(12)
    X = rng.integers(-4, 5, size=(9, 16, 3)).astype(np.float64)   # integers: every value on an edge of range (-4, 4), 8 bins
    X[0, 0, 0], X[1, 1, 0] = -0.0, 0.0
    X[2, 2, 1], X[3, 3, 1] = np.inf, -np.inf
    s = sampler_with_chain([X])
    cols = [0, 2, (0, 2)]
    check_histograms(s, [X], 1, 8, cols, rng=[(-4, 4), (-4, 4), (-8, 8)])
    check_histograms(s, [X], 1, 5, cols, rng=[(-1, 2), (0, 0), (-3.5, 1e-300)])   # excludes values; lo == hi widens
    check_histograms(s, [X], 1, 8, [0, 2, 1], rng=[(-4, 4), (-4, 4), (-4, 4)])  # +-inf in column 1: not counted
    check_histograms(s, [X], 1, 16, cols)                   # auto range: the max lands on the last edge
    X2 = np.full((4, 16, 2), 3.0)                           # a constant column with the auto range: (2.5, 3.5)
    X2[:, :, 1] = rng.standard_normal((4, 16))
    e, h1, _ = check_histograms(sampler_with_chain([X2]), [X2], 1, 4, [0, 1])
    assert e[0, 0, 0] == 2.5 and e[0, 0, -1] == 3.5 and h1[0, 0].sum() == 64


def test_histogram_errors():
    X = np.random.default_rng(13).standard_normal((5, 16, 3))
    X[2, 3, 1] = np.nan
    s = sampler_with_chain([X])
    with pytest.raises(ValueError, match=r"autodetected range of \[nan, nan\] is not finite \(source 0, column 1\)"):
        s.get_histograms(10, columns=[0, 1])
    s.get_histograms(10, columns=[0, 1], range=[(-3, 3), (-3, 3)])    # NaN is simply not counted with a range
    Xi = X.copy()
    Xi[2, 3, 1] = np.inf
    with pytest.raises(ValueError, match="not finite"):
        sampler_with_chain([Xi]).get_histograms(10, columns=[1])
    for bins in (0, _lib.RB_CHAIN_MAX_BINS + 1):
        with pytest.raises(ValueError, match="bins"):
            s.get_histograms(bins, columns=[0])
    with pytest.raises(ValueError, match="max must be larger than min"):
        s.get_histograms(10, columns=[0], range=[(1, 0)])
    with pytest.raises(ValueError, match="not finite"):
        s.get_histograms(10, columns=[0], range=[(0, np.inf)])
    with pytest.raises(ValueError):
        s.get_histograms(10, columns=[0, 2], range=[(0, 1)])
    with pytest.raises(ValueError, match="Too many bins for data range"):
        s.get_histograms(100, columns=[0], range=[(1.0, np.nextafter(1.0, 2.0))])
    with pytest.raises(ValueError):
        np.histogram([1.0], 100, range=(1.0, np.nextafter(1.0, 2.0)))


def test_covariance_matches_np_cov():
    rng = np.random.default_rng(14)
    X = rng.standard_normal((30, 3 * 16, 4)) @ rng.standard_normal((4, 4)) + [5.0, -1e3, 0.0, 1e-3]
    chunks = [X[:11], X[11:]]
    s = sampler_with_chain(chunks, nsources=3)
    for discard, thin in ((0, 1), (4, 3)):
        cov = s.get_covariance(discard, thin)
        for src, flat in enumerate(source_slices(chunks, 3, discard, thin)):
            np.testing.assert_allclose(cov[src], np.cov(flat, rowvar=False), rtol=1e-12, atol=0)
    X[3, 20, 2] = np.nan
    cov = sampler_with_chain([X], nsources=3).get_covariance()
    assert np.isnan(cov[1, 2]).all() and np.isfinite(cov[0]).all() and np.isfinite(cov[1, :2, :2]).all()


@pytest.mark.parametrize("metric", ["mahalanobis", "z", "euclidean"])
def test_nearest_sample_matches_driver(metric):
    rng = np.random.default_rng(15)
    X = rng.standard_normal((25, 3 * 16, 4)) @ rng.standard_normal((4, 4))
    X[:, 16:32, 3] = 2.0                                    # a constant parameter in source 1 (z metric: eps)
    chunks = [X[:9], X[9:]]
    s = sampler_with_chain(chunks, nsources=3)
    targets = rng.standard_normal((3, 4))
    for discard, thin in ((0, 1), (3, 2)):
        x, idx, d2 = s.get_nearest_sample(targets, discard, thin, metric=metric)
        for src, flat in enumerate(source_slices(chunks, 3, discard, thin)):
            if metric == "mahalanobis" and src == 1:
                continue                                    # singular covariance + eps: both sides ill-conditioned
            ref_x, ref_i, ref_d2 = driver.nearest_sample_to_vector(flat, targets[src], metric=metric)
            assert idx[src] == ref_i and np.array_equal(x[src], flat[idx[src]])
            np.testing.assert_allclose(d2[src], ref_d2, rtol=1e-10)
    # one target for every source
    x, idx, _ = s.get_nearest_sample(targets[0], metric=metric)
    assert idx.shape == (3,) and x.shape == (3, 4)


def test_nearest_sample_nan_and_ties():
    X = np.zeros((4, 16, 2))
    X[:, :, 0] = np.arange(16)
    s = sampler_with_chain([X])
    x, idx, d2 = s.get_nearest_sample([3.0, 0.0], metric="euclidean")
    assert idx[0] == 3 and d2[0] == 0.0                     # 4 samples at distance 0: the lowest index
    X[2, 9, 1] = np.nan
    X[3, 5, 1] = np.nan
    x, idx, d2 = sampler_with_chain([X]).get_nearest_sample([3.0, 0.0], metric="euclidean")
    assert idx[0] == 2 * 16 + 9 and np.isnan(d2[0]) and np.isnan(x[0, 1])     # NaN first, as np.argmin
    assert driver.nearest_sample_to_vector(X.reshape(-1, 2), [3.0, 0.0], metric="euclidean")[1] == idx[0]
    with pytest.raises(ValueError):
        s.get_nearest_sample([0.0, 0.0], metric="cosine")
    with pytest.raises(ValueError):
        s.get_nearest_sample([0.0, 0.0, 0.0])


def _two_call_run():
    """48 walkers, 3 sources of 16 (with two ranks, source 1 spans both), two run_mcmc calls (two chunks)."""
    rng = np.random.default_rng(9)
    s = StretchSampler(48, 3, MarginalsEngine(gauss_lnprob), seed=12, nsources=3, split_block=8)
    s.run_mcmc(rng.standard_normal((48, 3)), 9)
    s.run_mcmc(None, 12)
    return s


def _everything(s):
    e, h1, h2, _ = s.get_histograms(12, discard=3, thin=2, columns=[0, 1, 2, (0, 1)])
    cov = s.get_covariance(discard=2)
    near = [s.get_nearest_sample([0.1, -0.2, 0.3], discard=1, metric=m) for m in ("mahalanobis", "z", "euclidean")]
    return dict(e=e, h1=h1, h2=h2, cov=cov, **{"%s%d" % (k, i): v[j] for i, v in enumerate(near)
                                                for j, k in enumerate("xid")})


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        s = _two_call_run()
        assert s.world == world and s.gid_base == rank * 24
        res = _everything(s)
        if rank == 0:
            np.savez(out, **res)
    finally:
        dist.destroy_process_group()


def test_world_size_2_matches_single_process(tmp_path):
    ref = _two_call_run()
    want = _everything(ref)
    check_histograms(ref, [ref.get_chain()], 3, 12, [0, 1, 2, (0, 1)], 3, 2)
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    out = str(tmp_path / "marg2.npz")
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    got = np.load(out)
    for k, v in want.items():
        if k == "cov" or k.startswith("d"):
            np.testing.assert_allclose(got[k], v, rtol=1e-12, err_msg=k)
        else:
            np.testing.assert_array_equal(got[k], v, err_msg=k)


# ---- the C entry points -------------------------------------------------------------------------------------------
def _view(**kw):
    t = torch.zeros((5, 8, 3), dtype=torch.float64)
    v = ChainView([t, t], 8, 3, 0, 8, 0, 1).c_struct()
    for k, val in kw.items():
        setattr(v, k, val)
    return v, t


def _call(name, v, ncol=2, col_i=0, col_j=-1, nbins=4, null=False):
    L = _lib.load()
    buf = (C.c_double * 8192)()
    p = None if null else C.cast(buf, C.c_void_p)
    if name == "marginals":
        ci, cj = (C.c_int32 * ncol)(*([col_i] * ncol)), (C.c_int32 * ncol)(*([col_j] * ncol))
        return L.rb_chain_marginals_dev(None, C.byref(v), 1, ncol, ci, cj, nbins, p, p, p)
    if name == "sums":
        return L.rb_chain_sums_dev(None, C.byref(v), 1, p, p, p)
    return L.rb_chain_nearest_dev(None, C.byref(v), 1, p, p, p, p, p)


@pytest.mark.parametrize("name", ["marginals", "sums", "nearest"])
def test_entry_points_check_their_arguments(name):
    for bad in (dict(nchunks=_lib.RB_MAX_CHUNKS + 1), dict(thin=0), dict(ndim=0), dict(discard=-1),
                dict(walkers_per_source=4)):                  # nsrc = 1 does not cover walkers of 4 per source
        v, _ = _view(**bad)
        assert _call(name, v) == -1, bad                    # RB_ERR_ARG
    v, _ = _view()
    assert _call(name, v, null=True) == -1
    if name == "marginals":
        assert _call(name, v, col_i=3) == -1
        assert _call(name, v, col_j=3) == -1
        assert _call(name, v, ncol=0) == -1
        assert _call(name, v, ncol=_lib.RB_CHAIN_MAX_COLS + 1) == -1
        assert _call(name, v, nbins=0) == -1
        assert _call(name, v, nbins=_lib.RB_CHAIN_MAX_BINS + 1) == -1


@pytest.mark.parametrize("name", ["marginals", "sums", "nearest"])
def test_entry_points_need_a_device(name):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    v, _ = _view()
    assert _call(name, v) == -3                             # RB_ERR_CUDA
    assert "no CUDA device" in _lib.load().rb_last_error().decode()


def test_max_bins_matches_the_header(tmp_path):
    import subprocess
    from conftest import ROOT
    src = tmp_path / "bins.c"
    src.write_text('#include <stdio.h>\n#include "radex_b200.h"\n'
                   'int main(void) { printf("%d\\n", RB_CHAIN_MAX_BINS); return 0; }\n')
    exe = tmp_path / "bins"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe),
                           str(src)])
    assert int(subprocess.check_output([str(exe)], text=True)) == _lib.RB_CHAIN_MAX_BINS
