"""Corner-plot marginals, covariance and nearest sample on the device (csrc/chain_marginals.cuh through
StretchSampler.get_histograms / get_covariance / get_nearest_sample): the kernels against their numpy restatement
(tests/test_chain_marginals_cpu.py), np.histogram2d and np.cov on large columns, the driver's nearest-sample helper, a
real sampler run, the driver with and without the chain on the host, two ranks."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import MOLFILE, ROOT
from radex_emcee_b200 import _lib, driver
from radex_emcee_b200.data import DATA_DIR, read_data
from radex_emcee_b200.sampler import ChainView, CudaEngine, StretchSampler
from test_chain_marginals_cpu import MarginalsEngine, check_histograms, column, source_slices
from test_chain_stats_cpu import ar1_chain
from test_gpu_sampler import model1

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    return _lib.Context(_lib.MolData(MOLFILE), 0)


def device_sampler(ctx, chunks, nsources=1):
    nw, ndim = chunks[0].shape[1:]
    m, _ = model1()
    s = StretchSampler(nw, ndim, CudaEngine(ctx, m), nsources=nsources, randomize_split=False)
    s._chain = [torch.as_tensor(c, dtype=torch.float64).cuda().contiguous() for c in chunks]
    return s


def test_kernels_match_numpy_restatement(ctx):
    """Counts bit for bit, sums and the nearest sample to rounding, for a rank that owns walkers [70, 260) of sources of
    45 walkers (a source split at both ends).  100 bins x 10 columns takes several pair groups."""
    rng = np.random.default_rng(21)
    nlocal, ndim, W, gid_base = 190, 6, 45, 70
    X = ar1_chain(rng, 70, nlocal, [0.2, 0.7, 0.9, 0.5, 0.0, 0.3]) * [1, 1, 3, 1, 1, 1e-3]
    X[:, :, 3] = np.round(X[:, :, 3])                     # values on edges
    X[5, 7, 4], X[6, 8, 4], X[9, 9, 2] = np.inf, -np.inf, np.nan
    parts = [X[:30], X[30:31], X[31:]]
    m, _ = model1()
    eng, ref = CudaEngine(ctx, m), MarginalsEngine(None)
    nsrc = (gid_base + nlocal - 1) // W + 1
    every = [(i, -1) for i in range(ndim)] + [(0, 1), (2, 3), (4, 5), (1, 3)]
    for discard, thin in ((0, 1), (29, 2)):
        vd = ChainView([torch.from_numpy(p).cuda() for p in parts], nlocal, ndim, gid_base, W, discard, thin)
        vh = ChainView([torch.from_numpy(p) for p in parts], nlocal, ndim, gid_base, W, discard, thin)
        for bins in (1, 7, 20, 100):
            for ncol in (1, 5, 10):
                cols = every[:ncol]
                hi = rng.integers(1, 4, (nsrc, ncol, 1)).astype(np.float64)   # a last edge the rounded column hits
                edges = np.linspace(-hi - rng.uniform(0, 0.5, hi.shape), hi, bins + 1, axis=2)[..., 0]
                hd1, hd2 = eng.chain_marginals(vd, nsrc, cols, edges, pairs=ncol > 1)
                hh1, hh2 = ref.chain_marginals(vh, nsrc, cols, edges, pairs=ncol > 1)
                np.testing.assert_array_equal(hd1.cpu().numpy(), hh1.numpy(), err_msg=str((bins, ncol)))
                if ncol > 1:
                    np.testing.assert_array_equal(hd2.cpu().numpy(), hh2.numpy(), err_msg=str((bins, ncol)))
                    assert hd2[1:].sum() > 0
        center = rng.standard_normal((nsrc, ndim))
        Y = X.copy()
        Y[9, 9, 2] = 0.5                                    # finite sums and distances for the rounding comparison
        Y[5, 7, 4] = Y[6, 8, 4] = 0.25
        yparts = [Y[:30], Y[30:31], Y[31:]]
        vd = ChainView([torch.from_numpy(p).cuda() for p in yparts], nlocal, ndim, gid_base, W, discard, thin)
        vh = ChainView([torch.from_numpy(p) for p in yparts], nlocal, ndim, gid_base, W, discard, thin)
        s1d, s2d = eng.chain_sums(vd, nsrc, center)
        s1h, s2h = ref.chain_sums(vh, nsrc, center)
        np.testing.assert_allclose(s1d.cpu().numpy(), s1h.numpy(), rtol=1e-11, atol=1e-9)
        np.testing.assert_allclose(s2d.cpu().numpy(), s2h.numpy(), rtol=1e-11, atol=1e-9)
        assert (s1d[0] == 0).all() and (s2d[0] == 0).all()   # source 0 has no walker on this rank
        A = rng.standard_normal((nsrc, ndim, ndim)) * 0.1
        chol = np.tril(A) + 2 * np.eye(ndim)
        dd, idd, xd = eng.chain_nearest(vd, nsrc, center, chol)
        dh, idh, xh = ref.chain_nearest(vh, nsrc, center, chol)
        assert idd[0] == -1 and dd[0] == np.inf
        np.testing.assert_array_equal(idd.cpu().numpy(), idh.numpy())
        np.testing.assert_array_equal(xd.cpu().numpy(), xh.numpy())
        np.testing.assert_allclose(dd.cpu().numpy(), dh.numpy(), rtol=1e-12)


def test_histograms_large_columns(ctx):
    """Two sources of 1000 walkers, 16 800 steps (2^24 values per column and source) == np.histogram2d, with a
    column crowded into one bin."""
    g = torch.Generator(device="cuda").manual_seed(22)
    T, W = 16800, 1000
    X = torch.randn((T, 2 * W, 3), generator=g, device="cuda", dtype=torch.float64)
    X[:, :, 1] = 1.0 + 1e-9 * torch.round(0.3 * X[:, :, 1])   # 90 % in one bin of the auto range
    X[:, W:, 2] = torch.exp(X[:, W:, 2] * 3)                 # log-normal: a long tail
    assert T * W >= 1 << 24
    s = device_sampler(ctx, [X[:9000], X[9000:]], nsources=2)
    host = X.cpu().numpy()
    check_histograms(s, [host], 2, 20, [0, 1, 2], discard=3000)
    e, h1, h2, _ = s.get_histograms(20, columns=[0, 1, 2])
    assert h1[:, 1].max() > 0.6 * T * W


def test_covariance_and_nearest(ctx):
    rng = np.random.default_rng(23)
    T, W, ndim = 400, 3 * 50, 4
    X = ar1_chain(rng, T, W, [0.3, 0.5, 0.7, 0.1]) @ rng.standard_normal((4, 4)) + [5.0, -1e3, 0.0, 1e-3]
    chunks = [X[:150], X[150:]]
    s = device_sampler(ctx, chunks, nsources=3)
    a, b = s.get_covariance(discard=20, thin=2), s.get_covariance(discard=20, thin=2)
    assert a.tobytes() == b.tobytes()
    flats = source_slices(chunks, 3, 20, 2)
    for src, flat in enumerate(flats):
        np.testing.assert_allclose(a[src], np.cov(flat, rowvar=False), rtol=1e-12, atol=0)
    targets = np.array([np.median(f, axis=0) for f in flats]) + 0.01
    for metric in ("mahalanobis", "z", "euclidean"):
        x, idx, d2 = s.get_nearest_sample(targets, discard=20, thin=2, metric=metric)
        for src, flat in enumerate(flats):
            Xs, d = flat, flat - targets[src]
            if metric == "mahalanobis":
                cov = np.cov(Xs, rowvar=False) + 1e-9 * np.eye(ndim)
                w = np.linalg.solve(np.linalg.cholesky(cov), d.T)
                host = np.einsum("ij,ij->j", w, w)
            elif metric == "z":
                host = np.sum((d / Xs.std(axis=0, ddof=1)) ** 2, axis=1)
            else:
                host = np.sum(d * d, axis=1)
            order = np.argsort(host)
            assert np.array_equal(x[src], flat[idx[src]])
            np.testing.assert_allclose(host[idx[src]], host[order[0]], rtol=1e-10)
            np.testing.assert_allclose(d2[src], host[order[0]], rtol=1e-10)
            if host[order[1]] > host[order[0]] * (1 + 1e-8):
                assert idx[src] == order[0]
            assert driver.nearest_sample_to_vector(flat, targets[src], metric=metric)[1] in (idx[src], order[0])


def test_real_sampler_run(ctx):
    """Config-1 shape (100 walkers, two run_mcmc calls): histograms, covariance and nearest sample of the host chain."""
    model, p0 = model1()
    pos = p0 + 1e-3 * np.random.RandomState(20170914).randn(100, 4)
    s = StretchSampler(100, 4, CudaEngine(ctx, model), seed=20170914)
    s.run_mcmc(pos, 60)
    s.run_mcmc(None, 90)
    cols = driver.summary_columns(1)
    for discard, thin in ((0, 1), (50, 3)):
        check_histograms(s, [s.get_chain()], 1, 20, cols, discard, thin)
        flat = s.get_chain(flat=True, discard=discard, thin=thin)
        np.testing.assert_allclose(s.get_covariance(discard, thin)[0], np.cov(flat, rowvar=False), rtol=1e-12)
        med = np.percentile(flat, 50, axis=0)
        x, idx, d2 = s.get_nearest_sample(med, discard, thin)
        rx, ri, rd2 = driver.nearest_sample_to_vector(flat, med)
        np.testing.assert_allclose(d2[0], rd2, rtol=1e-10)
        assert np.array_equal(x[0], flat[idx[0]])


def test_driver_corner(tmp_path):
    data = read_data(os.path.join(DATA_DIR, "flux.dat"))
    kw = dict(ncomp=1, nwalkers=64, n_iter_burn=10, n_iter_walk=30, allow_synthetic=True, corner_bins=15)
    res = driver.fit_source("G09v1.97", data, outdir=str(tmp_path / "a"), **kw)
    lean = driver.fit_source("G09v1.97", data, outdir=str(tmp_path / "b"), chain_to_host=False, **kw)
    assert lean["chain"] is None
    c, cl = res["corner"], lean["corner"]
    for k in c:
        np.testing.assert_array_equal(np.asarray(cl[k], dtype=object if k == "columns" else None),
                                      np.asarray(c[k], dtype=object if k == "columns" else None), err_msg=k)
    flat = res["chain"].reshape(-1, 4)
    assert c["columns"] == driver.summary_columns(1) and c["hist2d"].shape == (10, 15, 15)
    h, _, _ = np.histogram2d(flat[:, 0], flat[:, 0] + flat[:, 1], 15)
    np.testing.assert_array_equal(c["hist2d"][3], h)
    x, i, d2 = driver.nearest_sample_to_vector(flat, res["theta_med"])
    np.testing.assert_allclose(c["theta_nearest_d2"], d2, rtol=1e-10)
    np.testing.assert_array_equal(c["theta_nearest"], flat[c["theta_nearest_index"]])
    z = np.load(os.path.join(str(tmp_path / "b"), "G09v1.97_corner.npz"))
    np.testing.assert_array_equal(z["hist2d"], c["hist2d"])
    np.testing.assert_array_equal(z["columns"], [(0, -1), (1, -1), (2, -1), (3, -1), (0, 1)])
    import io
    buf = io.StringIO()
    driver.print_summary(res, 1, file=buf)
    assert buf.getvalue().count("nearest") == 1
    out = driver.fit_sources_concurrently(list(data)[:2], data, ncomp=1, nwalkers=40, n_iter_burn=5, n_iter_walk=12,
                                          allow_synthetic=True, corner_bins=8, outdir=str(tmp_path / "c"))
    for r in out:
        flat = r["chain"].reshape(-1, 4)
        h, _ = np.histogram(flat[:, 2], 8)
        np.testing.assert_array_equal(r["corner"]["hist1d"][2], h)
        assert os.path.exists(r["corner_npz"])


WORKER = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["RB_ROOT"]); sys.path.insert(0, os.path.join(os.environ["RB_ROOT"], "tests"))
from test_gpu_chain_marginals import two_rank_run
lr = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
res = two_rank_run(lr)
if dist.get_rank() == 0:
    np.savez(os.environ["RB_OUT"], **res)
dist.destroy_process_group()
"""


def two_rank_run(device):
    """4 sources x 48 walkers, two run_mcmc calls: histograms, covariance, nearest samples."""
    from test_gpu_sampler import model2
    model, p0 = model2()
    ctx = _lib.Context(_lib.MolData(MOLFILE), device)
    pos = p0 + 0.02 * np.random.default_rng(3).standard_normal((192, 8))
    s = StretchSampler(192, 8, CudaEngine(ctx, [model] * 4), seed=11, nsources=4, split_block=8)
    s.run_mcmc(pos, 30)
    s.run_mcmc(None, 40)
    e, h1, h2, _ = s.get_histograms(20, discard=5, thin=2, columns=driver.summary_columns(2))
    x, i, d2 = s.get_nearest_sample(p0, discard=5)
    return dict(e=e, h1=h1, h2=h2, cov=s.get_covariance(discard=5), x=x, i=i, d2=d2)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs (NCCL refuses two ranks on one device)")
def test_nccl_two_ranks_match_single_process(tmp_path):
    want = two_rank_run(0)
    out = str(tmp_path / "marg2.npz")
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, RB_ROOT=ROOT, RB_OUT=out)
    subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                    "127.0.0.1", "--master-port", "29521", str(script)], check=True, env=env, timeout=600)
    got = np.load(out)
    for k, v in want.items():
        if k in ("cov", "d2"):
            np.testing.assert_allclose(got[k], v, rtol=1e-12, err_msg=k)
        else:
            np.testing.assert_array_equal(got[k], v, err_msg=k)
