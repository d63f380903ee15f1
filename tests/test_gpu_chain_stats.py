"""Device chain statistics (csrc/chain_stats.cuh through StretchSampler.get_quantiles / get_autocorr_time): exact
percentiles against np.percentile compared with ==, the kernels against their numpy restatement
(tests/test_chain_stats_cpu.py), emcee's integrated autocorrelation time, a real sampler run, the driver, two ranks."""
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import MOLFILE, ROOT
from radex_emcee_b200 import _lib, driver
from radex_emcee_b200.data import DATA_DIR, read_data
from radex_emcee_b200.sampler import AutocorrError, ChainView, CudaEngine, StretchSampler
from test_chain_stats_cpu import QS, StatsEngine, ar1_chain, emcee_integrated_time, percentile_ref
from test_gpu_sampler import model1

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    return _lib.Context(_lib.MolData(MOLFILE), 0)


def device_sampler(ctx, chunks, nsources=1):
    """A sampler whose stored chain is `chunks` (device or host arrays [steps, nwalkers, ndim])."""
    nw, ndim = chunks[0].shape[1:]
    m, _ = model1()
    s = StretchSampler(nw, ndim, CudaEngine(ctx, m), nsources=nsources, randomize_split=False)
    s._chain = [torch.as_tensor(c, dtype=torch.float64).cuda().contiguous() for c in chunks]
    return s


def test_quantiles_edge_values(ctx):
    """Ties, a constant column, mixed signs, +-0, +-inf, a NaN column; discard / thin across chunk boundaries."""
    rng = np.random.default_rng(3)
    T, nw, ndim = 61, 3 * 38, 5
    X = rng.standard_normal((T, nw, ndim)) * [1.0, 1e-3, 30.0, 1.0, 1e300] + [0.0, 5.0, -1.0, 0.0, 0.0]
    X[:, :, 3] = np.round(X[:, :, 3] * 2) / 2
    X[::3, ::5, 3] = -0.0
    X[:, 38:76, 1] = 7.25
    X[4, 80, 2], X[5, 81, 2], X[9, 3, 2] = np.inf, -np.inf, np.inf
    X[6, 100, 0] = np.nan
    chunks = [X[:7], X[7:8], X[8:30], X[30:]]
    s = device_sampler(ctx, chunks, nsources=3)
    cols = [0, 1, 2, 3, 4, (0, 1), (3, 3), (4, 4)]
    for discard, thin in ((0, 1), (5, 2), (6, 3), (29, 4), (0, 61)):
        got = s.get_quantiles(QS, discard=discard, thin=thin, columns=cols)
        ref = percentile_ref(chunks, 3, QS, cols, discard, thin)
        assert np.array_equal(got, ref, equal_nan=True), (discard, thin)
    assert np.isnan(s.get_quantiles(QS)[2, :, 0]).all()


def test_kernels_match_numpy_restatement(ctx):
    """Histogram counts bit for bit and moments / acf to rounding, for a rank that owns walkers [70, 70 + 190) of
    sources of 45 walkers (not a multiple of 32, a source split at both ends)."""
    rng = np.random.default_rng(5)
    nlocal, ndim, W, gid_base = 190, 4, 45, 70
    X = ar1_chain(rng, 90, nlocal, [0.2, 0.7, 0.9, 0.5])
    X[:, :, 3] = np.round(X[:, :, 3])
    parts = [X[:40], X[40:41], X[41:]]
    m, _ = model1()
    eng, ref = CudaEngine(ctx, m), StatsEngine(None)
    nsrc = (gid_base + nlocal - 1) // W + 1
    cols = [(0, -1), (1, -1), (3, -1), (1, 2)]
    for discard, thin in ((0, 1), (39, 2)):
        vd = ChainView([torch.from_numpy(p).cuda() for p in parts], nlocal, ndim, gid_base, W, discard, thin)
        vh = ChainView([torch.from_numpy(p) for p in parts], nlocal, ndim, gid_base, W, discard, thin)
        pre = np.zeros((nsrc, len(cols), 1), np.uint64)
        cd, nd = eng.chain_hist(vd, nsrc, cols, 0, pre)
        ch, nh = ref.chain_hist(vh, nsrc, cols, 0, pre)
        np.testing.assert_array_equal(cd.cpu().numpy(), ch.numpy())
        np.testing.assert_array_equal(nd.cpu().numpy(), nh.numpy())
        # pass 3 with two prefixes per column taken from real keys, one slot unused
        u = X[discard + thin - 1, 5, 0].view(np.uint64)
        key = ~u if u >> np.uint64(63) else u | np.uint64(1 << 63)
        pre = np.full((nsrc, len(cols), 3), np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64)
        pre[:, :, 0] = key >> np.uint64(40)
        pre[:, :, 1] = (key >> np.uint64(40)) ^ np.uint64(1)
        cd, _ = eng.chain_hist(vd, nsrc, cols, 3, pre)
        ch, _ = ref.chain_hist(vh, nsrc, cols, 3, pre)
        np.testing.assert_array_equal(cd.cpu().numpy(), ch.numpy())
        assert cd[:, 0, 0].sum() > 0
        md, c0d = eng.chain_moments(vd)
        mh, c0h = ref.chain_moments(vh)
        np.testing.assert_allclose(md.cpu().numpy(), mh.numpy(), rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(c0d.cpu().numpy(), c0h.numpy(), rtol=1e-12)
        for k0, k1 in ((0, vd.nsel), (3, 9)):
            rd = eng.chain_acf(vd, nsrc, md, c0d, k0, k1).cpu().numpy()
            rh = ref.chain_acf(vh, nsrc, md.cpu(), c0d.cpu(), k0, k1).numpy()
            np.testing.assert_allclose(rd, rh, rtol=1e-11, atol=1e-11)
            assert (rd[0] == 0).all()                      # source 0 has no walker on this rank


def test_quantiles_large_columns(ctx):
    """Two sources of 1000 walkers (not a multiple of 32), 16 800 steps: 2^24 values per column and source."""
    g = torch.Generator(device="cuda").manual_seed(11)
    T, W = 16800, 1000
    X = torch.randn((T, 2 * W, 4), generator=g, device="cuda", dtype=torch.float64)
    X[:, :, 2] = torch.round(X[:, :, 2] * 4)            # heavy ties
    X[:, W:, 3] *= -1e-7
    assert T * W >= 1 << 24
    s = device_sampler(ctx, [X[:9000], X[9000:]], nsources=2)
    cols = [0, 1, 2, 3, (0, 1)]
    got = s.get_quantiles(QS, discard=4000, thin=1, columns=cols)
    host = X.cpu().numpy()
    np.testing.assert_array_equal(got, percentile_ref([host], 2, QS, cols, 4000, 1))
    got = s.get_quantiles([16, 50, 84], columns=cols)
    np.testing.assert_array_equal(got, percentile_ref([host], 2, [16, 50, 84], cols))


def test_autocorr_time_matches_emcee(ctx):
    rng = np.random.default_rng(6)
    phis = [0.3, 0.8, 0.95, 0.0]
    X = ar1_chain(rng, 1500, 2 * 50, phis)
    chunks = [X[:250], X[250:260], X[260:]]
    s = device_sampler(ctx, chunks, nsources=2)
    for discard, thin in ((0, 1), (120, 1), (33, 2)):
        tau, win, n_t = s._integrated_time(discard, thin, 5)
        sel = X[discard + thin - 1::thin]
        for src in range(2):
            ref_tau, ref_win = emcee_integrated_time(sel[:, src * 50:(src + 1) * 50])
            np.testing.assert_array_equal(win[src], ref_win)
            np.testing.assert_allclose(tau[src], ref_tau, rtol=1e-10)
    a, b = s.get_autocorr_time(quiet=True), s.get_autocorr_time(quiet=True)
    assert a.tobytes() == b.tobytes()
    # AR(1): tau = (1 + phi) / (1 - phi); emcee's windowed estimate of 1500 steps x 50 walkers gets within 20 % for
    # phi <= 0.8 (for phi = 0.95 the window of 5 tau truncates noticeably and the estimate runs low)
    np.testing.assert_allclose(a[:, :2], np.broadcast_to([(1 + p) / (1 - p) for p in phis[:2]], (2, 2)), rtol=0.2)
    assert (a[:, 2] > 2 * a[:, 1]).all()
    # a stuck walker makes its source's tau NaN; a short chain raises (or warns with quiet)
    X[:, 7, 1] = 0.5
    s = device_sampler(ctx, [X], nsources=2)
    tau = s.get_autocorr_time(quiet=True)
    assert np.isnan(tau[0, 1]) and np.isfinite(tau[0, [0, 2, 3]]).all() and np.isfinite(tau[1]).all()
    s = device_sampler(ctx, [X[:80]], nsources=2)
    with pytest.raises(AutocorrError):
        s.get_autocorr_time()
    assert np.isfinite(s.get_autocorr_time(quiet=True)[:, 0]).all()


def test_real_sampler_run(ctx):
    """Config-1 shape (100 walkers, two run_mcmc calls): device percentiles == np.percentile of the host chain."""
    model, p0 = model1()
    pos = p0 + 1e-3 * np.random.RandomState(20170914).randn(100, 4)
    s = StretchSampler(100, 4, CudaEngine(ctx, model), seed=20170914)
    s.run_mcmc(pos, 60)
    s.run_mcmc(None, 90)
    assert len(s._chain) == 2
    cols = [0, 1, 2, 3, (0, 1)]
    for discard, thin in ((0, 1), (50, 3), (61, 1)):
        flat = s.get_chain(flat=True, discard=discard, thin=thin)
        cc = np.column_stack([flat, flat[:, 0] + flat[:, 1]])
        np.testing.assert_array_equal(s.get_quantiles(QS, discard=discard, thin=thin, columns=cols)[0],
                                      np.percentile(cc, QS, axis=0))
    tau = s.get_autocorr_time(quiet=True)
    assert tau.shape == (1, 4) and (tau > 1).all()


def test_driver_summaries(tmp_path):
    data = read_data(os.path.join(DATA_DIR, "flux.dat"))
    kw = dict(ncomp=1, nwalkers=64, n_iter_burn=10, n_iter_walk=30, allow_synthetic=True)
    res = driver.fit_source("G09v1.97", data, outdir=str(tmp_path / "a"), **kw)
    flat = res["chain"].reshape(-1, 4)
    ref = driver.posterior_summary(flat, 1)
    assert res["summary"] == ref
    for key in ref[0]:
        assert [type(v) for v in res["summary"][0][key]] == [type(v) for v in ref[0][key]]
    np.testing.assert_array_equal(res["theta_med"], np.percentile(flat, 50, axis=0))
    assert res["autocorr_time"].shape == (4,)
    with open(res["pickle"], "rb") as f:
        tup = pickle.load(f)
    np.testing.assert_array_equal(tup[6], res["theta_med"])
    np.testing.assert_array_equal(tup[-1][0], res["chain"])
    lean = driver.fit_source("G09v1.97", data, outdir=str(tmp_path / "b"), chain_to_host=False, **kw)
    assert lean["chain"] is None and lean["lnprobability"] is None
    assert lean["summary"] == ref
    np.testing.assert_array_equal(lean["theta_med"], res["theta_med"])
    with open(lean["pickle"], "rb") as f:
        assert pickle.load(f)[-1] == (None, None)
    out = driver.fit_sources_concurrently(list(data)[:2], data, ncomp=1, nwalkers=40, n_iter_burn=5, n_iter_walk=12,
                                          allow_synthetic=True)
    for r in out:
        assert r["summary"] == driver.posterior_summary(r["chain"].reshape(-1, 4), 1)
        assert r["autocorr_time"].shape == (4,)


WORKER = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["RB_ROOT"]); sys.path.insert(0, os.path.join(os.environ["RB_ROOT"], "tests"))
from test_gpu_chain_stats import two_rank_run
lr = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
q, tau = two_rank_run(lr)
if dist.get_rank() == 0:
    np.savez(os.environ["RB_OUT"], q=q, tau=tau)
dist.destroy_process_group()
"""


def two_rank_run(device):
    """4 sources x 48 walkers, two run_mcmc calls: quantiles and tau."""
    from test_gpu_sampler import model2
    model, p0 = model2()
    ctx = _lib.Context(_lib.MolData(MOLFILE), device)
    pos = p0 + 0.02 * np.random.default_rng(3).standard_normal((192, 8))
    s = StretchSampler(192, 8, CudaEngine(ctx, [model] * 4), seed=11, nsources=4, split_block=8)
    s.run_mcmc(pos, 30)
    s.run_mcmc(None, 40)
    q = s.get_quantiles(QS, discard=5, thin=2, columns=driver.summary_columns(2))
    return q, s.get_autocorr_time(quiet=True)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs (NCCL refuses two ranks on one device)")
def test_nccl_two_ranks_match_single_process(tmp_path):
    q_ref, tau_ref = two_rank_run(0)
    out = str(tmp_path / "stats2.npz")
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, RB_ROOT=ROOT, RB_OUT=out)
    subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                    "127.0.0.1", "--master-port", "29519", str(script)], check=True, env=env, timeout=600)
    got = np.load(out)
    np.testing.assert_array_equal(got["q"], q_ref)
    np.testing.assert_allclose(got["tau"], tau_ref, rtol=1e-12)
