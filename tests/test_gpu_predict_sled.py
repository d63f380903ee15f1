"""Posterior-predictive SLEDs on the GPU (csrc/predict_sled.cuh through rb_predict_sled_dev and
StretchSampler.get_predicted_fluxes / get_predictive_quantiles): per-sample fluxes against model_lvg through Radex, the
scheduled solve against the single launch, percentiles against np.percentile under ==, the total plane against the
stored log-probabilities, components out of range, the driver, two ranks."""
import ctypes as C
import io
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import MOLFILE, ROOT
from radex_emcee_b200 import _lib, driver
from radex_emcee_b200 import emcee_radex as er1
from radex_emcee_b200 import emcee_radex_2comp as er2
from radex_emcee_b200.data import DATA_DIR, get_source, read_data
from radex_emcee_b200.radex import Radex
from radex_emcee_b200.sampler import ChainView, CudaEngine, SLEDModel, StretchSampler
from test_chain_stats_cpu import QS
from test_gpu_sampler import model1, model2
from test_predict_sled_cpu import percentile_of_planes

pytestmark = pytest.mark.gpu

JUP = list(range(1, 12))
# model_lvg computes T, N and n(H2) with libm's pow, the kernels with CUDA's: the inputs of a solve can differ in the last
# bit, and the iteration's stop rule (sum |dx| < 1e-16) turns that into a difference of up to ~3e-11 of the brightest line of
# the SLED (measured on a B200; the weakest high-J lines, many decades fainter, carry it as a large relative error, most with
# the v1 solver)
HOST_RTOL = 1e-10


def assert_close_to_host(F, ref):
    """|F - ref| <= HOST_RTOL x the brightest line of the same sample's SLED, with the same NaNs."""
    peak = np.nanmax(np.abs(ref), axis=-1, keepdims=True)
    assert np.array_equal(np.isnan(F), np.isnan(ref))
    err = np.where(np.isnan(ref), 0.0, np.abs(F - ref))
    assert (err <= HOST_RTOL * peak).all(), float(np.nanmax(err / peak))


@pytest.fixture(scope="module")
def ctx():
    return _lib.Context(_lib.MolData(MOLFILE), 0)


def host_radex(tbg):
    return Radex(species="co", datapath=os.path.dirname(MOLFILE),
                 density={"oH2": er1.fortho * 1e10, "pH2": (1 - er1.fortho) * 1e10}, column=1e6, temperature=20.0,
                 tbackground=tbg, deltav=1.0, escapeProbGeom="lvg")


def host_components(R, jup, P, opts=None):
    """model_lvg of every component of the rows of P ([n, 4 ncomp]) -> [ncomp, n, nlines]; with opts, the same inputs
    and flux expression through rb_solve_batch under those opts."""
    out = []
    for c in range(P.shape[1] // 4):
        p = np.ascontiguousarray(P[:, 4 * c:4 * c + 4])
        if opts is None:
            out.append(np.atleast_2d(er1.model_lvg(jup, p, R)))
            continue
        R.set_params(density={"oH2": er1.fortho * 10. ** p[:, 0], "pH2": (1 - er1.fortho) * 10. ** p[:, 0]},
                     column=10. ** p[:, 2], temperature=10. ** p[:, 1])
        n, tk, dens, cd = R._batch_inputs()
        surf = np.empty((n, R.mol.nline))
        _lib.check(_lib.load().rb_solve_batch(R._ctx.handle, n, _lib.ptr(tk), _lib.ptr(dens), _lib.ptr(cd), 1.0, R.tbg,
                                              2, C.byref(opts), None, None, None, _lib.ptr(surf), None, None))
        out.append(surf[:, np.asarray(jup) - 1] * (10. ** p[:, 3])[:, None] * 1.0e23)
    return np.stack(out)


def planes_of(comp):
    return comp if comp.shape[0] == 1 else np.stack([comp[0] + comp[1], comp[0], comp[1]])


def injected(ctx, models, chunks, opts=None):
    """A sampler over `models` (one per source) whose stored chain is `chunks` ([steps, nwalkers, ndim] arrays)."""
    nw, ndim = chunks[0].shape[1:]
    if opts is not None:
        for m in models:
            m.opts = opts
    s = StretchSampler(nw, ndim, CudaEngine(ctx, models), nsources=len(models), randomize_split=False)
    s._chain = [torch.as_tensor(c, dtype=torch.float64).cuda().contiguous() for c in chunks]
    return s


def burnt_in(rng, p0, shape, spread=0.15):
    return p0 + spread * rng.standard_normal(shape + (p0.size,))


@pytest.mark.parametrize("ncomp", [1, 2])
def test_real_run_matches_host_model_and_log_prob(ctx, ncomp):
    """64 walkers x 30 steps of a flux.dat source: every predicted flux equals model_lvg through Radex at the source's
    tbg (assert_close_to_host), with the default opts and kernel = 1; the total plane at the observed lines rebuilds lnlike +
    lnprior of every stored sample to 1e-12."""
    model, p0 = model1() if ncomp == 1 else model2()
    ndim = 4 * ncomp
    s = StretchSampler(64, ndim, CudaEngine(ctx, model), seed=20170914)
    s.run_mcmc(p0 + 1e-3 * np.random.RandomState(1).randn(64, ndim), 12)
    s.run_mcmc(None, 18)
    P = s.get_chain(flat=True)
    R = host_radex(model.tbg)
    sampler_engine = s.engine
    for opts in (None, _lib.default_opts(kernel=1)):
        s.engine = sampler_engine if opts is None else CudaEngine(
            ctx, SLEDModel(ncomp, model.Jup, model.flux, model.eflux, model.bounds, model.tbg, model.T_d, opts=opts))
        F = s.get_predicted_fluxes(JUP, flat=True)
        ref = planes_of(host_components(R, JUP, P, opts))
        assert F.shape == ref.shape == ((1 if ncomp == 1 else 3), 30 * 64, len(JUP))
        assert_close_to_host(F, ref)
    # the likelihood the sampler stored, from the total plane at the observed lines, solved with the sampler's own opts
    s.engine = sampler_engine
    Fo = s.get_predicted_fluxes(model.Jup, flat=True)[0]
    e = np.maximum(np.abs(model.eflux), 1e-12)
    r = (model.flux - Fo) / e
    ll = -0.5 * (np.sum(r * r, axis=1) + 2.0 * np.sum(np.log(e)))
    lp = er1.lnprior(P, model.bounds) if ncomp == 1 else er2.lnprior(P, model.bounds, model.T_d)
    np.testing.assert_allclose(lp + ll, s.get_log_prob(flat=True), rtol=1e-12, atol=0)


def test_scheduled_solve_matches_single_launch(ctx):
    """12 288 models per call (2048 two-component walkers x 3 steps): the default schedule, park_max = 7 and the single
    launch (kernel = 3) give the same bits, and the same counters."""
    model, p0 = model2()
    rng = np.random.default_rng(2)
    X = burnt_in(rng, p0, (3, 2048))
    outs = []
    for kw in (dict(), dict(park_max=7), dict(kernel=3)):
        m, _ = model2()
        s = injected(ctx, [m], [X], opts=_lib.default_opts(**kw))
        view = s._chain_view(0, 1)
        cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
        F = s.engine.predict_sled(view, [4, 1, 9, 4], cnt).cpu().numpy()
        outs.append((F, cnt.cpu().numpy(), s.engine.ctx.counters()[0]))
    for F, cnt, iters in outs[1:]:
        assert F.tobytes() == outs[0][0].tobytes()
        np.testing.assert_array_equal(cnt, outs[0][1])
        assert iters == outs[0][2]
    assert outs[0][1].tolist() == [3 * 2048 * 2, 0] and np.isfinite(outs[0][0]).all()


def test_quantiles_three_sources(ctx):
    """Three sources with different tbg and 38 walkers each; discard / thin across chunk boundaries; unsorted and repeated
    J.  Quantiles == np.percentile of the gathered planes; per-sample fluxes == model_lvg at each source's tbg."""
    data = read_data(os.path.join(DATA_DIR, "flux.dat"))
    names = list(data)[:3]
    models = [model1(n)[0] for n in names]
    assert len({m.tbg for m in models}) == 3
    rng = np.random.default_rng(3)
    X = burnt_in(rng, model1()[1], (40, 3 * 38))
    chunks = [X[:7], X[7:8], X[8:30], X[30:]]
    s = injected(ctx, models, chunks)
    jup = [7, 2, 2, 11, 1]
    for discard, thin in ((0, 1), (5, 2), (6, 3), (29, 4)):
        F = s.get_predicted_fluxes(jup, discard=discard, thin=thin)
        got = s.get_predictive_quantiles(jup, QS, discard=discard, thin=thin)
        assert got.shape == (3, 1, len(QS), len(jup))
        assert np.array_equal(got, percentile_of_planes(F, 3, QS), equal_nan=True), (discard, thin)
    F = s.get_predicted_fluxes(jup, discard=5, thin=2)
    sel = X[6::2]
    for k, m in enumerate(models):
        P = sel[:, k * 38:(k + 1) * 38].reshape(-1, 4)
        ref = host_components(host_radex(m.tbg), jup, P)
        assert_close_to_host(F[0][:, k * 38:(k + 1) * 38].reshape(-1, len(jup)), ref[0])


def test_component_out_of_range(ctx):
    """One sample at T = 10^4.1 K: NaN in its component's plane and in the total, one count of a component out of
    range, a NaN column in its source's quantiles, as np.percentile gives."""
    model, p0 = model2()
    rng = np.random.default_rng(4)
    X = burnt_in(rng, p0, (6, 2 * 40))
    X[3, 45, 5] = 4.1                                       # source 1, warm component
    m2, _ = model2()
    s = injected(ctx, [model, m2], [X[:2], X[2:]])
    cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
    F = s.engine.predict_sled(s._chain_view(0, 1), JUP, cnt).cpu().numpy()
    assert cnt.cpu().tolist() == [6 * 80 * 2 - 1, 1]
    assert np.isnan(F[0, 3, 45]).all() and np.isnan(F[2, 3, 45]).all() and np.isfinite(F[1, 3, 45]).all()
    bad = np.isnan(F)
    assert bad.sum() == 2 * len(JUP)
    q = s.get_predictive_quantiles(JUP, [16, 50, 84])
    np.testing.assert_array_equal(q, percentile_of_planes(s.get_predicted_fluxes(JUP), 2, [16, 50, 84]))
    assert np.isnan(q[1, [0, 2]]).all() and np.isfinite(q[1, 1]).all() and np.isfinite(q[0]).all()


def test_entry_point_arguments_with_a_context(ctx):
    """The checks that need a context: J past the table, a set of another ncomp, a set without the view's sources."""
    model, _ = model1()
    eng = CudaEngine(ctx, model)
    X = torch.zeros((2, 8, 4), dtype=torch.float64, device="cuda")
    out = torch.empty(1024, dtype=torch.float64, device="cuda")
    L = _lib.load()

    def call(view, jup, engine=eng):
        j = (C.c_int32 * len(jup))(*jup)
        vs = view.c_struct()
        return L.rb_predict_sled_dev(ctx.handle, engine.srcset.handle, C.byref(vs), len(jup), j, None, out.data_ptr(),
                                     None)
    assert call(ChainView([X], 8, 4, 0, 8, 0, 1), [1, ctx.mol.nline]) == 0
    assert call(ChainView([X], 8, 4, 0, 8, 0, 1), [1, ctx.mol.nline + 1]) == -1
    assert call(ChainView([X], 8, 4, 0, 4, 0, 1), [1]) == -1     # walkers 4..7 belong to source 1: not in the set
    X8 = torch.zeros((2, 8, 8), dtype=torch.float64, device="cuda")
    assert call(ChainView([X8], 8, 8, 0, 8, 0, 1), [1]) == -1   # two components against a one-component set
    torch.cuda.synchronize()


def test_driver_sled_summary(tmp_path):
    data = read_data(os.path.join(DATA_DIR, "flux.dat"))
    kw = dict(ncomp=1, nwalkers=64, n_iter_burn=10, n_iter_walk=30, allow_synthetic=True)
    plain = driver.fit_source("G09v1.97", data, outdir=str(tmp_path / "a"), **kw)
    full = driver.fit_source("G09v1.97", data, outdir=str(tmp_path / "b"), predict_jup=JUP, **kw)
    lean = driver.fit_source("G09v1.97", data, outdir=str(tmp_path / "c"), predict_jup=JUP, chain_to_host=False, **kw)
    assert "sled_summary" not in plain and "sled_jup" not in plain
    assert set(full) - set(plain) == {"sled_jup", "sled_summary"}
    with open(plain["pickle"], "rb") as f, open(full["pickle"], "rb") as g:
        assert f.read() == g.read()                         # the pickle layout never changes
    np.testing.assert_array_equal(full["chain"], plain["chain"])
    assert lean["sled_summary"] == full["sled_summary"]
    np.testing.assert_array_equal(lean["sled_jup"], JUP)
    z = get_source("G09v1.97", data)[0]
    flux = host_components(host_radex(er1.source_setup(z)[0]), JUP, full["chain"].reshape(-1, 4))[0]
    ref = driver.percentile_summary(flux)
    (got,) = lean["sled_summary"]
    assert sorted(got) == JUP
    for J, r in zip(JUP, ref):
        np.testing.assert_allclose(got[J], r, rtol=1e-12, atol=1e-12 * abs(r[0]))
    buf_plain, buf_full = io.StringIO(), io.StringIO()
    driver.print_summary(plain, 1, file=buf_plain)
    driver.print_summary(lean, 1, file=buf_full)
    extra = buf_full.getvalue()[len(buf_plain.getvalue()):]
    assert buf_full.getvalue().startswith(buf_plain.getvalue())
    assert extra.count("xxx: J=") == len(JUP) and all(line.startswith("xxx:") for line in extra.splitlines())


WORKER = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["RB_ROOT"]); sys.path.insert(0, os.path.join(os.environ["RB_ROOT"], "tests"))
from test_gpu_predict_sled import two_rank_run
lr = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
F, q = two_rank_run(lr)
if dist.get_rank() == 0:
    np.savez(os.environ["RB_OUT"], F=F, q=q)
dist.destroy_process_group()
"""


def two_rank_run(device):
    """3 sources x 48 walkers of two components (with two ranks, source 1 spans both), two run_mcmc calls."""
    model, p0 = model2()
    ctx = _lib.Context(_lib.MolData(MOLFILE), device)
    pos = p0 + 0.02 * np.random.default_rng(3).standard_normal((144, 8))
    s = StretchSampler(144, 8, CudaEngine(ctx, [model] * 3), seed=11, nsources=3, split_block=8)
    s.run_mcmc(pos, 10)
    s.run_mcmc(None, 12)
    return s.get_predicted_fluxes([3, 1, 6], discard=3, thin=2), s.get_predictive_quantiles([3, 1, 6], QS, 3, 2)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs (NCCL refuses two ranks on one device)")
def test_nccl_two_ranks_match_single_process(tmp_path):
    F_ref, q_ref = two_rank_run(0)
    out = str(tmp_path / "sled2.npz")
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, RB_ROOT=ROOT, RB_OUT=out)
    subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                    "127.0.0.1", "--master-port", "29521", str(script)], check=True, env=env, timeout=600)
    got = np.load(out)
    assert got["F"].tobytes() == F_ref.tobytes()
    assert got["q"].tobytes() == q_ref.tobytes()
