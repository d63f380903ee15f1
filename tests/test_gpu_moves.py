"""Device moves beyond the stretch move: the DE propose / k-group accept kernels vs their numpy restatement
(tests/ref_moves.py), rb_moves_run_dev with one stretch move == rb_stretch_run_dev, DE and DE / stretch mixtures in the
library loop == the per-sub-step calls == the CPU reference sampler (oracle lnprob), sources kept apart, NCCL ranks."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import ref_engine
import ref_moves
from conftest import MOLFILE, ROOT
from radex_emcee_b200 import _lib
from radex_emcee_b200.data import get_source, read_data
from radex_emcee_b200 import emcee_radex as er1
from radex_emcee_b200.moves import DEMove, StretchMove
from radex_emcee_b200.sampler import CudaEngine, SLEDModel, SplitSpec, StretchSampler
from test_gpu_sampler import model1, model2

pytestmark = pytest.mark.gpu

MIX = [(DEMove(), 0.8), (StretchMove(), 0.2)]


@pytest.fixture(scope="module")
def ctx():
    return _lib.Context(_lib.MolData(MOLFILE), 0)


@pytest.mark.parametrize("N,W,B,randomize,gid_base,nlocal", [
    (100, 100, 100, True, 0, 100), (96, 48, 12, True, 48, 48), (4096, 4096, 512, True, 1024, 2048),
    (64, 64, 2, False, 32, 32), (1 << 16, 1 << 15, 1 << 12, True, 0, 1 << 16)])
def test_de_kernels_match_numpy(ctx, N, W, B, randomize, gid_base, nlocal):
    """rb_de_propose_dev / rb_group_accept_dev against the restatement, bit for bit: Q, source rows, X, lnp, per-walker
    acceptance counters and the NaN count (the Gaussian uses IEEE operations only, so gamma is exact as well)."""
    eng = CudaEngine(ctx, model1()[0])
    rng = np.random.default_rng(N + B)
    ndim = 4
    Xall = rng.standard_normal((N, ndim))
    X = Xall[gid_base:gid_base + nlocal].copy()
    sp = SplitSpec(N, W, B, randomize, 0xC0FFEE1234567)
    Xalld = torch.from_numpy(Xall).cuda()
    if B < 3:           # a block of 2 walkers would leave a DE group empty: refused
        with pytest.raises(_lib.RadexB200Error, match="blocks of >= 3"):
            eng.de_propose(sp, 0, 0, gid_base, torch.from_numpy(X).cuda(), Xalld, 1.0, 1e-5)
    for step in (0, 7, 2 ** 34 + 3):
        for g in range(3 if B >= 3 else 0):
            ns = ref_moves.nslots(sp, nlocal, 3, g)
            Xd = torch.from_numpy(X).cuda()
            for g0, sig in ((1.2, 1e-5), (0.5, 0.3)):
                Q, src = eng.de_propose(sp, step, g, gid_base, Xd, Xalld, g0, sig)
                Qn, srcn, i, gam, n, w1, w2 = ref_moves.de_propose_np(sp, step, g, gid_base, X, Xall, g0, sig)
                np.testing.assert_array_equal(Q.cpu().numpy(), Qn)
                np.testing.assert_array_equal(src.cpu().numpy(), srcn)
            assert (w1 // W == srcn).all() and (w2 // W == srcn).all() and (w1 != w2).all()
            lnp = rng.standard_normal(nlocal)
            lnp_new = lnp[i] + rng.standard_normal(ns)
            lnp_new[::11] = -np.inf
            lnp_new[5::29] = np.nan
            X2, l2 = Xd.clone(), torch.from_numpy(lnp).cuda()
            nacc = torch.zeros(nlocal, dtype=torch.int64, device="cuda")
            cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
            eng.group_accept(sp, _lib.RB_MOVE_DE, step, g, 3, gid_base, X2, l2, Q, torch.from_numpy(lnp_new).cuda(), None,
                             nacc, cnt)
            Xn, ln, nn = X.copy(), lnp.copy(), np.zeros(nlocal, np.int64)
            acc, nnan = ref_moves.group_accept_np(sp, ref_moves.RB_MOVE_DE, step, g, 3, gid_base, Xn, ln, Qn, lnp_new, None, nn)
            np.testing.assert_array_equal(X2.cpu().numpy(), Xn)
            np.testing.assert_array_equal(l2.cpu().numpy(), ln)
            np.testing.assert_array_equal(nacc.cpu().numpy(), nn)
            assert int(cnt[0].item()) == nnan == np.isnan(lnp_new).sum() and acc.sum() > ns // 20
        # the k-group accept with the stretch stream and two groups is rb_stretch_accept2_dev
        Xd = torch.from_numpy(X).cuda()
        Call = torch.from_numpy(rng.standard_normal((N // 2, ndim))).cuda()
        Q, lf, _ = eng.propose2(sp, step, 1, gid_base, Xd, Call, 2.0)
        lnp_new = torch.from_numpy(rng.standard_normal(nlocal // 2)).cuda()
        l0 = torch.from_numpy(rng.standard_normal(nlocal)).cuda()
        outs = []
        for f in ("accept2", "group"):
            X2, l2 = Xd.clone(), l0.clone()
            nacc = torch.zeros(nlocal, dtype=torch.int64, device="cuda")
            cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
            if f == "accept2":
                eng.accept2(sp, step, 1, gid_base, X2, l2, Q, lnp_new, lf, nacc, cnt)
            else:
                eng.group_accept(sp, _lib.RB_MOVE_STRETCH, step, 1, 2, gid_base, X2, l2, Q, lnp_new, lf, nacc, cnt)
            outs.append((X2.cpu().numpy(), l2.cpu().numpy(), nacc.cpu().numpy()))
        for a, b in zip(*outs):
            np.testing.assert_array_equal(a, b)
    # only (stretch, 2 groups) and (DE, 3 groups) have a random stream of their own per group
    for kind, ng in ((_lib.RB_MOVE_STRETCH, 3), (_lib.RB_MOVE_DE, 2), (_lib.RB_MOVE_DE, 5), (7, 2)):
        with pytest.raises(_lib.RadexB200Error, match="bad argument"):
            eng.group_accept(sp, kind, 0, 0, ng, gid_base, Xd, l0, Q, lnp_new, lf, nacc, cnt)


def _run(ctx, models, nw, nsteps, seed, moves, pos, nsources=1, native=True, **kw):
    s = StretchSampler(nw, models[0].ndim, CudaEngine(ctx, models if nsources > 1 else models[0]), seed=seed,
                       nsources=nsources, moves=moves, native=native, **kw)
    assert s.native == native
    s.run_mcmc(pos, nsteps)
    return s


@pytest.mark.parametrize("spec", [0, -1])
def test_one_stretch_move_equals_the_stretch_loop(ctx, spec):
    """rb_moves_run_dev([stretch]) is rb_stretch_run_dev: same chain, log-probabilities and counters, with and without the
    speculative second half-step, one source and four."""
    data = read_data(ROOT + "/data/flux.dat")
    for nsrc in (1, 4):
        models, starts = [], []
        for k, nm in enumerate(list(data)[:nsrc]):
            z, lw, jup, flux, eflux = get_source(nm, data)
            tbg, ra, bounds, p0 = er1.source_setup(z)
            models.append(SLEDModel(1, jup, flux, eflux, bounds, tbg, opts=_lib.default_opts(spec_half=spec)))
            starts.append(p0 + 0.02 * np.random.default_rng(11 + k).standard_normal((24, 4)))
        pos = np.vstack(starts)
        out = []
        for moves in (None, StretchMove(), [(StretchMove(), 1.0)]):
            s = _run(ctx, models, 24 * nsrc, 15, 9, moves, pos, nsources=nsrc)
            s.run_mcmc(None, 4)              # a second call: the captured graph is replayed
            out.append((s.get_chain(), s.get_log_prob(), s.acceptance_fraction, s.total_solves))
        for o in out[1:]:
            for a, b in zip(out[0], o):
                np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize("moves", ["de", "mix"])
def test_de_chain_matches_cpu_reference_sampler(ctx, oracle, moves):
    """Config 1 shortened (64 walkers x 12 steps) with DE and with a DE 0.8 / stretch 0.2 mixture: the in-library loop
    (one CUDA graph per move) equals the per-sub-step calls bit for bit, and against the CPU reference sampler (oracle
    lnprob, same streams) >= 95 % of the walker-steps agree to 1e-9 and the medians to 0.01 dex."""
    model, p0 = model1()
    mv = DEMove() if moves == "de" else MIX
    nw, nsteps = 64, 12
    pos = p0 + 1e-3 * np.random.default_rng(20170914).standard_normal((nw, 4))
    gpu = _run(ctx, [model], nw, nsteps, 42, mv, pos)
    py = _run(ctx, [model], nw, nsteps, 42, mv, pos, native=False)
    np.testing.assert_array_equal(gpu.get_chain(), py.get_chain())
    np.testing.assert_array_equal(gpu.get_log_prob(), py.get_log_prob())
    np.testing.assert_array_equal(gpu.acceptance_fraction, py.acceptance_fraction)
    cpu = StretchSampler(nw, 4, ref_moves.MovesNumpyEngine(
        ref_engine.oracle_lnprob1(oracle, model.Jup, model.flux, model.eflux, model.bounds, model.tbg)), seed=42, moves=mv)
    cpu.run_mcmc(pos, nsteps)
    cg, cc = gpu.get_chain(), cpu.get_chain()
    same = np.isclose(cg, cc, rtol=0, atol=1e-9).all(axis=2)
    assert same.mean() > 0.95, same.mean()
    assert np.abs(np.median(cg[-1], axis=0) - np.median(cc[-1], axis=0)).max() < 0.01
    assert np.abs(gpu.get_log_prob() - cpu.get_log_prob())[same].max() < 1e-4
    assert gpu.acceptance_fraction.mean() > 0.05
    # reset / thin, then a second run_mcmc call replays the captured graphs
    gpu.reset()
    gpu.run_mcmc(None, 6, thin=2)
    py.reset()
    py.run_mcmc(None, 6, thin=2)
    assert gpu.get_chain().shape == (3, nw, 4)
    np.testing.assert_array_equal(gpu.get_chain(), py.get_chain())


def test_two_component_de_chain_with_dust_prior(ctx, oracle):
    """emcee_radex_2comp.py's 8-parameter posterior (T_cold ~ N(T_d, T_d), T_cold < T_warm, size_cold >= size_warm)
    with the DE / stretch mixture: 48 walkers x 8 steps vs the CPU reference sampler."""
    model, p0 = model2()
    nw, nsteps = 48, 8
    pos = p0 + 1e-3 * np.random.default_rng(7).standard_normal((nw, 8))
    gpu = _run(ctx, [model], nw, nsteps, 5, MIX, pos)
    cpu = StretchSampler(nw, 8, ref_moves.MovesNumpyEngine(
        ref_engine.oracle_lnprob2(oracle, model.Jup, model.flux, model.eflux, model.bounds, model.T_d, model.tbg)), seed=5,
        moves=MIX)
    cpu.run_mcmc(pos, nsteps)
    cg, cc = gpu.get_chain(), cpu.get_chain()
    same = np.isclose(cg, cc, rtol=0, atol=1e-9).all(axis=2)
    assert same.mean() > 0.9, same.mean()
    assert np.abs(np.median(cg[-1], axis=0) - np.median(cc[-1], axis=0)).max() < 0.01
    assert np.abs(gpu.get_log_prob() - cpu.get_log_prob())[same].max() < 1e-4
    assert 0.05 < gpu.acceptance_fraction.mean() < 0.95


def test_de_partners_stay_in_their_source(ctx):
    """Five sources in one DE ensemble: every sub-ensemble's chain is the chain that source has in an ensemble of copies
    of itself (same global ids, same split) -- no partner is ever drawn from another source."""
    data = read_data(ROOT + "/data/flux.dat")
    names = list(data)[:5]
    W, nsteps = 42, 6
    models, starts = [], []
    for k, nm in enumerate(names):
        m, p0 = model1(nm)
        models.append(m)
        starts.append(p0 + 1e-3 * np.random.default_rng(100 + k).standard_normal((W, 4)))
    allsrc = _run(ctx, models, W * len(names), nsteps, 9, MIX, np.vstack(starts), nsources=len(names))
    chain, lnp = allsrc.get_chain(), allsrc.get_log_prob()
    assert np.isfinite(lnp).all()
    for k, m in enumerate(models):
        ref = _run(ctx, [m] * len(names), W * len(names), nsteps, 9, MIX, np.vstack([starts[k]] * len(names)),
                   nsources=len(names), native=False)
        np.testing.assert_array_equal(ref.get_chain()[:, k * W:(k + 1) * W], chain[:, k * W:(k + 1) * W])
        np.testing.assert_array_equal(ref.get_log_prob()[:, k * W:(k + 1) * W], lnp[:, k * W:(k + 1) * W])


WORKER = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["RB_ROOT"]); sys.path.insert(0, os.path.join(os.environ["RB_ROOT"], "tests"))
from test_gpu_sampler import model2
from radex_emcee_b200 import _lib
from radex_emcee_b200.moves import DEMove, StretchMove
from radex_emcee_b200.sampler import CudaEngine, StretchSampler
lr = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
model, p0 = model2()
nw = 4096
pos = p0 + 0.02 * np.random.default_rng(3).standard_normal((nw, 8))
ctx = _lib.Context(_lib.MolData(os.path.join(os.environ["RB_ROOT"], "radex_emcee_b200", "data", "co.dat")), lr)
s = StretchSampler(nw, 8, CudaEngine(ctx, model), seed=11, moves=[(DEMove(), 0.8), (StretchMove(), 0.2)])
s.run_mcmc(pos, 4)
chain, lnp, acc = s.get_chain(), s.get_log_prob(), s.acceptance_fraction
if dist.get_rank() == 0:
    np.savez(os.environ["RB_OUT"], chain=chain, lnp=lnp, acc=acc)
dist.destroy_process_group()
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs (NCCL refuses two ranks on one device)")
def test_nccl_two_ranks_match_single_process(ctx, tmp_path):
    """A DE / stretch mixture with the walkers sharded over two ranks (one NCCL all-gather of X per DE sub-step) == the
    single-process chain (library loop), bit for bit."""
    model, p0 = model2()
    nw = 4096
    pos = p0 + 0.02 * np.random.default_rng(3).standard_normal((nw, 8))
    ref = StretchSampler(nw, 8, CudaEngine(ctx, model), seed=11, moves=MIX)
    ref.run_mcmc(pos, 4)
    out = str(tmp_path / "nccl2.npz")
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, RB_ROOT=ROOT, RB_OUT=out)
    subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                    "127.0.0.1", "--master-port", "29519", str(script)], check=True, env=env, timeout=600)
    got = np.load(out)
    np.testing.assert_array_equal(got["chain"], ref.get_chain())
    np.testing.assert_array_equal(got["lnp"], ref.get_log_prob())
    np.testing.assert_array_equal(got["acc"], ref.acceptance_fraction)
