"""Moves beyond the stretch move on CPU: the k-group split, the move schedule (restatement == rb_move_schedule, which
needs no device), the DE and mixture samplers on a correlated Gaussian, gloo world_size 2 == one process, argument
errors and the rb_move layout."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

import ref_engine
import ref_moves
from conftest import ROOT
from radex_emcee_b200 import _lib
from radex_emcee_b200.moves import DEMove, StretchMove, normalize_moves, parse_moves
from radex_emcee_b200.sampler import SplitSpec, StretchSampler

SECOND_FORM_SHAPES = [(100, 100, 100, True, 0, 100), (96, 48, 12, True, 48, 48), (4096, 4096, 512, True, 1024, 2048),
                      (64, 64, 2, False, 32, 32), (1 << 16, 1 << 15, 1 << 12, True, 0, 1 << 16)]


@pytest.mark.parametrize("N,W,B,randomize,gid_base,nlocal", SECOND_FORM_SHAPES)
def test_two_group_split_is_the_red_blue_split(N, W, B, randomize, gid_base, nlocal):
    sp = SplitSpec(N, W, B, randomize, 0xC0FFEE1234567)
    for step in (0, 7, 2 ** 34 + 3):
        for half in (0, 1):
            k = np.arange(nlocal // 2)
            np.testing.assert_array_equal(ref_moves.slot_walker(sp, step, half, 2, gid_base, k),
                                          ref_engine.slot_walker(sp, step, half, gid_base, k))


@pytest.mark.parametrize("N,W,B", [(96, 48, 12), (100, 100, 100), (64, 32, 8), (4096, 2048, 512), (40, 20, 10)])
def test_three_group_split(N, W, B):
    """emcee's DE labelling (arange(N) % 3, shuffled): per block a partition into groups of B // 3 + (g < B % 3) walkers,
    new every step, inside each source; B need not be a multiple of 3."""
    sp = SplitSpec(N, W, B, True, 1234)
    sizes = [B // 3 + (g < B % 3) for g in range(3)]
    labels = []
    for step in range(5):
        lab = np.full(N, -1)
        for g in range(3):
            i = ref_moves.slot_walker(sp, step, g, 3, 0, np.arange(N // B * sizes[g]))
            assert (lab[i] == -1).all()
            lab[i] = g
            # slot order: block by block, so slot k of group g lies in block k // n_g
            np.testing.assert_array_equal(i // B, np.arange(i.size) // sizes[g])
        assert (lab >= 0).all()
        for g in range(3):
            assert ((lab.reshape(-1, B) == g).sum(axis=1) == sizes[g]).all()
        # a rank owning the second half evaluates the same labelling
        if (N // 2) % B == 0:
            for g in range(3):
                full = ref_moves.slot_walker(sp, step, g, 3, 0, np.arange(N // B * sizes[g]))
                j = ref_moves.slot_walker(sp, step, g, 3, N // 2, np.arange(N // 2 // B * sizes[g])) + N // 2
                np.testing.assert_array_equal(j, full[full.size // 2:])
        labels.append(lab)
    assert any((labels[0] != l).any() for l in labels[1:])
    # partners stay in the walker's source and in the other two groups
    X = np.arange(N, dtype=np.float64)[:, None] * np.ones((1, 2))
    for g in range(3):
        _, src, i, _, _, w1, w2 = ref_moves.de_propose_np(sp, 3, g, 0, X, X, 1.0, 1e-5)
        lab3 = np.full(N, -1)
        for h in range(3):
            lab3[ref_moves.slot_walker(sp, 3, h, 3, 0, np.arange(N // B * sizes[h]))] = h
        assert (w1 != w2).all()
        assert (w1 // W == src).all() and (w2 // W == src).all() and (i // W == src).all()
        assert (lab3[w1] != g).all() and (lab3[w2] != g).all()
        assert len(np.unique(w1)) > 0.5 * min(len(w1), W - N // B * sizes[g])


def test_unrandomized_de_split_block(monkeypatch):
    """DE without randomize_split: a block of 6 where it divides the sub-ensemble and every rank's share, one block per
    sub-ensemble where a rank holds whole sub-ensembles, a clear error otherwise."""
    mu, cov, lnprob = corr_gauss()
    eng = ref_moves.MovesNumpyEngine(lnprob)
    assert StretchSampler(48, 8, eng, moves=DEMove(), randomize_split=False).split.block == 6
    assert StretchSampler(40, 8, eng, moves=DEMove(), randomize_split=False).split.block == 40
    import radex_emcee_b200.sampler as smod

    class FakeDist:
        ReduceOp = None

        @staticmethod
        def get_world_size(group=None):
            return 2

        @staticmethod
        def get_rank(group=None):
            return 0
    monkeypatch.setattr(smod.torch.distributed, "is_initialized", lambda: True)
    monkeypatch.setattr(smod.torch.distributed, "get_world_size", FakeDist.get_world_size)
    monkeypatch.setattr(smod.torch.distributed, "get_rank", FakeDist.get_rank)
    assert StretchSampler(48, 8, eng, moves=DEMove(), randomize_split=False).split.block == 6     # 24 per rank
    with pytest.raises(ValueError, match="pass split_block"):
        StretchSampler(40, 8, eng, moves=DEMove(), randomize_split=False)                       # 20 per rank, W = 40
    assert StretchSampler(40, 8, eng, moves=DEMove(), randomize_split=False, split_block=4).split.block == 4


def test_unrandomized_three_group_split_is_emcee_labelling():
    sp = SplitSpec(48, 48, 6, False, 0)
    for g in range(3):
        np.testing.assert_array_equal(ref_moves.slot_walker(sp, 5, g, 3, 0, np.arange(16)), g + 3 * np.arange(16))


def test_ln_rn_and_gauss():
    x = np.concatenate([np.linspace(1e-300, 1, 10001)[1:-1], [0.5, 0.25, 1e-10, 0.7071067811865476, 0.9999999]])
    np.testing.assert_allclose(ref_moves.ln_rn(x), np.log(x), rtol=4e-16, atol=0)
    n = ref_moves.de_gauss(np.arange(200000, dtype=np.uint64), 3, 1, *ref_moves.de_keys(77))
    assert abs(n.mean()) < 0.01 and abs(n.std() - 1) < 0.01
    assert abs(np.mean(n ** 4) - 3) < 0.1 and (np.abs(n) > 3).mean() == pytest.approx(0.0027, abs=0.0008)


def test_schedule():
    w = [0.8, 0.2, 0.0, 1.0]
    s = ref_moves.schedule_np(99, 0, 100000, w)
    counts = np.bincount(s, minlength=4)
    assert counts[2] == 0
    p = np.array([0.8, 0.2, 1.0]) / 2.0
    obs = counts[[0, 1, 3]]
    chi2 = (((obs - 1e5 * p) ** 2) / (1e5 * p)).sum()
    assert chi2 < 13.8, chi2                        # 99.9 % point of chi^2 with 2 degrees of freedom
    assert (ref_moves.schedule_np(5, 17, 1000, [3.0]) == 0).all()
    # the library draws the same schedule (host only: no device needed), from any step on
    for seed, step0, ww in ((99, 0, w), (2 ** 63 + 12345, 2 ** 40, [1.0, 1.0]), (7, 3, [0.25, 0.5, 0.25]), (1, 0, [2.0])):
        np.testing.assert_array_equal(_lib.move_schedule(seed, step0, 5000, ww), ref_moves.schedule_np(seed, step0, 5000, ww))
    np.testing.assert_array_equal(_lib.move_schedule(99, 40, 10, w), ref_moves.schedule_np(99, 0, 50, w)[40:])
    for bad in ([0.0, 0.0], [-1.0, 2.0], [np.nan], [np.inf, 1.0], [1.0] * 9):
        with pytest.raises(_lib.RadexB200Error):
            _lib.move_schedule(1, 0, 10, bad)


def corr_gauss():
    rng = np.random.default_rng(4)
    A = rng.standard_normal((8, 8))
    cov = A @ A.T / 8 + 0.05 * np.eye(8)
    mu = rng.standard_normal(8)
    P = np.linalg.inv(cov)

    def lnprob(X):
        d = np.atleast_2d(X) - mu
        return -0.5 * np.einsum("ij,jk,ik->i", d, P, d)
    return mu, cov, lnprob


def _tau(x):
    """Integrated autocorrelation time of the walker-mean series (emcee's estimator, c = 5)."""
    f = np.zeros(x.shape[0])
    for w in range(x.shape[1]):
        y = x[:, w] - x[:, w].mean()
        n = 2 ** int(np.ceil(np.log2(2 * len(y))))
        a = np.fft.ifft(np.abs(np.fft.fft(y, n)) ** 2)[:len(y)].real
        f += a / a[0]
    f /= x.shape[1]
    taus = 2.0 * np.cumsum(f) - 1.0
    m = np.arange(len(taus)) < 5.0 * taus
    return taus[np.argmin(m)] if not m.all() else taus[-1]


@pytest.mark.parametrize("moves", [DEMove(), [(DEMove(), 0.8), (StretchMove(), 0.2)]])
def test_samplers_on_a_correlated_gaussian(moves):
    mu, cov, lnprob = corr_gauss()
    nw, nsteps, burn = 64, 2500, 500
    p0 = mu + 0.1 * np.random.default_rng(1).standard_normal((nw, 8))
    s = StretchSampler(nw, 8, ref_moves.MovesNumpyEngine(lnprob), seed=21, moves=moves)
    s.run_mcmc(p0, nsteps)
    c = s.get_chain(discard=burn)
    tau = max(_tau(c[:, :, d]) for d in range(8))
    neff = c.shape[0] * nw / tau
    assert neff > 2000, (tau, neff)
    flat = c.reshape(-1, 8)
    sd = np.sqrt(np.diag(cov))
    assert (np.abs(flat.mean(axis=0) - mu) / sd).max() < 5 / np.sqrt(neff)
    got = np.cov(flat, rowvar=False)
    # standard error of a covariance entry ~ sqrt((S_ii S_jj + S_ij^2) / neff)
    se = np.sqrt((np.outer(np.diag(cov), np.diag(cov)) + cov ** 2) / neff)
    assert (np.abs(got - cov) / se).max() < 5
    af = s.acceptance_fraction
    assert af.shape == (nw,) and 0.1 < af.mean() < 0.9


def _worker(rank, world, port, nw, nsteps, seed, out, kw):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        s = _chain(nw, nsteps, seed, **kw)
        assert s.world == world
        chain, lnp, acc = s.get_chain(), s.get_log_prob(), s.acceptance_fraction
        if rank == 0:
            np.savez(out, chain=chain, lnp=lnp, acc=acc)
    finally:
        dist.destroy_process_group()


def _chain(nw, nsteps, seed, moves, **kw):
    mu, cov, lnprob = corr_gauss()
    p0 = mu + 0.3 * np.random.default_rng(5).standard_normal((nw, 8))
    mv = {"de": DEMove(), "mix": [(DEMove(), 0.8), (StretchMove(), 0.2)], "de_g": DEMove(sigma=0.1, gamma0=0.5)}[moves]
    s = StretchSampler(nw, 8, ref_moves.MovesNumpyEngine(lnprob), seed=seed, moves=mv, **kw)
    s.run_mcmc(p0, nsteps)
    return s


@pytest.mark.parametrize("kw", [dict(moves="de", split_block=8), dict(moves="mix", split_block=12),
                                dict(moves="de", randomize_split=False), dict(moves="de_g", split_block=24)])
def test_world_size_2_matches_single_process(tmp_path, kw):
    """DE and a DE / stretch mixture sharded over two gloo ranks (one all-gather of X per DE sub-step) give the
    single-process chain bit for bit; split blocks of 8 and 12 walkers (8 is not a multiple of 3)."""
    nw, nsteps, seed = 48, 20, 77
    ref = _chain(nw, nsteps, seed, **kw)
    assert np.isfinite(ref.get_log_prob()).all() and ref.acceptance_fraction.mean() > 0
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    out = str(tmp_path / "w2.npz")
    mp.spawn(_worker, args=(2, port, nw, nsteps, seed, out, kw), nprocs=2, join=True)
    got = np.load(out)
    np.testing.assert_array_equal(got["chain"], ref.get_chain())
    np.testing.assert_array_equal(got["lnp"], ref.get_log_prob())
    np.testing.assert_array_equal(got["acc"], ref.acceptance_fraction)


def test_one_stretch_move_is_the_default_chain():
    mu, cov, lnprob = corr_gauss()
    p0 = mu + 0.3 * np.random.default_rng(5).standard_normal((32, 8))
    chains = []
    for moves in (None, StretchMove(), [StretchMove()], [(StretchMove(), 3.0)]):
        s = StretchSampler(32, 8, ref_engine.NumpyEngine(lnprob) if moves is None else ref_moves.MovesNumpyEngine(lnprob),
                           seed=3, moves=moves)
        s.run_mcmc(p0, 15)
        chains.append(s.get_chain())
    for c in chains[1:]:
        np.testing.assert_array_equal(c, chains[0])


def test_argument_errors():
    mu, cov, lnprob = corr_gauss()
    eng = ref_moves.MovesNumpyEngine(lnprob)
    for bad in ([(DEMove(), -1.0)], [(DEMove(), 0.0), (StretchMove(), 0.0)], ["de"], "stretch", [(DEMove(), np.nan)],
                [], [StretchMove()] * 9, [(DEMove(), 1.0, 2.0)], 3):
        with pytest.raises(ValueError):
            StretchSampler(48, 8, eng, moves=bad)
    with pytest.raises(ValueError):
        StretchMove(a=1.0)
    with pytest.raises(ValueError):
        DEMove(sigma=-1.0)
    with pytest.raises(ValueError):
        DEMove(gamma0=0.0)
    # a group whose complement holds fewer than 2 walkers of its source
    with pytest.raises(ValueError, match="DEMove"):                          # blocks of < 3 walkers: an empty group
        StretchSampler(48, 8, eng, moves=DEMove(), split_block=2)
    StretchSampler(48, 8, eng, moves=StretchMove(), split_block=2)           # fine for the stretch move

    assert [type(m).__name__ for m, _ in parse_moves(["de:0.8", "stretch:0.2"])] == ["DEMove", "StretchMove"]
    assert [w for _, w in parse_moves(["de:0.8", "stretch:0.2"])] == [0.8, 0.2]
    assert [w for _, w in normalize_moves([DEMove(), StretchMove()])] == [1.0, 1.0]
    with pytest.raises(ValueError):
        parse_moves(["walk:1"])


def test_move_layout_matches_the_header(tmp_path):
    import subprocess
    src = tmp_path / "layout.c"
    src.write_text(r'''
#include <stdio.h>
#include <stddef.h>
#include "radex_b200.h"
#define P(T, f) printf(#T "." #f " %zu\n", offsetof(T, f))
int main(void) {
  printf("rb_move %zu\n", sizeof(rb_move)); P(rb_move, kind); P(rb_move, a); P(rb_move, gamma0); P(rb_move, sigma); P(rb_move, weight);
  printf("kinds %d %d %d\n", RB_MOVE_STRETCH, RB_MOVE_DE, RB_MAX_MOVES);
  return 0;
}
''')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    lines = subprocess.check_output([str(exe)], text=True).strip().splitlines()
    got = dict(line.split(" ", 1) for line in lines)
    assert int(got["rb_move"]) == C.sizeof(_lib.rb_move)
    for key, off in got.items():
        if key.startswith("rb_move."):
            assert int(off) == getattr(_lib.rb_move, key.split(".")[1]).offset, key
    assert got["kinds"] == "%d %d %d" % (_lib.RB_MOVE_STRETCH, _lib.RB_MOVE_DE, _lib.RB_MAX_MOVES)
