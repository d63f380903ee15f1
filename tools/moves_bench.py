#!/usr/bin/env python
"""Stretch, DE and a DE 0.8 / stretch 0.2 mixture on G09v1.97 (one GPU, in-library loop): what a step costs and what it
buys in effective samples, on burnt-in chains of at least 50 integrated autocorrelation times.

Per ensemble: a 1e-3 ball around the drivers' starting point, burnt in with the stretch move, doubling until tau of its
second half has settled and the burn-in is 10 of it long; every move then starts from that same burnt-in ensemble and
runs until its stored chain is 50 tau long (emcee's tol = 50), checked after every chunk of steps.  The time caps are safety bounds; a run they stop
is marked reached_50_tau = false.  The results file is rewritten after every run.
Reported, with the card's name and power limit read in the same run:
  * wall time per step (host clock around run_mcmc, which ends in a device synchronise), walker-steps/s, solves per step;
  * acceptance fraction, tau per parameter (get_autocorr_time), steps / max tau, and effective samples per second =
    walkers x steps / max tau / wall time;
  * at 2^20 walkers (two components) a few steps of each move: walker-steps/s; on one GPU there is no all-gather.
    python tools/moves_bench.py --out profiles/r8_moves.json
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from chain_stats_bench import card  # noqa: E402
from radex_emcee_b200 import _lib  # noqa: E402
from radex_emcee_b200 import emcee_radex as er1  # noqa: E402
from radex_emcee_b200 import emcee_radex_2comp as er2  # noqa: E402
from radex_emcee_b200.data import DATA_DIR, get_source, read_data  # noqa: E402
from radex_emcee_b200.moves import DEMove, StretchMove  # noqa: E402
from radex_emcee_b200.sampler import CudaEngine, SLEDModel, StretchSampler  # noqa: E402

MOVES = {"stretch": None, "de": DEMove(), "de0.8+stretch0.2": [(DEMove(), 0.8), (StretchMove(), 0.2)]}


def model(ncomp):
    if ncomp == 1:
        z, _lw, jup, flux, eflux = get_source("G09v1.97", read_data(os.path.join(DATA_DIR, "flux.dat")))
        tbg, _ra, bounds, p0 = er1.source_setup(z)
        return SLEDModel(1, jup, flux, eflux, bounds, tbg), np.asarray(p0, dtype=np.float64)
    z, T_d, _lw, jup, flux, eflux = get_source("G09v1.97", read_data(os.path.join(DATA_DIR, "flux_for2p.dat")))
    tbg, _ra, bounds, p0 = er2.source_setup(z)
    p0 = np.array(p0, dtype=np.float64)
    p0[3] += 0.1      # cold size > warm size so the whole starting ball has a finite prior
    return SLEDModel(2, jup, flux, eflux, bounds, tbg, T_d=T_d), p0


def timed_run(s, pos, n, store=True, thin=1):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    s.run_mcmc(pos, n, store=store, thin=thin)
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def tau_of(s, thin=1, discard=0):
    """tau per parameter, in steps, of a chain stored every `thin` steps (run_mcmc(thin=...))."""
    return thin * s.get_autocorr_time(discard=discard // thin, quiet=True)[0]


def burn_in(ctx, ncomp, nw, seed, cap_s):
    """Stretch-move burn-in from the ball until it is 10 tau long, tau from its second half: (X, burn steps, tau, wall)."""
    m, p0 = model(ncomp)
    ndim = 4 * ncomp
    pos = p0 + 1e-3 * np.random.default_rng(seed).standard_normal((nw, ndim))
    s = StretchSampler(nw, ndim, CudaEngine(ctx, m), seed=seed)
    # a short window underestimates tau (emcee's auto_window is bounded by the chain): the burn-in doubles until the
    # estimate from its second half has settled (within 20 % of the previous one) and the burn-in is 10 of it long
    steps, chunk, wall, prev = 0, 1000, 0.0, None
    while True:
        wall += timed_run(s, pos if steps == 0 else None, chunk)
        steps += chunk
        tau = tau_of(s, discard=steps // 2)
        settled = prev is not None and np.all(np.isfinite(tau)) and tau.max() < 1.2 * prev
        if (settled and steps >= 10 * tau.max()) or wall >= cap_s:
            break
        prev = tau.max() if np.all(np.isfinite(tau)) else None
        chunk = steps
    X, _ = s.get_last_sample()
    return X, steps, tau, wall


def one(ctx, ncomp, nw, mvname, X0, thin, tau_hint, cap_s, seed):
    m, _ = model(ncomp)
    ndim = 4 * ncomp
    s = StretchSampler(nw, ndim, CudaEngine(ctx, m), seed=seed + 1, moves=MOVES[mvname])
    s.set_state(X0)
    solves0 = s.total_solves
    wall, steps = 0.0, 0
    chunk = max(10 * thin, int(20 * tau_hint) // thin * thin)
    while True:
        wall += timed_run(s, None, chunk, thin=thin)
        steps += chunk
        tau = tau_of(s, thin)
        enough = np.all(np.isfinite(tau)) and steps >= 50 * tau.max()
        if enough or wall >= cap_s:
            break
        need = 50 * tau.max() - steps if np.all(np.isfinite(tau)) else steps
        rate = steps / wall
        chunk = int(max(steps / 4, min(1.1 * need, (cap_s - wall) * rate))) // thin * thin + thin
    tmax = float(np.max(tau))
    return dict(ensemble="%d component%s, %d walkers" % (ncomp, "s" if ncomp > 1 else "", nw), ncomp=ncomp, walkers=nw,
                move=mvname, thin=thin, steps=steps, wall_s=wall, ms_per_step=1e3 * wall / steps,
                walker_steps_per_s=nw * steps / wall, solves_per_step=(s.total_solves - solves0) / steps,
                acceptance=float(s.acceptance_fraction.mean()), tau=[float(t) for t in tau], steps_over_max_tau=steps / tmax,
                reached_50_tau=bool(steps >= 50 * tmax), ess_per_s=nw * steps / tmax / wall)


def big(ctx, nw, mvname, steps, seed):
    m, p0 = model(2)
    pos = p0 + 1e-3 * np.random.default_rng(seed).standard_normal((nw, 8))
    s = StretchSampler(nw, 8, CudaEngine(ctx, m), seed=seed, moves=MOVES[mvname])
    timed_run(s, pos, 1, store=False)
    solves0 = s.total_solves
    wall = timed_run(s, None, steps, store=False)
    return dict(walkers=nw, move=mvname, steps=steps, ms_per_step=1e3 * wall / steps, walker_steps_per_s=nw * steps / wall,
                solves_per_step=(s.total_solves - solves0) / steps, gpus=1,
                all_gather_share="none on one GPU (the partners are read from X in place)",
                eight_gpus="not measured")


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--walkers", type=int, nargs="+", default=[100, 400, 16384],
                    help="ensembles: 100 is one component, the others two")
    ap.add_argument("--cap", type=float, default=600.0, help="safety bound in seconds per burn-in and per run")
    ap.add_argument("--deadline", type=float, default=1e9, help="seconds after which no new run starts")
    ap.add_argument("--big-walkers", type=int, default=1 << 20)
    ap.add_argument("--big-steps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=20170914)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    t_start = time.perf_counter()
    ctx = _lib.Context(_lib.MolData(os.path.join(ROOT, "radex_emcee_b200", "data", "co.dat")), 0)
    out = dict(card=card(), source="G09v1.97", burn_in=[], runs=[], big=[], not_run=[])
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)

    def save():
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    if a.big_steps > 0:
        for r in [big(ctx, a.big_walkers, mv, a.big_steps, a.seed) for mv in MOVES]:
            out["big"].append(r)
            print(json.dumps(r), flush=True)
        save()
    for nw in a.walkers:
        ncomp = 1 if nw == 100 else 2
        left = a.deadline - (time.perf_counter() - t_start)
        if left <= 0:
            out["not_run"].append(dict(walkers=nw, ncomp=ncomp, why="time budget of the run spent"))
            save()
            continue
        X, bsteps, btau, bwall = burn_in(ctx, ncomp, nw, a.seed, min(a.cap, left))
        b = dict(ncomp=ncomp, walkers=nw, move="stretch", steps=bsteps, wall_s=bwall, tau_second_half=[float(t) for t in btau],
                 reached_10_tau=bool(steps_ok(bsteps, btau, 10) and bwall < min(a.cap, left)))
        out["burn_in"].append(b)
        print(json.dumps(b), flush=True)
        save()
        thin = max(1, int(np.max(btau)) // 25)
        for mv in MOVES:
            left = a.deadline - (time.perf_counter() - t_start)
            if left <= 0:
                out["not_run"].append(dict(walkers=nw, ncomp=ncomp, move=mv, why="time budget of the run spent"))
                save()
                continue
            r = one(ctx, ncomp, nw, mv, X, thin, float(np.max(btau)), min(a.cap, left), a.seed)
            out["runs"].append(r)
            print(json.dumps(r), flush=True)
            save()
    out["card_after"] = card()
    save()


def steps_ok(steps, tau, k):
    return np.all(np.isfinite(tau)) and steps >= k * np.max(tau)


if __name__ == "__main__":
    main()
