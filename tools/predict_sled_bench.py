#!/usr/bin/env python
"""Posterior-predictive SLEDs at the config-5 shape: 2^20 two-component walkers, 16 stored steps thinned by 4 to 4
selected steps, 8.4e6 solves per call (one GPU).

The chain is seeded on the device: a burnt-in-like spread (0.15 dex) around the two-component starting point, clipped to
the two-component bounds of a flux_for2p.dat source.  Reported, with the card's name, power limit and max SM clock read
in the same run:
  * the predictive call (rb_predict_sled_dev, 11 lines) against rb_solve_batch_dev on the same models (every line's
    brightness and the status), alternated, CUDA events around each call, after one warm-up of each;
  * the share of k_predict_expand and k_predict_flux in the predictive call, from torch.profiler kernel times of one
    call in a profiled run of its own;
  * get_predictive_quantiles for 16 lines x 3 planes, CUDA events around the whole call (host narrowing included).
    python tools/predict_sled_bench.py --out profiles/r6_predict_sled.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from radex_emcee_b200 import _lib  # noqa: E402
from radex_emcee_b200 import emcee_radex_2comp as er2  # noqa: E402
from radex_emcee_b200.data import DATA_DIR, get_source, read_data  # noqa: E402
from radex_emcee_b200.sampler import CudaEngine, SLEDModel, StretchSampler  # noqa: E402

JUP = list(range(1, 12))


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        out["power_limit_and_max_sm_clock"] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit_and_max_sm_clock"] = "unavailable: %s" % e
    return out


def event_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return out, e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--walkers", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--thin", type=int, default=4)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    N, T, ndim = a.walkers, a.steps, 8
    ctx = _lib.Context(_lib.MolData(os.path.join(ROOT, "radex_emcee_b200", "data", "co.dat")), 0)
    z, T_d, _lw, jup, flux, eflux = get_source("G09v1.97", read_data(os.path.join(DATA_DIR, "flux_for2p.dat")))
    tbg, _ra, bounds, p0 = er2.source_setup(z)
    p0 = p0.copy()
    p0[3] += 0.1
    model = SLEDModel(2, jup, flux, eflux, bounds, tbg, T_d=T_d)
    eng = CudaEngine(ctx, model)
    res = {"shape": {"walkers": N, "steps": T, "thin": a.thin, "ncomp": 2, "lines": len(JUP)}, "card": card()}

    g = torch.Generator(device="cuda").manual_seed(a.seed)
    lo, hi = (torch.tensor(bounds[:, k], dtype=torch.float64, device="cuda") for k in (0, 1))
    chain = torch.tensor(p0, dtype=torch.float64, device="cuda") + 0.15 * torch.randn((T, N, ndim), generator=g,
                                                                                       dtype=torch.float64, device="cuda")
    chain = torch.minimum(torch.maximum(chain, lo), hi).contiguous()
    s = StretchSampler(N, ndim, eng, randomize_split=False)
    s._chain = [chain]
    view = s._chain_view(0, a.thin)
    nsel = view.nsel
    nmod = nsel * N * 2
    res["solves_per_call"] = nmod

    # the same models for rb_solve_batch_dev, component-major within a sample as the pipeline lays them out
    sel = chain[a.thin - 1::a.thin].reshape(-1, 2, 4).reshape(-1, 4)
    np_ = ctx.mol.npart
    dens_tot = torch.pow(10.0, sel[:, 0])
    frac = [0.0] * np_
    for q, pid in enumerate(ctx.mol.partner_id):
        frac[q] = 1.0 if pid == 1 else (1 - er2.fortho) if pid == 2 else er2.fortho if pid == 3 else 0.0
    dens = torch.stack([f * dens_tot for f in frac], dim=1).contiguous()
    tkin, cdmol = torch.pow(10.0, sel[:, 1]).contiguous(), torch.pow(10.0, sel[:, 2]).contiguous()
    del sel, dens_tot
    surf = torch.empty((nmod, ctx.mol.nline), dtype=torch.float64, device="cuda")
    status = torch.empty(nmod, dtype=torch.int32, device="cuda")
    opts = _lib.default_opts()
    L = _lib.load()

    def solve():
        ctx.set_stream(torch.cuda.current_stream().cuda_stream)
        _lib.check(L.rb_solve_batch_dev(ctx.handle, nmod, tkin.data_ptr(), dens.data_ptr(), cdmol.data_ptr(), 1.0, tbg,
                                        2, C.byref(opts), None, None, None, surf.data_ptr(), None, status.data_ptr()))

    cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
    predict = lambda: eng.predict_sled(view, JUP, cnt)   # noqa: E731
    predict()
    solve()
    torch.cuda.synchronize()
    ms_p, ms_s = [], []
    for _ in range(a.reps):
        F, t = event_ms(predict)
        ms_p.append(t)
        del F
        ms_s.append(event_ms(solve)[1])
    res["predict_vs_solve"] = {
        "predict_ms": ms_p, "solve_batch_ms": ms_s,
        "predict_solves_per_s": nmod / (min(ms_p) * 1e-3), "solve_batch_solves_per_s": nmod / (min(ms_s) * 1e-3),
        "predict_over_solve": min(ms_p) / min(ms_s),
        "counters_solved_out_of_range_over_all_calls": cnt.cpu().tolist(),
        "note": "same models (the selected samples, 2 components each); the solve batch writes the brightness of all "
                "%d lines and the status, the predictive call the fluxes of %d lines in 3 planes" % (ctx.mol.nline, len(JUP))}

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        predict()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.events():                               # device activities only: kernels and memsets
        us = getattr(ev, "device_time_total", 0.0) or 0.0
        if us > 0:
            kern[ev.name] = kern.get(ev.name, 0.0) + us / 1e3
    busy = sum(kern.values())
    exp = sum(v for k, v in kern.items() if "k_predict_expand" in k)
    flx = sum(v for k, v in kern.items() if "k_predict_flux" in k)
    res["kernel_share"] = {"device_busy_ms_summed": busy, "expand_ms": exp, "flux_ms": flx,
                           "expand_plus_flux_share_of_busy": (exp + flx) / busy if busy else None,
                           "kernels_ms": {k: v for k, v in sorted(kern.items(), key=lambda kv: -kv[1])[:12]},
                           "note": "kernel times of one profiled call, summed; launch B and the engine launches "
                                   "overlap, so the sum exceeds the call's wall time"}

    jq = list(range(1, 17))
    s.get_predictive_quantiles(jq, [16, 50, 84], thin=a.thin)
    ms_q = [event_ms(lambda: s.get_predictive_quantiles(jq, [16, 50, 84], thin=a.thin))[1] for _ in range(a.reps)]
    res["predictive_quantiles_16_lines_3_planes"] = {
        "ms": ms_q, "ms_min": min(ms_q),
        "note": "whole call: the predictive solve of every selected sample, then 8 radix passes per plane"}
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
