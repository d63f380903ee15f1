#!/usr/bin/env python
"""Device chain statistics at the config-5 shape (2^20 walkers x 1000 steps x 8 parameters, 67 GB in FP64, one GPU).

The chain is a seeded AR(1) series per (walker, parameter) built on the device (phi from 0.5 to 0.95 over the
parameters), stored as the sampler stores it.  Reported, with the card's name and power limit read in the same run:
  * get_quantiles((16, 50, 84)) on the 8 parameters + 2 log P columns, and get_autocorr_time: CUDA events around the
    whole call (host narrowing between passes included), after one warm-up call;
  * bytes read per radix pass against 7.7 TB/s (HGX B200 data sheet), acf FMAs against rb_fp64_peak (measured here);
  * on a 2^16-walker slice that fits on the host: get_quantiles == np.percentile, and the host time of np.percentile.
    python tools/chain_stats_bench.py --out profiles/r3_chain_stats.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from radex_emcee_b200 import _lib  # noqa: E402
from radex_emcee_b200 import emcee_radex_2comp as er2  # noqa: E402
from radex_emcee_b200.data import DATA_DIR, get_source, read_data  # noqa: E402
from radex_emcee_b200.driver import summary_columns  # noqa: E402
from radex_emcee_b200.sampler import CudaEngine, SLEDModel, StretchSampler  # noqa: E402

HBM_TBS = 7.7
Q = [16, 50, 84]


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        out["power_limit_and_max_sm_clock"] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit_and_max_sm_clock"] = "unavailable: %s" % e
    return out


def sampler_on(ctx, model, chain):
    """A sampler whose stored chain is `chain` [steps, nwalkers, ndim] (one chunk): the statistics read only that."""
    s = StretchSampler(chain.shape[1], chain.shape[2], CudaEngine(ctx, model), randomize_split=False)
    s._chain = [chain]
    return s


def timed(fn, reps):
    fn()                                                   # warm-up
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return out, ms


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--walkers", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--check-walkers", type=int, default=1 << 16)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=5)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    N, T, ndim = a.walkers, a.steps, 8
    ctx = _lib.Context(_lib.MolData(os.path.join(ROOT, "radex_emcee_b200", "data", "co.dat")), 0)
    z, T_d, _lw, jup, flux, eflux = get_source("G09v1.97", read_data(os.path.join(DATA_DIR, "flux_for2p.dat")))
    tbg, _ra, bounds, _p0 = er2.source_setup(z)
    model = SLEDModel(2, jup, flux, eflux, bounds, tbg, T_d=T_d)
    res = {"shape": {"walkers": N, "steps": T, "ndim": ndim}, "card": card()}

    g = torch.Generator(device="cuda").manual_seed(a.seed)
    phi = torch.linspace(0.5, 0.95, ndim, dtype=torch.float64, device="cuda")
    sig = torch.sqrt(1 - phi * phi)
    chain = torch.empty((T, N, ndim), dtype=torch.float64, device="cuda")
    x = torch.randn((N, ndim), generator=g, dtype=torch.float64, device="cuda")
    for t in range(T):
        chain[t] = x
        x = phi * x + sig * torch.randn((N, ndim), generator=g, dtype=torch.float64, device="cuda")
    del x
    torch.cuda.synchronize()
    chain_bytes = chain.numel() * 8
    res["chain_gb"] = chain_bytes / 1e9

    s = sampler_on(ctx, model, chain)
    cols = summary_columns(2)
    nranks = 2 * len(Q)                                    # two order statistics around each percentile (at most)
    groups = -(-nranks // max(1, _lib.RB_CHAIN_MAX_HIST // len(cols)))
    _, ms_q = timed(lambda: s.get_quantiles(Q, columns=cols), a.reps)
    passes = 8 * groups
    res["quantiles"] = {
        "columns": len(cols), "q": Q, "ms": ms_q, "ms_min": min(ms_q), "radix_passes": passes,
        "bytes_per_pass": chain_bytes, "bytes_per_pass_at_7.7TBs_ms": chain_bytes / (HBM_TBS * 1e12) * 1e3,
        "effective_TBs_whole_call": passes * chain_bytes / (min(ms_q) * 1e-3) / 1e12,
        "note": "ms covers the whole call: 8 histogram launches per group, their device-to-host copies and the host "
                "narrowing between passes"}

    l0 = s.engine.launches
    tau, ms_t = timed(lambda: s.get_autocorr_time(quiet=True), a.reps)
    acf_calls = (s.engine.launches - l0) // (a.reps + 1) - 1          # chain_moments is the other launch per call
    lags = min(T, acf_calls * 128)
    fmas = N * ndim * T * lags
    peak = ctx.fp64_peak_tflops()
    res["autocorr"] = {
        "ms": ms_t, "ms_min": min(ms_t), "lags_computed": lags, "acf_fma": fmas, "fp64_peak_tflops_measured": peak,
        "fma_at_peak_ms": 2 * fmas / (peak * 1e12) * 1e3, "achieved_fp64_tflops_whole_call": 2 * fmas / (min(ms_t) * 1e-3) / 1e12,
        "tau": tau.tolist(), "tau_ar1_exact": ((1 + phi) / (1 - phi)).tolist()}

    nc = a.check_walkers
    sl = chain[:, :nc].contiguous()
    del s
    s2 = sampler_on(ctx, model, sl)
    got = s2.get_quantiles(Q, columns=cols)[0]
    host = sl.cpu().numpy().reshape(-1, ndim)
    del sl, s2
    t0 = time.perf_counter()
    ref = np.empty((len(Q), len(cols)))
    for k, c in enumerate(cols):
        col = host[:, c] if isinstance(c, int) else host[:, c[0]] + host[:, c[1]]
        ref[:, k] = np.percentile(col, Q)
    host_s = time.perf_counter() - t0
    res["check_slice"] = {"walkers": nc, "values_per_column": nc * T, "equal_to_np_percentile": bool(np.array_equal(got, ref)),
                          "np_percentile_host_s": host_s}
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    if not res["check_slice"]["equal_to_np_percentile"]:
        raise SystemExit("device percentiles differ from np.percentile")


if __name__ == "__main__":
    main()
