#!/usr/bin/env python
"""Corner-plot marginals, covariance and nearest sample at the config-5 shape (2^20 walkers x 1000 steps x 8
parameters, 67 GB in FP64, one GPU); the chain generator of tools/chain_stats_bench.py.

Reported, with the card's name and power limit read in the same run:
  * get_histograms(20) on summary_columns(2) (10 columns, 45 pairs): CUDA events around the whole call after a warm-up,
    and the range pass (the exact min / max by radix select) on its own;
  * the marginal kernel's own time with and without the pairs, its chain reads x 67 GB against 7.7 TB/s (HGX B200 data
    sheet), and the warp-lane counter updates per read (before the warp merge): which of the two bounds it;
  * get_covariance and get_nearest_sample (Mahalanobis, to the median);
  * on a 2^16-walker slice that fits on the host: hist1d == np.histogram and hist2d == np.histogram2d, and numpy's time.
    python tools/corner_bench.py --out profiles/r7_corner.json
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

from chain_stats_bench import HBM_TBS, card, sampler_on, timed  # noqa: E402
from radex_emcee_b200 import _lib  # noqa: E402
from radex_emcee_b200 import emcee_radex_2comp as er2  # noqa: E402
from radex_emcee_b200.data import DATA_DIR, get_source, read_data  # noqa: E402
from radex_emcee_b200.driver import summary_columns  # noqa: E402
from radex_emcee_b200.sampler import SLEDModel  # noqa: E402

BINS = 20


def kernel_ms(ctx, fn, reps):
    """CUDA-event time of fn() and the launches it makes (ctx counter)."""
    fn()
    l0 = ctx.counters()[1]
    _, ms = timed(fn, reps)
    return ms, (ctx.counters()[1] - l0) // (reps + 1)


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
    hbm_ms = chain_bytes / (HBM_TBS * 1e12) * 1e3

    s = sampler_on(ctx, model, chain)
    cols = summary_columns(2)
    ncol, npair = len(cols), len(cols) * (len(cols) - 1) // 2
    (edges, h1, h2, _), ms_h = timed(lambda: s.get_histograms(BINS, columns=cols), a.reps)
    view = s._chain_view(0, 1)
    _, ms_r = timed(lambda: s._percentiles(view, s._columns(cols), [0, 100]), a.reps)
    eng = s.engine
    ms_k, reads = kernel_ms(ctx, lambda: eng.chain_marginals(view, 1, s._columns(cols), edges), a.reps)
    ms_k1, reads1 = kernel_ms(ctx, lambda: eng.chain_marginals(view, 1, s._columns(cols), edges, pairs=False), a.reps)
    samples = N * T
    res["histograms"] = {
        "bins": BINS, "columns": ncol, "pairs": npair, "ms": ms_h, "ms_min": min(ms_h),
        "range_pass_ms": ms_r, "range_pass_ms_min": min(ms_r),
        "marginal_kernel_ms": ms_k, "marginal_kernel_ms_min": min(ms_k), "chain_reads": reads,
        "chain_read_at_7.7TBs_ms": hbm_ms, "hbm_bound_ms": reads * hbm_ms,
        "marginal_kernel_effective_TBs": reads * chain_bytes / (min(ms_k) * 1e-3) / 1e12,
        "lane_updates_per_read": samples * (ncol + npair),
        "lane_updates_per_s": samples * (ncol + npair) / (min(ms_k) * 1e-3),
        "columns_only_kernel_ms": ms_k1, "columns_only_kernel_ms_min": min(ms_k1), "columns_only_chain_reads": reads1,
        "columns_only_effective_TBs": reads1 * chain_bytes / (min(ms_k1) * 1e-3) / 1e12,
        "columns_only_lane_updates_per_read": samples * ncol,
        "note": "ms covers the whole call (range pass included); kernel ms are CUDA events around CudaEngine."
                "chain_marginals (edges upload and zeroed counts included); lane updates are counted before the warp "
                "merge (__match_any_sync), one per (sample, column) and (sample, pair)"}

    cov, ms_c = timed(lambda: s.get_covariance(), a.reps)
    med = s.get_quantiles([50])[0, 0]
    (xn, idx, d2), ms_n = timed(lambda: s.get_nearest_sample(med), a.reps)
    res["covariance"] = {"ms": ms_c, "ms_min": min(ms_c), "chain_reads": 2, "hbm_bound_ms": 2 * hbm_ms}
    res["nearest"] = {"ms": ms_n, "ms_min": min(ms_n), "chain_reads": 3, "hbm_bound_ms": 3 * hbm_ms,
                      "note": "Mahalanobis: two covariance reads, then one distance read", "index": int(idx[0]),
                      "d2": float(d2[0])}

    nc = a.check_walkers
    sl = chain[:, :nc].contiguous()
    del s, view, chain
    torch.cuda.empty_cache()
    s2 = sampler_on(ctx, model, sl)
    e2, g1, g2, pairs = s2.get_histograms(BINS, columns=cols)
    host = sl.cpu().numpy().reshape(-1, ndim)
    del sl, s2
    t0 = time.perf_counter()
    vals = [host[:, c] if isinstance(c, int) else host[:, c[0]] + host[:, c[1]] for c in cols]
    ok = True
    for c in range(ncol):
        h, e = np.histogram(vals[c], BINS)
        ok &= bool(np.array_equal(h, g1[0, c]) and np.array_equal(e, e2[0, c]))
    for p, (ca, cb) in enumerate(pairs):
        h, _, _ = np.histogram2d(vals[ca], vals[cb], BINS, range=[(e2[0, ca, 0], e2[0, ca, -1]), (e2[0, cb, 0], e2[0, cb, -1])])
        ok &= bool(np.array_equal(h, g2[0, p]))
    host_s = time.perf_counter() - t0
    res["check_slice"] = {"walkers": nc, "values_per_column": nc * T, "equal_to_numpy": ok, "numpy_host_s": host_s}
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    if not ok:
        raise SystemExit("device histograms differ from numpy")


if __name__ == "__main__":
    main()
