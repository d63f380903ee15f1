"""Per-source fit pipeline: the body of the reference drivers' ``main()`` loops
(emcee/emcee_radex.py:389-531, emcee/emcee_radex_2comp.py:486-608) on top of the GPU hot path.

For one source: bounds and starting point -> ``scipy.optimize.curve_fit`` on the SLED model ->
``scipy.optimize.minimize`` of -lnprob -> walkers in a 1e-3 ball around the curve_fit point ->
burn-in, reset, production run of the stretch move -> pickle with the reference's tuple layout ->
16/50/84 percentiles of (log n, log T, log N, log P = log n + log T) printed with the same tags.

What differs from the reference, on purpose:
  * the optimisers' finite-difference Jacobians/gradients are evaluated as ONE batched launch per
    iteration (ndim + 1 models) instead of ndim + 1 serial RADEX calls; the step rules are scipy's
    own ('2-point', sign chosen to stay inside the bounds), so the iterates match a scipy run that
    differentiates numerically;
  * the sampler is the device-resident stretch move of ``sampler.py`` (emcee is not a dependency);
  * random numbers are seeded (the reference's are not);
  * fluxes in the pickle are plain float arrays in Jy km/s, not astropy Quantities.
With ``torchrun`` every rank takes the sources ``rank::world_size`` on its own GPU: replicas, no
communication (BASELINE.json configs[3]).

The 16/50/84 percentiles (``summary``) and ``theta_med`` are computed on the device from the stored chain
(``StretchSampler.get_quantiles``: the same values ``np.percentile`` gives on the host chain), and the result gains
``autocorr_time`` (emcee's integrated autocorrelation time per parameter).  With ``chain_to_host=False``
(CLI ``--summaries-only``) the chain is never gathered or copied to the host: ``chain`` and ``lnprobability`` of the
result are ``None``, and so is the pickle's ``(chain, lnprobability)`` slot.  That is the only way to run ensembles whose
chain does not fit in host memory (``--walkers 1048576``).

With ``predict_jup`` (CLI ``--predict-sled J ...``) the result also gains the posterior-predictive SLED: the 16/50/84
percentiles of the model flux of each requested line over the chain (``StretchSampler.get_predictive_quantiles``), per
component with two components -- the model SLEDs the reference's replot draws from the pickled chain.

With ``corner_bins`` (CLI ``--corner-bins B``) the result also gains ``corner``: the counts the replot's corner plots are
drawn from (B-bin marginals of every summary column and of every pair, ``StretchSampler.get_histograms``), the covariance
and the Mahalanobis-nearest sample to ``theta_med`` -- all computed on the device, so they work with ``--summaries-only``;
with ``outdir`` they are also written to ``<source>_corner.npz`` (``<source>_corner_2comp.npz`` with two components).
"""
from __future__ import annotations

import argparse
import logging
import os
import pickle
import sys

import numpy as np
from scipy.optimize import curve_fit, minimize

from . import _lib
from . import emcee_radex as _er1
from . import emcee_radex_2comp as _er2
from .data import get_source, read_data
from .moves import parse_moves

logger = logging.getLogger("radex_emcee_b200.driver")

SQRT_EPS = float(np.sqrt(np.finfo(np.float64).eps))


# ---- batched finite differences --------------------------------------------------------------------
def forward_steps(x, lo, hi, rel_step=None, abs_step=None):
    """scipy's '2-point' step rule: h = rel_step * sign(x) * max(1, |x|) (or an absolute step), flipped
    where x + h would leave [lo, hi]."""
    x = np.asarray(x, dtype=np.float64)
    if abs_step is not None:
        h = np.full_like(x, float(abs_step))
    else:
        rs = SQRT_EPS if rel_step is None else float(rel_step)
        h = rs * np.where(x >= 0, 1.0, -1.0) * np.maximum(1.0, np.abs(x))
    out = (x + h > hi) | (x + h < lo)
    return np.where(out, -h, h)


def batched_points(x, h):
    """Rows: x, x + h_0 e_0, ..., x + h_{n-1} e_{n-1}."""
    x = np.asarray(x, dtype=np.float64)
    P = np.tile(x, (x.size + 1, 1))
    P[np.arange(1, x.size + 1), np.arange(x.size)] += h
    return P


def fd_jacobian(model, x, lo, hi, rel_step=None):
    """Jacobian (m, n) of a vector model by forward differences, one batched model call."""
    h = forward_steps(x, lo, hi, rel_step=rel_step)
    F = np.atleast_2d(model(batched_points(x, h)))            # (n + 1, m)
    return ((F[1:] - F[0]) / h[:, None]).T


def fd_value_and_gradient(fun, x, lo, hi, abs_step=1e-8):
    """(f(x), grad f(x)) of a scalar batched function; L-BFGS-B's default numerical gradient
    (absolute step 1e-8, kept inside the bounds)."""
    h = forward_steps(x, lo, hi, abs_step=abs_step)
    f = np.asarray(fun(batched_points(x, h)), dtype=np.float64)
    with np.errstate(invalid="ignore"):
        g = (f[1:] - f[0]) / h
    return float(f[0]), g


# ---- summaries -------------------------------------------------------------------------------------
def percentile_summary(samples):
    """(median, +err, -err) per column from the 16/50/84 percentiles (emcee_radex.py:517-518)."""
    lo, med, hi = np.percentile(np.asarray(samples, dtype=np.float64), [16, 50, 84], axis=0)
    return [(m, h - m, m - l) for l, m, h in zip(lo, med, hi)]


def posterior_summary(flatchain, ncomp):
    """Per component: summaries of log n, log T, log N/dv and log P = log n + log T
    (emcee_radex.py:511-518, emcee_radex_2comp.py:588-597)."""
    flatchain = np.asarray(flatchain, dtype=np.float64)
    out = []
    for c in range(ncomp):
        blk = flatchain[:, 4 * c:4 * c + 3]
        out.append(dict(zip(("n_H2", "T_kin", "N_CO/dv", "P"),
                            percentile_summary(np.hstack((blk, blk[:, [0]] + blk[:, [1]]))))))
    return out


def summary_columns(ncomp):
    """get_quantiles columns of the drivers' summaries: the 4 ncomp parameters, then log P = log n + log T per
    component."""
    return list(range(4 * ncomp)) + [(4 * c, 4 * c + 1) for c in range(ncomp)]


def summaries_from_quantiles(Q, ncomp):
    """(summary, theta_med) from get_quantiles([16, 50, 84], columns=summary_columns(ncomp)) of one source ([3, ncol]):
    the same values and types posterior_summary and np.percentile(flatchain, 50, axis=0) give on the host chain."""
    ndim = 4 * ncomp
    out = []
    for c in range(ncomp):
        sel = [4 * c, 4 * c + 1, 4 * c + 2, ndim + c]
        lo, med, hi = Q[0, sel], Q[1, sel], Q[2, sel]
        out.append(dict(zip(("n_H2", "T_kin", "N_CO/dv", "P"), [(m, h - m, m - l) for l, m, h in zip(lo, med, hi)])))
    return out, np.array(Q[1, :ndim])


def sled_summaries(Q, jup):
    """Per plane of get_predictive_quantiles(jup, [16, 50, 84]) of one source ([nplanes, 3, nlines]): J -> (median, +err,
    -err) of the predicted flux, as percentile_summary gives on the host."""
    return [{int(J): (m, h - m, m - l) for J, l, m, h in zip(jup, *Qp)} for Qp in Q]


def sled_results(sampler, jup):
    """Per source: the result items of the posterior-predictive SLED, from the device-resident chain."""
    jup = [int(J) for J in jup]
    Q = sampler.get_predictive_quantiles(jup, [16, 50, 84])
    return [dict(sled_jup=np.array(jup), sled_summary=sled_summaries(Qs, jup)) for Qs in Q]


def corner_results(sampler, ncomp, theta_med, bins):
    """Per source: the ``corner`` result item from the device-resident chain -- B-bin marginals of the summary columns
    and of their pairs, the covariance and the sample nearest ``theta_med`` ([nsources, ndim]) in the Mahalanobis
    metric of nearest_sample_to_vector."""
    cols = summary_columns(ncomp)
    edges, h1, h2, _pairs = sampler.get_histograms(bins, columns=cols)
    cov = sampler.get_covariance()
    x, idx, d2 = sampler.get_nearest_sample(theta_med, metric="mahalanobis")
    return [dict(columns=cols, edges=edges[s], hist1d=h1[s], hist2d=h2[s], covariance=cov[s], theta_nearest=x[s],
                 theta_nearest_index=int(idx[s]), theta_nearest_d2=float(d2[s])) for s in range(len(edges))]


def write_corner(outdir, source, ncomp, corner):
    """<source>_corner.npz (<source>_corner_2comp.npz): the corner item, columns as (i, j) rows (j = -1: x[i] alone)."""
    name = os.path.join(outdir, "%s_corner%s.npz" % (source, "" if ncomp == 1 else "_2comp"))
    cols = np.array([(c, -1) if isinstance(c, int) else c for c in corner["columns"]], dtype=np.int64)
    np.savez(name, **dict(corner, columns=cols))
    return name


def log_autocorr(source, tau):
    logger.info("%s: integrated autocorrelation time (steps) %s", source, np.array2string(np.asarray(tau), precision=1))


def nearest_sample_to_vector(samples, target, metric="mahalanobis", eps=1e-9):
    """Sample closest to ``target``: (sample, index, squared distance); metrics as in
    emcee_radex.py:242-266 ('mahalanobis' with a regularised covariance, 'z' = per-axis standardised,
    'euclidean')."""
    X = np.asarray(samples, dtype=np.float64)
    d = X - np.asarray(target, dtype=np.float64)
    if metric == "mahalanobis":
        cov = np.cov(X, rowvar=False) + eps * np.eye(X.shape[1])
        white = np.linalg.solve(np.linalg.cholesky(cov), d.T)
        dist2 = np.einsum("ij,ij->j", white, white)
    elif metric == "z":
        s = X.std(axis=0, ddof=1)
        dist2 = np.sum((d / np.where(s > 0, s, eps)) ** 2, axis=1)
    else:
        dist2 = np.sum(d * d, axis=1)
    i = int(np.argmin(dist2))
    return X[i], i, float(dist2[i])


# ---- the pipeline ----------------------------------------------------------------------------------
def _modules(ncomp):
    if ncomp == 1:
        return _er1
    if ncomp == 2:
        return _er2
    raise ValueError("ncomp must be 1 or 2")


def prefit(ncomp, R, Jup, flux, eflux, bounds, p0, T_d=None, opts=None):
    """curve_fit then minimize(-lnprob), as emcee_radex.py:444-467 / emcee_radex_2comp.py:524-544.
    Returns (popt, pcov, pmin, info)."""
    mod = _modules(ncomp)
    lo, hi = bounds[:, 0], bounds[:, 1]
    info = {"model_launches": 0, "lnprob_launches": 0}

    def model_batch(P):
        info["model_launches"] += 1
        return mod.model_lvg(Jup, P, R)

    def f(_x, *params):
        return np.asarray(model_batch(np.asarray(params, dtype=np.float64)))

    def jac(_x, *params):
        return fd_jacobian(model_batch, np.asarray(params, dtype=np.float64), lo, hi)

    try:
        popt, pcov = curve_fit(f, Jup, flux, sigma=eflux, p0=p0, bounds=(lo, hi), jac=jac)
        logger.info("curve_fit : %s", popt)
    except Exception as e:                      # the 1-component script catches RuntimeError only; a
        logger.warning("curve_fit : failed (%s)", e)   # ValueError there would abort the whole run
        popt, pcov = np.asarray(p0, dtype=np.float64), None

    saved = mod.R
    mod.R = R

    def nll_batch(P):
        info["lnprob_launches"] += 1
        if ncomp == 1:
            return -np.asarray(mod.lnprob(P, Jup, flux, eflux, bounds, opts=opts))
        return -np.asarray(mod.lnprob(P, Jup, flux, eflux, bounds, T_d, opts=opts))

    try:
        res = minimize(lambda p: fd_value_and_gradient(nll_batch, p, lo, hi), popt, jac=True,
                       bounds=list(zip(lo, hi)), method="L-BFGS-B")
    finally:
        mod.R = saved
    pmin = res.x
    logger.info("minimize : %s", pmin)
    info["minimize_success"] = bool(res.success)
    info["minimize_nit"] = int(res.nit)
    return popt, pcov, pmin, info


def fit_source(source, data, ncomp=1, nwalkers=None, n_iter_burn=100, n_iter_walk=None, seed=20170914,
               device=0, datapath=None, opts=None, outdir=None, store_chain=True, allow_synthetic=False,
               chain_to_host=True, predict_jup=None, corner_bins=None, moves=None):
    """One pass of the reference's per-source loop.  Returns a dict with every item of the pickle plus
    the percentile summaries, the sampler's acceptance fraction and the integrated autocorrelation time.
    ``chain_to_host=False``: the chain stays on the device (``chain`` and ``lnprobability`` are None).
    ``predict_jup``: line indices J whose posterior-predictive fluxes the result gains (``sled_jup``, ``sled_summary``).
    ``corner_bins``: bins of the ``corner`` item the result gains (marginals, covariance, nearest sample).
    ``moves``: the sampler's moves as ``StretchSampler(moves=...)`` takes them (None: the stretch move)."""
    from .radex import Radex
    from .sampler import CudaEngine, SLEDModel, StretchSampler

    mod = _modules(ncomp)
    if ncomp == 1:
        z, line_width, Jup, flux, eflux = get_source(source, data)
        T_d = None
        nwalkers = 100 if nwalkers is None else nwalkers          # emcee_radex.py:472-474
        n_iter_walk = 500 if n_iter_walk is None else n_iter_walk
    else:
        z, T_d, line_width, Jup, flux, eflux = get_source(source, data)
        nwalkers = 400 if nwalkers is None else nwalkers          # emcee_radex_2comp.py:548-550
        n_iter_walk = 1000 if n_iter_walk is None else n_iter_walk
    tbg, _ra, bounds, p0 = mod.source_setup(z)
    R = Radex(species="co", datapath=datapath,
              density={"oH2": mod.fortho * 1e10, "pH2": (1 - mod.fortho) * 1e10}, column=1e6, temperature=20.0,
              tbackground=tbg, deltav=1.0, escapeProbGeom="lvg", device=device)
    if R.molfile_is_synthetic and not allow_synthetic:
        raise ValueError(
            "%s is the synthetic CO-like table shipped for tests (made-up collision rates): posteriors fitted with it are "
            "not physical.  Pass datapath= (or --datapath / RADEX_DATAPATH) pointing at the directory that holds the LAMDA "
            "co.dat, as the reference's radex_moldata/ does, or allow_synthetic=True (--allow-synthetic)." % R.molpath)
    if R.molfile_is_synthetic:
        logger.warning("fitting with the SYNTHETIC molecular table %s: results are not physical", R.molpath)
    popt, pcov, pmin, info = prefit(ncomp, R, Jup, flux, eflux, bounds, p0, T_d=T_d, opts=opts)

    ndim = 4 * ncomp
    rng = np.random.RandomState(seed)                       # the reference draws from numpy's global state
    pos = np.array([popt + 1e-3 * rng.randn(ndim) for _ in range(nwalkers)])
    eng = CudaEngine(R._ctx, SLEDModel(ncomp, Jup, flux, eflux, bounds, tbg, T_d=T_d, opts=opts))
    sampler = StretchSampler(nwalkers, ndim, eng, seed=seed, moves=moves)
    logger.info("burning samples")
    sampler.run_mcmc(pos, n_iter_burn, store=False)
    sampler.reset()
    logger.info("walking")
    sampler.run_mcmc(None, n_iter_walk, store=store_chain)
    summary, theta_med = summaries_from_quantiles(
        sampler.get_quantiles([16, 50, 84], columns=summary_columns(ncomp))[0], ncomp)
    tau = sampler.get_autocorr_time(quiet=True)[0]
    log_autocorr(source, tau)
    chain = sampler.get_chain() if chain_to_host else None
    lnprobability = sampler.get_log_prob() if chain_to_host else None
    result = dict(source=source, z=z, bounds=bounds, T_d=T_d, data=(Jup, flux, eflux), popt=popt, pcov=pcov,
                  pmin=pmin, theta_med=theta_med, chain=chain, lnprobability=lnprobability,
                  summary=summary, autocorr_time=tau,
                  acceptance_fraction=float(np.mean(sampler.acceptance_fraction)),
                  acceptance_fraction_per_walker=sampler.acceptance_fraction,
                  prefit_info=info, solves=int(eng.total_solves.item()) + sampler.total_solves,
                  molfile=R.molpath, molfile_synthetic=R.molfile_is_synthetic)
    if predict_jup is not None:
        result.update(sled_results(sampler, predict_jup)[0])
    if corner_bins is not None:
        result["corner"] = corner_results(sampler, ncomp, theta_med[None], corner_bins)[0]
    if outdir is not None:
        os.makedirs(outdir, exist_ok=True)
        if corner_bins is not None:
            result["corner_npz"] = write_corner(outdir, source, ncomp, result["corner"])
        if ncomp == 1:     # emcee_radex.py:504-509
            name = os.path.join(outdir, "%s_bounds.pickle" % source)
            payload = (source, z, bounds, (Jup, flux, eflux), (popt, pcov), pmin, theta_med, (chain, lnprobability))
        else:              # emcee_radex_2comp.py:580-585
            name = os.path.join(outdir, "%s_bounds_2comp.pickle" % source)
            payload = (source, z, bounds, T_d, (Jup, flux, eflux), (popt, pcov), pmin, theta_med, (chain, lnprobability))
        with open(name, "wb") as f:
            pickle.dump(payload, f)
        result["pickle"] = name
    return result


def fit_sources_concurrently(sources, data, ncomp=1, nwalkers=None, n_iter_burn=100, n_iter_walk=None, seed=20170914,
                             device=0, datapath=None, opts=None, outdir=None, allow_synthetic=False, chain_to_host=True,
                             predict_jup=None, corner_bins=None, moves=None):
    """BASELINE.json configs[3]: every source of the table in ONE ensemble.  The reference fits the sources one after the
    other (emcee_radex.py:389); here the pre-fits run per source (they are a few dozen batched launches each) and the
    walkers of all sources -- each with its own background temperature, bounds, line set and, with two components, dust
    temperature -- step together: ``nwalkers`` per source, partners drawn inside the source's own sub-ensemble, one fused
    lnprob launch per half-step for all of them.  Under torchrun the ensemble is sharded over the ranks (whole sources per
    rank).  Returns one result dict per source, the same items ``fit_source`` returns (``chain_to_host``, ``predict_jup``
    and ``corner_bins`` as there)."""
    from .radex import Radex
    from .sampler import CudaEngine, SLEDModel, StretchSampler

    mod = _modules(ncomp)
    if nwalkers is None:
        nwalkers = 100 if ncomp == 1 else 400
    if n_iter_walk is None:
        n_iter_walk = 500 if ncomp == 1 else 1000
    ndim = 4 * ncomp
    setups, models, starts = [], [], []
    R = None
    for k, source in enumerate(sources):
        if ncomp == 1:
            z, line_width, Jup, flux, eflux = get_source(source, data)
            T_d = None
        else:
            z, T_d, line_width, Jup, flux, eflux = get_source(source, data)
        tbg, _ra, bounds, p0 = mod.source_setup(z)
        if R is None:
            R = Radex(species="co", datapath=datapath, density={"oH2": mod.fortho * 1e10, "pH2": (1 - mod.fortho) * 1e10},
                      column=1e6, temperature=20.0, tbackground=tbg, deltav=1.0, escapeProbGeom="lvg", device=device)
            if R.molfile_is_synthetic and not allow_synthetic:
                raise ValueError("%s is the synthetic CO-like table shipped for tests: pass datapath= / --datapath, or "
                                 "allow_synthetic=True (--allow-synthetic)" % R.molpath)
        R.set_params(tbg=tbg)
        popt, pcov, pmin, info = prefit(ncomp, R, Jup, flux, eflux, bounds, p0, T_d=T_d, opts=opts)
        rng = np.random.RandomState(seed + k)
        starts.append(np.array([popt + 1e-3 * rng.randn(ndim) for _ in range(nwalkers)]))
        models.append(SLEDModel(ncomp, Jup, flux, eflux, bounds, tbg, T_d=T_d, opts=opts))
        setups.append(dict(source=source, z=z, bounds=bounds, T_d=T_d, data=(Jup, flux, eflux), popt=popt, pcov=pcov,
                           pmin=pmin, prefit_info=info))
    eng = CudaEngine(R._ctx, models)
    sampler = StretchSampler(nwalkers * len(sources), ndim, eng, seed=seed, nsources=len(sources), moves=moves)
    logger.info("burning samples (%d sources x %d walkers in one ensemble)", len(sources), nwalkers)
    sampler.run_mcmc(np.vstack(starts), n_iter_burn, store=False)
    sampler.reset()
    logger.info("walking")
    sampler.run_mcmc(None, n_iter_walk)
    Q = sampler.get_quantiles([16, 50, 84], columns=summary_columns(ncomp))
    taus = sampler.get_autocorr_time(quiet=True)
    acc = sampler.acceptance_fraction
    chain, lnp = (sampler.get_chain(), sampler.get_log_prob()) if chain_to_host else (None, None)
    sleds = sled_results(sampler, predict_jup) if predict_jup is not None else None
    corners = None
    if corner_bins is not None:
        meds = np.array([summaries_from_quantiles(Q[k], ncomp)[1] for k in range(len(setups))])
        corners = corner_results(sampler, ncomp, meds, corner_bins)
    results = []
    for k, st in enumerate(setups):
        sl = slice(k * nwalkers, (k + 1) * nwalkers)
        c, l = (np.ascontiguousarray(chain[:, sl]), np.ascontiguousarray(lnp[:, sl])) if chain_to_host else (None, None)
        summary, theta_med = summaries_from_quantiles(Q[k], ncomp)
        if sampler.rank == 0:
            log_autocorr(st["source"], taus[k])
        res = dict(st, theta_med=theta_med, chain=c, lnprobability=l, summary=summary, autocorr_time=taus[k],
                   acceptance_fraction=float(np.mean(acc[sl])),
                   acceptance_fraction_per_walker=acc[sl], molfile=R.molpath, molfile_synthetic=R.molfile_is_synthetic)
        if sleds is not None:
            res.update(sleds[k])
        if corners is not None:
            res["corner"] = corners[k]
        if outdir is not None and sampler.rank == 0:
            os.makedirs(outdir, exist_ok=True)
            if corners is not None:
                res["corner_npz"] = write_corner(outdir, st["source"], ncomp, corners[k])
            if ncomp == 1:
                name = os.path.join(outdir, "%s_bounds.pickle" % st["source"])
                payload = (st["source"], st["z"], st["bounds"], st["data"], (st["popt"], st["pcov"]), st["pmin"],
                           res["theta_med"], (c, l))
            else:
                name = os.path.join(outdir, "%s_bounds_2comp.pickle" % st["source"])
                payload = (st["source"], st["z"], st["bounds"], st["T_d"], st["data"], (st["popt"], st["pcov"]), st["pmin"],
                           res["theta_med"], (c, l))
            with open(name, "wb") as f:
                pickle.dump(payload, f)
            res["pickle"] = name
        results.append(res)
    return results


def print_summary(res, ncomp, file=None):
    """The 'xxx:' block of the reference (emcee_radex.py:520-531, emcee_radex_2comp.py:599-608)."""
    out = file or sys.stdout
    pmin = res["pmin"]
    print("xxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxxx", file=out)
    print("xxx: %s\nxxx: minimised results" % res["source"], file=out)
    for c in range(ncomp):
        blk = pmin[4 * c:4 * c + 3]
        print("xxx: %s" % np.hstack((blk, blk[0] + blk[1])), file=out)
    print("xxx: emcee results", file=out)
    for key in ("n_H2", "T_kin", "N_CO/dv", "P"):
        print("xxx: %s" % key, file=out)
        for c in range(ncomp):
            print("xxx: %s" % (tuple(float(v) for v in res["summary"][c][key]),), file=out)
    if "sled_summary" in res:
        names = ["flux"] if ncomp == 1 else ["total flux", "component 1 flux", "component 2 flux"]
        print("xxx: predicted SLED [Jy km/s]: (median, +err, -err)", file=out)
        for name, plane in zip(names, res["sled_summary"]):
            print("xxx: %s" % name, file=out)
            for J, v in plane.items():
                print("xxx: J=%d %s" % (J, tuple(float(x) for x in v)), file=out)
    if "corner" in res:
        print("xxx: sample nearest the median (Mahalanobis): %s" % res["corner"]["theta_nearest"], file=out)


def main(argv=None):
    ap = argparse.ArgumentParser(description="Fit every source of a flux table (reference: main() of the drivers)")
    ap.add_argument("--data", default=None, help="flux table (default: data/flux.dat or data/flux_for2p.dat)")
    ap.add_argument("--ncomp", type=int, default=1, choices=[1, 2])
    ap.add_argument("--out", default=None, help="directory for the pickles (default ./single or ./double)")
    ap.add_argument("--sources", nargs="*", default=None)
    ap.add_argument("--walkers", type=int, default=None)
    ap.add_argument("--burn", type=int, default=100)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--seed", type=int, default=20170914)
    ap.add_argument("--datapath", default=None, help="directory holding the LAMDA co.dat (the reference's radex_moldata/); "
                                                     "default: $RADEX_DATAPATH")
    ap.add_argument("--concurrent", action="store_true",
                    help="all sources in one ensemble (BASELINE configs[3]); with torchrun the ensemble is sharded over the ranks")
    ap.add_argument("--allow-synthetic", action="store_true",
                    help="fit with the synthetic test table shipped in the package (NOT physical)")
    ap.add_argument("--summaries-only", action="store_true",
                    help="keep the chain on the GPU: percentiles and autocorrelation times are computed there, the "
                         "pickles hold None for (chain, lnprobability); needed for ensembles whose chain does not fit "
                         "in host memory")
    ap.add_argument("--predict-sled", type=int, nargs="+", default=None, metavar="J",
                    help="also summarise the posterior-predictive flux of these lines (1-based J, at most 16), per "
                         "component with two; computed on the GPU, so it works with --summaries-only")
    ap.add_argument("--moves", nargs="+", default=None, metavar="MOVE[:WEIGHT]",
                    help="sampler moves, e.g. de:0.8 stretch:0.2 (emcee's DEMove / StretchMove mixture; default: the "
                         "stretch move)")
    ap.add_argument("--corner-bins", type=int, default=None, metavar="B",
                    help="also compute the corner-plot counts (B-bin marginals of the summary columns and their pairs), "
                         "the covariance and the sample nearest the median, on the GPU (works with --summaries-only); "
                         "written to <source>_corner.npz")
    args = ap.parse_args(argv)
    logging.basicConfig(level=logging.INFO)
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    device = int(os.environ.get("LOCAL_RANK", "0"))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    datafile = args.data or os.path.join(root, "data", "flux.dat" if args.ncomp == 1 else "flux_for2p.dat")
    outdir = args.out or ("./single" if args.ncomp == 1 else "./double")
    data = read_data(datafile)
    sources = [s for s in data if args.sources is None or s in args.sources]
    moves = None if args.moves is None else parse_moves(args.moves)
    if args.concurrent:
        if world > 1:
            import torch
            import torch.distributed as dist
            torch.cuda.set_device(device)
            dist.init_process_group("nccl", device_id=torch.device("cuda", device))
        for res in fit_sources_concurrently(sources, data, ncomp=args.ncomp, nwalkers=args.walkers, n_iter_burn=args.burn,
                                            n_iter_walk=args.steps, seed=args.seed, device=device, outdir=outdir,
                                            datapath=args.datapath, allow_synthetic=args.allow_synthetic,
                                            chain_to_host=not args.summaries_only, predict_jup=args.predict_sled,
                                            corner_bins=args.corner_bins, moves=moves):
            if rank == 0:
                print_summary(res, args.ncomp)
        if world > 1:
            dist.destroy_process_group()
        return
    for source in sources[rank::world]:          # replicas only: one source per GPU at a time, no communication
        logger.info("Processing %s on GPU %d", source, device)
        res = fit_source(source, data, ncomp=args.ncomp, nwalkers=args.walkers, n_iter_burn=args.burn,
                         n_iter_walk=args.steps, seed=args.seed, device=device, outdir=outdir, datapath=args.datapath,
                         allow_synthetic=args.allow_synthetic, chain_to_host=not args.summaries_only,
                         predict_jup=args.predict_sled, corner_bins=args.corner_bins, moves=moves)
        print_summary(res, args.ncomp)


if __name__ == "__main__":
    main()
