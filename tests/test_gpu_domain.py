"""The solve and lnprob kernels against the oracle over the whole input domain the C ABI and `Radex` accept, not only the
config-2 box the other parity tests draw from (T in [tbg, 1000] K, n 1e2..1e7, N 10^15.5..10^19.5, dv = 1 km/s):

  - collision temperatures on, just below and just above every point of the rate table, below its first point (the
    low clamp), in its last two intervals and above its last point (the high clamp), up to T = 1e4 K;
  - densities 1 .. 1e10 cm^-3 and columns 1e5 .. 1e25 cm^-2, the limits themselves included;
  - line widths of 0.1 and 30 km/s, and a background far colder (0.02 K) or hotter (60 K) than the gas;
  - observed SLEDs of 1 and 16 lines reaching J_up = 40 (all three 16-line trips), unsorted, with a duplicate;
  - several two-component sources in one launch, and components outside the solvable range under wide bounds.

Every set is seeded.  The bars are those of test_gpu_solve (1e-5 on models the reference resolves, classified with the
oracle alone) and test_gpu_lnprob (max(1e-4, 1e-9 relative) on walkers whose reference value reproduces itself and
whose components the solve parity resolves; see resolved_walkers).  profiles/r4_domain_parity.json holds the measured
class counts and worst errors of every set."""
import ctypes as C

import numpy as np
import pytest

from conftest import MOLFILE, draw_params
from radex_emcee_b200 import _lib
from radex_emcee_b200 import emcee_radex_2comp as er2
from radex_emcee_b200.radex import Radex
from test_gpu_solve import check_against_oracle, gpu_solve, record

pytestmark = pytest.mark.gpu

OUTPUTS = ("xpop", "tex", "tau", "surf", "niter", "status")
ATOL = 1e-4
TBG = 2.7315


@pytest.fixture(scope="module")
def ctx():
    return _lib.Context(_lib.MolData(MOLFILE), 0)


def collision_temperatures(path=MOLFILE):
    """Every temperature of the file's rate tables (the synthetic co.dat: 25 points, 2 .. 3000 K, for both partners)."""
    rows = open(path).read().split("\n")
    temps = [float(v) for i, r in enumerate(rows) if r.startswith("!COLL TEMPS") for v in rows[i + 1].split()]
    return np.unique(temps)


def _dens_col(rng, n):
    P = draw_params(rng, n, TBG)
    return P[:, 1], P[:, 2]


# name -> (T, n(H2), N, tbg, deltav_kms); about 400 models each
def edge_set(name):
    rng = np.random.default_rng({"grid": 501, "cold": 502, "warm": 503, "hot": 504, "nN": 505, "dv0.1": 506,
                                 "dv30": 507, "tbg0.02": 508, "tbg60": 509}[name])
    if name == "grid":          # on every table point and one ULP to either side of it
        t = collision_temperatures()
        T = np.tile(np.concatenate([t, np.nextafter(t, 0.0), np.nextafter(t, np.inf)]), 5)
        return (T,) + _dens_col(rng, T.size) + (TBG, 1.0)
    if name == "cold":          # below the first point: the low clamp
        T = 10 ** rng.uniform(np.log10(0.05), np.log10(2.0), 400)
        return (T,) + _dens_col(rng, 400) + (TBG, 1.0)
    if name == "warm":          # the last two intervals, 1000 .. 3000 K
        T = 10 ** rng.uniform(3.0, np.log10(3000.0), 400)
        return (T,) + _dens_col(rng, 400) + (TBG, 1.0)
    if name == "hot":           # above the last point: the high clamp, up to the 1e4 K limit itself
        T = 10 ** rng.uniform(np.log10(3000.0), 4.0, 400)
        T[-20:] = 1e4
        return (T,) + _dens_col(rng, 400) + (TBG, 1.0)
    if name == "nN":            # free densities and columns, the column limits themselves included
        T = 10 ** rng.uniform(np.log10(TBG), 3.0, 400)
        nh2, N = 10 ** rng.uniform(0.0, 10.0, 400), 10 ** rng.uniform(5.0, 25.0, 400)
        N[:10], N[10:20] = 1e5, 1e25
        return T, nh2, N, TBG, 1.0
    if name.startswith("dv"):
        P = draw_params(rng, 400, TBG)
        return P[:, 0], P[:, 1], P[:, 2], TBG, float(name[2:])
    tbg = float(name[3:])
    T = 10 ** rng.uniform(np.log10(max(tbg, 0.05)) if tbg < 1.0 else np.log10(TBG), 3.0, 400)
    return (T,) + _dens_col(rng, 400) + (tbg, 1.0)


T_SETS = ("grid", "cold", "warm", "hot")
DV_SETS = ("dv0.1", "dv30")
ALL_SETS = T_SETS + ("nN",) + DV_SETS + ("tbg0.02", "tbg60")
# least well-posed fraction per set and geometry (1 sphere, 2 LVG, 3 slab).  The classification is the oracle's alone;
# measured: grid .96/.91/.88, cold 1/1/1, warm .82/.62/.52, hot .75/.43/.34, nN .94, dv0.1 .98/.87/.87, dv30
# .98/.98/.97, tbg0.02 .98, tbg60 .99 (LVG/sphere/slab).  Above 1000 K most config-2 (n, N) draws end at the 200-call
# cap or mase, in sphere and slab most of all.
MIN_WELL_POSED = {("grid", 2): 0.9, ("grid", 1): 0.85, ("grid", 3): 0.8, ("cold", 2): 0.95, ("cold", 1): 0.95,
                  ("cold", 3): 0.95, ("warm", 2): 0.75, ("warm", 1): 0.55, ("warm", 3): 0.45, ("hot", 2): 0.7,
                  ("hot", 1): 0.4, ("hot", 3): 0.3, ("nN", 2): 0.9, ("dv0.1", 2): 0.95, ("dv0.1", 1): 0.8,
                  ("dv0.1", 3): 0.8, ("dv30", 2): 0.95, ("dv30", 1): 0.95, ("dv30", 3): 0.9, ("tbg0.02", 2): 0.95,
                  ("tbg60", 2): 0.95}
CASES = ([(s, 2, None) for s in ALL_SETS] + [(s, m, None) for s in T_SETS + DV_SETS for m in (1, 3)]
         + [(s, 2, 1) for s in T_SETS])


@pytest.mark.parametrize("name,method,kernel", CASES)
def test_edge_set_vs_oracle(ctx, name, method, kernel):
    """rb_solve_batch on each edge set against the oracle: 1e-5 on the well-posed models, excluded LVG models on one of
    the reference's own answers, non-finite brightness flagged.  kernel = 1 runs the general path (v1_rates has its own
    interpolation of the rate table)."""
    T, nh2, N, tbg, dv = edge_set(name)
    got = gpu_solve(ctx, T, nh2, N, tbg, method, dv, kernel=kernel)
    assert ((got["status"] & 3) == 0).all(), name
    label = "domain_%s_method%d%s" % (name, method, "_kernel1" if kernel == 1 else "")
    check_against_oracle(got, T, nh2, N, tbg, method, label, min_well_posed=MIN_WELL_POSED[name, method], deltav_kms=dv)


@pytest.mark.parametrize("kernel", [None, 1])
@pytest.mark.parametrize("method", [1, 2, 3])
def test_range_status_at_the_limits(ctx, method, kernel):
    """T = 1e4 K and N = 1e5 / 1e25 cm^-2 are solved; one ULP past them is the reference's ValueError: status
    T_RANGE / N_RANGE, NaN outputs, no iterations."""
    T = np.array([1e4, np.nextafter(1e4, np.inf), 50.0, 50.0, 50.0, 50.0])
    N = np.array([1e16, 1e16, 1e5, np.nextafter(1e5, 0.0), 1e25, np.nextafter(1e25, np.inf)])
    out = gpu_solve(ctx, T, np.full(6, 1e4), N, TBG, method, kernel=kernel)
    assert list(out["status"] & 3) == [0, 1, 0, 2, 0, 2], out["status"]
    bad = np.array([1, 3, 5])
    assert np.isnan(out["surf"][bad]).all() and np.isnan(out["xpop"][bad]).all() and (out["niter"][bad] == 0).all()
    assert np.isfinite(out["xpop"][[0, 2, 4]]).all() and (out["niter"][[0, 2, 4]] > 0).all()


# ---- the same models through the scheduled launches --------------------------------------------------------------------
SCHED_GROUPS = {"tbg2.7315": T_SETS + ("nN",), "dv0.1": ("dv0.1",), "dv30": ("dv30",), "tbg0.02": ("tbg0.02",),
                "tbg60": ("tbg60",)}


def replicated(names, n=20000):
    """The edge sets of one (tbg, dv) setting repeated to n models; copy k has its densities scaled by 1 + 1e-9 k, so
    every model is distinct while every copy keeps the sets' temperatures and columns exactly (grid points, 1e4 K,
    1e5 and 1e25 cm^-2)."""
    parts = [edge_set(s) for s in names]
    tbg, dv = parts[0][3], parts[0][4]
    assert all(p[3] == tbg and p[4] == dv for p in parts)
    base = np.column_stack([np.concatenate([p[i] for p in parts]) for i in range(3)])
    m = base.shape[0]
    P = base[np.arange(n) % m]
    P[:, 1] *= 1.0 + 1e-9 * (np.arange(n) // m)
    return P, m, tbg, dv


@pytest.mark.parametrize("group", list(SCHED_GROUPS))
def test_edge_sets_through_the_scheduled_launches(ctx, group):
    """>= 20000 edge models in one call: the default schedule, the 20/24/28-level lead blocks in their own launches
    (park_max = 7) and the ordering without the half-warp engines (kernel = 4) all repeat the single launch (kernel = 3)
    bit for bit -- outputs, iteration total and cache statistics; a sample of the scheduled run against the oracle."""
    P, m, tbg, dv = replicated(SCHED_GROUPS[group])
    T, nh2, N = P[:, 0], P[:, 1], P[:, 2]
    ref = gpu_solve(ctx, T, nh2, N, tbg, 2, dv, kernel=3)
    itr, _ = ctx.counters()
    sr = ctx.cache_stats()
    runs = {}
    for kw in ({}, {"park_max": 7}, {"kernel": 4}):
        a = gpu_solve(ctx, T, nh2, N, tbg, 2, dv, **kw)
        ita, _ = ctx.counters()
        runs[str(kw)] = a
        assert ita == itr, (group, kw, ita, itr)
        assert tuple(ctx.cache_stats()) == tuple(sr), (group, kw, ctx.cache_stats(), sr)
        for k in OUTPUTS:
            np.testing.assert_array_equal(a[k], ref[k], err_msg="%s %s %s" % (group, k, kw))
    assert sr[1] > 0, sr            # lead blocks were captured: the scheduled path ran
    got = runs["{}"]
    sel = np.sort(np.random.default_rng(600).choice(m, 300, replace=False))
    sample = {k: v[sel] for k, v in got.items()}
    check_against_oracle(sample, T[sel], nh2[sel], N[sel], tbg, 2, "domain_scheduled_%s" % group,
                         min_well_posed=0.85 if group == "tbg2.7315" else 0.95, deltav_kms=dv)   # measured .88, >= .97


# ---- N / dv: the physics and the code only use cdmol / deltav -----------------------------------------------------------
def _metamorphic_models(n, seed):
    rng = np.random.default_rng(seed)
    P = draw_params(rng, n, TBG)
    P[0::4, 0] = 10 ** rng.uniform(np.log10(0.05), np.log10(2.0), P[0::4].shape[0])
    P[1::4, 0] = 10 ** rng.uniform(3.0, 4.0, P[1::4].shape[0])
    return P


@pytest.mark.parametrize("path,method,n,kw", [("small", 2, 512, {}), ("scheduled", 2, 20000, {}),
                                              ("kernel1", 2, 256, {"kernel": 1}), ("sphere", 1, 512, {}),
                                              ("slab", 3, 512, {})])
def test_column_and_width_scale_together(ctx, path, method, n, kw):
    """Scaling N and dv by the same power of two leaves cdmol / deltav, and so every output, unchanged to the bit."""
    P = _metamorphic_models(n, 700 + method + n)
    T, nh2, N = P[:, 0], P[:, 1], P[:, 2]
    base = gpu_solve(ctx, T, nh2, N, TBG, method, 1.0, **kw)
    it0, _ = ctx.counters()
    assert ((base["status"] & 3) == 0).all()
    for k in (5, -3):
        s = 2.0 ** k
        assert (N * s >= 1e5).all() and (N * s <= 1e25).all()
        got = gpu_solve(ctx, T, nh2, N * s, TBG, method, s, **kw)
        assert ctx.counters()[0] == it0, (path, k)
        for key in OUTPUTS:
            np.testing.assert_array_equal(got[key], base[key], err_msg="%s %s dv=%g" % (path, key, s))


def test_radex_class_line_width(oracle):
    """Radex(column=..., deltav=5) against the oracle at deltav_kms = 5."""
    import warnings
    P = _metamorphic_models(96, 710)
    T, nh2, N = P[:, 0], P[:, 1], P[:, 2]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        R = Radex(species="co", density={"oH2": 0.75 * nh2, "pH2": 0.25 * nh2}, column=N, temperature=T,
                  tbackground=TBG, deltav=5.0)
    niter = R.run_radex()
    got = dict(xpop=R.level_population, tex=R.tex, tau=R.tau, surf=R.source_line_surfbrightness,
               niter=np.asarray(niter), status=np.asarray(R.status))
    check_against_oracle(got, T, nh2, N, TBG, 2, "domain_radex_deltav5", min_well_posed=0.9,   # measured .94
                         deltav_kms=5.0)


# ---- full SLEDs in the likelihood -------------------------------------------------------------------------------------
JUP = {1: np.array([40]),
       6: np.array([33, 1, 40, 16, 32, 17]),
       16: np.array([33, 1, 40, 17, 16, 32, 5, 9, 24, 28, 36, 12, 20, 3, 38, 17])}     # unsorted; 17 twice
TRUTH1 = np.array([6.0, 3.0, 18.0, -10.0])
TRUTH2 = np.array([3.0, 1.3, 16.5, -10.0, 5.5, 3.0, 18.5, -10.3])
T_D = 30.0


def sled_source(oracle, truth, jup, tbg, seed):
    """Fluxes (Jy km/s) of the oracle's model at `truth`, with 3 % noise and 5 % errors: chi^2 of order nobs there."""
    rng = np.random.default_rng(seed)
    model = np.zeros(jup.size)
    for c in range(truth.size // 4):
        n, t, col, size = truth[4 * c: 4 * c + 4]
        surf = oracle.solve_batch([10 ** t], [0.25 * 10 ** n], [0.75 * 10 ** n], [10 ** col], tbg=tbg)["surf"][0]
        model += surf[jup - 1] * 10 ** size * 1e23
    flux = model * (1 + 0.03 * rng.standard_normal(jup.size))
    return flux, 0.05 * np.abs(flux)


def sled_bounds(ncomp, tbg):
    b = np.array([[1.0, 8.0], [np.log10(tbg), 3.6], [13.0, 21.0], [-13.0, -7.0]])
    return np.vstack([b] * ncomp)


def sled_walkers(rng, truth, bounds, n_near, n_wide):
    near = truth + rng.standard_normal((n_near, truth.size)) * np.tile([0.3, 0.1, 0.3, 0.2], truth.size // 4)
    return np.vstack([near, rng.uniform(bounds[:, 0] - 0.05, bounds[:, 1] + 0.05, (n_wide, truth.size))])


def rb_lnprob(ctx, P, jup, flux, eflux, bounds, tbg, T_d=None, **optkw):
    ncomp = P.shape[1] // 4
    P = np.ascontiguousarray(P)
    out, ns = np.empty(P.shape[0]), C.c_int64(0)
    obs, opts, b = _lib.make_obs(jup, flux, eflux), _lib.default_opts(**optkw), np.ascontiguousarray(bounds)
    if ncomp == 1:
        _lib.check(_lib.load().rb_lnprob1(ctx.handle, P.shape[0], _lib.ptr(P), C.byref(obs), _lib.ptr(b), tbg,
                                          C.byref(opts), _lib.ptr(out), C.byref(ns)))
    else:
        _lib.check(_lib.load().rb_lnprob2(ctx.handle, P.shape[0], _lib.ptr(P), C.byref(obs), _lib.ptr(b),
                                          int(T_d is not None), float(T_d or 0.0), tbg, C.byref(opts), _lib.ptr(out),
                                          C.byref(ns)))
    return out, ns.value


def oracle_lnprob(oracle, P, jup, flux, eflux, bounds, tbg, T_d=None):
    if P.shape[1] == 4:
        return np.array([oracle.lnprob1(p, jup, flux, eflux, bounds, tbg) for p in P])
    return np.array([oracle.lnprob2(p, jup, flux, eflux, bounds, T_d, tbg) for p in P])


def resolved_walkers(P, jup, tbg):
    """Walkers whose model the solve parity vouches for.  Every solved component must be well_posed in parity.classify:
    no line of it a maser (tau < -3 anywhere, not only on the observed lines: a maser amplifies the rounding of the
    whole iteration, and the reference's own fluxes then move by ~1e-6 under its 1e-13 perturbations), brightness
    finite, the reference reproducing itself.  And on every observed line, the components whose upper level lies below
    the 1e-9 population floor of parity.rel_errors give less than 1e-6 of the model flux: high-J levels of cool gas sit
    far below that floor, where the reference's own populations carry no stated precision.  Far from the data chi^2
    with 5 % errors turns a relative model error e into a relative lnprob error of ~2 e, so the 1e-9 bar needs both."""
    from oracle import parity
    ok = np.ones(P.shape[0], dtype=bool)
    total, unresolved = np.zeros((P.shape[0], jup.size)), np.zeros((P.shape[0], jup.size))
    for c in range(P.shape[1] // 4):
        T, n, N = 10 ** P[:, 4 * c + 1], 10 ** P[:, 4 * c], 10 ** P[:, 4 * c + 2]
        run = (T > 0) & (T <= 1e4) & (N >= 1e5) & (N <= 1e25)
        ref, cls, _ = parity.classify(MOLFILE, np.where(run, T, 50.0), n, np.where(run, N, 1e15), tbg)
        ok &= ~run | cls["well_posed"]
        with np.errstate(all="ignore"):
            flux = np.abs(ref["surf"][:, jup - 1]) * 10 ** P[:, 4 * c + 3, None]
            total += np.where(run[:, None], flux, 0.0)
            unresolved += np.where(run[:, None] & ~(ref["xpop"][:, jup] > 1e-9), flux, 0.0)
    with np.errstate(all="ignore"):
        return ok & (unresolved <= 1e-6 * total).all(axis=1)


def check_lnprob_against_oracle(oracle, got, P, jup, flux, eflux, bounds, tbg, T_d, label, min_finite):
    """test_gpu_lnprob's comparison: the same -inf pattern; max(1e-4, 1e-9 relative) on the finite walkers whose reference
    value reproduces itself under a 1e-13 shift of the walker (and is not a maser blow-up), and whose components the
    solve parity resolves (resolved_walkers)."""
    ref = oracle_lnprob(oracle, P, jup, flux, eflux, bounds, tbg, T_d)
    assert not np.isnan(got).any(), label
    np.testing.assert_array_equal(got == -np.inf, ref == -np.inf, err_msg=label)
    fin = np.isfinite(ref)
    assert fin.sum() >= min_finite, (label, fin.sum())
    ref2 = oracle_lnprob(oracle, P + 1e-13, jup, flux, eflux, bounds, tbg, T_d)
    with np.errstate(invalid="ignore"):
        ok = fin & (np.abs(ref2 - ref) < 1e-7 * np.maximum(1.0, np.abs(ref))) & (np.abs(ref) < 1e12)
    ok &= resolved_walkers(P, jup, tbg)
    err = np.abs(got[ok] - ref[ok])
    bar = np.maximum(ATOL, 1e-9 * np.abs(ref[ok]))
    record(label, walkers=int(P.shape[0]), finite=int(fin.sum()), well_posed=int(ok.sum()),
           max_abs_err_well_posed=float(err.max()) if ok.any() else None,
           max_err_in_units_of_the_bar=float((err / bar).max()) if ok.any() else None)
    assert ok.sum() >= 0.6 * fin.sum(), (label, ok.sum(), fin.sum())
    assert (err < bar).all(), (label, err.max())
    return ref


SLED_CASES = [(1, None), (2, T_D), (2, None)]


@pytest.mark.parametrize("nobs", sorted(JUP))
@pytest.mark.parametrize("ncomp,T_d", SLED_CASES)
def test_full_sled_vs_oracle(ctx, oracle, ncomp, T_d, nobs):
    """Observed lines from all three 16-line trips (J_up 1 .. 40), up to RB_MAX_OBS of them, unsorted, one duplicated:
    the fused lnprob kernel against the oracle's lnprob1 / lnprob2."""
    jup, tbg = JUP[nobs], TBG * 1.8
    truth = TRUTH1 if ncomp == 1 else TRUTH2
    flux, eflux = sled_source(oracle, truth, jup, tbg, 800 + nobs)
    bounds = sled_bounds(ncomp, tbg)
    P = sled_walkers(np.random.default_rng(810 + nobs + ncomp), truth, bounds, 200 if ncomp == 1 else 160, 56)
    got, ns = rb_lnprob(ctx, P, jup, flux, eflux, bounds, tbg, T_d)
    check_lnprob_against_oracle(oracle, got, P, jup, flux, eflux, bounds, tbg, T_d,
                                "domain_sled_%dcomp_td%s_nobs%d" % (ncomp, T_d, nobs), min_finite=80)


@pytest.mark.parametrize("nobs", [1, 16])
@pytest.mark.parametrize("ncomp,T_d", SLED_CASES)
def test_full_sled_pipeline_equals_fused_kernel(ctx, oracle, ncomp, T_d, nobs):
    """Above 8192 walkers the same sources run as the pipeline (scheduled solve writing only the observed lines'
    fluxes, obs_surf stride RB_MAX_OBS): the -inf pattern, the solve count and the values of the fused launch."""
    jup, tbg = JUP[nobs], TBG * 1.8
    truth = TRUTH1 if ncomp == 1 else TRUTH2
    flux, eflux = sled_source(oracle, truth, jup, tbg, 800 + nobs)
    bounds = sled_bounds(ncomp, tbg)
    P = sled_walkers(np.random.default_rng(820 + nobs + ncomp), truth, bounds, 8000, 1500)
    a, na = rb_lnprob(ctx, P, jup, flux, eflux, bounds, tbg, T_d)
    b, nb = rb_lnprob(ctx, P, jup, flux, eflux, bounds, tbg, T_d, kernel=3)
    assert na == nb, (na, nb)
    np.testing.assert_array_equal(a == -np.inf, b == -np.inf)
    fin = np.isfinite(a)
    assert fin.sum() > 4000 and not np.isnan(a).any()
    np.testing.assert_allclose(a[fin], b[fin], rtol=1e-13, atol=0)


# ---- several two-component sources in one launch ----------------------------------------------------------------------
def test_sources_with_two_components_in_one_launch(ctx, oracle):
    """rb_lnprob_src_dev with ncomp = 2: sources that differ in nobs (up to 16), tbg, bounds and T_d, walkers assigned by
    a random permutation.  Every walker equals rb_lnprob2 of its own source bit for bit; a sample matches the oracle."""
    import torch
    from radex_emcee_b200.sampler import CudaEngine, SLEDModel
    specs = [(1, TBG * 1.5, T_D), (16, TBG * 3.0, None), (6, TBG * 2.2, 20.0), (3, TBG * 4.0, None)]
    srcs = []
    for s, (nobs, tbg, td) in enumerate(specs):
        jup = JUP[nobs] if nobs in JUP else np.array([2, 7, 21])
        truth = TRUTH2 + np.tile([0.2 * s, 0.0, 0.2 * s, 0.0], 2)     # denser and thicker; the temperatures stay
        flux, eflux = sled_source(oracle, truth, jup, tbg, 900 + s)
        bounds = sled_bounds(2, tbg)
        bounds[[2, 6]] = [[12.0 + 0.5 * s, 20.5 + 0.3 * s]] * 2
        srcs.append(dict(jup=jup, flux=flux, eflux=eflux, bounds=bounds, tbg=tbg, T_d=td, truth=truth))
    per = 2200
    rng = np.random.default_rng(910)
    src_id = rng.permutation(np.repeat(np.arange(len(srcs)), per)).astype(np.int32)
    P = np.empty((src_id.size, 8))
    for s, S in enumerate(srcs):
        P[src_id == s] = sled_walkers(rng, S["truth"], S["bounds"], per - 400, 400)
    eng = CudaEngine(ctx, [SLEDModel(2, S["jup"], S["flux"], S["eflux"], S["bounds"], S["tbg"], S["T_d"]) for S in srcs])
    dev = eng.device
    try:
        got = eng.lnprob(torch.from_numpy(P).to(dev), torch.from_numpy(src_id).to(dev)).cpu().numpy()
        ns_all = int(eng.nsolves.item())
    finally:
        ctx.reset_stream()
    assert not np.isnan(got).any()
    ns_sum = 0
    for s, S in enumerate(srcs):
        m = src_id == s
        own, ns = rb_lnprob(ctx, P[m], S["jup"], S["flux"], S["eflux"], S["bounds"], S["tbg"], S["T_d"])
        ns_sum += ns
        np.testing.assert_array_equal(got[m], own, err_msg="source %d" % s)
        k = np.nonzero(m)[0][:48]
        check_lnprob_against_oracle(oracle, got[k], P[k], S["jup"], S["flux"], S["eflux"], S["bounds"], S["tbg"],
                                    S["T_d"], "domain_srcset_2comp_source%d" % s, min_finite=10)
    assert ns_all == ns_sum, (ns_all, ns_sum)


# ---- components outside the solvable range under wide bounds ----------------------------------------------------------
def test_out_of_range_components_under_wide_bounds(ctx, oracle):
    """Bounds admitting log T up to 4.2 and log N from 4 to 25.5 leave the prior finite where a component is outside
    the reference's range (T <= 1e4 K, 1e5 <= N <= 1e25): pyradex raises ValueError at the first such component, so
    the walker is -inf and the components after it are never solved.  Fused launch and pipeline give the oracle's -inf
    pattern and count the solves the reference makes: both components, the first only, or none."""
    jup, tbg = JUP[6], TBG * 1.8
    flux, eflux = sled_source(oracle, TRUTH2, jup, tbg, 950)
    bounds = np.array([[-8.0, 17.0], [np.log10(tbg), 4.2], [4.0, 25.5], [-14.0, -6.0]] * 2)
    rng = np.random.default_rng(951)
    k = 500
    cases = {"in": TRUTH2 + rng.standard_normal((6000, 8)) * np.tile([0.3, 0.1, 0.3, 0.2], 2)}
    edge = np.tile(TRUTH2, (k, 1)) + rng.standard_normal((k, 8)) * np.tile([0.2, 0.05, 0.2, 0.0], 2)
    edge[:, 3], edge[:, 7] = -10.0, -10.5
    for name, (col, val) in {"c0_N_high": (2, 25.3), "c0_N_low": (2, 4.5), "c1_N_high": (6, 25.3),
                             "c1_T_high": (5, 4.1)}.items():
        e = edge.copy()
        e[:, col] = val + 0.05 * rng.uniform(-1, 1, k)
        if col in (2, 6):
            e[:, col - 2] = e[:, col] - 12.0
        cases[name] = e
    both = edge.copy()
    both[:, 1], both[:, 5] = 4.05, 4.15
    cases["both_T_high"] = both
    both = edge.copy()
    both[:, 2], both[:, 6] = 25.3, 4.5
    both[:, 0], both[:, 4] = 13.3, -7.5
    cases["both_N"] = both
    P = np.vstack(list(cases.values()))
    label = np.concatenate([np.full(len(v), i) for i, v in enumerate(cases.values())])
    lp_ok = np.isfinite(er2.lnprior(P, bounds))
    T, N = 10.0 ** P[:, [1, 5]], 10.0 ** P[:, [2, 6]]
    ok = (T > 0) & (T <= 1e4) & (N >= 1e5) & (N <= 1e25)
    for i, name in enumerate(cases):
        if name != "in":
            m = label == i
            assert lp_ok[m].mean() > 0.9 and not (ok[m].all(axis=1)).any(), name
    expected = int(np.where(lp_ok, np.where(ok[:, 0], 1 + ok[:, 1], 0), 0).sum())
    a, na = rb_lnprob(ctx, P, jup, flux, eflux, bounds, tbg)
    b, nb = rb_lnprob(ctx, P, jup, flux, eflux, bounds, tbg, kernel=3)
    assert P.shape[0] >= 8192
    assert nb == expected, (nb, expected)
    assert na == expected, (na, expected)
    np.testing.assert_array_equal(a == -np.inf, b == -np.inf)
    fin = np.isfinite(a)
    np.testing.assert_allclose(a[fin], b[fin], rtol=1e-13, atol=0)
    assert (a[lp_ok & ~ok.all(axis=1)] == -np.inf).all()
    # the oracle on every out-of-range walker and a sample of the others
    sel = np.concatenate([np.nonzero(label > 0)[0], np.arange(200)])
    ref = oracle_lnprob(oracle, P[sel], jup, flux, eflux, bounds, tbg)
    np.testing.assert_array_equal(a[sel] == -np.inf, ref == -np.inf)
