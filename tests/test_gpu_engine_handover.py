"""The cached engines (k_lvg_small<KP>) hand a model over while the previous one still iterates: each half-warp holds the
queue ticket of its next model, walks ticket -> order -> capture offset during the current model's calls, and copies the
parked capture into its slab with asynchronous 16-byte copies.  These tests give the engines queues of a few models per
half-warp, so every half hands over many times and ends holding a ticket past its queue, with odd model counts per lead
size, so a half idles while its partner finishes.  Each case repeats the single launch (kernel = 3) bit for bit: outputs,
iteration total and cache statistics."""
import numpy as np
import pytest

from conftest import MOLFILE, draw_params
from radex_emcee_b200 import _lib
from test_gpu_domain import JUP, TBG, TRUTH1, TRUTH2, T_D, rb_lnprob, sled_bounds, sled_source, sled_walkers
from test_gpu_solve import gpu_solve

pytestmark = pytest.mark.gpu

OUTPUTS = ("xpop", "tex", "tau", "surf", "niter", "status")


@pytest.fixture(scope="module")
def ctx():
    return _lib.Context(_lib.MolData(MOLFILE), 0)


@pytest.fixture(scope="module")
def pool(ctx):
    """Config-2 draws and the lead-block size (in panels, 3 .. 7) their converged optical depths call for."""
    P = draw_params(np.random.default_rng(95), 30000, 10.926)
    first = gpu_solve(ctx, P[:, 0], P[:, 1], P[:, 2], 10.926, kernel=3)
    thick = ~(np.abs(first["tau"]) * 0.5 < np.float32(0.01))
    top = np.where(thick.any(axis=1), thick.shape[1] - np.argmax(thick[:, ::-1], axis=1), -1)
    return P, np.minimum(7, np.maximum(3, (top + 1 + 4) >> 2))


def batch_of(P, key, counts, seed):
    """counts[k] distinct models of lead size k each (taken from the pool's models of that size), shuffled."""
    rows = []
    for k, c in counts.items():
        sel = np.nonzero(key == k)[0]
        assert sel.size > 20, (k, sel.size)
        rows.append(np.resize(sel, c))
    idx = np.random.default_rng(seed).permutation(np.concatenate(rows))
    Q = P[idx].copy()
    Q[:, 0] *= 1.0 + 1e-9 * np.arange(Q.shape[0])        # distinct models of the same class
    return Q


def check_bit_identical(ctx, Q, label, **kw):
    ref = gpu_solve(ctx, Q[:, 0], Q[:, 1], Q[:, 2], 10.926, kernel=3, **kw)
    itr, _ = ctx.counters()
    sr = tuple(ctx.cache_stats())
    for park_max in (None, 7):
        a = gpu_solve(ctx, Q[:, 0], Q[:, 1], Q[:, 2], 10.926, park_max=park_max, **kw)
        ita, _ = ctx.counters()
        assert ita == itr, (label, park_max, kw, ita, itr)
        assert tuple(ctx.cache_stats()) == sr, (label, park_max, kw)
        for k in OUTPUTS:
            np.testing.assert_array_equal(a[k], ref[k], err_msg="%s %s park_max %s %s" % (k, label, park_max, kw))
    assert sr[1] > 0.3 * Q.shape[0], (label, sr)     # the captures were made: the engines ran


# odd counts per lead size; 148 SMs hold 5328 / 4144 / 2960 / 2368 / 2072 half-warps of the 12 .. 28-level engines,
# so every queue is a few models per half (or fewer than one)
@pytest.mark.parametrize("counts", [
    {3: 9001, 4: 4001, 5: 1501, 6: 901, 7: 501},
    {3: 20001, 4: 7001, 5: 3001, 6: 2001, 7: 1001},
    {3: 2001, 4: 1001, 5: 3, 6: 1, 7: 2001},
], ids=["few", "several", "sparse"])
def test_engine_queues_of_a_few_models_per_half(ctx, pool, counts):
    P, key = pool
    Q = batch_of(P, key, counts, sum(counts.values()))
    check_bit_identical(ctx, Q, str(counts))
    check_bit_identical(ctx, Q, str(counts), stop_rule=_lib.STOP_RADEX)
    check_bit_identical(ctx, Q, str(counts), maxiter=12)


def test_capture_buffer_full_with_engines_running(ctx, pool):
    """Models of the 28-level class fill the capture buffer (832 doubles budgeted per model, 1312 taken): the ones that
    find it full finish in launch A while the rest, and every smaller lead size, hand over through the engines."""
    P, key = pool
    Q = batch_of(P, key, {7: 12001, 3: 3001, 4: 1001}, 7)
    check_bit_identical(ctx, Q, "ext full")


@pytest.mark.parametrize("nobs", [1, 16])
@pytest.mark.parametrize("ncomp,T_d", [(1, None), (2, T_D)])
def test_lnprob_pipeline_through_the_engines(ctx, oracle, ncomp, T_d, nobs):
    """At >= 8192 walkers lnprob runs as the pipeline, whose scheduled solve writes only the observed lines' brightness
    (obs_surf) from the engines' epilogue, here with every lead size in its engine (park_max = 7) and an odd walker
    count: the -inf pattern, the solve count and the values of the fused launch, as in test_gpu_domain."""
    jup, tbg = JUP[nobs], TBG * 1.8
    truth = TRUTH1 if ncomp == 1 else TRUTH2
    flux, eflux = sled_source(oracle, truth, jup, tbg, 800 + nobs)
    bounds = sled_bounds(ncomp, tbg)
    P = sled_walkers(np.random.default_rng(820 + nobs + ncomp), truth, bounds, 8000, 1501)
    a, na = rb_lnprob(ctx, P, jup, flux, eflux, bounds, tbg, T_d, park_max=7)
    c, nc = rb_lnprob(ctx, P, jup, flux, eflux, bounds, tbg, T_d, kernel=3)
    assert na == nc, (na, nc)
    np.testing.assert_array_equal(a == -np.inf, c == -np.inf)
    fin = np.isfinite(a)
    assert fin.sum() > 4000 and not np.isnan(a).any()
    np.testing.assert_allclose(a[fin], c[fin], rtol=1e-13, atol=0)


def test_table_whose_lead_lines_lie_elsewhere(ctx, tmp_path):
    """The engines keep per-line slots only for the lines that can be lead lines in a CO-like table (the first 16 or
    32).  A table listing its lines in another order runs its cached iterations in launch B instead: the same bits as
    kernel = 3 on that table, and the cache statistics of the CO-ordered table."""
    rows = open(MOLFILE).read().split("\n")
    k = next(i for i, r in enumerate(rows) if r.startswith("!NUMBER OF RADIATIVE"))
    nline = int(rows[k + 1])
    first = k + 3
    perm = np.arange(nline)[::-1]       # the lowest transitions last: lead lines in the third trip
    block = ["%5d %s" % (i + 1, " ".join(rows[first + p].split()[1:])) for i, p in enumerate(perm)]
    path = tmp_path / "co_reversed.dat"
    path.write_text("\n".join(rows[:first] + block + rows[first + nline:]))
    ctx2 = _lib.Context(_lib.MolData(str(path)), 0)
    P = draw_params(np.random.default_rng(96), 20001, 10.926)
    a = gpu_solve(ctx, P[:, 0], P[:, 1], P[:, 2], 10.926, park_max=7)
    sa = tuple(ctx.cache_stats())
    b = gpu_solve(ctx2, P[:, 0], P[:, 1], P[:, 2], 10.926, park_max=7)
    sb = tuple(ctx2.cache_stats())
    ref = gpu_solve(ctx2, P[:, 0], P[:, 1], P[:, 2], 10.926, kernel=3)
    assert sa == sb, (sa, sb)
    for key in OUTPUTS:
        np.testing.assert_array_equal(b[key], ref[key], err_msg=key)
    for key in ("xpop", "niter", "status"):
        np.testing.assert_array_equal(a[key], b[key], err_msg=key)
    for key in ("tex", "tau", "surf"):
        np.testing.assert_array_equal(a[key][:, perm], b[key], err_msg=key)
