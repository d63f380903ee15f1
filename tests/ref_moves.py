"""Test-only numpy restatement of the moves of csrc/stretch.cuh beyond the stretch move: the k-group split
(st2::slot_walker), the differential-evolution propose / accept (st2::k_de_propose, k_accept2 with the DE stream) and
the move schedule (rb_move_schedule).  Same Philox streams, same roundings.  ``MovesNumpyEngine`` adds the DE calls to
ref_engine.NumpyEngine so that the sampler's DE and mixture paths run on CPU.  Never imported by the package."""
import numpy as np
import torch

from ref_engine import MASK, NumpyEngine, _counters, philox4x32_10, split_perm, u01

DE_PAIR, DE_GAUSS, DE_ACCEPT, DE_MAX_TRIES = 0, 1, 255, 200
RB_MOVE_STRETCH, RB_MOVE_DE = 0, 1


def group_size(B, ngroups, g):
    return B // ngroups + (1 if g < B % ngroups else 0)


def group_off(B, ngroups, g):
    return g * (B // ngroups) + min(g, B % ngroups)


def _split_keys(split, gb, step):
    st = np.full(gb.shape, step, dtype=np.uint64)
    k0 = (split.seed & 0xFFFFFFFF) ^ 0x53504C54
    k1 = ((split.seed >> 32) & 0xFFFFFFFF) ^ 0x72616E64
    return philox4x32_10(gb & MASK, gb >> np.uint64(32), st & MASK, st >> np.uint64(32), k0, k1)


def block_walker(split, step, g, ngroups, gb, t):
    """Index within its block of slot t of group g in global block gb (arrays)."""
    t = np.asarray(t, dtype=np.int64)
    if not split.randomize:
        return g + ngroups * t
    gb = np.asarray(gb, dtype=np.uint64)
    x = (group_off(split.block, ngroups, g) + t).astype(np.uint64)
    return split_perm(x, split.block, _split_keys(split, gb, step)).astype(np.int64)


def slot_walker(split, step, g, ngroups, gid_base, k):
    """Local walker index of the local slots k (array) of group g of ngroups."""
    B = split.block
    n = group_size(B, ngroups, g)
    k = np.asarray(k, dtype=np.int64)
    lb, t = k // n, k % n
    return lb * B + block_walker(split, step, g, ngroups, (gid_base // B + lb).astype(np.uint64), t)


def nslots(split, nlocal, ngroups, g):
    return nlocal // split.block * group_size(split.block, ngroups, g)


# ---- differential evolution ---------------------------------------------------------------------------------------
def de_keys(seed):
    return (seed & 0xFFFFFFFF) ^ 0x44456D76, ((seed >> 32) & 0xFFFFFFFF) ^ 0x6D6F7665


def de_counter(gid, step, g, draw):
    gid = np.asarray(gid, dtype=np.uint64)
    sg = int(step) * 4 + g
    c2 = np.full(gid.shape, sg & 0xFFFFFFFF, dtype=np.uint64)
    c3 = np.full(gid.shape, ((sg >> 32) & 0x00FFFFFF) | (draw << 24), dtype=np.uint64)
    return gid & MASK, gid >> np.uint64(32), c2, c3


def ln_rn(x):
    """st2::ln_rn: ln x from IEEE operations only (numpy does not contract into FMA)."""
    m, e = np.frexp(np.asarray(x, dtype=np.float64))
    small = m < 0.70710678118654752
    m = np.where(small, m * 2.0, m)
    e = np.where(small, e - 1, e)
    s = (m - 1.0) / (m + 1.0)
    s2 = s * s
    p = np.full(s.shape, 1.0 / 21.0)
    for k in range(19, 0, -2):
        p = 1.0 / k + s2 * p
    return e.astype(np.float64) * 0.69314718055994531 + 2.0 * (s * p)


def de_gauss(gid, step, g, k0, k1):
    """st2::de_gauss: polar Box-Muller, one Philox call per try."""
    gid = np.asarray(gid, dtype=np.uint64)
    n = np.zeros(gid.shape)
    todo = np.ones(gid.shape, dtype=bool)
    for t in range(DE_MAX_TRIES):
        if not todo.any():
            break
        idx = np.nonzero(todo)[0]
        c = philox4x32_10(*de_counter(gid[idx], step, g, DE_GAUSS + t), k0, k1)
        v1 = 2.0 * u01(c[0], c[1]) - 1.0
        v2 = 2.0 * u01(c[2], c[3]) - 1.0
        r = v1 * v1 + v2 * v2
        ok = (r > 0.0) & (r < 1.0)
        with np.errstate(divide="ignore", invalid="ignore"):
            n[idx[ok]] = v1[ok] * np.sqrt((-2.0 * ln_rn(r[ok])) / r[ok])
        todo[idx[ok]] = False
    return n


def de_partner(split, step, g, src, j):
    """Global walker id of index j of the complement of group g within source src (arrays)."""
    W, B = split.walkers_per_source, split.block
    bps = W // B
    j = np.asarray(j, dtype=np.int64)
    src = np.asarray(src, dtype=np.int64)
    h1, h2 = (1 if g == 0 else 0), (1 if g == 2 else 2)
    n1 = bps * group_size(B, 3, h1)
    second = j >= n1
    out = np.empty(j.shape, dtype=np.int64)
    for h, m, jj in ((h1, ~second, j), (h2, second, j - n1)):
        if m.any():
            n = group_size(B, 3, h)
            lb, t = jj[m] // n, jj[m] % n
            gb = (src[m] * bps + lb).astype(np.uint64)
            out[m] = gb.astype(np.int64) * B + block_walker(split, step, h, 3, gb, t)
    return out


def de_propose_np(split, step, g, gid_base, X, Xall, gamma0, sigma):
    """(Q, src_id, local walker i, gamma, n, partner ids w1, w2) of the local slots of DE group g."""
    W, B = split.walkers_per_source, split.block
    ns = nslots(split, X.shape[0], 3, g)
    i = slot_walker(split, step, g, 3, gid_base, np.arange(ns))
    gid = (gid_base + i).astype(np.uint64)
    src = (gid // np.uint64(W)).astype(np.int64)
    nc = W - W // B * group_size(B, 3, g)
    k0, k1 = de_keys(split.seed)
    c = philox4x32_10(*de_counter(gid, step, g, DE_PAIR), k0, k1)
    npair = nc * (nc - 1)
    p = np.minimum((u01(c[0], c[1]) * float(npair)).astype(np.int64), npair - 1)
    j1 = p // (nc - 1)
    r = p - j1 * (nc - 1)
    j2 = r + (r >= j1)
    w1, w2 = de_partner(split, step, g, src, j1), de_partner(split, step, g, src, j2)
    n = de_gauss(gid, step, g, k0, k1)
    gamma = gamma0 * (1.0 + sigma * n)
    Q = X[i] + gamma[:, None] * (Xall[w2] - Xall[w1])
    return Q, src.astype(np.int32), i, gamma, n, w1, w2


def group_accept_np(split, kind, step, g, ngroups, gid_base, X, lnp, Q, lnp_new, logfac, naccept):
    """k_accept2 for group g of ngroups with the stretch (kind 0) or the DE (kind 1) stream; logfac None: 0."""
    ns = nslots(split, X.shape[0], ngroups, g)
    i = slot_walker(split, step, g, ngroups, gid_base, np.arange(ns))
    gid = (gid_base + i).astype(np.uint64)
    if kind == RB_MOVE_DE:
        r = philox4x32_10(*de_counter(gid, step, g, DE_ACCEPT), *de_keys(split.seed))
    else:
        r = philox4x32_10(*_counters(gid, step, g, True), split.seed & 0xFFFFFFFF, split.seed >> 32)
    with np.errstate(divide="ignore", invalid="ignore"):
        lnu = np.log(u01(r[0], r[1]))
        acc = ((0.0 if logfac is None else logfac) + lnp_new - lnp[i]) > lnu
    X[i[acc]] = Q[acc]
    lnp[i[acc]] = lnp_new[acc]
    naccept[i[acc]] += 1
    return acc, int(np.isnan(lnp_new).sum())


# ---- the move schedule ---------------------------------------------------------------------------------------------
def schedule_np(seed, step0, nsteps, weights):
    w = np.asarray(weights, dtype=np.float64)
    cum = np.cumsum(w)
    cum = cum / cum[-1]
    cum[-1] = 1.0
    st = np.uint64(step0) + np.arange(nsteps, dtype=np.uint64)
    z = np.zeros(st.shape, dtype=np.uint64)
    c = philox4x32_10(st & MASK, st >> np.uint64(32), z, z, (seed & 0xFFFFFFFF) ^ 0x4D4F5645,
                      ((seed >> 32) & 0xFFFFFFFF) ^ 0x53434844)
    u = u01(c[0], c[1])
    return np.minimum(np.searchsorted(cum, u, side="right"), w.size - 1).astype(np.int32)


class MovesNumpyEngine(NumpyEngine):
    """NumpyEngine with the DE propose and the k-group accept of CudaEngine."""

    def de_propose(self, split, step, group, gid_base, X, Xall, gamma0, sigma):
        Q, src = de_propose_np(split, step, group, gid_base, X.numpy(), Xall.numpy(), gamma0, sigma)[:2]
        return torch.from_numpy(Q), torch.from_numpy(src)

    def group_accept(self, split, kind, step, group, ngroups, gid_base, X, lnp, Q, lnp_new, logfac, naccept, counters):
        _, nn = group_accept_np(split, kind, step, group, ngroups, gid_base, X.numpy(), lnp.numpy(), Q.numpy(),
                                lnp_new.numpy(), None if logfac is None else logfac.numpy(), naccept.numpy())
        counters[0] += nn
