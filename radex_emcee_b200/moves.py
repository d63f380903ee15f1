"""Moves of the device-resident ensemble sampler, as emcee's ``EnsembleSampler(moves=...)`` takes them.

``StretchMove(a=2.0)`` is emcee's default move (the red/blue split of ``csrc/stretch.cuh``).  ``DEMove(sigma=1e-5,
gamma0=None)`` is emcee's differential-evolution move (ter Braak 2006, Nelson et al. 2013): three groups moved in turn,
q = s + gamma (c_j2 - c_j1) from two distinct walkers of the other groups, gamma = gamma0 (1 + sigma n), n ~ N(0, 1),
gamma0 = 2.38 / sqrt(2 ndim) by default.  A list of (move, weight) is a mixture: every step applies one move, drawn with
those probabilities, to the whole ensemble (``rb_move_schedule``)."""
from __future__ import annotations

import math

from . import _lib


class StretchMove:
    """emcee's ``StretchMove(a=2.0)``."""

    kind = _lib.RB_MOVE_STRETCH

    def __init__(self, a=2.0):
        self.a = float(a)
        if not self.a > 1.0:
            raise ValueError("StretchMove needs a > 1")

    def c_struct(self, weight):
        return _lib.rb_move(self.kind, 0, self.a, 0.0, 0.0, float(weight))

    def __repr__(self):
        return "StretchMove(a=%r)" % self.a


class DEMove:
    """emcee's ``DEMove(sigma=1e-5, gamma0=None)``; ``gamma0=None`` is 2.38 / sqrt(2 ndim)."""

    kind = _lib.RB_MOVE_DE

    def __init__(self, sigma=1e-5, gamma0=None):
        self.sigma = float(sigma)
        self.gamma0 = None if gamma0 is None else float(gamma0)
        if not (math.isfinite(self.sigma) and self.sigma >= 0.0):
            raise ValueError("DEMove needs a finite sigma >= 0")
        if self.gamma0 is not None and not (math.isfinite(self.gamma0) and self.gamma0 > 0.0):
            raise ValueError("DEMove needs a finite gamma0 > 0 (or None)")

    def gamma0_for(self, ndim):
        return 2.38 / math.sqrt(2.0 * ndim) if self.gamma0 is None else self.gamma0

    def c_struct(self, weight):
        return _lib.rb_move(self.kind, 0, 0.0, self.gamma0 or 0.0, self.sigma, float(weight))

    def __repr__(self):
        return "DEMove(sigma=%r, gamma0=%r)" % (self.sigma, self.gamma0)


def normalize_moves(moves):
    """emcee's three forms -- one move, a list of moves (equal weights), a list of (move, weight) -- as a list of
    (move, weight) with the weights as given (the schedule normalises them)."""
    if isinstance(moves, (StretchMove, DEMove)):
        pairs = [(moves, 1.0)]
    else:
        try:
            items = list(moves)
        except TypeError:
            raise ValueError("moves must be a move, a list of moves or a list of (move, weight)") from None
        if items and all(isinstance(m, (StretchMove, DEMove)) for m in items):
            pairs = [(m, 1.0) for m in items]
        else:
            pairs = []
            for it in items:
                if not (isinstance(it, (tuple, list)) and len(it) == 2 and isinstance(it[0], (StretchMove, DEMove))):
                    raise ValueError("unknown move %r: use StretchMove or DEMove, alone or as (move, weight)" % (it,))
                pairs.append((it[0], float(it[1])))
    if not 1 <= len(pairs) <= _lib.RB_MAX_MOVES:
        raise ValueError("between 1 and %d moves" % _lib.RB_MAX_MOVES)
    w = [p[1] for p in pairs]
    if not all(math.isfinite(x) and x >= 0.0 for x in w) or not sum(w) > 0.0:
        raise ValueError("move weights must be finite, >= 0 and not all 0")
    return pairs


def parse_moves(spec):
    """``["de:0.8", "stretch:0.2"]`` (the driver's ``--moves``) -> [(move, weight)]; a name without a weight gets 1."""
    out = []
    for item in spec:
        name, _, w = str(item).partition(":")
        name = name.strip().lower()
        if name == "stretch":
            mv = StretchMove()
        elif name == "de":
            mv = DEMove()
        else:
            raise ValueError("unknown move %r (stretch or de)" % name)
        out.append((mv, float(w) if w else 1.0))
    return normalize_moves(out)
