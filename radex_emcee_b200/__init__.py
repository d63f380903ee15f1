"""radex_emcee_b200: B200-native replacement for the hot path of yangcht/radex_emcee.

Public surface (mirrors the reference's):
  Radex                       pyradex.Radex-compatible batched solver      (radex.py)
  emcee_radex, emcee_radex_2comp   lnprob/lnprior/lnlike/model_lvg, vectorised  (emcee_radex*.py)
  StretchSampler              device-resident ensemble sampler (sampler.py)
  StretchMove, DEMove         its moves, alone or mixed (emcee's moves=)   (moves.py)
  read_data, get_source       flux table readers                           (data.py)
The CUDA library (libradex_b200.so) must be built; there is no CPU fallback.
"""
from . import _lib
from ._lib import RadexB200Error, STOP_PYRADEX, STOP_RADEX, default_opts
from .data import get_source, read_data
from .radex import Radex

__all__ = ["Radex", "RadexB200Error", "STOP_PYRADEX", "STOP_RADEX", "default_opts", "read_data", "get_source"]
