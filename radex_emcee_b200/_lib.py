"""ctypes binding of libradex_b200.so (include/radex_b200.h).  No CPU fallback: importing the
package without the built library, or creating a context without a B200, fails loudly."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libradex_b200.so")

RB_MAX_OBS = 16
RB_MAX_CHUNKS, RB_CHAIN_MAX_DIM, RB_CHAIN_MAX_COLS, RB_CHAIN_MAX_HIST = 64, 16, 32, 128
STOP_PYRADEX, STOP_RADEX = 0, 1
GEOM = {"sphere": 1, "lvg": 2, "slab": 3}
ST_T_RANGE, ST_N_RANGE, ST_MAXITER, ST_NONFINITE = 1, 2, 4, 8


class RadexB200Error(RuntimeError):
    pass


class rb_opts(C.Structure):
    _fields_ = [("stop_rule", C.c_int32), ("miniter", C.c_int32), ("maxiter", C.c_int32), ("kernel", C.c_int32),
                ("abs_tol", C.c_double), ("fk_epi", C.c_double), ("thc_epi", C.c_double),
                ("park_max", C.c_int32), ("spec_half", C.c_int32), ("lnprob_pipe_min", C.c_int64)]


class rb_obs(C.Structure):
    _fields_ = [("nobs", C.c_int32), ("jup", C.c_int32 * RB_MAX_OBS), ("flux", C.c_double * RB_MAX_OBS),
                ("eflux", C.c_double * RB_MAX_OBS)]


class rb_source(C.Structure):
    _fields_ = [("obs", rb_obs), ("bounds", C.c_double * 16), ("tbg", C.c_double), ("has_td", C.c_int32),
                ("reserved", C.c_int32), ("t_d", C.c_double)]


class rb_split(C.Structure):
    _fields_ = [("nwalkers", C.c_int64), ("walkers_per_source", C.c_int64), ("block", C.c_int64),
                ("randomize", C.c_int32), ("reserved", C.c_int32), ("seed", C.c_uint64)]


class rb_chain_view(C.Structure):
    _fields_ = [("chunk", C.c_void_p * RB_MAX_CHUNKS), ("steps", C.c_int64 * RB_MAX_CHUNKS), ("nchunks", C.c_int32),
                ("ndim", C.c_int32), ("nlocal", C.c_int64), ("gid_base", C.c_int64), ("walkers_per_source", C.c_int64),
                ("discard", C.c_int64), ("thin", C.c_int64)]


_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_lp = C.POINTER(C.c_int64)
_vp = C.c_void_p

# name -> (restype, argtypes); every symbol declared in include/radex_b200.h
SIGNATURES = {
    "rb_last_error": (C.c_char_p, []),
    "rb_default_opts": (None, [C.POINTER(rb_opts)]),
    "rb_device_count": (C.c_int, []),
    "rb_moldata_load": (C.c_int, [C.c_char_p, C.POINTER(_vp)]),
    "rb_moldata_free": (None, [_vp]),
    "rb_moldata_dims": (C.c_int, [_vp, _ip, _ip, _ip]),
    "rb_moldata_partners": (C.c_int, [_vp, _ip, _ip, _ip]),
    "rb_moldata_levels": (C.c_int, [_vp, _dp, _dp]),
    "rb_moldata_lines": (C.c_int, [_vp, _ip, _ip, _dp, _dp, _dp, _dp]),
    "rb_ctx_create": (C.c_int, [C.c_int, _vp, C.POINTER(_vp)]),
    "rb_ctx_destroy": (None, [_vp]),
    "rb_ctx_sync": (C.c_int, [_vp]),
    "rb_ctx_set_stream": (C.c_int, [_vp, _vp]),
    "rb_ctx_reset_stream": (C.c_int, [_vp]),
    "rb_solve_batch": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, C.c_double, C.c_double, C.c_int,
                                 C.POINTER(rb_opts), _vp, _vp, _vp, _vp, _vp, _vp]),
    "rb_solve_batch_dev": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, C.c_double, C.c_double, C.c_int,
                                     C.POINTER(rb_opts), _vp, _vp, _vp, _vp, _vp, _vp]),
    "rb_lnprob1": (C.c_int, [_vp, C.c_int64, _vp, C.POINTER(rb_obs), _vp, C.c_double, C.POINTER(rb_opts), _vp, _lp]),
    "rb_lnprob1_dev": (C.c_int, [_vp, C.c_int64, _vp, C.POINTER(rb_obs), _vp, C.c_double, C.POINTER(rb_opts), _vp, _vp]),
    "rb_lnprob2": (C.c_int, [_vp, C.c_int64, _vp, C.POINTER(rb_obs), _vp, C.c_int, C.c_double, C.c_double,
                             C.POINTER(rb_opts), _vp, _lp]),
    "rb_lnprob2_dev": (C.c_int, [_vp, C.c_int64, _vp, C.POINTER(rb_obs), _vp, C.c_int, C.c_double, C.c_double,
                                 C.POINTER(rb_opts), _vp, _vp]),
    "rb_stretch_propose_dev": (C.c_int, [_vp, C.c_int64, C.c_int32, _vp, C.c_int64, _vp, C.c_double, C.c_uint64,
                                         C.c_uint64, C.c_int32, C.c_int64, C.c_int64, _vp, _vp]),
    "rb_stretch_accept_dev": (C.c_int, [_vp, C.c_int64, C.c_int32, _vp, _vp, _vp, _vp, _vp, C.c_uint64, C.c_uint64,
                                        C.c_int32, C.c_int64, C.c_int64, _vp]),
    "rb_srcset_create": (C.c_int, [_vp, C.c_int32, C.c_int32, C.POINTER(rb_source), C.POINTER(_vp)]),
    "rb_srcset_destroy": (None, [_vp]),
    "rb_lnprob_src_dev": (C.c_int, [_vp, _vp, C.c_int64, _vp, _vp, C.POINTER(rb_opts), _vp, _vp]),
    "rb_stretch_pack_dev": (C.c_int, [_vp, C.POINTER(rb_split), C.c_uint64, C.c_int32, C.c_int64, C.c_int64, C.c_int32,
                                      _vp, _vp]),
    "rb_stretch_propose2_dev": (C.c_int, [_vp, C.POINTER(rb_split), C.c_uint64, C.c_int32, C.c_int64, C.c_int64,
                                          C.c_int32, _vp, _vp, C.c_double, _vp, _vp, _vp]),
    "rb_stretch_accept2_dev": (C.c_int, [_vp, C.POINTER(rb_split), C.c_uint64, C.c_int32, C.c_int64, C.c_int64,
                                         C.c_int32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rb_stretch_run_dev": (C.c_int, [_vp, _vp, C.POINTER(rb_split), C.c_double, C.c_uint64, C.c_int64,
                                     C.POINTER(rb_opts), _vp, _vp, _vp, _vp, C.c_int32, _vp, _vp]),
    "rb_ctx_counters": (C.c_int, [_vp, _lp, _lp]),
    "rb_ctx_cache_stats": (C.c_int, [_vp, _lp]),
    "rb_fp64_peak": (C.c_int, [_vp, _dp]),
    "rb_chain_hist_dev": (C.c_int, [_vp, C.POINTER(rb_chain_view), C.c_int32, C.c_int32, _ip, _ip, C.c_int32, C.c_int32,
                                    _vp, _vp, _vp]),
    "rb_chain_moments_dev": (C.c_int, [_vp, C.POINTER(rb_chain_view), _vp, _vp]),
    "rb_chain_acf_dev": (C.c_int, [_vp, C.POINTER(rb_chain_view), C.c_int32, _vp, _vp, C.c_int64, C.c_int64, _vp]),
}

_lib = None


def load():
    """dlopen the in-tree library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RadexB200Error(
                "libradex_b200.so is not built (%s). Run `python -m radex_emcee_b200.build` "
                "(needs nvcc); there is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise RadexB200Error("libradex_b200 error %d: %s" % (rc, load().rb_last_error().decode()))


def default_opts(**kw) -> rb_opts:
    o = rb_opts()
    load().rb_default_opts(C.byref(o))
    for k, v in kw.items():
        if v is not None:
            setattr(o, k, v)
    return o


def make_obs(jup, flux, eflux) -> rb_obs:
    jup = np.asarray(jup, dtype=np.int64).ravel()
    flux = np.asarray(flux, dtype=np.float64).ravel()
    eflux = np.asarray(eflux, dtype=np.float64).ravel()
    if not (jup.size == flux.size == eflux.size):
        raise ValueError("Jup, flux and eflux must have the same length")
    if not 1 <= jup.size <= RB_MAX_OBS:
        raise ValueError("between 1 and %d observed lines are supported" % RB_MAX_OBS)
    o = rb_obs()
    o.nobs = jup.size
    for i in range(jup.size):
        o.jup[i] = int(jup[i])
        o.flux[i] = float(flux[i])
        o.eflux[i] = float(eflux[i])
    return o


def make_source(ncomp, jup, flux, eflux, bounds, tbg, T_d=None) -> rb_source:
    b = np.ascontiguousarray(bounds, dtype=np.float64)
    if b.shape != (4 * ncomp, 2):
        raise ValueError("bounds must have shape (%d, 2)" % (4 * ncomp))
    s = rb_source()
    s.obs = make_obs(jup, flux, eflux)
    for i, v in enumerate(b.ravel()):
        s.bounds[i] = float(v)
    s.tbg = float(tbg)
    s.has_td = int(T_d is not None)
    s.t_d = float(T_d) if T_d is not None else 0.0
    return s


class SourceSet:
    """Device-resident table of fitted sources (rb_srcset): one row per source, same ncomp."""

    def __init__(self, ctx: "Context", ncomp: int, sources):
        L = load()
        self.ctx, self.ncomp, self.nsrc = ctx, int(ncomp), len(sources)
        arr = (rb_source * self.nsrc)(*sources)
        h = _vp()
        check(L.rb_srcset_create(ctx.handle, self.ncomp, self.nsrc, arr, C.byref(h)))
        self.handle = h

    def __del__(self):
        try:
            if self.handle:
                load().rb_srcset_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


def ptr(a):
    """void* of a C-contiguous numpy array (or None)."""
    if a is None:
        return None
    return a.ctypes.data_as(_vp)


class MolData:
    """Parsed LAMDA table (host side of rb_mol)."""

    def __init__(self, path):
        L = load()
        h = _vp()
        check(L.rb_moldata_load(os.fsencode(path), C.byref(h)))
        self.handle = h
        self.path = path
        nlev, nline, npart = C.c_int32(), C.c_int32(), C.c_int32()
        check(L.rb_moldata_dims(h, C.byref(nlev), C.byref(nline), C.byref(npart)))
        self.nlev, self.nline, self.npart = nlev.value, nline.value, npart.value
        self.partner_id = np.zeros(self.npart, np.int32)
        self.ncoll = np.zeros(self.npart, np.int32)
        self.ntemp = np.zeros(self.npart, np.int32)
        check(L.rb_moldata_partners(h, self.partner_id.ctypes.data_as(_ip), self.ncoll.ctypes.data_as(_ip),
                                    self.ntemp.ctypes.data_as(_ip)))
        self.eterm = np.zeros(self.nlev)
        self.gstat = np.zeros(self.nlev)
        check(L.rb_moldata_levels(h, self.eterm.ctypes.data_as(_dp), self.gstat.ctypes.data_as(_dp)))
        self.iupp = np.zeros(self.nline, np.int32)
        self.ilow = np.zeros(self.nline, np.int32)
        self.aeinst, self.spfreq, self.eup, self.xnu = (np.zeros(self.nline) for _ in range(4))
        check(L.rb_moldata_lines(h, self.iupp.ctypes.data_as(_ip), self.ilow.ctypes.data_as(_ip),
                                 self.aeinst.ctypes.data_as(_dp), self.spfreq.ctypes.data_as(_dp),
                                 self.eup.ctypes.data_as(_dp), self.xnu.ctypes.data_as(_dp)))

    def __del__(self):
        try:
            if self.handle:
                load().rb_moldata_free(self.handle)
                self.handle = None
        except Exception:
            pass


class Context:
    """One GPU: device-resident tables + stream (rb_ctx)."""

    def __init__(self, mol: MolData, device: int = 0):
        L = load()
        h = _vp()
        check(L.rb_ctx_create(int(device), mol.handle, C.byref(h)))
        self.handle = h
        self.mol = mol
        self.device = int(device)

    def __del__(self):
        try:
            if self.handle:
                load().rb_ctx_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def sync(self):
        check(load().rb_ctx_sync(self.handle))

    def set_stream(self, stream_ptr):
        """stream_ptr: cudaStream_t handle as int (0 = legacy default stream, PyTorch's default)."""
        check(load().rb_ctx_set_stream(self.handle, _vp(int(stream_ptr))))

    def reset_stream(self):
        check(load().rb_ctx_reset_stream(self.handle))

    def fp64_peak_tflops(self):
        v = C.c_double(0.0)
        check(load().rb_fp64_peak(self.handle, C.byref(v)))
        return v.value

    def cache_stats(self):
        """(cached iterations, captures, invalidations) of the last solve/lnprob call."""
        a = (C.c_int64 * 3)()
        check(load().rb_ctx_cache_stats(self.handle, a))
        return tuple(int(v) for v in a)

    def counters(self):
        it, ln = C.c_int64(), C.c_int64()
        check(load().rb_ctx_counters(self.handle, C.byref(it), C.byref(ln)))
        return it.value, ln.value
