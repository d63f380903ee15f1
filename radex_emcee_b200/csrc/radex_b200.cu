// libradex_b200 -- CUDA kernels (sm_100a) and C ABI for the RADEX escape-probability hot path.
//
// Reference path being replaced (all relative to /root/reference):
//   emcee/emcee_radex.py:120-181, emcee/emcee_radex_2comp.py:122-244   lnprob / lnprior / lnlike / model_lvg
//   emcee/pyradex/core.py:388-438, 856-925, 986-1003                   set_params / run_radex / brightness
//   emcee/pyradex/radex/radex.so  readdata@0x1cf90 backrad@0x1be30 matrix@0x17f70 escprob@0xa9c0
//                                 lubksb@0x17cb0 -> sgeir@0x16d50 -> sgefa@0xf3d0 / sgesl@0xdb70
//
// One warp (or half-warp) owns one model (walker component).  Small batches run as ONE launch in which nothing but
// the walker parameters and the requested outputs touches HBM; batches >= RB_SCHED_MIN run as ordered launches that
// park each model's state (and the capture of its frozen top) in HBM between them.  See DESIGN.md for the layout.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

#include "internal.h"

// ------------------------------------------------------------------------------------------------
// constants: exactly the values in the reference binary's constant pool (SURVEY.md 2.2)
// ------------------------------------------------------------------------------------------------
#define RB_FK 1.4387809925261357        // h c / k  (radex.inc)
#define RB_THC 3.972907393443411e-16    // 2 h c    (radex.inc)
#define RB_PI_TRUNC 3.14159265          // radex.inc's pi
#define RB_MINPOP 1.0e-20
#define RB_F32(x) ((double)(x##f))      // single-precision Fortran literal promoted to double
#define RB_FGAUS (RB_F32(1.0645) * 8.0 * RB_PI_TRUNC)

#define CUDA_TRY(expr)                                                                          \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) {                                                                    \
      rb_set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                         \
      return RB_ERR_CUDA;                                                                       \
    }                                                                                           \
  } while (0)

// ------------------------------------------------------------------------------------------------
// device-resident molecular table (SoA); passed to kernels by value
// ------------------------------------------------------------------------------------------------
struct MolDev {
  int nlev, nline, npart;
  int sorted_levels;                      // eterm strictly increasing (true for LAMDA files)
  const double *eterm, *gstat;            // [nlev]
  const int *iupp, *ilow;                 // [nline] 0-based
  const double *aeinst, *xnu;             // [nline]
  const int *lev_ptr;                     // [nlev+1] CSR: lines incident on each level, in line order
  const int *lev_line;                    // [2*nline] line index, bit 30 set when the level is the upper one
  int part_id[RB_MAXPART], ntemp[RB_MAXPART], ncoll[RB_MAXPART];
  double ln_frac[RB_MAXPART];             // lnprob: share of the walker's n(H2) that partner p receives (0 = no usable partner)
  const double *temps[RB_MAXPART];        // [ntemp]
  const int *lcu[RB_MAXPART], *lcl[RB_MAXPART];  // [ncoll] 0-based
  const double *rates_tc[RB_MAXPART];     // [ntemp][ncoll]
};

struct SolveCfg {
  double *bslab;   // v2: per-warp global copies of the collisional matrix (L2-resident)
  double deltav_cms, tbg;
  int method, stop_rule, miniter, maxiter;
  double abs_tol, fk_epi, thc_epi;
  int cache;                    // v2: frozen-top caching enabled (rb_opts.kernel != 2)
  int sched;                    // v2: launch scheduling allowed (rb_opts.kernel == 0 or 4)
  int small;                    // v2: cached engines as kernels of their own (lvg_small.cuh; kernel == 0)
  int park_max;                 // v2: largest lead block (in panels) handed to them: 4 (half-warp engines only) or 7;
                                //     0 = chosen from the batch size (rb_opts.park_max)
  long long lnprob_pipe_min;    // walkers per call from which lnprob runs as a pipeline (rb_opts.lnprob_pipe_min)
  unsigned long long *stats;    // v2: [0] cached iterations, [1] captures, [2] invalidations
};

struct rb_ctx {
  int device = 0;
  int sm_count = 0;
  int smem_optin = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  MolDev mol{};
  std::vector<void *> owned;              // device allocations of the tables
  // grow-only scratch for the host-pointer entry points
  void *scratch = nullptr;
  size_t scratch_bytes = 0;
  unsigned long long *counters = nullptr; // [0] work queue head, [1] total iterations, [2] solves
  double *bslab = nullptr;                // v2: sm_count x V2_WARPS x GSLAB doubles
  void *sched_buf = nullptr;              // v2 scheduling: parked state, keys, order (grow-only)
  size_t sched_bytes = 0;
  unsigned long long *sched_small = nullptr;   // 96 words: histogram, offsets, cursors, parked count
  cudaStream_t side[6] = {};              // launch B and the five cached-engine launches run side by side (independent models)
  cudaEvent_t ev_sorted = nullptr, ev_side[6] = {};
  cudaStream_t copy_stream = nullptr;     // host entry: results of one chunk travel while the next is solved
  std::vector<cudaEvent_t> chunk_done;
  void *ln_buf = nullptr;                 // lnprob pipeline: model parameters, observed-line brightness, status (grow-only)
  size_t ln_bytes = 0;
  rb_source *src_one = nullptr;           // device copy of the source of the last rb_lnprob1/2 call ...
  rb_source src_one_host{};               // ... and what it holds (no transfer while the caller keeps passing the same source)
  bool src_one_valid = false;
  bool ln_partners_ok = false;            // lnprob: the file has H2, or p-H2 / o-H2, as a collision partner
  bool engines_fit = false;               // v2: the lead lines of every cached engine lie in its lead trips (v2s::lead_lines_fit)
  void *samp_buf = nullptr;               // rb_stretch_run_dev: complementary half, proposals, their lnprob, step counter (grow-only)
  size_t samp_bytes = 0;
  cudaEvent_t ev_samp = nullptr;
  cudaGraphExec_t samp_graph[RB_MAX_MOVES] = {};   // one step of move m of the list, captured for the arguments in samp_key[m]
  std::vector<unsigned char> samp_key[RB_MAX_MOVES];
  void *cs_buf = nullptr;                 // rb_chain_acf_dev: per-block partial sums (grow-only)
  size_t cs_bytes = 0;
  long long launches = 0;
  long long last_total_iters = 0;
};

// ------------------------------------------------------------------------------------------------
// escape probability, three geometries (radex.so@0xa9c0; oracle/radex_oracle.c ro_escprob)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double rb_escprob(double tau, int method) {
  const double taur = tau * 0.5;
  double beta;
  if (method == RB_GEOM_LVG) {
    const double at = fabs(taur);
    if (at < RB_F32(0.01)) {
      beta = 1.0;
    } else if (at < 7.0) {
      beta = 2.0 * (1.0 - exp(-RB_F32(2.34) * taur)) / (RB_F32(4.68) * taur);
    } else {
      beta = 2.0 / (taur * 4.0 * sqrt(log(taur / sqrt(RB_PI_TRUNC))));
    }
  } else if (method == RB_GEOM_SPHERE) {
    const double at = fabs(taur);
    if (at < RB_F32(0.1)) {
      beta = 1.0 - 0.75 * taur + (taur * taur) / 2.5 - (taur * taur * taur) / 6.0 +
             (taur * taur * taur * taur) / 17.5;
    } else if (at > 50.0) {
      beta = 0.75 / taur;
    } else {
      beta = 0.75 / taur *
             (1.0 - 1.0 / (2.0 * (taur * taur)) + (1.0 / taur + 1.0 / (2.0 * (taur * taur))) * exp(-2.0 * taur));
    }
  } else {
    const double t3 = fabs(3.0 * tau);
    if (t3 < RB_F32(0.1)) {
      beta = 1.0 - 1.5 * (tau + tau * tau);
    } else if (t3 > 50.0) {
      beta = 1.0 / (3.0 * tau);
    } else {
      beta = (1.0 - exp(-3.0 * tau)) / (3.0 * tau);
    }
  }
  return beta;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ int warp_sum_int(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------------
// v1 solver: one warp per model, rate matrix in shared memory, partial-pivot LU exactly as the
// reference build does it (reduced nlev x nlev system, last equation replaced by conservation).
// ------------------------------------------------------------------------------------------------
struct WarpMem {             // carved out of dynamic shared memory, one per warp
  double *A;                 // [nlev*nlev] column-major work matrix (also holds crate[i*nlev+j] in the prologue)
  double *B;                 // [nlev*nlev] column-major collisional part incl. -eps (constant over iterations)
  double *ctot, *xpop, *xold, *rhs;  // [nlev]
  double *tex, *taul, *backi, *dn, *up, *upx;  // [nline]
};

__host__ __device__ inline size_t v1_warp_doubles(int nlev, int nline) {
  return (size_t)2 * nlev * nlev + 4 * (size_t)nlev + 6 * (size_t)nline;
}

__device__ __forceinline__ WarpMem carve(double *base, int nlev, int nline) {
  WarpMem w;
  w.A = base;
  w.B = w.A + nlev * nlev;
  w.ctot = w.B + nlev * nlev;
  w.xpop = w.ctot + nlev;
  w.xold = w.xpop + nlev;
  w.rhs = w.xold + nlev;
  w.tex = w.rhs + nlev;
  w.taul = w.tex + nline;
  w.backi = w.taul + nline;
  w.dn = w.backi + nline;
  w.up = w.dn + nline;
  w.upx = w.up + nline;
  return w;
}

// collision rates at tkin: clamped linear interpolation, partner mix, detailed balance, ctot
// (readdata, radex.so@0x1cf90; oracle ro_set_physics).  Result: crate in w.A (row-major
// crate[i*nlev+j] = rate i->j), ctot in w.ctot, returns totdens.
__device__ double v1_rates(const MolDev &mol, const WarpMem &w, int lane, double tkin, const double *dens) {
  const int nl = mol.nlev;
  for (int e = lane; e < nl * nl; e += 32) w.A[e] = 0.0;
  __syncwarp();
  double totdens = 0.0;
  for (int p = 0; p < mol.npart; ++p) {
    const double d = dens[p];
    totdens += d;
    const double *T = mol.temps[p];
    const int nt = mol.ntemp[p];
    int t0 = 0;
    double fint = 0.0;
    int mode;  // 0 low clamp, 1 high clamp, 2 interpolate
    if (tkin <= T[0]) {
      mode = 0;
    } else if (tkin >= T[nt - 1]) {
      mode = 1;
    } else {
      mode = 2;
      for (int t = 0; t < nt - 1; ++t)
        if (tkin > T[t] && tkin <= T[t + 1]) {
          t0 = t;
          fint = (tkin - T[t]) / (T[t + 1] - T[t]);
          break;
        }
    }
    const double *R = mol.rates_tc[p];
    const int nc = mol.ncoll[p];
    for (int c = lane; c < nc; c += 32) {
      double v;
      if (mode == 0) {
        v = __ldg(R + c);
      } else if (mode == 1) {
        v = __ldg(R + (size_t)(nt - 1) * nc + c);
      } else {
        const double r0 = __ldg(R + (size_t)t0 * nc + c), r1 = __ldg(R + (size_t)(t0 + 1) * nc + c);
        v = r0 + fint * (r1 - r0);
        if (v < 0.0) v = r0;
      }
      const int iu = mol.lcu[p][c], il = mol.lcl[p][c];
      w.A[iu * nl + il] += d * v;
    }
    __syncwarp();
  }
  for (int e = lane; e < nl * nl; e += 32) {
    const int iu = e / nl, il = e - iu * nl;
    const double ediff = mol.eterm[iu] - mol.eterm[il];
    if (ediff > 0.0) {
      const double x = RB_FK * ediff / tkin;
      w.A[il * nl + iu] = (x >= 160.0) ? 0.0 : mol.gstat[iu] / mol.gstat[il] * exp(-x) * w.A[iu * nl + il];
    }
  }
  __syncwarp();
  for (int i = lane; i < nl; i += 32) {
    double t = 0.0;
    for (int j = 0; j < nl; ++j) t += w.A[i * nl + j];
    w.ctot[i] = t;
  }
  __syncwarp();
  return totdens;
}

// LU with partial pivoting + solve on the nl x nl column-major matrix in w.A, rhs in w.rhs
// (sgefa/sgesl; oracle ro_gefa/ro_gesl).  Lanes run down the rows of a column.
__device__ void v1_lu_solve(const WarpMem &w, int nl, int lane) {
  double *A = w.A;
  double *b = w.rhs;
  for (int k = 0; k < nl - 1; ++k) {
    // pivot search: first index of max |A[i,k]|, i >= k
    double best = -1.0;
    int bi = k;
    for (int i = k + lane; i < nl; i += 32) {
      const double v = fabs(A[i + k * nl]);
      if (v > best) {
        best = v;
        bi = i;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > best || (ov == best && oi < bi)) {
        best = ov;
        bi = oi;
      }
    }
    const int l = bi;
    if (best == 0.0) continue;  // column already triangularised (sgefa's info path)
    // row interchange across all columns k..nl-1 and in the rhs (sgesl applies it to b)
    if (l != k) {
      for (int j = k + lane; j < nl; j += 32) {
        const double t = A[l + j * nl];
        A[l + j * nl] = A[k + j * nl];
        A[k + j * nl] = t;
      }
      if (lane == 0) {
        const double t = b[l];
        b[l] = b[k];
        b[k] = t;
      }
      __syncwarp();
    }
    const double piv = A[k + k * nl];
    const double t = -1.0 / piv;
    // multipliers for my rows (kept in registers), two passes cover nl <= 64
    const int i0 = k + 1 + lane, i1 = i0 + 32;
    double m0 = 0.0, m1 = 0.0;
    if (i0 < nl) {
      m0 = A[i0 + k * nl] * t;
      A[i0 + k * nl] = m0;
    }
    if (i1 < nl) {
      m1 = A[i1 + k * nl] * t;
      A[i1 + k * nl] = m1;
    }
    for (int j = k + 1; j < nl; ++j) {
      const double tj = A[k + j * nl];
      if (i0 < nl) A[i0 + j * nl] = fma(tj, m0, A[i0 + j * nl]);
      if (i1 < nl) A[i1 + j * nl] = fma(tj, m1, A[i1 + j * nl]);
    }
    // forward elimination of the rhs with the same multipliers
    const double bk = b[k];
    if (i0 < nl) b[i0] = fma(bk, m0, b[i0]);
    if (i1 < nl) b[i1] = fma(bk, m1, b[i1]);
    __syncwarp();
  }
  for (int k = nl - 1; k >= 0; --k) {
    const double xk = b[k] / A[k + k * nl];
    __syncwarp();
    if (lane == 0) b[k] = xk;
    for (int i = lane; i < k; i += 32) b[i] = fma(-xk, A[i + k * nl], b[i]);
    __syncwarp();
  }
}

// One full solve.  On return w.xpop/tex/taul/backi hold the state pyradex would read back.
// Returns the pyradex iteration counter; *status gets the rb_model_status bits.
__device__ int v1_solve(const MolDev &mol, const WarpMem &w, int lane, double tkin, const double *dens, double cdmol,
                        const double tbg, const SolveCfg &cfg, int *status) {
  const int nl = mol.nlev, nn = mol.nline;
  int st = 0;
  if (!(tkin > 0.0 && tkin <= 1.0e4)) st |= RB_ST_T_RANGE;
  if (!(cdmol >= 1.0e5 && cdmol <= 1.0e25)) st |= RB_ST_N_RANGE;
  if (st) {
    *status = st;
    return 0;
  }
  const double totdens = v1_rates(mol, w, lane, tkin, dens);
  const double eps_td = 1.0e-30 * totdens;
  // constant part of the rate matrix, column-major: B(i,j) = -eps - crate(j,i); the diagonal is rebuilt
  for (int e = lane; e < nl * nl; e += 32) {
    const int j = e / nl, i = e - j * nl;
    w.B[e] = (i == j) ? 0.0 : (-eps_td - w.A[j * nl + i]);
  }
  // background (backrad, tbg > 0 branch, radex.so@0x1be30): backi = totalb, trj = tbg
  for (int l = lane; l < nn; l += 32) {
    const double xnu = mol.xnu[l];
    const double hnu = RB_FK * xnu / tbg;
    w.backi[l] = (hnu >= 160.0) ? 1.0e-30 : RB_THC * (xnu * xnu * xnu) / (exp(hnu) - 1.0);
    w.tex[l] = 0.0;
    w.taul[l] = 0.0;
  }
  for (int i = lane; i < nl; i += 32) w.xpop[i] = 0.0;
  __syncwarp();

  const double cddv = cdmol / cfg.deltav_cms;
  int it = 0;
  int hit_max = 0;
  for (;;) {
    if (it >= cfg.maxiter) {
      hit_max = 1;
      break;
    }
    // ---- radiative rates per line ----------------------------------------------------------
    int nthick = 0;
    for (int l = lane; l < nn; l += 32) {
      const int m = mol.iupp[l], n = mol.ilow[l];
      const double a = mol.aeinst[l], gm = mol.gstat[m], gn = mol.gstat[n];
      const double xnu = mol.xnu[l];
      double beta, exr;
      if (it == 0) {
        const double etr = RB_FK * xnu / tbg;
        exr = (etr >= 160.0) ? 0.0 : 1.0 / (exp(etr) - 1.0);
        beta = 1.0;
      } else {
        const double xt = xnu * xnu * xnu;
        const double tau = cddv * (w.xpop[n] * gm / gn - w.xpop[m]) / (RB_FGAUS * xt / a);
        w.taul[l] = tau;
        if (tau > 1.0e-2) ++nthick;
        beta = rb_escprob(tau, cfg.method);
        exr = w.backi[l] * beta / (RB_THC * xt);
      }
      w.dn[l] = a * (beta + exr);
      w.up[l] = a * (gm * exr / gn);
      w.upx[l] = a * (gm / gn) * exr;
    }
    nthick = warp_sum_int(nthick);
    // ---- assemble: A = B, then diagonal and the line entries --------------------------------
    for (int e = lane; e < nl * nl; e += 32) w.A[e] = w.B[e];
    __syncwarp();
    for (int i = lane; i < nl; i += 32) {
      double s = -eps_td;
      for (int q = mol.lev_ptr[i]; q < mol.lev_ptr[i + 1]; ++q) {
        const int code = mol.lev_line[q];
        const int l = code & 0x3fffffff;
        s += (code & 0x40000000) ? w.dn[l] : w.up[l];
      }
      w.A[i + i * nl] = s + w.ctot[i];
    }
    for (int l = lane; l < nn; l += 32) {
      const int m = mol.iupp[l], n = mol.ilow[l];
      w.A[m + n * nl] -= w.upx[l];
      w.A[n + m * nl] -= w.dn[l];
    }
    __syncwarp();
    // reduced system of this build's lubksb: last equation := conservation, rhs = e_last
    for (int j = lane; j < nl; j += 32) {
      w.A[(nl - 1) + j * nl] = 1.0;
      w.rhs[j] = (j == nl - 1) ? 1.0 : 0.0;
    }
    __syncwarp();
    v1_lu_solve(w, nl, lane);
    // ---- populations ------------------------------------------------------------------------
    double part = 0.0;
    for (int i = lane; i < nl; i += 32) part += w.rhs[i];
    const double total = warp_sum(part);
    for (int i = lane; i < nl; i += 32) {
      double xo = fmax(RB_MINPOP, w.xpop[i]);
      const double xn = fmax(RB_MINPOP, w.rhs[i] / total);
      if (it == 0) xo = xn;
      w.xold[i] = xo;
      w.rhs[i] = xn;  // un-relaxed new populations
    }
    __syncwarp();
    // ---- excitation temperatures, optical depths ----------------------------------------------
    double tsum = 0.0;
    for (int l = lane; l < nn; l += 32) {
      const int m = mol.iupp[l], n = mol.ilow[l];
      const double gm = mol.gstat[m], gn = mol.gstat[n];
      const double xnu = mol.xnu[l];
      const double xm = w.rhs[m], xn = w.rhs[n];
      if (it == 0) {
        w.tex[l] = (xn <= RB_MINPOP || xm <= RB_MINPOP) ? w.backi[l] : RB_FK * xnu / log(xn * gm / (xm * gn));
      } else {
        const double told = w.tex[l];
        const double thistex =
            (xn <= RB_MINPOP || xm <= RB_MINPOP) ? told : RB_FK * xnu / log(xn * gm / (xm * gn));
        if (w.taul[l] > RB_F32(0.01)) tsum += fabs((thistex - told) / thistex);
        w.tex[l] = 0.5 * (thistex + told);
        w.taul[l] = cddv * (xn * gm / gn - xm) / (RB_FGAUS * (xnu * xnu * xnu) / mol.aeinst[l]);
      }
    }
    tsum = warp_sum(tsum);
    int conv = 0;
    if (it >= 10) {  // miniter of radex.inc
      if (nthick == 0) conv = 1;
      else if (tsum / nthick < RB_F32(1.0e-6)) conv = 1;
    }
    // ---- under-relaxation + pyradex's stop test ------------------------------------------------
    double diff = 0.0;
    for (int i = lane; i < nl; i += 32) {
      const double prev = w.xpop[i];
      const double xr = RB_F32(0.3) * w.rhs[i] + RB_F32(0.7) * w.xold[i];
      w.xpop[i] = xr;
      diff += fabs(prev - xr);
    }
    diff = warp_sum(diff);
    __syncwarp();
    if (cfg.stop_rule == RB_STOP_RADEX) {
      if (conv) break;
    } else if (diff < cfg.abs_tol && it > cfg.miniter) {
      break;
    }
    ++it;
  }
  if (hit_max) st |= RB_ST_MAXITER;
  *status = st;
  return it;
}

// source_line_surfbrightness for line l (core.py:986-1003, base_class.py:275-277): no guards
__device__ __forceinline__ double rb_surf(const MolDev &mol, const WarpMem &w, int l, const SolveCfg &cfg) {
  const double xnu = mol.xnu[l];
  const double ftau = exp(-w.taul[l]);
  const double earg = cfg.fk_epi * xnu / w.tex[l];
  const double bnutex = cfg.thc_epi * (xnu * xnu * xnu) / (exp(earg) - 1.0);
  const double toti = w.backi[l] * ftau + bnutex * (1.0 - ftau);
  return toti - w.backi[l];
}

#include "lvg_v2.cuh"
#include "lvg_small.cuh"

struct SolveIO {
  long long n;
  const double *tkin, *dens, *cdmol;
  double *xpop, *tex, *tau, *surf;
  int *niter, *status;
  unsigned long long *counters;
  // v2 two-launch scheduling (lvg_v2.cuh): 0 single launch; 1 = launch A (run to the engine choice, park);
  // 2 = launch B (resume the parked models in the order given)
  int sched;
  double *state;                       // n x v2::STATE_STRIDE
  int *keys;                           // n: Kp wanted by a parked model, -1 = finished in launch A
  const int *order;                    // launch B: model index of queue position q
  const unsigned long long *n_parked;  // launch B: number of parked models (device)
  // half-warp engine (lvg_small.cuh): launch B parks the captures of small-lead models in ext, k_lvg_small runs
  // them and appends the ones whose frozen lines turn thick to order_c for launch C (sched = 4)
  // observed-line mode (lnprob pipeline): only the brightness of nobs lines is written, obs_surf[n][RB_MAX_OBS]
  double *obs_surf;
  int nobs;
  int obs_line[RB_MAX_OBS];
  double *ext;                         // parked captures: v2::ext_size(n) doubles per cacheable model, at ext + ext_off[model]
  long long *ext_off;
  long long ext_cap;                   // doubles in ext
  unsigned long long *sched_small;     // [16+k] first queue position of key k, [48] parked, [49] models for launch C
  int *order_c;
  int queue;                           // work-queue head of this launch: counters[queue] (0, or 8.. when launches overlap)
};

__global__ void __launch_bounds__(256) k_lvg_solve_v1(MolDev mol, SolveCfg cfg, SolveIO io) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int nl = mol.nlev, nn = mol.nline;
  const WarpMem w = carve(smem + (size_t)wib * v1_warp_doubles(nl, nn), nl, nn);
  unsigned long long iters = 0;
  for (;;) {
    unsigned long long idx = 0;
    if (lane == 0) idx = atomicAdd(&io.counters[0], 1ULL);
    idx = __shfl_sync(0xffffffffu, idx, 0);
    if ((long long)idx >= io.n) break;
    double dens[RB_MAXPART];
    for (int p = 0; p < mol.npart; ++p) dens[p] = io.dens[idx * mol.npart + p];
    int st = 0;
    const int it = v1_solve(mol, w, lane, io.tkin[idx], dens, io.cdmol[idx], cfg.tbg, cfg, &st);
    const bool bad = (st & (RB_ST_T_RANGE | RB_ST_N_RANGE)) != 0;
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    int nonfinite = 0;
    for (int l = lane; l < nn; l += 32) {
      const double s = bad ? qnan : rb_surf(mol, w, l, cfg);
      if (!bad && !isfinite(s)) nonfinite = 1;
      if (io.surf) io.surf[idx * nn + l] = s;
      if (io.tex) io.tex[idx * nn + l] = bad ? qnan : w.tex[l];
      if (io.tau) io.tau[idx * nn + l] = bad ? qnan : w.taul[l];
    }
    if (io.xpop)
      for (int i = lane; i < nl; i += 32) io.xpop[idx * nl + i] = bad ? qnan : w.xpop[i];
    nonfinite = __any_sync(0xffffffffu, nonfinite);
    if (nonfinite) st |= RB_ST_NONFINITE;
    if (lane == 0) {
      if (io.niter) io.niter[idx] = it;
      if (io.status) io.status[idx] = st;
    }
    // pyradex calls matrix() for it = 0..it inclusive unless it stopped at maxiter
    iters += bad ? 0 : (unsigned long long)((st & RB_ST_MAXITER) ? it : it + 1);
    __syncwarp();
  }
  if (lane == 0 && iters) {
    atomicAdd(&io.counters[1], iters);
  }
}

// ------------------------------------------------------------------------------------------------
// fused lnprob kernels: prior -> (1 or 2) solves -> line fluxes -> chi^2
// ------------------------------------------------------------------------------------------------
struct LnprobIO {
  long long n;
  const double *P;        // n x (4*NCOMP)
  double *lnp;            // n
  const rb_source *srcs;  // device table: observed SLED, bounds, tbg, T_d per fitted source
  const int *src_id;      // n: row of each walker, or nullptr = row 0
  unsigned long long *counters;
};

__device__ __forceinline__ double neg_inf() { return __longlong_as_double(0xfff0000000000000LL); }

// lnprior, one component (emcee/emcee_radex.py:169-175)
__device__ double lnprior1(const double *p, const double *b) {
  for (int i = 0; i < 4; ++i)
    if (p[i] > b[2 * i + 1] || p[i] < b[2 * i]) return neg_inf();
  const double d = p[2] - p[0];
  if (d >= 17.5 || d <= 10.0) return neg_inf();
  return 0.0;
}

// lnprior, two components (emcee/emcee_radex_2comp.py:199-234)
__device__ double lnprior2(const double *p, const double *b, int has_td, double t_d) {
  for (int i = 0; i < 8; ++i)
    if (p[i] > b[2 * i + 1] || p[i] < b[2 * i]) return neg_inf();
  if (p[5] <= p[1]) return neg_inf();
  const double d1 = p[2] - p[0], d2 = p[6] - p[4];
  if (d1 >= 18.0 || d1 <= 9.0 || d2 >= 18.0 || d2 <= 9.0) return neg_inf();
  if (p[3] < p[7]) return neg_inf();
  double logp = 0.0;
  for (int i = 0; i < 8; ++i) {
    if (i == 1 && has_td) {
      const double tk = pow(10.0, p[i]);
      if (t_d <= 0.0) return neg_inf();
      const double sigma = 1.0 * t_d;
      const double z = (tk - t_d) / sigma;
      logp += (-0.5 * (z * z) - log(sigma * sqrt(2.0 * 3.141592653589793)));
    } else {
      logp += -(b[2 * i + 1] - b[2 * i]);
    }
  }
  return logp;
}

// lnlike (emcee_radex.py:132-167 / emcee_radex_2comp.py:169-196) by one warp: lane i < nobs holds the model flux of
// observed line i.  Returns lp + ll, or -inf wherever the reference does.
__device__ __forceinline__ double lnlike_warp(const rb_source &S, const double model, const double lp, const int lane) {
  int bad = 0;
  double r2 = 0.0, le = 0.0;
  if (lane < S.obs.nobs) {
    const double f = S.obs.flux[lane];
    const double e = fmax(fabs(S.obs.eflux[lane]), 1.0e-12);
    if (!isfinite(f) || !isfinite(model) || !isfinite(e)) {
      bad = 1;
    } else {
      const double r = (f - model) / e;
      const double max_safe = 1.3407807929942596e+153;  // sqrt(DBL_MAX)/10
      if (!isfinite(r) || fabs(r) > max_safe) bad = 1;
      r2 = r * r;
      le = log(e);
    }
  }
  bad = __any_sync(0xffffffffu, bad);
  const double chi2 = warp_sum(r2), logterm = 2.0 * warp_sum(le);
  if (bad) return neg_inf();
  const double ll = -0.5 * (chi2 + logterm);
  return isfinite(ll) ? lp + ll : neg_inf();
}

// collider densities of one walker component: total n(H2) split as the drivers do (opr = 3, emcee_radex.py:95-96)
// through the per-partner fractions worked out on the host (MolDev::ln_frac, see lnprob_partner_fractions)
__device__ __forceinline__ void lnprob_dens(const MolDev &mol, const double dens_tot, double *dens) {
#pragma unroll
  for (int q = 0; q < RB_MAXPART; ++q) dens[q] = (q < mol.npart) ? mol.ln_frac[q] * dens_tot : 0.0;
}

template <int NCOMP>
__global__ void __launch_bounds__(256) k_lnprob_v1(MolDev mol, SolveCfg cfg, LnprobIO io) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int nl = mol.nlev, nn = mol.nline;
  const WarpMem w = carve(smem + (size_t)wib * v1_warp_doubles(nl, nn), nl, nn);
  constexpr int ND = 4 * NCOMP;
  unsigned long long iters = 0, solves = 0;
  for (;;) {
    unsigned long long idx = 0;
    if (lane == 0) idx = atomicAdd(&io.counters[0], 1ULL);
    idx = __shfl_sync(0xffffffffu, idx, 0);
    if ((long long)idx >= io.n) break;
    const rb_source &S = io.srcs[io.src_id ? io.src_id[idx] : 0];
    double p[ND];
#pragma unroll
    for (int i = 0; i < ND; ++i) p[i] = io.P[idx * ND + i];
    const double lp = (NCOMP == 1) ? lnprior1(p, S.bounds) : lnprior2(p, S.bounds, S.has_td, S.t_d);
    double result = neg_inf();
    if (isfinite(lp)) {  // prior short-circuit: no solve (emcee_radex.py:178-180)
      double model = 0.0;  // lane i < nobs holds the model flux of observed line i
      bool value_error = false;
#pragma unroll
      for (int c = 0; c < NCOMP; ++c) {
        if (value_error) break;
        double dens[RB_MAXPART];
        lnprob_dens(mol, pow(10.0, p[4 * c + 0]), dens);
        int st = 0;
        const int it = v1_solve(mol, w, lane, pow(10.0, p[4 * c + 1]), dens, pow(10.0, p[4 * c + 2]), S.tbg, cfg, &st);
        if (st & (RB_ST_T_RANGE | RB_ST_N_RANGE)) {
          value_error = true;  // ValueError -> -inf (emcee_radex.py:134-137)
        } else {
          ++solves;
          iters += (unsigned long long)((st & RB_ST_MAXITER) ? it : it + 1);
          if (lane < S.obs.nobs) {
            const double sf = rb_surf(mol, w, S.obs.jup[lane] - 1, cfg);
            model += sf * pow(10.0, p[4 * c + 3]) * 1.0e23;  // x size [sr] x 1 km/s -> Jy km/s
          }
        }
        __syncwarp();
      }
      if (!value_error) result = lnlike_warp(S, model, lp, lane);
    }
    if (lane == 0) io.lnp[idx] = result;
  }
  if (lane == 0) {
    if (iters) atomicAdd(&io.counters[1], iters);
    if (solves) atomicAdd(&io.counters[2], solves);
  }
}

// ------------------------------------------------------------------------------------------------
// v2 kernels (41-level molecules): register-resident GTH elimination with DMMA updates
// ------------------------------------------------------------------------------------------------
#define V2_WARPS 12
#define RB_SCHED_MIN 8192   // batches smaller than this run as one launch
// walkers per call from which lnprob runs as a pipeline.  Measured (walker-steps/s, pipeline vs fused launch, with launch B
// and the engine launches overlapping): 1 component, 8192 walkers per call 4.35e6 vs 3.64e6; 2 components, 8192 per call
// 1.86e6 vs 1.66e6, 16384 per call 2.49e6 vs 1.80e6
#define RB_LNPROB_PIPE_MIN 8192
// rb_stretch_run_dev proposes the second half-step speculatively while 3 x (walkers / 2) candidates are at most this many warps per SM
#define RB_SPEC_WARPS_PER_SM 17

__global__ void __launch_bounds__(V2_WARPS * 32, 1) k_lvg_solve_v2(MolDev mol, SolveCfg cfg, SolveIO io) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  double *sm = smem + (size_t)wib * v2::SLAB;
  double *gB = cfg.bslab + ((size_t)blockIdx.x * V2_WARPS + wib) * v2::GSLAB;
  unsigned phase = 0;
  if (lane == 0) v2::mbar_init(sm + v2::O_MBAR, 1);
  __syncwarp();
  const int nl = mol.nlev, nn = mol.nline;
  unsigned long long iters = 0;
  const long long limit = (io.sched >= 2) ? (long long)*io.n_parked : io.n;
  for (;;) {
    unsigned long long idx = 0;
    if (lane == 0) idx = atomicAdd(&io.counters[io.queue], 1ULL);
    idx = __shfl_sync(0xffffffffu, idx, 0);
    if ((long long)idx >= limit) break;
    if (io.sched >= 2) idx = (unsigned long long)io.order[idx];
    double dens[RB_MAXPART];
#pragma unroll
    for (int p = 0; p < RB_MAXPART; ++p) dens[p] = (p < mol.npart) ? io.dens[idx * mol.npart + p] : 0.0;
    int st = 0, key = -1;
    const double cdmol = io.cdmol[idx];
    const v2::ExtPark xp{io.ext, io.sched_small ? io.sched_small + 50 : nullptr, io.ext_cap, io.ext_off};
    const int it = v2::solve(mol, sm, gB, phase, lane, io.tkin[idx], dens, cdmol, cfg.tbg, cfg, &st, io.sched,
                             io.state ? io.state + idx * v2::STATE_STRIDE : nullptr, &key,
                             (io.sched == 1 && io.ext) ? &xp : nullptr, (long long)idx);
    if (io.sched == 1 && lane == 0) io.keys[idx] = (st & v2::ST_PARKED) ? key : -1;
    if (st & v2::ST_PARKED) {   // launch B finishes this model
      iters += (unsigned long long)it;
      __syncwarp();
      continue;
    }
    const bool bad = (st & (RB_ST_T_RANGE | RB_ST_N_RANGE)) != 0;
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    int nonfinite = 0;
    if (io.obs_surf && lane < io.nobs) {
      double tex, tau, sf = qnan;
      if (!bad) v2::line_results(mol, sm, io.obs_line[lane], cdmol, cfg.tbg, cfg, tex, tau, sf);
      io.obs_surf[idx * RB_MAX_OBS + lane] = sf;
    }
#pragma unroll 1
    for (int l = io.obs_surf ? nn : lane; l < nn; l += 32) {
      double tex = qnan, tau = qnan, sf = qnan;
      if (!bad) {
        v2::line_results(mol, sm, l, cdmol, cfg.tbg, cfg, tex, tau, sf);
        if (!isfinite(sf)) nonfinite = 1;
      }
      if (io.surf) io.surf[idx * nn + l] = sf;
      if (io.tex) io.tex[idx * nn + l] = tex;
      if (io.tau) io.tau[idx * nn + l] = tau;
    }
    if (io.xpop)
      for (int i = lane; i < nl; i += 32) io.xpop[idx * nl + i] = bad ? qnan : sm[v2::O_X + i];
    nonfinite = __any_sync(0xffffffffu, nonfinite);
    if (nonfinite) st |= RB_ST_NONFINITE;
    if (lane == 0) {
      if (io.niter) io.niter[idx] = it;
      if (io.status) io.status[idx] = st;
    }
    // calls of matrix() made here; launch A already counted the first IT_DECIDE of a resumed model
    int it_before = (io.sched == 2) ? v2::IT_DECIDE : 0;   // calls counted by the launches that ran them
    if (io.sched == 4) it_before = (int)(reinterpret_cast<const long long *>(io.state + idx * v2::STATE_STRIDE)[123] & 0xffff);
    iters += bad ? 0 : (unsigned long long)(((st & RB_ST_MAXITER) ? it : it + 1) - it_before);
    __syncwarp();
  }
  if (lane == 0 && iters) atomicAdd(&io.counters[1], iters);
}

// ---- ordering of the parked models between the two launches: counting sort by key, heaviest first ------
constexpr int SCHED_NKEY = 16;
// small[0..15] histogram, [16..31] bin offsets, [32..47] bin cursors (from the front), [48] number of parked models,
// [64..79] bin cursors from the back.  Within a key the models whose next call has a NaN escape probability (bit 8 of the
// key: v2::solve, beta_nan) are placed from the front, the others from the back: those models mostly keep making calls whose
// solution is every level on the floor, and a cached engine skips the elimination of such a call only when BOTH models of the
// warp make one -- neighbours in the queue share a warp.
__global__ void k_sched_hist(const int *keys, long long n, unsigned long long *small) {
  __shared__ unsigned int h[SCHED_NKEY];
  if (threadIdx.x < SCHED_NKEY) h[threadIdx.x] = 0;
  __syncthreads();
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n && keys[i] >= 0) atomicAdd(&h[keys[i] & (SCHED_NKEY - 1)], 1u);
  __syncthreads();
  if (threadIdx.x < SCHED_NKEY && h[threadIdx.x]) atomicAdd(&small[threadIdx.x], (unsigned long long)h[threadIdx.x]);
}
__global__ void k_sched_scan(unsigned long long *small) {
  unsigned long long off = 0;
  for (int k = SCHED_NKEY - 1; k >= 0; --k) {   // heaviest key first: the tail of launch B is made of light models
    small[16 + k] = off;
    small[32 + k] = 0;
    off += small[k];
  }
  small[48] = off;
}
__global__ void k_sched_scatter(const int *keys, long long n, unsigned long long *small, int *order) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n && keys[i] >= 0) {
    const int k = keys[i] & (SCHED_NKEY - 1);
    if (keys[i] & 0x100) {
      const unsigned long long pos = atomicAdd(&small[32 + k], 1ULL);
      order[small[16 + k] + pos] = (int)i;
    } else {
      const unsigned long long pos = atomicAdd(&small[64 + k], 1ULL);
      order[small[16 + k] + small[k] - 1ULL - pos] = (int)i;
    }
  }
}


// ---- cached engines per lead-block size (lvg_small.cuh): G = 16 lanes per model up to 16 lead levels, else 32 ----
#ifdef V2S_TIMING
// debug build only (tools/timing.sh): cycles per section of the engine loop, summed over warps: [KP][0..7] = load, patch,
// pivots, back-substitution, relax, lines, rest of the loop body, iterations
__device__ unsigned long long g_tm[8][8];
#define TM(var) const long long var = clock64()
#else
#define TM(var)
#endif
template <int KP>
__global__ void __launch_bounds__(v2s::Lay<KP>::WARPS * 32, 1) k_lvg_small(MolDev mol, SolveCfg cfg, SolveIO io) {
  using namespace v2s;
  using L = Lay<KP>;
  static_assert(v2::IT_DECIDE >= 1, "the engines never run a model's first call (it == 0 has its own arithmetic in v2::solve)");
  constexpr int G = L::G, NT = L::NT;
  constexpr int SSLAB = L::SSLAB, S_LEAD = L::S_LEAD, S_X = L::S_X, S_XNEW = L::S_XNEW, S_BETA = L::S_BETA,
                S_DNB = L::S_DNB, S_UPB = L::S_UPB, S_TEX = L::S_TEX;
  extern __shared__ double smem[];
  double *cs = smem;   // per-line constants of this call, shared by the CTA
  const int lane = threadIdx.x & 31, hl = lane & (G - 1), half = lane / G, wib = threadIdx.x >> 5;
  const unsigned hmask = (G == 32) ? 0xffffffffu : 0xffffu << (16 * half);   // the lanes of this model
  double *sm = smem + CSLAB + (size_t)(L::MPW * wib + half) * SSLAB;
  int *lmn = reinterpret_cast<int *>(cs + C_LMN);
  const int nl = mol.nlev, nn = mol.nline;
  // the same expressions as the per-line set-up of v2::solve
  for (int l = threadIdx.x; l < nn; l += blockDim.x) {
    const int m = mol.iupp[l], n = mol.ilow[l];
    const double a = mol.aeinst[l], xnu = mol.xnu[l];
    const double xt = xnu * xnu * xnu;
    const double hnu = RB_FK * xnu / cfg.tbg;
    const double bi = (hnu >= 160.0) ? 1.0e-30 : RB_THC * xt / (exp(hnu) - 1.0);
    lmn[l] = m | (n << 8);
    cs[C_LA + l] = a;
    cs[C_LGR + l] = mol.gstat[m] / mol.gstat[n];
    cs[C_LTDEN + l] = 1.0 / (RB_FGAUS * xt / a);
    cs[C_LECOEF + l] = bi / (RB_THC * xt);
    cs[C_LFKXNU + l] = RB_FK * xnu;
    cs[C_XNU + l] = xnu;   // the epilogue's line constants: its backi is bi
    cs[C_BACKI + l] = bi;
  }
  // a slab that never receives a model still runs the arithmetic of its warp: give it finite numbers
  for (int e = hl; e < SSLAB; e += G) sm[e] = 1.0;
  __syncthreads();
  // trips over the lines (tt: lines G tt .. G tt + G - 1) that can hold a lead line, i.e. a line whose escape probability
  // can differ from 1 while the model stays in this engine: the first trip (KP <= 4) or the first two (the host runs the
  // engines only for tables where this holds, lead_lines_fit).  Only these trips are patched and evaluate escprob.
  constexpr unsigned LEAD_TRIPS = L::LEAD_TRIPS;
  // queue: the positions of key KP in the sorted order (heaviest key first; key 3 is the last block)
  const unsigned long long p_begin = io.sched_small[16 + KP], p_end = io.sched_small[(KP == 3) ? 48 : 16 + KP - 1];
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);

  // Hand-over.  Each half holds the queue ticket of its NEXT model while the current one iterates, and walks the chain
  // ticket -> order[] -> ext_off[] one link per call (pf: 1 ticket taken, 2 model index loaded, 3 capture offset loaded
  // and ready, 5 queue ended).  A model that ends before the chain does finishes it at once.  (An L2 prefetch of the next
  // model's state and capture as a further link measured 0.3 % slower on the sweep.)  A ticket is always used by the half that took it, so no model is lost at the queue's end.
  int pf = 0;
  unsigned long long tk = 0;
  long long nidx = 0, noff = 0;
  auto advance = [&]() {
    if (pf == 1) {
      const unsigned long long pos = p_begin + __shfl_sync(hmask, tk, 0, G);
      if (pos >= p_end) {
        pf = 5;
      } else {
        nidx = io.order[pos];
        pf = 2;
      }
    } else if (pf == 2) {
      noff = io.ext_off[nidx];
      pf = 3;
    }
  };
  auto take_ticket = [&]() {
    if (hl == 0) tk = atomicAdd(&io.counters[io.queue], 1ULL);
    pf = 1;
  };

  bool active = false, exhausted = false, need_load = false;
  long long idx = 0, off = 0;
  constexpr int Kp = KP, n = 4 * KP, pitch = n + 2;
  int it = 0, nthick = 0, topthick = -1;
  unsigned flags = 0;   // bit t: line hl + 16 t had tau > 0.01f after the last call (RADEX's own stop rule)
  bool beta_nan = false;   // the call about to be made has a NaN escape probability: its solution is every level on the floor (v2::solve)
  double cdmol = 1.0, cddv = 1.0;
  unsigned long long iters = 0, n_cached = 0, n_models = 0, n_inval = 0;
#ifdef V2S_TIMING
  unsigned long long tm[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  long long tm_prev = clock64();
#endif
  for (;;) {
    TM(tm0);
    // ---- a free half takes the next model of the queue -------------------------------------------------------------
    if (!active && !exhausted) {
      if (pf == 0) take_ticket();
      while (pf < 3) advance();
      if (pf == 5) {
        exhausted = true;
      } else {
        idx = nidx;
        off = noff;
        active = need_load = true;
        take_ticket();   // the next model's; its chain advances during this model's calls
      }
    }
    __syncwarp();
    if (!__any_sync(0xffffffffu, active)) break;   // nothing running and the queue is empty
    if (need_load) {
      need_load = false;
      const double *st = io.state + idx * v2::STATE_STRIDE;
      const double *ex = io.ext + off;
      // lead block + M (contiguous in ext and in the slab) and the lead lines' bases, as 16-byte asynchronous copies;
      // the state loads below are issued while they are in flight
      for (int c = hl; c < 22 * n; c += G) cp_async16(sm + S_LEAD + 2 * c, ex + EXT_LEAD + 2 * c);
      for (int c = hl; c < L::NLEAD; c += G) {
        const int o = (c < L::NLEAD / 2) ? 2 * c : v2::MAXLINE - L::NLEAD + 2 * c;   // DNB pairs, then UPB pairs
        cp_async16(sm + S_DNB + 2 * c, ex + o);
      }
      const unsigned long long bits = reinterpret_cast<const unsigned long long *>(st)[121];
      const long long packed = reinterpret_cast<const long long *>(st)[122];
      const double cdm = io.cdmol[idx];
      double xs[(NL + G - 1) / G], tex[NT], beta[NT];
#pragma unroll
      for (int t = 0; t < (NL + G - 1) / G; ++t) xs[t] = (hl + G * t < NL) ? st[hl + G * t] : 0.0;
#pragma unroll
      for (int t = 0; t < NT; ++t) {
        const int l = hl + G * t;
        tex[t] = (l < nn) ? st[41 + l] : 0.0;
        beta[t] = (l < nn) ? st[81 + l] : 0.0;
      }
#pragma unroll
      for (int t = 0; t < (NL + G - 1) / G; ++t)
        if (hl + G * t < NL) sm[S_X + hl + G * t] = xs[t];
      flags = 0;
      beta_nan = false;
#pragma unroll
      for (int t = 0; t < NT; ++t) {
        const int l = hl + G * t;
        if (l < nn) {
          sm[S_TEX + l] = tex[t];
          if (l < L::NLEAD) sm[S_BETA + l] = beta[t];
          if (beta[t] != beta[t]) beta_nan = true;
          flags |= (unsigned)((bits >> l) & 1ULL) << t;
        }
      }
      beta_nan = __any_sync(hmask, beta_nan);
      nthick = (int)(packed & 0xffffffffLL);
      topthick = (int)(packed >> 32);
      it = v2::IT_DECIDE;
      cdmol = cdm;
      cddv = cdmol / cfg.deltav_cms;
      ++n_models;
      cp_async_wait_all();
    } else if (active && pf < 3) {
      advance();
    }
    __syncwarp();
    TM(tm1);
    // ---- one call of matrix(): radiative rates of the lead lines, lead block, M -------------------------------
    double *B = sm + S_LEAD;
    // every model of the warp is about to make a call whose solution is NaN (v2::solve: beta_nan): no elimination
    const bool skip_solve = __all_sync(0xffffffffu, !active || beta_nan);
#pragma unroll
    for (int t = 0; t < L::NLEAD / G; ++t) {
      const int l = hl + G * t;
      if (l < nn && !skip_solve) {
        const int m = lmn[l] & 0xff, nlo = (lmn[l] >> 8) & 0xff;
        if (max(m, nlo) < n) {
          const double beta = sm[S_BETA + l], a = cs[C_LA + l];
          const double exr = cs[C_LECOEF + l] * beta;
          B[m * pitch + nlo] = sm[S_DNB + l] + a * (beta + exr);
          B[nlo * pitch + m] = sm[S_UPB + l] + a * cs[C_LGR + l] * exr;
        }
      }
    }
    __syncwarp();
    TM(tm2);
#ifdef V2S_TIMING
    long long tmid = clock64();
    const double tot = skip_solve ? __longlong_as_double(0x7ff8000000000000LL) : lead_solve<KP>(sm, hl, &tmid);
#else
    const double tot = skip_solve ? __longlong_as_double(0x7ff8000000000000LL) : lead_solve<KP>(sm, hl);
#endif
    __syncwarp();
    TM(tm3);
    const double rtot = v2::rcp1(tot);
    // ---- normalise, floor, under-relax + pyradex's stop test (v2::solve: lane l of 32 owns levels l and l + 32;
    // in a half-warp lane hl stands for lanes hl (dA) and hl + 16 (dB) of that warp)
    double dA = 0.0, dB = 0.0;
#pragma unroll
    for (int t = 0; t < ((G == 16) ? 3 : 2); ++t) {
      const int i = hl + ((t == 0) ? 0 : (t == 1) ? 32 : 16);
      if (i < NL) {
        const double xn = fmax(v2::KC[v2::KC_MINPOP], sm[S_XNEW + i] * rtot);
        const double prev = sm[S_X + i];
        const double xo = fmax(v2::KC[v2::KC_MINPOP], prev);   // it >= IT_DECIDE >= 1 here: never the first call
        const double xr = v2::KC[v2::KC_F03] * xn + v2::KC[v2::KC_F07] * xo;
        sm[S_XNEW + i] = xn;
        sm[S_X + i] = xr;
        if (t == 2) dB += fabs(prev - xr); else dA += fabs(prev - xr);
      }
    }
    __syncwarp();
    TM(tm4);
    // ---- per line: Tex of this call, optical depth and escape probability of the next ------------------------
    // Straight-line code over the NT trips (no branch per line or per trip): the logarithm of every trip's Tex and the
    // exponential of every trip's escape probability are independent dependency chains that the scheduler interleaves;
    // with a branch around each they ran one after the other and their latency was a third of the whole call.
    // The arithmetic per line is unchanged (a floored or out-of-range line computes on clamped inputs and discards).
    const int nthick_this = nthick;
    nthick = 0;
    topthick = -1;
    unsigned nflags = 0;
    double diff = 0.0, tsA = 0.0, tsB = 0.0;
    bool nan_next = false;
    {
      constexpr unsigned EM = LEAD_TRIPS;   // trips whose lines get their escape probability evaluated
      int ll[NT], lm[NT], ln[NT];
      bool lvalid[NT], lfloored[NT];
      double ltold[NT], larg[NT], ltaur[NT], ltex[NT], lmid[NT];
      bool thick_any = false;
#pragma unroll
      for (int t = 0; t < NT; ++t) {
        // half-warp: lines hl, hl + 32 (tsA), hl + 16 (tsB): the order of the 32-lane sums
        const int tt = (G == 16) ? ((t == 0) ? 0 : (t == 1) ? 2 : 1) : t;
        const int l = hl + G * tt;
        lvalid[t] = l < nn;
        ll[t] = lvalid[t] ? l : ((hl < nn) ? hl : 0);   // an out-of-range lane recomputes its OWN first-trip line (and discards): it
                                                        // reads no slot that another lane writes in this section
        const int mn = lmn[ll[t]];
        lm[t] = mn & 0xff;
        ln[t] = (mn >> 8) & 0xff;
        const double gr = cs[C_LGR + ll[t]];
        const double xm = sm[S_XNEW + lm[t]], xn = sm[S_XNEW + ln[t]];
        lfloored[t] = (xn <= v2::KC[v2::KC_MINPOP]) || (xm <= v2::KC[v2::KC_MINPOP]);
        ltold[t] = sm[S_TEX + ll[t]];
        larg[t] = xn * gr * v2::rcp1(xm);
        const double tau = cddv * (sm[S_X + ln[t]] * gr - sm[S_X + lm[t]]) * cs[C_LTDEN + ll[t]];
        ltaur[t] = tau * 0.5;
        if (lvalid[t]) {
          if (tau > v2::KC[v2::KC_D001]) ++nthick;
          if (tau > v2::KC[v2::KC_F001]) nflags |= 1u << tt;
          if (!(fabs(ltaur[t]) < v2::KC[v2::KC_F001])) topthick = max(topthick, max(lm[t], ln[t]));
          if (((EM >> tt) & 1u) && !(fabs(ltaur[t]) < 7.0)) thick_any = true;
        }
      }
      diff = (G == 16) ? group_sum<G>(dA + dB) : group_sum<G>(dA);
#pragma unroll
      for (int t = 0; t < NT; ++t) ltex[t] = cs[C_LFKXNU + ll[t]] * v2::rcp1(v2::fast_log(larg[t]));
#pragma unroll
      for (int t = 0; t < NT; ++t) {
        const int tt = (G == 16) ? ((t == 0) ? 0 : (t == 1) ? 2 : 1) : t;
        lmid[t] = ((EM >> tt) & 1u) ? v2::escprob_lvg_mid(ltaur[t]) : 1.0;
      }
      if (__any_sync(0xffffffffu, thick_any)) {   // a line with |tau/2| >= 7 (or NaN) somewhere in the warp: escprob's third branch
#pragma unroll
        for (int t = 0; t < NT; ++t) {
          const int tt = (G == 16) ? ((t == 0) ? 0 : (t == 1) ? 2 : 1) : t;
          if ((EM >> tt) & 1u) {
            const double bl = v2::escprob_lvg_thick(ltaur[t]);
            if (!(fabs(ltaur[t]) < 7.0)) lmid[t] = bl;
          }
        }
      }
#pragma unroll
      for (int t = 0; t < NT; ++t) {
        const int tt = (G == 16) ? ((t == 0) ? 0 : (t == 1) ? 2 : 1) : t;
        const double thistex = lfloored[t] ? ltold[t] : ltex[t];
        if (cfg.stop_rule == RB_STOP_RADEX && lvalid[t] && ((flags >> tt) & 1u)) {
          if (G == 16 && tt == 1) tsB += fabs((thistex - ltold[t]) / thistex); else tsA += fabs((thistex - ltold[t]) / thistex);
        }
        if (lvalid[t]) {
          sm[S_TEX + ll[t]] = 0.5 * (thistex + ltold[t]);
          // a trip without lead lines keeps beta = 1 (its lines are frozen; if one turns thick the model leaves this engine
          // and the leave path below evaluates escprob for it)
          if ((EM >> tt) & 1u) {
            const double beta_next = (fabs(ltaur[t]) < v2::KC[v2::KC_F001]) ? 1.0 : lmid[t];
            sm[S_BETA + ll[t]] = beta_next;
            if (beta_next != beta_next) nan_next = true;
          }
        }
      }
    }
    flags = nflags;
    beta_nan = __any_sync(hmask, nan_next);
    topthick = group_max_int(hmask, topthick);
    bool stop;
    if (cfg.stop_rule == RB_STOP_RADEX) {
      int conv = 0;
      nthick = group_sum_int(hmask, nthick);
      const double tsum = (G == 16) ? group_sum<G>(tsA + tsB) : group_sum<G>(tsA);
      if (it >= 10) {
        if (nthick_this == 0) conv = 1;
        else if (tsum / nthick_this < RB_F32(1.0e-6)) conv = 1;
      }
      stop = conv != 0;
    } else {
      stop = (diff < cfg.abs_tol) && (it > cfg.miniter);
    }
    __syncwarp();
#ifdef V2S_TIMING
    {
      const long long tm5 = clock64();
      tm[0] += tm1 - tm0; tm[1] += tm2 - tm1; tm[2] += tmid - tm2; tm[3] += tm3 - tmid; tm[4] += tm4 - tm3; tm[5] += tm5 - tm4;
      tm[6] += tm0 - tm_prev; tm[7] += 1;
      tm_prev = tm5;
    }
#endif
    if (!active) continue;
    ++n_cached;
    // ---- what v2::solve decides at the bottom of this call and at the top of the next ---------------------------
    bool hit_max = false, leave = false;
    if (!stop) {
      ++it;
      if (it >= cfg.maxiter) hit_max = true;
      else if (((topthick + 4) >> 2) > Kp) leave = true;
    }
    if (leave) {
      // a frozen line turned thick: park for launch C, which re-captures with a larger lead block
      double *st = io.state + idx * v2::STATE_STRIDE;
      for (int i = hl; i < NL; i += G) st[i] = sm[S_X + i];
      unsigned long long bits = 0;
#pragma unroll
      for (int t = 0; t < NT; ++t) {
        const int l = hl + G * t;
        if (l < nn) {
          // escape probability of the next call for EVERY line (the loop keeps it only for the trips with lead lines):
          // the expressions of the loop, from the same relaxed populations
          const int m = lmn[l] & 0xff, nlo = (lmn[l] >> 8) & 0xff;
          const double tau = cddv * (sm[S_X + nlo] * cs[C_LGR + l] - sm[S_X + m]) * cs[C_LTDEN + l];
          st[41 + l] = sm[S_TEX + l];
          st[81 + l] = v2::escprob_fast(tau, RB_GEOM_LVG);
        }
        const unsigned b = __ballot_sync(hmask, (flags >> t) & 1u);
        bits |= (unsigned long long)((G == 32) ? b : (b >> (16 * half)) & 0xffffu) << (G * t);
      }
      if (hl == 0) {
        reinterpret_cast<unsigned long long *>(st)[121] = bits;
        reinterpret_cast<long long *>(st)[122] = ((long long)topthick << 32) | (long long)(unsigned)nthick;
        reinterpret_cast<long long *>(st)[123] = v2::resume_word(it, 1);
        io.order_c[atomicAdd(&io.sched_small[49], 1ULL)] = (int)idx;
      }
      iters += (unsigned long long)(it - v2::IT_DECIDE);
      ++n_inval;
      active = false;
      __syncwarp(hmask);
      continue;
    }
    if (!(stop || hit_max)) continue;
    // ---- results (k_lvg_solve_v2's epilogue) --------------------------------------------------------------------
    int nonfinite = 0;
    const int l_first = io.obs_surf ? ((hl < io.nobs) ? io.obs_line[hl] : nn) : hl;
    const int l_step = io.obs_surf ? nn : G;
#pragma unroll 1
    for (int l = l_first; l < nn; l += l_step) {
      const int m = lmn[l] & 0xff, nlo = (lmn[l] >> 8) & 0xff;
      const double xnu = cs[C_XNU + l];
      const double xt = xnu * xnu * xnu;
      const double backi = cs[C_BACKI + l];
      const double tex = sm[S_TEX + l];
      const double tau = (cdmol / cfg.deltav_cms) * (sm[S_XNEW + nlo] * cs[C_LGR + l] - sm[S_XNEW + m]) * cs[C_LTDEN + l];
      const double ftau = exp(-tau);
      const double earg = cfg.fk_epi * xnu / tex;
      const double bnutex = cfg.thc_epi * xt / (exp(earg) - 1.0);
      const double toti = backi * ftau + bnutex * (1.0 - ftau);
      const double sf = toti - backi;
      if (io.obs_surf) {
        io.obs_surf[idx * RB_MAX_OBS + hl] = sf;
        continue;
      }
      if (!isfinite(sf)) nonfinite = 1;
      if (io.surf) io.surf[idx * nn + l] = sf;
      if (io.tex) io.tex[idx * nn + l] = tex;
      if (io.tau) io.tau[idx * nn + l] = tau;
    }
    if (io.xpop)
      for (int i = hl; i < nl; i += G) io.xpop[idx * nl + i] = sm[S_X + i];
    nonfinite = __any_sync(hmask, nonfinite);
    if (hl == 0) {
      if (io.niter) io.niter[idx] = it;
      if (io.status) io.status[idx] = (hit_max ? RB_ST_MAXITER : 0) | (nonfinite ? RB_ST_NONFINITE : 0);
    }
    iters += (unsigned long long)((hit_max ? it : it + 1) - v2::IT_DECIDE);
    active = false;
    __syncwarp(hmask);
  }
  (void)qnan;
#ifdef V2S_TIMING
  if (lane == 0)
    for (int i = 0; i < 8; ++i) atomicAdd(&g_tm[KP][i], tm[i]);
#endif
  if (hl == 0) {
    if (iters) atomicAdd(&io.counters[1], iters);
    if (cfg.stats && n_models) {
      atomicAdd(&cfg.stats[0], n_cached);
      atomicAdd(&cfg.stats[1], n_models);   // one capture each (made by launch A)
      if (n_inval) atomicAdd(&cfg.stats[2], n_inval);
    }
  }
}

template <int KP>
constexpr size_t small_smem() { return v2s::smem_bytes<KP>(); }

template <int NCOMP>
__global__ void __launch_bounds__(V2_WARPS * 32, 1) k_lnprob_v2(MolDev mol, SolveCfg cfg, LnprobIO io) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  double *sm = smem + (size_t)wib * v2::SLAB;
  double *gB = cfg.bslab + ((size_t)blockIdx.x * V2_WARPS + wib) * v2::GSLAB;
  unsigned phase = 0;
  if (lane == 0) v2::mbar_init(sm + v2::O_MBAR, 1);
  __syncwarp();
  constexpr int ND = 4 * NCOMP;
  unsigned long long iters = 0, solves = 0;
  for (;;) {
    unsigned long long idx = 0;
    if (lane == 0) idx = atomicAdd(&io.counters[0], 1ULL);
    idx = __shfl_sync(0xffffffffu, idx, 0);
    if ((long long)idx >= io.n) break;
    const rb_source &S = io.srcs[io.src_id ? io.src_id[idx] : 0];
    double p[ND];
#pragma unroll
    for (int i = 0; i < ND; ++i) p[i] = io.P[idx * ND + i];
    const double lp = (NCOMP == 1) ? lnprior1(p, S.bounds) : lnprior2(p, S.bounds, S.has_td, S.t_d);
    double result = neg_inf();
    if (isfinite(lp)) {  // prior short-circuit: no solve (emcee_radex.py:178-180)
      double model = 0.0;
      bool value_error = false;
      const double tbg = S.tbg;
#pragma unroll
      for (int c = 0; c < NCOMP; ++c) {
        if (value_error) break;
        double dens[RB_MAXPART];
        lnprob_dens(mol, pow(10.0, p[4 * c + 0]), dens);
        int st = 0;
        const double cdmol = pow(10.0, p[4 * c + 2]);
        const int it = v2::solve<true>(mol, sm, gB, phase, lane, pow(10.0, p[4 * c + 1]), dens, cdmol, tbg, cfg, &st);
        if (st & (RB_ST_T_RANGE | RB_ST_N_RANGE)) {
          value_error = true;  // ValueError -> -inf (emcee_radex.py:134-137)
        } else {
          ++solves;
          iters += (unsigned long long)((st & RB_ST_MAXITER) ? it : it + 1);
          // only the observed lines' fluxes are needed: lane i < nobs evaluates line Jup_i - 1
          if (lane < S.obs.nobs) {
            double tex, tau, sf;
            v2::line_results(mol, sm, S.obs.jup[lane] - 1, cdmol, tbg, cfg, tex, tau, sf);
            model += sf * pow(10.0, p[4 * c + 3]) * 1.0e23;
          }
        }
        __syncwarp();
      }
      if (!value_error) result = lnlike_warp(S, model, lp, lane);
    }
    if (lane == 0) io.lnp[idx] = result;
  }
  if (lane == 0) {
    if (iters) atomicAdd(&io.counters[1], iters);
    if (solves) atomicAdd(&io.counters[2], solves);
  }
}

// ---- lnprob as a pipeline for large ensembles: priors and walker -> model parameters (k_lnprob_expand), the
// scheduled solve of all n x NCOMP models with the half-warp engine (launch_solve_pipeline), fluxes -> chi^2
// (k_lnprob_combine).  Same expressions as the fused k_lnprob_v2, which stays the path of small ensembles.
struct LnprobPipe {
  double *tkin, *dens, *cdmol;   // n x NCOMP models
  double *obs_surf;              // [n x NCOMP][RB_MAX_OBS]
  int *status;
};

template <int NCOMP>
__global__ void k_lnprob_expand(MolDev mol, LnprobIO io, LnprobPipe pp) {
  constexpr int ND = 4 * NCOMP;
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (idx >= io.n) return;
  double p[ND];
#pragma unroll
  for (int i = 0; i < ND; ++i) p[i] = io.P[idx * ND + i];
  const rb_source &S = io.srcs[0];   // the pipeline serves one source per call
  const double lp = (NCOMP == 1) ? lnprior1(p, S.bounds) : lnprior2(p, S.bounds, S.has_td, S.t_d);
  io.lnp[idx] = lp;   // the prior waits here for k_lnprob_combine
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);
#pragma unroll
  for (int c = 0; c < NCOMP; ++c) {
    const long long m = idx * NCOMP + c;
    const bool go = isfinite(lp);   // prior short-circuit: a NaN temperature is refused before any work is done
    const double dens_tot = pow(10.0, p[4 * c + 0]);
    for (int q = 0; q < mol.npart; ++q) pp.dens[m * mol.npart + q] = mol.ln_frac[q] * dens_tot;
    pp.tkin[m] = go ? pow(10.0, p[4 * c + 1]) : qnan;
    pp.cdmol[m] = pow(10.0, p[4 * c + 2]);
  }
}

template <int NCOMP>
__global__ void k_lnprob_combine(LnprobIO io, LnprobPipe pp) {
  constexpr int ND = 4 * NCOMP;
  const int lane = threadIdx.x & 31;
  const long long idx = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;   // one warp per walker
  if (idx >= io.n) return;
  const rb_source &S = io.srcs[0];
  const double lp = io.lnp[idx];
  double result = neg_inf();
  unsigned long long solves = 0;
  if (isfinite(lp)) {
    double model = 0.0;
    bool value_error = false;
#pragma unroll
    for (int c = 0; c < NCOMP; ++c) {
      // the reference stops at the first ValueError: a later component was solved here but is not counted, as in
      // k_lnprob_v2
      if (value_error) break;
      const long long m = idx * NCOMP + c;
      if (pp.status[m] & (RB_ST_T_RANGE | RB_ST_N_RANGE)) {
        value_error = true;
      } else {
        ++solves;
        if (lane < S.obs.nobs) model += pp.obs_surf[m * RB_MAX_OBS + lane] * pow(10.0, io.P[idx * ND + 4 * c + 3]) * 1.0e23;
      }
    }
    if (!value_error) result = lnlike_warp(S, model, lp, lane);
  }
  if (lane == 0) {
    io.lnp[idx] = result;
    if (solves) atomicAdd(&io.counters[2], solves);
  }
}

// ------------------------------------------------------------------------------------------------
// stretch move (emcee StretchMove / RedBlueMove; SURVEY.md 3.5) with Philox4x32-10
// ------------------------------------------------------------------------------------------------
// host and device: the move schedule (rb_move_schedule) is drawn on the host from the same generator
__host__ __device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}

__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = mulhi32(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = mulhi32(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
}

__host__ __device__ __forceinline__ double u01(uint32_t hi, uint32_t lo) {  // 53-bit uniform in [0,1)
  const unsigned long long v = ((unsigned long long)hi << 32) | lo;
  return (double)(v >> 11) * 1.1102230246251565e-16;
}

__global__ void k_stretch_propose(long long ns, int ndim, const double *S, long long nc, const double *C, double a,
                                  unsigned long long seed, unsigned long long step, int half, long long gid0,
                                  long long gid_stride, double *Q, double *logfac) {
  const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= ns) return;
  const unsigned long long gid = (unsigned long long)(gid0 + k * gid_stride);
  uint32_t c[4] = {(uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)(step * 2ULL + (unsigned)half),
                   (uint32_t)((step * 2ULL + (unsigned)half) >> 32) & 0x7fffffffu};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  const double u = u01(c[0], c[1]);
  // explicit roundings (no FMA contraction) so a host restatement reproduces the proposal bit for bit
  const double sq = __dadd_rn(__dmul_rn(a - 1.0, u), 1.0);
  const double z = __dmul_rn(sq, sq) / a;
  long long j = (long long)(u01(c[2], c[3]) * (double)nc);
  if (j >= nc) j = nc - 1;
  for (int d = 0; d < ndim; ++d) {
    const double cj = C[j * ndim + d], s = S[k * ndim + d];
    Q[k * ndim + d] = __dsub_rn(cj, __dmul_rn(cj - s, z));
  }
  logfac[k] = (ndim - 1.0) * log(z);
}

__global__ void k_stretch_accept(long long ns, int ndim, double *S, double *lnp_old, const double *Q,
                                 const double *lnp_new, const double *logfac, unsigned long long seed,
                                 unsigned long long step, int half, long long gid0, long long gid_stride,
                                 unsigned long long *naccept) {
  const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  int acc = 0;
  if (k < ns) {
    const unsigned long long gid = (unsigned long long)(gid0 + k * gid_stride);
    uint32_t c[4] = {(uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)(step * 2ULL + (unsigned)half),
                     ((uint32_t)((step * 2ULL + (unsigned)half) >> 32) & 0x7fffffffu) | 0x80000000u};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    const double lnu = log(u01(c[0], c[1]));
    const double lnew = lnp_new[k];
    const double lnpdiff = logfac[k] + lnew - lnp_old[k];
    // emcee: accepted = lnpdiff > log(u).  -inf - -inf = NaN compares false -> rejected, like numpy.
    if (lnpdiff > lnu) {
      acc = 1;
      for (int d = 0; d < ndim; ++d) S[k * ndim + d] = Q[k * ndim + d];
      lnp_old[k] = lnew;
    }
  }
  const unsigned ballot = __ballot_sync(0xffffffffu, acc);
  if ((threadIdx.x & 31) == 0 && ballot && naccept) atomicAdd(naccept, (unsigned long long)__popc(ballot));
}


#include "stretch.cuh"
#include "chain_stats.cuh"
#include "chain_marginals.cuh"
#include "predict_sled.cuh"

// ------------------------------------------------------------------------------------------------
// FP64 FMA peak probe: the roofline denominator for the solve kernels is the vector FP64 pipe,
// which MEASURED_PEAKS.json does not cover, so bench.py measures it live with this kernel.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_fp64_peak(double *out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double b = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
      a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
namespace {

template <typename T>
int upload(rb_ctx *ctx, const std::vector<T> &v, const T **out) {
  void *d = nullptr;
  const size_t bytes = std::max<size_t>(v.size(), 1) * sizeof(T);
  CUDA_TRY(cudaMalloc(&d, bytes));
  ctx->owned.push_back(d);
  if (!v.empty()) CUDA_TRY(cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  *out = static_cast<const T *>(d);
  return RB_OK;
}

// the caller's options, or the defaults where it passes none
rb_opts resolve_opts(const rb_opts *o) {
  rb_opts d;
  rb_default_opts(&d);
  if (o) d = *o;
  return d;
}

SolveCfg make_cfg(const rb_ctx *ctx, const rb_opts *o, double deltav_kms, double tbg, int geometry) {
  const rb_opts d = resolve_opts(o);
  SolveCfg c;
  c.bslab = ctx->bslab;
  c.deltav_cms = deltav_kms * 1.0e5;  // km/s -> cm/s (core.py:447-454)
  c.tbg = tbg;
  c.method = geometry;
  c.stop_rule = d.stop_rule;
  c.miniter = d.miniter;
  c.maxiter = d.maxiter;
  c.abs_tol = d.abs_tol;
  c.fk_epi = d.fk_epi;
  c.thc_epi = d.thc_epi;
  c.cache = (d.kernel != 2);
  c.sched = (d.kernel == 0 || d.kernel == 4);
  c.small = (d.kernel == 0) && ctx->engines_fit;
  c.park_max = (d.park_max >= v2::KP_CACHE_MIN && d.park_max <= v2::KP_SMALL_MAX) ? d.park_max : 0;
  c.lnprob_pipe_min = (d.lnprob_pipe_min > 0) ? d.lnprob_pipe_min : RB_LNPROB_PIPE_MIN;
  c.stats = ctx->counters + 3;
  return c;
}

int check_common(rb_ctx *ctx, double deltav_kms, double tbg, int geometry) {
  if (!ctx) {
    rb_set_error("null context");
    return RB_ERR_ARG;
  }
  if (geometry < 1 || geometry > 3) {
    rb_set_error("Invalid escapeProbGeom, must be one of lvg,sphere,slab");
    return RB_ERR_ARG;
  }
  if (!(deltav_kms > 0.0) || !(tbg > 0.0)) {
    rb_set_error("deltav and tbg must be positive");
    return RB_ERR_ARG;
  }
  return RB_OK;
}

struct Launch {
  int warps_per_block;
  int blocks;
  size_t smem;
};

Launch v1_launch(rb_ctx *ctx, long long n) {
  const size_t per_warp = v1_warp_doubles(ctx->mol.nlev, ctx->mol.nline) * sizeof(double);
  int wpb = (int)(((size_t)ctx->smem_optin - 1024) / per_warp);
  if (wpb > 8) wpb = 8;
  if (wpb < 1) wpb = 1;
  Launch L;
  L.warps_per_block = wpb;
  L.smem = per_warp * wpb;
  long long need = (n + wpb - 1) / wpb;
  L.blocks = (int)std::min<long long>(need, ctx->sm_count);
  if (L.blocks < 1) L.blocks = 1;
  return L;
}

bool use_v2(const rb_ctx *ctx, const rb_opts *o) {
  const int kernel = o ? o->kernel : 0;
  return kernel != 1 && kernel <= 4 && kernel >= 0 && ctx->mol.nlev == v2::NL && ctx->mol.nline <= v2::MAXLINE;
}

// One CTA per SM; a batch with fewer models than 12 warps x SMs spreads them over the SMs (a small ensemble's
// half-step is 50 models: one warp each on 50 SMs, not 12 warps on each of 5)
Launch v2_launch(rb_ctx *ctx, long long n) {
  Launch L;
  const long long per_sm = (n + ctx->sm_count - 1) / ctx->sm_count;
  L.warps_per_block = (int)std::max<long long>(1, std::min<long long>(per_sm, V2_WARPS));
  L.smem = (size_t)L.warps_per_block * v2::SLAB * sizeof(double);
  const long long need = (n + L.warps_per_block - 1) / L.warps_per_block;
  L.blocks = (int)std::max<long long>(1, std::min<long long>(need, ctx->sm_count));
  return L;
}

// An lnprob call of n walkers runs as a pipeline (expand -> scheduled solve of n x ncomp models -> combine) rather
// than as one fused launch
bool lnprob_pipelined(const rb_ctx *ctx, const SolveCfg &cfg, const rb_opts *opts, int nsrc, long long n, int ncomp) {
  return nsrc == 1 && use_v2(ctx, opts) && cfg.sched && cfg.small && cfg.cache && n >= cfg.lnprob_pipe_min &&
         n * ncomp >= RB_SCHED_MIN;
}

// Grow-only device buffer p of cap bytes: a request for more replaces it with need + headroom bytes
int grow(void *&p, size_t &cap, size_t need, size_t headroom = 0) {
  if (need <= cap) return RB_OK;
  if (p) cudaFree(p);
  p = nullptr;
  cap = 0;
  CUDA_TRY(cudaMalloc(&p, need + headroom));
  cap = need + headroom;
  return RB_OK;
}

int ensure_scratch(rb_ctx *ctx, size_t bytes) { return grow(ctx->scratch, ctx->scratch_bytes, bytes, bytes / 4); }

// Hands out consecutive 256-byte-aligned arrays from base.  A layout is run once with a null base, which only adds up
// its size, and then with the buffer grown to that size.
struct Carve {
  void *base;
  size_t bytes = 0;
  template <typename T>
  T *take(long long count) {
    T *p = base ? reinterpret_cast<T *>(static_cast<char *>(base) + bytes) : nullptr;
    bytes += ((size_t)count * sizeof(T) + 255) & ~size_t(255);
    return p;
  }
};

// The model arrays of an expand -> solve -> combine call of m models, from ctx->ln_buf; the brightness holds `stride`
// lines per model
int model_arrays(rb_ctx *ctx, long long m, int stride, LnprobPipe *pp) {
  auto layout = [&](Carve c) {
    pp->tkin = c.take<double>(m);
    pp->cdmol = c.take<double>(m);
    pp->dens = c.take<double>(m * ctx->mol.npart);
    pp->obs_surf = c.take<double>(m * stride);
    pp->status = c.take<int>(m);
    return c.bytes;
  };
  const int rc = grow(ctx->ln_buf, ctx->ln_bytes, layout(Carve{nullptr}));
  if (rc != RB_OK) return rc;
  layout(Carve{ctx->ln_buf});
  return RB_OK;
}

// observed-line mode: only the brightness of lines jup[k] - 1 is written, at obs_surf[model][k]
void observe_lines(SolveIO &io, double *obs_surf, int nobs, const int32_t *jup) {
  io.obs_surf = obs_surf;
  io.nobs = nobs;
  for (int k = 0; k < nobs; ++k) io.obs_line[k] = jup[k] - 1;
}

// models [o, o + m) of io
SolveIO slice(const rb_ctx *ctx, const SolveIO &io, long long o, long long m) {
  const int np = ctx->mol.npart, nl = ctx->mol.nlev, nn = ctx->mol.nline;
  SolveIO part = io;
  part.n = m;
  part.tkin += o;
  part.dens += o * np;
  part.cdmol += o;
  if (part.xpop) part.xpop += o * nl;
  if (part.tex) part.tex += o * nn;
  if (part.tau) part.tau += o * nn;
  if (part.surf) part.surf += o * nn;
  if (part.niter) part.niter += o;
  if (part.status) part.status += o;
  if (part.obs_surf) part.obs_surf += o * RB_MAX_OBS;
  return part;
}

// After the work queued on ctx->stream: the iteration total of the last call (kept in the ctx) and its solves
int read_counters(rb_ctx *ctx, int64_t *nsolves = nullptr) {
  unsigned long long cnt[3] = {0, 0, 0};
  CUDA_TRY(cudaMemcpyAsync(cnt, ctx->counters, sizeof(cnt), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  ctx->last_total_iters = (long long)cnt[1];
  if (nsolves) *nsolves = (int64_t)cnt[2];
  return RB_OK;
}

}  // namespace

extern "C" {

void rb_default_opts(rb_opts *o) {
  if (!o) return;
  o->stop_rule = RB_STOP_PYRADEX;
  o->miniter = 10;
  o->maxiter = 200;
  o->kernel = 0;
  o->abs_tol = 1e-16;
  // astropy (CODATA 2018) h c / k_B and 2 h c in cgs, which is what core.py:981-984 evaluates to
  o->fk_epi = 1.4387768775039338;
  o->thc_epi = 3.9728917142978115e-16;
  o->park_max = 0;
  o->spec_half = 0;
  o->lnprob_pipe_min = 0;
}

int rb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int rb_ctx_create(int device, const rb_mol *mol, rb_ctx **out) {
  if (!mol || !out) {
    rb_set_error("rb_ctx_create: null argument");
    return RB_ERR_ARG;
  }
  *out = nullptr;
  if (mol->nlev > RB_MAXLEV) {
    rb_set_error("molecule has more levels than RB_MAXLEV");
    return RB_ERR_LIMIT;
  }
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) {
    rb_set_error("no such CUDA device");
    return RB_ERR_CUDA;
  }
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) {
    rb_set_error("libradex_b200 is built for sm_100a only; device is sm_" + std::to_string(prop.major * 10 + prop.minor));
    return RB_ERR_CUDA;
  }
  rb_ctx *ctx = new rb_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  ctx->smem_optin = (int)prop.sharedMemPerBlockOptin;
  if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
    rb_set_error("cudaStreamCreate failed");
    delete ctx;
    return RB_ERR_CUDA;
  }
  ctx->stream = ctx->own_stream;
  MolDev &m = ctx->mol;
  m.nlev = mol->nlev;
  m.nline = mol->nline;
  m.npart = mol->npart;
  m.sorted_levels = 1;
  ctx->engines_fit = v2s::lead_lines_fit(mol->iupp.data(), mol->ilow.data(), mol->nline);
  for (int i = 0; i + 1 < mol->nlev; ++i)
    if (!(mol->eterm[i + 1] > mol->eterm[i])) m.sorted_levels = 0;
  int rc = RB_OK;
#define UP(vec, dst)                                  \
  if (rc == RB_OK) rc = upload(ctx, vec, &dst);
  UP(mol->eterm, m.eterm);
  UP(mol->gstat, m.gstat);
  UP(mol->iupp, m.iupp);
  UP(mol->ilow, m.ilow);
  UP(mol->aeinst, m.aeinst);
  UP(mol->xnu, m.xnu);
  // CSR of lines incident on each level, in line order (keeps the reference's summation order)
  std::vector<int> ptr(mol->nlev + 1, 0), idx;
  for (int i = 0; i < mol->nlev; ++i) {
    for (int l = 0; l < mol->nline; ++l) {
      if (mol->iupp[l] == i) idx.push_back(l | 0x40000000);
      if (mol->ilow[l] == i) idx.push_back(l);
    }
    ptr[i + 1] = (int)idx.size();
  }
  UP(ptr, m.lev_ptr);
  UP(idx, m.lev_line);
  for (int p = 0; p < mol->npart && rc == RB_OK; ++p) {
    const rb_mol::Partner &pt = mol->partners[p];
    m.part_id[p] = pt.id;
    m.ntemp[p] = pt.ntemp;
    m.ncoll[p] = pt.ncoll;
    UP(pt.temps, m.temps[p]);
    UP(pt.lcu, m.lcu[p]);
    UP(pt.lcl, m.lcl[p]);
    UP(pt.rates_tc, m.rates_tc[p]);
  }
#undef UP
  {
    // lnprob's collider densities (emcee_radex.py:122-124 sets {'oH2': fortho n, 'pH2': (1 - fortho) n}, opr = 3):
    // pyradex folds them into H2 when the file lists that partner (core.py:551-556), else keeps them apart;
    // every other partner gets zero density
    const double fortho = 3.0 / (1.0 + 3.0);
    bool has_h2 = false;
    for (int p = 0; p < mol->npart; ++p) has_h2 |= (mol->partners[p].id == 1);
    for (int p = 0; p < RB_MAXPART; ++p) m.ln_frac[p] = 0.0;
    for (int p = 0; p < mol->npart; ++p) {
      const int id = mol->partners[p].id;
      if (has_h2) m.ln_frac[p] = (id == 1) ? 1.0 : 0.0;
      else m.ln_frac[p] = (id == 2) ? 1.0 - fortho : (id == 3) ? fortho : 0.0;
      if (m.ln_frac[p] > 0.0) ctx->ln_partners_ok = true;
    }
  }
  if (rc == RB_OK && cudaMalloc(&ctx->counters, 16 * sizeof(unsigned long long)) != cudaSuccess) {
    rb_set_error("cudaMalloc(counters) failed");
    rc = RB_ERR_CUDA;
  }
  if (rc == RB_OK) {
    // every kernel may use the whole opt-in shared memory of the device: the attribute belongs to the function, not to
    // the context, so it must not depend on which molecule this context holds
    const int smax = ctx->smem_optin;
    cudaError_t e = cudaFuncSetAttribute(k_lvg_solve_v1, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_lnprob_v1<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_lnprob_v1<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_lvg_solve_v2, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_lvg_small<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_lvg_small<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_lvg_small<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_lvg_small<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_lvg_small<7>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_lnprob_v2<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_lnprob_v2<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (e == cudaSuccess && (size_t)smax < (size_t)V2_WARPS * v2::SLAB * sizeof(double)) {
      rb_set_error("device offers less shared memory per block than the kernels need");
      rc = RB_ERR_LIMIT;
    }
    if (e == cudaSuccess && rc == RB_OK && mol->nlev == v2::NL && mol->nline <= v2::MAXLINE)
      e = cudaMalloc(&ctx->bslab, (size_t)ctx->sm_count * V2_WARPS * v2::GSLAB * sizeof(double));
    if (e != cudaSuccess) {
      rb_set_error(std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e));
      rc = RB_ERR_CUDA;
    }
  }
  if (rc != RB_OK) {
    rb_ctx_destroy(ctx);
    return rc;
  }
  *out = ctx;
  return RB_OK;
}

void rb_ctx_destroy(rb_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  for (void *p : ctx->owned) cudaFree(p);
  for (void *p : {ctx->scratch, ctx->sched_buf, ctx->ln_buf, ctx->samp_buf, ctx->cs_buf, (void *)ctx->counters,
                  (void *)ctx->bslab, (void *)ctx->sched_small, (void *)ctx->src_one})
    if (p) cudaFree(p);
  for (cudaGraphExec_t g : ctx->samp_graph)
    if (g) cudaGraphExecDestroy(g);
  if (ctx->ev_samp) cudaEventDestroy(ctx->ev_samp);
  for (cudaEvent_t ev : ctx->chunk_done) cudaEventDestroy(ev);
  for (int j = 0; j < 6; ++j) {
    if (ctx->side[j]) cudaStreamDestroy(ctx->side[j]);
    if (ctx->ev_side[j]) cudaEventDestroy(ctx->ev_side[j]);
  }
  if (ctx->ev_sorted) cudaEventDestroy(ctx->ev_sorted);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  delete ctx;
}

int rb_ctx_sync(rb_ctx *ctx) {
  if (!ctx) return RB_ERR_ARG;
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return RB_OK;
}

int rb_ctx_set_stream(rb_ctx *ctx, void *stream) {
  if (!ctx) return RB_ERR_ARG;
  ctx->stream = static_cast<cudaStream_t>(stream);   // 0 is CUDA's legacy default stream, used as given
  return RB_OK;
}

int rb_ctx_reset_stream(rb_ctx *ctx) {
  if (!ctx) return RB_ERR_ARG;
  ctx->stream = ctx->own_stream;
  return RB_OK;
}

// The scheduled solve of a large batch (lvg_v2.cuh, lvg_small.cuh): launch A, counting sort by lead-block size,
// launch B (large lead blocks), k_lvg_small (small ones, two per warp), launch C (invalidated small ones).
#define RB_MID_MIN (1LL << 17)   // batches from this size on also run the 20/24/28-level lead blocks in their own launches
                                 // (measured with the launches overlapping: 2^16 models 4 % slower with the three extra
                                 // launches, 2^17 2 % faster, 2^20 6 % faster)
#define RB_PIPE_MAX (1LL << 20)   // models per scheduled pass: bounds the parked state + captures at 1 + 7 GB

static int launch_solve_pipeline(rb_ctx *ctx, const SolveCfg &cfg_in, SolveIO io) {
  if (io.n > RB_PIPE_MAX && cfg_in.small) {   // larger batches: one pass per 2^20 models, totals keep accumulating
    for (long long o = 0; o < io.n; o += RB_PIPE_MAX) {
      if (o > 0) CUDA_TRY(cudaMemsetAsync(ctx->counters, 0, sizeof(unsigned long long), ctx->stream));   // queue head
      const int rc = launch_solve_pipeline(ctx, cfg_in, slice(ctx, io, o, std::min<long long>(RB_PIPE_MAX, io.n - o)));
      if (rc != RB_OK) return rc;
    }
    return RB_OK;
  }
  const long long n = io.n;
  const Launch L = v2_launch(ctx, n);
  SolveCfg cfg = cfg_in;
  if (cfg.park_max == 0) cfg.park_max = (n >= RB_MID_MIN) ? v2::KP_SMALL_MAX : 4;
  const bool small = cfg.small != 0;   // the parked captures take 4.9 .. 10.5 KB per cacheable model, EXT_AVG x 8 B budgeted
  int *order = nullptr;
  auto layout = [&](Carve c) {
    io.state = c.take<double>(n * v2::STATE_STRIDE);
    io.keys = c.take<int>(n);
    order = c.take<int>(n);
    if (small) {
      io.order_c = c.take<int>(n);
      io.ext_off = c.take<long long>(n);
      io.ext_cap = n * v2::EXT_AVG;
      io.ext = c.take<double>(io.ext_cap);
    }
    return c.bytes;
  };
  int rc = grow(ctx->sched_buf, ctx->sched_bytes, layout(Carve{nullptr}));
  if (rc != RB_OK) return rc;
  layout(Carve{ctx->sched_buf});
  if (!ctx->sched_small) CUDA_TRY(cudaMalloc(&ctx->sched_small, 96 * sizeof(unsigned long long)));
  io.sched_small = ctx->sched_small;
  CUDA_TRY(cudaMemsetAsync(ctx->sched_small, 0, 96 * sizeof(unsigned long long), ctx->stream));
  io.sched = 1;
  k_lvg_solve_v2<<<L.blocks, L.warps_per_block * 32, L.smem, ctx->stream>>>(ctx->mol, cfg, io);
  const int tpb = 256, nb = (int)((n + tpb - 1) / tpb);
  k_sched_hist<<<nb, tpb, 0, ctx->stream>>>(io.keys, n, ctx->sched_small);
  k_sched_scan<<<1, 1, 0, ctx->stream>>>(ctx->sched_small);
  k_sched_scatter<<<nb, tpb, 0, ctx->stream>>>(io.keys, n, ctx->sched_small, order);
  io.sched = 2;
  io.order = order;
  // heaviest key first: with the cached engines in kernels of their own launch B stops where their keys begin
  io.n_parked = ctx->sched_small + (small ? 16 + cfg.park_max : 48);
  if (!small) {
    CUDA_TRY(cudaMemsetAsync(ctx->counters, 0, sizeof(unsigned long long), ctx->stream));   // queue head only
    k_lvg_solve_v2<<<L.blocks, L.warps_per_block * 32, L.smem, ctx->stream>>>(ctx->mol, cfg, io);
  } else {
    // Launch B and the engine launches work on disjoint models: each gets its own stream and queue head, so the
    // tail of one (SMs idling while its last models finish their <= 200 calls) is filled by the CTAs of the next.
    cudaStream_t s = ctx->stream;
    if (!ctx->ev_sorted) {
      CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_sorted, cudaEventDisableTiming));
      for (int j = 0; j < 6; ++j) {
        CUDA_TRY(cudaStreamCreateWithFlags(&ctx->side[j], cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_side[j], cudaEventDisableTiming));
      }
    }
    CUDA_TRY(cudaMemsetAsync(ctx->counters + 8, 0, 8 * sizeof(unsigned long long), s));
    CUDA_TRY(cudaEventRecord(ctx->ev_sorted, s));
    for (int j = 0; j < 6; ++j) {
      if (j >= 1 && j <= 3 && cfg.park_max < 7) continue;   // keys 7, 6, 5 stay in launch B for small batches
      cudaStream_t sj = ctx->side[j];
      CUDA_TRY(cudaStreamWaitEvent(sj, ctx->ev_sorted, 0));
      io.queue = 8 + j;
      switch (j) {
        case 0: k_lvg_solve_v2<<<L.blocks, L.warps_per_block * 32, L.smem, sj>>>(ctx->mol, cfg, io); break;
        case 1: k_lvg_small<7><<<ctx->sm_count, v2s::Lay<7>::WARPS * 32, small_smem<7>(), sj>>>(ctx->mol, cfg, io); break;
        case 2: k_lvg_small<6><<<ctx->sm_count, v2s::Lay<6>::WARPS * 32, small_smem<6>(), sj>>>(ctx->mol, cfg, io); break;
        case 3: k_lvg_small<5><<<ctx->sm_count, v2s::Lay<5>::WARPS * 32, small_smem<5>(), sj>>>(ctx->mol, cfg, io); break;
        case 4: k_lvg_small<4><<<ctx->sm_count, v2s::Lay<4>::WARPS * 32, small_smem<4>(), sj>>>(ctx->mol, cfg, io); break;
        default: k_lvg_small<3><<<ctx->sm_count, v2s::Lay<3>::WARPS * 32, small_smem<3>(), sj>>>(ctx->mol, cfg, io); break;
      }
      CUDA_TRY(cudaEventRecord(ctx->ev_side[j], sj));
      CUDA_TRY(cudaStreamWaitEvent(s, ctx->ev_side[j], 0));
      ctx->launches += (j > 0);
    }
    io.queue = 0;
    CUDA_TRY(cudaMemsetAsync(ctx->counters, 0, sizeof(unsigned long long), s));
    io.sched = 4;
    io.order = io.order_c;
    io.n_parked = ctx->sched_small + 49;
    io.ext = nullptr;
    k_lvg_solve_v2<<<L.blocks, L.warps_per_block * 32, L.smem, ctx->stream>>>(ctx->mol, cfg, io);
    ctx->launches += 1;
  }
  ctx->launches += 4;
  CUDA_TRY(cudaGetLastError());
  return RB_OK;
}

// The solve of io.n models: k_lvg_solve_v1, one k_lvg_solve_v2 launch, or the scheduled pipeline
static int launch_solve(rb_ctx *ctx, const SolveCfg &cfg, const rb_opts *opts, const SolveIO &io) {
  if (!use_v2(ctx, opts)) {
    const Launch L = v1_launch(ctx, io.n);
    k_lvg_solve_v1<<<L.blocks, L.warps_per_block * 32, L.smem, ctx->stream>>>(ctx->mol, cfg, io);
  } else if (cfg.sched && cfg.cache && cfg.method == RB_GEOM_LVG && io.n >= RB_SCHED_MIN) {
    return launch_solve_pipeline(ctx, cfg, io);
  } else {
    const Launch L = v2_launch(ctx, io.n);
    k_lvg_solve_v2<<<L.blocks, L.warps_per_block * 32, L.smem, ctx->stream>>>(ctx->mol, cfg, io);
  }
  return RB_OK;
}

static int check_solve(rb_ctx *ctx, int64_t n, const double *tkin, const double *dens, const double *cdmol,
                       double deltav_kms, double tbg, int geometry) {
  const int rc = check_common(ctx, deltav_kms, tbg, geometry);
  if (rc != RB_OK) return rc;
  if (n < 0 || (n > 0 && (!tkin || !dens || !cdmol))) {
    rb_set_error("rb_solve_batch: null input");
    return RB_ERR_ARG;
  }
  return RB_OK;
}

// keep_totals: a further chunk of one host call -- only the work-queue head is reset, the iteration total and the
// cache statistics keep accumulating
static int solve_batch_dev_impl(rb_ctx *ctx, const SolveCfg &cfg, const rb_opts *opts, const SolveIO &io,
                                bool keep_totals) {
  CUDA_TRY(cudaMemsetAsync(ctx->counters, 0, (keep_totals ? 1 : 8) * sizeof(unsigned long long), ctx->stream));
  const int rc = launch_solve(ctx, cfg, opts, io);
  if (rc != RB_OK) return rc;
  CUDA_TRY(cudaGetLastError());
  ctx->launches += 1;
  return RB_OK;
}

int rb_solve_batch_dev(rb_ctx *ctx, int64_t n, const double *tkin, const double *dens, const double *cdmol,
                       double deltav_kms, double tbg, int geometry, const rb_opts *opts, double *xpop,
                       double *tex, double *tau, double *surf, int32_t *niter, int32_t *status) {
  const int rc = check_solve(ctx, n, tkin, dens, cdmol, deltav_kms, tbg, geometry);
  if (rc != RB_OK || n == 0) return rc;
  CUDA_TRY(cudaSetDevice(ctx->device));
  const SolveIO io{n, tkin, dens, cdmol, xpop, tex, tau, surf, niter, status, ctx->counters};
  return solve_batch_dev_impl(ctx, make_cfg(ctx, opts, deltav_kms, tbg, geometry), opts, io, false);
}

// Host-pointer entry.  Batches of more than 2 RB_HOST_CHUNK models are solved chunk by chunk, the results of one
// chunk travelling to the host (copy stream) while the next one is being solved.  The chunks shrink geometrically
// (half of what is left, down to RB_HOST_CHUNK_MIN): large chunks keep the scheduled launches efficient, and only the
// last, smallest chunk's results travel with nothing left to hide them behind.
#ifndef RB_HOST_CHUNK
#define RB_HOST_CHUNK (1LL << 18)
#endif
#ifndef RB_HOST_CHUNK_MIN
#define RB_HOST_CHUNK_MIN (1LL << 18)
#endif

int rb_solve_batch(rb_ctx *ctx, int64_t n, const double *tkin, const double *dens, const double *cdmol,
                   double deltav_kms, double tbg, int geometry, const rb_opts *opts, double *xpop, double *tex,
                   double *tau, double *surf, int32_t *niter, int32_t *status) {
  int rc = check_solve(ctx, n, tkin, dens, cdmol, deltav_kms, tbg, geometry);
  if (rc != RB_OK || n == 0) return rc;
  CUDA_TRY(cudaSetDevice(ctx->device));
  const int nl = ctx->mol.nlev, nn = ctx->mol.nline, np = ctx->mol.npart;
  double *d_t, *d_c, *d_d, *d_x, *d_tex, *d_tau, *d_s;
  int32_t *d_it, *d_st;
  auto layout = [&](Carve c) {
    d_t = c.take<double>(n);
    d_c = c.take<double>(n);
    d_d = c.take<double>(n * np);
    d_x = xpop ? c.take<double>(n * nl) : nullptr;
    d_tex = tex ? c.take<double>(n * nn) : nullptr;
    d_tau = tau ? c.take<double>(n * nn) : nullptr;
    d_s = surf ? c.take<double>(n * nn) : nullptr;
    d_it = c.take<int32_t>(n);
    d_st = c.take<int32_t>(n);
    return c.bytes;
  };
  rc = ensure_scratch(ctx, layout(Carve{nullptr}));
  if (rc != RB_OK) return rc;
  layout(Carve{ctx->scratch});
  cudaStream_t s = ctx->stream;
  CUDA_TRY(cudaMemcpyAsync(d_t, tkin, n * sizeof(double), cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaMemcpyAsync(d_c, cdmol, n * sizeof(double), cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaMemcpyAsync(d_d, dens, (size_t)n * np * sizeof(double), cudaMemcpyHostToDevice, s));
  std::vector<int64_t> c_off, c_len;
  if (n > 2 * RB_HOST_CHUNK) {
    int64_t left = n;
    while (left > 0) {
      int64_t m = RB_HOST_CHUNK_MIN;
      while (2 * m <= left / 2) m *= 2;          // largest power of two <= left / 2 ...
      if (left < 2 * RB_HOST_CHUNK_MIN) m = left;   // ... and the remainder in one piece
      m = std::min<int64_t>(m, RB_PIPE_MAX);
      c_off.push_back(n - left);
      c_len.push_back(m);
      left -= m;
    }
  } else {
    c_off.push_back(0);
    c_len.push_back(n);
  }
  const int64_t nchunk = (int64_t)c_len.size();
  if (nchunk > 1 && !ctx->copy_stream) CUDA_TRY(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  while (nchunk > 1 && (int64_t)ctx->chunk_done.size() < nchunk) {
    cudaEvent_t ev;
    CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    ctx->chunk_done.push_back(ev);
  }
  const SolveCfg cfg = make_cfg(ctx, opts, deltav_kms, tbg, geometry);
  const SolveIO io{n, d_t, d_d, d_c, d_x, d_tex, d_tau, d_s, d_it, d_st, ctx->counters};
  auto solve_chunk = [&](int64_t k) {
    return solve_batch_dev_impl(ctx, cfg, opts, slice(ctx, io, c_off[k], c_len[k]), k > 0);
  };
  rc = solve_chunk(0);
  if (rc != RB_OK) return rc;
  for (int64_t k = 0; k < nchunk; ++k) {
    const int64_t o = c_off[k], m = c_len[k];
    cudaStream_t cs = s;
    if (nchunk > 1) {
      // chunk k is queued: mark its end, queue chunk k + 1 behind it, then fetch chunk k on the copy stream
      CUDA_TRY(cudaEventRecord(ctx->chunk_done[k], s));
      if (k + 1 < nchunk) {
        rc = solve_chunk(k + 1);
        if (rc != RB_OK) return rc;
      }
      cs = ctx->copy_stream;
      CUDA_TRY(cudaStreamWaitEvent(cs, ctx->chunk_done[k], 0));
    }
    if (xpop) CUDA_TRY(cudaMemcpyAsync(xpop + o * nl, d_x + o * nl, (size_t)m * nl * sizeof(double), cudaMemcpyDeviceToHost, cs));
    if (tex) CUDA_TRY(cudaMemcpyAsync(tex + o * nn, d_tex + o * nn, (size_t)m * nn * sizeof(double), cudaMemcpyDeviceToHost, cs));
    if (tau) CUDA_TRY(cudaMemcpyAsync(tau + o * nn, d_tau + o * nn, (size_t)m * nn * sizeof(double), cudaMemcpyDeviceToHost, cs));
    if (surf) CUDA_TRY(cudaMemcpyAsync(surf + o * nn, d_s + o * nn, (size_t)m * nn * sizeof(double), cudaMemcpyDeviceToHost, cs));
    if (niter) CUDA_TRY(cudaMemcpyAsync(niter + o, d_it + o, m * sizeof(int32_t), cudaMemcpyDeviceToHost, cs));
    if (status) CUDA_TRY(cudaMemcpyAsync(status + o, d_st + o, m * sizeof(int32_t), cudaMemcpyDeviceToHost, cs));
  }
  if (nchunk > 1) CUDA_TRY(cudaStreamSynchronize(ctx->copy_stream));
  return read_counters(ctx);
}

struct rb_srcset {
  rb_ctx *ctx = nullptr;           // identity check only; never dereferenced after creation (the set may outlive it)
  int device = 0;
  int ncomp = 1, nsrc = 0;
  rb_source *d = nullptr;          // device table
  std::vector<rb_source> h;        // host copy (argument checks; row 0 drives the single-source pipeline)
};

static int check_source(const rb_ctx *ctx, const rb_source &S) {
  if (S.obs.nobs < 1 || S.obs.nobs > RB_MAX_OBS) {
    rb_set_error("rb_lnprob: nobs must be in 1..RB_MAX_OBS");
    return RB_ERR_ARG;
  }
  for (int i = 0; i < S.obs.nobs; ++i)
    if (S.obs.jup[i] < 1 || S.obs.jup[i] > ctx->mol.nline) {
      rb_set_error("rb_lnprob: Jup outside the molecule's line list");
      return RB_ERR_ARG;
    }
  if (!(S.tbg > 0.0)) {
    rb_set_error("deltav and tbg must be positive");
    return RB_ERR_ARG;
  }
  return RB_OK;
}

static int check_lnprob(const rb_ctx *ctx, int64_t n, const double *P, const double *lnp) {
  if (!ctx) {
    rb_set_error("null context");
    return RB_ERR_ARG;
  }
  if (n < 0 || (n > 0 && (!P || !lnp))) {
    rb_set_error("rb_lnprob: null argument");
    return RB_ERR_ARG;
  }
  return RB_OK;
}

// lnprob of n walkers against the device table d_srcs (row src_id[i], or row 0); h0 = host copy of row 0.
static int lnprob_core(rb_ctx *ctx, int ncomp, int64_t n, const double *P, const rb_source *d_srcs, int nsrc,
                       const rb_source &h0, const int *src_id, const rb_opts *opts, double *lnp) {
  int rc = check_lnprob(ctx, n, P, lnp);
  if (rc != RB_OK) return rc;
  if (!ctx->ln_partners_ok) {
    // the drivers set {'oH2', 'pH2'} (emcee_radex.py:122-124), which pyradex folds into H2 when the file has that
    // partner (core.py:551-556); a file with neither has all-zero colliders there (ValueError)
    rb_set_error("rb_lnprob: the molecular file has no H2 / p-H2 / o-H2 collision partner");
    return RB_ERR_ARG;
  }
  if (n == 0) return RB_OK;
  CUDA_TRY(cudaSetDevice(ctx->device));
  const SolveCfg cfg = make_cfg(ctx, opts, 1.0, h0.tbg, RB_GEOM_LVG);  // deltav=1 km/s, LVG (emcee_radex.py:108-117)
  CUDA_TRY(cudaMemsetAsync(ctx->counters, 0, 8 * sizeof(unsigned long long), ctx->stream));
  LnprobIO io;
  memset(&io, 0, sizeof(io));
  io.n = n;
  io.P = P;
  io.lnp = lnp;
  io.srcs = d_srcs;
  io.src_id = (nsrc > 1) ? src_id : nullptr;
  io.counters = ctx->counters;
  if (lnprob_pipelined(ctx, cfg, opts, nsrc, n, ncomp)) {
    // large ensembles: expand -> scheduled solve of all n x ncomp models (half-warp engine) -> combine
    const long long m = n * ncomp;
    LnprobPipe pp;
    rc = model_arrays(ctx, m, RB_MAX_OBS, &pp);
    if (rc != RB_OK) return rc;
    const int tpb = 256;
    SolveIO sio{m, pp.tkin, pp.dens, pp.cdmol, nullptr, nullptr, nullptr, nullptr, nullptr, pp.status, ctx->counters};
    observe_lines(sio, pp.obs_surf, h0.obs.nobs, h0.obs.jup);
    if (ncomp == 1)
      k_lnprob_expand<1><<<(unsigned)((n + tpb - 1) / tpb), tpb, 0, ctx->stream>>>(ctx->mol, io, pp);
    else
      k_lnprob_expand<2><<<(unsigned)((n + tpb - 1) / tpb), tpb, 0, ctx->stream>>>(ctx->mol, io, pp);
    rc = launch_solve(ctx, cfg, opts, sio);
    if (rc != RB_OK) return rc;
    const unsigned nbc = (unsigned)((n * 32 + tpb - 1) / tpb);
    if (ncomp == 1)
      k_lnprob_combine<1><<<nbc, tpb, 0, ctx->stream>>>(io, pp);
    else
      k_lnprob_combine<2><<<nbc, tpb, 0, ctx->stream>>>(io, pp);
    ctx->launches += 2;
  } else if (use_v2(ctx, opts)) {
    const Launch L = v2_launch(ctx, n);
    if (ncomp == 1)
      k_lnprob_v2<1><<<L.blocks, L.warps_per_block * 32, L.smem, ctx->stream>>>(ctx->mol, cfg, io);
    else
      k_lnprob_v2<2><<<L.blocks, L.warps_per_block * 32, L.smem, ctx->stream>>>(ctx->mol, cfg, io);
  } else {
    const Launch L = v1_launch(ctx, n);
    if (ncomp == 1)
      k_lnprob_v1<1><<<L.blocks, L.warps_per_block * 32, L.smem, ctx->stream>>>(ctx->mol, cfg, io);
    else
      k_lnprob_v1<2><<<L.blocks, L.warps_per_block * 32, L.smem, ctx->stream>>>(ctx->mol, cfg, io);
  }
  CUDA_TRY(cudaGetLastError());
  ctx->launches += 1;
  return RB_OK;
}

// rb_lnprob1/2: one source given by value.  Its device copy lives in the ctx and is refreshed only when the caller
// passes a different source than last time (a sampler passes the same one every half-step: no transfer, no sync).
static int lnprob_dev(rb_ctx *ctx, int ncomp, int64_t n, const double *P, const rb_obs *obs, const double *bounds,
                      int has_td, double t_d, double tbg, const rb_opts *opts, double *lnp) {
  int rc = check_common(ctx, 1.0, tbg, RB_GEOM_LVG);
  if (rc != RB_OK) return rc;
  if (!obs || !bounds) {
    rb_set_error("rb_lnprob: null argument");
    return RB_ERR_ARG;
  }
  rb_source S;
  memset(&S, 0, sizeof(S));
  S.obs = *obs;
  memcpy(S.bounds, bounds, sizeof(double) * 8 * ncomp);
  S.tbg = tbg;
  S.has_td = has_td;
  S.t_d = t_d;
  rc = check_source(ctx, S);
  if (rc != RB_OK) return rc;
  CUDA_TRY(cudaSetDevice(ctx->device));
  if (!ctx->src_one) CUDA_TRY(cudaMalloc(&ctx->src_one, sizeof(rb_source)));
  if (!ctx->src_one_valid || memcmp(&S, &ctx->src_one_host, sizeof(S)) != 0) {
    ctx->src_one_host = S;   // the copy reads the ctx's own (stable) host memory
    ctx->src_one_valid = true;
    CUDA_TRY(cudaMemcpyAsync(ctx->src_one, &ctx->src_one_host, sizeof(S), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  }
  return lnprob_core(ctx, ncomp, n, P, ctx->src_one, 1, S, nullptr, opts, lnp);
}

static int lnprob_host(rb_ctx *ctx, int ncomp, int64_t n, const double *P, const rb_obs *obs, const double *bounds,
                       int has_td, double t_d, double tbg, const rb_opts *opts, double *lnp, int64_t *nsolves) {
  int rc = check_lnprob(ctx, n, P, lnp);
  if (rc != RB_OK) return rc;
  if (n == 0) {
    if (nsolves) *nsolves = 0;
    return RB_OK;
  }
  CUDA_TRY(cudaSetDevice(ctx->device));
  double *d_p, *d_l;
  auto layout = [&](Carve c) {
    d_p = c.take<double>(n * 4 * ncomp);
    d_l = c.take<double>(n);
    return c.bytes;
  };
  rc = ensure_scratch(ctx, layout(Carve{nullptr}));
  if (rc != RB_OK) return rc;
  layout(Carve{ctx->scratch});
  CUDA_TRY(cudaMemcpyAsync(d_p, P, (size_t)n * 4 * ncomp * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  rc = lnprob_dev(ctx, ncomp, n, d_p, obs, bounds, has_td, t_d, tbg, opts, d_l);
  if (rc != RB_OK) return rc;
  CUDA_TRY(cudaMemcpyAsync(lnp, d_l, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  return read_counters(ctx, nsolves);
}

int rb_lnprob1(rb_ctx *ctx, int64_t n, const double *P, const rb_obs *obs, const double *bounds, double tbg,
               const rb_opts *opts, double *lnp, int64_t *nsolves) {
  return lnprob_host(ctx, 1, n, P, obs, bounds, 0, 0.0, tbg, opts, lnp, nsolves);
}

int rb_lnprob2(rb_ctx *ctx, int64_t n, const double *P, const rb_obs *obs, const double *bounds, int has_td,
               double t_d, double tbg, const rb_opts *opts, double *lnp, int64_t *nsolves) {
  return lnprob_host(ctx, 2, n, P, obs, bounds, has_td, t_d, tbg, opts, lnp, nsolves);
}

static int copy_nsolves(rb_ctx *ctx, int64_t *nsolves_dev) {
  if (nsolves_dev)
    CUDA_TRY(cudaMemcpyAsync(nsolves_dev, ctx->counters + 2, sizeof(int64_t), cudaMemcpyDeviceToDevice, ctx->stream));
  return RB_OK;
}

int rb_lnprob1_dev(rb_ctx *ctx, int64_t n, const double *P, const rb_obs *obs, const double *bounds, double tbg,
                   const rb_opts *opts, double *lnp, int64_t *nsolves_dev) {
  int rc = lnprob_dev(ctx, 1, n, P, obs, bounds, 0, 0.0, tbg, opts, lnp);
  if (rc != RB_OK || n == 0) return rc;
  return copy_nsolves(ctx, nsolves_dev);
}

int rb_lnprob2_dev(rb_ctx *ctx, int64_t n, const double *P, const rb_obs *obs, const double *bounds, int has_td,
                   double t_d, double tbg, const rb_opts *opts, double *lnp, int64_t *nsolves_dev) {
  int rc = lnprob_dev(ctx, 2, n, P, obs, bounds, has_td, t_d, tbg, opts, lnp);
  if (rc != RB_OK || n == 0) return rc;
  return copy_nsolves(ctx, nsolves_dev);
}

int rb_stretch_propose_dev(rb_ctx *ctx, int64_t ns, int32_t ndim, const double *S, int64_t nc, const double *C,
                           double a, uint64_t seed, uint64_t step, int32_t half, int64_t gid0, int64_t gid_stride,
                           double *Q, double *logfac) {
  if (!ctx || ns < 0 || nc < 1 || ndim < 1 || !S || !C || !Q || !logfac || !(a > 1.0)) {
    rb_set_error("rb_stretch_propose_dev: bad argument");
    return RB_ERR_ARG;
  }
  if (ns == 0) return RB_OK;
  CUDA_TRY(cudaSetDevice(ctx->device));
  const int tpb = 256;
  const int blocks = (int)((ns + tpb - 1) / tpb);
  k_stretch_propose<<<blocks, tpb, 0, ctx->stream>>>(ns, ndim, S, nc, C, a, seed, step, half, gid0, gid_stride, Q, logfac);
  CUDA_TRY(cudaGetLastError());
  ctx->launches += 1;
  return RB_OK;
}

int rb_stretch_accept_dev(rb_ctx *ctx, int64_t ns, int32_t ndim, double *S, double *lnp_old, const double *Q,
                          const double *lnp_new, const double *logfac, uint64_t seed, uint64_t step, int32_t half,
                          int64_t gid0, int64_t gid_stride, int64_t *naccept) {
  if (!ctx || ns < 0 || ndim < 1 || !S || !lnp_old || !Q || !lnp_new || !logfac) {
    rb_set_error("rb_stretch_accept_dev: bad argument");
    return RB_ERR_ARG;
  }
  if (ns == 0) return RB_OK;
  CUDA_TRY(cudaSetDevice(ctx->device));
  const int tpb = 256;
  const int blocks = (int)((ns + tpb - 1) / tpb);
  k_stretch_accept<<<blocks, tpb, 0, ctx->stream>>>(ns, ndim, S, lnp_old, Q, lnp_new, logfac, seed, step, half, gid0, gid_stride,
                                                    reinterpret_cast<unsigned long long *>(naccept));
  CUDA_TRY(cudaGetLastError());
  ctx->launches += 1;
  return RB_OK;
}


// ---- source sets, multi-source lnprob ---------------------------------------------------------------------------
int rb_srcset_create(rb_ctx *ctx, int32_t ncomp, int32_t nsrc, const rb_source *src, rb_srcset **out) {
  if (!ctx || !src || !out || nsrc < 1 || (ncomp != 1 && ncomp != 2)) {
    rb_set_error("rb_srcset_create: bad argument");
    return RB_ERR_ARG;
  }
  *out = nullptr;
  for (int i = 0; i < nsrc; ++i) {
    const int rc = check_source(ctx, src[i]);
    if (rc != RB_OK) return rc;
  }
  CUDA_TRY(cudaSetDevice(ctx->device));
  rb_srcset *set = new rb_srcset();
  set->ctx = ctx;
  set->device = ctx->device;
  set->ncomp = ncomp;
  set->nsrc = nsrc;
  set->h.assign(src, src + nsrc);
  if (cudaMalloc(&set->d, sizeof(rb_source) * nsrc) != cudaSuccess ||
      cudaMemcpy(set->d, set->h.data(), sizeof(rb_source) * nsrc, cudaMemcpyHostToDevice) != cudaSuccess) {
    rb_set_error("rb_srcset_create: device allocation failed");
    if (set->d) cudaFree(set->d);
    delete set;
    return RB_ERR_CUDA;
  }
  *out = set;
  return RB_OK;
}

void rb_srcset_destroy(rb_srcset *set) {
  if (!set) return;
  if (set->d) {
    cudaSetDevice(set->device);
    cudaFree(set->d);
  }
  delete set;
}

int rb_lnprob_src_dev(rb_ctx *ctx, const rb_srcset *set, int64_t n, const double *P, const int32_t *src_id,
                      const rb_opts *opts, double *lnp, int64_t *nsolves_dev) {
  if (!ctx || !set || set->ctx != ctx) {
    rb_set_error("rb_lnprob_src_dev: the source set belongs to another context");
    return RB_ERR_ARG;
  }
  if (set->nsrc > 1 && !src_id && n > 0) {
    rb_set_error("rb_lnprob_src_dev: src_id is required with more than one source");
    return RB_ERR_ARG;
  }
  int rc = lnprob_core(ctx, set->ncomp, n, P, set->d, set->nsrc, set->h[0], src_id, opts, lnp);
  if (rc != RB_OK || n == 0) return rc;
  return copy_nsolves(ctx, nsolves_dev);
}

// ---- stretch move, second form ----------------------------------------------------------------------------------
static int make_split(const rb_split *sp, int64_t gid_base, int64_t nlocal, int32_t ndim, st2::SplitDev *out) {
  if (!sp || sp->nwalkers < 2 || sp->walkers_per_source < 2 || sp->block < 2 || (sp->block & 1) ||
      sp->block > (1LL << 30) || sp->nwalkers % sp->walkers_per_source || sp->walkers_per_source % sp->block ||
      gid_base < 0 || nlocal < 0 || gid_base % sp->block || nlocal % sp->block || gid_base + nlocal > sp->nwalkers ||
      ndim < 1) {
    rb_set_error("rb_stretch: bad split (need block | walkers_per_source | nwalkers, block even, block | gid_base, nlocal)");
    return RB_ERR_ARG;
  }
  out->W = sp->walkers_per_source;
  out->B = (int)sp->block;
  int w = 1;
  while ((1LL << w) < sp->block) ++w;
  out->w = w;
  out->randomize = sp->randomize != 0;
  st2::split_key_words(sp->seed, out->k0, out->k1);
  return RB_OK;
}

// every group of the DE split has slots in every block and a complement of >= 2 walkers within its source (two distinct
// partners)
static int check_de_split(const char *who, const rb_split *split) {
  if (split->block < 3) {
    rb_set_error(std::string(who) + ": the 3-group split needs blocks of >= 3 walkers");
    return RB_ERR_ARG;
  }
  for (int g = 0; g < 3; ++g)
    if (split->walkers_per_source - (split->walkers_per_source / split->block) * st2::group_size((int)split->block, 3, g) < 2) {
      rb_set_error(std::string(who) + ": a group of the 3-group split leaves fewer than 2 walkers of its source to draw from");
      return RB_ERR_ARG;
    }
  return RB_OK;
}

static double de_gamma0(double gamma0, int ndim) { return gamma0 == 0.0 ? 2.38 / std::sqrt(2.0 * ndim) : gamma0; }

// The entry points below: argument checks (args_ok: the entry point's own arguments), the split, the device, then
// launch(sp, nslots, blocks) with blocks of 128 threads over the local slots of group g of ngroups (the stretch move: half g
// of 2)
extern "C++" {
template <typename F>
static int group_launch(const char *who, bool args_ok, rb_ctx *ctx, const rb_split *split, int32_t group, int32_t ngroups,
                        int64_t gid_base, int64_t nlocal, int32_t ndim, bool de, F launch) {
  if (!ctx || !args_ok || ngroups < 2 || group < 0 || group >= ngroups) {
    rb_set_error(std::string(who) + ": bad argument");
    return RB_ERR_ARG;
  }
  st2::SplitDev sp;
  int rc = make_split(split, gid_base, nlocal, ndim, &sp);
  if (rc != RB_OK) return rc;
  if (de && (rc = check_de_split(who, split)) != RB_OK) return rc;
  const long long nslots = nlocal / sp.B * st2::group_size(sp.B, ngroups, group);
  if (nslots == 0) return RB_OK;
  CUDA_TRY(cudaSetDevice(ctx->device));
  launch(sp, nslots, (unsigned)((nslots + 127) / 128));
  CUDA_TRY(cudaGetLastError());
  ctx->launches += 1;
  return RB_OK;
}
}

int rb_stretch_pack_dev(rb_ctx *ctx, const rb_split *split, uint64_t step, int32_t half, int64_t gid_base,
                        int64_t nlocal, int32_t ndim, const double *X, double *Chalf) {
  return group_launch("rb_stretch_pack_dev", X && Chalf, ctx, split, half, 2, gid_base, nlocal, ndim, false,
                         [&](const st2::SplitDev &sp, long long nhalf, unsigned nb) {
    st2::k_pack<<<nb, 128, 0, ctx->stream>>>(sp, nullptr, step, half, 2, gid_base, nhalf, ndim, X, Chalf);
  });
}

int rb_stretch_propose2_dev(rb_ctx *ctx, const rb_split *split, uint64_t step, int32_t half, int64_t gid_base,
                            int64_t nlocal, int32_t ndim, const double *X, const double *Call, double a, double *Q,
                            double *logfac, int32_t *src_id) {
  return group_launch("rb_stretch_propose2_dev", X && Call && Q && logfac && a > 1.0, ctx, split, half, 2, gid_base,
                         nlocal, ndim, false, [&](const st2::SplitDev &sp, long long nhalf, unsigned nb) {
    st2::k_propose2<<<nb, 128, 0, ctx->stream>>>(sp, nullptr, step, half, gid_base, nhalf, ndim, X, Call, a, split->seed,
                                                 Q, logfac, src_id);
  });
}

int rb_stretch_accept2_dev(rb_ctx *ctx, const rb_split *split, uint64_t step, int32_t half, int64_t gid_base,
                           int64_t nlocal, int32_t ndim, double *X, double *lnp, const double *Q, const double *lnp_new,
                           const double *logfac, int64_t *naccept, int64_t *nan_count) {
  return group_launch("rb_stretch_accept2_dev", X && lnp && Q && lnp_new && logfac, ctx, split, half, 2, gid_base,
                         nlocal, ndim, false, [&](const st2::SplitDev &sp, long long nhalf, unsigned nb) {
    st2::k_accept2<<<nb, 128, 0, ctx->stream>>>(sp, nullptr, step, half, 2, 0, gid_base, nhalf, ndim, X, lnp, Q, lnp_new, logfac,
                                                split->seed, reinterpret_cast<long long *>(naccept),
                                                reinterpret_cast<unsigned long long *>(nan_count), nullptr, nullptr);
  });
}

// One stretch-move step (both half-steps) on ctx->stream; the step index is *d_step + 0 (device-resident, so that the
// captured graph of one step can be replayed).
static int stretch_one_step(rb_ctx *ctx, const rb_srcset *set, const st2::SplitDev &sp, const rb_split *split, double a,
                            const rb_opts *opts, long long N, int ndim, double *X, double *lnp, long long *naccept,
                            unsigned long long *counters, double *Cbuf, double *Q, double *logfac, double *lnp_new,
                            int *src_id, unsigned long long *d_step) {
  const long long nhalf = N / 2;
  const int tpb = 128;
  const unsigned nb = (unsigned)((nhalf + tpb - 1) / tpb);
  cudaStream_t s = ctx->stream;
  for (int half = 0; half < 2; ++half) {
    st2::k_pack<<<nb, tpb, 0, s>>>(sp, d_step, 0, 1 - half, 2, 0, nhalf, ndim, X, Cbuf);
    st2::k_propose2<<<nb, tpb, 0, s>>>(sp, d_step, 0, half, 0, nhalf, ndim, X, Cbuf, a, split->seed, Q, logfac, src_id);
    int rc = lnprob_core(ctx, set->ncomp, nhalf, Q, set->d, set->nsrc, set->h[0], src_id, opts, lnp_new);
    if (rc != RB_OK) return rc;
    st2::k_accept2<<<nb, tpb, 0, s>>>(sp, d_step, 0, half, 2, 0, 0, nhalf, ndim, X, lnp, Q, lnp_new, logfac, split->seed, naccept,
                                      counters, ctx->counters + 2, counters ? counters + 1 : nullptr);
    ctx->launches += 3;
  }
  st2::k_step_inc<<<1, 1, 0, s>>>(d_step);
  ctx->launches += 1;
  CUDA_TRY(cudaGetLastError());
  return RB_OK;
}

// The same step with the second half-step proposed speculatively (stretch.cuh: k_propose_spec): one lnprob launch of
// 3 nhalf models per step.  Buffers: C1, Cold [nhalf x ndim]; Q3 [3 nhalf x ndim] = Q0 | Qa | Qb;
// L3 [3 nhalf]; logfac0, logfac1 [nhalf]; jpart, acc0 [nhalf]; the selected candidates overwrite C1 / its lnprob L3's head.
struct SpecBufs {
  double *C1, *Cold, *Q3, *L3, *logfac0, *logfac1, *Lsel;
  int *jpart, *acc0, *src3;   // src3 [3 nhalf]: source row of every candidate (several sources in one ensemble)
};
static int stretch_one_step_spec(rb_ctx *ctx, const rb_srcset *set, const st2::SplitDev &sp, const rb_split *split, double a,
                                 const rb_opts *opts, long long N, int ndim, double *X, double *lnp, long long *naccept,
                                 unsigned long long *counters, const SpecBufs &b, unsigned long long *d_step) {
  const long long nhalf = N / 2;
  const int tpb = 128;
  const unsigned nb = (unsigned)((nhalf + tpb - 1) / tpb);
  cudaStream_t s = ctx->stream;
  double *Q0 = b.Q3, *Qa = b.Q3 + nhalf * ndim, *Qb = b.Q3 + 2 * nhalf * ndim;
  st2::k_pack<<<nb, tpb, 0, s>>>(sp, d_step, 0, 1, 2, 0, nhalf, ndim, X, b.C1);
  int *src3 = (set->nsrc > 1) ? b.src3 : nullptr;
  st2::k_propose2<<<nb, tpb, 0, s>>>(sp, d_step, 0, 0, 0, nhalf, ndim, X, b.C1, a, split->seed, Q0, b.logfac0, src3);
  st2::k_pack<<<nb, tpb, 0, s>>>(sp, d_step, 0, 0, 2, 0, nhalf, ndim, X, b.Cold);
  st2::k_propose_spec<<<nb, tpb, 0, s>>>(sp, d_step, 0, 0, nhalf, ndim, X, b.Cold, Q0, a, split->seed, Qa, Qb, b.logfac1, b.jpart,
                                         src3 ? src3 + nhalf : nullptr, src3 ? src3 + 2 * nhalf : nullptr);
  int rc = lnprob_core(ctx, set->ncomp, 3 * nhalf, b.Q3, set->d, set->nsrc, set->h[0], src3, opts, b.L3);
  if (rc != RB_OK) return rc;
  st2::k_accept2<<<nb, tpb, 0, s>>>(sp, d_step, 0, 0, 2, 0, 0, nhalf, ndim, X, lnp, Q0, b.L3, b.logfac0, split->seed, naccept, counters,
                                    ctx->counters + 2, counters ? counters + 1 : nullptr, b.acc0);
  st2::k_select_spec<<<nb, tpb, 0, s>>>(nhalf, ndim, b.acc0, b.jpart, Qa, Qb, b.L3 + nhalf, b.L3 + 2 * nhalf, b.C1, b.Lsel);
  st2::k_accept2<<<nb, tpb, 0, s>>>(sp, d_step, 0, 1, 2, 0, 0, nhalf, ndim, X, lnp, b.C1, b.Lsel, b.logfac1, split->seed, naccept,
                                    counters, nullptr, nullptr);
  st2::k_step_inc<<<1, 1, 0, s>>>(d_step);
  ctx->launches += 9;
  CUDA_TRY(cudaGetLastError());
  return RB_OK;
}

// ---- moves: differential evolution, the k-group accept, the move schedule --------------------------------------------
int rb_de_propose_dev(rb_ctx *ctx, const rb_split *split, uint64_t step, int32_t group, int64_t gid_base, int64_t nlocal,
                      int32_t ndim, const double *X, const double *Xall, double gamma0, double sigma, double *Q,
                      int32_t *src_id) {
  const bool ok = X && Xall && Q && std::isfinite(gamma0) && gamma0 >= 0.0 && std::isfinite(sigma) && sigma >= 0.0;
  const double g0 = de_gamma0(gamma0, ndim);
  return group_launch("rb_de_propose_dev", ok, ctx, split, group, 3, gid_base, nlocal, ndim, true,
                      [&](const st2::SplitDev &sp, long long nslots, unsigned nb) {
    st2::k_de_propose<<<nb, 128, 0, ctx->stream>>>(sp, nullptr, step, group, gid_base, nslots, ndim, X, Xall, g0, sigma,
                                                   split->seed, Q, src_id);
  });
}

int rb_group_accept_dev(rb_ctx *ctx, const rb_split *split, int32_t kind, uint64_t step, int32_t group, int32_t ngroups,
                        int64_t gid_base, int64_t nlocal, int32_t ndim, double *X, double *lnp, const double *Q,
                        const double *lnp_new, const double *logfac, int64_t *naccept, int64_t *nan_count) {
  // the random streams have room for two groups per step (stretch: counter 2 step + group) and three (DE: 4 step + group)
  const bool ok = X && lnp && Q && lnp_new &&
                  ((kind == RB_MOVE_STRETCH && ngroups == 2) || (kind == RB_MOVE_DE && ngroups == 3));
  return group_launch("rb_group_accept_dev", ok, ctx, split, group, ngroups, gid_base, nlocal, ndim, kind == RB_MOVE_DE,
                      [&](const st2::SplitDev &sp, long long nslots, unsigned nb) {
    st2::k_accept2<<<nb, 128, 0, ctx->stream>>>(sp, nullptr, step, group, ngroups, kind == RB_MOVE_DE ? 1 : 0, gid_base, nslots,
                                                ndim, X, lnp, Q, lnp_new, logfac, split->seed,
                                                reinterpret_cast<long long *>(naccept),
                                                reinterpret_cast<unsigned long long *>(nan_count), nullptr, nullptr);
  });
}

int rb_move_schedule(uint64_t seed, uint64_t step0, int64_t nsteps, const double *weights, int32_t nmoves, int32_t *out) {
  if (nsteps < 0 || nmoves < 1 || nmoves > RB_MAX_MOVES || !weights || (nsteps > 0 && !out)) {
    rb_set_error("rb_move_schedule: bad argument");
    return RB_ERR_ARG;
  }
  double tot = 0.0;
  for (int m = 0; m < nmoves; ++m) {
    if (!(weights[m] >= 0.0) || !std::isfinite(weights[m])) {
      rb_set_error("rb_move_schedule: move weights must be finite and >= 0");
      return RB_ERR_ARG;
    }
    tot += weights[m];
  }
  if (!(tot > 0.0) || !std::isfinite(tot)) {
    rb_set_error("rb_move_schedule: the move weights must have a positive, finite sum");
    return RB_ERR_ARG;
  }
  double cum[RB_MAX_MOVES], acc = 0.0;
  for (int m = 0; m < nmoves; ++m) {
    acc += weights[m];
    cum[m] = acc / tot;
  }
  cum[nmoves - 1] = 1.0;
  const uint32_t k0 = (uint32_t)seed ^ 0x4D4F5645u, k1 = (uint32_t)(seed >> 32) ^ 0x53434844u;   // 'MOVE', 'SCHD'
  for (int64_t k = 0; k < nsteps; ++k) {
    const uint64_t step = step0 + (uint64_t)k;
    uint32_t c[4] = {(uint32_t)step, (uint32_t)(step >> 32), 0u, 0u};
    philox4x32_10(c, k0, k1);
    const double u = u01(c[0], c[1]);
    int m = 0;
    while (m < nmoves - 1 && !(u < cum[m])) ++m;
    out[k] = m;
  }
  return RB_OK;
}

// One DE step (three sub-steps) on ctx->stream; step index *d_step, as stretch_one_step
static int de_one_step(rb_ctx *ctx, const rb_srcset *set, const st2::SplitDev &sp, const rb_split *split, double gamma0,
                       double sigma, const rb_opts *opts, long long N, int ndim, double *X, double *lnp, long long *naccept,
                       unsigned long long *counters, double *Q, double *lnp_new, int *src_id, unsigned long long *d_step) {
  const int tpb = 128;
  cudaStream_t s = ctx->stream;
  for (int g = 0; g < 3; ++g) {
    const long long ns = N / sp.B * st2::group_size(sp.B, 3, g);
    if (ns == 0) continue;
    const unsigned nb = (unsigned)((ns + tpb - 1) / tpb);
    st2::k_de_propose<<<nb, tpb, 0, s>>>(sp, d_step, 0, g, 0, ns, ndim, X, X, gamma0, sigma, split->seed, Q, src_id);
    int rc = lnprob_core(ctx, set->ncomp, ns, Q, set->d, set->nsrc, set->h[0], src_id, opts, lnp_new);
    if (rc != RB_OK) return rc;
    st2::k_accept2<<<nb, tpb, 0, s>>>(sp, d_step, 0, g, 3, 1, 0, ns, ndim, X, lnp, Q, lnp_new, nullptr, split->seed, naccept,
                                      counters, ctx->counters + 2, counters ? counters + 1 : nullptr);
    ctx->launches += 2;
  }
  st2::k_step_inc<<<1, 1, 0, s>>>(d_step);
  ctx->launches += 1;
  CUDA_TRY(cudaGetLastError());
  return RB_OK;
}

static int moves_run_impl(const char *who, rb_ctx *ctx, const rb_srcset *set, const rb_split *split, const rb_move *moves,
                          int32_t nmoves, uint64_t step0, int64_t nsteps, const rb_opts *opts, double *X, double *lnp,
                          int64_t *naccept, int64_t *counters, int32_t thin, double *chain, double *lnp_chain);

// CUDA's legacy default stream (what PyTorch's default stream is) cannot be captured: the loop then runs on the ctx's own
// stream, ordered after the work already queued on the caller's stream and before what it queues next
static int moves_run(const char *who, rb_ctx *ctx, const rb_srcset *set, const rb_split *split, const rb_move *moves,
                     int32_t nmoves, uint64_t step0, int64_t nsteps, const rb_opts *opts, double *X, double *lnp,
                     int64_t *naccept, int64_t *counters, int32_t thin, double *chain, double *lnp_chain) {
  if (!ctx) {
    rb_set_error(std::string(who) + ": bad argument");
    return RB_ERR_ARG;
  }
  cudaStream_t caller = ctx->stream;
  if (caller != nullptr && caller != cudaStreamLegacy)
    return moves_run_impl(who, ctx, set, split, moves, nmoves, step0, nsteps, opts, X, lnp, naccept, counters, thin, chain,
                          lnp_chain);
  CUDA_TRY(cudaSetDevice(ctx->device));
  if (!ctx->ev_samp) CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_samp, cudaEventDisableTiming));
  CUDA_TRY(cudaEventRecord(ctx->ev_samp, caller));
  CUDA_TRY(cudaStreamWaitEvent(ctx->own_stream, ctx->ev_samp, 0));
  ctx->stream = ctx->own_stream;
  const int rc = moves_run_impl(who, ctx, set, split, moves, nmoves, step0, nsteps, opts, X, lnp, naccept, counters, thin,
                                chain, lnp_chain);
  ctx->stream = caller;
  CUDA_TRY(cudaEventRecord(ctx->ev_samp, ctx->own_stream));
  CUDA_TRY(cudaStreamWaitEvent(caller, ctx->ev_samp, 0));
  return rc;
}

int rb_stretch_run_dev(rb_ctx *ctx, const rb_srcset *set, const rb_split *split, double a, uint64_t step0,
                       int64_t nsteps, const rb_opts *opts, double *X, double *lnp, int64_t *naccept,
                       int64_t *counters, int32_t thin, double *chain, double *lnp_chain) {
  const rb_move stretch = {RB_MOVE_STRETCH, 0, a, 0.0, 0.0, 1.0};
  return moves_run("rb_stretch_run_dev", ctx, set, split, &stretch, 1, step0, nsteps, opts, X, lnp, naccept, counters, thin,
                   chain, lnp_chain);
}

int rb_moves_run_dev(rb_ctx *ctx, const rb_srcset *set, const rb_split *split, const rb_move *moves, int32_t nmoves,
                     uint64_t step0, int64_t nsteps, const rb_opts *opts, double *X, double *lnp, int64_t *naccept,
                     int64_t *counters, int32_t thin, double *chain, double *lnp_chain) {
  return moves_run("rb_moves_run_dev", ctx, set, split, moves, nmoves, step0, nsteps, opts, X, lnp, naccept, counters, thin,
                   chain, lnp_chain);
}

static int moves_run_impl(const char *who, rb_ctx *ctx, const rb_srcset *set, const rb_split *split, const rb_move *moves,
                          int32_t nmoves, uint64_t step0, int64_t nsteps, const rb_opts *opts, double *X, double *lnp,
                          int64_t *naccept, int64_t *counters, int32_t thin, double *chain, double *lnp_chain) {
  bool ok = ctx && set && set->ctx == ctx && split && X && lnp && nsteps >= 0 && thin >= 1 && moves && nmoves >= 1 &&
            nmoves <= RB_MAX_MOVES;
  bool has_de = false;
  for (int m = 0; ok && m < nmoves; ++m) {
    const rb_move &mv = moves[m];
    if (mv.kind == RB_MOVE_STRETCH) ok = mv.a > 1.0;
    else if (mv.kind == RB_MOVE_DE)
      ok = std::isfinite(mv.gamma0) && mv.gamma0 >= 0.0 && std::isfinite(mv.sigma) && mv.sigma >= 0.0;
    else ok = false;
    has_de |= mv.kind == RB_MOVE_DE;
  }
  if (!ok) {
    rb_set_error(std::string(who) + ": bad argument");
    return RB_ERR_ARG;
  }
  const long long N = split->nwalkers;
  const int ndim = 4 * set->ncomp;
  st2::SplitDev sp;
  int rc = make_split(split, 0, N, ndim, &sp);
  if (rc != RB_OK) return rc;
  if (N / split->walkers_per_source != set->nsrc) {
    rb_set_error(std::string(who) + ": nwalkers / walkers_per_source must equal the number of sources");
    return RB_ERR_ARG;
  }
  if (has_de && (rc = check_de_split(who, split)) != RB_OK) return rc;
  double weights[RB_MAX_MOVES];
  for (int m = 0; m < nmoves; ++m) weights[m] = moves[m].weight;
  std::vector<int32_t> sched((size_t)nsteps);
  rc = rb_move_schedule(split->seed, step0, nsteps, weights, nmoves, sched.data());
  if (rc != RB_OK) return rc;
  if (nsteps == 0) return RB_OK;
  CUDA_TRY(cudaSetDevice(ctx->device));
  const long long nhalf = N / 2;   // also >= every group of the 3-group split
  // speculative second half-step while the three candidates of every slot can run side by side (one warp each; measured
  // on B200, walker-steps/s with / without: 100 walkers 2.57e5 / 1.35e5, 800: 1.28e6 / 9.4e5, 1600: 1.74e6 / 1.51e6,
  // 3200: 2.22e6 / 2.38e6; two components, 800 walkers: 3.97e5 / 2.54e5), unless rb_opts.spec_half says otherwise
  const rb_opts od = resolve_opts(opts);
  const bool spec_fits = od.spec_half > 0 || (od.spec_half == 0 && 3 * nhalf <= (long long)RB_SPEC_WARPS_PER_SM * ctx->sm_count);
  double *Cbuf, *Q, *logfac, *lnp_new;
  int *src_id;
  unsigned long long *d_step;
  SpecBufs sb{};
  auto layout = [&](Carve c) {
    Cbuf = c.take<double>(nhalf * ndim);
    Q = c.take<double>(nhalf * ndim);
    logfac = c.take<double>(nhalf);
    lnp_new = c.take<double>(nhalf);
    src_id = c.take<int>(nhalf);
    d_step = c.take<unsigned long long>(1);
    if (spec_fits) {
      sb.C1 = c.take<double>(nhalf * ndim);
      sb.Cold = c.take<double>(nhalf * ndim);
      sb.Q3 = c.take<double>(3 * nhalf * ndim);
      sb.L3 = c.take<double>(3 * nhalf);
      sb.logfac0 = c.take<double>(nhalf);
      sb.logfac1 = c.take<double>(nhalf);
      sb.Lsel = c.take<double>(nhalf);
      sb.jpart = c.take<int>(nhalf);
      sb.acc0 = c.take<int>(nhalf);
      sb.src3 = c.take<int>(3 * nhalf);
    }
    return c.bytes;
  };
  const size_t need = layout(Carve{nullptr});
  if (need > ctx->samp_bytes)   // the captured steps hold pointers into the old buffer
    for (cudaGraphExec_t &g : ctx->samp_graph)
      if (g) {
        cudaGraphExecDestroy(g);
        g = nullptr;
      }
  rc = grow(ctx->samp_buf, ctx->samp_bytes, need);
  if (rc != RB_OK) return rc;
  layout(Carve{ctx->samp_buf});
  cudaStream_t s = ctx->stream;
  const unsigned long long step0_ = step0;
  CUDA_TRY(cudaMemcpyAsync(d_step, &step0_, sizeof(step0_), cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaStreamSynchronize(s));   // step0_ lives on this stack frame
  unsigned long long *cnt = reinterpret_cast<unsigned long long *>(counters);
  long long *nacc = reinterpret_cast<long long *>(naccept);
  int *srcp = (set->nsrc > 1) ? src_id : nullptr;
  bool spec = false;   // decided below, once it is known that the half-ensemble runs as one fused launch
  auto step_once = [&](int m) {
    const rb_move &mv = moves[m];
    if (mv.kind == RB_MOVE_DE)
      return de_one_step(ctx, set, sp, split, de_gamma0(mv.gamma0, ndim), mv.sigma, opts, N, ndim, X, lnp, nacc, cnt, Q,
                         lnp_new, srcp, d_step);
    if (spec) return stretch_one_step_spec(ctx, set, sp, split, mv.a, opts, N, ndim, X, lnp, nacc, cnt, sb, d_step);
    return stretch_one_step(ctx, set, sp, split, mv.a, opts, N, ndim, X, lnp, nacc, cnt, Cbuf, Q, logfac, lnp_new, srcp,
                            d_step);
  };
  auto store = [&](int64_t k) -> int {   // state after step k (0-based) -> chain slot
    if ((k + 1) % thin) return RB_OK;
    const int64_t slot = (k + 1) / thin - 1;
    if (chain)
      CUDA_TRY(cudaMemcpyAsync(chain + (size_t)slot * N * ndim, X, (size_t)N * ndim * sizeof(double), cudaMemcpyDeviceToDevice, s));
    if (lnp_chain)
      CUDA_TRY(cudaMemcpyAsync(lnp_chain + (size_t)slot * N, lnp, (size_t)N * sizeof(double), cudaMemcpyDeviceToDevice, s));
    return RB_OK;
  };
  // A half-ensemble that fits one fused lnprob launch is latency-bound (config 1: 50 models per half-step): the step of
  // every move of the list is captured once and replayed.  The key holds every argument the captured launches depend on.
  const SolveCfg cfg = make_cfg(ctx, opts, 1.0, set->h[0].tbg, RB_GEOM_LVG);
  const bool fused = !lnprob_pipelined(ctx, cfg, opts, set->nsrc, nhalf, set->ncomp);
  // (forced speculation on a large ensemble: the 1.5 N candidates must still be one fused launch, not the pipeline)
  spec = fused && spec_fits && !lnprob_pipelined(ctx, cfg, opts, set->nsrc, 3 * nhalf, set->ncomp);
  if (!(fused && nsteps >= 3)) {
    for (int64_t k = 0; k < nsteps; ++k) {
      rc = step_once(sched[k]);
      if (rc != RB_OK) return rc;
      rc = store(k);
      if (rc != RB_OK) return rc;
    }
    return RB_OK;
  }
  struct Key {
    const void *set, *X, *lnp, *naccept, *counters, *buf, *stream;
    rb_split split;
    rb_opts opts;
    rb_move move;
  };
  std::vector<Key> keys((size_t)nmoves);
  int ready[RB_MAX_MOVES] = {}, ran[RB_MAX_MOVES] = {};   // graph m matches its key / ran un-captured in this call
  long long per_step[RB_MAX_MOVES];
  for (int m = 0; m < nmoves; ++m) {
    Key &key = keys[m];
    memset(&key, 0, sizeof(key));
    key.set = set; key.X = X; key.lnp = lnp; key.naccept = naccept; key.counters = counters; key.buf = ctx->samp_buf;
    key.stream = s; key.split = *split; key.opts = od;
    key.move.kind = moves[m].kind;
    if (moves[m].kind == RB_MOVE_DE) {
      key.move.gamma0 = moves[m].gamma0;
      key.move.sigma = moves[m].sigma;
    } else {
      key.move.a = moves[m].a;
    }
    const unsigned char *kb = reinterpret_cast<const unsigned char *>(&key);
    ready[m] = ctx->samp_graph[m] && ctx->samp_key[m].size() == sizeof(key) &&
               memcmp(ctx->samp_key[m].data(), kb, sizeof(key)) == 0;
    // pack, propose2, lnprob, accept2 per half-step + the step counter (speculative: 9 as well); DE: propose, lnprob,
    // accept per non-empty group + the step counter
    per_step[m] = 9;
    if (moves[m].kind == RB_MOVE_DE) {
      per_step[m] = 1;
      for (int g = 0; g < 3; ++g) per_step[m] += st2::group_size(sp.B, 3, g) ? 3 : 0;
    }
  }
  for (int64_t k = 0; k < nsteps; ++k) {
    const int m = sched[k];
    if (!ready[m]) {
      if (!ran[m]) {   // un-captured first step of the move: every lazy allocation happens here
        if (ctx->samp_graph[m]) {
          cudaGraphExecDestroy(ctx->samp_graph[m]);
          ctx->samp_graph[m] = nullptr;
        }
        ran[m] = 1;
        rc = step_once(m);
        if (rc != RB_OK) return rc;
        rc = store(k);
        if (rc != RB_OK) return rc;
        continue;
      }
      cudaGraph_t g = nullptr;
      const long long launches_before = ctx->launches;
      CUDA_TRY(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
      rc = step_once(m);
      cudaError_t ce = cudaStreamEndCapture(s, &g);
      ctx->launches = launches_before;   // nothing ran
      if (rc != RB_OK || ce != cudaSuccess || !g) {
        if (g) cudaGraphDestroy(g);
        if (rc == RB_OK) rb_set_error(std::string(who) + ": graph capture failed: " + cudaGetErrorString(ce));
        return rc != RB_OK ? rc : RB_ERR_CUDA;
      }
      ce = cudaGraphInstantiate(&ctx->samp_graph[m], g, 0);
      cudaGraphDestroy(g);
      if (ce != cudaSuccess) {
        ctx->samp_graph[m] = nullptr;
        rb_set_error(std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ce));
        return RB_ERR_CUDA;
      }
      const unsigned char *kb = reinterpret_cast<const unsigned char *>(&keys[m]);
      ctx->samp_key[m].assign(kb, kb + sizeof(Key));
      ready[m] = 1;
    }
    CUDA_TRY(cudaGraphLaunch(ctx->samp_graph[m], s));
    ctx->launches += per_step[m];
    rc = store(k);
    if (rc != RB_OK) return rc;
  }
  return RB_OK;
}

#ifdef V2S_TIMING
int rb_debug_timing(unsigned long long *out64, int reset) {
  cudaDeviceSynchronize();
  if (out64) cudaMemcpyFromSymbol(out64, g_tm, sizeof(unsigned long long) * 64);
  if (out64) cudaMemcpyFromSymbol(out64 + 64, v2::g_tv, sizeof(unsigned long long) * 60);
  if (reset) {
    static unsigned long long z[64];
    cudaMemcpyToSymbol(g_tm, z, sizeof(z));
    cudaMemcpyToSymbol(v2::g_tv, z, sizeof(unsigned long long) * 60);
  }
  return 0;
}
#endif

int rb_fp64_peak(rb_ctx *ctx, double *tflops) {
  if (!ctx || !tflops) return RB_ERR_ARG;
  CUDA_TRY(cudaSetDevice(ctx->device));
  const int blocks = ctx->sm_count * 8, tpb = 256, iters = 4096;
  double *d = nullptr;
  CUDA_TRY(cudaMalloc(&d, (size_t)blocks * tpb * sizeof(double)));
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  float best = 1e30f;
  for (int rep = 0; rep < 5; ++rep) {
    CUDA_TRY(cudaEventRecord(e0, ctx->stream));
    k_fp64_peak<<<blocks, tpb, 0, ctx->stream>>>(d, iters);
    CUDA_TRY(cudaEventRecord(e1, ctx->stream));
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms = 0;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    if (rep > 0 && ms < best) best = ms;
  }
  ctx->launches += 5;
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  const double flops = 2.0 * 8 * 16 * (double)iters * (double)blocks * tpb;
  *tflops = flops / (best * 1e-3) * 1e-12;
  return RB_OK;
}

// ---- chain statistics (chain_stats.cuh) --------------------------------------------------------------------------
// Argument checks first (RB_ERR_ARG), then the device (RB_ERR_CUDA), then the context.
static int chain_view(const char *who, const rb_chain_view *in, int32_t nsrc, cs::View *v) {
  std::string e;
  if (!in) e = "null view";
  else if (in->nchunks < 0 || in->nchunks > RB_MAX_CHUNKS) e = "nchunks must be in 0..RB_MAX_CHUNKS";
  else if (in->ndim < 1 || in->ndim > RB_CHAIN_MAX_DIM) e = "ndim must be in 1..RB_CHAIN_MAX_DIM";
  else if (in->thin < 1) e = "thin must be positive";
  else if (in->discard < 0 || in->nlocal < 0 || in->gid_base < 0 || in->walkers_per_source < 1) e = "bad walker layout";
  if (e.empty()) {
    long long t = 0;
    for (int c = 0; c < in->nchunks && e.empty(); ++c) {
      if (in->steps[c] < 0 || (in->steps[c] > 0 && in->nlocal > 0 && !in->chunk[c])) e = "bad chunk";
      t += in->steps[c];
    }
    v->nchunks = in->nchunks;
    v->ndim = in->ndim;
    v->nlocal = in->nlocal;
    v->gid_base = in->gid_base;
    v->W = in->walkers_per_source;
    v->first = in->discard + in->thin - 1;
    v->thin = in->thin;
    v->nsel = t > v->first ? (t - v->first + v->thin - 1) / v->thin : 0;
    v->src0 = in->gid_base / in->walkers_per_source;
    long long acc = 0;
    for (int c = 0; c < RB_MAX_CHUNKS; ++c) {
      v->chunk[c] = c < in->nchunks ? in->chunk[c] : nullptr;
      v->start[c] = acc;
      if (c < in->nchunks) acc += in->steps[c];
    }
    v->start[RB_MAX_CHUNKS] = acc;
    if (e.empty() && in->nlocal > 0 && (in->gid_base + in->nlocal - 1) / in->walkers_per_source >= nsrc)
      e = "nsrc does not cover the rank's walkers";
  }
  if (!e.empty()) {
    rb_set_error(std::string(who) + ": " + e);
    return RB_ERR_ARG;
  }
  return RB_OK;
}

static int chain_device(const char *who, rb_ctx *ctx) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    rb_set_error(std::string(who) + ": no CUDA device");
    return RB_ERR_CUDA;
  }
  if (!ctx) {
    rb_set_error(std::string(who) + ": null context");
    return RB_ERR_ARG;
  }
  CUDA_TRY(cudaSetDevice(ctx->device));
  return RB_OK;
}

static long long local_sources(const cs::View &v) {
  return v.nlocal ? (v.gid_base + v.nlocal - 1) / v.W - v.src0 + 1 : 0;
}

int rb_chain_hist_dev(rb_ctx *ctx, const rb_chain_view *view, int32_t nsrc, int32_t ncol, const int32_t *col_i,
                      const int32_t *col_j, int32_t pass, int32_t nprefix, const uint64_t *prefix, uint64_t *counts,
                      uint64_t *nan_counts) {
  static const char *who = "rb_chain_hist_dev";
  cs::View v;
  int rc = chain_view(who, view, nsrc, &v);
  if (rc != RB_OK) return rc;
  cs::Cols cols;
  std::string e;
  if (ncol < 1 || ncol > RB_CHAIN_MAX_COLS || !col_i || !col_j) e = "ncol must be in 1..RB_CHAIN_MAX_COLS";
  else if (pass < 0 || pass > 7) e = "pass must be in 0..7";
  else if (nprefix < 1 || ncol * nprefix > RB_CHAIN_MAX_HIST || (pass == 0 && nprefix != 1)) e = "bad nprefix";
  else if (!prefix || !counts) e = "null output";
  for (int c = 0; e.empty() && c < ncol; ++c) {
    if (col_i[c] < 0 || col_i[c] >= v.ndim || col_j[c] < -1 || col_j[c] >= v.ndim) e = "column outside [0, ndim)";
    cols.i[c] = col_i[c];
    cols.j[c] = col_j[c];
  }
  cols.n = ncol;
  if (!e.empty()) {
    rb_set_error(std::string(who) + ": " + e);
    return RB_ERR_ARG;
  }
  if ((rc = chain_device(who, ctx)) != RB_OK) return rc;
  const long long nls = local_sources(v);
  if (nls == 0 || v.nsel == 0) return RB_OK;
  const int nh = ncol * nprefix;
  const size_t smem = (size_t)nh * 8 + (size_t)cs::HIST_THREADS * (v.ndim | 1) * 8 + ((size_t)nh * 256 + ncol) * 4;
  CUDA_TRY(cudaFuncSetAttribute(cs::k_hist, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // enough blocks to fill the GPU; at most 2^31 items per block so that the 32-bit shared counters cannot wrap
  const long long items = std::min<long long>(v.W, v.nlocal) * v.nsel;
  long long bx = std::max<long long>(1, (long long)ctx->sm_count * 4 / nls);
  bx = std::min<long long>(bx, (items + cs::HIST_THREADS - 1) / cs::HIST_THREADS);
  bx = std::max<long long>(bx, (items >> 31) + 1);
  if (nls > 65535 || bx > 0x7fffffffLL) {
    rb_set_error(std::string(who) + ": too many sources on this rank");
    return RB_ERR_ARG;
  }
  cs::k_hist<<<dim3((unsigned)bx, (unsigned)nls), cs::HIST_THREADS, smem, ctx->stream>>>(
      v, cols, pass, nprefix, reinterpret_cast<const unsigned long long *>(prefix),
      reinterpret_cast<unsigned long long *>(counts), reinterpret_cast<unsigned long long *>(nan_counts));
  CUDA_TRY(cudaGetLastError());
  ctx->launches += 1;
  return RB_OK;
}

int rb_chain_moments_dev(rb_ctx *ctx, const rb_chain_view *view, double *mean, double *c0) {
  static const char *who = "rb_chain_moments_dev";
  cs::View v;
  int rc = chain_view(who, view, INT32_MAX, &v);
  if (rc != RB_OK) return rc;
  if (!mean || !c0) {
    rb_set_error(std::string(who) + ": null output");
    return RB_ERR_ARG;
  }
  if ((rc = chain_device(who, ctx)) != RB_OK) return rc;
  const long long n = v.nlocal * v.ndim;
  if (n == 0) return RB_OK;
  cs::k_moments<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(v, mean, c0);
  CUDA_TRY(cudaGetLastError());
  ctx->launches += 1;
  return RB_OK;
}

int rb_chain_acf_dev(rb_ctx *ctx, const rb_chain_view *view, int32_t nsrc, const double *mean, const double *c0,
                     int64_t k0, int64_t k1, double *rho_sum) {
  static const char *who = "rb_chain_acf_dev";
  cs::View v;
  int rc = chain_view(who, view, nsrc, &v);
  if (rc != RB_OK) return rc;
  if (!mean || !c0 || !rho_sum || nsrc < 1 || k0 < 0 || k1 <= k0 || k1 > v.nsel) {
    rb_set_error(std::string(who) + ": bad argument (need 0 <= k0 < k1 <= selected steps)");
    return RB_ERR_ARG;
  }
  if ((rc = chain_device(who, ctx)) != RB_OK) return rc;
  const long long nl_all = k1 - k0;
  CUDA_TRY(cudaMemsetAsync(rho_sum, 0, (size_t)nsrc * nl_all * v.ndim * sizeof(double), ctx->stream));
  const long long nls = local_sources(v);
  if (nls == 0) return RB_OK;
  long long lo, hi;
  cs::local_range(v, 0, lo, hi);
  const long long ng0 = (hi - lo + cs::ACF_GROUP - 1) / cs::ACF_GROUP;
  const long long ngW = (v.W + cs::ACF_GROUP - 1) / cs::ACF_GROUP;
  // blocks: ng0 groups of the first local source, ngW of every later one but the last, which may hold fewer walkers
  long long nb = ng0;
  if (nls > 1) {
    long long l2, h2;
    cs::local_range(v, nls - 1, l2, h2);
    nb += (nls - 2) * ngW + (h2 - l2 + cs::ACF_GROUP - 1) / cs::ACF_GROUP;
  }
  const size_t need = (size_t)nb * std::min<long long>(nl_all, cs::ACF_LAGS) * v.ndim * sizeof(double);
  if ((rc = grow(ctx->cs_buf, ctx->cs_bytes, need)) != RB_OK) return rc;
  double *partial = static_cast<double *>(ctx->cs_buf);
  const size_t smem = (size_t)v.ndim * (2 * cs::ACF_TT + cs::ACF_LAGS + 2 * cs::ACF_R) * sizeof(double);
  CUDA_TRY(cudaFuncSetAttribute(cs::k_acf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  for (long long kb = k0; kb < k1; kb += cs::ACF_LAGS) {
    const int nl = (int)std::min<long long>(cs::ACF_LAGS, k1 - kb);
    cs::k_acf<<<(unsigned)nb, v.ndim * (cs::ACF_LAGS / cs::ACF_R), smem, ctx->stream>>>(v, mean, c0, kb, nl, ng0, ngW,
                                                                                         partial);
    CUDA_TRY(cudaGetLastError());
    // rho_sum is [nsrc][k1 - k0][ndim]; this launch fills lags [kb, kb + nl) through a temporary view of its rows
    const long long per = (long long)nl * v.ndim, nout = nls * per;
    cs::k_acf_reduce<<<(unsigned)((nout + 255) / 256), 256, 0, ctx->stream>>>(v, nl, ng0, ngW, nls, partial,
                                                                             rho_sum, nl_all, kb - k0);
    CUDA_TRY(cudaGetLastError());
    ctx->launches += 2;
  }
  return RB_OK;
}

// ---- corner-plot marginals, covariance sums, nearest sample (chain_marginals.cuh) ----------------------------------
// blocks per local source: enough to fill the GPU, at most one per `per` items of the largest local source
static long long blocks_per_source(const rb_ctx *ctx, const cs::View &v, long long nls, long long per) {
  const long long items = std::min<long long>(v.W, v.nlocal) * v.nsel;
  long long bx = std::max<long long>(1, (long long)ctx->sm_count * 4 / nls);
  return std::max<long long>(1, std::min<long long>(bx, (items + per - 1) / per));
}

int rb_chain_marginals_dev(rb_ctx *ctx, const rb_chain_view *view, int32_t nsrc, int32_t ncol, const int32_t *col_i,
                           const int32_t *col_j, int32_t nbins, const double *edges, uint64_t *counts1,
                           uint64_t *counts2) {
  static const char *who = "rb_chain_marginals_dev";
  cs::View v;
  int rc = chain_view(who, view, nsrc, &v);
  if (rc != RB_OK) return rc;
  cs::Cols cols;
  std::string e;
  if (ncol < 1 || ncol > RB_CHAIN_MAX_COLS || !col_i || !col_j) e = "ncol must be in 1..RB_CHAIN_MAX_COLS";
  else if (nbins < 1 || nbins > RB_CHAIN_MAX_BINS) e = "nbins must be in 1..RB_CHAIN_MAX_BINS";
  else if (!edges || !counts1) e = "null edges or counts";
  for (int c = 0; e.empty() && c < ncol; ++c) {
    if (col_i[c] < 0 || col_i[c] >= v.ndim || col_j[c] < -1 || col_j[c] >= v.ndim) e = "column outside [0, ndim)";
    cols.i[c] = col_i[c];
    cols.j[c] = col_j[c];
  }
  cols.n = ncol;
  if (!e.empty()) {
    rb_set_error(std::string(who) + ": " + e);
    return RB_ERR_ARG;
  }
  if ((rc = chain_device(who, ctx)) != RB_OK) return rc;
  const long long nls = local_sources(v);
  if (nls == 0 || v.nsel == 0) return RB_OK;
  // shared memory: edges, staged rows, 1-D counters, column bins; then 4 nbins^2 bytes of counters + 2 per pair
  const int nb = nbins, npair = counts2 ? ncol * (ncol - 1) / 2 : 0;
  const size_t fixed = (size_t)ncol * (nb + 1) * 8 + (size_t)cs::MARG_THREADS * (v.ndim | 1) * 8 + (size_t)ncol * nb * 4 +
                       (size_t)ncol * cs::MARG_THREADS;
  const size_t per_pair = (size_t)nb * nb * 4 + 2;
  const long long fit = ((long long)ctx->smem_optin - (long long)fixed) / (long long)per_pair;
  if (npair > 0 && fit < 1) {
    rb_set_error(std::string(who) + ": one pair's counters do not fit shared memory");
    return RB_ERR_LIMIT;
  }
  // pair groups of equal size, as few as fit: each group is one read of the chain
  const int ngroups = npair > 0 ? (int)((npair + fit - 1) / fit) : 1;
  const int per_group = npair > 0 ? (npair + ngroups - 1) / ngroups : 0;
  CUDA_TRY(cudaFuncSetAttribute(cs::k_marg, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)(fixed + per_group * per_pair)));
  // at most 2^31 items per block so that the 32-bit shared counters cannot wrap
  const long long items = std::min<long long>(v.W, v.nlocal) * v.nsel;
  long long bx = blocks_per_source(ctx, v, nls, cs::MARG_THREADS);
  bx = std::max<long long>(bx, (items >> 31) + 1);
  if (nls > 65535 || bx > 0x7fffffffLL) {
    rb_set_error(std::string(who) + ": too many sources on this rank");
    return RB_ERR_ARG;
  }
  for (int g = 0; g < ngroups; ++g) {
    const int p0 = g * per_group, npg = std::min(per_group, npair - p0);
    const size_t smem = fixed - (g ? (size_t)ncol * nb * 4 : 0) + (size_t)npg * per_pair;
    cs::k_marg<<<dim3((unsigned)bx, (unsigned)nls), cs::MARG_THREADS, smem, ctx->stream>>>(
        v, cols, nb, p0, npg, g == 0, edges, reinterpret_cast<unsigned long long *>(counts1),
        reinterpret_cast<unsigned long long *>(counts2));
    CUDA_TRY(cudaGetLastError());
    ctx->launches += 1;
  }
  return RB_OK;
}

int rb_chain_sums_dev(rb_ctx *ctx, const rb_chain_view *view, int32_t nsrc, const double *center, double *s1,
                      double *s2) {
  static const char *who = "rb_chain_sums_dev";
  cs::View v;
  int rc = chain_view(who, view, nsrc, &v);
  if (rc != RB_OK) return rc;
  if (nsrc < 1 || !center || !s1 || !s2) {
    rb_set_error(std::string(who) + ": bad argument (nsrc >= 1, non-null center, s1, s2)");
    return RB_ERR_ARG;
  }
  if ((rc = chain_device(who, ctx)) != RB_OK) return rc;
  const long long nls = local_sources(v);
  const int nent = v.ndim + v.ndim * (v.ndim + 1) / 2;
  const long long bx = (nls > 0 && v.nsel > 0) ? blocks_per_source(ctx, v, nls, cs::SUMS_THREADS) : 0;
  if (nls > 65535) {
    rb_set_error(std::string(who) + ": too many sources on this rank");
    return RB_ERR_ARG;
  }
  if ((rc = grow(ctx->cs_buf, ctx->cs_bytes, std::max<size_t>(8, (size_t)nls * bx * nent * sizeof(double)))) != RB_OK)
    return rc;
  double *partial = static_cast<double *>(ctx->cs_buf);
  if (bx > 0) {
    cs::k_sums<<<dim3((unsigned)bx, (unsigned)nls), cs::SUMS_THREADS, 0, ctx->stream>>>(v, center, partial);
    CUDA_TRY(cudaGetLastError());
    ctx->launches += 1;
  }
  const long long nout = (long long)nsrc * nent;
  cs::k_sums_reduce<<<(unsigned)((nout + 255) / 256), 256, 0, ctx->stream>>>(v, nsrc, bx > 0 ? nls : 0, (int)bx,
                                                                             partial, s1, s2);
  CUDA_TRY(cudaGetLastError());
  ctx->launches += 1;
  return RB_OK;
}

int rb_chain_nearest_dev(rb_ctx *ctx, const rb_chain_view *view, int32_t nsrc, const double *target, const double *chol,
                         double *d2, int64_t *index, double *x) {
  static const char *who = "rb_chain_nearest_dev";
  cs::View v;
  int rc = chain_view(who, view, nsrc, &v);
  if (rc != RB_OK) return rc;
  if (nsrc < 1 || !target || !chol || !d2 || !index || !x) {
    rb_set_error(std::string(who) + ": bad argument (nsrc >= 1, non-null target, chol, d2, index, x)");
    return RB_ERR_ARG;
  }
  if ((rc = chain_device(who, ctx)) != RB_OK) return rc;
  const long long nls = local_sources(v);
  const long long bx = (nls > 0 && v.nsel > 0) ? blocks_per_source(ctx, v, nls, cs::NEAR_THREADS) : 0;
  if (nls > 65535) {
    rb_set_error(std::string(who) + ": too many sources on this rank");
    return RB_ERR_ARG;
  }
  const size_t nblk = (size_t)nls * bx;
  if ((rc = grow(ctx->cs_buf, ctx->cs_bytes, std::max<size_t>(16, nblk * 16))) != RB_OK) return rc;
  double *pd2 = static_cast<double *>(ctx->cs_buf);
  long long *pidx = reinterpret_cast<long long *>(pd2 + nblk);
  if (bx > 0) {
    cs::k_near<<<dim3((unsigned)bx, (unsigned)nls), cs::NEAR_THREADS, 0, ctx->stream>>>(v, target, chol, pd2, pidx);
    CUDA_TRY(cudaGetLastError());
    ctx->launches += 1;
  }
  cs::k_near_reduce<<<(unsigned)((nsrc + 255) / 256), 256, 0, ctx->stream>>>(
      v, nsrc, bx > 0 ? nls : 0, (int)bx, pd2, pidx, d2, reinterpret_cast<long long *>(index), x);
  CUDA_TRY(cudaGetLastError());
  ctx->launches += 1;
  return RB_OK;
}

// ---- posterior-predictive SLEDs (predict_sled.cuh) ---------------------------------------------------------------
#define RB_PREDICT_MAX (2 * RB_PIPE_MAX)   // models per pipeline call: bounds ctx->ln_buf however long the chain is

int rb_predict_sled_dev(rb_ctx *ctx, const rb_srcset *set, const rb_chain_view *view, int32_t nlines, const int32_t *jup,
                        const rb_opts *opts, double *flux, int64_t *counters_dev) {
  static const char *who = "rb_predict_sled_dev";
  std::string e;
  if (!set || !jup || !flux) e = "null argument";
  else if (nlines < 1 || nlines > RB_MAX_OBS) e = "nlines must be in 1..RB_MAX_OBS";
  for (int k = 0; e.empty() && k < nlines; ++k)
    if (jup[k] < 1) e = "J must be in 1..nline";
  if (!e.empty()) {
    rb_set_error(std::string(who) + ": " + e);
    return RB_ERR_ARG;
  }
  cs::View v;
  int rc = chain_view(who, view, INT32_MAX, &v);
  if (rc != RB_OK) return rc;
  if ((rc = chain_device(who, ctx)) != RB_OK) return rc;
  if (set->ctx != ctx) e = "the source set belongs to another context";
  else if (view->ndim != 4 * set->ncomp) e = "ndim is not 4 x the source set's ncomp";
  else if (v.nlocal > 0 && (v.gid_base + v.nlocal - 1) / v.W >= set->nsrc) e = "the source set does not cover the rank's walkers";
  else if (!ctx->ln_partners_ok) e = "the molecular file has no H2 / p-H2 / o-H2 collision partner";
  for (int k = 0; e.empty() && k < nlines; ++k)
    if (jup[k] > ctx->mol.nline) e = "J must be in 1..nline";
  if (!e.empty()) {
    rb_set_error(std::string(who) + ": " + e);
    return RB_ERR_ARG;
  }
  CUDA_TRY(cudaMemsetAsync(ctx->counters, 0, 8 * sizeof(unsigned long long), ctx->stream));
  const long long nls = local_sources(v);
  if (nls == 0 || v.nsel == 0) return RB_OK;
  const int ncomp = set->ncomp;
  const bool v2 = use_v2(ctx, opts);
  // v2: observed-line mode, line k of model m at obs_surf[m][k]; v1: every line, at surf[m][J - 1]
  const int stride = v2 ? RB_MAX_OBS : ctx->mol.nline;
  long long total = 0;
  for (long long s = 0; s < nls; ++s) {
    long long lo, hi;
    cs::local_range(v, s, lo, hi);
    total = std::max(total, (hi - lo) * v.nsel);
  }
  const long long per_call = std::max<long long>(1, RB_PREDICT_MAX / ncomp);
  LnprobPipe pp;
  if ((rc = model_arrays(ctx, std::min(total, per_call) * ncomp, stride, &pp)) != RB_OK) return rc;
  PredictIO io;
  memset(&io, 0, sizeof(io));
  io.v = v;
  io.tkin = pp.tkin;
  io.cdmol = pp.cdmol;
  io.dens = pp.dens;
  io.surf = pp.obs_surf;
  io.status = pp.status;
  io.stride = stride;
  io.nlines = nlines;
  for (int k = 0; k < nlines; ++k) io.line[k] = v2 ? k : jup[k] - 1;
  io.flux = flux;
  io.counters = reinterpret_cast<unsigned long long *>(counters_dev);
  SolveIO sio{0, pp.tkin, pp.dens, pp.cdmol, nullptr, nullptr, nullptr, v2 ? nullptr : pp.obs_surf, nullptr, pp.status,
              ctx->counters};
  if (v2) observe_lines(sio, pp.obs_surf, nlines, jup);
  const int tpb = 256;
  for (long long s = 0; s < nls; ++s) {
    long long lo, hi;
    cs::local_range(v, s, lo, hi);
    io.w0 = lo;
    io.nw = hi - lo;
    const SolveCfg cfg = make_cfg(ctx, opts, 1.0, set->h[v.src0 + s].tbg, RB_GEOM_LVG);   // model_lvg: LVG, 1 km/s
    for (long long i0 = 0; i0 < io.nw * v.nsel; i0 += per_call) {
      io.i0 = i0;
      io.ni = std::min(per_call, io.nw * v.nsel - i0);
      const unsigned nbe = (unsigned)((io.ni + tpb - 1) / tpb);
      if (ncomp == 1)
        k_predict_expand<1><<<nbe, tpb, 0, ctx->stream>>>(ctx->mol, io);
      else
        k_predict_expand<2><<<nbe, tpb, 0, ctx->stream>>>(ctx->mol, io);
      CUDA_TRY(cudaMemsetAsync(ctx->counters, 0, sizeof(unsigned long long), ctx->stream));   // queue head only
      sio.n = io.ni * ncomp;
      if ((rc = launch_solve(ctx, cfg, opts, sio)) != RB_OK) return rc;
      const unsigned nbf = (unsigned)((io.ni * nlines + tpb - 1) / tpb);
      if (ncomp == 1)
        k_predict_flux<1><<<nbf, tpb, 0, ctx->stream>>>(io);
      else
        k_predict_flux<2><<<nbf, tpb, 0, ctx->stream>>>(io);
      CUDA_TRY(cudaGetLastError());
      ctx->launches += 3;
    }
  }
  return RB_OK;
}

int rb_ctx_counters(rb_ctx *ctx, int64_t *total_iters_last, int64_t *launches_total) {
  if (!ctx) return RB_ERR_ARG;
  CUDA_TRY(cudaSetDevice(ctx->device));
  const int rc = read_counters(ctx);
  if (rc != RB_OK) return rc;
  if (total_iters_last) *total_iters_last = ctx->last_total_iters;
  if (launches_total) *launches_total = ctx->launches;
  return RB_OK;
}

int rb_ctx_cache_stats(rb_ctx *ctx, int64_t *stats3) {
  if (!ctx || !stats3) return RB_ERR_ARG;
  CUDA_TRY(cudaSetDevice(ctx->device));
  unsigned long long cnt[3] = {0, 0, 0};
  CUDA_TRY(cudaMemcpyAsync(cnt, ctx->counters + 3, sizeof(cnt), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < 3; ++i) stats3[i] = (int64_t)cnt[i];
  return RB_OK;
}

}  // extern "C"
