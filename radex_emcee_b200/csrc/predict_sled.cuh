// predict_sled.cuh -- posterior-predictive SLEDs of the device-resident chain (rb_predict_sled_dev in radex_b200.h).
//
// What it replaces: the reference's replot, which draws model SLEDs from the pickled chain on the host through
// model_lvg, one serial Radex call per sample (emcee/emcee_radex.py:120-130, emcee/emcee_radex_2comp.py:122-147).
// Here the selected chain rows are read in place (chain_stats.cuh's View / row), expanded into the model arrays of the
// scheduled solve (k_predict_expand), solved with the same kernels as every other call, and turned into per-line fluxes
// (k_predict_flux).  The expressions are those of k_lnprob_expand and k_lnprob_combine, without the prior: the model SLED
// of a sample is what model_lvg returns for it, and a component out of pyradex's range gives NaN where model_lvg raises.
#pragma once

// One pipeline call covers the items [i0, i0 + ni) of one source: item i is local walker w0 + i % nw at selected step
// i / nw; its component c is model i * NCOMP + c, in [0, ni * NCOMP).
struct PredictIO {
  cs::View v;
  long long i0, ni, w0, nw;
  double *tkin, *dens, *cdmol;                 // models of the call
  const double *surf;                          // brightness of line k of model m: surf[m * stride + line[k]]
  const int *status;
  int stride, nlines;
  int line[RB_MAX_OBS];
  double *flux;                                // [nplanes][nsel][nlocal][nlines]
  unsigned long long *counters;                // [0] += models solved, [1] += models out of range; may be null
};

__device__ __forceinline__ const double *predict_row(const PredictIO &io, long long i) {
  const long long it = io.i0 + i;
  int cur = 0;
  return cs::row(io.v, it / io.nw, io.w0 + it % io.nw, cur);
}

template <int NCOMP>
__global__ void __launch_bounds__(256) k_predict_expand(MolDev mol, PredictIO io) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= io.ni) return;
  const double *p = predict_row(io, i);
#pragma unroll
  for (int c = 0; c < NCOMP; ++c) {
    const long long m = i * NCOMP + c;
    const double dens_tot = pow(10.0, p[4 * c + 0]);
    for (int q = 0; q < mol.npart; ++q) io.dens[m * mol.npart + q] = mol.ln_frac[q] * dens_tot;
    io.tkin[m] = pow(10.0, p[4 * c + 1]);
    io.cdmol[m] = pow(10.0, p[4 * c + 2]);
  }
}

// One thread per (item, line): plane 0 is the flux (one component) or the total flux_0 + flux_1 (two), planes 1 and 2
// the components.  A line's consecutive threads write consecutive doubles of one walker row.
template <int NCOMP>
__global__ void __launch_bounds__(256) k_predict_flux(PredictIO io) {
  const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const bool valid = t < io.ni * io.nlines;
  unsigned solved = 0, range = 0;
  if (valid) {
    const long long i = t / io.nlines;
    const int k = (int)(t % io.nlines);
    const double *p = predict_row(io, i);
    const long long it = io.i0 + i;
    const long long plane = io.v.nsel * io.v.nlocal * io.nlines;
    double *out = io.flux + ((it / io.nw) * io.v.nlocal + io.w0 + it % io.nw) * io.nlines + k;
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    double total = 0.0;
#pragma unroll
    for (int c = 0; c < NCOMP; ++c) {
      const long long m = i * NCOMP + c;
      const bool bad = (io.status[m] & (RB_ST_T_RANGE | RB_ST_N_RANGE)) != 0;
      const double f = bad ? qnan : io.surf[m * io.stride + io.line[k]] * pow(10.0, p[4 * c + 3]) * 1.0e23;
      if (NCOMP == 2) out[(c + 1) * plane] = f;
      total = (c == 0) ? f : total + f;
      if (k == 0) {
        solved += !bad;
        range += bad;
      }
    }
    out[0] = total;
  }
  if (io.counters) {
    solved = __reduce_add_sync(0xffffffffu, solved);
    range = __reduce_add_sync(0xffffffffu, range);
    if ((threadIdx.x & 31) == 0) {
      if (solved) atomicAdd(&io.counters[0], (unsigned long long)solved);
      if (range) atomicAdd(&io.counters[1], (unsigned long long)range);
    }
  }
}
