// chain_marginals.cuh -- corner-plot marginals, covariance and the sample nearest a target, computed where the chain
// lives (rb_chain_marginals_dev, rb_chain_sums_dev, rb_chain_nearest_dev in radex_b200.h).
//
// What it replaces: the reference's replot, which draws `corner` plots from the pickled chain, and the host search of
// driver.nearest_sample_to_vector (emcee_radex.py:242-266); both need the whole chain in host memory.  The kernels read
// the chain in place through chain_stats.cuh's View / row (emcee's discard / thin across chunks); only bin counts,
// per-block sums and one row per source leave the device.
//
// Marginals: bin k of x for the edges e[0..B] of (source, column) is (number of edges <= x) - 1, with x == e[B] in bin
// B - 1 -- np.searchsorted(e, x, 'right') - 1, how np.histogram(range=) and np.histogram2d(range=) bin.  NaN, +-inf and
// values outside [e[0], e[B]] are not counted.  One read of the chain counts every column and one group of pairs: each
// thread bins its row's columns once (binary search over the edges in shared memory), then feeds every 1-D and 2-D
// counter; equal bins of a warp are merged (__match_any_sync) before one shared-memory atomic, as k_hist does.
//
// Sums: per block, s1 = sum (x - c) and s2 = sum (x - c)(x - c)^T over its items in a fixed order (thread per entry of
// s1 and of the upper triangle of s2), then a second kernel adds the blocks of each source in block order: no
// floating-point atomics, so a repeated call gives the same bits.
//
// Nearest: w = L^-1 (x - t) by forward substitution, d2 = sum_r w_r^2 in r order; the minimum per source under the
// order NaN < numbers, ties to the lowest index j W + (gid - s W) (np.argmin over the source's flattened selection).
#pragma once

namespace cs {

constexpr int MARG_THREADS = 256;
constexpr int SUMS_THREADS = 256;
constexpr int NEAR_THREADS = 256;
constexpr unsigned char NO_BIN = 255;   // nbins <= RB_CHAIN_MAX_BINS < 255
constexpr long long NO_INDEX = 0x7fffffffffffffffLL;   // no sample yet (orders after every index)

// bin of x for the strictly increasing edges e[0..nb], or NO_BIN
__device__ __forceinline__ unsigned bin_of(const double *e, int nb, double x) {
  int n = 0;                                        // number of edges <= x (0 for NaN)
#pragma unroll
  for (int step = 64; step >= 1; step >>= 1)
    if (n + step <= nb + 1 && e[n + step - 1] <= x) n += step;
  int k = n - 1;
  if (n == nb + 1 && x == e[nb]) k = nb - 1;
  return (k >= 0 && k < nb) ? (unsigned)k : NO_BIN;
}

// pair p of (0,1), (0,2), ..., (0,n-1), (1,2), ...
__device__ __forceinline__ void pair_of(int p, int n, int &a, int &b) {
  a = 0;
  while (p >= n - 1 - a) {
    p -= n - 1 - a;
    ++a;
  }
  b = a + 1 + p;
}

// One source per blockIdx.y: counts1[src][c][k] (when do1) and counts2[src][p0 + q][ka][kb] for the pairs q < npg of
// this group, ADDED.  Shared: the source's edges, the staged rows, 32-bit block counters, each thread's column bins.
__global__ void __launch_bounds__(MARG_THREADS) k_marg(View v, Cols cols, int nb, int p0, int npg, int do1,
                                                       const double *__restrict__ edges,
                                                       unsigned long long *__restrict__ counts1,
                                                       unsigned long long *__restrict__ counts2) {
  extern __shared__ double smem_m[];
  const int ncol = cols.n, ne = nb + 1, rs = v.ndim | 1, n1 = do1 ? ncol * nb : 0, nbb = nb * nb;
  double *sedge = smem_m;                                                  // [ncol][nb + 1]
  double *srow = sedge + ncol * ne;                                        // [MARG_THREADS][rs]
  unsigned *h1 = reinterpret_cast<unsigned *>(srow + MARG_THREADS * rs);   // [ncol][nb] (do1)
  unsigned *h2 = h1 + n1;                                                  // [npg][nb][nb]
  unsigned char *sbin = reinterpret_cast<unsigned char *>(h2 + npg * nbb); // [ncol][MARG_THREADS]
  unsigned char *spa = sbin + ncol * MARG_THREADS, *spb = spa + npg;       // columns of the group's pairs
  const long long src = v.src0 + blockIdx.y;
  long long lo, hi;
  local_range(v, blockIdx.y, lo, hi);
  const long long nw = hi - lo, items = nw * v.nsel;
  for (int k = threadIdx.x; k < n1 + npg * nbb; k += blockDim.x) h1[k] = 0;
  for (int k = threadIdx.x; k < ncol * ne; k += blockDim.x) sedge[k] = edges[src * ncol * ne + k];
  for (int q = threadIdx.x; q < npg; q += blockDim.x) {
    int a, b;
    pair_of(p0 + q, ncol, a, b);
    spa[q] = (unsigned char)a;
    spb[q] = (unsigned char)b;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  double *my = srow + threadIdx.x * rs;
  unsigned char *mybin = sbin + threadIdx.x;                               // mybin[c * MARG_THREADS]: own entries only
  int cur = 0;
  for (long long base = (long long)blockIdx.x * blockDim.x; base < items; base += (long long)gridDim.x * blockDim.x) {
    const long long it = base + threadIdx.x;
    const bool valid = it < items;
    if (valid) {
      const double *p = row(v, it / nw, lo + it % nw, cur);
      for (int d = 0; d < v.ndim; ++d) my[d] = __ldg(p + d);
    }
    for (int c = 0; c < ncol; ++c) {
      const int cj = cols.j[c];
      const double x = valid ? (cj < 0 ? my[cols.i[c]] : my[cols.i[c]] + my[cj]) : 0.0;
      mybin[c * MARG_THREADS] = valid ? (unsigned char)bin_of(sedge + c * ne, nb, x) : NO_BIN;
    }
    if (do1) {
      for (int c = 0; c < ncol; ++c) {
        const unsigned k = mybin[c * MARG_THREADS];
        const bool hit = k != NO_BIN;
        if (!__any_sync(0xffffffffu, hit)) continue;
        const unsigned peers = __match_any_sync(0xffffffffu, hit ? k : 0xffffffffu);
        if (hit && lane == __ffs(peers) - 1) atomicAdd(&h1[c * nb + k], (unsigned)__popc(peers));
      }
    }
    for (int q = 0; q < npg; ++q) {
      const unsigned ka = mybin[spa[q] * MARG_THREADS], kb = mybin[spb[q] * MARG_THREADS];
      const bool hit = ka != NO_BIN && kb != NO_BIN;
      if (!__any_sync(0xffffffffu, hit)) continue;
      const unsigned k = ka * nb + kb;
      const unsigned peers = __match_any_sync(0xffffffffu, hit ? k : 0xffffffffu);
      if (hit && lane == __ffs(peers) - 1) atomicAdd(&h2[q * nbb + k], (unsigned)__popc(peers));
    }
  }
  __syncthreads();
  const long long npair = (long long)ncol * (ncol - 1) / 2;
  for (int k = threadIdx.x; k < n1; k += blockDim.x)
    if (h1[k]) atomicAdd(&counts1[src * ncol * nb + k], (unsigned long long)h1[k]);
  for (int k = threadIdx.x; k < npg * nbb; k += blockDim.x)
    if (h2[k]) atomicAdd(&counts2[(src * npair + p0) * nbb + k], (unsigned long long)h2[k]);
}

// entry e of the sums: e < nd is s1[e], else the upper-triangle element (d, f), d <= f, in row order
__device__ __forceinline__ void sums_entry(int e, int nd, int &d, int &f) {
  if (e < nd) {
    d = e;
    f = -1;
    return;
  }
  int q = e - nd;
  d = 0;
  while (q >= nd - d) {
    q -= nd - d;
    ++d;
  }
  f = d + q;
}

// partial[(blockIdx.y * gridDim.x + blockIdx.x)][e], e < nd + nd (nd + 1) / 2: the block's sums over the items of
// source blockIdx.y in tiles blockIdx.x, blockIdx.x + gridDim.x, ... (each a sequential sum in item order)
__global__ void __launch_bounds__(SUMS_THREADS) k_sums(View v, const double *__restrict__ center,
                                                       double *__restrict__ partial) {
  __shared__ double sy[SUMS_THREADS * (RB_CHAIN_MAX_DIM | 1)];
  __shared__ double sc[RB_CHAIN_MAX_DIM];
  const int nd = v.ndim, rs = nd | 1, nent = nd + nd * (nd + 1) / 2;
  const long long src = v.src0 + blockIdx.y;
  long long lo, hi;
  local_range(v, blockIdx.y, lo, hi);
  const long long nw = hi - lo, items = nw * v.nsel;
  int d = 0, f = -1;
  if (threadIdx.x < nent) sums_entry(threadIdx.x, nd, d, f);
  if (threadIdx.x < nd) sc[threadIdx.x] = center[src * nd + threadIdx.x];
  double acc = 0.0;
  int cur = 0;
  for (long long t0 = (long long)blockIdx.x * SUMS_THREADS; t0 < items; t0 += (long long)gridDim.x * SUMS_THREADS) {
    __syncthreads();
    const long long it = t0 + threadIdx.x;
    if (it < items) {
      const double *p = row(v, it / nw, lo + it % nw, cur);
      for (int k = 0; k < nd; ++k) sy[threadIdx.x * rs + k] = __ldg(p + k) - sc[k];
    }
    __syncthreads();
    const int n = items - t0 < SUMS_THREADS ? (int)(items - t0) : SUMS_THREADS;
    if (threadIdx.x < nent) {
      if (f < 0)
        for (int r = 0; r < n; ++r) acc += sy[r * rs + d];
      else
        for (int r = 0; r < n; ++r) acc = fma(sy[r * rs + d], sy[r * rs + f], acc);
    }
  }
  if (threadIdx.x < nent) partial[((long long)blockIdx.y * gridDim.x + blockIdx.x) * nent + threadIdx.x] = acc;
}

// s1[src][d], s2[src][d][f] of every source < nsrc: the partials of its nbx blocks in block order, 0 off this rank
__global__ void k_sums_reduce(View v, long long nsrc, long long nls, int nbx, const double *__restrict__ partial,
                              double *__restrict__ s1, double *__restrict__ s2) {
  const int nd = v.ndim, nent = nd + nd * (nd + 1) / 2;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= nsrc * nent) return;
  const long long src = idx / nent, s = src - v.src0;
  const int e = (int)(idx % nent);
  double acc = 0.0;
  if (s >= 0 && s < nls)
    for (int b = 0; b < nbx; ++b) acc += partial[(s * nbx + b) * nent + e];
  int d, f;
  sums_entry(e, nd, d, f);
  if (f < 0) {
    s1[src * nd + d] = acc;
  } else {
    s2[(src * nd + d) * nd + f] = acc;
    s2[(src * nd + f) * nd + d] = acc;
  }
}

// (d2, index) a orders before b: NaN before every number, then the smaller d2, then the lower index
__device__ __forceinline__ bool nearer(double da, long long ia, double db, long long ib) {
  const bool na = isnan(da), nb = isnan(db);
  if (na != nb) return na;
  if (!na && da != db) return da < db;
  return ia < ib;
}

// per block of source blockIdx.y: the nearest of its items, pd2[b], pidx[b] (NO_INDEX: none)
__global__ void __launch_bounds__(NEAR_THREADS) k_near(View v, const double *__restrict__ target,
                                                       const double *__restrict__ chol, double *__restrict__ pd2,
                                                       long long *__restrict__ pidx) {
  __shared__ double sL[RB_CHAIN_MAX_DIM * RB_CHAIN_MAX_DIM];
  __shared__ double st[RB_CHAIN_MAX_DIM];
  __shared__ double wd2[NEAR_THREADS / 32];
  __shared__ long long widx[NEAR_THREADS / 32];
  const int nd = v.ndim;
  const long long src = v.src0 + blockIdx.y;
  long long lo, hi;
  local_range(v, blockIdx.y, lo, hi);
  const long long nw = hi - lo, items = nw * v.nsel;
  const long long off = v.gid_base + lo - src * v.W;       // position of local walker lo within its source
  for (int k = threadIdx.x; k < nd * nd; k += blockDim.x) sL[k] = chol[src * nd * nd + k];
  if (threadIdx.x < nd) st[threadIdx.x] = target[src * nd + threadIdx.x];
  __syncthreads();
  double best = __longlong_as_double(0x7ff0000000000000LL);   // +inf
  long long bidx = NO_INDEX;
  int cur = 0;
  for (long long it = (long long)blockIdx.x * blockDim.x + threadIdx.x; it < items;
       it += (long long)gridDim.x * blockDim.x) {
    const long long j = it / nw, w = it % nw;
    const double *p = row(v, j, lo + w, cur);
    double y[RB_CHAIN_MAX_DIM];
    double d2 = 0.0;
#pragma unroll
    for (int r = 0; r < RB_CHAIN_MAX_DIM; ++r) {
      if (r < nd) {
        double s = __ldg(p + r) - st[r];
#pragma unroll
        for (int k = 0; k < r; ++k) s -= sL[r * nd + k] * y[k];
        y[r] = s / sL[r * nd + r];
        d2 += y[r] * y[r];
      }
    }
    const long long idx = j * v.W + off + w;
    if (nearer(d2, idx, best, bidx)) {
      best = d2;
      bidx = idx;
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const double od = __shfl_down_sync(0xffffffffu, best, o);
    const long long oi = __shfl_down_sync(0xffffffffu, bidx, o);
    if (nearer(od, oi, best, bidx)) {
      best = od;
      bidx = oi;
    }
  }
  if ((threadIdx.x & 31) == 0) {
    wd2[threadIdx.x >> 5] = best;
    widx[threadIdx.x >> 5] = bidx;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 1; k < NEAR_THREADS / 32; ++k)
      if (nearer(wd2[k], widx[k], best, bidx)) {
        best = wd2[k];
        bidx = widx[k];
      }
    const long long b = (long long)blockIdx.y * gridDim.x + blockIdx.x;
    pd2[b] = best;
    pidx[b] = bidx;
  }
}

// every source < nsrc: the nearest over its nbx blocks, its index and row; index -1, d2 = +inf, x = 0 without one
__global__ void k_near_reduce(View v, long long nsrc, long long nls, int nbx, const double *__restrict__ pd2,
                              const long long *__restrict__ pidx, double *__restrict__ d2, long long *__restrict__ index,
                              double *__restrict__ x) {
  const long long src = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (src >= nsrc) return;
  const long long s = src - v.src0;
  double best = __longlong_as_double(0x7ff0000000000000LL);
  long long bidx = NO_INDEX;
  if (s >= 0 && s < nls)
    for (int b = 0; b < nbx; ++b)
      if (nearer(pd2[s * nbx + b], pidx[s * nbx + b], best, bidx)) {
        best = pd2[s * nbx + b];
        bidx = pidx[s * nbx + b];
      }
  d2[src] = best;
  index[src] = bidx == NO_INDEX ? -1 : bidx;
  if (bidx == NO_INDEX) {
    for (int k = 0; k < v.ndim; ++k) x[src * v.ndim + k] = 0.0;
    return;
  }
  int cur = 0;
  const double *p = row(v, bidx / v.W, src * v.W + bidx % v.W - v.gid_base, cur);
  for (int k = 0; k < v.ndim; ++k) x[src * v.ndim + k] = p[k];
}

}  // namespace cs
