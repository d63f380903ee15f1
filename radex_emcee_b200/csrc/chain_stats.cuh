// chain_stats.cuh -- posterior statistics of the device-resident chain, computed where the chain lives
// (rb_chain_hist_dev, rb_chain_moments_dev, rb_chain_acf_dev in radex_b200.h).
//
// What it replaces: the drivers' np.percentile over the flattened chain (emcee/emcee_radex.py:511-531) and emcee's
// get_autocorr_time / integrated_time, which both need the whole chain in host memory.  The kernels read the chain in
// place, chunk by chunk (one chunk per run_mcmc call), with emcee's discard / thin applied to the concatenated step index;
// only digit histograms and per-lag sums leave the device.
//
// Exact percentiles by radix select: a double maps to an order-preserving 64-bit key; pass p (0..7) counts digit p
// (8 bits, most significant first) of the values whose higher digits equal a target prefix.  Between passes the caller
// sums the histograms over ranks and narrows prefix and remaining rank; after 8 passes the key, hence the value, of every
// requested order statistic is known exactly.
//
// Autocorrelation: per (walker, parameter) the mean and c_0 = sum_t (x_t - mu)^2 over the selected steps, then for a
// block of lags rho_k = c_k / c_0 with c_k = sum_t (x_t - mu)(x_{t+k} - mu) as a direct sum, summed over the walkers of
// each source in a fixed order (per-block partials, then a second pass): repeated calls give the same bits.
#pragma once

namespace cs {

constexpr int HIST_THREADS = 256;
constexpr int ACF_LAGS = 128;        // lags per acf launch
constexpr int ACF_R = 8;             // lags per thread (register tile)
constexpr int ACF_TT = 256;          // steps per shared-memory tile
constexpr int ACF_GROUP = 128;       // walkers summed per acf block (fixed: the partial order depends on it only)
constexpr unsigned long long NO_PREFIX = ~0ull;

struct View {
  const double *chunk[RB_MAX_CHUNKS];
  long long start[RB_MAX_CHUNKS + 1];  // concatenated step index of each chunk's first step; start[nchunks] = total
  int nchunks, ndim;
  long long nlocal, gid_base, W;
  long long first, thin, nsel;         // selected steps: first + j * thin, j < nsel (first = discard + thin - 1, emcee)
  long long src0;                      // global source of local walker 0
};

struct Cols {
  int n;
  int i[RB_CHAIN_MAX_COLS], j[RB_CHAIN_MAX_COLS];   // column c = x[i[c]] (+ x[j[c]] when j[c] >= 0)
};

// local walker range [lo, hi) of global source src0 + s on this rank
__device__ __host__ inline void local_range(const View &v, long long s, long long &lo, long long &hi) {
  const long long g = v.src0 + s;
  lo = g * v.W - v.gid_base;
  hi = lo + v.W;
  if (lo < 0) lo = 0;
  if (hi > v.nlocal) hi = v.nlocal;
}

// row of walker w at selected step j; `c` is a chunk cursor that only moves forward (j never decreases per caller)
__device__ __forceinline__ const double *row(const View &v, long long j, long long w, int &c) {
  const long long t = v.first + j * v.thin;
  while (t >= v.start[c + 1]) ++c;
  return v.chunk[c] + ((t - v.start[c]) * v.nlocal + w) * v.ndim;
}

// order-preserving key: flip every bit of a negative value, only the sign bit of a non-negative one
__device__ __forceinline__ unsigned long long order_key(double x) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(x);
  return (u >> 63) ? ~u : (u | (1ull << 63));
}

// One digit pass for every (column, prefix) of one source (blockIdx.y): counts[src][c][p][digit] += values whose
// higher digits equal prefix[src][c][p].  Each thread reads one walker row (ndim contiguous doubles) per item and feeds
// every column; equal bins of a warp are merged (__match_any_sync) before one shared-memory atomic.
__global__ void __launch_bounds__(HIST_THREADS) k_hist(View v, Cols cols, int pass, int nprefix,
                                                       const unsigned long long *__restrict__ prefix,
                                                       unsigned long long *__restrict__ counts,
                                                       unsigned long long *__restrict__ nan_counts) {
  extern __shared__ unsigned long long smem_u64[];
  const int ncol = cols.n, nh = ncol * nprefix, rs = v.ndim | 1;
  unsigned long long *spre = smem_u64;                                   // [nh]
  double *srow = reinterpret_cast<double *>(spre + nh);                  // [HIST_THREADS][rs]
  unsigned *shist = reinterpret_cast<unsigned *>(srow + HIST_THREADS * rs);   // [nh][256]
  unsigned *snan = shist + nh * 256;                                     // [ncol]
  const long long src = v.src0 + blockIdx.y;
  long long lo, hi;
  local_range(v, blockIdx.y, lo, hi);
  const long long nw = hi - lo, items = nw * v.nsel;
  for (int k = threadIdx.x; k < nh * 256 + ncol; k += blockDim.x) shist[k] = 0;
  for (int k = threadIdx.x; k < nh; k += blockDim.x) spre[k] = prefix[src * nh + k];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int shift = 56 - 8 * pass;
  double *my = srow + threadIdx.x * rs;
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
      const bool isn = valid && isnan(x);
      if (pass == 0) {
        const unsigned b = __ballot_sync(0xffffffffu, isn);
        if (lane == 0 && b) atomicAdd(&snan[c], (unsigned)__popc(b));
      }
      const unsigned long long key = order_key(x);
      const bool ok = valid && !isn;
      const unsigned bin = (unsigned)(key >> shift) & 255u;
      for (int p = 0; p < nprefix; ++p) {
        const unsigned long long pre = spre[c * nprefix + p];
        if (pre == NO_PREFIX) continue;                                   // uniform over the block
        const bool hit = ok && (pass == 0 || (key >> (shift + 8)) == pre);
        if (!__any_sync(0xffffffffu, hit)) continue;
        const unsigned peers = __match_any_sync(0xffffffffu, hit ? bin : 0xffffffffu);
        if (hit && lane == __ffs(peers) - 1) atomicAdd(&shist[(c * nprefix + p) * 256 + bin], (unsigned)__popc(peers));
      }
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < nh * 256; k += blockDim.x)
    if (shist[k]) atomicAdd(&counts[src * nh * 256 + k], (unsigned long long)shist[k]);
  if (pass == 0 && nan_counts)
    for (int k = threadIdx.x; k < ncol; k += blockDim.x)
      if (snan[k]) atomicAdd(&nan_counts[src * ncol + k], (unsigned long long)snan[k]);
}

// mean and c_0 of every (walker, parameter) over the selected steps, each a sequential sum in step order.  c_0 uses the
// same fma chain as the lag-0 sum of k_acf, so rho_0 is exactly 1 (emcee: acf /= acf[0]).
__global__ void __launch_bounds__(256) k_moments(View v, double *__restrict__ mean, double *__restrict__ c0) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= v.nlocal * v.ndim) return;
  const long long w = idx / v.ndim;
  const int d = (int)(idx % v.ndim);
  double s = 0.0;
  int cur = 0;
  for (long long j = 0; j < v.nsel; ++j) s += row(v, j, w, cur)[d];
  const double mu = s / (double)v.nsel;
  double q = 0.0;
  cur = 0;
  for (long long j = 0; j < v.nsel; ++j) {
    const double y = row(v, j, w, cur)[d] - mu;
    q = fma(y, y, q);
  }
  mean[idx] = mu;
  c0[idx] = q;
}

// centred values of walker w, parameter d, selected steps [j0, j0 + n) into dst (zero beyond nsel)
__device__ __forceinline__ void load_centred(const View &v, long long w, long long j0, int n, const double *mu,
                                             double *dst, int stride) {
  const int nd = v.ndim;
  int cur = 0;
  for (int k = threadIdx.x; k < n * nd; k += blockDim.x) {
    const int tl = k / nd, d = k % nd;
    const long long j = j0 + tl;
    dst[d * stride + tl] = (j < v.nsel) ? row(v, j, w, cur)[d] - mu[d] : 0.0;
  }
}

// Lags [k0, k0 + nl), nl <= ACF_LAGS.  Block b: up to ACF_GROUP walkers of one source; thread (d, g) owns lags
// k0 + ACF_R g + r of parameter d.  partial[b][l][d] = sum over the block's walkers (in walker order) of c_k / c_0.
__global__ void __launch_bounds__(256) k_acf(View v, const double *__restrict__ mean, const double *__restrict__ c0,
                                             long long k0, int nl, long long ng0, long long ngW,
                                             double *__restrict__ partial) {
  constexpr int SA = ACF_TT, SB = ACF_TT + ACF_LAGS + 2 * ACF_R;
  extern __shared__ double smem_d[];
  double *A = smem_d;                        // [ndim][SA]: y[t0 + t]
  double *B = smem_d + v.ndim * SA;          // [ndim][SB]: y[t0 + k0 + t]
  __shared__ double smu[RB_CHAIN_MAX_DIM];
  // block -> (source, group): the first local source has ng0 groups, every later one ngW
  const long long b = blockIdx.x;
  long long s, g;
  if (b < ng0) {
    s = 0;
    g = b;
  } else {
    s = 1 + (b - ng0) / ngW;
    g = (b - ng0) % ngW;
  }
  long long lo, hi;
  local_range(v, s, lo, hi);
  const long long w0 = lo + g * ACF_GROUP, w1 = min(hi, w0 + ACF_GROUP);
  const int d = threadIdx.x / (ACF_LAGS / ACF_R), lg = threadIdx.x % (ACF_LAGS / ACF_R);
  const bool active = d < v.ndim;
  double rsum[ACF_R];
#pragma unroll
  for (int r = 0; r < ACF_R; ++r) rsum[r] = 0.0;
  for (long long w = w0; w < w1; ++w) {
    double acc[ACF_R];
#pragma unroll
    for (int r = 0; r < ACF_R; ++r) acc[r] = 0.0;
    __syncthreads();
    if (threadIdx.x < v.ndim) smu[threadIdx.x] = mean[w * v.ndim + threadIdx.x];
    __syncthreads();
    for (long long t0 = 0; t0 < v.nsel - k0; t0 += ACF_TT) {
      __syncthreads();
      load_centred(v, w, t0, ACF_TT, smu, A, SA);
      load_centred(v, w, t0 + k0, SB, smu, B, SB);
      __syncthreads();
      if (active) {
        const double *a = A + d * SA;
        const double *bb = B + d * SB + ACF_R * lg;
        double win[2 * ACF_R];
#pragma unroll
        for (int r = 0; r < ACF_R; ++r) win[ACF_R + r] = bb[r];
        for (int t = 0; t < ACF_TT; t += ACF_R) {
#pragma unroll
          for (int r = 0; r < ACF_R; ++r) {
            win[r] = win[ACF_R + r];
            win[ACF_R + r] = bb[t + ACF_R + r];
          }
#pragma unroll
          for (int u = 0; u < ACF_R; ++u) {
            const double x = a[t + u];
#pragma unroll
            for (int r = 0; r < ACF_R; ++r) acc[r] = fma(x, win[u + r], acc[r]);
          }
        }
      }
    }
    if (active) {
      const double q = c0[w * v.ndim + d];
#pragma unroll
      for (int r = 0; r < ACF_R; ++r) rsum[r] += acc[r] / q;
    }
  }
  if (active) {
#pragma unroll
    for (int r = 0; r < ACF_R; ++r) {
      const int l = ACF_R * lg + r;
      if (l < nl) partial[(b * nl + l) * v.ndim + d] = rsum[r];
    }
  }
}

// rho_sum[src][off + l][d] (rows of nl_all lags) = sum of the partials of src's blocks, in block order
__global__ void k_acf_reduce(View v, int nl, long long ng0, long long ngW, long long nloc_src,
                             const double *__restrict__ partial, double *__restrict__ rho_sum, long long nl_all,
                             long long off) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per = (long long)nl * v.ndim;
  if (idx >= nloc_src * per) return;
  const long long s = idx / per, r = idx % per;
  const long long b0 = (s == 0) ? 0 : ng0 + (s - 1) * ngW;
  long long lo, hi;
  local_range(v, s, lo, hi);
  const long long nb = (hi - lo + ACF_GROUP - 1) / ACF_GROUP;
  double acc = 0.0;
  for (long long b = b0; b < b0 + nb; ++b) acc += partial[b * per + r];
  rho_sum[((v.src0 + s) * nl_all + off) * v.ndim + r] = acc;
}

}  // namespace cs
