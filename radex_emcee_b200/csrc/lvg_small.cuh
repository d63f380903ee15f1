// lvg_small.cuh -- the cached engine of lvg_v2.cuh as kernels of its own, one instantiation per lead-block size:
// one HALF-WARP per model for lead blocks of 12/16 levels, one warp per model for 20/24/28.
//
// 93 % of the matrix() calls of the forward sweep are cached iterations (lvg_v2.cuh: CACHED): a lead block of
// n = 4 KP levels eliminated one row per lane, the frozen levels through the response matrix.  Inside
// k_lvg_solve_v2 they pay for the full engine they do not use (an 18.8 KB slab, 168 registers: 12 warps per SM), and
// for n <= 16 -- three quarters of the sweep, nearly all of a converged ensemble -- half of the warp idles.  Here
// every lead size has its own instantiation and launch: the pivot loops are straight-line code with constant
// addresses, the slab holds just lead block + response matrix + pivot buffers + per-model line state (6.4 .. 15 KB),
// and for n <= 16 two models share a warp (lanes 0-15 / 16-31, each half with its own slab, iteration state and
// queue ticket): 36 / 28 / 20 / 16 / 14 models per SM for 12 / 16 / 20 / 24 / 28 lead levels.
// There is NO full elimination in these kernels: launch A (v2::solve, sched = 1) captures the frozen top of a model
// and parks lead block, response matrix and line bases (v2::ext_size(n) doubles); a model whose frozen lines turn thick is
// parked again and finished by launch C (v2::solve, sched = 4).
//
// Per model the arithmetic is the one of v2::lead_solve and of the iteration loop of v2::solve, operation for
// operation and in the same association (in a half-warp the 32-lane butterflies are reproduced as "pair, then
// 16-lane butterfly"), so the results are bit-identical to the single-launch path
// (tests/test_gpu_solve.py::test_two_launch_schedule_is_bit_identical, ::test_ordered_launches_...).
//
// What it replaces: the calls 2.. of matrix() + lubksb (emcee/pyradex/radex/radex.so@0x17f70, 0x17cb0) made
// by run_radex's loop (emcee/pyradex/core.py:856-925) for these models.
#pragma once

// V2S_TWO_ROWS = 1: the 20/24/28-level engines also run two models per warp, every lane of a half-warp holding TWO rows
// of its model's lead block (rows hl and hl + 16); 0: one model per warp, one row per lane (12 / 8 / 4 lanes idle)
#ifndef V2S_TWO_ROWS
#define V2S_TWO_ROWS 1
#endif
#ifndef V2S_WARPS5
#define V2S_WARPS5 (V2S_TWO_ROWS ? 10 : 20)
#endif
#ifndef V2S_WARPS6
#define V2S_WARPS6 (V2S_TWO_ROWS ? 8 : 17)
#endif
#ifndef V2S_WARPS7
#define V2S_WARPS7 (V2S_TWO_ROWS ? 7 : 15)
#endif

namespace v2s {

using v2::MP;
using v2::NL;
using v2::ld2;
using v2::st2;

using v2::KP_SMALL_MAX;               // largest lead block (in panels) with an engine here
using v2::EXT_LEAD;
// ---- per-model shared-memory slab (doubles), for a lead block of N = 4 KP levels -------------------------
// KP = 3: 796 doubles (6368 B, 36 models = 18 warps per SM); KP = 4: 1026 doubles (8208 B, 28 models = 14 warps)
template <int KP>
struct Lay {
  static constexpr int N = 4 * KP;
  static constexpr int G = (KP <= 4 || V2S_TWO_ROWS) ? 16 : 32;   // lanes per model: a half-warp (two rows per lane above 16 lead levels), or a warp
  static constexpr int MPW = 32 / G;                  // models per warp
  static constexpr int NT = (v2::MAXLINE + G - 1) / G;   // trips over the lines
  // lines that may be lead lines (both levels below N): the first 16 (KP <= 4) or 32.  A CO-like table has its N - 1
  // lead lines there; the engines only run tables that do (lead_lines_fit), so the per-line slots that only lead
  // lines read (S_BETA, S_DNB, S_UPB) exist for these lines only, and the trips LEAD_TRIPS are the only ones patched
  static constexpr int NLEAD = (KP <= 4) ? 16 : 32;
  static constexpr unsigned LEAD_TRIPS = (1u << (NLEAD / G)) - 1u;
  static constexpr int S_LEAD = 0;                    // lead block, row pitch N + 2
  static constexpr int S_M = N * (N + 2);             // M[i][f]: frozen populations from the lead ones, pitch 42 - N
  static constexpr int PBW = (N > 16) ? 32 : 16;      // a pivot row has up to N - 1 entries + 1/s_k in slot K
  static constexpr int S_PB = S_M + N * (MP - N);     // pivot-row broadcast buffers, 2 x PBW (1/s_k rides in slot K)
  static constexpr int S_VT = S_PB + 2 * PBW;         // raw pivot columns, triangular
  static constexpr int S_X = S_VT + N * (N - 1) / 2;  // relaxed populations
  static constexpr int S_XNEW = S_X + NL;             // un-relaxed populations of this call
  static constexpr int S_BETA = S_XNEW + NL;          // per line < NLEAD: escape probability of the call about to be made
  static constexpr int S_DNB = S_BETA + NLEAD;        //                   non-radiative part of q[m][n] (collisions + Schur term)
  static constexpr int S_UPB = S_DNB + NLEAD;         //                   non-radiative part of q[n][m]
  static constexpr int S_TEX = S_UPB + NLEAD;         // per line: excitation temperature
  static constexpr int SSLAB = S_TEX + 40;
  // warps per CTA: bounded by the 227 KB of shared memory and by 65536 registers / (32 x registers per thread)
  static constexpr int WARPS = (KP == 3) ? 18 : (KP == 4) ? 14 : (KP == 5) ? V2S_WARPS5 : (KP == 6) ? V2S_WARPS6 : V2S_WARPS7;
  static_assert(SSLAB % 2 == 0 && S_M % 2 == 0 && S_PB % 2 == 0 && S_X % 2 == 0 && S_DNB % 2 == 0 && S_UPB % 2 == 0,
                "16 B alignment of the slab parts");
};
// ---- per-CTA constants (the same for every model of a call) --------------------------------------------
constexpr int C_LA = 0, C_LGR = 40, C_LTDEN = 80, C_LECOEF = 120, C_LFKXNU = 160, C_LMN = 200, C_XNU = 220, C_BACKI = 260,
              CSLAB = 300;
// parked capture (global, per model; v2::ext_size(n) doubles at io.ext + io.ext_off[model]): DNB[40] UPB[40] lead[n(n+2)] M[n(42-n)]
template <int KP>
constexpr size_t smem_bytes() { return (size_t)(CSLAB + Lay<KP>::MPW * Lay<KP>::WARPS * Lay<KP>::SSLAB) * sizeof(double); }
static_assert(smem_bytes<3>() <= 232448 && smem_bytes<4>() <= 232448 && smem_bytes<5>() <= 232448 &&
                  smem_bytes<6>() <= 232448 && smem_bytes<7>() <= 232448,
              "slabs exceed the 227 KB of shared memory per CTA");

// Do the lead lines of every engine lie in its first NLEAD lines?  Decided once per molecule table; a table that fails
// runs its cached iterations in launch B instead (SolveCfg::small off), with the same arithmetic.
template <int KP>
inline bool lead_lines_fit_kp(const int *iupp, const int *ilow, int nline) {
  for (int l = Lay<KP>::NLEAD; l < nline; ++l)
    if (std::max(iupp[l], ilow[l]) < Lay<KP>::N) return false;
  return true;
}
inline bool lead_lines_fit(const int *iupp, const int *ilow, int nline) {
  return lead_lines_fit_kp<3>(iupp, ilow, nline) && lead_lines_fit_kp<4>(iupp, ilow, nline) &&
         lead_lines_fit_kp<5>(iupp, ilow, nline) && lead_lines_fit_kp<6>(iupp, ilow, nline) &&
         lead_lines_fit_kp<7>(iupp, ilow, nline);
}

// ---- hand-over of a model: 16-byte asynchronous copies global -> shared (SASS: LDGSTS), all in flight at once ----
__device__ __forceinline__ void cp_async16(double *dst_smem, const double *src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(v2::smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

template <int G>
__device__ __forceinline__ double group_sum(double v) {   // butterfly over the G lanes of a model
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// integer reductions over the lanes of a model: one REDUX instruction on the model's lane mask
__device__ __forceinline__ int group_sum_int(unsigned mask, int v) { return __reduce_add_sync(mask, v); }
__device__ __forceinline__ int group_max_int(unsigned mask, int v) { return __reduce_max_sync(mask, v); }

template <int LO, int HI, int NR>
__device__ __forceinline__ double sum_range(const double (&q)[NR]) {   // same association as v2::sum_range
  if constexpr (HI - LO == 1) {
    return q[LO];
  } else {
    constexpr int MID = (LO + HI) / 2;
    return sum_range<LO, MID, NR>(q) + sum_range<MID, HI, NR>(q);
  }
}

// v2::lead_pivots with hl = lane within the half; both halves run the same pivot on their own block.
template <int K, int LO, int NR, int G>
__device__ __forceinline__ void lead_pivots(double (&q)[NR], double &rmine, double *pbase, double *vt,
                                            const int hl) {
  if constexpr (K >= LO) {
    const double s = sum_range<0, K, NR>(q);
    const double rr = v2::rcp1(s);
    const double r = (s > 0.0) ? rr : 0.0;
    double *pb = pbase + (K & 1) * ((NR > 16) ? 32 : 16);
    if (hl == K) {
      rmine = r;
#pragma unroll
      for (int j = 0; j + 1 < K; j += 2) st2(pb + j, q[j], q[j + 1]);
      if (K & 1) pb[K - 1] = q[K - 1];
      pb[K] = r;
    }
    __syncwarp();
    const double w = q[K];
    if (hl < K) vt[K * (K - 1) / 2 + hl] = w;
    const double wv = w * pb[K];
#pragma unroll
    for (int j = 0; j < K; j += 2) {
      const double2 u = ld2(pb + j);
      q[j] = fma(wv, u.x, q[j]);
      if (j + 1 < K) q[j + 1] = fma(wv, u.y, q[j + 1]);
    }
    lead_pivots<K - 1, LO, NR, G>(q, rmine, pbase, vt, hl);
  }
}

// ---- two rows per lane: a half-warp eliminates a lead block of 17 .. 32 levels, lane hl holding rows hl and hl + 16 --------
// Pivot K belongs to lane K & 15, row slot K >> 4.  The arithmetic per row is that of lead_pivots (same sums, same
// reciprocal, same FMAs in the same order); only where a row lives changes.
template <int K, int NR>
__device__ __forceinline__ void lead_pivots2(double (&q0)[NR], double (&q1)[NR], double &r0, double &r1, double *pbase,
                                             double *vt, const int hl) {
  if constexpr (K >= 1) {
    constexpr int SLOT = K >> 4, OWN = K & 15;
    double s;
    if constexpr (SLOT) s = sum_range<0, K, NR>(q1); else s = sum_range<0, K, NR>(q0);
    const double rr = v2::rcp1(s);
    const double r = (s > 0.0) ? rr : 0.0;
    double *pb = pbase + (K & 1) * 32;
    if (hl == OWN) {
      if constexpr (SLOT) {
        r1 = r;
#pragma unroll
        for (int j = 0; j + 1 < K; j += 2) st2(pb + j, q1[j], q1[j + 1]);
        if (K & 1) pb[K - 1] = q1[K - 1];
      } else {
        r0 = r;
#pragma unroll
        for (int j = 0; j + 1 < K; j += 2) st2(pb + j, q0[j], q0[j + 1]);
        if (K & 1) pb[K - 1] = q0[K - 1];
      }
      pb[K] = r;
    }
    __syncwarp();
    const double pr = pb[K];
    const double w0 = q0[K];
    if (hl < K) vt[K * (K - 1) / 2 + hl] = w0;
    const double wv0 = w0 * pr;
    double wv1 = 0.0;
    if constexpr (K > 16) {
      const double w1 = q1[K];
      if (hl + 16 < K) vt[K * (K - 1) / 2 + hl + 16] = w1;
      wv1 = w1 * pr;
    }
#pragma unroll
    for (int j = 0; j < K; j += 2) {
      const double2 u = ld2(pb + j);
      q0[j] = fma(wv0, u.x, q0[j]);
      if (j + 1 < K) q0[j + 1] = fma(wv0, u.y, q0[j + 1]);
      if constexpr (K > 16) {
        q1[j] = fma(wv1, u.x, q1[j]);
        if (j + 1 < K) q1[j + 1] = fma(wv1, u.y, q1[j + 1]);
      }
    }
    lead_pivots2<K - 1, NR>(q0, q1, r0, r1, pbase, vt, hl);
  }
}

template <int I, int NM1>
__device__ __forceinline__ void lead_back2(double &Y0, double &Y1, double &F1, double &F2, double &xi, double &psum,
                                           double &x0, double &x1, const double r0, const double r1, const double *vt0,
                                           const double *vt1, const double *Mc1, const double *Mc2, const int pitch,
                                           const int hl) {
  if constexpr (I < NM1) {
    Y0 = fma(xi, vt0[I], Y0);
    Y1 = fma(xi, vt1[I], Y1);
    F1 = fma(xi, Mc1[I * pitch], F1);
    F2 = fma(xi, Mc2[I * pitch], F2);
    constexpr int LVL = I + 1, SLOT = LVL >> 4, OWN = LVL & 15;
    xi = __shfl_sync(0xffffffffu, SLOT ? r1 * Y1 : r0 * Y0, OWN, 16);
    psum += xi;
    if (hl == OWN) {
      if constexpr (SLOT) x1 = xi; else x0 = xi;
    }
    lead_back2<I + 1, NM1>(Y0, Y1, F1, F2, xi, psum, x0, x1, r0, r1, vt0, vt1, Mc1, Mc2, pitch, hl);
  }
}

template <int KP>
__device__ __forceinline__ double lead_solve2(double *sm, const int hl, long long *tmid = nullptr) {
  using L = Lay<KP>;
  constexpr int n = L::N;
  static_assert(n > 16 && n <= 32 && L::G == 16, "two rows per lane: 17 .. 32 lead levels in a half-warp");
  double *B = sm + L::S_LEAD;
  double q0[n], q1[n];
  {
    const double *row0 = B + hl * (n + 2), *row1 = B + ((hl + 16 < n) ? hl + 16 : 0) * (n + 2);
#pragma unroll
    for (int j = 0; j < n; j += 4) {
      const double2 a = ld2(row0 + j), b = ld2(row0 + j + 2), c = ld2(row1 + j), d = ld2(row1 + j + 2);
      q0[j] = a.x; q0[j + 1] = a.y; q0[j + 2] = b.x; q0[j + 3] = b.y;
      q1[j] = c.x; q1[j + 1] = c.y; q1[j + 2] = d.x; q1[j + 3] = d.y;
    }
  }
  double r0 = 0.0, r1 = 0.0;
  double *pbase = sm + L::S_PB, *vtb = sm + L::S_VT;
  lead_pivots2<n - 1, n>(q0, q1, r0, r1, pbase, vtb, hl);
  __syncwarp();   // Vt complete
#ifdef V2S_TIMING
  if (tmid) *tmid = clock64();
#endif
  constexpr int nf = NL - n, pitch = MP - n;
  const int l1 = hl + 16;
  const double *vt0 = vtb + hl * (hl - 1) / 2;
  const double *vt1 = vtb + ((l1 < n) ? l1 * (l1 - 1) / 2 : 0);   // lanes without a second row only go through the motions
  const bool one = hl < nf, two = hl + 16 < nf;
  const double *Mc1 = sm + L::S_M + (one ? hl : 0), *Mc2 = sm + L::S_M + (two ? hl + 16 : 0);
  double Y0 = 0.0, Y1 = 0.0, F1 = 0.0, F2 = 0.0, xi = 1.0, psum = 1.0, x0 = 1.0, x1 = 0.0;
  lead_back2<0, n - 1>(Y0, Y1, F1, F2, xi, psum, x0, x1, r0, r1, vt0, vt1, Mc1, Mc2, pitch, hl);
  F1 = fma(xi, Mc1[(n - 1) * pitch], F1);
  F2 = fma(xi, Mc2[(n - 1) * pitch], F2);
  sm[L::S_XNEW + hl] = x0;
  if (l1 < n) sm[L::S_XNEW + l1] = x1;
  if (one) sm[L::S_XNEW + n + hl] = F1;
  if (two) sm[L::S_XNEW + n + 16 + hl] = F2;
  // v2: psum + warp_sum(lane < nf ? F : 0): the first butterfly step pairs lane l with l + 16
  return psum + group_sum<16>((one ? F1 : 0.0) + (two ? F2 : 0.0));
}

// v2::lead_solve for the G lanes of one model and a lead block of N = 4 KP levels.
template <int KP>
__device__ __forceinline__ double lead_solve(double *sm, const int hl, long long *tmid = nullptr) {
  using L = Lay<KP>;
  constexpr int n = L::N, G = L::G;
  if constexpr (n > G) {
    return lead_solve2<KP>(sm, hl, tmid);
  } else {
    double *B = sm + L::S_LEAD;
    double q[n];
    {
      const double *row = B + ((hl < n) ? hl : 0) * (n + 2);
  #pragma unroll
      for (int j = 0; j < n; j += 4) {
        const double2 a = ld2(row + j), b = ld2(row + j + 2);
        q[j] = a.x; q[j + 1] = a.y; q[j + 2] = b.x; q[j + 3] = b.y;
      }
    }
    double rmine = 0.0;
    double *pbase = sm + L::S_PB, *vtb = sm + L::S_VT;
    lead_pivots<n - 1, 1, n, G>(q, rmine, pbase, vtb, hl);
    __syncwarp();   // Vt complete
#ifdef V2S_TIMING
    if (tmid) *tmid = clock64();
#endif
    // frozen levels: lane hl owns n + hl and, in a half-warp (29 or 25 of them), n + 16 + hl
    constexpr int nf = NL - n, pitch = MP - n;
    const double *vt = vtb + ((hl < n) ? hl * (hl - 1) / 2 : 0);   // lanes >= n only go through the motions: stay inside the slab
    const bool one = hl < nf, two = (G == 16) && (hl + 16 < nf);
    const double *Mc1 = sm + L::S_M + (one ? hl : 0), *Mc2 = sm + L::S_M + (two ? hl + 16 : 0);
    double Y = 0.0, F1 = 0.0, F2 = 0.0, xi = 1.0, psum = 1.0, xmine = 1.0;
  #pragma unroll
    for (int i = 0; i < n - 1; ++i) {
      Y = fma(xi, vt[i], Y);
      F1 = fma(xi, Mc1[i * pitch], F1);
      if (G == 16) F2 = fma(xi, Mc2[i * pitch], F2);
      xi = __shfl_sync(0xffffffffu, rmine * Y, i + 1, G);
      psum += xi;
      xmine = (hl == i + 1) ? xi : xmine;
    }
    F1 = fma(xi, Mc1[(n - 1) * pitch], F1);
    if (G == 16) F2 = fma(xi, Mc2[(n - 1) * pitch], F2);
    if (hl < n) sm[L::S_XNEW + hl] = xmine;
    if (one) sm[L::S_XNEW + n + hl] = F1;
    if (two) sm[L::S_XNEW + n + 16 + hl] = F2;
    // v2: psum + warp_sum(lane < nf ? F : 0); in a half-warp the first butterfly step pairs lane l with l + 16
    if (G == 16) return psum + group_sum<G>(F1 + (two ? F2 : 0.0));
    return psum + group_sum<G>(one ? F1 : 0.0);
  }
}

}  // namespace v2s
