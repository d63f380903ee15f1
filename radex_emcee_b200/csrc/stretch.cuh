// stretch.cuh -- the stretch move over an ensemble that stays in place (second form of the C ABI, radex_b200.h):
// red/blue split as a function of (seed, step, global walker id), sub-ensembles per fitted source, per-walker
// acceptance counters, NaN detection.
//
// What it replaces: emcee's RedBlueMove.propose + StretchMove.get_proposal with the default randomize_split=True
// (un-vendored; call sites emcee/emcee_radex.py:483-499, emcee/emcee_radex_2comp.py:557-574; SURVEY.md 3.5):
//     inds = arange(nwalkers) % 2 ; random.shuffle(inds)        -> a balanced random labelling, new every step
//     for split in (0, 1): s = coords[inds == split], c = coords[inds != split]
//         zz = ((a - 1) u + 1)^2 / a ; rint = randint(len(c)) ; q = c[rint] - (c[rint] - s) zz ; factors = (ndim - 1) ln zz
//         accept where factors + lnp_new - lnp_old > ln u'
// Here the labelling is balanced per BLOCK of consecutive walkers and is drawn from a keyed bijection, so that every
// rank can evaluate it for any walker without communication and the chain does not depend on the rank count.
#pragma once

namespace st2 {

struct SplitDev {
  long long W;        // walkers per source (sub-ensemble)
  int B;              // split block, B | W, even
  int w;              // bits: 2^w >= B
  int randomize;
  unsigned k0, k1;    // Philox key of the split stream
};

// keys of block gb at step `step`: one Philox call; the stream is separated from the proposal / accept streams by
// the key (seed ^ 'SPLTrand'), not by the counter
__device__ __host__ inline void split_key_words(unsigned long long seed, unsigned &k0, unsigned &k1) {
  k0 = (unsigned)seed ^ 0x53504C54u;
  k1 = (unsigned)(seed >> 32) ^ 0x72616E64u;
}

__device__ __forceinline__ void split_keys(const SplitDev &sp, unsigned long long gb, unsigned long long step, uint32_t k[4]) {
  k[0] = (uint32_t)gb;
  k[1] = (uint32_t)(gb >> 32);
  k[2] = (uint32_t)step;
  k[3] = (uint32_t)(step >> 32);
  philox4x32_10(k, sp.k0, sp.k1);
}

// keyed bijection of [0, B): four rounds of (odd multiply + key) mod 2^w and xor-shift, each invertible on w bits;
// values >= B walk the cycle until they are back inside (every cycle of a bijection of [0, 2^w) that starts inside
// [0, B) returns there)
__device__ __forceinline__ unsigned split_perm(unsigned x, const SplitDev &sp, const uint32_t k[4]) {
  const unsigned mask = (sp.w >= 32) ? 0xffffffffu : ((1u << sp.w) - 1u);
  const int s1 = (sp.w + 1) >> 1, s2 = (sp.w >= 3) ? sp.w / 3 : 1;
  do {
    x = (x * 0x9E3779B1u + k[0]) & mask; x ^= x >> s1;
    x = (x * 0x85EBCA6Bu + k[1]) & mask; x ^= x >> s2;
    x = (x * 0xC2B2AE35u + k[2]) & mask; x ^= x >> s1;
    x = (x * 0x27D4EB2Fu + k[3]) & mask; x ^= x >> s2;
  } while (x >= (unsigned)sp.B);
  return x;
}

// k-group split: in a block of B walkers group g of ngroups has n_g = B / ngroups + (g < B % ngroups) slots, which follow
// the off_g = sum_{h<g} n_h slots of the groups before it.  ngroups = 2 is the stretch move's red/blue split (n_g = B/2),
// ngroups = 3 the differential-evolution move's (emcee's DEMove: nsplits = 3).
__host__ __device__ inline int group_size(int B, int ngroups, int g) { return B / ngroups + (g < B % ngroups ? 1 : 0); }
__host__ __device__ inline int group_off(int B, int ngroups, int g) {
  return g * (B / ngroups) + (g < B % ngroups ? g : B % ngroups);
}

// index within its block of slot t of group g in global block gb: pi(off_g + t) (randomize), g + ngroups t otherwise
__device__ __forceinline__ long long block_walker(const SplitDev &sp, unsigned long long step, int g, int ngroups,
                                                  unsigned long long gb, int t) {
  if (!sp.randomize) return g + (long long)ngroups * t;
  uint32_t key[4];
  split_keys(sp, gb, step, key);
  return split_perm((unsigned)(group_off(sp.B, ngroups, g) + t), sp, key);
}

// local walker index of local slot k of group g (rank owns [gid_base, gid_base + nlocal), B | gid_base).  For ngroups = 2
// this is the red/blue split of the stretch move: half h, slot t of block b -> b B + pi(h B/2 + t), or 2t + h.
__device__ __forceinline__ long long slot_walker(const SplitDev &sp, unsigned long long step, int g, int ngroups,
                                                 long long gid_base, long long k) {
  const int n = group_size(sp.B, ngroups, g);
  const long long lb = k / n;
  const int t = (int)(k - lb * n);
  return lb * sp.B + block_walker(sp, step, g, ngroups, (unsigned long long)(gid_base / sp.B + lb), t);
}

__device__ __forceinline__ unsigned long long step_of(const unsigned long long *step_ptr, unsigned long long step) {
  return step + (step_ptr ? *step_ptr : 0ULL);
}

// ---- differential-evolution move (emcee's DEMove; ter Braak 2006, Nelson et al. 2013) -----------------------------------
// Three groups per step (the k-group split above with ngroups = 3), moved one after the other; group g's walker s moves
// to q = s + gamma (c[j2] - c[j1]), (j1, j2) uniform over the ordered pairs of distinct walkers of the complement c of
// group g within the walker's source (the other two groups as they stand after the earlier sub-steps, concatenated in
// group order, each in global slot order), gamma = gamma0 (1 + sigma n), n ~ N(0, 1) per walker; log factor 0.
// Its streams are separated from the stretch and split streams by the key (seed ^ 'DEmvmove'); the counter is
// (global id, 4 step + group, draw), draw DE_PAIR, then DE_GAUSS + t for the t-th try of the Gaussian, DE_ACCEPT.
enum { DE_PAIR = 0, DE_GAUSS = 1, DE_ACCEPT = 255, DE_MAX_TRIES = 200 };

__host__ __device__ inline void de_key_words(unsigned long long seed, unsigned &k0, unsigned &k1) {
  k0 = (unsigned)seed ^ 0x44456D76u;
  k1 = (unsigned)(seed >> 32) ^ 0x6D6F7665u;
}

__host__ __device__ inline void de_counter(uint32_t c[4], unsigned long long gid, unsigned long long step, int g, int draw) {
  const unsigned long long sg = step * 4ULL + (unsigned)g;
  c[0] = (uint32_t)gid;
  c[1] = (uint32_t)(gid >> 32);
  c[2] = (uint32_t)sg;
  c[3] = ((uint32_t)(sg >> 32) & 0x00ffffffu) | ((uint32_t)draw << 24);
}

// ln x for 0 < x < 1 from IEEE operations only (no library transcendental, whose last bit differs between CUDA and libm),
// so that the numpy restatement reproduces it bit for bit: x = m 2^e, m in [1/sqrt 2, sqrt 2), ln x = e ln 2 + 2 atanh(s)
// with s = (m - 1) / (m + 1), |s| < 0.1716, and the odd series of atanh to s^21 (truncation < 1e-17 relative)
__device__ __forceinline__ double ln_rn(double x) {
  int e;
  double m = frexp(x, &e);
  if (m < 0.70710678118654752) {
    m = __dmul_rn(m, 2.0);
    e -= 1;
  }
  const double s = __ddiv_rn(__dsub_rn(m, 1.0), __dadd_rn(m, 1.0)), s2 = __dmul_rn(s, s);
  double p = __ddiv_rn(1.0, 21.0);
#pragma unroll
  for (int k = 19; k >= 1; k -= 2) p = __dadd_rn(__ddiv_rn(1.0, (double)k), __dmul_rn(s2, p));
  return __dadd_rn(__dmul_rn((double)e, 0.69314718055994531), __dmul_rn(2.0, __dmul_rn(s, p)));
}

// one N(0, 1) draw of walker gid at sub-step (step, g): Box-Muller in Marsaglia's polar form (no cosine), tries
// DE_GAUSS, DE_GAUSS + 1, ... until v1^2 + v2^2 lies in (0, 1); P(reject) = 1 - pi/4 per try
__device__ __forceinline__ double de_gauss(unsigned long long gid, unsigned long long step, int g, unsigned k0, unsigned k1) {
  for (int t = 0; t < DE_MAX_TRIES; ++t) {
    uint32_t c[4];
    de_counter(c, gid, step, g, DE_GAUSS + t);
    philox4x32_10(c, k0, k1);
    const double v1 = __dsub_rn(__dmul_rn(2.0, u01(c[0], c[1])), 1.0), v2 = __dsub_rn(__dmul_rn(2.0, u01(c[2], c[3])), 1.0);
    const double r = __dadd_rn(__dmul_rn(v1, v1), __dmul_rn(v2, v2));
    if (r > 0.0 && r < 1.0) return __dmul_rn(v1, __dsqrt_rn(__ddiv_rn(__dmul_rn(-2.0, ln_rn(r)), r)));
  }
  // all DE_MAX_TRIES tries rejected: probability (1 - pi/4)^200 < 1e-130 per draw, never seen; n = 0 (gamma = gamma0)
  return 0.0;
}

// global walker id of index j of the complement of group g (of 3) within source src
__device__ __forceinline__ long long de_partner(const SplitDev &sp, unsigned long long step, int g, long long src, long long j) {
  const long long bps = sp.W / sp.B;   // blocks per source
  int h = (g == 0) ? 1 : 0;   // the complement: groups (1, 2), (0, 2) or (0, 1)
  const long long n_first = bps * group_size(sp.B, 3, h);
  if (j >= n_first) {
    j -= n_first;
    h = (g == 2) ? 1 : 2;
  }
  const int n = group_size(sp.B, 3, h);
  const long long lb = j / n;
  const unsigned long long gb = (unsigned long long)(src * bps + lb);
  return (long long)gb * sp.B + block_walker(sp, step, h, 3, gb, (int)(j - lb * n));
}

// one thread per local slot of group g: Q[k] = s + gamma (Xall[w2] - Xall[w1]); Xall[nwalkers, ndim] is the whole
// ensemble in global walker order (one rank: X itself)
__global__ void k_de_propose(SplitDev sp, const unsigned long long *step_ptr, unsigned long long step_, int g,
                             long long gid_base, long long nslots, int ndim, const double *X, const double *Xall,
                             double gamma0, double sigma, unsigned long long seed, double *Q, int *src_id) {
  const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= nslots) return;
  const unsigned long long step = step_of(step_ptr, step_);
  const long long i = slot_walker(sp, step, g, 3, gid_base, k);
  const unsigned long long gid = (unsigned long long)(gid_base + i);
  const long long src = (long long)(gid / (unsigned long long)sp.W);
  const long long nc = sp.W - (sp.W / sp.B) * group_size(sp.B, 3, g);
  unsigned k0, k1;
  de_key_words(seed, k0, k1);
  uint32_t c[4];
  de_counter(c, gid, step, g, DE_PAIR);
  philox4x32_10(c, k0, k1);
  const long long npair = nc * (nc - 1);
  long long p = (long long)(u01(c[0], c[1]) * (double)npair);
  if (p >= npair) p = npair - 1;
  const long long j1 = p / (nc - 1), r = p - j1 * (nc - 1), j2 = r + (r >= j1 ? 1 : 0);
  const long long w1 = de_partner(sp, step, g, src, j1), w2 = de_partner(sp, step, g, src, j2);
  const double gamma = __dmul_rn(gamma0, __dadd_rn(1.0, __dmul_rn(sigma, de_gauss(gid, step, g, k0, k1))));
  for (int d = 0; d < ndim; ++d)
    Q[k * ndim + d] = __dadd_rn(X[i * ndim + d], __dmul_rn(gamma, __dsub_rn(Xall[w2 * ndim + d], Xall[w1 * ndim + d])));
  if (src_id) src_id[k] = (int)src;
}

__global__ void k_pack(SplitDev sp, const unsigned long long *step_ptr, unsigned long long step_, int group, int ngroups,
                       long long gid_base, long long nslots, int ndim, const double *X, double *Chalf) {
  const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= nslots) return;
  const long long i = slot_walker(sp, step_of(step_ptr, step_), group, ngroups, gid_base, k);
  for (int d = 0; d < ndim; ++d) Chalf[k * ndim + d] = X[i * ndim + d];
}

__global__ void k_propose2(SplitDev sp, const unsigned long long *step_ptr, unsigned long long step_, int half,
                           long long gid_base, long long nhalf, int ndim, const double *X, const double *Call, double a,
                           unsigned long long seed, double *Q, double *logfac, int *src_id) {
  const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= nhalf) return;
  const unsigned long long step = step_of(step_ptr, step_);
  const long long i = slot_walker(sp, step, half, 2, gid_base, k);
  const unsigned long long gid = (unsigned long long)(gid_base + i);
  uint32_t c[4] = {(uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)(step * 2ULL + (unsigned)half),
                   (uint32_t)((step * 2ULL + (unsigned)half) >> 32) & 0x7fffffffu};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  const double u = u01(c[0], c[1]);
  const double sq = __dadd_rn(__dmul_rn(a - 1.0, u), 1.0);
  const double z = __dmul_rn(sq, sq) / a;
  const long long src = (long long)(gid / (unsigned long long)sp.W), nc = sp.W >> 1;
  long long j = (long long)(u01(c[2], c[3]) * (double)nc);
  if (j >= nc) j = nc - 1;
  j += src * nc;   // the complementary half of the walker's own sub-ensemble, in global slot order
  for (int d = 0; d < ndim; ++d) {
    const double cj = Call[j * ndim + d], s = X[i * ndim + d];
    Q[k * ndim + d] = __dsub_rn(cj, __dmul_rn(cj - s, z));
  }
  logfac[k] = (ndim - 1.0) * log(z);
  if (src_id) src_id[k] = (int)src;
}

// accept test of the slots of group `group` of ngroups.  de = 0: the stretch move's accept stream (key = seed); de = 1: the
// differential-evolution move's (key de_key_words(seed), counter de_counter(..., DE_ACCEPT)).  logfac NULL: a log factor
// of 0 (DEMove).
__global__ void k_accept2(SplitDev sp, const unsigned long long *step_ptr, unsigned long long step_, int group, int ngroups,
                          int de, long long gid_base, long long nslots, int ndim, double *X, double *lnp, const double *Q,
                          const double *lnp_new, const double *logfac, unsigned long long seed, long long *naccept,
                          unsigned long long *nan_count, const unsigned long long *nsolves_src,
                          unsigned long long *nsolves_sum, int *accepted = nullptr) {
  const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  int isnan_ = 0;
  if (k < nslots) {
    const unsigned long long step = step_of(step_ptr, step_);
    const long long i = slot_walker(sp, step, group, ngroups, gid_base, k);
    const unsigned long long gid = (unsigned long long)(gid_base + i);
    uint32_t c[4];
    if (de) {
      unsigned k0, k1;
      de_key_words(seed, k0, k1);
      de_counter(c, gid, step, group, DE_ACCEPT);
      philox4x32_10(c, k0, k1);
    } else {
      c[0] = (uint32_t)gid;
      c[1] = (uint32_t)(gid >> 32);
      c[2] = (uint32_t)(step * 2ULL + (unsigned)group);
      c[3] = ((uint32_t)((step * 2ULL + (unsigned)group) >> 32) & 0x7fffffffu) | 0x80000000u;
      philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    }
    const double lnu = log(u01(c[0], c[1]));
    const double lnew = lnp_new[k];
    isnan_ = (lnew != lnew);
    const double lnpdiff = (logfac ? logfac[k] : 0.0) + lnew - lnp[i];
    const bool acc = lnpdiff > lnu;   // -inf - -inf = NaN compares false -> rejected, like numpy
    if (acc) {
      for (int d = 0; d < ndim; ++d) X[i * ndim + d] = Q[k * ndim + d];
      lnp[i] = lnew;
      if (naccept) naccept[i] += 1;   // one slot per walker per sub-step: no atomics needed
    }
    if (accepted) accepted[k] = acc ? 1 : 0;
  }
  const unsigned nanb = __ballot_sync(0xffffffffu, isnan_);
  if ((threadIdx.x & 31) == 0 && nanb && nan_count) atomicAdd(nan_count, (unsigned long long)__popc(nanb));
  if (k == 0 && nsolves_sum && nsolves_src) atomicAdd(nsolves_sum, *nsolves_src);
}

// ---- speculative second half-step (small ensembles) -------------------------------------------------------------------
// A step of a small ensemble is bound by the latency of ONE solve per half-step (config 1: 50 models on 148 SMs, ~100
// sequential calls of matrix() each).  The second half-step depends on the first only through the partner c_j of every
// proposal, and c_j is one of two known points: where it stood, or the first half-step's proposal for it.  So both
// candidates are proposed before anything is solved, the nhalf + 2 nhalf models go through ONE lnprob launch, and after
// the first half-step's accept/reject the candidate the sequential move would have made is selected.  Same random
// numbers, same arithmetic per candidate: the chain is the sequential one bit for bit; a step costs one solve latency
// and 1.5 times the solves.
// Cold: the walkers of half 0 in slot order BEFORE their move (k_pack); Q0: half 0's proposals, same slot order.
__global__ void k_propose_spec(SplitDev sp, const unsigned long long *step_ptr, unsigned long long step_, long long gid_base,
                               long long nhalf, int ndim, const double *X, const double *Cold, const double *Q0, double a,
                               unsigned long long seed, double *Qa, double *Qb, double *logfac, int *jpart, int *src_a,
                               int *src_b) {
  const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= nhalf) return;
  const int half = 1;
  const unsigned long long step = step_of(step_ptr, step_);
  const long long i = slot_walker(sp, step, half, 2, gid_base, k);
  const unsigned long long gid = (unsigned long long)(gid_base + i);
  uint32_t c[4] = {(uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)(step * 2ULL + (unsigned)half),
                   (uint32_t)((step * 2ULL + (unsigned)half) >> 32) & 0x7fffffffu};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  const double u = u01(c[0], c[1]);
  const double sq = __dadd_rn(__dmul_rn(a - 1.0, u), 1.0);
  const double z = __dmul_rn(sq, sq) / a;
  const long long src = (long long)(gid / (unsigned long long)sp.W), nc = sp.W >> 1;
  long long j = (long long)(u01(c[2], c[3]) * (double)nc);
  if (j >= nc) j = nc - 1;
  j += src * nc;
  for (int d = 0; d < ndim; ++d) {
    const double s = X[i * ndim + d], co = Cold[j * ndim + d], cn = Q0[j * ndim + d];
    Qa[k * ndim + d] = __dsub_rn(co, __dmul_rn(co - s, z));
    Qb[k * ndim + d] = __dsub_rn(cn, __dmul_rn(cn - s, z));
  }
  logfac[k] = (ndim - 1.0) * log(z);
  jpart[k] = (int)j;
  if (src_a) src_a[k] = src_b[k] = (int)src;
}

// the candidate of slot k that the sequential move would have proposed: its partner moved (Qb) or stayed (Qa)
__global__ void k_select_spec(long long nhalf, int ndim, const int *acc0, const int *jpart, const double *Qa, const double *Qb,
                              const double *La, const double *Lb, double *Qsel, double *Lsel) {
  const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= nhalf) return;
  const bool moved = acc0[jpart[k]] != 0;
  for (int d = 0; d < ndim; ++d) Qsel[k * ndim + d] = moved ? Qb[k * ndim + d] : Qa[k * ndim + d];
  Lsel[k] = moved ? Lb[k] : La[k];
}

__global__ void k_step_inc(unsigned long long *step_ptr) { *step_ptr += 1ULL; }

}  // namespace st2
