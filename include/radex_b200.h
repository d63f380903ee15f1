/*
 * radex_b200.h -- C ABI of libradex_b200: the B200-native replacement for the hot path of
 * yangcht/radex_emcee (per-walker RADEX escape-probability solve + SLED likelihood + stretch move).
 *
 * Every entry point is extern "C", takes plain pointers and sizes, returns 0 on success and a
 * negative rb_status code on failure (rb_last_error() holds the message).  There is no CPU
 * fallback: every compute entry point fails with RB_ERR_CUDA if no sm_100 device is usable.
 *
 * "Replaces" citations are relative to the reference tree (/root/reference):
 *   core.py      = emcee/pyradex/core.py
 *   radex.so@X   = symbol at offset X of emcee/pyradex/radex/radex.so (the f2py-wrapped Fortran)
 *   er1 / er2    = emcee/emcee_radex.py / emcee/emcee_radex_2comp.py
 */
#ifndef RADEX_B200_H
#define RADEX_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rb_mol rb_mol; /* parsed LAMDA molecular table (host memory)          */
typedef struct rb_ctx rb_ctx; /* one GPU: device-resident SoA tables, stream, scratch */

enum rb_status_code {
  RB_OK = 0,
  RB_ERR_ARG = -1,   /* bad argument                                   */
  RB_ERR_IO = -2,    /* cannot open / parse the LAMDA file             */
  RB_ERR_CUDA = -3,  /* CUDA runtime error or no usable device         */
  RB_ERR_LIMIT = -4  /* molecule larger than the kernels support       */
};

/* per-model status bitmask written by the solve kernels (SURVEY.md 8b) */
enum rb_model_status {
  RB_ST_T_RANGE = 1,   /* T not in (0, 1e4]      -> reference raises ValueError, core.py:734-735 */
  RB_ST_N_RANGE = 2,   /* N not in [1e5, 1e25]   -> reference raises ValueError, core.py:771-772 */
  RB_ST_MAXITER = 4,   /* loop ended at maxiter (reference: silent, core.py:904-907)             */
  RB_ST_NONFINITE = 8  /* a returned brightness is NaN/inf                                       */
};

enum rb_stop_rule {
  RB_STOP_PYRADEX = 0, /* core.py:911-917: sum|dxpop| < abs_tol and iter > miniter (default)     */
  RB_STOP_RADEX = 1    /* Fortran matrix()'s own conv flag (radex.so@0x17f70), dropped by f2py   */
};

enum rb_geometry { RB_GEOM_SPHERE = 1, RB_GEOM_LVG = 2, RB_GEOM_SLAB = 3 }; /* core.py:690-700 */

typedef struct rb_opts {
  int32_t stop_rule;   /* rb_stop_rule                                                    */
  int32_t miniter;     /* 10  (core.py:460-461)                                           */
  int32_t maxiter;     /* 200 (core.py:462-463)                                           */
  int32_t kernel;      /* 0 = default (fastest validated: v2, launches ordered by lead-block size,
                              half-warp engine for small lead blocks),
                          1 = v1 shared-memory pivoted LU,
                          2 = v2 without frozen-top caching (cross-check / A-B),
                          3 = v2 with caching but as a single launch (no ordering),
                          4 = v2 with ordered launches but without the half-warp engine (A-B)  */
  double abs_tol;      /* 1e-16 (core.py:857)                                             */
  double fk_epi;       /* h c / k_B used by the brightness epilogue (astropy, core.py:981-984) */
  double thc_epi;      /* 2 h c     used by the brightness epilogue                        */
  int32_t park_max;    /* 0 = automatic.  3..7: largest lead block (in panels of 4 levels) that gets a cached-engine
                          launch of its own in a scheduled batch (tests force 7 on small batches)            */
  int32_t spec_half;   /* rb_stretch_run_dev: propose the second half-step speculatively (both candidates per walker: its
                          partner moved / stayed) so that a step is ONE lnprob launch of 1.5 N walkers -- same chain
                          bit for bit, half the latency.  0 = automatic (while the 1.5 N candidates are at most 17 warps
                          per SM: ~1600 walkers on a B200), -1 = never, 1 = whenever the half-ensemble runs as one fused
                          launch                                                                              */
  int64_t lnprob_pipe_min; /* 0 = automatic (8192).  walkers per call from which lnprob runs as
                          expand -> scheduled solve -> combine instead of one fused launch          */
} rb_opts;

/* observed SLED of one source (er1:229-240 get_source): up to RB_MAX_OBS CO lines */
#define RB_MAX_OBS 16
typedef struct rb_obs {
  int32_t nobs;
  int32_t jup[RB_MAX_OBS];    /* 1-based upper J == 1-based line index (er1:129)   */
  double flux[RB_MAX_OBS];    /* Jy km/s                                            */
  double eflux[RB_MAX_OBS];   /* Jy km/s                                            */
} rb_obs;

/* ---- library ---------------------------------------------------------------------------- */
const char *rb_last_error(void);
void rb_default_opts(rb_opts *opts);
int rb_device_count(void);

/* ---- LAMDA loader: replaces Fortran readdata's parse, radex.so@0x1cf90 (called from
 * core.py:570,744,887) and the collider discovery of emcee/pyradex/utils.py:53-62 ---------- */
int rb_moldata_load(const char *path, rb_mol **out);
void rb_moldata_free(rb_mol *mol);
int rb_moldata_dims(const rb_mol *mol, int32_t *nlev, int32_t *nline, int32_t *npart);
/* partner_id[npart]: LAMDA ids 1 H2, 2 p-H2, 3 o-H2, 4 e, 5 H, 6 He, 7 H+ */
int rb_moldata_partners(const rb_mol *mol, int32_t *partner_id, int32_t *ncoll, int32_t *ntemp);
int rb_moldata_levels(const rb_mol *mol, double *eterm, double *gstat);
int rb_moldata_lines(const rb_mol *mol, int32_t *iupp, int32_t *ilow, double *aeinst, double *spfreq_ghz,
                     double *eup_k, double *xnu);

/* ---- context: replaces init_radex()/Radex.__init__ (er1:104-117, core.py:209-378) ---------- */
int rb_ctx_create(int device, const rb_mol *mol, rb_ctx **out);
void rb_ctx_destroy(rb_ctx *ctx);
int rb_ctx_sync(rb_ctx *ctx);
/* launch on a caller-owned CUDA stream (cudaStream_t as void*; 0 = CUDA's legacy default stream,
 * which is what PyTorch's default stream is); rb_ctx_reset_stream goes back to the ctx's own. */
int rb_ctx_set_stream(rb_ctx *ctx, void *stream);
int rb_ctx_reset_stream(rb_ctx *ctx);

/* ---- batched solve: replaces set_params + run_radex + tex/tau/level_population +
 * source_line_surfbrightness (core.py:388-438, 856-925, 703-717, 986-1003; base_class.py:275-277)
 * and, inside, readdata's interpolation, backrad, matrix, escprob, lubksb/sgeir
 * (radex.so@0x1cf90, 0x1be30, 0x17f70, 0xa9c0, 0x17cb0).
 *   dens : n x npart, partner order of the file, cm^-3      tkin : K      cdmol : cm^-2
 *   outputs (any may be NULL): xpop n x nlev, tex/tau/surf n x nline
 *     surf = source_line_surfbrightness, erg s^-1 cm^-2 Hz^-1 sr^-1
 * Host-pointer form copies in/out on the ctx stream and synchronises; _dev takes device
 * pointers and is asynchronous on the ctx stream.                                              */
int rb_solve_batch(rb_ctx *ctx, int64_t n, const double *tkin, const double *dens, const double *cdmol,
                   double deltav_kms, double tbg, int geometry, const rb_opts *opts, double *xpop, double *tex,
                   double *tau, double *surf, int32_t *niter, int32_t *status);
int rb_solve_batch_dev(rb_ctx *ctx, int64_t n, const double *tkin, const double *dens, const double *cdmol,
                       double deltav_kms, double tbg, int geometry, const rb_opts *opts, double *xpop,
                       double *tex, double *tau, double *surf, int32_t *niter, int32_t *status);

/* ---- vectorised lnprob: replaces lnprob/lnprior/lnlike/model_lvg, one component (er1:120-181)
 * and two components (er2:122-244).  P is n x 4 / n x 8 (log10 n, T, N/dv, size per component);
 * bounds is 4 x 2 / 8 x 2 (lo, hi); opr fixed at 3 like the drivers (er1:95-96).
 * has_td = 0 reproduces T_d=None.  lnp[n] never holds NaN (emcee rejects NaN): every invalid
 * case maps to -inf exactly where the reference returns -inf.  nsolves (may be NULL) returns
 * the number of RADEX solves actually performed (prior short-circuit, er1:178-180).           */
int rb_lnprob1(rb_ctx *ctx, int64_t n, const double *P, const rb_obs *obs, const double *bounds, double tbg,
               const rb_opts *opts, double *lnp, int64_t *nsolves);
int rb_lnprob1_dev(rb_ctx *ctx, int64_t n, const double *P, const rb_obs *obs, const double *bounds,
                   double tbg, const rb_opts *opts, double *lnp, int64_t *nsolves_dev);
int rb_lnprob2(rb_ctx *ctx, int64_t n, const double *P, const rb_obs *obs, const double *bounds, int has_td,
               double t_d, double tbg, const rb_opts *opts, double *lnp, int64_t *nsolves);
int rb_lnprob2_dev(rb_ctx *ctx, int64_t n, const double *P, const rb_obs *obs, const double *bounds,
                   int has_td, double t_d, double tbg, const rb_opts *opts, double *lnp, int64_t *nsolves_dev);

/* ---- multi-source lnprob (BASELINE.json configs[3]: all flux.dat sources fitted concurrently; the reference
 * loops over the sources one after the other, er1:389).  A source set is a device-resident table of
 * (observed SLED, bounds, tbg, T_d) rows; src_id[n] (DEVICE int32, NULL = every walker belongs to source 0)
 * names the row of each walker.  Same arithmetic per walker as rb_lnprob1/2.  More than one source always
 * runs as one fused launch (the background temperature is a per-model quantity there).              */
typedef struct rb_source {
  rb_obs obs;
  double bounds[16];   /* (4 ncomp) x 2 : lo, hi                                  */
  double tbg;          /* 2.7315 (1 + z), er1:419                                  */
  int32_t has_td;      /* two components: Gaussian prior on T_cold (er2:213-224)   */
  int32_t reserved;
  double t_d;
} rb_source;
typedef struct rb_srcset rb_srcset;
int rb_srcset_create(rb_ctx *ctx, int32_t ncomp, int32_t nsrc, const rb_source *src, rb_srcset **out);
void rb_srcset_destroy(rb_srcset *set);
int rb_lnprob_src_dev(rb_ctx *ctx, const rb_srcset *set, int64_t n, const double *P, const int32_t *src_id,
                      const rb_opts *opts, double *lnp, int64_t *nsolves_dev);

/* ---- stretch move: replaces emcee.StretchMove.get_proposal + the accept loop of
 * emcee's RedBlueMove (un-vendored; call sites er1:483-499, er2:557-574; SURVEY.md 3.5).
 * All pointers are DEVICE pointers; asynchronous on the ctx stream.
 *   propose: for active walker k (global id gid0 + k*gid_stride) with position s = S[k,:], draw
 *            z = ((a-1)u+1)^2/a and a partner j uniformly from the nc complementary positions
 *            C[nc,ndim]; q = c_j - (c_j - s) z ; logfac[k] = (ndim-1) ln z.
 *   accept : accept iff logfac + lnp_new - lnp_old > ln u'; updates S, lnp_old in place and
 *            adds the number accepted to *naccept.
 * RNG is counter-based (Philox4x32-10) keyed by (seed, step, half, global walker id), so the
 * chain does not depend on how walkers are sharded over GPUs.                                  */
int rb_stretch_propose_dev(rb_ctx *ctx, int64_t ns, int32_t ndim, const double *S, int64_t nc,
                           const double *C, double a, uint64_t seed, uint64_t step, int32_t half,
                           int64_t gid0, int64_t gid_stride, double *Q, double *logfac);
int rb_stretch_accept_dev(rb_ctx *ctx, int64_t ns, int32_t ndim, double *S, double *lnp_old, const double *Q,
                          const double *lnp_new, const double *logfac, uint64_t seed, uint64_t step,
                          int32_t half, int64_t gid0, int64_t gid_stride, int64_t *naccept);

/* ---- stretch move, second form: the whole local ensemble X[nlocal, ndim] stays in place and the red/blue split
 * is a function of (seed, step, global walker id), so that emcee's default randomize_split=True
 * (RedBlueMove, SURVEY.md 3.5) is reproduced without communication and independently of the rank count.
 *   ensemble  : N = nwalkers walkers, global ids 0..N-1; nsrc = N / walkers_per_source independent
 *               sub-ensembles (one per fitted source) of W walkers each; a walker's partner comes from the
 *               complementary half of its own sub-ensemble.
 *   split     : blocks of `block` consecutive walkers (block | W, block even); in block b slot t of half h is
 *               walker b*block + pi(h*block/2 + t), pi a keyed bijection of [0, block) drawn per (seed, step, b)
 *               (randomize = 1), or 2t + h (randomize = 0: the parity split of the first form).
 *   a rank    : owns the contiguous ids [gid_base, gid_base + nlocal), block | nlocal.
 *   pack      : Chalf[nlocal/2, ndim] = positions of this rank's walkers of half `half`, in slot order; the
 *               all-gather of these over the ranks (rank order) is `Call` = the half in global slot order.
 *   propose2  : for every local slot of half `half`: walker s, partner c_j drawn from the W/2 slots of its
 *               source in Call (the complementary half), q = c_j - (c_j - s) z, logfac; src_id[k] = source.
 *   accept2   : accept test per slot; X, lnp updated in place; naccept[nlocal] per walker (emcee's
 *               acceptance_fraction is per walker); *nan_count += NaN log-probabilities seen (emcee raises).
 * RNG: Philox4x32-10 keyed by (seed, step, half, global walker id) exactly as in the first form.              */
typedef struct rb_split {
  int64_t nwalkers;
  int64_t walkers_per_source;
  int64_t block;
  int32_t randomize;
  int32_t reserved;
  uint64_t seed;
} rb_split;
int rb_stretch_pack_dev(rb_ctx *ctx, const rb_split *split, uint64_t step, int32_t half, int64_t gid_base,
                        int64_t nlocal, int32_t ndim, const double *X, double *Chalf);
int rb_stretch_propose2_dev(rb_ctx *ctx, const rb_split *split, uint64_t step, int32_t half, int64_t gid_base,
                            int64_t nlocal, int32_t ndim, const double *X, const double *Call, double a, double *Q,
                            double *logfac, int32_t *src_id);
int rb_stretch_accept2_dev(rb_ctx *ctx, const rb_split *split, uint64_t step, int32_t half, int64_t gid_base,
                           int64_t nlocal, int32_t ndim, double *X, double *lnp, const double *Q, const double *lnp_new,
                           const double *logfac, int64_t *naccept, int64_t *nan_count);

/* ---- the sampler loop itself, device-resident: replaces EnsembleSampler.run_mcmc (call sites er1:490-499,
 * er2:563-574) for one GPU -- nsteps stretch-move steps (two half-steps each: pack, propose2, lnprob of the
 * source set, accept2) without returning to the host; ensembles whose half fits one fused lnprob launch are
 * replayed from a CUDA graph of one step.  All pointers are DEVICE pointers.
 *   X[N, ndim], lnp[N] : state, in/out (lnp must hold lnprob(X) on entry: rb_lnprob_src_dev)
 *   naccept[N]         : += accepted proposals per walker        counters[2]: += NaN count, += solves
 *   chain, lnp_chain   : NULL, or [nsteps / thin][N, ndim] and [nsteps / thin][N]: state after every thin-th step
 * Multi-GPU runs call pack / all-gather (NCCL) / propose2 / rb_lnprob_src_dev / accept2 per half-step from one
 * process per GPU (radex_emcee_b200/sampler.py; INTEGRATION.md shows the C++ form).                           */
int rb_stretch_run_dev(rb_ctx *ctx, const rb_srcset *set, const rb_split *split, double a, uint64_t step0,
                       int64_t nsteps, const rb_opts *opts, double *X, double *lnp, int64_t *naccept,
                       int64_t *counters, int32_t thin, double *chain, double *lnp_chain);

/* ---- moves and move mixtures: emcee's EnsembleSampler(moves=...) for StretchMove(a) and DEMove(sigma, gamma0).
 *   rb_move        : one move of the list; weights >= 0 are normalised over the list (emcee's [(move, weight), ...]).
 *                    gamma0 = 0 means 2.38 / sqrt(2 ndim).
 *   schedule       : every step applies ONE move of the list to the whole ensemble, drawn from one Philox call keyed by
 *                    (seed ^ 'MOVESCHD', step) against the cumulative normalised weights (last bound 1): the same on
 *                    every rank and for any rank count.  rb_move_schedule writes the move index of steps step0 ..
 *                    step0 + nsteps - 1 to out[nsteps] (host memory, no device needed); a one-move list gives 0.
 *   DE split       : the split of rb_split generalised to k = 3 groups: in block b, group g holds
 *                    n_g = block / 3 + (g < block % 3) slots; slot t of group g is walker b*block + pi(off_g + t),
 *                    off_g = sum_{h<g} n_h, with the same keyed bijection pi of (seed, step, b) (randomize = 1), or
 *                    b*block + g + 3t (randomize = 0).  For k = 2 this is the red/blue split above.  Every group's
 *                    complement within its source must hold >= 2 walkers, and block >= 3 (RB_ERR_ARG otherwise).
 *   DE step        : groups g = 0, 1, 2 in turn: propose (rb_de_propose_dev), lnprob of the group, accept
 *                    (rb_group_accept_dev); partners are read from the positions as they stand after the earlier groups.
 *   rb_de_propose_dev   : Q[k] = s + gamma (c_j2 - c_j1) for the local slots k of group g (nslots = nlocal / block * n_g,
 *                    in slot order), (j1, j2) uniform over the ordered pairs of distinct walkers of the complement of
 *                    group g within the walker's source, gamma = gamma0 (1 + sigma n), n ~ N(0, 1).  Xall[nwalkers, ndim]
 *                    is the whole ensemble in global walker order (one rank: X; several: the all-gather of X).
 *                    src_id[nslots] may be NULL.
 *   rb_group_accept_dev : accept test of the local slots of group g of ngroups, as rb_stretch_accept2_dev (logfac NULL:
 *                    0); kind selects the random stream: RB_MOVE_STRETCH with ngroups = 2 (it IS rb_stretch_accept2_dev)
 *                    or RB_MOVE_DE with ngroups = 3 (and the DE split rules); any other pair is RB_ERR_ARG.
 *   rb_moves_run_dev    : rb_stretch_run_dev for a move list (arguments as there); one captured CUDA graph per entry of
 *                    the list, the host launches the scheduled move's graph step after step without a device sync.
 *                    rb_stretch_run_dev(a) is rb_moves_run_dev with the single move {RB_MOVE_STRETCH, a}.
 * DE random numbers: Philox4x32-10 keyed by seed ^ 'DEmvmove', counter (global id, 4 step + group, draw); the split
 * of a step stays keyed by (seed, step, block) whatever the move.                                                   */
enum rb_move_kind { RB_MOVE_STRETCH = 0, RB_MOVE_DE = 1 };
#define RB_MAX_MOVES 8
typedef struct rb_move {
  int32_t kind;      /* rb_move_kind                                    */
  int32_t reserved;
  double a;          /* RB_MOVE_STRETCH: scale, > 1 (emcee: 2)          */
  double gamma0;     /* RB_MOVE_DE: 0 = 2.38 / sqrt(2 ndim)             */
  double sigma;      /* RB_MOVE_DE: >= 0 (emcee: 1e-5)                  */
  double weight;     /* >= 0, normalised over the list                  */
} rb_move;
int rb_move_schedule(uint64_t seed, uint64_t step0, int64_t nsteps, const double *weights, int32_t nmoves, int32_t *out);
int rb_moves_run_dev(rb_ctx *ctx, const rb_srcset *set, const rb_split *split, const rb_move *moves, int32_t nmoves,
                     uint64_t step0, int64_t nsteps, const rb_opts *opts, double *X, double *lnp, int64_t *naccept,
                     int64_t *counters, int32_t thin, double *chain, double *lnp_chain);
int rb_de_propose_dev(rb_ctx *ctx, const rb_split *split, uint64_t step, int32_t group, int64_t gid_base, int64_t nlocal,
                      int32_t ndim, const double *X, const double *Xall, double gamma0, double sigma, double *Q,
                      int32_t *src_id);
int rb_group_accept_dev(rb_ctx *ctx, const rb_split *split, int32_t kind, uint64_t step, int32_t group, int32_t ngroups,
                        int64_t gid_base, int64_t nlocal, int32_t ndim, double *X, double *lnp, const double *Q,
                        const double *lnp_new, const double *logfac, int64_t *naccept, int64_t *nan_count);

/* ---- posterior statistics of the device-resident chain: replaces np.percentile over the flattened chain
 * (er1:511-531) and emcee's get_autocorr_time / integrated_time, without moving the chain.  DEVICE pointers,
 * asynchronous on the ctx stream.  Argument errors give RB_ERR_ARG, a machine without a CUDA device RB_ERR_CUDA.
 *   view   : the chain as this rank stores it: chunk[c] is [steps[c]][nlocal][ndim] (one chunk per run_mcmc call),
 *            read in place.  Selected steps over the concatenated step index are emcee's
 *            discard + thin - 1, discard + 2 thin - 1, ... (get_chain(discard=, thin=)).  Local walker w belongs to
 *            source (gid_base + w) / walkers_per_source, as in rb_split.
 *   hist   : one digit pass of a radix select over keys k(x) = bits(x) ^ (x < 0 ? ~0 : 1 << 63) (order-preserving; NaN is
 *            counted in nan_counts on pass 0 and in no histogram).  Column c is x[col_i[c]], or x[col_i[c]] + x[col_j[c]]
 *            (one IEEE add) when col_j[c] >= 0; col_i, col_j are HOST arrays.  Pass p counts digit p (bits 63-8p..56-8p)
 *            of the values whose higher digits equal prefix[src][c][t] (right-aligned; pass 0: nprefix = 1, prefix
 *            ignored; UINT64_MAX = unused slot):  counts[src][c][t][digit] += ..., nan_counts[src][c] += ... (pass 0,
 *            may be NULL).  ncol * nprefix <= RB_CHAIN_MAX_HIST.
 *   moments: mean[nlocal][ndim] and c0 = sum_t (x_t - mean)^2 over the selected steps.
 *   acf    : rho_sum[nsrc][k1 - k0][ndim] = sum over the walkers of each source of c_k / c_0, c_k = sum_t (x_t - mean)
 *            (x_{t+k} - mean), for lags k0 <= k < k1 <= selected steps; sources not on this rank get 0.  Fixed summation
 *            order: the same call on the same rank layout gives the same bits.  A walker with c_0 = 0 gives NaN.
 * The caller sums hist / acf outputs over ranks and finishes on the host; for a percentile q (numpy's default
 * 'linear' method) of n values:  v = (n - 1) (q / 100); i = floor(v), j = i + 1, or i = j = n - 1 when v >= n - 1
 * (then gamma = v + 1, else gamma = v - i); d = x_(j) - x_(i); result = gamma >= 0.5 ? x_(j) - d (1 - gamma)
 * : x_(i) + d gamma; NaN if the column holds a NaN.                                                               */
#define RB_MAX_CHUNKS 64
#define RB_CHAIN_MAX_DIM 16
#define RB_CHAIN_MAX_COLS 32
#define RB_CHAIN_MAX_HIST 128
typedef struct rb_chain_view {
  const double *chunk[RB_MAX_CHUNKS];
  int64_t steps[RB_MAX_CHUNKS];
  int32_t nchunks;
  int32_t ndim;
  int64_t nlocal;
  int64_t gid_base;
  int64_t walkers_per_source;
  int64_t discard;
  int64_t thin;
} rb_chain_view;
int rb_chain_hist_dev(rb_ctx *ctx, const rb_chain_view *view, int32_t nsrc, int32_t ncol, const int32_t *col_i,
                      const int32_t *col_j, int32_t pass, int32_t nprefix, const uint64_t *prefix, uint64_t *counts,
                      uint64_t *nan_counts);
int rb_chain_moments_dev(rb_ctx *ctx, const rb_chain_view *view, double *mean, double *c0);
int rb_chain_acf_dev(rb_ctx *ctx, const rb_chain_view *view, int32_t nsrc, const double *mean, const double *c0,
                     int64_t k0, int64_t k1, double *rho_sum);

/* ---- corner-plot marginals, covariance and the sample nearest a target, of the device-resident chain: replaces the
 * replot's `corner` over the pickled chain and the host search of nearest_sample_to_vector (er1:242-266), without
 * moving the chain.  The view, columns, sources, pointers and errors are as in rb_chain_hist_dev.
 *   marginals: bin k of a value x for the edges e[0..nbins] of its (source, column) is (number of edges <= x) - 1, and
 *            x == e[nbins] is in bin nbins - 1 (np.searchsorted(e, x, 'right') - 1: np.histogram / np.histogram2d with
 *            range=); NaN, +-inf and values outside [e[0], e[nbins]] are not counted.  One read of the chain counts every
 *            column and as many pairs as fit shared memory (all 45 pairs of 10 columns at 20 bins).
 *   sums   : s1 = sum (x - c), s2 = sum (x - c)(x - c)^T over each source's selected samples on this rank, c = center of
 *            the source.  Fixed summation order (per-block partials, then the blocks in order): a repeated call on the same
 *            rank layout gives the same bits.  Covariance: sums with c = 0 summed over ranks give the mean m = s1 / n;
 *            sums with c = m summed over ranks give cov = (s2 - s1 s1^T / n) / (n - 1).
 *   nearest: per selected sample w = L^-1 (x - t) by forward substitution (L = chol of the source, lower triangle), d2 =
 *            sum_r w_r^2 in r order; per source the minimum d2, NaN before every number (np.argmin), ties to the lowest
 *            index j W + (gid - s W): the row of the sample in get_chain(discard, thin)[:, s W:(s + 1) W].reshape(-1,
 *            ndim); x is that sample.  Across ranks: the minimum d2 (NaN first), then the lowest index. */
#define RB_CHAIN_MAX_BINS 100
/* edges: DEVICE [nsrc][ncol][nbins+1], finite, strictly increasing (the caller's precondition).
   counts1: DEVICE [nsrc][ncol][nbins].
   counts2: DEVICE [nsrc][npair][nbins][nbins] or NULL.
   Pairs are (a, b) with a < b, in the order (0,1), (0,2), ..., (0,n-1), (1,2), ...; npair = ncol (ncol - 1) / 2.
   counts2[s][p][ka][kb] counts the samples with column a in bin ka AND column b in bin kb.
   Counts are ADDED (the caller zeroes them), like rb_chain_hist_dev.  col_i, col_j are HOST arrays. */
int rb_chain_marginals_dev(rb_ctx *ctx, const rb_chain_view *view, int32_t nsrc, int32_t ncol, const int32_t *col_i,
                           const int32_t *col_j, int32_t nbins, const double *edges, uint64_t *counts1, uint64_t *counts2);
/* center: DEVICE [nsrc][ndim].  s1: [nsrc][ndim], s2: [nsrc][ndim][ndim].
   Both are written, not added; sources with no walkers on this rank get 0. */
int rb_chain_sums_dev(rb_ctx *ctx, const rb_chain_view *view, int32_t nsrc, const double *center, double *s1, double *s2);
/* target: DEVICE [nsrc][ndim].  chol: DEVICE [nsrc][ndim][ndim], lower triangle read.
   Outputs: d2 [nsrc], index [nsrc], x [nsrc][ndim].
   A source with no walkers on this rank gets index -1 and d2 = +inf (and x = 0). */
int rb_chain_nearest_dev(rb_ctx *ctx, const rb_chain_view *view, int32_t nsrc, const double *target, const double *chol,
                         double *d2, int64_t *index, double *x);

/* ---- posterior-predictive SLEDs of the device-resident chain: replaces the host replot's model_lvg over the pickled
 * chain (er1:120-130, er2:122-147), one Radex call per sample, without moving the chain.  DEVICE pointers except jup,
 * asynchronous on the ctx stream; rb_ctx_counters / rb_ctx_cache_stats report the call like any solve call.
 *   view   : the selected steps of the chain as in rb_chain_hist_dev; ndim = 4 x set->ncomp.  Local walker w belongs to
 *            source (gid_base + w) / walkers_per_source, whose row of `set` gives tbg.
 *   jup    : HOST int32[nlines], 1 <= nlines <= RB_MAX_OBS one-based line indices 1 <= J <= nline, in any order, repeats
 *            allowed.
 *   model  : per sample theta and component c: T = 10^theta[4c+1], N = 10^theta[4c+2], partner densities split from
 *            10^theta[4c] as rb_lnprob1/2 do (opr = 3), LVG, deltav = 1 km/s, opts as given;
 *            flux_c[J] = surf_c[J-1] * 10^theta[4c+3] * 1e23 (Jy km/s, er1:129).  No prior is applied.  A component out
 *            of pyradex's range (RB_ST_T_RANGE / RB_ST_N_RANGE, where model_lvg raises ValueError) gives NaN.
 *   flux   : [nplanes][nsel][nlocal][nlines], nsel = the view's selected steps.  One component: nplanes = 1, the flux.
 *            Two: nplanes = 3, the total flux_0 + flux_1 (er2:147, NaN if either is), then component 1 (theta[0:4]) and
 *            component 2 (theta[4:8]).  A plane is a chain chunk of ndim = nlines: rb_chain_hist_dev reads it as is.
 *   counters_dev : NULL, or int64[2]: [0] += components solved, [1] += components out of range.
 * Argument errors give RB_ERR_ARG (bad nlines or J, null pointers, a bad view, a set of another ctx, of another ncomp
 * or without the view's sources), a machine without a CUDA device RB_ERR_CUDA.                                        */
int rb_predict_sled_dev(rb_ctx *ctx, const rb_srcset *set, const rb_chain_view *view, int32_t nlines, const int32_t *jup,
                        const rb_opts *opts, double *flux, int64_t *counters_dev);

/* counters of the last solve/lnprob call on this ctx (device-measured, read back on request):
 * total matrix iterations summed over models, and kernels launched since ctx creation.        */
int rb_ctx_counters(rb_ctx *ctx, int64_t *total_iters_last, int64_t *launches_total);

/* frozen-top caching statistics of the last solve/lnprob call: stats3[0] matrix iterations that ran
 * on the cached path, [1] captures, [2] invalidations (a frozen line turned optically thick).  */
int rb_ctx_cache_stats(rb_ctx *ctx, int64_t *stats3);

/* measured FP64 FMA throughput of this GPU (TFLOP/s), the roofline denominator bench.py reports */
int rb_fp64_peak(rb_ctx *ctx, double *tflops);

#ifdef __cplusplus
}
#endif
#endif /* RADEX_B200_H */
