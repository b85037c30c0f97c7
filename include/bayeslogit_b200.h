/*
 * bayeslogit_b200.h -- C ABI of the B200-native Polya-Gamma engine.
 *
 * Part 1 is the DROP-IN BOUNDARY: exactly the symbols of the reference's
 * Code/C/LogitWrapper.h:23-64, the functions R reaches through
 * .C("rpg_devroye", ...), .C("gibbs", ...) etc. (Code/R/LogitWrapper.R:29,49,69,92,
 * 118,177,229,277,342,395).  Same names, same argument meaning, all arguments
 * pointers into caller-owned HOST memory, void return; errors are reported the
 * way the reference reports them (a message on the console, outputs left as
 * they were, LogitWrapper.cpp:226-229) and can additionally be read back with
 * bl_last_error().
 *
 * Part 2 are engine extensions (prefix bl_): seeding, device selection,
 * device-resident and streaming variants, and the injected-variate ("tape")
 * variants used for tier-1 parity.  There is NO CPU fallback anywhere in this
 * library: without a usable sm_100 device every entry point fails loudly.
 *
 * All matrices are column-major (R layout), see INTEGRATION.md.
 */
#ifndef BAYESLOGIT_B200_H
#define BAYESLOGIT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------ */
/* Part 1 -- reference entry points (Code/C/LogitWrapper.h)                  */
/* ------------------------------------------------------------------------ */

/* LogitWrapper.h:27 / LogitWrapper.cpp:39-62.  x[i] = n[i] != 0 ? truncated
 * sum-of-gammas PG(n[i], z[i]) with *trunc terms : 0. */
void rpg_gamma(double *x, double *n, double *z, int *num, int *trunc);

/* LogitWrapper.h:29 / LogitWrapper.cpp:66-85.  x[i] = n[i] != 0 ? sum of n[i]
 * Devroye PG(1, z[i]) draws : 0. */
void rpg_devroye(double *x, int *n, double *z, int *num);

/* LogitWrapper.h:31 / LogitWrapper.cpp:87-106.  Alternate sampler, h >= 1. */
void rpg_alt(double *x, double *h, double *z, int *num);

/* LogitWrapper.h:33 / LogitWrapper.cpp:108-127.  Saddle-point sampler; iter[i]
 * receives the proposal count (left untouched where h[i] == 0, as there). */
void rpg_sp(double *x, double *h, double *z, int *num, int *iter);

/* LogitWrapper.h:35 / LogitWrapper.cpp:129-167.  Regime dispatch on h[i]:
 * >170 normal approximation, >13 saddle point, ==1 or ==2 Devroye, >1 alternate,
 * >0 sum of gammas (200 terms), else 0. */
void rpg_hybrid(double *x, double *h, double *z, int *num);

/* LogitWrapper.h:39-43 / LogitWrapper.cpp:176-234.  Binomial-logit Gibbs.
 * wp: N x samp, betap: P x samp, yp: N (proportions), tXp: P x N, np: N,
 * m0p: P, P0p: P x P (precision). */
void gibbs(double *wp, double *betap, double *yp, double *tXp, double *np,
           double *m0p, double *P0p, int *N, int *P, int *samp, int *burn);

/* LogitWrapper.h:45-48 / LogitWrapper.cpp:238-273.  Posterior mode by EM. */
void EM(double *betap, double *yp, double *tXp, double *np, int *Np, int *Pp,
        double *tolp, int *max_iterp);

/* LogitWrapper.h:50-51 / LogitWrapper.cpp:279-310.  Merge duplicate rows. */
void combine(double *yp, double *tXp, double *np, int *N, int *P);

/* LogitWrapper.h:55-59 / LogitWrapper.cpp:316-374.  Multinomial-logit Gibbs.
 * wp: N x (J-1) x samp, betap: P x (J-1) x samp, typ: (J-1) x N, tXp: P x N,
 * m0p: P x (J-1), P0p: P x P x (J-1). */
void mult_gibbs(double *wp, double *betap, double *typ, double *tXp, double *np,
                double *m0p, double *P0p, int *N, int *P, int *J, int *sampp, int *burnp);

/* LogitWrapper.h:61-62 / LogitWrapper.cpp:376-409. */
void mult_combine(double *typ, double *tXp, double *np, int *N, int *P, int *J);

/* ------------------------------------------------------------------------ */
/* Part 2 -- engine extensions                                               */
/* ------------------------------------------------------------------------ */

/* Status: 0 = ok, nonzero = error (message through bl_last_error()). */
int bl_version(void);
const char *bl_last_error(void);
void bl_clear_error(void);

/* Select the CUDA device of this process (one process per GPU). */
int bl_set_device(int device);
int bl_get_device(void);

/* Seed of the Philox stream contract.  The reference has no seed argument: its
 * draws come from R's global generator (GetRNGstate/PutRNGstate,
 * LogitWrapper.cpp:44-46).  Here the drop-in entry points use (seed, call
 * counter); bl_set_seed() also resets the call counter to 0 so a sequence of
 * calls is reproducible. */
void bl_set_seed(uint64_t seed);
uint64_t bl_get_seed(void);
/* The same through R's .C() convention (an int vector of length 1): the shim an R front end calls next to
 * set.seed(), see INTEGRATION.md. */
void bl_set_seed_r(int *seed);
uint32_t bl_get_call_counter(void);

/* Device-resident batch draws: all pointers are DEVICE pointers; the work is
 * enqueued on `stream` (a cudaStream_t, NULL = legacy default stream) and the
 * call returns without synchronising.  Observation i uses the Philox stream of
 * global index obs0 + i, so shards of one logical batch can be drawn on
 * different GPUs with results independent of the sharding. */
int bl_rpg_devroye_dev(double *x, const int *n, const double *z, int64_t num,
                       uint64_t seed, uint32_t call_id, uint64_t obs0, void *stream);
/* The same draws through the unfiltered all-fp64 Devroye path (A/B check of the fp32
 * decision pre-filters: results must be identical). */
int bl_rpg_devroye_plain_dev(double *x, const int *n, const double *z, int64_t num,
                             uint64_t seed, uint32_t call_id, uint64_t obs0, void *stream);
/* ... and through the filtered sampler in a plain per-lane loop (no persistent-lane refill). */
int bl_rpg_devroye_loop_dev(double *x, const int *n, const double *z, int64_t num,
                            uint64_t seed, uint32_t call_id, uint64_t obs0, void *stream);
int bl_rpg_gamma_dev(double *x, const double *n, const double *z, int64_t num, int trunc,
                     uint64_t seed, uint32_t call_id, uint64_t obs0, void *stream);
int bl_rpg_alt_dev(double *x, const double *h, const double *z, int64_t num,
                   uint64_t seed, uint32_t call_id, uint64_t obs0, void *stream);
int bl_rpg_sp_dev(double *x, const double *h, const double *z, int64_t num, int *iter,
                  uint64_t seed, uint32_t call_id, uint64_t obs0, void *stream);
int bl_rpg_hybrid_dev(double *x, const double *h, const double *z, int64_t num,
                      uint64_t seed, uint32_t call_id, uint64_t obs0, void *stream);

/* Host-pointer draws with an explicit stream identity (what the drop-in entry
 * points call with the global seed / call counter). */
int bl_rpg_devroye_seeded(double *x, const int *n, const double *z, int64_t num,
                          uint64_t seed, uint32_t call_id, uint64_t obs0);
int bl_rpg_gamma_seeded(double *x, const double *n, const double *z, int64_t num, int trunc,
                        uint64_t seed, uint32_t call_id, uint64_t obs0);
int bl_rpg_alt_seeded(double *x, const double *h, const double *z, int64_t num,
                      uint64_t seed, uint32_t call_id, uint64_t obs0);
int bl_rpg_sp_seeded(double *x, const double *h, const double *z, int64_t num, int *iter,
                     uint64_t seed, uint32_t call_id, uint64_t obs0);
int bl_rpg_hybrid_seeded(double *x, const double *h, const double *z, int64_t num,
                         uint64_t seed, uint32_t call_id, uint64_t obs0);

/* Injected-variate ("tape") variants, host pointers.  Observation i consumes
 * uniforms tu[i*lu ..], exponentials te[i*le ..], normals tn[i*ln ..] and gamma
 * variates tg[i*lg ..] in the reference's statement order (SURVEY.md App. A).
 * trace (may be NULL) receives 6 ints per observation: #U, #E, #N, #G consumed,
 * a tape-exhausted flag, and an auxiliary count (saddle-point proposals).
 * Draws whose tape ran dry are returned as NaN. */
#define BL_TRACE_W 6
typedef struct bl_tape {
    const double *tu, *te, *tn, *tg;
    int32_t lu, le, ln, lg;
} bl_tape;

int bl_rpg_devroye_tape(double *x, const int *n, const double *z, int64_t num,
                        const bl_tape *tape, int *trace);
int bl_rpg_devroye_plain_tape(double *x, const int *n, const double *z, int64_t num,
                              const bl_tape *tape, int *trace);
int bl_rpg_gamma_tape(double *x, const double *n, const double *z, int64_t num, int trunc,
                      const bl_tape *tape, int *trace);
int bl_rpg_alt_tape(double *x, const double *h, const double *z, int64_t num,
                    const bl_tape *tape, int *trace);
int bl_rpg_sp_tape(double *x, const double *h, const double *z, int64_t num, int *iter,
                   const bl_tape *tape, int *trace);
int bl_rpg_hybrid_tape(double *x, const double *h, const double *z, int64_t num,
                       const bl_tape *tape, int *trace);

/* ---- Gibbs sweeps --------------------------------------------------------- */

/* flags */
#define BL_GIBBS_PLAIN_BETA 1   /* unconstrained beta ~ N(PP^-1 bP, PP^-1) (Logit.hpp:291-320) instead of
                                   the constrained coordinate-wise draw the reference calls (:322-400) */
#define BL_GIBBS_NO_W 2         /* do not return the omega chains (w may be NULL) */
#define BL_GIBBS_UNFUSED 4      /* measurement / A-B aid: psi = X beta and the omega draw as two kernels instead of
                                   the fused pass over X (same chain, bit for bit) */

#define BL_GIBBS_ONE_PASS 8      /* even P <= 64: psi, omega and X' Omega X from ONE TMA-staged read of X per iteration
                                   (k_logit_sweep, gibbs_sweep.cu) instead of two passes (k_logit_psi_draw + k_gram_partial);
                                   same chain up to the summation order of psi and the Gram.  Without either flag the
                                   one-pass kernel is used for shards of at most 2^18 rows, where it is the faster one. */
#define BL_GIBBS_TWO_PASS 16     /* the two-pass path whatever the shard size */

/* `gibbs` with an explicit seed and flags; host pointers, layouts as `gibbs`. */
int bl_logit_gibbs(double *w, double *beta, const double *y, const double *tX, const double *n,
                   const double *m0, const double *P0, int N, int P, int samp, int burn,
                   uint64_t seed, int flags);
/* The same with the omega chain thinned: omega of sampling iteration m (1-based) is returned only when
 * (m - 1) % w_every == 0, in slot (m - 1) / w_every; w: N x ceil(samp / w_every) (beta: every iteration, P x samp).
 * `gibbs` returns N x samp doubles of omega -- 40 GB at N = 1M, samp = 5000 (LogitWrapper.cpp:207-221); a caller
 * that wants beta and an occasional omega asks for w_every = 100, or passes BL_GIBBS_NO_W. */
int bl_logit_gibbs_thin(double *w, double *beta, const double *y, const double *tX, const double *n,
                        const double *m0, const double *P0, int N, int P, int samp, int burn,
                        uint64_t seed, int flags, int w_every);
/* `mult_gibbs` with an explicit seed (no duplicate-row merge: call mult_combine first). */
int bl_mlogit_gibbs(double *w, double *beta, const double *ty, const double *tX, const double *n,
                    const double *m0, const double *P0, int N, int P, int J, int samp, int burn,
                    uint64_t seed, int flags);
/* Negative-binomial regression sweep with fixed dispersion d (the reference has no C entry
 * for it: Code/R/NBPG-logmean.R:13-34,77-106).  y: counts [N]; beta: P x samp; w_last: N or NULL. */
int bl_nb_gibbs(double *w_last, double *beta, const double *y, const double *tX, double d,
                const double *m0, const double *P0, int N, int P, int samp, uint64_t seed);
/* The full NB.PG.gibbs of Code/R/NBPG-logmean.R:36-113: the dispersion d is sampled every
 * iteration by draw.df (Code/R/NB-Shape.R:21-53, random-walk Metropolis on the integers, two
 * uniforms per iteration from the stream (seed, obs 2^64-2, iteration)); burn iterations are
 * discarded.  d0: initial integer dispersion (the reference starts at 1); beta: P x samp;
 * d_out: samp; w_last: N (omega of the last iteration) or NULL. */
int bl_nb_gibbs_df(double *w_last, double *beta, double *d_out, const double *y, const double *tX, double d0,
                   const double *m0, const double *P0, int N, int P, int samp, int burn, uint64_t seed);

/* ... with the real-valued random walk draw.df.real.mean (Code/R/NB-Shape.R:86-96, the alternative the reference
 * keeps commented out at NBPG-logmean.R:87): rstar ~ U(d - 1, d + 1) (U(0, 2) for d <= 1), target
 * sum_i dnbinom(y_i, d, mu_i / (mu_i + d), log = TRUE) as written there; b = y + d is then non-integer, so omega comes
 * from the alternate / saddle-point samplers.  d0 > 0. */
int bl_nb_gibbs_dfreal(double *w_last, double *beta, double *d_out, const double *y, const double *tX, double d0,
                       const double *m0, const double *P0, int N, int P, int samp, int burn, uint64_t seed);
int bl_nb_gibbs_dfreal_dev(double *w_last, double *beta, double *d_out, const double *y, const double *tX, double d0,
                           const double *m0, const double *P0, int64_t N, int P, int samp, int burn, uint64_t seed,
                           uint64_t obs0, void *stream);

/* Device-resident shards (all pointers DEVICE pointers; one process per GPU).  Rank r holds
 * observations [obs0, obs0+N) of the global data set; with a communicator (bl_comm_init) the
 * ranks exchange one all-reduce of P*P+P doubles per beta draw and produce the same chain a
 * single GPU would. */
int bl_logit_gibbs_dev(double *w, double *beta, const double *y, const double *tX, const double *n,
                       const double *m0, const double *P0, int64_t N, int P, int samp, int burn,
                       uint64_t seed, int flags, uint64_t obs0, void *stream);
int bl_mlogit_gibbs_dev(double *w, double *beta, const double *ty, const double *tX, const double *n,
                        const double *m0, const double *P0, int64_t N, int P, int J, int samp, int burn,
                        uint64_t seed, int flags, uint64_t obs0, void *stream);
int bl_nb_gibbs_dev(double *w_last, double *beta, const double *y, const double *tX, double d,
                    const double *m0, const double *P0, int64_t N, int P, int samp, uint64_t seed,
                    uint64_t obs0, void *stream);
/* sharded rows: ymax, the count histogram and the four log-likelihood sums of every dispersion update are
 * all-reduced over the communicator (NCCL); d stays identical on every rank */
int bl_nb_gibbs_df_dev(double *w_last, double *beta, double *d_out, const double *y, const double *tX, double d0,
                       const double *m0, const double *P0, int64_t N, int P, int samp, int burn, uint64_t seed,
                       uint64_t obs0, void *stream);

/* A batch of independent logit chains (BASELINE config 5; no reference C symbol: the reference
 * would call gibbs() once per chain).  Chain c owns rows [c*N, (c+1)*N) of y, n (length chains*N)
 * and tX (P x chains*N), shares m0 / P0, and is the chain bl_logit_gibbs runs on those rows with
 * seed + c.  beta: [chains][samp][P] (chain c's P x samp block is what gibbs() would return);
 * omega is not returned.  flags: BL_GIBBS_PLAIN_BETA or 0 (the reference's constrained draw).
 * Block-distribute the chains over GPUs by calling with seed + first chain of the block. */
int bl_logit_chains(double *beta, const double *y, const double *tX, const double *n, const double *m0,
                    const double *P0, int chains, int N, int P, int samp, int burn, uint64_t seed, int flags);
int bl_logit_chains_dev(double *beta, const double *y, const double *tX, const double *n, const double *m0,
                        const double *P0, int chains, int64_t N, int P, int samp, int burn, uint64_t seed,
                        int flags, void *stream);

/* Several independent logit chains on ONE data set (the usual 4-8 chains from different seeds that R-hat and
 * effective-sample-size checks need).  y, n: [N], tX: P x N, shared by all chains, with m0 / P0.  Chain c is
 * bit for bit the chain bl_logit_chains runs when given `chains` copies of the data and the same seed, so it
 * uses the streams of seed + c; but X is held once and read once per iteration for all chains.
 * beta: [chains][samp][P]; omega is not returned.  flags: BL_GIBBS_PLAIN_BETA or 0 (the reference's constrained
 * draw), optionally BL_GIBBS_UNFUSED.  chains * N < 2^31; P as bl_logit_chains takes it (each chain's beta is drawn
 * by one CTA out of shared memory: P <= 91 with the constrained draw, P <= 111 with the plain one).  Duplicate rows
 * are not merged.  One chain runs faster through bl_logit_gibbs (a different, equally valid chain).
 * Spread the chains over GPUs by giving each rank the whole X and a block of chains, called with
 * seed + first chain of the block.  The host entry copies X to the device once. */
int bl_logit_multichain(double *beta, const double *y, const double *tX, const double *n, const double *m0,
                        const double *P0, int chains, int N, int P, int samp, int burn, uint64_t seed, int flags);
int bl_logit_multichain_dev(double *beta, const double *y, const double *tX, const double *n, const double *m0,
                            const double *P0, int chains, int64_t N, int P, int samp, int burn, uint64_t seed,
                            int flags, void *stream);

/* Several independent multinomial logit chains on ONE data set (the multinomial counterpart of
 * bl_logit_multichain).  ty: (J-1) x N, tX: P x N, n: [N], m0: P x (J-1), P0: P x P x (J-1), laid out as for
 * bl_mlogit_gibbs and shared by all chains.  beta: [chains][samp] blocks of P x (J-1); chain c's block is, bit for
 * bit, what bl_mlogit_gibbs(..., seed + c, BL_GIBBS_NO_W) returns.  omega is not returned.  X is held once and read
 * once per category update for up to 8 chains; the launches per iteration do not depend on the number of chains.
 * flags: 0 or BL_GIBBS_UNFUSED (separate psi and offsets kernels in every category update: the chains then equal
 * the single chain run with BL_MLOGIT_UNFUSED=1 in the environment); any other flag is refused.  Limits, checked
 * before anything is allocated: 1 <= chains <= 65535, J >= 2, chains * N < 2^31, P <= 111 (each chain's beta is drawn by one
 * CTA out of shared memory; the single-chain entry takes P <= 256).  Device memory beyond the data: 2 chains (J-1)
 * N doubles of linear predictors and their exponentials, and 32 bytes per (chain, row) of offsets, tilts, draws,
 * shapes and the draw's index list.  Duplicate rows are not
 * merged.  Spread the chains over GPUs by giving each rank the whole data set and a block of chains, called with
 * seed + first chain of the block.  The host entry copies ty, X and n to the device once. */
int bl_mlogit_multichain(double *beta, const double *ty, const double *tX, const double *n, const double *m0,
                         const double *P0, int chains, int N, int P, int J, int samp, int burn, uint64_t seed, int flags);
int bl_mlogit_multichain_dev(double *beta, const double *ty, const double *tX, const double *n, const double *m0,
                             const double *P0, int chains, int64_t N, int P, int J, int samp, int burn, uint64_t seed,
                             int flags, void *stream);

/* Several independent negative-binomial chains on ONE data set (the NB counterpart of bl_logit_multichain; R-hat on
 * the dispersion d is the usual first check).  y: counts [N], tX: P x N, shared by all chains with m0 / P0.
 * dmode picks the chain every chain runs:
 *   BL_NB_D_FIXED  d = d0 throughout: chain c's beta is rows burn .. burn + samp - 1 of
 *                  bl_nb_gibbs(..., samp + burn, seed + c), bit for bit (d_out, if given, is filled with d0);
 *   BL_NB_D_INT    draw.df on the integers: chain c's beta and d are bl_nb_gibbs_df(..., seed + c), bit for bit;
 *   BL_NB_D_REAL   draw.df.real.mean: chain c's beta and d are bl_nb_gibbs_dfreal(..., seed + c), bit for bit.
 * beta: [chains][samp][P]; d_out: [chains][samp] or NULL; omega is not returned.  X is held once and read once per
 * iteration for up to 8 chains; the launches per iteration do not depend on the number of chains.  Limits, checked
 * before anything is allocated or launched: 1 <= chains <= 65535, chains * N < 2^31, P <= 256, d0 as the matching
 * single-chain entry takes it.  Spread the chains over GPUs by giving each rank the whole data set and a block of
 * chains, called with seed + first chain of the block.  The host entry copies y and X to the device once. */
#define BL_NB_D_FIXED 0   /* d = d0 throughout: the chain of bl_nb_gibbs */
#define BL_NB_D_INT   1   /* draw.df on the integers: the chain of bl_nb_gibbs_df */
#define BL_NB_D_REAL  2   /* draw.df.real.mean: the chain of bl_nb_gibbs_dfreal */
int bl_nb_multichain(double *beta, double *d_out, const double *y, const double *tX, double d0,
                     const double *m0, const double *P0, int chains, int N, int P, int samp, int burn,
                     uint64_t seed, int dmode);
int bl_nb_multichain_dev(double *beta, double *d_out, const double *y, const double *tX, double d0,
                         const double *m0, const double *P0, int chains, int64_t N, int P, int samp, int burn,
                         uint64_t seed, int dmode, void *stream);

/* Binomial logit with group random intercepts (the GLMM with one grouping factor: patients within hospitals,
 * pupils within schools, repeated measures on a subject; the reference ships it only as Logit-MixedModel.R):
 *   logit P(success_i) = x_i' beta + u_{g_i},  u_g ~ N(0, tau2),  beta ~ N(m0, P0^-1),  tau2 ~ IG(a0, b0).
 * y: proportions [N], n: trials [N] (truncated to int), tX: P x N, group: ids in [0, G) [N], m0 [P], P0: P x P
 * (a precision).  The chain starts from beta = 0, u = 0, tau2 = tau2_0; each iteration draws omega | beta, u, then
 * u | omega, beta, tau2 (one normal per group), tau2 | u, then beta | omega, u with the unconstrained draw (streams:
 * DESIGN.md section 3).  After burn iterations, samp are kept: beta: samp x P (row t = iteration burn + t),
 * u: samp x G or NULL (no u draws stored), tau2: [samp].  One chain on the current GPU.  flags: 0 or
 * BL_GIBBS_UNFUSED (same chain, bit for bit).  Refused with their own messages, outputs untouched: G < 1, an id
 * outside [0, G) (checked on the host by bl_logit_ri_gibbs, on the device before the first iteration by the _dev
 * entry), a0 / b0 / tau2_0 not finite and positive, N outside [1, 2^31), P < 1, samp < 1, burn < 0, P > 256, any
 * other flag.  Duplicate rows are not merged. */
int bl_logit_ri_gibbs(double *beta, double *u, double *tau2, const double *y, const double *tX, const double *n,
                      const int *group, int G, const double *m0, const double *P0, double a0, double b0,
                      double tau2_0, int64_t N, int P, int samp, int burn, uint64_t seed, int flags);
/* The same on device-resident data (all pointers DEVICE pointers), enqueued on `stream` (a cudaStream_t). */
int bl_logit_ri_gibbs_dev(double *beta, double *u, double *tau2, const double *y, const double *tX, const double *n,
                          const int *group, int G, const double *m0, const double *P0, double a0, double b0,
                          double tau2_0, int64_t N, int P, int samp, int burn, uint64_t seed, int flags, void *stream);

/* Communicator over NCCL (NVLink/NVSwitch): rank 0 creates a 128-byte id, the host side
 * broadcasts it (e.g. torch.distributed), every rank calls bl_comm_init. */
int bl_comm_unique_id(void *out128);
int bl_comm_init(const void *id128, int rank, int world);
int bl_comm_destroy(void);
/* The same ranks WITHOUT an NCCL communicator: every exchange then goes through the peer windows
 * below, which must be opened (bl_comm_peer_handle / bl_comm_peer_open) before the first sharded
 * sweep.  For ranks NCCL cannot join -- several processes sharing one device (how the exchange is
 * tested on a one-GPU box) -- or to keep NCCL out of the process altogether. */
int bl_comm_init_local(int rank, int world);

/* Peer windows (ranks on one NVLink/NVSwitch node, at most 8): with them open, the sharded sweeps
 * exchange the P*P + P sums of each beta draw through one fused kernel pair instead of
 * ncclAllReduce -- the Gram reduce kernel stores its sums into every rank's window over NVLink and
 * the beta-draw kernel adds the windows' slots in rank order (bit-identical on every rank).
 * After bl_comm_init: every rank calls bl_comm_peer_handle (64-byte CUDA IPC handle of its
 * window), the host all-gathers the handles in rank order, every rank calls bl_comm_peer_open
 * with the world*64 bytes.  All ranks must open (or none): bl_comm_peer_close on failure anywhere.
 * bl_comm_peer_active() != 0 when the sweeps will use the windows. */
int bl_comm_peer_handle(void *out64);
int bl_comm_peer_open(const void *handles);
int bl_comm_peer_close(void);
int bl_comm_peer_active(void);

/* Virtual ranks -- a test aid for boxes with fewer GPUs than ranks.  bl_vcomm_create(world) makes a
 * communicator of `world` ranks that all live in THIS process on THIS device (windows = plain device
 * allocations); a host thread calls bl_vcomm_bind(r) and then the *_dev sweeps on its shard, every
 * thread passing the SAME CUDA stream.  The threads meet at a host barrier inside every exchange,
 * between enqueueing its producing and its consuming kernel, so in stream order all producers precede
 * all consumers and no kernel ever waits for a later one.  Kernels, slot/flag descriptors, epochs and
 * parities are those of the multi-GPU exchange.  bl_vcomm_bind(-1) unbinds the thread. */
int bl_vcomm_create(int world);
int bl_vcomm_bind(int rank);
int bl_vcomm_destroy(void);

/* Component probes for parity tests (host pointers, elementwise). */
int bl_probe_pg_moments(double *m1, double *m2, const double *b, const double *z, int64_t num);
int bl_probe_v_eval(double *v, const double *y, int64_t num);
int bl_probe_specfun(double *out, int which, const double *a, const double *b, const double *c,
                     int64_t num);
int bl_probe_philox(uint32_t *out4, const uint32_t *ctr4, const uint32_t *key2);
/* One negative-binomial dispersion step per chain (real_d = 0: draw.df on the integers, 1: draw.df.real.mean), run
 * with the kernels and grids of bl_nb_gibbs_df / bl_nb_gibbs_dfreal (chains = 1) and bl_nb_multichain, on given
 * phi [chains][N] (phi = X beta of chain c at phi + c N), counts y [N] and d [chains]; chain c keys its Metropolis
 * stream by seed + c and call.  out [chains][5] = {proposal d', accept variate (u; real walk: log u), llh(d),
 * llh(d'), new d}. */
int bl_probe_nb_dispersion(double *out, const double *phi, const double *y, const double *d, int chains, int64_t N,
                           uint64_t seed, uint32_t call, int real_d);

/* Pipe-throughput microbenchmarks on the current device, the denominators of the sampler's compute
 * roofline (bench.py): out6 = FP64 FMA TFLOP/s, FP32 FMA TFLOP/s, MUFU (ex2/lg2) Gop/s, FP64 tensor
 * (DMMA m8n8k4) TFLOP/s, 32x32->64 integer multiply + fold (one Philox round half) Gop/s, issued warp
 * instructions G/s.  Best of four launches each, ~10 ms in total. */
int bl_probe_peaks(double *out6);
/* FP64 tensor (DMMA) TFLOP/s with one, two, four and eight resident warps per scheduler: out8[0..4) with the
 * same A/B registers in every MMA, out16[4..8) with operands that change from MMA to MMA, [8..12) / [12..16) with a
 * DMUL forming the A operand in front of every 4 / 8 MMAs, as in a weighted Gram (design aid). */
int bl_probe_dmma_scaling(double *out16);

/* Host logic probe (no device needed): chunk sizes, in order, that the host-pointer entry points use to
 * stream a batch of num observations through HBM (small chunks open and close the batch so the pipeline
 * fills and drains quickly).  Writes at most cap sizes; returns the number of chunks, -1 for num < 0. */
int bl_probe_pipeline_schedule(int64_t num, int64_t *sizes, int cap);

/* Number of kernels this library has launched since load (bench accounting). */
uint64_t bl_kernel_launches(void);

/* Per-stage CUDA-event timing of the regime-binned rpg_hybrid path (measurement aid): after
 * bl_hybrid_timing(1), bl_hybrid_timing_last() returns, for the last launch, the milliseconds of
 * [binning, saddle-point set-up, saddle-point loop, alternate set-up, alternate loop,
 *  sum-of-gammas, normal, Devroye] and (launches8 may be null) the non-empty kernel launches
 * each figure sums over. */
void bl_hybrid_timing(int enable);
int bl_hybrid_timing_last(double *ms8, int *launches8);

#ifdef __cplusplus
}
#endif
#endif
