// Internal host-side interface between the C ABI (capi.cu) and the kernels.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "../../include/bayeslogit_b200.h"

namespace bl {

// kDevroyePlain: the unfiltered all-fp64 Devroye path, kept for A/B equality tests
// kDevroyeLoop: the filtered sampler in a plain per-lane loop (no persistent-lane refill)
enum Method { kDevroye = 0, kGamma = 1, kAlt = 2, kSP = 3, kHybrid = 4, kDevroyePlain = 5, kDevroyeLoop = 6 };

// Stream identity of a batch (see philox.cuh).
struct StreamId {
    uint64_t seed;
    uint64_t obs0;
    uint32_t call_id;
    // batched independent chains: > 0 means position i of the batch is observation i % chain_len of
    // chain i / chain_len, whose streams are keyed by seed + chain (batch size < 2^31)
    uint32_t chain_len = 0;
};

// Device-side tape descriptor (device pointers).
struct DevTape {
    const double *tu, *te, *tn, *tg;
    int lu, le, ln, lg;
};

// Batch draw, Philox streams.  shape: int32 for kDevroye, double otherwise.  id.chain_len keys the streams by chain for
// kDevroye and kHybrid (launch_hybrid_binned likewise).
cudaError_t launch_rpg(Method m, double *x, const void *shape, const double *z, int64_t num,
                       int trunc, int *iter, StreamId id, cudaStream_t stream);

// Batch draw from tapes; trace may be null.
cudaError_t launch_rpg_tape(Method m, double *x, const void *shape, const double *z, int64_t num,
                            int trunc, int *iter, DevTape tape, int *trace, cudaStream_t stream);

cudaError_t launch_probe_moments(double *m1, double *m2, const double *b, const double *z,
                                 int64_t num, cudaStream_t stream);
cudaError_t launch_probe_v_eval(double *v, const double *y, int64_t num, cudaStream_t stream);
cudaError_t launch_probe_specfun(double *out, int which, const double *a, const double *b,
                                 const double *c, int64_t num, cudaStream_t stream);
cudaError_t launch_probe_philox(uint32_t *out4, const uint32_t *ctr4, const uint32_t *key2,
                                cudaStream_t stream);

// `work` (optional, hybrid_workspace_bytes(num) bytes): enables branch-class binning for batches of at least
// `bin_min` draws (BL_DEVROYE_BIN_MIN overrides).  z ~ U(-5, 5) gains nothing below ~2^20 draws; the one-sided
// tilts of an mlogit sweep (eta = psi_j - log sum exp) gain 30 % at 10^6.
cudaError_t launch_devroye_refill(double *x, const int *n, const double *z, int64_t num,
                                  StreamId id, cudaStream_t stream, void *work = nullptr, int64_t bin_min = 1 << 20,
                                  bool prebinned = false);   // prebinned: work already holds the class-ordered index list
bool devroye_binned(int64_t num, int64_t bin_min);         // whether a batch of this size takes the binned path

// Fused psi = X beta + omega = PG(n, psi) of the logit sweeps (pg_devroye_kernel.cu); needs even P and a
// 16-byte aligned tX (logit_psi_draw_ok).  chains > 1: rows [c N, (c+1) N) meet beta + c * beta_stride and
// id.chain_len = N keys their streams by seed + c.  off (one chain): omega_i = PG(n_i, x_i . beta + off_i), psi_out
// keeps x_i . beta.
bool logit_psi_draw_ok(const double *tX, int P);
cudaError_t launch_logit_psi_draw(double *x, double *psi_out, const int *n, const double *tX, const double *beta,
                                  int64_t beta_stride, int chains, int64_t N, int P, StreamId id, cudaStream_t stream,
                                  const double *off = nullptr);
// The same for `chains` chains that share ONE set of N rows (n [N], tX P x N): chain c meets beta + c * beta_stride
// and the streams of id.seed + c; x: omega [chains][N].  Same conditions on P and tX.  off [chains][N] (the
// random-intercept logit): omega = PG(n_i, x_i . beta_c + off[c][i]), psi_out [chains][N] keeps x_i . beta_c.
cudaError_t launch_logit_psi_draw_shared(double *x, const int *n, const double *tX, const double *beta,
                                         int64_t beta_stride, int chains, int64_t N, int P, StreamId id, cudaStream_t stream,
                                         double *psi_out = nullptr, const double *off = nullptr);

// rpg_hybrid through regime binning (pg_hybrid.cu); num <= 2^31-1, `work` = device scratch of
// hybrid_workspace_bytes(num) bytes that stays valid until the stream has drained.
size_t hybrid_workspace_bytes(int64_t num);
cudaError_t launch_hybrid_binned(double *x, const double *h, const double *z, int num, StreamId id,
                                 void *work, cudaStream_t stream);

// Gibbs sweeps on device-resident data (gibbs.cu); return 0 on success, message in err.
int logit_gibbs_device(double *w_out, double *beta_out, const double *y, const double *tX,
                       const double *n, const double *m0, const double *P0, int64_t N, int P,
                       int samp, int burn, uint64_t seed, int flags, uint64_t obs0, bool sharded,
                       cudaStream_t st, std::string &err, int w_every = 1);   // w_out: N x ceil(samp / w_every)
int mlogit_gibbs_device(double *w_out, double *beta_out, const double *ty, const double *tX,
                        const double *n, const double *m0, const double *P0, int64_t N, int P, int J,
                        int samp, int burn, uint64_t seed, int flags, uint64_t obs0, bool sharded,
                        cudaStream_t st, std::string &err);
int nb_gibbs_device(double *w_out, double *beta_out, const double *y, const double *tX, double d,
                    const double *m0, const double *P0, int64_t N, int P, int samp, uint64_t seed,
                    uint64_t obs0, bool sharded, cudaStream_t st, std::string &err);
int nb_gibbs_df_device(double *w_out, double *beta_out, double *d_out, const double *y, const double *tX,
                       double d0, const double *m0, const double *P0, int64_t N, int P, int samp, int burn,
                       uint64_t seed, uint64_t obs0, bool sharded, int real_d, cudaStream_t st, std::string &err);
// Binomial logit with group random intercepts, one chain (gibbs.cu).  logit_ri_check refuses what the driver cannot
// run (every argument but the ids); the driver checks the ids on the device before anything else runs.
int logit_ri_check(int64_t N, int P, int G, int samp, int burn, double a0, double b0, double tau2_0, int flags,
                   std::string &err, const char *who = "logit_ri_gibbs");   // who: the messages' prefix
extern const char *const kLogitRiBadIdMsg;
int logit_ri_gibbs_device(double *beta_out, double *u_out, double *tau2_out, const double *y, const double *tX,
                          const double *n, const int *group, int G, const double *m0, const double *P0, double a0,
                          double b0, double tau2_0, int64_t N, int P, int samp, int burn, uint64_t seed, int flags,
                          cudaStream_t st, std::string &err);
// Several random-intercept chains on one data set (y, n, group [N], tX P x N, shared); beta_out: [chains][samp][P],
// u_out: [chains][samp][G] or null, tau2_out: [chains][samp].  The check refuses every argument the driver cannot run
// but the ids, before anything is allocated or launched; the driver checks the ids on the device first.
int logit_ri_multichain_check(int chains, int64_t N, int P, int G, int samp, int burn, double a0, double b0,
                              double tau2_0, int flags, std::string &err);
extern const char *const kLogitRiMultichainBadIdMsg;
int logit_ri_multichain_device(double *beta_out, double *u_out, double *tau2_out, const double *y, const double *tX,
                               const double *n, const int *group, int G, const double *m0, const double *P0, double a0,
                               double b0, double tau2_0, int chains, int64_t N, int P, int samp, int burn, uint64_t seed,
                               int flags, cudaStream_t st, std::string &err);
// Negative binomial with group random intercepts, one chain (gibbs.cu).  nb_ri_check refuses what the driver cannot
// run (every argument but the ids and the counts); the driver checks those on the device before anything else runs.
// dmode: BL_NB_D_FIXED / _INT / _REAL.  d_out: [samp] or null.
int nb_ri_check(int64_t N, int P, int G, int samp, int burn, double a0, double b0, double tau2_0, double d0, int dmode,
                std::string &err);
extern const char *const kNbRiBadIdMsg;
int nb_ri_gibbs_device(double *beta_out, double *u_out, double *tau2_out, double *d_out, const double *y,
                       const double *tX, const int *group, int G, const double *m0, const double *P0, double a0,
                       double b0, double tau2_0, double d0, int dmode, int64_t N, int P, int samp, int burn,
                       uint64_t seed, cudaStream_t st, std::string &err);
// shared_rows: every chain runs on the same N rows (y, n [N], tX P x N) instead of rows [c N, (c+1) N) of its own
int logit_chains_device(double *beta_out, const double *y, const double *tX, const double *n,
                        const double *m0, const double *P0, int chains, int64_t N, int P, int samp, int burn,
                        uint64_t seed, int flags, bool shared_rows, cudaStream_t st, std::string &err);
// Several multinomial logit chains on one data set (ty (J-1) x N, tX P x N, n [N], shared); beta_out: [chains][samp]
// blocks of P x (J-1).  The check refuses what the driver cannot run, before anything is allocated or launched.
int mlogit_multichain_check(int chains, int64_t N, int P, int J, int samp, int burn, int flags, std::string &err);
int mlogit_multichain_device(double *beta_out, const double *ty, const double *tX, const double *n, const double *m0,
                             const double *P0, int chains, int64_t N, int P, int J, int samp, int burn, uint64_t seed,
                             int flags, cudaStream_t st, std::string &err);
// Several negative-binomial chains on one data set (y [N], tX P x N, shared); beta_out: [chains][samp][P], d_out:
// [chains][samp] or null.  dmode: BL_NB_D_FIXED / _INT / _REAL.  The check refuses what the driver cannot run, before
// anything is allocated or launched.
int nb_multichain_check(int chains, int64_t N, int P, int samp, int burn, double d0, int dmode, std::string &err);
int nb_multichain_device(double *beta_out, double *d_out, const double *y, const double *tX, double d0, const double *m0,
                         const double *P0, int chains, int64_t N, int P, int samp, int burn, uint64_t seed, int dmode,
                         cudaStream_t st, std::string &err);
int nb_dispersion_probe(double *out, const double *phi, const double *y, const double *d, int chains, int64_t N,
                        uint64_t seed, uint32_t call, int real_d, cudaStream_t st, std::string &err);
int logit_em_device(double *beta, const double *y, const double *tX, const double *n, int64_t N,
                    int P, double tol, int max_iter, int *iters, cudaStream_t st, std::string &err);
// duplicate-row merge on device-resident data (merge.cu); returns M, -1 (CUDA error), -2 (needs the exact host merge)
int merge_rows_device(double *ty, double *tX, double *n, int N, int P, int ny, cudaStream_t st, std::string &err);
// stable sort of the rows 0..n-1 by key (0 <= key < nkeys) on the device (merge.cu): order[k] = row at sorted
// position k, key_sorted[k] = its key; rows with equal keys stay in increasing order
int sort_rows_by_key(int *order, int *key_sorted, const int *key, int n, int nkeys, cudaStream_t st, std::string &err);
int comm_unique_id(void *out128, std::string &err);
int comm_init(const void *id128, int rank, int world, std::string &err);
int comm_init_local(int rank, int world, std::string &err);
void comm_destroy();
int comm_peer_handle(void *out64, std::string &err);
int comm_peer_open(const void *handles, std::string &err);
void comm_peer_close();
int comm_peer_active();
int comm_virtual_create(int world, std::string &err);
int comm_virtual_bind(int rank, std::string &err);
void comm_virtual_destroy();

// pipe-throughput microbenchmarks (probe_peaks.cu)
int probe_peaks(double *out6, cudaStream_t stream, std::string &err);
int probe_dmma_scaling(double *out4, cudaStream_t stream, std::string &err);

void hybrid_timing_enable(bool on);
int hybrid_timing_last(double *ms8, int *launches8);

void count_launch(int n = 1);

// Programmatic dependent launch for the kernels of the Gibbs sweeps' inner loops: launch_pdl() sets the attribute
// (BL_GIBBS_NO_PDL in the environment drops it) and the kernel opens with BL_PDL_ENTER(), which waits until the kernel
// before it has completed and its writes are visible -- the launch latency between two kernels leaves the critical
// path.  No-op in a kernel launched without the attribute (<<< >>>).  The kernels do NOT trigger their dependents
// early (griddepcontrol.launch_dependents): the Gram kernels are sized for exactly one wave of CTAs, and a
// successor's CTAs that take their places while they wait cost a second, partial wave (measured: packed Gram 97 ->
// 148 us, N = 1M logit iteration 396 -> 449 us).
#define BL_PDL_ENTER() asm volatile("griddepcontrol.wait;" ::: "memory")

bool pdl_enabled();

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

}  // namespace bl

// internal hooks of the context in capi.cu
extern "C" {
int bl_ensure_ready_internal(void);
void bl_set_error_internal(const char *msg);
void *bl_stream_internal(void);
uint64_t bl_next_call_internal(void);
}

namespace bl {

}  // namespace bl
