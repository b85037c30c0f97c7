// C ABI of the Gibbs path: the reference's gibbs / EM / combine / mult_gibbs /
// mult_combine (LogitWrapper.h:39-62; bodies LogitWrapper.cpp:176-409) and the
// bl_* extensions (explicit seed, device-resident shards, NB sweep, communicator).
//
// Host-pointer entry points copy the caller's buffers to HBM once, run the whole
// chain on the device and copy the chains back; errors are reported like the
// reference does ("Error: ..." + "Aborting Gibbs sampler.", outputs untouched,
// LogitWrapper.cpp:226-229).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>

#include "engine.h"

using namespace bl;

namespace {

int report(const std::string &msg, const char *abort_line)
{
    bl_set_error_internal(msg.c_str());
    fprintf(stderr, "Error: %s\n", msg.c_str());
    if (abort_line) fprintf(stderr, "%s\n", abort_line);
    return 1;
}

struct Dev {
    std::vector<void *> ptrs;
    ~Dev() { for (void *p : ptrs) cudaFree(p); }
    void *put_bytes(const void *host, size_t bytes, std::string &err)
    {
        void *p = nullptr;
        cudaError_t e = cudaMalloc(&p, bytes ? bytes : 8);
        if (e == cudaSuccess && host) e = cudaMemcpy(p, host, bytes, cudaMemcpyHostToDevice);
        // pageable source: wait for the DMA itself, the sweeps run on a stream that does not order
        // against the legacy stream
        if (e == cudaSuccess && host) e = cudaStreamSynchronize(cudaStreamLegacy);
        if (e != cudaSuccess) { err = std::string("device buffer: ") + cudaGetErrorString(e); if (p) cudaFree(p); return nullptr; }
        ptrs.push_back(p);
        return p;
    }
    double *put(const double *host, size_t count, std::string &err)
    {
        return (double *)put_bytes(host, count * sizeof(double), err);
    }
};

// Merge observations with identical covariate rows, keeping first-occurrence order:
// y <- n-weighted mean, n <- sum.  Same result as the reference's O(N^2) list walk
// (Logit::compress, Logit.hpp:192-270; MultLogit::set_data, MultLogit.hpp:137-208),
// done in O(N P) with a hash of the row bytes.  ny = number of y rows per
// observation (1 for logit, J-1 for mlogit; ty is ny x N column-major).
int merge_rows(double *ty, double *tX, double *n, int N, int P, int ny)
{
    struct Key {
        const double *p; int len;
        bool operator==(const Key &o) const
        {
            for (int k = 0; k < len; ++k) if (!(p[k] == o.p[k])) return false;   // Matrix operator== : elementwise ==
            return true;
        }
    };
    struct Hash {
        size_t operator()(const Key &k) const
        {
            uint64_t h = 1469598103934665603ull;
            for (int i = 0; i < k.len; ++i) {
                double v = k.p[i] == 0.0 ? 0.0 : k.p[i];   // +0 and -0 compare equal
                uint64_t b;
                memcpy(&b, &v, 8);
                h = (h ^ b) * 1099511628211ull;
            }
            return (size_t)h;
        }
    };
    std::unordered_map<Key, int, Hash> first;
    first.reserve((size_t)N * 2);
    std::vector<int> keep;
    keep.reserve(N);
    for (int i = 0; i < N; ++i) {
        Key k{tX + (size_t)P * i, P};
        auto it = first.find(k);
        if (it == first.end()) {
            first.emplace(k, i);
            keep.push_back(i);
        } else {
            int f = it->second;
            double sum = n[f] + n[i];
            for (int r = 0; r < ny; ++r)
                ty[r + (size_t)ny * f] = (n[f] / sum) * ty[r + (size_t)ny * f] + (n[i] / sum) * ty[r + (size_t)ny * i];
            n[f] = sum;
        }
    }
    int M = (int)keep.size();
    if (M != N) {
        for (int k = 0; k < M; ++k) {
            int i = keep[k];
            if (i == k) continue;
            memmove(tX + (size_t)P * k, tX + (size_t)P * i, sizeof(double) * P);
            memmove(ty + (size_t)ny * k, ty + (size_t)ny * i, sizeof(double) * ny);
            n[k] = n[i];
        }
        printf("Warning: data was combined!\n");     // Logit.hpp:248-251
        printf("N: %i, P: %i \n", M, P);
    }
    return M;
}

// The merge the entry points use: on the device (merge.cu: row hashes, a stable radix sort by first occurrence,
// the reference's running weighted mean replayed per group -- bit-identical to merge_rows) for data sets large
// enough to pay for the upload; the exact host merge for small ones, when no device is usable, or when the device
// path reports rows it cannot decide by hash (a collision, NaN covariates).  BAYESLOGIT_MERGE=host|device forces one.
int merge_rows_auto(double *ty, double *tX, double *n, int N, int P, int ny)
{
    const char *mode = getenv("BAYESLOGIT_MERGE");
    const bool force_host = mode && !strcmp(mode, "host"), force_dev = mode && !strcmp(mode, "device");
    if (force_host || (!force_dev && (size_t)N * P < (1u << 16))) return merge_rows(ty, tX, n, N, P, ny);
    if (bl_ensure_ready_internal()) {
        if (force_dev) return N;                         // the error is set; nothing merged
        bl_set_error_internal("");
        return merge_rows(ty, tX, n, N, P, ny);
    }
    std::string err;
    Dev d;
    double *dy = d.put(ty, (size_t)N * ny, err), *dX = d.put(tX, (size_t)N * P, err), *dn = d.put(n, N, err);
    if (!err.empty()) { report(err, nullptr); return merge_rows(ty, tX, n, N, P, ny); }
    const int M = merge_rows_device(dy, dX, dn, N, P, ny, (cudaStream_t)bl_stream_internal(), err);
    if (M == -2) return merge_rows(ty, tX, n, N, P, ny);
    if (M < 0) { report(err, nullptr); return merge_rows(ty, tX, n, N, P, ny); }
    if (M != N) {
        cudaError_t e = cudaMemcpy(ty, dy, sizeof(double) * (size_t)M * ny, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(tX, dX, sizeof(double) * (size_t)M * P, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(n, dn, sizeof(double) * M, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) { report(cudaGetErrorString(e), nullptr); return N; }
        printf("Warning: data was combined!\n");     // Logit.hpp:248-251
        printf("N: %i, P: %i \n", M, P);
    }
    return M;
}

uint64_t dropin_seed()
{
    // the reference draws from R's global generator; here: (engine seed, call counter) -> chain seed.
    // Always through the mixer: the chain's streams (seed', obs i, call t) must never coincide with the
    // streams (seed, obs i, call c) of the drop-in rpg_* calls that share the engine seed.
    uint64_t s = bl_get_seed();
    uint64_t c = bl_next_call_internal();
    uint64_t x = s + 0x9E3779B97F4A7C15ull * (c + 1);
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;
    return x ? x : 0x9E3779B97F4A7C15ull;
}

int host_logit(double *w, double *beta, const double *y, const double *tX, const double *n,
               const double *m0, const double *P0, int N, int P, int samp, int burn, uint64_t seed,
               int flags, int w_every = 1)
{
    if (bl_ensure_ready_internal()) return 1;
    if (N <= 0 || P <= 0 || samp <= 0 || burn < 0 || w_every < 1) return report("gibbs: bad dimensions", "Aborting Gibbs sampler.");
    const size_t wslots = ((size_t)samp + w_every - 1) / w_every;
    std::string err;
    Dev d;
    double *dy = d.put(y, N, err), *dX = d.put(tX, (size_t)N * P, err), *dn = d.put(n, N, err);
    double *dm0 = d.put(m0, P, err), *dP0 = d.put(P0, (size_t)P * P, err);
    bool keep_w = w && !(flags & BL_GIBBS_NO_W);
    double *dw = keep_w ? d.put(nullptr, (size_t)N * wslots, err) : nullptr;
    double *dbeta = d.put(nullptr, (size_t)P * samp, err);
    if (!err.empty()) return report(err, "Aborting Gibbs sampler.");
    cudaStream_t st = (cudaStream_t)bl_stream_internal();
    if (logit_gibbs_device(dw, dbeta, dy, dX, dn, dm0, dP0, N, P, samp, burn, seed,
                           keep_w ? flags : (flags | BL_GIBBS_NO_W), 0, false, st, err, w_every))
        return report(err, "Aborting Gibbs sampler.");
    cudaError_t e = cudaMemcpy(beta, dbeta, sizeof(double) * (size_t)P * samp, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && keep_w) e = cudaMemcpy(w, dw, sizeof(double) * (size_t)N * wslots, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return report(cudaGetErrorString(e), "Aborting Gibbs sampler.");
    return 0;
}

int host_mlogit(double *w, double *beta, const double *ty, const double *tX, const double *n,
                const double *m0, const double *P0, int N, int P, int J, int samp, int burn,
                uint64_t seed, int flags)
{
    if (bl_ensure_ready_internal()) return 1;
    if (N <= 0 || P <= 0 || J < 2 || samp <= 0 || burn < 0) return report("mult_gibbs: bad dimensions", "Aborting Gibbs sampler.");
    const int U = J - 1;
    std::string err;
    Dev d;
    double *dy = d.put(ty, (size_t)N * U, err), *dX = d.put(tX, (size_t)N * P, err), *dn = d.put(n, N, err);
    double *dm0 = d.put(m0, (size_t)P * U, err), *dP0 = d.put(P0, (size_t)P * P * U, err);
    bool keep_w = w && !(flags & BL_GIBBS_NO_W);
    double *dw = keep_w ? d.put(nullptr, (size_t)N * U * samp, err) : nullptr;
    double *dbeta = d.put(nullptr, (size_t)P * U * samp, err);
    if (!err.empty()) return report(err, "Aborting Gibbs sampler.");
    cudaStream_t st = (cudaStream_t)bl_stream_internal();
    if (mlogit_gibbs_device(dw, dbeta, dy, dX, dn, dm0, dP0, N, P, J, samp, burn, seed,
                            keep_w ? flags : (flags | BL_GIBBS_NO_W), 0, false, st, err))
        return report(err, "Aborting Gibbs sampler.");
    cudaError_t e = cudaMemcpy(beta, dbeta, sizeof(double) * (size_t)P * U * samp, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && keep_w) e = cudaMemcpy(w, dw, sizeof(double) * (size_t)N * U * samp, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return report(cudaGetErrorString(e), "Aborting Gibbs sampler.");
    return 0;
}

}  // namespace

extern "C" {

// ---- reference entry points ---------------------------------------------------------

void gibbs(double *wp, double *betap, double *yp, double *tXp, double *np, double *m0p, double *P0p,
           int *N, int *P, int *samp, int *burn)
{
    if (!wp || !betap || !yp || !tXp || !np || !m0p || !P0p || !N || !P || !samp || !burn) {
        report("gibbs: null argument", "Aborting Gibbs sampler.");
        return;
    }
    // the reference's own compress() call is commented out here (LogitWrapper.cpp:202), so *N is unchanged
    host_logit(wp, betap, yp, tXp, np, m0p, P0p, *N, *P, *samp, *burn, dropin_seed(), 0);
}

void mult_gibbs(double *wp, double *betap, double *typ, double *tXp, double *np, double *m0p,
                double *P0p, int *N, int *P, int *J, int *sampp, int *burnp)
{
    if (!wp || !betap || !typ || !tXp || !np || !m0p || !P0p || !N || !P || !J || !sampp || !burnp) {
        report("mult_gibbs: null argument", "Aborting Gibbs sampler.");
        return;
    }
    // MultLogit's constructor merges duplicate rows (MultLogit.hpp:137-208); the reference works
    // on its own copies, so the caller's data buffers are left as they were
    int U = *J - 1;
    std::vector<double> ty(typ, typ + (size_t)U * *N), tX(tXp, tXp + (size_t)*P * *N), n(np, np + *N);
    int M = merge_rows_auto(ty.data(), tX.data(), n.data(), *N, *P, U);
    if (host_mlogit(wp, betap, ty.data(), tX.data(), n.data(), m0p, P0p, M, *P, *J, *sampp, *burnp,
                    dropin_seed(), 0) == 0)
        *N = M;
}

void combine(double *yp, double *tXp, double *np, int *N, int *P)
{
    if (!yp || !tXp || !np || !N || !P) { report("combine: null argument", "Aborting combine."); return; }
    *N = merge_rows_auto(yp, tXp, np, *N, *P, 1);
}

void mult_combine(double *typ, double *tXp, double *np, int *N, int *P, int *J)
{
    if (!typ || !tXp || !np || !N || !P || !J) { report("mult_combine: null argument", "Aborting combine."); return; }
    *N = merge_rows_auto(typ, tXp, np, *N, *P, *J - 1);
}

void EM(double *betap, double *yp, double *tXp, double *np, int *Np, int *Pp, double *tolp, int *max_iterp)
{
    if (!betap || !yp || !tXp || !np || !Np || !Pp || !tolp || !max_iterp) { report("EM: null argument", "Aborting EM."); return; }
    if (bl_ensure_ready_internal()) return;
    std::string err;
    Dev d;
    int N = *Np, P = *Pp;
    double *dy = d.put(yp, N, err), *dX = d.put(tXp, (size_t)N * P, err), *dn = d.put(np, N, err);
    double *dbeta = d.put(nullptr, P, err);
    if (!err.empty()) { report(err, "Aborting EM."); return; }
    int iters = 0;
    if (logit_em_device(dbeta, dy, dX, dn, N, P, *tolp, *max_iterp, &iters, (cudaStream_t)bl_stream_internal(), err)) {
        report(err, "Aborting EM.");
        return;
    }
    if (cudaMemcpy(betap, dbeta, sizeof(double) * P, cudaMemcpyDeviceToHost) != cudaSuccess) { report("EM: copy back failed", "Aborting EM."); return; }
    *max_iterp = iters;
}

// ---- extensions ------------------------------------------------------------------------

int bl_logit_gibbs(double *w, double *beta, const double *y, const double *tX, const double *n,
                   const double *m0, const double *P0, int N, int P, int samp, int burn,
                   uint64_t seed, int flags)
{
    return host_logit(w, beta, y, tX, n, m0, P0, N, P, samp, burn, seed, flags);
}

int bl_logit_gibbs_thin(double *w, double *beta, const double *y, const double *tX, const double *n,
                        const double *m0, const double *P0, int N, int P, int samp, int burn,
                        uint64_t seed, int flags, int w_every)
{
    return host_logit(w, beta, y, tX, n, m0, P0, N, P, samp, burn, seed, flags, w_every);
}

// R-side seeding shim: .C("bl_set_seed_r", as.integer(seed)) next to set.seed(seed) (INTEGRATION.md)
void bl_set_seed_r(int *seed)
{
    if (seed) bl_set_seed((uint64_t)(uint32_t)*seed);
}

int bl_mlogit_gibbs(double *w, double *beta, const double *ty, const double *tX, const double *n,
                    const double *m0, const double *P0, int N, int P, int J, int samp, int burn,
                    uint64_t seed, int flags)
{
    return host_mlogit(w, beta, ty, tX, n, m0, P0, N, P, J, samp, burn, seed, flags);
}

int bl_nb_gibbs(double *w_last, double *beta, const double *y, const double *tX, double d,
                const double *m0, const double *P0, int N, int P, int samp, uint64_t seed)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    Dev dv;
    double *dy = dv.put(y, N, err), *dX = dv.put(tX, (size_t)N * P, err);
    double *dm0 = dv.put(m0, P, err), *dP0 = dv.put(P0, (size_t)P * P, err);
    double *dw = dv.put(nullptr, N, err), *dbeta = dv.put(nullptr, (size_t)P * samp, err);
    if (!err.empty()) return report(err, "Aborting Gibbs sampler.");
    if (nb_gibbs_device(dw, dbeta, dy, dX, d, dm0, dP0, N, P, samp, seed, 0, false, (cudaStream_t)bl_stream_internal(), err))
        return report(err, "Aborting Gibbs sampler.");
    cudaError_t e = cudaMemcpy(beta, dbeta, sizeof(double) * (size_t)P * samp, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && w_last) e = cudaMemcpy(w_last, dw, sizeof(double) * N, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return report(cudaGetErrorString(e), "Aborting Gibbs sampler.");
    return 0;
}

static int host_nb_gibbs_df(double *w_last, double *beta, double *d_out, const double *y, const double *tX, double d0,
                            const double *m0, const double *P0, int N, int P, int samp, int burn, uint64_t seed, int real_d)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    Dev dv;
    double *dy = dv.put(y, N, err), *dX = dv.put(tX, (size_t)N * P, err);
    double *dm0 = dv.put(m0, P, err), *dP0 = dv.put(P0, (size_t)P * P, err);
    double *dw = dv.put(nullptr, N, err), *dbeta = dv.put(nullptr, (size_t)P * samp, err);
    double *dd = dv.put(nullptr, samp, err);
    if (!err.empty()) return report(err, "Aborting Gibbs sampler.");
    if (nb_gibbs_df_device(dw, dbeta, dd, dy, dX, d0, dm0, dP0, N, P, samp, burn, seed, 0, false, real_d,
                           (cudaStream_t)bl_stream_internal(), err))
        return report(err, "Aborting Gibbs sampler.");
    cudaError_t e = cudaMemcpy(beta, dbeta, sizeof(double) * (size_t)P * samp, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(d_out, dd, sizeof(double) * samp, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && w_last) e = cudaMemcpy(w_last, dw, sizeof(double) * N, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return report(cudaGetErrorString(e), "Aborting Gibbs sampler.");
    return 0;
}

int bl_nb_gibbs_df(double *w_last, double *beta, double *d_out, const double *y, const double *tX, double d0,
                   const double *m0, const double *P0, int N, int P, int samp, int burn, uint64_t seed)
{
    return host_nb_gibbs_df(w_last, beta, d_out, y, tX, d0, m0, P0, N, P, samp, burn, seed, 0);
}

int bl_nb_gibbs_dfreal(double *w_last, double *beta, double *d_out, const double *y, const double *tX, double d0,
                       const double *m0, const double *P0, int N, int P, int samp, int burn, uint64_t seed)
{
    return host_nb_gibbs_df(w_last, beta, d_out, y, tX, d0, m0, P0, N, P, samp, burn, seed, 1);
}

int bl_nb_gibbs_dfreal_dev(double *w_last, double *beta, double *d_out, const double *y, const double *tX, double d0,
                           const double *m0, const double *P0, int64_t N, int P, int samp, int burn, uint64_t seed,
                           uint64_t obs0, void *stream)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    if (nb_gibbs_df_device(w_last, beta, d_out, y, tX, d0, m0, P0, N, P, samp, burn, seed, obs0, true, 1, (cudaStream_t)stream, err))
        return report(err, nullptr);
    return 0;
}

int bl_probe_nb_dispersion(double *out, const double *phi, const double *y, const double *d, int chains, int64_t N,
                           uint64_t seed, uint32_t call, int real_d)
{
    if (bl_ensure_ready_internal()) return 1;
    if (!out || !phi || !y || !d) return report("probe_nb_dispersion: null argument", nullptr);
    if (chains < 1 || chains > 65535 || N < 1 || (int64_t)chains * N >= (1LL << 31))
        return report("probe_nb_dispersion: bad dimensions", nullptr);
    for (int c = 0; c < chains; ++c)
        if (real_d ? !(d[c] > 0.0) : (!(d[c] >= 1.0) || d[c] != floor(d[c])))
            return report(real_d ? "probe_nb_dispersion: d must be positive"
                                 : "probe_nb_dispersion: d must be a positive integer", nullptr);
    std::string err;
    Dev dv;
    double *dphi = dv.put(phi, (size_t)chains * N, err), *dy = dv.put(y, N, err);
    double *dout = dv.put(nullptr, (size_t)chains * 5, err);
    if (!err.empty()) return report(err, nullptr);
    if (nb_dispersion_probe(dout, dphi, dy, d, chains, N, seed, call, real_d, (cudaStream_t)bl_stream_internal(), err))
        return report(err, nullptr);
    cudaError_t e = cudaMemcpy(out, dout, sizeof(double) * (size_t)chains * 5, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return report(cudaGetErrorString(e), nullptr);
    return 0;
}

int bl_nb_gibbs_df_dev(double *w_last, double *beta, double *d_out, const double *y, const double *tX, double d0,
                       const double *m0, const double *P0, int64_t N, int P, int samp, int burn, uint64_t seed,
                       uint64_t obs0, void *stream)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    if (nb_gibbs_df_device(w_last, beta, d_out, y, tX, d0, m0, P0, N, P, samp, burn, seed, obs0, true, 0, (cudaStream_t)stream, err))
        return report(err, nullptr);
    return 0;
}

int bl_logit_gibbs_dev(double *w, double *beta, const double *y, const double *tX, const double *n,
                       const double *m0, const double *P0, int64_t N, int P, int samp, int burn,
                       uint64_t seed, int flags, uint64_t obs0, void *stream)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    if (logit_gibbs_device(w, beta, y, tX, n, m0, P0, N, P, samp, burn, seed, flags, obs0, true, (cudaStream_t)stream, err))
        return report(err, nullptr);
    return 0;
}

int bl_logit_chains_dev(double *beta, const double *y, const double *tX, const double *n, const double *m0,
                        const double *P0, int chains, int64_t N, int P, int samp, int burn, uint64_t seed,
                        int flags, void *stream)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    if (logit_chains_device(beta, y, tX, n, m0, P0, chains, N, P, samp, burn, seed, flags, false, (cudaStream_t)stream, err))
        return report(err, nullptr);
    return 0;
}

int bl_logit_chains(double *beta, const double *y, const double *tX, const double *n, const double *m0,
                    const double *P0, int chains, int N, int P, int samp, int burn, uint64_t seed, int flags)
{
    if (bl_ensure_ready_internal()) return 1;
    if (chains <= 0 || N <= 0 || P <= 0 || samp <= 0 || burn < 0) return report("logit_chains: bad dimensions", nullptr);
    std::string err;
    Dev d;
    const size_t T = (size_t)chains * N;
    double *dy = d.put(y, T, err), *dX = d.put(tX, T * P, err), *dn = d.put(n, T, err);
    double *dm0 = d.put(m0, P, err), *dP0 = d.put(P0, (size_t)P * P, err);
    double *dbeta = d.put(nullptr, (size_t)chains * P * samp, err);
    if (!err.empty()) return report(err, nullptr);
    if (logit_chains_device(dbeta, dy, dX, dn, dm0, dP0, chains, N, P, samp, burn, seed, flags, false,
                            (cudaStream_t)bl_stream_internal(), err))
        return report(err, nullptr);
    cudaError_t e = cudaMemcpy(beta, dbeta, sizeof(double) * (size_t)chains * P * samp, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return report(cudaGetErrorString(e), nullptr);
    return 0;
}

int bl_logit_multichain_dev(double *beta, const double *y, const double *tX, const double *n, const double *m0,
                            const double *P0, int chains, int64_t N, int P, int samp, int burn, uint64_t seed,
                            int flags, void *stream)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    if (logit_chains_device(beta, y, tX, n, m0, P0, chains, N, P, samp, burn, seed, flags, true, (cudaStream_t)stream, err))
        return report(err, nullptr);
    return 0;
}

int bl_logit_multichain(double *beta, const double *y, const double *tX, const double *n, const double *m0,
                        const double *P0, int chains, int N, int P, int samp, int burn, uint64_t seed, int flags)
{
    if (bl_ensure_ready_internal()) return 1;
    // checked before any buffer is made: the device driver repeats the checks
    if (chains <= 0 || N <= 0 || P <= 0 || samp <= 0 || burn < 0) return report("logit_multichain: bad dimensions", nullptr);
    if ((int64_t)chains * N >= (1LL << 31))
        return report("logit_multichain: chains * N must stay below 2^31 observations per call", nullptr);
    if (P > 256) return report("P > 256 covariates is not supported by the single-CTA beta draw", nullptr);
    std::string err;
    Dev d;
    double *dy = d.put(y, N, err), *dX = d.put(tX, (size_t)N * P, err), *dn = d.put(n, N, err);     // one copy of X
    double *dm0 = d.put(m0, P, err), *dP0 = d.put(P0, (size_t)P * P, err);
    double *dbeta = d.put(nullptr, (size_t)chains * P * samp, err);
    if (!err.empty()) return report(err, nullptr);
    if (logit_chains_device(dbeta, dy, dX, dn, dm0, dP0, chains, N, P, samp, burn, seed, flags, true,
                            (cudaStream_t)bl_stream_internal(), err))
        return report(err, nullptr);
    cudaError_t e = cudaMemcpy(beta, dbeta, sizeof(double) * (size_t)chains * P * samp, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return report(cudaGetErrorString(e), nullptr);
    return 0;
}

int bl_mlogit_multichain_dev(double *beta, const double *ty, const double *tX, const double *n, const double *m0,
                             const double *P0, int chains, int64_t N, int P, int J, int samp, int burn, uint64_t seed,
                             int flags, void *stream)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    if (mlogit_multichain_device(beta, ty, tX, n, m0, P0, chains, N, P, J, samp, burn, seed, flags, (cudaStream_t)stream, err))
        return report(err, nullptr);
    return 0;
}

int bl_mlogit_multichain(double *beta, const double *ty, const double *tX, const double *n, const double *m0,
                         const double *P0, int chains, int N, int P, int J, int samp, int burn, uint64_t seed, int flags)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    // checked before any buffer is made: the device driver repeats the checks
    if (mlogit_multichain_check(chains, N, P, J, samp, burn, flags, err)) return report(err, nullptr);
    const int U = J - 1;
    Dev d;
    double *dy = d.put(ty, (size_t)N * U, err), *dX = d.put(tX, (size_t)N * P, err), *dn = d.put(n, N, err);   // one copy
    double *dm0 = d.put(m0, (size_t)P * U, err), *dP0 = d.put(P0, (size_t)P * P * U, err);
    const size_t nb = (size_t)chains * samp * U * P;
    double *dbeta = d.put(nullptr, nb, err);
    if (!err.empty()) return report(err, nullptr);
    if (mlogit_multichain_device(dbeta, dy, dX, dn, dm0, dP0, chains, N, P, J, samp, burn, seed, flags,
                                 (cudaStream_t)bl_stream_internal(), err))
        return report(err, nullptr);
    cudaError_t e = cudaMemcpy(beta, dbeta, sizeof(double) * nb, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return report(cudaGetErrorString(e), nullptr);
    return 0;
}

int bl_nb_multichain_dev(double *beta, double *d_out, const double *y, const double *tX, double d0,
                         const double *m0, const double *P0, int chains, int64_t N, int P, int samp, int burn,
                         uint64_t seed, int dmode, void *stream)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    if (nb_multichain_device(beta, d_out, y, tX, d0, m0, P0, chains, N, P, samp, burn, seed, dmode, (cudaStream_t)stream, err))
        return report(err, nullptr);
    return 0;
}

int bl_nb_multichain(double *beta, double *d_out, const double *y, const double *tX, double d0,
                     const double *m0, const double *P0, int chains, int N, int P, int samp, int burn,
                     uint64_t seed, int dmode)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    // checked before any buffer is made: the device driver repeats the checks
    if (nb_multichain_check(chains, N, P, samp, burn, d0, dmode, err)) return report(err, nullptr);
    Dev d;
    double *dy = d.put(y, N, err), *dX = d.put(tX, (size_t)N * P, err);        // one copy of the data
    double *dm0 = d.put(m0, P, err), *dP0 = d.put(P0, (size_t)P * P, err);
    const size_t nb = (size_t)chains * samp * P, nd = (size_t)chains * samp;
    double *dbeta = d.put(nullptr, nb, err), *dd = d_out ? d.put(nullptr, nd, err) : nullptr;
    if (!err.empty()) return report(err, nullptr);
    if (nb_multichain_device(dbeta, dd, dy, dX, d0, dm0, dP0, chains, N, P, samp, burn, seed, dmode,
                             (cudaStream_t)bl_stream_internal(), err))
        return report(err, nullptr);
    cudaError_t e = cudaMemcpy(beta, dbeta, sizeof(double) * nb, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && d_out) e = cudaMemcpy(d_out, dd, sizeof(double) * nd, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return report(cudaGetErrorString(e), nullptr);
    return 0;
}

int bl_mlogit_gibbs_dev(double *w, double *beta, const double *ty, const double *tX, const double *n,
                        const double *m0, const double *P0, int64_t N, int P, int J, int samp, int burn,
                        uint64_t seed, int flags, uint64_t obs0, void *stream)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    if (mlogit_gibbs_device(w, beta, ty, tX, n, m0, P0, N, P, J, samp, burn, seed, flags, obs0, true, (cudaStream_t)stream, err))
        return report(err, nullptr);
    return 0;
}

int bl_nb_gibbs_dev(double *w_last, double *beta, const double *y, const double *tX, double d,
                    const double *m0, const double *P0, int64_t N, int P, int samp, uint64_t seed,
                    uint64_t obs0, void *stream)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    if (nb_gibbs_device(w_last, beta, y, tX, d, m0, P0, N, P, samp, seed, obs0, true, (cudaStream_t)stream, err))
        return report(err, nullptr);
    return 0;
}

// ---- binomial logit with group random intercepts ----------------------------------------------------------

int bl_logit_ri_gibbs(double *beta, double *u, double *tau2, const double *y, const double *tX, const double *n,
                      const int *group, int G, const double *m0, const double *P0, double a0, double b0,
                      double tau2_0, int64_t N, int P, int samp, int burn, uint64_t seed, int flags)
{
    if (bl_ensure_ready_internal()) return 1;
    if (!beta || !tau2 || !y || !tX || !n || !group || !m0 || !P0) return report("logit_ri_gibbs: null argument", nullptr);
    std::string err;
    if (logit_ri_check(N, P, G, samp, burn, a0, b0, tau2_0, flags, err)) return report(err, nullptr);
    for (int64_t i = 0; i < N; ++i)
        if (group[i] < 0 || group[i] >= G) return report(kLogitRiBadIdMsg, nullptr);
    Dev d;
    double *dy = d.put(y, N, err), *dX = d.put(tX, (size_t)N * P, err), *dn = d.put(n, N, err);
    double *dm0 = d.put(m0, P, err), *dP0 = d.put(P0, (size_t)P * P, err);
    int *dg = (int *)d.put_bytes(group, sizeof(int) * (size_t)N, err);
    double *dbeta = d.put(nullptr, (size_t)P * samp, err), *dtau2 = d.put(nullptr, samp, err);
    double *du = u ? d.put(nullptr, (size_t)G * samp, err) : nullptr;
    if (!err.empty()) return report(err, nullptr);
    if (logit_ri_gibbs_device(dbeta, du, dtau2, dy, dX, dn, dg, G, dm0, dP0, a0, b0, tau2_0, N, P, samp, burn, seed, flags,
                              (cudaStream_t)bl_stream_internal(), err))
        return report(err, nullptr);
    cudaError_t e = cudaMemcpy(beta, dbeta, sizeof(double) * (size_t)P * samp, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(tau2, dtau2, sizeof(double) * samp, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && u) e = cudaMemcpy(u, du, sizeof(double) * (size_t)G * samp, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return report(cudaGetErrorString(e), nullptr);
    return 0;
}

int bl_logit_ri_gibbs_dev(double *beta, double *u, double *tau2, const double *y, const double *tX, const double *n,
                          const int *group, int G, const double *m0, const double *P0, double a0, double b0,
                          double tau2_0, int64_t N, int P, int samp, int burn, uint64_t seed, int flags, void *stream)
{
    if (bl_ensure_ready_internal()) return 1;
    if (!beta || !tau2 || !y || !tX || !n || !group || !m0 || !P0) return report("logit_ri_gibbs: null argument", nullptr);
    std::string err;
    if (logit_ri_gibbs_device(beta, u, tau2, y, tX, n, group, G, m0, P0, a0, b0, tau2_0, N, P, samp, burn, seed, flags,
                              (cudaStream_t)stream, err))
        return report(err, nullptr);
    return 0;
}

int bl_logit_ri_multichain(double *beta, double *u, double *tau2, const double *y, const double *tX, const double *n,
                           const int *group, int G, const double *m0, const double *P0, double a0, double b0,
                           double tau2_0, int chains, int64_t N, int P, int samp, int burn, uint64_t seed, int flags)
{
    if (bl_ensure_ready_internal()) return 1;
    if (!beta || !tau2 || !y || !tX || !n || !group || !m0 || !P0) return report("logit_ri_multichain: null argument", nullptr);
    std::string err;
    // checked before any buffer is made: the device driver repeats the checks
    if (logit_ri_multichain_check(chains, N, P, G, samp, burn, a0, b0, tau2_0, flags, err)) return report(err, nullptr);
    for (int64_t i = 0; i < N; ++i)
        if (group[i] < 0 || group[i] >= G) return report(kLogitRiMultichainBadIdMsg, nullptr);
    Dev d;
    double *dy = d.put(y, N, err), *dX = d.put(tX, (size_t)N * P, err), *dn = d.put(n, N, err);   // one copy of the data
    double *dm0 = d.put(m0, P, err), *dP0 = d.put(P0, (size_t)P * P, err);
    int *dg = (int *)d.put_bytes(group, sizeof(int) * (size_t)N, err);
    const size_t nb = (size_t)chains * samp * P, nt = (size_t)chains * samp, nu = (size_t)chains * samp * G;
    double *dbeta = d.put(nullptr, nb, err), *dtau2 = d.put(nullptr, nt, err);
    double *du = u ? d.put(nullptr, nu, err) : nullptr;
    if (!err.empty()) return report(err, nullptr);
    if (logit_ri_multichain_device(dbeta, du, dtau2, dy, dX, dn, dg, G, dm0, dP0, a0, b0, tau2_0, chains, N, P, samp, burn,
                                   seed, flags, (cudaStream_t)bl_stream_internal(), err))
        return report(err, nullptr);
    cudaError_t e = cudaMemcpy(beta, dbeta, sizeof(double) * nb, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(tau2, dtau2, sizeof(double) * nt, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && u) e = cudaMemcpy(u, du, sizeof(double) * nu, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return report(cudaGetErrorString(e), nullptr);
    return 0;
}

int bl_logit_ri_multichain_dev(double *beta, double *u, double *tau2, const double *y, const double *tX, const double *n,
                               const int *group, int G, const double *m0, const double *P0, double a0, double b0,
                               double tau2_0, int chains, int64_t N, int P, int samp, int burn, uint64_t seed, int flags,
                               void *stream)
{
    if (bl_ensure_ready_internal()) return 1;
    if (!beta || !tau2 || !y || !tX || !n || !group || !m0 || !P0) return report("logit_ri_multichain: null argument", nullptr);
    std::string err;
    if (logit_ri_multichain_device(beta, u, tau2, y, tX, n, group, G, m0, P0, a0, b0, tau2_0, chains, N, P, samp, burn,
                                   seed, flags, (cudaStream_t)stream, err))
        return report(err, nullptr);
    return 0;
}

// ---- negative binomial with group random intercepts -------------------------------------------------------

int bl_nb_ri_gibbs(double *beta, double *u, double *tau2, double *d_out, const double *y, const double *tX,
                   const int *group, int G, const double *m0, const double *P0, double a0, double b0, double tau2_0,
                   double d0, int dmode, int64_t N, int P, int samp, int burn, uint64_t seed)
{
    if (bl_ensure_ready_internal()) return 1;
    if (!beta || !tau2 || !y || !tX || !group || !m0 || !P0) return report("nb_ri_gibbs: null argument", nullptr);
    std::string err;
    if (nb_ri_check(N, P, G, samp, burn, a0, b0, tau2_0, d0, dmode, err)) return report(err, nullptr);
    for (int64_t i = 0; i < N; ++i)
        if (group[i] < 0 || group[i] >= G) return report(kNbRiBadIdMsg, nullptr);
    Dev d;
    double *dy = d.put(y, N, err), *dX = d.put(tX, (size_t)N * P, err);
    double *dm0 = d.put(m0, P, err), *dP0 = d.put(P0, (size_t)P * P, err);
    int *dg = (int *)d.put_bytes(group, sizeof(int) * (size_t)N, err);
    double *dbeta = d.put(nullptr, (size_t)P * samp, err), *dtau2 = d.put(nullptr, samp, err);
    double *du = u ? d.put(nullptr, (size_t)G * samp, err) : nullptr;
    double *dd = d_out ? d.put(nullptr, samp, err) : nullptr;
    if (!err.empty()) return report(err, nullptr);
    if (nb_ri_gibbs_device(dbeta, du, dtau2, dd, dy, dX, dg, G, dm0, dP0, a0, b0, tau2_0, d0, dmode, N, P, samp, burn,
                           seed, (cudaStream_t)bl_stream_internal(), err))
        return report(err, nullptr);
    cudaError_t e = cudaMemcpy(beta, dbeta, sizeof(double) * (size_t)P * samp, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(tau2, dtau2, sizeof(double) * samp, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && u) e = cudaMemcpy(u, du, sizeof(double) * (size_t)G * samp, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && d_out) e = cudaMemcpy(d_out, dd, sizeof(double) * samp, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return report(cudaGetErrorString(e), nullptr);
    return 0;
}

int bl_nb_ri_gibbs_dev(double *beta, double *u, double *tau2, double *d_out, const double *y, const double *tX,
                       const int *group, int G, const double *m0, const double *P0, double a0, double b0, double tau2_0,
                       double d0, int dmode, int64_t N, int P, int samp, int burn, uint64_t seed, void *stream)
{
    if (bl_ensure_ready_internal()) return 1;
    if (!beta || !tau2 || !y || !tX || !group || !m0 || !P0) return report("nb_ri_gibbs: null argument", nullptr);
    std::string err;
    if (nb_ri_gibbs_device(beta, u, tau2, d_out, y, tX, group, G, m0, P0, a0, b0, tau2_0, d0, dmode, N, P, samp, burn,
                           seed, (cudaStream_t)stream, err))
        return report(err, nullptr);
    return 0;
}

int bl_comm_unique_id(void *out128)
{
    std::string err;
    if (comm_unique_id(out128, err)) return report(err, nullptr);
    return 0;
}

int bl_comm_init(const void *id128, int rank, int world)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    if (comm_init(id128, rank, world, err)) return report(err, nullptr);
    return 0;
}

int bl_comm_init_local(int rank, int world)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    if (comm_init_local(rank, world, err)) return report(err, nullptr);
    return 0;
}

int bl_comm_peer_handle(void *out64)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    if (comm_peer_handle(out64, err)) return report(err, nullptr);
    return 0;
}

int bl_comm_peer_open(const void *handles)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    if (comm_peer_open(handles, err)) return report(err, nullptr);
    return 0;
}

int bl_comm_peer_close(void)
{
    comm_peer_close();
    return 0;
}

int bl_comm_peer_active(void) { return comm_peer_active(); }

int bl_vcomm_create(int world)
{
    if (bl_ensure_ready_internal()) return 1;
    std::string err;
    if (comm_virtual_create(world, err)) return report(err, nullptr);
    return 0;
}

int bl_vcomm_bind(int rank)
{
    std::string err;
    if (comm_virtual_bind(rank, err)) return report(err, nullptr);
    return 0;
}

int bl_vcomm_destroy(void)
{
    comm_virtual_destroy();
    return 0;
}

int bl_comm_destroy(void)
{
    comm_destroy();
    return 0;
}

}  // extern "C"
