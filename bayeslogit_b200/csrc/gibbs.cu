// Gibbs sweeps on the device: binary/binomial logit, multinomial logit, negative
// binomial.  Host drivers + the reference's `gibbs` / `mult_gibbs` C entry points
// (LogitWrapper.cpp:176-234, :316-374) and their bl_* extensions.
//
// One iteration = psi = X beta (k_xbeta, HBM-bound) -> omega = PG(n, psi) (the
// sampler kernels of pg_devroye_kernel.cu / pg_hybrid.cu) -> X' Omega X (+ X'v)
// (k_gram_partial, FP64-pipe-bound; fixed-order reduce) -> [all-reduce of P^2+P
// doubles when observations are sharded across GPUs] -> beta draw (one CTA,
// replicated).  Nothing returns to the host inside the loop.
//
// Stream contract: iteration t draws omega_i from Philox (seed, obs i, call t)
// (mlogit: call t*(J-1)+j) and beta from (seed, obs 2^64-1, same call); i is the
// GLOBAL observation index, so sharding does not change the chain.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <condition_variable>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "engine.h"
#include "gibbs_beta.cuh"
#include "gibbs_kernels.cuh"
#include "gibbs_sweep.h"

namespace bl {

// ------------------------------------------------------------------------------------
// optional NCCL communicator (resolved at run time: no link-time dependency)
// ------------------------------------------------------------------------------------
namespace {

struct Nccl {
    void *lib = nullptr;
    int (*CommInitRank)(void **, int, char[128], int) = nullptr;   // ncclUniqueId by value (128 bytes)
    int (*GetUniqueId)(void *) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
} g_nccl;

struct UniqueId { char bytes[128]; };

bool nccl_load(std::string &err)
{
    if (g_nccl.lib) return true;
    g_nccl.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!g_nccl.lib) { err = std::string("cannot load libnccl.so.2: ") + dlerror(); return false; }
    g_nccl.GetUniqueId = (int (*)(void *))dlsym(g_nccl.lib, "ncclGetUniqueId");
    g_nccl.AllReduce = (int (*)(const void *, void *, size_t, int, int, void *, cudaStream_t))dlsym(g_nccl.lib, "ncclAllReduce");
    g_nccl.CommDestroy = (int (*)(void *))dlsym(g_nccl.lib, "ncclCommDestroy");
    g_nccl.GetErrorString = (const char *(*)(int))dlsym(g_nccl.lib, "ncclGetErrorString");
    void *init = dlsym(g_nccl.lib, "ncclCommInitRank");
    g_nccl.CommInitRank = (int (*)(void **, int, char[128], int))init;
    if (!g_nccl.GetUniqueId || !g_nccl.AllReduce || !init) { err = "libnccl.so.2 lacks expected symbols"; return false; }
    return true;
}

constexpr int kNcclFloat64 = 8, kNcclSum = 0;   // ncclDataType_t / ncclRedOp_t values (nccl.h)
constexpr int kNcclUint64 = 5, kNcclMax = 2;

// ------------------------------------------------------------------------------------
// Peer exchange over NVLink (one node): every rank owns one cudaMalloc'd window that its peers
// map through CUDA IPC.  Window = flags u32 [2 parities][8 ranks] (256 bytes reserved), then
// slots double [2 parities][8 ranks][slot_doubles].  Exchange e (parity e & 1): the Gram reduce
// kernel of rank r STORES its P^2 (+P) sums into slot [parity][r] of every rank's window (posted
// NVLink writes, spread over the reduce kernel's CTAs), fences, and the last CTA stores e into flag
// [parity][r] of every window; the beta-draw kernel of each rank waits on its LOCAL flags and adds
// the slots in rank order, so every rank forms bit-identical sums and the replicated beta draw
// needs no broadcast.  Parity double-buffering is enough: rank A starts exchange e+2 only after
// its beta draw e+1, which waited for every peer's flag e+1, which each peer raised after its own
// beta draw e (the reader of slots e) had completed in stream order.
// ------------------------------------------------------------------------------------
struct Peer {
    void *base = nullptr;                  // this rank's window
    void *win[kMaxPeers] = {};             // every rank's window as mapped here (win[rank] == base)
    unsigned *done = nullptr;              // CTA completion counter of the pushing kernel
    size_t slot_doubles = 0;
    uint32_t epoch = 0;                    // exchanges issued so far (identical on every rank: SPMD)
    bool open = false;
};

// Lock-step rendezvous of the host threads that drive VIRTUAL ranks (see VGroup below).
struct VBarrier {
    std::mutex mu;
    std::condition_variable cv;
    int world = 1, arrived = 0;
    uint64_t generation = 0;
    void wait()
    {
        std::unique_lock<std::mutex> lk(mu);
        const uint64_t g = generation;
        if (++arrived == world) { arrived = 0; ++generation; cv.notify_all(); }
        // a rank that left with an error never arrives: give up after two minutes rather than hang the test
        else if (!cv.wait_for(lk, std::chrono::seconds(120), [&] { return generation != g; })) { arrived = 0; ++generation; cv.notify_all(); }
    }
};

// Communicator state of one rank: the process-wide one (one process per GPU), or one of the virtual
// ranks a test binds its threads to.
struct CommState {
    void *comm = nullptr;          // ncclComm_t
    int rank = 0, world = 1;
    bool local = false;            // no NCCL communicator (bl_comm_init_local): peer windows only
    Peer peer;
    VBarrier *vbar = nullptr;      // virtual ranks only
};

CommState g_cs;
thread_local CommState *t_cs = nullptr;
inline CommState &cs() { return t_cs ? *t_cs : g_cs; }

// Virtual ranks (test aid for boxes with fewer GPUs than ranks): W ranks of one communicator live in ONE
// process on ONE device, each driven by its own host thread (bl_vcomm_bind) and ALL enqueueing into the
// same CUDA stream.  Their windows are plain device allocations of this process.  At every exchange the
// threads meet at a host barrier between enqueueing the producing kernel (slot stores + flags) and the
// consuming kernel (flag wait + rank-ordered sums), so in stream order every producer of an exchange
// precedes every consumer: no kernel ever waits for a kernel behind it, nothing relies on two kernels
// being resident at the same time.  Kernels, descriptors, epochs and parities are those of the real
// multi-GPU exchange.
struct VGroup {
    std::vector<std::unique_ptr<CommState>> ranks;
    VBarrier bar;
};
std::unique_ptr<VGroup> g_vgroup;

inline void exchange_rendezvous() { if (cs().vbar) cs().vbar->wait(); }

constexpr size_t kPeerFlagBytes = 256;
constexpr int kPeerMaxP = 256;

bool peer_active() { return cs().peer.open && cs().world > 1; }

// Descriptors of the next exchange through the windows (advances the epoch: call once per exchange,
// on every rank, in the same order).
void peer_next(PeerPush &px, PeerWait &pw)
{
    const unsigned e = ++cs().peer.epoch;
    const int par = (int)(e & 1u), me = cs().rank;
    px = PeerPush{};
    pw = PeerWait{};
    px.world = pw.world = cs().world;
    px.epoch = pw.epoch = e;
    px.done = cs().peer.done;
    for (int r = 0; r < cs().world; ++r) {
        char *w = (char *)cs().peer.win[r];
        px.flag[r] = (unsigned *)w + par * kMaxPeers + me;
        px.slot[r] = (double *)(w + kPeerFlagBytes) + ((size_t)par * kMaxPeers + me) * cs().peer.slot_doubles;
        pw.slot[r] = (const double *)((char *)cs().peer.base + kPeerFlagBytes) + ((size_t)par * kMaxPeers + r) * cs().peer.slot_doubles;
    }
    pw.flag = (const unsigned *)cs().peer.base + par * kMaxPeers;
}

}  // namespace

// Small all-reduce through the peer windows, two one-CTA kernels per rank.  k_peer_put: store the local
// words into this rank's slot of every window and raise the flags.  k_peer_combine: wait for the world's
// flags, combine the slots in rank order (bit-identical on every rank).  8-byte words; kOp 0: double sum,
// 1: uint64 sum, 2: uint64 max.
__global__ void __launch_bounds__(256)
k_peer_put(const unsigned long long *buf, int cnt, PeerPush px)
{
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
        const unsigned long long v = buf[i];
        for (int r = 0; r < px.world; ++r) reinterpret_cast<unsigned long long *>(px.slot[r])[i] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence_system();
        for (int r = 0; r < px.world; ++r) st_release_sys(px.flag[r], px.epoch);
    }
}

template <int kOp>
__global__ void __launch_bounds__(256)
k_peer_combine(unsigned long long *buf, int cnt, PeerWait pw, int *status)
{
    peer_wait(pw, status);
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
        unsigned long long a = __ldcg(reinterpret_cast<const unsigned long long *>(pw.slot[0]) + i);
        for (int r = 1; r < pw.world; ++r) {
            const unsigned long long b = __ldcg(reinterpret_cast<const unsigned long long *>(pw.slot[r]) + i);
            if (kOp == 0) a = (unsigned long long)__double_as_longlong(__longlong_as_double((long long)a) + __longlong_as_double((long long)b));
            else if (kOp == 1) a += b;
            else a = b > a ? b : a;
        }
        buf[i] = a;
    }
}

namespace {

enum SmallOp { kOpSumF64 = 0, kOpSumU64 = 1, kOpMaxU64 = 2 };

// All-reduce of cnt 8-byte words in place across the ranks (set-up sums, the NB dispersion step): the
// peer windows when they are open, else NCCL.  No-op without a communicator.
int small_allreduce(void *buf, size_t cnt, SmallOp op, int *status, cudaStream_t st, std::string &err)
{
    if (cs().world <= 1) return 0;
    if (peer_active()) {
        if (cnt > cs().peer.slot_doubles) { err = "peer all-reduce: vector longer than a window slot"; return 1; }
        PeerPush px;
        PeerWait pw;
        peer_next(px, pw);
        unsigned long long *b = (unsigned long long *)buf;
        k_peer_put<<<1, 256, 0, st>>>(b, (int)cnt, px);
        exchange_rendezvous();
        if (op == kOpSumF64) k_peer_combine<0><<<1, 256, 0, st>>>(b, (int)cnt, pw, status);
        else if (op == kOpSumU64) k_peer_combine<1><<<1, 256, 0, st>>>(b, (int)cnt, pw, status);
        else k_peer_combine<2><<<1, 256, 0, st>>>(b, (int)cnt, pw, status);
        count_launch(2);
        return 0;
    }
    if (!cs().comm) { err = "sharded sweep: no NCCL communicator and the peer windows are not open"; return 1; }
    const int r = g_nccl.AllReduce(buf, buf, cnt, op == kOpSumF64 ? kNcclFloat64 : kNcclUint64,
                                   op == kOpMaxU64 ? kNcclMax : kNcclSum, cs().comm, st);
    if (r != 0) { err = std::string("ncclAllReduce: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "error"); return 1; }
    return 0;
}

}  // namespace

// ------------------------------------------------------------------------------------
// kernels that need the single-CTA algebra
// ------------------------------------------------------------------------------------

// acc[0..P^2) = Gram sum (no prior), acc[P^2..P^2+P) = optional X'v sum.
// PP = acc + P0; rhs = base_rhs (+ acc tail); then the draw.
// SMEM = true: the workspace is the CTA's shared memory (address space known to the compiler ->
// LDS/STS); false: global scratch for P too large for shared memory.
#ifdef BL_BETA_SLOW
constexpr bool kSlowBeta = true;          // A/B build: the panel factorisation of cta_ldl_upper for every P
#else
constexpr bool kSlowBeta = false;
#endif

// Global scratch of one k_beta_draw<false> CTA: A, B (ld x P each), 5 P of vectors, the constrained draw's P^2 + 2P
// rejection normals.  Batched chains (grid = chains) take one such block each.
__host__ __device__ inline size_t beta_gwork_doubles(int P)
{
    return 2 * (size_t)(P + 1) * P + 5 * (size_t)P + (size_t)P * P + 2 * (size_t)P;
}

// kPlainOnly: the plain / mvn draw with P <= 64 alone (cta_plain_fast) -- a tenth of the code, and registers for two
// CTAs per SM: the batched chains run one CTA per chain.
template <bool SMEM, bool kPlainOnly = false>
__global__ void __launch_bounds__(256, kPlainOnly ? 2 : 1)
k_beta_draw(int mode, const double *__restrict__ acc, const double *__restrict__ P0,
            const double *__restrict__ base_rhs, int add_tail, const double *beta_prev,
            double *beta_out, double *gwork, int P, uint64_t seed, uint32_t call, int *status,
            PeerWait pw, int64_t chain_stride, const double *tn_pre, int tn_fast)
{
    extern __shared__ double sm[];
    // programmatic dependent launch (Sweep::beta_draw; no-ops otherwise): the next kernel's CTAs may be scheduled
    // from now on (they wait for this grid's completion themselves), and this one waits for the sums' producer
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    // batched independent chains: blockIdx.x = chain (own sums, own rhs, own beta, seed + chain; P0 shared)
    acc += (size_t)blockIdx.x * ((size_t)P * P + P);
    if (base_rhs) base_rhs += (size_t)blockIdx.x * P;
    if (beta_prev) beta_prev += blockIdx.x * chain_stride;
    beta_out += blockIdx.x * chain_stride;
    seed += blockIdx.x;
#ifdef BL_BETA_CLOCKS
    long long k0 = clock64();
#endif
    const int ld = P | 1;                     // odd leading dimension: row and column walks both conflict-free
    double *A = SMEM ? sm : gwork + blockIdx.x * beta_gwork_doubles(P);
    double *B = A + (size_t)ld * P;
    double *v = B + (size_t)ld * P;
    double *rhs = v + 4 * P;
    // constrained draw: P^2 + 2P precomputed rejection normals behind the workspace (gibbs_beta.cuh)
    double *nbuf = rhs + P;
    const int nbuf_len = mode == kBetaConstrained ? P * P + 2 * P : 0;
    // plain / mvn draw with P <= 64: the padded layout of cta_plain_fast (its normals live behind the workspace)
    const bool fast = SMEM && !kSlowBeta && mode != kBetaConstrained && P <= 64;
    double *efast = fast ? sm + beta_fast_e_offset(P) : nullptr;
    const bool rev = mode == kBetaMvn;
    if (pw.world > 1) {
        // sharded data: PP and the rhs tail are the rank-ordered sums of the slots the peers pushed
        peer_wait(pw, status);
        switch (pw.world) {
        case 2: peer_stage<2>(pw, A, rhs, P0, base_rhs, add_tail, P, ld); break;
        case 4: peer_stage<4>(pw, A, rhs, P0, base_rhs, add_tail, P, ld); break;
        case 8: peer_stage<8>(pw, A, rhs, P0, base_rhs, add_tail, P, ld); break;
        default: peer_stage<0>(pw, A, rhs, P0, base_rhs, add_tail, P, ld); break;
        }
        __syncthreads();
        cta_beta_draw<kPlainOnly>(mode, A, B, v, rhs, beta_prev, beta_out, P, ld, seed, call, status, nbuf, nbuf_len, efast, tn_pre, SMEM ? tn_fast : 0);
        return;
    }
    if (fast) {
        // straight into the padded layout: element (i = tid & 63, column (tid >> 6) + 4 u), every load issued
        // before the first is consumed; the mvn draw reads the index-reversed system
        const BetaFast w(sm, P);
        const int i = threadIdx.x & 63, cb = threadIdx.x >> 6;
        double g[16], q[16];
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            const int c = cb + 4 * u;
            const bool in = i < P && c < P;
            const int k = rev ? (P - 1 - i) + P * (P - 1 - c) : i + P * c;
            g[u] = in ? __ldcg(acc + k) : (i == c ? 1.0 : 0.0);
            q[u] = (in && P0) ? __ldg(P0 + k) : 0.0;
        }
        double rr = 0.0;
        if ((int)threadIdx.x < P) {
            const int k = rev ? P - 1 - (int)threadIdx.x : (int)threadIdx.x;
            rr = (base_rhs ? base_rhs[k] : 0.0) + (add_tail ? __ldcg(acc + (size_t)P * P + k) : 0.0);
        }
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            const int c = cb + 4 * u;
            if (i < w.Pp && c < w.Pp) w.F[i + w.LD * c] = g[u] + q[u];
        }
        if ((int)threadIdx.x < w.Pp) w.F[threadIdx.x + w.LD * w.Pp] = rr;
        if (threadIdx.x < 56) w.Sn[(threadIdx.x / 7) * kFastLdS + w.Pp + 1 + threadIdx.x % 7] = 0.0;
        __shared__ int ok_fast;
        if (threadIdx.x == 0) ok_fast = 1;
        __syncthreads();
#ifdef BL_BETA_CLOCKS
        if (threadIdx.x == 0 && call == 3) printf("[beta clocks] load %lld\n", clock64() - k0);
#endif
        cta_plain_fast(sm, efast, beta_out, P, rev, &ok_fast, seed, call);
        if (!ok_fast && threadIdx.x == 0) *status = 1;
        return;
    }
    if (kPlainOnly) return;                   // (the host picks this instantiation only when `fast` holds)
    // stage PP = Gram + P0.  P <= 64: every load of the thread (16 Gram entries, 16 prior entries) is issued before
    // the first use -- one L2 round trip instead of four.
    if (P <= 64) {
        double g[16], q[16];
        const int PP2 = P * P;
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            const int k = threadIdx.x + 256 * u;
            g[u] = k < PP2 ? __ldcg(acc + k) : 0.0;
            q[u] = (k < PP2 && P0) ? __ldg(P0 + k) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            const int k = threadIdx.x + 256 * u;
            if (k < PP2) A[k % P + (size_t)ld * (k / P)] = g[u] + q[u];
        }
    }
    if (P > 64)
        for (int k = threadIdx.x; k < P * P; k += blockDim.x)
            A[k % P + (size_t)ld * (k / P)] = acc[k] + (P0 ? P0[k] : 0.0);
    for (int k = threadIdx.x; k < P; k += blockDim.x)
        rhs[k] = (base_rhs ? base_rhs[k] : 0.0) + (add_tail ? acc[(size_t)P * P + k] : 0.0);
    __syncthreads();
#ifdef BL_BETA_CLOCKS
    if (threadIdx.x == 0 && call == 3) printf("[beta clocks] load %lld\n", clock64() - k0);
#endif
    cta_beta_draw(mode, A, B, v, rhs, beta_prev, beta_out, P, ld, seed, call, status, nbuf, nbuf_len, nullptr, tn_pre, SMEM ? tn_fast : 0);
}

// rejection normals of one constrained beta draw: normal m of the stream (seed, obs 2^64-3, call), gibbs_beta.cuh
__global__ void k_tn_normals(double *out, int n, uint64_t seed, uint32_t call)
{
    BL_PDL_ENTER();
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m < n) out[m] = stream_normal_obs(seed, kTnObs, call, m);
}

__global__ void k_matvec(double *out, const double *A, const double *x, int P)   // out = A x, col-major
{
    int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= P) return;
    double s = 0.0;
    for (int b = 0; b < P; ++b) s = fma(A[a + (size_t)P * b], x[b], s);
    out[a] = s;
}

namespace {

#define GB_CK(expr)                                                                  \
    do {                                                                             \
        cudaError_t e_ = (expr);                                                     \
        if (e_ != cudaSuccess) { err = std::string(#expr) + ": " + cudaGetErrorString(e_); return 1; } \
    } while (0)

// Stream-ordered scratch (cudaMallocAsync pool): no device-wide synchronisation per chain.
struct DevMem {
    std::vector<void *> ptrs;
    cudaStream_t st = nullptr;
    ~DevMem() { for (void *p : ptrs) cudaFreeAsync(p, st); }
    template <class T>
    cudaError_t get(T **p, size_t count)
    {
        void *q = nullptr;
        cudaError_t e = cudaMallocAsync(&q, (count ? count : 1) * sizeof(T), st);
        if (e == cudaSuccess) { ptrs.push_back(q); *p = (T *)q; }
        return e;
    }
};

inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// part[chain][slab][P] = per-slab sums of X'(c0 v0 + c1 v1 v2): streaming kernel for power-of-two P,
// tensor-core kernel for other even P, scalar kernel otherwise.  Chain c (grid.y) reads its rows at
// tX + c x_stride and its weights at + c N.
void launch_xtv(dim3 grid, cudaStream_t st, double *part, const double *tX, int64_t x_stride, const double *v0, double c0,
                const double *v1, const double *v2, double c1, int64_t N, int P, const double *c1_dev)
{
    const size_t smem = 8 * P * sizeof(double);
    // the streaming kernel indexes a slab's column pairs with 32 bits
    const int64_t slab_pairs = ((N + grid.x - 1) / grid.x) * (P / 2);
    const int l2 = slab_pairs < (1LL << 31) - 4096 ? xtv_stream_log2l(tX, P) : 0;
    const int mode = (v0 && !v1 && !v2) ? 0 : (!v0 && v1 && v2) ? 1 : (v0 && v1 && !v2) ? 2 : -1;
#define BL_XTV(L2, M) launch_pdl(k_xtv_stream<L2, M>, dim3(grid), dim3(256), smem, st, part, tX, x_stride, v0, c0, v1, v2, c1, N, c1_dev)
#define BL_XTV_L(L2) (mode == 0 ? BL_XTV(L2, 0) : mode == 1 ? BL_XTV(L2, 1) : BL_XTV(L2, 2))
    if (mode >= 0 && l2 == 2) BL_XTV_L(2);
    else if (mode >= 0 && l2 == 3) BL_XTV_L(3);
    else if (mode >= 0 && l2 == 4) BL_XTV_L(4);
    else if (mode >= 0 && l2 == 5) BL_XTV_L(5);
    else if (mode >= 0 && l2 == 6) BL_XTV_L(6);
    else if (mode >= 0 && l2 == 7) BL_XTV_L(7);
#undef BL_XTV_L
#undef BL_XTV
    else if (xbeta_mma_ok(tX, P)) launch_pdl(k_xtv_mma, dim3(grid), dim3(256), smem, st, part, tX, x_stride, v0, c0, v1, v2, c1, N, P, c1_dev);
    else launch_pdl(k_xtv_partial, dim3(grid), dim3(256), smem, st, part, tX, x_stride, v0, c0, v1, v2, c1, N, P, c1_dev);
}

// BL_GIBBS_TIMING=1: CUDA-event stage times of one iteration (the one armed by the driver), to stderr.
struct StageTimer {
    bool enabled = getenv("BL_GIBBS_TIMING") != nullptr, armed = false;
    cudaStream_t st = nullptr;
    std::vector<std::pair<const char *, cudaEvent_t>> marks;
    void arm(bool on) { armed = enabled && on; if (armed) mark("start"); }
    void mark(const char *name)
    {
        if (!armed) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, st);
        marks.emplace_back(name, e);
    }
    void report(const char *tag)
    {
        if (!armed || marks.size() < 2) return;
        cudaEventSynchronize(marks.back().second);
        fprintf(stderr, "[bl %s timing, us]", tag);
        for (size_t k = 1; k < marks.size(); ++k) {
            float ms = 0;
            cudaEventElapsedTime(&ms, marks[k - 1].second, marks[k].second);
            fprintf(stderr, " %s %.1f", marks[k].first, ms * 1e3);
        }
        fprintf(stderr, "\n");
        for (auto &m : marks) cudaEventDestroy(m.second);
        marks.clear();
        armed = false;
    }
};

// Gram and X'v slab partition of N rows: one wave of 2 CTAs per SM (Sweep::init; the multinomial multichain
// driver takes the single chain's partition so that every chain sums its rows in the single chain's order).
struct Slabs {
    int nt = 1, nslab = 1, nslab_diag = 0, xtv_slabs = 1;
};

Slabs slab_partition(int64_t N, int P)
{
    Slabs g;
    g.nt = cdiv(P, kGramTile);
    const int tiles = g.nt * (g.nt + 1) / 2;
    g.nslab = (int)std::min<int64_t>(std::max<int64_t>(1, 148 * 2 / tiles), std::max<int64_t>(1, N / (4 * kGramRows)));   // 2 CTAs/SM resident: one wave
    if (g.nslab < 1) g.nslab = 1;
    if (g.nt > 1) {
        // one wave of 2 CTAs per SM, slabs in proportion to the tile's cost (diagonal 36, off-diagonal 64
        // MMA tiles per k-step): P = 256 -> 4 x 20 + 6 x 35 CTAs instead of 10 x 29 of unequal length
        const int nd = g.nt, no = g.nt * (g.nt - 1) / 2, total = nd * 36 + no * 64;
        const int64_t cap = std::max<int64_t>(1, N / (4 * kGramRows));
        g.nslab = (int)std::min<int64_t>(std::max(1, 148 * 2 * 64 / total), cap);
        g.nslab_diag = (int)std::min<int64_t>(std::max(1, 148 * 2 * 36 / total), cap);
        if (g.nslab_diag > g.nslab) g.nslab_diag = g.nslab;
    }
    g.xtv_slabs = (int)std::min<int64_t>(148 * 2, std::max<int64_t>(1, N / 64));
    return g;
}

// The single chain's beta draw workspace: `plain` bytes of shared memory for the plain / mvn draw, `tn` with the
// constrained draw's rejection normals; above 200 KB of `tn` every draw runs out of global scratch (k_beta_draw<false>).
struct BetaSmem {
    size_t plain = 0, tn = 0;
    bool use_smem = true;
};

BetaSmem beta_smem_of(int P)
{
    BetaSmem b;
    // A, B (ld x P each), 5 P vector scratch; the constrained draw's P^2 + 2P rejection normals behind them
    b.plain = (2 * (size_t)(P | 1) * P + 5 * (size_t)P) * sizeof(double);
    if (P <= 64) b.plain = (beta_fast_e_offset(P) + 64) * sizeof(double);      // cta_plain_fast: + its normals
    b.tn = std::max(b.plain + ((size_t)P * P + 2 * (size_t)P) * sizeof(double), beta_tn_doubles(P) * sizeof(double));
    b.use_smem = b.tn <= 200 * 1024;
    return b;
}

// Shared machinery of the three sweeps.
struct Sweep {
    int64_t N = 0;          // local observations
    int P = 0;
    uint64_t obs0 = 0;      // global index of local observation 0
    cudaStream_t st = nullptr;
    const double *tX = nullptr;
    double *psi = nullptr, *w = nullptr, *acc = nullptr, *part = nullptr, *xtv_part = nullptr;
    double *gwork = nullptr;
    double *tnbuf = nullptr;   // the constrained draw's rejection normals of one iteration, made by k_tn_normals
    int *status = nullptr;
    int nt = 1, nslab = 1, nslab_diag = 0, xtv_slabs = 1;
    bool use_smem = true;
    size_t beta_smem = 0, beta_smem_tn = 0;   // workspace of the beta draw; the constrained draw adds its rejection normals
    bool exchange = false;  // sharded sweep: the Gram (+ tail) sums are exchanged between ranks before the beta draw
    PeerWait pending{};     // set by gram() when it pushed to the peers; consumed by beta_draw()

    int init(DevMem &m, std::string &err)
    {
        // the beta draws keep a vector in registers, 8 entries per lane of one warp (gibbs_beta.cuh)
        if (P > 256) { err = "P > 256 covariates is not supported by the single-CTA beta draw"; return 1; }
        const Slabs g = slab_partition(N, P);
        nt = g.nt; nslab = g.nslab; nslab_diag = g.nslab_diag; xtv_slabs = g.xtv_slabs;
        int tiles = nt * (nt + 1) / 2;
        GB_CK(m.get(&psi, N));
        GB_CK(m.get(&w, N));
        GB_CK(m.get(&acc, (size_t)P * P + P));
        GB_CK(m.get(&part, (size_t)tiles * nslab * 2 * kGramTile * kGramTile));
        GB_CK(m.get(&xtv_part, (size_t)xtv_slabs * P));
        GB_CK(m.get(&gwork, beta_gwork_doubles(P)));
        GB_CK(m.get(&status, 1));
        GB_CK(cudaMemsetAsync(status, 0, sizeof(int), st));
        GB_CK(cudaMemsetAsync(acc, 0, ((size_t)P * P + P) * sizeof(double), st));
        const BetaSmem bs = beta_smem_of(P);
        beta_smem = bs.plain;
        beta_smem_tn = bs.tn;
        GB_CK(m.get(&tnbuf, (size_t)P * P + 2 * (size_t)P));
        GB_CK(cudaFuncSetAttribute(k_gram_partial<kGramRows, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)gram_smem_bytes(true)));
        GB_CK(cudaFuncSetAttribute(k_gram_partial<kGramRowsDiag, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)gram_smem_bytes(false)));
        GB_CK(cudaFuncSetAttribute(k_gram_partial<kGramRowsDiag, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)gram_smem_bytes(false, true)));
        use_smem = bs.use_smem;
        if (use_smem && beta_smem_tn > 48 * 1024)
            GB_CK(cudaFuncSetAttribute(k_beta_draw<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)beta_smem_tn));
        if (use_smem && beta_smem > 48 * 1024)
            GB_CK(cudaFuncSetAttribute(k_beta_draw<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)beta_smem));
        return 0;
    }

    void xbeta(double *out, const double *beta, const double *off, double off_scale, double shift = 0.0)
    {
        int grid = (int)std::min<int64_t>(148 * 8, std::max<int64_t>(1, (N + 255) / 256));
        if (xbeta_mma_ok(tX, P))
            launch_pdl(k_xbeta_mma<false>, dim3(grid), dim3(256), 0, st, out, N, tX, N * P, beta, 0, 1, N, P, off, off_scale, shift, MlogitNext{});
        else
            k_xbeta<<<grid, 256, P * sizeof(double), st>>>(out, tX, beta, off, off_scale, shift, N, P);
        count_launch();
    }

    // mlogit: XB_j = X beta_j, E_j = exp(XB_j) and the next category's offset and tilt in one pass (k_xbeta_mma<true>)
    void xbeta_mlogit(double *out, const double *beta, const MlogitNext &mn)
    {
        int grid = (int)std::min<int64_t>(148 * 8, std::max<int64_t>(1, (N + 255) / 256));
        launch_pdl(k_xbeta_mma<true>, dim3(grid), dim3(256), 0, st, out, N, tX, N * P, beta, 0, 1, N, P, nullptr, 0.0, 0.0, mn);
        count_launch();
    }

    // acc[0..P^2) <- sum_i w_i x_i x_i'  (local shard).  Sharded sweeps with the peer windows open:
    // the reduce kernel stores the sums (and, with_tail, the P sums xtv() left in acc[P^2..]) into
    // every rank's window instead, and beta_draw() picks them up there -- call xtv() before gram().
    // cvec (packed kernel, P == 32, only): the X'v tail acc[P^2 ..) = X' (wv o cvec) comes out of the same pass
    // (gram_tail_fused() says whether that is possible); otherwise call xtv() first.
    bool gram_tail_fused() const { return gram_packed(P) && nt == 1; }
    void gram(const double *wv, bool with_tail = false, const double *cvec = nullptr)
    {
        int tiles = nt * (nt + 1) / 2;
        const bool packed = gram_packed(P);
        if (nt > 1)
            launch_pdl(k_gram_partial<kGramRows, false>, dim3(nslab, tiles), dim3(256), gram_smem_bytes(true), st, part, tX, N * P, wv, N, P, nt, nslab_diag, nullptr);
        else if (packed)
            launch_pdl(k_gram_partial<kGramRowsDiag, true, true>, dim3(nslab, tiles), dim3(256), gram_smem_bytes(false, true), st, part, tX, N * P, wv, N, P, nt, 0, cvec);
        else
            launch_pdl(k_gram_partial<kGramRowsDiag, true>, dim3(nslab, tiles), dim3(256), gram_smem_bytes(false), st, part, tX, N * P, wv, N, P, nt, 0, nullptr);
        const int tail_in_part = packed && cvec ? 1 : 0;
        PeerPush px{};
        pending = PeerWait{};
        if (exchange && peer_active()) {
            peer_next(px, pending);
            px.with_tail = with_tail ? 1 : 0;
        }
        launch_pdl(k_gram_reduce, dim3(cdiv((int64_t)P * P + (tail_in_part ? P : 0), 32)), dim3(256), 0, st, acc, nullptr, part, P, nt,
                   nt > 1 ? 2 * nslab : nslab, px, packed ? 1 : 0, 2 * nslab_diag, tail_in_part);
        count_launch(2);
        if (px.world > 1) exchange_rendezvous();     // virtual ranks: every producer is enqueued before any consumer
    }

    // acc[P^2..P^2+P) <- X'(c0 v0 + c1 v1 v2)
    void xtv(const double *v0, double c0, const double *v1, const double *v2, double c1,
             const double *c1_dev = nullptr)
    {
        launch_xtv(dim3(xtv_slabs), st, xtv_part, tX, N * P, v0, c0, v1, v2, c1, N, P, c1_dev);
        launch_pdl(k_xtv_reduce, dim3(cdiv(P, 128)), dim3(128), 0, st, acc + (size_t)P * P, nullptr, nullptr, xtv_part, P, xtv_slabs,
                   (int64_t)P);
        count_launch(2);
    }

    int allreduce(bool with_tail, std::string &err)
    {
        if (!exchange || cs().world <= 1) return 0;
        if (pending.world > 1) return 0;          // already pushed through the peer windows by gram()
        if (!cs().comm) { err = "sharded sweep: no NCCL communicator and the peer windows are not open"; return 1; }
        size_t cnt = (size_t)P * P + (with_tail ? P : 0);
        int r = g_nccl.AllReduce(acc, acc, cnt, kNcclFloat64, kNcclSum, cs().comm, st);
        if (r != 0) { err = std::string("ncclAllReduce: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "error"); return 1; }
        return 0;
    }

    void beta_draw(int mode, const double *P0, const double *base_rhs, bool add_tail,
                   const double *beta_prev, double *beta_out, uint64_t seed, uint32_t call)
    {
        if (use_smem) {
            const bool tn = mode == kBetaConstrained && tnbuf != nullptr;
            if (tn) {
                // the draw's P^2 + 2P rejection normals depend on (seed, call) alone: one thread each, a few
                // microseconds on the whole chip, instead of 17 in a row on each of the draw's 256 threads
                const int n = P * P + 2 * P;
                launch_pdl(k_tn_normals, dim3(cdiv(n, 128)), dim3(128), 0, st, tnbuf, n, seed, call);
                count_launch();
            }
            // programmatic dependent launch: the CTA is scheduled while the kernel that produces the sums drains and
            // waits for its completion on the device (griddepcontrol.wait at the top of k_beta_draw) -- the launch
            // latency of the one kernel that sits between two sweeps leaves the critical path
            static const bool pdl = getenv("BL_GIBBS_NO_PDL") == nullptr;
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(1); cfg.blockDim = dim3(256);
            cfg.dynamicSmemBytes = mode == kBetaConstrained ? beta_smem_tn : beta_smem;
            cfg.stream = st;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            at[0].val.programmaticStreamSerializationAllowed = 1;
            cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
            const bool lean = mode != kBetaConstrained && P <= 64 && !kSlowBeta;
            cudaLaunchKernelEx(&cfg, lean ? k_beta_draw<true, true> : k_beta_draw<true, false>, mode, (const double *)acc, P0,
                               base_rhs, add_tail ? 1 : 0, beta_prev,
                               beta_out, gwork, P, seed, call, status, pending, (int64_t)0,
                               (const double *)(tn ? tnbuf : nullptr), getenv("BL_BETA_NO_SPEC") ? 3 : 1);
        } else
            k_beta_draw<false><<<1, 256, 0, st>>>(mode, acc, P0, base_rhs, add_tail ? 1 : 0, beta_prev,
                                                  beta_out, gwork, P, seed, call, status, pending, 0, nullptr, 0);
        pending = PeerWait{};
        count_launch();
    }

    int check_status(std::string &err, const char *what)
    {
        int h = 0;
        GB_CK(cudaMemcpyAsync(&h, status, sizeof(int), cudaMemcpyDeviceToHost, st));
        GB_CK(cudaStreamSynchronize(st));
        if (h == 2) { err = std::string(what) + ": peer exchange timed out (a rank did not arrive)"; return 1; }
        if (h == 3) { err = std::string(what) + ": inverse of the posterior precision is not positive definite (constrained beta draw)"; return 1; }
        if (h != 0) { err = std::string(what) + ": posterior precision is not positive definite"; return 1; }
        return 0;
    }
};

}  // namespace

// ------------------------------------------------------------------------------------
// Binary / binomial logit (Logit::gibbs, Logit.hpp:460-481 with gibbs_block :402-457)
// ------------------------------------------------------------------------------------
// All pointers are DEVICE pointers.  y, n: local shard [N]; tX: P x N local shard;
// w_out: N x samp or null (flags & BL_GIBBS_NO_W); beta_out: P x samp.
int logit_gibbs_device(double *w_out, double *beta_out, const double *y, const double *tX,
                       const double *n, const double *m0, const double *P0, int64_t N, int P,
                       int samp, int burn, uint64_t seed, int flags, uint64_t obs0, bool sharded,
                       cudaStream_t st, std::string &err, int w_every)
{
    if (N <= 0 || P <= 0 || samp <= 0 || burn < 0 || w_every < 1) { err = "gibbs: bad dimensions"; return 1; }
    DevMem mem;
    mem.st = st;
    Sweep s;
    s.N = N; s.P = P; s.obs0 = obs0; s.st = st; s.tX = tX; s.exchange = sharded;
    if (s.init(mem, err)) return 1;
    double *kappa, *b0, *bP;
    int *shape;
    GB_CK(mem.get(&kappa, N));
    GB_CK(mem.get(&shape, N));
    GB_CK(mem.get(&b0, P));
    GB_CK(mem.get(&bP, P));
    const bool keep_w = !(flags & BL_GIBBS_NO_W) && w_out;
    const int mode = (flags & BL_GIBBS_PLAIN_BETA) ? kBetaPlain : kBetaConstrained;
    // psi = X beta and the omega draw as one pass over X (k_logit_psi_draw) unless asked otherwise
    const bool fused = !(flags & BL_GIBBS_UNFUSED) && logit_psi_draw_ok(tX, P);
    // ... or, for even P <= 64, psi, omega and the Gram from ONE TMA-staged read of X (k_logit_sweep, gibbs_sweep.cu):
    // exactly N P 8 bytes of HBM traffic and two launches per iteration.  Its rate is set by the latency of the draw
    // warps that fit beside the Gram warps, so on long shards the two-pass path is as fast or a little faster
    // (N = 1M: 378 us against 372; 500k rows per GPU: 219 against 216), while on short ones the launches and the
    // separate reduce it saves dominate (125k rows per GPU, 8 GPUs: 84 us against 106): default up to 2^18 local rows.
    // BL_GIBBS_ONE_PASS / BL_GIBBS_TWO_PASS force either.
    const bool one_pass = !(flags & (BL_GIBBS_UNFUSED | BL_GIBBS_TWO_PASS)) && logit_sweep_ok(tX, P) &&
                          ((flags & BL_GIBBS_ONE_PASS) || N <= (1 << 18));
    LogitSweep k3;
    if (one_pass && k3.init(tX, N, P, st, err)) return 1;

    // set_prior / set_bP: b0 = P0 m0, bP = b0 + X'(n (y - 1/2))   (Logit.hpp:174-190)
    k_kappa<<<cdiv(N, 256), 256, 0, st>>>(kappa, y, n, 0.0, N);
    k_shape_int<<<cdiv(N, 256), 256, 0, st>>>(shape, n, N);
    k_matvec<<<cdiv(P, 128), 128, 0, st>>>(b0, P0, m0, P);
    count_launch(3);
    s.xtv(kappa, 1.0, nullptr, nullptr, 0.0);
    if (sharded && small_allreduce(s.acc + (size_t)P * P, (size_t)P, kOpSumF64, s.status, st, err)) return 1;
    k_xtv_reduce<<<cdiv(P, 128), 128, 0, st>>>(bP, b0, s.acc + (size_t)P * P, s.xtv_part, P, 0, P);
    count_launch();

    GB_CK(cudaMemsetAsync(beta_out, 0, sizeof(double) * (size_t)P * samp, st));
    if (keep_w) GB_CK(cudaMemsetAsync(w_out, 0, sizeof(double) * (size_t)N * ((samp + w_every - 1) / w_every), st));
    const bool timing = getenv("BL_GIBBS_TIMING") != nullptr;
    cudaEvent_t ev[6];
    if (timing) for (auto &x : ev) cudaEventCreate(&x);
    uint32_t t = 0;
    for (int phase = 0; phase < 2; ++phase) {
        int iters = phase == 0 ? burn : samp;
        double *bcur = beta_out, *bprev = beta_out;
        const double *bpsi = bcur;                                    // the beta the next omega draw conditions on
        if (!fused && !one_pass) s.xbeta(s.psi, bcur, nullptr, 0.0);
        for (int m = 1; m <= iters; ++m, ++t) {
            const bool tm = timing && phase == 1 && m == iters;       // BL_GIBBS_TIMING=1: stage times
            // omega of sampling iteration m goes to slot m - 1 (Logit.hpp:402-457; burn-in overwrites slot 0); with
            // thinning only every w_every-th iteration is kept, in slot (m - 1) / w_every, the others stay in scratch
            double *wcur = !keep_w ? s.w : phase == 0 ? w_out
                           : ((m - 1) % w_every == 0 ? w_out + (size_t)N * ((m - 1) / w_every) : s.w);
            if (tm) cudaEventRecord(ev[0], st);
            if (one_pass) {
                PeerPush px{};
                s.pending = PeerWait{};
                if (s.exchange && peer_active()) peer_next(px, s.pending);
                cudaError_t e = k3.launch(wcur, s.acc, shape, bpsi, StreamId{seed, obs0, t}, px);
                if (e != cudaSuccess) { err = std::string("k_logit_sweep: ") + cudaGetErrorString(e); return 1; }
                if (px.world > 1) exchange_rendezvous();
                if (tm) cudaEventRecord(ev[1], st);
            } else {
                cudaError_t e = fused
                    ? launch_logit_psi_draw(wcur, nullptr, shape, tX, bpsi, 0, 1, N, P, StreamId{seed, obs0, t}, st)
                    : launch_devroye_refill(wcur, shape, s.psi, N, StreamId{seed, obs0, t}, st);
                if (e != cudaSuccess) { err = cudaGetErrorString(e); return 1; }
                if (tm) cudaEventRecord(ev[1], st);
                s.gram(wcur);
            }
            if (tm) cudaEventRecord(ev[2], st);
            if (s.allreduce(false, err)) return 1;
            if (tm) cudaEventRecord(ev[3], st);
            s.beta_draw(mode, P0, bP, false, bprev, bcur, seed, t);
            if (tm) cudaEventRecord(ev[4], st);
            bpsi = bcur;
            if (!fused && !one_pass) s.xbeta(s.psi, bcur, nullptr, 0.0);
            if (tm) {
                cudaEventRecord(ev[5], st);
                cudaEventSynchronize(ev[5]);
                float d[5];
                for (int k = 0; k < 5; ++k) cudaEventElapsedTime(&d[k], ev[k], ev[k + 1]);
                fprintf(stderr, "[bl gibbs timing, us] %s %.1f gram %.1f allreduce %.1f beta %.1f xbeta %.1f\n",
                        one_pass ? "psi+draw+gram (one pass)" : fused ? "psi+draw" : "draw", d[0] * 1e3, d[1] * 1e3, d[2] * 1e3, d[3] * 1e3, d[4] * 1e3);
                for (auto &x : ev) cudaEventDestroy(x);
            }
            if (phase == 1) {
                bprev = bcur;
                if (m < iters) bcur += P;
            }
        }
    }
    GB_CK(cudaGetLastError());
    return s.check_status(err, "gibbs");
}

// ------------------------------------------------------------------------------------
// A batch of independent binary / binomial logit chains (BASELINE config 5: 4096 chains of
// N = 10k, P = 32; SURVEY.md section 8e "independent chains").  Chain c owns rows [c N, (c+1) N)
// of tX / y / n, shares the prior, and is exactly the chain logit_gibbs_device runs on its rows
// with seed + c (same streams, same slot semantics); every kernel of the sweep is launched once
// for the whole batch with the chain as a grid dimension, so the one-CTA beta draws of the chains
// run side by side instead of sitting on each chain's critical path.  omega is not returned.
// shared_rows (bl_logit_multichain): every chain runs on the same N rows of tX / y / n -- the usual
// several chains from different seeds on one data set.  X is held and read once: kappa, the shapes and
// X' kappa are formed once, psi + omega of all chains come from one pass over X (k_logit_psi_draw_shared),
// the Gram kernels read X with a chain stride of 0.  Chain c is bit for bit the chain of the replicated
// call (chains copies of the rows, same seed).
// beta_out: [chains][samp][P].
// ------------------------------------------------------------------------------------
int logit_chains_device(double *beta_out, const double *y, const double *tX, const double *n,
                        const double *m0, const double *P0, int chains, int64_t N, int P, int samp, int burn,
                        uint64_t seed, int flags, bool shared_rows, cudaStream_t st, std::string &err)
{
    const char *who = shared_rows ? "logit_multichain" : "logit_chains";
    if (chains <= 0 || N <= 0 || P <= 0 || samp <= 0 || burn < 0) { err = std::string(who) + ": bad dimensions"; return 1; }
    const int64_t T = (int64_t)chains * N;
    if (T >= (1LL << 31)) { err = std::string(who) + ": chains * N must stay below 2^31 observations per call"; return 1; }
    if (P > 256) { err = "P > 256 covariates is not supported by the single-CTA beta draw"; return 1; }
    const int mode = (flags & BL_GIBBS_PLAIN_BETA) ? kBetaPlain : kBetaConstrained;
    const size_t beta_smem = mode == kBetaConstrained
        ? beta_tn_doubles(P) * sizeof(double)
        : std::max((2 * (size_t)(P | 1) * P + 5 * (size_t)P) * sizeof(double),
                   P <= 64 ? (beta_fast_e_offset(P) + 64) * sizeof(double) : (size_t)0);
    if (beta_smem > 200 * 1024) { err = std::string(who) + ": P too large for the shared-memory beta draw"; return 1; }
    DevMem mem;
    mem.st = st;
    const int nt = cdiv(P, kGramTile), tiles = nt * (nt + 1) / 2;
    int nslab = (int)std::min<int64_t>(std::max<int64_t>(1, cdiv(148 * 2, (int64_t)tiles * chains)),
                                       std::max<int64_t>(1, N / (4 * kGramRows)));
    const int slabs_total = nt > 1 ? 2 * nslab : nslab;
    const size_t accn = (size_t)P * P + P;
    const bool fused = !(flags & BL_GIBBS_UNFUSED) && logit_psi_draw_ok(tX, P);
    const int xchains = shared_rows ? 1 : chains;          // copies of the rows held
    const int64_t R = xchains * N;
    const int64_t x_stride = shared_rows ? 0 : N * P;      // chain c's rows: tX + c x_stride
    // the fused shared-rows kernel reads the N shapes of the shared rows; the refill kernel (unfused) walks all
    // chains * N (row, chain) pairs and reads one shape per pair
    const int64_t nshape = shared_rows && fused ? N : T;
    double *psi, *w, *kappa, *acc, *part, *xtv_part, *b0, *bP;
    int *shape, *status;
    void *work;
    GB_CK(mem.get(&psi, T));
    GB_CK(mem.get(&w, T));
    GB_CK(mem.get(&kappa, R));
    GB_CK(mem.get(&shape, nshape));
    GB_CK(mem.get(&acc, accn * chains));
    GB_CK(mem.get(&part, (size_t)chains * tiles * slabs_total * kGramTile * kGramTile));
    GB_CK(mem.get(&xtv_part, (size_t)xchains * P));
    GB_CK(mem.get(&b0, P));
    GB_CK(mem.get(&bP, (size_t)chains * P));
    GB_CK(mem.get(&status, 1));
    GB_CK(mem.get((char **)&work, (32 + (size_t)T) * sizeof(int)));      // branch-class binning of the draw: [meta][index list]
    GB_CK(cudaMemsetAsync(status, 0, sizeof(int), st));
    GB_CK(cudaFuncSetAttribute(k_gram_partial<kGramRows, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)gram_smem_bytes(true)));
    GB_CK(cudaFuncSetAttribute(k_gram_partial<kGramRowsDiag, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)gram_smem_bytes(false)));
    GB_CK(cudaFuncSetAttribute(k_gram_partial<kGramRowsDiag, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)gram_smem_bytes(false, true)));
    const bool packed = gram_packed(P);
    if (beta_smem > 48 * 1024) {
        GB_CK(cudaFuncSetAttribute(k_beta_draw<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)beta_smem));
        GB_CK(cudaFuncSetAttribute(k_beta_draw<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)beta_smem));
    }
    const int64_t bstride = (int64_t)P * samp;

    // bP_c = P0 m0 + X_c'(n (y - 1/2)); with shared rows the same for every chain: formed once, then copied
    k_kappa<<<cdiv(R, 256), 256, 0, st>>>(kappa, y, n, 0.0, R);
    k_shape_int<<<cdiv(R, 256), 256, 0, st>>>(shape, n, R);
    k_matvec<<<cdiv(P, 128), 128, 0, st>>>(b0, P0, m0, P);
    launch_xtv(dim3(1, xchains), st, xtv_part, tX, N * P, kappa, 1.0, nullptr, nullptr, 0.0, N, P, nullptr);
    k_xtv_reduce<<<dim3(cdiv(P, 128), xchains), 128, 0, st>>>(bP, b0, nullptr, xtv_part, P, 1, P);
    count_launch(5);
    for (int c = xchains; c < chains; ++c)
        GB_CK(cudaMemcpyAsync(bP + (size_t)c * P, bP, sizeof(double) * P, cudaMemcpyDeviceToDevice, st));
    for (int64_t c = R; c < nshape; c += N)
        GB_CK(cudaMemcpyAsync(shape + c, shape, sizeof(int) * N, cudaMemcpyDeviceToDevice, st));
    GB_CK(cudaMemsetAsync(beta_out, 0, sizeof(double) * (size_t)bstride * chains, st));

    auto xbeta = [&](const double *beta) {
        const int64_t trips = (int64_t)chains * ((N + 31) / 32);
        int grid = (int)std::min<int64_t>(148 * 8, std::max<int64_t>(1, (trips + 7) / 8));
        if (xbeta_mma_ok(tX, P))
            k_xbeta_mma<false><<<grid, 256, 0, st>>>(psi, N, tX, x_stride, beta, bstride, chains, N, P, nullptr, 0.0, 0.0, MlogitNext{});
        else
            k_xbeta_chains<<<grid, 256, 0, st>>>(psi, N, tX, x_stride, beta, bstride, chains, (int)N, P);
        count_launch();
    };
    const bool timing = getenv("BL_GIBBS_TIMING") != nullptr;
    cudaEvent_t ev[6];
    if (timing) for (auto &x : ev) cudaEventCreate(&x);
    uint32_t t = 0;
    for (int phase = 0; phase < 2; ++phase) {
        int iters = phase == 0 ? burn : samp;
        double *bcur = beta_out, *bprev = beta_out;
        const double *bpsi = bcur;
        if (!fused) xbeta(bcur);
        for (int m = 1; m <= iters; ++m, ++t) {
            const bool tm = timing && phase == 1 && m == iters;       // BL_GIBBS_TIMING=1: stage times
            if (tm) cudaEventRecord(ev[0], st);
            StreamId id{seed, 0, t, (uint32_t)N};
            // one chain: shared and own rows are the same layout, and k_logit_psi_draw is the faster kernel for it
            // (no trip through shared memory: 146 against 153 us at N = 1M, P = 64)
            cudaError_t e = !fused                    ? launch_devroye_refill(w, shape, psi, T, id, st, work)
                            : shared_rows && chains > 1 ? launch_logit_psi_draw_shared(w, shape, tX, bpsi, bstride, chains, N, P, id, st)
                                                        : launch_logit_psi_draw(w, nullptr, shape, tX, bpsi, bstride, chains, N, P, id, st);
            if (e != cudaSuccess) { err = cudaGetErrorString(e); return 1; }
            if (tm) cudaEventRecord(ev[1], st);
            if (nt > 1)
                k_gram_partial<kGramRows, false><<<dim3(nslab, tiles, chains), 256, gram_smem_bytes(true), st>>>(part, tX, x_stride, w, N, P, nt);
            else if (packed)
                k_gram_partial<kGramRowsDiag, true, true><<<dim3(nslab, tiles, chains), 256, gram_smem_bytes(false, true), st>>>(part, tX, x_stride, w, N, P, nt);
            else
                k_gram_partial<kGramRowsDiag, true><<<dim3(nslab, tiles, chains), 256, gram_smem_bytes(false), st>>>(part, tX, x_stride, w, N, P, nt);
            if (tm) cudaEventRecord(ev[2], st);
            k_gram_reduce<<<dim3(cdiv((int64_t)P * P, 32), chains), 256, 0, st>>>(acc, nullptr, part, P, nt, slabs_total, PeerPush{}, packed ? 1 : 0);
            if (tm) cudaEventRecord(ev[3], st);
            if (mode != kBetaConstrained && P <= 64 && !kSlowBeta)
                k_beta_draw<true, true><<<chains, 256, beta_smem, st>>>(mode, acc, P0, bP, 0, bprev, bcur, nullptr, P, seed, t, status,
                                                                     PeerWait{}, bstride, nullptr, 1);
            else
                k_beta_draw<true><<<chains, 256, beta_smem, st>>>(mode, acc, P0, bP, 0, bprev, bcur, nullptr, P, seed, t, status,
                                                               PeerWait{}, bstride, nullptr, getenv("BL_BETA_NO_SPEC") ? 3 : 1);
            count_launch(3);
            if (tm) cudaEventRecord(ev[4], st);
            bpsi = bcur;
            if (!fused) xbeta(bcur);
            if (tm) {
                cudaEventRecord(ev[5], st);
                cudaEventSynchronize(ev[5]);
                float d[5];
                for (int k = 0; k < 5; ++k) cudaEventElapsedTime(&d[k], ev[k], ev[k + 1]);
                fprintf(stderr, "[bl %s timing, us] draw %.1f gram %.1f reduce %.1f beta %.1f xbeta %.1f\n",
                        shared_rows ? "multichain" : "chains", d[0] * 1e3, d[1] * 1e3, d[2] * 1e3, d[3] * 1e3, d[4] * 1e3);
                for (auto &x : ev) cudaEventDestroy(x);
            }
            if (phase == 1) {
                bprev = bcur;
                if (m < iters) bcur += P;
            }
        }
    }
    GB_CK(cudaGetLastError());
    int h = 0;
    GB_CK(cudaMemcpyAsync(&h, status, sizeof(int), cudaMemcpyDeviceToHost, st));
    GB_CK(cudaStreamSynchronize(st));
    if (h != 0) { err = std::string(who) + ": a chain's posterior precision is not positive definite"; return 1; }
    return 0;
}

// ------------------------------------------------------------------------------------
// Multinomial logit (MultLogit::gibbs, MultLogit.hpp:261-372)
// ------------------------------------------------------------------------------------
// w_out: N x (J-1) x samp (or null), beta_out: P x (J-1) x samp, ty: (J-1) x N,
// m0: P x (J-1), P0: P x P x (J-1).
int mlogit_gibbs_device(double *w_out, double *beta_out, const double *ty, const double *tX,
                        const double *n, const double *m0, const double *P0, int64_t N, int P, int J,
                        int samp, int burn, uint64_t seed, int flags, uint64_t obs0, bool sharded,
                        cudaStream_t st, std::string &err)
{
    if (N <= 0 || P <= 0 || J < 2 || samp <= 0 || burn < 0) { err = "mult_gibbs: bad dimensions"; return 1; }
    const int U = J - 1;
    DevMem mem;
    mem.st = st;
    Sweep s;
    s.N = N; s.P = P; s.obs0 = obs0; s.st = st; s.tX = tX; s.exchange = sharded;
    if (s.init(mem, err)) return 1;
    double *Z, *b0, *XB, *cj, *eta, *yj, *base, *EX = nullptr;
    int *shape;
    // psi, exp(psi) and the next category's offsets from one pass over X (k_xbeta_mma<true>); BL_MLOGIT_UNFUSED
    // keeps the psi kernel and the offsets kernel per category (A/B: bit-identical chains)
    const bool fuse_next = xbeta_mma_ok(tX, P) && U <= kMlogitMaxU && !getenv("BL_MLOGIT_UNFUSED");
    const bool prebin = fuse_next && devroye_binned(N, 1 << 18);      // the psi pass also orders the next draw's rows by class
    GB_CK(mem.get(&Z, (size_t)P * U));
    GB_CK(mem.get(&b0, (size_t)P * U));
    GB_CK(mem.get(&base, (size_t)P * U));
    GB_CK(mem.get(&XB, (size_t)N * U));
    GB_CK(mem.get(&cj, N));
    GB_CK(mem.get(&eta, N));
    GB_CK(mem.get(&yj, N));
    GB_CK(mem.get(&shape, N));
    void *work = nullptr;                      // branch-class binning of the PG(1, eta) draws (large N)
    GB_CK(mem.get((char **)&work, (32 + (size_t)N) * sizeof(int)));          // [meta][index list]
    if (fuse_next) GB_CK(mem.get(&EX, (size_t)N * U));
    const bool keep_w = !(flags & BL_GIBBS_NO_W) && w_out;
    k_shape_int<<<cdiv(N, 256), 256, 0, st>>>(shape, n, N);
    count_launch();
    // Z_j = X'(n (y_j - 1/2)), b0_j = P0_j m0_j ; base_j = Z_j + b0_j   (MultLogit.hpp:214-219, :271-273)
    for (int j = 0; j < U; ++j) {
        GB_CK(cudaMemcpy2DAsync(yj, sizeof(double), ty + j, sizeof(double) * U, sizeof(double), N,
                                cudaMemcpyDeviceToDevice, st));
        k_kappa<<<cdiv(N, 256), 256, 0, st>>>(cj, yj, n, 0.0, N);
        k_matvec<<<cdiv(P, 128), 128, 0, st>>>(b0 + (size_t)P * j, P0 + (size_t)P * P * j, m0 + (size_t)P * j, P);
        count_launch(2);
        s.xtv(cj, 1.0, nullptr, nullptr, 0.0);
        if (sharded && small_allreduce(s.acc + (size_t)P * P, (size_t)P, kOpSumF64, s.status, st, err)) return 1;
        k_xtv_reduce<<<cdiv(P, 128), 128, 0, st>>>(base + (size_t)P * j, b0 + (size_t)P * j, s.acc + (size_t)P * P, s.xtv_part, P, 0, P);
        count_launch();
    }
    GB_CK(cudaMemsetAsync(beta_out, 0, sizeof(double) * (size_t)P * U * samp, st));
    if (keep_w) GB_CK(cudaMemsetAsync(w_out, 0, sizeof(double) * (size_t)N * U * samp, st));
    GB_CK(cudaMemsetAsync(XB, 0, sizeof(double) * (size_t)N * U, st));
    if (fuse_next) {
        k_fill<<<(int)std::min<int64_t>(148 * 8, cdiv((int64_t)N * U, 256)), 256, 0, st>>>(EX, 1.0, (int64_t)N * U);   // exp(0)
        count_launch();
    }
    const int total = burn + samp;
    StageTimer tmr;
    tmr.st = st;
    for (int t = 0; t < total; ++t) {
        int slice = t <= burn ? 0 : t - burn;
        double *bS = beta_out + (size_t)P * U * slice;
        double *wS = keep_w ? w_out + (size_t)N * U * slice : nullptr;
        for (int j = 0; j < U; ++j) {
            uint32_t call = (uint32_t)t * (uint32_t)U + (uint32_t)j;
            tmr.arm(t == total - 1 && j == U - 1);
            if (!fuse_next || (t == 0 && j == 0)) {
                k_mlogit_offsets<<<cdiv(N, 256), 256, 0, st>>>(cj, eta, XB, N, U, j);
                count_launch();
            }
            tmr.mark("offsets");
            double *wj = wS ? wS + (size_t)N * j : s.w;
            cudaError_t e = launch_devroye_refill(wj, shape, eta, N, StreamId{seed, obs0, call}, st, work, 1 << 18,
                                                  prebin && !(t == 0 && j == 0));
            if (e != cudaSuccess) { err = cudaGetErrorString(e); return 1; }
            tmr.mark("draw");
            if (s.gram_tail_fused()) {
                s.gram(wj, true, cj);                      // X' Omega X and X' Omega c_j from one pass (packed P = 32 kernel)
            } else {
                s.xtv(nullptr, 0.0, wj, cj, 1.0);          // X' Omega c_j
                tmr.mark("xtv");
                s.gram(wj, true);
            }
            tmr.mark("gram");
            if (s.allreduce(true, err)) return 1;
            s.beta_draw(kBetaMvn, P0 + (size_t)P * P * j, base + (size_t)P * j, true, nullptr,
                        bS + (size_t)P * j, seed, call);
            tmr.mark("beta");
            if (fuse_next) {
                // the next draw's class-ordered index list comes out of the same pass (cursors zeroed first)
                int *bm = prebin ? (int *)work : nullptr;
                if (prebin) GB_CK(cudaMemsetAsync(bm, 0, 32 * sizeof(int), st));
                s.xbeta_mlogit(XB + (size_t)N * j, bS + (size_t)P * j, MlogitNext{EX, XB, cj, eta, U, j, (j + 1) % U, bm, bm ? bm + 32 : nullptr});
            }
            else s.xbeta(XB + (size_t)N * j, bS + (size_t)P * j, nullptr, 0.0);
            tmr.mark("xbeta");
            tmr.report("mlogit");
        }
    }
    GB_CK(cudaGetLastError());
    return s.check_status(err, "mult_gibbs");
}

// ------------------------------------------------------------------------------------
// Several multinomial logit chains on ONE data set (bl_mlogit_multichain): chain c is, bit for bit, the chain
// mlogit_gibbs_device runs with seed + c and omega dropped (BL_GIBBS_UNFUSED: the one it runs with
// BL_MLOGIT_UNFUSED set).  Every category update is one launch per kernel for all chains:
//   psi   : XB_j of all chains from one pass over X (k_mlogit_psi_shared: 8 chains' beta_j in the 8 B columns
//           of the MMAs), which also forms E_j, the next category's offsets and the next draw's class-ordered
//           index list over all chains * N (chain, row) pairs.  Unfused: the single chain's psi kernel with an X
//           stride of 0, then k_mlogit_offsets, both with a chain dimension.
//   draw  : one refill over chains * N draws, stream of (chain, row) = (seed + c, row, t U + j).
//   sums  : the single chain's slab partition and kernels with a chain grid dimension (X stride 0).
//   beta  : one CTA per chain, the single chain's k_beta_draw instantiation out of shared memory; base_j =
//           P0_j m0_j + X' kappa_j is formed once and copied to every chain.
// The launches of an iteration do not depend on the number of chains.  beta_out: [chains][samp] blocks of P x U.
// ------------------------------------------------------------------------------------
// shared memory of one chain's mvn beta draw (A, B, 5 P of vectors; P <= 64: the layout of cta_plain_fast)
static size_t mlogit_multichain_beta_smem(int P)
{
    return std::max((2 * (size_t)(P | 1) * P + 5 * (size_t)P) * sizeof(double),
                    P <= 64 ? (beta_fast_e_offset(P) + 64) * sizeof(double) : (size_t)0);
}

constexpr int kMaxGridChains = 65535;   // largest y / z grid dimension

int mlogit_multichain_check(int chains, int64_t N, int P, int J, int samp, int burn, int flags, std::string &err)
{
    if (chains <= 0 || N <= 0 || P <= 0 || J < 2 || samp <= 0 || burn < 0) { err = "mlogit_multichain: bad dimensions"; return 1; }
    if (flags & ~BL_GIBBS_UNFUSED) { err = "mlogit_multichain: unsupported flags (only BL_GIBBS_UNFUSED is accepted)"; return 1; }
    if ((int64_t)chains * N >= (1LL << 31)) { err = "mlogit_multichain: chains * N must stay below 2^31 observations per call"; return 1; }
    // the chain is a y or z grid dimension of the offsets, X'v and Gram launches
    if (chains > kMaxGridChains) { err = "mlogit_multichain: chains must be at most 65535"; return 1; }
    // each chain's mvn draw runs in one CTA out of shared memory: P <= 111
    if (P > 256 || mlogit_multichain_beta_smem(P) > 200 * 1024) { err = "mlogit_multichain: P too large for the shared-memory beta draw"; return 1; }
    return 0;
}

int mlogit_multichain_device(double *beta_out, const double *ty, const double *tX, const double *n, const double *m0,
                             const double *P0, int chains, int64_t N, int P, int J, int samp, int burn, uint64_t seed,
                             int flags, cudaStream_t st, std::string &err)
{
    if (mlogit_multichain_check(chains, N, P, J, samp, burn, flags, err)) return 1;
    const int U = J - 1, K = chains;
    const int64_t T = (int64_t)K * N, UN = (int64_t)U * N;
    const size_t beta_smem = mlogit_multichain_beta_smem(P);
    const Slabs g = slab_partition(N, P);
    const int nt = g.nt, tiles = nt * (nt + 1) / 2, slabs_total = nt > 1 ? 2 * g.nslab : g.nslab;
    const bool packed = gram_packed(P);                 // P = 32: X'(Omega c_j) comes out of the Gram pass
    const size_t accn = (size_t)P * P + P;
    const bool fuse_next = !(flags & BL_GIBBS_UNFUSED) && xbeta_mma_ok(tX, P) && U <= kMlogitMaxU;
    const bool prebin = fuse_next && devroye_binned(T, 1 << 18);
    DevMem mem;
    mem.st = st;
    double *XB, *EX = nullptr, *cj, *eta, *w, *acc, *part, *xtv_part, *b0, *base, *yj;
    int *shape, *status;
    void *work;
    GB_CK(mem.get(&XB, (size_t)K * UN));
    if (fuse_next) GB_CK(mem.get(&EX, (size_t)K * UN));
    GB_CK(mem.get(&cj, T));
    GB_CK(mem.get(&eta, T));
    GB_CK(mem.get(&w, T));
    GB_CK(mem.get(&shape, T));                          // the refill reads one shape per (chain, row)
    GB_CK(mem.get(&acc, accn * K));
    GB_CK(mem.get(&part, (size_t)K * tiles * g.nslab * 2 * kGramTile * kGramTile));
    GB_CK(mem.get(&xtv_part, (size_t)K * g.xtv_slabs * P));
    GB_CK(mem.get(&b0, (size_t)P * U));
    GB_CK(mem.get(&base, (size_t)U * K * P));           // [U][K][P]: k_beta_draw reads chain c's rhs at + c P
    GB_CK(mem.get(&yj, N));
    GB_CK(mem.get(&status, 1));
    GB_CK(mem.get((char **)&work, (32 + (size_t)T) * sizeof(int)));      // branch-class binning: [meta][index list]
    GB_CK(cudaMemsetAsync(status, 0, sizeof(int), st));
    GB_CK(cudaFuncSetAttribute(k_gram_partial<kGramRows, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)gram_smem_bytes(true)));
    GB_CK(cudaFuncSetAttribute(k_gram_partial<kGramRowsDiag, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)gram_smem_bytes(false)));
    GB_CK(cudaFuncSetAttribute(k_gram_partial<kGramRowsDiag, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)gram_smem_bytes(false, true)));
    const bool lean = P <= 64 && !kSlowBeta;            // the single chain's mvn draw instantiation
    if (beta_smem > 48 * 1024)
        GB_CK(cudaFuncSetAttribute(lean ? k_beta_draw<true, true> : k_beta_draw<true, false>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, (int)beta_smem));
    const int64_t bstride = (int64_t)P * U * samp;      // chain stride of beta_out

    k_shape_int<<<cdiv(N, 256), 256, 0, st>>>(shape, n, N);
    count_launch();
    for (int64_t r = N; r < T; r += N)
        GB_CK(cudaMemcpyAsync(shape + r, shape, sizeof(int) * N, cudaMemcpyDeviceToDevice, st));
    // base_j = b0_j + X'(n (y_j - 1/2)), b0_j = P0_j m0_j, as the single chain forms it (MultLogit.hpp:214-219, :271-273)
    for (int j = 0; j < U; ++j) {
        GB_CK(cudaMemcpy2DAsync(yj, sizeof(double), ty + j, sizeof(double) * U, sizeof(double), N,
                                cudaMemcpyDeviceToDevice, st));
        k_kappa<<<cdiv(N, 256), 256, 0, st>>>(cj, yj, n, 0.0, N);
        k_matvec<<<cdiv(P, 128), 128, 0, st>>>(b0 + (size_t)P * j, P0 + (size_t)P * P * j, m0 + (size_t)P * j, P);
        launch_xtv(dim3(g.xtv_slabs), st, xtv_part, tX, N * P, cj, 1.0, nullptr, nullptr, 0.0, N, P, nullptr);
        launch_pdl(k_xtv_reduce, dim3(cdiv(P, 128)), dim3(128), 0, st, acc + (size_t)P * P, nullptr, nullptr, xtv_part, P,
                   g.xtv_slabs, (int64_t)P);
        double *bj = base + (size_t)K * P * j;
        k_xtv_reduce<<<cdiv(P, 128), 128, 0, st>>>(bj, b0 + (size_t)P * j, acc + (size_t)P * P, xtv_part, P, 0, P);
        count_launch(5);
        for (int c = 1; c < K; ++c)
            GB_CK(cudaMemcpyAsync(bj + (size_t)P * c, bj, sizeof(double) * P, cudaMemcpyDeviceToDevice, st));
    }
    GB_CK(cudaMemsetAsync(beta_out, 0, sizeof(double) * (size_t)bstride * K, st));
    GB_CK(cudaMemsetAsync(XB, 0, sizeof(double) * (size_t)K * UN, st));
    if (fuse_next) {
        k_fill<<<(int)std::min<int64_t>(148 * 8, cdiv((int64_t)K * UN, 256)), 256, 0, st>>>(EX, 1.0, (int64_t)K * UN);   // exp(0)
        count_launch();
    }
    static const int tn_flags = getenv("BL_BETA_NO_SPEC") ? 3 : 1;
    const int total = burn + samp;
    StageTimer tmr;
    tmr.st = st;
    for (int t = 0; t < total; ++t) {
        const int slice = t <= burn ? 0 : t - burn;
        double *bS = beta_out + (size_t)P * U * slice;
        for (int j = 0; j < U; ++j) {
            const uint32_t call = (uint32_t)t * (uint32_t)U + (uint32_t)j;
            const bool first = t == 0 && j == 0;
            tmr.arm(t == total - 1 && j == U - 1);
            if (!fuse_next || first) {
                k_mlogit_offsets<<<dim3(cdiv(N, 256), K), 256, 0, st>>>(cj, eta, XB, N, U, j);
                count_launch();
            }
            tmr.mark("offsets");
            cudaError_t e = launch_devroye_refill(w, shape, eta, T, StreamId{seed, 0, call, (uint32_t)N}, st, work, 1 << 18,
                                                  prebin && !first);
            if (e != cudaSuccess) { err = cudaGetErrorString(e); return 1; }
            tmr.mark("draw");
            if (!packed) {
                // X'(Omega c_j) of every chain into the tail of its sums
                launch_xtv(dim3(g.xtv_slabs, K), st, xtv_part, tX, 0, nullptr, 0.0, w, cj, 1.0, N, P, nullptr);
                launch_pdl(k_xtv_reduce, dim3(cdiv(P, 128), K), dim3(128), 0, st, acc + (size_t)P * P, nullptr, nullptr,
                           xtv_part, P, g.xtv_slabs, (int64_t)accn);
                count_launch(2);
                tmr.mark("xtv");
            }
            if (nt > 1)
                launch_pdl(k_gram_partial<kGramRows, false>, dim3(g.nslab, tiles, K), dim3(256), gram_smem_bytes(true), st,
                           part, tX, (int64_t)0, w, N, P, nt, g.nslab_diag, nullptr);
            else if (packed)
                launch_pdl(k_gram_partial<kGramRowsDiag, true, true>, dim3(g.nslab, tiles, K), dim3(256),
                           gram_smem_bytes(false, true), st, part, tX, (int64_t)0, w, N, P, nt, 0, cj);
            else
                launch_pdl(k_gram_partial<kGramRowsDiag, true>, dim3(g.nslab, tiles, K), dim3(256), gram_smem_bytes(false),
                           st, part, tX, (int64_t)0, w, N, P, nt, 0, nullptr);
            launch_pdl(k_gram_reduce, dim3(cdiv((int64_t)P * P + (packed ? P : 0), 32), K), dim3(256), 0, st, acc, nullptr,
                       part, P, nt, slabs_total, PeerPush{}, packed ? 1 : 0, 2 * g.nslab_diag, packed ? 1 : 0);
            count_launch(2);
            tmr.mark("gram");
            launch_pdl(lean ? k_beta_draw<true, true> : k_beta_draw<true, false>, dim3(K), dim3(256), beta_smem, st,
                       (int)kBetaMvn, (const double *)acc, P0 + (size_t)P * P * j, (const double *)(base + (size_t)K * P * j),
                       1, (const double *)nullptr, bS + (size_t)P * j, (double *)nullptr, P, seed, call, status, PeerWait{},
                       bstride, (const double *)nullptr, tn_flags);
            count_launch();
            tmr.mark("beta");
            const double *bj = bS + (size_t)P * j;
            if (fuse_next) {
                // the next draw's class-ordered index list comes out of the same pass (cursors zeroed first)
                int *bm = prebin ? (int *)work : nullptr;
                if (prebin) GB_CK(cudaMemsetAsync(bm, 0, 32 * sizeof(int), st));
                const MlogitNext mn{EX, XB, cj, eta, U, j, (j + 1) % U, bm, bm ? bm + 32 : nullptr};
                if (K == 1) {
                    // one chain: the single chain's kernel (no trip through shared memory)
                    const int grid = (int)std::min<int64_t>(148 * 8, std::max<int64_t>(1, (N + 255) / 256));
                    launch_pdl(k_xbeta_mma<true>, dim3(grid), dim3(256), 0, st, XB + (size_t)N * j, N, tX, N * P, bj,
                               (int64_t)0, 1, N, P, nullptr, 0.0, 0.0, mn);
                } else {
                    const int64_t items = (N + 31) / 32 * ((K + kGroupChains - 1) / kGroupChains);
                    const int grid = (int)std::min<int64_t>(148 * 8, std::max<int64_t>(1, (items + 7) / 8));
                    launch_pdl(k_mlogit_psi_shared, dim3(grid), dim3(256), 0, st, XB, tX, bj, bstride, K, N, P, mn);
                }
            } else {
                // XB_j of chain c at XB + c U N + j N: the single chain's psi kernel, rows shared (X stride 0)
                const int64_t trips = (int64_t)K * ((N + 31) / 32);
                const int grid = (int)std::min<int64_t>(148 * 8, std::max<int64_t>(1, (trips + 7) / 8));
                if (xbeta_mma_ok(tX, P))
                    launch_pdl(k_xbeta_mma<false>, dim3(grid), dim3(256), 0, st, XB + (size_t)N * j, UN, tX, (int64_t)0, bj,
                               bstride, K, N, P, nullptr, 0.0, 0.0, MlogitNext{});
                else
                    k_xbeta_chains<<<grid, 256, 0, st>>>(XB + (size_t)N * j, UN, tX, 0, bj, bstride, K, (int)N, P);
            }
            count_launch();
            tmr.mark("xbeta");
            tmr.report("mlogit multichain");
        }
    }
    GB_CK(cudaGetLastError());
    int h = 0;
    GB_CK(cudaMemcpyAsync(&h, status, sizeof(int), cudaMemcpyDeviceToHost, st));
    GB_CK(cudaStreamSynchronize(st));
    if (h != 0) { err = "mlogit_multichain: a chain's posterior precision is not positive definite"; return 1; }
    return 0;
}

// ------------------------------------------------------------------------------------
// Negative binomial, dispersion d fixed (NBPG-logmean.R:13-34, 77-106 without draw.df)
// ------------------------------------------------------------------------------------
// beta_out: P x samp (every iteration kept), w_out: N (last omega) or null.
int nb_gibbs_device(double *w_out, double *beta_out, const double *y, const double *tX, double d,
                    const double *m0, const double *P0, int64_t N, int P, int samp, uint64_t seed,
                    uint64_t obs0, bool sharded, cudaStream_t st, std::string &err)
{
    if (N <= 0 || P <= 0 || samp <= 0 || !(d > 0)) { err = "nb_gibbs: bad arguments"; return 1; }
    DevMem mem;
    mem.st = st;
    Sweep s;
    s.N = N; s.P = P; s.obs0 = obs0; s.st = st; s.tX = tX; s.exchange = sharded;
    if (s.init(mem, err)) return 1;
    double *kappa, *b0, *shape, *beta0;
    void *work;
    GB_CK(mem.get(&kappa, N));
    GB_CK(mem.get(&shape, N));
    GB_CK(mem.get(&b0, P));
    GB_CK(mem.get(&beta0, P));
    GB_CK(mem.get((char **)&work, hybrid_workspace_bytes(N)));
    const double ld = log(d);
    k_kappa<<<cdiv(N, 256), 256, 0, st>>>(kappa, y, nullptr, d, N);          // (y - d)/2
    k_shape_add<<<cdiv(N, 256), 256, 0, st>>>(shape, y, d, N);                // b = y + d
    k_matvec<<<cdiv(P, 128), 128, 0, st>>>(b0, P0, m0, P);
    count_launch(3);
    GB_CK(cudaMemsetAsync(beta0, 0, sizeof(double) * P, st));
    double *w = w_out ? w_out : s.w;
    StageTimer tmr;
    tmr.st = st;
    for (int t = 0; t < samp; ++t) {
        const double *bprev = t == 0 ? beta0 : beta_out + (size_t)P * (t - 1);
        tmr.arm(t == samp - 1);
        s.xbeta(s.psi, bprev, nullptr, 0.0, -ld);                              // psi = X beta - log d
        tmr.mark("xbeta");
        StreamId id{seed, obs0, (uint32_t)t};
        cudaError_t e = N >= (1 << 15)
            ? launch_hybrid_binned(w, shape, s.psi, (int)N, id, work, st)
            : launch_rpg(kHybrid, w, shape, s.psi, N, 0, nullptr, id, st);
        if (e != cudaSuccess) { err = cudaGetErrorString(e); return 1; }
        tmr.mark("draw");
        s.xtv(kappa, 1.0, w, nullptr, ld);                                     // X'(kappa + omega log d)
        tmr.mark("xtv");
        s.gram(w, true);
        tmr.mark("gram");
        if (s.allreduce(true, err)) return 1;
        s.beta_draw(kBetaPlain, P0, b0, true, nullptr, beta_out + (size_t)P * t, seed, (uint32_t)t);
        tmr.mark("beta");
        tmr.report("nb");
    }
    GB_CK(cudaGetLastError());
    return s.check_status(err, "nb_gibbs");
}

static const char *const kNbBadCountMsg = ": counts y must be finite, non-negative and below 2^31 - 1";

// ------------------------------------------------------------------------------------
// Negative binomial with the dispersion sampled (NB.PG.gibbs, NBPG-logmean.R:36-113, with
// draw.df, NB-Shape.R:9-53): per iteration phi = X beta; d | beta by one random-walk
// Metropolis step; psi = phi - log d; omega = PG(y + d, psi); beta | omega, d.  d, log d and
// everything derived from them stay on the device.  beta_out: P x samp, d_out: samp (recorded
// past burn-in), w_out: N (last omega) or null.  Sharded rows (communicator open): ymax, the histogram
// behind G and, every iteration, the four N-term log-likelihood sums are all-reduced (NCCL, 4 doubles);
// the Metropolis uniforms come from a stream every rank shares, so d stays identical on all ranks.
// ------------------------------------------------------------------------------------
int nb_gibbs_df_device(double *w_out, double *beta_out, double *d_out, const double *y, const double *tX,
                       double d0, const double *m0, const double *P0, int64_t N, int P, int samp, int burn,
                       uint64_t seed, uint64_t obs0, bool sharded_arg, int real_d, cudaStream_t st, std::string &err)
{
    if (N <= 0 || P <= 0 || samp <= 0 || burn < 0 || (real_d ? !(d0 > 0.0) : (!(d0 >= 1.0) || d0 != floor(d0)))) {
        err = real_d ? "nb_gibbs_dfreal: bad arguments (d0 must be positive)"
                     : "nb_gibbs_df: bad arguments (d0 must be a positive integer)";
        return 1;
    }
    const bool sharded = sharded_arg && cs().world > 1;
    DevMem mem;
    mem.st = st;
    Sweep s;
    s.N = N; s.P = P; s.obs0 = obs0; s.st = st; s.tX = tX; s.exchange = sharded;
    if (s.init(mem, err)) return 1;
    double *kappa, *b0, *shape, *bcur, *dpair, *G, *dfpart;
    unsigned long long *ymax_d;
    void *work;
    GB_CK(mem.get(&kappa, N));
    GB_CK(mem.get(&shape, N));
    GB_CK(mem.get(&b0, P));
    GB_CK(mem.get(&bcur, 2 * (size_t)P));
    GB_CK(mem.get(&dpair, 2));                 // d, log d
    GB_CK(mem.get(&ymax_d, 1));
    GB_CK(mem.get((char **)&work, hybrid_workspace_bytes(N)));
    const int nblk = (int)std::min<int64_t>(148 * 4, std::max<int64_t>(1, N / 1024));
    GB_CK(mem.get(&dfpart, (size_t)nblk * 4));
    double *dfsum;
    GB_CK(mem.get(&dfsum, 4));
    // ymax, G
    GB_CK(cudaMemsetAsync(ymax_d, 0, sizeof(unsigned long long), st));
    k_nb_ymax<<<148 * 2, 256, 0, st>>>(ymax_d, y, N);
    if (sharded && small_allreduce(ymax_d, 1, kOpMaxU64, s.status, st, err)) return 1;
    unsigned long long ymax64 = 0;
    GB_CK(cudaMemcpyAsync(&ymax64, ymax_d, sizeof(ymax64), cudaMemcpyDeviceToHost, st));
    GB_CK(cudaStreamSynchronize(st));
    if (ymax64 == kNbBadCount) {
        err = std::string(real_d ? "nb_gibbs_dfreal" : "nb_gibbs_df") + kNbBadCountMsg;
        return 1;
    }
    const int ymax = (int)ymax64;
    unsigned long long *hist;
    GB_CK(mem.get(&hist, (size_t)ymax + 2));
    GB_CK(mem.get(&G, (size_t)ymax + 1));
    GB_CK(cudaMemsetAsync(hist, 0, sizeof(unsigned long long) * ((size_t)ymax + 2), st));
    k_nb_hist<<<148 * 2, 256, 0, st>>>(hist, y, N);
    if (sharded && small_allreduce(hist, (size_t)ymax + 2, kOpSumU64, s.status, st, err)) return 1;
    k_nb_suffix<<<1, 1, 0, st>>>(G, hist, ymax);
    k_matvec<<<cdiv(P, 128), 128, 0, st>>>(b0, P0, m0, P);
    count_launch(4);
    const double dinit[2] = {d0, log(d0)};
    GB_CK(cudaMemcpyAsync(dpair, dinit, sizeof(dinit), cudaMemcpyHostToDevice, st));
    GB_CK(cudaMemsetAsync(bcur, 0, sizeof(double) * 2 * P, st));
    double *w = w_out ? w_out : s.w;
    for (int t = 0; t < samp + burn; ++t) {
        const double *bprev = bcur + (size_t)P * (t & 1);
        double *bnext = t >= burn ? beta_out + (size_t)P * (t - burn) : bcur + (size_t)P * ((t + 1) & 1);
        s.xbeta(s.psi, bprev, nullptr, 0.0);                                   // phi = X beta
        if (real_d) k_nb_dfreal_partial<<<nblk, 256, 0, st>>>(dfpart, s.psi, y, dpair, N, seed, (uint32_t)t);
        else k_nb_df_partial<<<nblk, 256, 0, st>>>(dfpart, s.psi, y, dpair, N, seed, (uint32_t)t);
        if (sharded) {
            k_nb_df_fold<<<1, 32, 0, st>>>(dfsum, dfpart, nblk);
            count_launch();
            if (small_allreduce(dfsum, 4, kOpSumF64, s.status, st, err)) return 1;
        }
        if (real_d)
            k_nb_dfreal_decide<<<1, 32, 0, st>>>(dpair, dpair + 1, t >= burn ? d_out + (t - burn) : nullptr,
                                                 sharded ? dfsum : dfpart, sharded ? 1 : nblk, seed, (uint32_t)t);
        else
            k_nb_df_decide<<<1, 32, 0, st>>>(dpair, dpair + 1, t >= burn ? d_out + (t - burn) : nullptr,
                                             sharded ? dfsum : dfpart, sharded ? 1 : nblk, G, ymax, seed, (uint32_t)t);
        k_nb_prepare<<<cdiv(N, 256), 256, 0, st>>>(s.psi, shape, kappa, y, dpair, dpair + 1, N);
        count_launch(3);
        StreamId id{seed, obs0, (uint32_t)t};
        cudaError_t e = N >= (1 << 15)
            ? launch_hybrid_binned(w, shape, s.psi, (int)N, id, work, st)
            : launch_rpg(kHybrid, w, shape, s.psi, N, 0, nullptr, id, st);
        if (e != cudaSuccess) { err = cudaGetErrorString(e); return 1; }
        s.xtv(kappa, 1.0, w, nullptr, 0.0, dpair + 1);                         // X'(kappa + omega log d)
        s.gram(w, true);
        if (s.allreduce(true, err)) return 1;
        s.beta_draw(kBetaPlain, P0, b0, true, nullptr, bnext, seed, (uint32_t)t);
        // the next iteration reads beta from where this one wrote it
        if (t >= burn) {
            GB_CK(cudaMemcpyAsync(bcur + (size_t)P * ((t + 1) & 1), bnext, sizeof(double) * P, cudaMemcpyDeviceToDevice, st));
        }
    }
    GB_CK(cudaGetLastError());
    return s.check_status(err, "nb_gibbs_df");
}

// ------------------------------------------------------------------------------------
// Several negative-binomial chains on ONE data set (bl_nb_multichain): chain c is, bit for bit, the chain
// nb_gibbs_df_device runs with seed + c (dmode BL_NB_D_INT / BL_NB_D_REAL), or, with d fixed (BL_NB_D_FIXED),
// iterations burn .. burn + samp - 1 of nb_gibbs_device with seed + c.  Every stage is one launch for all chains and
// follows the single chain's stage, with its summation order:
//   phi   : X beta of all chains from one read of X (k_xbeta_shared, 8 chains per pass; one chain: k_xbeta_mma; odd
//           P or unaligned X: k_xbeta with a chain grid dimension).  Fixed d: psi = phi - log d in the same pass.
//   d     : (sampled d) the single chain's dispersion kernels with a chain dimension over its nblk slabs; ymax, the
//           histogram and G depend on y alone and are formed once.
//   omega : one rpg_hybrid batch over chains * N (chain, row) pairs, the stream of (chain, row) keyed by (seed + c,
//           row).  The binned or per-lane sampler is picked by N, as the single chain picks it, so every draw runs
//           the single chain's sampler code.
//   sums  : the single chain's X'v and Gram slab partition and kernels with a chain grid dimension, X stride 0.
//   beta  : one plain draw per chain side by side, the single chain's instantiation (shared memory; above P ~ 92
//           global scratch, one block per chain).
// Per-chain state: psi, omega, kappa, shapes [chains][N]; d at dvec[c], log d at dvec[chains + c] (one chain: the
// single chain's (d, log d) pair).  beta_out: [chains][samp][P]; d_out: [chains][samp] or null.
// ------------------------------------------------------------------------------------
int nb_multichain_check(int chains, int64_t N, int P, int samp, int burn, double d0, int dmode, std::string &err)
{
    if (chains < 1) { err = "nb_multichain: chains must be at least 1"; return 1; }
    if (N < 1 || P < 1 || samp < 1 || burn < 0) { err = "nb_multichain: bad dimensions"; return 1; }
    if ((int64_t)chains * N >= (1LL << 31)) { err = "nb_multichain: chains * N must stay below 2^31 observations per call"; return 1; }
    // the chain is a y or z grid dimension of the dispersion, X'v and Gram launches
    if (chains > kMaxGridChains) { err = "nb_multichain: chains must be at most 65535"; return 1; }
    if (P > 256) { err = "nb_multichain: P > 256 covariates is not supported by the single-CTA beta draw"; return 1; }
    if (dmode != BL_NB_D_FIXED && dmode != BL_NB_D_INT && dmode != BL_NB_D_REAL) {
        err = "nb_multichain: unknown dmode (BL_NB_D_FIXED, BL_NB_D_INT or BL_NB_D_REAL)";
        return 1;
    }
    if (dmode == BL_NB_D_INT && (!(d0 >= 1.0) || d0 != floor(d0))) { err = "nb_multichain: bad arguments (d0 must be a positive integer)"; return 1; }
    if (dmode != BL_NB_D_INT && !(d0 > 0.0)) { err = "nb_multichain: bad arguments (d0 must be positive)"; return 1; }
    return 0;
}

int nb_multichain_device(double *beta_out, double *d_out, const double *y, const double *tX, double d0, const double *m0,
                         const double *P0, int chains, int64_t N, int P, int samp, int burn, uint64_t seed, int dmode,
                         cudaStream_t st, std::string &err)
{
    if (nb_multichain_check(chains, N, P, samp, burn, d0, dmode, err)) return 1;
    const int K = chains;
    const int64_t T = (int64_t)K * N;
    const bool fixed = dmode == BL_NB_D_FIXED, real_d = dmode == BL_NB_D_REAL;
    const Slabs g = slab_partition(N, P);
    const int nt = g.nt, tiles = nt * (nt + 1) / 2, slabs_total = nt > 1 ? 2 * g.nslab : g.nslab;
    const bool packed = gram_packed(P);
    const size_t accn = (size_t)P * P + P;
    const BetaSmem bs = beta_smem_of(P);
    const bool lean = P <= 64 && !kSlowBeta;            // Sweep::beta_draw's plain-draw instantiation
    const bool binned = N >= (1 << 15);                 // the single chain's choice of sampler path, by its own N
    const int nblk = (int)std::min<int64_t>(148 * 4, std::max<int64_t>(1, N / 1024));   // as nb_gibbs_df_device
    DevMem mem;
    mem.st = st;
    double *psi, *w, *kappa, *shape, *acc, *part, *xtv_part, *b0, *bscr, *dvec = nullptr, *dfpart = nullptr,
           *G = nullptr, *gwork = nullptr;
    int *status;
    void *work = nullptr;
    GB_CK(mem.get(&psi, T));
    GB_CK(mem.get(&w, T));
    GB_CK(mem.get(&kappa, T));
    GB_CK(mem.get(&shape, T));
    GB_CK(mem.get(&acc, accn * K));
    GB_CK(mem.get(&part, (size_t)K * tiles * g.nslab * 2 * kGramTile * kGramTile));
    GB_CK(mem.get(&xtv_part, (size_t)K * g.xtv_slabs * P));
    GB_CK(mem.get(&b0, (size_t)K * P));                 // P0 m0, one copy per chain: k_beta_draw reads chain c's at + c P
    GB_CK(mem.get(&bscr, (size_t)K * 2 * P));           // burn-in betas [chain][parity][P]
    GB_CK(mem.get(&status, 1));
    if (binned) GB_CK(mem.get((char **)&work, hybrid_workspace_bytes(T)));
    if (!bs.use_smem) GB_CK(mem.get(&gwork, beta_gwork_doubles(P) * K));
    GB_CK(cudaMemsetAsync(status, 0, sizeof(int), st));
    GB_CK(cudaFuncSetAttribute(k_gram_partial<kGramRows, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)gram_smem_bytes(true)));
    GB_CK(cudaFuncSetAttribute(k_gram_partial<kGramRowsDiag, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)gram_smem_bytes(false)));
    GB_CK(cudaFuncSetAttribute(k_gram_partial<kGramRowsDiag, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)gram_smem_bytes(false, true)));
    if (bs.use_smem && bs.plain > 48 * 1024)
        GB_CK(cudaFuncSetAttribute(lean ? k_beta_draw<true, true> : k_beta_draw<true, false>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bs.plain));

    k_matvec<<<cdiv(P, 128), 128, 0, st>>>(b0, P0, m0, P);
    count_launch();
    for (int c = 1; c < K; ++c)
        GB_CK(cudaMemcpyAsync(b0 + (size_t)P * c, b0, sizeof(double) * P, cudaMemcpyDeviceToDevice, st));
    const double ld0 = log(d0);
    int ymax = 0;
    if (fixed) {
        // kappa = (y - d)/2 and b = y + d are the same for every chain: formed once, then copied
        k_kappa<<<cdiv(N, 256), 256, 0, st>>>(kappa, y, nullptr, d0, N);
        k_shape_add<<<cdiv(N, 256), 256, 0, st>>>(shape, y, d0, N);
        count_launch(2);
        for (int64_t r = N; r < T; r += N) {
            GB_CK(cudaMemcpyAsync(kappa + r, kappa, sizeof(double) * N, cudaMemcpyDeviceToDevice, st));
            GB_CK(cudaMemcpyAsync(shape + r, shape, sizeof(double) * N, cudaMemcpyDeviceToDevice, st));
        }
        if (d_out) {
            k_fill<<<(int)std::min<int64_t>(148 * 8, cdiv((int64_t)K * samp, 256)), 256, 0, st>>>(d_out, d0, (int64_t)K * samp);
            count_launch();
        }
    } else {
        // ymax and G[j] = #{y_i > j}, as nb_gibbs_df_device forms them, shared by the chains
        unsigned long long *ymax_d, *hist;
        GB_CK(mem.get(&ymax_d, 1));
        GB_CK(cudaMemsetAsync(ymax_d, 0, sizeof(unsigned long long), st));
        k_nb_ymax<<<148 * 2, 256, 0, st>>>(ymax_d, y, N);
        count_launch();
        unsigned long long ymax64 = 0;
        GB_CK(cudaMemcpyAsync(&ymax64, ymax_d, sizeof(ymax64), cudaMemcpyDeviceToHost, st));
        GB_CK(cudaStreamSynchronize(st));
        if (ymax64 == kNbBadCount) { err = std::string("nb_multichain") + kNbBadCountMsg; return 1; }
        ymax = (int)ymax64;
        GB_CK(mem.get(&hist, (size_t)ymax + 2));
        GB_CK(mem.get(&G, (size_t)ymax + 1));
        GB_CK(cudaMemsetAsync(hist, 0, sizeof(unsigned long long) * ((size_t)ymax + 2), st));
        k_nb_hist<<<148 * 2, 256, 0, st>>>(hist, y, N);
        k_nb_suffix<<<1, 1, 0, st>>>(G, hist, ymax);
        count_launch(2);
        GB_CK(mem.get(&dfpart, (size_t)K * nblk * 4));
        GB_CK(mem.get(&dvec, 2 * (size_t)K));
        std::vector<double> dinit(2 * (size_t)K, d0);
        for (int c = 0; c < K; ++c) dinit[(size_t)K + c] = ld0;
        GB_CK(cudaMemcpyAsync(dvec, dinit.data(), sizeof(double) * 2 * K, cudaMemcpyHostToDevice, st));
        GB_CK(cudaStreamSynchronize(st));         // dinit is a pageable host buffer that leaves scope
    }
    GB_CK(cudaMemsetAsync(bscr, 0, sizeof(double) * 2 * P * (size_t)K, st));

    const int64_t bstride = (int64_t)P * samp;          // chain stride of beta_out
    const bool mma = xbeta_mma_ok(tX, P);
    const int xgrid = (int)std::min<int64_t>(148 * 8, std::max<int64_t>(1, (N + 255) / 256));     // Sweep::xbeta's grid
    const int64_t items = (N + 31) / 32 * ((K + kGroupChains - 1) / kGroupChains);
    const int sgrid = (int)std::min<int64_t>(148 * 8, std::max<int64_t>(1, (items + 7) / 8));
    const double shift = fixed ? -ld0 : 0.0;
    static const int tn_flags = getenv("BL_BETA_NO_SPEC") ? 3 : 1;
    StageTimer tmr;
    tmr.st = st;
    for (int t = 0; t < burn + samp; ++t) {
        // the beta every chain conditions on: the burn-in slot of parity t, or its last recorded draw
        const double *bprev = t <= burn ? bscr + (size_t)P * (t & 1) : beta_out + (size_t)P * (t - 1 - burn);
        const int64_t pstride = t <= burn ? 2 * (int64_t)P : bstride;
        const bool rec = t >= burn;
        double *bnext = rec ? beta_out + (size_t)P * (t - burn) : bscr + (size_t)P * ((t + 1) & 1);
        const int64_t nstride = rec ? bstride : 2 * (int64_t)P;
        tmr.arm(t == burn + samp - 1);
        if (mma && K == 1)
            launch_pdl(k_xbeta_mma<false>, dim3(xgrid), dim3(256), 0, st, psi, N, tX, N * P, bprev, (int64_t)0, 1, N, P,
                       (const double *)nullptr, 0.0, shift, MlogitNext{});
        else if (mma)
            launch_pdl(k_xbeta_shared, dim3(sgrid), dim3(256), 0, st, psi, tX, bprev, pstride, K, N, P, shift);
        else
            k_xbeta<<<dim3(xgrid, K), 256, P * sizeof(double), st>>>(psi, tX, bprev, nullptr, 0.0, shift, N, P, pstride);
        count_launch();
        tmr.mark("xbeta");
        if (!fixed) {
            // d | beta of every chain, then psi = phi - log d, b = y + d, kappa = (y - d)/2
            double *drec = rec && d_out ? d_out + (t - burn) : nullptr;
            if (real_d) {
                k_nb_dfreal_partial<<<dim3(nblk, K), 256, 0, st>>>(dfpart, psi, y, dvec, N, seed, (uint32_t)t);
                k_nb_dfreal_decide<<<K, 32, 0, st>>>(dvec, dvec + K, drec, dfpart, nblk, seed, (uint32_t)t, (int64_t)samp);
            } else {
                k_nb_df_partial<<<dim3(nblk, K), 256, 0, st>>>(dfpart, psi, y, dvec, N, seed, (uint32_t)t);
                k_nb_df_decide<<<K, 32, 0, st>>>(dvec, dvec + K, drec, dfpart, nblk, G, ymax, seed, (uint32_t)t, (int64_t)samp);
            }
            k_nb_prepare<<<dim3(cdiv(N, 256), K), 256, 0, st>>>(psi, shape, kappa, y, dvec, dvec + K, N);
            count_launch(3);
            tmr.mark("dispersion");
        }
        // one chain: the plain stream is the chain-keyed one, and the single chain's sampler kernels run
        const StreamId id{seed, 0, (uint32_t)t, K > 1 ? (uint32_t)N : 0u};
        cudaError_t e = binned ? launch_hybrid_binned(w, shape, psi, (int)T, id, work, st)
                               : launch_rpg(kHybrid, w, shape, psi, T, 0, nullptr, id, st);
        if (e != cudaSuccess) { err = cudaGetErrorString(e); return 1; }
        tmr.mark("draw");
        // X'(kappa + omega log d) of every chain into the tail of its sums
        launch_xtv(dim3(g.xtv_slabs, K), st, xtv_part, tX, 0, kappa, 1.0, w, nullptr, fixed ? ld0 : 0.0, N, P,
                   fixed ? nullptr : dvec + K);
        launch_pdl(k_xtv_reduce, dim3(cdiv(P, 128), K), dim3(128), 0, st, acc + (size_t)P * P, (const double *)nullptr,
                   (const double *)nullptr, xtv_part, P, g.xtv_slabs, (int64_t)accn);
        count_launch(2);
        tmr.mark("xtv");
        if (nt > 1)
            launch_pdl(k_gram_partial<kGramRows, false>, dim3(g.nslab, tiles, K), dim3(256), gram_smem_bytes(true), st,
                       part, tX, (int64_t)0, w, N, P, nt, g.nslab_diag, (const double *)nullptr);
        else if (packed)
            launch_pdl(k_gram_partial<kGramRowsDiag, true, true>, dim3(g.nslab, tiles, K), dim3(256),
                       gram_smem_bytes(false, true), st, part, tX, (int64_t)0, w, N, P, nt, 0, (const double *)nullptr);
        else
            launch_pdl(k_gram_partial<kGramRowsDiag, true>, dim3(g.nslab, tiles, K), dim3(256), gram_smem_bytes(false),
                       st, part, tX, (int64_t)0, w, N, P, nt, 0, (const double *)nullptr);
        launch_pdl(k_gram_reduce, dim3(cdiv((int64_t)P * P, 32), K), dim3(256), 0, st, acc, (const double *)nullptr,
                   part, P, nt, slabs_total, PeerPush{}, packed ? 1 : 0, 2 * g.nslab_diag, 0);
        count_launch(2);
        tmr.mark("gram");
        if (bs.use_smem)
            launch_pdl(lean ? k_beta_draw<true, true> : k_beta_draw<true, false>, dim3(K), dim3(256), bs.plain, st,
                       (int)kBetaPlain, (const double *)acc, P0, (const double *)b0, 1, (const double *)nullptr, bnext,
                       (double *)nullptr, P, seed, (uint32_t)t, status, PeerWait{}, nstride, (const double *)nullptr,
                       tn_flags);
        else
            k_beta_draw<false><<<K, 256, 0, st>>>(kBetaPlain, acc, P0, b0, 1, nullptr, bnext, gwork, P, seed, (uint32_t)t,
                                                  status, PeerWait{}, nstride, nullptr, 0);
        count_launch();
        tmr.mark("beta");
        tmr.report("nb multichain");
    }
    GB_CK(cudaGetLastError());
    int h = 0;
    GB_CK(cudaMemcpyAsync(&h, status, sizeof(int), cudaMemcpyDeviceToHost, st));
    GB_CK(cudaStreamSynchronize(st));
    if (h != 0) { err = "nb_multichain: a chain's posterior precision is not positive definite"; return 1; }
    return 0;
}

// One dispersion step of `chains` chains on given phi [chains][N] and d [chains] (host), with the kernels, grids and
// nblk of nb_gibbs_df_device (chains = 1) and nb_multichain_device: ymax, histogram, G, the N-term partials and the
// decide kernel, which writes out[c][5] = {d', accept variate (u; real walk: log u), llh(d), llh(d'), new d}.
// Arguments are checked by the caller (bl_probe_nb_dispersion).
int nb_dispersion_probe(double *out, const double *phi, const double *y, const double *d, int chains, int64_t N,
                        uint64_t seed, uint32_t call, int real_d, cudaStream_t st, std::string &err)
{
    const int K = chains;
    const int nblk = (int)std::min<int64_t>(148 * 4, std::max<int64_t>(1, N / 1024));   // as nb_gibbs_df_device
    DevMem mem;
    mem.st = st;
    unsigned long long *ymax_d, *hist;
    double *G, *dfpart, *dvec;
    GB_CK(mem.get(&ymax_d, 1));
    GB_CK(cudaMemsetAsync(ymax_d, 0, sizeof(unsigned long long), st));
    k_nb_ymax<<<148 * 2, 256, 0, st>>>(ymax_d, y, N);
    unsigned long long ymax64 = 0;
    GB_CK(cudaMemcpyAsync(&ymax64, ymax_d, sizeof(ymax64), cudaMemcpyDeviceToHost, st));
    GB_CK(cudaStreamSynchronize(st));
    if (ymax64 == kNbBadCount) { err = std::string("probe_nb_dispersion") + kNbBadCountMsg; return 1; }
    const int ymax = (int)ymax64;
    GB_CK(mem.get(&hist, (size_t)ymax + 2));
    GB_CK(mem.get(&G, (size_t)ymax + 1));
    GB_CK(cudaMemsetAsync(hist, 0, sizeof(unsigned long long) * ((size_t)ymax + 2), st));
    k_nb_hist<<<148 * 2, 256, 0, st>>>(hist, y, N);
    k_nb_suffix<<<1, 1, 0, st>>>(G, hist, ymax);
    GB_CK(mem.get(&dfpart, (size_t)K * nblk * 4));
    GB_CK(mem.get(&dvec, 2 * (size_t)K));
    std::vector<double> dinit(2 * (size_t)K);
    for (int c = 0; c < K; ++c) { dinit[c] = d[c]; dinit[(size_t)K + c] = log(d[c]); }
    GB_CK(cudaMemcpyAsync(dvec, dinit.data(), sizeof(double) * 2 * K, cudaMemcpyHostToDevice, st));
    if (real_d) {
        k_nb_dfreal_partial<<<dim3(nblk, K), 256, 0, st>>>(dfpart, phi, y, dvec, N, seed, call);
        k_nb_dfreal_decide<<<K, 32, 0, st>>>(dvec, dvec + K, out + 4, dfpart, nblk, seed, call, 5, out);
    } else {
        k_nb_df_partial<<<dim3(nblk, K), 256, 0, st>>>(dfpart, phi, y, dvec, N, seed, call);
        k_nb_df_decide<<<K, 32, 0, st>>>(dvec, dvec + K, out + 4, dfpart, nblk, G, ymax, seed, call, 5, out);
    }
    count_launch(5);
    GB_CK(cudaGetLastError());
    GB_CK(cudaStreamSynchronize(st));            // dinit is a pageable host buffer that leaves scope
    return 0;
}

// ------------------------------------------------------------------------------------
// Posterior mode by EM (Logit::EM, Logit.hpp:488-554): the same psi / Gram / Cholesky
// kernels with omega replaced by its conditional mean.
// ------------------------------------------------------------------------------------
__global__ void k_em_weights(double *__restrict__ w, const double *__restrict__ psi,
                             const double *__restrict__ n, int64_t N)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    double h = psi[i] * 0.5;
    if (fabs(h) < 0.01)
        w[i] = n[i] / cosh(h) * (1 + h * h / 6.0 + pow(h, 4.0) / 120.0 + pow(h, 6.0) / 5040.0) * 0.25;
    else
        w[i] = n[i] * tanh(h) / h * 0.25;
}

// beta_new = (acc)^-1 rhs by Cholesky; dist = max |beta_new - beta_old|  (Logit.hpp:538-548)
__global__ void __launch_bounds__(256)
k_em_solve(const double *__restrict__ acc, const double *__restrict__ rhs, double *beta, double *dist,
           double *gwork, int P, int *status, int use_smem)
{
    extern __shared__ double sm[];
    __shared__ int ok;
    const int ld = P | 1;
    double *A = use_smem ? sm : gwork;
    double *x = A + (size_t)ld * P;
    for (int k = threadIdx.x; k < P * P; k += blockDim.x) A[k % P + (size_t)ld * (k / P)] = acc[k];
    for (int k = threadIdx.x; k < P; k += blockDim.x) x[k] = rhs[k];
    if (threadIdx.x == 0) ok = 1;
    __syncthreads();
    cta_chol_upper(A, P, ld, &ok);
    if (!ok) { if (threadIdx.x == 0) *status = 1; return; }
    if (threadIdx.x < 32) {
        int lane = threadIdx.x;
        warp_solve_ut(A, x, P, ld, lane);
        warp_solve_u(A, x, P, ld, lane);
        double d = 0.0;
        for (int i = lane; i < P; i += 32) {
            d = fmax(d, fabs(x[i] - beta[i]));
            beta[i] = x[i];
        }
        for (int o = 16; o; o >>= 1) d = fmax(d, __shfl_xor_sync(0xffffffffu, d, o));
        if (lane == 0) *dist = d;
    }
}

int logit_em_device(double *beta, const double *y, const double *tX, const double *n, int64_t N,
                    int P, double tol, int max_iter, int *iters, cudaStream_t st, std::string &err)
{
    if (N <= 0 || P <= 0) { err = "EM: bad dimensions"; return 1; }
    DevMem mem;
    mem.st = st;
    Sweep s;
    s.N = N; s.P = P; s.st = st; s.tX = tX;
    if (s.init(mem, err)) return 1;
    double *kappa, *bP, *dist;
    GB_CK(mem.get(&kappa, N));
    GB_CK(mem.get(&bP, P));
    GB_CK(mem.get(&dist, 1));
    k_kappa<<<cdiv(N, 256), 256, 0, st>>>(kappa, y, n, 0.0, N);
    count_launch();
    s.xtv(kappa, 1.0, nullptr, nullptr, 0.0);                       // bP = X' kappa (default prior b0 = 0)
    k_xtv_reduce<<<cdiv(P, 128), 128, 0, st>>>(bP, s.acc + (size_t)P * P, nullptr, s.xtv_part, P, 0, P);
    count_launch();
    GB_CK(cudaMemsetAsync(beta, 0, sizeof(double) * P, st));
    size_t smem = ((size_t)(P | 1) * P + P) * sizeof(double);
    bool use_smem = smem <= 200 * 1024;
    if (use_smem && smem > 48 * 1024)
        GB_CK(cudaFuncSetAttribute(k_em_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    double hdist = tol + 1.0;
    int iter = 0;
    while (hdist > tol && iter < max_iter) {
        s.xbeta(s.psi, beta, nullptr, 0.0);
        k_em_weights<<<cdiv(N, 256), 256, 0, st>>>(s.w, s.psi, n, N);
        count_launch();
        s.gram(s.w);
        k_em_solve<<<1, 256, use_smem ? smem : 0, st>>>(s.acc, bP, beta, dist, s.gwork, P, s.status, use_smem ? 1 : 0);
        count_launch();
        GB_CK(cudaMemcpyAsync(&hdist, dist, sizeof(double), cudaMemcpyDeviceToHost, st));
        GB_CK(cudaStreamSynchronize(st));
        ++iter;
        int h = 0;
        GB_CK(cudaMemcpy(&h, s.status, sizeof(int), cudaMemcpyDeviceToHost));
        if (h) { err = "EM: X' Omega X is not positive definite"; return 1; }
    }
    *iters = iter;
    return 0;
}

// ------------------------------------------------------------------------------------
// communicator
// ------------------------------------------------------------------------------------
int comm_unique_id(void *out128, std::string &err)
{
    if (!nccl_load(err)) return 1;
    int r = g_nccl.GetUniqueId(out128);
    if (r != 0) { err = "ncclGetUniqueId failed"; return 1; }
    return 0;
}

int comm_init(const void *id128, int rank, int world, std::string &err)
{
    if (world <= 1) { cs().world = 1; cs().rank = 0; return 0; }
    if (!nccl_load(err)) return 1;
    UniqueId id;
    memcpy(id.bytes, id128, 128);
    // ncclCommInitRank(ncclComm_t*, int nranks, ncclUniqueId commId /*by value*/, int rank)
    typedef int (*init_fn)(void **, int, UniqueId, int);
    init_fn init = (init_fn)dlsym(g_nccl.lib, "ncclCommInitRank");
    int r = init(&cs().comm, world, id, rank);
    if (r != 0) { err = std::string("ncclCommInitRank: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "error"); return 1; }
    cs().rank = rank;
    cs().world = world;
    return 0;
}

// Ranks without NCCL (e.g. several processes sharing one device, which NCCL refuses): every exchange
// then goes through the peer windows, which must be opened before the first sharded sweep.
int comm_init_local(int rank, int world, std::string &err)
{
    if (world < 1 || world > kMaxPeers || rank < 0 || rank >= world) { err = "bl_comm_init_local: need 0 <= rank < world <= 8"; return 1; }
    cs().rank = rank;
    cs().world = world;
    cs().comm = nullptr;
    cs().local = world > 1;
    return 0;
}

// Allocate (once) and zero this rank's window; out64 receives its CUDA IPC handle.
int comm_peer_handle(void *out64, std::string &err)
{
    if (cs().world <= 1) { err = "peer windows need a communicator of more than one rank (bl_comm_init first)"; return 1; }
    if (cs().world > kMaxPeers) { err = "peer windows support at most 8 ranks"; return 1; }
    if (!cs().peer.base) {
        cs().peer.slot_doubles = (size_t)kPeerMaxP * kPeerMaxP + kPeerMaxP;
        size_t bytes = kPeerFlagBytes + 2 * (size_t)kMaxPeers * cs().peer.slot_doubles * sizeof(double);
        GB_CK(cudaMalloc(&cs().peer.base, bytes));
        GB_CK(cudaMalloc((void **)&cs().peer.done, sizeof(unsigned)));
        GB_CK(cudaMemset(cs().peer.base, 0, bytes));
        GB_CK(cudaMemset(cs().peer.done, 0, sizeof(unsigned)));
        GB_CK(cudaDeviceSynchronize());
    }
    cudaIpcMemHandle_t h;
    GB_CK(cudaIpcGetMemHandle(&h, cs().peer.base));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(out64, &h, 64);
    return 0;
}

// handles: world x 64 bytes, rank order (every rank's comm_peer_handle output, all-gathered by the host).
int comm_peer_open(const void *handles, std::string &err)
{
    if (!cs().peer.base) { err = "bl_comm_peer_handle has not been called"; return 1; }
    for (int r = 0; r < cs().world; ++r) {
        if (r == cs().rank) { cs().peer.win[r] = cs().peer.base; continue; }
        if (cs().peer.win[r]) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char *)handles + 64 * (size_t)r, 64);
        GB_CK(cudaIpcOpenMemHandle(&cs().peer.win[r], h, cudaIpcMemLazyEnablePeerAccess));
    }
    cs().peer.open = true;
    return 0;
}

void comm_peer_close()
{
    for (int r = 0; r < kMaxPeers; ++r) {
        if (cs().peer.win[r] && cs().peer.win[r] != cs().peer.base) cudaIpcCloseMemHandle(cs().peer.win[r]);
        cs().peer.win[r] = nullptr;
    }
    cs().peer.open = false;
}

int comm_peer_active() { return peer_active() ? 1 : 0; }

// ---- virtual ranks (see VGroup) ---------------------------------------------------------------
int comm_virtual_create(int world, std::string &err)
{
    if (world < 2 || world > kMaxPeers) { err = "bl_vcomm_create: need 2 <= world <= 8"; return 1; }
    if (g_vgroup) { err = "bl_vcomm_create: a virtual communicator already exists"; return 1; }
    std::unique_ptr<VGroup> g(new VGroup);
    g->bar.world = world;
    const size_t slot = (size_t)kPeerMaxP * kPeerMaxP + kPeerMaxP;
    const size_t bytes = kPeerFlagBytes + 2 * (size_t)kMaxPeers * slot * sizeof(double);
    for (int r = 0; r < world; ++r) {
        std::unique_ptr<CommState> c(new CommState);
        c->rank = r; c->world = world; c->local = true; c->vbar = &g->bar;
        c->peer.slot_doubles = slot;
        GB_CK(cudaMalloc(&c->peer.base, bytes));
        GB_CK(cudaMalloc((void **)&c->peer.done, sizeof(unsigned)));
        GB_CK(cudaMemset(c->peer.base, 0, bytes));
        GB_CK(cudaMemset(c->peer.done, 0, sizeof(unsigned)));
        g->ranks.push_back(std::move(c));
    }
    for (int r = 0; r < world; ++r) {
        for (int q = 0; q < world; ++q) g->ranks[r]->peer.win[q] = g->ranks[q]->peer.base;
        g->ranks[r]->peer.open = true;
    }
    GB_CK(cudaDeviceSynchronize());
    g_vgroup = std::move(g);
    return 0;
}

// Bind the calling host thread to virtual rank `rank` (rank < 0: back to the process communicator).
int comm_virtual_bind(int rank, std::string &err)
{
    if (rank < 0) { t_cs = nullptr; return 0; }
    if (!g_vgroup || rank >= (int)g_vgroup->ranks.size()) { err = "bl_vcomm_bind: no such virtual rank"; return 1; }
    t_cs = g_vgroup->ranks[rank].get();
    return 0;
}

void comm_virtual_destroy()
{
    t_cs = nullptr;
    if (!g_vgroup) return;
    cudaDeviceSynchronize();
    for (auto &c : g_vgroup->ranks) { cudaFree(c->peer.base); cudaFree(c->peer.done); }
    g_vgroup.reset();
}

void comm_destroy()
{
    comm_peer_close();
    if (cs().peer.base) { cudaDeviceSynchronize(); cudaFree(cs().peer.base); cudaFree(cs().peer.done); cs().peer.base = nullptr; cs().peer.done = nullptr; }
    cs().peer.epoch = 0;
    if (cs().comm && g_nccl.CommDestroy) g_nccl.CommDestroy(cs().comm);
    cs().comm = nullptr;
    cs().world = 1;
    cs().rank = 0;
    cs().local = false;
}

}  // namespace bl
