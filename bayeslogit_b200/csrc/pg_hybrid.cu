// rpg_hybrid on the device: regime binning + one kernel per regime.
//
// The reference dispatches per observation inside one serial loop
// (LogitWrapper.cpp:140-162; same logic in PolyaGammaHybrid.h:26-55).  Running that
// switch per lane makes every warp execute every sampler its 32 observations need
// and makes the kernel's code footprint the sum of all samplers (~400 KB of SASS,
// far beyond the instruction cache -- the profile in profiles/r1_00_* shows 65 of
// 70 stall cycles per instruction waiting on instruction fetch).  Instead:
//
//   1. k_hyb_count    histogram of regimes (block-aggregated atomics)
//   2. k_hyb_offsets  exclusive prefix -> list offsets
//   3. k_hyb_scatter  counting sort of observation indices by regime into one
//                     int32 list (block-level ballot ranking, ascending within a
//                     block so gathers stay nearly coalesced); b <= 0 -> x = 0
//   4. kernels per regime over its index list, so that every warp runs ONE sampler:
//        saddle point (13 < b <= 170) and alternate (1 < b <= 13, b != 2): a set-up kernel
//          (envelope / chunk constants -> struct-of-arrays state in HBM) followed by a rejection-loop
//          kernel that regroups draws by proposal piece across the CTA (k_loop_regroup), once per
//          state chunk of 2^23 draws;
//        sum of gammas (b < 1), normal approximation (b > 170), Devroye (b = 1, 2): one grid-stride
//          kernel each, on a low-priority side stream underneath the two heavy regimes.
//
// Results are unchanged by the re-ordering: each observation draws from the Philox
// stream keyed by its own global index (philox.cuh).
#include <algorithm>
#include <cstdlib>
#include <vector>

#include "engine.h"
#include "pg_devroye_fast.cuh"
#include "pg_stream.cuh"

namespace bl {

namespace {

constexpr int kBinThreads = 256;
constexpr int kMetaCounts = 0;    // meta[0..7]   regime counts
constexpr int kMetaOffsets = 8;   // meta[8..15]  list offsets
constexpr int kMetaCursor = 16;   // meta[16..23] scatter cursors

__global__ void __launch_bounds__(kBinThreads)
k_hyb_count(const double *__restrict__ h, int n, int *__restrict__ meta)
{
    __shared__ int cnt[8];
    if (threadIdx.x < 8) cnt[threadIdx.x] = 0;
    __syncthreads();
    int local[6] = {0, 0, 0, 0, 0, 0};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        local[regime_of(h[i])]++;
#pragma unroll
    for (int r = 0; r < 6; ++r) {
        int v = local[r];
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(&cnt[r], v);
    }
    __syncthreads();
    if (threadIdx.x < 6 && cnt[threadIdx.x]) atomicAdd(&meta[kMetaCounts + threadIdx.x], cnt[threadIdx.x]);
}

__global__ void k_hyb_offsets(int *meta)
{
    int acc = 0;
    for (int r = 1; r < 6; ++r) {   // regime 0 (b <= 0) needs no list
        meta[kMetaOffsets + r] = acc;
        meta[kMetaCursor + r] = 0;
        acc += meta[kMetaCounts + r];
    }
}

// Four observations per thread and tile (i = tile * 1024 + k * 256 + thread): one round of
// barriers and one cursor atomic per regime for 1024 observations.
constexpr int kBinPer = 4;

__global__ void __launch_bounds__(kBinThreads)
k_hyb_scatter(const double *__restrict__ h, int n, int *__restrict__ meta, int *__restrict__ idx,
              double *__restrict__ x)
{
    constexpr int kCells = kBinPer * (kBinThreads / 32);          // (k, warp) cells of a tile, ascending i
    __shared__ int wcnt[kCells][8];                                // counts, then exclusive prefixes
    __shared__ int base[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    const int tile_obs = kBinThreads * kBinPer;
    int tiles = (n + tile_obs - 1) / tile_obs;
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        int reg[kBinPer], rank[kBinPer];
#pragma unroll
        for (int k = 0; k < kBinPer; ++k) {
            int i = tile * tile_obs + k * kBinThreads + threadIdx.x;
            reg[k] = i < n ? regime_of(h[i]) : -1;
        }
#pragma unroll
        for (int k = 0; k < kBinPer; ++k) {
            int i = tile * tile_obs + k * kBinThreads + threadIdx.x;
            if (reg[k] == kRegZero) x[i] = 0.0;                   // LogitWrapper.cpp:159-161
            rank[k] = 0;
#pragma unroll
            for (int r = 1; r < 6; ++r) {
                unsigned m = __ballot_sync(0xffffffffu, reg[k] == r);
                if (reg[k] == r) rank[k] = __popc(m & lt);
                if (lane == 0) wcnt[k * (kBinThreads / 32) + warp][r] = __popc(m);
            }
        }
        __syncthreads();
        if (threadIdx.x >= 1 && threadIdx.x < 6) {
            int r = threadIdx.x, run = 0;
            for (int c = 0; c < kCells; ++c) {
                int v = wcnt[c][r];
                wcnt[c][r] = run;
                run += v;
            }
            base[r] = run ? meta[kMetaOffsets + r] + atomicAdd(&meta[kMetaCursor + r], run) : 0;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kBinPer; ++k) {
            if (reg[k] > 0) {
                int i = tile * tile_obs + k * kBinThreads + threadIdx.x;
                idx[base[reg[k]] + wcnt[k * (kBinThreads / 32) + warp][reg[k]] + rank[k]] = i;
            }
        }
        __syncthreads();
    }
}

// kChains: the batch holds independent chains side by side and id.chain_len keys their streams (open_batch_stream); a
// compile-time switch, so that the single-batch instantiations keep their code.
template <int R, bool kChains = false>
__global__ void __launch_bounds__(128)
k_hyb_regime(double *__restrict__ x, const double *__restrict__ h, const double *__restrict__ z,
             const int *__restrict__ idx, const int *__restrict__ meta, StreamId id)
{
    const int count = meta[kMetaCounts + R];
    const int *list = idx + meta[kMetaOffsets + R];
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < count; j += gridDim.x * blockDim.x) {
        int i = list[j];
        PhiloxSource s;
        if (kChains) open_batch_stream(s, id, i);
        else s.open(id.seed, id.obs0 + (uint64_t)i, id.call_id);
        double b = h[i], zi = z[i], v;
        if (R == kRegNormal) {
            double m = pg_m1(b, zi);
            double var = pg_m2(b, zi) - m * m;
            v = m + sqrt(var) * s.norm();
        } else if (R == kRegSP) {
            sp_draw(s, v, b, zi);
        } else if (R == kRegDevroye) {
            v = devroye_sum_fast(s, (int)b, zi);
        } else if (R == kRegAlt) {
            v = alt_draw(s, b, zi);
        } else {
            v = gamma_sum(s, b, zi, 200);
        }
        x[i] = v;
    }
}

// Saddle-point regime as two kernels (pg_sp.cuh): set-up -> 19-double state per draw in HBM
// (struct of arrays over the chunk, coalesced) -> rejection loop.  Each kernel's working set of
// code stays near the 32 KB instruction cache; the state costs 304 B of HBM traffic per draw,
// ~3 % of HBM bandwidth at the rates these kernels reach.
__global__ void __launch_bounds__(128, 8)
k_sp_setup(const double *__restrict__ h, const double *__restrict__ z, const int *__restrict__ idx,
           const int *__restrict__ meta, double *__restrict__ state, int c0, int cap)
{
    const int count = min(meta[kMetaCounts + kRegSP] - c0, cap);
    const int *list = idx + meta[kMetaOffsets + kRegSP] + c0;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < count; j += gridDim.x * blockDim.x) {
        int i = list[j];
        SpState s;
        sp_setup<true>(h[i], z[i], s);      // pl as an fp32 estimate + band where one is offered
#pragma unroll
        for (int k = 0; k < kSpStateDoubles; ++k) state[(size_t)k * cap + j] = s.f[k];
    }
}

constexpr int kLaneChunk = 128;   // consecutive list positions a warp works through

// Rejection loops with CTA-level regrouping by proposal piece.
//
// In the persistent-lane loops above a lane owns a draw, and every trip of a warp runs ALL the
// proposal generators of its sampler (saddle point: inverse Gaussian on the left piece, truncated
// gamma on the right; alternate: truncated gamma, inverse chi^2, inverse Gaussian) because its 32
// lanes are a coin-flip mix of them: 14 of 32 lanes were active in the average instruction of the
// saddle-point loop, 8 of 32 in the alternate one.  Here the draws live in SLOTS in shared memory
// -- envelope state, position in the loop, Philox position -- and any thread can advance any
// slot.  Every trip the CTA (i) refills empty slots (each warp from its own chunks of the list, as
// before), (ii) sorts the live slots by the piece their pending proposal comes from (ballot ranks
// + a small prefix over the warps; first piece from the front of `perm`, last piece from the back,
// a third one behind the first), (iii) lets thread t advance slot perm[t] by one trip.  All warps
// but those on a boundary then run a single generator.  The piece of a draw's NEXT proposal is
// decided (one uniform) by whichever thread finishes the previous one, so it is always known when
// the slots are sorted.  Variates are consumed per draw in the same order as everywhere else.
constexpr int kRgThreads = 256;

template <int F, int D, int I>
struct RgSlots {
    double f[F][kRgThreads];                   // envelope / chunk constants, [field][slot]
    double d[D][kRgThreads];                   // per-draw doubles of the sampler's lane state
    uint4 buf[kRgThreads];                     // Philox: current block
    uint32_t blk[kRgThreads];                  //         next block counter
    int pos[kRgThreads];                       //         next word of buf
    int i[I][kRgThreads];                      // per-draw ints of the lane state
    int obs[kRgThreads];
    int phase[kRgThreads];                     // -1 empty, else the pending piece (1, 2[, 3])
    int perm[kRgThreads];
    int wcnt[kRgThreads / 32][3];
};

// Saddle point: pieces 1 (left) and 2 (right); d = {n, |z|/2, X}, i = {proposals made}
struct SpRegroup {
    static constexpr int F = kSpStateDoubles, D = 3, I = 1, kClasses = 2, kRegime = kRegSP;
    using Slots = RgSlots<F, D, I>;
    // new draw: first piece (PolyaGammaSP.cpp:229-231)
    __device__ static void begin(Slots &S, int t, double shape, double zraw, PhiloxSource &src)
    {
        S.d[0][t] = shape;
        S.d[1][t] = 0.5 * fabs(zraw);
        S.d[2][t] = 2.0;
        S.i[0][t] = 1;
        SpStateRef st{&S.f[0][t], (size_t)kRgThreads};
        S.phase[t] = sp_pick_left(src.unif(), st, shape) ? 1 : 2;
    }
    // one trip of slot sl; returns true when the draw is complete and writes omega
    __device__ static bool advance(Slots &S, int sl, PhiloxSource &src, double &omega)
    {
        SpLane L;
        L.X = S.d[2][sl];
        L.iter = S.i[0][sl];
        L.phase = S.phase[sl];
        const double n = S.d[0][sl];
        SpStateRef st{&S.f[0][sl], (size_t)kRgThreads};
        bool done = sp_trip_staged(src, L, n, S.d[1][sl], st);
        if (!done && L.phase == 0) {                                    // rejected: piece of the next proposal
            if (L.iter >= 200) {
                done = true;
            } else {
                L.iter++;
                L.phase = sp_pick_left(src.unif(), st, n) ? 1 : 2;
            }
        }
        if (done) {
            omega = n * 0.25 * L.X;
        } else {
            S.d[2][sl] = L.X;
            S.i[0][sl] = L.iter;
            S.phase[sl] = L.phase;
        }
        return done;
    }
};

// Alternate: pieces 1 (truncated gamma), 2 (inverse chi^2), 3 (inverse Gaussian);
// d = {|z|/2, X, alpha, sum}, i = {trial, nfull, nrem}
struct AltRegroup {
    static constexpr int F = kAltStateDoubles, D = 4, I = 3, kClasses = 3, kRegime = kRegAlt;
    using Slots = RgSlots<F, D, I>;
    __device__ static void load(const Slots &S, int sl, AltLane &L)
    {
        L.X = S.d[1][sl]; L.alpha = S.d[2][sl]; L.sum = S.d[3][sl];
        L.trial = S.i[0][sl]; L.nfull = S.i[1][sl]; L.nrem = S.i[2][sl];
        L.phase = S.phase[sl];
    }
    __device__ static void store(Slots &S, int sl, const AltLane &L)
    {
        S.d[1][sl] = L.X; S.d[2][sl] = L.alpha; S.d[3][sl] = L.sum;
        S.i[0][sl] = L.trial; S.i[1][sl] = L.nfull; S.i[2][sl] = L.nrem;
        S.phase[sl] = L.phase;
    }
    __device__ static void begin(Slots &S, int t, double shape, double zraw, PhiloxSource &src)
    {
        int nfull, nrem;
        double hrem;
        alt_plan(shape, nfull, nrem, hrem);
        AltLane L;
        L.start(nfull, nrem);
        const double zh = 0.5 * fabs(zraw);
        S.d[0][t] = zh;
        AltStateRef st{&S.f[0][t], (size_t)kRgThreads};
        alt_pick(src, L, zh, st);                                       // first proposal: cannot hit the cap
        store(S, t, L);
    }
    __device__ static bool advance(Slots &S, int sl, PhiloxSource &src, double &omega)
    {
        AltLane L;
        load(S, sl, L);
        const double zh = S.d[0][sl];
        AltStateRef st{&S.f[0][sl], (size_t)kRgThreads};
        bool done = alt_trip<false>(src, L, zh, st);
        while (!done && L.phase == 0) done = alt_pick(src, L, zh, st);  // piece of the next proposal
        if (done)
            omega = L.sum;
        else
            store(S, sl, L);
        return done;
    }
};

template <class R, bool kChains = false>
__global__ void __launch_bounds__(kRgThreads)
k_loop_regroup(double *__restrict__ x, const double *__restrict__ h, const double *__restrict__ z,
               const int *__restrict__ idx, const int *__restrict__ meta, const double *__restrict__ state,
               int c0, int cap, StreamId id)
{
    using Slots = typename R::Slots;
    extern __shared__ __align__(16) unsigned char rg_raw[];
    Slots &S = *reinterpret_cast<Slots *>(rg_raw);
    const int count = min(meta[kMetaCounts + R::kRegime] - c0, cap);
    if (count <= 0) return;
    const int *list = idx + meta[kMetaOffsets + R::kRegime] + c0;
    const unsigned full = 0xffffffffu;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    constexpr int kWarps = kRgThreads / 32;
    const int gwarp = blockIdx.x * kWarps + warp;
    const int stride = gridDim.x * kWarps * kLaneChunk;
    int cur = gwarp * kLaneChunk, cend = cur + kLaneChunk;

    S.phase[t] = -1;
    __syncthreads();
    for (;;) {
        // (i) refill this warp's empty home slots from its chunk
        const bool empty = S.phase[t] < 0;
        const unsigned want = __ballot_sync(full, empty);
        if (want && cur < count) {
            int rank = __popc(want & lt_mask);
            int cand = cur + rank;
            if (cand >= cend) cand += stride - kLaneChunk;
            if (empty && cand < count) {
                const int obs = list[cand];
#pragma unroll
                for (int k = 0; k < R::F; ++k) S.f[k][t] = __ldg(state + (size_t)k * cap + cand);
                S.obs[t] = obs;
                PhiloxSource src;
                if (kChains) open_batch_stream(src, id, obs);
                else src.open(id.seed, id.obs0 + (uint64_t)obs, id.call_id);
                R::begin(S, t, h[obs], z[obs], src);
                S.buf[t] = src.buf;
                S.blk[t] = src.blk;
                S.pos[t] = src.pos;
            }
            cur += __popc(want);
            if (cur >= cend) {
                int over = cur - cend;
                cend += stride;
                cur = cend - kLaneChunk + over;
            }
        }
        // (ii) sort live slots by piece
        const int ph = S.phase[t];
        const unsigned m1 = __ballot_sync(full, ph == 1), m2 = __ballot_sync(full, ph == 2);
        const unsigned m3 = R::kClasses > 2 ? __ballot_sync(full, ph == 3) : 0u;
        if (lane == 0) { S.wcnt[warp][0] = __popc(m1); S.wcnt[warp][1] = __popc(m2); S.wcnt[warp][2] = __popc(m3); }
        __syncthreads();
        int tot1 = 0, tot2 = 0, tot3 = 0, b1 = 0, b2 = 0, b3 = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
            int a = S.wcnt[w][0], b = S.wcnt[w][1], c = S.wcnt[w][2];
            if (w < warp) { b1 += a; b2 += b; b3 += c; }
            tot1 += a;
            tot2 += b;
            tot3 += c;
        }
        if (tot1 + tot2 + tot3 == 0) {
            if (!__syncthreads_or(cur < count)) break;                  // nothing live, nothing left anywhere
            continue;
        }
        // piece 1 from the front, piece 3 right behind it, piece 2 from the back
        if (ph == 1) S.perm[b1 + __popc(m1 & lt_mask)] = t;
        else if (ph == 3) S.perm[tot1 + b3 + __popc(m3 & lt_mask)] = t;
        else if (ph == 2) S.perm[kRgThreads - 1 - (b2 + __popc(m2 & lt_mask))] = t;
        __syncthreads();
        // (iii) thread t advances slot perm[t] by one trip
        if (t < tot1 + tot3 || t >= kRgThreads - tot2) {
            const int sl = S.perm[t];
            PhiloxSource src;
            if (kChains) open_batch_stream(src, id, S.obs[sl]);
            else src.open(id.seed, id.obs0 + (uint64_t)S.obs[sl], id.call_id);
            src.buf = S.buf[sl];
            src.blk = S.blk[sl];
            src.pos = S.pos[sl];
            double omega;
            if (R::advance(S, sl, src, omega)) {
                x[S.obs[sl]] = omega;
                S.phase[sl] = -1;
            } else {
                S.buf[sl] = src.buf;
                S.blk[sl] = src.blk;
                S.pos[sl] = src.pos;
            }
        }
        __syncthreads();
    }
}

template <class R, bool kChains>
int regroup_grid()
{
    using Slots = typename R::Slots;
    cudaFuncSetAttribute(k_loop_regroup<R, kChains>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Slots));
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_loop_regroup<R, kChains>, kRgThreads, sizeof(Slots)) != cudaSuccess || per_sm < 1)
        per_sm = 1;
    int sms = 148, dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms * per_sm;
}

// Alternate regime, same two-kernel shape: the constants of the (at most) two chunk shapes of a
// draw -> 22 doubles per draw in HBM -> persistent-lane loop over chunks and proposals.
__global__ void __launch_bounds__(128)
k_alt_setup(const double *__restrict__ h, const double *__restrict__ z, const int *__restrict__ idx,
            const int *__restrict__ meta, double *__restrict__ state, int c0, int cap)
{
    const int count = min(meta[kMetaCounts + kRegAlt] - c0, cap);
    const int *list = idx + meta[kMetaOffsets + kRegAlt] + c0;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < count; j += gridDim.x * blockDim.x) {
        int i = list[j];
        int nfull, nrem;
        double hrem, zh = 0.5 * fabs(z[i]);
        alt_plan(h[i], nfull, nrem, hrem);
        double f[kAltSetupDoubles];
        // remainder shape first: every draw has one; the shape-4 constants only if it has a full chunk
        alt_setup<true>(hrem, zh, f);
#pragma unroll
        for (int k = 0; k < kAltSetupDoubles; ++k) state[(size_t)(kAltSetupDoubles + k) * cap + j] = f[k];
        if (nfull > 0) {
            alt_setup<true>(4.0, zh, f);
#pragma unroll
            for (int k = 0; k < kAltSetupDoubles; ++k) state[(size_t)k * cap + j] = f[k];
        }
    }
}

constexpr int kStateChunk = 1 << 23;   // draws per set-up/loop kernel pair (1.3 GB of state)
constexpr int kStateDoubles = kSpStateDoubles > kAltStateDoubles ? kSpStateDoubles : kAltStateDoubles;

// Persistent grids are sized to exactly the CTAs that are resident at once (148 SMs x occupancy):
// one CTA more per SM would run alone in a second wave at a fraction of the occupancy.
template <class K>
int resident_grid(K kernel, int threads, int need)
{
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0) != cudaSuccess || per_sm < 1)
        per_sm = 1;
    int sms = 148;
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int cap = sms * per_sm;
    return need < cap ? (need > 0 ? need : 1) : cap;
}

template <int R, bool kChains>
void launch_regime(double *x, const double *h, const double *z, const int *idx, const int *meta,
                   StreamId id, int n, cudaStream_t st)
{
    static const int cap = resident_grid(k_hyb_regime<R, kChains>, 128, 1 << 30);
    int need = (n + 127) / 128;
    k_hyb_regime<R, kChains><<<need < cap ? need : cap, 128, 0, st>>>(x, h, z, idx, meta, id);
    count_launch();
}

}  // namespace

// Optional per-kernel timing of the last binned launch (bench.py's roofline leg): CUDA events on
// the launch stream around every kernel, summed per stage.
enum HybStage { kStBin = 0, kStSpSetup, kStSpLoop, kStAltSetup, kStAltLoop, kStGamma, kStNormal, kStDevroye, kStCount };
static bool g_hyb_timing = false;
static std::vector<cudaEvent_t> g_hyb_pool;
struct HybSpan { int stage; int a, b; };
static std::vector<HybSpan> g_hyb_spans;
static int g_hyb_used = 0;

void hybrid_timing_enable(bool on) { g_hyb_timing = on; }

static int hyb_mark(cudaStream_t st)
{
    if ((int)g_hyb_pool.size() <= g_hyb_used) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        g_hyb_pool.push_back(e);
    }
    cudaEventRecord(g_hyb_pool[g_hyb_used], st);
    return g_hyb_used++;
}

struct HybTimer {
    bool on;
    cudaStream_t st;
    int stage, a;
    HybTimer(bool on_, cudaStream_t st_, int stage_) : on(on_), st(st_), stage(stage_), a(on_ ? hyb_mark(st_) : 0) {}
    ~HybTimer() { if (on) g_hyb_spans.push_back(HybSpan{stage, a, hyb_mark(st)}); }
};

// ms of [binning, SP set-up, SP loop, Alt set-up, Alt loop, sum-of-gammas, normal, Devroye] and the
// number of non-empty launches per stage of the last timed launch_hybrid_binned
int hybrid_timing_last(double *ms8, int *launches8)
{
    if (g_hyb_spans.empty()) return 1;
    for (int k = 0; k < kStCount; ++k) { ms8[k] = 0.0; if (launches8) launches8[k] = 0; }
    if (cudaEventSynchronize(g_hyb_pool[g_hyb_used - 1]) != cudaSuccess) return 1;
    for (const HybSpan &sp : g_hyb_spans) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, g_hyb_pool[sp.a], g_hyb_pool[sp.b]);
        ms8[sp.stage] += ms;
        if (launches8 && ms > 0.02f) launches8[sp.stage]++;   // pairs past the regime's count return in a few us
    }
    return 0;
}

// [meta: 32 ints][index list: num ints, padded to 16 B][sampler state: 20 x min(num, chunk) doubles]
static size_t hybrid_state_offset(int64_t num) { return ((32 + (size_t)num) * sizeof(int) + 15) / 16 * 16; }

size_t hybrid_workspace_bytes(int64_t num)
{
    size_t cap = (size_t)(num < kStateChunk ? num : kStateChunk);
    return hybrid_state_offset(num) + cap * kStateDoubles * sizeof(double);
}

// side stream of the light regimes, one per device context (created on first use)
struct SideStream {
    cudaStream_t s = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
    cudaStream_t get()
    {
        if (!s) {
            int lo = 0, hi = 0;   // lowest priority: its CTAs fill SM slots the main stream leaves free
            cudaDeviceGetStreamPriorityRange(&lo, &hi);
            cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, lo);
            cudaEventCreateWithFlags(&fork, cudaEventDisableTiming);
            cudaEventCreateWithFlags(&join, cudaEventDisableTiming);
        }
        return s;
    }
};
static SideStream g_side;

template <bool kChains>
static cudaError_t launch_hybrid_binned_k(double *x, const double *h, const double *z, int num, StreamId id,
                                          void *work, cudaStream_t st)
{
    if (num <= 0) return cudaSuccess;
    int *meta = (int *)work;
    int *idx = meta + 32;
    cudaError_t e = cudaMemsetAsync(meta, 0, 32 * sizeof(int), st);
    if (e != cudaSuccess) return e;
    int tiles = (num + kBinThreads - 1) / kBinThreads;
    int grid = tiles < 148 * 8 ? tiles : 148 * 8;
    int stiles = (num + kBinThreads * kBinPer - 1) / (kBinThreads * kBinPer);
    int sgrid = stiles < 148 * 8 ? stiles : 148 * 8;
    const bool tm = g_hyb_timing;
    if (tm) { g_hyb_spans.clear(); g_hyb_used = 0; }
    {
        HybTimer t(tm, st, kStBin);
        k_hyb_count<<<grid, kBinThreads, 0, st>>>(h, num, meta);
        k_hyb_offsets<<<1, 1, 0, st>>>(meta);
        k_hyb_scatter<<<sgrid, kBinThreads, 0, st>>>(h, num, meta, idx, x);
        count_launch(3);
    }
    // The three light regimes (0.15 % + 15 % + 0.5 % of this workload's draws; the sum of gammas
    // is 200 sequential gamma variates per draw at single-digit occupancy) run on a side stream
    // forked here and joined at the end, underneath the saddle-point and alternate kernels.
    static const bool use_side = getenv("BL_HYBRID_NO_SIDE_STREAM") == nullptr;
    cudaStream_t side = use_side ? g_side.get() : st;
    if (use_side) {
        cudaEventRecord(g_side.fork, st);
        cudaStreamWaitEvent(side, g_side.fork, 0);
    }
    {
        HybTimer t(tm, side, kStGamma);
        launch_regime<kRegGamma, kChains>(x, h, z, idx, meta, id, num, side);
    }
    {
        HybTimer t(tm, side, kStNormal);
        launch_regime<kRegNormal, kChains>(x, h, z, idx, meta, id, num, side);
    }
    {
        HybTimer t(tm, side, kStDevroye);
        launch_regime<kRegDevroye, kChains>(x, h, z, idx, meta, id, num, side);
    }
    double *state = (double *)((char *)work + hybrid_state_offset(num));
    const int cap = num < kStateChunk ? num : kStateChunk;
    static const int g_sp_setup = resident_grid(k_sp_setup, 128, 1 << 30);
    static const int g_alt_setup = resident_grid(k_alt_setup, 128, 1 << 30);
    static const int g_sp_regroup = regroup_grid<SpRegroup, kChains>();
    static const int g_alt_regroup = regroup_grid<AltRegroup, kChains>();
    const int rneed = (cap + kLaneChunk * (kRgThreads / 32) - 1) / (kLaneChunk * (kRgThreads / 32));
    const int sneed = (cap + 127) / 128;
    // One set-up/loop pair per state chunk.  The regime counts live on the device, so pairs are
    // issued for the largest possible count; those past the regime's count return at once.
    for (int c0 = 0; c0 < num; c0 += cap) {
        {
            HybTimer t(tm, st, kStSpSetup);
            k_sp_setup<<<std::min(sneed, g_sp_setup), 128, 0, st>>>(h, z, idx, meta, state, c0, cap);
        }
        {
            HybTimer t(tm, st, kStSpLoop);
            k_loop_regroup<SpRegroup, kChains><<<std::min(rneed, g_sp_regroup), kRgThreads, sizeof(SpRegroup::Slots), st>>>(x, h, z, idx, meta, state, c0, cap, id);
        }
        count_launch(2);
    }
    for (int c0 = 0; c0 < num; c0 += cap) {
        {
            HybTimer t(tm, st, kStAltSetup);
            k_alt_setup<<<std::min(sneed, g_alt_setup), 128, 0, st>>>(h, z, idx, meta, state, c0, cap);
        }
        {
            HybTimer t(tm, st, kStAltLoop);
            k_loop_regroup<AltRegroup, kChains><<<std::min(rneed, g_alt_regroup), kRgThreads, sizeof(AltRegroup::Slots), st>>>(x, h, z, idx, meta, state, c0, cap, id);
        }
        count_launch(2);
    }
    if (use_side) {
        cudaEventRecord(g_side.join, side);
        cudaStreamWaitEvent(st, g_side.join, 0);
    }
    return cudaGetLastError();
}

// One rpg_hybrid batch of at most 2^31-1 observations.  `work` holds
// hybrid_workspace_bytes(num) bytes of device scratch owned by the caller's stream.
cudaError_t launch_hybrid_binned(double *x, const double *h, const double *z, int num, StreamId id,
                                 void *work, cudaStream_t st)
{
    return id.chain_len ? launch_hybrid_binned_k<true>(x, h, z, num, id, work, st)
                        : launch_hybrid_binned_k<false>(x, h, z, num, id, work, st);
}

}  // namespace bl
