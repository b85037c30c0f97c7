// Persistent-lane Devroye kernel (the PG(1,z) / sum-of-PG(1) hot path).
//
// Replaces rpg_devroye's serial loop (LogitWrapper.cpp:75-80) and Logit::draw_w
// (Logit.hpp:285-288).  Rejection sampling makes lanes finish at different times;
// instead of letting a warp spin until its slowest lane accepts, every lane is a
// small state machine: one proposal + series test per trip, and a lane whose draw
// is complete immediately pulls the next observation of its warp's chunk through a
// ballot-compacted refill (popc of the lower-lane mask gives each requesting lane
// its offset).  All 32 lanes therefore carry live work on every trip.  Because the
// variate stream is keyed by the observation index (philox.cuh), the result does
// not depend on which lane ends up drawing which observation.
//
// Work split: the batch is cut into chunks of kChunkObs observations dealt
// round-robin to warps, so a drift of z along the array cannot unbalance the SMs.
// HBM traffic: z and n in, omega out -- coalesced in runs of consecutive indices.
#include <algorithm>
#include <cstdlib>

#include "engine.h"
#include "pg_devroye_fast.cuh"
#include "pg_stream.cuh"

namespace bl {

namespace {

constexpr int kThreads = 256;
constexpr int kChunkObs = 128;

// Branch-class binning (large batches): the left proposal is the inverse-chi^2 pair loop when
// Z = |z|/2 < 1/0.64 and the inverse-Gaussian loop otherwise (PolyaGamma.cpp:87), a property of
// the observation alone.  A counting sort of the observation indices by that class makes every
// warp's chunk class-pure, so a warp runs two proposal branches instead of three.
constexpr int kBinThreads = 256;

__device__ __forceinline__ int dev_class(double z) { return fabs(z) * 0.5 >= 1.0 / kTrunc ? 1 : 0; }

// idx = the observations ordered by branch class: class 0 from the front, class 1 from the back (two cursors in
// meta[1], meta[2]) -- no counting pass.  The order inside a class depends on the CTAs' timing; the draws do not
// (their streams are keyed by the observation).
__global__ void __launch_bounds__(kBinThreads)
k_cls_scatter(const double *__restrict__ z, int n, int *__restrict__ meta, int *__restrict__ idx)
{
    BL_PDL_ENTER();
    __shared__ int wcnt[kBinThreads / 32][2];
    __shared__ int base[2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    int tiles = (n + kBinThreads - 1) / kBinThreads;
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        int i = tile * kBinThreads + threadIdx.x;
        int cls = i < n ? dev_class(z[i]) : -1;
        unsigned m1 = __ballot_sync(0xffffffffu, cls == 1), m0 = __ballot_sync(0xffffffffu, cls == 0);
        int rank = __popc((cls == 1 ? m1 : m0) & lt);
        if (lane == 0) { wcnt[warp][0] = __popc(m0); wcnt[warp][1] = __popc(m1); }
        __syncthreads();
        if (threadIdx.x < 2) {
            int t = 0;
            for (int w = 0; w < kBinThreads / 32; ++w) t += wcnt[w][threadIdx.x];
            base[threadIdx.x] = t ? atomicAdd(&meta[1 + threadIdx.x], t) : 0;
        }
        __syncthreads();
        if (cls >= 0) {
            int off = base[cls];
            for (int w = 0; w < warp; ++w) off += wcnt[w][cls];
            idx[cls ? n - 1 - (off + rank) : off + rank] = i;
        }
        __syncthreads();
    }
}

template <bool kIndexed>
__global__ void __launch_bounds__(kThreads)
k_devroye_refill(double *__restrict__ x, const int *__restrict__ n, const double *__restrict__ z,
                 int64_t num, StreamId id, const int *__restrict__ idx, int chunk)
{
    BL_PDL_ENTER();
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int64_t warp = (int64_t)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
    const int64_t stride = (int64_t)gridDim.x * (kThreads / 32) * chunk;

    int64_t cur = warp * chunk;       // next unassigned observation of this warp (uniform)
    int64_t cend = cur + chunk;       // end of the current chunk (uniform)

    bool active = false;
    int64_t obs = 0;
    int remaining = 0;
    double sum = 0.0;
    DevSetup st;
    PhiloxSource src;

    for (;;) {
        unsigned want = __ballot_sync(full, !active);
        if (want && cur < num) {
            int rank = __popc(want & lt_mask);
            int64_t cand = cur + rank;
            if (cand >= cend) cand += stride - chunk;
            if (!active && cand < num) {
                if (kIndexed) cand = idx[cand];                  // position in the class-sorted list -> observation
                int ni = n[cand];
                if (ni == 0) {
                    x[cand] = 0.0;                    // LogitWrapper.cpp:76-79
                } else {
                    obs = cand;
                    remaining = ni < 1 ? 1 : ni;      // NTHROW clamp, PolyaGamma.cpp:128-135
                    sum = 0.0;
                    st = dev_setup(z[cand]);
                    if (id.chain_len) {
                        const uint32_t ch = (uint32_t)cand / id.chain_len;
                        src.open(id.seed + ch, id.obs0 + ((uint32_t)cand - ch * id.chain_len), id.call_id);
                    } else {
                        src.open(id.seed, id.obs0 + (uint64_t)cand, id.call_id);
                    }
                    active = true;
                }
            }
            cur += __popc(want);
            if (cur >= cend) {
                int64_t over = cur - cend;
                cend += stride;
                cur = cend - chunk + over;
            }
        }
        if (!__any_sync(full, active)) {
            if (cur >= num) break;
            continue;
        }
        if (active) {
            double X;
            if (dev_propose(src, st, X)) {
                sum += 0.25 * X;
                if (--remaining == 0) {
                    x[obs] = sum;
                    active = false;
                }
            }
        }
    }
}


// ---------------------------------------------------------------------------------------------
// PG(1,z) / sum of PG(1) with CTA-level regrouping by proposal piece (large batches).
//
// In k_devroye_refill a lane owns a draw, and every trip of a warp runs all the proposal pieces its
// 32 lanes happen to need -- the right piece (about half of the proposals for z ~ U(-5,5)) and one or
// both left pieces -- one after the other: 9-18 of 32 lanes were active in the average instruction.
// Here draws live in SLOTS in shared memory (Z, the fp32 right-mass estimate, the Philox position, the
// running sum of a Sigma PG(1) draw) and any thread can advance any slot.  Every trip the CTA
//   (i)   refills empty slots (each warp from its own chunks of the batch; set-up, first U_mix -> piece),
//   (ii)  sorts the live slots by the piece of their pending proposal: ballot ranks + a prefix over the
//         warps; piece 1 from the front of `perm`, piece 3 right behind it, piece 2 from the back,
//   (iii) lets thread t run the proposal of slot perm[t], the series test, and -- accepted or not -- the
//         U_mix that decides the piece of the slot's next proposal.
// All warps but the (at most two) on a boundary then run one piece.  Variates are consumed per draw in the
// reference's order, from the stream keyed by the draw's global index: results are bit-identical to
// k_devroye_refill and to the per-lane loops (test_devroye_regroup_equals_refill).
// ---------------------------------------------------------------------------------------------
constexpr int kDrThreads = 256;
constexpr int kDrChunk = 128;

struct DrSlots {
    double Z[kDrThreads];
    double sum[kDrThreads];
    uint4 buf[kDrThreads];
    uint32_t blk[kDrThreads];
    float pr32[kDrThreads];
    int pos[kDrThreads];
    int obs[kDrThreads];
    int remaining[kDrThreads];
    int phase[kDrThreads];                     // -1 empty, else the pending piece (1, 2, 3)
    int perm[kDrThreads];
    int wcnt[kDrThreads / 32][3];
};

__global__ void __launch_bounds__(kDrThreads)
k_devroye_regroup(double *__restrict__ x, const int *__restrict__ n, const double *__restrict__ z, int num, StreamId id)
{
    __shared__ DrSlots S;
    const unsigned full = 0xffffffffu;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    constexpr int kWarps = kDrThreads / 32;
    const int gwarp = blockIdx.x * kWarps + warp;
    const long long stride = (long long)gridDim.x * kWarps * kDrChunk;
    long long cur = (long long)gwarp * kDrChunk, cend = cur + kDrChunk;

    S.phase[t] = -1;
    __syncthreads();
    for (;;) {
        // (i) refill this warp's empty home slots from its chunk
        const bool empty = S.phase[t] < 0;
        const unsigned want = __ballot_sync(full, empty);
        if (want && cur < num) {
            const int rank = __popc(want & lt_mask);
            long long cand = cur + rank;
            if (cand >= cend) cand += stride - kDrChunk;
            if (empty && cand < num) {
                const int obs = (int)cand;
                const int ni = n[obs];
                if (ni == 0) {
                    x[obs] = 0.0;                                    // LogitWrapper.cpp:76-79
                } else {
                    DevSetup st = dev_setup(z[obs]);
                    PhiloxSource src;
                    open_batch_stream(src, id, obs);
                    S.phase[t] = dev_pick(src, st);
                    S.Z[t] = st.Z;
                    S.pr32[t] = st.pr32;
                    S.sum[t] = 0.0;
                    S.remaining[t] = ni < 1 ? 1 : ni;                // NTHROW clamp, PolyaGamma.cpp:128-135
                    S.obs[t] = obs;
                    S.buf[t] = src.buf;
                    S.blk[t] = src.blk;
                    S.pos[t] = src.pos;
                }
            }
            cur += __popc(want);
            if (cur >= cend) {
                const long long over = cur - cend;
                cend += stride;
                cur = cend - kDrChunk + over;
            }
        }
        // (ii) sort live slots by piece
        const int ph = S.phase[t];
        const unsigned m1 = __ballot_sync(full, ph == 1), m2 = __ballot_sync(full, ph == 2), m3 = __ballot_sync(full, ph == 3);
        if (lane == 0) { S.wcnt[warp][0] = __popc(m1); S.wcnt[warp][1] = __popc(m2); S.wcnt[warp][2] = __popc(m3); }
        __syncthreads();
        int tot1 = 0, tot2 = 0, tot3 = 0, b1 = 0, b2 = 0, b3 = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
            const int a = S.wcnt[w][0], b = S.wcnt[w][1], c = S.wcnt[w][2];
            if (w < warp) { b1 += a; b2 += b; b3 += c; }
            tot1 += a;
            tot2 += b;
            tot3 += c;
        }
        if (tot1 + tot2 + tot3 == 0) {
            if (!__syncthreads_or(cur < num)) break;                    // nothing live, nothing left anywhere
            continue;
        }
        if (ph == 1) S.perm[b1 + __popc(m1 & lt_mask)] = t;
        else if (ph == 3) S.perm[tot1 + b3 + __popc(m3 & lt_mask)] = t;
        else if (ph == 2) S.perm[kDrThreads - 1 - (b2 + __popc(m2 & lt_mask))] = t;
        __syncthreads();
        // (iii) thread t advances slot perm[t] by one proposal
        if (t < tot1 + tot3 || t >= kDrThreads - tot2) {
            const int sl = S.perm[t];
            const int obs = S.obs[sl];
            PhiloxSource src;
            open_batch_stream(src, id, obs);
            src.buf = S.buf[sl];
            src.blk = S.blk[sl];
            src.pos = S.pos[sl];
            DevSetup st;
            st.Z = S.Z[sl];
            st.fz = dev_fz(st.Z);
            st.pr32 = S.pr32[sl];
            st.pr64 = nan("");
            const int piece = S.phase[sl];
            double X;
            if (piece == 1) X = dev_piece_right(src, st);
            else if (piece == 2) X = dev_piece_pair(src, st);
            else X = dev_piece_ig(src, st);
            bool done = false;
            if (dev_series_test(X, src.unif())) {
                const double sum = S.sum[sl] + 0.25 * X;
                if (--S.remaining[sl] == 0) {
                    x[obs] = sum;
                    S.phase[sl] = -1;
                    done = true;
                } else {
                    S.sum[sl] = sum;
                }
            }
            if (!done) {
                S.phase[sl] = dev_pick(src, st);                        // piece of the next proposal
                S.buf[sl] = src.buf;
                S.blk[sl] = src.blk;
                S.pos[sl] = src.pos;
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// Fused sweep half-step of the logit samplers: psi_i = x_i . beta and omega_i = PG(n_i, psi_i) in one
// pass over X (Logit.hpp:421,431 then Logit::draw_w :283-289; the two statements are adjacent in
// gibbs_block and psi has no other reader).  Separately the two kernels are bound by different
// things -- k_xbeta_mma by HBM (N P 8 bytes, 18 % of the issue slots), the draw by the issue slots
// (16 bytes per row of HBM) -- so one kernel whose warps alternate between the two phases lets some
// warps' row loads fly while others draw.
//   trip  : a warp takes 32 consecutive rows.  psi exactly as k_xbeta_mma forms it (same fragment
//           layout, same MMA order: the bits of psi are those of the two-kernel path): lane
//           (gid, tig) loads X[i0 + 8 rb + gid][c0 + 2 tig, +1], every column of accumulator rb
//           holds psi of rows i0 + 8 rb + 0..7.
//   hand-over: lane l takes row i0 + l = accumulator l >> 3, row-in-tile l & 7, read from lane
//           (l & 7) << 2 by four shuffles.
//   draw  : the per-lane Devroye loop of the refill kernel (dev_propose), stream keyed by the global
//           observation index; PG(1, z) accepts 99.9 % of its first proposals, so the refill
//           machinery of k_devroye_refill buys nothing here -- lanes differ by proposal branch only.
// Chains: rows [c N, (c+1) N) meet beta + c * beta_stride and the streams of seed + c (trips never
// straddle two chains).  psi_out may be null.
// kOffset (the random-intercept logit): omega_i = PG(n_i, x_i . beta + off_i) and psi_out keeps x_i . beta.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void dmma884_f(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// The products of one 32-row trip, in k_xbeta_mma's fragment layout and MMA order: lane (gid, tig) feeds
// A = X[i0 + 8 rb + gid][c0 + 2 tig, +1] (base points at column 2 tig of row i0 + gid) and B[tig][gid] =
// bc[c0], bc[c0 + 1] (bc points at entry 2 tig of the beta of column gid; bv false: that column is zero).
// c[rb] then holds C[8 rb + gid][2 tig, +1] = row i0 + 8 rb + gid times the beta of columns 2 tig, 2 tig + 1.
__device__ __forceinline__ void psi_trip(double (&c)[4][2], const double *base, const double *bc, bool bv,
                                         const bool (&rv)[4], int P, int tig)
{
#pragma unroll 2
    for (int c0 = 0; c0 < P; c0 += 8) {
        const bool cv = c0 + 2 * tig < P;
        double2 a[4];
#pragma unroll
        for (int rb = 0; rb < 4; ++rb)
            a[rb] = (cv && rv[rb]) ? __ldg(reinterpret_cast<const double2 *>(base + (size_t)(8 * rb) * P + c0))
                                   : make_double2(0.0, 0.0);
        const bool bl = cv && bv;
        const double b0 = bl ? __ldg(bc + c0) : 0.0, b1 = bl ? __ldg(bc + c0 + 1) : 0.0;
#pragma unroll
        for (int rb = 0; rb < 4; ++rb) {
            dmma884_f(c[rb][0], c[rb][1], a[rb].x, b0);
            dmma884_f(c[rb][0], c[rb][1], a[rb].y, b1);
        }
    }
}

// omega = PG(n_i, z) as the sum of n_i PG(1, z) draws from the stream (seed, obs, call); n_i = 0 gives 0
// (LogitWrapper.cpp:76-79).  PG(1, z) accepts 99.9 % of its first proposals, so a lane loops on its own.
__device__ __forceinline__ double logit_omega(int ni, double z, uint64_t seed, uint64_t obs, uint32_t call)
{
    if (ni == 0) return 0.0;
    int remaining = ni < 1 ? 1 : ni;                                 // NTHROW clamp, PolyaGamma.cpp:128-135
    DevSetup st = dev_setup(z);
    PhiloxSource src;
    src.open(seed, obs, call);
    double sum = 0.0;
    do {
        double X;
        while (!dev_propose(src, st, X)) {}
        sum += 0.25 * X;
    } while (--remaining);
    return sum;
}

template <bool kOffset>
__global__ void __launch_bounds__(kThreads, 3)
k_logit_psi_draw(double *__restrict__ x, double *__restrict__ psi_out, const int *__restrict__ n,
                 const double *__restrict__ tX, const double *__restrict__ beta, int64_t beta_stride,
                 int chains, int64_t N, int P, StreamId id, const double *__restrict__ off)
{
    BL_PDL_ENTER();
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
    const int64_t tpc = (N + 31) >> 5;                               // 32-row trips per chain
    const int64_t trips = (int64_t)chains * tpc;
    const int64_t warps = (int64_t)gridDim.x * (kThreads >> 5);
    const int64_t wid = (int64_t)blockIdx.x * (kThreads >> 5) + (threadIdx.x >> 5);
    for (int64_t trip = wid; trip < trips; trip += warps) {
        const int64_t ch = chains > 1 ? trip / tpc : 0;
        const int64_t i0 = (trip - ch * tpc) << 5;
        const double *bc = beta + ch * beta_stride + 2 * tig;
        const double *base = tX + ((size_t)ch * N + i0 + gid) * P + 2 * tig;
        double c[4][2] = {};
        bool rv[4];
#pragma unroll
        for (int rb = 0; rb < 4; ++rb) rv[rb] = i0 + 8 * rb + gid < N;
        psi_trip(c, base, bc, true, rv, P, tig);
        double z = 0.0;
#pragma unroll
        for (int rb = 0; rb < 4; ++rb) {
            const double t = __shfl_sync(full, c[rb][0], (lane & 7) << 2);
            if ((lane >> 3) == rb) z = t;
        }
        const int64_t i = i0 + lane;
        if (i < N) {
            const int64_t g = ch * N + i;
            if (psi_out) psi_out[g] = z;
            if (kOffset) z += off[g];
            x[g] = logit_omega(n[g], z, id.chain_len ? id.seed + (uint64_t)ch : id.seed, id.obs0 + (uint64_t)i, id.call_id);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// The same half-step for `chains` chains on ONE set of rows (bl_logit_multichain): the chains multiply the
// same X and differ only in beta and in their streams, so the B operand that k_logit_psi_draw fills with one
// beta in all 8 columns carries 8 chains' betas instead -- lane (gid, tig) feeds B[tig][gid] = beta of chain
// g0 + gid -- and one read of X gives column k of every accumulator tile = psi of chain g0 + k.  More than 8
// chains: further passes over the trip's rows, 8 chains each.
//   hand-over: the warp's 32 x 8 psi tile goes through shared memory, and lane l draws row i0 + l for each
//           chain of the group in turn.  Every lane carries one draw per chain -- with fewer than 8 chains no
//           lane waits through the draws of others while holding only padding columns.
//   draw  : logit_omega, stream (seed + c, obs0 + i, call) as the replicated batch keys it, so chain c is
//           bit for bit the chain k_logit_psi_draw runs on a private copy of the rows (the MMA forms each
//           output element from its own row and column only).
// omega: [chains][N].
// ---------------------------------------------------------------------------------------------
constexpr int kGroup = 8;                       // chains per pass: the 8 columns of an m8n8k4 tile
constexpr int kTileLd = kGroup + 1;             // odd row stride: lane l reading row l is conflict-free

__global__ void __launch_bounds__(kThreads, 3)
k_logit_psi_draw_shared(double *__restrict__ x, const int *__restrict__ n, const double *__restrict__ tX,
                        const double *__restrict__ beta, int64_t beta_stride, int chains, int64_t N, int P, StreamId id)
{
    BL_PDL_ENTER();
    __shared__ double tile[kThreads / 32][32 * kTileLd];
    const int lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
    double *pt = tile[threadIdx.x >> 5];
    const int groups = (chains + kGroup - 1) / kGroup;
    // work item = (trip, group of 8 chains), the groups of a trip on neighbouring warps: little state lives
    // across the draws (80 registers), and the repeat reads of a trip's rows meet each other in L1 / L2
    const int64_t items = ((N + 31) >> 5) * groups;
    const int64_t warps = (int64_t)gridDim.x * (kThreads >> 5);
    const int64_t wid = (int64_t)blockIdx.x * (kThreads >> 5) + (threadIdx.x >> 5);
    for (int64_t item = wid; item < items; item += warps) {
        const int64_t trip = groups > 1 ? item / groups : item;
        const int g0 = (int)(item - trip * groups) * kGroup, kg = min(kGroup, chains - g0);
        const int64_t i0 = trip << 5, i = i0 + lane;
        bool rv[4];
#pragma unroll
        for (int rb = 0; rb < 4; ++rb) rv[rb] = i0 + 8 * rb + gid < N;
        double c[4][2] = {};
        psi_trip(c, tX + (i0 + gid) * P + 2 * tig, beta + (int64_t)(g0 + min(gid, kg - 1)) * beta_stride + 2 * tig,
                 gid < kg, rv, P, tig);
        __syncwarp();                                                // the previous item's reads of the tile are done
#pragma unroll
        for (int rb = 0; rb < 4; ++rb) {
            pt[(8 * rb + gid) * kTileLd + 2 * tig] = c[rb][0];
            pt[(8 * rb + gid) * kTileLd + 2 * tig + 1] = c[rb][1];
        }
        __syncwarp();
        if (i < N) {
            const int ni = n[i];
            for (int k = 0; k < kg; ++k)
                x[(int64_t)(g0 + k) * N + i] = logit_omega(ni, pt[lane * kTileLd + k], id.seed + (uint64_t)(g0 + k),
                                                           id.obs0 + (uint64_t)i, id.call_id);
        }
    }
}

}  // namespace

bool devroye_binned(int64_t num, int64_t bin_min_arg)
{
    static const int64_t bin_env = getenv("BL_DEVROYE_BIN_MIN") ? atoll(getenv("BL_DEVROYE_BIN_MIN")) : -1;
    const int64_t bin_min = bin_env >= 0 ? bin_env : bin_min_arg;
    return !getenv("BL_DEVROYE_REGROUP") && num >= bin_min && num < (1LL << 31);
}

cudaError_t launch_devroye_refill(double *x, const int *n, const double *z, int64_t num,
                                  StreamId id, cudaStream_t st, void *work, int64_t bin_min_arg, bool prebinned)
{
    if (num <= 0) return cudaSuccess;
    int64_t cap = 148LL * 4;                 // 148 SMs x resident CTAs
    // Chunks are dealt round-robin to warps; a warp should see at least ~8 of them or the last
    // round leaves part of the chip idle (N = 1M rows of a Gibbs sweep is only 1.65 chunks of 128
    // per resident warp).
    int chunk = num >= cap * (kThreads / 32) * kChunkObs * 8 ? kChunkObs : kChunkObs / 4;
    int64_t chunks = (num + chunk - 1) / chunk;
    int64_t blocks = (chunks + (kThreads / 32) - 1) / (kThreads / 32);
    int grid = (int)(blocks < cap ? blocks : cap);
    // BL_DEVROYE_REGROUP=1: slots regrouped by proposal piece across the CTA (k_devroye_regroup) -- bit-identical
    // results, but measured SLOWER than the per-lane kernel (1.14e10 against 1.26e10 draws/s at 2^27 draws; 113 us
    // against 105 us for the 1M draws of a Gibbs sweep): a PG(1,z) proposal is ~150 instructions, and the two
    // CTA barriers, the slot traffic and the wait for the slowest warp of every trip cost more than the
    // divergence they remove.  Kept as a measured alternative, not the default.
    const bool regroup = getenv("BL_DEVROYE_REGROUP") != nullptr;
    static const int64_t bin_env = getenv("BL_DEVROYE_BIN_MIN") ? atoll(getenv("BL_DEVROYE_BIN_MIN")) : -1;
    const int64_t bin_min = bin_env >= 0 ? bin_env : bin_min_arg;
    if (regroup && num >= (1 << 15) && num < (1LL << 31)) {
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_devroye_regroup, kDrThreads, 0) != cudaSuccess || per_sm < 1)
            per_sm = 1;
        const int64_t want = (num + kDrThreads - 1) / kDrThreads;
        const int rgrid = (int)std::min<int64_t>(148LL * per_sm, std::max<int64_t>(1, want));
        k_devroye_regroup<<<rgrid, kDrThreads, 0, st>>>(x, n, z, (int)num, id);
        count_launch();
    } else if (work && num >= bin_min && num < (1LL << 31)) {
        int *meta = (int *)work, *idx = meta + 32;
        if (!prebinned) {
            cudaError_t e = cudaMemsetAsync(meta, 0, 32 * sizeof(int), st);
            if (e != cudaSuccess) return e;
            int tiles = (int)((num + kBinThreads - 1) / kBinThreads);
            int bgrid = tiles < 148 * 8 ? tiles : 148 * 8;
            launch_pdl(k_cls_scatter, dim3(bgrid), dim3(kBinThreads), 0, st, z, (int)num, meta, idx);
            count_launch();
        }
        launch_pdl(k_devroye_refill<true>, dim3(grid), dim3(kThreads), 0, st, x, n, z, num, id, (const int *)idx, chunk);
        count_launch();
    } else {
        launch_pdl(k_devroye_refill<false>, dim3(grid), dim3(kThreads), 0, st, x, n, z, num, id, (const int *)nullptr, chunk);
        count_launch();
    }
    return cudaGetLastError();
}

}  // namespace bl

namespace bl {

bool logit_psi_draw_ok(const double *tX, int P) { return P % 2 == 0 && (reinterpret_cast<uintptr_t>(tX) & 15) == 0; }

// omega (and psi, when psi_out is given) for `chains` blocks of N rows each; see k_logit_psi_draw.
cudaError_t launch_logit_psi_draw(double *x, double *psi_out, const int *n, const double *tX, const double *beta,
                                  int64_t beta_stride, int chains, int64_t N, int P, StreamId id, cudaStream_t st,
                                  const double *off)
{
    if (N <= 0 || chains <= 0) return cudaSuccess;
    const int64_t trips = (int64_t)chains * ((N + 31) / 32);
    const int wpc = kThreads / 32;
    // three CTAs of 80 registers per SM: with 128 registers (the 16 loads of k_xbeta_mma in flight per
    // lane) only 16 warps are resident and the draw phases of some warps do not cover the load phases of
    // the others -- 189 us against 105 + 86 for the two kernels at N = 1M, P = 64; with 8 loads in flight
    // and 24 warps 172 us (P = 32: 104 against 122; P = 128: 252 against 281).
    int grid = (int)std::min<int64_t>(148 * 3, std::max<int64_t>(1, (trips + wpc - 1) / wpc));
    if (off)
        launch_pdl(k_logit_psi_draw<true>, dim3(grid), dim3(kThreads), 0, st, x, psi_out, n, tX, beta, beta_stride, chains, N, P, id, off);
    else
        launch_pdl(k_logit_psi_draw<false>, dim3(grid), dim3(kThreads), 0, st, x, psi_out, n, tX, beta, beta_stride, chains, N, P, id, off);
    count_launch();
    return cudaGetLastError();
}

// omega of `chains` chains on one set of N rows; see k_logit_psi_draw_shared.
cudaError_t launch_logit_psi_draw_shared(double *x, const int *n, const double *tX, const double *beta,
                                         int64_t beta_stride, int chains, int64_t N, int P, StreamId id, cudaStream_t st)
{
    if (N <= 0 || chains <= 0) return cudaSuccess;
    const int64_t items = (N + 31) / 32 * ((chains + kGroup - 1) / kGroup);
    const int wpc = kThreads / 32;
    // the occupancy of k_logit_psi_draw (three CTAs of 80 registers per SM)
    int grid = (int)std::min<int64_t>(148 * 3, std::max<int64_t>(1, (items + wpc - 1) / wpc));
    launch_pdl(k_logit_psi_draw_shared, dim3(grid), dim3(kThreads), 0, st, x, n, tX, beta, beta_stride, chains, N, P, id);
    count_launch();
    return cudaGetLastError();
}

}  // namespace bl
