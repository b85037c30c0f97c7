// Device kernels of the Gibbs sweeps that consume PG draws.
//
// Reference statements (all fp64):
//   psi = X beta                    Logit.hpp:421,431; MultLogit.hpp:277,307     (gemm 'T')
//   X' Omega X (+ P0)               Logit.hpp:293-301, :325-332; MultLogit.hpp:246-248,252
//   X' v                            Logit.hpp:174-183 (kappa), MultLogit.hpp:249,253 (Omega c_j),
//                                   NBPG-logmean.R:28 (kappa + omega log d)
//   c_j = log sum_{k != j} exp(XB_k), eta_j = XB_j - c_j      MultLogit.hpp:288,293-299,313
//   beta draws                      Logit.hpp:291-320 (plain), :322-400 (constrained, the one
//                                   called), Normal.hpp:98-131 (mlogit)
//
// Data layout in HBM: tX is P x N column-major exactly as R hands it over
// (LogitWrapper.R:226), i.e. observation i's P covariates are contiguous at
// tX[i*P .. i*P+P): every pass below streams X once, row by row, fully coalesced.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>

#include "philox.cuh"
#include "specfun.cuh"

namespace bl {

// ---------------------------------------------------------------------------------
// psi_i = x_i . beta (+ off_i).  A warp takes 32 consecutive rows per trip; lanes stride the
// columns (every load is a coalesced 256 B row segment), each lane keeps one partial sum per row,
// and the 32 x 32 partials are folded by a transposing butterfly (31 shuffle-adds per lane for 32
// rows, lane r ending up with row r) instead of a 5-step butterfly per row -- the per-row form
// spent 66 warp instructions per row and ran at 4.3 TB/s with the LSU and ALU pipes half busy.
// HBM-bound: N P 8 bytes.
// Several chains on shared rows (bl_nb_multichain, odd P or unaligned X): blockIdx.y = chain c, which meets
// beta + c beta_stride and writes psi + c N (off is read at + c N); every row sums in the single chain's order.
// ---------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256, 2)
k_xbeta(double *__restrict__ psi, const double *__restrict__ tX, const double *__restrict__ beta,
        const double *__restrict__ off, double off_scale, double shift, int64_t N, int P, int64_t beta_stride = 0)
{
    beta += blockIdx.y * beta_stride;
    psi += blockIdx.y * N;
    if (off) off += blockIdx.y * N;
    extern __shared__ __align__(16) double sbeta[];
    for (int p = threadIdx.x; p < P; p += blockDim.x) sbeta[p] = beta[p];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int64_t wid = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    for (int64_t i0 = wid * 32; i0 < N; i0 += warps * 32) {
        double acc[32];
#pragma unroll
        for (int r = 0; r < 32; ++r) acc[r] = 0.0;
        const bool whole = i0 + 32 <= N;
        for (int p = lane; p < P; p += 32) {
            const double bp = sbeta[p];
            const double *col = tX + i0 * P + p;
            if (whole) {
#pragma unroll
                for (int r = 0; r < 32; ++r) acc[r] = fma(__ldg(col + (int64_t)r * P), bp, acc[r]);
            } else {
#pragma unroll
                for (int r = 0; r < 32; ++r)
                    if (i0 + r < N) acc[r] = fma(__ldg(col + (int64_t)r * P), bp, acc[r]);
            }
        }
        // transposing butterfly: after the stage with offset o a lane holds the rows whose bit o
        // equals its own lane bit o
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
            const bool up = (lane & o) != 0;
#pragma unroll
            for (int k = 0; k < o; ++k) {
                double send = up ? acc[k] : acc[k + o];
                double keep = up ? acc[k + o] : acc[k];
                acc[k] = keep + __shfl_xor_sync(0xffffffffu, send, o);
            }
        }
        const int64_t i = i0 + lane;
        if (i < N) psi[i] = (off ? acc[0] + off_scale * off[i] : acc[0]) + shift;
    }
}

// The same for a batch of independent chains: chain c reads the N rows at tX + c * x_stride (N P: its own
// rows; 0: rows shared by all chains), meets beta_c = beta[c * beta_stride ..) and writes psi[c psi_stride ..)
// (N: chains side by side; U N: category j of a multinomial chain's [U][N] linear predictors).
// Trips of 32 rows never straddle two chains.
static __global__ void __launch_bounds__(256, 2)
k_xbeta_chains(double *__restrict__ psi, int64_t psi_stride, const double *__restrict__ tX, int64_t x_stride,
               const double *__restrict__ beta, int64_t beta_stride, int chains, int N, int P)
{
    const int lane = threadIdx.x & 31;
    const int tpc = (N + 31) >> 5;                                   // trips per chain
    const int64_t trips = (int64_t)chains * tpc;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int64_t wid = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    for (int64_t trip = wid; trip < trips; trip += warps) {
        const int ch = (int)(trip / tpc);
        const int i0 = (int)(trip - (int64_t)ch * tpc) << 5;
        const double *bc = beta + ch * beta_stride;
        const double *base = tX + ch * x_stride + (size_t)i0 * P;
        double acc[32];
#pragma unroll
        for (int r = 0; r < 32; ++r) acc[r] = 0.0;
        const bool whole = i0 + 32 <= N;
        for (int p = lane; p < P; p += 32) {
            const double bp = __ldg(bc + p);
            const double *col = base + p;
            if (whole) {
#pragma unroll
                for (int r = 0; r < 32; ++r) acc[r] = fma(__ldg(col + (int64_t)r * P), bp, acc[r]);
            } else {
#pragma unroll
                for (int r = 0; r < 32; ++r)
                    if (i0 + r < N) acc[r] = fma(__ldg(col + (int64_t)r * P), bp, acc[r]);
            }
        }
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
            const bool up = (lane & o) != 0;
#pragma unroll
            for (int k = 0; k < o; ++k) {
                double send = up ? acc[k] : acc[k + o];
                double keep = up ? acc[k + o] : acc[k];
                acc[k] = keep + __shfl_xor_sync(0xffffffffu, send, o);
            }
        }
        if (i0 + lane < N) psi[ch * psi_stride + i0 + lane] = acc[0];
    }
}

// ---------------------------------------------------------------------------------
// Weighted Gram, SYRK-shaped: G = sum_i w_i x_i x_i' over a slab of rows.
//
// Grid: blockIdx.y = output tile (bi, bj), bi <= bj, of 64 x 64; blockIdx.x = row slab.
// Row chunks of kGramRows rows (and their weights) stream HBM -> shared memory with cp.async
// (LDGSTS) through a three-stage ring -- two chunks in flight while one is multiplied, one
// barrier per chunk; the weight is folded into the row operand as it is read
// (w x_i) x_j', cf. MultLogit.hpp:246-248; Logit.hpp:325-332 scales by sqrt(w) instead).
// Compute: a 16 x 16 thread grid of 4 x 4 register tiles, thread (ty, tx) owning rows
// {ty + 16p} and columns {tx + 16q} (shared-memory reads are then conflict-free: lanes
// read consecutive doubles / broadcast).  On a diagonal tile thread (tx, ty) would only
// recompute the transpose of thread (ty, tx), so just the 136 threads with ty <= tx --
// packed into the first 4.25 warps -- run (P <= 64 launches 160-thread CTAs: no idle warps):
// the symmetry really frees FP64 issue slots.
// Per-CTA partial tiles go to `part`; k_gram_reduce sums them in a fixed order
// (deterministic, no atomics).  Bound by the FP64 pipe: ~N P^2 (1 + 1/16) FMA.
// ---------------------------------------------------------------------------------
constexpr int kGramRows = 32;       // rows per chunk when a CTA streams two column panels (P > 64)
constexpr int kGramRowsDiag = 64;   // P <= 64: one panel per chunk, so twice the rows fit and barriers halve
constexpr int kGramTile = 64;
constexpr int kGramLd = kGramTile;          // dense rows: column reads are lane-consecutive

__device__ __forceinline__ void cp_async8(double *smem_dst, const double *gsrc, bool valid)
{
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    int sz = valid ? 8 : 0;                 // src-size 0 -> zero fill
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(d), "l"(gsrc), "r"(sz));
}
__device__ __forceinline__ void cp_async16(double *smem_dst, const double *gsrc, bool valid)
{
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    int sz = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(gsrc), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

constexpr int kGramStages = 3;
constexpr int kGramLdm = 68;     // leading dimension (doubles): == 4 mod 16 -> conflict-free DMMA fragment loads

// D(8x8) += A(8x4) * B(4x8), fp64 tensor-core MMA.  Lane l: gid = l>>2, tig = l&3;
// a = A[gid][tig], b = B[tig][gid], c0/c1 = C[gid][2 tig], C[gid][2 tig + 1].
__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// ---------------------------------------------------------------------------------
// psi = X beta on the FP64 tensor cores, for even P and 16-byte aligned tX (else k_xbeta).
// The matrix-vector product is issued as m8n8k4 MMAs whose B operand repeats beta in every column:
// lane (gid, tig) loads the 16 bytes X[row0 + gid][c0 + 2 tig, +1] (four lanes cover 64 contiguous
// bytes of a row: full 32-byte sectors) and feeds them as the A fragments of two MMAs against
// beta[c0 + 2 tig] and beta[c0 + 2 tig + 1]; every column of the 8 x 8 accumulator then holds psi
// of the 8 rows.  No cross-lane reduction and two accumulator registers per 8 rows, so a warp
// keeps a whole 32-row trip of loads in flight; the lane-strided k_xbeta spends ~150 of its ~220
// instructions per trip in the transposing butterfly and idles HBM meanwhile (4.6 TB/s at P = 64,
// 2.4 TB/s at P = 32).  Chains: the N rows at tX + c * x_stride meet beta + c * beta_stride, psi goes to
// [c psi_stride ..) (off is read at [c N ..)).
// ---------------------------------------------------------------------------------
// mlogit epilogue (MultLogit.hpp:246-258, 275-277): the category whose coefficients were just drawn gets its new
// linear predictor XB_j = X beta_j and E_j = exp(XB_j) (cached so that no category's exponentials are recomputed
// until its own beta changes); the NEXT category jn gets its offset c = log(sum_{k != jn} E_k + 1) -- same
// summation order as k_mlogit_offsets, same exp() of the same numbers, same bits -- and eta = XB_jn - c.  One
// pass over X replaces the psi kernel and the offsets kernel of every category update.
constexpr int kMlogitMaxU = 16;       // categories - 1 the fused pass keeps in registers (more: the separate kernels)
struct MlogitNext {
    double *E;              // [N x U] exp(XB), column-major
    const double *XB;       // [N x U]
    double *c, *eta;        // [N] offset and PG tilt of category jn
    int U, j, jn;
    int *bin_meta, *bin_idx;   // optional: the next draw's rows ordered by branch class (two cursors + index list, as
                               // k_cls_scatter leaves them) -- the tilt is in a register here, so the ordering costs two
                               // shared cursors' atomics per 32 rows instead of a pass over eta
};

// The loads of the epilogue that do not depend on the new product: row i's exponentials of the categories other
// than j and jn, and XB_jn (zero for rows past N).
__device__ __forceinline__ void mlogit_next_load(double (&ek)[kMlogitMaxU], double &xbn, const MlogitNext &mn,
                                                 int64_t i, int64_t N)
{
#pragma unroll
    for (int k = 0; k < kMlogitMaxU; ++k)
        ek[k] = (k < mn.U && k != mn.j && k != mn.jn && i < N) ? __ldcg(mn.E + i + (size_t)N * k) : 0.0;
    xbn = 0.0;
    if (mn.jn != mn.j && i < N) xbn = __ldcg(mn.XB + i + (size_t)N * mn.jn);
}

// The epilogue of one row per lane, called by the whole warp: row i (< N) gets XB_j = xb (at psi[i]), E_j = exp(xb),
// the next category's offset c and tilt eta; with mn.bin_idx the warp's rows then enter the next draw's class-ordered
// index list of `total` entries as the values gi (class 0 from the front, class 1 from the back, one atomic per class).
__device__ __forceinline__ void mlogit_next_epilogue(double *psi, const MlogitNext &mn, double xb,
                                                     const double (&ek)[kMlogitMaxU], double xbn, int64_t i, int64_t N,
                                                     int gi, int total, int lane)
{
    int cls = -1;
    if (i < N) {
        psi[i] = xb;
        const double ej = exp(xb);
        mn.E[i + (size_t)N * mn.j] = ej;
        double A = 0.0;
#pragma unroll
        for (int k = 0; k < kMlogitMaxU; ++k)
            if (k < mn.U && k != mn.jn) A += k == mn.j ? ej : ek[k];
        A += 1.0;
        const double cj = log(A);
        mn.c[i] = cj;
        const double et = (mn.jn == mn.j ? xb : xbn) - cj;
        mn.eta[i] = et;
        if (mn.bin_idx) cls = fabs(et) * 0.5 >= 1.0 / 0.64 ? 1 : 0;        // dev_class (pg_devroye_kernel.cu), kTrunc = 0.64
    }
    if (mn.bin_idx) {
        const unsigned m1 = __ballot_sync(0xffffffffu, cls == 1), m0 = __ballot_sync(0xffffffffu, cls == 0);
        int b0 = 0, b1 = 0;
        if (lane == 0) {
            if (m0) b0 = atomicAdd(&mn.bin_meta[1], __popc(m0));
            if (m1) b1 = atomicAdd(&mn.bin_meta[2], __popc(m1));
        }
        b0 = __shfl_sync(0xffffffffu, b0, 0);
        b1 = __shfl_sync(0xffffffffu, b1, 0);
        const unsigned lt = (1u << lane) - 1u;
        if (cls == 0) mn.bin_idx[b0 + __popc(m0 & lt)] = gi;
        else if (cls == 1) mn.bin_idx[total - 1 - (b1 + __popc(m1 & lt))] = gi;
    }
}

template <bool kMlogit>
static __global__ void __launch_bounds__(256, 2)
k_xbeta_mma(double *__restrict__ psi, int64_t psi_stride, const double *__restrict__ tX, int64_t x_stride,
            const double *__restrict__ beta, int64_t beta_stride, int chains, int64_t N, int P,
            const double *__restrict__ off, double off_scale, double shift, MlogitNext mn)
{
    BL_PDL_ENTER();
    const int lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
    const int64_t tpc = (N + 31) >> 5;                               // 32-row trips per chain
    const int64_t trips = (int64_t)chains * tpc;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int64_t wid = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    for (int64_t trip = wid; trip < trips; trip += warps) {
        const int64_t ch = chains > 1 ? trip / tpc : 0;
        const int64_t i0 = (trip - ch * tpc) << 5;
        const double *bc = beta + ch * beta_stride + 2 * tig;
        const double *base = tX + ch * x_stride + (i0 + gid) * P + 2 * tig;
        double c[4][2] = {};
        bool rv[4];
#pragma unroll
        for (int rb = 0; rb < 4; ++rb) rv[rb] = i0 + 8 * rb + gid < N;
        // mlogit: this lane's row is 8 tig + gid; the other categories' exponentials and the next category's
        // linear predictor do not depend on this trip's product -- their loads go out with the first loads of X
        double ek[kMlogitMaxU], xbn = 0.0;
        if (kMlogit) mlogit_next_load(ek, xbn, mn, i0 + 8 * tig + gid, N);
#pragma unroll 4
        for (int c0 = 0; c0 < P; c0 += 8) {
            const bool cv = c0 + 2 * tig < P;
            double2 a[4];
#pragma unroll
            for (int rb = 0; rb < 4; ++rb)
                a[rb] = (cv && rv[rb]) ? __ldg(reinterpret_cast<const double2 *>(base + (size_t)(8 * rb) * P + c0))
                                       : make_double2(0.0, 0.0);
            const double b0 = cv ? __ldg(bc + c0) : 0.0, b1 = cv ? __ldg(bc + c0 + 1) : 0.0;
#pragma unroll
            for (int rb = 0; rb < 4; ++rb) {
                dmma884(c[rb][0], c[rb][1], a[rb].x, b0);
                dmma884(c[rb][0], c[rb][1], a[rb].y, b1);
            }
        }
        if (kMlogit) {
            // every column of an accumulator tile holds psi of its 8 rows: lane (gid, tig) takes row 8 tig + gid
            const double xb = tig == 0 ? c[0][0] : tig == 1 ? c[1][0] : tig == 2 ? c[2][0] : c[3][0];
            const int64_t i = i0 + 8 * tig + gid;
            mlogit_next_epilogue(psi, mn, xb, ek, xbn, i, N, (int)i, (int)N, lane);
        } else if (tig == 0) {
#pragma unroll
            for (int rb = 0; rb < 4; ++rb) {
                const int64_t i = i0 + 8 * rb + gid;
                if (i < N) {
                    psi[ch * psi_stride + i] = (off ? c[rb][0] + off_scale * off[ch * N + i] : c[rb][0]) + shift;
                }
            }
        }
    }
}

inline bool xbeta_mma_ok(const double *tX, int P) { return P % 2 == 0 && (reinterpret_cast<uintptr_t>(tX) & 15) == 0; }

// ---------------------------------------------------------------------------------
// k_xbeta_mma<true> for `chains` multinomial chains on ONE set of rows (bl_mlogit_multichain).  The chains multiply
// the same X by their own beta_j, so the B operand that k_xbeta_mma fills with one beta in all 8 columns carries the
// beta_j of 8 chains instead -- lane (gid, tig) feeds B[tig][gid] = beta_j of chain g0 + gid -- and one read of X
// gives column k of every accumulator tile = XB_j of chain g0 + k (the MMA forms each output element from its own
// row and column only: the bits of the single chain's XB_j).  More than 8 chains: further passes over the trip's
// rows, 8 chains each, on neighbouring warps.
//   hand-over: the warp's 32 x 8 tile goes through shared memory; lane l then runs row i0 + l's epilogue
//           (mlogit_next_epilogue, the single chain's arithmetic) for each chain of the group in turn.
//   state : chain c's XB and E at [c][U][N] (XB is also where XB_j is written), its c and eta at mn.c / mn.eta +
//           c N.  The next draw's index list (optional) holds all chains * N (chain, row) pairs as c N + i.
// ---------------------------------------------------------------------------------
constexpr int kGroupChains = 8;                  // chains per pass: the 8 columns of an m8n8k4 tile
constexpr int kGroupTileLd = kGroupChains + 1;   // odd row stride: lane l reading row l is conflict-free

// The MMA trip of the shared-rows kernels, called by the whole warp: rows i0 .. i0 + 31 of X (P x N, even P, 16-byte
// aligned) times the beta of chains g0 .. g0 + kg - 1 (B column gid = chain g0 + gid; padding columns multiply zeros).
// Leaves the 32 x 8 product in the warp's tile pt (row r, chain g0 + k at r kGroupTileLd + k).
__device__ __forceinline__ void shared_rows_tile(double *pt, const double *__restrict__ tX, const double *__restrict__ beta,
                                                 int64_t beta_stride, int g0, int kg, int64_t i0, int64_t N, int P, int lane)
{
    const int gid = lane >> 2, tig = lane & 3;
    bool rv[4];
#pragma unroll
    for (int rb = 0; rb < 4; ++rb) rv[rb] = i0 + 8 * rb + gid < N;
    const double *base = tX + (i0 + gid) * P + 2 * tig;
    const double *bc = beta + (int64_t)(g0 + min(gid, kg - 1)) * beta_stride + 2 * tig;
    const bool bv = gid < kg;                                         // padding columns multiply zeros
    double c[4][2] = {};
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
            dmma884(c[rb][0], c[rb][1], a[rb].x, b0);
            dmma884(c[rb][0], c[rb][1], a[rb].y, b1);
        }
    }
    __syncwarp();                                                    // the previous item's reads of the tile are done
#pragma unroll
    for (int rb = 0; rb < 4; ++rb) {
        pt[(8 * rb + gid) * kGroupTileLd + 2 * tig] = c[rb][0];
        pt[(8 * rb + gid) * kGroupTileLd + 2 * tig + 1] = c[rb][1];
    }
    __syncwarp();
}

static __global__ void __launch_bounds__(256, 2)
k_mlogit_psi_shared(double *XB, const double *__restrict__ tX, const double *__restrict__ beta,
                    int64_t beta_stride, int chains, int64_t N, int P, MlogitNext mn)
{
    BL_PDL_ENTER();
    __shared__ double tile[8][32 * kGroupTileLd];
    const int lane = threadIdx.x & 31;
    double *pt = tile[threadIdx.x >> 5];
    const int groups = (chains + kGroupChains - 1) / kGroupChains;
    const int64_t UN = (int64_t)mn.U * N;
    const int64_t items = ((N + 31) >> 5) * groups;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int64_t wid = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    for (int64_t item = wid; item < items; item += warps) {
        const int64_t trip = groups > 1 ? item / groups : item;
        const int g0 = (int)(item - trip * groups) * kGroupChains, kg = min(kGroupChains, chains - g0);
        const int64_t i0 = trip << 5, i = i0 + lane;
        // the first chain's loads of the epilogue go out with the first loads of X
        MlogitNext m = mn;
        m.E += g0 * UN; m.XB += g0 * UN; m.c += g0 * N; m.eta += g0 * N;
        double ek[kMlogitMaxU], xbn;
        mlogit_next_load(ek, xbn, m, i, N);
        shared_rows_tile(pt, tX, beta, beta_stride, g0, kg, i0, N, P, lane);
        for (int k = 0; k < kg; ++k) {
            const int ch = g0 + k;
            // the next chain's loads are in flight while this chain's epilogue runs
            MlogitNext mnext = m;
            mnext.E += UN; mnext.XB += UN; mnext.c += N; mnext.eta += N;
            double en[kMlogitMaxU], xn;
            mlogit_next_load(en, xn, mnext, k + 1 < kg ? i : N, N);
            mlogit_next_epilogue(XB + ch * UN + (int64_t)mn.j * N, m, pt[lane * kGroupTileLd + k], ek, xbn, i, N,
                                 (int)(ch * N + i), (int)(chains * N), lane);
            m = mnext;
#pragma unroll
            for (int u = 0; u < kMlogitMaxU; ++u) ek[u] = en[u];
            xbn = xn;
        }
    }
}

// ---------------------------------------------------------------------------------
// psi = X beta + shift for `chains` chains on ONE set of rows (bl_nb_multichain; even P, 16-byte aligned X): the
// MMAs of k_xbeta_mma with the beta of 8 chains in the 8 B columns, so one read of X gives psi of 8 chains, each
// element formed from its own row and column only (the single chain's bits).  The warp's 32 x 8 tile goes through
// shared memory and lane l stores row i0 + l of each chain in turn: every chain's psi is written in 256-byte runs.
// Chain c meets beta + c beta_stride and writes psi + c N.  More than 8 chains: further groups of 8.
// ---------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256, 2)
k_xbeta_shared(double *__restrict__ psi, const double *__restrict__ tX, const double *__restrict__ beta,
               int64_t beta_stride, int chains, int64_t N, int P, double shift)
{
    BL_PDL_ENTER();
    __shared__ double tile[8][32 * kGroupTileLd];
    const int lane = threadIdx.x & 31;
    double *pt = tile[threadIdx.x >> 5];
    const int groups = (chains + kGroupChains - 1) / kGroupChains;
    const int64_t items = ((N + 31) >> 5) * groups;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int64_t wid = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    for (int64_t item = wid; item < items; item += warps) {
        const int64_t trip = groups > 1 ? item / groups : item;
        const int g0 = (int)(item - trip * groups) * kGroupChains, kg = min(kGroupChains, chains - g0);
        const int64_t i0 = trip << 5, i = i0 + lane;
        shared_rows_tile(pt, tX, beta, beta_stride, g0, kg, i0, N, P, lane);
        if (i < N)
            for (int k = 0; k < kg; ++k) psi[(g0 + k) * N + i] = pt[lane * kGroupTileLd + k] + shift;
    }
}

// Weighted Gram on the FP64 tensor cores (DMMA).  A register-tiled DFMA version of this kernel
// was bound by shared-memory bandwidth (LSU data pipe 75% busy, FP64 pipe 11%: every 16 FMAs
// cost 8 shared loads); an 8x8x4 MMA reuses each fragment element across a whole tile, so
// the same shared traffic feeds 8x the math.
//   grid  : blockIdx.y = 64x64 output tile (bi <= bj), blockIdx.x = row slab
//   CTA   : 8 warps = 2 row-groups x 4 sub-tiles of 32x32; each warp holds a 4x4 grid of
//           8x8 accumulator tiles.  On a diagonal tile the sub-tile below the diagonal and
//           the MMA tiles below the diagonal of the two diagonal sub-tiles are skipped.
//   smem  : three-stage cp.async ring of 32-row chunks of X (+ their weights); one barrier
//           per chunk; row group g multiplies rows [16g, 16g+16) of each chunk.
//   C = sum_r (w_r x_r[i]) x_r[j]: A[i][r] = w_r X[r][i] (weight folded into the A fragment),
//   B[r][j] = X[r][j].
// Diagonal 64x64 tile, balanced over the CTA's warps.  Its 36 live 8x8 MMA tiles (mi <= mj) are
// dealt to four warp slots as the row pairs (A, 7 - A): (8 - A) + (A + 1) = 9 tiles each, and the
// two row groups split the chunk's rows, so all 8 warps issue the same 9 DMMAs per k-step.  (With
// 32x32 sub-tiles per warp, one of four warps had nothing to do and one had 16 tiles against
// 10: the DMMA pipe idled 44 % of the time waiting at the chunk barrier.)
// c[0 .. 8-A): tiles (A, A..7); c[8-A .. 9): tiles (7-A, 7-A..7)
template <int A, int kRows>
__device__ __forceinline__ void gram_diag_chunk(double (&c)[9][2], const double *chunk, const double *wts,
                                                int grp, int gid, int tig)
{
    constexpr int kLo = 8 - A;
#pragma unroll
    for (int kk = 0; kk < kRows / 8; ++kk) {
        const int r = grp * (kRows / 2) + kk * 4 + tig;          // this lane's k row
        const double wr = wts[r];
        const double *row = chunk + r * kGramLdm + gid;
        double b[8];
#pragma unroll
        for (int j = A; j < 8; ++j) b[j] = row[8 * j];
        const double alo = b[A] * wr, ahi = b[7 - A] * wr;
#pragma unroll
        for (int j = A; j < 8; ++j) dmma884(c[j - A][0], c[j - A][1], alo, b[j]);
#pragma unroll
        for (int j = 7 - A; j < 8; ++j) dmma884(c[kLo + j - (7 - A)][0], c[kLo + j - (7 - A)][1], ahi, b[j]);
    }
}

template <int A>
__device__ __forceinline__ void gram_diag_store(const double (&c)[9][2], double *out, int gid, int tig)
{
    constexpr int kLo = 8 - A;
#pragma unroll
    for (int j = A; j < 8; ++j) {
        int row = 8 * A + gid, col = 8 * j + 2 * tig;
        out[row * kGramTile + col] = c[j - A][0];
        out[row * kGramTile + col + 1] = c[j - A][1];
    }
#pragma unroll
    for (int j = 7 - A; j < 8; ++j) {
        int row = 8 * (7 - A) + gid, col = 8 * j + 2 * tig;
        out[row * kGramTile + col] = c[kLo + j - (7 - A)][0];
        out[row * kGramTile + col + 1] = c[kLo + j - (7 - A)][1];
    }
}

// P == 32: two observations per 64-wide shared-memory row.  X (N x 32, row-major) read as an
// (N/2) x 64 matrix Y = [x_2r | x_2r+1] is the same bytes, so the chunks stream in dense; with the
// A fragment scaled by the even row's weight in columns 0..31 and the odd row's in 32..63,
// Y' W Y = [[G_even, *], [*, G_odd]] and the Gram is G_even + G_odd (added by k_gram_reduce).
// Only the MMA tiles of the two diagonal 32 x 32 blocks are issued: warp slot A takes the row pair
// (A, 7 - A) as before, now (4 - A) + (A + 1) = 5 tiles per k-step for TWO observations -- 3.6x
// fewer DMMAs per observation than padding P = 32 to a 64 x 64 tile with zeros.
// wts: [2r] even-row weight, [2r + 1] odd-row weight of packed row r.
// xt (slots 0 and 3 only, cvs != nullptr): the same fragments also give X' (Omega c) -- slot 0 holds every column
// of the even observation of a packed row (b[0..3]), slot 3 every column of the odd one (b[4..7]) -- as four
// DFMAs per k-step: xt[j] += X[r][8 j + gid] w_r c_r.  That is MultLogit.hpp:249,253's tXOmC without a second
// pass over X (k_xtv_stream: 71 of the 380 us of a category update at N = 1M).
template <int A, int kRows>
__device__ __forceinline__ void gram_pack_chunk(double (&c)[9][2], const double *chunk, const double *wts,
                                                int grp, int gid, int tig, const double *cvs, double (&xt)[4])
{
    constexpr int kLo = 4 - A;
#pragma unroll
    for (int kk = 0; kk < kRows / 8; ++kk) {
        const int r = grp * (kRows / 2) + kk * 4 + tig;          // this lane's k row (packed)
        const double we = wts[2 * r], wo = wts[2 * r + 1];
        const double *row = chunk + r * kGramLdm + gid;
        double b[8];
#pragma unroll
        for (int j = A; j < 4; ++j) b[j] = row[8 * j];
#pragma unroll
        for (int j = 7 - A; j < 8; ++j) b[j] = row[8 * j];
        const double alo = b[A] * we, ahi = b[7 - A] * wo;
#pragma unroll
        for (int j = A; j < 4; ++j) dmma884(c[j - A][0], c[j - A][1], alo, b[j]);
#pragma unroll
        for (int j = 7 - A; j < 8; ++j) dmma884(c[kLo + j - (7 - A)][0], c[kLo + j - (7 - A)][1], ahi, b[j]);
        if (cvs && (A == 0 || A == 3)) {
            const double wc = A == 0 ? we * cvs[2 * r] : wo * cvs[2 * r + 1];
#pragma unroll
            for (int j = 0; j < 4; ++j) xt[j] = fma(b[A == 0 ? j : 4 + j], wc, xt[j]);
        }
    }
}

template <int A>
__device__ __forceinline__ void gram_pack_store(const double (&c)[9][2], double *out, int gid, int tig)
{
    constexpr int kLo = 4 - A;
#pragma unroll
    for (int j = A; j < 4; ++j) {
        int row = 8 * A + gid, col = 8 * j + 2 * tig;
        out[row * kGramTile + col] = c[j - A][0];
        out[row * kGramTile + col + 1] = c[j - A][1];
    }
#pragma unroll
    for (int j = 7 - A; j < 8; ++j) {
        int row = 8 * (7 - A) + gid, col = 8 * j + 2 * tig;
        out[row * kGramTile + col] = c[kLo + j - (7 - A)][0];
        out[row * kGramTile + col + 1] = c[kLo + j - (7 - A)][1];
    }
}

template <int kRows, bool kBalancedDiag, bool kPacked = false>
__global__ void __launch_bounds__(256)
k_gram_partial(double *__restrict__ part, const double *__restrict__ tX, int64_t x_stride, const double *__restrict__ w,
               int64_t N, int P, int nt, int nslab_diag = 0, const double *__restrict__ cv = nullptr)
{
    BL_PDL_ENTER();
    extern __shared__ __align__(16) double gsm[];
    const int nthr = blockDim.x;
    // batched independent chains: blockIdx.z = chain (its weights and partial tiles; its rows at tX + chain x_stride:
    // N P for rows of its own, 0 for rows shared by the chains)
    tX += (size_t)blockIdx.z * x_stride;
    w += (size_t)blockIdx.z * N;
    if (cv) cv += (size_t)blockIdx.z * N;
    part += (size_t)blockIdx.z * gridDim.y * gridDim.x * (kBalancedDiag ? 1 : 2) * (kGramTile * kGramTile);
    int t = blockIdx.y, bi = 0;
    while (t >= nt - bi) { t -= nt - bi; ++bi; }
    const int bj = bi + t;
    const bool diag = bi == bj;
    const int npanel = diag ? 1 : 2;
    static_assert(!kPacked || kBalancedDiag, "packed rows exist only for the single-tile kernel");
    constexpr int kObs = kPacked ? 2 * kRows : kRows;            // observations per chunk
    const int stage_elems = npanel * kRows * kGramLdm + (kPacked ? 2 : 1) * kObs;     // packed: weights, then the c vector
    const int w_off = npanel * kRows * kGramLdm;
    const int c_off = w_off + kObs;

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gid = lane >> 2, tig = lane & 3;
    const int grp = warp >> 2, sub = warp & 3, si = sub >> 1, sj = sub & 1;

    // P > 64: a diagonal tile costs 36 MMA tiles per k-step against 64 for an off-diagonal one, so its
    // rows are cut into fewer, longer slabs (nslab_diag of them; CTAs past that leave) and every CTA of
    // the single wave carries the same work.  Partial tiles keep the uniform stride of gridDim.x slabs.
    const int ns = (!kBalancedDiag && diag && nslab_diag > 0) ? nslab_diag : (int)gridDim.x;
    if ((int)blockIdx.x >= ns) return;
    double c[4][4][2] = {};
    double c9[9][2] = {};                               // kBalancedDiag: this warp's 9 tiles
    double xt[4] = {0.0, 0.0, 0.0, 0.0};                // packed + cv: this lane's part of X' (Omega c)
    int64_t slab = (N + ns - 1) / ns;
    if (kPacked) slab = (slab + 1) & ~(int64_t)1;               // packed rows pair observations (2r, 2r+1) of the chain
    const int64_t r0 = (int64_t)blockIdx.x * slab;
    const int64_t r1 = r0 + slab < N ? r0 + slab : N;
    const bool vec16 = (P % 2 == 0) && ((reinterpret_cast<uintptr_t>(tX) & 15) == 0);

    auto issue = [&](int64_t base, int sidx) {
        const int so = sidx * stage_elems;
        if (base < r1) {
            if (vec16) {
                for (int e = threadIdx.x; e < npanel * kRows * (kGramTile / 2); e += nthr) {
                    int pnl = e >= kRows * (kGramTile / 2);
                    int rem = e - pnl * (kRows * (kGramTile / 2));
                    int r = rem >> 5, cc = (rem & 31) * 2;
                    int64_t i = kPacked ? base + 2 * r + (cc >> 5) : base + r;
                    int col = kPacked ? (cc & 31) : (pnl == 0 ? bi : bj) * kGramTile + cc;
                    bool ok = i < r1 && col < P;
                    cp_async16(&gsm[so + (pnl * kRows + r) * kGramLdm + cc], ok ? tX + i * P + col : tX, ok);
                }
            } else {
                for (int e = threadIdx.x; e < npanel * kRows * kGramTile; e += nthr) {
                    int pnl = e >= kRows * kGramTile;
                    int rem = e - pnl * (kRows * kGramTile);
                    int r = rem >> 6, cc = rem & 63;
                    int64_t i = kPacked ? base + 2 * r + (cc >> 5) : base + r;
                    int col = kPacked ? (cc & 31) : (pnl == 0 ? bi : bj) * kGramTile + cc;
                    bool ok = i < r1 && col < P;
                    cp_async8(&gsm[so + (pnl * kRows + r) * kGramLdm + cc], ok ? tX + i * P + col : tX, ok);
                }
            }
            if (threadIdx.x < kObs) {
                int64_t i = base + threadIdx.x;
                cp_async8(&gsm[so + w_off + threadIdx.x], i < r1 ? w + i : w, i < r1);
                if (kPacked && cv) cp_async8(&gsm[so + c_off + threadIdx.x], i < r1 ? cv + i : cv, i < r1);
            }
        }
        cp_async_commit();
    };

    issue(r0, 0);
    issue(r0 + kObs, 1);
    int cur = 0;
    for (int64_t base = r0; base < r1; base += kObs) {
        cp_async_wait<1>();
        __syncthreads();
        int nxt = cur + 2 >= kGramStages ? cur + 2 - kGramStages : cur + 2;
        issue(base + 2 * kObs, nxt);
        if (kPacked) {
            const double *chunk = gsm + cur * stage_elems;
            const double *cvs = cv ? chunk + c_off : nullptr;
            switch (sub) {
            case 0: gram_pack_chunk<0, kRows>(c9, chunk, chunk + w_off, grp, gid, tig, cvs, xt); break;
            case 1: gram_pack_chunk<1, kRows>(c9, chunk, chunk + w_off, grp, gid, tig, cvs, xt); break;
            case 2: gram_pack_chunk<2, kRows>(c9, chunk, chunk + w_off, grp, gid, tig, cvs, xt); break;
            default: gram_pack_chunk<3, kRows>(c9, chunk, chunk + w_off, grp, gid, tig, cvs, xt); break;
            }
        } else if (kBalancedDiag) {
            const double *chunk = gsm + cur * stage_elems;
            switch (sub) {
            case 0: gram_diag_chunk<0, kRows>(c9, chunk, chunk + w_off, grp, gid, tig); break;
            case 1: gram_diag_chunk<1, kRows>(c9, chunk, chunk + w_off, grp, gid, tig); break;
            case 2: gram_diag_chunk<2, kRows>(c9, chunk, chunk + w_off, grp, gid, tig); break;
            default: gram_diag_chunk<3, kRows>(c9, chunk, chunk + w_off, grp, gid, tig); break;
            }
        } else if (diag) {
            // a diagonal tile of a P > 64 Gram: the balanced deal of its 36 live MMA tiles (9 per warp,
            // all 8 warps busy) instead of 32 x 32 sub-tiles (one warp of four idle, one with 16 tiles:
            // the tile then cost as much as an off-diagonal one).  The 9 accumulators live in c's registers.
            double (&cd)[9][2] = reinterpret_cast<double (&)[9][2]>(c);
            const double *chunk = gsm + cur * stage_elems;
            switch (sub) {
            case 0: gram_diag_chunk<0, kRows>(cd, chunk, chunk + w_off, grp, gid, tig); break;
            case 1: gram_diag_chunk<1, kRows>(cd, chunk, chunk + w_off, grp, gid, tig); break;
            case 2: gram_diag_chunk<2, kRows>(cd, chunk, chunk + w_off, grp, gid, tig); break;
            default: gram_diag_chunk<3, kRows>(cd, chunk, chunk + w_off, grp, gid, tig); break;
            }
        } else {
            const int so = cur * stage_elems;
            const int pa = so + si * 32 + gid;                                         // A: panel bi
            const int pb = so + (npanel - 1) * kRows * kGramLdm + sj * 32 + gid;   // B: panel bj
#pragma unroll
            for (int kk = 0; kk < kRows / 8; ++kk) {
                const int r = grp * (kRows / 2) + kk * 4 + tig;                    // this lane's k row
                const double wr = gsm[so + w_off + r];
                double a[4], b[4];
#pragma unroll
                for (int m = 0; m < 4; ++m) {
                    a[m] = gsm[pa + r * kGramLdm + 8 * m] * wr;
                    b[m] = gsm[pb + r * kGramLdm + 8 * m];
                }
#pragma unroll
                for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                    for (int mj = 0; mj < 4; ++mj)
                        dmma884(c[mi][mj][0], c[mi][mj][1], a[mi], b[mj]);
            }
        }
        cur = cur + 1 == kGramStages ? 0 : cur + 1;
    }
    cp_async_wait<0>();
    if (kBalancedDiag) {
        // fold the two row groups inside the CTA (through the drained pipeline buffers): one
        // partial tile per CTA instead of two halves the reduce kernel's traffic
        __syncthreads();
        double *fold = gsm + (sub * 32 + lane) * 19;          // odd stride: conflict-free
        if (grp == 1) {
#pragma unroll
            for (int t = 0; t < 9; ++t) { fold[2 * t] = c9[t][0]; fold[2 * t + 1] = c9[t][1]; }
        }
        __syncthreads();
        if (grp == 0) {
#pragma unroll
            for (int t = 0; t < 9; ++t) { c9[t][0] += fold[2 * t]; c9[t][1] += fold[2 * t + 1]; }
        }
        if (kPacked && cv) {
            // X' (Omega c): add the four k rows of a lane group (tig), then the two row groups, and park the 32 + 32
            // sums (even / odd observations of the packed rows) in the unused off-diagonal block of the partial tile:
            // rows 0 and 1, columns 32..63.  k_gram_reduce adds the two rows and the slabs.
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                xt[j] += __shfl_xor_sync(0xffffffffu, xt[j], 1);
                xt[j] += __shfl_xor_sync(0xffffffffu, xt[j], 2);
            }
            __syncthreads();
            double *tf = gsm + 4 * 32 * 19;                     // past the accumulator fold area
            if ((sub == 0 || sub == 3) && grp == 1 && tig == 0) {
#pragma unroll
                for (int j = 0; j < 4; ++j) tf[(sub == 3 ? 32 : 0) + 8 * j + gid] = xt[j];
            }
            __syncthreads();
            if ((sub == 0 || sub == 3) && grp == 0 && tig == 0) {
                double *o = part + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * (kGramTile * kGramTile) +
                            (sub == 3 ? kGramTile : 0) + 32;
#pragma unroll
                for (int j = 0; j < 4; ++j) o[8 * j + gid] = xt[j] + tf[(sub == 3 ? 32 : 0) + 8 * j + gid];
            }
        }
    }
    // partial tile of (slab[, row group]): entries exist where (row >> 3) <= (col >> 3) on diagonal tiles
    double *out = kBalancedDiag
        ? part + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * (kGramTile * kGramTile)
        : part + ((size_t)blockIdx.y * (gridDim.x * 2) + blockIdx.x * 2 + grp) * (kGramTile * kGramTile);
    if (kPacked) {
        if (grp == 0) switch (sub) {
        case 0: gram_pack_store<0>(c9, out, gid, tig); break;
        case 1: gram_pack_store<1>(c9, out, gid, tig); break;
        case 2: gram_pack_store<2>(c9, out, gid, tig); break;
        default: gram_pack_store<3>(c9, out, gid, tig); break;
        }
    } else if (kBalancedDiag) {
        if (grp == 0) switch (sub) {
        case 0: gram_diag_store<0>(c9, out, gid, tig); break;
        case 1: gram_diag_store<1>(c9, out, gid, tig); break;
        case 2: gram_diag_store<2>(c9, out, gid, tig); break;
        default: gram_diag_store<3>(c9, out, gid, tig); break;
        }
    } else if (diag) {
        const double (&cd)[9][2] = reinterpret_cast<const double (&)[9][2]>(c);
        switch (sub) {
        case 0: gram_diag_store<0>(cd, out, gid, tig); break;
        case 1: gram_diag_store<1>(cd, out, gid, tig); break;
        case 2: gram_diag_store<2>(cd, out, gid, tig); break;
        default: gram_diag_store<3>(cd, out, gid, tig); break;
        }
    } else {
#pragma unroll
        for (int mi = 0; mi < 4; ++mi)
#pragma unroll
            for (int mj = 0; mj < 4; ++mj) {
                int row = si * 32 + mi * 8 + gid, col = sj * 32 + mj * 8 + 2 * tig;
                out[row * kGramTile + col] = c[mi][mj][0];
                out[row * kGramTile + col + 1] = c[mi][mj][1];
            }
    }
}

inline int gram_rows(bool any_offdiag) { return any_offdiag ? kGramRows : kGramRowsDiag; }

inline size_t gram_smem_bytes(bool any_offdiag, bool packed = false)
{
    int rows = gram_rows(any_offdiag);
    return (size_t)kGramStages * ((any_offdiag ? 2 : 1) * rows * kGramLdm + (packed ? 4 : 1) * rows) * sizeof(double);
}

// P == 32 rows are packed two per shared-memory row (gram_pack_chunk)
inline bool gram_packed(int P) { return P == 32; }

// ---------------------------------------------------------------------------------
// Peer exchange (see the window layout in gibbs.cu).  PeerPush travels with the kernel that
// produces the sums, PeerWait with the kernel that consumes them.
// ---------------------------------------------------------------------------------
constexpr int kMaxPeers = 8;

struct PeerPush {
    double *slot[kMaxPeers];      // slot [parity][my rank] inside every rank's window
    unsigned *flag[kMaxPeers];    // flag [parity][my rank] inside every rank's window
    unsigned *done;               // local CTA counter (zero between launches)
    int with_tail;                // also publish the P extra sums xtv() left behind the P^2 (acc[P^2 ..))
    unsigned epoch;
    int world;                    // <= 1: no exchange
};

struct PeerWait {
    const double *slot[kMaxPeers];   // slot [parity][r] of the LOCAL window
    const unsigned *flag;            // flags [parity][0..world) of the local window
    unsigned epoch;
    int world;                       // <= 1: no exchange
};

__device__ __forceinline__ void st_release_sys(unsigned *p, unsigned v)
{
    asm volatile("st.release.sys.global.u32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long global_timer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t));
    return t;
}

// Called by every thread of every CTA of the reducing kernel once its part of `acc` is written.
// The last CTA to arrive copies the whole local result (cnt doubles) into this rank's slot
// of every window with coalesced 16-byte NVLink stores -- 512 contiguous bytes per warp instruction
// instead of the reducing CTAs' scattered 8-byte element stores -- then one system-scope fence and
// the flags.  (Scattering from all CTAs cost ~20 us at 8 GPUs: 2 x 8 small stores per element and a
// system fence in each of the 128 CTAs.)
__device__ __forceinline__ void peer_publish(const PeerPush &px, const double *acc, int cnt)
{
    __shared__ int last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();                    // this CTA's part of acc is visible device-wide
        unsigned prev = atomicAdd(px.done, 1u);
        last = prev == gridDim.x * gridDim.y - 1;
        if (last) *px.done = 0;             // next launch on this stream starts from zero
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    const double2 *src = reinterpret_cast<const double2 *>(acc);
    const int n2 = cnt >> 1;
    for (int i0 = threadIdx.x; i0 < n2; i0 += 4 * blockDim.x) {
        double2 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * blockDim.x;
            v[u] = i < n2 ? __ldcg(src + i) : make_double2(0.0, 0.0);
        }
        for (int r = 0; r < px.world; ++r) {
            double2 *dst = reinterpret_cast<double2 *>(px.slot[r]);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + u * blockDim.x;
                if (i < n2) dst[i] = v[u];
            }
        }
    }
    // odd cnt (logit sweep with odd P: P^2 sums, no tail): the last double travels on its own
    if ((cnt & 1) && (int)threadIdx.x < px.world) px.slot[threadIdx.x][cnt - 1] = __ldcg(acc + cnt - 1);
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence_system();             // the slot stores are performed system-wide before the flags
        for (int r = 0; r < px.world; ++r) st_release_sys(px.flag[r], px.epoch);
    }
}

// One CTA waits until every rank's flag has reached the epoch (flags only grow).  A peer that
// never arrives (crashed rank) turns into status 2 after 20 s instead of a hung GPU.
__device__ __forceinline__ void peer_wait(const PeerWait &pw, int *status)
{
    if ((int)threadIdx.x < pw.world) {
        const unsigned long long t0 = global_timer_ns();
        while ((int)(ld_acquire_sys(pw.flag + threadIdx.x) - pw.epoch) < 0) {
            if (global_timer_ns() - t0 > 20000000000ull) { *status = 2; break; }
            __nanosleep(40);
        }
    }
    __syncthreads();
}

// A (ld x P, column-major) = P0 + sum_r slot_r[0..P^2), rhs = base_rhs + sum_r slot_r[P^2..P^2+P),
// ranks added in index order (identical bits on every rank).  Slot loads bypass L1 (.cg): the
// lines were written by other GPUs.  W = 0: world known only at run time.
template <int W>
__device__ __forceinline__ void peer_stage(const PeerWait &pw, double *A, double *rhs,
                                           const double *__restrict__ P0, const double *__restrict__ base_rhs,
                                           int add_tail, int P, int ld)
{
    constexpr int WW = W ? W : kMaxPeers;
    const int world = W ? W : pw.world;
    const int PP = P * P;
    if ((P & 1) == 0) {
        // pairs (k, k+1) share a column; two pairs per thread per trip -> 2 W 16-byte loads in flight
        const int H = PP >> 1;
        for (int h0 = threadIdx.x; h0 < H; h0 += 2 * blockDim.x) {
            const int h1 = h0 + blockDim.x;
            const bool v1 = h1 < H;
            double2 x0[WW], x1[WW];
#pragma unroll
            for (int r = 0; r < WW; ++r) {
                x0[r] = r < world ? __ldcg(reinterpret_cast<const double2 *>(pw.slot[r]) + h0) : make_double2(0.0, 0.0);
                x1[r] = (r < world && v1) ? __ldcg(reinterpret_cast<const double2 *>(pw.slot[r]) + h1) : make_double2(0.0, 0.0);
            }
            // P0 is caller memory (8-byte alignment only)
            double2 q0 = P0 ? make_double2(P0[2 * h0], P0[2 * h0 + 1]) : make_double2(0.0, 0.0);
            double2 q1 = (P0 && v1) ? make_double2(P0[2 * h1], P0[2 * h1 + 1]) : make_double2(0.0, 0.0);
            double2 s0 = x0[0], s1 = x1[0];
#pragma unroll
            for (int r = 1; r < WW; ++r)
                if (r < world) { s0.x += x0[r].x; s0.y += x0[r].y; s1.x += x1[r].x; s1.y += x1[r].y; }
            int k = 2 * h0;
            double *d = A + k % P + (size_t)ld * (k / P);
            d[0] = s0.x + q0.x; d[1] = s0.y + q0.y;
            if (v1) {
                k = 2 * h1;
                d = A + k % P + (size_t)ld * (k / P);
                d[0] = s1.x + q1.x; d[1] = s1.y + q1.y;
            }
        }
    } else {
        for (int k = threadIdx.x; k < PP; k += blockDim.x) {
            double s = __ldcg(pw.slot[0] + k);
            for (int r = 1; r < world; ++r) s += __ldcg(pw.slot[r] + k);
            A[k % P + (size_t)ld * (k / P)] = s + (P0 ? P0[k] : 0.0);
        }
    }
    for (int k = threadIdx.x; k < P; k += blockDim.x) {
        double t = 0.0;
        if (add_tail) {
            t = __ldcg(pw.slot[0] + PP + k);
            for (int r = 1; r < world; ++r) t += __ldcg(pw.slot[r] + PP + k);
        }
        rhs[k] = (base_rhs ? base_rhs[k] : 0.0) + t;
    }
}

// PP = P0 + sum over slabs of the partial tiles, mirrored to a full symmetric P x P
// column-major matrix.  One warp-row of threads per output element group: each CTA owns
// 32 upper-triangle candidates, its 8 warps split the slabs, fixed summation order.
static __global__ void __launch_bounds__(256)
k_gram_reduce(double *__restrict__ PP, const double *__restrict__ P0,
              const double *__restrict__ part, int P, int nt, int nslab, PeerPush px, int packed = 0,
              int nslab_diag = 0,      // nslab: partial tiles per output tile (stride); diagonal tiles hold nslab_diag of them (0: nslab)
              int tail_in_part = 0)    // packed tiles also carry X'(Omega c): the CTAs past the P^2 entries sum it into PP[P^2 ..)
{
    BL_PDL_ENTER();
    __shared__ double red[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // batched independent chains: blockIdx.y = chain
    PP += (size_t)blockIdx.y * ((size_t)P * P + P);
    part += (size_t)blockIdx.y * (nt * (nt + 1) / 2) * nslab * (kGramTile * kGramTile);
    int e = blockIdx.x * 32 + lane;
    // consecutive lanes take consecutive COLUMNS of a tile row (the partial tiles are row-major: one 256-byte run per
    // warp load; with consecutive rows every lane touched its own 32-byte sector, four times the L2 traffic)
    int a = e / P, b = e % P;
    bool want = e < P * P && a <= b;
    const bool tail = tail_in_part && e >= P * P && e < P * P + P;
    double s = 0.0;
    if (tail) {
        // rows 0 (even observations) and 1 (odd) of the tile's unused off-diagonal block, columns 32 + p
        const double *src = part + 32 + (e - P * P);
        for (int k = warp; k < nslab; k += 8)
            s += src[(size_t)k * (kGramTile * kGramTile)] + src[(size_t)k * (kGramTile * kGramTile) + kGramTile];
    }
    if (want) {
        int bi = a / kGramTile, bj = b / kGramTile;
        int tile = 0;
        for (int k = 0; k < bi; ++k) tile += nt - k;
        tile += bj - bi;
        int la = a % kGramTile, lb = b % kGramTile;
        // a diagonal tile holds (row, col) wherever (row >> 3) <= (col >> 3): true for every la <= lb
        const double *src = part + (size_t)tile * nslab * (kGramTile * kGramTile) + la * kGramTile + lb;
        const int cnt = (bi == bj && nslab_diag > 0) ? nslab_diag : nslab;
#pragma unroll 8
        for (int k = warp; k < cnt; k += 8) s += src[(size_t)k * (kGramTile * kGramTile)];
        if (packed) {
            // the odd observations' sums sit in the second diagonal 32 x 32 block of the tile
            const double *src2 = src + 32 * kGramTile + 32;
            double s2 = 0.0;
#pragma unroll 8
            for (int k = warp; k < cnt; k += 8) s2 += src2[(size_t)k * (kGramTile * kGramTile)];
            s += s2;
        }
    }
    red[warp][lane] = s;
    __syncthreads();
    if (warp == 0 && want) {
        double v = 0.0;
        for (int k = 0; k < 8; ++k) v += red[k][lane];
        v += P0 ? P0[a + (size_t)P * b] : 0.0;
        PP[a + (size_t)P * b] = v;
        PP[b + (size_t)P * a] = v;
    }
    if (warp == 0 && tail) {
        double v = 0.0;
        for (int k = 0; k < 8; ++k) v += red[k][lane];
        PP[e] = v;
    }
    // sharded data: the finished sums (and the P sums behind them) go into every rank's window
    if (px.world > 1) peer_publish(px, PP, P * P + (px.with_tail ? P : 0));
}

// out_p = sum_i x_i[p] * v_i  (X'v), v_i = c0*v0_i + c1*v1_i*v2_i  (v1/v2 optional).
// Per-CTA partial sums then a fixed-order reduce (k_xtv_reduce).
// Batched chains (this kernel and the two below): blockIdx.y = chain, its rows at tX + chain x_stride (N P: rows of
// its own; 0: rows shared by the chains), its weights at + chain N, its c1_dev coefficient at c1_dev[chain].
static __global__ void __launch_bounds__(256)
k_xtv_partial(double *__restrict__ part, const double *__restrict__ tX, int64_t x_stride, const double *__restrict__ v0,
              double c0, const double *__restrict__ v1, const double *__restrict__ v2, double c1,
              int64_t N, int P, const double *__restrict__ c1_dev = nullptr)
{
    BL_PDL_ENTER();
    if (c1_dev) c1 = c1_dev[blockIdx.y];       // coefficient produced on the device, one per chain (NB: log d)
    tX += (size_t)blockIdx.y * x_stride;
    part += (size_t)blockIdx.y * gridDim.x * P;
    if (v0) v0 += (size_t)blockIdx.y * N;
    if (v1) v1 += (size_t)blockIdx.y * N;
    if (v2) v2 += (size_t)blockIdx.y * N;
    extern __shared__ double sacc[];   // [warps][P]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int p = threadIdx.x; p < nw * P; p += blockDim.x) sacc[p] = 0.0;
    __syncthreads();
    const int64_t slab = (N + gridDim.x - 1) / gridDim.x;
    const int64_t r0 = (int64_t)blockIdx.x * slab;
    const int64_t r1 = r0 + slab < N ? r0 + slab : N;
    for (int p = lane; p < P; p += 32) {
        double s = 0.0;
        for (int64_t i = r0 + warp; i < r1; i += nw) {
            double vi = (v0 ? c0 * v0[i] : 0.0) + (v1 ? c1 * v1[i] * (v2 ? v2[i] : 1.0) : 0.0);
            s = fma(tX[i * P + p], vi, s);
        }
        sacc[warp * P + p] = s;
    }
    __syncthreads();
    for (int p = threadIdx.x; p < P; p += blockDim.x) {
        double s = 0.0;
        for (int k = 0; k < nw; ++k) s += sacc[k * P + p];
        part[(size_t)blockIdx.x * P + p] = s;
    }
}

// The same on the FP64 tensor cores (even P, 16-byte aligned tX): out = X' v as m8n8k4 MMAs with
// the four k slots on four consecutive rows and v repeated in every column of B.  Lane (gid, tig)
// loads the 16 bytes X[i + tig][pc + 2 gid, +1] (the eight gid lanes cover 128 contiguous bytes
// of the row) and feeds .x to the MMA that accumulates the even columns of a 16-column block and
// .y to the one for the odd columns.  A warp owns one 64-column panel and every (8 / panels)-th
// group of 16 rows of the CTA's slab, 16 loads of 16 bytes in flight per lane; the scalar
// k_xtv_partial above keeps 4 rows in flight per warp and reaches 1.1 TB/s.
static __global__ void __launch_bounds__(256, 2)
k_xtv_mma(double *__restrict__ part, const double *__restrict__ tX, int64_t x_stride, const double *__restrict__ v0,
          double c0, const double *__restrict__ v1, const double *__restrict__ v2, double c1,
          int64_t N, int P, const double *__restrict__ c1_dev)
{
    BL_PDL_ENTER();
    if (c1_dev) c1 = c1_dev[blockIdx.y];
    tX += (size_t)blockIdx.y * x_stride;
    part += (size_t)blockIdx.y * gridDim.x * P;
    if (v0) v0 += (size_t)blockIdx.y * N;
    if (v1) v1 += (size_t)blockIdx.y * N;
    if (v2) v2 += (size_t)blockIdx.y * N;
    extern __shared__ double sacc[];                     // [row sub-groups][P]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, gid = lane >> 2, tig = lane & 3;
    const int panels = (P + 63) >> 6;                    // 1..4
    const int nsub = 8 / panels;
    const int panel = warp % panels, sub = warp / panels;
    const int64_t slab = (N + gridDim.x - 1) / gridDim.x;
    const int64_t r0 = (int64_t)blockIdx.x * slab;
    const int64_t r1 = r0 + slab < N ? r0 + slab : N;
    const int pc = panel * 64 + 2 * gid;                 // this lane's first column
    double acc[4][2][2] = {};                            // [16-column block][even / odd][c0, c1]
    if (sub < nsub) {
        for (int64_t i0 = r0 + sub * 16; i0 < r1; i0 += nsub * 16) {
            double2 a[4][4];
            double vv[4];
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const int64_t i = i0 + 4 * g + tig;
                const bool rv = i < r1;
#pragma unroll
                for (int cb = 0; cb < 4; ++cb)
                    a[g][cb] = (rv && pc + 16 * cb < P) ? __ldg(reinterpret_cast<const double2 *>(tX + i * P + pc + 16 * cb))
                                                        : make_double2(0.0, 0.0);
                vv[g] = rv ? (v0 ? c0 * v0[i] : 0.0) + (v1 ? c1 * v1[i] * (v2 ? v2[i] : 1.0) : 0.0) : 0.0;
            }
#pragma unroll
            for (int g = 0; g < 4; ++g)
#pragma unroll
                for (int cb = 0; cb < 4; ++cb)
                    if (panel * 64 + 16 * cb < P) {              // warp-uniform: no MMAs on column blocks past P
                        dmma884(acc[cb][0][0], acc[cb][0][1], a[g][cb].x, vv[g]);
                        dmma884(acc[cb][1][0], acc[cb][1][1], a[g][cb].y, vv[g]);
                    }
        }
        if (tig == 0) {
#pragma unroll
            for (int cb = 0; cb < 4; ++cb)
                if (pc + 16 * cb < P) {
                    sacc[sub * P + pc + 16 * cb] = acc[cb][0][0];
                    sacc[sub * P + pc + 16 * cb + 1] = acc[cb][1][0];
                }
        }
    }
    __syncthreads();
    for (int p = threadIdx.x; p < P; p += blockDim.x) {
        double s = 0.0;
        for (int k = 0; k < nsub; ++k) s += sacc[k * P + p];
        part[(size_t)blockIdx.x * P + p] = s;
    }
}

// Streaming form for P a power of two (8 <= P <= 256; kLog2L = log2(P / 2)) and 16-byte aligned tX:
// the CTA's slab is read as one flat run of 16-byte column pairs, 512 consecutive pairs (8 KB) per
// warp trip with all 16 loads of a lane in flight.  A lane meets the same column pair (P <= 64) or
// the same P/64 column pairs in rotation (P = 128, 256) on every trip, so its sums stay in registers,
// and with the row length a compile-time power of two every row index of a trip is the first one
// plus a constant: the loop is ~8 instructions per 16 bytes and HBM-bound.  (With a run-time shift
// and 64-bit element indices the same loop issued 48 instructions per 16 bytes and sat at 3 TB/s.)
// kMode: which of the weight arrays exist (compile-time, so the 16 weight fetches of a trip are
// issued together instead of one by one behind null tests): 0: c0 v0; 1: c1 v1 v2; 2: c0 v0 + c1 v1.
template <int kMode>
__device__ __forceinline__ double xtv_weight(const double *w0, double c0, const double *w1, const double *w2,
                                             double c1, int i)
{
    if (kMode == 0) return c0 * __ldg(w0 + i);
    if (kMode == 1) return c1 * __ldg(w1 + i) * __ldg(w2 + i);
    return c0 * __ldg(w0 + i) + c1 * __ldg(w1 + i);
}

template <int kLog2L, int kMode>
__global__ void __launch_bounds__(256, 2)
k_xtv_stream(double *__restrict__ part, const double *__restrict__ tX, int64_t x_stride, const double *__restrict__ v0,
             double c0, const double *__restrict__ v1, const double *__restrict__ v2, double c1,
             int64_t N, const double *__restrict__ c1_dev)
{
    BL_PDL_ENTER();
    constexpr int L = 1 << kLog2L, P = 2 * L;            // column pairs per row, columns
    constexpr int kQ = L > 32 ? L / 32 : 1;              // column pairs a lane rotates through
    if (c1_dev) c1 = c1_dev[blockIdx.y];
    tX += (size_t)blockIdx.y * x_stride;
    part += (size_t)blockIdx.y * gridDim.x * P;
    extern __shared__ double sacc[];                     // [warps][P]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int64_t slab = (N + gridDim.x - 1) / gridDim.x;
    const int64_t r0 = (int64_t)blockIdx.x * slab;
    const int64_t r1 = r0 + slab < N ? r0 + slab : N;
    const int np = r1 > r0 ? (int)((r1 - r0) << kLog2L) : 0;        // pairs in the slab (host keeps it < 2^31)
    const double2 *X2 = reinterpret_cast<const double2 *>(tX + r0 * P);
    const size_t voff = (size_t)blockIdx.y * N + r0;
    const double *w0 = v0 ? v0 + voff : nullptr, *w1 = v1 ? v1 + voff : nullptr, *w2 = v2 ? v2 + voff : nullptr;
    double2 acc[kQ];
#pragma unroll
    for (int q = 0; q < kQ; ++q) acc[q] = make_double2(0.0, 0.0);
    for (int e0 = warp * 512; e0 < np; e0 += nw * 512) {
        const double2 *Xw = X2 + e0 + lane;
        const int i0 = (e0 + lane) >> kLog2L;            // row of this lane's first pair (slab-relative)
        double2 x[16];
        if (e0 + 512 <= np) {
#pragma unroll
            for (int u = 0; u < 16; ++u) x[u] = __ldg(Xw + u * 32);
            // rows advance by a constant per u: at most 16 distinct weights per trip (one when P >= 64 ... 256)
            constexpr int kStep = L <= 32 ? 32 / L : 1, kEvery = L <= 32 ? 1 : L / 32;
            double vi[16 / kEvery];
#pragma unroll
            for (int r = 0; r < 16 / kEvery; ++r) vi[r] = xtv_weight<kMode>(w0, c0, w1, w2, c1, i0 + r * kStep);
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                acc[u % kQ].x = fma(x[u].x, vi[u / kEvery], acc[u % kQ].x);
                acc[u % kQ].y = fma(x[u].y, vi[u / kEvery], acc[u % kQ].y);
            }
        } else {
#pragma unroll
            for (int u = 0; u < 16; ++u) x[u] = e0 + u * 32 + lane < np ? __ldg(Xw + u * 32) : make_double2(0.0, 0.0);
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                const int i = i0 + ((u * 32) >> kLog2L);
                double vi = 0.0;
                if (e0 + u * 32 + lane < np) vi = xtv_weight<kMode>(w0, c0, w1, w2, c1, i);
                acc[u % kQ].x = fma(x[u].x, vi, acc[u % kQ].x);
                acc[u % kQ].y = fma(x[u].y, vi, acc[u % kQ].y);
            }
        }
    }
    // lanes that share a column pair (P < 64: pair = lane mod P/2)
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1)
        if (o >= L) {
#pragma unroll
            for (int q = 0; q < kQ; ++q) {
                acc[q].x += __shfl_xor_sync(0xffffffffu, acc[q].x, o);
                acc[q].y += __shfl_xor_sync(0xffffffffu, acc[q].y, o);
            }
        }
    if (lane < L) {
#pragma unroll
        for (int q = 0; q < kQ; ++q) {
            sacc[warp * P + 2 * (lane + 32 * q)] = acc[q].x;
            sacc[warp * P + 2 * (lane + 32 * q) + 1] = acc[q].y;
        }
    }
    __syncthreads();
    for (int p = threadIdx.x; p < P; p += blockDim.x) {
        double s = 0.0;
        for (int k = 0; k < nw; ++k) s += sacc[k * P + p];
        part[(size_t)blockIdx.x * P + p] = s;
    }
}

// 0: not eligible; else log2(P / 2) of k_xtv_stream
inline int xtv_stream_log2l(const double *tX, int P)
{
    if ((reinterpret_cast<uintptr_t>(tX) & 15) != 0 || P < 8 || P > 256 || (P & (P - 1)) != 0) return 0;
    int l = 0;
    while ((2 << l) < P) ++l;
    return l;
}

static __global__ void k_xtv_reduce(double *__restrict__ out, const double *__restrict__ add0,
                             const double *__restrict__ add1, const double *__restrict__ part,
                             int P, int nslab, int64_t out_stride)
{
    BL_PDL_ENTER();
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    // batched independent chains: blockIdx.y = chain (add0 is shared by the chains, add1 is not); chain c's sums go
    // to out + c out_stride (P: vectors side by side; P^2 + P: the X'v tail behind each chain's Gram sums)
    out += (size_t)blockIdx.y * out_stride;
    part += (size_t)blockIdx.y * nslab * P;
    if (add1) add1 += (size_t)blockIdx.y * P;
    double s = 0.0;
    for (int k = 0; k < nslab; ++k) s += part[(size_t)k * P + p];
    out[p] = s + (add0 ? add0[p] : 0.0) + (add1 ? add1[p] : 0.0);
}

// kappa_i = n_i (y_i - 1/2)   (Logit.hpp:180-181);  NB: kappa_i = (y_i - d)/2
static __global__ void k_kappa(double *__restrict__ kappa, const double *__restrict__ y,
                        const double *__restrict__ n, double d, int64_t N)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) kappa[i] = n ? n[i] * (y[i] - 0.5) : 0.5 * (y[i] - d);
}

// shape_i = (int) n_i  (Logit.hpp:287)  /  b_i = y_i + d  (NBPG-logmean.R:88)
static __global__ void k_shape_int(int *__restrict__ out, const double *__restrict__ n, int64_t N)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) out[i] = (int)n[i];
}
static __global__ void k_shape_add(double *__restrict__ out, const double *__restrict__ y, double d, int64_t N)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) out[i] = y[i] + d;
}

// ---------------------------------------------------------------------------------
// Negative-binomial dispersion update, draw.df of Code/R/NB-Shape.R:21-53 (kernel 1: random walk on
// the integers) with df.llh :9-19.  d lives in device memory; nothing returns to the host.
//   proposal: uniform on max(d-1,1) .. d+1 from the first uniform of stream (seed, 2^64-2, call)
//   llh(d) = sum_j log(d+j) G[j] + d sum_i (log d - log(e^phi_i + d)) + sum_i y_i (phi_i - log(e^phi_i + d))
// k_nb_df_partial: per-CTA sums of the two N-term series for d and the proposal (fixed order);
// k_nb_df_decide: one warp adds them up, adds the G series, applies the Metropolis test with the
// stream's second uniform and publishes d, log d (and the recorded draw).
// Several chains on shared rows (bl_nb_multichain): chain c reads phi + c N, its d at dptr[c] and log d at
// ldptr[c], draws from the Metropolis stream of seed + c and owns partials [c][gridDim.x][4]; the partial kernels
// take the chain as blockIdx.y, the decide kernels one warp per chain (blockIdx.x), and k_nb_prepare blockIdx.y.
// One chain: the single chain's layout (d, log d side by side) and summation order.
// ---------------------------------------------------------------------------------
constexpr uint64_t kDfObs = 0xFFFFFFFFFFFFFFFEull;

__device__ __forceinline__ double nb_df_proposal(double d, uint64_t seed, uint32_t call, double *u_accept)
{
    PhiloxSource s;
    s.open(seed, kDfObs, call);
    double lower = d - 1.0 > 1.0 ? d - 1.0 : 1.0;
    int nn = (int)(d + 1.0 - lower) + 1;
    int k = (int)floor(s.unif() * nn);
    if (k > nn - 1) k = nn - 1;
    if (u_accept) *u_accept = s.unif();
    return lower + k;
}

static __global__ void __launch_bounds__(256)
k_nb_df_partial(double *__restrict__ part, const double *__restrict__ phi, const double *__restrict__ y,
                const double *__restrict__ dptr, int64_t N, uint64_t seed, uint32_t call)
{
    __shared__ double red[8][4];
    phi += blockIdx.y * N;
    part += (size_t)blockIdx.y * gridDim.x * 4;
    const double d = dptr[blockIdx.y], dp = nb_df_proposal(d, seed + blockIdx.y, call, nullptr);
    const double ld = log(d), ldp = log(dp);
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    const int64_t slab = (N + gridDim.x - 1) / gridDim.x;
    const int64_t r0 = (int64_t)blockIdx.x * slab, r1 = r0 + slab < N ? r0 + slab : N;
    for (int64_t i = r0 + threadIdx.x; i < r1; i += blockDim.x) {
        double ph = phi[i], mu = exp(ph), yi = y[i];
        double l0 = log(mu + d), l1 = log(mu + dp);
        s[0] += ld - l0;
        s[1] += yi * (ph - l0);
        s[2] += ldp - l1;
        s[3] += yi * (ph - l1);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        double v = s[k];
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red[warp][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        double v = 0.0;
        for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
        part[(size_t)blockIdx.x * 4 + threadIdx.x] = v;
    }
}

// Sharded rows: the CTA partials of this rank's rows folded to the four sums (fixed order) that the
// ranks then all-reduce; k_nb_df_decide reads the result as a single partial.
static __global__ void k_nb_df_fold(double *__restrict__ sum4, const double *__restrict__ part, int nblk)
{
    const int lane = threadIdx.x;
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    for (int b = lane; b < nblk; b += 32)
        for (int k = 0; k < 4; ++k) s[k] += part[(size_t)b * 4 + k];
#pragma unroll
    for (int k = 0; k < 4; ++k)
        for (int o = 16; o; o >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
    if (lane == 0)
        for (int k = 0; k < 4; ++k) sum4[k] = s[k];
}

// probe (bl_probe_nb_dispersion; the drivers pass null): chain c's {d', u, llh(d), llh(d')} at probe + 5 c.
static __global__ void k_nb_df_decide(double *__restrict__ dptr, double *__restrict__ ldptr, double *__restrict__ d_rec,
                               const double *__restrict__ part, int nblk, const double *__restrict__ G, int ymax,
                               uint64_t seed, uint32_t call, int64_t rec_stride = 0, double *__restrict__ probe = nullptr)
{
    const int lane = threadIdx.x, ch = blockIdx.x;
    part += (size_t)ch * nblk * 4;
    const double d = dptr[ch];
    double u_acc;
    const double dp = nb_df_proposal(d, seed + ch, call, &u_acc);
    double s[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int b = lane; b < nblk; b += 32)
        for (int k = 0; k < 4; ++k) s[k] += part[(size_t)b * 4 + k];
    for (int j = lane; j < ymax; j += 32) {
        s[4] += log(d + j) * G[j];
        s[5] += log(dp + j) * G[j];
    }
#pragma unroll
    for (int k = 0; k < 6; ++k)
        for (int o = 16; o; o >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
    if (lane == 0) {
        double llh_prev = s[4] + d * s[0] + s[1];
        double llh_prop = s[5] + dp * s[2] + s[3];
        double lppsl = log(dp == 1.0 ? 0.5 : 1.0 / 3.0) - log(d == 1.0 ? 0.5 : 1.0 / 3.0);
        double dn = u_acc < exp(llh_prop - llh_prev + lppsl) ? dp : d;
        if (probe) { probe[5 * ch] = dp; probe[5 * ch + 1] = u_acc; probe[5 * ch + 2] = llh_prev; probe[5 * ch + 3] = llh_prop; }
        dptr[ch] = dn;
        ldptr[ch] = log(dn);
        if (d_rec) d_rec[ch * rec_stride] = dn;
    }
}

// draw.df.real.mean (NB-Shape.R:86-96; the alternative at NBPG-logmean.R:87): random walk on the reals,
// rstar ~ U(r - 1, r + 1) (U(0, 2) when r <= 1), target sum_i dnbinom(y_i, size r, prob mu_i / (mu_i + r), log) as
// written there; log density restated as lgamma(y + r) - lgamma(r) - lgamma(y + 1) + r log p + y log(1 - p).
// Same stream as draw.df: first uniform the proposal, second the one of lu = log(runif(1)).
__device__ __forceinline__ double nb_dfreal_proposal(double r, uint64_t seed, uint32_t call, double *lu)
{
    PhiloxSource s;
    s.open(seed, kDfObs, call);
    const double u = s.unif();
    const double rs = r > 1.0 ? (r - 1.0) + 2.0 * u : 2.0 * u;
    if (lu) *lu = log(s.unif());
    return rs;
}

// part[b] = {sum_i t_i(r), 0, sum_i t_i(rstar), 0} over the CTA's rows (the four-slot layout of k_nb_df_partial)
static __global__ void __launch_bounds__(256)
k_nb_dfreal_partial(double *__restrict__ part, const double *__restrict__ phi, const double *__restrict__ y,
                    const double *__restrict__ dptr, int64_t N, uint64_t seed, uint32_t call)
{
    __shared__ double red[8][2];
    phi += blockIdx.y * N;
    part += (size_t)blockIdx.y * gridDim.x * 4;
    const double r = dptr[blockIdx.y], rs = nb_dfreal_proposal(r, seed + blockIdx.y, call, nullptr);
    const double lgr = lgamma(r), lgs = lgamma(rs), lr = log(r), ls = log(rs);
    double s0 = 0.0, s1 = 0.0;
    const int64_t slab = (N + gridDim.x - 1) / gridDim.x;
    const int64_t r0 = (int64_t)blockIdx.x * slab, r1 = r0 + slab < N ? r0 + slab : N;
    for (int64_t i = r0 + threadIdx.x; i < r1; i += blockDim.x) {
        const double ph = phi[i], mu = exp(ph), yi = y[i], lgy = lgamma(yi + 1.0);
        const double l0 = log(mu + r), l1 = log(mu + rs);
        s0 += lgamma(yi + r) - lgr - lgy + r * (ph - l0) + yi * (lr - l0);
        s1 += lgamma(yi + rs) - lgs - lgy + rs * (ph - l1) + yi * (ls - l1);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int o = 16; o; o >>= 1) { s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o); }
    if (lane == 0) { red[warp][0] = s0; red[warp][1] = s1; }
    __syncthreads();
    if (threadIdx.x < 4) {
        double v = 0.0;
        if ((threadIdx.x & 1) == 0)
            for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x >> 1];
        part[(size_t)blockIdx.x * 4 + threadIdx.x] = v;
    }
}

// probe: chain c's {r*, lu, llh(r), llh(r*)} at probe + 5 c, as in k_nb_df_decide.
static __global__ void k_nb_dfreal_decide(double *__restrict__ dptr, double *__restrict__ ldptr, double *__restrict__ d_rec,
                                          const double *__restrict__ part, int nblk, uint64_t seed, uint32_t call,
                                          int64_t rec_stride = 0, double *__restrict__ probe = nullptr)
{
    const int lane = threadIdx.x, ch = blockIdx.x;
    part += (size_t)ch * nblk * 4;
    const double r = dptr[ch];
    double lu;
    const double rs = nb_dfreal_proposal(r, seed + ch, call, &lu);
    double s0 = 0.0, s1 = 0.0;
    for (int b = lane; b < nblk; b += 32) { s0 += part[(size_t)b * 4]; s1 += part[(size_t)b * 4 + 2]; }
    for (int o = 16; o; o >>= 1) { s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o); }
    if (lane == 0) {
        const double dn = lu < s1 - s0 ? rs : r;
        if (probe) { probe[5 * ch] = rs; probe[5 * ch + 1] = lu; probe[5 * ch + 2] = s0; probe[5 * ch + 3] = s1; }
        dptr[ch] = dn;
        ldptr[ch] = log(dn);
        if (d_rec) d_rec[ch * rec_stride] = dn;
    }
}

// psi <- phi - log d, shape <- y + d, kappa <- (y - d)/2 with d from device memory (NBPG-logmean.R:88-94)
static __global__ void k_nb_prepare(double *__restrict__ psi, double *__restrict__ shape, double *__restrict__ kappa,
                             const double *__restrict__ y, const double *__restrict__ dptr,
                             const double *__restrict__ ldptr, int64_t N)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const double d = dptr[blockIdx.y], ld = ldptr[blockIdx.y];
    const int64_t k = blockIdx.y * N + i;
    psi[k] -= ld;
    shape[k] = y[i] + d;
    kappa[k] = 0.5 * (y[i] - d);
}

// ymax and G[j] = #{y_i > j} (NBPG-logmean.R:65-67).  k_nb_hist indexes hist by (int)y, so a count that is negative,
// not finite or at least 2^31 - 1 sets *ymax to kNbBadCount instead, which no valid count reaches (an all-reduce by
// max carries it to every rank); the host refuses the data before it sizes the histogram.
constexpr unsigned long long kNbBadCount = ~0ull;
static __global__ void k_nb_ymax(unsigned long long *__restrict__ ymax, const double *__restrict__ y, int64_t N)
{
    int m = 0;
    bool bad = false;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        const double v = y[i];
        if (v >= 0.0 && v < 2147483647.0) m = max(m, (int)v);
        else bad = true;                          // NaN fails both comparisons
    }
    for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    bad = __any_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0 && (bad || m > 0)) atomicMax(ymax, bad ? kNbBadCount : (unsigned long long)m);
}
static __global__ void k_nb_hist(unsigned long long *__restrict__ hist, const double *__restrict__ y, int64_t N)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x)
        atomicAdd(&hist[(int)y[i]], 1ull);
}
static __global__ void k_nb_suffix(double *__restrict__ G, const unsigned long long *__restrict__ hist, int ymax)
{
    unsigned long long run = 0;                    // G[j] = sum_{k > j} hist[k], j = ymax-1 .. 0
    for (int j = ymax - 1; j >= 0; --j) {
        run += hist[j + 1];
        G[j] = (double)run;
    }
}

static __global__ void k_fill(double *__restrict__ x, double v, int64_t n)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) x[i] = v;
}

// mlogit offsets for category j: A = sum_{k != j, k < J-1} exp(XB_k) + exp(0),
// c = log A, eta = XB_j - c.  XB is N x (J-1) column-major (the reference's J-th
// column is identically 0, MultLogit.hpp:275-277).  No max-subtraction, as there.
// Several chains (blockIdx.y = chain): chain c's XB at XB + c U N, its c and eta at + c N.
static __global__ void k_mlogit_offsets(double *__restrict__ c, double *__restrict__ eta,
                                 const double *__restrict__ XB, int64_t N, int U, int j)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    XB += (size_t)blockIdx.y * U * N;
    c += (size_t)blockIdx.y * N;
    eta += (size_t)blockIdx.y * N;
    // the reference sums columns of XB_no_j in order: categories 0..J-1 without j, the
    // all-zero last column included (exp(0) = 1 added last)
    double A = 0.0;
    for (int k = 0; k < U; ++k)
        if (k != j) A += exp(XB[i + (size_t)N * k]);
    A += 1.0;
    double cj = log(A);
    c[i] = cj;
    eta[i] = XB[i + (size_t)N * j] - cj;
}

// ---------------------------------------------------------------------------------
// Random-intercept logit (logit_ri_gibbs_device): psi_i = x_i . beta + u_{g_i}, u_g ~ N(0, tau2), tau2 ~ IG(a0, b0).
// Per iteration, after the omega draw: group sums S_g = sum omega_i, R_g = sum (kappa_i - omega_i eta_i) over the
// rows of the group, u_g | . ~ N(R_g / (S_g + 1/tau2), 1 / (S_g + 1/tau2)), tau2 | u, then the rows' offsets and
// v_i = kappa_i - omega_i u_{g_i} for X'v.  Sums run over the rows sorted by group (a stable sort made once per
// chain), cut into fixed chunks of kRiChunk positions: a chunk sums the segments it holds in a fixed order and writes
// a group that lies inside it straight to S, R; a group that crosses chunk boundaries leaves its first piece as the
// tail of its first chunk and the rest as the heads of the following chunks, which k_ri_draw_u adds in chunk order.
// No floating-point atomics: every sum is bit-identical from run to run, whatever the group sizes.
// Several chains on one data set (logit_ri_multichain_device), kChains: the chain is a grid dimension of every
// per-iteration kernel (blockIdx.y; k_ri_draw_tau2: blockIdx.x), chain c keeps its own rows' state at + c N (eta, off,
// v, omega, psi), its groups' at + c G (S, R, u), its chunks' edges, partials and tau2, and draws from the streams of
// seed + c; the sorted order, the offsets and kappa are shared.  Chain c sums in the single chain's order: bit for bit
// its run.  The single chain's instantiations (kChains false) leave the chain arguments unread.
// ---------------------------------------------------------------------------------
constexpr uint64_t kRiGroupObs0 = 0x8000000000000000ull;   // u_g: first normal of the stream (seed, 2^63 + g, call)
constexpr uint64_t kRiTau2Obs = 0xFFFFFFFFFFFFFFFCull;     // tau2: the gamma variate of the stream (seed, 2^64 - 4, call)
constexpr int kRiItems = 8;                                // sorted positions per thread
constexpr int kRiThreads = 256;
constexpr int kRiChunk = kRiItems * kRiThreads;            // sorted positions per chunk (one CTA)
constexpr int kRiDrawWarps = 8;                            // groups per CTA of k_ri_draw_u (a warp each)

// *bad = 1 if an id lies outside [0, G)
static __global__ void k_ri_check_ids(int *__restrict__ bad, const int *__restrict__ group, int64_t N, int G)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x)
        if (group[i] < 0 || group[i] >= G) *bad = 1;
}

// goff[g] = first sorted position of group g, goff[G] = N (gs: the ids in sorted order).  Thread k writes the
// groups that start at position k -- the one at k and the empty ones before it -- so every entry is written once.
static __global__ void k_ri_offsets(int *__restrict__ goff, const int *__restrict__ gs, int64_t N, int G)
{
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k > N) return;
    const int lo = k == 0 ? 0 : gs[k - 1] + 1, hi = k == N ? G : gs[k];
    for (int g = lo; g <= hi; ++g) goff[g] = (int)k;
}

// unfused path: psi_i = eta_i + off_i (kChains: chain blockIdx.y at + c N)
template <bool kChains>
static __global__ void k_ri_psi(double *__restrict__ psi, const double *__restrict__ eta, const double *__restrict__ off,
                                int64_t N)
{
    BL_PDL_ENTER();
    if (kChains) {
        const size_t ch = (size_t)blockIdx.y * N;
        psi += ch;
        eta += ch;
        off += ch;
    }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x)
        psi[i] = eta[i] + off[i];
}

// Segment sum (s, r) with a flag: a segment starts inside the run it covers.  a then b: b alone if b holds a start.
struct RiSeg {
    double s, r;
    int f;
};
__device__ __forceinline__ RiSeg ri_seg_join(const RiSeg &a, const RiSeg &b)
{
    return b.f ? b : RiSeg{a.s + b.s, a.r + b.r, a.f};
}

// One CTA per chunk of kRiChunk sorted positions, kRiItems consecutive positions per thread.  edge[4 c ..]: head
// (s, r) and tail (s, r) pieces of chunk c (written only when a group crosses that edge).  kChains: chain blockIdx.y,
// S, R at + c G, edge at + 4 c gridDim.x, omega and eta at + c N.
template <bool kChains>
static __global__ void __launch_bounds__(kRiThreads)
k_ri_group_sums(double *__restrict__ S, double *__restrict__ R, double *__restrict__ edge, const int *__restrict__ order,
                const int *__restrict__ gs, const int *__restrict__ goff, const double *__restrict__ w,
                const double *__restrict__ eta, const double *__restrict__ kappa, int64_t N, int G)
{
    BL_PDL_ENTER();
    if (kChains) {
        S += (size_t)blockIdx.y * G;
        R += (size_t)blockIdx.y * G;
        edge += (size_t)blockIdx.y * 4 * gridDim.x;
        w += (size_t)blockIdx.y * N;
        eta += (size_t)blockIdx.y * N;
    }
    __shared__ RiSeg wtot[kRiThreads / 32], wcarry[kRiThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t p0 = (int64_t)blockIdx.x * kRiChunk, p1 = min(p0 + (int64_t)kRiChunk, N);
    const int64_t q0 = p0 + (int64_t)threadIdx.x * kRiItems;
    double sv[kRiItems], rv[kRiItems];
    int gv[kRiItems];
#pragma unroll
    for (int k = 0; k < kRiItems; ++k) {
        const int64_t p = q0 + k;
        gv[k] = -1;
        sv[k] = rv[k] = 0.0;
        if (p < p1) {
            const int row = order[p];
            const double om = w[row];
            gv[k] = gs[p];
            sv[k] = om;
            rv[k] = fma(-om, eta[row], kappa[row]);
        }
    }
    const int gprev = (q0 > p0 && q0 < p1) ? gs[q0 - 1] : -1;
    // the thread's own run: the sums since its last segment start
    RiSeg own{0.0, 0.0, 0};
#pragma unroll
    for (int k = 0; k < kRiItems; ++k) {
        if (gv[k] < 0) break;
        if (gv[k] != (k == 0 ? gprev : gv[k - 1])) own = RiSeg{0.0, 0.0, 1};
        own.s += sv[k];
        own.r += rv[k];
    }
    // segmented inclusive scan over the warp's runs, then over the warps (fixed order)
    RiSeg inc = own;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        RiSeg t{__shfl_up_sync(0xffffffffu, inc.s, o), __shfl_up_sync(0xffffffffu, inc.r, o),
                __shfl_up_sync(0xffffffffu, inc.f, o)};
        if (lane >= o) inc = ri_seg_join(t, inc);
    }
    if (lane == 31) wtot[warp] = inc;
    __syncthreads();
    if (threadIdx.x == 0) {
        RiSeg run{0.0, 0.0, 0};
        for (int v = 0; v < kRiThreads / 32; ++v) {
            wcarry[v] = run;
            run = ri_seg_join(run, wtot[v]);
        }
    }
    __syncthreads();
    RiSeg ex{__shfl_up_sync(0xffffffffu, inc.s, 1), __shfl_up_sync(0xffffffffu, inc.r, 1),
             __shfl_up_sync(0xffffffffu, inc.f, 1)};
    const RiSeg carry = lane == 0 ? wcarry[warp] : ri_seg_join(wcarry[warp], ex);
    // the segments that end in this thread's positions
    double rs = carry.s, rr = carry.r;
#pragma unroll
    for (int k = 0; k < kRiItems; ++k) {
        if (gv[k] < 0) break;
        if (gv[k] != (k == 0 ? gprev : gv[k - 1])) rs = rr = 0.0;
        rs += sv[k];
        rr += rv[k];
        const int64_t p = q0 + k;
        const int gnext = p + 1 >= p1 ? -1 : k + 1 < kRiItems ? gv[k + 1] : gs[p + 1];
        if (gnext != gv[k]) {
            const int g = gv[k];
            if (goff[g] < p0) { edge[4 * blockIdx.x] = rs; edge[4 * blockIdx.x + 1] = rr; }
            else if (goff[g + 1] > p1) { edge[4 * blockIdx.x + 2] = rs; edge[4 * blockIdx.x + 3] = rr; }
            else { S[g] = rs; R[g] = rr; }
        }
    }
}

// A warp per group: (S_g, R_g) -- the chunk's sums, or the pieces of a group that crosses chunks added in chunk order --
// then u_g = R_g / prec + z_g / sqrt(prec), prec = S_g + 1 / tau2 (an empty group draws from its prior), z_g the first
// normal of the stream (seed, 2^63 + g, call).  usq_part[b] = sum of u_g^2 over the CTA's groups, in group order.
// kChains: chain blockIdx.y, u, S, R at + c G, u_rec at + c rec_stride, usq_part at + c gridDim.x, edge at
// + 4 c nchunks, tau2 at + c, seed + c.
template <bool kChains>
static __global__ void __launch_bounds__(32 * kRiDrawWarps)
k_ri_draw_u(double *__restrict__ u, double *__restrict__ u_rec, double *__restrict__ usq_part,
            const double *__restrict__ S, const double *__restrict__ R, const double *__restrict__ edge,
            const int *__restrict__ goff, const double *__restrict__ tau2, int G, uint64_t seed, uint32_t call,
            int64_t rec_stride, int nchunks)
{
    BL_PDL_ENTER();
    if (kChains) {
        const unsigned ch = blockIdx.y;
        u += (size_t)ch * G;
        if (u_rec) u_rec += ch * rec_stride;
        usq_part += (size_t)ch * gridDim.x;
        S += (size_t)ch * G;
        R += (size_t)ch * G;
        edge += (size_t)ch * 4 * nchunks;
        tau2 += ch;
        seed += ch;
    }
    __shared__ double sq[kRiDrawWarps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = blockIdx.x * kRiDrawWarps + warp;
    double ug = 0.0;
    if (g < G) {
        const int a = goff[g], b = goff[g + 1];
        double s = 0.0, r = 0.0;
        if (b > a) {
            const int c0 = a / kRiChunk, c1 = (b - 1) / kRiChunk;
            if (c0 == c1) {
                s = S[g];
                r = R[g];
            } else {
                double hs = 0.0, hr = 0.0;
                for (int c = c0 + 1 + lane; c <= c1; c += 32) {
                    hs += edge[4 * (size_t)c];
                    hr += edge[4 * (size_t)c + 1];
                }
#pragma unroll
                for (int o = 16; o; o >>= 1) {
                    hs += __shfl_xor_sync(0xffffffffu, hs, o);
                    hr += __shfl_xor_sync(0xffffffffu, hr, o);
                }
                s = edge[4 * (size_t)c0 + 2] + hs;
                r = edge[4 * (size_t)c0 + 3] + hr;
            }
        }
        if (lane == 0) {
            const double prec = s + 1.0 / tau2[0];
            const double m = r / prec;
            PhiloxSource src;
            src.open(seed, kRiGroupObs0 + (uint64_t)g, call);
            ug = m + src.norm() / sqrt(prec);
            u[g] = ug;
            if (u_rec) u_rec[g] = ug;
        }
    }
    if (lane == 0) sq[warp] = ug * ug;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int v = 0; v < kRiDrawWarps; ++v) t += sq[v];
        usq_part[blockIdx.x] = t;
    }
}

// One CTA: sum of u_g^2 over the partials in a fixed order, then tau2 = (b0 + sum / 2) / gamma, gamma ~ Gamma(a0 + G/2, 1)
// from the stream (seed, 2^64 - 4, call) (Marsaglia-Tsang, PhiloxSource::gamma).  kChains: chain blockIdx.x, tau2 at
// + c, tau2_rec at + c rec_stride, usq_part at + c nparts, seed + c.
template <bool kChains>
static __global__ void __launch_bounds__(256)
k_ri_draw_tau2(double *__restrict__ tau2, double *__restrict__ tau2_rec, const double *__restrict__ usq_part, int nparts,
               int G, double a0, double b0, uint64_t seed, uint32_t call, int64_t rec_stride)
{
    BL_PDL_ENTER();
    if (kChains) {
        const unsigned ch = blockIdx.x;
        tau2 += ch;
        if (tau2_rec) tau2_rec += ch * rec_stride;
        usq_part += (size_t)ch * nparts;
        seed += ch;
    }
    __shared__ double red[256];
    double s = 0.0;
    for (int k = threadIdx.x; k < nparts; k += 256) s += usq_part[k];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        PhiloxSource src;
        src.open(seed, kRiTau2Obs, call);
        const double t2 = (b0 + 0.5 * red[0]) / src.gamma(a0 + 0.5 * (double)G);
        *tau2 = t2;
        if (tau2_rec) *tau2_rec = t2;
    }
}

// The rows after the u draw: off_i = u_{g_i} (the next iteration's psi offset), v_i = kappa_i - omega_i off_i.
// kChains: chain blockIdx.y, off, v, omega at + c N, u at + c G.
template <bool kChains>
static __global__ void k_ri_rows(double *__restrict__ off, double *__restrict__ v, const int *__restrict__ group,
                                 const double *__restrict__ u, const double *__restrict__ w,
                                 const double *__restrict__ kappa, int64_t N, int G)
{
    BL_PDL_ENTER();
    if (kChains) {
        const size_t ch = (size_t)blockIdx.y * N;
        off += ch;
        v += ch;
        w += ch;
        u += (size_t)blockIdx.y * G;
    }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        const double ug = u[group[i]];
        off[i] = ug;
        v[i] = fma(-w[i], ug, kappa[i]);
    }
}

// Negative-binomial random intercepts (nb_ri_gibbs_device), after the dispersion step on phi = eta + off, with
// (d, log d) at dptr: psi <- phi - log d, eta <- eta - log d (so that k_ri_group_sums forms
// R_g = sum (kappa_i - omega_i (eta_i - log d))), shape <- y + d, kappa <- (y - d)/2.
static __global__ void k_nb_ri_prepare(double *__restrict__ psi, double *__restrict__ eta, double *__restrict__ shape,
                                       double *__restrict__ kappa, const double *__restrict__ y,
                                       const double *__restrict__ dptr, int64_t N)
{
    BL_PDL_ENTER();
    const double d = dptr[0], ld = dptr[1];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        const double yi = y[i];
        psi[i] -= ld;
        eta[i] -= ld;
        shape[i] = yi + d;
        kappa[i] = 0.5 * (yi - d);
    }
}

}  // namespace bl
