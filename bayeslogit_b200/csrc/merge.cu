// Duplicate-row merge on the device (SURVEY.md section 8 row f1).
//
// Reference: Logit::compress (Logit.hpp:192-270) and the merge inside MultLogit::set_data
// (MultLogit.hpp:137-208), called by combine / mult_combine (LogitWrapper.cpp:279-310, 376-409) before every
// logit() / mlogit().  Observations with identical covariate rows collapse into the first one, in
// first-occurrence order: walking the later duplicates i in index order,
//     sum = n_f + n_i;  y_f = (n_f / sum) y_f + (n_i / sum) y_i;  n_f = sum.
// The reference does it with an O(N^2 P) list walk; here:
//   1. k_row_hash      64-bit hash of every row (a warp per row, coalesced; -0 hashes as +0)
//   2. k_hash_insert   open-addressing table keyed by the hash, value = smallest row index with that hash
//   3. k_resolve       rep[i] = that index if the two rows compare equal element by element (the reference's
//                      Matrix ==), else a conflict is flagged (hash collision, or rows holding NaN, which never
//                      equal themselves) and the caller falls back to the exact host merge
//   4. stable LSD radix sort of the row indices by rep: groups come out ordered by their first occurrence,
//      members in index order -- exactly the order the reference folds them in
//   5. k_fold          one thread per group replays the reference's running weighted mean with explicitly
//                      rounded operations (no FMA contraction): bit-identical y and n
//   6. k_gather_rows   the groups' first rows, compacted
// No library sort: the radix passes are two small kernels and a scan each.
#include <cuda_runtime.h>

#include <algorithm>
#include <string>
#include <vector>

#include "engine.h"

namespace bl {

namespace {

constexpr unsigned long long kEmpty = 0xFFFFFFFFFFFFFFFFull;

__device__ __forceinline__ unsigned long long mix64(unsigned long long x)
{
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;
    return x;
}

// hash[i] = sum over p of mix(bits(x_ip) + odd(p)): position dependent, order independent (a warp adds its lanes' parts)
__global__ void __launch_bounds__(256) k_row_hash(unsigned long long *__restrict__ hash, const double *__restrict__ tX, int N, int P)
{
    const int lane = threadIdx.x & 31;
    const int row = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (row >= N) return;
    unsigned long long h = 0;
    for (int p = lane; p < P; p += 32) {
        double v = tX[(size_t)row * P + p];
        if (v == 0.0) v = 0.0;                                   // -0 and +0 compare equal
        h += mix64((unsigned long long)__double_as_longlong(v) + 0x9E3779B97F4A7C15ull * (2ull * p + 1ull));
    }
    for (int o = 16; o; o >>= 1) h += __shfl_xor_sync(0xffffffffu, h, o);
    if (h == kEmpty) h = kEmpty - 1;
    if (lane == 0) hash[row] = h;
}

__global__ void k_hash_insert(unsigned long long *__restrict__ keys, int *__restrict__ first,
                              const unsigned long long *__restrict__ hash, int N, unsigned mask)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const unsigned long long h = hash[i];
    unsigned s = (unsigned)(h >> 17) & mask;
    for (;;) {
        const unsigned long long prev = atomicCAS(&keys[s], kEmpty, h);
        if (prev == kEmpty || prev == h) { atomicMin(&first[s], i); return; }
        s = (s + 1) & mask;
    }
}

// a warp per row: rep[i] = first row with the same hash if the rows are equal, else flag a conflict
__global__ void __launch_bounds__(256) k_resolve(int *__restrict__ rep, int *__restrict__ conflict,
                                                 const unsigned long long *__restrict__ keys, const int *__restrict__ first,
                                                 const unsigned long long *__restrict__ hash, const double *__restrict__ tX,
                                                 int N, int P, unsigned mask)
{
    const int lane = threadIdx.x & 31;
    const int row = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (row >= N) return;
    const unsigned long long h = hash[row];
    unsigned s = (unsigned)(h >> 17) & mask;
    while (keys[s] != h) s = (s + 1) & mask;
    const int f = first[s];
    bool same = true;
    if (f != row)
        for (int p = lane; p < P; p += 32) same = same && (tX[(size_t)row * P + p] == tX[(size_t)f * P + p]);
    same = __all_sync(0xffffffffu, same);
    if (lane == 0) {
        rep[row] = same ? f : row;
        if (!same) atomicExch(conflict, 1);
    }
}

// ---- exclusive scan of int32 (three kernels, 1024-element tiles) ------------------------------------
__global__ void __launch_bounds__(256) k_scan_tiles(int *__restrict__ out, int *__restrict__ tile_sum, const int *__restrict__ in, int n)
{
    __shared__ int wsum[8];
    const int base = blockIdx.x * 1024 + threadIdx.x * 4;
    int v[4], s = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) { v[k] = base + k < n ? in[base + k] : 0; s += v[k]; }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = s;
    for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int w = lane < 8 ? wsum[lane] : 0, wi = w;
        for (int o = 1; o < 8; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += t; }
        if (lane < 8) wsum[lane] = wi - w;
        if (lane == 7 && tile_sum) tile_sum[blockIdx.x] = wi;
    }
    __syncthreads();
    int run = wsum[warp] + inc - s;
#pragma unroll
    for (int k = 0; k < 4; ++k) { if (base + k < n) out[base + k] = run; run += v[k]; }
}

// one CTA: exclusive scan of the tile sums in place (sequential over 1024-element pieces)
__global__ void __launch_bounds__(1024) k_scan_top(int *__restrict__ a, int n, int *__restrict__ total)
{
    __shared__ int wsum[32];
    __shared__ int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int b = 0; b < n; b += 1024) {
        const int i = b + threadIdx.x;
        const int v = i < n ? a[i] : 0;
        int inc = v;
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        if (lane == 31) wsum[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            int w = wsum[lane], wi = w;
            for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += t; }
            wsum[lane] = wi - w;
        }
        __syncthreads();
        const int c = carry;
        if (i < n) a[i] = c + wsum[warp] + inc - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry = c + wsum[31] + inc;
        __syncthreads();
    }
    if (threadIdx.x == 0 && total) *total = carry;
}

__global__ void k_scan_add(int *__restrict__ out, const int *__restrict__ tile_off, int n)
{
    const int i = blockIdx.x * 1024 + threadIdx.x;
    if (i < n) out[i] += tile_off[blockIdx.x];
}

// ---- stable LSD radix sort of (key, value) by 8-bit digits ----------------------------------------------
constexpr int kSortTile = 2048;      // keys per block

__global__ void __launch_bounds__(256) k_digit_hist(int *__restrict__ hist, const int *__restrict__ key, int n, int shift, int nblk)
{
    __shared__ int h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const int base = blockIdx.x * kSortTile;
    for (int k = threadIdx.x; k < kSortTile && base + k < n; k += 256) atomicAdd(&h[(key[base + k] >> shift) & 255], 1);
    __syncthreads();
    hist[(size_t)threadIdx.x * nblk + blockIdx.x] = h[threadIdx.x];      // digit-major: a scan gives the global offsets
}

// one warp walks the block's keys in order, 32 at a time: rank inside the row from __match_any, running counts
// per digit in shared memory -- equal digits keep their input order (stable)
__global__ void __launch_bounds__(32) k_digit_scatter(int *__restrict__ key_out, int *__restrict__ val_out,
                                                      const int *__restrict__ key, const int *__restrict__ val,
                                                      const int *__restrict__ offs, int n, int shift, int nblk)
{
    __shared__ int cnt[256];
    const int lane = threadIdx.x;
    for (int d = lane; d < 256; d += 32) cnt[d] = offs[(size_t)d * nblk + blockIdx.x];
    __syncwarp();
    const int base = blockIdx.x * kSortTile;
    for (int k0 = 0; k0 < kSortTile && base + k0 < n; k0 += 32) {
        const int i = base + k0 + lane;
        const bool ok = i < n;
        const int kv = ok ? key[i] : 0, d = ok ? (kv >> shift) & 255 : 256 + lane;     // idle lanes match nobody
        const unsigned m = __match_any_sync(0xffffffffu, d);
        const int rank = __popc(m & ((1u << lane) - 1u));
        int pos = 0;
        if (ok) pos = cnt[d] + rank;
        __syncwarp();
        if (ok && rank == 0) cnt[d] += __popc(m);
        __syncwarp();
        if (ok) { key_out[pos] = kv; val_out[pos] = val[i]; }
    }
}

__global__ void k_iota(int *__restrict__ a, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = i;
}

// head[k] = 1 where position k of the sorted order starts a group
__global__ void k_heads(int *__restrict__ head, const int *__restrict__ rep_sorted, int n)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) head[k] = (k == 0 || rep_sorted[k] != rep_sorted[k - 1]) ? 1 : 0;
}

// One thread per group: the reference's running weighted mean over the group's later members in index order.
// yo: ny x M, no: M (compacted); order[k] = row index at sorted position k; gpos[k] = group number of position k.
__global__ void k_fold(double *__restrict__ yo, double *__restrict__ no, int *__restrict__ first_row,
                       const double *__restrict__ ty, const double *__restrict__ n, const int *__restrict__ order,
                       const int *__restrict__ head, const int *__restrict__ gpos, int N, int ny)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N || !head[k]) return;
    const int g = gpos[k], f = order[k];
    double nf = n[f];
    for (int r = 0; r < ny; ++r) yo[(size_t)ny * g + r] = ty[(size_t)ny * f + r];
    for (int q = k + 1; q < N && !head[q]; ++q) {
        const int i = order[q];
        const double ni = n[i], sum = __dadd_rn(nf, ni);
        const double a = __ddiv_rn(nf, sum), b = __ddiv_rn(ni, sum);
        for (int r = 0; r < ny; ++r)
            yo[(size_t)ny * g + r] = __dadd_rn(__dmul_rn(a, yo[(size_t)ny * g + r]), __dmul_rn(b, ty[(size_t)ny * i + r]));
        nf = sum;
    }
    no[g] = nf;
    first_row[g] = f;
}

__global__ void __launch_bounds__(256) k_gather_rows(double *__restrict__ out, const double *__restrict__ tX,
                                                     const int *__restrict__ first_row, int M, int P)
{
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (size_t)M * P) return;
    const int g = (int)(e / P), p = (int)(e % P);
    out[e] = tX[(size_t)first_row[g] * P + p];
}

#define MG_CK(expr)                                                                  \
    do {                                                                             \
        cudaError_t e_ = (expr);                                                     \
        if (e_ != cudaSuccess) { err = std::string(#expr) + ": " + cudaGetErrorString(e_); return -1; } \
    } while (0)

struct Bufs {
    std::vector<void *> p;
    ~Bufs() { for (void *q : p) cudaFree(q); }
    template <class T>
    cudaError_t get(T **out, size_t count)
    {
        void *q = nullptr;
        cudaError_t e = cudaMalloc(&q, (count ? count : 1) * sizeof(T));
        if (e == cudaSuccess) { p.push_back(q); *out = (T *)q; }
        return e;
    }
};

int cdiv(size_t a, size_t b) { return (int)((a + b - 1) / b); }

// out = exclusive scan of in (n ints); *total (device, optional) = the sum
int scan_exclusive(int *out, const int *in, int n, int *tile, int *total, cudaStream_t st)
{
    const int nt = cdiv(n, 1024);
    k_scan_tiles<<<nt, 256, 0, st>>>(out, tile, in, n);
    k_scan_top<<<1, 1024, 0, st>>>(tile, nt, total);
    k_scan_add<<<nt, 1024, 0, st>>>(out, tile, n);
    count_launch(3);
    return 0;
}

}  // namespace

// Stable LSD radix sort of (key, val) pairs by the low `bits` bits of key, 8 bits a pass.  The pointers are swapped
// pass by pass: on return key_a / val_a hold the sorted pairs.  hist: 256 cdiv(n, kSortTile) ints; tile: scan scratch
// of cdiv(max(n, 256 cdiv(n, kSortTile)), 1024) + 1 ints.
static void radix_sort_pairs(int *&key_a, int *&val_a, int *&key_b, int *&val_b, int n, int bits, int *hist, int *tile,
                             cudaStream_t st)
{
    const int nblk = cdiv(n, kSortTile);
    for (int shift = 0; shift < bits; shift += 8) {
        k_digit_hist<<<nblk, 256, 0, st>>>(hist, key_a, n, shift, nblk);
        scan_exclusive(hist, hist, 256 * nblk, tile, nullptr, st);
        k_digit_scatter<<<nblk, 32, 0, st>>>(key_b, val_b, key_a, val_a, hist, n, shift, nblk);
        count_launch(2);
        std::swap(key_a, key_b);
        std::swap(val_a, val_b);
    }
}

int sort_rows_by_key(int *order, int *key_sorted, const int *key, int n, int nkeys, cudaStream_t st, std::string &err)
{
    if (n <= 0) return 0;
    const int nblk = cdiv(n, kSortTile);
    int bits = 1;
    while ((1ll << bits) < nkeys) ++bits;
    int *scratch = nullptr;
    const size_t tile_n = (size_t)cdiv(std::max((size_t)n, (size_t)256 * nblk), 1024) + 1;
    cudaError_t e = cudaMallocAsync((void **)&scratch, sizeof(int) * (2 * (size_t)n + (size_t)256 * nblk + tile_n), st);
    if (e != cudaSuccess) { err = std::string("sort_rows_by_key scratch: ") + cudaGetErrorString(e); return 1; }
    int *key_a = key_sorted, *val_a = order, *key_b = scratch, *val_b = scratch + n;
    int *hist = scratch + 2 * (size_t)n, *tile = hist + (size_t)256 * nblk;
    e = cudaMemcpyAsync(key_a, key, sizeof(int) * n, cudaMemcpyDeviceToDevice, st);
    k_iota<<<cdiv(n, 256), 256, 0, st>>>(val_a, n);
    count_launch();
    radix_sort_pairs(key_a, val_a, key_b, val_b, n, bits, hist, tile, st);
    if (e == cudaSuccess && key_a != key_sorted) {
        e = cudaMemcpyAsync(key_sorted, key_a, sizeof(int) * n, cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(order, val_a, sizeof(int) * n, cudaMemcpyDeviceToDevice, st);
    }
    cudaFreeAsync(scratch, st);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) { err = std::string("sort_rows_by_key: ") + cudaGetErrorString(e); return 1; }
    return 0;
}

// Device-resident merge.  ty (ny x N), tX (P x N), n (N) are overwritten with the M merged observations in
// first-occurrence order; returns M, -1 on a CUDA error (message in err), -2 when the rows need the exact host
// merge (a hash collision, or rows holding NaN): the inputs are then untouched.
int merge_rows_device(double *ty, double *tX, double *n, int N, int P, int ny, cudaStream_t st, std::string &err)
{
    if (N <= 0) return 0;
    Bufs b;
    unsigned long long *hash, *keys;
    int *first, *rep, *conflict, *idx_a, *idx_b, *key_a, *key_b, *hist, *tile, *head, *gpos, *total, *first_row;
    unsigned cap = 1024;
    while (cap < 2u * (unsigned)N) cap <<= 1;
    const int nblk = cdiv(N, kSortTile);
    MG_CK(b.get(&hash, N)); MG_CK(b.get(&keys, cap)); MG_CK(b.get(&first, cap)); MG_CK(b.get(&rep, N));
    MG_CK(b.get(&conflict, 1)); MG_CK(b.get(&idx_a, N)); MG_CK(b.get(&idx_b, N)); MG_CK(b.get(&key_a, N)); MG_CK(b.get(&key_b, N));
    MG_CK(b.get(&hist, (size_t)256 * nblk)); MG_CK(b.get(&tile, (size_t)cdiv(std::max((size_t)N, (size_t)256 * nblk), 1024) + 1));
    MG_CK(b.get(&head, N)); MG_CK(b.get(&gpos, N)); MG_CK(b.get(&total, 1)); MG_CK(b.get(&first_row, N));
    MG_CK(cudaMemsetAsync(keys, 0xFF, sizeof(unsigned long long) * cap, st));
    MG_CK(cudaMemsetAsync(first, 0x7F, sizeof(int) * cap, st));
    MG_CK(cudaMemsetAsync(conflict, 0, sizeof(int), st));
    k_row_hash<<<cdiv((size_t)N * 32, 256), 256, 0, st>>>(hash, tX, N, P);
    k_hash_insert<<<cdiv(N, 256), 256, 0, st>>>(keys, first, hash, N, cap - 1);
    k_resolve<<<cdiv((size_t)N * 32, 256), 256, 0, st>>>(rep, conflict, keys, first, hash, tX, N, P, cap - 1);
    count_launch(3);
    int hconf = 0;
    MG_CK(cudaMemcpyAsync(&hconf, conflict, sizeof(int), cudaMemcpyDeviceToHost, st));
    MG_CK(cudaStreamSynchronize(st));
    if (hconf) return -2;
    // stable sort of the row indices by rep
    int bits = 1;
    while ((1ll << bits) < N) ++bits;
    k_iota<<<cdiv(N, 256), 256, 0, st>>>(idx_a, N);
    MG_CK(cudaMemcpyAsync(key_a, rep, sizeof(int) * N, cudaMemcpyDeviceToDevice, st));
    count_launch();
    radix_sort_pairs(key_a, idx_a, key_b, idx_b, N, bits, hist, tile, st);
    k_heads<<<cdiv(N, 256), 256, 0, st>>>(head, key_a, N);
    scan_exclusive(gpos, head, N, tile, total, st);
    int M = 0;
    MG_CK(cudaMemcpyAsync(&M, total, sizeof(int), cudaMemcpyDeviceToHost, st));
    MG_CK(cudaStreamSynchronize(st));
    count_launch();
    if (M == N) return N;                                  // nothing to merge: the inputs already are the answer
    double *yo, *no, *xo;
    MG_CK(b.get(&yo, (size_t)ny * M)); MG_CK(b.get(&no, M)); MG_CK(b.get(&xo, (size_t)P * M));
    k_fold<<<cdiv(N, 128), 128, 0, st>>>(yo, no, first_row, ty, n, idx_a, head, gpos, N, ny);
    k_gather_rows<<<cdiv((size_t)M * P, 256), 256, 0, st>>>(xo, tX, first_row, M, P);
    count_launch(2);
    MG_CK(cudaMemcpyAsync(ty, yo, sizeof(double) * ny * M, cudaMemcpyDeviceToDevice, st));
    MG_CK(cudaMemcpyAsync(n, no, sizeof(double) * M, cudaMemcpyDeviceToDevice, st));
    MG_CK(cudaMemcpyAsync(tX, xo, sizeof(double) * (size_t)P * M, cudaMemcpyDeviceToDevice, st));
    MG_CK(cudaStreamSynchronize(st));
    MG_CK(cudaGetLastError());
    return M;
}

}  // namespace bl
