// Batch Polya-Gamma draw kernels (sm_100a).
//
// One lane per observation, grid-stride.  Replaces the serial host loops
// rpg_gamma / rpg_devroye / rpg_alt / rpg_sp / rpg_hybrid of the reference
// (LogitWrapper.cpp:39-167).  HBM traffic per draw: z (8 B) + shape (4 or 8 B)
// in, omega (8 B) out, all coalesced; the kernels are bound by the fp64/ALU
// pipes, not by HBM (DESIGN.md "Rooflines").
#include "engine.h"
#include "pg_devroye_fast.cuh"
#include "pg_stream.cuh"

namespace bl {

namespace {

constexpr int kThreads = 128;

inline int grid_for(int64_t num, int threads, int ctas_per_sm)
{
    int64_t need = (num + threads - 1) / threads;
    int64_t cap = 148LL * ctas_per_sm;  // B200: 148 SMs
    return (int)(need < cap ? (need > 0 ? need : 1) : cap);
}

template <int M, class Src>
__device__ __forceinline__ double draw_one(Src &s, const void *shape, const double *z, int64_t i,
                                           int trunc, int *iter, int &aux)
{
    aux = 0;
    if (M == kDevroye || M == kDevroyeLoop) {
        int n = ((const int *)shape)[i];
        return n != 0 ? devroye_sum_fast(s, n, z[i]) : 0.0;
    } else if (M == kDevroyePlain) {
        int n = ((const int *)shape)[i];
        return n != 0 ? devroye_sum(s, n, z[i]) : 0.0;
    } else if (M == kGamma) {
        double n = ((const double *)shape)[i];
        return n != 0.0 ? gamma_sum(s, n, z[i], trunc) : 0.0;
    } else if (M == kAlt) {
        double h = ((const double *)shape)[i];
        return h != 0 ? alt_draw(s, h, z[i]) : 0.0;
    } else if (M == kSP) {
        double h = ((const double *)shape)[i];
        if (h != 0) {
            double d;
            aux = sp_draw(s, d, h, z[i]);
            if (iter) iter[i] = aux;
            return d;
        }
        return 0.0;
    } else {
        double h = ((const double *)shape)[i];
        return hybrid_draw(s, h, z[i], aux);
    }
}

// kChains: the batch holds independent chains side by side and id.chain_len keys their streams (open_batch_stream;
// batch < 2^31); a compile-time switch, so that the single-batch instantiations keep their code.
template <int M, bool kChains = false>
__global__ void __launch_bounds__(kThreads)
k_rpg_philox(double *__restrict__ x, const void *__restrict__ shape, const double *__restrict__ z,
             int64_t num, int trunc, int *__restrict__ iter, StreamId id)
{
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < num; i += stride) {
        PhiloxSource s;
        if (kChains) open_batch_stream(s, id, i);
        else s.open(id.seed, id.obs0 + (uint64_t)i, id.call_id);
        int aux;
        x[i] = draw_one<M>(s, shape, z, i, trunc, iter, aux);
    }
}

template <int M>
__global__ void __launch_bounds__(kThreads)
k_rpg_tape(double *__restrict__ x, const void *__restrict__ shape, const double *__restrict__ z,
           int64_t num, int trunc, int *__restrict__ iter, DevTape tp, int *__restrict__ trace)
{
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < num; i += stride) {
        TapeSource s;
        s.open(tp.tu, tp.lu, tp.te, tp.le, tp.tn, tp.ln, tp.tg, tp.lg, (size_t)i);
        int aux;
        double v = draw_one<M>(s, shape, z, i, trunc, iter, aux);
        x[i] = s.exhausted() ? nan("") : v;
        if (trace) {
            int *t = trace + i * BL_TRACE_W;
            s.counts(t);
            t[4] = s.exhausted() ? 1 : 0;
            t[5] = aux;
        }
    }
}

__global__ void k_probe_moments(double *m1, double *m2, const double *b, const double *z, int64_t num)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < num) {
        m1[i] = pg_m1(b[i], z[i]);
        m2[i] = pg_m2(b[i], z[i]);
    }
}

__global__ void k_probe_v_eval(double *v, const double *y, int64_t num)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < num) v[i] = v_eval(y[i]);
}

// which: 0 Phi(a), 1 log Phi(a), 2 P(shape=b, a*c) [= RNG::p_gamma_rate(a,b,c)],
//        3 p_igauss(a, mu=b, lambda=c), 4 lgamma(a), 5 tgamma(a), 6 right mass of the
//        Devroye proposal at Z=a, 7 Devroye coefficient a_n(x): n=b, x=a,
//        8 Gamma(b, a) e^a a^-b by the forward continued fraction (a >= b + 1),
//        9 p_igauss_direct(a, mu=b, lambda=c), 10 log cos_rt(v(a)) as the saddle-point sampler
//        takes it (table or reference iteration), 11 v(a) from the table path alone (NaN where
//        the table path hands over to the reference iteration), 12 / 13 mass of the saddle-point
//        sampler's left piece for shape a, tilt b: fp64, and the fp32 estimate (NaN: none offered),
//        14 / 15 mass of the alternate sampler's right piece for chunk shape a in [1,4], tilt b: same pair
__global__ void k_probe_specfun(double *out, int which, const double *a, const double *b,
                                const double *c, int64_t num)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= num) return;
    double r = 0.0;
    switch (which) {
    case 0: r = p_norm(a[i]); break;
    case 1: r = log_p_norm(a[i]); break;
    case 2: r = p_gamma_rate(a[i], b[i], c[i]); break;
    case 3: r = p_igauss(a[i], b[i], c[i]); break;
    case 4: r = lgamma(a[i]); break;
    case 5: r = tgamma(a[i]); break;
    case 6: r = dev_right_mass(a[i]); break;
    case 7: r = dev_coef((int)b[i], a[i]); break;
    case 8: r = upper_gamma_cf(b[i], a[i]); break;
    case 9: r = p_igauss_direct(a[i], b[i], c[i]); break;
    case 10: { double v, g; sp_vg(a[i], v, g); r = g; break; }
    case 11: { double v, g; r = sp_vg_table(a[i], v, g) ? v : nan(""); break; }
    case 12: { SpState st; sp_setup<false>(a[i], b[i], st); r = st.f[kSpPl]; break; }
    case 13: { SpState st; sp_setup<true>(a[i], b[i], st); r = st.f[kSpPlBand] > 0.0 ? st.f[kSpPl] : nan(""); break; }
    case 14: { double f[kAltSetupDoubles]; alt_setup<false>(a[i], 0.5 * fabs(b[i]), f); r = f[kAltPr]; break; }
    case 15: { double f[kAltSetupDoubles]; alt_setup<true>(a[i], 0.5 * fabs(b[i]), f); r = f[kAltPrBand] > 0.0 ? f[kAltPr] : nan(""); break; }
    }
    out[i] = r;
}

__global__ void k_probe_philox(uint32_t *out4, const uint32_t *ctr4, const uint32_t *key2)
{
    uint4 r = Philox4x32::block(make_uint4(ctr4[0], ctr4[1], ctr4[2], ctr4[3]),
                                make_uint2(key2[0], key2[1]));
    out4[0] = r.x; out4[1] = r.y; out4[2] = r.z; out4[3] = r.w;
}

template <int M, bool kChains = false>
cudaError_t launch_philox_m(double *x, const void *shape, const double *z, int64_t num, int trunc,
                            int *iter, StreamId id, cudaStream_t st)
{
    if (num <= 0) return cudaSuccess;
    k_rpg_philox<M, kChains><<<grid_for(num, kThreads, 16), kThreads, 0, st>>>(x, shape, z, num, trunc, iter, id);
    count_launch();
    return cudaGetLastError();
}

template <int M>
cudaError_t launch_tape_m(double *x, const void *shape, const double *z, int64_t num, int trunc,
                          int *iter, DevTape tp, int *trace, cudaStream_t st)
{
    if (num <= 0) return cudaSuccess;
    k_rpg_tape<M><<<grid_for(num, kThreads, 16), kThreads, 0, st>>>(x, shape, z, num, trunc, iter, tp, trace);
    count_launch();
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_rpg(Method m, double *x, const void *shape, const double *z, int64_t num,
                       int trunc, int *iter, StreamId id, cudaStream_t st)
{
    switch (m) {
    case kDevroye: return launch_devroye_refill(x, (const int *)shape, z, num, id, st);
    case kDevroyeLoop: return launch_philox_m<kDevroyeLoop>(x, shape, z, num, trunc, iter, id, st);
    case kGamma: return launch_philox_m<kGamma>(x, shape, z, num, trunc, iter, id, st);
    case kAlt: return launch_philox_m<kAlt>(x, shape, z, num, trunc, iter, id, st);
    case kSP: return launch_philox_m<kSP>(x, shape, z, num, trunc, iter, id, st);
    case kHybrid:
        return id.chain_len ? launch_philox_m<kHybrid, true>(x, shape, z, num, trunc, iter, id, st)
                            : launch_philox_m<kHybrid>(x, shape, z, num, trunc, iter, id, st);
    case kDevroyePlain: return launch_philox_m<kDevroyePlain>(x, shape, z, num, trunc, iter, id, st);
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_rpg_tape(Method m, double *x, const void *shape, const double *z, int64_t num,
                            int trunc, int *iter, DevTape tp, int *trace, cudaStream_t st)
{
    switch (m) {
    case kDevroye: return launch_tape_m<kDevroye>(x, shape, z, num, trunc, iter, tp, trace, st);
    case kGamma: return launch_tape_m<kGamma>(x, shape, z, num, trunc, iter, tp, trace, st);
    case kAlt: return launch_tape_m<kAlt>(x, shape, z, num, trunc, iter, tp, trace, st);
    case kSP: return launch_tape_m<kSP>(x, shape, z, num, trunc, iter, tp, trace, st);
    case kHybrid: return launch_tape_m<kHybrid>(x, shape, z, num, trunc, iter, tp, trace, st);
    case kDevroyePlain: return launch_tape_m<kDevroyePlain>(x, shape, z, num, trunc, iter, tp, trace, st);
    case kDevroyeLoop: return launch_tape_m<kDevroye>(x, shape, z, num, trunc, iter, tp, trace, st);
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_probe_moments(double *m1, double *m2, const double *b, const double *z,
                                 int64_t num, cudaStream_t st)
{
    if (num <= 0) return cudaSuccess;
    k_probe_moments<<<(unsigned)((num + 127) / 128), 128, 0, st>>>(m1, m2, b, z, num);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_probe_v_eval(double *v, const double *y, int64_t num, cudaStream_t st)
{
    if (num <= 0) return cudaSuccess;
    k_probe_v_eval<<<(unsigned)((num + 127) / 128), 128, 0, st>>>(v, y, num);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_probe_specfun(double *out, int which, const double *a, const double *b,
                                 const double *c, int64_t num, cudaStream_t st)
{
    if (num <= 0) return cudaSuccess;
    k_probe_specfun<<<(unsigned)((num + 127) / 128), 128, 0, st>>>(out, which, a, b, c, num);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_probe_philox(uint32_t *out4, const uint32_t *ctr4, const uint32_t *key2,
                                cudaStream_t st)
{
    k_probe_philox<<<1, 1, 0, st>>>(out4, ctr4, key2);
    count_launch();
    return cudaGetLastError();
}

}  // namespace bl
