/*
 * tests/ri_oracle/logit_ri_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Plain-loop restatement of the random-intercept logit chain (bl_logit_ri_gibbs):
 *   logit P(success_i) = x_i' beta + u_{g_i},  u_g ~ N(0, tau2),  beta ~ N(m0, P0^-1),  tau2 ~ IG(a0, b0).
 * Built from the oracle's own pieces -- its Philox streams, the Devroye PG draw, the Marsaglia-Tsang gamma, the
 * weighted Gram and the plain beta draw of oracle/gibbs_oracle.c, included here so that the shared oracle stays as it
 * is.  Iteration t (0-based, burn-in included), from beta = 0, u = 0, tau2 = tau2_0:
 *   1. eta = X beta; omega_i = PG(n_i, eta_i + u_{g_i})               stream (seed, i, t)
 *   2. S_g = sum omega_i, R_g = sum (kappa_i - omega_i eta_i) over the rows of g in row order;
 *      prec = S_g + 1/tau2, u_g = R_g / prec + z_g / sqrt(prec)       z_g: first normal of (seed, 2^63 + g, t)
 *   3. tau2 = (b0 + sum_g u_g^2 / 2) / gamma, gamma ~ Gamma(a0 + G/2, 1) from (seed, 2^64 - 4, t)
 *   4. beta ~ N(Q^-1 r, Q^-1), Q = P0 + X' Omega X, r = P0 m0 + X'(kappa - omega o u_g)   (seed, 2^64 - 1, t)
 * kappa_i - omega_i eta_i and kappa_i - omega_i u_g are single fused multiply-adds, as the engine forms them.
 * Iteration t >= burn goes to row t - burn of beta [samp][P], u [samp][G] (may be NULL) and tau2 [samp].
 */
#include "gibbs_oracle.c"

#define RI_GROUP_OBS0 0x8000000000000000ull
#define RI_TAU2_OBS 0xFFFFFFFFFFFFFFFCull

int pgb_logit_ri_gibbs(double *beta, double *u_out, double *tau2_out, const double *y, const double *tX,
                       const double *n, const int *group, int G, const double *m0, const double *P0, double a0,
                       double b0, double tau2_0, int N, int P, int samp, int burn, uint64_t seed, int nthreads)
{
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#else
    nthreads = 1;
#endif
    double *bprior = (double *)calloc(P, sizeof(double));
    double *bP = (double *)malloc(sizeof(double) * P);
    double *PP = (double *)malloc(sizeof(double) * P * P);
    double *bcur = (double *)calloc(P, sizeof(double));
    double *kappa = (double *)malloc(sizeof(double) * N);
    double *eta = (double *)malloc(sizeof(double) * N);
    double *w = (double *)malloc(sizeof(double) * N);
    double *u = (double *)calloc(G, sizeof(double));
    double *S = (double *)malloc(sizeof(double) * G);
    double *R = (double *)malloc(sizeof(double) * G);
    double tau2 = tau2_0;
    for (int a = 0; a < P; ++a)
        for (int b = 0; b < P; ++b) bprior[a] += P0[a + P * b] * m0[b];
    for (int i = 0; i < N; ++i) kappa[i] = n[i] * (y[i] - 0.5);
    int status = 0;
    for (int t = 0; t < samp + burn && !status; ++t) {
        xbeta(eta, tX, bcur, N, P, nthreads);
#pragma omp parallel for schedule(dynamic, 256) num_threads(nthreads)
        for (int i = 0; i < N; ++i) {
            pgo_src s;
            pgo_src_philox(&s, seed, (uint64_t)i, (uint32_t)t);
            w[i] = pgo_dev_draw(&s, (int)n[i], eta[i] + u[group[i]]);
        }
        for (int g = 0; g < G; ++g) S[g] = R[g] = 0.0;
        for (int i = 0; i < N; ++i) {
            S[group[i]] += w[i];
            R[group[i]] += fma(-w[i], eta[i], kappa[i]);
        }
        double usq = 0.0;
        for (int g = 0; g < G; ++g) {
            double prec = S[g] + 1.0 / tau2;
            double m = R[g] / prec;
            pgo_src sz;
            pgo_src_philox(&sz, seed, RI_GROUP_OBS0 + (uint64_t)g, (uint32_t)t);
            u[g] = m + pgo_norm(&sz) / sqrt(prec);
            usq += u[g] * u[g];
        }
        pgo_src sg;
        pgo_src_philox(&sg, seed, RI_TAU2_OBS, (uint32_t)t);
        tau2 = (b0 + 0.5 * usq) / pgo_gamma(&sg, a0 + 0.5 * (double)G);
        weighted_gram(PP, P0, tX, w, N, P, nthreads);
        memcpy(bP, bprior, sizeof(double) * P);
        for (int i = 0; i < N; ++i) {
            double v = fma(-w[i], u[group[i]], kappa[i]);
            for (int a = 0; a < P; ++a) bP[a] += tX[a + (size_t)P * i] * v;
        }
        pgo_src sb;
        pgo_src_philox(&sb, seed, BETA_OBS, (uint32_t)t);
        status = draw_beta_plain(bcur, PP, bP, P, &sb);
        if (t >= burn) {
            memcpy(beta + (size_t)P * (t - burn), bcur, sizeof(double) * P);
            if (u_out) memcpy(u_out + (size_t)G * (t - burn), u, sizeof(double) * G);
            tau2_out[t - burn] = tau2;
        }
    }
    free(bprior); free(bP); free(PP); free(bcur); free(kappa); free(eta); free(w); free(u); free(S); free(R);
    return status;
}
