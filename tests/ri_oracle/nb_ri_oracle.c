/*
 * tests/ri_oracle/nb_ri_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Plain-loop restatement of the random-intercept negative-binomial chain (bl_nb_ri_gibbs):
 *   log mu_i = x_i' beta + u_{g_i},  y_i ~ NB(d, mu_i / (mu_i + d)),  u_g ~ N(0, tau2),  beta ~ N(m0, P0^-1),
 *   tau2 ~ IG(a0, b0).
 * Built from the oracle's own pieces -- its Philox streams, the rpg_hybrid draw, the dispersion targets df_llh and
 * dfreal_ll, the Marsaglia-Tsang gamma, the weighted Gram and the plain beta draw of oracle/gibbs_oracle.c, included
 * here so that the shared oracle stays as it is.  dmode 0 keeps d = d0, 1 draws it by draw.df (the random walk on the
 * integers), 2 by draw.df.real.mean (the walk on the reals).  Iteration t (0-based, burn-in included), from beta = 0,
 * u = 0, tau2 = tau2_0, d = d0:
 *   1. eta = X beta; phi_i = eta_i + u_{g_i}
 *   2. d | phi (dmode 1, 2), the dispersion step of nb_gibbs_df_impl on mu_i = exp(phi_i)    stream (seed, 2^64 - 2, t)
 *   3. psi_i = phi_i - log d, b_i = y_i + d, kappa_i = (y_i - d)/2; omega_i = PG(b_i, psi_i)   stream (seed, i, t)
 *   4. S_g = sum omega_i, R_g = sum (kappa_i - omega_i (eta_i - log d)) over the rows of g in row order;
 *      prec = S_g + 1/tau2, u_g = R_g / prec + z_g / sqrt(prec)       z_g: first normal of (seed, 2^63 + g, t)
 *   5. tau2 = (b0 + sum_g u_g^2 / 2) / gamma, gamma ~ Gamma(a0 + G/2, 1) from (seed, 2^64 - 4, t)
 *   6. beta ~ N(Q^-1 r, Q^-1), Q = P0 + X' Omega X, r = P0 m0 + X'(kappa - omega o u_g + omega log d)
 *                                                                      (seed, 2^64 - 1, t)
 * Rounding as the engine forms the per-row values: eta_i - log d and (eta_i + u_{g_i}) - log d are single roundings,
 * kappa_i - omega_i (eta_i - log d) and kappa_i - omega_i u_{g_i} are single fused multiply-adds.
 * Iteration t >= burn goes to row t - burn of beta [samp][P], u [samp][G] (may be NULL), tau2 [samp] and d [samp].
 */
#include "gibbs_oracle.c"

#define RI_GROUP_OBS0 0x8000000000000000ull
#define RI_TAU2_OBS 0xFFFFFFFFFFFFFFFCull

int pgb_nb_ri_gibbs(double *beta, double *u_out, double *tau2_out, double *d_out, const double *y, const double *tX,
                    const int *group, int G, const double *m0, const double *P0, double a0, double b0, double tau2_0,
                    double d0, int dmode, int N, int P, int samp, int burn, uint64_t seed, int nthreads)
{
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#else
    nthreads = 1;
#endif
    int ymax = 0;
    for (int i = 0; i < N; ++i) if ((int)y[i] > ymax) ymax = (int)y[i];
    double *Gs = (double *)calloc(ymax > 0 ? ymax : 1, sizeof(double));
    for (int i = 0; i < N; ++i)
        for (int j = 0; j < (int)y[i]; ++j) Gs[j] += 1.0;
    double *bprior = (double *)calloc(P, sizeof(double));
    double *bP = (double *)malloc(sizeof(double) * P);
    double *PP = (double *)malloc(sizeof(double) * P * P);
    double *bcur = (double *)calloc(P, sizeof(double));
    double *eta = (double *)malloc(sizeof(double) * N);
    double *phi = (double *)malloc(sizeof(double) * N);
    double *w = (double *)malloc(sizeof(double) * N);
    double *u = (double *)calloc(G, sizeof(double));
    double *S = (double *)malloc(sizeof(double) * G);
    double *R = (double *)malloc(sizeof(double) * G);
    double tau2 = tau2_0, d = d0;
    for (int a = 0; a < P; ++a)
        for (int b = 0; b < P; ++b) bprior[a] += P0[a + P * b] * m0[b];
    int status = 0;
    for (int t = 0; t < samp + burn && !status; ++t) {
        xbeta(eta, tX, bcur, N, P, nthreads);
        for (int i = 0; i < N; ++i) phi[i] = eta[i] + u[group[i]];
        if (dmode == 2) {          /* draw.df.real.mean */
            pgo_src sd;
            pgo_src_philox(&sd, seed, DF_OBS, (uint32_t)t);
            double un = pgo_unif(&sd);
            double rstar = d > 1.0 ? (d - 1.0) + 2.0 * un : 2.0 * un;
            double lalpha = dfreal_ll(y, rstar, phi, N) - dfreal_ll(y, d, phi, N);
            if (log(pgo_unif(&sd)) < lalpha) d = rstar;
        } else if (dmode == 1) {   /* draw.df */
            pgo_src sd;
            pgo_src_philox(&sd, seed, DF_OBS, (uint32_t)t);
            double lower = d - 1.0 > 1.0 ? d - 1.0 : 1.0;
            int nn = (int)(d + 1.0 - lower) + 1;
            int k = (int)floor(pgo_unif(&sd) * nn);
            if (k > nn - 1) k = nn - 1;
            double dp = lower + k;
            double ltarget = df_llh(y, dp, phi, Gs, ymax, N) - df_llh(y, d, phi, Gs, ymax, N);
            double lppsl = log(dp == 1.0 ? 0.5 : 1.0 / 3.0) - log(d == 1.0 ? 0.5 : 1.0 / 3.0);
            if (pgo_unif(&sd) < exp(ltarget + lppsl)) d = dp;
        }
        double ld = log(d);
#pragma omp parallel for schedule(dynamic, 256) num_threads(nthreads)
        for (int i = 0; i < N; ++i) {
            pgo_src s;
            pgo_src_philox(&s, seed, (uint64_t)i, (uint32_t)t);
            w[i] = pgo_hybrid_draw(&s, y[i] + d, phi[i] - ld);
        }
        for (int g = 0; g < G; ++g) S[g] = R[g] = 0.0;
        for (int i = 0; i < N; ++i) {
            S[group[i]] += w[i];
            R[group[i]] += fma(-w[i], eta[i] - ld, 0.5 * (y[i] - d));
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
            double v = fma(-w[i], u[group[i]], 0.5 * (y[i] - d)) + w[i] * ld;
            for (int a = 0; a < P; ++a) bP[a] += tX[a + (size_t)P * i] * v;
        }
        pgo_src sb;
        pgo_src_philox(&sb, seed, BETA_OBS, (uint32_t)t);
        status = draw_beta_plain(bcur, PP, bP, P, &sb);
        if (t >= burn) {
            memcpy(beta + (size_t)P * (t - burn), bcur, sizeof(double) * P);
            if (u_out) memcpy(u_out + (size_t)G * (t - burn), u, sizeof(double) * G);
            tau2_out[t - burn] = tau2;
            d_out[t - burn] = d;
        }
    }
    free(Gs); free(bprior); free(bP); free(PP); free(bcur); free(eta); free(phi); free(w); free(u); free(S); free(R);
    return status;
}
