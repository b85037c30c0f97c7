"""The CPU restatement of the random-intercept negative-binomial chain (tests/ri_oracle/nb_ri_oracle.c) on simulated
data: it recovers the truth, and groups without rows draw u from the prior.  Deterministic at a fixed seed."""
import numpy as np

import _nb_ri_oracle as ro


def simulate(N, G, tau, beta, d, seed, ids=None):
    rng = np.random.default_rng(seed)
    P = len(beta)
    X = np.c_[np.ones(N), rng.standard_normal((N, P - 1))]
    u = rng.standard_normal(G)
    u = tau * (u - u.mean()) / u.std()                  # the realised intercepts have mean 0 and sd tau exactly
    g = rng.integers(0, G, N) if ids is None else ids
    mu = np.exp(X @ beta + u[g])
    return X, rng.negative_binomial(d, d / (mu + d)).astype(float), g, u


def test_recovers_beta_tau_and_d():
    """N = 20 000, G = 40, tau = 0.7, d = 3, P = 3 with an intercept, integer walk from d0 = 1: the posterior means of
    beta lie within 0.15 of the truth, sqrt(E[tau2]) within [0.5, 0.95] (40 groups pin tau to about +-12 %), E[d]
    within 0.5 of 3, and the posterior-mean u correlate with the true u above 0.95.  The true intercept is 0, where
    the chain starts: with 500 rows a group the chain moves along the intercept / mean-of-u ridge by a fraction of a
    per cent per iteration (the centred parametrisation), so a level far from the start would not be reached within
    the run (DESIGN.md section 11)."""
    beta = np.array([0.0, 0.5, -0.5])
    X, y, g, ut = simulate(20_000, 40, 0.7, beta, 3.0, 21)
    b, u, t2, d = ro.nb_ri(y, X, g, 40, np.zeros(3), 0.01 * np.eye(3), 2.0, 0.5, 1.0, 800, 200, 5, d0=1.0,
                           dmode="int")
    bm = b.mean(0)
    assert np.all(np.abs(bm - beta) < 0.15), bm
    assert 0.5 < np.sqrt(t2.mean()) < 0.95, t2.mean()
    assert abs(d.mean() - 3.0) < 0.5, d.mean()
    assert np.all(d == np.round(d)) and np.all(d >= 1)
    assert np.corrcoef(u.mean(0), ut)[0, 1] > 0.95
    assert u.shape == (800, 40) and np.all(np.isfinite(u))


def test_empty_groups_draw_from_the_prior():
    """Groups 20..29 hold no rows: their u draws have mean 0 and variance E[tau2] (tau2 of the iteration before),
    each within 5 standard errors (one effective draw per iteration for the variance, as the ten groups share
    tau2)."""
    rng = np.random.default_rng(3)
    ids = rng.integers(0, 20, 2000)
    X, y, g, _ = simulate(2000, 20, 0.7, np.array([0.0, 0.5]), 3.0, 4, ids=ids)
    samp = 4000
    b, u, t2, d = ro.nb_ri(y, X, g, 30, np.zeros(2), 0.01 * np.eye(2), 2.0, 1.0, 1.0, samp, 200, 9, d0=3.0,
                           dmode="fixed")
    assert np.all(d == 3.0)
    e = u[1:, 20:]                                       # u of iteration t was drawn with tau2 of iteration t - 1
    var_ref = t2[:-1].mean()
    assert abs(e.mean()) < 5 * np.sqrt(var_ref / e.size), (e.mean(), var_ref)
    sq = (e ** 2).mean(axis=1)
    assert abs(sq.mean() - var_ref) < 5 * sq.std() / np.sqrt(len(sq)), (sq.mean(), var_ref)
    assert np.all(u[:, :20].std(axis=0) < np.sqrt(var_ref))    # groups with rows are pinned down by their data
