"""The CPU restatement of the random-intercept logit chain (tests/ri_oracle/logit_ri_oracle.c) on simulated data:
it recovers the truth, and groups without rows draw u from the prior.  Deterministic at a fixed seed."""
import numpy as np

import _logit_ri_oracle as ro


def simulate(N, G, tau, beta, seed, ids=None):
    rng = np.random.default_rng(seed)
    P = len(beta)
    X = np.c_[np.ones(N), rng.standard_normal((N, P - 1))]
    u = rng.standard_normal(G)
    u = tau * (u - u.mean()) / u.std()                  # the realised intercepts have mean 0 and sd tau exactly
    g = rng.integers(0, G, N) if ids is None else ids
    p = 1.0 / (1.0 + np.exp(-(X @ beta + u[g])))
    return X, rng.binomial(1, p).astype(float), g


def test_recovers_beta_and_tau():
    """N = 3000, G = 30, tau = 1, P = 3 with an intercept: the posterior means of beta lie within 0.25 of the truth
    (about 3 posterior sd for the intercept, 5 for the slopes) and sqrt(E[tau2]) within [0.6, 1.6] (G = 30 groups
    pin tau to about +-25 %)."""
    beta = np.array([-0.5, 1.0, -0.7])
    X, y, g = simulate(3000, 30, 1.0, beta, 11)
    b, u, t2 = ro.logit_ri(y, X, np.ones(len(y)), g, 30, np.zeros(3), 0.01 * np.eye(3), 2.0, 2.0, 1.0, 2000, 300, 5)
    assert np.all(np.abs(b.mean(0) - beta) < 0.25), b.mean(0)
    assert 0.6 < np.sqrt(t2.mean()) < 1.6, t2.mean()
    assert u.shape == (2000, 30) and np.all(np.isfinite(u))


def test_empty_groups_draw_from_the_prior():
    """Groups 20..29 hold no rows: their u draws have mean 0 and variance E[tau2] (tau2 of the iteration before),
    each within 5 standard errors (one effective draw per iteration for the variance, as the ten groups share
    tau2)."""
    rng = np.random.default_rng(3)
    ids = rng.integers(0, 20, 2000)
    X, y, g = simulate(2000, 20, 1.0, np.array([0.2, 0.8]), 4, ids=ids)
    samp = 4000
    b, u, t2 = ro.logit_ri(y, X, np.ones(len(y)), g, 30, np.zeros(2), 0.01 * np.eye(2), 2.0, 2.0, 1.0, samp, 200, 9)
    e = u[1:, 20:]                                       # u of iteration t was drawn with tau2 of iteration t - 1
    var_ref = t2[:-1].mean()
    assert abs(e.mean()) < 5 * np.sqrt(var_ref / e.size), (e.mean(), var_ref)
    sq = (e ** 2).mean(axis=1)
    assert abs(sq.mean() - var_ref) < 5 * sq.std() / np.sqrt(len(sq)), (sq.mean(), var_ref)
    assert np.all(u[:, :20].std(axis=0) < np.sqrt(var_ref))    # groups with rows are pinned down by their data
