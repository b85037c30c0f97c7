"""Host-side mirror of the reference's R front end for the Gibbs path.

    logit_combine  <- logit.combine   (Code/R/LogitWrapper.R:160-190)
    logit          <- logit           (:197-244)
    logit_EM       <- logit.EM        (:248-286)
    mlogit_combine <- mlogit.combine  (:325-352)
    mlogit         <- mlogit          (:358-416)

Same argument meaning and return structure (dicts for R lists, -1 / NaN where R
returns -1 / NA), same validation messages, and the same C calls R makes through
.C(): column-major host buffers, t(X) handed over as tX.
"""
import ctypes as C

import numpy as np

from . import _lib

NA = float("nan")

PLAIN_BETA = 1   # BL_GIBBS_PLAIN_BETA
NO_W = 2         # BL_GIBBS_NO_W
UNFUSED = 4      # BL_GIBBS_UNFUSED (psi = X beta and the omega draw as two kernels; A/B aid)
ONE_PASS = 8     # BL_GIBBS_ONE_PASS (psi, omega and the Gram from one TMA-staged read of X; even P <= 64)
TWO_PASS = 16    # BL_GIBBS_TWO_PASS (never the one-pass kernel)


def _f(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _p(a):
    return a.ctypes.data


def _ci(v):
    return C.c_int(int(v))


def check_parameters(y, n, m0, P0, RX, CX, samp, burn):
    """check.parameters, LogitWrapper.R:130-157."""
    P0 = np.atleast_2d(P0)
    ok = [np.all(y >= 0), np.all(n > 0), CX == P0.shape[0], CX == P0.shape[1],
          len(y) == len(n) and len(y) == RX, CX == np.size(m0), samp > 0, burn >= 0, np.all(y <= 1)]
    if not ok[0]: print("y must be >= 0.")
    if not ok[8]: print("y is a proportion; it must be <= 1.")
    if not ok[1]: print("n must be > 0.")
    if not ok[2]: print(f"col(X) != row(P0) {CX} {P0.shape[0]}")
    if not ok[3]: print(f"col(X) != col(P0) {CX} {P0.shape[1]}")
    if not ok[4]: print(f"Dimensions do not conform for y, X, and n. len(y) = {len(y)} dim(x) = {RX} {CX} len(n) = {len(n)}")
    if not ok[5]: print(f"col(X) != length(m0) {CX} {np.size(m0)}")
    if not ok[6]: print("samp must be > 0.")
    if not ok[7]: print("burn must be >=0.")
    return all(ok)


def logit_combine(y, X, n=None):
    X = np.atleast_2d(_f(X)) if np.ndim(X) > 1 else _f(X).reshape(-1, 1)
    y = _f(y).ravel()
    n = np.ones(len(y)) if n is None else _f(n).ravel()
    N, P = X.shape
    if not check_parameters(y, n, np.zeros(P), np.zeros((P, P)), N, P, 1, 0):
        return -1
    y, n = y.copy(), n.copy()
    tX = np.ascontiguousarray(X)          # row-major N x P == column-major P x N == t(X)
    tX = tX.copy()
    cN, cP = _ci(N), _ci(P)
    _lib.lib().combine(_p(y), _p(tX), _p(n), C.byref(cN), C.byref(cP))
    _lib.check()
    M = cN.value
    return {"y": y[:M].copy(), "X": tX.reshape(N, P)[:M].copy(), "n": n[:M].copy()}


def logit(y, X, n=None, m0=None, P0=None, samp=1000, burn=500):
    X = np.atleast_2d(_f(X)) if np.ndim(X) > 1 else _f(X).reshape(-1, 1)
    new = logit_combine(y, X, n)
    if not isinstance(new, dict):
        return -1
    y, X, n = new["y"], new["X"], new["n"]
    N, P = X.shape
    m0 = np.zeros(P) if m0 is None else _f(m0).ravel()
    P0 = np.zeros((P, P)) if P0 is None else _f(P0)
    if not check_parameters(y, n, m0, P0, N, P, samp, burn):
        return -1
    w = np.zeros((samp, N))          # C view of the column-major N x samp array
    beta = np.zeros((samp, P))
    tX = np.ascontiguousarray(X)
    P0c = np.asfortranarray(P0)
    cN = _ci(N)
    _lib.lib().gibbs(_p(w), _p(beta), _p(y), _p(tX), _p(n), _p(m0), P0c.ctypes.data,
                     C.byref(cN), C.byref(_ci(P)), C.byref(_ci(samp)), C.byref(_ci(burn)))
    _lib.check()
    return {"w": w, "beta": beta, "y": y, "X": X, "n": n}      # w: samp x N, beta: samp x P, as R returns


def logit_EM(y, X, n=None, tol=1e-9, max_iter=100):
    X = np.atleast_2d(_f(X)) if np.ndim(X) > 1 else _f(X).reshape(-1, 1)
    new = logit_combine(y, X, n)
    if not isinstance(new, dict):
        return -1
    y, X, n = new["y"], new["X"], new["n"]
    N, P = X.shape
    if not check_parameters(y, n, np.zeros(P), np.zeros((P, P)), N, P, 1, 0):
        return -1
    beta = np.zeros(P)
    tX = np.ascontiguousarray(X)
    it = _ci(max_iter)
    _lib.lib().EM(_p(beta), _p(y), _p(tX), _p(n), C.byref(_ci(N)), C.byref(_ci(P)),
                  C.byref(C.c_double(tol)), C.byref(it))
    _lib.check()
    return {"beta": beta, "iter": it.value}


def mult_check_parameters(y, X, n, m0, P0, samp, burn):
    """mult.check.parameters, LogitWrapper.R:294-321."""
    ok = [np.all(y >= 0), np.all(n > 0), y.shape[0] == len(n) and y.shape[0] == X.shape[0], samp > 0,
          burn >= 0, np.all(y.sum(axis=1) <= 1),
          y.shape[1] == m0.shape[1] and X.shape[1] == m0.shape[0],
          X.shape[1] == P0.shape[0] and X.shape[1] == P0.shape[1] and y.shape[1] == P0.shape[2]]
    if not ok[0]: print("y must be >= 0.")
    if not ok[5]: print("y[i,] are proportions and must sum <= 1.")
    if not ok[1]: print("n must be > 0.")
    if not ok[2]: print("Dimensions do not conform for y, X, and n.")
    if not ok[3]: print("samp must be > 0.")
    if not ok[4]: print("burn must be >=0.")
    if not ok[6]: print("m.0 does not conform.")
    if not ok[7]: print("P.0 does not conform.")
    return all(ok)


def mlogit_combine(y, X, n=None):
    X = np.atleast_2d(_f(X))
    y = _f(y)
    y = y.reshape(-1, 1) if y.ndim == 1 else y
    n = np.ones(y.shape[0]) if n is None else _f(n).ravel()
    N, P = X.shape
    U = y.shape[1]
    if not mult_check_parameters(y, X, n, np.zeros((P, U)), np.zeros((P, P, U)), 1, 0):
        return NA
    ty = np.ascontiguousarray(y).copy()      # row-major N x U == column-major U x N == t(y)
    tX = np.ascontiguousarray(X).copy()
    n = n.copy()
    cN = _ci(N)
    _lib.lib().mult_combine(_p(ty), _p(tX), _p(n), C.byref(cN), C.byref(_ci(P)), C.byref(_ci(U + 1)))
    _lib.check()
    M = cN.value
    return {"y": ty.reshape(N, U)[:M].copy(), "X": tX.reshape(N, P)[:M].copy(), "n": n[:M].copy()}


def mlogit(y, X, n=None, m0=None, P0=None, samp=1000, burn=500):
    X = np.atleast_2d(_f(X))
    y = _f(y)
    y = y.reshape(-1, 1) if y.ndim == 1 else y
    new = mlogit_combine(y, X, n)
    if not isinstance(new, dict):
        return NA
    y, X, n = new["y"], new["X"], new["n"]
    N, P = X.shape
    U = y.shape[1]
    m0 = np.zeros((P, U)) if m0 is None else _f(m0)
    P0 = np.zeros((P, P, U)) if P0 is None else _f(P0)
    if not mult_check_parameters(y, X, n, m0, P0, samp, burn):
        return NA
    w = np.zeros((samp, U, N))       # C view of column-major N x U x samp
    beta = np.zeros((samp, U, P))
    ty = np.ascontiguousarray(y)
    tX = np.ascontiguousarray(X)
    m0c = np.asfortranarray(m0)
    P0c = np.asfortranarray(P0)
    cN = _ci(N)
    _lib.lib().mult_gibbs(_p(w), _p(beta), _p(ty), _p(tX), _p(n), m0c.ctypes.data, P0c.ctypes.data,
                          C.byref(cN), C.byref(_ci(P)), C.byref(_ci(U + 1)), C.byref(_ci(samp)),
                          C.byref(_ci(burn)))
    _lib.check()
    M = cN.value
    # R returns w as samp x N x (J-1) and beta as samp x P x (J-1)
    return {"w": np.transpose(w[:, :, :M], (0, 2, 1)).copy(), "beta": np.transpose(beta, (0, 2, 1)).copy(),
            "y": y, "X": X, "n": n}


# ---------------------------------------------------------------------------------
# engine extensions: explicit seeds / flags (column-major inputs as numpy Fortran or
# row-major-transposed arrays are handled here so tests read naturally)
# ---------------------------------------------------------------------------------

def logit_gibbs(y, X, n, m0, P0, samp, burn, seed, flags=0, keep_w=True, w_every=1):
    """Chain with an explicit seed.  Returns (w [ceil(samp / w_every) x N] or None, beta [samp x P]); w_every > 1
    thins the omega chain (row k = sampling iteration k * w_every + 1)."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    N, P = X.shape
    y, n, m0 = _f(y).ravel(), _f(n).ravel(), _f(m0).ravel()
    P0c = np.asfortranarray(_f(P0))
    beta = np.zeros((samp, P))
    w = np.zeros(((samp + w_every - 1) // w_every, N)) if keep_w else None
    st = _lib.lib().bl_logit_gibbs_thin(_p(w) if keep_w else None, _p(beta), _p(y), _p(X), _p(n), _p(m0),
                                        P0c.ctypes.data, N, P, samp, burn, int(seed),
                                        int(flags) | (0 if keep_w else NO_W), int(w_every))
    _lib.check(st)
    return w, beta


def logit_chains(y, X, n, m0, P0, samp, burn, seed, flags=0):
    """A batch of independent chains sharing the prior: y, n [chains x N], X [chains x N x P].
    Chain c is the chain logit_gibbs(y[c], X[c], n[c], ..., seed=seed + c) runs; all chains advance
    together, one launch per kernel per iteration for the whole batch.  Returns beta [chains x samp x P]."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    chains, N, P = X.shape
    y = np.ascontiguousarray(y, dtype=np.float64).reshape(chains, N)
    n = np.ascontiguousarray(n, dtype=np.float64).reshape(chains, N)
    m0 = _f(m0).ravel()
    P0c = np.asfortranarray(_f(P0))
    beta = np.zeros((chains, samp, P))
    st = _lib.lib().bl_logit_chains(_p(beta), _p(y), _p(X), _p(n), _p(m0), P0c.ctypes.data, chains, N, P,
                                    samp, burn, int(seed), int(flags))
    _lib.check(st)
    return beta


def logit_multichain(y, X, n, m0, P0, samp, burn, seed, chains, flags=0):
    """`chains` independent chains on one data set: y, n [N], X [N x P], shared by all chains.  Chain c is the
    chain logit_chains runs on `chains` copies of the data with the same seed (so it uses the streams of
    seed + c), bit for bit, with X held and read once.  Returns beta [chains x samp x P]."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    N, P = X.shape
    y, n, m0 = _f(y).ravel(), _f(n).ravel(), _f(m0).ravel()
    P0c = np.asfortranarray(_f(P0))
    beta = np.zeros((max(int(chains), 0), samp, P))
    st = _lib.lib().bl_logit_multichain(_p(beta), _p(y), _p(X), _p(n), _p(m0), P0c.ctypes.data, int(chains), N, P,
                                        samp, burn, int(seed), int(flags))
    _lib.check(st)
    return beta


def mlogit_gibbs(y, X, n, m0, P0, samp, burn, seed, flags=0, keep_w=True):
    """y: N x (J-1) proportions.  Returns (w [samp x (J-1) x N] or None, beta [samp x (J-1) x P])."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    N, P = X.shape
    U = y.shape[1]
    n = _f(n).ravel()
    m0c, P0c = np.asfortranarray(_f(m0)), np.asfortranarray(_f(P0))
    beta = np.zeros((samp, U, P))
    w = np.zeros((samp, U, N)) if keep_w else None
    st = _lib.lib().bl_mlogit_gibbs(_p(w) if keep_w else None, _p(beta), _p(y), _p(X), _p(n),
                                    m0c.ctypes.data, P0c.ctypes.data, N, P, U + 1, samp, burn, int(seed),
                                    int(flags) | (0 if keep_w else NO_W))
    _lib.check(st)
    return w, beta


def mlogit_multichain(y, X, n, m0, P0, samp, burn, seed, chains, flags=0):
    """`chains` independent multinomial logit chains on one data set: y [N x (J-1)], X [N x P], n [N], m0, P0 as
    mlogit_gibbs takes them, shared by all chains.  Chain c is, bit for bit, mlogit_gibbs(..., seed=seed + c,
    keep_w=False)[1], with X held once and read once per category update for up to 8 chains.  flags: 0 or UNFUSED.
    Returns beta [chains x samp x (J-1) x P]."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    N, P = X.shape
    U = y.shape[1]
    n = _f(n).ravel()
    m0c, P0c = np.asfortranarray(_f(m0)), np.asfortranarray(_f(P0))
    beta = np.zeros((max(int(chains), 0), samp, U, P))
    st = _lib.lib().bl_mlogit_multichain(_p(beta), _p(y), _p(X), _p(n), m0c.ctypes.data, P0c.ctypes.data, int(chains),
                                         N, P, U + 1, samp, burn, int(seed), int(flags))
    _lib.check(st)
    return beta


def nb_gibbs(y, X, d, m0, P0, samp, seed):
    """NB regression with fixed dispersion d.  Returns (w_last [N], beta [samp x P])."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    N, P = X.shape
    y, m0 = _f(y).ravel(), _f(m0).ravel()
    P0c = np.asfortranarray(_f(P0))
    beta = np.zeros((samp, P))
    w = np.zeros(N)
    st = _lib.lib().bl_nb_gibbs(_p(w), _p(beta), _p(y), _p(X), float(d), _p(m0), P0c.ctypes.data,
                                N, P, samp, int(seed))
    _lib.check(st)
    return w, beta


def nb_gibbs_df(y, X, m0, P0, samp, burn, seed, d0=1.0, real_d=False):
    """NB regression with the dispersion sampled (NB.PG.gibbs, NBPG-logmean.R:36-113): draw.df on the integers, or
    (real_d) draw.df.real.mean on the reals (NB-Shape.R:86-96).  Returns (w_last [N], beta [samp x P], d [samp])."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    N, P = X.shape
    y, m0 = _f(y).ravel(), _f(m0).ravel()
    P0c = np.asfortranarray(_f(P0))
    beta = np.zeros((samp, P))
    d = np.zeros(samp)
    w = np.zeros(N)
    fn = _lib.lib().bl_nb_gibbs_dfreal if real_d else _lib.lib().bl_nb_gibbs_df
    st = fn(_p(w), _p(beta), _p(d), _p(y), _p(X), float(d0), _p(m0), P0c.ctypes.data, N, P, samp, burn, int(seed))
    _lib.check(st)
    return w, beta, d


NB_DMODES = {"fixed": 0, "int": 1, "real": 2}     # BL_NB_D_FIXED, BL_NB_D_INT, BL_NB_D_REAL


def nb_multichain(y, X, m0, P0, samp, burn, seed, chains, d0=1.0, dmode="int"):
    """`chains` independent NB chains on one data set: y [N], X [N x P], m0, P0 shared by all chains.  dmode "int":
    chain c is, bit for bit, nb_gibbs_df(..., seed=seed + c)'s beta and d; "real": the same with real_d=True; "fixed":
    d = d0 throughout, beta is rows burn .. burn + samp - 1 of nb_gibbs(..., samp + burn, seed=seed + c) (d is d0).
    X is held once and read once per iteration for up to 8 chains.  Returns (beta [chains x samp x P],
    d [chains x samp])."""
    if dmode not in NB_DMODES:
        raise ValueError("dmode must be one of %s" % ", ".join(map(repr, NB_DMODES)))
    X = np.ascontiguousarray(X, dtype=np.float64)
    N, P = X.shape
    y, m0 = _f(y).ravel(), _f(m0).ravel()
    P0c = np.asfortranarray(_f(P0))
    K = max(int(chains), 0)
    beta = np.zeros((K, samp, P))
    d = np.zeros((K, samp))
    st = _lib.lib().bl_nb_multichain(_p(beta), _p(d), _p(y), _p(X), float(d0), _p(m0), P0c.ctypes.data, int(chains),
                                     N, P, samp, burn, int(seed), NB_DMODES[dmode])
    _lib.check(st)
    return beta, d


def logit_ri(y, X, n, group, G, m0, P0, a0, b0, tau2_0, samp, burn, seed, flags=0, keep_u=True):
    """Binomial logit with group random intercepts: logit P(success_i) = x_i' beta + u_{group_i}, u_g ~ N(0, tau2),
    beta ~ N(m0, P0^-1) (P0 a precision), tau2 ~ IG(a0, b0); y proportions, n trials, group ids in [0, G).  One chain
    from beta = 0, u = 0, tau2 = tau2_0; burn iterations are discarded.  flags: 0 or UNFUSED (same chain, bit for bit).
    Returns (beta [samp x P], u [samp x G] or None when keep_u is False, tau2 [samp])."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    N, P = X.shape
    y, n, m0 = _f(y).ravel(), _f(n).ravel(), _f(m0).ravel()
    group = np.ascontiguousarray(group, dtype=np.int32).ravel()
    if len(y) != N or len(n) != N or len(group) != N:
        raise ValueError("y, n and group need one entry per row of X")
    P0c = np.asfortranarray(_f(P0))
    beta = np.zeros((max(int(samp), 0), P))
    tau2 = np.zeros(max(int(samp), 0))
    u = np.zeros((max(int(samp), 0), max(int(G), 0))) if keep_u else None
    st = _lib.lib().bl_logit_ri_gibbs(_p(beta), _p(u) if keep_u else None, _p(tau2), _p(y), _p(X), _p(n), _p(group),
                                      int(G), _p(m0), P0c.ctypes.data, float(a0), float(b0), float(tau2_0), N, P,
                                      int(samp), int(burn), int(seed), int(flags))
    _lib.check(st)
    return beta, u, tau2
