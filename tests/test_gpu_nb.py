"""The single negative-binomial chain against the CPU oracle (oracle/gibbs_oracle.c) at every kernel choice, for all
three treatments of the dispersion d: fixed (bl_nb_gibbs), the random walk on the integers (bl_nb_gibbs_df) and the
walk on the reals (bl_nb_gibbs_dfreal).  The multichain and sharded NB tests compare outputs of the same kernels with
each other, so a wrong kernel path would leave them green; here every path meets the oracle.

  * shapes that each reach a different X'v, Gram, beta-draw or omega-sampler choice, with a non-zero prior mean and a
    dense prior precision (so b0 = P0 m0 matters), and edges of the dispersion step (d < 1, all-zero counts, one huge
    count, d0 = 1, burn = 0);
  * X at a pointer 8 bytes into its buffer (the scalar X beta / X'v kernels and the Gram's 8-byte loads);
  * bl_probe_nb_dispersion: the two log-likelihoods of one Metropolis step against a long-double reference with an
    exact sum, and the accept decision against the rule applied to the reference;
  * counts the histogram of G[j] = #{y_i > j} cannot index are refused at every entry that builds it;
  * sharded rows on virtual ranks, all three modes.
"""
import math
import threading

import numpy as np
import pytest
from scipy.special import gammaln

from oracle import loader

pytestmark = pytest.mark.gpu

MODES = ["fixed", "int", "real"]
D0 = {"fixed": 1.0, "int": 2.0, "real": 2.5}
SAMP, BURN = 4, 2
SEED = 7207

# (N, P), each reaching a different choice of kernels; N >= ~20 P keeps the posterior precision well conditioned, so
# the oracle's and the engine's summation orders give betas within the chain tolerance
SHAPES = [
    (2000, 5),       # odd P: k_xbeta, k_xtv_partial; per-lane rpg_hybrid
    (4001, 8),       # k_xtv_stream at the smallest power-of-two P
    (40_000, 16),    # regime-binned draw
    (30_011, 32),    # packed Gram
    (20_000, 64),    # one Gram tile, lean beta draw
    (10_007, 70),    # several Gram tiles, shared-memory beta draw at P > 64
    (6000, 128),     # beta drawn out of global scratch
    (30_000, 256),   # the same at the largest P
    (2000, 1),       # P = 1
    (2000, 2),       # P = 2
    (6000, 34),      # k_xtv_mma at an even P that is not a power of two
    (8000, 96),      # ragged second Gram tile, global-scratch beta draw
    (32_767, 16),    # the last N of the per-lane draw
    (32_768, 16),    # the first N of the regime-binned draw
    (700_003, 16),   # nblk = 592 binds: slabs of 1183 rows, the last one 850
]
REL_BETA = 1e-7
REL_DREAL = 1e-12


@pytest.fixture(scope="module")
def gapi(engine):
    from bayeslogit_b200 import gibbs_api
    return gibbs_api


def prior(P):
    """Non-zero prior mean and a dense SPD prior precision."""
    return np.linspace(-0.4, 0.4, P), 0.02 * np.eye(P) + 0.005 * np.ones((P, P))


def synth(N, P, seed, d=3.0):
    """Counts 0 .. ~1000: log-mean 2.6 + N(0, 1.2^2) (at P = 1 the spread is not explained by X)."""
    rng = np.random.default_rng(seed)
    X = np.c_[rng.standard_normal((N, P - 1)) / np.sqrt(max(P - 1, 1)), np.ones(N)]
    eta = X[:, :-1] @ (1.2 * rng.choice([-1.0, 1.0], P - 1)) + 2.6
    if P == 1:
        eta = eta + 1.2 * rng.standard_normal(N)
    mu = np.exp(eta)
    y = rng.negative_binomial(d, d / (mu + d)).astype(float)
    return X, y


REGIMES = {
    "gamma": lambda b: b < 1,                                  # sum of gammas
    "devroye": lambda b: (b == 1) | (b == 2),
    "alt": lambda b: (b > 1) & (b <= 13) & (b != 2),
    "sp": lambda b: (b > 13) & (b <= 170),                     # saddle point
    "normal": lambda b: b > 170,
}


def assert_regimes(y, d, *names):
    b = y + d
    for name in names:
        assert REGIMES[name](b).any(), (name, d)


def close(a, b, rel):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape
    err = np.abs(a - b) / np.maximum(np.abs(b), 1e-300)
    assert np.all(np.isfinite(a)) and err.max() <= rel, float(err.max())


def run_and_compare(gapi, mode, X, y, m0, P0, d0, samp, burn, seed):
    """The engine's chain and the oracle's: beta and the last omega within 1e-7, d equal step for step (integer
    walk) or within 1e-12 (real walk).  Returns the engine's d chain."""
    if mode == "fixed":
        w, b = gapi.nb_gibbs(y, X, d0, m0, P0, samp + burn, seed)
        wo, bo = loader.nb_gibbs(y, X, d0, m0, P0, samp + burn, seed=seed)
        d = np.full(samp, d0)
    else:
        real = mode == "real"
        w, b, d = gapi.nb_gibbs_df(y, X, m0, P0, samp, burn, seed, d0=d0, real_d=real)
        wo, bo, do = loader.nb_gibbs_df(y, X, m0, P0, samp, burn, seed=seed, d0=d0, real_d=real)
        if real:
            close(d, do, REL_DREAL)
        else:
            assert np.array_equal(d, do), (d, do)
    close(b, bo, REL_BETA)
    close(w, wo, REL_BETA)
    return d


_data = {}


def data(shape):
    if shape not in _data:
        _data[shape] = synth(*shape, 300 + shape[0] % 1000 + shape[1])
    return _data[shape]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "N%d-P%d" % s)
def test_nb_chain_matches_oracle(gapi, shape, mode):
    X, y = data(shape)
    m0, P0 = prior(shape[1])
    assert_regimes(y, D0[mode], "alt", "sp", "normal", *(["devroye"] if mode != "real" else []))
    run_and_compare(gapi, mode, X, y, m0, P0, D0[mode], SAMP, BURN, SEED + shape[1])


def test_nb_chain_matches_oracle_at_size(gapi):
    """N = 1 000 000, P = 64, integer walk: the binned draw at size, nblk capped, 1690-row slabs."""
    X, y = synth(1_000_000, 64, 41)
    m0, P0 = prior(64)
    run_and_compare(gapi, "int", X, y, m0, P0, 2.0, 2, 1, 43)


@pytest.mark.parametrize("shape", [(6000, 8), (40_000, 16)], ids=lambda s: "N%d-P%d" % s)
def test_nb_fixed_small_d_draws_sums_of_gammas(gapi, shape):
    """d = 0.4: rows with y = 0 have b = 0.4 < 1, the sum-of-gammas regime, inside the sweep."""
    X, y = data(shape)
    m0, P0 = prior(shape[1])
    assert_regimes(y, 0.4, "gamma", "alt", "sp", "normal")
    run_and_compare(gapi, "fixed", X, y, m0, P0, 0.4, 3, 0, 11)


@pytest.mark.parametrize("shape", [(6000, 8), (40_000, 16)], ids=lambda s: "N%d-P%d" % s)
def test_nb_real_walk_from_below_one(gapi, shape):
    """d0 = 0.5: the proposal is U(0, 2) (the r <= 1 branch), and b = y + d < 1 where y = 0."""
    X, y = data(shape)
    m0, P0 = prior(shape[1])
    assert_regimes(y, 0.5, "gamma", "alt", "sp", "normal")
    run_and_compare(gapi, "real", X, y, m0, P0, 0.5, 4, 2, 12)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("N", [5000, 40_000])
def test_nb_all_zero_counts(gapi, N, mode):
    """ymax = 0: no G series, b = d on every row."""
    X, _ = synth(N, 8, 13)
    m0, P0 = prior(8)
    run_and_compare(gapi, mode, X, np.zeros(N), m0, P0, D0[mode], SAMP, BURN, 14)


@pytest.mark.parametrize("mode", MODES)
def test_nb_one_huge_count(gapi, mode):
    """One count of 10^5: a G series of 10^5 terms, b ~ 10^5 in the normal regime."""
    X, y = synth(20_000, 16, 15)
    y[4321] = 1e5
    m0, P0 = prior(16)
    run_and_compare(gapi, mode, X, y, m0, P0, D0[mode], SAMP, BURN, 16)


def test_nb_integer_walk_from_one(gapi):
    """d0 = 1: proposals {1, 2}, and the proposal ratio lppsl is asymmetric (1/2 against 1/3)."""
    X, y = synth(20_000, 16, 17)
    m0, P0 = prior(16)
    assert_regimes(y, 1.0, "devroye", "alt", "sp", "normal")
    run_and_compare(gapi, "int", X, y, m0, P0, 1.0, 6, 2, 18)


@pytest.mark.parametrize("mode", MODES)
def test_nb_no_burn_one_sample(gapi, mode):
    X, y = data((4001, 8))
    m0, P0 = prior(8)
    run_and_compare(gapi, mode, X, y, m0, P0, D0[mode], 1, 0, 19)


# ---------------------------------------------------------------------------------------------------------------
# Device entries with X 8 bytes into its buffer
# ---------------------------------------------------------------------------------------------------------------
class Dev:
    """Device-resident inputs; X may start 8 bytes into its buffer."""

    def __init__(self):
        import torch
        from bayeslogit_b200 import _lib
        self.t, self.L, self.check = torch, _lib.lib(), _lib.check
        self.dev = torch.device("cuda")
        self.st = torch.cuda.current_stream().cuda_stream

    def put(self, a, offset=0):
        t = self.t
        a = np.ascontiguousarray(a, dtype=np.float64)
        buf = t.zeros(a.size + offset, dtype=t.float64, device=self.dev)
        buf[offset:] = t.from_numpy(a.ravel()).to(self.dev)
        ptr = buf.data_ptr() + 8 * offset
        assert ptr % 16 == (8 if offset % 2 else 0)
        return buf, ptr

    def chain(self, mode, X, y, m0, P0, d0, samp, burn, seed, x_offset):
        """bl_nb_gibbs_dev (fixed; every iteration recorded), bl_nb_gibbs_df_dev or bl_nb_gibbs_dfreal_dev.
        Returns (beta, d, last omega)."""
        t = self.t
        N, P = X.shape
        keep = [self.put(X, x_offset), self.put(y), self.put(m0), self.put(np.asfortranarray(P0).ravel(order="F"))]
        tX, ty, tm, tp = (k[1] for k in keep)
        w = t.zeros(N, dtype=t.float64, device=self.dev)
        if mode == "fixed":
            beta = t.zeros(samp + burn, P, dtype=t.float64, device=self.dev)
            self.check(self.L.bl_nb_gibbs_dev(w.data_ptr(), beta.data_ptr(), ty, tX, d0, tm, tp, N, P, samp + burn,
                                              seed, 0, self.st))
            t.cuda.synchronize()
            return beta.cpu().numpy(), np.full(samp, d0), w.cpu().numpy()
        beta = t.zeros(samp, P, dtype=t.float64, device=self.dev)
        d = t.zeros(samp, dtype=t.float64, device=self.dev)
        fn = self.L.bl_nb_gibbs_dfreal_dev if mode == "real" else self.L.bl_nb_gibbs_df_dev
        self.check(fn(w.data_ptr(), beta.data_ptr(), d.data_ptr(), ty, tX, d0, tm, tp, N, P, samp, burn, seed, 0,
                      self.st))
        t.cuda.synchronize()
        return beta.cpu().numpy(), d.cpu().numpy(), w.cpu().numpy()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("N,P", [(4001, 16), (6007, 32), (40_000, 64)])
def test_nb_unaligned_x_matches_oracle(engine, N, P, mode):
    """X 8 bytes into its buffer: k_xbeta, k_xtv_partial (with log d read from device memory when d is sampled) and
    the Gram's 8-byte loads.  Each chain matches the oracle, and the aligned call within 1e-9."""
    dev = Dev()
    X, y = synth(N, P, 90 + P)
    m0, P0 = prior(P)
    d0, samp, burn, seed = D0[mode], 4, 2, 91
    bu, du, wu = dev.chain(mode, X, y, m0, P0, d0, samp, burn, seed, x_offset=1)
    ba, da, _ = dev.chain(mode, X, y, m0, P0, d0, samp, burn, seed, x_offset=0)
    if mode == "fixed":
        wo, bo = loader.nb_gibbs(y, X, d0, m0, P0, samp + burn, seed=seed)
    else:
        wo, bo, do = loader.nb_gibbs_df(y, X, m0, P0, samp, burn, seed=seed, d0=d0, real_d=mode == "real")
        if mode == "int":
            assert np.array_equal(du, do)
        else:
            close(du, do, REL_DREAL)
    close(bu, bo, REL_BETA)
    close(wu, wo, REL_BETA)
    close(bu, ba, 1e-9)
    if mode == "int":
        assert np.array_equal(du, da)


# ---------------------------------------------------------------------------------------------------------------
# The dispersion step against a high-precision reference
# ---------------------------------------------------------------------------------------------------------------
# The engine's llh is within C_ULP * 2^-53 of the exact value times the sum of the operand magnitudes: per row
# |log d|, |log(mu + d)|, |y|, |phi|, each lgamma of the real walk, plus 1 for the relative error of mu = exp(phi)
# carried into log(mu + d) with weight mu / (mu + d) <= 1, and |log(d + j)| G[j] for the G series.  Operand
# magnitudes rather than term magnitudes, because log d - log(mu + d) cancels when phi << 0 and its rounding error is
# that of its operands.  The sums run over up to ~45 levels (a thread's rows, the warp and CTA reductions, the fold
# of the CTA partials); rounding errors of that depth are a few units of 2^-53 of the magnitude sum in practice.
C_ULP = 32
EPS = 2.0 ** -53


def exact_sum(t):
    """Sum of long-double terms, rounded once: each term split into two doubles, then math.fsum."""
    hi = t.astype(np.float64)
    lo = (t - hi.astype(np.longdouble)).astype(np.float64)
    return math.fsum(np.concatenate([hi, lo]))


def ref_llh(phi, y, d, real):
    """(llh, operand magnitude sum) of draw.df's df.llh (integer walk) or draw.df.real.mean's target (real walk)."""
    ph = phi.astype(np.longdouble)
    yl = y.astype(np.longdouble)
    dl = np.longdouble(d)
    lmd = np.log(np.exp(ph) + dl)
    ld = np.log(dl)
    if real:
        lg_yr, lg_r, lg_y1 = gammaln(y + d), gammaln(d), gammaln(y + 1.0)
        terms = (lg_yr.astype(np.longdouble) - np.longdouble(lg_r) - lg_y1.astype(np.longdouble)
                 + dl * (ph - lmd) + yl * (ld - lmd))
        mag = (np.abs(lg_yr) + abs(lg_r) + np.abs(lg_y1) + d * (np.abs(phi) + np.abs(lmd) + 1)
               + y * (abs(float(ld)) + np.abs(lmd) + 1))
        return exact_sum(terms), float(np.sum(mag.astype(np.float64)))
    terms = dl * (ld - lmd) + yl * (ph - lmd)
    mag = d * (abs(float(ld)) + np.abs(lmd) + 1) + y * (np.abs(phi) + np.abs(lmd) + 1)
    ymax = int(y.max())
    value, gmag = exact_sum(terms), 0.0
    if ymax > 0:
        hist = np.bincount(y.astype(np.int64), minlength=ymax + 1)
        G = np.cumsum(hist[::-1])[::-1][1:].astype(np.longdouble)       # G[j] = #{y_i > j}, j < ymax
        gterms = np.log(dl + np.arange(ymax, dtype=np.longdouble)) * G
        value = math.fsum([value, exact_sum(gterms)])
        gmag = float(np.sum(np.abs(gterms)))
    return value, float(np.sum(mag.astype(np.float64))) + gmag


def probe(phi, y, d, seed, call, real):
    from bayeslogit_b200 import _lib
    phi = np.ascontiguousarray(np.atleast_2d(phi), dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    d = np.ascontiguousarray(d, dtype=np.float64)
    K, N = phi.shape
    out = np.zeros((K, 5))
    _lib.check(_lib.lib().bl_probe_nb_dispersion(out.ctypes.data, phi.ctypes.data, y.ctypes.data, d.ctypes.data, K,
                                                 N, seed, call, int(real)))
    return out


def probe_data(N, counts, seed):
    """phi of 3 chains ~ N(1.5, 1.5^2) with rows at -30, 0 and +30 mixed in; counts from phi of chain 0."""
    rng = np.random.default_rng(seed)
    phi = rng.normal(1.5, 1.5, (3, N))
    for k, v in enumerate((-30.0, 0.0, 30.0)):
        phi[:, k::97] = v
    if counts == "zeros":
        return phi, np.zeros(N)
    mu = np.exp(np.clip(phi[0], -5, 5))
    y = rng.negative_binomial(3.0, 3.0 / (mu + 3.0)).astype(float)
    if counts == "big":
        y[N // 2] = 1e5
    return phi, y


PROBE_CASES = [(N, c) for N in (700, 1025, 5000) for c in ("nb", "zeros", "big")] + \
              [(606_209, "nb"), (1_000_000, "big")]
PROBE_D = {False: [1.0, 7.0, 1000.0], True: [0.3, 2.5, 1000.25]}


@pytest.mark.parametrize("real", [False, True], ids=["int", "real"])
@pytest.mark.parametrize("N,counts", PROBE_CASES, ids=lambda v: str(v))
def test_nb_dispersion_step_against_reference(engine, N, counts, real):
    """N < 1024 (one slab), 1025, not a multiple of 256, 606 209 (the nblk cap plus one), 10^6; ymax = 0 and one
    count of 10^5; d = 1, 7, 1000 (integer walk) and r = 0.3 (the U(0, 2) proposal), 2.5, 1000.25 (real walk)."""
    phi, y = probe_data(N, counts, N + len(counts))
    d = np.array(PROBE_D[real])
    seed = 808
    decided = 0
    for call in range(3):
        out = probe(phi, y, d, seed, call, real)
        for c in range(3):
            dp, u, llh, llhp, dn = out[c]
            if real:
                assert (0 < dp < 2) if d[c] <= 1 else (abs(dp - d[c]) <= 1), (c, dp)
                assert u < 0
            else:
                assert dp in {max(d[c] - 1, 1.0), d[c], d[c] + 1}, (c, dp)
                assert 0 < u < 1
            r0, mag0 = ref_llh(phi[c], y, d[c], real)
            r1, mag1 = ref_llh(phi[c], y, dp, real)
            tol0, tol1 = C_ULP * EPS * mag0, C_ULP * EPS * mag1
            assert abs(llh - r0) <= tol0, (c, call, llh, r0, tol0)
            assert abs(llhp - r1) <= tol1, (c, call, llhp, r1, tol1)
            # the Metropolis rule applied to the reference difference
            if real:
                x, lu = r1 - r0, u
            else:
                x = r1 - r0 + math.log(0.5 if dp == 1 else 1 / 3) - math.log(0.5 if d[c] == 1 else 1 / 3)
                lu = math.log(u)
            assert dn in (dp, d[c])
            if abs(x - lu) > tol0 + tol1 + 1e-12 * max(1.0, abs(lu)):
                assert dn == (dp if lu < x else d[c]), (c, call, x, lu, dn)
                decided += 1
        if call == 0:
            # three chains in one launch equal three one-chain probes bit for bit
            for c in range(3):
                one = probe(phi[c], y, d[c:c + 1], seed + c, call, real)
                assert np.array_equal(one[0], out[c]), (c, one[0], out[c])
    assert decided >= 6


# ---------------------------------------------------------------------------------------------------------------
# Counts the histogram cannot index
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bad", [-1.0, np.nan, 3e9, np.inf, 2147483647.0], ids=str)
def test_nb_refuses_counts_the_histogram_cannot_index(gapi, bad):
    """A count that is negative, not finite or >= 2^31 - 1 would index the count histogram out of bounds: every entry
    that builds it refuses the data, launching no sweep; a valid call afterwards still matches the oracle."""
    from bayeslogit_b200 import _lib
    N, P = 3001, 4
    X, y = synth(N, P, 21)
    m0, P0 = prior(P)
    yb = y.copy()
    yb[1234] = bad
    msg = "counts y must be finite, non-negative and below 2\\^31 - 1"
    with pytest.raises(_lib.EngineError, match="nb_gibbs_df: " + msg):
        gapi.nb_gibbs_df(yb, X, m0, P0, 2, 1, 5, d0=2.0)
    with pytest.raises(_lib.EngineError, match="nb_gibbs_dfreal: " + msg):
        gapi.nb_gibbs_df(yb, X, m0, P0, 2, 1, 5, d0=2.5, real_d=True)
    for chains in (1, 3):
        for dmode in ("int", "real"):
            with pytest.raises(_lib.EngineError, match="nb_multichain: " + msg):
                gapi.nb_multichain(yb, X, m0, P0, 2, 1, 5, chains, d0=D0[dmode], dmode=dmode)
    dev = Dev()
    for mode in ("int", "real"):
        with pytest.raises(_lib.EngineError, match=msg):
            dev.chain(mode, X, yb, m0, P0, D0[mode], 2, 1, 5, x_offset=0)
    with pytest.raises(_lib.EngineError, match="probe_nb_dispersion: " + msg):
        probe(np.zeros(N), yb, np.array([2.0]), 5, 0, False)
    for mode in ("int", "real"):
        run_and_compare(gapi, mode, X, y, m0, P0, D0[mode], 3, 1, 22)


# ---------------------------------------------------------------------------------------------------------------
# Sharded rows on virtual ranks
# ---------------------------------------------------------------------------------------------------------------
class _Runner:
    """The sharded NB sweeps on rows [lo, hi) of a data set, device pointers, one given stream."""

    def __init__(self, L, check, torch, dev, stream):
        self.L, self.check, self.torch, self.dev, self.st = L, check, torch, dev, stream

    def _up(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(self.dev)

    def run(self, mode, X, y, lo, hi, samp=4, burn=2, seed=4717):
        t, P = self.torch, X.shape[1]
        m0, P0 = prior(P)
        with t.cuda.stream(self.st):
            Xd, yd = self._up(X[lo:hi]), self._up(y[lo:hi])
            m0d, P0d = self._up(m0), self._up(np.asfortranarray(P0).ravel(order="F"))
            beta = t.zeros(samp + (burn if mode == "fixed" else 0), P, device=self.dev, dtype=t.float64)
            dd = t.zeros(samp, device=self.dev, dtype=t.float64)
        self.st.synchronize()
        if mode == "fixed":
            rc = self.L.bl_nb_gibbs_dev(None, beta.data_ptr(), yd.data_ptr(), Xd.data_ptr(), D0[mode],
                                        m0d.data_ptr(), P0d.data_ptr(), hi - lo, P, samp + burn, seed, lo,
                                        self.st.cuda_stream)
        else:
            fn = self.L.bl_nb_gibbs_dfreal_dev if mode == "real" else self.L.bl_nb_gibbs_df_dev
            rc = fn(None, beta.data_ptr(), dd.data_ptr(), yd.data_ptr(), Xd.data_ptr(), D0[mode], m0d.data_ptr(),
                    P0d.data_ptr(), hi - lo, P, samp, burn, seed, lo, self.st.cuda_stream)
        if rc:
            self.check(rc)
        self.st.synchronize()
        d = dd.cpu().numpy() if mode != "fixed" else np.full(samp, D0[mode])
        return beta.cpu().numpy(), d


def _shard_data():
    cases = {s: synth(*s, 500 + s[1]) for s in [(9001, 7), (12_001, 70), (40_003, 16)]}
    X, y = synth(12_001, 16, 533)
    y[: 12_001 * 3 // 5] = 0.0         # rank 0's counts are all zero at every world size tested
    cases["zero-shard"] = (X, y)
    return cases


@pytest.mark.parametrize("world", [2, 3, 8])
def test_nb_sharded_on_virtual_ranks(engine, world):
    """All three modes at W virtual ranks: beta bit-identical across ranks and within 1e-8 of the single-GPU chain,
    d equal step for step (within 1e-12 on the real walk); one shard with all counts zero (local ymax = 0, global
    ymax large); the (12 001, 70) integer-walk chain also against the oracle."""
    import torch
    from bayeslogit_b200 import _lib, dist as bdist
    L = _lib.lib()
    dev = torch.device("cuda", 0)
    st = torch.cuda.Stream(device=dev)
    run = _Runner(L, _lib.check, torch, dev, st)
    cases = _shard_data()
    full = {(k, m): run.run(m, X, y, 0, X.shape[0]) for k, (X, y) in cases.items() for m in MODES}
    lo0, hi0 = bdist.shard_range(0, world, 12_001)
    assert not cases["zero-shard"][1][lo0:hi0].any() and cases["zero-shard"][1].max() > 100

    _lib.check(L.bl_vcomm_create(world))
    results, errors = [None] * world, []

    def rank_main(r):
        try:
            _lib.check(L.bl_vcomm_bind(r))
            out = {}
            for k, (X, y) in cases.items():
                lo, hi = bdist.shard_range(r, world, X.shape[0])
                for m in MODES:
                    out[(k, m)] = run.run(m, X, y, lo, hi)
            results[r] = out
        except Exception as e:                       # noqa: BLE001 -- reported by the main thread
            errors.append((r, repr(e)))
        finally:
            L.bl_vcomm_bind(-1)

    threads = [threading.Thread(target=rank_main, args=(r,)) for r in range(world)]
    try:
        for t in threads:
            t.start()
        for t in threads:
            t.join(timeout=600)
        assert not errors, errors
        assert all(r is not None for r in results)
    finally:
        L.bl_vcomm_destroy()

    for key, (fb, fd) in full.items():
        for r in range(world):
            b, d = results[r][key]
            assert np.array_equal(b, results[0][key][0]), ("beta differs between ranks", key, r)
            close(b, fb, 1e-8)
            if key[1] == "real":
                close(d, fd, REL_DREAL)
            else:
                assert np.array_equal(d, fd), (key, r, d, fd)
        if key[1] != "fixed":
            assert np.any(fd != D0[key[1]]), key
    X, y = cases[(12_001, 70)]
    m0, P0 = prior(70)
    _, bo, do = loader.nb_gibbs_df(y, X, m0, P0, 4, 2, seed=4717, d0=D0["int"])
    b, d = results[world - 1][((12_001, 70), "int")]
    close(b, bo, REL_BETA)
    assert np.array_equal(d, do)
