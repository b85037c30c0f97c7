"""Negative binomial with group random intercepts on the GPU (bl_nb_ri_gibbs / bl_nb_ri_gibbs_dev) against the CPU
restatement of the same six steps (tests/ri_oracle/nb_ri_oracle.c), for all three treatments of the dispersion d:
fixed, the random walk on the integers and the walk on the reals.

  * every mode at P in {1, 2, 5, 8, 16, 32, 34, 64, 70, 128, 256}, which together reach each X'v, Gram and beta-draw
    choice; N = 32 767 and 32 768 (the last per-lane and the first regime-binned omega draw); the group layouts (one
    group, a group per row, empty groups, half the rows in one group, sorted ids); a group whose counts are all zero;
    counts that reach every rpg_hybrid regime; a non-zero m0 and a dense P0 throughout; N = 10^6, P = 64, G = 10^4.
    beta, u and tau2 agree within 1e-7 (|a - b| / max(1, |b|)); d is equal step for step on the integer walk and
    within 1e-12 on the real walk.  The engine sums in other orders than the restatement (MMA X beta, tiled Gram,
    chunked group sums), so the chains agree to rounding, not bit for bit;
  * the host and device entries, two runs of one seed, and runs without u or d stored agree bit for bit;
  * every refusal raises its own message and leaves the outputs untouched;
  * tau, d and the group effects are recovered at N = 2 * 10^5.
"""
import numpy as np
import pytest

import _nb_ri_oracle as ro

pytestmark = pytest.mark.gpu

MODES = ["fixed", "int", "real"]
D0 = {"fixed": 2.0, "int": 2.0, "real": 2.5}
A0, B0, TAU2_0 = 2.0, 0.5, 1.0
SAMP, BURN = 4, 2
REL = 1e-7
REL_DREAL = 1e-12

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


@pytest.fixture(scope="module")
def gapi(engine):
    from bayeslogit_b200 import gibbs_api
    return gibbs_api


def prior(P):
    """Non-zero prior mean and a dense SPD prior precision."""
    return np.linspace(-0.4, 0.4, P), 0.02 * np.eye(P) + 0.005 * np.ones((P, P))


def synth(N, P, G, seed, ids=None, d=3.0, tau=0.7, level=2.6):
    """Counts 0 .. ~1000: log-mean level + N(0, 1.2^2) from X + u_g (at P = 1 only the intercept and u_g)."""
    rng = np.random.default_rng(seed)
    X = np.c_[rng.standard_normal((N, P - 1)) / np.sqrt(max(P - 1, 1)), np.ones(N)]
    g = rng.integers(0, G, N).astype(np.int32) if ids is None else np.asarray(ids, dtype=np.int32)
    ut = tau * rng.standard_normal(G)
    eta = X[:, :-1] @ (1.2 * rng.choice([-1.0, 1.0], P - 1)) + level + ut[g]
    if P == 1:
        eta = eta + 1.2 * rng.standard_normal(N)
    mu = np.exp(eta)
    y = rng.negative_binomial(d, d / (mu + d)).astype(float)
    return X, y, g


def close(a, b, tol=REL):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape
    err = np.abs(a - b) / np.maximum(1.0, np.abs(b))
    assert np.all(np.isfinite(a)) and err.max() <= tol, float(err.max())


def parity(gapi, mode, X, y, g, G, seed, d0=None, samp=SAMP, burn=BURN):
    d0 = D0[mode] if d0 is None else d0
    m0, P0 = prior(X.shape[1])
    b, u, t2, d = gapi.nb_ri(y, X, g, G, m0, P0, A0, B0, TAU2_0, samp, burn, seed, d0=d0, dmode=mode)
    rb, ru, rt, rd = ro.nb_ri(y, X, g, G, m0, P0, A0, B0, TAU2_0, samp, burn, seed, d0=d0, dmode=mode)
    if mode == "real":
        assert np.all(np.abs(d - rd) <= REL_DREAL * np.abs(rd)), (d, rd)
    else:
        assert np.array_equal(d, rd), (d, rd)
    if mode == "fixed":
        assert np.all(d == d0)
    close(b, rb)
    close(u, ru)
    close(t2, rt)
    return b, u, t2, d


PS = [1, 2, 5, 8, 16, 32, 34, 64, 70, 128, 256]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("P", PS)
def test_parity_p(gapi, P, mode):
    """Odd P (k_xbeta, k_xtv_partial), P = 8, 16 (streaming X'v), 32 (packed Gram), 34 (k_xtv_mma), 64 (one Gram tile,
    lean beta draw), 70 (several tiles, shared-memory draw above 64), 128 and 256 (beta drawn out of global scratch);
    the per-lane omega draw below N = 2^15 and the binned one above."""
    N, G = max(4000, 100 * P), 60
    X, y, g = synth(N, P, G, 500 + P)
    assert_regimes(y, D0[mode], "alt", "sp", "normal", *(["devroye"] if mode != "real" else []))
    parity(gapi, mode, X, y, g, G, 71 + P)


@pytest.mark.parametrize("N", [32_767, 32_768])
def test_parity_sampler_switch(gapi, N):
    X, y, g = synth(N, 16, 200, 9)
    parity(gapi, "int", X, y, g, 200, 5)


def _ids(kind, N, rng):
    if kind == "one":
        return np.zeros(N, np.int32), 1
    if kind == "per_row":
        return rng.permutation(N).astype(np.int32), N
    if kind == "empty":                                  # even ids only, and the first and last groups empty
        return (2 * rng.integers(1, 150, N)).astype(np.int32), 301
    if kind == "skewed":                                 # half the rows in group 7, every other row its own group
        G = N // 2 + 8
        g = np.full(N, 7, np.int32)
        rest = rng.permutation(N)[: N - N // 2]
        g[rest] = np.arange(8, 8 + len(rest), dtype=np.int32)
        return g, G
    if kind == "sorted":
        return np.sort(rng.integers(0, 97, N)).astype(np.int32), 97
    raise ValueError(kind)


LAYOUT_SEED = {"one": 1, "per_row": 2, "empty": 3, "skewed": 4, "sorted": 5}


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("kind", list(LAYOUT_SEED))
def test_parity_group_layouts(gapi, kind, mode):
    N, P = 20_000, 8
    rng = np.random.default_rng(LAYOUT_SEED[kind])
    g, G = _ids(kind, N, rng)
    X, y, _ = synth(N, P, G, 7, ids=g)
    parity(gapi, mode, X, y, g, G, 17)


@pytest.mark.parametrize("mode", MODES)
def test_parity_all_zero_group(gapi, mode):
    """Group 3's counts are all zero (b = d on its rows, its u pulled down by the data)."""
    N, P, G = 12_000, 6, 40
    X, y, g = synth(N, P, G, 31)
    y[g == 3] = 0.0
    parity(gapi, mode, X, y, g, G, 33)


@pytest.mark.parametrize("shape", [(6000, 8), (40_000, 16)], ids=lambda s: "N%d-P%d" % s)
def test_parity_real_walk_from_below_one(gapi, shape):
    """d0 = 0.5: the real walk's U(0, 2) proposal, and b = y + d < 1 where y = 0 (the sum-of-gammas regime)."""
    X, y, g = synth(*shape, 50, 41)
    assert_regimes(y, 0.5, "gamma", "alt", "sp", "normal")
    parity(gapi, "real", X, y, g, 50, 43, d0=0.5)


def test_parity_large(gapi):
    """N = 10^6, P = 64, G = 10^4, integer walk, a short chain."""
    N, P, G = 1_000_000, 64, 10_000
    X, y, g = synth(N, P, G, 5)
    parity(gapi, "int", X, y, g, G, 99, samp=2, burn=1)


@pytest.mark.parametrize("mode", MODES)
def test_reproducible_and_optional_outputs(gapi, mode):
    """Two runs of one seed are identical; u = NULL and d_out = NULL leave the other outputs as they were."""
    from bayeslogit_b200 import _lib, gibbs_api
    N, P, G = 50_000, 16, 1000
    X, y, g = synth(N, P, G, 8)
    m0, P0 = prior(P)
    args = (y, X, g, G, m0, P0, A0, B0, TAU2_0, SAMP, BURN, 12)
    a = gapi.nb_ri(*args, d0=D0[mode], dmode=mode)
    b = gapi.nb_ri(*args, d0=D0[mode], dmode=mode)
    for x, z in zip(a, b):
        assert np.array_equal(x, z)
    c = gapi.nb_ri(*args, d0=D0[mode], dmode=mode, keep_u=False)
    assert c[1] is None and np.array_equal(c[0], a[0]) and np.array_equal(c[2], a[2]) and np.array_equal(c[3], a[3])
    beta, tau2 = np.zeros((SAMP, P)), np.zeros(SAMP)
    X, P0f = np.ascontiguousarray(X), np.asfortranarray(P0)      # kept alive across the call
    st = _lib.lib().bl_nb_ri_gibbs(beta.ctypes.data, None, tau2.ctypes.data, None, y.ctypes.data, X.ctypes.data,
                                   g.ctypes.data, G, m0.ctypes.data, P0f.ctypes.data, A0, B0, TAU2_0,
                                   D0[mode], gibbs_api.NB_DMODES[mode], N, P, SAMP, BURN, 12)
    _lib.check(st)
    assert np.array_equal(beta, a[0]) and np.array_equal(tau2, a[2])


class Dev:
    """Device-resident inputs; X may start 8 bytes into its buffer."""

    def __init__(self):
        import torch
        from bayeslogit_b200 import _lib
        self.t, self.L, self.check = torch, _lib.lib(), _lib.check
        self.dev = torch.device("cuda")
        self.st = torch.cuda.current_stream().cuda_stream

    def put(self, a, offset=0, dtype=np.float64):
        t = self.t
        a = np.ascontiguousarray(a, dtype=dtype)
        tdt = t.float64 if dtype == np.float64 else t.int32
        buf = t.zeros(a.size + offset, dtype=tdt, device=self.dev)
        buf[offset:] = t.from_numpy(a.ravel()).to(self.dev)
        return buf, buf.data_ptr() + a.itemsize * offset

    def run(self, X, y, g, G, m0, P0, samp, burn, seed, d0, dmode, x_offset=0):
        from bayeslogit_b200 import gibbs_api
        t = self.t
        N, P = X.shape
        keep = [self.put(X, x_offset), self.put(y), self.put(g, dtype=np.int32), self.put(m0), self.put(P0)]
        (_, tX), (_, ty), (_, tg), (_, tm), (_, tp) = keep
        outs = [t.zeros(s, dtype=t.float64, device=self.dev) for s in ((samp, P), (samp, G), (samp,), (samp,))]
        st = self.L.bl_nb_ri_gibbs_dev(*(o.data_ptr() for o in outs), ty, tX, tg, G, tm, tp, A0, B0, TAU2_0, d0,
                                       gibbs_api.NB_DMODES[dmode], N, P, samp, burn, seed, self.st)
        t.cuda.synchronize()
        self.check(st)
        return [o.cpu().numpy() for o in outs]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("P", [7, 32])
def test_device_entry(gapi, P, mode):
    """The device entry equals the host entry bit for bit; with X 8 bytes into its buffer (scalar X beta and X'v, the
    Gram's 8-byte loads) it still matches the restatement."""
    N, G = 12_000, 150
    X, y, g = synth(N, P, G, 60 + P)
    m0, P0 = prior(P)
    d = Dev()
    got = d.run(X, y, g, G, m0, P0, SAMP, BURN, 3, D0[mode], mode)
    host = gapi.nb_ri(y, X, g, G, m0, P0, A0, B0, TAU2_0, SAMP, BURN, 3, d0=D0[mode], dmode=mode)
    for x, z in zip(got, host):
        assert np.array_equal(x, z)
    b, u, t2, dd = d.run(X, y, g, G, m0, P0, SAMP, BURN, 3, D0[mode], mode, x_offset=1)
    rb, ru, rt, rd = ro.nb_ri(y, X, g, G, m0, P0, A0, B0, TAU2_0, SAMP, BURN, 3, d0=D0[mode], dmode=mode)
    close(b, rb)
    close(u, ru)
    close(t2, rt)
    if mode == "real":
        assert np.all(np.abs(dd - rd) <= REL_DREAL * np.abs(rd))
    else:
        assert np.array_equal(dd, rd)


REFUSALS = [
    ("G", dict(G=0), "G must be at least 1"),
    ("id", dict(bad_id=True), r"group ids must lie in \[0, G\)"),
    ("a0", dict(a0=0.0), "a0, b0 and tau2_0 must be finite and positive"),
    ("b0", dict(b0=float("inf")), "a0, b0 and tau2_0 must be finite and positive"),
    ("tau2_0", dict(tau2_0=-1.0), "a0, b0 and tau2_0 must be finite and positive"),
    ("samp", dict(samp=0), "bad dimensions"),
    ("burn", dict(burn=-1), "bad dimensions"),
    ("N", dict(N=0), "bad dimensions"),
    ("P", dict(P=257), "P > 256"),
    ("dmode", dict(dmode=3), "unknown dmode"),
    ("d0_int", dict(d0=2.5), r"d0 must be an integer >= 1"),
    ("d0_int_inf", dict(d0=float("inf")), r"d0 must be an integer >= 1"),
    ("d0_real", dict(d0=0.0, dmode=2), "d0 must be finite and positive"),
    ("d0_fixed", dict(d0=float("nan"), dmode=0), "d0 must be finite and positive"),
    ("count_negative", dict(bad_y=-1.0), "counts y must be finite, non-negative and below 2"),
    ("count_nan_fixed", dict(bad_y=float("nan"), dmode=0), "counts y must be finite, non-negative and below 2"),
    ("count_big_real", dict(bad_y=2.0 ** 31 - 1, dmode=2), "counts y must be finite, non-negative and below 2"),
]


@pytest.mark.parametrize("name,fault,msg", REFUSALS, ids=[r[0] for r in REFUSALS])
@pytest.mark.parametrize("where", ["host", "device"])
def test_refusals(engine, name, fault, msg, where):
    """Every refusal raises its own message and leaves the outputs as they were."""
    import torch
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    N0, P0_, G0 = 500, 3, 10
    X, y, g = synth(N0, P0_, G0, 1)
    a = dict(G=G0, a0=A0, b0=B0, tau2_0=TAU2_0, samp=3, burn=1, N=N0, P=P0_, d0=2.0, dmode=1)
    a.update({k: v for k, v in fault.items() if k not in ("bad_id", "bad_y")})
    if fault.get("bad_id"):
        g = g.copy()
        g[N0 // 2] = G0
    if "bad_y" in fault:
        y = y.copy()
        y[N0 // 3] = fault["bad_y"]
    P = a["P"]
    if P != P0_:
        X = np.ones((N0, P))
    m0, Pr = prior(P)
    sentinel = 1234.5
    S = max(a["samp"], 1)
    shp = [(S, P), (S, max(a["G"], 1)), (S,), (S,)]
    scal = (a["G"],)
    tail = (a["a0"], a["b0"], a["tau2_0"], a["d0"], a["dmode"], a["N"], P, a["samp"], a["burn"], 7)
    if where == "host":
        outs = [np.full(s, sentinel) for s in shp]
        ins = [np.ascontiguousarray(y), np.ascontiguousarray(X), np.ascontiguousarray(g, dtype=np.int32), m0,
               np.asfortranarray(Pr)]
        st = L.bl_nb_ri_gibbs(*(o.ctypes.data for o in outs), *(i.ctypes.data for i in ins[:3]), *scal,
                              ins[3].ctypes.data, ins[4].ctypes.data, *tail)
        got = outs
    else:
        dev = torch.device("cuda")
        outs = [torch.full(s, sentinel, dtype=torch.float64, device=dev) for s in shp]
        ins = [torch.from_numpy(np.ascontiguousarray(v)).to(dev) for v in (y, X, g.astype(np.int32), m0, Pr)]
        st = L.bl_nb_ri_gibbs_dev(*(o.data_ptr() for o in outs), *(i.data_ptr() for i in ins[:3]), *scal,
                                  ins[3].data_ptr(), ins[4].data_ptr(), *tail, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        got = [o.cpu().numpy() for o in outs]
    with pytest.raises(_lib.EngineError, match="nb_ri_gibbs: " + msg):
        _lib.check(st)
    assert st != 0
    for o in got:
        assert np.all(o == sentinel)


def test_recovers_tau_d_and_u(gapi):
    """N = 200 000 rows in G = 500 groups, tau = 0.7, d = 3, integer walk from d0 = 1, burn 300, samp 700: the
    posterior mean of tau lies within 0.1 of the truth (the realised intercepts have sd 0.7 exactly), that of d within
    0.5 of 3, and the posterior-mean u correlate with the true u above 0.9.  The true intercept is 0, where the chain
    starts: with 400 rows a group the centred chain moves slowly along the intercept / mean-of-u ridge (DESIGN.md
    section 11)."""
    N, P, G = 200_000, 3, 500
    rng = np.random.default_rng(77)
    X = np.c_[np.ones(N), rng.standard_normal((N, P - 1))]
    ut = rng.standard_normal(G)
    ut = 0.7 * (ut - ut.mean()) / ut.std()
    g = rng.integers(0, G, N).astype(np.int32)
    bt = np.array([0.0, 0.5, -0.5])
    mu = np.exp(X @ bt + ut[g])
    y = rng.negative_binomial(3.0, 3.0 / (mu + 3.0)).astype(float)
    b, u, t2, d = gapi.nb_ri(y, X, g, G, np.zeros(P), 0.01 * np.eye(P), 1.0, 1.0, 1.0, 700, 300, 4, d0=1.0,
                             dmode="int")
    assert abs(np.sqrt(t2).mean() - 0.7) < 0.1, np.sqrt(t2).mean()
    assert abs(d.mean() - 3.0) < 0.5, d.mean()
    assert np.corrcoef(u.mean(0), ut)[0, 1] > 0.9
    assert np.all(np.abs(b.mean(0) - bt) < 0.1), b.mean(0)
