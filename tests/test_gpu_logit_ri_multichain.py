"""Several random-intercept logit chains on one shared data set (bl_logit_ri_multichain / _dev): chain c must be, bit
for bit, the single chain bl_logit_ri_gibbs(..., seed + c) -- beta, u and tau2 -- at every kernel choice of the psi pass
(k_logit_psi_draw<true> for one chain, k_logit_psi_draw_shared<true> in groups of 8 chains, k_xbeta / k_xbeta_shared
then k_ri_psi and the refill draw when unfused), of X'v, the Gram and the beta draw, and at every group layout."""
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

A0, B0, TAU2_0 = 2.0, 1.5, 1.0
BURN, SAMP = 4, 6
SEED = 21
CHAINS = [1, 2, 3, 8, 9]          # 9 crosses the 8-chain group of the shared psi pass


@pytest.fixture(scope="module")
def gapi(engine):
    from bayeslogit_b200 import gibbs_api
    return gibbs_api


def synth(N, P, G, seed, tau=1.0, ids=None, nmax=1):
    rng = np.random.default_rng(seed)
    X = np.c_[np.ones(N), rng.standard_normal((N, P - 1)) / np.sqrt(max(P - 1, 1))]
    bt = rng.uniform(-1.0, 1.0, P)
    ut = tau * rng.standard_normal(G)
    g = rng.integers(0, G, N).astype(np.int32) if ids is None else np.asarray(ids, dtype=np.int32)
    n = rng.integers(1, nmax + 1, N).astype(float)
    p = 1.0 / (1.0 + np.exp(-(X @ bt + ut[g])))
    y = rng.binomial(n.astype(int), p) / n
    return X, y, n, g


def prior(P):
    return np.zeros(P), 0.05 * np.eye(P)


def assert_chains_equal(multi, singles):
    """multi: (beta [K,S,P], u [K,S,G], tau2 [K,S]); singles[c]: the single chain's (beta, u, tau2)."""
    b, u, t2 = multi
    assert b.shape[0] == len(singles)
    for c, (sb, su, st) in enumerate(singles):
        assert np.array_equal(b[c], sb), (c, float(np.abs(b[c] - sb).max()))
        assert np.array_equal(u[c], su), (c, float(np.abs(u[c] - su).max()))
        assert np.array_equal(t2[c], st), (c, float(np.abs(t2[c] - st).max()))


SHAPES = {1: 40, 7: 40, 2: 60, 16: 60, 64: 80, 70: 30, 128: 30}     # P -> G
N_SHAPE = 3001


@functools.lru_cache(maxsize=None)
def _shape_data(P):
    return synth(N_SHAPE, P, SHAPES[P], 500 + P, nmax=2)


@functools.lru_cache(maxsize=None)
def _single(P, seed, flags):
    from bayeslogit_b200 import gibbs_api
    X, y, n, g = _shape_data(P)
    return gibbs_api.logit_ri(y, X, n, g, SHAPES[P], *prior(P), A0, B0, TAU2_0, SAMP, BURN, seed, flags=flags)


@pytest.mark.parametrize("chains", CHAINS)
@pytest.mark.parametrize("P", list(SHAPES))
def test_equals_single_chains(gapi, P, chains):
    """P = 1, 7 (odd: k_xbeta, scalar X'v, unfused draw); 2, 16, 64 (fused shared pass, streaming X'v, packed Gram,
    lean beta draw); 70 (several Gram tiles, k_xtv_mma); 128 (global-scratch beta draw)."""
    X, y, n, g = _shape_data(P)
    G = SHAPES[P]
    got = gapi.logit_ri_multichain(y, X, n, g, G, *prior(P), A0, B0, TAU2_0, SAMP, BURN, SEED, chains)
    assert_chains_equal(got, [_single(P, SEED + c, 0) for c in range(chains)])
    if chains > 1:
        assert not np.array_equal(got[2][0], got[2][1])


@pytest.mark.parametrize("chains", [1, 3, 9])
@pytest.mark.parametrize("P", [2, 64])
def test_unfused_equals_single_chains(gapi, P, chains):
    """BL_GIBBS_UNFUSED: eta from k_xbeta_mma / k_xbeta_shared, k_ri_psi, the refill draw over chains * N pairs."""
    X, y, n, g = _shape_data(P)
    G = SHAPES[P]
    got = gapi.logit_ri_multichain(y, X, n, g, G, *prior(P), A0, B0, TAU2_0, SAMP, BURN, SEED, chains,
                                   flags=gapi.UNFUSED)
    assert_chains_equal(got, [_single(P, SEED + c, gapi.UNFUSED) for c in range(chains)])
    # the single chain's two paths are the same chain, so the unfused chains equal the fused single chains too
    assert_chains_equal(got, [_single(P, SEED + c, 0) for c in range(chains)])


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


@pytest.mark.parametrize("kind", list(LAYOUT_SEED))
def test_group_layouts(gapi, kind):
    N, P, K = 20_000, 8, 3
    rng = np.random.default_rng(LAYOUT_SEED[kind])
    g, G = _ids(kind, N, rng)
    X, y, n, _ = synth(N, P, G, 7, ids=g)
    m0, P0 = prior(P)
    got = gapi.logit_ri_multichain(y, X, n, g, G, m0, P0, A0, B0, TAU2_0, SAMP, BURN, 17, K)
    singles = [gapi.logit_ri(y, X, n, g, G, m0, P0, A0, B0, TAU2_0, SAMP, BURN, 17 + c) for c in range(K)]
    assert_chains_equal(got, singles)


def test_without_u(gapi):
    """u = NULL: no u draws are stored, beta and tau2 are unchanged."""
    P = 16
    X, y, n, g = _shape_data(P)
    G = SHAPES[P]
    a = gapi.logit_ri_multichain(y, X, n, g, G, *prior(P), A0, B0, TAU2_0, SAMP, BURN, SEED, 3)
    b = gapi.logit_ri_multichain(y, X, n, g, G, *prior(P), A0, B0, TAU2_0, SAMP, BURN, SEED, 3, keep_u=False)
    assert b[1] is None
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[2], b[2])


def test_reproducible(gapi):
    N, P, G, K = 50_000, 16, 1000, 4
    X, y, n, g = synth(N, P, G, 8)
    m0, P0 = prior(P)
    a = gapi.logit_ri_multichain(y, X, n, g, G, m0, P0, A0, B0, TAU2_0, SAMP, BURN, 12, K)
    b = gapi.logit_ri_multichain(y, X, n, g, G, m0, P0, A0, B0, TAU2_0, SAMP, BURN, 12, K)
    for x, z in zip(a, b):
        assert np.array_equal(x, z)


class Dev:
    """Device-resident inputs; X may start x_offset doubles into its buffer."""

    def __init__(self, X, y, n, g, G, m0, P0, x_offset=0):
        import torch
        from bayeslogit_b200 import _lib
        self.t, self.L, self.check = torch, _lib.lib(), _lib.check
        self.dev = torch.device("cuda")
        self.st = torch.cuda.current_stream().cuda_stream
        self.N, self.P = X.shape
        self.G = G
        self.keep = [self.put(X, x_offset), self.put(y), self.put(n), self.put(g, dtype=np.int32), self.put(m0),
                     self.put(np.asfortranarray(P0).ravel(order="F"))]

    def put(self, a, offset=0, dtype=np.float64):
        t = self.t
        a = np.ascontiguousarray(a, dtype=dtype)
        tdt = t.float64 if dtype == np.float64 else t.int32
        buf = t.zeros(a.size + offset, dtype=tdt, device=self.dev)
        buf[offset:] = t.from_numpy(a.ravel()).to(self.dev)
        return buf, buf.data_ptr() + a.itemsize * offset

    def _ptrs(self):
        return [p for _, p in self.keep]

    def single(self, samp, burn, seed, flags=0):
        t = self.t
        tX, ty, tn, tg, tm, tp = self._ptrs()
        beta = t.zeros((samp, self.P), dtype=t.float64, device=self.dev)
        u = t.zeros((samp, self.G), dtype=t.float64, device=self.dev)
        tau2 = t.zeros((samp,), dtype=t.float64, device=self.dev)
        self.check(self.L.bl_logit_ri_gibbs_dev(beta.data_ptr(), u.data_ptr(), tau2.data_ptr(), ty, tX, tn, tg, self.G,
                                                tm, tp, A0, B0, TAU2_0, self.N, self.P, samp, burn, seed, flags, self.st))
        t.cuda.synchronize()
        return beta.cpu().numpy(), u.cpu().numpy(), tau2.cpu().numpy()

    def multi(self, samp, burn, seed, chains, flags=0, keep_u=True):
        t = self.t
        tX, ty, tn, tg, tm, tp = self._ptrs()
        beta = t.zeros((chains, samp, self.P), dtype=t.float64, device=self.dev)
        u = t.zeros((chains, samp, self.G), dtype=t.float64, device=self.dev)
        tau2 = t.zeros((chains, samp), dtype=t.float64, device=self.dev)
        self.check(self.L.bl_logit_ri_multichain_dev(beta.data_ptr(), u.data_ptr() if keep_u else None,
                                                     tau2.data_ptr(), ty, tX, tn, tg, self.G, tm, tp, A0, B0, TAU2_0,
                                                     chains, self.N, self.P, samp, burn, seed, flags, self.st))
        t.cuda.synchronize()
        return beta.cpu().numpy(), u.cpu().numpy() if keep_u else None, tau2.cpu().numpy()


@pytest.mark.parametrize("P", [7, 32])
def test_device_entry(gapi, P):
    """The device entry equals the host entry bit for bit; with X 8 bytes into its buffer (k_xbeta, scalar X'v,
    unfused draw) the chains still equal the single chain's device entry on the same unaligned X."""
    N, G, K = 12_000, 150, 5
    X, y, n, g = synth(N, P, G, 60 + P, nmax=2)
    m0, P0 = prior(P)
    d = Dev(X, y, n, g, G, m0, P0)
    got = d.multi(SAMP, BURN, 3, K)
    host = gapi.logit_ri_multichain(y, X, n, g, G, m0, P0, A0, B0, TAU2_0, SAMP, BURN, 3, K)
    for x, z in zip(got, host):
        assert np.array_equal(x, z)
    nu = d.multi(SAMP, BURN, 3, K, keep_u=False)
    assert np.array_equal(nu[0], got[0]) and np.array_equal(nu[2], got[2])
    du = Dev(X, y, n, g, G, m0, P0, x_offset=1)
    assert_chains_equal(du.multi(SAMP, BURN, 3, K), [du.single(SAMP, BURN, 3 + c) for c in range(K)])


def test_large(gapi):
    """N = 10^6, P = 64, G = 10^4, 8 chains for a few iterations, on device-resident data."""
    N, P, G, K = 1_000_000, 64, 10_000, 8
    X, y, n, g = synth(N, P, G, 5, tau=0.7)
    d = Dev(X, y, n, g, G, *prior(P))
    got = d.multi(2, 1, 99, K)
    assert_chains_equal(got, [d.single(2, 1, 99 + c) for c in range(K)])


@pytest.mark.parametrize("flags", [0, 4], ids=["fused", "unfused"])     # 4: BL_GIBBS_UNFUSED
@pytest.mark.parametrize("P", [7, 16, 128])
def test_launches_do_not_depend_on_chains(gapi, P, flags):
    """One launch per kernel per iteration for all chains: K = 9 launches as many kernels as K = 1."""
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    X, y, n, g = _shape_data(P)
    G = SHAPES[P]

    def launches(chains, samp):
        before = L.bl_kernel_launches()
        gapi.logit_ri_multichain(y, X, n, g, G, *prior(P), A0, B0, TAU2_0, samp, 1, 5, chains, flags=flags)
        return L.bl_kernel_launches() - before

    per_iter = [(launches(K, 5) - launches(K, 2)) / 3 for K in (1, 9)]
    assert per_iter[0] == per_iter[1] and per_iter[0] > 0, per_iter
    assert launches(1, 2) == launches(9, 2)


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
    ("flags", dict(flags=1), "unknown flag"),
    ("chains0", dict(chains=0), "chains must be at least 1"),
    ("chains_grid", dict(chains=65536), "chains must be at most 65535"),
    ("chainsN", dict(chains=2, N=1 << 30), r"chains \* N must stay below 2\^31"),
    ("chainsG", dict(chains=2, G=1 << 30), r"chains \* G must stay below 2\^31"),
    ("null", dict(null=True), "null argument"),
]


@pytest.mark.parametrize("name,fault,msg", REFUSALS, ids=[r[0] for r in REFUSALS])
@pytest.mark.parametrize("where", ["host", "device"])
def test_refusals(engine, name, fault, msg, where):
    """Every refusal raises its own message and leaves the outputs as they were; the host entry launches nothing."""
    import torch
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    N0, P0_, G0 = 500, 3, 10
    X, y, n, g = synth(N0, P0_, G0, 1)
    a = dict(G=G0, a0=A0, b0=B0, tau2_0=TAU2_0, samp=3, burn=1, N=N0, P=P0_, flags=0, chains=2)
    a.update({k: v for k, v in fault.items() if k not in ("bad_id", "null")})
    if fault.get("bad_id"):
        g = g.copy()
        g[N0 // 2] = G0
    P = a["P"]
    if P != P0_:
        X = np.ones((N0, P))
    m0, Pr = prior(P)
    sentinel = 1234.5
    # the refusals come before any output is touched: small buffers stand in for the huge shapes
    K, S, G = min(max(a["chains"], 1), 4), max(a["samp"], 1), min(max(a["G"], 1), 64)
    shp = [(K, S, P), (K, S, G), (K, S)]
    args = lambda ins: [*ins[:4], a["G"], ins[4], ins[5], a["a0"], a["b0"], a["tau2_0"], a["chains"], a["N"], P,
                        a["samp"], a["burn"], 7, a["flags"]]
    before = L.bl_kernel_launches()
    if where == "host":
        outs = [np.full(s, sentinel) for s in shp]
        ins = [np.ascontiguousarray(y), np.ascontiguousarray(X), np.ascontiguousarray(n),
               np.ascontiguousarray(g, dtype=np.int32), m0, np.asfortranarray(Pr)]
        ptrs = [i.ctypes.data for i in ins]
        if fault.get("null"):
            ptrs[3] = None
        st = L.bl_logit_ri_multichain(*(o.ctypes.data for o in outs), *args(ptrs))
        got = outs
    else:
        dev = torch.device("cuda")
        outs = [torch.full(s, sentinel, dtype=torch.float64, device=dev) for s in shp]
        ins = [torch.from_numpy(np.ascontiguousarray(v)).to(dev) for v in (y, X, n, g.astype(np.int32), m0, Pr)]
        ptrs = [i.data_ptr() for i in ins]
        if fault.get("null"):
            ptrs[3] = None
        torch.cuda.synchronize()
        before = L.bl_kernel_launches()
        st = L.bl_logit_ri_multichain_dev(*(o.data_ptr() for o in outs), *args(ptrs),
                                          torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        got = [o.cpu().numpy() for o in outs]
    with pytest.raises(_lib.EngineError, match="logit_ri_multichain: " + msg):
        _lib.check(st)
    assert st != 0
    for o in got:
        assert np.all(o == sentinel)
    if where == "host" or not fault.get("bad_id"):
        assert L.bl_kernel_launches() == before


def split_rhat(draws):
    """Split-R-hat of draws [chains, n]: each chain cut into halves, then the Gelman-Rubin ratio."""
    K, n = draws.shape
    h = n // 2
    s = np.concatenate([draws[:, :h], draws[:, h:2 * h]], axis=0)
    W = s.var(axis=1, ddof=1).mean()
    B = h * s.mean(axis=1).var(ddof=1)
    return float(np.sqrt(((h - 1) / h * W + B / h) / W))


def test_tau2_rhat_and_recovery(gapi):
    """The use case: 4 chains on the single chain's recovery data (N = 200 000, G = 2000, tau = 0.8); split-R-hat of
    tau2 below 1.1 and the pooled posterior mean of tau within 0.1 of the truth."""
    N, P, G = 200_000, 4, 2000
    rng = np.random.default_rng(77)
    X = np.c_[np.ones(N), rng.standard_normal((N, P - 1))]
    ut = rng.standard_normal(G)
    ut = 0.8 * (ut - ut.mean()) / ut.std()
    g = rng.integers(0, G, N).astype(np.int32)
    bt = np.array([-0.3, 0.5, -0.5, 0.25])
    y = rng.binomial(1, 1.0 / (1.0 + np.exp(-(X @ bt + ut[g])))).astype(float)
    b, u, t2 = gapi.logit_ri_multichain(y, X, np.ones(N), g, G, np.zeros(P), 0.01 * np.eye(P), 1.0, 1.0, 1.0, 400,
                                        200, 4, 4)
    assert split_rhat(t2) < 1.1, split_rhat(t2)
    assert abs(np.sqrt(t2.mean()) - 0.8) < 0.1, np.sqrt(t2.mean())
