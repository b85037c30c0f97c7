"""Binomial logit with group random intercepts on the GPU (bl_logit_ri_gibbs / bl_logit_ri_gibbs_dev) against the CPU
restatement of the same four steps (tests/ri_oracle/logit_ri_oracle.c): beta, u and tau2 within 1e-8 over 20
iterations at every kernel choice and group layout -- one group, a group per row, empty groups, one group holding
half the rows beside thousands of singletons (its sums cross many chunks of the sorted rows), ids in random order.
The engine sums in other orders than the restatement (MMA psi, tiled Gram, chunked group sums), so the chains agree
to rounding, not bit for bit; the fused and unfused paths, the host and device entries and two runs of one seed
agree bit for bit."""
import numpy as np
import pytest

import _logit_ri_oracle as ro

pytestmark = pytest.mark.gpu

A0, B0, TAU2_0 = 2.0, 1.5, 1.0
BURN, SAMP = 8, 12


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


def close(a, b, tol=1e-8):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape
    err = np.abs(a - b) / np.maximum(1.0, np.abs(b))
    assert np.all(np.isfinite(a)) and err.max() <= tol, float(err.max())


def prior(P, dense=False, seed=0):
    if not dense:
        return np.zeros(P), 0.05 * np.eye(P)
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((P, P))
    return rng.uniform(-0.5, 0.5, P), A @ A.T / P + 0.2 * np.eye(P)


def parity(gapi, X, y, n, g, G, m0, P0, seed, flags=0, burn=BURN, samp=SAMP):
    b, u, t2 = gapi.logit_ri(y, X, n, g, G, m0, P0, A0, B0, TAU2_0, samp, burn, seed, flags=flags)
    rb, ru, rt = ro.logit_ri(y, X, n, g, G, m0, P0, A0, B0, TAU2_0, samp, burn, seed)
    close(b, rb)
    close(u, ru)
    close(t2, rt)
    return b, u, t2


@pytest.mark.parametrize("P", [1, 2, 7, 32, 64, 70, 128])
def test_parity_p(gapi, P):
    """Odd P (k_xbeta, k_xtv_partial, unfused draw), even P (fused draw, MMA X'v), power-of-two P (streaming X'v),
    P > 64 (several Gram tiles, the general beta draw)."""
    N, G = 5000, 40
    X, y, n, g = synth(N, P, G, 100 + P)
    parity(gapi, X, y, n, g, G, *prior(P), 31 + P)


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
def test_parity_group_layouts(gapi, kind):
    N, P = 20_000, 8
    rng = np.random.default_rng(LAYOUT_SEED[kind])
    g, G = _ids(kind, N, rng)
    X, y, n, _ = synth(N, P, G, 7, ids=g)
    parity(gapi, X, y, n, g, G, *prior(P), 17)


def test_parity_binomial_dense_prior(gapi):
    """Trials n in 1..5 and a non-zero m0 with a dense P0."""
    N, P, G = 6000, 6, 50
    X, y, n, g = synth(N, P, G, 21, nmax=5)
    parity(gapi, X, y, n, g, G, *prior(P, dense=True, seed=3), 23)


def test_parity_large(gapi):
    """N = 10^6, P = 64, G = 10^4, a short chain."""
    N, P, G = 1_000_000, 64, 10_000
    X, y, n, g = synth(N, P, G, 5, tau=0.7)
    parity(gapi, X, y, n, g, G, *prior(P), 99, burn=1, samp=2)


@pytest.mark.parametrize("P", [2, 16, 64])
def test_fused_equals_unfused(gapi, P):
    """psi + omega in one pass over X (k_logit_psi_draw with the offset) and as k_xbeta_mma, k_ri_psi and the refill
    draw give the same chain bit for bit."""
    N, G = 30_000, 300
    X, y, n, g = synth(N, P, G, 40 + P, nmax=3)
    m0, P0 = prior(P)
    a = gapi.logit_ri(y, X, n, g, G, m0, P0, A0, B0, TAU2_0, SAMP, BURN, 5, flags=0)
    b = gapi.logit_ri(y, X, n, g, G, m0, P0, A0, B0, TAU2_0, SAMP, BURN, 5, flags=gapi.UNFUSED)
    for x, z in zip(a, b):
        assert np.array_equal(x, z), float(np.abs(x - z).max())


def test_reproducible(gapi):
    N, P, G = 50_000, 16, 1000
    X, y, n, g = synth(N, P, G, 8)
    m0, P0 = prior(P)
    a = gapi.logit_ri(y, X, n, g, G, m0, P0, A0, B0, TAU2_0, SAMP, BURN, 12)
    b = gapi.logit_ri(y, X, n, g, G, m0, P0, A0, B0, TAU2_0, SAMP, BURN, 12)
    for x, z in zip(a, b):
        assert np.array_equal(x, z)
    c = gapi.logit_ri(y, X, n, g, G, m0, P0, A0, B0, TAU2_0, SAMP, BURN, 12, keep_u=False)
    assert c[1] is None and np.array_equal(c[0], a[0]) and np.array_equal(c[2], a[2])


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

    def run(self, X, y, n, g, G, m0, P0, samp, burn, seed, flags=0, x_offset=0, fill=0.0, check=True):
        t = self.t
        N, P = X.shape
        keep = [self.put(X, x_offset), self.put(y), self.put(n), self.put(g, dtype=np.int32), self.put(m0),
                self.put(P0)]
        (_, tX), (_, ty), (_, tn), (_, tg), (_, tm), (_, tp) = keep
        beta = t.full((samp, P), fill, dtype=t.float64, device=self.dev)
        u = t.full((samp, G), fill, dtype=t.float64, device=self.dev)
        tau2 = t.full((samp,), fill, dtype=t.float64, device=self.dev)
        st = self.L.bl_logit_ri_gibbs_dev(beta.data_ptr(), u.data_ptr(), tau2.data_ptr(), ty, tX, tn, tg, G, tm, tp,
                                          A0, B0, TAU2_0, N, P, samp, burn, seed, flags, self.st)
        t.cuda.synchronize()
        if check:
            self.check(st)
        return st, beta.cpu().numpy(), u.cpu().numpy(), tau2.cpu().numpy()


@pytest.mark.parametrize("P", [7, 32])
def test_device_entry(gapi, P):
    """The device entry equals the host entry bit for bit; with X 8 bytes into its buffer (scalar kernels, unfused
    draw) it still matches the restatement."""
    N, G = 12_000, 150
    X, y, n, g = synth(N, P, G, 60 + P, nmax=2)
    m0, P0 = prior(P)
    d = Dev()
    _, b, u, t2 = d.run(X, y, n, g, G, m0, P0, SAMP, BURN, 3)
    hb, hu, ht = gapi.logit_ri(y, X, n, g, G, m0, P0, A0, B0, TAU2_0, SAMP, BURN, 3)
    assert np.array_equal(b, hb) and np.array_equal(u, hu) and np.array_equal(t2, ht)
    _, b1, u1, t21 = d.run(X, y, n, g, G, m0, P0, SAMP, BURN, 3, x_offset=1)
    rb, ru, rt = ro.logit_ri(y, X, n, g, G, m0, P0, A0, B0, TAU2_0, SAMP, BURN, 3)
    close(b1, rb)
    close(u1, ru)
    close(t21, rt)


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
]


@pytest.mark.parametrize("name,fault,msg", REFUSALS, ids=[r[0] for r in REFUSALS])
@pytest.mark.parametrize("where", ["host", "device"])
def test_refusals(engine, name, fault, msg, where):
    """Every refusal raises its own message and leaves the outputs as they were."""
    import torch
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    N0, P0_, G0 = 500, 3, 10
    X, y, n, g = synth(N0, P0_, G0, 1)
    a = dict(G=G0, a0=A0, b0=B0, tau2_0=TAU2_0, samp=3, burn=1, N=N0, P=P0_, flags=0)
    a.update({k: v for k, v in fault.items() if k != "bad_id"})
    if fault.get("bad_id"):
        g = g.copy()
        g[N0 // 2] = G0
    P = a["P"]
    if P != P0_:
        X = np.ones((N0, P))
    m0, Pr = prior(P)
    sentinel = 1234.5
    shp = [(max(a["samp"], 1), P), (max(a["samp"], 1), max(a["G"], 1)), (max(a["samp"], 1),)]
    if where == "host":
        outs = [np.full(s, sentinel) for s in shp]
        ins = [np.ascontiguousarray(y), np.ascontiguousarray(X), np.ascontiguousarray(n),
               np.ascontiguousarray(g, dtype=np.int32), m0, np.asfortranarray(Pr)]
        st = L.bl_logit_ri_gibbs(*(o.ctypes.data for o in outs), *(i.ctypes.data for i in ins[:4]), a["G"],
                                 ins[4].ctypes.data, ins[5].ctypes.data, a["a0"], a["b0"], a["tau2_0"], a["N"], P,
                                 a["samp"], a["burn"], 7, a["flags"])
        got = outs
    else:
        dev = torch.device("cuda")
        outs = [torch.full(s, sentinel, dtype=torch.float64, device=dev) for s in shp]
        ins = [torch.from_numpy(np.ascontiguousarray(v)).to(dev) for v in (y, X, n, g.astype(np.int32), m0, Pr)]
        st = L.bl_logit_ri_gibbs_dev(*(o.data_ptr() for o in outs), *(i.data_ptr() for i in ins[:4]), a["G"],
                                     ins[4].data_ptr(), ins[5].data_ptr(), a["a0"], a["b0"], a["tau2_0"], a["N"], P,
                                     a["samp"], a["burn"], 7, a["flags"], torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        got = [o.cpu().numpy() for o in outs]
    with pytest.raises(_lib.EngineError, match=msg):
        _lib.check(st)
    assert st != 0
    for o in got:
        assert np.all(o == sentinel)


def test_recovers_tau(gapi):
    """N = 200 000 rows in G = 2000 groups, tau = 0.8: the posterior mean of tau lies within 0.1 of the truth (the
    realised intercepts have sd 0.8 exactly; 2000 groups pin tau to a few per cent)."""
    N, P, G = 200_000, 4, 2000
    rng = np.random.default_rng(77)
    X = np.c_[np.ones(N), rng.standard_normal((N, P - 1))]
    ut = rng.standard_normal(G)
    ut = 0.8 * (ut - ut.mean()) / ut.std()
    g = rng.integers(0, G, N).astype(np.int32)
    bt = np.array([-0.3, 0.5, -0.5, 0.25])
    y = rng.binomial(1, 1.0 / (1.0 + np.exp(-(X @ bt + ut[g])))).astype(float)
    b, u, t2 = gapi.logit_ri(y, X, np.ones(N), g, G, np.zeros(P), 0.01 * np.eye(P), 1.0, 1.0, 1.0, 400, 200, 4)
    assert abs(np.sqrt(t2.mean()) - 0.8) < 0.1, np.sqrt(t2.mean())
    assert np.all(np.abs(b.mean(0) - bt) < 0.1), b.mean(0)
    assert np.corrcoef(u.mean(0), ut)[0, 1] > 0.8
