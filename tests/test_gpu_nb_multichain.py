"""Several negative-binomial chains on one shared data set (bl_nb_multichain): chain c must be, bit for bit, the
single-chain sweep with seed + c -- bl_nb_gibbs_df (integer walk on d), bl_nb_gibbs_dfreal (real walk), or rows
burn .. burn + samp - 1 of bl_nb_gibbs (d fixed, every iteration recorded).

The equality rests on three things: the m8n8k4 f64 MMA forms each element of its output tile from that element's own
row and column only (k_xbeta_shared puts 8 chains' beta in the 8 B columns where the single chain repeats one beta);
every other stage runs the single chain's kernel with a chain grid dimension over the single chain's partition; and
the omega draw of every chain runs the sampler path the single chain picks by its own N.
"""
import numpy as np
import pytest

from oracle import loader

pytestmark = pytest.mark.gpu

DMODES = ["fixed", "int", "real"]
# int: from d = 2 the first proposals include d = 1, which the likelihood at beta = 0 prefers, so d moves at once
D0 = {"fixed": 1.0, "int": 2.0, "real": 2.5}

# (N, P), each reaching a different choice of kernels
SHAPES = [
    (2000, 5),       # odd P: k_xbeta with a chain dimension, k_xtv_partial; per-lane rpg_hybrid
    (4001, 8),       # per-lane draw although chains * N >= 2^15 at 9 chains (the path is picked by N)
    (40_000, 16),    # regime-binned draw
    (30_011, 32),    # packed Gram
    (20_000, 64),    # one Gram tile, lean beta draw
    (10_007, 70),    # several Gram tiles, shared-memory beta draw at P > 64
    (6000, 128),     # beta drawn out of global scratch, one block per chain
    (30_000, 256),   # the same at the largest P
]
CHAINS = [1, 2, 3, 8, 9]
SEED = 4343
SAMP, BURN = 4, 2
PRIOR = 0.01


@pytest.fixture(scope="module")
def gapi(engine):
    from bayeslogit_b200 import gibbs_api
    return gibbs_api


def synth_nb(N, P, seed, d=3.0):
    """Counts 0 .. ~500 (log-mean 2.6 + N(0, 1.2^2)): with d = 1 or 2, b = y + d spans the Devroye (b = 1, 2),
    alternate (b <= 13), saddle-point (b <= 170) and normal (b > 170) regimes of rpg_hybrid; with d = 2.5 all but
    Devroye."""
    rng = np.random.default_rng(seed)
    X = np.c_[rng.standard_normal((N, P - 1)) / np.sqrt(P - 1), np.ones(N)]
    bt = np.r_[1.2 * rng.choice([-1.0, 1.0], P - 1), 2.6]
    mu = np.exp(X @ bt)
    y = rng.negative_binomial(d, d / (mu + d)).astype(float)
    return X, y, np.zeros(P), PRIOR * np.eye(P)


def close(a, b, rel):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape
    err = np.abs(a - b) / np.maximum(np.abs(b), 1e-300)
    assert np.all(np.isfinite(a)) and err.max() <= rel, float(err.max())


_data = {}
_single = {}


def data(shape):
    if shape not in _data:
        _data[shape] = synth_nb(*shape, 200 + shape[0] + shape[1])
    return _data[shape]


def single_chain(gapi, X, y, m0, P0, samp, burn, seed, dmode):
    """(beta [samp x P], d [samp]) of the single-chain entry that dmode names."""
    d0 = D0[dmode]
    if dmode == "fixed":
        _, b = gapi.nb_gibbs(y, X, d0, m0, P0, samp + burn, seed)
        return b[burn:], np.full(samp, d0)
    _, b, d = gapi.nb_gibbs_df(y, X, m0, P0, samp, burn, seed, d0=d0, real_d=dmode == "real")
    return b, d


def cached_single(gapi, shape, seed, dmode):
    key = (shape, seed, dmode)
    if key not in _single:
        X, y, m0, P0 = data(shape)
        _single[key] = single_chain(gapi, X, y, m0, P0, SAMP, BURN, seed, dmode)
    return _single[key]


def test_counts_span_every_sampler_regime():
    for shape in SHAPES:
        _, y, _, _ = data(shape)
        for d0 in sorted(set(D0.values())):
            b = y + d0
            assert ((b > 1) & (b <= 13) & (b != 2)).any(), (shape, d0)
            assert ((b > 13) & (b <= 170)).any() and (b > 170).any(), (shape, d0)
            assert d0 not in (1.0, 2.0) or (b == 2).any(), shape
            assert d0 != 1.0 or (b == 1).any(), shape


@pytest.mark.parametrize("dmode", DMODES)
@pytest.mark.parametrize("chains", CHAINS)
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "N%d-P%d" % s)
def test_nb_multichain_equals_single_chains(gapi, shape, chains, dmode):
    """chains = 3 leaves padding columns in the MMA tile, 9 needs a second group of 8."""
    X, y, m0, P0 = data(shape)
    N, P = shape
    b, d = gapi.nb_multichain(y, X, m0, P0, SAMP, BURN, SEED, chains, d0=D0[dmode], dmode=dmode)
    assert b.shape == (chains, SAMP, P) and d.shape == (chains, SAMP)
    assert np.all(np.isfinite(b))
    for c in range(chains):
        rb, rd = cached_single(gapi, shape, SEED + c, dmode)
        assert np.array_equal(b[c], rb), (c, float(np.abs(b[c] - rb).max()))
        assert np.array_equal(d[c], rd), (c, d[c], rd)
    if dmode != "fixed":
        assert np.any(d != D0[dmode])                       # the dispersion moves


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

    def multichain(self, X, y, m0, P0, samp, burn, seed, chains, d0, dmode, x_offset):
        """bl_nb_multichain_dev with X x_offset doubles into its buffer.  Returns (beta, d, launches)."""
        t = self.t
        N, P = X.shape
        _bx, tX = self.put(X, x_offset)
        _by, ty = self.put(y)
        _bm, tm = self.put(m0)
        _bp, tp = self.put(P0)
        beta = t.zeros(chains, samp, P, dtype=t.float64, device=self.dev)
        d = t.zeros(chains, samp, dtype=t.float64, device=self.dev)
        before = self.L.bl_kernel_launches()
        self.check(self.L.bl_nb_multichain_dev(beta.data_ptr(), d.data_ptr(), ty, tX, d0, tm, tp, chains, N, P, samp,
                                               burn, seed, dmode, self.st))
        t.cuda.synchronize()
        return beta.cpu().numpy(), d.cpu().numpy(), self.L.bl_kernel_launches() - before

    def nb_df(self, X, y, m0, P0, samp, burn, seed, d0, x_offset):
        """bl_nb_gibbs_df_dev with X x_offset doubles into its buffer.  Returns (beta, d, launches)."""
        t = self.t
        N, P = X.shape
        _bx, tX = self.put(X, x_offset)
        _by, ty = self.put(y)
        _bm, tm = self.put(m0)
        _bp, tp = self.put(P0)
        beta = t.zeros(samp, P, dtype=t.float64, device=self.dev)
        d = t.zeros(samp, dtype=t.float64, device=self.dev)
        before = self.L.bl_kernel_launches()
        self.check(self.L.bl_nb_gibbs_df_dev(None, beta.data_ptr(), d.data_ptr(), ty, tX, d0, tm, tp, N, P, samp,
                                             burn, seed, 0, self.st))
        t.cuda.synchronize()
        return beta.cpu().numpy(), d.cpu().numpy(), self.L.bl_kernel_launches() - before


@pytest.mark.parametrize("N,P", [(4001, 16), (6007, 32)])
def test_nb_multichain_unaligned_x(engine, N, P):
    """X at a pointer 8 bytes into its buffer: the scalar kernels (k_xbeta with a chain dimension, k_xtv_partial)
    replace the MMA ones, with the same number of launches.  Chain c equals bl_nb_gibbs_df_dev(seed + c) at the same
    pointer bit for bit; it is within 1e-9 of the aligned call but not equal to it (other summation order), which
    shows that the scalar path ran."""
    d = Dev()
    X, y, m0, P0 = synth_nb(N, P, 70 + P)
    samp, burn, seed, chains = 4, 2, 61, 3
    bu, du, lu = d.multichain(X, y, m0, P0, samp, burn, seed, chains, 1.0, 1, x_offset=1)
    ba, da, la = d.multichain(X, y, m0, P0, samp, burn, seed, chains, 1.0, 1, x_offset=0)
    assert lu == la, (lu, la)
    for c in range(chains):
        b1, d1, l1 = d.nb_df(X, y, m0, P0, samp, burn, seed + c, 1.0, x_offset=1)
        assert np.array_equal(bu[c], b1), (c, float(np.abs(bu[c] - b1).max()))
        assert np.array_equal(du[c], d1)
        assert np.array_equal(du[c], da[c])
        close(bu[c], ba[c], 1e-9)
    assert not np.array_equal(bu, ba)


@pytest.mark.parametrize("dmode", DMODES)
def test_nb_multichain_matches_oracle(gapi, dmode):
    """Chain c against the CPU oracle's chain with seed + c: beta within 1e-7, d equal step by step (integer walk) or
    within 1e-12 (real walk); chains of different seeds differ."""
    N, P, chains, samp, burn = 2000, 5, 3, 6, 3
    X, y, m0, P0 = synth_nb(N, P, 6)
    d0 = D0[dmode]
    b, d = gapi.nb_multichain(y, X, m0, P0, samp, burn, 900, chains, d0=d0, dmode=dmode)
    for c in range(chains):
        if dmode == "fixed":
            _, bo = loader.nb_gibbs(y, X, d0, m0, P0, samp + burn, seed=900 + c)
            close(b[c], bo[burn:], 1e-7)
            assert np.all(d[c] == d0)
        else:
            _, bo, do = loader.nb_gibbs_df(y, X, m0, P0, samp, burn, seed=900 + c, d0=d0, real_d=dmode == "real")
            close(b[c], bo, 1e-7)
            if dmode == "int":
                assert np.array_equal(d[c], do)
            else:
                close(d[c], do, 1e-12)
    for c in range(1, chains):
        assert not np.allclose(b[0], b[c])


def test_nb_multichain_at_size(gapi):
    """N = 1 000 000, P = 64, 8 chains, integer walk: chains 0 and 7 equal the single-chain calls bit for bit."""
    N, P, chains = 1_000_000, 64, 8
    X, y, m0, P0 = synth_nb(N, P, 31)
    b, d = gapi.nb_multichain(y, X, m0, P0, 2, 1, 55, chains, d0=1.0, dmode="int")
    for c in (0, chains - 1):
        _, r, rd = gapi.nb_gibbs_df(y, X, m0, P0, 2, 1, 55 + c, d0=1.0)
        assert np.array_equal(b[c], r), (c, float(np.abs(b[c] - r).max()))
        assert np.array_equal(d[c], rd)
    assert not np.allclose(b[0], b[chains - 1])


@pytest.mark.parametrize("dmode", DMODES)
@pytest.mark.parametrize("shape", [(2000, 5), (40_000, 16), (6000, 128)], ids=lambda s: "N%d-P%d" % s)
def test_nb_multichain_launches_do_not_depend_on_chains(gapi, shape, dmode):
    """One launch per kernel per iteration for all chains: K = 9 launches as many kernels as K = 1.  (This holds up to
    chains * N = 2^23 draws; past that the binned sampler issues one more set-up / loop pair per 2^23 draws of the
    batch, as it does for any batch of that size.)"""
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    X, y, m0, P0 = data(shape)
    assert 9 * shape[0] <= 1 << 23
    counts = []
    for chains in (1, 9):
        before = L.bl_kernel_launches()
        gapi.nb_multichain(y, X, m0, P0, 2, 1, 5, chains, d0=D0[dmode], dmode=dmode)
        counts.append(L.bl_kernel_launches() - before)
    assert counts[0] == counts[1] and counts[0] > 0, counts


@pytest.mark.parametrize("dmode", DMODES)
def test_nb_multichain_dev_entry_equals_host_entry(gapi, dmode):
    """bl_nb_multichain_dev on torch device tensors gives the host entry's chains bit for bit."""
    N, P, chains, samp, burn = 5003, 16, 5, 3, 2
    X, y, m0, P0 = synth_nb(N, P, 77)
    code = {"fixed": 0, "int": 1, "real": 2}[dmode]
    b, d = gapi.nb_multichain(y, X, m0, P0, samp, burn, 13, chains, d0=D0[dmode], dmode=dmode)
    bd, dd, _ = Dev().multichain(X, y, m0, P0, samp, burn, 13, chains, D0[dmode], code, x_offset=0)
    assert np.array_equal(bd, b) and np.array_equal(dd, d)


def test_nb_multichain_refusals(gapi):
    """Each refusal carries its own message and launches nothing."""
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    N, P = 1 << 12, 4
    X, y, m0, P0 = synth_nb(N, P, 3)
    X257, y257, m0257, P0257 = synth_nb(300, 257, 4)

    def call(Xc, yc, m0c, P0c, chains=2, samp=2, burn=1, d0=1.0, dmode=1):
        Nc, Pc = Xc.shape
        beta = np.zeros((max(chains, 1), max(samp, 1), Pc))
        d = np.zeros((max(chains, 1), max(samp, 1)))
        _lib.check(L.bl_nb_multichain(beta.ctypes.data, d.ctypes.data, yc.ctypes.data, Xc.ctypes.data, d0,
                                      m0c.ctypes.data, P0c.ctypes.data, chains, Nc, Pc, samp, burn, 1, dmode))

    small = (X, y, m0, P0)
    cases = [
        (small, dict(chains=0), "chains must be at least 1"),
        (small, dict(samp=0), "bad dimensions"),
        (small, dict(burn=-1), "bad dimensions"),
        (small, dict(chains=1 << 19), r"2\^31"),
        ((X257, y257, m0257, P0257), dict(), "P > 256"),
        (small, dict(dmode=3), "unknown dmode"),
        (small, dict(dmode=1, d0=1.5), r"d0 must be a positive integer"),
        (small, dict(dmode=1, d0=0.0), r"d0 must be a positive integer"),
        (small, dict(dmode=2, d0=0.0), r"d0 must be positive\)"),
        (small, dict(dmode=0, d0=-1.0), r"d0 must be positive\)"),
    ]
    for args, kw, text in cases:
        before = L.bl_kernel_launches()
        with pytest.raises(_lib.EngineError, match=text):
            call(*args, **kw)
        assert L.bl_kernel_launches() == before, kw
    # N = 0
    before = L.bl_kernel_launches()
    with pytest.raises(_lib.EngineError, match="bad dimensions"):
        call(X[:0], y[:0], m0, P0)
    assert L.bl_kernel_launches() == before
    with pytest.raises(ValueError, match="dmode"):
        gapi.nb_multichain(y, X, m0, P0, 2, 1, 1, 2, dmode="integer")
