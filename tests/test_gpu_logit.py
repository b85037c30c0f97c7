"""The binary / binomial logit model against the CPU oracle (oracle/gibbs_oracle.c) on the paths the other files leave
unchecked: row-sharded sweeps, EM at every kernel choice, and the multichain / batched-chains device entries.

test_gpu_multi.py compares the sharded logit chain with the single-GPU chain only, at P = 16, 7 and 15, with m0 = 0;
test_gpu_multichain.py compares the multichain entry with the batched entry through the host entries, which copy X to
aligned memory.  A wrong kernel on any of these paths gives a wrong posterior without an error, and a comparison of
two outputs of the same wrong kernel stays green.  Here every path meets the plain-loop fp64 oracle:

  * sharded sweeps on 2, 3 and 8 virtual ranks (bl_vcomm_*) at shapes that reach each producer of the exchanged
    sums -- the one-pass k_logit_sweep publishing its own sums at every column-box count, the two-pass
    k_gram_reduce (packed, unpacked, several tiles), shards above 2^18 rows, shards smaller than one 32-row tile --
    and each consumer: the lean and the constrained draws in shared memory, the constrained draw at P > 64 and the
    global-scratch k_beta_draw<false> at P = 128, all waiting on peers;
  * EM (the C `EM` symbol) against pgb_logit_em: the same iteration count and beta, at P from 1 to 256, which
    reaches odd-P k_xbeta / k_xtv_partial, the packed P = 32 Gram, k_xtv_mma, one and several Gram tiles, and
    k_em_solve in static, opt-in and global memory; both branches of the conditional-mean weights; max_iter = 0
    and a rank-deficient X;
  * bl_logit_multichain_dev and bl_logit_chains_dev with X 8 bytes into its buffer (the two-kernel path:
    k_xbeta_chains with chain stride 0, k_xtv_partial, the Gram's 8-byte loads), and with chains * N >= 2^20,
    where the unfused draw goes through the class-binned, chain-keyed k_devroye_refill<true>.

Data and priors are those of test_gpu_gibbs.py: X with an intercept column, m0 = linspace(-0.1, 0.1, P) (so
b0 = P0 m0 is not zero), P0 = 0.5 I + 0.01 (dense), N >= ~20 P wherever the constrained draw runs.  Tolerance
CHAIN_REL = 1e-8 on beta and omega, as there.
"""
import ctypes as C
import threading

import numpy as np
import pytest

from oracle import loader

pytestmark = pytest.mark.gpu

CHAIN_REL = 1e-8
PLAIN_BETA = 1           # BL_GIBBS_PLAIN_BETA
UNFUSED = 4              # BL_GIBBS_UNFUSED
ONE_PASS = 8             # BL_GIBBS_ONE_PASS
TWO_PASS = 16            # BL_GIBBS_TWO_PASS


@pytest.fixture(scope="module")
def gapi(engine):
    from bayeslogit_b200 import gibbs_api
    return gibbs_api


def synth_logit(N, P, seed, binomial=False):
    """As test_gpu_gibbs.py: standard normal covariates, an intercept, n_i in {1..5} if binomial."""
    rng = np.random.default_rng(seed)
    X = np.c_[rng.standard_normal((N, P - 1)), np.ones(N)]
    bt = np.r_[np.abs(rng.normal(0, 0.4, P - 1)), -0.5]
    p = 1 / (1 + np.exp(-X @ bt))
    if binomial:
        n = rng.integers(1, 6, N).astype(float)
        y = rng.binomial(n.astype(int), p) / n
    else:
        n = np.ones(N)
        y = (rng.random(N) < p).astype(float)
    return X, y, n


def prior(P):
    return np.linspace(-0.1, 0.1, P), 0.5 * np.eye(P) + 0.01


def close(a, b, rel=CHAIN_REL):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape
    err = np.abs(a - b) / np.maximum(np.abs(b), 1e-300)
    assert np.all(np.isfinite(a)) and err.max() <= rel, float(err.max())


# ---------------------------------------------------------------------------------------------------------------
# A. Row-sharded sweeps on virtual ranks
# ---------------------------------------------------------------------------------------------------------------
# ((N, P, binomial), flag variants): each case reaches a different producer or consumer of the exchanged sums.  Every
# variant runs with both beta draws.  Without a flag the sweep takes the one-pass kernel for even P <= 64 on shards of
# at most 2^18 rows.
SHARD_CASES = [
    ((40_003, 2, False), (0,)),                # one-pass, one column box
    ((30_011, 6, True), (0,)),                 # one-pass, ragged last tile, PG(n) as sums of PG(1)
    ((50_000, 32, True), (0, TWO_PASS)),       # one-pass at P = 32; the packed Gram published by k_gram_reduce
    ((20_011, 34, False), (0, TWO_PASS)),      # one-pass; k_xtv_mma set-up sum, unpacked Gram
    ((24_001, 64, False), (0, TWO_PASS)),      # 4096 sums from the one-pass epilogue; the same from k_gram_reduce
    ((12_001, 70, False), (0,)),               # fused two-pass, several Gram tiles, constrained draw at P > 64
    ((12_001, 128, False), (0,)),              # k_beta_draw<false> (global scratch), both draws
    ((9_001, 7, False), (0,)),                 # unfused draw, odd P^2 count
    ((1_100, 1, False), (0,)),                 # P = 1: one sum, odd count
]
# world = 2 only: each shard has more than 2^18 rows -- the default two-pass sweep, and the one-pass kernel forced
# on a full grid
SHARD_BIG = ((600_011, 16, False), (0, ONE_PASS))
# world = 8 only, plain draw: 25 rows per shard, less than one 32-row tile and fewer rows than CTAs
SHARD_TINY = (200, 6, False)
SHARD_SEED = 4243

_shard_data, _shard_oracle, _shard_single = {}, {}, {}


def shard_samp_burn(shape):
    return (3, 2) if shape[0] > 100_000 else (5, 3)


def shard_data(shape):
    if shape not in _shard_data:
        N, P, binomial = shape
        _shard_data[shape] = synth_logit(N, P, 600 + P + N % 97, binomial)
    return _shard_data[shape]


def shard_oracle(shape, constrained):
    """The oracle's chain on all rows; it does not depend on the number of ranks."""
    key = (shape, constrained)
    if key not in _shard_oracle:
        X, y, n = shard_data(shape)
        m0, P0 = prior(shape[1])
        samp, burn = shard_samp_burn(shape)
        _shard_oracle[key] = loader.logit_gibbs(y, X, n, m0, P0, samp, burn, seed=SHARD_SEED, constrained=constrained)
    return _shard_oracle[key]


def shard_runs(world):
    """[(shape, flags)] every rank runs at this world size; flags include the beta draw."""
    runs = []
    cases = SHARD_CASES + ([SHARD_BIG] if world == 2 else [])
    for shape, variants in cases:
        for f in variants:
            runs += [(shape, f), (shape, f | PLAIN_BETA)]
    if world == 8:
        runs.append((SHARD_TINY, PLAIN_BETA))
    return runs


class _Runner:
    """bl_logit_gibbs_dev on rows [lo, hi) of a data set, device pointers, one given stream."""

    def __init__(self, L, check, torch, dev, stream):
        self.L, self.check, self.torch, self.dev, self.st = L, check, torch, dev, stream

    def _up(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(self.dev)

    def logit(self, shape, flags, lo, hi):
        t = self.torch
        X, y, n = shard_data(shape)
        m0, P0 = prior(shape[1])
        samp, burn = shard_samp_burn(shape)
        P = X.shape[1]
        with t.cuda.stream(self.st):
            Xd, yd, nd = self._up(X[lo:hi]), self._up(y[lo:hi]), self._up(n[lo:hi])
            m0d, P0d = self._up(m0), self._up(np.asfortranarray(P0).ravel(order="F"))
            beta = t.zeros(samp, P, device=self.dev, dtype=t.float64)
            w = t.zeros(samp, hi - lo, device=self.dev, dtype=t.float64)
        self.st.synchronize()
        rc = self.L.bl_logit_gibbs_dev(w.data_ptr(), beta.data_ptr(), yd.data_ptr(), Xd.data_ptr(), nd.data_ptr(),
                                       m0d.data_ptr(), P0d.data_ptr(), hi - lo, P, samp, burn, SHARD_SEED, flags, lo,
                                       self.st.cuda_stream)
        if rc:
            self.check(rc)
        self.st.synchronize()
        return beta.cpu().numpy(), w.cpu().numpy()


def rel(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


@pytest.mark.parametrize("world", [2, 3, 8])
def test_logit_sharded_matches_oracle(engine, world):
    """On every rank: beta bit-identical to rank 0's, within 1e-8 of the oracle and of the single-GPU chain with the
    same flags; the rank's omega rows within 1e-8 of the oracle's rows [lo, hi)."""
    import torch
    from bayeslogit_b200 import _lib, dist as bdist
    L = _lib.lib()
    dev = torch.device("cuda", 0)
    st = torch.cuda.Stream(device=dev)
    run = _Runner(L, _lib.check, torch, dev, st)
    runs = shard_runs(world)
    if world == 2:
        assert bdist.shard_range(1, 2, SHARD_BIG[0][0])[0] > 1 << 18
    if world == 8:
        assert all(np.diff(bdist.shard_range(r, 8, SHARD_TINY[0])) < 32 for r in range(8))
    # single-GPU chains: no communicator bound
    for key in runs:
        if key not in _shard_single:
            _shard_single[key] = run.logit(key[0], key[1], 0, key[0][0])

    _lib.check(L.bl_vcomm_create(world))
    results, errors = [None] * world, []

    def rank_main(r):
        try:
            _lib.check(L.bl_vcomm_bind(r))
            out = {}
            for shape, flags in runs:
                lo, hi = bdist.shard_range(r, world, shape[0])
                out[(shape, flags)] = (lo, hi) + run.logit(shape, flags, lo, hi)
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
            t.join(timeout=900)
        assert not errors, errors
        assert all(r is not None for r in results)
    finally:
        L.bl_vcomm_destroy()

    bad = []
    for key in runs:
        shape, flags = key
        wo, bo = shard_oracle(shape, constrained=not flags & PLAIN_BETA)
        fb = _shard_single[key][0]
        for r in range(world):
            lo, hi, b, w = results[r][key]
            if not np.array_equal(b, results[0][key][2]):
                bad.append((shape, flags, r, "beta differs between ranks"))
            errs = (rel(b, bo), rel(w, wo[:, lo:hi]), rel(b, fb))
            if not (np.all(np.isfinite(b)) and np.all(np.isfinite(w)) and max(errs) <= CHAIN_REL):
                bad.append((shape, flags, r, "beta / omega vs oracle, beta vs single GPU", errs))
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------
# B. EM against the oracle at every kernel choice
# ---------------------------------------------------------------------------------------------------------------
# The C symbol is called directly: logit_EM merges duplicate rows first, which at P = 1 (the intercept alone) turns
# every row into one.
def engine_em(y, X, n, tol, max_iter, beta=None):
    """`EM` on host arrays.  Returns (beta, iterations)."""
    from bayeslogit_b200 import _lib
    X = np.ascontiguousarray(X, dtype=np.float64)
    N, P = X.shape
    y, n = np.ascontiguousarray(y, dtype=np.float64), np.ascontiguousarray(n, dtype=np.float64)
    beta = np.zeros(P) if beta is None else beta
    it = C.c_int(max_iter)
    _lib.lib().EM(beta.ctypes.data, y.ctypes.data, X.ctypes.data, n.ctypes.data, C.byref(C.c_int(N)),
                  C.byref(C.c_int(P)), C.byref(C.c_double(tol)), C.byref(it))
    _lib.check()
    return beta, it.value


def synth_em(N, P, seed):
    """Binomial counts n_i in {0..5} (rows with n_i = 0 carry no weight), covariates scaled by 1/sqrt(P - 1)."""
    rng = np.random.default_rng(seed)
    X = np.c_[rng.standard_normal((N, P - 1)) / np.sqrt(max(P - 1, 1)), np.ones(N)]
    b = np.r_[rng.normal(0, 1.0, P - 1), -0.3]
    n = rng.integers(0, 6, N).astype(float)
    y = rng.binomial(n.astype(int), 1 / (1 + np.exp(-X @ b))) / np.maximum(n, 1)
    assert (n == 0).any()
    return X, y, n


# (P, N): each reaches a different kernel choice of the EM loop
EM_SHAPES = [
    (1, 5_000),          # one covariate (the intercept), no row merge
    (2, 3_000),          # smallest even P
    (7, 20_000),         # k_xbeta, k_xtv_partial, the Gram's 8-byte loads
    (32, 20_011),        # packed Gram
    (34, 20_011),        # k_xtv_mma, unpacked Gram
    (64, 40_000),        # one full Gram tile
    (70, 30_000),        # two Gram tiles, k_em_solve in < 48 KB of shared memory
    (128, 40_000),       # k_em_solve in opt-in shared memory
    (200, 60_000),       # k_em_solve from global memory: (P|1) P + P doubles exceed 200 KB from P = 160
    (256, 80_000),       # ... at the largest P
    (64, 1_000_000),     # multi-wave grids
]
# (tol, max_iter): converged at two tolerances, and cut by max_iter (tol = 0 is never met)
EM_STOPS = [(1e-6, 100), (1e-10, 200), (0.0, 4)]


def em_compare(y, X, n, tol, max_iter):
    b, it = engine_em(y, X, n, tol, max_iter)
    bo, ito = loader.logit_em(y, X, n, tol=tol, max_iter=max_iter)
    assert it == ito, (tol, max_iter, it, ito)
    assert np.allclose(b, bo, rtol=1e-9, atol=1e-12), float(np.max(np.abs(b - bo)))
    return b, it


@pytest.mark.parametrize("P,N", EM_SHAPES, ids=lambda v: str(v))
def test_em_matches_oracle(engine, P, N):
    X, y, n = synth_em(N, P, 70 + P + N % 1000)
    its = [em_compare(y, X, n, tol, max_iter)[1] for tol, max_iter in EM_STOPS]
    assert 1 < its[0] < its[1] < EM_STOPS[1][1] and its[2] == EM_STOPS[2][1], its


def tilt_data(b, seed, N=20_000):
    """y the exact success probabilities at b (so the mode is b), X uniform on [-1, 1] with an intercept."""
    rng = np.random.default_rng(seed)
    P = len(b)
    X = np.c_[rng.uniform(-1, 1, (N, P - 1)), np.ones(N)]
    n = rng.integers(0, 6, N).astype(float)
    y = 1 / (1 + np.exp(-X @ b))
    return X, y, n


@pytest.mark.parametrize("tilt", ["series", "straddle"])
def test_em_weight_branches(engine, tilt):
    """k_em_weights takes a series for |psi / 2| < 0.01 and tanh(h) / h above.  "series": every |psi / 2| stays
    below 0.01 in every iteration; "straddle": psi / 2 falls on both sides of +-0.01 at the mode.  With y the exact
    probabilities at b the mode is b itself, a check that does not lean on the oracle."""
    b = np.array([0.005, -0.004, 0.003, 0.002]) if tilt == "series" else np.array([0.03, -0.02, 0.025, 0.01])
    X, y, n = tilt_data(b, 5 if tilt == "series" else 6)
    out = {stop: em_compare(y, X, n, *stop) for stop in EM_STOPS}
    bt, it = out[EM_STOPS[1]]
    assert np.allclose(bt, b, rtol=0, atol=1e-12), float(np.max(np.abs(bt - b)))
    h = np.abs(X @ b) / 2
    if tilt == "series":
        for k in range(1, it + 1):              # the k-th weights are formed from the (k-1)-th iterate
            bk, _ = loader.logit_em(y, X, n, tol=0.0, max_iter=k - 1)
            assert np.max(np.abs(X @ bk)) / 2 < 0.01, k
        assert h.max() < 0.01
    else:
        assert (h < 0.01).mean() > 0.1 and (h >= 0.01).mean() > 0.1


def test_em_max_iter_zero(engine):
    X, y, n = synth_em(3000, 5, 9)
    beta = np.full(5, 7.0)
    b, it = engine_em(y, X, n, 1e-8, 0, beta=beta)
    assert it == 0 and np.array_equal(b, np.zeros(5))
    assert loader.logit_em(y, X, n, tol=1e-8, max_iter=0)[1] == 0


@pytest.mark.parametrize("col", [0, 3])
def test_em_rank_deficient(engine, col):
    """An all-zero covariate column: X' Omega X is singular.  The engine reports it and leaves the caller's beta and
    max_iter as they were; the oracle returns -1.  A good call afterwards still matches the oracle."""
    from bayeslogit_b200 import _lib
    X, y, n = synth_em(4000, 6, 11)
    Xz = X.copy()
    Xz[:, col] = 0.0
    beta = np.full(6, 7.0)
    it = C.c_int(50)
    with pytest.raises(_lib.EngineError, match="EM: X' Omega X is not positive definite"):
        _lib.lib().EM(beta.ctypes.data, y.ctypes.data, np.ascontiguousarray(Xz).ctypes.data, n.ctypes.data,
                      C.byref(C.c_int(4000)), C.byref(C.c_int(6)), C.byref(C.c_double(1e-8)), C.byref(it))
        _lib.check()
    assert np.array_equal(beta, np.full(6, 7.0)) and it.value == 50
    with pytest.raises(RuntimeError, match="not positive definite"):
        loader.logit_em(y, Xz, n, tol=1e-8, max_iter=50)
    em_compare(y, X, n, 1e-8, 50)


# ---------------------------------------------------------------------------------------------------------------
# C. The multichain and batched-chains device entries
# ---------------------------------------------------------------------------------------------------------------
class Dev:
    """Device-resident inputs; X may start `x_offset` doubles into its buffer."""

    def __init__(self):
        import torch
        from bayeslogit_b200 import _lib
        self.t, self.L, self.check = torch, _lib.lib(), _lib.check
        self.dev = torch.device("cuda")

    def put(self, a, offset=0):
        t = self.t
        a = np.ascontiguousarray(a, dtype=np.float64).ravel()
        buf = t.zeros(a.size + offset, dtype=t.float64, device=self.dev)
        buf[offset:] = t.from_numpy(a).to(self.dev)
        ptr = buf.data_ptr() + 8 * offset
        assert ptr % 16 == (8 if offset % 2 else 0)
        return buf, ptr

    def zeros(self, *shape):
        return self.t.zeros(*shape, dtype=self.t.float64, device=self.dev)

    def stream(self):
        return self.t.cuda.current_stream().cuda_stream

    def _inputs(self, X, y, n, m0, P0, x_offset):
        return [self.put(X, x_offset), self.put(y), self.put(n), self.put(m0),
                self.put(np.asfortranarray(P0).ravel(order="F"))]

    def _run(self, fn, out, *args):
        self.t.cuda.synchronize()
        before = self.L.bl_kernel_launches()
        self.check(fn(*args, self.stream()))
        self.t.cuda.synchronize()
        return out.cpu().numpy(), self.L.bl_kernel_launches() - before

    def logit(self, X, y, n, m0, P0, samp, burn, seed, flags, x_offset):
        """bl_logit_gibbs_dev.  Returns (beta, launches)."""
        N, P = X.shape
        keep = self._inputs(X, y, n, m0, P0, x_offset)
        tX, ty, tn, tm, tp = (k[1] for k in keep)
        beta = self.zeros(samp, P)
        return self._run(self.L.bl_logit_gibbs_dev, beta, None, beta.data_ptr(), ty, tX, tn, tm, tp, N, P, samp,
                         burn, seed, flags | 2, 0)

    def multichain(self, X, y, n, m0, P0, samp, burn, seed, chains, flags, x_offset):
        """bl_logit_multichain_dev on one copy of the rows.  Returns (beta [chains x samp x P], launches)."""
        N, P = X.shape
        keep = self._inputs(X, y, n, m0, P0, x_offset)
        tX, ty, tn, tm, tp = (k[1] for k in keep)
        beta = self.zeros(chains, samp, P)
        return self._run(self.L.bl_logit_multichain_dev, beta, beta.data_ptr(), ty, tX, tn, tm, tp, chains, N, P,
                         samp, burn, seed, flags)

    def chains(self, X, y, n, m0, P0, samp, burn, seed, chains, flags, x_offset):
        """bl_logit_chains_dev on `chains` copies of the rows, the copies side by side starting x_offset doubles
        into the buffer.  Returns (beta [chains x samp x P], launches)."""
        N, P = X.shape
        keep = self._inputs(np.broadcast_to(X, (chains, N, P)), np.tile(y, chains), np.tile(n, chains), m0, P0,
                            x_offset)
        tX, ty, tn, tm, tp = (k[1] for k in keep)
        beta = self.zeros(chains, samp, P)
        return self._run(self.L.bl_logit_chains_dev, beta, beta.data_ptr(), ty, tX, tn, tm, tp, chains, N, P, samp,
                         burn, seed, flags)


@pytest.mark.parametrize("constrained", [False, True])
@pytest.mark.parametrize("N,P,chains", [(900, 5, 3), (2101, 32, 3), (2115, 70, 2)])
def test_device_entries_equal_host_entries(gapi, N, P, chains, constrained):
    """X at offset 0: the device entries take the kernels the host entries take, so the same bits."""
    X, y, n = synth_logit(N, P, 3000 + N + P, binomial=True)
    m0, P0 = prior(P)
    samp, burn, seed = 4, 2, 811
    flags = 0 if constrained else PLAIN_BETA
    d = Dev()
    bm, _ = d.multichain(X, y, n, m0, P0, samp, burn, seed, chains, flags, 0)
    bc, _ = d.chains(X, y, n, m0, P0, samp, burn, seed, chains, flags, 0)
    hm = gapi.logit_multichain(y, X, n, m0, P0, samp, burn, seed=seed, chains=chains, flags=flags)
    hc = gapi.logit_chains(np.stack([y] * chains), np.stack([X] * chains), np.stack([n] * chains), m0, P0, samp,
                           burn, seed=seed, flags=flags)
    assert np.array_equal(bm, hm) and np.array_equal(bc, hc)
    assert np.array_equal(bm, bc)


@pytest.mark.parametrize("constrained", [False, True])
@pytest.mark.parametrize("N,P,chains", [(3001, 32, 3), (4099, 64, 5), (2115, 70, 2)])
def test_unaligned_multichain_matches_oracle(engine, N, P, chains, constrained):
    """X 8 bytes into its buffer: the two-kernel path (k_xbeta_chains with chain stride 0, the refill draw,
    k_xtv_partial, the Gram's 8-byte loads).  Chain c equals chain c of bl_logit_chains_dev on `chains` copies at the
    same offset bit for bit, and is within 1e-8 of the oracle and of bl_logit_gibbs_dev with seed + c at that
    offset.  Unfused costs one more launch per iteration (the omega draw apart from psi) and one psi pass ahead of
    each of the two phases."""
    X, y, n = synth_logit(N, P, 4000 + N + P, binomial=True)
    m0, P0 = prior(P)
    samp, burn, seed = 5, 3, 907
    flags = 0 if constrained else PLAIN_BETA
    d = Dev()
    bm, lm = d.multichain(X, y, n, m0, P0, samp, burn, seed, chains, flags, 1)
    _, la = d.multichain(X, y, n, m0, P0, samp, burn, seed, chains, flags, 0)
    assert lm - la == burn + samp + 2, (lm, la)
    bc, _ = d.chains(X, y, n, m0, P0, samp, burn, seed, chains, flags, 1)
    for c in range(chains):
        assert np.array_equal(bm[c], bc[c]), (c, float(np.abs(bm[c] - bc[c]).max()))
        _, bo = loader.logit_gibbs(y, X, n, m0, P0, samp, burn, seed=seed + c, constrained=constrained)
        close(bm[c], bo)
        b1, _ = d.logit(X, y, n, m0, P0, samp, burn, seed + c, flags, 1)
        close(bm[c], b1)
    assert not np.allclose(bm[0], bm[1])


@pytest.mark.parametrize("constrained", [False, True])
@pytest.mark.parametrize("x_offset", [0, 1])
def test_binned_chain_keyed_draw(engine, x_offset, constrained):
    """chains * N >= 2^20 with BL_GIBBS_UNFUSED: the draw bins the (chain, row) pairs by branch class and
    k_devroye_refill<true> keys each pair's stream by its chain (position % N), not by its place in the list.  Two more
    launches per iteration than the fused draw (the class scatter and the xbeta pass), one xbeta per phase."""
    N, P, chains = 300_007, 16, 4
    assert chains * N >= 1 << 20
    X, y, n = synth_logit(N, P, 5000, binomial=True)
    m0, P0 = prior(P)
    samp, burn, seed = 3, 2, 913
    flags = (0 if constrained else PLAIN_BETA) | UNFUSED
    d = Dev()
    bm, lm = d.multichain(X, y, n, m0, P0, samp, burn, seed, chains, flags, x_offset)
    _, lf = d.multichain(X, y, n, m0, P0, samp, burn, seed, chains, flags & ~UNFUSED, 0)
    assert lm - lf == 2 * (burn + samp) + 2, (lm, lf)
    bc, _ = d.chains(X, y, n, m0, P0, samp, burn, seed, chains, flags, x_offset)
    assert np.array_equal(bm, bc), float(np.abs(bm - bc).max())
    for c in range(chains):
        _, bo = loader.logit_gibbs(y, X, n, m0, P0, samp, burn, seed=seed + c, constrained=constrained)
        close(bm[c], bo)
