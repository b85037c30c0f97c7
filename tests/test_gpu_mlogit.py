"""The multinomial logit sweep against the CPU oracle at every kernel choice, on sharded rows and on device pointers
that are 8-byte but not 16-byte aligned.

The multichain tests compare chain c with the single-chain sweep bit for bit; that shows nothing if the single
chain is wrong.  Here the single chain meets the plain-loop fp64 oracle (oracle/gibbs_oracle.c) with the same seed
at shapes that reach each kernel choice of the sweep, with binomial counts n_i in {1..5} as well as n_i = 1:
  * odd P: k_xbeta + k_mlogit_offsets, k_xtv_partial, the Gram from 8-byte loads;
  * P = 64: one unpacked Gram tile and k_xtv_stream; P = 34: k_xtv_mma; P = 70: several Gram tiles;
  * P = 96, 128: the beta draw out of global scratch;
  * J - 1 = 16 (the most categories the fused psi pass keeps in registers) and 17 (separate kernels);
  * J = 2, where the next category is the category just drawn (offset c = 0);
  * >= 2^18 rows, where the psi pass builds the next draw's class-ordered index list.
Tolerance CHAIN_REL = 1e-8 on beta and omega, as in test_gpu_gibbs.py.  N is kept >= ~20 P there too.
"""
import os
import threading

import numpy as np
import pytest

from oracle import loader

pytestmark = pytest.mark.gpu

CHAIN_REL = 1e-8
NO_W = 2                 # BL_GIBBS_NO_W
PLAIN_BETA = 1           # BL_GIBBS_PLAIN_BETA
TWO_PASS = 16            # BL_GIBBS_TWO_PASS


@pytest.fixture(scope="module")
def gapi(engine):
    from bayeslogit_b200 import gibbs_api
    return gibbs_api


def synth_mlogit(N, P, J, seed, counts=False, scale=0.4):
    """X with an intercept column; counts: n ~ U{1..5} and y = multinomial(n, p)[:, :J-1] / n, else n = 1."""
    rng = np.random.default_rng(seed)
    X = np.c_[rng.standard_normal((N, P - 1)) / np.sqrt(max(P - 1, 1)), np.ones(N)]
    B = rng.normal(0, scale, (P, J - 1))
    eta = np.c_[X @ B, np.zeros(N)]
    pr = np.exp(eta)
    pr /= pr.sum(1, keepdims=True)
    if counts:
        n = rng.integers(1, 6, N)
        Y = rng.multinomial(n, pr)[:, :J - 1] / n[:, None]
        n = n.astype(float)
    else:
        cat = (pr.cumsum(1) < rng.random(N)[:, None]).sum(1)
        Y = np.eye(J)[np.minimum(cat, J - 1)][:, :J - 1]
        n = np.ones(N)
    m0 = rng.normal(0, 0.05, (P, J - 1))
    P0 = np.stack([(0.5 + 0.05 * j) * np.eye(P) for j in range(J - 1)], axis=2)
    return X, Y, n, m0, P0


def close(a, b, rel=CHAIN_REL):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape
    err = np.abs(a - b) / np.maximum(np.abs(b), 1e-300)
    assert np.all(np.isfinite(a)) and err.max() <= rel, float(err.max())


# (N, P, J, counts): each reaches a different choice of kernels
CASES = [
    (3001, 7, 3, False),       # odd P: k_xbeta, k_mlogit_offsets, k_xtv_partial, Gram from 8-byte loads
    (1100, 1, 3, False),       # P = 1
    (1200, 2, 3, True),        # P = 2
    (4001, 16, 2, True),       # J = 2: the next category is the same one, c = 0
    (4099, 64, 5, False),      # one Gram tile, not packed: k_xtv_stream
    (5003, 34, 3, False),      # even P not a power of two: k_xtv_mma
    (2115, 70, 3, False),      # several Gram tiles, cost-proportional slabs, P > 64 mvn draw
    (3000, 96, 3, False),      # beta draw out of global scratch
    (4000, 128, 3, False),     # ... with 2 x 2 Gram tiles
    (1500, 4, 17, False),      # U = 16: the largest U of the fused psi pass
    (1500, 4, 18, False),      # U = 17: separate psi and offsets kernels
    (300_007, 32, 4, False),   # >= 2^18 rows: the psi pass builds the next draw's class-ordered index list
    (20_011, 32, 10, True),    # packed Gram with X'(Omega c) from the same pass; PG(n) as sums of PG(1)
]
SEED = 2029


def case_id(c):
    return "N%d-P%d-J%d" % c[:3] + ("-counts" if c[3] else "")


def samp_burn(case):
    return (4, 2) if case[0] * case[1] <= 200_000 else (3, 2)


_data = {}


def data(case):
    if case not in _data:
        N, P, J, counts = case
        _data[case] = synth_mlogit(N, P, J, 300 + N + 7 * P + J, counts=counts)
    return _data[case]


_runs = {}


def run_single(gapi, case, unfused=False, keep_w=True):
    """bl_mlogit_gibbs on the case's data; unfused: under BL_MLOGIT_UNFUSED=1.  Cached."""
    key = (case, unfused, keep_w)
    if key not in _runs:
        X, Y, n, m0, P0 = data(case)
        samp, burn = samp_burn(case)
        if unfused:
            os.environ["BL_MLOGIT_UNFUSED"] = "1"
        try:
            _runs[key] = gapi.mlogit_gibbs(Y, X, n, m0, P0, samp, burn, seed=SEED, keep_w=keep_w)
        finally:
            os.environ.pop("BL_MLOGIT_UNFUSED", None)
    return _runs[key]


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_mlogit_chain_matches_oracle(gapi, case):
    X, Y, n, m0, P0 = data(case)
    N, P, J, _ = case
    samp, burn = samp_burn(case)
    w, b = run_single(gapi, case)
    wo, bo = loader.mlogit_gibbs(Y, X, n, m0, P0, samp, burn, seed=SEED)
    assert b.shape == (samp, J - 1, P) and w.shape == (samp, J - 1, N)
    close(b, bo)
    close(w, wo)
    if J == 2:
        assert np.all(np.isfinite(w)) and np.all(w > 0)


FUSED_CASES = [c for c in CASES if c[1] % 2 == 0 and c[2] - 1 <= 16]


@pytest.mark.parametrize("case", FUSED_CASES, ids=case_id)
def test_mlogit_fused_equals_unfused(gapi, case):
    """k_xbeta_mma<true> (psi_j, exp(psi_j), the next category's offset and tilt, at >= 2^18 rows the next draw's
    index list, from one pass over X) against the psi kernel + k_mlogit_offsets per category: the same bits.
    Dropping omega (keep_w=False) leaves beta unchanged."""
    w1, b1 = run_single(gapi, case)
    w2, b2 = run_single(gapi, case, unfused=True)
    assert np.array_equal(b1, b2), float(np.abs(b1 - b2).max())
    assert np.array_equal(w1, w2), float(np.abs(w1 - w2).max())
    w3, b3 = run_single(gapi, case, keep_w=False)
    assert w3 is None and np.array_equal(b3, b1)


# ---------------------------------------------------------------------------------------------------------------
# Device pointers that are 8-byte but not 16-byte aligned.  The kernels that read X 16 bytes at a time are chosen
# at dispatch by an alignment test; a caller of the _dev entries may pass a pointer into the middle of a buffer,
# and then the fallback kernels run: k_xbeta / k_xbeta_chains, k_mlogit_offsets per category, k_xtv_partial, the
# Gram's 8-byte loads, the unfused logit draw.  They sum in other orders, so the chain is the aligned chain to
# rounding; the multichain entry's chain c is the single chain at the same pointer bit for bit.
# ---------------------------------------------------------------------------------------------------------------
class Dev:
    def __init__(self):
        import torch
        from bayeslogit_b200 import _lib
        self.torch, self.L, self.check = torch, _lib.lib(), _lib.check
        self.dev = torch.device("cuda")

    def put(self, a, offset=0):
        """a (C order, float64) on the device, starting `offset` doubles into a buffer of a.size + offset.
        Returns (buffer, pointer)."""
        t = self.torch
        a = np.ascontiguousarray(a, dtype=np.float64).ravel()
        buf = t.zeros(a.size + offset, dtype=t.float64, device=self.dev)
        buf[offset:] = t.from_numpy(a).to(self.dev)
        ptr = buf.data_ptr() + 8 * offset
        assert ptr % 16 == (8 if offset % 2 else 0)
        return buf, ptr

    def zeros(self, *shape):
        t = self.torch
        return t.zeros(*shape, dtype=t.float64, device=self.dev)

    def stream(self):
        return self.torch.cuda.current_stream().cuda_stream

    def launches(self):
        return self.L.bl_kernel_launches()

    def mlogit(self, X, Y, n, m0, P0, samp, burn, seed, x_offset, keep_w=True):
        """bl_mlogit_gibbs_dev with X starting x_offset doubles into its buffer.  Returns (w, beta, launches)."""
        N, P = X.shape
        U = Y.shape[1]
        _bx, tX = self.put(X, x_offset)
        _by, ty = self.put(Y)
        _bn, tn = self.put(n)
        _bm, tm0 = self.put(np.asfortranarray(m0).ravel(order="F"))
        _bp, tP0 = self.put(np.asfortranarray(P0).ravel(order="F"))
        beta = self.zeros(samp, U, P)
        w = self.zeros(samp, U, N) if keep_w else None
        self.torch.cuda.synchronize()
        before = self.launches()
        self.check(self.L.bl_mlogit_gibbs_dev(w.data_ptr() if keep_w else None, beta.data_ptr(), ty, tX, tn, tm0, tP0,
                                              N, P, U + 1, samp, burn, seed, 0 if keep_w else NO_W, 0, self.stream()))
        self.torch.cuda.synchronize()
        launches = self.launches() - before
        return (w.cpu().numpy() if keep_w else None), beta.cpu().numpy(), launches

    def mlogit_multichain(self, X, Y, n, m0, P0, samp, burn, seed, chains, x_offset):
        N, P = X.shape
        U = Y.shape[1]
        _bx, tX = self.put(X, x_offset)
        _by, ty = self.put(Y)
        _bn, tn = self.put(n)
        _bm, tm0 = self.put(np.asfortranarray(m0).ravel(order="F"))
        _bp, tP0 = self.put(np.asfortranarray(P0).ravel(order="F"))
        beta = self.zeros(chains, samp, U, P)
        self.torch.cuda.synchronize()
        before = self.launches()
        self.check(self.L.bl_mlogit_multichain_dev(beta.data_ptr(), ty, tX, tn, tm0, tP0, chains, N, P, U + 1, samp, burn,
                                                   seed, 0, self.stream()))
        self.torch.cuda.synchronize()
        return beta.cpu().numpy(), self.launches() - before

    def logit(self, X, y, n, m0, P0, samp, burn, seed, flags, x_offset):
        N, P = X.shape
        _bx, tX = self.put(X, x_offset)
        _by, ty = self.put(y)
        _bn, tn = self.put(n)
        _bm, tm0 = self.put(m0)
        _bp, tP0 = self.put(np.asfortranarray(P0).ravel(order="F"))
        beta = self.zeros(samp, P)
        w = self.zeros(samp, N)
        self.torch.cuda.synchronize()
        before = self.launches()
        self.check(self.L.bl_logit_gibbs_dev(w.data_ptr(), beta.data_ptr(), ty, tX, tn, tm0, tP0, N, P, samp, burn, seed,
                                             flags, 0, self.stream()))
        self.torch.cuda.synchronize()
        return w.cpu().numpy(), beta.cpu().numpy(), self.launches() - before


@pytest.mark.parametrize("N,P,J", [(3001, 16, 4), (6007, 32, 5), (4099, 64, 3)], ids=lambda v: str(v))
def test_unaligned_device_pointers_mlogit(engine, N, P, J):
    d = Dev()
    X, Y, n, m0, P0 = synth_mlogit(N, P, J, 50 + P)
    samp, burn, seed, chains = 4, 2, 61, 3
    U = J - 1
    wa, ba, la = d.mlogit(X, Y, n, m0, P0, samp, burn, seed, x_offset=0)
    wu, bu, lu = d.mlogit(X, Y, n, m0, P0, samp, burn, seed, x_offset=1)
    wo, bo = loader.mlogit_gibbs(Y, X, n, m0, P0, samp, burn, seed=seed)
    close(bu, bo); close(wu, wo)
    close(bu, ba, 1e-9); close(wu, wa, 1e-9)
    # the fallback ran: k_mlogit_offsets on every category update instead of only the first, and no fill of the
    # cached exponentials (which only the fused pass keeps)
    assert lu - la == (burn + samp) * U - 2, (lu, la)
    # the multichain entry at the same unaligned pointer: chain c is the single chain with seed + c, bit for bit
    bm, lm = d.mlogit_multichain(X, Y, n, m0, P0, samp, burn, seed, chains, x_offset=1)
    bma, lma = d.mlogit_multichain(X, Y, n, m0, P0, samp, burn, seed, chains, x_offset=0)
    assert lm - lma == (burn + samp) * U - 2, (lm, lma)
    for c in range(chains):
        _, b1, _ = d.mlogit(X, Y, n, m0, P0, samp, burn, seed + c, x_offset=1, keep_w=False)
        assert np.array_equal(bm[c], b1), (c, float(np.abs(bm[c] - b1).max()))
        if c == 0:
            assert np.array_equal(b1, bu)
        else:
            _, bo_c = loader.mlogit_gibbs(Y, X, n, m0, P0, samp, burn, seed=seed + c)
            close(bm[c], bo_c)
        close(bm[c], bma[c], 1e-9)


def synth_logit(N, P, seed):
    rng = np.random.default_rng(seed)
    X = np.c_[rng.standard_normal((N, P - 1)), np.ones(N)]
    bt = np.r_[np.abs(rng.normal(0, 0.4, P - 1)), -0.5]
    y = (rng.random(N) < 1 / (1 + np.exp(-X @ bt))).astype(float)
    return X, y, np.ones(N)


@pytest.mark.parametrize("constrained", [False, True])
@pytest.mark.parametrize("N,P", [(3001, 32), (4099, 64)])
def test_unaligned_device_pointers_logit(engine, constrained, N, P):
    """The aligned call runs the two-pass sweep (the one-pass kernel needs 16-byte alignment too); unaligned, psi and
    omega come from k_xbeta + the refill kernel instead of the fused k_logit_psi_draw: one more launch per iteration
    and one psi pass ahead of each of the two phases."""
    d = Dev()
    X, y, n = synth_logit(N, P, 70 + P)
    m0 = np.linspace(-0.1, 0.1, P)
    P0 = 0.5 * np.eye(P) + 0.01
    samp, burn, seed = 5, 3, 19
    f = 0 if constrained else PLAIN_BETA
    wa, ba, la = d.logit(X, y, n, m0, P0, samp, burn, seed, f | TWO_PASS, x_offset=0)
    wu, bu, lu = d.logit(X, y, n, m0, P0, samp, burn, seed, f, x_offset=1)
    wo, bo = loader.logit_gibbs(y, X, n, m0, P0, samp, burn, seed=seed, constrained=constrained)
    close(bu, bo); close(wu, wo)
    close(bu, ba, 1e-9); close(wu, wa, 1e-9)
    assert lu - la == burn + samp + 2, (lu, la)


# ---------------------------------------------------------------------------------------------------------------
# Row-sharded mlogit and real-valued-dispersion NB on virtual ranks (bl_vcomm_*): W ranks in this process on one GPU,
# one host thread each, all enqueueing into one stream, meeting at a host barrier between the producing and the
# consuming kernel of every exchange.  The exchange kernels are those of the multi-GPU sweep: each category's X'kappa
# set-up through the small all-reduce, 2 (J - 1) exchanges per iteration, at P = 32 X'(Omega c_j) published from the
# packed Gram's partial tile with the P^2 sums, and on a shard of >= 2^18 rows the draw from the class-ordered index
# list with obs0 != 0.
# ---------------------------------------------------------------------------------------------------------------
def _make_nb(N, P, seed):
    rng = np.random.default_rng(seed)
    X = np.c_[rng.standard_normal((N, P - 1)), np.ones(N)]
    bt = np.r_[np.abs(rng.normal(0, 0.3, P - 1)), -0.5]
    yc = rng.poisson(np.exp(np.clip(X @ bt * 0.3 + 2.0, None, 4.0))).astype(float)
    return X, yc


class _Runner:
    """The sharded sweeps on rows [lo, hi) of a data set, device pointers, one given stream."""

    def __init__(self, L, check, torch, dev, stream):
        self.L, self.check, self.torch, self.dev, self.st = L, check, torch, dev, stream

    def _up(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(self.dev)

    def mlogit(self, X, Y, n, m0, P0, lo, hi, samp, burn, seed):
        t, P, U = self.torch, X.shape[1], Y.shape[1]
        with t.cuda.stream(self.st):
            Xd, yd, nd = self._up(X[lo:hi]), self._up(Y[lo:hi]), self._up(n[lo:hi])
            m0d = self._up(np.asfortranarray(m0).ravel(order="F"))
            P0d = self._up(np.asfortranarray(P0).ravel(order="F"))
            beta = t.zeros(samp, U, P, device=self.dev, dtype=t.float64)
            w = t.zeros(samp, U, hi - lo, device=self.dev, dtype=t.float64)
        self.st.synchronize()
        rc = self.L.bl_mlogit_gibbs_dev(w.data_ptr(), beta.data_ptr(), yd.data_ptr(), Xd.data_ptr(), nd.data_ptr(),
                                        m0d.data_ptr(), P0d.data_ptr(), hi - lo, P, U + 1, samp, burn, seed, 0, lo,
                                        self.st.cuda_stream)
        if rc:
            self.check(rc)
        self.st.synchronize()
        return beta.cpu().numpy(), w.cpu().numpy()

    def nb_dfreal(self, X, yc, lo, hi, samp=8, burn=4):
        t, P = self.torch, X.shape[1]
        with t.cuda.stream(self.st):
            Xd, yd = self._up(X[lo:hi]), self._up(yc[lo:hi])
            m0 = t.zeros(P, device=self.dev, dtype=t.float64)
            P0 = (0.1 * t.eye(P, device=self.dev, dtype=t.float64)).contiguous()
            beta = t.zeros(samp, P, device=self.dev, dtype=t.float64)
            dd = t.zeros(samp, device=self.dev, dtype=t.float64)
        self.st.synchronize()
        rc = self.L.bl_nb_gibbs_dfreal_dev(None, beta.data_ptr(), dd.data_ptr(), yd.data_ptr(), Xd.data_ptr(), 2.5,
                                           m0.data_ptr(), P0.data_ptr(), hi - lo, P, samp, burn, 4713, lo,
                                           self.st.cuda_stream)
        if rc:
            self.check(rc)
        self.st.synchronize()
        return beta.cpu().numpy(), dd.cpu().numpy()


SHARD_CASES = [
    (40_003, 16, 4),      # vectorised slot copy
    (9_001, 7, 3),        # odd P: odd P^2 count
    (30_011, 32, 5),      # packed Gram, X'(Omega c_j) in the partial tile
    (12_001, 70, 3),      # several Gram tiles
]
SHARD_BIG = (600_011, 32, 3)     # world = 2: each shard has >= 2^18 rows, the second starts at obs0 != 0
SHARD_ORACLE = (30_011, 32, 5)   # compared with the oracle at world = 3
SHARD_SAMP, SHARD_BURN, SHARD_SEED = 3, 2, 808

_shard_data = {}
_shard_full = {}


def shard_data(case):
    if case not in _shard_data:
        N, P, J = case
        _shard_data[case] = synth_mlogit(N, P, J, 500 + N + P + J, counts=(P == 7))
    return _shard_data[case]


def rel(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


@pytest.mark.parametrize("world", [2, 3, 8])
def test_mlogit_sharded_on_virtual_ranks(engine, world):
    import torch
    from bayeslogit_b200 import _lib, dist as bdist
    L = _lib.lib()
    dev = torch.device("cuda", 0)
    st = torch.cuda.Stream(device=dev)
    run = _Runner(L, _lib.check, torch, dev, st)
    cases = SHARD_CASES + ([SHARD_BIG] if world == 2 else [])
    if world == 2:
        assert bdist.shard_range(1, 2, SHARD_BIG[0])[0] >= 1 << 18
    nb_data = _make_nb(40_003, 16, 26)
    # single-GPU chains: no communicator bound
    for c in cases:
        if c not in _shard_full:
            X, Y, n, m0, P0 = shard_data(c)
            _shard_full[c] = run.mlogit(X, Y, n, m0, P0, 0, c[0], SHARD_SAMP, SHARD_BURN, SHARD_SEED)
    if "nb" not in _shard_full:
        _shard_full["nb"] = run.nb_dfreal(nb_data[0], nb_data[1], 0, 40_003)
    nb_full = _shard_full["nb"]
    assert len(set(nb_full[1])) > 1 and np.any(nb_full[1] != np.floor(nb_full[1]))      # d moves, on the reals

    _lib.check(L.bl_vcomm_create(world))
    results, errors = [None] * world, []

    def rank_main(r):
        try:
            _lib.check(L.bl_vcomm_bind(r))
            out = {}
            for c in cases:
                X, Y, n, m0, P0 = shard_data(c)
                lo, hi = bdist.shard_range(r, world, c[0])
                out[c] = (lo, hi) + run.mlogit(X, Y, n, m0, P0, lo, hi, SHARD_SAMP, SHARD_BURN, SHARD_SEED)
            lo, hi = bdist.shard_range(r, world, 40_003)
            out["nb"] = run.nb_dfreal(nb_data[0], nb_data[1], lo, hi)
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

    for c in cases:
        fb, fw = _shard_full[c]
        for r in range(world):
            lo, hi, b, w = results[r][c]
            assert np.array_equal(b, results[0][c][2]), ("beta differs between ranks", c, r)
            assert rel(b, fb) < 1e-8 and rel(w, fw[..., lo:hi]) < 1e-8, (c, r, rel(b, fb), rel(w, fw[..., lo:hi]))
    if world == 3:
        X, Y, n, m0, P0 = shard_data(SHARD_ORACLE)
        _, bo = loader.mlogit_gibbs(Y, X, n, m0, P0, SHARD_SAMP, SHARD_BURN, seed=SHARD_SEED)
        close(results[0][SHARD_ORACLE][2], bo)
    for r in range(world):
        b, d = results[r]["nb"]
        assert np.array_equal(d, results[0]["nb"][1]), "dispersion chain differs between ranks"
        assert np.array_equal(b, results[0]["nb"][0]), "beta differs between ranks"
        close(d, nb_full[1], 1e-12)
        close(b, nb_full[0], 1e-8)
