"""Several multinomial logit chains on one shared data set (bl_mlogit_multichain): chain c must be, bit for bit, the
single-chain sweep bl_mlogit_gibbs with seed + c and omega dropped; with BL_GIBBS_UNFUSED, the single chain run with
BL_MLOGIT_UNFUSED=1.

As for the logit multichain, the equality of the fused path rests on the m8n8k4 f64 MMA forming each element of its
output tile from that element's own row and column only: the single chain puts one beta_j in all 8 columns of the B
operand, the multichain kernel puts 8 chains' beta_j in the 8 columns.
"""
import os

import numpy as np
import pytest

from oracle import loader

pytestmark = pytest.mark.gpu

CHAIN_REL = 1e-8

# (N, P, J), each reaching a different choice of kernels
SHAPES = [
    (2500, 6, 4),        # fused psi pass, P <= 64 beta draw
    (3001, 7, 3),        # odd P: unfused psi (k_xbeta_chains)
    (20011, 32, 10),     # packed Gram with X'(Omega c) from the same pass
    (4099, 64, 5),       # one Gram tile, not packed: k_xtv_* with an X stride of 0
    (2115, 70, 3),       # several Gram tiles, P > 64 beta draw
    (3000, 96, 3),       # the single chain draws beta out of global memory, the multichain out of shared memory
    (1500, 4, 18),       # J - 1 = 17 > 16 categories: unfused
    (300_007, 32, 4),    # >= 2^18 rows: the psi pass bins the next draw's rows by class
]
CHAINS = [1, 2, 3, 8, 9]
SEED = 4242
SAMP, BURN = 3, 2


@pytest.fixture(scope="module")
def gapi(engine):
    from bayeslogit_b200 import gibbs_api
    return gibbs_api


def synth_mlogit(N, P, J, seed, scale=0.4):
    rng = np.random.default_rng(seed)
    X = np.c_[rng.standard_normal((N, P - 1)) / np.sqrt(max(P - 1, 1)), np.ones(N)]
    B = rng.normal(0, scale, (P, J - 1))
    eta = np.c_[X @ B, np.zeros(N)]
    pr = np.exp(eta)
    pr /= pr.sum(1, keepdims=True)
    cat = (pr.cumsum(1) < rng.random(N)[:, None]).sum(1)
    Y = np.eye(J)[np.minimum(cat, J - 1)][:, :J - 1]
    m0 = rng.normal(0, 0.05, (P, J - 1))
    P0 = np.stack([(0.5 + 0.05 * j) * np.eye(P) for j in range(J - 1)], axis=2)
    return X, Y, np.ones(N), m0, P0


def close(a, b, rel=CHAIN_REL):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape
    err = np.abs(a - b) / np.maximum(np.abs(b), 1e-300)
    assert np.all(np.isfinite(a)) and err.max() <= rel, float(err.max())


_data = {}
_single = {}


def data(shape):
    if shape not in _data:
        N, P, J = shape
        _data[shape] = synth_mlogit(N, P, J, 100 + N + P + J)
    return _data[shape]


def single_chain(gapi, shape, seed, unfused):
    """bl_mlogit_gibbs with omega dropped; unfused: under BL_MLOGIT_UNFUSED=1.  Cached across chain counts."""
    key = (shape, seed, unfused)
    if key not in _single:
        X, Y, n, m0, P0 = data(shape)
        if unfused:
            os.environ["BL_MLOGIT_UNFUSED"] = "1"
        try:
            _, b = gapi.mlogit_gibbs(Y, X, n, m0, P0, SAMP, BURN, seed=seed, keep_w=False)
        finally:
            os.environ.pop("BL_MLOGIT_UNFUSED", None)
        _single[key] = b
    return _single[key]


@pytest.mark.parametrize("unfused", [False, True])
@pytest.mark.parametrize("chains", CHAINS)
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "N%d-P%d-J%d" % s)
def test_mlogit_multichain_equals_single_chains(gapi, shape, chains, unfused):
    """chains = 3 leaves padding columns in the MMA tile, 9 needs a second group of 8."""
    X, Y, n, m0, P0 = data(shape)
    N, P, J = shape
    flags = gapi.UNFUSED if unfused else 0
    b = gapi.mlogit_multichain(Y, X, n, m0, P0, SAMP, BURN, seed=SEED, chains=chains, flags=flags)
    assert b.shape == (chains, SAMP, J - 1, P)
    assert np.all(np.isfinite(b))
    for c in range(chains):
        r = single_chain(gapi, shape, SEED + c, unfused)
        assert np.array_equal(b[c], r), (c, float(np.abs(b[c] - r).max()))


@pytest.mark.parametrize("N,P,J,chains", [(2500, 6, 4, 3), (6007, 32, 5, 9)])
def test_mlogit_multichain_matches_oracle(gapi, N, P, J, chains):
    """Chain c against the CPU oracle's chain with seed + c; chains of different seeds differ."""
    X, Y, n, m0, P0 = synth_mlogit(N, P, J, 7 + N)
    samp, burn = 4, 2
    b = gapi.mlogit_multichain(Y, X, n, m0, P0, samp, burn, seed=900, chains=chains)
    for c in range(chains):
        _, bo = loader.mlogit_gibbs(Y, X, n, m0, P0, samp, burn, seed=900 + c)
        close(b[c], bo)
    for c in range(1, chains):
        assert not np.allclose(b[0], b[c])


def test_mlogit_multichain_at_size(gapi):
    """N = 1 000 000, P = 32, J = 10, 8 chains: chains 0 and 7 equal the single-chain calls bit for bit."""
    N, P, J, chains = 1_000_000, 32, 10, 8
    X, Y, n, m0, P0 = synth_mlogit(N, P, J, 31, scale=0.25)
    b = gapi.mlogit_multichain(Y, X, n, m0, P0, 2, 1, seed=55, chains=chains)
    for c in (0, chains - 1):
        _, r = gapi.mlogit_gibbs(Y, X, n, m0, P0, 2, 1, seed=55 + c, keep_w=False)
        assert np.array_equal(b[c], r), (c, float(np.abs(b[c] - r).max()))
    assert not np.allclose(b[0], b[chains - 1])


@pytest.mark.parametrize("shape", [(2500, 6, 4), (3001, 7, 3), (300_007, 32, 4)], ids=lambda s: "N%d-P%d-J%d" % s)
def test_mlogit_multichain_launches_do_not_depend_on_chains(gapi, shape):
    """One launch per kernel per category update for all chains: a call at K = 9 launches as many kernels as at K = 1."""
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    X, Y, n, m0, P0 = data(shape)
    counts = []
    for chains in (1, 9):
        before = L.bl_kernel_launches()
        gapi.mlogit_multichain(Y, X, n, m0, P0, 2, 1, seed=5, chains=chains)
        counts.append(L.bl_kernel_launches() - before)
    assert counts[0] == counts[1] and counts[0] > 0, counts


def test_mlogit_multichain_dev_entry_equals_host_entry(gapi):
    """bl_mlogit_multichain_dev on torch device tensors gives the host entry's chains bit for bit."""
    import torch
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    N, P, J, chains, samp, burn = 5003, 16, 4, 5, 3, 2
    X, Y, n, m0, P0 = synth_mlogit(N, P, J, 77)
    b = gapi.mlogit_multichain(Y, X, n, m0, P0, samp, burn, seed=13, chains=chains)
    dev = torch.device("cuda")
    tX = torch.from_numpy(np.ascontiguousarray(X)).to(dev)                     # P x N column-major = N x P row-major
    ty = torch.from_numpy(np.ascontiguousarray(Y)).to(dev)                     # (J-1) x N column-major
    tn = torch.from_numpy(n).to(dev)
    tm0 = torch.from_numpy(np.asfortranarray(m0).ravel(order="F")).to(dev)
    tP0 = torch.from_numpy(np.asfortranarray(P0).ravel(order="F")).to(dev)
    beta = torch.zeros(chains, samp, J - 1, P, device=dev, dtype=torch.float64)
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(L.bl_mlogit_multichain_dev(beta.data_ptr(), ty.data_ptr(), tX.data_ptr(), tn.data_ptr(), tm0.data_ptr(),
                                          tP0.data_ptr(), chains, N, P, J, samp, burn, 13, 0, st))
    torch.cuda.synchronize()
    assert np.array_equal(beta.cpu().numpy(), b)


def test_mlogit_multichain_refusals(gapi):
    """Each refusal carries its message and launches nothing."""
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    N, P, J = 1 << 12, 4, 3
    X, Y, n, m0, P0 = synth_mlogit(N, P, J, 3)
    X112, Y112, n112, m0112, P0112 = synth_mlogit(300, 112, 3, 4)
    cases = [
        (dict(chains=0), "bad dimensions", (X, Y, n, m0, P0)),
        (dict(chains=1 << 19), r"2\^31", (X, Y, n, m0, P0)),
        (dict(chains=2), "P too large for the shared-memory beta draw", (X112, Y112, n112, m0112, P0112)),
        (dict(chains=2, flags=gapi.PLAIN_BETA), "flags", (X, Y, n, m0, P0)),
        (dict(chains=2, flags=64), "flags", (X, Y, n, m0, P0)),
    ]
    for kw, text, (Xc, Yc, nc, m0c, P0c) in cases:
        before = L.bl_kernel_launches()
        with pytest.raises(_lib.EngineError, match=text):
            gapi.mlogit_multichain(Yc, Xc, nc, m0c, P0c, 2, 1, seed=1, **kw)
        assert L.bl_kernel_launches() == before, kw
    # J = 1: no category to update
    before = L.bl_kernel_launches()
    beta = np.zeros((2, 2, 0, P))
    with pytest.raises(_lib.EngineError, match="bad dimensions"):
        _lib.check(L.bl_mlogit_multichain(beta.ctypes.data, Y[:, :0].ctypes.data, X.ctypes.data, n.ctypes.data,
                                          m0.ctypes.data, P0.ctypes.data, 2, N, P, 1, 2, 1, 1, 0))
    assert L.bl_kernel_launches() == before
