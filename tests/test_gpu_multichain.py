"""Several logit chains on one shared data set (bl_logit_multichain): chain c must be, bit for bit, chain c of the
replicated batch (bl_logit_chains on `chains` copies of the rows, same seed), and therefore the single-chain sweep
with seed + c.

The bit equality rests on one property of the hardware: an m8n8k4 f64 MMA forms each element of its output tile
from that element's own row and column only.  The replicated batch puts one chain's beta in all 8 columns of the
B operand and reads column 0; the shared-rows kernel puts 8 chains' betas in the 8 columns.
"""
import numpy as np
import pytest

from oracle import loader

pytestmark = pytest.mark.gpu

CHAIN_REL = 1e-8

# (P = 128 exceeds the batch's one-CTA shared-memory beta draw; see test_multichain_refuses_what_the_batch_refuses)
SHAPES = [(900, 5), (2101, 32), (1777, 34), (4099, 64), (2115, 70), (1100, 1), (1200, 2)]
CHAINS = [1, 2, 3, 5, 8, 11]


@pytest.fixture(scope="module")
def gapi(engine):
    from bayeslogit_b200 import gibbs_api
    return gibbs_api


def synth_binomial(N, P, seed, zeros=True):
    """Binomial data, n_i in {1..5}; with zeros, about one row in twenty has n_i = 0."""
    rng = np.random.default_rng(seed)
    X = np.c_[rng.standard_normal((N, P - 1)), np.ones(N)]
    bt = np.r_[np.abs(rng.normal(0, 0.4, P - 1)), -0.5]
    p = 1 / (1 + np.exp(-X @ bt))
    n = rng.integers(1, 6, N).astype(float)
    y = rng.binomial(n.astype(int), p) / n
    if zeros:
        n[rng.random(N) < 0.05] = 0.0
    return X, y, n


def close(a, b, rel=CHAIN_REL):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape
    err = np.abs(a - b) / np.maximum(np.abs(b), 1e-300)
    assert np.all(np.isfinite(a)) and err.max() <= rel, float(err.max())


def prior(P):
    return np.linspace(-0.1, 0.1, P), 0.5 * np.eye(P) + 0.01


@pytest.mark.parametrize("unfused", [False, True])
@pytest.mark.parametrize("constrained", [False, True])
@pytest.mark.parametrize("chains", CHAINS)
@pytest.mark.parametrize("N,P", SHAPES)
def test_multichain_equals_replicated_chains(gapi, N, P, chains, constrained, unfused):
    """Odd P (and P = 1) and unaligned rows take the two-kernel path whatever the flag; N not a multiple of 32 leaves
    a ragged last trip; P > 64 has several Gram tiles; chains = 3, 5 leave padding columns, 11 a second group of 8."""
    X, y, n = synth_binomial(N, P, 1000 + N + P)
    m0, P0 = prior(P)
    flags = (0 if constrained else gapi.PLAIN_BETA) | (gapi.UNFUSED if unfused else 0)
    samp, burn = 4, 2
    b = gapi.logit_multichain(y, X, n, m0, P0, samp, burn, seed=321, chains=chains, flags=flags)
    assert b.shape == (chains, samp, P)
    r = gapi.logit_chains(np.stack([y] * chains), np.stack([X] * chains), np.stack([n] * chains), m0, P0,
                          samp, burn, seed=321, flags=flags)
    assert np.array_equal(b, r), float(np.abs(b - r).max())
    assert np.all(np.isfinite(b))


@pytest.mark.parametrize("constrained", [False, True])
@pytest.mark.parametrize("N,P,chains", [(900, 5, 3), (2101, 32, 5), (4099, 64, 2), (2115, 70, 11)])
def test_multichain_matches_oracle_and_single_chain(gapi, N, P, chains, constrained):
    """Chain c against the oracle's chain and the engine's single-chain entry with seed + c."""
    X, y, n = synth_binomial(N, P, 2000 + N + P, zeros=False)
    m0, P0 = prior(P)
    samp, burn = (6, 3) if P < 64 else (4, 2)
    flags = 0 if constrained else gapi.PLAIN_BETA
    b = gapi.logit_multichain(y, X, n, m0, P0, samp, burn, seed=700, chains=chains, flags=flags)
    for c in range(chains):
        _, bo = loader.logit_gibbs(y, X, n, m0, P0, samp, burn, seed=700 + c, constrained=constrained)
        close(b[c], bo)
        _, b1 = gapi.logit_gibbs(y, X, n, m0, P0, samp, burn, seed=700 + c, flags=flags, keep_w=False)
        close(b[c], b1)
    for c in range(1, chains):
        assert not np.allclose(b[0], b[c])             # same data, different streams: different chains


def test_multichain_at_size(gapi):
    """N = 1 000 000, P = 64, 4 chains, the reference's constrained draw: bit equality with the replicated call
    (which holds 4 copies of X, 2 GB)."""
    N, P, chains = 1_000_000, 64, 4
    rng = np.random.default_rng(11)
    X = np.c_[rng.standard_normal((N, P - 1)), np.ones(N)]
    bt = np.r_[np.abs(rng.normal(0, 0.25, P - 1)), -0.5]
    y = (rng.random(N) < 1 / (1 + np.exp(-X @ bt))).astype(float)
    n = np.ones(N)
    m0, P0 = np.zeros(P), 0.01 * np.eye(P)
    b = gapi.logit_multichain(y, X, n, m0, P0, 2, 1, seed=99, chains=chains, flags=0)
    Xr = np.broadcast_to(X, (chains, N, P))
    r = gapi.logit_chains(np.broadcast_to(y, (chains, N)), Xr, np.broadcast_to(n, (chains, N)), m0, P0, 2, 1,
                          seed=99, flags=0)
    assert np.array_equal(b, r), float(np.abs(b - r).max())
    assert not np.allclose(b[0], b[1])


@pytest.mark.parametrize("constrained", [False, True])
def test_multichain_refuses_what_the_batch_refuses(gapi, constrained):
    """N = 3000, P = 128: the batched chains draw each chain's beta in one CTA out of shared memory, which holds
    P <= 91 (constrained draw) or P <= 111 (plain draw).  Both entries refuse the shape with the same message."""
    from bayeslogit_b200 import _lib
    N, P, chains = 3000, 128, 2
    X, y, n = synth_binomial(N, P, 4000)
    m0, P0 = prior(P)
    flags = 0 if constrained else gapi.PLAIN_BETA
    with pytest.raises(_lib.EngineError, match="P too large for the shared-memory beta draw"):
        gapi.logit_multichain(y, X, n, m0, P0, 2, 1, seed=3, chains=chains, flags=flags)
    with pytest.raises(_lib.EngineError, match="P too large for the shared-memory beta draw"):
        gapi.logit_chains(np.stack([y] * chains), np.stack([X] * chains), np.stack([n] * chains), m0, P0, 2, 1,
                          seed=3, flags=flags)


def test_multichain_rejects_bad_sizes(gapi):
    """chains = 0 and chains * N >= 2^31 fail with a message before anything is launched."""
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    N, P = 1 << 12, 2
    X, y, n = synth_binomial(N, P, 5, zeros=False)
    m0, P0 = prior(P)
    for chains, text in [(0, "bad dimensions"), (1 << 19, "2^31")]:
        before = L.bl_kernel_launches()
        with pytest.raises(_lib.EngineError, match=text.replace("^", r"\^")):
            gapi.logit_multichain(y, X, n, m0, P0, 1, 0, seed=1, chains=chains)
        assert L.bl_kernel_launches() == before
