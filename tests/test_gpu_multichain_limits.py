"""The multichain entries that give the chain its own y or z grid dimension refuse more than 65535 chains before
anything is allocated or launched, even when chains * N stays below 2^31."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_nb_multichain_refuses_more_chains_than_a_grid_dimension(engine):
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    N, P, chains, samp = 16, 2, 65536, 1
    X = np.ones((N, P))
    y = np.arange(N, dtype=float)
    m0, P0 = np.zeros(P), np.eye(P)
    beta, d = np.zeros((chains, samp, P)), np.zeros((chains, samp))
    before = L.bl_kernel_launches()
    with pytest.raises(_lib.EngineError, match="chains must be at most 65535"):
        _lib.check(L.bl_nb_multichain(beta.ctypes.data, d.ctypes.data, y.ctypes.data, X.ctypes.data, 1.0,
                                      m0.ctypes.data, P0.ctypes.data, chains, N, P, samp, 0, 1, 1))
    assert L.bl_kernel_launches() == before


def test_mlogit_multichain_refuses_more_chains_than_a_grid_dimension(engine):
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    N, P, J, chains, samp = 16, 2, 3, 65536, 1
    X = np.ones((N, P))
    Y = np.zeros((N, J - 1))
    n = np.ones(N)
    m0, P0 = np.zeros((P, J - 1)), np.stack([np.eye(P)] * (J - 1), axis=2)
    beta = np.zeros((chains, samp, J - 1, P))
    before = L.bl_kernel_launches()
    with pytest.raises(_lib.EngineError, match="chains must be at most 65535"):
        _lib.check(L.bl_mlogit_multichain(beta.ctypes.data, Y.ctypes.data, X.ctypes.data, n.ctypes.data,
                                          m0.ctypes.data, P0.ctypes.data, chains, N, P, J, samp, 0, 1, 0))
    assert L.bl_kernel_launches() == before
