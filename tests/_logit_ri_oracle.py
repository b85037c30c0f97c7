"""CPU restatement of the random-intercept logit chain (tests/ri_oracle/logit_ri_oracle.c), built on first use into
a temporary directory from that file and the oracle's sources (oracle/pg_oracle.c, oracle/l0.c, with
oracle/gibbs_oracle.c included), with the flags of oracle/Makefile."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE = os.path.join(os.path.dirname(HERE), "oracle")
_lib = None


def _build():
    cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
    out = tempfile.mkdtemp(prefix="logit_ri_oracle_")
    atexit.register(shutil.rmtree, out, True)
    so = os.path.join(out, "liblogit_ri_oracle.so")
    subprocess.run([cc, "-std=gnu11", "-O2", "-ffp-contract=off", "-fPIC", "-fopenmp", "-I", ORACLE,
                    os.path.join(HERE, "ri_oracle", "logit_ri_oracle.c"), os.path.join(ORACLE, "pg_oracle.c"),
                    os.path.join(ORACLE, "l0.c"), "-o", so, "-shared", "-Wl,-Bsymbolic", "-lm"], check=True)
    L = C.CDLL(so)
    vp, ci, cd = C.c_void_p, C.c_int, C.c_double
    L.pgb_logit_ri_gibbs.argtypes = [vp] * 7 + [ci, vp, vp, cd, cd, cd, ci, ci, ci, ci, C.c_uint64, ci]
    return L


def logit_ri(y, X, n, group, G, m0, P0, a0, b0, tau2_0, samp, burn, seed, nthreads=0):
    """Returns (beta [samp x P], u [samp x G], tau2 [samp]); arguments as gibbs_api.logit_ri."""
    global _lib
    if _lib is None:
        _lib = _build()
    X = np.ascontiguousarray(X, dtype=np.float64)
    N, P = X.shape
    f = lambda a: np.ascontiguousarray(a, dtype=np.float64).ravel()
    y, n, m0 = f(y), f(n), f(m0)
    group = np.ascontiguousarray(group, dtype=np.int32).ravel()
    P0c = np.asfortranarray(np.asarray(P0, dtype=np.float64))
    beta, u, tau2 = np.zeros((samp, P)), np.zeros((samp, G)), np.zeros(samp)
    st = _lib.pgb_logit_ri_gibbs(beta.ctypes.data, u.ctypes.data, tau2.ctypes.data, y.ctypes.data, X.ctypes.data,
                                 n.ctypes.data, group.ctypes.data, int(G), m0.ctypes.data, P0c.ctypes.data, float(a0),
                                 float(b0), float(tau2_0), N, P, int(samp), int(burn), int(seed), int(nthreads))
    if st:
        raise RuntimeError("oracle logit_ri_gibbs: precision not positive definite")
    return beta, u, tau2
