"""CPU tests that PIN the oracle.

1. The plain-C port (oracle/pg_oracle.c) reproduces the golden vectors that
   tests/golden/make_golden.py generated from the reference's own sources
   (oracle/_ref): identical variate consumption (= identical accept/reject
   decisions) and identical draws -- bit for bit under several threads, and on
   tapes cut short so that rows run dry.
2. The reference's own acceptance criterion (Code/C/test_pgomp.cpp:55-62): sample
   moments against pg_m1/pg_m2 -- and against the closed forms of BASELINE.md.
"""
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(__file__), "golden", "pg_golden.npz")


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(GOLD))


def same(a, b, rel=1e-14):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape
    nan = np.isnan(a)
    assert np.array_equal(nan, np.isnan(b))
    np.testing.assert_allclose(a[~nan], b[~nan], rtol=rel, atol=0)


def tape_of(g, p):
    return {k: g[f"{p}_t{k}"] for k in "ueng" if f"{p}_t{k}" in g}


def test_port_matches_golden_tapes(port, gold):
    g = gold
    x, tr = port.rpg_devroye(g["dev_n"], g["dev_z"], tape=tape_of(g, "dev"), trace=True)
    assert np.array_equal(tr, g["dev_trace"]); same(x, g["dev_x"])
    x, tr = port.rpg_alt(g["alt_h"], g["alt_z"], tape=tape_of(g, "alt"), trace=True)
    assert np.array_equal(tr, g["alt_trace"]); same(x, g["alt_x"])
    x, tr, it = port.rpg_sp(g["sp_h"], g["sp_z"], tape=tape_of(g, "sp"), trace=True)
    assert np.array_equal(tr, g["sp_trace"]); assert np.array_equal(it, g["sp_iter"]); same(x, g["sp_x"])
    x, tr = port.rpg_gamma(g["gam_h"], g["gam_z"], trunc=64, tape=tape_of(g, "gam"), trace=True)
    assert np.array_equal(tr, g["gam_trace"]); same(x, g["gam_x"])
    x, tr = port.rpg_hybrid(g["hyb_h"], g["hyb_z"], tape=tape_of(g, "hyb"), trace=True)
    assert np.array_equal(tr, g["hyb_trace"]); same(x, g["hyb_x"])


def test_port_matches_golden_philox(port, gold):
    g = gold
    same(port.rpg_devroye(g["pdev_n"], g["pdev_z"], seed=20240001, obs0=7, call_id=3), g["pdev_x"])
    same(port.rpg_alt(g["palt_h"], g["palt_z"], seed=20240002, obs0=1 << 33), g["palt_x"])
    x, it = port.rpg_sp(g["psp_h"], g["psp_z"], seed=20240003)
    same(x, g["psp_x"]); assert np.array_equal(it, g["psp_iter"])
    same(port.rpg_gamma(g["pgam_h"], g["pgam_z"], trunc=200, seed=20240004), g["pgam_x"])
    same(port.rpg_hybrid(g["phyb_h"], g["phyb_z"], seed=20240005, call_id=9), g["phyb_x"], rel=1e-9)


def test_port_helpers_match_golden(port, gold):
    g = gold
    same([port.pg_m1(b, z) for b, z in zip(g["mom_b"], g["mom_z"])], g["mom_m1"])
    same([port.pg_m2(b, z) for b, z in zip(g["mom_b"], g["mom_z"])], g["mom_m2"])
    same([port.v_eval(y) for y in g["vev_y"]], g["vev_v"])


# tape case -> (port method, shape array, extra arguments)
TAPE_CASES = {"dev": ("rpg_devroye", "dev_n", {}), "alt": ("rpg_alt", "alt_h", {}), "sp": ("rpg_sp", "sp_h", {}),
              "gam": ("rpg_gamma", "gam_h", {"trunc": 64}), "hyb": ("rpg_hybrid", "hyb_h", {})}


def test_port_equals_reference_bitwise(port, gold):
    """The port against the reference's own draws stored in the golden file, bit for bit under 1, 2 and 3
    threads: Philox streams and tapes in every regime, and tapes that run dry."""
    g = gold
    for nt in (1, 2, 3):
        assert np.array_equal(port.rpg_devroye(g["pdev_n"], g["pdev_z"], seed=20240001, obs0=7, call_id=3,
                                               nthreads=nt), g["pdev_x"])
        assert np.array_equal(port.rpg_alt(g["palt_h"], g["palt_z"], seed=20240002, obs0=1 << 33, nthreads=nt),
                              g["palt_x"])
        x, it = port.rpg_sp(g["psp_h"], g["psp_z"], seed=20240003, nthreads=nt)
        assert np.array_equal(x, g["psp_x"]) and np.array_equal(it, g["psp_iter"])
        assert np.array_equal(port.rpg_gamma(g["pgam_h"], g["pgam_z"], trunc=200, seed=20240004, nthreads=nt),
                              g["pgam_x"])
        assert np.array_equal(port.rpg_hybrid(g["phyb_h"], g["phyb_z"], seed=20240005, call_id=9, nthreads=nt),
                              g["phyb_x"])
        for p, (fn, shape, kw) in TAPE_CASES.items():
            out = getattr(port, fn)(g[shape], g[p + "_z"], tape=tape_of(g, p), trace=True, nthreads=nt, **kw)
            assert np.array_equal(out[0], g[p + "_x"]) and np.array_equal(out[1], g[p + "_trace"]), (p, nt)
    # Tapes that run dry: each stream's tape cut to the median count the reference consumed from it.  Up to
    # the first read past the cut a row runs as it did in the reference, so a row runs dry exactly when the
    # reference consumed more of some stream than the cut leaves; it then reports NaN and the exhausted flag,
    # and every other row the reference's draw and trace.
    for p in ("dev", "alt", "sp", "hyb"):
        fn, shape, kw = TAPE_CASES[p]
        used, tape = g[p + "_trace"], tape_of(g, p)
        cut = {k: max(1, int(np.median(used[:, "ueng".index(k)]))) for k in tape}
        dry = np.any([used[:, "ueng".index(k)] > w for k, w in cut.items()], axis=0)
        assert 0 < dry.sum() < len(dry)
        short = {k: np.ascontiguousarray(tape[k][:, :w]) for k, w in cut.items()}
        for nt in (1, 3):
            out = getattr(port, fn)(g[shape], g[p + "_z"], tape=short, trace=True, nthreads=nt, **kw)
            x, tr = out[0], out[1]
            assert np.array_equal(tr[:, 4] == 1, dry) and np.array_equal(np.isnan(x), dry), (p, nt)
            assert np.array_equal(x[~dry], g[p + "_x"][~dry]) and np.array_equal(tr[~dry], used[~dry]), (p, nt)
            if p == "sp":
                assert np.array_equal(out[2][~dry], g["sp_iter"][~dry])


@pytest.mark.parametrize("b,zs", [(1, (0.0, 0.7, 4.0, 25.0)), (3, (0.0, 2.0)), (2.5, (0.3, 5.0)),
                                  (9.0, (1.0,)), (40.0, (0.0, 3.0)), (150.0, (6.0,)), (0.4, (1.5,)),
                                  (300.0, (2.0,))])
def test_moments(oracle, b, zs):
    """Tier-2 criterion on the oracle itself: mean/variance within 5 sigma of
    E = b/(2z) tanh(z/2), Var = b/(4 z^3) (sinh z - z) sech^2(z/2)."""
    n = 4000 if b < 1 else 40000
    for z in zs:
        h = np.full(n, float(b))
        x = oracle.rpg_hybrid(h, np.full(n, z), seed=int(1000 * b + 10 * z), nthreads=4) if b != 3 else \
            oracle.rpg_devroye(np.full(n, 3, dtype=np.int32), np.full(n, z), seed=3, nthreads=4)
        if z == 0:
            m, v = b / 4.0, b / 24.0
        else:
            m = b / (2 * z) * np.tanh(z / 2)
            v = b / (4 * z ** 3) * (np.sinh(z) - z) / np.cosh(z / 2) ** 2
        assert m == pytest.approx(oracle.pg_m1(b, z), rel=1e-12)
        assert v == pytest.approx(oracle.pg_m2(b, z) - oracle.pg_m1(b, z) ** 2, rel=1e-6)
        assert abs(x.mean() - m) < 5 * np.sqrt(v / n)
        # variance of the sample variance ~ (mu4 - v^2)/n; PG kurtosis is modest: bound mu4 <= 12 v^2
        assert abs(x.var() - v) < 5 * np.sqrt(11 * v * v / n) + (0.02 * v if b < 1 else 0)
