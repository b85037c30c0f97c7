#!/usr/bin/env python3
"""Generate tests/golden/pg_golden.npz from the REFERENCE ITSELF.

Runs the reference's own sampler sources, compiled unmodified and in place from
/root/reference/Code/C into oracle/_ref/libpg_ref.so (oracle/Makefile), on small
seeded inputs, and stores inputs, injected variate tapes and outputs.  The
reference ships no golden vectors of its own (SURVEY.md section 4), so these are the pin
for the plain-C port (tests/test_oracle_port.py) and for the CUDA engine
(tests/test_gpu_parity.py); they also travel to the GPU box, where
/root/reference does not exist.

    python tests/golden/make_golden.py        # needs /root/reference mounted
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import loader  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "pg_golden.npz")


def main():
    loader.build(("ref",))
    R = loader.Oracle("reference")
    rng = np.random.default_rng(20240001)
    out = {}

    def zmix(n):
        z = rng.uniform(-5, 5, n)
        z[: n // 8] = rng.uniform(-50, 50, n // 8)
        z[n // 8] = 0.0
        z[n // 8 + 1] = 1e-9
        z[n // 8 + 2] = 3.125       # Z = 1/0.64: the truncated-IG branch switch
        z[n // 8 + 3] = -3.1250001
        return z

    # ---- tape cases (tier 1) -------------------------------------------------
    n = 192
    z = zmix(n)
    shape = rng.integers(0, 5, n).astype(np.int32)
    tape = loader.make_tape(n, lu=40, le=40, ln=12, seed=1)
    x, tr = R.rpg_devroye(shape, z, tape=tape, trace=True)
    out.update(dev_n=shape, dev_z=z, dev_tu=tape["u"], dev_te=tape["e"], dev_tn=tape["n"],
               dev_x=x, dev_trace=tr)

    z = zmix(n)
    h = rng.uniform(1, 13, n)
    h[:16] = rng.integers(1, 14, 16)
    h[16:20] = [1.0, 4.0, 4.99, 5.0]
    tape = loader.make_tape(n, lu=64, le=64, ln=16, seed=2)
    x, tr = R.rpg_alt(h, z, tape=tape, trace=True)
    out.update(alt_h=h, alt_z=z, alt_tu=tape["u"], alt_te=tape["e"], alt_tn=tape["n"],
               alt_x=x, alt_trace=tr)

    z = zmix(n)
    h = rng.uniform(13, 170, n)
    h[:16] = rng.integers(14, 171, 16)
    h[16:19] = [1.0, 2.5, 170.0]
    tape = loader.make_tape(n, lu=32, le=32, ln=12, seed=3)
    x, tr, it = R.rpg_sp(h, z, tape=tape, trace=True)
    out.update(sp_h=h, sp_z=z, sp_tu=tape["u"], sp_te=tape["e"], sp_tn=tape["n"],
               sp_x=x, sp_trace=tr, sp_iter=it)

    m = 48
    z = zmix(m)
    h = rng.uniform(0.05, 3.0, m)
    h[0] = 0.0
    tape = loader.make_tape(m, lg=64, g_shape=np.where(h > 0, h, 1.0), seed=4)
    x, tr = R.rpg_gamma(h, z, trunc=64, tape=tape, trace=True)
    out.update(gam_h=h, gam_z=z, gam_tg=tape["g"], gam_x=x, gam_trace=tr)

    z = zmix(n)
    h = np.where(rng.random(n) < 0.5, rng.uniform(0.5, 200, n), rng.integers(1, 201, n).astype(float))
    h[:8] = [0.0, -1.0, 1.0, 2.0, 13.0, 13.5, 170.0, 170.5]
    h[8:16] = rng.uniform(0.05, 1.0, 8)
    tape = loader.make_tape(n, lu=96, le=96, ln=24, lg=200, g_shape=np.where((h > 0) & (h < 1), h, 1.0),
                            seed=5)
    x, tr = R.rpg_hybrid(h, z, tape=tape, trace=True)
    out.update(hyb_h=h, hyb_z=z, hyb_tu=tape["u"], hyb_te=tape["e"], hyb_tn=tape["n"],
               hyb_tg=tape["g"], hyb_x=x, hyb_trace=tr)

    # ---- Philox-stream cases (stream contract) ----------------------------------
    k = 2048
    z = zmix(k)
    shape = rng.integers(0, 4, k).astype(np.int32)
    out.update(pdev_n=shape, pdev_z=z, pdev_x=R.rpg_devroye(shape, z, seed=20240001, obs0=7, call_id=3))
    h = rng.uniform(1, 13, k)
    out.update(palt_h=h, palt_z=z, palt_x=R.rpg_alt(h, z, seed=20240002, obs0=1 << 33, call_id=0))
    h = rng.uniform(13, 170, k)
    xs, its = R.rpg_sp(h, z, seed=20240003)
    out.update(psp_h=h, psp_z=z, psp_x=xs, psp_iter=its)
    h = rng.uniform(0.05, 2.0, 256)
    out.update(pgam_h=h, pgam_z=z[:256], pgam_x=R.rpg_gamma(h, z[:256], trunc=200, seed=20240004))
    h = np.where(rng.random(k) < 0.5, rng.uniform(0.5, 200, k), rng.integers(1, 201, k).astype(float))
    out.update(phyb_h=h, phyb_z=z, phyb_x=R.rpg_hybrid(h, z, seed=20240005, call_id=9))

    # ---- deterministic helpers -----------------------------------------------------
    b = rng.uniform(0.5, 400, 256)
    zz = zmix(256)
    out.update(mom_b=b, mom_z=zz, mom_m1=np.array([R.pg_m1(*p) for p in zip(b, zz)]),
               mom_m2=np.array([R.pg_m2(*p) for p in zip(b, zz)]))
    y = np.concatenate([2.0 ** rng.uniform(-6, 6, 500), [0.0625, 1.0, 15.999, 0.05, 17.0, 0.999999, 1.000001]])
    out.update(vev_y=y, vev_v=np.array([R.v_eval(t) for t in y]))

    zero_unread_tape_entries(out)
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, os.path.getsize(OUT), "bytes;",
          "exhausted:", {k: int(v[:, 4].sum()) for k, v in out.items() if k.endswith("_trace")})


def zero_unread_tape_entries(out):
    """Zero every tape entry past the count of variates its observation consumed (trace columns
    u, e, n, g): a tape row is read from its start, one entry per variate, so these entries never
    reach a sampler and the draws do not change, while the file shrinks to a quarter of its size."""
    for key in [k for k in out if k.endswith("_trace")]:
        p, used = key[:-len("_trace")], out[key]
        for col, k in enumerate("ueng"):
            t = out.get(f"{p}_t{k}")
            if t is not None:
                t[np.arange(t.shape[1])[None, :] >= used[:, col:col + 1]] = 0.0


if __name__ == "__main__":
    main()
