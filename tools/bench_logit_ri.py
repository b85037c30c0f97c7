#!/usr/bin/env python3
"""Cost of the random-intercept logit iteration (bl_logit_ri_gibbs_dev) beside the plain logit iteration
(bl_logit_gibbs_dev with BL_GIBBS_PLAIN_BETA | BL_GIBBS_NO_W) on the same data: N = 10^6 rows, P = 64, ids balanced
over G = 10^2, 10^4, 10^5 groups in random row order, and one skewed assignment (half the rows in one group, the rest
spread over 9 999 groups).  ms per iteration is the slope between a short and a long chain (set-up excluded), median
of --reps repeats (short and long chain alternating); the stage split is the CUDA-event timing of one iteration (BL_GIBBS_TIMING).  The card
name and power limit are read in the same run.

    python tools/bench_logit_ri.py [--short 10 --long 110 --reps 3 --out result.json]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N, P = 1_000_000, 64


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        return q
    except Exception as e:          # the timing stands without it, but say so
        return f"nvidia-smi unavailable: {e}"


def stage_lines(fn):
    """Run fn with BL_GIBBS_TIMING=1 and return the engine's timing lines (written to fd 2)."""
    os.environ["BL_GIBBS_TIMING"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["BL_GIBBS_TIMING"]
        f.seek(0)
        return [l.strip() for l in f if "timing, us]" in l]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--short", type=int, default=10)
    ap.add_argument("--long", type=int, default=110)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    dev = torch.device("cuda")
    st = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device=dev)
    g.manual_seed(20260101)
    X = torch.randn(N, P, generator=g, device=dev, dtype=torch.float64) / 8.0
    X[:, 0] = 1.0
    bt = torch.randn(P, generator=g, device=dev, dtype=torch.float64) * 0.5
    n = torch.ones(N, device=dev, dtype=torch.float64)
    m0 = torch.zeros(P, device=dev, dtype=torch.float64)
    P0 = (0.01 * torch.eye(P, device=dev, dtype=torch.float64)).contiguous()
    rng = np.random.default_rng(5)
    cases = {}
    for G in (100, 10_000, 100_000):
        cases[f"balanced G={G}"] = (rng.permutation(np.arange(N) % G), G)
    sk = rng.integers(1, 10_000, N)
    sk[rng.permutation(N)[: N // 2]] = 0
    cases["skewed G=10000 (half the rows in group 0)"] = (sk, 10_000)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def ri_call(grp, G, samp):
        beta = torch.empty(samp, P, device=dev, dtype=torch.float64)
        u = torch.empty(samp, G, device=dev, dtype=torch.float64)
        tau2 = torch.empty(samp, device=dev, dtype=torch.float64)
        y = grp[1]
        return lambda: _lib.check(L.bl_logit_ri_gibbs_dev(beta.data_ptr(), u.data_ptr(), tau2.data_ptr(), y.data_ptr(),
                                                          X.data_ptr(), n.data_ptr(), grp[0].data_ptr(), G,
                                                          m0.data_ptr(), P0.data_ptr(), 2.0, 2.0, 1.0, N, P, samp, 0,
                                                          7, 0, st))

    def plain_call(y, samp):
        beta = torch.empty(samp, P, device=dev, dtype=torch.float64)
        return lambda: _lib.check(L.bl_logit_gibbs_dev(None, beta.data_ptr(), y.data_ptr(), X.data_ptr(), n.data_ptr(),
                                                       m0.data_ptr(), P0.data_ptr(), N, P, samp, 0, 7, 3, 0, st))

    def per_iter(make):
        ms = []
        make(2)()                                       # warm-up of every kernel and the allocator
        for _ in range(a.reps):
            t0 = timed(make(a.short))
            t1 = timed(make(a.long))
            ms.append((t1 - t0) / (a.long - a.short))
        return ms

    res = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "N": N, "P": P, "cases": {}}
    for name, (ids, G) in cases.items():
        gid = torch.from_numpy(ids.astype(np.int32)).to(dev)
        ut = torch.randn(G, generator=g, device=dev, dtype=torch.float64)
        y = torch.bernoulli(torch.sigmoid(X @ bt + ut[gid.long()]), generator=g)
        grp = (gid, y)
        ri = per_iter(lambda s: ri_call(grp, G, s))
        pl = per_iter(lambda s: plain_call(y, s))
        r, p = float(np.median(ri)), float(np.median(pl))
        res["cases"][name] = {
            "G": G, "ri_ms_per_iter": r, "ri_ms_all": ri, "plain_logit_ms_per_iter": p, "plain_ms_all": pl,
            "ratio": r / p,
            "ri_stages_us": stage_lines(ri_call(grp, G, 3)),
            "plain_stages_us": stage_lines(plain_call(y, 3)),
        }
        print(json.dumps({name: res["cases"][name]}), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"]}))


if __name__ == "__main__":
    main()
