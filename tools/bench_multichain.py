#!/usr/bin/env python3
"""Several logit chains on one data set (bl_logit_multichain) against the two ways to get them without it.

    python tools/bench_multichain.py [--N 1000000 --P 64 --chains 1,2,4,8 --iters 20 --reps 3]
    python tools/bench_multichain.py --model mlogit [--N 1000000 --P 32 --J 10 --chains 1,2,4,8 --iters 20 --reps 3]
    python tools/bench_multichain.py --model nb [--dmode int|real|fixed --N 1000000 --P 64 --chains 1,2,4,8 ...]
    python tools/bench_multichain.py --model ri [--N 1000000 --P 64 --G 10000 --chains 1,2,4,8 --iters 20 --reps 3]

For every chain count K and both beta draws, three arms are timed alternately in the same process, on the same
device-resident data, and reported as ms per iteration of all K chains (median over the repetitions):
  (a) multichain: bl_logit_multichain_dev, one copy of X shared by the K chains;
  (b) replicated: bl_logit_chains_dev on K copies of X (the batch entry for chains that own their rows);
  (c) sequential: K calls of bl_logit_gibbs_dev, one chain after the other.
(a) and (b) start from the same seed and must give the same beta bit for bit (max_abs_diff_a_b).  The
BL_GIBBS_TIMING stage split of one iteration of (a) and (b) comes from a separate, untimed call.  X is 512 MB at
the default size, larger than L2, so every pass reads it from HBM.  Prints one JSON line.

--model mlogit: multinomial logit chains (bl_mlogit_multichain), two arms alternated the same way:
  (a) multichain: bl_mlogit_multichain_dev, one copy of X shared by the K chains;
  (b) sequential: K calls of bl_mlogit_gibbs_dev with seed + c and omega dropped.
Chain c of (a) must equal call c of (b) bit for bit (max_abs_diff_a_b).  Also reported: the stage split of the last
category update of both arms and the kernel launches per iteration (bl_kernel_launches over a timed call / its
iterations).  X is 256 MB at the default size (N = 1M, P = 32).

--model nb: negative-binomial chains (bl_nb_multichain) with the dispersion walk of --dmode, two arms alternated the
same way:
  (a) multichain: bl_nb_multichain_dev, one copy of X shared by the K chains;
  (b) sequential: K calls of bl_nb_gibbs_df_dev / bl_nb_gibbs_dfreal_dev / bl_nb_gibbs_dev with seed + c.
Both arms run without burn-in, so chain c of (a) must equal call c of (b) bit for bit, beta and d
(max_abs_diff_a_b).  Also reported: the multichain stage split of the last iteration and the kernel launches per
iteration.  Counts have mean ~ 100 (b = y + d mostly in the saddle-point range, as BASELINE config 4).

--model ri: random-intercept logit chains (bl_logit_ri_multichain), ids balanced over --G groups in random row order,
two arms alternated the same way:
  (a) multichain: bl_logit_ri_multichain_dev, one copy of X, y, n and the ids shared by the K chains;
  (b) sequential: K calls of bl_logit_ri_gibbs_dev with seed + c.
Both arms run without burn-in, so chain c of (a) must equal call c of (b) bit for bit, beta, u and tau2
(max_abs_diff_a_b).  Also reported: the stage split of the last iteration of both arms and the kernel launches per
iteration.

The card name, power limit and max SM clock are read in the same run.
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


def card():
    """Name, power limit (W) and max SM clock (MHz) of the device, read where the numbers are measured."""
    import torch
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        fields = out.stdout.strip().splitlines()[0].split(",") if out.returncode == 0 else []
        power = float(fields[0]) if fields else None
        clock = float(fields[1]) if len(fields) > 1 else None
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        power = clock = None
    return name, power, clock


def stage_split(fn):
    """Run fn() with BL_GIBBS_TIMING set and return the stage times (us) the driver prints to stderr."""
    import torch
    torch.cuda.synchronize()
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 2)
        os.environ["BL_GIBBS_TIMING"] = "1"
        try:
            fn()
            torch.cuda.synchronize()
        finally:
            del os.environ["BL_GIBBS_TIMING"]
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        text = f.read()
    lines = [l for l in text.splitlines() if "timing, us]" in l]
    if not lines:
        return None
    return {k: float(v) for k, v in re.findall(r"([a-z+]+) ([0-9.]+)", lines[-1].split("]", 1)[1])}


def run(N, P, ks, iters, reps):
    import torch
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    dev = torch.device("cuda")
    g = torch.Generator(device=dev); g.manual_seed(20240007)
    X = torch.randn(N, P, generator=g, device=dev, dtype=torch.float64)
    X[:, P - 1] = 1.0
    bt = torch.randn(P, generator=g, device=dev, dtype=torch.float64).abs() * 0.25
    bt[P - 1] = -0.5
    y = (torch.rand(N, generator=g, device=dev, dtype=torch.float64) < torch.sigmoid(X @ bt)).double()
    n = torch.ones(N, device=dev, dtype=torch.float64)
    m0 = torch.zeros(P, device=dev, dtype=torch.float64)
    P0 = (0.01 * torch.eye(P, device=dev, dtype=torch.float64)).contiguous()
    st = torch.cuda.current_stream().cuda_stream
    seed = 20240007
    row_bytes = (P + 2) * 8                                  # a row of X, its y and its n
    out = {"N": N, "P": P, "iters": iters, "reps": reps, "results": []}

    for constrained in (True, False):
        flags = 0 if constrained else 1
        for K in ks:
            Xr = X.unsqueeze(0).expand(K, N, P).contiguous()
            yr = y.unsqueeze(0).expand(K, N).contiguous()
            nr = n.unsqueeze(0).expand(K, N).contiguous()

            def multichain(k):
                beta = torch.zeros(K, k, P, device=dev, dtype=torch.float64)
                _lib.check(L.bl_logit_multichain_dev(beta.data_ptr(), y.data_ptr(), X.data_ptr(), n.data_ptr(),
                                                     m0.data_ptr(), P0.data_ptr(), K, N, P, k, 0, seed, flags, st))
                return beta

            def replicated(k):
                beta = torch.zeros(K, k, P, device=dev, dtype=torch.float64)
                _lib.check(L.bl_logit_chains_dev(beta.data_ptr(), yr.data_ptr(), Xr.data_ptr(), nr.data_ptr(),
                                                 m0.data_ptr(), P0.data_ptr(), K, N, P, k, 0, seed, flags, st))
                return beta

            def sequential(k):
                beta = torch.zeros(K, k, P, device=dev, dtype=torch.float64)
                for c in range(K):
                    _lib.check(L.bl_logit_gibbs_dev(None, beta[c].data_ptr(), y.data_ptr(), X.data_ptr(), n.data_ptr(),
                                                    m0.data_ptr(), P0.data_ptr(), N, P, k, 0, seed + c, flags | 2, 0, st))
                return beta

            arms = {"multichain": multichain, "replicated": replicated, "sequential": sequential}
            for fn in arms.values():                     # warm-up: modules, pools, every kernel of the timed window
                fn(2)
            torch.cuda.synchronize()
            times = {a: [] for a in arms}
            betas = {}
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for _ in range(reps):
                for a, fn in arms.items():               # alternated: drifts of the shared machine hit every arm
                    e0.record()
                    betas[a] = fn(iters)
                    e1.record()
                    torch.cuda.synchronize()
                    times[a].append(e0.elapsed_time(e1) / iters)
            med = {a: sorted(v)[len(v) // 2] for a, v in times.items()}
            diff = float((betas["multichain"] - betas["replicated"]).abs().max().item())
            out["results"].append({
                "beta_draw": "constrained" if constrained else "plain", "chains": K,
                "ms_per_iteration_of_all_chains": med,
                "ms_all_reps": times,
                "multichain_over_replicated": med["multichain"] / med["replicated"],
                "sequential_over_multichain": med["sequential"] / med["multichain"],
                "max_abs_diff_a_b": diff,
                "stages_us": {"multichain": stage_split(lambda: multichain(2)),
                              "replicated": stage_split(lambda: replicated(2))},
                "input_bytes_on_device": {"multichain": N * row_bytes, "replicated": K * N * row_bytes,
                                          "sequential": N * row_bytes},
            })
            del Xr, yr, nr
            torch.cuda.empty_cache()
    return out


def run_mlogit(N, P, J, ks, iters, reps):
    import torch
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    dev = torch.device("cuda")
    U = J - 1
    g = torch.Generator(device=dev); g.manual_seed(20240011)
    X = torch.randn(N, P, generator=g, device=dev, dtype=torch.float64) / (P - 1) ** 0.5
    X[:, P - 1] = 1.0
    B = torch.randn(P, U, generator=g, device=dev, dtype=torch.float64) * 0.5
    logits = torch.cat([X @ B, torch.zeros(N, 1, device=dev, dtype=torch.float64)], dim=1)
    cat = torch.multinomial(torch.softmax(logits, dim=1), 1, generator=g).squeeze(1)
    Y = torch.nn.functional.one_hot(cat, J)[:, :U].double().contiguous()     # N x U row-major = ty, U x N column-major
    n = torch.ones(N, device=dev, dtype=torch.float64)
    m0 = torch.zeros(U, P, device=dev, dtype=torch.float64)                  # P x U column-major
    P0 = (0.01 * torch.eye(P, device=dev, dtype=torch.float64)).expand(U, P, P).contiguous()
    st = torch.cuda.current_stream().cuda_stream
    seed = 20240011
    out = {"model": "mlogit", "N": N, "P": P, "J": J, "iters": iters, "reps": reps, "results": []}

    for K in ks:
        def multichain(k):
            beta = torch.zeros(K, k, U, P, device=dev, dtype=torch.float64)
            _lib.check(L.bl_mlogit_multichain_dev(beta.data_ptr(), Y.data_ptr(), X.data_ptr(), n.data_ptr(),
                                                  m0.data_ptr(), P0.data_ptr(), K, N, P, J, k, 0, seed, 0, st))
            return beta

        def sequential(k):
            beta = torch.zeros(K, k, U, P, device=dev, dtype=torch.float64)
            for c in range(K):
                _lib.check(L.bl_mlogit_gibbs_dev(None, beta[c].data_ptr(), Y.data_ptr(), X.data_ptr(), n.data_ptr(),
                                                 m0.data_ptr(), P0.data_ptr(), N, P, J, k, 0, seed + c, 2, 0, st))
            return beta

        arms = {"multichain": multichain, "sequential": sequential}
        for fn in arms.values():                         # warm-up: modules, pools, every kernel of the timed window
            fn(2)
        torch.cuda.synchronize()
        times = {a: [] for a in arms}
        launches = {}
        betas = {}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(reps):
            for a, fn in arms.items():                   # alternated: drifts of the shared machine hit every arm
                l0 = L.bl_kernel_launches()
                e0.record()
                betas[a] = fn(iters)
                e1.record()
                torch.cuda.synchronize()
                launches[a] = (L.bl_kernel_launches() - l0) / iters
                times[a].append(e0.elapsed_time(e1) / iters)
        med = {a: sorted(v)[len(v) // 2] for a, v in times.items()}
        diff = float((betas["multichain"] - betas["sequential"]).abs().max().item())
        out["results"].append({
            "chains": K,
            "ms_per_iteration_of_all_chains": med,
            "ms_all_reps": times,
            "sequential_over_multichain": med["sequential"] / med["multichain"],
            "max_abs_diff_a_b": diff,
            "launches_per_iteration": launches,
            "stages_us": {"multichain": stage_split(lambda: multichain(2)),
                          "sequential_one_chain": stage_split(lambda: sequential(2))},
        })
    return out


def run_nb(N, P, dmode, ks, iters, reps):
    import torch
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    dev = torch.device("cuda")
    g = torch.Generator(device=dev); g.manual_seed(20240013)
    X = torch.randn(N, P, generator=g, device=dev, dtype=torch.float64) / P ** 0.5
    X[:, P - 1] = 1.0
    bt = torch.randn(P, generator=g, device=dev, dtype=torch.float64) * 0.5
    bt[P - 1] = 4.6                                      # mean count ~ 100
    d_true = 10.0
    mu = torch.exp(X @ bt)
    torch.manual_seed(20240013)                          # the gamma draw below takes the global generator
    lam = torch.distributions.Gamma(torch.full_like(mu, d_true), d_true / mu).sample()     # NB = Poisson-gamma mix
    y = torch.poisson(lam, generator=g).contiguous()
    m0 = torch.zeros(P, device=dev, dtype=torch.float64)
    P0 = (0.01 * torch.eye(P, device=dev, dtype=torch.float64)).contiguous()
    st = torch.cuda.current_stream().cuda_stream
    seed = 20240013
    code = {"fixed": 0, "int": 1, "real": 2}[dmode]
    d0 = 10.0 if dmode == "fixed" else 3.0
    out = {"model": "nb", "dmode": dmode, "N": N, "P": P, "d0": d0, "iters": iters, "reps": reps, "results": []}

    for K in ks:
        def multichain(k):
            beta = torch.zeros(K, k, P, device=dev, dtype=torch.float64)
            d = torch.zeros(K, k, device=dev, dtype=torch.float64)
            _lib.check(L.bl_nb_multichain_dev(beta.data_ptr(), d.data_ptr(), y.data_ptr(), X.data_ptr(), d0,
                                              m0.data_ptr(), P0.data_ptr(), K, N, P, k, 0, seed, code, st))
            return beta, d

        def sequential(k):
            beta = torch.zeros(K, k, P, device=dev, dtype=torch.float64)
            d = torch.full((K, k), d0, device=dev, dtype=torch.float64)
            for c in range(K):
                if dmode == "fixed":
                    rc = L.bl_nb_gibbs_dev(None, beta[c].data_ptr(), y.data_ptr(), X.data_ptr(), d0, m0.data_ptr(),
                                           P0.data_ptr(), N, P, k, seed + c, 0, st)
                else:
                    fn = L.bl_nb_gibbs_dfreal_dev if dmode == "real" else L.bl_nb_gibbs_df_dev
                    rc = fn(None, beta[c].data_ptr(), d[c].data_ptr(), y.data_ptr(), X.data_ptr(), d0, m0.data_ptr(),
                            P0.data_ptr(), N, P, k, 0, seed + c, 0, st)
                _lib.check(rc)
            return beta, d

        arms = {"multichain": multichain, "sequential": sequential}
        for fn in arms.values():                         # warm-up: modules, pools, every kernel of the timed window
            fn(2)
        torch.cuda.synchronize()
        times = {a: [] for a in arms}
        launches = {}
        res = {}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(reps):
            for a, fn in arms.items():                   # alternated: drifts of the shared machine hit every arm
                l0 = L.bl_kernel_launches()
                e0.record()
                res[a] = fn(iters)
                e1.record()
                torch.cuda.synchronize()
                launches[a] = (L.bl_kernel_launches() - l0) / iters
                times[a].append(e0.elapsed_time(e1) / iters)
        med = {a: sorted(v)[len(v) // 2] for a, v in times.items()}
        diff = max(float((res["multichain"][i] - res["sequential"][i]).abs().max().item()) for i in (0, 1))
        out["results"].append({
            "chains": K,
            "ms_per_iteration_of_all_chains": med,
            "ms_all_reps": times,
            "sequential_over_multichain": med["sequential"] / med["multichain"],
            "max_abs_diff_a_b": diff,
            "d_moves": bool((res["multichain"][1] != res["multichain"][1][:, :1]).any().item()),
            "launches_per_iteration": launches,
            "stages_us": {"multichain": stage_split(lambda: multichain(2))},
        })
    return out


def run_ri(N, P, G, ks, iters, reps):
    import numpy as np
    import torch
    from bayeslogit_b200 import _lib
    L = _lib.lib()
    dev = torch.device("cuda")
    g = torch.Generator(device=dev); g.manual_seed(20240017)
    X = torch.randn(N, P, generator=g, device=dev, dtype=torch.float64) / P ** 0.5
    X[:, 0] = 1.0
    bt = torch.randn(P, generator=g, device=dev, dtype=torch.float64) * 0.5
    ids = np.random.default_rng(17).permutation(np.arange(N) % G)
    grp = torch.from_numpy(ids.astype(np.int32)).to(dev)
    ut = 0.8 * torch.randn(G, generator=g, device=dev, dtype=torch.float64)
    y = torch.bernoulli(torch.sigmoid(X @ bt + ut[grp.long()]), generator=g)
    n = torch.ones(N, device=dev, dtype=torch.float64)
    m0 = torch.zeros(P, device=dev, dtype=torch.float64)
    P0 = (0.01 * torch.eye(P, device=dev, dtype=torch.float64)).contiguous()
    st = torch.cuda.current_stream().cuda_stream
    seed = 20240017
    a0, b0, tau2_0 = 2.0, 2.0, 1.0
    out = {"model": "ri", "N": N, "P": P, "G": G, "iters": iters, "reps": reps, "results": []}

    for K in ks:
        def multichain(k):
            beta = torch.zeros(K, k, P, device=dev, dtype=torch.float64)
            u = torch.zeros(K, k, G, device=dev, dtype=torch.float64)
            tau2 = torch.zeros(K, k, device=dev, dtype=torch.float64)
            _lib.check(L.bl_logit_ri_multichain_dev(beta.data_ptr(), u.data_ptr(), tau2.data_ptr(), y.data_ptr(),
                                                    X.data_ptr(), n.data_ptr(), grp.data_ptr(), G, m0.data_ptr(),
                                                    P0.data_ptr(), a0, b0, tau2_0, K, N, P, k, 0, seed, 0, st))
            return beta, u, tau2

        def sequential(k):
            beta = torch.zeros(K, k, P, device=dev, dtype=torch.float64)
            u = torch.zeros(K, k, G, device=dev, dtype=torch.float64)
            tau2 = torch.zeros(K, k, device=dev, dtype=torch.float64)
            for c in range(K):
                _lib.check(L.bl_logit_ri_gibbs_dev(beta[c].data_ptr(), u[c].data_ptr(), tau2[c].data_ptr(), y.data_ptr(),
                                                   X.data_ptr(), n.data_ptr(), grp.data_ptr(), G, m0.data_ptr(),
                                                   P0.data_ptr(), a0, b0, tau2_0, N, P, k, 0, seed + c, 0, st))
            return beta, u, tau2

        arms = {"multichain": multichain, "sequential": sequential}
        for fn in arms.values():                         # warm-up: modules, pools, every kernel of the timed window
            fn(2)
        torch.cuda.synchronize()
        times = {a: [] for a in arms}
        launches = {}
        res = {}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(reps):
            for a, fn in arms.items():                   # alternated: drifts of the shared machine hit every arm
                l0 = L.bl_kernel_launches()
                e0.record()
                res[a] = fn(iters)
                e1.record()
                torch.cuda.synchronize()
                launches[a] = (L.bl_kernel_launches() - l0) / iters
                times[a].append(e0.elapsed_time(e1) / iters)
        med = {a: sorted(v)[len(v) // 2] for a, v in times.items()}
        diff = max(float((res["multichain"][i] - res["sequential"][i]).abs().max().item()) for i in (0, 1, 2))
        out["results"].append({
            "chains": K,
            "ms_per_iteration_of_all_chains": med,
            "ms_all_reps": times,
            "sequential_over_multichain": med["sequential"] / med["multichain"],
            "max_abs_diff_a_b": diff,
            "launches_per_iteration": launches,
            "stages_us": {"multichain": stage_split(lambda: multichain(2)),
                          "sequential_one_chain": stage_split(lambda: sequential(2))},
        })
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", choices=["logit", "mlogit", "nb", "ri"], default="logit")
    ap.add_argument("--dmode", choices=["int", "real", "fixed"], default="int", help="dispersion walk (nb)")
    ap.add_argument("--N", type=int, default=1_000_000)
    ap.add_argument("--P", type=int, default=None, help="default 64 (logit, nb), 32 (mlogit)")
    ap.add_argument("--J", type=int, default=10, help="categories (mlogit)")
    ap.add_argument("--G", type=int, default=10_000, help="groups (ri)")
    ap.add_argument("--chains", default="1,2,4,8")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_multichain: no CUDA device")
    name, power, clock = card()
    ks = [int(k) for k in a.chains.split(",")]
    if a.model == "mlogit":
        out = run_mlogit(a.N, a.P or 32, a.J, ks, a.iters, a.reps)
    elif a.model == "ri":
        out = run_ri(a.N, a.P or 64, a.G, ks, a.iters, a.reps)
    elif a.model == "nb":
        out = run_nb(a.N, a.P or 64, a.dmode, ks, a.iters, a.reps)
    else:
        out = run(a.N, a.P or 64, ks, a.iters, a.reps)
    out["device"] = name
    out["power_limit_w"] = power
    out["max_sm_clock_mhz"] = clock
    print(json.dumps(out))


if __name__ == "__main__":
    main()
