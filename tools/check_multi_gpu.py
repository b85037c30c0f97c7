#!/usr/bin/env python3
"""Multi-GPU check of the sharded sweeps (run under torchrun, one rank per GPU): the row-sharded logit /
multinomial logit / NB chains (the NB ones with the dispersion fixed, drawn on the integers and drawn on the reals) equal the single-GPU chains and beta is bit-identical on every rank -- on the peer-window
exchange (NCCL communicator + NVLink windows), on ncclAllReduce alone (BL_PEER_EXCHANGE=0), and on the
windows alone (bl_comm_init_local: no NCCL communicator, the set-up sums go through k_peer_put /
k_peer_combine too).  Prints MULTI_GPU_OK on rank 0.  One-GPU boxes: tests/test_gpu_multi.py runs the
same exchange kernels with virtual ranks (bl_vcomm_*)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bayeslogit_b200 import _lib, dist as bdist  # noqa: E402

LOCAL_MODE = False           # set below for the pass without an NCCL communicator
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
local = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
L = _lib.lib()
_lib.check(L.bl_set_device(local))
dist.init_process_group("nccl", device_id=dev)


def open_comm():
    if LOCAL_MODE:
        bdist.init_comm_local(rank, world, dev)
    else:
        bdist.init_comm(rank, world, dev)


def allmax(vals):
    t = torch.tensor(list(vals), dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t.cpu()]


def same_on_all_ranks(a):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    g = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(g, t)
    return all(torch.equal(g[0], x) for x in g)


st = torch.cuda.current_stream().cuda_stream
samp, burn = 12, 4


def make(N, P, seed):
    rng = np.random.default_rng(seed)
    X = np.c_[rng.standard_normal((N, P - 1)), np.ones(N)]
    bt = np.r_[np.abs(rng.normal(0, 0.3, P - 1)), -0.5]
    y = (rng.random(N) < 1 / (1 + np.exp(-X @ bt))).astype(float)
    yc = rng.poisson(np.exp(np.clip(X @ bt * 0.3 + 2.0, None, 4.0))).astype(float)
    return X, y, yc


def chain(X, y, lo, hi, flags):
    P = X.shape[1]
    Xd = torch.from_numpy(X[lo:hi].copy()).to(dev); yd = torch.from_numpy(y[lo:hi].copy()).to(dev)
    nd = torch.ones(hi - lo, device=dev, dtype=torch.float64)
    m0 = torch.zeros(P, device=dev, dtype=torch.float64)
    P0 = (0.1 * torch.eye(P, device=dev, dtype=torch.float64)).contiguous()
    beta = torch.zeros(samp, P, device=dev, dtype=torch.float64)
    w = torch.zeros(samp, hi - lo, device=dev, dtype=torch.float64)
    rc = L.bl_logit_gibbs_dev(w.data_ptr(), beta.data_ptr(), yd.data_ptr(), Xd.data_ptr(), nd.data_ptr(),
                              m0.data_ptr(), P0.data_ptr(), hi - lo, P, samp, burn, 4242, flags, lo, st)
    if rc:
        _lib.check(rc)
    torch.cuda.synchronize()
    return beta.cpu().numpy(), w.cpu().numpy()


def prior_chain(X, y, n, lo, hi, flags):
    """Logit sweep with a non-zero prior mean and a dense prior precision (b0 = P0 m0 must be added once, after the
    all-reduce of X'kappa) and binomial counts."""
    P = X.shape[1]
    Xd = torch.from_numpy(X[lo:hi].copy()).to(dev); yd = torch.from_numpy(y[lo:hi].copy()).to(dev)
    nd = torch.from_numpy(n[lo:hi].copy()).to(dev)
    m0 = torch.linspace(-0.1, 0.1, P, device=dev, dtype=torch.float64)
    P0 = (0.5 * torch.eye(P, device=dev, dtype=torch.float64) + 0.01).contiguous()
    beta = torch.zeros(6, P, device=dev, dtype=torch.float64)
    w = torch.zeros(6, hi - lo, device=dev, dtype=torch.float64)
    rc = L.bl_logit_gibbs_dev(w.data_ptr(), beta.data_ptr(), yd.data_ptr(), Xd.data_ptr(), nd.data_ptr(),
                              m0.data_ptr(), P0.data_ptr(), hi - lo, P, 6, 3, 4243, flags, lo, st)
    if rc:
        _lib.check(rc)
    torch.cuda.synchronize()
    return beta.cpu().numpy(), w.cpu().numpy()


def make_binomial(N, P, seed, binomial):
    rng = np.random.default_rng(seed)
    X = np.c_[rng.standard_normal((N, P - 1)), np.ones(N)]
    bt = np.r_[np.abs(rng.normal(0, 0.4, P - 1)), -0.5]
    p = 1 / (1 + np.exp(-X @ bt))
    n = rng.integers(1, 6, N).astype(float) if binomial else np.ones(N)
    y = rng.binomial(n.astype(int), p) / n
    return X, y, n


def nb_chain(X, yc, lo, hi):
    P = X.shape[1]
    Xd = torch.from_numpy(X[lo:hi].copy()).to(dev); yd = torch.from_numpy(yc[lo:hi].copy()).to(dev)
    m0 = torch.zeros(P, device=dev, dtype=torch.float64)
    P0 = (0.1 * torch.eye(P, device=dev, dtype=torch.float64)).contiguous()
    beta = torch.zeros(8, P, device=dev, dtype=torch.float64)
    w = torch.zeros(hi - lo, device=dev, dtype=torch.float64)
    rc = L.bl_nb_gibbs_dev(w.data_ptr(), beta.data_ptr(), yd.data_ptr(), Xd.data_ptr(), 5.0,
                           m0.data_ptr(), P0.data_ptr(), hi - lo, P, 8, 777, lo, st)
    if rc:
        _lib.check(rc)
    torch.cuda.synchronize()
    return beta.cpu().numpy(), w.cpu().numpy()


def nb_df_chain(X, yc, lo, hi):
    """NB sweep with the dispersion sampled on the device (draw.df): sharded, ymax / the count histogram /
    the log-likelihood sums of every Metropolis step are all-reduced."""
    P = X.shape[1]
    Xd = torch.from_numpy(X[lo:hi].copy()).to(dev); yd = torch.from_numpy(yc[lo:hi].copy()).to(dev)
    m0 = torch.zeros(P, device=dev, dtype=torch.float64)
    P0 = (0.1 * torch.eye(P, device=dev, dtype=torch.float64)).contiguous()
    beta = torch.zeros(10, P, device=dev, dtype=torch.float64)
    dd = torch.zeros(10, device=dev, dtype=torch.float64)
    rc = L.bl_nb_gibbs_df_dev(None, beta.data_ptr(), dd.data_ptr(), yd.data_ptr(), Xd.data_ptr(), 1.0,
                              m0.data_ptr(), P0.data_ptr(), hi - lo, P, 10, 6, 4711, lo, st)
    if rc:
        _lib.check(rc)
    torch.cuda.synchronize()
    return beta.cpu().numpy(), dd.cpu().numpy()


def nb_dfreal_chain(X, yc, lo, hi):
    """NB sweep with the dispersion walking on the reals (draw.df.real.mean): b = y + d is non-integer."""
    P = X.shape[1]
    Xd = torch.from_numpy(X[lo:hi].copy()).to(dev); yd = torch.from_numpy(yc[lo:hi].copy()).to(dev)
    m0 = torch.zeros(P, device=dev, dtype=torch.float64)
    P0 = (0.1 * torch.eye(P, device=dev, dtype=torch.float64)).contiguous()
    beta = torch.zeros(10, P, device=dev, dtype=torch.float64)
    dd = torch.zeros(10, device=dev, dtype=torch.float64)
    rc = L.bl_nb_gibbs_dfreal_dev(None, beta.data_ptr(), dd.data_ptr(), yd.data_ptr(), Xd.data_ptr(), 2.5,
                                  m0.data_ptr(), P0.data_ptr(), hi - lo, P, 10, 6, 4713, lo, st)
    if rc:
        _lib.check(rc)
    torch.cuda.synchronize()
    return beta.cpu().numpy(), dd.cpu().numpy()


def nb_mode_chain(mode, X, yc, lo, hi):
    """NB sweep in one of the three dispersion modes with a non-zero prior mean and a dense prior precision (so
    b0 = P0 m0 enters the beta draw).  Returns (beta, d)."""
    P = X.shape[1]
    Xd = torch.from_numpy(X[lo:hi].copy()).to(dev); yd = torch.from_numpy(yc[lo:hi].copy()).to(dev)
    m0 = torch.linspace(-0.4, 0.4, P, device=dev, dtype=torch.float64)
    P0 = (0.02 * torch.eye(P, device=dev, dtype=torch.float64) + 0.005).contiguous()
    beta = torch.zeros(6, P, device=dev, dtype=torch.float64)
    dd = torch.full((6,), 2.0, device=dev, dtype=torch.float64)
    if mode == "fixed":
        rc = L.bl_nb_gibbs_dev(None, beta.data_ptr(), yd.data_ptr(), Xd.data_ptr(), 2.0, m0.data_ptr(),
                               P0.data_ptr(), hi - lo, P, 6, 919, lo, st)
    else:
        fn = L.bl_nb_gibbs_dfreal_dev if mode == "real" else L.bl_nb_gibbs_df_dev
        rc = fn(None, beta.data_ptr(), dd.data_ptr(), yd.data_ptr(), Xd.data_ptr(), 2.5 if mode == "real" else 2.0,
                m0.data_ptr(), P0.data_ptr(), hi - lo, P, 6, 3, 919, lo, st)
    if rc:
        _lib.check(rc)
    torch.cuda.synchronize()
    return beta.cpu().numpy(), dd.cpu().numpy()


def make_mlogit(N, P, J, seed):
    rng = np.random.default_rng(seed)
    X = np.c_[rng.standard_normal((N, P - 1)) / np.sqrt(max(P - 1, 1)), np.ones(N)]
    eta = np.c_[X @ rng.normal(0, 0.4, (P, J - 1)), np.zeros(N)]
    pr = np.exp(eta)
    pr /= pr.sum(1, keepdims=True)
    cat = (pr.cumsum(1) < rng.random(N)[:, None]).sum(1)
    Y = np.eye(J)[np.minimum(cat, J - 1)][:, :J - 1]
    m0 = rng.normal(0, 0.05, (P, J - 1))
    P0 = np.stack([(0.5 + 0.05 * j) * np.eye(P) for j in range(J - 1)], axis=2)
    return X, Y, m0, P0


def mlogit_chain(X, Y, m0, P0, lo, hi):
    """Multinomial logit sweep: each category's X'kappa set-up and its 2 exchanges per update are all-reduced;
    at P = 32 X'(Omega c_j) travels in the packed Gram's partial tile with the P^2 sums."""
    P, U = X.shape[1], Y.shape[1]
    Xd = torch.from_numpy(X[lo:hi].copy()).to(dev); yd = torch.from_numpy(Y[lo:hi].copy()).to(dev)
    nd = torch.ones(hi - lo, device=dev, dtype=torch.float64)
    m0d = torch.from_numpy(np.asfortranarray(m0).ravel(order="F")).to(dev)
    P0d = torch.from_numpy(np.asfortranarray(P0).ravel(order="F")).to(dev)
    beta = torch.zeros(5, U, P, device=dev, dtype=torch.float64)
    w = torch.zeros(5, U, hi - lo, device=dev, dtype=torch.float64)
    rc = L.bl_mlogit_gibbs_dev(w.data_ptr(), beta.data_ptr(), yd.data_ptr(), Xd.data_ptr(), nd.data_ptr(),
                               m0d.data_ptr(), P0d.data_ptr(), hi - lo, P, U + 1, 5, 2, 808, 0, lo, st)
    if rc:
        _lib.check(rc)
    torch.cuda.synchronize()
    return beta.cpu().numpy(), w.cpu().numpy()


# P = 16: the vectorised slot copy; P = 7, 15: odd P (P*P sums without a tail is an odd count -- the last
# Gram entry travels on its own); N not a multiple of anything convenient
CASES = [(200_003, 16), (50_001, 7), (60_001, 15)]
data = {c: make(c[0], c[1], 10 + c[1]) for c in CASES}
full = {(c, f): chain(data[c][0], data[c][1], 0, c[0], f) for c in CASES for f in (0, 1)}   # no communicator yet
c0 = CASES[0]
nb_full = nb_chain(data[c0][0], data[c0][2], 0, c0[0])
nbdf_full = nb_df_chain(data[c0][0], data[c0][2], 0, c0[0])
nbdfreal_full = nb_dfreal_chain(data[c0][0], data[c0][2], 0, c0[0])
# (N, P, J): P = 16 vectorised slot copy; P = 7 odd P^2 count; P = 32 the packed Gram's X'(Omega c_j) tail
MCASES = [(200_003, 16, 4), (50_001, 7, 3), (60_001, 32, 5)]
mdata = {c: make_mlogit(c[0], c[1], c[2], 20 + c[1]) for c in MCASES}
mfull = {c: mlogit_chain(*mdata[c], 0, c[0]) for c in MCASES}
# NB in all three dispersion modes: P = 7 odd P^2 count (k_xtv_partial), P = 70 several Gram tiles
NBCASES = [(9_001, 7), (12_001, 70)]
NBMODES = ["fixed", "int", "real"]
nbdata = {c: make(c[0], c[1], 30 + c[1]) for c in NBCASES}
nbfull = {(c, m): nb_mode_chain(m, nbdata[c][0], nbdata[c][2], 0, c[0]) for c in NBCASES for m in NBMODES}
# logit with a non-zero m0 and a dense P0, both beta draws: (N, P, binomial, flag variants).  P = 32: the packed
# Gram, binomial counts; P = 64: the one-pass kernel's published sums and (BL_GIBBS_TWO_PASS) k_gram_reduce's;
# P = 70: several Gram tiles, the constrained draw at P > 64; P = 128: the beta draw out of global scratch
PCASES = [(60_001, 32, True, (0,)), (50_001, 64, False, (0, 16)), (24_001, 70, False, (0,)), (12_001, 128, False, (0,))]
pdata = {c: make_binomial(c[0], c[1], 40 + c[1], c[2]) for c in PCASES}
pruns = [(c, f | b) for c in PCASES for f in c[3] for b in (0, 1)]
pfull = {k: prior_chain(*pdata[k[0]], 0, k[0][0], k[1]) for k in pruns}

ok = True


def sharded_pass(tag):
    global ok
    for c in CASES:
        lo, hi = bdist.shard_range(rank, world, c[0])
        for f in (0, 1):
            b, w = chain(data[c][0], data[c][1], lo, hi, f)
            fb, fw = full[(c, f)]
            eb = np.max(np.abs(b - fb) / np.abs(fb))
            ew = np.max(np.abs(w - fw[:, lo:hi]) / fw[:, lo:hi])
            eb, ew = allmax([eb, ew])
            same = same_on_all_ranks(b)
            if rank == 0:
                print(f"[{tag}] logit N={c[0]} P={c[1]} flags={f}: world={world} max rel diff beta {eb:.2e} omega {ew:.2e}; "
                      f"beta bit-identical across ranks: {same}", flush=True)
            ok = ok and max(eb, ew) < 1e-8 and same
    for k in pruns:
        c, f = k
        lo, hi = bdist.shard_range(rank, world, c[0])
        b, w = prior_chain(*pdata[c], lo, hi, f)
        fb, fw = pfull[k]
        eb, ew = allmax([np.max(np.abs(b - fb) / np.abs(fb)), np.max(np.abs(w - fw[:, lo:hi]) / fw[:, lo:hi])])
        same = same_on_all_ranks(b)
        if rank == 0:
            print(f"[{tag}] logit (non-zero m0, dense P0) N={c[0]} P={c[1]} flags={f}: world={world} max rel diff "
                  f"beta {eb:.2e} omega {ew:.2e}; beta bit-identical across ranks: {same}", flush=True)
        ok = ok and max(eb, ew) < 1e-8 and same
    lo, hi = bdist.shard_range(rank, world, c0[0])
    b, w = nb_chain(data[c0][0], data[c0][2], lo, hi)
    eb = np.max(np.abs(b - nb_full[0]) / np.abs(nb_full[0]))
    ew = np.max(np.abs(w - nb_full[1][lo:hi]) / nb_full[1][lo:hi])
    eb, ew = allmax([eb, ew])
    same = same_on_all_ranks(b)
    if rank == 0:
        print(f"[{tag}] nb: max rel diff beta {eb:.2e} omega {ew:.2e}; beta bit-identical across ranks: {same}", flush=True)
    ok = ok and max(eb, ew) < 1e-8 and same
    b_df, d_df = nb_df_chain(data[c0][0], data[c0][2], lo, hi)
    e_df = float(np.max(np.abs(b_df - nbdf_full[0]) / np.abs(nbdf_full[0])))
    same_d = bool(np.array_equal(d_df, nbdf_full[1]))
    e_df, bad_d = allmax([e_df, 0.0 if same_d else 1.0])
    if rank == 0:
        print(f"[{tag}] nb with dispersion update: max rel diff beta {e_df:.2e}; d chain identical to the single-GPU chain "
              f"on every rank: {bad_d == 0.0} (d: {d_df[0]:.0f} .. {d_df[-1]:.0f})", flush=True)
    ok = ok and e_df < 1e-8 and bad_d == 0.0
    b_dr, d_dr = nb_dfreal_chain(data[c0][0], data[c0][2], lo, hi)
    e_dr = float(np.max(np.abs(b_dr - nbdfreal_full[0]) / np.abs(nbdfreal_full[0])))
    ed_dr = float(np.max(np.abs(d_dr - nbdfreal_full[1]) / np.abs(nbdfreal_full[1])))
    same_dr = same_on_all_ranks(d_dr) and same_on_all_ranks(b_dr)
    e_dr, ed_dr = allmax([e_dr, ed_dr])
    if rank == 0:
        print(f"[{tag}] nb with real-valued dispersion: max rel diff beta {e_dr:.2e} d {ed_dr:.2e}; beta and d "
              f"bit-identical across ranks: {same_dr} (d: {d_dr[0]:.3f} .. {d_dr[-1]:.3f})", flush=True)
    ok = ok and e_dr < 1e-8 and ed_dr < 1e-12 and same_dr
    for c in NBCASES:
        lo, hi = bdist.shard_range(rank, world, c[0])
        for m in NBMODES:
            b, d = nb_mode_chain(m, nbdata[c][0], nbdata[c][2], lo, hi)
            fb, fd = nbfull[(c, m)]
            eb, ed = allmax([np.max(np.abs(b - fb) / np.abs(fb)), np.max(np.abs(d - fd) / np.abs(fd))])
            same = same_on_all_ranks(b) and same_on_all_ranks(d)
            if rank == 0:
                print(f"[{tag}] nb ({m} d) N={c[0]} P={c[1]}: world={world} max rel diff beta {eb:.2e} d {ed:.2e}; "
                      f"beta and d bit-identical across ranks: {same}", flush=True)
            ok = ok and eb < 1e-8 and (ed < 1e-12 if m == "real" else ed == 0.0) and same
    for c in MCASES:
        lo, hi = bdist.shard_range(rank, world, c[0])
        b, w = mlogit_chain(*mdata[c], lo, hi)
        fb, fw = mfull[c]
        eb = np.max(np.abs(b - fb) / np.abs(fb))
        ew = np.max(np.abs(w - fw[..., lo:hi]) / fw[..., lo:hi])
        eb, ew = allmax([eb, ew])
        same = same_on_all_ranks(b)
        if rank == 0:
            print(f"[{tag}] mlogit N={c[0]} P={c[1]} J={c[2]}: world={world} max rel diff beta {eb:.2e} omega {ew:.2e}; "
                  f"beta bit-identical across ranks: {same}", flush=True)
        ok = ok and max(eb, ew) < 1e-8 and same


open_comm()
peer = bdist.peer_exchange_active()
sharded_pass("peer windows" if peer else "nccl")
if peer:
    # the NCCL path on the same shards
    bdist.destroy_comm()
    os.environ["BL_PEER_EXCHANGE"] = "0"
    bdist.init_comm(rank, world, dev)
    assert not bdist.peer_exchange_active()
    sharded_pass("nccl")
    # ... and the windows alone, without an NCCL communicator
    bdist.destroy_comm()
    os.environ["BL_PEER_EXCHANGE"] = "1"
    LOCAL_MODE = True
    open_comm()
    assert bdist.peer_exchange_active()
    sharded_pass("peer windows, no NCCL communicator")
if rank == 0:
    print(f"peer exchange active: {peer}")
    print("MULTI_GPU_OK" if ok else "MULTI_GPU_MISMATCH", flush=True)
bdist.destroy_comm()
dist.destroy_process_group()
